"""Diagnostics: times the pipelined dense playout step (rules_kernel + expand_kernel) under the caller patterns set by
the FPC_P_* variables below; FPC_LIB_PATH points it at another build of the library.  usage: [FPC_P_...=1] python
tools/overlap_probe.py [steps] [fast_forward_plies]"""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from alphazero_4_player_chess_b200 import _lib
from alphazero_4_player_chess_b200.env import BatchedEnv
from alphazero_4_player_chess_b200.fen import start_record

if int(os.environ.get("FPC_P_OWNSTREAM", "0")):  # 1: work on a non-blocking torch stream instead of the legacy default stream
    torch.cuda.set_stream(torch.cuda.Stream())
steps = int(sys.argv[1]) if len(sys.argv) > 1 else 300
ff = int(sys.argv[2]) if len(sys.argv) > 2 else 0
L = _lib.lib()
env = BatchedEnv(14, 4096)
env.reset_playout(start_record("STANDARD", castling=True))
for _ in range(ff):
    env.playout_step(planes=False, mask=False)
host_state = int(os.environ.get("FPC_P_HOST", "0"))  # bit 0: boards, bit 1: game/ply, bit 2: counts/status in pinned host memory
torch.cuda.synchronize()
def to_host(t):
    h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    h.copy_(t)
    return h
if host_state & 1:
    env.boards = to_host(env.boards)
if host_state & 2:
    env.game, env.ply = to_host(env.game), to_host(env.ply)
if host_state & 4:
    env.counts, env.status = to_host(env.counts), to_host(env.status)
for _ in range(20):
    env.playout_step(planes=True, mask=True, async_dense=True)
env.join()
torch.cuda.synchronize()
noprof = int(os.environ.get("FPC_P_NOPROF", "0"))  # 1: no per-launch CUDA events around the two kernels
prof = not noprof and int(os.environ.get("FPC_P_PROF", "1")) != 0  # FPC_P_PROF=0: the same as FPC_P_NOPROF=1
_lib.check(L.fpc_profile_enable(int(prof)))
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
env.counters.zero_()
sync_each = int(os.environ.get("FPC_P_SYNC", "0"))  # 1: the host waits for every step's compact results (rules kernel)
main = torch.cuda.current_stream()
e0.record()
cpu_delay = float(os.environ.get("FPC_P_CPUDELAY", "0")) * 1e-6  # busy-wait on the host after every step's launches
import time as _time
trace = int(os.environ.get("FPC_P_TRACE", "0"))  # 1: an event on the main stream after every step (fires when that step's rules kernel is done)
marks = []
for _ in range(steps):
    env.playout_step(planes=True, mask=True, async_dense=True)
    if trace:
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        marks.append(ev)
    if sync_each:
        main.synchronize()
    if cpu_delay:
        t_ = _time.perf_counter()
        while _time.perf_counter() - t_ < cpu_delay:
            pass
env.join()
e1.record()
torch.cuda.synchronize()
if trace:
    ts = [e0.elapsed_time(m) * 1e3 for m in marks]
    print("rules-done times (us since start):", " ".join(f"{t:.0f}" for t in ts[:24]), "... end", f"{e0.elapsed_time(e1) * 1e3:.0f}")
n, ex, ru = ctypes.c_int(0), ctypes.c_double(0), ctypes.c_double(0)
_lib.check(L.fpc_profile_read(ctypes.byref(n), ctypes.byref(ex), ctypes.byref(ru)))
r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
r0.record()
for _ in range(steps):
    env.playout_step(planes=False, mask=False)
r1.record()
torch.cuda.synchronize()
knobs = {k: v for k, v in os.environ.items() if k.startswith("FPC_P_")}
c = env.counters.cpu()
print(f"{knobs}: step {e0.elapsed_time(e1) / steps * 1e3:.1f} us, expand in-loop {ex.value / max(n.value, 1) * 1e3:.1f} us, "
      f"rules in-loop {ru.value / max(n.value, 1) * 1e3:.1f} us, rules-only step {r0.elapsed_time(r1) / steps * 1e3:.1f} us, "
      f"avg legal {float(c[6]) / max(float(c[0]), 1):.1f}", flush=True)
