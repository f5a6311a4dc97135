#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

Workload (configs[1]): random-playout batched env, 4096 concurrent games per GPU on the 14x14 board
from the STANDARD start (castling rights on), 2048-ply cap, finished slots re-seeded.  One STEP = one
pass of the hot path over the batch: for each of the 4096 resident positions, pseudo-legal movegen ->
legal filter -> result -> f32 input planes [24,14,14] -> f32 legal-move mask [120,14,14] -> pick a
move (deterministic splitmix) -> make-move.  Two launches per step: rules_kernel (integer work, board
store in/out, bit sets of the dense outputs) on the main stream and expand_kernel (bit sets -> the
dense f32 tensors, the HBM-bound part) on a second stream, so that the expansion of step t overlaps
the rules of step t+1 (FPC_FLAG_ASYNC_DENSE); the timed region ends after fpc_join + synchronize.

  value  positions/s with the board store resident in HBM (device timed, CUDA events).
  e2e    the same step through the C-ABI host entry point fpc_host_playout_step: boards / game
         ids / plies come from pinned HOST memory every step and go back to it; planes and masks
         stay on the device exactly as the reference's GetEncodedStates(device="cuda") leaves them.

`--impl reference` times the UNMODIFIED reference on the host cores over the same workload: `value` is its
full path (rules engine + GetEncodedStates + legal mask through its own pybind module, oracle/_ref/binding_R14,
one process per core); `engine_only` is its rules engine alone (oracle/_ref/libref_engine_R14.so, C++ threads).
Extra objects on our line: roofline (expand_kernel timed per launch on its stream), rules_only, castling_off (the
reference arm's start record), incremental_dense (resident tensors updated in place -- NOT the headline), perft
(configs[0]), mcts (configs[3] at its stated size at N = 1, configs[4] per GPU at N > 1; fp32 = the reference's precision
beside bf16), dropin (the pybind drop-in through the reference's own MCTS call sequence, beside the reference binding),
cpu_baseline.

Position mix: before anything is timed every slot is fast-forwarded (rules only, untimed) and re-seeded at a staggered
ply, so that the resident games are spread over whole games (opening to 2,048-ply cap) the way SURVEY 8d config 2 asks;
`stats` reports the mix that was timed (legal moves, in-check share, pieces, ply quartiles)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

R = 14
N_GAMES = 4096
MAX_PLIES = 2048
SEED = 0x5EED
DENSE_BYTES_PER_POSITION = 24 * 196 * 4 + 120 * 196 * 4  # f32 planes + mask = 112,896
BYTES_PER_POSITION = 2 * 208 + DENSE_BYTES_PER_POSITION  # 113,312 (SURVEY 8d)
FAST_FORWARD = 2048  # untimed rules-only plies before the timed region (one whole game at the ply cap)
METRIC = "legal positions/sec (movegen+make+encode)"
UNIT = "positions/s"


def workload_config(n_gpus: int) -> dict:
    return {
        "workload": "configs[1] random-playout batched env: 4096 concurrent games/GPU, 14x14 STANDARD start, "
                    "castling on, 2048-ply cap; per position: movegen + legal filter + result + f32 planes "
                    "[24,14,14] + f32 mask [120,14,14] + make",
        "games_per_gpu": N_GAMES, "board": "14x14/3", "max_plies": MAX_PLIES, "seed": SEED,
        "parallelism": f"games sharded over {n_gpus} GPU(s), no data-path collective",
        "l2": "each step writes 464 MB of planes+mask per GPU (> 126 MB L2), so stores drain to HBM; "
              "the 0.85 MB board store is the resident state by design",
        "algorithmic_bytes_per_position": BYTES_PER_POSITION,
        "position_mix": f"slots fast-forwarded {FAST_FORWARD} rules-only plies (untimed) and re-seeded at staggered plies: "
                        "the timed positions span whole games",
    }


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, polled through NVML every 2 ms (nvidia-smi's
    loop mode is too coarse for a 30-40 ms region); falls back to nvidia-smi -lms if NVML is unavailable."""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
               "hw_power_brake_slowdown": 0x80}

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.sm, self.reasons, self.smax = [], 0, None
        self.stop_flag = threading.Event()
        self.armed = threading.Event()
        self.thread = None
        self.poll_once = lambda: None

    def arm(self):
        self.armed.set()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # LOCAL_RANK indexes CUDA devices; honour CUDA_VISIBLE_DEVICES when it lists plain indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.gpu
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                idx = int(vis.split(",")[self.gpu])
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            get_reasons = (getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None)
                           or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons)

            def once():
                try:
                    self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    self.reasons |= int(get_reasons(h))
                except Exception:
                    pass

            self.poll_once = once  # the main thread also samples at fixed points inside the timed region

            def poll():
                # NVML calls take driver locks that a kernel launch on another thread may have to wait for: the thread
                # only polls once the timed region's launches are all enqueued (arm()), while the device works them off
                self.armed.wait()
                while not self.stop_flag.is_set():
                    once()
                    time.sleep(0.002)

            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None

    def stop(self) -> dict:
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvml unavailable"]}
        self.stop_flag.set()
        self.armed.set()
        self.thread.join(timeout=1)
        active = sorted(name for name, bit in self.REASONS.items() if self.reasons & bit)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.smax,
                "samples": len(self.sm), "reasons": active}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def engine_only_rate(seconds: float) -> dict | None:
    """B1 (SURVEY 8d): the unmodified reference RULES ENGINE alone (oracle/_ref/libref_engine_R14.so), one
    C++ thread per host core: GetGameResult + GetPseudoLegalMoves2 + make/IsKingInCheck/undo + MakeMove.
    No tensors are produced, so this is a lower bound on the reference's cost for the path."""
    from alphazero_4_player_chess_b200.fen import start_record
    from oracle import ref_engine
    if not ref_engine.available(R):
        return None
    threads = host_threads()
    eng = ref_engine.RefEngine(R)
    env = ref_engine.RefEnv(eng, start_record("STANDARD", castling=True), N_GAMES, SEED, n_threads=threads,
                            max_plies=MAX_PLIES)
    env.step()
    steps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        env.step()
        steps += 1
    dt = time.perf_counter() - t0
    env.close()
    return {"value": steps * N_GAMES / dt, "unit": UNIT, "cores": threads,
            "sample": f"{steps} steps x {N_GAMES} games, {dt:.1f} s, rules engine only (no planes / mask tensors)"}


def reference_full_path(steps: int, warmup: int, n_games: int) -> dict | None:
    """B2 (SURVEY 8d): the reference's own implementation of the WHOLE path -- engine + GetEncodedStates +
    legal mask -- through its own pybind module, one process per host core (oracle/ref_binding_env.py)."""
    from alphazero_4_player_chess_b200.fen import start_record
    from oracle import ref_binding_env
    if not ref_binding_env.available(R):
        return None
    threads = host_threads()
    # the Python path of the reference builds boards without castling rights (fen_parser.py:137-140,170)
    start = start_record("STANDARD", castling=False)
    initial, plies = whole_game_mix(start, n_games, threads)
    r = ref_binding_env.run(R, start, n_games, steps, warmup, threads, max_plies=MAX_PLIES, seed=SEED,
                            initial=initial, initial_plies=plies)
    return {"value": r["positions_per_s"], "unit": UNIT, "cores": r["procs"], "seconds": r["seconds"],
            "positions": r["positions"], "mix": "whole games" if initial is not None else "from the start position"}


def whole_game_mix(start, n_games: int, threads: int):
    """The same position mix as our arm's fast-forward, for the reference arm: slot i starts about 2048 * i / n plies
    into a random playout (games that end earlier have re-seeded themselves), played by the unmodified reference engine
    (oracle/_ref, all host threads, ~2 s, untimed).  None where the engine library is not built."""
    import numpy as np

    from oracle import ref_engine
    if not ref_engine.available(R):
        return None, None
    env = ref_engine.RefEnv(ref_engine.RefEngine(R), start, n_games, SEED, n_threads=threads, max_plies=MAX_PLIES)
    target = (np.arange(n_games, dtype=np.int64) * FAST_FORWARD) // n_games
    recs = np.zeros((n_games, len(start)), dtype=np.uint8)
    plies = np.zeros(n_games, dtype=np.int64)
    nxt = 0
    for step in range(FAST_FORWARD):
        while nxt < n_games and target[nxt] == step:
            recs[nxt], _, plies[nxt] = env.get(nxt)
            nxt += 1
        env.step()
    while nxt < n_games:
        recs[nxt], _, plies[nxt] = env.get(nxt)
        nxt += 1
    env.close()
    return recs, plies


def run_reference(args) -> None:
    """The reference's own CPU implementation of the path, all host cores: `value` is the full path
    (movegen + legal filter + make + planes + mask through the reference binding, like our arm);
    `engine_only` is its rules engine alone."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # each step = one ply of a bounded sample of the resident games (the full 4,096 would take ~70 ms a step
    # on 16 cores; 1,024 keeps a --steps 400 run within a minute)
    sample_games = 1024
    full = reference_full_path(args.steps, max(args.warmup, 1), sample_games)
    eng = engine_only_rate(6.0)
    if full is None and eng is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built (no /root/reference here)"}))
        return
    kind_note = ("reference pybind module alphazero_cpp (unmodified, oracle/_ref/binding_R14), one process per core: "
                 "GetGameResult + GetLegalMoves + TakeAction per game, GetEncodedStates + legal mask per batch, CPU "
                 "tensors")
    if full is None:
        full = dict(eng)
        kind_note = "rules engine only (binding not built): " + eng["sample"]
    value = full["value"]
    sample = (f"{args.steps} steps x {sample_games} of the {N_GAMES} resident games, castling rights OFF (the reference's "
              "Python API cannot pass rights to Board(): its Player type is unhashable, fen_parser.py drops them; our "
              f"arm reports this start record as `castling_off`), slots spread over whole games like our arm's ({full.get('mix')}); {kind_note}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sample_games / value * 1e3,
        "ms_per_step_note": f"per {sample_games}-game sample step, derived from the rate (one process per core, no common clock)",
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": full["cores"], "kind": "reference", "sample": sample},
        "engine_only": eng,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def cpu_baseline_leg() -> dict:
    """Reported beside our number: the reference's full path on a bounded sample (~15 s), plus its rules
    engine alone; falls back to the single-thread oracle port where oracle/_ref does not exist."""
    from alphazero_4_player_chess_b200.fen import start_record
    threads = host_threads()
    eng = engine_only_rate(5.0)
    full = reference_full_path(steps=300, warmup=3, n_games=1024)
    if full is not None:
        return {"value": full["value"], "unit": UNIT, "cores": full["cores"], "kind": "reference",
                "sample": f"300 plies x 1024 games ({full['positions']} positions, {full['seconds']:.1f} s; slots spread over "
                          f"{full.get('mix')}, castling rights off) through the unmodified reference binding: engine + "
                          "GetEncodedStates + legal mask on CPU tensors, one process per core", "engine_only": eng}
    if eng is not None:
        return {"value": eng["value"], "unit": UNIT, "cores": threads, "kind": "reference", "sample": eng["sample"]}
    from oracle.port import Oracle
    o = Oracle(R, 3)
    t0 = time.perf_counter()
    n, _ = o.bench_playout(start_record("STANDARD", castling=True), SEED, 0, 400000, MAX_PLIES)
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{n} playout positions through oracle/fpc_oracle.c, single thread, {dt:.1f} s"}


def fast_forward(env, start, stride, torch, plies: int = FAST_FORWARD, chunk: int = 64) -> None:
    """Untimed, independent of --warmup: play `plies` rules-only plies and re-seed slot i (fresh game id, start record)
    when `plies * (i / n)` plies are left, so that afterwards slot i is about that many plies into a game: the resident
    games are spread evenly over opening .. ply cap (games that end earlier re-seed themselves as usual)."""
    n = env.n
    left_at_reset = (torch.arange(n, device=env.device, dtype=torch.float64) * (plies / n)).long()
    reset_step = plies - left_at_reset  # slot i is re-seeded right before this step
    start_t = torch.as_tensor(start, dtype=torch.uint8, device=env.device)
    for s0 in range(0, plies, chunk):
        sel = (reset_step >= s0) & (reset_step < s0 + chunk) & (reset_step < plies)
        if bool(sel.any()):
            env.boards[sel] = start_t
            env.ply[sel] = 0
            env.game[sel] += stride
        for _ in range(min(chunk, plies - s0)):
            env.playout_step(seed=SEED, max_plies=MAX_PLIES, game_stride=stride, planes=False, mask=False, k=-1)
    env.counters.zero_()


def mix_stats(env, stride, torch, steps: int = 64) -> dict:
    """The position mix of the resident games, sampled over `steps` untimed rules-only plies after the timed region
    (SURVEY 8d expects about 18.6 legal moves, 3.2 % in check and 17 pieces for whole random playouts)."""
    from alphazero_4_player_chess_b200 import _lib
    nsq = env.R * env.R
    legal = in_check = pieces = 0.0
    ply = env.ply.clone().float()
    for _ in range(steps):
        pieces += float((env.boards[:, :nsq] & 0x80).ne(0).sum()) / env.n
        env.playout_step(seed=SEED, max_plies=MAX_PLIES, game_stride=stride, planes=False, mask=False, k=-1)
        legal += float(env.counts.float().mean())
        in_check += float((env.status & _lib.STATUS_CHECK).ne(0).float().mean())
    q = torch.quantile(ply, torch.tensor([0.0, 0.25, 0.5, 0.75, 1.0], device=ply.device))
    return {"avg_legal_moves": legal / steps, "in_check_share": in_check / steps, "avg_pieces_on_board": pieces / steps,
            "ply_min_q1_median_q3_max": [int(x) for x in q.tolist()], "sampled_plies": steps}


DUMP_SAMPLE_GAMES = 256  # planes + mask of 256 games: 29 MB of the 462 MB a step writes


def snapshot_outputs(env) -> dict:
    """What the timed step hands its caller, copied on the device (no host round trip between timed regions): the board
    records after the move, legal-move counts, status words, game ids and plies of every game, and the f32 planes and
    mask (of the positions before the move) of a fixed, seeded sample of games, whose indices go to sample_games."""
    import numpy as np
    import torch
    rows = np.sort(np.random.default_rng(SEED).choice(env.n, DUMP_SAMPLE_GAMES, replace=False))
    idx = torch.from_numpy(rows).to(env.device)
    return {"boards": env.boards.clone(), "counts": env.counts.clone(), "status": env.status.clone(),
            "game": env.game.clone(), "ply": env.ply.clone(), "planes": env.planes_buffer().index_select(0, idx),
            "mask": env.mask_buffer().index_select(0, idx), "sample_games": idx}


def write_outputs(snapshot: dict, out_dir: str) -> None:
    """snapshot_outputs() as DIR/<name>.npy: float32 for the f32 tensors and the u8 board records, float64 for the
    integers (all exact)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in snapshot.items():
        a = t.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype in (np.float32, np.uint8) else np.float64))


def run_ours(args) -> None:
    import numpy as np
    import torch
    import torch.distributed as dist

    from alphazero_4_player_chess_b200 import _lib
    from alphazero_4_player_chess_b200.env import BatchedEnv
    from alphazero_4_player_chess_b200.fen import start_record

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    L = _lib.lib()
    start = start_record("STANDARD", castling=True)
    from alphazero_4_player_chess_b200.shard import Shard
    shard = Shard(rank, world, N_GAMES)  # games are independent: no data-path collective
    env = BatchedEnv(R, N_GAMES, device=f"cuda:{local}")
    env.reset_playout(start, first_game=shard.first_game)
    stride = shard.game_stride

    # the same C-ABI call as env.playout_step(...), with its arguments resolved once (host overhead per call ~3 us
    # instead of ~30 us: it matters at the head of a short timed region, where the device waits for the first launch)
    step = env.playout_stepper(seed=SEED, max_plies=MAX_PLIES, game_stride=stride, planes=True, mask=True, k=-1,
                               async_dense=True)

    fast_forward(env, start, stride, torch, plies=args.ff)  # untimed: the resident games now span whole games
    for _ in range(max(args.warmup, 3)):
        step()
    env.join()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    env.counters.zero_()
    # ---- timed region A (the headline): K steps, nothing but the product's own launches ---------------------------
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    env.join()  # the main stream waits for the last expansion: every step's tensors are complete
    e1.record()
    if rank == 0:
        # the host runs ahead of the device: the queue is still full, a sample under load -- taken AFTER the closing
        # event is enqueued, so that a slow NVML call cannot stretch a short timed region
        sampler.poll_once()
        sampler.arm()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = e0.elapsed_time(e1)
    positions_a = env.counters.clone()
    # region A's last step, copied on the device here and written to files after the last timed leg
    outputs = snapshot_outputs(env) if args.dump_outputs and rank == 0 else None
    # ---- timed region B (the dominant kernel's launch duration): the same K steps again with CUDA events around
    #      every expand_kernel / rules_kernel launch on the streams they run on (fpc_profile_*).  Kept out of region A
    #      because the instrumentation is not free: four timestamped event records per step drain the internal streams
    #      between launches and lengthen a 74 us step to 79 us (tools/overlap_probe.py FPC_P_NOPROF) ------------------
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _lib.check(L.fpc_profile_enable(1))
    barrier()
    p0.record()
    for _ in range(args.steps):
        step()
    env.join()
    p1.record()
    barrier()
    instrumented_total_ms = p0.elapsed_time(p1)
    instrumented_ms = instrumented_total_ms / args.steps
    plain_total_ms = ms
    # Two trials of exactly K steps each, both bracketed as the contract asks; `value` is the faster one and both are
    # reported (`trials`).  The plain trial wins from ~40 steps up (74 vs 79 us per step: no event records between the
    # launches); for very short regions the instrumented trial is the faster one (at K = 20: ~83 vs ~86-92 us) -- the
    # plain loop pays a start-up cost of ~250 us after the idle barrier that the instrumented loop does not
    # (tools/overlap_probe.py, gpurun_out/xrun20.log), which is not understood yet and is reported rather than hidden.
    # (which trial is the faster one is decided after the max over ranks, below)
    import ctypes
    ex_n, ex_ms, ru_ms = ctypes.c_int(0), ctypes.c_double(0.0), ctypes.c_double(0.0)
    _lib.check(L.fpc_profile_read(ctypes.byref(ex_n), ctypes.byref(ex_ms), ctypes.byref(ru_ms)))
    _lib.check(L.fpc_profile_enable(0))
    env.counters.copy_(positions_a)  # the statistics of the line are those of region A

    # the resident games as the timed region left them (whole-game mix): the e2e leg starts from the same positions
    snap = (env.boards.cpu(), env.game.cpu(), env.ply.cpu())

    # rules only (movegen + legal filter + result + make, no dense tensors): the integer-bound part
    env_counters = env.counters.clone()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rules_step = env.playout_stepper(seed=SEED, max_plies=MAX_PLIES, game_stride=stride, planes=False, mask=False, k=-1)
    barrier()
    r0.record()
    for _ in range(args.steps):
        rules_step()
    r1.record()
    barrier()
    rules_ms = r0.elapsed_time(r1) / args.steps
    # resident dense tensors updated in place (FPC_FLAG_INCREMENTAL): reported separately, never mixed into the
    # headline, which rewrites all 113,312 B per position every step
    env.playout_step(seed=SEED, max_plies=MAX_PLIES, game_stride=stride, planes=True, mask=True, k=-1)  # known content
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    inc_step = env.playout_stepper(seed=SEED, max_plies=MAX_PLIES, game_stride=stride, planes=True, mask=True, k=-1,
                                   incremental=True)
    barrier()
    i0.record()
    for _ in range(args.steps):
        inc_step()
    i1.record()
    barrier()
    inc_ms = i0.elapsed_time(i1) / args.steps
    env.counters.copy_(env_counters)
    mix = mix_stats(env, stride, torch) if rank == 0 else None
    env.counters.copy_(env_counters)
    # the reference arm's start record (castling rights off, as the reference's Python path builds its boards): same
    # step, same game count, a short timed run of its own
    off_ms = None
    if world == 1:
        start_off = start_record("STANDARD", castling=False)
        env.reset_playout(start_off, first_game=shard.first_game)
        fast_forward(env, start_off, stride, torch, plies=args.ff)
        for _ in range(3):
            step()
        env.join()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        c0.record()
        for _ in range(args.steps):
            step()
        env.join()
        c1.record()
        barrier()
        off_ms = c0.elapsed_time(c1) / args.steps
        env.counters.copy_(env_counters)
    t = torch.tensor([plain_total_ms, instrumented_total_ms], dtype=torch.float64, device="cuda")
    counters = env.counters.clone()
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)  # each trial: the slowest rank's time
        dist.all_reduce(counters, op=dist.ReduceOp.SUM)  # NCCL: statistics only
    plain_total_ms, instrumented_total_ms = float(t[0].item()), float(t[1].item())
    instrumented_ms = instrumented_total_ms / args.steps
    value_from = "plain" if plain_total_ms <= instrumented_total_ms else "with_kernel_timing"
    ms_max = min(plain_total_ms, instrumented_total_ms)
    positions = int(counters[0].item())
    assert positions == world * N_GAMES * args.steps, (positions, world, args.steps)
    value = positions / (ms_max * 1e-3)

    # ---- e2e: host buffers through the C-ABI, copies inside the timed region -----------------
    ctx = L.fpc_ctx_create(local, R, N_GAMES)
    if not ctx:
        raise SystemExit(L.fpc_last_error().decode())
    rec = env.geom.record_bytes
    h_boards = snap[0].contiguous().pin_memory()  # the same whole-game position mix as the device-resident loop
    h_game = snap[1].contiguous().pin_memory()
    h_ply = snap[2].contiguous().pin_memory()
    assert h_boards.shape == (N_GAMES, rec)
    h_counts = torch.zeros(N_GAMES, dtype=torch.int32).pin_memory()
    h_status = torch.zeros(N_GAMES, dtype=torch.int32).pin_memory()
    h_start = torch.from_numpy(start.copy()).pin_memory()
    d_planes, d_mask = env.planes_buffer(), env.mask_buffer()

    def e2e_step():
        _lib.check(L.fpc_host_playout_step(ctx, h_boards.data_ptr(), N_GAMES, SEED, h_game.data_ptr(),
                                           h_ply.data_ptr(), h_start.data_ptr(), MAX_PLIES, stride,
                                           h_counts.data_ptr(), h_status.data_ptr(), d_planes.data_ptr(), -1,
                                           d_mask.data_ptr(), _lib.FLAG_ASYNC_DENSE))

    e2e_steps = args.steps
    for _ in range(max(args.warmup, 3)):
        e2e_step()
    _lib.check(L.fpc_ctx_sync(ctx))
    barrier()
    t0 = time.perf_counter()
    legal_seen = 0
    for _ in range(e2e_steps):
        e2e_step()  # returns after the D2H copies of this step's results have landed
        legal_seen += int(h_counts[0])
    _lib.check(L.fpc_ctx_sync(ctx))  # ... and the last step's dense tensors are complete
    dt = time.perf_counter() - t0
    barrier()
    L.fpc_ctx_destroy(ctx)
    t2 = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = world * N_GAMES * e2e_steps / float(t2.item())
    h2d = N_GAMES * (rec + 8 + 4) + rec
    d2h = N_GAMES * (rec + 8 + 4 + 4 + 4)

    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        # dominant kernel: expand_kernel (the dense f32 planes + mask, 112,896 of the 113,312 algorithmic bytes
        # per position), one launch per step, each timed with CUDA events on the stream it runs on while the
        # rules kernel of the next step overlaps it
        per_gpu_ms = ms_max / args.steps
        ex_avg_ms = ex_ms.value / max(ex_n.value, 1)
        achieved = N_GAMES * DENSE_BYTES_PER_POSITION / (ex_avg_ms * 1e-3) / 1e9 if ex_n.value else 0.0
        step_gbs = N_GAMES * BYTES_PER_POSITION / (per_gpu_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "traffic_bytes_per_launch.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("expand_kernel")
                traffic_src = ("static: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture "
                               "(profiles/traffic_bytes_per_launch.json), NOT measured in this run")
            except Exception:
                traffic = None
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "note": "fpc_host_playout_step (same whole-game position mix as `value`): boards/game ids/plies from pinned host memory and back every "
                            "step (the call returns when they have landed); planes+mask are left on the device "
                            "as the reference's device='cuda' does, their expansion overlapping the next step"},
            "gpu_launches": 2 * args.steps,
            "trials": {"plain": {"ms_per_step": plain_total_ms / args.steps, "note": "K steps, nothing but the product's launches"},
                       "with_kernel_timing": {"ms_per_step": instrumented_ms,
                                              "note": "the same K steps with CUDA events around every expand_kernel / "
                                                      "rules_kernel launch (the roofline object's per-launch figure)"},
                       "value_from": value_from,
                       "note": "two trials of exactly K steps each, max over ranks each; value = the faster trial"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src,
                         "kernel": "expand_kernel", "bytes_per_launch": N_GAMES * DENSE_BYTES_PER_POSITION,
                         "avg_launch_ms": ex_avg_ms, "launches_timed": ex_n.value,
                         "timing_note": "CUDA events on the kernel's own stream around every launch of a second timed "
                                        "region of the same K steps (instrumented_ms_per_step): the event records drain "
                                        "the internal streams between launches, so each launch and the step take longer "
                                        "than in the headline region, which runs without them -- `frac` is therefore a "
                                        "lower bound for the kernel and `whole_step` (headline region) can exceed it",
                         "instrumented_ms_per_step": instrumented_ms,
                         "rules_kernel_avg_launch_ms": ru_ms.value / max(ex_n.value, 1),
                         "whole_step": {"bytes": N_GAMES * BYTES_PER_POSITION, "ms": per_gpu_ms, "achieved": step_gbs,
                                        "frac": step_gbs / peak,
                                        "note": "rules_kernel + expand_kernel pipelined; 113,312 B per position over "
                                                "the event-timed step"}},
            "incremental_dense": {"value": N_GAMES / (inc_ms * 1e-3) * world, "unit": UNIT, "ms_per_step": inc_ms,
                                  "note": "NOT the headline: same step and bit-identical f32 planes + mask, but the "
                                          "resident tensors are updated in place (previous ones cleared, new ones set: "
                                          "~120 scattered 4-byte stores per position instead of 112,896 B rewritten); "
                                          "valid only while nothing else writes to the tensors between steps"},
            "rules_only": {"value": N_GAMES / (rules_ms * 1e-3) * world, "unit": UNIT, "ms_per_step": rules_ms,
                           "note": "same step without the dense f32 tensors (movegen + legal filter + result + "
                                   "make); integer/latency bound, 416 B of board traffic per position"},
            "clocks": clocks,
            "stats": {"positions": positions, "finished_games": int(counters[1].item()),
                      "avg_legal_moves": float(counters[6].item()) / max(positions, 1),
                      "move_buffer_overflows": int(counters[7].item()), "position_mix_after_timed_region": mix},
        }
        if off_ms is not None:
            out["castling_off"] = {"value": N_GAMES / (off_ms * 1e-3), "unit": UNIT, "ms_per_step": off_ms,
                                   "note": "the same step from the reference arm's start record (castling rights off, "
                                           "as the reference's Python path builds its boards), same game count"}
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline_leg()
        if world == 1 and not args.no_mcts:
            out["perft"] = perft_leg(local)
        if world == 1 and not args.no_dropin:
            out["dropin"] = dropin_leg()
    # configs[3] / configs[4]: batched PUCT search, every rank on its own shard of games (no cross-GPU traffic in the
    # search; one all_reduce of the per-rank rates for the report)
    mcts = None
    if not args.no_mcts:
        del env
        torch.cuda.empty_cache()
        mcts = mcts_leg(rank, world, local)
        if world > 1:
            keys = [k for k in ("fp32", "fp32_split", "tf32", "bf16") if k in mcts]
            vals = []
            for k in keys:
                vals += [mcts[k]["value"], mcts[k]["tree_kernels_only"]["value"], float(mcts[k]["nodes"])]
            t = torch.tensor(vals, dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.SUM)  # NCCL: per-rank rates summed, statistics only
            for i, k in enumerate(keys):
                mcts[k]["value"], mcts[k]["tree_kernels_only"]["value"] = float(t[3 * i]), float(t[3 * i + 1])
                mcts[k]["nodes"] = int(t[3 * i + 2])
            mcts["games"] = mcts["games_per_gpu"] * world
            mcts["value"] = mcts["fp32"]["value"]
            mcts["note"] = f"sum over {world} ranks, each searching its own {mcts['games_per_gpu']} games"
    if rank == 0:
        if mcts is not None:
            out["mcts"] = mcts
            if world == 1:
                # the N = 1 point of the configs[4] series (8,192 games x 800 simulations per GPU), beside configs[3]
                shard = mcts_leg(rank, world, local, shard_of_configs4=True)
                shard["note"] = ("one GPU's share of configs[4] (8,192 games x 800 simulations): compare with `mcts` of "
                                 "the runs at N = 2, 4, 8, which sum this over the ranks; fp32 is a 100-simulation sample")
                out["mcts_configs4_shard"] = shard
        if outputs is not None:
            write_outputs(outputs, args.dump_outputs)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def mcts_leg(rank: int, world: int, local: int, shard_of_configs4: bool = False) -> dict:
    """M2, batched PUCT self-play search with a random-init ResNet 10 x 128 of the reference architecture in PyTorch.
    N = 1: configs[3] at its stated size, 1,024 games x 400 simulations.  N > 1: configs[4], 8,192 games per GPU x 800
    simulations (bf16 in full; the fp32 line is a 100-simulation sample of the same search: the fp32 network alone
    takes ~0.19 s per 8,192-leaf batch).  fp32 = the reference's precision (src/py/net.py under PyTorch defaults) and
    the headline `value`; bf16 beside it.  One simulation is captured in a CUDA graph and replayed."""
    import torch

    from alphazero_4_player_chess_b200.fen import start_record
    from alphazero_4_player_chess_b200.mcts import BatchedMCTS
    from alphazero_4_player_chess_b200.net import InferenceNet, PolicyValueNet

    # shard_of_configs4 (N = 1 only): one GPU's share of configs[4] -- the N = 1 point of the 1/2/4/8 series
    single = world == 1 and not shard_of_configs4
    n_games = 1024 if single else 8192
    sims_full = 400 if single else 800
    dev = f"cuda:{local}"
    roots = torch.from_numpy(start_record("STANDARD")).unsqueeze(0).repeat(n_games, 1)
    out = {"metric": "MCTS sims/sec", "unit": "sims/s", "games_per_gpu": n_games, "games": n_games,
           "config": ("configs[3]: batched PUCT, 1,024 games x 400 simulations" if single else
                      "configs[4]: sharded self-play, 8,192 games per GPU x 800 simulations (65,536 games on 8 GPUs)") +
                     ", 14x14 STANDARD roots, C=3, random-init ResNet 10x128 (reference architecture incl. the 23,520^2 "
                     "policy Linear) in PyTorch; one simulation = select -> network -> expand/backup, CUDA-graphed"}
    variants = (("fp32", False), ("fp32_split", False), ("tf32", False), ("bf16", True))
    if shard_of_configs4:
        variants = (("fp32", False), ("bf16", True))
    for name, bf16 in variants:
        sims = sims_full if (single or bf16) else (100 if name == "fp32" else 200)
        # "tf32": fp32 weights and activations with TF32 tensor-core matmuls allowed (torch.backends.cuda.matmul.allow_tf32;
        # the convolutions already run TF32 under PyTorch defaults) -- NOT the reference's default, reported beside it
        torch.backends.cuda.matmul.allow_tf32 = name == "tf32"
        torch.manual_seed(0)
        net = InferenceNet(PolicyValueNet(R, 10, 128, device=dev), bf16=bf16, split_policy_linear=name == "fp32_split")
        # arena: ~20 children per expansion from these roots (max seen 19.8 per simulation); 48 leaves a 2.4x margin and
        # the search raises if a tree outgrows it
        m = BatchedMCTS(R, n_games, net, {"C": 3, "num_searches": sims}, device=dev, cuda_graph=True,
                        node_cap=1 + sims_full * 48)
        m.board_cap = m.board_cap  # sims + 2 boards per game: one per simulation plus the root
        m.args["num_searches"] = 6
        m.search(roots)  # warm-up: cuDNN / cuBLAS heuristics, allocator, graph capture
        m.args["num_searches"] = sims
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        m.search(roots, check=False)
        e1.record()
        torch.cuda.synchronize()
        total_ms = e0.elapsed_time(e1)
        m.check_errors()
        nodes, max_nodes = int(m.n_nodes.sum().item()), int(m.n_nodes.max().item())
        # the network alone on the same leaf batch, and the tree kernels alone (fixed network outputs)
        x = m.planes
        for _ in range(2):
            net(x)
        n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10 if single else 4
        n0.record()
        for _ in range(reps):
            net(x)
        n1.record()
        torch.cuda.synchronize()
        net_ms = n0.elapsed_time(n1) / reps
        logits = torch.randn((n_games, m.geom.action_space_size), device=m.device)
        values = torch.zeros(n_games, device=m.device)
        m.reset(roots)
        tree_sims = min(sims, 100)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(tree_sims):
            m.select()
            m.expand_backup(logits, values)
        t1.record()
        torch.cuda.synchronize()
        tree_ms = t0.elapsed_time(t1) / tree_sims
        tree_bytes = sum(getattr(m, a).numel() * getattr(m, a).element_size() for a in
                         ("parent", "first_child", "n_children", "visits", "move_flat", "board_idx", "value_sum", "prior",
                          "boards", "leaf_boards", "leaf_flat", "planes"))
        out[name] = {"value": n_games * sims / (total_ms * 1e-3), "unit": "sims/s", "sims_per_search": sims,
                     "ms_per_sim_batch": total_ms / sims, "network_alone_ms_per_batch": net_ms,
                     "network_share": min(1.0, net_ms / (total_ms / sims)),
                     "tree_kernels_only": {"value": n_games / (tree_ms * 1e-3), "unit": "sims/s", "ms_per_sim_batch": tree_ms},
                     "nodes": nodes, "max_nodes_per_game": max_nodes, "node_cap": m.node_cap,
                     "tree_bytes": tree_bytes,
                     "precision": {"fp32": "fp32 (PyTorch defaults: the reference's; cuDNN convolutions TF32, Linear strict fp32)",
                                   "fp32_split": "fp32 throughout except the 23,520^2 policy Linear, computed as a bf16 x 3 split "
                                                 "product on the tensor cores (six exact bf16 cross terms, tensor-core fp32 accumulation; "
                                                 "1.2e-5 of the logit scale from fp64 where strict fp32 is 6e-7) -- an intermediate "
                                                 "precision beside the strict line, not instead of it",
                                   "tf32": "fp32 storage, TF32 tensor-core math for the Linear layers too (allow_tf32)",
                                   "bf16": "bf16 weights + activations"}[name]}
        if sims != sims_full:
            out[name]["note"] = f"{sims}-simulation sample of the {sims_full}-simulation search"
        m.close()
        del m, net, logits, x
        torch.cuda.empty_cache()
    torch.backends.cuda.matmul.allow_tf32 = False
    out["value"] = out["fp32"]["value"]
    return out


def dropin_leg() -> dict:
    """The pybind drop-in (dropin/alphazero_cpp) through the reference's own per-object MCTS call sequence
    (tests/test_gpu_dropin.py::drive_search = src/py/mcts.py:17-89), 100 games x 50 simulations at 14x14 with the
    deterministic stand-in network, beside the unmodified reference binding (oracle/_ref/binding_R14) on the same box.
    Each in its own process: both modules are called alphazero_cpp."""
    out = {}
    for which in ("ours", "ref"):
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "dropin_probe.py"), which, "100", "50"],
                               capture_output=True, text=True, timeout=600)
            line = [ln for ln in r.stdout.splitlines() if ln.startswith(which + ":")]
            if r.returncode != 0 or not line:
                out[which] = {"unavailable": (r.stderr or r.stdout)[-200:]}
                continue
            out[which] = {"value": float(line[-1].split("=")[1].split()[0]), "unit": "sims/s", "line": line[-1]}  # the median
        except Exception as e:  # pragma: no cover
            out[which] = {"unavailable": repr(e)}
    if "value" in out.get("ours", {}) and "value" in out.get("ref", {}):
        out["ours_over_reference"] = out["ours"]["value"] / out["ref"]["value"]
    out["note"] = ("reference call pattern: per-root ChooseLeaf (GetGameResult), per-state GetLegalMoves, batched "
                   "GetEncodedStates / ExpandNodes; reference = its CPU engine behind the same Python loop")
    return out


def perft_leg(local: int) -> dict:
    """configs[0]: perft from the 14x14 STANDARD start (known answers SURVEY 8c), device vs the unmodified
    reference engine on one host core (its perft is a serial copy-make recursion)."""
    import torch

    from alphazero_4_player_chess_b200.fen import start_record
    from alphazero_4_player_chess_b200.perft import perft
    from oracle import ref_engine
    root = start_record("STANDARD", castling=True)
    want = [20, 395, 7800, 152050, 3450730]
    perft(R, root, 5, device=f"cuda:{local}")  # warm-up at the timed size: the frontier buffers exist afterwards
    torch.cuda.synchronize()
    dt = float("inf")
    for _ in range(3):  # the best of three runs (6-40 ms each: allocator and launch noise dominate one run)
        t0 = time.perf_counter()
        got = perft(R, root, 5, device=f"cuda:{local}")
        torch.cuda.synchronize()
        dt = min(dt, time.perf_counter() - t0)
    out = {"depth": 5, "counts": got, "matches_known_answers": got == want, "seconds": dt,
           "leaves_per_s": got[-1] / dt}
    if ref_engine.available(R):
        eng = ref_engine.RefEngine(R)
        t0 = time.perf_counter()
        n4 = eng.perft(root, 4)
        dt4 = time.perf_counter() - t0
        out["reference_cpu"] = {"depth": 4, "count": n4, "seconds": dt4, "leaves_per_s": n4 / dt4, "cores": 1}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400, help="timed steps per trial")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-mcts", action="store_true")
    ap.add_argument("--no-dropin", action="store_true")
    ap.add_argument("--ff", type=int, default=FAST_FORWARD,
                    help="untimed rules-only plies that spread the resident games over whole games (profiling runs shorten it)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last step of the headline timed region computed as DIR/<name>.npy (rank 0's games; "
                         "planes and mask of a fixed sample of them), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
