"""Leaf-parallel Gumbel search: BatchedMCTS(gumbel=True, gumbel_leaves=L) from the 14x14 start, ResNet 10 x 128 in bf16
(random weights, seed 0), gumbel_considered 16, every search in a CUDA graph.

For each (games, num_searches) the four variants L = 1, 4, 8, 16 are built and warmed up (eager batches, capture,
replays), then timed in alternation, REPS rounds of one search each, CUDA events around every search: wall time per
move as median [min - max].  Per variant: network batches and rows per move, the collision share of the slots, the
root visits a game gains (at most num_searches - L), device time per root visit, and the share of games whose
gumbel_result action equals L = 1's.  Every game starts from the same position with its own Gumbel keys, so the games
differ by their draws; agreement is reported, not judged (the network is untrained).

Then the select kernels' own time at 1,024 games x 32 simulations, from torch.profiler over one eager search each:
gumbel_leaves_descend_kernel (L = 8) against tree_descend_gumbel_kernel (sequential Gumbel) and leaves_descend_kernel
(leaf-parallel PUCT, L = 8), per launch and per root visit.

    python tools/gumbel_leaves_probe.py [--out DIR] [--games 1,16,128,1024] [--sims 32,64] [--leaves 1,4,8,16]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from alphazero_4_player_chess_b200.fen import start_record  # noqa: E402
from alphazero_4_player_chess_b200.mcts import BatchedMCTS  # noqa: E402
from alphazero_4_player_chess_b200.net import InferenceNet, PolicyValueNet  # noqa: E402

R, C_PUCT, CONSIDERED, REPS = 14, 3.0, 16, 7
SELECT_KERNELS = ("gumbel_leaves_descend_kernel", "tree_descend_gumbel_kernel", "leaves_descend_kernel")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the card name from torch is still printed
        q = f"nvidia-smi unavailable ({e})"
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def make(net, n, sims, L, graph=True, **kw):
    return BatchedMCTS(R, n, net, {"C": C_PUCT, "num_searches": sims}, cuda_graph=graph, gumbel=True,
                       gumbel_considered=CONSIDERED, gumbel_leaves=L, **kw)


def timed(m, roots, keys):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    m.search(roots, gumbel_keys=keys)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def pct(xs):
    xs = sorted(xs)
    return round(xs[len(xs) // 2], 3), round(xs[0], 3), round(xs[-1], 3)


def size_rows(net, n, sims, leaves, rec):
    roots = rec.unsqueeze(0).repeat(n, 1)
    keys = torch.arange(n, dtype=torch.int64, device="cuda")
    ms = {L: make(net, n, sims, L) for L in leaves}
    for L, m in ms.items():  # warm-up: eager batches, the capture, replays
        m.search(roots, gumbel_keys=keys)
        m.search(roots, gumbel_keys=keys)
    torch.cuda.synchronize()
    times = {L: [] for L in leaves}
    for _ in range(REPS):  # alternated: every round times each variant once
        for L, m in ms.items():
            times[L].append(timed(m, roots, keys))
    acts = {L: m.gumbel_result()[0].cpu() for L, m in ms.items()}
    rows = []
    for L, m in ms.items():
        m.check_errors()
        med, lo, hi = pct(times[L])
        visits = int((m.visits[:, 0] - 1).sum())  # every backup through the root, its own expansion included
        root_visits = float((m.visits[:, 0] - 2).float().mean())  # the visits its children gained
        row = dict(games=n, sims=sims, L=L, batches=sims // L, rows=n * L * (sims // L),
                   ms_per_move_median=med, ms_min=lo, ms_max=hi,
                   collision_share=round(int(m.collisions.sum()) / (n * sims), 4),
                   root_child_visits_per_game=round(root_visits, 2), leaf_visits=visits,
                   us_per_root_visit=round(med * 1e3 / max(visits, 1), 3),
                   agree_with_L1=round(float((acts[L] == acts[leaves[0]]).float().mean()), 4) if leaves[0] == 1
                   else None)
        print(json.dumps(row), flush=True)
        rows.append(row)
    del ms
    torch.cuda.empty_cache()
    return rows


def kernel_times(net, rec, n=1024, sims=32, L=8):
    from torch.profiler import ProfilerActivity, profile
    roots = rec.unsqueeze(0).repeat(n, 1)
    variants = {"gumbel_leaves L=8": make(net, n, sims, L, graph=False),
                "gumbel L=1": make(net, n, sims, 1, graph=False),
                "leaves_per_game L=8 (PUCT)": BatchedMCTS(R, n, net, {"C": C_PUCT, "num_searches": sims},
                                                          leaves_per_game=L)}
    out = []
    for name, m in variants.items():
        m.search(roots)  # warm-up
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            m.search(roots)
            torch.cuda.synchronize()
        tot, calls = 0.0, 0
        for ev in prof.key_averages():
            if any(k in ev.key for k in SELECT_KERNELS):
                tot += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                calls += ev.count
        visits = int((m.visits[:, 0] - 1).sum())
        row = dict(variant=name, games=n, sims=sims, select_launches=calls,
                   select_us_per_launch=round(tot / max(calls, 1), 1), select_us_per_search=round(tot, 1),
                   select_ns_per_root_visit=round(tot * 1e3 / max(visits, 1), 1))
        print(json.dumps(row), flush=True)
        out.append(row)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for gumbel_leaves_probe.json")
    ap.add_argument("--games", default="1,16,128,1024")
    ap.add_argument("--sims", default="32,64")
    ap.add_argument("--leaves", default="1,4,8,16")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "gumbel_leaves_probe needs a CUDA device"
    info = card()
    print(json.dumps(info), flush=True)
    torch.manual_seed(0)
    net = InferenceNet(PolicyValueNet(R, 10, 128, device="cuda"), bf16=True)
    rec = torch.from_numpy(start_record("STANDARD"))
    leaves = [int(x) for x in a.leaves.split(",")]
    rows = []
    t0 = time.time()
    for sims in (int(x) for x in a.sims.split(",")):
        for n in (int(x) for x in a.games.split(",")):
            rows += size_rows(net, n, sims, leaves, rec)
    kt = kernel_times(net, rec)
    info["after"] = card()["nvidia_smi"]
    print(json.dumps(dict(wall_s=round(time.time() - t0, 1))), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "gumbel_leaves_probe.json"), "w") as f:
            json.dump({"card": info, "settings": dict(R=R, considered=CONSIDERED, reps=REPS, net="ResNet 10x128 bf16",
                                                      start="STANDARD", graph=True),
                       "rows": rows, "select_kernels": kt}, f, indent=1)


if __name__ == "__main__":
    main()
