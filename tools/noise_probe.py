"""Cost of the Dirichlet root noise (fpc_tree_root_noise through BatchedMCTS.add_root_noise) at 1,024 games x 400
simulations (configs[3]) and 8,192 games x 800 (configs[4] per GPU): every game from the 14x14 start, one batch searched
(ResNet 10x128 in bf16, random initial weights) so that every root is expanded, then the noise call timed with CUDA
events, noise_done cleared (untimed) before each, median of --reps.

Two timings per call: `call_us` has the events around the Python call on an idle GPU (host enqueue included), and
`device_us` has the GPU held busy (torch.cuda._sleep) while the call is enqueued, so the events bracket the kernel.  For
scale, `batch_ms` is the median of --reps eager batches (select -> network -> expand/backup) of the same search; a move
is num_searches of them.  Usage: python tools/noise_probe.py [--reps 20] [--out FILE]"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from alphazero_4_player_chess_b200.fen import start_record  # noqa: E402
from alphazero_4_player_chess_b200.mcts import BatchedMCTS  # noqa: E402
from alphazero_4_player_chess_b200.net import InferenceNet, PolicyValueNet  # noqa: E402
from tools.reuse_probe import card, elapsed  # noqa: E402

SIZES = ((1024, 400), (8192, 800))


def stats(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "reps": len(xs)}


def probe(net, n, sims, reps):
    args = {"C": 3, "num_searches": sims, "dirichlet_alpha": 0.3, "dirichlet_epsilon": 0.25}
    m = BatchedMCTS(14, n, net, args, root_noise=True, noise_seed=1)
    m.reset(torch.from_numpy(start_record("STANDARD")).expand(n, -1).contiguous())
    m.simulate()  # the first batch expands every root
    keys = torch.arange(n, dtype=torch.int64, device="cuda")
    children = m.n_children[:, 0].float()
    call, device = [], []
    for r in range(reps + 3):  # three untimed warm-up calls
        m.noise_done.zero_()
        ms, _ = elapsed(lambda: m.add_root_noise(keys))
        m.noise_done.zero_()
        torch.cuda._sleep(2_000_000)  # the GPU is still busy when the call below is enqueued
        dev_ms, _ = elapsed(lambda: m.add_root_noise(keys))
        if r >= 3:
            call.append(ms * 1e3)
            # _sleep ran before the first event: what the events bracket is the kernel and its launch on the device
            device.append(dev_ms * 1e3)
    assert bool(m.noise_done.all()), "every root should have been noised"
    batches = [elapsed(m.simulate)[0] for _ in range(reps)]
    m.check_errors()
    return {"games": n, "sims": sims, "root_children_mean": float(children.mean()), "call_us": stats(call),
            "device_us": stats(device), "batch_ms": stats(batches),
            "device_call_over_move": float(np.median(device)) * 1e-3 / (float(np.median(batches)) * sims)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("noise_probe needs a GPU")
    info = card()
    print(json.dumps(info), flush=True)
    torch.manual_seed(0)
    net = InferenceNet(PolicyValueNet(14, 10, 128, device="cuda"), bf16=True)
    rows = []
    with torch.no_grad():
        for n, sims in SIZES:
            rows.append(probe(net, n, sims, args.reps))
            print(json.dumps(rows[-1]), flush=True)
    out = {"card": info, "rows": rows}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
