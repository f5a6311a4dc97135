"""Cost of the Gumbel root search (BatchedMCTS(gumbel=True)) and of Gumbel MuZero's interior selection
(gumbel_interior=True) with ResNet 10x128 in bf16 (random initial weights) from the 14x14 start, at 1,024 games x
num_searches 16, 32, 64 and 8,192 x 64.

1. The calls, on one tree state: every game searched for num_searches - 1 simulations, then the Gumbel select
   (fpc_tree_select_gumbel: descent + rules kernel + planes), the plain fpc_tree_select on the same state, and
   fpc_tree_gumbel_result, each timed with CUDA events with the GPU held busy (torch.cuda._sleep) while it is enqueued,
   so that the events bracket the device work; median, min and max of --reps.  A repeated select takes the same leaf
   (the only state it changes is the leaf's board, materialised once, and node_value entries rewritten with the same
   value), so the repetitions time the same work.  The interior select (fpc_tree_select_gumbel_interior) is timed the
   same way on a second tree searched with it, as its node_value cache requires.
2. One self-play move, graphed (cuda_graph=True, after one untimed search that warms up and captures): the wall time of
   search() + gumbel_result() at 32 Gumbel simulations, root-only and with the interior rule, the two timed in
   alternation, and search() at 400 PUCT simulations (configs[3]); median of --moves.

Usage: python tools/gumbel_probe.py [--reps 20] [--moves 5] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from alphazero_4_player_chess_b200 import _lib  # noqa: E402
from alphazero_4_player_chess_b200.fen import start_record  # noqa: E402
from alphazero_4_player_chess_b200.mcts import BatchedMCTS  # noqa: E402
from alphazero_4_player_chess_b200.net import InferenceNet, PolicyValueNet  # noqa: E402
from tools.reuse_probe import card, elapsed  # noqa: E402

CALLS = ((1024, 16), (1024, 32), (1024, 64), (8192, 64))


def stats(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "reps": len(xs)}


def roots(n):
    return torch.from_numpy(start_record("STANDARD")).expand(n, -1).contiguous()


def device_us(fn, reps):
    out = []
    for r in range(reps + 3):  # three untimed warm-up calls
        torch.cuda._sleep(2_000_000)  # the GPU is still busy when fn's work is enqueued
        ms, _ = elapsed(fn)
        if r >= 3:
            out.append(ms * 1e3)
    return stats(out)


def searched(net, n, sims, interior=False):
    """A BatchedMCTS whose games were searched for sims - 1 simulations."""
    m = BatchedMCTS(14, n, net, {"C": 3, "num_searches": sims}, gumbel=True, gumbel_seed=1, gumbel_interior=interior)
    m.reset(roots(n))
    m.gumbel_keys.copy_(torch.arange(n, dtype=torch.int64))
    for _ in range(sims - 1):
        m.simulate()
    m.check_errors()
    return m


def calls(net, n, sims, reps):
    m = searched(net, n, sims)

    def plain():
        _lib.check(m.L.fpc_tree_select(C.byref(m.desc), 0, m.planes.data_ptr(), _lib.FLAG_INCREMENTAL, m._track,
                                       m._stream()))

    row = {"games": n, "sims": sims, "root_visits_mean": float(m.visits[:, 0].float().mean()),
           "gumbel_select_us": device_us(m.select, reps), "plain_select_us": device_us(plain, reps),
           "gumbel_result_us": device_us(m.gumbel_result, reps)}
    m.check_errors()
    del m
    mi = searched(net, n, sims, interior=True)
    row["interior_root_visits_mean"] = float(mi.visits[:, 0].float().mean())
    row["interior_select_us"] = device_us(mi.select, reps)
    mi.check_errors()
    return row


def move_ms(net, n, sims, variants, moves):
    """{name: stats} of the graphed move of each variant (name, BatchedMCTS keyword arguments), timed in alternation."""
    r = roots(n)
    runs = {}
    for name, kw in variants:
        m = BatchedMCTS(14, n, net, {"C": 3, "num_searches": sims}, cuda_graph=True, gumbel_seed=1, **kw)

        def one(m=m):
            m.search(r)
            if m.gumbel:
                m.gumbel_result()
            torch.cuda.synchronize()

        one()  # warm-up and capture
        runs[name] = (one, [])
    for _ in range(moves):
        for one, out in runs.values():
            t0 = time.perf_counter()
            one()
            out.append((time.perf_counter() - t0) * 1e3)
    return {name: stats(out) for name, (_, out) in runs.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--moves", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("gumbel_probe needs a GPU")
    info = card()
    print(json.dumps(info), flush=True)
    torch.manual_seed(0)
    net = InferenceNet(PolicyValueNet(14, 10, 128, device="cuda"), bf16=True)
    rows = []
    with torch.no_grad():
        for n, sims in CALLS:
            rows.append(calls(net, n, sims, args.reps))
            print(json.dumps(rows[-1]), flush=True)
            torch.cuda.empty_cache()
        move = {"games": 1024}
        gumbel = move_ms(net, 1024, 32, [("gumbel_32_ms", {"gumbel": True}),
                                         ("gumbel_interior_32_ms", {"gumbel": True, "gumbel_interior": True})],
                         args.moves)
        move.update(gumbel)
        move["interior_over_root_only"] = gumbel["gumbel_interior_32_ms"]["median"] / gumbel["gumbel_32_ms"]["median"]
        torch.cuda.empty_cache()
        move.update(move_ms(net, 1024, 400, [("puct_400_ms", {})], args.moves))
        print(json.dumps(move), flush=True)
    out = {"card": info, "calls": rows, "move": move}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
