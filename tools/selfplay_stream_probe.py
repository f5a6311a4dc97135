"""Continuous self-play against lock-step rounds (DESIGN.md §6): `SelfPlay.play_games(k * n)` on n slots against k rounds
of `SelfPlay.play()` on the same n slots, timed in alternation within one run.  ResNet 10 x 128 in bf16 with random
initial weights, eager search (SelfPlay drives select / expand without CUDA graphs), temperature 1.

Per board (EIGHT_SIMPLE 8x8, where games end; STANDARD 14x14) and per method: replay entries per second (wall time
around the call, ended by a device synchronise), slot occupancy (live slot-plies over all slot-plies the network
evaluated: the entries over n times the plies searched), and the game-length quantiles.  Then the sampler kernel
(`fpc_tree_sample_root` via `BatchedMCTS.sample_root`) on a searched tree: CUDA events around the call, median of 50.
The card's name and power limit are read in the same run.

The network is random: game lengths say nothing about trained play.
Usage: python tools/selfplay_stream_probe.py [--slots 256] [--rounds 2] [--reps 3] [--out FILE]"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from alphazero_4_player_chess_b200.fen import start_record  # noqa: E402
from alphazero_4_player_chess_b200.net import InferenceNet, PolicyValueNet  # noqa: E402
from alphazero_4_player_chess_b200.selfplay import SelfPlay  # noqa: E402
from tools.reuse_probe import card  # noqa: E402

BOARDS = {"EIGHT_SIMPLE": (8, 300), "STANDARD": (14, 100)}  # board -> (R, max_game_length)
SIMS = 32


def quantiles(plies):
    q = np.quantile(np.asarray(plies), [0.1, 0.5, 0.9])
    return {"p10": float(q[0]), "p50": float(q[1]), "p90": float(q[2]), "max": int(np.max(plies))}


class Counted:
    """The SelfPlay with its per-ply search counted (one _search call per ply, for both methods)."""

    def __init__(self, sp):
        self.sp, self.plies = sp, 0
        search = sp._search

        def counted(*a, **kw):
            self.plies += 1
            return search(*a, **kw)

        sp._search = counted


def run_rounds(c, rounds):
    sp, entries, lengths = c.sp, 0, []
    for _ in range(rounds):
        out = sp.play()
        entries += out["boards"].shape[0]
        lengths += sp.hist_valid.sum(dim=0).tolist()
    return entries, lengths


def run_stream(c, games):
    out = c.sp.play_games(games)
    return out["boards"].shape[0], out["plies"].tolist()


def board(name, n, rounds, reps):
    R, T = BOARDS[name]
    torch.manual_seed(0)
    net = InferenceNet(PolicyValueNet(R, 10, 128, device="cuda"), bf16=True)
    args = {"C": 3, "num_searches": SIMS, "temperature": 1.0, "max_game_length": T, "heuristic_weight": 0.02}
    sp = SelfPlay(R, n, net, args, start_record(name))
    c = Counted(sp)
    with torch.no_grad():
        sp.play_games(n)  # warm-up: the network's kernels and the library's modules
    acc = {m: {"s": 0.0, "entries": 0, "plies": 0, "lengths": []} for m in ("rounds", "stream")}
    for r in range(2 * reps):
        method = "rounds" if r % 2 == 0 else "stream"
        c.plies = 0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        entries, lengths = run_rounds(c, rounds) if method == "rounds" else run_stream(c, rounds * n)
        torch.cuda.synchronize()
        a = acc[method]
        a["s"] += time.perf_counter() - t0
        a["entries"] += entries
        a["plies"] += c.plies
        a["lengths"] += lengths
        print(json.dumps({"board": name, "rep": r // 2, "method": method, "s": time.perf_counter() - t0,
                          "entries": entries, "plies_searched": c.plies}), flush=True)
    row = {"board": name, "R": R, "slots": n, "games_per_rep": rounds * n, "reps": reps, "num_searches": SIMS,
           "max_game_length": T}
    for method, a in acc.items():
        row[method] = {"entries_per_s": a["entries"] / a["s"], "occupancy": a["entries"] / (n * a["plies"]),
                       "entries": a["entries"], "plies_searched": a["plies"], "s": a["s"],
                       "game_length": quantiles(a["lengths"]),
                       "cut_off_share": float(np.mean(np.asarray(a["lengths"]) >= T))}
    row["stream_over_rounds"] = row["stream"]["entries_per_s"] / row["rounds"]["entries_per_s"]
    # the sampler kernel on the tree the last search left
    keys = torch.arange(n, dtype=torch.int64, device="cuda") * T
    times = []
    for _ in range(60):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sp.mcts.dropped.zero_()
        e0.record()
        sp.mcts.sample_root(1, keys, 1.0)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) * 1e3)
    row["sample_root_us"] = {"median": float(np.median(times[10:])), "min": float(np.min(times[10:])),
                             "max": float(np.max(times[10:])), "games": n}
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--slots", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--boards", default="EIGHT_SIMPLE,STANDARD")
    ap.add_argument("--out", default=None)
    opt = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("selfplay_stream_probe needs a GPU")
    out = {"card": card()}
    print(json.dumps(out["card"]), flush=True)
    for name in opt.boards.split(","):
        out[name] = board(name, opt.slots, opt.rounds, opt.reps)
        print(json.dumps(out[name]), flush=True)
        torch.cuda.empty_cache()
    out["card_after"] = card()
    if opt.out:
        os.makedirs(os.path.dirname(os.path.abspath(opt.out)), exist_ok=True)
        with open(opt.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
