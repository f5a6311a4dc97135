"""Cost of an Arena match (DESIGN.md §6): PUCT at 400 simulations against Gumbel at 32, one ResNet 10 x 128 in bf16
with random initial weights for both, CUDA graphs, 8 opening plies.

1. STANDARD 14x14, 512 pairs: the wall time of one ply (both searches, the move and the one host read) with the two
   searches on two streams and on one, alternating ply by ply after two warm-up plies (graph capture); median of
   --reps each.  Then the whole match at max_game_length 60 (the instances' graphs already captured).
2. EIGHT_SIMPLE 8x8, 256 pairs, the same pairing played to completion (max_game_length 300), with its summary().

The network is random: the match results say nothing about the strength of either search.
Usage: python tools/arena_probe.py [--reps 5] [--out FILE]"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from alphazero_4_player_chess_b200.arena import Arena, Player  # noqa: E402
from alphazero_4_player_chess_b200.fen import start_record  # noqa: E402
from alphazero_4_player_chess_b200.net import InferenceNet, PolicyValueNet  # noqa: E402
from tools.reuse_probe import card  # noqa: E402


def players(R):
    torch.manual_seed(0)
    net = InferenceNet(PolicyValueNet(R, 10, 128, device="cuda"), bf16=True)
    return (Player(net, {"C": 3, "num_searches": 400}, name="puct400", cuda_graph=True),
            Player(net, {"C": 3, "num_searches": 32}, name="gumbel32", cuda_graph=True, gumbel=True))


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def stats(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "reps": len(xs)}


def standard(reps):
    arena = Arena(14, 512, *players(14), start_record("STANDARD"), opening_plies=8, max_game_length=60)
    two = arena._streams
    out = {"two_streams_ms": [], "one_stream_ms": []}
    with torch.no_grad(), torch.cuda.device(arena.device):
        arena._begin()
        for t in range(2):  # warm-up: eager simulations and graph capture
            arena._ply(t)
        for r in range(2 * reps):
            name = "two_streams_ms" if r % 2 == 0 else "one_stream_ms"
            arena._streams = two if r % 2 == 0 else [None, None]
            ms, running = timed(lambda: arena._ply(2 + r))
            assert running
            out[name].append(ms)
    arena._streams = two
    row = {"board": "STANDARD", "pairs": 512, **{k: stats(v) for k, v in out.items()}}
    row["two_over_one"] = row["two_streams_ms"]["median"] / row["one_stream_ms"]["median"]
    ms, res = timed(arena.play)
    row.update(match_60_plies_s=ms / 1e3, plies=int(res.plies.max()), summary=res.summary())
    return row


def eight_simple():
    arena = Arena(8, 256, *players(8), start_record("EIGHT_SIMPLE"), opening_plies=8, max_game_length=300)
    ms, res = timed(arena.play)
    plies = res.plies.cpu().numpy()
    return {"board": "EIGHT_SIMPLE", "pairs": 256, "match_s": ms / 1e3, "max_plies": int(plies.max()),
            "mean_plies": float(plies.mean()), "summary": res.summary(), "result": res.to_json()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    opt = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("arena_probe needs a GPU")
    out = {"card": card()}
    print(json.dumps(out["card"]), flush=True)
    out["standard"] = standard(opt.reps)
    print(json.dumps(out["standard"]), flush=True)
    torch.cuda.empty_cache()
    out["eight_simple"] = eight_simple()
    print(json.dumps(out["eight_simple"]), flush=True)
    if opt.out:
        os.makedirs(os.path.dirname(os.path.abspath(opt.out)), exist_ok=True)
        with open(opt.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
