"""Tree reuse at configs[3] size: 1,024 games from the 14x14 start, 400 simulations per move, ResNet 10x128 in bf16, a
CUDA-graphed simulation.  Plays 8 moves of self-play (visit-count sampling at temperature 1) twice -- fresh roots every
move, then BatchedMCTS(reuse_tree=True) with advance() -- and reports per move the search time, the root visits at the
start of the search and the fresh-root fallbacks, and the time of fpc_tree_advance: CUDA events around each advance,
and the same advance repeated on a saved copy of the trees that is restored (untimed) before every launch.

Algorithmic bytes of an advance: the parent index of every node (4 B), the kept nodes read and written (36 B each way)
and the kept boards read and written (208 B each way); the share is of the measured 6,553 GB/s device copy rate
(DESIGN.md §6).  Usage: python tools/reuse_probe.py [--moves 8] [--sims 400] [--games 1024] [--reps 20]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from alphazero_4_player_chess_b200.env import BatchedEnv
from alphazero_4_player_chess_b200.fen import start_record
from alphazero_4_player_chess_b200.mcts import BatchedMCTS
from alphazero_4_player_chess_b200.net import InferenceNet, PolicyValueNet

COPY_PEAK_GBS = 6553.0
TREE = ("parent", "first_child", "n_children", "visits", "move_flat", "board_idx", "value_sum", "prior", "n_nodes",
        "n_boards", "leaf", "dropped", "error", "boards")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers are still printed, without the card's settings
        q = f"nvidia-smi unavailable ({e})"
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q}


def elapsed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def sample(m):
    flat, visits, _, _ = m.root_children()
    w = visits.float()
    has = w.sum(dim=1) > 0
    pick = torch.multinomial(torch.where(has[:, None], w, torch.ones_like(w)), 1)
    return torch.where(has, torch.gather(flat, 1, pick).squeeze(1), torch.full_like(has, -1, dtype=torch.int32))


def advance_bytes(nn_before, kept, nb_after, rec):
    k = kept > 0
    return float((4 * nn_before).sum() + (2 * 36 * kept).sum() + (2 * rec * nb_after[k]).sum())


def play(net, args, reuse, reps):
    n, sims, R = args.games, args.sims, 14
    m = BatchedMCTS(R, n, net, {"C": 3, "num_searches": sims}, cuda_graph=True, reuse_tree=reuse)
    env = BatchedEnv(R, n)
    env.load(start_record("STANDARD"))
    m.args["num_searches"] = 4
    m.search(env.boards)  # warm-up: cuDNN / cuBLAS heuristics, graph capture
    m.args["num_searches"] = sims
    torch.manual_seed(1)
    rec = m.geom.record_bytes
    moves, actions = [], None
    for move in range(args.moves):
        row = {"move": move}
        if reuse and move > 0:
            nn_before = m.n_nodes.clone()
            saved = {a: getattr(m, a).clone() for a in TREE} if move == args.moves // 2 else None
            ms, kept = elapsed(lambda: m.advance(actions, env.boards))
            kept_c, nb = kept.cpu().numpy(), m.n_boards.cpu().numpy()
            nbytes = advance_bytes(nn_before.cpu().numpy(), kept_c, nb, rec)
            row.update(advance_ms=ms, advance_bytes=nbytes, fresh_roots=int((kept_c == 0).sum()),
                       kept_nodes_mean=float(kept_c.mean()), kept_boards_mean=float(nb.mean()))
            if saved is not None:  # repeated on the same trees, restored before every launch (not timed)
                times = []
                for _ in range(reps):
                    for a, t in saved.items():
                        getattr(m, a).copy_(t)
                    times.append(elapsed(lambda: m.advance(actions, env.boards))[0])
                row["advance_repeated_ms"] = {"median": float(np.median(times)), "min": float(np.min(times)),
                                              "max": float(np.max(times)), "reps": reps}
                row["advance_repeated_share_of_copy_peak"] = nbytes / (np.median(times) * 1e-3) / (COPY_PEAK_GBS * 1e9)
            search = lambda: m.search(None, check=False)  # noqa: E731
        else:
            search = lambda: m.search(env.boards, check=False)  # noqa: E731
        if not reuse or move == 0:
            m.reset(env.boards)
        v0 = m.visits[:, 0].float()
        row["root_visits_at_start"] = {"mean": float(v0.mean()), "q10_50_90": [float(x) for x in
                                       torch.quantile(v0, torch.tensor([0.1, 0.5, 0.9], device=v0.device))],
                                       "max": float(v0.max())}
        ms, _ = elapsed(search)
        m.check_errors()
        row["search_ms"] = ms
        actions = sample(m)
        env.make_index(actions)
        moves.append(row)
        print(json.dumps({"reuse": reuse, **row}), flush=True)
    return moves


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--moves", type=int, default=8)
    ap.add_argument("--sims", type=int, default=400)
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("reuse_probe needs a GPU")
    info = card()
    print(json.dumps(info), flush=True)
    torch.manual_seed(0)
    net = InferenceNet(PolicyValueNet(14, 10, 128, device="cuda"), bf16=True)
    with torch.no_grad():
        runs = {name: play(net, args, reuse, args.reps) for name, reuse in (("fresh", False), ("reuse", True))}
    summary = {"card": info, "games": args.games, "sims": args.sims, "moves": args.moves}
    for name, rows in runs.items():
        later = rows[1:]
        summary[name] = {"search_ms_mean_after_move_0": float(np.mean([r["search_ms"] for r in later])),
                         "root_visits_at_start_mean_after_move_0":
                             float(np.mean([r["root_visits_at_start"]["mean"] for r in later]))}
    adv = runs["reuse"][1:]
    summary["reuse"].update(
        advance_ms_in_loop=[r["advance_ms"] for r in adv],
        advance_bytes_mean=float(np.mean([r["advance_bytes"] for r in adv])),
        fresh_root_rate=float(np.sum([r["fresh_roots"] for r in adv]) / (len(adv) * args.games)),
        advance_repeated=next(r["advance_repeated_ms"] for r in adv if "advance_repeated_ms" in r),
        advance_repeated_share_of_copy_peak=next(r["advance_repeated_share_of_copy_peak"] for r in adv
                                                 if "advance_repeated_share_of_copy_peak" in r))
    print(json.dumps({"summary": summary}), flush=True)


if __name__ == "__main__":
    main()
