"""Leaf-parallel PUCT at small game counts: BatchedMCTS(leaves_per_game=L) from the 14x14 start, 256 simulations per
game, ResNet 10 x 128 in bf16 (random weights, seed 0).

For each size (games x L) two runs of one search each:
  - timed: the search with the whole batch (select -> network -> expand/backup) in a CUDA graph, CUDA events around it:
    evaluated leaves per second (root visits gained), slots per second (games x L x batches), the collision rate;
  - split: the same search with the select, the network forward and the expand/backup each captured in a CUDA graph of
    its own and replayed one after the other, CUDA events between them: the tree time and the network time per batch
    without host launch gaps (each includes one graph launch, a few microseconds).
The most-visited root move of every game is compared with the L = 1 search of the same game count (same network):
reported, not a pass / fail test.  Every game of a size starts from the same position, so within a size the games
differ only by the rounding of their rows in the batch: the agreement is close to 0 or 1, not a rate over positions.

Then the cost of the commit kernel's serial backup (taken when a batch's leaf paths hold more than 4,096 nodes in all):
one game, root -> a chain of D single children -> a node with one child per legal move of the start position, L = 64
slots, so about 20 leaf slots with paths of D + 2 nodes.  D = 190 stays under the limit (sorted backup), D = 210 goes
over (serial backup); the expand/backup call is timed with CUDA events, the tree restored before every repetition.

    python tools/leaves_probe.py [--out DIR] [--sizes 1x1,1x16,...]"""
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

SIZES = "1x1,1x16,1x64,1x256,16x1,16x16,16x64,128x1,128x8,1024x1"
R, SIMS, C_PUCT = 14, 256, 3.0


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the card name from torch is still printed
        q = f"nvidia-smi unavailable ({e})"
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q}


class GraphedNet:
    """The network forward on a static input tensor, captured once in a CUDA graph."""

    def __init__(self, net, planes):
        self.planes = planes
        for _ in range(3):
            net(planes)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.logits, self.value = net(planes)

    def __call__(self, planes):
        assert planes.data_ptr() == self.planes.data_ptr()
        self.graph.replay()
        return self.logits, self.value


def timed_search(net, n, L, roots):
    m = BatchedMCTS(R, n, net, {"C": C_PUCT, "num_searches": SIMS}, cuda_graph=True, leaves_per_game=L)
    m.search(roots)  # warm-up: eager batches, capture, replays
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    m.search(roots)
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) / 1e3
    leaves = int((m.visits[:, 0] - 1).sum())
    coll = int(m.collisions.sum())
    flat, visits, _, _ = m.root_children()
    best = torch.gather(flat, 1, visits.argmax(dim=1, keepdim=True)).squeeze(1).cpu()
    return m, sec, leaves, coll, best


def capture(fn):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g  # capturing runs nothing


def split_search(net, n, L, roots):
    m = BatchedMCTS(R, n, None, {"C": C_PUCT, "num_searches": SIMS}, leaves_per_game=L)
    m.reset(roots)
    planes = m.select()  # the first select writes the planes in full
    m.expand_backup(*net(planes))  # cuDNN / cuBLAS pick their kernels
    torch.cuda.synchronize()
    g_net = GraphedNet(net, planes)
    g_sel = capture(m.select)
    g_exp = capture(lambda: m.expand_backup(g_net.logits, g_net.value))
    batches = SIMS // L
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(batches)]
    m.reset(roots)
    torch.cuda.synchronize()
    for b in range(batches):
        e = ev[b]
        e[0].record()
        g_sel.replay()
        e[1].record()
        g_net.graph.replay()
        e[2].record()
        g_exp.replay()
        e[3].record()
    torch.cuda.synchronize()
    m.check_errors()
    tree = sum(e[0].elapsed_time(e[1]) + e[2].elapsed_time(e[3]) for e in ev) / batches
    netms = sum(e[1].elapsed_time(e[2]) for e in ev) / batches
    return tree * 1e3, netms * 1e3


def fallback_cost(reps=20):
    L, out = 64, {}
    for depth in (190, 210):
        m = BatchedMCTS(R, 1, None, {"C": C_PUCT, "num_searches": L}, node_cap=8192, leaves_per_game=L)
        one = BatchedMCTS(R, 1, None, {"C": C_PUCT, "num_searches": 1})
        one.reset(torch.from_numpy(start_record("STANDARD"))[None])
        one.select()
        A = one.geom.action_space_size
        one.expand_backup(torch.zeros((1, A), device="cuda"), torch.zeros(1, device="cuda"))
        k = int(one.n_children[0, 0])
        flats, priors = one.move_flat[0, 1:1 + k].clone(), one.prior[0, 1:1 + k].clone()
        m.reset(torch.from_numpy(start_record("STANDARD"))[None])
        d, nn = depth, depth + 1 + k
        ar = torch.arange(nn, device="cuda", dtype=torch.int32)
        m.parent[0, :nn] = torch.where(ar <= d, ar - 1, torch.full_like(ar, d))
        m.first_child[0, :nn] = torch.where(ar <= d, ar + 1, torch.zeros_like(ar))
        m.n_children[0, :nn] = torch.where(ar < d, 1, torch.where(ar == d, k, 0)).int()
        m.visits[0, :nn] = torch.where(ar <= d, 50, 1).int()
        m.value_sum[0, :nn] = 0.0
        m.prior[0, :nn] = 0.5
        m.prior[0, d + 1:nn] = priors
        m.move_flat[0, :nn] = -1
        m.move_flat[0, d + 1:nn] = flats
        m.board_idx[0, :nn] = torch.where(ar <= d, 0, -1).int()  # the chain shares the root's board
        m.n_nodes[0] = nn
        saved = {name: getattr(m, name).clone() for name in ("parent", "first_child", "n_children", "visits",
                                                              "value_sum", "prior", "move_flat", "board_idx",
                                                              "n_nodes", "n_boards", "dropped", "error")}
        logits = torch.zeros((L, A), device="cuda")
        values = torch.zeros(L, device="cuda")
        times = []
        for _ in range(reps + 2):
            for name, t in saved.items():
                getattr(m, name).copy_(t)
            m.select()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            m.expand_backup(logits, values)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) * 1e3)
        m.check_errors()
        leaves = int(m.visits[0, 0]) - 50
        times = sorted(times[2:])
        out[depth] = dict(depth=depth, leaf_slots=leaves, backup_entries=leaves * (depth + 2),
                          path="serial" if leaves * (depth + 2) > 4096 else "sorted",
                          expand_backup_us_median=round(times[len(times) // 2], 1),
                          expand_backup_us_min=round(times[0], 1))
        print(json.dumps(out[depth]), flush=True)
    return list(out.values())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for leaves_probe.json")
    ap.add_argument("--sizes", default=SIZES)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "leaves_probe needs a CUDA device"
    info = card()
    print(json.dumps(info), flush=True)
    torch.manual_seed(0)
    net = InferenceNet(PolicyValueNet(R, 10, 128, device="cuda"), bf16=True)
    rec = torch.from_numpy(start_record("STANDARD"))
    sizes = [tuple(int(x) for x in s.split("x")) for s in a.sizes.split(",")]
    rows, ref = [], {}
    for n, L in sorted(sizes, key=lambda s: (s[0], s[1])):
        roots = rec.unsqueeze(0).repeat(n, 1)
        t0 = time.time()
        m, sec, leaves, coll, best = timed_search(net, n, L, roots)
        del m
        tree_us, net_us = split_search(net, n, L, roots)
        if L == 1:
            ref[n] = best
        slots = n * SIMS
        row = dict(games=n, L=L, batch_rows=n * L, batches=SIMS // L, seconds=round(sec, 4),
                   leaves_per_s=round(leaves / sec), slots_per_s=round(slots / sec),
                   collision_rate=round(coll / slots, 4), tree_us_per_batch=round(tree_us, 1),
                   net_us_per_batch=round(net_us, 1),
                   agree_with_L1=None if n not in ref else round(float((best == ref[n]).float().mean()), 4),
                   wall_s=round(time.time() - t0, 1))
        rows.append(row)
        print(json.dumps(row), flush=True)
    fb = fallback_cost()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "leaves_probe.json"), "w") as f:
            json.dump({"card": info, "settings": dict(R=R, sims=SIMS, net="ResNet 10x128 bf16", start="STANDARD"),
                       "rows": rows, "backup_fallback": fb}, f, indent=1)


if __name__ == "__main__":
    main()
