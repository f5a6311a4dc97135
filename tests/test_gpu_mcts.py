"""-m gpu: the batched PUCT kernels (fpc_tree_* through the C-ABI) against (1) the golden fixtures
produced by the reference's own MCTS.search and (2) the MCTS restatement oracle, node by node.

Integer state (tree shape, moves, visit counts) and the double value sums must be bit-exact.  Priors are
f32 softmax outputs: the kernel's fused softmax -> un-rotate -> mask -> renormalise differs from torch's
op-by-op f32 arithmetic by rounding only; tolerance rtol 2e-6."""
import os

import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200._lib import FPC_MAX_MOVES, FpcError
from alphazero_4_player_chess_b200.fen import start_record
from alphazero_4_player_chess_b200.geometry import GEOMETRIES
from alphazero_4_player_chess_b200.mcts import BatchedMCTS
from oracle.mcts_port import search as oracle_search
from tests.golden.fake_net import FakeNet
from tests.util import mixed_positions, oracle_for

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PRIOR_RTOL = 2e-6


def run_gpu(R, roots, sims, batch_rotation, C=3):
    net = FakeNet(R, device="cuda")
    m = BatchedMCTS(R, len(roots), net, {"C": C, "num_searches": sims}, batch_rotation=batch_rotation)
    m.search(torch.from_numpy(np.ascontiguousarray(roots)))
    torch.cuda.synchronize()
    m.check_errors()
    return m


@pytest.mark.parametrize("R", [8, 14])
@pytest.mark.parametrize("case", ["a", "b"])
def test_against_reference_mcts_fixtures(R, case):
    z = np.load(os.path.join(GOLDEN, f"mcts_R{R}.npz"))
    roots = z[f"{case}_roots"]
    m = run_gpu(R, roots, int(z[f"{case}_sims"]), batch_rotation=True)
    flat, visits, _, cnt = (t.cpu().numpy() for t in m.root_children())
    off = z[f"{case}_child_off"]
    for g in range(len(roots)):
        n = off[g + 1] - off[g]
        assert cnt[g] == n
        assert flat[g, :n].tolist() == z[f"{case}_child_flat"][off[g]: off[g + 1]].tolist(), g
        assert visits[g, :n].tolist() == z[f"{case}_child_visits"][off[g]: off[g + 1]].tolist(), g
    assert m.visits[:, 0].cpu().numpy().tolist() == z[f"{case}_root_visits"].tolist()
    assert m.n_nodes.cpu().numpy().tolist() == z[f"{case}_n_nodes"].tolist()


def search_roots(name, R, n_games):
    o = oracle_for(R)
    pool = mixed_positions(name, 600)
    # late positions: short games at 8x8 put terminal leaves (root dropping) inside the search horizon
    roots = np.ascontiguousarray(pool[len(pool) // 3:: max(1, len(pool) // (2 * n_games))][:n_games])
    return np.stack([r for r in roots if o.game_result(r)[0] == 0])


@pytest.mark.parametrize("name,R,n_games,sims", [("STANDARD", 14, 24, 48), ("EIGHT_SIMPLE", 8, 32, 80), ("TEN", 10, 16, 40),
                                                 ("THIRTEEN", 13, 16, 40)])
@pytest.mark.parametrize("batch_rotation", [True, False])
def test_whole_trees_match_the_oracle(name, R, n_games, sims, batch_rotation):
    o = oracle_for(R)
    roots = search_roots(name, R, n_games)
    trees = oracle_search(o, FakeNet(R), roots, 3, sims, batch_rotation=batch_rotation)
    m = run_gpu(R, roots, sims, batch_rotation)
    assert_trees_equal(m, trees)
    print(f"{name} rot={batch_rotation}: {len(trees)} games, {int(m.n_nodes.sum())} nodes, {int(m.dropped.sum())} dropped roots")


def assert_trees_equal(m, trees):
    n_nodes = m.n_nodes.cpu().numpy()
    parent, move_flat, visits = m.parent.cpu().numpy(), m.move_flat.cpu().numpy(), m.visits.cpu().numpy()
    value_sum, prior = m.value_sum.cpu().numpy(), m.prior.cpu().numpy()
    first_child, n_children = m.first_child.cpu().numpy(), m.n_children.cpu().numpy()
    for gi, t in enumerate(trees):
        nn = len(t.parent)
        assert n_nodes[gi] == nn, gi
        assert parent[gi, :nn].tolist() == t.parent
        assert move_flat[gi, :nn].tolist() == t.move_flat
        assert visits[gi, :nn].tolist() == t.visits
        assert value_sum[gi, :nn].tolist() == t.value_sum  # doubles, bit-exact
        np.testing.assert_allclose(prior[gi, :nn], np.array(t.prior), rtol=PRIOR_RTOL, atol=0)
        for node in range(nn):
            ch = t.children[node]
            assert n_children[gi, node] == len(ch)
            if ch:
                assert first_child[gi, node] == ch[0] and ch == list(range(ch[0], ch[0] + len(ch)))


class SharpMaskedNet(FakeNet):
    """FakeNet with logits x 8 (spread 64, so legal priors range down to e^-64) and -inf on every entry whose index is
    below 4 modulo 128 and on the eight planes no move reaches (8(R-1)+8 and up).  The first pattern covers the first
    16-value group lane 0 of every warp of tree_expand_backup_kernel streams, which is where a running maximum that
    starts at -inf turns into NaN.  At x16 the spread (128) would pass the f32 exponential's normal range (~87): priors
    then go through denormal intermediates, whose absolute precision no relative tolerance between two f32 pipelines
    can follow."""

    def __call__(self, encoded):
        logits, value = super().__call__(encoded)
        logits = logits * 8.0
        logits[:, (torch.arange(self.ASZ, device=logits.device) % 128) < 4] = -float("inf")
        logits[:, 8 * self.R * self.R * self.R:] = -float("inf")
        return logits, value


@pytest.mark.parametrize("batch_rotation", [True, False])
def test_sharp_masked_network_trees_match_the_oracle(batch_rotation):
    """A policy with -inf entries and a wide logit spread (before the soft-max started its running maximum at -FLT_MAX,
    every child got a NaN prior here and the next descent stopped the search with error bit 4)."""
    R, sims = 14, 48
    o = oracle_for(R)
    roots = search_roots("STANDARD", R, 24)
    trees = oracle_search(o, SharpMaskedNet(R), roots, 3, sims, batch_rotation=batch_rotation)
    for t in trees:  # every expanded leaf kept an unmasked legal move: finite priors that sum to 1
        for node, ch in enumerate(t.children):
            if ch:
                pr = np.array([t.prior[c] for c in ch])
                assert len(ch) <= FPC_MAX_MOVES and np.isfinite(pr).all() and abs(pr.sum() - 1.0) < 1e-5, node
    net = SharpMaskedNet(R, device="cuda")
    m = BatchedMCTS(R, len(roots), net, {"C": 3, "num_searches": sims}, batch_rotation=batch_rotation)
    m.search(torch.from_numpy(roots))
    torch.cuda.synchronize()
    assert_trees_equal(m, trees)
    print(f"sharp masked rot={batch_rotation}: {len(trees)} games, {int(m.n_nodes.sum())} nodes")


def test_fully_underflowing_policy_stops_the_search():
    """Every legal logit 200 below the row's maximum (which sits on a plane no move reaches): the soft-max underflows to 0
    on every legal move and the renormalisation divides 0 by 0, in the reference's f32 pipeline as in the kernel.  The
    leaf gets its children with NaN priors, the next descent can select none of them, and the search raises instead of
    returning a tree."""
    R = 8
    g = GEOMETRIES[R]

    def net(planes):
        logits = torch.zeros((planes.shape[0], g.action_space_size), device=planes.device)
        logits[:, -1] = 200.0
        return logits, torch.zeros((planes.shape[0], 1), device=planes.device)

    roots = np.stack([start_record("EIGHT_SIMPLE")] * 3)
    m = BatchedMCTS(R, 3, net, {"C": 3, "num_searches": 3})
    with pytest.raises(FpcError, match="tree error bits 0x4"):
        m.search(torch.from_numpy(roots))
    flat, _, prior, cnt = m.root_children()
    n_legal = len(set(oracle_for(R).move_flat_index(mv) for mv in oracle_for(R).legal_moves(roots[0])))
    assert cnt.tolist() == [n_legal] * 3
    assert torch.isnan(prior[:, :n_legal]).all()
    assert (m.error == 4).all() and (m.leaf == -1).all() and (m.dropped == 1).all()


def test_batch_rotation_ignores_terminal_leaves():
    """The reference encodes a leaf batch with the colour of states[0], and states holds only the leaves that are
    NOT terminal (mcts.py:18-26).  Game 0 here stands two plies before the end of a decisive game, so its selected
    leaf is terminal in many simulations while the games behind it (other sides to move) are not: the batch
    rotation must come from the first expandable leaf."""
    from alphazero_4_player_chess_b200.fen import start_record
    from tests.util import SEED
    R = 8
    o = oracle_for(R)
    start = start_record("EIGHT_SIMPLE")
    near_end, others = [], []
    for game in range(60):
        p = o.playout(start, SEED, game, 200)
        if p["result"][-1] in (1, 2) and p["n"] > 6:
            near_end.append(p["recs"][p["n"] - 3])
        others.append(p["recs"][min(5 + game % 3, p["n"] - 1)])
    assert near_end
    others = [r for r in others if o.game_result(r)[0] == 0 and r[R * R] != near_end[0][R * R]][:6]
    roots = np.stack([near_end[0]] + others + near_end[1:3])
    sims = 60
    trees = oracle_search(o, FakeNet(R), roots, 3, sims, batch_rotation=True)
    m = run_gpu(R, roots, sims, batch_rotation=True)
    assert int(m.dropped[0].item()) == 1 or any(v > 1 for v in trees[0].visits[1:])
    n_nodes = m.n_nodes.cpu().numpy()
    visits, value_sum, move_flat = m.visits.cpu().numpy(), m.value_sum.cpu().numpy(), m.move_flat.cpu().numpy()
    for gi, t in enumerate(trees):
        nn = len(t.parent)
        assert n_nodes[gi] == nn, gi
        assert move_flat[gi, :nn].tolist() == t.move_flat
        assert visits[gi, :nn].tolist() == t.visits
        assert value_sum[gi, :nn].tolist() == t.value_sum
    assert int(m.dropped.sum().item()) >= 1  # a root did reach a terminal leaf


def test_promotion_moves_collapse_into_one_child():
    """SURVEY 0.4: the four promotion moves share one (plane, from) index, so they become ONE child, made with an
    index-built move that does not promote.  Hand-made 14x14 position: a red pawn one step from its promotion row."""
    R = 14
    g = GEOMETRIES[R]
    o = oracle_for(R)
    rec = g.empty_record()
    def put(r, c, color, ptype):
        rec[r * R + c] = 0x80 | (color << 5) | (ptype << 2)
        if ptype == 5:
            rec[g.off_king + color] = r * R + c
    put(13, 7, 0, 5), put(7, 0, 1, 5), put(0, 6, 2, 5), put(6, 13, 3, 5)   # kings
    put(R // 4 + 1, 5, 0, 0)                                                # red pawn, promotion row is R/4
    put(R // 4, 6, 1, 3)                                                    # a blue rook it can capture with promotion
    legal = o.legal_moves(rec)
    promos = [m for m in legal if ((int(m) >> 24) & 0xff) != 6]
    assert len(promos) == 8  # push and capture, four promotion pieces each
    roots = np.stack([rec] * 3)
    trees = oracle_search(o, FakeNet(R), roots, 3, 20, batch_rotation=False)
    m = run_gpu(R, roots, 20, batch_rotation=False)
    flat, visits, prior, cnt = (t.cpu().numpy() for t in m.root_children())
    n_distinct = len(set(o.move_flat_index(mv) for mv in legal))
    assert n_distinct == len(legal) - 6
    for gi, t in enumerate(trees):
        ch = t.children[0]
        assert cnt[gi] == len(ch) == n_distinct
        assert flat[gi, : len(ch)].tolist() == [t.move_flat[c] for c in ch]
        assert visits[gi, : len(ch)].tolist() == [t.visits[c] for c in ch]
    # the child reached through the promotion index still holds a PAWN on the promotion row (index-built make)
    push = o.move_flat_index(promos[0])
    child = o.make_index(rec, push)
    assert (child[(R // 4) * R + 5] >> 2) & 7 == 0


def test_action_probs_and_capacity_errors():
    R = 8
    roots = np.stack([start_record("EIGHT_SIMPLE")] * 4)
    m = run_gpu(R, roots, 30, batch_rotation=False)
    probs = m.action_probs()
    flat, visits, _, cnt = m.root_children()
    assert torch.allclose(probs.sum(dim=1), torch.ones(4, device="cuda"))
    g0 = probs[0].cpu().numpy()
    n = int(cnt[0])
    want = visits[0, :n].float().cpu().numpy()
    assert np.allclose(g0[flat[0, :n].cpu().numpy()], want / want.sum())
    # a node arena that is too small is reported, not overrun
    small = BatchedMCTS(R, 4, FakeNet(R, device="cuda"), {"C": 3, "num_searches": 30}, node_cap=40)
    small.search(torch.from_numpy(roots), check=False)
    torch.cuda.synchronize()
    assert int(small.error.max().item()) & 1
    assert int(small.n_nodes.max().item()) <= 40


def test_cuda_graph_search_equals_eager_search():
    """One simulation captured in a CUDA graph and replayed gives the same trees as the eager loop."""
    R, sims = 14, 40
    roots = torch.from_numpy(np.ascontiguousarray(mixed_positions("STANDARD", 64)))
    trees = []
    for graph in (False, True):
        m = BatchedMCTS(R, 64, FakeNet(R, device="cuda"), {"C": 3, "num_searches": sims}, cuda_graph=graph)
        m.search(roots)
        m.search(roots)  # the second search replays the captured graph from its first simulation on
        torch.cuda.synchronize()
        trees.append(m)
    a, b = trees
    assert b._graph is not None
    assert torch.equal(a.n_nodes, b.n_nodes)
    nn = int(a.n_nodes.max())
    used = torch.arange(nn, device="cuda")[None, :] < a.n_nodes[:, None]  # the slabs are uninitialised past n_nodes
    for name in ("parent", "move_flat", "visits", "value_sum", "prior", "first_child", "n_children"):
        assert torch.equal(getattr(a, name)[:, :nn][used], getattr(b, name)[:, :nn][used]), name


def test_configs3_search_replayed_on_the_oracle():
    """BASELINE.json configs[3] at its stated size and the reference's precision: 1,024 games x 400 simulations with the
    random-init ResNet 10 x 128 in fp32 (PyTorch defaults, as src/py/net.py runs).  The network outputs of a sample of
    games are recorded and the same games are replayed on the CPU restatement of fpchess::Node / MCTS.search
    (oracle/mcts_port.py) with those outputs: tree shapes, moves, visit counts and value sums must be identical
    (SURVEY 8d: record / replay so that float noise of the network does not leak into the comparison)."""
    from alphazero_4_player_chess_b200.fen import start_record
    from alphazero_4_player_chess_b200.net import InferenceNet, PolicyValueNet
    R, n, sims = 14, 1024, 400
    o = oracle_for(R)
    torch.manual_seed(0)
    net = InferenceNet(PolicyValueNet(R, 10, 128, device="cuda"), bf16=False)
    pool = mixed_positions("STANDARD", 256)
    roots = np.ascontiguousarray(np.concatenate([pool] * (n // len(pool)))[:n])
    roots[::2] = start_record("STANDARD")  # half of the games search from the start position
    sample = torch.tensor([0, 1, 2, 3, 101, 255, 256, 511, 640, 777, 901, 1023], device="cuda")
    rec_logits, rec_values = [], []

    def record(sim, logits, value):
        rec_logits.append(logits[sample].cpu())
        rec_values.append(value[sample].reshape(-1, 1).cpu())

    m = BatchedMCTS(R, n, net, {"C": 3, "num_searches": sims})
    m.search(torch.from_numpy(roots), record=record)
    torch.cuda.synchronize()
    assert int(m.visits[:, 0].min()) >= 1 and int((m.visits[:, 0] == sims + 1).sum()) > n // 2
    idx = sample.cpu().numpy()
    pos = {int(g): i for i, g in enumerate(idx)}

    def replay(sim, games):
        rows = [pos[int(idx[g])] for g in games]
        return rec_logits[sim][rows], rec_values[sim][rows]

    prior = m.prior[sample].cpu().numpy()
    trees = oracle_search(o, None, roots[idx], 3, sims, batch_rotation=False, replay=replay, prior_source=prior)
    n_nodes, visits = m.n_nodes[sample].cpu().numpy(), m.visits[sample].cpu().numpy()
    move_flat, value_sum, parent = m.move_flat[sample].cpu().numpy(), m.value_sum[sample].cpu().numpy(), m.parent[sample].cpu().numpy()
    for i, t in enumerate(trees):
        nn = len(t.parent)
        assert n_nodes[i] == nn, (i, n_nodes[i], nn)
        assert parent[i, :nn].tolist() == t.parent
        assert move_flat[i, :nn].tolist() == t.move_flat
        assert visits[i, :nn].tolist() == t.visits  # the visit-count vectors, every node
        assert value_sum[i, :nn].tolist() == t.value_sum
    print(f"configs[3]: {n} games x {sims} sims, {int(m.n_nodes.sum())} nodes; {len(trees)} games replayed on the oracle, "
          f"{sum(len(t.parent) for t in trees)} nodes identical")


def test_inference_net_equals_the_module_it_wraps():
    """InferenceNet (BatchNorm folded, fused cuDNN conv+bias+ReLU(+residual), permuted head weights) against the plain
    eval-mode module.  fp32 = the reference's precision = PyTorch defaults, under which cuDNN convolutions use TF32 on both
    sides (torch.backends.cudnn.allow_tf32 is True by default, matmuls stay fp32): 3e-3 of the logit magnitude; with TF32
    off on both sides 2e-5; bf16 within 6e-2."""
    from alphazero_4_player_chess_b200.net import InferenceNet, PolicyValueNet
    torch.manual_seed(1)
    R = 14
    m = PolicyValueNet(R, 3, 32, device="cuda")
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.running_mean.normal_()
            mod.running_var.uniform_(0.5, 2.0)
            mod.weight.data.uniform_(0.5, 1.5)
            mod.bias.data.normal_()
    m.eval()
    x = (torch.rand(64, 24, R, R, device="cuda") < 0.05).float()
    with torch.no_grad():
        l0, v0 = m(x)
    def check(tol, bf16, want_l, want_v):
        for fused in (True, False):
            inf = InferenceNet(m, bf16=bf16, fused=fused)
            l1, v1 = inf(x)
            assert l1.dtype == torch.float32 and l1.shape == want_l.shape and v1.shape == want_v.shape
            assert float((l1 - want_l).abs().max()) < tol * max(1.0, float(want_l.abs().max())), (bf16, fused)
            assert float((v1 - want_v).abs().max()) < tol, (bf16, fused)

    check(3e-3, False, l0, v0)
    check(6e-2, True, l0, v0)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            l2, v2 = m(x)
        check(2e-5, False, l2, v2)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    assert next(m.parameters()).dtype == torch.float32  # the wrapped module is left as it was


def test_split_policy_linear_matches_strict_fp32():
    """InferenceNet(split_policy_linear=True): the policy Linear as a bf16 x 3 split product on the tensor cores against
    the strict-fp32 Linear of the same wrapper, and all variants against an fp64 Linear on the same activations: the
    split product sits between strict fp32 and TF32 (the ladder is printed and asserted below)."""
    from alphazero_4_player_chess_b200.net import InferenceNet, PolicyValueNet
    torch.manual_seed(2)
    R = 14
    m = PolicyValueNet(R, 2, 32, device="cuda").eval()
    x = (torch.rand(128, 24, R, R, device="cuda") < 0.05).float()
    strict = InferenceNet(m, bf16=False)
    split = InferenceNet(m, bf16=False, split_policy_linear=True)
    l0, v0 = strict(x)
    l1, v1 = split(x)
    scale = max(1.0, float(l0.abs().max()))
    err = float((l1 - l0).abs().max())
    # fp64 reference of the policy Linear on the same (fp32, TF32-convolved) activations
    n = x.shape[0]
    xx = x.contiguous(memory_format=torch.channels_last)
    xx = strict._conv_relu(xx, strict.stem)
    for a, b in strict.tower:
        xx = strict._conv_add_relu(strict._conv_relu(xx, a), b, xx)
    p = strict._conv_relu(xx, strict.p_conv).permute(0, 2, 3, 1).reshape(n, -1)
    l64 = (p.double() @ strict.p_lin[0].double().t() + strict.p_lin[1].double())
    e_strict = float((l0.double() - l64).abs().max())
    e_split = float((l1.double() - l64).abs().max())
    lb, _ = InferenceNet(m, bf16=True)(x)
    e_bf16 = float((lb.double() - l64).abs().max())
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        lt, _ = InferenceNet(m, bf16=False)(x)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = False
    e_tf32 = float((lt.double() - l64).abs().max())
    print(f"policy Linear vs fp64: strict fp32 {e_strict:.2e}, bf16x3 split {e_split:.2e}, tf32 {e_tf32:.2e}, bf16 {e_bf16:.2e} "
          f"(logit scale {scale:.2f})")
    # measured on B200: strict 6e-7, split 1.2e-5 (the tensor cores' fp32 accumulation over K = 3 x 23,520 is not IEEE
    # round-to-nearest), tf32 and bf16 orders of magnitude above: the split sits between strict fp32 and TF32
    assert err < 4e-5 * scale, (err, scale)
    assert e_strict < 5e-6 * scale
    assert e_split < 4e-5 * scale and e_split < e_bf16 / 20, (e_split, e_tf32, e_bf16)
    assert torch.equal(v0, v1)
