"""-m gpu: the two PUCT kernels on hand-built tree state, one launch at a time.

tree_expand_backup_kernel (through BatchedMCTS.expand_backup) against an f64 restatement of MCTS.step / expand
(src/py/mcts.py:66-89, node.cpp:79-154) written from the reference's Python -- soft-max over the whole row, rot90 by -k,
mask, renormalise, one child per non-zero prior in ascending flat order, backup with alternating sign -- and against the
same f32 pipeline in torch on the device, which gives the expected child set and the yardstick for the priors' precision.
tree_descend_kernel (through BatchedMCTS.select) against oracle/mcts_port.Tree.select_child.

Every slab is filled with sentinels before a launch (a NaN bit pattern in the float arrays, -7777 in the int arrays), so
that a write outside the region the reference says is written shows as a changed word."""
import functools

import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200._lib import FPC_MAX_MOVES
from alphazero_4_player_chess_b200.fen import start_record
from alphazero_4_player_chess_b200.geometry import GEOMETRIES
from alphazero_4_player_chess_b200.mcts import ERR_NO_CHILD, ERR_NODE_CAP, BatchedMCTS
from oracle.mcts_port import Tree
from tests.util import oracle_for

pytestmark = pytest.mark.gpu

START = {8: "EIGHT_SIMPLE", 10: "TEN", 13: "THIRTEEN", 14: "STANDARD"}
SENT_I32 = -7777
SENT_F32 = 0x7FC0DEAD                         # quiet NaN, f32 bits
SENT_F64 = 0x7FF8DEADBEEF0001               # quiet NaN, f64 bits
NODE_I32 = ("parent", "first_child", "n_children", "visits", "move_flat", "board_idx")
STATE = NODE_I32 + ("value_sum", "prior", "n_nodes", "n_boards", "leaf", "dropped", "error", "boards", "leaf_boards",
                    "leaf_flat", "leaf_counts", "leaf_status", "k")
UNDERFLOW = 1e-37  # f64 priors below this sit in f32's underflow band: the child may exist on one side only
C_PUCT = 3.0


def new_tree(R, n, node_cap):
    """A BatchedMCTS whose arrays the test writes by hand (the network is never called)."""
    m = BatchedMCTS(R, n, None, {"C": C_PUCT, "num_searches": 1}, node_cap=node_cap)
    for name in NODE_I32:
        getattr(m, name).fill_(SENT_I32)
    m.value_sum.view(torch.int64).fill_(SENT_F64)
    m.prior.view(torch.int32).fill_(SENT_F32)
    rec = torch.from_numpy(start_record(START[R])).to(m.device)
    m.boards[:] = rec
    m.leaf_boards[:] = rec
    m.n_boards.fill_(1)
    return m


def bits(t):
    """Host copy; floats as their bit patterns so that NaN sentinels compare exactly."""
    if t.dtype == torch.float64:
        t = t.view(torch.int64)
    elif t.dtype == torch.float32:
        t = t.view(torch.int32)
    return t.cpu().numpy().copy()


def snapshot(m):
    torch.cuda.synchronize()
    return {name: bits(getattr(m, name)) for name in STATE}


def put(m, name, array):
    t = getattr(m, name)
    src = torch.from_numpy(np.ascontiguousarray(array))
    if t.dtype == torch.float64:
        t.view(torch.int64).copy_(src.view(torch.int64))
    elif t.dtype == torch.float32:
        t.view(torch.int32).copy_(src.view(torch.int32))
    else:
        t.copy_(src)


def f64_bits(x):
    return np.float64(x).view(np.int64)


def assert_state(got, want, skip=()):
    for name in STATE:
        if name in skip:
            continue
        bad = np.argwhere(got[name] != want[name])
        assert len(bad) == 0, f"{name}: {len(bad)} words differ, first at {bad[:4].tolist()}"


# ---- the f64 reference of MCTS.step after the network + MCTS.expand ------------------------------------------------

@functools.lru_cache(maxsize=None)
def rot_index(R, A, k):
    """rot_index[flat] = the entry of the network's row that lands on `flat` after torch.rot90(., -k, (-2, -1)) over the
    [A, R, R] view (mcts.py:69, board.cpp:257-263)."""
    return np.ascontiguousarray(np.rot90(np.arange(A * R * R).reshape(A, R, R), -k, axes=(1, 2))).reshape(-1)


def reference_f64(row, R, A, k, flats):
    """(unique legal flats ascending, their f64 priors) for one leaf."""
    x = row.astype(np.float64)
    e = np.exp(x - x.max())
    p = (e / e.sum())[rot_index(R, A, k)]
    uniq = np.unique(flats)
    q = p[uniq]
    return uniq, q / q.sum()


def reference_torch_f32(logits, ks, flat_rows, counts, R, A):
    """The reference's own f32 arithmetic on the device: softmax, rot90 by -k, * legal mask, / sum.  [n, A*R*R]."""
    n = logits.shape[0]
    pol = torch.softmax(logits, dim=1).view(n, A, R, R)
    kt = torch.as_tensor(ks, device=logits.device)
    for k in range(4):
        sel = (kt == k).nonzero().view(-1)
        if len(sel):
            pol[sel] = torch.rot90(pol[sel], -k, (-2, -1))
    mask = np.zeros((n, A * R * R), np.float32)
    for g in range(n):
        mask[g, flat_rows[g][: counts[g]]] = 1.0
    pol = pol.view(n, -1) * torch.from_numpy(mask).to(logits.device)
    return (pol / pol.sum(dim=1, keepdim=True)).cpu().numpy()


# ---- cases ------------------------------------------------------------------------------------------------------------

KINDS = [("normal", 0.01), ("normal", 1.0), ("normal", 5.0), ("normal", 20.0), ("offset", 1e4), ("equal", 0.0),
         ("below", 60.0), ("below", 95.0), ("underflow", 120.0), ("neginf_illegal", 0.0), ("neginf_some_legal", 0.0),
         ("soft_mask", -1e30)]
COUNTS = [1, 2, 20, 31, 255, 256, 257, 300]
DEPTHS = [0, 1, 63, 64, 65, 129, 200]
NODE_CAP = 600  # >= the deepest chain + its off-path nodes + 300 children


def legal_layout(rng, R, A, cnt):
    """cnt legal-move entries, ascending, as the rules kernel lists them: the first and last plane, the four corners
    and the centre of a plane among them, and runs of four equal flats (a promotion's four moves share one index), one
    of them over entries 253-256 when there are more than 256."""
    nsq, asz = R * R, A * R * R
    p = int(rng.integers(1, A - 1)) * nsq
    special = [0, nsq - 1, (A - 1) * nsq, asz - 1, p, p + R - 1, p + (R - 1) * R, p + nsq - 1, p + (R // 2) * R + R // 2]
    runs = ([5] if cnt >= 31 else []) + ([253] if cnt >= 257 else [])
    need = cnt - 3 * len(runs)
    special = list(rng.permutation(special))[:need]
    rest = rng.choice(np.setdiff1d(np.arange(asz), special), need - len(special), replace=False)
    entries = []
    for f in np.sort(np.concatenate([special, rest]).astype(np.int64)):
        entries += [f] * (4 if len(entries) in runs else 1)
    assert len(entries) == cnt
    return np.array(entries, dtype=np.int32)


def make_logits(rng, kind, arg, R, A, k, flats):
    """One row in the network's (rotated) frame."""
    asz = A * R * R
    src = rot_index(R, A, k)[np.unique(flats)]  # the row entries the legal moves read
    illegal = np.setdiff1d(np.arange(asz), src)
    row = rng.normal(0.0, 1.0, asz)
    if kind == "normal":
        row = rng.normal(0.0, arg, asz)
    elif kind == "offset":
        row = row + arg
    elif kind == "equal":
        row = np.full(asz, 0.37)
    elif kind in ("below", "underflow"):  # every legal logit at least `arg` below the row's maximum, on an illegal entry
        row[illegal[rng.integers(len(illegal))]] = 10.0
        row[src] = 10.0 - arg - rng.uniform(0.0, 3.0, len(src))
    elif kind == "neginf_illegal":
        row[illegal] = -np.inf
        row[src] = rng.normal(0.0, 2.0, len(src))
    elif kind == "neginf_some_legal":
        row[illegal] = -np.inf
        if len(src) > 1:
            row[src[::3]] = -np.inf
    elif kind == "soft_mask":
        row[illegal] = arg
    return row.astype(np.float32)


def build_chain(rng, depth, n_nodes):
    """Node ids of the path root -> leaf (root = 0, the rest distinct random ids below n_nodes)."""
    return [0] + [int(x) for x in rng.choice(np.arange(1, n_nodes), depth, replace=False)]


def run_expand_case(R, n, seed):
    g = GEOMETRIES[R]
    A, asz = g.num_action_channels, g.action_space_size
    rng = np.random.default_rng(seed)
    m = new_tree(R, n, NODE_CAP)
    ks = np.zeros(n, np.int32)
    status = np.zeros(n, np.int32)
    leaf = np.zeros(n, np.int32)
    counts = np.zeros(n, np.int32)
    flat_rows = rng.integers(-5, asz, (n, FPC_MAX_MOVES)).astype(np.int32)  # entries past the count are stale garbage
    logits = np.zeros((n, asz), np.float32)
    kinds, depths, cap = [], [], [""] * n
    for gi in range(n):
        combo = gi // 4
        ks[gi] = gi % 4
        kind, arg = KINDS[combo % len(KINDS)]
        cnt = COUNTS[(combo // len(KINDS)) % len(COUNTS)]
        if n > 1 and gi % 64 in (17, 49):  # arena exactly full / one node over: a case with an unambiguous child set
            cap[gi] = "full" if gi % 64 == 17 else "over"
            kind, arg = "normal", 1.0
        elif n > 1 and gi % 11 == 3:
            status[gi] = 1 + (gi // 11) % 3  # terminal leaf: WIN_RY, WIN_BG, STALEMATE
        elif n > 1 and gi % 13 == 5:
            leaf[gi] = -1  # no leaf (root dropped): nothing may be written
        if n == 1:
            kind, arg, cnt = "neginf_illegal", 0.0, 300
        kinds.append((kind, arg))
        depths.append(DEPTHS[gi % len(DEPTHS)] if n > 1 else 65)
        counts[gi] = cnt
        flat_rows[gi, :cnt] = legal_layout(rng, R, A, cnt)
        logits[gi] = make_logits(rng, kind, arg, R, A, int(ks[gi]), flat_rows[gi, :cnt])
    values = rng.uniform(-1.0, 1.0, n).astype(np.float32)
    d_logits = torch.from_numpy(logits).cuda()
    t32 = reference_torch_f32(d_logits, ks, flat_rows, counts, R, A)
    torch_children = [np.flatnonzero(t32[gi]) for gi in range(n)]

    # the tree state: an ancestor chain per game plus off-path nodes, all with random contents
    n_nodes = np.zeros(n, np.int32)
    chains = []
    for gi in range(n):
        if cap[gi]:
            n_nodes[gi] = NODE_CAP - len(torch_children[gi]) + (cap[gi] == "over")
        else:
            n_nodes[gi] = depths[gi] + 1 + int(rng.integers(0, 50))
        chain = build_chain(rng, depths[gi], int(n_nodes[gi]))
        chains.append(chain)
        if leaf[gi] == 0:
            leaf[gi] = chain[-1]
    st = snapshot(m)
    for gi in range(n):
        nn = int(n_nodes[gi])
        for name in NODE_I32:
            st[name][gi, :nn] = rng.integers(-1, nn, nn)
        st["visits"][gi, :nn] = rng.integers(1, 1000, nn)
        st["value_sum"][gi, :nn] = rng.normal(0.0, 30.0, nn).view(np.int64)
        st["prior"][gi, :nn] = rng.uniform(0.0, 1.0, nn).astype(np.float32).view(np.int32)
        chain = chains[gi]
        st["parent"][gi, 0] = -1
        for a, b in zip(chain[:-1], chain[1:]):
            st["parent"][gi, b] = a
    st["n_nodes"][:] = n_nodes
    st["leaf"][:] = leaf
    st["leaf_status"][:] = status
    st["leaf_counts"][:] = counts
    st["leaf_flat"][:] = flat_rows
    st["k"][:] = ks
    st["dropped"][:] = 0
    st["error"][:] = np.where(np.arange(n) % 5 == 0, 8, 0)  # bits set before the launch stay set
    for name in STATE:
        put(m, name, st[name])
    before = snapshot(m)
    m.expand_backup(d_logits, torch.from_numpy(values).cuda())
    got = snapshot(m)

    # ---- the expected state ----
    want = {name: before[name].copy() for name in STATE}
    prec = []  # (kind, kernel max rel err vs f64, torch-f32 max rel err vs f64, row spread <= 8)
    n_band = n_nan = 0
    for gi in range(n):
        if leaf[gi] < 0:
            continue
        lf = int(leaf[gi])
        result = status[gi] & 3
        if result:
            v = 0.0 if result == 3 else -1.0
            want["dropped"][gi] = 1
        else:
            v = float(values[gi])
            kind, arg = kinds[gi]
            uniq, r64 = reference_f64(logits[gi], R, A, int(ks[gi]), flat_rows[gi, : counts[gi]])
            n0 = int(before["n_nodes"][gi])
            # every legal soft-max value underflows in f32 (by construction, or at sigma 20 with few legal moves): the
            # reference divides 0 by 0 and so does the kernel -- a child per legal move, NaN priors
            nan_row = bool(np.isnan(t32[gi, uniq]).all())
            assert nan_row == (kind == "underflow") or kind == "normal", (gi, kind)
            n_nan += nan_row
            if nan_row:
                kc = uniq
            else:
                # the kernel's children: those it wrote (capped games were chosen with an unambiguous set)
                nk = int(got["n_children"][gi, lf]) if cap[gi] != "over" else len(torch_children[gi])
                kc = got["move_flat"][gi, n0: n0 + nk] if cap[gi] != "over" else torch_children[gi]
                assert (np.diff(kc) > 0).all(), gi
                tc = torch_children[gi]
                r_of = dict(zip(uniq.tolist(), r64.tolist()))
                diff = np.setxor1d(kc, tc)
                assert all(r_of.get(int(f), 0.0) < UNDERFLOW for f in diff), (gi, kind, arg, diff[:8])
                n_band += len(diff)
                if kind == "neginf_some_legal":
                    lg = logits[gi][rot_index(R, A, int(ks[gi]))]
                    assert not np.isneginf(lg[kc]).any(), gi
            all_ = len(kc)
            if n0 + all_ > NODE_CAP:
                assert cap[gi] == "over"
                want["error"][gi] |= ERR_NODE_CAP
            else:
                assert cap[gi] != "over"
                sl = slice(n0, n0 + all_)
                want["n_nodes"][gi] = n0 + all_
                want["first_child"][gi, lf] = n0
                want["n_children"][gi, lf] = all_
                want["parent"][gi, sl] = lf
                want["first_child"][gi, sl] = 0
                want["n_children"][gi, sl] = 0
                want["visits"][gi, sl] = 1
                want["move_flat"][gi, sl] = kc
                want["board_idx"][gi, sl] = -1
                want["value_sum"][gi, sl] = 0
                kp = got["prior"][gi, sl].view(np.float32)
                if nan_row:
                    assert np.isnan(kp).all(), gi
                else:  # precision over the children both sides made, outside the underflow band
                    use = np.isin(kc, tc) & np.array([r_of[int(f)] >= UNDERFLOW for f in kc])
                    r = np.array([r_of[int(f)] for f in kc[use]])
                    tp = t32[gi, kc[use]].astype(np.float64)
                    ek = float(np.max(np.abs(kp[use] - r) / r))
                    et = float(np.max(np.abs(tp - r) / r))
                    fin = logits[gi][np.isfinite(logits[gi])]
                    narrow = np.isfinite(logits[gi]).all() and float(fin.max() - fin.min()) <= 8.0
                    prec.append((kind, arg, ek, et, narrow))
                    assert ek <= 2.0 * et + 2.0 ** -22, (gi, kind, arg, ek, et)
                    if narrow:
                        assert ek <= 1e-6, (gi, kind, arg, ek)
                    if kind == "equal":
                        assert (kp == np.float32(1.0 / all_)).all(), gi
                want["prior"][gi, sl] = got["prior"][gi, sl]  # checked above
        # Node::Backpropagate: float(np.float32(v)) at the leaf, the sign flipping at every ancestor
        vv = float(np.float32(v))
        for node in reversed(chains[gi]):
            want["value_sum"][gi, node] = f64_bits(before["value_sum"][gi, node].view(np.float64) + vv)
            want["visits"][gi, node] += 1
            vv = -vv
    assert_state(got, want)
    return prec, n_band, n_nan


@pytest.mark.parametrize("R", [8, 10, 13, 14])
def test_expand_backup_against_f64_reference(R):
    prec, n_band, n_nan = run_expand_case(R, 1024, seed=100 + R)
    p1, b1, _ = run_expand_case(R, 1, seed=200 + R)
    prec += p1
    n_band += b1
    lines = []
    for kind, arg in KINDS:
        rows = [(ek, et) for kd, a, ek, et, _ in prec if (kd, a) == (kind, arg)]
        if rows:
            ek, et = np.array(rows).T
            lines.append(f"{kind}({arg:g}): kernel {ek.max():.2e} torch-f32 {et.max():.2e} over {len(rows)} rows")
    print(f"R={R}: priors vs f64, max relative error per kind: " + "; ".join(lines))
    print(f"R={R}: {n_band} moves in the f32 underflow band (f64 prior < {UNDERFLOW:g}) with a child on one side only; "
          f"{n_nan} leaves whose every legal soft-max value underflows (NaN priors on both sides)")


# ---- tree_descend_kernel ----------------------------------------------------------------------------------------------

def put_trees(m, trees, dropped=None):
    """trees: per game dict of lists (parent, first_child, n_children, visits, value_sum, prior).  Every node's board is
    the root's (board_idx 0), so no lazy make runs."""
    st = snapshot(m)
    for gi, t in enumerate(trees):
        nn = len(t["parent"])
        for name in ("parent", "first_child", "n_children", "visits"):
            st[name][gi, :nn] = t[name]
        st["value_sum"][gi, :nn] = np.asarray(t["value_sum"], np.float64).view(np.int64)
        st["prior"][gi, :nn] = np.asarray(t["prior"], np.float32).view(np.int32)
        st["move_flat"][gi, :nn] = -1
        st["board_idx"][gi, :nn] = 0
        st["n_nodes"][gi] = nn
    st["dropped"][:] = 0 if dropped is None else dropped
    st["error"][:] = 0
    st["leaf"][:] = -5
    for name in STATE:
        put(m, name, st[name])
    return snapshot(m)


def oracle_tree(o, rec, t):
    tr = Tree(o, C_PUCT, rec)
    tr.parent = list(t["parent"])
    tr.visits = [int(x) for x in t["visits"]]
    tr.value_sum = [float(x) for x in t["value_sum"]]
    tr.prior = [float(np.float32(x)) for x in t["prior"]]
    tr.children = [list(range(fc, fc + nc)) for fc, nc in zip(t["first_child"], t["n_children"])]
    return tr


def ucb(tr, node, ch):
    n = tr.visits[ch]
    q = tr.value_sum[ch] / n if n > 0 else 0.0
    return q + tr.C * np.sqrt(np.log(np.sqrt(float(tr.visits[node]))) / (1 + n)) * tr.prior[ch]


def random_tree(rng, cap):
    parent, fc, nc, depth = [-1], [0], [0], [0]
    i = 0
    while i < len(parent):
        node = i
        i += 1
        if depth[node] >= 5 or (node and rng.random() < 0.8):
            continue
        k = int(rng.choice([rng.integers(1, 40), rng.integers(30, 70)]))
        if len(parent) + k > cap:
            break
        fc[node], nc[node] = len(parent), k
        parent += [node] * k
        fc += [0] * k
        nc += [0] * k
        depth += [depth[node] + 1] * k
    nn = len(parent)
    visits = np.maximum(rng.integers(0, 60, nn), np.array(nc) > 0)  # an expanded node has been visited
    visits[0] = rng.integers(1, 5000)
    return dict(parent=parent, first_child=fc, n_children=nc, visits=visits,
                value_sum=rng.normal(0.0, 1.0, nn) * visits * 0.4, prior=rng.uniform(0.0, 0.2, nn))


@pytest.mark.parametrize("R", [8, 13, 14])
def test_descend_random_trees_against_oracle(R):
    n, cap = 1024, 1500
    rng = np.random.default_rng(300 + R)
    o = oracle_for(R)
    rec = start_record(START[R])
    m = new_tree(R, n, cap)
    trees = [random_tree(rng, cap) for _ in range(n)]
    dropped = (np.arange(n) % 97 == 13).astype(np.int32)
    before = put_trees(m, trees, dropped)
    m.select()
    got = snapshot(m)
    assert_state(got, before, skip=("leaf", "k", "leaf_boards", "leaf_flat", "leaf_counts", "leaf_status"))
    near_ties = 0
    for gi, t in enumerate(trees):
        if dropped[gi]:
            assert got["leaf"][gi] == -1
            continue
        tr = oracle_tree(o, rec, t)
        path = [int(got["leaf"][gi])]
        while path[-1] > 0:
            path.append(tr.parent[path[-1]])
        path.reverse()
        assert path[0] == 0 and not tr.children[path[-1]], gi
        for node, kernel_choice in zip(path[:-1], path[1:]):
            want = tr.select_child(node)
            if want != kernel_choice:  # only a near-tie (CUDA log / sqrt against glibc's) may go the other way
                a, b = ucb(tr, node, want), ucb(tr, node, kernel_choice)
                assert abs(a - b) <= 8 * np.spacing(max(abs(a), abs(b))), (gi, node, want, kernel_choice, a, b)
                near_ties += 1
                break
    print(f"R={R}: {n} random trees, {int(dropped.sum())} dropped, {near_ties} near-ties resolved the other way")


TIE_NC = [1, 31, 32, 33, 64, 65, 300]


def tie_cases(rng):
    """(n_children, indices of the equal maxima): every single position, pairs in one lane (i, i+32), pairs in
    different lanes (either order of lane and index), triples."""
    out = []
    for nc in TIE_NC:
        out += [(nc, [j]) for j in range(nc)]
        out += [(nc, [i, i + 32]) for i in range(0, nc - 32, 7)]
        if nc > 1:
            for _ in range(12):
                i, j = (int(x) for x in rng.choice(nc, 2, replace=False))
                if i % 32 != j % 32:
                    out.append((nc, [i, j]))
            out += [(nc, [1, 0]), (nc, [nc - 1, nc - 2])]
        if nc > 2:
            out += [(nc, sorted(int(x) for x in rng.choice(nc, 3, replace=False))) for _ in range(6)]
            out.append((nc, [nc - 1, 0, nc // 2]))
    return out


def test_descend_ties_first_maximum_wins():
    R = 14
    rng = np.random.default_rng(5)
    cases = tie_cases(rng)
    n_nan = 8
    n = len(cases) + n_nan
    m = new_tree(R, n, 1 + max(TIE_NC))
    trees = []
    for nc, maxima in cases + [(TIE_NC[gi % len(TIE_NC)], []) for gi in range(n_nan)]:
        prior = np.full(nc, 0.01)
        prior[maxima] = 0.5
        if not maxima:
            prior[:] = np.nan  # no child is selectable
        trees.append(dict(parent=[-1] + [0] * nc, first_child=[1] + [0] * nc, n_children=[nc] + [0] * nc,
                          visits=[10] + [1] * nc, value_sum=[0.0] * (nc + 1), prior=np.concatenate([[0.0], prior])))
    before = put_trees(m, trees)
    m.select()
    got = snapshot(m)
    assert_state(got, before, skip=("leaf", "k", "leaf_boards", "leaf_flat", "leaf_counts", "leaf_status", "dropped",
                                    "error"))
    o = oracle_for(R)
    rec = start_record(START[R])
    for gi, (nc, maxima) in enumerate(cases):
        assert got["leaf"][gi] == 1 + min(maxima) == oracle_tree(o, rec, trees[gi]).select_child(0), (gi, nc, maxima)
    assert (got["error"][: len(cases)] == 0).all() and (got["dropped"][: len(cases)] == 0).all()
    assert (got["error"][len(cases):] == ERR_NO_CHILD).all()
    assert (got["leaf"][len(cases):] == -1).all() and (got["dropped"][len(cases):] == 1).all()
    print(f"{len(cases)} tie cases, {n_nan} all-NaN games")
