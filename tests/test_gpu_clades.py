"""Clade support and the maximum clade credibility score over forests of posterior trees (dphy_clade_table_*) against a plain
set-based counter: a frozenset of tips per node, counts, time sums, scores.  The counter is checked on the CPU against a 4-tip
example worked by hand; the device is compared with it on hand-worked and random forests (repeated topologies, SPR variants of one
tree, independent trees, permuted inner-node numbering), in batches, on never-added trees, after edits, from the wire format, and at
full size against an independent 128-bit key."""
import copy
import math
from collections import Counter, defaultdict

import numpy as np
import pytest

import delphy_b200 as db
from helpers import synth


# ---- reference (host) ---------------------------------------------------------------------------------------------------------------
def clades(emat):
    """frozenset of the tips (child0 == -1) below every node, node included, in host node order"""
    parent, child0, child1 = np.asarray(emat.parent), np.asarray(emat.child0), np.asarray(emat.child1)
    out = [None] * len(parent)
    stack = [(int(emat.root), False)]
    while stack:
        v, done = stack.pop()
        if child0[v] < 0:
            out[v] = frozenset([v])
        elif done:
            out[v] = out[child0[v]] | out[child1[v]]
        else:
            stack += [(v, True), (int(child0[v]), False), (int(child1[v]), False)]
    return out


class RefTable:
    def __init__(self):
        self.count, self.t_sum, self.num_trees = Counter(), defaultdict(float), 0

    def add(self, emats):
        for e in emats:
            for v, c in enumerate(clades(e)):
                self.count[c] += 1
                self.t_sum[c] += float(e.t[v])
            self.num_trees += 1

    def score(self, emat):
        cs = clades(emat)
        if any(self.count[c] == 0 for c in cs):
            return -math.inf
        return math.fsum(math.log(self.count[c] / self.num_trees) for c in cs)

    def node_support(self, emat):
        cs = clades(emat)
        count = np.array([self.count.get(c, 0) for c in cs], np.int64)
        mean_t = np.array([self.t_sum[c] / self.count[c] if self.count.get(c, 0) else math.nan for c in cs])
        return count, mean_t


# ---- trees --------------------------------------------------------------------------------------------------------------------------
def random_topology(rng, labels):
    """nested pairs over tip labels, joined two at a time at random"""
    nodes = list(labels)
    while len(nodes) > 1:
        i, j = sorted(rng.choice(len(nodes), 2, replace=False))
        b, a = nodes.pop(j), nodes.pop(i)
        nodes.append((a, b))
    return nodes[0]


def subtrees(t):
    out, stack = [], [t]
    while stack:
        x = stack.pop()
        out.append(x)
        if isinstance(x, tuple):
            stack += list(x)
    return out


def _remove(t, s):
    if not isinstance(t, tuple):
        return t
    a, b = t
    if a == s:
        return b
    if b == s:
        return a
    return (_remove(a, s), _remove(b, s))


def _insert(t, target, s):
    if t == target:
        return (t, s)
    if not isinstance(t, tuple):
        return t
    return (_insert(t[0], target, s), _insert(t[1], target, s))


def spr(rng, t):
    """prune a random subtree and regraft it on a random branch of the rest"""
    subs = [x for x in subtrees(t) if x != t]
    s = subs[rng.integers(len(subs))]
    rest = _remove(t, s)
    targets = subtrees(rest)
    return _insert(rest, targets[rng.integers(len(targets))], s)


def to_emat(topo, tip_idx, rng, permute_inner=True):
    """Host arrays of a nested-pairs topology: tip label i at host index tip_idx[i], inner nodes at the other indices (in random order
    when permute_inner), children in random order, times growing from 0 at the root."""
    n = len(tip_idx)
    N = 2 * n - 1
    inner = np.setdiff1d(np.arange(N), tip_idx)
    if permute_inner:
        inner = rng.permutation(inner)
    parent, child0, child1, t = np.full(N, -1), np.full(N, -1), np.full(N, -1), np.zeros(N)
    next_inner = iter(inner.tolist())
    root = None
    stack = [(topo, -1)]
    while stack:
        x, p = stack.pop()
        v = int(tip_idx[x]) if not isinstance(x, tuple) else next(next_inner)
        if p < 0:
            root = v
        else:
            parent[v] = p
            t[v] = t[p] + rng.uniform(0.1, 1.0)
            if child0[p] < 0:
                child0[p] = v
            else:
                child1[p] = v
        if isinstance(x, tuple):
            a, b = x if rng.random() < 0.5 else (x[1], x[0])
            stack += [(b, v), (a, v)]
    return bare_emat(root, parent, child0, child1, t)


def bare_emat(root, parent, child0, child1, t):
    """an EMAT without mutations or missing data: clades depend only on topology and times"""
    z = np.zeros(len(parent) + 1, np.int32)
    return db.HostEmat(root, parent=parent, child0=child0, child1=child1, t=t, mut_off=z, mut_site=[], mut_from=[], mut_to=[], mut_t=[],
                       miss_off=z, miss_start=[], miss_end=[], fs_off=z, fs_site=[], fs_from=[])


def tiny_sites(L=8):
    q = np.full((4, 4), 1.0 / 3.0)
    np.fill_diagonal(q, -1.0)
    return db.HostSites(np.zeros(L, np.uint8), np.zeros(L, np.int32), np.ones(L), [1.0], [0.25] * 4, q)


def mixed_forest(rng, n, num_trees=24):
    """one base tree, copies of it (new times and inner numbering), SPR variants of it, independent trees; tips at a fixed random
    subset of host indices"""
    tip_idx = rng.permutation(2 * n - 1)[:n]
    base = random_topology(rng, range(n))
    topos = []
    for k in range(num_trees):
        kind = k % 4
        if kind == 0:
            topos.append(base)
        elif kind in (1, 2):
            t = base
            for _ in range(int(rng.integers(1, 4))):
                t = spr(rng, t)
            topos.append(t)
        else:
            topos.append(random_topology(rng, range(n)))
    return [to_emat(t, tip_idx, rng) for t in topos], tip_idx


# the worked example: tips 0..3, inner nodes 4..6, root 6
def worked_forest():
    t = [3.0, 3.0, 3.0, 3.0, 1.0, 2.0, 0.0]
    a = bare_emat(6, [4, 4, 5, 5, 6, 6, -1], [-1, -1, -1, -1, 0, 2, 4], [-1, -1, -1, -1, 1, 3, 5], t)               # ((0,1),(2,3))
    b = bare_emat(6, [4, 4, 5, 6, 5, 6, -1], [-1, -1, -1, -1, 0, 4, 5], [-1, -1, -1, -1, 1, 2, 3], [3.0, 3.0, 3.0, 3.0, 2.0, 1.0, 0.0])  # (((0,1),2),3)
    c = bare_emat(6, [5, 5, 4, 4, 6, 6, -1], [-1, -1, -1, -1, 2, 0, 4], [-1, -1, -1, -1, 3, 1, 5], [3.0, 3.0, 3.0, 3.0, 1.5, 0.5, 0.0])  # ((0,1),(2,3)), renumbered
    return [a, b, c]


def test_reference_on_worked_example():
    ref = RefTable()
    trees = worked_forest()
    ref.add(trees)
    assert ref.num_trees == 3
    assert ref.count[frozenset({0, 1})] == 3 and ref.count[frozenset({2, 3})] == 2 and ref.count[frozenset({0, 1, 2})] == 1
    assert ref.count[frozenset({0, 1, 2, 3})] == 3 and all(ref.count[frozenset({i})] == 3 for i in range(4))
    assert len(ref.count) == 4 + 1 + 3
    assert ref.score(trees[0]) == math.log(2 / 3) and ref.score(trees[2]) == math.log(2 / 3)
    assert ref.score(trees[1]) == math.log(1 / 3)
    count, mean_t = ref.node_support(trees[1])
    assert count.tolist() == [3, 3, 3, 3, 3, 1, 3]
    assert mean_t[4] == (1.0 + 2.0 + 0.5) / 3 and mean_t[5] == 1.0 and mean_t[6] == 0.0
    # a clade never added: {0, 2}
    d = bare_emat(6, [4, 5, 4, 5, 6, 6, -1], [-1, -1, -1, -1, 0, 1, 4], [-1, -1, -1, -1, 2, 3, 5], [3.0] * 4 + [1.0, 1.0, 0.0])
    assert ref.score(d) == -math.inf
    count, mean_t = ref.node_support(d)
    assert count[4] == 0 and math.isnan(mean_t[4])


# ---- device -------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    with db.Context(0) as c:
        yield c


@pytest.fixture(scope="module")
def sites(ctx):
    s = db.DeviceSites(ctx, tiny_sites())
    yield s
    s.close()


def upload(ctx, sites, emats):
    return db.Forest(ctx, emats, [sites])


def check_against(table, ref, fo, emats, rtol=1e-12):
    assert table.num_trees == ref.num_trees
    got = table.score(fo)
    want = np.array([ref.score(e) for e in emats])
    assert np.array_equal(np.isneginf(got), np.isneginf(want))
    fin = np.isfinite(want)
    assert np.allclose(got[fin], want[fin], rtol=rtol, atol=1e-12)
    for k, e in enumerate(emats):
        c, m = table.node_support(fo, k)
        wc, wm = ref.node_support(e)
        assert np.array_equal(c, wc), k
        assert np.array_equal(np.isnan(m), np.isnan(wm)), k
        ok = ~np.isnan(wm)
        assert np.allclose(m[ok], wm[ok], rtol=rtol, atol=0), k
    return got


@pytest.mark.gpu
def test_worked_forest(ctx, sites):
    trees = worked_forest()
    fo = upload(ctx, sites, trees)
    tab = db.CladeTable(ctx)
    tab.add(fo)
    assert tab.num_trees == 3 and tab.num_clades == 8
    assert tab.device_bytes == 8 * 32 + 4
    s = tab.score(fo)                                                   # one non-zero term per tree: the device log to 1 ulp
    assert np.allclose(s, [math.log(2 / 3), math.log(1 / 3), math.log(2 / 3)], rtol=1e-15, atol=0)
    count, mean_t = tab.node_support(fo, 1)
    assert count.tolist() == [3, 3, 3, 3, 3, 1, 3]
    assert mean_t[4] == (1.0 + 2.0 + 0.5) / 3 and mean_t[5] == 1.0 and mean_t[6] == 0.0 and np.all(mean_t[:4] == 3.0)
    count, _ = tab.node_support(fo, 0)
    assert count.tolist() == [3, 3, 3, 3, 3, 2, 3]
    tab.close(); fo.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n,seed", [(64, 1), (150, 2), (400, 3)])
def test_random_forests(ctx, sites, n, seed):
    rng = np.random.default_rng(seed)
    emats, _ = mixed_forest(rng, n)
    fo = upload(ctx, sites, emats)
    tab = db.CladeTable(ctx)
    tab.add(fo)
    ref = RefTable()
    ref.add(emats)
    assert tab.num_clades == len(ref.count)
    assert tab.device_bytes == 32 * len(ref.count) + 4 * ((2 * n - 1 + 31) // 32)
    got = check_against(tab, ref, fo, emats)
    want = np.array([ref.score(e) for e in emats])
    # the MCC tree: copies of one topology tie up to the order of their terms, so any of the best is right
    assert math.isclose(want[int(np.argmax(got))], want.max(), rel_tol=1e-12)
    assert np.allclose(got[0::4], got[0], rtol=1e-12, atol=1e-12)      # copies of one topology score alike (up to term order)
    tab.close(); fo.close()


@pytest.mark.gpu
def test_batches_give_the_same_counts_and_repeat_bit_for_bit(ctx, sites):
    rng = np.random.default_rng(11)
    emats, _ = mixed_forest(rng, 120, num_trees=30)
    whole = upload(ctx, sites, emats)
    ref = RefTable()
    ref.add(emats)
    results = {}
    for nb in (1, 2, 5):
        runs = []
        for _ in range(2):
            tab = db.CladeTable(ctx)
            for part in np.array_split(np.arange(len(emats)), nb):
                fo = upload(ctx, sites, [emats[k] for k in part])
                tab.add(fo)
                fo.close()                                              # the table keeps no pointer to a forest
            assert tab.num_trees == len(emats) and tab.num_clades == len(ref.count)
            sup = [tab.node_support(whole, k) for k in range(len(emats))]
            runs.append((tab.score(whole), sup))
            tab.close()
        (s0, sup0), (s1, sup1) = runs
        assert s0.tobytes() == s1.tobytes()                             # same adds: bit-identical
        for (c0, m0), (c1, m1) in zip(sup0, sup1):
            assert c0.tobytes() == c1.tobytes() and m0.tobytes() == m1.tobytes()
        results[nb] = runs[0]
    for nb in (2, 5):
        for (c, m), (c1, m1) in zip(results[1][1], results[nb][1]):
            assert np.array_equal(c, c1)
            assert np.allclose(m, m1, rtol=1e-12, atol=0)
        assert np.allclose(results[1][0], results[nb][0], rtol=1e-12, atol=1e-12)
    whole.close()


@pytest.mark.gpu
def test_unseen_clades(ctx, sites):
    rng = np.random.default_rng(5)
    emats, tip_idx = mixed_forest(rng, 80, num_trees=12)
    tab = db.CladeTable(ctx)
    fo = upload(ctx, sites, emats)
    tab.add(fo)
    ref = RefTable()
    ref.add(emats)
    # never added: fresh random trees; and an added tree, which scores finite
    base = emats[0]
    others = [to_emat(random_topology(rng, range(80)), tip_idx, rng) for _ in range(3)]
    other_fo = upload(ctx, sites, others + [base])
    got = check_against(tab, ref, other_fo, others + [base])
    assert np.all(np.isneginf(got[:3])) and np.isfinite(got[3])
    c, m = tab.node_support(other_fo, 0)
    assert np.any(c == 0) and np.all(np.isnan(m[c == 0])) and not np.any(np.isnan(m[c > 0]))
    tab.close(); fo.close(); other_fo.close()


def _nni(emat, rng):
    """swap a child of an inner non-root node u with u's sibling; u takes its parent's time (no branch gets a negative length)"""
    e = copy.deepcopy(emat)
    cand = [v for v in range(e.num_nodes) if e.child0[v] >= 0 and e.parent[v] >= 0]
    u = int(cand[rng.integers(len(cand))])
    p = int(e.parent[u])
    s = int(e.child1[p]) if int(e.child0[p]) == u else int(e.child0[p])
    c = int(e.child0[u])
    if int(e.child0[p]) == s:
        e.child0[p] = c
    else:
        e.child1[p] = c
    e.child0[u] = s
    e.parent[c], e.parent[s] = p, u
    e.t[u] = e.t[p]
    return e, [p, u, c, s]


@pytest.mark.gpu
def test_edits_after_add_leave_the_table_alone(ctx, sites):
    rng = np.random.default_rng(9)
    emats, _ = mixed_forest(rng, 100, num_trees=8)
    fo = upload(ctx, sites, emats)
    tab = db.CladeTable(ctx)
    tab.add(fo)
    before = [tab.node_support(fo, k) for k in range(len(emats))], tab.score(fo), tab.num_clades
    # new times on tree 1: every non-root inner node halfway to its parent
    e1 = emats[1]
    nodes = np.array([v for v in range(e1.num_nodes) if e1.child0[v] >= 0 and e1.parent[v] >= 0], np.int32)
    new_t = 0.5 * (e1.t[nodes] + e1.t[e1.parent[nodes]])
    fo.set_node_times(1, nodes, new_t)
    # a new topology on tree 2
    e2, changed = _nni(emats[2], rng)
    fo.apply_rows([db.node_row(2, e2, v) for v in changed])
    after = [tab.node_support(fo, k) for k in (0, 3)], tab.num_clades, tab.num_trees
    assert after[1] == before[2] and after[2] == len(emats)
    for (c, m), k in zip(after[0], (0, 3)):
        assert c.tobytes() == before[0][k][0].tobytes() and m.tobytes() == before[0][k][1].tobytes()
    # adding the edited forest counts the edits
    e1_new = copy.deepcopy(e1)
    e1_new.t[nodes] = new_t
    edited = [emats[0], e1_new, e2] + emats[3:]
    tab.add(fo)
    ref = RefTable()
    ref.add(emats)
    ref.add(edited)
    assert tab.num_clades == len(ref.count)
    check_against(tab, ref, fo, edited)
    tab.close(); fo.close()


@pytest.mark.gpu
def test_wire_format_forest_counts_alike(ctx, sites):
    rng = np.random.default_rng(21)
    emats, _ = mixed_forest(rng, 90, num_trees=10)
    fo = upload(ctx, sites, emats)
    wire = db.Forest.from_api_trees(ctx, [fo.write_api_tree(k) for k in range(len(emats))], [sites])
    a, b = db.CladeTable(ctx), db.CladeTable(ctx)
    a.add(fo)
    b.add(wire)
    assert a.num_clades == b.num_clades and a.num_trees == b.num_trees
    for k in range(len(emats)):
        assert np.array_equal(a.node_support(fo, k)[0], b.node_support(wire, k)[0])
        assert np.array_equal(a.node_support(wire, k)[0], b.node_support(fo, k)[0])
    a.close(); b.close(); fo.close(); wire.close()


def _independent_keys(emat, tip_key):
    """per node: the sum of random 128-bit per-tip keys (another generator than the library's), mod 2^128 as two uint64 lanes"""
    parent, child0, child1 = emat.parent.tolist(), emat.child0.tolist(), emat.child1.tolist()
    n = len(parent)
    order, stack = [], [int(emat.root)]
    while stack:
        v = stack.pop()
        order.append(v)
        if child0[v] >= 0:
            stack += [child0[v], child1[v]]
    s = [0] * n
    for v in reversed(order):
        s[v] = tip_key[v] if child0[v] < 0 else s[child0[v]] + s[child1[v]]
    m = (1 << 64) - 1
    return np.array([[x & m, (x >> 64) & m] for x in s], np.uint64)


@pytest.mark.gpu
def test_full_size_against_an_independent_key(ctx, sites):
    trees = []
    for k in range(16):
        e = synth(4, seed=1000 + k, muts_per_tip=0.0, missing_mean_intervals_per_tip=0.0, num_sites=100)[0]
        trees.append(bare_emat(e.root, e.parent, e.child0, e.child1, e.t))
    trees += [trees[3], trees[11]]
    n_nodes = trees[0].num_nodes
    assert all(e.num_nodes == n_nodes and np.all(e.child0[:(n_nodes + 1) // 2] < 0) for e in trees)
    rng = np.random.default_rng(77)
    tip_key = [int(a) << 64 | int(b) for a, b in rng.integers(0, 2**64, size=(n_nodes, 2), dtype=np.uint64)]
    keys = np.concatenate([_independent_keys(e, tip_key) for e in trees])
    uniq, inverse, counts = np.unique(keys, axis=0, return_inverse=True, return_counts=True)
    want = counts[inverse.reshape(-1)].reshape(len(trees), n_nodes)
    fo = upload(ctx, sites, trees)
    tab = db.CladeTable(ctx)
    tab.add(fo)
    assert tab.num_trees == 18 and tab.num_clades == len(uniq)
    for k in range(len(trees)):
        c, m = tab.node_support(fo, k)
        assert np.array_equal(c, want[k]), k
        assert not np.any(np.isnan(m))
    s = tab.score(fo)
    assert np.all(np.isfinite(s)) and s[3] == s[16] and s[11] == s[17]
    tab.close(); fo.close()


@pytest.mark.gpu
def test_refusals_leave_the_table_unchanged(ctx, sites):
    trees = worked_forest()
    fo = upload(ctx, sites, trees)
    tab = db.CladeTable(ctx)
    tab.add(fo)
    L = db.lib()
    # a different number of nodes
    rng = np.random.default_rng(3)
    big = upload(ctx, sites, [to_emat(random_topology(rng, range(5)), np.arange(5), rng)])
    # the same number of nodes, tips at other indices (0, 1, 2, 4)
    moved = upload(ctx, sites, [bare_emat(3, [5, 5, 6, -1, 6, 3, 3], [-1, -1, -1, 5, -1, 0, 2], [-1, -1, -1, 6, -1, 1, 4],
                                          [2.0, 2.0, 2.0, 0.0, 2.0, 1.0, 1.0])])
    # and a forest whose second tree is the bad one: nothing of the first may be counted
    mixed = upload(ctx, sites, [trees[0], moved.emats[0]])
    i64p = db.C.POINTER(db.C.c_int64)
    cnt, mean, sc = np.zeros(16, np.int64), np.zeros(16), np.zeros(4)
    for f in (big, moved, mixed):
        for call in (lambda: L.dphy_clade_table_add(ctx._h, tab._h, f._h),
                     lambda: L.dphy_clade_table_score(ctx._h, tab._h, f._h, sc.ctypes.data_as(db.f64p)),
                     lambda: L.dphy_clade_table_node_support(ctx._h, tab._h, f._h, 0, cnt.ctypes.data_as(i64p), mean.ctypes.data_as(db.f64p))):
            assert call() == db.ERR_INVALID_ARGUMENT
            assert tab.num_trees == 3 and tab.num_clades == 8
    out = np.zeros(3)
    assert L.dphy_clade_table_add(None, tab._h, fo._h) == db.ERR_INVALID_ARGUMENT
    assert L.dphy_clade_table_add(ctx._h, None, fo._h) == db.ERR_INVALID_ARGUMENT
    assert L.dphy_clade_table_add(ctx._h, tab._h, None) == db.ERR_INVALID_ARGUMENT
    assert L.dphy_clade_table_score(ctx._h, tab._h, fo._h, None) == db.ERR_INVALID_ARGUMENT
    assert L.dphy_clade_table_score(ctx._h, None, fo._h, out.ctypes.data_as(db.f64p)) == db.ERR_INVALID_ARGUMENT
    assert L.dphy_clade_table_node_support(ctx._h, tab._h, fo._h, 0, None, out.ctypes.data_as(db.f64p)) == db.ERR_INVALID_ARGUMENT
    assert L.dphy_clade_table_node_support(ctx._h, tab._h, fo._h, 3, cnt.ctypes.data_as(i64p), mean.ctypes.data_as(db.f64p)) == db.ERR_INVALID_ARGUMENT
    assert L.dphy_clade_table_create(ctx._h, None) == db.ERR_INVALID_ARGUMENT
    assert L.dphy_clade_table_info(None, None, None, None) == db.ERR_INVALID_ARGUMENT
    assert tab.num_trees == 3 and tab.num_clades == 8
    # an empty table scores nothing
    empty = db.CladeTable(ctx)
    with pytest.raises(db.DphyError) as ei:
        empty.score(fo)
    assert ei.value.status == db.ERR_INVALID_ARGUMENT
    # the refused forests did not fix a tip set on a fresh table either: the first add after a refusal defines it
    fresh = db.CladeTable(ctx)
    assert L.dphy_clade_table_add(ctx._h, fresh._h, mixed._h) == db.ERR_INVALID_ARGUMENT
    assert fresh.num_trees == 0 and fresh.num_clades == 0
    fresh.add(big)
    assert fresh.num_trees == 1 and fresh.num_clades == 9
    for x in (empty, fresh, tab):
        x.close()
    for f in (fo, big, moved, mixed):
        f.close()
