"""The exponential-growth coalescent log-prior of device-resident trees (dphy_forest_log_coalescent_prior) against a float64 numpy
reference: one forest and batches of trees of different sizes; g = 0, tiny and large g; isochronous and heavily tied dates; a 2-tip tree
worked by hand; a tree grown by grafting samples where dphy_forest_place_samples puts them.  The references are checked on the CPU
first: the plain sorted-event loop against a branch-crossing count with the closed form of the integral, tie order, the 2-tip value."""
import math

import numpy as np
import pytest

import delphy_b200 as db
from helpers import synth

RTOL = 1e-10


# ---- references (float64, host) ---------------------------------------------------------------------------------------------------
def ref_log_prior(emat, n0, g, t0, tie_rng=None):
    """Walk the events in ascending time: an inner node (coalescence) adds a lineage above it going forward in time, a tip takes one
    away; k lineages on (a, b) contribute -C(k, 2) * integral_a^b dt / N(t), each coalescence -log N(t_c).  Ties are taken in index
    order, or in a random order drawn from tie_rng."""
    t = np.asarray(emat.t, np.float64)
    tip = np.asarray(emat.child0) < 0
    tie_key = tie_rng.random(len(t)) if tie_rng is not None else np.arange(len(t))
    order = np.lexsort((tie_key, t))
    k, total = 1, 0.0
    for j, v in enumerate(order):
        a = float(t[v])
        if tip[v]:
            k -= 1
        else:
            k += 1
            total -= math.log(n0) + g * (a - t0)
        if j + 1 < len(order) and k >= 2:
            b = float(t[order[j + 1]])
            if b > a:
                d = b - a
                w = d if g * d == 0.0 else -math.expm1(-g * d) / g
                total -= k * (k - 1) / 2 * math.exp(-g * (a - t0)) / n0 * w
    return total


def crossing_log_prior(emat, n0, g, t0):
    """The same density by another route: k on each interval between distinct event times is the number of branches spanning it, and
    the integral is the closed form C(k,2)/(n0 g) (exp(-g (a - t0)) - exp(-g (b - t0))) (g != 0) or C(k,2) (b - a) / n0."""
    t = np.asarray(emat.t, np.float64)
    parent = np.asarray(emat.parent)
    inner = np.asarray(emat.child0) >= 0
    nr = parent >= 0
    top, bottom = t[parent[nr]], t[nr]
    total = float(-np.sum(np.log(n0) + g * (t[inner] - t0)))
    times = np.unique(t)
    for a, b in zip(times[:-1], times[1:]):
        m = 0.5 * (a + b)
        k = int(np.count_nonzero((top < m) & (bottom > m)))
        integral = (b - a) / n0 if g == 0 else (math.exp(-g * (a - t0)) - math.exp(-g * (b - t0))) / (n0 * g)
        total -= k * (k - 1) / 2 * integral
    return total


def two_tip_tree(t_root, t_a, t_b):
    z = np.zeros(4, np.int32)
    return db.HostEmat(2, parent=[2, 2, -1], child0=[-1, -1, 0], child1=[-1, -1, 1], t=[t_a, t_b, t_root], mut_off=z, mut_site=[],
                       mut_from=[], mut_to=[], mut_t=[], miss_off=z, miss_start=[], miss_end=[], fs_off=z, fs_site=[], fs_from=[])


def two_tip_by_hand(n0, g, t0):
    """Root at 0, tips at 1 and 2: one coalescence at 0, two lineages on (0, 1), one on (1, 2)."""
    integral = 1.0 / n0 if g == 0 else math.exp(g * t0) * -math.expm1(-g) / (n0 * g)
    return -(math.log(n0) - g * t0) - integral


def with_times(emat, t):
    e = db.HostEmat(emat.root, emat.includes_run_root, **{k: getattr(emat, k) for k in db.HostEmat.FIELDS_I32 + db.HostEmat.FIELDS_U8 +
                                                           db.HostEmat.FIELDS_F64})
    e.t = np.ascontiguousarray(t, np.float64)
    return e


def isochronous(emat):
    """every tip moved to the latest tip date (later than before: no branch gets a negative length)"""
    tip = emat.child0 < 0
    t = emat.t.copy()
    t[tip] = t[tip].max()
    return with_times(emat, t)


def tied(emat, step):
    """tip dates rounded up to a grid of `step`, some inner nodes right above two tips of the same date moved onto it as well
    (mutation times are left alone: only node times enter the prior)"""
    t = emat.t.copy()
    tip = emat.child0 < 0
    t[tip] = np.ceil(t[tip] / step) * step
    for v in np.nonzero(~tip)[0]:
        c0, c1 = int(emat.child0[v]), int(emat.child1[v])
        if tip[c0] and tip[c1] and t[c0] == t[c1] and v % 3 == 0:
            t[v] = t[c0]                    # zero-length branches: a coalescence tied with its two samples
    return with_times(emat, t)


PARAMS = [(3.0, 0.0, 0.0), (3.0, 1e-12, 0.0), (3.0, -1e-12, 0.0), (0.7, 25.0, 0.0), (2.0, 4.0, -0.3), (5.0, -2.0, -0.5)]


# ---- the references themselves (CPU) -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n0,g,t0", [(1.0, 0.0, 0.0), (2.5, 0.8, 1.5), (0.3, -1.7, -2.0), (4.0, 1e-12, 0.5)])
def test_reference_two_tips_by_hand(n0, g, t0):
    e = two_tip_tree(0.0, 1.0, 2.0)
    assert math.isclose(ref_log_prior(e, n0, g, t0), two_tip_by_hand(n0, g, t0), rel_tol=1e-13)


@pytest.mark.parametrize("n0,g,t0", [p for p in PARAMS if abs(p[1]) == 0 or abs(p[1]) > 1e-6])
def test_reference_matches_branch_crossing_count(n0, g, t0):
    emat, _, _ = synth(0, num_tips=120, num_sites=200)
    for e in (emat, isochronous(emat), tied(emat, 0.05)):
        assert math.isclose(ref_log_prior(e, n0, g, t0), crossing_log_prior(e, n0, g, t0), rel_tol=1e-11)


def test_reference_tie_order_does_not_matter():
    emat, _, _ = synth(0, num_tips=150, num_sites=200)
    e = tied(emat, 0.1)
    want = ref_log_prior(e, 2.0, 3.0, 0.0)
    for seed in range(4):
        assert math.isclose(ref_log_prior(e, 2.0, 3.0, 0.0, np.random.default_rng(seed)), want, rel_tol=1e-13)


def test_reference_tiny_growth_is_constant_population():
    emat, _, _ = synth(0, num_tips=100, num_sites=200)
    base = ref_log_prior(emat, 3.0, 0.0, 0.0)
    for g in (1e-12, -1e-12):
        assert math.isclose(ref_log_prior(emat, 3.0, g, 0.0), base, rel_tol=1e-9)


# ---- device ----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    c = db.Context(0)
    yield c
    c.close()


class Resident:
    """trees uploaded as one forest, one sites table per tree"""

    def __init__(self, ctx, emats, sites):
        self.tables = [db.DeviceSites(ctx, s) for s in sites]
        self.forest = db.Forest(ctx, emats, self.tables, sites_index=np.arange(len(emats)))

    def close(self):
        self.forest.close()
        for t in self.tables:
            t.close()


def check_forest(ctx, emats, sites, params=PARAMS):
    r = Resident(ctx, emats, sites)
    try:
        for n0, g, t0 in params:
            got = r.forest.log_coalescent_prior(n0, g, t0)
            assert got.shape == (len(emats),) and got.dtype == np.float64
            want = np.array([ref_log_prior(e, n0, g, t0) for e in emats])
            np.testing.assert_allclose(got, want, rtol=RTOL, atol=0, err_msg=f"n0={n0} g={g} t0={t0}")
        return r.forest.log_coalescent_prior(*params[0])
    finally:
        r.close()


@pytest.mark.gpu
def test_two_tip_tree_by_hand(ctx):
    e = two_tip_tree(0.0, 1.0, 2.0)
    _, sites, _ = synth(0, num_tips=8, num_sites=50)
    r = Resident(ctx, [e], [sites])
    try:
        for n0, g, t0 in [(1.0, 0.0, 0.0), (2.5, 0.8, 1.5), (0.3, -1.7, -2.0), (4.0, 1e-12, 0.5)]:
            assert math.isclose(r.forest.log_coalescent_prior(n0, g, t0)[0], two_tip_by_hand(n0, g, t0), rel_tol=RTOL)
    finally:
        r.close()


@pytest.mark.gpu
def test_single_tree(ctx):
    emat, sites, _ = synth(1)                                       # 200 tips
    check_forest(ctx, [emat], [sites])


@pytest.mark.gpu
def test_batch_of_trees_of_different_sizes(ctx):
    shapes = [dict(num_tips=2), dict(num_tips=3), dict(num_tips=129), dict(num_tips=700), dict(num_tips=3000), dict(num_tips=40),
              dict(num_tips=1500, caterpillar=1)]
    trees = [synth(0, num_sites=300, seed=100 + k, **s) for k, s in enumerate(shapes)]
    emats, sites = [t[0] for t in trees], [t[1] for t in trees]
    batch = check_forest(ctx, emats, sites)
    # each tree alone gives the value it has inside the batch
    for k in range(len(emats)):
        alone = check_forest(ctx, [emats[k]], [sites[k]], params=PARAMS[:1])
        assert math.isclose(alone[0], batch[k], rel_tol=1e-13)


@pytest.mark.gpu
def test_large_tree(ctx):
    emat, sites, _ = synth(3, num_sites=500)                        # 10k tips: many tiles per tree, one scan carry per tile
    check_forest(ctx, [emat], [sites], params=[(3.0, 0.0, 0.0), (3.0, 1e-12, 0.0), (0.7, 25.0, 0.0)])


@pytest.mark.gpu
def test_tiny_growth_is_constant_population(ctx):
    emat, sites, _ = synth(1)
    r = Resident(ctx, [emat], [sites])
    try:
        base = r.forest.log_coalescent_prior(3.0, 0.0, 0.0)[0]
        for g in (1e-12, -1e-12, 1e-300):
            assert math.isclose(r.forest.log_coalescent_prior(3.0, g, 0.0)[0], base, rel_tol=1e-9)
    finally:
        r.close()


@pytest.mark.gpu
def test_isochronous_and_tied_dates(ctx):
    trees = [synth(0, num_tips=n, num_sites=300, seed=7 + n) for n in (64, 500, 2500)]
    emats = [isochronous(trees[0][0]), tied(trees[1][0], 0.05), tied(trees[2][0], 0.02), isochronous(trees[2][0])]
    sites = [trees[0][1], trees[1][1], trees[2][1], trees[2][1]]
    for e in emats[1:3]:                                              # the ties are there, and the tie order is immaterial
        assert len(np.unique(e.t)) < 0.75 * e.num_nodes
        want = ref_log_prior(e, 2.0, 3.0, 0.0)
        assert math.isclose(ref_log_prior(e, 2.0, 3.0, 0.0, np.random.default_rng(1)), want, rel_tol=1e-13)
    check_forest(ctx, emats, sites)


@pytest.mark.gpu
def test_follows_device_node_times(ctx):
    emat, sites, _ = synth(0, num_tips=300, num_sites=300)
    r = Resident(ctx, [emat], [sites])
    try:
        tips = np.nonzero(emat.child0 < 0)[0][:40]
        t = emat.t.copy()
        t[tips] += 0.01                                              # later tips stay later than their parents
        r.forest.set_node_times(0, tips, t[tips])
        got = r.forest.log_coalescent_prior(3.0, 4.0, 0.0)[0]
        assert math.isclose(got, ref_log_prior(with_times(emat, t), 3.0, 4.0, 0.0), rel_tol=RTOL)
    finally:
        r.close()


@pytest.mark.gpu
def test_rejects_bad_parameters(ctx):
    emat, sites, _ = synth(0, num_tips=20, num_sites=100)
    r = Resident(ctx, [emat], [sites])
    try:
        for n0, g, t0 in [(0.0, 1.0, 0.0), (-1.0, 1.0, 0.0), (math.inf, 1.0, 0.0), (1.0, math.nan, 0.0), (1.0, 1.0, math.inf)]:
            with pytest.raises(db.DphyError) as ei:
                r.forest.log_coalescent_prior(n0, g, t0)
            assert ei.value.status == db.ERR_INVALID_ARGUMENT
    finally:
        r.close()


# ---- composition with placement --------------------------------------------------------------------------------------------------
def root_path_deltas(emat, sites, v):
    """the sequence at node v as deltas from the reference"""
    path = []
    while v >= 0:
        path.append(v)
        v = int(emat.parent[v])
    diffs = {}
    for u in reversed(path):
        for i in range(int(emat.mut_off[u]), int(emat.mut_off[u + 1])):
            l, to = int(emat.mut_site[i]), int(emat.mut_to[i])
            if to == int(sites.ref[l]):
                diffs.pop(l, None)
            else:
                diffs[l] = to
    return sorted(diffs.items())


def graft(emat, grafts):
    """Attach one new tip per (branch, mut_idx, t_attach, t_tip): a new inner node on `branch` at t_attach taking the branch's
    mutations before mut_idx, and the tip below it (no mutations).  Branches are distinct and not the root."""
    n = emat.num_nodes
    parent, child0, child1 = list(emat.parent), list(emat.child0), list(emat.child1)
    t = list(emat.t)
    muts = {v: list(range(int(emat.mut_off[v]), int(emat.mut_off[v + 1]))) for v in range(n)}
    new_muts = {}
    for k, (b, mi, ta, tt) in enumerate(grafts):
        p, x, gp = n + 2 * k, n + 2 * k + 1, parent[b]
        if child0[gp] == b:
            child0[gp] = p
        else:
            child1[gp] = p
        parent += [gp, p]; child0 += [b, -1]; child1 += [x, -1]; t += [ta, tt]
        parent[b] = p
        new_muts[p], muts[b] = muts[b][:mi], muts[b][mi:]
        new_muts[x] = []
    muts.update(new_muts)
    N = len(parent)
    order = [i for v in range(N) for i in muts[v]]
    mut_off = np.cumsum([0] + [len(muts[v]) for v in range(N)])
    pad = lambda off: np.concatenate([off, np.full(N - n, off[-1], off.dtype)])      # new nodes: no missations, no from-states
    return db.HostEmat(emat.root, emat.includes_run_root, parent=parent, child0=child0, child1=child1, t=t, mut_off=mut_off,
                       mut_site=emat.mut_site[order], mut_from=emat.mut_from[order], mut_to=emat.mut_to[order], mut_t=emat.mut_t[order],
                       miss_off=pad(emat.miss_off), miss_start=emat.miss_start, miss_end=emat.miss_end, fs_off=pad(emat.fs_off),
                       fs_site=emat.fs_site, fs_from=emat.fs_from)


@pytest.mark.gpu
def test_tree_grown_by_placed_samples(ctx):
    emat, sites, _ = synth(0, num_tips=400, num_sites=2000, muts_per_tip=3.0, seed=11)
    rng = np.random.default_rng(5)
    r = Resident(ctx, [emat], [sites])
    try:
        before = r.forest.log_coalescent_prior(3.0, 4.0, 0.0)
        # new samples: existing tips' sequences with a few extra differences
        tips = rng.choice(np.nonzero(emat.child0 < 0)[0], 30, replace=False)
        samples = []
        for v in tips:
            d = dict(root_path_deltas(emat, sites, int(v)))
            for l in rng.integers(0, sites.num_sites, 2):
                d[int(l)] = int((sites.ref[l] + 1 + rng.integers(3)) % 4)
            samples.append(sorted(d.items()))
        arrays = dict(delta_off=np.cumsum([0] + [len(s) for s in samples]), delta_site=[l for s in samples for l, _ in s],
                      delta_to=[a for s in samples for _, a in s], miss_off=np.zeros(len(samples) + 1, np.int32), miss_start=[], miss_end=[])
        placed = r.forest.place_samples(arrays, can_change_root=False, max_best=1)
        assert np.array_equal(r.forest.log_coalescent_prior(3.0, 4.0, 0.0), before)     # placement leaves the tree as it was
        grafts, used = [], set()
        t_latest = float(emat.t.max())
        for k in range(len(samples)):
            reg = placed["best"][k, 0]
            b = int(reg["branch"])
            if b < 0 or b == emat.root or b in used:
                continue
            used.add(b)
            ta = 0.5 * (float(reg["t_min"]) + float(reg["t_max"]))
            grafts.append((b, int(reg["mut_idx"]), ta, max(ta, t_latest - 0.05 * (k % 4))))
        assert len(grafts) >= 10
        grown = graft(emat, grafts)
        assert grown.num_nodes == emat.num_nodes + 2 * len(grafts)
        check_forest(ctx, [grown, emat], [sites, sites])
    finally:
        r.close()
