"""GPU parity: dated maximum-parsimony placement (dphy_forest_place_dated_samples, Forest.place_samples(..., t_X=...)) vs the
oracle's region list of the unbounded study from the root after remove_regions_in_Xs_future with the sample's own t_X
(orc_spr_study_build), and, on a 100k-tip tree, vs the device's own dphy_spr_study_batch with the same per-request t_X.  Every
output is an integer or a copied (or clipped) double: all bit-exact."""
import ctypes as C
import os
import tempfile

import numpy as np
import pytest

import delphy_b200 as db
from delphy_b200 import maple
from emat_fixtures import A, T, DBL_MAX, complex_tree
from helpers import from_oracle, synth, to_oracle
from oracle_lib import Oracle
from test_gpu_placement import SYNTH_CASES, make_samples, relabel, sample_set, samples_of, tip_sample

pytestmark = pytest.mark.gpu
INF = 2**31 - 1


@pytest.fixture(scope="module")
def ctx():
    c = db.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def orc():
    return Oracle("oracle")


def _forest(ctx, emat, sites):
    ds = db.DeviceSites(ctx, sites)
    return db.Forest(ctx, [emat], [ds]), ds


# ---- what the study says ----------------------------------------------------------------------------------------------------------------
def oracle_place_dated(orc, e, s, emat, sample, t_X, ccr, max_best):
    """(min_muts, num_best, branch, mut_idx, first max_best regions) over the oracle's region list with date limit t_X."""
    deltas, ivls = sample
    ref = np.asarray(s.ref, np.uint8)
    L = len(ref)
    x = ref.copy()
    for l, t in deltas:
        x[l] = t
    miss = np.zeros(L + 2, bool)
    for a, b in ivls:
        miss[a + 1:b + 1] = True
    edges = np.diff(miss.astype(np.int8))
    ms = np.nonzero(edges == 1)[0].astype(np.int32)
    me = np.nonzero(edges == -1)[0].astype(np.int32)
    miss = miss[1:L + 1]
    root = int(emat.root)
    rs = ref.copy()
    for i in range(int(emat.mut_off[root]), int(emat.mut_off[root + 1])):
        rs[int(emat.mut_site[i])] = int(emat.mut_to[i])
    idx = np.nonzero(~miss & (rs != x))[0]
    init = [(int(l), int(rs[l]), int(x[l])) for l in idx]
    n_root = int(emat.mut_off[root + 1] - emat.mut_off[root])
    regs, _ = orc.spr_study(e, s, -1, float(t_X), (ms, me), root, n_root, init, INF, ccr)
    if len(regs) == 0:
        return -1, 0, -1, -1, regs
    m = regs["min_muts"].min()
    hits = np.nonzero(regs["min_muts"] == m)[0]
    return int(m), len(hits), int(regs["branch"][hits[0]]), int(regs["mut_idx"][hits[0]]), regs[hits[:max_best]]


def check_dated(orc, e, s, emat, samples, t_X, got, ccr, max_best):
    for k, smp in enumerate(samples):
        m, nb, br, mi, regs = oracle_place_dated(orc, e, s, emat, smp, t_X[k], ccr, max_best)
        assert (got["min_muts"][k], got["num_best"][k], got["branch"][k], got["mut_idx"][k]) == (m, nb, br, mi), (k, t_X[k])
        if max_best:
            b = got["best"][k]
            n = len(regs)
            for f in ("branch", "mut_idx", "min_muts"):
                np.testing.assert_array_equal(b[f][:n], regs[f], err_msg=f"{k} {f}")
            for f in ("t_min", "t_max"):
                assert np.array_equal(b[f][:n], regs[f]), (k, f)
            assert not b["log_W_over_Wmax"].any() and not b["W_over_Wmax"].any()
            assert (b["branch"][n:] == -1).all()
            for f in ("mut_idx", "min_muts", "t_min", "t_max"):
                assert not b[f][n:].any(), (k, f)


def assert_same(a, b):
    for f in ("min_muts", "num_best", "branch", "mut_idx"):
        np.testing.assert_array_equal(a[f], b[f], err_msg=f)
    assert a["best"].tobytes() == b["best"].tobytes()


def tree_times(emat):
    """every node time and every mutation time of the tree, distinct and ascending"""
    return np.unique(np.concatenate([emat.t, emat.mut_t]))


# ---- the reference's fixture ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ccr", [True, False])
def test_complex_tree(ctx, orc, ccr):
    e, s, n = complex_tree()
    emat, sites = from_oracle(e, s)
    fo, ds = _forest(ctx, emat, sites)
    samples = [([(0, T)], [(3, 4)])]
    samples += [tip_sample(emat, sites, v) for v in range(emat.num_nodes)]
    samples += [([], []), ([(0, T), (0, A), (1, 2)], [(2, 4), (3, 4)]), ([], [(0, 4)]), ([(2, 3)], [(0, 1)])]
    arrays = sample_set(samples)
    times = tree_times(emat)
    finite = times[times > -DBL_MAX]
    limits = list(times) + list(0.5 * (finite[1:] + finite[:-1])) + [float(emat.t[emat.root]) - 1.0, -DBL_MAX, np.inf, DBL_MAX]
    for tX in limits:
        t_X = np.full(len(samples), tX)
        for mb in (0, 7):
            got = fo.place_samples(arrays, can_change_root=ccr, max_best=mb, t_X=t_X)
            check_dated(orc, e, s, emat, samples, t_X, got, ccr, mb)
        if tX <= -DBL_MAX:
            assert (got["min_muts"] == -1).all() and (got["num_best"] == 0).all() and (got["branch"] == -1).all()
    # every limit in one call, in shuffled order
    rng = np.random.default_rng(5)
    big = samples * len(limits)
    t_X = rng.permutation(np.repeat(limits, len(samples)))
    got = fo.place_samples(sample_set(big), can_change_root=ccr, max_best=3, t_X=t_X)
    check_dated(orc, e, s, emat, big, t_X, got, ccr, 3)
    fo.close(); ds.close()


# ---- synthetic shapes -------------------------------------------------------------------------------------------------------------------
def dated_samples(emat, sites, rng, n_tips, n_perturbed):
    """tips with their own time as the limit, plus make_samples' exact / perturbed / edge-case samples with limits tied to a node or
    mutation time, or at a random quantile of the tree's times; in shuffled order"""
    tips = np.nonzero(emat.child0 < 0)[0]
    own = rng.choice(tips, min(n_tips, len(tips)), replace=False)
    samples = [tip_sample(emat, sites, v) for v in own]
    t_X = [float(emat.t[v]) for v in own]
    more, _ = make_samples(emat, sites, rng, n_tips, n_perturbed)
    times = tree_times(emat)
    for k in range(len(more)):
        c = k % 3
        if c == 0:
            t_X.append(float(rng.choice(emat.t)))
        elif c == 1:
            t_X.append(float(rng.choice(emat.mut_t)) if len(emat.mut_t) else float(rng.choice(emat.t)))
        else:
            t_X.append(float(np.quantile(times[times > -DBL_MAX], rng.random())))
    samples += more
    order = rng.permutation(len(samples))
    return [samples[i] for i in order], np.array(t_X)[order]


@pytest.mark.parametrize("cfg,ov", SYNTH_CASES)
def test_synthetic_trees(ctx, orc, cfg, ov):
    emat, sites, info = synth(cfg, **ov)
    e, s = to_oracle(emat, sites)
    fo, ds = _forest(ctx, emat, sites)
    rng = np.random.default_rng(101 + cfg)
    samples, t_X = dated_samples(emat, sites, rng, 8 if cfg == 3 else 16, 8 if cfg == 3 else 16)
    arrays = sample_set(samples)
    for ccr in (True, False):
        for mb in (0, 5):
            got = fo.place_samples(arrays, can_change_root=ccr, max_best=mb, t_X=t_X)
            check_dated(orc, e, s, emat, samples, t_X, got, ccr, mb)
    fo.close(); ds.close()


# ---- identity with the undated call -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", [0, 3])
def test_unbounded_limit_is_the_undated_call(ctx, cfg):
    emat, sites, _ = synth(cfg)
    fo, ds = _forest(ctx, emat, sites)
    samples, _ = make_samples(emat, sites, np.random.default_rng(9), 16, 16)
    arrays = sample_set(samples)
    S = len(samples)
    for ccr in (True, False):
        want = fo.place_samples(arrays, can_change_root=ccr, max_best=6)
        bytes0 = fo.device_bytes
        for tX in (DBL_MAX, np.inf):
            got = fo.place_samples(arrays, can_change_root=ccr, max_best=6, t_X=np.full(S, tX))
            assert_same(got, want)
        assert fo.device_bytes == bytes0            # no region dropped: the dated part is not built
    # a limit that drops regions builds it; DBL_MAX still gives the undated result through it
    fo.place_samples(arrays, t_X=np.full(S, float(np.median(emat.t))))
    assert fo.device_bytes > bytes0
    want = fo.place_samples(arrays, max_best=6)
    assert_same(fo.place_samples(arrays, max_best=6, t_X=np.full(S, DBL_MAX)), want)
    fo.close(); ds.close()


# ---- MAPLE ------------------------------------------------------------------------------------------------------------------------------
def test_maple_round_trip(ctx, orc):
    emat, sites, info = synth(0)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "tips.maple")
        n = maple.write_maple(emat, sites, path)
        with open(path, "rb") as f:
            parsed = db.maple_parse(f.read())
    assert len(parsed["delta_off"]) == n + 1 and len(parsed["t_max"]) == n
    # MAPLE dates are days since 2020-01-01 and write_maple puts the latest tip on 2021-01-01 (day 366): the tree goes to that unit
    tips = np.nonzero(emat.child0 < 0)[0]
    t_max_tip = float(emat.t[tips].max())
    emat.t[:] = (emat.t - t_max_tip) * 365.0 + 366.0
    emat.mut_t[:] = np.where(emat.mut_t > -DBL_MAX, (emat.mut_t - t_max_tip) * 365.0 + 366.0, emat.mut_t)
    e, s = to_oracle(emat, sites)
    fo, ds = _forest(ctx, emat, sites)
    got = fo.place_samples(parsed, max_best=3, t_X=parsed["t_max"])
    check_dated(orc, e, s, emat, samples_of(parsed), parsed["t_max"], got, True, 3)
    fo.close(); ds.close()


# ---- the dated part follows the tree ----------------------------------------------------------------------------------------------------
def test_node_time_edits(ctx, orc):
    emat, sites, _ = synth(0, seed=31)
    fo, ds = _forest(ctx, emat, sites)
    rng = np.random.default_rng(12)
    samples, t_X = dated_samples(emat, sites, rng, 16, 16)
    arrays = sample_set(samples)
    fo.place_samples(arrays, max_best=4, t_X=t_X)                  # builds the dated part
    bytes0 = fo.device_bytes
    # move inner nodes across the limits: each to a random point between its parent and its earliest child
    inner = [v for v in range(emat.num_nodes) if emat.child0[v] >= 0 and v != emat.root]
    moved = rng.choice(inner, min(40, len(inner)), replace=False)
    for v in moved:
        lo = float(emat.t[emat.parent[v]])
        hi = min(float(emat.t[emat.child0[v]]), float(emat.t[emat.child1[v]]))
        emat.t[v] = lo + rng.random() * (hi - lo)
    m = min(len(moved), len(t_X))
    t_X[:m] = emat.t[moved[:m]]                                     # ties with the new times
    fo.set_node_times(0, moved, emat.t[moved])
    got = fo.place_samples(arrays, max_best=4, t_X=t_X)
    fresh, ds2 = _forest(ctx, emat, sites)
    assert_same(got, fresh.place_samples(arrays, max_best=4, t_X=t_X))
    e, s = to_oracle(emat, sites)
    check_dated(orc, e, s, emat, samples, t_X, got, True, 4)
    assert fo.device_bytes == bytes0                                # rebuilt in the same block
    # an undated call in between changes nothing
    und = fo.place_samples(arrays, max_best=4)
    assert_same(fo.place_samples(arrays, max_best=4, t_X=t_X), got)
    assert_same(fo.place_samples(arrays, max_best=4), und)
    # a refused edit (a node later than its child) still changed the times: the next dated call sees them
    v = int(moved[0])
    emat.t[v] = float(max(emat.t[emat.child0[v]], emat.t[emat.child1[v]])) + 0.5
    with pytest.raises(db.DphyError):
        fo.set_node_times(0, [v], [emat.t[v]])
    t_X[0] = float(emat.t[v]) - 0.25
    got = fo.place_samples(arrays, max_best=4, t_X=t_X)
    e, s = to_oracle(emat, sites)
    check_dated(orc, e, s, emat, samples, t_X, got, True, 4)
    assert fo.device_bytes == bytes0
    fresh.close(); ds2.close(); fo.close(); ds.close()


def test_apply_rows(ctx, orc):
    a, _, _ = synth(0)
    b0, sites, _ = synth(0, seed=77)
    b = relabel(b0, np.random.default_rng(3).permutation(b0.num_nodes))
    ds = db.DeviceSites(ctx, sites)
    fo = db.Forest(ctx, [a], [ds])
    samples, t_X = dated_samples(b, sites, np.random.default_rng(8), 16, 16)
    arrays = sample_set(samples)
    fo.place_samples(arrays, max_best=2, t_X=t_X)                  # builds both parts for tree `a`
    fo.apply_rows([db.node_row(0, b, v) for v in range(b.num_nodes)], new_roots=[b.root])
    e, s = to_oracle(b, sites)
    got = fo.place_samples(arrays, max_best=5, t_X=t_X)
    check_dated(orc, e, s, b, samples, t_X, got, True, 5)
    fo.close(); ds.close()


def test_forest_of_three_trees(ctx, orc):
    items = [synth(0), synth(0, num_tips=300, seed=5), synth(2, num_tips=120, num_sites=4000)]
    tables = [db.DeviceSites(ctx, it[1]) for it in items]
    fo = db.Forest(ctx, [it[0] for it in items], tables, sites_index=[0, 1, 2])
    for k in (2, 0, 1):
        emat, sites, _ = items[k]
        e, s = to_oracle(emat, sites)
        samples, t_X = dated_samples(emat, sites, np.random.default_rng(k), 10, 10)
        got = fo.place_samples(sample_set(samples), tree=k, max_best=4, t_X=t_X)
        check_dated(orc, e, s, emat, samples, t_X, got, True, 4)
    fo.close()
    for t in tables:
        t.close()


# ---- refusals ---------------------------------------------------------------------------------------------------------------------------
def _raw_place_dated(ctx, fo, arrays, t_X, tree=0):
    a = {k: np.ascontiguousarray(v) for k, v in arrays.items()}
    S = len(a["delta_off"]) - 1
    ss = db.SampleSet(S, 0, a["delta_off"].ctypes.data_as(db.i32p), a["delta_site"].ctypes.data_as(db.i32p),
                      a["delta_to"].ctypes.data_as(db.u8p), a["miss_off"].ctypes.data_as(db.i32p),
                      a["miss_start"].ctypes.data_as(db.i32p), a["miss_end"].ctypes.data_as(db.i32p))
    out = np.full(S, -7, db.PLACEMENT_DTYPE)
    tx = None if t_X is None else np.ascontiguousarray(t_X, np.float64).ctypes.data_as(db.f64p)
    st = db.lib().dphy_forest_place_dated_samples(ctx._h, fo._h, tree, C.byref(ss), tx, 1, 0,
                                                  out.ctypes.data_as(C.POINTER(db.Placement)), None)
    return st, out


def test_refusals(ctx):
    emat, sites, _ = synth(0)
    L = sites.num_sites
    fo, ds = _forest(ctx, emat, sites)
    good = [([(5, 1)], [(10, 20)]), ([(7, 2)], [])]
    tx = [float(emat.t[emat.root]) + 0.1, DBL_MAX]
    st, out = _raw_place_dated(ctx, fo, sample_set(good), tx)
    assert st == db.DPHY_OK and (out["num_best"] > 0).all()
    cases = [
        (sample_set(good), None, 0, db.ERR_INVALID_ARGUMENT),                          # no limits
        (sample_set(good), [np.nan, 0.0], 0, db.ERR_INVALID_ARGUMENT),                # NaN
        (sample_set(good), [0.0, -np.nan], 0, db.ERR_INVALID_ARGUMENT),
        (sample_set(good), tx, 1, db.ERR_OUT_OF_RANGE),                                # tree index
        (sample_set(good), tx, -1, db.ERR_OUT_OF_RANGE),
        (sample_set([([(L, 1)], [])]), tx[:1], 0, db.ERR_OUT_OF_RANGE),                # site >= L
        (sample_set([([(3, 4)], [])]), tx[:1], 0, db.ERR_OUT_OF_RANGE),                # state > 3
        (sample_set([([], [(12, 9)])]), tx[:1], 0, db.ERR_OUT_OF_RANGE),               # start >= end
        (sample_set([([], [(L - 3, L + 1)])]), tx[:1], 0, db.ERR_OUT_OF_RANGE),        # end > L
    ]
    bad = sample_set(good)
    bad["delta_off"] = np.array([0, 2, 1], np.int32)                                  # offsets not monotone
    bad["delta_site"] = np.array([5, 7], np.int32); bad["delta_to"] = np.array([1, 2], np.uint8)
    cases.append((bad, tx, 0, db.ERR_INVALID_ARGUMENT))
    for arrays, t_X, tree, want in cases:
        st, out = _raw_place_dated(ctx, fo, arrays, t_X, tree)
        assert st == want, (arrays, t_X, tree)
        assert (out["min_muts"] == -7).all() and (out["branch"] == -7).all()
    with pytest.raises(ValueError):
        fo.place_samples(sample_set(good), t_X=[0.0])
    empty = fo.place_samples(sample_set([]), t_X=[])
    assert len(empty["min_muts"]) == 0
    st, _ = _raw_place_dated(ctx, fo, sample_set([]), None)                           # no samples: no limits needed
    assert st == db.DPHY_OK
    fo.close(); ds.close()


# ---- a 100k-tip tree (synthetic config 4, BASELINE.json configs[3]) -----------------------------------------------------------------------
@pytest.fixture(scope="module")
def big():
    return synth(4)


def test_large_tree(ctx, orc, big):
    emat, sites, info = big
    fo, ds = _forest(ctx, emat, sites)
    rng = np.random.default_rng(43)
    tips = rng.choice(np.nonzero(emat.child0 < 0)[0], 2000, replace=False)
    samples = [tip_sample(emat, sites, v) for v in tips]
    t_X = emat.t[tips].astype(np.float64)
    got = fo.place_samples(sample_set(samples), t_X=t_X)
    root = int(emat.root)
    n_root = int(emat.mut_off[root + 1] - emat.mut_off[root])
    ref = np.asarray(sites.ref, np.uint8)
    rs = ref.copy()
    for i in range(int(emat.mut_off[root]), int(emat.mut_off[root + 1])):
        rs[int(emat.mut_site[i])] = int(emat.mut_to[i])
    for b0 in range(0, len(samples), 64):
        reqs = []
        for (d, iv), tX in zip(samples[b0:b0 + 64], t_X[b0:b0 + 64]):
            x = ref.copy()
            for l, t in d:
                x[l] = t
            miss = np.zeros(len(ref), bool)
            for a, b in iv:
                miss[a:b] = True
            init = int((~miss & (rs != x)).sum())
            reqs.append(db.spr_request(0, -1, float(tX), root, n_root, init, 0.0, info["t_max_tip"], INF, True,
                                       x_deltas=d, x_missing=([a for a, _ in iv], [b for _, b in iv]), x_state_mode=db.SPR_X_REL_REF))
        batch = fo.spr_study_batch(reqs)
        summ = batch.summaries()
        regs = batch.regions()
        for i, sm in enumerate(summ):
            k = b0 + i
            r = regs[sm.region_offset:sm.region_offset + sm.num_regions]
            mm = r["min_muts"]
            m = mm.min()
            j = int(np.argmax(mm == m))
            assert (got["min_muts"][k], got["num_best"][k], got["branch"][k], got["mut_idx"][k]) == \
                (m, int((mm == m).sum()), r["branch"][j], r["mut_idx"][j]), k
        batch.close()
    e, s = to_oracle(emat, sites)
    sub = rng.choice(len(samples), 60, replace=False)
    got = fo.place_samples(sample_set([samples[i] for i in sub]), max_best=3, t_X=t_X[sub])
    check_dated(orc, e, s, emat, [samples[i] for i in sub], t_X[sub], got, True, 3)
    fo.close(); ds.close()
