"""GPU parity: maximum-parsimony placement of new samples (dphy_forest_place_samples) vs the unbounded study of the sample from
the root -- the oracle's builder (orc_spr_study_build, X == -1, t_X == DBL_MAX) and, on a 100k-tip tree, the device's own
dphy_spr_study_batch.  Every output is an integer or a copied double: all bit-exact."""
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


# ---- samples ----------------------------------------------------------------------------------------------------------------------
def tip_sample(emat, sites, v):
    """(deltas [(site, state)], missing intervals [(start, end)]) of node v: the reference overlaid with the root->v mutations."""
    path = []
    u = int(v)
    while u >= 0:
        path.append(u)
        u = int(emat.parent[u])
    diffs, ivls = {}, []
    for u in reversed(path):
        for i in range(int(emat.mut_off[u]), int(emat.mut_off[u + 1])):
            l, to = int(emat.mut_site[i]), int(emat.mut_to[i])
            if to == int(sites.ref[l]):
                diffs.pop(l, None)
            else:
                diffs[l] = to
        ivls += [(int(emat.miss_start[i]), int(emat.miss_end[i])) for i in range(int(emat.miss_off[u]), int(emat.miss_off[u + 1]))]
    return sorted(diffs.items()), ivls


def sample_set(samples):
    """list of (deltas, intervals) -> the six CSR arrays"""
    d_off = np.zeros(len(samples) + 1, np.int32)
    m_off = np.zeros(len(samples) + 1, np.int32)
    for k, (d, iv) in enumerate(samples):
        d_off[k + 1] = d_off[k] + len(d)
        m_off[k + 1] = m_off[k] + len(iv)
    ds = [l for d, _ in samples for l, _ in d]
    dt = [t for d, _ in samples for _, t in d]
    ms = [a for _, iv in samples for a, _ in iv]
    me = [b for _, iv in samples for _, b in iv]
    return dict(delta_off=d_off, delta_site=np.array(ds, np.int32), delta_to=np.array(dt, np.uint8), miss_off=m_off,
                miss_start=np.array(ms, np.int32), miss_end=np.array(me, np.int32))


def samples_of(arrays):
    """the six CSR arrays -> list of (deltas, intervals)"""
    out = []
    for k in range(len(arrays["delta_off"]) - 1):
        d0, d1 = int(arrays["delta_off"][k]), int(arrays["delta_off"][k + 1])
        i0, i1 = int(arrays["miss_off"][k]), int(arrays["miss_off"][k + 1])
        out.append(([(int(arrays["delta_site"][i]), int(arrays["delta_to"][i])) for i in range(d0, d1)],
                    [(int(arrays["miss_start"][i]), int(arrays["miss_end"][i])) for i in range(i0, i1)]))
    return out


def make_samples(emat, sites, rng, n_tips=24, n_perturbed=24):
    """Tips as they are (min_muts 0), perturbed tips, and the edge cases of the REL_REF input rules."""
    L = sites.num_sites
    tips = np.nonzero(emat.child0 < 0)[0]
    chosen = rng.choice(tips, min(n_tips, len(tips)), replace=False)
    exact = [tip_sample(emat, sites, v) for v in chosen]
    out = list(exact)
    for k in range(n_perturbed):
        d, iv = exact[k % len(exact)]
        d = list(d) + [(int(rng.integers(L)), int(rng.integers(4))) for _ in range(int(rng.integers(1, 8)))]
        iv = list(iv)
        for _ in range(int(rng.integers(0, 4))):
            a = int(rng.integers(L))
            iv.append((a, min(L, a + int(rng.integers(1, max(2, L // 50))))))
        rng.shuffle(d)
        rng.shuffle(iv)
        out.append((d, iv))
    d, iv = exact[0]
    s0 = int(rng.integers(L - 20))
    out.append((list(d) + [(s0, 1), (s0, 2), (s0, 3), (s0 + 1, 0), (s0 + 1, 3)], iv))                       # duplicated delta sites
    out.append((list(d), list(iv) + [(s0 + 5, s0 + 15), (s0, s0 + 10), (s0 + 2, s0 + 4), (s0, s0 + 10)]))   # overlapping, unsorted
    out.append((list(d) + [(s0 + 3, 2), (s0 + 7, 1)], list(iv) + [(s0 + 2, s0 + 9)]))                       # deltas inside their intervals
    out.append(([], []))                                                                                    # the reference itself
    out.append(([(0, 3)], [(0, L)]))                                                                        # nothing observed
    half = [(i * L // 20, i * L // 20 + L // 40) for i in range(20)]
    rng.shuffle(half)
    out.append((list(d), half))                                                                             # about half the sites missing
    return out, len(exact)


# ---- what the study says --------------------------------------------------------------------------------------------------------------
def oracle_place(orc, e, s, emat, sample, ccr, max_best):
    """(min_muts, num_best, branch, mut_idx, first max_best regions) from the oracle's full region list."""
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
    regs, _ = orc.spr_study(e, s, -1, DBL_MAX, (ms, me), root, n_root, init, INF, ccr)
    if len(regs) == 0:
        return -1, 0, -1, -1, regs
    m = regs["min_muts"].min()
    hits = np.nonzero(regs["min_muts"] == m)[0]
    return int(m), len(hits), int(regs["branch"][hits[0]]), int(regs["mut_idx"][hits[0]]), regs[hits[:max_best]]


def check_against_oracle(orc, e, s, emat, samples, got, ccr, max_best):
    for k, smp in enumerate(samples):
        m, nb, br, mi, regs = oracle_place(orc, e, s, emat, smp, ccr, max_best)
        assert (got["min_muts"][k], got["num_best"][k], got["branch"][k], got["mut_idx"][k]) == (m, nb, br, mi), k
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


def _forest(ctx, emat, sites):
    ds = db.DeviceSites(ctx, sites)
    return db.Forest(ctx, [emat], [ds]), ds


# ---- the reference's fixture ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ccr", [True, False])
def test_complex_tree(ctx, orc, ccr):
    e, s, n = complex_tree()
    emat, sites = from_oracle(e, s)
    fo, ds = _forest(ctx, emat, sites)
    samples = [([(0, T)], [(3, 4)])]                   # full_study_new_seq (tests/spr_study_tests.cpp:183-205)
    samples += [tip_sample(emat, sites, v) for v in range(emat.num_nodes)]
    samples += [([], []), ([(0, T), (0, A), (1, 2)], [(2, 4), (3, 4)]), ([], [(0, 4)]), ([(2, 3)], [(0, 1)])]
    for mb in (0, 1, 7, 20):
        got = fo.place_samples(sample_set(samples), can_change_root=ccr, max_best=mb)
        check_against_oracle(orc, e, s, emat, samples, got, ccr, mb)
    got = fo.place_samples(sample_set(samples[:1]), can_change_root=ccr)
    assert got["num_best"][0] >= 1
    fo.close(); ds.close()


SYNTH_CASES = [
    (0, {}),
    (0, dict(num_root_mutations=6, num_partitions=2)),
    (0, dict(caterpillar=1, num_tips=400)),
    (0, dict(num_tips=2500, muts_per_tip=24.0)),
    (1, {}),
    (2, {}),
    (3, {}),
    (5, dict(num_tips=60, num_sites=6000, num_partitions=1)),
]


@pytest.mark.parametrize("cfg,ov", SYNTH_CASES)
def test_synthetic_trees(ctx, orc, cfg, ov):
    emat, sites, info = synth(cfg, **ov)
    e, s = to_oracle(emat, sites)
    fo, ds = _forest(ctx, emat, sites)
    rng = np.random.default_rng(17 + cfg)
    samples, n_exact = make_samples(emat, sites, rng, n_tips=16 if cfg == 3 else 24, n_perturbed=8 if cfg == 3 else 24)
    arrays = sample_set(samples)
    R = emat.num_nodes + int(emat.mut_off[-1]) - int(emat.mut_off[emat.root + 1] - emat.mut_off[emat.root])
    for ccr in (True, False):
        mbs = (0, 1, 7, R + 1) if cfg == 0 and not ov else ((0, 7) if ccr else (1,))
        for mb in mbs:
            got = fo.place_samples(arrays, can_change_root=ccr, max_best=mb)
            assert (got["min_muts"][:n_exact] == 0).all()
            if mb == R + 1:      # larger than any num_best: every best region, the rest unused
                assert (got["best"]["branch"][np.arange(len(samples)), got["num_best"]] == -1).all()
            check_against_oracle(orc, e, s, emat, samples, got, ccr, mb)
            # the sample missing [0, L) ties every region of the study
            assert got["num_best"][len(samples) - 2] == R - (0 if ccr else 1)
    fo.close(); ds.close()


def test_maple_round_trip(ctx, orc):
    emat, sites, info = synth(0)
    e, s = to_oracle(emat, sites)
    fo, ds = _forest(ctx, emat, sites)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "tips.maple")
        n = maple.write_maple(emat, sites, path)
        with open(path, "rb") as f:
            parsed = db.maple_parse(f.read())
    assert len(parsed["delta_off"]) == n + 1
    got = fo.place_samples(parsed, max_best=3)
    assert (got["min_muts"] == 0).all()
    check_against_oracle(orc, e, s, emat, samples_of(parsed), got, True, 3)
    fo.close(); ds.close()


def test_forest_of_three_trees(ctx, orc):
    items = [synth(0), synth(0, num_tips=300, seed=5), synth(2, num_tips=120, num_sites=4000)]
    tables = [db.DeviceSites(ctx, it[1]) for it in items]
    fo = db.Forest(ctx, [it[0] for it in items], tables, sites_index=[0, 1, 2])
    for k in (1, 2):
        emat, sites, _ = items[k]
        e, s = to_oracle(emat, sites)
        samples, _ = make_samples(emat, sites, np.random.default_rng(k), 12, 12)
        got = fo.place_samples(sample_set(samples), tree=k, max_best=4)
        check_against_oracle(orc, e, s, emat, samples, got, True, 4)
    fo.close()
    for t in tables:
        t.close()


def relabel(emat, perm):
    """the same tree with node v renamed perm[v]"""
    N = emat.num_nodes
    inv = np.argsort(perm)
    mp = lambda a: np.where(a >= 0, perm[np.maximum(a, 0)], -1).astype(np.int32)

    def lists(off, *arrs):
        cnt = np.diff(off)[inv]
        noff = np.zeros(N + 1, np.int32)
        noff[1:] = np.cumsum(cnt)
        idx = np.concatenate([np.arange(off[v], off[v + 1]) for v in inv]).astype(np.int64) if noff[-1] else np.zeros(0, np.int64)
        return [noff] + [a[idx] for a in arrs]
    mo, ms, mf, mt, mtt = lists(emat.mut_off, emat.mut_site, emat.mut_from, emat.mut_to, emat.mut_t)
    io, ist, ien = lists(emat.miss_off, emat.miss_start, emat.miss_end)
    fo, fs, ff = lists(emat.fs_off, emat.fs_site, emat.fs_from)
    return db.HostEmat(int(perm[emat.root]), emat.includes_run_root, parent=mp(emat.parent)[inv], child0=mp(emat.child0)[inv],
                       child1=mp(emat.child1)[inv], t=emat.t[inv], mut_off=mo, mut_site=ms, mut_from=mf, mut_to=mt, mut_t=mtt,
                       miss_off=io, miss_start=ist, miss_end=ien, fs_off=fo, fs_site=fs, fs_from=ff)


def test_index_follows_edits(ctx, orc):
    a, _, _ = synth(0)
    b0, sites, _ = synth(0, seed=77)
    assert a.num_nodes == b0.num_nodes
    perm = np.random.default_rng(3).permutation(b0.num_nodes)
    b = relabel(b0, perm)
    assert b.root != a.root
    ds = db.DeviceSites(ctx, sites)
    fo = db.Forest(ctx, [a], [ds])
    samples, _ = make_samples(b, sites, np.random.default_rng(8), 16, 16)
    arrays = sample_set(samples)
    fo.place_samples(arrays, max_best=2)            # builds the index of tree `a`
    fo.apply_rows([db.node_row(0, b, v) for v in range(b.num_nodes)], new_roots=[b.root])
    e, s = to_oracle(b, sites)
    got = fo.place_samples(arrays, max_best=5)
    check_against_oracle(orc, e, s, b, samples, got, True, 5)
    # node times: only the reported t_min / t_max depend on them, and they follow
    tips = np.nonzero(b.child0 < 0)[0]
    b.t[tips] += 0.25
    fo.set_node_times(0, tips, b.t[tips])
    e, s = to_oracle(b, sites)
    got = fo.place_samples(arrays, max_best=5)
    check_against_oracle(orc, e, s, b, samples, got, True, 5)
    fo.close(); ds.close()


# ---- refusals --------------------------------------------------------------------------------------------------------------------------
def _raw_place(ctx, fo, arrays, tree=0):
    a = {k: np.ascontiguousarray(v) for k, v in arrays.items()}
    S = len(a["delta_off"]) - 1
    ss = db.SampleSet(S, 0, a["delta_off"].ctypes.data_as(db.i32p), a["delta_site"].ctypes.data_as(db.i32p),
                      a["delta_to"].ctypes.data_as(db.u8p), a["miss_off"].ctypes.data_as(db.i32p),
                      a["miss_start"].ctypes.data_as(db.i32p), a["miss_end"].ctypes.data_as(db.i32p))
    out = np.full(S, -7, db.PLACEMENT_DTYPE)
    st = db.lib().dphy_forest_place_samples(ctx._h, fo._h, tree, C.byref(ss), 1, 0, out.ctypes.data_as(C.POINTER(db.Placement)), None)
    return st, out


def test_refusals(ctx):
    emat, sites, _ = synth(0)
    L = sites.num_sites
    fo, ds = _forest(ctx, emat, sites)
    good = [([(5, 1)], [(10, 20)]), ([(7, 2)], [])]
    st, out = _raw_place(ctx, fo, sample_set(good))
    assert st == db.DPHY_OK and (out["num_best"] > 0).all()
    cases = [
        (sample_set(good), 1, db.ERR_OUT_OF_RANGE),                               # tree index
        (sample_set(good), -1, db.ERR_OUT_OF_RANGE),
        (sample_set([([(L, 1)], [])]), 0, db.ERR_OUT_OF_RANGE),                    # site >= L
        (sample_set([([(-1, 1)], [])]), 0, db.ERR_OUT_OF_RANGE),
        (sample_set([([(3, 4)], [])]), 0, db.ERR_OUT_OF_RANGE),                    # state > 3
        (sample_set([([], [(9, 9)])]), 0, db.ERR_OUT_OF_RANGE),                    # start >= end
        (sample_set([([], [(12, 9)])]), 0, db.ERR_OUT_OF_RANGE),
        (sample_set([([], [(L - 3, L + 1)])]), 0, db.ERR_OUT_OF_RANGE),            # end > L
    ]
    bad = sample_set(good)
    bad["delta_off"] = np.array([0, 2, 1], np.int32)                              # offsets not monotone
    bad["delta_site"] = np.array([5, 7], np.int32); bad["delta_to"] = np.array([1, 2], np.uint8)
    cases.append((bad, 0, db.ERR_INVALID_ARGUMENT))
    bad = sample_set(good)
    bad["miss_off"] = np.array([0, 1, 0], np.int32)
    cases.append((bad, 0, db.ERR_INVALID_ARGUMENT))
    for arrays, tree, want in cases:
        st, out = _raw_place(ctx, fo, arrays, tree)
        assert st == want, (arrays, tree)
        assert (out["min_muts"] == -7).all() and (out["branch"] == -7).all()
    empty = fo.place_samples(sample_set([]))
    assert len(empty["min_muts"]) == 0
    fo.close(); ds.close()


# ---- a 100k-tip tree (synthetic config 4, BASELINE.json configs[3]) -----------------------------------------------------------------------
@pytest.fixture(scope="module")
def big():
    emat, sites, info = synth(4)
    return emat, sites, info


def _perturbed_tips(emat, sites, rng, n):
    L = sites.num_sites
    tips = np.nonzero(emat.child0 < 0)[0]
    out = []
    for v in rng.choice(tips, n, replace=False):
        d, iv = tip_sample(emat, sites, v)
        d = list(d) + [(int(rng.integers(L)), int(rng.integers(4))) for _ in range(int(rng.integers(0, 4)))]
        if rng.random() < 0.5:
            a = int(rng.integers(L - 2000))
            iv = list(iv) + [(a, a + int(rng.integers(1, 2000)))]
        out.append((d, iv))
    return out


def test_large_tree_vs_oracle(ctx, orc, big):
    emat, sites, info = big
    e, s = to_oracle(emat, sites)
    fo, ds = _forest(ctx, emat, sites)
    samples = _perturbed_tips(emat, sites, np.random.default_rng(41), 200)
    got = fo.place_samples(sample_set(samples), max_best=3)
    check_against_oracle(orc, e, s, emat, samples, got, True, 3)
    fo.close(); ds.close()


def test_large_tree_vs_study_batches(ctx, big):
    emat, sites, info = big
    fo, ds = _forest(ctx, emat, sites)
    samples = _perturbed_tips(emat, sites, np.random.default_rng(42), 2000)
    got = fo.place_samples(sample_set(samples))
    root = int(emat.root)
    n_root = int(emat.mut_off[root + 1] - emat.mut_off[root])
    ref = np.asarray(sites.ref, np.uint8)
    rs = ref.copy()
    for i in range(int(emat.mut_off[root]), int(emat.mut_off[root + 1])):
        rs[int(emat.mut_site[i])] = int(emat.mut_to[i])
    for b0 in range(0, len(samples), 64):
        reqs = []
        for d, iv in samples[b0:b0 + 64]:
            x = ref.copy()
            for l, t in d:
                x[l] = t
            miss = np.zeros(len(ref), bool)
            for a, b in iv:
                miss[a:b] = True
            init = int((~miss & (rs != x)).sum())
            reqs.append(db.spr_request(0, -1, DBL_MAX, root, n_root, init, 0.0, info["t_max_tip"], INF, True,
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
    fo.close(); ds.close()
