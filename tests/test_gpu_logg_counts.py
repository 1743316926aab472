"""GPU: the folded log-G schedule reads lambda_i off per-node state counts (ForestDev::C, the root -> node prefix of every branch's
folded weights) that every upload and every re-flatten builds.  Checked against the general schedule, the oracle, and the same
tree uploaded alone, over forests whose trees differ in shape, partition count and upload path, and after edits."""
import numpy as np
import pytest

import delphy_b200 as db
from helpers import rel_err, synth, to_oracle
from oracle_lib import Oracle

pytestmark = pytest.mark.gpu

RTOL = 1e-9


@pytest.fixture(scope="module")
def orc():
    return Oracle("oracle")


def _outputs(fo, k):
    rp, br, lg = fo.log_G()
    return rp[k], br[k], lg[k], fo.lambda_i(k)


def _check_forest(c, orc, items, pinned=False):
    """Folded evaluation of the forest of `items`: every tree == the tree uploaded alone (bit for bit), == the general
    schedule (1e-12), == the oracle (1e-9)."""
    tables = [db.DeviceSites(c, it[1]) for it in items]
    idx = np.arange(len(items))
    fo = db.Forest(c, [it[0].pinned(c) if pinned else it[0] for it in items], tables, sites_index=idx)
    try:
        c.set_log_G_path("auto")
        launches = c.launches
        fo.eval_log_G()
        assert c.launches - launches == 2
        folded = [_outputs(fo, k) for k in range(len(items))]
        c.set_log_G_path("general")
        fo.eval_log_G()
        general = [_outputs(fo, k) for k in range(len(items))]
        c.set_log_G_path("auto")
        for k, (emat, sites, _) in enumerate(items):
            rp, br, lg, lam = folded[k]
            alone = db.Forest(c, [emat], [tables[k]])
            alone.eval_log_G()
            arp, abr, alg, alam = _outputs(alone, 0)
            alone.close()
            assert (rp, br, lg) == (arp, abr, alg)
            assert np.array_equal(lam, alam)
            grp, gbr, _, glam = general[k]
            assert rp == pytest.approx(grp, rel=1e-13)
            assert br == pytest.approx(gbr, rel=1e-12)
            np.testing.assert_allclose(lam, glam, rtol=1e-12)
            e, s = to_oracle(emat, sites)
            lam_o = orc.lambda_i(e, s)
            assert rel_err(lam, lam_o) <= RTOL
            assert rp == pytest.approx(orc.log_root_prior(e, s), rel=RTOL)
            assert br == pytest.approx(orc.log_G_below_root(e, s, lam_o), rel=RTOL)
    finally:
        fo.close()
        for t in tables:
            t.close()


def test_caterpillar_forest(orc):
    """Caterpillars between ordinary trees: their long paths end at tree boundaries, where the post-order lists of two trees meet."""
    items = [synth(0, seed=61, num_tips=700, caterpillar=1), synth(0, seed=62, num_tips=300), synth(0, seed=63, num_tips=1500, caterpillar=1),
             synth(0, seed=64, num_tips=2, num_sites=50, missing_len_max=20.0), synth(0, seed=65, num_tips=513, caterpillar=1)]
    with db.Context(0) as c:
        _check_forest(c, orc, items)


def test_two_partition_forest(orc):
    """A 2-partition tree next to 1-partition ones: the 1-partition trees' count rows are padded to the forest's width."""
    items = [synth(0, seed=71, num_partitions=2, num_root_mutations=5), synth(0, seed=72, num_tips=900), synth(3, seed=73),
             synth(0, seed=74, num_partitions=2, caterpillar=1, num_tips=600)]
    with db.Context(0) as c:
        _check_forest(c, orc, items)


def test_two_phase_pinned_upload(orc):
    """Page-locked arrays: the lists of every tree are folded as they land, the counts built once after the last tree."""
    items = [synth(3, seed=81), synth(0, seed=82, num_tips=300, caterpillar=1), synth(1, seed=83), synth(0, seed=84, num_partitions=2)]
    with db.Context(0) as c:
        _check_forest(c, orc, items, pinned=True)
        tables = [db.DeviceSites(c, it[1]) for it in items]
        idx = np.arange(len(items))
        fa = db.Forest(c, [it[0] for it in items], tables, sites_index=idx)
        fb = db.Forest(c, [it[0].pinned(c) for it in items], tables, sites_index=idx)
        for x, y in zip(fa.log_G(), fb.log_G()):
            assert np.array_equal(x, y)
        for k in range(len(items)):
            assert np.array_equal(fa.lambda_i(k), fb.lambda_i(k))
        fa.close(); fb.close()
        for t in tables:
            t.close()


def _edited(emat, rng, codes_and_missations):
    """A copy of `emat` with, per edit, either new mutation targets and missation intervals on a few branches (list lengths
    unchanged) or later times of a few tips; returns it with the edited nodes."""
    e = db.HostEmat(emat.root, emat.includes_run_root, **{k: getattr(emat, k).copy() for k in db.HostEmat.FIELDS_I32 + db.HostEmat.FIELDS_U8 + db.HostEmat.FIELDS_F64})
    n = e.num_nodes
    nodes = []
    if codes_and_missations:
        with_muts = [v for v in range(n) if e.mut_off[v + 1] > e.mut_off[v] and v != e.root]
        with_miss = [v for v in range(n) if e.miss_off[v + 1] > e.miss_off[v]]
        for v in rng.choice(with_muts, 6, replace=False):
            i = int(e.mut_off[v])
            e.mut_to[i] = (int(e.mut_from[i]) + 1 + int(rng.integers(3))) % 4
            nodes.append(int(v))
        L = int(e.miss_end.max()) if len(e.miss_end) else 1
        for v in rng.choice(with_miss, 6, replace=False):
            i = int(e.miss_off[v])
            s0 = int(e.miss_start[i])
            e.miss_end[i] = min(L, s0 + 1 + int(rng.integers(40)))
            if i + 1 < int(e.miss_off[v + 1]):
                e.miss_end[i] = min(int(e.miss_end[i]), int(e.miss_start[i + 1]))
            nodes.append(int(v))
    else:
        tips = [v for v in range(n) if e.child0[v] < 0]
        for v in rng.choice(tips, 8, replace=False):
            e.t[v] += 0.25
            nodes.append(int(v))
    return e, sorted(set(nodes))


@pytest.mark.parametrize("codes_and_missations", [True, False])
def test_apply_rows_rebuilds_the_counts(orc, codes_and_missations):
    """dphy_forest_apply_rows re-flattens the edited trees: the folded evaluation afterwards == a fresh upload of the edited trees
    (bit for bit) == the oracle; the untouched trees keep their values."""
    items = [synth(3, seed=91), synth(0, seed=92, num_tips=800, caterpillar=1), synth(0, seed=93, num_partitions=2)]
    rng = np.random.default_rng(7 if codes_and_missations else 8)
    with db.Context(0) as c:
        tables = [db.DeviceSites(c, it[1]) for it in items]
        idx = np.arange(len(items))
        fo = db.Forest(c, [it[0] for it in items], tables, sites_index=idx)
        before = [_outputs(fo, k) for k in range(len(items))]
        edited = []
        rows = []
        for k in (0, 1):
            e, nodes = _edited(items[k][0], rng, codes_and_missations)
            edited.append(e)
            rows += [db.node_row(k, e, v) for v in nodes]
        fo.apply_rows(rows)
        fo.eval_log_G()
        fresh = db.Forest(c, edited + [items[2][0]], tables, sites_index=idx)
        fresh.eval_log_G()
        for k in range(len(items)):
            got, want = _outputs(fo, k), _outputs(fresh, k)
            assert got[:3] == want[:3]
            assert np.array_equal(got[3], want[3])
            if k < 2:
                e, s = to_oracle(edited[k], items[k][1])
                lam_o = orc.lambda_i(e, s)
                assert rel_err(got[3], lam_o) <= RTOL
                assert got[1] == pytest.approx(orc.log_G_below_root(e, s, lam_o), rel=RTOL)
                assert got[0] == pytest.approx(orc.log_root_prior(e, s), rel=RTOL)
            else:
                assert got[:3] == before[k][:3] and np.array_equal(got[3], before[k][3])
        fo.close(); fresh.close()
        for t in tables:
            t.close()
