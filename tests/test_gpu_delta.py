"""Device-resident incremental edits (dphy_forest_apply_rows; SURVEY.md section 8f row 1): a forest patched row by row must equal a
fresh upload of the edited trees -- integers (nsmn, num_muts*, SPR regions and their order) bit for bit, log G / lambda_i to
1e-12 -- after 1,000 random edits of the kinds the reference's local moves make: node displacements (core/subrun.cpp:223-231),
branch reforms (one branch's mutation list rewritten, :316-319) and SPR regrafts (topology + times around P,
core/spr_move.cpp:1101-1156), including regrafts that change the root."""
import copy

import numpy as np
import pytest

import delphy_b200 as db
from helpers import synth

pytestmark = pytest.mark.gpu
F = db.HostEmat.FIELDS_I32 + db.HostEmat.FIELDS_U8 + db.HostEmat.FIELDS_F64


class Editable:
    """A HostEmat as python lists per node, so that edits are easy; rebuilds the flat arrays on demand."""

    def __init__(self, emat):
        n = emat.num_nodes
        self.root = emat.root
        self.includes_run_root = emat.includes_run_root
        self.parent = emat.parent.copy(); self.child0 = emat.child0.copy(); self.child1 = emat.child1.copy(); self.t = emat.t.copy()
        sl = lambda off, a, v: a[off[v]:off[v + 1]].copy()
        self.muts = [[sl(emat.mut_off, a, v) for a in (emat.mut_site, emat.mut_from, emat.mut_to, emat.mut_t)] for v in range(n)]
        self.miss = [[sl(emat.miss_off, a, v) for a in (emat.miss_start, emat.miss_end)] for v in range(n)]
        self.fs = [[sl(emat.fs_off, a, v) for a in (emat.fs_site, emat.fs_from)] for v in range(n)]

    def flat(self):
        n = len(self.parent)
        cat = lambda rows, k, dt: np.concatenate([r[k] for r in rows]).astype(dt) if n else np.zeros(0, dt)
        off = lambda rows: np.concatenate([[0], np.cumsum([len(r[0]) for r in rows])]).astype(np.int32)
        return db.HostEmat(self.root, self.includes_run_root, parent=self.parent, child0=self.child0, child1=self.child1, t=self.t,
                           mut_off=off(self.muts), mut_site=cat(self.muts, 0, np.int32), mut_from=cat(self.muts, 1, np.uint8),
                           mut_to=cat(self.muts, 2, np.uint8), mut_t=cat(self.muts, 3, np.float64),
                           miss_off=off(self.miss), miss_start=cat(self.miss, 0, np.int32), miss_end=cat(self.miss, 1, np.int32),
                           fs_off=off(self.fs), fs_site=cat(self.fs, 0, np.int32), fs_from=cat(self.fs, 1, np.uint8))

    def row(self, tree, v):
        m, i, f = self.muts[v], self.miss[v], self.fs[v]
        keep = [np.ascontiguousarray(a) for a in (m[0].astype(np.int32), m[1].astype(np.uint8), m[2].astype(np.uint8), m[3].astype(np.float64),
                                                  i[0].astype(np.int32), i[1].astype(np.int32), f[0].astype(np.int32), f[1].astype(np.uint8))]
        P = lambda a, ty: a.ctypes.data_as(ty)
        r = db.NodeRow(tree, v, int(self.parent[v]), int(self.child0[v]), int(self.child1[v]), len(m[0]), len(i[0]), len(f[0]), float(self.t[v]),
                       P(keep[0], db.i32p), P(keep[1], db.u8p), P(keep[2], db.u8p), P(keep[3], db.f64p), P(keep[4], db.i32p), P(keep[5], db.i32p),
                       P(keep[6], db.i32p), P(keep[7], db.u8p))
        r._keep = keep
        return r

    def is_ancestor(self, a, v):
        while v >= 0:
            if v == a:
                return True
            v = int(self.parent[v])
        return False

    def retime_muts(self, v, rng):
        """mutation times of branch v redrawn inside [t_parent, t_v], sorted"""
        k = len(self.muts[v][0])
        if k and self.parent[v] >= 0:
            lo, hi = self.t[self.parent[v]], self.t[v]
            self.muts[v][3] = np.sort(lo + (hi - lo) * rng.random(k))

    # ---- the three kinds of edit; each returns the set of nodes whose rows changed ----
    def displace(self, rng):
        v = int(rng.integers(len(self.parent)))
        if self.child0[v] < 0 or v == self.root:
            return set()
        lo = self.t[self.parent[v]]
        hi = min(self.t[self.child0[v]], self.t[self.child1[v]])
        self.t[v] = lo + (hi - lo) * (0.1 + 0.8 * rng.random())
        touched = {v, int(self.child0[v]), int(self.child1[v])}
        for u in touched:
            self.retime_muts(u, rng)
        return touched

    def reform(self, rng, L):
        v = int(rng.integers(len(self.parent)))
        if v == self.root:
            return set()
        k = int(rng.integers(0, 5))
        sites = rng.choice(L, size=k, replace=False) if k else np.zeros(0, int)
        fr = rng.integers(0, 4, size=k)
        to = (fr + 1 + rng.integers(0, 3, size=k)) % 4
        self.muts[v] = [sites.astype(np.int32), fr.astype(np.uint8), to.astype(np.uint8), np.zeros(k)]
        self.retime_muts(v, rng)
        return {v}

    def spr(self, rng):
        n = len(self.parent)
        X = int(rng.integers(n))
        if X == self.root:
            return set()
        P = int(self.parent[X])
        S = int(self.child1[P]) if self.child0[P] == X else int(self.child0[P])
        G = int(self.parent[P])
        for _ in range(20):
            S2 = int(rng.integers(n))
            if S2 in (X, P) or self.is_ancestor(X, S2) or self.t[self.parent[S2] if self.parent[S2] >= 0 else S2] >= self.t[X]:
                continue
            break
        else:
            return set()
        touched = {X, P, S}
        # detach P: S takes P's place below G
        if G >= 0:
            if self.child0[G] == P: self.child0[G] = S
            else: self.child1[G] = S
            touched.add(G)
        else:
            self.root = S
        self.parent[S] = G
        # S inherits P's branch contents (mutations first P's then S's), as Tree_editing_session does when P slides off
        self.muts[S] = [np.concatenate([self.muts[P][k], self.muts[S][k]]) for k in range(4)]
        self.muts[P] = [np.zeros(0, np.int32), np.zeros(0, np.uint8), np.zeros(0, np.uint8), np.zeros(0)]
        # regraft P above S2
        G2 = int(self.parent[S2])
        hi = min(self.t[X], self.t[S2])
        lo = self.t[G2] if G2 >= 0 else hi - 1.0
        if not lo < hi:
            lo = hi - 1e-3
        self.t[P] = lo + (hi - lo) * (0.2 + 0.6 * rng.random())
        self.parent[P] = G2
        if G2 >= 0:
            if self.child0[G2] == S2: self.child0[G2] = P
            else: self.child1[G2] = P
            touched.add(G2)
        else:
            self.root = P
        self.child0[P], self.child1[P] = (X, S2) if rng.random() < 0.5 else (S2, X)
        self.parent[S2] = P; self.parent[X] = P
        touched.add(S2)
        self.parent[self.root] = -1
        # the root carries no timed mutations: move whatever the new root has onto t = -DBL_MAX "root mutations"
        for u in touched | {self.root}:
            if u == self.root:
                self.muts[u][3] = np.full(len(self.muts[u][0]), -np.finfo(float).max)
                touched.add(u)
            else:
                self.retime_muts(u, rng)
        return touched


def _compare(ctx, fo, emats, tables, sites_index, infos, rng):
    fresh = db.Forest(ctx, emats, tables, sites_index=sites_index)
    a, b = fo.log_G(), fresh.log_G()
    for x, y in zip(a, b):
        np.testing.assert_allclose(x, y, rtol=1e-12, atol=1e-9)
    ta, tb = fo.tallies(), fresh.tallies()
    for k in range(len(emats)):
        assert ta[k]["num_muts"] == tb[k]["num_muts"]
        np.testing.assert_array_equal(ta[k]["num_muts_ab"], tb[k]["num_muts_ab"])
        assert ta[k]["T"] == pytest.approx(tb[k]["T"], rel=1e-12)
        np.testing.assert_array_equal(fo.num_sites_missing(k), fresh.num_sites_missing(k))
        np.testing.assert_allclose(fo.lambda_i(k), fresh.lambda_i(k), rtol=1e-12, atol=1e-9)
        np.testing.assert_allclose(fo.Ttwiddle_beta_a(k), fresh.Ttwiddle_beta_a(k), rtol=1e-12)
    # a full SPR study on each tree: regions and their order bit for bit
    reqs = []
    for k, e in enumerate(emats):
        lam = fresh.lambda_i(k)
        xs = [int(v) for v in rng.permutation(e.num_nodes) if v != e.root and e.parent[v] != e.root and lam[v] > 0][:2]
        reqs += db.spr_requests_for_attached(e, k, xs, lam, infos[k]["t_max_tip"])
    ba, bb = fo.spr_study_batch(reqs), fresh.spr_study_batch(reqs)
    for i in range(len(reqs)):
        ra, rb = ba.regions(i), bb.regions(i)
        assert len(ra) == len(rb)
        for key in ("branch", "mut_idx", "min_muts", "t_min", "t_max"):
            np.testing.assert_array_equal(ra[key], rb[key], err_msg=key)
        np.testing.assert_allclose(ra["W_over_Wmax"], rb["W_over_Wmax"], rtol=1e-12, atol=1e-300)
    ba.close(); bb.close(); fresh.close()


def test_a_thousand_random_edits_match_fresh_uploads():
    rng = np.random.default_rng(2026)
    items = [synth(1), synth(0, seed=77, num_tips=120, num_partitions=2, num_root_mutations=3), synth(3, num_tips=1500)]
    with db.Context(0) as ctx:
        tables = [db.DeviceSites(ctx, it[1]) for it in items]
        infos = [it[2] for it in items]
        eds = [Editable(it[0]) for it in items]
        sidx = np.arange(len(items))
        fo = db.Forest(ctx, [e.flat() for e in eds], tables, sites_index=sidx)
        fo.eval_log_G()
        total = 0
        for rnd in range(25):
            rows, roots_changed = [], False
            for _ in range(40):
                k = int(rng.integers(len(eds)))
                ed = eds[k]
                kind = rng.random()
                old_root = ed.root
                touched = ed.displace(rng) if kind < 0.45 else (ed.reform(rng, items[k][1].num_sites) if kind < 0.8 else ed.spr(rng))
                roots_changed |= ed.root != old_root
                total += 1 if touched else 0
                # a node edited twice in one batch: send its latest row once
                rows = [r for r in rows if (r.tree, r.node) not in {(k, v) for v in touched}]
                rows += [ed.row(k, v) for v in sorted(touched)]
            fo.apply_rows(rows, new_roots=[e.root for e in eds])
            if rnd % 5 == 4 or rnd == 0:
                _compare(ctx, fo, [e.flat() for e in eds], tables, sidx, infos, rng)
        assert total >= 700
        _compare(ctx, fo, [e.flat() for e in eds], tables, sidx, infos, rng)
        # node times set through the dedicated entry point survive a later row edit
        ed = eds[0]
        v = next(v for v in range(len(ed.parent)) if ed.child0[v] >= 0 and v != ed.root)
        ed.t[v] = 0.5 * (ed.t[ed.parent[v]] + min(ed.t[ed.child0[v]], ed.t[ed.child1[v]]))
        fo.set_node_times(0, [v], [ed.t[v]])
        touched = set()
        while not touched:
            touched = ed.reform(rng, items[0][1].num_sites)
        touched -= {v, int(ed.child0[v]), int(ed.child1[v])}
        if touched:
            fo.apply_rows([ed.row(0, u) for u in touched])
            np.testing.assert_allclose(fo.log_G()[2], db.Forest(ctx, [e.flat() for e in eds], tables, sites_index=sidx).log_G()[2], rtol=1e-12)
        # a broken edit is rejected and leaves the forest as it was
        before = fo.log_G()[2].copy()
        bad = ed.row(0, v)
        bad.parent = int(ed.child0[v])            # a cycle
        with pytest.raises(db.DphyError):
            fo.apply_rows([bad])
        np.testing.assert_array_equal(fo.log_G()[2], before)
        fo.close()
        for t in tables:
            t.close()


def test_a_refused_call_changes_no_list_length():
    """A call refused at a later tree (an out-of-range new root for tree 1) after tree 0's row was read must leave the forest's
    record of tree 0's list lengths as it was: the same row sent again alone then builds exactly the edited forest.  The row
    shortens a mutation list, so a length recorded by the refused call would size the rebuild for more mutations than it gets."""
    rng = np.random.default_rng(31)
    items = [synth(1), synth(0, seed=77, num_tips=120)]
    with db.Context(0) as ctx:
        tables = [db.DeviceSites(ctx, it[1]) for it in items]
        eds = [Editable(it[0]) for it in items]
        sidx = np.arange(len(items))
        fo = db.Forest(ctx, [e.flat() for e in eds], tables, sites_index=sidx)
        for _ in range(10000):                      # a reform may keep or grow the list: draw until one shortens it
            ed = copy.deepcopy(eds[0])
            touched = ed.reform(rng, items[0][1].num_sites)
            if touched and len(ed.muts[min(touched)][0]) < len(eds[0].muts[min(touched)][0]):
                break
        else:
            pytest.fail("no shortening reform drawn")
        v = min(touched)
        eds[0] = ed
        with pytest.raises(db.DphyError):
            fo.apply_rows([ed.row(0, v)], new_roots=[ed.root, len(eds[1].parent)])
        fo.apply_rows([ed.row(0, v)], new_roots=[e.root for e in eds])
        fresh = db.Forest(ctx, [e.flat() for e in eds], tables, sites_index=sidx)
        for k in range(len(eds)):
            got, want = fo.download_tree(k), fresh.download_tree(k)
            assert got.root == want.root
            for f in F:
                np.testing.assert_array_equal(getattr(got, f), getattr(want, f), err_msg=f"tree {k}: {f}")
        np.testing.assert_allclose(fo.log_G()[2], fresh.log_G()[2], rtol=1e-12, atol=0)
        fresh.close()
        fo.close()
        for t in tables:
            t.close()
