"""Shared helpers for the parity tests: synthetic EMATs (product-side generator) -> oracle structs."""
from __future__ import annotations

import copy
import functools

import numpy as np

import delphy_b200 as db
from oracle_lib import Emat, Sites


def to_oracle(emat: db.HostEmat, sites: db.HostSites):
    e = Emat(emat.root, emat.parent, emat.child0, emat.child1, emat.t, emat.mut_off, emat.mut_site, emat.mut_from,
             emat.mut_to, emat.mut_t, emat.miss_off, emat.miss_start, emat.miss_end, emat.fs_off, emat.fs_site,
             emat.fs_from, emat.includes_run_root)
    s = Sites(sites.ref, sites.partition_for_site, sites.nu_l, sites.mu, sites.pi_a, sites.q_ab)
    return e, s


def from_oracle(e: Emat, s: Sites):
    emat = db.HostEmat(e.root, e.includes_run_root, parent=e.parent, child0=e.child0, child1=e.child1, t=e.t,
                       mut_off=e.mut_off, mut_site=e.mut_site, mut_from=e.mut_from, mut_to=e.mut_to, mut_t=e.mut_t,
                       miss_off=e.miss_off, miss_start=e.miss_start, miss_end=e.miss_end, fs_off=e.fs_off,
                       fs_site=e.fs_site, fs_from=e.fs_from)
    sites = db.HostSites(s.ref, s.partition_for_site, s.nu_l, s.mu, s.pi_a, s.q_ab)
    return emat, sites


@functools.lru_cache(maxsize=32)
def _synth_cached(config=0, **overrides):
    p = db.synth_params(config, **overrides)
    return db.synth_generate(p)


def synth(config=0, **overrides):
    """(HostEmat, HostSites, info) of a synthetic shape.  Generated once, but every call gets its own copy: tests edit
    trees and models in place, and must not change what a later test in the same process is given."""
    return copy.deepcopy(_synth_cached(config, **overrides))


def rel_err(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    denom = np.maximum(np.abs(b), 1e-300)
    return float(np.max(np.abs(a - b) / denom)) if a.size else 0.0


# ---- delphy.api.Tree (core/api.fbs) test material -----------------------------------------------------------------------------------
# name -> (synthetic config, overrides): the trees behind tests/golden/api_tree_*.bin (written by the reference's own writer,
# tests/golden/make_api_tree_fixtures.py); few sites so that the reference sequence does not dominate the fixture
API_TREE_CASES = {
    "small": (0, dict(num_tips=40, num_sites=3000, muts_per_tip=3.0)),
    "missing_heavy": (5, dict(num_tips=60, num_sites=6000, muts_per_tip=6.0, num_partitions=1)),
    "root_muts": (2, dict(num_tips=50, num_sites=2500, muts_per_tip=4.0, num_root_mutations=7)),
}
EMAT_FIELDS = ["parent", "child0", "child1", "t", "mut_off", "mut_site", "mut_from", "mut_to", "mut_t", "miss_off", "miss_start", "miss_end",
               "fs_off", "fs_site", "fs_from"]


def assert_same_emat(a, b, float32_times_of_b=False):
    """Every array of two flat EMATs bit for bit (b's times first rounded to float32 when the other went through the wire format)."""
    assert int(a.root) == int(b.root)
    for f in EMAT_FIELDS:
        x, y = np.asarray(getattr(a, f)), np.asarray(getattr(b, f))
        if float32_times_of_b and f in ("t", "mut_t"):
            with np.errstate(over="ignore"):          # the root's rereferencing "mutations" sit at -DBL_MAX: -inf as float32, as in the reference
                y = y.astype(np.float32).astype(np.float64)
        assert x.shape == y.shape and np.array_equal(x, y), f


def with_extra_intervals(e: Emat, extra: dict) -> Emat:
    """A copy of `e` with extra missation intervals {node: [(start, end), ...]} merged (sorted) into the nodes' lists; from_states untouched."""
    n = e.num_nodes
    starts, ends, off = [], [], [0]
    for v in range(n):
        iv = [(int(e.miss_start[k]), int(e.miss_end[k])) for k in range(e.miss_off[v], e.miss_off[v + 1])] + list(extra.get(v, []))
        iv.sort()
        starts += [a for a, _ in iv]; ends += [b for _, b in iv]
        off.append(len(starts))
    return Emat(e.root, e.parent, e.child0, e.child1, e.t, e.mut_off, e.mut_site, e.mut_from, e.mut_to, e.mut_t,
                off, starts, ends, e.fs_off, e.fs_site, e.fs_from, e.includes_run_root)


def free_site_for(e: Emat, nodes, L, avoid_sites=()):
    """A site l such that [l, l+1) touches no missation interval of `nodes` nor of their ancestors / subtrees' roots given, and is not in avoid_sites."""
    taken = np.zeros(L + 2, bool)
    for v in nodes:
        a = v
        while a >= 0:
            for k in range(e.miss_off[a], e.miss_off[a + 1]):
                taken[max(int(e.miss_start[k]) - 1, 0):int(e.miss_end[k]) + 1] = True
            a = int(e.parent[a])
    for l in avoid_sites:
        taken[l] = True
    free = np.flatnonzero(~taken[:L])
    assert free.size
    return int(free[free.size // 2])
