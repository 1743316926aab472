"""delphy_b200 -- B200-native EMAT log-G + SPR-regraft engine (Python harness over the C ABI).

The product is ``libdelphy_b200.so`` (hand-written sm_100a CUDA behind ``include/delphy_b200.h``); the drop-in for
the reference is the C++ adapter described in INTEGRATION.md.  This module is the thin ctypes binding the tests and
bench.py use to drive that same C ABI.  It never imports anything from ``oracle/`` and has no CPU fallback: creating a
:class:`Context` without a usable CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdelphy_b200.so")
SYNTH_LIB_PATH = os.path.join(_HERE, "libdphy_synth.so")   # input generator only: no product code, no CUDA

i32p = C.POINTER(C.c_int32)
u8p = C.POINTER(C.c_uint8)
f64p = C.POINTER(C.c_double)


class DphyError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__(f"delphy_b200 status {status}: {msg}")
        self.status = status


DPHY_OK, ERR_INVALID_ARGUMENT, ERR_OUT_OF_RANGE, ERR_CUDA, ERR_OOM, ERR_INTERNAL = 0, -1, -2, -3, -4, -5
INT32_MAX = 2**31 - 1


class EmatHost(C.Structure):
    _fields_ = [
        ("num_nodes", C.c_int32), ("root", C.c_int32), ("includes_run_root", C.c_int32), ("reserved", C.c_int32),
        ("parent", i32p), ("child0", i32p), ("child1", i32p), ("t", f64p),
        ("mut_off", i32p), ("mut_site", i32p), ("mut_from", u8p), ("mut_to", u8p), ("mut_t", f64p),
        ("miss_off", i32p), ("miss_start", i32p), ("miss_end", i32p),
        ("fs_off", i32p), ("fs_site", i32p), ("fs_from", u8p),
    ]


class SitesHost(C.Structure):
    _fields_ = [
        ("num_sites", C.c_int32), ("num_partitions", C.c_int32),
        ("ref", u8p), ("partition_for_site", i32p), ("nu_l", f64p),
        ("mu", f64p), ("pi_a", f64p), ("q_ab", f64p),
    ]


class CandidateRegion(C.Structure):
    _fields_ = [
        ("branch", C.c_int32), ("mut_idx", C.c_int32), ("t_min", C.c_double), ("t_max", C.c_double),
        ("min_muts", C.c_int32), ("pad_", C.c_int32), ("log_W_over_Wmax", C.c_double), ("W_over_Wmax", C.c_double),
    ]


REGION_DTYPE = np.dtype([
    ("branch", "<i4"), ("mut_idx", "<i4"), ("t_min", "<f8"), ("t_max", "<f8"),
    ("min_muts", "<i4"), ("pad_", "<i4"), ("log_W_over_Wmax", "<f8"), ("W_over_Wmax", "<f8"),
])


class SprRequest(C.Structure):
    _fields_ = [
        ("tree", C.c_int32), ("X", C.c_int32), ("t_X", C.c_double),
        ("start_branch", C.c_int32), ("start_mut_idx", C.c_int32),
        ("init_min_muts", C.c_int32), ("max_muts_from_start", C.c_int32),
        ("can_change_root", C.c_int32), ("x_state_mode", C.c_int32),
        ("lambda_X", C.c_double), ("annealing_factor", C.c_double), ("t_max_tip", C.c_double),
        ("n_x_deltas", C.c_int32), ("x_delta_site", i32p), ("x_delta_to", u8p),
        ("n_x_missing", C.c_int32), ("x_missing_start", i32p), ("x_missing_end", i32p),
    ]


class SampleSet(C.Structure):
    _fields_ = [("num_samples", C.c_int32), ("reserved", C.c_int32), ("delta_off", i32p), ("delta_site", i32p), ("delta_to", u8p),
                ("miss_off", i32p), ("miss_start", i32p), ("miss_end", i32p)]


class Placement(C.Structure):
    _fields_ = [("min_muts", C.c_int32), ("num_best", C.c_int32), ("branch", C.c_int32), ("mut_idx", C.c_int32)]


PLACEMENT_DTYPE = np.dtype([("min_muts", "<i4"), ("num_best", "<i4"), ("branch", "<i4"), ("mut_idx", "<i4")])


class SprWeightParams(C.Structure):
    _fields_ = [("lambda_X", C.c_double), ("annealing_factor", C.c_double), ("t_max_tip", C.c_double)]


SPR_X_FROM_TREE, SPR_X_REL_REF, SPR_X_REL_START = 0, 1, 2


class NodeRow(C.Structure):
    _fields_ = [
        ("tree", C.c_int32), ("node", C.c_int32), ("parent", C.c_int32), ("child0", C.c_int32), ("child1", C.c_int32),
        ("n_muts", C.c_int32), ("n_miss", C.c_int32), ("n_fs", C.c_int32), ("t", C.c_double),
        ("mut_site", i32p), ("mut_from", u8p), ("mut_to", u8p), ("mut_t", f64p),
        ("miss_start", i32p), ("miss_end", i32p), ("fs_site", i32p), ("fs_from", u8p),
    ]


def node_row(tree: int, emat: "HostEmat", v: int) -> NodeRow:
    """The row of node v as `emat` (already edited on the host) has it."""
    m0, m1 = int(emat.mut_off[v]), int(emat.mut_off[v + 1])
    i0, i1 = int(emat.miss_off[v]), int(emat.miss_off[v + 1])
    f0, f1 = int(emat.fs_off[v]), int(emat.fs_off[v + 1])
    keep = [np.ascontiguousarray(a) for a in (emat.mut_site[m0:m1], emat.mut_from[m0:m1], emat.mut_to[m0:m1], emat.mut_t[m0:m1],
                                              emat.miss_start[i0:i1], emat.miss_end[i0:i1], emat.fs_site[f0:f1], emat.fs_from[f0:f1])]
    r = NodeRow(tree, v, int(emat.parent[v]), int(emat.child0[v]), int(emat.child1[v]), m1 - m0, i1 - i0, f1 - f0, float(emat.t[v]),
                _p(keep[0], i32p), _p(keep[1], u8p), _p(keep[2], u8p), _p(keep[3], f64p), _p(keep[4], i32p), _p(keep[5], i32p),
                _p(keep[6], i32p), _p(keep[7], u8p))
    r._keep = keep
    return r


class SprSummary(C.Structure):
    _fields_ = [
        ("mu", C.c_double), ("log_Wmax", C.c_double), ("sum_W_over_Wmax", C.c_double),
        ("num_regions", C.c_int32), ("num_missing_at_X", C.c_int32), ("region_offset", C.c_int64),
    ]


class Tallies(C.Structure):
    _fields_ = [
        ("num_muts", C.c_int32), ("reserved", C.c_int32), ("num_muts_ab", C.c_int32 * 16),
        ("T", C.c_double), ("log_root_prior", C.c_double), ("log_G_below_root", C.c_double),
    ]


class ApiTreeView(C.Structure):
    """dphy_api_tree_view: where the vectors of a delphy.api.Tree buffer (core/api.fbs:13-49) lie."""
    _fields_ = [("num_nodes", C.c_int32), ("root", C.c_int32), ("num_sites", C.c_int32), ("reserved", C.c_int32),
                ("num_mutations", C.c_int64), ("num_missation_intervals", C.c_int64),
                ("nodes", C.c_void_p), ("mutations", C.c_void_p), ("missation_intervals", C.c_void_p), ("ref_seq", C.c_void_p)]


class TreeCounts(C.Structure):
    _fields_ = [("num_nodes", C.c_int32), ("root", C.c_int32), ("num_mutations", C.c_int64),
                ("num_missation_intervals", C.c_int64), ("num_from_states", C.c_int64)]


def _bytes_ptr(data: bytes) -> C.c_void_p:
    """address of a bytes object's buffer (no copy; the caller keeps `data` alive)"""
    return C.cast(C.c_char_p(data), C.c_void_p)


def api_tree_parse(data: bytes) -> dict:
    """dphy_api_tree_parse (host only): the sizes, the root and the reference sequence of a delphy.api.Tree buffer."""
    data = bytes(data)
    v = ApiTreeView()
    st = lib().dphy_api_tree_parse(_bytes_ptr(data) if len(data) else None, len(data), C.byref(v))
    if st != DPHY_OK:
        raise DphyError(st, "malformed delphy.api.Tree buffer")
    ref = np.ctypeslib.as_array(C.cast(v.ref_seq, u8p), shape=(max(v.num_sites, 1),))[:v.num_sites].copy() if v.num_sites else np.zeros(0, np.uint8)
    return dict(num_nodes=v.num_nodes, root=v.root, num_sites=v.num_sites, num_mutations=int(v.num_mutations),
                num_missation_intervals=int(v.num_missation_intervals), ref_seq=ref)


class MapleView(C.Structure):
    _fields_ = [("num_sites", C.c_int32), ("num_tips", C.c_int32), ("num_warnings", C.c_int64),
                ("ref", u8p), ("t_min", f64p), ("t_max", f64p), ("name_off", C.POINTER(C.c_int64)), ("names", C.c_void_p),
                ("delta_off", i32p), ("delta_site", i32p), ("delta_from", u8p), ("delta_to", u8p),
                ("miss_off", i32p), ("miss_start", i32p), ("miss_end", i32p)]


def maple_parse(text: bytes) -> dict:
    """dphy_maple_parse (host only): read_maple (core/io.cpp:98-254) straight to CSR arrays.  Raises DphyError where the reference throws."""
    text = bytes(text)
    h = C.c_void_p()
    st = lib().dphy_maple_parse(text, len(text), C.byref(h))
    if st != DPHY_OK:
        raise DphyError(st, lib().dphy_maple_last_error().decode(errors="replace"))
    try:
        v = MapleView()
        lib().dphy_maple_get(h, C.byref(v))
        n, L = v.num_tips, v.num_sites
        name_off = _np_from(v.name_off, n + 1, np.int64)
        names_raw = C.string_at(v.names, int(name_off[-1])) if n and name_off[-1] else b""
        delta_off = _np_from(v.delta_off, n + 1, np.int32); miss_off = _np_from(v.miss_off, n + 1, np.int32)
        D, I = int(delta_off[-1]), int(miss_off[-1])
        return dict(num_warnings=int(v.num_warnings), ref=_np_from(v.ref, L, np.uint8), t_min=_np_from(v.t_min, n, np.float64),
                    t_max=_np_from(v.t_max, n, np.float64), names=[names_raw[name_off[k]:name_off[k + 1]] for k in range(n)],
                    delta_off=delta_off, delta_site=_np_from(v.delta_site, D, np.int32), delta_from=_np_from(v.delta_from, D, np.uint8),
                    delta_to=_np_from(v.delta_to, D, np.uint8), miss_off=miss_off, miss_start=_np_from(v.miss_start, I, np.int32),
                    miss_end=_np_from(v.miss_end, I, np.int32))
    finally:
        lib().dphy_maple_free(h)


class _ApiTreeShape:
    def __init__(self, num_nodes):
        self.num_nodes = num_nodes


class SynthParams(C.Structure):
    _fields_ = [
        ("num_tips", C.c_int32), ("num_sites", C.c_int32), ("seed", C.c_uint64),
        ("muts_per_tip", C.c_double), ("tip_date_span_years", C.c_double), ("growth_rate", C.c_double),
        ("n0_years", C.c_double), ("kappa", C.c_double), ("pi", C.c_double * 4),
        ("site_rate_heterogeneity", C.c_int32), ("gamma_alpha", C.c_double), ("num_partitions", C.c_int32),
        ("missing_mean_intervals_per_tip", C.c_double), ("missing_len_min", C.c_double), ("missing_len_max", C.c_double),
        ("end_gaps", C.c_int32), ("num_root_mutations", C.c_int32), ("caterpillar", C.c_int32),
    ]


class SynthEmat(C.Structure):
    _fields_ = [
        ("emat", EmatHost), ("sites", SitesHost), ("mu_used", C.c_double), ("t_max_tip", C.c_double),
        ("num_mutations", C.c_int64), ("num_intervals", C.c_int64), ("num_from_states", C.c_int64),
        ("num_missing_sites", C.c_int64), ("max_depth", C.c_int32), ("owner_", C.c_void_p),
    ]


def build(force: bool = False) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    src = os.path.join(_HERE, "csrc")
    args = ["make", "-s", "-C", src]
    if force:
        subprocess.run(args + ["clean"], check=True)
    subprocess.run(args, check=True)
    return LIB_PATH


_LIB = None
_SYNTH_LIB = None


def _bind_partition(L):
    vp = C.c_void_p
    L.dphy_partition_generate_stencil.argtypes = [C.POINTER(EmatHost), C.c_int32, C.c_uint64, i32p, i32p]
    L.dphy_partition_split.argtypes = [C.POINTER(EmatHost), C.POINTER(SitesHost), C.c_int32, i32p, C.POINTER(vp)]
    L.dphy_partition_num_parts.argtypes = [vp]; L.dphy_partition_num_parts.restype = C.c_int32
    L.dphy_partition_part.argtypes = [vp, C.c_int32]; L.dphy_partition_part.restype = C.POINTER(EmatHost)
    L.dphy_partition_orig_index.argtypes = [vp, C.c_int32]; L.dphy_partition_orig_index.restype = i32p
    L.dphy_partition_free.argtypes = [vp]; L.dphy_partition_free.restype = None
    L.dphy_partition_reassemble.argtypes = [vp, C.POINTER(EmatHost), C.c_int32, C.POINTER(EmatHost)]
    L.dphy_partition_reassemble.restype = C.POINTER(EmatHost)


def synth_lib() -> C.CDLL:
    """libdphy_synth.so: the synthetic-input generator (its own shared object, so that generating inputs loads no product code)."""
    global _SYNTH_LIB
    if _SYNTH_LIB is None:
        if not os.path.exists(SYNTH_LIB_PATH):
            raise FileNotFoundError(f"{SYNTH_LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'`")
        L = C.CDLL(SYNTH_LIB_PATH)
        L.dphy_synth_default_params.argtypes = [C.POINTER(SynthParams), C.c_int32]
        L.dphy_synth_default_params.restype = None
        L.dphy_synth_generate.argtypes = [C.POINTER(SynthParams), C.POINTER(C.POINTER(SynthEmat))]
        L.dphy_synth_free.argtypes = [C.POINTER(SynthEmat)]
        L.dphy_synth_free.restype = None
        _bind_partition(L)
        _SYNTH_LIB = L
    return _SYNTH_LIB


def lib() -> C.CDLL:
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.dphy_version.restype = C.c_char_p
    L.dphy_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.dphy_ctx_destroy.argtypes = [vp]
    L.dphy_last_error.argtypes = [vp]; L.dphy_last_error.restype = C.c_char_p
    L.dphy_ctx_synchronize.argtypes = [vp]
    L.dphy_ctx_join_side_streams.argtypes = [vp]
    L.dphy_arena_stats.argtypes = [vp, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    L.dphy_ctx_stream.argtypes = [vp]; L.dphy_ctx_stream.restype = vp
    L.dphy_ctx_launch_count.argtypes = [vp]; L.dphy_ctx_launch_count.restype = C.c_int64
    L.dphy_host_alloc.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
    L.dphy_host_free.argtypes = [vp, vp]; L.dphy_host_free.restype = None
    L.dphy_ctx_set_log_G_path.argtypes = [vp, C.c_int]
    L.dphy_sites_upload.argtypes = [vp, C.POINTER(SitesHost), C.POINTER(vp)]
    L.dphy_sites_destroy.argtypes = [vp, vp]
    L.dphy_sites_set_evo.argtypes = [vp, vp, f64p, f64p, f64p, f64p]
    L.dphy_sites_set_evo_many.argtypes = [vp, C.c_int32, C.POINTER(vp), C.POINTER(f64p), C.POINTER(f64p), C.POINTER(f64p)]
    L.dphy_calc_state_frequencies_per_partition.argtypes = [vp, vp, i32p]
    L.dphy_calc_cum_Q_l.argtypes = [vp, vp, f64p]
    L.dphy_forest_upload.argtypes = [vp, C.c_int32, C.POINTER(EmatHost), i32p, C.c_int32, C.POINTER(vp), C.POINTER(vp)]
    L.dphy_forest_destroy.argtypes = [vp, vp]
    L.dphy_forest_num_nodes.argtypes = [vp]; L.dphy_forest_num_nodes.restype = C.c_int64
    L.dphy_forest_device_bytes.argtypes = [vp]; L.dphy_forest_device_bytes.restype = C.c_int64
    L.dphy_forest_log_G_algorithmic_bytes.argtypes = [vp]; L.dphy_forest_log_G_algorithmic_bytes.restype = C.c_int64
    L.dphy_forest_set_node_times.argtypes = [vp, vp, C.c_int32, C.c_int32, i32p, f64p]
    L.dphy_forest_eval_log_G.argtypes = [vp, vp]
    L.dphy_forest_get_log_G.argtypes = [vp, vp, f64p, f64p, f64p]
    L.dphy_forest_get_lambda_i.argtypes = [vp, vp, C.c_int32, f64p]
    L.dphy_forest_get_num_sites_missing.argtypes = [vp, vp, C.c_int32, i32p]
    L.dphy_log_G_host.argtypes = [vp, C.POINTER(EmatHost), C.POINTER(SitesHost), f64p, f64p, f64p]
    L.dphy_forest_log_coalescent_prior.argtypes = [vp, vp, C.c_double, C.c_double, C.c_double, f64p]
    L.dphy_forest_calc_tallies.argtypes = [vp, vp, C.POINTER(Tallies)]
    L.dphy_forest_calc_num_muts_beta_ab.argtypes = [vp, vp, C.c_int32, i32p]
    L.dphy_forest_calc_num_muts_l.argtypes = [vp, vp, C.c_int32, i32p, i32p]
    L.dphy_forest_calc_Ttwiddle_beta_a.argtypes = [vp, vp, C.c_int32, f64p]
    L.dphy_forest_calc_Ttwiddle_l.argtypes = [vp, vp, C.c_int32, f64p, f64p]
    L.dphy_forest_calc_site_tallies.argtypes = [vp, vp, C.c_int64, f64p, i32p]
    L.dphy_spr_study_batch.argtypes = [vp, vp, C.c_int32, C.POINTER(SprRequest), C.POINTER(vp)]
    L.dphy_spr_batch_destroy.argtypes = [vp, vp]
    L.dphy_spr_batch_get_summaries.argtypes = [vp, vp, C.POINTER(SprSummary)]
    L.dphy_spr_batch_total_regions.argtypes = [vp, vp]; L.dphy_spr_batch_total_regions.restype = C.c_int64
    L.dphy_spr_batch_get_regions.argtypes = [vp, vp, C.c_int32, C.POINTER(CandidateRegion), C.c_int64]
    L.dphy_spr_batch_get_regions.restype = C.c_int64
    L.dphy_forest_apply_rows.argtypes = [vp, vp, C.c_int32, C.POINTER(NodeRow), i32p]
    L.dphy_sites_update.argtypes = [vp, vp, C.POINTER(SitesHost)]
    L.dphy_forest_cycle_tallies_device.argtypes = [vp, vp, vp, C.c_int32]
    L.dphy_spr_batch_set_weights.argtypes = [vp, vp, C.POINTER(SprWeightParams)]
    L.dphy_spr_batch_get_region_weights.argtypes = [vp, vp, C.c_int32, C.POINTER(CandidateRegion), C.c_int64]
    L.dphy_spr_batch_get_region_weights.restype = C.c_int64
    L.dphy_spr_batch_log_alpha_in_region.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_double, f64p]
    L.dphy_gamma_q.argtypes = [vp, C.c_int32, f64p, f64p, f64p]
    L.dphy_gamma_q_inv.argtypes = [vp, C.c_int32, f64p, f64p, f64p]
    L.dphy_spr_batch_pick_nexus_regions.argtypes = [vp, vp, f64p, i32p]
    L.dphy_spr_batch_find_region.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_double, i32p]
    L.dphy_api_tree_parse.argtypes = [vp, C.c_size_t, C.POINTER(ApiTreeView)]
    L.dphy_forest_upload_api_trees.argtypes = [vp, C.c_int32, C.POINTER(vp), C.POINTER(C.c_size_t), i32p, i32p, C.c_int32, C.POINTER(vp), C.c_uint32, C.POINTER(vp)]
    L.dphy_forest_write_api_tree.argtypes = [vp, vp, C.c_int32, vp, C.c_size_t]; L.dphy_forest_write_api_tree.restype = C.c_int64
    L.dphy_forest_tree_counts.argtypes = [vp, vp, C.c_int32, C.POINTER(TreeCounts)]
    L.dphy_forest_download_tree.argtypes = [vp, vp, C.c_int32, C.POINTER(EmatHost)]
    L.dphy_forest_place_samples.argtypes = [vp, vp, C.c_int32, C.POINTER(SampleSet), C.c_int32, C.c_int32, C.POINTER(Placement),
                                            C.POINTER(CandidateRegion)]
    L.dphy_forest_place_dated_samples.argtypes = [vp, vp, C.c_int32, C.POINTER(SampleSet), f64p, C.c_int32, C.c_int32,
                                                  C.POINTER(Placement), C.POINTER(CandidateRegion)]
    L.dphy_clade_table_create.argtypes = [vp, C.POINTER(vp)]
    L.dphy_clade_table_destroy.argtypes = [vp, vp]; L.dphy_clade_table_destroy.restype = None
    L.dphy_clade_table_add.argtypes = [vp, vp, vp]
    L.dphy_clade_table_info.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.dphy_clade_table_score.argtypes = [vp, vp, vp, f64p]
    L.dphy_clade_table_node_support.argtypes = [vp, vp, vp, C.c_int32, C.POINTER(C.c_int64), f64p]
    L.dphy_maple_parse.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(vp)]
    L.dphy_maple_get.argtypes = [vp, C.POINTER(MapleView)]
    L.dphy_maple_free.argtypes = [vp]; L.dphy_maple_free.restype = None
    L.dphy_maple_last_error.restype = C.c_char_p
    _bind_partition(L)
    _LIB = L
    return L


def _p(a, ty):
    return a.ctypes.data_as(ty)


def _np_from(ptr, n, dtype):
    if n == 0:
        return np.zeros(0, dtype)
    return np.ctypeslib.as_array(ptr, shape=(n,)).astype(dtype, copy=True)


class HostEmat:
    """Numpy-owned flat EMAT (host node order).  Field names follow include/delphy_b200.h."""
    FIELDS_I32 = ("parent", "child0", "child1", "mut_off", "mut_site", "miss_off", "miss_start", "miss_end", "fs_off", "fs_site")
    FIELDS_U8 = ("mut_from", "mut_to", "fs_from")
    FIELDS_F64 = ("t", "mut_t")

    def __init__(self, root, includes_run_root=1, **arrays):
        self.root = int(root)
        self.includes_run_root = int(includes_run_root)
        for k in self.FIELDS_I32:
            setattr(self, k, np.ascontiguousarray(arrays[k], np.int32))
        for k in self.FIELDS_U8:
            setattr(self, k, np.ascontiguousarray(arrays[k], np.uint8))
        for k in self.FIELDS_F64:
            setattr(self, k, np.ascontiguousarray(arrays[k], np.float64))

    @property
    def num_nodes(self):
        return int(self.parent.shape[0])

    def pinned(self, ctx) -> "HostEmat":
        """A copy whose arrays live in page-locked memory (dphy_host_alloc): dphy_forest_upload DMAs straight out of them."""
        arrays = {k: ctx.host_array_like(getattr(self, k)) for k in self.FIELDS_I32 + self.FIELDS_U8 + self.FIELDS_F64}
        return HostEmat(self.root, self.includes_run_root, **arrays)

    def as_struct(self) -> EmatHost:
        return EmatHost(self.num_nodes, self.root, self.includes_run_root, 0,
                        _p(self.parent, i32p), _p(self.child0, i32p), _p(self.child1, i32p), _p(self.t, f64p),
                        _p(self.mut_off, i32p), _p(self.mut_site, i32p), _p(self.mut_from, u8p), _p(self.mut_to, u8p),
                        _p(self.mut_t, f64p), _p(self.miss_off, i32p), _p(self.miss_start, i32p), _p(self.miss_end, i32p),
                        _p(self.fs_off, i32p), _p(self.fs_site, i32p), _p(self.fs_from, u8p))


class HostSites:
    def __init__(self, ref, partition_for_site, nu_l, mu, pi_a, q_ab):
        self.ref = np.ascontiguousarray(ref, np.uint8)
        self.partition_for_site = np.ascontiguousarray(partition_for_site, np.int32)
        self.nu_l = np.ascontiguousarray(nu_l, np.float64)
        self.mu = np.ascontiguousarray(mu, np.float64).reshape(-1)
        self.pi_a = np.ascontiguousarray(pi_a, np.float64).reshape(-1, 4)
        self.q_ab = np.ascontiguousarray(q_ab, np.float64).reshape(-1, 4, 4)

    @property
    def num_sites(self):
        return int(self.ref.shape[0])

    @property
    def num_partitions(self):
        return int(self.mu.shape[0])

    def as_struct(self) -> SitesHost:
        return SitesHost(self.num_sites, self.num_partitions, _p(self.ref, u8p), _p(self.partition_for_site, i32p),
                         _p(self.nu_l, f64p), _p(self.mu, f64p), _p(self.pi_a, f64p), _p(self.q_ab, f64p))


def _emat_from_struct(e: EmatHost) -> HostEmat:
    N = e.num_nodes
    M = int(e.mut_off[N]); I = int(e.miss_off[N]); F = int(e.fs_off[N])
    return HostEmat(
        e.root, e.includes_run_root,
        parent=_np_from(e.parent, N, np.int32), child0=_np_from(e.child0, N, np.int32), child1=_np_from(e.child1, N, np.int32),
        t=_np_from(e.t, N, np.float64),
        mut_off=_np_from(e.mut_off, N + 1, np.int32), mut_site=_np_from(e.mut_site, M, np.int32),
        mut_from=_np_from(e.mut_from, M, np.uint8), mut_to=_np_from(e.mut_to, M, np.uint8), mut_t=_np_from(e.mut_t, M, np.float64),
        miss_off=_np_from(e.miss_off, N + 1, np.int32), miss_start=_np_from(e.miss_start, I, np.int32), miss_end=_np_from(e.miss_end, I, np.int32),
        fs_off=_np_from(e.fs_off, N + 1, np.int32), fs_site=_np_from(e.fs_site, F, np.int32), fs_from=_np_from(e.fs_from, F, np.uint8))


def partition_emat(emat: HostEmat, sites: HostSites, num_parts: int, seed: int = 1):
    """Cut `emat` into <= num_parts independent parts (the reference's Run::repartition).  Returns
    (list of HostEmat parts, list of orig_tree_index arrays, cut_points); the last part holds the tree's root."""
    L = lib()
    es, ss = emat.as_struct(), sites.as_struct()
    cuts = np.zeros(max(num_parts, 1), np.int32)
    ncut = C.c_int32(0)
    st = L.dphy_partition_generate_stencil(C.byref(es), num_parts, seed, _p(cuts, i32p), C.byref(ncut))
    if st != DPHY_OK:
        raise DphyError(st, "dphy_partition_generate_stencil")
    h = C.c_void_p()
    st = L.dphy_partition_split(C.byref(es), C.byref(ss), ncut.value, _p(cuts, i32p), C.byref(h))
    if st != DPHY_OK:
        raise DphyError(st, "dphy_partition_split")
    try:
        parts, origs = [], []
        for i in range(L.dphy_partition_num_parts(h)):
            pe = L.dphy_partition_part(h, i).contents
            parts.append(_emat_from_struct(pe))
            origs.append(_np_from(L.dphy_partition_orig_index(h, i), pe.num_nodes, np.int32))
        return parts, origs, cuts[:ncut.value].copy()
    finally:
        L.dphy_partition_free(h)


class Partition:
    """A tree cut into parts that can be edited independently and merged back (Run::repartition / Run::reassemble,
    core/run.cpp:110-256).  parts[i] are HostEmat copies; origs[i] = orig_tree_index of every node of part i."""

    def __init__(self, emat: HostEmat, sites: HostSites, num_parts: int = 0, seed: int = 1, cut_points=None, host_only=False):
        # host_only: use the copy of the (host-only) tree cutter inside libdphy_synth.so, so that no product library is loaded
        L = synth_lib() if host_only else lib()
        self._L = L
        self.emat = emat
        es, ss = emat.as_struct(), sites.as_struct()
        if cut_points is None:
            cuts = np.zeros(max(num_parts, 1), np.int32)
            ncut = C.c_int32(0)
            st = L.dphy_partition_generate_stencil(C.byref(es), num_parts, seed, _p(cuts, i32p), C.byref(ncut))
            if st != DPHY_OK:
                raise DphyError(st, "dphy_partition_generate_stencil")
            cut_points = cuts[:ncut.value].copy()
        self.cut_points = np.ascontiguousarray(cut_points, np.int32)
        self._h = C.c_void_p()
        st = L.dphy_partition_split(C.byref(es), C.byref(ss), len(self.cut_points), _p(self.cut_points, i32p), C.byref(self._h))
        if st != DPHY_OK:
            raise DphyError(st, "dphy_partition_split")
        self.parts, self.origs = [], []
        for i in range(L.dphy_partition_num_parts(self._h)):
            pe = L.dphy_partition_part(self._h, i).contents
            self.parts.append(_emat_from_struct(pe))
            self.origs.append(_np_from(L.dphy_partition_orig_index(self._h, i), pe.num_nodes, np.int32))

    def reassemble(self, parts=None) -> HostEmat:
        parts = self.parts if parts is None else parts
        arr = (EmatHost * len(parts))(*[p.as_struct() for p in parts])
        es = self.emat.as_struct()
        r = self._L.dphy_partition_reassemble(self._h, C.byref(es), len(parts), arr)
        if not r:
            raise DphyError(ERR_INVALID_ARGUMENT, "dphy_partition_reassemble: parts do not match the split")
        return _emat_from_struct(r.contents)

    def close(self):
        if self._h:
            self._L.dphy_partition_free(self._h)
            self._h = C.c_void_p()


def synth_params(config: int = 0, **overrides) -> SynthParams:
    p = SynthParams()
    synth_lib().dphy_synth_default_params(C.byref(p), config)
    for k, v in overrides.items():
        if k == "pi":
            for i in range(4):
                p.pi[i] = v[i]
        else:
            setattr(p, k, v)
    return p


def synth_generate(params: SynthParams):
    """Returns (HostEmat, HostSites, info dict) -- numpy copies of a synthetic EMAT (SURVEY.md section 8d)."""
    L = synth_lib()
    out = C.POINTER(SynthEmat)()
    st = L.dphy_synth_generate(C.byref(params), C.byref(out))
    if st != DPHY_OK:
        raise DphyError(st, "dphy_synth_generate")
    try:
        s = out.contents
        e = s.emat
        N = e.num_nodes
        M = int(e.mut_off[N]); I = int(e.miss_off[N]); F = int(e.fs_off[N])
        emat = HostEmat(
            e.root, e.includes_run_root,
            parent=_np_from(e.parent, N, np.int32), child0=_np_from(e.child0, N, np.int32), child1=_np_from(e.child1, N, np.int32),
            t=_np_from(e.t, N, np.float64),
            mut_off=_np_from(e.mut_off, N + 1, np.int32), mut_site=_np_from(e.mut_site, M, np.int32),
            mut_from=_np_from(e.mut_from, M, np.uint8), mut_to=_np_from(e.mut_to, M, np.uint8), mut_t=_np_from(e.mut_t, M, np.float64),
            miss_off=_np_from(e.miss_off, N + 1, np.int32), miss_start=_np_from(e.miss_start, I, np.int32), miss_end=_np_from(e.miss_end, I, np.int32),
            fs_off=_np_from(e.fs_off, N + 1, np.int32), fs_site=_np_from(e.fs_site, F, np.int32), fs_from=_np_from(e.fs_from, F, np.uint8))
        ss = s.sites
        Ls, P = ss.num_sites, ss.num_partitions
        sites = HostSites(_np_from(ss.ref, Ls, np.uint8), _np_from(ss.partition_for_site, Ls, np.int32), _np_from(ss.nu_l, Ls, np.float64),
                          _np_from(ss.mu, P, np.float64), _np_from(ss.pi_a, P * 4, np.float64), _np_from(ss.q_ab, P * 16, np.float64))
        info = dict(mu=s.mu_used, t_max_tip=s.t_max_tip, num_mutations=int(s.num_mutations), num_intervals=int(s.num_intervals),
                    num_from_states=int(s.num_from_states), num_missing_sites=int(s.num_missing_sites), max_depth=int(s.max_depth))
        return emat, sites, info
    finally:
        L.dphy_synth_free(out)


class Context:
    """One CUDA device + stream + device arena (one per host thread / Subrun)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        self._host_blocks = []
        self.log_G_path = "auto"
        st = lib().dphy_ctx_create(device, C.byref(self._h))
        if st != DPHY_OK:
            raise DphyError(st, "dphy_ctx_create failed: a CUDA device is required (no CPU fallback)")

    def check(self, st: int):
        if st != DPHY_OK:
            raise DphyError(st, lib().dphy_last_error(self._h).decode())

    def join_side_streams(self):
        """dphy_ctx_join_side_streams: the main stream waits (on the device) for the library's side streams."""
        self.check(lib().dphy_ctx_join_side_streams(self._h))

    def synchronize(self):
        self.check(lib().dphy_ctx_synchronize(self._h))

    @property
    def stream(self) -> int:
        return int(lib().dphy_ctx_stream(self._h) or 0)

    @property
    def launches(self) -> int:
        return int(lib().dphy_ctx_launch_count(self._h))

    def host_array_like(self, a: np.ndarray) -> np.ndarray:
        """Page-locked copy of `a` (freed with the context)."""
        a = np.ascontiguousarray(a)
        p = C.c_void_p()
        self.check(lib().dphy_host_alloc(self._h, max(1, a.nbytes), C.byref(p)))
        self._host_blocks.append(p)
        buf = (C.c_char * max(1, a.nbytes)).from_address(p.value)
        out = np.frombuffer(buf, dtype=a.dtype, count=a.size).reshape(a.shape)
        out[...] = a
        return out

    def set_log_G_path(self, path: str = "auto"):
        """'auto': folded fast path when every site table has uniform nu_l; 'general': always the per-event kernels."""
        self.check(lib().dphy_ctx_set_log_G_path(self._h, {"auto": 0, "general": 1}[path]))
        self.log_G_path = path

    def arena_stats(self):
        cap, hw = C.c_size_t(), C.c_size_t()
        self.check(lib().dphy_arena_stats(self._h, C.byref(cap), C.byref(hw)))
        return cap.value, hw.value

    def close(self):
        if self._h:
            for p in self._host_blocks:        # numpy views into these blocks must not be used after close()
                lib().dphy_host_free(self._h, p)
            self._host_blocks = []
            lib().dphy_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- one-shot host-buffer call (what the C++ adapter does for Subrun::calc_cur_log_G)
    def gamma_q(self, a, x):
        a = np.ascontiguousarray(a, np.float64); x = np.ascontiguousarray(x, np.float64)
        out = np.zeros(len(a), np.float64)
        self.check(lib().dphy_gamma_q(self._h, len(a), _p(a, f64p), _p(x, f64p), _p(out, f64p)))
        return out

    def gamma_q_inv(self, a, q):
        a = np.ascontiguousarray(a, np.float64); q = np.ascontiguousarray(q, np.float64)
        out = np.zeros(len(a), np.float64)
        self.check(lib().dphy_gamma_q_inv(self._h, len(a), _p(a, f64p), _p(q, f64p), _p(out, f64p)))
        return out

    def log_G_host(self, emat: HostEmat, sites: HostSites, want_lambda=False):
        rp, br = C.c_double(), C.c_double()
        lam = np.zeros(emat.num_nodes, np.float64) if want_lambda else None
        es, ss = emat.as_struct(), sites.as_struct()
        self.check(lib().dphy_log_G_host(self._h, C.byref(es), C.byref(ss), C.byref(rp), C.byref(br),
                                         _p(lam, f64p) if want_lambda else None))
        return rp.value, br.value, lam


class DeviceSites:
    def __init__(self, ctx: Context, sites: HostSites):
        self.ctx = ctx
        # a private mirror of what the device table holds: set_evo / update must not write through to the caller's object
        self.host = HostSites(sites.ref.copy(), sites.partition_for_site.copy(), sites.nu_l.copy(), sites.mu.copy(),
                              sites.pi_a.copy(), sites.q_ab.copy())
        self._h = C.c_void_p()
        ss = sites.as_struct()
        ctx.check(lib().dphy_sites_upload(ctx._h, C.byref(ss), C.byref(self._h)))

    def set_evo(self, nu_l=None, mu=None, pi_a=None, q_ab=None):
        h = self.host
        if nu_l is not None:
            h.nu_l = np.ascontiguousarray(nu_l, np.float64)
        if mu is not None:
            h.mu = np.ascontiguousarray(mu, np.float64).reshape(-1)
        if pi_a is not None:
            h.pi_a = np.ascontiguousarray(pi_a, np.float64).reshape(-1, 4)
        if q_ab is not None:
            h.q_ab = np.ascontiguousarray(q_ab, np.float64).reshape(-1, 4, 4)
        # nu_l is passed only when it changed: the cumulative-nu tables are then left alone
        self.ctx.check(lib().dphy_sites_set_evo(self.ctx._h, self._h, _p(h.nu_l, f64p) if nu_l is not None else None,
                                                _p(h.mu, f64p), _p(h.pi_a, f64p), _p(h.q_ab, f64p)))

    def update(self, sites: HostSites):
        """New reference sequence / partitioning / model in place (same L and P): dphy_sites_update."""
        hs = sites.as_struct()
        self.ctx.check(lib().dphy_sites_update(self.ctx._h, self._h, C.byref(hs)))
        self.host = HostSites(sites.ref.copy(), sites.partition_for_site.copy(), sites.nu_l.copy(), sites.mu.copy(),
                              sites.pi_a.copy(), sites.q_ab.copy())

    def state_frequencies(self):
        out = np.zeros((self.host.num_partitions, 4), np.int32)
        self.ctx.check(lib().dphy_calc_state_frequencies_per_partition(self.ctx._h, self._h, _p(out, i32p)))
        return out

    def cum_Q_l(self):
        out = np.zeros(self.host.num_sites + 1, np.float64)
        self.ctx.check(lib().dphy_calc_cum_Q_l(self.ctx._h, self._h, _p(out, f64p)))
        return out

    def close(self):
        if self._h:
            lib().dphy_sites_destroy(self.ctx._h, self._h)
            self._h = C.c_void_p()


def sites_set_evo_many(ctx: Context, tables, mus=None, pis=None, qs=None):
    """dphy_sites_set_evo_many: new mu / pi / q (site rates kept) on several tables in one launch -- Run::push_global_params_to_subruns
    (core/run.cpp:267-275).  mus / pis / qs: one entry per table, or None to keep what the table has."""
    n = len(tables)
    for k, t in enumerate(tables):
        h = t.host
        if mus is not None and mus[k] is not None:
            h.mu = np.ascontiguousarray(mus[k], np.float64).reshape(-1)
        if pis is not None and pis[k] is not None:
            h.pi_a = np.ascontiguousarray(pis[k], np.float64).reshape(-1, 4)
        if qs is not None and qs[k] is not None:
            h.q_ab = np.ascontiguousarray(qs[k], np.float64).reshape(-1, 4, 4)
    hp = (C.c_void_p * max(n, 1))(*[t._h for t in tables])
    pm = (f64p * max(n, 1))(*[_p(t.host.mu, f64p) for t in tables])
    pp = (f64p * max(n, 1))(*[_p(t.host.pi_a, f64p) for t in tables])
    pq = (f64p * max(n, 1))(*[_p(t.host.q_ab, f64p) for t in tables])
    ctx.check(lib().dphy_sites_set_evo_many(ctx._h, n, hp, pm, pp, pq))


class Forest:
    """Device-resident batch of EMATs."""

    def __init__(self, ctx: Context, emats, sites_tables, sites_index=None):
        self.ctx = ctx
        self.emats = list(emats)
        self.sites_tables = list(sites_tables)
        n = len(self.emats)
        arr = (EmatHost * max(n, 1))(*[e.as_struct() for e in self.emats])
        idx = np.ascontiguousarray(sites_index if sites_index is not None else np.zeros(n), np.int32)
        self.sites_index = idx
        sp = (C.c_void_p * len(self.sites_tables))(*[s._h for s in self.sites_tables])
        self._h = C.c_void_p()
        ctx.check(lib().dphy_forest_upload(ctx._h, n, arr, _p(idx, i32p), len(self.sites_tables), sp, C.byref(self._h)))

    @classmethod
    def from_api_trees(cls, ctx: "Context", buffers, sites_tables, sites_index=None, includes_run_root=None, check_paths=False) -> "Forest":
        """dphy_forest_upload_api_trees: delphy.api.Tree buffers (core/api.fbs) straight to the device (check_paths:
        DPHY_API_TREE_CHECK_PATHS, the O(nodes x depth) half of the normal-form check)."""
        self = cls.__new__(cls)
        self.ctx = ctx
        # bytes are read in place (no copy); a uint8 numpy array too -- e.g. one in page-locked memory (Context.host_array_like), which
        # the library DMAs from where it lies instead of staging it
        buffers = [b if isinstance(b, np.ndarray) else bytes(b) for b in buffers]
        ptrs = [b.ctypes.data if isinstance(b, np.ndarray) else _bytes_ptr(b).value for b in buffers]
        sizes = [b.nbytes if isinstance(b, np.ndarray) else len(b) for b in buffers]
        self.emats = []
        for ptr, sz in zip(ptrs, sizes):
            v = ApiTreeView()
            if lib().dphy_api_tree_parse(ptr if sz else None, sz, C.byref(v)) != DPHY_OK:
                raise DphyError(ERR_INVALID_ARGUMENT, "api tree: malformed FlatBuffers Tree buffer")
            self.emats.append(_ApiTreeShape(v.num_nodes))
        self.sites_tables = list(sites_tables)
        n = len(buffers)
        bp = (C.c_void_p * n)(*ptrs)
        lens = (C.c_size_t * n)(*sizes)
        idx = np.ascontiguousarray(sites_index if sites_index is not None else np.zeros(n), np.int32)
        self.sites_index = idx
        irr = None if includes_run_root is None else np.ascontiguousarray(includes_run_root, np.int32)
        sp = (C.c_void_p * len(self.sites_tables))(*[s._h for s in self.sites_tables])
        self._h = C.c_void_p()
        ctx.check(lib().dphy_forest_upload_api_trees(ctx._h, n, bp, lens, None if irr is None else _p(irr, i32p), _p(idx, i32p),
                                                     len(self.sites_tables), sp, 1 if check_paths else 0, C.byref(self._h)))
        return self

    def write_api_tree(self, tree=0) -> bytes:
        """dphy_forest_write_api_tree: phylo_tree_to_api_tree (core/api.cpp:34-98) of a resident tree."""
        n = int(lib().dphy_forest_write_api_tree(self.ctx._h, self._h, tree, None, 0))
        if n < 0:
            self.ctx.check(n)
        buf = bytearray(n)
        got = int(lib().dphy_forest_write_api_tree(self.ctx._h, self._h, tree, (C.c_uint8 * n).from_buffer(buf), n))
        if got < 0:
            self.ctx.check(got)
        return bytes(buf) if got == n else bytes(memoryview(buf)[:got])

    def download_tree(self, tree=0) -> "HostEmat":
        """dphy_forest_download_tree: the host-order arrays of a tree as they are resident on the device."""
        c = TreeCounts()
        self.ctx.check(lib().dphy_forest_tree_counts(self.ctx._h, self._h, tree, C.byref(c)))
        N, M, I, F = c.num_nodes, int(c.num_mutations), int(c.num_missation_intervals), int(c.num_from_states)
        e = HostEmat(c.root, 1, parent=np.zeros(N, np.int32), child0=np.zeros(N, np.int32), child1=np.zeros(N, np.int32), t=np.zeros(N, np.float64),
                     mut_off=np.zeros(N + 1, np.int32), mut_site=np.zeros(M, np.int32), mut_from=np.zeros(M, np.uint8), mut_to=np.zeros(M, np.uint8),
                     mut_t=np.zeros(M, np.float64), miss_off=np.zeros(N + 1, np.int32), miss_start=np.zeros(I, np.int32), miss_end=np.zeros(I, np.int32),
                     fs_off=np.zeros(N + 1, np.int32), fs_site=np.zeros(F, np.int32), fs_from=np.zeros(F, np.uint8))
        st = e.as_struct()
        self.ctx.check(lib().dphy_forest_download_tree(self.ctx._h, self._h, tree, C.byref(st)))
        e.root = st.root; e.includes_run_root = st.includes_run_root
        return e

    @property
    def num_trees(self):
        return len(self.emats)

    @property
    def num_nodes(self):
        return int(lib().dphy_forest_num_nodes(self._h))

    @property
    def device_bytes(self):
        return int(lib().dphy_forest_device_bytes(self._h))

    @property
    def log_G_algorithmic_bytes(self):
        return int(lib().dphy_forest_log_G_algorithmic_bytes(self._h))

    def eval_log_G(self):
        """Asynchronous: enqueue one log-G evaluation of every tree."""
        self.ctx.check(lib().dphy_forest_eval_log_G(self.ctx._h, self._h))

    def log_G(self):
        n = self.num_trees
        rp, br, lg = np.zeros(n), np.zeros(n), np.zeros(n)
        self.ctx.check(lib().dphy_forest_get_log_G(self.ctx._h, self._h, _p(rp, f64p), _p(br, f64p), _p(lg, f64p)))
        return rp, br, lg

    def lambda_i(self, tree=0):
        out = np.zeros(self.emats[tree].num_nodes, np.float64)
        self.ctx.check(lib().dphy_forest_get_lambda_i(self.ctx._h, self._h, tree, _p(out, f64p)))
        return out

    def num_sites_missing(self, tree=0):
        out = np.zeros(self.emats[tree].num_nodes, np.int32)
        self.ctx.check(lib().dphy_forest_get_num_sites_missing(self.ctx._h, self._h, tree, _p(out, i32p)))
        return out

    def set_node_times(self, tree, nodes, t):
        nodes = np.ascontiguousarray(nodes, np.int32); t = np.ascontiguousarray(t, np.float64)
        self.ctx.check(lib().dphy_forest_set_node_times(self.ctx._h, self._h, tree, len(nodes), _p(nodes, i32p), _p(t, f64p)))

    def apply_rows(self, rows, new_roots=None):
        """dphy_forest_apply_rows: replace the given NodeRow rows (and optionally every tree's root) on the device."""
        n = len(rows)
        arr = (NodeRow * max(n, 1))(*rows)
        nr = None if new_roots is None else np.ascontiguousarray(new_roots, np.int32)
        self.ctx.check(lib().dphy_forest_apply_rows(self.ctx._h, self._h, n, arr, _p(nr, i32p) if nr is not None else None))

    def log_coalescent_prior(self, n0, g, t0=0.0):
        """dphy_forest_log_coalescent_prior: float64 array [num_trees], the log-density of each tree's node times under the
        exponential-growth coalescent N(t) = n0 * exp(g * (t - t0)).  Times grow toward the present (a parent is never later than
        its children), so g > 0 means growth toward the present; n0 is in the unit of the node times, g in its inverse.  Tips add a
        lineage going back in time, inner nodes (coalescences) remove one; with k lineages on the interval (a, b) between two
        consecutive events,
            log P = sum_c -log N(t_c) - sum_(a,b) C(k, 2) * exp(-g (a - t0)) / n0 * (1 - exp(-g (b - a))) / g,
        the last factor being b - a at g = 0 (evaluated as -expm1(-g (b - a)) / g: no cancellation for tiny |g|)."""
        out = np.zeros(max(self.num_trees, 1), np.float64)
        self.ctx.check(lib().dphy_forest_log_coalescent_prior(self.ctx._h, self._h, float(n0), float(g), float(t0), _p(out, f64p)))
        return out[:self.num_trees]

    def tallies(self):
        out = (Tallies * self.num_trees)()
        self.ctx.check(lib().dphy_forest_calc_tallies(self.ctx._h, self._h, out))
        return [dict(num_muts=o.num_muts, num_muts_ab=np.array(o.num_muts_ab[:], np.int32).reshape(4, 4), T=o.T,
                     log_root_prior=o.log_root_prior, log_G_below_root=o.log_G_below_root) for o in out]

    def num_muts_beta_ab(self, tree=0):
        P = self.sites_tables[self.sites_index[tree]].host.num_partitions
        out = np.zeros((P, 4, 4), np.int32)
        self.ctx.check(lib().dphy_forest_calc_num_muts_beta_ab(self.ctx._h, self._h, tree, _p(out, i32p)))
        return out

    def num_muts_l(self, tree=0, want_ab=True):
        L = self.sites_tables[self.sites_index[tree]].host.num_sites
        out_l = np.zeros(L, np.int32)
        out_ab = np.zeros((L, 4, 4), np.int32) if want_ab else None
        self.ctx.check(lib().dphy_forest_calc_num_muts_l(self.ctx._h, self._h, tree, _p(out_l, i32p),
                                                         _p(out_ab, i32p) if want_ab else None))
        return out_l, out_ab

    def Ttwiddle_beta_a(self, tree=0):
        P = self.sites_tables[self.sites_index[tree]].host.num_partitions
        out = np.zeros((P, 4), np.float64)
        self.ctx.check(lib().dphy_forest_calc_Ttwiddle_beta_a(self.ctx._h, self._h, tree, _p(out, f64p)))
        return out

    def Ttwiddle_l(self, tree=0, want_T_l_a=True):
        L = self.sites_tables[self.sites_index[tree]].host.num_sites
        out_l = np.zeros(L, np.float64)
        out_la = np.zeros((L, 4), np.float64) if want_T_l_a else None
        self.ctx.check(lib().dphy_forest_calc_Ttwiddle_l(self.ctx._h, self._h, tree, _p(out_l, f64p),
                                                         _p(out_la, f64p) if want_T_l_a else None))
        return out_l, out_la

    def cycle_tallies_device(self, device_ptr: int, cap: int):
        """Packs the forest's additive per-cycle tallies into device memory at `device_ptr` (>= 19 + 4P doubles), asynchronously
        on the ctx stream: [log_G, T, num_muts, num_muts_ab[16], Ttwiddle_beta_a[4P]] summed over the forest's trees."""
        self.ctx.check(lib().dphy_forest_cycle_tallies_device(self.ctx._h, self._h, C.c_void_p(device_ptr), cap))

    def site_tallies(self):
        """(Ttwiddle_l, num_muts_l) of every tree in one call: two [num_trees, max L] arrays (rows padded with zeros)."""
        ld = max(t.host.num_sites for t in self.sites_tables)
        tw = np.zeros((self.num_trees, ld), np.float64)
        nm = np.zeros((self.num_trees, ld), np.int32)
        self.ctx.check(lib().dphy_forest_calc_site_tallies(self.ctx._h, self._h, ld, _p(tw, f64p), _p(nm, i32p)))
        return tw, nm

    # -- placement of new samples
    def place_samples(self, samples, tree=0, can_change_root=True, max_best=0, t_X=None):
        """dphy_forest_place_samples: maximum-parsimony placement of new sequences on tree `tree`.  `samples` is the dict maple_parse
        returns, or any dict with its six arrays (delta_off / delta_site / delta_to, miss_off / miss_start / miss_end).  Returns a dict of
        numpy arrays: min_muts, num_best, branch, mut_idx (one entry per sample) and best, a [S, max_best] REGION_DTYPE array of the
        first max_best best regions in the study's emission order (unused slots: branch == -1).

        t_X: None places without a date limit.  Otherwise one float64 per sample, its date limit, in the tree's time unit
        (dphy_forest_place_dated_samples): only regions starting before t_X count, and t_max is clipped to t_X.  For a sample known
        by a date range, pass the end you want to hold it to -- usually maple_parse(...)["t_max"], the latest time it could have
        been taken; the library does not choose."""
        a = dict(delta_off=np.ascontiguousarray(samples["delta_off"], np.int32), delta_site=np.ascontiguousarray(samples["delta_site"], np.int32),
                 delta_to=np.ascontiguousarray(samples["delta_to"], np.uint8), miss_off=np.ascontiguousarray(samples["miss_off"], np.int32),
                 miss_start=np.ascontiguousarray(samples["miss_start"], np.int32), miss_end=np.ascontiguousarray(samples["miss_end"], np.int32))
        S = len(a["delta_off"]) - 1
        if S < 0 or len(a["miss_off"]) != S + 1:
            raise ValueError("place_samples: delta_off and miss_off must both have num_samples + 1 entries")
        ss = SampleSet(S, 0, _p(a["delta_off"], i32p), _p(a["delta_site"], i32p), _p(a["delta_to"], u8p), _p(a["miss_off"], i32p),
                       _p(a["miss_start"], i32p), _p(a["miss_end"], i32p))
        out = np.zeros(max(S, 1), PLACEMENT_DTYPE)
        best = np.zeros((max(S, 1), max_best), REGION_DTYPE)
        outs = (_p(out, C.POINTER(Placement)), _p(best, C.POINTER(CandidateRegion)) if max_best > 0 else None)
        if t_X is None:
            self.ctx.check(lib().dphy_forest_place_samples(self.ctx._h, self._h, tree, C.byref(ss), int(bool(can_change_root)), max_best,
                                                           *outs))
        else:
            tx = np.ascontiguousarray(t_X, np.float64)
            if tx.shape != (S,):
                raise ValueError("place_samples: t_X must hold one value per sample")
            self.ctx.check(lib().dphy_forest_place_dated_samples(self.ctx._h, self._h, tree, C.byref(ss), _p(tx, f64p),
                                                                 int(bool(can_change_root)), max_best, *outs))
        return dict(min_muts=out["min_muts"][:S].copy(), num_best=out["num_best"][:S].copy(), branch=out["branch"][:S].copy(),
                    mut_idx=out["mut_idx"][:S].copy(), best=best[:S])

    # -- SPR studies
    def spr_study_batch(self, requests):
        return SprBatch(self, requests)

    def close(self):
        if self._h:
            lib().dphy_forest_destroy(self.ctx._h, self._h)
            self._h = C.c_void_p()


class CladeTable:
    """dphy_clade_table: clade counts and summed clade times over every tree added, for clade support and the maximum clade
    credibility (MCC) tree.  A clade is the set of tips (nodes with child0 == -1, identified by host node index) below a node; the
    first add fixes the tip set, and every tree added or scored later must have the same number of nodes and the same tip indices.
    score(forest)[k] = sum over the nodes v of tree k of log(count(v) / num_trees): the MCC tree is the argmax over the added trees."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self._h = C.c_void_p()
        ctx.check(lib().dphy_clade_table_create(ctx._h, C.byref(self._h)))

    def add(self, forest: Forest):
        """Count every tree of `forest` as it is resident now."""
        self.ctx.check(lib().dphy_clade_table_add(self.ctx._h, self._h, forest._h))

    def _info(self):
        v = [C.c_int64() for _ in range(3)]
        self.ctx.check(lib().dphy_clade_table_info(self._h, *[C.byref(x) for x in v]))
        return [x.value for x in v]

    @property
    def num_trees(self):
        return self._info()[0]

    @property
    def num_clades(self):
        return self._info()[1]

    @property
    def device_bytes(self):
        return self._info()[2]

    def score(self, forest: Forest):
        """float64 [num_trees]: sum of log(count / num_trees) over each tree's nodes (-inf where a clade was never added)."""
        out = np.zeros(max(forest.num_trees, 1), np.float64)
        self.ctx.check(lib().dphy_clade_table_score(self.ctx._h, self._h, forest._h, _p(out, f64p)))
        return out[:forest.num_trees]

    def node_support(self, forest: Forest, tree=0):
        """(count int64 [num_nodes], mean_t float64 [num_nodes]) of tree `tree`, host node order: how many added trees contain each
        node's clade, and its mean node time over them (0 and NaN for a clade never added)."""
        n = forest.emats[tree].num_nodes if 0 <= tree < forest.num_trees else 1
        count, mean_t = np.zeros(max(n, 1), np.int64), np.zeros(max(n, 1), np.float64)
        self.ctx.check(lib().dphy_clade_table_node_support(self.ctx._h, self._h, forest._h, tree, _p(count, C.POINTER(C.c_int64)),
                                                           _p(mean_t, f64p)))
        return count[:n], mean_t[:n]

    def close(self):
        if self._h:
            lib().dphy_clade_table_destroy(self.ctx._h, self._h)
            self._h = C.c_void_p()


def spr_request(tree, X, t_X, start_branch, start_mut_idx, init_min_muts, lambda_X, t_max_tip,
                max_muts_from_start=INT32_MAX, can_change_root=True, annealing_factor=0.8,
                x_deltas=None, x_missing=None, x_state_mode=SPR_X_FROM_TREE):
    """x_deltas: [(site, to_state)], x_missing: (starts, ends); read only when x_state_mode != SPR_X_FROM_TREE or X == -1."""
    r = SprRequest()
    r.x_state_mode = x_state_mode
    r.tree, r.X, r.t_X = tree, X, t_X
    r.start_branch, r.start_mut_idx, r.init_min_muts = start_branch, start_mut_idx, init_min_muts
    r.max_muts_from_start, r.can_change_root = max_muts_from_start, int(can_change_root)
    r.lambda_X, r.annealing_factor, r.t_max_tip = lambda_X, annealing_factor, t_max_tip
    keep = []
    if x_deltas is not None:
        s = np.ascontiguousarray([d[0] for d in x_deltas], np.int32); t = np.ascontiguousarray([d[1] for d in x_deltas], np.uint8)
        r.n_x_deltas, r.x_delta_site, r.x_delta_to = len(s), _p(s, i32p), _p(t, u8p)
        keep += [s, t]
    if x_missing is not None:
        a = np.ascontiguousarray(x_missing[0], np.int32); b = np.ascontiguousarray(x_missing[1], np.int32)
        r.n_x_missing, r.x_missing_start, r.x_missing_end = len(a), _p(a, i32p), _p(b, i32p)
        keep += [a, b]
    r._keep = keep
    return r


class SprBatch:
    def __init__(self, forest: Forest, requests):
        self.forest = forest
        self.ctx = forest.ctx
        self.requests = list(requests)
        n = len(self.requests)
        arr = (SprRequest * max(n, 1))(*self.requests)
        self._h = C.c_void_p()
        self.ctx.check(lib().dphy_spr_study_batch(self.ctx._h, forest._h, n, arr, C.byref(self._h)))

    def summaries(self):
        out = (SprSummary * max(len(self.requests), 1))()
        self.ctx.check(lib().dphy_spr_batch_get_summaries(self.ctx._h, self._h, out))
        return list(out)[:len(self.requests)]

    def total_regions(self):
        return int(lib().dphy_spr_batch_total_regions(self.ctx._h, self._h))

    def total_regions_checked(self):
        n = self.total_regions()
        if n < 0:
            self.ctx.check(n)
        return n

    def regions(self, request=-1):
        n = self.total_regions() if request < 0 else self.summaries()[request].num_regions
        out = np.zeros(max(n, 1), REGION_DTYPE)
        got = lib().dphy_spr_batch_get_regions(self.ctx._h, self._h, request, _p(out, C.POINTER(CandidateRegion)), n)
        if got < 0:
            self.ctx.check(int(got))
        return out[:got]

    def pick_nexus_regions(self, r):
        r = np.ascontiguousarray(r, np.float64)
        out = np.zeros(len(self.requests), np.int32)
        self.ctx.check(lib().dphy_spr_batch_pick_nexus_regions(self.ctx._h, self._h, _p(r, f64p), _p(out, i32p)))
        return out

    def find_region(self, request, branch, t):
        out = C.c_int32(-2)
        self.ctx.check(lib().dphy_spr_batch_find_region(self.ctx._h, self._h, request, branch, t, C.byref(out)))
        return out.value

    def set_weights(self, params):
        """params: [(lambda_X, annealing_factor, t_max_tip)] per request -- the Spr_study constructor on enumerated regions."""
        n = len(self.requests)
        arr = (SprWeightParams * max(n, 1))(*[SprWeightParams(*p) for p in params])
        self.ctx.check(lib().dphy_spr_batch_set_weights(self.ctx._h, self._h, arr))

    def region_weights(self, request, regions):
        """Fills only the weight fields of `regions` (a REGION_DTYPE array from regions())."""
        got = lib().dphy_spr_batch_get_region_weights(self.ctx._h, self._h, request, _p(regions, C.POINTER(CandidateRegion)), len(regions))
        if got < 0:
            self.ctx.check(int(got))
        return regions

    def log_alpha_in_region(self, request, region_idx, t):
        out = C.c_double(0.0)
        self.ctx.check(lib().dphy_spr_batch_log_alpha_in_region(self.ctx._h, self._h, request, region_idx, t, C.byref(out)))
        return out.value

    def close(self):
        if self._h:
            lib().dphy_spr_batch_destroy(self.ctx._h, self._h)
            self._h = C.c_void_p()


def net_branch_deltas(emat: HostEmat, X: int):
    """Net (site -> (from, to)) deltas of the mutations on branch X, reversals cancelled
    (== calc_site_deltas_between(tree, parent(X), X), core/site_deltas.cpp:83-101)."""
    d = {}
    for i in range(int(emat.mut_off[X]), int(emat.mut_off[X + 1])):
        l, fr, to = int(emat.mut_site[i]), int(emat.mut_from[i]), int(emat.mut_to[i])
        if l in d:
            f0, _ = d[l]
            if f0 == to:
                del d[l]
            else:
                d[l] = (f0, to)
        else:
            d[l] = (fr, to)
    return d


def spr_requests_for_attached(emat: HostEmat, tree: int, xs, lambda_i, t_max_tip, max_muts_from_start=INT32_MAX,
                              can_change_root=True, annealing_factor=0.8):
    """Requests seeded exactly as Subrun::spr1_move seeds its study (core/subrun.cpp:540-553): start region = (sibling
    of X, 0), initial deltas = the net mutations on branch parent(X)->X."""
    reqs = []
    for X in xs:
        X = int(X)
        P = int(emat.parent[X])
        S = int(emat.child1[P]) if int(emat.child0[P]) == X else int(emat.child0[P])
        reqs.append(spr_request(tree, X, float(emat.t[X]), S, 0, len(net_branch_deltas(emat, X)), float(lambda_i[X]),
                                float(t_max_tip), max_muts_from_start, can_change_root, annealing_factor))
    return reqs
