/* delphy_b200.h -- C ABI of the B200-native EMAT log-G + SPR-regraft engine.
 *
 * This is the drop-in boundary for Delphy's data-parallel hot path (SURVEY.md section 8b).  The reference has
 * no plugin/FFI layer for this path: the boundary is the set of C++ free functions and structs declared in
 * core/phylo_tree_calc.h, core/spr_study.h and core/spr_move.h (all file:line citations below are relative
 * to the reference checkout).  A C++ adapter with the reference's exact signatures (INTEGRATION.md) flattens a
 * delphy::Phylo_tree / Global_evo_model into the plain arrays below and calls these entry points.
 *
 * Conventions (mirroring the reference's only extern "C" surface, tools/delphy_wasm.cpp:56-90):
 *   - context pointer first, raw pointers + sizes, no C++/torch types;
 *   - every call returns DPHY_OK (0) or a negative dphy_status; dphy_last_error() gives the message
 *     (the reference throws std::out_of_range / std::invalid_argument or CHECK-aborts, core/mutations.h:187-191;
 *      the adapter re-throws from the status);
 *   - host inputs are borrowed for the duration of the call only; outputs are caller-owned host buffers;
 *   - one dphy_ctx per host thread / Subrun (core/run.cpp:682-693 runs one Subrun per worker thread);
 *     a ctx owns one CUDA stream and one device arena (the device analogue of core/scratch_space.h:49-267).
 *   - there is NO CPU fallback: every compute entry point fails with DPHY_ERR_CUDA if no device is usable.
 */
#ifndef DELPHY_B200_H_
#define DELPHY_B200_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum dphy_status {
  DPHY_OK = 0,
  DPHY_ERR_INVALID_ARGUMENT = -1,   /* std::invalid_argument in the reference */
  DPHY_ERR_OUT_OF_RANGE = -2,       /* std::out_of_range in the reference (e.g. core/mutations.h:187-191) */
  DPHY_ERR_CUDA = -3,               /* no device / launch failure (no CPU fallback exists) */
  DPHY_ERR_OUT_OF_MEMORY = -4,
  DPHY_ERR_INTERNAL = -5            /* a CHECK(...) in the reference */
} dphy_status;

typedef struct dphy_ctx dphy_ctx;         /* device + stream + arena */
typedef struct dphy_sites dphy_sites;     /* device copy of ref_sequence + Global_evo_model + derived per-site tables */
typedef struct dphy_forest dphy_forest;   /* device-resident batch of EMATs (partition parts and/or independent chains) */
typedef struct dphy_spr_batch dphy_spr_batch; /* device-resident results of a batch of SPR studies */

/* One EMAT == one delphy::Phylo_tree (core/phylo_tree.h:14-63, core/tree.h:181-220) flattened to SoA + CSR,
 * in HOST node order.  Letters are Real_seq_letter codes A=0,C=1,G=2,T=3 (core/sequence.h:155). */
typedef struct dphy_emat_host {
  int32_t num_nodes;
  int32_t root;                /* Tree::root */
  int32_t includes_run_root;   /* Subrun::includes_run_root_ : add calc_log_root_prior to log G (core/subrun.cpp:58-68) */
  int32_t reserved;
  const int32_t* parent;       /* [N] Node::parent, -1 == k_no_node */
  const int32_t* child0;       /* [N] Binary_node::children[0], -1 for tips */
  const int32_t* child1;       /* [N] Binary_node::children[1] */
  const double*  t;            /* [N] Phylo_node::t */
  const int32_t* mut_off;      /* [N+1] CSR offsets into the mutation arrays (root's list included) */
  const int32_t* mut_site;     /* Mutation::site (core/mutations.h:21-29); per branch sorted by (t, site) */
  const uint8_t* mut_from;
  const uint8_t* mut_to;
  const double*  mut_t;
  const int32_t* miss_off;     /* [N+1] CSR offsets into Missation_map::intervals (core/mutations.h:124-137) */
  const int32_t* miss_start;
  const int32_t* miss_end;
  const int32_t* fs_off;       /* [N+1] CSR offsets into Missation_map::from_states */
  const int32_t* fs_site;
  const uint8_t* fs_from;
} dphy_emat_host;

/* Reference sequence + Global_evo_model (core/evo_model.h:12-48). */
typedef struct dphy_sites_host {
  int32_t num_sites;
  int32_t num_partitions;
  const uint8_t* ref;                  /* [L] Phylo_tree::ref_sequence */
  const int32_t* partition_for_site;   /* [L] */
  const double*  nu_l;                 /* [L] */
  const double*  mu;                   /* [P] Site_evo_model::mu */
  const double*  pi_a;                 /* [P][4] */
  const double*  q_ab;                 /* [P][4][4]; q_a(a) == -q_ab[a][a] */
} dphy_sites_host;

/* Byte-for-byte the layout of delphy::Candidate_region (core/spr_study.h:17-32), 48 bytes. */
typedef struct dphy_candidate_region {
  int32_t branch;
  int32_t mut_idx;
  double  t_min;
  double  t_max;
  int32_t min_muts;
  int32_t pad_;
  double  log_W_over_Wmax;
  double  W_over_Wmax;
} dphy_candidate_region;

/* Inputs of one SPR study == Spr_study_builder{tree, X, t_X, missing_at_X} + .max_muts_from_start +
 * .seed_fill_from(branch, mut_idx, deltas, can_change_root) + Spr_study{builder, lambda_X, f, t_X, t_max_tip}
 * (core/spr_study.h:69-205).
 *
 * Where X's sequence and missing set come from (x_state_mode):
 *   DPHY_SPR_X_FROM_TREE  X >= 0 is attached and the EMAT is self-consistent: both are reconstructed on the device
 *                         (reconstruct_missing_sites_at / view_of_sequence_at, core/phylo_tree_calc.cpp:19-56);
 *   DPHY_SPR_X_REL_REF    the caller passes X's sequence as deltas from the REFERENCE sequence plus its missing intervals
 *                         (a sequence that is not in the tree: X == -1 == k_no_node, build_usher_like_tree,
 *                         core/phylo_tree.cpp:918-932);
 *   DPHY_SPR_X_REL_START  exactly the builder's own inputs: x_delta_* is the Site_deltas `init_to_X_deltas` handed to
 *                         seed_fill_from -- deltas from the state at the START REGION (start_branch, start_mut_idx) to X --
 *                         and x_missing_* is `missing_at_X` (core/spr_study.cpp:9-24, core/subrun.cpp:543-554).  Nothing about X is
 *                         read from the tree, so this is the mode for studies on a tree mid-move (after Spr_move::peel_graft /
 *                         move, core/subrun.cpp:539-599) and it works for X >= 0 and X == -1 alike.
 * lambda_X == 0 enumerates the regions only (the builder without the Spr_study constructor): weights stay 0 until
 * dphy_spr_batch_set_weights. */
#define DPHY_SPR_X_FROM_TREE 0
#define DPHY_SPR_X_REL_REF 1
#define DPHY_SPR_X_REL_START 2
typedef struct dphy_spr_request {
  int32_t tree;                 /* index of the EMAT inside the forest */
  int32_t X;                    /* node being pruned (host node index), or -1 */
  double  t_X;
  int32_t start_branch;         /* seed_fill_from(init_branch, init_mut_idx, ...) */
  int32_t start_mut_idx;
  int32_t init_min_muts;        /* == ssize(init_to_X_deltas) */
  int32_t max_muts_from_start;  /* INT32_MAX == unbounded */
  int32_t can_change_root;
  int32_t x_state_mode;         /* DPHY_SPR_X_* */
  double  lambda_X;             /* > 0, or 0 for "enumerate only" */
  double  annealing_factor;
  double  t_max_tip;
  /* only read when x_state_mode != DPHY_SPR_X_FROM_TREE: */
  int32_t n_x_deltas;  const int32_t* x_delta_site;  const uint8_t* x_delta_to;
  int32_t n_x_missing; const int32_t* x_missing_start; const int32_t* x_missing_end;
} dphy_spr_request;

/* Inputs of the Spr_study constructor for a study whose regions are already enumerated (core/spr_study.cpp:226-239). */
typedef struct dphy_spr_weight_params {
  double lambda_X;
  double annealing_factor;
  double t_max_tip;
} dphy_spr_weight_params;

/* Outputs of Spr_study::Spr_study (core/spr_study.cpp:226-385). */
typedef struct dphy_spr_summary {
  double  mu;                 /* lambda_X / (L - #sites missing at X)  (:239) */
  double  log_Wmax;
  double  sum_W_over_Wmax;
  int32_t num_regions;
  int32_t num_missing_at_X;
  int64_t region_offset;      /* first region of this study inside the batch's region array */
} dphy_spr_summary;

/* Integer and floating tallies of Run::recalc_derived_quantities / global moves (core/run.cpp:437-478). */
typedef struct dphy_tallies {
  int32_t num_muts;                 /* calc_num_muts            core/phylo_tree_calc.cpp:577-585 */
  int32_t reserved;
  int32_t num_muts_ab[16];          /* calc_num_muts_ab         :587-597 */
  double  T;                        /* calc_T                   :120-128 */
  double  log_root_prior;           /* calc_log_root_prior      :467-504 (0 if !includes_run_root) */
  double  log_G_below_root;         /* calc_log_G_below_root    :515-543 */
} dphy_tallies;

/* ---- context ----------------------------------------------------------------------------------------- */
int  dphy_ctx_create(int device, dphy_ctx** out);
void dphy_ctx_destroy(dphy_ctx* ctx);
const char* dphy_last_error(const dphy_ctx* ctx);
int  dphy_ctx_synchronize(dphy_ctx* ctx);
/* Makes the ctx's main stream wait (on the device, no host block) for whatever the library has put on its side streams -- the
 * normalisation pass of the latest SPR batches runs on one, next to the set-up of the following batch.  Every accessor of a batch
 * joins on its own; callers that time a region with events on dphy_ctx_stream() call this before recording the closing event. */
int  dphy_ctx_join_side_streams(dphy_ctx* ctx);
/* Device arena replacing scratch_space (core/scratch_space.h:49-267): stats + explicit reset (scope close). */
int  dphy_arena_stats(const dphy_ctx* ctx, size_t* capacity, size_t* high_water);
/* cudaStream_t of the ctx as a void* (so callers can record CUDA events on the launching stream). */
void* dphy_ctx_stream(dphy_ctx* ctx);
/* number of kernels this ctx has launched so far (bench.py's gpu_launches) */
int64_t dphy_ctx_launch_count(const dphy_ctx* ctx);

/* Page-locked host memory for the arrays of dphy_emat_host.  dphy_forest_upload DMAs straight out of buffers obtained
 * here (or registered by the caller with cudaHostRegister); pageable buffers are staged through the ctx's own pinned slab by
 * worker threads.  The analogue on the reference side is the arena a Phylo_tree's vectors live in (core/scratch_space.h). */
int  dphy_host_alloc(dphy_ctx* ctx, size_t bytes, void** out);
void dphy_host_free(dphy_ctx* ctx, void* p);

/* Which kernels dphy_forest_eval_log_G uses.  AUTO: forests whose site tables all have uniform nu_l take the folded path
 * (per-branch state-count vectors built at upload; the per-event lists are only walked for the mutation times);
 * GENERAL: always the per-event path (the only one when there is site-rate heterogeneity).  Results agree to ~1e-13. */
#define DPHY_LOG_G_PATH_AUTO 0
#define DPHY_LOG_G_PATH_GENERAL 1
int  dphy_ctx_set_log_G_path(dphy_ctx* ctx, int path);

/* ---- sites / evo model ------------------------------------------------------------------------------- */
/* Lifetime: a forest keeps pointers to the sites tables it was uploaded against; destroy the forests first.  Inputs are validated
 * before anything is committed (ref in ACGT, partitions in range, mu / pi / nu finite and >= 0, q_ab a finite rate matrix). */
int  dphy_sites_upload(dphy_ctx* ctx, const dphy_sites_host* host, dphy_sites** out);
void dphy_sites_destroy(dphy_ctx* ctx, dphy_sites* sites);
/* Subrun::set_evo (core/subrun.h:29-30): new mu/pi/q/nu_l; recomputes cum_Q_l on the device.  nu_l == NULL keeps the current site
 * rates (the cumulative-nu tables are then not rebuilt).  Asynchronous: consumers are ordered after it on the ctx's stream. */
int  dphy_sites_set_evo(dphy_ctx* ctx, dphy_sites* sites, const double* nu_l, const double* mu,
                        const double* pi_a, const double* q_ab);
/* dphy_sites_set_evo (site rates kept) on `n` different tables in ONE launch: what Run::push_global_params_to_subruns does once per
 * cycle -- the new mu / pi / q go to every subrun's evo model (core/run.cpp:267-275).  mu[k] / pi_a[k] / q_ab[k] are table k's
 * arrays ([P_k], [P_k][4], [P_k][4][4]).  Everything is validated before anything is committed.  Asynchronous. */
int  dphy_sites_set_evo_many(dphy_ctx* ctx, int32_t n, dphy_sites* const* tables, const double* const* mu, const double* const* pi_a,
                             const double* const* q_ab);
/* Replace the reference sequence, the site partitioning and the whole model of an existing table in place (same number of sites
 * and partitions): what Run::normalize_root -> rereference_to_root_sequence does to every subrun's tables once per cycle
 * (core/run.cpp:258-265, core/phylo_tree.cpp:299-312).  No allocation; every derived table is rebuilt on the device.
 * Forests uploaded against the old sequence keep their folded weights and must be re-uploaded. */
int  dphy_sites_update(dphy_ctx* ctx, dphy_sites* sites, const dphy_sites_host* host);
/* calc_state_frequencies_per_partition_of (core/phylo_tree_calc.cpp:95-106) -> out[P*4] */
int  dphy_calc_state_frequencies_per_partition(dphy_ctx* ctx, dphy_sites* sites, int32_t* out);
/* calc_cum_Q_l_for_sequence (core/phylo_tree_calc.cpp:379-388) -> out[L+1] */
int  dphy_calc_cum_Q_l(dphy_ctx* ctx, dphy_sites* sites, double* out);

/* ---- forest (batch of EMATs) -------------------------------------------------------------------------- */
/* trees[i] uses sites[sites_index[i]].  All host arrays are copied; nothing is retained. */
int  dphy_forest_upload(dphy_ctx* ctx, int32_t num_trees, const dphy_emat_host* trees,
                        const int32_t* sites_index, int32_t num_sites_tables, dphy_sites* const* sites,
                        dphy_forest** out);
void dphy_forest_destroy(dphy_ctx* ctx, dphy_forest* forest);
int64_t dphy_forest_num_nodes(const dphy_forest* forest);
int64_t dphy_forest_device_bytes(const dphy_forest* forest);
/* algorithmic bytes of one log-G evaluation over the whole forest (SURVEY.md section 8d formula) */
int64_t dphy_forest_log_G_algorithmic_bytes(const dphy_forest* forest);
/* Update node times in place (accepted inner_node/tip displace moves, core/subrun.cpp:223-231,276-284).  Times must not
 * decrease away from the root (the reference's integrity CHECK, core/phylo_tree.cpp:131; the SPR kernels prune subtrees on it):
 * DPHY_ERR_INVALID_ARGUMENT if a displaced node ends up earlier than its parent or later than a child (the times are then
 * already changed -- set them again); dphy_forest_upload rejects such trees outright. */
int  dphy_forest_set_node_times(dphy_ctx* ctx, dphy_forest* forest, int32_t tree, int32_t count,
                                const int32_t* nodes, const double* t);

/* ---- incremental edits (device-resident; SURVEY.md section 8f row 1) --------------------------------------------------------------
 * One changed node of one tree: its new links, time and lists (the whole row).  What the reference's in-place edits change:
 * a branch-reform move = one row (core/subrun.cpp:316-319); an SPR move = the rows of X, P, G, the old and the new sibling and its
 * old parent, plus the nodes of the hot path whose lists peel_graft / apply_graft rewrite (core/spr_move.cpp:838-1156). */
typedef struct dphy_node_row {
  int32_t tree;                 /* index of the EMAT inside the forest */
  int32_t node;                 /* host node index */
  int32_t parent, child0, child1;   /* -1 == k_no_node */
  int32_t n_muts, n_miss, n_fs;
  double  t;
  const int32_t* mut_site; const uint8_t* mut_from; const uint8_t* mut_to; const double* mut_t;
  const int32_t* miss_start; const int32_t* miss_end;
  const int32_t* fs_site; const uint8_t* fs_from;
} dphy_node_row;
/* Replace `count` rows and (new_roots != NULL) set every tree's root (new_roots[num_trees]).  Only the rows cross PCIe: the
 * host-order arrays of every tree stay resident on the device, the edited trees' arrays are rebuilt there and the forest is
 * re-flattened from them with the validation of an upload (DPHY_ERR_INVALID_ARGUMENT for a broken topology / times, the forest
 * is then unchanged).  Results are those of a fresh dphy_forest_upload of the edited trees.  SPR batches made before the call
 * refer to the old forest and must be destroyed first. */
int  dphy_forest_apply_rows(dphy_ctx* ctx, dphy_forest* forest, int32_t count, const dphy_node_row* rows, const int32_t* new_roots);

/* ---- the reference's wire / on-disk tree format, straight to and from the device (SURVEY.md section 8f row 4) ------------------------
 * delphy.api.Tree (core/api.fbs:13-49): the size-prefixed FlatBuffers buffer phylo_tree_to_api_tree writes (core/api.cpp:34-98) --
 * `.dphy` files (core/delphy_output.cpp:111-121) and the WASM API (tools/delphy_wasm.cpp:500-534) carry it. */
typedef struct dphy_api_tree_view {
  int32_t num_nodes, root, num_sites, reserved;
  int64_t num_mutations, num_missation_intervals;
  const void* nodes;                  /* num_nodes x 16 B  {parent i32, left_child i32, right_child i32, t f32}            (core/api_generated.h:157-190) */
  const void* mutations;              /* 16 B each         {branch i32, site i32, from u8, to u8, 2 B padding, t f32}     (:192-236) */
  const void* missation_intervals;    /* 12 B each         {branch i32, start_site i32, end_site i32}                    (:238-265) */
  const uint8_t* ref_seq;             /* num_sites letters A=0 C=1 G=2 T=3 */
} dphy_api_tree_view;
/* Host only: GetSizePrefixedRoot<api::Tree> + the field accessors (core/api_generated.h:267-304) with every offset bounds-checked (the
 * buffer is untrusted).  The view points into `buf`.  DPHY_ERR_INVALID_ARGUMENT for a malformed buffer. */
int  dphy_api_tree_parse(const void* buf, size_t len, dphy_api_tree_view* out);
/* api_tree_and_tree_info_to_phylo_tree (core/api.cpp:127-186) + the flattening of dphy_forest_upload, without the AoS Phylo_tree in
 * between: the struct vectors of every buffer are DMA'd as they lie (from where they lie when the buffer is page-locked; through
 * the context's pinned slab otherwise); the struct-of-arrays split, the CSR offsets and the
 * Missation_map::from_states (which the format does not store; fix_up_missations, core/phylo_tree.cpp:446-459) are computed on the
 * device.  Tree k is loaded against sites[sites_index[k]], whose reference sequence must equal the buffer's ref_seq;
 * includes_run_root may be NULL (all 1).  Times are the format's float32 values widened to double, as in the reference.  The result is
 * the forest dphy_forest_upload would build from the reference's reloaded Phylo_tree.
 * Precondition, true of every buffer phylo_tree_to_api_tree wrote: fix_up_missations has nothing to rewrite beyond the from_states.
 * Always checked (DPHY_ERR_INVALID_ARGUMENT): records grouped by ascending branch, a branch's intervals ascending and apart; the
 * two children of a node share no missing site; no mutation on a site missing at its own node; every mutation's `from` equals the
 * state of the sequence above it (the reference CHECKs); plus everything dphy_forest_upload validates.  With
 * flags & DPHY_API_TREE_CHECK_PATHS also the half that needs every root path walked (O(nodes x depth)): no site missing at a node and
 * again at an ancestor, no mutation on a site missing at an ancestor. */
#define DPHY_API_TREE_CHECK_PATHS 1u
int  dphy_forest_upload_api_trees(dphy_ctx* ctx, int32_t num_trees, const void* const* bufs, const size_t* lens,
                                  const int32_t* includes_run_root, const int32_t* sites_index, int32_t num_sites_tables,
                                  dphy_sites* const* sites, uint32_t flags, dphy_forest** out);
/* phylo_tree_to_api_tree (core/api.cpp:34-98) of tree `tree` as it is resident on the device (edits applied by dphy_forest_apply_rows
 * included): the three struct vectors are packed on the device, the host adds the table header.  Returns the buffer length (out ==
 * NULL: size query) or a negative dphy_status.  Same content as the reference's writer; FlatBuffers readers follow offsets, so
 * the vectors' placement inside the buffer (ours: header first) is not part of the format. */
int64_t dphy_forest_write_api_tree(dphy_ctx* ctx, dphy_forest* forest, int32_t tree, void* out, size_t cap);
/* The host-order arrays of one tree as they are resident on the device (the inverse of dphy_forest_upload).  dphy_forest_tree_counts
 * gives the sizes; dphy_forest_download_tree WRITES through the array pointers of `out`, which the caller has pointed at buffers of
 * those sizes (parent / child0 / child1 / t: num_nodes; *_off: num_nodes + 1; lists: their totals), and fills the scalars. */
typedef struct dphy_tree_counts {
  int32_t num_nodes, root;
  int64_t num_mutations, num_missation_intervals, num_from_states;
} dphy_tree_counts;
int  dphy_forest_tree_counts(dphy_ctx* ctx, dphy_forest* forest, int32_t tree, dphy_tree_counts* out);
int  dphy_forest_download_tree(dphy_ctx* ctx, dphy_forest* forest, int32_t tree, dphy_emat_host* out);

/* ---- MAPLE input (host only) ------------------------------------------------------------------------------------------------------
 * read_maple (core/io.cpp:98-254): a MAPLE alignment -- reference sequence + per-sample differences -- parsed in one pass over the
 * text into CSR arrays in the shape the SPR studies of a sequence that is not in the tree yet take (dphy_spr_request with
 * DPHY_SPR_X_REL_REF: x_delta_site / x_delta_to and x_missing_start / x_missing_end of sample k are the slices
 * [delta_off[k], delta_off[k+1]) and [miss_off[k], miss_off[k+1]) below), i.e. what build_usher_like_tree feeds them tip by tip
 * (core/phylo_tree.cpp:918-932) without the vector<Tip_desc> in between.  Same tolerances and same dropped samples as the reference
 * (see maple.cpp).  DPHY_ERR_INVALID_ARGUMENT where read_maple throws; dphy_maple_last_error() then holds the message (per thread). */
typedef struct dphy_maple dphy_maple;
typedef struct dphy_maple_view {
  int32_t num_sites, num_tips;
  int64_t num_warnings;               /* calls the reference would have made to its warning hook (dropped samples, bad lines) */
  const uint8_t* ref;                 /* [num_sites] A=0 C=1 G=2 T=3; ambiguous reference letters read as A */
  const double* t_min;                /* [num_tips] Tip_desc::t_min / t_max (float precision), days since 2020-01-01 */
  const double* t_max;
  const int64_t* name_off;            /* [num_tips + 1] into names (not NUL-terminated) */
  const char* names;
  const int32_t* delta_off;           /* [num_tips + 1] Tip_desc::seq_deltas, file order */
  const int32_t* delta_site; const uint8_t* delta_from; const uint8_t* delta_to;
  const int32_t* miss_off;            /* [num_tips + 1] Tip_desc::missations.intervals: ascending, merged */
  const int32_t* miss_start; const int32_t* miss_end;
} dphy_maple_view;
int  dphy_maple_parse(const char* text, size_t len, dphy_maple** out);
int  dphy_maple_get(const dphy_maple* m, dphy_maple_view* out);      /* pointers stay valid until dphy_maple_free */
void dphy_maple_free(dphy_maple* m);
const char* dphy_maple_last_error(void);

/* ---- log G ------------------------------------------------------------------------------------------- */
/* One launch evaluates, for EVERY tree of the forest: calc_lambda_i (core/phylo_tree_calc.cpp:420-436),
 * calc_num_sites_missing_at_every_node (:67-76), calc_log_root_prior (:467-504) and calc_log_G_below_root
 * (:515-543).  Asynchronous on the ctx stream; results stay on the device until fetched. */
int  dphy_forest_eval_log_G(dphy_ctx* ctx, dphy_forest* forest);
/* out arrays are [num_trees]; any may be NULL.  log_G = (includes_run_root ? root_prior : 0) + below_root
 * (Subrun::calc_cur_log_G, core/subrun.cpp:58-68).  Synchronizes the ctx stream. */
int  dphy_forest_get_log_G(dphy_ctx* ctx, dphy_forest* forest, double* log_root_prior, double* log_G_below_root,
                           double* log_G);
/* calc_lambda_i result of the last eval for one tree, host node order, out[num_nodes]. */
int  dphy_forest_get_lambda_i(dphy_ctx* ctx, dphy_forest* forest, int32_t tree, double* out);
/* calc_num_sites_missing_at_every_node of the last eval for one tree, host node order. */
int  dphy_forest_get_num_sites_missing(dphy_ctx* ctx, dphy_forest* forest, int32_t tree, int32_t* out);

/* One-shot, host-buffers-in / host-scalars-out evaluation of a single EMAT (the call the C++ adapter makes for
 * Subrun::calc_cur_log_G when nothing is resident): uploads, evaluates, downloads.  lambda_i may be NULL. */
int  dphy_log_G_host(dphy_ctx* ctx, const dphy_emat_host* tree, const dphy_sites_host* sites,
                     double* log_root_prior, double* log_G_below_root, double* lambda_i);

/* ---- coalescent prior ---------------------------------------------------------------------------------------------------------------
 * Log-density of the node times of EVERY tree of the forest under the coalescent with exponential growth, N(t) = n0 exp(g (t - t0)),
 * in the time convention of the tree: t grows toward the present (a node is never earlier than its parent), so g > 0 is a population
 * growing toward the present.  n0 is in the unit of t, g in its inverse.  Tips are sampling events and add a lineage going back in
 * time; inner nodes are coalescences and remove one.  With k lineages on an interval (a, b) between consecutive events,
 *   out[k] = sum over inner nodes c of -log N(t_c)  -  sum over intervals of C(k, 2) * exp(-g (a - t0)) / n0 * (1 - exp(-g (b - a))) / g
 * (the last factor is b - a at g = 0; the device evaluates it as -expm1(-g (b - a)) / g, so tiny |g| loses nothing to cancellation).
 * Tied times give the same value in any order.  out[num_trees]; DPHY_ERR_INVALID_ARGUMENT unless n0 > 0 and n0, g, t0 are finite.
 * Synchronous: the node times as they are on the device (after dphy_forest_set_node_times / dphy_forest_apply_rows), one double per
 * tree back to the host.  Each tree is taken as a whole tree: for the parts of a partitioned tree the value is not that tree's prior. */
int  dphy_forest_log_coalescent_prior(dphy_ctx* ctx, dphy_forest* forest, double n0, double g, double t0, double* out);

/* ---- clade support and the maximum clade credibility (MCC) tree ----------------------------------------------------------------------
 * A clade table counts, over every tree added to it, how many trees contain each clade, and sums the clade's node time over them.
 *   Tips: a tip is a node with child0 == -1, identified by its HOST node index.  The first add fixes the table's tip set: N nodes per
 *     tree and which indices are tips.  Every tree later added or scored must have the same N and exactly the same tip indices;
 *     otherwise the call returns DPHY_ERR_INVALID_ARGUMENT before anything is changed.  Tips are not matched by name: renumber first.
 *   Clades: the clade of node v is the set of tips below it, v included -- tips, inner nodes and the root all have one.  Trees are
 *     rooted, so a binary tree contains each clade at most once.
 *   Key: a clade is keyed by 128 bits, two independent wrapping uint64 sums over its tips i of k_j(i) = splitmix64((uint64)i << 1 | j),
 *     j = 0 and 1, where splitmix64(x): z = x + 0x9e3779b97f4a7c15; z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9;
 *     z = (z ^ (z >> 27)) * 0x94d049bb133111eb; return z ^ (z >> 31)  (one step of SplitMix64 from state x).  Two different tip sets
 *     share a key with probability about 2^-128 per pair; such a collision is NOT detected (the two clades would count as one).
 *   Table: per distinct clade, count = how many of the trees added so far contain it, and the sum of its node time over them.
 *     T = the number of trees added.  Memory: 32 B per distinct clade plus a bitmap of N bits (dphy_clade_table_info's device_bytes);
 *     an add also takes stream-ordered scratch of about 90 B per node of the forest plus 64 B per clade of the merged table.
 *   Score: score(tree) = sum over every node v of log(count(v) / T), the log of the product of clade frequencies TreeAnnotator
 *     maximises for its MCC tree.  Tips and the root add exactly 0; a tree with a clade the table has never seen scores -inf.
 *   Node support (one tree, host node order): count(v) (0 for an unseen clade) and mean_t(v) = sum of t / count (NaN if count == 0).
 *   The MCC tree is the argmax of the scores over the added trees; its node support annotates it (frequency count / T, mean clade time).
 * Every call is synchronous with host results, and a table is used with the ctx that made it.  dphy_clade_table_add takes every tree of
 * the forest as it is resident now (after dphy_forest_set_node_times / dphy_forest_apply_rows); the table keeps no pointer to the forest,
 * so the forest may be edited or destroyed afterwards.  Adding forests one after another gives the counts of one forest holding all
 * their trees, which is how a posterior larger than HBM is summarised: add every batch, then score every batch.  The same sequence of
 * adds gives bit-identical mean_t and scores: time sums run in tree order within a batch, the table's sum before the batch's.
 * DPHY_ERR_OUT_OF_MEMORY for a failed allocation, the table then unchanged.  Scoring or node support before any add is
 * DPHY_ERR_INVALID_ARGUMENT. */
typedef struct dphy_clade_table dphy_clade_table;
int  dphy_clade_table_create(dphy_ctx* ctx, dphy_clade_table** out);
void dphy_clade_table_destroy(dphy_ctx* ctx, dphy_clade_table* table);
int  dphy_clade_table_add(dphy_ctx* ctx, dphy_clade_table* table, dphy_forest* forest);
int  dphy_clade_table_info(const dphy_clade_table* table, int64_t* num_trees, int64_t* num_clades, int64_t* device_bytes);
int  dphy_clade_table_score(dphy_ctx* ctx, dphy_clade_table* table, dphy_forest* forest, double* out /* [num_trees] */);
int  dphy_clade_table_node_support(dphy_ctx* ctx, dphy_clade_table* table, dphy_forest* forest, int32_t tree,
                                   int64_t* count /* [num_nodes] */, double* mean_t /* [num_nodes] */);

/* ---- tallies ------------------------------------------------------------------------------------------ */
/* calc_num_muts / _ab / calc_T + the log-G pieces for every tree; out[num_trees]. */
int  dphy_forest_calc_tallies(dphy_ctx* ctx, dphy_forest* forest, dphy_tallies* out);
/* calc_num_muts_beta_ab (core/phylo_tree_calc.cpp:599-610) -> out[P*16] for one tree */
int  dphy_forest_calc_num_muts_beta_ab(dphy_ctx* ctx, dphy_forest* forest, int32_t tree, int32_t* out);
/* calc_num_muts_l (:612-622) -> out[L];  calc_num_muts_l_ab (:624-634) -> out[L*16] (either may be NULL) */
int  dphy_forest_calc_num_muts_l(dphy_ctx* ctx, dphy_forest* forest, int32_t tree, int32_t* out_l, int32_t* out_l_ab);
/* calc_Ttwiddle_beta_a (:288-369) -> out[P*4] for one tree */
int  dphy_forest_calc_Ttwiddle_beta_a(dphy_ctx* ctx, dphy_forest* forest, int32_t tree, double* out);
/* calc_Ttwiddle_l (:176-222) -> out_l[L];  calc_T_l_a (:130-174) -> out_l_a[L*4] (either may be NULL) */
int  dphy_forest_calc_Ttwiddle_l(dphy_ctx* ctx, dphy_forest* forest, int32_t tree, double* out_l, double* out_l_a);
/* The per-site inputs of the reference's global Gibbs moves for EVERY tree of the forest in one call (what Run gathers from
 * its subruns each cycle for gibbs_sample_all_nus / alpha_moves, core/run.cpp:1105-1235): row k of out_Ttwiddle_l is
 * calc_Ttwiddle_l of tree k (core/phylo_tree_calc.cpp:176-222), row k of out_num_muts_l its calc_num_muts_l (:612-622).
 * Rows are `ld` elements apart (ld >= every tree's number of sites); either output may be NULL.  All trees' kernels and copies
 * are enqueued back to back with one synchronization at the end. */
int  dphy_forest_calc_site_tallies(dphy_ctx* ctx, dphy_forest* forest, int64_t ld, double* out_Ttwiddle_l, int32_t* out_num_muts_l);

/* The quantities the reference sums over its subruns once per cycle (Run::check_global_and_local_totals_match and the inputs of
 * the global moves, core/run.cpp:340-357,437-453), summed over the trees of this forest and packed as doubles in DEVICE memory
 * so that ranks holding different partition parts combine them with ONE all-reduce (NCCL over NVLink):
 *   d_out[0] = sum log_G   [1] = sum T   [2] = sum num_muts   [3..19) = sum num_muts_ab   [19 .. 19+4P) = sum Ttwiddle_beta_a
 * cap >= 19 + 4 P (DPHY_CYCLE_TALLIES_LEN).  Asynchronous on the ctx stream; no host round trip. */
#define DPHY_CYCLE_TALLIES_LEN(P) (19 + 4 * (P))
int  dphy_forest_cycle_tallies_device(dphy_ctx* ctx, dphy_forest* forest, double* d_out, int32_t cap);

/* ---- SPR regraft study -------------------------------------------------------------------------------- */
/* Runs a batch of SPR studies (Spr_study_builder::seed_fill_from + Spr_study ctor) in one pass over the forest.
 * Regions of study i are emitted in the reference's DFS order (core/spr_study.cpp:26-128) at
 * regions[summary[i].region_offset ...].  Asynchronous; results stay on the device. */
int  dphy_spr_study_batch(dphy_ctx* ctx, dphy_forest* forest, int32_t num_requests, const dphy_spr_request* requests,
                          dphy_spr_batch** out);
void dphy_spr_batch_destroy(dphy_ctx* ctx, dphy_spr_batch* batch);
/* summaries[num_requests]; synchronizes. */
int  dphy_spr_batch_get_summaries(dphy_ctx* ctx, dphy_spr_batch* batch, dphy_spr_summary* summaries);
/* total regions over the batch (after synchronizing) */
int64_t dphy_spr_batch_total_regions(dphy_ctx* ctx, dphy_spr_batch* batch);
/* copies the regions of study `request` (or of all studies if request < 0) to out[cap]; returns count or <0 */
int64_t dphy_spr_batch_get_regions(dphy_ctx* ctx, dphy_spr_batch* batch, int32_t request,
                                   dphy_candidate_region* out, int64_t cap);
/* Spr_study::pick_nexus_region (core/spr_study.cpp:404-422) with the caller's uniform draw r in [0,sum_W): the device replays
 * the reference's scan (if W_i >= r pick i, else r -= W_i) in the same order, so the index is the one the reference's code returns
 * for these weights; out_region_idx[i] for every study i given r[i]. */
int  dphy_spr_batch_pick_nexus_regions(dphy_ctx* ctx, dphy_spr_batch* batch, const double* r, int32_t* out_region_idx);
/* Spr_study::find_region (core/spr_study.cpp:474-484) for study `request` */
int  dphy_spr_batch_find_region(dphy_ctx* ctx, dphy_spr_batch* batch, int32_t request, int32_t branch, double t,
                                int32_t* out_region_idx);
/* The Spr_study constructor on its own (core/spr_study.cpp:226-385): (re)computes log_W_over_Wmax / W_over_Wmax, log_Wmax and
 * sum_W_over_Wmax of every study of the batch from its enumerated regions with params[num_requests].  Asynchronous. */
int  dphy_spr_batch_set_weights(dphy_ctx* ctx, dphy_spr_batch* batch, const dphy_spr_weight_params* params);
/* writes ONLY the (log_W_over_Wmax, W_over_Wmax) fields of out[0..count) (records already filled by dphy_spr_batch_get_regions
 * keep their other fields); returns count or <0 */
int64_t dphy_spr_batch_get_region_weights(dphy_ctx* ctx, dphy_spr_batch* batch, int32_t request,
                                          dphy_candidate_region* out, int64_t cap);
/* Spr_study::log_alpha_in_region (core/spr_study.cpp:486-549): log proposal density of attaching at time t in region_idx. */
int  dphy_spr_batch_log_alpha_in_region(dphy_ctx* ctx, dphy_spr_batch* batch, int32_t request, int32_t region_idx, double t,
                                        double* out);
/* Regularized upper incomplete gamma Q(a,x) and its inverse in x, fp64, evaluated on the device for n argument pairs: the two
 * special functions behind the above-root region (safe_gamma_q / safe_gamma_q_inv, core/safe_gamma_math.h:46-83, which the
 * reference takes from Boost.Math).  Spr_study::pick_time_in_region (core/spr_study.cpp:424-471) draws its uniform on the host
 * between Q(a, x_max) and Q(a, x_min) and inverts here. */
int  dphy_gamma_q(dphy_ctx* ctx, int32_t n, const double* a, const double* x, double* out);
int  dphy_gamma_q_inv(dphy_ctx* ctx, int32_t n, const double* a, const double* q, double* out);

/* ---- placement of new samples (maximum parsimony) ---------------------------------------------------------------------------------
 * Where on tree `tree` does each new sequence go, at how many mutations, and how many equally good places are there -- the per-tip step
 * of build_usher_like_tree (core/phylo_tree.cpp:918-932), UShER-style placement of fresh samples onto an existing or posterior tree.
 * For sample k, take the regions dphy_spr_study_batch enumerates for the request
 *   {tree, X = -1, x_state_mode = DPHY_SPR_X_REL_REF, start = (root, #root mutations), max_muts_from_start = INT32_MAX,
 *    t_X = DBL_MAX, lambda_X = 0, can_change_root, x deltas / missing intervals = sample k's}
 * (the region list of the reference's unbounded study from the root; core/spr_study.cpp:9-209).  Then out[k] holds
 *   min_muts = the least min_muts over those regions,  num_best = how many regions attain it,
 *   (branch, mut_idx) = the FIRST region attaining it in the study's emission order;
 * and, with max_best > 0, best[k * max_best + i] the first max_best such regions in emission order as full records (branch, mut_idx,
 * t_min, t_max, min_muts; weights 0); unused slots are zero with branch = -1.  A tree without regions (a lone root and
 * can_change_root == 0) gives min_muts = -1, num_best = 0, branch = mut_idx = -1.  Everything equals what the study gives, bit for bit.
 * Samples are those of a DPHY_SPR_X_REL_REF request: x = the reference overlaid with the deltas in array order (a later delta of
 * the same site wins); a site inside any interval is missing (intervals may overlap and come in any order).  Sample k's deltas are
 * [delta_off[k], delta_off[k+1]) and its intervals [miss_off[k], miss_off[k+1]) -- the arrays dphy_maple_view gives.
 * Validation as for a request, before anything is written: DPHY_ERR_OUT_OF_RANGE for a tree index, a site outside [0, L), a state
 * above 3 or an interval outside 0 <= start < end <= L; DPHY_ERR_INVALID_ARGUMENT for decreasing offsets or missing arrays.
 * Precondition (as for the study's own delta arithmetic): every mutation's `from` is the state of the sequence above it.
 * Cost: a per-tree index (mutations by site with the block of regions below each, and a min / count segment tree over the regions'
 * reference Hamming potential; 16 B per mutation + 8 B per segment-tree entry, 2 x the power of two >= R entries) is built by the first call on the tree and kept with the
 * forest (dphy_forest_apply_rows drops it, dphy_forest_set_node_times needs no rebuild: times are read when the records are made);
 * per sample the work is O(|A| log R), A = the tree's mutations at the sample's delta and missing sites, R = the number of regions.
 * Synchronous: host arrays in, host results out.
 * Dated placement, dphy_forest_place_dated_samples: sample k may only go where the tree is earlier than its date limit t_X[k].  Its
 * regions are those above after remove_regions_in_Xs_future (core/spr_study.cpp:211-224) with t_X = t_X[k]: a region with
 * t_min >= t_X[k] is dropped (a tie too), and t_max is clipped to t_X[k] where it is larger; the outputs are then as above over the
 * regions left, bit for bit, best records carrying the clipped t_max.  t_X[k] = +inf or DBL_MAX keeps every region (the undated
 * result); t_X[k] <= -DBL_MAX keeps none, not even the root region (t_min = -DBL_MAX), and gives min_muts = -1, num_best = 0,
 * branch = mut_idx = -1.  A sample with a date range passes the end it stands for (usually t_max of dphy_maple_view, the latest
 * time it could have been taken).  Validation, outputs and precondition as for dphy_forest_place_samples, and before anything is
 * written: DPHY_ERR_INVALID_ARGUMENT for t_X == NULL with num_samples > 0 or a NaN in it.  Node and mutation times are compared as
 * numbers (none may be NaN).  Cost: a dated part of the per-tree index, a merge-sort tree over the regions keyed by t_min (12 B per
 * entry, lg2(P2) levels of P2 entries, P2 = the power of two >= R, plus 8 B per region), is built by the first dated call that
 * drops a region of the tree and kept with the forest (dphy_forest_device_bytes includes it; dphy_forest_set_node_times marks it
 * stale and the next such call rebuilds it in the same memory); a sample that drops a region costs O(|A| log R) as well. */
typedef struct dphy_sample_set {
  int32_t num_samples;
  int32_t reserved;
  const int32_t* delta_off;           /* [num_samples + 1] */
  const int32_t* delta_site; const uint8_t* delta_to;
  const int32_t* miss_off;            /* [num_samples + 1] */
  const int32_t* miss_start; const int32_t* miss_end;
} dphy_sample_set;
typedef struct dphy_placement {
  int32_t min_muts, num_best, branch, mut_idx;   /* branch: host node index */
} dphy_placement;
int  dphy_forest_place_samples(dphy_ctx* ctx, dphy_forest* forest, int32_t tree, const dphy_sample_set* samples, int32_t can_change_root,
                               int32_t max_best, dphy_placement* out, dphy_candidate_region* best /* [num_samples * max_best] or NULL */);
int  dphy_forest_place_dated_samples(dphy_ctx* ctx, dphy_forest* forest, int32_t tree, const dphy_sample_set* samples,
                                     const double* t_X /* [num_samples] */, int32_t can_change_root, int32_t max_best,
                                     dphy_placement* out, dphy_candidate_region* best /* [num_samples * max_best] or NULL */);

/* ---- tree partitioning (one or more parts per GPU) ------------------------------------------------------------- */
/* generate_random_partition_stencil (core/tree_partitioning.h:139-194): up to num_parts-1 cut points.  The coin flips are the
 * reference's: std::bernoulli_distribution{0.5} drawn from std::mt19937{(uint32_t)seed} through absl::BitGenRef, interleaved with
 * the lazy randomized post-order traversal (core/tree.h:320-365), so the same seed gives the reference's cut points. */
typedef struct dphy_partition dphy_partition;
int  dphy_partition_generate_stencil(const dphy_emat_host* tree, int32_t num_parts, uint64_t seed, int32_t* cut_points,
                                     int32_t* num_cut_points);
/* partition_tree + the per-part Phylo_tree construction of Run::repartition (core/tree_partitioning.h:196-239,
 * core/run.cpp:133-176).  The last part is the one holding the tree's root. */
int  dphy_partition_split(const dphy_emat_host* tree, const dphy_sites_host* sites, int32_t num_cut_points,
                          const int32_t* cut_points, dphy_partition** out);
int32_t dphy_partition_num_parts(const dphy_partition* p);
const dphy_emat_host* dphy_partition_part(const dphy_partition* p, int32_t i);
/* orig_tree_index of every node of part i (core/tree_partitioning.h:20-34) */
const int32_t* dphy_partition_orig_index(const dphy_partition* p, int32_t i);
/* reassemble_tree / Run::reassemble (core/tree_partitioning.cpp:55-83, core/run.cpp:195-256): the whole tree with every part's
 * times, lists and topology transposed back through orig_tree_index.  parts[i] corresponds to dphy_partition_part(p, i) (same
 * node count; contents may have been edited by local moves).  The result is owned by `p` (valid until the next reassemble or
 * dphy_partition_free); NULL on a shape mismatch. */
const dphy_emat_host* dphy_partition_reassemble(dphy_partition* p, const dphy_emat_host* whole, int32_t num_parts,
                                                const dphy_emat_host* parts);
void dphy_partition_free(dphy_partition* p);

const char* dphy_version(void);

#ifdef __cplusplus
}
#endif
#endif /* DELPHY_B200_H_ */
