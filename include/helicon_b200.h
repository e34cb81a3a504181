/* helicon_b200 -- C ABI of the B200 (sm_100a) denovo3D solve+score hot path.
 *
 * Drop-in boundary for jianglab/helicon's denovo3D solver.  The reference is
 * pure Python (src/helicon/webApps/denovo3D/solver_linear_regression.py, "SLR"
 * below); a maintainer binds this library with ctypes (see INTEGRATION.md) from
 * the bodies of the reference functions named beside each entry point.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on
 * success or a negative hb2_status; hb2_last_error() gives the message.  All
 * host buffers are caller-owned.  `stream` is a cudaStream_t passed as void*
 * (NULL = legacy default stream).  Nothing here throws or calls back.
 *
 * Division of labour (DESIGN.md): the Python host plans the candidate exactly
 * as the reference does (ordered symmetry copies, ordered symmetry pairs,
 * rotation matrices from scipy, column->slice assignment); every O(pixels),
 * O(voxels) or O(iterations) step runs in CUDA kernels behind this ABI.
 */
#ifndef HELICON_B200_H
#define HELICON_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  HB2_OK = 0,
  HB2_ERR_CUDA = -1,        /* a CUDA runtime call failed */
  HB2_ERR_ARG = -2,         /* bad argument */
  HB2_ERR_GEOMETRY = -3,    /* geometry the path does not support (see message) */
  HB2_ERR_NO_DEVICE = -4,   /* no CUDA device: there is no CPU fallback */
  HB2_ERR_STATE = -5,       /* call order violated */
  HB2_ERR_CAPACITY = -6     /* an internal table overflowed */
} hb2_status;

/* per-candidate result flags (bit mask in hb2_result.flags) */
#define HB2_FLAG_TIE_XY 1u       /* an in-plane sample lies within 1e-9 of a rounding boundary (SURVEY F8) */
#define HB2_FLAG_TIE_Z 2u        /* a column's Z lies within 1e-9 of a rounding boundary (host planner sets it) */
#define HB2_FLAG_BOUNDED 4u      /* the bounded (TRF) branch ran (SLR:246-270, scipy lsq_linear) */
#define HB2_FLAG_NO_ROWS 8u      /* no data rows */
#define HB2_FLAG_TIE_Z_EXACT 16u /* column->slice ties resolved per sample from the reference's z table (exact) */
#define HB2_FLAG_NOT_CONVERGED 32u /* hb2_batch_solve_model: max_iter ended the fit before its stop rule held */

typedef struct hb2_problem hb2_problem; /* one image + in-plane geometry, shared by many candidates */
typedef struct hb2_batch hb2_batch;     /* a set of candidates solved together */

/* In-plane geometry shared by all candidates of a problem.
 * Mirrors the arguments of SLR:1304-1322 (build_A_data_matrix) and SLR:847-859
 * (build_A_helical_sym_matrix) that do not depend on (twist, rise, csym). */
typedef struct {
  int32_t ny, nx;          /* image shape */
  double scale2d_to_3d;    /* s */
  int32_t D2, L2;          /* reconstruct_diameter_2d_pixel, reconstruct_length_2d_pixel */
  int32_t D3;              /* reconstruct_diameter_3d_pixel */
  double rmin;             /* reconstruct_diameter_3d_inner_pixel / 2 (SLR:116) */
  int32_t rmax;            /* D3 // 2 - 1 (SLR:117) */
  int32_t interpolation;   /* 0 = "nn" (SLR:1514-1557, 1142-1218); 1 = "linear": a hint for the internal voxel order only
                            * (row-major tiles suit the footprint gathers of the matrix-free trilinear rows); every
                            * batch type works on either order */
} hb2_geometry;

/* One candidate (twist, rise, csym).  Views/pairs are slices of the flat
 * arrays given to hb2_batch_create, in the reference's order. */
typedef struct {
  int32_t view_begin, view_count;   /* data-operator symmetry copies actually used (after the row-count early stop, SLR:1647) */
  int32_t pair_begin, pair_count;   /* symmetry pairs in sorted_hsym_csym_pairs order (SLR:1749-1791) */
  int64_t min_sym_pairs;            /* SLR:168-170 */
  int32_t positive;                 /* resolved positive-constraint rule (SLR:352-355) */
  uint32_t flags_in;                /* HB2_FLAG_TIE_Z from the host planner */
} hb2_candidate;

/* One symmetry copy (h,c) of the data operator: in-plane rotation = angle
 * table entry `angle`, and the image column k feeding each (z-slice, slot):
 * colk[(z*MC + mc)] = k or -1, stored at col_begin in the flat colk array. */
typedef struct {
  int32_t angle;       /* index into the batch's unique-angle table */
  int32_t col_begin;   /* offset into colk (L3*MC entries) */
  int32_t tie;         /* -1, or index of the tie view this slot belongs to (hb2_batch_set_ties): colk then lists
                          the image COLUMNS of column slots tie_slot0 .. tie_slot0 + L3*MC - 1 */
  int32_t tie_slot0;
  int32_t dup_of;      /* -1, or the candidate-relative index of an EARLIER view with the same (h, c): the reference's
                          Halton re-indexing repeats symmetry copies (SLR:1559-1571), their rows are identical; the
                          projector kernels compute them once (forward: copy, adjoint: weight) */
  int32_t mult;        /* 1 + number of later duplicates of this view (0 for a duplicate) */
} hb2_view;

/* One symmetry pair ((h_i,c_i),(h_j,c_j)) of the regulariser (SLR:1223-1243):
 * rotation matrix entries (M00, M10) from scipy for each member and the z
 * shift rise_pixel*h. */
typedef struct {
  double ci, si, zi;
  double cj, sj, zj;
} hb2_pair;

typedef struct {
  int32_t max_iter;        /* lsmr_maxiter (SLR:266) = 1000 */
  double atol, btol;       /* 1e-2 * tol = 1e-4 (scipy lsq_linear.py:318-326) */
  double conlim;           /* 1e8 (scipy lsmr default) */
  int32_t check_every;     /* host polls convergence every this many iterations */
  int32_t clip_pred;       /* thresh_fraction >= 0: clip reprojection at 0 before scoring (SLR:502-503) */
  int32_t trf_max_iter;    /* max_iter of the bounded branch (SLR:241) = 200 */
  double trf_tol;          /* tol (SLR:240) = 1e-2 */
  int32_t fixed_iters;     /* >0: run exactly this many LSMR iterations, ignore stop tests (tests only) */
  int32_t profile;         /* 1: bracket every kernel launch with CUDA events (per-kernel-class device time) */
  int32_t norm_mode;       /* how LSMR's float32 norms ||u||, ||v|| (lsmr.py:239-340, numpy.linalg.norm) are formed:
                              1 (default) = as the reference EXECUTES them: numpy -> OpenBLAS sdot with 64 sequential
                              float32 FMA accumulators (biased low by ~1e-5 at 1e7 elements; LSMR amplifies that to
                              ~6e-3 in x), 0 = exactly rounded */
} hb2_solve_options;

typedef struct {
  float score;             /* cosine similarity of A_data x vs b_data (SLR:484-525, lib/analysis.py:802-821) */
  int32_t itn;             /* LSMR iterations of the unbounded solve */
  int32_t istop;           /* scipy lsmr istop code */
  int32_t trf_nit;         /* outer iterations of the bounded branch (0 if not taken) */
  uint32_t flags;
  int32_t n_data_rows;     /* real (unpadded) data rows */
  int32_t n_sym_rows;
  float normr, normar, normA, normx;
} hb2_result;

const char* hb2_last_error(void);
int hb2_device_count(void);
const char* hb2_build_info(void);

/* ---- streams / memory ------------------------------------------------------
 * Additive helpers for the batched grid driver (no reference counterpart: the
 * reference runs one candidate per ThreadPoolExecutor worker, app.py:2455-2523).
 * A batch does all its work on the stream given to hb2_batch_begin; batches on
 * different non-blocking streams overlap (setup of the next batch under the
 * solve of the current one).  Batch memory comes from the device's stream-
 * ordered pool and is kept cached between batches; hb2_device_trim returns it. */
int hb2_stream_create(int device, void** stream_out);
int hb2_stream_destroy(int device, void* stream);
int hb2_device_trim(int device);

/* ---- problem ------------------------------------------------------------- */
/* Uploads the image, crops pixel_vals (SLR:1706-1708) and builds the disk
 * tables of helicon.get_cylindrical_mask (lib/analysis.py:731-774). */
int hb2_problem_create(hb2_problem** out, const float* image_host, const hb2_geometry* geom, int device, void* stream);
void hb2_problem_destroy(hb2_problem* p);
int hb2_problem_ndisk(const hb2_problem* p);
/* rank table of the data grid: out[D2*D2], rank of voxel (y,x) in C order inside the disk, or -1 */
int hb2_problem_rank_table(const hb2_problem* p, int32_t* out_host);

/* ---- batch: step 1, in-plane maps for the batch's unique angles ---------- */
/* cos_sin[2*a+0] = M00, cos_sin[2*a+1] = M10 of scipy Rotation.from_euler('z', angle_a).
 * Builds the sample->voxel map of every angle (replaces the numba loop
 * SLR:1514-1557 and Rotation.apply SLR:1614-1620 for tilt=psi=dy=0).
 * Outputs (host, may be NULL): nvalid_rays[a] = rays with >=1 hit,
 * tie_samples[a] = samples within 1e-9 of a rounding boundary. */
int hb2_batch_begin(hb2_batch** out, hb2_problem* p, int32_t L3, int32_t MC, int32_t n_angles, const double* cos_sin,
                    int32_t* nvalid_rays, int32_t* tie_samples, void* stream);
/* ray validity per angle, out[n_angles*D2] (1 = the ray has projection data, SLR:1547) */
int hb2_batch_ray_valid(hb2_batch* b, uint8_t* out_host);
/* sample->voxel map of one angle, out[D2*D2] int32 (disk rank or -1), row j, depth i */
int hb2_batch_angle_map(hb2_batch* b, int32_t angle, int32_t* out_host);

/* In-plane tie views (SURVEY F8): at view angles where a sample coordinate cos*x0 + sin*y0 is a half-integer (30, 60,
 * ... degrees; angle 0/90/180 when s = 0.5) the reference's rounding follows the last-bit noise of its coordinate
 * table (SLR:1712-1719), which depends on (image column k, depth sample i).  For such a view the host requests one
 * EXACT map per image column: cos_sin[2e..] as in hb2_batch_begin, x0rows[e*D2 + i] = the table's x coordinate of
 * sample i in that column (taken from the same scipy call the reference makes).  The maps are appended to the angle
 * table (indices n_angles .. n_angles + n_extra - 1) and used by single-column views.  nvalid_rays[n_extra] out.
 * Call between hb2_batch_begin and hb2_batch_create. */
int hb2_batch_add_exact_maps(hb2_batch* b, int32_t n_extra, const double* cos_sin, const double* x0rows,
                             int32_t* nvalid_rays);

/* Tie views (SURVEY F8): a symmetry copy whose Z = s*(k - L2//2) - h*rise + L3//2 is a half-integer for its
 * columns lets every SAMPLE round by the last-bit noise of the reference's coordinate table (SLR:1712-1719), so a
 * row (column k, ray j) draws from two neighbouring slices.  The host resolves it from that table:
 * zlo[t*TS + s] = lower slice of column slot s (may be -1; <= -100 = unused slot), up[(t*TS + s)*D2 + i] in {0,1}
 * = sample i of the slot lands in zlo + up, rowvalid[(t*TS + s)*D2 + j] = the row exists.  Call between
 * hb2_batch_begin and hb2_batch_create; views refer to tie t through hb2_view.tie. */
int hb2_batch_set_ties(hb2_batch* b, int32_t n_tie, int32_t TS, const int8_t* zlo, const uint8_t* up,
                       const uint8_t* rowvalid);

/* ---- explicit data rows: general orientation and/or trilinear interpolation ---------------------------------
 * build_A_data_matrix (SLR:1301-1654) outside the grid-search case (tilt = psi = dy = 0, nearest neighbour), where a ray
 * crosses slices and the matrix-free projector does not apply: the rows are built ON THE GPU by the reference's float64
 * operation sequence (coords0[:,1] -= dy; R('yx',(tilt,psi)).apply(inverse); per copy R('z',angle).apply(inverse),
 * z -= h*rise; + n//2 offsets; round()/int(); SLR:1390-1395, 1576-1581, numba loops 1403-1557) into a CSR and its
 * transpose kept on the device; the solvers apply them in place of the projector kernels.  The batch then holds ONE
 * candidate whose hb2_candidate.view_count pseudo views (hb2_view.tie = 0, colk = -1) cover ceil(n_rows /
 * (D2 * ZMP)) chunks of the padded row space.
 * rot_yx / copy_mats: scipy's as_matrix() entries, row-major; xtab / ztab [L2*D2]: the reference's coordinate
 * tables (x and z of sample (column k, depth i)); copies in the reference's order (Halton re-indexed); the early stop
 * SLR:1647 is applied here.  Call between hb2_batch_begin (one dummy angle) and hb2_batch_create. */
typedef struct {
  int32_t interpolation;   /* 0 = "nn", 1 = "linear" (SLR:1403-1510) */
  double dy_pixel;
  double rot_yx[9];        /* Rotation.from_euler("yx", (tilt, psi), degrees=True).as_matrix() */
} hb2_explicit_geometry;
int hb2_batch_explicit_rows(hb2_batch* b, const hb2_explicit_geometry* g, int32_t n_copies, const double* copy_mats,
                            const double* zshift, const double* xtab, const double* ztab, int64_t min_projection_lines,
                            int32_t* copies_used, int32_t* rows_per_copy, int64_t* n_rows, int64_t* nnz);
/* Half sets for explicit rows (fsc_test): keep only the rows whose pixel id k*D2 + j is set in mask[L2*D2] (NULL: all);
 * applied after the early stop, as the reference splits the finished matrix (SLR:441-444).  Call before
 * hb2_batch_explicit_rows. */
int hb2_batch_explicit_pixel_mask(hb2_batch* b, const uint8_t* mask);
/* the rows as CSR in the reference's voxel order (entries unmerged: a voxel hit twice by one ray appears twice),
 * right-hand side and pixel ids (SLR:1651-1654); any pointer may be NULL */
int hb2_batch_explicit_export(hb2_batch* b, int64_t* indptr, int32_t* indices, float* data, float* b_out, int32_t* pid_out);

/* Trilinear symmetry rows (build_A_helical_sym_matrix with interpolation "linear", SLR:910-1138 + pair loop
 * 1221-1287), built on the GPU: per ordered pair and mask voxel the two images (scipy Rotation.apply arithmetic),
 * int() corners, all 16 corners valid, corner origins >= 3 apart on every axis, first-seen-wins on the rounded image
 * pair, 8 + 8 weights (incl. the reference's corner-110 expression xf*yf*(1-xf)).  pair_mats[p*12..] = M00, M01, M10,
 * M11, M22 of scipy's matrix and rise*h for member i, then the same for member j; pairs in sorted_hsym_csym_pairs
 * order; stops when the row count reaches min_sym_pairs.  In a batch with explicit data rows they are appended to
 * them (b = 0, not scored) and the candidate is created with pair_count = 0.  Call before hb2_batch_create. */
int hb2_batch_explicit_sym_rows(hb2_batch* b, int32_t n_pairs, const double* pair_mats, int64_t min_sym_pairs,
                                int64_t* n_rows);
/* the rows as 16 (column, weight) entries each, columns in the reference's voxel order; either may be NULL */
int hb2_batch_explicit_sym_export(hb2_batch* b, int32_t* cols, float* weights);

/* ---- matrix-free trilinear rows (interpolation "linear" in the grid-search case) -----------------------------
 * build_A_data_matrix with interpolation "linear" (numba loop SLR:1403-1510) at tilt = psi = dy = 0 and
 * scale2d_to_3d = 1: the row of (symmetry copy, image column k, ray j) factors into an in-plane bilinear footprint of
 * the ray -- a function of the view angle only, shared by the candidates of a batch -- times a two-slice blend
 * a_k P[zi_k] + b_k P[zi_k + 1] that depends on the column only (csrc/hb2_bilinear.cuh).  A batch of this kind holds
 * MANY candidates; the explicit matrix of hb2_batch_explicit_rows is never built.
 *
 * hb2_bilinear_map: m00..m22 = entries of Rotation.from_euler("z", angle, degrees=True).as_matrix() (SLR:1576); xrow /
 * zrow = -1 for a regular map, or the row of the coordinate tables passed along (xrows / zrows [n_tab_rows][D2] =
 * rows of the reference's x / z tables, SLR:1712-1719, for ONE image column) for an EXACT map: where sample
 * coordinates are integer-valued (angles 0 / 90 / 180 / 270, integer h * rise) the reference's int() truncation
 * follows the last-bit noise of those tables per (column, sample); zrow >= 0 additionally applies the reference's
 * slice-range test per sample with zshift = h * rise_pixel (SLR:1578, 1421-1428).
 * build_tables = 0 only reports, per map, the number of rays with data (SLR:1496) and the number of samples within 1e-9
 * of an integer coordinate (the host then replaces such views by single-column views with exact maps); 1 builds the
 * maps the kernels use (call once with all maps) and, if content_hash != NULL, a 64-bit hash of every map's content
 * (exact maps of neighbouring columns mostly come out identical -- the table noise has one sign per side of the image
 * centre -- and the host merges such columns into one view).  Call between hb2_batch_begin (one dummy angle) and
 * hb2_batch_create. */
typedef struct {
  double m00, m01, m10, m11, m22, zshift;
  int32_t xrow, zrow;
} hb2_bilinear_map;
int hb2_batch_bilinear_maps(hb2_batch* b, int32_t n_maps, const hb2_bilinear_map* maps, int32_t n_tab_rows,
                            const double* xrows, const double* zrows, int32_t build_tables, int32_t* nvalid_rays,
                            int32_t* tie_samples, uint64_t* content_hash);
/* ray validity of the maps built by hb2_batch_bilinear_maps(build_tables = 1), out[n_maps*D2] */
int hb2_batch_bilinear_ray_valid(hb2_batch* b, uint8_t* out_host);
/* Views of the batch, indexed like the views handed to hb2_batch_create (all of them pseudo views: hb2_view.tie = 0,
 * colk = -1): view_map[v] >= 0 -> bilinear view of that map, colk[v*ZMP + t] = image column of slot t (-1: unused),
 * ab[(v*ZMP + t)*2 ..] = (a, b) of its slice blend: row = a P[t-1] + b P[t] for t >= 1, a P[0] + b P[1] for t = 0
 * (a column with Z in (-1, 0): int() truncates toward zero, SLR:1418); view_map[v] = -1 -> pseudo view that holds
 * rows_per_view of the candidate's trilinear symmetry rows.  cand_nview[c] = bilinear views of candidate c (they come
 * first in its view range). */
int hb2_batch_bilinear_views(hb2_batch* b, int32_t n_views, const int32_t* view_map, const int32_t* colk,
                             const double* ab, int32_t n_cand, const int32_t* cand_nview);
/* Trilinear symmetry rows of candidate c (arguments as hb2_batch_explicit_sym_rows); call for c = 0, 1, ... in order. */
int hb2_batch_bilinear_sym_rows(hb2_batch* b, int32_t cand, int32_t n_pairs, const double* pair_mats,
                                int64_t min_sym_pairs, int64_t* n_rows);
int hb2_batch_bilinear_sym_export(hb2_batch* b, int32_t cand, int32_t* cols, float* weights);

/* ---- batch: step 2, candidates ----------------------------------------- */
/* Finalises the batch: adjoint maps, right-hand side, symmetry rows
 * (replaces SLR:1142-1218 + 1221-1287 incl. the first-seen-wins de-duplication
 * and the min_sym_pairs early stop) and their transpose lists. */
int hb2_batch_create(hb2_batch* b, int32_t n_cand, const hb2_candidate* cands, int32_t n_views, const hb2_view* views,
                     int32_t n_colk, const int32_t* colk, int32_t n_pairs, const hb2_pair* pairs);
void hb2_batch_destroy(hb2_batch* b);

/* Half-set solves (fsc_test, SLR:175-203 split_A_b + SLR:441-482): candidate c keeps only the data rows whose image
 * pixel id pid = k*D2 + j (b_data_pid, SLR:1548) is set in masks[cand_mask[c]][L2*D2]; cand_mask[c] = -1 keeps all
 * rows.  The host derives the sets from b_data_pid exactly as split_A_b does (incl. its np.random.shuffle for mode
 * 1); the kernels drop the rows (forward rows, right-hand side, max(b) of the positive bound, score).  Call after
 * hb2_batch_create, before hb2_batch_solve. */
int hb2_batch_set_pixel_masks(hb2_batch* b, int32_t n_masks, const uint8_t* masks, const int32_t* cand_mask);

/* number of symmetry rows of a candidate, and the rows themselves as (a,b)
 * voxel-index pairs in the reference's row order: A[r,a]=+1, A[r,b]=-1. */
int hb2_batch_sym_rows(hb2_batch* b, int32_t cand, int32_t* n_rows, int32_t* a_host, int32_t* b_host, int64_t capacity);
/* Stored position (inside the candidate's symmetry block of the row vectors) of the reference's r-th symmetry row:
 * the rows of one pair round are kept in the internal voxel order, SLR:1197-1202 enumerates them in mask order. */
int hb2_batch_sym_order(hb2_batch* b, int32_t cand, int32_t* order, int64_t capacity);
/* padded data-row count of a candidate (= view_count*D2*ZMP, ZMP = L3*MC rounded up to 4; row of (view v, ray j,
 * slice z, slot mc) = v*D2*ZMP + j*ZMP + z*MC + mc) and total padded rows incl. symmetry rows */
int64_t hb2_batch_rows_padded(hb2_batch* b, int32_t cand, int64_t* n_data_padded);
/* right-hand side in padded layout, out[n_data_padded] */
int hb2_batch_rhs(hb2_batch* b, int32_t cand, float* out_host);

/* ---- operators (tests, drop-in exports) --------------------------------- */
/* y = A x  (x in the reference's order z*ndisk + p; y in padded row layout: data rows [view][j][z*MC+mc], then
 * symmetry rows) */
int hb2_batch_apply_forward(hb2_batch* b, int32_t cand, const float* x_host, float* y_host);
/* x = A^T y */
int hb2_batch_apply_adjoint(hb2_batch* b, int32_t cand, const float* y_host, float* x_host);

/* ---- solve + score --------------------------------------------------------- */
/* For every candidate: LSMR on [A_data; A_hsym] x = [b; 0] with scipy's stopping
 * rules and precision map (replaces scipy lsq_linear as called at SLR:258-270),
 * the bounded TRF branch when cand.positive and the LSMR solution violates
 * [0, max(b)], then reprojection + cosine score (SLR:500-525).
 * results_host[n_cand].  Candidates stay resident for hb2_batch_get_x. */
int hb2_batch_solve(hb2_batch* b, const hb2_solve_options* opt, hb2_result* results_host);
/* solution vector x of one candidate as float32 in the reference's order (SLR:270, 538) */
int hb2_batch_get_x(hb2_batch* b, int32_t cand, float* x_host);
/* device time of the last hb2_batch_solve, out[16]:
 * [0] lsmr phase ms, [1] trf phase ms, [2] score phase ms, [3] kernels launched, [4] lsmr iterations run,
 * with opt.profile=1 also per kernel class, summed over launches (ms) and launch counts:
 * [5] fwd_data ms [6] fwd_sym ms [7] adjoint ms [8] update ms [9] scalar kernels ms,
 * [10] fwd_data launches [11] adjoint launches [12] update launches, [13..14] reserved,
 * [15] device ms of the last hb2_batch_score_metric (0 before one) */
int hb2_batch_timing(hb2_batch* b, double* out16);

/* debug/test: per outer iteration of the bounded branch of the last solve, out[row*8 + k] =
 * cost, g_norm, inner LSMR iterations, step kind (0 full Newton, 1 truncated Newton, 2 reflected, 3 anti-gradient),
 * p_value, r_value, ag_value, cost_change.  Returns nit*16 + (status+1). */
int hb2_batch_trf_trace(hb2_batch* b, int32_t cand, double* out, int32_t max_rows);

/* ---- ElasticNet / Lasso / Ridge (SLR:272-342) for every candidate of a nearest-neighbour batch ---------------
 * The reference's scikit-learn models on the stacked system [A_data; A_hsym] x = [b; 0] with the intercept profiled
 * out (X and y centred over the candidate's REAL rows), minimised as helicon_b200/regularized.py does on the host:
 * FISTA with adaptive restart and scikit-learn's duality gap for elastic net / lasso (and for ridge with the positive
 * constraint), CG on the normal equations for ridge, and the refit of an all-zero solution with alpha x 0.1
 * (SLR:331-335).  All candidates run at once on the device; the host only polls a counter every check_every iterations.
 * The positive constraint of each candidate is hb2_candidate.positive.  Afterwards the batch is solved as after
 * hb2_batch_solve: hb2_batch_get_x, hb2_batch_scatter_scores and the score (float32 w reprojected) are the model's,
 * hb2_result.itn = iterations of the final fit, flags |= HB2_FLAG_NOT_CONVERGED where max_iter ended it. */
#define HB2_MODEL_ENET 0   /* elastic net; lasso is l1_ratio = 1 */
#define HB2_MODEL_RIDGE 1
typedef struct {
  int32_t kind;               /* HB2_MODEL_ENET or HB2_MODEL_RIDGE */
  double alpha;               /* > 0 (scikit-learn's alpha) */
  double l1_ratio;            /* [0, 1], elastic net only */
  double gap_factor;          /* stop at gap <= gap_factor * 1e-2 * ||y_c||^2 (0.05: 20x tighter than the reference) */
  int32_t max_iter;           /* iterations per fit (4000) */
  int32_t check_every;        /* host polls the active-candidate counter every this many iterations */
  int32_t clip_pred;          /* as hb2_solve_options.clip_pred */
  const double* power_start;  /* [n] start vector of the power iteration for the Lipschitz constant, reference order,
                                 unit norm (regularized.py: default_rng(0).standard_normal(n) normalised) */
} hb2_model_options;
/* The candidate's real rows: real[m] over its padded row space (data rows then symmetry rows, m = the total of
 * hb2_batch_rows_padded), 1 where the row is an equation of the reference's system (Batch.data_row_index and every
 * symmetry row).  Required for every candidate before hb2_batch_solve_model. */
int hb2_batch_set_real_rows(hb2_batch* b, int32_t cand, const uint8_t* real, int64_t m);
int hb2_batch_solve_model(hb2_batch* b, const hb2_model_options* opt, hb2_result* results_host);
/* after hb2_batch_solve_model: out[4] = final alpha, iterations of the final fit, duality gap (elastic net; ridge: the
 * relative CG residual, or the last relative update with the positive constraint), Lipschitz estimate (0 for CG) */
int hb2_batch_model_info(hb2_batch* b, int32_t cand, double* out4);
/* test hook: the MODE_PLAIN products over ALL candidates in one launch each.  adjoint = 0: in = x of every candidate
 * ([nc][n], reference order), out = rows ([nc][total padded rows of hb2_batch_rows_padded] concatenated); adjoint = 1:
 * the other way round. */
int hb2_batch_apply_all(hb2_batch* b, int32_t adjoint, const float* in_host, float* out_host);

/* ---- 2-D score metrics (SLR:484-525, helicon_b200/imageprep.py) for every candidate of a solved batch -----------
 * The candidate's prediction A_data x (float32 x of hb2_batch_get_x, MODE_PLAIN forward, clipped at 0 when clip_pred)
 * is scattered into pred_2d[L2][D2] and scored against the transposed central (D2, L2) region of the problem's image
 * (the image hb2_problem_create received).  The metric's value replaces the candidate's score (the buffer that
 * hb2_batch_scatter_scores reads); composite is the mean of [cosine, ssim, ms_ssim, mutual information], its cosine
 * part the score the solve computed. */
#define HB2_METRIC_SSIM 1
#define HB2_METRIC_MS_SSIM 2
#define HB2_METRIC_MI 3
#define HB2_METRIC_COMPOSITE 4
/* The candidate's pixel table: last_row[k*D2 + j] = the padded data row (Batch.data_row_index) that writes pixel
 * (k, j) last in the reference's row order (copy, k, j), or -1 where no row does.  Every entry must be < the candidate's
 * padded data rows.  Required for every candidate before hb2_batch_score_metric. */
int hb2_batch_set_pixel_rows(hb2_batch* b, int32_t cand, const int32_t* last_row, int32_t L2, int32_t D2);
/* After hb2_batch_solve / hb2_batch_solve_model (HB2_ERR_STATE otherwise, or without the pixel tables).  scores_host
 * [nc] (nullable): the new scores; parts_host [nc][4] (nullable): cosine, ssim, ms_ssim, mutual information in
 * float64.  The device time of the call is hb2_batch_timing's out[15]. */
int hb2_batch_score_metric(hb2_batch* b, int32_t metric, int32_t clip_pred, float* scores_host, double* parts_host);

/* ---- test hook: the LSMR scalar recurrences run on the HOST --------------- */
/* Same code as the device path (compiled __host__ __device__).  state64 is an
 * opaque 64-double scratch the caller keeps between calls.
 * phase 0: initialise from alpha_1, beta_1 (lsmr.py:239-300);
 * phase 1: rotations + update coefficients from alpha_{k+1}, beta_{k+1} (lsmr.py:341-414);
 * phase 2: stopping tests given norm(x) (lsmr.py:416-457), returns istop. */
int hb2_lsmr_scalar_step(double* state64, int phase, float alpha, float beta, double normx, double atol, double btol,
                         double conlim, int maxiter, float* coef_hbar, float* coef_x, float* coef_h, double* trace8);

/* ---- post-solve display products (SURVEY.md section 8f rank 1) ------------------
 * helicon.apply_helical_symmetry (lib/transforms.py:58-165) as called by
 * pipeline.process_one_task (pipeline.py:405-427), plus the three sums the task
 * keeps of the symmetrised volume (pipeline.py:435-447): np.sum(vol, axis=2),
 * np.sum(vol, axis=1), np.sum(vol[zs0:zs1], axis=0) -- with numpy's summation
 * order, so results are bit-identical.  The host plans the z entries exactly as
 * the reference computes them (per OUTPUT slice k: the helical copies h whose
 * source slice k2 lies in the unit's z window, floor/ceil(k2), k2 - floor(k2))
 * and the 2x2 in-plane matrices of every (h, c); the kernels do the per-voxel
 * trilinear gather in the reference's float64 operation order. */
typedef struct {
  int32_t nz0, ny0, nx0;   /* asymmetric unit (rec3d) */
  int32_t nz, ny, nx;      /* working grid: max(unit, new_size) per axis (lib/transforms.py:74-80) */
  int32_t oz, oy, ox;      /* crop offset of the output in the working grid (lib/transforms.py:157-163) */
  int32_t nz1, ny1, nx1;   /* output size */
  double apix, new_apix;
  int32_t csym, n_ent;
  int32_t zs0, zs1;        /* z-section slab in output slices (pipeline.py:443-446) */
} hb2_symm_params;
/* k_begin[nz1+1]: CSR over output slices into ent_*; ent_h indexes mats in blocks of csym
 * (mats[(h*csym + c)*4 ..] = cos, sin, -sin, cos of deg2rad(twist*h + 360 c/csym)).
 * Any of the four outputs may be NULL. */
int hb2_helical_symmetrize(const float* data_host, const hb2_symm_params* p, const int64_t* k_begin,
                           const int32_t* ent_h, const int32_t* ent_floor, const int32_t* ent_ceil,
                           const double* ent_wk, const double* mats, int32_t n_mats, float* vol_out_host,
                           float* xsum_out, float* ysum_out, float* zsum_out, int device, void* stream);

/* ---- score map + top-K on the device (north-star item 3) -------------------
 * The grid driver the reference runs on the host (app.py:2482-2539: collect the task results, sort by score, keep the
 * top N, Z[twist, rise] = score) as device-resident state of ONE search: a float32 score map, an int32 iteration map
 * and a uint32 flag map over the flat task index (csym, twist, rise), NaN / 0 where a task was skipped or is solved by
 * another rank.
 * hb2_batch_scatter_scores writes the scores of a SOLVED batch into the map (one kernel on the batch's stream, no host
 * round trip per batch); hb2_scoremap_merge folds the maps of other ranks in (the buffer an NCCL all-gather filled:
 * n_maps maps of 3*n words back to back, device memory); hb2_scoremap_topk selects the K best (score descending, ties by
 * the lower task index = the reference's stable sort over its twist-major task list; NaN never selected). */
typedef struct hb2_scoremap hb2_scoremap;
int hb2_scoremap_create(hb2_scoremap** out, int64_t n, int device);
void hb2_scoremap_destroy(hb2_scoremap* m);
/* device pointer of the maps (float32[n] scores, int32[n] iterations, uint32[n] flags, contiguous: 3*n 4-byte words) */
void* hb2_scoremap_device_ptr(hb2_scoremap* m);
/* task_index_host[n_cand], flags_host[n_cand] (hb2_result.flags of the batch's solve) */
int hb2_batch_scatter_scores(hb2_batch* b, hb2_scoremap* m, const int64_t* task_index_host, const uint32_t* flags_host);
/* resume: entries of an earlier, interrupted search of the SAME grid (task index, score, iterations, flags; host
 * arrays of n_entries) written into the maps before the remaining candidates are solved -- replaces the reference's
 * on-disk function cache of finished candidates (lib/cache.py:132-209, used by app.py:2473-2539) */
int hb2_scoremap_restore(hb2_scoremap* m, int64_t n_entries, const int64_t* task_index_host, const float* scores_host,
                         const int32_t* itn_host, const uint32_t* flags_host);
int hb2_scoremap_merge(hb2_scoremap* m, const void* gathered_dev, int32_t n_maps, void* stream);
int hb2_scoremap_topk(hb2_scoremap* m, int32_t k, float* top_scores_host, int64_t* top_index_host, void* stream);
int hb2_scoremap_read(hb2_scoremap* m, float* scores_host, int32_t* itn_host, uint32_t* flags_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HELICON_B200_H */
