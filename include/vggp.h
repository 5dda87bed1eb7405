/*
 * vggp.h -- C ABI of libvggp.so: the sm_100a ELBO forward/backward hot path for variational Gaussian
 * processes with gridded (Kronecker-structured) inducing variables.
 *
 * This is the drop-in boundary.  The reference (maxnorman569/Variational-Gridded-Gaussian-Processes) is pure
 * Python and has no FFI; the entry points below are what a ctypes binding placed inside the reference's
 * model classes would call instead of the dense torch code (see INTEGRATION.md):
 *
 *   reference code replaced                                            entry point
 *   ------------------------------------------------------------------ ---------------------------------
 *   src/basis/bspline.py:92-94   SplineBasis.__call__ (B1 hats)         vggp_b1_stencil / vggp_b1_features_dense
 *   src/models/sparse/gridded_kronecker_structure.py:1325-1374          vggp_b0_features_dense
 *        _Kuf_along_dim (cell-integrated Matern-1/2 features)
 *   gridded_kronecker_structure.py:731-780, 1286-1323 _Kuu_along_dim    vggp_grid_forward (factor build)
 *   gridded_kronecker_structure.py:796-811, 1376-1390 _Kuu (torch.kron) vggp_grid_forward (never formed:
 *        + kronecker_structure.py:265-269 lazify(Kuu).inv_matmul         per-dimension Cholesky, inverse and
 *                                                                        Kronecker mode-n products instead)
 *   gridded_kronecker_structure.py:813-828, 1392-1407 _Kuf (Khatri-Rao) vggp_obs_fwd_bwd (never formed:
 *        + kronecker_structure.py:249-278 _elbo (N x N algebra)          per-observation fused kernel)
 *   elbow.backward()  (5_gridded_kronecker_structure_models.ipynb:445)  vggp_obs_fwd_bwd + vggp_grid_backward
 *   whole step with host buffers                                        vggp_elbo_host
 *
 * Conventions
 *   - every function returns int: 0 = ok, < 0 = invalid argument (VGGP_E_*), > 0 = a cudaError_t value;
 *     vggp_last_error() returns a static/thread-local message for the last non-zero status.
 *   - all work is asynchronous and ordered on the `stream` argument (a cudaStream_t passed as void*;
 *     NULL = the legacy default stream).  No entry point except vggp_plan_create/destroy, vggp_read_info,
 *     vggp_elbo_host, vggp_meanopt_solve, vggp_meanopt_solve_pc and vggp_logdet_system synchronises the host.
 *   - the caller owns every buffer passed in; the library allocates only inside vggp_plan_create (its
 *     grid-side workspace) and frees it in vggp_plan_destroy.
 *   - pointers are DEVICE pointers unless the parameter name ends in `_host`.
 *   - grid-side quantities (theta, m, L_d, their gradients, the ELBO) are always float64.  Observations,
 *     alpha as seen by the per-observation kernel and the per-observation gradient buffer use the plan's
 *     `obs_dtype` (VGGP_F32 or VGGP_F64).
 *   - index convention: flat inducing index u = ((i_1*M_2 + i_2)*M_3 + i_3), matching torch.kron(K_1, K_2)
 *     (gridded_kronecker_structure.py:1389) and the Khatri-Rao loop order (:1406).
 */
#ifndef VGGP_H
#define VGGP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VGGP_MAX_D 3

/* feature family */
#define VGGP_B1_ASVGP   0   /* B1-spline (hat) features, tridiagonal RKHS Kuu: GriddedMatern12ASVGP, Matern12B1SplineASVGP */
#define VGGP_B0_GRIDDED 1   /* cell-integrated Matern-1/2 features, Toeplitz Kuu: Matern12GriddedGP, Matern12B0SplineGriddedGP */
#define VGGP_SVGP_GRID  2   /* inducing POINTS on a product grid (kronecker_structure.py:287-338, Matern12SVGP): features
                             * phi_d(x)[i] = s2_d exp(-|x - z_i| / l_d), Kuu_d = s2_d exp(-|z_i - z_j| / l_d); the knots ARE the inducing
                             * locations z (M_d = n_knots[d]).  Dense-feature kernel (D <= 2, plain observation arrays); Z is fixed. */
#define VGGP_VFF_GRID   3   /* variational Fourier features (kronecker_structure.py:347-514 Matern12VFFGP, src/basis/fourier.py:58-88):
                             * per dimension M + 1 cosines and M sines of w_k = 2 pi k / (b - a) on the domain [a, b), exp(-r / l) outside,
                             * Kuu_d = diag(alpha) + beta beta^T.  The mesh of a dimension has 2 M + 1 knots spanning [a, b]: only its end
                             * points and its size are used (M_d = n_knots[d], odd).  Dense-feature kernel, D <= 2. */
#define VGGP_SVGP_MARKOV 4  /* the model of VGGP_SVGP_GRID (same knots-as-Z, theta layout and ELBO) in its O(1)-per-observation Markov
                             * form: K_d^-1 is tridiagonal and psi_d = K_d^-1 k_d(Z, x) has two non-zeros per dimension, so the
                             * per-observation kernel streams the binned layout (extended cells: observations outside the points
                             * contribute) and the grid side is O(M + sum M_d^2) elementwise work.  D = 1..3, Z fixed.  Takes the binned
                             * layout only: vggp_obs_fwd_bwd, vggp_obs_fwd_bwd_packed and vggp_elbo_host return VGGP_E_UNSUPPORTED, as do
                             * vggp_set_deterministic(plan, 1) and vggp_workspace_ptr; vggp_features_dense returns the dense k_d(Z, x). */

/* observation dtype */
#define VGGP_F32 0
#define VGGP_F64 1

/* status codes (< 0) */
#define VGGP_E_ARG        -1
#define VGGP_E_FAMILY     -2
#define VGGP_E_DTYPE      -3
#define VGGP_E_DIM        -4
#define VGGP_E_NOMEM      -5
#define VGGP_E_UNSUPPORTED -6

typedef struct vggp_plan vggp_plan;

/* ABI version of this header; vggp_abi_version() must return the same value. */
#define VGGP_ABI_VERSION 5
int vggp_abi_version(void);
const char* vggp_last_error(void);
/* Number of CUDA kernels this library has launched so far in this process (host-side counter). */
uint64_t vggp_launch_count(void);

/*
 * Plan = grid descriptor + workspace, one per (model, device).
 *   family      VGGP_B1_ASVGP | VGGP_B0_GRIDDED | VGGP_SVGP_GRID | VGGP_VFF_GRID | VGGP_SVGP_MARKOV
 *   D           number of input dimensions, 1..VGGP_MAX_D
 *   n_knots     [D] number of knots of each per-dimension mesh (B1: M_d = n_knots, B0: M_d = n_knots-1)
 *   knots_host  [D] host pointers to the float32 knot arrays, exactly as the reference builds them
 *               (torch.linspace without dtype, gridded_kronecker_structure.py:707-720, 1278-1279).  Knots are
 *               never regenerated on the device.
 *   obs_dtype   VGGP_F32 | VGGP_F64
 *   device      CUDA device ordinal
 */
int vggp_plan_create(vggp_plan** out, int family, int D, const int* n_knots,
                     const float* const* knots_host, int obs_dtype, int device);
int vggp_plan_destroy(vggp_plan* plan);

/* Device memory behind a plan (SURVEY.md section 8b): `plan_bytes` = everything vggp_plan_create allocated (factors, work
 * tensors, tables: the callee never allocates in a step), `gbuf_bytes` = the caller-owned gradient buffer a step needs
 * (= vggp_gbuf_layout total), `scratch_bytes` = what the opt-in paths have grown so far (plain-array staging of
 * vggp_obs_fwd_bwd / vggp_elbo_host, deterministic mode, B0 scan tables, the optimal-mean system).  Any output pointer may be null. */
int vggp_workspace_bytes(const vggp_plan* plan, int64_t* plan_bytes, int64_t* gbuf_bytes, int64_t* scratch_bytes);

/* M_d (inducing variables per dimension) and M = prod M_d. */
int vggp_plan_dims(const vggp_plan* plan, int* D, int* m_per_dim /*[D]*/, int64_t* M);

/*
 * Layout of the per-observation gradient buffer (`gbuf`) written by vggp_obs_fwd_bwd and all-reduced (sum)
 * across ranks before vggp_grid_backward:
 *     [ n_obs_elems values of obs_dtype | pad to 8 bytes | n_scalars float64 ]
 *   n_obs_elems = M (d alpha) + per-dimension band / factor-gradient blocks
 *   scalars     = { sum_n (r_n^2 - prod p + prod q), n_local, n_inside, reserved... }
 *   VGGP_SVGP_MARKOV: n_obs_elems = M (d m corner sums) + the band block [bp_d | bp_o | bq_d | bq_o] of every dimension (sums of
 *   prod_{e != d} p_e resp. q_e times wlo^2, wlo whi, whi^2 per node / node pair); scalars 3 + d hold
 *   sum_n d/dl_d [(y - mu)^2 + var] through the weights (bands held fixed).
 * `scalar_offset_bytes` is the byte offset of the float64 block, `total_bytes` the size to allocate.
 */
int vggp_gbuf_layout(const vggp_plan* plan, int64_t* n_obs_elems, int64_t* scalar_offset_bytes,
                     int64_t* n_scalars, int64_t* total_bytes);

/*
 * Grid-side forward: build K_d(theta), Cholesky, P_d = K_d^-1, R_d = P_d tril(L_d), Q_d = R_d R_d^T, S_d,
 * alpha = (kron_d P_d) m through mode-n products, the band tables the per-observation kernel reads, and the
 * KL ingredients (log-dets, traces, <m, alpha>).  Everything stays in the plan workspace.
 *   theta  [2D+1] float64: lengthscale_1..D, outputscale_1..D, noise   (constrained values)
 *   m      [M]    float64 variational mean (u-space, unwhitened; prior N(0, Kuu))
 *   L      [sum_d M_d^2] float64, the D row-major M_d x M_d factors back to back; lower triangle is used,
 *          S = kron_d L_d L_d^T
 */
int vggp_grid_forward(vggp_plan* plan, const double* theta, const double* m, const double* L, void* stream);

/*
 * Packed observation layout (setup, once per data set / minibatch partition; X is constant over optimisation
 * steps).  The fused kernel gives every lane one contiguous run of `run_len` observations and reads them
 * "warp-transposed" so that the loads stay coalesced; padding slots hold NaN.  With sort_by_cell != 0 the
 * observations are first ordered by flat grid-cell id (stable radix sort), so that a lane's run stays inside one
 * cell for as long as possible; this changes only the order of the summation, not the result.
 *   vggp_obs_pack_geometry  n -> padded length of every packed array and the run length (depends on the device)
 *   vggp_obs_pack           x[D], y (n values each) -> xp[D], yp (n_packed values each, caller-allocated).
 *                           May allocate temporary sort buffers (freed before returning, synchronises `stream`
 *                           in that case); with sort_by_cell == 0 it is allocation-free and asynchronous.
 */
int vggp_obs_pack_geometry(const vggp_plan* plan, int64_t n, int64_t* n_packed, int* run_len);
int vggp_obs_pack(vggp_plan* plan, const void* const* x, const void* y, int64_t n, int sort_by_cell,
                  void* const* xp, void* yp, void* stream);

/*
 * Per-observation fused forward+backward over one shard of the minibatch.
 *   x / xp [D] HOST array of device pointers to structure-of-arrays observations of obs_dtype
 *   y / yp     targets
 *   n          number of (real) observations in this shard (may be 0)
 *   gbuf       output, layout above; zeroed by this call, then accumulated.
 * Reads alpha / band tables produced by the last vggp_grid_forward on the same plan.
 * vggp_obs_fwd_bwd_packed consumes arrays produced by vggp_obs_pack (the hot-path form: nothing but the fused
 * kernel runs).  vggp_obs_fwd_bwd takes plain arrays in any order: it first transposes them into plan-owned
 * scratch (grown on demand -- the one allocation this call may make), then runs the same kernel.
 */
int vggp_obs_fwd_bwd_packed(vggp_plan* plan, const void* const* xp, const void* yp, int64_t n, void* gbuf, void* stream);
int vggp_obs_fwd_bwd(vggp_plan* plan, const void* const* x, const void* y, int64_t n, void* gbuf, void* stream);

/*
 * Binned observation layout (second form of the one-time setup, same gbuf as the other forms).
 * The observations are ordered by grid cell and cut into RUNS -- all observations of one cell, or an equal share of
 * them when the cell holds more than `run_cap` -- and 32 runs of (almost) equal length form one warp task, so that
 * the fused kernel enters and leaves cells with all lanes active and needs no per-observation cell test.  Padding
 * slots contribute nothing; observations outside the mesh are not streamed (their sum of y^2 is stored once).
 *   vggp_obs_bin_prepare   x[D] (n values each) -> desc: the layout of this data set and the size of the buffer the
 *                          caller must allocate (256-byte aligned).  Sorts by cell, reads the per-cell counts back
 *                          and plans the runs on the host: synchronises `stream`, allocates temporaries that live
 *                          until the matching vggp_obs_bin_pack (one pending layout per plan).
 *   vggp_obs_bin_pack      fills `binned` (desc->bytes) from x[D], y; synchronises, frees the temporaries.
 *   vggp_obs_fwd_bwd_binned  the fused forward+backward over a binned buffer (asynchronous, allocation-free);
 *                          gbuf is zeroed by the call, exactly as vggp_obs_fwd_bwd_packed.
 * VGGP_SVGP_MARKOV (D = 1..3): the same three calls with extended cells as for the B0 family below; the per-observation kernel is
 * k_obs_svgpm_binned (csrc/svgpm.cuh).  This is the only observation path of that family.
 * B0 family (D <= 2): the same three calls select the SCAN form of the cell-integrated features (csrc/b0scan.cuh,
 * DESIGN.md section 4): cells are extended by one virtual cell on each side (observations outside the mesh do
 * contribute in this family, n_inside == n), the per-observation kernel does O(1) work against per-cell tables built by
 * first-order recurrences on the grid side, and an adjoint stage writes the same gbuf blocks vggp_obs_fwd_bwd writes for this
 * family.  The tables live in the plan (allocated by vggp_plan_create).
 * Status: the default observation layout of both families since round 2 (GPU-verified against the oracle and against the
 * packed layout; DESIGN.md section 4).  run_cap: longest run of one cell; 0 = automatic (about two warp tasks per resident
 * warp: 256 from ~2^25.8 observations per shard up, smaller for thin or cell-range shards, never below 32).
 */
typedef struct vggp_binned_desc {
    int64_t bytes;          /* size of the device buffer `binned` */
    int64_t n;              /* observations given */
    int64_t n_inside;       /* of which inside the mesh (streamed) */
    int64_t n_tasks;        /* warp tasks of 32 runs */
    int64_t n_runs;         /* non-empty runs */
    int64_t data_elems;     /* streamed values of obs dtype, padding included: sum over tasks of 32 R_t (D + 1) */
    int64_t off_task_off, off_task_R, off_run_cell, off_run_n, off_run_start, off_data;   /* byte offsets */
    int32_t run_cap, D;
} vggp_binned_desc;
int vggp_obs_bin_prepare(vggp_plan* plan, const void* const* x, int64_t n, int run_cap, vggp_binned_desc* desc,
                         void* stream);
int vggp_obs_bin_pack(vggp_plan* plan, const vggp_binned_desc* desc, const void* const* x, const void* y,
                      void* binned, void* stream);
int vggp_obs_fwd_bwd_binned(vggp_plan* plan, const vggp_binned_desc* desc, const void* binned, void* gbuf,
                            void* stream);
/*
 * Epoch-shuffled minibatches in the binned layout (csrc/minibatch.cuh; B1, VGGP_SVGP_MARKOV and B0 with D <= 2).
 * Sampling law: epoch `epoch` of rank `rank` draws a pseudo-random permutation pi of the rank's n observations, a keyed
 * bijection computed inline (a balanced 4-round Feistel network on the smallest even number of bits k with 2^k >= n, round
 * function a 32-bit mixing hash of seed, epoch, rank, round and half, cycle-walking below n).  Batch b < P is
 * { i : pi(i) in [b B, (b + 1) B) }, the other n - P B observations are dropped, so every observation is in a given batch
 * with probability B / n: the expected log-likelihood of a batch scaled by n / B (ell_scale) is unbiased.
 * One device pass bins all P batches into one buffer: P 256-byte headers, then each batch's sections.  Batch b is the view
 * (binned + byte_offset, vggp_binned_desc) of vggp_epoch_batch, which every entry point taking a binned buffer accepts
 * (vggp_obs_fwd_bwd_binned in both modes, vggp_meanopt_assemble); its n is B.  Its bytes equal vggp_obs_bin_pack of that
 * batch's observations in ascending index order with the same run_cap.
 *   vggp_epoch_bin_prepare  x[D] (n values each), B = batch_size, n_batches = P (0 = n / B; a sharded run passes the
 *                           smallest shard's count so that every rank steps equally often), run_cap (0 = the automatic rule
 *                           of vggp_obs_bin_prepare applied to B) -> desc, and totals_host [VGGP_EPOCH_TOTALS * P]: per batch
 *                           { tasks, runs, observations inside the mesh, data elements, byte offset of its first section }.
 *                           Sorts by (batch, cell), plans the runs of every batch on the device and reads back only the
 *                           per-batch totals: synchronises `stream`, allocates temporaries that live until the matching
 *                           vggp_epoch_bin_pack (one pending epoch per plan).  VGGP_E_UNSUPPORTED for VGGP_SVGP_GRID,
 *                           VGGP_VFF_GRID and B0 with D = 3; VGGP_E_ARG for B < 1, B > n, n >= 2^31.
 *   vggp_epoch_bin_pack     fills `binned` (desc->bytes, 256-byte aligned) from x[D], y; synchronises, frees the temporaries.
 *   vggp_epoch_batch        host only: the descriptor of batch b and the byte offset of its view in `binned`.
 */
#define VGGP_EPOCH_TOTALS 5
typedef struct vggp_epoch_desc {
    int64_t bytes;          /* size of the epoch buffer */
    int64_t n;              /* observations given */
    int64_t batch_size;     /* B */
    int64_t n_batches;      /* P */
    int64_t n_tasks, n_runs, data_elems;   /* sums over the batches */
    uint64_t seed, epoch;
    int32_t rank, run_cap, D, elem_size;
} vggp_epoch_desc;
int vggp_epoch_bin_prepare(vggp_plan* plan, const void* const* x, int64_t n, int64_t batch_size, int64_t n_batches,
                           int run_cap, uint64_t seed, uint64_t epoch, int rank, vggp_epoch_desc* desc,
                           int64_t* totals_host, void* stream);
int vggp_epoch_bin_pack(vggp_plan* plan, const vggp_epoch_desc* desc, const int64_t* totals_host, const void* const* x,
                        const void* y, void* binned, void* stream);
int vggp_epoch_batch(const vggp_epoch_desc* desc, const int64_t* totals_host, int64_t b, vggp_binned_desc* batch,
                     int64_t* byte_offset);
/* How vggp_obs_fwd_bwd_binned streams the observations: 0 (default) coalesced 16-byte global loads into two register
 * buffers; 1 = a per-warp shared-memory ring filled by TMA bulk copies (cp.async.bulk + mbarrier), two stages ahead. */
int vggp_set_binned_stream(int mode);

/*
 * Deterministic mode (SURVEY.md section 8b): on = 1 makes a step of this plan -- vggp_grid_forward,
 * vggp_obs_fwd_bwd_binned, vggp_grid_backward -- bitwise reproducible from run to run, whatever the grid size, the work
 * stealing order or the load of the machine.  No floating-point atomic is left on the path: every run of the binned
 * layout writes its flush values as a record and the records are summed in the order of the cell-sorted stream
 * (csrc/obs_binned.cuh); the fibre passes leave per-CTA partials that are summed in tile order (csrc/grid_b1_fast.cuh).
 * Covered: the B1 (ASVGP) family with M_d <= 512 and the binned observation layout
 * (VGGP_E_UNSUPPORTED otherwise, also from vggp_obs_fwd_bwd / _packed while the mode is on).  The scratch is sized at the
 * first deterministic step (cudaMalloc): run one step eagerly before capturing a graph.  Costs a sort of the run list
 * and five small reductions per step; the default (0) is the atomics path.
 */
int vggp_set_deterministic(vggp_plan* plan, int on);

/*
 * The one collective of a sharded step as a single kernel over peer memory (csrc/collective.cuh): gbuf <- sum over the ranks
 * of one NVSwitch node, in place, on `stream`, between vggp_obs_fwd_bwd* and vggp_grid_backward.  It replaces the
 * ncclAllReduce the north star names (SURVEY.md section 8e) where the gradient buffers are SYMMETRIC allocations: same
 * size on every rank and mapped into every process (the host mirror uses torch.distributed._symmetric_memory for the
 * allocation and the handle exchange).  With a multicast address the reduction happens in the switch (multimem.ld_reduce /
 * multimem.st on slice `rank` of the buffer); without one, rank r reads slice r from every peer and writes the sum back to
 * every peer.  world <= 8.
 *   desc->pad_ptrs  every rank's signal pad (VGGP_AR_PAD_WORDS uint32 words, zeroed once at setup), mapped like the
 *                   buffers.  The barrier sequence numbers live in the pad and are advanced by the kernel itself, so the
 *                   call has no per-call argument and can be captured into a CUDA graph and replayed; all ranks must make
 *                   the same sequence of calls
 *   err_flag        DEVICE int, set to 1 if a barrier timed out (a rank is missing): the poll loops are bounded
 */
typedef struct vggp_ar_desc {
    void* mc_ptr;
    void* buf_ptrs[8];
    void* pad_ptrs[8];
    int32_t rank, world;
} vggp_ar_desc;
#define VGGP_AR_PAD_WORDS 576
int vggp_allreduce_gbuf(vggp_plan* plan, const vggp_ar_desc* desc, int* err_flag, void* stream);

/*
 * Grid-side backward + ELBO assembly from the (all-reduced) gbuf.
 *   ell_scale   N / B minibatch scaling of the expected log-likelihood (1 for full batch)
 *   out    [4]    float64: ELBO, ell_scale * ELL, KL, n_obs(all ranks)
 *   dtheta [2D+1] float64 d ELBO / d theta (constrained values)
 *   dm     [M]    float64
 *   dL     [sum_d M_d^2] float64 (strictly-upper triangles are zero)
 */
int vggp_grid_backward(vggp_plan* plan, const double* theta, const double* m, const double* L,
                       const void* gbuf, double ell_scale,
                       double* out, double* dtheta, double* dm, double* dL, void* stream);

/*
 * Device timing of the dominant kernel (the fused per-observation kernel), for roofline reporting: while enabled, every
 * vggp_obs_fwd_bwd* call records one CUDA event immediately before and one immediately after the launch of that kernel
 * on `stream` (not around the memsets / the band-replica reduction that belong to the same call).
 *   vggp_k1_timing     enable != 0: (re)start collecting; 0: stop.
 *   vggp_k1_time_read  mean duration in milliseconds over the launches recorded since the last (re)start (the most recent
 *                      256 at most) and their number; synchronises the recorded events.
 */
int vggp_k1_timing(vggp_plan* plan, int enable);
int vggp_k1_time_read(vggp_plan* plan, float* mean_ms, int* n_launches);
/* The same kernel inside a captured CUDA graph: when vggp_k1_timing is on while the caller's stream is being captured, the two
 * records become external event-record nodes of the graph (cudaEventRecordExternal), re-recorded by every replay.
 *   vggp_k1_graph_time_read  duration in milliseconds of the kernel in the most recent replay; synchronises its end event. */
int vggp_k1_graph_time_read(vggp_plan* plan, float* ms);

/* Failed-factorisation flag of the last forward (0 = ok, d+1 = factor d not positive definite).
 * Synchronises `stream`. */
int vggp_read_info(vggp_plan* plan, int* info_host, void* stream);
/* The same flag copied to `info_pinned_host` (page-locked host memory) in stream order WITHOUT synchronising: the host
 * mirror records an event after it and raises torch.linalg.LinAlgError from the next call that finds the event complete
 * (the reference raises at the failing Cholesky: 61_envisat_gulfstream_experiment.ipynb:746). */
int vggp_info_async(vggp_plan* plan, int* info_pinned_host, void* stream);

/*
 * Whole step through HOST buffers (the call a ctypes binding inside the reference's `_elbo` would make):
 * copies x/y/theta/m/L host->device into plan-owned staging buffers (grown on demand, the only call that
 * may allocate after plan creation), runs forward + per-observation + backward on `stream`, copies
 * out/dtheta/dm/dL back and synchronises.
 */
int vggp_elbo_host(vggp_plan* plan, const void* const* x_host, const void* y_host, int64_t n,
                   const double* theta_host, const double* m_host, const double* L_host, double ell_scale,
                   double* out_host, double* dtheta_host, double* dm_host, double* dL_host, void* stream);

/*
 * Optimal variational mean (B1 family and VGGP_SVGP_MARKOV; VGGP_E_UNSUPPORTED otherwise): the m that maximises the ELBO for
 * fixed theta, which is the mean of the reference's closed-form q_u(): m* = Kuu Sigma^-1 Kuf y / noise,
 * Sigma = Kuu + Kuf Kuf^T / noise.  The m-dependent part of the ELBO, -(1/2 noise) ||y - mu(m)||^2 - (1/2) m^T Kuu^-1 m, does
 * not depend on S, and every observation has 2^D non-zero weights w (the corners of its cell), so m* solves a symmetric
 * positive definite 3^D-point stencil system on the node grid (csrc/meanopt.cuh):
 *     B1:                (Kuu + G / noise) alpha = b / noise,   m* = Kuu alpha*      mu = Phi^T alpha,  Kuu = kron_d K_d
 *     VGGP_SVGP_MARKOV:  (Kuu^-1 + G / noise) m* = b / noise                         mu = Psi^T m,  Psi = Kuu^-1 Kuf
 * with G = sum_n w_n w_n^T and b = sum_n w_n y_n (B1: hat weights, observations outside the mesh contribute nothing; Markov:
 * the two weights per dimension of the extended cells, virtual corners dropped).
 *   vggp_meanopt_assemble  zeroes and fills G and b (plan-owned float64) in one pass over a binned buffer of this plan
 *                          (vggp_obs_bin_pack).  Asynchronous; the first call allocates the system and the solver's
 *                          vectors (about (3^D + 13) / 2 M float64, counted in scratch_bytes of vggp_workspace_bytes) and
 *                          must not be captured.  VGGP_SVGP_MARKOV uses the theta of the last vggp_grid_forward; the B1
 *                          system does not depend on theta.
 *   vggp_meanopt_solve     Jacobi-preconditioned conjugate gradients in float64 at the theta of the last vggp_grid_forward,
 *                          from the state of that forward (B1: its alpha; Markov: its m, in the observation dtype): a forward
 *                          at m = 0 is a cold start, a forward at a previous m* a warm start.  Stops once
 *                          ||r|| <= rtol ||b / noise|| or after max_iter iterations; writes m_out [M] (DEVICE, float64),
 *                          the iterations and the final relative residual.  Returns 0 also when it did not converge
 *                          (*iters_host == max_iter and *relres_host > rtol).  No data (b = 0): m* = 0, 0 iterations,
 *                          relres 0.  VGGP_E_ARG without a previous vggp_meanopt_assemble.  Synchronises `stream`.
 *   vggp_meanopt_solve_pc  the same solve with a choice of preconditioner `precond`; VGGP_E_ARG for any other value:
 *                          VGGP_MEANOPT_JACOBI      = vggp_meanopt_solve, bit for bit.
 *                          VGGP_MEANOPT_KRONECKER   kron_d (F_d + g I)^-1, applied exactly: F_d is the tridiagonal prior
 *                                                   factor of dimension d (B1: K_d; Markov: K_d^-1) and
 *                                                   g = (trace(G) / (noise M))^(1/D).  One application is D batched
 *                                                   tridiagonal solves along the modes of the node grid.  It converges on
 *                                                   3-D B1 grids where Jacobi does not (DESIGN.md section 4, K1m).  The
 *                                                   first call allocates its vector and factors (M + 3 sum M_d float64,
 *                                                   counted in scratch_bytes).
 *                          Synchronises `stream`.
 */
#define VGGP_MEANOPT_JACOBI    0
#define VGGP_MEANOPT_KRONECKER 1
int vggp_meanopt_assemble(vggp_plan* plan, const vggp_binned_desc* desc, const void* binned, void* stream);
int vggp_meanopt_solve(vggp_plan* plan, double rtol, int max_iter, double* m_out,
                       int* iters_host, double* relres_host, void* stream);
int vggp_meanopt_solve_pc(vggp_plan* plan, int precond, double rtol, int max_iter, double* m_out,
                          int* iters_host, double* relres_host, void* stream);

/* ---- optimal variational covariance within the Kronecker family (B1 and VGGP_SVGP_MARKOV) ------------------
 * One coordinate update of S_d = tril(L_d) tril(L_d)^T: with theta, m and every S_e, e != d, fixed, the ELBO is strictly
 * concave in S_d and maximised by S_d = (M / M_d) A_d^-1 (csrc/covopt.cuh, DESIGN.md section 4, K1s):
 *     T_d = (ell_scale / noise) H_d + c_d F_d,   H_d = sum_n (prod_{e != d} q_e(x_n)) w_d w_d^T,   c_d = prod_{e != d} tr(K_e^-1 S_e)
 *     VGGP_SVGP_MARKOV:  F_d = K_d^-1,  S_d = (M / M_d) T_d^-1;     B1:  F_d = K_d,  S_d = (M / M_d) K_d T_d^-1 K_d
 * Cycling d = 0..D-1 is coordinate ascent on the ELBO; with set_optimal_mean's m* it gives the ELBO-optimal q(u) of the
 * Kronecker family.  For D = 1 one update is the reference's S* = Kuu Sigma^-1 Kuu.
 *   vggp_covopt_update  reads `L` (DEVICE, float64, the concatenated [M_1^2 | M_2^2 | ...] blocks given to the last
 *                       vggp_grid_forward) and writes block `dim` of `L_out` (same layout; the other blocks are untouched;
 *                       `L_out` may alias `L`) with the lower-triangular Cholesky factor of the new S_d (positive diagonal,
 *                       strict upper triangle 0).  `gbuf` must be the gradient buffer of a step taken at exactly that
 *                       forward (vggp_obs_fwd_bwd_binned or another per-observation call after it), already all-reduced
 *                       when the observations are sharded; only its band block of dimension `dim` is read.  Adds
 *                       ||L_new / ||L_new||_F - L_old / ||L_old||_F||_F (lower triangles) to the DEVICE float64 scalar
 *                       `change`; the measure does not see the flat direction S_1 -> a S_1, S_2 -> S_2 / a of the family.
 *                       A pivot of T_d that is not positive and finite sets the flag of vggp_read_info to dim + 1, leaves
 *                       `L_out` untouched and adds +inf to `change`.  Asynchronous, no host synchronisation; the first call
 *                       allocates 6 max M_d + 8 float64 (counted in scratch_bytes) and must not be captured, later calls
 *                       may be.  VGGP_E_UNSUPPORTED for the B0, SVGP_GRID and VFF families and for M_d > 2560; VGGP_E_ARG
 *                       for a bad `dim`, a null pointer, or no previous vggp_grid_forward on the plan.
 */
int vggp_covopt_update(vggp_plan* plan, int dim, const void* gbuf, double ell_scale, const double* L, double* L_out,
                       double* change, void* stream);

/* ---- collapsed ELBO at any grid size (B1 and VGGP_SVGP_MARKOV; csrc/collapsed.cuh, DESIGN.md section 4, K1l) -------------
 * The reference's objective (its collapsed _elbo()) from the stencil system A = F + G / noise of the optimal mean (F = Kuu for
 * B1, F = Kuu^-1 for Markov) and the solver's iterate x* (B1: alpha*, Markov: m*), by the matrix determinant lemma:
 *     ELBO = -1/2 [N log 2 pi + N log noise + log det A - log det F + (y^T y - b^T x*) / noise] - (N prod_d s2_d - tr(F^-1 G)) / (2 noise)
 * with log det F = log det Kuu (B1) or -log det Kuu (Markov), tr(F^-1 G) = tr(Kuu^-1 G) (B1) or tr(Kuu G) (Markov).
 *   vggp_logdet_system    log det A by preconditioned stochastic Lanczos quadrature: log det A = log det P + tr log(C^-1 A C^-T)
 *                         with the preconditioner P = C C^T of vggp_meanopt_solve_pc (`precond`: VGGP_MEANOPT_JACOBI,
 *                         C = diag(A)^1/2; VGGP_MEANOPT_KRONECKER, C = kron_d L_d D_d^1/2 of the Thomas factors of F_d + g I).
 *                         log det P is exact; the trace is estimated from `n_probes` probes eps_j, each by Gauss quadrature on
 *                         its Lanczos tridiagonal.  probe_kind VGGP_PROBE_RADEMACHER: signs from a counter hash of
 *                         (seed_or_first, probe, node), estimate = log det P + mean_j eps_j^T log(B) eps_j, standard error =
 *                         sample deviation / sqrt(n_probes); VGGP_PROBE_UNIT: e_first .. e_{first + n_probes - 1}
 *                         (first = seed_or_first), estimate = log det P + sum_j, exact when the probes cover all M nodes,
 *                         standard error 0.  A probe has converged once its quadrature value moves by <= rtol (relative)
 *                         between two checks (8 steps apart, from 128 steps on steps / 8
 *                         apart), or when its Krylov space is exhausted; max_steps bounds the
 *                         iteration.  out_host[VGGP_LOGDET_FIELDS] = { estimate, standard error, log det P, Lanczos steps (max
 *                         over probes), probes converged, probes }; per_probe_host [n_probes] (or NULL) the per-probe values.
 *                         For one assembly and seed the output is bitwise reproducible (fixed-order reductions).  The first
 *                         call allocates (4 k + 1) M float64 and small arrays (k = n_probes; grown when k or max_steps grows;
 *                         counted in scratch_bytes, refused under stream capture).  Synchronises `stream`.
 *   vggp_collapsed_terms  out [VGGP_CT_FIELDS] (DEVICE float64) = { N (all observations of the binned set), sum y^2 (including
 *                         the observations outside the mesh), b^T x*, tr(F^-1 G), log det Kuu }: exact, fixed-order
 *                         reductions over the binned data section and the grid.  Needs a vggp_meanopt_solve /
 *                         vggp_meanopt_solve_pc on the current assembly after the last vggp_grid_forward (a forward
 *                         invalidates the solve), whose iterate it reads; `desc` / `binned` must be the set given to
 *                         vggp_meanopt_assemble (its n, n_tasks and data_elems are compared).  Asynchronous.
 * Both: VGGP_E_UNSUPPORTED for the B0, SVGP_GRID and VFF families; VGGP_E_ARG without a previous vggp_meanopt_assemble (and,
 * for the terms, without a solve on it or with another binned set), for n_probes outside 1 .. VGGP_MAX_PROBES, max_steps < 1, unit probes past M and an unknown precond.
 */
#define VGGP_PROBE_RADEMACHER 0
#define VGGP_PROBE_UNIT       1
#define VGGP_LOGDET_FIELDS    6
#define VGGP_MAX_PROBES       65535   /* the probe index is a grid dimension of the Lanczos kernels */
int vggp_logdet_system(vggp_plan* plan, int precond, int probe_kind, int n_probes, uint64_t seed_or_first,
                       int max_steps, double rtol, double* out_host, double* per_probe_host, void* stream);
#define VGGP_CT_FIELDS 5
int vggp_collapsed_terms(vggp_plan* plan, const vggp_binned_desc* desc, const void* binned, double* out, void* stream);

/* ---- feature evaluation (bit-exact restatement of the reference's basis calls) ------------------------- */

/* B1 stencil of dimension `dim`: for each x[n], c[n] (int32; -1 = outside the mesh), w_lo[n], w_hi[n] such
 * that column n of B1SplineBasis(mesh)(x) (bspline.py:92-94) has w_lo at row c, w_hi at row c+1. */
int vggp_b1_stencil(const vggp_plan* plan, int dim, const void* x, int64_t n,
                    int32_t* c, void* w_lo, void* w_hi, void* stream);

/* Dense (M_d, n) row-major feature matrix of dimension `dim`, numerically equal to the reference's
 * `_Kuf_along_dim` for the plan's family (B0 family needs theta for lengthscale/outputscale). */
int vggp_features_dense(const vggp_plan* plan, int dim, const void* x, int64_t n, const double* theta,
                        void* phi, void* stream);

/*
 * Point prediction at test points from the state of the last vggp_grid_forward: the marginal mean and variance of
 * q(f(x*)) -- kronecker_structure.py:199-230 `posterior` restricted to its diagonal --
 *   mean = <kron_d phi_d(x*), alpha>,   var = prod_d s2_d - prod_d phi_d^T P_d phi_d + prod_d phi_d^T Q_d phi_d.
 *   x [D] HOST array of device pointers (n values of obs_dtype each); mean, var: n values of obs_dtype.
 * B1 family: test points outside the mesh get mean 0 and the prior variance (their feature column is zero).
 * VGGP_SVGP_MARKOV: two weights per dimension against the per-cell tables of the last forward, O(1) per point.
 * B0 family (D <= 2): the cell-integrated features are non-zero everywhere; they are evaluated in their scan form
 *   (three local features per dimension against per-cell tables built by first-order recurrences on the grid side,
 *   csrc/b0scan.cuh),
 *   O(1) work per point.  The tables are part of the plan (DESIGN.md section 4; GPU-verified in round 2).
 */
int vggp_predict(vggp_plan* plan, const void* const* x, int64_t n, void* mean, void* var, void* stream);

/*
 * Evaluation metrics of the reference (src/utils/evaluationmetrics.py:6-54) as one fused reduction.  `out` (DEVICE,
 * 4 float64, zeroed by the call) receives the raw sums
 *     { sum (t - p)^2,  sum |t - p|,  sum (t - t_0),  sum (t - t_0)^2 }       t_0 = truth[0]
 * from which MSE = out0/n, MAE = out1/n, RMSE = sqrt(MSE), R^2 = 1 - out0 / (out3 - out2^2/n).
 *   vggp_metrics          truth, pred: n values of `dtype` (VGGP_F32 | VGGP_F64) each
 *   vggp_predict_metrics  the same sums for pred = posterior mean at the test points x[D] (state of the last
 *                         vggp_grid_forward, B1 and VGGP_SVGP_MARKOV families), without writing the predictions to memory
 */
int vggp_metrics(int dtype, const void* truth, const void* pred, int64_t n, double* out, void* stream);
int vggp_predict_metrics(vggp_plan* plan, const void* const* x, const void* y, int64_t n, double* out, void* stream);

/*
 * Min-max scaling of the reference's data preparation (src/utils/dataprocessors.py:3-44), in the tensor's own dtype
 * with separately rounded operations (bit for bit what torch computes).
 *   vggp_minmax        minmax (DEVICE, 2 values of `dtype`) <- { min(x), max(x) }, n > 0; synchronises `stream`
 *   vggp_minmax_scale  inverse == 0: y = (x - min) / (max - min);  inverse != 0: y = x * (max - min) + min.
 *                      minmax is read on the device; y may alias x.
 */
int vggp_minmax(int dtype, const void* x, int64_t n, void* minmax, void* stream);
int vggp_minmax_scale(int dtype, const void* x, int64_t n, const void* minmax, int inverse, void* y, void* stream);

/*
 * Synthetic satellite-track observations generated on the device (SURVEY.md section 8d, 8f row 4): the geometry of the
 * reference's generate_track (src/utils/dataloaders.py:290-377, notebook call trajectory_gradient = 2): `passes` ascending
 * passes x1 = j / passes + t / gradient (wrapped into [0, 1)), x2 = t, then as many descending ones (x2 = 1 - t), in
 * acquisition order; targets = a smooth field + noise of standard deviation 0.05; D = 3 adds the acquisition time as x3 and a
 * slow drift of the field.  Observation i of the data set is a pure function of (i, seed): a rank generates its shard
 * [lo, hi) of the same n_total observations whatever the sharding.
 *   x [D] HOST array of device pointers, hi - lo values of `dtype` each; y likewise.  Asynchronous on `stream`.
 */
int vggp_generate_tracks(int dtype, int D, int64_t n_total, int64_t lo, int64_t hi, int64_t seed, int passes, double gradient,
                         void* const* x, void* y, void* stream);

/* ---- workspace views and primitives (tests, predictions, debugging) ------------------------------------ */

/* Device pointer to a float64 workspace array of the last forward (VGGP_E_UNSUPPORTED for the Markov SVGP family).  which: */
#define VGGP_WS_K      0   /* Cholesky factor C_d of K_d (lower; upper triangle undefined); B0 / SVGP / VFF families only */
#define VGGP_WS_P      1   /* P_d = K_d^-1 */
#define VGGP_WS_R      2   /* R_d = P_d tril(L_d) */
#define VGGP_WS_Q      3   /* Q_d = R_d R_d^T; B0 / SVGP / VFF families only (the B1 family keeps just its band, VGGP_WS_QBAND) */
#define VGGP_WS_S      4   /* (retired: S_d is not materialised) */
#define VGGP_WS_ALPHA  5   /* alpha (M), dim ignored */
#define VGGP_WS_SCAL   6   /* scalars: logdet K_d [3], logdet S_d [3], tr(P_d S_d) [3], <m,alpha> */
#define VGGP_WS_KRAW   7   /* K_d as built (before factorisation) */
#define VGGP_WS_QBAND  8   /* main / first off diagonal of Q_d: [diag (M_d) | off (M_d)] */
int vggp_workspace_ptr(const vggp_plan* plan, int which, int dim, double** ptr, int64_t* n_elems);

/* Batched strided float64 GEMM on the tensor cores (DMMA m8n8k4) or the SIMT fallback used to cross-check it:
 *   C[b] = alpha * A[b] * B[b] + beta * C[b],  A: m x k, B: k x n, element (i,j) of X at X + b*bsX + i*rsX + j*csX */
int vggp_gemm_f64(int use_mma, int batch, int m, int n, int k, double alpha,
                  const double* A, int64_t rsA, int64_t csA, int64_t bsA,
                  const double* B, int64_t rsB, int64_t csB, int64_t bsB,
                  double beta, double* C, int64_t rsC, int64_t csC, int64_t bsC, int splitk, void* stream);

/* Apply a dense (M_d x M_d, row-major) matrix along mode `dim` of the M-tensor `src` -> `dst` (float64). */
int vggp_mode_product(vggp_plan* plan, int dim, const double* A, const double* src, double* dst, void* stream);

/* Select the GEMM inner loop used by the grid-side path: 1 = DMMA tensor cores (default), 0 = SIMT. */
int vggp_set_gemm_mode(int use_mma);

#ifdef __cplusplus
}
#endif
#endif /* VGGP_H */
