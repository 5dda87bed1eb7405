// libvggp.so -- plan, static launch schedules and the extern "C" entry points declared in include/vggp.h.
// sm_100a only; there is no CPU path in this library.
#include <vector>
#include <algorithm>
#include <new>
#include <mutex>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"
#include "gemm.cuh"
#include "grid.cuh"
#include "grid_b1.cuh"
#include "grid_b1_fast.cuh"
#include "obs.cuh"
#include "obs_binned.cuh"
#include "metrics.cuh"
#include "b0scan.cuh"
#include "svgpm.cuh"
#include "meanopt.cuh"
#include "covopt.cuh"
#include "collapsed.cuh"
#include "collective.cuh"
#include "minibatch.cuh"

// Every plan-taking entry point runs with the plan's device current and restores the caller's device on return
// (launches on a stream of another device fail with "invalid resource handle"; plan creation must not silently switch
// the process's current device).
struct DeviceGuard {
    int prev = -1, want = -1;
    explicit DeviceGuard(int dev) : want(dev) {
        if (dev < 0 || cudaGetDevice(&prev) != cudaSuccess) { prev = -1; return; }
        if (prev != dev) cudaSetDevice(dev); else prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-function attribute that lives as long as the process (per device):
// a second, smaller plan must never lower what an earlier, larger plan opted in.  Every opt-in goes through this
// high-water mark keyed by (function, device).
struct SmemHwm { const void* fn; int dev; int bytes; };
static std::vector<SmemHwm> g_smem_hwm;
static std::mutex g_smem_mu;
template <typename F>
int raise_dyn_smem(F fn, size_t bytes) {
    int dev = 0;
    VGGP_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_smem_mu);
    for (auto& e : g_smem_hwm)
        if (e.fn == (const void*)fn && e.dev == dev) {
            if ((int)bytes <= e.bytes) return 0;
            VGGP_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
            e.bytes = (int)bytes;
            return 0;
        }
    // first use: opt in whatever the size -- static shared memory counts against the 48 KB default too, so a kernel asking for
    // exactly 48 KB of dynamic memory already needs it
    VGGP_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    g_smem_hwm.push_back({(const void*)fn, dev, (int)bytes});
    return 0;
}

namespace vggp {
thread_local char g_err[512] = {0};
unsigned long long g_launches = 0;
static int g_use_mma = 1;
static int g_bin_stream = 0;       // binned K1: 0 = LDG.128 register ping-pong, 1 = TMA ring through shared memory

constexpr int BAND_REPLICAS = 128;

struct ZeroJob { void* ptr; size_t pitch, width, height; };      // cudaMemset2DAsync of a split-K destination (beta = 0)
// epoch binning planned by vggp_epoch_bin_prepare (minibatch.cuh): the device arrays the pack reads, until vggp_epoch_bin_pack
struct MbPending {
    bool active = false;
    vggp_epoch_desc desc = {};
    std::vector<void*> keep;
    uint32_t* perm = nullptr;                          // sorted position -> input index (batch b from position b B)
    unsigned long long *task_base = nullptr, *run_off = nullptr, *batch_runs = nullptr;
    long long* task_goff = nullptr;
    int32_t *task_R = nullptr, *run_len = nullptr;
    uint32_t *run_sorted = nullptr, *run_cell = nullptr, *run_start = nullptr;
    void clear() {
        for (void* a : keep) cudaFree(a);
        *this = MbPending();
    }
};
struct Phase {
    GemmDesc* d_descs = nullptr;
    int ndesc = 0;
    GemmGroupDims dims = {0, 0, 0};
    std::vector<ZeroJob> zero;
};
}  // namespace vggp

using namespace vggp;

struct vggp_plan {
    int family, D, obs_dtype, device;
    int K[VGGP_MAX_D], n[VGGP_MAX_D];
    i64 M, Lsize;
    i64 stride[VGGP_MAX_D];
    float* d_knots[VGGP_MAX_D];
    MeshView mesh[VGGP_MAX_D];
    GridDims g;
    int nmax;
    // M-sized float64 work tensors (the B1 family allocates alpha, pgA and pgB only)
    double *mws, *alpha, *Tm[VGGP_MAX_D], *tmpM[VGGP_MAX_D], *gM, *ghat, *pgA, *pgB;
    void* alphaT;
    double* theta_dev;                     // copy of theta of the last forward (the B0 features depend on it)
    unsigned int* obs_counter;             // work-stealing counter of the per-observation kernel
    int band_off[VGGP_MAX_D], band_total, knot_off[VGGP_MAX_D], knot_total;
    int tab_off[VGGP_MAX_D], tab_total;
    i64 gfac_off[VGGP_MAX_D], gfac_total;   // B0 family: full factor-gradient blocks [bP | bQ] per dim
    double* gfac_f64 = nullptr;            // dense-feature families, float32 observations: [bP | bQ] of k_obs_b0 in float64
    unsigned char* tables;                 // [band tables (obs dtype) | pad16 | knots (float32) | pad16]
    int table_bytes, knots_byte_off;
    int sm_count, obs_blocks_per_sm;
    // scratch for vggp_obs_fwd_bwd on unpacked observations (grown on demand)
    void* pk_x[VGGP_MAX_D] = {nullptr, nullptr, nullptr}; void* pk_y = nullptr; i64 pk_cap = 0;
    // binned layout: the layout planned by vggp_obs_bin_prepare and the cell-sorted order, until vggp_obs_bin_pack
    BinLayout bin_pending; uint32_t* bin_perm = nullptr; bool bin_has_pending = false;
    MbPending mb;                          // epoch minibatches: vggp_epoch_bin_prepare until vggp_epoch_bin_pack
    // B0 family, scan form (b0scan.cuh): per-dimension transform rows and products, per-cell tables; allocated at first use
    bool b0s_ready = false;
    double* b0s_G[VGGP_MAX_D][4] = {};     // GL, GR, dGL/dl, dGR/dl: (K+1) x (K-1)
    double* b0s_V[VGGP_MAX_D][4] = {};     // GL P, GR P, GL Q, GR Q: (K+1) x (K-1)
    double* b0s_eps[VGGP_MAX_D] = {};      // [eps | gam | d eps / d l], K-1 each
    double* b0s_U[2] = {};                 // A G2^y^T: M1 x E2
    double* b0s_B[2] = {};                 // G1^x A:   E1 x M2
    double* b0s_TT[4] = {};                // G1^x U^y: E1 x E2
    void* b0s_W[VGGP_MAX_D] = {};          // [2][6][E_d] obs dtype
    void* b0s_Tt = nullptr;                // D = 1: [3][E1], D = 2: [3][3][E1][E2] obs dtype
    void* b0s_raw = nullptr; i64 b0s_raw_bytes = 0;   // raw per-cell sums of k_obs_b0s (obs dtype): [GT | GW_0 | GW_1]
    double* b0s_GTd = nullptr;             // GT in float64
    double* b0s_H[3] = {};                 // M1 x E2
    double* b0s_dA = nullptr;              // M1 x M2
    double* b0s_Sx[4][3] = {};             // (K+1) x (K-1), largest dimension: one set per (dimension, matrix) pair
    double* b0s_bMx[4] = {};               // (K-1) x (K-1), largest dimension, likewise
    double* b0s_tan[6][4] = {};            // D = 2: scratch sets of the six tangent sweeps, E1 x E2 each (set 0 = b0s_TT)
    double* b0s_Gam[2] = {};               // (K+1) x (K-1), largest dimension
    int bin_blocks_per_sm[2] = {0, 0};     // resident CTAs of k_obs_b1_binned / k_obs_b1_binned_tma (queried at first use)
    // optional device timing of the per-observation kernel (vggp_k1_timing)
    bool k1_timing = false; std::vector<cudaEvent_t> k1_ev; int k1_count = 0;
    cudaEvent_t k1_gev[2] = {nullptr, nullptr};      // the pair recorded by event nodes of a captured graph (vggp_k1_graph_time_read)
    bool k1_gev_captured = false;
    // product-grid SVGP, Markov form (svgpm.cuh): per-cell tables (obs dtype), float64 bands per dimension, scalars
    void* svm_tab = nullptr; int svm_tab_off[VGGP_MAX_D] = {0, 0, 0};
    double* svm_W[VGGP_MAX_D] = {}; double* svm_sc = nullptr;
    int svm_blocks_per_sm = 0;
    double* b1_acc = nullptr; int b1_acc_total = 0;      // B1 family: band accumulators of dK_d, [3][n_d] per dimension
    cudaStream_t last_stream = nullptr;                  // stream of the last grid forward (on-demand workspace fills)
    // deterministic mode (vggp_set_deterministic): run records + sort scratch of the per-observation kernel, per-CTA partials
    // of the fibre passes; both grown on demand (the first deterministic step must not run inside a stream capture)
    size_t alloc_bytes = 0;                // device memory taken at plan creation (vggp_workspace_bytes)
    void* one_ws = nullptr; size_t one_ws_bytes = 0;      // fix-up workspace of ad-hoc k-split products (vggp_mode_product)
    double* phase_ws = nullptr; int* phase_cnt = nullptr; // fix-up workspace shared by the scheduled GEMM groups (make_phase)
    int det = 0;
    void* det_buf = nullptr; size_t det_bytes = 0;
    double* det_fp = nullptr; size_t det_fp_elems = 0;
    // optimal variational mean (meanopt.cuh): G, b, the CG vectors, the B1 prior bands and the CG status in one buffer,
    // allocated at the first vggp_meanopt_assemble (scratch_bytes of vggp_workspace_bytes)
    void* mo_buf = nullptr; size_t mo_bytes = 0; bool mo_assembled = false;
    // the Kronecker-preconditioned solve's z vector, Thomas factors and trace, allocated at its first call (scratch_bytes)
    void* mo_kbuf = nullptr; size_t mo_kbytes = 0;
    bool mo_solved = false;                // a solve ran on the current assembly at the theta of the last forward
    int64_t mo_set[3] = {0, 0, 0};         // n, n_tasks, data_elems of the binned set of the current assembly
    // collapsed ELBO (collapsed.cuh): exact-term scratch, Lanczos vectors and coefficients; grown by vggp_logdet_system /
    // vggp_collapsed_terms (scratch_bytes)
    void* ct_buf = nullptr; size_t ct_bytes = 0;
    // optimal covariance (covopt.cuh): F band, U^-T recurrence, B1 X diagonals, change sums; allocated at the first
    // vggp_covopt_update (scratch_bytes)
    void* co_buf = nullptr; size_t co_bytes = 0;
    bool forwarded = false;                // a vggp_grid_forward has run on this plan
    void* band_rep = nullptr;              // B1 family, binned kernel: BAND_REPLICAS copies of the band block (obs dtype), kept zero
                                           // between launches (k_band_reduce clears what it sums)
    // GEMM schedules of the dense families
    std::vector<Phase> chol_trailing;      // one per panel (may be empty phase)
    int n_panels;
    std::vector<Phase> triinv;             // two launches per recursion depth, deepest first
    Phase pinv, rs, qq, alpha_phase, bwdA, bwdMid, bwdB, Yp, dKp, dRp;
    std::vector<Phase> chains;             // D-1 launches building T_d = m x_{e != d} P_e
    double* dm_result;
    std::vector<void*> allocs;
    // staging for vggp_elbo_host
    void* st_x = nullptr; void* st_y = nullptr; i64 st_n = 0;
    cudaStream_t st_copy = nullptr; std::vector<cudaEvent_t> st_ev;      // vggp_elbo_host: copy stream + one event per chunk
    double n_real_override = -1.0;      // >= 0: the observation count a chunked launch reports (vggp_elbo_host)
    double *st_theta = nullptr, *st_m = nullptr, *st_L = nullptr, *st_out = nullptr, *st_dtheta = nullptr,
           *st_dm = nullptr, *st_dL = nullptr;
    void* st_gbuf = nullptr;
};

namespace {

template <typename T>
int dev_alloc(vggp_plan* p, T** out, i64 count) {
    void* ptr = nullptr;
    if (count <= 0) count = 1;
    VGGP_CUDA(cudaMalloc(&ptr, (size_t)count * sizeof(T)));
    VGGP_CUDA(cudaMemset(ptr, 0, (size_t)count * sizeof(T)));
    p->allocs.push_back(ptr);
    p->alloc_bytes += (size_t)count * sizeof(T);
    *out = reinterpret_cast<T*>(ptr);
    return 0;
}

// A group with fewer output tiles than SMs (one 512^3 product is 64 CTAs on 148 SMs, each at ~45 % of its SM's DMMA rate)
// is cut along k so that about two CTAs land on every SM: partial sums go through float64 atomics into a destination that
// already holds beta * C (beta = 1: nothing to do; beta = 0: zero-filled by a cudaMemset2DAsync queued before the launch).
int g_auto_splitk = 1;
int g_splitk_fixup = 1;       // 1: automatic splits use the workspace fix-up (no destination clear, no atomics); 0: the atomic form
// returns the split factor applied to every descriptor of the group (1: none).  `zero`: destinations the atomic form must clear.
int auto_splitk(std::vector<GemmDesc>& descs, std::vector<ZeroJob>& zero, bool fixup) {
    zero.clear();
    if (!g_auto_splitk) return 1;
    i64 ctas = 0;
    int kmin = 1 << 30;
    for (const GemmDesc& d : descs) {
        const i64 tm = (d.m + GBM - 1) / GBM, tn = (d.n + GBN - 1) / GBN;
        ctas += (d.lower_only ? (tm * (tm + 1)) / 2 : tm * tn) * std::max(1, d.batch) * std::max(1, d.splitk);
        kmin = std::min(kmin, d.tri_b ? d.k / 2 : d.k);
        if (d.splitk > 1 || d.kinner != 0) return 1;
        if (!fixup && !(d.beta == 0.0 || d.beta == 1.0)) return 1;
        if (!fixup && d.beta == 0.0 && !(d.csC == 1 || d.rsC == 1)) return 1;
    }
    if (ctas <= 0 || ctas >= 148) return 1;
    int sk = (int)std::min<i64>(4, (2 * 148) / ctas);
    while (sk > 1 && kmin / sk < 4 * GBK) --sk;
    if (sk <= 1) return 1;
    for (GemmDesc& d : descs) {
        d.splitk = sk;
        if (fixup || d.beta != 0.0) continue;
        for (int b = 0; b < std::max(1, d.batch); ++b) {
            ZeroJob z;
            z.ptr = d.C + (i64)b * d.bsC;
            if (d.csC == 1) { z.pitch = sizeof(double) * (size_t)d.rsC; z.width = sizeof(double) * (size_t)d.n; z.height = (size_t)d.m; }
            else { z.pitch = sizeof(double) * (size_t)d.csC; z.width = sizeof(double) * (size_t)d.m; z.height = (size_t)d.n; }
            zero.push_back(z);
        }
    }
    return sk;
}
// workspace of the fix-up form for one descriptor: partial tiles (doubles) and tile counters
inline void splitk_ws_size(const GemmDesc& d, i64* ws_elems, i64* n_cnt) {
    const i64 tiles = (i64)((d.m + GBM - 1) / GBM) * ((d.n + GBN - 1) / GBN) * std::max(1, d.batch);
    *ws_elems = tiles * d.splitk * 4096;
    *n_cnt = tiles;
}

int make_phase(vggp_plan* p, std::vector<GemmDesc>& descs, Phase& ph) {
    ph.ndesc = (int)descs.size();
    if (ph.ndesc == 0) return 0;
    const bool fixup = g_splitk_fixup != 0;
    const int sk = auto_splitk(descs, ph.zero, fixup);
    int rc;
    if (sk > 1 && fixup) {
        // One workspace for every phase of the plan: launches are stream-ordered and a launch consumes its partials before it
        // ends; an automatically split group has fewer than 148 computed tiles and at most 2 x 148 computed partial tiles
        // (auto_splitk); the workspace is indexed by the full tile grid, at most twice that for lower-triangular outputs.  The
        // counters start at zero (dev_alloc) and return to zero after every launch.
        constexpr i64 WS_TILES = 4 * 148 + 16, WS_CNT = 2 * 148 + 8;
        if (!p->phase_ws) {
            if ((rc = dev_alloc(p, &p->phase_ws, WS_TILES * 4096))) return rc;
            if ((rc = dev_alloc(p, &p->phase_cnt, WS_CNT))) return rc;
        }
        i64 woff = 0, coff = 0;
        for (GemmDesc& d : descs) {
            i64 we, nc;
            splitk_ws_size(d, &we, &nc);
            if (woff + we > WS_TILES * 4096 || coff + nc > WS_CNT) return fail(VGGP_E_NOMEM, "k-split workspace too small for this group");
            d.ws = p->phase_ws + woff;
            d.cnt = p->phase_cnt + coff;
            woff += we;
            coff += nc;
        }
    }
    ph.dims = gemm_finalize_group(descs.data(), ph.ndesc);
    rc = dev_alloc(p, &ph.d_descs, ph.ndesc);
    if (rc) return rc;
    VGGP_CUDA(cudaMemcpy(ph.d_descs, descs.data(), sizeof(GemmDesc) * ph.ndesc, cudaMemcpyHostToDevice));
    return 0;
}

int launch_phase(const Phase& ph, cudaStream_t st) {
    if (ph.ndesc == 0) return 0;
    dim3 grid(ph.dims.gx, ph.dims.gy, ph.dims.gz);
    for (const ZeroJob& z : ph.zero) VGGP_CUDA(cudaMemset2DAsync(z.ptr, z.pitch, 0, z.width, z.height, st));
    if (g_use_mma) {
        if (int rc = raise_dyn_smem(k_gemm_group<true>, GEMM_SMEM_BYTES)) return rc;
        k_gemm_group<true><<<grid, GEMM_THREADS_MMA, GEMM_SMEM_BYTES, st>>>(ph.d_descs, ph.ndesc);
    } else {
        if (int rc = raise_dyn_smem(k_gemm_group<false>, GEMM_SMEM_BYTES)) return rc;
        k_gemm_group<false><<<grid, GEMM_THREADS_SIMT, GEMM_SMEM_BYTES, st>>>(ph.d_descs, ph.ndesc);
    }
    VGGP_LAUNCH_CHECK();
    return 0;
}

int det_reserve(void** buf, size_t* have, size_t want, cudaStream_t st);
// `p` (may be null): the plan whose grow-only scratch holds the fix-up workspace of an automatic k-split; without a plan the
// split uses the atomic form.
int launch_one(GemmDesc d, int use_mma, cudaStream_t st, vggp_plan* p = nullptr) {
    if (d.m <= 0 || d.n <= 0) return 0;
    std::vector<GemmDesc> one(1, d);
    std::vector<ZeroJob> zero;
    const bool fixup = p != nullptr && g_splitk_fixup != 0;
    if (d.splitk <= 1) {
        const int sk = auto_splitk(one, zero, fixup);
        if (sk > 1 && fixup) {
            i64 we, nc;
            splitk_ws_size(one[0], &we, &nc);
            const size_t cnt_off = ((size_t)we * sizeof(double) + 255) / 256 * 256;
            const size_t want = cnt_off + (size_t)nc * sizeof(int);
            if (p->one_ws_bytes < want) {          // grown: the counters start at zero (and return to zero after every launch)
                if (int rc = det_reserve(&p->one_ws, &p->one_ws_bytes, want, st)) return rc;
                VGGP_CUDA(cudaMemsetAsync(p->one_ws, 0, p->one_ws_bytes, st));
            }
            one[0].ws = reinterpret_cast<double*>(p->one_ws);
            one[0].cnt = reinterpret_cast<int*>(reinterpret_cast<unsigned char*>(p->one_ws) + cnt_off);
        }
    }
    d = one[0];
    GemmGroupDims dims = gemm_finalize_group(&d, 1);
    for (const ZeroJob& z : zero) VGGP_CUDA(cudaMemset2DAsync(z.ptr, z.pitch, 0, z.width, z.height, st));
    dim3 grid(dims.gx, dims.gy, dims.gz);
    if (use_mma) {
        if (int rc = raise_dyn_smem(k_gemm_one<true>, GEMM_SMEM_BYTES)) return rc;
        k_gemm_one<true><<<grid, GEMM_THREADS_MMA, GEMM_SMEM_BYTES, st>>>(d);
    } else {
        if (int rc = raise_dyn_smem(k_gemm_one<false>, GEMM_SMEM_BYTES)) return rc;
        k_gemm_one<false><<<grid, GEMM_THREADS_SIMT, GEMM_SMEM_BYTES, st>>>(d);
    }
    VGGP_LAUNCH_CHECK();
    return 0;
}

// plain row-major square matrix product helper: C (n x n) = alpha * op(A) * op(B) + beta * C
GemmDesc square_desc(int n, const double* A, bool tA, const double* B, bool tB, double* C, double alpha, double beta) {
    GemmDesc d;
    gemm_desc_defaults(d);
    d.A = A; d.B = B; d.C = C;
    d.m = d.n = d.k = n;
    d.rsA = tA ? 1 : n; d.csA = tA ? n : 1;
    d.rsB = tB ? 1 : n; d.csB = tB ? n : 1;
    d.rsC = n; d.csC = 1;
    d.alpha = alpha; d.beta = beta;
    return d;
}

// dst = src x_e A   (apply the M_e x M_e matrix A along mode e of the M-tensor)
GemmDesc mode_desc(const vggp_plan* p, int e, const double* A, const double* src, double* dst) {
    i64 outer = 1, inner = 1;
    for (int f = 0; f < e; ++f) outer *= p->n[f];
    for (int f = e + 1; f < p->D; ++f) inner *= p->n[f];
    const int ne = p->n[e];
    GemmDesc d;
    gemm_desc_defaults(d);
    if (inner > 1) {
        d.A = A; d.B = src; d.C = dst;
        d.m = ne; d.n = (int)inner; d.k = ne;
        d.rsA = ne; d.csA = 1;
        d.rsB = inner; d.csB = 1;
        d.rsC = inner; d.csC = 1;
        d.batch = (int)outer;
        d.bsA = 0; d.bsB = (i64)ne * inner; d.bsC = (i64)ne * inner;
    } else {
        // dst (outer x ne) = src (outer x ne) * A^T
        d.A = src; d.B = A; d.C = dst;
        d.m = (int)outer; d.n = ne; d.k = ne;
        d.rsA = ne; d.csA = 1;
        d.rsB = 1; d.csB = ne;
        d.rsC = ne; d.csC = 1;
    }
    return d;
}

// dP_d[i][j] = sum_{o,r} ghat[o,i,r] * T_d[o,j,r]
GemmDesc gram_desc(const vggp_plan* p, int e, const double* ghat, const double* Td, double* dP, int n_descs_in_group) {
    i64 outer = 1, inner = 1;
    for (int f = 0; f < e; ++f) outer *= p->n[f];
    for (int f = e + 1; f < p->D; ++f) inner *= p->n[f];
    const int ne = p->n[e];
    GemmDesc d;
    gemm_desc_defaults(d);
    d.A = ghat; d.B = Td; d.C = dP;
    d.m = ne; d.n = ne; d.k = (int)(outer * inner);
    if (outer == 1) {
        // first mode: A(i, k=r) = ghat[i][r], B(k=r, j) = T[j][r]
        d.rsA = inner; d.csA = 1; d.rsB = 1; d.csB = inner;
    } else if (inner == 1) {
        // last mode: A(i, k=o) = ghat[o][i], B(k=o, j) = T[o][j]
        d.rsA = 1; d.csA = ne; d.rsB = ne; d.csB = 1;
    } else {
        d.kinner = (int)inner;
        d.rsA = inner; d.csA = 1; d.koA = (i64)ne * inner;
        d.csB = inner; d.rsB = 1; d.koB = (i64)ne * inner;
    }
    d.rsC = ne; d.csC = 1;
    d.alpha = 1.0; d.beta = 0.0;
    const int tiles = ((ne + GBM - 1) / GBM) * ((ne + GBN - 1) / GBN) * n_descs_in_group;
    int sk = (2 * 148 + tiles - 1) / tiles;
    const int max_sk = std::max(1, d.k / (GBK * 8));
    sk = std::max(1, std::min(sk, max_sk));
    d.splitk = sk;
    return d;
}

void build_leaves(int lo, int hi, std::vector<int>& bounds) {
    if (hi - lo <= NB) { bounds.push_back(lo); return; }
    const int half = (hi - lo + 1) / 2;
    const int mid = lo + (half + NB - 1) / NB * NB;
    build_leaves(lo, mid, bounds);
    build_leaves(mid, hi, bounds);
}

struct Node { int lo, mid, hi, depth; };
void build_nodes(int lo, int hi, int depth, std::vector<Node>& nodes) {
    if (hi - lo <= NB) return;
    const int half = (hi - lo + 1) / 2;
    const int mid = lo + (half + NB - 1) / NB * NB;
    nodes.push_back({lo, mid, hi, depth});
    build_nodes(lo, mid, depth + 1, nodes);
    build_nodes(mid, hi, depth + 1, nodes);
}

GemmDesc sub_desc(int n, const double* A, int ar, int ac, const double* B, int br, int bc, double* C, int cr, int cc,
                  int m, int nn, int k, double alpha, double beta) {
    GemmDesc d;
    gemm_desc_defaults(d);
    d.A = A + (i64)ar * n + ac; d.B = B + (i64)br * n + bc; d.C = C + (i64)cr * n + cc;
    d.m = m; d.n = nn; d.k = k;
    d.rsA = n; d.csA = 1; d.rsB = n; d.csB = 1; d.rsC = n; d.csC = 1;
    d.alpha = alpha; d.beta = beta;
    return d;
}

// GEMM schedules of the dense grid side (B0, SVGP and VFF families)
int build_schedules(vggp_plan* p) {
    const int D = p->D;
    GridDims& g = p->g;
    int rc;
    // ---- Cholesky trailing updates, one phase per panel ----
    p->n_panels = (p->nmax + NB - 1) / NB;
    p->chol_trailing.resize(p->n_panels);
    for (int j = 0; j < p->n_panels; ++j) {
        std::vector<GemmDesc> ds;
        const int j0 = j * NB;
        for (int d = 0; d < D; ++d) {
            const int n = p->n[d];
            const int r0 = j0 + NB;
            if (r0 >= n) continue;
            GemmDesc x;
            gemm_desc_defaults(x);
            x.A = g.Kc[d] + (i64)r0 * n + j0;                  // panel (n - r0) x NB
            x.B = x.A;                                         // panel^T: B(k, j) = panel[j][k]
            x.C = g.Kc[d] + (i64)r0 * n + r0;
            x.m = n - r0; x.n = n - r0; x.k = NB;
            x.rsA = n; x.csA = 1; x.rsB = 1; x.csB = n; x.rsC = n; x.csC = 1;
            x.alpha = -1.0; x.beta = 1.0; x.lower_only = 1;
            ds.push_back(x);
        }
        if ((rc = make_phase(p, ds, p->chol_trailing[j]))) return rc;
    }
    // ---- triangular inverse recursion ----
    int max_depth = -1;
    std::vector<std::vector<Node>> nodes(D);
    for (int d = 0; d < D; ++d) {
        build_nodes(0, p->n[d], 0, nodes[d]);
        for (auto& nd : nodes[d]) max_depth = std::max(max_depth, nd.depth);
    }
    for (int depth = max_depth; depth >= 0; --depth) {
        std::vector<GemmDesc> s1, s2;
        for (int d = 0; d < D; ++d) {
            const int n = p->n[d];
            for (auto& nd : nodes[d]) {
                if (nd.depth != depth) continue;
                const int m1 = nd.mid - nd.lo, m2 = nd.hi - nd.mid;
                // tmp21 = C21 * W11 ; W21 = -W22 * tmp21
                s1.push_back(sub_desc(n, g.Kc[d], nd.mid, nd.lo, g.W[d], nd.lo, nd.lo, g.tmp[d], nd.mid, nd.lo, m2, m1, m1, 1.0, 0.0));
                s2.push_back(sub_desc(n, g.W[d], nd.mid, nd.mid, g.tmp[d], nd.mid, nd.lo, g.W[d], nd.mid, nd.lo, m2, m1, m2, -1.0, 0.0));
            }
        }
        Phase a, b;
        if ((rc = make_phase(p, s1, a))) return rc;
        if ((rc = make_phase(p, s2, b))) return rc;
        p->triinv.push_back(a);
        p->triinv.push_back(b);
    }
    // ---- P = W^T W ; R = P Lt ; Q = R R^T ----
    {
        std::vector<GemmDesc> a, b, c;
        for (int d = 0; d < D; ++d) {
            const int n = p->n[d];
            a.push_back(square_desc(n, g.W[d], true, g.W[d], false, g.P[d], 1.0, 0.0));
            {
                GemmDesc r = square_desc(n, g.P[d], false, g.Lt[d], false, g.R[d], 1.0, 0.0);
                r.tri_b = 1;                            // B = Lt is lower-triangular
                b.push_back(r);
            }
            c.push_back(square_desc(n, g.R[d], false, g.R[d], true, g.Q[d], 1.0, 0.0));
        }
        if ((rc = make_phase(p, a, p->pinv))) return rc;
        if ((rc = make_phase(p, b, p->rs))) return rc;
        if ((rc = make_phase(p, c, p->qq))) return rc;
    }
    // ---- chains T_d = m x_{e != d} P_e, then alpha = T_{D-1} x_{D-1} P_{D-1} ----
    if (D == 1) {
        p->Tm[0] = p->mws;
    }
    for (int s = 0; s + 1 < D; ++s) {
        std::vector<GemmDesc> ds;
        for (int d = 0; d < D; ++d) {
            // modes e != d in increasing order; step s uses the s-th of them
            int e = s;
            if (e >= d) e += 1;
            const bool first = (s == 0), last = (s == D - 2);
            const double* src = first ? p->mws : p->tmpM[d];
            double* dst = last ? p->Tm[d] : p->tmpM[d];
            ds.push_back(mode_desc(p, e, g.P[e], src, dst));
        }
        Phase ph;
        if ((rc = make_phase(p, ds, ph))) return rc;
        p->chains.push_back(ph);
    }
    {
        std::vector<GemmDesc> ds;
        ds.push_back(mode_desc(p, D - 1, g.P[D - 1], p->Tm[D - 1], p->alpha));
        if ((rc = make_phase(p, ds, p->alpha_phase))) return rc;
    }
    // ---- reverse pass, three grouped launches:
    //   bwdA = { first mode of (kron P) g,  Gram contractions dP_d }
    //   bwdB = { remaining modes of (kron P) g (D = 2: the last one),  dP_d += dR_d Lt_d^T,  dLraw_d = P_d dR_d }
    //   Yp   = { Y_d = P_d sym(dP_d) },  dKp = { dK_d = -Y_d P_d }
    // For D = 3 the middle mode of (kron P) g gets its own launch between bwdA and bwdB.
    {
        std::vector<GemmDesc> A, B, mid, y, k, dr;
        const double* src = p->gM;
        for (int e = 0; e < D; ++e) {
            double* dst = (e % 2 == 0) ? p->pgA : p->pgB;
            GemmDesc md = mode_desc(p, e, g.P[e], src, dst);
            if (e == 0) A.push_back(md);
            else if (e == D - 1) B.push_back(md);
            else mid.push_back(md);
            src = dst;
            p->dm_result = dst;
        }
        for (int d = 0; d < D; ++d) {
            const int n = p->n[d];
            A.push_back(gram_desc(p, d, p->ghat, p->Tm[d], g.dP[d], D));
            GemmDesc x1 = square_desc(n, g.dR[d], false, g.Lt[d], true, g.dP[d], 1.0, 1.0);
            x1.tri_b = 2;                                   // B = Lt^T
            B.push_back(x1);
            GemmDesc x2 = square_desc(n, g.P[d], false, g.dR[d], false, g.dLraw[d], 1.0, 0.0);
            x2.lower_only = 1;                              // only tril(dL) is used
            B.push_back(x2);
            y.push_back(square_desc(n, g.P[d], false, g.X[d], false, g.Y[d], 1.0, 0.0));
            k.push_back(square_desc(n, g.Y[d], false, g.P[d], false, g.dK[d], -1.0, 0.0));
            dr.push_back(square_desc(n, g.X[d], false, g.R[d], false, g.dR[d], 1.0, 0.0));   // dense family: dR = 2 cQ sym(bQ) R
        }
        if ((rc = make_phase(p, dr, p->dRp))) return rc;
        if ((rc = make_phase(p, A, p->bwdA))) return rc;
        if ((rc = make_phase(p, mid, p->bwdMid))) return rc;
        if ((rc = make_phase(p, B, p->bwdB))) return rc;
        if ((rc = make_phase(p, y, p->Yp))) return rc;
        if ((rc = make_phase(p, k, p->dKp))) return rc;
    }
    return 0;
}


// ---- fused B1 grid side (grid_b1.cuh) -------------------------------------------------------------------
long long* g_fp_dbg = nullptr;        // debug: phase stamps of the next fibre passes (vggp_debug_fp_stamps)

int fp_tile_F(int n, int want) {
    int F = want;
    while (F > 2 && fp_smem_bytes(n, F, true) > (size_t)200 * 1024) F >>= 1;
    return F;
}

FpTask fp_task(const vggp_plan* p, int kind, int d, i64 outer, i64 inner) {
    FpTask t;
    memset(&t, 0, sizeof(t));
    t.kind = kind; t.d = d; t.n = p->n[d];
    t.inner = inner; t.nfib = outer * inner;
    t.F = fp_tile_F(t.n, 8);
    if (kind == FP_QROW) {
        t.ntiles = (t.n + FP_WARPS - 1) / FP_WARPS;
    } else {
        const int nsrc = (kind == FP_GA) ? t.F / 2 : t.F;
        t.ntiles = (int)((t.nfib + nsrc - 1) / nsrc);
    }
    return t;
}

// Fibre packing of k_fibre_pass_fast: how many fibres (2^pk) share one 512-slot row.  Only the mode-product kinds, only while
// the launch still has about two tiles per SM (small problems are latency-bound: more, smaller CTAs finish sooner).
int g_fp_pack = 1;                   // 0: never, 1: by the tile-count rule below, 2: always (tests)
int fp_pack_log2(const FpTask& t) {
    if (!g_fp_pack || t.n > 256) return 0;
    if (!(t.kind == FP_PROD || t.kind == FP_ALPHA || t.kind == FP_DM || t.kind == FP_GA || t.kind == FP_GAONLY)) return 0;
    int npad = 64;
    while (npad < t.n) npad <<= 1;
    const int nsrc = (t.kind == FP_GA) ? FF_F / 2 : FF_F;
    int pk = 0;
    while ((512 >> (pk + 1)) >= npad && (g_fp_pack == 2 || t.nfib / ((i64)nsrc << (pk + 1)) >= 296)) ++pk;
    return pk;
}

FpTask fp_mode_task(const vggp_plan* p, int kind, int e) {
    i64 outer = 1, inner = 1;
    for (int f = 0; f < e; ++f) outer *= p->n[f];
    for (int f = e + 1; f < p->D; ++f) inner *= p->n[f];
    return fp_task(p, kind, e, outer, inner);
}

void fp_pass_init(const vggp_plan* p, FpPass& P, const double* theta, double ell_scale) {
    memset(&P, 0, sizeof(P));
    P.D = p->D; P.obs_f32 = p->obs_dtype == VGGP_F32; P.M = p->M;
    P.ell_scale = ell_scale; P.theta = theta;
    int off = 0;
    for (int d = 0; d < p->D; ++d) {
        P.gen[d] = p->g.gen[d];
        P.acc[d] = p->b1_acc + off;
        off += 3 * p->n[d];
        P.Qb[d] = p->g.Qb[d];
        P.tab_off[d] = p->tab_off[d];
    }
    P.sc = p->g.sc;
    P.bandT = p->tables;
    P.dbg = g_fp_dbg;
}

int det_reserve(void** buf, size_t* have, size_t want, cudaStream_t st);
int g_fp_fast = 1;                   // use k_fibre_pass_fast where it applies (M_d <= 512); 0: always the generic kernel (cross-check)

int fp_launch(vggp_plan* p, FpPass& P, cudaStream_t st) {
    if (P.ntasks == 0) return 0;
    int tiles = 0;
    size_t smem = 0, smem_fast = 0;
    bool fast = g_fp_fast != 0;
    for (int i = 0; i < P.ntasks; ++i)
        if (P.t[i].kind != FP_QROW && (P.t[i].n > 512 || P.t[i].F != FF_F)) fast = false;
    for (int i = 0; i < P.ntasks; ++i) {
        FpTask& t = P.t[i];
        if (t.kind != FP_QROW) {
            const bool aux = fp_kind_has_aux(t.kind);
            smem = std::max(smem, fp_smem_bytes(t.n, t.F, aux));
            smem_fast = std::max(smem_fast, ff_smem_bytes(aux));
            const int nsrc = (t.kind == FP_GA) ? t.F / 2 : t.F;
            t.pk = fast ? fp_pack_log2(t) : 0;
            t.ntiles = (int)((t.nfib + ((i64)nsrc << t.pk) - 1) / ((i64)nsrc << t.pk));
        }
        t.tile0 = tiles;
        tiles += t.ntiles;
    }
    const int ti = p->obs_dtype == VGGP_F32 ? 0 : 1;
    if (p->det) {
        if (!fast) return fail(VGGP_E_UNSUPPORTED, "deterministic mode needs the fast fibre engine (M_d <= 512)");
        void* buf = p->det_fp; size_t have = p->det_fp_elems * sizeof(double);
        const int rc = det_reserve(&buf, &have, (size_t)tiles * FP_DET_SLOT * sizeof(double), st);
        p->det_fp = reinterpret_cast<double*>(buf); p->det_fp_elems = have / sizeof(double);      // whatever det_reserve left behind
        if (rc) return rc;
        P.det = p->det_fp;
    }
    if (fast) {
        if (int rc = ti == 0 ? raise_dyn_smem(k_fibre_pass_fast<float>, smem_fast) : raise_dyn_smem(k_fibre_pass_fast<double>, smem_fast)) return rc;
        if (ti == 0) k_fibre_pass_fast<float><<<tiles, FP_THREADS, smem_fast, st>>>(P);
        else k_fibre_pass_fast<double><<<tiles, FP_THREADS, smem_fast, st>>>(P);
        VGGP_LAUNCH_CHECK();
        if (P.det) {
            k_fp_det_reduce<<<dim3(P.D, FP_DET_YB), 256, 0, st>>>(P);
            VGGP_LAUNCH_CHECK();
        }
        return 0;
    }
    if (int rc = ti == 0 ? raise_dyn_smem(k_fibre_pass<float>, smem) : raise_dyn_smem(k_fibre_pass<double>, smem)) return rc;
    if (ti == 0) k_fibre_pass<float><<<tiles, FP_THREADS, smem, st>>>(P);
    else k_fibre_pass<double><<<tiles, FP_THREADS, smem, st>>>(P);
    VGGP_LAUNCH_CHECK();
    return 0;
}

int b1f_forward(vggp_plan* p, const double* theta, const double* m, const double* L, cudaStream_t st) {
    const int D = p->D;
    int rc;
    const size_t gsm = 4 * ((size_t)p->nmax + p->nmax / 32 + 1) * sizeof(double);
    if (p->obs_dtype == VGGP_F32) k_b1_gens<float><<<D, GEN_THREADS, gsm, st>>>(p->g, theta, p->b1_acc, p->b1_acc_total, p->theta_dev);
    else k_b1_gens<double><<<D, GEN_THREADS, gsm, st>>>(p->g, theta, p->b1_acc, p->b1_acc_total, p->theta_dev);
    VGGP_LAUNCH_CHECK();
    FpPass P;
    auto qrows = [&](FpPass& Q) {
        for (int d = 0; d < D; ++d) {
            FpTask t = fp_task(p, FP_QROW, d, 1, p->n[d]);
            t.s0 = p->g.R[d]; t.s1 = L + p->g.Loff[d];
            Q.t[Q.ntasks++] = t;
        }
    };
    // pass 1: R_d = P_d tril(L_d) for every d, and the first mode of alpha = (kron P) m
    fp_pass_init(p, P, theta, 1.0);
    for (int d = 0; d < D; ++d) {
        FpTask t = fp_task(p, FP_R, d, 1, p->n[d]);
        t.s0 = L + p->g.Loff[d]; t.o0 = p->g.R[d];
        P.t[P.ntasks++] = t;
    }
    {
        FpTask t = fp_mode_task(p, D == 1 ? FP_ALPHA : FP_PROD, 0);
        t.s0 = m; t.s1 = m;
        t.o0 = D == 1 ? p->alpha : p->pgA;
        t.t1 = p->alphaT;
        P.t[P.ntasks++] = t;
    }
    if ((rc = fp_launch(p, P, st))) return rc;
    const double* src = p->pgA;
    if (D == 3) {     // middle mode, with the row reductions of R_d riding along
        fp_pass_init(p, P, theta, 1.0);
        FpTask t = fp_mode_task(p, FP_PROD, 1);
        t.s0 = p->pgA; t.o0 = p->pgB;
        P.t[P.ntasks++] = t;
        qrows(P);
        if ((rc = fp_launch(p, P, st))) return rc;
        src = p->pgB;
    }
    // last pass: last mode of alpha (+ cast, <m, alpha>) and the row reductions of R_d
    fp_pass_init(p, P, theta, 1.0);
    if (D >= 2) {
        FpTask t = fp_mode_task(p, FP_ALPHA, D - 1);
        t.s0 = src; t.s1 = m; t.o0 = p->alpha; t.t1 = p->alphaT;
        P.t[P.ntasks++] = t;
    }
    if (D != 3) qrows(P);
    return fp_launch(p, P, st);
}

int b1f_backward(vggp_plan* p, const double* theta, const double* m, const double* L, const void* gbuf, double ell_scale,
                 double* out, double* dtheta, double* dm, double* dL, cudaStream_t st) {
    const int D = p->D;
    int rc;
    const size_t tsz = p->obs_dtype == VGGP_F32 ? 4 : 8;
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    const unsigned char* gb = reinterpret_cast<const unsigned char*>(gbuf);
    const double* gscal = reinterpret_cast<const double*>(gb + soff);
    auto band = [&](int d) { return (const void*)(gb + ((size_t)p->M + p->band_off[d]) * tsz); };
    FpPass P;
    // pass 1 (last mode): V = g x P, A = ghat x P contracted with alpha
    fp_pass_init(p, P, theta, ell_scale);
    {
        FpTask t = fp_mode_task(p, FP_GA, D - 1);
        t.s0 = m; t.s1 = p->alpha; t.t0 = gbuf;
        t.direct = (D == 1);
        t.o0 = D == 1 ? dm : p->pgA;
        P.t[P.ntasks++] = t;
    }
    if ((rc = fp_launch(p, P, st))) return rc;
    // pass 2: next mode of the dm chain, its A_e contraction, dL_d (the band of P_d X_d P_d is formed in k_b1_theta)
    fp_pass_init(p, P, theta, ell_scale);
    if (D >= 2) {
        const int e = D - 2;
        FpTask t = fp_mode_task(p, e == 0 ? FP_DM : FP_PROD, e);
        t.s0 = p->pgA; t.s1 = p->alpha; t.o0 = e == 0 ? dm : p->pgB;
        P.t[P.ntasks++] = t;
        FpTask a = fp_mode_task(p, FP_GAONLY, e);
        a.s0 = m; a.s1 = p->alpha; a.t0 = gbuf;
        P.t[P.ntasks++] = a;
    }
    for (int d = 0; d < D; ++d) {
        FpTask t = fp_task(p, FP_DL, d, 1, p->n[d]);
        t.s0 = p->g.R[d]; t.s1 = L + p->g.Loff[d]; t.t0 = band(d); t.o0 = dL + p->g.Loff[d];
        P.t[P.ntasks++] = t;
    }
    if ((rc = fp_launch(p, P, st))) return rc;
    if (D == 3) {
        fp_pass_init(p, P, theta, ell_scale);
        FpTask t = fp_mode_task(p, FP_DM, 0);
        t.s0 = p->pgB; t.s1 = p->alpha; t.o0 = dm;
        P.t[P.ntasks++] = t;
        FpTask a = fp_mode_task(p, FP_GAONLY, 0);
        a.s0 = m; a.s1 = p->alpha; a.t0 = gbuf;
        P.t[P.ntasks++] = a;
        if ((rc = fp_launch(p, P, st))) return rc;
    }
    const size_t tsm = 7 * ((size_t)p->nmax + 34) * sizeof(double);
    if (int rc = p->obs_dtype == VGGP_F32 ? raise_dyn_smem(k_b1_theta<float>, tsm) : raise_dyn_smem(k_b1_theta<double>, tsm)) return rc;
    if (p->obs_dtype == VGGP_F32)
        k_b1_theta<float><<<D, 512, tsm, st>>>(p->g, theta, p->b1_acc, reinterpret_cast<const float*>(gb) + p->M, gscal, ell_scale, out, dtheta, g_fp_dbg);
    else
        k_b1_theta<double><<<D, 512, tsm, st>>>(p->g, theta, p->b1_acc, reinterpret_cast<const double*>(gb) + p->M, gscal, ell_scale, out, dtheta, g_fp_dbg);
    VGGP_LAUNCH_CHECK();
    return 0;
}

constexpr int K1_EVENT_PAIRS = 256;
inline void k1_mark(vggp_plan* p, int which, cudaStream_t st) {
    if (!p->k1_timing || p->k1_ev.empty()) return;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusActive) {
        // inside a stream capture: an external event-record node; every replay of the graph re-records the same pair
        if (p->k1_gev[which]) { cudaEventRecordWithFlags(p->k1_gev[which], st, cudaEventRecordExternal); p->k1_gev_captured = true; }
        return;
    }
    cudaEventRecord(p->k1_ev[2 * (p->k1_count % K1_EVENT_PAIRS) + which], st);
    if (which == 1) ++p->k1_count;
}

PackGeom pack_geometry(const vggp_plan* p, i64 n) {
    PackGeom g;
    // Chunks of 32 lanes x R observations are handed out dynamically to the resident (persistent) warps.  R is chosen so
    // that the number of chunks is just below a whole multiple `waves` of the resident warps: with R simply capped at
    // 512, 2^26 observations made 4096 chunks for 2960 warps, i.e. 1.38 chunks per warp -- most warps idled at the final
    // block reduction while the rest ran a second chunk (ncu: 17 % of the warp-cycles stalled on the barrier, 16.6 of 20
    // warps resident on average).
    const i64 target_lanes = (i64)p->sm_count * p->obs_blocks_per_sm * OBS_THREADS;
    const i64 waves = std::max<i64>(1, (n + target_lanes * 512 - 1) / (target_lanes * 512));
    i64 R = (n + target_lanes * waves - 1) / (target_lanes * waves);
    R = (R + 3) / 4 * 4;
    if (R < 16) R = 16;
    if (R > 512) R = 512;
    const i64 lanes = (n + R - 1) / R;
    g.R = (int)R;
    g.nwarps = (lanes + 31) / 32;
    g.n_packed = g.nwarps * 32 * R;
    return g;
}

template <typename T, int D>
size_t obs_smem_bytes(const vggp_plan* p) {
    return (size_t)p->table_bytes;
}

template <typename T, int D>
int obs_prepare(vggp_plan* p) {
    const size_t smem = obs_smem_bytes<T, D>(p);
    if (smem > 200 * 1024) return fail(VGGP_E_UNSUPPORTED, "band tables do not fit in shared memory");
    if (int rc = raise_dyn_smem(k_obs_b1<T, D>, smem)) return rc;
    int nb = 0;
    VGGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_obs_b1<T, D>, OBS_THREADS, smem));
    p->obs_blocks_per_sm = nb < 1 ? 1 : nb;
    return 0;
}

template <typename T, int D>
int launch_obs_packed(vggp_plan* p, const void* const* xp, const void* yp, i64 n, void* gbuf, cudaStream_t st) {
    PackedArgs<T, D> a;
    a.geo = pack_geometry(p, n);
    for (int d = 0; d < D; ++d) {
        a.xp[d] = reinterpret_cast<const T*>(xp[d]);
        a.mesh[d] = p->mesh[d];
        a.stride[d] = (int)p->stride[d];
        a.band_off[d] = p->band_off[d];
        a.tab_off[d] = p->tab_off[d];
        a.knot_off[d] = p->knot_off[d];
    }
    a.yp = reinterpret_cast<const T*>(yp);
    a.table_bytes = p->table_bytes;
    a.knots_byte_off = p->knots_byte_off;
    a.tables = p->tables;
    a.alpha = reinterpret_cast<const T*>(p->alphaT);
    T* gb = reinterpret_cast<T*>(gbuf);
    a.galpha = gb;
    a.gband = gb + p->M;
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    a.gs = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(gbuf) + soff);
    a.n_real = p->n_real_override >= 0.0 ? p->n_real_override : (double)n;
    a.counter = p->obs_counter;
    VGGP_CUDA(cudaMemsetAsync(p->obs_counter, 0, sizeof(unsigned int), st));
    i64 blocks = (a.geo.nwarps + (OBS_THREADS / 32) - 1) / (OBS_THREADS / 32);
    blocks = std::min<i64>(blocks, (i64)p->sm_count * p->obs_blocks_per_sm);
    k1_mark(p, 0, st);
    k_obs_b1<T, D><<<(unsigned)blocks, OBS_THREADS, obs_smem_bytes<T, D>(p), st>>>(a);
    k1_mark(p, 1, st);
    VGGP_LAUNCH_CHECK();
    return 0;
}

// device temporaries of a setup call: freed on every exit path unless released to a longer-lived owner
struct DevTemps {
    std::vector<void*> ptrs;
    ~DevTemps() { for (void* q : ptrs) if (q) cudaFree(q); }
    template <typename P>
    cudaError_t alloc(P** out, size_t bytes) {
        void* q = nullptr;
        const cudaError_t e = cudaMalloc(&q, bytes ? bytes : 1);
        if (e == cudaSuccess) ptrs.push_back(q);
        *out = reinterpret_cast<P*>(q);
        return e;
    }
    void release(void* q) { for (void*& r : ptrs) if (r == q) r = nullptr; }
};

template <typename T, int D>
int pack_impl(vggp_plan* p, const void* const* x, const void* y, i64 n, int sort_by_cell, void* const* xp, void* yp,
              cudaStream_t st) {
    GatherArgs<T, D> ga;
    ga.geo = pack_geometry(p, n);
    ga.n = n;
    ga.perm = nullptr;
    for (int d = 0; d < D; ++d) {
        ga.x[d] = reinterpret_cast<const T*>(x[d]);
        ga.xp[d] = reinterpret_cast<T*>(xp[d]);
    }
    ga.y = reinterpret_cast<const T*>(y);
    ga.yp = reinterpret_cast<T*>(yp);
    uint32_t *keys_in = nullptr, *keys_out = nullptr, *idx_in = nullptr, *idx_out = nullptr;
    void* temp = nullptr;
    DevTemps tmp;                 // freed on every return path; the stream is drained first on the normal path
    if (sort_by_cell && n > 0) {
        if (n >= ((i64)1 << 31)) return fail(VGGP_E_UNSUPPORTED, "binning supports n < 2^31 observations per shard");
        i64 ncells = 1;
        KeyArgs<T, D> ka;
        ka.n = n;
        for (int d = 0; d < D; ++d) {
            ka.x[d] = ga.x[d];
            ka.mesh[d] = p->mesh[d];
            ncells *= (p->K[d] - 1);
        }
        if (ncells >= ((i64)1 << 32) - 1) return fail(VGGP_E_UNSUPPORTED, "too many cells for 32-bit keys");
        VGGP_CUDA(tmp.alloc(&keys_in, sizeof(uint32_t) * n));
        VGGP_CUDA(tmp.alloc(&keys_out, sizeof(uint32_t) * n));
        VGGP_CUDA(tmp.alloc(&idx_in, sizeof(uint32_t) * n));
        VGGP_CUDA(tmp.alloc(&idx_out, sizeof(uint32_t) * n));
        const int blocks = (int)std::min<i64>((n + 255) / 256, 148 * 16);
        k_cell_keys<T, D><<<blocks, 256, 0, st>>>(ka, (uint32_t)ncells, keys_in, idx_in);
        VGGP_LAUNCH_CHECK();
        int end_bit = 1;
        while (((i64)1 << end_bit) <= ncells) ++end_bit;
        size_t temp_bytes = 0;
        VGGP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys_in, keys_out, idx_in, idx_out, (int)n, 0, end_bit, st));
        VGGP_CUDA(tmp.alloc(&temp, temp_bytes));
        VGGP_CUDA(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys_in, keys_out, idx_in, idx_out, (int)n, 0, end_bit, st));
        ga.perm = idx_out;
    }
    if (ga.geo.n_packed > 0) {
        const int blocks = (int)std::min<i64>((ga.geo.n_packed + 255) / 256, 148 * 16);
        k_pack_gather<T, D><<<blocks, 256, 0, st>>>(ga);
        VGGP_LAUNCH_CHECK();
    }
    if (keys_in) VGGP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

template <typename T, int D>
int launch_obs_b0(vggp_plan* p, const void* const* x, const void* y, i64 n, void* gbuf, cudaStream_t st) {
    B0Args<T, D> a;
    int ntot = 0;
    for (int d = 0; d < D; ++d) {
        a.x[d] = reinterpret_cast<const T*>(x[d]);
        a.mesh[d] = p->mesh[d];
        a.nd[d] = p->n[d];
        a.P[d] = p->g.P[d];
        a.Q[d] = p->g.Q[d];
        a.gfac_off[d] = p->gfac_off[d];
        ntot += p->n[d];
    }
    a.family = p->family;
    a.y = reinterpret_cast<const T*>(y);
    a.n = n;
    a.theta = p->theta_dev;
    a.alpha = reinterpret_cast<const T*>(p->alphaT);
    T* gb = reinterpret_cast<T*>(gbuf);
    a.galpha = gb;
    constexpr bool f32 = sizeof(T) == 4;
    a.gfac = f32 ? p->gfac_f64 : reinterpret_cast<double*>(gb + p->M);
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    a.gs = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(gbuf) + soff);
    const size_t smem = (size_t)5 * ntot * B0_TN * sizeof(T);
    if (smem > 200 * 1024) return fail(VGGP_E_UNSUPPORTED, "B0 feature tiles do not fit in shared memory");
    if (int rc = raise_dyn_smem(k_obs_b0<T, D>, smem)) return rc;
    if (f32) VGGP_CUDA(cudaMemsetAsync(p->gfac_f64, 0, sizeof(double) * p->gfac_total, st));
    const i64 tiles = (n + B0_TN - 1) / B0_TN;
    const int blocks = (int)std::min<i64>(tiles, (i64)p->sm_count * 2);
    k1_mark(p, 0, st);
    k_obs_b0<T, D><<<blocks, 256, smem, st>>>(a);
    k1_mark(p, 1, st);
    VGGP_LAUNCH_CHECK();
    if (f32) {      // the caller cleared the gbuf (vggp_obs_fwd_bwd): the float64 sums replace its [bP | bQ] blocks
        k_b0s_from_double<T><<<ceil_div(p->gfac_total, 256), 256, 0, st>>>(p->gfac_f64, gb + p->M, p->gfac_total);
        VGGP_LAUNCH_CHECK();
    }
    return 0;
}

template <typename T, int D>
int launch_predict(vggp_plan* p, const void* const* x, i64 n, void* mean, void* var, cudaStream_t st) {
    PredictArgs<T, D> a;
    for (int d = 0; d < D; ++d) {
        a.x[d] = reinterpret_cast<const T*>(x[d]);
        a.mesh[d] = p->mesh[d];
        a.stride[d] = (int)p->stride[d];
        a.tab_off[d] = p->tab_off[d];
    }
    a.n = n;
    a.tab = reinterpret_cast<const T*>(p->tables);
    a.alpha = reinterpret_cast<const T*>(p->alphaT);
    a.theta = p->theta_dev;
    a.mean = reinterpret_cast<T*>(mean);
    a.var = reinterpret_cast<T*>(var);
    const int blocks = (int)std::min<i64>((n + 255) / 256, 148 * 8);
    k_predict_b1<T, D><<<blocks, 256, 0, st>>>(a);
    VGGP_LAUNCH_CHECK();
    return 0;
}
int predict_dispatch(vggp_plan* p, const void* const* x, i64 n, void* mean, void* var, cudaStream_t st);

template <typename T, int D>
int launch_predict_metrics(vggp_plan* p, const void* const* x, const void* y, i64 n, double* out, cudaStream_t st) {
    PredictMetricsArgs<T, D> m;
    for (int d = 0; d < D; ++d) {
        m.p.x[d] = reinterpret_cast<const T*>(x[d]);
        m.p.mesh[d] = p->mesh[d];
        m.p.stride[d] = (int)p->stride[d];
        m.p.tab_off[d] = p->tab_off[d];
    }
    m.p.n = n;
    m.p.tab = reinterpret_cast<const T*>(p->tables);
    m.p.alpha = reinterpret_cast<const T*>(p->alphaT);
    m.p.theta = p->theta_dev;
    m.p.mean = nullptr;
    m.p.var = nullptr;
    m.y = reinterpret_cast<const T*>(y);
    m.out = out;
    const int blocks = (int)std::min<i64>((n + 255) / 256, (i64)p->sm_count * 8);
    k_predict_metrics<T, D><<<blocks, 256, 0, st>>>(m);
    VGGP_LAUNCH_CHECK();
    return 0;
}
int predict_metrics_dispatch(vggp_plan* p, const void* const* x, const void* y, i64 n, double* out, cudaStream_t st);

int obs_b0_dispatch(vggp_plan* p, const void* const* x, const void* y, i64 n, void* gbuf, cudaStream_t st) {
    if (p->D > 2) return fail(VGGP_E_UNSUPPORTED, "the B0 (cell-integrated) family is built for D <= 2, as in the reference");
    if (p->obs_dtype == VGGP_F32) return p->D == 1 ? launch_obs_b0<float, 1>(p, x, y, n, gbuf, st) : launch_obs_b0<float, 2>(p, x, y, n, gbuf, st);
    return p->D == 1 ? launch_obs_b0<double, 1>(p, x, y, n, gbuf, st) : launch_obs_b0<double, 2>(p, x, y, n, gbuf, st);
}

#define VGGP_DISPATCH_TD(p, FN, ...)                                                        \
    do {                                                                                    \
        if ((p)->obs_dtype == VGGP_F32) {                                                   \
            switch ((p)->D) {                                                               \
                case 1: return FN<float, 1>(__VA_ARGS__);                                   \
                case 2: return FN<float, 2>(__VA_ARGS__);                                   \
                case 3: return FN<float, 3>(__VA_ARGS__);                                   \
            }                                                                               \
        } else {                                                                            \
            switch ((p)->D) {                                                               \
                case 1: return FN<double, 1>(__VA_ARGS__);                                  \
                case 2: return FN<double, 2>(__VA_ARGS__);                                  \
                case 3: return FN<double, 3>(__VA_ARGS__);                                  \
            }                                                                               \
        }                                                                                   \
        return fail(VGGP_E_DIM, "D must be 1..3");                                          \
    } while (0)

int obs_prepare_dispatch(vggp_plan* p) { VGGP_DISPATCH_TD(p, obs_prepare, p); }
int predict_dispatch(vggp_plan* p, const void* const* x, i64 n, void* mean, void* var, cudaStream_t st) {
    VGGP_DISPATCH_TD(p, launch_predict, p, x, n, mean, var, st);
}
int predict_metrics_dispatch(vggp_plan* p, const void* const* x, const void* y, i64 n, double* out, cudaStream_t st) {
    VGGP_DISPATCH_TD(p, launch_predict_metrics, p, x, y, n, out, st);
}
int obs_packed_dispatch(vggp_plan* p, const void* const* xp, const void* yp, i64 n, void* gbuf, cudaStream_t st) {
    VGGP_DISPATCH_TD(p, launch_obs_packed, p, xp, yp, n, gbuf, st);
}
int pack_dispatch(vggp_plan* p, const void* const* x, const void* y, i64 n, int sort, void* const* xp, void* yp, cudaStream_t st) {
    VGGP_DISPATCH_TD(p, pack_impl, p, x, y, n, sort, xp, yp, st);
}

// ---- binned layout (obs_binned.cuh) ---------------------------------------------------------------------
template <typename T, int D>
int bin_prepare_impl(vggp_plan* p, const void* const* x, i64 n, int run_cap, vggp_binned_desc* desc, cudaStream_t st) {
    i64 ncells = 1;
    // B0 and Markov-SVGP families: extended cells (observations outside the mesh contribute)
    const bool ext = p->family == VGGP_B0_GRIDDED || p->family == VGGP_SVGP_MARKOV;
    for (int d = 0; d < D; ++d) ncells *= (ext ? p->K[d] + 1 : p->K[d] - 1);
    if (ncells >= ((i64)1 << 32) - 1) return fail(VGGP_E_UNSUPPORTED, "too many cells for 32-bit keys");
    std::vector<uint32_t> count((size_t)ncells + 1, 0u);
    if (n > 0) {
        KeyArgs<T, D> ka;
        ka.n = n;
        for (int d = 0; d < D; ++d) {
            ka.x[d] = reinterpret_cast<const T*>(x[d]);
            ka.mesh[d] = p->mesh[d];
        }
        DevTemps tmp;
        uint32_t *keys_in = nullptr, *keys_out = nullptr, *idx_in = nullptr, *idx_out = nullptr, *d_count = nullptr;
        unsigned char* temp = nullptr;
        VGGP_CUDA(tmp.alloc(&keys_in, sizeof(uint32_t) * n));
        VGGP_CUDA(tmp.alloc(&keys_out, sizeof(uint32_t) * n));
        VGGP_CUDA(tmp.alloc(&idx_in, sizeof(uint32_t) * n));
        VGGP_CUDA(tmp.alloc(&idx_out, sizeof(uint32_t) * n));
        VGGP_CUDA(tmp.alloc(&d_count, sizeof(uint32_t) * (ncells + 1)));
        VGGP_CUDA(cudaMemsetAsync(d_count, 0, sizeof(uint32_t) * (ncells + 1), st));
        const int blocks = (int)std::min<i64>((n + 255) / 256, 148 * 16);
        if (ext) {       // extended cells: every observation has one (b0scan.cuh)
            B0sKeyArgs<T, D> kb;
            kb.n = n;
            for (int d = 0; d < D; ++d) { kb.x[d] = ka.x[d]; kb.mesh[d] = p->mesh[d]; }
            k_b0s_keys<T, D><<<blocks, 256, 0, st>>>(kb, keys_in, idx_in);
        } else {
            k_cell_keys<T, D><<<blocks, 256, 0, st>>>(ka, (uint32_t)ncells, keys_in, idx_in);
        }
        VGGP_LAUNCH_CHECK();
        k_bin_histogram<<<blocks, 256, 0, st>>>(keys_in, n, d_count);
        VGGP_LAUNCH_CHECK();
        int end_bit = 1;
        while (((i64)1 << end_bit) <= ncells) ++end_bit;
        size_t temp_bytes = 0;
        VGGP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys_in, keys_out, idx_in, idx_out, (int)n, 0, end_bit, st));
        VGGP_CUDA(tmp.alloc(&temp, temp_bytes));
        VGGP_CUDA(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys_in, keys_out, idx_in, idx_out, (int)n, 0, end_bit, st));
        VGGP_CUDA(cudaMemcpyAsync(count.data(), d_count, sizeof(uint32_t) * (ncells + 1), cudaMemcpyDeviceToHost, st));
        VGGP_CUDA(cudaStreamSynchronize(st));
        tmp.release(idx_out);                    // the cell-sorted order lives on until vggp_obs_bin_pack
        p->bin_perm = idx_out;
    }
    if (plan_bins(count.data(), ncells, run_cap, D, p->bin_pending) != 0) return fail(VGGP_E_ARG, "run_cap must be >= 4");
    if (p->bin_pending.n != n) return fail(VGGP_E_ARG, "internal: cell histogram does not add up to n");
    p->bin_has_pending = true;
    const BinLayout& L = p->bin_pending;
    const BinOffsets o = bin_offsets(L.n_tasks, L.data_elems, (int)sizeof(T));
    desc->bytes = o.bytes; desc->n = n; desc->n_inside = L.n_inside; desc->n_tasks = L.n_tasks; desc->n_runs = L.n_runs;
    desc->data_elems = L.data_elems;
    desc->off_task_off = o.task_off; desc->off_task_R = o.task_R; desc->off_run_cell = o.run_cell; desc->off_run_n = o.run_n;
    desc->off_run_start = o.run_start; desc->off_data = o.data;
    desc->run_cap = run_cap / 4 * 4; desc->D = D;
    return 0;
}

// data blocks of one binned set whose tables are already in `buf`: perm maps its stream positions to input indices
template <typename T, int D>
int launch_bin_gather(vggp_plan* p, const void* const* x, const void* y, const uint32_t* perm, unsigned char* buf,
                      const vggp_binned_desc* desc, i64 n_tasks, cudaStream_t st) {
    const int blocks = (int)std::min<i64>(n_tasks, (i64)p->sm_count * 8);
    if (p->family == VGGP_B0_GRIDDED || p->family == VGGP_SVGP_MARKOV) {
        B0sGatherArgs<T, D> gb0;
        for (int d = 0; d < D; ++d) {
            gb0.x[d] = reinterpret_cast<const T*>(x[d]);
            gb0.knots[d] = p->d_knots[d];
            gb0.K[d] = p->K[d];
        }
        gb0.y = reinterpret_cast<const T*>(y);
        gb0.perm = perm;
        gb0.buf = buf;
        gb0.off_task_off = desc->off_task_off; gb0.off_task_R = desc->off_task_R; gb0.off_run_cell = desc->off_run_cell;
        gb0.off_run_n = desc->off_run_n; gb0.off_run_start = desc->off_run_start; gb0.off_data = desc->off_data;
        gb0.n_tasks = (int)n_tasks;
        k_b0s_gather<T, D><<<blocks, 256, 0, st>>>(gb0);
    } else {
        BinGatherArgs<T, D> ga;
        for (int d = 0; d < D; ++d) {
            ga.x[d] = reinterpret_cast<const T*>(x[d]);
            ga.knots[d] = p->d_knots[d];
            ga.K[d] = p->K[d];
        }
        ga.y = reinterpret_cast<const T*>(y);
        ga.perm = perm;
        ga.buf = buf;
        ga.off_task_off = desc->off_task_off; ga.off_task_R = desc->off_task_R; ga.off_run_cell = desc->off_run_cell;
        ga.off_run_n = desc->off_run_n; ga.off_run_start = desc->off_run_start; ga.off_data = desc->off_data;
        ga.n_tasks = (int)n_tasks;
        k_bin_gather<T, D><<<blocks, 256, 0, st>>>(ga);
    }
    VGGP_LAUNCH_CHECK();
    return 0;
}

template <typename T, int D>
int bin_pack_impl(vggp_plan* p, const vggp_binned_desc* desc, const void* const* x, const void* y, void* binned,
                  cudaStream_t st) {
    const BinLayout& L = p->bin_pending;
    unsigned char* buf = reinterpret_cast<unsigned char*>(binned);
    VGGP_CUDA(cudaMemsetAsync(buf, 0, BIN_HEADER_BYTES, st));
    if (L.n_tasks > 0) {
        VGGP_CUDA(cudaMemcpyAsync(buf + desc->off_task_off, L.task_off.data(), sizeof(int64_t) * L.n_tasks, cudaMemcpyHostToDevice, st));
        VGGP_CUDA(cudaMemcpyAsync(buf + desc->off_task_R, L.task_R.data(), sizeof(int32_t) * L.n_tasks, cudaMemcpyHostToDevice, st));
        VGGP_CUDA(cudaMemcpyAsync(buf + desc->off_run_cell, L.run_cell.data(), sizeof(uint32_t) * 32 * L.n_tasks, cudaMemcpyHostToDevice, st));
        VGGP_CUDA(cudaMemcpyAsync(buf + desc->off_run_n, L.run_n.data(), sizeof(int32_t) * 32 * L.n_tasks, cudaMemcpyHostToDevice, st));
        VGGP_CUDA(cudaMemcpyAsync(buf + desc->off_run_start, L.run_start.data(), sizeof(uint32_t) * 32 * L.n_tasks, cudaMemcpyHostToDevice, st));
        if (int rc = launch_bin_gather<T, D>(p, x, y, p->bin_perm, buf, desc, L.n_tasks, st)) return rc;
    }
    if (L.n > L.n_inside) {
        const i64 nout = L.n - L.n_inside;
        const int blocks = (int)std::min<i64>((nout + 255) / 256, 148 * 4);
        k_bin_sum_y2<T><<<blocks, 256, 0, st>>>(reinterpret_cast<const T*>(y), p->bin_perm, L.n_inside, L.n,
                                                reinterpret_cast<double*>(buf));
        VGGP_LAUNCH_CHECK();
    }
    VGGP_CUDA(cudaStreamSynchronize(st));
    if (p->bin_perm) cudaFree(p->bin_perm);
    p->bin_perm = nullptr;
    p->bin_pending = BinLayout();
    p->bin_has_pending = false;
    return 0;
}

template <typename T, int D>
int launch_obs_binned(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, void* gbuf, cudaStream_t st) {
    const int mode = g_bin_stream ? 1 : 0;
    const size_t smem = mode ? bin_tma_smem_bytes<T, D>() : 0;
    if (p->bin_blocks_per_sm[mode] == 0) {
        int nb = 0;
        if (mode) {
            if (int rc2 = raise_dyn_smem(k_obs_b1_binned_tma<T, D>, smem)) return rc2;
            VGGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_obs_b1_binned_tma<T, D>, BIN_THREADS, smem));
        } else {
            VGGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_obs_b1_binned<T, D>, BIN_THREADS, smem));
        }
        p->bin_blocks_per_sm[mode] = nb < 1 ? 1 : nb;
    }
    BinnedArgs<T, D> a;
    for (int d = 0; d < D; ++d) {
        a.geo.K[d] = p->K[d];
        a.geo.stride[d] = (int)p->stride[d];
        a.geo.band_off[d] = p->band_off[d];
        a.geo.tab_off[d] = p->tab_off[d];
        a.geo.knot_off[d] = p->knot_off[d];
    }
    a.buf = reinterpret_cast<const unsigned char*>(binned);
    a.off_task_off = desc->off_task_off; a.off_task_R = desc->off_task_R; a.off_run_cell = desc->off_run_cell;
    a.off_run_n = desc->off_run_n; a.off_data = desc->off_data;
    a.n_tasks = (int)desc->n_tasks;
    a.knots_byte_off = p->knots_byte_off;
    a.tables = p->tables;
    a.alpha = reinterpret_cast<const T*>(p->alphaT);
    T* gb = reinterpret_cast<T*>(gbuf);
    a.galpha = gb;
    a.gband = reinterpret_cast<T*>(p->band_rep);
    a.n_rep = BAND_REPLICAS;
    a.band_rep_stride = p->band_total;
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    a.gs = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(gbuf) + soff);
    a.n_real = (double)desc->n;
    a.counter = p->obs_counter + 1;              // slot 1: reset by k_band_reduce after every launch (slot 0: the other kernels)
    i64 blocks = (desc->n_tasks + BIN_WARPS - 1) / BIN_WARPS;
    blocks = std::max<i64>(1, std::min<i64>(blocks, (i64)p->sm_count * p->bin_blocks_per_sm[mode]));
    k1_mark(p, 0, st);
    if (mode) k_obs_b1_binned_tma<T, D><<<(unsigned)blocks, BIN_THREADS, smem, st>>>(a);
    else k_obs_b1_binned<T, D><<<(unsigned)blocks, BIN_THREADS, 0, st>>>(a);
    k1_mark(p, 1, st);
    VGGP_LAUNCH_CHECK();
    k_band_reduce<T><<<ceil_div(p->band_total, 16), 256, 0, st>>>(a.gband, BAND_REPLICAS, a.band_rep_stride, p->band_total, gb + p->M, a.counter);
    VGGP_LAUNCH_CHECK();
    return 0;
}

int bin_prepare_dispatch(vggp_plan* p, const void* const* x, i64 n, int cap, vggp_binned_desc* desc, cudaStream_t st) {
    VGGP_DISPATCH_TD(p, bin_prepare_impl, p, x, n, cap, desc, st);
}
int bin_pack_dispatch(vggp_plan* p, const vggp_binned_desc* desc, const void* const* x, const void* y, void* binned, cudaStream_t st) {
    VGGP_DISPATCH_TD(p, bin_pack_impl, p, desc, x, y, binned, st);
}
// ---- epoch minibatches in the binned layout (minibatch.cuh) ----------------------------------------------
inline int mb_bits(uint64_t max_value) {        // tight end_bit of a radix sort whose largest key is max_value
    int b = 1;
    while (b < 64 && (max_value >> b) != 0) ++b;
    return b;
}

template <typename KT>
int mb_sort_pairs(const KT* kin, KT* kout, const uint32_t* vin, uint32_t* vout, i64 n, int end_bit, DevTemps& tmp,
                  cudaStream_t st) {
    size_t bytes = 0;
    VGGP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, kin, kout, vin, vout, (int)n, 0, end_bit, st));
    void* temp = nullptr;
    VGGP_CUDA(tmp.alloc(&temp, bytes));
    VGGP_CUDA(cub::DeviceRadixSort::SortPairs(temp, bytes, kin, kout, vin, vout, (int)n, 0, end_bit, st));
    return 0;
}

template <typename V, typename W>
int mb_exclusive_sum(const V* in, W* out, i64 n, DevTemps& tmp, cudaStream_t st) {
    size_t bytes = 0;
    VGGP_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, n, st));
    void* temp = nullptr;
    VGGP_CUDA(tmp.alloc(&temp, bytes));
    VGGP_CUDA(cub::DeviceScan::ExclusiveSum(temp, bytes, in, out, n, st));
    return 0;
}

// The per-batch binned descriptor and view offset (bytes from the epoch buffer) of batch b.  totals[MB_TOTALS b + 4] is the
// byte offset of the batch's first section; its sections follow in the order and alignment of bin_offsets.
void mb_batch_desc(const vggp_epoch_desc* e, const int64_t* totals, i64 b, vggp_binned_desc* out, int64_t* view_off) {
    const int64_t* t = totals + MB_TOTALS * b;
    const BinOffsets o = bin_offsets(t[0], t[3], e->elem_size);
    const i64 view = (i64)BIN_HEADER_BYTES * b, rel = t[4] - o.task_off - view;   // section offsets relative to the view
    memset(out, 0, sizeof(*out));
    out->bytes = o.bytes + rel;
    out->n = e->batch_size; out->n_inside = t[2]; out->n_tasks = t[0]; out->n_runs = t[1]; out->data_elems = t[3];
    out->off_task_off = o.task_off + rel; out->off_task_R = o.task_R + rel; out->off_run_cell = o.run_cell + rel;
    out->off_run_n = o.run_n + rel; out->off_run_start = o.run_start + rel; out->off_data = o.data + rel;
    out->run_cap = e->run_cap; out->D = e->D;
    *view_off = view;
}

template <typename T, int D, typename KT>
int epoch_prepare_kt(vggp_plan* p, const void* const* x, vggp_epoch_desc* e, int64_t* totals, cudaStream_t st) {
    const bool ext = p->family == VGGP_B0_GRIDDED || p->family == VGGP_SVGP_MARKOV;
    const i64 n = e->n, B = e->batch_size, P = e->n_batches, m = P * B;
    const uint32_t cap = (uint32_t)e->run_cap;
    i64 ncells = 1;
    for (int d = 0; d < D; ++d) ncells *= (ext ? p->K[d] + 1 : p->K[d] - 1);
    const i64 nck = ext ? ncells : ncells + 1;                  // cell keys per batch (B1: the outside key last)
    const int blocks_n = (int)std::min<i64>((n + 256) / 256, (i64)p->sm_count * 16);
    const int blocks_m = (int)std::min<i64>((m + 256) / 256, (i64)p->sm_count * 16);
    DevTemps tmp;
    // 1. keys (batch, cell) with the permutation fused in, one radix sort
    KT *keys_in = nullptr, *keys = nullptr;
    uint32_t *idx_in = nullptr, *perm = nullptr;
    VGGP_CUDA(tmp.alloc(&keys_in, sizeof(KT) * n));
    VGGP_CUDA(tmp.alloc(&keys, sizeof(KT) * n));
    VGGP_CUDA(tmp.alloc(&idx_in, sizeof(uint32_t) * n));
    VGGP_CUDA(tmp.alloc(&perm, sizeof(uint32_t) * n));
    MbKeyArgs<T, D> ka;
    for (int d = 0; d < D; ++d) { ka.x[d] = reinterpret_cast<const T*>(x[d]); ka.mesh[d] = p->mesh[d]; }
    ka.perm = mb_perm_make(n, e->seed, e->epoch, e->rank);
    ka.B = (uint32_t)B; ka.P = (uint32_t)P; ka.ncell_keys = (uint64_t)nck; ka.ext = ext ? 1 : 0;
    k_mb_keys<T, D, KT><<<blocks_n, 256, 0, st>>>(ka, keys_in, idx_in);
    VGGP_LAUNCH_CHECK();
    if (int rc = mb_sort_pairs<KT>(keys_in, keys, idx_in, perm, n, mb_bits((uint64_t)P * (uint64_t)nck), tmp, st)) return rc;
    // 2. segments of equal key among the m kept positions, runs per segment, per-batch sums
    uint32_t *flags = nullptr, *segid = nullptr, *seg_start = nullptr, *seg_nruns = nullptr, *run_base = nullptr;
    for (uint32_t** a : {&flags, &segid, &seg_start, &seg_nruns, &run_base}) VGGP_CUDA(tmp.alloc(a, sizeof(uint32_t) * (m + 1)));
    unsigned long long *batch_runs = nullptr, *batch_inside = nullptr, *run_off = nullptr, *batch_tasks = nullptr, *task_base = nullptr;
    for (unsigned long long** a : {&batch_runs, &batch_inside, &run_off, &batch_tasks, &task_base})
        VGGP_CUDA(tmp.alloc(a, sizeof(unsigned long long) * (P + 1)));
    VGGP_CUDA(cudaMemsetAsync(batch_runs, 0, sizeof(unsigned long long) * (P + 1), st));
    VGGP_CUDA(cudaMemsetAsync(batch_inside, 0, sizeof(unsigned long long) * (P + 1), st));
    VGGP_CUDA(cudaMemsetAsync(seg_nruns, 0, sizeof(uint32_t) * (m + 1), st));
    k_mb_heads<KT><<<blocks_m, 256, 0, st>>>(keys, m, flags);
    VGGP_LAUNCH_CHECK();
    if (int rc = mb_exclusive_sum(flags, segid, m + 1, tmp, st)) return rc;
    k_mb_seg_starts<<<blocks_m, 256, 0, st>>>(flags, segid, m, seg_start);
    VGGP_LAUNCH_CHECK();
    k_mb_seg_runs<KT><<<blocks_m, 256, 0, st>>>(keys, seg_start, segid + m, (uint64_t)nck, ext ? ~0ull : (uint64_t)ncells, cap,
                                              seg_nruns, batch_runs, batch_inside);
    VGGP_LAUNCH_CHECK();
    if (int rc = mb_exclusive_sum(seg_nruns, run_base, m + 1, tmp, st)) return rc;
    uint32_t n_runs_h = 0;
    VGGP_CUDA(cudaMemcpyAsync(&n_runs_h, run_base + m, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    VGGP_CUDA(cudaStreamSynchronize(st));
    const i64 R = n_runs_h;
    // 3. the runs in cell order, then a stable sort by (batch, longest first)
    KT *run_key = nullptr, *run_key_s = nullptr;
    uint32_t *run_idx = nullptr, *run_sorted = nullptr, *run_cell = nullptr, *run_start = nullptr;
    int32_t* run_len = nullptr;
    VGGP_CUDA(tmp.alloc(&run_key, sizeof(KT) * R));
    VGGP_CUDA(tmp.alloc(&run_key_s, sizeof(KT) * R));
    for (uint32_t** a : {&run_idx, &run_sorted, &run_cell, &run_start}) VGGP_CUDA(tmp.alloc(a, sizeof(uint32_t) * R));
    VGGP_CUDA(tmp.alloc(&run_len, sizeof(int32_t) * R));
    if (R > 0) {
        k_mb_emit_runs<KT><<<(int)std::min<i64>((R + 255) / 256, (i64)p->sm_count * 16), 256, 0, st>>>(
            keys, seg_start, run_base, segid + m, R, (uint64_t)nck, cap, (uint32_t)B, run_key, run_idx, run_cell, run_len, run_start);
        VGGP_LAUNCH_CHECK();
        if (int rc = mb_sort_pairs<KT>(run_key, run_key_s, run_idx, run_sorted, R, mb_bits((uint64_t)P * (cap + 1ull) - 1), tmp, st))
            return rc;
    }
    // 4. tasks: per-batch run and task offsets, padded run length and streamed elements of every task, their scan
    if (int rc = mb_exclusive_sum(batch_runs, run_off, P + 1, tmp, st)) return rc;
    const int blocks_p = (int)std::min<i64>((P + 256) / 256, (i64)p->sm_count * 16);
    k_mb_batch_tasks<<<blocks_p, 256, 0, st>>>(batch_runs, P, batch_tasks);
    VGGP_LAUNCH_CHECK();
    if (int rc = mb_exclusive_sum(batch_tasks, task_base, P + 1, tmp, st)) return rc;
    const i64 T_ub = (R + 31) / 32 + P;                         // >= sum over batches of ceil(runs / 32)
    int32_t* task_R = nullptr;
    long long *task_elems = nullptr, *task_goff = nullptr, *d_tot = nullptr;
    VGGP_CUDA(tmp.alloc(&task_R, sizeof(int32_t) * T_ub));
    VGGP_CUDA(tmp.alloc(&task_elems, sizeof(long long) * (T_ub + 1)));
    VGGP_CUDA(tmp.alloc(&task_goff, sizeof(long long) * (T_ub + 1)));
    VGGP_CUDA(tmp.alloc(&d_tot, sizeof(long long) * 4 * P));
    k_mb_task_R<<<(int)std::min<i64>((T_ub + 256) / 256, (i64)p->sm_count * 16), 256, 0, st>>>(
        task_base, run_off, run_sorted, run_len, P, T_ub, D, task_R, task_elems);
    VGGP_LAUNCH_CHECK();
    if (int rc = mb_exclusive_sum(task_elems, task_goff, T_ub + 1, tmp, st)) return rc;
    k_mb_totals<<<blocks_p, 256, 0, st>>>(batch_runs, batch_inside, task_base, task_goff, P, d_tot);
    VGGP_LAUNCH_CHECK();
    // 5. the per-batch totals back to the host, which lays the buffer out: P headers, then each batch's sections
    std::vector<long long> h((size_t)(4 * P));
    VGGP_CUDA(cudaMemcpyAsync(h.data(), d_tot, sizeof(long long) * 4 * P, cudaMemcpyDeviceToHost, st));
    VGGP_CUDA(cudaStreamSynchronize(st));
    i64 off = (i64)BIN_HEADER_BYTES * P;
    e->n_tasks = e->n_runs = e->data_elems = 0;
    for (i64 b = 0; b < P; ++b) {
        int64_t* t = totals + MB_TOTALS * b;
        for (int j = 0; j < 4; ++j) t[j] = h[(size_t)(4 * b + j)];
        t[4] = off;
        off += bin_offsets(t[0], t[3], (int)sizeof(T)).bytes - BIN_HEADER_BYTES;
        e->n_tasks += t[0]; e->n_runs += t[1]; e->data_elems += t[3];
    }
    e->bytes = off;
    // what the pack needs lives on in the plan until vggp_epoch_bin_pack
    MbPending& q = p->mb;
    q.perm = perm; q.task_base = task_base; q.task_goff = task_goff; q.task_R = task_R; q.run_off = run_off;
    q.batch_runs = batch_runs; q.run_sorted = run_sorted; q.run_cell = run_cell; q.run_len = run_len; q.run_start = run_start;
    for (void* a : {(void*)perm, (void*)task_base, (void*)task_goff, (void*)task_R, (void*)run_off, (void*)batch_runs,
                    (void*)run_sorted, (void*)run_cell, (void*)run_len, (void*)run_start}) {
        tmp.release(a);
        q.keep.push_back(a);
    }
    q.desc = *e;
    q.active = true;
    return 0;
}

template <typename T, int D>
int epoch_prepare_impl(vggp_plan* p, const void* const* x, vggp_epoch_desc* e, int64_t* totals, cudaStream_t st) {
    const bool ext = p->family == VGGP_B0_GRIDDED || p->family == VGGP_SVGP_MARKOV;
    uint64_t ncells = 1;
    for (int d = 0; d < D; ++d) ncells *= (uint64_t)(ext ? p->K[d] + 1 : p->K[d] - 1);
    const uint64_t P = (uint64_t)e->n_batches, kmax = std::max<uint64_t>(P * (ext ? ncells : ncells + 1), P * ((uint64_t)e->run_cap + 1));
    if (kmax < 0xffffffffull) return epoch_prepare_kt<T, D, uint32_t>(p, x, e, totals, st);
    return epoch_prepare_kt<T, D, unsigned long long>(p, x, e, totals, st);
}

template <typename T, int D>
int epoch_pack_impl(vggp_plan* p, const int64_t* totals, const void* const* x, const void* y, void* binned, cudaStream_t st) {
    MbPending& q = p->mb;
    const vggp_epoch_desc& e = q.desc;
    const i64 P = e.n_batches, B = e.batch_size;
    unsigned char* buf = reinterpret_cast<unsigned char*>(binned);
    DevTemps tmp;
    VGGP_CUDA(cudaMemsetAsync(buf, 0, (size_t)BIN_HEADER_BYTES * P, st));
    std::vector<long long> sec((size_t)(6 * P));
    std::vector<vggp_binned_desc> bd((size_t)P);
    for (i64 b = 0; b < P; ++b) {
        int64_t view = 0;
        mb_batch_desc(&e, totals, b, &bd[(size_t)b], &view);
        const vggp_binned_desc& d = bd[(size_t)b];
        const i64 o[6] = {d.off_task_off, d.off_task_R, d.off_run_cell, d.off_run_n, d.off_run_start, d.off_data};
        for (int j = 0; j < 6; ++j) sec[(size_t)(6 * b + j)] = view + o[j];
    }
    long long* d_sec = nullptr;
    VGGP_CUDA(tmp.alloc(&d_sec, sizeof(long long) * 6 * P));
    VGGP_CUDA(cudaMemcpyAsync(d_sec, sec.data(), sizeof(long long) * 6 * P, cudaMemcpyHostToDevice, st));
    if (e.n_tasks > 0) {
        k_mb_tables<<<(int)std::min<i64>((32 * e.n_tasks + 255) / 256, (i64)p->sm_count * 16), 256, 0, st>>>(
            q.task_base, q.task_goff, q.task_R, q.run_off, q.batch_runs, q.run_sorted, q.run_cell, q.run_len, q.run_start, d_sec, P,
            buf);
        VGGP_LAUNCH_CHECK();
    }
    for (i64 b = 0; b < P; ++b) {
        const vggp_binned_desc& d = bd[(size_t)b];
        unsigned char* view = buf + (i64)BIN_HEADER_BYTES * b;
        const uint32_t* perm = q.perm + b * B;
        if (d.n_tasks > 0)
            if (int rc = launch_bin_gather<T, D>(p, x, y, perm, view, &d, d.n_tasks, st)) return rc;
        if (d.n_inside < B) {                 // B1: sum of y^2 of the batch's observations outside the mesh, in its own header
            const i64 nout = B - d.n_inside;
            const int blocks = (int)std::min<i64>((nout + 255) / 256, 148 * 4);
            k_bin_sum_y2<T><<<blocks, 256, 0, st>>>(reinterpret_cast<const T*>(y), perm, d.n_inside, B, reinterpret_cast<double*>(view));
            VGGP_LAUNCH_CHECK();
        }
    }
    VGGP_CUDA(cudaStreamSynchronize(st));
    p->mb.clear();
    return 0;
}

int epoch_prepare_dispatch(vggp_plan* p, const void* const* x, vggp_epoch_desc* e, int64_t* totals, cudaStream_t st) {
    VGGP_DISPATCH_TD(p, epoch_prepare_impl, p, x, e, totals, st);
}
int epoch_pack_dispatch(vggp_plan* p, const int64_t* totals, const void* const* x, const void* y, void* binned, cudaStream_t st) {
    VGGP_DISPATCH_TD(p, epoch_pack_impl, p, totals, x, y, binned, st);
}
// grow-only scratch (never inside a stream capture: cudaMalloc is not capturable)
int det_reserve(void** buf, size_t* have, size_t want, cudaStream_t st) {
    if (*have >= want) return 0;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusActive)
        return fail(VGGP_E_UNSUPPORTED, "deterministic mode: run one eager step before capturing a graph (its scratch is sized at first use)");
    VGGP_CUDA(cudaStreamSynchronize(st));
    if (*buf) cudaFree(*buf);
    *buf = nullptr; *have = 0;
    VGGP_CUDA(cudaMalloc(buf, want));
    *have = want;
    return 0;
}

// Deterministic variant of launch_obs_binned: records, then reductions in an order fixed by the binned layout (obs_binned.cuh).
template <typename T, int D>
int launch_obs_binned_det(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, void* gbuf, cudaStream_t st) {
    constexpr int R = BinRec<D>::v;
    const i64 nslots = (i64)desc->n_tasks * 32;
    i64 ncells = 1, nplanes = 0;
    for (int d = 0; d < D; ++d) { ncells *= p->K[d] - 1; nplanes += p->K[d] - 1; }
    if (nslots >= ((i64)1 << 31)) return fail(VGGP_E_UNSUPPORTED, "deterministic mode: too many runs");
    if (ncells >= ((i64)1 << 31)) return fail(VGGP_E_UNSUPPORTED, "deterministic mode: too many cells");
    int key_bits = 1;
    while (((i64)1 << key_bits) <= ncells) ++key_bits;          // keys 0 .. ncells (ncells = empty slot)
    size_t temp_bytes = 0;
    {
        const uint32_t* k = nullptr; uint32_t* ko = nullptr;
        VGGP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, k, ko, k, ko, (int)nslots, 0, key_bits, st));
    }
    auto al = [](size_t v) { return (v + 255) / 256 * 256; };
    const size_t o_rec = 0, o_k0 = al(o_rec + sizeof(T) * (size_t)nslots * R), o_k1 = al(o_k0 + 4 * (size_t)nslots),
                 o_i0 = al(o_k1 + 4 * (size_t)nslots), o_i1 = al(o_i0 + 4 * (size_t)nslots), o_cf = al(o_i1 + 4 * (size_t)nslots),
                 o_ce = al(o_cf + 4 * (size_t)ncells), o_S = al(o_ce + 4 * (size_t)ncells), o_E = al(o_S + sizeof(T) * 6 * (size_t)nplanes), o_tmp = al(o_E + sizeof(double) * DET_EBLOCKS),
                 total_bytes = al(o_tmp + temp_bytes);
    if (int rc = det_reserve(&p->det_buf, &p->det_bytes, total_bytes, st)) return rc;
    unsigned char* base = reinterpret_cast<unsigned char*>(p->det_buf);
    T* rec = reinterpret_cast<T*>(base + o_rec);
    uint32_t *k0 = reinterpret_cast<uint32_t*>(base + o_k0), *k1 = reinterpret_cast<uint32_t*>(base + o_k1),
             *i0 = reinterpret_cast<uint32_t*>(base + o_i0), *i1 = reinterpret_cast<uint32_t*>(base + o_i1),
             *cf = reinterpret_cast<uint32_t*>(base + o_cf), *ce = reinterpret_cast<uint32_t*>(base + o_ce);
    T* S = reinterpret_cast<T*>(base + o_S);
    double* E = reinterpret_cast<double*>(base + o_E);
    if (p->bin_blocks_per_sm[0] == 0) {
        int nb = 0;
        VGGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_obs_b1_binned<T, D>, BIN_THREADS, 0));
        p->bin_blocks_per_sm[0] = nb < 1 ? 1 : nb;
    }
    BinnedArgs<T, D> a;
    for (int d = 0; d < D; ++d) {
        a.geo.K[d] = p->K[d];
        a.geo.stride[d] = (int)p->stride[d];
        a.geo.band_off[d] = p->band_off[d];
        a.geo.tab_off[d] = p->tab_off[d];
        a.geo.knot_off[d] = p->knot_off[d];
    }
    a.buf = reinterpret_cast<const unsigned char*>(binned);
    a.off_task_off = desc->off_task_off; a.off_task_R = desc->off_task_R; a.off_run_cell = desc->off_run_cell;
    a.off_run_n = desc->off_run_n; a.off_data = desc->off_data;
    a.n_tasks = (int)desc->n_tasks;
    a.knots_byte_off = p->knots_byte_off;
    a.tables = p->tables;
    a.alpha = reinterpret_cast<const T*>(p->alphaT);
    T* gb = reinterpret_cast<T*>(gbuf);
    a.galpha = gb;
    a.gband = gb + p->M;
    a.n_rep = 1;
    a.band_rep_stride = 0;
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    a.gs = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(gbuf) + soff);
    a.n_real = (double)desc->n;
    a.counter = p->obs_counter + 1;
    i64 blocks = (desc->n_tasks + BIN_WARPS - 1) / BIN_WARPS;
    blocks = std::max<i64>(1, std::min<i64>(blocks, (i64)p->sm_count * p->bin_blocks_per_sm[0]));
    const uint32_t* run_cell = reinterpret_cast<const uint32_t*>(a.buf + desc->off_run_cell);
    k1_mark(p, 0, st);
    k_obs_b1_binned_det<T, D><<<(unsigned)blocks, BIN_THREADS, 0, st>>>(a, rec);
    k1_mark(p, 1, st);
    VGGP_LAUNCH_CHECK();
    if (nslots > 0) {
        k_det_keys<<<ceil_div(nslots, 256), 256, 0, st>>>(run_cell, (uint32_t)ncells, nslots, k0, i0);
        VGGP_LAUNCH_CHECK();
        VGGP_CUDA(cub::DeviceRadixSort::SortPairs(base + o_tmp, temp_bytes, (const uint32_t*)k0, k1, (const uint32_t*)i0, i1, (int)nslots, 0, key_bits, st));
        VGGP_CUDA(cudaMemsetAsync(cf, 0, (o_S - o_cf), st));
        k_det_mark<<<ceil_div(nslots, 256), 256, 0, st>>>(run_cell, i1, nslots, cf, ce);
        VGGP_LAUNCH_CHECK();
        DetIndex ix;
        ix.sorted_slot = i1; ix.cell_first = cf; ix.cell_end = ce;
        k_det_alpha<T, D><<<ceil_div(p->M, 256), 256, 0, st>>>(a.geo, ix, rec, a.galpha, p->M);
        VGGP_LAUNCH_CHECK();
        k_det_band<T, D><<<(unsigned)nplanes, 256, 0, st>>>(a.geo, ix, rec, S);
        VGGP_LAUNCH_CHECK();
    } else {
        // every observation outside the mesh: no run, no record; the band block and d alpha stay zero (gbuf was cleared)
        VGGP_CUDA(cudaMemsetAsync(S, 0, sizeof(T) * 6 * (size_t)nplanes, st));
    }
    k_det_escal<T, D><<<DET_EBLOCKS, 256, 0, st>>>(rec, run_cell, nslots, E);
    VGGP_LAUNCH_CHECK();
    k_det_final<T, D><<<1, 256, 0, st>>>(a.geo, S, E, a.gband, a.gs, a.buf, a.counter);
    VGGP_LAUNCH_CHECK();
    return 0;
}

int obs_binned_dispatch(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, void* gbuf, cudaStream_t st) {
    if (p->det) { VGGP_DISPATCH_TD(p, launch_obs_binned_det, p, desc, binned, gbuf, st); }
    VGGP_DISPATCH_TD(p, launch_obs_binned, p, desc, binned, gbuf, st);
}

// ---- B0 family, scan form (b0scan.cuh) -------------------------------------------------------------------
int b0scan_alloc(vggp_plan* p) {
    if (p->b0s_ready) return 0;
    if (p->family != VGGP_B0_GRIDDED || p->D > 2) return fail(VGGP_E_UNSUPPORTED, "the scan form is built for the B0 family, D <= 2");
    const size_t tsz = p->obs_dtype == VGGP_F32 ? 4 : 8;
    int rc;
    for (int d = 0; d < p->D; ++d) {
        const i64 em = (i64)(p->K[d] + 1) * (p->K[d] - 1);
        for (int k = 0; k < 4; ++k) {
            if ((rc = dev_alloc(p, &p->b0s_G[d][k], em))) return rc;
            if ((rc = dev_alloc(p, &p->b0s_V[d][k], em))) return rc;
        }
        if ((rc = dev_alloc(p, &p->b0s_eps[d], (i64)3 * (p->K[d] - 1)))) return rc;
        unsigned char* w = nullptr;
        if ((rc = dev_alloc(p, &w, (i64)(12 * (p->K[d] + 1) * tsz)))) return rc;
        p->b0s_W[d] = w;
    }
    const i64 E1 = p->K[0] + 1, M1 = p->K[0] - 1;
    unsigned char* tt = nullptr;
    if (p->D == 1) {
        if ((rc = dev_alloc(p, &tt, (i64)(3 * E1 * tsz)))) return rc;
    } else {
        const i64 E2 = p->K[1] + 1, M2 = p->K[1] - 1;
        for (int k = 0; k < 2; ++k) {
            if ((rc = dev_alloc(p, &p->b0s_U[k], M1 * E2))) return rc;
            if ((rc = dev_alloc(p, &p->b0s_B[k], E1 * M2))) return rc;
        }
        for (int k = 0; k < 4; ++k)
            if ((rc = dev_alloc(p, &p->b0s_TT[k], E1 * E2))) return rc;
        if ((rc = dev_alloc(p, &tt, (i64)(9 * E1 * E2 * tsz)))) return rc;
    }
    p->b0s_Tt = tt;
    // reverse side
    i64 EE = E1, emmax = 0, mmmax = 0, gw_elems = 0;
    for (int d = 0; d < p->D; ++d) {
        emmax = std::max<i64>(emmax, (i64)(p->K[d] + 1) * (p->K[d] - 1));
        mmmax = std::max<i64>(mmmax, (i64)(p->K[d] - 1) * (p->K[d] - 1));
        gw_elems += 12 * (p->K[d] + 1);
    }
    if (p->D == 2) EE = E1 * (p->K[1] + 1);
    const i64 nt = p->D == 1 ? 3 : 9;
    unsigned char* raw = nullptr;
    p->b0s_raw_bytes = (nt * EE + gw_elems) * (i64)tsz;
    if ((rc = dev_alloc(p, &raw, p->b0s_raw_bytes))) return rc;
    p->b0s_raw = raw;
    if ((rc = dev_alloc(p, &p->b0s_GTd, nt * EE))) return rc;
    for (int pr = 0; pr < 2 * p->D; ++pr) {
        for (int k = 0; k < 3; ++k)
            if ((rc = dev_alloc(p, &p->b0s_Sx[pr][k], emmax))) return rc;
        if ((rc = dev_alloc(p, &p->b0s_bMx[pr], mmmax))) return rc;
    }
    for (int k = 0; k < 2; ++k)
        if ((rc = dev_alloc(p, &p->b0s_Gam[k], emmax))) return rc;
    if (p->D == 2) {
        const i64 E2 = p->K[1] + 1, M2 = p->K[1] - 1;
        for (int k = 0; k < 3; ++k)
            if ((rc = dev_alloc(p, &p->b0s_H[k], M1 * E2))) return rc;
        for (int k = 0; k < 4; ++k) p->b0s_tan[0][k] = p->b0s_TT[k];
        for (int set = 1; set < 6; ++set)
            for (int k = 0; k < 4; ++k)
                if ((rc = dev_alloc(p, &p->b0s_tan[set][k], E1 * E2))) return rc;
        if ((rc = dev_alloc(p, &p->b0s_dA, M1 * M2))) return rc;
    }
    p->b0s_ready = true;
    return 0;
}

// The sweeps of the scan form run segmented (k_b0s_scan_seg / k_b0s_scan_adj_seg: S = ceil(M / 16) threads per fibre);
// 0 selects the one-thread-per-fibre kernels they were derived from (cross-check, vggp_debug_b0s_seg).
int g_b0s_seg = 1;
i64 g_host_chunk = (i64)1 << 23;      // observations per PCIe chunk of vggp_elbo_host (vggp_debug_host_chunk)

struct B0sSegGeom { int S, F, f_fast; unsigned blocks; size_t smem; };
inline B0sSegGeom b0s_seg_geom(int M, i64 n_fibres, i64 n_lo, i64 lo_stride, bool tan) {
    B0sSegGeom g;
    g.S = (M + B0S_SEG - 1) / B0S_SEG;
    if (g.S < 1) g.S = 1;
    g.F = B0S_SEG_THREADS / g.S;
    g.f_fast = (n_lo > 1 && lo_stride == 1) ? 1 : 0;      // neighbouring fibres contiguous in memory
    g.blocks = (unsigned)((n_fibres + g.F - 1) / g.F);
    g.smem = b0s_seg_smem_bytes(M, tan);
    return g;
}

// Independent sweeps are queued and launched together (blockIdx.y = entry, up to B0S_MAX_BATCH per launch): forward / tangent
// transforms (k_b0s_scan_seg) and adjoint transforms (k_b0s_scan_adj_seg).  flush() is called wherever the next step reads
// what the queued sweeps write.
struct B0sBatcher {
    cudaStream_t st;
    std::vector<B0sScanArgs> scans;
    std::vector<B0sAdjArgs> adjs;
    explicit B0sBatcher(cudaStream_t s) : st(s) {}

    int flush_scans() {
        size_t i = 0;
        while (i < scans.size()) {
            const B0sScanArgs& a0 = scans[i];
            const bool tan = a0.tanL != nullptr;
            if (!g_b0s_seg || (a0.M + B0S_SEG - 1) / B0S_SEG > B0S_SEG_THREADS) {     // one-thread-per-fibre kernel, one at a time
                if (a0.n_fibres > 0 && a0.M > 0) {
                    k_b0s_scan<<<ceil_div(a0.n_fibres, 128), 128, 0, st>>>(a0);
                    VGGP_LAUNCH_CHECK();
                }
                ++i;
                continue;
            }
            B0sScanBatch bt;
            memset(&bt, 0, sizeof(bt));
            int n = 0;
            unsigned gx = 1;
            size_t smem = 0;
            while (i < scans.size() && n < B0S_MAX_BATCH && (scans[i].tanL != nullptr) == tan
                   && (scans[i].M + B0S_SEG - 1) / B0S_SEG <= B0S_SEG_THREADS) {
                const B0sScanArgs& a = scans[i];
                ++i;
                if (a.n_fibres <= 0 || a.M <= 0) continue;
                const B0sSegGeom g = b0s_seg_geom(a.M, a.n_fibres, a.n_lo, a.s_lo, tan);
                bt.a[n] = a;
                bt.g[n].S = g.S; bt.g[n].F = g.F; bt.g[n].f_fast = g.f_fast; bt.g[n].blocks = (int)g.blocks;
                gx = std::max(gx, g.blocks);
                smem = std::max(smem, g.smem);
                ++n;
            }
            if (n == 0) continue;
            if (tan) {
                if (int rc = raise_dyn_smem(k_b0s_scan_seg<true>, smem)) return rc;
                k_b0s_scan_seg<true><<<dim3(gx, n), B0S_SEG_THREADS, smem, st>>>(bt);
            } else {
                if (int rc = raise_dyn_smem(k_b0s_scan_seg<false>, smem)) return rc;
                k_b0s_scan_seg<false><<<dim3(gx, n), B0S_SEG_THREADS, smem, st>>>(bt);
            }
            VGGP_LAUNCH_CHECK();
        }
        scans.clear();
        return 0;
    }

    int flush_adjs() {
        size_t i = 0;
        while (i < adjs.size()) {
            const B0sAdjArgs& a0 = adjs[i];
            if (!g_b0s_seg || (a0.M + B0S_SEG - 1) / B0S_SEG > B0S_SEG_THREADS) {
                if (a0.n_fibres > 0 && a0.M > 0) {
                    k_b0s_scan_adj<<<ceil_div(a0.n_fibres, 128), 128, 0, st>>>(a0);
                    VGGP_LAUNCH_CHECK();
                }
                ++i;
                continue;
            }
            B0sAdjBatch bt;
            memset(&bt, 0, sizeof(bt));
            int n = 0;
            unsigned gx = 1;
            size_t smem = 0;
            while (i < adjs.size() && n < B0S_MAX_BATCH && (adjs[i].M + B0S_SEG - 1) / B0S_SEG <= B0S_SEG_THREADS) {
                const B0sAdjArgs& a = adjs[i];
                ++i;
                if (a.n_fibres <= 0 || a.M <= 0) continue;
                const B0sSegGeom g = b0s_seg_geom(a.M, a.n_fibres, a.n_lo, a.g_lo, false);
                bt.a[n] = a;
                bt.g[n].S = g.S; bt.g[n].F = g.F; bt.g[n].f_fast = g.f_fast; bt.g[n].blocks = (int)g.blocks;
                gx = std::max(gx, g.blocks);
                smem = std::max(smem, g.smem);
                ++n;
            }
            if (n == 0) continue;
            if (int rc = raise_dyn_smem(k_b0s_scan_adj_seg, smem)) return rc;
            k_b0s_scan_adj_seg<<<dim3(gx, n), B0S_SEG_THREADS, smem, st>>>(bt);
            VGGP_LAUNCH_CHECK();
        }
        adjs.clear();
        return 0;
    }

    int flush() {
        if (int rc = flush_scans()) return rc;
        return flush_adjs();
    }
};

// dstL = G^L src, dstR = G^R src along one mode (k_b0s_scan): n_hi x n_lo fibres of M elements -> M + 2 entries
void b0s_scan(B0sBatcher& q, const double* eps, int M, i64 n_hi, i64 n_lo, const double* src, i64 s_hi, i64 s_lo, i64 s_mode,
              double* dstL, double* dstR, i64 d_hi, i64 d_lo, i64 d_mode) {
    B0sScanArgs a;
    a.src = src; a.dstL = dstL; a.dstR = dstR; a.tanL = nullptr; a.tanR = nullptr; a.eps = eps; a.M = M;
    a.n_fibres = n_hi * n_lo; a.n_lo = n_lo;
    a.s_hi = s_hi; a.s_lo = s_lo; a.s_mode = s_mode;
    a.d_hi = d_hi; a.d_lo = d_lo; a.d_mode = d_mode;
    q.scans.push_back(a);
}

// Per-cell tables from the state of the last grid forward (alpha, P_d, Q_d, theta).  Every product with G^L / G^R is a
// first-order recurrence along a mode (k_b0s_scan, O(M) per mode); the dense G matrices are still written because the
// quadratic-form tables take row dots with them and the adjoint stage contracts with their lengthscale derivatives.
template <typename T>
int b0scan_tables(vggp_plan* p, cudaStream_t st) {
    int rc = b0scan_alloc(p);
    if (rc) return rc;
    const int D = p->D;
    B0sBatcher q(st);
    B0sGArgs ga;
    B0sEpsArgs ea;
    int emax = 0, mmax = 0;
    for (int d = 0; d < D; ++d) {
        ga.knots[d] = p->d_knots[d];
        ga.K[d] = p->K[d];
        ga.GL[d] = p->b0s_G[d][0]; ga.GR[d] = p->b0s_G[d][1]; ga.dGL[d] = p->b0s_G[d][2]; ga.dGR[d] = p->b0s_G[d][3];
        ea.knots[d] = p->d_knots[d];
        ea.K[d] = p->K[d];
        ea.out[d] = p->b0s_eps[d];
        emax = std::max(emax, (p->K[d] + 1) * (p->K[d] - 1));
        mmax = std::max(mmax, p->K[d] - 1);
    }
    ga.theta = p->theta_dev;
    ea.theta = p->theta_dev;
    k_b0s_G<<<dim3(ceil_div(emax, 256), D), 256, 0, st>>>(ga);
    VGGP_LAUNCH_CHECK();
    k_b0s_eps<<<dim3(ceil_div(mmax, 256), D), 256, 0, st>>>(ea);
    VGGP_LAUNCH_CHECK();
    B0sWArgs<T> wa;
    int kmax = 0;
    for (int d = 0; d < D; ++d) {
        const int M = p->K[d] - 1, E = p->K[d] + 1;
        const double* mats[2] = {p->g.P[d], p->g.Q[d]};
        for (int mat = 0; mat < 2; ++mat)       // V^x = G^x Mat (E x M): transform along the row index, fibres = columns
            b0s_scan(q, p->b0s_eps[d], M, 1, M, mats[mat], 0, 1, M, p->b0s_V[d][2 * mat], p->b0s_V[d][2 * mat + 1], 0, 1, M);
        wa.K[d] = p->K[d];
        wa.GL[d] = p->b0s_G[d][0]; wa.GR[d] = p->b0s_G[d][1];
        for (int k = 0; k < 4; ++k) wa.V[d][k] = p->b0s_V[d][k];
        wa.Mat[d][0] = p->g.P[d]; wa.Mat[d][1] = p->g.Q[d];
        wa.W[d] = reinterpret_cast<T*>(p->b0s_W[d]);
        kmax = std::max(kmax, E);
    }
    if ((rc = q.flush())) return rc;            // the 2 D transforms of P_d, Q_d: one launch
    k_b0s_W<T><<<dim3(ceil_div(kmax, 8), D), 256, 0, st>>>(wa);
    VGGP_LAUNCH_CHECK();
    const int E1 = p->K[0] + 1, M1 = p->K[0] - 1;
    if (D == 1) {
        k_b0s_T1<T><<<ceil_div(E1, 8), 256, 0, st>>>(p->K[0], p->b0s_G[0][0], p->b0s_G[0][1], p->alpha, reinterpret_cast<T*>(p->b0s_Tt));
        VGGP_LAUNCH_CHECK();
        return 0;
    }
    const int E2 = p->K[1] + 1, M2 = p->K[1] - 1;
    // U^y = A G2^y^T (M1 x E2): transform along dimension 2, fibres = rows of A
    b0s_scan(q, p->b0s_eps[1], M2, M1, 1, p->alpha, M2, 0, 1, p->b0s_U[0], p->b0s_U[1], E2, 0, 1);
    // B^x = G1^x A (E1 x M2): transform along dimension 1, fibres = columns of A
    b0s_scan(q, p->b0s_eps[0], M1, 1, M2, p->alpha, 0, 1, M2, p->b0s_B[0], p->b0s_B[1], 0, 1, M2);
    if ((rc = q.flush())) return rc;
    // TT[2x+y] = G1^x U^y (E1 x E2): transform along dimension 1 of U^y, fibres = its columns
    for (int y = 0; y < 2; ++y)
        b0s_scan(q, p->b0s_eps[0], M1, 1, E2, p->b0s_U[y], 0, 1, E2, p->b0s_TT[y], p->b0s_TT[2 + y], 0, 1, E2);
    if ((rc = q.flush())) return rc;
    B0sT2Args<T> ta;
    ta.E1 = E1; ta.E2 = E2; ta.M1 = M1; ta.M2 = M2;
    for (int k = 0; k < 4; ++k) ta.TT[k] = p->b0s_TT[k];
    for (int k = 0; k < 2; ++k) { ta.B[k] = p->b0s_B[k]; ta.U[k] = p->b0s_U[k]; }
    ta.A = p->alpha;
    ta.Tt = reinterpret_cast<T*>(p->b0s_Tt);
    k_b0s_T2<T><<<ceil_div((i64)E1 * E2, 256), 256, 0, st>>>(ta);
    VGGP_LAUNCH_CHECK();
    return 0;
}

template <typename T, int D>
void b0scan_point_tables(const vggp_plan* p, B0sPointTables<T, D>& t) {
    for (int d = 0; d < D; ++d) {
        t.mesh[d] = p->mesh[d];
        t.E[d] = p->K[d] + 1;
        t.W[d] = reinterpret_cast<const T*>(p->b0s_W[d]);
    }
    t.Tt = reinterpret_cast<const T*>(p->b0s_Tt);
    t.theta = p->theta_dev;
}

template <typename T, int D>
int launch_predict_b0s(vggp_plan* p, const void* const* x, i64 n, void* mean, void* var, cudaStream_t st) {
    int rc = b0scan_tables<T>(p, st);
    if (rc) return rc;
    B0sPredictArgs<T, D> a;
    b0scan_point_tables<T, D>(p, a.tab);
    for (int d = 0; d < D; ++d) a.x[d] = reinterpret_cast<const T*>(x[d]);
    a.n = n;
    a.mean = reinterpret_cast<T*>(mean);
    a.var = reinterpret_cast<T*>(var);
    const int blocks = (int)std::min<i64>((n + 255) / 256, (i64)p->sm_count * 8);
    k_predict_b0s<T, D><<<blocks, 256, 0, st>>>(a);
    VGGP_LAUNCH_CHECK();
    return 0;
}

void b0s_scan_tan(B0sBatcher& q, const double* eps, int M, i64 n_hi, i64 n_lo, const double* src, i64 s_hi, i64 s_lo, i64 s_mode,
                  double* dstL, double* dstR, double* tanL, double* tanR, i64 d_hi, i64 d_lo, i64 d_mode) {
    B0sScanArgs a;
    a.src = src; a.dstL = dstL; a.dstR = dstR; a.tanL = tanL; a.tanR = tanR; a.eps = eps; a.M = M;
    a.n_fibres = n_hi * n_lo; a.n_lo = n_lo;
    a.s_hi = s_hi; a.s_lo = s_lo; a.s_mode = s_mode;
    a.d_hi = d_hi; a.d_lo = d_lo; a.d_mode = d_mode;
    q.scans.push_back(a);
}

void b0s_scan_adj(B0sBatcher& q, const double* eps, int M, i64 n_hi, i64 n_lo, const double* gL, const double* gC, const double* gR,
                  i64 g_hi, i64 g_lo, i64 g_mode, double* dv, i64 v_hi, i64 v_lo, i64 v_mode) {
    B0sAdjArgs a;
    a.gL = gL; a.gC = gC; a.gR = gR; a.dv = dv; a.eps = eps; a.M = M;
    a.n_fibres = n_hi * n_lo; a.n_lo = n_lo;
    a.g_hi = g_hi; a.g_lo = g_lo; a.g_mode = g_mode;
    a.v_hi = v_hi; a.v_lo = v_lo; a.v_mode = v_mode;
    q.adjs.push_back(a);
}

// out[e] += <x_e, y_e> for up to B0S_MAX_BATCH pairs of n elements each, one launch
int b0s_dots(cudaStream_t st, const std::vector<const double*>& x, const std::vector<const double*>& y,
             const std::vector<double*>& out, i64 n) {
    size_t i = 0;
    while (i < x.size()) {
        B0sDotBatch b;
        memset(&b, 0, sizeof(b));
        int k = 0;
        for (; i < x.size() && k < B0S_MAX_BATCH; ++i, ++k) { b.x[k] = x[i]; b.y[k] = y[i]; b.out[k] = out[i]; }
        b.n = n;
        k_b0s_dot_batch<<<dim3(std::min<int>(ceil_div(n, 256), 64), k), 256, 0, st>>>(b);
        VGGP_LAUNCH_CHECK();
    }
    return 0;
}

// Adjoint of the table construction: raw per-cell sums of k_obs_b0s -> d alpha, [bP | bQ] and the table part of G_l, in
// the gbuf layout of the B0 family (what k_obs_b0 would have written).  Like the forward, every product with G^L / G^R or
// their lengthscale derivatives is a first-order recurrence along a mode (adjoint and tangent sweeps): O(M) per mode.
template <typename T, int D>
int b0scan_adjoint(vggp_plan* p, void* gbuf, cudaStream_t st) {
    int rc;
    const i64 E1 = p->K[0] + 1, M1 = p->K[0] - 1;
    const i64 E2 = D == 2 ? p->K[1] + 1 : 1, M2 = D == 2 ? p->K[1] - 1 : 1;
    const i64 EE = E1 * E2, NT = D == 1 ? 3 : 9;
    const T* rawT = reinterpret_cast<const T*>(p->b0s_raw);
    const T* GW[2] = {rawT + NT * EE, rawT + NT * EE + 12 * E1};
    double* GTd = p->b0s_GTd;
    k_b0s_to_double<T><<<ceil_div(NT * EE, 256), 256, 0, st>>>(rawT, GTd, NT * EE);
    VGGP_LAUNCH_CHECK();
    T* gb = reinterpret_cast<T*>(gbuf);
    T* galpha = gb;
    T* gfac = gb + p->M;
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    double* gs = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(gbuf) + soff);
    auto GT = [&](int X, int Y) { return GTd + (i64)(3 * X + Y) * EE; };
    B0sBatcher q(st);
    // the S^X = diag(gw^{X.}) G^. products of the four (dimension, matrix) pairs first: their adjoint sweeps then share launches
    // with the sweeps of d alpha
    int pair = 0;
    for (int d = 0; d < D; ++d) {
        const int K = p->K[d];
        const i64 M = K - 1, E = K + 1;
        for (int mat = 0; mat < 2; ++mat, ++pair) {
            k_b0s_S<T><<<ceil_div(E * M, 256), 256, 0, st>>>(K, p->b0s_G[d][0], p->b0s_G[d][1], GW[d] + (i64)mat * 6 * E,
                                                             p->b0s_Sx[pair][0], p->b0s_Sx[pair][1], p->b0s_Sx[pair][2]);
            VGGP_LAUNCH_CHECK();
        }
    }
    // ---- d alpha = sum_XY G1^X^T GT^{XY} G2^Y ----
    if (D == 1) {
        k_b0s_galpha1<T><<<ceil_div(M1, 256), 256, 0, st>>>(p->K[0], p->b0s_G[0][0], p->b0s_G[0][1], GTd, galpha);
        VGGP_LAUNCH_CHECK();
    } else {
        for (int Y = 0; Y < 3; ++Y)          // H^Y = sum_X G1^X^T GT^{XY}  (M1 x E2): adjoint sweep along dimension 1, fibres = columns
            b0s_scan_adj(q, p->b0s_eps[0], (int)M1, 1, E2, GT(B0S_L, Y), GT(B0S_C, Y), GT(B0S_R, Y), 0, 1, E2, p->b0s_H[Y], 0, 1, E2);
    }
    // ---- [bP | bQ]_d = sum_XY G^X^T diag(gw^{XY}) G^Y = sum_X G^X^T S^X ----
    pair = 0;
    for (int d = 0; d < D; ++d) {
        const i64 M = p->K[d] - 1;
        for (int mat = 0; mat < 2; ++mat, ++pair) {
            if (D == 2 && pair == 3) {        // H^Y are complete after the first launch: d alpha = sum_Y H^Y G2^Y rides with the last pair
                if ((rc = q.flush())) return rc;
                b0s_scan_adj(q, p->b0s_eps[1], (int)M2, M1, 1, p->b0s_H[B0S_L], p->b0s_H[B0S_C], p->b0s_H[B0S_R], E2, 0, 1, p->b0s_dA, M2, 0, 1);
            }
            b0s_scan_adj(q, p->b0s_eps[d], (int)M, 1, M, p->b0s_Sx[pair][B0S_L], p->b0s_Sx[pair][B0S_C], p->b0s_Sx[pair][B0S_R], 0, 1, M,
                         p->b0s_bMx[pair], 0, 1, M);
        }
    }
    if ((rc = q.flush())) return rc;
    if (D == 2) {
        k_b0s_from_double<T><<<ceil_div(M1 * M2, 256), 256, 0, st>>>(p->b0s_dA, galpha, M1 * M2);
        VGGP_LAUNCH_CHECK();
    }
    pair = 0;
    for (int d = 0; d < D; ++d) {
        const i64 M = p->K[d] - 1;
        for (int mat = 0; mat < 2; ++mat, ++pair) {
            k_b0s_from_double<T><<<ceil_div(M * M, 256), 256, 0, st>>>(p->b0s_bMx[pair], gfac + p->gfac_off[d] + (i64)mat * M * M, M * M);
            VGGP_LAUNCH_CHECK();
        }
    }
    // ---- table part of G_l[d] = <GT, dT / dl_d> + <GW_d, dW_d / dl_d> ----
    for (int d = 0; d < D; ++d) {
        const int K = p->K[d];
        k_b0s_gl_rows<T><<<ceil_div(K + 1, 8), 256, 0, st>>>(K, GW[d], p->b0s_V[d][0], p->b0s_V[d][1], p->b0s_V[d][2], p->b0s_V[d][3],
                                                             p->g.P[d], p->g.Q[d], p->b0s_G[d][2], p->b0s_G[d][3],
                                                             D == 1 ? GTd : nullptr, D == 1 ? p->alpha : nullptr, gs + 3 + d);
        VGGP_LAUNCH_CHECK();
    }
    if (D == 2) {
        // six tangent sweeps, each into its own scratch set [transform L | transform R | tangent L | tangent R] (the forward's corner
        // products in TT[] are no longer needed: they are set 0), one launch; then the twelve inner products in two launches
        std::vector<const double*> dx, dy;
        std::vector<double*> dout;
        // l_1: dT^{XY} / dl_1 = (dG1^X / dl_1) U^Y, X in {L, R}: tangent sweep along dimension 1 of U^Y (U^C = A in columns 1..M2)
        for (int Y = 0; Y < 3; ++Y) {
            double* const* sc = p->b0s_tan[Y];
            if (Y == B0S_C) {
                VGGP_CUDA(cudaMemsetAsync(sc[2], 0, sizeof(double) * EE, st));
                VGGP_CUDA(cudaMemsetAsync(sc[3], 0, sizeof(double) * EE, st));
                b0s_scan_tan(q, p->b0s_eps[0], (int)M1, 1, M2, p->alpha, 0, 1, M2, sc[0] + 1, sc[1] + 1, sc[2] + 1, sc[3] + 1, 0, 1, E2);
            } else {
                b0s_scan_tan(q, p->b0s_eps[0], (int)M1, 1, E2, p->b0s_U[Y == B0S_L ? 0 : 1], 0, 1, E2, sc[0], sc[1], sc[2], sc[3], 0, 1, E2);
            }
            dx.push_back(GT(B0S_L, Y)); dy.push_back(sc[2]); dout.push_back(gs + 3);
            dx.push_back(GT(B0S_R, Y)); dy.push_back(sc[3]); dout.push_back(gs + 3);
        }
        // l_2: dT^{XY} / dl_2 = B^X (dG2^Y / dl_2)^T, Y in {L, R}: tangent sweep along dimension 2 of B^X (B^C = A in rows 1..M1)
        for (int X = 0; X < 3; ++X) {
            double* const* sc = p->b0s_tan[3 + X];
            if (X == B0S_C) {
                VGGP_CUDA(cudaMemsetAsync(sc[2], 0, sizeof(double) * EE, st));
                VGGP_CUDA(cudaMemsetAsync(sc[3], 0, sizeof(double) * EE, st));
                b0s_scan_tan(q, p->b0s_eps[1], (int)M2, M1, 1, p->alpha, M2, 0, 1, sc[0] + E2, sc[1] + E2, sc[2] + E2, sc[3] + E2, E2, 0, 1);
            } else {
                b0s_scan_tan(q, p->b0s_eps[1], (int)M2, E1, 1, p->b0s_B[X == B0S_L ? 0 : 1], M2, 0, 1, sc[0], sc[1], sc[2], sc[3], E2, 0, 1);
            }
            dx.push_back(GT(X, B0S_L)); dy.push_back(sc[2]); dout.push_back(gs + 4);
            dx.push_back(GT(X, B0S_R)); dy.push_back(sc[3]); dout.push_back(gs + 4);
        }
        if ((rc = q.flush())) return rc;
        if ((rc = b0s_dots(st, dx, dy, dout, EE))) return rc;
    }
    return 0;
}

template <typename T, int D>
int launch_obs_b0s(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, void* gbuf, cudaStream_t st) {
    int rc = b0scan_tables<T>(p, st);
    if (rc) return rc;
    VGGP_CUDA(cudaMemsetAsync(p->b0s_raw, 0, (size_t)p->b0s_raw_bytes, st));
    B0sObsArgs<T, D> a;
    b0scan_point_tables<T, D>(p, a.tab);
    a.buf = reinterpret_cast<const unsigned char*>(binned);
    a.off_task_off = desc->off_task_off; a.off_task_R = desc->off_task_R; a.off_run_cell = desc->off_run_cell;
    a.off_run_n = desc->off_run_n; a.off_data = desc->off_data;
    a.n_tasks = (int)desc->n_tasks;
    const i64 E1 = p->K[0] + 1, EE = D == 1 ? E1 : E1 * (p->K[D - 1] + 1), NT = D == 1 ? 3 : 9;
    T* rawT = reinterpret_cast<T*>(p->b0s_raw);
    a.GT = rawT;
    a.GW[0] = rawT + NT * EE;
    if (D == 2) a.GW[D - 1] = rawT + NT * EE + 12 * E1;
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    a.gs = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(gbuf) + soff);
    a.n_real = (double)desc->n;
    a.counter = p->obs_counter;
    VGGP_CUDA(cudaMemsetAsync(p->obs_counter, 0, sizeof(unsigned int), st));
    i64 blocks = (desc->n_tasks + (B0S_THREADS / 32) - 1) / (B0S_THREADS / 32);
    int per_sm = 0;                             // as many persistent CTAs as fit (167 registers: 3 per SM; the first version launched 2)
    VGGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_obs_b0s<T, D>, B0S_THREADS, 0));
    blocks = std::max<i64>(1, std::min<i64>(blocks, (i64)p->sm_count * std::max(1, per_sm)));
    k1_mark(p, 0, st);
    k_obs_b0s<T, D><<<(unsigned)blocks, B0S_THREADS, 0, st>>>(a);
    k1_mark(p, 1, st);
    VGGP_LAUNCH_CHECK();
    return b0scan_adjoint<T, D>(p, gbuf, st);
}

int obs_b0s_dispatch(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, void* gbuf, cudaStream_t st) {
    if (p->obs_dtype == VGGP_F32)
        return p->D == 1 ? launch_obs_b0s<float, 1>(p, desc, binned, gbuf, st) : launch_obs_b0s<float, 2>(p, desc, binned, gbuf, st);
    return p->D == 1 ? launch_obs_b0s<double, 1>(p, desc, binned, gbuf, st) : launch_obs_b0s<double, 2>(p, desc, binned, gbuf, st);
}

int predict_b0s_dispatch(vggp_plan* p, const void* const* x, i64 n, void* mean, void* var, cudaStream_t st) {
    if (p->D > 2) return fail(VGGP_E_UNSUPPORTED, "the B0 (cell-integrated) family is built for D <= 2, as in the reference");
    if (p->obs_dtype == VGGP_F32)
        return p->D == 1 ? launch_predict_b0s<float, 1>(p, x, n, mean, var, st) : launch_predict_b0s<float, 2>(p, x, n, mean, var, st);
    return p->D == 1 ? launch_predict_b0s<double, 1>(p, x, n, mean, var, st) : launch_predict_b0s<double, 2>(p, x, n, mean, var, st);
}

}  // namespace

// =========================================================================================================
template <typename T, int D>
int launch_tracks(void* const* x, void* y, i64 lo, i64 hi, i64 n_total, i64 seed, int passes, double gradient, cudaStream_t st) {
    TrackArgs<T, D> a;
    for (int d = 0; d < D; ++d) a.x[d] = reinterpret_cast<T*>(x[d]);
    a.y = reinterpret_cast<T*>(y);
    a.lo = lo; a.hi = hi; a.n_total = n_total; a.seed = seed; a.passes = passes; a.gradient = gradient;
    const int blocks = (int)std::min<i64>((hi - lo + 255) / 256, 148 * 16);
    k_generate_tracks<T, D><<<blocks, 256, 0, st>>>(a);
    VGGP_LAUNCH_CHECK();
    return 0;
}

// ---- product-grid SVGP, Markov form (svgpm.cuh) -------------------------------------------------------------
template <int D>
SvgpmGeom<D> svgpm_geom(const vggp_plan* p) {
    SvgpmGeom<D> g;
    for (int d = 0; d < D; ++d) {
        g.M[d] = p->n[d];
        g.stride[d] = (int)p->stride[d];
        g.band_off[d] = p->band_off[d];
        g.tab_off[d] = p->svm_tab_off[d];
    }
    return g;
}

SvgpmBwd svgpm_bwd(const vggp_plan* p) {
    SvgpmBwd g;
    memset(&g, 0, sizeof(g));
    g.D = p->D;
    g.Mtot = p->M;
    for (int d = 0; d < p->D; ++d) {
        g.M[d] = p->n[d];
        g.stride[d] = (int)p->stride[d];
        g.band_off[d] = p->band_off[d];
        g.Loff[d] = p->g.Loff[d];
        g.W[d] = p->svm_W[d];
    }
    g.sc = p->svm_sc;
    return g;
}

// K_d band and K_d^-1 band in closed form, S_d band from tril(L_d), per-cell tables, log-dets and traces, m in the
// observation dtype.  Four launches, no allocation, no synchronisation.
int svgpm_forward(vggp_plan* p, const double* theta, const double* m, const double* L, cudaStream_t st) {
    const int D = p->D;
    VGGP_CUDA(cudaMemsetAsync(p->svm_sc, 0, sizeof(double) * SVS_MKM, st));
    VGGP_CUDA(cudaMemsetAsync(p->g.info, 0, sizeof(int), st));
    VGGP_CUDA(cudaMemcpyAsync(p->theta_dev, theta, sizeof(double) * (2 * D + 1), cudaMemcpyDeviceToDevice, st));
    SvgpmGrid g;
    memset(&g, 0, sizeof(g));
    g.D = D;
    for (int d = 0; d < D; ++d) {
        g.M[d] = p->n[d];
        g.z[d] = p->d_knots[d];
        g.Loff[d] = p->g.Loff[d];
        g.W[d] = p->svm_W[d];
        g.tab_off[d] = p->svm_tab_off[d];
    }
    g.tab = p->svm_tab;
    g.sc = p->svm_sc;
    g.info = p->g.info;
    const dim3 grid(ceil_div(p->nmax, 8), D);
    const int cblocks = (int)std::min<i64>((p->M + 255) / 256, 148 * 4);
    if (p->obs_dtype == VGGP_F32) {
        k_svgpm_fwd<float><<<grid, 256, 0, st>>>(g, theta, L);
        VGGP_LAUNCH_CHECK();
        k_b0s_from_double<float><<<cblocks, 256, 0, st>>>(m, reinterpret_cast<float*>(p->alphaT), p->M);
    } else {
        k_svgpm_fwd<double><<<grid, 256, 0, st>>>(g, theta, L);
        VGGP_LAUNCH_CHECK();
        k_b0s_from_double<double><<<cblocks, 256, 0, st>>>(m, reinterpret_cast<double*>(p->alphaT), p->M);
    }
    VGGP_LAUNCH_CHECK();
    return 0;
}

template <typename T, int D>
int svgpm_backward_impl(vggp_plan* p, const double* theta, const double* m, const double* L, const void* gbuf,
                        double ell_scale, double* out, double* dtheta, double* dm, double* dL, cudaStream_t st) {
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    const double* gs = reinterpret_cast<const double*>(reinterpret_cast<const unsigned char*>(gbuf) + soff);
    const T* gm = reinterpret_cast<const T*>(gbuf);
    const T* gband = gm + p->M;
    const SvgpmBwd g = svgpm_bwd(p);
    VGGP_CUDA(cudaMemsetAsync(p->svm_sc + SVS_MKM, 0, sizeof(double) * (SVS_COUNT - SVS_MKM), st));
    const int mblocks = (int)std::min<i64>((p->M + 255) / 256, (i64)p->sm_count * 4);
    k_svgpm_dm<T, D><<<mblocks, 256, 0, st>>>(g, gm, m, theta, ell_scale, dm);
    VGGP_LAUNCH_CHECK();
    k_svgpm_dL<T><<<dim3(ceil_div((i64)p->nmax * p->nmax, 256), D), 256, 0, st>>>(g, gband, L, theta, ell_scale, dL);
    VGGP_LAUNCH_CHECK();
    k_svgpm_theta<T><<<1, 256, 0, st>>>(g, gband, gs, theta, ell_scale, out, dtheta);
    VGGP_LAUNCH_CHECK();
    return 0;
}
int svgpm_backward(vggp_plan* p, const double* theta, const double* m, const double* L, const void* gbuf, double ell_scale,
                   double* out, double* dtheta, double* dm, double* dL, cudaStream_t st) {
    VGGP_DISPATCH_TD(p, svgpm_backward_impl, p, theta, m, L, gbuf, ell_scale, out, dtheta, dm, dL, st);
}

template <typename T, int D>
int launch_obs_svgpm(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, void* gbuf, cudaStream_t st) {
    if (p->svm_blocks_per_sm == 0) {
        int nb = 0;
        VGGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_obs_svgpm_binned<T, D>, BIN_THREADS, 0));
        p->svm_blocks_per_sm = nb < 1 ? 1 : nb;
    }
    SvgpmArgs<T, D> a;
    memset(&a, 0, sizeof(a));
    a.bin.buf = reinterpret_cast<const unsigned char*>(binned);
    a.bin.off_task_off = desc->off_task_off; a.bin.off_task_R = desc->off_task_R; a.bin.off_run_cell = desc->off_run_cell;
    a.bin.off_run_n = desc->off_run_n; a.bin.off_data = desc->off_data;
    a.bin.n_tasks = (int)desc->n_tasks;
    T* gb = reinterpret_cast<T*>(gbuf);
    a.bin.galpha = gb;
    a.bin.gband = reinterpret_cast<T*>(p->band_rep);
    a.bin.n_rep = BAND_REPLICAS;
    a.bin.band_rep_stride = p->band_total;
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    a.bin.gs = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(gbuf) + soff);
    a.bin.n_real = (double)desc->n;
    a.bin.counter = p->obs_counter + 1;          // reset by k_band_reduce after every launch
    a.geo = svgpm_geom<D>(p);
    a.tab = reinterpret_cast<const T*>(p->svm_tab);
    a.m = reinterpret_cast<const T*>(p->alphaT);
    a.theta = p->theta_dev;
    i64 blocks = (desc->n_tasks + BIN_WARPS - 1) / BIN_WARPS;
    blocks = std::max<i64>(1, std::min<i64>(blocks, (i64)p->sm_count * p->svm_blocks_per_sm));
    k1_mark(p, 0, st);
    k_obs_svgpm_binned<T, D><<<(unsigned)blocks, BIN_THREADS, 0, st>>>(a);
    k1_mark(p, 1, st);
    VGGP_LAUNCH_CHECK();
    k_band_reduce<T><<<ceil_div(p->band_total, 16), 256, 0, st>>>(a.bin.gband, BAND_REPLICAS, p->band_total, p->band_total, gb + p->M,
                                                                  a.bin.counter);
    VGGP_LAUNCH_CHECK();
    return 0;
}
int obs_svgpm_dispatch(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, void* gbuf, cudaStream_t st) {
    VGGP_DISPATCH_TD(p, launch_obs_svgpm, p, desc, binned, gbuf, st);
}

template <typename T, int D>
int launch_predict_svgpm(vggp_plan* p, const void* const* x, const void* y, i64 n, void* mean, void* var, double* out,
                         cudaStream_t st) {
    SvgpmPredictArgs<T, D> a;
    memset(&a, 0, sizeof(a));
    a.geo = svgpm_geom<D>(p);
    for (int d = 0; d < D; ++d) {
        a.z[d] = p->d_knots[d];
        a.x[d] = reinterpret_cast<const T*>(x[d]);
    }
    a.y = reinterpret_cast<const T*>(y);
    a.n = n;
    a.tab = reinterpret_cast<const T*>(p->svm_tab);
    a.m = reinterpret_cast<const T*>(p->alphaT);
    a.theta = p->theta_dev;
    a.mean = reinterpret_cast<T*>(mean);
    a.var = reinterpret_cast<T*>(var);
    a.out = out;
    const int blocks = (int)std::min<i64>((n + 255) / 256, (i64)p->sm_count * 8);
    if (out) k_predict_svgpm<T, D, true><<<blocks, 256, 0, st>>>(a);
    else k_predict_svgpm<T, D, false><<<blocks, 256, 0, st>>>(a);
    VGGP_LAUNCH_CHECK();
    return 0;
}
int predict_svgpm_dispatch(vggp_plan* p, const void* const* x, const void* y, i64 n, void* mean, void* var, double* out,
                           cudaStream_t st) {
    VGGP_DISPATCH_TD(p, launch_predict_svgpm, p, x, y, n, mean, var, out, st);
}


// ---- optimal variational mean (meanopt.cuh) ---------------------------------------------------------------------
struct MoLayout {
    double *G, *b, *x, *r, *p, *q, *dinv, *band;
    MoStatus* st;
    int band_stride;
    size_t bytes;
};

MoLayout mo_layout(const vggp_plan* p) {
    const int slots = p->D == 1 ? MoSlots<1>::v : (p->D == 2 ? MoSlots<2>::v : MoSlots<3>::v);
    MoLayout L;
    double* base = reinterpret_cast<double*>(p->mo_buf);
    const i64 M = p->M;
    L.G = base;
    L.b = L.G + (i64)slots * M;
    L.x = L.b + M; L.r = L.x + M; L.p = L.r + M; L.q = L.p + M; L.dinv = L.q + M;
    L.band = L.dinv + M;
    L.band_stride = 2 * p->nmax;
    L.st = reinterpret_cast<MoStatus*>(L.band + (i64)p->D * L.band_stride);
    L.bytes = (size_t)((i64)(slots + 6) * M + (i64)p->D * L.band_stride) * sizeof(double) + sizeof(MoStatus);
    return L;
}

// Kronecker buffer: z [M] | Thomas factors [3 sum M_d] | MoKron
struct MoKronLayout {
    double *z, *fac;
    MoKron* k;
    int fac_off[VGGP_MAX_D];
    size_t bytes;
};

MoKronLayout mo_kron_layout(const vggp_plan* p) {
    MoKronLayout K;
    double* base = reinterpret_cast<double*>(p->mo_kbuf);
    i64 nf = 0;
    for (int d = 0; d < p->D; ++d) { K.fac_off[d] = (int)nf; nf += 3 * (i64)p->n[d]; }
    K.z = base;
    K.fac = K.z + p->M;
    K.k = reinterpret_cast<MoKron*>(K.fac + nf);
    K.bytes = (size_t)(p->M + nf) * sizeof(double) + sizeof(MoKron);
    return K;
}

constexpr int MO_SWEEP_SMEM = 32000;    // dynamic shared memory of a staged sweep; with its 16.6 KB static arrays <= 48 KB
// a row of the longest mesh, cut into 32 segments, fits: the contiguous mode is always staged
static_assert(32 * ((((NB * MAX_LEAVES) + 31) / 32) | 1) * sizeof(double) <= (size_t)MO_SWEEP_SMEM,
              "a row of the longest mesh must fit the staged sweep");

// launch shape of the tridiagonal sweep along mode d: S segments per fibre (a power of two <= 32, chosen so that the
// fibres x segments fill the GPU while segments keep >= 4 nodes).  The contiguous mode (d = D - 1) is staged through shared
// memory in tiles of whole rows, at least 32 / S rows per CTA; where such a tile exceeds MO_SWEEP_SMEM, S doubles (shorter
// padded segments, fewer rows) until it fits, which S = 32 always does (static_assert above).
struct MoSweepCfg {
    MoSweep w;
    unsigned blocks, threads;
    size_t smem;
};

MoSweepCfg mo_sweep_cfg(const vggp_plan* p, const MoKronLayout& K, int d, i64 nvec = 1) {
    MoSweepCfg c;
    MoSweep& w = c.w;
    w.n = p->n[d];
    w.inner = p->stride[d];
    w.F = nvec * (p->M / w.n);       // nvec vectors of M back to back: the outer index runs over them as well
    w.fac = K.fac + K.fac_off[d];
    const i64 target = (i64)p->sm_count * 1024;
    int S = 1;
    while (S < 32 && w.F * S < target && (w.n + 2 * S - 1) / (2 * S) >= 4) S *= 2;
    const bool staged = d == p->D - 1;
    if (staged) {
        for (;; S *= 2) {
            const int P = ((w.n + S - 1) / S) | 1;
            if (S == 32 || (size_t)32 * P * sizeof(double) <= (size_t)MO_SWEEP_SMEM) break;
        }
    }
    w.S = S;
    w.Ls = (w.n + S - 1) / S;
    w.P = w.Ls | 1;
    if (staged) {
        const size_t row = (size_t)S * w.P * sizeof(double);
        int rows = 256 / S;
        while (rows > 32 / S && rows * row > (size_t)MO_SWEEP_SMEM) rows /= 2;
        c.threads = (unsigned)(rows * S);
        c.smem = rows * row;
        c.blocks = (unsigned)((w.F + rows - 1) / rows);
    } else {
        c.threads = (unsigned)(32 * S);
        c.smem = 0;
        c.blocks = (unsigned)((w.F + 31) / 32);
    }
    return c;
}

// z = kron_d (F_d + g I)^-1 r, one sweep per mode (the first reads r, the others work in place on z); adds r.z to rz_acc
int mo_kron_apply(const vggp_plan* p, const MoKronLayout& K, const double* r, double* z, MoStatus* mst, cudaStream_t st) {
    for (int d = 0; d < p->D; ++d) {
        const MoSweepCfg c = mo_sweep_cfg(p, K, d);
        const double* in = d == 0 ? r : z;
        const bool last = d == p->D - 1;
        if (last) k_mo_kron_sweep<true, true><<<c.blocks, c.threads, c.smem, st>>>(c.w, in, z, r, mst);
        else k_mo_kron_sweep<false, false><<<c.blocks, c.threads, 0, st>>>(c.w, in, z, r, mst);
        VGGP_LAUNCH_CHECK();
    }
    return 0;
}

template <typename T, int D>
int mo_assemble_impl(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, cudaStream_t st) {
    const MoLayout L = mo_layout(p);
    unsigned int* counter = p->obs_counter + 2;          // slot 2: this kernel's work-stealing counter, cleared here
    VGGP_CUDA(cudaMemsetAsync(counter, 0, sizeof(unsigned int), st));
    VGGP_CUDA(cudaMemsetAsync(L.G, 0, sizeof(double) * (size_t)(L.x - L.G), st));
    if (desc->n_tasks == 0) return 0;
    BinnedArgs<T, D> a;
    memset(&a, 0, sizeof(a));
    a.buf = reinterpret_cast<const unsigned char*>(binned);
    a.off_task_off = desc->off_task_off; a.off_task_R = desc->off_task_R; a.off_run_cell = desc->off_run_cell;
    a.off_run_n = desc->off_run_n; a.off_data = desc->off_data;
    a.n_tasks = (int)desc->n_tasks;
    a.counter = counter;
    i64 blocks = (desc->n_tasks + BIN_WARPS - 1) / BIN_WARPS;
    if (p->family == VGGP_B1_ASVGP) {
        for (int d = 0; d < D; ++d) {
            a.geo.K[d] = p->K[d];
            a.geo.stride[d] = (int)p->stride[d];
            a.geo.tab_off[d] = p->tab_off[d];
            a.geo.knot_off[d] = p->knot_off[d];
        }
        a.tables = p->tables;
        a.knots_byte_off = p->knots_byte_off;
        int nb = 0;
        VGGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_mo_b1_assemble<T, D>, BIN_THREADS, 0));
        blocks = std::max<i64>(1, std::min<i64>(blocks, (i64)p->sm_count * std::max(nb, 1)));
        k_mo_b1_assemble<T, D><<<(unsigned)blocks, BIN_THREADS, 0, st>>>(a, L.G, L.b, p->M);
    } else {
        SvgpmArgs<T, D> sa;
        memset(&sa, 0, sizeof(sa));
        sa.bin = a;
        sa.geo = svgpm_geom<D>(p);
        sa.tab = reinterpret_cast<const T*>(p->svm_tab);
        sa.theta = p->theta_dev;
        int nb = 0;
        VGGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_mo_svm_assemble<T, D>, BIN_THREADS, 0));
        blocks = std::max<i64>(1, std::min<i64>(blocks, (i64)p->sm_count * std::max(nb, 1)));
        k_mo_svm_assemble<T, D><<<(unsigned)blocks, BIN_THREADS, 0, st>>>(sa, L.G, L.b, p->M);
    }
    VGGP_LAUNCH_CHECK();
    return 0;
}
int mo_assemble_dispatch(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, cudaStream_t st) {
    VGGP_DISPATCH_TD(p, mo_assemble_impl, p, desc, binned, st);
}

// ---- optimal covariance (covopt.cuh) -------------------------------------------------------------------------
template <typename T>
int covopt_impl(vggp_plan* p, int dim, const void* gbuf, double ell_scale, const double* L, double* L_out, double* change,
                cudaStream_t st) {
    const int n = p->n[dim];
    double* base = reinterpret_cast<double*>(p->co_buf);
    CoArgs a;
    a.n = n; a.d = dim; a.D = p->D; a.family = p->family;
    a.scale = sqrt((double)p->M / (double)n);
    a.fd = base; a.fo = base + n; a.ib = base + 2 * n; a.rr = base + 3 * n; a.xd = base + 4 * n; a.xs = base + 5 * n;
    a.acc = base + 6 * n;
    a.Lold = L + p->g.Loff[dim];
    a.Lout = L_out + p->g.Loff[dim];
    const bool b1 = p->family == VGGP_B1_ASVGP;
    const T* band = reinterpret_cast<const T*>(gbuf) + p->M + p->band_off[dim];
    const double* trs = b1 ? p->g.sc + SC_TR : p->svm_sc + SVS_TR;
    k_co_factor<T><<<1, CO_THREADS, 0, st>>>(a, p->g, b1 ? nullptr : p->svm_W[dim], band, p->theta_dev, trs, ell_scale,
                                             p->g.info);
    VGGP_LAUNCH_CHECK();
    const unsigned cols = (unsigned)ceil_div(n, CO_THREADS);
    if (b1) {
        k_co_b1_x<<<cols, CO_THREADS, 0, st>>>(a);
        VGGP_LAUNCH_CHECK();
        k_co_b1_rq<<<1, CO_THREADS, 0, st>>>(a);
    } else {
        k_co_markov<<<cols, CO_THREADS, 0, st>>>(a);
    }
    VGGP_LAUNCH_CHECK();
    k_co_change<<<1, 32, 0, st>>>(a.acc, change);
    VGGP_LAUNCH_CHECK();
    return 0;
}

// the assembled system at the theta of the last forward (the B1 bands are filled by k_mo_b1_bands)
template <int D>
MoSys<D> mo_system(const vggp_plan* p, const MoLayout& L) {
    const bool b1 = p->family == VGGP_B1_ASVGP;
    MoSys<D> s;
    memset(&s, 0, sizeof(s));
    s.M = p->M;
    for (int d = 0; d < D; ++d) {
        s.n[d] = p->n[d];
        s.stride[d] = (int)p->stride[d];
        if (b1) {
            s.bd[d] = L.band + (i64)d * L.band_stride;
            s.bo[d] = s.bd[d] + p->n[d];
        } else {
            s.bd[d] = p->svm_W[d] + (i64)SVW_PD * p->n[d];
            s.bo[d] = p->svm_W[d] + (i64)SVW_PO * p->n[d];
        }
    }
    s.G = L.G;
    s.theta = p->theta_dev;
    return s;
}

constexpr int MO_BATCH = 64;        // CG iterations launched between two reads of the status record

// precond: VGGP_MEANOPT_JACOBI or VGGP_MEANOPT_KRONECKER (the Jacobi launches are those of the solve before the choice)
template <int D>
int mo_solve_impl(vggp_plan* p, int precond, double rtol, int max_iter, double* m_out, int* iters_host, double* relres_host,
                  cudaStream_t st) {
    const bool kron = precond == VGGP_MEANOPT_KRONECKER;
    if (kron && !p->mo_kbuf) {
        const size_t want = mo_kron_layout(p).bytes;
        VGGP_CUDA(cudaMalloc(&p->mo_kbuf, want));
        p->mo_kbytes = want;
    }
    const MoLayout L = mo_layout(p);
    const bool b1 = p->family == VGGP_B1_ASVGP;
    const MoSys<D> s = mo_system<D>(p, L);
    const unsigned blocks = (unsigned)std::min<i64>((p->M + 255) / 256, (i64)p->sm_count * 8);
    if (b1) {
        k_mo_b1_bands<<<dim3(ceil_div(p->nmax, 256), D), 256, 0, st>>>(p->g, p->theta_dev, L.band, L.band_stride);
        VGGP_LAUNCH_CHECK();
    }
    VGGP_CUDA(cudaMemsetAsync(L.st, 0, sizeof(MoStatus), st));
    MoKronLayout K{};
    if (kron) {
        K = mo_kron_layout(p);
        MoFacOff<D> fo;
        for (int d = 0; d < D; ++d) fo.off[d] = K.fac_off[d];
        VGGP_CUDA(cudaMemsetAsync(K.k, 0, sizeof(MoKron), st));
        k_mo_kron_trace<<<blocks, 256, 0, st>>>(p->M, L.G, K.k);
        VGGP_LAUNCH_CHECK();
        k_mo_kron_factors<D><<<1, 32, 0, st>>>(s, K.k, K.fac, fo);
        VGGP_LAUNCH_CHECK();
        // initial guess as below; z0 = P r0 adds r0.z0 to rz_acc, p0 = z0
        if (b1) k_mo_kron_init<double, D><<<blocks, 256, 0, st>>>(s, L.b, p->alpha, L.x, L.r, L.st);
        else if (p->obs_dtype == VGGP_F32)
            k_mo_kron_init<float, D><<<blocks, 256, 0, st>>>(s, L.b, reinterpret_cast<const float*>(p->alphaT), L.x, L.r, L.st);
        else k_mo_kron_init<double, D><<<blocks, 256, 0, st>>>(s, L.b, reinterpret_cast<const double*>(p->alphaT), L.x, L.r, L.st);
        VGGP_LAUNCH_CHECK();
        if (int rc = mo_kron_apply(p, K, L.r, K.z, L.st, st)) return rc;
        VGGP_CUDA(cudaMemcpyAsync(L.p, K.z, sizeof(double) * (size_t)p->M, cudaMemcpyDeviceToDevice, st));
    } else {
        // initial guess: the state of the last grid forward (B1: alpha = Kuu^-1 m in float64; Markov: m as the kernels read it)
        if (b1) k_mo_init<double, D><<<blocks, 256, 0, st>>>(s, L.b, p->alpha, L.x, L.r, L.p, L.dinv, L.st);
        else if (p->obs_dtype == VGGP_F32)
            k_mo_init<float, D><<<blocks, 256, 0, st>>>(s, L.b, reinterpret_cast<const float*>(p->alphaT), L.x, L.r, L.p, L.dinv, L.st);
        else k_mo_init<double, D><<<blocks, 256, 0, st>>>(s, L.b, reinterpret_cast<const double*>(p->alphaT), L.x, L.r, L.p, L.dinv, L.st);
        VGGP_LAUNCH_CHECK();
    }
    MoStatus h;
    VGGP_CUDA(cudaMemcpyAsync(&h, L.st, sizeof(MoStatus), cudaMemcpyDeviceToHost, st));
    VGGP_CUDA(cudaStreamSynchronize(st));
    if (h.bb == 0.0) {          // no data: m* = 0
        VGGP_CUDA(cudaMemsetAsync(m_out, 0, sizeof(double) * (size_t)p->M, st));
        VGGP_CUDA(cudaStreamSynchronize(st));
        *iters_host = 0;
        *relres_host = 0.0;
        return 0;
    }
    double relres = sqrt(h.rr_acc / h.bb);
    int iters = 0;
    while (relres > rtol && iters < max_iter) {
        const int nb = std::min(MO_BATCH, max_iter - iters);
        for (int k = 0; k < nb; ++k) {
            k_mo_matvec<D><<<blocks, 256, 0, st>>>(s, L.p, L.q, L.st);
            VGGP_LAUNCH_CHECK();
            if (kron) {
                k_mo_kron_update<<<blocks, 256, 0, st>>>(p->M, L.p, L.q, L.x, L.r, L.st);
                VGGP_LAUNCH_CHECK();
                if (int rc = mo_kron_apply(p, K, L.r, K.z, L.st, st)) return rc;
                k_mo_kron_direction<<<blocks, 256, 0, st>>>(p->M, K.z, L.p, rtol, L.st);
                VGGP_LAUNCH_CHECK();
            } else {
                k_mo_update<<<blocks, 256, 0, st>>>(p->M, L.p, L.q, L.dinv, L.x, L.r, L.st);
                VGGP_LAUNCH_CHECK();
                k_mo_direction<<<blocks, 256, 0, st>>>(p->M, L.r, L.dinv, L.p, rtol, L.st);
                VGGP_LAUNCH_CHECK();
            }
        }
        VGGP_CUDA(cudaMemcpyAsync(&h, L.st, sizeof(MoStatus), cudaMemcpyDeviceToHost, st));
        VGGP_CUDA(cudaStreamSynchronize(st));
        iters = h.iters;
        relres = h.relres;
        if (h.done) break;
    }
    if (b1) {
        k_mo_prior_apply<D><<<blocks, 256, 0, st>>>(s, L.x, m_out);
        VGGP_LAUNCH_CHECK();
    } else {
        VGGP_CUDA(cudaMemcpyAsync(m_out, L.x, sizeof(double) * (size_t)p->M, cudaMemcpyDeviceToDevice, st));
    }
    VGGP_CUDA(cudaStreamSynchronize(st));
    *iters_host = iters;
    *relres_host = relres;
    return 0;
}

// ---- collapsed ELBO (collapsed.cuh) ---------------------------------------------------------------------------------
// One buffer, grown on demand: [inverse bands 4 sum M_d | d'^-1/2 sum M_d | log det F_d 4 | term partials 3 NB | diag(A)^-1/2 M |
//                               Lanczos partials 2 k NB | alpha k S | beta k S | v0, v1, t, y: 4 k M | nsteps k | done k]
// with NB = CT_NB_PER_SM * SMs CTAs at most per probe and S = max_steps.
constexpr int CT_NB_PER_SM = 8;
constexpr int CT_CHECK = 8;             // Lanczos steps launched between the first reads of the coefficients

struct CtLayout {
    double *ib, *rs, *ldf, *tpart, *sdiag, *part, *alpha, *beta, *v[4];
    int *nsteps, *done;
    int nb;
    size_t bytes;
};

CtLayout ct_layout(const vggp_plan* p, void* buf, int k, int max_steps) {
    CtLayout c;
    c.nb = p->sm_count * CT_NB_PER_SM;
    i64 nf = 0;
    for (int d = 0; d < p->D; ++d) nf += 4 * (i64)p->n[d];
    double* q = reinterpret_cast<double*>(buf);
    c.ib = q; q += nf;
    c.rs = q; q += nf / 4;
    c.ldf = q; q += 4;
    c.tpart = q; q += 3 * (i64)c.nb;
    c.sdiag = q; q += p->M;
    c.part = q; q += 2 * (i64)k * c.nb;
    c.alpha = q; q += (i64)k * max_steps;
    c.beta = q; q += (i64)k * max_steps;
    for (int i = 0; i < 4; ++i) { c.v[i] = q; q += (i64)k * p->M; }
    c.nsteps = reinterpret_cast<int*>(q);
    c.done = c.nsteps + k;
    c.bytes = (size_t)(reinterpret_cast<char*>(c.done + k) - reinterpret_cast<char*>(buf));
    return c;
}

int ct_reserve(vggp_plan* p, int k, int max_steps, cudaStream_t st) {
    const size_t want = ct_layout(p, nullptr, k, max_steps).bytes;
    if (p->ct_buf && p->ct_bytes >= want) return 0;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusActive)
        return fail(VGGP_E_UNSUPPORTED, "the collapsed-ELBO scratch grows here: call it outside a stream capture");
    if (p->ct_buf) {
        VGGP_CUDA(cudaStreamSynchronize(st));
        VGGP_CUDA(cudaFree(p->ct_buf));
        p->ct_buf = nullptr;
        p->ct_bytes = 0;
    }
    VGGP_CUDA(cudaMalloc(&p->ct_buf, want));
    p->ct_bytes = want;
    return 0;
}

// Eigenvalues theta_i of the symmetric tridiagonal (a [n], b [n - 1]) and the squared first components tau_i^2 of its
// eigenvectors, by the implicit QL method with Wilkinson shifts (Golub-Welsch: only the first row of the eigenvector matrix
// is carried).  Returns sum_i tau_i^2 log theta_i, NaN if an eigenvalue is not positive or the iteration does not settle.
double ct_gauss_log(int n, const double* a, const double* b, std::vector<double>& d, std::vector<double>& e,
                    std::vector<double>& z) {
    d.assign(a, a + n);
    e.assign(n, 0.0);
    for (int i = 0; i + 1 < n; ++i) e[i] = b[i];
    z.assign(n, 0.0);
    z[0] = 1.0;
    for (int l = 0; l < n; ++l) {
        int iter = 0, m;
        do {
            for (m = l; m < n - 1; ++m) {
                const double dd = fabs(d[m]) + fabs(d[m + 1]);
                if (fabs(e[m]) <= 1e-16 * dd) break;
            }
            if (m != l) {
                if (iter++ == 100) return NAN;
                double g = (d[l + 1] - d[l]) / (2.0 * e[l]);
                double r = hypot(g, 1.0);
                g = d[m] - d[l] + e[l] / (g + copysign(r, g));
                double sn = 1.0, c = 1.0, pp = 0.0;
                int i;
                for (i = m - 1; i >= l; --i) {
                    double f = sn * e[i];
                    const double bb = c * e[i];
                    r = hypot(f, g);
                    e[i + 1] = r;
                    if (r == 0.0) {
                        d[i + 1] -= pp;
                        e[m] = 0.0;
                        break;
                    }
                    sn = f / r;
                    c = g / r;
                    g = d[i + 1] - pp;
                    r = (d[i] - g) * sn + 2.0 * c * bb;
                    pp = sn * r;
                    d[i + 1] = g + pp;
                    g = c * r - bb;
                    f = z[i + 1];
                    z[i + 1] = sn * z[i] + c * f;
                    z[i] = c * z[i] - sn * f;
                }
                if (r == 0.0 && i >= l) continue;
                d[l] -= pp;
                e[l] = g;
                e[m] = 0.0;
            }
        } while (m != l);
    }
    double acc = 0.0;
    for (int i = 0; i < n; ++i) {
        if (!(d[i] > 0.0)) return NAN;
        acc += z[i] * z[i] * log(d[i]);
    }
    return acc;
}

template <int D>
int ct_logdet_impl(vggp_plan* p, int precond, int kind, int k, uint64_t seed, int max_steps, double rtol, double* out,
                   double* per_probe, cudaStream_t st) {
    const bool kron = precond == VGGP_MEANOPT_KRONECKER;
    if (kron && !p->mo_kbuf) {
        const size_t want = mo_kron_layout(p).bytes;
        VGGP_CUDA(cudaMalloc(&p->mo_kbuf, want));
        p->mo_kbytes = want;
    }
    if (int rc = ct_reserve(p, k, max_steps, st)) return rc;
    const CtLayout c = ct_layout(p, p->ct_buf, k, max_steps);
    const MoLayout L = mo_layout(p);
    const MoSys<D> s = mo_system<D>(p, L);
    const i64 M = p->M;
    const unsigned nb = (unsigned)std::min<i64>((M + CT_THREADS - 1) / CT_THREADS, (i64)c.nb);
    if (p->family == VGGP_B1_ASVGP) {
        k_mo_b1_bands<<<dim3(ceil_div(p->nmax, 256), D), 256, 0, st>>>(p->g, p->theta_dev, L.band, L.band_stride);
        VGGP_LAUNCH_CHECK();
    }
    // preconditioner and log det P
    double logdet_p = 0.0;
    MoKronLayout K{};
    if (kron) {
        K = mo_kron_layout(p);
        MoFacOff<D> fo;
        for (int d = 0; d < D; ++d) fo.off[d] = K.fac_off[d];
        k_ct_gtrace<<<nb, CT_THREADS, 0, st>>>(M, L.G, c.tpart);
        VGGP_LAUNCH_CHECK();
        k_ct_gtrace_final<<<1, CT_THREADS, 0, st>>>(c.tpart, (int)nb, K.k);
        VGGP_LAUNCH_CHECK();
        k_mo_kron_factors<D><<<1, 32, 0, st>>>(s, K.k, K.fac, fo);
        VGGP_LAUNCH_CHECK();
        k_ct_rsqrt_pivots<D><<<dim3(ceil_div(p->nmax, CT_THREADS), D), CT_THREADS, 0, st>>>(s, K.fac, fo, c.rs);
        VGGP_LAUNCH_CHECK();
        i64 nf = 0;
        for (int d = 0; d < D; ++d) nf += 3 * (i64)p->n[d];
        std::vector<double> fac((size_t)nf);
        VGGP_CUDA(cudaMemcpyAsync(fac.data(), K.fac, sizeof(double) * (size_t)nf, cudaMemcpyDeviceToHost, st));
        VGGP_CUDA(cudaStreamSynchronize(st));
        for (int d = 0; d < D; ++d) {
            double ld = 0.0;
            for (int i = 0; i < p->n[d]; ++i) ld -= log(fac[(size_t)K.fac_off[d] + p->n[d] + i]);
            logdet_p += ((double)M / (double)p->n[d]) * ld;
        }
    } else {
        k_ct_jacobi<D><<<nb, CT_THREADS, 0, st>>>(s, c.sdiag, c.tpart);
        VGGP_LAUNCH_CHECK();
        std::vector<double> part(nb);
        VGGP_CUDA(cudaMemcpyAsync(part.data(), c.tpart, sizeof(double) * nb, cudaMemcpyDeviceToHost, st));
        VGGP_CUDA(cudaStreamSynchronize(st));
        for (unsigned i = 0; i < nb; ++i) logdet_p += part[i];
    }
    // Lanczos on B = C^-1 A C^-T from the probes
    CtLanczos z;
    z.M = M; z.k = k; z.max_steps = max_steps;
    z.alpha = c.alpha; z.beta = c.beta; z.nsteps = c.nsteps; z.done = c.done; z.part = c.part; z.nb = (int)nb;
    VGGP_CUDA(cudaMemsetAsync(c.nsteps, 0, sizeof(int) * 2 * (size_t)k, st));
    double *v0 = c.v[0], *v1 = c.v[1], *y = c.v[3], *t = c.v[2];
    k_ct_probe_init<<<dim3(nb, k), CT_THREADS, 0, st>>>(M, kind, seed, v0, v1);
    VGGP_LAUNCH_CHECK();
    const unsigned sb = (unsigned)std::min<i64>((M + CT_THREADS - 1) / CT_THREADS, (i64)p->sm_count * 8);
    auto apply = [&](const double* in, double* outv) -> int {
        if (!kron) {
            k_ct_stencil<D, true><<<sb, CT_THREADS, 0, st>>>(s, k, in, outv, c.sdiag, c.done);
            VGGP_LAUNCH_CHECK();
            return 0;
        }
        auto sweep = [&](int d, bool fwd, const double* src, double* dst) -> int {
            const MoSweepCfg cf = mo_sweep_cfg(p, K, d, k);
            const double* rs = c.rs + K.fac_off[d] / 3;
            if (d == D - 1) {
                if (fwd) k_ct_kron_half<true, true><<<cf.blocks, cf.threads, cf.smem, st>>>(cf.w, M, rs, src, dst, c.done);
                else k_ct_kron_half<false, true><<<cf.blocks, cf.threads, cf.smem, st>>>(cf.w, M, rs, src, dst, c.done);
            } else {
                if (fwd) k_ct_kron_half<true, false><<<cf.blocks, cf.threads, 0, st>>>(cf.w, M, rs, src, dst, c.done);
                else k_ct_kron_half<false, false><<<cf.blocks, cf.threads, 0, st>>>(cf.w, M, rs, src, dst, c.done);
            }
            VGGP_LAUNCH_CHECK();
            return 0;
        };
        for (int d = D - 1; d >= 0; --d)            // t = C^-T in
            if (int rc = sweep(d, false, d == D - 1 ? in : t, t)) return rc;
        k_ct_stencil<D, false><<<sb, CT_THREADS, 0, st>>>(s, k, t, outv, nullptr, c.done);
        VGGP_LAUNCH_CHECK();
        for (int d = 0; d < D; ++d)                 // out = C^-1 A t
            if (int rc = sweep(d, true, outv, outv)) return rc;
        return 0;
    };
    std::vector<double> ha((size_t)k * max_steps), hb((size_t)k * max_steps), q(k, NAN), qprev(k, NAN);
    std::vector<int> hn(2 * (size_t)k), conv(k, 0), fin(k, 0);
    std::vector<double> wd, we, wz;
    const double norm2 = kind == 0 ? (double)M : 1.0;
    int step = 0;
    while (step < max_steps) {
        // checks every 8 steps up to 128, then every step / 8 rounded down to a multiple of 8: the host quadrature of a
        // probe costs O(steps^2), so the checks stay a small share of long runs
        const int nsb = std::min(CT_CHECK * std::max(1, step / (8 * CT_CHECK)), max_steps - step);
        for (int i = 0; i < nsb; ++i, ++step) {
            if (int rc = apply(v1, y)) return rc;
            k_ct_dot<<<dim3(nb, k), CT_THREADS, 0, st>>>(z, y, v1);
            VGGP_LAUNCH_CHECK();
            k_ct_alpha<<<k, CT_THREADS, 0, st>>>(z, step);
            VGGP_LAUNCH_CHECK();
            k_ct_update<<<dim3(nb, k), CT_THREADS, 0, st>>>(z, step, y, v1, v0);
            VGGP_LAUNCH_CHECK();
            k_ct_beta<<<k, CT_THREADS, 0, st>>>(z, step);
            VGGP_LAUNCH_CHECK();
            k_ct_next<<<dim3(nb, k), CT_THREADS, 0, st>>>(z, step, y);
            VGGP_LAUNCH_CHECK();
            double* old = v0;
            v0 = v1; v1 = y; y = old;
        }
        VGGP_CUDA(cudaMemcpyAsync(ha.data(), c.alpha, sizeof(double) * ha.size(), cudaMemcpyDeviceToHost, st));
        VGGP_CUDA(cudaMemcpyAsync(hb.data(), c.beta, sizeof(double) * hb.size(), cudaMemcpyDeviceToHost, st));
        VGGP_CUDA(cudaMemcpyAsync(hn.data(), c.nsteps, sizeof(int) * hn.size(), cudaMemcpyDeviceToHost, st));
        VGGP_CUDA(cudaStreamSynchronize(st));
        // a probe converges once its quadrature moves by <= rtol (relative) from one check to the next, or when its Krylov
        // space is exhausted; the host then marks it done for the kernels.  done = 3 (step limit) ends it unconverged.
        bool all = true, changed = false;
        for (int j = 0; j < k; ++j) {
            int& dn = hn[(size_t)k + j];
            if (fin[j]) continue;
            qprev[j] = q[j];
            q[j] = norm2 * ct_gauss_log(hn[j], ha.data() + (size_t)j * max_steps, hb.data() + (size_t)j * max_steps, wd, we, wz);
            conv[j] = dn == 2 || fabs(q[j] - qprev[j]) <= rtol * fabs(q[j]);
            if (conv[j] && dn == 0) { dn = 1; changed = true; }
            fin[j] = conv[j] || dn != 0;
            all = all && fin[j];
        }
        if (all) break;
        if (changed) VGGP_CUDA(cudaMemcpyAsync(c.done, hn.data() + k, sizeof(int) * (size_t)k, cudaMemcpyHostToDevice, st));
    }
    VGGP_CUDA(cudaStreamSynchronize(st));
    double sum = 0.0, sq = 0.0;
    int steps = 0, nconv = 0;
    for (int j = 0; j < k; ++j) {
        sum += q[j];
        steps = std::max(steps, hn[j]);
        nconv += conv[j];
        if (per_probe) per_probe[j] = q[j];
    }
    const double mean = sum / k;
    for (int j = 0; j < k; ++j) sq += (q[j] - mean) * (q[j] - mean);
    out[0] = logdet_p + (kind == 0 ? mean : sum);
    out[1] = kind == 0 && k > 1 ? sqrt(sq / (k - 1) / k) : 0.0;
    out[2] = logdet_p;
    out[3] = steps;
    out[4] = nconv;
    out[5] = k;
    return 0;
}

template <typename T, int D>
int ct_terms_impl(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, double* out, cudaStream_t st) {
    if (int rc = ct_reserve(p, 0, 0, st)) return rc;
    const CtLayout c = ct_layout(p, p->ct_buf, 0, 0);
    const MoLayout L = mo_layout(p);
    const MoSys<D> s = mo_system<D>(p, L);
    if (p->family == VGGP_B1_ASVGP) {
        k_mo_b1_bands<<<dim3(ceil_div(p->nmax, 256), D), 256, 0, st>>>(p->g, p->theta_dev, L.band, L.band_stride);
        VGGP_LAUNCH_CHECK();
    }
    k_ct_inv_bands<D><<<1, 32, 0, st>>>(s, c.ib, c.ldf);
    VGGP_LAUNCH_CHECK();
    CtTermArgs a;
    a.data = reinterpret_cast<const unsigned char*>(binned) + desc->off_data;
    a.elems = desc->n_tasks > 0 ? desc->data_elems : 0;
    a.b = L.b;
    a.x = L.x;
    a.ib = c.ib;
    a.part = c.tpart;
    const i64 work = std::max<i64>(p->M, a.elems / (D + 1));
    const unsigned nb = (unsigned)std::max<i64>(1, std::min<i64>((work + CT_THREADS - 1) / CT_THREADS, (i64)c.nb));
    k_ct_terms<T, D><<<nb, CT_THREADS, 0, st>>>(s, a);
    VGGP_LAUNCH_CHECK();
    const double* outside = desc->n_inside < desc->n ? reinterpret_cast<const double*>(binned) : nullptr;
    k_ct_terms_final<D><<<1, CT_THREADS, 0, st>>>(s, c.tpart, (int)nb, c.ldf, (double)desc->n, outside,
                                                  p->family == VGGP_SVGP_MARKOV ? 1 : 0, out);
    VGGP_LAUNCH_CHECK();
    return 0;
}
int ct_terms_dispatch(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, double* out, cudaStream_t st) {
    VGGP_DISPATCH_TD(p, ct_terms_impl, p, desc, binned, out, st);
}


extern "C" {

int vggp_abi_version(void) { return VGGP_ABI_VERSION; }
const char* vggp_last_error(void) { return g_err; }
uint64_t vggp_launch_count(void) { return (uint64_t)g_launches; }

int vggp_set_gemm_mode(int use_mma) {
    g_use_mma = use_mma ? 1 : 0;
    return 0;
}

int vggp_set_binned_stream(int mode) {
    g_bin_stream = mode ? 1 : 0;
    return 0;
}

int vggp_workspace_bytes(const vggp_plan* p, int64_t* plan_bytes, int64_t* gbuf_bytes, int64_t* scratch_bytes) {
    if (!p) return fail(VGGP_E_ARG, "null plan");
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    if (plan_bytes) *plan_bytes = (int64_t)p->alloc_bytes;
    if (gbuf_bytes) *gbuf_bytes = total;
    if (scratch_bytes) {
        const size_t tsz = p->obs_dtype == VGGP_F32 ? 4 : 8;
        size_t sc = p->det_bytes + p->det_fp_elems * sizeof(double) + (size_t)p->pk_cap * tsz * (p->D + 1) + (size_t)p->b0s_raw_bytes + p->mo_bytes + p->mo_kbytes + p->co_bytes + p->ct_bytes;
        if (p->st_x) sc += (size_t)p->st_n * tsz * (p->D + 1) + sizeof(double) * (2 * (size_t)p->M + 2 * (size_t)p->Lsize) + (size_t)total;
        *scratch_bytes = (int64_t)sc;
    }
    return 0;
}

int vggp_set_deterministic(vggp_plan* p, int on) {
    if (!p) return fail(VGGP_E_ARG, "null plan");
    if (on && p->family != VGGP_B1_ASVGP)
        return fail(VGGP_E_UNSUPPORTED, "deterministic mode covers the B1 (ASVGP) family");
    if (on)
        for (int d = 0; d < p->D; ++d)
            if (p->n[d] > 512) return fail(VGGP_E_UNSUPPORTED, "deterministic mode needs M_d <= 512");
    p->det = on ? 1 : 0;
    return 0;
}

int vggp_plan_create(vggp_plan** out, int family, int D, const int* n_knots, const float* const* knots_host,
                     int obs_dtype, int device) {
    if (!out || !n_knots || !knots_host) return fail(VGGP_E_ARG, "null argument");
    if (family != VGGP_B1_ASVGP && family != VGGP_B0_GRIDDED && family != VGGP_SVGP_GRID && family != VGGP_VFF_GRID &&
        family != VGGP_SVGP_MARKOV)
        return fail(VGGP_E_FAMILY, "unknown feature family");
    if ((family == VGGP_SVGP_GRID || family == VGGP_VFF_GRID) && D > 2)
        return fail(VGGP_E_UNSUPPORTED, "the SVGP and VFF families are built for D <= 2, as in the reference");
    if (family == VGGP_VFF_GRID)
        for (int d = 0; d < D; ++d)
            if (n_knots && n_knots[d] % 2 == 0) return fail(VGGP_E_ARG, "a VFF mesh has 2 * nfrequencies + 1 knots");
    if (D < 1 || D > VGGP_MAX_D) return fail(VGGP_E_DIM, "D must be 1..3");
    if (obs_dtype != VGGP_F32 && obs_dtype != VGGP_F64) return fail(VGGP_E_DTYPE, "obs_dtype must be VGGP_F32 or VGGP_F64");
    for (int d = 0; d < D; ++d) {
        if (n_knots[d] < 3) return fail(VGGP_E_ARG, "each mesh needs at least 3 knots");
        if (n_knots[d] > NB * MAX_LEAVES) return fail(VGGP_E_ARG, "mesh too large");
        for (int k = 1; k < n_knots[d]; ++k)
            if (!(knots_host[d][k] > knots_host[d][k - 1])) return fail(VGGP_E_ARG, "knots must be strictly increasing");
    }
    {
        double Mchk = 1.0;
        for (int d = 0; d < D; ++d) Mchk *= (double)n_knots[d];
        if (Mchk >= 2147483647.0) return fail(VGGP_E_ARG, "M = prod M_d must be below 2^31");
    }
    DeviceGuard dev_guard(device);
    { int cur = -1; VGGP_CUDA(cudaGetDevice(&cur)); if (cur != device) return fail(VGGP_E_ARG, "cannot select the device"); }
    vggp_plan* p = new (std::nothrow) vggp_plan();
    if (!p) return fail(VGGP_E_NOMEM, "out of host memory");
    p->family = family; p->D = D; p->obs_dtype = obs_dtype; p->device = device;
    const bool markov = family == VGGP_SVGP_MARKOV;     // O(M + sum M_d^2) grid side: no factor arrays, no GEMM schedules
    const bool b1 = family == VGGP_B1_ASVGP;            // fused grid side (grid_b1.cuh): generators and R_d, no GEMM schedules
    p->M = 1; p->Lsize = 0; p->nmax = 0;
    int rc = 0;
    GridDims& g = p->g;
    memset(&g, 0, sizeof(g));
    g.D = D; g.family = family; g.obs_dtype = obs_dtype;
    int boff = 0, koff = 0, toff = 0;
    i64 foff = 0;
    for (int d = 0; d < D; ++d) {
        p->K[d] = n_knots[d];
        p->n[d] = (family == VGGP_B0_GRIDDED) ? n_knots[d] - 1 : n_knots[d];      // B0: cells; B1 / SVGP: one inducing variable per knot
        p->M *= p->n[d];
        g.n[d] = p->n[d]; g.K[d] = p->K[d];
        g.delta32[d] = knots_host[d][1] - knots_host[d][0];
        g.Loff[d] = p->Lsize;
        p->Lsize += (i64)p->n[d] * p->n[d];
        p->nmax = std::max(p->nmax, p->n[d]);
        p->band_off[d] = boff; g.band_off[d] = boff;
        boff += 4 * p->n[d];
        p->tab_off[d] = toff; g.tab_off[d] = toff;
        toff += 8 * p->n[d];
        p->gfac_off[d] = foff; g.gfac_off[d] = foff;
        foff += 2 * (i64)p->n[d] * p->n[d];
        p->knot_off[d] = koff;
        koff += p->K[d];
    }
    p->band_total = boff;
    p->tab_total = toff;
    p->gfac_total = foff;
    p->knot_total = koff;
    g.M = p->M;
    for (int d = 0; d < D; ++d) {
        i64 s = 1;
        for (int f = d + 1; f < D; ++f) s *= p->n[f];
        p->stride[d] = s;
    }
#define TRY(expr) do { rc = (expr); if (rc) { vggp_plan_destroy(p); return rc; } } while (0)
    for (int d = 0; d < D; ++d) {
        const int K = p->K[d];
        TRY(dev_alloc(p, &p->d_knots[d], K));
        rc = (int)cudaMemcpy(p->d_knots[d], knots_host[d], sizeof(float) * K, cudaMemcpyHostToDevice);
        if (rc) { vggp_plan_destroy(p); return fail(rc, "cudaMemcpy(knots) failed"); }
        g.knots[d] = p->d_knots[d];
        MeshView& mv = p->mesh[d];
        mv.t = p->d_knots[d]; mv.K = K; mv.t0 = knots_host[d][0];
        mv.inv_h = (float)((double)(K - 1) / ((double)knots_host[d][K - 1] - (double)knots_host[d][0]));
        mv.nearly_uniform = 1;
        mv.tfirst = knots_host[d][0];
        mv.tlast = knots_host[d][K - 1];
        for (int k = 0; k < K; ++k) {
            const float gf = (knots_host[d][k] - mv.t0) * mv.inv_h;
            if (fabsf(gf - (float)k) > 1.25f) mv.nearly_uniform = 0;
        }
        if (markov) continue;
        const i64 nn = (i64)p->n[d] * p->n[d];
        TRY(dev_alloc(p, &g.Kraw[d], nn)); TRY(dev_alloc(p, &g.P[d], nn)); TRY(dev_alloc(p, &g.R[d], nn));
        TRY(dev_alloc(p, &g.Qb[d], 2 * (i64)p->n[d]));
        if (b1) {
            TRY(dev_alloc(p, &g.gen[d], 3 * (i64)p->n[d]));
            continue;
        }
        TRY(dev_alloc(p, &g.Kc[d], nn)); TRY(dev_alloc(p, &g.W[d], nn));
        TRY(dev_alloc(p, &g.cdiag[d], (i64)NB * NB));
        TRY(dev_alloc(p, &g.Lt[d], nn)); TRY(dev_alloc(p, &g.Q[d], nn)); TRY(dev_alloc(p, &g.dP[d], nn));
        TRY(dev_alloc(p, &g.dR[d], nn)); TRY(dev_alloc(p, &g.X[d], nn)); TRY(dev_alloc(p, &g.Y[d], nn));
        TRY(dev_alloc(p, &g.dK[d], nn)); TRY(dev_alloc(p, &g.dLraw[d], nn)); TRY(dev_alloc(p, &g.tmp[d], nn));
        std::vector<int> bounds;
        build_leaves(0, p->n[d], bounds);
        bounds.push_back(p->n[d]);
        g.leaf_cnt[d] = (int)bounds.size() - 1;
        for (size_t i = 0; i < bounds.size(); ++i) g.leaf_lo[d][i] = bounds[i];
    }
    TRY(dev_alloc(p, &g.sc, SC_COUNT));
    TRY(dev_alloc(p, &g.info, 1));
    const size_t tsz = obs_dtype == VGGP_F32 ? 4 : 8;
    if (markov) {
        int toff2 = 0;
        for (int d = 0; d < D; ++d) {
            p->svm_tab_off[d] = toff2;
            toff2 += SVM_TAB * (p->n[d] + 1);
            TRY(dev_alloc(p, &p->svm_W[d], (i64)SVM_W * p->n[d]));
        }
        unsigned char* t = nullptr;
        TRY(dev_alloc(p, &t, (i64)toff2 * (i64)tsz));
        p->svm_tab = t;
        TRY(dev_alloc(p, &p->svm_sc, SVS_COUNT));
        unsigned char* a = nullptr;
        TRY(dev_alloc(p, &a, p->M * (i64)tsz));
        p->alphaT = a;
        unsigned char* br = nullptr;
        TRY(dev_alloc(p, &br, (i64)BAND_REPLICAS * p->band_total * (i64)tsz));
        p->band_rep = br;
        TRY(dev_alloc(p, &p->theta_dev, 2 * VGGP_MAX_D + 1));
        TRY(dev_alloc(p, &p->obs_counter, 4));
        cudaDeviceProp prop;
        rc = (int)cudaGetDeviceProperties(&prop, device);
        if (rc) { vggp_plan_destroy(p); return fail(rc, "cudaGetDeviceProperties failed"); }
        p->sm_count = prop.multiProcessorCount;
        *out = p;
        return 0;
    }
    {
        const int band_bytes = (int)(((size_t)p->tab_total * tsz + 15) / 16 * 16);
        const int knot_bytes = (int)(((size_t)p->knot_total * 4 + 15) / 16 * 16);
        p->knots_byte_off = band_bytes;
        p->table_bytes = band_bytes + knot_bytes;
        TRY(dev_alloc(p, &p->tables, p->table_bytes));
        g.bandT = p->tables;
        for (int d = 0; d < D; ++d) {
            rc = (int)cudaMemcpy(p->tables + band_bytes + 4 * (size_t)p->knot_off[d], knots_host[d],
                                 sizeof(float) * p->K[d], cudaMemcpyHostToDevice);
            if (rc) { vggp_plan_destroy(p); return fail(rc, "cudaMemcpy(knot table) failed"); }
            // static per-cell tables: h = (T)(float32 knot difference), rh = correctly rounded 1 / h
            const int n = p->n[d];
            std::vector<unsigned char> hb(2 * (size_t)n * tsz, 0);
            for (int c = 0; c + 1 < p->K[d] && c < n; ++c) {
                const float hf = knots_host[d][c + 1] - knots_host[d][c];
                if (obs_dtype == VGGP_F32) {
                    reinterpret_cast<float*>(hb.data())[c] = hf;
                    reinterpret_cast<float*>(hb.data())[n + c] = 1.0f / hf;
                } else {
                    reinterpret_cast<double*>(hb.data())[c] = (double)hf;
                    reinterpret_cast<double*>(hb.data())[n + c] = 1.0 / (double)hf;
                }
            }
            rc = (int)cudaMemcpy(p->tables + ((size_t)p->tab_off[d] + 6 * (size_t)n) * tsz, hb.data(), hb.size(),
                                 cudaMemcpyHostToDevice);
            if (rc) { vggp_plan_destroy(p); return fail(rc, "cudaMemcpy(cell table) failed"); }
        }
        unsigned char* a = nullptr;
        TRY(dev_alloc(p, &a, p->M * (i64)tsz));
        p->alphaT = a;
    }
    if (b1) {
        int acc_total = 0;
        for (int d = 0; d < D; ++d) acc_total += 3 * p->n[d];
        p->b1_acc_total = acc_total;
        TRY(dev_alloc(p, &p->b1_acc, acc_total));
        unsigned char* br = nullptr;
        TRY(dev_alloc(p, &br, (i64)BAND_REPLICAS * p->band_total * (i64)tsz));
        p->band_rep = br;
    } else if (obs_dtype == VGGP_F32) {
        TRY(dev_alloc(p, &p->gfac_f64, p->gfac_total));
    }
    TRY(dev_alloc(p, &p->theta_dev, 2 * VGGP_MAX_D + 1));
    TRY(dev_alloc(p, &p->obs_counter, 4));
    TRY(dev_alloc(p, &p->alpha, p->M));
    TRY(dev_alloc(p, &p->pgA, p->M)); TRY(dev_alloc(p, &p->pgB, p->M));
    if (!b1) {
        TRY(dev_alloc(p, &p->mws, p->M));
        TRY(dev_alloc(p, &p->gM, p->M)); TRY(dev_alloc(p, &p->ghat, p->M));
        for (int d = 0; d < D; ++d) {
            if (D > 1) TRY(dev_alloc(p, &p->Tm[d], p->M));
            if (D > 2) TRY(dev_alloc(p, &p->tmpM[d], p->M)); else p->tmpM[d] = nullptr;
        }
        TRY(build_schedules(p));
    }
    {
        cudaDeviceProp prop;
        rc = (int)cudaGetDeviceProperties(&prop, device);
        if (rc) { vggp_plan_destroy(p); return fail(rc, "cudaGetDeviceProperties failed"); }
        p->sm_count = prop.multiProcessorCount;
        p->obs_blocks_per_sm = 1;
        if (b1) TRY(obs_prepare_dispatch(p));
        // the scan form of the cell-integrated family (default for binned observations and for point prediction): its tables
        // (~75 MB at 512 x 512) belong to the plan's one allocation phase, not to the first stream-ordered call that needs them
        if (family == VGGP_B0_GRIDDED && D <= 2) TRY(b0scan_alloc(p));
    }
    rc = raise_dyn_smem(k_chol_panel, (2 * NB * CHOL_PITCH + 2 * NB) * sizeof(double));
    if (!rc) rc = raise_dyn_smem(k_triinv_leaf, 2 * NB * (NB + 1) * sizeof(double));
    if (rc) { vggp_plan_destroy(p); return fail(rc, "cudaFuncSetAttribute failed (is this an sm_100a device?)"); }
#undef TRY
    *out = p;
    return 0;
}

int vggp_plan_destroy(vggp_plan* p) {
    if (!p) return 0;
    DeviceGuard dev_guard(p->device);
    for (void* ptr : p->allocs) cudaFree(ptr);
    for (int d = 0; d < VGGP_MAX_D; ++d)
        if (p->pk_x[d]) cudaFree(p->pk_x[d]);
    if (p->pk_y) cudaFree(p->pk_y);
    if (p->bin_perm) cudaFree(p->bin_perm);
    p->mb.clear();
    if (p->det_buf) cudaFree(p->det_buf);
    if (p->one_ws) cudaFree(p->one_ws);
    if (p->det_fp) cudaFree(p->det_fp);
    if (p->mo_buf) cudaFree(p->mo_buf);
    if (p->mo_kbuf) cudaFree(p->mo_kbuf);
    if (p->ct_buf) cudaFree(p->ct_buf);
    if (p->co_buf) cudaFree(p->co_buf);
    for (auto& e : p->k1_ev) cudaEventDestroy(e);
    for (auto& e : p->k1_gev) if (e) cudaEventDestroy(e);
    for (auto& e : p->st_ev) cudaEventDestroy(e);
    if (p->st_copy) cudaStreamDestroy(p->st_copy);
    void* st[] = {p->st_x, p->st_y, p->st_theta, p->st_m, p->st_L, p->st_out, p->st_dtheta, p->st_dm, p->st_dL, p->st_gbuf};
    for (void* ptr : st)
        if (ptr) cudaFree(ptr);
    delete p;
    return 0;
}

int vggp_plan_dims(const vggp_plan* p, int* D, int* m_per_dim, int64_t* M) {
    if (!p) return fail(VGGP_E_ARG, "null plan");
    if (D) *D = p->D;
    if (m_per_dim) for (int d = 0; d < p->D; ++d) m_per_dim[d] = p->n[d];
    if (M) *M = p->M;
    return 0;
}

int vggp_gbuf_layout(const vggp_plan* p, int64_t* n_obs_elems, int64_t* scalar_offset_bytes, int64_t* n_scalars,
                     int64_t* total_bytes) {
    if (!p) return fail(VGGP_E_ARG, "null plan");
    const i64 tsz = p->obs_dtype == VGGP_F32 ? 4 : 8;
    const bool band = p->family == VGGP_B1_ASVGP || p->family == VGGP_SVGP_MARKOV;
    const i64 ne = p->M + (band ? (i64)p->band_total : p->gfac_total);
    const i64 soff = (ne * tsz + 7) / 8 * 8;
    if (n_obs_elems) *n_obs_elems = ne;
    if (scalar_offset_bytes) *scalar_offset_bytes = soff;
    if (n_scalars) *n_scalars = 8;
    if (total_bytes) *total_bytes = soff + 8 * 8;
    return 0;
}

int vggp_grid_forward(vggp_plan* p, const double* theta, const double* m, const double* L, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !theta || !m || !L) return fail(VGGP_E_ARG, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int D = p->D;
    int rc;
    p->last_stream = st;
    p->forwarded = true;
    p->mo_solved = false;                   // a new theta: the iterate of the last optimal-mean solve no longer belongs to it
    if (p->family == VGGP_SVGP_MARKOV) return svgpm_forward(p, theta, m, L, st);
    if (p->family == VGGP_B1_ASVGP) return b1f_forward(p, theta, m, L, st);
    VGGP_CUDA(cudaMemcpyAsync(p->mws, m, sizeof(double) * p->M, cudaMemcpyDeviceToDevice, st));
    VGGP_CUDA(cudaMemcpyAsync(p->theta_dev, theta, sizeof(double) * (2 * D + 1), cudaMemcpyDeviceToDevice, st));
    const i64 nn = (i64)p->nmax * p->nmax;
    dim3 egrid(ceil_div(nn, 256), D);
    k_build_factors<<<egrid, 256, 0, st>>>(p->g, theta, L);
    VGGP_LAUNCH_CHECK();
    const size_t csm = 2 * NB * (NB + 1) * sizeof(double), cpsm = (2 * NB * CHOL_PITCH + 2 * NB) * sizeof(double);
    for (int j = 0; j < p->n_panels; ++j) {
        const int j0 = j * NB;
        dim3 grid(ceil_div(p->nmax - j0, NB), D);
        k_chol_panel<<<grid, 256, cpsm, st>>>(p->g, j0);
        VGGP_LAUNCH_CHECK();
        if ((rc = launch_phase(p->chol_trailing[j], st))) return rc;
    }
    int max_leaves = 0;
    for (int d = 0; d < D; ++d) max_leaves = std::max(max_leaves, p->g.leaf_cnt[d]);
    k_triinv_leaf<<<dim3(max_leaves, D), NB, csm, st>>>(p->g);
    VGGP_LAUNCH_CHECK();
    for (auto& ph : p->triinv) if ((rc = launch_phase(ph, st))) return rc;
    if ((rc = launch_phase(p->pinv, st))) return rc;
    if ((rc = launch_phase(p->rs, st))) return rc;
    if ((rc = launch_phase(p->qq, st))) return rc;
    {
        dim3 rgrid(ceil_div(p->nmax, 8), D), tgrid(ceil_div(p->nmax, 256), D);
        if (p->obs_dtype == VGGP_F32) {
            k_fwd_reduce<float><<<rgrid, 256, 0, st>>>(p->g);
            VGGP_LAUNCH_CHECK();
            k_fwd_qtable<float><<<tgrid, 256, 0, st>>>(p->g);
        } else {
            k_fwd_reduce<double><<<rgrid, 256, 0, st>>>(p->g);
            VGGP_LAUNCH_CHECK();
            k_fwd_qtable<double><<<tgrid, 256, 0, st>>>(p->g);
        }
        VGGP_LAUNCH_CHECK();
    }
    for (auto& ph : p->chains) if ((rc = launch_phase(ph, st))) return rc;
    if ((rc = launch_phase(p->alpha_phase, st))) return rc;
    const int cblocks = (int)std::min<i64>((p->M + 255) / 256, 148 * 4);
    if (p->obs_dtype == VGGP_F32)
        k_cast_alpha<float><<<cblocks, 256, 0, st>>>(p->alpha, p->mws, reinterpret_cast<float*>(p->alphaT), p->M, p->g.sc);
    else
        k_cast_alpha<double><<<cblocks, 256, 0, st>>>(p->alpha, p->mws, reinterpret_cast<double*>(p->alphaT), p->M, p->g.sc);
    VGGP_LAUNCH_CHECK();
    return 0;
}

int vggp_obs_pack_geometry(const vggp_plan* p, int64_t n, int64_t* n_packed, int* run_len) {
    if (!p || n < 0) return fail(VGGP_E_ARG, "bad argument");
    const PackGeom g = pack_geometry(p, n);
    if (n_packed) *n_packed = g.n_packed;
    if (run_len) *run_len = g.R;
    return 0;
}

int vggp_obs_pack(vggp_plan* p, const void* const* x, const void* y, int64_t n, int sort_by_cell, void* const* xp,
                  void* yp, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || n < 0) return fail(VGGP_E_ARG, "bad argument");
    if (n == 0) return 0;
    if (p->family != VGGP_B1_ASVGP) return fail(VGGP_E_UNSUPPORTED, "the packed layout is used by the B1 family only");
    if (!x || !y || !xp || !yp) return fail(VGGP_E_ARG, "null argument");
    for (int d = 0; d < p->D; ++d)
        if (!x[d] || !xp[d]) return fail(VGGP_E_ARG, "null observation pointer");
    return pack_dispatch(p, x, y, n, sort_by_cell, xp, yp, (cudaStream_t)stream);
}

int vggp_obs_fwd_bwd_packed(vggp_plan* p, const void* const* xp, const void* yp, int64_t n, void* gbuf, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (p && p->det) return fail(VGGP_E_UNSUPPORTED, "deterministic mode takes the binned layout (vggp_obs_fwd_bwd_binned)");
    if (!p || !gbuf || n < 0) return fail(VGGP_E_ARG, "bad argument");
    if (p->family == VGGP_SVGP_MARKOV) return fail(VGGP_E_UNSUPPORTED, "the Markov SVGP family takes the binned layout (vggp_obs_bin_prepare / _pack, vggp_obs_fwd_bwd_binned)");
    if (n > 0 && (!xp || !yp)) return fail(VGGP_E_ARG, "null observation pointers");
    cudaStream_t st = (cudaStream_t)stream;
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    VGGP_CUDA(cudaMemsetAsync(gbuf, 0, (size_t)total, st));
    if (n == 0) return 0;
    for (int d = 0; d < p->D; ++d)
        if (!xp[d]) return fail(VGGP_E_ARG, "null observation pointer");
    if (p->family != VGGP_B1_ASVGP)
        return fail(VGGP_E_UNSUPPORTED, "the packed layout is used by the B1 family only; call vggp_obs_fwd_bwd");
    return obs_packed_dispatch(p, xp, yp, n, gbuf, st);
}

int vggp_obs_fwd_bwd(vggp_plan* p, const void* const* x, const void* y, int64_t n, void* gbuf, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (p && p->det) return fail(VGGP_E_UNSUPPORTED, "deterministic mode takes the binned layout (vggp_obs_fwd_bwd_binned)");
    if (!p || !gbuf || n < 0) return fail(VGGP_E_ARG, "bad argument");
    if (p->family == VGGP_SVGP_MARKOV) return fail(VGGP_E_UNSUPPORTED, "the Markov SVGP family takes the binned layout (vggp_obs_bin_prepare / _pack, vggp_obs_fwd_bwd_binned)");
    if (n > 0 && (!x || !y)) return fail(VGGP_E_ARG, "null observation pointers");
    if (n == 0 || p->family != VGGP_B1_ASVGP) {
        cudaStream_t st0 = (cudaStream_t)stream;
        i64 ne0, so0, ns0, tot0;
        vggp_gbuf_layout(p, &ne0, &so0, &ns0, &tot0);
        VGGP_CUDA(cudaMemsetAsync(gbuf, 0, (size_t)tot0, st0));
        if (n == 0) return 0;
        for (int d = 0; d < p->D; ++d)
            if (!x[d]) return fail(VGGP_E_ARG, "null observation pointer");
        return obs_b0_dispatch(p, x, y, n, gbuf, st0);
    }
    // unpacked input: transpose into the packed layout (input order kept) in plan-owned scratch, grown on demand
    const PackGeom g = pack_geometry(p, n);
    const size_t tsz = p->obs_dtype == VGGP_F32 ? 4 : 8;
    if (g.n_packed > p->pk_cap) {
        VGGP_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
        for (int d = 0; d < p->D; ++d) {
            if (p->pk_x[d]) cudaFree(p->pk_x[d]);
            p->pk_x[d] = nullptr;
        }
        if (p->pk_y) cudaFree(p->pk_y);
        p->pk_y = nullptr;
        p->pk_cap = 0;
        for (int d = 0; d < p->D; ++d) VGGP_CUDA(cudaMalloc(&p->pk_x[d], tsz * (size_t)g.n_packed));
        VGGP_CUDA(cudaMalloc(&p->pk_y, tsz * (size_t)g.n_packed));
        p->pk_cap = g.n_packed;
    }
    int rc = vggp_obs_pack(p, x, y, n, 0, p->pk_x, p->pk_y, stream);
    if (rc) return rc;
    return vggp_obs_fwd_bwd_packed(p, p->pk_x, p->pk_y, n, gbuf, stream);
}

// run_cap = 0 of the binned layouts: about two tasks (of 32 runs) per resident warp, so that thin shards and cell-range shards
// (few, full cells) still spread over the whole GPU; 256 (the value the 1-GPU measurements settled on) from 2^25.8 observations up
static int auto_run_cap(const vggp_plan* p, i64 n) {
    const i64 warps = (i64)p->sm_count * 24;
    const i64 want = (n + 64 * warps - 1) / (64 * warps);
    return (int)std::min<i64>(256, std::max<i64>(32, (want + 3) / 4 * 4));
}

int vggp_obs_bin_prepare(vggp_plan* p, const void* const* x, int64_t n, int run_cap, vggp_binned_desc* desc, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !desc || n < 0) return fail(VGGP_E_ARG, "bad argument");
    if (p->family == VGGP_B0_GRIDDED && p->D > 2) return fail(VGGP_E_UNSUPPORTED, "the B0 (cell-integrated) family is built for D <= 2, as in the reference");
    if (p->family == VGGP_SVGP_GRID || p->family == VGGP_VFF_GRID)
        return fail(VGGP_E_UNSUPPORTED, "the SVGP and VFF families take plain observation arrays (vggp_obs_fwd_bwd)");
    if (run_cap == 0) run_cap = auto_run_cap(p, n);
    if (run_cap < 4) return fail(VGGP_E_ARG, "run_cap must be >= 4 (0 = automatic)");
    if (n >= ((i64)1 << 31)) return fail(VGGP_E_UNSUPPORTED, "binning supports n < 2^31 observations per shard");
    if (n > 0) {
        if (!x) return fail(VGGP_E_ARG, "null observation pointers");
        for (int d = 0; d < p->D; ++d)
            if (!x[d]) return fail(VGGP_E_ARG, "null observation pointer");
    }
    if (p->bin_perm) { cudaFree(p->bin_perm); p->bin_perm = nullptr; }
    p->bin_has_pending = false;
    memset(desc, 0, sizeof(*desc));
    return bin_prepare_dispatch(p, x, n, run_cap, desc, (cudaStream_t)stream);
}

int vggp_obs_bin_pack(vggp_plan* p, const vggp_binned_desc* desc, const void* const* x, const void* y, void* binned,
                      void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !desc || !binned) return fail(VGGP_E_ARG, "bad argument");
    if (!p->bin_has_pending) return fail(VGGP_E_ARG, "vggp_obs_bin_pack without a pending vggp_obs_bin_prepare on this plan");
    const BinLayout& L = p->bin_pending;
    if (desc->n != L.n || desc->n_tasks != L.n_tasks || desc->data_elems != L.data_elems || desc->D != p->D)
        return fail(VGGP_E_ARG, "descriptor does not match the pending layout");
    if (L.n > 0) {
        if (!x || !y) return fail(VGGP_E_ARG, "null observation pointers");
        for (int d = 0; d < p->D; ++d)
            if (!x[d]) return fail(VGGP_E_ARG, "null observation pointer");
    }
    return bin_pack_dispatch(p, desc, x, y, binned, (cudaStream_t)stream);
}

int vggp_obs_fwd_bwd_binned(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, void* gbuf, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !desc || !gbuf) return fail(VGGP_E_ARG, "bad argument");
    if (p->family == VGGP_B0_GRIDDED && p->D > 2) return fail(VGGP_E_UNSUPPORTED, "the B0 (cell-integrated) family is built for D <= 2, as in the reference");
    if (desc->D != p->D) return fail(VGGP_E_ARG, "descriptor belongs to a plan of another dimension");
    cudaStream_t st = (cudaStream_t)stream;
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    VGGP_CUDA(cudaMemsetAsync(gbuf, 0, (size_t)total, st));
    if (desc->n == 0) return 0;
    if (!binned) return fail(VGGP_E_ARG, "null binned buffer");
    if (p->family == VGGP_SVGP_GRID || p->family == VGGP_VFF_GRID)
        return fail(VGGP_E_UNSUPPORTED, "the SVGP and VFF families take plain observation arrays (vggp_obs_fwd_bwd)");
    if (p->family == VGGP_SVGP_MARKOV) return obs_svgpm_dispatch(p, desc, binned, gbuf, st);  // Markov form (svgpm.cuh)
    if (p->family == VGGP_B0_GRIDDED) return obs_b0s_dispatch(p, desc, binned, gbuf, st);     // scan form (b0scan.cuh)
    return obs_binned_dispatch(p, desc, binned, gbuf, st);
}

int vggp_epoch_bin_prepare(vggp_plan* p, const void* const* x, int64_t n, int64_t batch_size, int64_t n_batches, int run_cap,
                           uint64_t seed, uint64_t epoch, int rank, vggp_epoch_desc* desc, int64_t* totals_host, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !desc || !totals_host) return fail(VGGP_E_ARG, "bad argument");
    if (p->family == VGGP_SVGP_GRID || p->family == VGGP_VFF_GRID)
        return fail(VGGP_E_UNSUPPORTED, "the SVGP and VFF families have no binned layout: index their plain arrays");
    if (p->family == VGGP_B0_GRIDDED && p->D > 2) return fail(VGGP_E_UNSUPPORTED, "the B0 (cell-integrated) family is built for D <= 2, as in the reference");
    if (n < 1 || n >= ((i64)1 << 31)) return fail(VGGP_E_ARG, "epoch binning needs 1 <= n < 2^31 observations per shard");
    if (batch_size < 1 || batch_size > n) return fail(VGGP_E_ARG, "batch_size must be in 1..n");
    if (n_batches < 0 || n_batches > n / batch_size) return fail(VGGP_E_ARG, "n_batches must be in 0..n / batch_size (0 = n / batch_size)");
    if (rank < 0) return fail(VGGP_E_ARG, "rank must be >= 0");
    if (run_cap == 0) run_cap = auto_run_cap(p, batch_size);
    if (run_cap < 4) return fail(VGGP_E_ARG, "run_cap must be >= 4 (0 = automatic)");
    if (!x) return fail(VGGP_E_ARG, "null observation pointers");
    for (int d = 0; d < p->D; ++d)
        if (!x[d]) return fail(VGGP_E_ARG, "null observation pointer");
    p->mb.clear();
    memset(desc, 0, sizeof(*desc));
    desc->n = n; desc->batch_size = batch_size; desc->n_batches = n_batches ? n_batches : n / batch_size;
    desc->seed = seed; desc->epoch = epoch; desc->rank = rank;
    desc->run_cap = run_cap / 4 * 4; desc->D = p->D; desc->elem_size = p->obs_dtype == VGGP_F32 ? 4 : 8;
    const int rc = epoch_prepare_dispatch(p, x, desc, totals_host, (cudaStream_t)stream);
    if (rc) p->mb.clear();
    return rc;
}

int vggp_epoch_bin_pack(vggp_plan* p, const vggp_epoch_desc* desc, const int64_t* totals_host, const void* const* x, const void* y,
                        void* binned, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !desc || !totals_host || !binned) return fail(VGGP_E_ARG, "bad argument");
    if (!p->mb.active) return fail(VGGP_E_ARG, "vggp_epoch_bin_pack without a pending vggp_epoch_bin_prepare on this plan");
    if (memcmp(desc, &p->mb.desc, sizeof(*desc)) != 0) return fail(VGGP_E_ARG, "descriptor does not match the pending epoch");
    if (!x || !y) return fail(VGGP_E_ARG, "null observation pointers");
    for (int d = 0; d < p->D; ++d)
        if (!x[d]) return fail(VGGP_E_ARG, "null observation pointer");
    const int rc = epoch_pack_dispatch(p, totals_host, x, y, binned, (cudaStream_t)stream);
    if (rc) p->mb.clear();
    return rc;
}

int vggp_epoch_batch(const vggp_epoch_desc* desc, const int64_t* totals_host, int64_t b, vggp_binned_desc* batch,
                     int64_t* byte_offset) {
    if (!desc || !totals_host || !batch || !byte_offset) return fail(VGGP_E_ARG, "bad argument");
    if (b < 0 || b >= desc->n_batches) return fail(VGGP_E_ARG, "batch index out of range");
    mb_batch_desc(desc, totals_host, b, batch, byte_offset);
    return 0;
}

int vggp_allreduce_gbuf(vggp_plan* p, const vggp_ar_desc* desc, int* err_flag, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !desc || !err_flag) return fail(VGGP_E_ARG, "null argument");
    if (desc->world < 1 || desc->world > AR_MAX_RANKS || desc->rank < 0 || desc->rank >= desc->world)
        return fail(VGGP_E_ARG, "world must be 1..8 and rank inside it");
#ifdef VGGP_EMUL
    (void)stream;
    return fail(VGGP_E_UNSUPPORTED, "the peer-memory collective needs NVLink peers");
#else
    if (desc->world == 1) return 0;
    ArArgs a;
    memset(&a, 0, sizeof(a));
    a.mc = desc->mc_ptr;
    for (int r = 0; r < desc->world; ++r) {
        if (!desc->buf_ptrs[r] || !desc->pad_ptrs[r]) return fail(VGGP_E_ARG, "null peer pointer");
        a.buf[r] = desc->buf_ptrs[r];
        a.pad[r] = reinterpret_cast<unsigned int*>(desc->pad_ptrs[r]);
    }
    a.rank = desc->rank; a.world = desc->world;
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    a.n_obs = n_elems; a.obs_f32 = p->obs_dtype == VGGP_F32; a.scal_off = soff; a.n_scal = (int)nsc;
    a.err = err_flag;
    k_allreduce_gbuf<<<ar_blocks(n_elems, a.obs_f32 ? 4 : 8, a.world), AR_THREADS, 0, (cudaStream_t)stream>>>(a);
    VGGP_LAUNCH_CHECK();
    return 0;
#endif
}

int vggp_grid_backward(vggp_plan* p, const double* theta, const double* m, const double* L, const void* gbuf,
                       double ell_scale, double* out, double* dtheta, double* dm, double* dL, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !theta || !m || !L || !gbuf || !out || !dtheta || !dm || !dL) return fail(VGGP_E_ARG, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int D = p->D;
    int rc;
    if (p->family == VGGP_SVGP_MARKOV) return svgpm_backward(p, theta, m, L, gbuf, ell_scale, out, dtheta, dm, dL, st);
    if (p->family == VGGP_B1_ASVGP) return b1f_backward(p, theta, m, L, gbuf, ell_scale, out, dtheta, dm, dL, st);
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    const double* gscal = reinterpret_cast<const double*>(reinterpret_cast<const unsigned char*>(gbuf) + soff);
    const int mblocks = (int)std::min<i64>((p->M + 255) / 256, 148 * 4);
    if (p->obs_dtype == VGGP_F32)
        k_bwd_prep<float><<<mblocks, 256, 0, st>>>(reinterpret_cast<const float*>(gbuf), p->mws, theta, D, ell_scale, p->gM, p->ghat, p->M);
    else
        k_bwd_prep<double><<<mblocks, 256, 0, st>>>(reinterpret_cast<const double*>(gbuf), p->mws, theta, D, ell_scale, p->gM, p->ghat, p->M);
    VGGP_LAUNCH_CHECK();
    const i64 nn = (i64)p->nmax * p->nmax;
    dim3 egrid(ceil_div(nn, 256), D);
    for (int d = 0; d < D; ++d)
        VGGP_CUDA(cudaMemsetAsync(p->g.dP[d], 0, sizeof(double) * (size_t)p->n[d] * p->n[d], st));
    if ((rc = launch_phase(p->bwdA, st))) return rc;
    if ((rc = launch_phase(p->bwdMid, st))) return rc;
    if (p->obs_dtype == VGGP_F32)
        k_bwd_dense_prep<float><<<egrid, 256, 0, st>>>(p->g, reinterpret_cast<const float*>(gbuf) + p->M, theta, ell_scale);
    else
        k_bwd_dense_prep<double><<<egrid, 256, 0, st>>>(p->g, reinterpret_cast<const double*>(gbuf) + p->M, theta, ell_scale);
    VGGP_LAUNCH_CHECK();
    if ((rc = launch_phase(p->dRp, st))) return rc;
    if ((rc = launch_phase(p->bwdB, st))) return rc;
    k_bwd_dm<<<mblocks, 256, 0, st>>>(p->dm_result, p->alpha, dm, p->M);
    VGGP_LAUNCH_CHECK();
    k_sym<<<egrid, 256, 0, st>>>(p->g);
    VGGP_LAUNCH_CHECK();
    if ((rc = launch_phase(p->Yp, st))) return rc;
    if ((rc = launch_phase(p->dKp, st))) return rc;
    k_bwd_dL<<<egrid, 256, 0, st>>>(p->g, dL);
    VGGP_LAUNCH_CHECK();
    VGGP_CUDA(cudaMemsetAsync(dtheta, 0, sizeof(double) * (2 * D + 1), st));
    k_bwd_theta<<<dim3(64, D), 256, 0, st>>>(p->g, theta, gscal, ell_scale, out, dtheta);
    VGGP_LAUNCH_CHECK();
    return 0;
}

int vggp_k1_timing(vggp_plan* p, int enable) {
    if (!p) return fail(VGGP_E_ARG, "null plan");
    if (enable && p->k1_ev.empty()) {
        p->k1_ev.resize(2 * K1_EVENT_PAIRS);
        for (auto& e : p->k1_ev) VGGP_CUDA(cudaEventCreate(&e));
        for (auto& e : p->k1_gev) VGGP_CUDA(cudaEventCreate(&e));
    }
    p->k1_timing = enable != 0;
    if (enable) p->k1_count = 0;
    return 0;
}

int vggp_k1_time_read(vggp_plan* p, float* mean_ms, int* n_launches) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !mean_ms || !n_launches) return fail(VGGP_E_ARG, "null argument");
    const int n = std::min(p->k1_count, K1_EVENT_PAIRS);
    double acc = 0.0;
    for (int i = 0; i < n; ++i) {
        float ms = 0.f;
        VGGP_CUDA(cudaEventSynchronize(p->k1_ev[2 * i + 1]));
        VGGP_CUDA(cudaEventElapsedTime(&ms, p->k1_ev[2 * i], p->k1_ev[2 * i + 1]));
        acc += ms;
    }
    *mean_ms = n > 0 ? (float)(acc / n) : 0.f;
    *n_launches = p->k1_count;
    return 0;
}

int vggp_k1_graph_time_read(vggp_plan* p, float* ms) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !ms) return fail(VGGP_E_ARG, "null argument");
    if (!p->k1_gev_captured) return fail(VGGP_E_ARG, "no captured graph holds the timing events (enable vggp_k1_timing before the capture)");
    VGGP_CUDA(cudaEventSynchronize(p->k1_gev[1]));
    VGGP_CUDA(cudaEventElapsedTime(ms, p->k1_gev[0], p->k1_gev[1]));
    return 0;
}

int vggp_read_info(vggp_plan* p, int* info_host, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !info_host) return fail(VGGP_E_ARG, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    VGGP_CUDA(cudaMemcpyAsync(info_host, p->g.info, sizeof(int), cudaMemcpyDeviceToHost, st));
    VGGP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

/* debugging aid, not part of the documented ABI: every k_fibre_pass launched afterwards writes 8 int64 per CTA
 * (clock64 at the phase boundaries, globaltimer, kind) to `buf` (device, >= 8 * tiles of the largest pass); NULL switches it off */
int vggp_debug_fp_stamps(long long* buf) { g_fp_dbg = buf; return 0; }
/* debugging aid: 0 = run every fibre pass through the generic kernel (cross-check of k_fibre_pass_fast), 1 = default */
// 0: generic kernel; 1: fast kernel, fibre packing by rule (default); 3: fast, no packing; 5: fast, packing forced (tests)
/* debugging aid: 0 = one-thread-per-fibre sweeps of the B0 scan form (cross-check of the segmented kernels), 1 = default */
int vggp_debug_b0s_seg(int on) { g_b0s_seg = on ? 1 : 0; return 0; }
/* debugging aid: 0 = never cut a small GEMM group along k (plans created afterwards), 1 = default */
int vggp_debug_auto_splitk(int on) { g_auto_splitk = on ? 1 : 0; return 0; }
/* debugging aid: how an automatic k-split combines its partial sums in plans created afterwards: 1 (default) workspace fix-up by
 * the last CTA of a tile (deterministic, no destination clear), 0 float64 atomics into a cleared destination */
int vggp_debug_splitk_fixup(int on) { g_splitk_fixup = on ? 1 : 0; return 0; }
/* debugging aid: observations per host-to-device chunk of vggp_elbo_host (default 2^23; tests use small values) */
int vggp_debug_host_chunk(long long n) { g_host_chunk = n > 4 ? n : 4; return 0; }
int vggp_debug_fp_fast(int on) { g_fp_fast = (on & 1); g_fp_pack = (on & 2) ? 0 : ((on & 4) ? 2 : 1); return 0; }

int vggp_info_async(vggp_plan* p, int* info_pinned_host, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !info_pinned_host) return fail(VGGP_E_ARG, "null argument");
    VGGP_CUDA(cudaMemcpyAsync(info_pinned_host, p->g.info, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return 0;
}

int vggp_elbo_host(vggp_plan* p, const void* const* x_host, const void* y_host, int64_t n, const double* theta_host,
                   const double* m_host, const double* L_host, double ell_scale, double* out_host,
                   double* dtheta_host, double* dm_host, double* dL_host, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !theta_host || !m_host || !L_host || !out_host || !dtheta_host || !dm_host || !dL_host || n < 0)
        return fail(VGGP_E_ARG, "bad argument");
    if (p->family == VGGP_SVGP_MARKOV) return fail(VGGP_E_UNSUPPORTED, "the Markov SVGP family takes the binned layout (vggp_obs_bin_prepare / _pack, vggp_obs_fwd_bwd_binned)");
    if (n > 0 && (!x_host || !y_host)) return fail(VGGP_E_ARG, "null observation pointers");
    cudaStream_t st = (cudaStream_t)stream;
    const int D = p->D;
    const size_t tsz = p->obs_dtype == VGGP_F32 ? 4 : 8;
    i64 n_elems, soff, nsc, total;
    vggp_gbuf_layout(p, &n_elems, &soff, &nsc, &total);
    if (!p->st_theta) {
        VGGP_CUDA(cudaMalloc(&p->st_theta, sizeof(double) * (2 * D + 1)));
        VGGP_CUDA(cudaMalloc(&p->st_dtheta, sizeof(double) * (2 * D + 1)));
        VGGP_CUDA(cudaMalloc(&p->st_out, sizeof(double) * 4));
        VGGP_CUDA(cudaMalloc(&p->st_m, sizeof(double) * p->M));
        VGGP_CUDA(cudaMalloc(&p->st_dm, sizeof(double) * p->M));
        VGGP_CUDA(cudaMalloc(&p->st_L, sizeof(double) * p->Lsize));
        VGGP_CUDA(cudaMalloc(&p->st_dL, sizeof(double) * p->Lsize));
        VGGP_CUDA(cudaMalloc(&p->st_gbuf, (size_t)total));
    }
    if (n > p->st_n) {
        if (p->st_x) cudaFree(p->st_x);
        if (p->st_y) cudaFree(p->st_y);
        p->st_x = p->st_y = nullptr; p->st_n = 0;
        VGGP_CUDA(cudaMalloc(&p->st_x, tsz * (size_t)n * D));
        VGGP_CUDA(cudaMalloc(&p->st_y, tsz * (size_t)n));
        p->st_n = n;
    }
    // parameters first (6 MB at 512^2), so that the grid-side forward runs while the observations are still on their way
    VGGP_CUDA(cudaMemcpyAsync(p->st_theta, theta_host, sizeof(double) * (2 * D + 1), cudaMemcpyHostToDevice, st));
    VGGP_CUDA(cudaMemcpyAsync(p->st_m, m_host, sizeof(double) * p->M, cudaMemcpyHostToDevice, st));
    VGGP_CUDA(cudaMemcpyAsync(p->st_L, L_host, sizeof(double) * p->Lsize, cudaMemcpyHostToDevice, st));
    int rc;
    if ((rc = vggp_grid_forward(p, p->st_theta, p->st_m, p->st_L, stream))) return rc;
    // The observations cross PCIe in chunks on a second stream; the per-observation kernel of chunk c runs on `stream` as
    // soon as its copy has landed, accumulating into one gradient buffer, so only the last chunk's kernel, the backward and
    // the read-back are not hidden behind the transfer.  (B1 family; the B0 kernels take the whole shard in one call.)
    const i64 chunk_target = g_host_chunk;
    const int nchunks = (p->family == VGGP_B1_ASVGP && n > chunk_target) ? (int)std::min<i64>(32, (n + chunk_target - 1) / chunk_target) : 1;
    if (nchunks == 1) {
        const void* xdev[VGGP_MAX_D] = {nullptr, nullptr, nullptr};
        for (int d = 0; d < D && n > 0; ++d) {
            unsigned char* dst = reinterpret_cast<unsigned char*>(p->st_x) + (size_t)d * n * tsz;
            VGGP_CUDA(cudaMemcpyAsync(dst, x_host[d], tsz * (size_t)n, cudaMemcpyHostToDevice, st));
            xdev[d] = dst;
        }
        if (n > 0) VGGP_CUDA(cudaMemcpyAsync(p->st_y, y_host, tsz * (size_t)n, cudaMemcpyHostToDevice, st));
        if ((rc = vggp_obs_fwd_bwd(p, xdev, p->st_y, n, p->st_gbuf, stream))) return rc;
    } else {
        if (!p->st_copy) VGGP_CUDA(cudaStreamCreateWithFlags(&p->st_copy, cudaStreamNonBlocking));
        while ((int)p->st_ev.size() < nchunks + 1) {
            cudaEvent_t e;
            VGGP_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            p->st_ev.push_back(e);
        }
        // the copy stream starts after whatever `stream` already holds (earlier users of the staging buffers)
        VGGP_CUDA(cudaEventRecord(p->st_ev[nchunks], st));
        VGGP_CUDA(cudaStreamWaitEvent(p->st_copy, p->st_ev[nchunks], 0));
        VGGP_CUDA(cudaMemsetAsync(p->st_gbuf, 0, (size_t)total, st));
        const i64 per = ((n + nchunks - 1) / nchunks + 3) / 4 * 4;
        const PackGeom g = pack_geometry(p, per);
        if (g.n_packed > p->pk_cap) {
            VGGP_CUDA(cudaStreamSynchronize(st));
            for (int d = 0; d < D; ++d) { if (p->pk_x[d]) cudaFree(p->pk_x[d]); p->pk_x[d] = nullptr; }
            if (p->pk_y) cudaFree(p->pk_y);
            p->pk_y = nullptr; p->pk_cap = 0;
            for (int d = 0; d < D; ++d) VGGP_CUDA(cudaMalloc(&p->pk_x[d], tsz * (size_t)g.n_packed));
            VGGP_CUDA(cudaMalloc(&p->pk_y, tsz * (size_t)g.n_packed));
            p->pk_cap = g.n_packed;
        }
        for (int c = 0; c < nchunks; ++c) {
            const i64 lo = (i64)c * per, hi = std::min<i64>(n, lo + per);
            if (lo >= hi) break;
            const void* xdev[VGGP_MAX_D] = {nullptr, nullptr, nullptr};
            for (int d = 0; d < D; ++d) {
                unsigned char* dst = reinterpret_cast<unsigned char*>(p->st_x) + ((size_t)d * n + lo) * tsz;
                VGGP_CUDA(cudaMemcpyAsync(dst, reinterpret_cast<const unsigned char*>(x_host[d]) + lo * tsz, tsz * (size_t)(hi - lo),
                                          cudaMemcpyHostToDevice, p->st_copy));
                xdev[d] = dst;
            }
            unsigned char* ydst = reinterpret_cast<unsigned char*>(p->st_y) + lo * tsz;
            VGGP_CUDA(cudaMemcpyAsync(ydst, reinterpret_cast<const unsigned char*>(y_host) + lo * tsz, tsz * (size_t)(hi - lo),
                                      cudaMemcpyHostToDevice, p->st_copy));
            VGGP_CUDA(cudaEventRecord(p->st_ev[c], p->st_copy));
            VGGP_CUDA(cudaStreamWaitEvent(st, p->st_ev[c], 0));
            if ((rc = vggp_obs_pack(p, xdev, ydst, hi - lo, 0, p->pk_x, p->pk_y, stream))) return rc;
            p->n_real_override = (double)n;                    // every launch stores the shard's count, not its chunk's
            rc = obs_packed_dispatch(p, p->pk_x, p->pk_y, hi - lo, p->st_gbuf, st);        // accumulates: no memset
            p->n_real_override = -1.0;
            if (rc) return rc;
        }
    }
    if ((rc = vggp_grid_backward(p, p->st_theta, p->st_m, p->st_L, p->st_gbuf, ell_scale, p->st_out, p->st_dtheta,
                                 p->st_dm, p->st_dL, stream))) return rc;
    VGGP_CUDA(cudaMemcpyAsync(out_host, p->st_out, sizeof(double) * 4, cudaMemcpyDeviceToHost, st));
    VGGP_CUDA(cudaMemcpyAsync(dtheta_host, p->st_dtheta, sizeof(double) * (2 * D + 1), cudaMemcpyDeviceToHost, st));
    VGGP_CUDA(cudaMemcpyAsync(dm_host, p->st_dm, sizeof(double) * p->M, cudaMemcpyDeviceToHost, st));
    VGGP_CUDA(cudaMemcpyAsync(dL_host, p->st_dL, sizeof(double) * p->Lsize, cudaMemcpyDeviceToHost, st));
    VGGP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int vggp_b1_stencil(const vggp_plan* p, int dim, const void* x, int64_t n, int32_t* c, void* w_lo, void* w_hi,
                    void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || dim < 0 || dim >= p->D || n < 0) return fail(VGGP_E_ARG, "bad argument");
    if (n == 0) return 0;
    if (!x || !c || !w_lo || !w_hi) return fail(VGGP_E_ARG, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = (int)std::min<i64>((n + 255) / 256, 148 * 8);
    if (p->obs_dtype == VGGP_F32)
        k_b1_stencil<float><<<blocks, 256, 0, st>>>(p->mesh[dim], (const float*)x, n, c, (float*)w_lo, (float*)w_hi);
    else
        k_b1_stencil<double><<<blocks, 256, 0, st>>>(p->mesh[dim], (const double*)x, n, c, (double*)w_lo, (double*)w_hi);
    VGGP_LAUNCH_CHECK();
    return 0;
}

int vggp_features_dense(const vggp_plan* p, int dim, const void* x, int64_t n, const double* theta, void* phi,
                        void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || dim < 0 || dim >= p->D || n < 0) return fail(VGGP_E_ARG, "bad argument");
    if (n == 0) return 0;
    if (!x || !phi) return fail(VGGP_E_ARG, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t tsz = p->obs_dtype == VGGP_F32 ? 4 : 8;
    if (p->family == VGGP_B1_ASVGP) {
        VGGP_CUDA(cudaMemsetAsync(phi, 0, tsz * (size_t)n * p->n[dim], st));
        const int blocks = (int)std::min<i64>((n + 255) / 256, 148 * 8);
        if (p->obs_dtype == VGGP_F32) k_b1_dense<float><<<blocks, 256, 0, st>>>(p->mesh[dim], (const float*)x, n, (float*)phi);
        else k_b1_dense<double><<<blocks, 256, 0, st>>>(p->mesh[dim], (const double*)x, n, (double*)phi);
    } else {
        if (!theta) return fail(VGGP_E_ARG, "theta required for the B0 family");
        double th[2 * VGGP_MAX_D + 1];
        VGGP_CUDA(cudaMemcpyAsync(th, theta, sizeof(double) * (2 * p->D + 1), cudaMemcpyDeviceToHost, st));
        VGGP_CUDA(cudaStreamSynchronize(st));
        dim3 grid(ceil_div(n, 256), p->n[dim]);
        if (p->family == VGGP_VFF_GRID) {
            if (p->obs_dtype == VGGP_F32) k_vff_dense<float><<<grid, 256, 0, st>>>(p->mesh[dim], (const float*)x, n, th[dim], (float*)phi);
            else k_vff_dense<double><<<grid, 256, 0, st>>>(p->mesh[dim], (const double*)x, n, th[dim], (double*)phi);
        } else if (p->family == VGGP_SVGP_GRID || p->family == VGGP_SVGP_MARKOV) {     // the dense k_d(Z, x)
            if (p->obs_dtype == VGGP_F32)
                k_svgp_dense<float><<<grid, 256, 0, st>>>(p->mesh[dim], (const float*)x, n, th[dim], th[p->D + dim], (float*)phi);
            else
                k_svgp_dense<double><<<grid, 256, 0, st>>>(p->mesh[dim], (const double*)x, n, th[dim], th[p->D + dim], (double*)phi);
        } else if (p->obs_dtype == VGGP_F32)
            k_b0_dense<float><<<grid, 256, 0, st>>>(p->mesh[dim], (const float*)x, n, th[dim], th[p->D + dim], (float*)phi);
        else
            k_b0_dense<double><<<grid, 256, 0, st>>>(p->mesh[dim], (const double*)x, n, th[dim], th[p->D + dim], (double*)phi);
    }
    VGGP_LAUNCH_CHECK();
    return 0;
}

int vggp_predict(vggp_plan* p, const void* const* x, int64_t n, void* mean, void* var, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || n < 0) return fail(VGGP_E_ARG, "bad argument");
    if (n == 0) return 0;
    if (!x || !mean || !var) return fail(VGGP_E_ARG, "null argument");
    for (int d = 0; d < p->D; ++d)
        if (!x[d]) return fail(VGGP_E_ARG, "null test-point pointer");
    if (p->family == VGGP_SVGP_MARKOV)      // Markov form, O(1) per point (svgpm.cuh)
        return predict_svgpm_dispatch(p, x, nullptr, n, mean, var, nullptr, (cudaStream_t)stream);
    if (p->family >= VGGP_SVGP_GRID)
        return fail(VGGP_E_UNSUPPORTED, "SVGP / VFF families: predictions are assembled from vggp_features_dense by the host mirror");
    if (p->family != VGGP_B1_ASVGP)      // B0 family: scan form, O(1) per point (b0scan.cuh)
        return predict_b0s_dispatch(p, x, n, mean, var, (cudaStream_t)stream);
    return predict_dispatch(p, x, n, mean, var, (cudaStream_t)stream);
}

int vggp_meanopt_assemble(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !desc) return fail(VGGP_E_ARG, "null argument");
    if (p->family != VGGP_B1_ASVGP && p->family != VGGP_SVGP_MARKOV)
        return fail(VGGP_E_UNSUPPORTED, "the optimal mean is built for the B1 and VGGP_SVGP_MARKOV families (3^D-stencil system)");
    if (desc->D != p->D || desc->n_tasks < 0 || (desc->n_tasks > 0 && !binned))
        return fail(VGGP_E_ARG, "binned buffer does not match the plan");
    cudaStream_t st = (cudaStream_t)stream;
    if (!p->mo_buf) {
        const size_t want = mo_layout(p).bytes;
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusActive)
            return fail(VGGP_E_UNSUPPORTED, "the first vggp_meanopt_assemble allocates: call it outside a stream capture");
        VGGP_CUDA(cudaMalloc(&p->mo_buf, want));
        p->mo_bytes = want;
    }
    p->mo_assembled = false;
    p->mo_solved = false;
    if (int rc = mo_assemble_dispatch(p, desc, binned, st)) return rc;
    p->mo_set[0] = desc->n; p->mo_set[1] = desc->n_tasks; p->mo_set[2] = desc->data_elems;
    p->mo_assembled = true;
    return 0;
}

int vggp_meanopt_solve(vggp_plan* p, double rtol, int max_iter, double* m_out, int* iters_host, double* relres_host,
                       void* stream) {
    return vggp_meanopt_solve_pc(p, VGGP_MEANOPT_JACOBI, rtol, max_iter, m_out, iters_host, relres_host, stream);
}

int vggp_meanopt_solve_pc(vggp_plan* p, int precond, double rtol, int max_iter, double* m_out, int* iters_host,
                          double* relres_host, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !m_out || !iters_host || !relres_host) return fail(VGGP_E_ARG, "null argument");
    if (p->family != VGGP_B1_ASVGP && p->family != VGGP_SVGP_MARKOV)
        return fail(VGGP_E_UNSUPPORTED, "the optimal mean is built for the B1 and VGGP_SVGP_MARKOV families (3^D-stencil system)");
    if (!(rtol >= 0.0) || max_iter < 0) return fail(VGGP_E_ARG, "rtol must be >= 0 and max_iter >= 0");
    if (precond != VGGP_MEANOPT_JACOBI && precond != VGGP_MEANOPT_KRONECKER)
        return fail(VGGP_E_ARG, "precond must be VGGP_MEANOPT_JACOBI or VGGP_MEANOPT_KRONECKER");
    if (!p->mo_assembled) return fail(VGGP_E_ARG, "vggp_meanopt_solve needs a previous vggp_meanopt_assemble on this plan");
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    switch (p->D) {
        case 1: rc = mo_solve_impl<1>(p, precond, rtol, max_iter, m_out, iters_host, relres_host, st); break;
        case 2: rc = mo_solve_impl<2>(p, precond, rtol, max_iter, m_out, iters_host, relres_host, st); break;
        default: rc = mo_solve_impl<3>(p, precond, rtol, max_iter, m_out, iters_host, relres_host, st); break;
    }
    p->mo_solved = rc == 0;
    return rc;
}

int vggp_logdet_system(vggp_plan* p, int precond, int probe_kind, int n_probes, uint64_t seed_or_first, int max_steps,
                       double rtol, double* out_host, double* per_probe_host, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !out_host) return fail(VGGP_E_ARG, "null argument");
    if (p->family != VGGP_B1_ASVGP && p->family != VGGP_SVGP_MARKOV)
        return fail(VGGP_E_UNSUPPORTED, "the collapsed ELBO is built for the B1 and VGGP_SVGP_MARKOV families (3^D-stencil system)");
    if (precond != VGGP_MEANOPT_JACOBI && precond != VGGP_MEANOPT_KRONECKER)
        return fail(VGGP_E_ARG, "precond must be VGGP_MEANOPT_JACOBI or VGGP_MEANOPT_KRONECKER");
    if (probe_kind != VGGP_PROBE_RADEMACHER && probe_kind != VGGP_PROBE_UNIT)
        return fail(VGGP_E_ARG, "probe_kind must be VGGP_PROBE_RADEMACHER or VGGP_PROBE_UNIT");
    if (n_probes < 1 || n_probes > VGGP_MAX_PROBES || max_steps < 1 || !(rtol >= 0.0))
        return fail(VGGP_E_ARG, "1 <= n_probes <= VGGP_MAX_PROBES, max_steps >= 1 and rtol >= 0");
    if (probe_kind == VGGP_PROBE_UNIT && (seed_or_first >= (uint64_t)p->M || (uint64_t)n_probes > (uint64_t)p->M - seed_or_first))
        return fail(VGGP_E_ARG, "unit probes e_first .. e_{first + n_probes - 1} must lie below M");
    if (!p->mo_assembled) return fail(VGGP_E_ARG, "vggp_logdet_system needs a previous vggp_meanopt_assemble on this plan");
    cudaStream_t st = (cudaStream_t)stream;
    switch (p->D) {
        case 1: return ct_logdet_impl<1>(p, precond, probe_kind, n_probes, seed_or_first, max_steps, rtol, out_host, per_probe_host, st);
        case 2: return ct_logdet_impl<2>(p, precond, probe_kind, n_probes, seed_or_first, max_steps, rtol, out_host, per_probe_host, st);
        default: return ct_logdet_impl<3>(p, precond, probe_kind, n_probes, seed_or_first, max_steps, rtol, out_host, per_probe_host, st);
    }
}

int vggp_collapsed_terms(vggp_plan* p, const vggp_binned_desc* desc, const void* binned, double* out, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !desc || !out) return fail(VGGP_E_ARG, "null argument");
    if (p->family != VGGP_B1_ASVGP && p->family != VGGP_SVGP_MARKOV)
        return fail(VGGP_E_UNSUPPORTED, "the collapsed ELBO is built for the B1 and VGGP_SVGP_MARKOV families (3^D-stencil system)");
    if (desc->D != p->D || desc->n_tasks < 0 || (desc->n_tasks > 0 && !binned) || (desc->n_inside < desc->n && !binned))
        return fail(VGGP_E_ARG, "binned buffer does not match the plan");
    if (!p->mo_assembled) return fail(VGGP_E_ARG, "vggp_collapsed_terms needs a previous vggp_meanopt_assemble on this plan");
    if (!p->mo_solved)
        return fail(VGGP_E_ARG, "vggp_collapsed_terms needs a vggp_meanopt_solve on the current assembly after the last "
                                "vggp_grid_forward");
    if (desc->n != p->mo_set[0] || desc->n_tasks != p->mo_set[1] || desc->data_elems != p->mo_set[2])
        return fail(VGGP_E_ARG, "vggp_collapsed_terms takes the binned set given to vggp_meanopt_assemble");
    return ct_terms_dispatch(p, desc, binned, out, (cudaStream_t)stream);
}

int vggp_covopt_update(vggp_plan* p, int dim, const void* gbuf, double ell_scale, const double* L, double* L_out,
                       double* change, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !gbuf || !L || !L_out || !change) return fail(VGGP_E_ARG, "null argument");
    if (p->family != VGGP_B1_ASVGP && p->family != VGGP_SVGP_MARKOV)
        return fail(VGGP_E_UNSUPPORTED, "the optimal covariance is built for the B1 and VGGP_SVGP_MARKOV families (tridiagonal "
                                        "T_d); the dense families have the reference's dense q_u()");
    if (dim < 0 || dim >= p->D) return fail(VGGP_E_ARG, "bad dim");
    if (!p->forwarded) return fail(VGGP_E_ARG, "vggp_covopt_update needs a previous vggp_grid_forward on this plan");
    if (p->n[dim] > CO_MAX_N) return fail(VGGP_E_UNSUPPORTED, "vggp_covopt_update supports M_d <= 2560");
    cudaStream_t st = (cudaStream_t)stream;
    if (!p->co_buf) {
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusActive)
            return fail(VGGP_E_UNSUPPORTED, "the first vggp_covopt_update allocates: call it outside a stream capture");
        const size_t want = sizeof(double) * (6 * (size_t)p->nmax + 8);
        VGGP_CUDA(cudaMalloc(&p->co_buf, want));
        p->co_bytes = want;
    }
    if (p->obs_dtype == VGGP_F32) return covopt_impl<float>(p, dim, gbuf, ell_scale, L, L_out, change, st);
    return covopt_impl<double>(p, dim, gbuf, ell_scale, L, L_out, change, st);
}

int vggp_metrics(int dtype, const void* truth, const void* pred, int64_t n, double* out, void* stream) {
    if (!out || n < 0) return fail(VGGP_E_ARG, "bad argument");
    if (dtype != VGGP_F32 && dtype != VGGP_F64) return fail(VGGP_E_DTYPE, "dtype must be VGGP_F32 or VGGP_F64");
    cudaStream_t st = (cudaStream_t)stream;
    VGGP_CUDA(cudaMemsetAsync(out, 0, 4 * sizeof(double), st));
    if (n == 0) return 0;
    if (!truth || !pred) return fail(VGGP_E_ARG, "null argument");
    const int blocks = (int)std::min<i64>((n + 255) / 256, 148 * 8);
    if (dtype == VGGP_F32) k_metrics<float><<<blocks, 256, 0, st>>>((const float*)truth, (const float*)pred, n, out);
    else k_metrics<double><<<blocks, 256, 0, st>>>((const double*)truth, (const double*)pred, n, out);
    VGGP_LAUNCH_CHECK();
    return 0;
}

int vggp_predict_metrics(vggp_plan* p, const void* const* x, const void* y, int64_t n, double* out, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !out || n < 0) return fail(VGGP_E_ARG, "bad argument");
    if (p->family != VGGP_B1_ASVGP && p->family != VGGP_SVGP_MARKOV)
        return fail(VGGP_E_UNSUPPORTED, "fused prediction metrics are built for the B1 and Markov SVGP families");
    cudaStream_t st = (cudaStream_t)stream;
    VGGP_CUDA(cudaMemsetAsync(out, 0, 4 * sizeof(double), st));
    if (n == 0) return 0;
    if (!x || !y) return fail(VGGP_E_ARG, "null argument");
    for (int d = 0; d < p->D; ++d)
        if (!x[d]) return fail(VGGP_E_ARG, "null test-point pointer");
    if (p->family == VGGP_SVGP_MARKOV) return predict_svgpm_dispatch(p, x, y, n, nullptr, nullptr, out, st);
    return predict_metrics_dispatch(p, x, y, n, out, st);
}

int vggp_minmax(int dtype, const void* x, int64_t n, void* minmax, void* stream) {
    if (!x || !minmax || n <= 0) return fail(VGGP_E_ARG, "bad argument (n must be > 0)");
    if (dtype != VGGP_F32 && dtype != VGGP_F64) return fail(VGGP_E_DTYPE, "dtype must be VGGP_F32 or VGGP_F64");
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = (int)std::min<i64>((n + 255) / 256, 1024);
    const size_t tsz = dtype == VGGP_F32 ? 4 : 8;
    DevTemps tmp;                            // 2 values per block; setup-time call, freed after the stream has drained
    unsigned char* partial = nullptr;
    VGGP_CUDA(tmp.alloc(&partial, 2 * (size_t)blocks * tsz));
    if (dtype == VGGP_F32) {
        k_minmax_partial<float><<<blocks, 256, 0, st>>>((const float*)x, n, (float*)partial);
        VGGP_LAUNCH_CHECK();
        k_minmax_final<float><<<1, 256, 0, st>>>((const float*)partial, blocks, (float*)minmax);
    } else {
        k_minmax_partial<double><<<blocks, 256, 0, st>>>((const double*)x, n, (double*)partial);
        VGGP_LAUNCH_CHECK();
        k_minmax_final<double><<<1, 256, 0, st>>>((const double*)partial, blocks, (double*)minmax);
    }
    VGGP_LAUNCH_CHECK();
    VGGP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int vggp_minmax_scale(int dtype, const void* x, int64_t n, const void* minmax, int inverse, void* y, void* stream) {
    if (n < 0 || !minmax) return fail(VGGP_E_ARG, "bad argument");
    if (dtype != VGGP_F32 && dtype != VGGP_F64) return fail(VGGP_E_DTYPE, "dtype must be VGGP_F32 or VGGP_F64");
    if (n == 0) return 0;
    if (!x || !y) return fail(VGGP_E_ARG, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = (int)std::min<i64>((n + 255) / 256, 148 * 8);
    if (dtype == VGGP_F32) k_minmax_scale<float><<<blocks, 256, 0, st>>>((const float*)x, n, (const float*)minmax, inverse, (float*)y);
    else k_minmax_scale<double><<<blocks, 256, 0, st>>>((const double*)x, n, (const double*)minmax, inverse, (double*)y);
    VGGP_LAUNCH_CHECK();
    return 0;
}

int vggp_generate_tracks(int dtype, int D, int64_t n_total, int64_t lo, int64_t hi, int64_t seed, int passes, double gradient,
                         void* const* x, void* y, void* stream) {
    if (dtype != VGGP_F32 && dtype != VGGP_F64) return fail(VGGP_E_DTYPE, "dtype must be VGGP_F32 or VGGP_F64");
    if (D < 1 || D > VGGP_MAX_D) return fail(VGGP_E_DIM, "D must be 1..3");
    if (n_total < 1 || lo < 0 || hi < lo || hi > n_total || passes < 1 || !(gradient > 0.0)) return fail(VGGP_E_ARG, "bad argument");
    if (hi == lo) return 0;
    if (!x || !y) return fail(VGGP_E_ARG, "null argument");
    for (int d = 0; d < D; ++d)
        if (!x[d]) return fail(VGGP_E_ARG, "null coordinate pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == VGGP_F32) {
        if (D == 1) return launch_tracks<float, 1>(x, y, lo, hi, n_total, seed, passes, gradient, st);
        if (D == 2) return launch_tracks<float, 2>(x, y, lo, hi, n_total, seed, passes, gradient, st);
        return launch_tracks<float, 3>(x, y, lo, hi, n_total, seed, passes, gradient, st);
    }
    if (D == 1) return launch_tracks<double, 1>(x, y, lo, hi, n_total, seed, passes, gradient, st);
    if (D == 2) return launch_tracks<double, 2>(x, y, lo, hi, n_total, seed, passes, gradient, st);
    return launch_tracks<double, 3>(x, y, lo, hi, n_total, seed, passes, gradient, st);
}

int vggp_workspace_ptr(const vggp_plan* p, int which, int dim, double** ptr, int64_t* n_elems) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !ptr) return fail(VGGP_E_ARG, "null argument");
    if (p->family == VGGP_SVGP_MARKOV)
        return fail(VGGP_E_UNSUPPORTED, "the Markov SVGP family keeps bands and per-cell tables only: no dense workspace array");
    if (which != VGGP_WS_ALPHA && which != VGGP_WS_SCAL && (dim < 0 || dim >= p->D)) return fail(VGGP_E_ARG, "bad dim");
    const bool b1 = p->family == VGGP_B1_ASVGP;
    if (b1 && (which == VGGP_WS_K || which == VGGP_WS_Q))
        return fail(VGGP_E_UNSUPPORTED, "the B1 family has no Cholesky factor and keeps only the band of Q_d (VGGP_WS_QBAND)");
    const i64 nn = (which == VGGP_WS_ALPHA || which == VGGP_WS_SCAL) ? 0 : (i64)p->n[dim] * p->n[dim];
    switch (which) {
        case VGGP_WS_K: *ptr = p->g.Kc[dim]; if (n_elems) *n_elems = nn; return 0;
        case VGGP_WS_P:
            if (b1) {      // not materialised in a step: filled now, ordered on the stream of the last forward
                k_b1_fill_P<<<dim3(ceil_div(p->nmax, 256), p->D), 256, 0, p->last_stream>>>(p->g);
                VGGP_LAUNCH_CHECK();
            }
            *ptr = p->g.P[dim]; if (n_elems) *n_elems = nn; return 0;
        case VGGP_WS_R: *ptr = p->g.R[dim]; if (n_elems) *n_elems = nn; return 0;
        case VGGP_WS_Q: *ptr = p->g.Q[dim]; if (n_elems) *n_elems = nn; return 0;
        case VGGP_WS_S: return fail(VGGP_E_UNSUPPORTED, "S_d is no longer materialised");
        case VGGP_WS_KRAW:
            if (b1) {      // as VGGP_WS_P
                k_b1_fill_Kraw<<<dim3(ceil_div((i64)p->nmax * p->nmax, 256), p->D), 256, 0, p->last_stream>>>(p->g, p->theta_dev);
                VGGP_LAUNCH_CHECK();
            }
            *ptr = p->g.Kraw[dim]; if (n_elems) *n_elems = nn; return 0;
        case VGGP_WS_QBAND: *ptr = p->g.Qb[dim]; if (n_elems) *n_elems = 2 * (i64)p->n[dim]; return 0;
        case VGGP_WS_ALPHA: *ptr = p->alpha; if (n_elems) *n_elems = p->M; return 0;
        case VGGP_WS_SCAL: *ptr = p->g.sc; if (n_elems) *n_elems = SC_COUNT; return 0;
    }
    return fail(VGGP_E_ARG, "unknown workspace id");
}

int vggp_gemm_f64(int use_mma, int batch, int m, int n, int k, double alpha, const double* A, int64_t rsA, int64_t csA,
                  int64_t bsA, const double* B, int64_t rsB, int64_t csB, int64_t bsB, double beta, double* C,
                  int64_t rsC, int64_t csC, int64_t bsC, int splitk, void* stream) {
    if (!A || !B || !C || m < 0 || n < 0 || k < 0 || batch < 1) return fail(VGGP_E_ARG, "bad argument");
    GemmDesc d;
    gemm_desc_defaults(d);
    d.A = A; d.B = B; d.C = C; d.m = m; d.n = n; d.k = k;
    d.rsA = rsA; d.csA = csA; d.bsA = bsA; d.rsB = rsB; d.csB = csB; d.bsB = bsB; d.rsC = rsC; d.csC = csC; d.bsC = bsC;
    d.alpha = alpha; d.beta = beta; d.batch = batch; d.splitk = splitk < 1 ? 1 : splitk;
    return launch_one(d, use_mma, (cudaStream_t)stream);
}

int vggp_mode_product(vggp_plan* p, int dim, const double* A, const double* src, double* dst, void* stream) {
    DeviceGuard dev_guard(p ? p->device : -1);
    if (!p || !A || !src || !dst || dim < 0 || dim >= p->D) return fail(VGGP_E_ARG, "bad argument");
    return launch_one(mode_desc(p, dim, A, src, dst), g_use_mma, (cudaStream_t)stream, p);
}

}  // extern "C"
