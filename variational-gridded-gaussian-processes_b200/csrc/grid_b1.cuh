// Fused grid side of the B1 (ASVGP) family: the whole replicated part of a step in a handful of launches.
//
// The per-dimension factor K_d of this family is tridiagonal (gridded_kronecker_structure.py:731-780), so P_d = K_d^-1 is
// semiseparable and every product with it is a pair of first-order recurrences along a fibre.  Round 1 ran those as 14
// dependent small launches (0.2 ms per step: the Amdahl term of the multi-GPU run).  Here
//   k_b1_gens     pivots of the twisted factorisation by a chunk-parallel scan (2 x 2 Moebius composition for the chunk
//                 carries, the plain recurrence inside a chunk), generators, log det K_d, the P-band tables
//   k_fibre_pass  ONE engine for every product with P_d: a CTA stages a tile of F fibres in shared memory (coalesced for
//                 strided and for contiguous modes), one warp per fibre runs the two recurrences (lane-local sweeps + a
//                 5-step affine scan across lanes), and a kind-specific prologue / epilogue fuses what round 1 did in
//                 separate elementwise kernels (tril mask, casts, <m, alpha>, g / ghat from the gradient buffer, band
//                 scatter, dR from R, tril / diagonal terms of dL, band dot products for dK)
//   k_b1_theta    band of P_d X_d P_d by two first-order recurrences, band of dK_d -> d theta, ELBO scalars
// A step is: gens, pass F1 (R_d = P_d tril L_d, first mode of alpha), pass F2 (last mode of alpha + casts + row reductions
// of R_d), the per-observation kernel, pass B1 (last mode of (kron P) g, A_e), pass B2 (first mode, dL), theta (which also
// forms the band of P X P by O(n) recurrences): 6 launches for D = 2 (one more forward and backward pass for D = 3).
// This is the only grid side of the family; the reference it is tested against is the float64 oracle (oracle/vggp_oracle.py).
// Maths: SURVEY.md appendix A.
#pragma once
#include "grid.cuh"

namespace vggp {

constexpr int FP_THREADS = 256;
constexpr int FP_WARPS = FP_THREADS / 32;
constexpr int FP_MAX_TASKS = 14;
constexpr int GEN_CHUNK = 32;            // pivots per thread in k_b1_gens
constexpr int GEN_THREADS = 256;
// deterministic mode: what one CTA of a fibre pass leaves for k_fp_det_reduce (grid_b1_fast.cuh)
constexpr int FP_DET_BAND = 0;                     // [3][512] band partials (dl + 1, i)
constexpr int FP_DET_MALPHA = 3 * 512;             // <m, alpha> partial
constexpr int FP_DET_TR = FP_DET_MALPHA + 1;       // [FP_WARPS] tr terms of the rows of a QROW tile
constexpr int FP_DET_LOGDET = FP_DET_TR + 8;       // [FP_WARPS] log det terms
constexpr int FP_DET_SLOT = FP_DET_LOGDET + 8;

enum FpKind {
    FP_R = 0,       // R_d = P_d tril(L_d): column k of tril(L_d) -> column k of R_d
    FP_PROD,        // dst = src x_e P_e
    FP_ALPHA,       // alpha = src x_e P_e, + cast to the observation dtype + <m, alpha>
    FP_GA,          // g = c galpha, ghat = g - m / 2 from the gradient buffer; V = g x_e P_e (or dm = V - alpha), A_e = ghat x_e P_e
                    // is only contracted: acc_e[i][i + dl] += sum_rest A_e[.. i ..] alpha[.. i + dl ..]
    FP_GAONLY,      // the A_e contraction alone (modes other than the one the dm chain starts with)
    FP_DM,          // dm = src x_e P_e - alpha
    FP_DL,          // column k of dR_d = 2 cQ tridiag(bq) R_d -> dLraw = P_d dR; dL = tril(dLraw - c_d R + (M/M_d) diag(1/L_ii));
                    // acc_d[i][i + dl] += dLraw[i][k] R[i + dl][k]
    FP_QROW         // no product: row reductions of R_d (band of Q_d, tr(P_d S_d), log det S_d, Q-band tables)
};

struct FpTask {
    int kind, d, n, F;            // d: dimension whose P_d is applied; n = M_d; F = fibres of one tile (in shared memory)
    i64 inner, nfib;              // fibre f = (o, r): element i at (o n + i) inner + r; nfib = outer * inner
    int tile0, ntiles;
    const double* s0;             // PROD / ALPHA / DM: source tensor;  R / DL: L_d resp. R_d;  GA*: m
    const double* s1;             // ALPHA: m;  GA / GAONLY / DM: alpha;  DL: L_d
    double* o0;                   // PROD / ALPHA / R: destination;  GA: V (or dm when `direct`);  DM: dm;  DL: dL
    const void* t0;               // GA*: galpha;  DL: band sums of dimension d [bp_d | bp_o | bq_d | bq_o] (obs dtype)
    void* t1;                     // ALPHA: alpha in the observation dtype
    int direct;                   // GA with D == 1: o0 receives dm = V - alpha
    int pk;                       // k_fibre_pass_fast only: a 512-slot row of the tile holds 2^pk fibres (mode-product kinds, M_d <= 256)
};

struct FpPass {
    FpTask t[FP_MAX_TASKS];
    int ntasks;
    int D, obs_f32;
    i64 M;
    double ell_scale;
    const double* theta;
    double* gen[VGGP_MAX_D];      // generators of P_d: [pd | ru | rl], n each
    double* acc[VGGP_MAX_D];      // band accumulators of dK_d: [3][n], slot (dl + 1, i) = W[i][i + dl]
    double* sc;                   // SC_* scalars
    double* Qb[VGGP_MAX_D];
    void* bandT;                  // per-cell tables (obs dtype)
    int tab_off[VGGP_MAX_D];
    double* det;                  // deterministic mode: per-CTA partials [FP_DET_SLOT] instead of atomics (summed by k_fp_det_reduce), or null
    long long* dbg;               // optional phase stamps (tools/gpu_phase_stamps.py): [tile][8] of clock64 / globaltimer, or null
};

// ---------------------------------------------------------------------------------------------------------
// Generators.  Top-down pivots d_k = a_k - b_{k-1}^2 / d_{k-1} and bottom-up pivots e_k = a_k - b_k^2 / e_{k+1} are
// Moebius maps of the previous pivot; a chunk of GEN_CHUNK of them composes to one 2 x 2 matrix (entries are minors of
// K_d, rescaled by exact powers of two), a single thread chains the 2 x n/GEN_CHUNK carries, and every chunk then runs the
// plain recurrence from its carry -- which contracts the (already small) error of the carry.  512 pivots: 3 x 32
// dependent steps instead of 512.
// grid (D), GEN_THREADS threads, dynamic smem 4 (n + n / 32 + 1) doubles.
// ---------------------------------------------------------------------------------------------------------
struct Mob { double a, b, c, d; };     // x -> (a x + b) / (c x + d)

// 2^-e for the binary exponent e of |x| (x normal, non-zero): an exact scaling that brings x into [1, 2)
__device__ __forceinline__ double pow2_inv_scale(double x) {
    const int e = (__double2hiint(x) >> 20) & 0x7ff;
    return __hiloint2double((2046 - e) << 20, 0);
}
__device__ __forceinline__ void mob_rescale(Mob& m) {
    const double sc = pow2_inv_scale(fmax(fmax(fabs(m.a), fabs(m.b)), fmax(fabs(m.c), fabs(m.d))));
    m.a *= sc; m.b *= sc; m.c *= sc; m.d *= sc;
}
// apply x -> p - q / x after m:  (p (a x + b) - q (c x + d)) / (a x + b)
__device__ __forceinline__ void mob_push(Mob& m, double p, double q) {
    const double na = fma(p, m.a, -q * m.c), nb = fma(p, m.b, -q * m.d);
    m.c = m.a; m.d = m.b; m.a = na; m.b = nb;
}

// The factor of this family is Toeplitz apart from its two corner entries (one knot spacing delta32 for the whole matrix,
// as in the reference): three numbers describe it.
struct B1Coef { double a_in, a_bd, b; };      // interior diagonal, corner diagonal, off-diagonal
__device__ __forceinline__ B1Coef b1_coef(const GridDims& g, const double* theta, int d) {
    B1Coef c;
    const int n = g.n[d];
    c.a_bd = factor_entry(g, theta, d, 0, 0);
    c.a_in = factor_entry(g, theta, d, 1, 1);
    c.b = factor_entry(g, theta, d, 0, 1);
    if (n < 3) c.a_in = c.a_bd;
    return c;
}

template <typename T>
__global__ void __launch_bounds__(GEN_THREADS) k_b1_gens(const __grid_constant__ GridDims g, const double* __restrict__ theta,
                                                         double* __restrict__ acc_all, int acc_total,
                                                         double* __restrict__ theta_copy) {
    extern __shared__ double sm[];
    __shared__ double red[32];
    __shared__ double carry_d[GEN_THREADS], carry_e[GEN_THREADS];
    __shared__ Mob comp_d[GEN_THREADS / 2], comp_e[GEN_THREADS / 2];
    __shared__ int bad_flag;
    const int d = blockIdx.x;
    const int n = g.n[d];
    const int tid = threadIdx.x;
    // position of pivot k: one pad slot per chunk, so that the chunk-strided accesses of the sweeps (thread = chunk) spread
    // over the banks
    auto G = [](int k) { return k + (k >> 5); };
    const int npad = n + (n >> 5) + 1;
    double* dd = sm;                 // top-down pivots, later ru
    double* ee = dd + npad;          // bottom-up pivots
    double* rd = ee + npad;          // 1 / dd
    double* re = rd + npad;          // 1 / ee
    if (tid == 0) bad_flag = 0;
    if (d == 0) {
        if (tid < SC_COUNT) g.sc[tid] = 0.0;
        if (tid == 0) *g.info = 0;
        if (tid < 2 * g.D + 1) theta_copy[tid] = theta[tid];       // the plan's copy of theta (features / predictions read it)
    }
    // the band accumulators of every dimension are cleared here, at the start of the step
    for (int i = (int)blockIdx.x * GEN_THREADS + tid; i < acc_total; i += (int)gridDim.x * GEN_THREADS) acc_all[i] = 0.0;
    const B1Coef cf = b1_coef(g, theta, d);
    const double b2 = cf.b * cf.b;
    auto diag = [&](int k) { return (k == 0 || k == n - 1) ? cf.a_bd : cf.a_in; };
    const int nch = (n + GEN_CHUNK - 1) / GEN_CHUNK;      // <= GEN_THREADS / 2 (n <= 2560: 80 chunks)
    // threads [0, nch): top-down chunk composites; threads [128, 128 + nch): bottom-up
    const bool up = tid >= GEN_THREADS / 2;
    const int ch = up ? tid - GEN_THREADS / 2 : tid;
    if (ch < nch) {
        Mob m = {1.0, 0.0, 0.0, 1.0};
        const int k0 = ch * GEN_CHUNK, k1 = min(n, k0 + GEN_CHUNK);
        if (!up) {
            // chunk covers k in [k0, k1); maps d_{k0 - 1} -> d_{k1 - 1}
            for (int k = max(k0, 1); k < k1; ++k) {
                mob_push(m, diag(k), b2);
                if ((k & 7) == 7) mob_rescale(m);
            }
            mob_rescale(m);            // entries in [1, 2): the serial chain below cannot overflow between its own rescalings
            comp_d[ch] = m;
        } else {
            // chunk covers k in [k0, k1) walked downwards; maps e_{k1} -> e_{k0}
            for (int k = min(k1 - 1, n - 2); k >= k0; --k) {
                mob_push(m, diag(k), b2);
                if ((k & 7) == 0) mob_rescale(m);
            }
            mob_rescale(m);
            comp_e[ch] = m;
        }
    }
    __syncthreads();
    // the carries are chained in homogeneous coordinates x = num / den (no division on the serial path; exact power-of-two
    // rescaling), every chunk divides its own carry afterwards
    if (tid == 0) {
        double num = cf.a_bd, den = 1.0;                   // d_0; chunk 0's composite starts from it
        for (int c = 0; c < nch; ++c) {
            carry_d[c] = num; carry_d[GEN_THREADS / 2 + c] = den;    // value entering chunk c (d_{k0 - 1}; for c = 0: d_0 itself)
            const Mob m = comp_d[c];
            const double nn = fma(m.a, num, m.b * den), dn = fma(m.c, num, m.d * den);
            const double sc = pow2_inv_scale(fmax(fabs(nn), fabs(dn)));
            num = nn * sc; den = dn * sc;
        }
    } else if (tid == 32) {
        double num = cf.a_bd, den = 1.0;                   // e_{n-1}
        for (int c = nch - 1; c >= 0; --c) {
            carry_e[c] = num; carry_e[GEN_THREADS / 2 + c] = den;    // value entering chunk c from above (e_{k1}; top chunk: e_{n-1})
            const Mob m = comp_e[c];
            const double nn = fma(m.a, num, m.b * den), dn = fma(m.c, num, m.d * den);
            const double sc = pow2_inv_scale(fmax(fabs(nn), fabs(dn)));
            num = nn * sc; den = dn * sc;
        }
    }
    __syncthreads();
    // plain recurrences inside the chunks.  1 / pivot is carried along by one Newton step from the previous reciprocal
    // (the pivots change slowly) with an exact division whenever the residual is not at rounding level; the reciprocals
    // are kept: the generators need them.
    if (ch < nch) {
        const int k0 = ch * GEN_CHUNK, k1 = min(n, k0 + GEN_CHUNK);
        bool bad = false;
        if (!up) {
            double prev = carry_d[ch] / carry_d[GEN_THREADS / 2 + ch];
            double r = 1.0 / prev;
            int k = k0;
            if (ch == 0) { dd[G(0)] = prev; rd[G(0)] = r; bad = !(prev > 0.0); k = 1; }
            for (; k < k1; ++k) {
                const double nxt = fma(-b2, r, diag(k));
                bad = bad || !(nxt > 0.0);
                double e = fma(-nxt, r, 1.0);
                double rn = fma(r, e, r);
                e = fma(-nxt, rn, 1.0);
                if (!(fabs(e) < 3e-16)) rn = 1.0 / nxt;
                r = rn;
                dd[G(k)] = nxt; rd[G(k)] = r;
            }
        } else {
            double nxt = carry_e[ch] / carry_e[GEN_THREADS / 2 + ch];
            double r = 1.0 / nxt;
            int k = k1 - 1;
            if (k1 == n) { ee[G(n - 1)] = nxt; re[G(n - 1)] = r; bad = !(nxt > 0.0); k = n - 2; }
            for (; k >= k0; --k) {
                const double cur = fma(-b2, r, diag(k));
                bad = bad || !(cur > 0.0);
                double e = fma(-cur, r, 1.0);
                double rn = fma(r, e, r);
                e = fma(-cur, rn, 1.0);
                if (!(fabs(e) < 3e-16)) rn = 1.0 / cur;
                r = rn;
                ee[G(k)] = cur; re[G(k)] = r;
            }
        }
        if (bad) bad_flag = 1;
    }
    __syncthreads();
    if (tid == 0 && bad_flag) atomicMax(g.info, d + 1);
    double* gen = g.gen[d];
    double prod = 1.0;
    double ld = 0.0;
    for (int i = tid; i < n; i += GEN_THREADS) {
        const double di = dd[G(i)];
        const double pdv = 1.0 / (di + ee[G(i)] - diag(i));
        const double ruv = (i + 1 < n) ? -cf.b * rd[G(i)] : 0.0;
        const double rlv = (i + 1 < n) ? -cf.b * re[G(i + 1)] : 0.0;
        gen[i] = pdv; gen[n + i] = ruv; gen[2 * n + i] = rlv;
        ee[G(i)] = pdv; dd[G(i)] = ruv;          // reuse (only this thread reads dd[G(i)], ee[G(i)] above): ee = pd, dd = ru for the tables
        prod *= di;                        // log det K_d = sum log d_k: one log per thread
        if (prod > 1e200 || prod < 1e-200) { ld += log(prod); prod = 1.0; }
    }
    ld += log(prod);
    __syncthreads();
    // per-cell tables of the band of P_d, monomial basis in the hat weight (same as k_fwd_reduce)
    T* tab = reinterpret_cast<T*>(g.bandT) + g.tab_off[d];
    for (int i = tid; i < n; i += GEN_THREADS) {
        const bool last = (i + 1 >= n);
        const double A = ee[G(i)];
        const double B2 = last ? 0.0 : 2.0 * ee[G(i + 1)] * dd[G(i)];        // 2 P[i][i+1] = 2 pd[i+1] ru[i]
        const double Cc = last ? 0.0 : ee[G(i + 1)];
        tab[i] = (T)A; tab[n + i] = (T)(B2 - 2.0 * A); tab[2 * n + i] = (T)(A - B2 + Cc);
    }
    ld = block_sum(ld, red);
    if (tid == 0) g.sc[SC_LOGDETK + d] = ld;
}

// ---------------------------------------------------------------------------------------------------------
// The fibre engine.
// Shared memory (dynamic):  [pd | ru | rl] padded, then tile arrays X (source -> result), C (auxiliary fibres), U (upper
// sweep values, only when a lane owns more than 16 elements), then F fibre bases.
// Padded index of element i of a fibre: i + i / S, S = ceil(n / 32) elements per lane (lane l owns [l S, (l+1) S)); the
// extra slot per lane makes the lane-strided accesses of the sweeps conflict-free.
// ---------------------------------------------------------------------------------------------------------
struct FpGeom {
    int n, S, pitch;     // pitch of one fibre in shared memory (doubles)
    unsigned magic;      // ceil(2^32 / S): i / S == umulhi(i, magic) for 0 <= i < 2^16
};
__host__ __device__ inline FpGeom fp_geom(int n) {
    FpGeom q;
    q.n = n;
    q.S = (n + 31) / 32;
    int len = n + (n + q.S - 1) / q.S + 1;
    if (len < 32 * (q.S + 1) + 16) len = 32 * (q.S + 1) + 16;      // every lane may read 16 slots from its segment start
    len = (len + 15) / 16 * 16 + 2;            // consecutive fibres start 2 banks (of 8 bytes) apart: transposed stores spread
    q.pitch = len;
    q.magic = (unsigned)((0x100000000ull + (unsigned long long)q.S - 1) / (unsigned long long)q.S);
    return q;
}
__host__ __device__ inline size_t fp_smem_bytes(int n, int F, bool aux) {
    const FpGeom q = fp_geom(n);
    const int narr = 1 + (aux ? 1 : 0) + (q.S > 16 ? 1 : 0);
    return sizeof(double) * ((size_t)5 * q.pitch + (size_t)narr * F * q.pitch);      // [pd | ru | rl | bq_diag | bq_off] + tiles
}
// padded index; `SM` = FpGeom::magic (S == 1 gives magic 2^32, which does not fit: n <= 32 is handled by the S == 1 branch)
__device__ __forceinline__ int fp_pidx(int i, unsigned SM) { return SM ? i + (int)__umulhi((unsigned)i, SM) : 2 * i; }

__host__ __device__ inline bool fp_kind_has_aux(int kind) { return kind == FP_GA || kind == FP_GAONLY || kind == FP_DL; }

// one warp, one fibre: X holds x_i on entry and y_i = (P x)_i on exit
__device__ __forceinline__ void fp_fibre(const FpGeom& q, const double* __restrict__ pd, const double* __restrict__ ru,
                                         const double* __restrict__ rl, double* __restrict__ X, double* __restrict__ U, int lane) {
    const int S = q.S, n = q.n;
    const int i0 = lane * S;
    const int cnt = max(0, min(S, n - i0));
    const int p0 = lane * (S + 1);
    // phase 1: affine summaries of the lane's segment for both sweeps.  Up to 16 elements per lane (n <= 512) live in
    // registers and the loops are fully unrolled, so the shared-memory loads are issued ahead of the dependent chains.
    double lA = 1.0, lB = 0.0, uA = 1.0, uB = 0.0;
    double sv[16];
    if (S <= 16) {
        // straight-line code: every shared-memory load is unconditional (the slots exist, fp_geom) and the updates are
        // selects, so the loads are scheduled ahead of the dependent chains instead of one branch region per element
#pragma unroll
        for (int j = 0; j < 16; ++j) sv[j] = pd[p0 + j] * X[p0 + j];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const double r = rl[p0 + j];
            const double nb = fma(r, lB, r * sv[j]), na = lA * r;
            lB = (j < cnt) ? nb : lB;
            lA = (j < cnt) ? na : lA;
        }
#pragma unroll
        for (int j = 15; j >= 0; --j) {
            const double rr = ru[j > 0 ? p0 + j - 1 : (p0 >= 2 ? p0 - 2 : 0)];     // slot of element i - 1
            const double r = (i0 + j > 0) ? rr : 0.0;
            const double nb = fma(r, uB, r * sv[j]), na = uA * r;
            uB = (j < cnt) ? nb : uB;
            uA = (j < cnt) ? na : uA;
        }
    } else {
        for (int j = 0; j < cnt; ++j) {
            const double r = rl[p0 + j];
            const double s = pd[p0 + j] * X[p0 + j];
            lB = fma(r, lB, r * s);
            lA *= r;
        }
        for (int j = cnt - 1; j >= 0; --j) {
            const double r = (i0 + j > 0) ? ru[j > 0 ? p0 + j - 1 : p0 - 2] : 0.0;     // slot of element i - 1
            const double s = pd[p0 + j] * X[p0 + j];
            uB = fma(r, uB, r * s);
            uA *= r;
        }
    }
    // inclusive scans of the affine maps across lanes (ascending for l, descending for u)
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double Ap = __shfl_sync(0xffffffffu, lA, (lane - o) & 31), Bp = __shfl_sync(0xffffffffu, lB, (lane - o) & 31);
        const double Aq = __shfl_sync(0xffffffffu, uA, (lane + o) & 31), Bq = __shfl_sync(0xffffffffu, uB, (lane + o) & 31);
        if (lane >= o) { lB = fma(lA, Bp, lB); lA *= Ap; }
        if (lane + o < 32) { uB = fma(uA, Bq, uB); uA *= Aq; }
    }
    double l = __shfl_sync(0xffffffffu, lB, (lane - 1) & 31);
    double u = __shfl_sync(0xffffffffu, uB, (lane + 1) & 31);
    if (lane == 0) l = 0.0;
    if (lane == 31) u = 0.0;
    // phase 2: the sweeps with their true carries
    if (S <= 16) {
        double uu[16];
#pragma unroll
        for (int j = 15; j >= 0; --j) {
            uu[j] = u;
            const double rr = ru[j > 0 ? p0 + j - 1 : (p0 >= 2 ? p0 - 2 : 0)];     // slot of element i - 1
            const double r = (i0 + j > 0) ? rr : 0.0;
            const double nu = fma(r, u, r * sv[j]);
            u = (j < cnt) ? nu : u;
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const double r = rl[p0 + j];
            if (j < cnt) X[p0 + j] = sv[j] + l + uu[j];
            const double nl = fma(r, l, r * sv[j]);
            l = (j < cnt) ? nl : l;
        }
    } else {
        for (int j = cnt - 1; j >= 0; --j) {
            U[p0 + j] = u;
            const double r = (i0 + j > 0) ? ru[j > 0 ? p0 + j - 1 : p0 - 2] : 0.0;     // slot of element i - 1
            const double s = pd[p0 + j] * X[p0 + j];
            u = fma(r, u, r * s);
        }
        for (int j = 0; j < cnt; ++j) {
            const double r = rl[p0 + j];
            const double s = pd[p0 + j] * X[p0 + j];
            X[p0 + j] = s + l + U[p0 + j];
            l = fma(r, l, r * s);
        }
    }
}


// Element-parallel loop with U independent global loads in flight per thread before the first use: without it the
// compiler issues one load per iteration and the warp waits for each (16 serialised L2 / HBM round trips per phase).
struct FpNoHook { __device__ __forceinline__ void operator()() const {} };
template <int U, typename LoadF, typename StoreF, typename HookF = FpNoHook>
__device__ __forceinline__ void fp_batched(int total, LoadF ld, StoreF st, HookF after_first_loads = HookF()) {
    bool first = true;
    for (int e0 = threadIdx.x; e0 < total; e0 += U * FP_THREADS) {
        double v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int e = e0 + u * FP_THREADS;
            v[u] = (e < total) ? ld(e) : 0.0;
        }
        if (first) { after_first_loads(); first = false; }      // e.g. the stores of values whose loads were issued earlier
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int e = e0 + u * FP_THREADS;
            if (e < total) st(e, v[u]);
        }
    }
}
constexpr int FP_U = 8;

template <typename T>
__device__ __forceinline__ void fp_qrow(const FpPass& P, const FpTask& tk, int tile);

// acc[dl + 1][i] += sum over the fibres [f0, f1) of Y[f][i] * Cx[f - f0][i + dl]
__device__ __forceinline__ void fp_band_dots(const FpGeom& q, const double* __restrict__ Y, const double* __restrict__ Cx,
                                             int f0, int f1, double* __restrict__ acc) {
    const int n = q.n;
    const unsigned SM = q.magic;
    for (int i = threadIdx.x; i < n; i += FP_THREADS) {
        const int p = fp_pidx(i, SM);
        const int pm = (i > 0) ? fp_pidx(i - 1, SM) : p, pp = (i + 1 < n) ? fp_pidx(i + 1, SM) : p;
        double am = 0.0, a0 = 0.0, ap = 0.0;
        for (int f = f0; f < f1; ++f) {
            const double y = Y[(size_t)f * q.pitch + p];
            const double* c = Cx + (size_t)(f - f0) * q.pitch;
            am = fma(y, c[pm], am);
            a0 = fma(y, c[p], a0);
            ap = fma(y, c[pp], ap);
        }
        if (i > 0) atomicAdd(acc + i, am);
        atomicAdd(acc + n + i, a0);
        if (i + 1 < n) atomicAdd(acc + 2 * n + i, ap);
    }
}

template <typename T>
__global__ void __launch_bounds__(FP_THREADS) k_fibre_pass(const __grid_constant__ FpPass P) {
    extern __shared__ __align__(128) unsigned char smraw[];
    __shared__ double red[32];
    // which task does this tile belong to
    int ti = 0;
    while (ti + 1 < P.ntasks && (int)blockIdx.x >= P.t[ti + 1].tile0) ++ti;
    const FpTask& tk = P.t[ti];
    const int tile = (int)blockIdx.x - tk.tile0;
    if (tile >= tk.ntiles) return;
    if (tk.kind == FP_QROW) { fp_qrow<T>(P, tk, tile); return; }
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = tk.n, d = tk.d, F = tk.F;
#ifndef VGGP_EMUL
    long long* stamp = (P.dbg && tid == 0) ? P.dbg + (size_t)blockIdx.x * 8 : nullptr;
#define FP_STAMP(k) do { if (stamp) { stamp[k] = clock64(); } } while (0)
    if (stamp) { unsigned long long gt; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt)); stamp[6] = (long long)gt; stamp[7] = tk.kind; }
#else
#define FP_STAMP(k) do { } while (0)
#endif
    FP_STAMP(0);
    const FpGeom q = fp_geom(n);
    const int S = q.S;
    const unsigned SM = q.magic;
    double* pd = reinterpret_cast<double*>(smraw);
    double* ru = pd + q.pitch;
    double* rl = ru + q.pitch;
    double* bqs = rl + q.pitch;                                         // DL: 2 cQ [bq_diag | bq_off], plain indexing
    double* X = bqs + 2 * q.pitch;
    const bool aux = fp_kind_has_aux(tk.kind);
    double* Cx = X + (size_t)F * q.pitch;                               // valid only if aux
    double* U = X + (size_t)(aux ? 2 : 1) * F * q.pitch;                // valid only if S > 16
    const double noise = P.theta[2 * P.D];
    const double cg = P.ell_scale / noise;
    const double cQ = -P.ell_scale / (2.0 * noise);
    const bool contiguous = (tk.inner == 1);
    // ---- source fibres of this tile: GA carries g and ghat of the same F / 2 source fibres
    const int nsrc = (tk.kind == FP_GA) ? F / 2 : F;
    const i64 fib0 = (i64)tile * nsrc;
    const int nf = (int)min((i64)nsrc, tk.nfib - fib0);                 // source fibres present in this tile
    // element-parallel loops over (fibre, element): for strided modes consecutive threads take consecutive fibres of one
    // element index (they are adjacent in memory), for the contiguous mode consecutive elements of one fibre
    const int total = nsrc * n;
    // element index of the tile -> (element of the fibre, fibre of the tile) without integer divisions: nsrc is a power of
    // two, e / n goes through a multiply-high (e < 2^16)
    const int nsrc_sh = 31 - __clz(nsrc);
    const unsigned n_magic = (unsigned)((0x100000000ull + (unsigned)n - 1) / (unsigned)n);
    auto split_s = [&](int e, int& i, int& f) { i = e >> nsrc_sh; f = e & (nsrc - 1); };                 // strided modes
    auto split_c = [&](int e, int& i, int& f) { f = (int)__umulhi((unsigned)e, n_magic); i = e - f * n; };  // contiguous mode
    auto split = [&](int e, int& i, int& f) { if (contiguous) split_c(e, i, f); else split_s(e, i, f); };
    // address of element i of tile fibre f.  Strided modes: FP_THREADS is a multiple of nsrc, so a thread only ever touches
    // fibre tid & (nsrc - 1) and keeps its base in a register; contiguous mode: fibre f starts at f n.
    i64 my_base = 0;
    bool my_ok = false;
    if (!contiguous) {
        const i64 fg = fib0 + (tid & (nsrc - 1));
        my_ok = fg < tk.nfib;
        const i64 o = fg / tk.inner, r = fg - o * tk.inner;
        my_base = o * (i64)n * tk.inner + r;
    }
    auto addr = [&](int i, int f) -> i64 { return contiguous ? (fib0 + f) * (i64)n + i : my_base + (i64)i * tk.inner; };
    auto live = [&](int f) -> bool { return contiguous ? f < nf : my_ok; };
    // ---- generators of dimension d ([pd | ru | rl], 3 n contiguous doubles): the loads are issued before those of the
    // tile, the shared-memory stores follow, so that both round trips to L2 overlap
    const double* __restrict__ gen = P.gen[d];
    constexpr int GB = 6;                       // 3 n / FP_THREADS for n <= 512
    double gq[GB];
#pragma unroll
    for (int u = 0; u < GB; ++u) {
        const int e = tid + u * FP_THREADS;
        gq[u] = (e < 3 * n) ? gen[e] : 0.0;
    }
    FP_STAMP(1);
    auto gens_store = [&]() {
#pragma unroll
        for (int u = 0; u < GB; ++u) {
            const int e = tid + u * FP_THREADS;
            if (e < 3 * n) {
                const int arr = (int)__umulhi((unsigned)e, n_magic), i = e - arr * n;
                pd[arr * q.pitch + fp_pidx(i, SM)] = gq[u];
            }
        }
        for (int e = tid + GB * FP_THREADS; e < 3 * n; e += FP_THREADS) {      // n > 512
            const int arr = (int)__umulhi((unsigned)e, n_magic), i = e - arr * n;
            pd[arr * q.pitch + fp_pidx(i, SM)] = gen[e];
        }
    };
    switch (tk.kind) {
        case FP_R: {
            const double* __restrict__ L = tk.s0;
            fp_batched<FP_U>(total,
                [&](int e) { int i, f; split_s(e, i, f); const i64 k = fib0 + f;
                             return (f < nf && (i64)i >= k) ? L[(i64)i * n + k] : 0.0; },
                [&](int e, double v) { int i, f; split_s(e, i, f); X[(size_t)f * q.pitch + fp_pidx(i, SM)] = v; }, gens_store);
        } break;
        case FP_PROD: case FP_ALPHA: case FP_DM: {
            const double* __restrict__ src = tk.s0;
            fp_batched<FP_U>(total,
                [&](int e) { int i, f; split(e, i, f); return live(f) ? src[addr(i, f)] : 0.0; },
                [&](int e, double v) { int i, f; split(e, i, f); X[(size_t)f * q.pitch + fp_pidx(i, SM)] = v; }, gens_store);
        } break;
        case FP_GA: case FP_GAONLY: {
            const T* __restrict__ ga = reinterpret_cast<const T*>(tk.t0);
            const double* __restrict__ m = tk.s0;
            const double* __restrict__ al = tk.s1;
            const bool both = (tk.kind == FP_GA);
            bool first = true;
            for (int e0 = tid; e0 < total; e0 += 8 * FP_THREADS) {
                double gv[8], mv[8], av[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int e = e0 + u * FP_THREADS;
                    gv[u] = mv[u] = av[u] = 0.0;
                    if (e < total) {
                        int i, f; split(e, i, f);
                        if (live(f)) {
                            const i64 a = addr(i, f);
                            gv[u] = (double)ga[a]; mv[u] = m[a]; av[u] = al[a];
                        }
                    }
                }
                if (first) { gens_store(); first = false; }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int e = e0 + u * FP_THREADS;
                    if (e < total) {
                        int i, f; split(e, i, f);
                        const int p = fp_pidx(i, SM);
                        const double g1 = cg * gv[u], h1 = g1 - 0.5 * mv[u];
                        if (both) {
                            X[(size_t)f * q.pitch + p] = g1;
                            X[(size_t)(nsrc + f) * q.pitch + p] = h1;
                        } else {
                            X[(size_t)f * q.pitch + p] = h1;
                        }
                        Cx[(size_t)f * q.pitch + p] = av[u];
                    }
                }
            }
        } break;
        case FP_DL: {
            // column k of R_d -> Cx and the bq band (scaled by 2 cQ) -> shared; then column k of dR_d = 2 cQ tridiag(bq) R_d -> X
            const double* __restrict__ R = tk.s0;
            const T* __restrict__ bnd = reinterpret_cast<const T*>(tk.t0) + 2 * n;        // [bq_diag | bq_off]
            constexpr int BB = 4;               // 2 n / FP_THREADS for n <= 512
            T bq[BB];
#pragma unroll
            for (int u = 0; u < BB; ++u) {
                const int e = tid + u * FP_THREADS;
                bq[u] = (e < 2 * n) ? bnd[e] : (T)0;
            }
            fp_batched<FP_U>(total,
                [&](int e) { int i, f; split_s(e, i, f); return (f < nf) ? R[(i64)i * n + (fib0 + f)] : 0.0; },
                [&](int e, double v) { int i, f; split_s(e, i, f); Cx[(size_t)f * q.pitch + fp_pidx(i, SM)] = v; }, gens_store);
#pragma unroll
            for (int u = 0; u < BB; ++u) {
                const int e = tid + u * FP_THREADS;
                if (e < 2 * n) bqs[e] = 2.0 * cQ * (double)bq[u];
            }
            for (int e = tid + BB * FP_THREADS; e < 2 * n; e += FP_THREADS) bqs[e] = 2.0 * cQ * (double)bnd[e];      // n > 512
            __syncthreads();
            for (int e = tid; e < total; e += FP_THREADS) {
                int i, f; split_c(e, i, f);
                const double* c = Cx + (size_t)f * q.pitch;
                double r = bqs[i] * c[fp_pidx(i, SM)];
                if (i > 0) r = fma(bqs[n + i - 1], c[fp_pidx(i - 1, SM)], r);
                if (i + 1 < n) r = fma(bqs[n + i], c[fp_pidx(i + 1, SM)], r);
                X[(size_t)f * q.pitch + fp_pidx(i, SM)] = r;
            }
        } break;
        default: break;
    }
    __syncthreads();
    FP_STAMP(2);
    // ---- recurrences: one warp per fibre
    for (int f = warp; f < F; f += FP_WARPS)
        fp_fibre(q, pd, ru, rl, X + (size_t)f * q.pitch, U + (size_t)f * q.pitch, lane);
    __syncthreads();
    FP_STAMP(3);
    // ---- epilogues
    switch (tk.kind) {
        case FP_R: {
            double* __restrict__ R = tk.o0;
            for (int e = tid; e < total; e += FP_THREADS) {
                int i, f; split_s(e, i, f);
                if (f < nf) R[(i64)i * n + (fib0 + f)] = X[(size_t)f * q.pitch + fp_pidx(i, SM)];
            }
        } break;
        case FP_PROD: case FP_DM: case FP_ALPHA: {
            double* __restrict__ dst = tk.o0;
            const double* __restrict__ al = tk.s1;            // DM: alpha; ALPHA: m
            T* __restrict__ aT = reinterpret_cast<T*>(tk.t1);
            double dot = 0.0;
            const int kind = tk.kind;
            fp_batched<FP_U>(total,
                [&](int e) { int i, f; split(e, i, f);
                             return (kind != FP_PROD && live(f)) ? al[addr(i, f)] : 0.0; },
                [&](int e, double v) {
                    int i, f; split(e, i, f);
                    if (!live(f)) return;
                    const i64 a = addr(i, f);
                    const double y = X[(size_t)f * q.pitch + fp_pidx(i, SM)];
                    if (kind == FP_DM) {
                        dst[a] = y - v;
                    } else {
                        dst[a] = y;
                        if (kind == FP_ALPHA) { aT[a] = (T)y; dot = fma(y, v, dot); }
                    }
                });
            if (kind == FP_ALPHA) {
                dot = block_sum(dot, red);
                if (tid == 0) atomicAdd(P.sc + SC_MALPHA, dot);
            }
        } break;
        case FP_GA: {
            double* __restrict__ dst = tk.o0;
            const double* __restrict__ al = tk.s1;
            (void)al;
            for (int e = tid; e < total; e += FP_THREADS) {
                int i, f; split(e, i, f);
                if (!live(f)) continue;
                const i64 a = addr(i, f);
                const int pp = fp_pidx(i, SM);
                const double y = X[(size_t)f * q.pitch + pp];
                dst[a] = tk.direct ? y - Cx[(size_t)f * q.pitch + pp] : y;      // Cx holds alpha of these fibres
            }
            fp_band_dots(q, X, Cx, nsrc, nsrc + nf, P.acc[d]);
        } break;
        case FP_GAONLY:
            fp_band_dots(q, X, Cx, 0, nf, P.acc[d]);
            break;
        case FP_DL: {
            double* __restrict__ dL = tk.o0;
            const double* __restrict__ L = tk.s1;
            double trO = 1.0;
            for (int e2 = 0; e2 < P.D; ++e2)
                if (e2 != d) trO *= P.sc[SC_TR + e2];
            const double ratio = (double)P.M / (double)n;
            for (int e = tid; e < total; e += FP_THREADS) {
                int i, f; split_s(e, i, f);
                if (f >= nf) continue;
                const i64 k = fib0 + f;
                const int p = fp_pidx(i, SM);
                double v = 0.0;
                if ((i64)i >= k) {
                    v = X[(size_t)f * q.pitch + p] - trO * Cx[(size_t)f * q.pitch + p];
                    if ((i64)i == k) v += ratio / L[(i64)i * n + k];
                }
                dL[(i64)i * n + k] = v;
            }
            fp_band_dots(q, X, Cx, 0, nf, P.acc[d]);
        } break;
        default: break;
    }
    __syncthreads();
    FP_STAMP(4);
#undef FP_STAMP
}

// Row reductions of R_d: one warp per row i (tile = 8 rows).  tk.s0 = R_d, tk.s1 = L_d.
template <typename T>
__device__ __forceinline__ void fp_qrow(const FpPass& P, const FpTask& tk, int tile) {
    const int d = tk.d, n = tk.n;
    const int lane = threadIdx.x & 31;
    const int i = tile * FP_WARPS + (threadIdx.x >> 5);
    if (i >= n) return;
    const double* __restrict__ R = tk.s0;
    const double* __restrict__ L = tk.s1;
    const bool last = (i + 1 >= n);
    const double* Ri = R + (i64)i * n;
    const double* Rn = R + (i64)(last ? i : i + 1) * n;
    const double* Li = L + (i64)i * n;
    double qd = 0.0, qo = 0.0, qn = 0.0, tr = 0.0;
#pragma unroll 8
    for (int k = lane; k < n; k += 32) {
        const double r = Ri[k], rn = Rn[k];
        qd = fma(r, r, qd);
        qo = fma(r, rn, qo);
        qn = fma(rn, rn, qn);
        if (k <= i) tr = fma(r, Li[k], tr);
    }
    qd = warp_sum(qd); qo = warp_sum(qo); qn = warp_sum(qn); tr = warp_sum(tr);
    if (lane == 0) {
        if (last) { qo = 0.0; qn = 0.0; }
        P.Qb[d][i] = qd;
        P.Qb[d][n + i] = qo;
        T* tab = reinterpret_cast<T*>(P.bandT) + P.tab_off[d];
        const double B2 = 2.0 * qo;
        tab[3 * n + i] = (T)qd; tab[4 * n + i] = (T)(B2 - 2.0 * qd); tab[5 * n + i] = (T)(qd - B2 + qn);
        if (P.det) {
            double* ds = P.det + (i64)blockIdx.x * FP_DET_SLOT;
            ds[FP_DET_TR + (threadIdx.x >> 5)] = tr;
            ds[FP_DET_LOGDET + (threadIdx.x >> 5)] = 2.0 * log(fabs(Li[i]));
        } else {
            atomicAdd(P.sc + SC_TR + d, tr);
            atomicAdd(P.sc + SC_LOGDETS + d, 2.0 * log(fabs(Li[i])));
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// First-order linear recurrence t_i = b_i + a_i t_prev over i = 0 .. n-1 (ascending: t_prev = t_{i-1}; descending: t_{i+1}),
// t_prev = 0 at the start, by ONE warp: lane-local sweeps + a 5-step affine scan across lanes.  a(i), b(i) are functors.
// ---------------------------------------------------------------------------------------------------------
template <bool ASC, typename FA, typename FB>
__device__ __forceinline__ void warp_recurrence(int n, FA a, FB b, double* __restrict__ out, int lane) {
    const int S = (n + 31) / 32;
    // lane l owns [l S, (l + 1) S); for the descending sweep the lane order is reversed so that the scan still runs upwards.
    // a(i, p), b(i, p) and out[] use the padded position p = i + i / S of element i (lane stride S + 1: the lane-strided
    // shared-memory accesses of the sweeps are then conflict-free; unpadded they were 32-way conflicts)
    const int seg = ASC ? lane : 31 - lane;
    const int i0 = seg * S, cnt = max(0, min(S, n - i0));
    const int q0 = seg * (S + 1);
    double A = 1.0, B = 0.0;
    for (int j = 0; j < cnt; ++j) {
        const int jj = ASC ? j : cnt - 1 - j;
        const double ai = a(i0 + jj, q0 + jj);
        B = fma(ai, B, b(i0 + jj, q0 + jj));
        A *= ai;
    }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double Ap = __shfl_sync(0xffffffffu, A, (lane - o) & 31), Bp = __shfl_sync(0xffffffffu, B, (lane - o) & 31);
        if (lane >= o) { B = fma(A, Bp, B); A *= Ap; }
    }
    double t = __shfl_sync(0xffffffffu, B, (lane - 1) & 31);
    if (lane == 0) t = 0.0;
    for (int j = 0; j < cnt; ++j) {
        const int jj = ASC ? j : cnt - 1 - j;
        t = fma(a(i0 + jj, q0 + jj), t, b(i0 + jj, q0 + jj));
        out[q0 + jj] = t;
    }
}

// ---------------------------------------------------------------------------------------------------------
// d theta and the ELBO scalars.
//   dK_d[i][j] = -W_d[i][j] + (c_d / 2) Q_d[i][j] - (M / (2 M_d)) P_d[i][j]   on |i - j| <= 1   (K_d and dK_d / d theta are tridiagonal)
// W_d = band of P_d (dP_d) P_d.  Its Gram and dR L^T parts arrive in the accumulators `acc` (fibre passes); the part that
// goes through the band scatter X_d = cP tridiag(bp_diag, bp_off) of the per-observation sums is formed here in O(n):
// with P semiseparable, the quadratic forms of a row of P_d restricted to the indices >= i (T_i) and <= i (S_i) obey
//   T_i = xd_i pd_i^2 + 2 xo_i pd_i P[i][i+1] + ru_i^2 T_{i+1},      S_i = xd_i pd_i^2 + 2 xo_{i-1} pd_i P[i][i-1] + rl_{i-1}^2 S_{i-1}
//   (P X P)[i][i]   = T_i + rl_{i-1}^2 S_{i-1} + 2 xo_{i-1} P[i][i-1] pd_i
//   (P X P)[i][i+1] = ru_i T_{i+1} + rl_i S_i + xo_i (pd_i pd_{i+1} + P[i][i+1]^2)
// grid (D), 512 threads, dynamic smem 7 (n + n / S + 2) doubles.
// ---------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(512) k_b1_theta(const __grid_constant__ GridDims g, const double* __restrict__ theta,
                                                  const double* __restrict__ acc, const T* __restrict__ gband,
                                                  const double* __restrict__ gscal,
                                                  double ell_scale, double* __restrict__ out, double* __restrict__ dtheta,
                                                  long long* __restrict__ dbg) {
    extern __shared__ double sm[];
    const int d = blockIdx.x;
    const int n = g.n[d];
    const int D = g.D;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#ifndef VGGP_EMUL
#define TH_STAMP(k) do { if (dbg && threadIdx.x == 0) dbg[blockIdx.x * 8 + (k)] = clock64(); } while (0)
#else
#define TH_STAMP(k) do { } while (0)
#endif
    TH_STAMP(0);
    // shared: generators, the band scatter X_d and the two recurrences, 7 arrays in PADDED positions p(i) = i + i / S
    // (S = elements per lane of the sweeps): the serial sweeps must neither wait for global memory nor collide on banks
    const int S = (n + 31) / 32;
    const int np = n + (n + S - 1) / S + 2;
    const unsigned SM = (unsigned)((0x100000000ull + (unsigned)S - 1) / (unsigned)S);
    auto P_ = [&](int i) { return fp_pidx(i, SM); };
    double* Tt = sm;
    double* Ss = sm + np;
    double* pd = sm + 2 * np;
    double* ru = sm + 3 * np;
    double* rl = sm + 4 * np;
    double* xd = sm + 5 * np;
    double* xo = sm + 6 * np;
    const double half_ratio = 0.5 * (double)g.M / (double)n;
    const double half_c = 0.5 * tr_others(g, d);
    const double cP = ell_scale / (2.0 * theta[2 * D]);
    {
        const double* __restrict__ gen = g.gen[d];
        const T* __restrict__ bp = gband + g.band_off[d];           // [bp_diag | bp_off | bq_diag | bq_off]
        for (int i = threadIdx.x; i < n; i += 512) {
            const int p = P_(i);
            pd[p] = gen[i]; ru[p] = gen[n + i]; rl[p] = gen[2 * n + i];
            xd[p] = cP * (double)bp[i]; xo[p] = cP * (double)bp[n + i];
        }
    }
    for (int e = 0; e < d; ++e) acc += 3 * g.n[e];          // this dimension's block of the accumulators
    __syncthreads();
    TH_STAMP(1);
    // neighbours of element i in padded positions: i + 1 is p + 1 unless i closes a lane segment (then p + 2); likewise i - 1
    if (warp == 0) {
        warp_recurrence<false>(n,
            [&](int i, int p) { return (i + 1 < n) ? ru[p] * ru[p] : 0.0; },
            [&](int i, int p) { const double x = xd[p] * pd[p] * pd[p];
                                return (i + 1 < n) ? x + 2.0 * xo[p] * pd[p] * (ru[p] * pd[P_(i + 1)]) : x; },
            Tt, lane);
    } else if (warp == 1) {
        warp_recurrence<true>(n,
            [&](int i, int p) { return (i > 0) ? rl[P_(i - 1)] * rl[P_(i - 1)] : 0.0; },
            [&](int i, int p) { const double x = xd[p] * pd[p] * pd[p];
                                if (i == 0) return x;
                                const int pm = P_(i - 1);
                                return x + 2.0 * xo[pm] * pd[p] * (rl[pm] * pd[pm]); },
            Ss, lane);
    }
    // d K / d l and d K / d s2 take three distinct values each (corner diagonal, interior diagonal, off-diagonal)
    double gl[3], gs[3];
    factor_entry_grad(g, theta, d, 0, 0, gl[0], gs[0]);
    factor_entry_grad(g, theta, d, 1, 1, gl[1], gs[1]);
    factor_entry_grad(g, theta, d, 0, 1, gl[2], gs[2]);
    const double* __restrict__ Qb = g.Qb[d];
    TH_STAMP(2);
    __syncthreads();
    TH_STAMP(3);
    double sl = 0.0, ss = 0.0;
#pragma unroll 3
    for (int e = threadIdx.x; e < 3 * n; e += 512) {
        const int dl = (e >= 2 * n) ? 1 : (e >= n ? 0 : -1);
        const int i = e - (dl + 1) * n;
        const int j = i + dl;
        if (j < 0 || j >= n) continue;
        const int lo = i < j ? i : j;
        double qv, pij, w;
        if (dl == 0) {
            const int p = P_(i);
            qv = Qb[i];
            pij = pd[p];
            w = Tt[p];
            if (i > 0) {
                const int pm = P_(i - 1);
                const double pl = rl[pm] * pd[pm];                             // P[i][i-1]
                w += rl[pm] * rl[pm] * Ss[pm] + 2.0 * xo[pm] * pl * pd[p];
            }
        } else {
            const int p = P_(lo), pn = P_(lo + 1);
            qv = Qb[n + lo];
            const double pu = ru[p] * pd[pn];                                  // P[lo][lo+1]
            pij = pu;
            w = ru[p] * Tt[pn] + rl[p] * Ss[p] + xo[p] * (pd[p] * pd[pn] + pu * pu);
        }
        const double v = -(acc[e] + w) + half_c * qv - half_ratio * pij;
        const bool corner = (i == 0 || i == n - 1);
        sl = fma(v, (dl != 0) ? gl[2] : (corner ? gl[0] : gl[1]), sl);
        ss = fma(v, (dl != 0) ? gs[2] : (corner ? gs[0] : gs[1]), ss);
    }
    sl = warp_sum(sl);
    ss = warp_sum(ss);
    __shared__ double red2[2][16];
    if (lane == 0) { red2[0][warp] = sl; red2[1][warp] = ss; }
    __syncthreads();
    TH_STAMP(4);
    if (threadIdx.x == 0) {
        sl = 0.0; ss = 0.0;
        for (int w = 0; w < 16; ++w) { sl += red2[0][w]; ss += red2[1][w]; }
        const double noise = theta[2 * D];
        double kff = 1.0;
        for (int e = 0; e < D; ++e) kff *= theta[D + e];
        const double E = gscal[0], nobs = gscal[1];
        const double dkff = -ell_scale * nobs / (2.0 * noise);
        dtheta[d] = sl;
        dtheta[D + d] = ss + dkff * kff / theta[D + d];
        if (d == 0) {
            const double tot = E + nobs * kff;
            const double ell = -0.5 * nobs * log(2.0 * 3.14159265358979323846 * noise) - tot / (2.0 * noise);
            dtheta[2 * D] = ell_scale * (-nobs / (2.0 * noise) + tot / (2.0 * noise * noise));
            double trp = 1.0, lds = 0.0;
            for (int e = 0; e < D; ++e) {
                trp *= g.sc[SC_TR + e];
                lds += ((double)g.M / (double)g.n[e]) * (g.sc[SC_LOGDETK + e] - g.sc[SC_LOGDETS + e]);
            }
            const double kl = 0.5 * (trp + g.sc[SC_MALPHA] - (double)g.M + lds);
            out[0] = ell_scale * ell - kl;
            out[1] = ell_scale * ell;
            out[2] = kl;
            out[3] = nobs;
        }
    }
    TH_STAMP(5);
#undef TH_STAMP
}

// Explicit P_d from the generators (O(n^2)), on demand (vggp_workspace_ptr): the fused path never materialises it in a step.
//   P[i][j] = pd[j] prod_{k=i}^{j-1} ru[k] (i < j),  pd[i] (i == j),  pd[j] prod_{k=j}^{i-1} rl[k] (i > j)
// grid (ceil(nmax / 256), D), 256 threads
__global__ void __launch_bounds__(256) k_b1_fill_P(const __grid_constant__ GridDims g) {
    const int d = blockIdx.y;
    const int n = g.n[d];
    const int j = (int)blockIdx.x * 256 + threadIdx.x;
    if (j >= n) return;
    const double* __restrict__ gen = g.gen[d];
    double* __restrict__ P = g.P[d];
    const double pj = gen[j];
    double p = pj;
    P[(i64)j * n + j] = p;
    for (int i = j - 1; i >= 0; --i) {
        p *= gen[n + i];
        P[(i64)i * n + j] = p;
    }
    p = pj;
    for (int i = j + 1; i < n; ++i) {
        p *= gen[2 * n + i - 1];
        P[(i64)i * n + j] = p;
    }
}

// K_d as a dense matrix, on demand (vggp_workspace_ptr), like P_d.
// grid (ceil(nmax^2 / 256), D)
__global__ void __launch_bounds__(256) k_b1_fill_Kraw(const __grid_constant__ GridDims g, const double* __restrict__ theta) {
    const int d = blockIdx.y;
    const int n = g.n[d];
    const i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (i64)n * n) return;
    g.Kraw[d][e] = factor_entry(g, theta, d, (int)(e / n), (int)(e % n));
}

}  // namespace vggp
