// Per-observation kernels: B1 interpolation stencil (bit-exact restatement of bspline.py:23-77, 92-94),
// dense feature matrices (tests / small predictions), the observation packing pass and the fused ELBO
// forward+backward over packed observations.
#pragma once
#include "common.cuh"

namespace vggp {

struct MeshView {
    const float* t;      // knots (float32, exactly as uploaded)
    int K;
    float t0, inv_h;     // arithmetic guess of the cell: floor((x - t0) * inv_h)
    int nearly_uniform;  // guess is within +-2 cells of the truth (checked at plan creation)
    float tfirst, tlast; // mesh[0], mesh[K-1]
};

// c = clamp(searchsorted(mesh, x, right=False) - 1, 0, K-2);  inside = mesh[0] <= x <= mesh[K-1].
// Comparisons are done in T against the float32 knots promoted to T (exact), like torch does.
template <typename T>
__device__ __forceinline__ int find_cell(const float* __restrict__ t, int K, float t0, float inv_h,
                                         int nearly_uniform, T x, bool& inside) {
    inside = (x >= (T)t[0]) && (x <= (T)t[K - 1]);
    int c;
    if (nearly_uniform) {
        float gf = ((float)x - t0) * inv_h;
        gf = fminf(fmaxf(gf, 0.0f), (float)(K - 2));     // NaN -> 0
        c = (int)gf;
#pragma unroll
        for (int it = 0; it < 3; ++it)
            if (c > 0 && x <= (T)t[c]) --c;
#pragma unroll
        for (int it = 0; it < 3; ++it)
            if (c < K - 2 && x > (T)t[c + 1]) ++c;
    } else {
        // lower_bound: first index with t[idx] >= x
        int lo = 0, hi = K;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if ((T)t[mid] < x) lo = mid + 1; else hi = mid;
        }
        c = min(max(lo - 1, 0), K - 2);
    }
    return c;
}

// Correctly rounded u / h for float from the correctly rounded reciprocal rh = RN(1/h) (Markstein): one
// multiply and two fused multiply-adds.  Valid for the operand ranges of the stencil (0 <= u <= h, h a normal
// float32 knot spacing); bit-exactness against IEEE division is asserted by the stencil tests.
__device__ __forceinline__ float div_by_cached_rcp(float u, float h, float rh) {
    const float q0 = u * rh;
    const float rem = fmaf(-q0, h, u);
    return fmaf(rem, rh, q0);
}
__device__ __forceinline__ double div_by_cached_rcp(double u, double h, double rh) {
    (void)rh;
    return u / h;
}

// Interpolation weights of the two hats overlapping cell c.  The denominator is the float32 knot
// difference promoted to T (0-dim float32 arithmetic in the reference), the numerators are computed in T;
// true IEEE subtraction and division (no fma contraction is possible here).
template <typename T>
__device__ __forceinline__ void b1_weights(const float* __restrict__ t, int c, T x, bool inside, T& w_lo, T& w_hi) {
    const float tl = t[c], th = t[c + 1];
    const T h = (T)(th - tl);
    const T rh = (T)1 / h;
    const T wh = div_by_cached_rcp(x - (T)tl, h, rh);
    const T wl = div_by_cached_rcp((T)th - x, h, rh);
    w_hi = inside ? wh : (T)0;
    w_lo = inside ? wl : (T)0;
}

template <typename T>
__global__ void __launch_bounds__(256) k_b1_stencil(MeshView mv, const T* __restrict__ x, i64 n,
                                                    int32_t* __restrict__ c_out, T* __restrict__ w_lo,
                                                    T* __restrict__ w_hi) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        const T xv = x[i];
        bool inside;
        const int c = find_cell<T>(mv.t, mv.K, mv.t0, mv.inv_h, mv.nearly_uniform, xv, inside);
        T wl, wh;
        b1_weights<T>(mv.t, c, xv, inside, wl, wh);
        c_out[i] = inside ? c : -1;
        w_lo[i] = wl;
        w_hi[i] = wh;
    }
}

// Dense (M_d, n) B1 feature matrix (zero-filled first by the caller).
template <typename T>
__global__ void __launch_bounds__(256) k_b1_dense(MeshView mv, const T* __restrict__ x, i64 n, T* __restrict__ phi) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        const T xv = x[i];
        bool inside;
        const int c = find_cell<T>(mv.t, mv.K, mv.t0, mv.inv_h, mv.nearly_uniform, xv, inside);
        T wl, wh;
        b1_weights<T>(mv.t, c, xv, inside, wl, wh);
        if (inside) {
            phi[(i64)c * n + i] = wl;
            phi[(i64)(c + 1) * n + i] = wh;
        }
    }
}

// B0 cell-integrated Matern-1/2 feature of cell k at x (gridded_kronecker_structure.py:1325-1374).
// idx = searchsorted(mesh, x, right=False).
template <typename T>
__device__ __forceinline__ T b0_feature(const float* __restrict__ t, int k, int idx, T x, T l, T s2) {
    const T a = (T)t[k], b = (T)t[k + 1];
    const T e1 = l * exp(-fabs(x - a) / l);
    const T e2 = l * exp(-fabs(x - b) / l);
    const int sgn = idx - k - 1;                // indicator = -sign(sgn)
    T v;
    if (sgn == 0) v = (T)2 * l - (e1 + e2);
    else if (sgn > 0) v = -(e1 - e2);
    else v = (e1 - e2);
    return v * s2;
}

template <typename T>
__device__ __forceinline__ int lower_bound_knots(const float* __restrict__ t, int K, T x) {
    int lo = 0, hi = K;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((T)t[mid] < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Dense (K-1, n) B0 feature matrix.  grid (ceil(n/256), K-1)
template <typename T>
__global__ void __launch_bounds__(256) k_b0_dense(MeshView mv, const T* __restrict__ x, i64 n, double l, double s2,
                                                  T* __restrict__ phi) {
    const int k = blockIdx.y;
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const T xv = x[i];
    const int idx = lower_bound_knots<T>(mv.t, mv.K, xv);
    phi[(i64)k * n + i] = b0_feature<T>(mv.t, k, idx, xv, (T)l, (T)s2);
}

// Dense (K, n) Fourier feature matrix (K = 2 M + 1 rows: cosines, then sines).  grid (ceil(n/256), K)
template <typename T>
__global__ void __launch_bounds__(256) k_vff_dense(MeshView mv, const T* __restrict__ x, i64 n, double l, T* __restrict__ phi) {
    const int k = blockIdx.y, Mf = (mv.K - 1) / 2;
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const T xa = (T)mv.t[0], xb = (T)mv.t[mv.K - 1], xv = x[i];
    T f = (T)0;
    if (xv >= xa && xv < xb) {
        const int kf = k <= Mf ? k : k - Mf;
        const T arg = ((T)6.283185307179586476925286766559 * (T)kf / (xb - xa)) * (xv - xa);
        f = k <= Mf ? cos(arg) : sin(arg);
    } else if (k <= Mf) {
        f = exp(-fmin(fabs(xv - xa), fabs(xv - xb)) / (T)l);
    }
    phi[(i64)k * n + i] = f;
}

// Dense (K, n) SVGP feature matrix: phi[k][i] = s2 exp(-|x_i - z_k| / l).  grid (ceil(n/256), K)
template <typename T>
__global__ void __launch_bounds__(256) k_svgp_dense(MeshView mv, const T* __restrict__ x, i64 n, double l, double s2,
                                                    T* __restrict__ phi) {
    const int k = blockIdx.y;
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    phi[(i64)k * n + i] = (T)s2 * exp(-fabs(x[i] - (T)mv.t[k]) / (T)l);
}

// ---------------------------------------------------------------------------------------------------------
// Packed observation layout.
//
// The fused kernel gives every lane one contiguous RUN of R observations of the (optionally cell-sorted)
// stream and walks it sequentially, so that per-cell state and gradient accumulators live in registers and are
// flushed only when the run leaves a cell.  To keep the global loads coalesced the stream is stored
// "warp-transposed": observation j of lane l of warp w (stream position (32 w + l) R + j) lives at
//      w * 32 R + (j / 4) * 128 + l * 4 + (j % 4)
// so one 16-byte (float4) load per lane fetches 4 consecutive observations of its run and a warp reads 512
// contiguous bytes.  Padding slots hold x = NaN (outside every mesh), y = 0.
// ---------------------------------------------------------------------------------------------------------
struct PackGeom {
    int R;          // run length per lane (multiple of 4)
    i64 nwarps;     // number of warps of runs
    i64 n_packed;   // nwarps * 32 * R
};

// key = flat cell id (row-major over cells) or `ncells` for observations outside the mesh
template <typename T, int D>
struct KeyArgs {
    const T* x[D];
    i64 n;
    MeshView mesh[D];
};

template <typename T, int D>
__global__ void __launch_bounds__(256) k_cell_keys(const __grid_constant__ KeyArgs<T, D> a, uint32_t ncells,
                                                   uint32_t* __restrict__ keys, uint32_t* __restrict__ idx) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (i64)gridDim.x * blockDim.x) {
        uint32_t key = 0;
        bool all_in = true;
#pragma unroll
        for (int d = 0; d < D; ++d) {
            bool inside;
            const int c = find_cell<T>(a.mesh[d].t, a.mesh[d].K, a.mesh[d].t0, a.mesh[d].inv_h,
                                       a.mesh[d].nearly_uniform, a.x[d][i], inside);
            key = key * (uint32_t)(a.mesh[d].K - 1) + (uint32_t)c;
            all_in = all_in && inside;
        }
        keys[i] = all_in ? key : ncells;
        idx[i] = (uint32_t)i;
    }
}

template <typename T, int D>
struct GatherArgs {
    const T* x[D];
    const T* y;
    T* xp[D];
    T* yp;
    i64 n;
    const uint32_t* perm;   // nullptr: keep the input order
    PackGeom geo;
};

template <typename T, int D>
__global__ void __launch_bounds__(256) k_pack_gather(const __grid_constant__ GatherArgs<T, D> a) {
    const i64 per_warp = (i64)32 * a.geo.R;
    T nanv;
    if (sizeof(T) == 4) nanv = (T)__int_as_float(0x7fc00000); else nanv = (T)__longlong_as_double(0x7ff8000000000000LL);
    for (i64 q = (i64)blockIdx.x * blockDim.x + threadIdx.x; q < a.geo.n_packed; q += (i64)gridDim.x * blockDim.x) {
        const i64 w = q / per_warp;
        const int rem = (int)(q - w * per_warp);
        const int g4 = rem >> 7, lane = (rem & 127) >> 2, jj = rem & 3;
        const i64 s = (w * 32 + lane) * (i64)a.geo.R + (g4 * 4 + jj);
        if (s < a.n) {
            const i64 src = a.perm ? (i64)a.perm[s] : s;
#pragma unroll
            for (int d = 0; d < D; ++d) a.xp[d][q] = a.x[d][src];
            a.yp[q] = a.y[src];
        } else {
#pragma unroll
            for (int d = 0; d < D; ++d) a.xp[d][q] = nanv;
            a.yp[q] = (T)0;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// TMA (bulk async copy) helpers: the per-CTA tables (band tables of P_d, Q_d and the knots) are staged into
// shared memory with one cp.async.bulk completing on an mbarrier.
// ---------------------------------------------------------------------------------------------------------
#ifndef VGGP_EMUL   // tests/host_emul supplies CPU stand-ins for these six PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok)
                     : "r"(smem_u32(bar)), "r"(phase)
                     : "memory");
    } while (!ok);
}
#endif

// ---------------------------------------------------------------------------------------------------------
// K1: fused per-observation ELBO forward + backward, B1 (ASVGP) family, packed layout.
//
// Per observation (hat weight a_d = w_hi of dimension d, w_lo = 1 - a_d):
//   mu   = sum_S am[S] prod_{d in S} a_d                 (alpha at the 2^D cell corners, monomial basis)
//   p_d  = pe[d][0] + pe[d][1] a_d + pe[d][2] a_d^2      (main / first off diagonal of P_d at the cell)
//   q_d  likewise from Q_d;   v = kff - prod p_d + prod q_d;   r = y - mu
// and, in the same pass, the reverse-mode sums kept in registers while the run stays in one cell:
//   gm[S]    += r prod_{d in S} a_d        -> d alpha at the corners
//   bp[d][k] += (prod_{e != d} p_e) a_d^k  -> main / off-diagonal gradients of P_d   (bq likewise for Q_d)
//   E        += r^2 - prod p + prod q
// 1/noise, ell_scale and kff are applied on the grid side.  On leaving a cell the sums are converted back to
// the corner / band bases and flushed: d alpha with global float atomics (L2-resident M-vector), band sums
// into per-CTA shared accumulators that are added to the global buffer once at the end.
// ---------------------------------------------------------------------------------------------------------
template <typename T, int D>
struct PackedArgs {
    const T* xp[D];
    const T* yp;
    PackGeom geo;
    MeshView mesh[D];
    int stride[D];         // row-major strides of alpha (M < 2^31, checked at plan creation)
    int band_off[D];       // offset of dim d inside the gradient band block: [bp_d | bp_o | bq_d | bq_o] each n_d long
    int tab_off[D];        // offset (elements of T) of dim d inside the cell tables: [pe0 pe1 pe2 qe0 qe1 qe2 h rh] each n_d long
    int knot_off[D];
    int table_bytes;       // bytes of [cell tables (T) | pad16 | knots (float) | pad16] in `tables`
    int knots_byte_off;
    const unsigned char* tables;
    const T* alpha;
    T* galpha;
    T* gband;
    double* gs;
    double n_real;
    unsigned int* counter;   // work-stealing counter over warp chunks (zeroed before the launch)
};

template <typename T>
__device__ __forceinline__ void load4(const T* p, T (&v)[4]);
template <>
__device__ __forceinline__ void load4<float>(const float* p, float (&v)[4]) {
    const float4 t = __ldcs(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <>
__device__ __forceinline__ void load4<double>(const double* p, double (&v)[4]) {
    const double2 a = __ldcs(reinterpret_cast<const double2*>(p));
    const double2 b = __ldcs(reinterpret_cast<const double2*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

template <typename T, int D>
struct LaneState {
    int c[D];
    T tlo[D], tlo_chk[D], thi[D], h[D], rh[D];
    T am[1 << D];
    T pe[D][3], qe[D][3];
    // accumulators
    T gm[1 << D];
    T bp[D][3], bq[D][3];
    T accE;
    bool valid;
};

// Leave the cached cell: convert the monomial moments back to corner / band sums and add them to the global
// gradient buffer with fire-and-forget float atomics (RED; the buffer is L2-resident).  The band sums of dimension
// d are indexed by c_d alone, so they are flushed only when c_d itself changes (`newc`; nullptr = flush everything):
// in cell-sorted order the slow dimensions change rarely, which removes most of the same-address RED traffic.
template <typename T, int D>
__device__ __forceinline__ void lane_flush(const PackedArgs<T, D>& a, LaneState<T, D>& s, const int* newc) {
    if (!s.valid) return;
    // per dimension (m0, m1) -> (m0 - m1, m1)
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const int bit = 1 << (D - 1 - d);
#pragma unroll
        for (int i = 0; i < (1 << D); ++i)
            if (!(i & bit)) s.gm[i] -= s.gm[i | bit];
    }
    int base = 0;
#pragma unroll
    for (int d = 0; d < D; ++d) base += s.c[d] * a.stride[d];
    T* ga = a.galpha + base;
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) {
        int off = 0;
#pragma unroll
        for (int d = 0; d < D; ++d) off += (i & (1 << (D - 1 - d))) ? a.stride[d] : 0;
        atomicAdd(ga + off, s.gm[i]);
        s.gm[i] = (T)0;
    }
#pragma unroll
    for (int d = 0; d < D; ++d) {
        if (newc != nullptr && newc[d] == s.c[d]) continue;
        const int n = a.mesh[d].K;
        T* gb = a.gband + (a.band_off[d] + s.c[d]);
        // sums of w (1-a)^2, w (1-a) a, w a^2 from the moments s0, s1, s2
        atomicAdd(gb, s.bp[d][0] - (T)2 * s.bp[d][1] + s.bp[d][2]);
        atomicAdd(gb + n, s.bp[d][1] - s.bp[d][2]);
        atomicAdd(gb + 1, s.bp[d][2]);
        atomicAdd(gb + 2 * n, s.bq[d][0] - (T)2 * s.bq[d][1] + s.bq[d][2]);
        atomicAdd(gb + 3 * n, s.bq[d][1] - s.bq[d][2]);
        atomicAdd(gb + 2 * n + 1, s.bq[d][2]);
#pragma unroll
        for (int k = 0; k < 3; ++k) { s.bp[d][k] = (T)0; s.bq[d][k] = (T)0; }
    }
}

// Enter cell c: knots and per-cell tables from shared memory, alpha corners from L2.
template <typename T, int D>
__device__ __forceinline__ void lane_load_cell(const PackedArgs<T, D>& a, LaneState<T, D>& s, const int (&c)[D],
                                               const T (&tl)[D], const T (&th)[D], const T* s_tab) {
    int base = 0;
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const int n = a.mesh[d].K;
        const T* tb = s_tab + (a.tab_off[d] + c[d]);
        s.c[d] = c[d];
        s.tlo[d] = tl[d];
        s.tlo_chk[d] = tl[d];
        s.thi[d] = th[d];
        s.pe[d][0] = tb[0]; s.pe[d][1] = tb[n]; s.pe[d][2] = tb[2 * n];
        s.qe[d][0] = tb[3 * n]; s.qe[d][1] = tb[4 * n]; s.qe[d][2] = tb[5 * n];
        s.h[d] = tb[6 * n];          // (T)(float32 knot difference), reference semantics
        s.rh[d] = tb[7 * n];         // correctly rounded 1 / h
        base += c[d] * a.stride[d];
    }
    const T* al = a.alpha + base;
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) {
        int off = 0;
#pragma unroll
        for (int d = 0; d < D; ++d) off += (i & (1 << (D - 1 - d))) ? a.stride[d] : 0;
        s.am[i] = __ldg(al + off);
    }
    // corner values -> monomial coefficients: per dimension (lo, hi) -> (lo, hi - lo)
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const int bit = 1 << (D - 1 - d);
#pragma unroll
        for (int i = 0; i < (1 << D); ++i)
            if (i & bit) s.am[i] -= s.am[i ^ bit];
    }
    s.valid = true;
}

// the largest value strictly below a finite v (one step in the ordered bit pattern; -denorm_min below +-0)
__device__ __forceinline__ float just_below(float v) {
    const int b = __float_as_int(v);
    return __int_as_float(v > 0.0f ? b - 1 : (v < 0.0f ? b + 1 : (int)0x80000001u));
}
__device__ __forceinline__ double just_below(double v) {
    const long long b = __double_as_longlong(v);
    return __longlong_as_double(v > 0.0 ? b - 1 : (v < 0.0 ? b + 1 : (long long)0x8000000000000001ull));
}

template <typename T, int D>
__device__ __forceinline__ bool lane_in_cell(const LaneState<T, D>& s, const T (&x)[D]) {
    bool same = true;
#pragma unroll
    for (int d = 0; d < D; ++d) same = same && (x[d] > s.tlo_chk[d]) && (x[d] <= s.thi[d]);
    return same;
}

// Slow path: the observation is not inside the cached cell.  Returns true when the observation has been consumed
// here (outside the mesh: zero feature column, mu = 0, p = q = 0).
// Cell search: walk from the cached cell (cell-sorted or along-track data move to a neighbouring cell), falling back
// to the arithmetic guess after 4 steps; the loop ends when t[c] < x <= t[c+1] (exact comparisons against the float32
// knots, same result as searchsorted(mesh, x, right=False) - 1 clamped to [0, K-2]).
template <typename T, int D>
__device__ __forceinline__ bool lane_switch(const PackedArgs<T, D>& a, LaneState<T, D>& s, const T (&x)[D], T y,
                                            const T* s_tab, const float* s_knots) {
    bool all_in = true;
#pragma unroll
    for (int d = 0; d < D; ++d) all_in = all_in && (x[d] >= (T)a.mesh[d].tfirst) && (x[d] <= (T)a.mesh[d].tlast);
    if (!all_in) {               // also catches NaN padding
        s.accE += y * y;
        return true;
    }
    int c[D];
    T tl[D], th[D];
    bool moved = !s.valid;
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const float* t = s_knots + a.knot_off[d];
        const int K = a.mesh[d].K;
        int cc;
        T lo, hi;
        if (s.valid) {
            cc = s.c[d]; lo = s.tlo[d]; hi = s.thi[d];
        } else {
            cc = 0; lo = (T)t[0]; hi = (T)t[1];
        }
        int steps = 0;
#pragma unroll 1
        while (true) {
            if (cc > 0 && x[d] <= lo) { --cc; hi = lo; lo = (T)t[cc]; }
            else if (cc < K - 2 && x[d] > hi) { ++cc; lo = hi; hi = (T)t[cc + 1]; }
            else break;
            if (++steps == 4) {          // far jump: restart from the arithmetic guess
                float gf = ((float)x[d] - a.mesh[d].t0) * a.mesh[d].inv_h;
                gf = fminf(fmaxf(gf, 0.0f), (float)(K - 2));
                cc = (int)gf; lo = (T)t[cc]; hi = (T)t[cc + 1];
            }
        }
        c[d] = cc; tl[d] = lo; th[d] = hi;
        moved = moved || (cc != s.c[d]);
    }
    if (moved) {
        lane_flush<T, D>(a, s, c);
        lane_load_cell<T, D>(a, s, c, tl, th, s_tab);
    } else {
        // x == first knot of the mesh: it belongs to cell 0 although x > t_lo fails; lower the cached bound by one ulp
        // so that the fast check accepts x >= t_0 (the weight formula is unchanged: a = (x - t_0) / h = 0) and still
        // rejects everything left of the mesh.  (Up to round 1 the bound was widened to -inf, which let an observation
        // left of the mesh through when it followed a first-knot hit inside the same run of an unsorted stream.)
#pragma unroll
        for (int d = 0; d < D; ++d)
            if (c[d] == 0 && x[d] == s.tlo[d]) s.tlo_chk[d] = just_below(s.tlo[d]);
    }
    return false;
}

// Fast path: straight-line arithmetic for an observation inside the cached cell.
template <typename T, int D>
__device__ __forceinline__ void lane_math(LaneState<T, D>& s, const T (&x)[D], T y) {
    T w[D], p[D], q[D];
#pragma unroll
    for (int d = 0; d < D; ++d) {
        w[d] = div_by_cached_rcp(x[d] - s.tlo[d], s.h[d], s.rh[d]);
        p[d] = fma(fma(s.pe[d][2], w[d], s.pe[d][1]), w[d], s.pe[d][0]);
        q[d] = fma(fma(s.qe[d][2], w[d], s.qe[d][1]), w[d], s.qe[d][0]);
    }
    // monomials prod_{d in S} a_d, S indexed by bits (dimension 0 = most significant bit)
    T mono[1 << D];
    mono[0] = (T)1;
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const int bit = 1 << (D - 1 - d);
#pragma unroll
        for (int i = 0; i < (1 << D); ++i)
            if ((i & bit) && !(i & (bit - 1))) mono[i] = (i ^ bit) ? mono[i ^ bit] * w[d] : w[d];
    }
    T mu = s.am[0];
#pragma unroll
    for (int i = 1; i < (1 << D); ++i) mu = fma(s.am[i], mono[i], mu);
    const T r = y - mu;
    s.gm[0] += r;
#pragma unroll
    for (int i = 1; i < (1 << D); ++i) s.gm[i] = fma(r, mono[i], s.gm[i]);
    T pp = p[0], qq = q[0];
#pragma unroll
    for (int d = 1; d < D; ++d) { pp *= p[d]; qq *= q[d]; }
    s.accE += fma(r, r, qq - pp);
#pragma unroll
    for (int d = 0; d < D; ++d) {
        T op = (T)1, oq = (T)1;
        bool first = true;
#pragma unroll
        for (int e = 0; e < D; ++e)
            if (e != d) {
                op = first ? p[e] : op * p[e];
                oq = first ? q[e] : oq * q[e];
                first = false;
            }
        const T t1 = op * w[d], u1 = oq * w[d];
        s.bp[d][0] += op;
        s.bp[d][1] += t1;
        s.bp[d][2] = fma(t1, w[d], s.bp[d][2]);
        s.bq[d][0] += oq;
        s.bq[d][1] += u1;
        s.bq[d][2] = fma(u1, w[d], s.bq[d][2]);
    }
}

// One group of 4 consecutive observations of this lane's run: per observation an exact cell-membership check, the
// (rare, divergent) cell switch, then the straight-line arithmetic with all lanes reconverged.
template <typename T, int D>
__device__ __forceinline__ void lane_group(const PackedArgs<T, D>& a, LaneState<T, D>& s, const T (&xg)[D][4],
                                           const T (&yg)[4], const T* s_tab, const float* s_knots) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        T xx[D];
#pragma unroll
        for (int d = 0; d < D; ++d) xx[d] = xg[d][j];
        bool consumed = false;
        if (!lane_in_cell<T, D>(s, xx)) consumed = lane_switch<T, D>(a, s, xx, yg[j], s_tab, s_knots);
        if (!consumed) lane_math<T, D>(s, xx, yg[j]);
    }
}

constexpr int OBS_THREADS = 128;

template <typename T, int D>
__global__ void __launch_bounds__(OBS_THREADS, (sizeof(T) == 4 ? (D == 3 ? 4 : 5) : (D == 1 ? 4 : 2))) k_obs_b1(const __grid_constant__ PackedArgs<T, D> a) {
    extern __shared__ __align__(128) unsigned char smraw[];
    // [cell tables (T) | knots (float)], staged by one TMA bulk copy
    const T* s_tab = reinterpret_cast<const T*>(smraw);
    const float* s_knots = reinterpret_cast<const float*>(smraw + a.knots_byte_off);
    __shared__ __align__(8) uint64_t bar;
    __shared__ double red[32];

    if (threadIdx.x == 0) {
        mbar_init(&bar, 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(&bar, (uint32_t)a.table_bytes);
        bulk_g2s(smraw, a.tables, (uint32_t)a.table_bytes, &bar);
    }
    mbar_wait(&bar, 0);

    const int lane = threadIdx.x & 31;
    LaneState<T, D> s;
    s.valid = false;
    s.accE = (T)0;
#pragma unroll
    for (int d = 0; d < D; ++d) {
        s.c[d] = -1;
        s.tlo[d] = s.h[d] = s.rh[d] = (T)0;
        s.tlo_chk[d] = (T)INFINITY;      // nothing is inside the (empty) initial cell
        s.thi[d] = -(T)INFINITY;
#pragma unroll
        for (int k = 0; k < 3; ++k) { s.bp[d][k] = (T)0; s.bq[d][k] = (T)0; s.pe[d][k] = (T)0; s.qe[d][k] = (T)0; }
    }
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) { s.gm[i] = (T)0; s.am[i] = (T)0; }

    // persistent warps: every warp takes the next chunk (32 lanes x R observations) from a global counter, so the
    // data-dependent cost of the cell switches balances over the SMs
    const int groups = a.geo.R >> 2;
    bool first = true;                  // first chunk = the warp's global index, later ones from the counter (see bin_next_task)
    const unsigned int nwarps_all = gridDim.x * (blockDim.x >> 5);
    for (;;) {
        unsigned int chunk = 0;
        if (first) {
            chunk = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
            first = false;
        } else {
            if (lane == 0) chunk = atomicAdd(a.counter, 1u) + nwarps_all;
            chunk = __shfl_sync(0xffffffffu, chunk, 0);
        }
        if ((i64)chunk >= a.geo.nwarps) break;
        const i64 base = (i64)chunk * 32 * a.geo.R + lane * 4;
        T xa[D][4], ya[4], xb[D][4], yb[4];
#pragma unroll
        for (int d = 0; d < D; ++d) load4<T>(a.xp[d] + base, xa[d]);
        load4<T>(a.yp + base, ya);
        // software pipeline over groups of 4 observations: the loads of the next group are in flight while this one
        // is processed (one copy of the group code; rotating the buffers costs 3 register moves per observation)
#pragma unroll 1
        for (int gi = 0; gi < groups; ++gi) {
            if (gi + 1 < groups) {
                const i64 o = base + (i64)(gi + 1) * 128;
#pragma unroll
                for (int d = 0; d < D; ++d) load4<T>(a.xp[d] + o, xb[d]);
                load4<T>(a.yp + o, yb);
            }
            lane_group<T, D>(a, s, xa, ya, s_tab, s_knots);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
#pragma unroll
                for (int d = 0; d < D; ++d) xa[d][j] = xb[d][j];
                ya[j] = yb[j];
            }
        }
        lane_flush<T, D>(a, s, nullptr);
        s.valid = false;
#pragma unroll
        for (int d = 0; d < D; ++d) { s.tlo_chk[d] = (T)INFINITY; s.thi[d] = -(T)INFINITY; s.c[d] = -1; }
    }
    const double e = block_sum((double)s.accE, red);
    if (threadIdx.x == 0) {
        atomicAdd(a.gs + 0, e);
        if (blockIdx.x == 0) a.gs[1] = a.n_real;      // single writer; summed over ranks by the all-reduce
    }
}

// ---------------------------------------------------------------------------------------------------------
// Point prediction (the forward half of K1 at arbitrary test points, kronecker_structure.py:199-230 restricted to the
// marginals): mean = <kron phi_d(x*), alpha>,  var = kff - prod_d phi_d^T P_d phi_d + prod_d phi_d^T Q_d phi_d.
// Plain structure-of-arrays input in any order; one thread per test point.
// ---------------------------------------------------------------------------------------------------------
template <typename T, int D>
struct PredictArgs {
    const T* x[D];
    i64 n;
    MeshView mesh[D];
    int stride[D];
    int tab_off[D];
    const T* tab;            // per-cell tables (global memory)
    const T* alpha;
    const double* theta;     // l[D], s2[D], noise
    T* mean;
    T* var;
};

template <typename T, int D>
__global__ void __launch_bounds__(256) k_predict_b1(const __grid_constant__ PredictArgs<T, D> a) {
    T kff = (T)1;
#pragma unroll
    for (int d = 0; d < D; ++d) kff *= (T)a.theta[D + d];
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (i64)gridDim.x * blockDim.x) {
        int c[D];
        T w[D];
        bool all_in = true;
        T pp = (T)1, qq = (T)1;
#pragma unroll
        for (int d = 0; d < D; ++d) {
            const T xv = a.x[d][i];
            bool inside;
            c[d] = find_cell<T>(a.mesh[d].t, a.mesh[d].K, a.mesh[d].t0, a.mesh[d].inv_h, a.mesh[d].nearly_uniform, xv, inside);
            all_in = all_in && inside;
            const int n = a.mesh[d].K;
            const T* tb = a.tab + (a.tab_off[d] + c[d]);
            w[d] = div_by_cached_rcp(xv - (T)a.mesh[d].t[c[d]], tb[6 * n], tb[7 * n]);
            pp *= fma(fma(tb[2 * n], w[d], tb[n]), w[d], tb[0]);
            qq *= fma(fma(tb[5 * n], w[d], tb[4 * n]), w[d], tb[3 * n]);
        }
        T mu = (T)0, v = kff;
        if (all_in) {
            int base = 0;
#pragma unroll
            for (int d = 0; d < D; ++d) base += c[d] * a.stride[d];
#pragma unroll
            for (int corner = 0; corner < (1 << D); ++corner) {
                T wt = (T)1;
                int off = base;
#pragma unroll
                for (int d = 0; d < D; ++d) {
                    const bool hi = (corner >> (D - 1 - d)) & 1;
                    wt *= hi ? w[d] : ((T)1 - w[d]);
                    off += hi ? a.stride[d] : 0;
                }
                mu += wt * a.alpha[off];
            }
            v = kff - pp + qq;
        }
        a.mean[i] = mu;
        a.var[i] = v;
    }
}

// ---------------------------------------------------------------------------------------------------------
// K1 for the B0 (cell-integrated Matern-1/2) family: dense features phi_d(x) in R^{M_d} that depend on
// (l_d, s2_d).  This is the reference's own O(N (M + sum M_d^2)) dense algorithm (gridded_kronecker_structure.py:
// 1392-1407 + kronecker_structure.py:265-275) restated per tile of observations -- features live in shared memory and
// never reach HBM -- with the reverse pass fused in.  D <= 2 (as the reference).  It is the correctness baseline for
// this family; the tensor-core / semiseparable-scan forms (DESIGN.md section 7) replace it later.
//
// Per observation n:  mu = phi_1^T A phi_2,  p_d = phi_d^T P_d phi_d,  q_d = phi_d^T Q_d phi_d,  r = y - mu.
// Outputs (raw sums; 1/noise, ell_scale applied on the grid side):
//   g_alpha[i][j] += r phi_1[i] phi_2[j]
//   bP_d[i][j]    += (prod_{e!=d} p_e) phi_d[i] phi_d[j]        bQ_d likewise with q
//   E             += r^2 - prod p + prod q
//   G_l[d]        += sum_i gphi_d[i] dphi_d[i]/dl,   G_s[d] += sum_i gphi_d[i] phi_d[i]      (features depend on theta)
//        with gphi_d = r V_d + (prod_{e!=d} p_e) P_d phi_d - (prod_{e!=d} q_e) Q_d phi_d,  V_1 = A phi_2, V_2 = A^T phi_1
// ---------------------------------------------------------------------------------------------------------
constexpr int B0_TN = 4;        // observations per tile

template <typename T, int D>
struct B0Args {
    const T* x[D];
    const T* y;
    i64 n;
    MeshView mesh[D];
    int nd[D];               // M_d = K_d - 1 (B0 cells) or K_d (SVGP points)
    int family;              // VGGP_B0_GRIDDED, VGGP_SVGP_GRID or VGGP_VFF_GRID
    const double* theta;     // l[D], s2[D], noise
    const T* alpha;          // (M_1, M_2) row-major, obs dtype
    const double* P[D];
    const double* Q[D];
    T* galpha;
    double* gfac;            // per dim [bP (n_d^2) | bQ (n_d^2)], float64 whatever T: the gbuf block itself for float64
                             // observations, a plan-owned buffer rounded once into the gbuf for float32 ones
    i64 gfac_off[D];
    double* gs;              // [E, n, -, G_l[0..1], G_s[0..1]]
};

template <typename T, int D>
__global__ void __launch_bounds__(256) k_obs_b0(const __grid_constant__ B0Args<T, D> a) {
    extern __shared__ __align__(128) unsigned char smraw[];
    __shared__ double red[32];
    __shared__ T s_r[B0_TN], s_op[D][B0_TN], s_oq[D][B0_TN];
    // shared arrays, each [sum_d n_d][B0_TN]
    int off[D], ntot = 0;
#pragma unroll
    for (int d = 0; d < D; ++d) { off[d] = ntot; ntot += a.nd[d]; }
    T* phi = reinterpret_cast<T*>(smraw);
    T* dphi = phi + (size_t)ntot * B0_TN;
    T* V = dphi + (size_t)ntot * B0_TN;
    T* Zp = V + (size_t)ntot * B0_TN;
    T* Zq = Zp + (size_t)ntot * B0_TN;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const i64 ntiles = (a.n + B0_TN - 1) / B0_TN;
    double accE = 0.0, accGl[D], accGs[D];
#pragma unroll
    for (int d = 0; d < D; ++d) { accGl[d] = 0.0; accGs[d] = 0.0; }

    for (i64 tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const i64 n0 = tile * B0_TN;
        // ---- 1. features and their lengthscale derivative ----
#pragma unroll
        for (int d = 0; d < D; ++d) {
            const T l = (T)a.theta[d], s2 = (T)a.theta[D + d];
            for (int e = tid; e < a.nd[d] * B0_TN; e += blockDim.x) {
                const int k = e / B0_TN, t = e % B0_TN;
                T f = (T)0, df = (T)0;
                if (n0 + t < a.n && a.family == VGGP_VFF_GRID) {
                    // FourierBasisMatern12(x), fourier.py:16-19, 30-48, 58-88: cosines then sines on [a, b), exp(-r / l) outside
                    const int Kk = a.mesh[d].K, Mf = (Kk - 1) / 2;
                    const T xa = (T)a.mesh[d].t[0], xb = (T)a.mesh[d].t[Kk - 1];
                    const T xv = a.x[d][n0 + t];
                    if (xv >= xa && xv < xb) {
                        const int kf = k <= Mf ? k : k - Mf;
                        const T arg = ((T)6.283185307179586476925286766559 * (T)kf / (xb - xa)) * (xv - xa);
                        f = k <= Mf ? cos(arg) : sin(arg);
                    } else if (k <= Mf) {
                        const T r = fmin(fabs(xv - xa), fabs(xv - xb));
                        f = exp(-r / l);
                        df = f * r / (l * l);
                    }
                } else if (n0 + t < a.n && a.family == VGGP_SVGP_GRID) {
                    // k(z_k, x) of a ScaleKernel(MaternKernel(1/2)) and its lengthscale derivative (kronecker_structure.py:337-338)
                    const T A1 = fabs(a.x[d][n0 + t] - (T)a.mesh[d].t[k]);
                    f = s2 * exp(-A1 / l);
                    df = f * A1 / (l * l);
                } else if (n0 + t < a.n) {
                    const T xv = a.x[d][n0 + t];
                    const int idx = lower_bound_knots<T>(a.mesh[d].t, a.mesh[d].K, xv);
                    const T A1 = fabs(xv - (T)a.mesh[d].t[k]), A2 = fabs(xv - (T)a.mesh[d].t[k + 1]);
                    const T e1 = exp(-A1 / l), e2 = exp(-A2 / l);
                    const T g1 = e1 * ((T)1 + A1 / l), g2 = e2 * ((T)1 + A2 / l);     // d/dl of l exp(-A/l)
                    const int sgn = idx - k - 1;
                    if (sgn == 0) { f = (T)2 * l - (l * e1 + l * e2); df = (T)2 - (g1 + g2); }
                    else if (sgn > 0) { f = -(l * e1 - l * e2); df = -(g1 - g2); }
                    else { f = l * e1 - l * e2; df = g1 - g2; }
                    f *= s2;
                    df *= s2;
                }
                phi[(size_t)(off[d] + k) * B0_TN + t] = f;
                dphi[(size_t)(off[d] + k) * B0_TN + t] = df;
            }
        }
        __syncthreads();
        // ---- 2. V_d: contraction of alpha with the other dimension's features; Zp, Zq ----
        if (D == 1) {
            for (int e = tid; e < a.nd[0] * B0_TN; e += blockDim.x) V[e] = a.alpha[e / B0_TN];
        } else {
            const int n1 = a.nd[0], n2 = a.nd[D - 1];
            for (int i = warp; i < n1; i += nwarps) {            // V_1[i][t] = sum_j A[i][j] phi_2[j][t]
                T acc[B0_TN];
#pragma unroll
                for (int t = 0; t < B0_TN; ++t) acc[t] = (T)0;
                for (int j = lane; j < n2; j += 32) {
                    const T av = a.alpha[(i64)i * n2 + j];
#pragma unroll
                    for (int t = 0; t < B0_TN; ++t) acc[t] += av * phi[(size_t)(off[D - 1] + j) * B0_TN + t];
                }
#pragma unroll
                for (int t = 0; t < B0_TN; ++t) {
                    const T v = warp_sum(acc[t]);
                    if (lane == 0) V[(size_t)(off[0] + i) * B0_TN + t] = v;
                }
            }
            for (int j = tid; j < n2; j += blockDim.x) {         // V_2[j][t] = sum_i A[i][j] phi_1[i][t]
                T acc[B0_TN];
#pragma unroll
                for (int t = 0; t < B0_TN; ++t) acc[t] = (T)0;
                for (int i = 0; i < n1; ++i) {
                    const T av = a.alpha[(i64)i * n2 + j];
#pragma unroll
                    for (int t = 0; t < B0_TN; ++t) acc[t] += av * phi[(size_t)(off[0] + i) * B0_TN + t];
                }
#pragma unroll
                for (int t = 0; t < B0_TN; ++t) V[(size_t)(off[D - 1] + j) * B0_TN + t] = acc[t];
            }
        }
#pragma unroll
        for (int d = 0; d < D; ++d) {
            const int nn = a.nd[d];
            for (int i = warp; i < nn; i += nwarps) {
                T ap[B0_TN], aq[B0_TN];
#pragma unroll
                for (int t = 0; t < B0_TN; ++t) { ap[t] = (T)0; aq[t] = (T)0; }
                for (int j = lane; j < nn; j += 32) {
                    const T pv = (T)a.P[d][(i64)i * nn + j], qv = (T)a.Q[d][(i64)i * nn + j];
#pragma unroll
                    for (int t = 0; t < B0_TN; ++t) {
                        const T f = phi[(size_t)(off[d] + j) * B0_TN + t];
                        ap[t] += pv * f;
                        aq[t] += qv * f;
                    }
                }
#pragma unroll
                for (int t = 0; t < B0_TN; ++t) {
                    const T vp = warp_sum(ap[t]), vq = warp_sum(aq[t]);
                    if (lane == 0) {
                        Zp[(size_t)(off[d] + i) * B0_TN + t] = vp;
                        Zq[(size_t)(off[d] + i) * B0_TN + t] = vq;
                    }
                }
            }
        }
        __syncthreads();
        // ---- 3. per-observation scalars: one warp per observation of the tile ----
        if (warp < B0_TN) {
            const int t = warp;
            T mu = (T)0, p[D], q[D];
#pragma unroll
            for (int d = 0; d < D; ++d) { p[d] = (T)0; q[d] = (T)0; }
            for (int i = lane; i < a.nd[0]; i += 32) mu += phi[(size_t)(off[0] + i) * B0_TN + t] * V[(size_t)(off[0] + i) * B0_TN + t];
            mu = warp_sum(mu);
#pragma unroll
            for (int d = 0; d < D; ++d) {
                for (int i = lane; i < a.nd[d]; i += 32) {
                    const T f = phi[(size_t)(off[d] + i) * B0_TN + t];
                    p[d] += f * Zp[(size_t)(off[d] + i) * B0_TN + t];
                    q[d] += f * Zq[(size_t)(off[d] + i) * B0_TN + t];
                }
                p[d] = warp_sum(p[d]);
                q[d] = warp_sum(q[d]);
            }
            if (lane == 0) {
                const bool live = (n0 + t < a.n);
                const T r = live ? a.y[n0 + t] - mu : (T)0;
                T pp = (T)1, qq = (T)1;
#pragma unroll
                for (int d = 0; d < D; ++d) { pp *= p[d]; qq *= q[d]; }
                if (live) accE += (double)(r * r - pp + qq);
                s_r[t] = r;
#pragma unroll
                for (int d = 0; d < D; ++d) {
                    T op = (T)1, oq = (T)1;
#pragma unroll
                    for (int e = 0; e < D; ++e)
                        if (e != d) { op *= p[e]; oq *= q[e]; }
                    s_op[d][t] = live ? op : (T)0;
                    s_oq[d][t] = live ? oq : (T)0;
                }
            }
        }
        __syncthreads();
        // ---- 4. reverse pass ----
#pragma unroll
        for (int d = 0; d < D; ++d) {
            double gl = 0.0, gsv = 0.0;
            for (int e = tid; e < a.nd[d] * B0_TN; e += blockDim.x) {
                const int t = e % B0_TN;
                const size_t o = (size_t)off[d] * B0_TN + e;
                const T gphi = s_r[t] * V[o] + s_op[d][t] * Zp[o] - s_oq[d][t] * Zq[o];
                gl += (double)(gphi * dphi[o]);
                gsv += (double)(gphi * phi[o]);
            }
            accGl[d] += gl;
            accGs[d] += gsv;
            const int nn = a.nd[d];
            // float64 sums: the l / s2 gradients go through P bP P and Q bQ Q, which amplify a relative error of bQ by about four
            // orders of magnitude; float32 atomics over the tiles put the 1-D s2 gradient ~ 1 % off the oracle, varying with their order
            double* gP = a.gfac + a.gfac_off[d];
            double* gQ = gP + (i64)nn * nn;
            for (int e = tid; e < nn * nn; e += blockDim.x) {
                const int i = e / nn, j = e % nn;
                double vp = 0.0, vq = 0.0;
#pragma unroll
                for (int t = 0; t < B0_TN; ++t) {
                    const double ff = (double)phi[(size_t)(off[d] + i) * B0_TN + t] * phi[(size_t)(off[d] + j) * B0_TN + t];
                    vp += s_op[d][t] * ff;
                    vq += s_oq[d][t] * ff;
                }
                atomicAdd(gP + e, vp);
                atomicAdd(gQ + e, vq);
            }
        }
        if (D == 1) {
            for (int i = tid; i < a.nd[0]; i += blockDim.x) {
                T v = (T)0;
#pragma unroll
                for (int t = 0; t < B0_TN; ++t) v += s_r[t] * phi[(size_t)i * B0_TN + t];
                atomicAdd(a.galpha + i, v);
            }
        } else {
            const int n1 = a.nd[0], n2 = a.nd[D - 1];
            for (int e = tid; e < n1 * n2; e += blockDim.x) {
                const int i = e / n2, j = e % n2;
                T v = (T)0;
#pragma unroll
                for (int t = 0; t < B0_TN; ++t)
                    v += s_r[t] * phi[(size_t)(off[0] + i) * B0_TN + t] * phi[(size_t)(off[D - 1] + j) * B0_TN + t];
                atomicAdd(a.galpha + e, v);
            }
        }
        __syncthreads();
    }
    double e = block_sum(accE, red);
    if (tid == 0) atomicAdd(a.gs + 0, e);
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const double gl = block_sum(accGl[d], red);
        const double gsv = block_sum(accGs[d], red);
        if (tid == 0) {
            atomicAdd(a.gs + 3 + d, gl);
            atomicAdd(a.gs + 5 + d, gsv);
        }
    }
    if (tid == 0 && blockIdx.x == 0) a.gs[1] = (double)a.n;
}

}  // namespace vggp
