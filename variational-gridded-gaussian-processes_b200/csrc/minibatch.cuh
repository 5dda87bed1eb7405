// Epoch-shuffled minibatches in the binned layout (include/vggp.h, vggp_epoch_bin_prepare / _pack).
//
// Sampling law: epoch e of rank r draws a pseudo-random permutation pi of the rank's n observations; batch b (b < P) is
// { i : pi(i) in [b B, (b + 1) B) }, the remainder n - P B is dropped.  pi is a keyed bijection computed inline: a balanced
// Feistel network of MB_ROUNDS rounds on the smallest even number of bits k with 2^k >= n, round function = a 32-bit mixing
// hash of (seed, epoch, rank, round, half), cycle-walking until the value is below n.  tests/test_minibatch.py restates it
// in numpy.
//
// One pass bins all P batches of an epoch: composite key (batch, cell) with the permutation fused into the key kernel, one
// radix sort, then a device run planner that reproduces plan_bins (binplan.hpp) within every batch:
//   segment heads of the sorted keys -> each non-empty (batch, cell) with its start and count
//   ceil(count / run_cap) runs of equal share per inside cell, emitted in cell order
//   a stable radix sort of the runs by (batch, longest first): ties keep cell order, as std::stable_sort does there
//   32 runs per task, R = first run's length rounded up to a multiple of 4, task offsets as a per-batch exclusive scan
// Only the per-batch totals go back to the host; the pack writes each batch's tables and gathers its data with the gather
// kernels of the single-set layout (k_bin_gather / k_b0s_gather, the sorted indices offset to the batch).
#ifndef VGGP_MINIBATCH_CUH
#define VGGP_MINIBATCH_CUH
#include <stdint.h>
#include "obs_binned.cuh"
#include "b0scan.cuh"

namespace vggp {

constexpr int MB_ROUNDS = 4;
constexpr int MB_TOTALS = 5;    // per batch in the caller's totals array: tasks, runs, n_inside, data elements, section offset

__host__ __device__ __forceinline__ uint32_t mb_mix32(uint32_t x) {
    x ^= x >> 16;
    x *= 0x7feb352du;
    x ^= x >> 15;
    x *= 0x846ca68bu;
    x ^= x >> 16;
    return x;
}

struct MbPerm {
    uint32_t n;                    // observations of this rank (< 2^31)
    int half;                      // bits of one Feistel half
    uint32_t mask;
    uint32_t key[MB_ROUNDS];       // round keys: hash of (seed, epoch, rank, round)
};

inline MbPerm mb_perm_make(int64_t n, uint64_t seed, uint64_t epoch, int rank) {
    MbPerm p;
    p.n = (uint32_t)n;
    int k = 2;
    while (((int64_t)1 << k) < n) k += 2;
    p.half = k / 2;
    p.mask = (uint32_t)(((uint64_t)1 << p.half) - 1);
    uint32_t h = mb_mix32((uint32_t)seed);
    h = mb_mix32(h ^ (uint32_t)(seed >> 32));
    h = mb_mix32(h ^ (uint32_t)epoch);
    h = mb_mix32(h ^ (uint32_t)(epoch >> 32));
    h = mb_mix32(h ^ (uint32_t)rank);
    for (int r = 0; r < MB_ROUNDS; ++r) p.key[r] = mb_mix32(h ^ (uint32_t)(r + 1) * 0x9e3779b9u);
    return p;
}

__host__ __device__ __forceinline__ uint32_t mb_perm(const MbPerm& p, uint32_t i) {
    uint32_t v = i;
    do {
        uint32_t L = v >> p.half, R = v & p.mask;
#pragma unroll
        for (int r = 0; r < MB_ROUNDS; ++r) {
            const uint32_t F = mb_mix32(p.key[r] ^ R) & p.mask;
            const uint32_t nL = R;
            R = L ^ F;
            L = nL;
        }
        v = (L << p.half) | R;
    } while (v >= p.n);
    return v;
}

// key of observation i: (batch, cell) as batch * ncell_keys + cell, or P * ncell_keys for a dropped observation.  The cell is
// the flat inside-mesh cell with `ncells` for outside (B1, the cell of k_cell_keys), or the extended cell of k_b0s_keys.
template <typename T, int D>
struct MbKeyArgs {
    const T* x[D];
    MeshView mesh[D];
    MbPerm perm;
    uint32_t B, P;
    uint64_t ncell_keys;           // cells + 1 (B1: the outside key) or extended cells
    int ext;
};
template <typename T, int D, typename KT>
__global__ void __launch_bounds__(256) k_mb_keys(const __grid_constant__ MbKeyArgs<T, D> a, KT* __restrict__ keys,
                                                 uint32_t* __restrict__ idx) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < (i64)a.perm.n; i += (i64)gridDim.x * blockDim.x) {
        const uint32_t q = mb_perm(a.perm, (uint32_t)i);
        const uint32_t b = q / a.B;
        KT key;
        if (b >= a.P) {
            key = (KT)a.P * (KT)a.ncell_keys;
        } else {
            uint32_t cell = 0;
            bool all_in = true;
#pragma unroll
            for (int d = 0; d < D; ++d) {
                if (a.ext) {
                    cell = cell * (uint32_t)(a.mesh[d].K + 1) + (uint32_t)lower_bound_knots<T>(a.mesh[d].t, a.mesh[d].K, a.x[d][i]);
                } else {
                    bool inside;
                    const int c = find_cell<T>(a.mesh[d].t, a.mesh[d].K, a.mesh[d].t0, a.mesh[d].inv_h,
                                               a.mesh[d].nearly_uniform, a.x[d][i], inside);
                    cell = cell * (uint32_t)(a.mesh[d].K - 1) + (uint32_t)c;
                    all_in = all_in && inside;
                }
            }
            if (!all_in) cell = (uint32_t)(a.ncell_keys - 1);
            key = (KT)b * (KT)a.ncell_keys + (KT)cell;
        }
        keys[i] = key;
        idx[i] = (uint32_t)i;
    }
}

// flags[i] = 1 at the first sorted position of every (batch, cell) segment among the m = P B kept positions; flags[m] = 0
template <typename KT>
__global__ void __launch_bounds__(256) k_mb_heads(const KT* __restrict__ keys, i64 m, uint32_t* __restrict__ flags) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i <= m; i += (i64)gridDim.x * blockDim.x)
        flags[i] = (i < m && (i == 0 || keys[i] != keys[i - 1])) ? 1u : 0u;
}

// seg_start[s] = first position of segment s, seg_start[S] = m (S = segid[m] segments)
__global__ void __launch_bounds__(256) k_mb_seg_starts(const uint32_t* __restrict__ flags, const uint32_t* __restrict__ segid,
                                                       i64 m, uint32_t* __restrict__ seg_start) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i <= m; i += (i64)gridDim.x * blockDim.x) {
        if (i == m) seg_start[segid[m]] = (uint32_t)m;
        else if (flags[i]) seg_start[segid[i]] = (uint32_t)i;
    }
}

// runs per segment (0 for the outside key of B1) and per-batch sums of runs and of streamed observations
template <typename KT>
__global__ void __launch_bounds__(256) k_mb_seg_runs(const KT* __restrict__ keys, const uint32_t* __restrict__ seg_start,
                                                     const uint32_t* __restrict__ n_seg, uint64_t ncell_keys, uint64_t outside,
                                                     uint32_t cap, uint32_t* __restrict__ seg_nruns,
                                                     unsigned long long* __restrict__ batch_runs,
                                                     unsigned long long* __restrict__ batch_inside) {
    const i64 S = *n_seg;
    for (i64 s = (i64)blockIdx.x * blockDim.x + threadIdx.x; s < S; s += (i64)gridDim.x * blockDim.x) {
        const uint32_t start = seg_start[s], cnt = seg_start[s + 1] - start;
        const KT key = keys[start];
        const uint64_t b = (uint64_t)(key / (KT)ncell_keys), c = (uint64_t)(key % (KT)ncell_keys);
        if (c == outside) { seg_nruns[s] = 0u; continue; }
        const uint32_t k = (cnt + cap - 1) / cap;
        seg_nruns[s] = k;
        atomicAdd(batch_runs + b, (unsigned long long)k);
        atomicAdd(batch_inside + b, (unsigned long long)cnt);
    }
}

// run r of the epoch (cell order within each batch): its cell, length, start relative to its batch, and the key of the
// (batch, longest first) sort
template <typename KT>
__global__ void __launch_bounds__(256) k_mb_emit_runs(const KT* __restrict__ keys, const uint32_t* __restrict__ seg_start,
                                                      const uint32_t* __restrict__ run_base, const uint32_t* __restrict__ n_seg,
                                                      i64 n_runs, uint64_t ncell_keys, uint32_t cap, uint32_t B,
                                                      KT* __restrict__ run_key, uint32_t* __restrict__ run_idx,
                                                      uint32_t* __restrict__ run_cell, int32_t* __restrict__ run_len,
                                                      uint32_t* __restrict__ run_start) {
    const uint32_t S = *n_seg;
    for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < n_runs; r += (i64)gridDim.x * blockDim.x) {
        uint32_t lo = 0, hi = S;                  // last segment s with run_base[s] <= r (run_base[S] = n_runs > r)
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (run_base[mid] <= (uint32_t)r) lo = mid; else hi = mid;
        }
        const uint32_t s = lo, i = (uint32_t)r - run_base[s];
        const uint32_t start = seg_start[s], cnt = seg_start[s + 1] - start;
        const KT key = keys[start];
        const uint64_t b = (uint64_t)(key / (KT)ncell_keys);
        const uint32_t k = (cnt + cap - 1) / cap, base = cnt / k, extra = cnt % k;
        const uint32_t len = base + (i < extra ? 1u : 0u);
        run_cell[r] = (uint32_t)(key % (KT)ncell_keys);
        run_len[r] = (int32_t)len;
        run_start[r] = start - (uint32_t)(b * B) + i * base + (i < extra ? i : extra);
        run_key[r] = (KT)b * (KT)(cap + 1) + (KT)(cap - len);
        run_idx[r] = (uint32_t)r;
    }
}

// tasks per batch = ceil(runs / 32); entry P = 0 (the exclusive scan then ends in the total)
__global__ void __launch_bounds__(256) k_mb_batch_tasks(const unsigned long long* __restrict__ batch_runs, i64 P,
                                                        unsigned long long* __restrict__ batch_tasks) {
    for (i64 b = (i64)blockIdx.x * blockDim.x + threadIdx.x; b <= P; b += (i64)gridDim.x * blockDim.x)
        batch_tasks[b] = b < P ? (batch_runs[b] + 31) / 32 : 0ull;
}

__device__ __forceinline__ i64 mb_batch_of(const unsigned long long* __restrict__ base, i64 P, unsigned long long v) {
    i64 lo = 0, hi = P;                           // last b with base[b] <= v
    while (hi - lo > 1) {
        const i64 mid = (lo + hi) >> 1;
        if (base[mid] <= v) lo = mid; else hi = mid;
    }
    return lo;
}

// padded run length and streamed elements of every task (global task index g over all batches; slots past the total are 0)
__global__ void __launch_bounds__(256) k_mb_task_R(const unsigned long long* __restrict__ task_base,
                                                   const unsigned long long* __restrict__ run_off, const uint32_t* __restrict__ run_sorted,
                                                   const int32_t* __restrict__ run_len, i64 P, i64 n_slots, int D,
                                                   int32_t* __restrict__ task_R, long long* __restrict__ task_elems) {
    const unsigned long long T = task_base[P];
    for (i64 g = (i64)blockIdx.x * blockDim.x + threadIdx.x; g <= n_slots; g += (i64)gridDim.x * blockDim.x) {
        if ((unsigned long long)g >= T) { task_elems[g] = 0; continue; }
        const i64 b = mb_batch_of(task_base, P, (unsigned long long)g);
        const unsigned long long t = (unsigned long long)g - task_base[b];
        const int R = (run_len[run_sorted[run_off[b] + 32 * t]] + 3) / 4 * 4;
        task_R[g] = R;
        task_elems[g] = (long long)32 * R * (D + 1);
    }
}

// per-batch totals for the host: tasks, runs, streamed observations, data elements
__global__ void __launch_bounds__(256) k_mb_totals(const unsigned long long* __restrict__ batch_runs,
                                                   const unsigned long long* __restrict__ batch_inside,
                                                   const unsigned long long* __restrict__ task_base,
                                                   const long long* __restrict__ task_goff, i64 P, long long* __restrict__ out) {
    for (i64 b = (i64)blockIdx.x * blockDim.x + threadIdx.x; b < P; b += (i64)gridDim.x * blockDim.x) {
        out[4 * b + 0] = (long long)(task_base[b + 1] - task_base[b]);
        out[4 * b + 1] = (long long)batch_runs[b];
        out[4 * b + 2] = (long long)batch_inside[b];
        out[4 * b + 3] = task_goff[task_base[b + 1]] - task_goff[task_base[b]];
    }
}

// the tables of every batch, one thread per run slot: task_off / task_R (lane 0), run_cell / run_n / run_start.
// sec[6 b + j]: absolute byte offsets of batch b's sections task_off, task_R, run_cell, run_n, run_start, data.
__global__ void __launch_bounds__(256) k_mb_tables(const unsigned long long* __restrict__ task_base,
                                                   const long long* __restrict__ task_goff, const int32_t* __restrict__ task_R,
                                                   const unsigned long long* __restrict__ run_off,
                                                   const unsigned long long* __restrict__ batch_runs,
                                                   const uint32_t* __restrict__ run_sorted, const uint32_t* __restrict__ run_cell,
                                                   const int32_t* __restrict__ run_len, const uint32_t* __restrict__ run_start,
                                                   const long long* __restrict__ sec, i64 P, unsigned char* __restrict__ buf) {
    const i64 nslots = (i64)task_base[P] * 32;
    for (i64 slot = (i64)blockIdx.x * blockDim.x + threadIdx.x; slot < nslots; slot += (i64)gridDim.x * blockDim.x) {
        const i64 g = slot / 32;
        const int lane = (int)(slot % 32);
        const i64 b = mb_batch_of(task_base, P, (unsigned long long)g);
        const i64 t = g - (i64)task_base[b];
        const long long* o = sec + 6 * b;
        if (lane == 0) {
            reinterpret_cast<i64*>(buf + o[0])[t] = task_goff[g] - task_goff[task_base[b]];
            reinterpret_cast<int32_t*>(buf + o[1])[t] = task_R[g];
        }
        const i64 j = 32 * t + lane;
        uint32_t cell = BIN_EMPTY, start = 0u;
        int32_t len = 0;
        if (j < (i64)batch_runs[b]) {
            const uint32_t r = run_sorted[run_off[b] + j];
            cell = run_cell[r];
            len = run_len[r];
            start = run_start[r];
        }
        reinterpret_cast<uint32_t*>(buf + o[2])[j] = cell;
        reinterpret_cast<int32_t*>(buf + o[3])[j] = len;
        reinterpret_cast<uint32_t*>(buf + o[4])[j] = start;
    }
}

}  // namespace vggp
#endif
