// select.cu -- ordering primitives of the sampler bookkeeping (SURVEY.md K3, K7):
//   * stable LSD radix sort of (fp64 key, int32 index) pairs  -> np.argsort replacement used by
//     Rejection._merge_batch (samplers.py:232-237) and weighted_sample_quantile (utils.py:397);
//   * row gather (the fancy-index permutation `v[:] = v[sort_mask]`, samplers.py:236-237, and
//     `batch[node][accepted]`, samplers.py:228-230);
//   * weighted sample quantile (methods/utils.py:379-411).
//
// Keys are distances (>= 0, possibly +inf / NaN).  They are mapped to order-preserving uint64
// (NaN last, like NumPy) and sorted 8 bits per pass.  All working sets at the BASELINE sizes
// (<= 2e6 pairs = 24 MB) are L2 resident, so the sort is latency/issue bound, not HBM bound;
// passes whose digit is constant over all keys (typical for the high exponent bits of
// distances) degenerate to a copy.
#include "eqweight.h"
#include "pairwise.cuh"

namespace elfi {

constexpr int SORT_CHUNK = 1024;   // keys per warp sub-chunk
constexpr int SORT_WARPS = 8;      // warps per block

__device__ __forceinline__ uint64_t key_to_u64(double d) {
    if (d != d) return ~uint64_t(0);                 // NaN sorts last
    uint64_t u = static_cast<uint64_t>(__double_as_longlong(d));
    return (u >> 63) ? ~u : (u | (uint64_t(1) << 63));
}
__device__ __forceinline__ double u64_to_key(uint64_t u) {
    if (u == ~uint64_t(0)) return __longlong_as_double(0x7ff8000000000000LL);
    u = (u >> 63) ? (u & ~(uint64_t(1) << 63)) : ~u;
    return __longlong_as_double(static_cast<long long>(u));
}

// keys -> u64, vals -> iota, and the 8 x 256 global digit histograms in one read.
__global__ void __launch_bounds__(256)
sort_prepare_kernel(const double* __restrict__ keys, int64_t n, uint64_t* __restrict__ ukeys,
                    int32_t* __restrict__ vals, uint32_t* __restrict__ ghist) {
    __shared__ uint32_t h[8 * 256];
    for (int i = threadIdx.x; i < 8 * 256; i += blockDim.x) h[i] = 0;
    __syncthreads();
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint64_t u = key_to_u64(keys[i]);
        ukeys[i] = u;
        vals[i] = int32_t(i);
#pragma unroll
        for (int p = 0; p < 8; ++p) atomicAdd(&h[p * 256 + ((u >> (8 * p)) & 255)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 8 * 256; i += blockDim.x)
        if (h[i]) atomicAdd(&ghist[i], h[i]);
}

// A pass is trivial when one bin of its histogram holds all n keys.
__device__ __forceinline__ bool pass_trivial(const uint32_t* ghist, int pass, int64_t n,
                                             uint64_t first_key) {
    return ghist[pass * 256 + ((first_key >> (8 * pass)) & 255)] == uint32_t(n);
}

// Per-warp digit counts of each sub-chunk, written digit-major: whist[digit * nw + warp].
__global__ void __launch_bounds__(SORT_WARPS * 32)
sort_upsweep_kernel(const uint64_t* __restrict__ ukeys, int64_t n, int pass, int64_t nw,
                    const uint32_t* __restrict__ ghist, uint32_t* __restrict__ whist) {
    if (pass_trivial(ghist, pass, n, ukeys[0])) return;
    __shared__ uint32_t h[SORT_WARPS][256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t gw = int64_t(blockIdx.x) * SORT_WARPS + warp;
    for (int i = lane; i < 256; i += 32) h[warp][i] = 0;
    __syncwarp();
    if (gw < nw) {
        const int64_t lo = gw * SORT_CHUNK;
        const int64_t hi = (lo + SORT_CHUNK < n) ? lo + SORT_CHUNK : n;
        for (int64_t i = lo + lane; i < hi; i += 32)
            atomicAdd(&h[warp][(ukeys[i] >> (8 * pass)) & 255], 1u);
        __syncwarp();
        for (int d = lane; d < 256; d += 32) whist[int64_t(d) * nw + gw] = h[warp][d];
    }
}

// Block d turns whist[d * nw + *] into global start offsets for digit d.
__global__ void __launch_bounds__(1024)
sort_scan_kernel(const uint64_t* __restrict__ ukeys, int64_t n, int pass, int64_t nw,
                 const uint32_t* __restrict__ ghist, uint32_t* __restrict__ whist) {
    if (pass_trivial(ghist, pass, n, ukeys[0])) return;
    __shared__ uint32_t warp_tot[32];
    __shared__ uint32_t carry_s;
    const int d = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    // base = number of keys with a smaller digit
    uint32_t part = 0;
    for (int i = tid; i < d; i += 1024) part += ghist[pass * 256 + i];
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) warp_tot[wid] = part;
    __syncthreads();
    if (tid == 0) {
        uint32_t t = 0;
        for (int i = 0; i < 32; ++i) t += warp_tot[i];
        carry_s = t;
    }
    __syncthreads();
    uint32_t* row = whist + int64_t(d) * nw;
    for (int64_t base = 0; base < nw; base += 1024) {
        const int64_t i = base + tid;
        const uint32_t v = i < nw ? row[i] : 0u;
        uint32_t incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        __syncthreads();  // warp_tot / carry_s reads of the previous round are done
        if (lane == 31) warp_tot[wid] = incl;
        __syncthreads();
        uint32_t woff = 0;
        for (int k = 0; k < wid; ++k) woff += warp_tot[k];
        const uint32_t carry = carry_s;
        if (i < nw) row[i] = carry + woff + incl - v;
        __syncthreads();
        if (tid == 1023) carry_s = carry + woff + incl;
    }
}

// Stable scatter: each warp walks its sub-chunk in order; equal digits keep their order
// (match_any groups + rank by lane id).  Trivial passes copy.
__global__ void __launch_bounds__(SORT_WARPS * 32)
sort_scatter_kernel(const uint64_t* __restrict__ kin, const int32_t* __restrict__ vin, int64_t n,
                    int pass, int64_t nw, const uint32_t* __restrict__ ghist,
                    const uint32_t* __restrict__ whist, uint64_t* __restrict__ kout,
                    int32_t* __restrict__ vout) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t gw = int64_t(blockIdx.x) * SORT_WARPS + warp;
    if (gw >= nw) return;
    const int64_t lo = gw * SORT_CHUNK;
    const int64_t hi = (lo + SORT_CHUNK < n) ? lo + SORT_CHUNK : n;
    if (pass_trivial(ghist, pass, n, kin[0])) {
        for (int64_t i = lo + lane; i < hi; i += 32) {
            kout[i] = kin[i];
            vout[i] = vin[i];
        }
        return;
    }
    __shared__ uint32_t off[SORT_WARPS][256];
    for (int d = lane; d < 256; d += 32) off[warp][d] = whist[int64_t(d) * nw + gw];
    __syncwarp();
    for (int64_t base = lo; base < hi; base += 32) {
        const int64_t i = base + lane;
        const bool valid = i < hi;
        const uint64_t k = valid ? kin[i] : 0;
        const int32_t v = valid ? vin[i] : 0;
        const uint32_t digit = valid ? uint32_t((k >> (8 * pass)) & 255) : 256u + lane;
        const uint32_t peers = __match_any_sync(0xffffffffu, digit);
        const uint32_t rank = __popc(peers & ((1u << lane) - 1));
        uint32_t pos = 0;
        if (valid) pos = off[warp][digit] + rank;
        __syncwarp();
        if (valid && rank == 0) off[warp][digit] += __popc(peers);
        __syncwarp();
        if (valid) {
            kout[pos] = k;
            vout[pos] = v;
        }
    }
}

__global__ void sort_finish_kernel(const uint64_t* __restrict__ ukeys, const int32_t* __restrict__ vals,
                                   int64_t n, double* __restrict__ keys_out,
                                   int32_t* __restrict__ perm_out) {
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (keys_out) keys_out[i] = u64_to_key(ukeys[i]);
        if (perm_out) perm_out[i] = vals[i];
    }
}

struct SortScratch {
    uint64_t* k[2];
    int32_t* v[2];
    uint32_t* ghist;
    uint32_t* whist;
    int64_t nw;
};

static size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

static size_t sort_scratch_bytes(int64_t n) {
    const int64_t nw = (n + SORT_CHUNK - 1) / SORT_CHUNK;
    return 2 * align256(size_t(n) * 8) + 2 * align256(size_t(n) * 4) + align256(8 * 256 * 4) +
           align256(size_t(256) * nw * 4);
}

static SortScratch carve_sort(uint8_t* base, int64_t n) {
    SortScratch s;
    s.nw = (n + SORT_CHUNK - 1) / SORT_CHUNK;
    size_t o = 0;
    for (int i = 0; i < 2; ++i) { s.k[i] = reinterpret_cast<uint64_t*>(base + o); o += align256(size_t(n) * 8); }
    for (int i = 0; i < 2; ++i) { s.v[i] = reinterpret_cast<int32_t*>(base + o); o += align256(size_t(n) * 4); }
    s.ghist = reinterpret_cast<uint32_t*>(base + o); o += align256(8 * 256 * 4);
    s.whist = reinterpret_cast<uint32_t*>(base + o);
    return s;
}

// Sorts ascending; results are left in s.k[0] / s.v[0] (8 passes = even number of swaps).
int sort_pairs_device(const double* keys, int64_t n, const SortScratch& s, int sm_count,
                      cudaStream_t stream) {
    ELFI_CUDA_OK(cudaMemsetAsync(s.ghist, 0, 8 * 256 * 4, stream));
    int blocks = int((n + 256 * 8 - 1) / (256 * 8));
    if (blocks > sm_count * 4) blocks = sm_count * 4;
    if (blocks < 1) blocks = 1;
    sort_prepare_kernel<<<blocks, 256, 0, stream>>>(keys, n, s.k[0], s.v[0], s.ghist);
    const unsigned wblocks = unsigned((s.nw + SORT_WARPS - 1) / SORT_WARPS);
    int cur = 0;
    for (int pass = 0; pass < 8; ++pass) {
        sort_upsweep_kernel<<<wblocks, SORT_WARPS * 32, 0, stream>>>(s.k[cur], n, pass, s.nw, s.ghist, s.whist);
        sort_scan_kernel<<<256, 1024, 0, stream>>>(s.k[cur], n, pass, s.nw, s.ghist, s.whist);
        sort_scatter_kernel<<<wblocks, SORT_WARPS * 32, 0, stream>>>(
            s.k[cur], s.v[cur], n, pass, s.nw, s.ghist, s.whist, s.k[cur ^ 1], s.v[cur ^ 1]);
        cur ^= 1;
    }
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

// dst[i, 0:width] = src[idx[i], 0:width]
__global__ void __launch_bounds__(256)
gather_rows_kernel(const double* __restrict__ src, int64_t ld_src, const int32_t* __restrict__ idx,
                   int64_t n, int64_t width, double* __restrict__ dst, int64_t ld_dst) {
    const int64_t total = n * width;
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < total; t += stride) {
        const int64_t i = t / width, j = t - i * width;
        dst[i * ld_dst + j] = src[int64_t(idx[i]) * ld_src + j];
    }
}

// Accepted rows of a batch -> tail of a candidate buffer, with the counts read on the device.
// Up to APPEND_MAX_SRC source arrays (each (B, width_k) with its own leading dimension) are laid
// side by side in the packed destination row.
constexpr int APPEND_MAX_SRC = 8;
struct AppendSources {
    const double* ptr[APPEND_MAX_SRC];
    int64_t ld[APPEND_MAX_SRC];
    int32_t width[APPEND_MAX_SRC];
    int32_t col0[APPEND_MAX_SRC];
    int32_t n_src, total_width;
};

__global__ void __launch_bounds__(256)
accept_append_kernel(const int32_t* __restrict__ acc_idx, const int64_t* __restrict__ n_acc,
                     AppendSources src, double* __restrict__ dst, int64_t ld_dst, int64_t capacity,
                     const int64_t* __restrict__ count) {
    const int64_t base = *count;
    int64_t room = capacity - base;
    if (room < 0) room = 0;
    const int64_t rows = *n_acc < room ? *n_acc : room;
    const int64_t total = rows * src.total_width;
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < total; t += stride) {
        const int64_t j = t / src.total_width;
        const int c = int(t - j * src.total_width);
        const int64_t row = acc_idx ? int64_t(acc_idx[j]) : j;
        int k = 0;
#pragma unroll
        for (int q = 1; q < APPEND_MAX_SRC; ++q)
            if (q < src.n_src && c >= src.col0[q]) k = q;
        dst[(base + j) * ld_dst + c] = src.ptr[k][row * src.ld[k] + (c - src.col0[k])];
    }
}

// count += rows appended; dropped[0] += rows that did not fit (runs after accept_append_kernel)
__global__ void accept_count_kernel(const int64_t* __restrict__ n_acc, int64_t capacity,
                                    int64_t* __restrict__ count, int64_t* __restrict__ dropped) {
    int64_t room = capacity - *count;
    if (room < 0) room = 0;
    const int64_t rows = *n_acc < room ? *n_acc : room;
    if (dropped) *dropped += *n_acc - rows;
    *count += rows;
}

// Two-source gather for the running top-n merge: logical row r < nA is A[r], otherwise
// B[mapB ? mapB[r - nA] : r - nA]  (B = the new batch, mapB = its accepted row indices).
__global__ void __launch_bounds__(256)
gather2_rows_kernel(const double* __restrict__ A, int64_t ldA, int64_t nA,
                    const double* __restrict__ Bm, int64_t ldB, const int32_t* __restrict__ mapB,
                    const int32_t* __restrict__ perm, int64_t n, int64_t width,
                    double* __restrict__ dst, int64_t ld_dst) {
    const int64_t total = n * width;
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < total; t += stride) {
        const int64_t i = t / width, j = t - i * width;
        const int64_t r = perm ? perm[i] : i;
        double v;
        if (r < nA) {
            v = A[r * ldA + j];
        } else {
            const int64_t rb = mapB ? int64_t(mapB[r - nA]) : (r - nA);
            v = Bm[rb * ldB + j];
        }
        dst[i * ld_dst + j] = v;
    }
}

// keys of the virtual concatenation [A (nA rows); B[mapB] (nB rows)] of a top-n merge; a key is
// the last of kw columns (the reference ranks by the last distance column, samplers.py:232)
__global__ void __launch_bounds__(256)
merge_keys_kernel(const double* __restrict__ keysA, int64_t ldA, int64_t nA,
                  const double* __restrict__ keysB, int64_t ldB, const int32_t* __restrict__ mapB,
                  int64_t nB, double* __restrict__ out) {
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < nA + nB; i += stride) {
        if (i < nA) {
            out[i] = keysA[i * ldA];
        } else {
            const int64_t rb = mapB ? int64_t(mapB[i - nA]) : (i - nA);
            out[i] = keysB[rb * ldB];
        }
    }
}

// ---- weighted quantile ---------------------------------------------------------------------
// The reference normalises with np.sum (pairwise order) and accumulates with np.cumsum
// (strictly sequential); with equal weights and round alphas (e.g. SMC round 0, alpha = 0.5)
// alpha sits exactly on a cumulative weight, so the rounding of that sequential sum decides
// which order statistic is returned.  Both are therefore reproduced in the reference's order:
// one warp streams the data through shared memory (coalesced loads, double buffered) and lane 0
// performs the order-dependent adds.  Cost ~5 ns per element (1e6 weights: a few ms per
// generation), negligible next to the O(N^2) weight update it feeds.
constexpr int WQ_CHUNK = 1024;

__device__ __forceinline__ void wq_stage(const double* __restrict__ src, int64_t n, int64_t base,
                                         double* buf, int lane) {
    for (int t = lane; t < WQ_CHUNK; t += 32) {
        const int64_t i = base + t;
        buf[t] = i < n ? src[i] : 0.0;
    }
}

// out[0] = np.sum(w) in NumPy's pairwise order (w == NULL: n, exactly).  One warp: the control
// state of the pairwise tree is uniform, lane k < 8 owns the strided accumulator r[k] of the
// current <=128-term leaf, the fold ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) is three shuffle steps.
__global__ void __launch_bounds__(32)
wq_total_kernel(const double* __restrict__ w, int64_t n64, double* __restrict__ out) {
    __shared__ double buf[2][WQ_CHUNK];
    __shared__ double left_val[32];
    __shared__ int pending_right[32];
    const int lane = threadIdx.x;
    const int n = int(n64);
    if (w == nullptr) {
        if (lane == 0) out[0] = double(n);
        return;
    }
    uint32_t has_left = 0;
    int depth = 0, leaf_start = 0, leaf_end = 0, tail_start = 0;
    bool in_tail = false;
    double r = 0.0, res = 0.0;   // r: lanes 0..7; res: meaningful in every lane (kept uniform)
    auto descend = [&](int start, int len) {
        while (len > 128) {
            int n2 = len / 2;
            n2 -= n2 % 8;
            if (lane == 0) pending_right[depth] = len - n2;
            has_left &= ~(1u << depth);
            ++depth;
            len = n2;
        }
        __syncwarp();
        leaf_start = start;
        leaf_end = start + len;
        tail_start = len < 8 ? start : start + (len - len % 8);
        in_tail = len < 8;
        res = 0.0;
    };
    auto fold = [&]() -> double {
        double t = r + __shfl_down_sync(0xffffffffu, r, 1);      // lanes 0,2,4,6: r_k + r_{k+1}
        t = t + __shfl_down_sync(0xffffffffu, t, 2);             // lanes 0,4
        t = t + __shfl_down_sync(0xffffffffu, t, 4);             // lane 0
        return __shfl_sync(0xffffffffu, t, 0);
    };
    auto leaf_value = [&]() -> double { return in_tail ? res : fold(); };
    descend(0, n);
    wq_stage(w, n64, 0, buf[0], lane);
    __syncwarp();
    int cur = 0;
    for (int base = 0; base < n; base += WQ_CHUNK, cur ^= 1) {
        if (int64_t(base) + WQ_CHUNK < n64) wq_stage(w, n64, int64_t(base) + WQ_CHUNK, buf[cur ^ 1], lane);
        const int lim = (n - base) < WQ_CHUNK ? (n - base) : WQ_CHUNK;
        for (int j = 0; j < lim; j += 8) {
            const int j0 = base + j;
            const int cnt = (lim - j) < 8 ? (lim - j) : 8;
            if (j0 == leaf_end) {                       // close the leaf, open the next one
                double v = leaf_value();
                bool opened = false;
                while (depth > 0 && !opened) {
                    if (!((has_left >> (depth - 1)) & 1u)) {
                        if (lane == 0) left_val[depth - 1] = v;
                        has_left |= 1u << (depth - 1);
                        __syncwarp();
                        descend(j0, pending_right[depth - 1]);
                        opened = true;
                    } else {
                        v = left_val[depth - 1] + v;
                        --depth;
                    }
                }
            }
            if (!in_tail && j0 == tail_start && tail_start != leaf_start) {
                res = fold();
                in_tail = true;
            }
            if (in_tail) {
                for (int k = 0; k < cnt; ++k) res = res + buf[cur][j + k];   // uniform, sequential
            } else if (lane < 8) {
                const double t = buf[cur][j + lane];
                r = (j0 == leaf_start) ? t : r + t;
            }
        }
        __syncwarp();
    }
    double v = leaf_value();
    while (depth > 0) {
        v = left_val[depth - 1] + v;
        --depth;
    }
    if (lane == 0) out[0] = v;
}

// ws[i] = w[perm[i]] / total   (weights[index] of utils.py:401-402; exact IEEE division)
__global__ void wq_normalise_kernel(const double* __restrict__ w, const int32_t* __restrict__ perm,
                                    int64_t n, const double* __restrict__ total,
                                    double* __restrict__ ws) {
    const double t = total[0];
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
        ws[i] = (w ? w[perm[i]] : 1.0) / t;
}

// index_alpha = #{ k in [0, n-2] : cumsum(ws)[k] < alpha }, cumsum strictly sequential
// (utils.py:403-406; the last cumulative weight is forced to 1.0 there, hence n-2).
// Lane 0 carries the running sum; terms are fetched eight at a time so the shared-memory
// latency is paid once per eight dependent adds.
__global__ void __launch_bounds__(32)
wq_seqscan_kernel(const double* __restrict__ ws, int64_t n, double alpha,
                  const uint64_t* __restrict__ ukeys, double* __restrict__ out) {
    __shared__ double buf[2][WQ_CHUNK];
    __shared__ int done_s;
    const int lane = threadIdx.x;
    int64_t count = 0;
    double c = 0.0;
    if (lane == 0) done_s = (alpha == 0.0) ? 1 : 0;
    wq_stage(ws, n, 0, buf[0], lane);
    __syncwarp();
    int cur = 0;
    for (int64_t base = 0; base < n - 1; base += WQ_CHUNK, cur ^= 1) {
        if (done_s) break;
        if (base + WQ_CHUNK < n - 1) wq_stage(ws, n, base + WQ_CHUNK, buf[cur ^ 1], lane);
        if (lane == 0) {
            const int lim = int((n - 1 - base) < WQ_CHUNK ? (n - 1 - base) : WQ_CHUNK);
            int j = 0;
            for (; j + 8 <= lim; j += 8) {
                double t[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) t[k] = buf[cur][j + k];
                int below = 0;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    c = __dadd_rn(c, t[k]);
                    below += (c < alpha) ? 1 : 0;   // non-decreasing: a prefix of the 8 is below
                }
                count += below;
                if (below < 8) { done_s = 1; break; }
            }
            if (!done_s) {
                for (; j < lim; ++j) {
                    c = __dadd_rn(c, buf[cur][j]);
                    if (c < alpha) ++count; else { done_s = 1; break; }
                }
            }
        }
        __syncwarp();
    }
    if (lane == 0) {
        out[0] = u64_to_key(ukeys[count]);
        out[1] = double(count);
    }
}

// ---- per-row sort (order-statistic summaries, e.g. the g-and-k model: np.sort(y, axis=1)) ---------
// One warp per row: keys go to shared memory as order-preserving u64 (NaN last, like np.sort),
// padded to a power of two, bitonic network with __syncwarp between stages.
__global__ void __launch_bounds__(256)
rowsort_kernel(const double* __restrict__ X, int64_t ldX, int64_t B, int n, int npow2,
               double* __restrict__ out, int64_t ld_out) {
    extern __shared__ uint64_t sk_all[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint64_t* sk = sk_all + size_t(warp) * npow2;
    for (int64_t row = int64_t(blockIdx.x) * 8 + warp; row < B; row += int64_t(gridDim.x) * 8) {
        for (int i = lane; i < npow2; i += 32) sk[i] = i < n ? key_to_u64(X[row * ldX + i]) : ~uint64_t(0);
        __syncwarp();
        for (int k = 2; k <= npow2; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int t = lane; t < (npow2 >> 1); t += 32) {
                    const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                    const int l = i | j;
                    const bool up = (i & k) == 0;
                    const uint64_t a = sk[i], b = sk[l];
                    if ((a > b) == up) { sk[i] = b; sk[l] = a; }
                }
                __syncwarp();
            }
        }
        for (int i = lane; i < n; i += 32) out[row * ld_out + i] = u64_to_key(sk[i]);
        __syncwarp();
    }
}

// Rows of up to 512 keys: the same network with the keys in REGISTERS.  Lane L holds the KPL
// consecutive elements L*KPL .. L*KPL + KPL-1, so compare-exchange distances j < KPL stay inside
// a thread and j >= KPL are one shuffle per key with lane L ^ (j / KPL): no shared memory, no
// bank conflicts, no __syncwarp between stages (the shared-memory network above spends its time
// there: 6.9 ms for 1e6 x 256).  A lane's elements are contiguous in memory: 16-byte loads and
// stores when the row is aligned and entirely inside [0, n).
__device__ __forceinline__ uint64_t shfl_xor_u64(uint64_t v, int m) {
    uint32_t lo = uint32_t(v), hi = uint32_t(v >> 32);
    asm volatile("shfl.sync.bfly.b32 %0, %0, %2, 0x1f, 0xffffffff;\n\t"
                 "shfl.sync.bfly.b32 %1, %1, %2, 0x1f, 0xffffffff;"
                 : "+r"(lo), "+r"(hi) : "r"(m));
    return (uint64_t(hi) << 32) | lo;
}

template <int KPL>
__device__ __forceinline__ void bitonic_in_registers(uint64_t (&key)[KPL], int lane) {
    constexpr int N = KPL * 32;
#pragma unroll
    for (int k = 2; k <= N; k <<= 1) {
        // sort direction of the k-block the element sits in: bit k of i = L*KPL + r
        const bool lane_up = (k >= N) ? true : ((lane & (k >= KPL ? k / KPL : 1)) == 0);
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= KPL) {
                const int m = j / KPL;
                const bool keep_min = ((lane & m) == 0) == lane_up;
#pragma unroll
                for (int r = 0; r < KPL; ++r) {
                    const uint64_t o = shfl_xor_u64(key[r], m);
                    key[r] = ((o < key[r]) == keep_min) ? o : key[r];
                }
            } else {
#pragma unroll
                for (int r = 0; r < KPL; ++r) {
                    if ((r & j) == 0) {
                        const bool up = (k < KPL) ? ((r & k) == 0) : lane_up;
                        const uint64_t a = key[r], b = key[r | j];
                        const bool sw = (a > b) == up;
                        key[r] = sw ? b : a;
                        key[r | j] = sw ? a : b;
                    }
                }
            }
        }
    }
}

template <int KPL>
__global__ void __launch_bounds__(256)
rowsort_regs_kernel(const double* __restrict__ X, int64_t ldX, int64_t B, int n_,
                    double* __restrict__ out, int64_t ld_out, int vec_in, int vec_out) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = int64_t(gridDim.x) * 8;
    const int first = lane * KPL;
    // block-uniform loop bounds: the shuffles below sit in provably convergent code (a per-warp
    // row loop makes ptxas bracket every shuffle with WARPSYNC.COLLECTIVE / ENDCOLLECTIVE)
    for (int64_t base = int64_t(blockIdx.x) * 8; base < B; base += nwarps) {
        const int64_t row = base + (threadIdx.x >> 5);
        const bool live = row < B;
        const int n = live ? n_ : 0;
        const bool whole = first + KPL <= n;
        uint64_t key[KPL];
        const double* x = X + row * ldX + first;
        bool loaded = false;
        if constexpr (KPL >= 2) {
            if (vec_in && whole) {
#pragma unroll
                for (int r = 0; r < KPL; r += 2) {
                    const double2 v = __ldg(reinterpret_cast<const double2*>(x + r));
                    key[r] = key_to_u64(v.x);
                    key[r + 1] = key_to_u64(v.y);
                }
                loaded = true;
            }
        }
        if (!loaded) {
#pragma unroll
            for (int r = 0; r < KPL; ++r)
                key[r] = first + r < n ? key_to_u64(__ldg(x + r)) : ~uint64_t(0);
        }
        bitonic_in_registers<KPL>(key, lane);
        double* y = out + row * ld_out + first;
        bool stored = false;
        if constexpr (KPL >= 2) {
            if (vec_out && whole) {
#pragma unroll
                for (int r = 0; r < KPL; r += 2)
                    *reinterpret_cast<double2*>(y + r) =
                        make_double2(u64_to_key(key[r]), u64_to_key(key[r + 1]));
                stored = true;
            }
        }
        if (!stored) {
#pragma unroll
            for (int r = 0; r < KPL; ++r)
                if (first + r < n) y[r] = u64_to_key(key[r]);
        }
    }
}

template <int KPL>
static void launch_rowsort_regs(const double* X, int64_t ldX, int64_t B, int n, double* out,
                                int64_t ld_out, int sm_count, cudaStream_t stream) {
    int64_t blocks = (B + 7) / 8;
    if (blocks > int64_t(sm_count) * 8) blocks = int64_t(sm_count) * 8;
    const int vec_in = (reinterpret_cast<uintptr_t>(X) % 16 == 0) && (ldX % 2 == 0);
    const int vec_out = (reinterpret_cast<uintptr_t>(out) % 16 == 0) && (ld_out % 2 == 0);
    rowsort_regs_kernel<KPL><<<unsigned(blocks), 256, 0, stream>>>(X, ldX, B, n, out, ld_out,
                                                                   vec_in, vec_out);
}

// ---- fast path of the weighted quantile -----------------------------------------------------------
// A blocked parallel scan gives cumulative weights c~_k whose distance to the reference's
// sequential np.cumsum values is bounded by eps = 4 n 2^-53 (both are within ~n u of the exact
// real sums).  If no c~_k falls within eps of alpha the selected order statistic is provably the
// same as the reference's and the sequential kernel above is skipped; otherwise (alpha sitting on
// a cumulative weight: equal weights + round alpha) the exact path decides.
__global__ void __launch_bounds__(1024)
wq_par_block_sums_kernel(const double* __restrict__ w, const int32_t* __restrict__ perm, int64_t n,
                         double* __restrict__ partial) {
    __shared__ double ws[32];
    const int64_t lo = int64_t(blockIdx.x) * 4096;
    double acc = 0.0;
    for (int k = 0; k < 4; ++k) {
        const int64_t i = lo + k * 1024 + threadIdx.x;
        if (i < n) acc += w ? w[perm[i]] : 1.0;
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = ws[threadIdx.x];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) partial[blockIdx.x] = v;
    }
}

// exclusive scan of the block sums (single block); total in partial[nb]; zeroes the two counters
__global__ void __launch_bounds__(1024)
wq_par_scan_kernel(double* __restrict__ partial, int64_t nb, int32_t* __restrict__ counts) {
    __shared__ double ws[32];
    __shared__ double carry_s;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) { carry_s = 0.0; counts[0] = 0; counts[1] = 0; }
    __syncthreads();
    for (int64_t base = 0; base < nb; base += 1024) {
        const int64_t i = base + tid;
        const double v = i < nb ? partial[i] : 0.0;
        double incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const double t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) ws[wid] = incl;
        __syncthreads();
        double woff = 0.0;
        for (int k = 0; k < wid; ++k) woff += ws[k];
        const double carry = carry_s;
        if (i < nb) partial[i] = carry + woff + incl - v;
        __syncthreads();
        if (tid == 1023) carry_s = carry + woff + incl;
        __syncthreads();
    }
    if (tid == 0) partial[nb] = carry_s;
}

// counts[0] = #{k <= n-2 : c~_k < alpha - eps}, counts[1] = #{k <= n-2 : c~_k < alpha + eps}
__global__ void __launch_bounds__(1024)
wq_par_count_kernel(const double* __restrict__ w, const int32_t* __restrict__ perm, int64_t n,
                    const double* __restrict__ partial, int64_t nb, double alpha, double eps,
                    int32_t* __restrict__ counts) {
    __shared__ double ws[32];
    __shared__ double carry_s;
    __shared__ int c0_s, c1_s;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const double total = partial[nb];
    if (tid == 0) { carry_s = partial[blockIdx.x]; c0_s = 0; c1_s = 0; }
    __syncthreads();
    int l0 = 0, l1 = 0;
    const int64_t lo = int64_t(blockIdx.x) * 4096;
    for (int k = 0; k < 4; ++k) {
        const int64_t i = lo + k * 1024 + tid;
        const double v = i < n ? (w ? w[perm[i]] : 1.0) : 0.0;
        double incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const double t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) ws[wid] = incl;
        __syncthreads();
        double woff = 0.0;
        for (int q = 0; q < wid; ++q) woff += ws[q];
        const double carry = carry_s;
        const double c = (carry + woff + incl) / total;
        if (i < n - 1) {
            l0 += (c < alpha - eps) ? 1 : 0;
            l1 += (c < alpha + eps) ? 1 : 0;
        }
        __syncthreads();
        if (tid == 1023) carry_s = carry + woff + incl;
        __syncthreads();
    }
    for (int o = 16; o > 0; o >>= 1) {
        l0 += __shfl_xor_sync(0xffffffffu, l0, o);
        l1 += __shfl_xor_sync(0xffffffffu, l1, o);
    }
    if (lane == 0) { atomicAdd(&c0_s, l0); atomicAdd(&c1_s, l1); }
    __syncthreads();
    if (tid == 0) { atomicAdd(&counts[0], c0_s); atomicAdd(&counts[1], c1_s); }
}

__global__ void wq_pick_kernel(const uint64_t* __restrict__ ukeys, int64_t idx, double* __restrict__ out) {
    out[0] = u64_to_key(ukeys[idx]);
    out[1] = double(idx);
}

}  // namespace elfi

extern "C" {

int elfi_b200_sort_pairs_f64(elfi_b200_ctx* ctx, const double* keys, int64_t n,
                             double* keys_sorted, int32_t* perm, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx != nullptr, "sort: ctx is NULL");
    ELFI_REQUIRE(n >= 0 && n < (int64_t(1) << 31), "sort: n=%lld out of range", (long long)n);
    if (n == 0) return ELFI_B200_OK;
    ELFI_REQUIRE(keys != nullptr, "sort: keys is NULL");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    uint8_t* base = static_cast<uint8_t*>(ctx_scratch(ctx, sort_scratch_bytes(n)));
    if (!base) return ELFI_B200_ERR_NOMEM;
    SortScratch s = carve_sort(base, n);
    int rc = sort_pairs_device(keys, n, s, ctx->sm_count, stream);
    if (rc) return rc;
    int blocks = int((n + 255) / 256);
    if (blocks > ctx->sm_count * 8) blocks = ctx->sm_count * 8;
    sort_finish_kernel<<<blocks, 256, 0, stream>>>(s.k[0], s.v[0], n, keys_sorted, perm);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_gather_rows_f64(elfi_b200_ctx* ctx, const double* src, int64_t ld_src,
                              const int32_t* idx, int64_t n, int64_t width, double* dst,
                              int64_t ld_dst, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx != nullptr, "gather: ctx is NULL");
    ELFI_REQUIRE(n >= 0 && width >= 1 && ld_src >= width && ld_dst >= width, "gather: bad shape");
    if (n == 0) return ELFI_B200_OK;
    ELFI_REQUIRE(src && idx && dst, "gather: NULL argument");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    int64_t blocks = (n * width + 255) / 256;
    if (blocks > int64_t(ctx->sm_count) * 16) blocks = int64_t(ctx->sm_count) * 16;
    gather_rows_kernel<<<unsigned(blocks), 256, 0, stream>>>(src, ld_src, idx, n, width, dst, ld_dst);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_gather2_rows_f64(elfi_b200_ctx* ctx, const double* A, int64_t ldA, int64_t nA,
                               const double* Bm, int64_t ldB, const int32_t* mapB,
                               const int32_t* perm, int64_t n, int64_t width, double* dst,
                               int64_t ld_dst, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx != nullptr, "gather2: ctx is NULL");
    ELFI_REQUIRE(n >= 0 && nA >= 0 && width >= 1 && ld_dst >= width, "gather2: bad shape");
    if (n == 0) return ELFI_B200_OK;
    ELFI_REQUIRE(dst != nullptr && (nA == 0 || A != nullptr), "gather2: NULL argument");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    int64_t blocks = (n * width + 255) / 256;
    if (blocks > int64_t(ctx->sm_count) * 16) blocks = int64_t(ctx->sm_count) * 16;
    gather2_rows_kernel<<<unsigned(blocks), 256, 0, stream>>>(A, ldA, nA, Bm, ldB, mapB, perm, n,
                                                             width, dst, ld_dst);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_topn_merge_f64(elfi_b200_ctx* ctx, const double* keysA, int64_t ld_keysA, int64_t nA,
                             const double* keysB, int64_t ld_keysB, const int32_t* mapB, int64_t nB,
                             int64_t n_keep, int64_t n_out, const double* const* A_host,
                             const int64_t* ldA_host, const double* const* B_host,
                             const int64_t* ldB_host, const int64_t* width_host,
                             double* const* dst_host, const int64_t* ld_dst_host, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx != nullptr, "topn_merge: ctx is NULL");
    ELFI_REQUIRE(nA >= 0 && nB >= 0 && n_keep >= 0 && n_keep <= nA + nB && n_out >= 0,
                 "topn_merge: bad sizes (nA=%lld nB=%lld n_keep=%lld)", (long long)nA, (long long)nB,
                 (long long)n_keep);
    const int64_t n = nA + nB;
    ELFI_REQUIRE(n < (int64_t(1) << 31), "topn_merge: too many rows");
    if (n == 0 || n_keep == 0) return ELFI_B200_OK;
    ELFI_REQUIRE((nA == 0 || keysA) && (nB == 0 || keysB), "topn_merge: keys are NULL");
    ELFI_REQUIRE(n_out == 0 || (A_host && ldA_host && B_host && ldB_host && width_host && dst_host &&
                                ld_dst_host), "topn_merge: output descriptors are NULL");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    const size_t sort_bytes = sort_scratch_bytes(n);
    uint8_t* base = static_cast<uint8_t*>(ctx_scratch(ctx, sort_bytes + align256(size_t(n) * 8) + 256));
    if (!base) return ELFI_B200_ERR_NOMEM;
    SortScratch s = carve_sort(base, n);
    double* keys = reinterpret_cast<double*>(base + sort_bytes);
    int blocks = int((n + 255) / 256);
    if (blocks > ctx->sm_count * 8) blocks = ctx->sm_count * 8;
    merge_keys_kernel<<<blocks, 256, 0, stream>>>(keysA, ld_keysA, nA, keysB, ld_keysB, mapB, nB, keys);
    int rc = sort_pairs_device(keys, n, s, ctx->sm_count, stream);
    if (rc) return rc;
    const int32_t* perm = s.v[0];
    for (int64_t k = 0; k < n_out; ++k) {
        const int64_t width = width_host[k];
        ELFI_REQUIRE(width >= 1 && dst_host[k] && ld_dst_host[k] >= width &&
                     (nA == 0 || (A_host[k] && ldA_host[k] >= width)) &&
                     (nB == 0 || (B_host[k] && ldB_host[k] >= width)),
                     "topn_merge: bad descriptor of output %lld", (long long)k);
        int64_t gb = (n_keep * width + 255) / 256;
        if (gb > int64_t(ctx->sm_count) * 16) gb = int64_t(ctx->sm_count) * 16;
        gather2_rows_kernel<<<unsigned(gb), 256, 0, stream>>>(A_host[k], ldA_host[k], nA, B_host[k],
                                                              ldB_host[k], mapB, perm, n_keep, width,
                                                              dst_host[k], ld_dst_host[k]);
    }
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_accept_append_f64(elfi_b200_ctx* ctx, const int32_t* acc_idx, const int64_t* n_acc,
                                int64_t max_rows, int64_t n_src, const double* const* src_host,
                                const int64_t* ld_src_host, const int64_t* width_host, double* dst,
                                int64_t ld_dst, int64_t capacity, int64_t* count, int64_t* dropped,
                                void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && n_acc && src_host && ld_src_host && width_host && dst && count,
                 "accept_append: NULL argument");
    ELFI_REQUIRE(n_src >= 1 && n_src <= APPEND_MAX_SRC, "accept_append: 1..%d sources", APPEND_MAX_SRC);
    ELFI_REQUIRE(max_rows >= 0 && capacity >= 0, "accept_append: bad shape");
    AppendSources src;
    memset(&src, 0, sizeof(src));
    src.n_src = int32_t(n_src);
    int64_t col = 0;
    for (int k = 0; k < n_src; ++k) {
        ELFI_REQUIRE(src_host[k] && width_host[k] >= 1 && ld_src_host[k] >= width_host[k],
                     "accept_append: bad source %d", k);
        src.ptr[k] = src_host[k];
        src.ld[k] = ld_src_host[k];
        src.width[k] = int32_t(width_host[k]);
        src.col0[k] = int32_t(col);
        col += width_host[k];
    }
    ELFI_REQUIRE(col <= ld_dst && col < (int64_t(1) << 30), "accept_append: ld_dst < total width");
    src.total_width = int32_t(col);
    if (max_rows == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    int64_t blocks = (max_rows * col + 255) / 256;
    if (blocks > int64_t(ctx->sm_count) * 8) blocks = int64_t(ctx->sm_count) * 8;
    accept_append_kernel<<<unsigned(blocks), 256, 0, stream>>>(acc_idx, n_acc, src, dst, ld_dst,
                                                              capacity, count);
    accept_count_kernel<<<1, 1, 0, stream>>>(n_acc, capacity, count, dropped);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

// One batch of a threshold-mode rejection round in ONE call: distances + acceptance + compaction
// (elfi_b200_dist_euclid_thr[_dev]_f64) and the append of the accepted rows [d | extra sources]
// to the candidate buffer (elfi_b200_accept_append_f64); four launches, no synchronisation.
extern "C" int elfi_b200_dist_euclid_thr_f64(elfi_b200_ctx*, const double*, int64_t, int64_t, int64_t,
                                             const double*, const double*, int64_t, const double*,
                                             double*, int32_t*, int64_t*, void*);
extern "C" int elfi_b200_dist_euclid_thr_dev_f64(elfi_b200_ctx*, const double*, int64_t, int64_t,
                                                 int64_t, const double*, const double*, int64_t,
                                                 const double*, double*, int32_t*, int64_t*, void*);

int elfi_b200_rejection_batch_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B,
                                  int64_t D, const double* obs, const double* W, int64_t K,
                                  const double* thr_host, const double* thr_dev, double* d_out,
                                  int32_t* acc_idx, int64_t* n_acc, int64_t n_extra,
                                  const double* const* extra_host, const int64_t* ld_extra_host,
                                  const int64_t* width_extra_host, double* dst, int64_t ld_dst,
                                  int64_t capacity, int64_t* count, int64_t* dropped,
                                  void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && acc_idx && n_acc && d_out, "rejection_batch: NULL argument");
    ELFI_REQUIRE((thr_host != nullptr) != (thr_dev != nullptr),
                 "rejection_batch: thresholds on the host OR on the device");
    ELFI_REQUIRE(n_extra >= 0 && n_extra < APPEND_MAX_SRC, "rejection_batch: 0..%d extra sources",
                 APPEND_MAX_SRC - 1);
    int rc = thr_host
        ? elfi_b200_dist_euclid_thr_f64(ctx, S, ldS, B, D, obs, W, K, thr_host, d_out, acc_idx, n_acc,
                                        stream_)
        : elfi_b200_dist_euclid_thr_dev_f64(ctx, S, ldS, B, D, obs, W, K, thr_dev, d_out, acc_idx,
                                            n_acc, stream_);
    if (rc) return rc;
    const double* src[APPEND_MAX_SRC];
    int64_t ld[APPEND_MAX_SRC], width[APPEND_MAX_SRC];
    src[0] = d_out; ld[0] = K; width[0] = K;
    for (int64_t k = 0; k < n_extra; ++k) {
        src[k + 1] = extra_host[k];
        ld[k + 1] = ld_extra_host[k];
        width[k + 1] = width_extra_host[k];
    }
    return elfi_b200_accept_append_f64(ctx, acc_idx, n_acc, B, n_extra + 1, src, ld, width, dst,
                                       ld_dst, capacity, count, dropped, stream_);
}

int elfi_b200_wquantile_f64(elfi_b200_ctx* ctx, const double* x, const double* w, int64_t n,
                            double alpha, double* out, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx != nullptr && x != nullptr && out != nullptr, "wquantile: NULL argument");
    ELFI_REQUIRE(n >= 1 && n < (int64_t(1) << 31), "wquantile: n=%lld out of range", (long long)n);
    ELFI_REQUIRE(alpha >= 0.0 && alpha <= 1.0, "wquantile: alpha=%g outside [0, 1]", alpha);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    const size_t sort_bytes = sort_scratch_bytes(n);
    const size_t extra = align256(size_t(n + 2) * 8) + 256;
    uint8_t* base = static_cast<uint8_t*>(ctx_scratch(ctx, sort_bytes + extra));
    if (!base) return ELFI_B200_ERR_NOMEM;
    SortScratch s = carve_sort(base, n);
    double* ws = reinterpret_cast<double*>(base + sort_bytes);
    double* total = reinterpret_cast<double*>(base + sort_bytes + align256(size_t(n) * 8));
    int rc = sort_pairs_device(x, n, s, ctx->sm_count, stream);
    if (rc) return rc;
    if (w == nullptr && alpha > 0.0) {
        // equal weights: the position in NumPy's sequential cumulative sum is known in closed form
        // (eqweight.h), so neither a scan nor a host round trip is needed
        wq_pick_kernel<<<1, 1, 0, stream>>>(s.k[0], equal_weight_cum_index(n, alpha) - 1, out);
        ELFI_CUDA_OK(cudaGetLastError());
        return ELFI_B200_OK;
    }
    if (alpha > 0.0 && n > 1) {
        // fast path: parallel scan + error bound; falls through to the exact kernels only when
        // alpha is within eps of a cumulative weight
        const int64_t nb = (n + 4095) / 4096;
        double* partial = ws;                               // reuse: nb + 1 doubles (<= n)
        int32_t* counts = reinterpret_cast<int32_t*>(total) + 4;
        const double eps = (4.0 * double(n) + 64.0) * 1.1102230246251565e-16;
        wq_par_block_sums_kernel<<<unsigned(nb), 1024, 0, stream>>>(w, s.v[0], n, partial);
        wq_par_scan_kernel<<<1, 1024, 0, stream>>>(partial, nb, counts);
        wq_par_count_kernel<<<unsigned(nb), 1024, 0, stream>>>(w, s.v[0], n, partial, nb, alpha, eps, counts);
        int32_t hc[2] = {0, -1};
        ELFI_CUDA_OK(cudaMemcpyAsync(hc, counts, 8, cudaMemcpyDeviceToHost, stream));
        ELFI_CUDA_OK(cudaStreamSynchronize(stream));
        if (hc[0] == hc[1]) {
            wq_pick_kernel<<<1, 1, 0, stream>>>(s.k[0], int64_t(hc[0]), out);
            ELFI_CUDA_OK(cudaGetLastError());
            return ELFI_B200_OK;
        }
    }
    wq_total_kernel<<<1, 32, 0, stream>>>(w, n, total);
    int blocks = int((n + 255) / 256);
    if (blocks > ctx->sm_count * 8) blocks = ctx->sm_count * 8;
    wq_normalise_kernel<<<blocks, 256, 0, stream>>>(w, s.v[0], n, total, ws);
    wq_seqscan_kernel<<<1, 32, 0, stream>>>(ws, n, alpha, s.k[0], out);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_rowsort_f64(elfi_b200_ctx* ctx, const double* X, int64_t ldX, int64_t B, int64_t n,
                          double* out, int64_t ld_out, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && (B == 0 || (X && out)), "rowsort: NULL argument");
    ELFI_REQUIRE(B >= 0 && n >= 1 && n <= 2048 && ldX >= n && ld_out >= n,
                 "rowsort: bad shape (1 <= n <= 2048)");
    if (B == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    int npow2 = 2;
    while (npow2 < n) npow2 <<= 1;
    if (npow2 <= 512) {
        const int kpl = npow2 <= 32 ? 1 : npow2 / 32;
        switch (kpl) {
            case 1: launch_rowsort_regs<1>(X, ldX, B, int(n), out, ld_out, ctx->sm_count, stream); break;
            case 2: launch_rowsort_regs<2>(X, ldX, B, int(n), out, ld_out, ctx->sm_count, stream); break;
            case 4: launch_rowsort_regs<4>(X, ldX, B, int(n), out, ld_out, ctx->sm_count, stream); break;
            case 8: launch_rowsort_regs<8>(X, ldX, B, int(n), out, ld_out, ctx->sm_count, stream); break;
            default: launch_rowsort_regs<16>(X, ldX, B, int(n), out, ld_out, ctx->sm_count, stream); break;
        }
        ELFI_CUDA_OK(cudaGetLastError());
        return ELFI_B200_OK;
    }
    const size_t smem = size_t(8) * npow2 * 8;
    ELFI_CUDA_OK(cudaFuncSetAttribute(rowsort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      int(smem)));
    int64_t blocks = (B + 7) / 8;
    if (blocks > int64_t(ctx->sm_count) * 8) blocks = int64_t(ctx->sm_count) * 8;
    rowsort_kernel<<<unsigned(blocks), 256, smem, stream>>>(X, ldX, B, int(n), npow2, out, ld_out);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

}  // extern "C"
