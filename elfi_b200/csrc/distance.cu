// distance.cu -- Euclidean / nested weighted distances fused with the acceptance test
// (SURVEY.md K1, K2, K4).
//
// Reference semantics restated (see include/elfi_b200.h for the call sites):
//   d[i,k] = sqrt( sum_j W[k,j] * ((S[i,j]-obs[j]) * (S[i,j]-obs[j])) ), j strictly ascending,
// one rounding per multiply and per add (SciPy's cdist 'euclidean' with optional `w`).
// The CUDA code uses __dmul_rn/__dadd_rn/__dsub_rn so nvcc cannot contract into FMA.
//
// Algorithmic traffic per particle: D*8 bytes read + K*8 bytes written (+ 1 bit of mask).
// Roofline: HBM.  The fp64 pipe does 3 (unweighted) or 4 (weighted) issue slots per element,
// ~20 % of the memory time at D=128 on B200, so the kernel is bandwidth bound as long as
// the TMA pipeline keeps >= ~45 KiB in flight per SM (see rowstream.cuh).
#include "rowstream.cuh"

extern "C" int elfi_b200_colmoments_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B,
                                        int64_t D, double* out, void* stream);

namespace elfi {

struct DistParams {
    const double* obs;   // (D)
    const double* W;     // (K, D) or nullptr
    double* d_out;       // (B, K)
    uint32_t* mask;      // ceil(B/32) words or nullptr
    int K;
    int has_thr;
    const double* shift_src;   // fused column moments: row 0 of S (the shift of the power sums)
    double* mom_partial;       // (warps, 2, D) shifted power sums per warp, or nullptr
    const double* thr_dev;   // K thresholds in device memory (e.g. a quantile computed on the
                             // device), or nullptr: then thr[] below, copied from the host
    double thr[ELFI_B200_MAX_NESTED];
    __device__ __forceinline__ double threshold(int k) const {
        return thr_dev ? __ldg(thr_dev + k) : thr[k];
    }
};

// Shared consumer area: obs padded to G*16 doubles with zeros, then W rows padded likewise.
// Padding matters: TMA zero-fills columns >= D, obs pad 0 => (0-0)^2 = +0 is added, which
// leaves a non-negative accumulator unchanged bit for bit.
__device__ __forceinline__ void dist_setup_shared(uint8_t* aux, const DistParams& p, int D,
                                                  bool weighted) {
    const int Dp = ((D + RS_BOX_COLS - 1) / RS_BOX_COLS) * RS_BOX_COLS;
    double* obs_s = reinterpret_cast<double*>(aux);
    for (int j = threadIdx.x; j < Dp; j += blockDim.x) obs_s[j] = j < D ? p.obs[j] : 0.0;
    if (weighted) {
        double* w_s = obs_s + Dp;
        for (int k = 0; k < p.K; ++k)
            for (int j = threadIdx.x; j < Dp; j += blockDim.x)
                w_s[size_t(k) * Dp + j] = j < D ? p.W[size_t(k) * D + j] : 0.0;
    }
}

// Epilogue shared by all consumers.  KMAX is a compile-time bound so that acc[] and thr[] are
// indexed by constants (a runtime-indexed acc[] would be demoted to local memory).
template <int KMAX>
__device__ __forceinline__ void dist_finish(const DistParams& p, const double (&acc)[KMAX], int K,
                                            int64_t row, int64_t B, int lane) {
    bool ok = row < B;
    if (ok) {
#pragma unroll
        for (int k = 0; k < KMAX; ++k) {
            if (k < K) {
                const double d = sqrt(acc[k]);
                p.d_out[row * K + k] = d;
                if (p.has_thr) ok = ok && (d <= p.threshold(k));
            }
        }
    }
    if (p.mask != nullptr) {
        const uint32_t bits = __ballot_sync(0xffffffffu, ok && p.has_thr);
        if (lane == 0) p.mask[row >> 5] = bits;
    }
}

// K = 1, unweighted: the headline kernel (config #2: 1e6 x 128).
struct EuclidConsumer {
    typedef DistParams Params;
    static constexpr int PASSES = 1;
    const Params& p;
    const double* obs_s;
    double acc;

    static __device__ void setup_shared(uint8_t* aux, const Params& p, int D) {
        dist_setup_shared(aux, p, D, false);
    }
    __device__ EuclidConsumer(const Params& p_, const uint8_t* aux, int, int)
        : p(p_), obs_s(reinterpret_cast<const double*>(aux)), acc(0.0) {}
    __device__ __forceinline__ void begin_row() { acc = 0.0; }
    __device__ __forceinline__ void consume(int, int cg, const uint8_t* box_row, int sw) {
        const double2* o = reinterpret_cast<const double2*>(obs_s + cg * RS_BOX_COLS);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const double2 v = *reinterpret_cast<const double2*>(box_row + ((c ^ sw) << 4));
            const double2 ob = o[c];
            const double d0 = __dsub_rn(v.x, ob.x);
            const double d1 = __dsub_rn(v.y, ob.y);
            acc = __dadd_rn(acc, __dmul_rn(d0, d0));
            acc = __dadd_rn(acc, __dmul_rn(d1, d1));
        }
    }
    __device__ __forceinline__ void end_row(int64_t row, int64_t B, int lane) {
        const double a1[1] = {acc};
        dist_finish<1>(p, a1, 1, row, B, lane);
    }
};

// K = 1 with weights (cdist's `w`): acc += w_j * (diff * diff).
struct WeightedConsumer {
    typedef DistParams Params;
    static constexpr int PASSES = 1;
    const Params& p;
    const double* obs_s;
    const double* w_s;
    double acc;

    static __device__ void setup_shared(uint8_t* aux, const Params& p, int D) {
        dist_setup_shared(aux, p, D, true);
    }
    __device__ WeightedConsumer(const Params& p_, const uint8_t* aux, int D, int)
        : p(p_), obs_s(reinterpret_cast<const double*>(aux)), acc(0.0) {
        w_s = obs_s + ((D + RS_BOX_COLS - 1) / RS_BOX_COLS) * RS_BOX_COLS;
    }
    __device__ __forceinline__ void begin_row() { acc = 0.0; }
    __device__ __forceinline__ void consume(int, int cg, const uint8_t* box_row, int sw) {
        const double2* o = reinterpret_cast<const double2*>(obs_s + cg * RS_BOX_COLS);
        const double2* wv = reinterpret_cast<const double2*>(w_s + cg * RS_BOX_COLS);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const double2 v = *reinterpret_cast<const double2*>(box_row + ((c ^ sw) << 4));
            const double2 ob = o[c];
            const double2 w = wv[c];
            const double d0 = __dsub_rn(v.x, ob.x);
            const double d1 = __dsub_rn(v.y, ob.y);
            acc = __dadd_rn(acc, __dmul_rn(w.x, __dmul_rn(d0, d0)));
            acc = __dadd_rn(acc, __dmul_rn(w.y, __dmul_rn(d1, d1)));
        }
    }
    __device__ __forceinline__ void end_row(int64_t row, int64_t B, int lane) {
        const double a1[1] = {acc};
        dist_finish<1>(p, a1, 1, row, B, lane);
    }
};

// 1 <= K <= KMAX weighted columns sharing one pass over S (AdaptiveDistance: the reference
// re-reads S once per column, elfi_model.py:1150).
template <int KMAX>
struct NestedConsumer {
    typedef DistParams Params;
    static constexpr int PASSES = 1;
    const Params& p;
    const double* obs_s;
    const double* w_s;
    int Dp;
    double acc[KMAX];

    static __device__ void setup_shared(uint8_t* aux, const Params& p, int D) {
        dist_setup_shared(aux, p, D, true);
    }
    __device__ NestedConsumer(const Params& p_, const uint8_t* aux, int D, int)
        : p(p_), obs_s(reinterpret_cast<const double*>(aux)) {
        Dp = ((D + RS_BOX_COLS - 1) / RS_BOX_COLS) * RS_BOX_COLS;
        w_s = obs_s + Dp;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) acc[k] = 0.0;
    }
    __device__ __forceinline__ void begin_row() {
#pragma unroll
        for (int k = 0; k < KMAX; ++k) acc[k] = 0.0;
    }
    __device__ __forceinline__ void consume(int, int cg, const uint8_t* box_row, int sw) {
        const double2* o = reinterpret_cast<const double2*>(obs_s + cg * RS_BOX_COLS);
        const int K = p.K;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const double2 v = *reinterpret_cast<const double2*>(box_row + ((c ^ sw) << 4));
            const double2 ob = o[c];
            const double d0 = __dsub_rn(v.x, ob.x);
            const double d1 = __dsub_rn(v.y, ob.y);
            const double s0 = __dmul_rn(d0, d0);
            const double s1 = __dmul_rn(d1, d1);
#pragma unroll
            for (int k = 0; k < KMAX; ++k) {
                if (k < K) {
                    const double2 w = *reinterpret_cast<const double2*>(
                        w_s + size_t(k) * Dp + cg * RS_BOX_COLS + 2 * c);
                    acc[k] = __dadd_rn(acc[k], __dmul_rn(w.x, s0));
                    acc[k] = __dadd_rn(acc[k], __dmul_rn(w.y, s1));
                }
            }
        }
    }
    __device__ __forceinline__ void end_row(int64_t row, int64_t B, int lane) {
        dist_finish<KMAX>(p, acc, p.K, row, B, lane);
    }
};

// NestedConsumer + the per-column moments of AdaptiveDistance.add_data (elfi_model.py:1104-1125)
// from the SAME staged boxes: S is read from HBM once for the K distance columns and the
// (count, mean, M2) update, where the reference reads it K + 1 times.  After a lane has walked its
// row of the box, the warp sweeps the box again DOWN the rows: lane L owns the 16-byte chunk
// c2 = L & 7 (two columns) of the eight rows 8 (L >> 3) .. + 7 -- with the 128-byte swizzle the
// eight lanes of a quarter read one 128-byte row and the four quarters four different rows, so
// the LDS.128 is conflict-free like the row-wise read.  Shifted power sums
// (sum (x - c), sum (x - c)^2 with c = first row of S) go through two shuffles into per-warp
// shared accumulators (one per column, only lanes 0..7 write, no atomics); each warp flushes them
// once at the end and colmoments_flush_kernel adds the warps in a fixed order: deterministic.
template <int KMAX>
struct NestedMomentsConsumer : NestedConsumer<KMAX> {
    typedef NestedConsumer<KMAX> Base;
    typedef DistParams Params;
    static constexpr bool RS_TILE_INFO = true;
    static constexpr bool RS_FINISH = true;
    const double* shift_s;
    double* acc_s;          // this warp's [2][Dp]
    int64_t row0, nrows;
    int D;

    // aux: obs [Dp] | W [K][Dp] | shift [Dp] | accumulators [warps][2][Dp]
    static __host__ __device__ size_t aux_bytes(int64_t Dp, int64_t K, int warps = RS_WARPS) {
        return size_t(Dp) * 8 * (1 + K + 1 + 2 * warps);
    }
    static __device__ void setup_shared(uint8_t* aux, const Params& p, int D) {
        dist_setup_shared(aux, p, D, true);
        const int Dp = ((D + RS_BOX_COLS - 1) / RS_BOX_COLS) * RS_BOX_COLS;
        double* shift = reinterpret_cast<double*>(aux) + size_t(1 + p.K) * Dp;
        for (int j = threadIdx.x; j < Dp; j += blockDim.x) shift[j] = j < D ? p.shift_src[j] : 0.0;
        double* acc = shift + Dp;
        const int warps = blockDim.x >> 5;
        for (int j = threadIdx.x; j < 2 * warps * Dp; j += blockDim.x) acc[j] = 0.0;
    }
    __device__ NestedMomentsConsumer(const Params& p_, const uint8_t* aux, int D_, int lane)
        : Base(p_, aux, D_, lane), row0(0), nrows(0), D(D_) {
        shift_s = this->obs_s + size_t(1 + p_.K) * this->Dp;
        acc_s = const_cast<double*>(shift_s) + this->Dp + size_t(threadIdx.x >> 5) * 2 * this->Dp;
    }
    __device__ __forceinline__ void set_tile(int64_t r0, int64_t B) { row0 = r0; nrows = B; }
    __device__ __forceinline__ void consume(int pass, int cg, const uint8_t* box_row, int sw) {
        Base::consume(pass, cg, box_row, sw);
        const int lane = threadIdx.x & 31;
        const int c2 = lane & 7, h = lane >> 3;
        const uint8_t* box = box_row - lane * 128;
        const double2 sh = *reinterpret_cast<const double2*>(shift_s + cg * RS_BOX_COLS + 2 * c2);
        double s1x = 0.0, s1y = 0.0, s2x = 0.0, s2y = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int r = h * 8 + i;
            const double2 v = *reinterpret_cast<const double2*>(box + r * 128 + ((c2 ^ i) << 4));
            if (row0 + r < nrows) {
                const double dx = v.x - sh.x, dy = v.y - sh.y;
                s1x += dx;
                s1y += dy;
                s2x = fma(dx, dx, s2x);
                s2y = fma(dy, dy, s2y);
            }
        }
#pragma unroll
        for (int o = 8; o <= 16; o <<= 1) {
            s1x += __shfl_xor_sync(0xffffffffu, s1x, o);
            s1y += __shfl_xor_sync(0xffffffffu, s1y, o);
            s2x += __shfl_xor_sync(0xffffffffu, s2x, o);
            s2y += __shfl_xor_sync(0xffffffffu, s2y, o);
        }
        if (lane < 8) {
            double2* a1 = reinterpret_cast<double2*>(acc_s + cg * RS_BOX_COLS + 2 * c2);
            double2* a2 = reinterpret_cast<double2*>(acc_s + this->Dp + cg * RS_BOX_COLS + 2 * c2);
            double2 t1 = *a1, t2 = *a2;
            t1.x += s1x; t1.y += s1y; t2.x += s2x; t2.y += s2y;
            *a1 = t1;
            *a2 = t2;
        }
    }
    __device__ __forceinline__ void finish(int64_t gw, int lane) {
        double* out = this->p.mom_partial + gw * 2 * int64_t(D);
        for (int j = lane; j < D; j += 32) {
            out[j] = acc_s[j];
            out[D + j] = acc_s[this->Dp + j];
        }
    }
};

// out[0*D + j] = mean_j, out[1*D + j] = M2_j from the per-warp shifted power sums.
// Block (32 columns, 32 slices): slice y adds the warps y, y + 32, ... of its column, the slices
// are then added in order -- a fixed summation tree, ~nwarps / 32 dependent loads per thread
// (a single thread per column walking all ~1200 warps cost 0.15 ms of pure latency).
__global__ void __launch_bounds__(1024)
colmoments_flush_kernel(const double* __restrict__ S, const double* __restrict__ partial,
                        int64_t nwarps, int64_t B, int64_t D, double* __restrict__ out) {
    __shared__ double r1[32][33], r2[32][33];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int64_t c = int64_t(blockIdx.x) * 32 + tx;
    double s1 = 0.0, s2 = 0.0;
    if (c < D)
        for (int64_t b = ty; b < nwarps; b += 32) {
            s1 += partial[(b * 2 + 0) * D + c];
            s2 += partial[(b * 2 + 1) * D + c];
        }
    r1[ty][tx] = s1;
    r2[ty][tx] = s2;
    __syncthreads();
    if (ty == 0 && c < D) {
        for (int k = 1; k < 32; ++k) { s1 += r1[k][tx]; s2 += r2[k][tx]; }
        const double n = double(B);
        out[c] = S[c] + s1 / n;
        out[D + c] = s2 - s1 * s1 / n;
    }
}

// Warps per CTA of the fused kernel: 12 when the ring still gets >= 3 slots next to the per-warp
// accumulators (two warps per scheduler leave the fp64 pipe half idle: long dependent chains of
// K + 2 accumulators per lane), else 8.  Measured at 5e5 x 256: K = 2 0.232 -> 0.214 ms, K = 6
// 0.297 -> 0.279 ms; 16 warps (128 registers, 2-slot ring) gives the 8-warp time back, and the
// plain nested kernels do not gain from either.
template <int KMAX>
static int fused_moments_warps(elfi_b200_ctx* ctx, int64_t Dp, int64_t K) {
    constexpr int warps = 12;
    if (KMAX > 8) return RS_WARPS;
    const size_t aux = NestedMomentsConsumer<KMAX>::aux_bytes(Dp, K, warps);
    return rs_pick_stages(ctx->smem_optin, aux, warps) >= 3 ? warps : RS_WARPS;
}

template <int KMAX>
static int launch_nested_moments(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B,
                                 int64_t D, DistParams p, double* moments, cudaStream_t stream) {
    const int64_t Dp = ((D + RS_BOX_COLS - 1) / RS_BOX_COLS) * RS_BOX_COLS;
    const int warps = fused_moments_warps<KMAX>(ctx, Dp, p.K);
    const size_t aux = NestedMomentsConsumer<KMAX>::aux_bytes(Dp, p.K, warps);
    const int64_t ntiles = (B + RS_BOX_ROWS - 1) / RS_BOX_ROWS;
    int64_t ctas = (ntiles + warps - 1) / warps;
    if (ctas > ctx->sm_count) ctas = ctx->sm_count;
    const int64_t nwarps = ctas * warps;
    int rc;
    if constexpr (KMAX <= 8) {
        if (warps == 12)
            rc = rowstream_launch<NestedMomentsConsumer<KMAX>, 12>(ctx, S, ldS, B, D, aux, p, stream);
        else
            rc = rowstream_launch<NestedMomentsConsumer<KMAX>>(ctx, S, ldS, B, D, aux, p, stream);
    } else {
        rc = rowstream_launch<NestedMomentsConsumer<KMAX>>(ctx, S, ldS, B, D, aux, p, stream);
    }
    if (rc) return rc;
    colmoments_flush_kernel<<<unsigned((D + 31) / 32), dim3(32, 32), 0, stream>>>(
        S, p.mom_partial, nwarps, B, D, moments);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

// Fallback for narrow (D < 16) or TMA-incompatible matrices: one thread per row, direct
// loads.  For D <= 8 a warp still touches a contiguous span, so sectors are fully used.
__global__ void __launch_bounds__(256)
dist_direct_kernel(const double* __restrict__ S, int64_t ld, int64_t B, int D, DistParams p) {
    const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int K = p.K;
    bool ok = row < B;
    if (ok) {
        const double* r = S + row * ld;
        for (int k = 0; k < K; ++k) {
            double acc = 0.0;
            if (p.W != nullptr) {
                const double* w = p.W + size_t(k) * D;
                for (int j = 0; j < D; ++j) {
                    const double d = __dsub_rn(__ldg(r + j), __ldg(p.obs + j));
                    acc = __dadd_rn(acc, __dmul_rn(__ldg(w + j), __dmul_rn(d, d)));
                }
            } else {
                for (int j = 0; j < D; ++j) {
                    const double d = __dsub_rn(__ldg(r + j), __ldg(p.obs + j));
                    acc = __dadd_rn(acc, __dmul_rn(d, d));
                }
            }
            const double dist = sqrt(acc);
            p.d_out[row * K + k] = dist;
            if (p.has_thr) ok = ok && (dist <= p.threshold(k));
        }
    }
    if (p.mask != nullptr) {
        const uint32_t bits = __ballot_sync(0xffffffffu, ok && p.has_thr);
        if (lane == 0 && (row - lane) < B) p.mask[row >> 5] = bits;
    }
}

// Mask words -> ascending accepted row indices.  CTA b owns words [b*1024, (b+1)*1024):
// it first totals the popcounts of all earlier words (the whole mask is B/8 bytes, L2
// resident), then scans its own and scatters.  Deterministic order, no atomics.
__global__ void __launch_bounds__(1024)
compact_mask_kernel(const uint32_t* __restrict__ mask, int64_t nwords, int64_t B,
                    int32_t* __restrict__ idx, int64_t* __restrict__ n_out) {
    __shared__ int64_t warp_sums[32];
    __shared__ int64_t base_s;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int wid = tid >> 5;
    const int64_t first = int64_t(blockIdx.x) * 1024;

    int64_t before = 0;
    for (int64_t w = tid; w < first; w += 1024) before += __popc(mask[w]);
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    if (lane == 0) warp_sums[wid] = before;
    __syncthreads();
    if (tid == 0) {
        int64_t t = 0;
        for (int i = 0; i < 32; ++i) t += warp_sums[i];
        base_s = t;
    }
    __syncthreads();
    const int64_t base = base_s;
    __syncthreads();

    const int64_t w = first + tid;
    const uint32_t bits = w < nwords ? mask[w] : 0u;
    const int cnt = __popc(bits);
    int incl = cnt;
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sums[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        int64_t v = warp_sums[lane];
        int64_t inc2 = v;
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t t = __shfl_up_sync(0xffffffffu, inc2, o);
            if (lane >= o) inc2 += t;
        }
        warp_sums[lane] = inc2 - v;  // exclusive
        if (lane == 31 && blockIdx.x == gridDim.x - 1 && n_out != nullptr) *n_out = base + inc2;
    }
    __syncthreads();
    int64_t pos = base + warp_sums[wid] + (incl - cnt);
    if (idx != nullptr) {
        uint32_t b = bits;
        while (b) {
            const int bit = __ffs(b) - 1;
            b &= b - 1;
            idx[pos++] = int32_t(w * 32 + bit);
        }
    }
}

int launch_compact_mask(const uint32_t* mask, int64_t B, int32_t* idx, int64_t* n_out,
                        cudaStream_t stream) {
    const int64_t nwords = (B + 31) / 32;
    if (nwords == 0) {
        if (n_out) ELFI_CUDA_OK(cudaMemsetAsync(n_out, 0, sizeof(int64_t), stream));
        return ELFI_B200_OK;
    }
    const unsigned blocks = unsigned((nwords + 1023) / 1024);
    compact_mask_kernel<<<blocks, 1024, 0, stream>>>(mask, nwords, B, idx, n_out);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

// Distances (+ mask when thresholds are given) for a device-resident matrix.
int launch_dist(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B, int64_t D,
                const double* obs, const double* W, int64_t K, const double* thr_host,
                double* d_out, uint32_t* mask, cudaStream_t stream,
                const double* thr_dev = nullptr) {
    DistParams p;
    memset(&p, 0, sizeof(p));
    p.obs = obs;
    p.W = W;
    p.d_out = d_out;
    p.mask = mask;
    p.K = int(K);
    p.has_thr = thr_host != nullptr || thr_dev != nullptr;
    p.thr_dev = thr_dev;
    if (thr_host)
        for (int k = 0; k < K; ++k) p.thr[k] = thr_host[k];
    if (B == 0) return ELFI_B200_OK;

    const int64_t Dp = ((D + RS_BOX_COLS - 1) / RS_BOX_COLS) * RS_BOX_COLS;
    const bool use_tma = D >= RS_BOX_COLS && tma_compatible(S, ldS);
    if (use_tma) {
        const size_t aux = size_t(Dp) * 8 * (W ? (1 + K) : 1);
        if (rs_pick_stages(ctx->smem_optin, aux) >= 2) {
            if (W == nullptr) return rowstream_launch<EuclidConsumer>(ctx, S, ldS, B, D, aux, p, stream);
            if (K == 1) return rowstream_launch<WeightedConsumer>(ctx, S, ldS, B, D, aux, p, stream);
            if (K <= 2) return rowstream_launch<NestedConsumer<2>>(ctx, S, ldS, B, D, aux, p, stream);
            if (K <= 3) return rowstream_launch<NestedConsumer<3>>(ctx, S, ldS, B, D, aux, p, stream);
            if (K <= 4) return rowstream_launch<NestedConsumer<4>>(ctx, S, ldS, B, D, aux, p, stream);
            if (K <= 5) return rowstream_launch<NestedConsumer<5>>(ctx, S, ldS, B, D, aux, p, stream);
            if (K <= 6) return rowstream_launch<NestedConsumer<6>>(ctx, S, ldS, B, D, aux, p, stream);
            if (K <= 8) return rowstream_launch<NestedConsumer<8>>(ctx, S, ldS, B, D, aux, p, stream);
            if (K <= 16) return rowstream_launch<NestedConsumer<16>>(ctx, S, ldS, B, D, aux, p, stream);
            return rowstream_launch<NestedConsumer<32>>(ctx, S, ldS, B, D, aux, p, stream);
        }
    }
    const unsigned blocks = unsigned((B + 255) / 256);
    dist_direct_kernel<<<blocks, 256, 0, stream>>>(S, ldS, B, int(D), p);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

// ---- other cdist metrics (elfi/model/elfi_model.py:1037: Distance passes any metric string to
// scipy.spatial.distance.cdist) ------------------------------------------------------------------
// SciPy 1.18 accumulates 'sqeuclidean', 'cityblock', 'chebyshev' and 'minkowski' left to right in
// fp64 like 'euclidean' (probed: bit-identical to a sequential loop at 2000 x 128), so they are
// variants of EuclidConsumer with another per-term operation and another finish.  Unweighted,
// one column (K = 1).  Zero padding (TMA fill, obs pad) adds |0|, 0^2, 0^p or max(acc, 0): no-ops.
struct MetricParams : DistParams {
    double pexp;       // Minkowski exponent
    const double* V;   // (D) component variances of 'seuclidean', else nullptr
};

template <int METRIC>
__device__ __forceinline__ double metric_term(double acc, double d, double pexp) {
    if (METRIC == ELFI_B200_METRIC_SQEUCLIDEAN) return __dadd_rn(acc, __dmul_rn(d, d));
    if (METRIC == ELFI_B200_METRIC_CITYBLOCK) return __dadd_rn(acc, fabs(d));
    if (METRIC == ELFI_B200_METRIC_CHEBYSHEV) return fabs(d) > acc ? fabs(d) : acc;
    return __dadd_rn(acc, pow(fabs(d), pexp));                       // Minkowski
}

template <int METRIC>
__device__ __forceinline__ double metric_value(double acc, double pexp) {
    return METRIC == ELFI_B200_METRIC_MINKOWSKI ? pow(acc, 1.0 / pexp) : acc;
}

template <int METRIC>
__device__ __forceinline__ void metric_finish(const MetricParams& p, double acc, int64_t row,
                                              int64_t B, int lane, bool whole_warp) {
    bool ok = row < B;
    if (ok) {
        const double d = metric_value<METRIC>(acc, p.pexp);
        p.d_out[row] = d;
        if (p.has_thr) ok = d <= p.threshold(0);
    }
    if (p.mask != nullptr) {
        const uint32_t bits = __ballot_sync(0xffffffffu, ok && p.has_thr);
        if (lane == 0 && (whole_warp || (row - lane) < B)) p.mask[row >> 5] = bits;
    }
}

template <int METRIC>
struct MetricConsumer {
    typedef MetricParams Params;
    static constexpr int PASSES = 1;
    const Params& p;
    const double* obs_s;
    double acc;

    static __device__ void setup_shared(uint8_t* aux, const Params& p, int D) {
        dist_setup_shared(aux, p, D, false);
    }
    __device__ MetricConsumer(const Params& p_, const uint8_t* aux, int, int)
        : p(p_), obs_s(reinterpret_cast<const double*>(aux)), acc(0.0) {}
    __device__ __forceinline__ void begin_row() { acc = 0.0; }
    __device__ __forceinline__ void consume(int, int cg, const uint8_t* box_row, int sw) {
        const double2* o = reinterpret_cast<const double2*>(obs_s + cg * RS_BOX_COLS);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const double2 v = *reinterpret_cast<const double2*>(box_row + ((c ^ sw) << 4));
            const double2 ob = o[c];
            acc = metric_term<METRIC>(acc, __dsub_rn(v.x, ob.x), p.pexp);
            acc = metric_term<METRIC>(acc, __dsub_rn(v.y, ob.y), p.pexp);
        }
    }
    __device__ __forceinline__ void end_row(int64_t row, int64_t B, int lane) {
        metric_finish<METRIC>(p, acc, row, B, lane, true);
    }
};

template <int METRIC>
__global__ void __launch_bounds__(256)
metric_direct_kernel(const double* __restrict__ S, int64_t ld, int64_t B, int D, MetricParams p) {
    const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    double acc = 0.0;
    if (row < B) {
        const double* r = S + row * ld;
        for (int j = 0; j < D; ++j)
            acc = metric_term<METRIC>(acc, __dsub_rn(__ldg(r + j), __ldg(p.obs + j)), p.pexp);
    }
    metric_finish<METRIC>(p, acc, row, B, threadIdx.x & 31, false);
}

template <int METRIC>
static int launch_metric_t(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B, int64_t D,
                           const MetricParams& p, cudaStream_t stream) {
    const int64_t Dp = ((D + RS_BOX_COLS - 1) / RS_BOX_COLS) * RS_BOX_COLS;
    const size_t aux = size_t(Dp) * 8;
    if (D >= RS_BOX_COLS && tma_compatible(S, ldS) && rs_pick_stages(ctx->smem_optin, aux) >= 2)
        return rowstream_launch<MetricConsumer<METRIC>>(ctx, S, ldS, B, D, aux, p, stream);
    metric_direct_kernel<METRIC><<<unsigned((B + 255) / 256), 256, 0, stream>>>(S, ldS, B, int(D), p);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

static int launch_metric(elfi_b200_ctx* ctx, int metric, double pexp, const double* S, int64_t ldS,
                         int64_t B, int64_t D, const double* obs, const double* thr_host,
                         double* d_out, uint32_t* mask, cudaStream_t stream) {
    MetricParams p;
    memset(&p, 0, sizeof(p));
    p.obs = obs;
    p.d_out = d_out;
    p.mask = mask;
    p.K = 1;
    p.has_thr = thr_host != nullptr;
    if (thr_host) p.thr[0] = thr_host[0];
    p.pexp = pexp;
    if (B == 0) return ELFI_B200_OK;
    switch (metric) {
        case ELFI_B200_METRIC_SQEUCLIDEAN:
            return launch_metric_t<ELFI_B200_METRIC_SQEUCLIDEAN>(ctx, S, ldS, B, D, p, stream);
        case ELFI_B200_METRIC_CITYBLOCK:
            return launch_metric_t<ELFI_B200_METRIC_CITYBLOCK>(ctx, S, ldS, B, D, p, stream);
        case ELFI_B200_METRIC_CHEBYSHEV:
            return launch_metric_t<ELFI_B200_METRIC_CHEBYSHEV>(ctx, S, ldS, B, D, p, stream);
        default:
            return launch_metric_t<ELFI_B200_METRIC_MINKOWSKI>(ctx, S, ldS, B, D, p, stream);
    }
}

// 'seuclidean' (cdist(..., 'seuclidean', V=V)): SciPy 1.18's compiled loop keeps TWO running sums,
// terms (d*d)/V_j with even j in one and odd j in the other over the first D - D%2 columns, adds
// the two, then adds the last term when D is odd, then takes the root (probed against the
// installed SciPy for D = 1..69, 127..129, 255, 1000: bit-identical; tests/test_oracle.py pins
// it).  The division is IEEE (__ddiv_rn), so a weight row 1/V through WeightedConsumer differs in
// the last bits.  Padding: TMA zero-fills columns >= D, obs pads with 0 and V with 1, so a padded
// term is (0*0)/1 = +0, a no-op on the non-negative sums.
struct SeuclidTerm {
    double even, odd, last;
    int j_last;   // D - 1 when D is odd (that term is added after the two sums meet), else -1
    __device__ __forceinline__ void begin(int D) {
        even = 0.0;
        odd = 0.0;
        last = 0.0;
        j_last = (D & 1) ? D - 1 : -1;
    }
    // j0 is even; (t0, t1) are the terms of columns j0 and j0 + 1
    __device__ __forceinline__ void pair(int j0, double t0, double t1) {
        if (j0 == j_last) {
            last = t0;
        } else {
            even = __dadd_rn(even, t0);
            odd = __dadd_rn(odd, t1);
        }
    }
    __device__ __forceinline__ double value() const {
        const double s = __dadd_rn(even, odd);
        return sqrt(j_last >= 0 ? __dadd_rn(s, last) : s);
    }
};

__device__ __forceinline__ double seuclid_term(double x, double o, double v) {
    const double d = __dsub_rn(x, o);
    return __ddiv_rn(__dmul_rn(d, d), v);
}

__device__ __forceinline__ void seuclid_finish(const MetricParams& p, double dist, int64_t row,
                                               int64_t B, int lane, bool whole_warp) {
    bool ok = row < B;
    if (ok) {
        p.d_out[row] = dist;
        if (p.has_thr) ok = dist <= p.threshold(0);
    }
    if (p.mask != nullptr) {
        const uint32_t bits = __ballot_sync(0xffffffffu, ok && p.has_thr);
        if (lane == 0 && (whole_warp || (row - lane) < B)) p.mask[row >> 5] = bits;
    }
}

struct SeuclidConsumer {
    typedef MetricParams Params;
    static constexpr int PASSES = 1;
    const Params& p;
    const double* obs_s;
    const double* v_s;
    int D;
    SeuclidTerm acc;

    static __device__ void setup_shared(uint8_t* aux, const Params& p, int D) {
        const int Dp = ((D + RS_BOX_COLS - 1) / RS_BOX_COLS) * RS_BOX_COLS;
        double* obs_s = reinterpret_cast<double*>(aux);
        for (int j = threadIdx.x; j < Dp; j += blockDim.x) {
            obs_s[j] = j < D ? p.obs[j] : 0.0;
            obs_s[Dp + j] = j < D ? p.V[j] : 1.0;
        }
    }
    __device__ SeuclidConsumer(const Params& p_, const uint8_t* aux, int D_, int)
        : p(p_), obs_s(reinterpret_cast<const double*>(aux)), D(D_) {
        v_s = obs_s + ((D + RS_BOX_COLS - 1) / RS_BOX_COLS) * RS_BOX_COLS;
        acc.begin(D);
    }
    __device__ __forceinline__ void begin_row() { acc.begin(D); }
    __device__ __forceinline__ void consume(int, int cg, const uint8_t* box_row, int sw) {
        const double2* o = reinterpret_cast<const double2*>(obs_s + cg * RS_BOX_COLS);
        const double2* vv = reinterpret_cast<const double2*>(v_s + cg * RS_BOX_COLS);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const double2 x = *reinterpret_cast<const double2*>(box_row + ((c ^ sw) << 4));
            const double2 ob = o[c];
            const double2 v = vv[c];
            acc.pair(cg * RS_BOX_COLS + 2 * c, seuclid_term(x.x, ob.x, v.x),
                     seuclid_term(x.y, ob.y, v.y));
        }
    }
    __device__ __forceinline__ void end_row(int64_t row, int64_t B, int lane) {
        seuclid_finish(p, acc.value(), row, B, lane, true);
    }
};

__global__ void __launch_bounds__(256)
seuclid_direct_kernel(const double* __restrict__ S, int64_t ld, int64_t B, int D, MetricParams p) {
    const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    SeuclidTerm acc;
    acc.begin(D);
    if (row < B) {
        const double* r = S + row * ld;
        for (int j = 0; j < D; j += 2) {
            const double t0 = seuclid_term(__ldg(r + j), __ldg(p.obs + j), __ldg(p.V + j));
            const double t1 = j + 1 < D
                ? seuclid_term(__ldg(r + j + 1), __ldg(p.obs + j + 1), __ldg(p.V + j + 1)) : 0.0;
            acc.pair(j, t0, t1);
        }
    }
    seuclid_finish(p, acc.value(), row, B, threadIdx.x & 31, false);
}

static int launch_seuclid(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B, int64_t D,
                          const double* obs, const double* V, const double* thr_host,
                          double* d_out, uint32_t* mask, cudaStream_t stream) {
    MetricParams p;
    memset(&p, 0, sizeof(p));
    p.obs = obs;
    p.V = V;
    p.d_out = d_out;
    p.mask = mask;
    p.K = 1;
    p.has_thr = thr_host != nullptr;
    if (thr_host) p.thr[0] = thr_host[0];
    if (B == 0) return ELFI_B200_OK;
    const int64_t Dp = ((D + RS_BOX_COLS - 1) / RS_BOX_COLS) * RS_BOX_COLS;
    const size_t aux = size_t(Dp) * 8 * 2;
    if (D >= RS_BOX_COLS && tma_compatible(S, ldS) && rs_pick_stages(ctx->smem_optin, aux) >= 2)
        return rowstream_launch<SeuclidConsumer>(ctx, S, ldS, B, D, aux, p, stream);
    seuclid_direct_kernel<<<unsigned((B + 255) / 256), 256, 0, stream>>>(S, ldS, B, int(D), p);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

static int check_dist_args(const void* S, int64_t ldS, int64_t B, int64_t D, const void* obs,
                           const void* W, int64_t K, const void* thr, const void* acc_idx) {
    ELFI_REQUIRE(B >= 0 && D >= 1, "dist: bad shape B=%lld D=%lld", (long long)B, (long long)D);
    ELFI_REQUIRE(B == 0 || S != nullptr, "dist: S is NULL");
    ELFI_REQUIRE(obs != nullptr, "dist: obs is NULL");
    ELFI_REQUIRE(ldS >= D, "dist: ldS (%lld) < D (%lld)", (long long)ldS, (long long)D);
    ELFI_REQUIRE(K >= 1 && K <= ELFI_B200_MAX_NESTED, "dist: K=%lld outside [1, %d]",
                 (long long)K, ELFI_B200_MAX_NESTED);
    ELFI_REQUIRE(W != nullptr || K == 1, "dist: K=%lld needs a weight matrix", (long long)K);
    ELFI_REQUIRE(acc_idx == nullptr || thr != nullptr, "dist: acc_idx requires thresholds");
    ELFI_REQUIRE(B < (int64_t(1) << 31), "dist: B must fit int32 row indices");
    return ELFI_B200_OK;
}

}  // namespace elfi

extern "C" {

int elfi_b200_dist_euclid_thr_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B,
                                  int64_t D, const double* obs, const double* W, int64_t K,
                                  const double* thr_host, double* d_out, int32_t* acc_idx,
                                  int64_t* n_acc, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx != nullptr, "dist: ctx is NULL");
    int rc = check_dist_args(S, ldS, B, D, obs, W, K, thr_host, acc_idx);
    if (rc) return rc;
    ELFI_REQUIRE(B == 0 || d_out != nullptr, "dist: d_out is NULL");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    uint32_t* mask = nullptr;
    if (thr_host != nullptr) {
        const size_t nwords = size_t((B + 31) / 32);
        mask = static_cast<uint32_t*>(ctx_scratch(ctx, nwords * 4 + 256));
        if (!mask) return ELFI_B200_ERR_NOMEM;
    }
    rc = launch_dist(ctx, S, ldS, B, D, obs, W, K, thr_host, d_out, mask, stream);
    if (rc) return rc;
    if (thr_host != nullptr && (acc_idx != nullptr || n_acc != nullptr))
        return launch_compact_mask(mask, B, acc_idx, n_acc, stream);
    return ELFI_B200_OK;
}

int elfi_b200_dist_euclid_thr_dev_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B,
                                      int64_t D, const double* obs, const double* W, int64_t K,
                                      const double* thr_dev, double* d_out, int32_t* acc_idx,
                                      int64_t* n_acc, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx != nullptr && thr_dev != nullptr, "dist: ctx or thr_dev is NULL");
    int rc = check_dist_args(S, ldS, B, D, obs, W, K, thr_dev, acc_idx);
    if (rc) return rc;
    ELFI_REQUIRE(B == 0 || d_out != nullptr, "dist: d_out is NULL");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    const size_t nwords = size_t((B + 31) / 32);
    uint32_t* mask = static_cast<uint32_t*>(ctx_scratch(ctx, nwords * 4 + 256));
    if (!mask) return ELFI_B200_ERR_NOMEM;
    rc = launch_dist(ctx, S, ldS, B, D, obs, W, K, nullptr, d_out, mask, stream, thr_dev);
    if (rc) return rc;
    if (acc_idx != nullptr || n_acc != nullptr)
        return launch_compact_mask(mask, B, acc_idx, n_acc, stream);
    return ELFI_B200_OK;
}

int elfi_b200_dist_euclid_mom_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B,
                                  int64_t D, const double* obs, const double* W, int64_t K,
                                  const double* thr_host, const double* thr_dev, double* d_out,
                                  int32_t* acc_idx, int64_t* n_acc, double* moments,
                                  void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx != nullptr && moments != nullptr, "dist_mom: ctx or moments is NULL");
    ELFI_REQUIRE(!(thr_host && thr_dev), "dist_mom: give thresholds on the host OR on the device");
    const void* thr = thr_host ? static_cast<const void*>(thr_host) : thr_dev;
    int rc = check_dist_args(S, ldS, B, D, obs, W, K, thr, acc_idx);
    if (rc) return rc;
    ELFI_REQUIRE(B >= 1 && d_out != nullptr, "dist_mom: needs at least one row and d_out");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    const int64_t Dp = ((D + RS_BOX_COLS - 1) / RS_BOX_COLS) * RS_BOX_COLS;
    const size_t aux = NestedMomentsConsumer<2>::aux_bytes(Dp, K);
    const bool fused = W != nullptr && D >= RS_BOX_COLS && tma_compatible(S, ldS) &&
                       rs_pick_stages(ctx->smem_optin, aux) >= 2;
    const size_t mask_bytes = (size_t((B + 31) / 32) * 4 + 255) & ~size_t(255);
    const size_t part_bytes = fused ? size_t(ctx->sm_count) * 16 * 2 * D * 8 : 0;   // <= 16 warps
    uint8_t* base = static_cast<uint8_t*>(ctx_scratch(ctx, mask_bytes + part_bytes + 256));
    if (!base) return ELFI_B200_ERR_NOMEM;
    uint32_t* mask = thr ? reinterpret_cast<uint32_t*>(base) : nullptr;
    if (!fused) {
        // narrow / unaligned / unweighted matrices: distances, then the stand-alone moments pass
        rc = launch_dist(ctx, S, ldS, B, D, obs, W, K, thr_host, d_out, mask, stream, thr_dev);
        if (rc) return rc;
        if (thr && (acc_idx != nullptr || n_acc != nullptr)) {
            rc = launch_compact_mask(mask, B, acc_idx, n_acc, stream);
            if (rc) return rc;
        }
        return elfi_b200_colmoments_f64(ctx, S, ldS, B, D, moments, stream_);
    }
    DistParams p;
    memset(&p, 0, sizeof(p));
    p.obs = obs;
    p.W = W;
    p.d_out = d_out;
    p.mask = mask;
    p.K = int(K);
    p.has_thr = thr != nullptr;
    p.thr_dev = thr_dev;
    if (thr_host)
        for (int k = 0; k < K; ++k) p.thr[k] = thr_host[k];
    p.shift_src = S;
    p.mom_partial = reinterpret_cast<double*>(base + mask_bytes);
    if (K <= 2) rc = launch_nested_moments<2>(ctx, S, ldS, B, D, p, moments, stream);
    else if (K <= 4) rc = launch_nested_moments<4>(ctx, S, ldS, B, D, p, moments, stream);
    else if (K <= 6) rc = launch_nested_moments<6>(ctx, S, ldS, B, D, p, moments, stream);
    else if (K <= 8) rc = launch_nested_moments<8>(ctx, S, ldS, B, D, p, moments, stream);
    else if (K <= 16) rc = launch_nested_moments<16>(ctx, S, ldS, B, D, p, moments, stream);
    else rc = launch_nested_moments<32>(ctx, S, ldS, B, D, p, moments, stream);
    if (rc) return rc;
    if (thr && (acc_idx != nullptr || n_acc != nullptr))
        return launch_compact_mask(mask, B, acc_idx, n_acc, stream);
    return ELFI_B200_OK;
}

int elfi_b200_dist_euclid_thr_f64_host(elfi_b200_ctx* ctx, const double* S_host, int64_t ldS,
                                       int64_t B, int64_t D, const double* obs_host,
                                       const double* W_host, int64_t K, const double* thr_host,
                                       double* d_out_host, int32_t* acc_idx_host,
                                       int64_t* n_acc_host) {
    using namespace elfi;
    ELFI_REQUIRE(ctx != nullptr, "dist_host: ctx is NULL");
    int rc = check_dist_args(S_host, ldS, B, D, obs_host, W_host, K, thr_host, acc_idx_host);
    if (rc) return rc;
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));

    // Device staging: two row chunks (ping-pong), obs, W, distances, mask, indices, count.
    const int64_t row_bytes = D * 8;
    int64_t chunk_rows = (int64_t(32) << 20) / row_bytes;
    chunk_rows = (chunk_rows / 32) * 32;
    if (chunk_rows < 32) chunk_rows = 32;
    if (chunk_rows > B) chunk_rows = ((B + 31) / 32) * 32;
    const size_t chunk_bytes = size_t(chunk_rows) * row_bytes;
    const size_t nwords = size_t((B + 31) / 32);
    auto align = [](size_t v) { return (v + 255) & ~size_t(255); };
    const size_t off_chunk1 = align(chunk_bytes);
    const size_t off_obs = off_chunk1 + align(chunk_bytes);
    const size_t off_w = off_obs + align(size_t(D) * 8);
    const size_t off_d = off_w + align(size_t(K) * D * 8);
    const size_t off_mask = off_d + align(size_t(B) * K * 8);
    const size_t off_idx = off_mask + align(nwords * 4 + 4);
    const size_t off_n = off_idx + align(size_t(B) * 4 + 4);
    const size_t total = off_n + 256;
    if (total > ctx->dev_stage_bytes) {
        ELFI_CUDA_OK(cudaDeviceSynchronize());
        if (ctx->dev_stage) ELFI_CUDA_OK(cudaFree(ctx->dev_stage));
        ctx->dev_stage = nullptr;
        ctx->dev_stage_bytes = 0;
        ELFI_CUDA_OK(cudaMalloc(&ctx->dev_stage, total));
        ctx->dev_stage_bytes = total;
    }
    uint8_t* base = static_cast<uint8_t*>(ctx->dev_stage);
    double* chunk[2] = {reinterpret_cast<double*>(base), reinterpret_cast<double*>(base + off_chunk1)};
    double* obs_d = reinterpret_cast<double*>(base + off_obs);
    double* w_d = W_host ? reinterpret_cast<double*>(base + off_w) : nullptr;
    double* d_d = reinterpret_cast<double*>(base + off_d);
    uint32_t* mask_d = thr_host ? reinterpret_cast<uint32_t*>(base + off_mask) : nullptr;
    int32_t* idx_d = reinterpret_cast<int32_t*>(base + off_idx);
    int64_t* n_d = reinterpret_cast<int64_t*>(base + off_n);

    cudaStream_t s0 = ctx->copy_stream[0], s1 = ctx->copy_stream[1];
    ELFI_CUDA_OK(cudaMemcpyAsync(obs_d, obs_host, size_t(D) * 8, cudaMemcpyHostToDevice, s0));
    if (W_host)
        ELFI_CUDA_OK(cudaMemcpyAsync(w_d, W_host, size_t(K) * D * 8, cudaMemcpyHostToDevice, s0));
    ELFI_CUDA_OK(cudaEventRecord(ctx->copy_event[0], s0));
    ELFI_CUDA_OK(cudaStreamWaitEvent(s1, ctx->copy_event[0], 0));

    int which = 0;
    for (int64_t r0 = 0; r0 < B; r0 += chunk_rows, which ^= 1) {
        const int64_t rows = (B - r0) < chunk_rows ? (B - r0) : chunk_rows;
        cudaStream_t st = which ? s1 : s0;
        if (ldS == D) {
            ELFI_CUDA_OK(cudaMemcpyAsync(chunk[which], S_host + r0 * ldS, size_t(rows) * row_bytes,
                                         cudaMemcpyHostToDevice, st));
        } else {
            ELFI_CUDA_OK(cudaMemcpy2DAsync(chunk[which], size_t(row_bytes), S_host + r0 * ldS,
                                           size_t(ldS) * 8, size_t(row_bytes), size_t(rows),
                                           cudaMemcpyHostToDevice, st));
        }
        rc = launch_dist(ctx, chunk[which], D, rows, D, obs_d, w_d, K, thr_host, d_d + r0 * K,
                         mask_d ? mask_d + r0 / 32 : nullptr, st);
        if (rc) return rc;
    }
    // join s1 into s0, compact, copy back
    ELFI_CUDA_OK(cudaEventRecord(ctx->copy_event[1], s1));
    ELFI_CUDA_OK(cudaStreamWaitEvent(s0, ctx->copy_event[1], 0));
    ELFI_CUDA_OK(cudaEventRecord(ctx->copy_event[2], s0));
    ELFI_CUDA_OK(cudaStreamWaitEvent(s1, ctx->copy_event[2], 0));
    if (d_out_host && B > 0)
        ELFI_CUDA_OK(cudaMemcpyAsync(d_out_host, d_d, size_t(B) * K * 8, cudaMemcpyDeviceToHost, s1));
    int64_t n_acc = 0;
    if (thr_host != nullptr) {
        rc = launch_compact_mask(mask_d, B, acc_idx_host ? idx_d : nullptr, n_d, s0);
        if (rc) return rc;
        ELFI_CUDA_OK(cudaMemcpyAsync(&n_acc, n_d, 8, cudaMemcpyDeviceToHost, s0));
        ELFI_CUDA_OK(cudaStreamSynchronize(s0));
        if (acc_idx_host && n_acc > 0)
            ELFI_CUDA_OK(cudaMemcpyAsync(acc_idx_host, idx_d, size_t(n_acc) * 4,
                                         cudaMemcpyDeviceToHost, s0));
        if (n_acc_host) *n_acc_host = n_acc;
    }
    ELFI_CUDA_OK(cudaStreamSynchronize(s0));
    ELFI_CUDA_OK(cudaStreamSynchronize(s1));
    return ELFI_B200_OK;
}

int elfi_b200_dist_metric_thr_f64(elfi_b200_ctx* ctx, int32_t metric, double pexp, const double* S,
                                  int64_t ldS, int64_t B, int64_t D, const double* obs,
                                  const double* thr_host, double* d_out, int32_t* acc_idx,
                                  int64_t* n_acc, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx != nullptr, "dist_metric: ctx is NULL");
    ELFI_REQUIRE(metric >= ELFI_B200_METRIC_SQEUCLIDEAN && metric <= ELFI_B200_METRIC_MINKOWSKI,
                 "dist_metric: unknown metric code %d", int(metric));
    ELFI_REQUIRE(metric != ELFI_B200_METRIC_MINKOWSKI || (pexp > 0.0 && pexp < 1e308),
                 "dist_metric: Minkowski exponent must be positive and finite");
    int rc = check_dist_args(S, ldS, B, D, obs, nullptr, 1, thr_host, acc_idx);
    if (rc) return rc;
    ELFI_REQUIRE(B == 0 || d_out != nullptr, "dist_metric: d_out is NULL");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    uint32_t* mask = nullptr;
    if (thr_host != nullptr) {
        mask = static_cast<uint32_t*>(ctx_scratch(ctx, size_t((B + 31) / 32) * 4 + 256));
        if (!mask) return ELFI_B200_ERR_NOMEM;
    }
    rc = launch_metric(ctx, int(metric), pexp, S, ldS, B, D, obs, thr_host, d_out, mask, stream);
    if (rc) return rc;
    if (thr_host != nullptr && (acc_idx != nullptr || n_acc != nullptr))
        return launch_compact_mask(mask, B, acc_idx, n_acc, stream);
    return ELFI_B200_OK;
}

int elfi_b200_dist_seuclidean_thr_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B,
                                      int64_t D, const double* obs, const double* V,
                                      const double* thr_host, double* d_out, int32_t* acc_idx,
                                      int64_t* n_acc, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx != nullptr, "dist_seuclidean: ctx is NULL");
    ELFI_REQUIRE(V != nullptr, "dist_seuclidean: V is NULL");
    int rc = check_dist_args(S, ldS, B, D, obs, nullptr, 1, thr_host, acc_idx);
    if (rc) return rc;
    ELFI_REQUIRE(B == 0 || d_out != nullptr, "dist_seuclidean: d_out is NULL");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    uint32_t* mask = nullptr;
    if (thr_host != nullptr) {
        mask = static_cast<uint32_t*>(ctx_scratch(ctx, size_t((B + 31) / 32) * 4 + 256));
        if (!mask) return ELFI_B200_ERR_NOMEM;
    }
    rc = launch_seuclid(ctx, S, ldS, B, D, obs, V, thr_host, d_out, mask, stream);
    if (rc) return rc;
    if (thr_host != nullptr && (acc_idx != nullptr || n_acc != nullptr))
        return launch_compact_mask(mask, B, acc_idx, n_acc, stream);
    return ELFI_B200_OK;
}

}  // extern "C"
