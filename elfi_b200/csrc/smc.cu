// smc.cu -- SMC-ABC population arithmetic (SURVEY.md K5, K8, K9):
//   * column moments for AdaptiveDistance.add_data      (elfi/model/elfi_model.py:1104-1125)
//   * weighted mean / unbiased weighted variance         (elfi/methods/utils.py:108-139)
//   * Gaussian-mixture proposal density  q(x_i) = sum_j w_j N(x_i; m_j, Sigma)
//     (GMDistribution.pdf/logpdf, elfi/methods/utils.py:146-197) and the importance weights
//     w_i = exp(logprior_i - log q_i)  (elfi/methods/inference/samplers.py:511-514).
//
// The mixture density is the only O(N_new * N_prev) object on the path (1e12 pair terms per
// generation at 1e6 particles): it is bound by the FP64 pipe, not by HBM.  Per pair and
// parameter dimension p: p DFMA + 1 DADD for the (expanded, centred) squared whitened distance
// with the log-weight folded in, then 2^(-nt) by range reduction (round via the 2^52 trick, no
// 64-bit conversions, which run at quarter rate) and a degree-6 minimax polynomial: relative
// error < 2e-9 per term, far inside the 1e-5 relative tolerance on the weights.  Accumulation
// is fp64.
#include "common.cuh"

namespace elfi {

// ---------------------------------------------------------------------------------------------
// K5: per-column shifted power sums of a (B, D) batch: s1_j = sum_i (x_ij - c_j),
// s2_j = sum_i (x_ij - c_j)^2 with the shift c = first row (keeps s2 - s1^2/B well conditioned).
// Grid (row slabs, column groups of 32); block (32, 8).
__global__ void __launch_bounds__(256)
colmoments_partial_kernel(const double* __restrict__ S, int64_t ld, int64_t B, int64_t D,
                          int64_t rows_per_block, double* __restrict__ partial) {
    __shared__ double s1s[8][33], s2s[8][33];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int64_t c = int64_t(blockIdx.y) * 32 + tx;
    const int64_t r0 = int64_t(blockIdx.x) * rows_per_block;
    const int64_t r1 = (r0 + rows_per_block < B) ? r0 + rows_per_block : B;
    double s1 = 0.0, s2 = 0.0;
    if (c < D) {
        const double shift = S[c];
        for (int64_t r = r0 + ty; r < r1; r += 8) {
            const double d = S[r * ld + c] - shift;
            s1 += d;
            s2 = fma(d, d, s2);
        }
    }
    s1s[ty][tx] = s1;
    s2s[ty][tx] = s2;
    __syncthreads();
    if (ty == 0 && c < D) {
        for (int k = 1; k < 8; ++k) { s1 += s1s[k][tx]; s2 += s2s[k][tx]; }
        partial[(int64_t(blockIdx.x) * 2 + 0) * D + c] = s1;
        partial[(int64_t(blockIdx.x) * 2 + 1) * D + c] = s2;
    }
}

// out[0*D + j] = batch mean_j, out[1*D + j] = batch M2_j = sum_i (x_ij - mean_j)^2
__global__ void colmoments_final_kernel(const double* __restrict__ S, const double* __restrict__ partial,
                                        int64_t nblocks, int64_t B, int64_t D,
                                        double* __restrict__ out) {
    const int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (c >= D) return;
    double s1 = 0.0, s2 = 0.0;
    for (int64_t b = 0; b < nblocks; ++b) {
        s1 += partial[(b * 2 + 0) * D + c];
        s2 += partial[(b * 2 + 1) * D + c];
    }
    const double n = double(B);
    out[c] = S[c] + s1 / n;
    out[D + c] = s2 - s1 * s1 / n;
}

// ---------------------------------------------------------------------------------------------
// K8: weighted statistics.  pass 0: V1 = sum w, V2 = sum w^2, xw_j = sum w x_j.
//     pass 1: num_j = sum w (x_j - xbar_j)^2.   p <= 16.
constexpr int WS_MAXP = 16;

__global__ void __launch_bounds__(256)
wstats_partial_kernel(const double* __restrict__ x, int64_t ld, const double* __restrict__ w,
                      int64_t N, int p, int pass, const double* __restrict__ stats,
                      double* __restrict__ partial) {
    __shared__ double red[8][WS_MAXP + 2];
    double acc[WS_MAXP + 2];
#pragma unroll
    for (int k = 0; k < WS_MAXP + 2; ++k) acc[k] = 0.0;
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < N; i += stride) {
        const double wi = w ? w[i] : 1.0;
        if (pass == 0) {
            acc[0] += wi;
            acc[1] = fma(wi, wi, acc[1]);
#pragma unroll
            for (int j = 0; j < WS_MAXP; ++j)
                if (j < p) acc[2 + j] = fma(wi, x[i * ld + j], acc[2 + j]);
        } else {
#pragma unroll
            for (int j = 0; j < WS_MAXP; ++j)
                if (j < p) {
                    const double d = x[i * ld + j] - stats[2 + j];
                    acc[2 + j] = fma(wi, d * d, acc[2 + j]);
                }
        }
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < WS_MAXP + 2; ++k) {
        double v = acc[k];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[wid][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < p + 2) {
        double v = 0.0;
        for (int k = 0; k < 8; ++k) v += red[k][threadIdx.x];
        partial[int64_t(blockIdx.x) * (WS_MAXP + 2) + threadIdx.x] = v;
    }
}

// stats layout: [V1, V2, xbar_0..p-1, s2_0..p-1]
__global__ void wstats_final_kernel(const double* __restrict__ partial, int nblocks, int p, int pass,
                                    double* __restrict__ stats) {
    const int k = threadIdx.x;
    if (k >= p + 2) return;
    double v = 0.0;
    for (int b = 0; b < nblocks; ++b) v += partial[int64_t(b) * (WS_MAXP + 2) + k];
    if (pass == 0) {
        if (k < 2) stats[k] = v;
        __syncthreads();
        if (k >= 2) stats[k] = v / stats[0];                 // np.average: sum(w x) / sum(w)
    } else if (k >= 2) {
        const double V1 = stats[0], V2 = stats[1];
        stats[p + k] = v / (V1 - (V2 / V1));                 // utils.py:138
    }
}

// ---------------------------------------------------------------------------------------------
// K9: Gaussian mixture density.
// Coordinates are centred at the first component (any point of the cloud: the proposal covariance
// is twice the population's own variance, so after centring |y| is a few units), whitened with
// Linv and pre-scaled by sqrt(log2(e)/2), so that for a pair
//   w_j exp(-maha/2) = 2^(-nt),  nt = |y_i|^2 + (|m_j|^2 - log2 w_j) - 2 y_i . m_j.
// The squared distance is expanded: per component the kernel reads (-2 m_j, c_j = |m_j|^2 -
// log2 w_j), per point it keeps (y_i, |y_i|^2), and a pair costs P DFMA + 1 DADD instead of P DSUB
// + P DFMA + the weight multiply.  The cancellation error is |y|^2 * 2^-52 ~ 1e-14 ABSOLUTE in nt,
// i.e. 1e-14 relative in the term (what matters for a density), thanks to the centring.
// 2^(-nt): k = rint(-nt) through the 2^52 trick (no 64-bit conversions, which run on the slow
// XU pipe), f = -nt - k in [-.5, .5], 2^f by the degree-6 minimax polynomial (relative error
// < 1.9e-9, Remez on [-.5, .5]), scaled by 2^k through the exponent field; nt > 1020 flushes to 0
// (and so does a zero weight, whose c_j is +inf).
// fp64-pipe instructions per pair: P + 1 (distance) + 3 (range reduction) + 6 (polynomial)
// + 1 (compare) + 1 (accumulate) = P + 12  (round 1: 2P + 12).
__device__ __forceinline__ double exp2_neg(double nt) {
    const double magic = 6755399441055744.0;  // 1.5 * 2^52
    const double tm = magic - nt;
    const double kd = tm - magic;             // rint(-nt)
    const double f = -nt - kd;
    double pz = 1.5345812158740182e-04;
    pz = fma(pz, f, 1.3399931209474140e-03);
    pz = fma(pz, f, 9.6184889565227916e-03);
    pz = fma(pz, f, 5.5503287769976638e-02);
    pz = fma(pz, f, 2.4022646890639572e-01);
    pz = fma(pz, f, 6.9314720573725268e-01);
    pz = fma(pz, f, 1.0000000005541663e+00);
    const int k = __double2loint(tm);         // low word of (magic - nt) holds rint(-nt)
    const int hi = __double2hiint(pz) + (k << 20);
    const double r = __hiloint2double(hi, __double2loint(pz));
    return (nt <= 1020.0) ? r : 0.0;
}

// Mixed-precision variant of exp2_neg (elfi_b200_gm_logpdf_mixed_f64): the range reduction
// stays in fp64 (the integer / fraction split of nt needs it), but 2^f for f in [-.5, .5] comes
// from the special-function unit in fp32 (ex2.approx: 2 ulp, ~1.7e-7 relative) and is widened
// back to fp64 with integer operations while the exponent k is added -- no polynomial: the
// fp64 pipe issues 8 instructions per pair at P = 2 instead of 14, the rest runs on the
// XU (F2F + MUFU) and integer pipes concurrently.  Accuracy ~2e-7 per term against the 1e-5
// relative tolerance on the weights; the fp64 path (1.9e-9) stays the default.
__device__ __forceinline__ double exp2_neg_mixed(double nt) {
    const double magic = 6755399441055744.0;  // 1.5 * 2^52
    const double tm = magic - nt;
    const double kd = tm - magic;             // rint(-nt)
    const float f = __double2float_rn(-nt - kd);
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(f));     // in [0.707, 1.415]
    const unsigned eb = __float_as_uint(e);
    const int k = __double2loint(tm);
    const int hi = int(((eb >> 23) + unsigned(1023 - 127 + k)) << 20) | int((eb >> 3) & 0xFFFFFu);
    const double r = __hiloint2double(hi, int(eb << 29));
    return (nt <= 1020.0) ? r : 0.0;
}

// Whitened, centred, scaled coordinates y = s Linv (x - centre) with s = sqrt(log2(e)/2).
//   points     (mode 0): out[i] = (y_0 .. y_{p-1}, |y|^2)
//   components (mode 1): out[j] = (-2 y_0 .. -2 y_{p-1}, |y|^2 - log2(w_j / sum w))
__global__ void gm_whiten_kernel(const double* __restrict__ x, int64_t ld, int64_t n, int p,
                                 const double* __restrict__ Linv, const double* __restrict__ centre,
                                 int mode, const double* __restrict__ w,
                                 const double* __restrict__ wsum, double* __restrict__ out) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double scale = 0.8493218002880191;   // sqrt(log2(e) / 2)
    double yy = 0.0;
    for (int a = 0; a < p; ++a) {
        double s = 0.0;
        for (int b = 0; b <= a; ++b) s = fma(Linv[a * p + b], x[i * ld + b] - centre[b], s);
        s *= scale;
        yy = fma(s, s, yy);
        out[i * (p + 1) + a] = mode ? -2.0 * s : s;
    }
    if (mode) {
        const double wn = w ? w[i] / wsum[0] : 1.0 / double(n);
        yy -= log2(wn);                        // w = 0: +inf, the component never contributes
    }
    out[i * (p + 1) + p] = yy;
}

// grid = (point blocks, component chunks).  Each CTA accumulates its chunk of the mixture for
// 128 * R points and writes one partial sum per point; gm_finish_kernel adds the chunks in a
// fixed order (deterministic) and takes the log.  The 2-D grid keeps >= 8 CTAs per SM even when a
// rank owns only ~1e5 points, which the dependent polynomial chains need to fill the fp64 pipe.
template <int P, int R, bool MIXED = false>
__global__ void __launch_bounds__(128)
gm_pdf_kernel(const double* __restrict__ xw, int64_t N, const double* __restrict__ mw, int64_t M,
              int64_t chunk_len, double* __restrict__ partial) {
    constexpr int TILE = 512;
    __shared__ double sm[TILE * (P + 1)];
    double x[R][P + 1];
    double acc[R];
    const int64_t i0 = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) * R;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        acc[r] = 0.0;
#pragma unroll
        for (int a = 0; a <= P; ++a) x[r][a] = (i0 + r < N) ? xw[(i0 + r) * (P + 1) + a] : 0.0;
    }
    const int64_t jbeg = int64_t(blockIdx.y) * chunk_len;
    const int64_t jend = (jbeg + chunk_len < M) ? jbeg + chunk_len : M;
    for (int64_t j0 = jbeg; j0 < jend; j0 += TILE) {
        const int cnt = int((jend - j0) < TILE ? (jend - j0) : TILE);
        __syncthreads();
        for (int t = threadIdx.x; t < cnt * (P + 1); t += blockDim.x)
            sm[t] = mw[j0 * (P + 1) + t];
        __syncthreads();
#pragma unroll 2
        for (int j = 0; j < cnt; ++j) {
            double m[P];
#pragma unroll
            for (int a = 0; a < P; ++a) m[a] = sm[j * (P + 1) + a];
            const double cj = sm[j * (P + 1) + P];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                double g = cj;
#pragma unroll
                for (int a = 0; a < P; ++a) g = fma(x[r][a], m[a], g);
                acc[r] += MIXED ? exp2_neg_mixed(g + x[r][P]) : exp2_neg(g + x[r][P]);
            }
        }
    }
#pragma unroll
    for (int r = 0; r < R; ++r)
        if (i0 + r < N) partial[int64_t(blockIdx.y) * N + i0 + r] = acc[r];
}

__global__ void gm_finish_kernel(const double* __restrict__ partial, int64_t N, int chunks,
                                 double lognorm, double* __restrict__ logq) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= N) return;
    double s = 0.0;
    for (int c = 0; c < chunks; ++c) s += partial[int64_t(c) * N + i];
    logq[i] = log(s) + lognorm;
}

// generic p (<= 16), one point per thread
__global__ void __launch_bounds__(128)
gm_pdf_generic_kernel(const double* __restrict__ xw, int64_t N, const double* __restrict__ mw,
                      int64_t M, int p, double lognorm, double* __restrict__ logq) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= N) return;
    double x[WS_MAXP + 1];
    for (int a = 0; a <= p; ++a) x[a] = xw[i * (p + 1) + a];
    double acc = 0.0;
    for (int64_t j = 0; j < M; ++j) {
        double g = __ldg(mw + j * (p + 1) + p);
        for (int a = 0; a < p; ++a) g = fma(x[a], __ldg(mw + j * (p + 1) + a), g);
        acc += exp2_neg(g + x[p]);
    }
    logq[i] = log(acc) + lognorm;
}

__global__ void sum_kernel(const double* __restrict__ v, int64_t n, double* __restrict__ out) {
    // single block, deterministic
    __shared__ double ws[32];
    double acc = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc += v[i];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        double t = threadIdx.x < (blockDim.x >> 5) ? ws[threadIdx.x] : 0.0;
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (threadIdx.x == 0) out[0] = t;
    }
}

__global__ void smc_weights_kernel(const double* __restrict__ logprior, const double* __restrict__ logq,
                                   int64_t n, double* __restrict__ w) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) w[i] = exp(logprior[i] - logq[i]);
}

}  // namespace elfi

extern "C" {

int elfi_b200_colmoments_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B, int64_t D,
                             double* out, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && S && out, "colmoments: NULL argument");
    ELFI_REQUIRE(B >= 1 && D >= 1 && ldS >= D, "colmoments: bad shape");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    const int64_t colgroups = (D + 31) / 32;
    int64_t slabs = (int64_t(ctx->sm_count) * 8 + colgroups - 1) / colgroups;
    int64_t rows_per_block = (B + slabs - 1) / slabs;
    if (rows_per_block < 64) rows_per_block = 64;
    slabs = (B + rows_per_block - 1) / rows_per_block;
    double* partial = static_cast<double*>(ctx_scratch(ctx, size_t(slabs) * 2 * D * 8 + 256));
    if (!partial) return ELFI_B200_ERR_NOMEM;
    colmoments_partial_kernel<<<dim3(unsigned(slabs), unsigned(colgroups)), dim3(32, 8), 0, stream>>>(
        S, ldS, B, D, rows_per_block, partial);
    colmoments_final_kernel<<<unsigned((D + 127) / 128), 128, 0, stream>>>(S, partial, slabs, B, D, out);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_weighted_stats_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, const double* w,
                                 int64_t N, int64_t p, double* stats, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && x && stats, "weighted_stats: NULL argument");
    ELFI_REQUIRE(N >= 1 && p >= 1 && p <= WS_MAXP && ldx >= p, "weighted_stats: bad shape (p <= %d)",
                 WS_MAXP);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    int blocks = int((N + 255) / 256);
    if (blocks > ctx->sm_count * 4) blocks = ctx->sm_count * 4;
    double* partial = static_cast<double*>(ctx_scratch(ctx, size_t(blocks) * (WS_MAXP + 2) * 8 + 256));
    if (!partial) return ELFI_B200_ERR_NOMEM;
    for (int pass = 0; pass < 2; ++pass) {
        wstats_partial_kernel<<<blocks, 256, 0, stream>>>(x, ldx, w, N, int(p), pass, stats, partial);
        wstats_final_kernel<<<1, 32, 0, stream>>>(partial, blocks, int(p), pass, stats);
    }
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

static int gm_logpdf_impl(elfi_b200_ctx* ctx, const double* x, int64_t ldx, int64_t N,
                          const double* means, int64_t ldm, const double* w, int64_t M, int64_t p,
                          const double* Linv_host, double logdet, double* logq, void* stream_,
                          bool mixed) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && x && means && Linv_host && logq, "gm_logpdf: NULL argument");
    ELFI_REQUIRE(N >= 0 && M >= 1 && p >= 1 && p <= WS_MAXP && ldx >= p && ldm >= p,
                 "gm_logpdf: bad shape (p <= %d)", WS_MAXP);
    if (N == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    auto align = [](size_t v) { return (v + 255) & ~size_t(255); };
    // Component chunks.  The chunk length depends on M ONLY, never on N: a point's partial sums are
    // then added in the same order whether a rank evaluates all N points or a shard of them, so
    // the sharded multi-GPU density is bit-identical to the single-GPU one.  M / 64 components per
    // chunk (clamped to [2048, 16384], multiple of the 512-component smem tile) gives >= 8 CTAs
    // per SM from N ~ 1e4 points per rank upwards while a CTA's prologue stays negligible.
    constexpr int R = 4;
    const int64_t xblocks = (N + 128 * R - 1) / (128 * R);
    int64_t chunks = 1, chunk_len = M;
    if (p <= 4) {
        chunk_len = ((M / 64 + 511) / 512) * 512;
        if (chunk_len < 2048) chunk_len = 2048;
        if (chunk_len > 16384) chunk_len = 16384;
        chunks = (M + chunk_len - 1) / chunk_len;
        ELFI_REQUIRE(chunks <= 65535, "gm_logpdf: too many component chunks (%lld)", (long long)chunks);
    }
    const size_t off_xw = align(size_t(p) * p * 8);
    const size_t off_mw = off_xw + align(size_t(N) * (p + 1) * 8);
    const size_t off_ws = off_mw + align(size_t(M) * (p + 1) * 8);
    const size_t off_part = off_ws + 256;
    uint8_t* base = static_cast<uint8_t*>(ctx_scratch(ctx, off_part + size_t(chunks) * N * 8 + 256));
    if (!base) return ELFI_B200_ERR_NOMEM;
    double* Linv = reinterpret_cast<double*>(base);
    double* xw = reinterpret_cast<double*>(base + off_xw);
    double* mw = reinterpret_cast<double*>(base + off_mw);
    double* wsum = reinterpret_cast<double*>(base + off_ws);
    double* partial = reinterpret_cast<double*>(base + off_part);
    ELFI_CUDA_OK(cudaMemcpyAsync(Linv, Linv_host, size_t(p) * p * 8, cudaMemcpyHostToDevice, stream));
    if (w) sum_kernel<<<1, 1024, 0, stream>>>(w, M, wsum);
    gm_whiten_kernel<<<unsigned((N + 255) / 256), 256, 0, stream>>>(x, ldx, N, int(p), Linv, means, 0,
                                                                   nullptr, nullptr, xw);
    gm_whiten_kernel<<<unsigned((M + 255) / 256), 256, 0, stream>>>(means, ldm, M, int(p), Linv, means,
                                                                   1, w, wsum, mw);
    const double lognorm = -0.5 * (double(p) * 1.8378770664093453 + logdet);  // log(2 pi)
    if (p <= 4) {
        dim3 grid(static_cast<unsigned>(xblocks), static_cast<unsigned>(chunks));
        if (mixed) {
            switch (p) {
                case 1: gm_pdf_kernel<1, R, true><<<grid, 128, 0, stream>>>(xw, N, mw, M, chunk_len, partial); break;
                case 2: gm_pdf_kernel<2, R, true><<<grid, 128, 0, stream>>>(xw, N, mw, M, chunk_len, partial); break;
                case 3: gm_pdf_kernel<3, R, true><<<grid, 128, 0, stream>>>(xw, N, mw, M, chunk_len, partial); break;
                default: gm_pdf_kernel<4, R, true><<<grid, 128, 0, stream>>>(xw, N, mw, M, chunk_len, partial); break;
            }
        } else {
            switch (p) {
                case 1: gm_pdf_kernel<1, R><<<grid, 128, 0, stream>>>(xw, N, mw, M, chunk_len, partial); break;
                case 2: gm_pdf_kernel<2, R><<<grid, 128, 0, stream>>>(xw, N, mw, M, chunk_len, partial); break;
                case 3: gm_pdf_kernel<3, R><<<grid, 128, 0, stream>>>(xw, N, mw, M, chunk_len, partial); break;
                default: gm_pdf_kernel<4, R><<<grid, 128, 0, stream>>>(xw, N, mw, M, chunk_len, partial); break;
            }
        }
        gm_finish_kernel<<<unsigned((N + 255) / 256), 256, 0, stream>>>(partial, N, int(chunks), lognorm, logq);
    } else {
        gm_pdf_generic_kernel<<<unsigned((N + 127) / 128), 128, 0, stream>>>(xw, N, mw, M, int(p),
                                                                          lognorm, logq);
    }
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_gm_logpdf_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, int64_t N,
                            const double* means, int64_t ldm, const double* w, int64_t M, int64_t p,
                            const double* Linv_host, double logdet, double* logq, void* stream_) {
    return gm_logpdf_impl(ctx, x, ldx, N, means, ldm, w, M, p, Linv_host, logdet, logq, stream_, false);
}

int elfi_b200_gm_logpdf_mixed_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, int64_t N,
                                  const double* means, int64_t ldm, const double* w, int64_t M,
                                  int64_t p, const double* Linv_host, double logdet, double* logq,
                                  void* stream_) {
    return gm_logpdf_impl(ctx, x, ldx, N, means, ldm, w, M, p, Linv_host, logdet, logq, stream_, true);
}

int elfi_b200_smc_weights_f64(elfi_b200_ctx* ctx, const double* logprior, const double* logq,
                              int64_t n, double* w, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && (n == 0 || (logprior && logq && w)), "smc_weights: NULL argument");
    if (n == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    smc_weights_kernel<<<unsigned((n + 255) / 256), 256, 0, stream>>>(logprior, logq, n, w);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

}  // extern "C"
