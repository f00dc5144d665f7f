// synlik.cu -- batched Gaussian synthetic likelihood of BSL (elfi/methods/bsl/pdf_methods.py:77-176,
// cov_warton.py:6-30), fp64.
//
// One CTA per group of n simulated summary rows (d columns, d <= 128):
//   1. one pass over the rows, shifted by the group's first row s: the column sums of (x - s) and
//      the upper triangle of the Gram matrix sum (x - s)(x - s)^T on the DMMA pipe (8 x 8 tiles,
//      four rows per instruction); Sigma = (G - n (m - s)(m - s)^T) / (n - 1) is np.cov with
//      ddof = 1 from ONE read of the rows (np.cov reads them twice);
//   2. optional whitening Sigma' = Wh Sigma Wh^T, r' = Wh r (algebraically the reference's whitening
//      of every row, pdf_methods.py:106-108);
//   3. per Warton parameter gamma: A = gamma Sigma + (1 - gamma) diag(Sigma_ii + 1e-5) (closed form of
//      cov_warton incl. its `np.diag(S + eps)`), Cholesky A = L L^T, z = L^-1 (obs - mu),
//      loglik = -(|z|^2 + log det A + d log 2 pi) / 2; the Ghurye-Olkin estimator takes
//      log|det psi| from the same factor (matrix determinant lemma).
// Sigma lives in the strict upper triangle of a d x d shared buffer plus a diagonal vector; each
// factorisation writes L into the strict lower triangle and its diagonal into a second vector, so
// the L penalties refactor from the saved Sigma.  A group with a non-finite value, or a pivot at or
// below 1e6 eps max_j A_jj (SciPy's _PSD cutoff constant applied to pivots), gives -inf.
//
// Roofline per group: bytes n d 8; FMAs n d (d + 1) / 2 (Gram) + L d^3 / 6 (Cholesky).
#include "common.cuh"
#include "dmma.cuh"

#include <cmath>

namespace elfi {

constexpr int SL_WARPS = 8;
constexpr int SL_THREADS = 32 * SL_WARPS;
constexpr int SL_ROWS = 32;                  // rows staged per pass (a multiple of 4)
// Gram tiles per warp (accumulators held in registers): ceil(136 / 8) = 17 at d = 128, 5 up to
// d = 64.  The small instance needs a third of the registers, so several CTAs share an SM.
constexpr int SL_MAXT_SMALL = 5, SL_MAXT_LARGE = 17, SL_SMALL_MAX_D = 64;

struct SynlikArgs {
    const double* S; int64_t ldS;
    int64_t n, group_stride;
    int d, dpad, ldx;
    const double* obs;
    const double* Wh;
    const double* gammas;   // device, L entries, or NULL
    int L;
    int estimator;
    double* loglik;
};

// Tile index t of the upper triangle of an nt x nt tile grid, row-major: (I, J), I <= J.
__device__ __forceinline__ void tile_of(int t, int nt, int& I, int& J) {
    I = 0;
    while (t >= nt - I) {
        t -= nt - I;
        ++I;
    }
    J = I + t;
}

__device__ __forceinline__ double wcon(int k, double nu) {
    double s = 0.0;
    for (int x = 0; x < k; ++x) s += lgamma(0.5 * (nu - x));
    return -k * nu / 2 * log(2.0) - k * (k - 1) / 4.0 * log(M_PI) - s;
}

template <int SL_MAXT>
__global__ void __launch_bounds__(SL_THREADS) synlik_kernel(SynlikArgs a) {
    extern __shared__ double sm[];
    const int d = a.d, dpad = a.dpad, ldx = a.ldx;
    double* M = sm;                              // d x d: Sigma strict upper, L strict lower
    double* X = M + d * d;                       // SL_ROWS x ldx staged (x - s), zero padded
    double* vs = X + SL_ROWS * ldx;              // shift s, then the residual obs - mu
    double* vsum = vs + dpad;                    // column sums of (x - s)
    double* vdiag = vsum + dpad;                 // Sigma_ii
    double* vl = vdiag + dpad;                   // diag of L (and of Sigma' while whitening)
    double* vt = vl + dpad;                      // scratch vector (z, whitening row)
    double* part = vt + dpad;                    // SL_WARPS x 64 partial Gram tiles
    __shared__ int bad;
    __shared__ double red[SL_WARPS];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t n = a.n;
    const double* base = a.S + int64_t(blockIdx.x) * a.group_stride * a.ldS;
    if (tid == 0) bad = 0;
    for (int j = tid; j < dpad; j += SL_THREADS) vs[j] = j < d ? base[j] : 0.0;

    // Gram tiles of this warp: all k-steps of tiles warp, warp + 8, ... when there are at least 8
    // tiles; otherwise `slices` warps share one tile and split its k-steps (summed in order below)
    const int nt = dpad / 8, T = nt * (nt + 1) / 2;
    const int slices = T >= SL_WARPS ? 1 : SL_WARPS / T;
    const int slice = T >= SL_WARPS ? 0 : warp / T;
    const int first = T >= SL_WARPS ? warp : warp % T;
    const int step = T >= SL_WARPS ? SL_WARPS : T;   // any value > T - first ends the list
    int nmine = 0;
    if (slice < slices)
        for (int t = first; t < T; t += step) ++nmine;
    int off[SL_MAXT];   // fragment columns of tile q: I * 8 + lane / 4 | (J * 8 + lane / 4) << 16
    double acc[SL_MAXT][2];
#pragma unroll
    for (int q = 0; q < SL_MAXT; ++q) {
        int I = 0, J = 0;
        if (q < nmine) tile_of(first + q * step, nt, I, J);
        off[q] = (I * 8 + (lane >> 2)) | ((J * 8 + (lane >> 2)) << 16);
        acc[q][0] = acc[q][1] = 0.0;
    }
    double csum = 0.0;
    __syncthreads();

    for (int64_t r0 = 0; r0 < n; r0 += SL_ROWS) {
        const int rows = n - r0 < SL_ROWS ? int(n - r0) : SL_ROWS;
        __syncthreads();   // the previous chunk has been consumed
        for (int e = tid; e < SL_ROWS * dpad; e += SL_THREADS) {
            const int rr = e / dpad, c = e - rr * dpad;
            double v = 0.0;
            if (rr < rows && c < d) {
                const double x = base[(r0 + rr) * a.ldS + c];
                if (!isfinite(x)) bad = 1;
                v = x - vs[c];
            }
            X[rr * ldx + c] = v;
        }
        __syncthreads();
        if (tid < d)
            for (int rr = 0; rr < rows; ++rr) csum += X[rr * ldx + tid];
        const int nk = (rows + 3) >> 2;
        for (int ks = slice; ks < nk; ks += slices) {
            const double* xr = X + (ks * 4 + (lane & 3)) * ldx;
#pragma unroll
            for (int q = 0; q < SL_MAXT; ++q)
                if (q < nmine)
                    dmma_m8n8k4(acc[q][0], acc[q][1], xr[off[q] & 0xffff], xr[off[q] >> 16]);
        }
    }
    if (tid < d) vsum[tid] = csum;

    // Gram entries (i <= j < d) -> M[i][j] (strict upper) / vdiag[i]
    const int gi = lane >> 2, gj = (lane & 3) * 2;
    if (slices == 1) {
#pragma unroll
        for (int q = 0; q < SL_MAXT; ++q) {
            if (q < nmine) {
                const int i = off[q] & 0xffff, j0 = (off[q] >> 16) - gi + gj;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int j = j0 + h;
                    if (i < d && j < d && i <= j) {
                        if (i == j) vdiag[i] = acc[q][h];
                        else M[i * d + j] = acc[q][h];
                    }
                }
            }
        }
    } else {
        if (nmine) {
            part[warp * 64 + lane * 2] = acc[0][0];
            part[warp * 64 + lane * 2 + 1] = acc[0][1];
        }
        __syncthreads();
        // warp w held slice w / T of tile w % T; sum the slices of each tile in slice order
        for (int e = tid; e < T * 64; e += SL_THREADS) {
            const int t = e >> 6, l = (e & 63) >> 1, h = e & 1;
            double v = 0.0;
            for (int s = 0; s < slices; ++s) v += part[(s * T + t) * 64 + l * 2 + h];
            int I, J;
            tile_of(t, nt, I, J);
            const int i = I * 8 + (l >> 2), j = J * 8 + (l & 3) * 2 + h;
            if (i < d && j < d && i <= j) {
                if (i == j) vdiag[i] = v;
                else M[i * d + j] = v;
            }
        }
    }
    __syncthreads();

    // np.cov (ddof = 1) and the residual obs - mean
    const double dn = double(n), inv_n1 = 1.0 / double(n - 1);
    for (int e = tid; e < d * d; e += SL_THREADS) {
        const int i = e / d, j = e - i * d;
        if (i < j) M[e] = (M[e] - vsum[i] * vsum[j] / dn) * inv_n1;
    }
    if (tid < d) {
        vdiag[tid] = (vdiag[tid] - vsum[tid] * vsum[tid] / dn) * inv_n1;
        vs[tid] = a.obs[tid] - (vs[tid] + vsum[tid] / dn);
    }
    __syncthreads();

    if (a.Wh) {
        // r' = Wh r;  Sigma' = Wh Sigma Wh^T row by row into the strict lower triangle + vl
        if (tid < d) {
            double v = 0.0;
            for (int k = 0; k < d; ++k) v = fma(a.Wh[tid * d + k], vs[k], v);
            vt[tid] = v;
        }
        __syncthreads();
        if (tid < d) vs[tid] = vt[tid];
        for (int i = 0; i < d; ++i) {
            __syncthreads();
            if (tid < d) {   // u_l = sum_k Wh_ik Sigma_kl
                double v = 0.0;
                for (int k = 0; k < d; ++k) {
                    const double s = k < tid ? M[k * d + tid] : (k > tid ? M[tid * d + k] : vdiag[k]);
                    v = fma(a.Wh[i * d + k], s, v);
                }
                vt[tid] = v;
            }
            __syncthreads();
            for (int j = i + tid; j < d; j += SL_THREADS) {
                double v = 0.0;
                for (int l = 0; l < d; ++l) v = fma(vt[l], a.Wh[j * d + l], v);
                if (j == i) vl[i] = v;
                else M[j * d + i] = v;
            }
        }
        __syncthreads();
        for (int e = tid; e < d * d; e += SL_THREADS) {
            const int i = e / d, j = e - i * d;
            if (i < j) M[e] = M[j * d + i];
        }
        if (tid < d) vdiag[tid] = vl[tid];
        __syncthreads();
    }

    const double log2pi = 1.8378770664093453;
    for (int l = 0; l < a.L; ++l) {
        const double g = a.gammas ? a.gammas[l] : 1.0;
        __syncthreads();   // the previous factor is no longer read
        for (int e = tid; e < d * d; e += SL_THREADS) {
            const int i = e / d, j = e - i * d;
            if (j < i) M[e] = g * M[j * d + i];
        }
        if (tid < d)
            vt[tid] = a.gammas ? g * vdiag[tid] + (1.0 - g) * (vdiag[tid] + 1e-5) : vdiag[tid];
        __syncthreads();
        if (warp == 0) {
            double m = 0.0;
            for (int j = lane; j < d; j += 32) m = fmax(m, vt[j]);
            for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
            if (lane == 0) red[0] = m;
        }
        __syncthreads();
        const double tol = 1e6 * 2.220446049250313e-16 * red[0];
        // right-looking Cholesky: column k of L in M[i][k] (i > k), L_kk in vl[k]; vt holds the
        // running diagonal of the trailing matrix
        bool singular = false;
        for (int k = 0; k < d; ++k) {
            const double piv = vt[k];
            if (!(piv > tol)) {
                singular = true;
                break;
            }
            const double lkk = sqrt(piv);
            if (tid == 0) vl[k] = lkk;
            for (int i = k + 1 + tid; i < d; i += SL_THREADS) M[i * d + k] /= lkk;
            __syncthreads();
            const int m = d - k - 1;
            for (int e = tid; e < m * m; e += SL_THREADS) {
                const int ii = e / m, jj = e - ii * m;
                if (jj < ii) {
                    const int i = k + 1 + ii, j = k + 1 + jj;
                    M[i * d + j] -= M[i * d + k] * M[j * d + k];
                } else if (jj == ii) {
                    const int i = k + 1 + ii;
                    vt[i] -= M[i * d + k] * M[i * d + k];
                }
            }
            __syncthreads();
        }
        if (warp == 0) {
            double out = -INFINITY;
            if (!singular && !bad) {
                // forward substitution z = L^-1 r (z in part[], warp 0 only), q = |z|^2
                double q = 0.0, logdet = 0.0;
                for (int i = 0; i < d; ++i) {
                    double s = 0.0;
                    for (int k = lane; k < i; k += 32) s = fma(M[i * d + k], part[k], s);
                    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                    const double z = (vs[i] - s) / vl[i];
                    __syncwarp();
                    if (lane == 0) part[i] = z;
                    __syncwarp();
                    q = fma(z, z, q);
                    logdet += 2.0 * log(vl[i]);
                }
                if (a.estimator == ELFI_B200_SYNLIK_GAUSSIAN) {
                    out = -0.5 * (q + logdet + d * log2pi);
                } else {
                    const double n1 = dn - 1.0;
                    const double logdet_psi = d * log(n1) + logdet + log(fabs(1.0 - q * dn / (n1 * n1)));
                    const double A = wcon(d, dn - 2.0) - wcon(d, n1) - 0.5 * d * log(1.0 - 1.0 / dn);
                    const double B = -0.5 * (dn - d - 2.0) * (log(n1) + logdet);
                    const double C = 0.5 * (dn - d - 3.0) * logdet_psi;
                    out = -0.5 * d * log2pi + A + B + C;
                }
            }
            if (lane == 0) a.loglik[int64_t(blockIdx.x) * a.L + l] = out;
        }
    }
}

}  // namespace elfi

extern "C" int elfi_b200_synlik_f64(elfi_b200_ctx* ctx, int32_t estimator, const double* S,
                                    int64_t ldS, int64_t P, int64_t n, int64_t group_stride,
                                    int64_t d, const double* obs, const double* Wh,
                                    const double* gamma_host, int64_t L, double* loglik,
                                    void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx, "synlik: NULL context");
    ELFI_REQUIRE(estimator == ELFI_B200_SYNLIK_GAUSSIAN || estimator == ELFI_B200_SYNLIK_GHURYE_OLKIN,
                 "synlik: unknown estimator %d", int(estimator));
    ELFI_REQUIRE(d >= 1 && d <= ELFI_B200_SYNLIK_MAX_D, "synlik: d = %lld outside [1, %d]",
                 (long long)d, ELFI_B200_SYNLIK_MAX_D);
    ELFI_REQUIRE(n >= 2, "synlik: n = %lld, at least 2 rows per group are needed", (long long)n);
    ELFI_REQUIRE(group_stride >= n, "synlik: group_stride %lld < n %lld", (long long)group_stride,
                 (long long)n);
    ELFI_REQUIRE(P >= 0, "synlik: P = %lld < 0", (long long)P);
    ELFI_REQUIRE(L >= 1, "synlik: L = %lld < 1", (long long)L);
    ELFI_REQUIRE(gamma_host || L == 1, "synlik: without gammas L must be 1 (got %lld)", (long long)L);
    ELFI_REQUIRE(ldS >= d, "synlik: ldS %lld < d %lld", (long long)ldS, (long long)d);
    ELFI_REQUIRE(estimator == ELFI_B200_SYNLIK_GAUSSIAN || (!Wh && !gamma_host),
                 "synlik: the Ghurye-Olkin estimator takes neither whitening nor shrinkage");
    if (gamma_host)
        for (int64_t l = 0; l < L; ++l)
            ELFI_REQUIRE(gamma_host[l] >= 0.0 && gamma_host[l] <= 1.0,
                         "synlik: gamma[%lld] = %g outside [0, 1]", (long long)l, gamma_host[l]);
    if (P == 0) return ELFI_B200_OK;
    ELFI_REQUIRE(S && obs && loglik, "synlik: NULL argument");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));

    SynlikArgs a;
    a.S = S; a.ldS = ldS; a.n = n; a.group_stride = group_stride;
    a.d = int(d);
    a.dpad = int((d + 7) / 8 * 8);
    a.ldx = (a.dpad + 15) / 16 * 16 + 4;   // row pitch = 4 mod 16 doubles: conflict-free fragments
    a.obs = obs; a.Wh = Wh; a.gammas = nullptr; a.L = int(L); a.estimator = estimator;
    a.loglik = loglik;
    if (gamma_host) {
        double* g = static_cast<double*>(ctx_scratch(ctx, size_t(L) * sizeof(double)));
        if (!g) return ELFI_B200_ERR_NOMEM;
        ELFI_CUDA_OK(cudaMemcpyAsync(g, gamma_host, size_t(L) * sizeof(double),
                                     cudaMemcpyHostToDevice, stream));
        a.gammas = g;
    }
    const size_t smem = (size_t(d) * d + size_t(SL_ROWS) * a.ldx + 5 * size_t(a.dpad) +
                         SL_WARPS * 64) * sizeof(double);
    auto kern = d <= SL_SMALL_MAX_D ? synlik_kernel<SL_MAXT_SMALL> : synlik_kernel<SL_MAXT_LARGE>;
    ELFI_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    kern<<<unsigned(P), SL_THREADS, smem, stream>>>(a);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}
