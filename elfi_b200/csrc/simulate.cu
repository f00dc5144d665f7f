// simulate.cu -- device-side generation for the throughput mode (SURVEY.md section 8f, row N2):
// MA2 prior draws, the MA2 simulator fused with its autocovariance summaries, and Gaussian-mixture
// proposals with the MA2 prior support, so that a whole SMC-ABC batch is born in HBM and only
// accepted particles ever leave the device.
//
// Reference functions mirrored (statistically, not bit-wise: the reference draws from a host
// MT19937 RandomState, here a counter-based Philox4x32-10 stream keyed by (seed, batch, row)):
//   elfi/examples/ma2.py:11-37    MA2(t1, t2)              x_i = w_i + t1 w_{i-1} + t2 w_{i-2}
//   elfi/examples/ma2.py:40-59    autocov (lags 1, 2), NumPy pairwise summation order kept
//   elfi/examples/ma2.py:96-186   CustomPrior1 (triangular t1), CustomPrior2 (uniform t2 | t1)
//   elfi/methods/utils.py:200-261 GMDistribution.rvs (choice by weights + MVN perturbation +
//                                 rejection of draws outside the prior support)
// The random numbers are a pure function of (seed, stream, row, index): the simulator can be
// replayed (e.g. to materialise X for a test) and any sharding of rows gives the same particles.
#include "gnkmath.cuh"
#include "leafsum.cuh"
#include "pairwise.cuh"

namespace elfi {

struct Philox {
    uint32_t key0, key1;
    __device__ __forceinline__ Philox(uint64_t seed) : key0(uint32_t(seed)), key1(uint32_t(seed >> 32)) {}
    __device__ __forceinline__ uint4 operator()(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) const {
        uint32_t k0 = key0, k1 = key1;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
            const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
            const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
            c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
            k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
        }
        return make_uint4(c0, c1, c2, c3);
    }
};

__device__ __forceinline__ double u01(uint32_t a, uint32_t b) {   // (0, 1], 53 bits
    const uint64_t v = (uint64_t(a) << 21) ^ uint64_t(b >> 11);
    return (double(v & ((uint64_t(1) << 53) - 1)) + 1.0) * (1.0 / 9007199254740992.0);
}

// two standard normals from one Philox block (Box-Muller)
__device__ __forceinline__ void normal2(const uint4& r, double& n0, double& n1) {
    const double u = u01(r.x, r.y), v = u01(r.z, r.w);
    const double rad = sqrt(-2.0 * log(u));
    double s, c;
    sincospi(2.0 * v, &s, &c);
    n0 = rad * c;
    n1 = rad * s;
}

// ---- MA2 prior ------------------------------------------------------------------------------
// mode 0: joint draw (t1, t2); mode 1: t1 only; mode 2: t2 given the t1 passed in.
__global__ void prior_ma2_kernel(int64_t B, uint64_t seed, uint64_t offset, int mode,
                                 double* __restrict__ t1, double* __restrict__ t2) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= B) return;
    const Philox ph(seed);
    const uint64_t row = offset + uint64_t(i);
    const uint4 r = ph(uint32_t(row), uint32_t(row >> 32), 0u, 0x50524931u);
    const double u = u01(r.x, r.y), v = u01(r.z, r.w);
    const double b = 2.0, a = 1.0;
    double x1;
    if (mode == 2) {
        x1 = t1[i];
    } else {
        x1 = u < 0.5 ? sqrt(2.0 * u) * b - b : -sqrt(2.0 * (1.0 - u)) * b + b;
        t1[i] = x1;
    }
    if (mode != 1) {
        const double loc = fmax(-a - x1, -a + x1);
        t2[i] = loc + (a - loc) * v;
    }
}

__device__ __forceinline__ bool ma2_in_support(double x1, double x2) {
    const double ax = fabs(x1);
    return ax < 2.0 && x2 >= -1.0 + ax && x2 <= 1.0;
}

// log p(t1) + log p(t2 | t1) of the MA2 priors (b = 2, a = 1); -inf outside the support
__global__ void logprior_ma2_kernel(const double* __restrict__ x, int64_t ld, int64_t B,
                                    double* __restrict__ out) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= B) return;
    const double x1 = x[i * ld], x2 = x[i * ld + 1];
    const double ax = fabs(x1);
    double lp = -INFINITY;
    if (ma2_in_support(x1, x2)) lp = log(0.5 - ax * 0.25) - log(2.0 - ax);
    out[i] = lp;
}

// Elements k0 + E .. k0 + 7 of a group of eight: their lag-1 / lag-2 products into the leaf sums
// (E is a template parameter because the slot of a product, index % 8, must be static).
template <int E>
__device__ __forceinline__ void ma2_leaf_products(LeafSum& l1, LeafSum& l2, const double (&x)[8],
                                                  double xm1, double xm2, bool mid, int k0,
                                                  int cnt) {
    const double prev1 = (E == 0) ? xm1 : x[E >= 1 ? E - 1 : 0];
    const double prev2 = (E == 0) ? xm2 : (E == 1 ? xm1 : x[E >= 2 ? E - 2 : 0]);
    if (mid) {
        l1.push_mid<(E + 7) & 7>(__dmul_rn(x[E], prev1));
        l2.push_mid<(E + 6) & 7>(__dmul_rn(x[E], prev2));
    } else if (E < cnt) {
        const int k = k0 + E;
        if (k >= 1) l1.push<(E + 7) & 7>(k - 1, __dmul_rn(x[E], prev1));
        if (k >= 2) l2.push<(E + 6) & 7>(k - 2, __dmul_rn(x[E], prev2));
    }
    if constexpr (E + 1 < 8) ma2_leaf_products<E + 1>(l1, l2, x, xm1, xm2, mid, k0, cnt);
}

// ---- MA2 simulator (+ fused autocovariance) ---------------------------------------------------
// One thread per row; normals are generated eight at a time (4 Philox blocks).
// LEAF: both product rows fit one leaf of NumPy's pairwise sum (n_obs - 1 <= 128, e.g. the 99 / 98
// products of the benchmark model): eight running sums per lag (leafsum.cuh) instead of the general
// PairwiseStream tree with its per-level stack -- the kernel drops from 255 registers to well under
// half, i.e. more than two resident blocks per SM for a kernel whose Box-Muller chains need the
// latency hiding (0.79 ms for 1e6 x 100 at 8 warps per SM against ~0.3 ms of fp64-pipe time).
template <bool WRITE_X, bool SUMMARIES, bool LEAF>
__global__ void __launch_bounds__(128)
sim_ma2_kernel(const double* __restrict__ t1, const double* __restrict__ t2, int64_t B, int n_obs,
               uint64_t seed, uint64_t offset, double* __restrict__ X, int64_t ldX,
               double* __restrict__ S, int64_t ldS) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= B) return;
    const Philox ph(seed);
    const uint64_t row = offset + uint64_t(i);
    const uint32_t r0 = uint32_t(row), r1 = uint32_t(row >> 32);
    const double a1 = t1[i], a2 = t2[i];
    PairwiseStream<6> p1, p2;      // lag-1 and lag-2 product sums (rows up to 7688 terms)
    LeafSum l1, l2;                // the same sums when a row is a single leaf
    if (SUMMARIES) {
        if constexpr (LEAF) {
            l1.begin(n_obs - 1);
            l2.begin(n_obs - 2);
        } else {
            p1.begin(n_obs - 1);
            p2.begin(n_obs - 2);
        }
    }
    // w has n_obs + 2 entries; x_k = w_{k+2} + a1 w_{k+1} + a2 w_k
    double wm2, wm1;   // w_{k}, w_{k+1} before the current group
    {
        double n0, n1;
        normal2(ph(r0, r1, 0u, 0x4d413257u), n0, n1);
        wm2 = n0;
        wm1 = n1;
    }
    double xm1 = 0.0, xm2 = 0.0;   // x_{k-1}, x_{k-2}
    double b1[8], b2[8];
    for (int k0 = 0; k0 < n_obs; k0 += 8) {
        double w[8];
#pragma unroll
        for (int q = 0; q < 4; ++q)
            normal2(ph(r0, r1, uint32_t(1 + (k0 >> 1) + q), 0x4d413257u), w[2 * q], w[2 * q + 1]);
        double x[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const double wk = (e == 0) ? wm2 : (e == 1 ? wm1 : w[e >= 2 ? e - 2 : 0]);
            const double wk1 = (e == 0) ? wm1 : w[e >= 1 ? e - 1 : 0];
            // (w2 + t1*w1) + t2*w0 with separate roundings, like the NumPy expression in ma2.py:36
            x[e] = __dadd_rn(__dadd_rn(w[e], __dmul_rn(a1, wk1)), __dmul_rn(a2, wk));
        }
        wm2 = w[6];
        wm1 = w[7];
        const int cnt = (n_obs - k0) < 8 ? (n_obs - k0) : 8;
        if (WRITE_X) {
#pragma unroll
            for (int e = 0; e < 8; ++e)
                if (e < cnt) X[i * ldX + k0 + e] = x[e];
        }
        if constexpr (SUMMARIES && LEAF) {
            // product index k - 1 (lag 1) / k - 2 (lag 2) of element k = k0 + e goes straight into
            // its running sum; slot = index % 8 is static because k0 is a multiple of 8
            const bool mid = cnt == 8 && l1.all_mid(k0 - 1, k0 + 6) && l2.all_mid(k0 - 2, k0 + 5);
            ma2_leaf_products<0>(l1, l2, x, xm1, xm2, mid, k0, cnt);
        }
        if constexpr (SUMMARIES && !LEAF) {
            // lag-1 products p[j] = x[j+1] x[j], j = k - 1 for element k; lag-2: j = k - 2.
            // Feed aligned groups of 8 products: group g of lag 1 needs x[8g .. 8g+8].
            // b1[] holds products with indices 8(g) .. 8g+7 once x[8g+8] is known, so products are
            // emitted one group late: element k contributes product index k-1 (lag 1), k-2 (lag 2).
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int k = k0 + e;
                if (e < cnt) {
                    const double prev1 = (e == 0) ? xm1 : x[e >= 1 ? e - 1 : 0];
                    const double prev2 = (e == 0) ? xm2 : (e == 1 ? xm1 : x[e >= 2 ? e - 2 : 0]);
                    // product index for lag 1 is k-1: slot (k-1) & 7 == (e + 7) & 7
                    if (k >= 1) {
                        b1[(e + 7) & 7] = __dmul_rn(x[e], prev1);
                        if (((e + 7) & 7) == 7) p1.feed8(k - 8, b1, 8);
                    }
                    if (k >= 2) {
                        b2[(e + 6) & 7] = __dmul_rn(x[e], prev2);
                        if (((e + 6) & 7) == 7) p2.feed8(k - 9, b2, 8);
                    }
                }
            }
        }
        xm2 = x[6];
        xm1 = x[7];
    }
    if constexpr (SUMMARIES && LEAF) {
        S[i * ldS + 0] = l1.finish(n_obs - 1) / double(n_obs - 1);
        S[i * ldS + 1] = l2.finish(n_obs - 2) / double(n_obs - 2);
    }
    if constexpr (SUMMARIES && !LEAF) {
        const int m1 = n_obs - 1, m2 = n_obs - 2;
        if (m1 % 8) p1.feed8(m1 - m1 % 8, b1, m1 % 8);
        if (m2 % 8) p2.feed8(m2 - m2 % 8, b2, m2 % 8);
        S[i * ldS + 0] = p1.finish() / double(m1);
        S[i * ldS + 1] = p2.finish() / double(m2);
    }
}

// ---- Gaussian-mixture proposals ------------------------------------------------------------------
// cumw: inclusive cumulative sum of the normalised weights (N); Lc: lower Cholesky factor of the
// shared covariance (p x p, row-major, p <= 4).  support: 0 none, 1 MA2 prior support.
struct BoxSupport { double lo[4], hi[4]; };
struct LowerFactor4 { double v[16]; };   // row-major p x p (p <= 4), passed by value

__global__ void gm_rvs_kernel(const double* __restrict__ means, int64_t ldm, const double* __restrict__ cumw,
                              int64_t N, int p, const LowerFactor4 Lc, int64_t B,
                              uint64_t seed, uint64_t offset, int support, BoxSupport box,
                              double* __restrict__ out, int64_t ldo) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= B) return;
    const Philox ph(seed);
    const uint64_t row = offset + uint64_t(i);
    const double total = cumw[N - 1];
    double x[4];
    for (uint32_t trial = 0; trial < 1000u; ++trial) {
        const uint4 r = ph(uint32_t(row), uint32_t(row >> 32), trial * 4u, 0x474d5256u);
        const double u = u01(r.x, r.y) * total;
        int64_t lo = 0, hi = N - 1;               // first index with cumw >= u
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (cumw[mid] < u) lo = mid + 1; else hi = mid;
        }
        double z[4];
        normal2(ph(uint32_t(row), uint32_t(row >> 32), trial * 4u + 1u, 0x474d5256u), z[0], z[1]);
        if (p > 2) normal2(ph(uint32_t(row), uint32_t(row >> 32), trial * 4u + 2u, 0x474d5256u), z[2], z[3]);
        for (int a = 0; a < p; ++a) {
            double s = means[lo * ldm + a];
            for (int b = 0; b <= a; ++b) s = fma(Lc.v[a * p + b], z[b], s);
            x[a] = s;
        }
        bool ok = support == 0 || (support == 1 && ma2_in_support(x[0], x[1]));
        if (support == 2) {
            ok = true;
            for (int a = 0; a < p; ++a) ok = ok && x[a] >= box.lo[a] && x[a] <= box.hi[a];
        }
        if (ok) break;
    }
    for (int a = 0; a < p; ++a) out[i * ldo + a] = x[a];
}

// ---- Gaussian noise model (elfi/examples/gauss.py) --------------------------------------------------
// priors of get_model(): mu ~ U(mu_lo, mu_lo + mu_w); sigma ~ truncnorm(a, b) (standard normal
// truncated to [a, b], scipy convention with loc 0, scale 1).
struct GaussPrior { double mu_lo, mu_w, a, b, cdf_a, cdf_w; };

__global__ void prior_gauss_kernel(int64_t B, uint64_t seed, uint64_t offset, GaussPrior g,
                                   double* __restrict__ mu, double* __restrict__ sigma) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= B) return;
    const Philox ph(seed);
    const uint64_t row = offset + uint64_t(i);
    const uint4 r = ph(uint32_t(row), uint32_t(row >> 32), 0u, 0x47415553u);
    const double u = u01(r.x, r.y), v = u01(r.z, r.w);
    mu[i] = g.mu_lo + g.mu_w * u;
    double sgm = normcdfinv(g.cdf_a + v * g.cdf_w);     // inverse-CDF sampling of the truncation
    sigma[i] = fmin(fmax(sgm, g.a), g.b);
}

__global__ void logprior_gauss_kernel(const double* __restrict__ x, int64_t ld, int64_t B, GaussPrior g,
                                      double* __restrict__ out) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= B) return;
    const double m = x[i * ld], s = x[i * ld + 1];
    double lp = -INFINITY;
    if (m >= g.mu_lo && m <= g.mu_lo + g.mu_w && s >= g.a && s <= g.b)
        lp = -log(g.mu_w) - 0.5 * s * s - 0.9189385332046727 - log(g.cdf_w);
    out[i] = lp;
}

// y_ij = mu_i + sigma_i z_ij (gauss.py:11-35) with np.mean / np.var summaries (gauss.py:142-173,
// NumPy pairwise order).  The variance needs the mean first: the counter-based normals are simply
// generated a second time instead of being stored.
// Terms k0 + E .. k0 + 7 of a group of eight into a single-leaf sum (static slots).
template <int E>
__device__ __forceinline__ void leaf_feed8(LeafSum& s, int k0, const double (&t)[8], int cnt,
                                           bool mid) {
    if (mid) s.push_mid<E>(t[E]);
    else if (E < cnt) s.push<E>(k0 + E, t[E]);
    if constexpr (E + 1 < 8) leaf_feed8<E + 1>(s, k0, t, cnt, mid);
}

// LEAF: n_obs <= 128, the row sums are single leaves of NumPy's pairwise sum (fewer registers, more
// resident blocks; keeping the draws in registers to generate them only once was tried and is
// slower -- 180 registers, two blocks per SM: the Box-Muller chains need the occupancy more than
// they need the halved work: 0.715 against 0.562 ms for 1e6 x 50).
template <bool WRITE_Y, bool LEAF>
__global__ void __launch_bounds__(128)
sim_gauss_kernel(const double* __restrict__ mu, const double* __restrict__ sigma, int64_t B, int n_obs,
                 uint64_t seed, uint64_t offset, double* __restrict__ Y, int64_t ldY,
                 double* __restrict__ S, int64_t ldS) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= B) return;
    const Philox ph(seed);
    const uint64_t row = offset + uint64_t(i);
    const uint32_t r0 = uint32_t(row), r1 = uint32_t(row >> 32);
    const double m = mu[i], sg = sigma[i];
    PairwiseStream<6> pw;
    LeafSum lf;
    double mean = 0.0;
    for (int pass = 0; pass < (S ? 2 : 1); ++pass) {
        if (S) {
            if constexpr (LEAF) lf.begin(n_obs); else pw.begin(n_obs);
        }
        double t[8];
        for (int k0 = 0; k0 < n_obs; k0 += 8) {
            double y[8];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                double z0, z1;
                normal2(ph(r0, r1, uint32_t((k0 >> 1) + q), 0x47534d55u), z0, z1);
                y[2 * q] = __dadd_rn(m, __dmul_rn(sg, z0));
                y[2 * q + 1] = __dadd_rn(m, __dmul_rn(sg, z1));
            }
            const int cnt = (n_obs - k0) < 8 ? (n_obs - k0) : 8;
            if (WRITE_Y && pass == 0) {
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    if (e < cnt) Y[i * ldY + k0 + e] = y[e];
            }
            if (S) {
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    if (pass == 0) {
                        t[e] = y[e];
                    } else {
                        const double c = __dsub_rn(y[e], mean);
                        t[e] = __dmul_rn(c, c);
                    }
                }
                if constexpr (LEAF)
                    leaf_feed8<0>(lf, k0, t, cnt, cnt == 8 && lf.all_mid(k0, k0 + 7));
                else
                    pw.feed8(k0, t, cnt);
            }
        }
        if (S) {
            const double v = (LEAF ? lf.finish(n_obs) : pw.finish()) / double(n_obs);
            if (pass == 0) { mean = v; S[i * ldS] = v; } else { S[i * ldS + 1] = v; }
        }
    }
}

// ---- g-and-k model (elfi/examples/gnk.py) -------------------------------------------------------
// y_ij = Q(z_ij; A_i, B_i, g_i, k_i, c) with the quantile function of gnkmath.cuh (gnk.py:60-66).
// One thread per pair of observations: Philox block (row, pair) -> two normals -> two adjacent
// outputs, so a warp writes 512 contiguous bytes of a row.  The draws of a row do not depend on
// n_obs or on how rows are sharded.
__global__ void __launch_bounds__(256)
sim_gnk_kernel(const double* __restrict__ A, const double* __restrict__ Bs, const double* __restrict__ g,
               const double* __restrict__ k, double c, int64_t B, int n_obs, uint64_t seed,
               uint64_t offset, double* __restrict__ Y, int64_t ldY) {
    const int half = (n_obs + 1) >> 1;
    const int64_t total = B * half;
    const Philox ph(seed);
    const bool vec = (ldY & 1) == 0 && (reinterpret_cast<uintptr_t>(Y) & 15) == 0;
    for (int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
         idx += int64_t(gridDim.x) * blockDim.x) {
        const int64_t i = idx / half;
        const int q = int(idx - i * half);
        const uint64_t row = offset + uint64_t(i);
        double z0, z1;
        normal2(ph(uint32_t(row), uint32_t(row >> 32), uint32_t(q), 0x474e4b30u), z0, z1);
        const double a = A[i], b = Bs[i], gg = g[i], kk = k[i];
        const double y0 = gnk_quantile(a, b, gg, kk, c, z0);
        double* dst = Y + i * ldY + 2 * q;
        if (2 * q + 1 < n_obs) {
            const double y1 = gnk_quantile(a, b, gg, kk, c, z1);
            if (vec) {
                *reinterpret_cast<double2*>(dst) = make_double2(y0, y1);
            } else {
                dst[0] = y0;
                dst[1] = y1;
            }
        } else {
            dst[0] = y0;
        }
    }
}

// log density of independent uniform priors U(lo_a, lo_a + width_a), a < p <= 8
// (gnk.py:99-103: A, B, g, k ~ uniform(0, 10)); -inf outside the box like scipy's logpdf.
struct BoxPrior { double lo[8], hi[8]; double logdens; };

__global__ void logprior_box_kernel(const double* __restrict__ x, int64_t ld, int64_t B, int p,
                                    BoxPrior box, double* __restrict__ out) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= B) return;
    bool inside = true;
    for (int a = 0; a < p; ++a) {
        const double v = x[i * ld + a];
        inside = inside && v >= box.lo[a] && v <= box.hi[a];   // NaN -> outside
    }
    out[i] = inside ? box.logdens : -INFINITY;
}

// inclusive scan of w / sum(w) (single block; N up to a few million is fine: one pass each)
__global__ void __launch_bounds__(1024)
cumsum_kernel(const double* __restrict__ w, int64_t n, double* __restrict__ out) {
    __shared__ double ws[32];
    __shared__ double carry_s;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) carry_s = 0.0;
    __syncthreads();
    for (int64_t base = 0; base < n; base += 1024) {
        const int64_t i = base + tid;
        const double v = i < n ? (w ? w[i] : 1.0) : 0.0;
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
        if (i < n) out[i] = carry + woff + incl;
        __syncthreads();
        if (tid == 1023) carry_s = carry + woff + incl;
        __syncthreads();
    }
}

}  // namespace elfi

extern "C" {

int elfi_b200_prior_ma2_f64(elfi_b200_ctx* ctx, int64_t B, uint64_t seed, uint64_t offset,
                            int32_t mode, double* t1, double* t2, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && mode >= 0 && mode <= 2, "prior_ma2: bad argument");
    ELFI_REQUIRE(B == 0 || (t1 && (mode == 1 || t2)), "prior_ma2: NULL argument");
    if (B == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    prior_ma2_kernel<<<unsigned((B + 255) / 256), 256, 0, stream>>>(B, seed, offset, mode, t1, t2);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_logprior_ma2_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, int64_t B,
                               double* out, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && (B == 0 || (x && out)) && ldx >= 2, "logprior_ma2: bad argument");
    if (B == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    logprior_ma2_kernel<<<unsigned((B + 255) / 256), 256, 0, stream>>>(x, ldx, B, out);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_sim_ma2_f64(elfi_b200_ctx* ctx, const double* t1, const double* t2, int64_t B,
                          int64_t n_obs, uint64_t seed, uint64_t offset, double* X, int64_t ldX,
                          double* S, int64_t ldS, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && (B == 0 || (t1 && t2)), "sim_ma2: NULL argument");
    ELFI_REQUIRE(n_obs >= 3 && n_obs <= PairwiseStream<6>::max_terms(),
                 "sim_ma2: n_obs=%lld outside [3, 7688]", (long long)n_obs);
    ELFI_REQUIRE(X || S, "sim_ma2: nothing to produce (X and S are both NULL)");
    ELFI_REQUIRE((!X || ldX >= n_obs) && (!S || ldS >= 2), "sim_ma2: bad leading dimension");
    if (B == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    const unsigned blocks = unsigned((B + 127) / 128);
    const bool leaf = n_obs - 1 <= LEAF_MAX_TERMS;
#define ELFI_SIM_MA2(WX, SM, LF) \
    sim_ma2_kernel<WX, SM, LF><<<blocks, 128, 0, stream>>>(t1, t2, B, int(n_obs), seed, offset, X, ldX, S, ldS)
    if (X && S) { if (leaf) ELFI_SIM_MA2(true, true, true); else ELFI_SIM_MA2(true, true, false); }
    else if (X) ELFI_SIM_MA2(true, false, false);
    else { if (leaf) ELFI_SIM_MA2(false, true, true); else ELFI_SIM_MA2(false, true, false); }
#undef ELFI_SIM_MA2
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_gm_cdf_f64(elfi_b200_ctx* ctx, const double* weights, int64_t N, double* cumw,
                         void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && cumw && N >= 1, "gm_cdf: bad argument");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    cumsum_kernel<<<1, 1024, 0, stream>>>(weights, N, cumw);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_gm_rvs_cdf_f64(elfi_b200_ctx* ctx, const double* means, int64_t ldm, const double* cumw,
                             int64_t N, int64_t p, const double* Lchol_host, int64_t B, uint64_t seed,
                             uint64_t offset, int32_t support, const double* box_host, double* out,
                             int64_t ldo, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && means && cumw && Lchol_host && (B == 0 || out), "gm_rvs: NULL argument");
    ELFI_REQUIRE(N >= 1 && p >= 1 && p <= 4 && ldm >= p && ldo >= p, "gm_rvs: bad shape (p <= 4)");
    ELFI_REQUIRE(support == 0 || (support == 1 && p == 2) || (support == 2 && box_host),
                 "gm_rvs: unknown support %d", support);
    BoxSupport box;
    memset(&box, 0, sizeof(box));
    if (support == 2)
        for (int a = 0; a < p; ++a) { box.lo[a] = box_host[a]; box.hi[a] = box_host[p + a]; }
    if (B == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    LowerFactor4 Lc;
    memset(&Lc, 0, sizeof(Lc));
    for (int a = 0; a < p; ++a)
        for (int b = 0; b <= a; ++b) Lc.v[a * p + b] = Lchol_host[a * p + b];
    gm_rvs_kernel<<<unsigned((B + 127) / 128), 128, 0, stream>>>(means, ldm, cumw, N, int(p), Lc, B,
                                                                seed, offset, support, box, out, ldo);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_gm_rvs_f64(elfi_b200_ctx* ctx, const double* means, int64_t ldm, const double* weights,
                         int64_t N, int64_t p, const double* Lchol_host, int64_t B, uint64_t seed,
                         uint64_t offset, int32_t support, const double* box_host, double* out,
                         int64_t ldo, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && N >= 1, "gm_rvs: bad argument");
    if (B == 0) return ELFI_B200_OK;
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    double* cumw = static_cast<double*>(ctx_scratch(ctx, size_t(N) * 8 + 256));
    if (!cumw) return ELFI_B200_ERR_NOMEM;
    int rc = elfi_b200_gm_cdf_f64(ctx, weights, N, cumw, stream_);
    if (rc != ELFI_B200_OK) return rc;
    return elfi_b200_gm_rvs_cdf_f64(ctx, means, ldm, cumw, N, p, Lchol_host, B, seed, offset, support,
                                    box_host, out, ldo, stream_);
}

static elfi::GaussPrior make_gauss_prior(const double* prm) {
    elfi::GaussPrior g;
    g.mu_lo = prm[0]; g.mu_w = prm[1]; g.a = prm[2]; g.b = prm[3];
    g.cdf_a = 0.5 * erfc(-g.a * 0.7071067811865476);
    g.cdf_w = 0.5 * erfc(-g.b * 0.7071067811865476) - g.cdf_a;
    return g;
}

/* prm_host = [mu_lo, mu_width, a, b] of mu ~ U(mu_lo, mu_lo + mu_width), sigma ~ truncnorm(a, b) */
int elfi_b200_prior_gauss_f64(elfi_b200_ctx* ctx, int64_t B, uint64_t seed, uint64_t offset,
                              const double* prm_host, double* mu, double* sigma, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && prm_host && (B == 0 || (mu && sigma)), "prior_gauss: NULL argument");
    ELFI_REQUIRE(prm_host[1] > 0 && prm_host[3] > prm_host[2], "prior_gauss: bad prior parameters");
    if (B == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    prior_gauss_kernel<<<unsigned((B + 255) / 256), 256, 0, stream>>>(B, seed, offset,
                                                                     make_gauss_prior(prm_host), mu, sigma);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_logprior_gauss_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, int64_t B,
                                 const double* prm_host, double* out, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && prm_host && (B == 0 || (x && out)) && ldx >= 2, "logprior_gauss: bad argument");
    if (B == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    logprior_gauss_kernel<<<unsigned((B + 255) / 256), 256, 0, stream>>>(x, ldx, B,
                                                                        make_gauss_prior(prm_host), out);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_sim_gauss_f64(elfi_b200_ctx* ctx, const double* mu, const double* sigma, int64_t B,
                            int64_t n_obs, uint64_t seed, uint64_t offset, double* Y, int64_t ldY,
                            double* S, int64_t ldS, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && (B == 0 || (mu && sigma)), "sim_gauss: NULL argument");
    ELFI_REQUIRE(n_obs >= 1 && n_obs <= PairwiseStream<6>::max_terms(),
                 "sim_gauss: n_obs=%lld outside [1, 7688]", (long long)n_obs);
    ELFI_REQUIRE(Y || S, "sim_gauss: nothing to produce (Y and S are both NULL)");
    ELFI_REQUIRE((!Y || ldY >= n_obs) && (!S || ldS >= 2), "sim_gauss: bad leading dimension");
    if (B == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    const unsigned blocks = unsigned((B + 127) / 128);
    const bool leaf = n_obs <= LEAF_MAX_TERMS;
#define ELFI_SIM_GAUSS(WY, LF) \
    sim_gauss_kernel<WY, LF><<<blocks, 128, 0, stream>>>(mu, sigma, B, int(n_obs), seed, offset, Y, ldY, S, ldS)
    if (Y) { if (leaf) ELFI_SIM_GAUSS(true, true); else ELFI_SIM_GAUSS(true, false); }
    else { if (leaf) ELFI_SIM_GAUSS(false, true); else ELFI_SIM_GAUSS(false, false); }
#undef ELFI_SIM_GAUSS
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_sim_gnk_f64(elfi_b200_ctx* ctx, const double* A, const double* Bs, const double* g,
                          const double* k, double c, int64_t B, int64_t n_obs, uint64_t seed,
                          uint64_t offset, double* Y, int64_t ldY, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && (B == 0 || (A && Bs && g && k && Y)), "sim_gnk: NULL argument");
    ELFI_REQUIRE(B >= 0 && n_obs >= 1 && n_obs < (int64_t(1) << 30), "sim_gnk: bad shape B=%lld n_obs=%lld",
                 (long long)B, (long long)n_obs);
    ELFI_REQUIRE(ldY >= n_obs, "sim_gnk: bad leading dimension");
    if (B == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    const int64_t total = B * ((n_obs + 1) / 2);
    int64_t blocks = (total + 255) / 256;
    const int64_t cap = int64_t(ctx->sm_count) * 64;   // grid-stride beyond 8 waves of 8 CTAs/SM
    if (blocks > cap) blocks = cap;
    sim_gnk_kernel<<<unsigned(blocks), 256, 0, stream>>>(A, Bs, g, k, c, B, int(n_obs), seed, offset, Y, ldY);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

int elfi_b200_logprior_box_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, int64_t B, int64_t p,
                               const double* box_host, double* out, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && box_host && (B == 0 || (x && out)), "logprior_box: NULL argument");
    ELFI_REQUIRE(B >= 0 && p >= 1 && p <= 8 && ldx >= p, "logprior_box: bad shape (p <= 8)");
    BoxPrior box;
    memset(&box, 0, sizeof(box));
    box.logdens = 0.0;
    for (int a = 0; a < p; ++a) {
        ELFI_REQUIRE(box_host[p + a] > 0.0, "logprior_box: width[%d] must be positive", a);
        box.lo[a] = box_host[a];
        box.hi[a] = box_host[a] + box_host[p + a];
        box.logdens -= log(box_host[p + a]);
    }
    if (B == 0) return ELFI_B200_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    logprior_box_kernel<<<unsigned((B + 255) / 256), 256, 0, stream>>>(x, ldx, B, int(p), box, out);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

}  // extern "C"
