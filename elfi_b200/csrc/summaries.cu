// summaries.cu -- row-wise summary statistics with NumPy's pairwise summation order
// (SURVEY.md K6): MA2 autocovariance (elfi/examples/ma2.py:40-59) and the Gaussian model's
// mean / variance (elfi/examples/gauss.py:142-173).
//
// NumPy reduces each row with DOUBLE_pairwise_sum: blocks of <= 128 elements are summed with
// 8 strided accumulators r[0..7] combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) plus a
// sequential tail; longer rows are split recursively at n/2 rounded down to a multiple of 8.
// Every left part is a multiple of 8 long, so every leaf starts at an index that is a multiple
// of 8 and only the last leaf has a tail.  The row-stream consumers below reproduce that tree bit
// for bit with the accumulators of leafsum.cuh / treesum.cuh, indexed by compile-time constants
// (the term index modulo 8 is fixed by the column position and the lag); the generic fallback
// feeds the same tree through PairwiseStream (pairwise.cuh).
//
// Traffic: n*8 bytes read per row (variance re-reads the tile from L2), 8 bytes written per
// statistic.  Roofline: HBM.
#include "leafsum.cuh"
#include "pairwise.cuh"
#include "rowstream.cuh"
#include "treesum.cuh"

namespace elfi {

constexpr int RS_PW_DEPTH = 6;   // rows of up to 7688 terms on the row-stream path (max_terms())

struct SummaryParams {
    double* out;      // out[row * ld_out + col0 (+1)]
    int64_t ld_out;
    int n;            // row length
    int col_a;        // output column of the first statistic
    int col_b;        // output column of the second statistic (or -1)
};

__device__ __forceinline__ void load_box_row(const uint8_t* box_row, int sw, double* cur) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const double2 v = *reinterpret_cast<const double2*>(box_row + ((c ^ sw) << 4));
        cur[2 * c] = v.x;
        cur[2 * c + 1] = v.y;
    }
}

// Term-wise consumers: the per-lane state is one of the accumulators of leafsum.cuh / treesum.cuh
// and the box logic is AutocovBoxes / MeanVarBoxes, which also compile for the host.
//   Sum = LeafSum   every reduced run has <= 128 terms, so NumPy's tree is one leaf and the state
//                   is 8 accumulators per sum (profiles/r1_summ_instruction_mix.md).
//   Sum = TreeSum   rows of 129..7688 terms, same front end.
template <class Sum, int LAG_A, int LAG_B>
struct AutocovBoxConsumer {
    typedef SummaryParams Params;
    static constexpr int PASSES = 1;
    const Params& p;
    AutocovBoxes<Sum, LAG_A, LAG_B> st;

    static __device__ void setup_shared(uint8_t*, const Params&, int) {}
    __device__ AutocovBoxConsumer(const Params& p_, const uint8_t*, int, int) : p(p_) {}
    __device__ __forceinline__ void begin_row() { st.begin(p.n); }
    __device__ __forceinline__ void consume(int, int cg, const uint8_t* box_row, int sw) {
        double cur[16];
        load_box_row(box_row, sw, cur);
        st.box(cg * RS_BOX_COLS, cur);
    }
    __device__ __forceinline__ void end_row(int64_t row, int64_t B, int) {
        if (row < B) {
            p.out[row * p.ld_out + p.col_a] = st.sum_a() / double(p.n - LAG_A);
            if constexpr (LAG_B >= 0)
                p.out[row * p.ld_out + p.col_b] = st.sum_b() / double(p.n - LAG_B);
        }
    }
};

template <class Sum>
struct MeanVarBoxConsumer {
    typedef SummaryParams Params;
    static constexpr int PASSES = 2;
    const Params& p;
    MeanVarBoxes<Sum> st;

    static __device__ void setup_shared(uint8_t*, const Params&, int) {}
    __device__ MeanVarBoxConsumer(const Params& p_, const uint8_t*, int, int) : p(p_) {}
    __device__ __forceinline__ void begin_row() { st.begin(p.n); }
    __device__ __forceinline__ void consume(int pass, int cg, const uint8_t* box_row, int sw) {
        double cur[16];
        load_box_row(box_row, sw, cur);
        st.box(pass, cg * RS_BOX_COLS, cur);
    }
    __device__ __forceinline__ void end_row(int64_t row, int64_t B, int) {
        const double var = st.variance();
        if (row < B) {
            if (p.col_a >= 0) p.out[row * p.ld_out + p.col_a] = st.mean;
            if (p.col_b >= 0) p.out[row * p.ld_out + p.col_b] = var;
        }
    }
};

// Rows of <= 64 observations: one sweep, the row stays in registers (MeanVarRegs, leafsum.cuh).
// The box index selects the register block through a switch so that every index is a constant.
template <int NBOX>
struct MeanVarRegsConsumer {
    typedef SummaryParams Params;
    static constexpr int PASSES = 1;
    const Params& p;
    MeanVarRegs<NBOX> st;

    static __device__ void setup_shared(uint8_t*, const Params&, int) {}
    __device__ MeanVarRegsConsumer(const Params& p_, const uint8_t*, int, int) : p(p_) {}
    __device__ __forceinline__ void begin_row() { st.begin(p.n); }
    __device__ __forceinline__ void consume(int, int cg, const uint8_t* box_row, int sw) {
        double cur[16];
        load_box_row(box_row, sw, cur);
        switch (cg) {
            case 0: st.template box<0>(cur); break;
            case 1: if constexpr (NBOX > 1) st.template box<1>(cur); break;
            case 2: if constexpr (NBOX > 2) st.template box<2>(cur); break;
            default: if constexpr (NBOX > 3) st.template box<3>(cur); break;
        }
    }
    __device__ __forceinline__ void end_row(int64_t row, int64_t B, int) {
        double mean, var;
        st.finish(mean, var);
        if (row < B) {
            if (p.col_a >= 0) p.out[row * p.ld_out + p.col_a] = mean;
            if (p.col_b >= 0) p.out[row * p.ld_out + p.col_b] = var;
        }
    }
};

// Contiguous rows whose pitch is an odd multiple of 16 bytes (n = 2 mod 4; the Gaussian model
// has n = 50: 400-byte rows).  Through the 2-D tensor map such a matrix costs ceil(n/16) boxes
// per 32 rows, the last one nearly empty (n = 50: 4 boxes for 3.125 boxes of data -- the
// kernel ran at 0.6 of the HBM peak against 0.8 at n = 64), and no box row is line aligned.
// Here a tile is what it is in memory: 32 rows = ONE contiguous run of 32 * 8n bytes, fetched
// by one 1-D bulk copy into the warp's ring slot.  No swizzle is needed: lane l reads 16-byte
// chunk c of its row at l * 8n + 16c, and with 8n / 16 odd the eight lanes of a quarter-warp
// fall into eight distinct 16-byte bank groups (LDS.128 without conflicts).  Arithmetic and
// order are MeanVarRegs', i.e. the same bits as the row-stream consumers.
constexpr int RG_WARPS = 8;         // 6 for the widest rows (two ring slots of 8 warps would not fit)
constexpr int RG_SLACK = 256;   // the last box of lane 31 reads up to (16*NBOX - n) doubles past its row

__host__ __device__ inline size_t rg_slot_bytes(int n) { return size_t(32) * n * 8; }

template <int NBOX, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, 1)
meanvar_rowgroup_kernel(const double* __restrict__ X, int64_t B, int ns, SummaryParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int n = p.n;
    const uint32_t slot = uint32_t(rg_slot_bytes(n));
    uint8_t* bars_generic = smem + size_t(WARPS) * ns * slot + RG_SLACK;
    const uint32_t box0 = smem_u32(smem) + uint32_t(warp) * ns * slot;
    const uint32_t bar0 = smem_u32(bars_generic) + uint32_t(warp) * ns * 8;
    const uint8_t* box0_generic = smem + size_t(warp) * ns * slot;
    if (lane == 0) {
        for (int s = 0; s < ns; ++s) mbar_init(bar0 + s * 8, 1);
        mbar_fence_init();
    }
    __syncwarp();

    const int64_t ntiles = (B + 31) / 32;
    const int64_t gw = int64_t(blockIdx.x) * WARPS + warp;
    const int64_t GW = int64_t(gridDim.x) * WARPS;
    const int64_t my_tiles = gw < ntiles ? (ntiles - gw + GW - 1) / GW : 0;

    int64_t p_tile = gw;   // producer cursor (lane 0)
    int64_t p_q = 0;
    int p_s = 0;
    auto issue = [&]() {
        const int64_t row0 = p_tile * 32;
        const int64_t rows = (B - row0 < 32) ? (B - row0) : 32;
        const uint32_t bytes = uint32_t(rows) * uint32_t(n) * 8u;
        mbar_arrive_expect_tx(bar0 + p_s * 8, bytes);
        bulk_load_1d(box0 + p_s * slot, X + row0 * n, bytes, bar0 + p_s * 8);
        ++p_q;
        p_tile += GW;
        if (++p_s == ns) p_s = 0;
    };
    if (lane == 0) {
        const int64_t pre = my_tiles < ns ? my_tiles : ns;
        for (int64_t i = 0; i < pre; ++i) issue();
    }

    MeanVarRegs<NBOX> st;
    const uint32_t row_off = uint32_t(lane) * uint32_t(n) * 8u;
    int s = 0;
    uint32_t parity = 0;
    int64_t tile = gw;
    for (int64_t q = 0; q < my_tiles; ++q) {
        mbar_wait(bar0 + s * 8, parity);
        const double2* row = reinterpret_cast<const double2*>(box0_generic + size_t(s) * slot + row_off);
        st.begin(n);
        double cur[16];
#pragma unroll
        for (int g = 0; g < NBOX; ++g) {
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const double2 v = row[g * 8 + c];
                cur[2 * c] = v.x;
                cur[2 * c + 1] = v.y;
            }
            if (g == 0) st.template box<0>(cur);
            if constexpr (NBOX > 1) if (g == 1) st.template box<1>(cur);
            if constexpr (NBOX > 2) if (g == 2) st.template box<2>(cur);
            if constexpr (NBOX > 3) if (g == 3) st.template box<3>(cur);
        }
        __syncwarp();
        if (lane == 0 && p_q < my_tiles) issue();
        double mean, var;
        st.finish(mean, var);
        const int64_t r = tile * 32 + lane;
        if (r < B) {
            if (p.col_a >= 0) p.out[r * p.ld_out + p.col_a] = mean;
            if (p.col_b >= 0) p.out[r * p.ld_out + p.col_b] = var;
        }
        tile += GW;
        if (++s == ns) { s = 0; parity ^= 1; }
    }
}

static size_t rg_smem_bytes(int warps, int ns, int64_t n) {
    return size_t(warps) * ns * rg_slot_bytes(int(n)) + RG_SLACK + size_t(warps) * ns * 8;
}

static bool rowgroup_ok(elfi_b200_ctx* ctx, const double* X, int64_t ld, int64_t n) {
    if (ld != n || n > 64 || (n & 3) != 2 || (reinterpret_cast<uintptr_t>(X) & 15)) return false;
    return rg_smem_bytes(6, 2, n) + 1024 <= ctx->smem_optin;
}

template <int NBOX, int WARPS>
static int rowgroup_launch_w(elfi_b200_ctx* ctx, const double* X, int64_t B, int64_t n,
                             const SummaryParams& p, cudaStream_t stream) {
    int ns = 4;
    while (rg_smem_bytes(WARPS, ns, n) + 1024 > ctx->smem_optin) --ns;
    const size_t smem_bytes = rg_smem_bytes(WARPS, ns, n);
    auto kern = meanvar_rowgroup_kernel<NBOX, WARPS>;
    ELFI_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      int(smem_bytes)));
    const int64_t ntiles = (B + 31) / 32;
    int64_t ctas = (ntiles + WARPS - 1) / WARPS;
    if (ctas > ctx->sm_count) ctas = ctx->sm_count;
    kern<<<dim3(unsigned(ctas)), dim3(WARPS * 32), smem_bytes, stream>>>(X, B, ns, p);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

template <int NBOX>
static int rowgroup_launch(elfi_b200_ctx* ctx, const double* X, int64_t B, int64_t n,
                           const SummaryParams& p, cudaStream_t stream) {
    if (rg_smem_bytes(RG_WARPS, 2, n) + 1024 <= ctx->smem_optin)
        return rowgroup_launch_w<NBOX, RG_WARPS>(ctx, X, B, n, p, stream);
    return rowgroup_launch_w<NBOX, 6>(ctx, X, B, n, p, stream);
}

typedef TreeSum<RS_PW_DEPTH> RowTreeSum;

// Rows of 129..7688 terms take the term-wise TreeSum front end (autocov(1,2) 4e5 x 256: 0.152 ms =
// 0.83 of the HBM peak against 0.225 ms = 0.56 for the round-1 group-of-8 consumers; mean/var
// 0.183 against 0.350 ms; profiles/r2_kernels.md).

// Generic fallback (any lag, any alignment): one thread per row straight from global memory,
// same tree through PairwiseStream so results are identical.  mode 0 = autocov(lag), 1 = mean+var.
__global__ void __launch_bounds__(128)
summary_direct_kernel(const double* __restrict__ X, int64_t ld, int64_t B, int n, int lag,
                      int mode, SummaryParams p) {
    const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (row >= B) return;
    const double* x = X + row * ld;
    PairwiseStream<24> pw;
    double buf[8];
    auto run = [&](int m, auto term) -> double {
        pw.begin(m);
        for (int j0 = 0; j0 < m; j0 += 8) {
            const int cnt = (m - j0) < 8 ? (m - j0) : 8;
#pragma unroll
            for (int k = 0; k < 8; ++k) buf[k] = k < cnt ? term(j0 + k) : 0.0;
            pw.feed8(j0, buf, cnt);
        }
        return __dadd_rn(0.0, pw.finish());   // np.add.reduce starts from the identity 0.0
    };
    if (mode == 0) {
        const int m = n - lag;
        const double s = run(m, [&](int j) { return __dmul_rn(__ldg(x + j + lag), __ldg(x + j)); });
        p.out[row * p.ld_out + p.col_a] = s / double(m);
    } else {
        const double mean = run(n, [&](int j) { return __ldg(x + j); }) / double(n);
        const double ss = run(n, [&](int j) {
            const double c = __dsub_rn(__ldg(x + j), mean);
            return __dmul_rn(c, c);
        });
        if (p.col_a >= 0) p.out[row * p.ld_out + p.col_a] = mean;
        if (p.col_b >= 0) p.out[row * p.ld_out + p.col_b] = ss / double(n);
    }
}

static bool rowstream_ok(elfi_b200_ctx* ctx, const double* X, int64_t ld, int64_t n) {
    return n >= RS_BOX_COLS && n <= PairwiseStream<RS_PW_DEPTH>::max_terms() &&
           tma_compatible(X, ld) && rs_pick_stages(ctx->smem_optin, 0) >= 2;
}

// One row-stream launch for lag pair (LA, LB): single-leaf consumer when every run fits a leaf.
template <int LA, int LB>
static int autocov_launch(elfi_b200_ctx* ctx, const double* X, int64_t ld, int64_t B, int64_t n,
                          const SummaryParams& p, cudaStream_t stream) {
    if (n - LA <= LEAF_MAX_TERMS)   // LA is the smaller lag: the longer run
        return rowstream_launch<AutocovBoxConsumer<LeafSum, LA, LB>>(ctx, X, ld, B, n, 0, p, stream);
    return rowstream_launch<AutocovBoxConsumer<RowTreeSum, LA, LB>>(ctx, X, ld, B, n, 0, p, stream);
}

}  // namespace elfi

extern "C" {

int elfi_b200_summary_autocov_f64(elfi_b200_ctx* ctx, const double* X, int64_t ldX, int64_t B,
                                  int64_t n, const int32_t* lags_host, int64_t nlags, double* out,
                                  int64_t ld_out, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && (B == 0 || (X && out)), "autocov: NULL argument");
    ELFI_REQUIRE(B >= 0 && n >= 1 && ldX >= n, "autocov: bad shape B=%lld n=%lld ld=%lld",
                 (long long)B, (long long)n, (long long)ldX);
    ELFI_REQUIRE(nlags >= 1 && lags_host != nullptr && ld_out >= nlags, "autocov: bad lags/ld_out");
    ELFI_REQUIRE(n <= PairwiseStream<24>::max_terms(), "autocov: row too long");
    for (int64_t l = 0; l < nlags; ++l)
        ELFI_REQUIRE(lags_host[l] >= 1 && lags_host[l] < n, "autocov: lag %d outside [1, n)",
                     lags_host[l]);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    if (B == 0) return ELFI_B200_OK;
    SummaryParams p;
    p.out = out;
    p.ld_out = ld_out;
    p.n = int(n);
    const bool fast = rowstream_ok(ctx, X, ldX, n);
    int64_t l = 0;
    while (l < nlags) {
        p.col_a = int(l);
        p.col_b = -1;
        const int la = lags_host[l];
        const int lb = (l + 1 < nlags) ? lags_host[l + 1] : -1;
        int rc = -100;
        if (fast) {
            if (la == 1 && lb == 2) {
                p.col_b = int(l + 1);
                rc = autocov_launch<1, 2>(ctx, X, ldX, B, n, p, stream);
                if (rc == 0) l += 2;
            } else if (la == 1) {
                rc = autocov_launch<1, -1>(ctx, X, ldX, B, n, p, stream);
                if (rc == 0) l += 1;
            } else if (la == 2) {
                rc = autocov_launch<2, -1>(ctx, X, ldX, B, n, p, stream);
                if (rc == 0) l += 1;
            } else if (la == 3) {
                rc = autocov_launch<3, -1>(ctx, X, ldX, B, n, p, stream);
                if (rc == 0) l += 1;
            } else if (la == 4) {
                rc = autocov_launch<4, -1>(ctx, X, ldX, B, n, p, stream);
                if (rc == 0) l += 1;
            }
            if (rc != -100 && rc != 0) return rc;
        }
        if (rc == -100) {
            summary_direct_kernel<<<unsigned((B + 127) / 128), 128, 0, stream>>>(X, ldX, B, int(n),
                                                                                la, 0, p);
            ELFI_CUDA_OK(cudaGetLastError());
            l += 1;
        }
    }
    return ELFI_B200_OK;
}

int elfi_b200_summary_meanvar_f64(elfi_b200_ctx* ctx, const double* X, int64_t ldX, int64_t B,
                                  int64_t n, double* out, int64_t ld_out, int32_t col_mean,
                                  int32_t col_var, void* stream_) {
    using namespace elfi;
    ELFI_REQUIRE(ctx && (B == 0 || (X && out)), "meanvar: NULL argument");
    ELFI_REQUIRE(B >= 0 && n >= 1 && ldX >= n, "meanvar: bad shape B=%lld n=%lld ld=%lld",
                 (long long)B, (long long)n, (long long)ldX);
    ELFI_REQUIRE(col_mean < ld_out && col_var < ld_out && (col_mean >= 0 || col_var >= 0),
                 "meanvar: bad output columns");
    ELFI_REQUIRE(n <= PairwiseStream<24>::max_terms(), "meanvar: row too long");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    ELFI_CUDA_OK(cudaSetDevice(ctx->device));
    if (B == 0) return ELFI_B200_OK;
    SummaryParams p;
    p.out = out;
    p.ld_out = ld_out;
    p.n = int(n);
    p.col_a = col_mean;
    p.col_b = col_var;
    if (rowgroup_ok(ctx, X, ldX, n)) {
        if (n <= 16) return rowgroup_launch<1>(ctx, X, B, n, p, stream);
        if (n <= 32) return rowgroup_launch<2>(ctx, X, B, n, p, stream);
        if (n <= 48) return rowgroup_launch<3>(ctx, X, B, n, p, stream);
        return rowgroup_launch<4>(ctx, X, B, n, p, stream);
    }
    if (rowstream_ok(ctx, X, ldX, n)) {
        if (n <= 16) return rowstream_launch<MeanVarRegsConsumer<1>>(ctx, X, ldX, B, n, 0, p, stream);
        if (n <= 32) return rowstream_launch<MeanVarRegsConsumer<2>>(ctx, X, ldX, B, n, 0, p, stream);
        if (n <= 48) return rowstream_launch<MeanVarRegsConsumer<3>>(ctx, X, ldX, B, n, 0, p, stream);
        if (n <= 64) return rowstream_launch<MeanVarRegsConsumer<4>>(ctx, X, ldX, B, n, 0, p, stream);
        if (n <= LEAF_MAX_TERMS)
            return rowstream_launch<MeanVarBoxConsumer<LeafSum>>(ctx, X, ldX, B, n, 0, p, stream);
        return rowstream_launch<MeanVarBoxConsumer<RowTreeSum>>(ctx, X, ldX, B, n, 0, p, stream);
    }
    summary_direct_kernel<<<unsigned((B + 127) / 128), 128, 0, stream>>>(X, ldX, B, int(n), 0, 1, p);
    ELFI_CUDA_OK(cudaGetLastError());
    return ELFI_B200_OK;
}

}  // extern "C"
