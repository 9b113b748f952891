// K2 (exact-fp32 CUDA-core path): the stacked-K projection of the Chebyshev GCN, reference GCN.py:37-42.
//   forward : out = act( sum_k (T_k X) W_k + b )  -- reads T_0X..T_KX as K+1 A-segments (no torch.cat copy)
//   backward: dZ = dOut (.) [out>0];  db = sum dZ;  dW_k = (T_k X)^T dZ;  U_k = dZ W_k^T  (SURVEY.md 8(a))
#include "gemm_tall.cuh"

using namespace stmgcn;

namespace {

struct ProjEpi {
    const float* bias;       // (q) or nullptr
    int act;
    float* out;              // (rows, q)
    int half_cols;

    __device__ __forceinline__ void operator()(float (&acc)[8][8], int64_t row0, int mg, int MG, int col0,
                                               int tn, int64_t rows, int nc) const {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int64_t r = row0 + mg + (int64_t)i * MG;
            if (r >= rows) continue;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int n = col0 + (j < 4 ? 4 * tn + j : half_cols + 4 * tn + (j - 4));
                if (n >= nc) continue;
                float v = acc[i][j] + (bias ? bias[n] : 0.f);
                if (act == STMGCN_ACT_RELU) v = fmaxf(v, 0.f);
                out[r * nc + n] = v;
            }
        }
    }
};

// U_k[r, i] = acc column n = k*p + i
struct StoreSegEpi {
    float* u;
    int64_t stride_u;
    int p;
    int half_cols;

    __device__ __forceinline__ void operator()(float (&acc)[8][8], int64_t row0, int mg, int MG, int col0,
                                               int tn, int64_t rows, int nc) const {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int64_t r = row0 + mg + (int64_t)i * MG;
            if (r >= rows) continue;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int n = col0 + (j < 4 ? 4 * tn + j : half_cols + 4 * tn + (j - 4));
                if (n >= nc) continue;
                const int k = n / p;
                u[(int64_t)k * stride_u + r * p + (n - k * p)] = acc[i][j];
            }
        }
    }
};

// pool[(r % B) * q + j] += x[r, j] + g[r, j]: column sums of an (N x B*q) matrix.
// grid.x: column chunks of blockDim, grid.y: region chunks.
__global__ void pool_kernel(const float* __restrict__ x, const float* __restrict__ g, int64_t n_regions,
                            int64_t cols, float* __restrict__ pool) {
    const int64_t col = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= cols) return;
    float acc = 0.f;
    for (int64_t n = blockIdx.y; n < n_regions; n += gridDim.y) acc += x[n * cols + col] + g[n * cols + col];
    atomicAdd(&pool[col], acc);
}

// dZ = dOut (.) mask, plus column sums into dbias.  thread -> (row lane, column j): j fastest.
__global__ void __launch_bounds__(256)
dz_kernel(const float* __restrict__ out, const float* __restrict__ d_out, const float* __restrict__ d_bcast,
          float scale, int64_t b_inner, int64_t rows, int q, int act, float* __restrict__ dz,
          float* __restrict__ dbias) {
    extern __shared__ float s_db[];          // q
    for (int e = threadIdx.x; e < q; e += blockDim.x) s_db[e] = 0.f;
    __syncthreads();
    const int64_t total = rows * q;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    // stride is a multiple of q only by luck; track the column explicitly
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        const int64_t r = e / q;
        const int j = (int)(e - r * q);
        float v = d_out ? d_out[e] : d_bcast[(r % b_inner) * q + j] * scale;
        if (act == STMGCN_ACT_RELU && !(out[e] > 0.f)) v = 0.f;
        dz[e] = v;
        if (v != 0.f) atomicAdd(&s_db[j], v);
    }
    __syncthreads();
    if (dbias)
        for (int e = threadIdx.x; e < q; e += blockDim.x) atomicAdd(&dbias[e], s_db[e]);
}

// dW (kd x q) += S^T dZ for SMALL kd*q (the temporal GCN: kd = Ks*T = 48, q = T = 12): each CTA streams row chunks of
// S and dZ through shared memory; thread e owns outputs e, e + blockDim, ...  (i = out / q, j = out % q).
constexpr int kSmallRows = 64;
constexpr int kSmallThreads = 256;
constexpr int kSmallMaxPerThread = 8;
__global__ void __launch_bounds__(kSmallThreads)
small_wgrad_kernel(ASegs a, int64_t rows, int kd, const float* __restrict__ dz, int q, float* __restrict__ dw) {
    extern __shared__ float sm[];                    // S chunk [kSmallRows][kd] | dZ chunk [kSmallRows][q]
    float* ss = sm;
    float* ds = sm + kSmallRows * kd;
    const int n_out = kd * q;
    float acc[kSmallMaxPerThread];
#pragma unroll
    for (int o = 0; o < kSmallMaxPerThread; ++o) acc[o] = 0.f;
    for (int64_t r0 = (int64_t)blockIdx.x * kSmallRows; r0 < rows; r0 += (int64_t)gridDim.x * kSmallRows) {
        for (int e = threadIdx.x; e < kSmallRows * kd; e += kSmallThreads) {
            const int rr = e / kd, k = e % kd;
            const int sg = k / a.segw;
            const int64_t r = r0 + rr;
            ss[e] = (r < rows && a.seg[sg]) ? a.seg[sg][r * a.lda + (k - sg * a.segw)] : 0.f;
        }
        for (int e = threadIdx.x; e < kSmallRows * q; e += kSmallThreads) {
            const int64_t r = r0 + e / q;
            ds[e] = r < rows ? dz[r * q + e % q] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int o = 0; o < kSmallMaxPerThread; ++o) {
            const int out = threadIdx.x + o * kSmallThreads;
            if (out < n_out) {
                const int i = out / q, j = out % q;
                float s_acc = acc[o];
#pragma unroll 8
                for (int rr = 0; rr < kSmallRows; ++rr) s_acc = fmaf(ss[rr * kd + i], ds[rr * q + j], s_acc);
                acc[o] = s_acc;
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int o = 0; o < kSmallMaxPerThread; ++o) {
        const int out = threadIdx.x + o * kSmallThreads;
        if (out < n_out) atomicAdd(&dw[out], acc[o]);
    }
}

template <class Epi>
int32_t launch_tall_auto(const ASegs& a, int64_t rows, int kd, const float* b, int ldb, int nc, Epi epi,
                         cudaStream_t st, const char* what) {
    const bool vec = vec_ok(a, b, ldb, nc);
    if (nc <= 64) {
        epi.half_cols = 32;
        return vec ? launch_tall<64, true>(a, rows, kd, b, ldb, nc, epi, st, what)
                   : launch_tall<64, false>(a, rows, kd, b, ldb, nc, epi, st, what);
    }
    if (nc <= 128) {
        epi.half_cols = 64;
        return vec ? launch_tall<128, true>(a, rows, kd, b, ldb, nc, epi, st, what)
                   : launch_tall<128, false>(a, rows, kd, b, ldb, nc, epi, st, what);
    }
    epi.half_cols = 128;
    return vec ? launch_tall<256, true>(a, rows, kd, b, ldb, nc, epi, st, what)
               : launch_tall<256, false>(a, rows, kd, b, ldb, nc, epi, st, what);
}

}  // namespace

extern "C" {

int32_t stmgcn_proj_fwd(const float* s, int64_t stride_k, int32_t ks, int64_t rows, int32_t p, const float* w,
                        const float* bias, int32_t q, int32_t act, float* out, float* pool, int64_t b_inner,
                        void* stream) {
    STMGCN_REQUIRE(s && w && out, STMGCN_ERR_ARG, "proj_fwd: null pointer");
    STMGCN_REQUIRE(ks >= 1 && ks <= kMaxSegs, STMGCN_ERR_SHAPE, "proj_fwd: %d supports (max %d)", ks, kMaxSegs);
    STMGCN_REQUIRE(rows > 0 && p > 0 && q > 0, STMGCN_ERR_SHAPE, "proj_fwd: bad shape");
    STMGCN_REQUIRE(act == STMGCN_ACT_NONE || act == STMGCN_ACT_RELU, STMGCN_ERR_ARG, "proj_fwd: act=%d", act);
    cudaStream_t st = (cudaStream_t)stream;
    ASegs a{};
    a.nseg = ks;
    a.segw = p;
    a.lda = p;
    for (int k = 0; k < ks; ++k) a.seg[k] = s + (int64_t)k * stride_k;
    ProjEpi epi;
    epi.bias = bias;
    epi.act = act;
    epi.out = out;
    epi.half_cols = 0;
    if (int32_t rc = launch_tall_auto(a, rows, ks * p, w, q, q, epi, st, "proj_fwd")) return rc;
    if (pool) {
        STMGCN_REQUIRE(q == p, STMGCN_ERR_SHAPE, "proj_fwd: pooling needs q == p (got %d, %d)", q, p);
        STMGCN_REQUIRE(b_inner > 0 && rows % b_inner == 0, STMGCN_ERR_SHAPE, "proj_fwd: rows %% b_inner != 0");
        const int64_t cols = b_inner * q, n_regions = rows / b_inner;
        int64_t gy = (int64_t)sm_count() * 8 / ceil_div(cols, 256);
        if (gy < 1) gy = 1;
        if (gy > n_regions) gy = n_regions;
        if (gy > 65535) gy = 65535;
        dim3 grid((unsigned)ceil_div(cols, 256), (unsigned)gy);
        pool_kernel<<<grid, 256, 0, st>>>(s, out, n_regions, cols, pool);
        count_launch();
        return check_launch("proj_fwd pool");
    }
    return 0;
}

int32_t stmgcn_proj_bwd(const float* s, int64_t stride_k, int32_t ks, int64_t rows, int32_t p, const float* wt,
                        int32_t q, int32_t act, const float* out, const float* d_out, const float* d_out_bcast,
                        float bcast_scale, int64_t b_inner, float* dz_work, float* dw, float* dbias, float* u,
                        int64_t stride_u, void* stream) {
    STMGCN_REQUIRE(s && out && dz_work && dw, STMGCN_ERR_ARG, "proj_bwd: null pointer");
    STMGCN_REQUIRE((d_out != nullptr) != (d_out_bcast != nullptr), STMGCN_ERR_ARG,
                   "proj_bwd: exactly one of d_out / d_out_bcast");
    STMGCN_REQUIRE(ks >= 1 && ks <= kMaxSegs, STMGCN_ERR_SHAPE, "proj_bwd: %d supports (max %d)", ks, kMaxSegs);
    STMGCN_REQUIRE(rows > 0 && p > 0 && q > 0 && q <= 8192, STMGCN_ERR_SHAPE, "proj_bwd: bad shape");
    STMGCN_REQUIRE(!d_out_bcast || (b_inner > 0 && rows % b_inner == 0), STMGCN_ERR_SHAPE, "proj_bwd: b_inner");
    STMGCN_REQUIRE(!u || wt, STMGCN_ERR_ARG, "proj_bwd: u requested without wt");
    cudaStream_t st = (cudaStream_t)stream;
    {
        const int64_t total = rows * q;
        int64_t blocks = ceil_div(total, 256 * 8);
        const int64_t cap = (int64_t)sm_count() * 8;
        if (blocks > cap) blocks = cap;
        if (blocks < 1) blocks = 1;
        dz_kernel<<<(unsigned)blocks, 256, q * sizeof(float), st>>>(out, d_out, d_out_bcast, bcast_scale,
                                                                    b_inner > 0 ? b_inner : 1, rows, q, act,
                                                                    dz_work, dbias);
        count_launch();
        if (int32_t rc = check_launch("proj_bwd dz")) return rc;
    }
    if (ks * p * q <= kSmallThreads * kSmallMaxPerThread && (size_t)kSmallRows * (ks * p + q) * 4 <= 48 * 1024) {
        // small outputs (temporal GCN): dedicated streaming kernel instead of the 512-row-tile reduce GEMM
        ASegs a{};
        a.nseg = ks;
        a.segw = p;
        a.lda = p;
        for (int k = 0; k < ks; ++k) a.seg[k] = s + (int64_t)k * stride_k;
        int64_t blocks = ceil_div(rows, kSmallRows);
        const int64_t cap = (int64_t)sm_count() * 4;
        if (blocks > cap) blocks = cap;
        small_wgrad_kernel<<<(unsigned)blocks, kSmallThreads, (size_t)kSmallRows * (ks * p + q) * 4, st>>>(
            a, rows, ks * p, dz_work, q, dw);
        count_launch();
        if (int32_t rc = check_launch("proj_bwd dW(small)")) return rc;
    } else {   // dW (ks*p, q) += S^T dZ
        ASegs a{};
        a.nseg = ks;
        a.segw = p;
        a.lda = p;
        for (int k = 0; k < ks; ++k) a.seg[k] = s + (int64_t)k * stride_k;
        ReduceTime tm{};
        tm.n_t = 1;
        const int kd = ks * p;
        bool vec = (p % 4 == 0) && (q % 4 == 0) && aligned16(s) && aligned16(dz_work) && (stride_k % 4 == 0);
        int32_t rc;
        if (q <= 64)
            rc = vec ? launch_reduce<64, true>(a, tm, rows, kd, dz_work, q, q, dw, q, st, "proj_bwd dW")
                     : launch_reduce<64, false>(a, tm, rows, kd, dz_work, q, q, dw, q, st, "proj_bwd dW");
        else
            rc = vec ? launch_reduce<256, true>(a, tm, rows, kd, dz_work, q, q, dw, q, st, "proj_bwd dW")
                     : launch_reduce<256, false>(a, tm, rows, kd, dz_work, q, q, dw, q, st, "proj_bwd dW");
        if (rc) return rc;
    }
    if (u) {    // U_k = dZ W_k^T : A = dZ (rows x q), B = W^T (q x ks*p)
        ASegs a{};
        a.nseg = 1;
        a.segw = q;
        a.lda = q;
        a.seg[0] = dz_work;
        StoreSegEpi epi;
        epi.u = u;
        epi.stride_u = stride_u;
        epi.p = p;
        epi.half_cols = 0;
        return launch_tall_auto(a, rows, q, wt, ks * p, ks * p, epi, st, "proj_bwd U");
    }
    return 0;
}

}  // extern "C"
