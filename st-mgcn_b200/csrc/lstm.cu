// K3b: the shared-weight LSTM of CG_LSTM (reference STMGCN.py:21-22, :44, :47-50; nn.LSTM semantics: gate
// order i,f,g,o, b_ih + b_hh, zero initial state STMGCN.py:53-57), exact-fp32 CUDA-core path: every shape the
// tensor-core kernels of lstm16.cu do not cover (H != 64, C > 4), and the on-device reference the parity tests
// compare those kernels with.  Own tape: hs, cs (L,T,R,H) and post-activation gates (L,T,R,4H), fp32 row-major.
//
// Rows r = n*B + b (node-major) so the top layer's last hidden state IS the (N,B,H) operand of the spatial
// Chebyshev GCN (STMGCN.py:114) with no permute.  The context-gate modulation obs * s[b,t] (STMGCN.py:44)
// is folded into the layer-0 input read.  Weights arrive packed (see include/stmgcn_b200.h):
//   wx  (C, 4H)      = W_ih_l0^T, columns gate-interleaved (col = 4*unit + gate)
//   wp[l] (kd_l, 4H) = [W_ih_l^T ; W_hh_l^T] (l > 0) or W_hh_0^T (l = 0), same column order
//   wpt[l] (4H, kd_l)= wp[l]^T               (backward data GEMM operand)
#include "gemm_tall.cuh"

using namespace stmgcn;


namespace {

constexpr int kMaxLayers = 8;
constexpr int kMaxC = 4;
constexpr int kMaxUnitsPerLane = 4;      // hid <= 128

// ---- forward cell epilogue -----------------------------------------------------------------------------
struct LstmCellEpi {
    const float* bias;       // (4H) interleaved
    const float* wx;         // (C,4H) interleaved or nullptr (layers > 0)
    const float* xo;         // (R,T,C)
    const float* sg;         // (B,T)
    int c_in, t, t_len;
    int64_t b_inner;
    const float* c_prev;     // (R,H) or nullptr
    float* h_out;            // (R,H)
    float* c_out;            // (R,H)
    float* gates_out;        // (R,4H) or nullptr
    int hid;
    int half_units;          // TN/8

    __device__ __forceinline__ void operator()(float (&acc)[8][8], int64_t row0, int mg, int MG, int col0,
                                               int tn, int64_t rows, int nc) const {
        const int h4 = 4 * hid;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int64_t r = row0 + mg + (int64_t)i * MG;
            if (r >= rows) continue;
            float xs[kMaxC];
            if (wx != nullptr) {
                const float sv = sg[(r % b_inner) * t_len + t];
#pragma unroll
                for (int c = 0; c < kMaxC; ++c)
                    xs[c] = (c < c_in) ? xo[(r * t_len + t) * c_in + c] * sv : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int unit = col0 / 4 + (u ? half_units + tn : tn);
                if (unit >= hid) continue;
                const float4 bv = *reinterpret_cast<const float4*>(bias + 4 * unit);
                float pi = acc[i][4 * u + 0] + bv.x, pf = acc[i][4 * u + 1] + bv.y;
                float pg = acc[i][4 * u + 2] + bv.z, po = acc[i][4 * u + 3] + bv.w;
                if (wx != nullptr) {
#pragma unroll
                    for (int c = 0; c < kMaxC; ++c) {
                        if (c < c_in) {
                            const float4 wv = *reinterpret_cast<const float4*>(wx + (int64_t)c * h4 + 4 * unit);
                            pi = fmaf(xs[c], wv.x, pi);
                            pf = fmaf(xs[c], wv.y, pf);
                            pg = fmaf(xs[c], wv.z, pg);
                            po = fmaf(xs[c], wv.w, po);
                        }
                    }
                }
                const float gi = sigmoidf_(pi), gf = sigmoidf_(pf), gg = tanhf_(pg), go = sigmoidf_(po);
                const float cp = c_prev ? c_prev[r * hid + unit] : 0.f;
                const float cn = fmaf(gf, cp, gi * gg);
                const float hn = go * tanhf_(cn);
                c_out[r * hid + unit] = cn;
                h_out[r * hid + unit] = hn;
                if (gates_out) *reinterpret_cast<float4*>(gates_out + r * h4 + 4 * unit) = make_float4(gi, gf, gg, go);
            }
        }
    }
};

// ---- backward data epilogue: columns [0,w0) -> dst0, [w0, nc) -> dst1 ----------------------------------
struct StoreSplitEpi {
    float* dst0;
    int64_t ld0;
    int w0;
    float* dst1;
    int64_t ld1;
    int half_cols;           // TN/2

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
                if (n < w0) dst0[r * ld0 + n] = acc[i][j];
                else dst1[r * ld1 + (n - w0)] = acc[i][j];
            }
        }
    }
};

// ---- backward pointwise: gates (post-activation) -> dA (pre-activation gradient), in place ----------------
// one warp per row; lane owns units lane, lane+32, ...
__global__ void __launch_bounds__(256)
lstm_bwd_pointwise_kernel(int64_t rows, int hid, float* __restrict__ gates, const float* __restrict__ c_t,
                          const float* __restrict__ c_prev, const float* __restrict__ dh_in,
                          const float* __restrict__ dh_rec, float* __restrict__ dc,
                          float* __restrict__ dbp,            // (4H) +=
                          // layer-0 extras (wx == nullptr otherwise)
                          const float* __restrict__ wx, float* __restrict__ dwx, const float* __restrict__ xo,
                          const float* __restrict__ sg, float* __restrict__ d_s, int c_in, int t, int t_len,
                          int64_t b_inner) {
    const bool first = (t == t_len - 1);     // the incoming dh_rec / dc are zero by definition at the last time step
    extern __shared__ float sm[];            // [4H] dbias | [C*4H] dwx | [b_inner] ds (if it fits)
    const int h4 = 4 * hid;
    float* s_db = sm;
    float* s_dwx = sm + h4;
    float* s_ds = s_dwx + (wx ? c_in * h4 : 0);
    const bool ds_in_smem = (wx != nullptr) && (b_inner <= 2048);
    for (int e = threadIdx.x; e < h4 * (1 + (wx ? c_in : 0)); e += blockDim.x) sm[e] = 0.f;
    if (ds_in_smem)
        for (int e = threadIdx.x; e < b_inner; e += blockDim.x) s_ds[e] = 0.f;
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int ul = (hid + 31) / 32;
    float4 acc_b[kMaxUnitsPerLane];
    float4 acc_x[kMaxC][kMaxUnitsPerLane];
#pragma unroll
    for (int u = 0; u < kMaxUnitsPerLane; ++u) {
        acc_b[u] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int c = 0; c < kMaxC; ++c) acc_x[c][u] = make_float4(0.f, 0.f, 0.f, 0.f);
    }

    for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows;
         r += (int64_t)gridDim.x * (blockDim.x >> 5)) {
        float xs[kMaxC];
        float dxs[kMaxC];
        if (wx != nullptr) {
            const float sv = sg[(r % b_inner) * t_len + t];
#pragma unroll
            for (int c = 0; c < kMaxC; ++c) {
                xs[c] = (c < c_in) ? xo[(r * t_len + t) * c_in + c] * sv : 0.f;
                dxs[c] = 0.f;
            }
        }
#pragma unroll
        for (int u = 0; u < kMaxUnitsPerLane; ++u) {
            const int unit = lane + 32 * u;
            if (u >= ul || unit >= hid) continue;
            const int64_t e = r * hid + unit;
            const float4 g = *reinterpret_cast<const float4*>(gates + r * h4 + 4 * unit);   // i,f,g,o
            float dh = first ? 0.f : dh_rec[e];
            if (dh_in) dh += dh_in[e];
            const float tc = tanhf_(c_t[e]);
            const float cp = c_prev ? c_prev[e] : 0.f;
            const float dcv = (first ? 0.f : dc[e]) + dh * g.w * (1.f - tc * tc);
            float4 da;
            da.x = dcv * g.z * g.x * (1.f - g.x);
            da.y = dcv * cp * g.y * (1.f - g.y);
            da.z = dcv * g.x * (1.f - g.z * g.z);
            da.w = dh * tc * g.w * (1.f - g.w);
            dc[e] = dcv * g.y;
            *reinterpret_cast<float4*>(gates + r * h4 + 4 * unit) = da;
            acc_b[u].x += da.x; acc_b[u].y += da.y; acc_b[u].z += da.z; acc_b[u].w += da.w;
            if (wx != nullptr) {
#pragma unroll
                for (int c = 0; c < kMaxC; ++c) {
                    if (c < c_in) {
                        acc_x[c][u].x = fmaf(xs[c], da.x, acc_x[c][u].x);
                        acc_x[c][u].y = fmaf(xs[c], da.y, acc_x[c][u].y);
                        acc_x[c][u].z = fmaf(xs[c], da.z, acc_x[c][u].z);
                        acc_x[c][u].w = fmaf(xs[c], da.w, acc_x[c][u].w);
                        const float4 wv = *reinterpret_cast<const float4*>(wx + (int64_t)c * h4 + 4 * unit);
                        dxs[c] += da.x * wv.x + da.y * wv.y + da.z * wv.z + da.w * wv.w;
                    }
                }
            }
        }
        if (wx != nullptr) {
            // d s[b,t] += sum_c dxmod[r,c] * xo[r,t,c]   (xs = xo*s  =>  xo = xs/s is avoided: reload xo)
            float contrib = 0.f;
#pragma unroll
            for (int c = 0; c < kMaxC; ++c) {
                if (c < c_in) {
                    const float dx = warp_sum(dxs[c]);
                    contrib = fmaf(dx, xo[(r * t_len + t) * c_in + c], contrib);
                }
            }
            if (lane == 0) {
                const int64_t b = r % b_inner;
                if (ds_in_smem) atomicAdd(&s_ds[b], contrib);
                else atomicAdd(&d_s[b * t_len + t], contrib);
            }
        }
    }
    // CTA reduction of the bias / wx gradients through shared memory, then one global atomic per entry
#pragma unroll
    for (int u = 0; u < kMaxUnitsPerLane; ++u) {
        const int unit = lane + 32 * u;
        if (u >= ul || unit >= hid) continue;
        atomicAdd(&s_db[4 * unit + 0], acc_b[u].x);
        atomicAdd(&s_db[4 * unit + 1], acc_b[u].y);
        atomicAdd(&s_db[4 * unit + 2], acc_b[u].z);
        atomicAdd(&s_db[4 * unit + 3], acc_b[u].w);
        if (wx != nullptr) {
#pragma unroll
            for (int c = 0; c < kMaxC; ++c) {
                if (c < c_in) {
                    atomicAdd(&s_dwx[c * h4 + 4 * unit + 0], acc_x[c][u].x);
                    atomicAdd(&s_dwx[c * h4 + 4 * unit + 1], acc_x[c][u].y);
                    atomicAdd(&s_dwx[c * h4 + 4 * unit + 2], acc_x[c][u].z);
                    atomicAdd(&s_dwx[c * h4 + 4 * unit + 3], acc_x[c][u].w);
                }
            }
        }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < h4; e += blockDim.x) atomicAdd(&dbp[e], s_db[e]);
    if (wx != nullptr) {
        for (int e = threadIdx.x; e < c_in * h4; e += blockDim.x) atomicAdd(&dwx[e], s_dwx[e]);
        if (ds_in_smem)
            for (int e = threadIdx.x; e < b_inner; e += blockDim.x) atomicAdd(&d_s[(int64_t)e * t_len + t], s_ds[e]);
    }
}

int32_t check_dims(const char* who, int32_t t_len, int32_t n_layers, int64_t rows, int32_t hid, int32_t c_in,
                   int64_t b_inner) {
    STMGCN_REQUIRE(t_len >= 1, STMGCN_ERR_SHAPE, "%s: T=%d", who, t_len);
    STMGCN_REQUIRE(n_layers >= 1 && n_layers <= kMaxLayers, STMGCN_ERR_SHAPE, "%s: layers=%d (max %d)", who,
                   n_layers, kMaxLayers);
    STMGCN_REQUIRE(rows > 0 && b_inner > 0 && rows % b_inner == 0, STMGCN_ERR_SHAPE, "%s: rows=%lld b=%lld", who,
                   (long long)rows, (long long)b_inner);
    STMGCN_REQUIRE(hid > 0 && hid % 4 == 0 && hid <= 32 * kMaxUnitsPerLane, STMGCN_ERR_SHAPE,
                   "%s: lstm hidden=%d unsupported (need multiple of 4, <= %d)", who, hid, 32 * kMaxUnitsPerLane);
    STMGCN_REQUIRE(c_in >= 1 && c_in <= kMaxC, STMGCN_ERR_SHAPE, "%s: input_dim=%d unsupported (max %d)", who,
                   c_in, kMaxC);
    return 0;
}

}  // namespace

extern "C" {

int32_t stmgcn_lstm_fwd(int32_t t_len, int32_t n_layers, int64_t rows, int32_t hid, int32_t c_in, int64_t b_inner,
                        const float* xo, const float* s_gate, const float* wx, const float* const* wp,
                        const float* const* bp, const float* h0, const float* c0, float* hs, float* cs, float* gates,
                        void* stream) {
    STMGCN_REQUIRE(xo && s_gate && wx && wp && bp && hs && cs, STMGCN_ERR_ARG, "lstm_fwd: null pointer");
    if (int32_t rc = check_dims("lstm_fwd", t_len, n_layers, rows, hid, c_in, b_inner)) return rc;
    for (int l = 0; l < n_layers; ++l) STMGCN_REQUIRE(wp[l] && bp[l], STMGCN_ERR_ARG, "lstm_fwd: wp/bp[%d] null", l);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t rh = rows * hid;
    const int h4 = 4 * hid;
    for (int t = 0; t < t_len; ++t)
        for (int l = 0; l < n_layers; ++l) {
            const float* h_prev = t > 0 ? hs + ((int64_t)(l * t_len + t - 1)) * rh : (h0 ? h0 + (int64_t)l * rh : nullptr);
            const float* c_prev = t > 0 ? cs + ((int64_t)(l * t_len + t - 1)) * rh : (c0 ? c0 + (int64_t)l * rh : nullptr);
            ASegs a{};
            a.segw = hid;
            a.lda = hid;
            if (l == 0) {
                a.nseg = 1;
                a.seg[0] = h_prev;
            } else {
                a.nseg = 2;
                a.seg[0] = hs + ((int64_t)((l - 1) * t_len + t)) * rh;
                a.seg[1] = h_prev;
            }
            LstmCellEpi epi;
            epi.bias = bp[l];
            epi.wx = (l == 0) ? wx : nullptr;
            epi.xo = xo;
            epi.sg = s_gate;
            epi.c_in = c_in;
            epi.t = t;
            epi.t_len = t_len;
            epi.b_inner = b_inner;
            epi.c_prev = c_prev;
            epi.h_out = hs + ((int64_t)(l * t_len + t)) * rh;
            epi.c_out = cs + ((int64_t)(l * t_len + t)) * rh;
            epi.gates_out = gates ? gates + ((int64_t)(l * t_len + t)) * rows * h4 : nullptr;
            epi.hid = hid;
            epi.half_units = 256 / 8;
            const int kd = a.nseg * hid;
            int32_t rc;
            if (vec_ok(a, wp[l], h4, h4))
                rc = launch_tall<256, true>(a, rows, kd, wp[l], h4, h4, epi, st, "lstm_fwd");
            else
                rc = launch_tall<256, false>(a, rows, kd, wp[l], h4, h4, epi, st, "lstm_fwd");
            if (rc) return rc;
        }
    return 0;
}

int32_t stmgcn_lstm_bwd(int32_t t_len, int32_t n_layers, int64_t rows, int32_t hid, int32_t c_in, int64_t b_inner,
                        const float* xo, const float* s_gate, const float* wx, const float* const* wpt, const float* h0,
                        const float* c0, const float* hs, const float* cs, float* gates, const float* d_top,
                        float* dh_rec, float* dc, float* dx_work, float* d_s, float* dwx, float* const* dbp,
                        float* const* dwp, void* stream) {
    STMGCN_REQUIRE(xo && s_gate && wx && wpt && hs && cs && gates && d_top && dh_rec && dc && dx_work && d_s && dwx && dbp &&
                       dwp,
                   STMGCN_ERR_ARG, "lstm_bwd: null pointer");
    if (int32_t rc = check_dims("lstm_bwd", t_len, n_layers, rows, hid, c_in, b_inner)) return rc;
    for (int l = 0; l < n_layers; ++l)
        STMGCN_REQUIRE(wpt[l] && dbp[l] && dwp[l], STMGCN_ERR_ARG, "lstm_bwd: wpt/dbp/dwp[%d] null", l);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t rh = rows * hid;
    const int h4 = 4 * hid;
    const int grid_pw = (int)((ceil_div(rows, 8) < (int64_t)sm_count() * 4) ? ceil_div(rows, 8) : (int64_t)sm_count() * 4);
    // BPTT, t = T-1 .. 0, layers top-down; dx_work carries a layer's input gradient to the layer below
    for (int t = t_len - 1; t >= 0; --t)
        for (int l = n_layers - 1; l >= 0; --l) {
            float* g_lt = gates + ((int64_t)(l * t_len + t)) * rows * h4;
            const float* c_t = cs + ((int64_t)(l * t_len + t)) * rh;
            const float* c_prev = t > 0 ? cs + ((int64_t)(l * t_len + t - 1)) * rh : (c0 ? c0 + (int64_t)l * rh : nullptr);
            const float* dh_in = (l == n_layers - 1) ? ((t == t_len - 1) ? d_top : nullptr) : dx_work;
            const bool l0 = (l == 0);
            size_t smem = (size_t)h4 * (1 + (l0 ? c_in : 0)) * sizeof(float);
            if (l0 && b_inner <= 2048) smem += (size_t)b_inner * sizeof(float);
            lstm_bwd_pointwise_kernel<<<grid_pw, 256, smem, st>>>(
                rows, hid, g_lt, c_t, c_prev, dh_in, dh_rec + (int64_t)l * rh, dc + (int64_t)l * rh, dbp[l],
                l0 ? wx : nullptr, l0 ? dwx : nullptr, xo, s_gate, d_s, c_in, t, t_len, b_inner);
            count_launch();
            if (int32_t rc = check_launch("lstm_bwd (pointwise)")) return rc;
            // data gradients: [dx_below | dh_rec] = dA . wpt[l]      (dA: rows x 4H, wpt[l]: 4H x kd_l)
            ASegs a{};
            a.nseg = 1;
            a.segw = h4;
            a.lda = h4;
            a.seg[0] = g_lt;
            StoreSplitEpi epi;
            epi.dst0 = l0 ? nullptr : dx_work;
            epi.ld0 = hid;
            epi.w0 = l0 ? 0 : hid;
            epi.dst1 = dh_rec + (int64_t)l * rh;
            epi.ld1 = hid;
            const int nc = l0 ? hid : 2 * hid;
            int32_t rc;
            if (nc > 64) {
                epi.half_cols = 64;
                if (vec_ok(a, wpt[l], nc, nc)) rc = launch_tall<128, true>(a, rows, h4, wpt[l], nc, nc, epi, st, "lstm_bwd (data)");
                else rc = launch_tall<128, false>(a, rows, h4, wpt[l], nc, nc, epi, st, "lstm_bwd (data)");
            } else {
                epi.half_cols = 32;
                if (vec_ok(a, wpt[l], nc, nc)) rc = launch_tall<64, true>(a, rows, h4, wpt[l], nc, nc, epi, st, "lstm_bwd (data)");
                else rc = launch_tall<64, false>(a, rows, h4, wpt[l], nc, nc, epi, st, "lstm_bwd (data)");
            }
            if (rc) return rc;
        }
    // weight gradients, one layer at a time: dwp[l] += [h_below_t | h_{t-1}]^T dA summed over all (t, r)
    for (int l = 0; l < n_layers; ++l) {
        ASegs a{};
        ReduceTime tm{};
        a.segw = hid;
        a.lda = hid;
        tm.n_t = t_len;
        tm.d_tstride = rows * h4;
        int s = 0;
        if (l > 0) {                           // input from the layer below, same step
            a.seg[s] = hs + ((int64_t)(l - 1) * t_len) * rh;
            tm.a_tstride[s] = rh;
            tm.a_shift[s] = 0;
            tm.a_t0[s] = nullptr;
            ++s;
        }
        a.seg[s] = hs + ((int64_t)l * t_len) * rh;      // h_{t-1} of this layer
        tm.a_tstride[s] = rh;
        tm.a_shift[s] = 1;
        tm.a_t0[s] = h0 ? h0 + (int64_t)l * rh : nullptr;
        ++s;
        a.nseg = s;
        const int kd = s * hid;
        const float* d = gates + ((int64_t)l * t_len) * rows * h4;
        const bool vec = (hid % 4 == 0) && aligned16(d) && aligned16(hs) && (!h0 || aligned16(h0));
        const int32_t rc = vec ? launch_reduce<256, true>(a, tm, rows, kd, d, h4, h4, dwp[l], h4, st, "lstm_bwd (weights)")
                               : launch_reduce<256, false>(a, tm, rows, kd, d, h4, h4, dwp[l], h4, st, "lstm_bwd (weights)");
        if (rc) return rc;
    }
    return 0;
}

}  // extern "C"
