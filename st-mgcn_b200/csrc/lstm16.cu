// K3b, second generation (H = 64): the shared LSTM of CG_LSTM (reference STMGCN.py:21-22, :47-50; nn.LSTM semantics)
// on tcgen05 with bf16 hi/lo PLANES ("3xBF16", see tc16.cuh) and NO gate tape.
//
// Tape written by the forward (all the backward needs; it recomputes the gates from it):
//   hp : (L, T, P, rows, 64) bf16  -- the hidden state of every layer-step as P planes (P = 2: hi | lo, fp32-grade
//        arithmetic; P = 1: hi only, the bf16 mode).  A 128-row x 64-column piece of a plane IS a K-major, 128-byte
//        swizzled tcgen05 operand tile once a TMA tensor load has put it into shared memory -- no splitter warps, no
//        per-thread loads, no proxy fences on the operand path.
//   cs : (L, T, rows_pad, 64) fp32, tile-blocked ([tile][unit/4][128 rows][4 units], see below): the 32 lanes of a warp
//        (32 consecutive rows, the same 4 units) touch ONE contiguous 512-byte run per access.  (With 8-unit groups every
//        access was 16 bytes at a 32-byte stride: 32 half-used sectors and ~22 L1 data-pipe wavefronts per request; ncu
//        showed the L1 data pipe -- tensor-core operand reads + LSU -- at 77 % (forward) / 90 % (backward) of its peak.)
// 4 + 4 bytes per (row, unit, layer-step) instead of 4 + 4 + 16 with the gate tape of the first-generation (3xTF32)
// kernels: 4.8 GB instead of 14.5 GB per graph branch at BASELINE configs[2], and configs[4] fits.
//
// forward kernel (one launch per layer-step, persistent, one CTA per SM):
//   producer warp : loads the layer's weight image ONCE (resident for the whole launch: [256 gate cols][64 k] bf16 tiles,
//                   hi and lo, per K segment = 128 KB) and streams the A planes of every tile through a ring of 16 KB
//                   stages with TMA tensor loads (h_below hi, h_below lo, h_prev hi, h_prev lo)
//   MMA warp      : per tile 8 (P = 1) or 24 (P = 2) tcgen05.mma kind::f16 (M 128, N 256, K 16) into one of two TMEM
//                   accumulators: Ahi.Whi + Ahi.Wlo + Alo.Whi
//   16 epilogue warps: TMEM -> registers -> bias (+ layer 0: x*s . W_ih in exact fp32) -> gates -> c, h -> h split into
//                   bf16 planes -> coalesced global stores.  Nothing of the gates leaves the SM.
#include "tc16.cuh"
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

using namespace stmgcn;
using namespace stmgcn::tc;

namespace {

constexpr int kTileM = 128;
constexpr int kHid = 64;
constexpr int kGateCols = 256;
constexpr int kMaxC = 4;
constexpr int kWTileBytes = kGateCols * 128;          // [256 gate cols][64 k] bf16 = 32 KB
constexpr int kATileBytes = kTile16Bytes;             // [128 rows][64 k] bf16 = 16 KB

// element (row r, unit u) of a tile-blocked (rows_pad x 64) fp32 workspace lives at
//   (((r >> 7) * 16 + (unit >> 2)) * 128 + (r & 127)) * 4 + (unit & 3)        (host side: ops.to_blocked / from_blocked)

__device__ __forceinline__ void tma_load_3d(void* smem_dst, const void* tmap, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 :: "r"(smem_u32(smem_dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// ---- LSTM cell with 8 MUFU operations instead of 10 ------------------------------------------------------------
// sigmoid(v) = 1 / (1 + e^-v), tanh(v) = (1 - e^-2v) / (1 + e^-2v).  Five exponentials per cell are unavoidable (i, f, g, o,
// tanh(c)); the five reciprocals are not: reciprocals of PRODUCTS of two (1 + e) terms serve two activations at once.
// The exponentials are capped at e^30 (the capped activations differ from the exact ones by < 1e-13) so that a
// product of two (1 + e^30) terms stays far below the fp32 overflow threshold.  The cell epilogue is MUFU-bound
// (16 MUFU results per clock and SM), so this is 20 % off its critical resource.
// (one-sided: only a large NEGATIVE argument makes e^-v large; for large positive v the exponential underflows to 0, which is exact)
// The kernels keep bias and W_ih PRE-SCALED by the exponent factor of their gate (kGateScale: -log2(e) for i, f, o and
// -2 log2(e) for g), so "accumulator + bias, times -log2(e)" is ONE fma per gate: arg = fma(acc, scale, bias_scaled).
__device__ __forceinline__ float gate_scale(int col) { return (col & 3) == 2 ? -2.8853900817779268f : -1.4426950408889634f; }
__device__ __forceinline__ float exp_arg_(float a) { return ex2_ftz_(fminf(a, 43.28f)); }      // e^(-v) or e^(-2v), <= e^30
// forward: exponent arguments of (i, f, g, o) and c_{t-1} -> c_t, h_t
__device__ __forceinline__ void lstm_cell_fwd8(float ai, float af, float ag, float ao, float cp, float& c, float& h) {
    const float ei = exp_arg_(ai), ef = exp_arg_(af), eg = exp_arg_(ag), eo = exp_arg_(ao);
    const float ig = (1.f - eg) * rcp_ftz_((1.f + ei) * (1.f + eg));          // sigmoid(pi) * tanh(pg)
    c = fmaf(rcp_ftz_(1.f + ef), cp, ig);
    const float ec = exp_arg_(-2.8853900817779268f * c);
    h = (1.f - ec) * rcp_ftz_((1.f + eo) * (1.f + ec));                      // sigmoid(po) * tanh(c)
}
// backward recompute: all four gate activations, c_t and tanh(c_t)
__device__ __forceinline__ void lstm_cell_gates8(float ai, float af, float ag, float ao, float cp, float& gi, float& gf,
                                                 float& gg, float& go, float& tc) {
    const float ei = 1.f + exp_arg_(ai), ef = 1.f + exp_arg_(af), eo = 1.f + exp_arg_(ao);
    const float eg = exp_arg_(ag);
    const float r1 = rcp_ftz_(ei * (1.f + eg));
    const float r2 = rcp_ftz_(ef * eo);
    gi = r1 * (1.f + eg);
    gg = (1.f - eg) * (r1 * ei);
    gf = r2 * eo;
    go = r2 * ef;
    const float ec = exp_arg_(-2.8853900817779268f * fmaf(gf, cp, gi * gg));
    tc = (1.f - ec) * rcp_ftz_(1.f + ec);
}

// L2 prefetch of a tensor-map box (no shared memory, no barrier): the later TMA load of the same box finds it in L2
__device__ __forceinline__ void tma_prefetch_3d(const void* tmap, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];"
                 :: "l"(tmap), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// =====================================================================================================
// forward
// =====================================================================================================
constexpr int kFEpiWarps = 16;
constexpr int kFThreads = (kFEpiWarps + 2) * 32;       // + MMA warp + producer warp
constexpr int kFStages = 5;

struct F16Tail {
    float bias[kGateCols];
    float wih[kMaxC * kGateCols];
    uint64_t full[kFStages];
    uint64_t empty[kFStages];
    uint64_t tmem_full[2];
    uint64_t tmem_empty[2];
    uint64_t w_full;
    uint32_t tmem_base;
};
constexpr size_t kFSmem = 1024 + 4 * (size_t)kWTileBytes + (size_t)kFStages * kATileBytes + sizeof(F16Tail);
static_assert(kFSmem <= 232448, "lstm16 forward kernel exceeds the 227 KB shared-memory limit");

struct Fwd16Params {
    alignas(64) CUtensorMap amap[2];   // per K segment: (64, rows, slices) bf16 view of a plane tensor, box 64 x 128 x 1, 128B swizzle
    int aslice[2];                     // slice of the segment's hi plane (lo plane = +1)
    int nseg;                          // K segments present: layer 0: h_prev; layers > 0: h_below, h_prev (absent at t = 0 without h0)
    const uint8_t* wimg;               // tiles [(seg*2 + plane)] of 32 KB
    const float* bias;                 // (256) gate-interleaved b_ih + b_hh
    const float* wih;                  // layer 0: (C, 256) gate-interleaved W_ih^T; else nullptr
    const float* xo;                   // (rows, T, C)
    const float* sg;                   // (B, T)
    int c_in, t, t_len;
    int64_t b_inner;
    const float* c_prev;               // tile-blocked or nullptr (zeros)
    float* c_out;                      // tile-blocked
    uint16_t* h_hi;                    // (rows, 64) bf16 plane
    uint16_t* h_lo;                    // (rows, 64) bf16 plane (PLANES = 2)
    float* h_f32;                      // (rows, 64) fp32 copy of h or nullptr
    int64_t rows;
    int n_tiles;
};

// CIN: 0 = not layer 0; 1 = layer 0 with one input channel (the reference's input_dim, compile-time: no predicated-off
// W_ih FMAs / loads in the cell loop); kMaxC = layer 0 with a runtime channel count <= kMaxC
template <int PLANES, int CIN>
__global__ void __launch_bounds__(kFThreads, 1) lstm16_fwd_kernel(const __grid_constant__ Fwd16Params p) {
    constexpr bool L0 = CIN > 0;
    constexpr int kC = (CIN == 1) ? 1 : kMaxC;
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment by pointer arithmetic on the __shared__ array (an integer round trip would make every access through
    // `smem` a generic LD/ST/ATOM instead of LDS/STS/ATOMS: ncu showed the bias loads as long-scoreboard stalls)
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* wsm = smem;                                           // resident weight tiles
    uint8_t* stages = smem + 4 * (size_t)kWTileBytes;
    F16Tail* tail = (F16Tail*)(stages + (size_t)kFStages * kATileBytes);
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;
    constexpr int kMmaWarp = kFEpiWarps;
    constexpr int kProdWarp = kFEpiWarps + 1;

    if (tid == 0) {
        for (int s = 0; s < kFStages; ++s) {
            mbar_init(&tail->full[s], 1);
            mbar_init(&tail->empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tail->tmem_full[a], 1);
            mbar_init(&tail->tmem_empty[a], kFEpiWarps);       // one arrival per epilogue warp
        }
        mbar_init(&tail->w_full, 1);
        fence_barrier_init();
    }
    if (warp == kMmaWarp) tmem_alloc(&tail->tmem_base, 512);
    for (int i = tid; i < kGateCols; i += kFThreads) tail->bias[i] = p.bias[i] * gate_scale(i);
    if (L0)
        for (int i = tid; i < p.c_in * kGateCols; i += kFThreads) tail->wih[i] = p.wih[i] * gate_scale(i);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tail->tmem_base;
    const int my_tiles = (p.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

    if (warp == kProdWarp) {
        // ===================== producer: resident weights once, then the A planes of every tile =====================
        TC_PROF_DECL
        const bool leader = elect_one_sync();
        if (leader && p.nseg > 0) {
            mbar_arrive_expect_tx(&tail->w_full, (uint32_t)(p.nseg * PLANES * kWTileBytes));
            for (int s = 0; s < p.nseg; ++s)
                for (int pl = 0; pl < PLANES; ++pl)
                    bulk_g2s(wsm + (size_t)(s * 2 + pl) * kWTileBytes, p.wimg + (size_t)(s * 2 + pl) * kWTileBytes, kWTileBytes,
                             &tail->w_full);
            uint32_t it = 0;
            for (int i = 0; i < my_tiles; ++i) {
                const int tile = blockIdx.x + i * gridDim.x;
                if (p.c_prev != nullptr && i + 2 < my_tiles)     // c_{t-1} of the tile after next -> L2 (a tile is contiguous)
                    prefetch_l2(p.c_prev + (int64_t)(tile + 2 * (int)gridDim.x) * kTileM * kHid, kTileM * kHid * 4);
                for (int s = 0; s < p.nseg; ++s)
                    for (int pl = 0; pl < PLANES; ++pl, ++it) {
                        const int stg = it % kFStages;
                        const uint32_t ph = (it / kFStages) & 1;
                        mbar_wait_p(&tail->empty[stg], ph ^ 1, 0);
                        mbar_arrive_expect_tx(&tail->full[stg], kATileBytes);
                        tma_load_3d(stages + (size_t)stg * kATileBytes, &p.amap[s], 0, tile * kTileM, p.aslice[s] + pl,
                                    &tail->full[stg]);
                    }
            }
        }
        TC_PROF_FLUSH(0, leader)
    } else if (warp == kMmaWarp) {
        // ===================== MMA issuer =====================
        TC_PROF_DECL
        const bool leader = elect_one_sync();
        if (p.nseg > 0) {
            constexpr uint32_t idesc = idesc_bf16(kTileM, kGateCols);
            mbar_wait_p(&tail->w_full, 0, 0);
            tc_fence_after();
            uint32_t it = 0;
            for (int i = 0; i < my_tiles; ++i) {
                const int a = i & 1;
                const uint32_t aph = (uint32_t)(i >> 1) & 1;
                mbar_wait_p(&tail->tmem_empty[a], aph ^ 1, 2);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)a * kGateCols;
                for (int s = 0; s < p.nseg; ++s) {
                    const uint64_t w_hi = desc16_k(smem_u32(wsm + (size_t)(s * 2) * kWTileBytes));
                    const uint64_t w_lo = desc16_k(smem_u32(wsm + (size_t)(s * 2 + 1) * kWTileBytes));
                    {   // hi plane of the segment: against W hi (and W lo)
                        const int stg = it % kFStages;
                        const uint32_t ph = (it / kFStages) & 1;
                        mbar_wait_p(&tail->full[stg], ph, 1);
                        tc_fence_after();
                        if (leader) {
                            const uint64_t a_d = desc16_k(smem_u32(stages + (size_t)stg * kATileBytes));
                            if (PLANES == 2) {
                                // per k-step: A_hi . W_hi keeps A in the collector, A_hi . W_lo re-uses it (one A read, not two)
#pragma unroll
                                for (int kk = 0; kk < 4; ++kk) {
                                    mma_bf16_keep_a(d_tmem, a_d + (uint64_t)(2 * kk), w_hi + (uint64_t)(2 * kk), idesc, (s > 0 || kk > 0) ? 1u : 0u);
                                    mma_bf16_reuse_a(d_tmem, a_d + (uint64_t)(2 * kk), w_lo + (uint64_t)(2 * kk), idesc, 1u);
                                }
                            } else {
#pragma unroll
                                for (int kk = 0; kk < 4; ++kk)
                                    mma_bf16(d_tmem, a_d + (uint64_t)(2 * kk), w_hi + (uint64_t)(2 * kk), idesc, (s > 0 || kk > 0) ? 1u : 0u);
                            }
                            mma_commit(&tail->empty[stg]);
                        }
                        __syncwarp();
                        ++it;
                    }
                    if (PLANES == 2) {   // lo plane of the segment: against W hi
                        const int stg = it % kFStages;
                        const uint32_t ph = (it / kFStages) & 1;
                        mbar_wait_p(&tail->full[stg], ph, 1);
                        tc_fence_after();
                        if (leader) {
                            const uint64_t a_d = desc16_k(smem_u32(stages + (size_t)stg * kATileBytes));
#pragma unroll
                            for (int kk = 0; kk < 4; ++kk)
                                mma_bf16(d_tmem, a_d + (uint64_t)(2 * kk), w_hi + (uint64_t)(2 * kk), idesc, 1u);
                            mma_commit(&tail->empty[stg]);
                        }
                        __syncwarp();
                        ++it;
                    }
                }
                if (leader) mma_commit(&tail->tmem_full[a]);
                __syncwarp();
            }
        }
        TC_PROF_FLUSH(1, leader)
    } else {
        // ===================== epilogue: LSTM cell =====================
        TC_PROF_DECL
        // TMEM lane quadrant q = warp & 3 (rows 32q .. 32q+31 of the tile), column quarter part = warp >> 2
        // (gate columns 64*part .. +63 = units 16*part .. +15), four pieces of 16 columns = 4 units each
        const int q = warp & 3, part = warp >> 2;
        constexpr bool l0 = L0;
        // c_{t-1} of this thread's row (16 units) lives in registers; the four floats a piece has just consumed are
        // reloaded at once with the NEXT tile's values, so the loads are in flight for most of a tile (loading all 16 at the
        // end of a tile exposed the full DRAM latency at the top of the next one: ncu showed 21 % of the samples there)
        float cpv[16];
        float xs[kMaxC], xs_next[kMaxC], sv_next = 0.f;    // xs_next: raw x of the next tile; scaled by sv_next at the swap
        // 32-bit element offsets (rows <= 2^25 is checked on the host): 64-bit address pairs cost registers, and the few
        // that spilled were re-read from local memory in the tile loop at full L1-miss latency (ncu: 18 % of the samples)
        const uint32_t row_in_tile = (uint32_t)(q * 32 + lane);
        const uint32_t rows32 = (uint32_t)p.rows;
        // tile-blocked (rows_pad x 64): element (tile, row, unit) at tile*8192 + (unit/4)*512 + row*4 + unit%4
        const uint32_t thr_c = row_in_tile * 4u + (uint32_t)part * 2048u;
        auto load_c4 = [&](int tile_n, int j) {
            const uint32_t rn = (uint32_t)tile_n * kTileM + row_in_tile;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.c_prev != nullptr && tile_n < p.n_tiles && rn < rows32)
                v = *reinterpret_cast<const float4*>(p.c_prev + ((uint32_t)tile_n * 8192u + thr_c + (uint32_t)j * 512u));
            cpv[4 * j] = v.x; cpv[4 * j + 1] = v.y; cpv[4 * j + 2] = v.z; cpv[4 * j + 3] = v.w;
        };
        // loads only: the product x * s is formed when the tile starts (multiplying here waited for the loads on the spot:
        // 14 % of the layer-0 kernel's stall samples)
        auto load_xs = [&](int tile_n) {
            const uint32_t rn = (uint32_t)tile_n * kTileM + row_in_tile;
            const bool ok = tile_n < p.n_tiles && rn < rows32;
            sv_next = 0.f;
            if (ok) sv_next = p.sg[(rn % (uint32_t)p.b_inner) * (uint32_t)p.t_len + (uint32_t)p.t];    // (32-bit: a 64-bit % is a call)
#pragma unroll
            for (int c = 0; c < kMaxC; ++c)
                xs_next[c] = (c < kC && ok && (CIN == 1 || c < p.c_in)) ? p.xo[((int64_t)rn * p.t_len + p.t) * p.c_in + c] : 0.f;
        };
#pragma unroll
        for (int j = 0; j < 4; ++j) load_c4((int)blockIdx.x, j);
        if (l0) {
            load_xs((int)blockIdx.x);
#pragma unroll
            for (int c = 0; c < kMaxC; ++c) xs[c] = xs_next[c] * sv_next;
        }
        const int gstep = (int)gridDim.x;
        int tile = (int)blockIdx.x;                // carried in a register: re-reading %ctaid every tile is a long-scoreboard stall
        for (int i = 0; i < my_tiles; ++i, tile += gstep) {
            const int a = i & 1;
            const uint32_t aph = (uint32_t)(i >> 1) & 1;
            const uint32_t r = (uint32_t)tile * kTileM + row_in_tile;
            const bool valid = r < rows32;
            if (p.nseg > 0) {
                mbar_wait(&tail->tmem_full[a], aph, 3);
                tc_fence_after();
            }
            const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)a * kGateCols + (uint32_t)part * 64;
            // (measured and rejected: software-pipelining the tcgen05.ld of the next piece under this piece's arithmetic with
            //  per-piece 8-byte h stores -- 3.77 ms per branch forward against 2.86 ms for this load-then-wait form)
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int pc = 0; pc < 4; ++pc) {
                uint32_t v[16];
                if (p.nseg > 0) {
                    tmem_ld16(t_row + pc * 16, v);
                    tmem_ld_wait();
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = 0u;
                }
                const int unit0 = part * 16 + pc * 4;
                float hn[4], cn[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int col = 4 * (unit0 + u);
                    const float4 bv = *reinterpret_cast<const float4*>(&tail->bias[col]);      // pre-scaled (gate_scale)
                    float pi = fmaf(__uint_as_float(v[4 * u + 0]), -1.4426950408889634f, bv.x);
                    float pf = fmaf(__uint_as_float(v[4 * u + 1]), -1.4426950408889634f, bv.y);
                    float pg = fmaf(__uint_as_float(v[4 * u + 2]), -2.8853900817779268f, bv.z);
                    float po = fmaf(__uint_as_float(v[4 * u + 3]), -1.4426950408889634f, bv.w);
                    if (l0) {
#pragma unroll
                        for (int c = 0; c < kC; ++c)
                            if (CIN == 1 || c < p.c_in) {
                                const float4 wv = *reinterpret_cast<const float4*>(&tail->wih[c * kGateCols + col]);
                                pi = fmaf(xs[c], wv.x, pi); pf = fmaf(xs[c], wv.y, pf);
                                pg = fmaf(xs[c], wv.z, pg); po = fmaf(xs[c], wv.w, po);
                            }
                    }
                    lstm_cell_fwd8(pi, pf, pg, po, cpv[4 * pc + u], cn[u], hn[u]);
                }
                if (PLANES == 2) {
                    split_bf16x2(hn[0], hn[1], hi[2 * pc], lo[2 * pc]);
                    split_bf16x2(hn[2], hn[3], hi[2 * pc + 1], lo[2 * pc + 1]);
                } else {
                    hi[2 * pc] = pack_bf16x2(hn[0], hn[1]);
                    hi[2 * pc + 1] = pack_bf16x2(hn[2], hn[3]);
                }
                if (valid) {
                    *reinterpret_cast<float4*>(p.c_out + ((uint32_t)tile * 8192u + thr_c + (uint32_t)pc * 512u)) =
                        make_float4(cn[0], cn[1], cn[2], cn[3]);
                    if (p.h_f32 != nullptr)
                        *reinterpret_cast<float4*>(p.h_f32 + (r * (uint32_t)kHid + (uint32_t)unit0)) = make_float4(hn[0], hn[1], hn[2], hn[3]);
                }
                load_c4(tile + gstep, pc);                      // this piece's registers are free: next tile's values
                if (l0 && pc == 0) load_xs(tile + gstep);
            }
            if (p.nseg > 0) {          // all TMEM reads of this accumulator are done (one mbarrier arrival per warp: 512
                tc_fence_before();     // per-thread arrivals are 512 serialised shared-memory atomics per tile)
                __syncwarp();
                if (lane == 0) mbar_arrive(&tail->tmem_empty[a]);
            }
            if (valid) {
                // 16 bf16 = 32 bytes per row and plane: one 256-bit store (a full sector) instead of two 128-bit ones
                st_global_v8(p.h_hi + (r * (uint32_t)kHid + (uint32_t)part * 16u), hi);
                if (PLANES == 2) st_global_v8(p.h_lo + (r * (uint32_t)kHid + (uint32_t)part * 16u), lo);
            }
            if (l0) {
#pragma unroll
                for (int c = 0; c < kMaxC; ++c) xs[c] = xs_next[c] * sv_next;
            }
        }
        TC_PROF_FLUSH(2, tid == 0)
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == kMmaWarp) tmem_dealloc(tmem_base, 512);
}

// ---- weight image packer: nn.LSTM parameters of one layer -> resident operand tiles + interleaved bias / W_ih^T ----
// tile (seg, plane): [256 rows n = 4*unit + gate][64 k] bf16, 128-byte swizzle; seg 0 = W_ih (layers > 0) or W_hh (layer 0),
// seg 1 = W_hh (layers > 0).  Native row of gate-interleaved column n: (n & 3) * 64 + (n >> 2)  (gate order i, f, g, o).
__global__ void lstm16_pack_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh,
                                   const float* __restrict__ b_ih, const float* __restrict__ b_hh, int layer, int c_in,
                                   uint8_t* __restrict__ wimg, float* __restrict__ bias, float* __restrict__ wih_t) {
    const int nseg = layer == 0 ? 1 : 2;
    const int total = nseg * kGateCols * kHid;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int s = e / (kGateCols * kHid), n = (e / kHid) % kGateCols, k = e % kHid;
        const int nat = (n & 3) * kHid + (n >> 2);
        const float* src = (layer > 0 && s == 0) ? w_ih : w_hh;
        const float v = src[(int64_t)nat * kHid + k];
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
        const uint32_t off = sw128_off16((uint32_t)n, (uint32_t)k);
        *reinterpret_cast<__nv_bfloat16*>(wimg + (size_t)(s * 2) * kWTileBytes + off) = h;
        *reinterpret_cast<__nv_bfloat16*>(wimg + (size_t)(s * 2 + 1) * kWTileBytes + off) = l;
    }
    for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < kGateCols; n += gridDim.x * blockDim.x) {
        const int nat = (n & 3) * kHid + (n >> 2);
        bias[n] = b_ih[nat] + b_hh[nat];
        if (layer == 0 && wih_t != nullptr)
            for (int c = 0; c < c_in; ++c) wih_t[c * kGateCols + n] = w_ih[(int64_t)nat * c_in + c];
    }
}


// =====================================================================================================
// backward: gate recompute + BPTT pointwise + data gradient + weight gradient in ONE kernel, time-fused per layer
// (a launch = one layer x a run of timesteps, see Bwd16Params; "tile" below = one (step, tile) work item)
// =====================================================================================================
// Per 128-row tile, the 256 gate columns are processed as four chunks of 64 (16 units x i,f,g,o):
//   R_c : recompute the chunk's pre-activations  G_c[128 x 64] = [h_below | h_prev] . Wp[:, chunk]     (TMEM, 64 columns)
//   P_c : 16 compute warps: TMEM -> gates -> c_t, tanh(c_t) -> BPTT pointwise -> dA_c (fp32) -> bf16 hi/lo planes in a
//         128-byte-swizzled shared-memory tile; dc in place
//   W_c : weight gradient   dWp[:, chunk] += [h_below | h_prev]^T . dA_c   -- BOTH operands are the MN-major view of tiles
//         that are already in shared memory (the A planes, dA_c); one 256-column TMEM accumulator lives for the launch
//   D_c : data gradient     [dx_below | dh_prev] += dA_c . Wp[:, chunk]^T  -- B is the MN-major view of the weight chunk
//         R_c used; 128-column TMEM accumulator, drained by the compute warps at the start of the next tile
//   B_c : bias gradient     db[chunk] += dA_c^T . ones   -- 8 small MMAs (M = 64 hi + 64 lo columns, N = 16) on the W warp
// dA never leaves the SM; the gates are never stored.  HBM traffic per tile: A planes 64 KB + c_prev, dh_in, dh_rec, dc
// (4 x 32 KB) in, dc, dh_rec, dx_below (3 x 32 KB) out = 288 KB (the first-generation pair of kernels moved 640 KB).
// Weight chunks stream from L2 twice, into one single-buffered slot for R_c and one for D_c (see the producer).
// Partial weight gradients: every CTA adds its TMEM accumulator into its OWN slice of a scratch buffer (vector reductions,
// no contention; the slice layout is the accumulator's register layout); after the last layer, stmgcn_lstm16_bwd sums the
// slices once per layer (lstm16_wgrad_reduce_kernel) and writes nn.LSTM-native gradients.
// The kernel is bound by the L1 / shared-memory data pipe (ncu: 94 %: tensor-core operand reads 61 % + LSU 33 %).
constexpr int kBCompWarps = 16;
constexpr int kBThreads = (kBCompWarps + 2) * 32;       // + MMA-issuing warp + producer warp
constexpr int kBWStages = 2;                            // two single-buffered slots: the recompute's and the data gradient's copy
constexpr int kBWChunkTile = 64 * 128;                  // [64 gate cols][64 k] bf16 = 8 KB
constexpr int kBWStageBytes = 4 * kBWChunkTile;         // (seg0 hi | seg0 lo | seg1 hi | seg1 lo) = 32 KB
constexpr int kBSgMax = 1024;

struct B16Tail {
    uint16_t ones[1024];                       // [16][64] bf16 tile of 1.0: B operand of the bias-gradient MMA (first member:
                                               // the tail starts 1024-byte aligned, as a swizzled K-major operand must)
    float bias[kGateCols];
    float wih[kMaxC * kGateCols];
    float s_ds[kBSgMax];
    uint64_t ahi_full[2], ahi_empty[2];        // A hi planes: double-buffered by tile parity
    uint64_t alo_full, alo_empty;              // A lo planes: single buffer
    uint64_t w_full[kBWStages], w_empty[kBWStages];
    uint64_t r_full, r_empty;
    uint64_t d_full, d_empty;
    uint64_t g_full, g_empty;
    uint64_t done;
    uint32_t tmem_base;
};
constexpr int kBATiles = 6;                             // hi planes of two tiles (2 x 2 segments) + lo planes of one (2 segments)
constexpr size_t kBSmem = 1024 + kBATiles * (size_t)kATileBytes + (size_t)kBWStages * kBWStageBytes + 2 * (size_t)kATileBytes + sizeof(B16Tail);
static_assert(kBSmem <= 232448, "lstm16 backward kernel exceeds the 227 KB shared-memory limit");

// One launch = one LAYER, all timesteps T-1 .. 0 (the tiles of a CTA are its own through time: rows never mix).  A step
// of a tile needs what the SAME CTA produced for that tile one step later (dh_rec, dc: global, in place), so nothing but
// the launch order of the layers (top down) synchronises; what a per-step launch paid 36 times per branch -- prologue,
// first-tile latency, the 128 KB weight-gradient flush per CTA, the launch gap: 22 us of a 169 us launch, measured by
// scaling the row count -- is paid 3 times.
constexpr int kBMaxSteps = 64;
struct Bwd16Step {
    int32_t slice[2];          // plane slice of K segment s in its tensor map (hi plane; lo = + 1)
    int8_t src[2];             // 0: maps[0] (hp), 1: maps[1] (h0p), 2: zeros (h_prev at t = 0 without an initial state)
    int8_t first;              // t == T-1: incoming dh_rec / dc are zero and not read
    int8_t store_dh;           // write dh_prev (t > 0 or an initial state exists)
    int32_t t;
    const float* c_prev;       // blocked or nullptr (zeros)
    const float* dh_in;        // blocked or nullptr: gradient from the layer above at this step (top layer: d_top at T-1)
    float* dx_out;             // blocked or nullptr (layer 0)
};
struct Bwd16Params {
    alignas(64) CUtensorMap maps[2];
    const uint8_t* zero_tile;  // 16 KB of zeros
    const uint8_t* wimg;
    const float* bias;
    const float* wih;          // layer 0: (C,256) gate-interleaved
    const float* xo;           // (rows, T, C)
    const float* sg;           // (B, T)
    float* d_s;                // (B, T) +=   (layer 0)
    int c_in, t_len, n_steps;
    int64_t b_inner;
    float* dh_rec;             // blocked, in (unless first) / out, in place through the steps
    float* dc;                 // blocked, in (unless first) / out, in place through the steps
    float* dbp;                // (256) +=  gate-interleaved bias gradient
    float* dw_slice;           // gridDim.x slices of 128*256 floats (accumulator register layout)
    int dw_first;              // 1: first launch of this layer: slices are written, not accumulated
    int64_t rows;
    int n_tiles;
    Bwd16Step steps[kBMaxSteps];   // in execution order: steps[0] is t = T-1
};
static_assert(sizeof(Bwd16Params) <= 4096, "kernel parameter block exceeds 4 KB");

template <int PLANES, int CIN>                                  // CIN: see lstm16_fwd_kernel
__global__ void __launch_bounds__(kBThreads, 1) lstm16_bwd_kernel(const __grid_constant__ Bwd16Params p) {
    constexpr bool L0 = CIN > 0;
    constexpr int kC = (CIN == 1) ? 1 : kMaxC;
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment by pointer arithmetic on the __shared__ array (an integer round trip would make every access through
    // `smem` a generic LD/ST/ATOM instead of LDS/STS/ATOMS: ncu showed the bias loads as long-scoreboard stalls)
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    // A planes: tiles [hi buffer 0: seg0, seg1 (aux)] [hi buffer 1: seg0, seg1 (aux)] [lo: seg0, seg1 (aux)].  The hi planes
    // of the NEXT tile load while this tile is processed; the lo planes (needed by one of three passes) are single-buffered
    // and released by the FIRST pass of the tile's last weight-gradient MMA group.  Fully single-buffered planes cost the
    // compute warps 16 % of their lifetime waiting for the first recompute of every tile (role accounting, profiles/).
    uint8_t* a_sm = smem;
    uint8_t* w_sm = a_sm + kBATiles * (size_t)kATileBytes;         // weight chunk ring
    uint8_t* da_sm = w_sm + (size_t)kBWStages * kBWStageBytes;     // dA chunk: hi tile | lo tile
    B16Tail* tail = (B16Tail*)(da_sm + 2 * (size_t)kATileBytes);
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;
    constexpr int kMmaWarp = kBCompWarps;
    constexpr int kProdWarp = kBCompWarps + 1;
    // TMEM columns: weight grad (256) | data grad (128) | recompute (64, single buffer: the compute warps hold it only for
    // the TMEM -> register copy at the start of a chunk) | bias grad (4 chunks x 16)
    constexpr uint32_t kWgCol = 0, kDgCol = 256, kRcCol = 384, kDbCol = 448;

    if (tid == 0) {
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tail->ahi_full[b], 1);
            mbar_init(&tail->ahi_empty[b], 1);
        }
        mbar_init(&tail->alo_full, 1);
        mbar_init(&tail->alo_empty, 1);
        for (int s = 0; s < kBWStages; ++s) {
            mbar_init(&tail->w_full[s], 1);
            mbar_init(&tail->w_empty[s], 1);
        }
        mbar_init(&tail->r_full, 1);
        mbar_init(&tail->r_empty, kBCompWarps);                // one arrival per compute warp
        mbar_init(&tail->d_full, kBCompWarps);
        mbar_init(&tail->d_empty, 1);
        mbar_init(&tail->g_full, 1);
        mbar_init(&tail->g_empty, kBCompWarps);
        mbar_init(&tail->done, 1);
        fence_barrier_init();
    }
    if (warp == kMmaWarp) tmem_alloc(&tail->tmem_base, 512);
    for (int i = tid; i < kGateCols; i += kBThreads) tail->bias[i] = p.bias[i] * gate_scale(i);
    for (int i = tid; i < 1024; i += kBThreads) tail->ones[i] = 0x3f80u;           // bf16 1.0 (layout-invariant)
    if (L0) {
        for (int i = tid; i < p.c_in * kGateCols; i += kBThreads) tail->wih[i] = p.wih[i] * gate_scale(i);
        for (int i = tid; i < kBSgMax; i += kBThreads) tail->s_ds[i] = 0.f;
    }
    fence_proxy_async_smem();                   // the ones tile is read by the tensor pipe (async proxy)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tail->tmem_base;
    const int my_tiles = (p.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const bool have_aux = L0;
    // K segments of the gate GEMM: layers > 0: [h_below | h_prev]; layer 0: [h_prev] (at t = 0 without an initial state the
    // h_prev tiles are loaded as zeros: every step of a layer has the same operand geometry and accumulates into the same
    // weight-gradient rows)
    constexpr int kNseg = L0 ? 1 : 2;
    const int n_items = my_tiles * p.n_steps;                      // work items (step, tile), step-major
    // operand tiles of the weight-gradient GEMM (MN-major view): atom 0 and atom 1 along M = kd
    // layers > 0: atom 0 = h_below, atom 1 = h_prev;  layer 0: atom 0 = h_prev, atom 1 = auxiliary [x*s] tile
    constexpr uint32_t wg_a0 = 0u;                                 // segment slot of atom 0
    constexpr uint32_t wg_lbo = kATileBytes;

    if (warp == kProdWarp) {
        // ===================== producer =====================
        TC_PROF_DECL
        const bool leader = elect_one_sync();
        if (leader && n_items > 0) {
            const int first = (int)blockIdx.x, gstep = (int)gridDim.x;
            // work item w = (step w / my_tiles, tile first + (w % my_tiles) * gstep)
            auto seg_load = [&](uint8_t* dst, const Bwd16Step& sp, int sg, int plane, int tile, uint64_t* bar) {
                if (sp.src[sg] == 2) bulk_g2s(dst, p.zero_tile, kATileBytes, bar);
                else tma_load_3d(dst, &p.maps[sp.src[sg]], 0, tile * kTileM, sp.slice[sg] + plane, bar);
            };
            auto load_hi = [&](int w) {                 // hi planes of item w -> hi buffer w & 1
                const int b = w & 1;
                const int st = w / my_tiles, tile = first + (w - st * my_tiles) * gstep;
                const Bwd16Step& sp = p.steps[st];
                if (w >= 2) mbar_wait_p(&tail->ahi_empty[b], (uint32_t)((w >> 1) - 1) & 1, 1);
                mbar_arrive_expect_tx(&tail->ahi_full[b], (uint32_t)(kNseg * kATileBytes));
                for (int sg = 0; sg < kNseg; ++sg)
                    seg_load(a_sm + (size_t)(b * 2 + sg) * kATileBytes, sp, sg, 0, tile, &tail->ahi_full[b]);
            };
            auto load_lo = [&](int w) {                 // lo planes of item w -> the single lo buffer
                const int st = w / my_tiles, tile = first + (w - st * my_tiles) * gstep;
                const Bwd16Step& sp = p.steps[st];
                if (w >= 1) mbar_wait_p(&tail->alo_empty, (uint32_t)(w - 1) & 1, 1);
                mbar_arrive_expect_tx(&tail->alo_full, (uint32_t)(kNseg * kATileBytes));
                for (int sg = 0; sg < kNseg; ++sg)
                    seg_load(a_sm + (size_t)(4 + sg) * kATileBytes, sp, sg, 1, tile, &tail->alo_full);
            };
            auto load_w = [&](int stg, uint32_t wc) {   // weight chunk wc & 3 -> buffer stg (0: the recompute's copy, 1: the
                const int c = wc & 3;                   // data gradient's copy); use wc of a buffer waits for release wc - 1
                mbar_wait_p(&tail->w_empty[stg], (wc & 1) ^ 1, 0);
                mbar_arrive_expect_tx(&tail->w_full[stg], (uint32_t)(kNseg * PLANES * kBWChunkTile));
                for (int sg = 0; sg < kNseg; ++sg)
                    for (int pl = 0; pl < PLANES; ++pl)
                        bulk_g2s(w_sm + (size_t)stg * kBWStageBytes + (size_t)(sg * 2 + pl) * kBWChunkTile,
                                 p.wimg + (size_t)(sg * 2 + pl) * kWTileBytes + (size_t)c * kBWChunkTile, kBWChunkTile, &tail->w_full[stg]);
            };
            auto prefetch_next = [&](int w) {           // item w's lo planes and per-row inputs -> L2
                const int st = w / my_tiles, tile = first + (w - st * my_tiles) * gstep;
                const Bwd16Step& sp = p.steps[st];
                if (PLANES == 2)
                    for (int sg = 0; sg < kNseg; ++sg)
                        if (sp.src[sg] != 2) tma_prefetch_3d(&p.maps[sp.src[sg]], 0, tile * kTileM, sp.slice[sg] + 1);
                // the compute warps' per-row inputs (a tile is one contiguous 32 KB run in every workspace): their
                // one-chunk-ahead register prefetch then costs an L2 hit, not a DRAM round trip
                const int64_t o = (int64_t)tile * kTileM * kHid;
                constexpr uint32_t kB = kTileM * kHid * 4;
                if (sp.c_prev) prefetch_l2(sp.c_prev + o, kB);
                if (sp.dh_in) prefetch_l2(sp.dh_in + o, kB);
                if (!sp.first && my_tiles > 2) {         // (written by this CTA more than a tile-time ago)
                    prefetch_l2(p.dh_rec + o, kB);
                    prefetch_l2(p.dc + o, kB);
                }
            };
            // Every weight chunk is loaded TWICE (L2 hits), into two single-buffered slots: one copy for the recompute R_c, one
            // for the data gradient D_c.  With one shared ring a stage was held from R_c until D_c (a whole chunk-time later), so
            // R_{c+2} had to wait for D_c + a reload + its own MMAs inside one chunk-time: the recompute warp spent 40 % of its
            // life waiting for weights and the compute warps 11 % waiting for the recompute.  Now R_{c+1} only needs the compute
            // warps to have copied G_c out of TMEM.
            // Flat schedule: every wait below is on an event that lies in the PAST of what the consumers need next, in time
            // order: R(g+2) is released at the start of chunk-time g+1, D(g+1)'s buffer at the end of chunk-time g.
            load_hi(0);
            if (PLANES == 2) load_lo(0);
            load_w(0, 0);
            load_w(1, 0);
            load_w(0, 1);
            for (int i = 0; i < n_items; ++i) {
                const bool more = i + 1 < n_items;
                const uint32_t g0 = 4u * (uint32_t)i;
                if (more) {
                    load_hi(i + 1);
                    prefetch_next(i + 1);
                }
                load_w(0, g0 + 2);
                load_w(1, g0 + 1);
                load_w(0, g0 + 3);
                load_w(1, g0 + 2);
                if (more) load_w(0, g0 + 4);
                load_w(1, g0 + 3);
                if (more) {
                    if (PLANES == 2) load_lo(i + 1);
                    load_w(0, g0 + 5);
                    load_w(1, g0 + 4);
                }
            }
        }
        TC_PROF_FLUSH(5, leader)
    } else if (warp == kMmaWarp) {
        // ===================== the MMA issuer: recompute (R) | weight gradient (W) | bias gradient | data gradient (D) =====================
        // ONE thread issues every tcgen05.mma of the CTA, in the order the work becomes ready:
        //     R_{g+1} (hi passes [+ lo pass])  ->  W_g lo pass, D_g, W_g hi passes, bias gradient  ->  [tile boundary: R_{g+1} lo pass]
        // R_{g+1} is released when the compute warps have copied G_g out of TMEM (start of chunk-time g), W_g / D_g when dA_g is in
        // shared memory (its end).  (An earlier version used three issuing warps because an issue cost ~90 cycles -- that was the
        // ELECT / BRA.U.ANY loop ptxas wraps around `lane == 0`-guarded UTCHMMAs, gone with elect.sync.)  A single in-order issuer
        // is what makes the A-operand collector usable: in the 3xBF16 scheme the products A_hi.B_hi and A_hi.B_lo share A, so
        // the second MMA of each pair takes A from the tensor core's collector buffer instead of re-reading 4 KB of shared memory
        // -- the kernel is bound by the shared-memory data pipe (ncu: 94 %, 61 % of it tensor-core operand reads).
        // Everything that does not change is hoisted into 64-bit descriptor constants; a k-step is one add on the descriptor's
        // address field (encoded address = bytes >> 4; all operands live below 256 KB: no carry).
        TC_PROF_DECL
        const bool leader = elect_one_sync();
        constexpr uint32_t idesc_rc = idesc_bf16(kTileM, 64);              // recompute: A K-major, B K-major, N = 64
        constexpr uint32_t idesc_wg = idesc_bf16(kTileM, 64, 1, 1);        // weight gradient: both MN-major, M = kd (128), N = 64
        constexpr uint32_t idesc_db = idesc_bf16(kTileM, 16, 1, 0);        // bias gradient: A = dA^T (hi | lo atoms), B = ones
        constexpr uint32_t idesc_dg = idesc_bf16(kTileM, 64 * kNseg, 0, 1);   // data gradient: B MN-major, N = 64 * nseg
        const uint32_t a_u = smem_u32(a_sm), w_u = smem_u32(w_sm), da_u = smem_u32(da_sm);
        constexpr uint64_t kStepK = 2;                                     // K-major: 16 bf16 = 32 bytes
        constexpr uint64_t kStepMN = 2048 >> 4;                            // MN-major: 16 rows of 128 bytes
        constexpr uint64_t kTileEnc = kATileBytes >> 4, kChunkEnc = kBWChunkTile >> 4, kStageEnc = kBWStageBytes >> 4;
        constexpr int nseg = kNseg;
        const uint64_t rc_a = desc16_k(a_u);                               // hi: + (buffer*2 + s) * kTileEnc; lo: + (4 + s) * kTileEnc
        const uint64_t rc_b = desc16_k(w_u);                               // buffer 0 (the recompute's copy): + (s*2 + plane) * kChunkEnc
        const uint64_t wg_hi0 = desc16_mn(a_u + wg_a0 * kATileBytes, wg_lbo);              // hi buffer 0; buffer 1: + 2 * kTileEnc
        const uint64_t wg_lo = desc16_mn(a_u + (4 + wg_a0) * kATileBytes, wg_lbo);         // lo planes
        const uint64_t wg_b = desc16_mn(da_u, kATileBytes);                                  // dA hi; lo: + kTileEnc
        const uint64_t db_b = desc16_k(smem_u32(tail->ones));
        const uint64_t dg_a = desc16_k(da_u);                              // dA hi; lo: + kTileEnc
        const uint64_t dg_b = desc16_mn(w_u, 2 * kBWChunkTile) + kStageEnc;   // buffer 1 (the data gradient's copy) (+ kChunkEnc: lo plane)
        const uint32_t t_rc = tmem_base + kRcCol, t_wg = tmem_base + kWgCol, t_db = tmem_base + kDbCol, t_dg = tmem_base + kDgCol;
        const bool a_sync = nseg > 0 || L0;          // someone waits for the A buffers (producer and / or the aux-tile writers)
        const uint32_t total = 4u * (uint32_t)n_items;    // chunks; "tile" below = work item (step, tile): the hand-offs do
                                                          // not care which timestep an item belongs to

        // hi-plane passes of the recompute of chunk wc (tile wc >> 2): G = A_hi . (W_hi + W_lo)
        auto issue_r_hi = [&](uint32_t wc) {
            const int ab = (int)((wc >> 2) & 1);
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                if (s < nseg) {
                    const uint64_t a_hi = rc_a + (uint64_t)(ab * 2 + s) * kTileEnc;
                    const uint64_t b_hi = rc_b + (uint64_t)(s * 2) * kChunkEnc, b_lo = b_hi + kChunkEnc;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const uint32_t acc = (s > 0 || kk > 0) ? 1u : 0u;
                        if (PLANES == 2) {
                            mma_bf16_keep_a(t_rc, a_hi + kk * kStepK, b_hi + kk * kStepK, idesc_rc, acc);
                            mma_bf16_reuse_a(t_rc, a_hi + kk * kStepK, b_lo + kk * kStepK, idesc_rc, 1u);
                        } else {
                            mma_bf16(t_rc, a_hi + kk * kStepK, b_hi + kk * kStepK, idesc_rc, acc);
                        }
                    }
                }
            }
        };
        // lo-plane pass (PLANES == 2): G += A_lo . W_hi; then the chunk's weight slot and the accumulator are handed over
        auto issue_r_lo_and_commit = [&]() {
            if (PLANES == 2) {
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                    if (s < nseg) {
                        const uint64_t a_lo = rc_a + (uint64_t)(4 + s) * kTileEnc;
                        const uint64_t b_hi = rc_b + (uint64_t)(s * 2) * kChunkEnc;
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) mma_bf16(t_rc, a_lo + kk * kStepK, b_hi + kk * kStepK, idesc_rc, 1u);
                    }
                }
            }
            mma_commit(&tail->w_empty[0]);
            mma_commit(&tail->r_full);
        };

        if (n_items > 0) {                           // R_0
            mbar_wait_p(&tail->ahi_full[0], 0, 3);
            mbar_wait_p(&tail->w_full[0], 0, 0);
            if (PLANES == 2) mbar_wait_p(&tail->alo_full, 0, 3);
            tc_fence_after();
            if (leader) {
                issue_r_hi(0);
                issue_r_lo_and_commit();
            }
            __syncwarp();
        }
        for (uint32_t g = 0; g < total; ++g) {
            const int i = (int)(g >> 2), c = (int)(g & 3);
            const bool have_next = nseg > 0 && g + 1 < total;
            // ---- (1) recompute of the next chunk ----
            if (have_next) {
                const uint32_t wc = g + 1;
                mbar_wait_p(&tail->w_full[0], wc & 1, 0);
                if (c == 3) mbar_wait_p(&tail->ahi_full[(i + 1) & 1], (uint32_t)((i + 1) >> 1) & 1, 3);
                mbar_wait_p(&tail->r_empty, (wc & 1) ^ 1, 2);
                tc_fence_after();
                if (leader) {
                    issue_r_hi(wc);
                    if (c != 3) issue_r_lo_and_commit();         // (c == 3: the next tile's lo planes land after W_g's lo pass)
                }
                __syncwarp();
            }
            // ---- (2) dA_g is in shared memory: weight gradient, data gradient, bias gradient ----
            if (nseg > 0) mbar_wait_p(&tail->w_full[1], g & 1, 0);
            mbar_wait_p(&tail->d_full, g & 1, 1);
            if (c == 0 && nseg > 0 && i > 0) mbar_wait_p(&tail->g_empty, (uint32_t)(i - 1) & 1, 2);
            tc_fence_after();
            if (leader) {
                const uint64_t wg_hi = wg_hi0 + (uint64_t)((i & 1) * 2) * kTileEnc;
                const uint32_t d_wg = t_wg + (uint32_t)c * 64;
                const uint32_t acc0 = (i > 0) ? 1u : 0u;
                if (PLANES == 2) {                   // W_g, lo-plane pass first: the tile's last one releases the single lo buffer a.s.a.p.
                    mma_bf16(d_wg, wg_lo, wg_b, idesc_wg, acc0);
#pragma unroll
                    for (int ks = 1; ks < 8; ++ks) mma_bf16(d_wg, wg_lo + ks * kStepMN, wg_b + ks * kStepMN, idesc_wg, 1u);
                    if (c == 3 && a_sync) mma_commit(&tail->alo_empty);
                }
                if (nseg > 0) {                      // D_g: [dx_below | dh_prev] += (dA_hi + dA_lo) . W_hi^T + dA_hi . W_lo^T
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const uint32_t acc = (c > 0 || kk > 0) ? 1u : 0u;
                        if (PLANES == 2) {
                            mma_bf16_keep_a(t_dg, dg_a + kk * kStepK, dg_b + kk * kStepMN, idesc_dg, acc);
                            mma_bf16_reuse_a(t_dg, dg_a + kk * kStepK, dg_b + kChunkEnc + kk * kStepMN, idesc_dg, 1u);
                        } else {
                            mma_bf16(t_dg, dg_a + kk * kStepK, dg_b + kk * kStepMN, idesc_dg, acc);
                        }
                    }
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)                       // dA lo plane: always (it never leaves the SM)
                        mma_bf16(t_dg, dg_a + kTileEnc + kk * kStepK, dg_b + kk * kStepMN, idesc_dg, 1u);
                    mma_commit(&tail->w_empty[1]);
                    if (c == 3) mma_commit(&tail->g_full);
                }
                // W_g, hi planes: A_hi^T . (dA_hi + dA_lo); dA always has its lo plane: in the single-plane (bf16 storage) mode
                // only the STORED operands are rounded to bf16
#pragma unroll
                for (int ks = 0; ks < 8; ++ks) {
                    mma_bf16_keep_a(d_wg, wg_hi + ks * kStepMN, wg_b + ks * kStepMN, idesc_wg, (PLANES == 2 || ks > 0) ? 1u : acc0);
                    mma_bf16_reuse_a(d_wg, wg_hi + ks * kStepMN, wg_b + kTileEnc + ks * kStepMN, idesc_wg, 1u);
                }
                if (c == 3 && a_sync) mma_commit(&tail->ahi_empty[i & 1]);       // this tile's hi buffer may be refilled
                // bias gradient on the tensor pipe: D[128 x 16] += dA_c^T (MN-major A, M = 64 columns of the hi plane | 64 of the
                // lo plane: the two planes are the two 64-element atoms, LBO = one tile) . ones[K = 16 rows][16].  Lane m < 64 of
                // the accumulator holds sum_rows hi(dA)[:, m], lane 64 + m the lo plane's sum; all 16 columns are equal.
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)
                    mma_bf16(t_db + (uint32_t)c * 16, wg_b + ks * kStepMN, db_b, idesc_db, (i > 0 || ks > 0) ? 1u : 0u);
                mma_commit(&tail->d_empty);
            }
            __syncwarp();
            // ---- (3) tile boundary: the next tile's lo planes were requested when W_g's lo pass released the buffer ----
            if (have_next && c == 3) {
                if (PLANES == 2) {
                    mbar_wait_p(&tail->alo_full, (uint32_t)(i + 1) & 1, 3);
                    tc_fence_after();
                }
                if (leader) issue_r_lo_and_commit();
                __syncwarp();
            }
        }
        if (leader && n_items > 0) mma_commit(&tail->done);
        __syncwarp();
        TC_PROF_FLUSH(4, leader)
    } else {
        // ===================== compute warps =====================
        TC_PROF_DECL
        // TMEM lane quadrant q = warp & 3 (row 32q + lane of the tile), part = warp >> 2: units 4*part .. +3 of every chunk
        const int q = warp & 3, part = warp >> 2;
        const int ctid = tid;
        (void)ctid;
        float xs[kMaxC], xraw[kMaxC], dxs[kMaxC];
        uint32_t dcount = 0, rcount = 0;
        // raw inputs of one chunk: c_prev, dh_in, dh_rec, dc of this thread's 4 units
        struct Raw { float4 cp, dhi, dhr, dcv; };
        // tile-blocked workspaces: element (tile, row, unit) at tile*8192 + (unit/4)*512 + row*4 + unit%4
        const uint32_t row_in_tile = (uint32_t)(q * 32 + lane);
        const uint32_t rows32 = (uint32_t)p.rows;       // (rows <= 2^25 is checked on the host: 32-bit element offsets)
        const uint32_t thr_off = row_in_tile * 4u + (uint32_t)part * 512u;
        float xraw_next[kMaxC], sv_next = 0.f;      // layer 0: x and gate value of the next tile, loaded a chunk ahead
        // layer 0: when b_inner divides the tile height, a thread's row belongs to the same window b in every tile: its share
        // of d_s is summed in a register and added once (one shared-memory float atomic = a CAS loop; 16 per address and tile
        // were 6 % of the layer-0 kernel's stall samples)
        const bool ds_fixed = L0 && (kTileM % (uint32_t)p.b_inner) == 0u;
        const bool ds_smem = L0 && (int64_t)p.n_steps * p.b_inner <= kBSgMax;    // s_ds holds [step][window]
        float ds_acc = 0.f;
        // (st, tile): step index and tile of a work item; a step index >= n_steps marks "no such item"
        auto load_x = [&](int st, int tile_n) {
            const uint32_t rn = (uint32_t)tile_n * kTileM + row_in_tile;
            const bool ok = st < p.n_steps && rn < rows32;
            const uint32_t t = ok ? (uint32_t)p.steps[st].t : 0u;
            sv_next = 0.f;
            if (ok) sv_next = p.sg[(rn % (uint32_t)p.b_inner) * (uint32_t)p.t_len + t];      // (32-bit: a 64-bit % is a call)
#pragma unroll
            for (int c = 0; c < kMaxC; ++c)
                xraw_next[c] = (c < kC && ok && (CIN == 1 || c < p.c_in)) ? p.xo[((int64_t)rn * p.t_len + t) * p.c_in + c] : 0.f;
        };
        auto load_raw = [&](int st, int tile, int c, Raw& rw) {
            const uint32_t r = (uint32_t)tile * kTileM + row_in_tile;
            const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
            rw.cp = rw.dhi = rw.dhr = rw.dcv = z;
            if (st < p.n_steps && r < rows32) {
                const Bwd16Step& sp = p.steps[st];
                const uint32_t o = (uint32_t)tile * 8192u + (uint32_t)c * 2048u + thr_off;
                if (sp.c_prev) rw.cp = *reinterpret_cast<const float4*>(sp.c_prev + o);
                if (sp.dh_in) rw.dhi = *reinterpret_cast<const float4*>(sp.dh_in + o);
                if (!sp.first) {
                    rw.dhr = *reinterpret_cast<const float4*>(p.dh_rec + o);
                    rw.dcv = *reinterpret_cast<const float4*>(p.dc + o);
                }
            }
        };
        // [dx_below | dh_prev] of work item w_prev (step st_prev, tile tile_prev): TMEM -> tile-blocked workspaces
        auto drain = [&](int w_prev, int st_prev, int tile_prev) {
            const uint32_t r = (uint32_t)tile_prev * kTileM + row_in_tile;
            const Bwd16Step& sp = p.steps[st_prev];
            mbar_wait(&tail->g_full, (uint32_t)w_prev & 1, 2);
            tc_fence_after();
            constexpr int ncols = 64 * kNseg;
            if (part * 32 < ncols) {
                uint32_t v[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + kDgCol + (uint32_t)part * 32, v);
                tmem_ld_wait();
                const int col = part * 32;
                // layers > 0: columns [0,64) = dx_below, [64,128) = dh_prev; layer 0: [0,64) = dh_prev
                const bool is_dx = !L0 && col < 64;
                float* base = is_dx ? sp.dx_out : p.dh_rec;
                const int unit0 = col & 63;
                if (r < rows32 && base != nullptr && (is_dx || sp.store_dh)) {
                    const uint32_t o = (uint32_t)tile_prev * 8192u + row_in_tile * 4u + (uint32_t)(unit0 >> 2) * 512u;
#pragma unroll
                    for (int k = 0; k < 8; ++k)          // units unit0 + 4k .. +3: the warp writes one contiguous 512-byte run
                        *reinterpret_cast<uint4*>(base + (o + (uint32_t)k * 512u)) = make_uint4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tail->g_empty);
        };
        Raw cur, nxt;              // (measured and rejected: loading two chunks ahead -- the 16 extra registers at the 96-register
                                   //  cap cost more than the covered latency gained: 8.43 -> 8.68 ms per branch)
        const int gstep = (int)gridDim.x;
        // work items in step-major order: (st, i) = (step index, this CTA's i-th tile); (st_n, tile_n) = the item after it
        int st = 0, i = 0, tile = (int)blockIdx.x;
        if (n_items == 0) st = p.n_steps;
        load_raw(st, tile, 0, nxt);
        if (L0) load_x(st, tile);
        for (int w = 0; w < n_items; ++w) {
            const bool last_of_step = (i + 1 == my_tiles);
            const int st_n = last_of_step ? st + 1 : st;
            const int tile_n = last_of_step ? (int)blockIdx.x : tile + gstep;
            const int st_p = (i == 0) ? st - 1 : st;                                   // the item before this one
            const int tile_p = (i == 0) ? (int)blockIdx.x + (my_tiles - 1) * gstep : tile - gstep;
            const Bwd16Step& sp = p.steps[st];
            const uint32_t r = (uint32_t)tile * kTileM + row_in_tile;
            const bool valid = r < rows32;
            if (L0) {
#pragma unroll
                for (int c = 0; c < kMaxC; ++c) {
                    xraw[c] = xraw_next[c];
                    xs[c] = xraw[c] * sv_next;
                    dxs[c] = 0.f;
                }
            }
            // (the drain sits in the tile-boundary bubble: the first recompute of this tile cannot finish before the lo planes
            // have been reloaded; moved behind chunk 0 it cost 2.3 k cycles of real time per tile, measured)
            if (w > 0) drain(w - 1, st_p, tile_p);
            if (i == 0 && w > 0) {
                // step boundary: this step reads the dh_rec the CTA's own drains wrote during the previous step (other threads'
                // stores): a barrier of the 512 compute threads orders them, and the first chunk's inputs -- not prefetched
                // across the boundary (with one tile per CTA they did not exist yet) -- are loaded behind it
                asm volatile("bar.sync 1, %0;" ::"n"(kBCompWarps * 32) : "memory");
                load_raw(st, tile, 0, nxt);
            }
            if (have_aux && part == 0) {
                // auxiliary weight-gradient operand: the seg-1 slot of this tile's hi buffer and of the lo buffer; row = this
                // thread's row, columns 0..C-1 = x*s (hi / lo split)
                if (w >= 2) mbar_wait(&tail->ahi_empty[w & 1], (uint32_t)((w >> 1) - 1) & 1, 3);
                uint32_t hi[2], lo[2];
                split_bf16x2(xs[0], xs[1], hi[0], lo[0]);
                split_bf16x2(xs[2], xs[3], hi[1], lo[1]);
                const uint32_t row = (uint32_t)(q * 32 + lane);
                const uint32_t off = row * 128u + ((0u ^ (row & 7u)) << 4);
                *reinterpret_cast<uint4*>(a_sm + (size_t)((w & 1) * 2 + 1) * kATileBytes + off) = make_uint4(hi[0], hi[1], 0u, 0u);
                if (PLANES == 2) {
                    if (w >= 1) mbar_wait(&tail->alo_empty, (uint32_t)(w - 1) & 1, 3);
                    *reinterpret_cast<uint4*>(a_sm + (size_t)5 * kATileBytes + off) = make_uint4(lo[0], lo[1], 0u, 0u);
                }
            }
            for (int c = 0; c < 4; ++c, ++dcount) {
                cur = nxt;
                uint32_t v[16];
                {
                    mbar_wait(&tail->r_full, rcount & 1, c == 0 ? 3 : 1);      // (profile builds: class 3 = first chunk of a tile)
                    tc_fence_after();
                    tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + kRcCol + (uint32_t)part * 16, v);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tail->r_empty);
                    ++rcount;
                }
                const int unit0 = 16 * c + 4 * part;
                const float cp[4] = {cur.cp.x, cur.cp.y, cur.cp.z, cur.cp.w};
                const float dhi[4] = {cur.dhi.x, cur.dhi.y, cur.dhi.z, cur.dhi.w};
                const float dhr[4] = {cur.dhr.x, cur.dhr.y, cur.dhr.z, cur.dhr.w};
                const float dci[4] = {cur.dcv.x, cur.dcv.y, cur.dcv.z, cur.dcv.w};
                float da[16], dcn[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int col = 4 * (unit0 + u);
                    const float4 bv = *reinterpret_cast<const float4*>(&tail->bias[col]);      // pre-scaled (gate_scale)
                    float pi = fmaf(__uint_as_float(v[4 * u + 0]), -1.4426950408889634f, bv.x);
                    float pf = fmaf(__uint_as_float(v[4 * u + 1]), -1.4426950408889634f, bv.y);
                    float pg = fmaf(__uint_as_float(v[4 * u + 2]), -2.8853900817779268f, bv.z);
                    float po = fmaf(__uint_as_float(v[4 * u + 3]), -1.4426950408889634f, bv.w);
                    if (L0) {
#pragma unroll
                        for (int cc = 0; cc < kC; ++cc)
                            if (CIN == 1 || cc < p.c_in) {
                                const float4 wv = *reinterpret_cast<const float4*>(&tail->wih[cc * kGateCols + col]);
                                pi = fmaf(xs[cc], wv.x, pi); pf = fmaf(xs[cc], wv.y, pf);
                                pg = fmaf(xs[cc], wv.z, pg); po = fmaf(xs[cc], wv.w, po);
                            }
                    }
                    float gi, gf, gg, go, tc_;
                    lstm_cell_gates8(pi, pf, pg, po, cp[u], gi, gf, gg, go, tc_);
                    // rows past the end: load_raw returned zeros for dh_rec / dh_in / dc, so dh = dcv = 0 and dA = 0 without selects
                    const float dh = dhr[u] + dhi[u];
                    const float dcv = fmaf(dh * go, 1.f - tc_ * tc_, dci[u]);
                    da[4 * u + 0] = dcv * gg * gi * (1.f - gi);
                    da[4 * u + 1] = dcv * cp[u] * gf * (1.f - gf);
                    da[4 * u + 2] = dcv * gi * (1.f - gg * gg);
                    da[4 * u + 3] = dh * tc_ * go * (1.f - go);
                    dcn[u] = dcv * gf;
                    if (L0) {
#pragma unroll
                        for (int cc = 0; cc < kC; ++cc)
                            if (CIN == 1 || cc < p.c_in) {
                                // W_ih is stored pre-scaled: undo -log2(e) (and the g gate's extra factor 2)
                                const float4 wv = *reinterpret_cast<const float4*>(&tail->wih[cc * kGateCols + col]);
                                dxs[cc] = fmaf(da[4 * u] * wv.x + da[4 * u + 1] * wv.y + 0.5f * (da[4 * u + 2] * wv.z) + da[4 * u + 3] * wv.w,
                                               -0.6931471805599453f, dxs[cc]);
                            }
                    }
                }
                // dA chunk -> bf16 planes, 128-byte-swizzled tile: row = this thread's row, columns 16*part .. +15
                uint32_t hi[8], lo[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) split_bf16x2(da[2 * j], da[2 * j + 1], hi[j], lo[j]);
                if (dcount > 0) mbar_wait(&tail->d_empty, (dcount - 1) & 1, 0);     // W_{c-1}, D_{c-1} have read the dA tile
                {
                    const uint32_t row = (uint32_t)(q * 32 + lane);
                    const uint32_t o0 = row * 128u + ((((uint32_t)(2 * part)) ^ (row & 7u)) << 4);
                    const uint32_t o1 = row * 128u + ((((uint32_t)(2 * part + 1)) ^ (row & 7u)) << 4);
                    *reinterpret_cast<uint4*>(da_sm + o0) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<uint4*>(da_sm + o1) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
                    *reinterpret_cast<uint4*>(da_sm + kATileBytes + o0) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                    *reinterpret_cast<uint4*>(da_sm + kATileBytes + o1) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tail->d_full);
                // next chunk's inputs: issued AFTER the proxy fence -- fence.proxy.async implies MEMBAR.ALL.CTA, which waits for
                // every outstanding load of the thread, so a prefetch issued before it is simply waited for at the fence
                if (c < 3) load_raw(st, tile, c + 1, nxt);
                else {
                    // (across a step boundary the first chunk is loaded behind the step's barrier, see above)
                    if (!last_of_step) load_raw(st_n, tile_n, 0, nxt);
                    if (L0) load_x(st_n, tile_n);
                }
                if (valid)
                    *reinterpret_cast<float4*>(p.dc + ((uint32_t)tile * 8192u + (uint32_t)c * 2048u + thr_off)) =
                        make_float4(dcn[0], dcn[1], dcn[2], dcn[3]);
            }
            if (L0 && valid) {
                // gate adjoint: d s[b, t] += sum_c dxmod[r, c] * xo[r, t, c]   (STMGCN.py:44)
                float contrib = 0.f;
#pragma unroll
                for (int cc = 0; cc < kC; ++cc) contrib += dxs[cc] * xraw[cc];
                if (ds_fixed) {
                    ds_acc += contrib;
                } else {
                    const int64_t b = (int64_t)(r % (uint32_t)p.b_inner);
                    if (ds_smem) atomicAdd(&tail->s_ds[(int64_t)st * p.b_inner + b], contrib);
                    else atomicAdd(&p.d_s[b * p.t_len + sp.t], contrib);
                }
            }
            if (L0 && ds_fixed && last_of_step) {       // this thread's share of d_s[b, t] for the step that ends here
                const int64_t b = (int64_t)(row_in_tile % (uint32_t)p.b_inner);
                if (ds_smem) atomicAdd(&tail->s_ds[(int64_t)st * p.b_inner + b], ds_acc);
                else atomicAdd(&p.d_s[b * p.t_len + sp.t], ds_acc);
                ds_acc = 0.f;
            }
            // next work item
            if (last_of_step) { st = st + 1; i = 0; tile = (int)blockIdx.x; }
            else { ++i; tile += gstep; }
        }
        if (n_items > 0) drain(n_items - 1, p.n_steps - 1, (int)blockIdx.x + (my_tiles - 1) * gstep);
        TC_PROF_FLUSH(3, tid == 0)
        // ---- weight-gradient accumulator -> this CTA's scratch slice (register layout: [part][piece][vec][row m][4]) ----
        if (n_items > 0) {
            mbar_wait_raw(&tail->done, 0);
            tc_fence_after();
            float* slice = p.dw_slice + (size_t)blockIdx.x * (kTileM * kGateCols);
            const int m = q * 32 + lane;
            if (part == 0) {                       // bias gradient: lanes [0,64) hold the hi-plane sums, [64,128) the lo-plane sums
                uint32_t v[16];
#pragma unroll 1
                for (int c = 0; c < 4; ++c) {
                    tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + kDbCol + (uint32_t)c * 16, v);
                    tmem_ld_wait();
                    atomicAdd(&p.dbp[64 * c + (m & 63)], __uint_as_float(v[0]));
                }
            }
#pragma unroll 1
            for (int j = 0; j < 4; ++j) {
                uint32_t v[16];
                tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + kWgCol + (uint32_t)part * 64 + (uint32_t)j * 16, v);
                tmem_ld_wait();
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    float4* dst = reinterpret_cast<float4*>(slice + ((size_t)((part * 4 + j) * 4 + e) * kTileM + m) * 4);
                    float4 acc = make_float4(__uint_as_float(v[4 * e]), __uint_as_float(v[4 * e + 1]), __uint_as_float(v[4 * e + 2]),
                                             __uint_as_float(v[4 * e + 3]));
                    // later launches of the layer add with a fire-and-forget vector reduction (the slice is private to this
                    // CTA: no contention, no read latency at the end of the launch)
                    if (p.dw_first) *dst = acc;
                    else red_add_f32x4(dst, acc);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == kMmaWarp) tmem_dealloc(tmem_base, 512);
    if (L0 && (int64_t)p.n_steps * p.b_inner <= kBSgMax)
        for (int e = tid; e < p.n_steps * (int)p.b_inner; e += kBThreads) {
            const int st = e / (int)p.b_inner, b = e - st * (int)p.b_inner;
            atomicAdd(&p.d_s[(int64_t)b * p.t_len + p.steps[st].t], tail->s_ds[e]);
        }
}

// Sum the per-CTA weight-gradient slices of one layer and write nn.LSTM-native gradients:
//   d_w_ih (256, in), d_w_hh (256, 64), d_b_ih = d_b_hh (256); native row of gate-interleaved column n: (n & 3) * 64 + (n >> 2).
// Accumulator row m = kd index: layers > 0: m < 64 -> W_ih[:, m], m >= 64 -> W_hh[:, m - 64]; layer 0: m < 64 -> W_hh[:, m],
// m = 64 + c -> W_ih[:, c].
__global__ void lstm16_wgrad_reduce_kernel(const float* __restrict__ slices, int n_slices, int layer, int c_in,
                                           const float* __restrict__ dbp, float* __restrict__ d_w_ih,
                                           float* __restrict__ d_w_hh, float* __restrict__ d_b_ih, float* __restrict__ d_b_hh) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;           // index in the slice layout
    if (e < kTileM * kGateCols) {
        float s = 0.f;
        for (int i = 0; i < n_slices; ++i) s += slices[(size_t)i * (kTileM * kGateCols) + e];
        const int x = e & 3, m = (e >> 2) & 127, rest = e >> 9;    // rest = (part*4 + j)*4 + vec
        const int n = (rest >> 2) * 16 + (rest & 3) * 4 + x;       // gate-interleaved column
        const int nat = (n & 3) * kHid + (n >> 2);
        if (layer > 0) {
            if (m < 64) d_w_ih[(size_t)nat * kHid + m] = s;
            else d_w_hh[(size_t)nat * kHid + (m - 64)] = s;
        } else {
            if (m < 64) d_w_hh[(size_t)nat * kHid + m] = s;
            else if (m - 64 < c_in) d_w_ih[(size_t)nat * c_in + (m - 64)] = s;
        }
    }
    if (e < kGateCols) {
        const int nat = (e & 3) * kHid + (e >> 2);
        d_b_ih[nat] = dbp[e];
        d_b_hh[nat] = dbp[e];
    }
}

typedef CUresult (*EncodeTiledFn16)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn16 encode_fn16() {
    static EncodeTiledFn16 fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn16)sym;
    }
    return fn;
}
// (slices, rows, 64) bf16 plane tensor, box = 1 x 128 x 64, 128-byte swizzle (rows past the end read as zeros)
bool make_plane_map(CUtensorMap* map, const void* base, int64_t rows, int64_t slices) {
    EncodeTiledFn16 fn = encode_fn16();
    if (fn == nullptr) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)kHid, (cuuint64_t)rows, (cuuint64_t)slices};
    const cuuint64_t strides[2] = {(cuuint64_t)kHid * 2, (cuuint64_t)rows * kHid * 2};
    const cuuint32_t box[3] = {(cuuint32_t)kHid, (cuuint32_t)kTileM, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// kernel variant for (planes, cin): cin = 0 (not layer 0), 1 (layer 0, one input channel), kMaxC (layer 0, runtime count)
using FwdFn = void (*)(const Fwd16Params);
using BwdFn = void (*)(const Bwd16Params);
FwdFn fwd_kernel_for(int planes, int cin) {
    if (planes == 2) return cin == 0 ? lstm16_fwd_kernel<2, 0> : (cin == 1 ? lstm16_fwd_kernel<2, 1> : lstm16_fwd_kernel<2, kMaxC>);
    return cin == 0 ? lstm16_fwd_kernel<1, 0> : (cin == 1 ? lstm16_fwd_kernel<1, 1> : lstm16_fwd_kernel<1, kMaxC>);
}
BwdFn bwd_kernel_for(int planes, int cin) {
    if (planes == 2) return cin == 0 ? lstm16_bwd_kernel<2, 0> : (cin == 1 ? lstm16_bwd_kernel<2, 1> : lstm16_bwd_kernel<2, kMaxC>);
    return cin == 0 ? lstm16_bwd_kernel<1, 0> : (cin == 1 ? lstm16_bwd_kernel<1, 1> : lstm16_bwd_kernel<1, kMaxC>);
}

// CTAs of every lstm16 launch for `rows` rows (persistent: at most one per SM)
int grid_for(int64_t rows) {
    const int64_t n_tiles = ceil_div(rows, kTileM);
    return (int)(n_tiles < sm_count() ? n_tiles : sm_count());
}

// What the forward and the backward entry check alike, before any CUDA call
int32_t check_args(const char* who, int32_t t_len, int32_t n_layers, int64_t rows, int32_t c_in, int64_t b_inner,
                   int32_t planes, const void* const* wimg, const float* const* bias, const void* h0p, const float* c0) {
    STMGCN_REQUIRE(planes == 1 || planes == 2, STMGCN_ERR_ARG, "%s: planes=%d", who, planes);
    STMGCN_REQUIRE(t_len >= 1 && n_layers >= 1 && n_layers <= 8 && rows > 0 && c_in >= 1 && c_in <= kMaxC && b_inner > 0,
                   STMGCN_ERR_SHAPE, "%s: T=%d L=%d rows=%lld C=%d", who, t_len, n_layers, (long long)rows, c_in);
    STMGCN_REQUIRE(rows <= (1LL << 25), STMGCN_ERR_SHAPE, "%s: rows=%lld too large (32-bit element offsets)", who, (long long)rows);
    STMGCN_REQUIRE((h0p == nullptr) == (c0 == nullptr), STMGCN_ERR_ARG, "%s: h0p and c0 go together", who);
    for (int l = 0; l < n_layers; ++l) STMGCN_REQUIRE(wimg[l] && bias[l], STMGCN_ERR_ARG, "%s: wimg/bias[%d] null", who, l);
    return 0;
}

// tensor maps of the hidden-state tape hp and, when there is one, of the initial state h0p (else left zero)
int32_t make_state_maps(const char* who, CUtensorMap* hp_map, CUtensorMap* h0_map, const void* hp, const void* h0p,
                        int64_t rows, int t_len, int n_layers, int planes) {
    STMGCN_REQUIRE(make_plane_map(hp_map, hp, rows, (int64_t)n_layers * t_len * planes), STMGCN_ERR_STATE,
                   "%s: cuTensorMapEncodeTiled failed (hp)", who);
    if (h0p != nullptr)
        STMGCN_REQUIRE(make_plane_map(h0_map, h0p, rows, (int64_t)n_layers * planes), STMGCN_ERR_STATE,
                       "%s: cuTensorMapEncodeTiled failed (h0p)", who);
    return 0;
}

// The K segments of layer-step (l, t), in weight-image order ([seg0 hi | seg0 lo | seg1 hi | seg1 lo]): layers > 0 first
// read h of the layer below at step t; every layer then reads its own h_prev -- h at t - 1, at t = 0 the initial state, or,
// without one, zeros (STMGCN.py:53-57).  The forward leaves a zero segment out (layers > 0 then use only W_ih, layer 0 has
// no MMA at all); the backward reads the zero tile there.
enum : int8_t { kSegHp = 0, kSegH0 = 1, kSegZero = 2 };         // Bwd16Step::src
struct StepPlan {
    int nseg;
    int8_t src[2];
    int32_t slice[2];          // plane slice of the segment's hi plane in its tensor map (lo = + 1)
    const float* c_prev;       // tile-blocked c_{t-1} of this layer, or nullptr (zeros)
};
StepPlan plan_step(int l, int t, int t_len, int planes, const float* c0, const float* cs, int64_t cslice) {
    StepPlan s;
    memset(&s, 0, sizeof(s));
    if (l > 0) {
        s.src[s.nseg] = kSegHp;
        s.slice[s.nseg] = ((l - 1) * t_len + t) * planes;
        ++s.nseg;
    }
    if (t > 0) {
        s.src[s.nseg] = kSegHp;
        s.slice[s.nseg] = (l * t_len + t - 1) * planes;
    } else if (c0 != nullptr) {                                    // c0 and h0p go together
        s.src[s.nseg] = kSegH0;
        s.slice[s.nseg] = l * planes;
    } else {
        s.src[s.nseg] = kSegZero;
    }
    ++s.nseg;
    s.c_prev = t > 0 ? cs + (int64_t)(l * t_len + t - 1) * cslice : (c0 ? c0 + (int64_t)l * cslice : nullptr);
    return s;
}

}  // namespace

extern "C" int32_t stmgcn_lstm16_pack(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh,
                                      int32_t layer, int32_t c_in, void* wimg, float* bias, float* wih_t, void* stream) {
    STMGCN_REQUIRE(w_ih && w_hh && b_ih && b_hh && wimg && bias, STMGCN_ERR_ARG, "lstm16_pack: null pointer");
    STMGCN_REQUIRE(layer >= 0 && c_in >= 1 && c_in <= kMaxC, STMGCN_ERR_SHAPE, "lstm16_pack: layer=%d c_in=%d", layer, c_in);
    STMGCN_REQUIRE(layer > 0 || wih_t != nullptr, STMGCN_ERR_ARG, "lstm16_pack: layer 0 needs wih_t");
    lstm16_pack_kernel<<<64, 256, 0, (cudaStream_t)stream>>>(w_ih, w_hh, b_ih, b_hh, layer, c_in, (uint8_t*)wimg, bias, wih_t);
    count_launch();
    return check_launch("lstm16_pack");
}

extern "C" int32_t stmgcn_lstm16_fwd(int32_t t_len, int32_t n_layers, int64_t rows, int32_t c_in, int64_t b_inner,
                                     int32_t planes, const float* xo, const float* s_gate, const void* const* wimg,
                                     const float* const* bias, const float* wih_t, const void* h0p, const float* c0,
                                     void* hp, float* cs, float* h_top, float* h_n, void* stream) {
    STMGCN_REQUIRE(xo && s_gate && wimg && bias && wih_t && hp && cs, STMGCN_ERR_ARG, "lstm16_fwd: null pointer");
    if (int32_t rc = check_args("lstm16_fwd", t_len, n_layers, rows, c_in, b_inner, planes, wimg, bias, h0p, c0)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int n_tiles = (int)ceil_div(rows, kTileM);
    const int64_t plane_elems = rows * kHid;                       // bf16 elements per plane
    const int64_t cslice = (int64_t)n_tiles * kTileM * kHid;
    const FwdFn fn0 = fwd_kernel_for(planes, c_in == 1 ? 1 : kMaxC), fn1 = fwd_kernel_for(planes, 0);
    if (int32_t rc = ensure_dyn_smem((const void*)fn0, kFSmem)) return rc;
    if (int32_t rc = ensure_dyn_smem((const void*)fn1, kFSmem)) return rc;
    CUtensorMap maps[2] = {};                                      // indexed by StepPlan::src: hp, h0p
    if (int32_t rc = make_state_maps("lstm16_fwd", &maps[kSegHp], &maps[kSegH0], hp, h0p, rows, t_len, n_layers, planes))
        return rc;
    const int grid = grid_for(rows);
    for (int t = 0; t < t_len; ++t)
        for (int l = 0; l < n_layers; ++l) {
            const StepPlan sp = plan_step(l, t, t_len, planes, c0, cs, cslice);
            Fwd16Params p;
            memset(&p, 0, sizeof(p));
            for (int s = 0; s < sp.nseg; ++s)
                if (sp.src[s] != kSegZero) {
                    p.amap[p.nseg] = maps[sp.src[s]];
                    p.aslice[p.nseg] = sp.slice[s];
                    ++p.nseg;
                }
            p.wimg = (const uint8_t*)wimg[l];
            p.bias = bias[l];
            p.wih = (l == 0) ? wih_t : nullptr;
            p.xo = xo;
            p.sg = s_gate;
            p.c_in = c_in;
            p.t = t;
            p.t_len = t_len;
            p.b_inner = b_inner;
            p.c_prev = sp.c_prev;
            p.c_out = cs + (int64_t)(l * t_len + t) * cslice;
            uint16_t* hbase = (uint16_t*)hp + (int64_t)(l * t_len + t) * planes * plane_elems;
            p.h_hi = hbase;
            p.h_lo = planes == 2 ? hbase + plane_elems : nullptr;
            p.h_f32 = nullptr;
            if (t == t_len - 1) {
                if (h_n != nullptr) p.h_f32 = h_n + (int64_t)l * rows * kHid;
                else if (l == n_layers - 1) p.h_f32 = h_top;
            }
            p.rows = rows;
            p.n_tiles = n_tiles;
            (l == 0 ? fn0 : fn1)<<<grid, kFThreads, kFSmem, st>>>(p);
            count_launch();
            if (int32_t rc = check_launch("lstm16_fwd")) return rc;
        }
    return 0;
}

extern "C" int32_t stmgcn_lstm16_grid(int64_t rows) { return grid_for(rows); }

extern "C" int32_t stmgcn_lstm16_bwd(int32_t t_len, int32_t n_layers, int64_t rows, int32_t c_in, int64_t b_inner,
                                     int32_t planes, const float* xo, const float* s_gate, const void* const* wimg,
                                     const float* const* bias, const float* wih_t, const void* h0p, const float* c0,
                                     const void* hp, const float* cs, const float* d_top, float* dh_rec, float* dc,
                                     float* dx_work, float* d_s, float* dbp, float* dw_scratch, const void* zero_tile,
                                     float* const* grads, void* stream) {
    STMGCN_REQUIRE(xo && s_gate && wimg && bias && wih_t && hp && cs && d_top && dh_rec && dc && d_s && dbp && dw_scratch &&
                       zero_tile && grads,
                   STMGCN_ERR_ARG, "lstm16_bwd: null pointer");
    if (int32_t rc = check_args("lstm16_bwd", t_len, n_layers, rows, c_in, b_inner, planes, wimg, bias, h0p, c0)) return rc;
    STMGCN_REQUIRE(t_len <= kBMaxSteps, STMGCN_ERR_SHAPE, "lstm16_bwd: T=%d (max %d)", t_len, kBMaxSteps);
    STMGCN_REQUIRE((n_layers > 1) == (dx_work != nullptr), STMGCN_ERR_ARG, "lstm16_bwd: dx_work is needed exactly when L > 1 (L=%d)",
                   n_layers);
    for (int i = 0; i < 4 * n_layers; ++i) STMGCN_REQUIRE(grads[i], STMGCN_ERR_ARG, "lstm16_bwd: grads[%d] null", i);
    cudaStream_t st = (cudaStream_t)stream;
    const int n_tiles = (int)ceil_div(rows, kTileM);
    const int64_t cslice = (int64_t)n_tiles * kTileM * kHid;
    CUtensorMap maps[2] = {};                                      // Bwd16Params::maps: hp, h0p
    if (int32_t rc = make_state_maps("lstm16_bwd", &maps[kSegHp], &maps[kSegH0], hp, h0p, rows, t_len, n_layers, planes))
        return rc;
    const int grid = grid_for(rows);
    const int64_t wg_slices = (int64_t)grid * (kTileM * kGateCols);  // one layer's dw_scratch
    // Steps per launch: the weight-gradient accumulator of a CTA lives in TMEM for the whole launch, and the tensor core's fp32
    // accumulation loses precision with the length of the chain (all T steps of cfg5's 7 tiles per CTA = 21.5 k rows in one
    // chain put 1.3e-4 into the LSTM weight gradients, measured; per-step launches, 1.8 k rows: 1.4e-5).  A launch therefore
    // covers at most kMaxChainItems (step, tile) items per CTA; the slices are summed across launches in fp32 memory.
    constexpr int kMaxChainItems = 48;                             // 6144 rows per accumulation chain
    const int tiles_per_cta = (int)ceil_div(n_tiles, grid);
    int steps_per_launch = kMaxChainItems / tiles_per_cta;
    if (steps_per_launch < 1) steps_per_launch = 1;
    // Layers top-down.  A layer reads the gradient of its output from the layer above -- the top layer d_top at T-1 only --
    // and writes the gradient of its input (dx, every step) for the layer below: two slices of dx_work alternate.
    const float* dh_in = d_top;
    for (int l = n_layers - 1; l >= 0; --l) {
        const bool top = (l == n_layers - 1);
        float* dx_out = l > 0 ? dx_work + (int64_t)((n_layers - 1 - l) % 2) * t_len * cslice : nullptr;
        const BwdFn fn = bwd_kernel_for(planes, l == 0 ? (c_in == 1 ? 1 : kMaxC) : 0);
        if (int32_t rc = ensure_dyn_smem((const void*)fn, kBSmem)) return rc;
        Bwd16Params p;
        memset(&p, 0, sizeof(p));
        p.maps[0] = maps[0];
        p.maps[1] = maps[1];
        p.zero_tile = (const uint8_t*)zero_tile;
        p.wimg = (const uint8_t*)wimg[l];
        p.bias = bias[l];
        p.wih = (l == 0) ? wih_t : nullptr;
        p.xo = xo;
        p.sg = s_gate;
        p.d_s = d_s;
        p.c_in = c_in;
        p.t_len = t_len;
        p.b_inner = b_inner;
        p.dh_rec = dh_rec;
        p.dc = dc;
        p.dbp = dbp + (int64_t)l * kGateCols;
        p.dw_slice = dw_scratch + l * wg_slices;
        p.rows = rows;
        p.n_tiles = n_tiles;
        for (int s0 = 0; s0 < t_len; s0 += steps_per_launch) {
            const int ns_launch = (t_len - s0 < steps_per_launch) ? (t_len - s0) : steps_per_launch;
            p.n_steps = ns_launch;
            p.dw_first = (s0 == 0) ? 1 : 0;
            for (int sj = 0; sj < ns_launch; ++sj) {
                const int t = t_len - 1 - (s0 + sj);
                const StepPlan plan = plan_step(l, t, t_len, planes, c0, cs, cslice);
                Bwd16Step& sp = p.steps[sj];
                for (int s = 0; s < 2; ++s) {
                    sp.src[s] = plan.src[s];
                    sp.slice[s] = plan.slice[s];
                }
                sp.t = t;
                sp.first = (t == t_len - 1) ? 1 : 0;
                sp.store_dh = (t > 0 || h0p != nullptr) ? 1 : 0;
                sp.c_prev = plan.c_prev;
                sp.dh_in = top ? (t == t_len - 1 ? dh_in : nullptr) : dh_in + (int64_t)t * cslice;
                sp.dx_out = l > 0 ? dx_out + (int64_t)t * cslice : nullptr;
            }
            fn<<<grid, kBThreads, kBSmem, st>>>(p);
            count_launch();
            if (int32_t rc = check_launch("lstm16_bwd")) return rc;
        }
        dh_in = dx_out;
    }
    // per layer: sum the CTAs' scratch slices into the nn.LSTM-native gradients w_ih, w_hh, b_ih, b_hh
    for (int l = 0; l < n_layers; ++l) {
        float* const* g = grads + 4 * l;
        lstm16_wgrad_reduce_kernel<<<(kTileM * kGateCols) / 256, 256, 0, st>>>(dw_scratch + l * wg_slices, grid, l, c_in,
                                                                             dbp + (int64_t)l * kGateCols, g[0], g[1], g[2], g[3]);
        count_launch();
        if (int32_t rc = check_launch("lstm16_bwd (weight-gradient reduction)")) return rc;
    }
    return 0;
}

#ifdef STMGCN_TC_PROFILE
// per-role wait accounting of THIS translation unit's kernels (see tc_common.cuh); instrumented builds only
extern "C" int32_t stmgcn_dbg_tc_prof16(unsigned long long* host_out, int32_t reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(host_out, stmgcn::tc::g_tc_prof, sizeof(unsigned long long) * 64);
    if (reset) {
        unsigned long long z[64] = {0};
        cudaMemcpyToSymbol(stmgcn::tc::g_tc_prof, z, sizeof(z));
    }
    return 0;
}
#endif
