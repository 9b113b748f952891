// K2 on the 5th-gen tensor cores (p = q = 64, the reference's lstm_hidden_dim / gcn_hidden_dim, Main.py:62-63):
//   forward : out[128 x 64]  = act( [T_0X | T_1X | ... | T_KX][128 x Ks*64] . W[Ks*64 x 64] + b )   (GCN.py:37-42)
//             -- the A operand is read segment by segment straight from the Chebyshev stack the SpMM steps wrote
//             (no torch.cat), split to tf32 hi/lo in the loader, accumulated in TMEM
//   backward: dZ = dOut (.) [out > 0] is formed in the loader (and written out for the weight-gradient kernel, with
//             the bias gradient as a by-product);  U[128 x Ks*64] = dZ[128 x 64] . W^T  -> U_k segments
//   weight gradient: dW[kd x 64] += [T_kX | T_{k+1}X]^T . dZ  per 128-row block of W (proj_tc_wgrad_kernel)
// CTA anatomy: register loader warps in two groups, 1 MMA warp, epilogue warps.
//
// Precision scheme "3xTF32": every fp32 operand v is split into hi = v with the low 13 mantissa bits cleared
// (exactly representable in tf32, so the tensor core's own fp32->tf32 conversion cannot change it) and
// lo = v - hi (exact in fp32; <= 13 significant bits, again masked to tf32).  A.B is accumulated in fp32
// TMEM as Ahi.Bhi + Alo.Bhi + Ahi.Blo; the dropped Alo.Blo term is ~2^-22 relative (the 1e-4 parity bar forbids
// single-pass TF32, SURVEY.md section 0.5).
//
// Loader groups and the proxy fence: fence.proxy.async (which makes the loaders' shared-memory stores visible to the
// tensor core) compiles to MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC, and the MEMBAR waits for every outstanding memory
// operation of the thread.  Loads a thread issued ahead for its next k-block / row chunk would be waited for at the
// current one's fence, so the loaders are split into two GROUPS that alternate k-blocks (row chunks): while one group
// waits for its global loads, the other converts, stores and fences.  For the same reason global stores a loader has to
// make go after its fence and barrier arrive, not before.
#include "tc_common.cuh"

using namespace stmgcn;
using namespace stmgcn::tc;

namespace {

// ---- 3xTF32 helpers ----------------------------------------------------------------------------------------
__device__ __forceinline__ float tf32_hi(float v) { return __uint_as_float(__float_as_uint(v) & 0xffffe000u); }
__device__ __forceinline__ float tf32_lo(float v, float hi) {
    return __uint_as_float(__float_as_uint(v - hi) & 0xffffe000u);
}

// kind::tf32, fp32 accumulate, M x N tile; mn_major = 0: A and B K-major, 1: both MN-major
__host__ __device__ constexpr uint32_t idesc_tf32(int m, int n, int mn_major = 0) {
    return (1u << 4)                               // c_format  = F32
           | (2u << 7)                             // a_format  = TF32
           | (2u << 10)                            // b_format  = TF32
           | ((uint32_t)(mn_major & 1) << 15)      // a_major
           | ((uint32_t)(mn_major & 1) << 16)      // b_major
           | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// D[tmem] (+)= A[smem] . B[smem], tf32 inputs, fp32 accumulate; one thread issues for the CTA.
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                         uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// MN-major tile for 32-bit operands: layout type SWIZZLE_128B_BASE32B (1), Swizzle<2,5,2> on the byte address:
// atoms of 128 B (32 consecutive M/N elements) x 4 K-rows = 512 B; inside an atom the 32-byte chunk index is XORed
// with the K-row index.  Atoms are laid out [mn atom][k atom]: LBO = (k_rows/4)*512 bytes, SBO = 512 bytes.
__host__ __device__ __forceinline__ uint32_t mn32_offset(uint32_t q /*float4 index along M/N*/, uint32_t k,
                                                         uint32_t k_rows) {
    const uint32_t atom_mn = q >> 3, c16 = q & 7;            // 8 float4 per 128-byte row
    const uint32_t atom_k = k >> 2, kr = k & 3;
    return atom_mn * (k_rows >> 2) * 512u + atom_k * 512u + kr * 128u + ((((c16 >> 1) ^ kr) & 3u) << 5) + ((c16 & 1u) << 4);
}

// byte offset of element (row, k) inside a [rows][32 fp32] K-major tile with the 128-byte swizzle
__host__ __device__ __forceinline__ uint32_t sw128_offset(uint32_t row, uint32_t k) {
    return row * 128u + ((((k >> 2) ^ (row & 7u)) & 7u) << 4) + ((k & 3u) << 2);
}

// ---- forward / backward-data pipeline ----------------------------------------------------------------------
constexpr int kTileM = 128;
constexpr int kKB = 32;              // k-block: one 128-byte swizzle row of fp32
constexpr int kMaxStages = 4;
constexpr int kAccs = 2;
constexpr int kABytes = kTileM * kKB * 4;            // 16 KB per hi or lo A tile

struct Barriers {
    uint64_t full[kMaxStages];
    uint64_t empty[kMaxStages];
    uint64_t tmem_full[kAccs];
    uint64_t tmem_empty[kAccs];
    uint32_t tmem_base;
};

__device__ __forceinline__ void init_barriers(Barriers* b, int stages, int n_epi_threads, int n_loaders) {
    for (int s = 0; s < stages; ++s) {
        mbar_init(&b->full[s], n_loaders + 1);
        mbar_init(&b->empty[s], 1);
    }
    for (int a = 0; a < kAccs; ++a) {
        mbar_init(&b->tmem_full[a], 1);
        mbar_init(&b->tmem_empty[a], n_epi_threads);
    }
    fence_barrier_init();
}

// The MMA warp: for every tile, for every k-block: wait operands, issue 3 x 4 MMAs, release the stage.
template <int N, int STAGES>
__device__ __forceinline__ void mma_issuer(Barriers* bar, uint8_t* smem, int stage_bytes, int b_bytes, int nkb,
                                           int n_tiles, uint32_t tmem_base) {
    constexpr uint32_t idesc = idesc_tf32(kTileM, N);
    const bool leader = elect_one_sync();      // (not `lane == 0`: see elect_one_sync in tc_common.cuh)
    uint32_t it = 0, tcount = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
        const int a = tcount & 1;
        const uint32_t aph = (tcount >> 1) & 1;
        mbar_wait_raw(&bar->tmem_empty[a], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)a * N;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
            const int s = it % STAGES;
            const uint32_t ph = (it / STAGES) & 1;
            mbar_wait_raw(&bar->full[s], ph);
            tc_fence_after();
            if (leader) {
                const uint32_t st = smem_u32(smem + (size_t)s * stage_bytes);
                const uint64_t a_hi = smem_desc_k_sw128(st);
                const uint64_t a_lo = smem_desc_k_sw128(st + kABytes);
                const uint64_t b_hi = smem_desc_k_sw128(st + 2 * kABytes);
                const uint64_t b_lo = smem_desc_k_sw128(st + 2 * kABytes + b_bytes);
#pragma unroll
                for (int pass = 0; pass < 3; ++pass) {
                    const uint64_t da = (pass == 1) ? a_lo : a_hi;
                    const uint64_t db = (pass == 2) ? b_lo : b_hi;
#pragma unroll
                    for (int k = 0; k < kKB / 8; ++k) {
                        const uint32_t acc = (kb > 0 || pass > 0 || k > 0) ? 1u : 0u;
                        mma_tf32(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, acc);
                    }
                }
                mma_commit(&bar->empty[s]);
            }
            __syncwarp();
        }
        if (leader) mma_commit(&bar->tmem_full[a]);
        __syncwarp();
    }
}

// split v into tf32 hi / lo and store them at st + off (hi tile) and st + kABytes + off (lo tile)
__device__ __forceinline__ void split_store(uint8_t* st, uint32_t off, const float4& v) {
    float4 hi, lo;
    hi.x = tf32_hi(v.x); hi.y = tf32_hi(v.y); hi.z = tf32_hi(v.z); hi.w = tf32_hi(v.w);
    lo.x = tf32_lo(v.x, hi.x); lo.y = tf32_lo(v.y, hi.y); lo.z = tf32_lo(v.z, hi.z); lo.w = tf32_lo(v.w, hi.w);
    *reinterpret_cast<float4*>(st + off) = hi;
    *reinterpret_cast<float4*>(st + kABytes + off) = lo;
}

// K-major hi/lo image of a logical B[n][k] = src[n*rs + k*cs]: per 32-wide k-block [hi | lo], each an
// [n_rows][32] fp32 tile with the 128-byte swizzle.
__global__ void pack_image_kernel(const float* __restrict__ src, int n_rows, int k_cols, int64_t rs, int64_t cs,
                                  float* __restrict__ img, int tile_rows) {
    const int total = n_rows * k_cols;
    const int tile_floats = tile_rows * kKB;      // tile_rows >= n_rows: extra rows keep what the caller put there (zeros)
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int n = e / k_cols, k = e % k_cols;
        const float v = src[(int64_t)n * rs + (int64_t)k * cs];
        const float hi = tf32_hi(v);
        const float lo = tf32_lo(v, hi);
        const int kb = k / kKB, kk = k % kKB;
        const uint32_t off = sw128_offset((uint32_t)n, (uint32_t)kk) / 4;
        float* base = img + (size_t)kb * (2 * tile_floats);
        base[off] = hi;
        base[tile_floats + off] = lo;
    }
}

constexpr int kPLoaderWarps = 8;
constexpr int kPLoaders = kPLoaderWarps * 32;
constexpr int kMaxSeg = 8;

template <int N>
struct PCfg {
    static constexpr int kEpiWarps = (N == 64) ? 4 : 8;
    static constexpr int kThreads = (kEpiWarps + kPLoaderWarps + 1) * 32;
    static constexpr int kBBytes = N * kKB * 4;
    static constexpr int kStageBytes = 2 * kABytes + 2 * kBBytes;
    static constexpr int kStages = (N == 64) ? 4 : 2;
    static constexpr int kTmemCols = (2 * N < 32) ? 32 : 2 * N;
};

struct PTail {
    float bias[64];
    float s_db[kPLoaderWarps][64];
    Barriers bar;
};
template <int N>
constexpr size_t psmem() { return 1024 + (size_t)PCfg<N>::kStages * PCfg<N>::kStageBytes + sizeof(PTail); }

struct PParams {
    const float* seg[kMaxSeg];   // forward: A segments (rows x 64)
    int nkb;                     // k-blocks (2 per 64-wide segment)
    // backward (dz mode): A = d_out (.) [out > 0]
    const float* d_out;          // (rows, 64) or nullptr
    const float* out_act;        // (rows, 64) forward output (mask source)
    int act;
    float* dz_out;               // (rows, 64) or nullptr (second pass of a > 4-support backward: dZ is already stored)
    float* dbias;                // (64) += or nullptr
    const float* wimg;
    const float* bias;           // forward epilogue
    float* out;                  // forward: (rows, 64)
    float* u;                    // backward: U_k = u + k*stride_u, (rows, 64) each
    int64_t stride_u;
    int ks_out;                  // backward: number of valid U segments (<= 4)
    int64_t rows;
    int n_tiles;
};

template <int N, bool DZ>
__global__ void __launch_bounds__(PCfg<N>::kThreads, 1) proj_rows_tc_kernel(const __grid_constant__ PParams p) {
    using Cfg = PCfg<N>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // keeps the __shared__ address space (LDS/STS, not generic LD/ST)
    PTail* tail = (PTail*)(smem + (size_t)Cfg::kStages * Cfg::kStageBytes);
    Barriers* bar = &tail->bar;
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;
    constexpr int kMmaWarp = Cfg::kEpiWarps + kPLoaderWarps;

    if (tid == 0) init_barriers(bar, Cfg::kStages, Cfg::kEpiWarps * 32, kPLoaders / 2);   // one loader group per k-block
    if (warp == kMmaWarp) tmem_alloc(&bar->tmem_base, Cfg::kTmemCols);
    for (int i = tid; i < 64; i += Cfg::kThreads) tail->bias[i] = (!DZ && p.bias) ? p.bias[i] : 0.f;
    for (int i = tid; i < kPLoaderWarps * 64; i += Cfg::kThreads) (&tail->s_db[0][0])[i] = 0.f;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = bar->tmem_base;

    if (warp >= Cfg::kEpiWarps && warp < kMmaWarp) {
        // ===================== loaders: two groups alternate k-blocks (the proxy fence, see the top of the file) =====
        constexpr int kGroups = 2, kGT = kPLoaders / kGroups, kPer = 1024 / kGT;
        const int ltid = tid - Cfg::kEpiWarps * 32;
        const int grp = ltid / kGT, gtid = ltid % kGT;
        const int c = gtid & 7, rsub = gtid >> 3, lwarp = ltid >> 5;
        const int my_tiles = (p.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
        const int total = my_tiles * p.nkb;
        for (int j = grp; j < total; j += kGroups) {
            const int tile = blockIdx.x + (j / p.nkb) * gridDim.x, kb = j % p.nkb;
            const int koff = (kb & 1) * kKB + c * 4;
            float4 v[kPer];
            if (DZ) {
                float4 sb = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int i = 0; i < kPer; ++i) {
                    const int64_t r = (int64_t)tile * kTileM + rsub + (kGT / 8) * i;
                    float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (r < p.rows) {
                        d = *reinterpret_cast<const float4*>(p.d_out + r * 64 + koff);
                        if (p.act == STMGCN_ACT_RELU) {
                            const float4 m = *reinterpret_cast<const float4*>(p.out_act + r * 64 + koff);
                            if (!(m.x > 0.f)) d.x = 0.f;
                            if (!(m.y > 0.f)) d.y = 0.f;
                            if (!(m.z > 0.f)) d.z = 0.f;
                            if (!(m.w > 0.f)) d.w = 0.f;
                        }
                    }
                    v[i] = d;
                    sb.x += d.x; sb.y += d.y; sb.z += d.z; sb.w += d.w;
                }
#pragma unroll
                for (int o = 8; o <= 16; o <<= 1) {
                    sb.x += __shfl_xor_sync(0xffffffffu, sb.x, o); sb.y += __shfl_xor_sync(0xffffffffu, sb.y, o);
                    sb.z += __shfl_xor_sync(0xffffffffu, sb.z, o); sb.w += __shfl_xor_sync(0xffffffffu, sb.w, o);
                }
                if (lane < 8) {
                    float4* acc = reinterpret_cast<float4*>(&tail->s_db[lwarp][koff]);
                    float4 t = *acc;
                    t.x += sb.x; t.y += sb.y; t.z += sb.z; t.w += sb.w;
                    *acc = t;
                }
            } else {
                const float* seg = p.seg[kb >> 1];
#pragma unroll
                for (int i = 0; i < kPer; ++i) {
                    const int64_t r = (int64_t)tile * kTileM + rsub + (kGT / 8) * i;
                    v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (seg != nullptr && r < p.rows) v[i] = *reinterpret_cast<const float4*>(seg + r * 64 + koff);
                }
            }
            const int s = j % Cfg::kStages;
            const uint32_t ph = (j / Cfg::kStages) & 1;
            mbar_wait_raw(&bar->empty[s], ph ^ 1);
            uint8_t* st = smem + (size_t)s * Cfg::kStageBytes;
            if (gtid == 0) {
                mbar_arrive_expect_tx(&bar->full[s], 2 * Cfg::kBBytes);
                const float* src = p.wimg + (size_t)kb * (2 * Cfg::kBBytes / 4);
                bulk_g2s(st + 2 * kABytes, src, Cfg::kBBytes, &bar->full[s]);
                bulk_g2s(st + 2 * kABytes + Cfg::kBBytes, src + Cfg::kBBytes / 4, Cfg::kBBytes, &bar->full[s]);
            }
#pragma unroll
            for (int i = 0; i < kPer; ++i) {
                const int row = rsub + (kGT / 8) * i;
                split_store(st, (uint32_t)row * 128u + (uint32_t)((c ^ (row & 7)) << 4), v[i]);
            }
            fence_proxy_async_smem();
            mbar_arrive(&bar->full[s]);
            if (DZ) {          // dZ tape for the weight-gradient kernel, stored after the fence (see the top of the file)
#pragma unroll
                for (int i = 0; i < kPer; ++i) {
                    const int64_t r = (int64_t)tile * kTileM + rsub + (kGT / 8) * i;
                    if (r < p.rows && p.dz_out != nullptr) *reinterpret_cast<float4*>(p.dz_out + r * 64 + koff) = v[i];
                }
            }
        }
    } else if (warp == kMmaWarp) {
        mma_issuer<N, Cfg::kStages>(bar, smem, Cfg::kStageBytes, Cfg::kBBytes, p.nkb, p.n_tiles, tmem_base);
    } else {
        // ===================== epilogue =====================
        const int q = warp & 3, part = warp >> 2;          // N = 256: two column halves
        uint32_t tcount = 0;
        for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++tcount) {
            const int a = tcount & 1;
            const uint32_t aph = (tcount >> 1) & 1;
            const int64_t r = (int64_t)tile * kTileM + q * 32 + lane;
            const bool valid = r < p.rows;
            mbar_wait_raw(&bar->tmem_full[a], aph);
            tc_fence_after();
            const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)a * N;
            constexpr int kChunksPerWarp = (N == 64) ? 2 : 4;
#pragma unroll 1
            for (int ci = 0; ci < kChunksPerWarp; ++ci) {
                const int chunk = part * kChunksPerWarp + ci;
                uint32_t v[32];
                tmem_ld32(t_row + chunk * 32, v);
                tmem_ld_wait();
                if (!valid) continue;
                if (N == 64) {
                    float* dst = p.out + r * 64 + chunk * 32;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        float4 o;
                        o.x = __uint_as_float(v[4 * j + 0]) + tail->bias[chunk * 32 + 4 * j + 0];
                        o.y = __uint_as_float(v[4 * j + 1]) + tail->bias[chunk * 32 + 4 * j + 1];
                        o.z = __uint_as_float(v[4 * j + 2]) + tail->bias[chunk * 32 + 4 * j + 2];
                        o.w = __uint_as_float(v[4 * j + 3]) + tail->bias[chunk * 32 + 4 * j + 3];
                        if (p.act == STMGCN_ACT_RELU) {
                            o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f);
                        }
                        *reinterpret_cast<float4*>(dst + 4 * j) = o;
                    }
                } else {
                    const int col = chunk * 32;                    // U_k, k = col / 64
                    if ((col >> 6) >= p.ks_out) continue;
                    float* dst = p.u + (int64_t)(col >> 6) * p.stride_u + r * 64 + (col & 63);
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<uint4*>(dst + 4 * j) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                }
            }
            tc_fence_before();
            mbar_arrive(&bar->tmem_empty[a]);
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == kMmaWarp) tmem_dealloc(tmem_base, Cfg::kTmemCols);
    if (DZ && p.dbias != nullptr) {
        for (int i = tid; i < 64; i += Cfg::kThreads) {
            float v = 0.f;
#pragma unroll
            for (int w = 0; w < kPLoaderWarps; ++w) v += tail->s_db[w][i];
            atomicAdd(&p.dbias[i], v);
        }
    }
}

// ---- weight gradient ------------------------------------------------------------------------------------------
// dW[kd x 64] += sum over rows r of [seg0 | seg1][r, :]^T . dZ[r, :]
// M = kd index (padded to 128), N = 64 output columns, K = rows.  Both operands are row-major in HBM, i.e. K is the slow
// dimension: they are MN-major operands.  The loaders copy rows with coalesced float4 loads and store them as MN-major
// atoms with the 32-byte-base 128B swizzle (layout type SWIZZLE_128B_BASE32B = 1, see mn32_offset; with the plain
// SWIZZLE_128B type and the MN-major descriptor bits the tf32 MMA returns zeros).  One TMEM accumulator lives for the
// whole kernel and is flushed with atomicAdd.
constexpr int kWgLoaderWarps = 16;
constexpr int kWgLoaders = kWgLoaderWarps * 32;
constexpr int kWgThreads = kWgLoaders + 32;                        // 544: loaders + the MMA warp
constexpr int kWgN = 64;
constexpr int kWgStages = 2;
constexpr int kWgRows = 32;                                        // K per stage
constexpr int kWgABytes = 128 * kWgRows * 4;                       // 16 KB  [128 m][32 k]
constexpr int kWgBBytes = kWgN * kWgRows * 4;                      // 8 KB   [64 n][32 k]
constexpr int kWgStageBytes = 2 * kWgABytes + 2 * kWgBBytes;
constexpr size_t kWgSmem = 1024 + (size_t)kWgStages * kWgStageBytes + 64;

struct WgTail {
    uint64_t full[kWgStages];
    uint64_t empty[kWgStages];
    uint64_t done;
    uint32_t tmem_base;
};
static_assert(sizeof(WgTail) <= 64, "WgTail");

struct WgParams {
    const float* seg0;       // (rows, 64): dW rows 0..63 of this block
    const float* seg1;       // (rows, 64): dW rows 64..127, or nullptr (a 64-row block)
    const float* dz;         // (rows, 64)
    float* dw;               // (kd, 64) +=, kd = 64 per segment
    int kd;
    int64_t rows;
    int n_chunks;            // ceil(rows / kWgRows)
};

__global__ void __launch_bounds__(kWgThreads, 1) proj_tc_wgrad_kernel(const __grid_constant__ WgParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // keeps the __shared__ address space (LDS/STS, not generic LD/ST)
    WgTail* tail = (WgTail*)(smem + (size_t)kWgStages * kWgStageBytes);
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;
    constexpr int kMmaWarp = kWgLoaderWarps;

    if (tid == 0) {
        for (int s = 0; s < kWgStages; ++s) {
            mbar_init(&tail->full[s], kWgLoaders / 2);       // one loader group per chunk
            mbar_init(&tail->empty[s], 1);
        }
        mbar_init(&tail->done, 1);
        fence_barrier_init();
    }
    if (warp == kMmaWarp) tmem_alloc(&tail->tmem_base, kWgN);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tail->tmem_base;
    const bool has_work = (int)blockIdx.x < p.n_chunks;

    if (warp < kMmaWarp) {
        // ===================== loaders: HBM rows -> tf32 hi/lo -> MN-major swizzled atoms =====================
        // two groups alternate row chunks (the proxy fence, see the top of the file)
        constexpr int kGroups = 2, kGT = kWgLoaders / kGroups;
        constexpr int kNA = 1024 / kGT, kNB = (32 * kWgN / 4) / kGT;
        static_assert(kNB >= 1, "loader mapping");
        const int grp = tid / kGT, gtid = tid % kGT;
        const int my_chunks = (p.n_chunks - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
        for (int j = grp; j < my_chunks; j += kGroups) {
            const int64_t r0 = (int64_t)(blockIdx.x + j * gridDim.x) * kWgRows;
            float4 va[kNA], vb[kNB];
#pragma unroll
            for (int i = 0; i < kNA; ++i) {                   // A': 32 rows x 32 float4 (128 kd values), coalesced
                const int idx = gtid + i * kGT;
                const int row = idx >> 5, q = idx & 31;
                const int64_t r = r0 + row;
                const float* src = q < 16 ? p.seg0 : p.seg1;   // m 0..63 from seg0, 64..127 from seg1
                va[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (src != nullptr && r < p.rows) va[i] = *reinterpret_cast<const float4*>(src + r * 64 + (q & 15) * 4);
            }
#pragma unroll
            for (int i = 0; i < kNB; ++i) {                   // B': 32 rows x 16 float4, coalesced
                const int idx = gtid + i * kGT;
                const int row = idx / (kWgN / 4), q = idx % (kWgN / 4);
                const int64_t r = r0 + row;
                vb[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r < p.rows) vb[i] = *reinterpret_cast<const float4*>(p.dz + r * kWgN + q * 4);
            }
            const int s = j % kWgStages;
            const uint32_t ph = (j / kWgStages) & 1;
            mbar_wait_raw(&tail->empty[s], ph ^ 1);
            uint8_t* st = smem + (size_t)s * kWgStageBytes;
#pragma unroll
            for (int i = 0; i < kNA; ++i) {
                const int idx = gtid + i * kGT;
                split_store(st, mn32_offset(idx & 31, idx >> 5, kWgRows), va[i]);      // hi at st, lo at st + kWgABytes
            }
#pragma unroll
            for (int i = 0; i < kNB; ++i) {
                const int idx = gtid + i * kGT;
                const uint32_t off = mn32_offset(idx % (kWgN / 4), idx / (kWgN / 4), kWgRows);
                float4 hi, lo;
                const float4 v = vb[i];
                hi.x = tf32_hi(v.x); hi.y = tf32_hi(v.y); hi.z = tf32_hi(v.z); hi.w = tf32_hi(v.w);
                lo.x = tf32_lo(v.x, hi.x); lo.y = tf32_lo(v.y, hi.y); lo.z = tf32_lo(v.z, hi.z); lo.w = tf32_lo(v.w, hi.w);
                *reinterpret_cast<float4*>(st + 2 * kWgABytes + off) = hi;
                *reinterpret_cast<float4*>(st + 2 * kWgABytes + kWgBBytes + off) = lo;
            }
            fence_proxy_async_smem();
            mbar_arrive(&tail->full[s]);
        }
        // ===================== epilogue (warps 0-3): accumulator rows = kd index -> atomicAdd into dW =====================
        if (warp < 4 && has_work) {
            mbar_wait_raw(&tail->done, 0);
            tc_fence_after();
            const int m = warp * 32 + lane;
            const uint32_t t_row = tmem_base + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
            for (int chunk32 = 0; chunk32 < kWgN / 32; ++chunk32) {
                uint32_t v[32];
                tmem_ld32(t_row + chunk32 * 32, v);
                tmem_ld_wait();
                if (m < p.kd) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) atomicAdd(p.dw + (int64_t)m * kWgN + chunk32 * 32 + j, __uint_as_float(v[j]));
                }
            }
        }
    } else {
        // ===================== MMA issuer =====================
        constexpr uint32_t idesc = idesc_tf32(128, kWgN, 1);       // both operands MN-major
        constexpr uint32_t kLbo = (kWgRows / 4) * 512, kSbo = 512;
        const bool leader = elect_one_sync();      // (not `lane == 0`: see elect_one_sync in tc_common.cuh)
        uint32_t it = 0;
        for (int chunk = blockIdx.x; chunk < p.n_chunks; chunk += gridDim.x, ++it) {
            const int s = it % kWgStages;
            const uint32_t ph = (it / kWgStages) & 1;
            mbar_wait_raw(&tail->full[s], ph);
            tc_fence_after();
            if (leader) {
                const uint32_t st = smem_u32(smem + (size_t)s * kWgStageBytes);
#pragma unroll
                for (int pass = 0; pass < 3; ++pass) {
                    const uint32_t a_base = st + ((pass == 1) ? kWgABytes : 0);
                    const uint32_t b_base = st + 2 * kWgABytes + ((pass == 2) ? kWgBBytes : 0);
#pragma unroll
                    for (int ks = 0; ks < kWgRows / 8; ++ks) {      // one MMA consumes K = 8 rows = two 4-row atoms
                        const uint64_t da = smem_desc_mn_sw128(a_base + ks * 2 * kSbo, kLbo, kSbo, 1);
                        const uint64_t db = smem_desc_mn_sw128(b_base + ks * 2 * kSbo, kLbo, kSbo, 1);
                        mma_tf32(tmem_base, da, db, idesc, (it > 0 || pass > 0 || ks > 0) ? 1u : 0u);
                    }
                }
                mma_commit(&tail->empty[s]);
            }
            __syncwarp();
        }
        if (leader && has_work) mma_commit(&tail->done);
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == kMmaWarp) tmem_dealloc(tmem_base, kWgN);
}

// ---- host launchers ----------------------------------------------------------------------------------------
// forward: out = act(sum_k S_k W_k + bias); wimg = image of B[n][k] = W[k][n] (2*ks k-blocks of [hi|lo] [64][32])
int32_t launch_proj_fwd_tc(const float* s, int64_t stride_k, int ks, int64_t rows, const float* wimg, const float* bias,
                           int act, float* out, cudaStream_t st) {
    auto kern = proj_rows_tc_kernel<64, false>;
    if (int32_t rc = ensure_dyn_smem((const void*)kern, psmem<64>())) return rc;
    PParams p{};
    for (int k = 0; k < ks; ++k) p.seg[k] = s + (int64_t)k * stride_k;
    p.nkb = 2 * ks;
    p.wimg = wimg;
    p.bias = bias;
    p.act = act;
    p.out = out;
    p.rows = rows;
    p.n_tiles = (int)ceil_div(rows, kTileM);
    const int grid = p.n_tiles < sm_count() ? p.n_tiles : sm_count();
    kern<<<grid, PCfg<64>::kThreads, psmem<64>(), st>>>(p);
    count_launch();
    return check_launch("proj_fwd_tc");
}

// backward data: dZ = d_out (.) mask (written to dz_out, bias gradient accumulated), U_k = dZ W_k^T (if u != nullptr);
// wimg_t = image of B[n = k*64+i][k' = j] = W[n][j]  (2 k-blocks of [hi|lo] [ks*64][32])
int32_t launch_proj_bwd_tc(const float* d_out, const float* out_act, int act, int64_t rows, int ks, const float* wimg_t,
                           float* dz_out, float* dbias, float* u, int64_t stride_u, cudaStream_t st) {
    auto kern = proj_rows_tc_kernel<256, true>;
    if (int32_t rc = ensure_dyn_smem((const void*)kern, psmem<256>())) return rc;
    PParams p{};
    p.nkb = 2;
    p.ks_out = ks;
    p.d_out = d_out;
    p.out_act = out_act;
    p.act = act;
    p.dz_out = dz_out;
    p.dbias = dbias;
    p.wimg = wimg_t;
    p.u = u;
    p.stride_u = stride_u;
    p.rows = rows;
    p.n_tiles = (int)ceil_div(rows, kTileM);
    const int grid = p.n_tiles < sm_count() ? p.n_tiles : sm_count();
    kern<<<grid, PCfg<256>::kThreads, psmem<256>(), st>>>(p);
    count_launch();
    return check_launch("proj_bwd_tc");
}

// weight gradient of one 128-row block of W (seg0 and seg1) or of a 64-row tail block (seg1 = nullptr):
// dw[kd x 64] += [seg0 | seg1]^T . dz
int32_t launch_proj_tc_wgrad(const float* seg0, const float* seg1, const float* dz, int64_t rows, float* dw,
                             cudaStream_t st) {
    if (int32_t rc = ensure_dyn_smem((const void*)proj_tc_wgrad_kernel, kWgSmem)) return rc;
    WgParams p;
    p.seg0 = seg0;
    p.seg1 = seg1;
    p.dz = dz;
    p.dw = dw;
    p.kd = seg1 ? 128 : 64;
    p.rows = rows;
    p.n_chunks = (int)ceil_div(rows, kWgRows);
    const int grid = p.n_chunks < sm_count() ? p.n_chunks : sm_count();
    proj_tc_wgrad_kernel<<<grid, kWgThreads, kWgSmem, st>>>(p);
    count_launch();
    return check_launch("proj_tc_wgrad");
}

int32_t launch_pack_image(const float* src, int n_rows, int k_cols, int64_t rs, int64_t cs, float* img, int tile_rows,
                          cudaStream_t st) {
    pack_image_kernel<<<(n_rows * k_cols + 255) / 256, 256, 0, st>>>(src, n_rows, k_cols, rs, cs, img, tile_rows);
    count_launch();
    return check_launch("pack_image");
}

}  // namespace

extern "C" {

int32_t stmgcn_proj_pack_tc(const float* w, int32_t ks, float* img_fwd, float* img_bwd, void* stream) {
    STMGCN_REQUIRE(w && img_fwd, STMGCN_ERR_ARG, "proj_pack_tc: null pointer");
    STMGCN_REQUIRE(ks >= 1 && ks <= 8, STMGCN_ERR_SHAPE, "proj_pack_tc: ks=%d (tensor-core path supports 1..8 supports)", ks);
    cudaStream_t st = (cudaStream_t)stream;
    // forward operand B[n = out col][k = ks*64 index] = W[k][n]
    if (int32_t rc = launch_pack_image(w, 64, ks * 64, 1, 64, img_fwd, 64, st)) return rc;
    // backward operand B[n = k*64+i][k' = out col] = W[n][k'], one 256-row image per group of 4 supports (caller
    // zero-fills img_bwd: rows beyond the last support stay zero)
    if (img_bwd) {
        const int k0 = ks < 4 ? ks : 4;
        if (int32_t rc = launch_pack_image(w, k0 * 64, 64, 64, 1, img_bwd, 256, st)) return rc;
        if (ks > 4) return launch_pack_image(w + (int64_t)256 * 64, (ks - 4) * 64, 64, 64, 1, img_bwd + 2 * 2 * 256 * 32, 256, st);
    }
    return 0;
}

int32_t stmgcn_proj_fwd_tc(const float* s, int64_t stride_k, int32_t ks, int64_t rows, const float* wimg,
                           const float* bias, int32_t act, float* out, void* stream) {
    STMGCN_REQUIRE(s && wimg && out, STMGCN_ERR_ARG, "proj_fwd_tc: null pointer");
    STMGCN_REQUIRE(act == STMGCN_ACT_NONE || act == STMGCN_ACT_RELU, STMGCN_ERR_ARG, "proj_fwd_tc: act=%d", act);
    STMGCN_REQUIRE(ks >= 1 && ks <= 8 && rows > 0, STMGCN_ERR_SHAPE, "proj_fwd_tc: ks=%d rows=%lld (1..8 supports)", ks,
                   (long long)rows);
    STMGCN_REQUIRE(aligned16(s) && aligned16(wimg) && aligned16(out) && stride_k % 4 == 0, STMGCN_ERR_ALIGN,
                   "proj_fwd_tc: s, wimg and out must be 16-byte aligned and stride_k a multiple of 4");
    return launch_proj_fwd_tc(s, stride_k, ks, rows, wimg, bias, act, out, (cudaStream_t)stream);
}

int32_t stmgcn_proj_bwd_tc(const float* s, int64_t stride_k, int32_t ks, int64_t rows, const float* wimg_t, int32_t act,
                           const float* out, const float* d_out, float* dz_work, float* dw, float* dbias, float* u,
                           int64_t stride_u, void* stream) {
    STMGCN_REQUIRE(s && wimg_t && out && d_out && dz_work && dw && u, STMGCN_ERR_ARG, "proj_bwd_tc: null pointer");
    STMGCN_REQUIRE(act == STMGCN_ACT_NONE || act == STMGCN_ACT_RELU, STMGCN_ERR_ARG, "proj_bwd_tc: act=%d", act);
    STMGCN_REQUIRE(ks >= 1 && ks <= 8 && rows > 0, STMGCN_ERR_SHAPE, "proj_bwd_tc: ks=%d rows=%lld (1..8 supports)", ks,
                   (long long)rows);
    STMGCN_REQUIRE(aligned16(s) && aligned16(wimg_t) && aligned16(out) && aligned16(d_out) && aligned16(dz_work) &&
                       aligned16(u) && stride_k % 4 == 0 && stride_u % 4 == 0,
                   STMGCN_ERR_ALIGN, "proj_bwd_tc: s, wimg_t, out, d_out, dz_work and u must be 16-byte aligned, "
                   "stride_k and stride_u multiples of 4");
    cudaStream_t st = (cudaStream_t)stream;
    // dZ + bias gradient + U in one kernel.  U has 64*ks columns; one launch produces up to 256 of them (supports 0..3), a
    // second one the rest (it re-forms dZ in its loader but neither stores it nor accumulates the bias gradient again)
    if (int32_t rc = launch_proj_bwd_tc(d_out, out, act, rows, ks < 4 ? ks : 4, wimg_t, dz_work, dbias, u, stride_u, st)) return rc;
    if (ks > 4)
        if (int32_t rc = launch_proj_bwd_tc(d_out, out, act, rows, ks - 4, wimg_t + 2 * 2 * 256 * 32, nullptr, nullptr,
                                            u + 4 * stride_u, stride_u, st))
            return rc;
    // dW per 128-row block of W
    for (int k0 = 0; k0 < ks; k0 += 2) {
        const float* s0 = s + (int64_t)k0 * stride_k;
        const float* s1 = k0 + 1 < ks ? s0 + stride_k : nullptr;     // nullptr: the 64-row tail block of W
        if (int32_t rc = launch_proj_tc_wgrad(s0, s1, dz_work, rows, dw + (int64_t)k0 * 64 * 64, st)) return rc;
    }
    return 0;
}

}  // extern "C"
