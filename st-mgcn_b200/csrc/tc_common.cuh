// Blackwell (sm_100a) primitives shared by the tensor-core kernels (lstm16.cu through tc16.cuh, proj_tc.cu): mbarrier
// and bounded waits, 1-D bulk async copy (TMA unit, SASS UBLKCP), L2 prefetch, wide global stores / reductions,
// tcgen05 (alloc / commit / ld / fences), the elected single issuing thread and the 128-byte-swizzle UMMA descriptors.
// The MMA instructions themselves live with their precision scheme: kind::f16 in tc16.cuh, kind::tf32 in proj_tc.cu.
#pragma once
#include "common.cuh"

namespace stmgcn {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier -----------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (the launch fails with an error) instead of hanging the GPU.
// (fast polls first, then a nanosleep back-off: ~20 s before the trap, so profiler / sanitizer slow-downs of 100x do not
// kill the context -- VERDICT r1)
__device__ __forceinline__ void mbar_wait_raw(uint64_t* bar, uint32_t parity) {
    for (uint32_t it = 0; it < (1u << 16); ++it)
        if (mbar_try_wait(bar, parity)) return;
    for (uint32_t it = 0; it < (1u << 26); ++it) {
        if (mbar_try_wait(bar, parity)) return;
        __nanosleep(256);
    }
    __trap();
}
// Polite wait for the single-thread roles (TMA producer, MMA issuer): a spinning warp competes for issue slots with the
// warps doing the arithmetic on the same SM sub-partition (ncu: a quarter of all executed instructions were try_wait /
// branch pairs), so back off ~40 ns between polls; the bound is the same ~20 s.
__device__ __forceinline__ void mbar_wait_polite(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    for (uint32_t it = 0; it < (1u << 28); ++it) {
        __nanosleep(40);
        if (mbar_try_wait(bar, parity)) return;
    }
    __trap();
}
// Optional wait-time accounting (built with -DSTMGCN_TC_PROFILE): cycles each role spends blocked on each barrier
// class, summed per launch into g_tc_prof[slot]; slot = role*4 + barrier class.  The library is built without relocatable
// device code, so every translation unit has its own g_tc_prof: the instrumented kernels are lstm16.cu's, read with
// stmgcn_dbg_tc_prof16() (tools/tc_role_profile16.py).
#ifdef STMGCN_TC_PROFILE
__device__ unsigned long long g_tc_prof[64];
struct WaitProf {
    unsigned long long acc[4] = {0, 0, 0, 0};
    long long t_start;
    __device__ WaitProf() { t_start = clock64(); }
    __device__ void flush(int role, bool leader) {
        if (leader) {
            for (int i = 0; i < 4; ++i) atomicAdd(&g_tc_prof[role * 4 + i], acc[i]);
            atomicAdd(&g_tc_prof[48 + role], (unsigned long long)(clock64() - t_start));
        }
    }
};
#define TC_PROF_DECL WaitProf _wp;
#define TC_PROF_FLUSH(role, leader) _wp.flush(role, leader);
#define mbar_wait(bar, parity, cls) do { long long _t0 = clock64(); mbar_wait_raw(bar, parity); _wp.acc[cls] += clock64() - _t0; } while (0)
#define mbar_wait_p(bar, parity, cls) do { long long _t0 = clock64(); mbar_wait_polite(bar, parity); _wp.acc[cls] += clock64() - _t0; } while (0)
#else
#define TC_PROF_DECL
#define TC_PROF_FLUSH(role, leader)
#define mbar_wait(bar, parity, cls) mbar_wait_raw(bar, parity)
#define mbar_wait_p(bar, parity, cls) mbar_wait_polite(bar, parity)
#endif

// generic-proxy smem writes -> visible to the async proxy (tcgen05.mma / bulk copies read smem through it)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- 1-D bulk async copy global -> shared, completion on an mbarrier (TMA unit; SASS: UBLKCP) -----------
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// One elected lane of a fully converged warp.  Guarding the single-thread tcgen05 / TMA / mbarrier instructions with this
// instead of `lane == 0` matters: ptxas cannot prove `lane == 0` selects one thread, and wraps EVERY uniform-datapath
// instruction (UTCHMMA, UTCBAR, UBLKCP, UTMALDG) in an ELECT / BRA.U.ANY serialisation loop -- ~10 extra instructions and
// a branch per MMA, measured as ~90 cycles per issued tcgen05.mma.  After elect.sync the instructions issue back to back.
// The elected lane is the same on every call of a converged warp, so MMAs and their tcgen05.commit come from one thread.
__device__ __forceinline__ bool elect_one_sync() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}
// 256-bit global store / load (sm_100: STG.E.ENL2.256 / LDG.E.ENL2.256): 8 consecutive 32-bit words, 32-byte aligned
__device__ __forceinline__ void st_global_v8(void* dst, const uint32_t* v) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
                 "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
// fire-and-forget 16-byte reduction into global memory (REDG.E.ADD.F32x4: the add happens in L2, nothing returns)
__device__ __forceinline__ void red_add_f32x4(float4* dst, const float4& v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// L2 prefetch of a contiguous global range (no registers, no shared memory; SASS UBLKPF)
__device__ __forceinline__ void prefetch_l2(const void* gmem, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gmem), "r"(bytes) : "memory");
}

// ---- tcgen05 --------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {   // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {      // same warp that allocated
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// all previously issued MMAs of this thread complete -> one arrival on the mbarrier
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets row (lane base + i), columns [c, c+32)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, "
        "[%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- UMMA descriptors (field layout: cute/arch/mma_sm100_desc.hpp in the vendored CUTLASS tree) --------------
// K-major operand tile, 128-byte swizzle: rows of 128 B (32 fp32 along K), 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t smem_desc_k_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);          // start address  [0,14)
    d |= (uint64_t)1 << 16;                              // leading byte offset (unused for swizzled K-major) [16,30)
    d |= (uint64_t)(1024 >> 4) << 32;                    // stride byte offset: 8 rows x 128 B [32,46)
    d |= (uint64_t)1 << 46;                              // descriptor version 1 (Blackwell) [46,48)
    d |= (uint64_t)2 << 61;                              // layout type SWIZZLE_128B [61,64)
    return d;
}
// MN-major operand, 128-byte swizzle.  Canonical layout (cute/atom/mma_traits_sm100.hpp, in 16-byte units):
// ((8,n),(8,k)) : ((1,LBO),(8,SBO)) -- a 1024-byte atom holds 32 consecutive M/N elements (one 128-byte row)
// for each of 8 consecutive K; LBO = byte distance between atoms along M/N, SBO = between atoms along K.
__device__ __forceinline__ uint64_t smem_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                       uint32_t layout_type = 2) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)layout_type << 61;
    return d;
}

}  // namespace tc
}  // namespace stmgcn
