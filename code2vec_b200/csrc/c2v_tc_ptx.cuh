// c2v_tc_ptx.cuh -- raw PTX wrappers shared by the sm_100a tensor-core kernels: mbarrier, proxy fences,
// cp.async.bulk (TMA), tcgen05 (MMA / TMEM / commit), UMMA shared-memory descriptors.
#pragma once
#include <cuda_fp16.h>

#include "c2v_common.cuh"

namespace c2v {

// ------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Wait for the phase with the given parity; a watchdog turns a protocol bug into a trap instead of a hung GPU.
// A bare try_wait returns after ~30 cycles, so a waiting warp re-polls ~30x per microsecond: in the K1e profile two
// thirds of all executed warp instructions were these poll loops, taking issue slots from the warps that had work.
// Measured alternatives (cfg2, K1e): try_wait with a suspend-time hint of 1 or 20 us: 82.6-83.1 us (the hardware
// wake-up is slower than a poll); nanosleep 500: 74.1 us; nanosleep 64: 72.9 us  -> wake-up latency matters more than
// the issue slots the polls take.
constexpr unsigned C2V_SPIN_NS = 64;
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, long long *status) {
    uint32_t ok = 0;
    long long t0 = 0;
    for (uint32_t spins = 0;; ++spins) {
        asm volatile("{\n\t.reg .pred p;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) break;
        __nanosleep(C2V_SPIN_NS);
#ifndef C2V_NO_WATCHDOG                               // (compute-sanitizer slows kernels 100x: build the variant without it)
        if ((spins & 0x3ff) == 0x3ff) {
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000LL) {           // ~2 s: certainly a deadlock
                status[1] = 0xDEAD0000LL | (long long)(bar & 0xffff);
                __threadfence();
                __trap();
            }
        }
#endif
    }
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
// start>>4 [0,14) | LBO>>4 [16,30) (unused for swizzled K-major, 1) | SBO>>4 [32,46) = 1024 B
// (stride between 8-row groups) | version=1 [46,48) | layout_type=2 (SWIZZLE_128B) [61,64)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) |
           (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float *v) {
    uint32_t r[32];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float *v) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float *v) {
    uint32_t r[4];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float *v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
                 "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
                 "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
                 ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]),
                   "f"(v[8]), "f"(v[9]), "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]),
                   "f"(v[16]), "f"(v[17]), "f"(v[18]), "f"(v[19]), "f"(v[20]), "f"(v[21]), "f"(v[22]), "f"(v[23]),
                   "f"(v[24]), "f"(v[25]), "f"(v[26]), "f"(v[27]), "f"(v[28]), "f"(v[29]), "f"(v[30]), "f"(v[31]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait_all() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float4 ldg_nc_v4(const float4 *p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ void sts_v2(uint32_t addr, uint32_t a, uint32_t b) {
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ uint32_t pack_h2(__half2 h) { return *reinterpret_cast<uint32_t *>(&h); }

// byte offset of fp16 element (row, k) inside a [rows x 64] K-major SWIZZLE_128B tile
__host__ __device__ __forceinline__ uint32_t sw128_offset(int row, int k) {
    return (uint32_t)((row >> 3) * 1024 + (row & 7) * 128 + ((((k >> 3) ^ (row & 7)) & 7) << 4) + (k & 7) * 2);
}

// In-place transpose-reduce across the 32 lanes of a warp: on entry lane i holds v[0..31]
// (32 columns of its row); on exit v[0] of lane i is the sum over all 32 lanes of column i.
// 31 shuffles instead of 32 x 5.
__device__ __forceinline__ void butterfly_reduce32(float (&v)[32], int lane) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int j = 0; j < off; ++j) {
            const float send = upper ? v[j] : v[j + off];
            const float keep = upper ? v[j + off] : v[j];
            v[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
}

__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// tanh(v) given w = 2*log2(e)*v :  1 - 2/(2^w + 1); 2^w = inf -> 1, 2^w = 0 -> -1.  Two MUFU ops,
// absolute error ~2e-7 (same formula as tanh_accurate, constants folded into gamma/beta).
__device__ __forceinline__ float tanh_from_scaled(float w) {
    return fmaf(-2.0f, rcp_approx(ex2_approx(w) + 1.0f), 1.0f);
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}


}  // namespace c2v
