// c2v_label_tcgen05.cu -- K2: label logits  outputs = cv . W_out^T + b  (model.py:83) on tcgen05.
//
// Same fp32-accurate scheme as the encode kernel: both operands are split into fp16 hi + lo and
// three kind::f16 MMAs (hi.hi + lo.hi + hi.lo) accumulate in fp32 in TMEM.  W_out is scaled by a
// power of two (from its absmax) before the split; the epilogue multiplies by the exact inverse
// and adds the bias.  Plain TF32 fails the 1e-4 bar on trained weights (SURVEY.md 8d).
//
// Three launches: absmax(W_out) -> split cv and W_out into UMMA K-major SWIZZLE_128B tile images
// ([128 rows x 64 k] fp16, hi then lo, per k-block) -> one CTA per 128x128 output tile: two 64 KB
// cp.async.bulk copies, 24 tcgen05.mma, TMEM -> registers -> padded smem -> coalesced 512-B row
// stores with the bias added.  Output-write bound (B*C*4 bytes).
#include <cuda_fp16.h>

#include <cstring>

#include "c2v_common.cuh"

namespace c2v {

namespace lt {
constexpr int TM = 128, TN = 128, KB = 64;
constexpr int TILE_BYTES = 128 * KB * 2;          // 16 KB
constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
}  // namespace lt

__host__ __device__ __forceinline__ uint32_t lt_sw128(int row, int k) {
    return (uint32_t)((row >> 3) * 1024 + (row & 7) * 128 + ((((k >> 3) ^ (row & 7)) & 7) << 4) + (k & 7) * 2);
}
__device__ __forceinline__ uint32_t lt_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__global__ void absmax_kernel(const float *__restrict__ x, long long n, unsigned *__restrict__ out_bits)
{
    float m = 0.0f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        m = fmaxf(m, fabsf(x[i]));
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0) atomicMax(out_bits, __float_as_uint(m));   // non-negative floats order as uints
}

// X [R, K] fp32 row-major -> image: for each 128-row tile, for each k-block: {hi tile, lo tile}.
// scale_bits == nullptr: no scaling.  Rows >= R are zero-filled.  hdr[0] = 1/scale, hdr[1] = scale.
__global__ void split_rows_kernel(const float *__restrict__ X, long long R, int K, int nkb,
                                  const unsigned *__restrict__ scale_bits, uint8_t *__restrict__ img,
                                  float *__restrict__ hdr, unsigned long long *__restrict__ zero_u64, int n_zero)
{
    pdl_wait();                                   // (no-op unless launched as a programmatic dependent)
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_zero; i += gridDim.x * blockDim.x) zero_u64[i] = 0ull;
    float scale = 1.0f;
    if (scale_bits) {
        const float mx = __uint_as_float(*scale_bits);
        if (mx > 0.0f && mx < 3.0e38f) {
            int e;
            frexpf(mx, &e);
            int k = 14 - e;
            k = k > 60 ? 60 : (k < -60 ? -60 : k);
            scale = ldexpf(1.0f, k);
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) { hdr[0] = 1.0f / scale; hdr[1] = scale; }
    }
    const long long tiles = (R + 127) / 128;
    const long long total = tiles * 128 * (long long)(nkb * 16);          // float4 groups
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
        const int k4 = (int)(g % (nkb * 16));
        const long long row = g / (nkb * 16);
        const int k = k4 * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row < R && k < K) v = *reinterpret_cast<const float4 *>(X + row * K + k);
        v.x *= scale; v.y *= scale; v.z *= scale; v.w *= scale;
        const __half2 h01 = __floats2half2_rn(v.x, v.y), h23 = __floats2half2_rn(v.z, v.w);
        const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
        const __half2 l01 = __floats2half2_rn(v.x - f01.x, v.y - f01.y), l23 = __floats2half2_rn(v.z - f23.x, v.w - f23.y);
        const long long tile = row >> 7;
        const int r = (int)(row & 127), kb = k / lt::KB, kk = k % lt::KB;
        uint8_t *base = img + (tile * nkb + kb) * (size_t)(2 * lt::TILE_BYTES);
        const uint32_t off = lt_sw128(r, kk);
        *reinterpret_cast<uint2 *>(base + off) = make_uint2(*reinterpret_cast<const unsigned *>(&h01), *reinterpret_cast<const unsigned *>(&h23));
        *reinterpret_cast<uint2 *>(base + lt::TILE_BYTES + off) = make_uint2(*reinterpret_cast<const unsigned *>(&l01), *reinterpret_cast<const unsigned *>(&l23));
    }
}

__device__ __forceinline__ void lt_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
    for (unsigned spins = 0; !ok; ++spins) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
#ifndef C2V_NO_WATCHDOG
        if (!ok && spins > (1u << 26)) __trap();
#endif
    }
}
__device__ __forceinline__ bool lt_elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}
// monotone float -> uint32 map, so that (key(value) << 32 | ~column) ordered as uint64 picks the largest value and,
// among equal values, the smallest column: torch.max(dim=1) semantics (main.py:285)
__device__ __forceinline__ uint32_t lt_orderable(float v) {
    const uint32_t u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float lt_from_orderable(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// Tile order: groups of NT_GROUP consecutive n-tiles; inside a group m-tile major, n-tile minor.  A CTA's consecutive
// tiles then write adjacent 512-B pieces of the same 128 output rows within a few microseconds (L2 merges them into
// long DRAM bursts: with n-tile-major order the label GEMM wrote at 2.2 TB/s, with contiguous 4 KB runs at 4.2 TB/s),
// and the W_out tiles of a group (NT_GROUP x 64 KB) are re-read from L2 by the n_mt m-tiles.
// Lane order (per_m > 0, what the launcher picks whenever n_mt * per_m CTAs cover >= 95 % of the SMs): CTA c owns m-tile
// c % n_mt for the whole launch and walks the n-tiles of slice c / n_mt of the label range one after the other.  The n_mt
// CTAs of a slice (adjacent CTA ids, same pace) ask for the same W_out tile within a few microseconds: one DRAM read and
// n_mt - 1 L2 hits, where the group order re-read the whole 100 MB image n_mt times at C = 195,299 (the 800 MB of streaming
// logits evict a group's tiles between a CTA's visits: 809 MB read per launch under ncu); and every CTA extends each of its
// 128 output rows by 512 contiguous bytes per tile.
struct LtTile { long long nt; int mt; };
struct LtRange { long long t_lo; int my_tiles; int mt; };         // lane order: t_lo = first n-tile, mt fixed; group order: mt = -1
__device__ __forceinline__ LtRange lt_range(long long n_tiles, int n_mt, long long n_nt, int per_m) {
    LtRange r;
    if (per_m > 0) {
        const int slice = (int)blockIdx.x / n_mt;
        r.mt = (int)blockIdx.x % n_mt;
        if (slice >= per_m) { r.t_lo = 0; r.my_tiles = 0; return r; }
        r.t_lo = n_nt * slice / per_m;
        r.my_tiles = (int)(n_nt * (slice + 1) / per_m - r.t_lo);
        return r;
    }
    r.mt = -1;
    r.t_lo = n_tiles * blockIdx.x / gridDim.x;
    r.my_tiles = (int)(n_tiles * (blockIdx.x + 1) / gridDim.x - r.t_lo);
    return r;
}
__device__ __forceinline__ LtTile lt_tile(long long t, int n_mt, long long n_nt, int group) {
    const long long per_group = (long long)group * n_mt;
    const long long g = t / per_group;
    const long long rem = t - g * per_group;
    long long gs = n_nt - g * group; if (gs > group) gs = group;           // the last group may be narrower
    LtTile r;
    r.mt = (int)(rem / gs);
    r.nt = g * group + (rem - (long long)r.mt * gs);
    return r;
}

// Loss fusion (SURVEY.md 8f row 1, main.py:251-264): what the epilogue adds when the caller wants the mean NLL without
// re-reading (or without ever writing) the [B, C] logits.
//   part != NULL : per (row, n-tile, 32-column block) the block's (max, sum exp(v - max)) -> part[(nt * 4 + cq) * Mpad + row],
//                  and the target logit v[row, label[row]] -> tgt[row]; merged by loss_partials_reduce / loss_finalize.
//   lse  != NULL : dlogits mode (backward): the value stored is (exp(v - lse[row]) - [col == label[row]]) * dscale
//                  instead of the logit (main.py:174 through log_softmax + NLLLoss, weights == 1).
struct LtLoss {
    float2 *part; float *tgt; const long long *label; const float *lse; const float *dscale_ptr; float dscale; int Mpad;
    unsigned *gmax_bits;      // dlogits mode: bits of max |value stored| over the launch (what the label backward's fp16 split scales by)
};
constexpr float LT_LOG2E = 1.4426950408889634f;
__device__ __forceinline__ float lt_ex2(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

namespace lt2 {
constexpr int NT_GROUP = 8;
constexpr int N_EPI_WARPS = 16;                 // warp w: TMEM lane quarter w & 3, column quarter w >> 2 (32 columns)
constexpr int LOAD_WARP = 16, MMA_WARP = 17;
constexpr int THREADS = 18 * 32;
constexpr int OP_STAGES = 2, ACC_STAGES = 4;
constexpr int STAGE_BYTES = 4 * lt::TILE_BYTES;              // one k-block: {A_hi, A_lo | B_hi, B_lo}, 64 KB
constexpr int STG_LD = 36;                                   // padded fp32 row of a warp's [32 x 32] staging tile
constexpr int BAND_LD = 132;                                 // padded fp32 row of a row band's [32 x 128] staging tile (4 warps)
constexpr int STG_BYTES = N_EPI_WARPS * 32 * STG_LD * 4;     // 72 KB
constexpr int MAX_MT = 16;                                   // running arg-max table: 16 m-tiles x 128 rows x u64
constexpr int TAB_BYTES = MAX_MT * 128 * 8;
constexpr int SMEM_STG_OFF = OP_STAGES * STAGE_BYTES;
constexpr int SMEM_TAB_OFF = SMEM_STG_OFF + STG_BYTES;
constexpr int SMEM_BIAS_OFF = SMEM_TAB_OFF + TAB_BYTES;      // [16 warps][32] bias of the current tile
constexpr int SMEM_BAR_OFF = SMEM_BIAS_OFF + N_EPI_WARPS * 32 * 4;
constexpr int SMEM_BYTES = SMEM_BAR_OFF + 128 + 1024;
}  // namespace lt2

// K2 v2: persistent label GEMM with the arg-max folded in.  The 128 x 128 output tiles are numbered n-tile major /
// m-tile minor and cut into one contiguous range per CTA (all SMs busy for any B, C; a CTA's consecutive tiles share
// their W_out tile, which is therefore read from HBM once and re-read from L2).  Warp 16 streams {cv tile, W_out tile}
// k-block images through a 2-stage ring (one 32 KB cp.async.bulk each), warp 17 issues 12 tcgen05.mma per k-block into one of
// four TMEM accumulators, 16 epilogue warps (32 rows x 32 columns each) do TMEM -> registers -> *1/scale + bias ->
// running arg-max (smem table, 64-bit atomicMax) -> padded smem tile -> row-contiguous 128-B stores.
// Bound: the logits write (B*C*4 bytes); the arg-max costs no extra pass over them.
__global__ void __launch_bounds__(lt2::THREADS, 1)
label_gemm_v2_kernel(const uint8_t *__restrict__ imgA, const uint8_t *__restrict__ imgB,
                     const float *__restrict__ bias, const float *__restrict__ hdr, float *__restrict__ out,
                     int M, long long N, int nkb, int n_mt, long long n_nt, long long n_tiles,
                     unsigned long long *__restrict__ keys, unsigned *__restrict__ ticket,
                     long long *__restrict__ argmax, float *__restrict__ maxval, const LtLoss ls, const int per_m)
{
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = lt_smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char *smem = smem_raw + (base - raw);
    float *stage_all = reinterpret_cast<float *>(smem + lt2::SMEM_STG_OFF);
    unsigned long long *tab = reinterpret_cast<unsigned long long *>(smem + lt2::SMEM_TAB_OFF);
    const uint32_t bars = base + lt2::SMEM_BAR_OFF;
    // op_full[2] @0, op_empty[2] @16, t_full[4] @32, t_empty[4] @64, tmem ptr @96
    const uint32_t bar_ofull = bars, bar_oempty = bars + 16, bar_tfull = bars + 32, bar_tempty = bars + 64;
    uint32_t *tmem_ptr_smem = reinterpret_cast<uint32_t *>(smem + lt2::SMEM_BAR_OFF + 96);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const LtRange rg = lt_range(n_tiles, n_mt, n_nt, per_m);
    const long long t_lo = rg.t_lo;
    const int my_tiles = rg.my_tiles;
    auto tile_of = [&](int i) {
        if (rg.mt >= 0) { LtTile r; r.nt = t_lo + i; r.mt = rg.mt; return r; }
        return lt_tile(t_lo + i, n_mt, n_nt, lt2::NT_GROUP);
    };
    const bool want_arg = keys != nullptr;

    if (tid == 0) {
        for (int s = 0; s < lt2::OP_STAGES; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_ofull + 8 * s));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_oempty + 8 * s));
        }
        for (int s = 0; s < lt2::ACC_STAGES; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_tfull + 8 * s));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_tempty + 8 * s), "r"((uint32_t)lt2::N_EPI_WARPS));
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (want_arg)
        for (int i = tid; i < lt2::MAX_MT * 128; i += lt2::THREADS) tab[i] = 0ull;
    if (warp == lt2::MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(lt_smem_u32(tmem_ptr_smem)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_ptr_smem;
    pdl_wait();                                   // everything above overlapped the tail of the cv-image kernel

    const int kb_bytes = 2 * lt::TILE_BYTES;                          // {hi, lo} of one k-block of one operand
    if (warp == lt2::LOAD_WARP) {
        if (lane == 0) {
            int it = 0;
            for (int i = 0; i < my_tiles; ++i) {
                const LtTile tt = tile_of(i);
                const long long nt = tt.nt; const int mt = tt.mt;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int st = it & 1;
                    const uint32_t dst = base + st * lt2::STAGE_BYTES;
                    lt_mbar_wait(bar_oempty + 8 * st, ((uint32_t)(it >> 1) & 1u) ^ 1u);
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_ofull + 8 * st), "r"((uint32_t)(2 * kb_bytes)) : "memory");
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                 ::"r"(dst), "l"(imgA + ((size_t)mt * nkb + kb) * kb_bytes), "r"((uint32_t)kb_bytes), "r"(bar_ofull + 8 * st) : "memory");
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                 ::"r"(dst + kb_bytes), "l"(imgB + ((size_t)nt * nkb + kb) * kb_bytes), "r"((uint32_t)kb_bytes), "r"(bar_ofull + 8 * st) : "memory");
                }
            }
        }
        __syncwarp();
    } else if (warp == lt2::MMA_WARP) {
        // converged warp, one elected lane issues (a divergent `if (lane == 0)` makes ptxas wrap every UTCHMMA in an
        // ELECT / BRA.U.ANY loop and rebuild the descriptors through R2UR: the issuer becomes the slowest stage)
        auto desc = [](uint32_t a) {
            return (uint64_t)((a & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
        };
        int it = 0;
        for (int i = 0; i < my_tiles; ++i) {
            const int acc = i & (lt2::ACC_STAGES - 1);
            lt_mbar_wait(bar_tempty + 8 * acc, ((uint32_t)(i / lt2::ACC_STAGES) & 1u) ^ 1u);
            const uint32_t d_tmem = tmem + (uint32_t)(acc * lt::TN);
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int st = it & 1;
                lt_mbar_wait(bar_ofull + 8 * st, (uint32_t)(it >> 1) & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (lt_elect_one()) {
                    const uint64_t a0 = desc(base + st * lt2::STAGE_BYTES);
                    const uint64_t b0 = a0 + (uint64_t)(kb_bytes >> 4);
#pragma unroll
                    for (int k = 0; k < lt::KB / 16; ++k) {
                        const uint64_t a_hi = a0 + (uint64_t)(k * 2), a_lo = a_hi + (lt::TILE_BYTES >> 4);
                        const uint64_t b_hi = b0 + (uint64_t)(k * 2), b_lo = b_hi + (lt::TILE_BYTES >> 4);
                        auto mma = [&](uint64_t ad, uint64_t bd, uint32_t accum) {
                            asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                                         "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                                         ::"r"(d_tmem), "l"(ad), "l"(bd), "r"(lt::IDESC), "r"(accum) : "memory");
                        };
                        mma(a_hi, b_hi, (kb | k) != 0 ? 1u : 0u);
                        mma(a_lo, b_hi, 1u);
                        mma(a_hi, b_lo, 1u);
                    }
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_oempty + 8 * st) : "memory");
                    if (kb == nkb - 1)
                        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_tfull + 8 * acc) : "memory");
                }
                __syncwarp();
            }
        }
    } else {
        // ---- epilogue: thread = output row (TMEM lane) x 32 columns.  Bounds and addresses are hoisted out of the
        //      per-element code (the first version spent 1100 instructions per warp and tile, 60 % issue-bound).
        const int q = warp & 3, cq = warp >> 2;
        const float inv_scale = hdr[0];
        const bool vec_ok = (N % 4 == 0);
        float *stg = stage_all + warp * 32 * lt2::STG_LD;
        float *sbias = reinterpret_cast<float *>(smem + lt2::SMEM_BIAS_OFF) + warp * 32;
        float gmax = 0.0f;                                    // dlogits mode: running max |d logit| of this thread
        // bias of the NEXT tile's 32 columns is fetched one tile ahead (a dependent global load at the top of every tile
        // otherwise sits on each warp's critical path: ~0.7 us of the ~4 us a tile takes)
        auto bias_of = [&](int i) {
            if (!bias || i >= my_tiles) return 0.0f;
            const LtTile t2 = tile_of(i);
            const long long c2 = t2.nt * lt::TN + cq * 32 + lane;
            return c2 < N ? __ldg(bias + c2) : 0.0f;
        };
        float bias_next = bias_of(0);
        for (int i = 0; i < my_tiles; ++i) {
            const LtTile tt = tile_of(i);
            const long long nt = tt.nt; const int mt = tt.mt;
            const int acc = i & (lt2::ACC_STAGES - 1);
            const long long col0 = nt * lt::TN + cq * 32;              // first column of this warp's block
            const long long row0 = (long long)mt * lt::TM + q * 32;    // first row
            const int n_cols = (int)(N - col0 < 32 ? N - col0 : 32);   // valid columns / rows of the block (may be <= 0)
            const int n_rows = (int)(M - row0 < 32 ? M - row0 : 32);
            // bias of this warp's 32 columns: one element per lane -> smem -> broadcast float4 reads
            sbias[lane] = bias_next;
            __syncwarp();
            bias_next = bias_of(i + 1);
            lt_mbar_wait(bar_tfull + 8 * acc, (uint32_t)(i / lt2::ACC_STAGES) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * lt::TN + cq * 32);
            uint32_t r[32];
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                         "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                         "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                         : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                           "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                           "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                           "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                         : "r"(taddr));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_tempty + 8 * acc) : "memory");
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; j += 4) {                                                       // model.py:83
                const float4 b4 = *reinterpret_cast<const float4 *>(sbias + j);
                v[j] = fmaf(__uint_as_float(r[j]), inv_scale, b4.x); v[j + 1] = fmaf(__uint_as_float(r[j + 1]), inv_scale, b4.y);
                v[j + 2] = fmaf(__uint_as_float(r[j + 2]), inv_scale, b4.z); v[j + 3] = fmaf(__uint_as_float(r[j + 3]), inv_scale, b4.w);
            }
            if (ls.part || ls.lse) {
                const long long grow = row0 + lane;                                     // this thread's output row
                const long long lab = (grow < M && ls.label) ? ls.label[grow] : -1;
                const long long tj = lab - col0;                                        // label's column inside this block
                if (ls.part) {
                    float m = -INFINITY, ssum = 0.0f;
#pragma unroll
                    for (int j = 0; j < 32; ++j) m = fmaxf(m, j < n_cols ? v[j] : -INFINITY);
                    const float mb = m * LT_LOG2E;
#pragma unroll
                    for (int j = 0; j < 32; ++j) ssum += j < n_cols ? lt_ex2(fmaf(v[j], LT_LOG2E, -mb)) : 0.0f;
                    ls.part[(size_t)(nt * 4 + cq) * ls.Mpad + grow] = make_float2(m, n_cols > 0 ? ssum : 0.0f);
                    if (__any_sync(0xffffffffu, tj >= 0 && tj < n_cols)) {
                        // select chain in PTX: written in C++ the compiler turns it into v[tj], a dynamically indexed read
                        // that puts all of v[] in local memory -- 8 x STL.128 per thread and tile in EVERY mode of this
                        // kernel (64 KB of local stores per tile and SM, as much as the logits themselves)
                        float t = 0.0f;
                        const int tji = (int)tj;
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.s32 p, %2, %3;\n\tselp.f32 %0, %1, %0, p;\n\t}"
                                         : "+f"(t) : "f"(v[j]), "r"(tji), "r"(j));
                        if (tj >= 0 && tj < n_cols) ls.tgt[grow] = t;
                    }
                }
                if (ls.lse) {                                                           // dlogits (overwrites v)
                    const float lb = (grow < M ? ls.lse[grow] : 0.0f) * LT_LOG2E;
                    const float sc = ls.dscale_ptr ? ls.dscale * *ls.dscale_ptr : ls.dscale;
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = (lt_ex2(fmaf(v[j], LT_LOG2E, -lb)) - ((j == (int)tj) ? 1.0f : 0.0f)) * sc;
                    if (ls.gmax_bits && grow < M) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) gmax = fmaxf(gmax, j < n_cols ? fabsf(v[j]) : 0.0f);
                    }
                }
            }
            if (want_arg && lane < n_rows && n_cols > 0) {
                float m = -INFINITY;
                if (n_cols == 32) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) m = fmaxf(m, v[j]);
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) m = fmaxf(m, j < n_cols ? v[j] : -INFINITY);
                }
                unsigned long long *slot = tab + mt * 128 + q * 32 + lane;
                const uint32_t mk = lt_orderable(m);
                if (mk >= (uint32_t)(*reinterpret_cast<volatile unsigned long long *>(slot) >> 32)) {
                    int jm = 31;
#pragma unroll
                    for (int j = 31; j >= 0; --j) jm = (v[j] == m && j < n_cols) ? j : jm;        // first maximum
                    atomicMax(slot, ((unsigned long long)mk << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)(col0 + jm)));
                }
            }
            if (out == nullptr) { __syncwarp(); continue; }   // loss-only mode: the logits are never written
            if (!vec_ok) {
                // Rows that are only 4-byte aligned (label_count % 4 != 0, e.g. top11's 195,299): the four column-quarter
                // warps of a row band stage the whole [32 rows x 128 columns] band, then every warp writes 8 rows of it in
                // segments that start on 128-byte boundaries of GLOBAL memory (5 store instructions per row instead of 4;
                // only the tile's two edge sectors per row stay partial).  Per-warp 128-B pieces at the row's own misalignment
                // wrote every sector in two halves: 412 us instead of 318 us for the 800 MB of logits at that label count.
                float *band = stage_all + q * (32 * lt2::BAND_LD);
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4 *>(band + lane * lt2::BAND_LD + cq * 32 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                asm volatile("bar.sync %0, 128;" ::"r"(1 + q) : "memory");
                const long long base_col = nt * lt::TN;
                const int tile_cols = (int)(N - base_col < lt::TN ? N - base_col : lt::TN);
#pragma unroll 1
                for (int rr = cq * 8; rr < cq * 8 + 8; ++rr) {
                    const long long grow = (long long)mt * lt::TM + q * 32 + rr;
                    if (grow >= M) break;
                    float *grow_p = out + (size_t)grow * N + base_col;
                    const int a = (int)(((size_t)grow * N + base_col) & 31);        // floats past a 128-byte boundary
                    const float *sp = band + rr * lt2::BAND_LD;
#pragma unroll
                    for (int sg = 0; sg < 5; ++sg) {
                        const int col = sg * 32 - a + lane;
                        if (col >= 0 && col < tile_cols) grow_p[col] = sp[col];
                    }
                }
                asm volatile("bar.sync %0, 128;" ::"r"(1 + q) : "memory");     // the band is restaged by the next tile
                continue;
            }
            // registers -> padded smem tile (thread = row), then row-contiguous stores
#pragma unroll
            for (int j = 0; j < 32; j += 4)
                *reinterpret_cast<float4 *>(stg + lane * lt2::STG_LD + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            __syncwarp();
            if (n_rows > 0 && n_cols > 0) {
                if (vec_ok && n_cols == 32) {
                    const int rr0 = lane >> 3, c4 = (lane & 7) * 4;          // 4 rows x 128 B per store instruction
                    float *gp = out + (size_t)(row0 + rr0) * N + col0 + c4;
                    const float *sp = stg + rr0 * lt2::STG_LD + c4;
                    const size_t gstep = (size_t)4 * N;
#pragma unroll
                    for (int it = 0; it < 8; ++it) {
                        if (it * 4 + rr0 < n_rows) *reinterpret_cast<float4 *>(gp) = *reinterpret_cast<const float4 *>(sp + it * 4 * lt2::STG_LD);
                        gp += gstep;
                    }
                } else if (lane < n_cols) {                                  // one <= 128-B row segment per store instruction
                    float *gp = out + (size_t)row0 * N + col0 + lane;
                    const float *sp = stg + lane;
#pragma unroll
                    for (int rr = 0; rr < 32; ++rr) {
                        if (rr < n_rows) *gp = sp[rr * lt2::STG_LD];
                        gp += N;
                    }
                }
            }
            __syncwarp();                         // staging tile is rewritten by the next tile
        }
        if (ls.lse && ls.gmax_bits) {                 // one atomic per warp and launch (non-negative floats order as uints)
            gmax = warp_max(gmax);
            if (lane == 0 && gmax > 0.0f && gmax < 3.0e38f) atomicMax(ls.gmax_bits, __float_as_uint(gmax));
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == lt2::MMA_WARP) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
    }
    if (want_arg) {
        // flush this CTA's table, then the last CTA to arrive decodes keys -> (argmax, maxval)
        __shared__ unsigned s_last;
        for (int i = tid; i < n_mt * 128; i += lt2::THREADS) {
            const unsigned long long k = tab[i];
            if (k != 0ull && i < M) atomicMax(keys + i, k);
        }
        __threadfence();
        __syncthreads();
        if (tid == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1 ? 1u : 0u;
        __syncthreads();
        if (s_last) {
            __threadfence();
            for (int b = tid; b < M; b += lt2::THREADS) {
                const unsigned long long k = *reinterpret_cast<volatile unsigned long long *>(keys + b);
                if (argmax) argmax[b] = (long long)(0xFFFFFFFFu - (uint32_t)(k & 0xFFFFFFFFull));
                if (maxval) maxval[b] = lt_from_orderable((uint32_t)(k >> 32));
            }
        }
    }
}

// ---- merging the loss partials: (max, sum exp) pairs are merged online-softmax style ----------------------------------
__device__ __forceinline__ void lt_merge(float &M, float &S, float m, float sv) {
    if (m > M) { S = S * __expf(M - m) + sv; M = m; }          // (M = -inf, S = 0 start: exp(-inf) = 0)
    else if (m > -INFINITY) S += sv * __expf(m - M);
}
constexpr int LT_PSPLIT = 16;
// grid (Mpad / 32, LT_PSPLIT), 256 threads: lane = row, the 8 warps stride over this CTA's share of the partial index
__global__ void __launch_bounds__(256)
loss_partials_reduce_kernel(const float2 *__restrict__ part, int P, int Mpad, float2 *__restrict__ part2)
{
    __shared__ float2 sh[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int row = blockIdx.x * 32 + lane;
    const int p0 = (int)((long long)P * blockIdx.y / gridDim.y), p1 = (int)((long long)P * (blockIdx.y + 1) / gridDim.y);
    float M = -INFINITY, S = 0.0f;
    for (int p = p0 + warp; p < p1; p += 8) {
        const float2 v = part[(size_t)p * Mpad + row];
        lt_merge(M, S, v.x, v.y);
    }
    sh[warp][lane] = make_float2(M, S);
    __syncthreads();
    if (warp == 0) {
        for (int w = 1; w < 8; ++w) lt_merge(M, S, sh[w][lane].x, sh[w][lane].y);      // fixed order: deterministic
        part2[(size_t)blockIdx.y * Mpad + row] = make_float2(M, S);
    }
}
// one CTA: lse[b] = M + log S, loss = mean_b (lse[b] - target logit[b])   (main.py:251-264 with weights == 1)
__global__ void __launch_bounds__(1024)
loss_finalize_kernel(const float2 *__restrict__ part2, int nsplit, int Mpad, const float *__restrict__ tgt, int B,
                     float *__restrict__ lse, float *__restrict__ loss)
{
    __shared__ float red[32];
    float acc = 0.0f;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        float M = -INFINITY, S = 0.0f;
        for (int k = 0; k < nsplit; ++k) { const float2 v = part2[(size_t)k * Mpad + b]; lt_merge(M, S, v.x, v.y); }
        const float l = M + logf(S);
        if (lse) lse[b] = l;
        acc += l - tgt[b];
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0f;
        v = warp_sum(v);
        if (threadIdx.x == 0 && loss) *loss = v / (float)B;
    }
}

// K (= encode_size) is zero-padded to a multiple of 64 inside the operand images
bool label_tcgen05_shape_ok(const c2v_dims *d) { return d->encode >= 4 && d->encode <= 256 && (d->encode & 3) == 0; }

// ticket (first 64 bytes) + arg-max keys [B] u64.  This region sits AFTER the W_out image: the image is reused across calls
// while the weights are unchanged (C2V_FLAG_REUSE_PREP), so its offset must not depend on the batch size (a ragged last
// batch of an evaluation pass has a different B).
static size_t lt_keys_bytes(int B) { return (64 + (size_t)B * 8 + 1023) / 1024 * 1024; }

// loss partials (behind the cv image): part [nt * 4][Mpad] float2 | part2 [LT_PSPLIT][Mpad] float2 | tgt [Mpad] float
static size_t lt_loss_bytes(int B, long long C)
{
    const size_t Mpad = (size_t)(B + 127) / 128 * 128, nt = (size_t)((C + 127) / 128);
    return (nt * 4 + LT_PSPLIT) * Mpad * sizeof(float2) + Mpad * sizeof(float) + 1024;
}
size_t label_tcgen05_workspace_bytes(const c2v_dims *d, int B)
{
    const size_t nkb = (size_t)(d->encode + 63) / 64;
    const size_t mt = (size_t)(B + 127) / 128, nt = (size_t)(d->label_count + 127) / 128;
    return 1024 + lt_keys_bytes(B) + (mt + nt) * nkb * 2 * lt::TILE_BYTES + lt_loss_bytes(B, d->label_count);
}

int launch_loss_argmax(const float *out, const long long *label, int B, long long C, float *loss,
                       long long *argmax, float *maxval, float *d_out, cudaStream_t st);

// argmax / maxval (torch.max(dim=1), main.py:285) are folded into the GEMM epilogue (label_gemm_v2_kernel) for up to
// 16 m-tiles (B <= 2048); beyond that they are a second pass over the logits.
int launch_label_tcgen05_ex(const c2v_dims *d, const float *cv, int B, const float *Wout, const float *bias,
                            float *out, long long *argmax, float *maxval, void *ws, size_t ws_bytes, bool reuse_prep,
                            cudaStream_t st, const LabelLossArgs *la);

// The cached W_out image of a label workspace (built here unless reuse_prep): what the tensor-core label backward streams.
int label_w_image(const c2v_dims *d, const float *Wout, int B, void *ws, size_t ws_bytes, bool reuse_prep, cudaStream_t st,
                  const uint8_t **img, const float **hdr, unsigned **scratch, const uint8_t **cv_img)
{
    if (!label_tcgen05_shape_ok(d) || !ws || ws_bytes < label_tcgen05_workspace_bytes(d, B)) {
        set_error("label backward: workspace missing or too small");
        return C2V_EWORKSPACE;
    }
    const int H = d->encode, nkb = (H + 63) / 64;
    const long long C = d->label_count;
    uint8_t *p = static_cast<uint8_t *>(ws);
    float *h = reinterpret_cast<float *>(p);
    unsigned *mxbits = reinterpret_cast<unsigned *>(p + 256);
    uint8_t *imgB = p + 1024;
    if (!reuse_prep) {
        int dev = 0, sms = 0;
        C2V_CUDA_OK(cudaGetDevice(&dev));
        C2V_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        C2V_CUDA_OK(cudaMemsetAsync(mxbits, 0, 4, st));
        absmax_kernel<<<sms * 4, 256, 0, st>>>(Wout, C * H, mxbits);
        C2V_LAUNCH_OK("absmax_kernel");
        split_rows_kernel<<<sms * 8, 256, 0, st>>>(Wout, C, H, nkb, mxbits, imgB, h, nullptr, 0);
        C2V_LAUNCH_OK("split_rows_kernel");
    }
    *img = imgB; *hdr = h; *scratch = reinterpret_cast<unsigned *>(p + 768);
    // where launch_label_tcgen05_ex keeps the fp16 image of the code vectors of its last call with this B (same layout math)
    if (cv_img) *cv_img = imgB + (size_t)((C + 127) / 128) * nkb * 2 * lt::TILE_BYTES + lt_keys_bytes(B);
    return C2V_OK;
}

int launch_label_tcgen05(const c2v_dims *d, const float *cv, int B, const float *Wout, const float *bias,
                         float *out, long long *argmax, float *maxval, void *ws, size_t ws_bytes, bool reuse_prep,
                         cudaStream_t st)
{
    return launch_label_tcgen05_ex(d, cv, B, Wout, bias, out, argmax, maxval, ws, ws_bytes, reuse_prep, st, nullptr);
}

// What the last label GEMM launched from this host thread left in its workspace: the fp16 image of `cv` (every call) and, in
// dlogits mode, max |d logit|.  c2v_label_backward_ws only believes C2V_FLAG_GRAD_ABSMAX_READY when this record matches its
// own workspace / code_vector / B -- a wrong flag then costs the skipped shortcuts, not the result.
static thread_local struct { const void *ws; const float *cv; int B; bool dlogits; } g_label_last = {nullptr, nullptr, 0, false};
bool label_ws_holds_dlogits_of(const void *ws, const float *cv, int B)
{
    return g_label_last.dlogits && g_label_last.ws == ws && g_label_last.cv == cv && g_label_last.B == B;
}

// la != NULL: la->loss (mean NLL) / la->lse [B] are produced from the fused partials (out may then be NULL: the logits
// are never written); la->dlogits_lse != NULL: `out` receives d(loss)/d(logits) instead of the logits.
int launch_label_tcgen05_ex(const c2v_dims *d, const float *cv, int B, const float *Wout, const float *bias,
                            float *out, long long *argmax, float *maxval, void *ws, size_t ws_bytes, bool reuse_prep,
                            cudaStream_t st, const LabelLossArgs *la)
{
    if (!label_tcgen05_shape_ok(d)) {
        set_error("tcgen05 label GEMM needs encode_size %% 4 == 0 and <= 256 (got %d)", d->encode);
        return C2V_EUNSUPPORTED;
    }
    const int H = d->encode, nkb = (H + 63) / 64;
    const long long C = d->label_count;
    if (!ws || ws_bytes < label_tcgen05_workspace_bytes(d, B)) {
        set_error("label workspace too small: %zu < %zu", ws_bytes, label_tcgen05_workspace_bytes(d, B));
        return C2V_EWORKSPACE;
    }
    g_label_last.ws = ws; g_label_last.cv = cv; g_label_last.B = B; g_label_last.dlogits = la && la->dlogits_lse;
    uint8_t *p = static_cast<uint8_t *>(ws);
    float *hdr = reinterpret_cast<float *>(p);
    unsigned *mxbits = reinterpret_cast<unsigned *>(p + 256);

    const size_t mt = (size_t)(B + 127) / 128, nt = (size_t)((C + 127) / 128);
    // W_out image first (reusable across calls while the weights are unchanged), then the cv image
    uint8_t *imgB = p + 1024;                                           // batch-size independent offset
    uint8_t *key_region = imgB + nt * nkb * 2 * lt::TILE_BYTES;
    unsigned *ticket = reinterpret_cast<unsigned *>(key_region);
    unsigned long long *keys = reinterpret_cast<unsigned long long *>(key_region + 64);
    uint8_t *imgA = key_region + lt_keys_bytes(B);
    const int Mpad = (int)mt * 128;
    float2 *part = reinterpret_cast<float2 *>(imgA + mt * nkb * 2 * lt::TILE_BYTES);
    float2 *part2 = part + nt * 4 * (size_t)Mpad;
    float *tgt = reinterpret_cast<float *>(part2 + (size_t)LT_PSPLIT * Mpad);
    LtLoss ls;
    memset(&ls, 0, sizeof(ls));
    ls.Mpad = Mpad;
    const bool want_loss = la && (la->loss || la->lse_out);
    if (want_loss) {
        if (!la->label) { set_error("label loss: label is NULL"); return C2V_EINVAL; }
        ls.part = part; ls.tgt = tgt; ls.label = la->label;
        // a label outside [0, C) leaves its target logit unwritten: NaN then makes the loss NaN (the reference's NLLLoss
        // raises "Target out of bounds")
        C2V_CUDA_OK(cudaMemsetAsync(tgt, 0xFF, (size_t)Mpad * sizeof(float), st));
    }
    if (la && la->dlogits_lse) {
        if (!la->label || !out) { set_error("label dlogits: label / output is NULL"); return C2V_EINVAL; }
        ls.lse = la->dlogits_lse; ls.label = la->label; ls.dscale = la->dscale; ls.dscale_ptr = la->dscale_ptr;
        // max |d logit| for the label backward (c2v_label_backward_ws with C2V_FLAG_GRAD_ABSMAX_READY skips its own pass
        // over the [B, C] gradient: 220 us at C = 195,299); same word label_w_image hands to the backward as `scratch`
        ls.gmax_bits = reinterpret_cast<unsigned *>(p + 768);
        C2V_CUDA_OK(cudaMemsetAsync(ls.gmax_bits, 0, 4, st));
    }
    const bool want_arg = argmax || maxval;
    const bool fused_arg = want_arg && mt <= (size_t)lt2::MAX_MT;
    int dev = 0, sms = 0;
    C2V_CUDA_OK(cudaGetDevice(&dev));
    C2V_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));

    if (!reuse_prep) {
        C2V_CUDA_OK(cudaMemsetAsync(mxbits, 0, 4, st));
        absmax_kernel<<<sms * 4, 256, 0, st>>>(Wout, C * H, mxbits);
        C2V_LAUNCH_OK("absmax_kernel");
        split_rows_kernel<<<sms * 8, 256, 0, st>>>(Wout, C, H, nkb, mxbits, imgB, hdr, nullptr, 0);
        C2V_LAUNCH_OK("split_rows_kernel");
    }
    // cv image (+ zeroes the ticket and the arg-max keys, which sit contiguously in key_region)
    C2V_CUDA_OK(launch_pdl(split_rows_kernel, dim3((unsigned)((mt * 128 * nkb * 16 + 255) / 256)), dim3(256), 0, st, cv,
                           (long long)B, H, nkb, (const unsigned *)nullptr, imgA, hdr,
                           reinterpret_cast<unsigned long long *>(key_region), fused_arg ? 8 + B : 0));
    C2V_COUNT_LAUNCH();

    C2V_CUDA_OK(cudaFuncSetAttribute(label_gemm_v2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, lt2::SMEM_BYTES));
    const long long n_tiles = (long long)mt * (long long)nt;
    const int grid = (int)(n_tiles < sms ? n_tiles : sms);
    // tile order (see lt_range): lanes when that keeps >= 95 % of the CTAs busy, else groups
    int per_m = (mt <= (size_t)grid) ? grid / (int)mt : 0;
    if (per_m > 0 && (long long)per_m * (long long)mt * 100 < 95ll * grid) per_m = 0;
    C2V_CUDA_OK(launch_pdl(label_gemm_v2_kernel, dim3((unsigned)grid), dim3(lt2::THREADS), (size_t)lt2::SMEM_BYTES, st,
                           (const uint8_t *)imgA, (const uint8_t *)imgB, bias, (const float *)hdr, out, B, C, nkb, (int)mt,
                           (long long)nt, n_tiles, fused_arg ? keys : (unsigned long long *)nullptr, ticket,
                           fused_arg ? argmax : (long long *)nullptr, fused_arg ? maxval : (float *)nullptr, ls, per_m));
    C2V_LAUNCH_OK("label_gemm_v2_kernel");
    if (want_loss) {
        loss_partials_reduce_kernel<<<dim3((unsigned)(Mpad / 32), LT_PSPLIT), 256, 0, st>>>(part, (int)(nt * 4), Mpad, part2);
        C2V_LAUNCH_OK("loss_partials_reduce_kernel");
        loss_finalize_kernel<<<1, 1024, 0, st>>>(part2, LT_PSPLIT, Mpad, tgt, B, la->lse_out, la->loss);
        C2V_LAUNCH_OK("loss_finalize_kernel");
    }
    if (want_arg && !fused_arg) {
        if (!out) { set_error("label loss without logits: arg-max needs B <= %d", lt2::MAX_MT * 128); return C2V_EUNSUPPORTED; }
        return launch_loss_argmax(out, nullptr, B, C, nullptr, argmax, maxval, nullptr, st);
    }
    return C2V_OK;
}

}  // namespace c2v
