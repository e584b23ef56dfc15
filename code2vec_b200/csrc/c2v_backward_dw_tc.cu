// c2v_backward_dw_tc.cu -- K3b: dW = dX^T . C on the tensor cores (terminal_embed = path_embed = E <= 256, encode = H <= 256,
// both multiples of 4: the reference's default 100/100/100 runs here with the panels zero-padded to 128; sizes above 128
// run as 128-wide windows of h and of d, one window pair per blockIdx.y -- see "windows" below).
//
// The weight gradient of input_linear (what autograd computes for model.py:54 under loss.backward(), main.py:174):
//   dW[h, d] = sum over context rows r of dX[r, h] * C[r, d],   C[r] = [E_t[s_r]; E_p[p_r]; E_t[e_r]]
// i.e. a [128 x 384] output with K = B*L = 204,800 rows at cfg2: 20 GFLOP that the CUDA-core kernel (backward_dw_kernel)
// needs 1.05 ms for.  Here: M = h, N = d, K = rows -- both operands are "MN-major" (the row index is K, the 128
// columns of a row are contiguous).  The shared-memory image is the same [128 rows x 64 columns] fp16 SWIZZLE_128B
// panel the forward kernels build (one 128-byte line per row); only the descriptors change: major = MN in the
// instruction descriptor (bits 15, 16), LBO = stride between 64-column panels, SBO = 1024 B between 8-row groups, and a
// K step of 16 rows advances the start address by 2 KB.  Same 3-pass fp16 hi/lo split as everywhere else
// (dX and C are fp32; fp32 accumulation in TMEM).  dX is scaled by a power of two before the split, the gathered C is
// split as it is: each element of C keeps an absolute precision of about 2^-25 (its lo half is an fp16 subnormal below
// 2^-14), so dW's relative error is about max(1e-6, 2^-25 / std(C)): by estimate 4e-6 at an embedding std of 2^-8
// (the smallest the tests use), 7.5e-5 at 2^-12.  |C| must stay below 65504 (fp16 overflow).  C is not scaled as well:
// embeddings at the reference's init (std 1) sit far inside that range (DESIGN.md "Numerics at the edges").
//
// One persistent CTA per SM walks 128-row tiles and keeps its partial dW [128 h x 384 d] in TMEM (384 columns) for
// the whole launch; at the end 4 warps add it to the global gradient with 128-bit vector atomics.
// Warps: 0-15 producers (8 rows each: LDG.128 -> hi/lo split -> STS.64; warps 0-3 also do the final reduction) | 16 MMA
// issuer.  17 warps leave 96 registers per thread: a producer keeps TWO panels of loads in flight (both dX panels of a tile
// before it waits for the stage; gathered panel kb+1 while it converts panel kb) -- with one panel at a time the eight
// dependent load -> convert -> store rounds per tile were the whole kernel (ncu: 40 % of the stall samples on the first
// use of a load, tensor pipe 26 %).
// smem: 2 tile-stages of the dX operand {hi p0, hi p1, lo p0, lo p1} (128 KB) + 2 slots of one gathered panel {hi, lo}
// (64 KB); per tile 6 gathered panels (start / path / end x 2 halves) stream through the slots: 144 MMAs (N = 64).
// Windows: blockIdx.y = hb * n_db + db selects rows h in [128 hb, 128 hb + 128) of dW and, inside each of the three
// sub-vectors, columns d in [128 db, 128 db + 128); the CTAs of one window pair (gridDim.x of them) share the row tiles.
// At E = H = 256 that is four window pairs: dX and the gathered rows are each read twice, the MMAs are the same 2 H D.
#include <cuda_fp16.h>

#include "c2v_tc_ptx.cuh"

namespace c2v {

namespace dwt {
constexpr int ROWS = 128, H = 128, E = 128, D = 3 * E;
constexpr int PANEL = ROWS * 64 * 2;                  // 16 KB: [128 rows x 64 cols] fp16
constexpr int A_STAGE = 4 * PANEL;                    // hi p0 | hi p1 | lo p0 | lo p1
constexpr int B_SLOT = 2 * PANEL;                     // hi | lo
constexpr int N_PROD_WARPS = 16, PROD_WARP0 = 0, MMA_WARP = 16;
constexpr int THREADS = 17 * 32;
constexpr int ROWS_PER_PW = ROWS / N_PROD_WARPS;      // 8
constexpr int NB = 6;                                 // gathered panels per tile
constexpr int SMEM_A_OFF = 0, SMEM_B_OFF = 2 * A_STAGE, SMEM_BAR_OFF = SMEM_B_OFF + 2 * B_SLOT;
constexpr int SMEM_BYTES = SMEM_BAR_OFF + 128 + 1024;
// kind::f16, D = f32, A and B MN-major, N = 64, M = 128
constexpr uint32_t IDESC = (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(ROWS >> 4) << 24);
}  // namespace dwt

// MN-major SWIZZLE_128B descriptor: LBO = byte stride between 64-element MN groups, SBO = between 8-row K groups
__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t saddr, uint32_t lbo_bytes) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) |
           (1ull << 46) | (2ull << 61);
}

__global__ void __launch_bounds__(dwt::THREADS, 1)
backward_dw_tc_kernel(const EncodeArgs a, const float *__restrict__ dx, const unsigned *__restrict__ dx_absmax,
                      float *__restrict__ dW, const int n_db)
{
    const int hb = (int)blockIdx.y / n_db, db = (int)blockIdx.y % n_db;       // this CTA's 128-wide windows of h and of d
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char *smem = smem_raw + (base - raw);
    const uint32_t bars = base + dwt::SMEM_BAR_OFF;
    // a_full[2] @0, a_empty[2] @16, b_full[2] @32, b_empty[2] @48, acc_full @64, tmem ptr @72
    const uint32_t bar_afull = bars, bar_aempty = bars + 16, bar_bfull = bars + 32, bar_bempty = bars + 48, bar_acc = bars + 64;
    uint32_t *tmem_ptr_smem = reinterpret_cast<uint32_t *>(smem + dwt::SMEM_BAR_OFF + 72);
    __shared__ long long s_status[2];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int my_tiles = (a.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    long long *status = s_status;                      // watchdog scratch of mbar_wait (no workspace status here)

    if (tid == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(bar_afull + 8 * s, 2 * dwt::N_PROD_WARPS);      // two panels per tile, one arrival per warp each
            mbar_init(bar_aempty + 8 * s, 1);
            mbar_init(bar_bfull + 8 * s, dwt::N_PROD_WARPS);
            mbar_init(bar_bempty + 8 * s, 1);
        }
        mbar_init(bar_acc, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == dwt::MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(tmem_ptr_smem)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;
    // Gradients are small (mean NLL over 1024 bags: |dx| ~ 1e-6) and would sit in fp16's subnormals: dX is multiplied by
    // the power of two that brings max |dx| (found by backward_rows_kernel) just below 2^14 before the hi/lo split, and
    // the accumulated dW by its exact inverse.
    float dx_scale = 1.0f;
    {
        const float mx = __uint_as_float(*dx_absmax);
        if (mx > 0.0f && mx < 3.0e38f) {
            int e;
            frexpf(mx, &e);
            int k = 14 - e;
            k = k > 100 ? 100 : (k < -100 ? -100 : k);
            dx_scale = ldexpf(1.0f, k);
        }
    }

    if (warp >= dwt::PROD_WARP0 && warp < dwt::MMA_WARP) {
        // =============================== PRODUCERS ===============================
        const int pw = warp - dwt::PROD_WARP0;        // rows 8*pw .. 8*pw+7 of every tile
        const int sub_row = lane >> 4, q = lane & 15; // lanes 0-15: row 2j, lanes 16-31: row 2j+1; q = 16-B column
        uint32_t st_off[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = pw * dwt::ROWS_PER_PW + 2 * j + sub_row;
            st_off[j] = (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((((q >> 1) ^ (r & 7)) & 7) << 4) + (q & 1) * 8);
        }
        auto split_store = [&](uint32_t hi, uint32_t lo, const float4 (&buf)[4]) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 v = buf[j];
                const __half2 h01 = __floats2half2_rn(v.x, v.y), h23 = __floats2half2_rn(v.z, v.w);
                const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
                const __half2 l01 = __floats2half2_rn(v.x - f01.x, v.y - f01.y);
                const __half2 l23 = __floats2half2_rn(v.z - f23.x, v.w - f23.y);
                sts_v2(hi + st_off[j], pack_h2(h01), pack_h2(h23));
                sts_v2(lo + st_off[j], pack_h2(l01), pack_h2(l23));
            }
        };
        const int E4 = a.Et / 4, H4 = a.H / 4;        // row lengths in 16-byte pieces (columns beyond them are zero padding)
        const int h04 = hb * 32, d04 = db * 32;       // window starts, in 16-byte pieces
        const float4 *tab_t = reinterpret_cast<const float4 *>(a.emb_t);
        const float4 *tab_p = reinterpret_cast<const float4 *>(a.emb_p);
        const float4 *dx4 = reinterpret_cast<const float4 *>(dx);
        int itb = 0;                                  // running gathered-panel counter (B ring position)
        for (int tl = 0; tl < my_tiles; ++tl) {
            const long long row0 = ((long long)blockIdx.x + (long long)tl * gridDim.x) * dwt::ROWS + pw * dwt::ROWS_PER_PW;
            // this lane's copy of the row indices of its warp's 8 rows (lane & 7)
            const long long myrow = row0 + (lane & 7);
            long long is = 0, ip = 0, ie = 0;
            if (myrow < a.N) { is = a.starts[myrow]; ip = a.paths[myrow]; ie = a.ends[myrow]; }
            // ---- dX operand: both panels (h 0..63, 64..127 of the window) in flight before the stage wait
            float4 buf[2][4];
#pragma unroll
            for (int p = 0; p < 2; ++p)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const long long r = row0 + 2 * j + sub_row;
                    buf[p][j] = (r < a.N && h04 + p * 16 + q < H4) ? ldg_nc_v4(dx4 + (size_t)r * H4 + h04 + p * 16 + q)
                                                                   : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            if (is < 0 || is >= a.T) is = 0;
            if (ip < 0 || ip >= a.P) ip = 0;
            if (ie < 0 || ie >= a.T) ie = 0;
            const uint32_t off_s = (uint32_t)(is * E4), off_p = (uint32_t)(ip * E4), off_e = (uint32_t)(ie * E4);
            const int as = tl & 1;
            mbar_wait(bar_aempty + 8 * as, (((uint32_t)(tl >> 1)) & 1u) ^ 1u, status);
#pragma unroll
            for (int p = 0; p < 2; ++p) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    buf[p][j].x *= dx_scale; buf[p][j].y *= dx_scale; buf[p][j].z *= dx_scale; buf[p][j].w *= dx_scale;
                }
                const uint32_t hi = base + dwt::SMEM_A_OFF + as * dwt::A_STAGE + p * dwt::PANEL;
                split_store(hi, hi + 2 * dwt::PANEL, buf[p]);
                fence_proxy_async_smem();             // writer side: generic-proxy stores -> visible to the tensor core's async proxy
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_afull + 8 * as);
            }
            // ---- gathered operand: 6 panels through the 2-slot ring, panel kb+1's loads in flight while kb is converted
            auto gather = [&](float4 (&dst)[4], int kb) {
                const int sv = kb >> 1;
                const float4 *tab = sv == 1 ? tab_p : tab_t;
                const uint32_t off = sv == 0 ? off_s : (sv == 1 ? off_p : off_e);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t o = __shfl_sync(0xffffffffu, off, 2 * j + sub_row);
                    const long long r = row0 + 2 * j + sub_row;
                    dst[j] = (r < a.N && d04 + (kb & 1) * 16 + q < E4) ? ldg_nc_v4(tab + (size_t)o + d04 + (kb & 1) * 16 + q)
                                                                       : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            };
            gather(buf[0], 0);
#pragma unroll
            for (int kb = 0; kb < dwt::NB; ++kb, ++itb) {
                if (kb + 1 < dwt::NB) gather(buf[(kb + 1) & 1], kb + 1);
                const int bs = itb & 1;
                mbar_wait(bar_bempty + 8 * bs, (((uint32_t)(itb >> 1)) & 1u) ^ 1u, status);
                const uint32_t hi = base + dwt::SMEM_B_OFF + bs * dwt::B_SLOT;
                split_store(hi, hi + dwt::PANEL, buf[kb & 1]);
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_bfull + 8 * bs);
            }
        }
        if (warp < 4 && my_tiles > 0) {
            // =============================== FINAL REDUCTION ===============================
            // thread = row h of dW (TMEM lane); 384 accumulator columns = d; added to the global gradient with 128-bit atomics
            mbar_wait(bar_acc, 0u, status);
            tc_fence_after();
            // Through a padded shared-memory tile (the operand stages are idle by now), so that one instruction adds 4 rows x
            // 128 contiguous bytes instead of 16 bytes of 32 different rows (same reason as the scatter of K3c).
            const float inv = 1.0f / dx_scale;
            const int E = a.Et;
            constexpr int STG_LD = 36;
            float *stg = reinterpret_cast<float *>(smem + dwt::SMEM_A_OFF) + warp * (32 * STG_LD);
            const int wr = lane >> 3, cp = lane & 7;
#pragma unroll 1
            for (int c = 0; c < dwt::D / 32; ++c) {
                float v[32];
                tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(c * 32), v);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4 *>(stg + lane * STG_LD + j) = make_float4(v[j] * inv, v[j + 1] * inv, v[j + 2] * inv, v[j + 3] * inv);
                __syncwarp();
                const int sv = c >> 2, d = db * 128 + (c & 3) * 32 + cp * 4;    // accumulator column sv * 128 + (d - 128 db)
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                    const int h = hb * 128 + warp * 32 + 4 * it + wr;
                    const float4 w = *reinterpret_cast<const float4 *>(stg + (4 * it + wr) * STG_LD + cp * 4);
                    if (h < a.H && d < E) red_add_v4(dW + (size_t)h * (3 * E) + sv * E + d, w);      // dW is [H][3E]
                }
                __syncwarp();
            }
            tc_fence_before();
        }
    } else if (warp == dwt::MMA_WARP) {
        // =============================== MMA ISSUER (converged, one elected lane) ===============================
        int itb = 0;
        for (int tl = 0; tl < my_tiles; ++tl) {
            const int as = tl & 1;
            mbar_wait(bar_afull + 8 * as, ((uint32_t)(tl >> 1)) & 1u, status);
#pragma unroll 1
            for (int kb = 0; kb < dwt::NB; ++kb, ++itb) {
                const int bs = itb & 1;
                mbar_wait(bar_bfull + 8 * bs, ((uint32_t)(itb >> 1)) & 1u, status);
                fence_proxy_async_smem();             // the producers' generic-proxy stores -> async proxy (tensor core)
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t sa = base + dwt::SMEM_A_OFF + as * dwt::A_STAGE;
                    const uint32_t sb = base + dwt::SMEM_B_OFF + bs * dwt::B_SLOT;
                    const uint32_t d_tmem = tmem_base + (uint32_t)(kb * 64);
#pragma unroll
                    for (int k = 0; k < dwt::ROWS / 16; ++k) {
                        const uint64_t a_hi = umma_desc_mn(sa + k * 2048, dwt::PANEL);
                        const uint64_t a_lo = umma_desc_mn(sa + 2 * dwt::PANEL + k * 2048, dwt::PANEL);
                        const uint64_t b_hi = umma_desc_mn(sb + k * 2048, dwt::PANEL);
                        const uint64_t b_lo = umma_desc_mn(sb + dwt::PANEL + k * 2048, dwt::PANEL);
                        const uint32_t acc = (tl | k) != 0 ? 1u : 0u;
                        umma_f16(d_tmem, a_hi, b_hi, dwt::IDESC, acc);
                        umma_f16(d_tmem, a_lo, b_hi, dwt::IDESC, 1u);
                        umma_f16(d_tmem, a_hi, b_lo, dwt::IDESC, 1u);
                    }
                    umma_commit(bar_bempty + 8 * bs);
                    if (kb == dwt::NB - 1) {
                        umma_commit(bar_aempty + 8 * as);
                        if (tl == my_tiles - 1) umma_commit(bar_acc);
                    }
                }
                __syncwarp();
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == dwt::MMA_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

bool backward_dw_tc_ok(const EncodeArgs &a) {
    return a.Et == a.Ep && a.Et <= 2 * dwt::E && a.H <= 2 * dwt::H && (a.Et & 3) == 0 && (a.H & 3) == 0 &&
           (long long)a.T * a.Et * 4 < (1ll << 32) && (long long)a.P * a.Et * 4 < (1ll << 32);
}

int launch_backward_dw_tc(const EncodeArgs &a_in, const float *dx, const unsigned *dx_absmax, float *dW, cudaStream_t st)
{
    EncodeArgs a = a_in;
    a.n_tiles = (int)((a.N + dwt::ROWS - 1) / dwt::ROWS);
    int dev = 0, sms = 0;
    C2V_CUDA_OK(cudaGetDevice(&dev));
    C2V_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    C2V_CUDA_OK(cudaFuncSetAttribute(backward_dw_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dwt::SMEM_BYTES));
    const int n_hb = (a.H + dwt::H - 1) / dwt::H, n_db = (a.Et + dwt::E - 1) / dwt::E;
    int grid = sms / (n_hb * n_db);                        // one CTA per SM over all window pairs
    if (grid > a.n_tiles) grid = a.n_tiles;
    if (grid < 1) grid = 1;
    backward_dw_tc_kernel<<<dim3(grid, n_hb * n_db), dwt::THREADS, dwt::SMEM_BYTES, st>>>(a, dx, dx_absmax, dW, n_db);
    C2V_LAUNCH_OK("backward_dw_tc_kernel");
    return C2V_OK;
}

}  // namespace c2v
