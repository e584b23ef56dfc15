// c2v_encode_tm.cu -- K1e: the fused gather + encode + attention kernel on the 5th-gen tensor cores (sm_100a), with
// its shape check (tcgen05_shape_ok) and its weight preparation (split_w_kernel).
//
// What it replaces: model.py:48-69 + get_attention (model.py:90-96) of the reference.
//
// Numerics.  The reference contraction x = c . W^T is fp32; plain TF32/BF16 miss the 1e-4 parity bar (SURVEY.md 8d).
// Here both operands are split into fp16 hi + fp16 lo (a = a_hi + a_lo exactly to ~2^-22) and three kind::f16 MMAs
// with fp32 accumulation are issued per k-step:  a_hi.w_hi + a_lo.w_hi + a_hi.w_lo  (the dropped a_lo.w_lo term is
// 2^-22 relative).  W is pre-multiplied by a power of two so its lo part stays out of the fp16 subnormals; the
// epilogue (c2v_tc_epilogue.cuh) folds the exact inverse into the LayerNorm scale.
// Measured distance to the reference: ~5e-7 (tests/test_forward_parity_gpu.py).
//
// The gathered-and-split A operand lives in TENSOR MEMORY: the converter warps write the fp16 hi/lo halves straight
// into TMEM with tcgen05.st and the MMAs read A from TMEM (tcgen05.mma [d], [a_tmem], b_desc).
// Why (profiles/README.md): K1d, the earlier variant with A in shared memory, moved 224 KB through shared memory per
// k-block (cp.async 32 + LDS 32 + STS 32 + W copy 32 + MMA operand reads 96) = ~60 us per cfg2 batch at 128 B/clk,
// and its two 32 KB raw stages kept only 64 KB of gathers in flight per SM (loaders alone: 69 us).  Here the STS and
// the MMA's A reads are gone (144 KB per k-block) and the 64 KB of smem they occupied became two more raw stages
// (128 KB in flight).
//
// Warps (24):  0-7 epilogue | 8-15 converters | 16-19 loaders | 20 MMA issuer (+ TMEM alloc) | 21 W producer |
//              22-23 idle register donors.  Registers (pool 768 x 80): 120 | 72 | 56 | 40 | 40 | 24
// smem (201 KB): 4 raw stages [128 rows x 64 fp32], 16-B chunks XOR-swizzled by (row & 7) (128 KB) |
//                2 W stages {W_hi, W_lo} K-major SWIZZLE_128B (64 KB) | gamma'/beta'/attn | LN exchange | mbarriers
// TMEM (512 columns): 2 accumulators [128 lanes x 128 fp32] | 4 A stages {hi: 32 columns, lo: 32 columns},
//                one 32-bit column = two consecutive k of one context row (lane)

#include "c2v_tc_epilogue.cuh"

namespace c2v {

// WIDE = false: terminal_embed = path_embed <= 128, encode_size 100 / 128 (two 128-column accumulators, 4 x 32 KB
// gather stages).  WIDE = true: embed <= 256, encode_size 256 (BASELINE.json configs[3]): one 256-column accumulator
// (UMMA N = 256), 64 KB W k-blocks, 2 gather stages; tensor-bound (393 K FLOP per context x 3 passes).
template <bool WIDE>
struct TmCfg {
    static constexpr int ROWS = tce::ROWS;
    static constexpr int EP = WIDE ? 256 : 128;              // padded sub-vector width (k per start / path / end)
    static constexpr int HP = WIDE ? 256 : 128;              // padded encode size = UMMA N
    static constexpr int KB = 64, NQ = EP / KB, NKB = 3 * NQ; // k-blocks per sub-vector / per tile
    static constexpr int RAW_STAGES = WIDE ? 2 : 4, W_STAGES = 2, A_STAGES = 4, ACC_STAGES = WIDE ? 1 : 2;
    static constexpr int RAW_ROW_BYTES = KB * 4;             // 256 B of an embedding row
    static constexpr int RAW_BYTES = ROWS * RAW_ROW_BYTES;   // 32 KB
    static constexpr int TILE_BYTES = HP * KB * 2;           // one fp16 W tile [HP n x 64 k]: 16 / 32 KB
    static constexpr int W_KB_BYTES = 2 * TILE_BYTES;        // {hi, lo} of one k-block of W
    static constexpr int N_CONV_WARPS = 8;
    static constexpr int CONV_WARP0 = tce::N_EPI_WARPS;      // 8 (multiple of 4: warp & 3 is the TMEM lane quarter)
    static constexpr int N_LOAD_WARPS = 4;
    static constexpr int LOAD_WARP0 = CONV_WARP0 + N_CONV_WARPS; // 16
    static constexpr int MISC_WARP0 = LOAD_WARP0 + N_LOAD_WARPS; // 20
    static constexpr int THREADS = (MISC_WARP0 + 4) * 32;    // 768: warps 22-23 only donate their registers (setmaxnreg pool)
    static constexpr int CPA_PER_ITEM = ROWS / N_LOAD_WARPS / 2; // 16 x LDGSTS.128 (two 256-B row pieces per instruction)
    static constexpr int TMEM_COLS = 512;
    static constexpr int A_COL0 = ACC_STAGES * HP;           // first A-stage column (256)
    static constexpr int A_STAGE_COLS = KB;                  // hi: KB/2 columns, lo: KB/2 columns
    static constexpr int VEC_BYTES = 3 * HP * 4;             // gamma' | beta' | attn
    static constexpr int SMEM_RAW_OFF = 0;
    static constexpr int SMEM_W_OFF = RAW_STAGES * RAW_BYTES;
    static constexpr int SMEM_VEC_OFF = SMEM_W_OFF + W_STAGES * W_KB_BYTES;
    static constexpr int SMEM_XCH_OFF = SMEM_VEC_OFF + VEC_BYTES;
    static constexpr int SMEM_BAR_OFF = SMEM_XCH_OFF + tce::XCH_BYTES;
    static constexpr int SMEM_BYTES = SMEM_BAR_OFF + 256 + 1024;
    static constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(HP >> 3) << 17) | ((uint32_t)(ROWS >> 4) << 24);
    static_assert((RAW_STAGES & (RAW_STAGES - 1)) == 0 && (A_STAGES & (A_STAGES - 1)) == 0 && W_STAGES == 2, "ring index math");
    static_assert(A_COL0 + A_STAGES * A_STAGE_COLS <= TMEM_COLS, "TMEM budget");
    static_assert(SMEM_BYTES <= 232448, "shared memory budget");
};

// K1e pads every sub-vector and the encode size to 128 -- or to 256 in its wide configuration -- so it serves the
// reference's default 100/100/100 (main.py:56-58) and BASELINE.json's 256/256/256 as well:
// terminal_embed == path_embed = E, E % 4 == 0; (E <= 128 and encode_size in {100, 128}) or (E <= 256 and encode_size
// == 256).  Row offsets are 32-bit inside the kernels: tables up to 4 GB.
static bool tm_wide(int E, int H) { return H > TmCfg<false>::HP || E > TmCfg<false>::EP; }
bool tcgen05_shape_ok(const c2v_dims *d)
{
    const int E = d->terminal_embed, H = d->encode;
    if (d->path_embed != E || E < 4 || (E & 3)) return false;
    const bool narrow = E <= 128 && (H == 100 || H == 128), wide = E <= 256 && H == 256;
    if (!narrow && !wide) return false;
    const long long row_bytes = (long long)E * 4;
    return d->terminal_count * row_bytes < (1ll << 32) && d->path_count * row_bytes < (1ll << 32);
}

// ------------------------------------------------------------------------------------
// weight preparation: W [H, 3E] fp32 -> 3*NQ k-block images {hi tile, lo tile} of [HP n x 64 k] fp16 in the exact
// shared-memory layout (K-major SWIZZLE_128B), scaled by 2^k; EP = HP = 128 (NQ = 2) or 256 (NQ = 4).  Sub-vector sv
// (start / path / end) owns k-blocks NQ*sv .. NQ*sv + NQ-1; k >= E and n >= H are zero padding.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
split_w_kernel(const float *__restrict__ W, uint8_t *__restrict__ img, float *__restrict__ hdr, int E, int H, int EP, int HP)
{
    // Several CTAs (the image is rebuilt every training step: one CTA took 22 us at 128/128/128 and 87 us at 256/256/256).
    // Every CTA finds max |W| over the whole matrix itself (<= 768 KB, L2 hits after the first CTA): no second launch, no
    // atomics, no pre-zeroed word.  Then one item = 4 consecutive k of one row n of the PADDED [HP][3 EP] matrix (zeros
    // beyond E / H), i.e. 8 contiguous bytes of the hi tile and of the lo tile: every byte of the image is written once.
    constexpr int KB = TmCfg<false>::KB;
    __shared__ float red[32];
    const int tid = threadIdx.x;
    const int D = 3 * E, NQ = EP / KB;
    const int tile_bytes = HP * KB * 2, kb_bytes = 2 * tile_bytes;
    const bool vec = (reinterpret_cast<uintptr_t>(W) & 15) == 0;       // E % 4 == 0 on this path: rows are 16-B multiples
    float mx = 0.0f;
    if (vec) {
        const float4 *W4 = reinterpret_cast<const float4 *>(W);
        for (int i = tid; i < H * D / 4; i += 1024) {
            const float4 v = W4[i];
            mx = fmaxf(mx, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
        }
    } else {
        for (int i = tid; i < H * D; i += 1024) mx = fmaxf(mx, fabsf(W[i]));
    }
    mx = warp_max(mx);
    if ((tid & 31) == 0) red[tid >> 5] = mx;
    __syncthreads();
    mx = red[0];
    for (int i = 1; i < 32; ++i) mx = fmaxf(mx, red[i]);
    // largest power of two with max|W| * scale < 2^14 (fp16 max is 65504)
    float scale = 1.0f;
    if (mx > 0.0f && mx < 3.0e38f) {
        int e;
        frexpf(mx, &e);                       // mx = f * 2^e, f in [0.5, 1)
        int k = 14 - e;
        k = k > 60 ? 60 : (k < -60 ? -60 : k);
        scale = ldexpf(1.0f, k);
    }
    if (blockIdx.x == 0 && tid == 0) { hdr[0] = 1.0f / scale; hdr[1] = scale; }
    const int per_row = 3 * EP / 4;
    for (int g = blockIdx.x * 1024 + tid; g < HP * per_row; g += gridDim.x * 1024) {
        const int n = g / per_row, kp = (g % per_row) * 4;
        const int sv = kp / EP, e = kp % EP;
        float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
        if (n < H && e < E) {
            const float *src = W + (size_t)n * D + sv * E + e;
            w = vec ? *reinterpret_cast<const float4 *>(src) : make_float4(src[0], src[1], src[2], src[3]);
        }
        w.x *= scale; w.y *= scale; w.z *= scale; w.w *= scale;
        const __half2 h01 = __floats2half2_rn(w.x, w.y), h23 = __floats2half2_rn(w.z, w.w);
        const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
        const __half2 l01 = __floats2half2_rn(w.x - f01.x, w.y - f01.y), l23 = __floats2half2_rn(w.z - f23.x, w.w - f23.y);
        const int kb = NQ * sv + e / KB, kk = e % KB;
        uint8_t *dst = img + (size_t)kb * kb_bytes + sw128_offset(n, kk);
        *reinterpret_cast<uint2 *>(dst) = make_uint2(pack_h2(h01), pack_h2(h23));
        *reinterpret_cast<uint2 *>(dst + tile_bytes) = make_uint2(pack_h2(l01), pack_h2(l23));
    }
}

int launch_split_w_tcgen05(const c2v_dims *d, const float *W, EncodeWorkspace &ws, cudaStream_t st)
{
    const int P = tm_wide(d->terminal_embed, d->encode) ? 256 : 128;
    split_w_kernel<<<P == 256 ? 24 : 12, 1024, 0, st>>>(W, reinterpret_cast<uint8_t *>(ws.w_hi), ws.prep_hdr, d->terminal_embed, d->encode, P, P);
    C2V_LAUNCH_OK("split_w_kernel");
    return C2V_OK;
}

__device__ __forceinline__ void tm_cp_async_cg16(uint32_t dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void tm_cp_async_mbar_arrive_noinc(uint32_t bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ float4 tm_lds_v4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
// D[tmem] (+)= A[tmem] . B[smem]^T : A is [128 lanes x 16 k] fp16, two k per 32-bit column (8 columns)
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// 16 consecutive 32-bit columns of this thread's TMEM lane (lane = 32 * (warp & 3) + laneid)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
                 "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
                   "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// FULL_E: terminal_embed = path_embed = EP (no padding chunks); HV = encode_size (100, 128 or 256).
template <bool DROPOUT, bool FULL_E, int HV>
__global__ void __launch_bounds__(TmCfg<(HV > 128)>::THREADS, 1)
encode_tm_kernel(const EncodeArgs a)
{
    constexpr bool WIDE = HV > 128;
    using tm = TmCfg<WIDE>;
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char *smem = smem_raw + (base - raw);
    float *s_vec = reinterpret_cast<float *>(smem + tm::SMEM_VEC_OFF);
    float *s_xch = reinterpret_cast<float *>(smem + tm::SMEM_XCH_OFF);
    const uint32_t bar_base = base + tm::SMEM_BAR_OFF;
    // 8-byte barriers: raw_full[4] @0, raw_empty[4] @32, a_full[4] @64, a_empty[4] @96, w_full[2] @128,
    //                  w_empty[2] @144, tmem_full[2] @160, tmem_empty[2] @176, tmem ptr @192
    const uint32_t bar_rfull = bar_base, bar_rempty = bar_base + 32, bar_afull = bar_base + 64,
                   bar_aempty = bar_base + 96, bar_wfull = bar_base + 128, bar_wempty = bar_base + 144,
                   bar_tfull = bar_base + 160, bar_tempty = bar_base + 176;
    uint32_t *tmem_ptr_smem = reinterpret_cast<uint32_t *>(smem + tm::SMEM_BAR_OFF + 192);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int my_tiles = (a.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int n_items = my_tiles * tm::NKB;
    long long *status = a.ws.status;

    if (tid == 0) {
        for (int s = 0; s < tm::RAW_STAGES; ++s) {
            mbar_init(bar_rfull + 8 * s, tm::N_LOAD_WARPS * 32);
            mbar_init(bar_rempty + 8 * s, tm::N_CONV_WARPS);
        }
        for (int s = 0; s < tm::A_STAGES; ++s) {
            mbar_init(bar_afull + 8 * s, tm::N_CONV_WARPS);
            mbar_init(bar_aempty + 8 * s, 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(bar_wfull + 8 * s, 1);
            mbar_init(bar_wempty + 8 * s, 1);
            mbar_init(bar_tfull + 8 * s, 1);                  // (WIDE uses stage 0 only)
            mbar_init(bar_tempty + 8 * s, tce::N_EPI_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == tm::MISC_WARP0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(tmem_ptr_smem)), "r"((uint32_t)tm::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    pdl_wait();              // barrier init and the TMEM allocation above overlap the previous kernel's tail
    tce_fill_vectors<tm::HP>(a, s_vec, tid);
    if (!FULL_E) {      // padding chunks of the raw stages (k >= embed size) are read by the converters but never written
        uint4 *z = reinterpret_cast<uint4 *>(smem + tm::SMEM_RAW_OFF);
        for (int i = tid; i < tm::RAW_STAGES * tm::RAW_BYTES / 16; i += tm::THREADS) z[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    // item it = tl * NKB + kb.  Raw ring / A ring: stage it & 3, use count it >> 2; W ring: stage it & 1, use it >> 1.
    if (warp < tce::N_EPI_WARPS) {
        // =============================== EPILOGUE ===============================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 120;");
        if constexpr (WIDE)
            tce_epilogue_loop_wide<DROPOUT>(a, s_vec, s_xch, tmem_base, bar_tfull, bar_tempty, warp, lane, my_tiles, status);
        else
            tce_epilogue_loop<DROPOUT, 2, HV>(a, s_vec, s_xch, tmem_base, bar_tfull, bar_tempty, warp, lane, my_tiles, status);
    } else if (warp < tm::LOAD_WARP0) {
        // =============================== CONVERTERS ===============================
        // thread = one context row (TMEM lane) x 32 consecutive k of the k-block (8 x LDS.128, conflict-free
        // through the chunk swizzle) -> 16 hi + 16 lo packed columns -> 2 x tcgen05.st.32x32b.x16
        asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
        const int qd = warp & 3, hf = (warp - tm::CONV_WARP0) >> 2;
        const int r = qd * 32 + lane;
        uint32_t ld_off[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) ld_off[c] = (uint32_t)(r * tm::RAW_ROW_BYTES + ((8 * hf + (c ^ (r & 7))) << 4));
        const uint32_t t_lane = tmem_base + ((uint32_t)(qd * 32) << 16) + (uint32_t)(tm::A_COL0 + hf * (tm::KB / 4));
        for (int it = 0; it < n_items; ++it) {
            const int st = it & (tm::RAW_STAGES - 1);
            const uint32_t phase = (uint32_t)(it / tm::RAW_STAGES) & 1u;
            const uint32_t rawb = base + tm::SMEM_RAW_OFF + st * tm::RAW_BYTES;
            mbar_wait(bar_rfull + 8 * st, phase, status);          // gathered fp32 rows have landed
            float4 v[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) v[c] = tm_lds_v4(rawb + ld_off[c]);
            // the asm volatile loads above complete in order before this arrive: the raw stage can be
            // refilled by the next gather while this warp converts out of registers
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_rempty + 8 * st);
            const int as = it & (tm::A_STAGES - 1);
            const uint32_t aphase = (uint32_t)(it / tm::A_STAGES) & 1u;
            const uint32_t t_st = t_lane + as * tm::A_STAGE_COLS;
            // two halves of 4 chunks (16 k) each, so that 72 registers are enough
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                uint32_t hi[8], lo[8];
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    const float4 x = v[4 * g + cc];
                    const __half2 h01 = __floats2half2_rn(x.x, x.y), h23 = __floats2half2_rn(x.z, x.w);
                    const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
                    hi[2 * cc] = pack_h2(h01);
                    hi[2 * cc + 1] = pack_h2(h23);
                    lo[2 * cc] = pack_h2(__floats2half2_rn(x.x - f01.x, x.y - f01.y));
                    lo[2 * cc + 1] = pack_h2(__floats2half2_rn(x.z - f23.x, x.w - f23.y));
                }
                if (g == 0) {
                    mbar_wait(bar_aempty + 8 * as, aphase ^ 1u, status);   // MMAs of the previous use retired
                    tc_fence_after();
                }
                tmem_st8(t_st + g * 8, hi);
                tmem_st8(t_st + tm::KB / 2 + g * 8, lo);
            }
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_afull + 8 * as);
        }
    } else if (warp < tm::MISC_WARP0) {
        // =============================== LOADERS (cp.async) ===============================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
        const int lw = warp - tm::LOAD_WARP0;        // rows 32*lw .. 32*lw+31 of every tile; lane l owns row 32*lw+l's indices
        // Instruction j copies rows 32*lw + 2j (lanes 0-15) and 2j+1 (lanes 16-31): 512 contiguous bytes of the raw
        // stage in lane order (a permuted smem destination falls off the LDGSTS fast path: 177 us instead of 69).
        // The chunk swizzle is applied on the GLOBAL side instead: the lane that writes chunk position q of row r
        // fetches chunk q ^ (r & 7) of the embedding row; r & 7 = (2j & 7) | sub, so q ^ (r & 7) = (q ^ sub) ^ (2j & 7).
        const int sub = lane >> 4, q = lane & 15;
        const char *tab_t = reinterpret_cast<const char *>(a.emb_t);
        const char *tab_p = reinterpret_cast<const char *>(a.emb_p);
        uint32_t qoff[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) qoff[c] = (uint32_t)(((q ^ sub) ^ (2 * c)) << 4);
        const uint32_t dst_lane = (uint32_t)((lw * 32 + sub) * tm::RAW_ROW_BYTES + q * 16);
        const uint32_t row_bytes = FULL_E ? (uint32_t)(tm::EP * 4) : (uint32_t)(a.Et * 4);    // Et == Ep
        long long rs = 0, rp = 0, re = 0;            // raw indices of the NEXT tile (prefetched)
        uint32_t off_s = 0, off_p = 0, off_e = 0;    // byte offsets of this lane's row in the tables
        auto fetch_idx = [&](int tl) {
            rs = rp = re = 0;
            if (tl < my_tiles) {
                const long long row = ((long long)blockIdx.x + (long long)tl * gridDim.x) * tm::ROWS + lw * 32 + lane;
                if (row < a.N) { rs = a.starts[row]; rp = a.paths[row]; re = a.ends[row]; }
            }
        };
        auto adopt_idx = [&]() {
            int bad = 0;
            if (rs < 0 || rs >= a.T) { rs = 0; ++bad; }
            if (rp < 0 || rp >= a.P) { rp = 0; ++bad; }
            if (re < 0 || re >= a.T) { re = 0; ++bad; }
            if (bad) atomicAdd((unsigned long long *)status, (unsigned long long)bad);
            off_s = (uint32_t)rs * row_bytes; off_p = (uint32_t)rp * row_bytes; off_e = (uint32_t)re * row_bytes;
        };
        fetch_idx(0);
        int it = 0;
        for (int tl = 0; tl < my_tiles; ++tl) {
            adopt_idx();
            fetch_idx(tl + 1);
            // One sub-vector (start / path / end embedding) = two k-blocks.  The 16 row offsets a lane needs are
            // fetched with 16 back-to-back shuffles per sub-vector (with 40 registers ptxas chained SHFL -> IADD ->
            // LDGSTS one at a time and the loaders, ~115 cycles per LDGSTS, paced the whole pipeline).
#pragma unroll
            for (int sv = 0; sv < 3; ++sv) {
                const uint32_t off = sv == 0 ? off_s : (sv == 1 ? off_p : off_e);
                const char *tab = sv == 1 ? tab_p : tab_t;
                uint32_t o[tm::CPA_PER_ITEM];
#pragma unroll
                for (int j = 0; j < tm::CPA_PER_ITEM; ++j) o[j] = __shfl_sync(0xffffffffu, off, 2 * j + sub);
#pragma unroll
                for (int h = 0; h < tm::NQ; ++h, ++it) {
                    const int st = it & (tm::RAW_STAGES - 1);
                    const uint32_t phase = (uint32_t)(it / tm::RAW_STAGES) & 1u;
                    const uint32_t dst = base + tm::SMEM_RAW_OFF + st * tm::RAW_BYTES + dst_lane;
                    mbar_wait(bar_rempty + 8 * st, phase ^ 1u, status);
#pragma unroll
                    for (int j = 0; j < tm::CPA_PER_ITEM; ++j) {
                        const uint32_t chunk = (uint32_t)(h * tm::RAW_ROW_BYTES) + qoff[j & 3];   // byte offset in the row
                        if (FULL_E || chunk < row_bytes)    // chunk positions at or beyond the embedding size are never
                            tm_cp_async_cg16(dst + j * 2 * tm::RAW_ROW_BYTES, tab + (o[j] + chunk));   // written: zero since start
                    }
                    tm_cp_async_mbar_arrive_noinc(bar_rfull + 8 * st);
                }
            }
        }
    } else if (warp >= tm::MISC_WARP0 + 2) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
    } else {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        if (warp == tm::MISC_WARP0) {
            // =============================== MMA ISSUER ===============================
            // The whole warp runs the loop converged and one elected lane issues: inside an `if (lane == 0)` region
            // ptxas wraps every UTCHMMA in an ELECT / BRA.U.ANY loop and rebuilds the descriptors through R2UR
            // (~25 instructions per MMA); the issuer thread was then the slowest stage of the pipeline
            // (cycle counters around the barrier waits: it waited only 15 % of the time while converters and loaders
            // waited ~50 %).
            const uint64_t wdesc0 = umma_desc(base + tm::SMEM_W_OFF);       // stage 0, W_hi, k-step 0
            const uint32_t ta0 = tmem_base + (uint32_t)tm::A_COL0;
            int it = 0;
            for (int tl = 0; tl < my_tiles; ++tl) {
                const int acc = WIDE ? 0 : (tl & 1);
                const uint32_t acc_phase = (uint32_t)(tl / tm::ACC_STAGES) & 1u;
                mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1u, status);
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * tm::HP);
#pragma unroll 1
                for (int kb = 0; kb < tm::NKB; ++kb, ++it) {
                    const int as = it & (tm::A_STAGES - 1), ws = it & 1;
                    mbar_wait(bar_afull + 8 * as, (uint32_t)(it / tm::A_STAGES) & 1u, status);
                    mbar_wait(bar_wfull + 8 * ws, (uint32_t)(it >> 1) & 1u, status);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint64_t w_hi0 = wdesc0 + (uint64_t)(ws * (tm::W_KB_BYTES >> 4));
                        const uint32_t ta = ta0 + (uint32_t)(as * tm::A_STAGE_COLS);
#pragma unroll
                        for (int k = 0; k < tm::KB / 16; ++k) {
                            if (!FULL_E && (kb % tm::NQ) * tm::KB + k * 16 >= a.Et) break;  // k-steps of pure padding
                            const uint32_t a_hi = ta + k * 8, a_lo = ta + tm::KB / 2 + k * 8;
                            const uint64_t w_hi = w_hi0 + (uint64_t)(k * 2);                  // + 32 B
                            const uint64_t w_lo = w_hi + (uint64_t)(tm::TILE_BYTES >> 4);
                            umma_f16_ts(d_tmem, a_hi, w_hi, tm::IDESC, (kb | k) != 0 ? 1u : 0u);
                            umma_f16_ts(d_tmem, a_lo, w_hi, tm::IDESC, 1u);
                            umma_f16_ts(d_tmem, a_hi, w_lo, tm::IDESC, 1u);
                        }
                        umma_commit(bar_aempty + 8 * as);
                        umma_commit(bar_wempty + 8 * ws);
                        if (kb == tm::NKB - 1) umma_commit(bar_tfull + 8 * acc);
                    }
                    __syncwarp();
                }
            }
        } else if (warp == tm::MISC_WARP0 + 1) {
            // =============================== W PRODUCER ===============================
            if (lane == 0) {
                const uint8_t *img = reinterpret_cast<const uint8_t *>(a.ws.w_hi);
                int kb = 0;
                for (int it = 0; it < n_items; ++it) {
                    const int ws = it & 1;
                    mbar_wait(bar_wempty + 8 * ws, ((uint32_t)(it >> 1) & 1u) ^ 1u, status);
                    mbar_arrive_expect_tx(bar_wfull + 8 * ws, tm::W_KB_BYTES);
                    bulk_copy_g2s(base + tm::SMEM_W_OFF + ws * tm::W_KB_BYTES, img + (size_t)kb * tm::W_KB_BYTES,
                                  tm::W_KB_BYTES, bar_wfull + 8 * ws);
                    if (++kb == tm::NKB) kb = 0;
                }
            }
            __syncwarp();
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == tm::MISC_WARP0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)tm::TMEM_COLS) : "memory");
    }
}

template <bool WIDE>
static int launch_tm(void (*kern)(const EncodeArgs), const EncodeArgs &a, cudaStream_t st)
{
    using C = TmCfg<WIDE>;
    int dev = 0, sms = 0;
    C2V_CUDA_OK(cudaGetDevice(&dev));
    C2V_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    C2V_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    int grid = a.n_tiles < sms ? a.n_tiles : sms;
    if (grid < 1) grid = 1;
    C2V_CUDA_OK(launch_pdl(kern, dim3((unsigned)grid), dim3(C::THREADS), (size_t)C::SMEM_BYTES, st, a));
    C2V_COUNT_LAUNCH();
    return C2V_OK;
}

int launch_encode_tm(const EncodeArgs &a, cudaStream_t st)
{
    const bool drop = a.drop_p > 0.0f;
    if (a.H == 256) {
        const bool full = a.Et == 256;
        return launch_tm<true>(full ? (drop ? encode_tm_kernel<true, true, 256> : encode_tm_kernel<false, true, 256>)
                                    : (drop ? encode_tm_kernel<true, false, 256> : encode_tm_kernel<false, false, 256>), a, st);
    }
    const bool full = a.Et == 128;
    if (a.H == 128)
        return launch_tm<false>(full ? (drop ? encode_tm_kernel<true, true, 128> : encode_tm_kernel<false, true, 128>)
                                     : (drop ? encode_tm_kernel<true, false, 128> : encode_tm_kernel<false, false, 128>), a, st);
    if (a.H == 100)
        return launch_tm<false>(full ? (drop ? encode_tm_kernel<true, true, 100> : encode_tm_kernel<false, true, 100>)
                                     : (drop ? encode_tm_kernel<true, false, 100> : encode_tm_kernel<false, false, 100>), a, st);
    set_error("encode_tm_kernel: encode_size %d not supported (100, 128 or 256)", a.H);
    return C2V_EUNSUPPORTED;
}

}  // namespace c2v
