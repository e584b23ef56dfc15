// c2v_tc_epilogue.cuh -- the epilogue role of the tcgen05 encode kernel (K1e, c2v_encode_tm.cu; 8 warps):
// TMEM -> registers, LayerNorm (model.py:55-56), tanh (:57), dropout (:60-61), score and NINF
// masking (:64, :92-93), per-warp online-softmax partials of the weighted sum (:68-69, :96).
#pragma once
#include "c2v_tc_ptx.cuh"

namespace c2v {

namespace tce {
constexpr int ROWS = 128;     // context rows per tile (UMMA M)
constexpr int H = 128;        // encode size (UMMA N)
constexpr int VROWS = 32;     // rows per softmax partial = one TMEM lane quarter
constexpr int N_EPI_WARPS = 8;             // default: 2 column slices per TMEM lane quarter
constexpr float TWO_LOG2E = 2.8853900817779268f;
constexpr int VEC_BYTES = 3 * H * 4;               // gamma' | beta' | attn
constexpr int XCH_BYTES = 4 * 4 * 3 * 32 * 4;      // [4 quarters][<=4 slices][3][32] floats
}  // namespace tce

// LayerNorm affine pre-multiplied by 2*log2(e) so tanh needs no extra multiply; columns >= a.H (padding of the
// HP-wide tile when encode_size < HP) get gamma' = beta' = attn = 0.  Layout: gamma'[HP] | beta'[HP] | attn[HP].
template <int HP = tce::H>
__device__ __forceinline__ void tce_fill_vectors(const EncodeArgs &a, float *s_vec, int tid) {
    if (tid < 3 * HP) {
        const int which = tid / HP, c = tid % HP;
        float v = 0.0f;
        if (c < a.H) v = which == 0 ? a.ln_g[c] * tce::TWO_LOG2E : which == 1 ? a.ln_b[c] * tce::TWO_LOG2E : a.attn[c];
        s_vec[tid] = v;
    }
}

// One tile of one epilogue thread: row `row` of the tile, columns [hf * HC, hf * HC + HC) of the accumulator.
// The NS slices of a row are equally wide (HC = 64 at encode_size 128, 52 at 100), so all epilogue warps run the same
// code for the same time; columns >= a.H (only in the last 4-column group of the last slice) are padding: their
// accumulators are exactly 0 (zero rows of the W image), so they add nothing to the LayerNorm sums and are left out
// of the squared deviations, gamma' = beta' = attn = 0 makes their tanh output 0, and they are not written anywhere.
template <bool DROPOUT, int NS, int HC, int HV>
__device__ __forceinline__ void tce_tile_body(const EncodeArgs &a, const float *s_vec, float *my_x, const float *qx,
                                              float (&x)[(HC + 31) / 32 * 32], int q, int hf, int lane, long long vrow0,
                                              long long row, bool in_range, long long st_idx, float inv_scale,
                                              float inv_h, int n_valid)
{
    namespace tc = tce;
    static_assert(HC % 4 == 0 && HC >= 4, "columns per slice");
    constexpr int HCR = (HC + 31) / 32 * 32;                    // rounded up to whole 32-column butterfly groups
    const float4 *sG = reinterpret_cast<const float4 *>(s_vec + hf * HC);
    const float4 *sB = reinterpret_cast<const float4 *>(s_vec + tc::H + hf * HC);
    const float4 *sA = reinterpret_cast<const float4 *>(s_vec + 2 * tc::H + hf * HC);
    auto xsum = [&](int slot) {
        float t = 0.0f;
#pragma unroll
        for (int s = 0; s < NS; ++s) t += qx[(s * 3 + slot) * 32];
        return t;
    };
    // LayerNorm (model.py:55-56) moments, two-pass within the slice: the slice's sum over its n_valid columns, then
    // M2_s = sum (x - m_s)^2 about the slice mean m_s from the same registers.  The slices exchange (sum_s, M2_s) once and
    // combine them with Chan's formula M2 = sum M2_s + sum n_s (m_s - mean)^2.  Unlike E[x^2] - mean^2 this does not
    // cancel when a row's |mean| / std is large (a component shared by all rows of input_linear.weight, which LayerNorm
    // removes and the loss never sees): the variance keeps fp32 relative accuracy there.  Padding columns (zero
    // accumulators) are masked out of M2_s and n_s.
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
    for (int c = 0; c < HC; c += 4) {
        s0 += x[c]; s1 += x[c + 1]; s2 += x[c + 2]; s3 += x[c + 3];
    }
    float part = (s0 + s1) + (s2 + s3);
    const float m_s = part / (float)n_valid;
    s0 = s1 = s2 = s3 = 0.f;
#pragma unroll
    for (int c = 0; c < HC; c += 4) {
        if (c + 4 < HC || c < n_valid) {                          // only the last 4-column group can be padding
            const float d0 = x[c] - m_s, d1 = x[c + 1] - m_s, d2 = x[c + 2] - m_s, d3 = x[c + 3] - m_s;
            s0 = fmaf(d0, d0, s0); s1 = fmaf(d1, d1, s1); s2 = fmaf(d2, d2, s2); s3 = fmaf(d3, d3, s3);
        }
    }
    my_x[0] = part;
    my_x[32] = (s0 + s1) + (s2 + s3);
    named_bar_sync(1 + q, 32 * NS);
    const float mean = xsum(0) * inv_h;
    float m2 = 0.0f;
#pragma unroll
    for (int s = 0; s < NS; ++s) {                               // slice order: the same bits in every slice
        const float n_s = (float)(HV - s * HC < HC ? HV - s * HC : HC);
        const float d = qx[(s * 3) * 32] / n_s - mean;
        m2 += fmaf(n_s * d, d, qx[(s * 3 + 1) * 32]);
    }
    const float var = m2 * inv_h * inv_scale * inv_scale;
    const float nrm = inv_scale / sqrtf(var + C2V_LN_EPS);
    const float shift = -mean * nrm;
    // tanh (model.py:57), dropout (model.py:60-61), score h.a (model.py:92-93)
    float u0 = 0.f, u1 = 0.f;
#pragma unroll
    for (int c4 = 0; c4 < HC / 4; ++c4) {
        const float4 g = sG[c4], b = sB[c4], at = sA[c4];
        float y0 = tanh_from_scaled(fmaf(fmaf(x[4 * c4 + 0], nrm, shift), g.x, b.x));
        float y1 = tanh_from_scaled(fmaf(fmaf(x[4 * c4 + 1], nrm, shift), g.y, b.y));
        float y2 = tanh_from_scaled(fmaf(fmaf(x[4 * c4 + 2], nrm, shift), g.z, b.z));
        float y3 = tanh_from_scaled(fmaf(fmaf(x[4 * c4 + 3], nrm, shift), g.w, b.w));
        if (DROPOUT) {
            const uint4 bits = dropout_bits(a.seed, row, hf * (HC / 4) + c4);
            y0 *= dropout_mul(bits.x, a.drop_p, a.drop_scale);
            y1 *= dropout_mul(bits.y, a.drop_p, a.drop_scale);
            y2 *= dropout_mul(bits.z, a.drop_p, a.drop_scale);
            y3 *= dropout_mul(bits.w, a.drop_p, a.drop_scale);
        }
        x[4 * c4 + 0] = y0; x[4 * c4 + 1] = y1; x[4 * c4 + 2] = y2; x[4 * c4 + 3] = y3;
        u0 = fmaf(y0, at.x, u0); u1 = fmaf(y1, at.y, u1);
        u0 = fmaf(y2, at.z, u0); u1 = fmaf(y3, at.w, u1);
    }
#pragma unroll
    for (int c = HC; c < HCR; ++c) x[c] = 0.0f;                 // fill the last 32-column butterfly group
    part = u0 + u1;
    my_x[64] = part;
    named_bar_sync(1 + q, 32 * NS);
    const float u = xsum(2);                                     // same order => same bits in every slice
    // model.py:93  score*mask + (1-mask)*NINF
    const float z = (in_range && st_idx > 0) ? u : C2V_NINF;
    if (hf == 0 && in_range) a.attention[row] = z;

    // per-(warp, bag) online-softmax partial -> slot (vtile + bag); each slice writes its valid columns
    if (vrow0 < a.N) {
        const long long vt = vrow0 / tc::VROWS;
        long long last = vrow0 + tc::VROWS - 1; if (last > a.N - 1) last = a.N - 1;
        const long long bag_lo = vrow0 / a.L, bag_hi = last / a.L;
        const long long my_bag = row / a.L;
        for (long long bag = bag_lo; bag <= bag_hi; ++bag) {
            const bool in_seg = in_range && my_bag == bag;
            const float m = warp_max(in_seg ? z : -INFINITY);
            const float e = in_seg ? __expf(z - m) : 0.0f;
            const size_t slot = (size_t)(vt + bag);
            float *pv = a.ws.part_v + slot * a.H + hf * HC;
#pragma unroll
            for (int c = 0; c < HCR / 32; ++c) {
                float t[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) t[j] = e * x[c * 32 + j];
                butterfly_reduce32(t, lane);
                if (c * 32 + lane < n_valid) pv[c * 32 + lane] = t[0];
            }
            if (hf == 0) {
                const float ssum = warp_sum(e);
                if (lane == 0) { a.ws.part_m[slot] = m; a.ws.part_s[slot] = ssum; }
            }
        }
    }
}

// Runs on warps 0..7 (warp q and q+4 share TMEM lane quarter q and split the columns).
// tile(tl) = blockIdx.x + tl * gridDim.x; accumulator stage tl & 1 at tmem_base + (tl & 1) * 128.
// DROPOUT is a template parameter so the eval instantiation carries no Philox code: the unrolled epilogue
// shrinks from ~3000 to ~1500 SASS instructions (it was missing the instruction cache, 16 % stall_no_inst).
// NS = column slices per lane quarter (epilogue warps = 4 * NS): warp w handles rows of quarter w & 3 and
// columns [(w >> 2) * HC, ...); LayerNorm moments and the score are summed across the NS warps of a
// quarter through smem + a named barrier, always in slice order so every warp gets the same bits.
// HV = encode_size (multiple of 4); the accumulator tile is always 128 wide, HC = ceil4(HV / NS) columns per slice.
template <bool DROPOUT, int NS = 2, int HV = 128>
__device__ __forceinline__ void tce_epilogue_loop(const EncodeArgs &a, float *s_vec, float *s_xch,
                                                  uint32_t tmem_base, uint32_t bar_tfull, uint32_t bar_tempty,
                                                  int warp, int lane, int my_tiles, long long *status)
{
    namespace tc = tce;
        const int q = warp & 3;                 // TMEM lane quarter: rows 32q .. 32q+31 of the tile
        const int hf = warp >> 2;               // column slice: HC*hf .. HC*hf+HC-1
        constexpr int HC = ((HV + NS - 1) / NS + 3) / 4 * 4;     // columns per thread (64 at 128, 52 at 100)
        constexpr int HCR = (HC + 31) / 32 * 32;
        static_assert(NS * HC <= tc::H && NS * HC - HV <= 4, "padding stays inside the last 4-column group of the last slice");
        static_assert(HC % 32 == 0 || HC % 32 == 16 + 4 || HC % 32 == 16 || HC % 32 == 4, "TMEM load shapes: x32, x16, x4");
        const int n_valid = (HV - hf * HC) < HC ? (HV - hf * HC) : HC;   // valid columns of this slice
        const float inv_scale = a.ws.prep_hdr[0];
        float *my_x = s_xch + ((q * NS + hf) * 3) * 32 + lane;          // [3][32] per (quarter, slice)
        const float *qx = s_xch + (q * NS * 3) * 32 + lane;             // slice s, slot k at qx[(s*3+k)*32]
        for (int tl = 0; tl < my_tiles; ++tl) {
            const int tile = (int)blockIdx.x + tl * (int)gridDim.x;
            const int acc = tl & 1;
            const uint32_t acc_phase = (uint32_t)(tl >> 1) & 1u;
            const long long vrow0 = (long long)tile * tc::ROWS + q * tc::VROWS;
            const long long row = vrow0 + lane;
            const bool in_range = row < a.N;
            const long long st_idx = in_range ? a.starts[row] : 0;       // model.py:64 mask = starts > 0

            mbar_wait(bar_tfull + 8 * acc, acc_phase, status);
            tc_fence_after();
            float x[HCR];
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * tc::H + hf * HC);
#pragma unroll
            for (int c = 0; c < HC / 32; ++c) tmem_ld32(taddr + c * 32, x + c * 32);
            if (HC % 32 >= 16) tmem_ld16(taddr + HC / 32 * 32, x + HC / 32 * 32);
            if (HC % 16 == 4) tmem_ld4(taddr + HC / 16 * 16, x + HC / 16 * 16);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);           // accumulator is free again
            if (a.stash_x && in_range) {       // training forward: keep x = c . W^T for the backward (no recompute)
                float4 *dst = reinterpret_cast<float4 *>(a.stash_x + (size_t)row * a.H + hf * HC);
#pragma unroll
                for (int c = 0; c < HC; c += 4)
                    if (c < n_valid) dst[c / 4] = make_float4(x[c] * inv_scale, x[c + 1] * inv_scale, x[c + 2] * inv_scale, x[c + 3] * inv_scale);
            }

            tce_tile_body<DROPOUT, NS, HC, HV>(a, s_vec, my_x, qx, x, q, hf, lane, vrow0, row, in_range, st_idx,
                                               inv_scale, 1.0f / (float)HV, n_valid);
        }
}

// ------------------------------------------------------------------------------------------------------------------
// encode_size 256 (BASELINE.json configs[3]): the accumulator is [128 rows x 256 columns] and there is only one of it
// (TMEM: 256 accumulator + 256 A-stage columns), so the epilogue cannot keep a row in registers.  Warp (q, hf) owns rows
// 32q.. and columns [128 hf, 128 hf + 128), walks them in 64-column chunks and goes over the accumulator three times:
// LayerNorm moments | LayerNorm + tanh (+ dropout) + score, tanh output written BACK into the accumulator
// (tcgen05.st) | softmax partials of the weighted sum from that output.  The MMAs of the next tile wait
// for the last pass (bar_tempty), the loaders and converters keep running (4 A stages in TMEM).
// ------------------------------------------------------------------------------------------------------------------
template <bool DROPOUT>
__device__ __forceinline__ void tce_epilogue_loop_wide(const EncodeArgs &a, float *s_vec, float *s_xch,
                                                       uint32_t tmem_base, uint32_t bar_tfull, uint32_t bar_tempty,
                                                       int warp, int lane, int my_tiles, long long *status)
{
    namespace tc = tce;
    constexpr int HP = 256, NS = 2, HS = HP / NS, CH = 64, NCH = HS / CH;
    const int q = warp & 3, hf = warp >> 2;
    const float inv_scale = a.ws.prep_hdr[0];
    const float inv_h = 1.0f / (float)HP;
    float *my_x = s_xch + ((q * NS + hf) * 3) * 32 + lane;
    const float *qx = s_xch + (q * NS * 3) * 32 + lane;
    auto xsum = [&](int slot) {
        float t = 0.0f;
#pragma unroll
        for (int s = 0; s < NS; ++s) t += qx[(s * 3 + slot) * 32];
        return t;
    };
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(hf * HS);
    auto load_chunk = [&](int ch, float (&x)[CH]) {
        tmem_ld32(taddr + ch * CH, x);
        tmem_ld32(taddr + ch * CH + 32, x + 32);
        tmem_ld_wait();
    };
    for (int tl = 0; tl < my_tiles; ++tl) {
        const int tile = (int)blockIdx.x + tl * (int)gridDim.x;
        const long long vrow0 = (long long)tile * tc::ROWS + q * tc::VROWS;
        const long long row = vrow0 + lane;
        const bool in_range = row < a.N;
        const long long st_idx = in_range ? a.starts[row] : 0;       // model.py:64 mask = starts > 0
        mbar_wait(bar_tfull, (uint32_t)tl & 1u, status);
        tc_fence_after();
        float x[CH];
        // pass 1: LayerNorm moments (model.py:55-56), two-pass within each 64-column chunk held in registers (sum, then
        // squared deviations about the chunk mean), chunks and then slices combined with Chan's formula as in
        // tce_tile_body: no cancellation at large |mean| / std, and still one walk over the accumulator
        float ssum = 0.f, m2 = 0.f;
#pragma unroll 1
        for (int ch = 0; ch < NCH; ++ch) {
            load_chunk(ch, x);
            if (a.stash_x && in_range) {
                float4 *dst = reinterpret_cast<float4 *>(a.stash_x + (size_t)row * a.H + hf * HS + ch * CH);
#pragma unroll
                for (int c = 0; c < CH; c += 4)
                    dst[c / 4] = make_float4(x[c] * inv_scale, x[c + 1] * inv_scale, x[c + 2] * inv_scale, x[c + 3] * inv_scale);
            }
            float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
            for (int c = 0; c < CH; c += 4) {
                s0 += x[c]; s1 += x[c + 1]; s2 += x[c + 2]; s3 += x[c + 3];
            }
            const float csum = (s0 + s1) + (s2 + s3);
            const float m_c = csum * (1.0f / CH);
            s0 = s1 = s2 = s3 = 0.f;
#pragma unroll
            for (int c = 0; c < CH; c += 4) {
                const float d0 = x[c] - m_c, d1 = x[c + 1] - m_c, d2 = x[c + 2] - m_c, d3 = x[c + 3] - m_c;
                s0 = fmaf(d0, d0, s0); s1 = fmaf(d1, d1, s1); s2 = fmaf(d2, d2, s2); s3 = fmaf(d3, d3, s3);
            }
            m2 += (s0 + s1) + (s2 + s3);
            if (ch > 0) {                       // merge with the chunks before: + n_a n_b / (n_a + n_b) (m_c - m_a)^2
                const float d = m_c - ssum / (float)(ch * CH);
                m2 = fmaf((float)(ch * CH) / (float)(ch + 1) * d, d, m2);
            }
            ssum += csum;
        }
        my_x[0] = ssum;
        my_x[32] = m2;
        named_bar_sync(1 + q, 32 * NS);
        const float mean = xsum(0) * inv_h;
        m2 = 0.0f;
#pragma unroll
        for (int s = 0; s < NS; ++s) {                           // slice order: the same bits in every slice
            const float d = qx[(s * 3) * 32] * (1.0f / HS) - mean;
            m2 += fmaf(HS * d, d, qx[(s * 3 + 1) * 32]);
        }
        const float var = m2 * inv_h * inv_scale * inv_scale;
        const float nrm = inv_scale / sqrtf(var + C2V_LN_EPS);
        const float shift = -mean * nrm;
        // pass 2: tanh (model.py:57), dropout (:60-61), score h.a (:92-93); h goes back into the accumulator
        float u0 = 0.f, u1 = 0.f;
#pragma unroll 1
        for (int ch = 0; ch < NCH; ++ch) {
            load_chunk(ch, x);
            const float4 *sG = reinterpret_cast<const float4 *>(s_vec + hf * HS + ch * CH);
            const float4 *sB = reinterpret_cast<const float4 *>(s_vec + HP + hf * HS + ch * CH);
            const float4 *sA = reinterpret_cast<const float4 *>(s_vec + 2 * HP + hf * HS + ch * CH);
#pragma unroll
            for (int c4 = 0; c4 < CH / 4; ++c4) {
                const float4 g = sG[c4], b = sB[c4], at = sA[c4];
                float y0 = tanh_from_scaled(fmaf(fmaf(x[4 * c4 + 0], nrm, shift), g.x, b.x));
                float y1 = tanh_from_scaled(fmaf(fmaf(x[4 * c4 + 1], nrm, shift), g.y, b.y));
                float y2 = tanh_from_scaled(fmaf(fmaf(x[4 * c4 + 2], nrm, shift), g.z, b.z));
                float y3 = tanh_from_scaled(fmaf(fmaf(x[4 * c4 + 3], nrm, shift), g.w, b.w));
                if (DROPOUT) {
                    const uint4 bits = dropout_bits(a.seed, row, (hf * HS + ch * CH) / 4 + c4);
                    y0 *= dropout_mul(bits.x, a.drop_p, a.drop_scale);
                    y1 *= dropout_mul(bits.y, a.drop_p, a.drop_scale);
                    y2 *= dropout_mul(bits.z, a.drop_p, a.drop_scale);
                    y3 *= dropout_mul(bits.w, a.drop_p, a.drop_scale);
                }
                x[4 * c4 + 0] = y0; x[4 * c4 + 1] = y1; x[4 * c4 + 2] = y2; x[4 * c4 + 3] = y3;
                u0 = fmaf(y0, at.x, u0); u1 = fmaf(y1, at.y, u1);
                u0 = fmaf(y2, at.z, u0); u1 = fmaf(y3, at.w, u1);
            }
            tmem_st32(taddr + ch * CH, x);
            tmem_st32(taddr + ch * CH + 32, x + 32);
        }
        tmem_st_wait_all();
        my_x[64] = u0 + u1;
        named_bar_sync(1 + q, 32 * NS);
        const float u = xsum(2);
        const float z = (in_range && st_idx > 0) ? u : C2V_NINF;     // model.py:93
        if (hf == 0 && in_range) a.attention[row] = z;
        // pass 3: per-(warp, bag) online-softmax partials of the weighted sum
        if (vrow0 < a.N) {
            const long long vt = vrow0 / tc::VROWS;
            long long last = vrow0 + tc::VROWS - 1; if (last > a.N - 1) last = a.N - 1;
            const long long bag_lo = vrow0 / a.L, bag_hi = last / a.L;
            const long long my_bag = row / a.L;
            for (long long bag = bag_lo; bag <= bag_hi; ++bag) {
                const bool in_seg = in_range && my_bag == bag;
                const float m = warp_max(in_seg ? z : -INFINITY);
                const float e = in_seg ? __expf(z - m) : 0.0f;
                const size_t slot = (size_t)(vt + bag);
                float *pv = a.ws.part_v + slot * a.H + hf * HS;
#pragma unroll 1
                for (int ch = 0; ch < NCH; ++ch) {
                    load_chunk(ch, x);
#pragma unroll
                    for (int c = 0; c < CH / 32; ++c) {
                        float t[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) t[j] = e * x[c * 32 + j];
                        butterfly_reduce32(t, lane);
                        pv[ch * CH + c * 32 + lane] = t[0];
                    }
                }
                if (hf == 0) {
                    const float ssum = warp_sum(e);
                    if (lane == 0) { a.ws.part_m[slot] = m; a.ws.part_s[slot] = ssum; }
                }
            }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_tempty);                     // the (only) accumulator is free again
    }
}

}  // namespace c2v
