// c2v_backward.cu -- K3: backward of the fused encode path (what loss.backward(), main.py:174,
// runs through model.py:48-69 + 90-96 in the reference), CUDA-core version.
//
// Formulas (SURVEY.md A.1; pinned against the reference's autograd by tests/golden/grad_*.npz).
// Per context j of a bag, with m_j = [starts_j > 0], d_j the dropout multiplier, g_v = dL/dcv:
//   c_j = [E_t[s_j]; E_p[p_j]; E_t[e_j]],  x_j = W c_j,  xh_j = (x_j - mu_j) r_j,
//   t_j = tanh(gamma*xh_j + beta),  h_j = d_j*t_j,  u_j = h_j.a,  alpha = softmax(masked u),
//   v = sum_j alpha_j h_j
//   dalpha_j = g_v.h_j (+ dL/dattention_j);  dz_j = alpha_j (dalpha_j - sum_k alpha_k dalpha_k)
//   du_j = m_j dz_j;  dh_j = alpha_j g_v + du_j a;  da += du_j h_j
//   dy_j = d_j*dh_j*(1 - t_j^2);  dgamma += dy_j*xh_j;  dbeta += dy_j;  dxh_j = dy_j*gamma
//   dx_j = r_j (dxh_j - mean(dxh_j) - xh_j mean(dxh_j*xh_j))
//   dW += dx_j c_j^T ;  dc_j = W^T dx_j scattered into the three embedding-row gradients.
// Nothing but code_vector / attention is stashed by forward: x_j is recomputed per 64-row tile
// (the same tile GEMM as the FFMA forward) and the dropout mask is regenerated from (seed,row,col).
//
// Two kernels:
//   backward_rows_kernel : recompute + dx (kept in smem and written to a [N,H] buffer) +
//                          da/dgamma/dbeta + dC = dX.W scattered with 128-bit vector atomics
//   backward_dw_kernel   : dW = dX^T . C  (split over context rows, gathered C operand)
#include <cstdlib>
#include <cstring>

#include "c2v_ffma_tile.cuh"

namespace c2v {

int launch_transpose_w(const float *W, float *Wt, int H, int D, int Hs, cudaStream_t st);
bool backward_dw_tc_ok(const EncodeArgs &a);
bool backward_dc_tc_ok(const EncodeArgs &a);
size_t backward_dc_tc_workspace_bytes();
int launch_backward_dc_tc(const EncodeArgs &a, const float *W, const float *dx, const unsigned *dx_absmax, void *ws,
                          float *g_emb_t, float *g_emb_p, cudaStream_t st, int sv_mask, bool build_image);
int launch_backward_dw_tc(const EncodeArgs &a, const float *dx, const unsigned *dx_absmax, float *dW, cudaStream_t st);

struct BackwardArgs {
    const float *cv, *att, *d_cv, *d_att, *sb;   // sb[b] = sum_j att[b,j] d_att[b,j] (or null)
    const float *x_stash;                        // [N, H] x = c . W^T kept by the training forward (or null: recompute)
    unsigned *dx_absmax;                         // bits of max |dx| over the batch (atomicMax; for the fp16 split of K3b)
    int skip_dc;                                 // dC = dX . W + scatter is done by K3c (c2v_backward_dc_tc.cu)
    const float *W;                              // [H, D] row-major (B operand of dC = dX . W)
    float *dx;                                   // [N, H]
    float *g_emb_t, *g_emb_p, *g_attn, *g_ln_g, *g_ln_b;
};

constexpr int MAXC = 8;   // columns per lane: encode_size <= 256
// lane owns 4 consecutive columns per 128-column group (k = 0..3, 4..7): one Philox4x32 block gives the dropout masks of
// all four (it is keyed by column / 4), and rows of X are read as one 16-byte piece per lane and group
__device__ __forceinline__ int bk_col(int lane, int k) { return (k >> 2) * 128 + lane * 4 + (k & 3); }

__global__ void bag_dot_kernel(const float *__restrict__ att, const float *__restrict__ d_att, int L,
                               float *__restrict__ sb)
{
    const int b = blockIdx.x, lane = threadIdx.x;
    float s = 0.0f;
    for (int j = lane; j < L; j += 32) s = fmaf(att[(size_t)b * L + j], d_att[(size_t)b * L + j], s);
    s = warp_sum(s);
    if (lane == 0) sb[b] = s;
}

__device__ __forceinline__ void load_wrow_chunk(const float *__restrict__ W, int H, int D, float *Wc, int hc, int cb)
{
    // KC rows (h) x NB columns (d) of W [H][D]
    for (int i = threadIdx.x; i < KC * (NB / 4); i += THREADS) {
        const int kk = i / (NB / 4), cq = i % (NB / 4);
        const int h = hc * KC + kk, col = cb * NB + cq * 4;
        float *dst = Wc + kk * NB + cq * 4;
        // 16-byte copies only when every row of W starts 16-byte aligned (D % 4 == 0: the rows are D floats apart)
        if (h < H && col + 3 < D && (D & 3) == 0) cp_async16(dst, W + (size_t)h * D + col);
        else {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (h < H) {
                if (col < D) v.x = W[(size_t)h * D + col];
                if (col + 1 < D) v.y = W[(size_t)h * D + col + 1];
                if (col + 2 < D) v.z = W[(size_t)h * D + col + 2];
                if (col + 3 < D) v.w = W[(size_t)h * D + col + 3];
            }
            *reinterpret_cast<float4 *>(dst) = v;
        }
    }
}

template <bool VEC>
__global__ void __launch_bounds__(THREADS)
backward_rows_kernel(const EncodeArgs a, const BackwardArgs b, const int Hs)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const FfmaSmem lay = ffma_smem_layout(Hs);
    long long *sidx = reinterpret_cast<long long *>(smem + lay.idx);
    float *Ac = reinterpret_cast<float *>(smem + lay.ac);
    float *Wc = reinterpret_cast<float *>(smem + lay.wc);
    // lite mode (x from the stash, dC done by K3c): no GEMM operand buffers, so X moves up behind the reduction scratch
    // and the CTA needs ~46 KB instead of ~85 KB of shared memory (4 CTAs per SM instead of 2)
    const bool lite = b.x_stash != nullptr && b.skip_dc;
    float *X = reinterpret_cast<float *>(smem + (lite ? lay.ac + 3 * 8 * Hs * 4 : lay.x));
    float *red = reinterpret_cast<float *>(smem + lay.ac);     // reused at the very end (3 x 8 warps x H)

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = tid & 15, ty = tid >> 4;
    const int H = a.H, D = a.D, L = a.L, Et = a.Et, Ep = a.Ep;
    const float invH = 1.0f / (float)H;

    float acc_a[MAXC], acc_g[MAXC], acc_b[MAXC];              // per-lane partial da / dgamma / dbeta
    float dx_max = 0.0f;
#pragma unroll
    for (int k = 0; k < MAXC; ++k) acc_a[k] = acc_g[k] = acc_b[k] = 0.0f;

    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const long long row0 = (long long)tile * TM;
        tile_load_indices(a, row0, sidx);
        __syncthreads();
        if (b.x_stash) {                                       // x kept by the forward: one coalesced tile load
            for (int i = tid; i < TM * H; i += THREADS) {
                const int r = i / H, c = i % H;
                X[r * Hs + c] = row0 + r < a.N ? b.x_stash[(size_t)(row0 + r) * H + c] : 0.0f;
            }
            __syncthreads();
        } else {
            tile_gemm_xw<VEC>(a, sidx, Ac, Wc, X, Hs);         // recompute x = c . W^T
        }

        // ---- per row: forward recompute of LN / tanh / dropout, then dx (one warp per row)
        for (int r = warp; r < TM; r += THREADS / 32) {
            const long long row = row0 + r;
            float *xr = X + r * Hs;
            if (row >= a.N) {
                for (int c = lane; c < Hs; c += 32) xr[c] = 0.0f;
                continue;
            }
            const long long bag = row / L;
            const float *gv = b.d_cv + bag * H, *cvb = b.cv + bag * H;
            const float alpha = b.att[row];
            float s = 0.0f;
            for (int c = lane; c < H; c += 32) s += xr[c];
            const float mean = warp_sum(s) * invH;
            float v = 0.0f;
            for (int c = lane; c < H; c += 32) { const float d = xr[c] - mean; v = fmaf(d, d, v); }
            const float rstd = 1.0f / sqrtf(warp_sum(v) * invH + C2V_LN_EPS);
            float xh[MAXC], tt[MAXC], dm[MAXC];
            float dal = 0.0f, gvv = 0.0f;
            uint4 dbits = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
            for (int k = 0; k < MAXC; ++k) {
                const int c = bk_col(lane, k);
                xh[k] = tt[k] = 0.0f; dm[k] = 1.0f;
                if (c < H) {
                    xh[k] = (xr[c] - mean) * rstd;
                    tt[k] = tanh_accurate(fmaf(xh[k], a.ln_g[c], a.ln_b[c]));
                    if (a.drop_p > 0.0f) {
                        if ((k & 3) == 0) dbits = dropout_bits(a.seed, row, c >> 2);       // columns c .. c+3
                        const unsigned w = (k & 3) == 0 ? dbits.x : (k & 3) == 1 ? dbits.y : (k & 3) == 2 ? dbits.z : dbits.w;
                        dm[k] = dropout_mul(w, a.drop_p, a.drop_scale);
                    }
                    dal = fmaf(gv[c], dm[k] * tt[k], dal);
                    gvv = fmaf(gv[c], cvb[c], gvv);
                }
            }
            dal = warp_sum(dal); gvv = warp_sum(gvv);
            float extra = 0.0f, sbag = 0.0f;
            if (b.d_att) { extra = b.d_att[row]; sbag = b.sb[bag]; }
            const float dz = alpha * (dal + extra - gvv - sbag);
            const float du = sidx[r] > 0 ? dz : 0.0f;            // mask = starts > 0 (model.py:64)
            float dxh[MAXC];
            float m1 = 0.0f, m2 = 0.0f;
#pragma unroll
            for (int k = 0; k < MAXC; ++k) {
                const int c = bk_col(lane, k);
                dxh[k] = 0.0f;
                if (c < H) {
                    const float h = dm[k] * tt[k];
                    const float dh = fmaf(alpha, gv[c], du * a.attn[c]);
                    acc_a[k] = fmaf(du, h, acc_a[k]);
                    const float dy = dm[k] * dh * (1.0f - tt[k] * tt[k]);
                    acc_g[k] = fmaf(dy, xh[k], acc_g[k]);
                    acc_b[k] += dy;
                    dxh[k] = dy * a.ln_g[c];
                    m1 += dxh[k];
                    m2 = fmaf(dxh[k], xh[k], m2);
                }
            }
            m1 = warp_sum(m1) * invH; m2 = warp_sum(m2) * invH;
#pragma unroll
            for (int k = 0; k < MAXC; ++k) {
                const int c = bk_col(lane, k);
                if (c < H) {
                    const float dxv = rstd * (dxh[k] - m1 - xh[k] * m2);
                    xr[c] = dxv;
                    b.dx[row * H + c] = dxv;
                    dx_max = fmaxf(dx_max, fabsf(dxv));
                }
            }
            for (int c = H + lane; c < Hs; c += 32) xr[c] = 0.0f;
        }
        __syncthreads();

        // ---- dC = dX . W  (K = H), 128 columns of D at a time, scattered into the embedding grads
        const int n_cb = b.skip_dc ? 0 : (D + NB - 1) / NB, n_hc = (H + KC - 1) / KC;
        for (int cb = 0; cb < n_cb; ++cb) {
            float acc[4][8];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
            load_wrow_chunk(b.W, H, D, Wc, 0, cb);
            cp_async_commit();
            for (int hc = 0; hc < n_hc; ++hc) {
                const int buf = hc & 1;
                if (hc + 1 < n_hc) {
                    load_wrow_chunk(b.W, H, D, Wc + (buf ^ 1) * KC * NB, hc + 1, cb);
                    cp_async_commit();
                    cp_async_wait<1>();
                } else {
                    cp_async_wait<0>();
                }
                __syncthreads();
                const float *Wb = Wc + buf * KC * NB;
#pragma unroll
                for (int k4 = 0; k4 < KC; k4 += 4) {
                    const int h0 = hc * KC + k4;
                    float4 av[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        av[i] = h0 < Hs ? *reinterpret_cast<const float4 *>(X + (ty * 4 + i) * Hs + h0) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const float4 w0 = *reinterpret_cast<const float4 *>(Wb + (k4 + kk) * NB + tx * 4);
                        const float4 w1 = *reinterpret_cast<const float4 *>(Wb + (k4 + kk) * NB + 64 + tx * 4);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float ai = kk == 0 ? av[i].x : kk == 1 ? av[i].y : kk == 2 ? av[i].z : av[i].w;
                            acc[i][0] = fmaf(ai, w0.x, acc[i][0]); acc[i][1] = fmaf(ai, w0.y, acc[i][1]);
                            acc[i][2] = fmaf(ai, w0.z, acc[i][2]); acc[i][3] = fmaf(ai, w0.w, acc[i][3]);
                            acc[i][4] = fmaf(ai, w1.x, acc[i][4]); acc[i][5] = fmaf(ai, w1.y, acc[i][5]);
                            acc[i][6] = fmaf(ai, w1.z, acc[i][6]); acc[i][7] = fmaf(ai, w1.w, acc[i][7]);
                        }
                    }
                }
                __syncthreads();
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = ty * 4 + i;
                if (row0 + r >= a.N) continue;
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    const int c = cb * NB + g * 64 + tx * 4;
                    if (c >= D) continue;
                    const float v0 = acc[i][g * 4], v1 = acc[i][g * 4 + 1], v2 = acc[i][g * 4 + 2], v3 = acc[i][g * 4 + 3];
                    if (v0 == 0.0f && v1 == 0.0f && v2 == 0.0f && v3 == 0.0f) continue;   // padded contexts
                    if (VEC) {
                        float *dst;
                        if (c < Et) dst = b.g_emb_t + (size_t)sidx[r] * Et + c;
                        else if (c < Et + Ep) dst = b.g_emb_p + (size_t)sidx[TM + r] * Ep + (c - Et);
                        else dst = b.g_emb_t + (size_t)sidx[2 * TM + r] * Et + (c - Et - Ep);
                        red_add_v4(dst, make_float4(v0, v1, v2, v3));
                    } else {
                        const float vv[4] = {v0, v1, v2, v3};
                        for (int q = 0; q < 4; ++q) {
                            const int cc = c + q;
                            if (cc >= D) break;
                            float *dst;
                            if (cc < Et) dst = b.g_emb_t + (size_t)sidx[r] * Et + cc;
                            else if (cc < Et + Ep) dst = b.g_emb_p + (size_t)sidx[TM + r] * Ep + (cc - Et);
                            else dst = b.g_emb_t + (size_t)sidx[2 * TM + r] * Et + (cc - Et - Ep);
                            atomicAdd(dst, vv[q]);
                        }
                    }
                }
            }
        }
        __syncthreads();
    }

    dx_max = warp_max(dx_max);
    if (lane == 0 && dx_max > 0.0f) atomicMax(b.dx_absmax, __float_as_uint(dx_max));   // non-negative floats order as uints
    // ---- da / dgamma / dbeta: 8 warps -> smem -> one atomic per column per CTA
    __syncthreads();
#pragma unroll
    for (int k = 0; k < MAXC; ++k) {
        const int c = bk_col(lane, k);
        if (c < H) {
            red[(0 * 8 + warp) * H + c] = acc_a[k];
            red[(1 * 8 + warp) * H + c] = acc_g[k];
            red[(2 * 8 + warp) * H + c] = acc_b[k];
        }
    }
    __syncthreads();
    for (int i = tid; i < 3 * H; i += THREADS) {
        const int which = i / H, c = i % H;
        float s = 0.0f;
        for (int w = 0; w < 8; ++w) s += red[(which * 8 + w) * H + c];
        float *dst = which == 0 ? b.g_attn : which == 1 ? b.g_ln_g : b.g_ln_b;
        if (s != 0.0f) atomicAdd(dst + c, s);
    }
}

// ------------------------------------------------------------------------------------
// backward_rows_lite_kernel: the same per-row math when x comes from the forward's stash and dC / dW run on the tensor
// cores (K3b, K3c), i.e. no GEMM in this kernel at all.  One warp per context row, rows strided over all warps; lane l
// owns columns 4l..4l+3 of every 128-column group, so x, d_cv, cv and dx move as 16-byte pieces, gamma / beta / attn sit
// in registers for the whole launch, one Philox block serves four columns, and padded contexts (attention weight
// exactly 0) cost one zero store.  encode_size % 4 == 0, <= 256.
// ------------------------------------------------------------------------------------
template <int NG>                                             // 128-column groups: 1 (encode_size <= 128) or 2
__global__ void __launch_bounds__(256, NG == 1 ? 4 : 2)
backward_rows_lite_kernel(const EncodeArgs a, const BackwardArgs b)
{
    constexpr int MAXC = 4 * NG;
    __shared__ float red[3 * 8 * 32 * MAXC];
    // warp index through a lane-0 broadcast, so that the compiler sees the row loop and its branches as warp-uniform
    // (otherwise every shuffle of the six warp sums per row is wrapped in WARPSYNC.COLLECTIVE / ENDCOLLECTIVE)
    const int tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int H = a.H, L = a.L;
    const float invH = 1.0f / (float)H;
    float4 g4[NG], b4[NG], at4[NG];
    bool on[NG];
#pragma unroll
    for (int g = 0; g < NG; ++g) {
        const int c0 = g * 128 + lane * 4;
        on[g] = c0 < H;
        g4[g] = b4[g] = at4[g] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (on[g]) {
            g4[g] = *reinterpret_cast<const float4 *>(a.ln_g + c0);
            b4[g] = *reinterpret_cast<const float4 *>(a.ln_b + c0);
            at4[g] = *reinterpret_cast<const float4 *>(a.attn + c0);
        }
    }
    float acc_a[MAXC], acc_g[MAXC], acc_b[MAXC];
#pragma unroll
    for (int k = 0; k < MAXC; ++k) acc_a[k] = acc_g[k] = acc_b[k] = 0.0f;
    float dx_max = 0.0f;
    const long long n_warps = (long long)gridDim.x * 8;
    // the attention weight of the NEXT row is fetched one iteration ahead: alpha gates the row's other loads (padded rows
    // skip them), so fetched in place it put two dependent memory latencies on every row (ncu: the top stalls were the
    // first uses of these loads)
    const long long row_first = (long long)blockIdx.x * 8 + warp;
    float alpha_next = row_first < a.N ? b.att[row_first] : 0.0f;
    for (long long row = row_first; row < a.N; row += n_warps) {
        const float alpha = alpha_next;
        alpha_next = row + n_warps < a.N ? b.att[row + n_warps] : 0.0f;
        const long long start_idx = a.starts[row];              // (used late: issued here so that it overlaps the row loads)
        float4 *dxr = reinterpret_cast<float4 *>(b.dx + row * H);
        if (__all_sync(0xffffffffu, alpha == 0.0f)) {                                   // padded context of a bag with valid ones: dx == 0
#pragma unroll
            for (int g = 0; g < NG; ++g) if (on[g]) dxr[g * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
            continue;
        }
        const long long bag = row / L;
        const float4 *xr = reinterpret_cast<const float4 *>(b.x_stash + row * H);
        const float4 *gvp = reinterpret_cast<const float4 *>(b.d_cv + bag * H), *cvp = reinterpret_cast<const float4 *>(b.cv + bag * H);
        float x[MAXC], gv[MAXC], cvv[MAXC];
        float s = 0.0f;
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            float4 xv = make_float4(0.f, 0.f, 0.f, 0.f), gg = xv, cc = xv;
            if (on[g]) { xv = xr[g * 32 + lane]; gg = gvp[g * 32 + lane]; cc = cvp[g * 32 + lane]; }
            x[4 * g] = xv.x; x[4 * g + 1] = xv.y; x[4 * g + 2] = xv.z; x[4 * g + 3] = xv.w;
            gv[4 * g] = gg.x; gv[4 * g + 1] = gg.y; gv[4 * g + 2] = gg.z; gv[4 * g + 3] = gg.w;
            cvv[4 * g] = cc.x; cvv[4 * g + 1] = cc.y; cvv[4 * g + 2] = cc.z; cvv[4 * g + 3] = cc.w;
            s += (xv.x + xv.y) + (xv.z + xv.w);
        }
        const float mean = warp_sum(s) * invH;
        float v = 0.0f;
#pragma unroll
        for (int k = 0; k < MAXC; ++k) if (on[k >> 2]) { const float d = x[k] - mean; v = fmaf(d, d, v); }
        const float rstd = 1.0f / sqrtf(warp_sum(v) * invH + C2V_LN_EPS);
        float xh[MAXC], tt[MAXC], dm[MAXC];
        float dal = 0.0f, gvv = 0.0f;
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            uint4 bits = make_uint4(0u, 0u, 0u, 0u);
            if (on[g] && a.drop_p > 0.0f) bits = dropout_bits(a.seed, row, g * 32 + lane);
            const float gam[4] = {g4[g].x, g4[g].y, g4[g].z, g4[g].w}, bet[4] = {b4[g].x, b4[g].y, b4[g].z, b4[g].w};
            const unsigned bw[4] = {bits.x, bits.y, bits.z, bits.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int k = 4 * g + q;
                xh[k] = tt[k] = 0.0f; dm[k] = 1.0f;
                if (on[g]) {
                    xh[k] = (x[k] - mean) * rstd;
                    tt[k] = tanh_accurate(fmaf(xh[k], gam[q], bet[q]));
                    if (a.drop_p > 0.0f) dm[k] = dropout_mul(bw[q], a.drop_p, a.drop_scale);
                    dal = fmaf(gv[k], dm[k] * tt[k], dal);
                    gvv = fmaf(gv[k], cvv[k], gvv);
                }
            }
        }
        dal = warp_sum(dal); gvv = warp_sum(gvv);
        float extra = 0.0f, sbag = 0.0f;
        if (b.d_att) { extra = b.d_att[row]; sbag = b.sb[bag]; }
        const float dz = alpha * (dal + extra - gvv - sbag);
        const float du = start_idx > 0 ? dz : 0.0f;              // mask = starts > 0 (model.py:64)
        float dxh[MAXC];
        float m1 = 0.0f, m2 = 0.0f;
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            const float gam[4] = {g4[g].x, g4[g].y, g4[g].z, g4[g].w}, att[4] = {at4[g].x, at4[g].y, at4[g].z, at4[g].w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int k = 4 * g + q;
                dxh[k] = 0.0f;
                if (on[g]) {
                    const float h = dm[k] * tt[k];
                    const float dh = fmaf(alpha, gv[k], du * att[q]);
                    acc_a[k] = fmaf(du, h, acc_a[k]);
                    const float dy = dm[k] * dh * (1.0f - tt[k] * tt[k]);
                    acc_g[k] = fmaf(dy, xh[k], acc_g[k]);
                    acc_b[k] += dy;
                    dxh[k] = dy * gam[q];
                    m1 += dxh[k];
                    m2 = fmaf(dxh[k], xh[k], m2);
                }
            }
        }
        m1 = warp_sum(m1) * invH; m2 = warp_sum(m2) * invH;
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            if (!on[g]) continue;
            float o[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                o[q] = rstd * (dxh[4 * g + q] - m1 - xh[4 * g + q] * m2);
                dx_max = fmaxf(dx_max, fabsf(o[q]));
            }
            dxr[g * 32 + lane] = make_float4(o[0], o[1], o[2], o[3]);
        }
    }
    dx_max = warp_max(dx_max);
    if (lane == 0 && dx_max > 0.0f) atomicMax(b.dx_absmax, __float_as_uint(dx_max));
    // da / dgamma / dbeta: 8 warps -> smem -> one atomic per column per CTA
#pragma unroll
    for (int k = 0; k < MAXC; ++k) {
        red[((0 * 8 + warp) * MAXC + k) * 32 + lane] = acc_a[k];
        red[((1 * 8 + warp) * MAXC + k) * 32 + lane] = acc_g[k];
        red[((2 * 8 + warp) * MAXC + k) * 32 + lane] = acc_b[k];
    }
    __syncthreads();
    for (int i = tid; i < 3 * MAXC * 32; i += 256) {
        const int which = i / (MAXC * 32), k = (i / 32) % MAXC, l = i % 32;
        const int c = bk_col(l, k);
        if (c >= H) continue;
        float sum = 0.0f;
        for (int w = 0; w < 8; ++w) sum += red[((which * 8 + w) * MAXC + k) * 32 + l];
        float *dst = which == 0 ? b.g_attn : which == 1 ? b.g_ln_g : b.g_ln_b;
        if (sum != 0.0f) atomicAdd(dst + c, sum);
    }
}

// dW[h][d] += sum over this CTA's rows of dx[row][h] * c[row][d]
constexpr int DW_T = 64, DW_R = 16;
__global__ void __launch_bounds__(256)
backward_dw_kernel(const EncodeArgs a, const float *__restrict__ dx, float *__restrict__ dW, const long long rows_per_cta)
{
    __shared__ float As[DW_R][DW_T + 4];
    __shared__ float Bs[DW_R][DW_T + 4];
    __shared__ long long sidx[3][DW_R];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int H = a.H, D = a.D, Et = a.Et, Ep = a.Ep;
    const int d0 = blockIdx.x * DW_T, h0 = blockIdx.y * DW_T;
    const long long r_begin = (long long)blockIdx.z * rows_per_cta;
    long long r_end = r_begin + rows_per_cta; if (r_end > a.N) r_end = a.N;
    float acc[4][4] = {};
    for (long long rc = r_begin; rc < r_end; rc += DW_R) {
        if (tid < 3 * DW_R) {
            const int which = tid / DW_R, r = tid % DW_R;
            const long long row = rc + r;
            long long v = 0;
            if (row < r_end) {
                v = (which == 0 ? a.starts : which == 1 ? a.paths : a.ends)[row];
                const long long lim = which == 1 ? a.P : a.T;
                if (v < 0 || v >= lim) v = 0;
            }
            sidx[which][r] = v;
        }
        __syncthreads();
        for (int i = tid; i < DW_R * DW_T; i += 256) {
            const int r = i / DW_T, q = i % DW_T;
            const long long row = rc + r;
            float av = 0.0f, bv = 0.0f;
            if (row < r_end) {
                const int h = h0 + q, d = d0 + q;
                if (h < H) av = dx[row * H + h];
                if (d < D) {
                    if (d < Et) bv = a.emb_t[(size_t)sidx[0][r] * Et + d];
                    else if (d < Et + Ep) bv = a.emb_p[(size_t)sidx[1][r] * Ep + (d - Et)];
                    else bv = a.emb_t[(size_t)sidx[2][r] * Et + (d - Et - Ep)];
                }
            }
            As[r][q] = av; Bs[r][q] = bv;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < DW_R; ++r) {
            const float4 av = *reinterpret_cast<const float4 *>(&As[r][ty * 4]);
            const float4 bv = *reinterpret_cast<const float4 *>(&Bs[r][tx * 4]);
            const float a4[4] = {av.x, av.y, av.z, av.w}, b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], b4[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int h = h0 + ty * 4 + i;
        if (h >= H) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int d = d0 + tx * 4 + j;
            if (d < D && acc[i][j] != 0.0f) atomicAdd(dW + (size_t)h * D + d, acc[i][j]);
        }
    }
}

size_t encode_backward_workspace_bytes(const c2v_dims *d, int B, int L)
{
    const size_t N = (size_t)B * L, H = d->encode, D = 2 * (size_t)d->terminal_embed + d->path_embed;
    const size_t Hs = (H + 3) / 4 * 4;
    return align_up(N * H * 4, 1024) + align_up((size_t)B * 4, 1024) + align_up(D * Hs * 4, 1024) + 1024 +   // 1 KB: dx absmax word
           align_up(backward_dc_tc_workspace_bytes(), 1024);
}

int launch_encode_backward(const c2v_dims *d, const c2v_params *p, const EncodeArgs &a_in, int B,
                           const float *cv, const float *attention, const float *d_cv, const float *d_att,
                           const c2v_grads *g, void *ws, size_t ws_bytes, cudaStream_t st, const float *x_stash, int phase)
{
    // phase 0: the whole backward.  Phases 1 / 2 split it where the path table's gradient is complete (all state between
    // the two calls lives in the workspace): 1 = per-row work + dC of the path sub-vector + dW, 2 = dC of start / end.
    // dW gathers rows of BOTH embedding tables, so it must run before a caller may start updating path_embedding between
    // the phases; phase 2 reads only dx, the W^T image and the indices.  Only the tensor-core path with a stashed x
    // splits; every other path does everything in phase 1.
    EncodeArgs a = a_in;
    if (a.H > 32 * MAXC) {
        set_error("encode backward supports encode_size <= %d (got %d)", 32 * MAXC, a.H);
        return C2V_EUNSUPPORTED;
    }
    if (ws_bytes < encode_backward_workspace_bytes(d, B, a.L)) {
        set_error("backward workspace too small: %zu < %zu", ws_bytes, encode_backward_workspace_bytes(d, B, a.L));
        return C2V_EWORKSPACE;
    }
    const int Hs = (a.H + 3) / 4 * 4;
    char *base = static_cast<char *>(ws);
    float *dx = reinterpret_cast<float *>(base);
    size_t o = align_up((size_t)a.N * a.H * 4, 1024);
    float *sb = reinterpret_cast<float *>(base + o); o += align_up((size_t)B * 4, 1024);
    float *w_t = reinterpret_cast<float *>(base + o); o += align_up((size_t)a.D * Hs * 4, 1024);
    unsigned *dx_absmax = reinterpret_cast<unsigned *>(base + o); o += 1024;
    void *dc_ws = base + o;
    // dC = dX . W and dW = dX^T . C run on the tensor cores when the shape allows.  C2V_BACKWARD=ffma keeps both on the
    // CUDA cores: the reference the tensor-core tests compare against.
    const char *impl = getenv("C2V_BACKWARD");
    const bool ffma = impl && !strcmp(impl, "ffma");
    const bool dc_tc = !ffma && backward_dc_tc_ok(a), dw_tc = !ffma && backward_dw_tc_ok(a);
    const bool split_ok = x_stash && (a.H & 3) == 0 && dc_tc && dw_tc;
    if (phase == 2) {
        if (!split_ok) return C2V_OK;                           // phase 1 already did everything
        a.n_tiles = (int)((a.N + TM - 1) / TM);
        return launch_backward_dc_tc(a, p->input_linear, dx, dx_absmax, dc_ws, g->terminal_embedding, g->path_embedding, st,
                                     5, false);
    }
    if (phase == 1 && !split_ok) phase = 0;
    C2V_CUDA_OK(cudaMemsetAsync(dx_absmax, 0, 4, st));
    memset(&a.ws, 0, sizeof(a.ws));
    a.ws.w_t = w_t;
    a.ws.status = nullptr;
    a.n_tiles = (int)((a.N + TM - 1) / TM);

    int rc = launch_transpose_w(p->input_linear, w_t, a.H, a.D, Hs, st);
    if (rc != C2V_OK) return rc;
    BackwardArgs b;
    b.cv = cv; b.att = attention; b.d_cv = d_cv; b.d_att = d_att; b.sb = nullptr; b.x_stash = x_stash; b.dx_absmax = dx_absmax;
    b.skip_dc = dc_tc ? 1 : 0;
    b.W = p->input_linear; b.dx = dx;
    b.g_emb_t = g->terminal_embedding; b.g_emb_p = g->path_embedding;
    b.g_attn = g->attention; b.g_ln_g = g->ln_weight; b.g_ln_b = g->ln_bias;
    if (d_att) {
        bag_dot_kernel<<<B, 32, 0, st>>>(attention, d_att, a.L, sb);
        C2V_LAUNCH_OK("bag_dot_kernel");
        b.sb = sb;
    }
    // the three small gradients are overwritten (header contract): zero, then accumulate
    C2V_CUDA_OK(cudaMemsetAsync(g->attention, 0, (size_t)a.H * 4, st));
    C2V_CUDA_OK(cudaMemsetAsync(g->ln_weight, 0, (size_t)a.H * 4, st));
    C2V_CUDA_OK(cudaMemsetAsync(g->ln_bias, 0, (size_t)a.H * 4, st));

    const FfmaSmem lay = ffma_smem_layout(Hs);
    int smem = lay.total;
    const int need_red = lay.ac + 3 * 8 * a.H * 4;
    if (need_red > smem) smem = need_red;
    if (x_stash && dc_tc) smem = lay.ac + 3 * 8 * Hs * 4 + TM * Hs * 4;        // lite layout (see the kernel)
    if (smem > 227 * 1024) { set_error("backward: shared memory %d B too large", smem); return C2V_EUNSUPPORTED; }
    const bool vec = (a.Et % 4 == 0) && (a.Ep % 4 == 0);
    int dev = 0, sms = 0;
    C2V_CUDA_OK(cudaGetDevice(&dev));
    C2V_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    if (x_stash && dc_tc && (a.H & 3) == 0) {                  // no GEMM left in this kernel: one warp per row
        if (a.H <= 128) backward_rows_lite_kernel<1><<<sms * 16, 256, 0, st>>>(a, b);
        else backward_rows_lite_kernel<2><<<sms * 8, 256, 0, st>>>(a, b);
        C2V_LAUNCH_OK("backward_rows_lite_kernel");
        if (phase == 1) {                                       // path sub-vector + dW; start / end follow in phase 2
            rc = launch_backward_dc_tc(a, p->input_linear, dx, dx_absmax, dc_ws, g->terminal_embedding, g->path_embedding, st, 2, true);
            if (rc != C2V_OK) return rc;
            return launch_backward_dw_tc(a, dx, dx_absmax, g->input_linear, st);
        }
        rc = launch_backward_dc_tc(a, p->input_linear, dx, dx_absmax, dc_ws, g->terminal_embedding, g->path_embedding, st, 7, true);
        if (rc != C2V_OK) return rc;
    } else {
        auto kern = vec ? backward_rows_kernel<true> : backward_rows_kernel<false>;
        C2V_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        int occ = 1;
        C2V_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, THREADS, smem));
        if (occ < 1) occ = 1;
        int grid = a.n_tiles < sms * occ ? a.n_tiles : sms * occ;
        kern<<<grid, THREADS, smem, st>>>(a, b, Hs);
        C2V_LAUNCH_OK("backward_rows_kernel");
        if (dc_tc) {
            rc = launch_backward_dc_tc(a, p->input_linear, dx, dx_absmax, dc_ws, g->terminal_embedding, g->path_embedding, st, 7, true);
            if (rc != C2V_OK) return rc;
        }
    }

    // dW = dX^T . C
    if (dw_tc) return launch_backward_dw_tc(a, dx, dx_absmax, g->input_linear, st);
    const int gx = (a.D + DW_T - 1) / DW_T, gy = (a.H + DW_T - 1) / DW_T;
    long long split = (8LL * sms) / (gx * gy);
    if (split < 1) split = 1;
    long long rows_per = (a.N + split - 1) / split;
    rows_per = (rows_per + DW_R - 1) / DW_R * DW_R;
    if (rows_per < DW_R) rows_per = DW_R;
    const long long gz = (a.N + rows_per - 1) / rows_per;
    backward_dw_kernel<<<dim3(gx, gy, (unsigned)gz), 256, 0, st>>>(a, dx, g->input_linear, rows_per);
    C2V_LAUNCH_OK("backward_dw_kernel");
    return C2V_OK;
}

}  // namespace c2v
