// c2v_common.cuh -- shared device helpers and internal launch declarations.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/c2v_b200.h"

#define C2V_NINF (-3.4e38f)   // model.py:12 (finite fp32, NOT -inf)
#define C2V_LN_EPS 1e-5f       // nn.LayerNorm default, model.py:24
#define C2V_MIRROR_MAGIC 0x0C2B200C0FFEE5A5LL   // guards the status-mirror pointer stored in the workspace header

namespace c2v {

// ---------------------------------------------------------------------------------
// error plumbing (host)
// ---------------------------------------------------------------------------------
void set_error(const char *fmt, ...);
extern long long g_launches;
#define C2V_COUNT_LAUNCH() (__atomic_add_fetch(&::c2v::g_launches, 1, __ATOMIC_RELAXED))
#define C2V_CUDA_OK(expr)                                                                     \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            ::c2v::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                             __LINE__);                                                       \
            return C2V_ECUDA;                                                                 \
        }                                                                                     \
    } while (0)
#define C2V_LAUNCH_OK(name)                                                                   \
    do {                                                                                      \
        C2V_COUNT_LAUNCH();                                                                   \
        cudaError_t _e = cudaGetLastError();                                                  \
        if (_e != cudaSuccess) {                                                              \
            ::c2v::set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));        \
            return C2V_ECUDA;                                                                 \
        }                                                                                     \
    } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

#ifdef __CUDACC__
// Programmatic dependent launch: the kernel may start (prologue, block scheduling) while the previous kernel of the
// stream is still draining; it must execute griddepcontrol.wait (pdl_wait()) before touching anything the previous
// kernel wrote.  Per-call switch (thread local, set by the extern "C" entry points): the calls that feed autograd -- the
// stashing training forward, or any call with C2V_FLAG_NO_PDL -- use plain stream-ordered launches.
extern thread_local bool g_pdl_this_call;
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = g_pdl_this_call ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#endif

// ---------------------------------------------------------------------------------
// workspace layout of one encode call (all offsets 256-B aligned)
// ---------------------------------------------------------------------------------
struct EncodeWorkspace {
    long long *status;     // [0] out-of-range index count
    float *prep_hdr;       // [0] 1/w_scale (tcgen05 path), [1] w_scale
    float *w_t;            // FFMA: W transposed, [D][Hs] fp32 (Hs = H rounded up to 4)
    uint16_t *w_hi;        // tcgen05: per k-block {hi, lo} fp16 tiles of W*scale, UMMA K-major SW128
    float *part_m;         // [slots] running max of each (tile, bag) segment
    float *part_s;         // [slots] sum of exp(z - m)
    float *part_v;         // [slots][H] sum of exp(z - m) * h
    int tile_rows;         // rows per softmax partial (64: FFMA CTA tile / 32: tcgen05 epilogue warp)
    size_t bytes;
};
// Partial slot of (tile t, bag b): t + b.  Walking the context rows in order, each new
// (tile, bag) pair increments t or b (or both), so t + b is unique; needs n_tiles + B slots.
EncodeWorkspace carve_encode_workspace(const c2v_dims *d, int B, int L, void *base);

struct EncodeArgs {
    const long long *starts, *paths, *ends;
    const float *emb_t, *emb_p, *ln_g, *ln_b, *attn;
    long long T, P;
    int Et, Ep, H, D;
    int L;
    long long N;            // B * L context rows
    int n_tiles;
    float drop_p;           // 0 => no dropout
    float drop_scale;       // 1/(1-p)
    unsigned long long seed;
    float *attention;       // [N] raw masked scores z (finalize turns them into softmax weights)
    float *stash_x;         // optional [N, H]: x = c . W^T (model.py:54) of every row, kept for the backward
    EncodeWorkspace ws;
};

int launch_encode_ffma(const EncodeArgs &a, cudaStream_t st);
int launch_encode_tm(const EncodeArgs &a, cudaStream_t st);
bool tcgen05_shape_ok(const c2v_dims *d);
int launch_encode_finalize(const EncodeArgs &a, int B, float *code_vector, cudaStream_t st);

// Generic fp32 GEMM with bias on CUDA cores: C[m,n] = sum_k A(m,k) * B(k,n) (+ bias[n]),
// element strides given explicitly so every transpose combination is one kernel.
int launch_sgemm(int M, int N, int K, const float *A, long long a_sm, long long a_sk,
                 const float *B, long long b_sk, long long b_sn, const float *bias, float *C,
                 long long c_sm, bool accumulate, cudaStream_t st);
// fused loss / dlogits modes of the label GEMM (c2v_label_tcgen05.cu)
struct LabelLossArgs {
    const long long *label;      // [B]
    float *loss;                 // out: mean NLL (or NULL)
    float *lse_out;              // out: [B] logsumexp of every row (or NULL)
    const float *dlogits_lse;    // in: [B] -> `out` receives d loss / d logits instead of the logits (or NULL)
    float dscale;                // dlogits scale: 1 / B (mean) ...
    const float *dscale_ptr;     // ... times *dscale_ptr when not NULL (the upstream gradient of the scalar loss, on the device)
};
int launch_label_tcgen05_ex(const c2v_dims *d, const float *cv, int B, const float *Wout, const float *bias,
                            float *out, long long *argmax, float *maxval, void *ws, size_t ws_bytes, bool reuse_prep,
                            cudaStream_t st, const LabelLossArgs *la);
int launch_label_tcgen05(const c2v_dims *d, const float *cv, int B, const float *Wout,
                         const float *bias, float *out, long long *argmax, float *maxval, void *ws,
                         size_t ws_bytes, bool reuse_prep, cudaStream_t st);

// ---------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// tanh with <= ~3e-7 absolute error from two MUFU ops: 1 - 2/(e^{2x}+1).
// (tanh.approx.f32 has 2^-11 relative error and would eat the 1e-4 parity budget.)
__device__ __forceinline__ float tanh_accurate(float x) {
    const float e = __expf(2.0f * x);            // inf for large x -> 1, 0 for very negative -> -1
    return 1.0f - __fdividef(2.0f, e + 1.0f);
}

// Philox4x32-10 (Salmon et al. 2011), counter-based: the dropout mask of element
// (row, col) is output [col & 3] of the block with counter (row_lo, row_hi, col >> 2, 0)
// and key (seed_lo, seed_hi); backward regenerates it from the same triple.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const unsigned M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        const unsigned hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0; key.y += W1;
    }
    return ctr;
}
__device__ __forceinline__ uint4 dropout_bits(unsigned long long seed, long long row, int col4) {
    return philox4x32_10(make_uint4((unsigned)row, (unsigned)((unsigned long long)row >> 32),
                                    (unsigned)col4, 0u),
                         make_uint2((unsigned)seed, (unsigned)(seed >> 32)));
}
// keep iff uniform24(bits) >= p ; returns the multiplicative mask (0 or 1/(1-p))
__device__ __forceinline__ float dropout_mul(unsigned bits, float p, float scale) {
    const float u = (float)(bits >> 8) * (1.0f / 16777216.0f);
    return u >= p ? scale : 0.0f;
}
__device__ __forceinline__ float dropout_mask_at(unsigned long long seed, long long row, int col,
                                                 float p, float scale) {
    const uint4 b = dropout_bits(seed, row, col >> 2);
    const unsigned w = (col & 3) == 0 ? b.x : (col & 3) == 1 ? b.y : (col & 3) == 2 ? b.z : b.w;
    return dropout_mul(w, p, scale);
}

// 128-bit reduction without a return value (REDG.E.ADD.F32x4): the scatter-add of gradient rows needs no old value, and
// atomicAdd(float4 *) compiles to ATOMG (the returning form) even when the result is dropped.
__device__ __forceinline__ void red_add_v4(float *addr, float4 v) {
    asm volatile("red.relaxed.gpu.global.add.v4.f32 [%0], {%1, %2, %3, %4};"
                 ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async4(void *smem, const void *gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}
#endif  // __CUDACC__

}  // namespace c2v
