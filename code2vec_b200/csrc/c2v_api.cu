// c2v_api.cu -- the extern "C" surface declared in include/c2v_b200.h.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>

#include "c2v_common.cuh"

namespace c2v {

long long g_launches = 0;
static thread_local char g_err[512] = "";
thread_local bool g_pdl_this_call = true;

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int launch_transpose_w(const float *W, float *Wt, int H, int D, int Hs, cudaStream_t st);
int launch_split_w_tcgen05(const c2v_dims *d, const float *W, EncodeWorkspace &ws, cudaStream_t st);
int launch_angular(const c2v_dims *d, const c2v_params *p, const float *cv, const long long *label,
                   int B, float margin, float inverse_temp, float *out, float *scratch,
                   cudaStream_t st, float *cos_out);
int launch_angular_backward(const c2v_dims *d, const c2v_params *p, const float *cv, const long long *label, int B,
                            float margin, float inverse_temp, const float *cosine, const float *inv_cv, const float *inv_w,
                            float *d_out_inplace, float *d_cv, float *d_w, float *sums, cudaStream_t st);
int launch_loss_argmax(const float *out, const long long *label, int B, long long C, float *loss,
                       long long *argmax, float *maxval, float *d_out, cudaStream_t st);
int launch_colsum(const float *X, int B, long long C, float *out, cudaStream_t st);
int launch_encode_backward(const c2v_dims *d, const c2v_params *p, const EncodeArgs &a, int B,
                           const float *cv, const float *attention, const float *d_cv,
                           const float *d_att, const c2v_grads *g, void *ws, size_t ws_bytes,
                           cudaStream_t st, const float *x_stash, int phase);
size_t encode_backward_workspace_bytes(const c2v_dims *d, int B, int L);
bool label_tcgen05_shape_ok(const c2v_dims *d);
bool label_backward_tc_ok(const c2v_dims *d);
int label_w_image(const c2v_dims *d, const float *Wout, int B, void *ws, size_t ws_bytes, bool reuse_prep, cudaStream_t st,
                  const uint8_t **img, const float **hdr, unsigned **scratch, const uint8_t **cv_img);
int launch_label_backward_tc(const c2v_dims *d, const float *cv, const float *G, int B, const uint8_t *w_img,
                             const float *w_hdr, float *d_cv, float *d_w, float *d_b, unsigned *scratch, cudaStream_t st,
                             bool absmax_ready, const uint8_t *cv_img);
size_t label_tcgen05_workspace_bytes(const c2v_dims *d, int B);
bool label_ws_holds_dlogits_of(const void *ws, const float *cv, int B);

// ---- profiling hook (c2v_profile_enable / c2v_profile_read) ----------------------------
static const int kProfRing = 4096;
static bool g_prof_on = false;
static int g_prof_stride = 1;          // time every n-th encode launch (events between launches defeat
static long long g_prof_calls = 0;     // programmatic dependent launch, so a bench samples instead)
static cudaEvent_t g_prof_ev[kProfRing][2];
static bool g_prof_made = false;
static int g_prof_pending = 0;
static double g_prof_ms = 0.0;
static long long g_prof_count = 0;

static int prof_drain()
{
    for (int i = 0; i < g_prof_pending; ++i) {
        float ms = 0.0f;
        C2V_CUDA_OK(cudaEventSynchronize(g_prof_ev[i][1]));
        C2V_CUDA_OK(cudaEventElapsedTime(&ms, g_prof_ev[i][0], g_prof_ev[i][1]));
        g_prof_ms += ms;
        g_prof_count += 1;
    }
    g_prof_pending = 0;
    return C2V_OK;
}

static bool dims_ok(const c2v_dims *d)
{
    if (!d) { set_error("dims is NULL"); return false; }
    if (d->terminal_count < 1 || d->path_count < 1 || d->terminal_embed < 1 || d->path_embed < 1 ||
        d->encode < 1) {
        set_error("bad dims: T=%lld P=%lld Et=%d Ep=%d H=%d", (long long)d->terminal_count,
                  (long long)d->path_count, d->terminal_embed, d->path_embed, d->encode);
        return false;
    }
    return true;
}

// tile rows used for sizing: the smallest tile any algorithm uses (64) gives the most slots
static const int kMinTileRows = 32;   // tcgen05 path: one partial per 32-row epilogue warp

EncodeWorkspace carve_encode_workspace(const c2v_dims *d, int B, int L, void *base)
{
    EncodeWorkspace w;
    memset(&w, 0, sizeof(w));
    const int H = d->encode, D = 2 * d->terminal_embed + d->path_embed;
    const int Hs = (H + 3) / 4 * 4;
    const long long N = (long long)B * L;
    const size_t n_tiles = (size_t)((N + kMinTileRows - 1) / kMinTileRows);
    const size_t slots = n_tiles + (size_t)B + 1;
    // tcgen05 split weights: K padded to 64-element blocks, N padded to 128 rows... sized generously
    size_t kblocks = (size_t)(D + 63) / 64 + 3;                // +3: per-sub-vector padding
    const size_t padded = (H > 128 || d->terminal_embed > 128) ? 12 : 6;   // K1e pads each sub-vector to 128 / 256 k
    if (kblocks < padded) kblocks = padded;
    const size_t hp = (size_t)(H + 127) / 128 * 128;
    char *p = static_cast<char *>(base);
    size_t o = 0;
    auto take = [&](size_t bytes) { char *r = p ? p + o : nullptr; o += align_up(bytes, 1024); return r; };
    w.status = reinterpret_cast<long long *>(take(256));
    w.prep_hdr = reinterpret_cast<float *>(take(256));
    w.w_t = reinterpret_cast<float *>(take((size_t)D * Hs * sizeof(float)));
    // per k-block: {hi tile, lo tile}, each [hp x 64] fp16 in the UMMA shared-memory layout
    w.w_hi = reinterpret_cast<uint16_t *>(take(2 * kblocks * hp * 64 * sizeof(uint16_t)));
    w.part_m = reinterpret_cast<float *>(take(slots * sizeof(float)));
    w.part_s = reinterpret_cast<float *>(take(slots * sizeof(float)));
    w.part_v = reinterpret_cast<float *>(take(slots * (size_t)H * sizeof(float)));
    w.bytes = o;
    return w;
}

}  // namespace c2v

using namespace c2v;

extern "C" {

int c2v_abi_version(void) { return C2V_ABI_VERSION; }
const char *c2v_last_error(void) { return g_err; }
int64_t c2v_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }

int c2v_get_device_info(int device, c2v_device_info *out)
{
    if (!out) { set_error("out is NULL"); return C2V_EINVAL; }
    cudaDeviceProp pr;
    C2V_CUDA_OK(cudaGetDeviceProperties(&pr, device));
    out->cc_major = pr.major; out->cc_minor = pr.minor; out->sm_count = pr.multiProcessorCount;
    out->reserved = 0;
    out->global_mem_bytes = (int64_t)pr.totalGlobalMem;
    out->smem_per_block_optin = (int64_t)pr.sharedMemPerBlockOptin;
    return C2V_OK;
}

int c2v_encode_supports_tcgen05(const c2v_dims *d)
{
    if (!dims_ok(d)) return 0;
    return tcgen05_shape_ok(d) ? 1 : 0;
}

size_t c2v_encode_workspace_bytes(const c2v_dims *d, int32_t B, int32_t L)
{
    if (!dims_ok(d) || B < 1 || L < 1) return 0;
    return carve_encode_workspace(d, B, L, nullptr).bytes;
}

int c2v_encode_forward(const c2v_dims *d, const c2v_params *p, const int64_t *starts,
                       const int64_t *paths, const int64_t *ends, int32_t B, int32_t L,
                       const c2v_dropout *drop, float *code_vector, float *attention,
                       void *workspace, size_t workspace_bytes, int32_t algo, void *stream)
{
    return c2v_encode_forward_stash(d, p, starts, paths, ends, B, L, drop, code_vector, attention, nullptr, workspace,
                                    workspace_bytes, algo, stream);
}

int c2v_encode_forward_stash(const c2v_dims *d, const c2v_params *p, const int64_t *starts,
                             const int64_t *paths, const int64_t *ends, int32_t B, int32_t L,
                             const c2v_dropout *drop, float *code_vector, float *attention, float *x_stash,
                             void *workspace, size_t workspace_bytes, int32_t algo, void *stream)
{
    if (!dims_ok(d)) return C2V_EINVAL;
    if (!p || !starts || !paths || !ends || !code_vector || !attention || !workspace) {
        set_error("c2v_encode_forward: NULL pointer argument");
        return C2V_EINVAL;
    }
    if (!p->terminal_embedding || !p->path_embedding || !p->input_linear || !p->ln_weight ||
        !p->ln_bias || !p->attention) {
        set_error("c2v_encode_forward: NULL parameter pointer");
        return C2V_EINVAL;
    }
    if (B < 1 || L < 1) { set_error("c2v_encode_forward: B=%d L=%d", B, L); return C2V_EINVAL; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    EncodeWorkspace ws = carve_encode_workspace(d, B, L, workspace);
    if (ws.bytes > workspace_bytes) {
        set_error("workspace too small: %zu < %zu", workspace_bytes, ws.bytes);
        return C2V_EWORKSPACE;
    }
    const bool reuse_prep = (algo & C2V_FLAG_REUSE_PREP) != 0;
    g_pdl_this_call = (algo & C2V_FLAG_NO_PDL) == 0 && x_stash == nullptr;
    algo &= 0xff;
    bool use_tc;
    if (algo == C2V_ALGO_TCGEN05) {
        if (!tcgen05_shape_ok(d)) {
            set_error("tcgen05 encode does not support Et=%d Ep=%d H=%d", d->terminal_embed,
                      d->path_embed, d->encode);
            return C2V_EUNSUPPORTED;
        }
        use_tc = true;
    } else if (algo == C2V_ALGO_FFMA) {
        use_tc = false;
    } else if (algo == C2V_ALGO_AUTO) {
        use_tc = tcgen05_shape_ok(d);
    } else {
        set_error("unknown algo %d", algo);
        return C2V_EINVAL;
    }

    EncodeArgs a;
    memset(&a, 0, sizeof(a));
    a.starts = reinterpret_cast<const long long *>(starts);
    a.paths = reinterpret_cast<const long long *>(paths);
    a.ends = reinterpret_cast<const long long *>(ends);
    a.emb_t = p->terminal_embedding; a.emb_p = p->path_embedding;
    a.ln_g = p->ln_weight; a.ln_b = p->ln_bias; a.attn = p->attention;
    a.T = d->terminal_count; a.P = d->path_count;
    a.Et = d->terminal_embed; a.Ep = d->path_embed; a.H = d->encode;
    a.D = 2 * a.Et + a.Ep;
    a.L = L; a.N = (long long)B * L;
    a.drop_p = 0.0f; a.drop_scale = 1.0f; a.seed = 0;
    if (drop && drop->training && drop->p > 0.0f && drop->p < 1.0f) {   // model.py:26-29
        a.drop_p = drop->p; a.drop_scale = 1.0f / (1.0f - drop->p); a.seed = drop->seed;
    }
    a.attention = attention;
    a.stash_x = x_stash;
    // rows per softmax partial: 64-row CTA tiles (FFMA) or 32-row epilogue warps (tcgen05)
    ws.tile_rows = use_tc ? 32 : 64;
    const int cta_rows = use_tc ? 128 : 64;
    a.n_tiles = (int)((a.N + cta_rows - 1) / cta_rows);
    a.ws = ws;

    // status[0] accumulates out-of-range indices during the encode kernel; the finalize kernel publishes it to
    // status[3] and clears it for the next call, so a steady-state call (REUSE_PREP) needs no memset and the encode
    // kernel can be launched as a programmatic dependent of whatever ran before it on the stream.
    if (!reuse_prep) C2V_CUDA_OK(cudaMemsetAsync(ws.status, 0, 256, st));
    int rc = C2V_OK;
    if (!reuse_prep)
        rc = use_tc ? launch_split_w_tcgen05(d, p->input_linear, a.ws, st)
                    : launch_transpose_w(p->input_linear, ws.w_t, a.H, a.D, (a.H + 3) / 4 * 4, st);
    if (rc != C2V_OK) return rc;
    int slot = -1;
    if (g_prof_on && (g_prof_calls++ % g_prof_stride) == 0) {
        if (g_prof_pending == kProfRing) { rc = prof_drain(); if (rc != C2V_OK) return rc; }
        slot = g_prof_pending;
        C2V_CUDA_OK(cudaEventRecord(g_prof_ev[slot][0], st));
    }
    rc = use_tc ? launch_encode_tm(a, st) : launch_encode_ffma(a, st);
    if (rc != C2V_OK) return rc;
    if (slot >= 0) {
        C2V_CUDA_OK(cudaEventRecord(g_prof_ev[slot][1], st));
        g_prof_pending = slot + 1;
    }
    return launch_encode_finalize(a, B, code_vector, st);
}

int c2v_profile_enable(int32_t on)
{
    if (on && !g_prof_made) {
        for (int i = 0; i < kProfRing; ++i)
            for (int j = 0; j < 2; ++j) C2V_CUDA_OK(cudaEventCreate(&g_prof_ev[i][j]));
        g_prof_made = true;
    }
    g_prof_on = on != 0;
    g_prof_stride = on > 1 ? on : 1;
    g_prof_calls = 0;
    g_prof_pending = 0; g_prof_ms = 0.0; g_prof_count = 0;
    return C2V_OK;
}

int c2v_profile_read(double *kernel_ms, int64_t *launches)
{
    int rc = prof_drain();
    if (rc != C2V_OK) return rc;
    if (kernel_ms) *kernel_ms = g_prof_ms;
    if (launches) *launches = g_prof_count;
    return C2V_OK;
}

int64_t c2v_workspace_status(void *workspace, void *stream)
{
    if (!workspace) { set_error("workspace is NULL"); return C2V_EINVAL; }
    long long v = 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    C2V_CUDA_OK(cudaMemcpyAsync(&v, static_cast<const char *>(workspace) + 24, sizeof(v), cudaMemcpyDeviceToHost, st));
    C2V_CUDA_OK(cudaStreamSynchronize(st));
    return v;
}

int c2v_workspace_set_status_mirror(void *workspace, int64_t *pinned_host_word, void *stream)
{
    if (!workspace) { set_error("workspace is NULL"); return C2V_EINVAL; }
    long long hdr[2] = {0, 0};
    if (pinned_host_word) {
        cudaPointerAttributes at;
        C2V_CUDA_OK(cudaPointerGetAttributes(&at, pinned_host_word));
        if (at.type != cudaMemoryTypeHost || !at.devicePointer) {
            set_error("c2v_workspace_set_status_mirror: the mirror must be pinned (page-locked, device-mapped) host memory");
            return C2V_EINVAL;
        }
        hdr[0] = (long long)reinterpret_cast<uintptr_t>(at.devicePointer);
        hdr[1] = hdr[0] ^ C2V_MIRROR_MAGIC;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // pageable source: the copy is staged before the call returns, so the stack buffer may go away
    C2V_CUDA_OK(cudaMemcpyAsync(static_cast<char *>(workspace) + 512, hdr, sizeof(hdr), cudaMemcpyHostToDevice, st));
    return C2V_OK;
}

size_t c2v_label_workspace_bytes(const c2v_dims *d, int32_t B)
{
    if (!dims_ok(d) || B < 1) return 0;
    // split fp16 images of cv and W_out for the tcgen05 label GEMM (unused by the FFMA path)
    return align_up(label_tcgen05_workspace_bytes(d, B), 1024);
}

int c2v_label_logits(const c2v_dims *d, const c2v_params *p, const float *code_vector, int32_t B,
                     float *outputs, void *workspace, size_t workspace_bytes, int32_t algo,
                     void *stream)
{
    if (!dims_ok(d)) return C2V_EINVAL;
    if (!p || !p->output_weight || !code_vector || !outputs || B < 1 || d->label_count < 1) {
        set_error("c2v_label_logits: bad argument");
        return C2V_EINVAL;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int H = d->encode;
    const long long C = d->label_count;
    const bool reuse_prep = (algo & C2V_FLAG_REUSE_PREP) != 0;
    g_pdl_this_call = (algo & C2V_FLAG_NO_PDL) == 0;
    algo &= 0xff;
    if (algo == C2V_ALGO_TCGEN05 || (algo == C2V_ALGO_AUTO && label_tcgen05_shape_ok(d))) {
        return launch_label_tcgen05(d, code_vector, B, p->output_weight, p->output_bias, outputs, nullptr,
                                    nullptr, workspace, workspace_bytes, reuse_prep, st);
    }
    // outputs[b,c] = sum_h cv[b,h] * W_out[c,h] + bias[c]   (model.py:83)
    return launch_sgemm(B, (int)C, H, code_vector, H, 1, p->output_weight, 1, H, p->output_bias,
                        outputs, C, false, st);
}

int c2v_label_logits_argmax(const c2v_dims *d, const c2v_params *p, const float *code_vector, int32_t B,
                            float *outputs, int64_t *argmax, float *maxval, void *workspace,
                            size_t workspace_bytes, int32_t algo, void *stream)
{
    if (!dims_ok(d)) return C2V_EINVAL;
    if (!p || !p->output_weight || !code_vector || B < 1 || d->label_count < 1 || (!outputs && !argmax && !maxval)) {
        set_error("c2v_label_logits_argmax: bad argument");
        return C2V_EINVAL;
    }
    if (!outputs && !c2v_label_loss_supported(d, B)) {       // arg-max without the logits needs the fused tensor-core epilogue
        set_error("c2v_label_logits_argmax: outputs == NULL needs encode_size %% 4 == 0, <= 256 and B <= 2048");
        return C2V_EUNSUPPORTED;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool reuse_prep = (algo & C2V_FLAG_REUSE_PREP) != 0;
    g_pdl_this_call = (algo & C2V_FLAG_NO_PDL) == 0;
    const int base_algo = algo & 0xff;
    if (base_algo == C2V_ALGO_TCGEN05 || (base_algo == C2V_ALGO_AUTO && label_tcgen05_shape_ok(d)))
        return launch_label_tcgen05(d, code_vector, B, p->output_weight, p->output_bias, outputs,
                                    reinterpret_cast<long long *>(argmax), maxval, workspace, workspace_bytes,
                                    reuse_prep, st);
    int rc = c2v_label_logits(d, p, code_vector, B, outputs, workspace, workspace_bytes, algo, stream);
    if (rc != C2V_OK || (!argmax && !maxval)) return rc;
    return launch_loss_argmax(outputs, nullptr, B, d->label_count, nullptr,
                              reinterpret_cast<long long *>(argmax), maxval, nullptr, st);
}

int c2v_label_loss_supported(const c2v_dims *d, int32_t B)
{
    if (!dims_ok(d) || B < 1) return 0;
    return (label_tcgen05_shape_ok(d) && B <= 2048) ? 1 : 0;
}

int c2v_label_loss_argmax(const c2v_dims *d, const c2v_params *p, const float *code_vector, const int64_t *label,
                          int32_t B, float *outputs, float *loss, float *lse, int64_t *argmax, float *maxval,
                          void *workspace, size_t workspace_bytes, int32_t algo, void *stream)
{
    if (!dims_ok(d)) return C2V_EINVAL;
    if (!p || !p->output_weight || !code_vector || !label || B < 1 || d->label_count < 1 || (!loss && !lse)) {
        set_error("c2v_label_loss_argmax: bad argument");
        return C2V_EINVAL;
    }
    if (!c2v_label_loss_supported(d, B)) {
        set_error("c2v_label_loss_argmax: the fused loss needs encode_size %% 4 == 0, <= 256 and B <= 2048 (got %d, %d); use "
                  "c2v_label_logits + c2v_loss_argmax", d->encode, B);
        return C2V_EUNSUPPORTED;
    }
    const bool reuse_prep = (algo & C2V_FLAG_REUSE_PREP) != 0;
    g_pdl_this_call = (algo & C2V_FLAG_NO_PDL) == 0;
    LabelLossArgs la;
    memset(&la, 0, sizeof(la));
    la.label = reinterpret_cast<const long long *>(label); la.loss = loss; la.lse_out = lse;
    return launch_label_tcgen05_ex(d, code_vector, B, p->output_weight, p->output_bias, outputs,
                                   reinterpret_cast<long long *>(argmax), maxval, workspace, workspace_bytes, reuse_prep,
                                   static_cast<cudaStream_t>(stream), &la);
}

int c2v_label_dlogits(const c2v_dims *d, const c2v_params *p, const float *code_vector, const int64_t *label,
                      const float *lse, int32_t B, float scale, const float *scale_device, float *d_outputs,
                      void *workspace, size_t workspace_bytes, int32_t algo, void *stream)
{
    if (!dims_ok(d)) return C2V_EINVAL;
    if (!p || !p->output_weight || !code_vector || !label || !lse || !d_outputs || B < 1 || d->label_count < 1) {
        set_error("c2v_label_dlogits: bad argument");
        return C2V_EINVAL;
    }
    if (!label_tcgen05_shape_ok(d)) {
        set_error("c2v_label_dlogits: needs encode_size %% 4 == 0 and <= 256 (got %d)", d->encode);
        return C2V_EUNSUPPORTED;
    }
    const bool reuse_prep = (algo & C2V_FLAG_REUSE_PREP) != 0;
    g_pdl_this_call = false;
    LabelLossArgs la;
    memset(&la, 0, sizeof(la));
    la.label = reinterpret_cast<const long long *>(label); la.dlogits_lse = lse; la.dscale = scale; la.dscale_ptr = scale_device;
    return launch_label_tcgen05_ex(d, code_vector, B, p->output_weight, p->output_bias, d_outputs, nullptr, nullptr,
                                   workspace, workspace_bytes, reuse_prep, static_cast<cudaStream_t>(stream), &la);
}

int c2v_angular_logits(const c2v_dims *d, const c2v_params *p, const float *code_vector,
                       const int64_t *label, int32_t B, float margin, float inverse_temp,
                       float *outputs, void *stream)
{
    if (!dims_ok(d)) return C2V_EINVAL;
    if (!p || !p->output_weight || !code_vector || !outputs || !label || B < 1) {
        set_error("c2v_angular_logits: bad argument");
        return C2V_EINVAL;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    float *scratch = nullptr;
    C2V_CUDA_OK(cudaMallocAsync(&scratch, (size_t)(B + d->label_count) * sizeof(float), st));
    int rc = launch_angular(d, p, code_vector, reinterpret_cast<const long long *>(label), B, margin,
                            inverse_temp, outputs, scratch, st, nullptr);
    cudaFreeAsync(scratch, st);
    return rc;
}

int c2v_angular_forward_train(const c2v_dims *d, const c2v_params *p, const float *code_vector, const int64_t *label,
                              int32_t B, float margin, float inverse_temp, float *outputs, float *cosine,
                              float *inv_norms, void *stream)
{
    if (!dims_ok(d)) return C2V_EINVAL;
    if (!p || !p->output_weight || !code_vector || !outputs || !label || !cosine || !inv_norms || B < 1) {
        set_error("c2v_angular_forward_train: bad argument");
        return C2V_EINVAL;
    }
    return launch_angular(d, p, code_vector, reinterpret_cast<const long long *>(label), B, margin, inverse_temp, outputs,
                          inv_norms, static_cast<cudaStream_t>(stream), cosine);
}

int c2v_angular_backward(const c2v_dims *d, const c2v_params *p, const float *code_vector, const int64_t *label,
                         int32_t B, float margin, float inverse_temp, const float *cosine, const float *inv_norms,
                         float *d_outputs, float *d_code_vector, float *d_output_weight, float *scratch, void *stream)
{
    if (!dims_ok(d)) return C2V_EINVAL;
    if (!p || !p->output_weight || !code_vector || !label || !cosine || !inv_norms || !d_outputs || !scratch || B < 1) {
        set_error("c2v_angular_backward: bad argument");
        return C2V_EINVAL;
    }
    return launch_angular_backward(d, p, code_vector, reinterpret_cast<const long long *>(label), B, margin, inverse_temp,
                                   cosine, inv_norms, inv_norms + B, d_outputs, d_code_vector, d_output_weight, scratch,
                                   static_cast<cudaStream_t>(stream));
}

int c2v_loss_argmax(const float *outputs, const int64_t *label, int32_t B, int64_t C, float *loss,
                    int64_t *argmax, float *maxval, float *d_outputs, void *stream)
{
    if (!outputs || B < 1 || C < 1) { set_error("c2v_loss_argmax: bad argument"); return C2V_EINVAL; }
    if ((loss || d_outputs) && !label) {
        set_error("c2v_loss_argmax: loss / d_outputs need label");
        return C2V_EINVAL;
    }
    return launch_loss_argmax(outputs, reinterpret_cast<const long long *>(label), B, C, loss,
                              reinterpret_cast<long long *>(argmax), maxval, d_outputs,
                              static_cast<cudaStream_t>(stream));
}

int c2v_label_backward(const c2v_dims *d, const c2v_params *p, const float *code_vector,
                       const float *d_outputs, int32_t B, float *d_code_vector,
                       float *d_output_weight, float *d_output_bias, void *stream)
{
    if (!dims_ok(d)) return C2V_EINVAL;
    if (!p || !p->output_weight || !code_vector || !d_outputs || B < 1) {
        set_error("c2v_label_backward: bad argument");
        return C2V_EINVAL;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int H = d->encode;
    const long long C = d->label_count;
    int rc = C2V_OK;
    if (d_code_vector)   // d_cv[b,h] = sum_c d_out[b,c] W_out[c,h]
        rc = launch_sgemm(B, H, (int)C, d_outputs, C, 1, p->output_weight, H, 1, nullptr,
                          d_code_vector, H, false, st);
    if (rc != C2V_OK) return rc;
    if (d_output_weight) // dW_out[c,h] = sum_b d_out[b,c] cv[b,h]
        rc = launch_sgemm((int)C, H, B, d_outputs, 1, C, code_vector, H, 1, nullptr, d_output_weight,
                          H, false, st);
    if (rc != C2V_OK) return rc;
    if (d_output_bias) rc = launch_colsum(d_outputs, B, C, d_output_bias, st);
    return rc;
}

int c2v_label_backward_ws(const c2v_dims *d, const c2v_params *p, const float *code_vector, const float *d_outputs,
                          int32_t B, float *d_code_vector, float *d_output_weight, float *d_output_bias, void *workspace,
                          size_t workspace_bytes, int32_t algo, void *stream)
{
    if (!dims_ok(d)) return C2V_EINVAL;
    if (!p || !p->output_weight || !code_vector || !d_outputs || B < 1) {
        set_error("c2v_label_backward_ws: bad argument");
        return C2V_EINVAL;
    }
    const int base_algo = algo & 0xff;
    const bool tc = base_algo != C2V_ALGO_FFMA && workspace != nullptr && label_backward_tc_ok(d) &&
                    (d_output_weight != nullptr || d_output_bias == nullptr);
    if (!tc) {
        if (base_algo == C2V_ALGO_TCGEN05) {
            set_error("tensor-core label backward needs a label workspace, encode_size %% 4 == 0 and <= 256");
            return C2V_EUNSUPPORTED;
        }
        return c2v_label_backward(d, p, code_vector, d_outputs, B, d_code_vector, d_output_weight, d_output_bias, stream);
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const uint8_t *img = nullptr, *cv_img = nullptr; const float *hdr = nullptr; unsigned *scratch = nullptr;
    int rc = label_w_image(d, p->output_weight, B, workspace, workspace_bytes, (algo & C2V_FLAG_REUSE_PREP) != 0, st, &img, &hdr,
                           &scratch, &cv_img);
    if (rc != C2V_OK) return rc;
    // after c2v_label_dlogits on this workspace (the flag's contract: same code_vector, nothing in between) the workspace also
    // holds max |d_outputs| and the fp16 image of code_vector: the backward reads both instead of recomputing them
    const bool from_dlogits = (algo & C2V_FLAG_GRAD_ABSMAX_READY) != 0 && label_ws_holds_dlogits_of(workspace, code_vector, B);
    return launch_label_backward_tc(d, code_vector, d_outputs, B, img, hdr, d_code_vector, d_output_weight, d_output_bias,
                                    scratch, st, from_dlogits, from_dlogits ? cv_img : nullptr);
}

size_t c2v_encode_backward_workspace_bytes(const c2v_dims *d, int32_t B, int32_t L)
{
    if (!dims_ok(d) || B < 1 || L < 1) return 0;
    return encode_backward_workspace_bytes(d, B, L);
}

int c2v_encode_backward(const c2v_dims *d, const c2v_params *p, const int64_t *starts,
                        const int64_t *paths, const int64_t *ends, int32_t B, int32_t L,
                        const c2v_dropout *drop, const float *code_vector, const float *attention,
                        const float *d_code_vector, const float *d_attention, const c2v_grads *grads,
                        void *workspace, size_t workspace_bytes, void *stream)
{
    return c2v_encode_backward_stashed(d, p, starts, paths, ends, B, L, drop, code_vector, attention, nullptr,
                                       d_code_vector, d_attention, grads, workspace, workspace_bytes, stream);
}

int c2v_encode_backward_stashed(const c2v_dims *d, const c2v_params *p, const int64_t *starts,
                                const int64_t *paths, const int64_t *ends, int32_t B, int32_t L,
                                const c2v_dropout *drop, const float *code_vector, const float *attention,
                                const float *x_stash, const float *d_code_vector, const float *d_attention,
                                const c2v_grads *grads, void *workspace, size_t workspace_bytes, void *stream)
{
    return c2v_encode_backward_phased(d, p, starts, paths, ends, B, L, drop, code_vector, attention, x_stash, d_code_vector,
                                      d_attention, grads, workspace, workspace_bytes, 0, stream);
}

int c2v_encode_backward_phased(const c2v_dims *d, const c2v_params *p, const int64_t *starts,
                               const int64_t *paths, const int64_t *ends, int32_t B, int32_t L,
                               const c2v_dropout *drop, const float *code_vector, const float *attention,
                               const float *x_stash, const float *d_code_vector, const float *d_attention,
                               const c2v_grads *grads, void *workspace, size_t workspace_bytes, int32_t phase, void *stream)
{
    if (phase < 0 || phase > 2) { set_error("c2v_encode_backward_phased: phase %d", phase); return C2V_EINVAL; }
    if (!dims_ok(d)) return C2V_EINVAL;
    if (!p || !starts || !paths || !ends || !code_vector || !attention || !d_code_vector || !grads ||
        !workspace || B < 1 || L < 1) {
        set_error("c2v_encode_backward: bad argument");
        return C2V_EINVAL;
    }
    if (!grads->terminal_embedding || !grads->path_embedding || !grads->input_linear ||
        !grads->ln_weight || !grads->ln_bias || !grads->attention) {
        set_error("c2v_encode_backward: NULL gradient pointer");
        return C2V_EINVAL;
    }
    EncodeArgs a;
    memset(&a, 0, sizeof(a));
    a.starts = reinterpret_cast<const long long *>(starts);
    a.paths = reinterpret_cast<const long long *>(paths);
    a.ends = reinterpret_cast<const long long *>(ends);
    a.emb_t = p->terminal_embedding; a.emb_p = p->path_embedding;
    a.ln_g = p->ln_weight; a.ln_b = p->ln_bias; a.attn = p->attention;
    a.T = d->terminal_count; a.P = d->path_count;
    a.Et = d->terminal_embed; a.Ep = d->path_embed; a.H = d->encode;
    a.D = 2 * a.Et + a.Ep;
    a.L = L; a.N = (long long)B * L;
    a.drop_p = 0.0f; a.drop_scale = 1.0f;
    if (drop && drop->training && drop->p > 0.0f && drop->p < 1.0f) {
        a.drop_p = drop->p; a.drop_scale = 1.0f / (1.0f - drop->p); a.seed = drop->seed;
    }
    return launch_encode_backward(d, p, a, B, code_vector, attention, d_code_vector, d_attention,
                                  grads, workspace, workspace_bytes,
                                  static_cast<cudaStream_t>(stream), x_stash, phase);
}

}  // extern "C"
