/*
 * c2v_b200.h -- C ABI of the B200-native code2vec path-attention encoder.
 *
 * This is the drop-in boundary for ONE hot path of sonoisa/code2vec:
 *   Code2Vec.forward(starts, paths, ends, label) -> (outputs, code_vector, attention)
 *   /root/reference/model/model.py:44-88 (+ get_attention, model.py:90-105),
 * its autograd backward (what loss.backward() at main.py:174 runs through it) and
 * the loss/argmax consumers next to it (main.py:251-264, main.py:285).
 *
 * The reference has no FFI of its own (it is pure PyTorch, SURVEY.md 8b); the
 * binding a maintainer adds is the ctypes stub in INTEGRATION.md, which is what
 * code2vec_b200/_lib.py contains.  No torch types appear here: plain pointers
 * and sizes, `void* stream` is a cudaStream_t.
 *
 * Conventions
 *   - all tensors are dense row-major fp32 / int64, exactly the reference's
 *     dtypes (dataset_builder.py:206-209 builds int64 indices; parameters fp32);
 *   - "device" entry points take device pointers and never synchronise or
 *     allocate: the caller passes a workspace of c2v_*_workspace_bytes();
 *   - "host" entry points take host pointers, copy in/out on the given stream
 *     and synchronise before returning;
 *   - every function returns C2V_OK (0) or a negative C2V_E* code;
 *     c2v_last_error() gives the message for the calling thread.
 *   - index semantics: starts/ends in [0,T), paths in [0,P).  The reference
 *     raises IndexError (CPU) / device-asserts (CUDA) on violations
 *     (SURVEY.md 8b "Call"); here out-of-range indices are clamped to row 0 and
 *     counted in the workspace status word, which the host entry points turn
 *     into C2V_EINDEX and c2v_workspace_status() exposes to device callers.
 */
#ifndef C2V_B200_H
#define C2V_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define C2V_ABI_VERSION 1

enum {
    C2V_OK = 0,
    C2V_EINVAL = -1,   /* bad argument (shape, null pointer, alignment)            */
    C2V_ECUDA = -2,    /* a CUDA runtime call or launch failed                     */
    C2V_EWORKSPACE = -3, /* workspace too small                                    */
    C2V_EINDEX = -4,   /* an index was out of range (reference: IndexError)        */
    C2V_EUNSUPPORTED = -5 /* requested algorithm cannot run this shape / device    */
};

/* Which encode / GEMM implementation to run. AUTO picks TCGEN05 when the shape
 * is supported (see c2v_encode_supports_tcgen05) and FFMA otherwise. */
enum {
    C2V_ALGO_AUTO = 0,
    C2V_ALGO_FFMA = 1,    /* fp32 CUDA-core path, any shape                         */
    C2V_ALGO_TCGEN05 = 2  /* tcgen05.mma kind::f16, 3-pass hi/lo split, fp32-accurate */
};

/* OR-ed into `algo`: the caller guarantees that the parameters behind this workspace have not
 * changed since the previous call that used it, so the derived weight images (transposed /
 * hi-lo split copies of input_linear and output_linear kept in the workspace) are reused
 * instead of rebuilt.  The torch module sets it from the parameters' version counters. */
#define C2V_FLAG_REUSE_PREP 0x100
/* OR-ed into `algo`: launch this call's kernels as plain stream-ordered launches instead of programmatic dependent
 * launches (the default overlaps each kernel's prologue with its predecessor's tail).  The training forward
 * (c2v_encode_forward_stash with a stash) always does. */
#define C2V_FLAG_NO_PDL 0x200
/* OR-ed into `algo` of c2v_label_backward_ws: `d_outputs` is what c2v_label_dlogits wrote with this same workspace for
 * this same `code_vector` and B (and no other call has used the workspace since).  The workspace then already holds
 * max |d_outputs| -- the scale of the fp16 split -- and the fp16 image of code_vector, so the pass over the [B, C] gradient
 * that finds the former and the per-tile conversion of the latter are skipped.  Same results either way.  The library
 * checks the claim against what its last label call on this host thread used (workspace, code_vector, B) and ignores the
 * flag when they differ. */
#define C2V_FLAG_GRAD_ABSMAX_READY 0x400

/* Sizes read from the reference's Option (main.py:93-115) by Code2Vec.__init__
 * (model.py:18-42). */
typedef struct c2v_dims {
    int64_t terminal_count;   /* T: rows of terminal_embedding   (model.py:21) */
    int64_t path_count;       /* P: rows of path_embedding       (model.py:22) */
    int64_t label_count;      /* C: rows of output_linear        (model.py:41) */
    int32_t terminal_embed;   /* E_t                                            */
    int32_t path_embed;       /* E_p                                            */
    int32_t encode;           /* H: input_linear out features    (model.py:23) */
    int32_t reserved;
} c2v_dims;

/* Parameters, named as in the reference state_dict (SURVEY.md section 5). */
typedef struct c2v_params {
    const float *terminal_embedding;  /* [T, E_t]              model.py:21 */
    const float *path_embedding;      /* [P, E_p]              model.py:22 */
    const float *input_linear;        /* [H, 2E_t+E_p] no bias model.py:23 */
    const float *ln_weight;           /* [H]                   model.py:24 */
    const float *ln_bias;             /* [H]                   model.py:24 */
    const float *attention;           /* [H]                   model.py:31 */
    const float *output_weight;       /* [C, H]                model.py:33/41 */
    const float *output_bias;         /* [C] or NULL (angular) model.py:41-42 */
} c2v_params;

/* Gradients, same shapes as c2v_params.  The embedding / linear gradients are
 * ACCUMULATED into (atomics), so the caller zero-fills them (optimizer.zero_grad,
 * main.py:171); the small ones are overwritten. */
typedef struct c2v_grads {
    float *terminal_embedding;
    float *path_embedding;
    float *input_linear;
    float *ln_weight;
    float *ln_bias;
    float *attention;
} c2v_grads;

/* Dropout after tanh (model.py:26-29, :60-61): keep-prob 1-p, survivors scaled by
 * 1/(1-p).  The mask is a counter-based hash of (seed, context row, column), so
 * backward regenerates it instead of storing it. training==0 or p outside (0,1)
 * means identity, as in the reference. */
typedef struct c2v_dropout {
    float p;
    int32_t training;
    uint64_t seed;
} c2v_dropout;

int c2v_abi_version(void);
const char *c2v_last_error(void);

/* Device facts the host side sizes grids with. */
typedef struct c2v_device_info {
    int32_t cc_major, cc_minor, sm_count, reserved;
    int64_t global_mem_bytes;
    int64_t smem_per_block_optin;
} c2v_device_info;
int c2v_get_device_info(int device, c2v_device_info *out);

/* 1 if the tcgen05 encode kernel handles this shape on this device. */
int c2v_encode_supports_tcgen05(const c2v_dims *d);

/* ---- encode: model.py:48-69 + 90-96 as one fused pass ------------------------------
 * gathers -> concat -> input_linear -> LayerNorm -> tanh -> dropout -> masked
 * attention softmax over the bag -> weighted sum.
 *   starts/paths/ends : int64 [B, L] device
 *   code_vector [B, H], attention [B, L] : fp32 device, overwritten
 * Workspace holds the split weights, the per-(tile,bag) softmax partials and a
 * status word; contents are needed by c2v_encode_backward for the same batch.
 * Operand range of the tensor-core path (algo TCGEN05 / AUTO; the FFMA path is plain fp32): every fp32 operand
 * of a GEMM is split into fp16 hi + lo.  input_linear.weight, W_out and the gradients are first scaled by a power
 * of two from their max |value|; the gathered embeddings (here and in the dW backward) and the code vectors (label
 * GEMM and its backward) are split as they are.  So those must satisfy |value| < 65504 (fp16 overflow; not
 * checked), and they keep full fp32-level accuracy only above about 2^-8 in magnitude: below 2^-14 the lo half is
 * an fp16 subnormal, which caps each element's absolute precision at about 2^-25.  LayerNorm makes the forward
 * insensitive to that (tested at embedding std 2^-8 .. 2^8); the dW backward's relative error grows as about
 * 2^-25 / std(embedding). */
size_t c2v_encode_workspace_bytes(const c2v_dims *d, int32_t B, int32_t L);
int c2v_encode_forward(const c2v_dims *d, const c2v_params *p,
                       const int64_t *starts, const int64_t *paths, const int64_t *ends,
                       int32_t B, int32_t L, const c2v_dropout *drop,
                       float *code_vector, float *attention,
                       void *workspace, size_t workspace_bytes, int32_t algo, void *stream);
/* Training forward: additionally keeps the input_linear output x = c . W^T (model.py:54, before LayerNorm) of every
 * context row in x_stash [B*L, H] (fp32, device) for c2v_encode_backward_stashed; x_stash == NULL: c2v_encode_forward. */
int c2v_encode_forward_stash(const c2v_dims *d, const c2v_params *p, const int64_t *starts,
                             const int64_t *paths, const int64_t *ends, int32_t B, int32_t L,
                             const c2v_dropout *drop, float *code_vector, float *attention, float *x_stash,
                             void *workspace, size_t workspace_bytes, int32_t algo, void *stream);

/* Reads the status word of the last encode on this workspace (synchronises the
 * stream): returns the number of out-of-range indices seen, or a negative code. */
int64_t c2v_workspace_status(void *workspace, void *stream);
/* Deferred error surface for device callers: registers a pinned (page-locked) host int64 with an encode workspace; every
 * later c2v_encode_forward* on that workspace ADDS its count of out-of-range indices to the host word (nothing is written
 * when the count is 0), so the caller can poll the word at its next call -- no synchronisation -- and raise IndexError, as
 * late as the reference's own CUDA device assert would (SURVEY.md 8b "Call").  NULL unregisters. */
int c2v_workspace_set_status_mirror(void *workspace, int64_t *pinned_host_word, void *stream);

/* ---- label head --------------------------------------------------------------------
 * plain:   outputs = cv . W_out^T + b                                   model.py:83
 * angular: cosine head with margin on the true class, times inverse_temp model.py:71-80
 *          (needs label, also in eval).
 * cv [B,H], outputs [B,C] device fp32; label int64 [B] device. */
size_t c2v_label_workspace_bytes(const c2v_dims *d, int32_t B);
int c2v_label_logits(const c2v_dims *d, const c2v_params *p, const float *code_vector, int32_t B,
                     float *outputs, void *workspace, size_t workspace_bytes, int32_t algo,
                     void *stream);
/* Training through the angular-margin head (model.py:71-80 under loss.backward(), main.py:174).
 * c2v_angular_forward_train = c2v_angular_logits that also keeps cosine [B, C] and inv_norms [B + C]
 * (1 / max(|cv_b|, 1e-12) then 1 / max(|W_c|, 1e-12), F.normalize's clamp) for the backward.
 * c2v_angular_backward: d_outputs [B, C] is OVERWRITTEN (it becomes d loss / d (cv . W^T)); d_code_vector [B, H] and
 * d_output_weight [C, H] are written (either may be NULL); scratch: B + C floats. */
int c2v_angular_forward_train(const c2v_dims *d, const c2v_params *p, const float *code_vector, const int64_t *label,
                              int32_t B, float margin, float inverse_temp, float *outputs, float *cosine,
                              float *inv_norms, void *stream);
int c2v_angular_backward(const c2v_dims *d, const c2v_params *p, const float *code_vector, const int64_t *label,
                         int32_t B, float margin, float inverse_temp, const float *cosine, const float *inv_norms,
                         float *d_outputs, float *d_code_vector, float *d_output_weight, float *scratch, void *stream);

/* Loss fused into the label GEMM (SURVEY.md 8f row 1): model.py:83 + calculate_loss (main.py:251-264: log_softmax +
 * NLLLoss with weights == 1, mean over the batch) + torch.max(dim=1) (main.py:285) in one pass.  The epilogue of the
 * label kernel keeps, per row, (max, sum exp) partials, the target logit and the running arg-max, so the [B, C] logits
 * are never re-read -- and with outputs == NULL never written (800 MB per batch at the top11 label count).
 * loss: mean NLL (device scalar), lse: [B] logsumexp per row (what the backward needs), either may be NULL (not both).
 * Same workspace as c2v_label_logits.  c2v_label_loss_supported: encode_size % 4 == 0, <= 256, B <= 2048. */
int c2v_label_loss_supported(const c2v_dims *d, int32_t B);
int c2v_label_loss_argmax(const c2v_dims *d, const c2v_params *p, const float *code_vector, const int64_t *label,
                          int32_t B, float *outputs, float *loss, float *lse, int64_t *argmax, float *maxval,
                          void *workspace, size_t workspace_bytes, int32_t algo, void *stream);
/* Backward companion: recomputes the logits tile by tile and writes d loss / d outputs [B, C] =
 * (softmax(outputs) - onehot(label)) * scale (* *scale_device when not NULL: the upstream gradient of the scalar loss;
 * scale = 1 / B for the mean) straight from the accumulators; feed it to c2v_label_backward. */
int c2v_label_dlogits(const c2v_dims *d, const c2v_params *p, const float *code_vector, const int64_t *label,
                      const float *lse, int32_t B, float scale, const float *scale_device, float *d_outputs,
                      void *workspace, size_t workspace_bytes, int32_t algo, void *stream);
/* Label logits + the prediction the reference takes from them (`torch.max(preds, dim=1)`,
 * main.py:285; first maximum wins) in one call: the argmax pass runs right behind the GEMM while the
 * [B,C] logits are still in L2.  argmax int64 [B], maxval fp32 [B] (either may be NULL).
 * outputs == NULL (tensor-core path, B <= 2048: c2v_label_loss_supported): only the prediction is produced and the
 * logits are never written -- what predict() and the host-buffer calls do when the caller does not ask for them. */
int c2v_label_logits_argmax(const c2v_dims *d, const c2v_params *p, const float *code_vector, int32_t B,
                            float *outputs, int64_t *argmax, float *maxval, void *workspace,
                            size_t workspace_bytes, int32_t algo, void *stream);
int c2v_angular_logits(const c2v_dims *d, const c2v_params *p, const float *code_vector,
                       const int64_t *label, int32_t B, float margin, float inverse_temp,
                       float *outputs, void *stream);

/* ---- loss / predict next to the path ----------------------------------------------
 * main.py:251-264: mean over the batch of -log_softmax(outputs)[label] (NLLLoss
 * weights are identically 1, SURVEY.md 8a row 16); main.py:285: torch.max(dim=1).
 * Any of loss / argmax / maxval / d_outputs may be NULL.  d_outputs [B,C] receives
 * dLoss/doutputs = (softmax - onehot) / B. */
int c2v_loss_argmax(const float *outputs, const int64_t *label, int32_t B, int64_t C,
                    float *loss, int64_t *argmax, float *maxval, float *d_outputs, void *stream);

/* ---- backward ----------------------------------------------------------------------
 * Label head: d_cv = d_out . W_out ; dW_out = d_out^T . cv ; d_bias = sum_b d_out. */
int c2v_label_backward(const c2v_dims *d, const c2v_params *p, const float *code_vector,
                       const float *d_outputs, int32_t B, float *d_code_vector,
                       float *d_output_weight, float *d_output_bias, void *stream);
/* c2v_label_backward on the tensor cores (dW_out = d_out^T . cv with the column sums d_b folded in, d_cv = d_out . W_out
 * streaming the cached W_out image): `workspace` is the label workspace of c2v_label_logits* for this weight
 * (C2V_FLAG_REUSE_PREP in `algo` = its image is current, e.g. the forward of the same step built it;
 * C2V_FLAG_GRAD_ABSMAX_READY = d_outputs comes from c2v_label_dlogits on this workspace).  Falls back to
 * c2v_label_backward (CUDA cores) when workspace == NULL, encode_size % 4 != 0 or > 256, or algo == C2V_ALGO_FFMA. */
int c2v_label_backward_ws(const c2v_dims *d, const c2v_params *p, const float *code_vector, const float *d_outputs,
                          int32_t B, float *d_code_vector, float *d_output_weight, float *d_output_bias, void *workspace,
                          size_t workspace_bytes, int32_t algo, void *stream);

/* Encode: gradients of every encode parameter given d_code_vector [B,H] and
 * (optionally, may be NULL) d_attention [B,L]; formulas in DESIGN.md "Backward".
 * Recomputes the forward per context row (nothing but code_vector / attention is
 * stashed) and regenerates the dropout mask from `drop`. */
size_t c2v_encode_backward_workspace_bytes(const c2v_dims *d, int32_t B, int32_t L);
int c2v_encode_backward(const c2v_dims *d, const c2v_params *p,
                        const int64_t *starts, const int64_t *paths, const int64_t *ends,
                        int32_t B, int32_t L, const c2v_dropout *drop,
                        const float *code_vector, const float *attention,
                        const float *d_code_vector, const float *d_attention,
                        const c2v_grads *grads, void *workspace, size_t workspace_bytes,
                        void *stream);
/* The same with x = c . W^T (model.py:54) of every context row read from x_stash [B*L, H] -- written by
 * c2v_encode_forward_stash for the same batch -- instead of re-gathering the rows and redoing the GEMM
 * (x_stash == NULL: identical to c2v_encode_backward). */
int c2v_encode_backward_stashed(const c2v_dims *d, const c2v_params *p, const int64_t *starts,
                                const int64_t *paths, const int64_t *ends, int32_t B, int32_t L,
                                const c2v_dropout *drop, const float *code_vector, const float *attention,
                                const float *x_stash, const float *d_code_vector, const float *d_attention,
                                const c2v_grads *grads, void *workspace, size_t workspace_bytes, void *stream);
/* The same backward in two calls on the same workspace and gradient buffers (phase 0 = all at once = the call above):
 * phase 1 runs the per-row work, the path sub-vector of dC and dW -- afterwards the gradients of path_embedding and
 * input_linear are complete and nothing reads the embedding tables any more --, phase 2 the start / end sub-vectors
 * (terminal_embedding).  A data-parallel caller starts reducing
 * the path table between the two (ShardedFlatAdam.early_step).  Shapes that do not run on the tensor cores do
 * everything in phase 1. */
int c2v_encode_backward_phased(const c2v_dims *d, const c2v_params *p, const int64_t *starts,
                               const int64_t *paths, const int64_t *ends, int32_t B, int32_t L,
                               const c2v_dropout *drop, const float *code_vector, const float *attention,
                               const float *x_stash, const float *d_code_vector, const float *d_attention,
                               const c2v_grads *grads, void *workspace, size_t workspace_bytes, int32_t phase, void *stream);

/* ---- host-buffer call: what a reference-side caller with CPU tensors uses ----------
 * One whole Code2Vec.forward + torch.max for a batch held in HOST memory (pinned
 * for full speed): copies the int64 indices in, runs encode + label head +
 * argmax on `device`, copies code_vector / attention / prediction (and the
 * logits, if `outputs` is not NULL) back, synchronises.  Parameters stay on the
 * device (p holds device pointers).  Returns C2V_EINDEX if an index was out of
 * range.  `session` keeps the device staging buffers between calls. */
typedef struct c2v_session c2v_session;
int c2v_session_create(int device, const c2v_dims *d, int32_t max_B, int32_t L, c2v_session **out);
void c2v_session_destroy(c2v_session *s);
int c2v_forward_host(c2v_session *s, const c2v_params *p,
                     const int64_t *starts, const int64_t *paths, const int64_t *ends,
                     const int64_t *label, int32_t B,
                     float *outputs /* [B,C] or NULL */, float *code_vector /* [B,H] */,
                     float *attention /* [B,L] */, int64_t *pred_label /* [B] or NULL */,
                     float *pred_score /* [B] or NULL */, int32_t algo);
/* Pipelined variant: enqueue only (H2D, kernels, D2H on the session's streams);
 * c2v_session_wait() blocks until batch `ticket` has fully landed in the host
 * buffers.  Lets step i+1's H2D overlap step i's kernels (double buffered). */
int c2v_forward_host_async(c2v_session *s, const c2v_params *p,
                           const int64_t *starts, const int64_t *paths, const int64_t *ends,
                           const int64_t *label, int32_t B,
                           float *outputs, float *code_vector, float *attention,
                           int64_t *pred_label, float *pred_score, int32_t algo, int64_t *ticket);
int c2v_session_wait(c2v_session *s, int64_t ticket);

/* On-GPU batch construction for the method-name task: replaces DatasetBuilder.build_data
 * (model/dataset_builder.py:112-150, infer_method branch; SURVEY.md 8f row 2).  The corpus stays on the device as CSR:
 * offsets [n_items + 1] (int64), contexts [offsets[n_items]][3] (int32: start, path, end), item_labels [n_items]
 * (int64, may be NULL).  Row b of starts / paths / ends [B, L] (int64, device) receives a uniformly random subset of
 * min(n, L) contexts of method item_ids[b] -- the reference shuffles and truncates -- with @method_0 rewritten to
 * @question (:136-143) and a zero-padded suffix (:212-219); label[b] = item_labels[item_ids[b]] (label may be NULL).
 * The choice is a pure function of (seed, item, context index); an item id outside [0, n_items) yields an all-pad row. */
int c2v_build_batch(const int64_t *offsets, const int32_t *contexts, int64_t n_items,
                    const int64_t *item_ids, const int64_t *item_labels, int32_t B, int32_t L,
                    uint64_t seed, int64_t method_token, int64_t question_token, int64_t *starts,
                    int64_t *paths, int64_t *ends, int64_t *label, void *stream);

/* The variable-name task of the same builder (/root/reference/model/dataset_builder.py:152-204, `--infer_variable_name`):
 * a unit is an (item, @var_k alias) pair -- unit_item / unit_var (terminal index of @var_k) / unit_label [n_units], in the
 * reference's order (items in order, aliases in CodeData.aliases order).  Row b of the outputs is the bag of unit
 * unit_ids[b]: the contexts of the item whose start or end is @var_k, @var_k rewritten to @question (:181-182, :190-191),
 * every other token t with var_pos[t] >= 0 mapped to variable_indexes[sigma(var_pos[t])] when shuffle_variable_indexes
 * != 0 (sigma: a per-(seed, item) permutation, :166-168; var_pos is int32 [terminal_count], -1 for non-variables), a
 * uniformly random subset of min(n, L) of them (:193-195) and a zero-padded suffix (:196-198). */
int c2v_build_batch_vars(const int64_t *offsets, const int32_t *contexts, int64_t n_items,
                         const int64_t *unit_item, const int64_t *unit_var, const int64_t *unit_label,
                         int64_t n_units, const int64_t *unit_ids, int32_t B, int32_t L, uint64_t seed,
                         int64_t question_token, const int32_t *var_pos, int64_t terminal_count,
                         const int64_t *variable_indexes, int32_t n_vars, int32_t shuffle_variable_indexes,
                         int64_t *starts, int64_t *paths, int64_t *ends, int64_t *label, void *stream);

/* Fused flat-buffer Adam (SURVEY.md 8f row 3): torch.optim.Adam(..., lr, betas, weight_decay) of main.py:138 +
 * optimizer.step() (:175) + optimizer.zero_grad() (:171) for all parameters in one launch.  param / grad / exp_avg /
 * exp_avg_sq: fp32 [n] device buffers, 16-byte aligned; `step` is the 1-based step count (bias corrections);
 * the gradient is read as grad * grad_scale (1/world after a summing all_reduce) and, if zero_grad != 0, left zeroed. */
int c2v_adam_step(float *param, float *grad, float *exp_avg, float *exp_avg_sq, int64_t n, float lr,
                  float beta1, float beta2, float eps, float weight_decay, int64_t step, float grad_scale,
                  int32_t zero_grad, void *stream);

/* The same optimizer for data-parallel training, fused with its collective (SURVEY.md 8e: "one all_reduce per step"
 * becomes one kernel per rank): for the rank's slice [slice_begin, slice_begin + slice_n) of the flat buffers the kernel
 * (1) sums the gradients of all ranks -- `multimem.ld_reduce` on grad_multicast (NVSwitch in-switch reduction) or, when
 * the multicast pointers are NULL, loads from grad_peers[0..world) in rank order over NVLink peer mappings --, (2) runs
 * Adam on param_local[slice] with exp_avg_slice / exp_avg_sq_slice (optimizer state is sharded: slice_n elements),
 * (3) stores the new parameters into every rank's buffer (`multimem.st` on param_multicast, or param_peers[r]), and
 * (4) zero-fills zero_buffer[0..zero_n) (the rank's other gradient bucket) while the links are busy.  param_peers /
 * grad_peers are HOST arrays of `world` device pointers.  slice_begin, slice_n, zero_n: multiples of 4 elements.
 * The caller provides the two cross-GPU barriers around the launch (all gradients complete / all stores landed). */
int c2v_adam_step_sharded(const float *param_local, float *param_multicast, const float *grad_multicast,
                          float *const *param_peers, const float *const *grad_peers, int32_t world,
                          float *exp_avg_slice, float *exp_avg_sq_slice, int64_t slice_begin, int64_t slice_n,
                          float *zero_buffer, int64_t zero_n, float lr, float beta1, float beta2, float eps,
                          float weight_decay, int64_t step, float grad_scale, void *stream);

/* The same sharded step for one slice, driven by bulk-async copies: one warp and 28 KB of shared memory per CTA, so that
 * it fits on SMs that a persistent tensor-core kernel already occupies (used on a side stream for the gradients that are
 * complete before the backward ends: ShardedFlatAdam.early_step).  Peer pointers only; no zero-fill.  max_ctas <= 0: one
 * CTA per SM. */
int c2v_adam_step_sharded_bulk(const float *param_local, float *const *param_peers, const float *const *grad_peers,
                               int32_t world, float *exp_avg_slice, float *exp_avg_sq_slice, int64_t slice_begin,
                               int64_t slice_n, float lr, float beta1, float beta2, float eps, float weight_decay,
                               int64_t step, float grad_scale, int32_t max_ctas, void *stream);

/* ---- corpus reader / code-vector writer (SURVEY.md 8f row 4): the data formats either side of the path ----------
 * c2v_corpus_parse_*: DatasetReader.load (/root/reference/model/dataset_reader.py:72-128) for the `corpus.txt` format
 * (`#id`, `label:`, `class:`, `paths:` + `start\tpath\tend` lines, `vars:` + `original\talias` lines, blank line between
 * items).  Several files are read as one concatenated stream (README: `cat splitted_corpus_*`).  question_shift =
 * QUESTION_TOKEN_INDEX (dataset_reader.py:11, added to start and end, :113-115).  A malformed line is C2V_EINVAL with
 * the line number in c2v_last_error() (the reference raises ValueError / IndexError there).  Host-only: no GPU needed. */
typedef struct c2v_corpus c2v_corpus;
typedef struct c2v_corpus_info {
    int64_t n_items, n_contexts, n_aliases, label_bytes, alias_bytes, alias_name_bytes;
} c2v_corpus_info;
int c2v_corpus_parse_buffer(const char *text, size_t n, int32_t question_shift, c2v_corpus **out);
int c2v_corpus_parse_files(const char *const *paths, int32_t n_paths, int32_t question_shift, c2v_corpus **out);
void c2v_corpus_free(c2v_corpus *c);
int c2v_corpus_get_info(const c2v_corpus *c, c2v_corpus_info *info);
/* Copies the parsed corpus into caller buffers (any pointer may be NULL = skip): ids [n_items] (-1: no `#` line),
 * ctx_offsets [n_items+1], contexts int32 [n_contexts][3] (the CSR image c2v_build_batch reads), label_offsets
 * [n_items+1] + label_blob (raw text after `label:`), has_label [n_items], label_pos [n_items] (aliases of the item that
 * precede its label line: vocabulary insertion order), alias_item_offsets [n_items+1], and per alias the original
 * variable name (alias_orig_offsets [n_aliases+1] + alias_blob) and the alias (alias_name_offsets + alias_name_blob). */
int c2v_corpus_export(const c2v_corpus *c, int64_t *ids, int64_t *ctx_offsets, int32_t *contexts,
                      int64_t *label_offsets, char *label_blob, uint8_t *has_label, int32_t *label_pos,
                      int64_t *alias_item_offsets, int64_t *alias_orig_offsets, char *alias_blob,
                      int64_t *alias_name_offsets, char *alias_name_blob);
/* Binary cache of a parsed corpus (one flat little-endian file). */
int c2v_corpus_save(const c2v_corpus *c, const char *path);
int c2v_corpus_load(const char *path, c2v_corpus **out);
/* Python's str(float) of an fp32 value (shortest round trip of the double it converts to); returns the length. */
int c2v_format_float(float value, char *out, size_t out_bytes);
/* write_code_vectors (/root/reference/main.py:393-423) for n rows: vector file lines `name\tv0 v1 ...` (:416) opened
 * with `mode` ("w" / "a"), preceded by the `n_items\tencode_size` header (main.py:227-228) when header_items >= 0; and,
 * when result_path != NULL, the test TSV `id\tTrue|False\tlabel\tpred\tmax_logit` (:420).  All pointers are HOST
 * memory; label / pred_label index the vocabulary given as names_blob + name_offsets [n_names+1]. */
int c2v_write_code_vectors(const char *vector_path, const char *mode, int64_t header_items, int64_t n, int32_t H,
                           const float *code_vectors, const int64_t *label, const char *names_blob,
                           const int64_t *name_offsets, int64_t n_names, const char *result_path, const char *result_mode,
                           const int64_t *ids, const int64_t *pred_label, const float *pred_score);

/* Counts kernels launched by this library since load (bench.py's gpu_launches). */
int64_t c2v_launch_count(void);

/* Measurement hook for bench.py's roofline: while enabled, every c2v_encode_forward brackets
 * its dominant kernel (the fused gather+encode+attention kernel, not the weight prep or the
 * per-bag finalize) with CUDA events on the launching stream.  c2v_profile_read synchronises
 * those events and returns the summed kernel milliseconds and the launch count since the last
 * enable; timing never runs under a profiler and adds no device work.  on > 1 samples every
 * on-th call only: an event between two launches keeps the second from starting as a
 * programmatic dependent of the first, so a throughput loop should sample, not bracket every step. */
int c2v_profile_enable(int32_t on);
int c2v_profile_read(double *kernel_ms, int64_t *launches);

#ifdef __cplusplus
}
#endif
#endif /* C2V_B200_H */
