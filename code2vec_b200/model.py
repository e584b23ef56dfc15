"""Drop-in `Code2Vec` for the reference's `model/model.py`, backed by the sm_100a kernels.

Boundary mirrored (SURVEY.md 8b):
  * constructor `Code2Vec(option)` reads the same Option fields (model.py:18-42) and creates
    the same submodules in the same order, so `torch.manual_seed(s); Code2Vec(option)` gives
    bit-identical initial weights and `state_dict()` keys/shapes interchange with the reference;
  * `forward(starts, paths, ends, label) -> (outputs, code_vector, attention)` (model.py:44-88),
    int64 [b, L] inputs, fp32 outputs, autograd-connected to every parameter;
  * `model.train()/eval()` toggle dropout only (model.py:60-61);
  * `from code2vec_b200.model import *` also exports `nn`, `F`, `torch`, `math`, `Parameter`,
    `NINF`, because the reference's main.py uses `nn` / `F` from that star import
    (main.py:22, :130, :261).

There is no CPU path: parameters and inputs must live on a CUDA (B200) device.
"""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.nn.parameter import Parameter

from . import _lib
from . import functional as CF

NINF = - 3.4 * math.pow(10, 38)  # model.py:12

__all__ = ["Code2Vec", "NINF", "torch", "nn", "F", "Parameter", "math"]


class _EncodeFn(torch.autograd.Function):
    """gathers -> concat -> input_linear -> LayerNorm -> tanh -> dropout -> attention -> code vector."""

    @staticmethod
    def forward(ctx, emb_t, emb_p, W, ln_g, ln_b, attn, starts, paths, ends, dims, drop_p, training, seed, algo, cache):
        params = CF.make_params(emb_t, emb_p, W, ln_g, ln_b, attn)
        # when a gradient will be asked for, keep x = c . W^T (105 MB per 1024 x 200 batch at encode_size 128) so that
        # the backward neither re-gathers the embedding rows nor redoes the input_linear GEMM
        stash = any(ctx.needs_input_grad[:6])
        res = CF.encode_forward(dims, params, starts, paths, ends, drop_p, training, seed, algo,
                                cache=cache, weight=W, stash=stash)
        cv, att = res[0], res[1]
        ctx.x_stash = res[2] if stash else None
        ctx.save_for_backward(emb_t, emb_p, W, ln_g, ln_b, attn, starts, paths, ends, cv, att)
        ctx.cfg = (dims, drop_p, training, seed)
        ctx.cache = cache
        return cv, att

    @staticmethod
    def backward(ctx, d_cv, d_att):
        emb_t, emb_p, W, ln_g, ln_b, attn, starts, paths, ends, cv, att = ctx.saved_tensors
        dims, drop_p, training, seed = ctx.cfg
        if ctx.cache is not None:
            ctx.cache.raise_deferred()               # bad indices in the forward this backward belongs to
        params = CF.make_params(emb_t, emb_p, W, ln_g, ln_b, attn)
        shapes = {"terminal_embedding": emb_t.shape, "path_embedding": emb_p.shape, "input_linear": W.shape,
                  "ln_weight": ln_g.shape, "ln_bias": ln_b.shape, "attention": attn.shape}
        if d_cv is None:
            d_cv = torch.zeros_like(cv)
        # Fused gradient accumulation (opt-in, Code2Vec.fuse_grad_accumulation; what ddp_step switches on for the flat
        # optimizers): the embedding-table and input_linear gradients -- 99.9 % of the bytes -- are scatter-added straight into
        # the existing dense .grad buffers instead of into fresh zero-filled tensors that autograd would then add to .grad
        # (at cfg2: a 360 MB fill plus a 1.1 GB read-modify-write per step).  Autograd gets None for those three inputs.
        big = (("terminal_embedding", emb_t), ("path_embedding", emb_p), ("input_linear", W))
        fuse = bool(getattr(ctx.cache, "fuse_grad_accumulation", False)) and all(
            t.grad is not None and t.grad.dtype == torch.float32 and t.grad.is_contiguous() and t.grad.shape == t.shape
            and t.grad.device == t.device for _, t in big)
        grads_out = None
        if fuse:
            grads_out = {k: t.grad for k, t in big}
            for k in ("ln_weight", "ln_bias", "attention"):
                grads_out[k] = torch.empty(shapes[k], dtype=torch.float32, device=cv.device)   # overwritten by the kernels
        hook = getattr(ctx.cache, "on_path_grads_ready", None) if fuse else None
        g = CF.encode_backward(dims, params, starts, paths, ends, cv, att, d_cv, d_att, shapes, drop_p, training, seed,
                               grads_out=grads_out, x_stash=ctx.x_stash, between_phases=hook)
        ctx.x_stash = None
        if fuse:
            return (None, None, None, g["ln_weight"], g["ln_bias"], g["attention"], None, None, None, None, None, None,
                    None, None, None)
        return (g["terminal_embedding"], g["path_embedding"], g["input_linear"], g["ln_weight"], g["ln_bias"],
                g["attention"], None, None, None, None, None, None, None, None, None)


class _LabelFn(torch.autograd.Function):
    """outputs = cv . W_out^T + b   (model.py:83)"""

    @staticmethod
    def forward(ctx, cv, w_out, b_out, dims, algo, cache):
        params = CF.make_params(None, None, None, None, None, None, w_out, b_out)
        if any(ctx.needs_input_grad[:3]):
            algo = int(algo) | CF.NO_PDL            # the calls that feed autograd use plain stream-ordered launches
        out = CF.label_logits(dims, params, cv, algo, cache=cache, weight=w_out)
        ctx.save_for_backward(cv, w_out)
        ctx.dims, ctx.cache, ctx.algo = dims, cache, int(algo) & 0xff
        return out

    @staticmethod
    def backward(ctx, d_out):
        cv, w_out = ctx.saved_tensors
        params = CF.make_params(None, None, None, None, None, None, w_out, None)
        d_cv, d_w, d_b = CF.label_backward(ctx.dims, params, cv, d_out, ctx.needs_input_grad[0],
                                           ctx.needs_input_grad[1], ctx.needs_input_grad[2], algo=ctx.algo, cache=ctx.cache,
                                           weight=w_out)
        return d_cv, d_w, d_b, None, None, None


class _AngularFn(torch.autograd.Function):
    """angular-margin head (model.py:71-80) with its hand-written backward (c2v_angular_backward)"""

    @staticmethod
    def forward(ctx, cv, w_out, label, dims, margin, inverse_temp):
        params = CF.make_params(None, None, None, None, None, None, w_out, None)
        out, cos, inv = CF.angular_forward_train(dims, params, cv, label, margin, inverse_temp)
        ctx.save_for_backward(cv, w_out, label, cos, inv)
        ctx.cfg = (dims, margin, inverse_temp)
        return out

    @staticmethod
    def backward(ctx, d_out):
        cv, w_out, label, cos, inv = ctx.saved_tensors
        dims, margin, inverse_temp = ctx.cfg
        params = CF.make_params(None, None, None, None, None, None, w_out, None)
        d_cv, d_w = CF.angular_backward(dims, params, cv, label, margin, inverse_temp, cos, inv, d_out,
                                        ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        return d_cv, d_w, None, None, None, None


class _LabelLossFn(torch.autograd.Function):
    """mean NLL of log_softmax(cv . W_out^T + b) (model.py:83 + main.py:251-264) without materialising the logits:
    the label GEMM's epilogue produces loss / logsumexp / arg-max; the backward recomputes the tile-wise softmax."""

    @staticmethod
    def forward(ctx, cv, w_out, b_out, label, dims, algo, cache):
        params = CF.make_params(None, None, None, None, None, None, w_out, b_out)
        if any(ctx.needs_input_grad[:3]):
            algo = int(algo) | CF.NO_PDL
        loss, lse, am, mx, _ = CF.label_loss(dims, params, cv, label, want_logits=False, algo=algo, cache=cache, weight=w_out)
        ctx.save_for_backward(cv, w_out, b_out, label, lse)
        ctx.dims, ctx.cache, ctx.algo = dims, cache, algo
        ctx.mark_non_differentiable(am, mx)
        return loss, am, mx

    @staticmethod
    def backward(ctx, d_loss, _d_am, _d_mx):
        cv, w_out, b_out, label, lse = ctx.saved_tensors
        params = CF.make_params(None, None, None, None, None, None, w_out, b_out)
        B = cv.shape[0]
        d_out = CF.label_dlogits(ctx.dims, params, cv, label, lse, 1.0 / B, scale_device=d_loss.reshape(1),
                                 algo=ctx.algo, cache=ctx.cache, weight=w_out)
        d_cv, d_w, d_b = CF.label_backward(ctx.dims, params, cv, d_out, ctx.needs_input_grad[0], ctx.needs_input_grad[1],
                                           ctx.needs_input_grad[2], algo=int(ctx.algo) & 0xff, cache=ctx.cache, weight=w_out,
                                           absmax_ready=True)
        return d_cv, d_w, d_b, None, None, None, None


class Code2Vec(nn.Module):
    """the code2vec model (B200-native drop-in for model.py:15-105)"""

    def __init__(self, option, algo="auto"):
        super(Code2Vec, self).__init__()
        self.option = option
        # same submodules, same order => same RNG consumption as model.py:21-42
        self.terminal_embedding = nn.Embedding(option.terminal_count, option.terminal_embed_size)
        self.path_embedding = nn.Embedding(option.path_count, option.path_embed_size)
        self.input_linear = nn.Linear(option.terminal_embed_size * 2 + option.path_embed_size, option.encode_size, bias=False)
        self.input_layer_norm = nn.LayerNorm(option.encode_size)

        if 0.0 < option.dropout_prob < 1.0:
            self.input_dropout = nn.Dropout(p=option.dropout_prob)   # holds p; the mask is made in-kernel
        else:
            self.input_dropout = None

        self.attention_parameter = Parameter(torch.nn.init.xavier_normal_(torch.zeros(option.encode_size, 1, dtype=torch.float32, requires_grad=True)).view(-1), requires_grad=True)

        if option.angular_margin_loss:
            self.output_linear = Parameter(torch.empty(option.label_count, option.encode_size, dtype=torch.float32))
            nn.init.xavier_uniform_(self.output_linear)
            self.cos_m = math.cos(option.angular_margin)
            self.sin_m = math.sin(option.angular_margin)
            self.th = math.cos(math.pi - option.angular_margin)
            self.mm = math.sin(math.pi - option.angular_margin) * option.angular_margin
        else:
            self.output_linear = nn.Linear(option.encode_size, option.label_count, bias=True)
            self.output_linear.bias.data.fill_(0.0)

        self.algo = {"auto": _lib.ALGO_AUTO, "ffma": _lib.ALGO_FFMA, "tcgen05": _lib.ALGO_TCGEN05}[algo]
        self._dropout_calls = 0
        # persistent workspaces: the hi/lo split images of input_linear / output_linear are rebuilt
        # only when the optimizer changed the weights (tracked by the tensors' version counters)
        self._enc_cache = CF.PrepCache(mirror_errors=True)
        # True: the backward adds the table / input_linear gradients directly into the parameters' existing .grad buffers
        # (see _EncodeFn.backward); needs dense fp32 .grad tensors to exist before the backward, e.g. a flat gradient bucket
        self.fuse_grad_accumulation = False
        # callable run by the backward once path_embedding's gradient is complete (fused accumulation only): the sharded
        # optimizer starts that table's data-parallel reduction there (ShardedFlatAdam.early_step)
        self.on_path_grads_ready = None
        self._lab_cache = CF.PrepCache()

    # -- helpers ---------------------------------------------------------------------------
    def _dims(self):
        o = self.option
        return CF.make_dims(o.terminal_count, o.path_count, o.label_count, o.terminal_embed_size,
                            o.path_embed_size, o.encode_size)

    def _next_seed(self):
        # one Philox key per training forward, drawn from torch's CPU generator so that
        # torch.manual_seed (main.py:120) makes runs repeatable
        self._dropout_calls += 1
        return int(torch.randint(0, 2 ** 62, (1,)).item())

    # -- the reference surface -------------------------------------------------------------
    def check_indices(self):
        """Synchronise and raise IndexError if any forward so far saw an index outside the embedding tables
        (`forward` itself raises it one call late, without synchronising: see functional.PrepCache.raise_deferred)."""
        self._enc_cache.raise_deferred(synchronize=True)

    def forward(self, starts, paths, ends, label):
        self._enc_cache.raise_deferred()
        self._enc_cache.fuse_grad_accumulation = self.fuse_grad_accumulation
        self._enc_cache.on_path_grads_ready = self.on_path_grads_ready
        option = self.option
        dims = self._dims()
        training = self.training and self.input_dropout is not None
        drop_p = float(option.dropout_prob) if training else 0.0
        seed = self._next_seed() if training else 0

        code_vector, attention = _EncodeFn.apply(
            self.terminal_embedding.weight, self.path_embedding.weight, self.input_linear.weight,
            self.input_layer_norm.weight, self.input_layer_norm.bias, self.attention_parameter,
            starts, paths, ends, dims, drop_p, training, seed, self.algo, self._enc_cache)

        if option.angular_margin_loss:
            if torch.is_grad_enabled() and (code_vector.requires_grad or self.output_linear.requires_grad):
                outputs = _AngularFn.apply(code_vector, self.output_linear, label, dims, option.angular_margin,
                                           option.inverse_temp)
            else:
                params = CF.make_params(None, None, None, None, None, None, self.output_linear, None)
                outputs = CF.angular_logits(dims, params, code_vector, label, option.angular_margin, option.inverse_temp)
        else:
            outputs = _LabelFn.apply(code_vector, self.output_linear.weight, self.output_linear.bias, dims,
                                     _lib.ALGO_FFMA if self.algo == _lib.ALGO_FFMA else _lib.ALGO_AUTO,
                                     self._lab_cache)

        return outputs, code_vector, attention

    # -- additive fast path (SURVEY.md 8f row 1): forward + calculate_loss (main.py:251-264) + torch.max (main.py:285) -----
    def forward_loss(self, starts, paths, ends, label):
        """-> (loss, pred_label [b], pred_score [b], code_vector [b,H], attention [b,L]); loss is the mean NLL the
        reference's `calculate_loss(preds, label, criterion, option)` returns (criterion weights are all 1, SURVEY 8a
        row 16) and is autograd-connected; the [b, C] logits are never written.  Plain label head only; shapes the fused
        kernel does not take fall back to forward() + c2v_loss_argmax."""
        if self.option.angular_margin_loss:
            raise NotImplementedError("forward_loss() needs the plain label head")
        self._enc_cache.raise_deferred()
        self._enc_cache.fuse_grad_accumulation = self.fuse_grad_accumulation
        self._enc_cache.on_path_grads_ready = self.on_path_grads_ready
        dims = self._dims()
        training = self.training and self.input_dropout is not None
        drop_p = float(self.option.dropout_prob) if training else 0.0
        seed = self._next_seed() if training else 0
        code_vector, attention = _EncodeFn.apply(
            self.terminal_embedding.weight, self.path_embedding.weight, self.input_linear.weight,
            self.input_layer_norm.weight, self.input_layer_norm.bias, self.attention_parameter,
            starts, paths, ends, dims, drop_p, training, seed, self.algo, self._enc_cache)
        if self.algo != _lib.ALGO_FFMA and CF.label_loss_supported(dims, starts.shape[0]):
            loss, am, mx = _LabelLossFn.apply(code_vector, self.output_linear.weight, self.output_linear.bias, label, dims,
                                              _lib.ALGO_AUTO, self._lab_cache)
        else:
            outputs = _LabelFn.apply(code_vector, self.output_linear.weight, self.output_linear.bias, dims,
                                     _lib.ALGO_FFMA if self.algo == _lib.ALGO_FFMA else _lib.ALGO_AUTO, self._lab_cache)
            loss = F.nll_loss(F.log_softmax(outputs, dim=1), label)
            mx, am = torch.max(outputs.detach(), dim=1)
        return loss, am, mx, code_vector, attention

    # -- additive convenience (the reference does torch.max(preds, dim=1) at main.py:285) ----
    @torch.no_grad()
    def predict(self, starts, paths, ends):
        """-> (pred_label [b], pred_score [b], code_vector [b,H], attention [b,L])"""
        if self.option.angular_margin_loss:
            raise NotImplementedError("predict() needs the plain label head (the angular head needs labels)")
        self._enc_cache.raise_deferred()
        dims = self._dims()
        params = CF.make_params(self.terminal_embedding.weight, self.path_embedding.weight, self.input_linear.weight,
                                self.input_layer_norm.weight, self.input_layer_norm.bias, self.attention_parameter,
                                self.output_linear.weight, self.output_linear.bias)
        code_vector, attention = CF.encode_forward(dims, params, starts, paths, ends, algo=self.algo,
                                                   cache=self._enc_cache, weight=self.input_linear.weight)
        _, am, mx = CF.label_logits_argmax(dims, params, code_vector,
                                           _lib.ALGO_FFMA if self.algo == _lib.ALGO_FFMA else _lib.ALGO_AUTO,
                                           cache=self._lab_cache, weight=self.output_linear.weight, want_logits=False)
        return am, mx, code_vector, attention
