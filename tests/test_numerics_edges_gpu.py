"""-m gpu: the kernels on ill-conditioned inputs, against high-precision references of the same operation.

Every other parity test feeds well-conditioned operands.  These cover the numerical edges the kernels meet in training:
 (a) LayerNorm rows whose |mean| / std is large.  The row mean of x = c . W^T comes from a component u shared by all
     rows of input_linear.weight.  LayerNorm removes it and the loss never sees it, so nothing keeps it small, and
     W + 1_H (x) u must give the outputs of W;
 (b) the gradients on such rows;
 (c) rows whose variance is below LayerNorm's eps;
 (d) operand magnitudes far from 1 for every fp16 hi/lo-split GEMM, all-zero operands, a power-of-two absmax;
 (e) attention scores of ~1e3 (a nearly one-hot softmax) and single-context bags.
Forward references: the C oracle (double accumulation, two-pass LayerNorm).  Gradients: fp64 torch on the CPU."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from gpu_util import ALGOS, cuda, model_from_golden, random_batch, random_params
from code2vec_b200 import _lib
from code2vec_b200 import functional as CF

pytestmark = pytest.mark.gpu

TOL = 1e-4          # the project's bar
EXPECT = 2e-5       # what the kernels deliver (regression guard)
KEYS = ["terminal_embedding.weight", "path_embedding.weight", "input_linear.weight", "input_layer_norm.weight",
        "input_layer_norm.bias", "attention_parameter", "output_linear.weight", "output_linear.bias"]
NAMES = {"terminal_embedding": "terminal_embedding.weight", "path_embedding": "path_embedding.weight",
         "input_linear": "input_linear.weight", "ln_weight": "input_layer_norm.weight",
         "ln_bias": "input_layer_norm.bias", "attention": "attention_parameter"}
RATIOS = [0, 3, 10, 30, 100]


def _ratio_bar(ratio, bar=EXPECT):
    """The bar at |mean| / std = ratio.  x = c . W^T itself is accumulated in fp32 (on the CUDA cores and on the tensor
    cores alike): its rounding error is relative to |x| ~ ratio * std, and LayerNorm divides by std.  Measured on a B200
    with the FFMA kernel: cv errors of 2e-5 at ratio 30 (encode_size 128) and 1.1e-4 to 2.1e-4 at ratio 100.  So the
    bar grows with the ratio beyond 5; a variance that cancels (E[x^2] - mean^2 in fp32) misses it at ratio 10 to 100."""
    return bar * max(1.0, ratio / 5.0)
SHAPES = [(128, 128), (100, 100), (256, 256)]      # narrow epilogue; padded columns (n_valid < HC); wide epilogue


def _dims_params(p, with_head=True):
    o = p["output_linear.weight"].shape[0]
    E, H = p["terminal_embedding.weight"].shape[1], p["input_linear.weight"].shape[0]
    dims = CF.make_dims(p["terminal_embedding.weight"].shape[0], p["path_embedding.weight"].shape[0], o, E, E, H)
    tp = {k: cuda(v) for k, v in p.items()}
    head = (tp["output_linear.weight"], tp["output_linear.bias"]) if with_head else ()
    params = CF.make_params(tp["terminal_embedding.weight"], tp["path_embedding.weight"], tp["input_linear.weight"],
                            tp["input_layer_norm.weight"], tp["input_layer_norm.bias"], tp["attention_parameter"], *head)
    return dims, params


def _shapes(p):
    return {k: p[v].shape for k, v in NAMES.items()}


def _contexts(p, starts, paths, ends):
    """c = [emb_t[start] | emb_p[path] | emb_t[end]] of the valid contexts, fp64 (model.py:48-51)"""
    v = starts > 0
    return np.concatenate([p["terminal_embedding.weight"][starts[v]], p["path_embedding.weight"][paths[v]],
                           p["terminal_embedding.weight"][ends[v]]], axis=1).astype(np.float64)


def _row_ratio(c, W):
    """median over context rows of |mean| / std of x = c . W^T, in fp64"""
    x = c @ W.astype(np.float64).T
    return float(np.median(np.abs(x.mean(1)) / x.std(1)))


def _with_common_mode(p, starts, paths, ends, ratio, rng):
    """-> (params with input_linear.weight = W + 1_H (x) u, params with W alone, the ratio reached).  u is scaled so
    that the median |mean| / std of the rows of x reaches `ratio`.  W and u are rounded to one power-of-two grid coarse
    enough that W + u is exact in fp32, so the two parameter sets give the same outputs in exact arithmetic."""
    c = _contexts(p, starts, paths, ends)
    W = p["input_linear.weight"].astype(np.float64)
    u0 = rng.standard_normal(W.shape[1]) / np.sqrt(W.shape[1])
    lo, hi = 0.0, 1.0
    while ratio and _row_ratio(c, W + hi * u0) < ratio:
        hi *= 2
    for _ in range(50 if ratio else 0):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if _row_ratio(c, W + mid * u0) < ratio else (lo, mid)
    u = hi * u0 if ratio else 0.0 * u0
    grid = 2.0 ** (np.ceil(np.log2(np.abs(W).max() + np.abs(u).max())) - 23)
    Wq, uq = np.round(W / grid) * grid, np.round(u / grid) * grid
    base = dict(p, **{"input_linear.weight": Wq.astype(np.float32)})
    shifted = dict(p, **{"input_linear.weight": (Wq + uq[None, :]).astype(np.float32)})
    assert np.array_equal(shifted["input_linear.weight"].astype(np.float64), Wq + uq[None, :])
    return shifted, base, _row_ratio(c, shifted["input_linear.weight"])


def _fp64_reference(p, starts, paths, ends, wa, wc, w_out_sq=0.1, dropmask=None):
    """fp64 evaluation of model.py:44-88 (LayerNorm written out) and the gradients of
    loss = sum(att * wa) + sum(cv * wc) + w_out_sq * sum(outputs^2) -> (grads, (outputs, cv, att))"""
    dt = torch.float64
    tp = {k: torch.from_numpy(v).to(dt).requires_grad_(True) for k, v in p.items()}
    s, pp, e = (torch.from_numpy(a) for a in (starts, paths, ends))
    H = p["input_linear.weight"].shape[0]
    c = torch.cat((F.embedding(s, tp["terminal_embedding.weight"]), F.embedding(pp, tp["path_embedding.weight"]),
                   F.embedding(e, tp["terminal_embedding.weight"])), 2)
    x = F.linear(c, tp["input_linear.weight"])
    xv = x.view(-1, H)
    mu = xv.mean(1, keepdim=True); var = xv.var(1, unbiased=False, keepdim=True)
    y = (xv - mu) / torch.sqrt(var + 1e-5) * tp["input_layer_norm.weight"] + tp["input_layer_norm.bias"]
    h = torch.tanh(y).view(x.shape)
    if dropmask is not None:
        h = h * torch.from_numpy(dropmask).to(dt)
    mask = (s > 0).to(dt)
    z = (h * tp["attention_parameter"]).sum(2) * mask + (1 - mask) * (-3.4e38)
    att = F.softmax(z, 1)
    cv = (h * att.unsqueeze(-1)).sum(1)
    out = F.linear(cv, tp["output_linear.weight"], tp["output_linear.bias"])
    loss = (att * torch.from_numpy(wa).to(dt)).sum() + (cv * torch.from_numpy(wc).to(dt)).sum()
    if w_out_sq:
        loss = loss + w_out_sq * out.square().sum()
    loss.backward()
    return ({k: (v.grad.numpy() if v.grad is not None else np.zeros_like(p[k], np.float64)) for k, v in tp.items()},
            (out.detach().numpy(), cv.detach().numpy(), att.detach().numpy()))


def _assert_grads_close(got, ref, keys, rel=2e-5):
    """every gradient within rel * max|ref| of the fp64 reference (NaN fails)"""
    bad = {}
    for k in keys:
        g, r = got[k], ref[k]
        err = float(np.nanmax(np.abs(g - r))) if not np.isnan(g).any() else float("nan")
        if not err <= rel * float(np.abs(r).max()):
            bad[k] = (err, rel * float(np.abs(r).max()))
    assert not bad, bad


def _case(rng, E, H, B=9, L=200, T=900, P=700, C=33):
    p = random_params(rng, T, P, C, E, E, H)
    starts, paths, ends, label = random_batch(rng, B, L, T, P, C)
    starts[1, :] = 0                                   # an all-pad bag
    starts[2, 1:] = 0                                  # a bag with one valid context
    return p, starts, paths, ends, label


def _forward_errors(p, starts, paths, ends, label, algo, dropmask=None, seed=0, prob=0.0):
    from oracle import oracle
    dims, params = _dims_params(p)
    cv, att = CF.encode_forward(dims, params, cuda(starts), cuda(paths), cuda(ends), drop_p=prob,
                                training=dropmask is not None, seed=seed, algo=ALGOS[algo])
    out = CF.label_logits(dims, params, cv, algo=ALGOS[algo])
    ref_out, ref_cv, ref_att = oracle.forward(p, starts, paths, ends, label, dropmask=dropmask)
    return (float(np.abs(cv.cpu().numpy() - ref_cv).max()), float(np.abs(att.cpu().numpy() - ref_att).max()),
            float(np.abs(out.cpu().numpy() - ref_out).max()), (cv, att))


# ---------------------------------------------------------------------------------------------------- (a) common mode
@pytest.mark.parametrize("ratio", RATIOS)
@pytest.mark.parametrize("E,H", SHAPES)
@pytest.mark.parametrize("algo", ["ffma", "tcgen05"])
def test_common_mode_rows_match_the_oracle(algo, E, H, ratio, record_property):
    """Rows of x with median |mean| / std = ratio, eval and training (the kernel's own dropout mask), ragged bags, an
    all-pad bag and a single-context bag: code vectors, attention and logits against the oracle."""
    from philox_ref import dropout_mask
    rng = np.random.default_rng(100 * E + ratio)
    p, starts, paths, ends, label = _case(rng, E, H)
    p, _, reached = _with_common_mode(p, starts, paths, ends, ratio, rng)
    assert (reached < 0.5) if ratio == 0 else (abs(reached - ratio) <= 0.02 * ratio), reached
    e_cv, e_att, e_out, _ = _forward_errors(p, starts, paths, ends, label, algo)
    seed, prob = 0x5EED + ratio, 0.25
    mask = dropout_mask(seed, starts.size, H, prob).reshape(*starts.shape, H)
    d_cv, d_att, d_out, _ = _forward_errors(p, starts, paths, ends, label, algo, dropmask=mask, seed=seed, prob=prob)
    record_property("errors", dict(eval=(e_cv, e_att, e_out), train=(d_cv, d_att, d_out)))
    assert max(e_cv, e_att, d_cv, d_att) <= _ratio_bar(ratio) and max(e_out, d_out) <= 4 * _ratio_bar(ratio), \
        dict(eval=(e_cv, e_att, e_out), train=(d_cv, d_att, d_out))


@pytest.mark.parametrize("E,H", SHAPES)
def test_tensor_core_outputs_do_not_depend_on_the_common_mode(E, H, record_property):
    """LayerNorm removes 1_H (x) u exactly: W and W + 1_H (x) u (both exact in fp32) give the same outputs, up to the
    fp32 contraction's rounding at ratio 100 (_ratio_bar)."""
    rng = np.random.default_rng(7 * E)
    p, starts, paths, ends, label = _case(rng, E, H)
    shifted, base, reached = _with_common_mode(p, starts, paths, ends, 100, rng)
    res = []
    for q in (base, shifted):
        dims, params = _dims_params(q, with_head=False)
        cv, att = CF.encode_forward(dims, params, cuda(starts), cuda(paths), cuda(ends), algo=_lib.ALGO_TCGEN05)
        res.append((cv.cpu().numpy(), att.cpu().numpy()))
    errs = [float(np.abs(a - b).max()) for a, b in zip(*res)]
    record_property("errors", errs)
    assert max(errs) <= _ratio_bar(100), errs


# ---------------------------------------------------------------------------------------------------- (b) gradients
@pytest.mark.parametrize("E,H", [(128, 128), (100, 100)])
@pytest.mark.parametrize("algo", ["auto", "ffma"])
def test_gradients_on_common_mode_rows_through_the_module(algo, E, H, record_property):
    rng = np.random.default_rng(31 * E)
    p, starts, paths, ends, label = _case(rng, E, H, B=7, L=90, T=300, P=200, C=11)
    p, _, reached = _with_common_mode(p, starts, paths, ends, 30, rng)
    assert abs(reached - 30) <= 0.6, reached
    B, L = starts.shape
    wa = rng.standard_normal((B, L)).astype(np.float32); wc = rng.standard_normal((B, H)).astype(np.float32)
    ref, (ref_out, ref_cv, ref_att) = _fp64_reference(p, starts, paths, ends, wa, wc)
    rec = {"opt": {"T": 300, "P": 200, "C": 11, "Et": E, "Ep": E, "H": H}, "params": p}
    m = model_from_golden(rec, algo=algo).train()
    out, cv, att = m.forward(cuda(starts), cuda(paths), cuda(ends), cuda(label))
    ((att * cuda(wa)).sum() + (cv * cuda(wc)).sum() + 0.1 * out.square().sum()).backward()
    assert np.abs(cv.detach().cpu().numpy() - ref_cv).max() <= _ratio_bar(30)
    assert np.abs(att.detach().cpu().numpy() - ref_att).max() <= _ratio_bar(30)
    got = {k: v.grad.cpu().numpy() for k, v in m.named_parameters()}
    record_property("errors", {k: float(np.abs(got[k] - ref[k]).max() / np.abs(ref[k]).max()) for k in KEYS})
    _assert_grads_close(got, ref, KEYS, rel=_ratio_bar(30))


@pytest.mark.parametrize("E,H", [(128, 128), (100, 100), (256, 256)])
@pytest.mark.parametrize("algo", ["ffma", "tcgen05"])
def test_encode_backward_on_common_mode_rows_with_and_without_the_stash(algo, E, H, record_property):
    rng = np.random.default_rng(37 * E)
    p, starts, paths, ends, label = _case(rng, E, H, B=7, L=90, T=300, P=200, C=11)
    p, _, reached = _with_common_mode(p, starts, paths, ends, 30, rng)
    B, L = starts.shape
    wa = rng.standard_normal((B, L)).astype(np.float32); wc = rng.standard_normal((B, H)).astype(np.float32)
    ref, _ = _fp64_reference(p, starts, paths, ends, wa, wc, w_out_sq=0.0)
    dims, params = _dims_params(p, with_head=False)
    s, pp, e = cuda(starts), cuda(paths), cuda(ends)
    cv, att, xs = CF.encode_forward(dims, params, s, pp, e, training=True, algo=ALGOS[algo], stash=True)
    errs = {}
    for name, stash in (("recompute", None), ("stash", xs)):
        g = CF.encode_backward(dims, params, s, pp, e, cv, att, cuda(wc), cuda(wa), _shapes(p), training=True,
                               x_stash=stash)
        got = {NAMES[k]: v.cpu().numpy() for k, v in g.items()}
        errs[name] = {k: float(np.abs(got[k] - ref[k]).max() / np.abs(ref[k]).max()) for k in got}
        _assert_grads_close(got, ref, list(got), rel=_ratio_bar(30))
    record_property("errors", errs)


# ---------------------------------------------------------------------------------------------------- (c) near-constant
@pytest.mark.parametrize("E,H", SHAPES)
@pytest.mark.parametrize("algo", ["ffma", "tcgen05"])
def test_rows_with_variance_below_eps_match_the_oracle(algo, E, H, record_property):
    """input_linear.weight = one row repeated plus noise of 1e-4: var(x) ~ 1e-6 < eps = 1e-5, so LayerNorm's output is
    decided by eps and by the small deviations of a row around a mean of order 1.  LayerNorm amplifies the fp32
    rounding of x by up to 1 / sqrt(eps) ~ 316 here: the FFMA kernel measured 8e-5 to 1.8e-4 on a B200, a cancelling
    variance 3e-4 to 1e-3."""
    rng = np.random.default_rng(11 * E + 1)
    p, starts, paths, ends, label = _case(rng, E, H)
    W = p["input_linear.weight"]
    p["input_linear.weight"] = (W[:1] + 1e-4 * rng.standard_normal(W.shape)).astype(np.float32)
    x = _contexts(p, starts, paths, ends) @ p["input_linear.weight"].astype(np.float64).T
    assert np.median(x.var(1)) < 1e-5 < np.median(np.abs(x.mean(1)))
    e_cv, e_att, e_out, _ = _forward_errors(p, starts, paths, ends, label, algo)
    record_property("errors", (e_cv, e_att, e_out))
    assert max(e_cv, e_att) <= 2.5 * TOL and e_out <= 4 * 2.5 * TOL, (e_cv, e_att, e_out)


# ---------------------------------------------------------------------------------------------------- (d) magnitudes
SCALES = [2.0 ** k for k in (-8, -4, 0, 4, 8)]


@pytest.mark.parametrize("emb_scale,w_scale", [(s, 1.0) for s in SCALES] + [(1.0, s) for s in SCALES if s != 1.0])
@pytest.mark.parametrize("E,H", [(128, 128), (256, 256)])
def test_encode_forward_over_operand_magnitudes(E, H, emb_scale, w_scale, record_property):
    """K1e splits both operands of c . W^T into fp16 hi + lo; W is scaled by a power of two first, the gathered
    embeddings are split as they are.  LayerNorm makes the result scale-free, so the bars do not move."""
    rng = np.random.default_rng(int(np.log2(emb_scale) + 8) * 17 + int(np.log2(w_scale) + 8) + E)
    p, starts, paths, ends, label = _case(rng, E, H)
    for k in ("terminal_embedding.weight", "path_embedding.weight"):
        p[k] = (p[k] * emb_scale).astype(np.float32)
    p["input_linear.weight"] = (p["input_linear.weight"] * w_scale).astype(np.float32)
    e_cv, e_att, e_out, _ = _forward_errors(p, starts, paths, ends, label, "tcgen05")
    record_property("errors", (e_cv, e_att, e_out))
    assert max(e_cv, e_att) <= EXPECT and e_out <= 4 * EXPECT, (e_cv, e_att, e_out)


@pytest.mark.parametrize("emb_scale", SCALES)
@pytest.mark.parametrize("E,H", [(128, 128), (256, 256)])
def test_tensor_core_weight_and_embedding_gradients_over_operand_magnitudes(E, H, emb_scale, record_property):
    """K3b (dW = dX^T . C: dX scaled, the gathered C split unscaled) and K3c (dC = dX . W) against fp64 and against the
    CUDA-core kernels, at embedding magnitudes 2^-8 .. 2^8.  Below ~2^-8 the lo half of C is subnormal in fp16 and
    dW's relative error grows as 2^-25 / std(C) (DESIGN.md)."""
    rng = np.random.default_rng(int(np.log2(emb_scale) + 8) + 40 + E)
    T, P, C, B, L = 3000, 2000, 16, 24, 200
    p = random_params(rng, T, P, C, E, E, H, scale=emb_scale)
    starts, paths, ends, label = random_batch(rng, B, L, T, P, C)
    starts[7, :] = 0
    wc = (1e-6 * rng.standard_normal((B, H))).astype(np.float32)
    ref, _ = _fp64_reference(p, starts, paths, ends, np.zeros((B, L), np.float32), wc, w_out_sq=0.0)
    dims, params = _dims_params(p, with_head=False)
    s, pp, e = cuda(starts), cuda(paths), cuda(ends)
    cv, att = CF.encode_forward(dims, params, s, pp, e)
    os.environ["C2V_BACKWARD"] = "ffma"
    try:
        g_ffma = CF.encode_backward(dims, params, s, pp, e, cv, att, cuda(wc), None, _shapes(p))
    finally:
        del os.environ["C2V_BACKWARD"]
    g_tc = CF.encode_backward(dims, params, s, pp, e, cv, att, cuda(wc), None, _shapes(p))
    got = {NAMES[k]: v.cpu().numpy() for k, v in g_tc.items()}
    record_property("errors", {k: float(np.abs(got[k] - ref[k]).max() / np.abs(ref[k]).max()) for k in got})
    _assert_grads_close(got, ref, list(got))
    for k in g_tc:
        b = g_ffma[k]
        assert torch.allclose(g_tc[k], b, rtol=0, atol=2e-5 * float(b.abs().max())), k


def _gemm_floor(a, b):
    """The absolute error floor of a 3-product fp16 hi/lo GEMM a . b^T whose unscaled operand is small: each element of
    that operand carries up to 2^-25 of absolute error (its lo half is subnormal).  Whichever operand the kernel leaves
    unscaled, the floor is at most 2^-25 times the largest row sum of |the other operand|."""
    return 2.0 ** -25 * (np.abs(a).sum(1).max() + np.abs(b).sum(1).max())


MAGS = [2.0 ** k for k in (-10, -5, 0, 5, 10)]


@pytest.mark.parametrize("w_scale,cv_scale", [(s, 1.0) for s in MAGS] + [(1.0, s) for s in MAGS if s != 1.0])
def test_label_gemms_over_operand_magnitudes(w_scale, cv_scale, record_property):
    """K2 (logits, fused loss, d logits) and LB1 (label backward: d cv = dout . W_out, dW_out = dout^T . cv) on the
    tensor cores against fp64, W_out and cv from 2^-10 to 2^10; the label backward with a freshly built and with a
    reused W_out image."""
    rng = np.random.default_rng(int(np.log2(w_scale) + 10) * 100 + int(np.log2(cv_scale) + 10))
    B, C, H = 130, 1000, 128
    cvn = (np.tanh(rng.standard_normal((B, H))) * cv_scale).astype(np.float32)
    w = (rng.standard_normal((C, H)) * 0.7 * w_scale).astype(np.float32)
    bias = (0.3 * rng.standard_normal(C) * w_scale * cv_scale).astype(np.float32)
    label = rng.integers(0, C, B).astype(np.int64)
    dims = CF.make_dims(10, 10, C, H, H, H)
    wt, bt = cuda(w), cuda(bias)
    params = CF.make_params(None, None, None, None, None, None, wt, bt)
    c64, w64 = cvn.astype(np.float64), w.astype(np.float64)
    ref = c64 @ w64.T + bias
    floor = _gemm_floor(c64, w64)
    errs = {}
    out = CF.label_logits(dims, params, cuda(cvn), algo=_lib.ALGO_TCGEN05).cpu().numpy()
    tol = 3e-6 * np.abs(ref).max() + floor                # on a logit; the loss and lse carry it along
    errs["logits"] = float(np.abs(out - ref).max())
    assert errs["logits"] <= tol, errs
    assert CF.label_loss_supported(dims, B)
    loss, lse, am, mx, out2 = CF.label_loss(dims, params, cuda(cvn), cuda(label), want_logits=True)
    m = ref.max(1, keepdims=True)
    ref_lse = (m + np.log(np.exp(ref - m).sum(1, keepdims=True)))[:, 0]
    ref_loss = float((ref_lse - ref[np.arange(B), label]).mean())
    errs["loss"] = abs(loss.item() - ref_loss)
    assert np.abs(out2.cpu().numpy() - ref).max() <= tol
    assert errs["loss"] <= 1e-5 * max(1.0, abs(ref_loss)) + 2 * tol, errs
    assert np.abs(lse.cpu().numpy() - ref_lse).max() <= 1e-6 * max(1.0, np.abs(ref_lse).max()) + tol
    dout = CF.label_dlogits(dims, params, cuda(cvn), cuda(label), lse, 1.0 / B)
    sm = np.exp(ref - ref_lse[:, None]); sm[np.arange(B), label] -= 1.0
    # d logits = (softmax - onehot) / B: a logit error delta moves softmax by at most ~delta
    errs["dlogits"] = float(np.abs(dout.cpu().numpy() - sm / B).max())
    assert errs["dlogits"] <= (1e-6 + 2 * tol) / B, errs
    d64 = dout.cpu().numpy().astype(np.float64)
    ref_dcv, ref_dw, ref_db = d64 @ w64, d64.T @ c64, d64.sum(0)
    cache = CF.PrepCache()
    for image in ("fresh", "reused"):
        d_cv, d_w, d_b = CF.label_backward(dims, params, cuda(cvn), dout, cache=cache, weight=wt)
        e = (float(np.abs(d_cv.cpu().numpy() - ref_dcv).max()), float(np.abs(d_w.cpu().numpy() - ref_dw).max()),
             float(np.abs(d_b.cpu().numpy() - ref_db).max()))
        errs[image] = e
        assert e[0] <= 2e-5 * np.abs(ref_dcv).max() + _gemm_floor(d64, w64.T), errs
        assert e[1] <= 2e-5 * np.abs(ref_dw).max() + _gemm_floor(d64.T, c64.T), errs
        assert e[2] <= 2e-5 * np.abs(ref_db).max() + 1e-6 * np.abs(d64).sum(0).max(), errs
    record_property("errors", errs)


def test_all_zero_output_weight():
    """absmax(W_out) = 0: no scale can be derived from it; the logits are the bias and the gradients are exact zeros."""
    rng = np.random.default_rng(3)
    B, C, H = 37, 77, 128
    cvn = np.tanh(rng.standard_normal((B, H))).astype(np.float32)
    w = np.zeros((C, H), np.float32); bias = (0.3 * rng.standard_normal(C)).astype(np.float32)
    label = rng.integers(0, C, B).astype(np.int64)
    dims = CF.make_dims(10, 10, C, H, H, H)
    wt = cuda(w)
    params = CF.make_params(None, None, None, None, None, None, wt, cuda(bias))
    for algo in (_lib.ALGO_TCGEN05, _lib.ALGO_FFMA):
        out = CF.label_logits(dims, params, cuda(cvn), algo=algo).cpu().numpy()
        assert np.array_equal(out, np.broadcast_to(bias, (B, C))), algo
    loss, lse, am, mx, _ = CF.label_loss(dims, params, cuda(cvn), cuda(label))
    ref = bias.astype(np.float64)
    ref_lse = ref.max() + np.log(np.exp(ref - ref.max()).sum())
    assert abs(loss.item() - float((ref_lse - ref[label]).mean())) <= 1e-5
    dout = CF.label_dlogits(dims, params, cuda(cvn), cuda(label), lse, 1.0 / B)
    d_cv, d_w, d_b = CF.label_backward(dims, params, cuda(cvn), dout, cache=CF.PrepCache(), weight=wt)
    assert float(d_cv.abs().max()) == 0.0
    d64 = dout.cpu().numpy().astype(np.float64)
    assert np.abs(d_w.cpu().numpy() - d64.T @ cvn.astype(np.float64)).max() <= 2e-5 * np.abs(d64.T @ cvn).max()


@pytest.mark.parametrize("algo", ["ffma", "tcgen05"])
def test_all_zero_code_vector_gradient(algo):
    """d_cv = 0 (max |dx| = 0: no scale for dX): every encode gradient is exactly zero, without NaN."""
    rng = np.random.default_rng(4)
    p, starts, paths, ends, label = _case(rng, 128, 128)
    B, L = starts.shape
    dims, params = _dims_params(p, with_head=False)
    s, pp, e = cuda(starts), cuda(paths), cuda(ends)
    cv, att = CF.encode_forward(dims, params, s, pp, e, algo=ALGOS[algo])
    zero = torch.zeros((B, 128), dtype=torch.float32, device="cuda:0")
    for d_att in (None, torch.zeros((B, L), dtype=torch.float32, device="cuda:0")):
        g = CF.encode_backward(dims, params, s, pp, e, cv, att, zero, d_att, _shapes(p))
        for k, v in g.items():
            assert float(v.abs().max()) == 0.0, k


@pytest.mark.parametrize("E,H", SHAPES)
def test_input_linear_absmax_exactly_a_power_of_two(E, H):
    """The W scale is a power of two found from max |W|; at max |W| = 2^k exactly the scaled maximum sits on the fp16
    range's binade edge."""
    rng = np.random.default_rng(5 * E)
    p, starts, paths, ends, label = _case(rng, E, H)
    W = p["input_linear.weight"]
    W[3, 5] = 0.5; W[H - 1, 0] = -0.5
    assert np.abs(W).max() == 0.5
    for algo in ("ffma", "tcgen05"):
        e_cv, e_att, e_out, _ = _forward_errors(p, starts, paths, ends, label, algo)
        assert max(e_cv, e_att) <= EXPECT and e_out <= 4 * EXPECT, (algo, e_cv, e_att, e_out)


# ---------------------------------------------------------------------------------------------------- (e) attention
@pytest.mark.parametrize("E,H", SHAPES)
@pytest.mark.parametrize("algo", ["ffma", "tcgen05"])
def test_nearly_one_hot_attention_matches_the_oracle(algo, E, H, record_property):
    """attention_parameter x 1e3: scores of order 1e3, so each bag's softmax is nearly one-hot; bag 2 has a single
    valid context (attention exactly 1 there).  A score error dz moves the attention by att (1 - att) dz, and scores
    of 1e3 turn an h error of 1e-7 into dz ~ 1e-4: the bar is TOL (measured on a B200: up to 2.2e-5 on the FFMA
    kernel, 4.4e-5 on the tensor cores, at encode_size 100)."""
    rng = np.random.default_rng(13 * E)
    p, starts, paths, ends, label = _case(rng, E, H)
    p["attention_parameter"] = (p["attention_parameter"] * 1e3).astype(np.float32)
    e_cv, e_att, e_out, (cv, att) = _forward_errors(p, starts, paths, ends, label, algo)
    record_property("errors", (e_cv, e_att, e_out))
    a = att.cpu().numpy()
    assert abs(a[2, 0] - 1.0) <= 1e-7 and (a[2, 1:] == 0).all()
    assert (a.max(1)[[0, 3, 4]] > 0.9).all()           # the softmax is as peaked as intended
    assert max(e_cv, e_att) <= TOL and e_out <= 4 * TOL, (e_cv, e_att, e_out)
