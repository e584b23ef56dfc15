"""-m gpu parity tests of the CUDA path (through the C ABI) against
 (1) the committed outputs of the unmodified reference (tests/golden/), bar: 1e-4 fp32 abs
     (BASELINE.json north_star), observed ~1e-6;
 (2) the CPU oracle on fresh seeded inputs at sizes it finishes in seconds;
 (3) size-independent properties at BASELINE.json's full batch (1024 x 200)."""
import numpy as np
import pytest
import torch

from conftest import golden_names, load_golden
from gpu_util import ALGOS, algos_for, cuda, model_from_golden, random_batch, random_params, supports_tcgen05
from code2vec_b200 import _lib
from code2vec_b200 import functional as CF

pytestmark = pytest.mark.gpu

TOL = 1e-4          # the north_star's bar
EXPECT = 2e-5       # what the kernels actually deliver (tighter regression guard)

FWD_CASES = [(n, a) for n in golden_names() for a in ("ffma", "tcgen05")]


@pytest.mark.parametrize("name,algo", FWD_CASES)
def test_forward_matches_reference_golden(name, algo):
    rec = load_golden(name)
    m = model_from_golden(rec, algo=algo).eval()
    if algo == "tcgen05" and not supports_tcgen05(rec["opt"]):
        # the FFMA cases cover this shape; asking for the tensor-core kernel is refused, never silently served by another
        with pytest.raises(NotImplementedError, match="tcgen05"), torch.no_grad():
            m.forward(cuda(rec["starts"]), cuda(rec["paths"]), cuda(rec["ends"]), cuda(rec["label"]))
        return
    with torch.no_grad():
        out, cv, att = m.forward(cuda(rec["starts"]), cuda(rec["paths"]), cuda(rec["ends"]), cuda(rec["label"]))
    torch.cuda.synchronize()
    scale = max(1.0, float(np.abs(rec["outputs"]).max()))
    e_cv = np.abs(cv.cpu().numpy() - rec["code_vector"]).max()
    e_att = np.abs(att.cpu().numpy() - rec["attention"]).max()
    e_out = np.abs(out.cpu().numpy() - rec["outputs"]).max()
    assert e_cv <= EXPECT and e_att <= EXPECT and e_out <= EXPECT * scale * 4, (e_cv, e_att, e_out)
    assert e_cv <= TOL and e_att <= TOL
    # padded slots are exactly zero whenever the bag has a valid context (SURVEY.md 8a row 11)
    a = att.cpu().numpy()
    valid = rec["starts"] > 0
    has_valid = valid.any(1)
    assert (a[has_valid][~valid[has_valid]] == 0.0).all()
    assert np.allclose(a.sum(1), 1.0, atol=1e-5)


@pytest.mark.parametrize("algo", ["ffma", "tcgen05"])
@pytest.mark.parametrize("B,L", [(1, 1), (3, 200), (64, 200), (37, 50), (130, 31), (7, 333)])
def test_forward_matches_oracle_on_seeded_inputs(algo, B, L):
    from oracle import oracle
    rng = np.random.default_rng(1000 + B * 7 + L)
    T, P, C, E, H = 5000, 3000, 77, 128, 128
    p = random_params(rng, T, P, C, E, E, H)
    starts, paths, ends, label = random_batch(rng, B, L, T, P, C)
    if B > 2:
        starts[1, :] = 0                      # an all-pad bag
        starts[2, ::3] = 0                    # holes
    dims = CF.make_dims(T, P, C, E, E, H)
    tp = {k: cuda(v) for k, v in p.items()}
    params = CF.make_params(tp["terminal_embedding.weight"], tp["path_embedding.weight"], tp["input_linear.weight"],
                            tp["input_layer_norm.weight"], tp["input_layer_norm.bias"], tp["attention_parameter"],
                            tp["output_linear.weight"], tp["output_linear.bias"])
    cv, att = CF.encode_forward(dims, params, cuda(starts), cuda(paths), cuda(ends), algo=ALGOS[algo], check_indices=True)
    out = CF.label_logits(dims, params, cv, algo=_lib.ALGO_FFMA)
    ref_out, ref_cv, ref_att = oracle.forward(p, starts, paths, ends, label)
    assert np.abs(cv.cpu().numpy() - ref_cv).max() <= EXPECT
    assert np.abs(att.cpu().numpy() - ref_att).max() <= EXPECT
    assert np.abs(out.cpu().numpy() - ref_out).max() <= EXPECT * 4


@pytest.mark.parametrize("E,H", [(100, 100), (128, 100), (100, 128), (64, 128), (36, 100), (4, 100),
                                 (256, 256), (200, 256), (64, 256)])
@pytest.mark.parametrize("B,L", [(3, 200), (37, 50), (130, 31)])
def test_padded_shapes_on_the_tensor_core_path(E, H, B, L):
    """K1e pads every sub-vector to 128 k (zero-filled cp.async chunks) and the encode size to 128 columns
    (masked LayerNorm moments): the reference's default 100/100/100 (main.py:56-58) and other E % 4 == 0,
    H in {100, 128} shapes against the oracle, through the C ABI with algo = TCGEN05 (no fallback)."""
    from oracle import oracle
    rng = np.random.default_rng(E * 1000 + H * 10 + B)
    T, P, C = 5000, 3000, 77
    p = random_params(rng, T, P, C, E, E, H)
    starts, paths, ends, label = random_batch(rng, B, L, T, P, C)
    starts[1, :] = 0                          # an all-pad bag
    starts[2, ::3] = 0                        # holes
    dims = CF.make_dims(T, P, C, E, E, H)
    assert supports_tcgen05(dict(T=T, P=P, C=C, Et=E, Ep=E, H=H))
    tp = {k: cuda(v) for k, v in p.items()}
    params = CF.make_params(tp["terminal_embedding.weight"], tp["path_embedding.weight"], tp["input_linear.weight"],
                            tp["input_layer_norm.weight"], tp["input_layer_norm.bias"], tp["attention_parameter"],
                            tp["output_linear.weight"], tp["output_linear.bias"])
    cv, att = CF.encode_forward(dims, params, cuda(starts), cuda(paths), cuda(ends), algo=_lib.ALGO_TCGEN05, check_indices=True)
    out = CF.label_logits(dims, params, cv, algo=_lib.ALGO_TCGEN05)
    ref_out, ref_cv, ref_att = oracle.forward(p, starts, paths, ends, label)
    assert np.abs(cv.cpu().numpy() - ref_cv).max() <= EXPECT
    assert np.abs(att.cpu().numpy() - ref_att).max() <= EXPECT
    assert np.abs(out.cpu().numpy() - ref_out).max() <= EXPECT * 4
    cvf, attf = CF.encode_forward(dims, params, cuda(starts), cuda(paths), cuda(ends), algo=_lib.ALGO_FFMA)
    assert np.abs(cvf.cpu().numpy() - cv.cpu().numpy()).max() <= EXPECT


@pytest.mark.parametrize("algo", ["ffma", "tcgen05"])
def test_full_size_properties(algo):
    """BASELINE.json cfg2 batch (1024 x 200, E=H=128): too big for the scalar oracle, so check
    properties: rows of attention sum to 1, code vectors are convex combinations of tanh outputs
    (|cv| <= 1), the two algorithms agree, bags are independent of their batch neighbours, and a
    random sample of bags matches the oracle."""
    from oracle import oracle
    rng = np.random.default_rng(7)
    T, P, C, E, H, B, L = 50000, 40000, 512, 128, 128, 1024, 200
    p = random_params(rng, T, P, C, E, E, H)
    starts, paths, ends, label = random_batch(rng, B, L, T, P, C, ragged=False)
    dims = CF.make_dims(T, P, C, E, E, H)
    tp = {k: cuda(v) for k, v in p.items()}
    params = CF.make_params(tp["terminal_embedding.weight"], tp["path_embedding.weight"], tp["input_linear.weight"],
                            tp["input_layer_norm.weight"], tp["input_layer_norm.bias"], tp["attention_parameter"],
                            tp["output_linear.weight"], tp["output_linear.bias"])
    s, pp, e = cuda(starts), cuda(paths), cuda(ends)
    cv, att = CF.encode_forward(dims, params, s, pp, e, algo=ALGOS[algo], check_indices=True)
    a = att.cpu().numpy(); v = cv.cpu().numpy()
    assert np.allclose(a.sum(1), 1.0, atol=2e-5) and (a >= 0).all()
    assert np.abs(v).max() <= 1.0 + 1e-6
    sel = rng.choice(B, 12, replace=False)
    ref_cv, ref_att = oracle.encode_forward(starts[sel], paths[sel], ends[sel], p["terminal_embedding.weight"],
                                            p["path_embedding.weight"], p["input_linear.weight"],
                                            p["input_layer_norm.weight"], p["input_layer_norm.bias"],
                                            p["attention_parameter"])
    assert np.abs(v[sel] - ref_cv).max() <= EXPECT and np.abs(a[sel] - ref_att).max() <= EXPECT
    # independence: the same bags in a different batch position / batch size give the same rows
    perm = rng.permutation(B)[:300]
    cv2, att2 = CF.encode_forward(dims, params, s[perm].contiguous(), pp[perm].contiguous(), e[perm].contiguous(),
                                  algo=ALGOS[algo])
    assert np.abs(cv2.cpu().numpy() - v[perm]).max() <= 2e-6
    other = "ffma" if algo == "tcgen05" else "tcgen05"
    cv3, att3 = CF.encode_forward(dims, params, s, pp, e, algo=ALGOS[other])
    assert np.abs(cv3.cpu().numpy() - v).max() <= EXPECT and np.abs(att3.cpu().numpy() - a).max() <= EXPECT


def test_out_of_range_index_is_reported_like_the_reference():
    rec = load_golden("cfg2_small")
    m = model_from_golden(rec).eval()
    bad = rec["starts"].copy(); bad[0, 0] = rec["opt"]["T"]
    o = rec["opt"]
    dims = CF.make_dims(o["T"], o["P"], o["C"], o["Et"], o["Ep"], o["H"])
    params = CF.make_params(m.terminal_embedding.weight.data, m.path_embedding.weight.data, m.input_linear.weight.data,
                            m.input_layer_norm.weight.data, m.input_layer_norm.bias.data, m.attention_parameter.data)
    for algo in algos_for(o):
        with pytest.raises(IndexError):
            CF.encode_forward(dims, params, cuda(bad), cuda(rec["paths"]), cuda(rec["ends"]), algo=ALGOS[algo],
                              check_indices=True)


@pytest.mark.parametrize("E,H", [(128, 128), (100, 100), (256, 256)])
@pytest.mark.parametrize("algo", ["ffma", "tcgen05"])
def test_training_mode_dropout_matches_oracle_with_same_mask(algo, E, H):
    """model.py:60-61.  The kernel's mask is a pure function of (seed, row, col); the test rebuilds
    it in numpy (tests/philox_ref.py) and hands it to the oracle, so parity is exact."""
    from oracle import oracle
    from philox_ref import dropout_mask
    rng = np.random.default_rng(3)
    T, P, C, B, L = 900, 700, 33, 9, 200
    p = random_params(rng, T, P, C, E, E, H)
    starts, paths, ends, label = random_batch(rng, B, L, T, P, C)
    dims = CF.make_dims(T, P, C, E, E, H)
    tp = {k: cuda(v) for k, v in p.items()}
    params = CF.make_params(tp["terminal_embedding.weight"], tp["path_embedding.weight"], tp["input_linear.weight"],
                            tp["input_layer_norm.weight"], tp["input_layer_norm.bias"], tp["attention_parameter"])
    seed, prob = 0x1234567890ABCDEF, 0.25
    cv, att = CF.encode_forward(dims, params, cuda(starts), cuda(paths), cuda(ends), drop_p=prob, training=True,
                                seed=seed, algo=ALGOS[algo])
    mask = dropout_mask(seed, B * L, H, prob).reshape(B, L, H)
    assert abs((mask > 0).mean() - 0.75) < 0.01
    ref_cv, ref_att = oracle.encode_forward(starts, paths, ends, p["terminal_embedding.weight"],
                                            p["path_embedding.weight"], p["input_linear.weight"],
                                            p["input_layer_norm.weight"], p["input_layer_norm.bias"],
                                            p["attention_parameter"], dropmask=mask)
    assert np.abs(cv.cpu().numpy() - ref_cv).max() <= EXPECT
    assert np.abs(att.cpu().numpy() - ref_att).max() <= EXPECT
    # eval mode ignores p
    cv_e, _ = CF.encode_forward(dims, params, cuda(starts), cuda(paths), cuda(ends), drop_p=prob, training=False,
                                seed=seed, algo=ALGOS[algo])
    cv_0, _ = CF.encode_forward(dims, params, cuda(starts), cuda(paths), cuda(ends), algo=ALGOS[algo])
    assert torch.equal(cv_e, cv_0)


def test_loss_and_argmax_match_oracle():
    from oracle import oracle
    rec = load_golden("trained_scale")
    out = cuda(rec["outputs"]); label = cuda(rec["label"])
    loss, am, mx, dout = CF.loss_argmax(out, label, want_grad=True)
    ref_loss, ref_am, ref_mx = oracle.loss_argmax(rec["outputs"], rec["label"])
    assert abs(loss.item() - ref_loss) <= 1e-5 * max(1.0, abs(ref_loss))
    assert np.array_equal(am.cpu().numpy(), ref_am) and np.array_equal(mx.cpu().numpy(), ref_mx)
    t = torch.from_numpy(rec["outputs"]).double().requires_grad_(True)
    torch.nn.functional.nll_loss(torch.log_softmax(t, 1), torch.from_numpy(rec["label"])).backward()
    assert np.abs(dout.cpu().numpy() - t.grad.numpy()).max() <= 1e-6


def test_host_buffer_api_matches_device_api():
    """c2v_forward_host: the call a reference-side user with CPU tensors makes."""
    import ctypes
    rec = load_golden("cfg2_small")
    m = model_from_golden(rec).eval()
    o = rec["opt"]
    B, L = rec["starts"].shape
    dims = CF.make_dims(o["T"], o["P"], o["C"], o["Et"], o["Ep"], o["H"])
    params = CF.make_params(m.terminal_embedding.weight.data, m.path_embedding.weight.data, m.input_linear.weight.data,
                            m.input_layer_norm.weight.data, m.input_layer_norm.bias.data, m.attention_parameter.data,
                            m.output_linear.weight.data, m.output_linear.bias.data)
    lib = _lib.load()
    sess = ctypes.c_void_p()
    _lib.check(lib.c2v_session_create(0, ctypes.byref(dims), 16, L, ctypes.byref(sess)), "session_create")
    try:
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        hs, hp, he, hl = pin(rec["starts"]), pin(rec["paths"]), pin(rec["ends"]), pin(rec["label"])
        out = torch.empty((B, o["C"]), dtype=torch.float32).pin_memory()
        cv = torch.empty((B, o["H"]), dtype=torch.float32).pin_memory()
        att = torch.empty((B, L), dtype=torch.float32).pin_memory()
        pred = torch.empty((B,), dtype=torch.int64).pin_memory()
        score = torch.empty((B,), dtype=torch.float32).pin_memory()
        P = lambda t: ctypes.c_void_p(t.data_ptr())
        for _ in range(3):   # exercises both staging slots
            rc = lib.c2v_forward_host(sess, ctypes.byref(params), P(hs), P(hp), P(he), P(hl), B, P(out), P(cv), P(att),
                                      P(pred), P(score), _lib.ALGO_AUTO)
            _lib.check(rc, "c2v_forward_host")
        assert np.abs(cv.numpy() - rec["code_vector"]).max() <= EXPECT
        assert np.abs(att.numpy() - rec["attention"]).max() <= EXPECT
        assert np.abs(out.numpy() - rec["outputs"]).max() <= EXPECT * 4
        assert np.array_equal(pred.numpy(), rec["outputs"].argmax(1))
        bad = rec["starts"].copy(); bad[1, 2] = -5
        hb = pin(bad)
        rc = lib.c2v_forward_host(sess, ctypes.byref(params), P(hb), P(hp), P(he), P(hl), B, None, P(cv), P(att),
                                  None, None, _lib.ALGO_AUTO)
        assert rc == _lib.C2V_EINDEX
    finally:
        lib.c2v_session_destroy(sess)


@pytest.mark.parametrize("B,C,H", [(1, 5, 128), (37, 77, 128), (130, 1000, 128), (1024, 8192, 128), (64, 300, 64), (9, 50, 100),
                                   (200, 2279, 100), (33, 70, 36), (5, 40, 130), (130, 1000, 256), (40, 300, 200)])
def test_label_logits_tcgen05_vs_ffma_vs_oracle(B, C, H):
    """model.py:83 on the tensor cores (3-pass fp16 split) against the CUDA-core GEMM and the oracle,
    incl. ragged tile edges and weights at 'trained' scale."""
    from oracle import oracle
    rng = np.random.default_rng(B * 31 + C)
    cvn = np.tanh(rng.standard_normal((B, H))).astype(np.float32)
    w = (rng.standard_normal((C, H)) * 0.7).astype(np.float32)
    bias = (0.3 * rng.standard_normal(C)).astype(np.float32)
    dims = CF.make_dims(10, 10, C, H, H, H)
    params = CF.make_params(None, None, None, None, None, None, cuda(w), cuda(bias))
    ref = oracle.label_logits(cvn, w, bias)
    tol = 3e-6 * max(1.0, float(np.abs(ref).max()))      # fp32 relative: logits reach +-30 here
    out_f = CF.label_logits(dims, params, cuda(cvn), algo=_lib.ALGO_FFMA).cpu().numpy()
    assert np.abs(out_f - ref).max() <= tol
    if H % 4 == 0 and H <= 256:
        out_t = CF.label_logits(dims, params, cuda(cvn), algo=_lib.ALGO_TCGEN05).cpu().numpy()
        assert np.abs(out_t - ref).max() <= tol, np.abs(out_t - ref).max()
        out_a = CF.label_logits(dims, params, cuda(cvn), algo=_lib.ALGO_AUTO).cpu().numpy()
        assert np.array_equal(out_a, out_t)
    else:
        with pytest.raises(NotImplementedError):
            CF.label_logits(dims, params, cuda(cvn), algo=_lib.ALGO_TCGEN05)


@pytest.mark.parametrize("B,C", [(1, 5), (37, 77), (1024, 8192), (130, 1000), (300, 1001), (2100, 300), (1024, 19531)])
def test_fused_label_argmax_matches_torch_max(B, C):
    """main.py:285 folded into the label GEMM epilogue: same logits, first maximum wins, ties included."""
    rng = np.random.default_rng(B + C)
    H = 128
    cvn = np.tanh(rng.standard_normal((B, H))).astype(np.float32)
    w = (rng.standard_normal((C, H)) * 0.3).astype(np.float32)
    if C > 3:
        w[C - 1] = w[1]                    # duplicate class -> exact tie: the lower index must win
    bias = np.zeros(C, np.float32)
    dims = CF.make_dims(10, 10, C, H, H, H)
    params = CF.make_params(None, None, None, None, None, None, cuda(w), cuda(bias))
    out, am, mx = CF.label_logits_argmax(dims, params, cuda(cvn), algo=_lib.ALGO_AUTO)
    ref = CF.label_logits(dims, params, cuda(cvn), algo=_lib.ALGO_TCGEN05)
    assert torch.equal(out, ref)
    tv, ti = torch.max(out, dim=1)
    assert torch.equal(mx, tv) and torch.equal(am, ti)
    out2, am2, mx2 = CF.label_logits_argmax(dims, params, cuda(cvn), algo=_lib.ALGO_FFMA)
    tv2, ti2 = torch.max(out2, dim=1)
    assert torch.equal(mx2, tv2) and torch.equal(am2, ti2)


def test_predict_surface():
    rec = load_golden("cfg2_small")
    m = model_from_golden(rec).eval()
    am, mx, cv, att = m.predict(cuda(rec["starts"]), cuda(rec["paths"]), cuda(rec["ends"]))
    assert np.array_equal(am.cpu().numpy(), rec["outputs"].argmax(1))
    assert np.abs(cv.cpu().numpy() - rec["code_vector"]).max() <= EXPECT


@pytest.mark.parametrize("name,T,P,E,H", [("cfg5", 2_000_000, 500_000, 128, 128), ("cfg3", 360_633, 342_846, 100, 100)])
def test_baseline_vocab_sizes_sampled_against_the_oracle(name, T, P, E, H):
    """BASELINE.json configs[4] (2M terminals / 500K paths: 1.28 GB of tables, every gather misses L2) and configs[2]
    (top11 vocabulary sizes at the reference's default 100/100/100) at the full 1024 x 200 batch: a sample of bags against
    the oracle, all rows against the size-independent properties, and the 32-bit row-offset arithmetic at its largest."""
    from oracle import oracle
    g = torch.Generator(device="cuda:0").manual_seed(5)
    B, L, C = 1024, 200, 64
    emb_t = torch.randn(T, E, generator=g, device="cuda:0"); emb_p = torch.randn(P, E, generator=g, device="cuda:0")
    rng = np.random.default_rng(11)
    p = random_params(rng, 8, 8, C, E, E, H)
    starts = torch.randint(1, T, (B, L), generator=g, device="cuda:0"); paths = torch.randint(1, P, (B, L), generator=g, device="cuda:0")
    ends = torch.randint(1, T, (B, L), generator=g, device="cuda:0")
    starts[:, -1] = T - 1; paths[:, -1] = P - 1; ends[0, :] = T - 1           # the last rows of both tables
    starts[5, 100:] = 0                                                        # a padded suffix
    dims = CF.make_dims(T, P, C, E, E, H)
    assert supports_tcgen05(dict(T=T, P=P, C=C, Et=E, Ep=E, H=H))
    tp = {k: cuda(v) for k, v in p.items()}
    params = CF.make_params(emb_t, emb_p, tp["input_linear.weight"], tp["input_layer_norm.weight"],
                            tp["input_layer_norm.bias"], tp["attention_parameter"])
    cv, att = CF.encode_forward(dims, params, starts, paths, ends, algo=_lib.ALGO_TCGEN05, check_indices=True)
    a = att.cpu().numpy(); v = cv.cpu().numpy()
    assert np.allclose(a.sum(1), 1.0, atol=2e-5) and (a >= 0).all() and np.abs(v).max() <= 1.0 + 1e-6
    assert (a[5, 100:] == 0).all()
    sel = np.array([0, 5, 17, 511, 1023])
    sn, pn, en = starts[sel].cpu().numpy(), paths[sel].cpu().numpy(), ends[sel].cpu().numpy()
    # compact the sampled bags' rows so that the scalar oracle does not need the whole table on the host
    ut, it = np.unique(np.concatenate([sn.ravel(), en.ravel()]), return_inverse=True)
    up, ip = np.unique(pn.ravel(), return_inverse=True)
    et_small = emb_t[torch.from_numpy(ut).cuda()].cpu().numpy(); ep_small = emb_p[torch.from_numpy(up).cuda()].cpu().numpy()
    s2 = it[:sn.size].reshape(sn.shape).astype(np.int64); e2 = it[sn.size:].reshape(en.shape).astype(np.int64)
    p2 = ip.reshape(pn.shape).astype(np.int64)
    # index 0 means padding to the mask (model.py:64): keep real rows away from compact index 0
    et_small = np.concatenate([emb_t[:1].cpu().numpy(), et_small]); ep_small = np.concatenate([emb_p[:1].cpu().numpy(), ep_small])
    s2 = np.where(sn == 0, 0, s2 + 1); e2 = np.where(en == 0, 0, e2 + 1); p2 = np.where(pn == 0, 0, p2 + 1)
    ref_cv, ref_att = oracle.encode_forward(s2, p2, e2, et_small, ep_small, p["input_linear.weight"],
                                            p["input_layer_norm.weight"], p["input_layer_norm.bias"], p["attention_parameter"])
    assert np.abs(v[sel] - ref_cv).max() <= EXPECT and np.abs(a[sel] - ref_att).max() <= EXPECT


def test_fused_argmax_at_top11_label_count():
    """configs[2]'s label vocabulary (C = 195,299: odd, so output rows are only 4-byte aligned; 800 MB of logits at
    B = 1024): logits against the CUDA-core GEMM on a row sample, arg-max against torch.max on all rows."""
    B, C, H = 1024, 195_299, 100
    g = torch.Generator(device="cuda:0").manual_seed(9)
    cvt = torch.tanh(torch.randn(B, H, generator=g, device="cuda:0"))
    w = torch.randn(C, H, generator=g, device="cuda:0") * 0.2
    w[C - 1] = w[3]                                    # exact tie between class 3 and the last class
    bias = torch.randn(C, generator=g, device="cuda:0") * 0.05; bias[C - 1] = bias[3]
    dims = CF.make_dims(10, 10, C, H, H, H)
    params = CF.make_params(None, None, None, None, None, None, w, bias)
    out, am, mx = CF.label_logits_argmax(dims, params, cvt, algo=_lib.ALGO_AUTO)
    tv, ti = torch.max(out, dim=1)
    assert torch.equal(mx, tv) and torch.equal(am, ti)
    ref = cvt[:64].double() @ w.double().T + bias.double()
    assert (out[:64].double() - ref).abs().max().item() <= 3e-6 * max(1.0, ref.abs().max().item())


def test_wide_configuration_full_shard_properties():
    """BASELINE.json configs[3] per-GPU shard (512 x 200, embed = encode = 256) on the 256-wide tensor-core configuration
    (one TMEM accumulator, 4-pass chunked epilogue): size-independent properties on all rows, the CUDA-core kernel on
    all rows, the oracle on a sample of bags, and bit-identical relaunches."""
    from oracle import oracle
    rng = np.random.default_rng(21)
    T, P, C, E, H, B, L = 30000, 20000, 64, 256, 256, 512, 200
    p = random_params(rng, T, P, C, E, E, H)
    starts, paths, ends, label = random_batch(rng, B, L, T, P, C, ragged=True)
    starts[3, :] = 0
    dims = CF.make_dims(T, P, C, E, E, H)
    tp = {k: cuda(v) for k, v in p.items()}
    params = CF.make_params(tp["terminal_embedding.weight"], tp["path_embedding.weight"], tp["input_linear.weight"],
                            tp["input_layer_norm.weight"], tp["input_layer_norm.bias"], tp["attention_parameter"])
    s, pp, e = cuda(starts), cuda(paths), cuda(ends)
    cv, att = CF.encode_forward(dims, params, s, pp, e, algo=_lib.ALGO_TCGEN05, check_indices=True)
    cv2, att2 = CF.encode_forward(dims, params, s, pp, e, algo=_lib.ALGO_TCGEN05)
    assert torch.equal(cv, cv2) and torch.equal(att, att2)
    a = att.cpu().numpy(); v = cv.cpu().numpy()
    assert np.allclose(a.sum(1), 1.0, atol=2e-5) and (a >= 0).all() and np.abs(v).max() <= 1.0 + 1e-6
    assert np.allclose(a[3], 1.0 / L, atol=1e-7)                 # all-pad bag: uniform attention (model.py:93-96)
    cvf, attf = CF.encode_forward(dims, params, s, pp, e, algo=_lib.ALGO_FFMA)
    assert np.abs(cvf.cpu().numpy() - v).max() <= EXPECT and np.abs(attf.cpu().numpy() - a).max() <= EXPECT
    sel = rng.choice(B, 6, replace=False)
    ref_cv, ref_att = oracle.encode_forward(starts[sel], paths[sel], ends[sel], p["terminal_embedding.weight"],
                                            p["path_embedding.weight"], p["input_linear.weight"],
                                            p["input_layer_norm.weight"], p["input_layer_norm.bias"], p["attention_parameter"])
    assert np.abs(v[sel] - ref_cv).max() <= EXPECT and np.abs(a[sel] - ref_att).max() <= EXPECT


def test_weight_image_reuse_survives_a_smaller_last_batch():
    """An evaluation pass ends with a ragged batch (main.py:162, drop_last unset): the cached W_out image (REUSE_PREP)
    must be found again when B shrinks -- its workspace offset may not depend on the batch size."""
    rng = np.random.default_rng(77)
    C, H = 700, 128
    w = cuda((rng.standard_normal((C, H)) * 0.3).astype(np.float32)); bias = cuda((0.1 * rng.standard_normal(C)).astype(np.float32))
    dims = CF.make_dims(10, 10, C, H, H, H)
    params = CF.make_params(None, None, None, None, None, None, w, bias)
    cache = CF.PrepCache()
    for B in (300, 7, 129, 1):
        cvt = cuda(np.tanh(rng.standard_normal((B, H))).astype(np.float32))
        out, am, mx = CF.label_logits_argmax(dims, params, cvt, cache=cache, weight=w)
        ref = CF.label_logits(dims, params, cvt)                       # fresh workspace, images rebuilt
        assert torch.equal(out, ref)
        tv, ti = torch.max(ref, dim=1)
        assert torch.equal(mx, tv) and torch.equal(am, ti)
