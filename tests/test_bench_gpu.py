"""-m gpu: bench.py's own arm on the tiny workload.  --steps sets the number of timed steps (the timed region holds
exactly K steps' launches), and --dump-outputs writes what the last timed step computed: checked against the C oracle
on the batch that step used."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu

POOL = 5            # shares no factor with the step counts below: a timed region of several K-step passes would end on
                    # another batch than W+K-1 unless the pass count were a multiple of 5, for all three (K, W) at once
REUSE = 0x100       # C2V_FLAG_REUSE_PREP, as bench.py's timed steps pass it


def _bench(steps, warmup, out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", str(steps),
                        "--warmup", str(warmup), "--pool-batches", str(POOL), "--no-cpu-baseline", "--no-e2e",
                        "--no-gpu-eager", "--train-steps", "0", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = r.stdout.splitlines()
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def _launches_per_step(w, p, s, pth, e):
    """kernel launches of one bench step (encode + label logits / arg-max) once the weight images exist"""
    from code2vec_b200 import _lib
    from code2vec_b200 import functional as CF
    lib = _lib.load()
    B, L, H, C = w["B"], w["L"], w["H"], w["C"]
    dev = s.device
    dims = CF.make_dims(w["T"], w["P"], C, w["Et"], w["Ep"], H)
    params = CF.make_params(p["terminal_embedding.weight"], p["path_embedding.weight"], p["input_linear.weight"],
                            p["input_layer_norm.weight"], p["input_layer_norm.bias"], p["attention_parameter"],
                            p["output_linear.weight"], p["output_linear.bias"])
    cv, att = torch.empty((B, H), device=dev), torch.empty((B, L), device=dev)
    out, am, mx = torch.empty((B, C), device=dev), torch.empty((B,), dtype=torch.int64, device=dev), torch.empty((B,), device=dev)
    ws_n = lib.c2v_encode_workspace_bytes(ctypes.byref(dims), B, L); ws = torch.empty((ws_n,), dtype=torch.uint8, device=dev)
    wl_n = lib.c2v_label_workspace_bytes(ctypes.byref(dims), B); wl = torch.empty((wl_n,), dtype=torch.uint8, device=dev)
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def step(reuse):
        _lib.check(lib.c2v_encode_forward(ctypes.byref(dims), ctypes.byref(params), P(s[:B]), P(pth[:B]), P(e[:B]), B, L,
                                          None, P(cv), P(att), P(ws), ws_n, _lib.ALGO_AUTO | reuse, st), "encode")
        _lib.check(lib.c2v_label_logits_argmax(ctypes.byref(dims), ctypes.byref(params), P(cv), B, P(out), P(am), P(mx),
                                               P(wl), wl_n, _lib.ALGO_AUTO | reuse, st), "label+argmax")
    step(0)                                   # builds the weight images, as bench.py's first step does
    l0 = lib.c2v_launch_count()
    step(REUSE)
    n = lib.c2v_launch_count() - l0
    torch.cuda.synchronize()
    return n


def test_steps_set_the_timed_region_and_the_dump_is_its_last_step(tmp_path):
    import bench
    from oracle import oracle
    w = dict(bench.WORKLOADS["tiny"])
    dev = torch.device("cuda", 0)
    tp = bench.synth_params(w, dev)
    ts, tpth, te, tlab = bench.synth_pool(w, POOL, dev, 1234)
    per_step = _launches_per_step(w, tp, ts, tpth, te)
    assert per_step > 0
    p = {k: v.cpu().numpy() for k, v in tp.items()}
    s, pth, e, lab = (t.cpu().numpy() for t in (ts, tpth, te, tlab))
    B = w["B"]
    for k, warmup in ((2, 1), (3, 2), (4, 0)):
        out_dir = tmp_path / f"k{k}"
        d = _bench(k, warmup, out_dir)
        assert d["steps"] == k and d["warmup"] == warmup and d["parity"]["ok"]
        assert d["gpu_launches"] == k * per_step, (d["gpu_launches"], k, per_step)
        o = ((warmup + k - 1) % POOL) * B          # the timed pass runs batches W .. W+K-1 of the pool
        got = {n: np.load(out_dir / f"{n}.npy") for n in ("outputs", "code_vector", "attention", "predicted_label",
                                                             "predicted_score")}
        assert all(a.dtype in (np.float32, np.float64) for a in got.values())
        ro, rc, ra = oracle.forward(p, s[o:o + B], pth[o:o + B], e[o:o + B], lab[o:o + B])
        for n, ref in (("outputs", ro), ("code_vector", rc), ("attention", ra)):
            assert got[n].shape == ref.shape and float(np.abs(got[n] - ref).max()) <= 1e-4, n
        assert np.array_equal(got["predicted_label"], got["outputs"].argmax(1).astype(np.float64))
        assert np.array_equal(got["predicted_score"], got["outputs"].max(1))
