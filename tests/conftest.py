import glob
import hashlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run by the driver with -m gpu)")


def golden_names(prefix=None, exclude_prefix=("init_", "builder_", "reader_", "writer")):
    names = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))
    names = [n for n in names if not n.startswith(tuple(exclude_prefix))]
    if prefix is not None:
        names = [n for n in names if n.startswith(prefix)]
    return names


def params_sha256(params):
    """Digest of a state dict's arrays (fp32 bytes, in order): pins the parameters a golden file stores by seed."""
    h = hashlib.sha256()
    for k, v in params.items():
        h.update(k.encode())
        h.update(np.ascontiguousarray(v, dtype=np.float32).tobytes())
    return h.hexdigest()


def reference_init_params(opt, seed):
    """The reference's initial weights of a plain-head model under torch.manual_seed(seed): its modules in its order
    (model.py:21-42), output bias zero-filled.  Golden files whose parameters are too large to store keep only the seed."""
    import torch
    import torch.nn as nn
    torch.manual_seed(seed)
    te = nn.Embedding(opt["T"], opt["Et"])
    pe = nn.Embedding(opt["P"], opt["Ep"])
    lin = nn.Linear(2 * opt["Et"] + opt["Ep"], opt["H"], bias=False)
    ln = nn.LayerNorm(opt["H"])
    att = nn.init.xavier_normal_(torch.zeros(opt["H"], 1)).view(-1)
    out = nn.Linear(opt["H"], opt["C"], bias=True)
    out.bias.data.fill_(0.0)
    p = {"attention_parameter": att, "terminal_embedding.weight": te.weight, "path_embedding.weight": pe.weight,
         "input_linear.weight": lin.weight, "input_layer_norm.weight": ln.weight, "input_layer_norm.bias": ln.bias,
         "output_linear.weight": out.weight, "output_linear.bias": out.bias}
    return {k: v.detach().numpy().copy() for k, v in p.items()}


def load_golden(name):
    """-> dict(opt=..., params={state_dict key: array}, grads={...}, inputs..., outputs...)"""
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    rec = {"opt": {}, "params": {}, "grads": {}}
    for k in z.files:
        if k.startswith("opt_"):
            rec["opt"][k[4:]] = z[k].item()
        elif k.startswith("param."):
            rec["params"][k[6:]] = z[k]
        elif k.startswith("grad."):
            rec["grads"][k[5:]] = z[k]
        elif k not in ("param_seed", "param_sha256"):
            rec[k] = z[k]
    if "param_seed" in z.files:
        rec["params"] = reference_init_params(rec["opt"], int(z["param_seed"]))
        assert params_sha256(rec["params"]) == str(z["param_sha256"]), \
            f"{name}: torch.manual_seed({int(z['param_seed'])}) no longer yields the reference's initial weights"
    return rec


@pytest.fixture(scope="session")
def golden_loader():
    return load_golden


@pytest.fixture(scope="session", autouse=True)
def _warm_up_aten_cpu_reference():
    """The torch-CPU restatement (oracle.torch_forward) is the reference of several tests.  On the many-core GPU-box host
    the first fp32 evaluation of its LayerNorm + autograd in a fresh process was found to be occasionally off by ~1e-4
    relative (profiles/r2_flake_root_cause.txt); every later evaluation in the same process is right.  Run it once, on
    sizes that exercise the parallel paths, before any test uses it as a reference."""
    import torch
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(0)
    for _ in range(2):
        x = torch.randn(640, 128, generator=g, requires_grad=True)
        w = torch.randn(128, generator=g, requires_grad=True)
        b = torch.randn(128, generator=g, requires_grad=True)
        emb = torch.randn(300, 128, generator=g, requires_grad=True)
        idx = torch.randint(0, 300, (640,), generator=g)
        y = torch.tanh(F.layer_norm(F.linear(F.embedding(idx, emb) + x, torch.eye(128)), (128,), w, b, 1e-5))
        (y.sum() + F.softmax(y, 1).square().sum()).backward()
    yield
