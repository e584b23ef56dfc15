"""Kernel-only timing of the fused encode kernel K1e (CUDA events through the c2v_profile hook) + parity vs FFMA.

    python scripts/time_encode.py
"""
import ctypes
import os
import sys

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, R)
import torch

from bench import WORKLOADS, synth_params, synth_pool
from code2vec_b200 import _lib, functional as CF

wl = os.environ.get("WORKLOAD", "cfg2")
w = dict(WORKLOADS[wl]); w["B"] = int(os.environ.get("BATCH", w["B"])); dev = torch.device("cuda:0")
nb = 64
p = synth_params(w, dev); s, pth, e, lab = synth_pool(w, nb, dev, 99)
B, L = w["B"], w["L"]
dims = CF.make_dims(w["T"], w["P"], w["C"], w["Et"], w["Ep"], w["H"])
params = CF.make_params(p["terminal_embedding.weight"], p["path_embedding.weight"], p["input_linear.weight"],
                        p["input_layer_norm.weight"], p["input_layer_norm.bias"], p["attention_parameter"])
lib = _lib.load()
print("lib:", _lib.LIB_PATH, flush=True)
peak = 6570.3
D = 2 * w["Et"] + w["Ep"]
alg_bytes = B * L * (24 + 4 * D) + B * (4 * w["H"] + 4 * L)
ref = CF.encode_forward(dims, params, s[:B], pth[:B], e[:B], algo=_lib.ALGO_FFMA)
cache = CF.PrepCache()
W = p["input_linear.weight"]
a = CF.encode_forward(dims, params, s[:B], pth[:B], e[:B], algo=_lib.ALGO_TCGEN05)
err = max((a[0] - ref[0]).abs().max().item(), (a[1] - ref[1]).abs().max().item())
for i in range(20):
    o = (i % nb) * B
    CF.encode_forward(dims, params, s[o:o + B], pth[o:o + B], e[o:o + B], algo=_lib.ALGO_TCGEN05, cache=cache, weight=W)
torch.cuda.synchronize()
lib.c2v_profile_enable(1)
n = 400
for i in range(n):
    o = (i % nb) * B
    CF.encode_forward(dims, params, s[o:o + B], pth[o:o + B], e[o:o + B], algo=_lib.ALGO_TCGEN05, cache=cache, weight=W)
torch.cuda.synchronize()
ms = ctypes.c_double(0); cnt = ctypes.c_int64(0)
lib.c2v_profile_read(ctypes.byref(ms), ctypes.byref(cnt))
lib.c2v_profile_enable(0)
us = ms.value / cnt.value * 1e3
print(f"{wl} encode_tm_kernel: {us:.2f} us/launch  {alg_bytes / us / 1e3:.0f} GB/s  frac={alg_bytes / us / 1e3 / peak:.3f}  max|err vs ffma|={err:.2e}", flush=True)
if os.environ.get("TIME_FFMA"):
    for i in range(3):
        CF.encode_forward(dims, params, s[:B], pth[:B], e[:B], algo=_lib.ALGO_FFMA, cache=cache, weight=p["input_linear.weight"])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(10):
        o = (i % nb) * B
        CF.encode_forward(dims, params, s[o:o + B], pth[o:o + B], e[o:o + B], algo=_lib.ALGO_FFMA)
    e1.record(); torch.cuda.synchronize()
    print(f"{wl} ffma (whole call): {e0.elapsed_time(e1) / 10 * 1e3:.1f} us", flush=True)
