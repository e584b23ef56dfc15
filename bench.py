#!/usr/bin/env python
"""bench.py -- path-contexts/sec of the code2vec path-attention forward on B200.

Metric (BASELINE.json): path-contexts/sec = batch x bag x steps / seconds, every slot valid,
plus the fused-kernel HBM GB/s against the measured roofline.

A "step" is one Code2Vec.forward (fused gather+encode+attention kernel, per-bag finalize,
label logits, argmax) over one batch of 1024 synthetic bags of 200 contexts.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]    # our arm
    python bench.py --impl reference [...]                          # the reference's CPU path
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Our arm prints ONE JSON line with `value` (inputs resident in HBM), `e2e` (host buffers through
the C-ABI c2v_forward_host, H2D/D2H inside the timed region), `roofline` (dominant kernel timed
with CUDA events on its stream), `cpu_baseline` (the oracle's torch-CPU restatement on a bounded
sample, rank 0, N=1 only), `clocks`, `gpu_launches`.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on (single GPU)
    "cfg2": dict(T=360633, P=342846, C=8192, Et=128, Ep=128, H=128, B=1024, L=200,
                 desc="synthetic methods x 200 contexts, embed=128/128, encode=128, batch=1024 "
                      "(top11-sized vocab: T=360,633 P=342,846; C=8,192)"),
    # configs[4]: large-vocab stress (gather-bound)
    "cfg5": dict(T=2000000, P=500000, C=8192, Et=128, Ep=128, H=128, B=1024, L=200,
                 desc="large-vocab stress: 2M terminals / 500K paths, embed=128, encode=128, batch=1024"),
    # configs[2]: top11 corpus sizes (the reference's default embed/encode 100), synthetic uniform indices
    "cfg3": dict(T=360633, P=342846, C=195299, Et=100, Ep=100, H=100, B=1024, L=200,
                 desc="top11_dataset sizes: T=360,633 P=342,846 C=195,299, embed=100/100, encode=100, batch=1024 "
                      "(synthetic uniform indices; the corpus itself is not shipped)"),
    # configs[3]: embed=encode=256, global batch 4096 over 8 GPUs = 512 per rank (the per-rank shard is what one GPU runs)
    "cfg4": dict(T=360633, P=342846, C=8192, Et=256, Ep=256, H=256, B=512, L=200,
                 desc="synthetic methods x 200 contexts, embed=256/256, encode=256, batch=512 per GPU (4096 over 8), "
                      "top11-sized vocab, C=8,192"),
    # small variant for quick functional runs
    "tiny": dict(T=5000, P=4000, C=256, Et=128, Ep=128, H=128, B=64, L=200, desc="tiny functional run"),
}


def bytes_per_ctx(w):
    """SURVEY.md 8(d): 3 int64 indices + three fp32 rows per context, + per-bag outputs."""
    D = 2 * w["Et"] + w["Ep"]
    return 24 + 4 * D + (4 * w["H"] + 4 * w["L"]) / w["L"]


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            j = json.load(open(path))
            return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region: started before the warm-up so the
    process is already looping when the region begins; only samples whose timestamp falls inside
    [mark_begin, mark_end] count (if the region is shorter than the sampling interval, the nearest sample is
    reported and flagged)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t0, self.t1 = index, [], None, None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        parsed = []
        for ts, r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                parsed.append((ts, float(f[1]), float(f[2]), [n for n, v in zip(names, f[4:8]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        if not parsed:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        t0, t1 = self.t0 or 0.0, self.t1 or 1e18
        # a row is printed when its query completes; the query itself took a few ms, hence the small slack
        inside = [p for p in parsed if t0 <= p[0] <= t1 + 0.03]
        note = None
        if not inside:
            mid = 0.5 * (t0 + min(t1, time.time()))
            inside = [min(parsed, key=lambda p: abs(p[0] - mid))]
            note = "timed region shorter than the sampling interval: nearest sample"
        sm = sorted(p[1] for p in inside)
        out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(p[2] for p in inside),
               "reasons": sorted({r for p in inside for r in p[3]}), "samples": len(inside)}
        if note:
            out["note"] = note
        return out


def synth_params(w, device, seed=1):
    """Random-init weights of the reference architecture (model.py:18-42 init distributions)."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    D = 2 * w["Et"] + w["Ep"]
    r = lambda *s: torch.randn(*s, generator=g, device=device, dtype=torch.float32)
    u = lambda bound, *s: (torch.rand(*s, generator=g, device=device, dtype=torch.float32) * 2 - 1) * bound
    return {
        "terminal_embedding.weight": r(w["T"], w["Et"]), "path_embedding.weight": r(w["P"], w["Ep"]),
        "input_linear.weight": u(D ** -0.5, w["H"], D),
        "input_layer_norm.weight": torch.ones(w["H"], device=device), "input_layer_norm.bias": torch.zeros(w["H"], device=device),
        "attention_parameter": r(w["H"]) * (2.0 / (w["H"] + 1)) ** 0.5,
        "output_linear.weight": u(w["H"] ** -0.5, w["C"], w["H"]), "output_linear.bias": torch.zeros(w["C"], device=device),
    }


def synth_pool(w, n_batches, device, seed):
    """Device-resident index pool: every slot valid (SURVEY.md 8d), uniform over the vocab."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    n = n_batches * w["B"]
    mk = lambda hi: torch.randint(1, hi, (n, w["L"]), generator=g, device=device, dtype=torch.int64)
    return mk(w["T"]), mk(w["P"]), mk(w["T"]), torch.randint(0, w["C"], (n,), generator=g, device=device, dtype=torch.int64)


def bench_config(w, args):
    """the `config` object of the JSON line -- ONE function for both arms, so the driver's same_config check holds"""
    nb = args.pool_batches
    return {"workload": w["name"], "detail": w["desc"], "batch_per_gpu": w["B"], "bag": w["L"],
            "step": "Code2Vec.forward: encode + finalize + label logits + argmax",
            "sharding": "methods sharded by rank, parameters replicated, no collective in forward",
            "l2": f"inputs larger than L2: {(w['T'] * w['Et'] + w['P'] * w['Ep']) * 4 / 1e6:.0f} MB of tables, "
                  f"{nb} distinct batches ({nb * w['B'] * w['L'] * 24 / 1e6:.0f} MB of indices) cycled"}


DUMP_BYTES = 64 << 20         # at most this much is written by --dump-outputs


def dump_outputs(d, tensors):
    """--dump-outputs: every result of the timed path's last step as <d>/<name>.npy, floating point as float32 and integers
    as float64 (exact below 2**53).  If together they exceed DUMP_BYTES, the largest keeps a fixed, seeded sample of its
    rows, whose indices go to <d>/<name>_rows.npy: two builds run with the same arguments write the same entries."""
    import numpy as np
    arrays = {k: t.detach().cpu().numpy() for k, t in tensors.items()}
    arrays = {k: a.astype(np.float32 if a.dtype.kind == "f" else np.float64) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        big = max(arrays, key=lambda k: arrays[k].nbytes)
        a = arrays[big]
        row_bytes = a.nbytes // a.shape[0] + 8
        n = max(1, (DUMP_BYTES - (total - a.nbytes)) // row_bytes)
        rows = np.sort(np.random.default_rng(0).choice(a.shape[0], size=n, replace=False))
        arrays[big] = a[rows]
        arrays[big + "_rows"] = rows.astype(np.float64)
    os.makedirs(d, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(d, k + ".npy"), a)


def find_reference_module():
    """The UNMODIFIED reference `model.model.Code2Vec` if it can be imported on this box: baseline/_ref first, then
    /root/reference (BASELINE.md section 3.1).  The reference has neither setup.py nor pyproject.toml, so the offline pip
    install into baseline/_ref fails ("not installable", DESIGN.md) and the GPU box has neither path: -> None there."""
    for root in (os.path.join(ROOT, "baseline", "_ref"), os.environ.get("C2V_REFERENCE", "/root/reference")):
        if os.path.exists(os.path.join(root, "model", "model.py")):
            try:
                sys.dont_write_bytecode = True
                sys.path.insert(0, root)
                from model.model import Code2Vec as RefCode2Vec          # noqa: the reference, unmodified
                return RefCode2Vec, root
            except Exception:
                sys.path.remove(root)
    return None, None


def run_reference(args, w):
    """The reference's own CPU implementation of the path, timed on this box's host cores: the unmodified
    /root/reference/model/model.py when this box has it (kind "reference"), else oracle.torch_forward, the same ATen CPU
    ops in the same order, pinned to the reference by tests/test_oracle_golden.py (kind "port")."""
    import types
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    dev = torch.device("cpu")
    p = synth_params(w, dev)
    s, pth, e, lab = synth_pool(w, 2, dev, 1234)
    B, L = w["B"], w["L"]
    RefCode2Vec, ref_root = find_reference_module()
    if RefCode2Vec is not None:
        o = types.SimpleNamespace(terminal_count=w["T"], path_count=w["P"], label_count=w["C"], terminal_embed_size=w["Et"],
                                  path_embed_size=w["Ep"], encode_size=w["H"], dropout_prob=0.25, angular_margin_loss=False,
                                  angular_margin=0.5, inverse_temp=30.0, device=dev)
        ref = RefCode2Vec(o)
        ref.load_state_dict(p)
        ref.eval()
        fwd = lambda a, b, c, d: ref.forward(a, b, c, d)
        kind, how = "reference", f"unmodified {ref_root}/model/model.py Code2Vec.forward (eval, no_grad)"
    else:
        from oracle import oracle
        fwd = lambda a, b, c, d: oracle.torch_forward(p, a, b, c, d)
        kind, how = "port", "torch-CPU restatement (oracle.torch_forward; the reference is not installable and absent on this box)"
    # all the host threads it can use: the fastest of {all, 1/2, 1/4, 16} threads, each judged by the best of 3 passes
    best_nt, best_t = cores, None
    for nt in sorted({cores, max(1, cores // 2), max(1, cores // 4), min(cores, 16)}, reverse=True):
        torch.set_num_threads(nt)
        with torch.no_grad():
            fwd(s[:B], pth[:B], e[:B], lab[:B])
            dtp = None
            for _ in range(3):
                t0 = time.perf_counter()
                fwd(s[:B], pth[:B], e[:B], lab[:B])
                d1 = time.perf_counter() - t0
                dtp = d1 if dtp is None else min(dtp, d1)
        if best_t is None or dtp < best_t * 0.97:             # prefer more threads unless clearly slower
            best_nt, best_t = nt, dtp
    torch.set_num_threads(best_nt)
    cores_used = best_nt

    def step(i):
        o = (i % 2) * B
        with torch.no_grad():
            out, cv, att = fwd(s[o:o + B], pth[o:o + B], e[o:o + B], lab[o:o + B])
            return out.max(dim=1)
    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i)
    dt = time.perf_counter() - t0
    val = B * L * args.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": "path-contexts/sec", "value": val, "unit": "ctx/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(w, args),
        "cpu_baseline": {"value": val, "unit": "ctx/s", "cores": cores_used, "host_cores": cores, "kind": kind,
                         "sample": f"{args.steps} forward passes of {B}x{L} batches, {how}, {torch.get_num_threads()} threads"},
        "e2e": {"value": val, "unit": "ctx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, help="timed steps (default: 2000 on the GPU, 20 for --impl reference)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--algo", default="auto", choices=["auto", "ffma", "tcgen05"])
    ap.add_argument("--pool-batches", type=int, default=64, help="distinct batches in the device index pool")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--train-steps", type=int, default=8, help="also time K training steps (0 = skip)")
    ap.add_argument("--train-unfused-loss", action="store_true", help="training leg: forward() + eager loss instead of forward_loss()")
    ap.add_argument("--early-reduce", action="store_true",
                    help="training leg: reduce path_embedding's gradient on a side stream while the backward is still running "
                         "(ShardedFlatAdam early region; experimental: slower today, see DESIGN.md section 5)")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the ATen/cuBLAS eager comparator on this GPU")
    ap.add_argument("--transport", default="auto", choices=["auto", "nvls", "p2p", "nccl"],
                    help="gradient reduction of the training leg (ShardedFlatAdam)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step (rank 0) to DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.impl == "reference" else 2000
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes what the CUDA path computed; --impl reference has no such outputs")
    w = dict(WORKLOADS[args.workload]); w["name"] = args.workload

    if args.impl == "reference":
        return run_reference(args, w)

    # The measured loops are CUDA-API-bound on ONE host thread; a 128-thread OpenMP/ATen pool in the same
    # process slows the host-buffer (e2e) loop by ~60 % (measured), so this process keeps one host thread and
    # the CPU baseline runs in its own process with all of them.
    saved_omp = os.environ.get("OMP_NUM_THREADS")
    os.environ["OMP_NUM_THREADS"] = "1"
    import numpy as np
    import torch
    torch.set_num_threads(1)
    from code2vec_b200 import _lib
    from code2vec_b200 import functional as CF

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            sys.exit("--gpus N>1 must be launched with torch.distributed.run --nproc-per-node N")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    algo = {"auto": _lib.ALGO_AUTO, "ffma": _lib.ALGO_FFMA, "tcgen05": _lib.ALGO_TCGEN05}[args.algo]

    B, L, H, C = w["B"], w["L"], w["H"], w["C"]
    dims = CF.make_dims(w["T"], w["P"], C, w["Et"], w["Ep"], H)
    p = synth_params(w, dev)                        # same weights on every rank (replicated parameters)
    params = CF.make_params(p["terminal_embedding.weight"], p["path_embedding.weight"], p["input_linear.weight"],
                            p["input_layer_norm.weight"], p["input_layer_norm.bias"], p["attention_parameter"],
                            p["output_linear.weight"], p["output_linear.bias"])
    s, pth, e, lab = synth_pool(w, args.pool_batches, dev, 1234 + rank)   # each rank: its own shard of methods
    nb = args.pool_batches

    # preallocated outputs / workspaces: the timed region launches kernels only
    cv = torch.empty((B, H), dtype=torch.float32, device=dev)
    att = torch.empty((B, L), dtype=torch.float32, device=dev)
    out = torch.empty((B, C), dtype=torch.float32, device=dev)
    am = torch.empty((B,), dtype=torch.int64, device=dev); mx = torch.empty((B,), dtype=torch.float32, device=dev)
    ws_n = lib.c2v_encode_workspace_bytes(ctypes.byref(dims), B, L)
    ws = torch.empty((ws_n,), dtype=torch.uint8, device=dev)
    wl_n = lib.c2v_label_workspace_bytes(ctypes.byref(dims), B)
    wl = torch.empty((wl_n,), dtype=torch.uint8, device=dev)
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    stream = torch.cuda.current_stream(dev)
    st = ctypes.c_void_p(stream.cuda_stream)
    label_algo = _lib.ALGO_FFMA if algo == _lib.ALGO_FFMA else _lib.ALGO_AUTO

    REUSE = 0x100   # C2V_FLAG_REUSE_PREP: weights are frozen during the run (inference), as the torch
                    # module does when the parameters' version counters are unchanged

    def step(i, reuse=REUSE):
        o = (i % nb) * B
        _lib.check(lib.c2v_encode_forward(ctypes.byref(dims), ctypes.byref(params), P(s[o:o + B]), P(pth[o:o + B]),
                                          P(e[o:o + B]), B, L, None, P(cv), P(att), P(ws), ws_n, algo | reuse, st), "encode")
        _lib.check(lib.c2v_label_logits_argmax(ctypes.byref(dims), ctypes.byref(params), P(cv), B, P(out), P(am), P(mx),
                                               P(wl), wl_n, label_algo | reuse, st), "label+argmax")

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- parity gate on the first batch (rank 0): CUDA vs the pinned C oracle ---------------------
    parity = None
    if rank == 0:
        from oracle import oracle
        step(0, reuse=0); torch.cuda.synchronize(dev)     # first call builds the weight images
        nchk = min(B, 32)
        npar = {k: v.cpu().numpy() for k, v in p.items()}
        ro, rc_, ra = oracle.forward(npar, s[:nchk].cpu().numpy(), pth[:nchk].cpu().numpy(), e[:nchk].cpu().numpy(),
                                     lab[:nchk].cpu().numpy())
        parity = {"max_abs_err": {"outputs": float(np.abs(out[:nchk].cpu().numpy() - ro).max()),
                                  "code_vector": float(np.abs(cv[:nchk].cpu().numpy() - rc_).max()),
                                  "attention": float(np.abs(att[:nchk].cpu().numpy() - ra).max())},
                  "bags_checked": nchk, "tolerance": 1e-4, "checker": "oracle/c2v_oracle.c (pinned to the reference)"}
        parity["ok"] = max(parity["max_abs_err"].values()) <= 1e-4

    # ---- device-resident throughput ("value") --------------------------------------------------
    # --warmup steps, then the timed region: exactly --steps steps (batches W .. W+K-1 of the pool, so the same arguments
    # give the same inputs), bracketed by barrier + synchronize and timed with CUDA events on the launch stream.
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(args.warmup):
        step(i)
    barrier()

    def timed_pass(first):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for i in range(args.steps):
            step(first + i)
        ev1.record(stream)
        barrier()
        return ev0.elapsed_time(ev1)

    sampler.mark_begin()
    l0 = lib.c2v_launch_count()
    t_wall0 = time.perf_counter()
    pass_ms = timed_pass(args.warmup)
    timed_region_s = time.perf_counter() - t_wall0
    sampler.mark_end()
    launches = lib.c2v_launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([pass_ms], dtype=torch.float64, device=dev)
    lt = torch.tensor([float(launches)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX); dist.all_reduce(lt, op=dist.ReduceOp.SUM)   # the slowest rank
    ms_max = float(t.item())
    value = world * B * L * args.steps / (ms_max * 1e-3)
    if rank == 0 and args.dump_outputs:
        # the last timed step's results, before the legs below reuse the buffers (.gitignore lists these file names)
        dump_outputs(args.dump_outputs, {"outputs": out, "code_vector": cv, "attention": att, "predicted_label": am,
                                         "predicted_score": mx})

    # ---- roofline of the dominant kernel (this rank) -----------------------------------------------
    # CUDA events around every 8th launch of the kernel, in untimed passes of K steps after the timed one (>= 0.6 s of GPU
    # time: hundreds of samples), so that no extra event sits inside the timed region
    lib.c2v_profile_enable(8)
    for r in range(int(min(2000, max(1, -(-600.0 // max(ms_max, 1e-3)))))):     # ms_max: the same count on every rank
        timed_pass(args.warmup + (r + 1) * args.steps)
    kms, kcnt = ctypes.c_double(0), ctypes.c_int64(0)
    lib.c2v_profile_read(ctypes.byref(kms), ctypes.byref(kcnt))
    lib.c2v_profile_enable(0)
    peak, peak_src = measured_peaks()
    k_ms = kms.value / max(1, kcnt.value)
    alg_bytes = bytes_per_ctx(w) * B * L
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    kvar = {"ldg": "encode_tcgen05_kernel", "tma": "encode_tma_kernel", "cpa": "encode_cpa_kernel"}.get(
        os.environ.get("C2V_ENCODE_KERNEL", ""), "encode_tm_kernel")
    traffic = None
    for tf in ("r2_traffic.json", "r1_traffic.json"):   # DRAM traffic of the dominant kernel from the committed ncu capture
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", tf)))
            if tj["kernel"] == kvar and tj.get("workload", "cfg2") == args.workload:
                traffic = tj["traffic_bytes_per_launch"]
                break
        except Exception:
            pass
    roofline = {"bound": "hbm", "kernel": kvar if lib.c2v_encode_supports_tcgen05(ctypes.byref(dims)) and algo != _lib.ALGO_FFMA else "encode_ffma_kernel",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "kernel_ms": k_ms, "kernel_samples": int(kcnt.value), "algorithmic_bytes_per_launch": alg_bytes,
                "peak_source": peak_src, "ctx_per_s_kernel_only": B * L / (k_ms * 1e-3) if k_ms > 0 else 0.0,
                "how": "CUDA events on the launch stream around every 8th launch of the kernel, in untimed passes after the timed one "
                       "(launch + prologue inside the interval, no dependent-launch overlap for the bracketed launch)"}

    # ---- the same kernel launched back to back (no bracketing events between launches, dependent-launch overlap intact):
    #      what it costs the step, as opposed to what a bracketed launch shows; reported beside `frac`, not instead of it
    def enc_only(i):
        o = (i % nb) * B
        _lib.check(lib.c2v_encode_forward(ctypes.byref(dims), ctypes.byref(params), P(s[o:o + B]), P(pth[o:o + B]),
                                          P(e[o:o + B]), B, L, None, P(cv), P(att), P(ws), ws_n, algo | REUSE, st), "encode")
    n_b2b = 256
    for i in range(8):
        enc_only(i)
    torch.cuda.synchronize(dev)
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record(stream)
    for i in range(n_b2b):
        enc_only(8 + i)
    b1.record(stream)
    torch.cuda.synchronize(dev)
    b2b_ms = b0.elapsed_time(b1) / n_b2b                       # encode kernel + its 4 us finalize kernel per call
    roofline["encode_call_ms_back_to_back"] = b2b_ms
    roofline["frac_back_to_back"] = alg_bytes / (b2b_ms * 1e-3) / 1e9 / peak
    roofline["back_to_back_note"] = (f"{n_b2b} c2v_encode_forward calls (encode_tm_kernel + encode_finalize_kernel) between two CUDA events, "
                                     "no events in between; includes the finalize kernel, so it is an upper bound of the kernel's own time")

    # ---- the same path on the existing Blackwell kernels: ATen/cuBLAS eager on this GPU (BASELINE.md 3.5) ----------
    gpu_eager = None
    if rank == 0 and not args.no_gpu_eager:
        try:
            from oracle import oracle as _or                 # baseline leg only: the torch restatement dispatches to ATen
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.allow_tf32 = False
            def estep(i):
                o = (i % nb) * B
                with torch.no_grad():
                    o_, _, _ = _or.torch_forward(p, s[o:o + B], pth[o:o + B], e[o:o + B], lab[o:o + B])
                    return o_.max(dim=1)
            for i in range(3):
                estep(i)
            torch.cuda.synchronize(dev)
            n_e = max(5, min(args.steps, 50))
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record(stream)
            for i in range(n_e):
                estep(3 + i)
            g1.record(stream)
            torch.cuda.synchronize(dev)
            gms = g0.elapsed_time(g1) / n_e
            gpu_eager = {"value": B * L / (gms * 1e-3), "unit": "ctx/s", "ms_per_step": gms, "steps": n_e, "n_gpus": 1,
                         "what": "the reference's op sequence (model.py:48-83 + torch.max) as eager ATen/cuBLAS kernels on this "
                                 "B200, fp32, allow_tf32=False (oracle.torch_forward on cuda; the reference itself is absent here)"}
            torch.cuda.empty_cache()
        except Exception as ex:
            gpu_eager = {"value": None, "unit": "ctx/s", "what": f"failed: {type(ex).__name__}: {ex}"}

    # ---- end to end through the host-buffer C-ABI call (pinned host inputs, H2D + D2H inside) ------
    e2e = None
    if not args.no_e2e:
        bound = bind_to_gpu_numa_node(local)             # before the pinned staging buffers and the session exist
        sess = ctypes.c_void_p()
        _lib.check(lib.c2v_session_create(local, ctypes.byref(dims), B, L, ctypes.byref(sess)), "session")
        hb = min(nb, 8)
        hs, hp, he = s[:hb * B].cpu().pin_memory(), pth[:hb * B].cpu().pin_memory(), e[:hb * B].cpu().pin_memory()
        DEPTH = 4                              # batches in flight (the session has 4 staging slots)
        hcv = [torch.empty((B, H), dtype=torch.float32).pin_memory() for _ in range(DEPTH)]
        hat = [torch.empty((B, L), dtype=torch.float32).pin_memory() for _ in range(DEPTH)]
        hpr = [torch.empty((B,), dtype=torch.int64).pin_memory() for _ in range(DEPTH)]
        hsc = [torch.empty((B,), dtype=torch.float32).pin_memory() for _ in range(DEPTH)]
        tick = ctypes.c_int64(0)

        def host_loop(n):
            pending = []
            for i in range(n):
                o = (i % hb) * B; k = i % DEPTH
                _lib.check(lib.c2v_forward_host_async(sess, ctypes.byref(params), P(hs[o:o + B]), P(hp[o:o + B]),
                                                      P(he[o:o + B]), None, B, None, P(hcv[k]), P(hat[k]), P(hpr[k]),
                                                      P(hsc[k]), algo | REUSE, ctypes.byref(tick)), "forward_host_async")
                pending.append(tick.value)
                if len(pending) == DEPTH:   # results of step i-3 are consumed while steps i-2..i are in flight
                    _lib.check(lib.c2v_session_wait(sess, pending.pop(0)), "session_wait")
            for tk in pending:
                _lib.check(lib.c2v_session_wait(sess, tk), "session_wait")

        def host_pass():
            barrier()
            t0 = time.perf_counter()
            host_loop(args.steps)
            torch.cuda.synchronize(dev)
            return time.perf_counter() - t0
        # warm up until two consecutive passes agree within 5 % (first passes pay page faults / the copy engines' ramp)
        prev, n_warm = host_pass(), 1
        while n_warm < 12:
            cur = host_pass(); n_warm += 1
            tw = torch.tensor([1.0 if abs(cur - prev) <= 0.05 * prev else 0.0], dtype=torch.float64, device=dev)
            if dist is not None:
                dist.all_reduce(tw, op=dist.ReduceOp.MIN)      # every rank takes the same number of passes
            prev = cur
            if tw.item() > 0:
                break
        te = torch.tensor([host_pass()], dtype=torch.float64, device=dev)   # the timed pass: exactly --steps steps
        if dist is not None:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)           # the slowest rank
        dt = float(te.item())
        lib.c2v_session_destroy(sess)
        e2e = {"value": world * B * L * args.steps / dt, "unit": "ctx/s",
               "h2d_bytes_per_step": 3 * B * L * 8, "d2h_bytes_per_step": B * H * 4 + B * L * 4 + B * 8 + B * 4 + 8,
               "api": "c2v_forward_host_async (4 batches in flight on upload / compute / download streams; pinned host int64 indices in, code_vector + "
                      "attention + argmax/score out; the [B, C] logits stay on the device: this is the predict surface of main.py:282-285)",
               "ms_per_step": dt / args.steps * 1e3, "warmup_passes": n_warm, "cpu_binding": bound}

    # ---- training step (reported beside the metric, not the metric): main.py:171-175 on this rank's shard; the gradient
    #      reduction over the ranks is fused into the optimizer kernel (ShardedFlatAdam, NVLS) -- no NCCL call in the step
    train = None
    if args.train_steps > 0:
        import types
        import torch.nn.functional as F
        from code2vec_b200.model import Code2Vec
        from code2vec_b200.distributed import ShardedFlatAdam, ddp_step
        opt_ns = types.SimpleNamespace(terminal_count=w["T"], path_count=w["P"], label_count=C,
                                       terminal_embed_size=w["Et"], path_embed_size=w["Ep"], encode_size=H,
                                       dropout_prob=0.25, angular_margin_loss=False, angular_margin=0.5,
                                       inverse_temp=30.0, device=dev)
        model = Code2Vec(opt_ns, algo=args.algo)
        model.load_state_dict(p)
        model = model.to(dev).train()
        optim = ShardedFlatAdam(model.parameters(), lr=0.01, betas=(0.9, 0.999), transport=args.transport,   # main.py:138
                                early=[model.path_embedding.weight] if args.early_reduce else [])
        # main.py:251-264: by default through Code2Vec.forward_loss (loss fused into the label GEMM, logits never written);
        # --train-unfused-loss: forward() + eager log_softmax + nll_loss on the [b, C] logits, like the reference's loop
        loss_fn = (lambda o_, l_: F.nll_loss(F.log_softmax(o_, dim=1), l_)) if args.train_unfused_loss else None
        def tstep(i):
            o = (i % nb) * B
            return ddp_step(model, optim, None, s[o:o + B], pth[o:o + B], e[o:o + B], lab[o:o + B], loss_fn)
        for i in range(3):
            tstep(i)
        barrier()
        def train_pass(first):
            tv0, tv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            tv0.record(stream)
            for i in range(args.train_steps):
                last = tstep(first + i)
            tv1.record(stream)
            barrier()
            return tv0.elapsed_time(tv1), last
        t_reps = 5
        res = [train_pass(3 + r * args.train_steps) for r in range(t_reps)]
        tt = torch.tensor([r[0] for r in res], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        tms = float(tt.median().item())
        train = {"value": world * B * L * args.train_steps / (tms * 1e-3), "unit": "ctx/s",
                 "ms_per_step": tms / args.train_steps, "steps": args.train_steps, "passes": t_reps,
                 "loss": "forward + eager log_softmax/nll_loss" if args.train_unfused_loss else "fused into the label GEMM (forward_loss)",
                 "step": "forward(dropout .25) + mean NLL + backward + gradient reduction over the ranks + dense Adam "
                         "(optimizer state sharded 1/world; reduction + Adam + parameter broadcast = one kernel per rank)",
                 "early_region": len(optim.regions) > 1, "transport": optim.transport, "transport_calibration_ms": optim.calibration, "gradient_bytes": 4 * optim.numel, "loss_value": float(res[-1][1].item())}
        del model, optim
        torch.cuda.empty_cache()

    # ---- CPU baseline beside it: rank 0, N=1 only, bounded sample, in its own process (all host threads)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        env = dict(os.environ)
        if saved_omp is None:
            env.pop("OMP_NUM_THREADS", None)
        else:
            env["OMP_NUM_THREADS"] = saved_omp
        env["CUDA_VISIBLE_DEVICES"] = ""
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload",
                                args.workload, "--steps", "8", "--warmup", "2"], env=env, capture_output=True,
                               text=True, timeout=600)
            cpu = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as ex:      # keep the GPU numbers even if the host leg fails
            cpu = {"value": None, "unit": "ctx/s", "cores": None, "kind": "port", "sample": f"failed: {ex}"}

    if rank == 0:
        cfg = bench_config(w, args)
        print(json.dumps({
            "metric": "path-contexts/sec", "value": value, "unit": "ctx/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "timing": {"pass_ms": ms_max, "timed_region_s": timed_region_s, "algo": args.algo,
                       "how": f"one pass of exactly {args.steps} steps after {args.warmup} warm-up steps, bracketed by barrier + "
                              "synchronize and timed with CUDA events on the launch stream; max over ranks"},
            "roofline": roofline, "cpu_baseline": cpu, "gpu_eager_baseline": gpu_eager, "e2e": e2e, "train": train,
            "clocks": clocks, "gpu_launches": int(round(lt.item())), "parity": parity,
        }))
    if dist is not None:
        dist.destroy_process_group()


def bind_to_gpu_numa_node(local):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off (GPUs 4-7 of an 8-GPU box sit on node 1): the host
    loop of the e2e leg and its pinned staging buffers then live next to the GPU.  Returns what was done."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return f"gpu {bdf}: no NUMA affinity reported"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return f"gpu {bdf}: node {node} has no CPUs this process may use"
        os.sched_setaffinity(0, cpus)
        return f"gpu {bdf} -> NUMA node {node}, {len(cpus)} cpus"
    except Exception as ex:
        return f"not bound ({type(ex).__name__}: {ex})"


if __name__ == "__main__":
    # stdout carries the ONE JSON line and nothing else: libraries that write to file descriptor 1 during the run (NCCL's
    # "NCCL version ..." banner at communicator creation) are sent to stderr; print() goes to the real stdout at the end.
    import io
    sys.dont_write_bytecode = True      # the tree may be read-only: the run writes nothing into it
    sys.stdout.flush()
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    _buf = io.StringIO()
    _py_stdout, sys.stdout = sys.stdout, _buf
    try:
        main()
    finally:
        sys.stdout = _py_stdout
        os.dup2(_real_stdout, 1)
        os.close(_real_stdout)
        sys.stdout.write(_buf.getvalue())
        sys.stdout.flush()
