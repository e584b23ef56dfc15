#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference/model/model.py, imported -- never copied) on seeded inputs.

Run in the dev container only (the GPU box has no /root/reference):
    PYTHONDONTWRITEBYTECODE=1 python oracle/gen_golden.py
The committed .npz files are what pins oracle/c2v_oracle.c and what the
`-m gpu` parity tests compare the CUDA path against.

Each file holds: the Option values, every parameter (reference state_dict keys),
the int64 inputs, and the reference outputs (outputs, code_vector, attention);
grad_* files also hold d(mean NLL)/d(param) from the reference's autograd.
"""
import os
import sys
import types

import numpy as np
import torch
import torch.nn.functional as F

REF = os.environ.get("C2V_REFERENCE", "/root/reference")
sys.dont_write_bytecode = True
sys.path.insert(0, REF)
from model.model import Code2Vec  # noqa: E402  (the reference, unmodified)

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")
sys.path.insert(0, os.path.join(OUT, ".."))
from conftest import params_sha256  # noqa: E402  (the digest tests/conftest.py checks)
os.makedirs(OUT, exist_ok=True)


def option(T, P, C, Et, Ep, H, dropout=0.0, angular=False, margin=0.5, inv_temp=30.0):
    o = types.SimpleNamespace()
    o.terminal_count, o.path_count, o.label_count = T, P, C
    o.terminal_embed_size, o.path_embed_size, o.encode_size = Et, Ep, H
    o.dropout_prob = dropout
    o.angular_margin_loss, o.angular_margin, o.inverse_temp = angular, margin, inv_temp
    o.device = torch.device("cpu")
    return o


def make_inputs(gen, B, L, T, P, C, pad="suffix", holes=False, allpad_rows=()):
    starts = torch.randint(1, T, (B, L), generator=gen)
    paths = torch.randint(1, P, (B, L), generator=gen)
    ends = torch.randint(1, T, (B, L), generator=gen)
    if pad == "suffix":  # what dataset_builder.py:145-147 produces
        n = torch.randint(1, L + 1, (B,), generator=gen)
        n[0] = L
        for b in range(B):
            starts[b, n[b]:] = 0; paths[b, n[b]:] = 0; ends[b, n[b]:] = 0
    if holes:  # mask depends on starts only (model.py:64): holes, and paths/ends nonzero under a pad start
        hm = torch.rand((B, L), generator=gen) < 0.2
        starts[hm] = 0
    for b in allpad_rows:
        starts[b, :] = 0
        if b % 2 == 0:
            paths[b, :] = 0; ends[b, :] = 0
    label = torch.randint(0, C, (B,), generator=gen)
    return starts, paths, ends, label


def dump(name, opt, model, starts, paths, ends, label, grads=False, scale=None, param_seed=None):
    """param_seed: the torch.manual_seed the model was built under (plain head, unscaled).  A record that would exceed
    1 MB then stores the seed and a digest of the parameters instead of the parameters (tests/conftest.py rebuilds them)."""
    model.eval()
    if scale:
        with torch.no_grad():
            for k, v in model.state_dict().items():
                v.mul_(scale.get(k, 1.0))
            if "output_linear.bias" in model.state_dict():
                model.output_linear.bias.normal_(0.0, 0.3)
    rec = {
        "opt_T": opt.terminal_count, "opt_P": opt.path_count, "opt_C": opt.label_count,
        "opt_Et": opt.terminal_embed_size, "opt_Ep": opt.path_embed_size, "opt_H": opt.encode_size,
        "opt_angular": int(opt.angular_margin_loss), "opt_margin": opt.angular_margin,
        "opt_inverse_temp": opt.inverse_temp,
        "starts": starts.numpy(), "paths": paths.numpy(), "ends": ends.numpy(), "label": label.numpy(),
    }
    for k, v in model.state_dict().items():
        rec["param." + k] = v.detach().numpy().copy()
    if grads:
        model.zero_grad()
        out, cv, att = model.forward(starts, paths, ends, label)
        # main.py:251-264 with weight == 1 (SURVEY.md 8a row 16)
        loss = F.nll_loss(F.log_softmax(out, dim=1), label)
        loss.backward()
        rec["loss"] = np.float32(loss.item())
        for k, p in model.named_parameters():
            rec["grad." + k] = p.grad.detach().numpy().copy()
    else:
        with torch.no_grad():
            out, cv, att = model.forward(starts, paths, ends, label)
    rec["outputs"] = out.detach().numpy(); rec["code_vector"] = cv.detach().numpy()
    rec["attention"] = att.detach().numpy()
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **rec)
    if param_seed is not None and os.path.getsize(path) > 1_000_000:
        params = {k[6:]: v for k, v in rec.items() if k.startswith("param.")}
        rec = {k: v for k, v in rec.items() if not k.startswith("param.")}
        rec["param_seed"] = np.int64(param_seed)
        rec["param_sha256"] = np.str_(params_sha256(params))
        np.savez_compressed(path, **rec)
    print(f"{name:22s} B={starts.shape[0]:3d} L={starts.shape[1]:3d} -> {os.path.getsize(path)/1024:.0f} KiB")


def kat():
    """RNG-free known-answer test, SURVEY.md section 8(c)."""
    opt = option(7, 5, 3, 2, 3, 4)
    m = Code2Vec(opt)
    fills = {
        "terminal_embedding.weight": (0.37, 0.1), "path_embedding.weight": (0.53, 0.2),
        "input_linear.weight": (0.29, 0.3), "input_layer_norm.weight": (0.41, 1.0),
        "input_layer_norm.bias": (0.23, -0.5), "attention_parameter": (0.61, 0.4),
        "output_linear.weight": (0.47, 0.6), "output_linear.bias": (0.31, -0.2),
    }
    with torch.no_grad():
        for k, t in m.state_dict().items():
            a, b = fills[k]
            t.copy_(torch.sin(torch.arange(t.numel(), dtype=torch.float64) * a + b).float().view_as(t))
    starts = torch.tensor([[1, 3, 6, 0, 0], [2, 0, 5, 4, 1], [0, 0, 0, 0, 0]])
    paths = torch.tensor([[1, 2, 4, 0, 0], [3, 0, 1, 2, 4], [0, 0, 0, 0, 0]])
    ends = torch.tensor([[2, 5, 1, 0, 0], [6, 0, 3, 1, 2], [0, 0, 0, 0, 0]])
    label = torch.tensor([0, 2, 1])
    dump("kat", opt, m, starts, paths, ends, label)


def seeded(name, seed, B, L, T, P, C, Et, Ep, H, grads=False, scale=None, angular=False, **kw):
    torch.manual_seed(seed)
    opt = option(T, P, C, Et, Ep, H, angular=angular)
    m = Code2Vec(opt)
    gen = torch.Generator().manual_seed(seed + 1000)
    starts, paths, ends, label = make_inputs(gen, B, L, T, P, C, **kw)
    dump(name, opt, m, starts, paths, ends, label, grads=grads, scale=scale,
         param_seed=seed if scale is None and not angular else None)


def real_batch():
    """A real batch built by the reference's own reader/builder from dataset/corpus.txt
    (dataset_reader.py:44-128, dataset_builder.py:112-210), tables compacted to the
    rows the batch touches so the fixture stays small."""
    import random
    import logging
    logging.disable(logging.CRITICAL)
    from model.dataset_builder import DatasetBuilder
    from model.dataset_reader import DatasetReader
    random.seed(7)
    torch.manual_seed(7)
    reader = DatasetReader(f"{REF}/dataset/corpus.txt", f"{REF}/dataset/path_idxs.txt",
                           f"{REF}/dataset/terminal_idxs.txt", infer_method=True, infer_variable=False,
                           shuffle_variable_indexes=False)
    o = option(reader.terminal_vocab.len(), reader.path_vocab.len(), reader.label_vocab.len(), 100, 100, 100)
    o.max_path_length, o.eval_method, o.batch_size = 200, "exact", 32
    builder = DatasetBuilder(reader, o)
    builder.refresh_test_dataset()
    ds = builder.test_dataset
    B = 32
    starts = torch.stack([ds[i]["starts"] for i in range(B)])
    paths = torch.stack([ds[i]["paths"] for i in range(B)])
    ends = torch.stack([ds[i]["ends"] for i in range(B)])
    label = torch.tensor([int(ds[i]["label"]) for i in range(B)])
    full = Code2Vec(o)
    # compact: remap indices to the unique rows used (PAD row 0 kept at 0)
    ut = torch.unique(torch.cat([starts.flatten(), ends.flatten(), torch.tensor([0])]))
    up = torch.unique(torch.cat([paths.flatten(), torch.tensor([0])]))
    ul = torch.unique(label)
    tmap = torch.full((o.terminal_count,), -1, dtype=torch.long); tmap[ut] = torch.arange(len(ut))
    pmap = torch.full((o.path_count,), -1, dtype=torch.long); pmap[up] = torch.arange(len(up))
    lmap = torch.full((o.label_count,), -1, dtype=torch.long); lmap[ul] = torch.arange(len(ul))
    o2 = option(len(ut), len(up), len(ul), 100, 100, 100)
    small = Code2Vec(o2)
    with torch.no_grad():
        sd, fd = small.state_dict(), full.state_dict()
        sd["terminal_embedding.weight"].copy_(fd["terminal_embedding.weight"][ut])
        sd["path_embedding.weight"].copy_(fd["path_embedding.weight"][up])
        sd["output_linear.weight"].copy_(fd["output_linear.weight"][ul])
        sd["output_linear.bias"].copy_(fd["output_linear.bias"][ul])
        for k in ("input_linear.weight", "input_layer_norm.weight", "input_layer_norm.bias", "attention_parameter"):
            sd[k].copy_(fd[k])
    dump("real_batch", o2, small, tmap[starts], pmap[paths], tmap[ends], lmap[label])


def builder_corpus():
    """The reference's own reader + builder on dataset/corpus.txt (dataset_reader.py:44-128, dataset_builder.py:112-150):
    the contexts of 64 methods (all the long ones first, so that n > max_path_length is covered) as CSR, and what
    `DatasetBuilder.build_data` made of them under random.seed(11) -- the pin of oracle/batch_oracle.py."""
    import random
    import logging
    import numpy as np
    logging.disable(logging.CRITICAL)
    from model.dataset_builder import DatasetBuilder
    from model.dataset_reader import DatasetReader
    random.seed(11)
    reader = DatasetReader(f"{REF}/dataset/corpus.txt", f"{REF}/dataset/path_idxs.txt",
                           f"{REF}/dataset/terminal_idxs.txt", infer_method=True, infer_variable=False,
                           shuffle_variable_indexes=False)
    o = option(reader.terminal_vocab.len(), reader.path_vocab.len(), reader.label_vocab.len(), 100, 100, 100)
    o.max_path_length, o.eval_method, o.batch_size = 200, "exact", 32
    builder = DatasetBuilder(reader, o)
    items = sorted(reader.items, key=lambda it: -len(it.path_contexts))
    items = items[:6] + [it for it in items if 150 <= len(it.path_contexts) <= 260][:10] + items[len(items) // 2:len(items) // 2 + 40] + items[-8:]
    offsets = np.zeros(len(items) + 1, dtype=np.int64)
    ctx = []
    for i, it in enumerate(items):
        offsets[i + 1] = offsets[i] + len(it.path_contexts)
        ctx.extend(it.path_contexts)                       # stored order BEFORE build_data shuffles in place
    ctx = np.asarray(ctx, dtype=np.int32).reshape(-1, 3)
    ids, starts, paths, ends, label = builder.build_data(reader, items, o.max_path_length)
    np.savez_compressed(os.path.join(OUT, "builder_corpus.npz"), offsets=offsets, contexts=ctx,
                        method_token=np.int64(reader.terminal_vocab.stoi["@method_0"]),
                        question_token=np.int64(reader.QUESTION_TOKEN_INDEX), max_path_length=np.int64(o.max_path_length),
                        ref_starts=starts.numpy(), ref_paths=paths.numpy(), ref_ends=ends.numpy(), ref_label=label.numpy(),
                        item_label=np.asarray([reader.label_vocab.stoi[it.normalized_label] for it in items], dtype=np.int64))
    print("builder_corpus:", len(items), "items,", len(ctx), "contexts, longest", int(np.diff(offsets).max()))


def init_fingerprint():
    """Initial weights under torch.manual_seed (main.py:120): the boundary module must
    create its parameters in the same RNG order (SURVEY.md 8a row 1)."""
    torch.manual_seed(123)
    m = Code2Vec(option(50, 40, 9, 6, 10, 8, dropout=0.25))
    rec = {"param." + k: v.numpy().copy() for k, v in m.state_dict().items()}
    torch.manual_seed(123)
    m = Code2Vec(option(50, 40, 9, 6, 10, 8, angular=True))
    rec.update({"angular." + k: v.numpy().copy() for k, v in m.state_dict().items()})
    np.savez_compressed(os.path.join(OUT, "init_seed123.npz"), **rec)
    print("init_seed123")


if __name__ == "__main__":
    kat()
    seeded("tiny", 1, 5, 7, 11, 9, 6, 8, 12, 16, holes=True, allpad_rows=(2, 3))
    seeded("odd", 2, 9, 13, 37, 23, 10, 20, 36, 24, holes=True, allpad_rows=(4,))
    seeded("cfg1_small", 3, 8, 200, 500, 700, 50, 100, 100, 100)
    seeded("cfg2_small", 4, 6, 200, 1000, 800, 64, 128, 128, 128, allpad_rows=(5,))
    seeded("cfg2_full_bags", 5, 5, 200, 600, 500, 40, 128, 128, 128, pad="none")
    seeded("cfg4_small", 6, 3, 200, 300, 200, 32, 256, 256, 256)
    seeded("trained_scale", 7, 6, 200, 400, 300, 48, 128, 128, 128,
           scale={"terminal_embedding.weight": 3.0, "path_embedding.weight": 3.0, "input_linear.weight": 8.0,
                  "attention_parameter": 6.0, "output_linear.weight": 10.0})
    seeded("angular", 8, 6, 11, 30, 20, 7, 8, 8, 16, angular=True, holes=True)
    seeded("shortbag", 9, 40, 3, 30, 20, 7, 128, 128, 128, holes=True, allpad_rows=(7,))
    seeded("grad_tiny", 11, 5, 7, 11, 9, 6, 8, 12, 16, grads=True, holes=True, allpad_rows=(2,))
    seeded("grad_odd", 12, 9, 13, 37, 23, 10, 20, 36, 24, grads=True, holes=True)
    seeded("grad_cfg2", 13, 4, 50, 200, 150, 24, 128, 128, 128, grads=True)
    seeded("grad_cfg1", 14, 3, 40, 120, 90, 12, 100, 100, 100, grads=True, allpad_rows=(1,))
    init_fingerprint()
    real_batch()
    builder_corpus()
