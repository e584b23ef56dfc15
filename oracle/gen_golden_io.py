#!/usr/bin/env python
"""Generate the fixtures that pin the corpus reader / variable-task builder / code-vector writer (SURVEY.md 8f rows 2, 4)
by running the UNMODIFIED reference (imported from /root/reference, never copied) in the dev container:

    PYTHONDONTWRITEBYTECODE=1 python oracle/gen_golden_io.py

  tests/golden/reader_synth.npz   reference DatasetReader on oracle.corpus_oracle.synthetic_corpus(seed) (seeds 1, 2)
  tests/golden/builder_vars.npz   reference DatasetBuilder.build_data, infer_variable branch (dataset_builder.py:152-204)
  tests/golden/writer.npz         reference write_code_vectors (main.py:393-423) output for fixed vectors
  tests/golden/unaligned.npz, grad_unaligned.npz   forward / gradient goldens with embed / encode sizes not divisible by 4
  tests/golden/grad_wide.npz, grad_e200.npz        gradient goldens with embed / encode sizes above 128
"""
import ast
import json
import os
import random
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE); sys.path.insert(0, os.path.dirname(HERE))
import gen_golden as gg                         # noqa: E402  (puts /root/reference on sys.path, imports the reference model)
from oracle import corpus_oracle as co          # noqa: E402
import logging                                   # noqa: E402
logging.disable(logging.CRITICAL)
from model.dataset_builder import DatasetBuilder  # noqa: E402
from model.dataset_reader import DatasetReader    # noqa: E402

REF, OUT = gg.REF, gg.OUT


def _reader_record(reader):
    items = reader.items
    off = np.zeros(len(items) + 1, np.int64)
    for i, it in enumerate(items):
        off[i + 1] = off[i] + len(it.path_contexts)
    ctx = np.asarray([pc for it in items for pc in it.path_contexts], dtype=np.int64).reshape(-1, 3)
    lv = reader.label_vocab
    return {
        "ids": [it.id for it in items],
        "labels": [it.label for it in items],
        "normalized_labels": [it.normalized_label for it in items],
        "aliases": [list(it.aliases.items()) for it in items],
        "label_names": [lv.itos[i] for i in range(lv.len())],
        "label_subtokens": [lv.itosubtokens[i] for i in range(lv.len())],
        "variable_indexes": list(reader.variable_indexes),
        "terminal_count": reader.terminal_vocab.len(), "path_count": reader.path_vocab.len(),
        "question": reader.terminal_vocab.stoi["@question"], "method0": reader.terminal_vocab.stoi["@method_0"],
    }, off, ctx


def _write_synth(seed, d):
    text, term, path = co.synthetic_corpus(seed)
    paths = [os.path.join(d, n) for n in ("corpus.txt", "terminal_idxs.txt", "path_idxs.txt")]
    for p, t in zip(paths, (text, term, path)):
        with open(p, "w", encoding="utf-8", newline="") as f:      # newline="": keep the \r\n lines as generated
            f.write(t)
    return paths


def reader_synth():
    rec = {}
    for seed in (1, 2):
        with tempfile.TemporaryDirectory() as d:
            cp, tp, pp = _write_synth(seed, d)
            for tag, im, iv in (("mv", True, True), ("m", True, False), ("v", False, True)):
                r = DatasetReader(cp, pp, tp, infer_method=im, infer_variable=iv, shuffle_variable_indexes=False)
                meta, off, ctx = _reader_record(r)
                rec[f"s{seed}_{tag}_meta"] = np.array(json.dumps(meta, ensure_ascii=False))
                rec[f"s{seed}_{tag}_offsets"] = off
                rec[f"s{seed}_{tag}_contexts"] = ctx
    np.savez_compressed(os.path.join(OUT, "reader_synth.npz"), **rec)
    print("reader_synth:", len(rec), "arrays")


def builder_vars():
    """dataset_builder.py:152-204 on the synthetic corpus (seed 1) and on 48 methods of dataset/corpus.txt."""
    rec = {}
    for tag in ("synth", "real"):
        with tempfile.TemporaryDirectory() as d:
            if tag == "synth":
                cp, tp, pp = _write_synth(1, d)
            else:
                cp, tp, pp = (f"{REF}/dataset/{n}" for n in ("corpus.txt", "terminal_idxs.txt", "path_idxs.txt"))
            random.seed(5)
            r = DatasetReader(cp, pp, tp, infer_method=False, infer_variable=True, shuffle_variable_indexes=False)
            o = gg.option(r.terminal_vocab.len(), r.path_vocab.len(), r.label_vocab.len(), 8, 8, 8)
            o.max_path_length, o.eval_method, o.batch_size = (5 if tag == "synth" else 200), "exact", 32
            items = list(r.items)
            if tag == "real":
                items = sorted(items, key=lambda it: -len(it.path_contexts))[:8] + items[100:140]
            r.items = list(items)
            b = DatasetBuilder(r, o)                                # shuffles r.items (a copy) in place: `items` keeps our order
            off = np.zeros(len(items) + 1, np.int64)
            for i, it in enumerate(items):
                off[i + 1] = off[i] + len(it.path_contexts)
            ctx = np.asarray([pc for it in items for pc in it.path_contexts], dtype=np.int32).reshape(-1, 3)
            ids, s, p, e, lab = b.build_data(r, items, o.max_path_length)
            units = [(i, r.terminal_vocab.stoi[a], r.label_vocab.stoi[it.aliases[a]])
                     for i, it in enumerate(items) for a in it.aliases if a.startswith("@var_")]
            rec.update({f"{tag}_offsets": off, f"{tag}_contexts": ctx, f"{tag}_units": np.asarray(units, np.int64).reshape(-1, 3),
                        f"{tag}_ref_starts": s.numpy(), f"{tag}_ref_paths": p.numpy(), f"{tag}_ref_ends": e.numpy(),
                        f"{tag}_ref_label": lab.numpy(), f"{tag}_ref_ids": np.asarray([-1 if v is None else v for v in ids], np.int64),
                        f"{tag}_item_ids": np.asarray([-1 if it.id is None else it.id for it in items], np.int64),
                        f"{tag}_variable_indexes": np.asarray(r.variable_indexes, np.int64),
                        f"{tag}_L": np.int64(o.max_path_length), f"{tag}_question": np.int64(r.QUESTION_TOKEN_INDEX)})
            print("builder_vars", tag, len(items), "items", len(units), "units")
    np.savez_compressed(os.path.join(OUT, "builder_vars.npz"), **rec)


def writer():
    """Runs the reference's own write_code_vectors (main.py:393-423) -- the function's source is taken from the reference
    file with ast at generation time (main.py itself parses argv and trains at import, so it cannot be imported)."""
    src = open(f"{REF}/main.py", encoding="utf-8").read()
    fn = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "write_code_vectors")
    ns = {"torch": torch}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), f"{REF}/main.py", "exec"), ns)
    rng = np.random.default_rng(3)
    names = ["getvalue", "tostring", "größeändern", "a", "run"]
    n, H = 11, 7
    vec = rng.standard_normal((n, H)).astype(np.float32)
    vec[0, :] = [0.0, -0.0, 1.0, 1e-5, 123456789.0, 1e16, 3.4e38]
    vec[1, :] = [1e-4, 0.1, 0.5, 2.5e-7, 16777216.0, 9.999999e15, 1.17549435e-38]
    vec[2, :3] = [float("nan"), float("inf"), float("-inf")]
    label = rng.integers(0, len(names), n)
    logits = rng.standard_normal((n, len(names))).astype(np.float32) * 5
    ids = rng.integers(0, 10000, n)

    class M:
        def eval(self): pass
        def forward(self, s, p, e, lab):
            i = int(s[0, 0])
            k = len(s)
            return torch.from_numpy(logits[i:i + k]), torch.from_numpy(vec[i:i + k]), None
    reader = types.SimpleNamespace(label_vocab=types.SimpleNamespace(itos=dict(enumerate(names))))
    loader, i = [], 0
    for k in (4, 4, 3):                       # ragged last batch; starts[0, 0] carries the row offset for the stub model
        loader.append({"id": torch.from_numpy(ids[i:i + k]), "starts": torch.full((k, 2), i), "paths": torch.zeros(k, 2),
                       "ends": torch.zeros(k, 2), "label": torch.from_numpy(label[i:i + k])})
        i += k
    opt = types.SimpleNamespace(device=torch.device("cpu"))
    with tempfile.TemporaryDirectory() as d:
        vf, rf = os.path.join(d, "code.vec"), os.path.join(d, "result.tsv")
        with open(vf, "w") as f:
            f.write("{0}\t{1}\n".format(n, H))                     # main.py:227-228
        ns["write_code_vectors"](reader, M(), loader, opt, vf, "a", rf)
        vtxt, rtxt = open(vf, encoding="utf-8").read(), open(rf, encoding="utf-8").read()
    np.savez_compressed(os.path.join(OUT, "writer.npz"), vec=vec, label=label, logits=logits, ids=ids,
                        names=np.array(json.dumps(names, ensure_ascii=False)), vector_text=np.array(vtxt),
                        result_text=np.array(rtxt))
    print("writer:", len(vtxt), "bytes,", len(rtxt), "bytes")


if __name__ == "__main__":
    reader_synth()
    builder_vars()
    writer()
    gg.seeded("unaligned", 21, 6, 9, 23, 17, 5, 10, 7, 9, holes=True, allpad_rows=(3,))
    gg.seeded("grad_unaligned", 22, 5, 11, 23, 17, 5, 10, 7, 9, grads=True, holes=True, allpad_rows=(2,))
    gg.seeded("grad_e50", 23, 3, 12, 40, 30, 6, 50, 50, 50, grads=True)
    # embed / encode sizes above 128: the tensor-core backward runs them as 128-wide windows (c2v_backward_d{w,c}_tc.cu)
    gg.seeded("grad_wide", 24, 5, 70, 80, 60, 12, 256, 256, 256, grads=True, allpad_rows=(3,))
    gg.seeded("grad_e200", 25, 4, 60, 90, 70, 10, 200, 200, 192, grads=True, holes=True)
