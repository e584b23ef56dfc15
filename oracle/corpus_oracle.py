"""CPU restatement (plain Python) of the reference's corpus reader and code-vector writer --
TEST INFRASTRUCTURE ONLY: the checker of `c2v_corpus_parse_*` / `c2v_write_code_vectors`
(code2vec_b200/csrc/c2v_corpus.cpp) and of their Python mirror, never the product path.

  parse_corpus   DatasetReader.load, /root/reference/model/dataset_reader.py:72-128, line for line
                 (strip -> blank closes the item -> '#', 'label:', 'class:', 'paths:', 'vars:', 'doc:' -> mode lines)
  label_vocab    the label vocabulary those lines build (:94-100, :120-124) with Vocab.append semantics (dataset.py:64-74)
  format_vectors write_code_vectors, /root/reference/main.py:393-423 (+ header :227-228)
  synthetic_corpus  seeded generator of a small corpus.txt / *_idxs.txt triple with the edge cases the format allows

Pinned to the reference by tests/golden/reader_synth.npz (the reference's own DatasetReader run on synthetic_corpus(seed)
by oracle/gen_golden_io.py).
"""
import re

import numpy as np

_REDUNDANT = re.compile(r"[_0-9]+")                                             # dataset.py:56
_SUBTOKEN = re.compile(r"([a-z]+)([A-Z][a-z]+)|([A-Z][a-z]+)")                  # dataset.py:57
QUESTION_TOKEN_INDEX = 1


def normalize(name):
    return _REDUNDANT.sub("", name)


def subtokens(name):
    return [x.lower() for x in _SUBTOKEN.split(name) if x is not None and x != ""]


def parse_corpus(text, question_shift=QUESTION_TOKEN_INDEX):
    """-> list of items: dict(id, label, normalized_label, path_contexts [(s, p, e)], aliases [(alias, normalized)] in
    dict order, events [('label', norm, subtokens) | ('var', alias, norm, subtokens)] in line order)."""
    items, cur, mode = [], None, 0
    # text-mode universal newlines: '\r\n' and a lone '\r' both end a line
    for line in text.replace("\r\n", "\n").replace("\r", "\n").split("\n"):
        line = line.strip(" \r\n\t")
        if line == "":
            if cur is not None:
                items.append(cur)
                cur = None
            continue
        if cur is None:
            cur = {"id": None, "label": None, "normalized_label": None, "path_contexts": [], "aliases": {}, "events": []}
        if line.startswith("#"):
            cur["id"] = int(line[1:])
        elif line.startswith("label:"):
            label = line[6:]
            n = normalize(label)
            cur["label"], cur["normalized_label"] = label, n.lower()
            cur["events"].append(("label", n.lower(), subtokens(n)))
        elif line.startswith("class:"):
            pass
        elif line.startswith("paths:"):
            mode = 1
        elif line.startswith("vars:"):
            mode = 2
        elif line.startswith("doc:"):
            pass
        elif mode == 1:
            f = line.split("\t")
            cur["path_contexts"].append((int(f[0]) + question_shift, int(f[1]), int(f[2]) + question_shift))
        elif mode == 2:
            f = line.split("\t")
            n = normalize(f[0])
            cur["aliases"][f[1]] = n.lower()
            cur["events"].append(("var", f[1], n.lower(), subtokens(n)))
    if cur is not None:
        items.append(cur)
    return items


def label_vocab(items, infer_method=True, infer_variable=False):
    """-> (names in index order, subtokens per index)"""
    stoi, subs = {}, {}
    for it in items:
        for ev in it["events"]:
            if ev[0] == "label" and infer_method:
                name, st = ev[1], ev[2]
            elif ev[0] == "var" and infer_variable and ev[1].startswith("@var_"):
                name, st = ev[2], ev[3]
            else:
                continue
            if name not in stoi:
                stoi[name] = len(stoi)
                subs[stoi[name]] = st
    names = sorted(stoi, key=stoi.get)
    return names, [subs[i] for i in range(len(names))]


def format_vectors(code_vectors, labels, names, header_items=None, ids=None, pred_labels=None, pred_scores=None):
    """-> (vector file text, result file text or None); floats printed as str(python float) of the fp32 value"""
    vec = np.asarray(code_vectors, dtype=np.float32)
    out = []
    if header_items is not None:
        out.append("{0}\t{1}\n".format(header_items, vec.shape[1]))
    res = [] if pred_labels is not None else None
    for i in range(vec.shape[0]):
        name = names[int(labels[i])]
        out.append(name + "\t" + " ".join([str(float(e)) for e in vec[i]]) + "\n")
        if res is not None:
            pred = names[int(pred_labels[i])]
            res.append("{0}\t{1}\t{2}\t{3}\t{4}\n".format(int(ids[i]), name == pred, name, pred,
                                                       float(np.float32(pred_scores[i]))))
    return "".join(out), (None if res is None else "".join(res))


def synthetic_corpus(seed, n_items=60, n_terminals=40, n_paths=50, n_vars=6):
    """-> (corpus text, terminal_idxs text, path_idxs text).  Deterministic in `seed` (numpy PCG64)."""
    rng = np.random.default_rng(seed)
    terms = ["<PAD/>", "@method_0"] + ["@var_%d" % k for k in range(n_vars)] + \
            ["tok%d" % k for k in range(n_terminals - 2 - n_vars)]
    term_txt = "".join("%d\t%s\n" % (i, t) for i, t in enumerate(terms))
    path_txt = "0\t<PAD/>\n" + "".join("%d\tName↑Decl↓P%d\n" % (i, i) for i in range(1, n_paths))
    label_pool = ["getValue", "set_value2", "toString", "HTTPServer_start", "run", "größeÄndern", "parse_JSON_2_xml",
                  "a", "İnit", "computeHash256", "__init__", "main", "getvalue", "x_1_y_2"]
    var_pool = ["index", "count_1", "resultList", "tmpVar2", "i", "bufferSize", "ÜberWert", "node"]
    nl = ["\n", "\n", "\n", "\r\n"]
    out = []
    for it in range(n_items):
        e = nl[int(rng.integers(0, len(nl)))]
        kind = int(rng.integers(0, 12))
        if kind != 0:
            out.append("#%d%s" % (it * 3 + int(rng.integers(0, 3)), e))          # (kind 0: no id line)
        vars_first = kind == 1
        n_ctx = int(rng.choice([0, 1, 3, 7, 25, 230])) if kind != 2 else 0
        n_var = int(rng.integers(0, 4))
        var_lines = []
        for k in rng.permutation(n_vars)[:n_var]:
            var_lines.append("%s\t@var_%d%s" % (var_pool[int(rng.integers(0, len(var_pool)))], int(k), e))
        if n_var and kind == 3:
            var_lines.append("other\tnot_a_var" + e)                               # alias that is not @var_*
            var_lines.append("again\t@var_%d%s" % (int(rng.integers(0, n_vars)), e))  # may overwrite an alias
        if vars_first and var_lines:
            out.append("vars:" + e); out.extend(var_lines)
        lab = label_pool[int(rng.integers(0, len(label_pool)))]
        out.append(("  label:%s \t%s" if kind == 4 else "label:%s%s") % (lab, e))
        out.append("class:some/File%d.java%s" % (it, e))
        if kind == 5:
            out.append("doc:a comment line" + e)
        if n_ctx or kind == 6:
            out.append("paths:" + e)
            for _ in range(n_ctx):
                s, p, t = int(rng.integers(1, n_terminals)), int(rng.integers(1, n_paths)), int(rng.integers(1, n_terminals))
                out.append("%d\t%d\t%d%s" % (s, p, t, e) if kind != 7 else "\t%d\t%d\t%d  %s" % (s, p, t, e))
        if not vars_first and var_lines:
            out.append("vars:" + e); out.extend(var_lines)
        out.append(e if kind != 8 else e + " \t" + e + e)                         # runs of blank lines
    if seed % 2:
        out[-1] = ""                                                               # file ends without a blank line
    return "".join(out), term_txt, path_txt
