"""Overflowing windows (TKZ_HF_OVERFLOW) restated on top of the oracle's hf encodings without truncation or padding, the
reference the overflow tests compare with: each document's real tokens are cut into windows of L = max_length minus the
template's tokens that overlap by `stride` (Encoding::truncate(max_length, stride, Right) of Hugging Face `tokenizers`), and
every window gets the template's special tokens and its own padding.  As in `tokenizers`, the template's sequence type id goes
to the tokens of a document's first row only: the tokens of its overflowing rows keep type id 0.  Also flattens the rows of
hf_overflow_vectors.json.gz."""
import gzip
import json
import os

import numpy as np

from oracle import oracle as orc
from word_ids_ref import NONE, restated

HERE = os.path.dirname(os.path.abspath(__file__))
FIELDS = ("ids", "type_ids", "offsets", "attention_mask", "special_tokens_mask", "word_ids")


def windows(n, L, stride):
    """[(start, stop)] of a document of n tokens: one window when n <= L, else windows k * (L - stride) until one reaches n"""
    if n <= L:
        return [(0, n)]
    step, out = L - stride, []
    while not out or out[-1][1] < n:
        a = len(out) * step
        out.append((a, min(a + L, n)))
    return out


def flatten(rows_per_doc):
    """{doc_row_off, row_tok_off, doc_tok_off, ids, type_ids, offsets (n, 2), attention_mask, special_tokens_mask, word_ids}
    from a list (documents) of lists (rows) of per-row dicts"""
    doc_row_off, row_tok_off, cols = [0], [0], {f: [] for f in FIELDS}
    for rows in rows_per_doc:
        for r in rows:
            for f in FIELDS:
                cols[f] += r[f]
            row_tok_off.append(len(cols["ids"]))
        doc_row_off.append(len(row_tok_off) - 1)
    out = {f: np.array(v, np.uint32) for f, v in cols.items()}
    out["offsets"] = out["offsets"].reshape(-1, 2)
    out["doc_row_off"] = np.array(doc_row_off, np.uint64)
    out["row_tok_off"] = np.array(row_tok_off, np.uint64)
    out["doc_tok_off"] = out["row_tok_off"][out["doc_row_off"].astype(np.int64)]
    return out


def overflow_rows(o: orc.OracleTokenizer, docs, max_length, stride, prefix=(), suffix=(), seq_type=0, padding=None, doc_offsets=True,
                  word_ids=True, threads=1):
    """the rows of docs as flat arrays (see flatten).  prefix / suffix = [(id, type id)] of the template's special tokens (empty:
    reference mode, or a template encoded without add_special_tokens); padding = {"length", "pad_id", "pad_type_id",
    "direction"} or None; word_ids=False leaves every word id NONE (faster on large corpora).  Sets o's hf mode and clears its
    truncation / padding."""
    o.set_hf_compat(1 | (2 if doc_offsets else 0), list(prefix), list(suffix), seq_type)
    o.truncation, o.padding = None, None
    enc = o.encode_batch(docs, algo=1, threads=threads)
    wid = restated(o, docs, len(prefix), len(suffix))[0] if word_ids else np.full(len(enc.ids), NONE, np.uint32)
    L = max_length - len(prefix) - len(suffix)
    assert 0 <= stride < L
    out = []
    for d in range(len(docs)):
        a, b = int(enc.doc_tok_off[d]), int(enc.doc_tok_off[d + 1])
        real = enc.special_tokens_mask[a:b] == 0
        ids, offs, w = enc.ids[a:b][real].tolist(), enc.offsets[a:b][real].tolist(), wid[a:b][real].tolist()
        rows = []
        for k, (s, e) in enumerate(windows(len(ids), L, stride)):
            n = e - s
            r = {"ids": [p[0] for p in prefix] + ids[s:e] + [q[0] for q in suffix],
                 "type_ids": [p[1] for p in prefix] + [seq_type if k == 0 else 0] * n + [q[1] for q in suffix],
                 "offsets": [[0, 0]] * len(prefix) + offs[s:e] + [[0, 0]] * len(suffix),
                 "attention_mask": [1] * (len(prefix) + n + len(suffix)),
                 "special_tokens_mask": [1] * len(prefix) + [0] * n + [1] * len(suffix),
                 "word_ids": [NONE] * len(prefix) + w[s:e] + [NONE] * len(suffix)}
            npad = padding["length"] - len(r["ids"]) if padding is not None else 0
            if npad > 0:
                fill = {"ids": padding["pad_id"], "type_ids": padding["pad_type_id"], "offsets": [0, 0], "attention_mask": 0,
                        "special_tokens_mask": 1, "word_ids": NONE}
                for f in FIELDS:
                    r[f] = [fill[f]] * npad + r[f] if padding.get("direction") == "left" else r[f] + [fill[f]] * npad
            rows.append(r)
        out.append(rows)
    return flatten(out)


def load_vectors():
    """(hf_overflow_vectors.json.gz with each suite's tokenizer_json from hf_compat_vectors.json, [(suite, case)])"""
    vec = json.load(gzip.open(os.path.join(HERE, "golden", "hf_overflow_vectors.json.gz")))
    compat = {s["name"]: s for s in json.load(open(os.path.join(HERE, "golden", "hf_compat_vectors.json")))["suites"]}
    for s in vec["suites"]:
        s["tokenizer_json"] = compat[s["name"]]["tokenizer_json"]
    return vec, [(s, c) for s in vec["suites"] for c in s["cases"]]


def expected(case):
    """a vector case's rows as flat arrays (word ids: -1 -> NONE)"""
    rows = [[{f: ([NONE if x < 0 else x for x in r[f]] if f == "word_ids" else r[f]) for f in FIELDS} for r in d] for d in case["docs"]]
    return flatten(rows)


def template_for(suite, case):
    """(prefix, suffix, seq_type) the case encodes with: the suite's template, its special tokens only with add_special_tokens"""
    pre, suf, seq = orc.hf_template_from_json(suite["tokenizer_json"])
    return (pre, suf, seq) if case["add_special_tokens"] else ([], [], seq)
