"""Word ids restated on top of the oracle's stage probes, the reference the word-id tests compare with: normalise a document,
pre-tokenize it, tokenize every pre-token on its own (a tokenizer with the same model and no normalizer / pre-tokenizer: the
model is a pure function of the normalised pre-token), and give each token the ordinal of its pre-token.  Then the
encoding's layout as the oracle builds it: truncation to max_length minus the template's tokens, the template's special
tokens and the padding slots with no word (0xFFFFFFFF).  Also loads the Hugging Face word ids of the hf_compat vectors."""
import gzip
import os

import numpy as np

from oracle import oracle as orc

NONE = 0xFFFFFFFF
HERE = os.path.dirname(os.path.abspath(__file__))


def restated(t: orc.OracleTokenizer, docs, n_pre=0, n_suf=0):
    """(word ids, ids of the real tokens) of t.encode_batch(docs) under t's truncation / padding and a template of n_pre +
    n_suf special tokens (0 / 0: reference mode, or a template encoded without add_special_tokens)"""
    m = orc.OracleTokenizer(t.cfg)
    m.normalizers, m.pretokenizers = [], None
    pieces, owner = [], []
    for d, doc in enumerate(docs):
        for q, piece in enumerate(t.pre_tokenize(t.normalize(doc))):
            pieces.append(piece)
            owner.append((d, q))
    enc = m.encode_batch(pieces, algo=1)
    off = enc.doc_tok_off.astype(np.int64)
    words, ids = [[] for _ in docs], [[] for _ in docs]
    for k, (d, q) in enumerate(owner):
        words[d] += [q] * int(off[k + 1] - off[k])
        ids[d] += enc.ids[off[k]:off[k + 1]].tolist()
    out_w, out_ids = [], []
    for w, i in zip(words, ids):
        if t.truncation is not None:
            keep = max(t.truncation - n_pre - n_suf, 0)
            w, i = w[:keep], i[:keep]
        out_ids += i
        w = [NONE] * n_pre + w + [NONE] * n_suf
        if t.padding is not None and t.padding.get("length") is not None and len(w) < t.padding["length"]:
            pad = [NONE] * (t.padding["length"] - len(w))
            w = pad + w if t.padding.get("direction") == "left" else w + pad
        out_w += w
    return np.array(out_w, np.uint32), np.array(out_ids, np.uint32)


def hf_word_ids(vec):
    """{(suite name, case name): u32 word ids of all its encodings back to back} from tests/golden/hf_compat_word_ids.i32.gz
    (made by tests/golden/make_hf_word_ids.py from the same encodings as hf_compat_vectors.json)"""
    flat = np.frombuffer(gzip.open(os.path.join(HERE, "golden", "hf_compat_word_ids.i32.gz")).read(), "<i4").astype(np.int64)
    out, k = {}, 0
    for s in vec["suites"]:
        for c in s["cases"]:
            n = sum(len(e["ids"]) for e in c["encodings"])
            out[(s["name"], c["name"])] = np.where(flat[k:k + n] < 0, NONE, flat[k:k + n]).astype(np.uint32)
            k += n
    assert k == len(flat)
    return out
