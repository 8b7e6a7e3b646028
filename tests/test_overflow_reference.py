"""The restatement of overflowing windows (tests/overflow_ref.py) against what Hugging Face `tokenizers` 0.22.2 returned with
a truncation stride (tests/golden/hf_overflow_vectors.json.gz, made by tests/golden/make_hf_overflow_vectors.py), and, on random
corpora, the first row of every document against the oracle's hf encoding with ordinary truncation."""
import json

import numpy as np
import pytest

from oracle import oracle as orc
from overflow_ref import FIELDS, expected, load_vectors, overflow_rows, template_for, windows
from test_gpu_hf_compat import ascii_corpus

VEC, CASES = load_vectors()


def case_id(s, c):
    return f"{s['name']}-add{int(c['add_special_tokens'])}-s{c['stride']}-{(c['padding'] or {}).get('direction', 'nopad')}"


def test_windows():
    assert windows(10, 4, 2) == [(0, 4), (2, 6), (4, 8), (6, 10)]
    assert windows(5, 4, 2) == [(0, 4), (2, 5)]
    assert windows(4, 4, 3) == [(0, 4)] and windows(0, 4, 0) == [(0, 0)]
    assert windows(9, 4, 0) == [(0, 4), (4, 8), (8, 9)]
    for n in range(0, 60):
        for L in range(1, 9):
            for s in range(L):
                w = windows(n, L, s)
                assert len(w) == (1 if n <= L else 1 + -(-(n - L) // (L - s)))
                assert w[-1][1] == n and all(b - a == L for a, b in w[:-1])


def test_vectors_cover_the_cases():
    for s in VEC["suites"]:
        assert len(s["cases"]) == 18
        for c in s["cases"]:
            L = s["max_length"] - (len(sum(template_for(s, c)[:2], [])))
            assert c["stride"] in (0, L // 2, L - 1)
            n_rows = [len(d) for d in c["docs"]]
            assert n_rows[0] == 1 and max(n_rows) >= 5


@pytest.mark.parametrize("suite,case", CASES, ids=[case_id(s, c) for s, c in CASES])
def test_restatement_equals_tokenizers(suite, case):
    o = orc.OracleTokenizer.from_json(suite["tokenizer_json"])
    pre, suf, seq = template_for(suite, case)
    got = overflow_rows(o, [t.encode() for t in suite["texts"]], suite["max_length"], case["stride"], pre, suf, seq, case["padding"])
    want = expected(case)
    for k in ("doc_row_off", "row_tok_off") + FIELDS:
        assert np.array_equal(got[k], want[k]), k


@pytest.mark.parametrize("si", [0, 2, 3])
@pytest.mark.parametrize("pad", [None, {"length": 40, "pad_id": 1, "pad_type_id": 1, "direction": "left"},
                                 {"length": 24, "pad_id": 0, "pad_type_id": 0, "direction": "right"}])
def test_first_rows_are_ordinary_truncation(si, pad):
    suite = VEC["suites"][si]
    js = suite["tokenizer_json"]
    vocab = json.loads(js)["model"]["vocab"]
    words = [w for w in vocab if w.isalpha() and w.islower()][:400] + ["zzqx"]
    docs = ascii_corpus(900 + si, 200, words)
    pre, suf, seq = orc.hf_template_from_json(js)
    for max_length, stride in ((24, 0), (24, 7), (16, 16 - len(pre) - len(suf) - 1)):
        o = orc.OracleTokenizer.from_json(js)
        rows = overflow_rows(o, docs, max_length, stride, pre, suf, seq, pad)
        o.set_hf_compat(3, pre, suf, seq)
        o.truncation, o.padding = max_length, pad
        ref = o.encode_batch(docs, algo=1)
        first = rows["doc_row_off"][:-1].astype(np.int64)
        for d in range(len(docs)):
            a, b = int(rows["row_tok_off"][first[d]]), int(rows["row_tok_off"][first[d] + 1])
            ra, rb = int(ref.doc_tok_off[d]), int(ref.doc_tok_off[d + 1])
            assert np.array_equal(rows["ids"][a:b], ref.ids[ra:rb])
            assert np.array_equal(rows["offsets"][a:b], ref.offsets[ra:rb])
            assert np.array_equal(rows["type_ids"][a:b], ref.type_ids[ra:rb])
            assert np.array_equal(rows["attention_mask"][a:b], ref.attention_mask[ra:rb])
            assert np.array_equal(rows["special_tokens_mask"][a:b], ref.special_tokens_mask[ra:rb])
