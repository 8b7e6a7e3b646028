"""hf_compat on the GPU (SURVEY.md section 8(f) row 4; beyond the reference, opt-in): the CUDA path with TKZ_HF_TEMPLATE |
TKZ_HF_DOC_OFFSETS against (a) what Hugging Face `tokenizers` 0.22.2 returned for the same tokenizer.json and texts
(tests/golden/hf_compat_vectors.json) and (b) the oracle's hf mode on larger random ASCII corpora.  Everything goes through the
C ABI (tkzh_set_hf_compat + tkzh_encode_batch -> tkz_encode_params.hf_flags / tpl_*)."""
import json
import os
import random

import numpy as np
import pytest

import tokzig_b200 as tz
from oracle import oracle as orc
from test_hf_compat_oracle import CASES, VEC, expected_arrays, oracle_for

pytestmark = pytest.mark.gpu


MODES = ("slices", "occurrence")


def gpu_for(suite, case, mode="slices"):
    """both device pipelines serve the mode: the slice pipeline (default) and the per-occurrence pipeline (TKZ_NO_DEDUP=1)"""
    os.environ["TKZ_NO_DEDUP"] = "1" if mode == "occurrence" else "0"
    try:
        t = tz.Tokenizer.from_json(suite["tokenizer_json"], device=0)
    finally:
        os.environ["TKZ_NO_DEDUP"] = "0"
    assert t.set_hf_compat(tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS)
    t.truncation = None if case["truncation"] is None else {"max_length": case["truncation"]}
    t.padding = case["padding"]
    return t


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("suite,case", CASES, ids=[f"{s['name']}-{c['name']}" for s, c in CASES])
def test_gpu_hf_mode_equals_tokenizers(suite, case, mode):
    t = gpu_for(suite, case, mode)
    r = t.encode_batch([x.encode() for x in suite["texts"]], add_special_tokens=case["add_special_tokens"])
    doc_off, ids, offs, attn, tids, spec = expected_arrays(case)
    assert r.doc_tok_off.tolist() == doc_off.tolist()
    assert r.ids.tolist() == ids.tolist()
    assert r.offsets.tolist() == offs.tolist()
    assert r.attention_mask.tolist() == attn.tolist()
    assert r.type_ids.tolist() == tids.tolist()
    assert r.special_tokens_mask.tolist() == spec.tolist()
    t.close()


def ascii_corpus(seed, n_docs, words, long_word_every=0):
    rng = random.Random(seed)
    docs = []
    for d in range(n_docs):
        parts = []
        for _ in range(rng.randint(0, 60)):
            w = rng.choice(words)
            if rng.random() < 0.2:
                w = w.upper()
            if rng.random() < 0.1:
                w += rng.choice(",.;!?")
            parts.append(w)
        if long_word_every and d % long_word_every == 1:
            parts.insert(len(parts) // 2, "".join(rng.choice("abcdefghij") for _ in range(rng.choice([300, 3000, 9000]))))
        docs.append((" " if rng.random() < 0.8 else "\n").join(parts).encode())
    return docs


@pytest.mark.parametrize("si", [0, 2, 3])
@pytest.mark.parametrize("trunc,pad", [(None, None), (32, {"length": 40, "pad_id": 0, "pad_type_id": 0, "direction": "right"}),
                                       (20, {"length": 33, "pad_id": 1, "pad_type_id": 1, "direction": "left"}),
                                       (None, {"length": 256, "pad_id": 1, "pad_type_id": 1, "direction": "left"})])   # (mostly padding: whole-array fill)
@pytest.mark.parametrize("mode", MODES)
def test_gpu_hf_mode_equals_oracle_on_random_corpora(si, trunc, pad, mode):
    suite = VEC["suites"][si]
    js = suite["tokenizer_json"]
    vocab = json.loads(js)["model"]["vocab"]
    words = [w for w in vocab if w.isalpha() and w.islower()][:400] + ["zzqx", "unknownword"]
    docs = ascii_corpus(100 + si, 700, words, long_word_every=50 if si == 3 else 0)      # (BPE: words of thousands of tokens -> the grid-wide copy)
    for add in (True, False):
        case = {"add_special_tokens": add, "truncation": trunc, "padding": pad}
        o = oracle_for(suite, case)
        t = gpu_for(suite, case, mode)
        ref = o.encode_batch(docs, algo=1)
        got = t.encode_batch(docs, add_special_tokens=add)
        assert t.stats().path == (0 if mode == "occurrence" else 2)
        assert np.array_equal(got.doc_tok_off, ref.doc_tok_off)
        assert np.array_equal(got.ids, ref.ids)
        assert np.array_equal(got.offsets, ref.offsets)
        assert np.array_equal(got.attention_mask, ref.attention_mask)
        assert np.array_equal(got.type_ids, ref.type_ids)
        assert np.array_equal(got.special_tokens_mask, ref.special_tokens_mask)
        t.close()


@pytest.mark.parametrize("mode", MODES)
def test_span_tokens_carry_the_template(mode):
    suite = VEC["suites"][2]                                      # [CLS]:0 [MASK]:1 $A:1 [SEP]:1 [SEP]:0
    case = {"add_special_tokens": True, "truncation": 8, "padding": {"length": 12, "pad_id": 0, "pad_type_id": 0, "direction": "right"}}
    t = gpu_for(suite, case, mode)
    r = t.encode_batch([b"ka lo mi", b""], outputs=tz.OUT_ALL | tz.OUT_SPAN_TOKENS)
    sp = r.span_tokens.reshape(-1, 4)
    assert len(sp) == 24
    for k in range(24):
        sid, s, e, tf = (int(x) for x in sp[k])
        assert sid == int(r.ids[k]) and (s, e) == tuple(int(x) for x in r.offsets[k])
        assert (tf & 0xFF) == int(r.type_ids[k])
        flags = tf >> 8
        if r.attention_mask[k] == 0:
            assert flags == 0x04                                  # SpanToken.initPadding
        elif r.special_tokens_mask[k]:
            assert flags == 0x01                                  # SpanToken.initSpecial
        else:
            assert flags == 0
    t.close()


def test_mode_off_is_the_reference_and_the_other_entry_points_refuse_the_mode():
    suite = VEC["suites"][0]
    t = tz.Tokenizer.from_json(suite["tokenizer_json"], device=0)
    o = orc.OracleTokenizer.from_json(suite["tokenizer_json"])
    docs = [x.encode() for x in suite["texts"]]
    ref = o.encode_batch(docs)
    for add in (True, False):                                     # the reference: add_special_tokens changes nothing
        got = t.encode_batch(docs, add_special_tokens=add)
        assert np.array_equal(got.ids, ref.ids) and np.array_equal(got.offsets, ref.offsets) and np.array_equal(got.special_tokens_mask, ref.special_tokens_mask)
    import ctypes as C
    text, off = tz.pack_docs(docs)
    L, h = tz.lib(), t.context_handle()
    p = t.params()
    p.hf_flags = tz.HF_DOC_OFFSETS
    cr, br = tz.CompactResult(), tz.BatchResult()
    assert L.tkz_encode_batch_compact(h, text.ctypes.data, off.ctypes.data, len(off) - 1, C.byref(p), 1, C.byref(cr)) == tz.ERR_INVALID_ARG
    p.fast = 1
    assert L.tkz_encode_batch(h, text.ctypes.data, off.ctypes.data, len(off) - 1, C.byref(p), C.byref(br)) == tz.ERR_INVALID_ARG
    p.fast, p.hf_flags = 0, 8
    assert L.tkz_encode_batch(h, text.ctypes.data, off.ctypes.data, len(off) - 1, C.byref(p), C.byref(br)) == tz.ERR_INVALID_ARG
    p.hf_flags = tz.HF_DOC_OFFSETS
    assert L.tkz_encode_batch(h, text.ctypes.data, off.ctypes.data, len(off) - 1, C.byref(p), C.byref(br)) == tz.OK
    t.close()
