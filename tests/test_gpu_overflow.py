"""Overflowing windows on the GPU (TKZ_HF_OVERFLOW), through the slice pipeline and the per-occurrence pipeline (TKZ_NO_DEDUP=1):
against what Hugging Face `tokenizers` 0.22.2 returned with a truncation stride (tests/golden/hf_overflow_vectors.json.gz) and, on
random corpora, against the restated rows of tests/overflow_ref.py -- empty documents and documents of exactly L and L + 1
tokens, stride 0 up to L - 1, padding on both sides (also mostly padding: the array-wide fill), pre-tokens for the block and
grid kernels, word ids and document offsets carried into every window, the packed-offset fallback, the device-resident call
and the chunked host path.  A call without the flag is unchanged whatever its stride; the calls the flag cannot serve are
refused."""
import ctypes as C
import json
import random

import numpy as np
import pytest

import tokzig_b200 as tz
from oracle import oracle as orc
from gen_util import rand_bpe_json
from overflow_ref import FIELDS, expected, load_vectors, overflow_rows
from test_gpu_hf_compat import ascii_corpus
from test_gpu_word_ids import long_words_corpus, make_gpu

pytestmark = pytest.mark.gpu

MODES = ("slices", "occurrence")
OUT = tz.OUT_ALL | tz.OUT_WORD_IDS
VEC, CASES = load_vectors()
CSR = ("doc_row_off", "row_tok_off", "doc_tok_off")


def assert_rows(r, want, what, fields=FIELDS):
    for k in CSR + tuple(fields):
        got = getattr(r, k) if hasattr(r, k) else r[k]
        assert got is not None and got.shape == want[k].shape and np.array_equal(got, want[k]), f"{what}: {k}"


def configure(t, js, hf, add, max_length, stride, pad):
    """hf_compat flags + overflow, truncation with stride and padding on the GPU tokenizer; returns the (prefix, suffix, seq_type)
    the restatement needs"""
    t.set_hf_compat(hf | tz.HF_OVERFLOW)
    t.truncation = {"max_length": max_length, "stride": stride}
    t.padding = pad
    pre, suf, seq = orc.hf_template_from_json(js) if hf & tz.HF_TEMPLATE else ([], [], 0)
    return (pre, suf, seq) if add else ([], [], seq)


def case_id(s, c):
    return f"{s['name']}-add{int(c['add_special_tokens'])}-s{c['stride']}-{(c['padding'] or {}).get('direction', 'nopad')}"


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("suite,case", CASES, ids=[case_id(s, c) for s, c in CASES])
def test_gpu_overflow_equals_tokenizers(suite, case, mode):
    js = suite["tokenizer_json"]
    t = make_gpu(js, mode)
    configure(t, js, tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS, case["add_special_tokens"], suite["max_length"], case["stride"], case["padding"])
    r = t.encode_batch([x.encode() for x in suite["texts"]], add_special_tokens=case["add_special_tokens"], outputs=OUT)
    want = expected(case)
    assert_rows(r, want, case_id(suite, case))
    assert r.overflow_to_sample_mapping.tolist() == [d for d, rows in enumerate(case["docs"]) for _ in rows]
    t.close()


def exact_length_docs(o, docs, counts):
    """word prefixes of docs whose real token counts are exactly those in `counts` (one each, where one exists)"""
    out = []
    for doc in docs:
        words = doc.split(b" ")
        pre = [b" ".join(words[:i]) for i in range(len(words) + 1)]
        enc = o.encode_batch(pre, algo=1)
        n = [int(((enc.special_tokens_mask[a:b]) == 0).sum()) for a, b in zip(enc.doc_tok_off[:-1], enc.doc_tok_off[1:])]
        for c in counts:
            if c in n:
                out.append(pre[n.index(c)])
    return out


def check_random(t, o, docs, js, hf, max_length, stride, pad, what):
    for add in ((True, False) if hf & tz.HF_TEMPLATE else (True,)):
        pre, suf, seq = configure(t, js, hf, add, max_length, stride, pad)
        want = overflow_rows(o, docs, max_length, stride, pre, suf, seq, pad, doc_offsets=bool(hf & tz.HF_DOC_OFFSETS))
        r = t.encode_batch(docs, add_special_tokens=add, outputs=OUT)
        assert_rows(r, want, f"{what} add {add}")
        r = t.encode_batch(docs, add_special_tokens=add, outputs=tz.OUT_IDS)
        assert_rows(r, want, f"{what} add {add} ids only", fields=("ids",))
        assert r.offsets is None and r.word_ids is None and r.attention_mask is None
        # the one-u16 offsets fall back to 32-bit pairs; u16 ids stay
        r = t.encode_batch(docs, add_special_tokens=add, outputs=tz.OUT_IDS | tz.OUT_OFFSETS_PACKED | tz.OUT_IDS_U16)
        assert r.offsets_packed is None and r.offsets is not None
        assert_rows(r, want, f"{what} add {add} packed", fields=("ids", "offsets"))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("si", [0, 2, 3])
@pytest.mark.parametrize("hf", [tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS, tz.HF_TEMPLATE, 0])
@pytest.mark.parametrize("max_length,stride,pad", [(24, "mid", None),
                                                   (16, "max", {"length": 20, "pad_id": 1, "pad_type_id": 1, "direction": "left"}),
                                                   (32, "zero", {"length": 32, "pad_id": 0, "pad_type_id": 0, "direction": "right"}),
                                                   (12, "max", {"length": 256, "pad_id": 0, "pad_type_id": 0, "direction": "right"})])
def test_random_corpora(mode, si, hf, max_length, stride, pad):
    suite = VEC["suites"][si]
    js = suite["tokenizer_json"]
    vocab = json.loads(js)["model"]["vocab"]
    words = [w for w in vocab if w.isalpha() and w.islower()][:400] + ["zzqx", "unknownword"]
    docs = ascii_corpus(500 + si, 400, words, long_word_every=50 if si == 3 else 0)
    o = orc.OracleTokenizer.from_json(js)
    n_tpl = sum(map(len, orc.hf_template_from_json(js)[:2])) if hf & tz.HF_TEMPLATE else 0
    L = max_length - n_tpl
    docs += [b""] + exact_length_docs(o, docs[:40], (L, L + 1, max_length, max_length + 1))
    s = {"zero": 0, "mid": L // 2, "max": L - 1}[stride]
    t = make_gpu(js, mode)
    check_random(t, o, docs, js, hf, max_length, s, pad, f"{suite['name']} hf {hf} L {L} stride {s} pad {pad}")
    t.close()


@pytest.mark.parametrize("mode", MODES)
def test_long_pre_tokens(mode):
    """BPE on WhitespaceSplit, reference mode: pre-tokens of 256..12288 bytes (block kernels), above 12288 (grid kernel) and of
    thousands of tokens (grid-wide copy) end up in windows of their own and across them"""
    rng = random.Random(8100)
    js, _ = rand_bpe_json(rng, n_merges=40, alphabet=list("abcdefghij"), unk=None, pretok="WhitespaceSplit")
    docs = long_words_corpus(rng, 600)
    t, o = make_gpu(js, mode), orc.OracleTokenizer.from_json(js)
    for max_length, stride, pad in ((64, 63, None), (300, 100, {"length": 310, "pad_id": 1, "pad_type_id": 0, "direction": "left"})):
        check_random(t, o, docs, js, 0, max_length, stride, pad, f"long words L {max_length} stride {stride}")
    t.close()


def cudart():
    tz.lib()                                  # (loads the CUDA runtime the library links)
    rt = C.CDLL("libcudart.so.12")
    rt.cudaMemcpy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
    return rt


def d2h(rt, ptr, n, dtype):
    a = np.zeros(n, dtype)
    if n:
        assert rt.cudaMemcpy(a.ctypes.data, ptr, a.nbytes, 2) == 0
    return a


@pytest.mark.parametrize("mode", MODES)
def test_device_call(mode):
    import torch
    suite = VEC["suites"][0]
    js = suite["tokenizer_json"]
    words = [w for w in json.loads(js)["model"]["vocab"] if w.isalpha() and w.islower()][:300]
    docs = ascii_corpus(61, 700, words)
    t, o = make_gpu(js, mode), orc.OracleTokenizer.from_json(js)
    pad = {"length": 30, "pad_id": 0, "pad_type_id": 1, "direction": "left"}
    pre, suf, seq = configure(t, js, tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS, True, 28, 9, pad)
    want = overflow_rows(o, docs, 28, 9, pre, suf, seq, pad)
    p = t.params(outputs=OUT)
    p.hf_flags = tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS | tz.HF_OVERFLOW
    p.tpl_n_prefix, p.tpl_n_suffix, p.tpl_seq_type = len(pre), len(suf), seq
    for i, (a, b) in enumerate(pre):
        p.tpl_prefix_id[i], p.tpl_prefix_type[i] = a, b
    for i, (a, b) in enumerate(suf):
        p.tpl_suffix_id[i], p.tpl_suffix_type[i] = a, b
    text, off = tz.pack_docs(docs)
    d_text, d_off = torch.from_numpy(text).cuda(), torch.from_numpy(off.astype(np.int64)).cuda()
    r = tz.BatchResult()
    L = tz.lib()
    assert L.tkz_encode_batch_device(t.context_handle(), C.c_void_p(d_text.data_ptr()), C.c_void_p(d_off.data_ptr()), len(docs), len(text),
                                     C.byref(p), C.byref(r)) == tz.OK
    rt = cudart()
    T, R = int(r.n_tokens), int(r.n_rows)
    assert R == len(want["row_tok_off"]) - 1 and T == int(want["row_tok_off"][-1])
    got = {"doc_row_off": d2h(rt, r.doc_row_off, len(docs) + 1, np.uint64), "row_tok_off": d2h(rt, r.row_tok_off, R + 1, np.uint64),
           "doc_tok_off": d2h(rt, r.doc_tok_off, len(docs) + 1, np.uint64), "offsets": d2h(rt, r.offsets, 2 * T, np.uint32).reshape(-1, 2)}
    for k, f in (("ids", "ids"), ("type_ids", "type_ids"), ("attention_mask", "attention_mask"), ("special_tokens_mask", "special_tokens_mask"),
                 ("word_ids", "word_ids")):
        got[k] = d2h(rt, getattr(r, f), T, np.uint32)
    assert_rows(got, want, "device call")
    t.close()


@pytest.mark.parametrize("mode", MODES)
def test_host_buffer_chunks(mode):
    """the chunked host path (64 KiB chunks): row offsets and document-row offsets continue across chunks"""
    suite = VEC["suites"][3]
    js = suite["tokenizer_json"]
    words = [w for w in json.loads(js)["model"]["vocab"] if w.isalpha() and w.islower()][:300]
    docs = ascii_corpus(78, 4500, words)
    assert sum(map(len, docs)) > 8 * 65536
    o = orc.OracleTokenizer.from_json(js)
    for hf, max_length, stride, pad in ((tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS, 20, 5, {"length": 24, "pad_id": 0, "pad_type_id": 0, "direction": "left"}),
                                        (0, 16, 15, None)):
        t = make_gpu(js, mode, chunk_bytes=65536)
        pre, suf, seq = configure(t, js, hf, True, max_length, stride, pad)
        want = overflow_rows(o, docs, max_length, stride, pre, suf, seq, pad, doc_offsets=bool(hf & tz.HF_DOC_OFFSETS))
        assert_rows(t.encode_batch(docs, outputs=OUT), want, f"chunked hf {hf}")
        t.close()


def test_without_the_flag_stride_changes_nothing():
    suite = VEC["suites"][0]
    js = suite["tokenizer_json"]
    docs = [x.encode() for x in suite["texts"]] * 3
    t = make_gpu(js, "slices")
    t.set_hf_compat(tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS)
    t.padding = {"length": 16, "pad_id": 0, "pad_type_id": 0, "direction": "right"}
    for outputs in (OUT, tz.OUT_IDS | tz.OUT_OFFSETS_PACKED | tz.OUT_IDS_U16):
        t.truncation = {"max_length": 12}
        base = t.encode_batch(docs, outputs=outputs)
        t.truncation = {"max_length": 12, "stride": 5}
        got = t.encode_batch(docs, outputs=outputs)
        for k in ("doc_tok_off", "ids", "offsets", "attention_mask", "type_ids", "special_tokens_mask", "offsets_packed", "word_ids"):
            a, b = getattr(got, k), getattr(base, k)
            assert (a is None) == (b is None) and (a is None or np.array_equal(a, b)), k
        assert got.row_tok_off is None and got.doc_row_off is None and got.overflow_to_sample_mapping is None
    text, off = tz.pack_docs(docs)
    r = tz.BatchResult()
    p = t.params(outputs=OUT)
    p.hf_flags = tz.HF_DOC_OFFSETS
    assert tz.lib().tkz_encode_batch(t.context_handle(), text.ctypes.data, off.ctypes.data, len(docs), C.byref(p), C.byref(r)) == tz.OK
    assert r.n_rows == 0 and not r.row_tok_off and not r.doc_row_off
    t.close()


def test_refusals():
    suite = VEC["suites"][0]
    t = tz.Tokenizer.from_json(suite["tokenizer_json"], device=0)
    L, h = tz.lib(), t.context_handle()
    text, off = tz.pack_docs([b"ka lo mi ne", b"mi"])

    def call(**kw):
        p = tz.EncodeParams(has_truncation=1, max_length=6, stride=2, outputs=OUT, hf_flags=tz.HF_TEMPLATE | tz.HF_OVERFLOW,
                            tpl_n_prefix=1, tpl_n_suffix=1)
        p.tpl_prefix_id[0], p.tpl_suffix_id[0] = 2, 3
        for k, v in kw.items():
            setattr(p, k, v)
        return L.tkz_encode_batch(h, text.ctypes.data, off.ctypes.data, 2, C.byref(p), C.byref(tz.BatchResult())), p

    assert call()[0] == tz.OK
    assert call(stride=3)[0] == tz.OK                                   # L = 6 - 2 = 4: stride 3 is the largest
    assert call(stride=4)[0] == tz.ERR_INVALID_ARG
    assert call(max_length=2, stride=0)[0] == tz.ERR_INVALID_ARG        # L = 0
    assert call(has_truncation=0)[0] == tz.ERR_INVALID_ARG
    assert call(fast=1)[0] == tz.ERR_INVALID_ARG
    assert call(outputs=tz.OUT_ALL | tz.OUT_SPAN_TOKENS)[0] == tz.ERR_INVALID_ARG
    _, p = call()
    assert L.tkz_encode_batch_compact(h, text.ctypes.data, off.ctypes.data, 2, C.byref(p), 1, C.byref(tz.CompactResult())) == tz.ERR_INVALID_ARG
    pool = tz.MultiPool(t, [0])
    bounds, res = np.zeros(2, np.uint64), (tz.CompactResult * 1)()
    assert L.tkzm_encode_batch_compact(pool._h, text.ctypes.data, off.ctypes.data, 2, C.byref(p), 1, 0, bounds.ctypes.data,
                                       C.cast(res, C.c_void_p), None) == tz.ERR_INVALID_ARG
    pool.close()
    t.close()
