"""Word ids on the GPU (TKZ_OUT_WORD_IDS), through the slice pipeline and the per-occurrence pipeline (TKZ_NO_DEDUP=1): against
what Hugging Face `tokenizers` 0.22.2 returned (tests/golden/hf_compat_word_ids.i32.gz) and, on random corpora, against the
oracle's encodings and the restated word ids of tests/word_ids_ref.py --
documents that start mid-slice, empty documents, words across slice boundaries, a slice of 1024 one-byte punctuation
pre-tokens, pre-tokens without tokens, long pre-tokens (block kernels, grid kernel, more than 2048 tokens), truncation and
padding on both sides with and without the template and document offsets, the chunked host-buffer path.  Every other array
is the same with and without the bit; the calls that cannot carry word ids are refused."""
import ctypes as C
import json
import os
import random

import numpy as np
import pytest

import tokzig_b200 as tz
from oracle import oracle as orc
from gen_util import rand_bpe_json, rand_text
from test_gpu_hf_compat import ascii_corpus, gpu_for
from test_hf_compat_oracle import CASES, VEC, expected_arrays
from word_ids_ref import hf_word_ids, restated

pytestmark = pytest.mark.gpu

MODES = ("slices", "occurrence")
ARRAYS = ("ids", "offsets", "attention_mask", "type_ids", "special_tokens_mask", "offsets_packed", "span_tokens", "wide_tokens")


def make_gpu(js, mode, chunk_bytes=None):
    env = {"TKZ_NO_DEDUP": "1" if mode == "occurrence" else "0"}
    if chunk_bytes:
        env["TKZ_CHUNK_BYTES"] = str(chunk_bytes)
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return tz.Tokenizer.from_json(js, device=0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def configure(js, t, o, hf, add, trunc, pad):
    """the same truncation / padding / hf_compat flags on the GPU tokenizer t and the oracle o; returns the number of template
    tokens before and after each document"""
    pre, suf = [], []
    if hf:
        t.set_hf_compat(hf)
        pre, suf, seq = orc.hf_template_from_json(js) if hf & tz.HF_TEMPLATE else ([], [], 0)
        if not add:
            pre, suf = [], []
        o.set_hf_compat(hf, pre, suf, seq)
    t.truncation = None if trunc is None else {"max_length": trunc}
    t.padding = pad
    o.truncation = trunc
    o.padding = pad
    return len(pre), len(suf)


def check(t, o, docs, add=True, tpl=(0, 0), outputs=tz.OUT_ALL, what="", path=None):
    """word ids equal the restated ones; every other array equal with and without the bit (and to the oracle's)"""
    got = t.encode_batch(docs, add_special_tokens=add, outputs=outputs | tz.OUT_WORD_IDS)
    if path is not None:
        assert t.stats().path == path, what
    base = t.encode_batch(docs, add_special_tokens=add, outputs=outputs)
    ref = o.encode_batch(docs, algo=1)
    want, real_ids = restated(o, docs, *tpl)
    assert np.array_equal(real_ids, ref.ids[ref.special_tokens_mask == 0]), what
    assert base.word_ids is None
    assert np.array_equal(got.doc_tok_off, ref.doc_tok_off), what
    if not np.array_equal(got.word_ids, want):
        bad = np.nonzero(got.word_ids != want)[0] if len(got.word_ids) == len(want) else [-1]
        raise AssertionError(f"{what}: word ids differ at {len(bad)} slots, first {int(bad[0])}")
    assert np.array_equal(got.doc_tok_off, base.doc_tok_off), what
    for k in ARRAYS:
        a, b = getattr(got, k), getattr(base, k)
        assert (a is None) == (b is None) and (a is None or np.array_equal(a, b)), f"{what}: {k} changed with word ids"
    assert np.array_equal(got.ids, ref.ids), what
    if got.offsets is not None:
        assert np.array_equal(got.offsets, ref.offsets), what


HF = hf_word_ids(VEC)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("suite,case", CASES, ids=[f"{s['name']}-{c['name']}" for s, c in CASES])
def test_gpu_word_ids_equal_tokenizers(suite, case, mode):
    t = gpu_for(suite, case, mode)
    r = t.encode_batch([x.encode() for x in suite["texts"]], add_special_tokens=case["add_special_tokens"], outputs=tz.OUT_ALL | tz.OUT_WORD_IDS)
    doc_off, ids, offs, attn, tids, spec = expected_arrays(case)
    assert r.doc_tok_off.tolist() == doc_off.tolist() and r.ids.tolist() == ids.tolist() and r.offsets.tolist() == offs.tolist()
    assert r.word_ids.tolist() == HF[(suite["name"], case["name"])].tolist()
    t.close()


def long_words_corpus(rng, n_docs):
    """ASCII documents of words from a..j with punctuation, empty documents, and now and then a pre-token of 256..12288 bytes
    (block kernels), above 12288 (grid kernel), or of thousands of tokens (grid-wide copy)"""
    docs = []
    for d in range(n_docs):
        if rng.random() < 0.05:
            docs.append(b"")
            continue
        parts = [rand_text(rng, list("abcdefghij"), rng.randint(1, 12), seps="", p_sep=0.0, p_unknown=0.1) for _ in range(rng.randint(0, 80))]
        if d % 37 == 5:
            parts.insert(rng.randint(0, len(parts)), b"".join(rng.choice([b"a", b"b", b"c", b"j"]) for _ in range(rng.choice([300, 3000, 9000, 14000]))))
        docs.append(b" ".join(p + (rng.choice([b",", b".", b""]) if rng.random() < 0.1 else b"") for p in parts))
    return docs


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("trunc,pad", [(None, None), (7, None), (None, {"length": 64, "pad_id": 1, "pad_type_id": 0, "direction": "right"}),
                                       (50, {"length": 60, "pad_id": 1, "pad_type_id": 1, "direction": "left"}),
                                       (None, {"length": 512, "pad_id": 0, "pad_type_id": 0, "direction": "right"})])   # (mostly padding: array-wide fill)
def test_random_bpe_corpora_with_long_and_empty_words(mode, trunc, pad):
    """BPE without unk (pre-tokens of unknown bytes only have no token) on WhitespaceSplit, reference mode"""
    rng = random.Random(7000 + (trunc or 0) + (pad or {}).get("length", 0))
    js, _ = rand_bpe_json(rng, n_merges=40, alphabet=list("abcdefghij"), unk=None, pretok="WhitespaceSplit")
    t, o = make_gpu(js, mode), orc.OracleTokenizer.from_json(js)
    configure(js, t, o, 0, True, trunc, pad)
    docs = long_words_corpus(rng, 900)
    check(t, o, docs, what=f"{mode} trunc {trunc} pad {pad}", path=0 if mode == "occurrence" else 2)
    check(t, o, docs, outputs=tz.OUT_IDS, what="ids only")
    check(t, o, docs, outputs=tz.OUT_IDS | tz.OUT_OFFSETS_PACKED | tz.OUT_IDS_U16, what="packed")
    t.close()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("si", [0, 2, 3])
@pytest.mark.parametrize("hf", [0, tz.HF_TEMPLATE, tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS, tz.HF_DOC_OFFSETS])
@pytest.mark.parametrize("trunc,pad", [(None, None), (20, {"length": 33, "pad_id": 1, "pad_type_id": 1, "direction": "left"}),
                                       (32, {"length": 40, "pad_id": 0, "pad_type_id": 0, "direction": "right"})])
def test_hf_suites_on_random_corpora(mode, si, hf, trunc, pad):
    suite = VEC["suites"][si]
    js = suite["tokenizer_json"]
    vocab = json.loads(js)["model"]["vocab"]
    words = [w for w in vocab if w.isalpha() and w.islower()][:400] + ["zzqx", "unknownword"]
    docs = ascii_corpus(300 + si, 500, words, long_word_every=40 if si == 3 else 0)
    for add in ((True, False) if hf & tz.HF_TEMPLATE else (True,)):
        t, o = make_gpu(js, mode), orc.OracleTokenizer.from_json(js)
        tpl = configure(js, t, o, hf, add, trunc, pad)
        check(t, o, docs, add=add, tpl=tpl, what=f"{suite['name']} hf {hf} add {add} trunc {trunc} pad {pad}")
        t.close()


@pytest.mark.parametrize("mode", MODES)
def test_slices_full_of_punctuation_words(mode):
    """BertPreTokenizer: every punctuation byte is its own word -> slices of 1024 words (last index 1023), documents that start
    in the middle of such runs"""
    suite = VEC["suites"][0]
    js = suite["tokenizer_json"]
    rng = random.Random(11)
    docs = [b"," * 3000, b"ka" + b"!" * 2500 + b"lo", b"", b"." * 1024, b"mi ne"] + [b"?" * rng.randint(0, 2000) + b" ka lo" for _ in range(30)]
    for hf in (0, tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS):
        t, o = make_gpu(js, mode), orc.OracleTokenizer.from_json(js)
        tpl = configure(js, t, o, hf, True, None, None)
        check(t, o, docs, tpl=tpl, what=f"hf {hf}")
        r = t.encode_batch(docs[:1], outputs=tz.OUT_IDS | tz.OUT_WORD_IDS)
        assert r.word_ids[-1 if not hf else -2] == 2999
        t.close()


@pytest.mark.parametrize("mode", MODES)
def test_host_buffer_chunks(mode):
    """the chunked host path (64 KiB chunks): documents land in several chunks, word ids need no per-chunk shift"""
    suite = VEC["suites"][0]
    js = suite["tokenizer_json"]
    vocab = json.loads(js)["model"]["vocab"]
    words = [w for w in vocab if w.isalpha() and w.islower()][:300]
    docs = ascii_corpus(77, 3000, words)
    assert sum(map(len, docs)) > 8 * 65536
    for hf, trunc, pad in ((0, None, None), (tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS, 24, {"length": 30, "pad_id": 0, "pad_type_id": 0, "direction": "left"})):
        t, o = make_gpu(js, mode, chunk_bytes=65536), orc.OracleTokenizer.from_json(js)
        tpl = configure(js, t, o, hf, True, trunc, pad)
        check(t, o, docs, tpl=tpl, what=f"chunked hf {hf}")
        t.close()


def test_refusals():
    suite = VEC["suites"][0]
    t = tz.Tokenizer.from_json(suite["tokenizer_json"], device=0)
    L, h = tz.lib(), t.context_handle()
    text, off = tz.pack_docs([b"ka lo", b"mi"])
    p = t.params(outputs=tz.OUT_ALL | tz.OUT_WORD_IDS)
    br, cr = tz.BatchResult(), tz.CompactResult()
    assert L.tkz_encode_batch(h, text.ctypes.data, off.ctypes.data, 2, C.byref(p), C.byref(br)) == tz.OK
    p.fast = 1
    assert L.tkz_encode_batch(h, text.ctypes.data, off.ctypes.data, 2, C.byref(p), C.byref(br)) == tz.ERR_INVALID_ARG
    p.fast = 0
    assert L.tkz_encode_batch_compact(h, text.ctypes.data, off.ctypes.data, 2, C.byref(p), 1, C.byref(cr)) == tz.ERR_INVALID_ARG
    pool = tz.MultiPool(t, [0])
    bounds, res = np.zeros(2, np.uint64), (tz.CompactResult * 1)()
    assert L.tkzm_encode_batch_compact(pool._h, text.ctypes.data, off.ctypes.data, 2, C.byref(p), 1, 0, bounds.ctypes.data,
                                       C.cast(res, C.c_void_p), None) == tz.ERR_INVALID_ARG
    pool.close()
    t.close()


@pytest.mark.parametrize("mode", MODES)
def test_ids_at_or_above_2_pow_22_are_refused(mode):
    """a hand-made vocabulary with sparse ids: the largest id decides"""
    for top, ok in (((1 << 22) - 1, True), (1 << 22, False)):
        js = json.dumps({"model": {"type": "BPE", "vocab": {"a": 0, "b": 1, "ab": top, "c": 5}, "merges": ["a b"]},
                         "pre_tokenizer": {"type": "WhitespaceSplit"}})
        t, o = make_gpu(js, mode), orc.OracleTokenizer.from_json(js)
        docs = [b"ab c ab", b"", b"cab ba"]
        if ok:
            check(t, o, docs, what=f"top id {top}")
        else:
            with pytest.raises(tz.TokzigError) as e:
                t.encode_batch(docs, outputs=tz.OUT_ALL | tz.OUT_WORD_IDS)
            assert e.value.code == tz.ERR_INVALID_ARG
            assert np.array_equal(t.encode_batch(docs).ids, o.encode_batch(docs).ids)
        t.close()
