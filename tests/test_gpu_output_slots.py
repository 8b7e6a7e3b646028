"""Every slot of every output form is written, whatever the output buffers held before the call.  The device-resident call
(tkz_encode_batch_device) runs once, every per-slot value array it returned is filled with the byte 0xA5, and the same call
runs again into the same buffers; what it returns is then compared in full with the CPU oracle.  An unwritten slot reads as
a plausible wrong value: 0xA5A5 as packed offsets is (165, 165), not the 0xFFFF of a wide token; as a u32 it is neither 0,
1 nor 0xFFFFFFFF.  The CSR arrays and the wide-token side list are compared but never poisoned: kernels read them as indices.

One context per (model, pipeline) goes through the whole case table -- output masks x hf_compat flags x truncation / padding,
both sides of the whole-array padding fill -- so that what one call leaves behind is in the buffers of the next.  The models:
a WordPiece and a BPE suite of hf_compat_vectors.json, a BPE with ids just below 65536 and one with ids above it.  Also: the
host-buffer call into the same (poisoned) buffers, overflowing windows, the FastTokenizer mode through the device call, text
at every 16-byte misalignment (the staging copy, with and without the byte-dropping normalizer), and a caller-owned stream
whose input copies are still in flight when the call starts."""
import ctypes as C
import functools
import json
import os
import random

import numpy as np
import pytest

import tokzig_b200 as tz
from oracle import oracle as orc
from overflow_ref import overflow_rows
from test_gpu_hf_compat import ascii_corpus
from test_gpu_overflow import configure as configure_overflow
from test_gpu_overflow import cudart, d2h, exact_length_docs
from test_gpu_token_records import SMALL_BPE
from test_gpu_word_ids import configure
from test_hf_compat_oracle import VEC
from word_ids_ref import restated

POISON = 0xA5
OUT_PACKED, OUT_U16, OUT_SPAN, OUT_WID = tz.OUT_OFFSETS_PACKED, tz.OUT_IDS_U16, tz.OUT_SPAN_TOKENS, tz.OUT_WORD_IDS
MASKS = (tz.OUT_IDS, tz.OUT_IDS | OUT_U16, tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION, tz.OUT_IDS | OUT_PACKED,
         tz.OUT_IDS | OUT_U16 | OUT_PACKED, tz.OUT_ALL, tz.OUT_ALL | OUT_SPAN, tz.OUT_ALL | OUT_WID,
         tz.OUT_ALL | OUT_U16 | OUT_PACKED | OUT_SPAN | OUT_WID)
HOST_MASKS = (tz.OUT_IDS | OUT_PACKED, tz.OUT_ALL | OUT_U16 | OUT_PACKED | OUT_SPAN | OUT_WID)   # also through tkz_encode_batch
# (name, hf_flags, add_special_tokens)
HF = (("ref", 0, True), ("tpl", tz.HF_TEMPLATE, True), ("tpl_noadd", tz.HF_TEMPLATE, False),
      ("tpl_doc", tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS, True), ("doc", tz.HF_DOC_OFFSETS, True))
# truncation max_length, padding; "dominates": so many padding slots (T >= 2 x real tokens) that the arrays are filled whole first
TP = {"none": (None, None),
      "trunc": (16, None),
      "pad_right": (None, {"length": 40, "pad_id": 1, "pad_type_id": 1, "direction": "right"}),
      "pad_left": (None, {"length": 40, "pad_id": 0, "pad_type_id": 0, "direction": "left"}),
      "trunc_pad_left": (20, {"length": 24, "pad_id": 1, "pad_type_id": 1, "direction": "left"}),
      "pad_dominates": (None, {"length": 256, "pad_id": 0, "pad_type_id": 1, "direction": "right"}),
      "trunc_pad_dominates_left": (16, {"length": 128, "pad_id": 1, "pad_type_id": 0, "direction": "left"})}
PIPELINES = {"slices": {}, "slices_wide_records": {"TKZ_TOK_RECORD": "wide"}, "slices_lut": {"TKZ_CLASSIFY": "lut"},
             "occurrence": {"TKZ_NO_DEDUP": "1"}}
ENV_KEYS = ("TKZ_NO_DEDUP", "TKZ_TOK_RECORD", "TKZ_CLASSIFY")


def with_template(js, cls_id, sep_id):
    """js with a TemplateProcessing post_processor  [CLS]:0 $A:1 [SEP]:1"""
    j = json.loads(js)
    j["post_processor"] = {"type": "TemplateProcessing",
                           "single": [{"SpecialToken": {"id": "[CLS]", "type_id": 0}}, {"Sequence": {"id": "A", "type_id": 1}},
                                      {"SpecialToken": {"id": "[SEP]", "type_id": 1}}],
                           "pair": [], "special_tokens": {"[CLS]": {"id": "[CLS]", "ids": [cls_id], "tokens": ["[CLS]"]},
                                                          "[SEP]": {"id": "[SEP]", "ids": [sep_id], "tokens": ["[SEP]"]}}}
    return json.dumps(j)


_WIDE = json.loads(SMALL_BPE)
_WIDE["model"]["vocab"] = {**{c: 65536 + i for i, c in enumerate("abcdefgh")}, "ab": 3, "cd": 1000000, "abcd": 65535, "ee": 100000}
MODELS = {
    "wordpiece": VEC["suites"][2]["tokenizer_json"],            # [CLS]:0 [MASK]:1 $A:1 [SEP]:1 [SEP]:0, BertPreTokenizer
    "bpe": VEC["suites"][3]["tokenizer_json"],                  # <s> $A </s>, WhitespaceSplit, <unk>
    "bpe16": with_template(SMALL_BPE, 65535, 65534),            # ids up to 65535 (u16 ids, narrow token records)
    "bpe_wide": with_template(json.dumps(_WIDE), 1000001, 70000),   # ids above 65535: TKZ_OUT_IDS_U16 is ignored
}
IDS16_OK = {"wordpiece": True, "bpe": True, "bpe16": True, "bpe_wide": False}
BIG_WORD = {"bpe": b"a" * 2500, "bpe16": b"ab" * 2500, "bpe_wide": b"ab" * 2500}   # pre-tokens of more than 2048 tokens


def template(name, hf, add):
    """(prefix, suffix, seq_type) the call passes: the tokenizer.json's template, its special tokens only with add"""
    if not hf & tz.HF_TEMPLATE:
        return [], [], 0
    pre, suf, seq = orc.hf_template_from_json(MODELS[name])
    return (pre, suf, seq) if add else ([], [], seq)


def n_template(name):
    pre, suf, _ = orc.hf_template_from_json(MODELS[name])
    return len(pre) + len(suf)


@functools.lru_cache(maxsize=None)
def corpus(name):
    """seeded documents: ordinary words; empty documents and documents without a token; documents of exactly L and L + 1
    real tokens for every max_length of TP with and without the template (L = max_length minus its tokens); pre-tokens of
    256 bytes or more at the start of documents (their tokens are kept by truncation and shifted by left padding and the
    template); and for the BPE models one pre-token of more than 2048 tokens (the grid-wide copy)"""
    js = MODELS[name]
    rng = random.Random(4400 + len(name))
    if name in ("wordpiece", "bpe"):
        words = [w for w in json.loads(js)["model"]["vocab"] if w.isalpha() and w.islower()][:400] + ["zzqx", "unknownword"]
    else:
        words = ["ab", "cd", "abcd", "ee", "a", "abh", "fgh", "hgfe", "cab", "zq"]
    base = ascii_corpus(4500 + len(name), 300, words)
    maxlens = sorted({m for m, _ in TP.values() if m is not None})
    counts = sorted({m - k + d for m in maxlens for k in (0, n_template(name)) for d in (0, 1)})
    docs = exact_length_docs(orc.OracleTokenizer.from_json(js), base[:80], counts)
    docs += [b"", b" \t\n ", b"", b"ZZ Zq QQ", b"\x7f"]
    # a long pre-token first: WordPiece makes it one [UNK] (0, n); the small BPEs drop the unknown bytes, so its first token
    # ends beyond 255; the suite's BPE has an <unk> for every byte (wide tokens only behind 255 bytes of it)
    for n in (254, 256, 300, 700):
        lead = (b"Z" * n + b"abcd") if name in ("bpe16", "bpe_wide") else bytes(rng.choice(b"abcdefghij") for _ in range(n))
        docs.append(lead + b" " + " ".join(rng.choice(words) for _ in range(rng.randint(0, 30))).encode())
    if name in BIG_WORD:
        docs.append(b"ab " + BIG_WORD[name] + b" cd")
    for d in docs:                                   # (spread among the ordinary documents)
        base.insert(rng.randrange(0, len(base) + 1), d)
    return base


def long_piece_tokens(o, docs):
    """token count of every pre-token of 256 bytes or more (the slice pipeline's long words)"""
    m = orc.OracleTokenizer(o.cfg)
    m.normalizers, m.pretokenizers = [], None
    pieces = [p for d in docs for p in o.pre_tokenize(o.normalize(d)) if len(p) >= 256]
    return np.diff(m.encode_batch(pieces, algo=1).doc_tok_off.astype(np.int64)) if pieces else np.zeros(0, np.int64)


@functools.lru_cache(maxsize=None)
def oracle_case(name, hf_name, tp, normalizer=None, docs_key=None):
    """(expected arrays of the full case, the template the call passes) for corpus(name) or docs_key (a tuple of documents)"""
    js = MODELS[name]
    docs = list(docs_key) if docs_key is not None else corpus(name)
    _, hf, add = next(h for h in HF if h[0] == hf_name)
    trunc, pad = TP[tp]
    t, o = tz.Tokenizer.from_json(js, device=None), orc.OracleTokenizer.from_json(js)
    if normalizer:
        o.normalizers = [normalizer]
    n_pre, n_suf = configure(js, t, o, hf, add, trunc, pad)
    t.close()
    ref = o.encode_batch(docs, algo=1)
    wid = restated(o, docs, n_pre, n_suf)[0]
    base = orc.OracleTokenizer.from_json(js)
    if normalizer:
        base.normalizers = [normalizer]
    return expected(ref, wid, len(base.encode_batch(docs, algo=1).ids)), template(name, hf, add)


def expected(ref, wid, t_real):
    """every output form of an oracle encoding: template tokens are special but attended, padding slots are not attended"""
    pad = ref.attention_mask == 0
    tpl = (ref.special_tokens_mask == 1) & ~pad
    real = ~pad & ~tpl
    s, e = ref.offsets[:, 0].astype(np.uint64), ref.offsets[:, 1].astype(np.uint64)
    slots = np.flatnonzero(real & (e >= 256)).astype(np.uint64)
    ty = ref.type_ids & 0xFF
    return {"doc_tok_off": ref.doc_tok_off, "ids": ref.ids, "ids16": ref.ids.astype(np.uint16), "offsets": ref.offsets.reshape(-1),
            "offsets_packed": np.where(real, np.where(e < 256, s | (e << np.uint64(8)), 0xFFFF), 0).astype(np.uint16),
            "attention_mask": ref.attention_mask, "type_ids": ref.type_ids, "special_tokens_mask": ref.special_tokens_mask,
            "span_tokens": np.stack([ref.ids, ref.offsets[:, 0], ref.offsets[:, 1],
                                     np.where(pad, 0x0400, np.where(tpl, ty | 0x0100, ty))], 1).astype(np.uint32).reshape(-1),
            "word_ids": wid,
            "wide_tokens": np.stack([slots & np.uint64(0xFFFFFFFF), slots >> np.uint64(32), s[slots.astype(np.int64)],
                                     e[slots.astype(np.int64)]], 1).astype(np.uint32),
            "kind": np.where(pad, 2, np.where(tpl, 1, 0)), "n_real": t_real}


# per-slot value arrays of tkz_batch_result: dtype, elements per slot
ARRAYS = {"ids": (np.uint32, 1), "ids16": (np.uint16, 1), "offsets": (np.uint32, 2), "offsets_packed": (np.uint16, 1),
          "attention_mask": (np.uint32, 1), "type_ids": (np.uint32, 1), "special_tokens_mask": (np.uint32, 1),
          "span_tokens": (np.uint32, 4), "word_ids": (np.uint32, 1)}


def delivered(name, pipeline, mask, hf):
    """which arrays the call returns: u16 ids when the vocabulary allows; packed offsets from the slice pipeline without
    document offsets, else 32-bit pairs"""
    u16 = bool(mask & OUT_U16) and IDS16_OK[name]
    packed = bool(mask & OUT_PACKED) and pipeline != "occurrence" and not hf & (tz.HF_DOC_OFFSETS | tz.HF_OVERFLOW)
    return {"ids": not u16, "ids16": u16, "offsets": bool(mask & tz.OUT_OFFSETS) or (bool(mask & OUT_PACKED) and not packed),
            "offsets_packed": packed, "attention_mask": bool(mask & tz.OUT_ATTENTION), "type_ids": bool(mask & tz.OUT_TYPE_IDS),
            "special_tokens_mask": bool(mask & tz.OUT_SPECIAL), "span_tokens": bool(mask & OUT_SPAN), "word_ids": bool(mask & OUT_WID)}


KIND = ("real token", "template token", "padding")


def compare(got, exp, form, what):
    """got: {array: host copy or None}; exp: expected(...); form: delivered(...)"""
    assert np.array_equal(got["doc_tok_off"], exp["doc_tok_off"]), f"{what}: doc_tok_off"
    for k, (_, w) in ARRAYS.items():
        g = got[k]
        assert (g is not None) == form[k], f"{what}: {k} {'missing' if form[k] else 'delivered though not asked for'}"
        if g is None:
            continue
        want = exp[k]
        assert g.shape == want.shape, f"{what}: {k} has {g.shape}, want {want.shape}"
        if not np.array_equal(g, want):
            bad = np.flatnonzero(g != want)
            slot = int(bad[0]) // w
            msg = f"{what}: {k} differs at {len(bad)} elements; first slot {slot} ({KIND[exp['kind'][slot]]}): got {g[slot * w:(slot + 1) * w].tolist()}"
            if k == "offsets_packed":
                msg += f" = offsets ({int(g[slot]) & 0xFF}, {int(g[slot]) >> 8})"
            raise AssertionError(msg + f", want {want[slot * w:(slot + 1) * w].tolist()}")
    if form["offsets_packed"]:
        p = got["offsets_packed"]
        assert np.all(p[exp["kind"] != 0] == 0), f"{what}: packed offsets of template tokens / padding are not 0"
        wide = got["wide_tokens"]
        if not got.get("sorted"):
            wide = wide[np.lexsort((wide[:, 0], wide[:, 1]))]       # device results: in no particular order
        slots = wide[:, 0].astype(np.uint64) | (wide[:, 1].astype(np.uint64) << np.uint64(32))
        assert np.array_equal(slots, np.flatnonzero(p == 0xFFFF)), f"{what}: the wide list is not the set of 0xFFFF slots"
        assert np.array_equal(wide, exp["wide_tokens"]), f"{what}: wide tokens"
    else:
        assert len(got["wide_tokens"]) == 0, f"{what}: wide tokens without packed offsets"


def context(js, pipeline, stream):
    """a tokenizer whose context runs the given pipeline on the caller's stream (the switches are read when it is created)"""
    old = {k: os.environ.pop(k, None) for k in ENV_KEYS}
    os.environ.update(PIPELINES[pipeline])
    try:
        return tz.Tokenizer.from_json(js, device=0, stream=stream.cuda_stream)
    finally:
        for k, v in old.items():
            os.environ.pop(k, None)
            if v is not None:
                os.environ[k] = v


class Poisoner:
    """device calls on one stream, and the poisoning of what they returned"""

    def __init__(self, stream):
        self.rt = cudart()
        self.rt.cudaMemsetAsync.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_void_p]
        self.rt.cudaStreamSynchronize.argtypes = [C.c_void_p]
        self.stream = C.c_void_p(stream.cuda_stream)
        self.self_checked = False

    def call(self, t, d_text, d_off, n_docs, n_bytes, p):
        r = tz.BatchResult()
        rc = tz.lib().tkz_encode_batch_device(t.context_handle(), C.c_void_p(d_text), C.c_void_p(d_off), n_docs, n_bytes, C.byref(p), C.byref(r))
        assert rc == tz.OK, (rc, tz.lib().tkz_last_error(t.context_handle()))
        return r

    def poison(self, r):
        for k, (dt, w) in ARRAYS.items():
            if getattr(r, k) and r.n_tokens:
                assert self.rt.cudaMemsetAsync(getattr(r, k), POISON, int(r.n_tokens) * w * np.dtype(dt).itemsize, self.stream) == 0

    def read(self, r):
        T, n = int(r.n_tokens), int(r.n_docs)
        got = {k: d2h(self.rt, getattr(r, k), T * w, dt) if getattr(r, k) else None for k, (dt, w) in ARRAYS.items()}
        got["doc_tok_off"] = d2h(self.rt, r.doc_tok_off, n + 1, np.uint64)
        got["wide_tokens"] = d2h(self.rt, r.wide_tokens, 4 * int(r.n_wide), np.uint32).reshape(-1, 4)
        if r.n_rows:
            got["row_tok_off"] = d2h(self.rt, r.row_tok_off, int(r.n_rows) + 1, np.uint64)
            got["doc_row_off"] = d2h(self.rt, r.doc_row_off, n + 1, np.uint64)
        return got

    def run(self, t, d_text, d_off, n_docs, n_bytes, p, what):
        """call, poison what it returned, call again into the same buffers; the second result, read back"""
        r1 = self.call(t, d_text, d_off, n_docs, n_bytes, p)
        self.poison(r1)
        r2 = self.call(t, d_text, d_off, n_docs, n_bytes, p)
        assert r2.n_tokens == r1.n_tokens, what
        for k in ARRAYS:
            assert getattr(r2, k) == getattr(r1, k), f"{what}: {k} moved to a new buffer between the calls: the poison missed it"
        got = self.read(r2)
        if not self.self_checked:
            # the memset reaches the buffers this harness reads
            self.poison(r2)
            assert self.rt.cudaStreamSynchronize(self.stream) == 0
            for k, (dt, w) in ARRAYS.items():
                if getattr(r2, k) and r2.n_tokens:
                    assert np.all(d2h(self.rt, getattr(r2, k), int(r2.n_tokens) * w, dt).view(np.uint8) == POISON), k
            self.self_checked = True
        return r2, got


def params(t, mask, hf, tpl, **kw):
    p = t.params(outputs=mask)
    p.hf_flags = hf
    pre, suf, seq = tpl
    p.tpl_n_prefix, p.tpl_n_suffix, p.tpl_seq_type = len(pre), len(suf), seq
    for i, (a, b) in enumerate(pre):
        p.tpl_prefix_id[i], p.tpl_prefix_type[i] = a, b
    for i, (a, b) in enumerate(suf):
        p.tpl_suffix_id[i], p.tpl_suffix_type[i] = a, b
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def set_tp(t, tp):
    trunc, pad = TP[tp]
    t.truncation = None if trunc is None else {"max_length": trunc}
    t.padding = pad


def host_batch(r):
    """a host-buffer result in the form of Poisoner.read (its wide list comes sorted)"""
    T, n = int(r.n_tokens), int(r.n_docs)
    got = {k: tz._copy(getattr(r, k), T * w, dt) if getattr(r, k) else None for k, (dt, w) in ARRAYS.items()}
    got["doc_tok_off"] = tz._copy(r.doc_tok_off, n + 1, np.uint64)
    got["wide_tokens"] = tz._copy(r.wide_tokens, 4 * int(r.n_wide), np.uint32).reshape(-1, 4)
    got["sorted"] = True
    return got


def upload(docs):
    """the documents packed on the host and copied to the device: text, doc_off, d_text, d_doc_off (int64)"""
    import torch
    text, off = tz.pack_docs(docs)
    d_text, d_off = torch.from_numpy(text.copy()).cuda(), torch.from_numpy(off.astype(np.int64)).cuda()
    torch.cuda.synchronize()
    return text, off, d_text, d_off


@pytest.fixture
def stream():
    import torch
    s = torch.cuda.Stream()
    yield s
    s.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", list(PIPELINES))
@pytest.mark.parametrize("name", list(MODELS))
def test_case_table(name, pipeline, stream):
    docs = corpus(name)
    text, off, d_text, d_off = upload(docs)
    t, pz = context(MODELS[name], pipeline, stream), Poisoner(stream)
    L = tz.lib()
    failed, n_cases = [], 0
    for hf_name, hf, add in HF:
        for tp in TP:
            set_tp(t, tp)
            exp, tpl = oracle_case(name, hf_name, tp)
            for mask in MASKS:
                what = f"{name} {pipeline} hf {hf_name} {tp} mask {mask}"
                n_cases += 1
                p = params(t, mask, hf, tpl)
                r, got = pz.run(t, d_text.data_ptr(), d_off.data_ptr(), len(docs), len(text), p, what)
                assert t.stats().path == (0 if pipeline == "occurrence" else 2), what
                form = delivered(name, pipeline, mask, hf)
                try:
                    assert int(r.n_real_tokens) == exp["n_real"], what
                    compare(got, exp, form, what)
                    if mask in HOST_MASKS:
                        # the host-buffer call (one output set: encode_host_single) into the buffers just poisoned
                        pz.poison(r)
                        hr = tz.BatchResult()
                        assert L.tkz_encode_batch(t.context_handle(), text.ctypes.data, off.ctypes.data, len(docs), C.byref(p), C.byref(hr)) == tz.OK
                        compare(host_batch(hr), exp, form, what + " host buffers")
                except AssertionError as e:
                    failed.append(str(e).split("\n")[0])
    t.close()
    assert not failed, f"{len(failed)} of {n_cases} cases failed:\n" + "\n".join(failed[:40])


def test_case_table_has_the_edges():
    """the corpus and the case table reach the edges they are there for (oracle only)"""
    for name, js in MODELS.items():
        docs = corpus(name)
        o = orc.OracleTokenizer.from_json(js)
        ref = o.encode_batch(docs, algo=1)
        n = np.diff(ref.doc_tok_off.astype(np.int64))
        t_real = int(n.sum())
        assert b"" in docs and any(len(d) and k == 0 for d, k in zip(docs, n)), name
        for m in {m for m, _ in TP.values() if m is not None}:
            for L in (m, m - n_template(name)):
                assert L in n and L + 1 in n, (name, m, L)
        long_n = long_piece_tokens(o, docs)
        assert len(long_n), name
        if name in BIG_WORD:
            assert long_n.max() > 2048, name
        # (so many tokens of long pre-tokens that packed offsets fall back to 32-bit pairs: not here)
        assert long_n.sum() <= t_real // 8 + 4096, name
        for hf_name, hf, add in HF:
            sides = set()
            for tp, (trunc, pad) in TP.items():
                exp, _ = oracle_case(name, hf_name, tp)
                assert exp["n_real"] == t_real
                wide = len(exp["wide_tokens"])
                # wide tokens next to the template, left padding and (where the model can have one early) truncation
                if trunc is None or name != "bpe":
                    assert wide, (name, hf_name, tp)
                if pad is not None:
                    sides.add(len(exp["ids"]) >= 2 * t_real)
            assert sides == {True, False}, (name, hf_name)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["slices", "occurrence"])
@pytest.mark.parametrize("name", ["wordpiece", "bpe16"])
def test_overflow_rows(name, pipeline, stream):
    """TKZ_HF_OVERFLOW into poisoned buffers: two strides, with and without padding"""
    js = MODELS[name]
    docs = corpus(name)
    text, off, d_text, d_off = upload(docs)
    t, pz = context(js, pipeline, stream), Poisoner(stream)
    for hf in (tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS, tz.HF_TEMPLATE):
        for max_length, stride, pad in ((16, 0, None), (16, 5, {"length": 20, "pad_id": 1, "pad_type_id": 1, "direction": "left"}),
                                        (24, 11, {"length": 24, "pad_id": 0, "pad_type_id": 0, "direction": "right"})):
            pre, suf, seq = configure_overflow(t, js, hf, True, max_length, stride, pad)
            want = overflow_rows(orc.OracleTokenizer.from_json(js), docs, max_length, stride, pre, suf, seq, pad,
                                 doc_offsets=bool(hf & tz.HF_DOC_OFFSETS))
            for mask in (tz.OUT_ALL | OUT_WID, tz.OUT_IDS | OUT_U16 | OUT_PACKED):
                what = f"{name} {pipeline} hf {hf} L {max_length} stride {stride} pad {pad} mask {mask}"
                p = params(t, mask, hf | tz.HF_OVERFLOW, (pre, suf, seq), stride=stride)
                r, got = pz.run(t, d_text.data_ptr(), d_off.data_ptr(), len(docs), len(text), p, what)
                form = delivered(name, pipeline, mask, hf | tz.HF_OVERFLOW)
                for k in ("doc_row_off", "row_tok_off", "doc_tok_off"):
                    assert np.array_equal(got[k], want[k]), f"{what}: {k}"
                for k, f in (("ids16" if form["ids16"] else "ids", "ids"), ("offsets", "offsets"), ("attention_mask", "attention_mask"),
                             ("type_ids", "type_ids"), ("special_tokens_mask", "special_tokens_mask"), ("word_ids", "word_ids")):
                    assert (got[k] is not None) == form[k], f"{what}: {k}"
                    if form[k]:
                        assert np.array_equal(got[k], want[f].reshape(-1).astype(got[k].dtype)), f"{what}: {k}"
                assert got["offsets_packed"] is None and got["span_tokens"] is None
    t.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["wordpiece", "bpe16"])
def test_fast_mode_device_call(name, stream):
    """FastTokenizer.encode (params.fast) through the device call into poisoned buffers, against the oracle's algo 2"""
    js = MODELS[name]
    docs = corpus(name)
    text, off, d_text, d_off = upload(docs)
    t, pz, o = context(js, "slices", stream), Poisoner(stream), orc.OracleTokenizer.from_json(js)
    for max_seq, max_tok in ((8192, 512), (64, 7)):
        o.set_fast_options(max_seq, max_tok)
        ref = o.encode_batch(docs, algo=2, threads=4)
        for mask in (tz.OUT_ALL, tz.OUT_ALL | OUT_SPAN):
            what = f"{name} fast {max_seq}/{max_tok} mask {mask}"
            p = params(t, mask, 0, ([], [], 0), fast=1, fast_max_sequence_length=max_seq, fast_max_tokens=max_tok)
            r, got = pz.run(t, d_text.data_ptr(), d_off.data_ptr(), len(docs), len(text), p, what)
            T = len(ref.ids)
            assert np.array_equal(got["doc_tok_off"], ref.doc_tok_off), what
            assert np.array_equal(got["ids"], ref.ids) and np.array_equal(got["offsets"], ref.offsets.reshape(-1)), what
            assert np.all(got["attention_mask"] == 1) and np.all(got["type_ids"] == 0) and np.all(got["special_tokens_mask"] == 0), what
            assert len(got["attention_mask"]) == T, what
            if mask & OUT_SPAN:
                sp = got["span_tokens"].reshape(-1, 4)
                assert np.array_equal(sp[:, 0], ref.ids) and np.array_equal(sp[:, 1:3], ref.offsets) and np.all(sp[:, 3] == 0), what
            else:
                assert got["span_tokens"] is None
    t.close()


# the device-entry cases: (hf name, tp, mask)
ENTRY_CASES = (("ref", "none", tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION), ("tpl_doc", "trunc_pad_left", tz.OUT_ALL | OUT_WID),
               ("tpl", "pad_left", tz.OUT_IDS | OUT_U16 | OUT_PACKED | OUT_SPAN))
BERT_CLEAN = (orc.NORM_BERT_STRUCT, 3)       # clean_text (drops control bytes) | lowercase: the normalizer kernel K0 runs


def with_control_bytes(docs, seed):
    rng = random.Random(seed)
    out = []
    for d in docs:
        d = bytearray(d)
        for _ in range(rng.randint(0, 3)):
            d.insert(rng.randint(0, len(d)), rng.choice(b"\x00\x01\x08\x1f\x7f"))
        out.append(bytes(d))
    return out + [b"\x01\x02\x7f"]


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["slices", "occurrence"])
@pytest.mark.parametrize("name,normalizer", [("bpe", None), ("wordpiece", None), ("wordpiece", BERT_CLEAN)],
                         ids=["bpe", "wordpiece", "wordpiece-clean_text"])
def test_misaligned_document_ranges(name, normalizer, pipeline, stream):
    """the corpus uploaded once, as bench.py does; document ranges that start at every residue mod 16 are encoded from
    d_text + off[a] (staged into an aligned copy) with offsets rebased on the device"""
    import torch
    docs = corpus(name) if normalizer is None else with_control_bytes(corpus(name), 17)
    text, off, d_text, d_full = upload(docs)
    t, pz = context(MODELS[name], pipeline, stream), Poisoner(stream)
    if normalizer is not None:
        t.set_normalizer([(tz.NORM_BERT_STRUCT, normalizer[1])])
        t.encode_batch([b"a"])                                   # (the host mirror uploads the changed model with its next encode)
    starts = {}
    for a in range(len(docs) - 40):
        starts.setdefault(int(off[a]) % 16, a)
    assert sorted(starts) == list(range(16))
    for res, a in sorted(starts.items()):
        b = a + 40
        sub = tuple(docs[a:b])
        d_off = (d_full[a:b + 1] - d_full[a]).contiguous()
        torch.cuda.synchronize()
        n_bytes = int(off[b] - off[a])
        for hf_name, tp, mask in ENTRY_CASES:
            hf = next(h for h in HF if h[0] == hf_name)[1]
            set_tp(t, tp)
            exp, tpl = oracle_case(name, hf_name, tp, normalizer, sub)
            what = f"{name} norm {normalizer} {pipeline} start {a} (mod 16: {res}) hf {hf_name} {tp} mask {mask}"
            r, got = pz.run(t, d_text.data_ptr() + int(off[a]), d_off.data_ptr(), b - a, n_bytes, params(t, mask, hf, tpl), what)
            compare(got, exp, delivered(name, pipeline, mask, hf), what)
    t.close()


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["slices", "occurrence"])
def test_caller_stream_with_input_in_flight(pipeline, stream):
    """a context on the caller's stream; the text (3 MiB, pinned) and the rebased offsets are produced on that stream
    just before the call, with no synchronisation in between"""
    import torch
    name = "wordpiece"
    docs = corpus(name) * 40
    text, off = tz.pack_docs(docs)
    h_text = torch.from_numpy(text.copy()).pin_memory()
    h_off = torch.from_numpy(off.astype(np.int64)).pin_memory()
    a, b = 3, len(docs) - 5
    t, pz = context(MODELS[name], pipeline, stream), Poisoner(stream)
    hf_name, tp, mask = ENTRY_CASES[1]
    hf = next(h for h in HF if h[0] == hf_name)[1]
    set_tp(t, tp)
    exp, tpl = oracle_case(name, hf_name, tp, None, tuple(docs[a:b]))
    p = params(t, mask, hf, tpl)
    ptrs = None
    for k in range(2):
        with torch.cuda.stream(stream):
            d_text = h_text.to("cuda", non_blocking=True)
            d_full = h_off.to("cuda", non_blocking=True)
            d_off = d_full[a:b + 1] - d_full[a]
            r = pz.call(t, d_text.data_ptr() + int(off[a]), d_off.data_ptr(), b - a, int(off[b] - off[a]), p)
        what = f"{pipeline} caller stream, call {k}"
        assert ptrs is None or ptrs == [getattr(r, f) for f in ARRAYS], f"{what}: the poison missed the buffers"
        ptrs = [getattr(r, f) for f in ARRAYS]
        compare(pz.read(r), exp, delivered(name, pipeline, mask, hf), what)
        pz.poison(r)                                             # (the second call writes into poisoned buffers)
    t.close()
