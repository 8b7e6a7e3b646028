"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle, bit-exact on ids / offsets / masks / CSR offsets.
Covers the reference's own known-answer vectors, random vocabularies and texts (proper, improper, degenerate and aliased
merge tables; every normalizer / pre-tokenizer chain; truncation and padding), ragged and empty inputs, words longer
than the shared-memory path, equal-symbol runs across warp chunks, malformed UTF-8, and the real-size synthesised
tokenizers on corpus samples."""
import json
import random

import numpy as np
import pytest

import tokzig_b200 as tz
from oracle import oracle as orc
from gen_util import rand_bpe_json, rand_docs, rand_text, rand_wp_json
from kat_util import NORM_OPS, PT_OPS, check_encoding_against_case, load_kats, model_case_to_json, norm_flags
from tools import corpus, tokenizers_io

pytestmark = pytest.mark.gpu
CASES = load_kats()


def assert_same(got: tz.BatchEncoding, ref: orc.BatchEncoding, what=""):
    assert np.array_equal(got.doc_tok_off, ref.doc_tok_off), f"{what}: doc_tok_off"
    if not np.array_equal(got.ids, ref.ids):
        bad = int(np.nonzero(got.ids != ref.ids)[0][0]) if len(got.ids) == len(ref.ids) else -1
        raise AssertionError(f"{what}: ids differ (first at {bad}, {len(got.ids)} vs {len(ref.ids)} tokens)")
    assert np.array_equal(got.offsets, ref.offsets), f"{what}: offsets"
    assert np.array_equal(got.attention_mask, ref.attention_mask), f"{what}: attention_mask"
    assert np.array_equal(got.type_ids, ref.type_ids), f"{what}: type_ids"
    assert np.array_equal(got.special_tokens_mask, ref.special_tokens_mask), f"{what}: special_tokens_mask"


MODES = ("slices", "lut", "occurrence")


def pair(js, mode="slices"):
    """(GPU tokenizer, oracle).  The context reads its pipeline switches when it is created: mode "slices" = the slice
    pipeline (tkz_slices.cuh, default: byte classes by packed range compares when the class table allows it), "lut" = the
    same pipeline with the per-byte class look-up forced (TKZ_CLASSIFY=lut), "occurrence" = the per-occurrence pipeline
    (TKZ_NO_DEDUP=1).  All device pipelines are held to the same oracle."""
    import os
    os.environ["TKZ_NO_DEDUP"] = "1" if mode == "occurrence" else "0"
    os.environ["TKZ_CLASSIFY"] = "lut" if mode == "lut" else "auto"
    try:
        t = tz.Tokenizer.from_json(js, device=0)
    finally:
        os.environ["TKZ_NO_DEDUP"] = "0"
        os.environ["TKZ_CLASSIFY"] = "auto"
    return t, orc.OracleTokenizer.from_json(js)


# ----------------------------------------------------------------------------- the reference's known-answer vectors
@pytest.mark.parametrize("c", [c for c in CASES if c["kind"] in ("json", "model") and any(a in (0, 1) for a in c["algos"])], ids=lambda c: c["id"])
def test_reference_kats_on_gpu(c):
    js = c["json"] if c["kind"] == "json" else model_case_to_json(c["model"])
    t = tz.Tokenizer.from_json(js, device=0)
    if c.get("truncation") is not None:
        t.truncation = {"max_length": c["truncation"]}
    if c.get("padding") is not None:
        t.padding = c["padding"]
    text = bytes.fromhex(c["input_hex"])
    for add in (True, False):        # examples/basic_tokenize.zig calls encode(text, true); no post-processor does anything
        e = t.encode(text, add_special_tokens=add)
        check_encoding_against_case(c, e.ids, e.offsets, e.attention_mask, e.type_ids, e.special_tokens_mask)
    t.close()


def test_example_basic_tokenize_call_sequence(tmp_path):
    """examples/basic_tokenize.zig:24-45: fromFile -> encode("Hello, world!", true) -> ids / tokens."""
    js = tokenizers_io.tokenizer_json("gpt2_bytelevel")
    p = tmp_path / "tokenizer.json"
    p.write_text(js, encoding="utf-8")
    t = tz.Tokenizer.from_file(str(p), device=0)
    o = orc.OracleTokenizer.from_json(js)
    e = t.encode("Hello, world!", True)
    ids, offs, *_ = o.encode(b"Hello, world!")
    assert e.ids.tolist() == ids.tolist() and e.offsets.tolist() == offs.tolist()
    assert len(e.get_tokens()) == len(e.ids)
    # tokens[i] == idToToken(ids[i])  (bpe.zig:258)
    assert b"".join(e.get_tokens()) == b"Hello,world!"       # the space is not a vocab key of a byte-level vocab: dropped
    t.close()


def test_encoding_tokens_come_from_the_model_vocabulary_not_the_added_one():
    """Encoding.tokens[i] = the MODEL's vocab_r[id] (bpe.zig:258), while idToToken consults the added vocabulary first
    (lib.zig:217-223): an added token that shares an id with a model token must not change Encoding.tokens."""
    js = json.dumps({"model": {"type": "BPE", "vocab": {"a": 0, "b": 1, "ab": 2}, "merges": ["a b"]}, "pre_tokenizer": {"type": "Whitespace"},
                     "added_tokens": [{"id": 2, "content": "<special>", "special": True}, {"id": 7, "content": "<only-added>", "special": True}]})
    t = tz.Tokenizer.from_json(js, device=0)
    e = t.encode("ab a", True)
    assert e.ids.tolist() == [2, 0]
    assert e.get_tokens() == [b"ab", b"a"]
    assert t.id_to_token(2) == b"<special>" and t.id_to_token(7) == b"<only-added>" and t._model_id_to_token(7) is None
    t.close()


# ----------------------------------------------------------------------------- random property tests
@pytest.mark.parametrize("seed", range(48))
def test_bpe_random(seed):
    rng = random.Random(seed)
    mode = seed % 4
    js, alpha = rand_bpe_json(rng, n_merges=rng.randint(0, 80), unk="<unk>" if seed % 3 == 0 else None,
                              improper=[0.0, 0.3, 0.0, 0.5][mode], degenerate=[0.0, 0.0, 0.3, 0.2][mode], alias=[0.0, 0.0, 0.1, 0.2][mode],
                              pretok=[None, "Whitespace", "BertPreTokenizer", "ByteLevel"][(seed // 4) % 4],
                              normalizer=[None, "Lowercase"][(seed // 16) % 2])
    t, o = pair(js, mode=MODES[seed % 3])
    docs = rand_docs(rng, alpha, 400, max_len=90, p_upper=0.2)
    assert_same(t.encode_batch(docs), o.encode_batch(docs), f"seed {seed}")
    t.close()


@pytest.mark.parametrize("seed", range(32))
def test_wordpiece_random(seed):
    rng = random.Random(500 + seed)
    js, alpha = rand_wp_json(rng, n_words=rng.randint(5, 120), prefix=["##", "", "@@@", "#"][seed % 4], max_chars=[None, 4, 7, 100][(seed // 4) % 4],
                             pretok=["BertPreTokenizer", "Whitespace", None, "BertPreTokenizer"][(seed // 2) % 4],
                             normalizer=["BertNormalizer", None][(seed // 8) % 2])
    t, o = pair(js, mode=MODES[seed % 3])
    docs = rand_docs(rng, alpha, 400, max_len=70, p_upper=0.3)
    assert_same(t.encode_batch(docs), o.encode_batch(docs), f"seed {seed}")
    t.close()


@pytest.mark.parametrize("seed", range(24))
def test_truncation_and_padding(seed):
    rng = random.Random(900 + seed)
    if seed % 2:
        js, alpha = rand_wp_json(rng)
    else:
        js, alpha = rand_bpe_json(rng, n_merges=30, pretok="Whitespace")
    t, o = pair(js, mode="slices" if seed % 4 != 3 else "occurrence")
    docs = rand_docs(rng, alpha, 300, max_len=60)
    trunc = [None, 0, 1, 5, 8, 64][seed % 6]
    pad = [None, {"length": 8, "pad_id": 7, "pad_type_id": 3, "direction": "right"}, {"length": 5, "pad_id": 0, "direction": "left"},
           {"length": None, "pad_id": 9}][(seed // 2) % 4]
    if seed >= 16:      # mostly padding: the whole-array fill, in the per-occurrence pipeline at seeds 19 and 23
        pad = {"length": 256, "pad_id": 4, "pad_type_id": 2, "direction": "left"}
    t.truncation = None if trunc is None else {"max_length": trunc}
    o.truncation = trunc
    t.padding = pad
    o.padding = pad
    assert_same(t.encode_batch(docs), o.encode_batch(docs), f"seed {seed} trunc {trunc} pad {pad}")
    # a subset of the output arrays can be requested; ids always come back
    sub = t.encode_batch(docs, outputs=tz.OUT_IDS | tz.OUT_ATTENTION)
    ref = o.encode_batch(docs)
    assert np.array_equal(sub.ids, ref.ids) and np.array_equal(sub.attention_mask, ref.attention_mask) and sub.offsets is None
    t.close()


@pytest.mark.parametrize("seed", range(24))
def test_struct_chains(seed):
    """hand-wired normalizer_impl / pretokenizer_impl (struct variants and Sequences), incl. byte-dropping normalizers."""
    rng = random.Random(1300 + seed)
    tzn = {"cfg_lower": tz.NORM_CFG_LOWER, "bert_struct": tz.NORM_BERT_STRUCT, "lower_struct": tz.NORM_LOWER_STRUCT}
    tzp = {"ws_cfg": tz.PT_WS_CFG, "bert_cfg": tz.PT_BERT_CFG, "ws_struct": tz.PT_WS_STRUCT, "bert_struct": tz.PT_BERT_STRUCT,
           "bytelevel_struct": tz.PT_BYTELEVEL_STRUCT}
    if seed % 2:
        js, alpha = rand_wp_json(rng, pretok=None, normalizer=None)
    else:
        js, alpha = rand_bpe_json(rng, n_merges=30, unk="<unk>" if seed % 4 == 0 else None)
    t, o = pair(js, mode="slices" if seed % 3 != 1 else "occurrence")
    nn = [rng.choice(list(tzn)) for _ in range(rng.randint(0, 3))]
    fl = [rng.randint(0, 3) for _ in nn]
    pn = [rng.choice(list(tzp)) for _ in range(rng.randint(0, 3))]
    use_norm, use_pt = seed % 3 != 0, seed % 5 != 0
    t.set_normalizer([(tzn[n], f) for n, f in zip(nn, fl)] if use_norm else None)
    o.normalizers = [(NORM_OPS[n], f) for n, f in zip(nn, fl)] if use_norm else []
    t.set_pretokenizer([tzp[n] for n in pn] if use_pt else None)
    o.pretokenizers = [PT_OPS[n] for n in pn] if use_pt else None
    docs = []
    for _ in range(300):
        d = bytearray(rand_text(rng, alpha, rng.randint(0, 60), p_upper=0.3))
        for _ in range(rng.randint(0, 3)):          # control bytes (ASCII, keeps UTF-8 valid) for clean_text
            d.insert(rng.randint(0, len(d)), rng.choice(b"\x00\x01\x08\x1f\x7f\x0b\x0c"))
        docs.append(_fix_utf8(bytes(d)))
    assert_same(t.encode_batch(docs), o.encode_batch(docs), f"seed {seed} norm {nn}{fl} pt {pn}")
    t.close()


def _fix_utf8(b: bytes) -> bytes:
    return b.decode("utf-8", "ignore").encode("utf-8")


# ----------------------------------------------------------------------------- edge cases
@pytest.mark.parametrize("mode", MODES)
def test_empty_and_ragged_inputs(mode):
    js, alpha = rand_bpe_json(random.Random(1), n_merges=20, pretok="Whitespace")
    t, o = pair(js, mode=mode)
    for docs in ([], [b""], [b"", b"", b""], [b" "], [b"  \n\t "], [b"a"], [b"", b"a", b""], [b"ab", b"", b"", b"ba ab"], [b"a" * 5000, b"", b"b"]):
        assert_same(t.encode_batch(docs), o.encode_batch(docs), repr(docs)[:40])
    t.close()


@pytest.mark.parametrize("mode", MODES)
def test_document_boundary_splits_words(mode):
    js = json.dumps({"model": {"type": "BPE", "vocab": {"a": 0, "b": 1, "ab": 2, "ba": 3, "abab": 4}, "merges": ["a b", "b a", "ab ab"]},
                     "pre_tokenizer": {"type": "Whitespace"}})
    t, o = pair(js, mode=mode)
    docs = [b"abab", b"ab", b"ab", b"a", b"b", b"", b"a b", b"ab"] * 700        # boundaries fall inside tiles and on tile edges
    assert_same(t.encode_batch(docs), o.encode_batch(docs))
    t.close()


@pytest.mark.parametrize("n", [31, 32, 33, 63, 64, 65, 95, 96, 97, 511, 512, 513, 1000, 5000])
def test_equal_symbol_runs_across_chunks(n):
    # aaaaa -> aa aa a (SURVEY.md 2.3); runs crossing 32-lane chunks, the shared-memory limit and the HBM path
    js = json.dumps({"model": {"type": "BPE", "vocab": {"a": 0, "b": 1, "aa": 2, "aaaa": 3, "ab": 4}, "merges": ["a a", "aa aa", "a b"]}})
    t, o = pair(js)
    docs = [b"a" * n, b"b" + b"a" * n, b"a" * n + b"b", (b"a" * 7 + b"b") * (n // 8 + 1), b"ab" * n]
    assert_same(t.encode_batch(docs), o.encode_batch(docs), f"n {n}")
    t.close()


def test_survey_adversarial_cascades():
    v = {"w": 0, "x": 1, "y": 2, "z": 3, "u": 4, "wx": 5, "wxy": 6, "wxyz": 7, "zu": 8, "xy": 9, "yz": 10}
    merges = [["w", "x"], ["wx", "y"], ["wxy", "z"], ["z", "u"], ["x", "y"], ["y", "z"]]
    t, o = pair(json.dumps({"model": {"type": "BPE", "vocab": v, "merges": merges}}))
    docs = [b"wxyzu", b"wxyzu" * 40, b"uzyxw" * 30, b"xyzuwxyzu" * 100]
    assert_same(t.encode_batch(docs), o.encode_batch(docs))
    assert t.encode(b"wxyzu").ids.tolist() == [7, 4]
    t.close()
    v = {"d": 0, "a": 1, "b": 2, "c": 3, "bc": 4, "ab": 5, "da": 6, "abc": 7}
    t, o = pair(json.dumps({"model": {"type": "BPE", "vocab": v, "merges": ["b c", "a b", "x x", "d a", "y y", "a bc"]}}))
    assert t.encode(b"dabc").ids.tolist() == [6, 4]           # canonical BPE.tokenize answer, not tokenizeFast's [d, abc]
    t.close()


def test_long_words_take_the_hbm_path():
    rng = random.Random(5)
    js, alpha = rand_bpe_json(rng, n_merges=150, alphabet=list("abcdefgh") + ["é", "中"], dead_merges=0.0)
    t, o = pair(js)
    docs = ["".join(rng.choice(alpha) for _ in range(n)).encode() for n in (600, 1500, 4000, 20000, 3, 0, 513)]
    assert_same(t.encode_batch(docs), o.encode_batch(docs, algo=1))
    t.close()


def test_malformed_utf8():
    js = json.dumps({"model": {"type": "BPE", "vocab": {"a": 0, "b": 1, "é": 2, "ab": 3, "Ã(": 4}, "merges": ["a b"]}}, ensure_ascii=False)
    t, o = pair(js)
    # malformed but in bounds: the reference's iterator takes the length from the lead byte only -> defined behaviour
    ok_docs = [b"ab\xc3(ab", b"a\xe4ab", b"\xc3\xa9ab\xc3\xa9", b"ab\xf0abcab"]
    assert_same(t.encode_batch(ok_docs), o.encode_batch(ok_docs))
    # invalid lead byte / truncated tail: `unreachable` in the reference -> an error here, with the document index
    for bad, where in (([b"ab", b"a\x80b"], 1), ([b"ab\xc3"], 0), ([b"ok", b"ok", b"\xff"], 2), ([b"a\xe4\xb8"], 0)):
        with pytest.raises(tz.TokzigError) as e:
            t.encode_batch(bad)
        assert e.value.code == tz.ERR_INVALID_UTF8 and e.value.doc == where
        with pytest.raises(orc.OracleError) as e2:
            o.encode_batch(bad)
        assert e2.value.code == orc.ERR_INVALID_UTF8 and e2.value.doc == where
    t.close()


@pytest.mark.parametrize("dedup", ["slices", "lut", "occurrence"])
def test_wordpiece_missing_unk_is_an_error(dedup):
    js = json.dumps({"model": {"type": "WordPiece", "vocab": {"hello": 1, "##s": 2}, "unk_token": "[UNK]"}, "pre_tokenizer": {"type": "Whitespace"}})
    t, o = pair(js, mode=dedup)
    assert_same(t.encode_batch([b"hello hellos"]), o.encode_batch([b"hello hellos"]))
    with pytest.raises(tz.TokzigError) as e:
        t.encode_batch([b"hello", b"hello xyz", b"q"])
    assert e.value.code == tz.ERR_MISSING_UNK and e.value.doc == 1
    with pytest.raises(orc.OracleError) as e2:
        o.encode_batch([b"hello", b"hello xyz", b"q"])
    assert e2.value.code == orc.ERR_MISSING_UNK and e2.value.doc == 1
    t.close()


def test_wordpiece_long_keys_and_512_byte_rule():
    long_piece = "x" * 600
    vocab = {"[UNK]": 0, "a": 1, "##" + long_piece: 2, long_piece: 3, "##b": 4, "ab": 5}
    js = json.dumps({"model": {"type": "WordPiece", "vocab": vocab, "max_input_chars_per_word": 5000}})
    t, o = pair(js)
    docs = [long_piece.encode(), b"a" + long_piece.encode(), b"ab", b"a" + b"b" * 3, (long_piece + long_piece).encode()]
    assert_same(t.encode_batch(docs), o.encode_batch(docs))
    t.close()


# ----------------------------------------------------------------------------- real-size tokenizers on corpus samples
@pytest.mark.parametrize("name,cname,algo,nbytes", [("gpt2_whitespace", "c2", 0, 3 << 20), ("gpt2_bytelevel", "c2", 1, 3 << 20),
                                                     ("bert_wordpiece", "c3", 0, 3 << 20), ("llama3_whitespace", "c4", 0, 2 << 20),
                                                     ("llama3_sequence", "c4", 1, 2 << 20), ("gpt2_whitespace", "c5", 1, 6 << 20),
                                                     ("gpt2_bytelevel", "c5", 1, 6 << 20)])
def test_synthesised_tokenizers_on_corpus(name, cname, algo, nbytes):
    js = tokenizers_io.tokenizer_json(name)
    t, o = pair(js)
    text, off = corpus.generate(cname, nbytes, seed=2024)
    if name == "bert_wordpiece":
        t.truncation = {"max_length": 512}
        o.truncation = 512
        t.padding = {"length": 64, "pad_id": 0}
        o.padding = {"length": 64, "pad_id": 0}
    got = t.encode_packed(text, off)
    ref = o.encode_packed(text, off, algo=algo, threads=8)
    assert_same(got, ref, name)
    t.close()


def test_batch_split_invariance_and_roundtrip_property():
    """size-independent properties at a larger size: encoding a batch == concatenating the encodings of its halves, and
    (BPE, no unk) the token strings of a document concatenate to the document minus the characters the vocab lacks."""
    js = tokenizers_io.tokenizer_json("gpt2_whitespace")
    t = tz.Tokenizer.from_json(js, device=0)
    text, off = corpus.generate("c2", 48 << 20, seed=77)
    full = t.encode_packed(text, off)
    nd = len(off) - 1
    h = nd // 2
    a = t.encode_packed(text[: int(off[h])], off[: h + 1])
    b = t.encode_packed(text[int(off[h]):], off[h:] - off[h])
    assert np.array_equal(full.ids, np.concatenate([a.ids, b.ids]))
    assert np.array_equal(full.offsets, np.concatenate([a.offsets, b.offsets]))
    assert np.array_equal(full.doc_tok_off, np.concatenate([a.doc_tok_off, b.doc_tok_off[1:] + a.doc_tok_off[-1]]))
    # round trip on a sample of documents
    d = t.model_desc()
    id2tok = {int(i): k for k, i in zip(d["keys"], d["ids"])}
    single = {k for k in d["keys"] if len(k.decode("utf-8", "ignore")) == 1}
    rng = random.Random(3)
    raw = text.tobytes()
    for i in rng.sample(range(nd), 200):
        doc = raw[int(off[i]):int(off[i + 1])]
        kept = b"".join(ch.encode() for w in doc.split() for ch in w.decode("utf-8") if ch.encode() in single)
        sl = full.doc_slice(i)
        assert b"".join(id2tok[int(x)] for x in full.ids[sl]) == kept
    t.close()


# ----------------------------------------------------------------------------- dedup pipeline specifics
@pytest.mark.parametrize("mode", ["slices", "lut"])
@pytest.mark.parametrize("model", ["bpe", "wp"])
def test_dedup_word_lengths_around_the_key_limit(model, mode):
    """words of 14 / 15 / 16 / 17 bytes straddle the 128-bit key (15 bytes + length), incl. NUL bytes inside words,
    words crossing 4 KiB tile edges and document boundaries inside a run."""
    rng = random.Random(17)
    if model == "bpe":
        js, alpha = rand_bpe_json(rng, n_merges=60, alphabet=list("abcde") + ["é"], pretok="Whitespace", dead_merges=0.0)
    else:
        js, alpha = rand_wp_json(rng, n_words=80, alphabet=list("abcde") + ["é"], pretok="Whitespace", normalizer=None)
    t, o = pair(js, mode=mode)
    docs = []
    for i in range(3000):
        words = []
        for _ in range(rng.randint(0, 12)):
            L = rng.choice([1, 2, 3, 7, 13, 14, 15, 16, 17, 31, 40, 63, 64, 65, 66, 100, 101, 255, 256, 257])
            w = "".join(rng.choice(alpha) for _ in range(L)).encode()[:L]
            words.append(w.decode("utf-8", "ignore").encode())
        d = b" ".join(words)
        if model == "wp" and rng.random() < 0.2:
            d = d.replace(b"a", b"\x00", 1)          # NUL is an ordinary word byte for the whitespace split
        docs.append(d)
    assert_same(t.encode_batch(docs), o.encode_batch(docs), model)
    t.close()


def test_dedup_and_per_occurrence_pipelines_agree_on_errors():
    js = json.dumps({"model": {"type": "BPE", "vocab": {"a": 0, "b": 1, "ab": 2}, "merges": ["a b"]}, "pre_tokenizer": {"type": "Whitespace"}})
    for mode in MODES:
        t, o = pair(js, mode=mode)
        docs = [b"ab ab", b"ab \xffab ab", b"a\x80 ab", b"ab"]            # first failing document in TEXT order is 1
        with pytest.raises(tz.TokzigError) as e:
            t.encode_batch(docs)
        assert e.value.code == tz.ERR_INVALID_UTF8 and e.value.doc == 1
        # a long failing word (>15 bytes) in an earlier document wins over a short failing word later
        docs = [b"ab", b"ab " + b"a" * 20 + b"\xc3", b"\xff"]
        with pytest.raises(tz.TokzigError) as e:
            t.encode_batch(docs)
        assert e.value.doc == 1
        t.close()


@pytest.mark.parametrize("mode", ["slices", "lut"])
@pytest.mark.parametrize("n_words", [60000, 200000])
def test_dedup_table_pressure_and_overflow(n_words, mode):
    """more unique words than the batch's table holds: insertions that find no slot fall back to the long list, and when
    the long list overflows as well the batch is re-run by the per-occurrence pipeline -- results stay exact."""
    rng = random.Random(23)
    js, alpha = rand_bpe_json(rng, n_merges=100, alphabet=list("abcdefghijklmnop"), pretok="Whitespace", dead_merges=0.0)
    t, o = pair(js, mode=mode)
    chars = "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789"
    words = ["".join(rng.choice(chars) for _ in range(4)) for _ in range(n_words)]
    docs = [" ".join(words[i:i + 50]).encode() for i in range(0, len(words), 50)]
    assert_same(t.encode_batch(docs), o.encode_batch(docs, threads=8))
    t.close()


# ----------------------------------------------------------------------------- windowed block kernels (long words)
def _long_docs(rng, alpha, lengths, p_run=0.1):
    docs = []
    for n in lengths:
        out = []
        while len(out) < n:
            if rng.random() < p_run:
                out.extend([rng.choice(alpha)] * rng.randint(2, 40))          # equal-symbol runs
            elif rng.random() < 0.03:
                out.append(rng.choice(["z", "Z", "語", " "]))                  # not in the vocab: dropped or <unk>
            else:
                out.append(rng.choice(alpha))
        docs.append("".join(out[:n]).encode())
    return docs


@pytest.mark.parametrize("seed", range(12))
def test_windowed_block_kernel_random_proper_tables(seed):
    rng = random.Random(4000 + seed)
    alpha = list("abcdefgh")[: rng.randint(2, 8)] + (["é", "中"] if seed % 2 else [])
    js, alpha = rand_bpe_json(rng, n_merges=rng.randint(5, 400), alphabet=alpha, unk="<unk>" if seed % 4 == 0 else None,
                              dead_merges=0.0, unique_products=True, pretok=[None, "Whitespace"][seed % 2])
    t, o = pair(js)
    lengths = [65, 66, 100, 255, 256, 257, 1000, 2047, 2048, 2049, 5000, 12287, 12288, 12289, 30000, 3, 0, 64]
    docs = _long_docs(rng, alpha, lengths)
    got = t.encode_batch(docs)
    assert t.stats().model_flags & 1, "a table with unique producers listed in creation order must be recognised as proper"
    assert_same(got, o.encode_batch(docs, algo=1), f"seed {seed}")
    t.close()


@pytest.mark.parametrize("seed", range(6))
def test_long_words_with_improper_tables_use_literal_rounds(seed):
    rng = random.Random(4100 + seed)
    js, alpha = rand_bpe_json(rng, n_merges=80, alphabet=list("abcdef"), improper=0.4, degenerate=0.1 * (seed % 2), dead_merges=0.0)
    t, o = pair(js)
    docs = _long_docs(rng, alpha, [70, 300, 2100, 4000, 13000])
    assert_same(t.encode_batch(docs), o.encode_batch(docs, algo=1), f"seed {seed}")
    t.close()


def test_windowed_cascades_and_runs_at_length():
    # the SURVEY.md section 7 cascade (local minima merged in parallel would give [wxy, zu]) repeated past every kernel boundary
    v = {"w": 0, "x": 1, "y": 2, "z": 3, "u": 4, "wx": 5, "wxy": 6, "wxyz": 7, "zu": 8, "xy": 9, "yz": 10}
    merges = [["w", "x"], ["wx", "y"], ["wxy", "z"], ["z", "u"], ["x", "y"], ["y", "z"]]
    t, o = pair(json.dumps({"model": {"type": "BPE", "vocab": v, "merges": merges}}))
    docs = [b"wxyzu" * k for k in (13, 14, 410, 2500, 7000)] + [b"uzyxw" * 3000, b"xyzuwxyzu" * 1500, b"wxyzuzu" * 2000]
    got = t.encode_batch(docs)
    assert t.stats().model_flags & 1
    assert_same(got, o.encode_batch(docs, algo=1))
    t.close()
    v = {"a": 0, "b": 1, "aa": 2, "aaaa": 3, "ab": 4, "aab": 5}
    t, o = pair(json.dumps({"model": {"type": "BPE", "vocab": v, "merges": ["a a", "aa aa", "a b", "aa b"]}}))
    docs = [b"a" * n for n in (65, 66, 67, 1023, 1024, 1025, 4097, 20001)] + [(b"a" * 9 + b"b") * 700, b"b" + b"a" * 3000 + b"b" * 5, (b"aab" * 5 + b"aaaab") * 600]
    assert_same(t.encode_batch(docs), o.encode_batch(docs, algo=1))
    t.close()


# ----------------------------------------------------------------------------- grid-wide kernel (huge words, tkz_bpe_grid.cuh)
def _huge_docs(rng, alpha, lengths, p_run=0.08, drop=("z", "語")):
    """Unbroken words (no white space): random symbols, equal-symbol runs of 2..90 (longer than the kernel's walk limit of
    32), characters that are not in the vocabulary (dropped, or <unk>)."""
    docs = []
    for n in lengths:
        out = []
        while len(out) < n:
            x = rng.random()
            if x < p_run:
                out.extend([rng.choice(alpha)] * rng.randint(2, 90))
            elif x < p_run + 0.02:
                out.append(rng.choice(drop))
            else:
                out.append(rng.choice(alpha))
        docs.append("".join(out[:n]).encode())
    return docs


@pytest.mark.parametrize("seed", range(10))
def test_grid_kernel_random_proper_tables(seed):
    """Several words above the shared-memory capacity (12288 bytes) in one batch go through bpe_grid_kernel together; as
    whole documents (no pre-tokenizer, per-occurrence pipeline) and as words of the slice pipeline's long list."""
    rng = random.Random(7000 + seed)
    alpha = list("abcdefgh")[: rng.randint(2, 8)] + (["é", "中"] if seed % 2 else [])
    js, alpha = rand_bpe_json(rng, n_merges=rng.randint(5, 400), alphabet=alpha, unk="<unk>" if seed % 4 == 0 else None,
                              dead_merges=0.0, unique_products=True, pretok=[None, "Whitespace"][(seed // 2) % 2])
    t, o = pair(js)
    lengths = [12289, 13000, 40000, 3, 150000, 12288, 0, 20000, 65, 70001, 2500]
    docs = _huge_docs(rng, alpha, lengths)
    docs.append(b" ".join(_huge_docs(rng, alpha, [15000, 100, 30000, 14000])))      # several huge words in one document
    got = t.encode_batch(docs)
    st = t.stats()
    assert st.model_flags & 1, "the generated table must be recognised as proper"
    assert st.model_flags & 2, "the huge words must have taken the grid-wide kernel"
    assert_same(got, o.encode_batch(docs, algo=1, threads=8), f"seed {seed}")
    t.close()


def test_grid_kernel_runs_empty_words_and_malformed_words(monkeypatch):
    v = {"a": 0, "b": 1, "aa": 2, "aaaa": 3, "ab": 4, "aab": 5, "Ã(": 6}
    js = json.dumps({"model": {"type": "BPE", "vocab": v, "merges": ["a a", "aa aa", "a b", "aa b"]}}, ensure_ascii=False)
    t, o = pair(js)
    docs = [b"a" * 20001, b"a" * 300000, (b"a" * 9 + b"b") * 5000, b"b" + b"a" * 70000 + b"b" * 5, (b"aab" * 5 + b"aaaab") * 3000,
            "語".encode() * 10000,                          # 30000 bytes, no symbol at all
            b"a" * 13001 + "語".encode() * 5 + b"a" * 13000, b"ab" * 40000,
            b"ab" * 7000 + b"\xc3(" + b"ab" * 7000,         # malformed but in bounds: left to the block kernel (sequential re-decode)
            b"", b"ab"]
    got = t.encode_batch(docs)
    assert t.stats().model_flags & 2
    assert_same(got, o.encode_batch(docs, algo=1, threads=8))
    # invalid lead byte inside a huge word: still an error with the document index
    bad = [b"ab" * 9000, b"ab" * 9000 + b"\xff" + b"ab" * 10]
    with pytest.raises(tz.TokzigError) as e:
        t.encode_batch(bad)
    assert e.value.code == tz.ERR_INVALID_UTF8 and e.value.doc == 1
    t.close()
    # A/B: the same batch with one block per huge word
    monkeypatch.setenv("TKZ_NO_GRID", "1")
    t2 = tz.Tokenizer.from_json(js, device=0)
    got2 = t2.encode_batch(docs)
    assert not (t2.stats().model_flags & 2)
    assert_same(got2, got)
    t2.close()


def test_grid_kernel_sparse_phase_falls_back_for_a_long_late_run(monkeypatch):
    """(a, a) has the highest rank: its runs wait until every other pair of the word is done, i.e. until the kernel is in its
    sparse in-place phase; a run longer than the sparse walk limit must send it back to the dense steps (run scan)."""
    rng = random.Random(99)
    toks = list("bcdefgh")
    vocab = {c: i for i, c in enumerate("abcdefgh")}
    merges = []
    while len(merges) < 150:
        x, y = rng.choice(toks), rng.choice(toks)
        if x + y in vocab or len(x + y) > 12:
            continue
        vocab[x + y] = len(vocab)
        toks.append(x + y)
        merges.append(f"{x} {y}")
    vocab["aa"] = len(vocab)
    vocab["aaaa"] = len(vocab)
    merges += ["a a", "aa aa"]
    js = json.dumps({"model": {"type": "BPE", "vocab": vocab, "merges": merges}})
    t, o = pair(js)
    rnd = lambda n: "".join(rng.choice("bcdefgh") for _ in range(n))
    docs = [(rnd(60000) + "a" * 3001 + rnd(9000) + "a" * 700 + rnd(50) + "a" * 5000).encode(), (rnd(20000) + "a" * 40 + rnd(100)).encode(),
            ("a" * 2100 + rnd(30000)).encode()]
    got = t.encode_batch(docs)
    assert t.stats().model_flags & 3 == 3
    ref = o.encode_batch(docs, algo=1, threads=8)
    assert_same(got, ref)
    t.close()
    # the same with a walk limit of 2: the phase changes (sparse -> compaction -> dense run scan -> sparse ...) happen dozens
    # of times per launch (regression: a flag reset that raced with slower blocks still reading the flag)
    monkeypatch.setenv("TKZ_GRID_SPARSE_WALK", "2")
    for rep in range(3):
        t2 = tz.Tokenizer.from_json(js, device=0)
        assert_same(t2.encode_batch(docs + _huge_docs(rng, list("bcdefgha"), [15000, 40000], p_run=0.3)[:0]), ref, f"walk limit 2, repetition {rep}")
        t2.close()


def test_grid_kernel_on_the_skewed_corpus():
    """c5 generator (documents 1 B .. 4 MiB with long unbroken words) through the GPT-2-shaped tokenizers: Whitespace
    (slice pipeline + long list) and ByteLevel JSON (whole documents)."""
    text, off = corpus.generate("c5", 24 << 20, seed=77)
    for name in ("gpt2_whitespace", "gpt2_bytelevel"):
        js = tokenizers_io.tokenizer_json(name)
        t = tz.Tokenizer.from_json(js, device=0)
        o = orc.OracleTokenizer.from_json(js)
        got = t.encode_packed(text, off)
        assert t.stats().model_flags & 2, name
        assert_same(got, o.encode_packed(text, off, algo=1, threads=8), name)
        t.close()


def test_windowed_vs_literal_switch(monkeypatch):
    """TKZ_NO_WINDOWED=1 forces the literal round kernel for long words: both schedules must give the oracle's answer."""
    js = tokenizers_io.tokenizer_json("gpt2_bytelevel")
    text, off = corpus.generate("c2", 1 << 20, seed=31)
    o = orc.OracleTokenizer.from_json(js)
    ref = o.encode_packed(text, off, algo=1, threads=8)
    for flag in ("0", "1"):
        monkeypatch.setenv("TKZ_NO_WINDOWED", flag)
        t = tz.Tokenizer.from_json(js, device=0)
        got = t.encode_packed(text, off)
        assert bool(t.stats().model_flags & 1) == (flag == "0")
        assert_same(got, ref, f"TKZ_NO_WINDOWED={flag}")
        t.close()


# ----------------------------------------------------------------------------- chunked (pipelined) host path
@pytest.mark.parametrize("chunk", [4096, 65536])
def test_chunked_host_path_matches_single_shot(monkeypatch, chunk):
    monkeypatch.setenv("TKZ_CHUNK_BYTES", str(chunk))
    for name, cname, trunc, pad in (("gpt2_whitespace", "c2", None, None), ("bert_wordpiece", "c3", 16, {"length": 24, "pad_id": 0, "direction": "left"})):
        js = tokenizers_io.tokenizer_json(name)
        t = tz.Tokenizer.from_json(js, device=0)
        o = orc.OracleTokenizer.from_json(js)
        t.truncation = None if trunc is None else {"max_length": trunc}
        o.truncation = trunc
        t.padding = pad
        o.padding = pad
        text, off = corpus.generate(cname, 1 << 20, seed=5)
        assert_same(t.encode_packed(text, off), o.encode_packed(text, off, threads=8), f"{name} chunk {chunk}")
        t.close()
    # the error position is reported in whole-batch document numbering
    js = json.dumps({"model": {"type": "BPE", "vocab": {"a": 0, "b": 1, "ab": 2}, "merges": ["a b"]}, "pre_tokenizer": {"type": "Whitespace"}})
    t = tz.Tokenizer.from_json(js, device=0)
    docs = [b"ab ab ab"] * 3000 + [b"ab \xff"] + [b"ab"] * 10
    with pytest.raises(tz.TokzigError) as e:
        t.encode_batch(docs)
    assert e.value.code == tz.ERR_INVALID_UTF8 and e.value.doc == 3000
    t.close()


# ----------------------------------------------------------------------------- slice pipeline (tkz_slices.cuh)
@pytest.mark.parametrize("name,cname,mib", [("gpt2_whitespace", "c2", 96), ("llama3_whitespace", "c4", 64), ("bert_wordpiece", "c3", 48)])
def test_tiles_equal_per_occurrence_at_size(name, cname, mib, monkeypatch):
    """the slice pipeline against the per-occurrence pipeline (one warp per pre-token, no word table) on the same batch
    (one device call for the whole batch), every output array compared in full (both are held to the oracle at
    oracle-feasible sizes above)."""
    monkeypatch.setenv("TKZ_CHUNK_BYTES", str(1 << 31))
    js = tokenizers_io.tokenizer_json(name)
    text, off = corpus.generate(cname, mib << 20, seed=31)
    t1, _ = pair(js, mode="slices")
    t0, _ = pair(js, mode="occurrence")
    for rep in range(2):                                  # second call: table sized from history, output estimate from density
        a = t1.encode_packed(text, off)
        b = t0.encode_packed(text, off)
        assert t0.stats().path == 0
        assert t1.stats().path == 2, "the slice pipeline gave up on a corpus it is meant to handle"
        for k in ("doc_tok_off", "ids", "offsets", "attention_mask", "type_ids", "special_tokens_mask"):
            assert np.array_equal(getattr(a, k), getattr(b, k)), f"{name} call {rep}: {k}"
    t1.close(); t0.close()


def test_tiles_words_between_65_and_255_bytes_and_the_long_list():
    """65..255-byte words are tokenized inside pass A (symbols in global scratch, not deduplicated); longer words go to
    the long list (word-list kernels between the passes, counts folded back per tile and per document start)."""
    rng = random.Random(41)
    for model in ("bpe", "wp"):
        if model == "bpe":
            js, alpha = rand_bpe_json(rng, n_merges=80, alphabet=list("abcdefgh") + ["é", "語"], pretok="Whitespace", dead_merges=0.0)
        else:
            js, alpha = rand_wp_json(rng, n_words=100, alphabet=list("abcdefgh") + ["é"], pretok="BertPreTokenizer", max_chars=300)
        t, o = pair(js)

        def word(L):
            return "".join(rng.choice(alpha) for _ in range(L)).encode()[:L].decode("utf-8", "ignore").encode()

        inline = [b" ".join(word(rng.choice([3, 9, 64, 65, 90, 128, 200, 254, 255])) for _ in range(rng.randint(1, 9))) for _ in range(800)]
        assert_same(t.encode_batch(inline), o.encode_batch(inline, threads=8), model + " inline")
        assert t.stats().path == 2 and t.stats().n_long_words == 0
        # long words in front of document starts inside the same tile, at tile edges, back to back
        longer = inline[:300] + [b"ab " + word(256) + b" cd", word(257) + b" " + word(256) + b" " + word(256) + b" " + word(256), word(3000), b"", word(5), word(300) + b" " + word(400), b"x", word(9000)] + inline[300:500]
        for trunc, pad in ((None, None), (7, {"length": 9, "pad_id": 3})):
            t.truncation = None if trunc is None else {"max_length": trunc}
            o.truncation = trunc
            t.padding = pad; o.padding = pad
            assert_same(t.encode_batch(longer), o.encode_batch(longer, threads=8), model + f" long list trunc={trunc}")
            assert t.stats().path == 2 and t.stats().n_long_words >= 2
        t.close()


def test_tiles_wordpiece_words_above_max_chars_any_length():
    """WordPiece only needs the length of a word above max_input_chars_per_word (wordpiece.zig:149-158): one [UNK] with
    offsets (0, len), whatever the length -- handled inside pass A up to 255 bytes, by the word-list kernel beyond."""
    js, alpha = rand_wp_json(random.Random(5), n_words=60, pretok="Whitespace", max_chars=100, normalizer=None)
    t, o = pair(js)
    docs = [b"x" * n + b" " + b"ab" for n in (99, 100, 101, 255, 256, 257, 1000, 4095, 4096, 4097, 20000, 65535)] * 3
    assert_same(t.encode_batch(docs), o.encode_batch(docs))
    assert t.stats().path == 2
    docs.append(b"y" * 70000)
    assert_same(t.encode_batch(docs), o.encode_batch(docs))
    t.close()


def test_tiles_dense_isolated_bytes_and_first_wave_contention():
    """tiles where every byte is its own pre-token (512 words per warp slice), and thousands of tiles that meet the same
    few new words at the same time (owner / polling protocol)."""
    js, alpha = rand_wp_json(random.Random(6), n_words=60, pretok="BertPreTokenizer")
    t, o = pair(js)
    docs = [b"!" * 9000, b"?!.,;" * 2000, b"a!b?c.d" * 1500, b"...", b""] + [b"hello, world! " * 300] * 400
    assert_same(t.encode_batch(docs), o.encode_batch(docs, threads=8))
    assert t.stats().path == 2
    t.close()
    js = tokenizers_io.tokenizer_json("gpt2_whitespace")
    t, o = pair(js)
    docs = [b"the quick brown fox jumps over the lazy dog " * 100] * 3000
    for rep in range(3):
        assert_same(t.encode_batch(docs), o.encode_batch(docs, threads=8), f"contention call {rep}")
    t.close()


def test_tiles_errors_report_the_first_document_in_text_order():
    js = json.dumps({"model": {"type": "BPE", "vocab": {"a": 0, "b": 1, "ab": 2}, "merges": ["a b"]}, "pre_tokenizer": {"type": "Whitespace"}})
    t, o = pair(js)
    filler = [b"ab ab a b"] * 5000
    for bad_at, bad in ((4000, b"ab \xff"), (1234, b"ab " + b"a" * 30 + b"\xc3"), (0, b"\x80"), (4999, b"a" * 100 + b"\xff")):
        docs = list(filler); docs[bad_at] = bad; docs[4500] = b"\xfe"
        with pytest.raises(tz.TokzigError) as e:
            t.encode_batch(docs)
        assert e.value.code == tz.ERR_INVALID_UTF8 and e.value.doc == min(bad_at, 4500)
    assert_same(t.encode_batch(filler), o.encode_batch(filler), "after errors")
    t.close()


def test_full_size_properties_1gib():
    """BASELINE.json configs[1] at its full size (1 GiB of the c2 corpus, GPT-2-shaped tokenizer), through properties that
    need no oracle run: (1) batch-split invariance -- the encoding of the whole batch equals the concatenation of the
    encodings of its halves (different slice / chunk / table-occupancy layout); (2) the slice pipeline equals the
    per-occurrence pipeline on all 235 M tokens; (3) token strings of sampled documents concatenate to the document minus
    the characters the vocabulary lacks; (4) CSR offsets are monotone and end at the token count; (5) the oracle on the same GiB, every id and offset."""
    js = tokenizers_io.tokenizer_json("gpt2_whitespace")
    text, off = corpus.generate("c2", 1 << 30, seed=1234)
    nd = len(off) - 1
    t = tz.Tokenizer.from_json(js, device=0)
    full = t.encode_packed(text, off, outputs=3)
    assert t.stats().path == 2
    assert int(full.doc_tok_off[-1]) == len(full.ids) and np.all(np.diff(full.doc_tok_off.astype(np.int64)) >= 0)
    h = nd // 2
    a = t.encode_packed(text[: int(off[h])], off[: h + 1], outputs=3)
    b = t.encode_packed(text[int(off[h]):], off[h:] - off[h], outputs=3)
    na = len(a.ids)
    assert na + len(b.ids) == len(full.ids)
    assert np.array_equal(full.ids[:na], a.ids) and np.array_equal(full.ids[na:], b.ids)
    assert np.array_equal(full.offsets[:na], a.offsets) and np.array_equal(full.offsets[na:], b.offsets)
    assert np.array_equal(full.doc_tok_off[: h + 1], a.doc_tok_off) and np.array_equal(full.doc_tok_off[h:], b.doc_tok_off + a.doc_tok_off[-1])
    del a, b
    t0, _ = pair(js, mode="occurrence")
    old = t0.encode_packed(text, off, outputs=3)
    assert t0.stats().path == 0
    assert np.array_equal(old.ids, full.ids) and np.array_equal(old.offsets, full.offsets) and np.array_equal(old.doc_tok_off, full.doc_tok_off)
    del old
    t0.close()
    # (5) and the oracle itself on the whole GiB (literal BPE.tokenize on all host cores: a few seconds per GiB here)
    import os
    o = orc.OracleTokenizer.from_json(js)
    ref = o.encode_packed(text, off, algo=0, threads=os.cpu_count() or 1)
    assert np.array_equal(ref.ids, full.ids) and np.array_equal(ref.offsets, full.offsets) and np.array_equal(ref.doc_tok_off, full.doc_tok_off)
    del ref
    d = t.model_desc()
    id2tok = {int(i): k for k, i in zip(d["keys"], d["ids"])}
    single = {k for k in d["keys"] if len(k.decode("utf-8", "ignore")) == 1}
    rng = random.Random(5)
    for i in rng.sample(range(nd), 300):
        doc = text[int(off[i]):int(off[i + 1])].tobytes()
        kept = b"".join(ch.encode() for w in doc.split() for ch in w.decode("utf-8") if ch.encode() in single)
        sl = full.doc_slice(i)
        assert b"".join(id2tok[int(x)] for x in full.ids[sl]) == kept
    t.close()


@pytest.mark.parametrize("model", ["bpe", "wp"])
def test_tiles_words_of_16_to_31_bytes_share_prefixes(model):
    """words of 16..31 bytes take the lane-parallel 64-byte slots: the first half of the key ([length, bytes 0..14]) is
    claimed by CAS, the second half compared afterwards -- so words that share their first 15 bytes (and length), words
    with NUL bytes in either half, and the neighbours 15 / 32 bytes long must all stay distinct."""
    rng = random.Random(77)
    if model == "bpe":
        js, alpha = rand_bpe_json(rng, n_merges=60, alphabet=list("abcd") + ["é"], pretok="Whitespace", dead_merges=0.0)
    else:
        js, alpha = rand_wp_json(rng, n_words=80, alphabet=list("abcd") + ["é"], pretok="Whitespace", normalizer=None, max_chars=40)
    t, o = pair(js)
    stems = ["".join(rng.choice("abcd") for _ in range(15)) for _ in range(6)] + ["a" * 15, "\x00" * 15 if model == "wp" else "b" * 15]
    words = []
    for st in stems:
        for L in (15, 16, 17, 20, 30, 31, 32, 33):
            for _ in range(6):
                tail = "".join(rng.choice("abcd" + ("\x00" if model == "wp" else "")) for _ in range(L - 15))
                words.append((st + tail).encode())
    docs = [b" ".join(rng.choice(words) for _ in range(rng.randint(1, 40))) for _ in range(6000)]
    for rep in range(2):
        assert_same(t.encode_batch(docs), o.encode_batch(docs, threads=8), f"{model} call {rep}")
    assert t.stats().path == 2
    t.close()


def test_tiles_capacity_estimate_exceeded_falls_back_then_adapts():
    """a batch that needs more token records than the slice pipeline reserved (millions of distinct multi-token words in
    a few MiB) is run again with worst-case capacities -- same result -- and the context sizes the next batch from what
    this one needed, so the same batch then needs no second run."""
    rng = random.Random(99)
    v = {c: i for i, c in enumerate("abcdefghijklmnopqrstuvwxyz")}
    js = json.dumps({"model": {"type": "BPE", "vocab": v, "merges": []}, "pre_tokenizer": {"type": "Whitespace"}})
    t, o = pair(js)
    n_words = 300000                                   # 15 one-character tokens each: 4.5 M records > N / 8 + 2^20
    raw = rng.randbytes(n_words * 15)
    letters = bytes(97 + (b % 26) for b in raw)
    docs = [b" ".join(letters[i * 15:(i + 1) * 15] for i in range(j, min(j + 40, n_words))) for j in range(0, n_words, 40)]
    ref = o.encode_batch(docs, threads=8)
    assert_same(t.encode_batch(docs), ref, "first call")
    assert t.stats().path == 2 and t.stats().model_flags & 4, "expected the worst-case re-run on the first call"
    assert_same(t.encode_batch(docs), ref, "second call")
    assert t.stats().path == 2 and not (t.stats().model_flags & 4), "the second call should fit the adapted capacities"
    t.close()


# ----------------------------------------------------------------------------- decode on the GPU (tkz_decode.cuh)
def test_decode_batch_on_gpu_matches_host_decode_and_oracle():
    """Tokenizer.decode (src/lib.zig:163-189) for a batch: the reference's known answers, then random id sequences with
    every decoder kind, ids outside the vocabulary, special ids, '#' runs and C4 A0 pairs that only form ACROSS token
    boundaries, sequences longer than one 32-byte step, empty sequences -- against the host decode and the oracle."""
    js = json.dumps({"model": {"type": "WordPiece", "vocab": {"[PAD]": 0, "[CLS]": 1, "[SEP]": 2, "hello": 3}},
                     "added_tokens": [{"id": 1, "content": "[CLS]", "special": True}, {"id": 2, "content": "[SEP]", "special": True}]})
    t, o = pair(js)
    assert t.decode_batch([[1, 3, 2], [], [3]], False) == [b"[CLS]hello[SEP]", b"", b"hello"]          # src/lib.zig:652-686
    assert t.decode_batch([[1, 3, 2], [], [3]], True) == [b"hello", b"", b"hello"]
    t.close()
    rng = random.Random(11)
    for dec in (None, "WordPiece", "BPE", "ByteLevel"):
        vocab = {"[UNK]": 0, "a": 1, "##b": 2, "#": 3, "\u0120c": 4, "d##": 5, "[X]": 6, "\u00c4": 7, "###": 8, "x" * 40: 9, "": 10}
        root = {"model": {"type": "WordPiece", "vocab": vocab},
                "added_tokens": [{"id": 6, "content": "[X]", "special": True}, {"id": 1, "content": "a", "special": False}, {"id": 40, "content": "[Y]", "special": True}]}
        if dec:
            root["decoder"] = {"type": dec}
        t, o = pair(json.dumps(root, ensure_ascii=False))
        seqs = [[rng.randrange(0, 13) for _ in range(rng.choice([0, 1, 2, 5, 12, 40, 200]))] for _ in range(300)]
        seqs += [[3] * n for n in (1, 2, 3, 31, 32, 33, 64, 65, 1000)] + [[5, 2] * 20, [7, 4] * 30, [], [10, 10], [99, 40]]
        for skip in (False, True):
            got = t.decode_batch(seqs, skip)
            for ids, g in zip(seqs, got):
                assert g == t.decode(ids, skip) == o.decode(ids, skip), (dec, skip, ids[:20])
        t.close()


def test_decode_round_trip_at_size():
    """encode a corpus sample on the GPU, decode every document's ids on the GPU: with a vocabulary whose single-codepoint
    keys cover the text and no decoder rewriting, the decoded bytes are the document without its separators."""
    js = tokenizers_io.tokenizer_json("gpt2_whitespace")
    t = tz.Tokenizer.from_json(js, device=0)
    text, off = corpus.generate("c2", 24 << 20, seed=3)
    enc = t.encode_packed(text, off, outputs=1)
    nd = len(off) - 1
    seqs = [enc.ids[enc.doc_slice(i)] for i in range(nd)]
    dec = t.decode_batch(seqs)
    d = t.model_desc()
    single = {k for k in d["keys"] if len(k.decode("utf-8", "ignore")) == 1}
    rng = random.Random(4)
    for i in rng.sample(range(nd), 300):
        doc = text[int(off[i]):int(off[i + 1])].tobytes()
        kept = b"".join(ch.encode() for w in doc.split() for ch in w.decode("utf-8") if ch.encode() in single)
        assert t.decode(seqs[i]) == dec[i]
        if b"\xc4\xa0" not in kept and b"##" not in kept:               # whatever decoder the JSON names leaves these documents alone
            assert dec[i] == kept
    t.close()


# ----------------------------------------------------------------------------- compact result / packed formats
@pytest.mark.parametrize("seed", range(12))
def test_compact_result_expands_to_the_reference_encoding(seed):
    """tkz_encode_batch_compact ships kept ids (u16 when the vocabulary allows) + one u16 of offsets per token and nothing that is a
    constant of the parameters; tkz_compact_expand must rebuild the reference's six arrays bit-exactly (truncation, left and
    right padding, documents without tokens), for the whole batch and for any document range."""
    rng = random.Random(4200 + seed)
    if seed % 2:
        js, alpha = rand_wp_json(rng)
    else:
        js, alpha = rand_bpe_json(rng, n_merges=30, pretok="Whitespace")
    t, o = pair(js, mode=MODES[seed % 3])
    docs = rand_docs(rng, alpha, 300, max_len=60) + [b"", b"   "]
    trunc = [None, 0, 1, 5, 8, 64][seed % 6]
    pad = [None, {"length": 8, "pad_id": 7, "pad_type_id": 3, "direction": "right"}, {"length": 5, "pad_id": 0, "direction": "left"},
           {"length": None, "pad_id": 9}][(seed // 2) % 4]
    t.truncation = None if trunc is None else {"max_length": trunc}
    o.truncation = trunc
    t.padding = pad
    o.padding = pad
    ref = o.encode_batch(docs)
    text, off = tz.pack_docs(docs)
    r = t.encode_compact(text, off)
    assert r.ids16 and not r.ids, "small vocabulary: ids must travel as u16"
    if MODES[seed % 3] != "occurrence":
        assert r.offsets_packed and not r.offsets
    assert_same(tz.expand_compact(r), ref, f"seed {seed} trunc {trunc} pad {pad}")
    lo, hi = 17, 203
    part = tz.expand_compact(r, lo, hi)
    a, b = int(ref.doc_tok_off[lo]), int(ref.doc_tok_off[hi])
    assert np.array_equal(part.doc_tok_off, ref.doc_tok_off[lo:hi + 1] - ref.doc_tok_off[lo])
    assert np.array_equal(part.ids, ref.ids[a:b]) and np.array_equal(part.offsets, ref.offsets[a:b])
    assert np.array_equal(part.attention_mask, ref.attention_mask[a:b]) and np.array_equal(part.type_ids, ref.type_ids[a:b])
    assert np.array_equal(part.special_tokens_mask, ref.special_tokens_mask[a:b])
    # ids only
    r2 = t.encode_compact(text, off, want_offsets=False)
    assert not r2.offsets_packed and not r2.offsets
    assert np.array_equal(tz.expand_compact(r2).ids, ref.ids)
    t.close()


def test_packed_formats_fall_back_when_they_cannot_hold_the_values(monkeypatch):
    """offsets_packed: tokens of pre-tokens of 256 bytes or more carry 0xFFFF and their offsets travel in a side list; when
    such tokens are many (an eighth of the call's tokens) the whole call -- every chunk of the host path -- delivers 32-bit
    offsets; ids16 needs every vocabulary id below 65536."""
    rng = random.Random(77)
    js, alpha = rand_bpe_json(rng, n_merges=40, alphabet=list("abcdefg"), pretok="Whitespace", dead_merges=0.0)
    t, o = pair(js)
    short = [b" ".join(bytes(rng.choice(b"abcdefg") for _ in range(rng.randint(1, 40))) for _ in range(rng.randint(1, 30))) for _ in range(2000)]
    long_doc = b"ab " + bytes(rng.choice(b"abcdefg") for _ in range(300)) + b" cd"
    many_long = [b"x " + bytes(rng.choice(b"abcdefg") for _ in range(rng.randint(256, 2000))) for _ in range(1500)]
    for docs, packed, wide in ((short, True, False), (short[:1000] + [long_doc] + short[1000:] + [long_doc, b"", long_doc[3:]], True, True),
                               (short[:50] + many_long + short[50:100], False, False)):
        for chunk in (1 << 31, 16384):
            monkeypatch.setenv("TKZ_CHUNK_BYTES", str(chunk))
            t2 = tz.Tokenizer.from_json(js, device=0)
            text, off = tz.pack_docs(docs)
            got = t2.encode_packed(text, off, outputs=tz.OUT_IDS | tz.OUT_OFFSETS_PACKED | tz.OUT_IDS_U16)
            ref = o.encode_batch(docs, threads=4)
            assert (got.offsets_packed is not None) == packed and (got.offsets is not None) == (not packed)
            assert (got.wide_tokens is not None and len(got.wide_tokens) > 0) == wide
            if wide:
                slots = got.wide_tokens[:, 0].astype(np.int64) | (got.wide_tokens[:, 1].astype(np.int64) << 32)
                assert np.all(np.diff(slots) > 0)                       # sorted by slot, no duplicates
                assert int((got.offsets_packed == 0xFFFF).sum()) == len(slots)
            assert np.array_equal(got.ids, ref.ids) and np.array_equal(got.unpacked_offsets(), ref.offsets) and np.array_equal(got.doc_tok_off, ref.doc_tok_off)
            r = t2.encode_compact(text, off)
            assert bool(r.offsets_packed) == packed and (r.n_wide > 0) == wide
            assert_same(tz.expand_compact(r), ref, f"packed={packed} chunk={chunk}")
            if wide:                                                    # expansion of document ranges that start behind a wide token
                nd = len(docs)
                for d0, d1 in ((1001, nd), (nd - 3, nd - 1), (nd - 1, nd), (0, 1000)):
                    part = tz.expand_compact(r, d0, d1)
                    a, b = int(ref.doc_tok_off[d0]), int(ref.doc_tok_off[d1])
                    assert np.array_equal(part.ids, ref.ids[a:b]) and np.array_equal(part.offsets, ref.offsets[a:b])
            t2.close()
    t.close()
    # vocabulary ids above 65535: ids stay u32
    v = {c: 70000 + i for i, c in enumerate("abcd")}
    v["ab"] = 70010
    js2 = json.dumps({"model": {"type": "BPE", "vocab": v, "merges": ["a b"]}, "pre_tokenizer": {"type": "Whitespace"}})
    t3, o3 = pair(js2)
    docs = [b"ab abcd", b"", b"dcba ab"]
    text, off = tz.pack_docs(docs)
    r = t3.encode_compact(text, off)
    assert r.ids and not r.ids16
    assert_same(tz.expand_compact(r), o3.encode_batch(docs))
    t3.close()
    # no pre-tokenizer: a pre-token can have any length, offsets are always 32-bit
    js3 = json.dumps({"model": {"type": "BPE", "vocab": {"a": 0, "b": 1, "ab": 2}, "merges": ["a b"]}})
    t4, o4 = pair(js3)
    docs = [b"abab" * 100, b"ba"]
    text, off = tz.pack_docs(docs)
    r = t4.encode_compact(text, off)
    assert r.offsets and not r.offsets_packed
    assert_same(tz.expand_compact(r), o4.encode_batch(docs))
    t4.close()


# ----------------------------------------------------------------------------- several contexts, one host thread each (tkzm_*)
@pytest.mark.parametrize("cost_balanced", [False, True])
def test_multi_context_pool_matches_the_oracle(cost_balanced):
    """tkzm_encode_batch_compact: the batch cut into shards (by bytes / by the cost model), one context and one host thread
    per shard running concurrently (here: three contexts on the same GPU), shard results expanded and concatenated in
    document order == the oracle; the caller's current device is left alone; errors carry the batch-wide document index."""
    import torch
    text, off = corpus.generate("c5", 12 << 20, seed=5)
    for name, trunc, pad in (("gpt2_whitespace", None, None), ("bert_wordpiece", 16, {"length": 24, "pad_id": 0, "direction": "left"})):
        js = tokenizers_io.tokenizer_json(name)
        cfg = tz.Tokenizer.from_json(js, device=None)
        cfg.truncation = None if trunc is None else {"max_length": trunc}
        cfg.padding = pad
        o = orc.OracleTokenizer.from_json(js)
        o.truncation = trunc; o.padding = pad
        ng = torch.cuda.device_count()
        pool = tz.MultiPool(cfg, [k % ng for k in range(3)])            # distinct GPUs when the box has them
        before = torch.cuda.current_device()
        got = pool.encode_expanded(text, off, cost_balanced=cost_balanced)
        assert torch.cuda.current_device() == before
        assert_same(got, o.encode_packed(text, off, algo=1, threads=8), f"{name} cost_balanced={cost_balanced}")
        bounds, results, ms = pool.encode_compact(text, off, cost_balanced=cost_balanced)
        assert bounds[0] == 0 and bounds[-1] == len(off) - 1 and np.all(np.diff(bounds.astype(np.int64)) >= 0) and np.all(ms > 0)
        pool.close(); cfg.close()
    # error in the last shard: document index of the whole batch
    js = json.dumps({"model": {"type": "BPE", "vocab": {"a": 0, "b": 1, "ab": 2}, "merges": ["a b"]}, "pre_tokenizer": {"type": "Whitespace"}})
    cfg = tz.Tokenizer.from_json(js, device=None)
    pool = tz.MultiPool(cfg, [0, 0])
    docs = [b"ab ab"] * 50 + [b"ab \xffab"] + [b"ab"] * 3
    t_, o_ = tz.pack_docs(docs)
    with pytest.raises(tz.TokzigError) as e:
        pool.encode_compact(t_, o_)
    assert e.value.code == tz.ERR_INVALID_UTF8 and e.value.doc == 50
    pool.close(); cfg.close()


def test_decode_batch_refuses_a_batch_that_decodes_to_4gib_or_more():
    """token byte offsets of the decode path are 32-bit: a batch whose decoded bytes reach 4 GiB (here 4100 ids of a 1 MiB
    token) must be refused with the request to split it, not wrapped; the same ids in two halves decode."""
    big = "x" * (1 << 20)
    js = json.dumps({"model": {"type": "WordPiece", "vocab": {"[UNK]": 0, big: 1, "ab": 2}, "unk_token": "[UNK]"}})
    t = tz.Tokenizer.from_json(js, device=0)
    with pytest.raises(tz.TokzigError) as e:
        t.decode_batch([[1] * 2050, [2], [1] * 2050])
    assert e.value.code == tz.ERR_INVALID_ARG and "split" in str(e.value)
    out = t.decode_batch([[1] * 40, [2, 1, 2]])
    assert len(out[0]) == 40 << 20 and out[1] == b"ab" + big.encode() + b"ab"
    t.close()


# ----------------------------------------------------------------------------- FastTokenizer mode (tkz_fast.cuh)
@pytest.mark.parametrize("c", [c for c in CASES if c["kind"] in ("json", "model") and 2 in c["algos"]], ids=lambda c: c["id"])
def test_reference_fast_kats_on_gpu(c):
    """the reference's own known answers for tokenizeFast / FastTokenizer (bpe.zig:709-866, wordpiece.zig tests, lib.zig:957-1174)"""
    js = c["json"] if c["kind"] == "json" else model_case_to_json(c["model"])
    t = tz.Tokenizer.from_json(js, device=0)
    text = bytes.fromhex(c["input_hex"])
    if c.get("error"):
        t.close()
        pytest.skip("error cases belong to Tokenizer.encode (the arena variants do not raise)")
    e = t.encode_fast_batch([text])
    check_encoding_against_case(c, e.ids, e.offsets, e.attention_mask, e.type_ids, np.zeros(len(e.ids), np.uint32))
    t.close()


@pytest.mark.parametrize("seed", range(24))
def test_fast_mode_random_against_the_arena_oracle(seed):
    """FastTokenizer.encode on the GPU == the oracle's restatement of the arena variants (algo 2): heap pop order with equal
    ranks, stale entries merged at their old priority, improper / aliased / degenerate tables, the symbol / pre-token / token
    caps of the arena (small values so that they bind), the WordPiece word that crosses max_tokens before it turns out bad,
    and the 16-byte SpanToken records."""
    rng = random.Random(8100 + seed)
    if seed % 3 == 2:
        js, alpha = rand_wp_json(rng, n_words=rng.choice([20, 80]), with_unk=seed % 6 != 5)
    else:
        js, alpha = rand_bpe_json(rng, n_merges=rng.choice([5, 40, 120]), improper=[0.0, 0.3][seed % 2], degenerate=[0.0, 0.1][(seed // 2) % 2],
                                  alias=[0.0, 0.2][(seed // 4) % 2], pretok=[None, "Whitespace"][(seed // 3) % 2], unk="<unk>" if seed % 5 == 0 else None)
    t = tz.Tokenizer.from_json(js, device=0)
    o = orc.OracleTokenizer.from_json(js)
    docs = rand_docs(rng, alpha, 300, max_len=120) + [b"", b"aaaaa", b"dabc", b"a" * 300, (b"ab " * 200)]
    for max_seq, max_tok in ((8192, 512), (64, 7), (16, 3), (400, 1), (8, 100)):
        o.set_fast_options(max_seq, max_tok)
        ref = o.encode_batch(docs, algo=2, threads=4)
        got = t.encode_fast_batch(docs, max_sequence_length=max_seq, max_tokens=max_tok)
        assert np.array_equal(got.doc_tok_off, ref.doc_tok_off), f"seed {seed} caps {max_seq}/{max_tok}: doc_tok_off"
        assert np.array_equal(got.ids, ref.ids), f"seed {seed} caps {max_seq}/{max_tok}: ids"
        assert np.array_equal(got.offsets, ref.offsets), f"seed {seed} caps {max_seq}/{max_tok}: offsets"
        assert np.all(got.attention_mask == 1) and np.all(got.type_ids == 0)
        sp = got.span_tokens
        assert np.array_equal(sp[:, 0], ref.ids) and np.array_equal(sp[:, 1:3], ref.offsets) and np.all(sp[:, 3] == 0)
    t.close()


def test_span_token_records_of_the_padded_encoding():
    """TKZ_OUT_SPAN_TOKENS next to the CSR arrays of Tokenizer.encode: real slots {id, start, end, 0}, padding slots
    SpanToken.initPadding(pad_id) = {pad_id, 0, 0, flags.is_padding} (token.zig:52-54)."""
    rng = random.Random(3)
    js, alpha = rand_wp_json(rng)
    t, o = pair(js)
    t.truncation = {"max_length": 6}; o.truncation = 6
    pad = {"length": 9, "pad_id": 5, "pad_type_id": 2, "direction": "right"}
    t.padding = pad; o.padding = pad
    docs = rand_docs(rng, alpha, 200, max_len=60)
    got = t.encode_batch(docs, outputs=tz.OUT_ALL | tz.OUT_SPAN_TOKENS)
    ref = o.encode_batch(docs)
    assert_same(got, ref)
    sp = got.span_tokens
    real = ref.attention_mask == 1
    assert np.array_equal(sp[:, 0], ref.ids) and np.array_equal(sp[:, 1:3], ref.offsets)
    assert np.all(sp[real, 3] == 0) and np.all(sp[~real, 3] == 0x0400)
    t.close()
