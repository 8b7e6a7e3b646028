"""GPU: the token stream between the two passes of the slice pipeline (tkz_slices.cuh) in both record forms.  A 16-bit
vocabulary gets 4-byte records (id u16 + offsets u8,u8) or u16 ids; TKZ_TOK_RECORD=wide forces u32 ids and 8-byte records.
Each case runs in both forms and is held to the CPU oracle on every array the call delivers: the output masks that pass B
has compile-time forms for, hf_compat with and without document offsets, truncation and padding, words of 0..6 tokens,
words at the 15 / 16-byte slot boundary, 65..255-byte words (end offsets up to 255), errors, and the contention and
table-pressure shapes.  Vocabularies with ids of 65536 and more (llama3_whitespace) keep the wide records: a narrow record
would cut their ids, which the oracle comparison would see."""
import json
import os
import random

import numpy as np
import pytest

import tokzig_b200 as tz
from oracle import oracle as orc
from gen_util import rand_bpe_json
from test_hf_compat_oracle import VEC, oracle_for
from tools import corpus, tokenizers_io

pytestmark = pytest.mark.gpu

RECORDS = ("narrow", "wide")
MASKS = (tz.OUT_IDS, tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION, tz.OUT_IDS | tz.OUT_OFFSETS_PACKED,
         tz.OUT_IDS | tz.OUT_IDS_U16 | tz.OUT_OFFSETS_PACKED, tz.OUT_IDS | tz.OUT_IDS_U16, tz.OUT_ALL)

# ids at the top of the 16-bit range: a narrow record must keep every id bit apart from the offset bytes
LETTERS = "abcdefgh"
SMALL_VOCAB = {c: 65528 + i for i, c in enumerate(LETTERS)}
SMALL_VOCAB.update({"ab": 40000, "cd": 300, "abcd": 7, "ee": 65000})
SMALL_BPE = json.dumps({"model": {"type": "BPE", "vocab": SMALL_VOCAB, "merges": ["a b", "c d", "ab cd", "e e"]},
                        "pre_tokenizer": {"type": "Whitespace"}})


def gpu(js, record):
    """a context whose token stream takes the given record form (read when the context is created)"""
    if record == "wide":
        os.environ["TKZ_TOK_RECORD"] = "wide"
    try:
        t = tz.Tokenizer.from_json(js, device=0)
    finally:
        os.environ.pop("TKZ_TOK_RECORD", None)
    return t


def assert_same(got, ref, mask, what=""):
    assert np.array_equal(got.doc_tok_off, ref.doc_tok_off), f"{what}: doc_tok_off"
    assert np.array_equal(got.ids, ref.ids), f"{what}: ids"
    if mask & (tz.OUT_OFFSETS | tz.OUT_OFFSETS_PACKED):
        assert np.array_equal(got.unpacked_offsets(), ref.offsets), f"{what}: offsets"
    for name, bit in (("attention_mask", tz.OUT_ATTENTION), ("type_ids", tz.OUT_TYPE_IDS), ("special_tokens_mask", tz.OUT_SPECIAL)):
        if mask & bit:
            assert np.array_equal(getattr(got, name), getattr(ref, name)), f"{what}: {name}"


def small_docs(rng, n_docs):
    """words of 0..6 tokens, of 15 and 16 bytes, of 65..255 bytes, next to each other and at document ends"""
    def word(L, alpha=LETTERS):
        return "".join(rng.choice(alpha) for _ in range(L))
    shapes = [lambda: "zz",                                  # no token: bytes outside the vocabulary are dropped
              lambda: "a", lambda: "ab", lambda: "abh", lambda: "abcdh", lambda: "abcdabcdfg", lambda: "fghfgh",
              lambda: "hgfedc"[:rng.randint(1, 6)], lambda: word(rng.randint(1, 6)),
              lambda: word(15), lambda: word(16), lambda: word(14) + "z", lambda: "ab" * 7 + "c", lambda: "ab" * 8,
              lambda: word(rng.randint(65, 255)), lambda: word(255), lambda: "ee" * 100]
    docs = []
    for _ in range(n_docs):
        docs.append(" ".join(rng.choice(shapes)() for _ in range(rng.randint(0, 40))).encode())
    return docs


@pytest.mark.parametrize("record", RECORDS)
@pytest.mark.parametrize("mask", MASKS)
def test_word_shapes_every_output_form(record, mask):
    rng = random.Random(11)
    docs = small_docs(rng, 3000) + [b"", b"abcd", b"z"]
    t, o = gpu(SMALL_BPE, record), orc.OracleTokenizer.from_json(SMALL_BPE)
    ref = o.encode_batch(docs)
    lens = {int(ref.doc_tok_off[i + 1] - ref.doc_tok_off[i]) for i in range(len(docs))}
    assert len(lens) > 50
    assert_same(t.encode_batch(docs, outputs=mask), ref, mask, f"{record} mask {mask}")
    t.close()


@pytest.mark.parametrize("record", RECORDS)
@pytest.mark.parametrize("mask", [tz.OUT_IDS | tz.OUT_IDS_U16, tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION, tz.OUT_ALL])
@pytest.mark.parametrize("trunc,pad", [(5, None), (None, {"length": 64, "pad_id": 3, "direction": "right"}),
                                       (9, {"length": 12, "pad_id": 0, "pad_type_id": 1, "direction": "left"}),
                                       (None, {"length": 600, "pad_id": 1})])
def test_truncation_and_padding(record, mask, trunc, pad):
    rng = random.Random(12)
    docs = small_docs(rng, 1500)
    t, o = gpu(SMALL_BPE, record), orc.OracleTokenizer.from_json(SMALL_BPE)
    t.truncation = None if trunc is None else {"max_length": trunc}
    o.truncation = trunc
    t.padding = pad
    o.padding = pad
    assert_same(t.encode_batch(docs, outputs=mask), o.encode_batch(docs), mask, f"{record} trunc {trunc} pad {pad}")
    t.close()


@pytest.mark.parametrize("record", RECORDS)
@pytest.mark.parametrize("name,cname,nbytes", [("gpt2_whitespace", "c2", 3 << 20), ("bert_wordpiece", "c3", 3 << 20), ("llama3_whitespace", "c4", 2 << 20)])
@pytest.mark.parametrize("mask", [tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION, tz.OUT_IDS | tz.OUT_IDS_U16 | tz.OUT_OFFSETS_PACKED, tz.OUT_IDS])
def test_synthesised_tokenizers_on_corpus(record, name, cname, nbytes, mask):
    js = tokenizers_io.tokenizer_json(name)
    t, o = gpu(js, record), orc.OracleTokenizer.from_json(js)
    text, off = corpus.generate(cname, nbytes, seed=2025)
    if name == "bert_wordpiece":
        t.truncation = {"max_length": 128}
        o.truncation = 128
        t.padding = {"length": 64, "pad_id": 0}
        o.padding = {"length": 64, "pad_id": 0}
    got = t.encode_packed(text, off, outputs=mask)
    assert t.stats().path == 2
    assert_same(got, o.encode_packed(text, off, threads=8), mask, f"{name} {record}")
    t.close()


@pytest.mark.parametrize("record", RECORDS)
@pytest.mark.parametrize("flags", [tz.HF_TEMPLATE, tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS])
@pytest.mark.parametrize("trunc,pad", [(None, None), (20, {"length": 33, "pad_id": 1, "pad_type_id": 1, "direction": "left"})])
def test_hf_compat_with_and_without_document_offsets(record, flags, trunc, pad):
    """template only: narrow records (pre-token offsets); document offsets: the wide records carry the word's position"""
    suite = VEC["suites"][0]
    js = suite["tokenizer_json"]
    words = [w for w in json.loads(js)["model"]["vocab"] if w.isalpha() and w.islower()][:300] + ["zzqx"]
    rng = random.Random(13)
    docs = [" ".join(rng.choice(words) for _ in range(rng.randint(0, 50))).encode() for _ in range(800)]
    case = {"add_special_tokens": True, "truncation": trunc, "padding": pad}
    o = oracle_for(suite, case)
    prefix, suffix, seq_type = orc.hf_template_from_json(js)
    o.set_hf_compat(flags, prefix, suffix, seq_type)
    t = gpu(js, record)
    assert t.set_hf_compat(flags)
    t.truncation = None if trunc is None else {"max_length": trunc}
    t.padding = pad
    got = t.encode_batch(docs)
    assert t.stats().path == 2
    assert_same(got, o.encode_batch(docs, algo=1), tz.OUT_ALL, f"{record} flags {flags}")
    t.close()


@pytest.mark.parametrize("record", RECORDS)
def test_errors_are_reported_as_before(record):
    t = gpu(SMALL_BPE, record)
    filler = [b"ab cd abcd " * 20] * 2000
    for bad_at, bad in ((1500, b"ab \xff"), (700, b"ab " + b"a" * 30 + b"\xc3"), (1999, b"a" * 100 + b"\xff")):
        docs = list(filler)
        docs[bad_at] = bad
        with pytest.raises(tz.TokzigError) as e:
            t.encode_batch(docs, outputs=tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION)
        assert e.value.code == tz.ERR_INVALID_UTF8 and e.value.doc == bad_at
    t.close()
    js = json.dumps({"model": {"type": "WordPiece", "vocab": {"hello": 1, "##s": 2}, "unk_token": "[UNK]"}, "pre_tokenizer": {"type": "Whitespace"}})
    t, o = gpu(js, record), orc.OracleTokenizer.from_json(js)
    assert_same(t.encode_batch([b"hello hellos"]), o.encode_batch([b"hello hellos"]), tz.OUT_ALL)
    with pytest.raises(tz.TokzigError) as e:
        t.encode_batch([b"hello", b"hello xyz", b"q"], outputs=tz.OUT_IDS)
    assert e.value.code == tz.ERR_MISSING_UNK and e.value.doc == 1
    t.close()


@pytest.mark.parametrize("record", RECORDS)
def test_first_wave_contention(record):
    """thousands of slices meet the same few new words at once: most of them read the value of a word another warp owns"""
    js = tokenizers_io.tokenizer_json("gpt2_whitespace")
    t, o = gpu(js, record), orc.OracleTokenizer.from_json(js)
    docs = [b"the quick brown fox jumps over the lazy dog " * 100] * 3000
    ref = o.encode_batch(docs, threads=8)
    for mask in (tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION, tz.OUT_IDS | tz.OUT_IDS_U16):
        assert_same(t.encode_batch(docs, outputs=mask), ref, mask, f"contention {record}")
    t.close()


@pytest.mark.parametrize("record", RECORDS)
@pytest.mark.parametrize("n_words", [60000, 200000])
def test_table_pressure(record, n_words):
    rng = random.Random(23)
    js, alpha = rand_bpe_json(rng, n_merges=100, alphabet=list("abcdefghijklmnop"), pretok="Whitespace", dead_merges=0.0)
    t, o = gpu(js, record), orc.OracleTokenizer.from_json(js)
    chars = "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789"
    words = ["".join(rng.choice(chars) for _ in range(4)) for _ in range(n_words)]
    docs = [" ".join(words[i:i + 50]).encode() for i in range(0, len(words), 50)]
    mask = tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION
    assert_same(t.encode_batch(docs, outputs=mask), o.encode_batch(docs, threads=8), mask, f"pressure {record}")
    t.close()
