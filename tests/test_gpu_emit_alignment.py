"""GPU: pass B of the slice pipeline (tkz_slices.cuh, slice_emit_kernel) at the edges of its copy.  Without truncation or
padding, the ids + offsets + attention form and the generic form read each slice's run of the token stream through 1 KiB
shared-memory windows that start at a 16-byte boundary of the stream; ids + offsets + attention is written 4 tokens per
lane at 4-aligned destination slots, token by token at the ends of a range.  The other forms keep per-lane loads and
stores.  The text below is laid out slice by slice (1 KiB each) so that the slices have chosen token counts -- 0, 1, 3,
4, 5, 255, 256, 257 and 1274 (next to TW_SLICE_TOK_MAX) -- in an order that puts every run at every destination residue
mod 8, next to long words (more than 255 bytes, copied from the pool) and a partial last slice; one batch has enough
slices that every warp of pass B walks several of them.  Every result is held to the CPU oracle, in both record forms,
for every output mask the benchmark uses, with truncation and padding left and right."""
import json
import os
import random

import numpy as np
import pytest

import tokzig_b200 as tz
from oracle import oracle as orc

SLICE = 1024
# one token per letter (no merges among f, g, h), "ab" and "ee" merge; "z" is outside the vocabulary: its words give no token
VOCAB = {c: 65520 + i for i, c in enumerate("abcdefgh")}
VOCAB.update({"ab": 40000, "ee": 9, ".": 77})
BPE = json.dumps({"model": {"type": "BPE", "vocab": VOCAB, "merges": ["a b", "e e"]}, "pre_tokenizer": {"type": "Whitespace"}})
COUNTS = (0, 1, 3, 4, 5, 255, 256, 257)
MASKS = (tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION, tz.OUT_IDS, tz.OUT_IDS | tz.OUT_IDS_U16,
         tz.OUT_IDS | tz.OUT_IDS_U16 | tz.OUT_OFFSETS_PACKED, tz.OUT_IDS | tz.OUT_OFFSETS_PACKED, tz.OUT_ALL)


def gpu(record):
    """a context whose token stream takes the given record form (read when the context is created)"""
    if record == "wide":
        os.environ["TKZ_TOK_RECORD"] = "wide"
    try:
        return tz.Tokenizer.from_json(BPE, device=0)
    finally:
        os.environ.pop("TKZ_TOK_RECORD", None)


def slice_bytes(rng, k):
    """1 KiB whose words starting in it have k tokens: k words "a" or "f" (1 token, 2 bytes) and "z" filler"""
    assert 2 * k <= SLICE
    words = [rng.choice("af") for _ in range(k)]
    body = " ".join(words) + " " if k else ""
    fill = SLICE - len(body)
    while fill > 0:                                       # filler words of up to 15 bytes, each followed by a space
        n = min(fill, rng.randint(2, 16))
        body += "z" * (n - 1) + " " if n > 1 else " "
        fill -= n
    assert len(body) == SLICE
    return body


DENSE = " ".join(["fgh" * 85] * 3 + ["fgh" * 84 + "fg"]) + " " + "fgh" * 85 + " "
"""a slice of words of 254 and 255 single-letter tokens (words longer than 255 bytes would leave pass A for the long-word
list), the last one starting at the slice's last byte: 3 * 255 + 254 + 255 = 1274 tokens start in it, next to the bound
pass A reserves for one slice (TW_SLICE_TOK_MAX = 1280)"""
DENSE_TOKENS = 3 * 255 + 254 + 255
assert DENSE.rindex(" f") + 1 == SLICE - 1


def layout(seed, n_slices=600):
    """the text of a batch slice by slice, cut into documents at random byte positions (a cut splits no token of these
    words: every letter but "ab" is a token of its own).  Returns the documents and, for every slice laid out with a chosen
    count, (count, tokens before it)."""
    rng = random.Random(seed)
    text, plan, before = "", [], 0
    for i in range(n_slices):
        r = rng.random()
        if r < 0.03:                                      # a long word (> 255 bytes) in the middle of a slice: pool pieces
            n = rng.randint(90, 200)
            text += "a " * 100 + "fgh" * n + " "
            before += 100 + 3 * n
        elif r < 0.05:
            text += DENSE
            before += DENSE_TOKENS
        else:
            k = rng.choice(COUNTS)
            plan.append((k, before))
            text += slice_bytes(rng, k)
            before += k
        text += " " * (-len(text) % SLICE)                # the next slice starts at a slice boundary
    text += "ab a f " * rng.randint(1, 60)                 # a partial last slice
    data = text.encode()
    cuts = sorted(rng.sample(range(1, len(data)), 150))
    bounds = [0] + cuts + [len(data)]
    return [data[bounds[i]:bounds[i + 1]] for i in range(len(bounds) - 1)], plan


def assert_same(got, ref, mask, what):
    assert np.array_equal(got.doc_tok_off, ref.doc_tok_off), f"{what}: doc_tok_off"
    if not np.array_equal(got.ids, ref.ids):
        bad = int(np.nonzero(got.ids != ref.ids)[0][0]) if len(got.ids) == len(ref.ids) else -1
        raise AssertionError(f"{what}: ids differ (first at {bad}, {len(got.ids)} vs {len(ref.ids)} tokens)")
    if mask & (tz.OUT_OFFSETS | tz.OUT_OFFSETS_PACKED):
        assert np.array_equal(got.unpacked_offsets(), ref.offsets), f"{what}: offsets"
    for name, bit in (("attention_mask", tz.OUT_ATTENTION), ("type_ids", tz.OUT_TYPE_IDS), ("special_tokens_mask", tz.OUT_SPECIAL)):
        if mask & bit:
            assert np.array_equal(getattr(got, name), getattr(ref, name)), f"{what}: {name}"


def test_layout_has_the_edges():
    """(CPU) the layout keeps its promise: slices of every chosen count, each at every destination residue mod 8, and the
    token total the oracle finds"""
    docs, plan = layout(2)
    for k in COUNTS:
        assert {b % 8 for kk, b in plan if kk == k} == set(range(8)), k
    ref = orc.OracleTokenizer.from_json(BPE).encode_batch(docs)
    assert len(ref.ids) > plan[-1][1] + plan[-1][0]


@pytest.mark.gpu
@pytest.mark.parametrize("record", ("narrow", "wide"))
@pytest.mark.parametrize("mask", MASKS)
def test_every_slice_shape_and_residue(record, mask):
    docs, _ = layout(2)
    t, o = gpu(record), orc.OracleTokenizer.from_json(BPE)
    ref = o.encode_batch(docs)
    assert_same(t.encode_batch(docs, outputs=mask), ref, mask, f"{record} mask {mask}")
    assert t.stats().path == 2 and t.stats().n_long_words > 0
    # the same batch shifted by 1..7 tokens at the front: every run moves to every other destination residue
    for k in range(1, 8):
        lead = [(" ".join(["a"] * k)).encode()]
        assert_same(t.encode_batch(lead + docs, outputs=mask), o.encode_batch(lead + docs), mask, f"{record} mask {mask} lead {k}")
    t.close()


@pytest.mark.gpu
@pytest.mark.parametrize("record", ("narrow", "wide"))
def test_slice_at_the_token_bound(record):
    """the dense slice alone and between sparse ones: 1274 tokens of one slice, all of them inline (no long word)"""
    rng = random.Random(5)
    text = DENSE + " " * (-len(DENSE) % SLICE)
    docs = [text.encode(), (slice_bytes(rng, 3) + text + slice_bytes(rng, 257)).encode(), text.encode() * 3]
    t, o = gpu(record), orc.OracleTokenizer.from_json(BPE)
    ref = o.encode_batch(docs)
    assert int(ref.doc_tok_off[1]) == DENSE_TOKENS
    for mask in (tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION, tz.OUT_ALL, tz.OUT_IDS):
        assert_same(t.encode_batch(docs, outputs=mask), ref, mask, f"{record} mask {mask}")
        assert t.stats().path == 2 and t.stats().n_long_words == 0
    t.close()


@pytest.mark.gpu
@pytest.mark.parametrize("record", ("narrow", "wide"))
@pytest.mark.parametrize("mask", [tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION, tz.OUT_ALL, tz.OUT_IDS | tz.OUT_IDS_U16])
def test_warps_walk_many_slices(record, mask):
    """pass B runs at most 16 blocks of 8 warps per SM, each warp taking every (grid warps)-th slice: with three times
    as many slices every warp writes several, so the first window of a warp's next slice is issued while the current one
    is written, across empty, tiny, dense and long-word slices"""
    import torch
    n_slices = 3 * 16 * 8 * torch.cuda.get_device_properties(0).multi_processor_count
    docs, _ = layout(4, n_slices=n_slices)
    t, o = gpu(record), orc.OracleTokenizer.from_json(BPE)
    assert_same(t.encode_batch(docs, outputs=mask), o.encode_batch(docs, threads=8), mask, f"{record} mask {mask}")
    assert t.stats().path == 2
    t.close()


@pytest.mark.gpu
@pytest.mark.parametrize("record", ("narrow", "wide"))
@pytest.mark.parametrize("mask", [tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION, tz.OUT_IDS | tz.OUT_IDS_U16, tz.OUT_ALL])
@pytest.mark.parametrize("trunc,pad", [(7, None), (300, {"length": 301, "pad_id": 3, "direction": "right"}),
                                       (250, {"length": 260, "pad_id": 0, "pad_type_id": 1, "direction": "left"}),
                                       (None, {"length": 2000, "pad_id": 1, "direction": "left"})])
def test_truncation_and_padding_pieces(record, mask, trunc, pad):
    docs, _ = layout(3, n_slices=300)
    t, o = gpu(record), orc.OracleTokenizer.from_json(BPE)
    t.truncation = None if trunc is None else {"max_length": trunc}
    o.truncation = trunc
    t.padding = pad
    o.padding = pad
    assert_same(t.encode_batch(docs, outputs=mask), o.encode_batch(docs), mask, f"{record} trunc {trunc} pad {pad}")
    t.close()


@pytest.mark.gpu
def test_worst_case_retry_writes_the_same_tokens():
    """a batch whose first pass A runs out of its record pool is run again with worst-case capacities; pass B then reads
    runs that lie anywhere in a larger token stream"""
    rng = random.Random(99)
    v = {c: i for i, c in enumerate("abcdefghijklmnopqrstuvwxyz")}
    js = json.dumps({"model": {"type": "BPE", "vocab": v, "merges": []}, "pre_tokenizer": {"type": "Whitespace"}})
    t, o = tz.Tokenizer.from_json(js, device=0), orc.OracleTokenizer.from_json(js)
    n_words = 300000
    letters = bytes(97 + (b % 26) for b in rng.randbytes(n_words * 15))
    docs = [b" ".join(letters[i * 15:(i + 1) * 15] for i in range(j, min(j + rng.randint(1, 60), n_words))) for j in range(0, n_words, 40)]
    mask = tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION
    assert_same(t.encode_batch(docs, outputs=mask), o.encode_batch(docs, threads=8), mask, "retry")
    assert t.stats().path == 2 and t.stats().model_flags & 4, "expected the worst-case re-run"
    t.close()
