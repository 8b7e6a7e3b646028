#!/usr/bin/env python3
"""Generates tests/golden/hf_overflow_vectors.json.gz: what Hugging Face `tokenizers` (0.22.2) returns with
enable_truncation(max_length, stride) -- the main encoding and every overflowing one of each document -- for the four tokenizers
of tests/golden/hf_compat_vectors.json (the file stores only the suite names; the tokenizer.json comes from there).

Texts: ASCII documents of words from each suite's texts (fixed seed) with exactly 0, L, L + 1, 2 * max_length + 1 and
4 * max_length + 1 tokens (L = max_length minus the template's tokens, with and without add_special_tokens), and the suite's
first four texts.  Cases: add_special_tokens true / false x no
padding, padding right / left to a fixed length x stride 0, L // 2 and L - 1.  Every row records ids, type ids, offsets, attention
mask, special tokens mask and word ids (-1 for None).  Compact JSON, gzip with mtime 0: a rerun writes the same bytes.

    python tests/golden/make_hf_overflow_vectors.py        # needs `tokenizers`; the tests only read the output
"""
import gzip
import json
import os
import random

from tokenizers import Tokenizer

HERE = os.path.dirname(os.path.abspath(__file__))
MAX_LENGTH = {"wordpiece_template_cls_sep": 12, "wordpiece_bert_processing": 11, "wordpiece_template_typed": 13,
              "bpe_whitespace_split_template": 10}


def n_tokens(tok, text):
    return len(tok.encode(text, add_special_tokens=False).ids)


def text_of(tok, words, rng, target):
    """an ASCII text of exactly `target` tokens (without specials), words drawn from `words`"""
    out = []
    for _ in range(2000):
        if n_tokens(tok, " ".join(out)) == target:
            return " ".join(out)
        w = rng.choice(words)
        if n_tokens(tok, " ".join(out + [w])) <= target:
            out.append(w)
    raise RuntimeError(f"no text of {target} tokens")


def row_record(e):
    return {"ids": e.ids, "type_ids": e.type_ids, "offsets": [list(o) for o in e.offsets], "attention_mask": e.attention_mask,
            "special_tokens_mask": e.special_tokens_mask, "word_ids": [-1 if w is None else w for w in e.word_ids]}


def main():
    vec = json.load(open(os.path.join(HERE, "hf_compat_vectors.json")))
    out = {"generator": "tests/golden/make_hf_overflow_vectors.py", "tokenizers_version": __import__("tokenizers").__version__, "suites": []}
    for si, s in enumerate(vec["suites"]):
        rng = random.Random(1000 + si)
        tok = Tokenizer.from_str(s["tokenizer_json"])
        tok.no_truncation()
        tok.no_padding()
        max_length = MAX_LENGTH[s["name"]]
        added = tok.post_processor.num_special_tokens_to_add(False)
        words = sorted({w for t in s["texts"] for w in t.split()})
        texts = ["", text_of(tok, words, rng, max_length - added), text_of(tok, words, rng, max_length - added + 1),
                 text_of(tok, words, rng, max_length), text_of(tok, words, rng, max_length + 1)]
        texts += [text_of(tok, words, rng, k * max_length + 1) for k in (2, 4)]      # many windows' worth
        texts += s["texts"][:4]
        suite = {"name": s["name"], "max_length": max_length, "texts": texts, "cases": []}
        for add in (True, False):
            L = max_length - (added if add else 0)
            for pad in (None, "right", "left"):
                for stride in sorted({0, L // 2, L - 1}):
                    # (through the tokenizer.json: enable_truncation refuses a stride that only fits without add_special_tokens)
                    cfg = json.loads(s["tokenizer_json"])
                    cfg["truncation"] = {"direction": "Right", "max_length": max_length, "strategy": "LongestFirst", "stride": stride}
                    tok = Tokenizer.from_str(json.dumps(cfg))
                    padding = None
                    if pad is not None:
                        padding = {"length": max_length + 3, "pad_id": 0, "pad_type_id": 1 if pad == "left" else 0, "direction": pad}
                        tok.enable_padding(length=padding["length"], pad_id=0, pad_type_id=padding["pad_type_id"], pad_token="[PAD]", direction=pad)
                    docs = []
                    for t in texts:
                        e = tok.encode(t, add_special_tokens=add)
                        assert all(not o.overflowing for o in e.overflowing)
                        docs.append([row_record(e)] + [row_record(o) for o in e.overflowing])
                    suite["cases"].append({"add_special_tokens": add, "stride": stride, "padding": padding, "docs": docs})
        out["suites"].append(suite)
    path = os.path.join(HERE, "hf_overflow_vectors.json.gz")
    with open(path, "wb") as f, gzip.GzipFile(filename="", mode="wb", fileobj=f, mtime=0) as g:
        g.write(json.dumps(out, separators=(",", ":")).encode())
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
