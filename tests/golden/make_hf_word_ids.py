#!/usr/bin/env python3
"""Generates tests/golden/hf_compat_word_ids.i32.gz: Encoding.word_ids as Hugging Face `tokenizers` (0.22.2) returns them for
every encoding of tests/golden/hf_compat_vectors.json (same tokenizer.json, texts, truncation, padding and add_special_tokens;
the ids are checked against the stored ones, so both files describe the same encodings).  Little-endian int32, suites -> cases
-> encodings -> tokens in file order, -1 for None (special tokens and padding); gzip with mtime 0, so a rerun is byte-identical.

    python tests/golden/make_hf_word_ids.py        # needs `tokenizers`; the tests only read the output
"""
import gzip
import json
import os

import numpy as np
from tokenizers import Tokenizer

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    vec = json.load(open(os.path.join(HERE, "hf_compat_vectors.json")))
    out, n = [], 0
    for s in vec["suites"]:
        tok = Tokenizer.from_str(s["tokenizer_json"])
        for c in s["cases"]:
            tok.no_truncation()
            tok.no_padding()
            if c["truncation"] is not None:
                tok.enable_truncation(max_length=c["truncation"])
            if c["padding"] is not None:
                p = c["padding"]
                tok.enable_padding(length=p["length"], pad_id=p["pad_id"], pad_type_id=p["pad_type_id"], pad_token=p["pad_token"], direction=p["direction"])
            for text, e in zip(s["texts"], c["encodings"]):
                enc = tok.encode(text, add_special_tokens=c["add_special_tokens"])
                assert enc.ids == e["ids"], (s["name"], c["name"], text)
                out += [-1 if w is None else w for w in enc.word_ids]
                n += 1
    path = os.path.join(HERE, "hf_compat_word_ids.i32.gz")
    with open(path, "wb") as f, gzip.GzipFile(filename="", mode="wb", fileobj=f, mtime=0) as g:
        g.write(np.array(out, "<i4").tobytes())
    print(path, os.path.getsize(path), "bytes;", n, "encodings,", len(out), "word ids")


if __name__ == "__main__":
    main()
