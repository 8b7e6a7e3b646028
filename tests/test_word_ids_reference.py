"""Word ids (TKZ_OUT_WORD_IDS, Hugging Face Encoding.word_ids for a single sequence): the restatement the GPU tests compare with
(tests/word_ids_ref.py: every token's pre-token ordinal in its document, 0xFFFFFFFF for template special tokens and padding)
against what `tokenizers` 0.22.2 returned for every encoding of tests/golden/hf_compat_vectors.json, and on random normalizer /
pre-tokenizer chains against the oracle's encodings, including pre-tokens that yield no token."""
import json
import random

import numpy as np
import pytest

from gen_util import rand_bpe_json, rand_text, rand_wp_json
from kat_util import NORM_OPS, PT_OPS
from oracle import oracle as orc
from test_hf_compat_oracle import CASES, VEC, oracle_for
from word_ids_ref import NONE, hf_word_ids, restated

HF = hf_word_ids(VEC)


def template_sizes(suite, add):
    pre, suf, _ = orc.hf_template_from_json(suite["tokenizer_json"])
    return (len(pre), len(suf)) if add else (0, 0)


@pytest.mark.parametrize("suite,case", CASES, ids=[f"{s['name']}-{c['name']}" for s, c in CASES])
def test_restated_word_ids_equal_tokenizers(suite, case):
    t = oracle_for(suite, case)
    docs = [x.encode() for x in suite["texts"]]
    w, ids = restated(t, docs, *template_sizes(suite, case["add_special_tokens"]))
    r = t.encode_batch(docs)
    assert ids.tolist() == r.ids[r.special_tokens_mask == 0].tolist()
    assert w.tolist() == HF[(suite["name"], case["name"])].tolist()


@pytest.mark.parametrize("seed", range(16))
def test_restatement_on_random_chains(seed):
    rng = random.Random(4100 + seed)
    if seed % 2:
        js, alpha = rand_wp_json(rng, pretok=None, normalizer=None)
    else:
        # BPE without unk: a pre-token of unknown characters only yields no token and still uses up its index
        js, alpha = rand_bpe_json(rng, n_merges=30, unk=None)
    t = orc.OracleTokenizer.from_json(js)
    t.normalizers = [(NORM_OPS[rng.choice(list(NORM_OPS))], rng.randint(0, 3)) for _ in range(rng.randint(0, 2))]
    t.pretokenizers = [PT_OPS[rng.choice(list(PT_OPS))] for _ in range(rng.randint(1, 3))]
    t.truncation = [None, 3, 17][seed % 3]
    t.padding = [None, {"length": 24, "pad_id": 0, "direction": "right"}, {"length": 20, "pad_id": 0, "direction": "left"}][(seed // 3) % 3]
    docs = [rand_text(rng, alpha, rng.randint(0, 50), p_unknown=0.2, p_upper=0.2) for _ in range(120)] + [b"", b" ", b"zz", b"ab zz ab a"]
    w, ids = restated(t, docs)
    r = t.encode_batch(docs)
    assert ids.tolist() == r.ids[r.special_tokens_mask == 0].tolist()
    assert np.array_equal(w == NONE, r.special_tokens_mask == 1)


def test_zero_token_pre_token_keeps_its_index():
    """BPE without unk on "ab zz ab a": word ids [0, 2, 3] ("zz" yields no token and still uses up index 1)"""
    js = json.dumps({"model": {"type": "BPE", "vocab": {"a": 0, "b": 1, "ab": 2}, "merges": ["a b"]}, "pre_tokenizer": {"type": "WhitespaceSplit"}})
    t = orc.OracleTokenizer.from_json(js)
    assert restated(t, [b"ab zz ab a"])[0].tolist() == [0, 2, 3]
    t.pretokenizers = None                                          # no pre-tokenizer: the document is word 0
    assert restated(t, [b"ab zz ab a"])[0].tolist() == [0, 0, 0]
