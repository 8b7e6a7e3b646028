#!/usr/bin/env python3
"""Cost of overflowing windows (TKZ_HF_OVERFLOW) on the device-resident path: the c3 WordPiece tokenizer with its [CLS] / [SEP]
template on long documents (the c2 corpus: median ~700 B), truncated and padded to max_length 128 (stride 32) and 512 (stride
128), timed with and without the flag, alternating A B in one process.  Without the flag each document keeps its first window;
with it every window is a row.  Reports rows, slots, the emit stage (ms_emit, which includes the window stage) and step times
from the library's stage events and CUDA events, the card's name and power limit read in the same run, and a parity check of
the rows against tests/overflow_ref.py on the first --parity-mib of the corpus.  Prints one JSON line.

    python tools/bench_overflow.py [--mib 1024] [--steps 5] [--warmup 2] [--rounds 2] [--parity-mib 64]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

OUTPUTS_NAMES = "ids + offsets + attention + type ids"


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:                      # (the timing itself does not depend on it)
        return f"unknown ({e})"


def params(tz, tpl, max_length, stride, overflow, outputs):
    pre, suf, seq = tpl
    p = tz.EncodeParams(has_truncation=1, max_length=max_length, has_padding=1, pad_length=max_length, outputs=outputs,
                        hf_flags=tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS | (tz.HF_OVERFLOW if overflow else 0), tpl_n_prefix=len(pre),
                        tpl_n_suffix=len(suf), tpl_seq_type=seq, stride=stride)
    for i, (a, b) in enumerate(pre):
        p.tpl_prefix_id[i], p.tpl_prefix_type[i] = a, b
    for i, (a, b) in enumerate(suf):
        p.tpl_suffix_id[i], p.tpl_suffix_type[i] = a, b
    return p


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mib", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2, help="A B pairs per setting")
    ap.add_argument("--parity-mib", type=int, default=64)
    args = ap.parse_args()

    import torch
    import tokzig_b200 as tz
    from bench import make_corpus
    from oracle import oracle as orc
    from overflow_ref import overflow_rows
    from tools import tokenizers_io

    js = tokenizers_io.tokenizer_json("bert_wordpiece")
    tpl = orc.hf_template_from_json(js)
    text, off = make_corpus("c2", args.mib << 20, 1234, pinned=False)
    lens = np.diff(off.astype(np.int64))
    stream = torch.cuda.Stream(device=0)
    tok = tz.Tokenizer.from_json(js, device=0, stream=stream.cuda_stream)
    L, h = tz.lib(), tok.context_handle()
    d_text = torch.from_numpy(text).cuda()
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    nd, nb = len(off) - 1, int(off[-1])
    outputs = tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION | tz.OUT_TYPE_IDS
    out = {"card": card(), "tokenizer": "bert_wordpiece (c3) + [CLS] $A [SEP]", "corpus": "c2", "bytes": nb, "docs": nd,
           "doc_bytes_median": int(np.median(lens)), "outputs": OUTPUTS_NAMES, "steps": args.steps, "rounds": args.rounds, "settings": {}}
    r, st = tz.BatchResult(), tz.Stats()

    def step(p):
        rc = L.tkz_encode_batch_device(h, C.c_void_p(d_text.data_ptr()), C.c_void_p(d_off.data_ptr()), nd, nb, C.byref(p), C.byref(r))
        if rc != tz.OK:
            raise RuntimeError(f"rc {rc}: {L.tkz_last_error(h)}")

    def timed(p):
        for _ in range(args.warmup):
            step(p)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        emit = total = 0.0
        torch.cuda.synchronize()
        ev0.record(stream)
        for _ in range(args.steps):
            step(p)
            L.tkz_ctx_get_stats(h, C.byref(st))
            emit += st.ms_emit; total += st.ms_total
        ev1.record(stream)
        ev1.synchronize()
        return {"ms_per_step": round(ev0.elapsed_time(ev1) / args.steps, 3), "ms_emit": round(emit / args.steps, 3),
                "ms_kernels": round(total / args.steps, 3), "rows": int(r.n_rows) if r.n_rows else nd, "slots": int(r.n_tokens),
                "real_tokens": int(r.n_real_tokens), "launches": int(st.kernel_launches)}

    with torch.cuda.stream(stream):
        for max_length, stride in ((128, 32), (512, 128)):
            runs = {"without": [], "with": []}
            for _ in range(args.rounds):
                for label, ovf in (("without", False), ("with", True)):
                    runs[label].append(timed(params(tz, tpl, max_length, stride, ovf, outputs)))
            out["settings"][f"max_length {max_length} stride {stride}"] = runs
    torch.cuda.synchronize()

    # parity: the host-buffer call on the first parity-mib of the corpus against the restatement
    k = int(np.searchsorted(off, args.parity_mib << 20, side="right")) - 1
    docs = [bytes(text[off[i]:off[i + 1]]) for i in range(k)]
    o = orc.OracleTokenizer.from_json(js)
    parity = {}
    for max_length, stride in ((128, 32), (512, 128)):
        tok.set_hf_compat(tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS | tz.HF_OVERFLOW)
        tok.truncation = {"max_length": max_length, "stride": stride}
        tok.padding = {"length": max_length, "pad_id": 0, "pad_type_id": 0, "direction": "right"}
        got = tok.encode_batch(docs, outputs=tz.OUT_ALL)
        want = overflow_rows(o, docs, max_length, stride, tpl[0], tpl[1], tpl[2], tok.padding, word_ids=False, threads=os.cpu_count() or 1)
        ok = all(np.array_equal(getattr(got, f), want[f]) for f in ("doc_row_off", "row_tok_off", "doc_tok_off", "ids", "offsets", "attention_mask",
                                                                     "type_ids", "special_tokens_mask"))
        parity[f"max_length {max_length} stride {stride}"] = {"docs": k, "bytes": int(off[k]), "rows": int(len(want["row_tok_off"]) - 1), "equal": ok}
    out["parity"] = parity
    tok.close()
    print(json.dumps(out), flush=True)
    if not all(v["equal"] for v in parity.values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
