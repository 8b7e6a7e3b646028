#!/usr/bin/env python3
"""Cost of word ids (TKZ_OUT_WORD_IDS) on the device-resident path: the same workload timed with and without the bit,
alternating A B A B in one process, with the library's stage events (pass A = ms_split, pass B = ms_emit in the slice
pipeline).  Workloads as bench.py builds them: c2b (1 GiB, ids + offsets + attention) and c3 (BERT WordPiece, truncate / pad
512).  Prints one JSON line; the card's name and power limit are read in the same run.

    python tools/bench_word_ids.py [--steps 5] [--warmup 2] [--rounds 2] [--c2b-mib 1024] [--c3-mib 1600]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:                      # (the timing itself does not depend on it)
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2, help="A B pairs per workload")
    ap.add_argument("--c2b-mib", type=int, default=1024)
    ap.add_argument("--c3-mib", type=int, default=1600)
    args = ap.parse_args()

    import torch
    import tokzig_b200 as tz
    from bench import Work

    stream = torch.cuda.Stream(device=0)
    out = {"card": card(), "steps": args.steps, "rounds": args.rounds, "workloads": {}}
    base = tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION
    for name, mib in (("c2b", args.c2b_mib), ("c3", args.c3_mib)):
        with torch.cuda.stream(stream):
            W = Work(name, mib, 0, 0, stream)
            runs = {"without": [], "with": []}
            for _ in range(args.rounds):
                for label, outputs in (("without", base), ("with", base | tz.OUT_WORD_IDS)):
                    a = W.time_device(outputs, args.steps, args.warmup, stream, lambda: None)
                    st = dict(zip(["pass_a_split", "model", "scan", "pass_b_emit", "total_kernels"], [round(x, 4) for x in a["stage_ms"]]))
                    runs[label].append({"ms_per_step": round(a["ms_step"], 3), "stage_ms_per_step": st, "slots": int(a["tokens"])})
            out["workloads"][name] = {"bytes": W.nbytes, "docs": W.nd, "sub_batches": len(W.batches), "outputs_mask": base, **runs}
            W.close()
        torch.cuda.synchronize()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
