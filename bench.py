#!/usr/bin/env python3
"""bench.py -- BASELINE.json's metric (input GB/s + tokens/s of batch encode) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2b|c2a|c3|c4a|c4b|c5a|c5b] [--size-mib M] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      the reference's algorithm (C restatement, oracle/) on the host cores

A step = one pass of the encode hot path over one synthetic batch.  The headline workload is configs[1] of BASELINE.json
(c2b: GPT-2-shaped byte-level BPE, 1 GiB of synthetic UTF-8 per GPU); the other BASELINE configs (c2a, c3 at 10 M sentences,
c5b, and c4b when N > 1) are measured in the same run with fewer steps and reported under "configs", each checked against
the oracle on a sample.  One process per GPU, documents sharded by rank with NO collective on the data path; NCCL only
carries the barrier and the max-over-ranks of the timings.

  value      device-resident: inputs in HBM, CUDA events on the stream the kernels run on, ids + offsets + attention (16 B/token)
  e2e        the host-buffer C-ABI call tkz_encode_batch_compact: pinned text H2D, kept ids (u16 when the vocabulary allows) +
             packed offsets D2H, inside the timed region; the full Encoding is rebuilt from it by tkz_compact_expand
  roofline   frac = ALL kernels of a step: (input bytes + 4 B per id slot) / device time of the step / measured HBM peak
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (tokenizer, corpus, description, truncation, padding, docs per sub-batch (0 = whole shard), max docs (0 = by size))
    "c2b": ("gpt2_whitespace", "c2", "GPT-2-shaped byte-level BPE 50,257/50k merges, pre_tokenizer Whitespace (words split on whitespace)", None, None, 0, 0),
    "c2a": ("gpt2_bytelevel", "c2", "GPT-2-shaped byte-level BPE 50,257/50k merges, pre_tokenizer ByteLevel (reference: null => whole document = one pre-token)", None, None, 0, 0),
    "c3": ("bert_wordpiece", "c3", "BERT-shaped WordPiece 30,522, ASCII-lowercase + ws/punct split, truncate/pad 512, 10 M sentences", 512, {"length": 512, "pad_id": 0}, 2097152, 10_000_000),
    "c4b": ("llama3_whitespace", "c4", "Llama-3-shaped byte-level BPE 128,256, pre_tokenizer Whitespace, multilingual", None, None, 0, 0),
    "c4a": ("llama3_sequence", "c4", "Llama-3-shaped byte-level BPE 128,256, pre_tokenizer Sequence (reference: null => whole document)", None, None, 0, 0),
    "c5b": ("gpt2_whitespace", "c5", "GPT-2-shaped BPE, skewed documents 1 B..4 MiB with long unbroken words, Whitespace", None, None, 0, 0),
    "c5a": ("gpt2_bytelevel", "c5", "GPT-2-shaped BPE, skewed documents 1 B..4 MiB, whole-document pre-tokens", None, None, 0, 0),
}
DEFAULT_MIB = {"c2b": 1024, "c2a": 1024, "c3": 1600, "c4b": 2048, "c4a": 2048, "c5b": 1024, "c5a": 256}
VERIFY_MIB = 64           # per workload: the GPU encoding of this much text is compared with the oracle, every array
DUMP_BYTES = 60 << 20     # --dump-outputs: all sampled arrays of one step together, float64 (under 64 MB with the .npy headers)
DUMP_DOC_ROWS = 1 << 18   # CSR entries (doc_tok_off) of the sample; the token slots share what the CSR and wide rows leave
DUMP_WIDE_ROWS = 1 << 16  # wide-offset records (only with packed offsets)
DUMP_SEED = 1234
# per-token-slot arrays of tkz_batch_result: (field, values per slot, element type as the C ABI writes it)
SLOT_ARRAYS = (("ids", 1, "u4"), ("ids16", 1, "u2"), ("offsets", 2, "u4"), ("offsets_packed", 1, "u2"), ("attention_mask", 1, "u4"),
               ("type_ids", 1, "u4"), ("special_tokens_mask", 1, "u4"), ("span_tokens", 4, "u4"))


def env_int(k, d):
    try:
        return int(os.environ.get(k, d))
    except ValueError:
        return d


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = threading.Event()

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            p = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                 stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            return
        while not self.stop_flag.is_set():
            line = p.stdout.readline()
            if not line:
                break
            self.rows.append([x.strip() for x in line.split(",")])
        p.terminate()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def make_corpus(cname, nbytes, seed, pinned=True, max_docs=0):
    from tools import corpus
    out = None
    if pinned:
        import torch
        out = torch.empty(nbytes + 4096, dtype=torch.uint8, pin_memory=True).numpy()
    text, off = corpus.generate(cname, nbytes, seed, max_docs=max_docs or None, out=out)
    return text, off


def sub_batches(off, docs_per_batch):
    nd = len(off) - 1
    if docs_per_batch <= 0 or docs_per_batch >= nd:
        return [(0, nd)]
    return [(a, min(nd, a + docs_per_batch)) for a in range(0, nd, docs_per_batch)]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def config_of(workload, size_mib):
    """the workload description both arms print (no measured values in it)"""
    tok_name, cname, desc, trunc, pad, _, max_docs = WORKLOADS[workload]
    return {"workload": f"{workload}: {desc}", "tokenizer": tok_name, "corpus": cname, "corpus_target_mib": size_mib,
            "corpus_max_docs": max_docs or None, "seed": "1234 + rank", "truncation": trunc, "padding": pad,
            "l2": "inputs (>= 1 GiB per step) larger than the 126 MB L2; no flush needed", "parallelism": "documents sharded by rank, no collective"}


def oracle_for(tok_name, trunc, pad):
    from oracle import oracle as orc
    from tools import tokenizers_io
    o = orc.OracleTokenizer.from_json(tokenizers_io.tokenizer_json(tok_name))
    o.truncation = trunc
    o.padding = pad
    return o


def cpu_sample(o, text, off, algo, budget_s, cores):
    """documents [0, k) of the shard such that one pass of the oracle on all host cores takes about budget_s"""
    nd = len(off) - 1
    probe = max(1, min(nd, int(np.searchsorted(off, min(int(off[-1]), 256 << 10)))))
    probe = max(probe, min(nd, cores * 4))
    t0 = time.perf_counter()
    o.count_tokens(text, off[: probe + 1], algo=algo, threads=cores)
    dt = max(time.perf_counter() - t0, 1e-4)
    rate = float(off[probe]) / dt
    want = int(min(float(off[-1]), rate * budget_s))
    return max(probe, min(nd, int(np.searchsorted(off, want))))


def cpu_baseline(workload, text, off, budget_s=10.0):
    """The reference algorithm (C restatement, oracle/) on the host cores, bounded sample of the same workload."""
    tok_name, cname, desc, trunc, pad, _, _ = WORKLOADS[workload]
    o = oracle_for(tok_name, trunc, pad)
    cores = os.cpu_count() or 1
    algo = 0 if workload in ("c2b", "c3", "c4b") else 1
    ndocs = cpu_sample(o, text, off, algo, budget_s, cores)
    t0 = time.perf_counter()
    ntok = o.count_tokens(text, off[: ndocs + 1], algo=algo, threads=cores)
    dt = time.perf_counter() - t0
    nbytes = int(off[ndocs])
    return {"value": nbytes / dt / 1e9, "unit": "GB/s", "cores": cores, "kind": "port",
            "sample": f"first {ndocs} documents ({nbytes / 2**20:.1f} MiB) of the seed-1234 shard, one pass on all {cores} host threads, {dt:.1f} s, "
                      f"{'BPE.tokenize / WordPiece.tokenize literal restatement' if algo == 0 else 'fast-exact restatement (same rounds, O(n log n)): the literal O(n^2) loop does not finish on whole-document words'}",
            "tokens_per_s": ntok / dt, "note": "C restatement of tokenizer-zig's Tokenizer.encode (oracle/), not the Zig binary: no zig toolchain in the image"}


def run_reference(args, rank, world):
    """--impl reference: the same workload and config keys; each step = the bounded sample of cpu_baseline, all host threads."""
    if rank != 0:
        return
    tok_name, cname, desc, trunc, pad, _, max_docs = WORKLOADS[args.workload]
    text, off = make_corpus(cname, args.size_mib << 20, 1234, pinned=False, max_docs=max_docs)
    o = oracle_for(tok_name, trunc, pad)
    cores = os.cpu_count() or 1
    algo = 0 if args.workload in ("c2b", "c3", "c4b") else 1
    ndocs = cpu_sample(o, text, off, algo, args.ref_step_s, cores)
    sub = off[: ndocs + 1]
    nbytes = int(sub[-1])
    for _ in range(args.warmup):
        o.count_tokens(text, sub, algo=algo, threads=cores)
    t0 = time.perf_counter()
    ntok = 0
    for _ in range(args.steps):
        ntok = o.count_tokens(text, sub, algo=algo, threads=cores)
    dt = (time.perf_counter() - t0) / args.steps
    v = nbytes / dt / 1e9
    line = {"impl": "reference", "metric": "encode_input_throughput", "value": v, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": f"synthetic ({cname} generator, seed 1234)", "tokens_per_s": ntok / dt,
            "config": config_of(args.workload, args.size_mib),
            "cpu_baseline": {"value": v, "unit": "GB/s", "cores": cores, "kind": "port",
                             "sample": f"each step = first {ndocs} documents ({nbytes / 2**20:.1f} MiB) of the seed-1234 shard, all {cores} host threads, "
                                       f"{'BPE.tokenize / WordPiece.tokenize literal restatement' if algo == 0 else 'fast-exact restatement'}"},
            "e2e": {"value": v, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


class DeviceArray:
    """A (rows, cols) array the C ABI returned in device memory, seen by torch.as_tensor without a copy (CUDA array interface).
    It is typed as the signed integer of the same width: torch gathers no unsigned type wider than a byte."""

    def __init__(self, ptr, rows, cols, utype):
        self.__cuda_array_interface__ = {"shape": (rows, cols), "typestr": "<" + utype.replace("u", "i"), "data": (ptr, False), "version": 3}


class OutputSample:
    """--dump-outputs: a fixed, seeded sample of what the timed path hands its caller in its last step, i.e. the device result of
    every sub-batch, read right after its call because the next call on the context reuses the buffers.  Written as
    DIR/<name>.npy in float64: one file per array of tkz_batch_result, and slot_rows / doc_rows / wide_rows holding the row
    numbers of the sample counted over the whole step (doc_tok_off is made step-wide the same way).  A shard no larger than
    the budget is written whole."""

    def __init__(self, n_batches, stream):
        self.n_batches, self.stream = n_batches, stream
        self.parts = {}
        self.slot0 = self.wide0 = 0
        self.ms = 0.0                  # device-timeline time spent here; the caller takes it out of the timed window

    @staticmethod
    def pick(rng, n, k):
        return np.arange(n, dtype=np.int64) if n <= k else np.unique(rng.integers(0, n, size=k))

    @staticmethod
    def gather(ptr, n, cols, utype, rows):
        import torch
        if len(rows) == 0:
            return np.zeros((0, cols) if cols > 1 else 0)
        t = torch.as_tensor(DeviceArray(ptr, n, cols, utype))
        v = t.index_select(0, torch.from_numpy(rows).to(t.device)).cpu().numpy().view("<" + utype).astype(np.float64)
        return v if cols > 1 else v.ravel()

    def add(self, r, i, doc0):
        """sub-batch i of the step, whose first document is doc0 of the shard"""
        import torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        rng = np.random.default_rng([DUMP_SEED, i])
        nt, nd = int(r.n_tokens), int(r.n_docs)
        slot = [(f, c, u) for f, c, u in SLOT_ARRAYS if getattr(r, f)]
        k = (DUMP_BYTES - 16 * DUMP_DOC_ROWS - 40 * DUMP_WIDE_ROWS) // (8 * (1 + sum(c for _, c, _ in slot))) // self.n_batches
        rows = self.pick(rng, nt, k)
        out = {"slot_rows": rows + self.slot0}
        for f, c, u in slot:
            out[f] = self.gather(getattr(r, f), nt, c, u, rows)
        # a sub-batch's closing CSR entry is the next one's first: only the last sub-batch contributes it
        rows = self.pick(rng, nd + (i == self.n_batches - 1), DUMP_DOC_ROWS // self.n_batches)
        out["doc_rows"] = rows + doc0
        out["doc_tok_off"] = self.gather(r.doc_tok_off, nd + 1, 1, "u8", rows) + self.slot0
        if r.wide_tokens and r.n_wide:
            rows = self.pick(rng, int(r.n_wide), DUMP_WIDE_ROWS // self.n_batches)
            out["wide_rows"] = rows + self.wide0
            out["wide_tokens"] = self.gather(r.wide_tokens, int(r.n_wide), 4, "u4", rows)
            self.wide0 += int(r.n_wide)
        self.slot0 += nt
        for name, a in out.items():
            self.parts.setdefault(name, []).append(np.asarray(a, dtype=np.float64))
        e1.record(self.stream)
        e1.synchronize()
        self.ms += e0.elapsed_time(e1)

    def save(self, out_dir):
        os.makedirs(out_dir, exist_ok=True)
        for name, parts in self.parts.items():
            np.save(os.path.join(out_dir, name + ".npy"), np.concatenate(parts))


class Work:
    """one workload on one rank: corpus in pinned host memory and in HBM, tokenizer, parameters"""

    def __init__(self, workload, size_mib, rank, local_rank, stream):
        import torch
        import tokzig_b200 as tz
        from tools import tokenizers_io
        self.tz, self.torch = tz, torch
        self.name = workload
        self.tok_name, self.cname, self.desc, self.trunc, self.pad, self.docs_per_batch, self.max_docs = WORKLOADS[workload]
        t0 = time.time()
        self.text, self.off = make_corpus(self.cname, size_mib << 20, 1234 + rank, max_docs=self.max_docs)
        self.t_gen = time.time() - t0
        self.nd = len(self.off) - 1
        self.nbytes = int(self.off[-1])
        self.dev = torch.device("cuda", local_rank)
        self.tok = tz.Tokenizer.from_json(tokenizers_io.tokenizer_json(self.tok_name), device=local_rank, stream=stream.cuda_stream)
        self.tok.truncation = None if self.trunc is None else {"max_length": self.trunc}
        self.tok.padding = self.pad
        self.L = tz.lib()
        self.ctx = self.tok.context_handle()
        self.d_text = torch.from_numpy(self.text).to(self.dev)
        d_off = torch.from_numpy(self.off.astype(np.int64)).to(self.dev)
        self.batches = sub_batches(self.off, self.docs_per_batch)
        self.d_offs = [(d_off[a: b + 1] - d_off[a]).contiguous() for a, b in self.batches]
        self.h_offs = [(self.off[a: b + 1] - self.off[a]).astype(np.uint64) for a, b in self.batches]
        self.stats = tz.Stats()

    def close(self):
        self.tok.close()
        del self.d_text, self.d_offs

    def device_step(self, params, collect=None, sink=None):
        tot_tokens = tot_real = 0
        for i, ((a, b), doff) in enumerate(zip(self.batches, self.d_offs)):
            r = self.tz.BatchResult()
            base = int(self.off[a]); nb = int(self.off[b]) - base
            rc = self.L.tkz_encode_batch_device(self.ctx, C.c_void_p(self.d_text.data_ptr() + base), C.c_void_p(doff.data_ptr()), b - a, nb, C.byref(params), C.byref(r))
            if rc != 0:
                raise RuntimeError(f"tkz_encode_batch_device rc={rc}: {self.L.tkz_last_error(self.ctx)}")
            tot_tokens += r.n_tokens; tot_real += r.n_real_tokens
            if collect is not None:
                self.L.tkz_ctx_get_stats(self.ctx, C.byref(self.stats))
                s = self.stats
                collect["launches"] += s.kernel_launches; collect["words"] += s.n_words
                collect["uniq"] = int(s.n_unique_words); collect["long"] = int(s.n_long_words); collect["path"] = int(s.path)
                for j, k in enumerate(("ms_split", "ms_model", "ms_scan", "ms_emit", "ms_total")):
                    collect["ms"][j] += getattr(s, k)
            if sink is not None:
                sink.add(r, i, a)
        return tot_tokens, tot_real

    def time_device(self, outputs, steps, warmup, stream, barrier, params=None, sink=None):
        """K steps with everything resident in HBM; returns local ms per step and the counters of the steps.  `sink` (an
        OutputSample) reads the results of the last step; the time it takes is not counted."""
        torch = self.torch
        if params is None:
            params = self.tok.params(outputs)
        for _ in range(warmup):
            self.device_step(params)
        agg = {"launches": 0, "words": 0, "ms": [0.0] * 5}
        barrier(); torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for s in range(steps):
            agg["words"] = 0
            tokens, real = self.device_step(params, collect=agg, sink=sink if s == steps - 1 else None)
        ev1.record(stream)
        torch.cuda.synchronize(); barrier()
        agg["tokens"], agg["real"] = tokens, real
        agg["ms_step"] = (ev0.elapsed_time(ev1) - (sink.ms if sink else 0.0)) / steps
        agg["stage_ms"] = [x / steps for x in agg["ms"]]
        agg["launches_per_step"] = agg["launches"] / steps
        return agg

    def host_step(self, mode):
        """one pass through the host-buffer C ABI; returns (h2d bytes, d2h bytes).  mode: compact | compact_ids | full16"""
        tz, L = self.tz, self.L
        h2d = d2h = 0
        # the compact result has no padding slots, so the whole shard is ONE call (the device-resident steps of a padded workload
        # are cut into sub-batches only because their padded slot count would pass 2^32)
        whole = mode != "full16" and len(self.batches) > 1 and self.nbytes < (1 << 32) - (1 << 20)
        if whole and not hasattr(self, "h_off_all"):
            self.h_off_all = self.off.astype(np.uint64)
        for (a, b), ob in ([((0, self.nd), self.h_off_all)] if whole else zip(self.batches, self.h_offs)):
            base = int(self.off[a])
            h2d += int(ob[-1]) + ob.nbytes
            if mode == "full16":
                r = tz.BatchResult()
                p = self.tok.params(tz.OUT_IDS | tz.OUT_OFFSETS | tz.OUT_ATTENTION)
                rc = L.tkz_encode_batch(self.ctx, C.c_void_p(self.text.ctypes.data + base), C.c_void_p(ob.ctypes.data), b - a, C.byref(p), C.byref(r))
                d2h += int(r.n_tokens) * 16 + (b - a + 1) * 8
            else:
                r = tz.CompactResult()
                p = self.tok.params()
                rc = L.tkz_encode_batch_compact(self.ctx, C.c_void_p(self.text.ctypes.data + base), C.c_void_p(ob.ctypes.data), b - a, C.byref(p),
                                                1 if mode == "compact" else 0, C.byref(r))
                per = (2 if r.ids16 else 4) + (2 if r.offsets_packed else (8 if r.offsets else 0))
                d2h += int(r.n_kept) * per + (b - a + 1) * 8 + int(r.n_wide) * 16
            if rc != 0:
                raise RuntimeError(f"host encode rc={rc}: {L.tkz_last_error(self.ctx)}")
            self.last = r
        return h2d, d2h

    def time_host(self, mode, steps, barrier):
        torch = self.torch
        self.host_step(mode)                       # warm-up: sizes the pinned result buffers
        barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            h2d, d2h = self.host_step(mode)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        return dt, h2d, d2h

    def verify(self, mib):
        """GPU == oracle on the first `mib` MiB of the shard: the six arrays through the full-array call AND through the compact
        result + tkz_compact_expand"""
        tz = self.tz
        o = oracle_for(self.tok_name, self.trunc, self.pad)
        k = max(1, min(self.nd, int(np.searchsorted(self.off, mib << 20))))
        text, off = self.text[: int(self.off[k])], self.off[: k + 1]
        algo = 0 if self.name in ("c2b", "c3", "c4b") else 1
        ref = o.encode_packed(text, off, algo=algo, threads=os.cpu_count() or 1)
        got = self.tok.encode_packed(text, off)
        exp = tz.expand_compact(self.tok.encode_compact(text, off))
        ok = True
        for g in (got, exp):
            ok = ok and all(np.array_equal(getattr(g, f), getattr(ref, f)) for f in ("doc_tok_off", "ids", "offsets", "attention_mask", "type_ids", "special_tokens_mask"))
        return bool(ok), int(off[-1]), k


def traffic_table():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}


def roofline_of(W, agg, ms_step_max, outputs, peak, peak_src, size_mib):
    """SURVEY.md 8(d): B_alg = input bytes + 4 B per id slot over the CUDA-event span of ALL kernels of the step"""
    b_alg = W.nbytes + 4 * agg["tokens"]
    per_tok = (4 if outputs & 1 and not outputs & 64 else 0) + (2 if outputs & 64 else 0) + (8 if outputs & 2 else 0) + (4 if outputs & 4 else 0) + (2 if outputs & 32 else 0)
    b_full = W.nbytes + per_tok * agg["tokens"]
    ach = b_alg / (ms_step_max * 1e-3) / 1e9
    st = agg["stage_ms"]
    tj = traffic_table().get(f"{W.name}:{size_mib}:{outputs}", {})
    if agg.get("path") == 2:
        kernels = [{"name": "slice_words_kernel (pass A: stage + classify + split + word-table probe + inline model -> token stream)", "ms": round(st[0], 4),
                    "algorithmic_bytes": W.nbytes, "note": "reads the text once; its output is the token stream, not counted"},
                   {"name": "word-list kernels (pre-tokens > 255 B: bpe_block / bpe_grid / wordpiece_warp)", "ms": round(st[1], 4), "algorithmic_bytes": 0},
                   {"name": "scans", "ms": round(st[2], 4), "algorithmic_bytes": 0},
                   {"name": "slice_emit_kernel (pass B: token stream -> ids [+ offsets, attention], truncate / pad)", "ms": round(st[3], 4),
                    "algorithmic_bytes": 4 * agg["tokens"], "note": "writes the id slots"}]
    else:
        kernels = [{"name": "split (K0 + K1)", "ms": round(st[0], 4), "algorithmic_bytes": W.nbytes},
                   {"name": "model (K3 bpe_warp / bpe_block / bpe_grid | K4 wordpiece)", "ms": round(st[1], 4), "algorithmic_bytes": 0},
                   {"name": "scans", "ms": round(st[2], 4), "algorithmic_bytes": 0},
                   {"name": "emit (K5)", "ms": round(st[3], 4), "algorithmic_bytes": 4 * agg["tokens"]}]
    for k in kernels:
        k["achieved"] = k["algorithmic_bytes"] / (k["ms"] * 1e-3) / 1e9 if k["ms"] > 0 else 0.0
        k["frac"] = k["achieved"] / peak
        k["traffic"] = tj.get(k["name"].split(" ")[0])
    dom = max(kernels, key=lambda k: k["ms"])
    return {"bound": "hbm", "kernel": "whole step (all kernels between the first and the last CUDA event); dominant: " + dom["name"].split(" (")[0],
            "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": tj.get("step"), "peak_source": peak_src,
            "algorithmic_bytes_per_step": b_alg, "delivered_bytes_per_step": b_full, "kernels": kernels,
            "stage_ms_per_step": dict(zip(["split", "model", "scan", "emit", "total_kernels"], [round(x, 4) for x in st]))}


def strong_scaling(n_gpus, total_mib, workload="c5b"):
    """tkzm_encode_batch_compact over n_gpus GPUs on one seed-fixed corpus, two cuts; wall time per shard (host buffers in,
    compact result out: an e2e figure), slowest over mean = the load imbalance the cut leaves"""
    import tokzig_b200 as tz
    from tools import tokenizers_io
    tok_name, cname, desc, trunc, pad, _, _ = WORKLOADS[workload]
    t0 = time.time()
    text, off = make_corpus(cname, total_mib << 20, 99, pinned=True)
    t_gen = time.time() - t0
    cfg = tz.Tokenizer.from_json(tokenizers_io.tokenizer_json(tok_name), device=None)
    pool = tz.MultiPool(cfg, list(range(n_gpus)))
    out = {"workload": f"{workload}: {desc}", "corpus_bytes": int(off[-1]), "docs": len(off) - 1, "n_gpus": n_gpus, "corpus_generated_s": round(t_gen, 1),
           "api": "tkzm_encode_batch_compact (rank 0 drives every GPU: one context + one host thread per GPU; pinned text in, compact results out)", "cuts": {}}
    o = oracle_for(tok_name, trunc, pad)
    rc_ = pool.raw_class()
    for label, cb in (("bytes", False), ("cost_model", True)):
        # the cut, timed on its own (bytes: a few binary searches; cost model: one sparse pass over the text on all host threads)
        t0 = time.perf_counter()
        cut = tz.shard_bounds_c(off, n_gpus, tz.document_costs_c(text, off, rc_) if cb else None)
        cut_ms = (time.perf_counter() - t0) * 1e3
        pool.encode_compact(text, off, bounds=cut)                     # warm-up: arenas, pinned buffers
        best = None
        for _ in range(2):
            t0 = time.perf_counter()
            bounds, results, ms = pool.encode_compact(text, off, bounds=cut)
            wall = time.perf_counter() - t0
            if best is None or wall < best[0]:
                best = (wall, bounds.copy(), ms.copy(), sum(int(r.n_kept) for r in results), pool.shard_kernel_ms())
        wall, bounds, ms, kept, kms = best
        shard_bytes = [int(off[int(bounds[k + 1])] - off[int(bounds[k])]) for k in range(n_gpus)]
        # parity of the sharded path: the first and the last documents of every shard against the oracle
        ok = True
        for k in range(n_gpus):
            d0, d1 = int(bounds[k]), int(bounds[k + 1])
            for lo, hi in ((d0, min(d1, d0 + 40)), (max(d0, d1 - 40), d1)):
                if hi <= lo:
                    continue
                ref = o.encode_packed(text[int(off[lo]):int(off[hi])], off[lo:hi + 1] - off[lo], algo=1, threads=os.cpu_count() or 1)
                got = tz.expand_compact(results[k], lo - d0, hi - d0)
                ok = ok and np.array_equal(got.ids, ref.ids) and np.array_equal(got.offsets, ref.offsets) and np.array_equal(got.doc_tok_off, ref.doc_tok_off)
        out["cuts"][label] = {"value": int(off[-1]) / wall / 1e9, "unit": "GB/s", "wall_ms": wall * 1e3, "shard_ms": [round(float(x), 2) for x in ms],
                              "imbalance_slowest_over_mean": float(ms.max() / ms.mean()),
                              "shard_kernel_ms": [round(float(x), 2) for x in kms], "kernel_imbalance_slowest_over_mean": float(kms.max() / max(kms.mean(), 1e-9)), "shard_bytes": shard_bytes, "kept_tokens": kept,
                              "cut_ms": cut_ms, "parity_checked_vs_oracle": bool(ok)}
    pool.close(); cfg.close()
    return out


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import tokzig_b200 as tz

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.current_stream()
    peak, peak_src = peaks()

    def barrier():
        if world > 1:
            dist.barrier()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(xs):
        t = torch.tensor([float(x) for x in xs], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(x) for x in t.tolist()]

    def measure(workload, size_mib, steps, warmup, outputs, headline):
        """device-resident + e2e numbers of one workload; every rank runs it on its own shard"""
        W = Work(workload, size_mib, rank, local_rank, stream)
        parity = None
        if rank == 0 and not args.no_verify:
            ok, vbytes, vdocs = W.verify(VERIFY_MIB)
            parity = {"ok": ok, "bytes": vbytes, "docs": vdocs, "arrays": "doc_tok_off, ids, offsets, attention_mask, type_ids, special_tokens_mask; full-array call and compact result + tkz_compact_expand"}
            if not ok:
                raise SystemExit(f"PARITY FAILURE ({workload}): GPU encoding differs from the oracle on the verification sample")
        sampler = None
        if headline:
            sampler = ClockSampler(local_rank)
            sampler.start()
        sink = OutputSample(len(W.batches), stream) if headline and args.dump_outputs and rank == 0 else None
        agg = W.time_device(outputs, steps, warmup, stream, barrier, sink=sink)
        if sampler:
            sampler.stop_flag.set()
        if sink:
            sink.save(args.dump_outputs)
        ms_step = allmax(agg["ms_step"])
        all_bytes, all_real, all_slots = allsum([W.nbytes, agg["real"], agg["tokens"]])
        out = {"value": all_bytes / (ms_step * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms_step, "steps": steps,
               "tokens_per_s": all_real / (ms_step * 1e-3), "slots_per_s": all_slots / (ms_step * 1e-3), "outputs_mask": outputs,
               "bytes_per_gpu": W.nbytes, "docs_per_gpu": W.nd, "words_per_gpu": agg["words"], "tokens_per_gpu": agg["real"],
               "unique_words_last_batch": agg.get("uniq"), "long_words_last_batch": agg.get("long"), "sub_batches": len(W.batches),
               "pipeline": {0: "per-occurrence pipeline", 2: "slice pipeline (2 passes)"}.get(agg.get("path"), "?"),
               "roofline": roofline_of(W, agg, ms_step, outputs, peak, peak_src, size_mib), "gpu_launches_per_step": agg["launches_per_step"],
               "parity_checked_vs_oracle": parity, "corpus_generated_s": round(W.t_gen, 1)}
        extra = {}
        if headline:
            # the same step delivering less: ids only (what B_alg counts) and the compact device form (ids16 + packed offsets)
            for label, o2 in (("ids_only", tz.OUT_IDS), ("ids16_packed_offsets", tz.OUT_IDS | tz.OUT_IDS_U16 | tz.OUT_OFFSETS_PACKED)):
                a2 = W.time_device(o2, max(3, steps // 2), 2, stream, barrier)
                ms2 = allmax(a2["ms_step"])
                b_alg = W.nbytes + 4 * a2["tokens"]
                extra[label] = {"outputs_mask": o2, "ms_per_step": ms2, "value": all_bytes / (ms2 * 1e-3) / 1e9, "unit": "GB/s",
                                "roofline_frac": b_alg / (ms2 * 1e-3) / 1e9 / peak, "stage_ms_per_step": dict(zip(["split", "model", "scan", "emit", "total_kernels"], [round(x, 4) for x in a2["stage_ms"]]))}
            out["device_variants"] = extra
        if workload == "c3":
            # the same batch in hf_compat mode (beyond the reference, opt-in: [CLS] $A [SEP] from the JSON's TemplateProcessing and
            # document-relative offsets) through the same slice pipeline.  Parity: tests/test_gpu_hf_compat.py
            ph = W.tok.params(outputs)
            ph.hf_flags = tz.HF_TEMPLATE | tz.HF_DOC_OFFSETS
            ph.tpl_n_prefix, ph.tpl_n_suffix = 1, 1
            ph.tpl_prefix_id[0], ph.tpl_suffix_id[0] = W.tok.token_to_id(b"[CLS]"), W.tok.token_to_id(b"[SEP]")
            a3 = W.time_device(outputs, max(2, steps // 2), 1, stream, barrier, params=ph)
            ms3 = allmax(a3["ms_step"])
            out["hf_compat"] = {"ms_per_step": ms3, "value": all_bytes / (ms3 * 1e-3) / 1e9, "unit": "GB/s", "flags": "TKZ_HF_TEMPLATE | TKZ_HF_DOC_OFFSETS",
                                "pipeline": {0: "per-occurrence pipeline", 2: "slice pipeline (2 passes)"}.get(a3.get("path"), "?"),
                                "stage_ms_per_step": dict(zip(["split", "model", "scan", "emit", "total_kernels"], [round(x, 4) for x in a3["stage_ms"]]))}
        e2e = None
        if not args.no_e2e:
            e_steps = max(1, min(steps, args.e2e_steps))
            dt, h2d, d2h = W.time_host("compact", e_steps, barrier)
            dt = allmax(dt)
            r = W.last
            e2e = {"value": all_bytes / dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": dt * 1e3, "steps": e_steps,
                   "tokens_per_s": all_real / dt,
                   "api": "tkz_encode_batch_compact (host pointers; pinned text H2D + kept ids and packed offsets D2H inside the timed region; "
                          "attention / type / special masks and padding slots are constants of (kept count, parameters) and are rebuilt by tkz_compact_expand)",
                   "wire_format": {"ids": "u16" if r.ids16 else "u32", "offsets": "u16 (start | end << 8)" if r.offsets_packed else ("2 x u32" if r.offsets else None),
                                   "wide_offset_records": int(r.n_wide)}}
            if headline:
                dt2, _, d2h2 = W.time_host("full16", max(1, e_steps - 1), barrier)
                e2e["full_arrays"] = {"value": W.nbytes / dt2 / 1e9, "unit": "GB/s", "ms_per_step": dt2 * 1e3, "d2h_bytes_per_step": d2h2,
                                      "api": "tkz_encode_batch with ids + offsets + attention as u32 arrays (16 B/token over PCIe: round 1's e2e)", "note": "rank-local"}
                dt3, _, d2h3 = W.time_host("compact_ids", max(1, e_steps - 1), barrier)
                e2e["ids_only"] = {"value": W.nbytes / dt3 / 1e9, "unit": "GB/s", "ms_per_step": dt3 * 1e3, "d2h_bytes_per_step": d2h3, "note": "rank-local"}
                if rank == 0 and not args.no_materialise:
                    e2e["binding_shape"] = binding_shape_e2e(W)
        out["e2e"] = e2e
        clocks = sampler.summary() if sampler else None
        return W, out, clocks

    def binding_shape_e2e(W):
        """what the Zig binding does for its caller (INTEGRATION.md): PAGEABLE text in, compact result, then every document's six
        arrays materialised on the host (tkz_compact_expand, one call per range of documents, on all host threads)"""
        from concurrent.futures import ThreadPoolExecutor
        L = W.L
        text = np.array(W.text, copy=True)             # pageable copy
        ob = W.h_offs[0] if len(W.batches) == 1 else None
        if ob is None:
            return None
        nthreads = min(32, os.cpu_count() or 1)
        r = tz.CompactResult()
        p = W.tok.params()

        def once():
            rc = L.tkz_encode_batch_compact(W.ctx, C.c_void_p(text.ctypes.data), C.c_void_p(ob.ctypes.data), W.nd, C.byref(p), 1, C.byref(r))
            if rc != 0:
                raise RuntimeError("compact encode failed")
            n = int(L.tkz_compact_slots(C.byref(r), 0, W.nd))
            ids, attn, typ, sp = (np.empty(n, np.uint32) for _ in range(4))
            offs = np.empty(2 * n, np.uint32)
            dto = np.empty(W.nd + 1, np.uint64)
            kept = np.ctypeslib.as_array(C.cast(r.doc_kept_off, C.POINTER(C.c_uint64)), shape=(W.nd + 1,))
            cuts = np.searchsorted(kept, np.linspace(0, float(kept[-1]), nthreads + 1)[1:-1]).tolist()
            bounds = [0] + cuts + [W.nd]

            def part(i):
                d0, d1 = int(bounds[i]), int(bounds[i + 1])
                if d1 <= d0:
                    return
                s0 = int(L.tkz_compact_slots(C.byref(r), 0, d0))
                L.tkz_compact_expand(C.byref(r), d0, d1, C.c_void_p(dto.ctypes.data + 8 * d0), C.c_void_p(ids.ctypes.data + 4 * s0), C.c_void_p(offs.ctypes.data + 8 * s0),
                                     C.c_void_p(attn.ctypes.data + 4 * s0), C.c_void_p(typ.ctypes.data + 4 * s0), C.c_void_p(sp.ctypes.data + 4 * s0))
            with ThreadPoolExecutor(nthreads) as ex:
                list(ex.map(part, range(nthreads)))
            return n
        once()
        t0 = time.perf_counter()
        n = once()
        dt = time.perf_counter() - t0
        return {"value": W.nbytes / dt / 1e9, "unit": "GB/s", "ms_per_step": dt * 1e3, "host_threads": nthreads, "slots_materialised": n,
                "api": "pageable text -> tkz_encode_batch_compact -> tkz_compact_expand of every document into six freshly allocated u32 arrays", "note": "rank 0 only"}

    # ---- headline
    W, head, clocks = measure(args.workload, args.size_mib, args.steps, args.warmup, args.outputs, True)
    cb = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = cpu_baseline(args.workload, W.text, W.off)
    desc = W.desc
    cname = W.cname
    nbytes, nd = W.nbytes, W.nd
    W.close(); del W
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, same run, fewer steps
    configs = {}
    if not args.no_configs and args.workload == "c2b":
        names = ["c2a", "c3", "c5b"] + (["c4b"] if world > 1 else [])
        for name in names:
            W2, o2, _ = measure(name, DEFAULT_MIB[name], args.config_steps, 3, args.outputs, False)
            keep = ("value", "unit", "ms_per_step", "steps", "tokens_per_s", "slots_per_s", "bytes_per_gpu", "docs_per_gpu", "tokens_per_gpu", "long_words_last_batch",
                    "sub_batches", "pipeline", "parity_checked_vs_oracle", "corpus_generated_s")
            c = {k: o2[k] for k in keep}
            c["workload"] = f"{name}: {W2.desc}"
            c["roofline"] = {"frac": o2["roofline"]["frac"], "achieved": o2["roofline"]["achieved"], "algorithmic_bytes_per_step": o2["roofline"]["algorithmic_bytes_per_step"],
                             "stage_ms_per_step": o2["roofline"]["stage_ms_per_step"]}
            c["e2e"] = None if o2["e2e"] is None else {k: o2["e2e"][k] for k in ("value", "unit", "ms_per_step", "h2d_bytes_per_step", "d2h_bytes_per_step", "wire_format")}
            if "hf_compat" in o2:
                c["hf_compat"] = o2["hf_compat"]
            configs[name] = c
            W2.close(); del W2
            torch.cuda.empty_cache()

    # ---- strong scaling + skew through the product's multi-GPU entry point (tkzm_*): ONE fixed corpus (BASELINE config 5: 4 GiB,
    # documents 1 B .. 4 MiB with long unbroken words) cut over the N GPUs by bytes and by the cost model; rank 0 drives all GPUs
    # (one context + one host thread each) while the other ranks wait on a CPU barrier with their GPUs idle
    strong = None
    if world > 1 and not args.no_strong and args.workload == "c2b":
        gloo = dist.new_group(backend="gloo")
        torch.cuda.synchronize()
        dist.barrier(group=gloo)
        if rank == 0:
            strong = strong_scaling(world, args.strong_mib)
        dist.barrier(group=gloo)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    line = {"metric": "encode_input_throughput", "value": head["value"], "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": f"synthetic ({cname} generator, seed 1234+rank, generated in {head['corpus_generated_s']} s)",
            "tokens_per_s": head["tokens_per_s"], "slots_per_s": head["slots_per_s"],
            "config": config_of(args.workload, args.size_mib),
            "workload_stats": {k: head[k] for k in ("bytes_per_gpu", "docs_per_gpu", "words_per_gpu", "tokens_per_gpu", "unique_words_last_batch", "long_words_last_batch",
                                                    "sub_batches", "outputs_mask", "pipeline")},
            "roofline": head["roofline"], "device_variants": head.get("device_variants"), "hf_compat": head.get("hf_compat"), "cpu_baseline": cb, "e2e": head["e2e"],
            "gpu_launches": int(round(head["gpu_launches_per_step"] * args.steps)), "clocks": clocks,
            "parity_checked_vs_oracle": None if head["parity_checked_vs_oracle"] is None else head["parity_checked_vs_oracle"]["ok"],
            "parity": head["parity_checked_vs_oracle"], "configs": configs, "strong_scaling": strong}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2b", choices=sorted(WORKLOADS))
    ap.add_argument("--size-mib", type=int, default=0)
    ap.add_argument("--outputs", type=int, default=7, help="TKZ_OUT_* mask of the device-resident headline: ids|offsets|attention = 7 (16 B/token)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--config-steps", type=int, default=3, help="timed steps of each workload under \"configs\"")
    ap.add_argument("--ref-step-s", type=float, default=10.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline workload only")
    ap.add_argument("--no-materialise", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling / skew measurement (N > 1 only)")
    ap.add_argument("--strong-mib", type=int, default=4096, help="size of the fixed corpus of the strong-scaling measurement")
    ap.add_argument("--multi", type=int, default=0, help="single process: only the strong-scaling measurement over this many GPUs (tkzm_*)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the headline's timed steps, write a seeded sample (at most 64 MB, float64) "
                    "of what its last step computed to DIR/<name>.npy (rank 0's shard)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.multi > 0):
        ap.error("--dump-outputs samples the device-resident headline; --impl reference and --multi have none")
    if args.size_mib <= 0:
        args.size_mib = DEFAULT_MIB[args.workload]
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if args.impl == "reference":
        # the reference arm loads nothing of the product: only the oracle and the corpus generator are built
        if rank == 0:
            subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
            subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tools")])
        run_reference(args, rank, world)
        return
    import __graft_entry__ as g
    if rank == 0:
        g.build()
    elif world > 1:
        time.sleep(0.5)
    if args.multi > 0:
        print(json.dumps({"strong_scaling": strong_scaling(args.multi, args.strong_mib, "c5b" if args.workload == "c2b" else args.workload)}), flush=True)
        return
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
