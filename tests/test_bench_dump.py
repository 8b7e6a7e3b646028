"""bench.py --dump-outputs: the files hold what the timed device-resident path computed (held to the oracle), row numbers and
CSR offsets count over the whole step when it is cut into sub-batches, and the dump stays within 64 MB."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


@pytest.mark.gpu
@pytest.mark.parametrize("workload,mib", [("c2b", 4), ("c3", 2)])      # c2b: the whole shard; c3 (padded to 512): a sample
def test_dump_is_the_encoding_of_the_timed_path(tmp_path, workload, mib):
    subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--size-mib", str(mib), "--steps", "2",
                    "--no-configs", "--no-e2e", "--no-cpu-baseline", "--no-verify", "--dump-outputs", str(tmp_path)],
                   check=True, cwd=ROOT, stdout=subprocess.DEVNULL)
    assert sum(os.path.getsize(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)) <= 64_000_000
    d = load(tmp_path)
    assert set(d) == {"slot_rows", "ids", "offsets", "attention_mask", "doc_rows", "doc_tok_off"}
    assert all(a.dtype == np.float64 for a in d.values())
    tok_name, cname, _, trunc, pad, _, max_docs = bench.WORKLOADS[workload]
    text, off = bench.make_corpus(cname, mib << 20, 1234, pinned=False, max_docs=max_docs)
    ref = bench.oracle_for(tok_name, trunc, pad).encode_packed(text, off, algo=0, threads=os.cpu_count() or 1)
    rows, docs = d["slot_rows"].astype(np.int64), d["doc_rows"].astype(np.int64)
    if workload == "c2b":
        assert np.array_equal(rows, np.arange(len(ref.ids))) and np.array_equal(docs, np.arange(len(off)))
    else:
        assert 0 < len(rows) < len(ref.ids) and np.all(np.diff(rows) > 0)
    assert np.array_equal(d["ids"], ref.ids[rows])
    assert np.array_equal(d["offsets"], ref.offsets[rows])
    assert np.array_equal(d["attention_mask"], ref.attention_mask[rows])
    assert np.array_equal(d["doc_tok_off"], ref.doc_tok_off[docs])


@pytest.mark.gpu
def test_sample_of_several_sub_batches_counts_over_the_step(tmp_path):
    import torch
    import tokzig_b200 as tz
    keep, doc0 = [], 0
    parts = [[0, 2, 5, 5], [0, 4, 7]]                                     # doc_tok_off of two sub-batches as the C ABI returns them
    s = bench.OutputSample(len(parts), torch.cuda.current_stream())
    for i, dto in enumerate(parts):
        ids = torch.arange(100 * i, 100 * i + dto[-1], dtype=torch.int32, device="cuda")
        d_off = torch.tensor(dto, dtype=torch.int64, device="cuda")
        keep += [ids, d_off]
        s.add(tz.BatchResult(n_docs=len(dto) - 1, n_tokens=dto[-1], doc_tok_off=d_off.data_ptr(), ids=ids.data_ptr()), i, doc0)
        doc0 += len(dto) - 1
    s.save(tmp_path)
    d = load(tmp_path)
    assert set(d) == {"slot_rows", "ids", "doc_rows", "doc_tok_off"}
    assert np.array_equal(d["slot_rows"], np.arange(12))
    assert np.array_equal(d["ids"], list(range(5)) + list(range(100, 107)))
    assert np.array_equal(d["doc_rows"], np.arange(6))
    assert np.array_equal(d["doc_tok_off"], [0, 2, 5, 5, 9, 12])
