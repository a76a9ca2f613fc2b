"""bench.py contract on CPU: the reference arm (--impl reference) needs no GPU — it runs the reference's own exec_query (oracle/_ref) on
the host cores and must print one JSON line with the keys the driver reads; the product arm must fail loudly without a CUDA device."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.parametrize("workload", ["and2", "or10"])
def test_reference_arm_prints_the_contract_line(real_ref, workload):
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", workload, "--ndocs", "200000", "--nterms", "64",
                        "--nq", "16", "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "queries/s" and line["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline", "gpu_launches"):
        assert key in line, key
    assert line["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["cores"] >= 1 and "workload" in line["config"]


def test_product_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--ndocs", "200000", "--nterms", "64", "--nq", "8", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode != 0  # no CPU fallback
    assert not [l for l in p.stdout.splitlines() if l.startswith('{"metric"')]


def test_full_size_parity_checker_is_exact_in_uint64(ref):
    """the checker bench.py hangs on its cpu_baseline leg: fed the reference's own results it must report equality, and one flipped docID
    must flip the checksum verdict even when the running sum is beyond 2^53 (a float64 detour would lose it)"""
    import types

    import numpy as np

    sys.path.insert(0, str(ROOT))
    import bench
    import trinity_b200 as tb

    nq = 6
    counts = np.array([3, 0, 2, 4, 1, 2], np.uint64)
    ids = np.array([4_000_000_000 - i for i in range(int(counts.sum()))][::-1], np.uint32)  # large docIDs
    big = np.repeat(ids, 1)  # one copy is enough: prepend a huge constant through a fake first query below
    off = np.concatenate([np.zeros(1, np.int64), np.cumsum(counts).astype(np.int64)])
    sums = np.array([int(big[off[q]:off[q + 1]].astype(np.uint64).sum()) for q in range(nq)], np.uint64)
    def result(match_counts, offsets, docids):  # what bench.py holds: a BatchResult (its checksums() is the code under test)
        return tb.BatchResult(len(match_counts), tb.MODE_DOCS_ONLY, 0, offsets, docids, None, match_counts, 0, 0, 0, 0.0)

    res = result(counts.copy(), off, big.copy())
    out = bench.full_size_parity(res, tb.MODE_DOCS_ONLY, 100, counts, sums, None, None, nq)
    assert out == {"queries_checked": nq, "match_counts_equal": True, "docid_checksums_equal": True}
    res.docids[5] ^= 1
    assert bench.full_size_parity(res, tb.MODE_DOCS_ONLY, 100, counts, sums, None, None, nq)["docid_checksums_equal"] is False
    # sums past 2^53: 3e6 documents near 4e9 each
    n = 3_000_000
    d = np.full(n, 3_999_999_999, np.uint32)
    d[-1] = 3_999_999_998
    res = result(np.array([n - 1, 1], np.uint64), np.array([0, n - 1, n], np.int64), d)
    sums = np.array([int(d[: n - 1].astype(np.uint64).sum()), 3_999_999_998], np.uint64)
    assert bench.full_size_parity(res, tb.MODE_DOCS_ONLY, 100, res.match_counts, sums, None, None, 2)["docid_checksums_equal"] is True
    sums[1] += 1
    assert bench.full_size_parity(res, tb.MODE_DOCS_ONLY, 100, res.match_counts, sums, None, None, 2)["docid_checksums_equal"] is False


def test_reference_side_binding_fails_loudly_without_a_gpu(real_ref):
    """oracle/_ref/libtrinity_ref_gpu.so = the reference + integration/gpu_exec.cpp: attaching the device twin of an index source needs
    a CUDA device; without one it reports the engine's error (no silent CPU detour), and the library's exec_query() keeps using the
    reference's own span for sources that have no twin"""
    import numpy as np
    import torch

    sys.path.insert(0, str(ROOT / "tests"))
    from refharness import RefIndex, load_ref_gpu

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    refg = load_ref_gpu()
    r = RefIndex(refg, 0)
    r.add_term("a", np.arange(2, 2000, 2, dtype=np.uint32), np.ones(999, np.uint32))
    r.add_term("b", np.arange(3, 2000, 3, dtype=np.uint32), np.ones(666, np.uint32))
    r.finish(2000)
    assert refg.L.tref_gpu_attach(r.h, 0, 2000) != 0
    assert "CUDA" in refg.err()
    ids, _ = r.exec("a AND b", False, 4000)  # no twin registered: the stock CPU span
    assert np.array_equal(ids, np.arange(6, 2000, 6, dtype=np.uint32))
