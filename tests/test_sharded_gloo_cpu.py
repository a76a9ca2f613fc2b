"""World-size-2 gloo test (CPU) of the docID-sharded path's host logic: shard ranges, global df for BM25, DocumentsOnly
concatenation and the single all-gather + merge of per-shard top-k.  Each rank evaluates its shard with the reference oracle
(the GPU kernels are covered by the -m gpu tests); the merged result must equal the unsharded reference exec_query."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parent.parent
NDOCS, NTERMS, MIN_DF, K = 150_000, 24, 60, 10
QUERIES = ["t0001 AND t0002", "t0003 OR t0009 OR t0017", "t0002 AND t0005 NOT t0007", "t0001 OR t0002 OR t0004 OR t0008 OR t0016"]


def _numpy_merge(gd, gs):
    world, nq, k = gd.shape
    od, os_ = np.zeros((nq, k), np.int32), np.full((nq, k), -1.0, np.float32)
    for q in range(nq):
        d, s = gd[:, q, :].reshape(-1).numpy(), gs[:, q, :].reshape(-1).numpy()
        keep = s >= 0
        d, s = d[keep], s[keep]
        order = np.lexsort((d, -s))[:k]
        od[q, : len(order)], os_[q, : len(order)] = d[order], s[order]
    import torch
    return torch.from_numpy(od), torch.from_numpy(os_)


def _worker(rank, world, port, out):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import torch
        import trinity_b200 as tb
        from refharness import RefIndex, load_golden_ref
        from trinity_b200.sharded import concat_docs_only, gather_and_merge_topk, global_document_frequencies, shard_range

        lo, hi = shard_range(NDOCS, rank, world)
        s = tb.SynthIndex(tb.CODEC_GOOGLE, NDOCS, NTERMS, min_df=MIN_DF, threads=1, doc_range=(lo, hi))
        gdf = global_document_frequencies(dist, s.terms["documents"])
        want_df = np.array([max(MIN_DF, NDOCS // (2 * r)) for r in range(1, NTERMS + 1)])
        assert np.array_equal(gdf, want_df), "summed shard dfs must equal the unsharded dfs"
        # the shard as an IndexSource of its own; docsCnt = GLOBAL collection size, like IndexSourcesCollectionBM25Scorer::reset
        r = RefIndex.from_bytes(load_golden_ref(), tb.CODEC_GOOGLE, np.asarray(s.index), None, s.names, np.asarray(s.terms), NDOCS, s.sum_hits)
        docs_parts, topd, tops = [], np.zeros((len(QUERIES), K), np.int32), np.full((len(QUERIES), K), -1.0, np.float32)
        for qi, q in enumerate(QUERIES):
            ids, _ = r.exec(q, False, NDOCS + 1)
            docs_parts.append(concat_docs_only(dist, ids))
            if "NOT" in q:
                continue
            # shard-local scores with GLOBAL idf: every match's score = sum over its matching terms of bm25(global idf, freq)
            sid, _ = r.exec(q, True, NDOCS + 1)
            terms = [t for t in q.replace("AND", " ").replace("OR", " ").split()]
            sc = np.zeros(len(sid))
            for t in terms:
                ti = s.names.index(t)
                d, f = r.decode(ti, int(s.terms["documents"][ti]) + 1)
                idf = tb.bm25_idf(int(gdf[ti]), NDOCS)
                pos = np.searchsorted(d, sid)
                hit = (pos < len(d)) & (d[np.minimum(pos, len(d) - 1)] == sid) if len(d) else np.zeros(len(sid), bool)
                sc[hit] += [tb.bm25_score(idf, int(x)) for x in f[pos[hit]]]
            order = np.lexsort((sid, -sc))[:K]
            topd[qi, : len(order)], tops[qi, : len(order)] = sid[order], sc[order]
        md, ms = gather_and_merge_topk(dist, torch.from_numpy(topd), torch.from_numpy(tops), K, _numpy_merge)
        if rank == 0:
            np.savez(out, **{f"docs_{i}": d for i, d in enumerate(docs_parts)}, topd=md.numpy(), tops=ms.numpy())
    finally:
        dist.destroy_process_group()


def test_two_rank_sharded_path_equals_unsharded_reference(ref, tmp_path):
    sys.path.insert(0, str(ROOT / "tests"))
    import trinity_b200 as tb
    from refharness import RefIndex

    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    out = str(tmp_path / "r0.npz")
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    z = np.load(out)
    full = tb.SynthIndex(tb.CODEC_GOOGLE, NDOCS, NTERMS, min_df=MIN_DF, threads=2)
    r = RefIndex.from_bytes(ref, tb.CODEC_GOOGLE, np.asarray(full.index), None, full.names, np.asarray(full.terms), NDOCS, full.sum_hits)
    for qi, q in enumerate(QUERIES):
        want, _ = r.exec(q, False, NDOCS + 1)
        assert np.array_equal(z[f"docs_{qi}"], want), q
        if "NOT" in q:
            continue
        wd, ws = r.exec(q, True, NDOCS + 1)
        order = np.lexsort((wd, -ws))[:K]
        assert np.allclose(z["tops"][qi], ws[order], rtol=1e-5), q
        assert np.array_equal(z["topd"][qi][:3], wd[order][:3]) or np.allclose(ws[order][:3], z["tops"][qi][:3], rtol=1e-6)


def test_shard_ranges_partition_docid_space():
    from trinity_b200.sharded import shard_range
    for n, w in ((100_000_000, 8), (1000, 3), (17, 4)):
        rs = [shard_range(n, r, w) for r in range(w)]
        assert rs[0][0] == 1 and rs[-1][1] == n
        assert all(rs[i][1] + 1 == rs[i + 1][0] for i in range(w - 1))
    with pytest.raises(ValueError):
        shard_range(10, 3, 3)
