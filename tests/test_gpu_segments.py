"""Segment ingestion (SURVEY.md 8f row 2): directories written by the reference's own indexer, read by trn_segment_open, executed
on the GPU, compared with the reference's SegmentIndexSource / IndexSourcesCollection exec on the same directories."""
import numpy as np
import pytest

import trinity_b200 as tb
from trinity_b200.segments import SegmentCollection
from util import assert_close_scores, assert_same_docs, assert_topk_equal

pytestmark = pytest.mark.gpu


@pytest.fixture
def ref(real_ref):
    """these tests run the reference's own code, not its recorded outputs"""
    return real_ref


NDOCS = 200_000
QUERIES = ["w1 AND w2", "w3 OR w7 OR w9", "w1 AND (w2 OR w3) NOT w5", "w10", "(w1 AND w2) OR (w3 AND w4)", "w2 AND onlyold", "w1 OR onlynew",
           "missing AND w1", "missing OR w4"]


def lists(seed, lo, hi, extra):
    rng = np.random.default_rng(seed)
    out = {}
    for t in range(1, 13):
        df = max(1, (hi - lo) // (t + 1))
        docs = np.sort(rng.choice(np.arange(lo, hi), size=df, replace=False)).astype(np.uint32)
        out[f"w{t}"] = (docs, rng.integers(1, 9, size=df).astype(np.uint32))
    docs = np.sort(rng.choice(np.arange(lo, hi), size=5000, replace=False)).astype(np.uint32)
    out[extra] = (docs, np.ones(5000, np.uint32))
    return out


@pytest.mark.parametrize("codec", [tb.CODEC_GOOGLE, tb.CODEC_LUCENE], ids=["google", "lucene"])
def test_single_segment(ref, tmp_path, codec):
    path = tmp_path / "3"
    path.mkdir()
    ref.segment_write(codec, path, lists(1, 1, NDOCS, "onlyold"))
    col = SegmentCollection([path])
    rseg = ref.segment_open(path)
    for mode, scored in ((tb.MODE_DOCS_ONLY, False), (tb.MODE_SCORED_ALL, True)):
        (res,) = col.exec_batch(QUERIES, mode)
        for i, q in enumerate(QUERIES):
            wd, ws = rseg.exec(q, scored, NDOCS + 1)
            gd, gs = res.query(i)
            assert_same_docs(gd, wd, f"[{q}]")
            if scored:
                assert_close_scores(gs, ws, f"[{q}]")


@pytest.mark.parametrize("codec", [tb.CODEC_GOOGLE, tb.CODEC_LUCENE], ids=["google", "lucene"])
def test_collection_of_two_segments_with_updates(ref, tmp_path, codec):
    """generation 2 re-indexes a docID range of generation 1 and erases some of its documents: generation 1 is scanned with
    generation 2's updated_documents masked; BM25 uses the collection's statistics"""
    old, new = tmp_path / "1", tmp_path / "2"
    old.mkdir(), new.mkdir()
    ref.segment_write(codec, old, lists(1, 1, NDOCS, "onlyold"))
    erased = np.arange(5, 90_000, 7, dtype=np.uint32)           # deleted documents of generation 1
    ref.segment_write(codec, new, lists(2, 150_000, 260_000, "onlynew"), erased, replace_below=NDOCS)   # 150000..199999: updated documents
    col = SegmentCollection([old, new])
    assert col.generations == [2, 1]
    rcol = ref.collection_open([old, new])
    cap = 600_000
    for mode, scored in ((tb.MODE_DOCS_ONLY, False), (tb.MODE_SCORED_ALL, True)):
        res = col.exec_batch(QUERIES, mode)
        for i, q in enumerate(QUERIES):
            want = rcol.collection_exec(q, scored, cap)
            for s, (wd, ws) in enumerate(want):
                gd, gs = res[s].query(i)
                assert_same_docs(gd, wd, f"[{q}] source {s}")
                if scored:
                    assert_close_scores(gs, ws, f"[{q}] source {s}")
    # the older generation really was masked
    (plain,) = SegmentCollection([old]).exec_batch(["w1"], tb.MODE_DOCS_ONLY)
    assert len(res[1].query(QUERIES.index("w10"))[0]) < len(ref.segment_open(old).exec("w10", False, cap)[0])
    assert len(plain.query(0)[0]) == col.segments[1].terms["documents"][col.segments[1].names.index("w1")]
    tres = col.exec_batch(QUERIES, tb.MODE_SCORED_TOPK, k=25)
    for i, q in enumerate(QUERIES):
        want = rcol.collection_exec(q, True, cap)
        for s, (wd, ws) in enumerate(want):
            td, ts = tres[s].query(i)
            assert_topk_equal(td, ts, wd, ws, 25, f"[{q}] source {s} top-25")
