"""The drop-in boundary, EXECUTED: oracle/_ref/libtrinity_ref_gpu.so is the reference itself (same objects as the oracle) with the one
span-building call site of exec_query() (exec.cpp:1083-1086) going through the reference-side binding of libtrinity_b200.so
(integration/gpu_exec.{h,cpp}: GpuAccessProxy / PlanBuilder / GpuDocsSetSpan).  The reference's own query -> compile_query -> exec_node
tree is turned into a plan by PlanBuilder (not by this repo's parser), runs through trn_exec_batch, and is replayed through
MatchesProxy::process -> the stock exec Handlers -> MatchedIndexDocumentsFilter::consider().  The stream consider() sees must equal the
stock library's, for every golden query shape, both ExecFlags modes, both codecs, with and without masked documents."""
import ctypes as C

import numpy as np
import pytest

import trinity_b200 as tb
from refharness import RefIndex, load_ref_gpu
from test_frontend_cpu import EXTRA, OPTIONAL_QUERIES, SOME_QUERIES
from test_gpu_parity import TEMPLATES
from util import assert_close_scores, assert_same_docs, closed_form_lists

pytestmark = pytest.mark.gpu


@pytest.fixture
def ref(real_ref):
    """these tests run the reference's own code, not its recorded outputs"""
    return real_ref


NDOCS = 400_000


def _twin(rl, codec, lists, names):
    r = RefIndex(rl, codec)
    for n, (d, f) in zip(names, lists):
        r.add_term(n, d, f)
    r.finish(NDOCS)
    return r


@pytest.mark.parametrize("codec", [tb.CODEC_GOOGLE, tb.CODEC_LUCENE], ids=["google", "lucene"])
def test_exec_query_through_the_gpu_span_equals_stock_exec_query(ref, codec):
    refg = load_ref_gpu()
    lists = closed_form_lists(NDOCS)
    names = [f"t{i + 1}" for i in range(len(lists))]
    stock = _twin(ref, codec, lists, names)
    gpu = _twin(refg, codec, lists, names)
    assert refg.L.tref_gpu_attach(gpu.h, 0, NDOCS) == 0, refg.err()
    try:
        shapes = [(q, 0, 0) for q in TEMPLATES + EXTRA] + [(q, 8, 0) for q in OPTIONAL_QUERIES] + [(q, 16, m) for q, m in SOME_QUERIES]
        before = refg.L.tref_gpu_spans_executed(gpu.h)
        ran = 0
        for q, pflags, mm in shapes:
            for scored in (False, True):
                if scored and "nosuchterm" in q:
                    continue
                wd, ws = stock.exec(q, scored, NDOCS + 1, parser_flags=pflags, min_match=mm)
                gd, gs = gpu.exec(q, scored, NDOCS + 1, parser_flags=pflags, min_match=mm)
                assert_same_docs(gd, wd, f"[{q}] scored={scored}")
                if scored:
                    assert_close_scores(gs, ws, f"[{q}]")
                ran += 1
        executed = refg.L.tref_gpu_spans_executed(gpu.h) - before
        # single-term DocumentsOnly queries take exec_query's own specialisation (exec.cpp:894-1080) before any span is built, and a query
        # whose tree collapses to nothing never reaches the span site; everything else must have gone through the GPU span
        assert executed >= ran - 8, (executed, ran)
        # masked documents: the Handler's registry test stays where it is (exec.cpp:1108-1116) and filters the replayed stream
        rng = np.random.default_rng(5)
        masked = np.unique(rng.integers(1, NDOCS + 1, 9000)).astype(np.uint32)
        for q in ("t1 AND t2", "t3 OR t7 OR t9", "t1 AND (t2 OR t3) NOT t5"):
            for scored in (False, True):
                wd, ws = stock.exec_masked(q, scored, masked, NDOCS + 1)
                gd, gs = gpu.exec_masked(q, scored, masked, NDOCS + 1)
                assert_same_docs(gd, wd, f"[{q}] masked scored={scored}")
                if scored:
                    assert_close_scores(gs, ws, f"[{q}] masked")
    finally:
        refg.L.tref_gpu_detach(gpu.h)


def _phrase_twins(rl_stock, rl_gpu, codec, ndocs, vocab=9, seed=33, lo=3, hi=40):
    rng = np.random.default_rng(seed)
    prob = 1.0 / np.arange(1, vocab + 1)
    prob /= prob.sum()
    per_term = [dict() for _ in range(vocab)]
    for d in range(1, ndocs + 1):
        toks = rng.choice(vocab, size=int(rng.integers(lo, hi)), p=prob)
        for pos, t in enumerate(toks, start=1):
            per_term[int(t)].setdefault(d, []).append(pos)
    out = []
    for rl in (rl_stock, rl_gpu):
        r = RefIndex(rl, codec)
        for t in range(vocab):
            docs = np.array(sorted(per_term[t]), np.uint32)
            freqs = np.array([len(per_term[t][int(d)]) for d in docs], np.uint32)
            flat = np.array([p for d in docs for p in per_term[t][int(d)]], np.uint32)
            r.add_term(f"w{t + 1}", docs, freqs, flat)
        r.finish(ndocs)
        out.append(r)
    return out


def test_phrases_through_the_gpu_span(ref):
    """ENT::matchphrase / matchanyphrases / matchallphrases -> TRN_NODE_PHRASE: positions checked on the device for a GOOGLE source (inline
    hits) and for a LUCENE source whose hits.data the binding uploaded; a LUCENE source WITHOUT its hits on the device makes the binding
    decline and the reference's own span runs: the same stream in all three cases"""
    from test_phrase_cpu import QUERIES
    refg = load_ref_gpu()
    refg.L.tref_gpu_attach2.restype = C.c_int
    refg.L.tref_gpu_attach2.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_int]
    ndocs = 20_000
    for codec, with_hits in ((tb.CODEC_GOOGLE, 1), (tb.CODEC_LUCENE, 1), (tb.CODEC_LUCENE, 0)):
        stock, gpu = _phrase_twins(ref, refg, codec, ndocs)
        assert refg.L.tref_gpu_attach2(gpu.h, 0, ndocs, with_hits) == 0, refg.err()
        try:
            before = refg.L.tref_gpu_spans_executed(gpu.h)
            nonempty = 0
            for q in QUERIES:
                for scored in (False, True):
                    wd, ws = stock.exec(q, scored, ndocs + 1)
                    gd, gs = gpu.exec(q, scored, ndocs + 1)
                    assert_same_docs(gd, wd, f"[{q}] scored={scored} codec={codec} hits={with_hits}")
                    if scored:
                        assert_close_scores(gs, ws, f"[{q}] codec={codec} hits={with_hits}")
                    nonempty += len(wd) > 0
            executed = refg.L.tref_gpu_spans_executed(gpu.h) - before
            assert nonempty >= 9
            if with_hits:  # '"w1 nosuch"' collapses before the span site; '"w1"' is a term (DocumentsOnly: exec_query's own specialisation)
                assert executed >= 2 * len(QUERIES) - 4, (executed, len(QUERIES))
            else:  # only '"w1"' (a plain term) may have gone to the device
                assert executed <= 2, executed
        finally:
            refg.L.tref_gpu_detach(gpu.h)
