"""Segment directories written by the reference's own indexer (SegmentIndexSession::commit, indexer.cpp:241-300) are read by the
product's host reader (trn_segment_open) into exactly what the reference's SegmentIndexSource (segment_index_source.cpp:5-186)
restores: terms dictionary, term_index_ctx per term, field statistics, codec, masked documents."""
import numpy as np
import pytest

import trinity_b200 as tb
from refharness import load_golden_ref


ERASED = np.array([3, 17, 4000, 40000, 70001, 1 << 20], np.uint32)  # a session cannot erase a document it also indexes


def make_lists(seed, nterms=40, ndocs=6000):
    rng = np.random.default_rng(seed)
    lists = {}
    pool = np.setdiff1d(np.arange(1, ndocs + 1), ERASED)
    for t in range(nterms):
        df = int(rng.integers(1, ndocs // (1 + t % 7)))
        docs = np.sort(rng.choice(pool, size=df, replace=False)).astype(np.uint32)
        freqs = rng.integers(1, 6, size=df).astype(np.uint32)
        # mixed-length names exercise the front coding of terms.data
        name = ("t%d" % t) if t % 3 else ("term_prefix_%03d" % t)
        lists[name] = (docs, freqs)
    return lists


@pytest.mark.parametrize("codec", [0, 1])
def test_segment_reader_matches_reference(tmp_path, codec):
    ref = load_golden_ref()
    lists = make_lists(7 + codec, ndocs=1500)   # the segment directories it reads are stored in tests/golden: keep them small
    erased = ERASED
    path = tmp_path / "100"
    path.mkdir()
    ref.segment_write(codec, path, lists, erased, replace_below=100)   # documents 1..99 are updates of an older segment's
    seg = tb.Segment(str(path))
    rseg = ref.segment_open(path)
    assert seg.codec == codec
    assert sorted(seg.names) == sorted(lists)
    assert seg.names == sorted(seg.names), "terms.data is in dictionary order"
    for name, t in zip(seg.names, seg.terms):
        assert (int(t["documents"]), int(t["chunk_off"]), int(t["chunk_len"])) == rseg.resolve(name), name
        assert int(t["documents"]) == len(lists[name][0])
    assert rseg.resolve("no-such-term")[0] == 0
    assert seg.field_statistics == rseg.field_stats()
    assert seg.field_statistics["totalTerms"] == len(lists)
    assert seg.field_statistics["sumTermsDocs"] == sum(len(v[0]) for v in lists.values())
    updated = np.unique(np.concatenate([d[d < 100] for d, _ in lists.values()]))
    assert np.array_equal(seg.masked_documents, np.union1d(erased, updated))
    assert seg.index.size == (path / "index").stat().st_size


def test_segment_without_updates_and_errors(tmp_path):
    ref = load_golden_ref()
    path = tmp_path / "7"
    path.mkdir()
    ref.segment_write(0, path, {"a": ([1, 2, 3], [1, 1, 2]), "ab": ([2], [1])})
    seg = tb.Segment(str(path))
    assert seg.masked_documents.size == 0 and seg.names == ["a", "ab"]
    with pytest.raises(tb.TrinityError):
        tb.Segment(str(tmp_path / "nope"))
    (path / "id").write_bytes(b"\x02\x06GOOGLE" + b"\0" * 24)
    with pytest.raises(tb.TrinityError):
        tb.Segment(str(path))


def test_segment_reader_survives_truncated_and_corrupted_files(tmp_path):
    """the reader parses files it did not write: every truncation / byte flip must end in a TrinityError or a consistent segment,
    never in an out-of-bounds read (the process would die)"""
    ref = load_golden_ref()
    src = tmp_path / "9"
    src.mkdir()
    ref.segment_write(0, src, make_lists(3, nterms=12, ndocs=3000), ERASED, replace_below=50)
    good = {f: (src / f).read_bytes() for f in ("id", "index", "terms.data", "updated_documents.ids")}
    rng = np.random.default_rng(0)
    dst = tmp_path / "10"
    dst.mkdir()
    ok = bad = 0
    for trial in range(300):
        for f, b in good.items():
            (dst / f).write_bytes(b)
        f = ("id", "terms.data", "updated_documents.ids", "index")[trial % 4]
        b = bytearray(good[f])
        if trial % 3 == 0 and len(b):
            b = b[: int(rng.integers(0, len(b)))]
        else:
            for _ in range(int(rng.integers(1, 4))):
                if len(b):
                    b[int(rng.integers(0, len(b)))] = int(rng.integers(0, 256))
        (dst / f).write_bytes(bytes(b))
        try:
            seg = tb.Segment(str(dst))
            # whatever was accepted must be self-consistent
            assert len(seg.names) == len(seg.terms)
            for t in seg.terms:
                assert int(t["chunk_off"]) + int(t["chunk_len"]) <= seg.index.size
            ok += 1
        except tb.TrinityError:
            bad += 1
    assert ok + bad == 300 and bad > 50
