"""GPU tests of how a caller reads results back (run with -m gpu on the B200 box): KMerIndex / EdgeIndex lookups of stored and
absent keys, ranged downloads of multi-chunk k-mer sets, and every read-input path of the C ABI. The checker is the C oracle,
whose lookups tests/test_oracle_vs_reference.py pins to the unmodified reference."""
import numpy as np
import pytest

import golden_util as G
import oracle as O
from query_sets import query_set
from spades_b200.kmer_index import (Context, DeBruijnKMerKMerSplitter, DeBruijnReadKMerSplitter, KMerDiskCounter, KMerIndexBuilder,
                                    ParallelSortingSplitter, SpadesGpuError, _p)
from spades_b200.packing import pack_fixed, pack_reads, synthetic_reads

pytestmark = pytest.mark.gpu

NOT_FOUND = np.uint64((1 << 64) - 1)


def _bucket(key, B):
    w = np.ascontiguousarray(key, np.uint64)
    return int(O.lib().orc_bucket(O._p(w), len(w), B))


def _assert_same_lookups(got, want, q, bsz, what):
    """got == want row by row; otherwise name the first mismatching keys with their bucket and its size"""
    bad = np.nonzero(np.asarray(got) != np.asarray(want))[0]
    if len(bad) == 0:
        return
    B = len(bsz)
    lines = []
    for i in bad[:8]:
        b = _bucket(q[i], B)
        lines.append("key %s bucket %d (size %d): gpu %d, oracle %d" % (" ".join("%016x" % x for x in q[i]), b, bsz[b], int(got[i]),
                                                                       np.int64(want[i].astype(np.int64))))
    empty = sum(1 for i in bad if bsz[_bucket(q[i], B)] == 0)
    pytest.fail("%s: %d of %d lookups differ (%d of them in empty buckets)\n  " % (what, len(bad), len(q), empty) + "\n  ".join(lines))


def _check_index_lookups(c, st, ks, K, seed, what, n_derived=None):
    """KMerIndex.seq_idx of the query set of tests/query_sets.py against the oracle's index of the same keys"""
    assert np.array_equal(st.kmers().ravel(), ks.keys.ravel()) and np.array_equal(st.bucket_sizes(), ks.bsz), what
    idx = KMerIndexBuilder(c).BuildIndex(st)
    m = O.Mphf(ks)
    assert G.index_equal(m.serialize(), idx.serialize(), len(ks.bsz)), what
    q = query_set(ks.keys, K, ks.nw, seed, n_derived)
    want = m.lookup_many(q)
    _assert_same_lookups(idx.seq_idx(q), want, q, ks.bsz, what)
    if ks.n:
        assert np.array_equal(np.sort(want[:ks.n]), np.arange(ks.n, dtype=np.uint64))
    idx.free()
    return want


def _reads(seed, n=60, genome_len=500):
    return synthetic_reads(n, 150, genome_len, 0.01, seed=seed)


# (set kind, K, B, seed): canonical = sgpu_count(SGPU_CANONICAL), all = sgpu_count(SGPU_ALL_WINDOWS), from_kp = sgpu_kmers_from_kpomers
# of a canonical (K+1)-mer set. K from 3 to 128 (one to four words, odd and even), B from 1 to far more buckets than keys.
LOOKUP_CASES = [
    ("canonical", 3, 1, 1), ("canonical", 3, 64, 2), ("all", 4, 300, 3), ("canonical", 21, 1, 4), ("canonical", 21, 4000, 5),
    ("all", 22, 5000, 6), ("from_kp", 21, 3000, 7), ("canonical", 32, 3000, 8), ("all", 33, 2500, 9), ("from_kp", 55, 3000, 10),
    ("canonical", 64, 7, 11), ("all", 64, 6000, 12), ("canonical", 65, 4000, 13), ("from_kp", 77, 16, 14), ("all", 96, 2000, 15),
    ("from_kp", 97, 3000, 16), ("canonical", 100, 2500, 17), ("from_kp", 127, 2000, 18), ("canonical", 128, 1500, 19), ("all", 128, 9, 20),
]


@pytest.mark.parametrize("kind,K,B,seed", LOOKUP_CASES)
def test_kmer_index_lookups_match_oracle(kind, K, B, seed):
    from gpu_util import ctx
    c = ctx()
    words, offs, lens = pack_reads(_reads(seed))
    c.set_reads(words, offs, lens)
    if kind == "from_kp":
        kp = KMerDiskCounter(c, DeBruijnReadKMerSplitter(K + 1)).Count(B)
        st = KMerDiskCounter(c, DeBruijnKMerKMerSplitter(K, kp)).Count(B)
        ks = O.kmers_from_kpomers(O.count(words, offs, lens, K + 1, B, 0), B)
    else:
        splitter = DeBruijnReadKMerSplitter(K) if kind == "canonical" else ParallelSortingSplitter(K)
        st = KMerDiskCounter(c, splitter).Count(B)
        ks = O.count(words, offs, lens, K, B, 0 if kind == "canonical" else 1)
    _check_index_lookups(c, st, ks, K, 100 + seed, "%s K=%d B=%d" % (kind, K, B))


def test_lookups_in_a_set_without_kmers():
    from gpu_util import ctx
    c = ctx()
    words, offs, lens = pack_reads(["ACGT", "AC", "GGGTTT", "A" * 20])
    c.set_reads(words, offs, lens)
    for K, B in ((21, 1), (33, 40)):
        st = KMerDiskCounter(c, DeBruijnReadKMerSplitter(K)).Count(B)
        ks = O.count(words, offs, lens, K, B, 0)
        assert ks.n == 0 and st.total_kmers() == 0
        want = _check_index_lookups(c, st, ks, K, 7, "empty set K=%d B=%d" % (K, B))
        assert (want == NOT_FOUND).all()


# ---- a set counted in several bucket-group passes (one result chunk per pass) ----------------------------------------------------
@pytest.fixture(scope="module")
def multichunk():
    """60 k reads x 150 bp, K = 56, B = 80, counted in a context whose HBM budget holds only a part of the records"""
    codes = synthetic_reads(60_000, 150, 60_000, 0.01, seed=94, as_codes=True)
    words, offs, lens = pack_fixed(codes)
    K, B = 56, 80
    c = Context(0, hbm_budget_bytes=128 << 20)
    c.set_reads(words, offs, lens)
    st = KMerDiskCounter(c, DeBruijnReadKMerSplitter(K)).Count(B)
    passes = int(c.times()["passes"])
    ks = O.count(words, offs, lens, K, B, 0)
    yield c, st, ks, passes
    st.free()
    c.close()


def test_multichunk_ranged_downloads(multichunk):
    """records and multiplicities of every range that starts 0, 1 or 7 records before a bucket boundary (the passes, and with them
    the result chunks, split the set at bucket boundaries) and ends 0, 1 or 7 records after it"""
    c, st, ks, passes = multichunk
    assert passes >= 3, passes
    n = st.total_kmers()
    assert n == ks.n
    bounds = np.unique(np.cumsum(ks.bsz)[:-1])
    bounds = bounds[(bounds > 0) & (bounds < n)]
    assert len(bounds) >= passes - 1
    ranges = [(0, n), (0, 0), (n, 0), (n - 1, 1), (0, 1)]
    for x in bounds:
        for a in (0, 1, 7):
            for b in (0, 1, 7):
                lo, hi = max(0, int(x) - a), min(n, int(x) + b)
                ranges.append((lo, hi - lo))
    for first, cnt in ranges:
        keys, counts = st.kmers(first, cnt), st.counts(first, cnt)
        assert keys.shape == (cnt, ks.nw) and np.array_equal(keys, ks.keys[first:first + cnt]), (first, cnt)
        assert np.array_equal(counts, ks.counts[first:first + cnt]), (first, cnt)
    for first, cnt in ((n - 5, 6), (n, 1), (n + 1, 0), (-1, 2), (0, n + 1)):
        with pytest.raises(SpadesGpuError):
            st.kmers(first, cnt)
        with pytest.raises(SpadesGpuError):
            st.counts(first, cnt)


def test_multichunk_checksum_and_files(multichunk, tmp_path):
    c, st, ks, passes = multichunk
    wsum = int((ks.keys * (2 * np.arange(ks.nw, dtype=np.uint64) + 1)[None, :]).sum(dtype=np.uint64))
    xr = 0
    for q in range(ks.nw):
        r = 7 * q + 1
        col = ks.keys[:, q]
        xr ^= int(np.bitwise_xor.reduce((col << np.uint64(r)) | (col >> np.uint64(64 - r))))
    assert st.checksum() == [ks.n, wsum, xr, int(ks.counts.astype(np.uint64).sum())]
    st.write_buckets(tmp_path / "kmers")
    start = np.concatenate([[0], np.cumsum(ks.bsz)])
    for b in range(len(ks.bsz)):
        assert (tmp_path / ("kmers.%d" % b)).read_bytes() == ks.keys[start[b]:start[b + 1]].tobytes(), b
    st.merge(tmp_path / "final_kmers")
    assert (tmp_path / "final_kmers").read_bytes() == ks.keys.tobytes()


def test_multichunk_index_lookups(multichunk):
    c, st, ks, passes = multichunk
    _check_index_lookups(c, st, ks, 56, 95, "multi-chunk K=56 B=80", n_derived=200_000)


# ---- EdgeIndex ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,K,B,seed", [(21, None, 6, 81), (33, 25, 5000, 82), (55, 40, 3000, 83), (77, None, 3, 84), (63, 47, 4000, 85)])
def test_edge_index_lookups_match_oracle(k, K, B, seed):
    """EdgeIndex.seq_idx of the K-mers of the graph's edges and of absent ones: K = k+1 (one index segment) and K != k+1 counted into
    B buckets, many of them empty"""
    from gpu_util import ctx
    from spades_b200.graph import DeBruijnGraphConstructor, EdgeIndex
    c = ctx()
    c.set_reads(*pack_reads(synthetic_reads(800, 150, 1500, 0.01, seed=seed)))
    gr = DeBruijnGraphConstructor(c, k, 4).ConstructGraph()
    ei = EdgeIndex(gr, K, B)
    ks, m, _, _ = O.edge_index(gr.unitigs(), k, K, 1 if K is None else B)
    assert ei.size() == ks.n
    Kx = k + 1 if K is None else K
    q = query_set(ks.keys, Kx, ks.nw, seed)
    want = m.lookup_many(q)
    _assert_same_lookups(ei.seq_idx(q), want, q, ks.bsz, "edge index k=%d K=%d B=%d" % (k, Kx, B))
    assert np.array_equal(np.sort(want[:ks.n]), np.arange(ks.n, dtype=np.uint64)) and (want == NOT_FOUND).any()
    ei.free(); gr.free()


# ---- read-input paths -----------------------------------------------------------------------------------------------------------
def _ragged_reads(seed):
    rng = np.random.default_rng(seed)
    reads = [r[:int(rng.integers(1, 151))] for r in synthetic_reads(600, 150, 1500, 0.01, seed=seed)]
    return reads + ["A", "ACGT", "ACGTACGTACGTACGTACGTACGT"]


PATH_K, PATH_B = 22, 6


def _count_and_compare(c, reads, what):
    """(keys, counts, bsz), the serialized KMerIndex and seq_idx of every key of the context's current read set against the oracle"""
    words, offs, lens = pack_reads(reads)
    ks = O.count(words, offs, lens, PATH_K, PATH_B, 0)
    st = KMerDiskCounter(c, DeBruijnReadKMerSplitter(PATH_K)).Count(PATH_B)
    assert np.array_equal(st.kmers().ravel(), ks.keys.ravel()), what
    assert np.array_equal(st.counts(), ks.counts) and np.array_equal(st.bucket_sizes(), ks.bsz), what
    idx = KMerIndexBuilder(c).BuildIndex(st)
    m = O.Mphf(ks)
    assert G.index_equal(m.serialize(), idx.serialize(), PATH_B), what
    assert np.array_equal(idx.seq_idx(ks.keys), m.lookup_many(ks.keys)), what
    idx.free(); st.free()


def _append_in_batches(c, reads, nbatch=3):
    """sgpu_reads_append_packed in batches, each with offsets relative to its own words"""
    c.check(c.L.sgpu_reads_clear(c.h))
    cut = np.linspace(0, len(reads), nbatch + 1).astype(int)
    for i in range(nbatch):
        w, o, l = pack_reads(reads[cut[i]:cut[i + 1]])
        c.check(c.L.sgpu_reads_append_packed(c.h, _p(w), len(w), _p(o), _p(l), len(l)))


def _upload_pageable(c, reads):
    words, offs, lens = pack_reads(reads)
    c.upload_reads(words.ctypes.data, len(words), offs.ctypes.data, lens.ctypes.data, len(lens))
    return words, offs, lens                       # must stay alive until the next count has returned


def _upload_pinned(c, torch, reads):
    words, offs, lens = pack_reads(reads)
    t = [torch.from_numpy(words.view(np.int64)).pin_memory(), torch.from_numpy(offs.view(np.int64)).pin_memory(),
         torch.from_numpy(lens.view(np.int32)).pin_memory()]
    c.upload_reads(t[0].data_ptr(), len(words), t[1].data_ptr(), t[2].data_ptr(), len(lens))
    return t


def _adopt(c, torch, s, reads):
    """device tensors written on stream s (the context's stream): int64 words with zero padding, int64 offs, int32 lens"""
    words, offs, lens = pack_reads(reads)
    with torch.cuda.stream(s):
        dw = torch.zeros(len(words) + 8, dtype=torch.int64, device="cuda")
        dw[:len(words)] = torch.from_numpy(words.view(np.int64)).to("cuda")
        do = torch.from_numpy(offs.view(np.int64)).to("cuda")
        dl = torch.from_numpy(lens.view(np.int32)).to("cuda")
    c.adopt_device_reads(dw.data_ptr(), len(words), do.data_ptr(), dl.data_ptr(), len(lens))
    return dw, do, dl


def test_read_input_paths_match_oracle():
    """set_reads, append_packed in three batches, upload from pageable and from pinned host memory, adopt device tensors, all on one
    context that runs on a caller's non-default stream; then set_reads -> adopt -> upload -> set_reads with a different read set each
    time, so that a switch that left reads of the previous set behind would show"""
    import torch
    s = torch.cuda.Stream()
    c = Context(0, stream=s.cuda_stream)
    try:
        reads = _ragged_reads(41)
        c.set_reads(*pack_reads(reads))
        _count_and_compare(c, reads, "set_reads")
        _append_in_batches(c, reads)
        _count_and_compare(c, reads, "append_packed x3")
        keep = _upload_pageable(c, reads)
        _count_and_compare(c, reads, "upload pageable")
        keep = _upload_pinned(c, torch, reads)
        _count_and_compare(c, reads, "upload pinned")
        keep = _adopt(c, torch, s, reads)
        _count_and_compare(c, reads, "adopt device")
        sets = [_ragged_reads(42), synthetic_reads(300, 150, 900, 0.01, seed=43), _ragged_reads(44), synthetic_reads(50, 100, 400, 0.0, seed=45)]
        c.set_reads(*pack_reads(sets[0]))
        _count_and_compare(c, sets[0], "set_reads after adopt")
        keep = _adopt(c, torch, s, sets[1])
        _count_and_compare(c, sets[1], "adopt after set_reads")
        keep = _upload_pageable(c, sets[2])
        _count_and_compare(c, sets[2], "upload after adopt")
        c.set_reads(*pack_reads(sets[3]))
        _count_and_compare(c, sets[3], "set_reads after upload")
        del keep
    finally:
        c.close()
        s.synchronize()
