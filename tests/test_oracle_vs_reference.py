"""CPU test: the C oracle against the UNMODIFIED reference (oracle/_ref/ref_probe) on fresh seeded inputs. The reads are regenerated
here from their seeds; tests/golden/seeded_reference.json holds what the reference produced for them (the SHA-256 of every artefact,
the serialized indices with their uninitialised bytes zeroed, and the small integers), written by tests/golden/make_golden_seeded.py."""
import json
import os

import numpy as np
import pytest

import golden_util as G
import oracle as O
from spades_b200.packing import pack_reads, revcomp, synthetic_reads
from test_oracle_golden import oracle_artifacts

GRAPH = [(21, 16, 11), (31, 5, 12), (55, 30, 13), (63, 9, 14), (77, 4, 15), (127, 6, 16)]
COUNT = [(21, 16, 21), (55, 16, 22), (100, 3, 23)]
TIP_CLIPPER = [(21, 16, 3000, 100, 4000, 0.01, 41, 1), (21, 8, 3000, 100, 2000, 0.03, 42, 8), (55, 30, 3000, 150, 5000, 0.01, 43, 3),
               (77, 4, 1500, 150, 2000, 0.01, 44, 8), (9, 3, 1000, 60, 600, 0.1, 45, 8)]
COVERAGE_PREFILTER = [(21, 2, 51, 1), (20, 3, 52, 8), (55, 2, 53, 3), (63, 4, 54, 8), (69, 2, 55, 2), (127, 3, 56, 8), (11, 6, 57, 8)]
# index lookups: far more buckets than keys in most cases (k = 21, 33, 63, 99, 127: one to four words per record), so that many
# absent keys fall into empty buckets
LOOKUP = [(21, 5000, 61), (33, 3000, 62), (63, 8000, 63), (99, 2000, 64), (127, 1500, 65)]


def case_id(params):
    return "_".join(str(p) for p in params)


def graph_reads(seed):
    return synthetic_reads(1500, 150, 3000, 0.01, seed=seed)


def count_reads(seed):
    return synthetic_reads(800, 150, 2000, 0.01, seed=seed)


def coverage_prefilter_reads(seed):
    rng = np.random.default_rng(seed)
    reads = synthetic_reads(2500, 150, 4000, 0.01, seed=seed) + synthetic_reads(400, 150, 40000, 0.02, seed=seed + 1)
    x = "".join("ACGT"[i] for i in rng.integers(0, 4, 90))
    return reads + [x + revcomp(x)] * 3 + ["A" * 150, "AC" * 70, "ACGTACGT"]


def lookup_reads(seed):
    return synthetic_reads(40, 150, 400, 0.01, seed=seed)


def lookup_queries(keys, K, seed):
    """the query set of one index of a LOOKUP case (tests/query_sets.py), from the keys that index holds"""
    from query_sets import query_set
    return query_set(keys, K, (K + 31) // 32, seed)


def lookup_digests(queries, idx):
    idx = np.asarray(idx, np.uint64)
    return {"queries": G.sha256(np.ascontiguousarray(queries, np.uint64).tobytes()), "n": int(len(queries)),
            "idx": G.sha256(idx.tobytes()), "not_found": int((idx == np.uint64((1 << 64) - 1)).sum())}


def count_digests(keys, bsz):
    return {"final_kmers": G.sha256(np.ascontiguousarray(np.asarray(keys, np.uint64).ravel()).tobytes()),
            "bucket_sizes": G.sha256(np.asarray(bsz, np.int64).tobytes())}


def _want(kind, params):
    fx = json.load(open(os.path.join(G.GOLDEN_DIR, "seeded_reference.json")))
    return fx[kind][case_id(params)]


@pytest.mark.parametrize("k,B,seed", GRAPH)
def test_oracle_vs_live_reference_graph(k, B, seed):
    art, _ = oracle_artifacts(graph_reads(seed), k, B)
    assert G.graph_digests(art, B) == _want("graph", (k, B, seed))


@pytest.mark.parametrize("k,B,seed", COUNT)
def test_oracle_vs_live_reference_kmercount(k, B, seed):
    words, offs, lens = pack_reads(count_reads(seed))
    ks = O.count(words, offs, lens, k, B, 1)
    assert count_digests(ks.keys, ks.bsz) == _want("count", (k, B, seed))


@pytest.mark.parametrize("k,B,n,L,glen,err,seed,T", TIP_CLIPPER)
def test_oracle_vs_live_reference_early_tip_clipper(k, B, n, L, glen, err, seed, T):
    """the reference's clipper runs racily on T threads; its result (and the oracle's) must not depend on T"""
    reads = synthetic_reads(n, L, glen, err, seed=seed)
    art, r = oracle_artifacts(reads, k, B, early_tc=L - k)
    assert G.graph_digests(art, B) == _want("early_tip_clipper", (k, B, n, L, glen, err, seed, T))
    assert r["tc"]["removed"] > 0


@pytest.mark.parametrize("k,thr,seed,T", COVERAGE_PREFILTER)
def test_oracle_vs_live_reference_coverage_prefilter(k, thr, seed, T):
    """SURVEY 8f-3: the CoverageFilter phase of the unmodified reference (HLL bound -> qf::cqf -> median filter, filled by T racing
    threads) against the oracle's restatement: the cardinality bound, the key width, the verdict for every read and the rolling hash
    itself, for k+1 below, at and above 64 (rotation by (k+1) mod 64)"""
    reads = coverage_prefilter_reads(seed)
    want = _want("coverage_prefilter", (k, thr, seed, T))
    words, offs, lens = pack_reads(reads)
    keep, st = O.cov_filter(words, offs, lens, k + 1, thr)
    assert st[0] == want["card"] and st[1] == want["key_bits"] and (1 << st[1]) - 1 == want["range_mask"]
    assert G.sha256(np.asarray(keep, np.uint8).tobytes()) == want["keep"]
    hh = [O.cyclic_hash(words[int(offs[i]):], j, k + 1) for i in range(64) for j in range(max(0, len(reads[i]) - k))]
    assert G.sha256(np.array(hh, dtype=np.uint64).tobytes()) == want["hashes"]


@pytest.mark.parametrize("k,B,seed", LOOKUP)
def test_oracle_vs_live_reference_index_lookups(k, B, seed):
    """KMerIndex::seq_idx of stored keys, their reverse complements, one-base substitutions and random keys, under the k-mer and the
    (k+1)-mer index KMerIndexBuilder::BuildIndex built in memory, against the oracle's orc_mphf_lookup. An absent key whose bucket
    holds no key is NOT_FOUND there (the bucket's mphf was never built, BooPHF.h:425-426,467)."""
    want = _want("lookup", (k, B, seed))
    words, offs, lens = pack_reads(lookup_reads(seed))
    kp = O.count(words, offs, lens, k + 1, B, 0)
    km = O.kmers_from_kpomers(kp, B)
    for name, ks, K, qseed in (("kmer", km, k, 10 * seed + 1), ("kpomer", kp, k + 1, 10 * seed + 2)):
        q = lookup_queries(ks.keys, K, qseed)
        got = lookup_digests(q, O.Mphf(ks).lookup_many(q))
        assert got == want[name], name
        assert (ks.bsz == 0).sum() > 0 and got["not_found"] > 0
