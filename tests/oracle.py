"""ctypes front end of oracle/liboracle.so -- TEST INFRASTRUCTURE (checker only, never the product path)."""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORC_DIR = os.path.join(os.path.dirname(_HERE), "oracle")
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(_ORC_DIR, "liboracle.so")
        src = os.path.join(_ORC_DIR, "spades_oracle.c")
        if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
            subprocess.check_call(["make", "-C", _ORC_DIR, "oracle"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        L = C.CDLL(so)
        vp, i64, i32, u64 = C.c_void_p, C.c_int64, C.c_int, C.c_uint64
        L.orc_xxh3_64.restype = u64; L.orc_xxh3_64.argtypes = [vp, i32]
        L.orc_xxh3_128.restype = None; L.orc_xxh3_128.argtypes = [vp, i32, vp, vp]
        L.orc_bucket.restype = u64; L.orc_bucket.argtypes = [vp, i32, u64]
        L.orc_is_minimal.restype = i32; L.orc_is_minimal.argtypes = [vp, i32]
        L.orc_rc.restype = None; L.orc_rc.argtypes = [vp, i32, vp]
        L.orc_count.restype = vp; L.orc_count.argtypes = [vp, vp, vp, i64, i32, i32, i32]
        L.orc_kmers_from_kpomers.restype = vp; L.orc_kmers_from_kpomers.argtypes = [vp, i32]
        for f in ("orc_kset_keys", "orc_kset_counts", "orc_kset_bsz"):
            getattr(L, f).restype = vp; getattr(L, f).argtypes = [vp]
        L.orc_kset_n.restype = i64; L.orc_kset_n.argtypes = [vp]
        L.orc_kset_nw.restype = i32; L.orc_kset_nw.argtypes = [vp]
        L.orc_kset_free.restype = None; L.orc_kset_free.argtypes = [vp]
        L.orc_mphf_build.restype = vp; L.orc_mphf_build.argtypes = [vp]
        L.orc_mphf_free.restype = None; L.orc_mphf_free.argtypes = [vp]
        L.orc_mphf_lookup.restype = u64; L.orc_mphf_lookup.argtypes = [vp, vp]
        L.orc_mphf_lookup_many.restype = None; L.orc_mphf_lookup_many.argtypes = [vp, vp, i64, vp]
        L.orc_mphf_nfinal.restype = u64; L.orc_mphf_nfinal.argtypes = [vp]
        L.orc_mphf_serialize.restype = i64; L.orc_mphf_serialize.argtypes = [vp, vp]
        L.orc_masks.restype = None; L.orc_masks.argtypes = [vp, vp, vp, i64]
        L.orc_coverage.restype = None; L.orc_coverage.argtypes = [vp, vp, vp]
        L.orc_histogram.restype = i64; L.orc_histogram.argtypes = [vp, i64, vp, i64]
        L.orc_early_tip_clip.restype = i64; L.orc_early_tip_clip.argtypes = [vp, vp, vp, i64, i32, vp, vp]
        L.orc_unitigs.restype = vp; L.orc_unitigs.argtypes = [vp, vp, vp, i32]
        L.orc_unitigs_n.restype = i64; L.orc_unitigs_n.argtypes = [vp]
        L.orc_unitig_len.restype = i64; L.orc_unitig_len.argtypes = [vp, i64]
        L.orc_unitig_seq.restype = vp; L.orc_unitig_seq.argtypes = [vp, i64]
        L.orc_unitigs_free.restype = None; L.orc_unitigs_free.argtypes = [vp]
        L.orc_gfa.restype = vp; L.orc_gfa.argtypes = [vp, vp, vp, vp, C.c_char_p, vp]
        L.orc_free.restype = None; L.orc_free.argtypes = [vp]
        L.orc_cyclic_hash.restype = u64; L.orc_cyclic_hash.argtypes = [vp, i64, i32]
        L.orc_cov_filter.restype = None; L.orc_cov_filter.argtypes = [vp, vp, vp, i64, i32, C.c_uint, vp, vp]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def xxh3_64(words):
    w = np.ascontiguousarray(words, dtype=np.uint64)
    return int(lib().orc_xxh3_64(_p(w), len(w)))


def xxh3_128(words):
    w = np.ascontiguousarray(words, dtype=np.uint64)
    lo, hi = C.c_uint64(), C.c_uint64()
    lib().orc_xxh3_128(_p(w), len(w), C.byref(lo), C.byref(hi))
    return lo.value, hi.value


class KSet:
    def __init__(self, h, K, B):
        self.h, self.K, self.B = h, K, B
        L = lib()
        self.n = L.orc_kset_n(h)
        self.nw = L.orc_kset_nw(h)
        self.keys = np.ctypeslib.as_array(C.cast(L.orc_kset_keys(h), C.POINTER(C.c_uint64)), shape=(max(self.n, 1) * self.nw,))[: self.n * self.nw].reshape(self.n, self.nw).copy()
        cp = L.orc_kset_counts(h)
        self.counts = None if not cp else np.ctypeslib.as_array(C.cast(cp, C.POINTER(C.c_uint32)), shape=(max(self.n, 1),))[: self.n].copy()
        self.bsz = np.ctypeslib.as_array(C.cast(L.orc_kset_bsz(h), C.POINTER(C.c_int64)), shape=(B,)).copy()

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_kset_free(self.h); self.h = None


def count(words, offs, lens, K, B, mode):
    words = np.ascontiguousarray(words, np.uint64); offs = np.ascontiguousarray(offs, np.uint64); lens = np.ascontiguousarray(lens, np.uint32)
    h = lib().orc_count(_p(words), _p(offs), _p(lens), len(lens), K, B, mode)
    return KSet(h, K, B)


def kmers_from_kpomers(kp: KSet, B):
    return KSet(lib().orc_kmers_from_kpomers(kp.h, B), kp.K - 1, B)


class Mphf:
    def __init__(self, ks: KSet):
        self.ks = ks
        self.h = lib().orc_mphf_build(ks.h)

    def serialize(self) -> bytes:
        n = lib().orc_mphf_serialize(self.h, None)
        buf = np.zeros(n, np.uint8)
        lib().orc_mphf_serialize(self.h, _p(buf))
        return buf.tobytes()

    def lookup(self, key_words):
        w = np.ascontiguousarray(key_words, np.uint64)
        return int(lib().orc_mphf_lookup(self.h, _p(w)))

    def lookup_many(self, keys):
        """seq_idx of every row of keys [n, nw] (stored form); -1 as 2^64 - 1"""
        w = np.ascontiguousarray(keys, np.uint64).reshape(-1, self.ks.nw)
        out = np.zeros(max(len(w), 1), np.uint64)
        lib().orc_mphf_lookup_many(self.h, _p(w), len(w), _p(out))
        return out[: len(w)]

    def nfinal(self):
        return int(lib().orc_mphf_nfinal(self.h))

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_mphf_free(self.h); self.h = None


def masks(kp: KSet, mk: Mphf, nk):
    out = np.zeros(max(nk, 1), np.uint8)
    lib().orc_masks(kp.h, mk.h, _p(out), nk)
    return out[:nk]


def coverage(kp: KSet, mkp: Mphf):
    out = np.zeros(max(kp.n, 1), np.uint32)
    lib().orc_coverage(kp.h, mkp.h, _p(out))
    return out[: kp.n]


def histogram(cov):
    cov = np.ascontiguousarray(cov, np.uint32)
    mx = lib().orc_histogram(_p(cov), len(cov), None, 0)
    hist = np.zeros(max(mx, 1), np.uint64)
    lib().orc_histogram(_p(cov), len(cov), _p(hist), mx)
    return hist[:mx]


def early_tip_clip(km: KSet, mk: Mphf, masks_arr, length_bound, snapshot=False):
    """EarlyTipClipperProcessor::ClipTips on a copy of the mask array -> (masks, removed k-mers, tipped junctions, clipped links)"""
    m = np.array(masks_arr, np.uint8, copy=True)
    if m.size == 0:
        return m, 0, 0, 0
    nt, nc = C.c_int64(), C.c_int64()
    removed = lib().orc_early_tip_clip(km.h, mk.h, _p(m), int(length_bound), 1 if snapshot else 0, C.byref(nt), C.byref(nc))
    return m, int(removed), int(nt.value), int(nc.value)


def early_at_clip(km: KSet, mk: Mphf, masks_arr, ratio=0.8, min_len=10, max_len=200, snapshot=False):
    """EarlyLowComplexityClipperProcessor::RemoveATEdges + RemoveATTips on a copy of the mask array
    -> (masks, [edges collected, links removed, k-mers removed, clipped tips])"""
    m = np.array(masks_arr, np.uint8, copy=True)
    out = np.zeros(4, np.int64)
    if m.size:
        L = lib()
        L.orc_early_at_clip.restype = None
        L.orc_early_at_clip.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int64, C.c_int64, C.c_int, C.c_void_p]
        L.orc_early_at_clip(km.h, mk.h, _p(m), float(ratio), int(min_len), int(max_len), 1 if snapshot else 0, _p(out))
    return m, [int(x) for x in out]


class Unitigs:
    def __init__(self, km: KSet, mk: Mphf, masks_arr, keep_loops=True):
        m = np.ascontiguousarray(masks_arr, np.uint8)
        self.h = lib().orc_unitigs(km.h, mk.h, _p(m), 1 if keep_loops else 0)
        L = lib()
        self.seqs = []
        lut = np.frombuffer(b"ACGT", np.uint8)
        for i in range(L.orc_unitigs_n(self.h)):
            n = L.orc_unitig_len(self.h, i)
            a = np.ctypeslib.as_array(C.cast(L.orc_unitig_seq(self.h, i), C.POINTER(C.c_uint8)), shape=(n,))
            self.seqs.append(lut[a].tobytes().decode())

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_unitigs_free(self.h); self.h = None


def gfa(u: Unitigs, mk: Mphf, mkp: Mphf = None, cov=None, version="SPAdes-4.3.0-dev") -> str:
    n = C.c_int64()
    covp = None
    if cov is not None:
        cov = np.ascontiguousarray(cov, np.uint32); covp = _p(cov)
    p = lib().orc_gfa(u.h, mk.h, mkp.h if mkp else None, covp, version.encode(), C.byref(n))
    s = C.string_at(p, n.value).decode()
    lib().orc_free(p)
    return s


def full_graph(reads, k, B, early_tc=0, early_at=False):
    """Whole path on a list of ACGT strings; returns dict of artefacts named like ref_probe's files.
    early_tc > 0: run the early tip clipper with that length bound between the mask fill and the unitig extraction
    (stages/construction.cpp:289-302); `masks` then holds the clipped array and `masks_raw` the one before."""
    from spades_b200.packing import pack_reads
    if k % 2 == 0:
        raise ValueError("k must be odd (projects/spades_tools/gbuilder.cpp:125): with even k a k-mer can be its own reverse complement")
    words, offs, lens = pack_reads(reads)
    kp = count(words, offs, lens, k + 1, B, 0)
    km = kmers_from_kpomers(kp, B)
    mk = Mphf(km)
    mkp = Mphf(kp)
    mk_arr = masks(kp, mk, km.n)
    raw = mk_arr
    tc = None
    at = None
    if early_at:                  # the RNA pipeline's EarlyATClipper runs before the tip clipper (stages/construction.cpp:447-450)
        mk_arr, at = early_at_clip(km, mk, mk_arr)
    if early_tc:
        mk_arr, removed, tipped, clipped = early_tip_clip(km, mk, mk_arr, early_tc)
        tc = dict(removed=removed, tipped=tipped, clipped=clipped)
    cov = coverage(kp, mkp)
    u = Unitigs(km, mk, mk_arr, True)
    return dict(kp=kp, km=km, mk=mk, mkp=mkp, masks=mk_arr, masks_raw=raw, tc=tc, at=at, cov=cov, hist=histogram(cov), unitigs=u,
                gfa=gfa(u, mk, mkp, cov))


def edge_index(unitig_seqs, k, K=None, B=1):
    """EdgeIndex refill restated on top of the oracle's count / MPHF (test infrastructure; python loops: small cases only).
    keys   = the minimal form of every K-mer of every edge (GraphPositionFillingIndexBuilder::BuildIndexFromGraph,
             assembly_graph/index/edge_index_builders.hpp:154-307; KmerFreeEdgeIndex is an InvertableStoring map, storing_traits.hpp:74,
             92-101) = the canonical count over the primary strands; K = k+1 -> one index segment (KMerFullGraphStorage:
             segment_policy_.reset(1)), else B buckets.
    values = EdgeInfoUpdater::UpdateKMers (edge_info_updater.hpp:38-48: windows that are minimal as they stand, on every edge and its
             conjugate) + PutInIndex (edge_position_index.hpp:152-167): one put -> (edge id, offset), more -> TOMBSTONE. Edge ids:
             edge i -> 3 + 2i, conjugate +1, self-conjugate edges once (graph_core.hpp:233,514-531).
    Returns (KSet, Mphf, ids u64[n], offsets u32[n]) in slot order."""
    from spades_b200.packing import pack_reads, revcomp
    K = k + 1 if K is None else K
    words, offs, lens = pack_reads(unitig_seqs)
    ks = count(words, offs, lens, K, B, 0)
    m = Mphf(ks)
    ids = np.full(ks.n, (1 << 64) - 1, np.uint64)
    off = np.full(ks.n, 0x7FFFFFFF, np.uint32)
    occ = np.zeros(ks.n, np.int64)
    puts = []
    for i, s in enumerate(unitig_seqs):
        strands = [(s, 3 + 2 * i)]
        if revcomp(s) != s:
            strands.append((revcomp(s), 3 + 2 * i + 1))
        for seq, eid in strands:
            for j in range(len(seq) - K + 1):
                kmer = seq[j:j + K]
                if kmer > revcomp(kmer):              # RtSeq::IsMinimal: nucleotide order from position 0, ties (self-RC) are minimal
                    continue
                w, _, _ = pack_reads([kmer])
                slot = m.lookup(w)
                occ[slot] += 1
                puts.append((slot, eid, j))
    for slot, eid, j in puts:
        if occ[slot] == 1:
            ids[slot] = eid; off[slot] = j
        else:
            ids[slot] = (1 << 64) - 2; off[slot] = 0x7FFFFFFE
    return ks, m, ids, off


def cyclic_hash(words, pos, K):
    """SymmetricCyclicHash<NDNASeqHash>(K) of the window at base `pos` of a packed sequence (adt/cyclichash.hpp:187-259)"""
    w = np.ascontiguousarray(words, dtype=np.uint64)
    return int(lib().orc_cyclic_hash(_p(w), pos, K))


def cov_filter(words, offs, lens, K, thr):
    """the pipeline's coverage pre-filter over K-mers (K = k+1): (keep flag per read, [cardinality bound, key bits, distinct keys, kept])"""
    words = np.ascontiguousarray(words, dtype=np.uint64)
    offs = np.ascontiguousarray(offs, dtype=np.uint64)
    lens = np.ascontiguousarray(lens, dtype=np.uint32)
    keep = np.zeros(len(lens), dtype=np.uint8)
    stats = np.zeros(4, dtype=np.uint64)
    lib().orc_cov_filter(_p(words), _p(offs), _p(lens), len(lens), K, thr, _p(keep), _p(stats))
    return keep, [int(x) for x in stats]
