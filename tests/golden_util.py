"""Load tests/golden/*.npz (reference outputs) and compare an implementation's artefacts against them."""
import glob
import hashlib
import os
import struct

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def names(mode=None):
    out = []
    for p in sorted(glob.glob(os.path.join(GOLDEN_DIR, "*.npz"))):
        n = os.path.basename(p)[:-4]
        if mode is None or n.endswith("_" + mode) or (mode == "graph" and n.startswith("gtest_")):
            out.append(n)
    return out


def load(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    g = {k: z[k] for k in z.files}
    g["reads"] = g["reads"].tobytes().decode().split("\n")
    g["k"] = int(g["k"][0]); g["B"] = int(g["B"][0]) if "B" in g else 0; g["mode"] = g["mode"].tobytes().decode()
    if "tc_bound" in g:
        g["tc_bound"] = int(g["tc_bound"][0])
    for f in ("ei_k", "ei_chunks"):
        if f in g:
            g[f] = np.asarray(g[f])
    return g


def _txt_ints(a):
    s = a.tobytes().decode().split()
    return np.array([int(x) for x in s], dtype=np.int64)


def strip_uleb_k(ref_bytes, k):
    """IndexWrapper::BinWrite prefixes KMerIndex::serialize with ULEB128(k) (io/binary/binary.hpp:109-146)."""
    v, shift, i = 0, 0, 0
    while True:
        b = ref_bytes[i]; i += 1
        v |= (b & 0x7F) << shift; shift += 7
        if not (b & 0x80):
            break
    assert v == k
    return bytes(ref_bytes[i:])


def index_equal(ref: bytes, mine: bytes, nbuckets: int):
    """Byte compare of KMerIndex::serialize output; the reference writes an UNINITIALISED _lastbitsetrank for
    empty buckets (BooPHF.h:514-517 with build() returning early at :426), so those 8 bytes are masked."""
    if len(ref) != len(mine):
        return False
    ref = bytearray(ref); mine = bytearray(mine)
    p = 8
    for _ in range(nbuckets):
        n = struct.unpack_from("<Q", mine, p + 20)[0]
        if n == 0:
            ref[p + 12:p + 20] = b"\0" * 8
            mine[p + 12:p + 20] = b"\0" * 8
        p += 28
        if n:
            for _l in range(25):
                _size, nchar = struct.unpack_from("<QQ", mine, p); p += 16 + 8 * nchar
                nr = struct.unpack_from("<Q", mine, p)[0]; p += 8 + 8 * nr
        p += 8
    return ref == mine


def sha256(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def _same_keys(g, name, keys):
    """large key arrays are stored as their SHA-256 (`<name>_sha256`) to keep each fixture under 1 MB"""
    mine = np.ascontiguousarray(np.asarray(keys, np.uint64).ravel()).tobytes()
    if name in g:
        return g[name].tobytes() == mine
    return g[name + "_sha256"].tobytes().decode() == sha256(mine)


def canonical_index(blob, nbuckets):
    """KMerIndex::serialize bytes with the uninitialised _lastbitsetrank of empty buckets zeroed (see index_equal)"""
    b = bytearray(blob)
    p = 8
    for _ in range(nbuckets):
        n = struct.unpack_from("<Q", b, p + 20)[0]
        if n == 0:
            b[p + 12:p + 20] = b"\0" * 8
        p += 28
        if n:
            for _l in range(25):
                _size, nchar = struct.unpack_from("<QQ", b, p); p += 16 + 8 * nchar
                nr = struct.unpack_from("<Q", b, p)[0]; p += 8 + 8 * nr
        p += 8
    return bytes(b)


def ref_graph_art(g):
    """ref_probe graph output (file name -> bytes, dots as underscores) as the artefact dict check_graph takes"""
    k, B = g["k"], g["B"]
    art = dict(kpomers=np.frombuffer(g["kpomers"].tobytes(), np.uint64), kp_bsz=_txt_ints(g["kpomer_bucket_sizes_txt"]),
               kmers=np.frombuffer(g["kmers"].tobytes(), np.uint64), kmer_index=strip_uleb_k(g["kmer_index_bin"].tobytes(), k),
               kpomer_index=strip_uleb_k(g["kpomer_index_bin"].tobytes(), k + 1),
               masks=g["masks_tc_bin"] if "masks_tc_bin" in g else (g["masks_at_bin"] if "masks_at_bin" in g else g["masks_bin"]),
               cov=np.frombuffer(g["coverage_bin"].tobytes(), np.uint32), hist=_txt_ints(g["histogram_txt"]),
               unitigs=g["unitigs_txt"].tobytes().decode().split(), gfa=g["graph_gfa"].tobytes().decode())
    if "masks_tc_bin" in g:
        art.update(masks_raw=g["masks_bin"], tc_removed=int(g["tc_removed_txt"].tobytes().decode().split()[0]))
    return art


def graph_digests(art, B):
    """SHA-256 of every artefact of check_graph's dict (the serialized indices canonicalised), integers as they are"""
    out = {}
    for key, v in art.items():
        if key in ("kpomers", "kmers"):
            out[key] = sha256(np.ascontiguousarray(np.asarray(v, np.uint64).ravel()).tobytes())
        elif key in ("kp_bsz", "hist"):
            out[key] = sha256(np.asarray(v, np.int64).tobytes())
        elif key in ("masks", "masks_raw"):
            out[key] = sha256(np.asarray(v, np.uint8).tobytes())
        elif key == "cov":
            out[key] = sha256(np.asarray(v, np.uint32).tobytes())
        elif key in ("kmer_index", "kpomer_index"):
            out[key] = sha256(canonical_index(v, B))
        elif key == "unitigs":
            out[key] = sha256("\n".join(v).encode())
        elif key == "gfa":
            out[key] = sha256(v.encode())
        elif key == "tc_removed":
            out[key] = int(v)
    return out


def check_graph(g, art):
    """art: dict with kpomers,kp_bsz,kmers,kmer_index,kpomer_index,masks,cov,hist,unitigs,gfa (any subset)."""
    k, B = g["k"], g["B"]
    bad = []
    def chk(name, ok):
        if not ok:
            bad.append(name)
    if "kpomers" in art:
        chk("kpomers", _same_keys(g, "kpomers", art["kpomers"]))
    if "kp_bsz" in art:
        chk("kp_bsz", np.array_equal(_txt_ints(g["kpomer_bucket_sizes_txt"]), np.asarray(art["kp_bsz"], np.int64)))
    if "kp_counts_sorted" in art:
        pass
    if "kmers" in art:
        chk("kmers", _same_keys(g, "kmers", art["kmers"]))
    if "kmer_index" in art:
        chk("kmer_index", index_equal(strip_uleb_k(g["kmer_index_bin"].tobytes(), k), art["kmer_index"], B))
    if "kpomer_index" in art:
        chk("kpomer_index", index_equal(strip_uleb_k(g["kpomer_index_bin"].tobytes(), k + 1), art["kpomer_index"], B))
    if "masks" in art:     # clipper fixtures: `masks` is the array after the last clipper that ran (masks_tc.bin, else masks_at.bin)
        want = g["masks_tc_bin"] if "masks_tc_bin" in g else (g["masks_at_bin"] if "masks_at_bin" in g else g["masks_bin"])
        chk("masks", np.array_equal(want, np.asarray(art["masks"], np.uint8)))
    if "at_removed" in art:    # (RemoveATEdges' return value, RemoveATTips' return value)
        chk("at_removed", [int(x) for x in g["at_removed_txt"].tobytes().decode().split()] == [int(x) for x in art["at_removed"]])
    if "masks_raw" in art and "masks_tc_bin" in g:
        chk("masks_raw", np.array_equal(g["masks_bin"], np.asarray(art["masks_raw"], np.uint8)))
    if "tc_removed" in art:
        chk("tc_removed", int(g["tc_removed_txt"].tobytes().decode().split()[0]) == int(art["tc_removed"]))
    if "cov" in art:
        chk("cov", np.array_equal(np.frombuffer(g["coverage_bin"].tobytes(), np.uint32), np.asarray(art["cov"], np.uint32)))
    if "hist" in art:
        chk("hist", np.array_equal(_txt_ints(g["histogram_txt"]), np.asarray(art["hist"], np.int64)))
    if "unitigs" in art:
        chk("unitigs", g["unitigs_txt"].tobytes().decode().split() == list(art["unitigs"]))
    if "gfa" in art:
        chk("gfa", g["graph_gfa"].tobytes().decode() == art["gfa"])
    return bad


def check_edge_index(g, ei_bytes, ids, offs, nbuckets):
    """EdgeIndex fixtures: edge_index.bin = ULEB(K) + KMerIndex::serialize, edge_index_values.bin = per slot {u64 edge id, u32 offset}"""
    bad = []
    K = int(g["ei_k"][0])
    if not index_equal(strip_uleb_k(g["edge_index_bin"].tobytes(), K), ei_bytes, nbuckets):
        bad.append("edge_index")
    v = g["edge_index_values_bin"].reshape(-1, 12)
    want_ids = v[:, :8].copy().view(np.uint64).ravel(); want_off = v[:, 8:].copy().view(np.uint32).ravel()
    if not np.array_equal(want_ids, np.asarray(ids, np.uint64)):
        bad.append("edge_ids")
    if not np.array_equal(want_off, np.asarray(offs, np.uint32)):
        bad.append("edge_offsets")
    return bad


def check_count(g, art):
    bad = []
    if not np.array_equal(np.frombuffer(g["final_kmers"].tobytes(), np.uint64), np.asarray(art["final_kmers"], np.uint64).ravel()):
        bad.append("final_kmers")
    if not np.array_equal(_txt_ints(g["bucket_sizes_txt"]), np.asarray(art["bsz"], np.int64)):
        bad.append("bucket_sizes")
    return bad
