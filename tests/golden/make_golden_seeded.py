"""Results of the UNMODIFIED reference (oracle/_ref/ref_probe, oracle/_ref/ref_fastx) on the seeded inputs of
tests/test_oracle_vs_reference.py and of the reference-format tests of tests/test_ingest.py.

    make -C oracle ref && python tests/golden/make_golden_seeded.py        (needs the reference sources to build oracle/_ref)

Writes tests/golden/seeded_reference.json (SHA-256 of every artefact, the serialized indices with their uninitialised bytes zeroed,
the small integers, and for the index lookups the SHA-256 of the queries and of the slots returned with the number of NOT_FOUND) and tests/golden/seqfile_reference.npz (the reference's read-back text of our .seq/.off, that .off, and its
own .seq of the same reads).
"""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
import golden_util as G  # noqa: E402
import test_ingest as I  # noqa: E402
import test_oracle_vs_reference as V  # noqa: E402
from spades_b200.packing import synthetic_reads  # noqa: E402
from spades_b200.reads_io import read_fastx  # noqa: E402

PROBE = os.path.join(ROOT, "oracle", "_ref", "ref_probe")
REF_FASTX = os.path.join(ROOT, "oracle", "_ref", "ref_fastx")


def run_probe(mode, reads, k, B, T=3, env_extra=None):
    with tempfile.TemporaryDirectory() as d:
        rf = os.path.join(d, "reads.txt")
        open(rf, "w").write("\n".join(reads) + "\n")
        out = os.path.join(d, "out")
        env = dict(os.environ)
        env.update(env_extra or {})
        subprocess.check_call([PROBE, mode, rf, str(k), str(B), str(T), out], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env, timeout=600)
        g = {f.replace(".", "_"): np.frombuffer(open(os.path.join(out, f), "rb").read(), np.uint8)
             for f in os.listdir(out) if os.path.isfile(os.path.join(out, f))}
    g.update(k=k, B=B)
    return g


def graph_digests(reads, k, B, T=3, early_tc=0):
    g = run_probe("graph", reads, k, B, T, {"PROBE_EARLY_TC": str(early_tc)} if early_tc else None)
    return G.graph_digests(G.ref_graph_art(g), B)


def lookup_digests(k, B, seed):
    """seq_idx under the reference's in-memory k-mer and (k+1)-mer index (PROBE_QUERIES) of the query sets built from the keys it
    stored: the graph run is done twice, first for the keys, then with the queries"""
    reads = V.lookup_reads(seed)
    g = run_probe("graph", reads, k, B)
    nw = (k + 32) // 32                      # k odd: a k-mer and a (k+1)-mer have the same number of words
    qk = V.lookup_queries(np.frombuffer(g["kmers"].tobytes(), np.uint64).reshape(-1, nw), k, 10 * seed + 1)
    qkp = V.lookup_queries(np.frombuffer(g["kpomers"].tobytes(), np.uint64).reshape(-1, nw), k + 1, 10 * seed + 2)
    with tempfile.TemporaryDirectory() as d:
        q = os.path.join(d, "queries")
        qk.tofile(q)
        qkp.tofile(q + ".kp1")
        g = run_probe("graph", reads, k, B, env_extra={"PROBE_QUERIES": q})
    return {"kmer": V.lookup_digests(qk, np.frombuffer(g["kmer_queries_idx_bin"].tobytes(), np.uint64)),
            "kpomer": V.lookup_digests(qkp, np.frombuffer(g["kpomer_queries_idx_bin"].tobytes(), np.uint64))}


def main():
    out = {"graph": {}, "count": {}, "early_tip_clipper": {}, "coverage_prefilter": {}, "parser": {}, "lookup": {}}
    for p in V.LOOKUP:
        out["lookup"][V.case_id(p)] = lookup_digests(*p)
    for p in V.GRAPH:
        k, B, seed = p
        out["graph"][V.case_id(p)] = graph_digests(V.graph_reads(seed), k, B)
    for p in V.COUNT:
        k, B, seed = p
        g = run_probe("count", V.count_reads(seed), k, B)
        out["count"][V.case_id(p)] = V.count_digests(np.frombuffer(g["final_kmers"].tobytes(), np.uint64), G._txt_ints(g["bucket_sizes_txt"]))
    for p in V.TIP_CLIPPER:
        k, B, n, L, glen, err, seed, T = p
        out["early_tip_clipper"][V.case_id(p)] = graph_digests(synthetic_reads(n, L, glen, err, seed=seed), k, B, T, early_tc=L - k)
    for p in V.COVERAGE_PREFILTER:
        k, thr, seed, T = p
        with tempfile.TemporaryDirectory() as d:
            rf = os.path.join(d, "reads.txt")
            open(rf, "w").write("\n".join(V.coverage_prefilter_reads(seed)) + "\n")
            env = dict(os.environ); env["PROBE_COV_THR"] = str(thr)
            subprocess.check_call([PROBE, "covfilter", rf, str(k), "4", str(T), os.path.join(d, "out")], stdout=subprocess.DEVNULL,
                                  stderr=subprocess.DEVNULL, env=env, timeout=600)
            card, bits, mask, _ = [int(v) for v in open(os.path.join(d, "out", "covfilter.txt")).read().split()]
            keep = np.array([int(v) for v in open(os.path.join(d, "out", "keep.txt")).read().split()], dtype=np.uint8)
            hashes = np.fromfile(os.path.join(d, "out", "hashes.bin"), dtype=np.uint64)
        out["coverage_prefilter"][V.case_id(p)] = {"card": card, "key_bits": bits, "range_mask": mask, "keep": G.sha256(keep.tobytes()),
                                                   "hashes": G.sha256(hashes.tobytes())}
    with tempfile.TemporaryDirectory() as d:
        from pathlib import Path
        for f in I.parser_case_files(Path(d)):
            po = os.path.join(d, "ref_parsed.txt")
            subprocess.check_call([REF_FASTX, f, po], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            lines = open(po).read().split("\n")
            recs = int([ln for ln in lines if ln.startswith("#records")][0].split()[1])
            want = [ln for ln in lines if ln and not ln.startswith("#")]
            out["parser"][os.path.basename(f)] = {"sha256": G.sha256("\n".join(want).encode()), "records": recs}
    json.dump(out, open(os.path.join(HERE, "seeded_reference.json"), "w"), indent=1, sort_keys=True)

    reads = I.seqfile_case_reads()
    with tempfile.TemporaryDirectory() as d:
        txt = os.path.join(d, "reads.txt")
        open(txt, "w").write("\n".join(reads) + "\n")
        fa = os.path.join(d, "r.fa")
        open(fa, "w").write("".join(">%d\n%s\n" % (i, s) for i, s in enumerate(reads)))
        prefix = os.path.join(d, "lib")
        read_fastx(fa).write_seqfile(prefix)
        subprocess.check_call([PROBE, "binreads", txt, "21", "1", "3", os.path.join(d, "out"), prefix], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        np.savez_compressed(os.path.join(HERE, "seqfile_reference.npz"),
                            readback=np.frombuffer(open(prefix + "_readback.txt", "rb").read(), np.uint8),
                            off=np.frombuffer(open(prefix + ".off", "rb").read(), np.uint8),
                            ref_seq=np.frombuffer(open(prefix + "_ref.seq", "rb").read(), np.uint8))


if __name__ == "__main__":
    main()
