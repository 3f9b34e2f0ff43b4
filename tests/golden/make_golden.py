"""Generates tests/golden/*.npz from the UNMODIFIED reference (oracle/_ref/ref_probe).

Needs the reference sources to have built oracle/_ref:
    make -C oracle ref && python tests/golden/make_golden.py
Each fixture holds the input reads and every artefact ref_probe dumps for them (key arrays over 1 MB as their SHA-256), so the
oracle and the CUDA path can be pinned against reference output on machines without the reference.
"""
import gzip
import hashlib
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from spades_b200.packing import longest_valid, revcomp, synthetic_reads  # noqa: E402

PROBE = os.path.join(ROOT, "oracle", "_ref", "ref_probe")


def ecoli_reads():
    """the reference's own test data set (src/projects/spades/test_dataset), stored next to this script"""
    reads = []
    for f in ("ecoli_1K_1.fq.gz", "ecoli_1K_2.fq.gz"):
        lines = gzip.open(os.path.join(HERE, f), "rt").read().split("\n")
        for i in range(1, len(lines), 4):
            s = longest_valid(lines[i].strip().upper())
            if s:
                reads.append(s)
    return reads


def loops_reads():
    rng = np.random.default_rng(5)
    g = "".join("ACGT"[i] for i in rng.integers(0, 4, 500))
    gg = g + g
    reads = [gg[i:i + 120] for i in range(0, 500, 7)]
    x = "".join("ACGT"[i] for i in rng.integers(0, 4, 200))
    h = x + revcomp(x)
    hh = h + h
    reads += [hh[i:i + 150] for i in range(0, 400, 5)]
    return reads


# the six literal-read cases of src/test/debruijn/construction_test.cpp:30-64 (k=5) with their etalon edges
GTEST_CASES = {
    "SimpleThread": (["ACAAACCACCA"], ["ACAAACCACCA"]),
    "SimpleThread2": (["ACAAACCACCC", "AAACCACCCAC"], ["ACAAACCACCCAC"]),
    "SplitThread": (["ACAAACCACCA", "ACAAACAACCC"], ["ACAAAC", "CAAACCACCA", "CAAACAACCC"]),
    "SplitThread2": (["ACAAACCACCA", "ACAAACAACCA"], ["AACCACCA", "ACAAAC", "CAAACCA", "CAAACAACCA"]),
    "Buldge": (["ACAAAACACCA", "ACAAACCACCA"], ["ACAAAACACCA", "ACAAACCACCA"]),
    "CondenseSimple": (["CGAAACCAC", "CGAAAACAC", "AACCACACC", "AAACACACC"], ["CGAAAACACAC", "CACACC", "CGAAACCACAC"]),
}


def at_reads(n, L, glen, err, seed):
    """RNA-like reads: poly-A tails, poly-T heads, A-rich noisy tails and pure low-complexity reads on top of the SURVEY 8(d) generator"""
    rng = np.random.default_rng(seed)
    out = []
    for r in synthetic_reads(n, L, glen, err, seed=seed):
        x = rng.random()
        if x < 0.15:
            cut = int(rng.integers(L // 3, L - 5)); r = r[:cut] + "A" * (L - cut)
        elif x < 0.25:
            cut = int(rng.integers(5, L // 2)); r = "T" * cut + r[cut:]
        elif x < 0.30:
            cut = int(rng.integers(L // 3, L - 5)); r = r[:cut] + "".join(rng.choice(list("AAAAAAAT"), L - cut))
        out.append(r)
    return out + ["A" * L] * 5 + ["AT" * (L // 2)] * 3


def run_probe(mode, reads, k, B, T=2, early_tc=0, early_at=False, edge_index=None):
    with tempfile.TemporaryDirectory() as d:
        rf = os.path.join(d, "reads.txt")
        open(rf, "w").write("\n".join(reads) + "\n")
        out = os.path.join(d, "out")
        env = dict(os.environ)
        if edge_index is not None:
            env["PROBE_EDGE_INDEX"] = str(edge_index)  # EdgeIndex refill over the constructed graph: 0 = (k+1)-mers, else that K (counting path)
        if early_at:
            env["PROBE_EARLY_AT"] = "1"                # EarlyLowComplexityClipperProcessor (RNA pipeline), before the tip clipper
        if early_tc:
            env["PROBE_EARLY_TC"] = str(early_tc)      # EarlyTipClipperProcessor between mask fill and unitig extraction
        subprocess.check_call([PROBE, mode, rf, str(k), str(B), str(T), out], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
        res = {}
        for f in os.listdir(out):
            p = os.path.join(out, f)
            if os.path.isfile(p):
                res[f.replace(".", "_")] = np.frombuffer(open(p, "rb").read(), dtype=np.uint8)
        return res


def save(name, mode, reads, k, B, early_tc=0, edge_index=None):
    """mode "tcgraph" = graph mode with the pipeline's early tip clipper (length bound early_tc); masks_bin is the array
    before the clipper, masks_tc_bin after it, everything downstream (unitigs, GFA) comes from the clipped index.
    mode "atgraph" = graph mode with the RNA pipeline's early A/T clipper (masks_at_bin, at_removed_txt), followed by the tip clipper
    when early_tc is given (then masks_tc_bin is the array after both)."""
    res = run_probe("graph" if mode in ("tcgraph", "atgraph", "eigraph") else mode, reads, k, B, early_tc=early_tc, early_at=(mode == "atgraph"),
                    edge_index=edge_index)
    if edge_index is not None:
        res["ei_k"] = np.array([edge_index if edge_index else k + 1])
        res["ei_chunks"] = np.array([10 * 2])          # run_probe's T = 2: the (k+1)-mer path walks the edges in 10 x T vertex chunks
    if early_tc:
        res["tc_bound"] = np.array([early_tc])
    for key in ("kpomers", "kmers"):
        if key in res and res[key].size > (1 << 20):
            res[key + "_sha256"] = np.frombuffer(hashlib.sha256(res.pop(key).tobytes()).hexdigest().encode(), dtype=np.uint8)
    res["reads"] = np.frombuffer("\n".join(reads).encode(), dtype=np.uint8)
    res["k"] = np.array([k]); res["B"] = np.array([B]); res["mode"] = np.frombuffer(mode.encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **res)
    print(name, {a: len(b) for a, b in res.items() if a not in ("k", "B", "mode")})


def save_covfilter(name, reads, k, thr):
    """SURVEY 8f-3: ref_probe covfilter = the pipeline's CoverageFilter phase (EstimateCardinalityUpperBound -> qf::cqf ->
    FillCoverageHistogram -> CoverageFilter on every read) over (k+1)-mers; keeps the cardinality bound, the filter's key bits, the
    verdict per read and the SymmetricCyclicHash of every window of the first 64 reads."""
    with tempfile.TemporaryDirectory() as d:
        rf = os.path.join(d, "reads.txt")
        open(rf, "w").write("\n".join(reads) + "\n")
        out = os.path.join(d, "out")
        env = dict(os.environ); env["PROBE_COV_THR"] = str(thr)
        subprocess.check_call([PROBE, "covfilter", rf, str(k), "4", "2", out], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
        card, bits, mask, _ = [int(x) for x in open(os.path.join(out, "covfilter.txt")).read().split()]
        keep = np.array([int(x) for x in open(os.path.join(out, "keep.txt")).read().split()], dtype=np.uint8)
        hashes = np.fromfile(os.path.join(out, "hashes.bin"), dtype=np.uint64)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), reads=np.frombuffer("\n".join(reads).encode(), dtype=np.uint8), k=np.array([k]),
                        thr=np.array([thr]), card=np.array([card], dtype=np.uint64), key_bits=np.array([bits]), range_mask=np.array([mask], dtype=np.uint64),
                        keep=keep, hashes=hashes, mode=np.frombuffer(b"covfilter", dtype=np.uint8))
    print(name, "reads", len(reads), "kept", int(keep.sum()), "card", card, "key bits", bits)


def covfilter_reads(seed):
    """a well-covered genome, a thinly covered one, palindromes (self-RC (k+1)-mers), short and low-complexity reads"""
    rng = np.random.default_rng(seed)
    reads = synthetic_reads(2500, 100, 4000, 0.01, seed=seed) + synthetic_reads(400, 100, 30000, 0.01, seed=seed + 1)
    x = "".join("ACGT"[i] for i in rng.integers(0, 4, 60))
    pal = x + revcomp(x)
    reads += [pal] * 4 + [pal[10:110]] * 2 + ["A" * 100] * 3 + ["ACGT" * 10, "ACGTACGTAC", "AC" * 45]
    order = rng.permutation(len(reads))
    return [reads[i] for i in order]


REF_FASTX = os.path.join(ROOT, "oracle", "_ref", "ref_fastx")


def ingest_case_files():
    """small FASTA/FASTQ files that exercise the vendored kseq's corner semantics (see tests/test_ingest.py)"""
    rng = np.random.default_rng(11)
    def rnd(n, pn=0.0, lower=0.0):
        s = rng.choice(list("ACGT"), n)
        s = np.where(rng.random(n) < pn, "N", s)
        s = np.where(rng.random(n) < lower, np.char.lower(s), s)
        return "".join(s)
    seqs = [rnd(int(rng.integers(1, 200)), 0.03, 0.2) for _ in range(120)] + ["", "NNNN", "n", "ACGT ACGTA"]
    fq = "".join("@r%d c\n%s\n+\n%s\n" % (i, s, ("@>+I" * (len(s) // 4 + 1))[:len(s)]) for i, s in enumerate(seqs))
    fa = "junk before the first record\n" + "".join(">s%d\n%s\n%s" % (i, "\n".join(s[j:j + 40] for j in range(0, len(s), 40)), "\n" if i % 4 == 0 else "")
                                                    for i, s in enumerate(seqs)) + ">last\nACGTTGCA"
    mq = "".join("@m%d\n%s\n+m%d\n%s\nnoise without markers\n" % (i, "\n".join((s or "A")[j:j + 30] for j in range(0, len(s or "A"), 30)), i,
                                                                      "\n".join(("I" * len(s or "A"))[j:j + 30] for j in range(0, len(s or "A"), 30)))
                 for i, s in enumerate(seqs[:60]))
    return {"fastq": fq.encode(), "fastq_crlf_gz": gzip.compress(fq.replace("\n", "\r\n").encode()), "fasta_multiline": fa.encode(), "fastq_multiline": mq.encode()}


def save_ingest():
    res = {}
    with tempfile.TemporaryDirectory() as d:
        for name, data in ingest_case_files().items():
            f = os.path.join(d, name + (".gz" if name.endswith("_gz") else ".txt"))
            open(f, "wb").write(data)
            out = os.path.join(d, "out.txt")
            subprocess.check_call([REF_FASTX, f, out], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            res["file_" + name] = np.frombuffer(data, np.uint8)
            res["parsed_" + name] = np.frombuffer(open(out, "rb").read(), np.uint8)
    np.savez_compressed(os.path.join(HERE, "ingest_cases.npz"), **res)
    print("ingest_cases", {a: len(b) for a, b in res.items()})


if __name__ == "__main__":
    save_ingest()
    ec = ecoli_reads()
    save("ecoli_k21_B40_graph", "graph", ec, 21, 40)          # BASELINE.json configs[0]
    save("ecoli_k21_B16_count", "count", ec, 21, 16)          # spades-kmercount defaults (kmercount.cpp:220)
    save("ecoli_k55_B16_graph", "graph", ec[:1500], 55, 16)
    save("ecoli_k77_B7_graph", "graph", ec[:800], 77, 7)
    save("ecoli_k99_B3_graph", "graph", ec[:800], 99, 3)
    save("syn_k21_B10_graph", "graph", synthetic_reads(400, 100, 1500, 0.01, seed=1), 21, 10)
    save("syn_k33_B5_count", "count", synthetic_reads(300, 100, 1500, 0.01, seed=2), 33, 5)
    save("loops_k21_B10_graph", "graph", loops_reads(), 21, 10)
    save("dense_k5_B4_graph", "graph", synthetic_reads(200, 60, 200, 0.02, seed=3), 5, 4)
    save("dense_k3_B1_graph", "graph", synthetic_reads(100, 40, 100, 0.02, seed=4), 3, 1)
    # Construction stage with early_tc (stages/construction.cpp:289-302): length bound = read length - k
    save("ecoli_k21_B40_tcgraph", "tcgraph", ec, 21, 40, early_tc=100 - 21)
    save("ecoli_k55_B16_tcgraph", "tcgraph", ec[:1500], 55, 16, early_tc=100 - 55)
    save("syn_k21_B10_tcgraph", "tcgraph", synthetic_reads(2000, 100, 3000, 0.02, seed=6), 21, 10, early_tc=79)
    save("loops_k21_B10_tcgraph", "tcgraph", loops_reads() + synthetic_reads(300, 120, 700, 0.02, seed=3), 21, 10, early_tc=99)
    save("dense_k7_B4_tcgraph", "tcgraph", synthetic_reads(800, 60, 400, 0.03, seed=14), 7, 4, early_tc=10)
    # RNA pipeline: EarlyATClipper (stages/construction.cpp:317-340), alone and followed by the tip clipper (:447-450)
    save("rna_k21_B8_atgraph", "atgraph", at_reads(3000, 100, 3000, 0.01, 1), 21, 8)
    save("rna_k33_B5_atgraph", "atgraph", at_reads(2000, 150, 3000, 0.02, 2), 33, 5, early_tc=150 - 33)
    save("rna_k55_B16_atgraph", "atgraph", at_reads(2000, 150, 4000, 0.01, 3), 55, 16, early_tc=150 - 55)
    save("rna_k11_B3_atgraph", "atgraph", at_reads(1500, 60, 800, 0.05, 4), 11, 3)
    # EdgeIndex refill (SURVEY 8f-1): the (k+1)-mer index of the pipeline and the counting path with a smaller K; B = 10 x 2 threads
    save("syn_k21_B20_eigraph", "eigraph", synthetic_reads(600, 100, 1500, 0.01, seed=5), 21, 20, edge_index=0)
    save("syn_k21_B20_K15_eigraph", "eigraph", synthetic_reads(600, 100, 1500, 0.01, seed=5), 21, 20, edge_index=15)
    save("loops_k21_B10_eigraph", "eigraph", loops_reads(), 21, 10, edge_index=0)
    save("ecoli_k55_B20_K33_eigraph", "eigraph", ec[:1200], 55, 20, edge_index=33)
    for nm, (rd, _) in GTEST_CASES.items():
        save("gtest_" + nm + "_k5", "graph", rd, 5, 2)
    # construction_test.cpp:97-105 (SimpleTestEarlyPairedInfo, k=3): its coverage table is the known answer in tests/test_oracle_golden.py
    save("gtest_EarlyPairedInfo_k3", "graph", ["CCCAC", "CCACG", "ACCAC", "CCACA"], 3, 2)
    # coverage pre-filter (SURVEY 8f-3), thresholds 2..5, odd and even k+1 (self-RC windows exist only for even k+1)
    save_covfilter("cov_k21_t2_covfilter", covfilter_reads(31), 21, 2)
    save_covfilter("cov_k20_t3_covfilter", covfilter_reads(32), 20, 3)
    save_covfilter("cov_k55_t2_covfilter", covfilter_reads(33), 55, 2)
    save_covfilter("cov_k31_t5_covfilter", ecoli_reads()[:1500] + covfilter_reads(34)[:800], 31, 5)
