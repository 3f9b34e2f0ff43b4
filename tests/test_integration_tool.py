"""The reference-side adapters of INTEGRATION.md as real code: integration/gpu_kmer_counter.hpp compiled against the UNMODIFIED
reference headers into a spades-kmercount-compatible tool (integration/spades_kmercount_gpu.cpp) that links libspades_b200.so.
The binaries are built under oracle/_ref/integration where the reference sources are available, like the rest of oracle/_ref.

CPU: it exists, and without a GPU it refuses loudly (no CPU fallback).
GPU: reference C++ host code -> C ABI -> CUDA: final_kmers byte-identical to the reference's spades-kmercount golden output, the
     reference's own KMerIndexBuilder accepts the GPU-written bucket files, and the GPU-built MPHF loaded through the reference's
     own KMerIndex::deserialize agrees with it on every k-mer (the tool's exit code)."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import golden_util as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILT = os.path.join(ROOT, "oracle", "_ref", "integration")
PROBE = os.path.join(ROOT, "oracle", "_ref", "ref_probe")
TOOL = os.path.join(BUILT, "spades_kmercount_gpu")
GBUILDER = os.path.join(BUILT, "spades_gbuilder_gpu")
needs_tool = pytest.mark.skipif(not os.path.exists(TOOL), reason="oracle/_ref/integration/spades_kmercount_gpu not built (make -C integration; needs the reference sources)")


@needs_tool
def test_tool_refuses_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with tempfile.TemporaryDirectory() as d:
        rf = os.path.join(d, "r.txt")
        open(rf, "w").write("ACGTACGTACGTAGCTAGCTAGCTAGCATCGATCGATCAGCTAGC\n")
        p = subprocess.run([TOOL, rf, "21", os.path.join(d, "w")], capture_output=True, text=True)
    assert p.returncode == 3 and "no CPU fallback" in p.stderr


def test_adapter_is_built_where_the_reference_is():
    if os.path.exists(PROBE):
        assert os.path.exists(TOOL), "run __graft_entry__.build()"


def test_construction_phase_subclass_compiles_against_the_reference():
    """integration/construction_gpu_phase.cpp (KMerCountingGpu : Construction::Phase, the pipeline seam) is compiled against the
    UNMODIFIED reference wherever the reference exists; the object must define the phase's run()"""
    obj = os.path.join(BUILT, "construction_gpu_phase.o")
    if not os.path.exists(PROBE) and not os.path.exists(obj):
        pytest.skip("needs the reference sources to build (oracle/_ref)")
    assert os.path.exists(obj), "run __graft_entry__.build()"
    syms = subprocess.run(["nm", "-C", obj], capture_output=True, text=True).stdout
    assert "KMerCountingGpu::run" in syms and "CoverageFilterGpu::run" in syms and "GpuKMerDiskCounterT<" in syms


@needs_tool
@pytest.mark.gpu
@pytest.mark.parametrize("name", G.names("count"))
def test_reference_host_code_over_the_c_abi(name):
    g = G.load(name)
    with tempfile.TemporaryDirectory() as d:
        rf = os.path.join(d, "reads.txt")
        open(rf, "w").write("\n".join(g["reads"]) + "\n")
        w = os.path.join(d, "w")
        p = subprocess.run([TOOL, rf, str(g["k"]), w, str(g["B"])], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
        fk = np.fromfile(os.path.join(w, "final_kmers"), np.uint8)
    assert np.array_equal(fk, g["final_kmers"])
    assert "reference-built and GPU-built KMerIndex agree" in p.stdout
    assert "reference KMerDiskCounter over GpuKMerSplitter: identical final_kmers" in p.stdout        # the KMerSplitter-level seam
    assert "MTS client (k-mer file -> canonical set, 16 buckets): GPU counter == reference" in p.stdout   # SURVEY 8f-4 clients
    if g["k"] == 21:
        assert "hammer::KMer client (Seq<21>): GPU counter == reference KMerDiskCounter<Seq<21>>" in p.stdout


@needs_tool
@pytest.mark.gpu
def test_tool_takes_gzipped_fastq_like_the_original():
    """same reads as a gzipped FASTQ with N-containing reads added: the library's ingest (kseq semantics + LongestValid) in front of
    the same adapter; the N reads are cut to their longest valid run, which here is shorter than k and so contributes nothing"""
    import gzip
    g = G.load("ecoli_k21_B16_count")
    with tempfile.TemporaryDirectory() as d:
        fq = os.path.join(d, "reads.fq.gz")
        with gzip.open(fq, "wt") as f:
            for i, r in enumerate(g["reads"]):
                f.write("@r%d\n%s\n+\n%s\n" % (i, r, "I" * len(r)))
            f.write("@n1\nACGTACGTNNNNACGTACGTACNNNN\n+\nIIIIIIIIIIIIIIIIIIIIIIIIII\n")
        w = os.path.join(d, "w")
        p = subprocess.run([TOOL, fq, str(g["k"]), w, str(g["B"])], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
        fk = np.fromfile(os.path.join(w, "final_kmers"), np.uint8)
    assert np.array_equal(fk, g["final_kmers"])


@pytest.mark.skipif(not os.path.exists(GBUILDER), reason="oracle/_ref/integration/spades_gbuilder_gpu not built")
def test_gbuilder_tool_refuses_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with tempfile.TemporaryDirectory() as d:
        rf = os.path.join(d, "r.txt")
        open(rf, "w").write("ACGTACGTACGTAGCTAGCTAGCTAGCATCGATCGATCAGCTAGC\n")
        p = subprocess.run([GBUILDER, rf, "21", os.path.join(d, "w")], capture_output=True, text=True)
    assert p.returncode == 3 and "no CPU fallback" in p.stderr


@pytest.mark.skipif(not os.path.exists(GBUILDER), reason="oracle/_ref/integration/spades_gbuilder_gpu not built")
@pytest.mark.gpu
@pytest.mark.parametrize("name,early_tc", [("ecoli_k21_B40_graph", 0), ("loops_k21_B10_graph", 0), ("ecoli_k55_B16_graph", 0), ("syn_k21_B10_tcgraph", 79)])
def test_reference_graph_construction_over_gpu_arrays(name, early_tc):
    """spades-gbuilder's flow with the hot path on the GPU and the UNMODIFIED reference doing everything downstream on the GPU's
    arrays (its own KMerIndexBuilder over the GPU-written buckets, UnbranchingPathExtractor over the GPU's masks, graph
    constructor, coverage filler, GFA writer): the tool exits 0 iff the reference reproduces the GPU's unitigs and GFA, and the GFA
    must also be the golden one (the reference end to end on the CPU)."""
    g = G.load(name)
    with tempfile.TemporaryDirectory() as d:
        rf = os.path.join(d, "reads.txt")
        open(rf, "w").write("\n".join(g["reads"]) + "\n")
        w = os.path.join(d, "w")
        p = subprocess.run([GBUILDER, rf, str(g["k"]), w, str(g["B"]), str(early_tc)], capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-2000:]
        gfa = open(os.path.join(w, "graph.gfa")).read()
    assert gfa == g["graph_gfa"].tobytes().decode()
