"""CPU: the host-side read ingest (spades_b200/csrc/ingest.cpp) -- FASTA/FASTQ(.gz) parsing with kseq semantics, LongestValid,
2-bit packing, and the reference's binary read-stream format.
Checked against (1) a line-level Python model on adversarial inputs, (2) the reference's own test data set (ecoli_1K_*.fq.gz, stored
under tests/golden) parsed with Python's gzip, (3) the UNMODIFIED reference reading our .seq/.off through io::BinaryFileSingleStream
and writing the same reads through SingleReadSeq::BinWrite, and (4) the reference's parser on seeded awkward files; (3) and (4) as
oracle/_ref/ref_probe binreads and oracle/_ref/ref_fastx produced them (tests/golden/make_golden_seeded.py)."""
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

from spades_b200.packing import longest_valid, pack_reads
from spades_b200.reads_io import read_fastx, read_seqfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _model(records):
    return [s for s in (longest_valid("".join(r).upper()) for r in records) if s]


def _canonical_seqfile(path):
    raw = open(path, "rb").read()
    out = bytearray(raw[:24])
    n = int(np.frombuffer(raw[:8], np.uint64)[0])
    p = 24
    for _ in range(n):
        size = int(np.frombuffer(raw[p:p + 8], np.uint64)[0])
        nw = (size + 31) // 32
        w = np.frombuffer(raw[p + 8:p + 8 + 8 * nw], np.uint64).copy()
        if size % 32:
            w[-1] &= np.uint64((1 << (2 * (size % 32))) - 1)
        out += raw[p:p + 8] + w.tobytes() + raw[p + 8 + 8 * nw:p + 8 + 8 * nw + 12]
        p += 8 + 8 * nw + 12
    assert p == len(raw)
    return bytes(out)


def test_fastq_fasta_variants(tmp_path):
    rng = np.random.default_rng(1)
    def rnd(n, pn=0.0, lower=0.0):
        s = rng.choice(list("ACGT"), n)
        s = np.where(rng.random(n) < pn, "N", s)
        s = np.where(rng.random(n) < lower, np.char.lower(s), s)
        return "".join(s)
    seqs = [rnd(150), rnd(150, 0.02), rnd(100, 0.0, 0.5), rnd(33, 0.3), "N" * 50, "", rnd(32), rnd(64), rnd(65), rnd(1), "ACGTNNACGTACNNNACGTACGTA",
            "NACGTN", rnd(1000, 0.005)]
    seqs += [rnd(int(rng.integers(1, 300)), 0.01) for _ in range(300)]
    want = _model([[s] for s in seqs])
    # FASTQ, qualities that start with '@' / '+' / '>' (the classic ambiguity kseq resolves by length)
    fq = tmp_path / "a.fq"
    with open(fq, "w") as f:
        for i, s in enumerate(seqs):
            q = ("@+>" * (len(s) // 3 + 1))[:len(s)]
            f.write("@r%d some comment\n%s\n+\n%s\n" % (i, s, q))
    b = read_fastx(fq)
    assert b.strings() == want and b.records == len(seqs)
    assert b.dropped == sum(1 for s in seqs if not longest_valid(s.upper()))
    # the packed layout is the one pack_reads produces
    w, o, l = pack_reads(want)
    assert np.array_equal(b.words, w) and np.array_equal(b.offs, o) and np.array_equal(b.lens, l)
    # gzip, CRLF, multi-line FASTA with blank lines
    gz = tmp_path / "a.fq.gz"
    with gzip.open(gz, "wt") as f:
        f.write(open(fq).read().replace("\n", "\r\n"))
    assert read_fastx(gz).strings() == want
    fa = tmp_path / "a.fa"
    with open(fa, "w") as f:
        f.write("; leading junk that is not a record\n")
        for i, s in enumerate(seqs):
            f.write(">s%d\n" % i)
            for j in range(0, len(s), 60):
                f.write(s[j:j + 60] + "\n")
            if i % 7 == 0:
                f.write("\n")
    assert read_fastx(fa).strings() == want
    # without N handling an invalid read contributes nothing
    nolv = read_fastx(fq, longest_valid=False).strings()
    assert nolv == [s.upper() for s in seqs if s and set(s.upper()) <= set("ACGT")]
    with pytest.raises(IOError):
        read_fastx(tmp_path / "missing.fq")


def test_kseq_corner_semantics(tmp_path):
    """the vendored kseq keeps blanks inside a sequence line (they are invalid characters for LongestValid), strips one trailing CR
    per line, skips empty lines, finds the next record at the next '>' / '@' anywhere after a FASTQ record, and rejects a
    quality string of another length (ext/include/kseq/kseq.h:171-213)"""
    p = tmp_path / "c.fq"
    open(p, "wb").write(b"junk line\nmore >r0 header found mid-line\nACGT ACGTA\n\nAC\tGGGGGG\r\n+\nIIIIIIIIII\nIIIIIIIII\n"
                        b"trailing junk @r1\nacgtnacg\n+r1\nIIIIIIII\n>r2\nAAAA\nCCCC\n>r3\n>r4\nTTTT")
    b = read_fastx(p)
    # r0: "ACGT ACGTA" + "AC\tGGGGGG" -> longest valid run "GGGGGG"; r1: "ACGTNACG" -> "ACGT"; r2: "AAAACCCC"; r3: empty (dropped); r4: "TTTT"
    assert b.strings() == ["ACGTAAC", "ACGT", "AAAACCCC", "TTTT"]
    assert (b.records, b.dropped) == (5, 1)
    bad = tmp_path / "bad.fq"
    open(bad, "w").write("@r\nACGTACGT\n+\nIIIIIIIIII\n")
    with pytest.raises(IOError):
        read_fastx(bad)


def test_truncated_fastq_is_an_error(tmp_path):
    p = tmp_path / "t.fq"
    open(p, "w").write("@r\nACGTACGT\n+\nIIII")
    with pytest.raises(IOError):
        read_fastx(p)


def test_truncated_or_corrupt_gzip_is_an_error_not_a_smaller_read_set(tmp_path):
    """a .gz cut in the middle of the deflate stream (or with flipped bytes) must fail with SGPU_EIO -- zlib's gzread() <= 0 is only a
    clean end of input when gzerror() agrees (ADVICE r01)"""
    import gzip
    import random
    rnd = random.Random(5)
    fq = "".join("@r%d\n%s\n+\n%s\n" % (i, "".join(rnd.choice("ACGT") for _ in range(100)), "I" * 100) for i in range(3000))
    blob = gzip.compress(fq.encode())
    good = tmp_path / "ok.fq.gz"; good.write_bytes(blob)
    assert len(read_fastx(good)) == 3000
    cut = tmp_path / "cut.fq.gz"; cut.write_bytes(blob[: len(blob) // 2])
    with pytest.raises(IOError, match="read error|truncated|different length"):
        read_fastx(cut)
    bad = bytearray(blob)
    for i in range(len(bad) // 2, len(bad) // 2 + 64):
        bad[i] ^= 0x5A
    corrupt = tmp_path / "corrupt.fq.gz"; corrupt.write_bytes(bytes(bad))
    with pytest.raises(IOError):
        read_fastx(corrupt)


def test_ecoli_test_dataset_matches_python_gzip():
    for f in ("ecoli_1K_1.fq.gz", "ecoli_1K_2.fq.gz"):
        lines = gzip.open(os.path.join(GOLDEN, f), "rt").read().split("\n")
        want = _model([[lines[i].strip()] for i in range(1, len(lines), 4)])
        assert read_fastx(os.path.join(GOLDEN, f)).strings() == want


def test_seqfile_round_trip(tmp_path):
    rng = np.random.default_rng(2)
    reads = ["".join(rng.choice(list("ACGT"), int(n))) for n in rng.integers(1, 400, 731)]
    fa = tmp_path / "r.fa"
    open(fa, "w").write("".join(">%d\n%s\n" % (i, s) for i, s in enumerate(reads)))
    b = read_fastx(fa)
    b.write_seqfile(tmp_path / "lib")
    assert os.path.getsize(tmp_path / "lib.off") == 8 * ((len(reads) + 99) // 100)          # one offset per 100 reads
    back = read_seqfile(tmp_path / "lib")
    assert back.strings() == reads
    assert np.array_equal(back.words, b.words) and np.array_equal(back.lens, b.lens)


def seqfile_case_reads():
    rng = np.random.default_rng(3)
    return ["".join(rng.choice(list("ACGT"), int(n))) for n in rng.integers(1, 300, 457)]


def test_seqfile_format_against_the_unmodified_reference(tmp_path):
    """tests/golden/seqfile_reference.npz: what the reference read from our .seq/.off of these reads (3 portions through the .off
    index), that .off, and the .seq it wrote for the same reads itself"""
    reads = seqfile_case_reads()
    fa = tmp_path / "r.fa"
    open(fa, "w").write("".join(">%d\n%s\n" % (i, s) for i, s in enumerate(reads)))
    prefix = str(tmp_path / "lib")
    read_fastx(fa).write_seqfile(prefix)
    z = np.load(os.path.join(GOLDEN, "seqfile_reference.npz"))
    # the reference reads our files (the .off index it read is the one we write) ...
    assert open(prefix + ".off", "rb").read() == z["off"].tobytes()
    assert z["readback"].tobytes().decode().split() == reads          # guards the fixture: it holds the reads these seeds make
    # ... and writes the same bytes itself, up to the padding bits above the last base of a read: a reference Sequence of <= 60
    # bases lives inline in 16 bytes whose top byte is its metadata (sequence.hpp:194-262), and Sequence::BinWrite dumps that
    # byte along with the data; BinRead restores the metadata afterwards (:808-815), so the padding is "don't care" on input
    open(prefix + "_ref.seq", "wb").write(z["ref_seq"].tobytes())
    assert _canonical_seqfile(prefix + "_ref.seq") == _canonical_seqfile(prefix + ".seq")
    assert read_seqfile(prefix + "_ref").strings() == reads            # and we read the reference's bytes


def parser_case_files(tmp_path):
    """well-formed and deliberately awkward FASTA/FASTQ files, and the reference's own test data"""
    rng = np.random.default_rng(7)
    def rnd(n, pn=0.0, lower=0.0):
        s = rng.choice(list("ACGT"), n)
        s = np.where(rng.random(n) < pn, "N", s)
        s = np.where(rng.random(n) < lower, np.char.lower(s), s)
        return "".join(s)
    files = []
    # 1. plain FASTQ, qualities full of marker characters, some N / lowercase reads, an empty read
    seqs = [rnd(int(rng.integers(1, 250)), 0.02, 0.2) for _ in range(400)] + ["", "NNNN", "n"]
    p = tmp_path / "a.fq"
    with open(p, "w") as f:
        for i, s in enumerate(seqs):
            f.write("@r%d c\n%s\n+\n%s\n" % (i, s, ("@>+I" * (len(s) // 4 + 1))[:len(s)]))
    files.append(p)
    # 2. the same gzipped with CRLF line ends
    gz = tmp_path / "a_crlf.fq.gz"
    with gzip.open(gz, "wb") as f:
        f.write(open(p, "rb").read().replace(b"\n", b"\r\n"))
    files.append(gz)
    # 3. multi-line FASTA with blank lines, blanks inside lines, leading junk, no final newline
    fa = tmp_path / "b.fa"
    with open(fa, "w") as f:
        f.write("junk before the first record\n")
        for i, s in enumerate(seqs[:200]):
            f.write(">s%d\n" % i)
            for j in range(0, len(s), 50):
                f.write(s[j:j + 50] + ("  " if j % 100 == 0 else "") + "\n")
            if i % 5 == 0:
                f.write("\n")
        f.write(">last\nACGTTGCA")
    files.append(fa)
    # 4. multi-line FASTQ (sequence and quality wrapped), junk between records
    mq = tmp_path / "c.fq"
    with open(mq, "w") as f:
        for i, s in enumerate(seqs[:100]):
            s = s or "A"
            f.write("@m%d\n" % i + "\n".join(s[j:j + 30] for j in range(0, len(s), 30)) + "\n+m%d\n" % i)
            q = "I" * len(s)
            f.write("\n".join(q[j:j + 30] for j in range(0, len(s), 30)) + "\nnoise without markers\n")
    files.append(mq)
    # 5. the reference's own test data
    files += [os.path.join(GOLDEN, "ecoli_1K_1.fq.gz"), os.path.join(GOLDEN, "ecoli_1K_2.fq.gz")]
    return [str(f) for f in files]


def test_parser_against_the_unmodified_reference_parser(tmp_path):
    """our ingest against io::FastaFastqGzParser (the reference's vendored kseq + zlib) + io::LongestValid: the SHA-256 of the reads
    and the record count oracle/_ref/ref_fastx reported for each file (tests/golden/seeded_reference.json)"""
    want = json.load(open(os.path.join(GOLDEN, "seeded_reference.json")))["parser"]
    for f in parser_case_files(tmp_path):
        b = read_fastx(f)
        w = want[os.path.basename(f)]
        assert (hashlib.sha256("\n".join(b.strings()).encode()).hexdigest(), b.records) == (w["sha256"], w["records"]), f


def test_parser_against_reference_golden(tmp_path):
    """tests/golden/ingest_cases.npz: awkward input files and what the unmodified reference's parser + LongestValid made of them
    (generated by tests/golden/make_golden.py::save_ingest through oracle/_ref/ref_fastx)"""
    z = np.load(os.path.join(ROOT, "tests", "golden", "ingest_cases.npz"))
    names = [k[5:] for k in z.files if k.startswith("file_")]
    assert len(names) >= 4
    for name in names:
        f = tmp_path / (name + (".gz" if name.endswith("_gz") else ".txt"))
        open(f, "wb").write(z["file_" + name].tobytes())
        lines = z["parsed_" + name].tobytes().decode().split("\n")
        want = [l for l in lines if l and not l.startswith("#")]
        recs = int([l for l in lines if l.startswith("#records")][0].split()[1])
        b = read_fastx(f)
        assert b.strings() == want and b.records == recs, name


def test_parallel_parse_is_exact(tmp_path):
    """uncompressed files are parsed in parallel pieces that are only accepted where the sequential parser provably stands at the
    same place: the result must be identical to the sequential parse on four-line FASTQ (qualities full of marker characters),
    wrapped FASTQ, multi-line FASTA and on files with junk between the records"""
    rng = np.random.default_rng(21)
    def rnd(n, pn=0.01):
        s = rng.choice(list("ACGT"), n)
        return "".join(np.where(rng.random(n) < pn, "N", s))
    seqs = [rnd(int(rng.integers(50, 251))) for _ in range(12000)]
    quals = ["".join(rng.choice(list("@+>I#5"), len(s))) for s in seqs]
    files = {}
    files["four_line.fq"] = "".join("@r%d\n%s\n+\n%s\n" % (i, s, q) for i, (s, q) in enumerate(zip(seqs, quals)))
    files["wrapped.fq"] = "".join("@w%d\n%s\n+\n%s\n" % (i, "\n".join(s[j:j + 60] for j in range(0, len(s), 60)), "\n".join(q[j:j + 60] for j in range(0, len(q), 60)))
                                  for i, (s, q) in enumerate(zip(seqs, quals)))
    files["multi.fa"] = "".join(">s%d desc\n%s\n" % (i, "\n".join(s[j:j + 70] for j in range(0, len(s), 70))) for i, s in enumerate(seqs))
    files["junk.fq"] = "".join("@j%d\n%s\n+\n%s\n%s" % (i, s, q, "noise, no markers\n" if i % 3 == 0 else "") for i, (s, q) in enumerate(zip(seqs, quals)))
    for name, text in files.items():
        p = tmp_path / name
        open(p, "w").write(text)
        assert os.path.getsize(p) > (8 << 16)
        one = read_fastx(p, threads=1)
        many = read_fastx(p, threads=8)
        assert one.records == len(seqs), name
        assert many.records == one.records and many.trimmed == one.trimmed and many.dropped == one.dropped, name
        assert np.array_equal(many.words, one.words) and np.array_equal(many.offs, one.offs) and np.array_equal(many.lens, one.lens), name
        three = read_fastx(p, threads=3)
        assert np.array_equal(three.words, one.words) and np.array_equal(three.lens, one.lens), name
    # an error inside a piece is reported by the sequential parse
    bad = tmp_path / "bad.fq"
    open(bad, "w").write(files["four_line.fq"] + "@last\nACGT\n+\nII\n")
    with pytest.raises(IOError):
        read_fastx(bad, threads=8)


def _awkward_fastq(n=400, seed=9):
    import random
    rnd = random.Random(seed)
    recs = []
    for i in range(n):
        L = rnd.choice([0, 1, 31, 32, 33, 64, 100, 150, 151, 300])
        seq = "".join(rnd.choice("ACGTacgtNn.") if rnd.random() < 0.1 else rnd.choice("ACGT") for _ in range(L))
        recs.append((seq, "".join(chr(33 + rnd.randrange(40)) for _ in range(L))))
    return recs


def test_text_index_of_strict_fastx_and_refusal_of_everything_else(tmp_path):
    """host half of the GPU packer (sgpu_text_index_fastx): sequence ranges of strict 4-line FASTQ / 2-line FASTA (also with CRLF and
    without a final newline) equal what the general parser sees; multi-line records, junk and truncated records are refused"""
    from spades_b200.reads_io import index_text
    recs = _awkward_fastq()
    fq = "".join("@r%d x\n%s\n+\n%s\n" % (i, s, q) for i, (s, q) in enumerate(recs))
    fa = "".join(">s%d\n%s\n" % (i, s) for i, (s, q) in enumerate(recs))
    for text in (fq, fq.replace("\n", "\r\n"), fq[:-1], fa, fa[:-1]):
        data = text.encode()
        off, ln = index_text(data)
        assert [data[int(o):int(o) + int(l)].decode() for o, l in zip(off, ln)] == [s for s, _ in recs]
    f = tmp_path / "x.fq"; f.write_text(fq)
    want = [longest_valid(s) for s, _ in recs]
    assert read_fastx(f).strings() == [w.upper() for w in want if w]
    assert index_text(b"@r\nACGT\nACGT\n+\nIIIIIIII\n") is None            # multi-line sequence
    assert index_text(b"junk\n@r\nACGT\n+\nIIII\n") is None
    assert index_text(b"@r\nACGT\n+\nIII\n") is None                        # quality of another length
    assert index_text(b"@r\nACGT\n+\n") is None                              # truncated
    assert index_text(b"")[0].size == 0


@pytest.mark.gpu
def test_gpu_packer_matches_host_ingest():
    """sgpu_reads_pack_text (LongestValid + 2-bit packing in CUDA kernels) against the host ingest on the same awkward FASTQ: identical
    words / lengths for every read with a valid base, and identical k-mers downstream"""
    import tempfile
    from gpu_util import ctx
    from spades_b200.kmer_index import KMerDiskCounter, ParallelSortingSplitter
    from spades_b200.reads_io import download_reads, pack_text_on_gpu
    recs = _awkward_fastq(3000, seed=10)
    fq = "".join("@r%d\n%s\n+\n%s\n" % (i, s, q) for i, (s, q) in enumerate(recs)).encode()
    c = ctx()
    for lv in (True, False):
        n = pack_text_on_gpu(c, fq, longest_valid=lv)
        assert n == len(recs)
        words, offs, lens = download_reads(c)
        want = [longest_valid(s) if lv else (s if all(ch in "ACGTacgt" for ch in s) else "") for s, _ in recs]
        assert [int(x) for x in lens] == [len(w) for w in want]
        hw, ho, hl = pack_reads([w.upper() for w in want if w])
        got = np.concatenate([words[int(o):int(o) + (int(l) + 31) // 32] for o, l in zip(offs, lens) if l]) if len(hw) else np.zeros(0, np.uint64)
        assert np.array_equal(got, hw)
        st = KMerDiskCounter(c, ParallelSortingSplitter(21)).Count(7)
        k_gpu = st.kmers(); st.free()
        c.set_reads(hw, ho, hl)
        st = KMerDiskCounter(c, ParallelSortingSplitter(21)).Count(7)
        assert np.array_equal(k_gpu, st.kmers()); st.free()
