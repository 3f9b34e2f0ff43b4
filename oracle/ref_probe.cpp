// oracle/ref_probe.cpp -- TEST INFRASTRUCTURE ONLY (never linked into the product).
//
// A thin driver (our code) over the UNMODIFIED reference headers under /root/reference:
// it runs the reference's own KMerDiskCounter / DeBruijnExtensionIndexBuilder /
// UnbranchingPathExtractor / FastGraphFromSequencesConstructor / CoverageHashMapBuilder /
// GFAWriter on a plain-text read file and dumps every intermediate artefact so that
// oracle/*.c (the CPU restatement) and the CUDA path can be compared byte for byte.
//
// Mirrors what spades-kmercount (projects/spades_tools/kmercount.cpp:48-122,191-230) and
// spades-gbuilder (projects/spades_tools/gbuilder.cpp:157-225) do, minus their CLI / YAML /
// binary-read-conversion front ends (reads here come from an in-memory VectorReadStream
// wrapped in RCWrap, the same fixture the reference's own construction_test uses,
// test/debruijn/test_utils.cpp:128-138).
//
// usage: ref_probe <mode: count|graph|bench> <reads.txt> <k> <num_buckets> <nthreads> <outdir>   (env PROBE_EARLY_TC=<bound>: graph mode
//        also runs EarlyTipClipperProcessor before the unitig extraction; PROBE_QUERIES=<file>: graph mode also answers index
//        lookups, see below)
//   reads.txt: one ACGT read per line (N-trimming is the ingest layer's job)
#include "io/reads/vector_reader.hpp"
#include "io/reads/rc_reader_wrapper.hpp"
#include "io/reads/read_stream_vector.hpp"
#include "io/reads/single_read.hpp"
#include "io/reads/binary_streams.hpp"
#include "io/reads/coverage_filtering_read_wrapper.hpp"
#include "kmer_index/kmer_counting.hpp"
#include "kmer_index/ph_map/kmer_maps.hpp"
#include "kmer_index/kmer_mph/kmer_index_builder.hpp"
#include "kmer_index/kmer_mph/kmer_splitters.hpp"
#include "kmer_index/ph_map/coverage_hash_map_builder.hpp"
#include "kmer_index/extension_index/kmer_extension_index.hpp"
#include "kmer_index/extension_index/kmer_extension_index_builder.hpp"
#include "assembly_graph/core/graph.hpp"
#include "assembly_graph/construction/debruijn_graph_constructor.hpp"
#include "assembly_graph/construction/early_simplification.hpp"
#include "assembly_graph/graph_support/coverage_filling.hpp"
#include "assembly_graph/index/edge_index_builders.hpp"
#include "io/graph/gfa_writer.hpp"
#include "utils/logger/log_writers.hpp"
#include "utils/filesystem/temporary.hpp"

#include <fstream>
#include <sstream>
#include <string>
#include <vector>
#include <omp.h>

using namespace debruijn_graph;

static void create_console_logger() {
    using namespace logging;
    logger *lg = create_logger("");
    lg->add_writer(std::make_shared<console_writer>());
    attach_logger(lg);
}

static void probe_copy(const std::filesystem::path &from, const std::filesystem::path &to) {
    std::filesystem::copy_file(from, to, std::filesystem::copy_options::overwrite_existing);
}

// all windows of reads + RC, no filter: the splitter of kmercount.cpp:48-122 restated over
// an in-memory vector (the original parses files through ReadProcessor).
class AllWindowsSplitter : public kmers::KMerSortingSplitter<RtSeq> {
    const std::vector<Sequence> &reads_;
  public:
    AllWindowsSplitter(fs::TmpDir dir, unsigned K, const std::vector<Sequence> &reads)
            : kmers::KMerSortingSplitter<RtSeq>(dir, K), reads_(reads) {}
    RawKMers Split(size_t num_files, unsigned nthreads) override {
        auto out = PrepareBuffers(num_files, 1, 0);
        for (const auto &fw : reads_) {
            for (int rc = 0; rc < 2; ++rc) {
                Sequence seq = rc ? !fw : fw;
                if (seq.size() < this->K_) continue;
                RtSeq kmer = seq.start<RtSeq>(this->K_) >> 'A';
                bool stop = false;
                for (size_t j = this->K_ - 1; j < seq.size(); ++j) {
                    kmer <<= seq[j];
                    stop |= push_back_internal(kmer, 0);
                }
                if (stop) DumpBuffers(out);
            }
        }
        DumpBuffers(out);
        ClearBuffers();
        (void)nthreads;
        return out;
    }
};

template<class Index>
static void dump_index(const Index &idx, const std::filesystem::path &p) {
    std::ofstream os(p, std::ios::binary);
    idx.BinWrite(os);   // u32 k, then KMerIndex::serialize (kmer_index.hpp:102-108)
}

// KMerIndex::seq_idx (kmer_index.hpp:88-93) of raw records read from `qpath` (ceil(K/32) u64 words each, the stored form) under the
// index an IndexWrapper holds; one u64 per record to `out` (-1 = NOT_FOUND). The wrapper keeps its KMerIndex protected
// (perfect_hash_map.hpp:32-34), so a derived accessor reaches it through a member pointer.
using SlimIndex = kmers::IndexWrapper<RtSeq, kmers::slim_kmer_index_traits<RtSeq>>;
struct SlimIndexPeek : SlimIndex {
    static const KMerIndexT &of(const SlimIndex &w) { return *(w.*(&SlimIndexPeek::index_ptr_)); }
};
static void dump_queries(const SlimIndex &idx, unsigned K, const std::string &qpath, const std::filesystem::path &out) {
    const size_t nw = RtSeq::GetDataSize(K);
    std::ifstream is(qpath, std::ios::binary);
    std::vector<uint64_t> rec(nw);
    std::ofstream os(out, std::ios::binary);
    const auto &index = SlimIndexPeek::of(idx);
    while (is.read((char *)rec.data(), (std::streamsize)(nw * 8))) {
        const uint64_t v = index.seq_idx(RtSeq(K, rec.data()));
        os.write((const char *)&v, 8);
    }
}

int main(int argc, char **argv) {
    if (argc < 7) { fprintf(stderr, "usage: %s count|graph reads.txt k B T outdir\n", argv[0]); return 2; }
    std::string mode = argv[1];
    std::string reads_path = argv[2];
    unsigned k = atoi(argv[3]);
    unsigned B = atoi(argv[4]);
    unsigned T = atoi(argv[5]);
    std::filesystem::path outdir = argv[6];
    std::filesystem::create_directories(outdir);
    create_console_logger();
    omp_set_num_threads(T);

    std::vector<Sequence> seqs;
    {
        std::ifstream is(reads_path);
        std::string line;
        while (std::getline(is, line)) {
            if (line.empty()) continue;
            seqs.emplace_back(line);
        }
    }
    std::filesystem::create_directories(outdir / "tmp");
    auto workdir = fs::tmp::make_temp_dir(outdir / "tmp", "probe");

    if (mode == "binreads") {
        // format pin for the binary read streams (SURVEY a2/a3): argv[7] = prefix. (1) <prefix>_ref.seq = ReadStreamStat header +
        // every read of reads.txt through the reference's own SingleReadSeq::BinWrite (what BinaryWriter::ToBinary emits per read,
        // binary_converter.cpp:96-110); (2) <prefix>.seq/.off -- written by OUR library -- read back through the reference's own
        // io::BinaryFileStream in T portions (uses the .off index) and dumped as text.
        std::string prefix = argc > 7 ? argv[7] : argv[6];
        {
            std::ofstream os(prefix + "_ref.seq", std::ios::binary);
            io::ReadStreamStat stat;
            for (const auto &s : seqs) { stat.read_count++; stat.max_len = std::max(stat.max_len, s.size()); stat.total_len += s.size(); }
            stat.write(os);
            for (const auto &s : seqs) io::SingleReadSeq(s).BinWrite(os);
        }
        std::ofstream txt(prefix + "_readback.txt");
        for (unsigned t = 0; t < T; ++t) {
            io::BinaryFileSingleStream st(prefix, T, t);
            st.reset();
            io::SingleReadSeq r;
            while (!st.eof()) { st >> r; txt << r.sequence().str() << "\n"; }
        }
        return 0;
    }

    if (mode == "count") {
        kmers::KMerDiskCounter<RtSeq> counter(workdir, AllWindowsSplitter(workdir, k, seqs));
        auto storage = counter.Count(B, T);
        {
            std::ofstream sz(outdir / "bucket_sizes.txt");
            for (unsigned i = 0; i < B; ++i) sz << storage.bucket_size(i) << "\n";
        }
        storage.merge();
        probe_copy(storage.final_kmers()->file(), outdir / "final_kmers");
        return 0;
    }

    // graph mode
    typedef io::SingleReadSeq Read;
    typedef io::VectorReadStream<Read> RawStream;
    io::ReadStreamList<Read> streams;
    {
        size_t n = seqs.size(), per = (n + T - 1) / T;
        for (unsigned t = 0; t < T; ++t) {
            std::vector<Read> chunk;
            for (size_t i = t * per; i < std::min(n, (t + 1) * per); ++i) chunk.emplace_back(seqs[i]);
            streams.push_back(io::RCWrap<Read>(RawStream(chunk)));
        }
    }

    if (mode == "covfilter") {
        // SURVEY 8f-3, the pipeline's CoverageFilter phase (stages/construction.cpp:167-198) on the reads + RC streams above:
        // HLL upper bound of the distinct (k+1)-mers -> qf::cqf sized from it -> counts up to the threshold -> reads whose median
        // (k+1)-mer multiplicity reaches the threshold survive (io/reads/coverage_filtering_read_wrapper.hpp). PROBE_COV_THR = threshold.
        // covfilter.txt: "<cardinality upper bound> <hash bits> <range mask> <distinct fingerprints>"; keep.txt: one 0/1 per input read;
        // hashes.bin: the SymmetricCyclicHash of every (k+1)-window of the first 64 reads (u64 each, read by read).
        const unsigned thr = getenv("PROBE_COV_THR") ? (unsigned)atoi(getenv("PROBE_COV_THR")) : 2u;
        const unsigned kp1 = k + 1;
        rolling_hash::SymmetricCyclicHash<rolling_hash::NDNASeqHash> hasher(kp1);
        using KmerFilter = kmers::StoringTypeFilter<kmers::InvertableStoring>;
        const size_t card = kmers::EstimateCardinalityUpperBound(kp1, streams, hasher, KmerFilter());
        qf::cqf cqf(card);
        kmers::FillCoverageHistogram(cqf, kp1, hasher, streams, thr, KmerFilter());
        {
            std::ofstream os(outdir / "covfilter.txt");
            os << card << " " << cqf.hash_bits() << " " << cqf.range_mask() << " " << cqf.distinct() << "\n";
        }
        io::CoverageFilter<Read, decltype(hasher)> filter(kp1, hasher, cqf, thr);
        {
            std::ofstream os(outdir / "keep.txt");
            for (const auto &s : seqs) os << (filter(Read(s)) ? 1 : 0) << "\n";
        }
        {
            std::ofstream os(outdir / "hashes.bin", std::ios::binary);
            for (size_t i = 0; i < seqs.size() && i < 64; ++i) {
                const Sequence &s = seqs[i];
                if (s.size() < kp1) continue;
                RtSeq kmer = s.start<RtSeq>(kp1) >> 'A';
                auto hash = hasher.hash(kmer);
                for (size_t j = kp1 - 1; j < s.size(); ++j) {
                    hash = hasher.hash_update(hash, (rolling_hash::chartype)kmer[0], (rolling_hash::chartype)s[j]);
                    kmer <<= s[j];
                    const uint64_t v = (uint64_t)hash;
                    os.write((const char *)&v, 8);
                }
            }
        }
        return 0;
    }

    using Splitter = kmers::DeBruijnReadKMerSplitter<Read, kmers::StoringTypeFilter<kmers::InvertableStoring>>;
    if (mode == "bench") {
        // timed region == the GPU bench step: extract + count the (k+1)-mers (KMerDiskCounter::Count) and index them
        // (KMerIndexBuilder::BuildIndex over the storage, as CoverageHashMapBuilder does, coverage_hash_map_builder.hpp:46).
        // Input parsing / packing above is outside the region, like "reads resident" on the GPU side.
        int reps = argc > 7 ? atoi(argv[7]) : 1;
        for (int rep = 0; rep < reps; ++rep) {
            auto wd = fs::tmp::make_temp_dir(outdir / "tmp", "bench");
            streams.reset();
            double t0 = omp_get_wtime();
            kmers::KMerDiskCounter<RtSeq> counter(wd, Splitter(wd, k + 1, streams, 0));
            auto kpomers = counter.Count(B, T);
            double t1 = omp_get_wtime();
            using CoverageMap = kmers::PerfectHashMap<RtSeq, uint32_t, kmers::slim_kmer_index_traits<RtSeq>, kmers::DefaultStoring>;
            CoverageMap cm(k + 1);
            kmers::PerfectHashMapBuilder().BuildIndex(cm, kpomers, T);
            double t2 = omp_get_wtime();
            size_t windows = 0;
            for (const auto &s : seqs) if (s.size() >= k + 1) windows += s.size() - k;
            printf("BENCH {\"rep\": %d, \"count_s\": %.6f, \"index_s\": %.6f, \"total_s\": %.6f, \"windows\": %zu, \"distinct\": %zu, \"threads\": %u, \"buckets\": %u}\n",
                   rep, t1 - t0, t2 - t1, t2 - t0, windows, kpomers.total_kmers(), T, B);
            fflush(stdout);
        }
        return 0;
    }
    kmers::KMerDiskCounter<RtSeq> counter(workdir, Splitter(workdir, k + 1, streams, 0));
    auto kpomers = counter.Count(B, T);
    {
        std::ofstream sz(outdir / "kpomer_bucket_sizes.txt");
        std::ofstream all(outdir / "kpomers", std::ios::binary);
        for (unsigned i = 0; i < B; ++i) {
            sz << kpomers.bucket_size(i) << "\n";
            if (!kpomers.bucket_size(i)) continue;        // inserting an empty streambuf sets failbit and drops all later buckets
            std::ifstream in(kpomers.bucket_file(i)->file(), std::ios::binary);
            all << in.rdbuf();
        }
    }

    kmers::DeBruijnExtensionIndex<> ext(k);
    kmers::DeBruijnExtensionIndexBuilder().BuildExtensionIndexFromKPOMers(workdir, ext, kpomers, T);
    {
        // final_kmers of the k-mer index, in index iteration order
        std::ofstream os(outdir / "kmers", std::ios::binary);
        size_t W = RtSeq::GetDataSize(k) * sizeof(RtSeq::DataType);
        auto its = ext.kmer_begin(1);
        for (auto &it = its[0]; it.good(); ++it) os.write((const char *)*it, W);
        dump_index(static_cast<const kmers::IndexWrapper<RtSeq, kmers::slim_kmer_index_traits<RtSeq>>&>(ext), outdir / "kmer_index.bin");
        std::ofstream ms(outdir / "masks.bin", std::ios::binary);
        ms.write(ext.raw_data(), ext.raw_size());
    }

    // PROBE_EARLY_AT=1: the RNA pipeline's early low-complexity clipper (stages/construction.cpp:317-340: at_ratio 0.8, min 10, max 200)
    // between the mask fill and everything downstream; masks_at.bin = the array after it, at_removed.txt = the two return values
    if (getenv("PROBE_EARLY_AT")) {
        EarlyLowComplexityClipperProcessor at(ext, 0.8, 10, 200);
        size_t e = at.RemoveATEdges();
        size_t t = at.RemoveATTips();
        std::ofstream ms(outdir / "masks_at.bin", std::ios::binary);
        ms.write(ext.raw_data(), ext.raw_size());
        std::ofstream rs(outdir / "at_removed.txt");
        rs << e << "\n" << t << "\n";
    }

    // PROBE_EARLY_TC=<length bound>: the pipeline's early tip clipper (stages/construction.cpp:289-302) between the mask
    // fill and the unitig extraction; masks.bin above is the array before, masks_tc.bin the array after
    if (const char *tc = getenv("PROBE_EARLY_TC")) {
        size_t bound = (size_t)atoll(tc);
        size_t removed = EarlyTipClipperProcessor(ext, bound).ClipTips();
        std::ofstream ms(outdir / "masks_tc.bin", std::ios::binary);
        ms.write(ext.raw_data(), ext.raw_size());
        std::ofstream rs(outdir / "tc_removed.txt");
        rs << removed << "\n";
    }

    unsigned nchunks = 16 * omp_get_max_threads();
    std::vector<Sequence> edges = UnbranchingPathExtractor(ext, k).ExtractUnbranchingPathsAndLoops(nchunks);
    {
        std::ofstream os(outdir / "unitigs.txt");
        for (const auto &e : edges) os << e.str() << "\n";
    }

    DeBruijnGraph g(k);
    FastGraphFromSequencesConstructor<DeBruijnGraph>(k, ext).ConstructGraph(g, edges);

    using CoverageMap = kmers::PerfectHashMap<RtSeq, uint32_t, kmers::slim_kmer_index_traits<RtSeq>, kmers::DefaultStoring>;
    CoverageMap coverage_map(k + 1);
    omnigraph::FlankingCoverage<DeBruijnGraph> flanking_cov(g, 50);
    kmers::CoverageHashMapBuilder().BuildIndex(coverage_map, kpomers, streams);
    {
        std::ofstream cs(outdir / "coverage.bin", std::ios::binary);
        for (auto I = coverage_map.value_cbegin(), E = coverage_map.value_cend(); I != E; ++I) {
            uint32_t v = *I; cs.write((const char *)&v, 4);
        }
        dump_index(static_cast<const kmers::IndexWrapper<RtSeq, kmers::slim_kmer_index_traits<RtSeq>>&>(coverage_map), outdir / "kpomer_index.bin");
        // histogram exactly as stages/construction.cpp:404-418
        std::vector<size_t> hist; size_t maxcov = 0;
        for (auto I = coverage_map.value_cbegin(), E = coverage_map.value_cend(); I != E; ++I) {
            size_t ccov = *I;
            if (!ccov) continue;
            maxcov = std::max(ccov, maxcov);
            if (maxcov > hist.size()) hist.resize(maxcov, 0);
            hist[ccov - 1] += 2;
        }
        std::ofstream hs(outdir / "histogram.txt");
        for (size_t v : hist) hs << v << "\n";
    }
    // PROBE_QUERIES=<file>: seq_idx of every record of <file> under the k-mer index (kmer_queries_idx.bin) and of every record of
    // <file>.kp1 under the (k+1)-mer index (kpomer_queries_idx.bin). Both indices are the ones KMerIndexBuilder::BuildIndex built in
    // memory above: a deserialized index marks empty buckets as built (BooPHF.h:537-577) and answers absent keys differently.
    if (const char *q = getenv("PROBE_QUERIES")) {
        dump_queries(ext, k, q, outdir / "kmer_queries_idx.bin");
        dump_queries(coverage_map, k + 1, std::string(q) + ".kp1", outdir / "kpomer_queries_idx.bin");
    }
    // PROBE_EDGE_INDEX=<kk> (0 = k+1): the EdgeIndex refill of the pipeline (modules/graph_construction.hpp:74-82, alignment/edge_index.hpp:
    // Refill -> GraphPositionFillingIndexBuilder, assembly_graph/index/edge_index_builders.hpp:274-307). kk == k+1 takes the (k+1)-mers
    // straight from the edges (one MPHF, no counting); any other kk goes through DeBruijnGraphKMerSplitter + KMerDiskCounter with B buckets.
    // edge_index.bin = KMerIndex::serialize; edge_index_values.bin = per slot { u64 edge id, u32 offset } (EdgeInfo, edge_position_index.hpp)
    if (const char *ei = getenv("PROBE_EDGE_INDEX")) {
        const unsigned kk = atoi(ei) ? (unsigned)atoi(ei) : k + 1;
        using Index = KmerFreeEdgeIndex<DeBruijnGraph>;
        Index index(g, kk);
        omp_set_num_threads(kk == k + 1 ? T : (int)std::max(1u, B / 10));      // the counting path uses 10 x omp_get_max_threads() buckets
        if (kk == k + 1) GraphPositionFillingIndexBuilder<Index>().BuildIndexFromGraph(index, g);
        else GraphPositionFillingIndexBuilder<Index>().BuildIndexFromGraph(index, g, fs::tmp::make_temp_dir(outdir / "tmp", "edge_index"));
        omp_set_num_threads(T);
        dump_index(static_cast<const kmers::IndexWrapper<RtSeq, kmers::kmer_index_traits<RtSeq>>&>(index), outdir / "edge_index.bin");
        std::ofstream vs(outdir / "edge_index_values.bin", std::ios::binary);
        for (auto I = index.value_cbegin(), E = index.value_cend(); I != E; ++I) {
            const uint64_t id = I->valid() ? (uint64_t)I->edge().int_id() : (I->removed() ? ~1ull : ~0ull);
            const uint32_t off = I->offset();
            vs.write((const char *)&id, 8); vs.write((const char *)&off, 4);
        }
        std::ofstream es(outdir / "edge_ids.txt");      // edge ids in graph iteration order with their sequences: the id <-> unitig mapping
        for (EdgeId e : g.edges()) es << e.int_id() << " " << g.EdgeNucls(e).str() << "\n";
    }
    FillCoverageAndFlankingFromPHM(coverage_map, g, flanking_cov);
    {
        std::ofstream f(outdir / "graph.gfa");
        gfa::GFAWriter w(g, f);
        w.WriteSegmentsAndLinks();
    }
    return 0;
}

// The reference's LLVM time-trace hooks (utils/perf/timetracer.hpp:9-42) live in the vendored LLVM
// support library (ext/src/llvm, ~60 files + cmake-generated config). They are profiling no-ops
// when the profiler was never initialised (the standalone tools never initialise it), so the probe
// supplies the three entry points as no-ops instead of building that library.
namespace llvm {
TimeTraceProfiler *getTimeTraceProfilerInstance() { return nullptr; }
void timeTraceProfilerBegin(StringRef, StringRef) {}
void timeTraceProfilerEnd() {}
}
