/*
 * spades_b200.h -- C ABI of libspades_b200.so: the B200-native k-mer counting / de Bruijn construction path.
 *
 * Plain pointers and sizes only; every function returns 0 on success or a positive error code (never exits,
 * never throws); sgpu_last_error() gives the message. One sgpu_ctx per process per GPU, used from one host
 * thread at a time (the reference calls this path from a single thread too, SURVEY 8b).
 *
 * Each entry point replaces one piece of the reference (paths relative to the SPAdes source tree):
 *
 *   sgpu_reads_*            io/reads binary read records: Sequence::BinRead (common/sequence/sequence.hpp:808-830),
 *                           SingleReadSeq (common/io/reads/single_read.hpp:307-323) -- 2-bit packed reads
 *   sgpu_count              kmers::KMerDiskCounter<RtSeq>::Count over a DeBruijnReadKMerSplitter<..., StoringTypeFilter<
 *                           InvertableStoring>> (SGPU_CANONICAL; common/kmer_index/kmer_mph/kmer_index_builder.hpp:306-332,
 *                           kmer_splitters.hpp:112-136) or over spades-kmercount's ParallelSortingSplitter (SGPU_ALL_WINDOWS;
 *                           projects/spades_tools/kmercount.cpp:48-122,219-220)
 *   sgpu_kmers_from_kpomers KMerDiskCounter::Count over DeBruijnKMerKMerSplitter (kmer_splitters.hpp:138-207), as called by
 *                           DeBruijnExtensionIndexBuilder::BuildExtensionIndexFromKPOMers (extension_index/
 *                           kmer_extension_index_builder.hpp:83-96)
 *   sgpu_kset_*             kmers::KMerDiskStorage<RtSeq> (kmer_index_builder.hpp:47-256): bucket_size, bucket files, merge()
 *   sgpu_mphf_build         kmers::KMerIndexBuilder<Index>::BuildIndex(index, storage) (kmer_index_builder.hpp:448-498)
 *   sgpu_mphf_serialize     kmers::KMerIndex::serialize (kmer_mph/kmer_index.hpp:102-108), byte compatible
 *   sgpu_mphf_lookup        kmers::KMerIndex::seq_idx (kmer_index.hpp:88-93)
 *   sgpu_graph_build        FillExtensionsFromIndex (kmer_extension_index_builder.hpp:45-60,102-105) +
 *                           UnbranchingPathExtractor::ExtractUnbranchingPathsAndLoops (assembly_graph/construction/
 *                           debruijn_graph_constructor.hpp:399-406) + CoverageHashMapBuilder::BuildIndex
 *                           (ph_map/coverage_hash_map_builder.hpp:42-56) + FillCoverageAndFlankingFromPHM (raw coverage part,
 *                           assembly_graph/graph_support/coverage_filling.hpp:90-96)
 *   sgpu_graph_build_ex     the same preceded by EarlyTipClipperProcessor::ClipTips (assembly_graph/construction/
 *                           early_simplification.hpp:38-162; stages/construction.cpp:289-302)
 *   sgpu_graph_build_opts   the same preceded, optionally, by EarlyLowComplexityClipperProcessor::RemoveATEdges / RemoveATTips
 *                           (early_simplification.hpp:164-347; EarlyATClipper of the RNA pipeline, stages/construction.cpp:317-340)
 *   sgpu_graph_masks        DeBruijnExtensionIndex::raw_data() (extension_index/kmer_extension_index.hpp:83-84)
 *   sgpu_graph_coverage     PerfectHashMap<RtSeq,uint32_t>::values() of the coverage map (stages/construction.cpp:371-395)
 *   sgpu_graph_histogram    the multiplicity histogram of PHMCoverageFiller (stages/construction.cpp:404-418)
 *   sgpu_graph_unitig*      std::vector<Sequence> returned by ExtractUnbranchingPathsAndLoops
 *   sgpu_edge_index_*       EdgeIndex<Graph>::Refill (alignment/edge_index.hpp:88-110; assembly_graph/index/edge_index_builders.hpp:154-307,
 *                           edge_info_updater.hpp:38-101)
 *   sgpu_graph_gfa          FastGraphFromSequencesConstructor::ConstructGraph (debruijn_graph_constructor.hpp:506-567) +
 *                           gfa::GFAWriter::WriteSegmentsAndLinks (io/graph/gfa_writer.cpp:36-116)
 */
#ifndef SPADES_B200_H_
#define SPADES_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sgpu_ctx sgpu_ctx;
typedef struct sgpu_kset sgpu_kset;     /* a counted k-mer set resident in HBM (== KMerDiskStorage contents) */
typedef struct sgpu_mphf sgpu_mphf;     /* a boomphf-compatible KMerIndex resident in HBM */
typedef struct sgpu_graph sgpu_graph;   /* masks + coverage + unitigs + link records */

typedef struct sgpu_config {
    int device;                 /* CUDA device ordinal */
    uint64_t hbm_budget_bytes;  /* 0 = whatever is free on the device */
    int verbose;
    uint64_t stream;            /* a cudaStream_t to run on (e.g. the caller's timing stream); 0 = create a private stream */
} sgpu_config;

enum { SGPU_CANONICAL = 0, SGPU_ALL_WINDOWS = 1 };

enum {
    SGPU_OK = 0, SGPU_EINVAL = 2, SGPU_ENODEV = 3, SGPU_ENOMEM = 4, SGPU_ECUDA = 5, SGPU_EINTERNAL = 6, SGPU_EUNSUPPORTED = 7,
    SGPU_EIO = 8
};

/* device-side milliseconds of the last sgpu_count / sgpu_kmers_from_kpomers / sgpu_mphf_build, measured with CUDA events
 * on the context's stream, plus the number of kernels launched since the context was created */
typedef struct sgpu_times {
    float extract_count_ms, extract_scatter_ms, refine_ms, local_sort_ms, compact_ms, mphf_ms, exchange_ms;
    uint64_t instances;   /* records the partition kernel wrote */
    uint64_t passes;      /* bucket-group passes */
    uint64_t launches;    /* kernels launched by this context so far */
    uint64_t peak_bytes;  /* peak device memory held by this context */
    uint64_t cached_bytes;/* freed device blocks kept by the context's caching allocator (reusable) */
} sgpu_times;

int sgpu_create(const sgpu_config *cfg, sgpu_ctx **out);
/* k-mer sets, indexes, graphs and distributed counts created from a context keep device memory of that context. Destroying the
 * context while some are alive is safe in any order: the context is torn down when the last of them has been freed. */
void sgpu_destroy(sgpu_ctx *ctx);
const char *sgpu_last_error(const sgpu_ctx *ctx);
int sgpu_get_times(const sgpu_ctx *ctx, sgpu_times *out);

/* reads: read r occupies words[offs[r] .. offs[r]+ceil(lens[r]/32)), nucleotide i at bits 2(i%32) of word i/32, A=0 C=1 G=2 T=3
 * (N-free: apply LongestValid first, io/reads/longest_valid_wrapper.hpp:16-53). offs are relative to `words`. */
int sgpu_reads_clear(sgpu_ctx *ctx);
int sgpu_reads_append_packed(sgpu_ctx *ctx, const uint64_t *words, uint64_t nwords, const uint64_t *offs, const uint32_t *lens, int64_t nreads);
/* replace the read set with these HOST buffers, copied straight to the device (pinned buffers copy at full PCIe rate). The copies
 * are enqueued on the context's stream and the call returns: the buffers must stay valid and unmodified until the next
 * sgpu_count / sgpu_dist_begin on this context has returned (both synchronise the stream). */
int sgpu_reads_upload(sgpu_ctx *ctx, const uint64_t *words, uint64_t nwords, const uint64_t *offs, const uint32_t *lens, int64_t nreads);
/* GPU-side packing (SURVEY 8f-2): the host only locates the sequence of every read inside a text buffer (FASTA/FASTQ file contents:
 * byte offset + length of each single-line sequence; sgpu_text_index_fastx does it for 2-line FASTA / 4-line FASTQ); the device applies
 * io::LongestValid (io/reads/longest_valid_wrapper.hpp:16-53; longest_valid = 0: a read with any non-ACGT symbol contributes nothing)
 * and packs 2 bits per base (Sequence::BinWrite payload). Replaces the context's read set; reads without a valid base keep a slot of
 * length 0. */
int sgpu_reads_pack_text(sgpu_ctx *ctx, const char *text, uint64_t text_bytes, const uint64_t *seq_off, const uint32_t *seq_len, int64_t nreads,
                         int longest_valid);
/* the context's current (packed) read set: sizes, and a copy to host arrays of those sizes (any pointer may be NULL) */
int sgpu_reads_info(sgpu_ctx *ctx, int64_t *nreads, uint64_t *nwords);
int sgpu_reads_download(sgpu_ctx *ctx, uint64_t *words, uint64_t *offs, uint32_t *lens);
/* Coverage pre-filter of the construction stage (SURVEY 8f-3; the pipeline's CoverageFilter phase, stages/construction.cpp:167-198, active
 * when read_cov_threshold > 0): K = k + 1. (1) HyperLogLog upper bound of the distinct K-mers (EstimateCardinalityUpperBound,
 * kmer_index/kmer_counting.hpp:215-249; adt/hll.hpp) with rolling_hash::SymmetricCyclicHash (adt/cyclichash.hpp:187-259); (2) the counting
 * quotient filter sized from it (qf::cqf, adt/cqf.hpp:28-37) filled up to `threshold` per key (FillCoverageHistogram, kmer_counting.hpp:251-282);
 * (3) io::CovFilteringWrap (io/reads/coverage_filtering_read_wrapper.hpp): a read survives iff the median multiplicity of its K-mers is >=
 * threshold. keep_out (may be NULL): one byte per read of the CURRENT read set, 1 = survives. apply != 0: the survivors (order kept) become
 * the context's read set, as the wrapper does to the pipeline's streams. stats (may be NULL): [0] cardinality upper bound, [1] key bits of
 * the filter (qbits + 8), [2] distinct keys counted, [3] reads kept. */
int sgpu_reads_cov_filter(sgpu_ctx *ctx, int K, unsigned threshold, int apply, uint8_t *keep_out, uint64_t *stats);
/* use a read set that already lives in device memory (not copied, must stay valid while the context uses it) */
int sgpu_reads_adopt_device(sgpu_ctx *ctx, const uint64_t *d_words, uint64_t nwords, const uint64_t *d_offs, const uint32_t *d_lens, int64_t nreads);

/* ---- read ingest (pure host code: no GPU, no context needed). Replaces the front end of the tools: io::FastaFastqGzParser
 * over kseq + zlib (io/reads/fasta_fastq_gz_parser.hpp:25-150), io::LongestValid (io/reads/longest_valid_wrapper.hpp:16-53, applied
 * by io_helper.cpp:30-31 and read_converter.cpp:115,121) and the binary read streams <prefix>.seq / <prefix>.off that
 * io::BinaryWriter::ToBinary writes and io::BinaryFileStream<SingleReadSeq> reads (io/reads/binary_converter.cpp:84-145,
 * binary_streams.hpp:54-102; record = Sequence::BinWrite + SingleReadSeq::BinWrite, sequence.hpp:817-830, single_read.hpp:325-338).
 * A batch holds 2-bit packed reads in the layout sgpu_reads_append_packed / sgpu_reads_upload take. Reads without any valid
 * base are dropped (they contribute no k-mer). On failure *out is still a batch whose sgpu_read_batch_error() says why. */
typedef struct sgpu_read_batch sgpu_read_batch;
int sgpu_fastx_parse(const char *path, int longest_valid, sgpu_read_batch **out);      /* FASTA / FASTQ, plain or gzip */
/* nthreads > 1: an uncompressed file is parsed in parallel pieces, accepted only where the sequential parser provably stands at
 * the same place (otherwise, and for gzip, the sequential parse runs); 0 = hardware threads (SGPU_INGEST_THREADS overrides), 1 = sequential */
int sgpu_fastx_parse_threads(const char *path, int longest_valid, int nthreads, sgpu_read_batch **out);
int sgpu_seqfile_parse(const char *prefix, sgpu_read_batch **out);                     /* <prefix>.seq of the reference */
int sgpu_read_batch_write_seqfile(const sgpu_read_batch *b, const char *prefix);       /* <prefix>.seq + <prefix>.off */
int64_t sgpu_read_batch_num_reads(const sgpu_read_batch *b);
uint64_t sgpu_read_batch_num_words(const sgpu_read_batch *b);
const uint64_t *sgpu_read_batch_words(const sgpu_read_batch *b);
const uint64_t *sgpu_read_batch_offs(const sgpu_read_batch *b);
const uint32_t *sgpu_read_batch_lens(const sgpu_read_batch *b);
int sgpu_read_batch_stats(const sgpu_read_batch *b, uint64_t *out3);   /* records in the file, reads trimmed by LongestValid, reads dropped */
const char *sgpu_read_batch_error(const sgpu_read_batch *b);
void sgpu_read_batch_free(sgpu_read_batch *b);
/* host side of sgpu_reads_pack_text: sequence ranges of a strictly 2-line FASTA ('>') / 4-line FASTQ ('@', '+', quality as long as the
 * sequence) text; a trailing '\r' is excluded. out arrays must hold max_reads entries; returns the number of reads, -1 if the text is
 * not in that strict layout (then use sgpu_fastx_parse, which implements kseq's general record semantics), -2 if max_reads is too small */
int64_t sgpu_text_index_fastx(const char *text, uint64_t text_bytes, uint64_t *seq_off, uint32_t *seq_len, int64_t max_reads);
/* sgpu_reads_append_packed of a whole batch */
int sgpu_reads_append_batch(sgpu_ctx *ctx, const sgpu_read_batch *b);

int sgpu_count(sgpu_ctx *ctx, int K, int num_buckets, int mode, sgpu_kset **out);
int sgpu_kmers_from_kpomers(sgpu_ctx *ctx, const sgpu_kset *kpomers, int num_buckets, sgpu_kset **out);

int64_t sgpu_kset_size(const sgpu_kset *s);
int sgpu_kset_k(const sgpu_kset *s);
int sgpu_kset_num_buckets(const sgpu_kset *s);
int sgpu_kset_record_bytes(const sgpu_kset *s);                       /* KMerCounter::kmer_size(): 8*ceil(K/32) */
int sgpu_kset_bucket_sizes(const sgpu_kset *s, int64_t *out);         /* num_buckets entries */
/* records [first, first+n) of final_kmers order (KMerDiskStorage::merge, kmer_index_builder.hpp:190-203) to host memory */
/* order-independent checksums computed on the device: out4 = { number of records, weighted sum of all record words, xor of
 * the rotated record words, sum of the multiplicities } (mod 2^64). Disjoint bucket sets add / xor up, so the per-rank sets of a
 * multi-GPU count can be checked against a single-GPU count of the union without moving records. */
int sgpu_kset_checksum(const sgpu_kset *s, uint64_t *out4);
int sgpu_kset_download_keys(const sgpu_kset *s, int64_t first, int64_t n, uint64_t *out);
int sgpu_kset_download_counts(const sgpu_kset *s, int64_t first, int64_t n, uint32_t *out);   /* SGPU_CANONICAL sets only */
/* writes <prefix>.<b> for every bucket in the reference's bucket file format (raw W-byte records) */
int sgpu_kset_write_buckets(const sgpu_kset *s, const char *prefix);
int sgpu_kset_write_final(const sgpu_kset *s, const char *path);      /* final_kmers */
void sgpu_kset_free(sgpu_kset *s);

int sgpu_mphf_build(sgpu_ctx *ctx, const sgpu_kset *s, sgpu_mphf **out);
int64_t sgpu_mphf_serialized_size(const sgpu_mphf *m);
int sgpu_mphf_serialize(const sgpu_mphf *m, uint8_t *out, int64_t cap);
/* host keys, stored (minimal) form. A key of the set gets its slot; any other key gets what KMerIndex::seq_idx gives: -1 (2^64 - 1),
 * always so when its bucket holds no key, or the slot of some other key of the set */
int sgpu_mphf_lookup(const sgpu_mphf *m, const uint64_t *keys, int64_t n, uint64_t *out_idx);
void sgpu_mphf_free(sgpu_mphf *m);

/* kpomers must come from sgpu_count(k+1, B, SGPU_CANONICAL); kmers/kmer_index from sgpu_kmers_from_kpomers / sgpu_mphf_build.
 * kpomer_index may be NULL (then no coverage: DP/KC are 0 and sgpu_graph_coverage fails). The graph borrows its inputs. */
int sgpu_graph_build(sgpu_ctx *ctx, const sgpu_kset *kpomers, const sgpu_kset *kmers, const sgpu_mphf *kmer_index,
                     const sgpu_mphf *kpomer_index, int keep_perfect_loops, sgpu_graph **out);
/* sgpu_graph_build plus the pipeline's early tip clipper between the mask fill and the unitig extraction:
 * EarlyTipClipperProcessor::ClipTips (assembly_graph/construction/early_simplification.hpp:38-162) as run by the Construction
 * stage (stages/construction.cpp:289-302, modules/graph_construction.hpp:32-36) with length_bound = read length - k.
 * early_tip_length_bound = 0 switches it off (== sgpu_graph_build, what spades-gbuilder does). sgpu_graph_masks then returns
 * the clipped array. stats: removed k-mers (ClipTips' return value), tipped junctions, clipped links (its INFO counters). */
int sgpu_graph_build_ex(sgpu_ctx *ctx, const sgpu_kset *kpomers, const sgpu_kset *kmers, const sgpu_mphf *kmer_index,
                        const sgpu_mphf *kpomer_index, int keep_perfect_loops, uint64_t early_tip_length_bound, sgpu_graph **out);
int sgpu_graph_tip_clipper_stats(const sgpu_graph *g, uint64_t *out3);
/* all options of the Construction stage's graph phases in one call. early_at_clipper: EarlyLowComplexityClipperProcessor::
 * RemoveATEdges + RemoveATTips (assembly_graph/construction/early_simplification.hpp:164-347), the EarlyATClipper phase the RNA
 * pipeline runs before the tip clipper (stages/construction.cpp:317-340,447-448 with at_ratio 0.8, min_length 10, max_length 200;
 * min_length must not exceed k). sgpu_graph_masks then returns the array after both clippers. */
typedef struct sgpu_graph_options {
    int keep_perfect_loops;
    uint64_t early_tip_length_bound;   /* 0 = off */
    int early_at_clipper;              /* 0 = off */
    double at_ratio;
    uint64_t at_min_length, at_max_length;
} sgpu_graph_options;
int sgpu_graph_build_opts(sgpu_ctx *ctx, const sgpu_kset *kpomers, const sgpu_kset *kmers, const sgpu_mphf *kmer_index,
                          const sgpu_mphf *kpomer_index, const sgpu_graph_options *opts, sgpu_graph **out);
/* stats: edges collected (RemoveATEdges' return value), links removed, k-mers removed (RemoveATTips' return value), clipped tips */
int sgpu_graph_at_clipper_stats(const sgpu_graph *g, uint64_t *out4);
int sgpu_graph_masks(const sgpu_graph *g, uint8_t *out, int64_t n);           /* n = number of k-mers */
int sgpu_graph_coverage(const sgpu_graph *g, uint32_t *out, int64_t n);       /* n = number of (k+1)-mers */
int64_t sgpu_graph_histogram(const sgpu_graph *g, uint64_t *out, int64_t cap);/* returns the histogram length (max coverage) */
int64_t sgpu_graph_num_unitigs(const sgpu_graph *g);
int64_t sgpu_graph_unitig_bases(const sgpu_graph *g);
/* ASCII unitigs concatenated into out (sgpu_graph_unitig_bases() bytes) and their lengths */
int sgpu_graph_unitigs(const sgpu_graph *g, char *out, uint32_t *lens);
int64_t sgpu_graph_gfa(const sgpu_graph *g, const char *version, char *out, int64_t cap);   /* returns the text size */
int sgpu_graph_write_gfa(const sgpu_graph *g, const char *version, const char *path);
void sgpu_graph_free(sgpu_graph *g);

/* ---- EdgeIndex refill (the next consumer of the graph in the pipeline): debruijn_graph::EdgeIndex<Graph>::Refill
 * (alignment/edge_index.hpp:88-110, modules/graph_construction.hpp:74-82) = GraphPositionFillingIndexBuilder::BuildIndexFromGraph
 * (assembly_graph/index/edge_index_builders.hpp:154-307) + EdgeInfoUpdater::UpdateAll (edge_info_updater.hpp:38-101) over the
 * graph's own unitigs. num_buckets = 10 x the reference's threads in both cases: K = 0 means k+1 -- the reference then walks the
 * edges in that many vertex chunks and builds ONE index segment (num_buckets only decides a serialization detail, see
 * edge_index.cu); any other K counts through DeBruijnGraphKMerSplitter + KMerDiskCounter into num_buckets buckets. The index holds every K-mer of every edge
 * and of its conjugate (KmerFreeEdgeIndex, DefaultStoring); a slot's value is (EdgeId::int_id(), offset) -- edge i of
 * sgpu_graph_unitigs has id 3 + 2i, its conjugate 3 + 2i + 1 -- or (~1, 0x7ffffffe) when the K-mer occurs more than once in the
 * graph (EdgeInfo TOMBSTONE, edge_position_index.hpp:29-30,152-167). The graph may be freed afterwards. */
typedef struct sgpu_edge_index sgpu_edge_index;
int sgpu_edge_index_build(sgpu_ctx *ctx, const sgpu_graph *g, int K, int num_buckets, sgpu_edge_index **out);
int sgpu_edge_index_k(const sgpu_edge_index *e);
int64_t sgpu_edge_index_size(const sgpu_edge_index *e);                              /* number of K-mers = number of slots */
int64_t sgpu_edge_index_serialized_size(const sgpu_edge_index *e);
int sgpu_edge_index_serialize(const sgpu_edge_index *e, uint8_t *out, int64_t cap);   /* KMerIndex::serialize bytes */
int sgpu_edge_index_values(const sgpu_edge_index *e, uint64_t *edge_ids, uint32_t *offsets, int64_t n);   /* slot order */
/* host keys (stored form) -> slots; a K-mer not in the index gets -1 or the slot of some other K-mer, as in sgpu_mphf_lookup */
int sgpu_edge_index_lookup(const sgpu_edge_index *e, const uint64_t *keys, int64_t n, uint64_t *out_idx);
void sgpu_edge_index_free(sgpu_edge_index *e);

/* ---- multi-GPU count (one process per GPU; SURVEY 8e). Replaces hpcspades' shared-filesystem + MPI pattern
 * (projects/hpcspades/mpi/stages/construction_mpi.cpp:222-300, mpi/kmer_index/kmer_extension_index_builder_mpi.hpp:87,190):
 * buckets are owned by ranks; every rank partitions its own reads into a staging buffer (same kernels as sgpu_count), then
 * sgpu_dist_exchange is ONE kernel on the owner that pulls its pieces from all peers' staging buffers over NVLink peer memory
 * (cudaIpc mappings of the peers' memory arenas, opened once per process) and merges them partition by partition. The host
 * language only moves small tables between ranks (torch.distributed / MPI all_gather) and provides the barriers:
 *   begin -> local_counts -> [all_gather counts] -> plan ->
 *   repeat: free_bytes -> [all_reduce MIN] -> next_pass (-1 = done) -> ipc_handle -> [all_gather descriptors] -> open_peers ->
 *           scatter [barrier] exchange [barrier] sort
 *   -> end (k-mer set holding this rank's buckets)
 * Passes are planned one at a time against the memory every rank has free at that moment (like sgpu_count's bucket-group passes). */
typedef struct sgpu_dist sgpu_dist;
int sgpu_dist_begin(sgpu_ctx *ctx, int K, int num_buckets, int mode, int world, int rank, sgpu_dist **out);
int64_t sgpu_dist_num_partitions(const sgpu_dist *d);
int sgpu_dist_local_counts(sgpu_dist *d, uint64_t *out);                 /* num_partitions host entries */
int sgpu_dist_plan(sgpu_dist *d, const uint64_t *all_counts /* world x num_partitions, rank-major, host */, uint64_t *total_records);
int sgpu_dist_free_bytes(sgpu_dist *d, uint64_t *out);                  /* device bytes this rank can allocate for the next pass */
/* budget_bytes: the MINIMUM of sgpu_dist_free_bytes over the ranks (identical inputs give identical decisions on every rank).
 * *pass = index of the pass that was planned and whose buffers were allocated, or -1 when all buckets are done */
int sgpu_dist_next_pass(sgpu_dist *d, uint64_t budget_bytes, int *pass);
#define SGPU_IPC_BYTES 96
/* this rank's descriptor for the current pass: cudaIpcMemHandle_t of its memory arena + the offsets of its staging buffer and
 * piece tables inside it */
int sgpu_dist_ipc_handle(sgpu_dist *d, uint8_t *out /* SGPU_IPC_BYTES */);
int sgpu_dist_open_peers(sgpu_dist *d, const uint8_t *descriptors /* world x SGPU_IPC_BYTES, rank-major */);
int sgpu_dist_scatter(sgpu_dist *d, int pass);                          /* partition this rank's shard into its staging buffer */
int sgpu_dist_exchange(sgpu_dist *d, int pass);                         /* fused NVLink exchange + merge: pulls the owned pieces from every peer */
int sgpu_dist_sort(sgpu_dist *d, int pass);                             /* refinement + local sort + compaction of what arrived */
int sgpu_dist_end(sgpu_dist *d, sgpu_kset **out);
void sgpu_dist_free(sgpu_dist *d);
/* the planning step alone (pure host arithmetic, no GPU): returns npass and fills pass_bounds[0..npass] */
int sgpu_dist_plan_host(int world, int num_buckets, int key_bits_in_partition, const uint64_t *all_counts, uint64_t budget_bytes,
                        int record_bytes, int *pass_bounds, uint64_t *max_recv);

/* self tests of the shared host/device arithmetic (tests only): op 0 = xxh3_64, 1 = xxh3_128 lo, 2 = xxh3_128 hi, 3 = bucket(arg),
 * 4 = is_minimal, 5.. = rc word j. keys: n records of ceil(K/32) words. on_device != 0 runs the same code in a kernel. */
int sgpu_selftest(sgpu_ctx *ctx, int on_device, int op, int K, uint64_t arg, const uint64_t *keys, int64_t n, uint64_t *out);

#ifdef __cplusplus
}
#endif
#endif
