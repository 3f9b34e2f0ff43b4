/*
 * oracle/spades_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * Plain-C, single-threaded, obviously-correct restatement of the SPAdes k-mer counting /
 * de Bruijn construction hot path (ablab/spades 4.3.0-dev). It exists so that the CUDA path can be
 * checked bit-for-bit on machines where /root/reference is absent (the GPU box). Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline leg may load it; the product
 * (spades_b200/) never does.
 *
 * Parity of this file is PINNED against the unmodified reference (oracle/_ref/ref_probe, built from the
 * reference's own sources) by tests/test_oracle_vs_reference.py and the fixtures under tests/golden/.
 *
 * Every function cites the reference file:line it restates (paths relative to /root/reference).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#include <math.h>

typedef unsigned __int128 u128;

/* ------------------------------------------------------------------------------------------------
 * 2-bit k-mers.  src/common/sequence/rtseq.hpp:379-382 : nucleotide i lives at bits 2(i%32)..+1 of
 * word i/32, A=0 C=1 G=2 T=3 (src/common/sequence/nucl.hpp:132-142); unused high bits are zero.
 * ---------------------------------------------------------------------------------------------- */
#define MAXW 4
static inline int nwords(int K) { return (K + 31) >> 5; }             /* rtseq.hpp:131-133 */
static inline int getnuc(const uint64_t *w, int i) { return (int)((w[i >> 5] >> ((i & 31) << 1)) & 3); }
static inline void orc_setnuc(uint64_t *w, int i, int c) { w[i >> 5] |= (uint64_t)c << ((i & 31) << 1); }

/* reverse complement, the slow definition (rtseq.hpp:391-404 commented body == FastRC :81-117) */
void orc_rc(const uint64_t *in, int K, uint64_t *out) {
    for (int i = 0; i < nwords(K); ++i) out[i] = 0;
    for (int i = 0; i < K; ++i) orc_setnuc(out, i, 3 - getnuc(in, K - 1 - i));
}

/* RtSeq::IsMinimal, rtseq.hpp:409-417 */
int orc_is_minimal(const uint64_t *w, int K) {
    for (int i = 0; (i << 1) + 1 <= K; ++i) {
        int front = getnuc(w, i), end = 3 - getnuc(w, K - 1 - i);
        if (front != end) return front < end;
    }
    return 1;
}

/* operator<(RtSeq,RtSeq), rtseq.hpp:740-748 : nucleotide-lexicographic */
static int kmer_nuc_less(const uint64_t *a, const uint64_t *b, int K) {
    for (int i = 0; i < K; ++i) {
        int x = getnuc(a, i), y = getnuc(b, i);
        if (x != y) return x < y;
    }
    return 0;
}

/* word-lexicographic order used inside buckets: ext/include/pdqsort/pdqsort_pod.h:725-734,
 * src/common/adt/array_vector.hpp:115-124 */
static int g_cmp_nw;
static int cmp_words(const void *pa, const void *pb) {
    const uint64_t *a = (const uint64_t *)pa, *b = (const uint64_t *)pb;
    for (int i = 0; i < g_cmp_nw; ++i) {
        if (a[i] != b[i]) return a[i] < b[i] ? -1 : 1;
    }
    return 0;
}

/* ------------------------------------------------------------------------------------------------
 * XXH3 (xxHash 0.8.2, ext/include/xxh/xxhash.h) short-input paths for 8/16/24/32-byte inputs, seed 0.
 * ---------------------------------------------------------------------------------------------- */
static const uint8_t kSecret[192] = { /* xxhash.h:4239-4252 */
    0xb8, 0xfe, 0x6c, 0x39, 0x23, 0xa4, 0x4b, 0xbe, 0x7c, 0x01, 0x81, 0x2c, 0xf7, 0x21, 0xad, 0x1c,
    0xde, 0xd4, 0x6d, 0xe9, 0x83, 0x90, 0x97, 0xdb, 0x72, 0x40, 0xa4, 0xa4, 0xb7, 0xb3, 0x67, 0x1f,
    0xcb, 0x79, 0xe6, 0x4e, 0xcc, 0xc0, 0xe5, 0x78, 0x82, 0x5a, 0xd0, 0x7d, 0xcc, 0xff, 0x72, 0x21,
    0xb8, 0x08, 0x46, 0x74, 0xf7, 0x43, 0x24, 0x8e, 0xe0, 0x35, 0x90, 0xe6, 0x81, 0x3a, 0x26, 0x4c,
    0x3c, 0x28, 0x52, 0xbb, 0x91, 0xc3, 0x00, 0xcb, 0x88, 0xd0, 0x65, 0x8b, 0x1b, 0x53, 0x2e, 0xa3,
    0x71, 0x64, 0x48, 0x97, 0xa2, 0x0d, 0xf9, 0x4e, 0x38, 0x19, 0xef, 0x46, 0xa9, 0xde, 0xac, 0xd8,
    0xa8, 0xfa, 0x76, 0x3f, 0xe3, 0x9c, 0x34, 0x3f, 0xf9, 0xdc, 0xbb, 0xc7, 0xc7, 0x0b, 0x4f, 0x1d,
    0x8a, 0x51, 0xe0, 0x4b, 0xcd, 0xb4, 0x59, 0x31, 0xc8, 0x9f, 0x7e, 0xc9, 0xd9, 0x78, 0x73, 0x64,
    0xea, 0xc5, 0xac, 0x83, 0x34, 0xd3, 0xeb, 0xc3, 0xc5, 0x81, 0xa0, 0xff, 0xfa, 0x13, 0x63, 0xeb,
    0x17, 0x0d, 0xdd, 0x51, 0xb7, 0xf0, 0xda, 0x49, 0xd3, 0x16, 0x55, 0x26, 0x29, 0xd4, 0x68, 0x9e,
    0x2b, 0x16, 0xbe, 0x58, 0x7d, 0x47, 0xa1, 0xfc, 0x8f, 0xf8, 0xb8, 0xd1, 0x7a, 0xd0, 0x31, 0xce,
    0x45, 0xcb, 0x3a, 0x8f, 0x95, 0x16, 0x04, 0x28, 0xaf, 0xd7, 0xfb, 0xca, 0xbb, 0x4b, 0x40, 0x7e,
};
#define P64_1 0x9E3779B185EBCA87ULL  /* xxhash.h:3353-3357 */
#define P64_2 0xC2B2AE3D27D4EB4FULL
#define P64_4 0x85EBCA77C2B2AE63ULL
#define P32_2 0x85EBCA77U            /* xxhash.h:2834 */
#define PMX1  0x165667919E3779F9ULL  /* xxhash.h:4254-4255 */
#define PMX2  0x9FB21C651E98DF25ULL

static inline uint64_t sec64(int off) { uint64_t v; memcpy(&v, kSecret + off, 8); return v; } /* little-endian host */
static inline uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
static inline uint64_t swap64(uint64_t x) { return __builtin_bswap64(x); }
static inline uint64_t mul128_fold64(uint64_t a, uint64_t b) { u128 p = (u128)a * b; return (uint64_t)p ^ (uint64_t)(p >> 64); } /* :4440 */
static inline uint64_t xorshift64(uint64_t v, int s) { return v ^ (v >> s); }
static inline uint64_t avalanche(uint64_t h) { h = xorshift64(h, 37); h *= PMX1; return xorshift64(h, 32); } /* :4457 */
static inline uint64_t rrmxmx(uint64_t h, uint64_t len) {  /* :4470-4478 */
    h ^= rotl64(h, 49) ^ rotl64(h, 24); h *= PMX2; h ^= (h >> 35) + len; h *= PMX2; return xorshift64(h, 28);
}
static inline uint64_t mix16B(const uint64_t *in, int soff) { /* :4606-4623, seed 0 */
    return mul128_fold64(in[0] ^ sec64(soff), in[1] ^ sec64(soff + 8));
}

/* XXH3_64bits_withSeed(words, 8*nw, 0): rtseq.hpp:690-696 calls it on the first ceil(K/32) words */
uint64_t orc_xxh3_64(const uint64_t *w, int nw) {
    uint64_t len = 8ULL * nw;
    if (nw == 1) { /* XXH3_len_4to8_64b, :4537-4550 */
        uint32_t in1 = (uint32_t)w[0], in2 = (uint32_t)(w[0] >> 32);
        uint64_t bitflip = sec64(8) ^ sec64(16);
        uint64_t in64 = in2 + ((uint64_t)in1 << 32);
        return rrmxmx(in64 ^ bitflip, len);
    }
    if (nw == 2) { /* XXH3_len_9to16_64b, :4553-4567 */
        uint64_t lo = w[0] ^ (sec64(24) ^ sec64(32));
        uint64_t hi = w[1] ^ (sec64(40) ^ sec64(48));
        uint64_t acc = len + swap64(lo) + hi + mul128_fold64(lo, hi);
        return avalanche(acc);
    }
    /* XXH3_len_17to128_64b, :4640-4675 ; len 24 or 32 (<=32 so only the last two mixes) */
    uint64_t acc = len * P64_1;
    acc += mix16B(w, 0);
    acc += mix16B(w + nw - 2, 16);
    return avalanche(acc);
}

/* XXH3_128bits(words, 8*nw): src/common/kmer_index/kmer_mph/kmer_index.hpp:39-52 (returns {high64, low64}) */
void orc_xxh3_128(const uint64_t *w, int nw, uint64_t *low64, uint64_t *high64) {
    uint64_t len = 8ULL * nw;
    if (nw == 1) { /* XXH3_len_4to8_128b, :6449-6473 */
        uint32_t ilo = (uint32_t)w[0], ihi = (uint32_t)(w[0] >> 32);
        uint64_t in64 = ilo + ((uint64_t)ihi << 32);
        uint64_t bitflip = sec64(16) ^ sec64(24);
        uint64_t keyed = in64 ^ bitflip;
        u128 m = (u128)keyed * (P64_1 + (len << 2));
        uint64_t lo = (uint64_t)m, hi = (uint64_t)(m >> 64);
        hi += (lo << 1);
        lo ^= (hi >> 3);
        lo = xorshift64(lo, 35); lo *= PMX2; lo = xorshift64(lo, 28);
        hi = avalanche(hi);
        *low64 = lo; *high64 = hi; return;
    }
    if (nw == 2) { /* XXH3_len_9to16_128b, :6476-6545 */
        uint64_t bitflipl = sec64(32) ^ sec64(40);
        uint64_t bitfliph = sec64(48) ^ sec64(56);
        uint64_t ilo = w[0], ihi = w[1];
        u128 m = (u128)(ilo ^ ihi ^ bitflipl) * P64_1;
        uint64_t mlo = (uint64_t)m, mhi = (uint64_t)(m >> 64);
        mlo += (uint64_t)(len - 1) << 54;
        ihi ^= bitfliph;
        mhi += ihi + (uint64_t)(uint32_t)ihi * (uint64_t)(P32_2 - 1);
        mlo ^= swap64(mhi);
        u128 h = (u128)mlo * P64_2;
        uint64_t hlo = (uint64_t)h, hhi = (uint64_t)(h >> 64);
        hhi += mhi * P64_2;
        *low64 = avalanche(hlo); *high64 = avalanche(hhi); return;
    }
    /* XXH3_len_17to128_128b, :6570-6625 ; len<=32 so one XXH128_mix32B(acc, input, input+len-16, secret) */
    uint64_t alo = len * P64_1, ahi = 0;
    const uint64_t *in1 = w, *in2 = w + nw - 2;
    alo += mix16B(in1, 0);
    alo ^= in2[0] + in2[1];
    ahi += mix16B(in2, 16);
    ahi ^= in1[0] + in1[1];
    uint64_t hlo = alo + ahi;
    uint64_t hhi = alo * P64_1 + ahi * P64_4 + (len - 0) * P64_2;
    *low64 = avalanche(hlo);
    *high64 = (uint64_t)0 - avalanche(hhi);
}

/* KMerSegmentPolicy::operator(), src/common/kmer_index/kmer_mph/kmer_buckets.hpp:41-61 ;
 * multiply_high_u64, src/common/adt/lemiere_mod_reduce.hpp:18-21 */
uint64_t orc_bucket(const uint64_t *w, int nw, uint64_t B) {
    if (B == 1) return 0;
    return (uint64_t)(((u128)orc_xxh3_64(w, nw) * (u128)B) >> 64);
}

/* ------------------------------------------------------------------------------------------------
 * k-mer sets: what KMerDiskCounter::Count leaves on disk (B bucket files of strictly increasing records,
 * kmer_index_builder.hpp:306-332) plus, for the canonical mode, the multiplicities the reference obtains in
 * a second pass (coverage_hash_map_builder.hpp:18-40).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int K, nw, B;
    int64_t n;
    uint64_t *keys;     /* n*nw words, bucket-major, sorted inside a bucket == final_kmers (:190-203) */
    uint32_t *counts;   /* n, or NULL */
    int64_t *bsz;       /* B bucket sizes */
} kset_t;

void orc_kset_free(kset_t *s) { if (!s) return; free(s->keys); free(s->counts); free(s->bsz); free(s); }
int64_t orc_kset_n(const kset_t *s) { return s->n; }
int orc_kset_nw(const kset_t *s) { return s->nw; }
const uint64_t *orc_kset_keys(const kset_t *s) { return s->keys; }
const uint32_t *orc_kset_counts(const kset_t *s) { return s->counts; }
const int64_t *orc_kset_bsz(const kset_t *s) { return s->bsz; }

typedef struct { uint64_t *rec; int64_t n, cap; int rw; } recvec_t;   /* records: [bucket, w0..w(nw-1)] */
static void rv_push(recvec_t *v, uint64_t b, const uint64_t *w, int nw) {
    if (v->n == v->cap) { v->cap = v->cap ? v->cap * 2 : 1024; v->rec = (uint64_t *)realloc(v->rec, (size_t)v->cap * v->rw * 8); }
    uint64_t *r = v->rec + v->n * v->rw;
    r[0] = b; memcpy(r + 1, w, 8 * nw); v->n++;
}

/* sort by (bucket, words), unique, count run lengths */
static kset_t *finish_set(recvec_t *v, int K, int B, int want_counts) {
    int nw = nwords(K);
    g_cmp_nw = nw + 1;
    qsort(v->rec, (size_t)v->n, (size_t)v->rw * 8, cmp_words);
    kset_t *s = (kset_t *)calloc(1, sizeof(kset_t));
    s->K = K; s->nw = nw; s->B = B;
    s->bsz = (int64_t *)calloc((size_t)B, 8);
    s->keys = (uint64_t *)malloc((size_t)(v->n ? v->n : 1) * nw * 8);
    s->counts = want_counts ? (uint32_t *)malloc((size_t)(v->n ? v->n : 1) * 4) : NULL;
    int64_t m = 0;
    for (int64_t i = 0; i < v->n; ++i) {
        const uint64_t *r = v->rec + i * v->rw;
        if (i && memcmp(r, r - v->rw, (size_t)v->rw * 8) == 0) {   /* std::unique, kmer_splitter.hpp:140 / kmer_index_builder.hpp:381-403 */
            if (want_counts) s->counts[m - 1] += 1;                  /* uint32 wrap, construction.cpp:26 */
            continue;
        }
        memcpy(s->keys + m * nw, r + 1, 8 * nw);
        if (want_counts) s->counts[m] = 1;
        s->bsz[r[0]] += 1;
        m++;
    }
    s->n = m;
    free(v->rec);
    return s;
}

/* shift-left-and-append: RtSeq::operator<<=, rtseq.hpp:459-476 */
static void kmer_shl(uint64_t *w, int K, int c) {
    int nw = nwords(K);
    for (int i = 0; i < nw - 1; ++i) w[i] = (w[i] >> 2) | ((w[i + 1] & 3) << 62);
    int sh = ((K + 31) & 31) << 1;
    w[nw - 1] = (w[nw - 1] >> 2) | ((uint64_t)c << sh);
}

/*
 * mode 0 (graph path): DeBruijnReadKMerSplitter over RCWrap'ed reads with StoringTypeFilter<InvertableStoring>
 *   (kmer_splitters.hpp:28-44,112-136; storing_traits.hpp:92-101; rc_reader_wrapper.hpp:34-43): every window of the
 *   read and of its reverse complement that IsMinimal() is pushed. The run length of a key in the resulting multiset
 *   is exactly what CoverageHashMapBuilder::FillCoverageFromStream (coverage_hash_map_builder.hpp:18-40) adds up, so
 *   `counts` == the reference's coverage value of the key (self-RC (k+1)-mers get 2 per occurrence, SURVEY section 0.6).
 * mode 1 (spades-kmercount): every window of read and RC, no filter (projects/spades_tools/kmercount.cpp:65-83,103).
 * reads: read r occupies words[offs[r] .. offs[r]+ceil(lens[r]/32)) in the rtseq packing; reads shorter than K are
 *   skipped (kmer_splitters.hpp:30-31).
 */
kset_t *orc_count(const uint64_t *words, const uint64_t *offs, const uint32_t *lens, int64_t nreads,
                  int K, int B, int mode) {
    int nw = nwords(K);
    recvec_t v = {0, 0, 0, nw + 1};
    uint64_t *rcbuf = NULL; size_t rccap = 0;
    for (int64_t r = 0; r < nreads; ++r) {
        int L = (int)lens[r];
        if (L < K) continue;
        const uint64_t *fw = words + offs[r];
        size_t need = (size_t)((L + 31) >> 5);
        if (need > rccap) { rccap = need * 2; rcbuf = (uint64_t *)realloc(rcbuf, rccap * 8); }
        memset(rcbuf, 0, need * 8);
        for (int i = 0; i < L; ++i) orc_setnuc(rcbuf, i, 3 - getnuc(fw, L - 1 - i));
        for (int strand = 0; strand < 2; ++strand) {
            const uint64_t *s = strand ? rcbuf : fw;
            uint64_t km[MAXW] = {0, 0, 0, 0};
            for (int i = 0; i < K - 1; ++i) orc_setnuc(km, i + 1, getnuc(s, i));   /* seq.start(K) >> 'A' */
            for (int j = K - 1; j < L; ++j) {
                kmer_shl(km, K, getnuc(s, j));
                if (mode == 0 && !orc_is_minimal(km, K)) continue;
                rv_push(&v, orc_bucket(km, nw, (uint64_t)B), km, nw);
            }
        }
    }
    free(rcbuf);
    return finish_set(&v, K, B, mode == 0);
}

/* DeBruijnKMerKMerSplitter(K_target=k, K_source=k+1, add_rc=true) + IsMinimal filter, kmer_splitters.hpp:163-179,28-62 */
kset_t *orc_kmers_from_kpomers(const kset_t *kp, int B) {
    int K1 = kp->K, K = K1 - 1, nw = nwords(K);
    recvec_t v = {0, 0, 0, nw + 1};
    for (int64_t i = 0; i < kp->n; ++i) {
        const uint64_t *x = kp->keys + i * kp->nw;
        uint64_t rc[MAXW];
        orc_rc(x, K1, rc);
        for (int strand = 0; strand < 2; ++strand) {
            const uint64_t *s = strand ? rc : x;
            for (int st = 0; st < 2; ++st) {
                uint64_t km[MAXW] = {0, 0, 0, 0};
                for (int t = 0; t < K; ++t) orc_setnuc(km, t, getnuc(s, st + t));
                if (!orc_is_minimal(km, K)) continue;
                rv_push(&v, orc_bucket(km, nw, (uint64_t)B), km, nw);
            }
        }
    }
    return finish_set(&v, K, B, 0);
}

/* ------------------------------------------------------------------------------------------------
 * boomphf (ext/include/boomphf/BooPHF.h) as instantiated by KMerIndexBuilder::BuildIndex
 * (kmer_index_builder.hpp:462-475): one mphf(n, Ignore, gamma=4.0, perc=0.03, nb_levels=25) per bucket.
 * ---------------------------------------------------------------------------------------------- */
#define NLEVELS 25
typedef struct {
    uint64_t n;
    uint64_t lastrank;
    uint64_t dom[NLEVELS];      /* hash_domain per level, BooPHF.h:586-595 */
    uint64_t nchar[NLEVELS];    /* 1 + dom/64, :142 */
    uint64_t *bits[NLEVELS];
    uint64_t nranks[NLEVELS];
    uint64_t *ranks[NLEVELS];
    uint64_t nfinal;            /* keys that fell through all 24 bitset levels (order-dependent map, :659-678) */
} mphf1_t;

typedef struct {
    int K, nw, B;
    mphf1_t *seg;               /* B */
    uint64_t *starts;           /* B+1, kmer_index_builder.hpp:468,492-493 (last entry is NOT accumulated) */
} mphf_t;

static inline uint64_t fastrange64(uint64_t w, uint64_t p) { return (uint64_t)(((u128)w * (u128)p) >> 64); } /* :354-356 */

/* iterate_hash, BooPHF.h:606-613 + XorshiftHashFunctors::next :94-100. s[0]=high64, s[1]=low64 (kmer_index.hpp:39-52) */
static inline uint64_t level_hash(uint64_t s[2], int level) {
    if (level == 0) return s[0];
    if (level == 1) return s[1];
    uint64_t s1 = s[0]; const uint64_t s0 = s[1];
    s[0] = s0;
    s1 ^= s1 << 23;
    s[1] = s1 ^ s0 ^ (s1 >> 17) ^ (s0 >> 26);
    return s[1] + s0;
}

/* getLevel, BooPHF.h:616-630 */
static uint64_t get_level(const mphf1_t *m, const uint64_t *key, int nw, int *res_level, int maxlevel) {
    uint64_t s[2], lo, hi;
    orc_xxh3_128(key, nw, &lo, &hi);
    s[0] = hi; s[1] = lo;
    int level; uint64_t h = 0;
    for (level = 0; level < NLEVELS - 1 && level < maxlevel; ++level) {
        h = level_hash(s, level);
        uint64_t p = fastrange64(h, m->dom[level]);
        if ((m->bits[level][p >> 6] >> (p & 63)) & 1) { *res_level = level; return h; }
    }
    *res_level = level;
    return level_hash(s, level);
}

static void mphf1_build(mphf1_t *m, const uint64_t *keys, uint64_t n, int nw) {
    memset(m, 0, sizeof(*m));
    m->n = n;
    if (n == 0) return;                                        /* build() returns early, :426-427 */
    double gamma = 4.0;
    uint64_t hash_domain = (uint64_t)ceil((double)n * gamma);  /* :415 */
    double p = 1.0 - pow(((gamma * (double)n - 1) / (gamma * (double)n)), (double)(n - 1)); /* :586 */
    for (int l = 0; l < NLEVELS; ++l) {
        uint64_t d = (((uint64_t)((double)hash_domain * pow(p, l)) + 63) / 64) * 64;   /* :592 */
        if (d == 0) d = 64;
        m->dom[l] = d;
        m->nchar[l] = 1 + d / 64;
        m->bits[l] = (uint64_t *)calloc(m->nchar[l], 8);
    }
    uint64_t offset = 0;
    for (int l = 0; l < NLEVELS; ++l) {
        uint64_t *coll = (uint64_t *)calloc(m->nchar[l], 8);
        for (uint64_t i = 0; i < n; ++i) {                      /* processLevel/processHash, :684-703,641-682 */
            int lev; uint64_t h = get_level(m, keys + i * nw, nw, &lev, l);
            if (lev != l) continue;
            if (l == NLEVELS - 1) { m->nfinal++; continue; }
            uint64_t pos = fastrange64(h, m->dom[l]);           /* insertIntoLevel, :633-639 */
            uint64_t bit = 1ULL << (pos & 63);
            if (m->bits[l][pos >> 6] & bit) coll[pos >> 6] |= bit; else m->bits[l][pos >> 6] |= bit;
        }
        for (uint64_t w = 0; w < m->dom[l] / 64; ++w) m->bits[l][w] &= ~coll[w];   /* clearCollisions, :219-229 */
        free(coll);
        /* build_ranks, :289-301 */
        m->nranks[l] = (m->nchar[l] + 7) / 8;
        m->ranks[l] = (uint64_t *)malloc(m->nranks[l] * 8);
        uint64_t cur = offset, nr = 0;
        for (uint64_t w = 0; w < m->nchar[l]; ++w) {
            if (((w * 64) % 512) == 0) m->ranks[l][nr++] = cur;
            cur += (uint64_t)__builtin_popcountll(m->bits[l][w]);
        }
        offset = cur;
    }
    m->lastrank = offset;
}

/* mphf::lookup, BooPHF.h:465-487 + bitVector::rank :303-314 */
static uint64_t mphf1_lookup(const mphf1_t *m, const uint64_t *key, int nw) {
    if (m->n == 0) return (uint64_t)-1;
    int lev; uint64_t h = get_level(m, key, nw, &lev, NLEVELS);
    if (lev == NLEVELS - 1) return (uint64_t)-1;
    uint64_t pos = fastrange64(h, m->dom[lev]);
    uint64_t widx = pos / 64, woff = pos % 64, block = pos / 512;
    uint64_t r = m->ranks[lev][block];
    for (uint64_t w = block * 512 / 64; w < widx; ++w) r += (uint64_t)__builtin_popcountll(m->bits[lev][w]);
    r += (uint64_t)__builtin_popcountll(m->bits[lev][widx] & ((1ULL << woff) - 1));
    return r;
}

mphf_t *orc_mphf_build(const kset_t *s) {
    mphf_t *m = (mphf_t *)calloc(1, sizeof(mphf_t));
    m->K = s->K; m->nw = s->nw; m->B = s->B;
    m->seg = (mphf1_t *)calloc((size_t)s->B, sizeof(mphf1_t));
    m->starts = (uint64_t *)calloc((size_t)s->B + 1, 8);
    int64_t off = 0;
    for (int b = 0; b < s->B; ++b) {
        mphf1_build(&m->seg[b], s->keys + off * s->nw, (uint64_t)s->bsz[b], s->nw);
        m->starts[b + 1] = (uint64_t)s->bsz[b];               /* kmer_index_builder.hpp:468 */
        off += s->bsz[b];
    }
    for (int i = 1; i < s->B; ++i) m->starts[i] += m->starts[i - 1];   /* :492-493 (sic: stops before B) */
    return m;
}

void orc_mphf_free(mphf_t *m) {
    if (!m) return;
    for (int b = 0; b < m->B; ++b) for (int l = 0; l < NLEVELS; ++l) { free(m->seg[b].bits[l]); free(m->seg[b].ranks[l]); }
    free(m->seg); free(m->starts); free(m);
}

/* KMerIndex::seq_idx, kmer_index.hpp:88-93 (key must already be the stored (minimal) form) */
uint64_t orc_mphf_lookup(const mphf_t *m, const uint64_t *key) {
    uint64_t b = orc_bucket(key, m->nw, (uint64_t)m->B);
    uint64_t i = mphf1_lookup(&m->seg[b], key, m->nw);
    return i == (uint64_t)-1 ? i : m->starts[b] + i;
}

/* orc_mphf_lookup of n keys of nw words each (one call instead of n from the test harness) */
void orc_mphf_lookup_many(const mphf_t *m, const uint64_t *keys, int64_t n, uint64_t *out) {
    for (int64_t i = 0; i < n; ++i) out[i] = orc_mphf_lookup(m, keys + i * m->nw);
}

uint64_t orc_mphf_nfinal(const mphf_t *m) { uint64_t t = 0; for (int b = 0; b < m->B; ++b) t += m->seg[b].nfinal; return t; }

/* KMerIndex::serialize (kmer_index.hpp:102-108) -> mphf::save (BooPHF.h:514-535) -> bitVector::save (:316-323).
 * Returns the byte count; writes when buf != NULL. For an EMPTY bucket the reference writes its uninitialised
 * _lastbitsetrank member; we write 0 there (comparisons must mask those 8 bytes). */
int64_t orc_mphf_serialize(const mphf_t *m, uint8_t *buf) {
    int64_t p = 0;
#define PUT(ptr, nbytes) do { if (buf) memcpy(buf + p, (ptr), (size_t)(nbytes)); p += (int64_t)(nbytes); } while (0)
    uint64_t nseg = (uint64_t)m->B; PUT(&nseg, 8);
    for (int b = 0; b < m->B; ++b) {
        const mphf1_t *s = &m->seg[b];
        double gamma = 4.0; int nl = NLEVELS;
        PUT(&gamma, 8); PUT(&nl, 4); PUT(&s->lastrank, 8); PUT(&s->n, 8);
        if (s->n != 0) {
            for (int l = 0; l < NLEVELS; ++l) {
                PUT(&s->dom[l], 8); PUT(&s->nchar[l], 8); PUT(s->bits[l], 8 * s->nchar[l]);
                PUT(&s->nranks[l], 8); PUT(s->ranks[l], 8 * s->nranks[l]);
            }
        }
        uint64_t nf = 0; PUT(&nf, 8);   /* final hash map: must be empty (orc_mphf_nfinal()==0) for byte parity */
    }
    PUT(m->starts, 8 * ((size_t)m->B + 1));
#undef PUT
    return p;
}

/* ------------------------------------------------------------------------------------------------
 * Extension masks: DeBruijnExtensionIndexBuilder::FillExtensionsFromIndex (kmer_extension_index_builder.hpp:45-60),
 * InOutMask::AddOutgoing/AddIncoming + inv_position (inout_mask.hpp:92-131), InvertableKeyWithHash::CountIdx
 * (key_with_hash.hpp:120-128). out[] is indexed by the k-mer MPHF index (PerfectHashMap::data_).
 * ---------------------------------------------------------------------------------------------- */
static uint64_t canon_idx(const mphf_t *m, const uint64_t *km, int K, int *is_min) {
    *is_min = orc_is_minimal(km, K);
    if (*is_min) return orc_mphf_lookup(m, km);
    uint64_t rc[MAXW]; orc_rc(km, K, rc);
    return orc_mphf_lookup(m, rc);
}

void orc_masks(const kset_t *kp, const mphf_t *mk, uint8_t *out, int64_t nk) {
    int K1 = kp->K, K = K1 - 1;
    memset(out, 0, (size_t)nk);
    for (int64_t i = 0; i < kp->n; ++i) {
        const uint64_t *x = kp->keys + i * kp->nw;
        int pnucl = getnuc(x, 0), nnucl = getnuc(x, K1 - 1);
        uint64_t pre[MAXW] = {0, 0, 0, 0}, suf[MAXW] = {0, 0, 0, 0};
        for (int t = 0; t < K; ++t) { orc_setnuc(pre, t, getnuc(x, t)); orc_setnuc(suf, t, getnuc(x, t + 1)); }
        int mn; uint64_t idx = canon_idx(mk, pre, K, &mn);
        out[idx] |= (uint8_t)(1u << (mn ? nnucl : 7 - nnucl));
        idx = canon_idx(mk, suf, K, &mn);
        out[idx] |= (uint8_t)(1u << (mn ? pnucl + 4 : 7 - (pnucl + 4)));
    }
}

/* coverage array in MPHF order + histogram (stages/construction.cpp:404-418: hist[cov-1] += 2) */
void orc_coverage(const kset_t *kp, const mphf_t *mkp, uint32_t *out) {
    memset(out, 0, (size_t)kp->n * 4);
    for (int64_t i = 0; i < kp->n; ++i) out[orc_mphf_lookup(mkp, kp->keys + i * kp->nw)] = kp->counts[i];
}
int64_t orc_histogram(const uint32_t *cov, int64_t n, uint64_t *hist, int64_t cap) {
    int64_t maxcov = 0;
    for (int64_t i = 0; i < n; ++i) if (cov[i] > maxcov) maxcov = cov[i];
    if (!hist) return maxcov;
    memset(hist, 0, (size_t)cap * 8);
    for (int64_t i = 0; i < n; ++i) if (cov[i] && cov[i] - 1 < cap) hist[cov[i] - 1] += 2;
    return maxcov;
}

/* ------------------------------------------------------------------------------------------------
 * Unitigs: UnbranchingPathExtractor (assembly_graph/construction/debruijn_graph_constructor.hpp:184-410).
 * Sequences are kept as 0..3 byte strings.
 * ---------------------------------------------------------------------------------------------- */
typedef struct { uint8_t *s; int64_t len; } seq_t;
typedef struct { seq_t *v; int64_t n, cap; } seqvec_t;
static void sv_push(seqvec_t *sv, const uint8_t *s, int64_t len) {
    if (sv->n == sv->cap) { sv->cap = sv->cap ? sv->cap * 2 : 64; sv->v = (seq_t *)realloc(sv->v, (size_t)sv->cap * sizeof(seq_t)); }
    sv->v[sv->n].s = (uint8_t *)malloc((size_t)len ? (size_t)len : 1); memcpy(sv->v[sv->n].s, s, (size_t)len); sv->v[sv->n].len = len; sv->n++;
}
static uint8_t inv_byte(uint8_t a) { uint8_t r = 0; for (int i = 0; i < 8; ++i) { r = (uint8_t)((r << 1) | (a & 1)); a >>= 1; } return r; } /* inout_mask.hpp:18-27 */

typedef struct { const mphf_t *m; uint8_t *masks; int K; } gctx_t;
/* get_value(kwh): InvertableStoring::get_value (storing_traits.hpp:44-51) with InOutMask::conjugate */
static uint8_t g_mask(const gctx_t *g, const uint64_t *km) {
    int mn; uint64_t idx = canon_idx(g->m, km, g->K, &mn);
    return mn ? g->masks[idx] : inv_byte(g->masks[idx]);
}
static const int8_t UNIQ[16] = {-1, 0, 1, -1, 2, -1, -1, -1, 3, -1, -1, -1, -1, -1, -1, -1};   /* inout_mask.hpp:61-81 */
static int m_unique_out(uint8_t m) { return UNIQ[m & 15]; }
static int m_unique_in(uint8_t m) { return UNIQ[m >> 4]; }
static int m_is_junction(uint8_t m) { return m_unique_out(m) < 0 || m_unique_in(m) < 0; }

typedef struct { uint8_t *b; int64_t n, cap; } bytes_t;
static void by_push(bytes_t *b, uint8_t c) { if (b->n == b->cap) { b->cap = b->cap ? b->cap * 2 : 256; b->b = (uint8_t *)realloc(b->b, (size_t)b->cap); } b->b[b->n++] = c; }

/* ConstructSequenceWithEdge, :264-273 (edge = (start k-mer, start<<c)) ; loop guard `edge != initial` */
static void construct_seq(const gctx_t *g, const uint64_t *start, int c, bytes_t *out) {
    int K = g->K, nw = nwords(K);
    out->n = 0;
    for (int i = 0; i < K; ++i) by_push(out, (uint8_t)getnuc(start, i));
    by_push(out, (uint8_t)c);
    uint64_t es[MAXW], ee[MAXW], is[MAXW], ie[MAXW];
    memcpy(es, start, 8 * nw); memcpy(ee, start, 8 * nw); kmer_shl(ee, K, c);
    memcpy(is, es, 8 * nw); memcpy(ie, ee, 8 * nw);
    for (;;) {
        uint8_t m = g_mask(g, ee);                               /* StepRightIfPossible(DeEdge&), :247-255 */
        int uo = m_unique_out(m), ui = m_unique_in(m);
        if (uo < 0 || ui < 0) break;
        memcpy(es, ee, 8 * nw); kmer_shl(ee, K, uo);
        if (memcmp(es, is, 8 * nw) == 0 && memcmp(ee, ie, 8 * nw) == 0) break;
        by_push(out, (uint8_t)getnuc(ee, K - 1));
    }
}
static void seq_rc(const uint8_t *s, int64_t n, uint8_t *o) { for (int64_t i = 0; i < n; ++i) o[i] = (uint8_t)(3 - s[n - 1 - i]); }
static int seq_less(const uint8_t *a, int64_t na, const uint8_t *b, int64_t nb) {    /* Sequence::operator<, sequence.hpp:592-600 */
    int64_t s = na < nb ? na : nb;
    for (int64_t i = 0; i < s; ++i) if (a[i] != b[i]) return a[i] < b[i];
    return na < nb;
}
static void seq_to_kmer(const uint8_t *s, int K, uint64_t *w) { for (int i = 0; i < nwords(K); ++i) w[i] = 0; for (int i = 0; i < K; ++i) orc_setnuc(w, i, s[i]); }

/* RemoveSequence, kmer_extension_index.hpp:131-138 */
static void remove_seq(gctx_t *g, const uint8_t *s, int64_t n) {
    uint64_t km[MAXW]; seq_to_kmer(s, g->K, km);
    int mn; g->masks[canon_idx(g->m, km, g->K, &mn)] = 0;
    for (int64_t pos = g->K; pos < n; ++pos) { kmer_shl(km, g->K, s[pos]); g->masks[canon_idx(g->m, km, g->K, &mn)] = 0; }
}

/* ------------------------------------------------------------------------------------------------
 * Early tip clipper: EarlyTipClipperProcessor (assembly_graph/construction/early_simplification.hpp:38-162) +
 * RemoveInconsistentForwardLinks (:21-36). Works on the mask array in place. Iteration order of the reference with one
 * thread: k-mers in final_kmers order (index_.kmer_begin), each as seq then !seq (:69-71).
 *   snapshot == 0 : the reference's sequential semantics (walks see the removals made so far)
 *   snapshot != 0 : every walk sees the masks as they were before the clipper started (what a data-parallel
 *                   implementation computes); tests assert both give the same array.
 * Returns the number of removed k-mers (ClipTips' return value, :57,102-103); *n_tipped / *n_clipped = the two INFO counters.
 * ---------------------------------------------------------------------------------------------- */
static int etc_find_forward(const gctx_t *g, const uint64_t *first, int64_t bound, uint64_t *idx_out /* bound+1 */) {
    /* FindForward, :115-125. returns the tip size (0 = not a tip) and the canonical indices of its vertices */
    int K = g->K, nw = nwords(K);
    uint64_t kh[MAXW]; memcpy(kh, first, 8 * nw);
    int64_t n = 0; int mn;
    for (;;) {
        uint8_t m = g_mask(g, kh);
        if (!(n < bound && m_unique_in(m) >= 0 && m_unique_out(m) >= 0)) break;
        idx_out[n++] = canon_idx(g->m, kh, K, &mn);
        kmer_shl(kh, K, m_unique_out(m));
    }
    idx_out[n++] = canon_idx(g->m, kh, K, &mn);
    uint8_t m = g_mask(g, kh);
    if (m_unique_in(m) < 0 || (m & 15) != 0) return 0;
    return (int)n;
}
int64_t orc_early_tip_clip(const kset_t *km, const mphf_t *mk, uint8_t *masks, int64_t length_bound, int snapshot,
                           int64_t *n_tipped, int64_t *n_clipped) {
    int K = km->K, nw = km->nw;
    uint8_t *view = masks;
    if (snapshot) { view = (uint8_t *)malloc((size_t)(km->n ? km->n : 1)); memcpy(view, masks, (size_t)km->n); }
    gctx_t g; g.m = mk; g.K = K; g.masks = view;
    uint64_t *tips[4];
    for (int c = 0; c < 4; ++c) tips[c] = (uint64_t *)malloc((size_t)(length_bound + 2) * 8);
    uint64_t *tj = NULL; int64_t ntj = 0, ctj = 0;          /* tipped junctions: k-mer words */
    int64_t removed = 0;
    for (int64_t i = 0; i < km->n; ++i) {
        for (int o = 0; o < 2; ++o) {
            uint64_t kh[MAXW];
            if (o == 0) memcpy(kh, km->keys + i * nw, 8 * nw); else orc_rc(km->keys + i * nw, K, kh);
            uint8_t m = g_mask(&g, kh);
            if (__builtin_popcount(m & 15) < 2) continue;
            /* RemoveForward, :143-155 */
            size_t max = 0; int sz[4] = {0, 0, 0, 0};
            for (int c = 0; c < 4; ++c) {
                if (!(m & (1 << c))) continue;
                uint64_t khc[MAXW]; memcpy(khc, kh, 8 * nw); kmer_shl(khc, K, c);
                sz[c] = etc_find_forward(&g, khc, length_bound, tips[c]);
                size_t len = sz[c] ? (size_t)sz[c] : (size_t)-1;
                if (len > max) max = len;
            }
            int64_t rem = 0;
            for (int c = 0; c < 4; ++c)
                if ((size_t)sz[c] < max) { for (int t = 0; t < sz[c]; ++t) masks[tips[c][t]] = 0; rem += sz[c]; }   /* IsolateVertex */
            removed += rem;
            if (rem) {
                if (ntj == ctj) { ctj = ctj ? 2 * ctj : 64; tj = (uint64_t *)realloc(tj, (size_t)ctj * nw * 8); }
                memcpy(tj + ntj * nw, kh, 8 * nw); ++ntj;
            }
        }
    }
    /* RemoveInconsistentForwardLinks over the tipped junctions, :21-36,88-96 (sees the final masks) */
    g.masks = masks;
    int64_t clipped = 0;
    for (int64_t j = 0; j < ntj; ++j) {
        const uint64_t *kh = tj + j * nw;
        uint8_t m = g_mask(&g, kh);
        int mn; uint64_t idx = canon_idx(mk, kh, K, &mn);
        for (int c = 0; c < 4; ++c) {
            if (!(m & (1 << c))) continue;
            uint64_t nx[MAXW]; memcpy(nx, kh, 8 * nw); kmer_shl(nx, K, c);
            if (!(g_mask(&g, nx) & (1 << (4 + getnuc(kh, 0))))) { masks[idx] &= (uint8_t)~(1u << (mn ? c : 7 - c)); ++clipped; }
        }
    }
    if (n_tipped) *n_tipped = ntj;
    if (n_clipped) *n_clipped = clipped;
    for (int c = 0; c < 4; ++c) free(tips[c]);
    free(tj);
    if (snapshot) free(view);
    return removed;
}

/* ------------------------------------------------------------------------------------------------
 * Early low-complexity (poly A/T) clipper of the RNA pipeline: EarlyLowComplexityClipperProcessor
 * (assembly_graph/construction/early_simplification.hpp:164-347; phase EarlyATClipper, stages/construction.cpp:317-340,448:
 * at_ratio 0.8, min_length 10, max_length 200). Works on the mask array in place; k-mers are visited in final_kmers order, each
 * as seq then !seq (:190-191, :277-278).
 *   RemoveATEdges (:185-256): collects (junction k-mer, c) edges of length 1 on a read-only pass, then deletes each link once.
 *   RemoveATTips  (:269-334): from every dead end with a unique incoming edge walk back to the junction; low-complexity tips
 *                 are isolated on the fly, then the phantom links of their roots are removed (RemoveInconsistentForwardLinks).
 *   snapshot != 0 : the tip decisions see the masks as they were after RemoveATEdges (what a data-parallel implementation
 *                   computes); tests assert both modes give the same array.
 * out4 = { edges collected (RemoveATEdges' return value), links removed, k-mers removed (RemoveATTips' return value), clipped tips }
 * ---------------------------------------------------------------------------------------------- */
static int almost_equals_d(double a, double b) {      /* gtest FloatingPoint<double>::AlmostEquals, 4 ULPs (math/xmath.h:283-299) */
    if (isnan(a) || isnan(b)) return 0;
    uint64_t x, y; memcpy(&x, &a, 8); memcpy(&y, &b, 8);
    const uint64_t sign = 0x8000000000000000ull;
    uint64_t bx = (x & sign) ? (~x + 1) : (sign | x), by = (y & sign) ? (~y + 1) : (sign | y);
    uint64_t d = bx >= by ? bx - by : by - bx;
    return d <= 4;
}
static int math_ls(double a, double b) { return !almost_equals_d(a, b) && a < b; }    /* math::ls, xmath.h:300-306 */
static void kmer_shr(uint64_t *w, int K, int c) {          /* kwh >> c: c enters at position 0, the last nucleotide drops (rtseq.hpp:569-588) */
    int nw = nwords(K);
    uint64_t carry = (uint64_t)c;
    for (int j = 0; j < nw; ++j) { uint64_t nc = w[j] >> 62; w[j] = (w[j] << 2) | carry; carry = nc; }
    int bits = 2 * K - 64 * (nw - 1);
    if (bits < 64) w[nw - 1] &= (1ULL << bits) - 1;
}
void orc_early_at_clip(const kset_t *km, const mphf_t *mk, uint8_t *masks, double ratio, int64_t min_len, int64_t max_len, int snapshot, int64_t *out4) {
    int K = km->K, nw = km->nw;
    gctx_t g; g.m = mk; g.K = K; g.masks = masks;
    /* ---- RemoveATEdges */
    uint64_t *ek = NULL; uint8_t *ec = NULL; int64_t ne = 0, ce = 0;
    double thr = (double)K * ratio;
    for (int64_t i = 0; i < km->n; ++i) {
        for (int o = 0; o < 2; ++o) {
            uint64_t kh[MAXW];
            if (o == 0) memcpy(kh, km->keys + i * nw, 8 * nw); else orc_rc(km->keys + i * nw, K, kh);
            uint8_t m = g_mask(&g, kh);
            if (!m_is_junction(m)) continue;
            size_t counts[4] = {0, 0, 0, 0};
            for (int p = 0; p < K; ++p) counts[getnuc(kh, p)]++;
            size_t curm = counts[0];
            for (int c = 1; c < 4; ++c) if (counts[c] > curm) curm = counts[c];
            if (math_ls((double)curm, thr)) continue;
            for (int c = 0; c < 4; ++c) {
                if (!(m & (1 << c))) continue;
                uint64_t nx[MAXW]; memcpy(nx, kh, 8 * nw); kmer_shl(nx, K, c);
                uint8_t mn = g_mask(&g, nx);
                if (!m_is_junction(mn) && (mn & 15) != 0) continue;       /* next must be a junction or a dead end */
                if (ne == ce) { ce = ce ? 2 * ce : 64; ek = (uint64_t *)realloc(ek, (size_t)ce * nw * 8); ec = (uint8_t *)realloc(ec, (size_t)ce); }
                memcpy(ek + ne * nw, kh, 8 * nw); ec[ne] = (uint8_t)c; ++ne;
            }
        }
    }
    int64_t removed_links = 0;
    for (int64_t e = 0; e < ne; ++e) {
        const uint64_t *kh = ek + e * nw; int c = ec[e];
        if (!(g_mask(&g, kh) & (1 << c))) continue;
        uint64_t nx[MAXW]; memcpy(nx, kh, 8 * nw); kmer_shl(nx, K, c);
        int mn; uint64_t idx = canon_idx(mk, kh, K, &mn);
        masks[idx] &= (uint8_t)~(1u << (mn ? c : 7 - c));                                  /* DeleteOutgoing(kh, c) */
        int first = getnuc(kh, 0);
        idx = canon_idx(mk, nx, K, &mn);
        masks[idx] &= (uint8_t)~(1u << (mn ? 4 + first : 7 - (4 + first)));               /* DeleteIncoming(next, kh[0]) */
        removed_links += 2;
    }
    free(ek); free(ec);
    /* ---- RemoveATTips */
    uint8_t *view = masks;
    if (snapshot) { view = (uint8_t *)malloc((size_t)(km->n ? km->n : 1)); memcpy(view, masks, (size_t)km->n); }
    g.masks = view;
    uint64_t *tip = (uint64_t *)malloc((size_t)(max_len + 1) * 8);
    uint64_t *roots = NULL; int64_t nr = 0, cr = 0;
    int64_t removed_kmers = 0;
    for (int64_t i = 0; i < km->n; ++i) {
        for (int o = 0; o < 2; ++o) {
            uint64_t kh[MAXW];
            if (o == 0) memcpy(kh, km->keys + i * nw, 8 * nw); else orc_rc(km->keys + i * nw, K, kh);
            uint8_t m = g_mask(&g, kh);
            if ((m & 15) != 0 || m_unique_in(m) < 0) continue;             /* IsDeadEnd && CheckUniqueIncoming */
            size_t counts[4] = {0, 0, 0, 0};
            int64_t tsz = 0; int mn;
            do {
                tip[tsz++] = canon_idx(mk, kh, K, &mn);
                counts[getnuc(kh, K - 1)]++;
                kmer_shr(kh, K, m_unique_in(g_mask(&g, kh)));                /* GetUniqueIncoming (8 -> garbage when not unique: the loop then stops) */
            } while (tsz < max_len && !m_is_junction(g_mask(&g, kh)));
            uint8_t mr = g_mask(&g, kh);
            if ((mr >> 4) == 0 || !m_is_junction(mr)) continue;            /* dead start, or the tip is too long */
            for (int64_t p = tsz - 1; p < min_len; ++p) counts[getnuc(kh, (int)(K - 1 - p))]++;
            size_t curm = counts[0];
            for (int c = 1; c < 4; ++c) if (counts[c] > curm) curm = counts[c];
            double thr2 = (double)(tsz > min_len ? tsz : min_len) * ratio;
            if (math_ls((double)curm, thr2)) continue;
            if (nr == cr) { cr = cr ? 2 * cr : 64; roots = (uint64_t *)realloc(roots, (size_t)cr * nw * 8); }
            memcpy(roots + nr * nw, kh, 8 * nw); ++nr;
            removed_kmers += tsz;
            for (int64_t t = 0; t < tsz; ++t) masks[tip[t]] = 0;            /* IsolateVertex */
        }
    }
    g.masks = masks;
    int64_t clipped = 0;
    for (int64_t j = 0; j < nr; ++j) {                                       /* RemoveInconsistentForwardLinks, :21-36 */
        const uint64_t *kh = roots + j * nw;
        uint8_t m = g_mask(&g, kh);
        int mn; uint64_t idx = canon_idx(mk, kh, K, &mn);
        for (int c = 0; c < 4; ++c) {
            if (!(m & (1 << c))) continue;
            uint64_t nx[MAXW]; memcpy(nx, kh, 8 * nw); kmer_shl(nx, K, c);
            if (!(g_mask(&g, nx) & (1 << (4 + getnuc(kh, 0))))) { masks[idx] &= (uint8_t)~(1u << (mn ? c : 7 - c)); ++clipped; }
        }
    }
    free(tip); free(roots);
    if (snapshot) free(view);
    if (out4) { out4[0] = ne; out4[1] = removed_links; out4[2] = removed_kmers; out4[3] = clipped; }
}

typedef struct { seqvec_t seqs; } unitigs_t;

unitigs_t *orc_unitigs(const kset_t *km, const mphf_t *mk, const uint8_t *masks_in, int keep_loops) {
    int K = km->K, nw = km->nw;
    gctx_t g; g.m = mk; g.K = K;
    g.masks = (uint8_t *)malloc((size_t)(km->n ? km->n : 1)); memcpy(g.masks, masks_in, (size_t)km->n);
    unitigs_t *u = (unitigs_t *)calloc(1, sizeof(unitigs_t));
    bytes_t buf = {0, 0, 0};
    uint8_t *rcb = NULL; int64_t rccap = 0;
    /* ExtractUnbranchingPaths / CalculateSequences :295-314, AddStartDeEdges :214-235 ; order = final_kmers order */
    for (int64_t i = 0; i < km->n; ++i) {
        const uint64_t *kh = km->keys + i * nw;
        uint8_t ext = g_mask(&g, kh);
        if (!m_is_junction(ext)) continue;
        uint64_t inv[MAXW]; orc_rc(kh, K, inv);
        for (int side = 0; side < 2; ++side) {
            const uint64_t *st = side ? inv : kh;
            /* `if (!kh_inv.is_minimal())` :230 is always taken: kh is the stored minimal form and k is odd (gbuilder.cpp:125) */
            uint8_t m = side ? g_mask(&g, inv) : ext;
            for (int c = 0; c < 4; ++c) {
                if (!(m & (1u << c))) continue;
                construct_seq(&g, st, c, &buf);
                if (buf.n > rccap) { rccap = buf.n * 2; rcb = (uint8_t *)realloc(rcb, (size_t)rccap); }
                seq_rc(buf.b, buf.n, rcb);
                if (seq_less(buf.b, buf.n, rcb, buf.n)) continue;   /* `if (s < !s) continue;` :307 */
                sv_push(&u->seqs, buf.b, buf.n);
            }
        }
    }
    if (keep_loops) {
        /* RemoveSequences, kmer_extension_index.hpp:141-147 */
        int64_t npaths = u->seqs.n;
        for (int64_t i = 0; i < npaths; ++i) {
            seq_t *s = &u->seqs.v[i];
            if (s->len > rccap) { rccap = s->len * 2; rcb = (uint8_t *)realloc(rcb, (size_t)rccap); }
            remove_seq(&g, s->s, s->len);
            seq_rc(s->s, s->len, rcb);
            remove_seq(&g, rcb, s->len);
        }
        /* CollectLoops :359-397 */
        for (int64_t i = 0; i < km->n; ++i) {
            const uint64_t *kh = km->keys + i * nw;
            if (m_is_junction(g_mask(&g, kh))) continue;
            /* FindMinimalKMerInLoop :252-262 */
            uint64_t minimal[MAXW], cur[MAXW], tmp[MAXW];
            orc_rc(kh, K, tmp);
            memcpy(minimal, kmer_nuc_less(kh, tmp, K) ? kh : tmp, 8 * nw);
            memcpy(cur, kh, 8 * nw);
            { uint8_t m = g_mask(&g, cur); if (m_unique_out(m) >= 0 && m_unique_in(m) >= 0) kmer_shl(cur, K, m_unique_out(m)); }
            while (memcmp(cur, kh, 8 * nw) != 0) {
                if (kmer_nuc_less(cur, minimal, K)) memcpy(minimal, cur, 8 * nw);
                orc_rc(cur, K, tmp);
                if (kmer_nuc_less(tmp, minimal, K)) memcpy(minimal, tmp, 8 * nw);
                uint8_t m = g_mask(&g, cur);
                if (m_unique_out(m) >= 0 && m_unique_in(m) >= 0) kmer_shl(cur, K, m_unique_out(m));
            }
            /* ConstructLoopFromVertex :283-293 */
            construct_seq(&g, minimal, m_unique_out(g_mask(&g, minimal)), &buf);
            int64_t n = buf.n;
            uint8_t *s = (uint8_t *)malloc((size_t)n); memcpy(s, buf.b, (size_t)n);
            int64_t split = -1;
            {
                int K1 = K + 1;
                uint64_t a[MAXW] = {0, 0, 0, 0}, b[MAXW];
                for (int t = 0; t < K1 - 1; ++t) orc_setnuc(a, t + 1, s[t]);   /* s.start(K+1) >> 'A' */
                for (int64_t p = K; p < n; ++p) {
                    kmer_shl(a, K1, s[p]);
                    orc_rc(a, K1, b);
                    if (memcmp(a, b, 8 * (size_t)nwords(K1)) == 0) { split = p - K; break; }
                }
            }
            /* pieces: SplitLoop :276-281 */
            int64_t npieces = split >= 0 ? 2 : 1;
            for (int64_t pc = 0; pc < npieces; ++pc) {
                uint8_t *q; int64_t qn;
                if (split < 0) { q = s; qn = n; }
                else if (pc == 0) { q = s + split; qn = K + 1; }
                else {
                    /* s.Subseq(pos+1, size-K) + s.Subseq(0, pos+K) */
                    int64_t n1 = (n - K) - (split + 1), n2 = split + K;
                    q = (uint8_t *)malloc((size_t)(n1 + n2 > 0 ? n1 + n2 : 1));
                    memcpy(q, s + split + 1, (size_t)n1); memcpy(q + n1, s, (size_t)n2); qn = n1 + n2;
                }
                if (qn > rccap) { rccap = qn * 2; rcb = (uint8_t *)realloc(rcb, (size_t)rccap); }
                seq_rc(q, qn, rcb);
                if (seq_less(q, qn, rcb, qn)) sv_push(&u->seqs, rcb, qn); else sv_push(&u->seqs, q, qn);
                remove_seq(&g, q, qn);
                remove_seq(&g, rcb, qn);
                if (split >= 0 && pc == 1) free(q);
            }
            free(s);
        }
    }
    free(buf.b); free(rcb); free(g.masks);
    return u;
}
int64_t orc_unitigs_n(const unitigs_t *u) { return u->seqs.n; }
int64_t orc_unitig_len(const unitigs_t *u, int64_t i) { return u->seqs.v[i].len; }
const uint8_t *orc_unitig_seq(const unitigs_t *u, int64_t i) { return u->seqs.v[i].s; }
void orc_unitigs_free(unitigs_t *u) { if (!u) return; for (int64_t i = 0; i < u->seqs.n; ++i) free(u->seqs.v[i].s); free(u->seqs.v); free(u); }

/* ------------------------------------------------------------------------------------------------
 * Graph linking + coverage + GFA text: FastGraphFromSequencesConstructor::ConstructGraph
 * (debruijn_graph_constructor.hpp:412-568), GraphCoverageFiller (graph_support/coverage_filling.hpp:52-70),
 * GFAWriter (io/graph/gfa_writer.cpp:19-116), ids: graph_core.hpp:233 (ID_BIAS=3), :459-479, :514-531.
 * ---------------------------------------------------------------------------------------------- */
typedef struct { uint64_t hm; uint64_t edge; } linkrec_t;
static uint64_t lr_edge_and_mask(const linkrec_t *r) { return (r->edge << 2) | (r->hm & 3); }
static int cmp_link(const void *a, const void *b) {
    const linkrec_t *x = (const linkrec_t *)a, *y = (const linkrec_t *)b;
    uint64_t hx = x->hm >> 2, hy = y->hm >> 2;
    if (hx != hy) return hx < hy ? -1 : 1;
    uint64_t ex = lr_edge_and_mask(x), ey = lr_edge_and_mask(y);
    if (ex != ey) return ex < ey ? -1 : 1;
    return 0;
}
static const linkrec_t *g_recs;
static int cmp_group(const void *a, const void *b) {
    uint64_t x = lr_edge_and_mask(&g_recs[*(const int64_t *)a]), y = lr_edge_and_mask(&g_recs[*(const int64_t *)b]);
    return x < y ? -1 : (x > y ? 1 : 0);
}
static int cmp_u64(const void *a, const void *b) { uint64_t x = *(const uint64_t *)a, y = *(const uint64_t *)b; return x < y ? -1 : (x > y ? 1 : 0); }

typedef struct { char *b; int64_t n, cap; } text_t;
static void tx_put(text_t *t, const char *s, int64_t n) {
    if (t->n + n + 1 > t->cap) { t->cap = (t->n + n + 1) * 2; t->b = (char *)realloc(t->b, (size_t)t->cap); }
    memcpy(t->b + t->n, s, (size_t)n); t->n += n; t->b[t->n] = 0;
}
static void tx_printf_u(text_t *t, uint64_t v) { char tmp[32]; int n = snprintf(tmp, sizeof tmp, "%llu", (unsigned long long)v); tx_put(t, tmp, n); }

/* returns malloc'ed NUL-terminated GFA text. mkp/cov may be NULL (then DP/KC are 0). version e.g. "SPAdes-4.3.0-dev" */
char *orc_gfa(const unitigs_t *u, const mphf_t *mk, const mphf_t *mkp, const uint32_t *cov, const char *version, int64_t *out_len) {
    int K = mk->K;
    int64_t E = u->seqs.n;
    const uint64_t MINID = 3;
    linkrec_t *recs = (linkrec_t *)malloc((size_t)(2 * E ? 2 * E : 1) * sizeof(linkrec_t));
    uint8_t *selfc = (uint8_t *)calloc((size_t)(E ? E : 1), 1);
    uint8_t *rcb = NULL; int64_t rccap = 0;
    for (int64_t i = 0; i < E; ++i) {
        const seq_t *s = &u->seqs.v[i];
        if (s->len > rccap) { rccap = s->len * 2; rcb = (uint8_t *)realloc(rcb, (size_t)rccap); }
        seq_rc(s->s, s->len, rcb);
        selfc[i] = memcmp(rcb, s->s, (size_t)s->len) == 0;
        uint64_t edge = MINID + 2 * (uint64_t)i;
        uint64_t km[MAXW], kr[MAXW];
        seq_to_kmer(s->s, K, km); orc_rc(km, K, kr);                       /* StartLink :455-462 */
        if (kmer_nuc_less(km, kr, K)) recs[2 * i].hm = (orc_mphf_lookup(mk, km) << 2) | 1; else recs[2 * i].hm = (orc_mphf_lookup(mk, kr) << 2) | 2 | 1;
        recs[2 * i].edge = edge;
        if (!selfc[i]) {                                                   /* EndLink :464-471 */
            seq_to_kmer(s->s + s->len - K, K, km); orc_rc(km, K, kr);
            if (kmer_nuc_less(km, kr, K)) recs[2 * i + 1].hm = (orc_mphf_lookup(mk, km) << 2); else recs[2 * i + 1].hm = (orc_mphf_lookup(mk, kr) << 2) | 2;
            recs[2 * i + 1].edge = edge;
        } else { recs[2 * i + 1].hm = (uint64_t)-1; recs[2 * i + 1].edge = 0; }   /* LinkRecord() :447-448 */
    }
    qsort(recs, (size_t)(2 * E), sizeof(linkrec_t), cmp_link);
    int64_t *groups = (int64_t *)malloc((size_t)(2 * E ? 2 * E : 1) * 8); int64_t V = 0;
    for (int64_t i = 0; i < 2 * E; ++i) {
        if (i == 0 || (recs[i].hm >> 2) != (recs[i - 1].hm >> 2)) {
            int invalid = (recs[i].hm + 1 == 0) && recs[i].edge == 0;
            if (!invalid) groups[V++] = i;
        }
    }
    g_recs = recs;
    qsort(groups, (size_t)V, 8, cmp_group);
    /* per (vertex, side) outgoing lists; side 0 = v, side 1 = conjugate(v) */
    uint64_t **outl = (uint64_t **)calloc((size_t)(2 * V ? 2 * V : 1), sizeof(uint64_t *));
    int *outn = (int *)calloc((size_t)(2 * V ? 2 * V : 1), sizeof(int));
    for (int64_t vn = 0; vn < V; ++vn) {
        int64_t i = groups[vn];
        for (int64_t j = i; j < 2 * E && (recs[j].hm >> 2) == (recs[i].hm >> 2); ++j) {
            int is_start = (int)(recs[j].hm & 1), is_rc = (int)((recs[j].hm >> 1) & 1);
            uint64_t e = recs[j].edge;
            int64_t ei = (int64_t)((e - MINID) / 2);
            uint64_t ce = selfc[ei] ? e : e + 1;
            /* LinkEdge :486-496 + ConstructionHelper::Link{Outgoing,Incoming}Edge (core/construction_helper.hpp:87-97) */
            int side = is_rc ? 1 : 0;            /* v1 = is_rc ? conj(v) : v */
            int tgt; uint64_t add;
            if (is_start) { tgt = side; add = e; } else { tgt = side ^ 1; add = ce; }
            int64_t slot = 2 * vn + tgt;
            outl[slot] = (uint64_t *)realloc(outl[slot], (size_t)(outn[slot] + 1) * 8);
            outl[slot][outn[slot]++] = add;
        }
        qsort(outl[2 * vn], (size_t)outn[2 * vn], 8, cmp_u64);            /* PairedVertex::AddOutgoingEdge keeps ids sorted, graph_core.hpp:206-209 */
        qsort(outl[2 * vn + 1], (size_t)outn[2 * vn + 1], 8, cmp_u64);
    }
    text_t t = {0, 0, 0};
    tx_put(&t, "H\tsp:Z:", 7); tx_put(&t, version, (int64_t)strlen(version)); tx_put(&t, "\n", 1);
    int K1 = K + 1;
    for (int64_t i = 0; i < E; ++i) {
        const seq_t *s = &u->seqs.v[i];
        uint32_t raw = 0;
        if (mkp && cov) {
            uint64_t a[MAXW] = {0, 0, 0, 0}, b[MAXW];
            for (int q = 0; q < K1 - 1; ++q) orc_setnuc(a, q + 1, s->s[q]);
            for (int64_t p = K1 - 1; p < s->len; ++p) {
                kmer_shl(a, K1, s->s[p]);
                if (orc_is_minimal(a, K1)) raw += cov[orc_mphf_lookup(mkp, a)]; else { orc_rc(a, K1, b); raw += cov[orc_mphf_lookup(mkp, b)]; }
            }
        }
        tx_put(&t, "S\t", 2); tx_printf_u(&t, MINID + 2 * (uint64_t)i); tx_put(&t, "\t", 1);
        { char *tmp = (char *)malloc((size_t)s->len + 1); for (int64_t q = 0; q < s->len; ++q) tmp[q] = "ACGT"[s->s[q]]; tx_put(&t, tmp, s->len); free(tmp); }
        double c = (double)raw / (double)(s->len - K);                      /* coverage(): core/coverage.hpp:59-61 */
        char tmp[64]; int n = snprintf(tmp, sizeof tmp, "\tDP:f:%g\tKC:i:%u\n", (double)(float)c, raw);   /* gfa_writer.cpp:19-26 */
        tx_put(&t, tmp, n);
    }
    for (int64_t vn = 0; vn < V; ++vn) {                                     /* WriteVertexLinks, gfa_writer.cpp:77-91 */
        for (int a = 0; a < outn[2 * vn + 1]; ++a) {
            uint64_t x = outl[2 * vn + 1][a];
            int64_t xi = (int64_t)((x - MINID) / 2);
            uint64_t inc = selfc[xi] ? x : (((x - MINID) & 1) ? x - 1 : x + 1);        /* conjugate */
            for (int b = 0; b < outn[2 * vn]; ++b) {
                uint64_t oe = outl[2 * vn][b];
                uint64_t ends[2] = {inc, oe};
                tx_put(&t, "L", 1);
                for (int q = 0; q < 2; ++q) {
                    uint64_t e = ends[q]; int64_t ei = (int64_t)((e - MINID) / 2);
                    int canon = selfc[ei] || (((e - MINID) & 1) == 0);
                    tx_put(&t, "\t", 1); tx_printf_u(&t, MINID + 2 * (uint64_t)ei); tx_put(&t, canon ? "\t+" : "\t-", 2);
                }
                char tmp[32]; int n = snprintf(tmp, sizeof tmp, "\t%dM\n", K); tx_put(&t, tmp, n);
            }
        }
    }
    for (int64_t i = 0; i < 2 * V; ++i) free(outl[i]);
    free(outl); free(outn); free(groups); free(recs); free(selfc); free(rcb);
    if (out_len) *out_len = t.n;
    if (!t.b) { t.b = (char *)calloc(1, 1); }
    return t.b;
}
/* ------------------------------------------------------------------------------------------------
 * Coverage pre-filter (SURVEY 8f-3): stages/construction.cpp:167-198 (CoverageFilter phase).
 *   hash      adt/cyclichash.hpp:187-259  SymmetricCyclicHash<NDNASeqHash>(n = K): value = fwd + rvs,
 *             fwd = XOR_p rol(h(s_p), n-1-p), rvs = XOR_p rol(h(3 - s_p), p); character hashes :24-27 (seed 0 -> :51 is the identity).
 *             KmerSequenceProcessor (kmer_index/kmer_counting.hpp:38-52) rolls it from the hash of 'A' + the first K-1 bases; the
 *             rolled value equals the direct one (the update :250-256 is exact), which is what is restated here.
 *   HLL       adt/hll.hpp:16-77: 2^24 one-byte registers, id = top 24 bits, rho = clz of the low 40 bits (as a 64-bit word) - 24 + 1
 *             (64 - 24 + 1 when they are zero); cardinality :50-64 (sequential double sum in register order), upper bound = 1.1 x.
 *             EstimateCardinalityUpperBound (kmer_counting.hpp:215-249) adds every window that passes the IsMinimal filter of reads and
 *             their reverse complements; the hash is symmetric, so that is every window of the forward reads.
 *   CQF       adt/cqf.hpp:28-37: qbits = max(7, ceil(log2(maxn))) + 1, key = hash & (2^(qbits+8) - 1): an EXACT multiset of keys
 *             (ext/src/gqf/gqf.c:1430-1477: range = nslots << remainder bits = 2^key_bits). FillCoverageHistogram + CQFProcessor
 *             (kmer_counting.hpp:96-121,251-282) stop counting a key at the threshold; only ">= threshold" is ever asked.
 *             A self-RC window passes the filter in the read and in its reverse complement: counted twice (as in coverage, SURVEY 0.6).
 *   filter    io/reads/coverage_filtering_read_wrapper.hpp:37-72: multiplicities of ALL windows of a read, nth_element at size/2,
 *             keep the read iff that element >= threshold; reads shorter than K are dropped (median 0).
 * out_stats: [0] cardinality upper bound (size_t(1.1 * cardinality)), [1] key bits, [2] distinct keys, [3] reads kept.
 * ---------------------------------------------------------------------------------------------- */
static const uint64_t CYC_H[4] = {0x3c8bfbb395c60474ULL, 0x3193c18562a02b4cULL, 0x20323ed082572324ULL, 0x295549f54be24456ULL};
static inline uint64_t rol64(uint64_t x, unsigned s) { s &= 63; return s ? (x << s) | (x >> (64 - s)) : x; }
uint64_t orc_cyclic_hash(const uint64_t *seq, int64_t pos, int K) {
    uint64_t fwd = 0, rvs = 0;
    for (int i = 0; i < K; ++i) fwd = rol64(fwd, 1) ^ CYC_H[getnuc(seq, (int)pos + i)];
    for (int i = 0; i < K; ++i) rvs = rol64(rvs, 1) ^ CYC_H[3 - getnuc(seq, (int)pos + K - 1 - i)];
    return fwd + rvs;
}
typedef struct { uint64_t key; uint32_t cnt; } cfent_t;
static int cfent_cmp(const void *a, const void *b) { uint64_t x = *(const uint64_t *)a, y = *(const uint64_t *)b; return x < y ? -1 : x > y; }
void orc_cov_filter(const uint64_t *words, const uint64_t *offs, const uint32_t *lens, int64_t nreads, int K, unsigned thr,
                    uint8_t *keep, uint64_t *out_stats) {
    /* 1. HLL */
    const unsigned P = 24;
    const uint64_t m = 1ull << P, mask = (m - 1) << (64 - P);
    uint8_t *reg = (uint8_t *)calloc(m, 1);
    size_t nwin = 0;
    for (int64_t r = 0; r < nreads; ++r) if ((int)lens[r] >= K) nwin += (size_t)lens[r] - K + 1;
    uint64_t *keys = (uint64_t *)malloc((nwin * 2 + 1) * 8);
    size_t nk = 0;
    for (int64_t r = 0; r < nreads; ++r) {
        const int L = (int)lens[r];
        if (L < K) continue;
        const uint64_t *s = words + offs[r];
        for (int j = 0; j + K <= L; ++j) {
            const uint64_t d = orc_cyclic_hash(s, j, K);
            const size_t id = (d & mask) >> (64 - P);
            const uint64_t low = d & ~mask;
            const uint8_t rho = (uint8_t)((low == 0 ? 64 : __builtin_clzll(low)) - P + 1);
            if (reg[id] < rho) reg[id] = rho;
            keys[nk++] = d;
            /* self-RC window: minimal in both streams */
            uint64_t km[MAXW] = {0, 0, 0, 0}, rc[MAXW];
            for (int i = 0; i < K; ++i) orc_setnuc(km, i, getnuc(s, j + i));
            orc_rc(km, K, rc);
            if (memcmp(km, rc, (size_t)nwords(K) * 8) == 0) keys[nk++] = d;
        }
    }
    const double alpha = 0.7213 / (1.0 + 1.079 / (double)m);
    double res = alpha * (double)m * (double)m, E = 0.0;
    uint64_t zeros = 0;
    for (uint64_t i = 0; i < m; ++i) { E += exp2(-(double)reg[i]); zeros += reg[i] == 0; }
    res /= E;
    if (res <= 5.0 * (double)m / 2 && zeros > 0) res = (double)m * (log((double)m) - log((double)zeros));
    free(reg);
    const size_t maxn = (size_t)(1.1 * res);
    /* 2. CQF geometry + exact key multiset */
    unsigned lg = maxn > 1 ? (unsigned)ceil(log2((double)maxn)) : 0u;
    unsigned qbits = (lg > 7u ? lg : 7u) + 1;
    const unsigned key_bits = qbits + 8;
    const uint64_t range_mask = key_bits >= 64 ? ~0ull : ((1ull << key_bits) - 1);
    for (size_t i = 0; i < nk; ++i) keys[i] &= range_mask;
    qsort(keys, nk, 8, cfent_cmp);
    size_t nd = 0;
    uint32_t *cnt = (uint32_t *)malloc((nk + 1) * 4);
    for (size_t i = 0; i < nk;) { size_t j = i; while (j < nk && keys[j] == keys[i]) ++j; keys[nd] = keys[i]; cnt[nd] = (uint32_t)(j - i); ++nd; i = j; }
    /* 3. filter */
    uint64_t kept = 0;
    uint32_t *ml = NULL; size_t mlcap = 0;
    for (int64_t r = 0; r < nreads; ++r) {
        const int L = (int)lens[r];
        keep[r] = 0;
        if (L < K) { if (thr == 0) { keep[r] = 1; ++kept; } continue; }
        const uint64_t *s = words + offs[r];
        const size_t w = (size_t)(L - K + 1);
        if (w > mlcap) { mlcap = w * 2; ml = (uint32_t *)realloc(ml, mlcap * 4); }
        for (size_t j = 0; j < w; ++j) {
            const uint64_t d = orc_cyclic_hash(s, (int64_t)j, K) & range_mask;
            size_t lo = 0, hi = nd;
            while (lo < hi) { size_t mid = (lo + hi) >> 1; if (keys[mid] < d) lo = mid + 1; else hi = mid; }
            uint32_t c = (lo < nd && keys[lo] == d) ? cnt[lo] : 0;
            ml[j] = c < thr ? c : thr;                     /* the filter stops counting at the threshold */
        }
        /* nth_element at w/2 == element w/2 of the sorted array */
        size_t below = 0;
        for (size_t j = 0; j < w; ++j) below += ml[j] < thr;
        if (below <= w / 2) { keep[r] = 1; ++kept; }
    }
    free(ml); free(cnt); free(keys);
    out_stats[0] = maxn; out_stats[1] = key_bits; out_stats[2] = nd; out_stats[3] = kept;
}

void orc_free(void *p) { free(p); }
