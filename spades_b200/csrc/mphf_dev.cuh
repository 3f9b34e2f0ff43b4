// mphf_dev.cuh -- device-side view of a k-mer set and of its boomphf index (shared by mphf.cu and graph.cu)
#pragma once
#include "sgpu_internal.h"

namespace sg {

static const int kMaxChunks = 128;
struct KeyTable {
    int nchunks;
    int64_t first[kMaxChunks + 1];
    const uint64_t *keys[kMaxChunks];
};

template <int NW>
__device__ __forceinline__ Kmer<NW> table_key(const KeyTable &t, int64_t i) {
    int c = 0, hi = t.nchunks - 1;
    while (c < hi) {                                  // last chunk whose first record index is <= i
        const int mid = (c + hi + 1) >> 1;
        if (t.first[mid] <= i) c = mid; else hi = mid - 1;
    }
    const uint64_t *p = t.keys[c] + (i - t.first[c]) * NW;
    Kmer<NW> k;
#pragma unroll
    for (int q = 0; q < NW; ++q) k.w[q] = p[q];
    return k;
}

struct MphfDev {
    const uint64_t *dom;      // [level*B + b]
    const uint64_t *woff;     // [level*B + b] word offset of the piece in bits
    const uint64_t *starts;   // [B+1]
    uint64_t *bits;
    const uint64_t *ranks;
    uint32_t B;
};

template <int NW>
__device__ __forceinline__ uint64_t level_pos(const MphfDev &m, const Kmer<NW> &k, uint32_t b, int level, uint64_t *word_index) {
    LevelHasher lh(xxh3_128<NW>(k));
    uint64_t h = 0;
    for (int l = 0; l <= level; ++l) h = lh.next();
    const uint64_t pos = mulhi64(h, m.dom[(size_t)level * m.B + b]);
    *word_index = m.woff[(size_t)level * m.B + b] + (pos >> 6);
    return pos;
}

// mphf::lookup (BooPHF.h:465-487) + bitVector::rank (:303-314) + KMerIndex::seq_idx (kmer_index.hpp:88-93)
template <int NW>
__device__ __forceinline__ uint64_t mphf_lookup_dev(const MphfDev &m, const Kmer<NW> &k) {
    const uint32_t b = kmer_bucket<NW>(k, m.B);
    // an empty bucket owns no words (its woff is where the next piece starts) and its mphf was never built: NOT_FOUND
    // (BooPHF.h:425-426,467). A non-empty piece owns >= 8 words; woff has kLevels * B + 1 entries, so b = B - 1 is covered too.
    if (m.woff[b + 1] == m.woff[b]) return ~0ull;
    LevelHasher lh(xxh3_128<NW>(k));
    for (int l = 0; l < kLevels - 1; ++l) {
        const uint64_t h = lh.next();
        const size_t p = (size_t)l * m.B + b;
        const uint64_t pos = mulhi64(h, m.dom[p]);
        const uint64_t wbase = m.woff[p];
        const uint64_t wi = pos >> 6;
        const uint64_t word = m.bits[wbase + wi];
        if ((word >> (pos & 63)) & 1ull) {
            uint64_t r = m.ranks[(wbase >> 3) + (pos >> 9)];
            for (uint64_t w = (pos >> 9) << 3; w < wi; ++w) r += __popcll(m.bits[wbase + w]);
            r += __popcll(word & ((1ull << (pos & 63)) - 1));
            return m.starts[b] + r;
        }
    }
    return ~0ull;
}


MphfDev mphf_dev(const Mphf *m);

inline KeyTable make_table(const KSet *ks) {
    SG_CHECK((int)ks->chunks.size() <= kMaxChunks, 6, "too many result chunks for the key table");
    KeyTable t;
    t.nchunks = (int)ks->chunks.size();
    for (int c = 0; c < t.nchunks; ++c) { t.first[c] = ks->chunks[c].first; t.keys[c] = ks->chunks[c].keys.p; }
    t.first[t.nchunks] = ks->n;
    if (t.nchunks == 0) { t.nchunks = 1; t.first[0] = 0; t.first[1] = 0; t.keys[0] = nullptr; }
    return t;
}

}  // namespace sg
