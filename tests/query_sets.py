"""Seeded lookup query sets for a k-mer index (test infrastructure): stored keys, keys that are absent but close to stored ones,
and random keys. KMerIndex::seq_idx of an absent key is -1 or the slot of some other key, decided by the key's bucket and the
bitsets stored there, so the absent keys are what tells two implementations of the lookup apart."""
import numpy as np


def _bases(keys, K):
    """[n, nw] packed records -> [n, K] nucleotide codes (nucleotide i at bits 2(i%32) of word i/32)"""
    keys = np.asarray(keys, np.uint64).reshape(len(keys), -1)
    out = np.empty((len(keys), K), np.uint8)
    for i in range(K):
        out[:, i] = (keys[:, i // 32] >> np.uint64(2 * (i % 32))) & np.uint64(3)
    return out


def _pack(bases, nw):
    n, K = bases.shape
    out = np.zeros((n, nw), np.uint64)
    for i in range(K):
        out[:, i // 32] |= bases[:, i].astype(np.uint64) << np.uint64(2 * (i % 32))
    return out


def revcomp_keys(keys, K):
    keys = np.asarray(keys, np.uint64).reshape(len(keys), -1)
    return _pack(3 - _bases(keys, K)[:, ::-1], keys.shape[1])


def key_mask(K, nw):
    """the 2K low bits of an nw-word record"""
    m = np.full(nw, ~np.uint64(0), np.uint64)
    top = 2 * K - 64 * (nw - 1)
    if top < 64:
        m[nw - 1] = (np.uint64(1) << np.uint64(top)) - np.uint64(1)
    return m


def isin_rows(a, b):
    """a[i] is one of the rows of b"""
    a = np.ascontiguousarray(a, np.uint64)
    b = np.ascontiguousarray(b, np.uint64)
    if len(a) == 0 or len(b) == 0:
        return np.zeros(len(a), bool)
    v = np.dtype((np.void, a.shape[1] * 8))
    return np.isin(a.view(v).ravel(), b.view(v).ravel())


def query_set(keys, K, nw, seed, n_derived=None):
    """[m, nw] queries: every stored key; the reverse complement of each stored key that is not itself stored; as many stored keys
    with one base substituted; max(1000, #keys) uniform random keys masked to 2K bits. n_derived < #keys: the reverse complements
    and substitutions come from that many stored keys drawn at random, and as many random keys are added."""
    rng = np.random.default_rng(seed)
    keys = np.asarray(keys, np.uint64).reshape(-1, nw)
    n = len(keys)
    nd = n if n_derived is None else min(n, n_derived)
    parts = [keys]
    if n:
        base = keys if nd == n else keys[np.sort(rng.choice(n, nd, replace=False))]
        rc = revcomp_keys(base, K)
        parts.append(rc[~isin_rows(rc, keys)])
        ns = nd
        src = base[rng.integers(0, nd, ns)]
        b = _bases(src, K)
        pos = rng.integers(0, K, ns)
        rows = np.arange(ns)
        b[rows, pos] = (b[rows, pos] + rng.integers(1, 4, ns).astype(np.uint8)) & 3
        parts.append(_pack(b, nw))
    nr = max(1000, nd)
    rnd = rng.integers(0, 1 << 63, (nr, nw), dtype=np.uint64) << np.uint64(1) | rng.integers(0, 2, (nr, nw), dtype=np.uint64)
    parts.append(rnd & key_mask(K, nw)[None, :])
    return np.ascontiguousarray(np.concatenate(parts), np.uint64)
