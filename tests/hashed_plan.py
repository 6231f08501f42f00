"""Numpy statement of how the hashed multi-GPU merge (csrc/fuse_hash_peers.cu) splits the key space over the ranks:
samples, splitters and the exact cut of every splitter in every rank's sorted records."""

import numpy as np


def samples_of(keys: np.ndarray, S: int) -> np.ndarray:
    """key[floor(i M / S)] for i < S (empty for M = 0)."""
    m = len(keys)
    return keys[(np.arange(S, dtype=np.int64) * m) // S] if m else np.zeros(0, np.uint64)


def splitters(ranks: list, S: int) -> list:
    """[k_0 = 0, k_1 .. k_{R-1}, k_R = 2^64 - 1]: rank b owns the keys in [k_b, k_{b+1}).  k_b is the smallest key k with
    E(k) >= floor(total b / R) (0 when that target is 0), E(k) = sum over ranks q of floor(j_q(k) M_q / S), j_q(k) = the
    number of q's samples below k.  E only changes at keys s + 1 of a sample s, so those are the candidates."""
    R = len(ranks)
    total = sum(len(k) for k in ranks)
    samp = [samples_of(k, S) for k in ranks]
    cand = np.unique(np.concatenate([s for s in samp if len(s)] + [np.zeros(0, np.uint64)]).astype(np.uint64)) + np.uint64(1)

    def E(k):
        return sum((int(np.searchsorted(s, k, side="left")) * len(q)) // S for s, q in zip(samp, ranks) if len(q))

    e = np.array([E(k) for k in cand], dtype=np.int64)
    out = [np.uint64(0)]
    for b in range(1, R):
        t = total * b // R
        if t == 0:
            out.append(np.uint64(0))
            continue
        hit = np.nonzero(e >= t)[0]
        out.append(cand[hit[0]] if len(hit) else np.uint64(2**64 - 1))
    out.append(np.uint64(2**64 - 1))
    return out


def cut(keys: np.ndarray, key, S: int) -> int:
    """Records of `keys` below `key`, found as the kernel finds it: the samples bound it to a window of fewer than
    ceil(M / S) records, of which only the keys below `key` are counted."""
    m = len(keys)
    if m == 0:
        return 0
    s = samples_of(keys, S)
    j = int(np.searchsorted(s, np.uint64(key), side="left"))
    if j == 0:
        return 0
    lo, hi = (j - 1) * m // S + 1, j * m // S
    assert hi - lo < -(-m // S)
    return lo + int((keys[lo:hi] < np.uint64(key)).sum())


def shares(ranks: list, S: int) -> list:
    """Per owner b, the records it receives from every rank q: (begin, count)."""
    k = splitters(ranks, S)
    R = len(ranks)
    return [[(cut(q, k[b], S), cut(q, k[b + 1], S) - cut(q, k[b], S)) for q in ranks] for b in range(R)]


def share_bound(total: int, R: int, S: int) -> float:
    return total / R + 2 * (total / S + R)
