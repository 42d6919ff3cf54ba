"""numpy restatement of generate.ratio_split (the counter-based draws of bmf_split_bits), shared by the CPU and GPU
tests.  Pure functions of (seed, global row, column): rows [r0, r1) of an m x n matrix give the same bits whatever the
row range they are computed in."""
import numpy as np
import scipy.sparse as sp

MASK32 = np.uint64(0xFFFFFFFF)


def splitmix64(z):
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def draws(seed, stream, r0, r1, n):
    """u[i - r0, j]: the 32-bit draw of stream `stream` for bit (i, j), i in [r0, r1) (bernoulli_word's scheme)."""
    cw = (n + 63) // 64
    rows = np.arange(r0, r1, dtype=np.uint64)[:, None]
    cols = np.arange(n, dtype=np.uint64)[None, :]
    b = rows * np.uint64(cw * 64) + cols
    with np.errstate(over="ignore"):
        key = np.uint64(seed) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(stream) * np.uint64(0xD1B54A32D192ED03)
        h = splitmix64(key + (b >> np.uint64(1)))
    return np.where(b & np.uint64(1), h >> np.uint64(32), h & MASK32)


def ratio_split_rows(x, r0, n, seed, thresholds, streams=(5, 6)):
    """(train, val ones, val zeros, test ones, test zeros) as bool arrays for the dense rows x = X[r0:r0 + len(x)]."""
    t_v, t_t, q_v, q_t = (np.uint64(t) for t in thresholds)
    x = np.asarray(x) != 0
    r1 = r0 + x.shape[0]
    u1, u0 = draws(seed, streams[0], r0, r1, n), draws(seed, streams[1], r0, r1, n)
    v1 = x & (u1 < t_v)
    s1 = x & ~v1 & (u1 < t_v + t_t)
    v0 = ~x & (u0 < q_v)
    s0 = ~x & ~v0 & (u0 < q_v + q_t)
    return x & ~v1 & ~s1, v1, v0, s1, s0


def stored_csr(ones, zeros):
    """csr int64 of the dense bool arrays: 1 where `ones`, an explicitly stored 0 where `zeros` (sparse addition would
    drop the zeros, so the matrix is built from triplets)."""
    r1, c1 = np.nonzero(ones)
    r0, c0 = np.nonzero(zeros)
    data = np.concatenate([np.ones(len(r1), np.int64), np.zeros(len(r0), np.int64)])
    return sp.coo_matrix((data, (np.concatenate([r1, r0]), np.concatenate([c1, c0]))), shape=ones.shape).tocsr()
