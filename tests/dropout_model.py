"""Host model of the fused dropout mask (include/egc_b200.h, egc_dropout), written from the contract alone: Philox4x32-10
(Salmon, Moraes, Dror, Shaw, "Parallel random numbers: as easy as 1, 2, 3", SC'11; the Random123 constants) in numpy."""
import numpy as np

_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Four uint32 output words for counters (c0, c1, c2, c3) (broadcastable integer arrays) under key (k0, k1)."""
    c = [np.asarray(v, dtype=np.uint64) & _M32 for v in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(int(k0) & 0xFFFFFFFF), np.uint64(int(k1) & 0xFFFFFFFF)
    for r in range(10):
        if r:
            k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _M32, (k1 + np.uint64(0xBB67AE85)) & _M32
        p0 = np.uint64(0xD2511F53) * c[0]                 # < 2^64: exact in uint64
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _M32]
    return [v.astype(np.uint32) for v in c]


def dropout_constants(p):
    """(threshold, scale): from the fp32 p widened to double, keep iff word < floor((1 - p) 2^32), scale = fp32(1 / (1 - p))."""
    keep = 1.0 - float(np.float32(p))
    return min(int(np.floor(keep * 2.0 ** 32)), 2 ** 32 - 1), float(np.float32(1.0 / keep))


def keep_mask(seed, row0, n_rows, n_cols, p):
    """bool [n_rows, n_cols]: element (i, c) is kept, i = local row of a block whose first global row is row0."""
    t, _ = dropout_constants(p)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    nq = (n_cols + 3) // 4
    rows = np.arange(row0, row0 + n_rows, dtype=np.uint64)[:, None]
    q = np.arange(nq, dtype=np.uint64)[None, :]
    words = philox4x32_10(q, rows, 0, 0, seed & 0xFFFFFFFF, seed >> 32)     # word w of group q = column 4q + w
    r = np.stack(words, axis=-1).reshape(n_rows, 4 * nq)[:, :n_cols]
    return r < np.uint32(t)
