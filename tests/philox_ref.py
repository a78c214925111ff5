"""numpy restatement of the library's counter-based random numbers (csrc/common.cuh): Philox4x32-10 and the keep-mask of the
dense-layer dropout, vectorised over elements.  The tests compare the kernels' masks with this bit for bit."""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c, k):
    """c: 4 uint32 arrays (broadcastable), k: 2 uint32 scalars or arrays -> 4 uint32 arrays"""
    c = [np.asarray(x, dtype=np.uint64) for x in c]
    k0, k1 = np.uint64(k[0]), np.uint64(k[1])
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & M32
        hi1, lo1 = p1 >> np.uint64(32), p1 & M32
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return [x.astype(np.uint32) for x in c]


def drop_threshold(p):
    """floor(p * 2^32) of the float32 p the C ABI receives"""
    return int(np.floor(float(np.float32(p)) * 4294967296.0))


def dropout_words(seed, offset, rows, cols):
    """(rows.size, cols.size) uint32: word (col & 3) of Philox(counter (col >> 2, row, offset_lo, offset_hi),
    key (seed_lo, seed_hi)), the random word that decides element (row, col) of the call at stream position `offset`"""
    rows = np.asarray(rows, dtype=np.uint64).reshape(-1, 1)
    cols = np.asarray(cols, dtype=np.uint64).reshape(1, -1)
    seed, offset = int(seed), int(offset)
    quad = np.arange(int(cols.max()) // 4 + 1, dtype=np.uint64).reshape(1, -1)
    words = philox4x32_10((quad, rows, np.uint64(offset & 0xFFFFFFFF), np.uint64(offset >> 32)),
                          (seed & 0xFFFFFFFF, seed >> 32))
    words = np.stack(np.broadcast_arrays(*words), -1)                      # (rows, quads, 4)
    r = words[:, (cols >> np.uint64(2)).ravel().astype(np.int64), (cols & np.uint64(3)).ravel().astype(np.int64)]
    return r


def keep_of(words, p):
    return words.astype(np.uint64) >= np.uint64(drop_threshold(p))      # p == 1: 2^32 exceeds every word


def dropout_keep(seed, offset, rows, cols, p):
    """keep-mask (rows.size, cols.size) bool: dropout_words >= floor(p * 2^32)"""
    return keep_of(dropout_words(seed, offset, rows, cols), p)
