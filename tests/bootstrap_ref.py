"""CPU restatement of the bootstrap resampler (strawberry_b200/csrc/sbq_bootstrap.cuh, DESIGN.md "Bootstrap replicates"), bit for
bit: replicate b of locus l draws N = sum n_i fragments with

    key    = sm64(sm64(sm64(seed ^ 0xD1B54A32D192ED03) + b) + l)
    draw k : h = sm64(key + k), r = umulhi64(h, N)              k = 0 .. N - 1
             row i of the locus with C_i <= r < C_{i+1}         C = exclusive prefix of the locus' counts

resample() is the numpy form (every draw of the batch at once), resample_locus_scalar() the same function in Python ints, one
draw at a time, to cross-check it. sm64 is strawberry_b200.synth._sm64, the restatement of sbq_synth.cuh::sm64."""
import bisect

import numpy as np

from strawberry_b200.synth import _sm64

BOOT_SALT = 0xD1B54A32D192ED03
_M32 = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)
_M64 = (1 << 64) - 1


def umulhi64(a, b):
    """floor(a * b / 2^64) of uint64 arrays, exactly, from 32-bit limbs (every partial product fits 64 bits)."""
    a, b = np.asarray(a, np.uint64), np.asarray(b, np.uint64)
    a0, a1, b0, b1 = a & _M32, a >> _S32, b & _M32, b >> _S32
    with np.errstate(over="ignore"):
        p00, p01, p10, p11 = a0 * b0, a0 * b1, a1 * b0, a1 * b1
        mid = (p00 >> _S32) + (p01 & _M32) + (p10 & _M32)          # < 3 * 2^32
        return p11 + (p01 >> _S32) + (p10 >> _S32) + (mid >> _S32)


def boot_key(seed, replicate, locus):
    with np.errstate(over="ignore"):
        k = _sm64(np.uint64(int(seed) & _M64) ^ np.uint64(BOOT_SALT)) + np.uint64(int(replicate) & _M64)
        return _sm64(_sm64(k) + np.asarray(locus, np.uint64))


def resample(batch, seed, replicate, locus_ids=None):
    """Resampled class counts (int32, one per row of the flat batch) of one replicate. locus_ids: the hash position of every locus
    (default: its index in the batch)."""
    cnt = np.asarray(batch["count"], np.int64)
    lro = np.asarray(batch["loc_row_off"], np.int64)
    C = np.zeros(len(cnt) + 1, np.int64)
    np.cumsum(cnt, out=C[1:])
    base = C[lro]                                  # first draw of every locus
    N = np.diff(base)
    ids = np.arange(len(lro) - 1) if locus_ids is None else np.asarray(locus_ids, np.int64)
    total = int(C[-1])
    out = np.zeros(len(cnt), np.int64)
    step = 1 << 24                                 # bounded memory for large batches
    keys = boot_key(seed, replicate, ids)
    for g0 in range(0, total, step):
        g = np.arange(g0, min(total, g0 + step), dtype=np.int64)
        l = np.searchsorted(base, g, side="right") - 1
        with np.errstate(over="ignore"):
            h = _sm64(keys[l] + (g - base[l]).astype(np.uint64))
        r = umulhi64(h, N[l].astype(np.uint64)).astype(np.int64)
        row = np.searchsorted(C, base[l] + r, side="right") - 1
        out += np.bincount(row, minlength=len(cnt))
    return out.astype(np.int32)


def _sm64_int(x):
    x = (x + 0x9E3779B97F4A7C15) & _M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & _M64
    return x ^ (x >> 31)


def resample_locus_scalar(counts, seed, replicate, locus):
    """The same function for one locus, in Python ints: big-int product for umulhi64, bisect for the row."""
    key = _sm64_int((_sm64_int((_sm64_int((seed & _M64) ^ BOOT_SALT) + replicate) & _M64) + locus) & _M64)
    C = [0]
    for n in counts:
        C.append(C[-1] + int(n))
    N = C[-1]
    out = [0] * len(counts)
    for k in range(N):
        h = _sm64_int((key + k) & _M64)
        out[bisect.bisect_right(C, (h * N) >> 64) - 1] += 1
    return out


def resampled_batch(batch, seed, replicate, locus_ids=None):
    """The batch with its counts replaced by replicate `replicate` (for a fresh solve or the oracle)."""
    b = dict(batch)
    b["count"] = resample(batch, seed, replicate, locus_ids)
    return b
