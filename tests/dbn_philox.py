"""numpy restatement of bb_philox_keep (csrc/bb_train_f64.cuh): the AE_Dropout_BN keep-bits of the fused and the
layer-by-layer fp32 steps, Philox4x32-10 (curand_Philox4x32_10) keyed by (seed, step), counter (column / 4, row, layer,
step), one 32-bit word per column compared with (1 - p) x 2^32."""
import numpy as np

KEEP = (0.5, 0.6, 0.7, 0.8)  # 1 - p of models.py:263-275
WIDTHS = (200, 100, 50, 15)
_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(c, key):
    """c: 4 uint64 arrays holding 32-bit words, key: 2 ints -> 4 uint64 arrays"""
    c = [np.asarray(v, dtype=np.uint64) for v in c]
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for i in range(10):
        p0, p1 = np.uint64(_M0) * c[0], np.uint64(_M1) * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & _MASK, p1 >> np.uint64(32), p1 & _MASK
        c = [hi1 ^ c[1] ^ np.uint64(k0), lo1, hi0 ^ c[3] ^ np.uint64(k1), lo0]
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return c


def philox_masks(seed, step, rows, widths=WIDTHS, row0=0):
    """the 4 boolean keep-masks [rows][width_l] of one step (batch rows row0 .. row0 + rows - 1)"""
    out = []
    key = (seed & 0xFFFFFFFF, ((seed >> 32) ^ (step >> 32)) & 0xFFFFFFFF)
    for l, w in enumerate(widths):
        r, j = np.meshgrid(np.arange(row0, row0 + rows, dtype=np.uint64), np.arange(w, dtype=np.uint64), indexing="ij")
        words = philox4x32_10([j >> np.uint64(2), r, np.full_like(r, l), np.full_like(r, step & 0xFFFFFFFF)], key)
        lane = (j & np.uint64(3)).astype(np.int64)
        v = np.choose(lane, words)
        thr = np.uint64(int(np.float32(KEEP[l]) * 4294967296.0))
        out.append(v < thr)
    return out
