"""numpy restatement of the tuning rotation T (include/ookd_gpu.h, "Tuning"), independent of the library's C form."""
import math

import numpy as np


def quarter_table():
    """S[j] = round(32767 sin(2 pi j / 1024)), j = 0..256, ties away from zero (all values are >= 0)."""
    return np.array([math.floor(32767 * math.sin(2 * math.pi * j / 1024) + 0.5) for j in range(257)], np.int64)


def cos_sin(k):
    """(c, s) of table phases k (array, 0..1023) by the quadrant rule of the header."""
    S = quarter_table()
    k = np.asarray(k, np.int64)
    q, r = k >> 8, k & 255
    a, b = S[r], S[256 - r]
    c = np.select([q == 0, q == 1, q == 2, q == 3], [b, -a, -b, a])
    s = np.select([q == 0, q == 1, q == 2, q == 3], [a, b, -a, -b])
    return c, s


def tune(iq, step, first_sample=0):
    """SC16Q11 samples (int16, shape (n, 2) or flat interleaved) whose first one is global sample first_sample -> T(x),
    same shape.  phi(n) = low 32 bits of n * step; k = phi >> 22."""
    a = np.asarray(iq, np.int16)
    x = a.reshape(-1, 2).astype(np.int64)
    n = np.arange(x.shape[0], dtype=np.uint64) + np.uint64(first_sample)
    with np.errstate(over="ignore"):
        phi = (n * np.uint64(step)) & np.uint64(0xFFFFFFFF)
    c, s = cos_sin((phi >> np.uint64(22)).astype(np.int64))
    I, Q = x[:, 0], x[:, 1]
    i2 = np.clip((I * c + Q * s + 16384) >> 15, -32768, 32767)
    q2 = np.clip((Q * c - I * s + 16384) >> 15, -32768, 32767)
    return np.stack([i2, q2], -1).astype(np.int16).reshape(a.shape)


def widen(b, fmt):
    """8-bit capture -> its SC16Q11 words (CS8 16 k, CU8 16 v - 2040)."""
    return (16 * np.asarray(b).astype(np.int32) - (0 if fmt == "cs8" else 2040)).astype(np.int16)
