"""Test infrastructure: a numpy restatement of the crop rule of include/bsq.h (bsq_crop).

``crop(bytes, offsets, crop_len, random, seed, seq_index_base)`` returns ``(bytes', offsets', starts)``, vectorised over
the batch.  Philox4x32-10 is the vectorised one of tests/mlm_reference.py; tests/test_crop_host.py pins this rule to a
scalar restatement written directly from the header's text in Python integers.
"""
import numpy as np

from mlm_reference import philox4x32_10


def starts(lens, crop_len, random, seed=0, seq_index_base=0):
    """start_i of every sequence (int64): 0 unless random and len_i > crop_len, else floor(d * span / 2^64)."""
    lens = np.asarray(lens, dtype=np.int64)
    out = np.zeros(lens.size, dtype=np.int64)
    if not random:
        return out
    idx = np.flatnonzero(lens > crop_len)
    if idx.size == 0:
        return out
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    g = (np.int64(seq_index_base) + idx.astype(np.int64)).astype(np.uint64)
    x0, x1, _, _ = philox4x32_10(g & np.uint64(0xFFFFFFFF), g >> np.uint64(32), 0, 3, seed & 0xFFFFFFFF, seed >> 32)
    d = x0.astype(np.uint64) | (x1.astype(np.uint64) << np.uint64(32))
    span = (lens[idx] - crop_len + 1).astype(np.uint64)
    # floor(d * span / 2^64) in exact integers: split d into 32-bit halves (span < 2^63)
    d_hi, d_lo = d >> np.uint64(32), d & np.uint64(0xFFFFFFFF)
    s_hi, s_lo = span >> np.uint64(32), span & np.uint64(0xFFFFFFFF)
    ll = d_lo * s_lo
    lh = d_lo * s_hi
    hl = d_hi * s_lo
    hh = d_hi * s_hi
    mid = (ll >> np.uint64(32)) + (lh & np.uint64(0xFFFFFFFF)) + (hl & np.uint64(0xFFFFFFFF))
    out[idx] = (hh + (lh >> np.uint64(32)) + (hl >> np.uint64(32)) + (mid >> np.uint64(32))).astype(np.int64)
    return out


def crop(buf, offs, crop_len, random, seed=0, seq_index_base=0):
    """The cropped batch: ``(bytes', offsets' (from 0), starts)``."""
    buf = np.asarray(buf, dtype=np.uint8)
    offs = np.asarray(offs, dtype=np.int64)
    lens = np.diff(offs)
    st = starts(lens, crop_len, random, seed, seq_index_base)
    kept = np.minimum(lens, crop_len)
    out_offs = np.zeros(lens.size + 1, dtype=np.int64)
    np.cumsum(kept, out=out_offs[1:])
    total = int(out_offs[-1])
    if total == 0:
        return np.zeros(0, np.uint8), out_offs, st
    row = np.repeat(np.arange(lens.size), kept)
    j = np.arange(total, dtype=np.int64) - np.repeat(out_offs[:-1], kept)
    return buf[offs[:-1][row] + st[row] + j], out_offs, st
