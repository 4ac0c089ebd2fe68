"""Test infrastructure: a numpy restatement of the reverse-complement rule of include/bsq.h (bsq_revcomp).

``revcomp(bytes, offsets, mode, rc_prob, seed, seq_index_base)`` returns ``(bytes', offsets', flipped)``, vectorised over
the batch.  The coin is word 0 of the vectorised Philox4x32-10 of tests/mlm_reference.py at counter word 3 = 4;
tests/test_revcomp_host.py pins the table to a scalar restatement of the header's pairs and the coin to the oracle's C
Philox.
"""
import math

import numpy as np

from mlm_reference import philox4x32_10

ALWAYS, RANDOM, BOTH = "always", "random", "both"


def table():
    """comp[256]: A<->T, C<->G, R<->Y, K<->M, B<->V, D<->H, U->A, the same in lower case, every other byte to itself."""
    t = np.arange(256, dtype=np.uint8)
    for x, y in ("AT", "CG", "RY", "KM", "BV", "DH"):
        for a, b in ((x, y), (x.lower(), y.lower())):
            t[ord(a)], t[ord(b)] = ord(b), ord(a)
    t[ord("U")], t[ord("u")] = ord("A"), ord("a")
    return t


def gate(rc_prob):
    return 1 << 32 if rc_prob >= 1.0 else math.floor(rc_prob * 2.0 ** 32)


def coins(n, rc_prob, seed=0, seq_index_base=0):
    """flip bits (bool) of sequences 0 .. n-1 in random mode: x0 < gate, x0 = Philox4x32-10 word 0 at (g_lo, g_hi, 0, 4)."""
    if n == 0:
        return np.zeros(0, bool)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    g = (np.int64(seq_index_base) + np.arange(n, dtype=np.int64)).astype(np.uint64)
    x0 = philox4x32_10(g & np.uint64(0xFFFFFFFF), g >> np.uint64(32), 0, 4, seed & 0xFFFFFFFF, seed >> 32)[0]
    return x0.astype(np.uint64) < np.uint64(gate(rc_prob))


def revcomp(buf, offs, mode, rc_prob=0.5, seed=0, seq_index_base=0):
    """The flipped batch: ``(bytes', offsets' (from 0), flipped)`` with 2n sequences in "both" mode."""
    buf = np.asarray(buf, dtype=np.uint8)
    offs = np.asarray(offs, dtype=np.int64)
    n = offs.size - 1
    lens = np.diff(offs)
    if mode == BOTH:
        src = np.concatenate([offs[:-1], offs[:-1]])
        lens = np.concatenate([lens, lens])
        flipped = np.arange(2 * n) >= n
    else:
        src = offs[:-1]
        flipped = np.ones(n, bool) if mode == ALWAYS else coins(n, rc_prob, seed, seq_index_base)
    out_offs = np.zeros(lens.size + 1, dtype=np.int64)
    np.cumsum(lens, out=out_offs[1:])
    total = int(out_offs[-1])
    if total == 0:
        return np.zeros(0, np.uint8), out_offs, flipped
    row = np.repeat(np.arange(lens.size), lens)
    j = np.arange(total, dtype=np.int64) - np.repeat(out_offs[:-1], lens)
    f = flipped[row]
    idx = src[row] + np.where(f, lens[row] - 1 - j, j)
    out = buf[idx]
    out[f] = table()[out[f]]
    return out, out_offs, flipped
