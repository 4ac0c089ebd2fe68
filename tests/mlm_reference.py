"""Test infrastructure: a numpy restatement of the masked-language-model rule of include/bsq.h (bsq_tokenize_mlm).

It applies the rule to padded batch-first tokens -- for example the oracle's ``OracleTokenizer.batch_tokenize(...,
batch_first=True)`` -- of any element type, and returns the masked inputs and the int64 labels.  The padding-free
expectation is the padded one cut per row.  Philox4x32-10 is vectorised here over all residues at once;
tests/test_mlm_host.py pins it to the oracle's C Philox (itself pinned to the Random123 known-answer vectors) and the
whole rule to a scalar restatement written directly from the header's text.
"""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of counters (c0, c1, c2, c3) (uint32 arrays, broadcast) under key (k0, k1) -> 4 uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & MASK32 for x in (c0, c1, c2, c3)]
    c = list(np.broadcast_arrays(*c))
    k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0 = M0 * c[0]
        p1 = M1 * c[2]
        n0 = (p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0)
        n1 = p1 & MASK32
        n2 = (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1)
        n3 = p0 & MASK32
        c = [n0, n1, n2, n3]
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    return [x.astype(np.uint32) for x in c]


def _store(dtype, values):
    """int64 values as the element type, wrapping like the C stores (int8 <- 200 is -56, uint64 <- -1 is 2^64 - 1)."""
    v = np.asarray(values, dtype=np.int64)
    if np.dtype(dtype).kind == "f":
        return v.astype(dtype)
    return v.astype(dtype, casting="unsafe")


def mlm(tokens, offs, bos, nchars, thresholds, mask_id, ignore_index=-100, seed=0, seq_index_base=0):
    """The rule on padded batch-first ``tokens`` (n, padlen) of the sequences delimited by ``offs``.  Returns
    ``(inputs, labels)``: a masked copy of ``tokens`` and the int64 labels.  ``thresholds``: the integers
    ``(t_select, t_mask, t_random)``."""
    tokens = np.ascontiguousarray(tokens)
    offs = np.asarray(offs, dtype=np.int64)
    n, padlen = tokens.shape
    ts, tm, tr = (int(t) for t in thresholds)
    inputs = tokens.copy()
    labels = np.full((n, padlen), ignore_index, dtype=np.int64)
    lens = np.diff(offs)
    if n == 0 or int(lens.sum()) == 0:
        return inputs, labels
    row = np.repeat(np.arange(n, dtype=np.int64), lens)
    start = np.repeat(np.cumsum(lens) - lens, lens)
    j = np.arange(row.size, dtype=np.int64) - start  # residue index within its row
    col = int(bos) + j
    g = (np.int64(seq_index_base) + row).astype(np.uint64)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    g_lo, g_hi, blk, w = g & MASK32, g >> np.uint64(32), (j >> 2).astype(np.uint64), j & 3
    words = philox4x32_10(g_lo, g_hi, blk, 1, k0, k1)
    u = np.choose(w, words).astype(np.int64)
    sel = u < ts
    r_sel, c_sel, u_sel = row[sel], col[sel], u[sel]
    labels[r_sel, c_sel] = tokens[r_sel, c_sel].astype(np.int64)
    masked = u_sel < tm
    inputs[r_sel[masked], c_sel[masked]] = _store(tokens.dtype, np.full(int(masked.sum()), mask_id))
    rnd = ~masked & (u_sel < tr)
    if rnd.any():
        idx = np.flatnonzero(sel)[rnd]
        rw = philox4x32_10(g_lo[idx], g_hi[idx], blk[idx], 2, k0, k1)
        word = np.choose(w[idx], rw).astype(np.uint64)
        rid = ((word * np.uint64(nchars)) >> np.uint64(32)).astype(np.int64)
        inputs[r_sel[rnd], c_sel[rnd]] = _store(tokens.dtype, rid)
    return inputs, labels
