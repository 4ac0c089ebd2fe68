"""The k-mer rule of include/bsq.h (bsq_kmer) in numpy, independent of libbsq: codes come from the C oracle's alphabet
tables (oracle.OracleTokenizer(key).lut), k-mers from sliding_window_view with a stride."""
import numpy as np
from numpy.lib.stride_tricks import sliding_window_view

from oracle.oracle import OracleTokenizer


def codes(key):
    """byte -> code of the alphabet, -1 for an invalid byte (bytes >= 0x80 are invalid)."""
    lut = OracleTokenizer(key).lut.astype(np.int64)
    lut[0x80:] = -1
    return lut


def ids(nchars, k, bos, eos, padchar):
    """-> dict(nkmers, unk, bos, eos, pad, vocab_size); bos / eos None when absent."""
    nk = nchars ** k
    unk = nk + nchars
    return dict(nkmers=nk, unk=unk, bos=unk + 1 if bos else None, eos=unk + 1 + bos if eos else None, pad=unk + 1 + bos + eos,
                vocab_size=nk + nchars + 1 + bos + eos + padchar)


def count(n, k, s, single, bos, eos):
    """T(n) in numpy (n: an array of lengths)."""
    n = np.asarray(n, np.int64)
    m = np.where(n >= k, (n - k) // s + 1, 0)
    covered = np.where(m > 0, (m - 1) * s + k, 0)
    return m + (n - covered if single else 0) + bos + eos


def row(c, nchars, k, s, single, idd):
    """The tokens between BOS and EOS of one sequence given as codes c (-1 invalid)."""
    n = c.size
    parts = []
    if n >= k:
        win = sliding_window_view(c, k)[::s]
        val = (np.maximum(win, 0) * nchars ** np.arange(k - 1, -1, -1, dtype=np.int64)).sum(1)
        parts.append(np.where((win < 0).any(1), idd["unk"], val))
        covered = (win.shape[0] - 1) * s + k
    else:
        covered = 0
    if single:
        t = c[covered:]
        parts.append(np.where(t < 0, idd["unk"], idd["nkmers"] + t))
    return np.concatenate(parts).astype(np.int64) if parts else np.zeros(0, np.int64)


def rows(buf, offs, key, k, s, single, bos, eos, padchar=False):
    """Every sequence's full row [BOS] tokens [EOS] as int64 arrays."""
    lut = codes(key)
    nchars = OracleTokenizer(key).nchars()
    idd = ids(nchars, k, bos, eos, padchar)
    out = []
    for i in range(len(offs) - 1):
        c = lut[np.asarray(buf[int(offs[i]):int(offs[i + 1])], np.uint8)]
        r = row(c, nchars, k, s, single, idd)
        out.append(np.concatenate([[idd["bos"]] * bos, r, [idd["eos"]] * eos]).astype(np.int64))
    return out


def padded(buf, offs, key, k, s, single, bos, eos, padchar, padlen):
    """(nseq, padlen) int64: rows, then pad (padchar) or 0."""
    rs = rows(buf, offs, key, k, s, single, bos, eos, padchar)
    fill = ids(OracleTokenizer(key).nchars(), k, bos, eos, padchar)["pad"] if padchar else 0
    out = np.full((len(rs), padlen), fill, np.int64)
    for i, r in enumerate(rs):
        assert r.size <= padlen
        out[i, :r.size] = r
    return out


def varlen(buf, offs, key, k, s, single, bos, eos):
    """(tokens int64, cu_seqlens int32, max_seqlen)."""
    rs = rows(buf, offs, key, k, s, single, bos, eos)
    lens = np.array([r.size for r in rs], np.int64)
    cu = np.zeros(len(rs) + 1, np.int64)
    np.cumsum(lens, out=cu[1:])
    toks = np.concatenate(rs) if rs else np.zeros(0, np.int64)
    return toks, cu.astype(np.int32), int(lens.max()) if lens.size else 0
