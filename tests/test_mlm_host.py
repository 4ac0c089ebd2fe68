"""CPU: masked-language-model batches (batch_tokenize_mlm / bsq_tokenize_mlm, kernel K8) without a device.

The entry points are declared, exported and bound; the integer thresholds and the argument checks are pinned; the
vectorised reference of the rule (tests/mlm_reference.py, what the GPU tests compare with) is checked against a scalar
restatement built on the oracle's C Philox, and its statistics (selected share, 80/10/10 split, uniform random ids,
specials never selected) on about 10^6 residues."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from bioseq_b200 import capi, consumers
from oracle import oracle
from oracle.oracle import OracleTokenizer
from helpers import gen
from mlm_reference import mlm as reference_mlm, philox4x32_10 as np_philox

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TWO32 = 1 << 32


def test_mlm_entry_points_declared_exported_and_bound():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bsq.h")).read(), flags=re.S)
    assert re.search(r"typedef\s+struct\s+bsq_mlm\s*\{", src)
    L = C.CDLL(capi.LIB_PATH)
    for name in ("bsq_tokenize_mlm", "bsq_tokenize_varlen_mlm"):
        assert re.search(r"\b" + name + r"\s*\(", src), f"{name} not declared in include/bsq.h"
        assert hasattr(L, name) and name in capi.EXPORTS
        assert getattr(capi.lib(), name).argtypes is not None
    # struct bsq_mlm: 7 eight-byte fields
    assert C.sizeof(capi.MLMDesc) == 56


def test_thresholds_known_answers():
    assert consumers._mlm_thresholds() == (644245094, 515396075, 579820584)
    assert consumers._mlm_thresholds(0.15, 0.8, 0.1) == (644245094, 515396075, 579820584)
    assert consumers._mlm_thresholds(0.0) == (0, 0, 0)
    assert consumers._mlm_thresholds(1.0) == (TWO32, math.floor(TWO32 * 0.8), math.floor(TWO32 * (0.8 + 0.1)))
    assert consumers._mlm_thresholds(1.0, 1.0, 0.0) == (TWO32, TWO32, TWO32)
    assert consumers._mlm_thresholds(0.5, 0.0, 0.0) == (TWO32 // 2, 0, 0)
    # t_random never passes t_select
    ts, tm, tr = consumers._mlm_thresholds(0.3, 0.6, 0.4)
    assert tm <= tr <= ts


@pytest.mark.parametrize("args", [(-0.01, 0.8, 0.1), (1.01, 0.8, 0.1), (float("nan"), 0.8, 0.1), (0.15, -0.1, 0.1),
                                  (0.15, 0.8, -0.1), (0.15, 0.8, 0.3), (0.15, float("nan"), 0.1)])
def test_thresholds_errors(args):
    with pytest.raises(ValueError):
        consumers._mlm_thresholds(*args)


def desc(key="PROTEIN", bos=True, eos=True, pad=True):
    return capi.tokenizer(key, eos=eos, bos=bos, padchar=pad)


@pytest.mark.parametrize("destchar,limit", [("B", 255), ("b", 127), ("h", 32767), ("H", 32767), ("i", 2 ** 31 - 1),
                                            ("l", 2 ** 31 - 1), ("f", 2 ** 24), ("d", 2 ** 31 - 1)])
def test_mask_token_range(destchar, limit):
    t = desc()
    kw = dict(maskfrac=0.15, mask_prob=0.8, random_prob=0.1, ignore_index=-100, seed=0, seq_index_base=0)
    assert consumers._mlm_desc(t, destchar, mask_token=limit, **kw).mask_id == limit
    assert consumers._mlm_desc(t, destchar, mask_token=0, **kw).mask_id == 0
    for bad in (limit + 1, -1):
        with pytest.raises(ValueError, match="mask_token"):
            consumers._mlm_desc(t, destchar, mask_token=bad, **kw)


def test_mlm_desc_defaults_and_errors():
    kw = dict(maskfrac=0.15, mask_prob=0.8, random_prob=0.1, seed=5, seq_index_base=7)
    d = consumers._mlm_desc(desc(), "B", mask_token=None, ignore_index=-100, **kw)
    assert (d.mask_id, d.ignore_index, d.seed, d.seq_index_base) == (23, -100, 5, 7)  # PROTEIN pbeos: 20 + 3
    assert (d.t_select, d.t_mask, d.t_random) == (644245094, 515396075, 579820584)
    # BYTES: alphabet_size 256 + specials does not fit 'B' -> an explicit token is needed
    with pytest.raises(ValueError, match="mask_token"):
        consumers._mlm_desc(desc("BYTES", False, False, False), "B", mask_token=None, ignore_index=-100, **kw)
    assert consumers._mlm_desc(desc("BYTES"), "i", mask_token=None, ignore_index=-100, **kw).mask_id == 259
    for bad in (2 ** 63, -(2 ** 63) - 1):
        with pytest.raises(ValueError, match="int64"):
            consumers._mlm_desc(desc(), "B", mask_token=None, ignore_index=bad, **kw)
    assert consumers._mlm_desc(desc(), "B", mask_token=None, ignore_index=-(2 ** 63), **kw).ignore_index == -(2 ** 63)
    with pytest.raises(ValueError, match="integers"):
        consumers._mlm_desc(desc(), "B", mask_token=1.5, ignore_index=-100, **kw)


def test_argument_errors_before_any_device_work():
    # every ValueError of batch_tokenize_mlm is raised before the batch is staged (no device is touched here)
    from bioseq_b200 import cbioseq
    tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    batch = (np.frombuffer(b"ACDE", np.uint8).copy(), np.array([0, 4], np.int64))
    capi.lib().bsq_launch_count_reset()
    for kw in (dict(maskfrac=1.5), dict(mask_prob=0.95, random_prob=0.1), dict(random_prob=-1.0), dict(mask_token=256),
               dict(destchar="b", mask_token=128), dict(ignore_index=2 ** 64), dict(varlen=True, padlen=64),
               dict(destchar="z")):
        with pytest.raises(ValueError):
            consumers.batch_tokenize_mlm(tok, batch, **{"padlen": 16, **kw})
    with pytest.raises(ValueError):  # BYTES + 'B': alphabet_size() does not fit a byte
        consumers.batch_tokenize_mlm(cbioseq.Tokenizer("BYTES"), batch, padlen=16)
    assert capi.lib().bsq_launch_count() == 0


def test_c_abi_rejects_bad_arguments():
    t = desc()
    L = capi.lib()
    good = capi.mlm_desc(0, 0, (100, 50, 60), 23, -100)
    cases = [capi.mlm_desc(0, 0, (TWO32 + 1, 0, 0), 23, -100), capi.mlm_desc(0, 0, (100, 70, 60), 23, -100),
             capi.mlm_desc(0, 0, (100, 50, 101), 23, -100), capi.mlm_desc(0, 0, (100, 50, 60), -1, -100),
             capi.mlm_desc(0, 0, (100, 50, 60), 256, -100)]
    for m in cases:
        assert L.bsq_tokenize_mlm(0, None, None, None, 1, 16, C.byref(t), capi.I8, C.byref(m), None, None) == capi.ERR_ARG
        assert L.bsq_tokenize_varlen_mlm(0, None, None, None, 1, C.byref(t), capi.I8, C.byref(m), None, None, None) == capi.ERR_ARG
    m16 = capi.mlm_desc(0, 0, (100, 50, 60), 32768, -100)
    assert L.bsq_tokenize_mlm(0, None, None, None, 1, 16, C.byref(t), capi.I16, C.byref(m16), None, None) == capi.ERR_ARG
    mf = capi.mlm_desc(0, 0, (100, 50, 60), 2 ** 24 + 1, -100)
    assert L.bsq_tokenize_mlm(0, None, None, None, 1, 16, C.byref(t), capi.F32, C.byref(mf), None, None) == capi.ERR_ARG
    assert L.bsq_tokenize_mlm(0, None, None, None, 1, 16, C.byref(t), capi.I8, None, None, None) == capi.ERR_ARG
    assert L.bsq_tokenize_mlm(0, None, None, None, 1, 16, C.byref(t), 9, C.byref(good), None, None) == capi.ERR_ARG


# ------------------------------------------------------------------------------------------------------------------
def restate(tokens, offs, bos, nchars, thresholds, mask_id, ignore, seed, base):
    """The rule of include/bsq.h, written again from the text with numpy and the oracle's Philox block function."""
    ts, tm, tr = thresholds
    inputs = tokens.copy()
    labels = np.full(tokens.shape, ignore, np.int64)
    key = (seed & 0xFFFFFFFF, seed >> 32)
    for i in range(offs.size - 1):
        g = base + i
        for j in range(int(offs[i + 1] - offs[i])):
            u = int(oracle.philox4x32_10((g & 0xFFFFFFFF, g >> 32, j // 4, 1), key)[j % 4])
            col = bos + j
            if u >= ts:
                continue
            labels[i, col] = int(tokens[i, col])
            if u < tm:
                inputs[i, col] = mask_id
            elif u < tr:
                w = int(oracle.philox4x32_10((g & 0xFFFFFFFF, g >> 32, j // 4, 2), key)[j % 4])
                inputs[i, col] = (w * nchars) >> 32
    return inputs, labels


@pytest.mark.parametrize("flags", [(True, True, True), (False, False, False), (True, False, True), (False, True, False)])
@pytest.mark.parametrize("destchar", ["B", "i", "f"])
def test_reference_matches_scalar_restatement(flags, destchar):
    bos, eos, pad = flags
    orc = OracleTokenizer("PROTEIN", bos=bos, eos=eos, padchar=pad)
    buf, offs = gen(11, 30, 0, 70, b"ACDEFGHIKLMNPQRSTVWYXBZ*")
    padlen = 72
    toks = orc.batch_tokenize((buf, offs), padlen=padlen, destchar=destchar, batch_first=True)
    th = consumers._mlm_thresholds(0.3, 0.5, 0.3)  # large random share: the second stream is exercised
    seed, base = 0x1234_5678_9ABC_DEF0, 2 ** 32 + 5
    got_in, got_lab = reference_mlm(toks, offs, bos, orc.nchars(), th, 21, -7, seed, base)
    want_in, want_lab = restate(toks, offs, int(bos), orc.nchars(), th, 21, -7, seed, base)
    assert np.array_equal(got_lab, want_lab)
    assert got_in.dtype == toks.dtype and np.array_equal(got_in, want_in)
    sel = got_lab != -7
    assert sel.any() and (got_in == 21).any() and ((got_in != toks) & (got_in != 21)).any()


def test_vectorised_philox_matches_the_oracle():
    rng = np.random.default_rng(1)
    ctr = rng.integers(0, 2 ** 32, size=(4, 200), dtype=np.uint64)
    key = (0x9ABCDEF0, 0x12345678)
    got = np_philox(*ctr, *key)
    for i in range(200):
        want = oracle.philox4x32_10(ctr[:, i], key)
        assert [int(w[i]) for w in got] == [int(x) for x in want]


def test_known_philox_streams_are_disjoint_from_augmentation():
    # K7 draws from counter word 3 = 0; the mask from 1 and 2: the same (seed, g, block) gives three different blocks
    a = oracle.philox4x32_10((5, 0, 0, 0), (9, 0))
    b = oracle.philox4x32_10((5, 0, 0, 1), (9, 0))
    c = oracle.philox4x32_10((5, 0, 0, 2), (9, 0))
    assert not np.array_equal(a, b) and not np.array_equal(b, c)


@pytest.fixture(scope="module")
def big():
    orc = OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    buf, offs = gen(21, 2000, 400, 600, b"ACDEFGHIKLMNPQRSTVWY")
    toks = orc.batch_tokenize((buf, offs), padlen=602, destchar="B", batch_first=True)
    return orc, buf, offs, toks


def _residue_mask(offs, padlen, bos):
    lens = np.diff(offs)
    cols = np.arange(padlen)[None, :]
    return (cols >= bos) & (cols < bos + lens[:, None])


def _within(x, n, p, sigmas=5.0):
    return abs(x - n * p) <= sigmas * math.sqrt(n * p * (1 - p))


def test_statistics(big):
    orc, buf, offs, toks = big
    res = _residue_mask(offs, toks.shape[1], 1)
    nres = int(res.sum())
    assert nres > 900_000
    inputs, labels = reference_mlm(toks, offs, 1, orc.nchars(), consumers._mlm_thresholds(), orc.alphabet_size(), -100, 3, 0)
    sel = labels != -100
    assert not (sel & ~res).any()                 # specials and padding are never selected
    assert np.array_equal(labels[sel], toks[sel].astype(np.int64))
    assert np.array_equal(inputs[~sel], toks[~sel])
    nsel = int(sel.sum())
    assert _within(nsel, nres, 0.15)
    masked = int((inputs[sel] == orc.alphabet_size()).sum())
    changed = int(((inputs[sel] != toks[sel]) & (inputs[sel] != orc.alphabet_size())).sum())
    assert _within(masked, nsel, 0.8)
    # a random id equals the original 1 time in 20 (residues uniform over the 20 amino acids)
    assert _within(changed, nsel, 0.1 * 19 / 20)
    assert _within(nsel - masked - changed, nsel, 0.1 + 0.1 / 20)


def test_random_ids_uniform(big):
    scipy_stats = pytest.importorskip("scipy.stats")
    orc, buf, offs, toks = big
    inputs, labels = reference_mlm(toks, offs, 1, orc.nchars(), consumers._mlm_thresholds(0.15, 0.0, 1.0), 99, -100, 4, 0)
    ids = inputs[labels != -100].astype(np.int64)
    assert ids.size > 100_000 and ids.min() >= 0 and ids.max() < orc.nchars()
    counts = np.bincount(ids, minlength=orc.nchars())
    assert scipy_stats.chisquare(counts).pvalue > 1e-4
    # BYTES: 256 residue ids
    ob = OracleTokenizer("BYTES")
    t2 = ob.batch_tokenize((buf, offs), padlen=600, destchar="i", batch_first=True)
    in2, lab2 = reference_mlm(t2, offs, 0, ob.nchars(), consumers._mlm_thresholds(0.5, 0.0, 1.0), 300, -100, 4, 0)
    c2 = np.bincount(in2[lab2 != -100].astype(np.int64), minlength=256)
    assert c2.size == 256 and scipy_stats.chisquare(c2).pvalue > 1e-4


def test_all_selected_and_none_selected(big):
    orc, buf, offs, toks = big
    res = _residue_mask(offs, toks.shape[1], 1)
    inputs, labels = reference_mlm(toks, offs, 1, orc.nchars(), consumers._mlm_thresholds(1.0, 1.0, 0.0), 23, -100, 1, 0)
    assert (inputs[res] == 23).all() and np.array_equal(inputs[~res], toks[~res])
    assert np.array_equal(labels[res], toks[res].astype(np.int64)) and (labels[~res] == -100).all()
    inputs, labels = reference_mlm(toks, offs, 1, orc.nchars(), consumers._mlm_thresholds(0.0), 23, -100, 1, 0)
    assert np.array_equal(inputs, toks) and (labels == -100).all()


def test_shift_invariance(big):
    orc, buf, offs, toks = big
    th = consumers._mlm_thresholds()
    full_in, full_lab = reference_mlm(toks, offs, 1, orc.nchars(), th, 23, -100, 77, 0)
    for a in (1, 999, 1500):
        part_in, part_lab = reference_mlm(toks[a:], offs[a:], 1, orc.nchars(), th, 23, -100, 77, a)
        assert np.array_equal(part_in, full_in[a:]) and np.array_equal(part_lab, full_lab[a:])
    # ... and a different seed or base gives a different mask
    other_in, _ = reference_mlm(toks, offs, 1, orc.nchars(), th, 23, -100, 78, 0)
    assert not np.array_equal(other_in, full_in)
