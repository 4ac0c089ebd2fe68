"""CPU: sequence packing (batch_tokenize_seqpack / bsq_seqpack_plan, kernel K10) without a device.

The library's planner (bucketed best-fit decreasing in C) is checked against tests/seqpack_reference.py, a plain
statement of the rule of include/bsq.h, on random and edge-case lengths; the fill it reaches on protein-like lengths;
and every argument error, raised before anything is staged or launched."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from bioseq_b200 import capi, consumers
from seqpack_reference import plan as reference_plan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_seqpack_entry_points_declared_exported_and_bound():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bsq.h")).read(), flags=re.S)
    L = C.CDLL(capi.LIB_PATH)
    for name in ("bsq_seqpack_plan", "bsq_tokenize_seqpack", "bsq_tokenize_seqpack_mlm"):
        assert re.search(r"\b" + name + r"\s*\(", src), f"{name} not declared in include/bsq.h"
        assert hasattr(L, name) and name in capi.EXPORTS
        assert getattr(capi.lib(), name).argtypes is not None
    import bioseq_b200
    for name in ("batch_tokenize_seqpack", "SeqPackBatch"):
        assert name in bioseq_b200.__all__ and hasattr(bioseq_b200, name)


def offsets_of(lens, lead=0):
    o = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=o[1:])
    return o + lead


def library_plan(lens, k, L, rows=None, lead=0):
    o = offsets_of(lens, lead)
    n = len(lens)
    R, nseg, mx = capi.seqpack_plan(o, n, k, L, rows or 0)
    starts, row_ptr = np.full(n, 7, np.int64), np.full(R + 1, 7, np.int64)
    row_seq, cu = np.full(max(n, 1), 7, np.int64), np.full(nseg + 1, 7, np.int32)
    assert capi.seqpack_plan(o, n, k, L, rows or 0, starts, row_ptr, row_seq, cu) == (R, nseg, mx)
    return dict(R=R, starts=starts, row_ptr=row_ptr, row_seq=row_seq[:row_ptr[-1]], cu_seqlens=cu, max_seqlen=mx)


def assert_same_plan(got, want):
    assert got["R"] == want["R"] and got["max_seqlen"] == want["max_seqlen"]
    for key in ("starts", "row_ptr", "row_seq", "cu_seqlens"):
        assert np.array_equal(got[key], want[key]), key


def check_invariants(p, lens, k, L):
    need = np.asarray(lens, np.int64) + k
    st, R = p["starts"], p["R"]
    placed = need > 0
    assert np.all(st[~placed] == -1) and np.all(st[placed] >= 0)
    cover = np.zeros(R * L, np.int32)
    for i in np.flatnonzero(placed):
        assert st[i] // L == (st[i] + need[i] - 1) // L  # never split across rows
        cover[st[i]:st[i] + need[i]] += 1
    assert cover.max(initial=0) <= 1
    cu = p["cu_seqlens"]
    assert cu[0] == 0 and cu[-1] == R * L and np.all(np.diff(cu) > 0)
    assert p["max_seqlen"] == (int(np.diff(cu).max()) if R else 0)


@pytest.mark.parametrize("k", [0, 1, 2])
@pytest.mark.parametrize("L", [1, 2, 7, 16, 64, 1024])
def test_planner_matches_reference_on_random_lengths(k, L):
    if L <= k:
        return
    rng = np.random.default_rng(1000 * k + L)
    for trial in range(6):
        n = int(rng.integers(0, 300))
        hi = L - k
        lens = rng.integers(0, hi + 1, size=n)
        if trial == 1:
            lens = np.where(rng.random(n) < 0.3, 0, lens)  # zeros
        if trial == 2 and n:
            lens[: n // 3] = hi  # need == L
        got = library_plan(lens, k, L, lead=trial)
        assert_same_plan(got, reference_plan(lens, k, L))
        check_invariants(got, lens, k, L)
        extra = got["R"] + 3
        assert_same_plan(library_plan(lens, k, L, rows=extra), reference_plan(lens, k, L, rows=extra))


def test_planner_edge_cases():
    L = 32
    # n = 0: no rows, or only padding rows
    for rows in (None, 1, 4):
        got = library_plan([], 2, L, rows)
        assert_same_plan(got, reference_plan([], 2, L, rows))
    assert library_plan([], 2, L)["cu_seqlens"].tolist() == [0]
    # every row exactly full: no padding segments
    got = library_plan([30, 14, 14, 6, 6, 6, 6], 2, L)
    assert_same_plan(got, reference_plan([30, 14, 14, 6, 6, 6, 6], 2, L))
    assert got["R"] == 3 and got["cu_seqlens"].size == 8
    # everything in one row
    got = library_plan([3, 0, 5, 1], 1, L)
    assert got["R"] == 1 and got["starts"].tolist() == [6, 12, 0, 10]
    # empty sequences occupy nothing when k = 0
    got = library_plan([0, 4, 0], 0, L)
    assert got["starts"].tolist() == [-1, 0, -1] and got["R"] == 1 and got["row_seq"].tolist() == [1]
    # best fit, not first fit: the 2 goes into row 2 (2 left), not row 0 (3 left, first fit's choice)
    got = library_plan([28, 15, 29, 15, 2], 0, L)
    assert got["starts"].tolist() == [32, 64, 0, 79, 94]
    # very wide rows take the sparse buckets; row widths beyond them still match the reference
    rng = np.random.default_rng(3)
    for L2 in (300_000, 5_000_000):
        lens = rng.integers(0, L2 // 3, size=200)
        assert_same_plan(library_plan(lens, 2, L2), reference_plan(lens, 2, L2))


@pytest.mark.parametrize("W", [None, 100, 1022])
def test_planner_with_crop(W):
    # the planner takes the cropped offsets; the consumer derives them with the crop's host arithmetic
    rng = np.random.default_rng(9)
    lens = rng.integers(0, 3000, size=500)
    o = offsets_of(lens, 11)
    L = 1024
    if W is None:
        lens = np.minimum(lens, L - 2)
        o = offsets_of(lens, 11)
        cropped = o
    else:
        cropped, _ = consumers._crop_host_extent(o, lens.size, W)
    got = library_plan(np.diff(cropped), 2, L)
    assert_same_plan(got, reference_plan(np.minimum(lens, W or L), 2, L))


def lognormal_protein_lengths(n, seed):
    rng = np.random.default_rng(seed)
    return np.clip(np.round(rng.lognormal(np.log(300), 0.8, size=n)), 1, None).astype(np.int64)


def test_fill_on_protein_lengths():
    L, k = 1024, 2
    lens = np.minimum(lognormal_protein_lengths(65_536, 0), L - k)
    p = library_plan(lens, k, L)
    fill = float((lens + k).sum()) / (p["R"] * L)
    assert fill >= 0.99, fill
    check_invariants(p, lens, k, L)


def test_planner_argument_errors():
    o = offsets_of([5, 10, 3])
    lib = capi.lib()
    R, ns, mx = C.c_int64(), C.c_int64(), C.c_int64()
    out = [C.byref(R), C.byref(ns), C.byref(mx)]
    with pytest.raises(ValueError, match=r"seq len \+ bos \+ eos > padlen: 12, vs padlen 11"):
        capi.seqpack_plan(o, 3, 2, 11)
    with pytest.raises(ValueError, match="rows"):
        capi.seqpack_plan(o, 3, 0, 10, rows=1)
    assert capi.seqpack_plan(o, 3, 0, 10, rows=2)[0] == 2
    with pytest.raises(ValueError, match="2\\^31"):
        capi.seqpack_plan(offsets_of([2 ** 20] * 3000), 3000, 0, 2 ** 20)
    with pytest.raises(ValueError, match="2\\^31"):
        capi.seqpack_plan(o, 3, 0, 2 ** 30, rows=2)
    for L in (0, -5):
        assert lib.bsq_seqpack_plan(o.ctypes.data, 3, 0, L, 0, *out, None, None, None, None) == capi.ERR_ARG
    assert lib.bsq_seqpack_plan(None, 3, 0, 16, 0, *out, None, None, None, None) == capi.ERR_ARG
    assert lib.bsq_seqpack_plan(o.ctypes.data, -1, 0, 16, 0, *out, None, None, None, None) == capi.ERR_ARG
    assert lib.bsq_seqpack_plan(o.ctypes.data, 3, 3, 16, 0, *out, None, None, None, None) == capi.ERR_ARG
    assert lib.bsq_seqpack_plan(o.ctypes.data, 3, 0, 16, 0, None, out[1], out[2], None, None, None, None) == capi.ERR_ARG
    buf = np.zeros(64, np.int64)
    p = buf.ctypes.data
    assert lib.bsq_seqpack_plan(o.ctypes.data, 3, 0, 16, 0, *out, p, p, None, p) == capi.ERR_ARG  # some arrays only
    bad = np.array([0, 5, 4], np.int64)
    assert lib.bsq_seqpack_plan(bad.ctypes.data, 2, 0, 16, 0, *out, None, None, None, None) == capi.ERR_ARG
    # n = 0 needs no offsets
    assert lib.bsq_seqpack_plan(None, 0, 2, 16, 0, *out, None, None, None, None) == capi.OK and R.value == 0


def test_kernel_entry_rejects_bad_arguments_without_a_device():
    lib = capi.lib()
    tok = capi.tokenizer("PROTEIN", eos=True, bos=True, padchar=True)
    d = C.c_void_p(16)
    odd = C.c_void_p(17)
    mlm = capi.mlm_desc(0, 0, consumers._mlm_thresholds(), 25, -100)
    assert lib.bsq_tokenize_seqpack(0, None, d, d, C.byref(tok), 0, 0, 4, d, d, d, d) == capi.ERR_ARG  # row_len < 1
    assert lib.bsq_tokenize_seqpack(0, None, d, d, C.byref(tok), 0, 16, -1, d, d, d, d) == capi.ERR_ARG
    assert lib.bsq_tokenize_seqpack(0, None, d, d, C.byref(tok), 9, 16, 4, d, d, d, d) == capi.ERR_ARG  # kind
    assert lib.bsq_tokenize_seqpack(0, None, d, d, None, 0, 16, 4, d, d, d, d) == capi.ERR_ARG
    assert lib.bsq_tokenize_seqpack(0, None, d, d, C.byref(tok), 0, 16, 4, None, d, d, d) == capi.ERR_ARG
    assert lib.bsq_tokenize_seqpack(0, None, d, d, C.byref(tok), 0, 16, 4, d, d, odd, d) == capi.ERR_ARG
    assert lib.bsq_tokenize_seqpack(0, None, d, d, C.byref(tok), 0, 16, 4, d, d, d, None) == capi.ERR_ARG
    assert lib.bsq_tokenize_seqpack(0, None, d, d, C.byref(tok), 0, 2 ** 20, 2 ** 12, d, d, d, d) == capi.ERR_ARG
    assert lib.bsq_tokenize_seqpack(0, None, None, None, C.byref(tok), 0, 16, 0, None, None, None, None) == capi.OK  # nothing
    assert lib.bsq_tokenize_seqpack_mlm(0, None, d, d, C.byref(tok), 0, None, 16, 4, d, d, d, d, d) == capi.ERR_ARG
    assert lib.bsq_tokenize_seqpack_mlm(0, None, d, d, C.byref(tok), 0, C.byref(mlm), 16, 4, d, d, d, d, odd) == capi.ERR_ARG
    bad = capi.mlm_desc(0, 0, (1, 2, 0), 25, -100)  # thresholds out of order
    assert lib.bsq_tokenize_seqpack_mlm(0, None, d, d, C.byref(tok), 0, C.byref(bad), 16, 4, d, d, d, d, d) == capi.ERR_ARG


def test_consumer_argument_errors_before_any_device_work():
    from bioseq_b200 import cbioseq
    tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    batch = (np.frombuffer(b"ACDEFGHIKLMNPQRSTVWY", np.uint8).copy(), np.array([0, 9, 20], np.int64))
    capi.lib().bsq_launch_count_reset()
    bad = (dict(row_len=10), dict(row_len=13, rows=1), dict(row_len=0), dict(row_len=16, rows=0), dict(row_len=2.5),
           dict(row_len=16, rows=1.5), dict(row_len=16, destchar="x"), dict(row_len=16, mlm=True, maskfrac=2.0),
           dict(row_len=16, mlm=True, mask_token=300), dict(row_len=16, crop="middle"), dict(row_len=16, crop="head", crop_len=15),
           dict(row_len=16, crop_len=4), dict(row_len=2 ** 30, rows=2), dict(row_len=2, crop="head"))
    for kw in bad:
        with pytest.raises(ValueError):
            consumers.batch_tokenize_seqpack(tok, batch, **kw)
    # a cropped batch fits where the uncropped one does not
    with pytest.raises(ValueError, match="padlen 8"):
        consumers.batch_tokenize_seqpack(tok, batch, 8)
    assert capi.lib().bsq_launch_count() == 0


def test_dataset_arguments():
    from bioseq_b200 import cbioseq, loaders
    from oracle import oracle
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "x.ff")
        with open(path, "wb") as f:
            f.write(oracle.flatfile_image([b"ACDEFGHIKLMN" * 10, b"ACD"]))
        ff = cbioseq.FlatFile(path)
        tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
        assert loaders.FlatFileDataset(ff, tok, seqpack=True, max_seq_len=64).seqpack
        for kw in (dict(seqpack=True, varlen=True), dict(seqpack=True, cnn=True)):
            with pytest.raises(ValueError):
                loaders.FlatFileDataset(ff, tok, **kw)
