"""CPU: cropping over-long sequences (crop_packed / crop= / bsq_crop, kernel K9) without a device.

The entry points are declared, exported and bound; the vectorised reference of the rule (tests/crop_reference.py, what
the GPU tests compare with) is checked against a scalar restatement of the header's text in Python integers and the
oracle's C Philox, and its statistics (uniform starts, independence of slicing); every argument error is raised
before anything is staged or launched, and the C ABI rejects bad arguments without a device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from bioseq_b200 import capi, consumers
from oracle import oracle
from helpers import gen
from crop_reference import crop as reference_crop, starts as reference_starts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_crop_entry_points_declared_exported_and_bound():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bsq.h")).read(), flags=re.S)
    L = C.CDLL(capi.LIB_PATH)
    for name in ("bsq_crop", "bsq_crop_extent_device"):
        assert re.search(r"\b" + name + r"\s*\(", src), f"{name} not declared in include/bsq.h"
        assert hasattr(L, name) and name in capi.EXPORTS
        assert getattr(capi.lib(), name).argtypes is not None
    import bioseq_b200
    for name in ("crop_packed", "batch_tokenize_cropped", "CroppedBatch"):
        assert name in bioseq_b200.__all__ and hasattr(bioseq_b200, name)


# ------------------------------------------------------------------------------------------------------------------
def restate(buf, offs, W, random, seed, base):
    """The rule of include/bsq.h written again from its text, one sequence at a time in Python integers."""
    out, out_offs, starts = bytearray(), [0], []
    key = (seed & 0xFFFFFFFF, seed >> 32)
    for i in range(len(offs) - 1):
        length = int(offs[i + 1]) - int(offs[i])
        start = 0
        if random and length > W:
            g = base + i
            x = oracle.philox4x32_10((g & 0xFFFFFFFF, g >> 32, 0, 3), key)
            d = int(x[0]) | (int(x[1]) << 32)
            start = (d * (length - W + 1)) >> 64
        kept = min(length, W)
        out += bytes(buf[int(offs[i]) + start:int(offs[i]) + start + kept])
        out_offs.append(out_offs[-1] + kept)
        starts.append(start)
    return np.frombuffer(bytes(out), np.uint8), np.array(out_offs, np.int64), np.array(starts, np.int64)


@pytest.mark.parametrize("W", [1, 15, 16, 17, 40])
@pytest.mark.parametrize("random", [False, True])
def test_reference_matches_scalar_restatement(W, random):
    buf, offs = gen(5, 120, 0, 3 * W + 2, b"ACDEFGHIKLMNPQRSTVWY")
    offs = offs + 3  # offsets[0] != 0: the rule indexes bytes with the offsets as given
    buf = np.concatenate([np.frombuffer(b"xyz", np.uint8), buf])
    seed, base = 0x1234_5678_9ABC_DEF0, 2 ** 32 + 11
    got = reference_crop(buf, offs, W, random, seed, base)
    want = restate(buf, offs, W, random, seed, base)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
    lens = np.diff(offs)
    assert np.array_equal(np.diff(got[1]), np.minimum(lens, W))
    if not random:
        assert not got[2].any()
    elif (lens > W).sum() > 10:
        assert got[2].any()


def test_known_window_of_a_long_span():
    # spans near 2^40: the product d * span needs all 104 bits
    lens = np.array([2 ** 40 + 12345, 5, 2 ** 40], np.int64)
    got = reference_starts(lens, 7, True, seed=99, seq_index_base=3)
    for i, length in enumerate(lens):
        if length <= 7:
            assert got[i] == 0
            continue
        g = 3 + i
        x = oracle.philox4x32_10((g, 0, 0, 3), (99, 0))
        assert int(got[i]) == ((int(x[0]) | (int(x[1]) << 32)) * (int(length) - 7 + 1)) >> 64


def test_starts_uniform():
    scipy_stats = pytest.importorskip("scipy.stats")
    n, W, span = 1_000_000, 100, 37
    st = reference_starts(np.full(n, W + span - 1, np.int64), W, True, seed=2024)
    assert st.min() >= 0 and st.max() < span
    counts = np.bincount(st, minlength=span)
    assert counts.size == span and scipy_stats.chisquare(counts).pvalue > 1e-4
    # a different seed gives different windows
    assert not np.array_equal(st, reference_starts(np.full(n, W + span - 1, np.int64), W, True, seed=2025))


def test_starts_independent_of_slicing():
    buf, offs = gen(8, 3000, 0, 400, b"ACGT")
    full = reference_crop(buf, offs, 100, True, 77, 0)
    for a, b in ((0, 1), (1, 999), (999, 2500), (2500, 3000)):
        part = reference_crop(buf, offs[a:b + 1], 100, True, 77, a)
        assert np.array_equal(part[2], full[2][a:b])
        assert np.array_equal(part[0], full[0][full[1][a]:full[1][b]])
        assert np.array_equal(part[1], full[1][a:b + 1] - full[1][a])


def test_head_is_truncation_and_long_crop_is_identity():
    buf, offs = gen(9, 200, 0, 90, b"ACDEFGHIKLMNPQRSTVWY")
    b, o, s = reference_crop(buf, offs, 30, False)
    items = [bytes(buf[offs[i]:offs[i + 1]])[:30] for i in range(200)]
    assert b.tobytes() == b"".join(items) and not s.any()
    b, o, s = reference_crop(buf, offs, int(np.diff(offs).max()), True, 5)
    assert np.array_equal(b, buf[offs[0]:offs[-1]]) and np.array_equal(o, offs - offs[0]) and not s.any()


def test_crop_extent_host_arithmetic():
    o, (total, mx) = consumers._crop_host_extent(np.array([3, 10, 10, 40, 41], np.int64), 4, 20)
    assert o.tolist() == [0, 7, 7, 27, 28] and (total, mx) == (28, 20)
    o, ext = consumers._crop_host_extent(np.array([5], np.int64), 0, 20)
    assert o.tolist() == [0] and ext == (0, 0)
    for bad in ([3, 2], [-1, 4]):
        with pytest.raises(ValueError):
            consumers._crop_host_extent(np.array(bad, np.int64), 1, 20)


# ------------------------------------------------------------------------------------------------------------------
def test_crop_spec():
    assert consumers._crop_spec(None, None, 1, 2) is None
    assert consumers._crop_spec(None, None, 1, 2, 10) is None
    assert consumers._crop_spec("head", None, 1, 2, 10) == (False, 10, 1, 2)
    assert consumers._crop_spec("random", 7, 1, 2, 10) == (True, 7, 1, 2)
    assert consumers._crop_spec("random", 7, 1, 2) == (True, 7, 1, 2)
    for args in (("tail", None, 0, 0, 10), (True, None, 0, 0, 10), (None, 5, 0, 0, 10), ("head", 0, 0, 0, 10),
                 ("head", 11, 0, 0, 10), ("random", None, 0, 0, None), ("head", 2.5, 0, 0, 10), ("head", None, 0, 0, 0)):
        with pytest.raises(ValueError):
            consumers._crop_spec(*args)


def test_argument_errors_before_any_device_work():
    # every crop ValueError of the consumers is raised before the batch is staged (no device is touched here)
    from bioseq_b200 import cbioseq
    tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    batch = (np.frombuffer(b"ACDEFGHIK", np.uint8).copy(), np.array([0, 9], np.int64))
    weight = np.zeros((32, 16), np.float32)
    capi.lib().bsq_launch_count_reset()
    bad = (dict(crop="middle"), dict(crop="head", crop_len=0), dict(crop="random", crop_len=-3), dict(crop_len=4),
           dict(crop="head", crop_len=15))  # padlen 16 - bos - eos = 14
    for kw in bad:
        calls = [lambda: consumers.batch_onehot_encode_bcl(tok, batch, 16, **kw),
                 lambda: consumers.batch_tokenize_mlm(tok, batch, 16, **kw),
                 lambda: consumers.batch_embed(tok, batch, weight, 16, **kw)]
        if "crop" in kw:  # (batch_tokenize_cropped crops by default: crop_len alone is valid there)
            calls.append(lambda: consumers.batch_tokenize_cropped(tok, batch, 16, **kw))
        for call in calls:
            with pytest.raises(ValueError):
                call()
    for kw in (dict(crop="middle", crop_len=4), dict(crop="head"), dict(crop="head", crop_len=0), dict(crop_len=4)):
        with pytest.raises(ValueError):
            consumers.batch_tokenize_varlen(tok, batch, **kw)
        with pytest.raises(ValueError):
            consumers.batch_tokenize_mlm(tok, batch, varlen=True, **kw)
    with pytest.raises(ValueError):
        consumers.batch_tokenize_cropped(tok, batch, 16, crop=None)
    with pytest.raises(ValueError):  # a residue mask covers the uncropped batch
        consumers.batch_onehot_encode_bcl(tok, batch, 16, mask=np.ones(9, np.uint8), crop="head")
    with pytest.raises(ValueError):
        consumers.crop_packed(batch[0], batch[1], 4)  # host arrays: crop_packed works on CUDA tensors
    assert capi.lib().bsq_launch_count() == 0


def test_c_abi_rejects_bad_arguments():
    L = capi.lib()
    d = C.c_void_p(16)  # never dereferenced: the checks run before any device call
    total, mx = C.c_int64(), C.c_int64()
    for W in (0, -1):
        assert L.bsq_crop(0, None, d, d, 1, W, 1, 0, 0, d, d, None) == capi.ERR_ARG
        assert L.bsq_crop_extent_device(0, None, d, 1, -1, W, C.byref(total), C.byref(mx)) == capi.ERR_ARG
    assert L.bsq_crop(0, None, d, d, -1, 4, 1, 0, 0, d, d, None) == capi.ERR_ARG
    for args in ((None, d, d, d), (d, None, d, d), (d, d, None, d), (d, d, d, None)):
        b, o, ob, oo = args
        assert L.bsq_crop(0, None, b, o, 3, 4, 0, 0, 0, ob, oo, None) == capi.ERR_ARG
    assert L.bsq_crop_extent_device(0, None, None, 3, -1, 4, C.byref(total), C.byref(mx)) == capi.ERR_ARG
    assert L.bsq_crop_extent_device(0, None, d, -1, -1, 4, C.byref(total), C.byref(mx)) == capi.ERR_ARG
    assert L.bsq_crop_extent_device(0, None, d, 3, -1, 4, None, C.byref(mx)) == capi.ERR_ARG
    assert L.bsq_crop_extent_device(0, None, d, 3, -1, 4, C.byref(total), None) == capi.ERR_ARG
    assert "crop_len" in capi.last_error() or "null" in capi.last_error()


def test_dataset_arguments():
    from bioseq_b200 import cbioseq, loaders
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "x.ff")
        with open(path, "wb") as f:
            f.write(oracle.flatfile_image([b"ACDEFGHIKLMN" * 10, b"ACD"]))
        ff = cbioseq.FlatFile(path)
        tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
        ds = loaders.FlatFileDataset(ff, tok, max_seq_len=3)
        assert (ds.max_seq_len, ds.crop, ds.crop_len) == (3, "random", 1)
        ds = loaders.FlatFileDataset(ff, tok, max_seq_len=64, crop="head")
        assert (ds.max_seq_len, ds.crop, ds.crop_len) == (64, "head", 62)
        assert loaders.FlatFileDataset(ff, tok).crop is None
        assert loaders.FlatFileDataset(ff, tok).max_seq_len == 122
        for kw in (dict(max_seq_len=2), dict(max_seq_len=0), dict(max_seq_len=64, crop="tail"),
                   dict(max_seq_len=64, crop=None)):
            with pytest.raises(ValueError):
                loaders.FlatFileDataset(ff, tok, **kw)
