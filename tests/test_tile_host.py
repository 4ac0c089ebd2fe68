"""CPU: sliding-window tiling and stitching (tile_packed / batch_tokenize_tiled / untile / bsq_tile, kernel K13) without
a device.

The entry points are declared, exported and bound; the numpy reference (tests/tile_reference.py, what the GPU tests
compare with) is pinned to a scalar restatement of the header's rule and to its worked answers, and
bsq_tile_extent_host to the reference on edge and random lengths (counts only near 2^62, and past INT64_MAX); every
argument error is raised before anything is staged or launched, and the C ABI rejects bad arguments without a device."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from bioseq_b200 import capi, consumers
import tile_reference as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("bsq_tile_extent_host", "bsq_tile_extent_device", "bsq_tile", "bsq_untile_mean")


def test_tile_entry_points_declared_exported_and_bound():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bsq.h")).read(), flags=re.S)
    L = C.CDLL(capi.LIB_PATH)
    for name in NEW:
        assert re.search(r"\b" + name + r"\s*\(", src), f"{name} not declared in include/bsq.h"
        assert hasattr(L, name) and name in capi.EXPORTS
        assert getattr(capi.lib(), name).argtypes is not None
    for name, value in (("BSQ_TILE_SHORT", capi.TILE_SHORT), ("BSQ_TILE_END", capi.TILE_END), ("BSQ_TILE_DROP", capi.TILE_DROP),
                        ("BSQ_UNTILE_F32", capi.UNTILE_F32), ("BSQ_UNTILE_BF16", capi.UNTILE_BF16),
                        ("BSQ_UNTILE_F16", capi.UNTILE_F16)):
        assert re.search(r"#define\s+" + name + r"\s+" + str(value) + r"\b", src)
    import bioseq_b200
    for name in ("tile_packed", "batch_tokenize_tiled", "untile", "TiledBatch", "TiledTokens", "UntiledBatch"):
        assert name in bioseq_b200.__all__ and hasattr(bioseq_b200, name)


# ------------------------------------------------------------------------------------------------------------------
def scalar_windows(n, W, S, tail):
    """The header's rule word for word, one window at a time."""
    if n <= W:
        return [(0, n)]
    if tail == "drop":
        m = math.floor((n - W) / S) + 1
    else:
        m = math.ceil((n - W) / S) + 1
    out = []
    for j in range(m):
        if tail == "short":
            out.append((j * S, min(W, n - j * S)))
        elif tail == "end" and j == m - 1:
            out.append((n - W, W))
        else:
            out.append((j * S, W))
    return out


@pytest.mark.parametrize("tail", ["short", "end", "drop"])
def test_reference_matches_scalar_rule(tail):
    for W in (1, 2, 3, 4, 7, 16, 64):
        for S in sorted(s for s in {1, 2, 3, W // 2 or 1, W - 1 or 1, W} if s <= W):
            for n in range(0, 3 * W + 20):
                got = ref.windows(n, W, S, tail)
                assert got == scalar_windows(n, W, S, tail), (n, W, S, tail)
                # every window lies in the sequence, starts ascend, and (but for DROP) every residue is covered
                assert all(0 <= st and st + ln <= n for st, ln in got)
                assert [st for st, _ in got] == sorted(st for st, _ in got)
                covered = set(p for st, ln in got for p in range(st, st + ln))
                if tail != "drop":
                    assert covered == set(range(n))
                if tail == "end" and n > W and (n - W) % S == 0:
                    assert got == ref.windows(n, W, S, "short")


@pytest.mark.parametrize("tail,want", [
    ("short", [(0, "ACGT"), (3, "TACG"), (6, "GTAC"), (9, "CG")]),
    ("end", [(0, "ACGT"), (3, "TACG"), (6, "GTAC"), (7, "TACG")]),
    ("drop", [(0, "ACGT"), (3, "TACG"), (6, "GTAC")]),
])
def test_worked_answers(tail, want):
    s = b"ACGTACGTACG"
    b, o, sp, si, st = ref.tile(np.frombuffer(s, np.uint8), [0, 11], 4, 3, tail)
    assert [(int(st[w]), b[o[w]:o[w + 1]].tobytes().decode()) for w in range(len(si))] == want
    assert sp.tolist() == [0, len(want)] and si.tolist() == [0] * len(want)
    five = {"short": [(0, 4), (3, 2)], "end": [(0, 4), (1, 4)], "drop": [(0, 4)]}
    assert ref.windows(5, 4, 3, tail) == five[tail]
    assert ref.windows(4, 4, 3, tail) == [(0, 4)] and ref.windows(0, 4, 3, tail) == [(0, 0)]


@pytest.mark.parametrize("tail,want", [
    ("short", [0, 0, 0, 0.5, 1, 1, 1.5, 2, 2, 2.5, 3]),
    ("end", [0, 0, 0, 0.5, 1, 1, 1.5, 2.5, 2.5, 2.5, 3]),
    ("drop", [0, 0, 0, 0.5, 1, 1, 1.5, 2, 2, 2, float("nan")]),
])
def test_untile_worked_answer(tail, want):
    W, S = 4, 3
    M = len(ref.windows(11, W, S, tail))
    y = np.repeat(np.arange(M, dtype=np.float32), W)[:, None]  # padded (M, W, 1): window w reports w everywhere
    got = ref.untile(y, [11], W, S, tail, lambda w: w * W, 0)[:, 0]
    np.testing.assert_array_equal(got, np.array(want, np.float32))


def test_untile_reference_order_and_flips():
    # two strands, the second flipped: each residue's mean is its own position when windows report source positions
    W, S, lens = 5, 2, [0, 3, 12, 7]
    wins = [ref.windows(n, W, S, "end") for n in lens]
    flat = [(st, ln) for w in wins for st, ln in w]
    M = len(flat)
    y = np.zeros((2 * M, W), np.float32)
    for w, (st, ln) in enumerate(flat):
        y[w, :ln] = np.arange(st, st + ln)
        y[M + w, :ln] = np.arange(st, st + ln)[::-1]
    flipped = np.array([0] * M + [1] * M, np.uint8)
    got = ref.untile(y.reshape(-1, 1), lens, W, S, "end", lambda w: w * W, 0, strands=2, flipped=flipped)[:, 0]
    np.testing.assert_array_equal(got, np.concatenate([np.arange(n, dtype=np.float32) for n in lens]))


# ------------------------------------------------------------------------------------------------------------------
def ref_extent(lens, W, S, tail):
    wins = [ref.windows(int(n), W, S, tail) for n in lens]
    return (sum(len(w) for w in wins), sum(ln for w in wins for _, ln in w), max((min(int(n), W) for n in lens), default=0))


@pytest.mark.parametrize("tail", ["short", "end", "drop"])
def test_extent_host_matches_reference(tail):
    rng = np.random.default_rng(7)
    t = consumers._TILE_TAILS[tail]
    for W, S in ((1, 1), (4, 3), (16, 16), (64, 1), (100, 37), (1000, 500)):
        edge = {0, 1, W - 1, W, W + 1, W + S - 1, W + S, W + S + 1, 2 * W, 3 * W + S + 1}
        lens = np.array(sorted(x for x in edge if x >= 0) + list(rng.integers(0, 5 * W + 3, 200)), np.int64)
        offs = np.concatenate([[5], 5 + np.cumsum(lens)]).astype(np.int64)
        assert capi.tile_extent_host(offs, lens.size, W, S, t) == ref_extent(lens, W, S, tail)
        assert capi.tile_extent_host(offs, 0, W, S, t) == (0, 0, 0)


def scalar_count(n, W, S, tail):
    """m of the header's rule in exact integers (math.ceil of a float would round at these sizes)."""
    if n <= W:
        return 1
    return ((n - W) // S if tail == "drop" else -(-(n - W) // S)) + 1


def test_extent_host_near_2_62_and_past_int64():
    n = 2 ** 62 + 12345
    W = 1000
    offs = np.array([0, n], np.int64)
    for S in (W, 999, 600):  # bytes ~ n * W / S stay below 2^63
        for tail in ("short", "end", "drop"):
            wins = scalar_count(n, W, S, tail)
            nbytes = {"short": (wins - 1) * W + n - (wins - 1) * S, "end": wins * W, "drop": wins * W}[tail]
            assert capi.tile_extent_host(offs, 1, W, S, consumers._TILE_TAILS[tail]) == (wins, nbytes, W)
    # windows fit but their bytes do not: S = 7 makes ~n / 7 windows of W bytes
    for tail in (capi.TILE_SHORT, capi.TILE_END, capi.TILE_DROP):
        with pytest.raises(ValueError, match="INT64_MAX"):
            capi.tile_extent_host(offs, 1, W, 7, tail)
    # (no more windows than residues, so the count is bounded by offsets[n]): exactly INT64_MAX windows and bytes fit
    big = np.array([0, 2 ** 62, 2 ** 63 - 1], np.int64)
    assert capi.tile_extent_host(big, 2, 1, 1, capi.TILE_SHORT) == (2 ** 63 - 1, 2 ** 63 - 1, 1)
    with pytest.raises(ValueError, match="INT64_MAX"):  # one byte more: the second sequence in windows of 2 at stride 1
        capi.tile_extent_host(big, 2, 2, 1, capi.TILE_SHORT)


def test_extent_host_rejects_bad_arguments():
    o = np.array([0, 5, 9], np.int64)
    for W, S, tail in ((0, 1, 0), (4, 0, 0), (4, 5, 0), (4, 2, 3), (4, 2, -1), (-3, -3, 0)):
        with pytest.raises(ValueError):
            capi.tile_extent_host(o, 2, W, S, tail)
    with pytest.raises(ValueError):
        capi.tile_extent_host(np.array([0, 5, 3], np.int64), 2, 4, 2, 0)
    with pytest.raises(ValueError):
        capi.tile_extent_host(np.array([-1, 5], np.int64), 1, 4, 2, 0)
    L = capi.lib()
    w, b, m = C.c_int64(), C.c_int64(), C.c_int64()
    assert L.bsq_tile_extent_host(None, 2, 4, 2, 0, C.byref(w), C.byref(b), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_tile_extent_host(None, -1, 4, 2, 0, C.byref(w), C.byref(b), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_tile_extent_host(o.ctypes.data, 2, 4, 2, 0, None, C.byref(b), C.byref(m)) == capi.ERR_ARG


def test_c_abi_rejects_bad_arguments():
    L = capi.lib()
    d = C.c_void_p(16)  # never dereferenced: the checks run before any device call
    w, b, m = C.c_int64(), C.c_int64(), C.c_int64()
    for W, S, tail in ((0, 1, 0), (4, 0, 0), (4, 5, 0), (4, 2, 3)):
        assert L.bsq_tile(0, None, d, d, 1, W, S, tail, d, d, None, None, None) == capi.ERR_ARG
        assert L.bsq_tile_extent_device(0, None, d, 1, -1, W, S, tail, C.byref(w), C.byref(b), C.byref(m)) == capi.ERR_ARG
        assert L.bsq_untile_mean(0, None, 0, d, 1, 8, None, 0, d, 1, W, S, tail, d, 1, 1, None, d) == capi.ERR_ARG
    assert L.bsq_tile(0, None, d, d, -1, 4, 2, 0, d, d, None, None, None) == capi.ERR_ARG
    for bb, o, ob, oo in ((None, d, d, d), (d, None, d, d), (d, d, None, d), (d, d, d, None)):
        assert L.bsq_tile(0, None, bb, o, 3, 4, 2, 0, ob, oo, None, None, None) == capi.ERR_ARG
    assert L.bsq_tile_extent_device(0, None, None, 3, -1, 4, 2, 0, C.byref(w), C.byref(b), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_tile_extent_device(0, None, d, -1, -1, 4, 2, 0, C.byref(w), C.byref(b), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_tile_extent_device(0, None, d, 3, -1, 4, 2, 0, None, C.byref(b), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_tile_extent_device(0, None, None, 0, -1, 4, 2, 0, C.byref(w), C.byref(b), C.byref(m)) == capi.OK
    U = L.bsq_untile_mean
    good = dict(dtype=0, y=d, C=1, stride=8, cu=None, col0=0, offs=d, n=1, W=4, S=2, tail=0, sp=d, nwin=1, strands=1, fl=None, out=d)
    for k, v in (("dtype", 3), ("dtype", -1), ("C", 0), ("col0", -1), ("strands", 0), ("strands", 3), ("n", -1), ("nwin", 0),
                 ("stride", 0), ("y", None), ("offs", None), ("sp", None), ("out", None)):
        args = dict(good, **{k: v})
        assert U(0, None, *args.values()) == capi.ERR_ARG, k
    assert U(0, None, *dict(good, n=0, nwin=0).values()) == capi.OK  # nothing to do


def test_argument_errors_before_any_device_work():
    from bioseq_b200 import cbioseq
    dna = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
    prot = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    batch = (np.frombuffer(b"ACGTACGTA", np.uint8).copy(), np.array([0, 9], np.int64))
    capi.lib().bsq_launch_count_reset()
    bad = [dict(window=0), dict(window=4, stride=0), dict(window=4, stride=5), dict(window=4, tail="middle"), dict(window=4, tail=1),
           dict(window=4.5), dict(window=4, stride="2"), dict(window=4, padlen=5), dict(window=4, varlen=True, padlen=8),
           dict(window=4, crop="head"), dict(window=4, rc="flip"), dict(window=4, rc_prob=0.5), dict(window=4, rc="always", rc_prob=0.5),
           dict(window=4, rc="random", rc_prob=2.0), dict(window=4, rc="random", rc_prob=float("nan"))]
    for kw in bad:
        with pytest.raises(ValueError):
            consumers.batch_tokenize_tiled(dna, batch, **kw)
    with pytest.raises(ValueError):  # no complement for proteins
        consumers.batch_tokenize_tiled(prot, batch, 4, rc="both")
    for kw in (dict(window=0), dict(window=4, stride=7), dict(window=4, tail="none")):
        with pytest.raises(ValueError):
            consumers.tile_packed(batch[0], batch[1], **kw)
    with pytest.raises(ValueError):
        consumers.tile_packed(batch[0], batch[1], 4)  # host arrays: tile_packed works on CUDA tensors
    with pytest.raises(ValueError):
        consumers.untile(np.zeros((1, 6), np.float32), None)
    assert capi.lib().bsq_launch_count() == 0


def test_tile_spec():
    assert consumers._tile_spec(8, None, "short") == (8, 8, capi.TILE_SHORT)
    assert consumers._tile_spec(8, 1, "end") == (8, 1, capi.TILE_END)
    assert consumers._tile_spec(np.int64(8), np.int32(3), "drop") == (8, 3, capi.TILE_DROP)
