"""CPU: the padding-free token entry points of the C ABI are exported and bound, and the host-side extent arithmetic of
batch_tokenize_varlen is pinned to the oracle's padded tokens trimmed per row.  No device is used."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from bioseq_b200 import capi, consumers
from oracle.oracle import OracleTokenizer
from helpers import gen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_varlen_entry_points_declared_exported_and_bound():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bsq.h")).read(), flags=re.S)
    L = C.CDLL(capi.LIB_PATH)
    for name in ("bsq_tokenize_varlen", "bsq_varlen_extent_device"):
        assert re.search(r"\b" + name + r"\s*\(", src), f"{name} not declared in include/bsq.h"
        assert hasattr(L, name) and name in capi.EXPORTS
        assert getattr(capi.lib(), name).argtypes is not None


def oracle_varlen(orc, buf, offs, destchar="B"):
    """The oracle's padded batch-first tokens, each row cut to len + bos + eos, concatenated; and cu_seqlens."""
    k = int(orc.bos() >= 0) + int(orc.eos() >= 0)
    lens = np.diff(offs)
    n = lens.size
    padlen = int(lens.max()) + k if n else 1
    padded = orc.batch_tokenize((buf, offs), padlen=max(padlen, 1), destchar=destchar, batch_first=True)
    rows = [padded[i, :int(lens[i]) + k] for i in range(n)]
    tokens = np.concatenate(rows) if rows else padded.reshape(-1)[:0]
    cu = np.zeros(n + 1, np.int64)
    np.cumsum(lens + k, out=cu[1:])
    return tokens, cu.astype(np.int32)


def test_readme_known_answer():
    orc = OracleTokenizer("DNA", bos=True, eos=True, padchar=True)
    buf = np.frombuffer(b"ACGTGGGG", np.uint8).copy()
    offs = np.array([0, 4, 8], np.int64)
    tokens, cu = oracle_varlen(orc, buf, offs)
    assert tokens.tolist() == [4, 0, 1, 2, 3, 5, 4, 2, 2, 2, 2, 5]
    assert cu.tolist() == [0, 6, 12]
    assert consumers._varlen_extent_host(offs, 2, 2) == (12, 6)


@pytest.mark.parametrize("k", [0, 1, 2])
def test_extent_arithmetic(k):
    buf, offs = gen(5, 300, 0, 40, b"ACGT")
    offs = offs + 7  # a range that does not start at 0
    total, max_seqlen = consumers._varlen_extent_host(offs, 300, k)
    lens = np.diff(offs)
    assert total == int(lens.sum()) + 300 * k
    assert max_seqlen == int(lens.max()) + k
    # cu_seqlens[i] = (offsets[i] - offsets[0]) + i * k
    cu = (offs - offs[0]) + np.arange(301) * k
    assert cu[-1] == total and np.all(np.diff(cu) == lens + k)
    assert consumers._varlen_extent_host(offs[:1], 0, k) == (0, 0)
    assert consumers._varlen_extent_host(np.zeros(4, np.int64), 3, k) == (3 * k, k)


def test_extent_errors():
    with pytest.raises(ValueError, match="non-decreasing"):
        consumers._varlen_extent_host(np.array([0, 5, 3], np.int64), 2, 1)
    with pytest.raises(ValueError, match="at or after 0"):
        consumers._varlen_extent_host(np.array([-1, 5], np.int64), 1, 1)
    # 2^31 - 1 tokens fit, one more does not
    assert consumers._varlen_extent_host(np.array([0, 2 ** 31 - 3], np.int64), 1, 2)[0] == 2 ** 31 - 1
    with pytest.raises(ValueError, match="2\\^31 - 1"):
        consumers._varlen_extent_host(np.array([0, 2 ** 31 - 2], np.int64), 1, 2)
