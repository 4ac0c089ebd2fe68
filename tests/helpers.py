"""Shared helpers for the parity tests (test infrastructure; may import oracle/)."""
import hashlib
import json
import os

import numpy as np

from bioseq_b200.synth import gen, gen_mask, as_list  # noqa: F401

REFERENCE_JSON = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference.json")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def sha_strs(strs):
    return hashlib.sha256("\n".join(strs).encode("latin-1")).hexdigest()[:16]


def raw(a):
    """Raw bytes + shape view used for bit-exact comparison across sign conventions."""
    a = np.ascontiguousarray(a)
    return a.shape, a.view(np.uint8).reshape(-1)


def assert_same_bits(a, b):
    sa, ra = raw(a)
    sb, rb = raw(b)
    assert sa == sb, (sa, sb)
    assert a.itemsize == b.itemsize
    if not np.array_equal(ra, rb):
        bad = np.flatnonzero(ra != rb)
        raise AssertionError(f"{bad.size} differing bytes, first at {bad[:8]} (shape {sa})")


def golden_inputs(rec):
    seed, n, lo, hi, alpha = rec["gen"]
    buf, offs = gen(seed, n, lo, hi, alpha.encode("latin-1"))
    assert sha(buf) == rec["buf_sha"] and sha(offs) == rec["offs_sha"], "synthetic generator drifted"
    mask = gen_mask(rec["mask_seed"], buf.size) if "mask_seed" in rec else None
    return buf, offs, mask


def _plain(x):
    if isinstance(x, (bytes, bytearray, memoryview)):
        return bytes(x)
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    if isinstance(x, np.integer):
        return int(x)
    return x


def digest(x):
    """Arrays: item size, shape and SHA-256 of the raw bytes (the terms of assert_same_bits); anything else (text,
    lists of strings or bytes, numbers, error messages): SHA-256 of its repr."""
    if isinstance(x, np.ndarray):
        a = np.ascontiguousarray(x)
        return f"{a.itemsize}:{'x'.join(map(str, a.shape))}:{sha(a)}"
    return "repr:" + hashlib.sha256(repr(_plain(x)).encode("utf-8", "surrogatepass")).hexdigest()[:16]


class Reference:
    """What the original project's compiled tokenizer (oracle/_ref, built by `make -C oracle ref` from its sources)
    returned at each comparison of one test, in call order, kept as digests in tests/golden/reference.json so that the
    comparison runs without it.  When oracle/_ref is present the live reference is compared as well.

    BSQ_RECORD_REFERENCE=<file> rewrites the test's entry of that file (created from tests/golden/reference.json) from
    the outputs the test compares instead of checking them.  It needs oracle/_ref: each recorded output must first
    equal the live reference's, so what is recorded is the reference's output."""

    def __init__(self, test, ref_module):
        self.test, self.live = test, ref_module is not None
        self.record_to = os.environ.get("BSQ_RECORD_REFERENCE")
        assert self.live or not self.record_to, "BSQ_RECORD_REFERENCE needs the compiled reference (make -C oracle ref)"
        with open(REFERENCE_JSON) as f:
            self.want = json.load(f)["tests"].get(test, [])
        self.got = []

    def check(self, ours, reference):
        """`ours`: this project's output; `reference`: a call that returns the reference's (made only when oracle/_ref
        is present).  Returns the reference's output, or None."""
        d = digest(ours)
        where = f"{self.test}, comparison {len(self.got)}"
        theirs = None
        if self.live:
            theirs = reference()
            if isinstance(ours, np.ndarray) and isinstance(theirs, np.ndarray):
                assert_same_bits(theirs, ours)
            assert digest(theirs) == d, f"{where}: reference {digest(theirs)}, ours {d}"
        if not self.record_to:
            assert len(self.got) < len(self.want), f"{self.test}: more comparisons than recorded"
            assert d == self.want[len(self.got)], f"{where}: recorded reference {self.want[len(self.got)]}, ours {d}"
        self.got.append(d)
        return theirs

    def done(self):
        if self.record_to:
            path = self.record_to if os.path.exists(self.record_to) else REFERENCE_JSON
            with open(path) as f:
                rec = json.load(f)
            rec["tests"][self.test] = self.got
            with open(self.record_to, "w") as f:
                json.dump(rec, f, indent=0, sort_keys=True)
        else:
            assert len(self.got) == len(self.want), f"{self.test}: {len(self.got)} comparisons, {len(self.want)} recorded"


def table_cap_lens():
    """Output bytes per row for the flat map's row-table cap (K12, K13a, K14b): tiles of 2046, 2047 and 2048 rows, 16
    bytes each but the tile's last.  With the output aligned a 64 KiB tile's row table needs as many rows, misaligned one
    more (the previous tile's last row), so 2047 rows (the table's cap) and 2048 (the first over-full count) occur at every
    output alignment."""
    lens = []
    for k in (2046, 2047, 2048, 2047, 2046):
        lens += [16] * (k - 1) + [65536 - 16 * (k - 1)]
    return lens
