"""CPU: k-mer tokens (batch_tokenize_kmer / bsq_kmer, kernel K11) without a device.

The entry points are declared, exported and bound; the numpy reference of the rule (tests/kmer_reference.py, what the
GPU tests compare with) is checked against a scalar restatement of the header's text and against the header's worked
answers; bsq_kmer_init's ids, limits and errors, bsq_kmer_extent_host against the reference (also past 2^31 tokens),
kmer_ids / kmer_vocab, and the C ABI's argument checks, which must fail before any device call."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import bioseq_b200
from bioseq_b200 import capi, consumers
from oracle.oracle import OracleTokenizer
import kmer_reference as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("bsq_kmer_init", "bsq_tokenize_kmer", "bsq_tokenize_kmer_varlen", "bsq_kmer_extent_host", "bsq_kmer_extent_device")
# the largest k of each alphabet whose vocabulary fits int32 (b^k + b + 1 + 3 - 1 <= 2^31 - 1)
KMAX = {"DNA": 15, "DNA5": 13, "SEB6": 11, "PROTEIN": 7, "PURPYR": 30}
MIX = b"ACGTUNacgtunRYKMSW-*.\x00\x7f\x80\xc3\xffDEFHIKLMPQVXZ"


def test_kmer_entry_points_declared_exported_and_bound():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bsq.h")).read(), flags=re.S)
    L = C.CDLL(capi.LIB_PATH)
    for name in NEW:
        assert re.search(r"\b" + name + r"\s*\(", src), f"{name} not declared in include/bsq.h"
        assert hasattr(L, name) and name in capi.EXPORTS
        assert getattr(capi.lib(), name).argtypes is not None
    for name in ("batch_tokenize_kmer", "kmer_ids", "kmer_vocab", "KmerIds"):
        assert name in bioseq_b200.__all__ and hasattr(bioseq_b200, name)
    assert C.sizeof(capi.KmerDesc) == 7 * 4 + 4 + 6 * 8


# ------------------------------------------------------------------------------------------------------------------
def restate(seq, key, k, s, single, bos, eos, padchar):
    """The rule of include/bsq.h written again from its text, for one sequence, in Python integers."""
    o = OracleTokenizer(key)
    b = o.nchars()

    def code(x):
        return int(o.lut[x]) if x < 0x80 else -1

    unk = b ** k + b
    out = [unk + 1] if bos else []
    n = len(seq)
    m = (n - k) // s + 1 if n >= k else 0
    for j in range(m):
        v, bad = 0, False
        for t in range(k):
            c = code(seq[j * s + t])
            bad |= c < 0
            v += max(c, 0) * b ** (k - 1 - t)
        out.append(unk if bad else v)
    covered = (m - 1) * s + k if m else 0
    if single:
        for x in seq[covered:]:
            c = code(x)
            out.append(unk if c < 0 else b ** k + c)
    if eos:
        out.append(unk + 1 + bos)
    return out


def lengths_for(k, s):
    ls = {0, 1, max(k - 1, 0), k, k + 1}
    for j in range(1, 4):
        ls |= {k + j * s - 1, k + j * s, k + j * s + 1}
    return sorted(ls)


def random_batch(lens, seed, alphabet=MIX):
    rng = np.random.default_rng(seed)
    table = np.frombuffer(alphabet, np.uint8)
    offs = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    # mostly valid residues, so that k-mers without an invalid byte occur for every k
    valid = np.frombuffer(b"ACGTacgt" if b"A" in alphabet else alphabet, np.uint8)
    buf = np.where(rng.random(int(offs[-1])) < 0.9, valid[rng.integers(0, valid.size, int(offs[-1]))],
                   table[rng.integers(0, table.size, int(offs[-1]))]).astype(np.uint8)
    return buf, offs


CASES = [(key, k) for key, kmax in KMAX.items() for k in range(1, kmax + 1)
         if key == "DNA" or k in (1, 2, 3, kmax - 1, kmax)]


@pytest.mark.parametrize("key,k", CASES)
def test_reference_matches_scalar_restatement(key, k):
    valid = {"DNA": b"ACGTacgt", "DNA5": b"ACGTNacgtn", "SEB6": b"ACDEFGHIKLMNPQRSTVWY", "PROTEIN": b"ACDEFGHIKLMNPQRSTVWYacdy",
             "PURPYR": b"ACGTRYacgt"}[key]
    for s in range(1, k + 1):
        lens = lengths_for(k, s)
        buf, offs = random_batch(lens, 1000 * k + s, valid + b"NnUu\x80\xff-")
        for single in (False, True):
            for bos, eos in ((True, True), (False, False), (True, False)):
                got = ref.rows(buf, offs, key, k, s, single, bos, eos)
                for i in range(len(lens)):
                    want = restate(bytes(buf[offs[i]:offs[i + 1]]), key, k, s, single, bos, eos, False)
                    assert got[i].tolist() == want, (key, k, s, single, lens[i])
                assert np.array_equal([g.size for g in got], ref.count(np.diff(offs), k, s, single, bos, eos))


WORKED = [("ACGTNAG", 1, "drop", [69, 6, 27, 68, 68, 68, 70]), ("ACGTNAG", 1, "single", [69, 6, 27, 68, 68, 68, 70]),
          ("ACGTNAG", 3, "single", [69, 6, 68, 66, 70]), ("ACGTNAG", 3, "drop", [69, 6, 68, 70]),
          ("AC", 1, "single", [69, 64, 65, 70]), ("AC", 2, "single", [69, 64, 65, 70]), ("AC", 3, "single", [69, 64, 65, 70]),
          ("AC", 1, "drop", [69, 70]), ("AC", 3, "drop", [69, 70]), ("", 1, "single", [69, 70]), ("", 3, "drop", [69, 70])]


@pytest.mark.parametrize("seq,s,tail,want", WORKED)
def test_worked_answers(seq, s, tail, want):
    buf = np.frombuffer(seq.encode(), np.uint8)
    offs = np.array([0, len(seq)], np.int64)
    assert ref.rows(buf, offs, "DNA", 3, s, tail == "single", True, True)[0].tolist() == want
    assert restate(seq.encode(), "DNA", 3, s, tail == "single", True, True, True) == want
    km = capi.kmer_desc(consumers.descriptor(bioseq_b200.pbeos_tokenizers["DNA"]), 3, s, consumers._KMER_TAILS[tail])
    assert capi.kmer_extent_host(offs, 1, km) == (len(want), len(want))


# ------------------------------------------------------------------------------------------------------------------
def test_kmer_init_ids():
    for key in ("DNA", "PROTEIN", "SEB6", "PURPYR", "DNA5"):
        for bos, eos, pad in [(b, e, p) for b in (0, 1) for e in (0, 1) for p in (0, 1)]:
            tok = capi.tokenizer(key, eos=eos, bos=bos, padchar=pad)
            for k in (1, 2, KMAX[key]):
                km = capi.kmer_desc(tok, k, k, capi.KMER_SINGLE)
                want = ref.ids(tok.nchars, k, bos, eos, pad)
                assert (km.nkmers, km.unk_id, km.pad_id, km.vocab_size) == (want["nkmers"], want["unk"], want["pad"], want["vocab_size"])
                assert km.bos_id == (want["bos"] if bos else -1) and km.eos_id == (want["eos"] if eos else -1)
                assert (km.k, km.stride, km.tail, km.nchars, km.bos, km.eos, km.padchar) == (k, k, 1, tok.nchars, bos, eos, pad)
    # the worked example
    ids = bioseq_b200.kmer_ids(bioseq_b200.pbeos_tokenizers["DNA"], 3)
    assert ids == (64, 64, 68, 69, 70, 71, 72)
    ids = bioseq_b200.kmer_ids(bioseq_b200.DNATokenizer, 6)
    assert ids == (4096, 4096, 4100, None, None, 4101, 4101)


@pytest.mark.parametrize("key", sorted(KMAX))
def test_kmer_init_limits(key):
    tok = capi.tokenizer(key, eos=True, bos=True, padchar=True)
    km = capi.kmer_desc(tok, KMAX[key], 1)
    assert km.vocab_size - 1 <= 2 ** 31 - 1
    with pytest.raises(ValueError, match="2\\^31"):
        capi.kmer_desc(tok, KMAX[key] + 1, 1)
    with pytest.raises(ValueError, match="2\\^31"):
        bioseq_b200.kmer_ids(bioseq_b200.pbeos_tokenizers[key], KMAX[key] + 1)


def test_kmer_init_errors():
    tok = capi.tokenizer("DNA")
    for k, s, tail in [(0, 1, 0), (-1, 1, 0), (3, 0, 0), (3, 4, 0), (3, -1, 0), (3, 1, 2), (3, 1, -1)]:
        with pytest.raises(ValueError):
            capi.kmer_desc(tok, k, s, tail)
    with pytest.raises(ValueError, match="BYTES"):
        capi.kmer_desc(capi.tokenizer("BYTES"), 1, 1)
    assert capi.lib().bsq_kmer_init(None, C.byref(tok), 3, 1, 0) == capi.ERR_ARG
    assert capi.lib().bsq_kmer_init(C.byref(capi.KmerDesc()), None, 3, 1, 0) == capi.ERR_ARG
    t = bioseq_b200.DNATokenizer
    for kw in (dict(k=0), dict(k=3, stride=4), dict(k=3, stride=0), dict(k=3, tail="keep"), dict(k=3.0), dict(k=3, stride=None)):
        k = kw.pop("k")
        with pytest.raises(ValueError):
            consumers._kmer_desc(t, k, **kw)


# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,s,single", [(1, 1, False), (3, 1, True), (3, 3, True), (6, 6, True), (6, 1, False), (5, 2, True)])
def test_extent_host_matches_reference(k, s, single):
    rng = np.random.default_rng(k * 10 + s)
    lens = rng.integers(0, 40, 3000)
    offs = np.zeros(lens.size + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    offs += 7  # offsets[0] != 0
    for bos, eos in ((0, 0), (1, 1), (1, 0)):
        tok = capi.tokenizer("DNA", eos=eos, bos=bos)
        km = capi.kmer_desc(tok, k, s, int(single))
        t = ref.count(lens, k, s, single, bos, eos)
        assert capi.kmer_extent_host(offs, lens.size, km) == (int(t.sum()), int(t.max()))
    assert capi.kmer_extent_host(offs, 0, km) == (0, 0)


def test_extent_host_past_int32_and_the_python_limit():
    # no residues are needed to size a batch: lengths of 2^30 give totals past 2^31 - 1
    tok = capi.tokenizer("DNA", eos=True, bos=True)
    km = capi.kmer_desc(tok, 1, 1)
    offs = np.array([0, 2 ** 30, 2 ** 31 - 4, 2 ** 31 - 3], np.int64)
    total, mx = capi.kmer_extent_host(offs, 3, km)
    assert (total, mx) == (2 ** 31 - 3 + 6, 2 ** 30 + 2) and total > 2 ** 31 - 1
    with pytest.raises(ValueError, match="2\\^31 - 1"):
        consumers._kmer_check_extent((total, mx), 0, True)
    consumers._kmer_check_extent((2 ** 31 - 1, mx), 0, True)  # exactly the limit fits
    km = capi.kmer_desc(tok, 15, 15, capi.KMER_SINGLE)
    big = np.array([0, 3 * 2 ** 31 + 7], np.int64)  # lengths past int32: the host count is exact
    assert capi.kmer_extent_host(big, 1, km) == ((3 * 2 ** 31 + 7 - 15) // 15 + 1 + (3 * 2 ** 31 + 7 - 15) % 15 + 2,) * 2
    with pytest.raises(ValueError, match="> padlen: 9, vs padlen 8"):
        consumers._kmer_check_extent((9, 9), 8, False)


def test_extent_host_rejects_bad_offsets():
    km = capi.kmer_desc(capi.tokenizer("DNA"), 3, 1)
    with pytest.raises(ValueError, match="non-decreasing"):
        capi.kmer_extent_host(np.array([0, 5, 3], np.int64), 2, km)
    with pytest.raises(ValueError, match="start at or after 0"):
        capi.kmer_extent_host(np.array([-1, 5], np.int64), 1, km)
    t, m = C.c_int64(), C.c_int64()
    assert capi.lib().bsq_kmer_extent_host(None, 2, C.byref(km), C.byref(t), C.byref(m)) == capi.ERR_ARG
    assert capi.lib().bsq_kmer_extent_host(None, -1, C.byref(km), C.byref(t), C.byref(m)) == capi.ERR_ARG
    assert capi.lib().bsq_kmer_extent_host(None, 0, None, C.byref(t), C.byref(m)) == capi.ERR_ARG


# ------------------------------------------------------------------------------------------------------------------
def test_kmer_vocab_known_answers():
    v = bioseq_b200.kmer_vocab(bioseq_b200.pbeos_tokenizers["DNA"], 3)
    assert len(v) == 72 and v[0] == "AAA" and v[6] == "ACG" and v[27] == "CGT" and v[63] == "TTT"
    assert v[64:68] == ["A", "C", "G", "T"] and v[68:] == ["<UNK>", "<BOS>", "<EOS>", "<PAD>"]
    v = bioseq_b200.kmer_vocab(bioseq_b200.DNATokenizer, 1)
    assert v == ["A", "C", "G", "T", "A", "C", "G", "T", "<UNK>"]
    v = bioseq_b200.kmer_vocab(bioseq_b200.beos_tokenizers["PROTEIN"], 2)
    ids = bioseq_b200.kmer_ids(bioseq_b200.beos_tokenizers["PROTEIN"], 2)
    assert len(v) == ids.vocab_size == 400 + 20 + 1 + 2 and v[-3:] == ["<UNK>", "<BOS>", "<EOS>"]
    # k-mer j is spelled by its digits, first residue most significant
    letters = v[400:420]
    assert all(v[a * 20 + b] == letters[a] + letters[b] for a in range(20) for b in range(20))
    assert len(set(v[:420])) == 420


# ------------------------------------------------------------------------------------------------------------------
def test_c_abi_rejects_bad_arguments_before_any_device_call():
    L = capi.lib()
    tok = capi.tokenizer("DNA", eos=True, bos=True)
    km = capi.kmer_desc(tok, 6, 1)
    p, offs = 0x1000, 0x2000
    assert L.bsq_tokenize_kmer(0, None, p, offs, 4, 16, C.byref(tok), None, capi.I32, p) == capi.ERR_ARG
    assert L.bsq_tokenize_kmer(0, None, p, offs, 4, 16, None, C.byref(km), capi.I32, p) == capi.ERR_ARG
    assert L.bsq_tokenize_kmer(0, None, p, offs, -1, 16, C.byref(tok), C.byref(km), capi.I32, p) == capi.ERR_ARG
    assert L.bsq_tokenize_kmer(0, None, p, offs, 4, 0, C.byref(tok), C.byref(km), capi.I32, p) == capi.ERR_ARG
    assert L.bsq_tokenize_kmer(0, None, p, offs, 4, 16, C.byref(tok), C.byref(km), capi.I32, p + 4) == capi.ERR_ARG
    assert L.bsq_tokenize_kmer(0, None, None, offs, 4, 16, C.byref(tok), C.byref(km), capi.I32, p) == capi.ERR_ARG
    assert L.bsq_tokenize_kmer(0, None, p, offs, 4, 16, C.byref(tok), C.byref(km), 9, p) == capi.ERR_ARG
    # kinds too narrow for 4 096 + 4 + 3 ids
    assert L.bsq_tokenize_kmer(0, None, p, offs, 4, 16, C.byref(tok), C.byref(km), capi.I8, p) == capi.ERR_ARG
    assert "do not fit" in capi.last_error()
    km_big = capi.kmer_desc(tok, 12, 1)  # 4^12 + 7 ids: too many for int16 and float32
    for kind in (capi.I16, capi.F32):
        assert L.bsq_tokenize_kmer(0, None, p, offs, 4, 16, C.byref(tok), C.byref(km_big), kind, p) == capi.ERR_ARG
    # a descriptor made for another tokenizer
    other = capi.kmer_desc(capi.tokenizer("DNA"), 6, 1)
    assert L.bsq_tokenize_kmer(0, None, p, offs, 4, 16, C.byref(tok), C.byref(other), capi.I32, p) == capi.ERR_ARG
    bad = capi.kmer_desc(tok, 6, 1)
    bad.stride = 7
    assert L.bsq_tokenize_kmer(0, None, p, offs, 4, 16, C.byref(tok), C.byref(bad), capi.I32, p) == capi.ERR_ARG
    cu = 0x3000
    assert L.bsq_tokenize_kmer_varlen(0, None, p, offs, 4, C.byref(tok), C.byref(km), capi.I32, p, None) == capi.ERR_ARG
    assert L.bsq_tokenize_kmer_varlen(0, None, p, offs, -1, C.byref(tok), C.byref(km), capi.I32, p, cu) == capi.ERR_ARG
    assert L.bsq_tokenize_kmer_varlen(0, None, p, offs, 4, C.byref(tok), C.byref(km), capi.I32, p + 8, cu) == capi.ERR_ARG
    assert L.bsq_tokenize_kmer_varlen(0, None, None, offs, 4, C.byref(tok), C.byref(km), capi.I32, p, cu) == capi.ERR_ARG
    assert L.bsq_tokenize_kmer_varlen(0, None, p, offs, 4, C.byref(tok), C.byref(km), capi.I8, p, cu) == capi.ERR_ARG
    t, m = C.c_int64(), C.c_int64()
    assert L.bsq_kmer_extent_device(0, None, offs, 4, -1, None, C.byref(t), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_kmer_extent_device(0, None, None, 4, -1, C.byref(km), C.byref(t), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_kmer_extent_device(0, None, offs, -1, -1, C.byref(km), C.byref(t), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_kmer_extent_device(0, None, offs, 4, -1, C.byref(km), None, C.byref(m)) == capi.ERR_ARG
    # nothing to do: no device call either
    assert L.bsq_kmer_extent_device(0, None, None, 0, -1, C.byref(km), C.byref(t), C.byref(m)) == capi.OK
    assert (t.value, m.value) == (0, 0)
    assert L.bsq_tokenize_kmer(0, None, None, None, 0, 16, C.byref(tok), C.byref(km), capi.I32, None) == capi.OK
