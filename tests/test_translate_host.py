"""CPU: translation of DNA into protein reading frames (translate_packed / batch_tokenize_translated / translate= /
bsq_translate, kernel K14) without a device.

The entry points are declared, exported and bound; the built-in genetic codes equal the header's strings;
bsq_translate_table equals a scalar itertools.product restatement of the rule over every triple of base sets; the numpy
reference (tests/translate_reference.py, what the GPU tests compare with) reproduces every worked answer of the header;
bsq_translate_extent_host matches the reference on edge and random lengths; every argument error is raised before
anything is staged or launched, and the C ABI rejects bad arguments without a device."""
import ctypes as C
import itertools
import os
import re

import numpy as np
import pytest

from bioseq_b200 import capi, consumers
import translate_reference as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("bsq_genetic_code", "bsq_translate_table", "bsq_translate_extent_host", "bsq_translate_extent_device", "bsq_translate")
SIX = (1, 2, 3, -1, -2, -3)


def test_translate_entry_points_declared_exported_and_bound():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bsq.h")).read(), flags=re.S)
    L = C.CDLL(capi.LIB_PATH)
    for name in NEW:
        assert re.search(r"\b" + name + r"\s*\(", src), f"{name} not declared in include/bsq.h"
        assert hasattr(L, name) and name in capi.EXPORTS
        assert getattr(capi.lib(), name).argtypes is not None
    assert re.search(r"#define\s+BSQ_ABI_VERSION\s+5\b", src)
    import bioseq_b200
    for name in ("translate_packed", "batch_tokenize_translated", "TranslatedBatch"):
        assert name in bioseq_b200.__all__ and hasattr(bioseq_b200, name)


@pytest.mark.parametrize("code", [1, 2, 4, 5, 6, 11])
def test_builtin_codes_equal_header_strings(code):
    header = open(os.path.join(ROOT, "include", "bsq.h")).read()
    got = capi.genetic_code(code)
    assert got == ref.CODES[code].encode() and len(got) == 64
    assert consumers._genetic_code(code) == got
    assert ref.CODES[code] in open(os.path.join(ROOT, "bioseq_b200", "csrc", "bsq_translate.cu")).read()
    assert "bsq_genetic_code" in header


def test_genetic_code_rejects_other_ids():
    buf = C.create_string_buffer(64)
    for code in (0, 3, 7, 12, -1, 100):
        assert capi.lib().bsq_genetic_code(code, buf) == capi.ERR_ARG
        with pytest.raises(ValueError):
            consumers._genetic_code(code)
    assert capi.lib().bsq_genetic_code(1, None) == capi.ERR_ARG


def scalar_letter(m0, m1, m2, code):
    """The header's rule for a triple of 4-bit base sets (A = 1, C = 2, G = 4, T = 8), word for word."""
    bases = "ACGT"
    sets = [[bases[b] for b in range(4) if (m >> b) & 1] for m in (m0, m1, m2)]
    if not all(sets):
        return "X"
    idx = {"T": 0, "C": 1, "A": 2, "G": 3}
    letters = set(code[16 * idx[a] + 4 * idx[b] + idx[c]] for a, b, c in itertools.product(*sets))
    return letters.pop() if len(letters) == 1 else "X"


@pytest.mark.parametrize("code", [1, 2, 6, "custom"])
def test_table_equals_scalar_rule(code):
    s = ref.CODES[code] if code != "custom" else "".join(chr(0x21 + (7 * i) % 94) for i in range(64))
    masks, codons = capi.translate_table(s.encode())
    want_masks = np.zeros(256, np.uint8)
    for c, bs in ref.IUPAC.items():
        m = sum({"A": 1, "C": 2, "G": 4, "T": 8}[b] for b in bs)
        want_masks[ord(c)] = want_masks[ord(c.lower())] = m
    np.testing.assert_array_equal(masks, want_masks)
    for m0, m1, m2 in itertools.product(range(16), repeat=3):  # all 15^3 base-set triples, and the invalid ones
        assert chr(codons[m0 << 8 | m1 << 4 | m2]) == scalar_letter(m0, m1, m2, s), (m0, m1, m2)
    rm, rc = ref.tables(s)
    np.testing.assert_array_equal(masks, rm)
    np.testing.assert_array_equal(codons, rc)


def test_table_rejects_bad_codes():
    m, c = np.zeros(256, np.uint8), np.zeros(4096, np.uint8)
    L = capi.lib()
    good = ref.CODES[1].encode()
    assert L.bsq_translate_table(good, m.ctypes.data, c.ctypes.data) == capi.OK
    for bad in (None, good[:63] + b" ", good[:10] + b"\x7f" + good[11:], b"\x80" * 64, good[:20] + b"\0" + good[21:]):
        assert L.bsq_translate_table(bad, m.ctypes.data, c.ctypes.data) == capi.ERR_ARG
    assert L.bsq_translate_table(good, None, c.ctypes.data) == capi.ERR_ARG
    assert L.bsq_translate_table(good, m.ctypes.data, None) == capi.ERR_ARG


# ------------------------------------------------------------------------------------------------------------------
WORKED = "ATGGCCATTGTAATGGGCCGCTGAAAGGGTGCCCGATAG"


def test_worked_answers():
    assert [ref.translate_seq(WORKED, f) for f in SIX] == ["MAIVMGR*KGAR*", "WPL*WAAERVPD", "GHCNGPLKGCPI", "LSGTLSAAHYNGH",
                                                          "YRAPFQRPITMA", "IGHPFSGPLQWP"]
    assert [ref.translate_seq("ATGA", f) for f in SIX] == ["M", "*", "", "S", "H", ""]
    assert [ref.translate_seq("ATGAA", f) for f in SIX] == ["M", "*", "E", "F", "S", "H"]
    for s in ("", "A", "AT"):
        assert [ref.translate_seq(s, f) for f in SIX] == [""] * 6
    table = [("GCN", "A", "A", "X"), ("TAR", "*", "*", "L"), ("TRA", "*", "X", "X"), ("YTG", "L", "L", "Q"), ("atg", "M", "M", "H"),
             ("AUG", "M", "M", "H"), ("A-G", "X", "X", "X"), ("TGA", "*", "W", "S"), ("AGA", "R", "*", "S")]
    for codon, c1, c2, r1 in table:
        assert (ref.translate_seq(codon, 1, 1), ref.translate_seq(codon, 1, 2), ref.translate_seq(codon, -1, 1)) == (c1, c2, r1), codon
    assert ref.translate_seq("ATAAGATGA", 1, 1) == "IR*" and ref.translate_seq("ATAAGATGA", 1, 2) == "M*W"
    assert ref.translate_seq("TAATAG", 1, 6) == "QQ"


def test_vectorised_reference_equals_scalar_one():
    rng = np.random.default_rng(3)
    alphabet = np.frombuffer(b"ACGTUNRYSWKMBDHVacgtun-*.X0\x80\xff", np.uint8)
    lens = np.concatenate([np.arange(8), rng.integers(0, 80, 60)])
    buf = alphabet[rng.integers(0, alphabet.size, int(lens.sum()) + 5)]
    offs = np.concatenate([[5], 5 + np.cumsum(lens)]).astype(np.int64)
    for frames in (SIX, (-2, 3), (-1,), (3, -3, 1)):
        for code in (1, 2, 6, ref.CODES[5]):
            b, o = ref.translate(buf, offs, frames, code)
            assert o[0] == 0 and o.size == lens.size * len(frames) + 1
            for i in range(lens.size):
                for fi, f in enumerate(frames):
                    w = i * len(frames) + fi
                    want = ref.translate_seq(buf[offs[i]:offs[i + 1]].tobytes(), f, code)
                    assert b[o[w]:o[w + 1]].tobytes().decode("latin-1") == want, (i, f, code)


# ------------------------------------------------------------------------------------------------------------------
def ref_extent(lens, frames, crop_len=(1 << 63) - 1):
    L = [max(0, (int(n) - (abs(f) - 1)) // 3) for n in lens for f in frames]
    return sum(L), sum(min(x, crop_len) for x in L), max((min(x, crop_len) for x in L), default=0)


@pytest.mark.parametrize("frames", [SIX, (1,), (-3,), (2, -1), (3, 2, 1, -3, -2)])
def test_extent_host_matches_reference(frames):
    rng = np.random.default_rng(11)
    lens = np.array(list(range(0, 12)) + [47, 48, 49, 50, 51, 150, 151, 152] + list(rng.integers(0, 5000, 300)), np.int64)
    offs = np.concatenate([[7], 7 + np.cumsum(lens)]).astype(np.int64)
    assert capi.translate_extent_host(offs, lens.size, frames) == ref_extent(lens, frames)
    for crop_len in (1, 2, 16, 49, 1000):
        assert capi.translate_extent_host(offs, lens.size, frames, crop_len) == ref_extent(lens, frames, crop_len)
    assert capi.translate_extent_host(offs, 0, frames) == (0, 0, 0)
    # the numpy sizing of host batches agrees
    o = consumers._translate_host_offsets(offs, lens.size, frames)
    assert int(o[-1]) == ref_extent(lens, frames)[0] and o.size == lens.size * len(frames) + 1
    np.testing.assert_array_equal(o, ref.translate(np.zeros(int(offs[-1]), np.uint8), offs, frames)[1])


def test_extent_host_near_int64_max():
    big = np.array([0, 2 ** 62, 2 ** 63 - 1], np.int64)
    assert capi.translate_extent_host(big, 2, (1,)) == ((2 ** 62) // 3 + (2 ** 63 - 1 - 2 ** 62) // 3,) * 2 + ((2 ** 62) // 3,)
    with pytest.raises(ValueError, match="INT64_MAX"):  # six frames of 2^63 - 1 nucleotides: about 2^64 amino acids
        capi.translate_extent_host(big, 2, SIX)


def test_extent_host_rejects_bad_arguments():
    o = np.array([0, 5, 9], np.int64)
    for frames in ((), (0,), (4,), (-4,), (1, 1), (1, 2, 3, -1, -2, -3, 1)):
        with pytest.raises(ValueError):
            capi.translate_extent_host(o, 2, frames)
    with pytest.raises(ValueError):
        capi.translate_extent_host(o, 2, (1,), 0)
    with pytest.raises(ValueError):
        capi.translate_extent_host(np.array([0, 5, 3], np.int64), 2, (1,))
    with pytest.raises(ValueError):
        capi.translate_extent_host(np.array([-1, 5], np.int64), 1, (1,))
    L = capi.lib()
    fa = (C.c_int8 * 1)(1)
    t, c, m = C.c_int64(), C.c_int64(), C.c_int64()
    assert L.bsq_translate_extent_host(None, 2, fa, 1, 5, C.byref(t), C.byref(c), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_translate_extent_host(o.ctypes.data, -1, fa, 1, 5, C.byref(t), C.byref(c), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_translate_extent_host(o.ctypes.data, 2, None, 1, 5, C.byref(t), C.byref(c), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_translate_extent_host(o.ctypes.data, 2, fa, 1, 5, None, C.byref(c), C.byref(m)) == capi.ERR_ARG


def test_c_abi_rejects_bad_arguments():
    L = capi.lib()
    d = C.c_void_p(16)  # never dereferenced: the checks run before any device call
    code = ref.CODES[1].encode()
    t, c, m = C.c_int64(), C.c_int64(), C.c_int64()
    for frames in ((), (0,), (4,), (2, 2), (1, 2, 3, -1, -2, -3, -1)):
        fa = (C.c_int8 * max(len(frames), 1))(*frames)
        assert L.bsq_translate(0, None, d, d, 1, fa, len(frames), code, d, d) == capi.ERR_ARG
        assert L.bsq_translate_extent_device(0, None, d, 1, -1, fa, len(frames), 1, C.byref(t), C.byref(c), C.byref(m)) == capi.ERR_ARG
    fa = (C.c_int8 * 2)(1, -1)
    assert L.bsq_translate(0, None, d, d, 1, None, 2, code, d, d) == capi.ERR_ARG
    assert L.bsq_translate(0, None, d, d, 1, fa, 2, None, d, d) == capi.ERR_ARG
    assert L.bsq_translate(0, None, d, d, 1, fa, 2, b"\x01" * 64, d, d) == capi.ERR_ARG
    assert L.bsq_translate(0, None, d, d, -1, fa, 2, code, d, d) == capi.ERR_ARG
    for bb, o, ob, oo in ((None, d, d, d), (d, None, d, d), (d, d, None, d), (d, d, d, None)):
        assert L.bsq_translate(0, None, bb, o, 3, fa, 2, code, ob, oo) == capi.ERR_ARG
    assert L.bsq_translate_extent_device(0, None, None, 3, -1, fa, 2, 1, C.byref(t), C.byref(c), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_translate_extent_device(0, None, d, -1, -1, fa, 2, 1, C.byref(t), C.byref(c), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_translate_extent_device(0, None, d, 3, -1, fa, 2, 0, C.byref(t), C.byref(c), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_translate_extent_device(0, None, d, 3, -1, fa, 2, 1, None, C.byref(c), C.byref(m)) == capi.ERR_ARG
    assert L.bsq_translate_extent_device(0, None, None, 0, -1, fa, 2, 1, C.byref(t), C.byref(c), C.byref(m)) == capi.OK


def test_frames_and_codes_parsing():
    assert consumers._frames(1) == (1,) and consumers._frames(-3) == (-3,) and consumers._frames(np.int8(2)) == (2,)
    assert consumers._frames("forward") == (1, 2, 3) and consumers._frames("six") == SIX
    assert consumers._frames([-1, 3]) == (-1, 3) and consumers._frames((3, 2, 1)) == (3, 2, 1)
    for bad in (0, 4, -4, "both", "Six", [], [1, 1], (1, 2, 3, -1, -2, -3, 1), 1.0, [1, "2"], None):
        with pytest.raises(ValueError):
            consumers._frames(bad)
    assert consumers._genetic_code(ref.CODES[4]) == ref.CODES[4].encode()
    assert consumers._genetic_code(ref.CODES[4].encode()) == ref.CODES[4].encode()
    for bad in ("ABC", ref.CODES[1] + "A", ref.CODES[1][:63] + " ", 3, 1.0, None):
        with pytest.raises(ValueError):
            consumers._genetic_code(bad)


def test_argument_errors_before_any_device_work():
    from bioseq_b200 import cbioseq
    dna = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
    prot = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    byts = cbioseq.Tokenizer("BYTES")
    seb = cbioseq.Tokenizer("SEB8", bos=True)
    batch = (np.frombuffer(b"ACGTACGTA", np.uint8).copy(), np.array([0, 9], np.int64))
    capi.lib().bsq_launch_count_reset()
    for tok in (dna, cbioseq.Tokenizer("DNA5"), cbioseq.Tokenizer("KETO")):  # nucleotide tokenizers
        with pytest.raises(ValueError, match="protein tokenizer"):
            consumers.batch_tokenize_translated(tok, batch)
        with pytest.raises(ValueError, match="protein tokenizer"):
            consumers.batch_tokenize_varlen(tok, batch, translate=1)
    for tok in (prot, byts, seb):
        consumers._translate_spec("six", 1, tok)
    bad = [dict(frames=0), dict(frames=[1, 1]), dict(frames="all"), dict(genetic_code=3), dict(genetic_code="ACGT"),
           dict(seq_index_base=2 ** 62, frames="six"), dict(padlen=0), dict(varlen=True, padlen=8),
           dict(crop="random"), dict(crop="middle", crop_len=4), dict(crop_len=4), dict(padlen=8, crop="head", crop_len=9)]
    for kw in bad:
        with pytest.raises(ValueError):
            consumers.batch_tokenize_translated(prot, batch, **kw)
    calls = [lambda **kw: consumers.batch_tokenize_cropped(prot, batch, 16, **kw), lambda **kw: consumers.batch_tokenize_varlen(prot, batch, **kw),
             lambda **kw: consumers.batch_tokenize_mlm(prot, batch, 16, **kw), lambda **kw: consumers.batch_tokenize_seqpack(prot, batch, 16, **kw),
             lambda **kw: consumers.batch_tokenize_kmer(prot, batch, 2, 16, **kw),
             lambda **kw: consumers.batch_onehot_encode_bcl(prot, batch, 16, **kw),
             lambda **kw: consumers.batch_embed(prot, batch, _FakeWeight(), 16, **kw)]
    for call in calls:
        for kw in (dict(translate=0), dict(translate="six", genetic_code=7), dict(translate=1, rc="always"),
                   dict(genetic_code=2), dict(translate=(1, -1), seq_index_base=-(2 ** 62) - 1)):
            with pytest.raises(ValueError):
                call(**kw)
    for kw in (dict(translate=1, rc="random"), dict(translate=1, rc="always")):  # nucleotide tokenizer and rc: still rejected
        with pytest.raises(ValueError):
            consumers.batch_tokenize_cropped(dna, batch, 16, **kw)
    with pytest.raises(ValueError, match="mask"):
        consumers.batch_onehot_encode_bcl(prot, batch, 16, mask=np.ones(9, np.uint8), translate=1)
    with pytest.raises(ValueError):
        consumers.translate_packed(batch[0], batch[1])  # host arrays: translate_packed works on CUDA tensors
    for kw in (dict(frames=7), dict(genetic_code=0)):
        with pytest.raises(ValueError):
            consumers.translate_packed(batch[0], batch[1], **kw)
    assert capi.lib().bsq_launch_count() == 0


class _FakeWeight:
    """Stands in for an embedding weight: batch_embed validates its arguments before it touches the weight."""

    def detach(self):
        raise AssertionError("reached the weight")


def test_protein_alphabets_have_no_stop_or_x():
    """AMINO20 / PROTEIN tokenize '*' and 'X' as every invalid byte (id 0, like the reference's LUT); reduced protein
    alphabets do the same, BYTES keeps them."""
    for key in ("PROTEIN", "AMINO20"):
        tok = capi.tokenizer(key)
        assert tok.lut[ord("*")] == -1 and tok.lut[ord("X")] == -1
    tok = capi.tokenizer("BYTES")
    assert tok.nchars == 256


def test_out_base():
    assert consumers._out_base(5, None) == 5
    assert consumers._out_base(5, ((1, -1, 2), b"")) == 15
