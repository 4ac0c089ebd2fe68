"""CPU: reverse complement (revcomp_packed / rc= / bsq_revcomp, kernel K12) without a device.

The entry points are declared, exported and bound; the numpy reference of the rule (tests/revcomp_reference.py, what the
GPU tests compare with) is checked against the library's own table, a scalar restatement of the header's pairs, the
header's worked answers and the oracle's C Philox, and its statistics (the flip rate, independence of slicing); every
argument error is raised before anything is staged or launched, and the C ABI rejects bad arguments without a device."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from bioseq_b200 import capi, consumers
from oracle import oracle
from helpers import gen
from revcomp_reference import revcomp as reference_revcomp, coins as reference_coins, table as reference_table

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_revcomp_entry_points_declared_exported_and_bound():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bsq.h")).read(), flags=re.S)
    L = C.CDLL(capi.LIB_PATH)
    for name in ("bsq_revcomp", "bsq_revcomp_table"):
        assert re.search(r"\b" + name + r"\s*\(", src), f"{name} not declared in include/bsq.h"
        assert hasattr(L, name) and name in capi.EXPORTS
        assert getattr(capi.lib(), name).argtypes is not None
    for name, value in (("BSQ_RC_ALWAYS", capi.RC_ALWAYS), ("BSQ_RC_RANDOM", capi.RC_RANDOM), ("BSQ_RC_BOTH", capi.RC_BOTH)):
        assert re.search(r"#define\s+" + name + r"\s+" + str(value) + r"\b", src)
    import bioseq_b200
    for name in ("revcomp_packed", "batch_tokenize_revcomp", "RevCompBatch"):
        assert name in bioseq_b200.__all__ and hasattr(bioseq_b200, name)


# ------------------------------------------------------------------------------------------------------------------
def test_table_matches_library_and_header_pairs():
    lib_table = capi.revcomp_table()
    assert np.array_equal(reference_table(), lib_table)
    # the header's text, byte by byte
    pairs = {"A": "T", "T": "A", "C": "G", "G": "C", "R": "Y", "Y": "R", "K": "M", "M": "K", "B": "V", "V": "B", "D": "H",
             "H": "D", "S": "S", "W": "W", "N": "N", "U": "A"}
    for b in range(256):
        c = chr(b)
        if c in pairs:
            want = ord(pairs[c])
        elif c.isascii() and c.islower() and c.upper() in pairs:
            want = ord(pairs[c.upper()].lower())
        else:
            want = b
        assert int(lib_table[b]) == want, (b, int(lib_table[b]), want)


@pytest.mark.parametrize("seq,want", [("ACGTN", "NACGT"), ("GATTACA", "TGTAATC"), ("ACGU", "ACGT"),
                                      ("acgRYkmBDHVswn-*", "*-nwsBDHVkmRYcgt"), ("", "")])
def test_worked_answers(seq, want):
    b = np.frombuffer(seq.encode(), np.uint8)
    out, offs, flipped = reference_revcomp(b, [0, b.size], "always")
    assert out.tobytes() == want.encode() and offs.tolist() == [0, b.size] and flipped.tolist() == [True]
    out, offs, flipped = reference_revcomp(b, [0, b.size], "both")
    assert out.tobytes() == (seq + want).encode() and offs.tolist() == [0, b.size, 2 * b.size]
    assert flipped.tolist() == [False, True]


def scalar_coins(n, rc_prob, seed, base):
    """The header's coin written again from its text with the oracle's C Philox, one sequence at a time."""
    gate = 1 << 32 if rc_prob >= 1 else math.floor(rc_prob * 2 ** 32)
    out = []
    for i in range(n):
        g = base + i
        x0 = int(oracle.philox4x32_10((g & 0xFFFFFFFF, g >> 32, 0, 4), (seed & 0xFFFFFFFF, seed >> 32))[0])
        out.append(x0 < gate)
    return out


def test_worked_coins_against_the_oracle_philox():
    assert reference_coins(8, 0.5, 7, 0).astype(int).tolist() == [1, 0, 1, 1, 1, 1, 1, 1]
    assert [int(oracle.philox4x32_10((g, 0, 0, 4), (7, 0))[0]) for g in range(3)] == [407685168, 3339964855, 305774060]
    assert reference_coins(8, 0.5, 0x123456789ABCDEF0, 2 ** 32 + 11).astype(int).tolist() == [1, 0, 0, 0, 1, 0, 1, 1]
    for rc_prob, seed, base in ((0.5, 7, 0), (0.3, 0x123456789ABCDEF0, 2 ** 32 + 11), (0.0, 1, 5), (1.0, 2, 6), (0.999, 3, 2 ** 40)):
        assert reference_coins(300, rc_prob, seed, base).tolist() == scalar_coins(300, rc_prob, seed, base)
    assert not reference_coins(1000, 0.0, 9).any() and reference_coins(1000, 1.0, 9).all()


@pytest.mark.parametrize("rc_prob", [0.5, 0.3])
def test_flip_rate_within_binomial_bounds(rc_prob):
    n = 200_000
    k = int(reference_coins(n, rc_prob, seed=2024).sum())
    sd = math.sqrt(n * rc_prob * (1 - rc_prob))
    assert abs(k - n * rc_prob) < 5 * sd
    # another seed draws other coins
    assert not np.array_equal(reference_coins(n, rc_prob, 2024), reference_coins(n, rc_prob, 2025))


def test_flips_independent_of_slicing_and_length():
    buf, offs = gen(8, 3000, 0, 400, b"ACGT")
    full = reference_revcomp(buf, offs, "random", 0.5, 77, 0)
    for a, b in ((0, 1), (1, 999), (999, 2500), (2500, 3000)):
        part = reference_revcomp(buf, offs[a:b + 1], "random", 0.5, 77, a)
        assert np.array_equal(part[2], full[2][a:b])
        assert np.array_equal(part[0], full[0][full[1][a]:full[1][b]])
        assert np.array_equal(part[1], full[1][a:b + 1] - full[1][a])
    # the coin of a sequence does not depend on its length
    other = reference_revcomp(buf[:10], np.minimum(offs, 10), "random", 0.5, 77, 0)
    assert np.array_equal(other[2], full[2])


def test_flip_twice_is_identity():
    # every byte but U / u (U -> A -> T) is an involution of the table
    alphabet = bytes(b for b in range(256) if b not in (ord("U"), ord("u")))
    buf, offs = gen(3, 500, 0, 300, alphabet)
    offs = offs + 2
    buf = np.concatenate([np.zeros(2, np.uint8), buf])
    once = reference_revcomp(buf, offs, "always")
    twice = reference_revcomp(once[0], once[1], "always")
    assert np.array_equal(twice[0], buf[offs[0]:offs[-1]]) and np.array_equal(twice[1], offs - offs[0])
    # in random mode the same coins undo their own flips
    once = reference_revcomp(buf, offs, "random", 0.5, 11, 4)
    twice = reference_revcomp(once[0], once[1], "random", 0.5, 11, 4)
    assert np.array_equal(twice[0], buf[offs[0]:offs[-1]])


# ------------------------------------------------------------------------------------------------------------------
def test_rc_spec():
    assert consumers._rc_spec(None, None, 1, 2) is None
    assert consumers._rc_spec("always", None, 1, 2) == (capi.RC_ALWAYS, 0.0, 1, 2)
    assert consumers._rc_spec("random", None, 1, 2) == (capi.RC_RANDOM, 0.5, 1, 2)
    assert consumers._rc_spec("random", 0.25, 1, 2) == (capi.RC_RANDOM, 0.25, 1, 2)
    assert consumers._rc_spec("both", None, 1, 2) == (capi.RC_BOTH, 0.0, 1, 2)
    for key in ("DNA", "DNA4", "DNA5", "DNAMETH", "C", "KETO", "PURPYR", "dna5"):
        assert consumers._rc_spec("random", None, 0, 0, capi.tokenizer(key.upper())) is not None
    for args in (("flip", None), (True, None), (["both"], None), (None, 0.5), ("always", 0.5), ("both", 0.5),
                 ("random", -0.1), ("random", 1.5), ("random", float("nan")), ("random", "half")):
        with pytest.raises(ValueError):
            consumers._rc_spec(*args, 0, 0)


def test_argument_errors_before_any_device_work():
    # every rc ValueError of the consumers is raised before the batch is staged (no device is touched here)
    from bioseq_b200 import cbioseq
    dna = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
    batch = (np.frombuffer(b"ACGTACGTA", np.uint8).copy(), np.array([0, 9], np.int64))
    weight = np.zeros((32, 16), np.float32)
    capi.lib().bsq_launch_count_reset()
    bad = [dict(rc="flip"), dict(rc=None, rc_prob=0.5), dict(rc="always", rc_prob=0.5), dict(rc="random", rc_prob=2.0),
           dict(rc="random", rc_prob=float("nan")), dict(rc="random", augment=1), dict(rc="both", augment=1)]
    for kw in bad:
        calls = [lambda: consumers.batch_onehot_encode_bcl(dna, batch, 16, **kw),
                 lambda: consumers.batch_tokenize_mlm(dna, batch, 16, **kw),
                 lambda: consumers.batch_embed(dna, batch, weight, 16, **kw),
                 lambda: consumers.batch_tokenize_cropped(dna, batch, 16, **kw),
                 lambda: consumers.batch_tokenize_seqpack(dna, batch, 16, **kw)]
        if "augment" not in kw:
            calls += [lambda: consumers.batch_tokenize_varlen(dna, batch, **kw),
                      lambda: consumers.batch_tokenize_mlm(dna, batch, varlen=True, **kw),
                      lambda: consumers.batch_tokenize_kmer(dna, batch, 3, 16, **kw),
                      lambda: consumers.batch_tokenize_kmer(dna, batch, 3, varlen=True, **kw)]
            if kw.get("rc") is not None:
                calls.append(lambda: consumers.batch_tokenize_revcomp(dna, batch, 16, **kw))
        for call in calls:
            with pytest.raises(ValueError):
                call()
    # protein, reduced-protein and byte alphabets have no complement
    for key in ("PROTEIN", "AMINO20", "SEB6", "DAYHOFF", "BYTES"):
        tok = cbioseq.Tokenizer(key, bos=True, eos=True, padchar=True)
        for call in (lambda: consumers.batch_tokenize_revcomp(tok, batch, 16),
                     lambda: consumers.batch_tokenize_varlen(tok, batch, rc="always"),
                     lambda: consumers.batch_onehot_encode_bcl(tok, batch, 16, rc="both"),
                     lambda: consumers.batch_tokenize_mlm(tok, batch, 16, rc="random")):
            with pytest.raises(ValueError):
                call()
    # "both" doubles the batch for inference: not with a masked-language-model batch
    for call in (lambda: consumers.batch_tokenize_mlm(dna, batch, 16, rc="both"),
                 lambda: consumers.batch_tokenize_mlm(dna, batch, varlen=True, rc="both"),
                 lambda: consumers.batch_tokenize_seqpack(dna, batch, 16, mlm=True, rc="both")):
        with pytest.raises(ValueError):
            call()
    with pytest.raises(ValueError):  # a residue mask covers the unflipped batch
        consumers.batch_onehot_encode_bcl(dna, batch, 16, mask=np.ones(9, np.uint8), rc="always")
    with pytest.raises(ValueError):
        consumers.batch_tokenize_revcomp(dna, batch, 16, rc=None)
    with pytest.raises(ValueError):
        consumers.revcomp_packed(batch[0], batch[1])  # host arrays: revcomp_packed works on CUDA tensors
    assert capi.lib().bsq_launch_count() == 0


def test_c_abi_rejects_bad_arguments():
    L = capi.lib()
    d = C.c_void_p(16)  # never dereferenced: the checks run before any device call
    for mode in (-1, 3, 7):
        assert L.bsq_revcomp(0, None, d, d, 1, mode, 0.5, 0, 0, d, d, None) == capi.ERR_ARG
    assert "mode" in capi.last_error()
    for p in (float("nan"), -0.5, -1e-300):
        assert L.bsq_revcomp(0, None, d, d, 1, capi.RC_RANDOM, p, 0, 0, d, d, None) == capi.ERR_ARG
        assert L.bsq_revcomp(0, None, d, d, 1, capi.RC_ALWAYS, p, 0, 0, d, d, None) == capi.ERR_ARG
    assert "rc_prob" in capi.last_error()
    assert L.bsq_revcomp(0, None, d, d, -1, capi.RC_ALWAYS, 0.5, 0, 0, d, d, None) == capi.ERR_ARG
    for b, o, ob, oo in ((None, d, d, d), (d, None, d, d), (d, d, None, d), (d, d, d, None)):
        assert L.bsq_revcomp(0, None, b, o, 3, capi.RC_BOTH, 0.5, 0, 0, ob, oo, None) == capi.ERR_ARG
    assert L.bsq_revcomp(0, None, None, None, 0, capi.RC_ALWAYS, 0.5, 0, 0, None, None, None) == capi.ERR_ARG
    assert L.bsq_revcomp_table(None) == capi.ERR_ARG


def test_dataset_arguments():
    from bioseq_b200 import cbioseq, loaders
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "x.ff")
        with open(path, "wb") as f:
            f.write(oracle.flatfile_image([b"ACGTACGTAC" * 10, b"ACG"]))
        ff = cbioseq.FlatFile(path)
        dna = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
        ds = loaders.FlatFileDataset(ff, dna, rc="random")
        assert (ds.rc, ds.rc_prob) == ("random", 0.5)
        assert loaders.FlatFileDataset(ff, dna, rc="random", rc_prob=0.25, max_seq_len=32).rc_prob == 0.25
        assert loaders.FlatFileDataset(ff, dna).rc is None
        prot = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
        for tok, kw in ((dna, dict(rc="both")), (dna, dict(rc="always")), (dna, dict(rc="flip")), (prot, dict(rc="random")),
                        (dna, dict(rc="random", augment=1)), (dna, dict(rc="random", rc_prob=1.5))):
            with pytest.raises(ValueError):
                loaders.FlatFileDataset(ff, tok, **kw)
