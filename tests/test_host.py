"""CPU: the C-ABI library loads and exports what include/bsq.h declares; host logic (alphabet
tables, ids, pack layer, length checks, dtype dispatch) and the Python drop-in surface.
No compute entry point is called here (no GPU in the build container)."""
import ctypes as C
import os
import pickle
import re

import numpy as np
import pytest

import bioseq_b200
from bioseq_b200 import capi
from helpers import gen, as_list

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "bsq.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(bsq_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    L = C.CDLL(capi.LIB_PATH)
    names = declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/bsq.h but not exported by libbsq.so"
    assert sorted(capi.EXPORTS) == names, "capi.py binding list out of sync with include/bsq.h"
    assert capi.lib().bsq_abi_version() == 5


def test_alphabet_registry_and_luts(golden):
    L = capi.lib()
    keys = [L.bsq_alphabet_key(i).decode() for i in range(L.bsq_alphabet_count())]
    assert keys == sorted(golden["alphabets"])          # CAMAP is a std::map: lexicographic order
    for key, g in golden["alphabets"].items():
        for k in (key, key.lower()):
            t = capi.tokenizer(k, eos=True, bos=True, padchar=True)
            assert bytes(np.frombuffer(t.lut, dtype=np.uint8)).hex() == g["lut_hex"], key
            assert (t.nchars, t.bos_id, t.eos_id, t.pad_id, t.alphabet_size) == \
                (g["nchars"], g["bos"], g["eos"], g["pad"], g["alphabet_size"])
            assert t.key.decode() == key
    t = capi.tokenizer("DNA")
    assert (t.bos_id, t.eos_id, t.pad_id, t.alphabet_size, t.padchar) == (-1, -1, 4, 4, 0)
    t = capi.tokenizer("DNA", eos=True)
    assert (t.bos_id, t.eos_id, t.pad_id, t.alphabet_size) == (-1, 4, 5, 5)
    with pytest.raises(RuntimeError, match="Invalid tokenizer type; select one fromAMINO;AMINO20;BYTES;"):
        capi.tokenizer("nope")


def test_lookup_matches_reference_map(golden):
    buf = C.create_string_buffer(8)
    for key, g in golden["alphabets"].items():
        if g["lookup"] is None:
            continue
        t = capi.tokenizer(key, eos=True, bos=True, padchar=True)
        got = {}
        for i in range(-128, 300):
            n = capi.lib().bsq_tokenizer_lookup(C.byref(t), i, buf, 8)
            if n:
                got[str(i)] = buf.raw[:n].decode("latin-1")
        assert got == g["lookup"], key


def test_destchar_dispatch():
    want = {"b": 0, "B": 0, "h": 1, "H": 1, "i": 2, "I": 2, "l": 3, "L": 3, "q": 3, "Q": 3, "f": 4, "F": 4, "d": 5, "D": 5}
    for ch, k in want.items():
        assert capi.kind_of(ch) == k
    for ch in "xuUe?1":
        with pytest.raises(ValueError, match="Unsupported dtype: "):
            capi.kind_of(ch)
    assert [capi.lib().bsq_kind_size(k) for k in range(7)] == [1, 2, 4, 8, 4, 8, 0]


def test_pack_layer_pageable():
    buf, offs = gen(7, 3000, 0, 900, b"ACGTN")
    seqs = as_list(buf, offs)
    for nthreads in (1, 4):
        p = capi.Pack(pinned=False).gather(seqs, nthreads=nthreads)
        b, o = p.to_numpy()
        assert p.nseq == len(seqs) and p.nbytes == buf.size and p.maxlen == int(np.diff(offs).max())
        assert np.array_equal(b, buf) and np.array_equal(o, offs)
        p.gather([])            # reusable; empty batch
        assert p.nseq == 0 and p.nbytes == 0
        p.close()


def test_length_checks_host():
    offs = np.array([0, 4, 4, 10], dtype=np.int64)
    t = capi.tokenizer("DNA", eos=True, bos=True)
    capi.check_lengths_host(offs, 3, 8, t)
    with pytest.raises(RuntimeError, match=r"seq len \+ bos \+ eos > padlen: 8, vs padlen 7"):
        capi.check_lengths_host(offs, 3, 7, t)
    with pytest.raises(ValueError, match=r"seq len \+ bos \+ eos > padlen: 8, vs padlen 7"):
        capi.check_lengths_host(offs, 3, 7, t, onehot=True)
    with pytest.raises(ValueError, match="batch tokenize requires padlen is provded."):
        capi.check_lengths_host(offs, 3, 0, t)
    with pytest.raises(ValueError):
        capi.check_lengths_host(np.array([0, 5, 3], dtype=np.int64), 2, 10, t)
    with pytest.raises(ValueError, match="offsets must start at or after 0"):
        capi.check_lengths_host(np.array([-1, 2, 3], dtype=np.int64), 2, 10, t)


def test_python_surface_names_and_keys():
    b = bioseq_b200
    fams = {"pbeos_tokenizers": (1, 1, 1), "beos_tokenizers": (1, 1, 0), "pbos_tokenizers": (1, 0, 1),
            "bos_tokenizers": (1, 0, 0), "peos_tokenizers": (0, 1, 1), "eos_tokenizers": (0, 1, 0),
            "pos_tokenizers": (0, 0, 1)}
    assert len(b.bkeys) == 34 and len(set(b.bkeys)) == 32
    for name, (bos, eos, pad) in fams.items():
        d = getattr(b, name)
        assert set(d) == set(b.bkeys)
        for k, t in d.items():
            assert t.key == k.upper()
            assert (t.includes_bos(), t.includes_eos(), t.is_padded()) == (bool(bos), bool(eos), bool(pad))
        assert b.get_tokenizer_dict(bos, eos, pad) is d
    assert b.get_tokenizer_dict(0, 0, 0) is b.default_tokenizers
    assert set(b.default_tokenizers) == {"DNA", "AMINO20", "AMINE", "PROTEIN", "SEB6", "SEB8", "SEB10", "SEB14",
                                         "LIA10", "LIA", "LIB10", "LIB"}
    assert len(b.total_tokenizer_dict) == 8 * 32
    t = b.pbeos_tokenizers["PROTEIN"]
    assert (t.nchars(), t.bos(), t.eos(), t.pad(), t.alphabet_size()) == (20, 20, 21, 22, 23)
    t = b.Tokenizer("dna")            # kwarg order key, eos, bos, padchar (src/tokenize.cpp:23)
    assert (t.bos(), t.eos(), t.pad(), t.alphabet_size()) == (-1, -1, 4, 4)
    t = b.Tokenizer("DNA", True, False, True)
    assert (t.includes_eos(), t.includes_bos(), t.is_padded(), t.eos(), t.pad()) == (True, False, True, 4, 5)


def test_tokenizer_introspection_and_pickle(golden):
    for key, g in golden["alphabets"].items():
        if g["lookup"] is None:
            continue
        t = bioseq_b200.Tokenizer(key, bos=True, eos=True, padchar=True)
        assert {str(k): v for k, v in t.lut().items()} == g["lookup"]
        assert sorted(t.token_map().split(";")) == sorted(f"{k}:{v}" for k, v in g["lookup"].items())
        dec = t.token_decoder()
        lut = np.frombuffer(bytes.fromhex(g["lut_hex"]), dtype=np.int8)
        for ident, members in dec.items():
            assert all(lut[m] == ident for m in members)
        assert sum(len(v) for v in dec.values()) == 256
        t2 = pickle.loads(pickle.dumps(t))
        assert (t2.key, t2.includes_eos(), t2.includes_bos(), t2.is_padded()) == (key, True, True, True)
    assert bioseq_b200.Tokenizer("DNA", eos=True).__getstate__() == ("DNA", True, False, False)


def test_argument_errors_precede_device_use():
    t = bioseq_b200.pbeos_tokenizers["DNA"]
    with pytest.raises(ValueError, match="batch tokenize requires padlen is provded."):
        t.batch_tokenize(["ACGT"])
    with pytest.raises(ValueError, match="Unsupported dtype: x"):
        t.batch_tokenize(["ACGT"], padlen=8, destchar="x")
    with pytest.raises(ValueError, match="Unsupported dtype: u"):
        t.batch_onehot_encode(["ACGT"], padlen=8, destchar="u")
    with pytest.raises(ValueError, match="item was none of string, bytes, or numpy array of 8-bit integers. "):
        t.batch_tokenize(["ACGT", 5], padlen=8)
    with pytest.raises(ValueError, match="item was none of string"):
        t.batch_tokenize([np.frombuffer(b"ACGT", dtype=np.uint8)], padlen=8)   # src/tokenize.h:406-416


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    t = bioseq_b200.pbeos_tokenizers["DNA"]
    with pytest.raises(RuntimeError, match="no CUDA device available"):
        t.batch_tokenize(["ACGT"], padlen=8, batch_first=True)
    with pytest.raises(RuntimeError, match="no CUDA device available"):
        t.decode_tokens(np.zeros(4, dtype=np.uint8))


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "bioseq_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle" not in text.lower() or f == "synth.py", f"{f} mentions the oracle"


def test_library_reads_only_the_documented_environment_variable():
    # The shipped kernels run one measured configuration each; no environment variable may select another.
    # BSQ_POOL_CAP (INTEGRATION.md) sizes the host worker pool and is the one variable the library reads.
    csrc = os.path.join(ROOT, "bioseq_b200", "csrc")
    calls = []
    for f in sorted(os.listdir(csrc)):
        text = open(os.path.join(csrc, f), errors="ignore").read()
        calls += [(f, arg.strip()) for arg in re.findall(r"\b\w*getenv\s*\(([^)]*)\)", text)]
    assert [arg for _, arg in calls] == ['"BSQ_POOL_CAP"'], calls


def test_parallel_for_runs_every_share_once():
    # the persistent host worker pool behind the gather / scatter loops (no GPU involved)
    L = capi.lib()
    CB = C.CFUNCTYPE(None, C.c_int, C.c_int, C.c_void_p)
    for nthreads in (1, 2, 5):
        seen = []
        cb = CB(lambda t, nt, ctx: seen.append((t, nt)))
        for _ in range(3):                       # the pool is reused job after job
            seen.clear()
            assert L.bsq_parallel_for(nthreads, C.cast(cb, C.c_void_p), None) == 0
            nt = seen[0][1]
            assert 1 <= nt <= nthreads           # capped at half the hardware threads
            assert sorted(seen) == [(t, nt) for t in range(nt)]
    assert L.bsq_parallel_for(2, None, None) == capi.ERR_ARG


@pytest.mark.filterwarnings("ignore::DeprecationWarning")
def test_parallel_for_after_fork():
    # a forked child has none of the parent's pool threads: it must start its own instead of waiting for them
    import os
    L = capi.lib()
    CB = C.CFUNCTYPE(None, C.c_int, C.c_int, C.c_void_p)
    hits = []
    cb = CB(lambda t, nt, ctx: hits.append(t))
    assert L.bsq_parallel_for(4, C.cast(cb, C.c_void_p), None) == 0      # parent's pool exists now
    pid = os.fork()
    if pid == 0:
        ok = 1
        try:
            import signal
            signal.alarm(20)                                            # a deadlock ends the child, not the test run
            hits.clear()
            if L.bsq_parallel_for(4, C.cast(cb, C.c_void_p), None) == 0 and sorted(hits) == list(range(len(hits))) and hits:
                ok = 0
        finally:
            os._exit(ok)
    _, status = os.waitpid(pid, 0)
    assert os.WIFEXITED(status) and os.WEXITSTATUS(status) == 0
