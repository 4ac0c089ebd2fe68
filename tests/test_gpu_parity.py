"""GPU parity: the CUDA path, driven through the C ABI (bioseq_b200.capi -> libbsq.so) and
through the drop-in Python class, against the oracle (oracle/bsq_oracle.c, pinned to the
reference by tests/test_oracle.py) and the committed golden fixtures.  Bit-exact everywhere:
raw bytes + shape for arrays, string equality for decoded text."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import bioseq_b200  # noqa: E402
from bioseq_b200 import capi  # noqa: E402
from oracle.oracle import OracleTokenizer, alphabet_keys, load_ref  # noqa: E402
from helpers import sha, sha_strs, assert_same_bits, golden_inputs, gen, gen_mask, as_list, Reference  # noqa: E402

TORCH_DT = {0: torch.int8, 1: torch.int16, 2: torch.int32, 3: torch.int64, 4: torch.float32, 5: torch.float64}
MIX = b"ACDEFGHIKLMNPQRSTVWYacdefghiklmnpqrstvwyXBZOUJ*-NnUu .\x00\x7f\x80\xc3\xff"


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests selected but no CUDA device is visible")


def to_dev(a):
    a = np.ascontiguousarray(a)
    return torch.from_numpy(a.copy()).cuda() if a.size else torch.empty(0, dtype=torch.from_numpy(a).dtype, device="cuda")


def stream():
    return torch.cuda.current_stream().cuda_stream


def abi_tokenize(tok, buf, offs, padlen, batch_first, destchar, d_bytes=None):
    kind = capi.kind_of(destchar)
    n = len(offs) - 1
    d_bytes = to_dev(buf) if d_bytes is None else d_bytes
    d_offs = to_dev(offs)
    out = torch.empty((n, padlen) if batch_first else (padlen, n), dtype=TORCH_DT[kind], device="cuda")
    capi.tokenize(0, stream(), d_bytes, d_offs, n, padlen, tok, batch_first, kind, out)
    torch.cuda.synchronize()
    return out


def abi_onehot(tok, buf, offs, mask, padlen, destchar):
    kind = capi.kind_of(destchar)
    n = len(offs) - 1
    out = torch.empty((padlen, n, tok.alphabet_size), dtype=TORCH_DT[kind], device="cuda")
    capi.onehot(0, stream(), to_dev(buf), to_dev(offs), None if mask is None else to_dev(mask), n, padlen, tok, kind, out)
    torch.cuda.synchronize()
    return out


def abi_decode(tok, d_tokens):
    """decode a 1-D/2-D CUDA tensor through bsq_decode_lengths + bsq_decode_chars."""
    nd = d_tokens.dim()
    es = d_tokens.element_size()
    rows, cols = (1, d_tokens.shape[0]) if nd == 1 else d_tokens.shape
    rs, cs = (0, d_tokens.stride(0) * es) if nd == 1 else (d_tokens.stride(0) * es, d_tokens.stride(1) * es)
    d_offs = torch.empty(rows + 1, dtype=torch.int64, device="cuda")
    outs = []
    for with_tail in (True, False):   # with and without the trailing-run hint buffer: the text must not depend on it
        d_tail = torch.empty(rows, dtype=torch.int32, device="cuda") if with_tail else None
        total = capi.decode_lengths(0, stream(), d_tokens, es, rows, cols, rs, cs, tok, d_offs, d_tail)
        d_chars = torch.full((total,), 0x7e, dtype=torch.uint8, device="cuda")
        capi.decode_chars(0, stream(), d_tokens, es, rows, cols, rs, cs, tok, d_offs, d_chars, d_tail)
        raw = d_chars.cpu().numpy().tobytes()
        o = d_offs.cpu().numpy()
        outs.append([raw[o[i]:o[i + 1]].decode("latin-1") for i in range(rows)])
    assert outs[0] == outs[1]
    # the one-call form (bsq_decode_text): a buffer that is large enough is filled; one that is too small is not
    # touched and the exactly sized second pass gives the same text
    d_tail = torch.empty(rows, dtype=torch.int32, device="cuda")
    cap = 5 * rows * cols + 16
    d_chars = torch.full((cap,), 0x7e, dtype=torch.uint8, device="cuda")
    total = capi.decode_text(0, stream(), d_tokens, es, rows, cols, rs, cs, tok, d_offs, d_tail, d_chars, cap)
    raw = d_chars.cpu().numpy().tobytes()
    o = d_offs.cpu().numpy()
    assert total == o[rows] and [raw[o[i]:o[i + 1]].decode("latin-1") for i in range(rows)] == outs[0]
    assert raw[total:] == b"\x7e" * (cap - total)
    if total > 1:
        small = torch.full((total - 1,), 0x7e, dtype=torch.uint8, device="cuda")
        assert capi.decode_text(0, stream(), d_tokens, es, rows, cols, rs, cs, tok, d_offs, d_tail, small, total - 1) == total
        assert bool((small == 0x7e).all())
        exact = torch.empty(total, dtype=torch.uint8, device="cuda")
        capi.decode_chars(0, stream(), d_tokens, es, rows, cols, rs, cs, tok, d_offs, exact, d_tail)
        assert exact.cpu().numpy().tobytes() == raw[:total]
    out = outs[0]
    return out[0] if nd == 1 else out


def split_mask(mask, offs):
    return None if mask is None else [mask[offs[i]:offs[i + 1]] for i in range(len(offs) - 1)]


# ------------------------------------------------------------------------------------- golden
def test_golden_kats_python_api(golden):
    for rec in golden["kats"]:
        t = bioseq_b200.Tokenizer(rec["key"], **rec["flags"])
        if rec["op"] == "tokenize":
            out = t.batch_tokenize(rec["seqs"], padlen=rec["padlen"], **rec["kw"])
            assert out.is_cuda
            assert out.cpu().numpy().tolist() == rec["out"], rec
            assert t.decode_tokens(out) == rec["decoded"], rec
            assert t.decode_tokens(out.cpu().numpy()) == rec["decoded"], rec
        else:
            out = t.batch_onehot_encode(rec["seqs"], padlen=rec["padlen"], **rec["kw"])
            assert out.cpu().numpy().tolist() == rec["out"], rec
        assert out.element_size() == np.dtype(rec["dtype"]).itemsize


def test_readme_example():
    # /root/reference/README.md:38-44
    t = bioseq_b200.pbeos_tokenizers["DNA"]
    out = t.batch_tokenize(["ACGT", "GGGG"], padlen=7, batch_first=True)
    assert out.dtype == torch.uint8 and out.device.type == "cuda"
    assert out.cpu().tolist() == [[4, 0, 1, 2, 3, 5, 6], [4, 2, 2, 2, 2, 5, 6]]
    assert t.decode_tokens(out) == ["<BOS>ACGT<EOS><PAD>", "<BOS>GGGG<EOS><PAD>"]


def test_golden_hashes_all_entry_points(golden):
    stager = capi.Stager(0)
    for rec in golden["hashes"]:
        buf, offs, mask = golden_inputs(rec)
        n = len(offs) - 1
        tok = capi.tokenizer(rec["key"], **rec["flags"])
        pt = bioseq_b200.Tokenizer(rec["key"], **rec["flags"])
        dc = rec["kw"].get("destchar", "B")
        kind = capi.kind_of(dc)
        if rec["op"] == "tokenize":
            bf = rec["kw"]["batch_first"]
            a = abi_tokenize(tok, buf, offs, rec["padlen"], bf, dc)
            b = torch.empty_like(a)
            stager.tokenize_host(stream(), buf, offs, n, rec["padlen"], tok, bf, kind, b)
            c = pt.batch_tokenize(as_list(buf, offs), padlen=rec["padlen"], **rec["kw"])
            d = pt.batch_tokenize_packed(buf, offs, padlen=rec["padlen"], **rec["kw"])
            e = pt.batch_tokenize_packed(to_dev(buf), to_dev(offs), padlen=rec["padlen"], **rec["kw"])
            if "decode_sha" in rec:
                assert sha_strs(abi_decode(tok, a)) == rec["decode_sha"], rec["name"]
                assert sha_strs(pt.decode_tokens(c)) == rec["decode_sha"], rec["name"]
        else:
            a = abi_onehot(tok, buf, offs, mask, rec["padlen"], dc)
            b = torch.empty_like(a)
            stager.onehot_host(stream(), buf, offs, mask, n, rec["padlen"], tok, kind, b)
            kw = dict(rec["kw"])
            c = pt.batch_onehot_encode(as_list(buf, offs), padlen=rec["padlen"], mask=split_mask(mask, offs), **kw)
            d = pt.batch_onehot_encode_packed(buf, offs, padlen=rec["padlen"], mask=mask, **kw)
            e = pt.batch_onehot_encode_packed(to_dev(buf), to_dev(offs), padlen=rec["padlen"],
                                              mask=None if mask is None else to_dev(mask), **kw)
        torch.cuda.synchronize()
        for name, x in (("abi", a), ("staged", b), ("py-list", c), ("py-packed-host", d), ("py-packed-dev", e)):
            x = x.cpu().numpy()
            assert list(x.shape) == rec["shape"] and x.itemsize == rec["itemsize"], (rec["name"], name)
            assert sha(x) == rec["sha"], (rec["name"], name)
    stager.close()


# ------------------------------------------------------------------------------------- differential
@pytest.mark.parametrize("seed", range(8))
def test_random_batches_vs_oracle(seed):
    rng = np.random.default_rng(4200 + seed)
    keys = alphabet_keys()
    for trial in range(10):
        key = keys[int(rng.integers(len(keys)))]
        flags = dict(bos=bool(rng.integers(2)), eos=bool(rng.integers(2)), padchar=bool(rng.integers(2)))
        n = int(rng.choice([0, 1, 2, 15, 16, 17, 127, 128, 129, 200, 333]))
        hi = int(rng.choice([0, 1, 5, 15, 16, 17, 31, 64, 100, 257]))
        buf, offs = gen(int(rng.integers(1 << 30)), n, 0, hi, MIX)
        padlen = max(1, hi + 2 + int(rng.choice([0, 0, 1, 3, 14, 16, 30])))
        dc = "bBhilqfd"[int(rng.integers(8))]
        bf = bool(rng.integers(2))
        tok, orc = capi.tokenizer(key, **flags), OracleTokenizer(key, **flags)
        want = orc.batch_tokenize((buf, offs), padlen=padlen, destchar=dc, batch_first=bf)
        got = abi_tokenize(tok, buf, offs, padlen, bf, dc)
        assert_same_bits(want, got.cpu().numpy())
        if dc not in "fd" and n:
            assert abi_decode(tok, got) == orc.decode_tokens(want)
            assert abi_decode(tok, got.t()) == orc.decode_tokens(want.T)
            assert abi_decode(tok, got[::2, 1::3]) == orc.decode_tokens(want[::2, 1::3])
            assert abi_decode(tok, got[0]) == orc.decode_tokens(want[0])
        mask = gen_mask(int(rng.integers(1 << 30)), buf.size, 0.7) if rng.integers(2) else None
        want = orc.batch_onehot_encode((buf, offs), padlen=padlen, destchar=dc, mask=split_mask(mask, offs))
        got = abi_onehot(tok, buf, offs, mask, padlen, dc)
        assert_same_bits(want, got.cpu().numpy())


def test_every_alphabet_every_dtype_both_layouts():
    buf, offs = gen(99, 261, 0, 140, MIX)
    for key in alphabet_keys():
        for flags in (dict(), dict(bos=True, eos=True, padchar=True), dict(eos=True), dict(bos=True, padchar=True)):
            tok, orc = capi.tokenizer(key, **flags), OracleTokenizer(key, **flags)
            for dc in "bhiqfd":
                for padlen in (144, 147):
                    for bf in (True, False):
                        want = orc.batch_tokenize((buf, offs), padlen=padlen, destchar=dc, batch_first=bf)
                        assert_same_bits(want, abi_tokenize(tok, buf, offs, padlen, bf, dc).cpu().numpy())
                want = orc.batch_onehot_encode((buf, offs), padlen=143, destchar=dc)
                assert_same_bits(want, abi_onehot(tok, buf, offs, None, 143, dc).cpu().numpy())


def test_unaligned_device_buffers_and_offset_base():
    # residues starting at every byte alignment, offsets that do not start at zero
    buf, offs = gen(5, 300, 0, 70, MIX)
    tok, orc = capi.tokenizer("PROTEIN", bos=True, eos=True, padchar=True), OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    want_t = orc.batch_tokenize((buf, offs), padlen=80, batch_first=True)
    want_s = orc.batch_tokenize((buf, offs), padlen=80, batch_first=False)
    want_o = orc.batch_onehot_encode((buf, offs), padlen=80, destchar="f")
    for shift in range(0, 18):
        big = torch.zeros(buf.size + 64, dtype=torch.uint8, device="cuda")
        big[shift:shift + buf.size] = to_dev(buf)
        view = big[shift:]
        n = len(offs) - 1
        assert_same_bits(want_t, abi_tokenize(tok, buf, offs, 80, True, "B", d_bytes=view).cpu().numpy())
        assert_same_bits(want_s, abi_tokenize(tok, buf, offs, 80, False, "B", d_bytes=view).cpu().numpy())
        # same bytes, but offsets carry a base: pass a pointer moved back by `shift`
        out = torch.empty((80, n, 23), dtype=torch.float32, device="cuda")
        capi.onehot(0, stream(), big.data_ptr(), to_dev(offs + shift), None, n, 80, tok, capi.F32, out)
        torch.cuda.synchronize()
        assert_same_bits(want_o, out.cpu().numpy())


@pytest.mark.parametrize("flags", [dict(), dict(bos=True, eos=True, padchar=True), dict(eos=True), dict(bos=True)])
def test_tma_row_kernel_shapes(flags):
    # one-byte batch-first output with padlen % 16 == 0 and > 256 goes through the persistent
    # TMA-fed kernel: empty rows, rows that fill padlen exactly, every source alignment, more rows
    # than one 32-row batch per warp of the persistent grid, and an unaligned residue buffer
    tok, orc = capi.tokenizer("PROTEIN", **flags), OracleTokenizer("PROTEIN", **flags)
    extra = int(flags.get("bos", False)) + int(flags.get("eos", False))
    # ... and padlens that are not a multiple of 16 (rows own the aligned vectors that END inside them; a
    # nearly full previous row reaches into the next row's first vector)
    for n, padlen, hi in ((1, 272, 270), (3000, 272, 270 - extra + extra), (777, 1024, 1024), (65, 4096, 4096), (200_000, 272, 40),
                          (1, 1026, 1000), (2, 257, 257), (3001, 273, 273), (777, 1026, 1026), (513, 1001, 1001), (100_000, 259, 30)):
        hi = min(hi, padlen) - extra
        buf, offs = gen(1234 + n, n, 0, hi, MIX)
        lens = np.diff(offs)
        lens[:: max(1, n // 7)] = hi          # some rows exactly fill padlen
        if n > 100 and hi >= 40:
            lens[5:40] = np.arange(hi - 34, hi + 1)   # a run of nearly full rows, every tail length
        offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        buf = np.resize(buf, int(offs[-1]))
        want = orc.batch_tokenize((buf, offs), padlen=padlen, batch_first=True)
        assert_same_bits(want, abi_tokenize(tok, buf, offs, padlen, True, "B").cpu().numpy())
        big = torch.zeros(buf.size + 64, dtype=torch.uint8, device="cuda")
        big[5:5 + buf.size] = to_dev(buf)
        assert_same_bits(want, abi_tokenize(tok, buf, offs, padlen, True, "B", d_bytes=big[5:]).cpu().numpy())


def test_staged_pipeline_multi_chunk_and_reuse():
    # > 4 MiB of residues so the host-staged path runs several pipeline stages; odd batch size so the
    # last range is not a whole tile; pageable and pinned sources; back-to-back reuse of one stager.
    buf, offs = gen(11, 20011, 100, 1000, b"ACDEFGHIKLMNPQRSTVWYX")
    n = len(offs) - 1
    assert buf.size > 10 * (1 << 20)
    orc = OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    tok = capi.tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    stager = capi.Stager(0)
    pin_b = torch.from_numpy(buf.copy()).pin_memory()
    pin_o = torch.from_numpy(offs.copy()).pin_memory()
    for bf, dc in ((True, "B"), (False, "B"), (False, "i"), (True, "h")):
        want = orc.batch_tokenize((buf, offs), padlen=1002, destchar=dc, batch_first=bf)
        for hb, ho in ((buf, offs), (pin_b, pin_o)):
            out = torch.empty(want.shape, dtype=TORCH_DT[capi.kind_of(dc)], device="cuda")
            stager.tokenize_host(stream(), hb, ho, n, 1002, tok, bf, capi.kind_of(dc), out)
            torch.cuda.synchronize()
            assert_same_bits(want, out.cpu().numpy())
    mask = gen_mask(3, buf.size)
    want = orc.batch_onehot_encode((buf[:offs[3001]], offs[:3002]), padlen=1002, destchar="b", mask=split_mask(mask, offs[:3002]))
    out = torch.empty(want.shape, dtype=torch.int8, device="cuda")
    stager.onehot_host(stream(), buf, offs, mask, 3001, 1002, tok, capi.I8, out)
    torch.cuda.synchronize()
    assert_same_bits(want, out.cpu().numpy())
    stager.close()


def test_non_default_stream_and_python_list_inputs():
    t = bioseq_b200.pbeos_tokenizers["protein"]
    orc = OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    buf, offs = gen(21, 5000, 0, 400, MIX)
    seqs = as_list(buf, offs)
    mixed = [s if i % 3 else bytearray(s) for i, s in enumerate(seqs)]
    want = orc.batch_tokenize((buf, offs), padlen=402, batch_first=True)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got = t.batch_tokenize(mixed, padlen=402, batch_first=True, nthreads=4)
        got2 = t.batch_tokenize(tuple(seqs), padlen=402, batch_first=False)
    s.synchronize()
    assert_same_bits(want, got.cpu().numpy())
    assert_same_bits(want.T, got2.cpu().numpy())
    # str items are taken as UTF-8 (src/tokenize.h:397)
    strs = ["ACGT", "ACéGT", "", "中N"]
    want = OracleTokenizer("DNA", bos=True, padchar=True).batch_tokenize(strs, padlen=9, batch_first=True)
    got = bioseq_b200.Tokenizer("DNA", bos=True, padchar=True).batch_tokenize(strs, padlen=9, batch_first=True)
    assert_same_bits(want, got.cpu().numpy())


def test_dtypes_returned_by_python_api():
    t = bioseq_b200.Tokenizer("DNA")
    want = {"B": torch.uint8, "b": torch.int8, "h": torch.int16, "H": torch.int16, "i": torch.int32, "I": torch.int32,
            "l": torch.int64, "q": torch.int64, "L": torch.int64, "Q": torch.int64, "f": torch.float32, "d": torch.float64}
    for dc, dt in want.items():
        assert t.batch_tokenize(["ACGT"], padlen=5, destchar=dc).dtype == dt
        assert t.batch_onehot_encode(["ACGT"], padlen=5, destchar=dc).dtype == dt
    assert t.batch_tokenize(["ACGT"], padlen=5).shape == (5, 1)                      # batch_first defaults to False
    assert t.batch_tokenize([], padlen=5, batch_first=True).shape == (0, 5)
    assert t.batch_tokenize([], padlen=5).shape == (5, 0)
    assert t.batch_onehot_encode([], padlen=5).shape == (5, 0, 4)


# ------------------------------------------------------------------------------------- errors
def test_errors_raise_instead_of_aborting():
    t = bioseq_b200.Tokenizer("DNA", bos=True, eos=True)
    with pytest.raises(RuntimeError, match=r"seq len \+ bos \+ eos > padlen: 6, vs padlen 5"):
        t.batch_tokenize(["AC", "ACGT"], padlen=5, batch_first=True)
    with pytest.raises(ValueError, match=r"seq len \+ bos \+ eos > padlen: 6, vs padlen 5"):
        t.batch_onehot_encode(["AC", "ACGT"], padlen=5)
    offs = np.array([0, 2, 6], dtype=np.int64)
    buf = np.frombuffer(b"ACACGT", dtype=np.uint8)
    with pytest.raises(RuntimeError, match=r"seq len \+ bos \+ eos > padlen: 6, vs padlen 5"):
        t.batch_tokenize_packed(to_dev(buf), to_dev(offs), padlen=5)
    with pytest.raises(RuntimeError, match=r"seq len \+ bos \+ eos > padlen: 6, vs padlen 5"):
        t.batch_tokenize_packed(buf, offs, padlen=5)
    tok = capi.tokenizer("DNA")
    out = torch.empty(64, dtype=torch.int8, device="cuda")
    with pytest.raises(ValueError, match="16-byte aligned"):
        capi.tokenize(0, stream(), to_dev(buf), to_dev(offs), 2, 8, tok, True, 0, out.data_ptr() + 1)
    with pytest.raises(ValueError, match="batch tokenize requires padlen is provded."):
        capi.tokenize(0, stream(), to_dev(buf), to_dev(offs), 2, 0, tok, True, 0, out)


def test_decode_errors_and_itemsizes():
    t = bioseq_b200.pbeos_tokenizers["PROTEIN"]
    orc = OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    base = np.array([[20, 0, 5, 19, 21, 22, 22], [20, 21, 22, 22, 22, 22, 22]])
    for dt in (np.uint8, np.int8, np.int16, np.int32, np.int64, np.uint16, np.uint32, np.uint64):
        x = base.astype(dt)
        assert t.decode_tokens(x) == orc.decode_tokens(x)
        assert t.decode_tokens(x[1]) == orc.decode_tokens(x[1])
        if dt in (np.uint8, np.int8, np.int16, np.int32, np.int64):
            assert t.decode_tokens(torch.from_numpy(x).cuda()) == orc.decode_tokens(x)
            assert t.decode_tokens(torch.from_numpy(x)) == orc.decode_tokens(x)
    for bad, dt in ((23, np.uint8), (-1, np.int8), (-1, np.int16), (300, np.int32), (1.0, np.float32), (70000, np.int64)):
        x = np.array([[0, 1], [0, bad], [bad, 0]], dtype=dt)
        with pytest.raises(RuntimeError) as e1:
            orc.decode_tokens(x)
        with pytest.raises(RuntimeError) as e2:
            t.decode_tokens(x)
        assert str(e1.value) == str(e2.value)
    for dt in (np.int32, np.int64):                     # -1 -> "\0" entry (src/tokenize.h:83-88)
        assert t.decode_tokens(np.array([0, -1, 3], dtype=dt)) == "A\x00E"
    with pytest.raises(ValueError, match="Currently supported: 1 or 2 dimensions"):
        t.decode_tokens(np.zeros((2, 2, 2), dtype=np.uint8))
    assert t.decode_tokens(np.zeros((0, 4), dtype=np.uint8)) == []
    assert t.decode_tokens(np.zeros((3, 0), dtype=np.uint8)) == ["", "", ""]
    assert t.decode_tokens(np.zeros(0, dtype=np.uint8)) == ""


def test_single_sequence_onehot_encode():
    R = load_ref()
    ref = Reference("test_gpu_parity::test_single_sequence_onehot_encode", R)
    for key, flags in (("DNA", {}), ("DNA", dict(bos=True, eos=True, padchar=True)), ("PROTEIN", dict(eos=True, padchar=True))):
        ref_t, t = R and R.Tokenizer(key, **flags), bioseq_b200.Tokenizer(key, **flags)
        for seq in ("ACGT", "", "ACGTACGTAC", b"GATTACA", bytearray(b"CCGG")):
            # len + 1: with BOS + EOS + padchar the EOS row lies at `padlen` itself (ADVICE r1: it must not be zeroed)
            for padlen in (0, 3, 12, len(seq) + 1, len(seq)):
                if padlen and len(seq) > padlen:
                    with pytest.raises(RuntimeError, match="padlen is too short"):
                        t.onehot_encode(seq, padlen)
                    continue
                for dc in ("f", "B", "H", "i", "d"):
                    ref.check(t.onehot_encode(seq, padlen, dc).cpu().numpy(), lambda: ref_t.onehot_encode(seq, padlen, dc))
                ref.check(t.onehot_encode(seq, padlen).cpu().numpy(), lambda: ref_t.onehot_encode(seq, padlen))
    ref.done()


# ------------------------------------------------------------------------------------- BASELINE.json sizes
def test_config1_dna_full_size():
    buf, offs = gen(101, 4096, 1000, 1000, b"ACGT")
    tok, orc = capi.tokenizer("DNA"), OracleTokenizer("DNA")
    want = orc.batch_tokenize((buf, offs), padlen=1024, batch_first=True)
    got = abi_tokenize(tok, buf, offs, 1024, True, "B")
    assert_same_bits(want, got.cpu().numpy())
    assert_same_bits(want.T, abi_tokenize(tok, buf, offs, 1024, False, "B").cpu().numpy())


@pytest.mark.parametrize("hi,padlen", [(1022, 1024), (1024, 1026)])
def test_config2_protein_ragged_full_size(hi, padlen):
    buf, offs = gen(102, 65536, 50, hi, b"ACDEFGHIKLMNPQRSTVWY")
    tok = capi.tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    orc = OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    want = orc.batch_tokenize((buf, offs), padlen=padlen, batch_first=True)
    got = abi_tokenize(tok, buf, offs, padlen, True, "B")
    assert_same_bits(want, got.cpu().numpy())
    # properties that do not need the oracle: row structure and a checksum of checksums
    g = got.long()
    lens = torch.from_numpy(np.diff(offs)).cuda()
    assert bool((g[:, 0] == 20).all())
    assert bool((g.gather(1, (lens + 1).unsqueeze(1)).squeeze(1) == 21).all())
    assert bool(((g == 22).sum(1) == padlen - lens - 2).all())
    assert int(g.sum()) == int(want.astype(np.int64).sum())
    got_sf = abi_tokenize(tok, buf, offs, padlen, False, "B")
    assert torch.equal(got_sf, got.t())
    dec = abi_decode(tok, got[:2048])
    assert dec == orc.decode_tokens(want[:2048])


def test_config3_onehot_f32_full_size():
    buf, offs = gen(103, 16384, 4096, 4096, b"ACGT")
    tok, orc = capi.tokenizer("DNA"), OracleTokenizer("DNA")
    got = abi_onehot(tok, buf, offs, None, 4096, "f")          # (4096, 16384, 4) float32, 1 GiB
    assert got.shape == (4096, 16384, 4)
    toks = abi_tokenize(tok, buf, offs, 4096, False, "B")
    assert torch.equal(got.argmax(2).to(torch.uint8), toks)     # one-hot <-> tokens
    assert bool((got.sum(2) == 1).all())
    assert float(got.sum()) == 4096 * 16384
    want = orc.batch_onehot_encode((buf[:offs[2048]], offs[:2049]), padlen=4096, destchar="f")
    assert_same_bits(want, got[:, :2048].contiguous().cpu().numpy())
    del got
    torch.cuda.empty_cache()


def test_config4_reduced_alphabets_roundtrip():
    buf, offs = gen(104, 200_000, 50, 1024, b"ACDEFGHIKLMNPQRSTVWY")
    rng = np.random.default_rng(4)
    noisy = buf.copy()                                            # 5 % lower-case / invalid residues
    idx = rng.random(buf.size) < 0.05
    noisy[idx] = np.frombuffer(b"acdefghiklmnpqrstvwyXBZOU*-", dtype=np.uint8)[rng.integers(0, 27, int(idx.sum()))]
    d_bytes, d_noisy = to_dev(buf), to_dev(noisy)
    n = len(offs) - 1
    for key in ("SEB6", "SEB8", "SEB10", "SEB14", "SEV10", "MURPHY", "LIA10", "LIB10", "DAYHOFF"):
        for flags, padlen in ((dict(padchar=True), 1024), (dict(bos=True, eos=True, padchar=True), 1026)):
            tok, orc = capi.tokenizer(key, **flags), OracleTokenizer(key, **flags)
            got = abi_tokenize(tok, buf, offs, padlen, True, "B", d_bytes=d_bytes)
            # decode o tokenize maps every residue to its group representative (not the identity)
            rep = np.zeros(256, dtype=np.uint8)
            first = {}
            for b in range(256):
                first.setdefault(int(orc.lut[b]), b)
            for b in range(256):
                rep[b] = first[int(orc.lut[b])] if orc.lut[b] >= 0 else first[0]
            sub = slice(0, 20000)
            dec = abi_decode(tok, got[sub])
            want_tok = orc.batch_tokenize((buf[:offs[20000]], offs[:20001]), padlen=padlen, batch_first=True)
            assert_same_bits(want_tok, got[sub].cpu().numpy())
            assert dec == orc.decode_tokens(want_tok)
            bos = "<BOS>" if flags.get("bos") else ""
            eos = "<EOS>" if flags.get("eos") else ""
            for i in (0, 1, 19999):
                body = rep[buf[offs[i]:offs[i + 1]]].tobytes().decode()
                npad = padlen - len(body) - (len(bos) > 0) - (len(eos) > 0)
                assert dec[i] == bos + body + eos + "<PAD>" * npad
            if key in ("SEB10", "DAYHOFF"):
                gn = abi_tokenize(tok, noisy, offs, padlen, True, "B", d_bytes=d_noisy)
                wn = orc.batch_tokenize((noisy[:offs[20000]], offs[:20001]), padlen=padlen, batch_first=True)
                assert_same_bits(wn, gn[sub].cpu().numpy())
                # whole-batch checksum against the oracle
                wfull = orc.batch_tokenize((noisy, offs), padlen=padlen, batch_first=True)
                assert int(gn.long().sum()) == int(wfull.astype(np.int64).sum())
                assert_same_bits(wfull, gn.cpu().numpy())
    del d_bytes, d_noisy
    torch.cuda.empty_cache()


def test_python_decode_many_rows():
    t = bioseq_b200.pbeos_tokenizers["SEB10"]
    orc = OracleTokenizer("SEB10", bos=True, eos=True, padchar=True)
    buf, offs = gen(44, 50_000, 1, 300, b"ACDEFGHIKLMNPQRSTVWY")
    toks = t.batch_tokenize_packed(buf, offs, padlen=304, batch_first=True)
    want = orc.decode_tokens(orc.batch_tokenize((buf, offs), padlen=304, batch_first=True))
    assert t.decode_tokens(toks) == want
    assert t.decode_tokens(toks.to(torch.int32)) == want


def test_sharded_equals_single_device():
    # SURVEY 8(e): shards are independent; concatenating them reproduces the unsharded output.
    from bioseq_b200.shard import tokenize_sharded
    t = bioseq_b200.pbeos_tokenizers["PROTEIN"]
    buf, offs = gen(88, 30_001, 0, 600, b"ACDEFGHIKLMNPQRSTVWYX")
    full_bf = t.batch_tokenize_packed(buf, offs, padlen=608, batch_first=True)
    full_sf = t.batch_tokenize_packed(buf, offs, padlen=608, batch_first=False)
    for world in (2, 3, 8):
        parts = [tokenize_sharded(t, buf, offs, 608, world, r, batch_first=True) for r in range(world)]
        assert [p[1][0] for p in parts][0] == 0 and parts[-1][1][1] == 30_001
        assert torch.equal(torch.cat([p[0] for p in parts], dim=0), full_bf)
        parts = [tokenize_sharded(t, buf, offs, 608, world, r, batch_first=False)[0] for r in range(world)]
        assert torch.equal(torch.cat(parts, dim=1), full_sf)


@pytest.mark.parametrize("nthreads", [1, 3, 16])
def test_list_api_pipelined_gather(nthreads):
    # the reference's calling convention (a Python list of bytes) on a batch of several staged ranges:
    # gather -> copy -> kernel pipelined range by range (bsq_tokenize_items / bsq_onehot_items), every
    # thread count, both layouts, back-to-back calls reusing the pinned pack, one-hot without a mask
    buf, offs = gen(300 + nthreads, 30_011, 0, 1000, MIX)
    assert buf.size > 12 * (1 << 20)
    seqs = as_list(buf, offs)
    t = bioseq_b200.pbeos_tokenizers["PROTEIN"]
    dev_bf = t.batch_tokenize_packed(to_dev(buf), to_dev(offs), padlen=1002, batch_first=True)
    for _ in range(2):
        got = t.batch_tokenize(seqs, padlen=1002, batch_first=True, nthreads=nthreads)
        got_sf = t.batch_tokenize(seqs, padlen=1002, destchar="h", nthreads=nthreads)
        assert torch.equal(got, dev_bf)
        assert torch.equal(got_sf, dev_bf.T.to(torch.int16))
    small = seqs[:2001]
    orc = OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    want = orc.batch_onehot_encode((buf[:offs[2001]], offs[:2002]), padlen=1002, destchar="B")
    assert_same_bits(want, t.batch_onehot_encode(small, padlen=1002, nthreads=nthreads).cpu().numpy())
    # the length check fires before anything is copied, with the reference's text
    with pytest.raises(RuntimeError, match=r"seq len \+ bos \+ eos > padlen: 1002, vs padlen 1001"):
        t.batch_tokenize(seqs + [b"A" * 1000], padlen=1001, nthreads=nthreads)
    assert torch.equal(t.batch_tokenize(seqs, padlen=1002, batch_first=True, nthreads=nthreads), dev_bf)


def test_python_decode_streams_many_stages():
    # decoded characters leave the device through the pinned ring in 8 MiB stages (bsq_fetch_rows): enough rows
    # for > 3 stages (ring reuse), ragged rows with 5-character specials, rows straddling stage boundaries
    t = bioseq_b200.pbeos_tokenizers["DAYHOFF"]
    orc = OracleTokenizer("DAYHOFF", bos=True, eos=True, padchar=True)
    buf, offs = gen(45, 40_000, 0, 500, b"ACDEFGHIKLMNPQRSTVWY")
    toks = t.batch_tokenize_packed(buf, offs, padlen=512, batch_first=True)
    got = t.decode_tokens(toks)
    assert sum(map(len, got)) > 4 * (8 << 20)
    ref_rows = np.r_[0:300, 20_000:20_300, 39_700:40_000]
    sub = orc.batch_tokenize((buf, offs), padlen=512, batch_first=True)[ref_rows]
    assert [got[i] for i in ref_rows] == orc.decode_tokens(sub)
    assert got == abi_decode(capi.tokenizer("DAYHOFF", bos=True, eos=True, padchar=True), toks)
    # 1-D input, one row, and empty rows
    assert t.decode_tokens(toks[7]) == got[7]
    assert t.decode_tokens(toks[:1]) == got[:1]
    assert t.decode_tokens(toks[:0]) == []


@pytest.mark.parametrize("cols,row_pad,shift", [(1024, 0, 0), (1040, 0, 0), (1000, 0, 0), (1024, 16, 0), (1024, 4, 0), (640, 1, 0),
                                                (1024, 0, 4), (1024, 0, 3), (130, 0, 0), (512, 0, 0)])
def test_decode_fast_steps_every_alignment(cols, row_pad, shift):
    # K4 lays plain-text steps and runs of one special into its stage as whole words (512-token steps for
    # 16-byte aligned rows, 128-token steps for 4-byte aligned ones) and falls back to the byte-wise step for
    # mixed ones: random mixtures of text runs, special runs and single specials, every row/carry alignment,
    # against a direct table decode
    flags = dict(bos=True, eos=True, padchar=True)
    tok = capi.tokenizer("PROTEIN", **flags)
    orc = OracleTokenizer("PROTEIN", **flags)
    rng = np.random.default_rng(cols * 31 + row_pad * 7 + shift)
    rows = 300
    a = np.empty((rows, cols), dtype=np.uint8)
    for r in range(rows):
        c = 0
        while c < cols:
            kind = rng.integers(0, 10)
            n = int(rng.integers(1, 700)) if kind < 8 else int(rng.integers(1, 4))
            n = min(n, cols - c)
            if kind < 5:
                a[r, c:c + n] = rng.integers(0, 20, size=n)
            elif kind < 8:
                a[r, c:c + n] = rng.integers(20, 23)
            else:
                a[r, c:c + n] = rng.integers(0, 23, size=n)
            c += n
    a[0] = 22
    a[1] = 3
    a[2, :] = np.arange(cols) % 20
    a[3, :] = (np.arange(cols) * 7) % 20            # one special in the very first position, then plain text
    a[3, 0] = 20
    a[4, :] = (np.arange(cols) * 3) % 20            # ... then text, EOS and a PAD run
    a[4, 0] = 20
    a[4, cols // 2] = 21
    a[4, cols // 2 + 1:] = 22
    a[5, :] = 22                                    # specials only, two kinds
    a[5, ::2] = 21
    for r in range(6, 130):                         # rows as batch_tokenize writes them: <BOS> text <EOS> <PAD>...
        L = int(rng.integers(0, cols - 1)) if r > 12 else (0, 1, 13, 14, 15, cols - 2, cols - 3)[r - 6]
        a[r, 0] = 20
        a[r, 1:1 + L] = rng.integers(0, 20, size=L)
        a[r, 1 + L] = 21
        a[r, 2 + L:] = 22
    for r in range(130, 180):                       # ... and without BOS / EOS: text, then the PAD run
        L = int(rng.integers(0, cols + 1))
        a[r, :L] = rng.integers(0, 20, size=L)
        a[r, L:] = 22
    want = orc.decode_tokens(a)
    assert want[0] == "<PAD>" * cols and want[1] == "E" * cols
    flat = torch.zeros(rows * (cols + row_pad) + 64, dtype=torch.uint8, device="cuda")
    view = flat[shift:shift + rows * (cols + row_pad)].view(rows, cols + row_pad)[:, :cols]
    view.copy_(torch.from_numpy(a))
    assert abi_decode(tok, view) == want
    # a token without an entry: reported with the reference's message, at its first position in row-major order
    for (r, c) in ((rows - 1, cols - 1), (5, 17), (5, 16)):
        old = int(view[r, c])
        view[r, c] = 23
        with pytest.raises(RuntimeError, match="Unexpected/invalid token 23"):
            abi_decode(tok, view)
        view[r, c] = old
    assert abi_decode(tok, view) == want


def test_concurrent_python_threads_share_pool_and_stager():
    # four Python threads hammer the list API (worker pool + pinned pack + stager, per-device mutex) and
    # decode_tokens (pinned device->host ring) at once, each on its own stream: no deadlock, no cross-talk
    import threading
    t = bioseq_b200.pbeos_tokenizers["PROTEIN"]
    work = []
    for k in range(4):
        buf, offs = gen(500 + k, 9000 + 1000 * k, 0, 800, MIX)
        seqs = as_list(buf, offs)
        want = t.batch_tokenize_packed(to_dev(buf), to_dev(offs), padlen=802, batch_first=True)
        work.append((seqs, want, t.decode_tokens(want[:2000])))
    errors = []

    def run(k):
        try:
            seqs, want, want_txt = work[k]
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                for it in range(6):
                    got = t.batch_tokenize(seqs, padlen=802, batch_first=True, nthreads=2 + 3 * (it % 3))
                    s.synchronize()
                    assert torch.equal(got, want), f"thread {k} iteration {it}: tokens differ"
                    assert t.decode_tokens(got[:2000]) == want_txt, f"thread {k} iteration {it}: text differs"
        except Exception as e:  # noqa: BLE001
            errors.append(repr(e))

    threads = [threading.Thread(target=run, args=(k,)) for k in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join(timeout=120)
    assert not any(th.is_alive() for th in threads), "deadlock in the host pipeline"
    assert not errors, errors


# ------------------------------------------------------------------------------------- the reference on the GPU machine
def test_oracle_pinned_to_live_reference_on_this_box():
    """The oracle <-> reference pin of tests/test_oracle.py, run in a GPU-only test pass (`-m gpu`) as well: it is the
    reference (recorded in tests/golden/reference.json; live when oracle/_ref is built) that makes the oracle an oracle."""
    import test_oracle as TO
    for seed in range(6):
        TO.test_live_reference_tokenize_onehot_decode(seed)
    TO.test_live_reference_str_inputs_utf8()
    TO.test_live_reference_decode_itemsizes()


@pytest.mark.parametrize("seed", range(4))
def test_gpu_vs_live_reference_dropin_calls(seed):
    """The drop-in Python class against the reference's own class, same calls, same arguments: list of str / bytes /
    bytearray items in, arrays (tokens in both layouts and every dtype, one-hot with and without mask) and decoded
    strings out."""
    R = load_ref()
    ref = Reference(f"test_gpu_parity::test_gpu_vs_live_reference_dropin_calls[{seed}]", R)
    rng = np.random.default_rng(4242 + seed)
    keys = [k for k in alphabet_keys() if k != "BYTES"]   # BYTES ids wrap differently by design (DESIGN.md section 5)
    for trial in range(10):
        key = keys[int(rng.integers(len(keys)))]
        flags = dict(bos=bool(rng.integers(2)), eos=bool(rng.integers(2)), padchar=bool(rng.integers(2)))
        n = int(rng.integers(0, 300))
        hi = int(rng.integers(0, 700))
        buf, offs = gen(int(rng.integers(1 << 30)), n, 0, hi, MIX[:-3])   # (bytes >= 0x80 are undefined in the reference)
        seqs = as_list(buf, offs)
        kind = int(rng.integers(3))
        if kind == 1:
            seqs = [bytearray(s) for s in seqs]
        elif kind == 2:
            seqs = [s.decode("latin-1") if all(c < 0x80 for c in s) else s for s in seqs]
        padlen = hi + 2 + int(rng.integers(0, 40))
        dc = "bhilqfd"[int(rng.integers(7))]
        bf = bool(rng.integers(2))
        ref_t, t = R and R.Tokenizer(key, **flags), bioseq_b200.Tokenizer(key, **flags)
        b = t.batch_tokenize(seqs, padlen=padlen, destchar=dc, batch_first=bf, nthreads=int(rng.integers(1, 9)))
        a = ref.check(b.cpu().numpy(), lambda: ref_t.batch_tokenize(seqs, padlen=padlen, destchar=dc, batch_first=bf, nthreads=2))
        if dc not in "fd":
            ref.check(t.decode_tokens(b), lambda: ref_t.decode_tokens(a))
        mask = None
        if rng.integers(2) and n:
            m = gen_mask(int(rng.integers(1 << 30)), buf.size, 0.7)
            mask = [m[offs[i]:offs[i + 1]] for i in range(n)]
        b = t.batch_onehot_encode(seqs, padlen=padlen, destchar=dc, mask=mask)
        ref.check(b.cpu().numpy(), lambda: ref_t.batch_onehot_encode(seqs, padlen=padlen, destchar=dc, mask=mask))
    ref.done()


def test_streamed_items_ranges_and_growth():
    """bsq_tokenize_stream_items: many ranges, pinned-pack growth in the middle of a call, batches that shrink and grow
    from call to call, every host thread count; always equal to the packed device call."""
    tok = bioseq_b200.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    for n, lo, hi, padlen in ((70000, 0, 120, 128), (9000, 900, 1000, 1002), (3, 0, 5, 8), (200000, 0, 30, 32), (20000, 500, 2000, 2048)):
        buf, offs = gen(n + hi, n, lo, hi, b"ACDEFGHIKLMNPQRSTVWYXacd")
        seqs = as_list(buf, offs)
        want = tok.batch_tokenize_packed(torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda(), padlen=padlen, batch_first=True)
        for nt in (1, 3, 8, 16):
            assert torch.equal(tok.batch_tokenize(seqs, padlen=padlen, batch_first=True, nthreads=nt), want)
        assert torch.equal(tok.batch_tokenize(seqs, padlen=padlen, nthreads=5), want.t())


def test_sharded_single_process_entry():
    """Tokenizer.batch_tokenize_sharded: one packed host batch -> one shard per device (here: the same device twice is
    refused; one device = the whole batch; with 2+ GPUs the shards concatenate to the single-device result)."""
    tok = bioseq_b200.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    buf, offs = gen(9, 5000, 0, 300, b"ACDEFGHIKLMNPQRSTVWY")
    want = tok.batch_tokenize_packed(torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda(), padlen=304, batch_first=True)
    outs, bounds = tok.batch_tokenize_sharded(buf, offs, padlen=304, batch_first=True, devices=[0])
    assert list(bounds) == [0, 5000] and torch.equal(outs[0], want)
    ndev = torch.cuda.device_count()
    if ndev >= 2:
        outs, bounds = tok.batch_tokenize_sharded(buf, offs, padlen=304, batch_first=True)
        assert len(outs) == ndev and bounds[0] == 0 and bounds[-1] == 5000
        assert torch.equal(torch.cat([o.to("cuda:0") for o in outs], dim=0), want)
        sizes = [int(offs[bounds[g + 1]] - offs[bounds[g]]) for g in range(ndev)]
        assert max(sizes) - min(sizes) <= 2 * 300
        outs, _ = tok.batch_tokenize_sharded(buf, offs, padlen=304, batch_first=False)
        assert torch.equal(torch.cat([o.to("cuda:0") for o in outs], dim=1), want.t())
    with pytest.raises(ValueError):
        tok.batch_tokenize_sharded(buf, offs, padlen=304, devices=[0, 0])


@pytest.mark.parametrize("padlen,batch_first,destchar", [(1024, True, "B"), (1026, True, "B"), (300, True, "B"), (1024, False, "B"), (1024, True, "i")])
def test_tokenize_many_equals_single_launches(padlen, batch_first, destchar):
    """bsq_tokenize_many: k small batches, one launch (groups of 32); other layouts / dtypes fall back to one launch each."""
    tok, orc = capi.tokenizer("PROTEIN", bos=True, eos=True, padchar=True), OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    kind = capi.kind_of(destchar)
    rng = np.random.default_rng(padlen)
    sizes = [int(x) for x in rng.integers(0, 400, size=40)] + [0, 1, 4096]
    batches, wants = [], []
    for k, n in enumerate(sizes):
        buf, offs = gen(1000 + k, n, 0, padlen - 2, MIX)
        d_b = to_dev(np.concatenate([buf, np.zeros(32, np.uint8)]))
        d_o = to_dev(offs)
        out = torch.full((n, padlen) if batch_first else (padlen, n), 77, dtype=TORCH_DT[kind], device="cuda")
        batches.append((d_b, d_o, n, out))
        wants.append(orc.batch_tokenize((buf, offs), padlen=padlen, destchar=destchar, batch_first=batch_first))
    capi.tokenize_many(0, stream(), batches, padlen, tok, batch_first, kind)
    torch.cuda.synchronize()
    for (d_b, d_o, n, out), want in zip(batches, wants):
        assert_same_bits(want, out.cpu().numpy())


def test_packed_offsets_are_validated_before_any_kernel_indexes_bytes():
    # device-resident and host packed inputs: negative first offset, decreasing offsets, offsets past the end of bytes
    tok = bioseq_b200.Tokenizer("DNA")
    b = np.frombuffer(b"ACGTACGTAC", dtype=np.uint8).copy()
    good = np.array([0, 4, 10], dtype=np.int64)
    want = tok.batch_tokenize_packed(b, good, padlen=8, batch_first=True).cpu().numpy()
    for side in ("host", "cuda"):
        conv = (lambda x: x) if side == "host" else (lambda x: torch.from_numpy(x).cuda())
        assert np.array_equal(tok.batch_tokenize_packed(conv(b), conv(good), padlen=8, batch_first=True).cpu().numpy(), want)
        for bad in ([-2, 4, 10], [0, 6, 4], [0, 4, 11], [3, 2, 10]):
            with pytest.raises((ValueError, RuntimeError), match="offsets"):
                tok.batch_tokenize_packed(conv(b), conv(np.array(bad, dtype=np.int64)), padlen=16, batch_first=True)
            with pytest.raises((ValueError, RuntimeError), match="offsets"):
                tok.batch_onehot_encode_packed(conv(b), conv(np.array(bad, dtype=np.int64)), padlen=16)


def test_cuda_graph_of_small_batches_replays_bit_exact():
    # INTEGRATION.md "Small batches": a train of bsq_tokenize calls captured once and replayed (the launches are
    # capturable; under capture the span kernel uses its static tile order), against the same calls made directly
    tok = capi.tokenizer("DNA", bos=True, eos=True, padchar=True)
    st_default = torch.cuda.current_stream().cuda_stream
    batches = []
    for i in range(6):
        buf, offs = gen(900 + i, 512, 0, 998, b"ACGTN")
        d_b, d_o = torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda()
        direct = torch.empty((512, 1000), dtype=torch.uint8, device="cuda")
        capi.tokenize(0, st_default, d_b, d_o, 512, 1000, tok, True, 0, direct)
        batches.append((d_b, d_o, direct, torch.zeros_like(direct)))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        st = torch.cuda.current_stream().cuda_stream
        for d_b, d_o, _, out in batches:
            capi.tokenize(0, st, d_b, d_o, 512, 1000, tok, True, 0, out)
    for rep in range(3):
        for b in batches:
            b[3].zero_()
        g.replay()
        torch.cuda.synchronize()
        for _, _, direct, out in batches:
            assert torch.equal(direct, out)


def test_python_decode_text_guess_overflow_falls_back_to_exact_pass():
    # Tokenizer.decode_tokens sizes its text buffer by a guess (3 characters per token) and runs both passes in one
    # call; a batch that is nearly all <PAD> (5 characters per token) does not fit: nothing is written, and the
    # exactly sized second pass must give the same strings
    t = bioseq_b200.pbeos_tokenizers["PROTEIN"]
    o = OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    rows, cols = 300, 777
    a = np.full((rows, cols), 22, dtype=np.uint8)           # <PAD> everywhere ...
    a[:, 0] = 20                                            # ... behind <BOS> X <EOS>
    a[:, 1] = np.arange(rows) % 20
    a[:, 2] = 21
    want = o.decode_tokens(a)
    assert sum(map(len, want)) > 3 * rows * cols
    assert t.decode_tokens(torch.from_numpy(a).cuda()) == want
    assert t.decode_tokens(a) == want


@pytest.mark.parametrize("seed", range(6))
def test_random_mid_size_batches_span_kernel_and_decode(seed):
    # the regime of the headline kernel (padlen >= 257: tokenize_span_kernel, several tiles, rows that straddle tiles and
    # warps) and of the staged decode: random padlens (16-byte aligned or not), row counts, length distributions with
    # empty and full rows, every flag combination -- tokens against the oracle, text against the oracle's decode
    rng = np.random.default_rng(9100 + seed)
    for trial in range(4):
        key = ("PROTEIN", "DNA", "DAYHOFF", "BYTES")[int(rng.integers(4))]
        flags = dict(bos=bool(rng.integers(2)), eos=bool(rng.integers(2)), padchar=bool(rng.integers(2)))
        padlen = int(rng.choice([257, 272, 511, 512, 513, 652, 656, 1000, 1024, 1026, 1500, 2048, 2999]))
        n = int(rng.choice([1, 7, 64, 500, 1777, 3000]))
        room = padlen - flags["bos"] - flags["eos"]
        shape = int(rng.integers(4))
        lo, hi = ((0, room), (room, room), (0, min(room, 40)), (max(0, room - 20), room))[shape]
        buf, offs = gen(int(rng.integers(1 << 30)), n, lo, hi, MIX)
        tok, orc = capi.tokenizer(key, **flags), OracleTokenizer(key, **flags)
        want = orc.batch_tokenize((buf, offs), padlen=padlen, destchar="B", batch_first=True)
        got = abi_tokenize(tok, buf, offs, padlen, True, "B")
        assert_same_bits(want, got.cpu().numpy())
        if key != "BYTES":
            assert abi_decode(tok, got) == orc.decode_tokens(want)


def test_span_kernel_on_concurrent_streams():
    # the span kernel's dynamic tile scheduler keeps its counters per stream (two slots, alternating): launches that
    # run concurrently on several streams, back to back on each, must not disturb one another
    tok = capi.tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    orc = OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    streams = [torch.cuda.Stream() for _ in range(4)]
    work = []
    for k, (n, padlen) in enumerate(((3000, 1024), (2500, 1026), (4000, 652), (1500, 2048))):
        buf, offs = gen(7700 + k, n, 0, padlen - 2, MIX)
        want = orc.batch_tokenize((buf, offs), padlen=padlen, destchar="B", batch_first=True)
        work.append((torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda(), n, padlen, want,
                     [torch.zeros((n, padlen), dtype=torch.uint8, device="cuda") for _ in range(6)]))
    torch.cuda.synchronize()
    for rep in range(6):
        for s, (d_b, d_o, n, padlen, _, outs) in zip(streams, work):
            capi.tokenize(0, s.cuda_stream, d_b, d_o, n, padlen, tok, True, 0, outs[rep])
    torch.cuda.synchronize()
    for d_b, d_o, n, padlen, want, outs in work:
        for o in outs:
            assert_same_bits(want, o.cpu().numpy())
