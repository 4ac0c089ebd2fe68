"""K-mer tokens (batch_tokenize_kmer / bsq_tokenize_kmer / bsq_tokenize_kmer_varlen, kernel K11), bit for bit against
the rule of include/bsq.h (tests/kmer_reference.py).

K11's padded kernel fills the flat (nseq, padlen) output 16 elements per thread, one row segment at a time where a
chunk crosses a row end; the padding-free form scans T(len_i) into cu_seqlens (K9's scan and carry) and writes each
row with one warp, element stores where two rows share a 16-element vector.  The cases cover every output kind that
holds the vocabulary with every bos / eos / padchar combination, the alphabets up to their largest k with strides 1, 2
and k and both tails, empty batches and rows, rows shorter than k, a sequence of 100 000 residues, every source
alignment, an unaligned padlen, batch sizes around the scan's block of 1024 rows and past 1024^2 rows, every batch
form, crops, the errors, back-to-back launches and a replayed CUDA graph."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import bioseq_b200  # noqa: E402
from bioseq_b200 import capi, cbioseq, consumers, batch_tokenize_kmer, crop_packed, VarlenBatch  # noqa: E402
from oracle.oracle import flatfile_image  # noqa: E402
from helpers import assert_same_bits  # noqa: E402
import kmer_reference as ref  # noqa: E402

FLAGS = [(b, e, p) for b in (False, True) for e in (False, True) for p in (False, True)]
NP = {"B": np.uint8, "b": np.int8, "h": np.int16, "i": np.int32, "l": np.int64, "f": np.float32, "d": np.float64}
VALID = {"DNA": b"ACGTacgt", "DNA5": b"ACGTNacgtn", "SEB6": b"ACDEFGHIKLMNPQRSTVWY", "PROTEIN": b"ACDEFGHIKLMNPQRSTVWYacdy",
         "PURPYR": b"ACGTRYacgt"}
NOISE = b"NnUuXx-*.\x00\x7f\x80\xc3\xff"


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests selected but no CUDA device is visible")


def cuda(buf, offs):
    return torch.from_numpy(np.ascontiguousarray(buf)).cuda(), torch.from_numpy(np.ascontiguousarray(offs)).cuda()


def batch_of(lens, seed, valid=b"ACGTacgt", lead=0, noise=0.05):
    lens = np.asarray(lens, np.int64)
    offs = np.zeros(lens.size + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    rng = np.random.default_rng(seed)
    v, x = np.frombuffer(valid, np.uint8), np.frombuffer(NOISE, np.uint8)
    size = int(offs[-1]) + lead
    buf = np.where(rng.random(size) < noise, x[rng.integers(0, x.size, size)], v[rng.integers(0, v.size, size)]).astype(np.uint8)
    return buf, offs + lead


def tokenizer(key, bos, eos, pad):
    return cbioseq.Tokenizer(key, bos=bos, eos=eos, padchar=pad)


def check_padded(got, buf, offs, key, k, s, tail, flags, padlen, destchar="i"):
    want = ref.padded(buf, offs, key, k, s, tail == "single", *flags, padlen)
    torch.cuda.synchronize()
    assert_same_bits(want.astype(NP[destchar]), got.cpu().numpy())


def check_varlen(vb, buf, offs, key, k, s, tail, flags, destchar="i"):
    toks, cu, mx = ref.varlen(buf, offs, key, k, s, tail == "single", flags[0], flags[1])
    torch.cuda.synchronize()
    assert isinstance(vb, VarlenBatch)
    assert_same_bits(cu, vb.cu_seqlens.cpu().numpy())
    assert_same_bits(toks.astype(NP[destchar]), vb.tokens.cpu().numpy())
    assert vb.max_seqlen == mx


def run_both(batch, buf, offs, key, k, s, tail, flags, padlen=None, destchar="i"):
    t = tokenizer(key, *flags)
    T = ref.count(np.diff(offs), k, s, tail == "single", flags[0], flags[1])
    padlen = padlen or int(T.max(initial=0)) + 3
    check_padded(batch_tokenize_kmer(t, batch, k, padlen, destchar, stride=s, tail=tail), buf, offs, key, k, s, tail, flags, padlen,
                 destchar)
    check_varlen(batch_tokenize_kmer(t, batch, k, destchar=destchar, stride=s, tail=tail, varlen=True), buf, offs, key, k, s, tail,
                 flags, destchar)


# ------------------------------------------------------------------------------------------------------------------
def test_worked_answers():
    t = bioseq_b200.pbeos_tokenizers["DNA"]
    for seq, s, tail, want in [("ACGTNAG", 1, "drop", [69, 6, 27, 68, 68, 68, 70]), ("ACGTNAG", 3, "single", [69, 6, 68, 66, 70]),
                               ("ACGTNAG", 3, "drop", [69, 6, 68, 70]), ("AC", 2, "single", [69, 64, 65, 70]),
                               ("AC", 1, "drop", [69, 70]), ("", 3, "single", [69, 70])]:
        out = batch_tokenize_kmer(t, [seq], 3, 9, stride=s, tail=tail)
        assert out.dtype == torch.int32 and out[0].tolist() == want + [71] * (9 - len(want))
        vb = batch_tokenize_kmer(t, [seq], 3, stride=s, tail=tail, varlen=True)
        assert vb.tokens.tolist() == want and vb.cu_seqlens.tolist() == [0, len(want)] and vb.max_seqlen == len(want)


@pytest.mark.parametrize("flags", FLAGS)
@pytest.mark.parametrize("destchar", ["B", "b", "h", "i", "l", "f", "d"])
def test_every_kind_and_flags(destchar, flags):
    lens = np.random.default_rng(3).integers(0, 70, 700)
    lens[:5] = [0, 1, 2, 3, 4]
    buf, offs = batch_of(lens, 11)
    for s, tail in ((1, "drop"), (3, "single"), (2, "single")):
        run_both((buf, offs), buf, offs, "DNA", 3, s, tail, flags, destchar=destchar)


def test_kinds_too_narrow_raise():
    t = bioseq_b200.pbeos_tokenizers["DNA"]
    with pytest.raises(ValueError, match="do not fit"):
        batch_tokenize_kmer(t, ["ACGT"], 4, 16, "b")  # 256 + 4 + 1 + 3 ids
    with pytest.raises(ValueError, match="do not fit"):
        batch_tokenize_kmer(t, ["ACGT"], 8, 16, "h")
    with pytest.raises(ValueError, match="do not fit"):
        batch_tokenize_kmer(t, ["ACGT"], 12, 16, "f", varlen=True)


KS = [("DNA", 1), ("DNA", 6), ("DNA", 15), ("DNA5", 13), ("SEB6", 11), ("PROTEIN", 3), ("PROTEIN", 7), ("PURPYR", 30)]


@pytest.mark.parametrize("key,k", KS)
@pytest.mark.parametrize("tail", ["drop", "single"])
def test_alphabets_strides_and_tails(key, k, tail):
    rng = np.random.default_rng(k)
    lens = rng.integers(0, 6 * k + 40, 500)
    lens[:6] = [0, 1, k - 1, k, k + 1, 2 * k + 1]
    buf, offs = batch_of(lens, 17 * k, VALID[key])
    for s in sorted({1, 2, k} & set(range(1, k + 1))):
        run_both((buf, offs), buf, offs, key, k, s, tail, (True, True, True))


def test_empty_batches_short_rows_and_a_long_sequence():
    t = bioseq_b200.pbeos_tokenizers["DNA"]
    e = batch_tokenize_kmer(t, [], 3, 8)
    assert e.shape == (0, 8)
    vb = batch_tokenize_kmer(t, [], 3, varlen=True)
    assert vb.tokens.numel() == 0 and vb.cu_seqlens.tolist() == [0] and vb.max_seqlen == 0
    for flags in ((True, True, True), (False, False, False)):
        buf, offs = batch_of([0] * 37, 1)
        run_both((buf, offs), buf, offs, "DNA", 3, 1, "drop", flags)
        run_both(cuda(buf, offs), buf, offs, "DNA", 3, 3, "single", flags)
        buf, offs = batch_of([1, 2, 0, 5, 4, 3, 0, 1] * 40, 2)  # all shorter than k = 6
        for tail in ("drop", "single"):
            run_both((buf, offs), buf, offs, "DNA", 6, 6, tail, flags)
    buf, offs = batch_of([100_003, 5, 70_001], 3)
    for s, tail in ((1, "drop"), (6, "single"), (4, "single")):
        run_both(cuda(buf, offs), buf, offs, "DNA", 6, s, tail, (True, True, True))


@pytest.mark.parametrize("shift", range(16))
def test_every_source_alignment_and_unaligned_padlen(shift):
    lens = np.random.default_rng(shift).integers(0, 1000, 300)
    buf, offs = batch_of(lens, 40 + shift, lead=shift)
    for s, tail in ((1, "drop"), (6, "single")):
        run_both(cuda(buf, offs), buf, offs, "DNA", 6, s, tail, (True, True, shift % 2 == 0), padlen=1026, destchar="i")
        run_both((buf, offs), buf, offs, "DNA", 6, s, tail, (shift % 3 == 0, True, True), padlen=1026 + shift, destchar="h")


@pytest.mark.parametrize("n", [1023, 1024, 1025, 2049])
def test_batch_sizes_around_the_scan_block(n):
    lens = np.random.default_rng(n).integers(0, 300, n)
    buf, offs = batch_of(lens, n)
    for flags in ((False, False, False), (True, True, False)):
        t = tokenizer("DNA", *flags)
        check_varlen(batch_tokenize_kmer(t, cuda(buf, offs), 5, stride=2, tail="single", varlen=True), buf, offs, "DNA", 5, 2,
                     "single", flags)


def test_more_than_a_million_short_rows():
    # 1 100 000 rows of 0..3 residues over {A, C, N}: the carry loops over more than 1024 scan blocks
    alpha = [b""] + [bytes(p) for L in (1, 2, 3) for p in np.array(np.meshgrid(*[[65, 67, 78]] * L)).reshape(L, -1).T.tolist()]
    n = 1_100_000
    pick = np.random.default_rng(9).integers(0, len(alpha), n)
    seqs = [alpha[i] for i in range(len(alpha))]
    lens = np.array([len(s) for s in seqs], np.int64)[pick]
    offs = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    buf = np.frombuffer(b"".join(seqs[i] for i in pick), np.uint8).copy()
    for tail in ("single", "drop"):
        table = ref.rows(np.frombuffer(b"".join(seqs), np.uint8), np.concatenate([[0], np.cumsum([len(s) for s in seqs])]), "DNA", 2,
                         2, tail == "single", True, False)
        want = np.concatenate([table[i] for i in pick]).astype(np.int32)
        cu = np.zeros(n + 1, np.int64)
        np.cumsum(np.array([table[i].size for i in range(len(table))])[pick], out=cu[1:])
        vb = batch_tokenize_kmer(tokenizer("DNA", True, False, False), cuda(buf, offs), 2, stride=2, tail=tail, varlen=True)
        torch.cuda.synchronize()
        assert_same_bits(cu.astype(np.int32), vb.cu_seqlens.cpu().numpy())
        assert_same_bits(want, vb.tokens.cpu().numpy())


# ------------------------------------------------------------------------------------------------------------------
def forms(buf, offs, tmp_path, name):
    """The batch as a list of bytes, host numpy, pinned torch, CUDA tensors and a FlatFile range (offsets[0] != 0)."""
    seqs = [buf[offs[i]:offs[i + 1]].tobytes() for i in range(offs.size - 1)]
    path = tmp_path / f"{name}.ff"
    path.write_bytes(flatfile_image([b"ACGTACGT"] + seqs))
    ff = cbioseq.FlatFile(str(path))
    return [("list", seqs), ("host", (buf, offs)), ("pinned", (torch.from_numpy(buf).pin_memory(), torch.from_numpy(offs).pin_memory())),
            ("cuda", cuda(buf, offs)), ("flatfile", (ff, 1, 1 + len(seqs)))]


def test_every_batch_form(tmp_path):
    lens = np.random.default_rng(4).integers(0, 400, 900)
    buf, offs = batch_of(lens, 4)
    for name, batch in forms(buf, offs, tmp_path, "f"):
        run_both(batch, buf, offs, "DNA", 6, 1, "drop", (True, True, True))
        run_both(batch, buf, offs, "DNA", 6, 6, "single", (True, False, False))


@pytest.mark.parametrize("mode", ["head", "random"])
def test_crop_equals_crop_packed_then_kmer(mode, tmp_path):
    lens = np.random.default_rng(5).integers(0, 3000, 700)
    buf, offs = batch_of(lens, 5)
    W, seed, base = 1000, 1234, 7
    cb = crop_packed(*cuda(buf, offs), W, crop=mode, seed=seed, seq_index_base=base)
    cbuf, coffs = cb.bytes.cpu().numpy(), cb.offsets.cpu().numpy()
    t = bioseq_b200.pbeos_tokenizers["DNA"]
    for name, batch in forms(buf, offs, tmp_path, mode):
        if name == "flatfile":
            continue  # (its sequence indices start at 1: a different random window)
        for s, tail in ((1, "drop"), (6, "single")):
            out = batch_tokenize_kmer(t, batch, 6, 1002, stride=s, tail=tail, crop=mode, crop_len=W, seed=seed, seq_index_base=base)
            check_padded(out, cbuf, coffs, "DNA", 6, s, tail, (True, True, True), 1002)
            vb = batch_tokenize_kmer(t, batch, 6, stride=s, tail=tail, varlen=True, crop=mode, crop_len=W, seed=seed,
                                     seq_index_base=base)
            check_varlen(vb, cbuf, coffs, "DNA", 6, s, tail, (True, True, True))


def test_errors_for_host_and_cuda_batches():
    t = bioseq_b200.pbeos_tokenizers["DNA"]
    buf, offs = batch_of([10, 20, 30], 6)
    for batch in ((buf, offs), cuda(buf, offs), [buf[offs[i]:offs[i + 1]].tobytes() for i in range(3)]):
        with pytest.raises(ValueError, match="k-mer tokens \\+ bos \\+ eos > padlen: 30, vs padlen 29"):
            batch_tokenize_kmer(t, batch, 3, 29)
        batch_tokenize_kmer(t, batch, 3, 30)
        with pytest.raises(ValueError, match="padlen"):
            batch_tokenize_kmer(t, batch, 3)
        with pytest.raises(ValueError, match="padlen must not be given"):
            batch_tokenize_kmer(t, batch, 3, 40, varlen=True)
        with pytest.raises(ValueError, match="crop_len"):
            batch_tokenize_kmer(t, batch, 3, varlen=True, crop="head")
    bad = np.array([0, 10, 5, 30], np.int64)
    for batch in ((buf, bad), cuda(buf, bad)):
        with pytest.raises(ValueError, match="non-decreasing"):
            batch_tokenize_kmer(t, batch, 3, 64)
    with pytest.raises(ValueError, match="past the end"):
        batch_tokenize_kmer(t, cuda(buf, np.array([0, 10, 20, 61], np.int64)), 3, 64)
    # more than 2^31 - 1 tokens: k = 1, no specials, 2^31 residues
    t0 = bioseq_b200.DNATokenizer
    offs = np.array([0, 2 ** 30, 2 ** 31], np.int64)
    host = np.zeros(2 ** 31, np.uint8)  # (never staged: the size check comes first)
    with pytest.raises(ValueError, match="2\\^31 - 1"):
        batch_tokenize_kmer(t0, (host, offs), 1, varlen=True)
    del host
    dev = torch.full((2 ** 31,), 65, dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError, match="2\\^31 - 1"):
        batch_tokenize_kmer(t0, (dev, torch.from_numpy(offs).cuda()), 1, varlen=True)
    ok = batch_tokenize_kmer(t0, (dev, torch.from_numpy(offs - np.array([0, 0, 1])).cuda()), 1, varlen=True)
    assert ok.tokens.numel() == 2 ** 31 - 1 and ok.cu_seqlens.tolist() == [0, 2 ** 30, 2 ** 31 - 1]
    assert bool((ok.tokens[-1000:] == 0).all()) and bool((ok.tokens[:1000] == 0).all())
    del dev, ok
    torch.cuda.empty_cache()


def test_back_to_back_launches_and_a_cuda_graph():
    tok = consumers.descriptor(bioseq_b200.pbeos_tokenizers["DNA"])
    lens = np.random.default_rng(8).integers(0, 2000, 3000)
    buf_a, offs = batch_of(lens, 80)
    buf_b, _ = batch_of(lens, 81)
    km1, km6 = capi.kmer_desc(tok, 6, 1, capi.KMER_DROP), capi.kmer_desc(tok, 6, 6, capi.KMER_SINGLE)
    n = lens.size
    P = int(ref.count(lens, 6, 1, False, 1, 1).max())
    total6 = int(ref.count(lens, 6, 6, True, 1, 1).sum())
    want = {}
    for name, buf in (("a", buf_a), ("b", buf_b)):
        want[name] = (ref.padded(buf, offs, "DNA", 6, 1, False, True, True, True, P).astype(np.int32),
                      ref.varlen(buf, offs, "DNA", 6, 6, True, True, True))
    da, db = cuda(buf_a, offs), cuda(buf_b, offs)
    out = torch.zeros((n, P), dtype=torch.int32, device="cuda")
    vt = torch.zeros(total6, dtype=torch.int32, device="cuda")
    cu = torch.zeros(n + 1, dtype=torch.int32, device="cuda")

    def launch(st, d):
        capi.tokenize_kmer(0, st, d[0], d[1], n, P, tok, km1, capi.I32, out)
        capi.tokenize_kmer_varlen(0, st, d[0], d[1], n, tok, km6, capi.I32, vt, cu)

    def expect(name):
        torch.cuda.synchronize()
        p, (toks, c, _) = want[name]
        assert_same_bits(p, out.cpu().numpy())
        assert_same_bits(toks.astype(np.int32), vt.cpu().numpy())
        assert_same_bits(c, cu.cpu().numpy())

    st = torch.cuda.current_stream().cuda_stream
    for i in range(50):
        launch(st, da if i % 2 == 0 else db)
    expect("b")
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch(torch.cuda.current_stream().cuda_stream, da)
    for _ in range(2):
        for x in (out, vt, cu):
            x.zero_()
        g.replay()
        expect("a")
        launch(torch.cuda.current_stream().cuda_stream, db)
        expect("b")
