"""Cropping over-long sequences (crop_packed / crop= / bsq_crop, kernel K9), bit for bit against the rule of
include/bsq.h (tests/crop_reference.py).

K9 scans the cropped lengths per block of 1024 rows, carries the block totals over (one CTA, only with more than one
block) and copies each row's window with one warp: destination-aligned 16-byte stores from realigned source words,
byte stores at either end of a row.  The cases cover window lengths around the 16-byte vector, every source
alignment, offsets[0] != 0, empty batches and rows, more than one scan block, a sequence over 10^6 residues, slicing,
every consumer with crop= against the same consumer on the reference-cropped batch (and the oracle), back-to-back
launches, concurrent streams, a CUDA graph captured through the C ABI, and the dataset."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from bioseq_b200 import capi, cbioseq, consumers, crop_packed, batch_tokenize_cropped, CroppedBatch  # noqa: E402
from bioseq_b200 import batch_tokenize_varlen, batch_tokenize_mlm, batch_onehot_encode_bcl, batch_embed  # noqa: E402
from bioseq_b200.loaders import FlatFileDataset  # noqa: E402
from oracle import oracle  # noqa: E402
from oracle.oracle import OracleTokenizer, flatfile_image  # noqa: E402
from helpers import assert_same_bits, gen  # noqa: E402
from crop_reference import crop as reference_crop  # noqa: E402

AA = b"ACDEFGHIKLMNPQRSTVWY"
MIX = b"ACDEFGHIKLMNPQRSTVWYacdefghiklmnpqrstvwyXBZOUJ*-NnUu .\x00\x7f\x80\xc3\xff"
FLAGS = [(b, e, p) for b in (False, True) for e in (False, True) for p in (False, True)]


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests selected but no CUDA device is visible")


def cuda(buf, offs):
    return torch.from_numpy(np.ascontiguousarray(buf)).cuda(), torch.from_numpy(np.ascontiguousarray(offs)).cuda()


def check_crop(cb, buf, offs, W, random, seed=0, base=0):
    wb, wo, ws = reference_crop(buf, offs, W, random, seed, base)
    torch.cuda.synchronize()
    assert isinstance(cb, CroppedBatch)
    assert_same_bits(wo, cb.offsets.cpu().numpy())
    assert_same_bits(ws, cb.starts.cpu().numpy())
    assert_same_bits(wb, cb.bytes.cpu().numpy())


def lengths_0_to_3w(W, seed, n=600):
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 3 * W + 1, size=n)
    lens[:6] = [W - 1 if W > 1 else 0, W, W + 1, 0, 3 * W, 1]
    return lens


def batch_of(lens, seed, alphabet=MIX, lead=0):
    offs = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    rng = np.random.default_rng(seed)
    table = np.frombuffer(alphabet, np.uint8)
    buf = table[rng.integers(0, table.size, size=int(offs[-1]) + lead)]
    return buf, offs + lead


@pytest.mark.parametrize("W", [1, 15, 16, 17, 1022, 4096])
@pytest.mark.parametrize("random", [False, True])
def test_crop_packed_matches_reference(W, random):
    lens = lengths_0_to_3w(W, W, n=600 if W < 1000 else 150)
    for lead in (0, 5):  # offsets[0] != 0
        buf, offs = batch_of(lens, W + lead, lead=lead)
        b, o = cuda(buf, offs)
        check_crop(crop_packed(b, o, W, crop="random" if random else "head", seed=0x9E3779B97F4A7C15, seq_index_base=17),
                   buf, offs, W, random, 0x9E3779B97F4A7C15, 17)


@pytest.mark.parametrize("shift", range(16))
def test_every_source_and_destination_alignment(shift):
    # shifted inputs move every row's source alignment; ragged kept lengths move the destination alignment
    lens = lengths_0_to_3w(37, 100 + shift, n=2500)  # 2500 rows: three scan blocks
    buf, offs = batch_of(lens, shift, lead=shift)
    b, o = cuda(buf, offs)
    for random in (False, True):
        check_crop(crop_packed(b, o, 37, crop="random" if random else "head", seed=shift), buf, offs, 37, random, shift)
    # a base pointer that is not 16-byte aligned either
    bb = torch.zeros(buf.size + 16, dtype=torch.uint8, device="cuda")
    bb[shift:shift + buf.size] = b
    o2 = o + shift
    check_crop(crop_packed(bb, o2, 23, seed=3), np.concatenate([np.zeros(shift, np.uint8), buf]), offs + shift, 23, True, 3)


def test_empty_batch_empty_rows_and_one_huge_row():
    e = crop_packed(torch.zeros(0, dtype=torch.uint8, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda"), 8)
    assert e.bytes.numel() == 0 and e.offsets.tolist() == [0] and e.starts.numel() == 0
    buf, offs = batch_of([0, 0, 0], 1)
    b, o = cuda(buf, offs)
    check_crop(crop_packed(b, o, 8), buf, offs, 8, True)
    # one sequence over 10^6 residues among short ones
    buf, offs = batch_of([5, 1_234_567, 0, 99, 3000], 2, alphabet=AA, lead=3)
    b, o = cuda(buf, offs)
    for W in (1, 4096, 1_000_000, 2_000_000):
        for random in (False, True):
            check_crop(crop_packed(b, o, W, crop="random" if random else "head", seed=W), buf, offs, W, random, W)
    # many scan blocks (rows > 1024 * 1024 would need a second carry round; 300 000 rows take 293 blocks)
    lens = np.random.default_rng(4).integers(0, 60, size=300_000)
    buf, offs = batch_of(lens, 4, alphabet=b"ACGT")
    b, o = cuda(buf, offs)
    check_crop(crop_packed(b, o, 31, seed=8), buf, offs, 31, True, 8)


def test_slicing_and_identity():
    buf, offs = batch_of(lengths_0_to_3w(100, 9, n=5000), 9)
    b, o = cuda(buf, offs)
    full = crop_packed(b, o, 100, seed=44)
    torch.cuda.synchronize()
    fo = full.offsets.cpu().numpy()
    for a, z in ((0, 1), (1, 1025), (1000, 4999), (4000, 5000)):
        part = crop_packed(b, o[a:z + 1].contiguous(), 100, seed=44, seq_index_base=a)
        torch.cuda.synchronize()
        assert torch.equal(part.starts, full.starts[a:z])
        assert torch.equal(part.bytes, full.bytes[int(fo[a]):int(fo[z])])
        assert torch.equal(part.offsets, full.offsets[a:z + 1] - int(fo[a]))
    W = int(np.diff(offs).max())
    for mode in ("head", "random"):
        same = crop_packed(b, o, W, crop=mode, seed=1)
        torch.cuda.synchronize()
        assert torch.equal(same.bytes, b[int(offs[0]):int(offs[-1])]) and torch.equal(same.offsets, o - int(offs[0]))
        assert not same.starts.any()


# ------------------------------------------------------------------------------------------------------------------
def forms(buf, offs, tmp_path, name):
    """The batch as a list of bytes, host numpy, pinned torch, CUDA tensors and a FlatFile range (offsets[0] != 0)."""
    seqs = [buf[offs[i]:offs[i + 1]].tobytes() for i in range(offs.size - 1)]
    path = tmp_path / f"{name}.ff"
    path.write_bytes(flatfile_image([b"MKV"] + seqs))
    ff = cbioseq.FlatFile(str(path))
    return [("list", seqs, 0), ("host", (buf, offs), 0), ("pinned", (torch.from_numpy(buf).pin_memory(), torch.from_numpy(offs).pin_memory()), 0),
            ("cuda", cuda(buf, offs), 0), ("flatfile", (ff, 1, 1 + len(seqs)), 1)]


def ascii_batch(n, lo, hi, seed):
    return gen(seed, n, lo, hi, AA + b"xbz*")


@pytest.mark.parametrize("flags", FLAGS)
def test_padded_consumers_match_uncropped_on_cropped_batch(flags, tmp_path):
    bos, eos, pad = flags
    tok = cbioseq.Tokenizer("PROTEIN", bos=bos, eos=eos, padchar=pad)
    orc = OracleTokenizer("PROTEIN", bos=bos, eos=eos, padchar=pad)
    k = int(bos) + int(eos)
    buf, offs = ascii_batch(700, 0, 300, 11)
    P = 128
    W = P - k
    weight = torch.randn(tok.alphabet_size(), 16, device="cuda")
    for name, batch, base in forms(buf, offs, tmp_path, "p"):
        for mode in ("head", "random"):
            random = mode == "random"
            kw = dict(crop=mode, seed=5, seq_index_base=base)
            cb, co, _ = reference_crop(buf, offs, W, random, 5, base)
            ref = (cb, co)
            for destchar in ("B", "i", "f"):
                got = batch_tokenize_cropped(tok, batch, P, destchar, batch_first=True, **kw)
                want = orc.batch_tokenize(ref, padlen=P, destchar=destchar, batch_first=True)  # the oracle on the cropped items
                torch.cuda.synchronize()
                assert_same_bits(want, got.cpu().numpy())
            got = batch_tokenize_cropped(tok, batch, P, "B", batch_first=False, crop_len=W - 7, **kw)
            cb7, co7, _ = reference_crop(buf, offs, W - 7, random, 5, base)
            torch.cuda.synchronize()
            assert_same_bits(orc.batch_tokenize((cb7, co7), padlen=P, destchar="B", batch_first=False), got.cpu().numpy())
            got = batch_onehot_encode_bcl(tok, batch, P, "f", **kw)
            want = batch_onehot_encode_bcl(tok, cuda(*ref), P, "f")
            assert torch.equal(got, want)
            got = batch_embed(tok, batch, weight, P, **kw)
            assert torch.equal(got, batch_embed(tok, cuda(*ref), weight, P))
            got = batch_tokenize_mlm(tok, batch, P, "l", **kw)
            want = batch_tokenize_mlm(tok, cuda(*ref), P, "l", seed=5, seq_index_base=base)
            assert torch.equal(got.inputs, want.inputs) and torch.equal(got.labels, want.labels)


@pytest.mark.parametrize("flags", [(True, True, True), (False, False, False), (True, False, False)])
def test_varlen_consumers_match_uncropped_on_cropped_batch(flags, tmp_path):
    bos, eos, pad = flags
    tok = cbioseq.Tokenizer("PROTEIN", bos=bos, eos=eos, padchar=pad)
    k = int(bos) + int(eos)
    buf, offs = ascii_batch(900, 0, 400, 12)
    W = 150
    for name, batch, base in forms(buf, offs, tmp_path, "v"):
        for mode in ("head", "random"):
            cb, co, _ = reference_crop(buf, offs, W, mode == "random", 6, base)
            ref = cuda(cb, co)
            for destchar in ("B", "l"):
                got = batch_tokenize_varlen(tok, batch, destchar, crop=mode, crop_len=W, seed=6, seq_index_base=base)
                want = batch_tokenize_varlen(tok, ref, destchar)
                assert torch.equal(got.tokens, want.tokens) and torch.equal(got.cu_seqlens, want.cu_seqlens)
                lens = np.minimum(np.diff(offs), W) + k
                assert got.max_seqlen == int(lens.max())
                assert got.cu_seqlens.cpu().numpy().tolist() == np.concatenate([[0], np.cumsum(lens)]).tolist()
            got = batch_tokenize_mlm(tok, batch, varlen=True, crop=mode, crop_len=W, seed=6, seq_index_base=base)
            want = batch_tokenize_mlm(tok, ref, varlen=True, seed=6, seq_index_base=base)
            assert torch.equal(got.inputs.tokens, want.inputs.tokens) and torch.equal(got.labels, want.labels)


def test_augment_and_mlm_after_crop():
    tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    orc = OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    buf, offs = gen(31, 1500, 1, 900, AA)
    W, P = 254, 256
    cb, co, _ = reference_crop(buf, offs, W, True, 11, 40)
    mut = oracle.augment(cb, co, chain_len=2, augment_frac=0.7, seed=11, seq_index_base=40)
    for batch in ((buf, offs), cuda(buf, offs)):
        got = batch_tokenize_cropped(tok, batch, P, augment=2, augment_frac=0.7, seed=11, seq_index_base=40)
        torch.cuda.synchronize()
        assert_same_bits(orc.batch_tokenize((mut, co), padlen=P, destchar="B", batch_first=True), got.cpu().numpy())
        got = batch_tokenize_mlm(tok, batch, P, augment=2, augment_frac=0.7, seed=11, seq_index_base=40, crop="random")
        want = batch_tokenize_mlm(tok, cuda(mut, co), P, seed=11, seq_index_base=40)
        assert torch.equal(got.inputs, want.inputs) and torch.equal(got.labels, want.labels)
    d = cuda(buf, offs)
    batch_tokenize_cropped(tok, d, P, augment=2, seed=11)
    torch.cuda.synchronize()
    assert np.array_equal(d[0].cpu().numpy(), buf)  # the caller's residues are not mutated


def test_crop_extent_device_and_errors():
    buf, offs = gen(3, 500, 0, 300, AA)
    b, o = cuda(buf, offs)
    assert capi.crop_extent_device(0, torch.cuda.current_stream().cuda_stream, o, 500, 100, nbytes=b.numel()) == (
        int(np.minimum(np.diff(offs), 100).sum()), 100)
    bad = o.clone()
    bad[10] = bad[11] + 1
    with pytest.raises(ValueError):
        crop_packed(b, bad, 100)
    with pytest.raises(ValueError):
        crop_packed(b[:-1], o, 100)  # offsets run past the end of bytes
    tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    with pytest.raises(ValueError):
        batch_tokenize_cropped(tok, (b, bad), 64)


def test_back_to_back_graph_and_streams():
    tok_py = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    orc = OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    tok = consumers.descriptor(tok_py)
    lens = np.random.default_rng(5).integers(10, 3000, size=4000)
    buf_a, offs = batch_of(lens, 50, alphabet=AA)
    buf_b, _ = batch_of(lens, 51, alphabet=AA)
    W, P, n = 1022, 1024, lens.size
    seeds = (7, 8)
    want = {}
    for name, buf in (("a", buf_a), ("b", buf_b)):
        for s in seeds:
            cb, co, cs = reference_crop(buf, offs, W, True, s, 0)
            want[name, s] = (cb, co, cs, orc.batch_tokenize((cb, co), padlen=P, destchar="B", batch_first=True))
    da, db = cuda(buf_a, offs), cuda(buf_b, offs)
    total = int(np.minimum(lens, W).sum())
    ob = torch.zeros(total, dtype=torch.uint8, device="cuda")
    oo = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    os_ = torch.zeros(n, dtype=torch.int64, device="cuda")
    out = torch.zeros((n, P), dtype=torch.uint8, device="cuda")

    def launch(st, d, seed):
        capi.crop(0, st, d[0], d[1], n, W, True, seed, 0, ob, oo, os_)
        capi.tokenize(0, st, ob, oo, n, P, tok, True, capi.I8, out)

    def expect(key):
        torch.cuda.synchronize()
        cb, co, cs, t = want[key]
        assert_same_bits(cb, ob.cpu().numpy())
        assert_same_bits(co, oo.cpu().numpy())
        assert_same_bits(cs, os_.cpu().numpy())
        assert_same_bits(t, out.cpu().numpy())

    st = torch.cuda.current_stream().cuda_stream
    for i in range(20):
        launch(st, da if i % 2 == 0 else db, seeds[i % 2])
    expect(("b", 8))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(5):
            launch(torch.cuda.current_stream().cuda_stream, da if i % 2 == 0 else db, seeds[i % 2])
    for _ in range(2):
        for t in (ob, oo, os_, out):
            t.zero_()
        g.replay()
        expect(("a", 7))
        launch(torch.cuda.current_stream().cuda_stream, db, 7)
        expect(("b", 7))
    streams = [torch.cuda.Stream() for _ in range(4)]
    outs = [(torch.zeros(total, dtype=torch.uint8, device="cuda"), torch.zeros(n + 1, dtype=torch.int64, device="cuda"))
            for _ in streams]
    torch.cuda.synchronize()
    for rep in range(3):
        for j, (s, (b_, o_)) in enumerate(zip(streams, outs)):
            capi.crop(0, s.cuda_stream, (da if j % 2 == 0 else db)[0], da[1], n, W, True, seeds[j % 2], 0, b_, o_)
    torch.cuda.synchronize()
    for j, (b_, o_) in enumerate(outs):
        cb, co, _, _ = want["a" if j % 2 == 0 else "b", seeds[j % 2]]
        assert_same_bits(cb, b_.cpu().numpy())
        assert_same_bits(co, o_.cpu().numpy())


# ------------------------------------------------------------------------------------------------------------------
def test_dataset_on_long_sequences(tmp_path):
    tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    rng = np.random.default_rng(77)
    lens = rng.integers(1, 400, size=1200)
    lens[[3, 500, 1100]] = [34_000, 5000, 1023]
    table = np.frombuffer(AA, np.uint8)
    seqs = [table[rng.integers(0, 20, size=int(n))].tobytes() for n in lens]
    path = tmp_path / "long.ff"
    path.write_bytes(flatfile_image(seqs))
    ff = cbioseq.FlatFile(str(path))
    assert ff.maxseqlen == 34_000
    L = 1024

    def seed_of(draw, base=13):
        return (base & 0xFFFFFFFF) | (draw << 32)

    ds = FlatFileDataset(ff, tok, max_seq_len=L, mlm=True)
    mb = ds[0:600]
    assert mb.inputs.shape == (600, L) and mb.labels.shape == (600, L)
    ds = FlatFileDataset(ff, tok, max_seq_len=L, mlm=True, varlen=True)
    vb = ds[0:600].inputs
    assert vb.max_seqlen == L and vb.cu_seqlens[-1].item() == int(np.minimum(lens[:600], L - 2).sum()) + 2 * 600
    ds = FlatFileDataset(ff, tok, max_seq_len=L, varlen=True)
    assert ds[0:600].max_seqlen == L and ds[3].numel() == L
    ds = FlatFileDataset(ff, tok, max_seq_len=L, cnn=True)
    assert ds[0:64].shape == (64, tok.alphabet_size(), L) and ds[3].shape == (L, tok.alphabet_size())
    # head mode is truncation
    ds = FlatFileDataset(ff, tok, max_seq_len=L, crop="head")
    got = ds[0:1200]
    want = tok.batch_tokenize([s[:L - 2] for s in seqs], padlen=L, batch_first=True, destchar="B").to(torch.long)
    assert got.shape == (1200, L) and torch.equal(got, want)
    # random mode: a new window every fetch, reproducible from the seed, always a substring of the stored sequence
    ds = FlatFileDataset(ff, tok, max_seq_len=L)
    a, b = ds[0:1200], ds[0:1200]
    assert a.shape == (1200, L) and not torch.equal(a, b)
    assert torch.equal(a, batch_tokenize_cropped(tok, (ff, 0, 1200), L, seed=seed_of(1)).to(torch.long))
    again = FlatFileDataset(ff, tok, max_seq_len=L)[0:1200]
    assert torch.equal(again, a)
    text = tok.decode_tokens(a.to(torch.uint8))
    for i in (3, 500, 1100, 7):
        window = text[i].replace("<BOS>", "").replace("<EOS>", "").replace("<PAD>", "").encode()
        assert window in seqs[i] and len(window) == min(int(lens[i]), L - 2)
    item, raw = ds.fetch(3, return_items=True)
    assert item.shape == (L,) and bytes(raw) == seqs[3]  # the stored, uncropped item
    # without max_seq_len nothing changes: rows are as wide as the longest sequence
    assert FlatFileDataset(ff, tok)[0:4].shape == (4, 34_002)
