"""Reverse complement (revcomp_packed / rc= / bsq_revcomp, kernel K12), bit for bit against the rule of include/bsq.h
(tests/revcomp_reference.py).

K12 is a flat map over 16-byte output vectors in 64 KiB tiles: each tile searches its first row, keeps its rows' starts
and flip bits in shared memory (or, past 2047 rows, reads them in global memory), and builds each vector from one
whole-vector result per row it touches.  The cases cover lengths around the 16-byte vector and the tile, a row of
2^24 + 3 bytes, empty rows and batches, every source and destination alignment, all 256 byte values, each mode at
rc_prob 0, 1 and 0.5, over-full tiles, a batch past 2^31 bytes into its buffer, the caller's tensors, a side stream, a
CUDA graph captured through the C ABI, every consumer with rc= against the same consumer on the reference-flipped batch,
and the dataset."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from bioseq_b200 import capi, cbioseq, consumers, revcomp_packed, batch_tokenize_revcomp, RevCompBatch  # noqa: E402
from bioseq_b200 import batch_tokenize_cropped, batch_tokenize_varlen, batch_tokenize_mlm, batch_tokenize_seqpack  # noqa: E402
from bioseq_b200 import batch_tokenize_kmer, batch_onehot_encode_bcl, batch_embed  # noqa: E402
from bioseq_b200.loaders import FlatFileDataset  # noqa: E402
from oracle.oracle import OracleTokenizer, flatfile_image  # noqa: E402
from helpers import assert_same_bits, gen, table_cap_lens  # noqa: E402
from revcomp_reference import revcomp as reference_revcomp  # noqa: E402
from crop_reference import crop as reference_crop  # noqa: E402

DNA = b"ACGTNacgtnRYKMBVDHSWUu-*"
ALL = bytes(range(256))
MODES = [("always", None), ("both", None), ("random", 0.0), ("random", 1.0), ("random", 0.5)]


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests selected but no CUDA device is visible")


def cuda(buf, offs):
    return torch.from_numpy(np.ascontiguousarray(buf)).cuda(), torch.from_numpy(np.ascontiguousarray(offs)).cuda()


def batch_of(lens, seed, alphabet=DNA, lead=0):
    offs = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    rng = np.random.default_rng(seed)
    table = np.frombuffer(alphabet, np.uint8)
    buf = table[rng.integers(0, table.size, size=int(offs[-1]) + lead)]
    return buf, offs + lead


def check(rb, buf, offs, mode, rc_prob=None, seed=0, base=0):
    wb, wo, wf = reference_revcomp(buf, offs, mode, 0.5 if rc_prob is None else rc_prob, seed, base)
    torch.cuda.synchronize()
    assert isinstance(rb, RevCompBatch) and rb.flipped.dtype == torch.bool
    assert_same_bits(wo, rb.offsets.cpu().numpy())
    assert_same_bits(wf, rb.flipped.cpu().numpy())
    assert_same_bits(wb, rb.bytes.cpu().numpy())


EDGE = [0, 1, 15, 16, 17, 31, 32, 33, 511, 512, 513, 10_000]


@pytest.mark.parametrize("mode,rc_prob", MODES)
def test_edge_lengths_every_source_alignment(mode, rc_prob):
    rng = np.random.default_rng(1)
    lens = np.concatenate([EDGE, rng.choice(EDGE, size=400), rng.integers(0, 200, size=400)])
    for lead in range(16):  # every offsets[0] % 16
        buf, offs = batch_of(lens, lead, alphabet=ALL, lead=lead)
        b, o = cuda(buf, offs)
        b0, o0 = b.clone(), o.clone()
        check(revcomp_packed(b, o, rc=mode, rc_prob=rc_prob, seed=0x9E3779B97F4A7C15, seq_index_base=17), buf, offs, mode, rc_prob,
              0x9E3779B97F4A7C15, 17)
        assert torch.equal(b, b0) and torch.equal(o, o0)  # the caller's tensors are unchanged


# random rows; the same ending in a run of empty rows (every alignment but one leaves the last vector partial); rows that
# fill tiles to the row table's cap and one past it
DEST_LENS = [np.random.default_rng(2).integers(0, 300, size=2000),
             np.concatenate([np.random.default_rng(2).integers(0, 300, size=500), np.zeros(40, np.int64)]), table_cap_lens()]


@pytest.mark.parametrize("mode,rc_prob", MODES)
def test_every_destination_alignment(mode, rc_prob):
    for lens in DEST_LENS:
        buf, offs = batch_of(lens, 3, lead=5)
        b, o = cuda(buf, offs)
        wb, wo, wf = reference_revcomp(buf, offs, mode, 0.5 if rc_prob is None else rc_prob, 4, 9)
        st = torch.cuda.current_stream().cuda_stream
        for shift in range(16):
            ob = torch.full((wb.size + 64,), 0xA5, dtype=torch.uint8, device="cuda")
            oo = torch.empty(wo.size, dtype=torch.int64, device="cuda")
            of = torch.empty(wf.size, dtype=torch.uint8, device="cuda")
            mode_i = consumers._RC_MODES[mode]
            capi.revcomp(0, st, b, o, offs.size - 1, mode_i, rc_prob or 0.0, 4, 9, ob.data_ptr() + shift, oo, of)
            torch.cuda.synchronize()
            got = ob.cpu().numpy()
            assert_same_bits(wb, got[shift:shift + wb.size])
            assert (got[:shift] == 0xA5).all() and (got[shift + wb.size:] == 0xA5).all()  # nothing written outside
            assert_same_bits(wo, oo.cpu().numpy())
            assert_same_bits(wf.astype(np.uint8), of.cpu().numpy())


def test_empty_batches_huge_row_and_overfull_tiles():
    for mode, rc_prob in MODES:
        e = revcomp_packed(torch.zeros(0, dtype=torch.uint8, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda"),
                           rc=mode, rc_prob=rc_prob)
        assert e.bytes.numel() == 0 and e.offsets.tolist() == [0] and e.flipped.numel() == 0
        buf, offs = batch_of([0, 0, 0], 1)
        check(revcomp_packed(*cuda(buf, offs), rc=mode, rc_prob=rc_prob), buf, offs, mode, rc_prob)
    # one row of 2^24 + 3 bytes among short ones: one row spans hundreds of tiles
    buf, offs = batch_of([5, 2 ** 24 + 3, 0, 99], 2, lead=3)
    b, o = cuda(buf, offs)
    for mode, rc_prob in MODES:
        check(revcomp_packed(b, o, rc=mode, rc_prob=rc_prob, seed=3), buf, offs, mode, rc_prob, 3)
    # tiles of more than 2047 rows (short and empty rows): rows and coins read in global memory, several rows per vector
    lens = np.random.default_rng(4).integers(0, 12, size=300_000)
    lens[1000:60_000] = 0
    buf, offs = batch_of(lens, 4, alphabet=ALL, lead=9)
    b, o = cuda(buf, offs)
    for mode, rc_prob in MODES:
        check(revcomp_packed(b, o, rc=mode, rc_prob=rc_prob, seed=8, seq_index_base=2 ** 33), buf, offs, mode, rc_prob, 8, 2 ** 33)


def test_batch_past_2_pow_31_bytes_into_its_buffer():
    lens = np.random.default_rng(6).integers(0, 5000, size=3000)
    buf, offs = batch_of(lens, 6)
    lead = 2 ** 31 + 5
    big = torch.empty(lead + buf.size, dtype=torch.uint8, device="cuda")
    big[lead:] = torch.from_numpy(buf).cuda()
    o = torch.from_numpy(offs + lead).cuda()
    for mode, rc_prob in (("always", None), ("both", None), ("random", 0.5)):
        check(revcomp_packed(big, o, rc=mode, rc_prob=rc_prob, seed=12), buf, offs, mode, rc_prob, 12)
    del big
    torch.cuda.empty_cache()


def test_slicing_and_double_flip():
    buf, offs = batch_of(np.random.default_rng(9).integers(0, 400, size=5000), 9, alphabet=b"ACGTNacgtn")
    b, o = cuda(buf, offs)
    full = revcomp_packed(b, o, rc="random", seed=44)
    torch.cuda.synchronize()
    fo = full.offsets.cpu().numpy()
    for a, z in ((0, 1), (1, 1025), (1000, 4999), (4000, 5000)):
        part = revcomp_packed(b, o[a:z + 1].contiguous(), rc="random", seed=44, seq_index_base=a)
        torch.cuda.synchronize()
        assert torch.equal(part.flipped, full.flipped[a:z])
        assert torch.equal(part.bytes, full.bytes[int(fo[a]):int(fo[z])])
    twice = revcomp_packed(*revcomp_packed(b, o)[:2])
    torch.cuda.synchronize()
    assert torch.equal(twice.bytes, b) and torch.equal(twice.offsets, o - int(offs[0]))


def test_side_stream_graph_and_back_to_back():
    lens = np.random.default_rng(5).integers(10, 3000, size=4000)
    buf_a, offs = batch_of(lens, 50)
    buf_b, _ = batch_of(lens, 51)
    n, total = lens.size, int(lens.sum())
    want = {(name, s): reference_revcomp(buf, offs, "random", 0.5, s, 0) for name, buf in (("a", buf_a), ("b", buf_b)) for s in (7, 8)}
    da, db = cuda(buf_a, offs), cuda(buf_b, offs)
    ob = torch.zeros(total, dtype=torch.uint8, device="cuda")
    oo = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    of = torch.zeros(n, dtype=torch.uint8, device="cuda")

    def launch(st, d, seed):
        capi.revcomp(0, st, d[0], d[1], n, capi.RC_RANDOM, 0.5, seed, 0, ob, oo, of)

    def expect(key):
        torch.cuda.synchronize()
        wb, wo, wf = want[key]
        assert_same_bits(wb, ob.cpu().numpy())
        assert_same_bits(wo, oo.cpu().numpy())
        assert_same_bits(wf.astype(np.uint8), of.cpu().numpy())

    for i in range(20):
        launch(torch.cuda.current_stream().cuda_stream, da if i % 2 == 0 else db, 7 + i % 2)
    expect(("b", 8))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        launch(side.cuda_stream, da, 8)
    torch.cuda.current_stream().wait_stream(side)
    expect(("a", 8))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(5):
            launch(torch.cuda.current_stream().cuda_stream, da if i % 2 == 0 else db, 7)
    for _ in range(2):
        for t in (ob, oo, of):
            t.zero_()
        g.replay()
        expect(("a", 7))
        launch(torch.cuda.current_stream().cuda_stream, db, 8)
        expect(("b", 8))
    da[0].copy_(db[0])  # a replay reads the inputs as they are now
    g.replay()
    expect(("b", 7))


# ------------------------------------------------------------------------------------------------------------------
def forms(buf, offs, tmp_path, name):
    """The batch as a list of bytes, host numpy, CUDA tensors and a FlatFile range (offsets[0] != 0)."""
    seqs = [buf[offs[i]:offs[i + 1]].tobytes() for i in range(offs.size - 1)]
    path = tmp_path / f"{name}.ff"
    path.write_bytes(flatfile_image([b"ACG"] + seqs))
    ff = cbioseq.FlatFile(str(path))
    return [("list", seqs, 0), ("host", (buf, offs), 0), ("cuda", cuda(buf, offs), 0), ("flatfile", (ff, 1, 1 + len(seqs)), 1)]


@pytest.mark.parametrize("flags", [(True, True, True), (False, False, False), (True, False, True)])
def test_padded_consumers_match_on_flipped_batch(flags, tmp_path):
    bos, eos, pad = flags
    tok = cbioseq.Tokenizer("DNA5", bos=bos, eos=eos, padchar=pad)
    orc = OracleTokenizer("DNA5", bos=bos, eos=eos, padchar=pad)
    k = int(bos) + int(eos)
    buf, offs = gen(11, 700, 0, 126, DNA)
    P = 128
    weight = torch.randn(tok.alphabet_size(), 16, device="cuda")
    for name, batch, base in forms(buf, offs, tmp_path, "p"):
        for mode, rc_prob in MODES:
            kw = dict(rc=mode, rc_prob=rc_prob, seed=5, seq_index_base=base)
            ref = reference_revcomp(buf, offs, mode, 0.5 if rc_prob is None else rc_prob, 5, base)[:2]
            got = batch_tokenize_revcomp(tok, batch, P, "B", **kw)
            torch.cuda.synchronize()
            assert_same_bits(orc.batch_tokenize(ref, padlen=P, destchar="B", batch_first=True), got.cpu().numpy())
            got = batch_tokenize_revcomp(tok, batch, P, "i", batch_first=False, **kw)
            torch.cuda.synchronize()
            assert_same_bits(orc.batch_tokenize(ref, padlen=P, destchar="i", batch_first=False), got.cpu().numpy())
            assert torch.equal(batch_onehot_encode_bcl(tok, batch, P, "f", **kw), batch_onehot_encode_bcl(tok, cuda(*ref), P, "f"))
            assert torch.equal(batch_embed(tok, batch, weight, P, **kw), batch_embed(tok, cuda(*ref), weight, P))
            if mode != "both":
                got = batch_tokenize_mlm(tok, batch, P, "l", **kw)
                want = batch_tokenize_mlm(tok, cuda(*ref), P, "l", seed=5, seq_index_base=base)
                assert torch.equal(got.inputs, want.inputs) and torch.equal(got.labels, want.labels)
            for varlen in (False, True):
                got = batch_tokenize_kmer(tok, batch, 3, None if varlen else P, stride=2, tail="single", varlen=varlen, **kw)
                want = batch_tokenize_kmer(tok, cuda(*ref), 3, None if varlen else P, stride=2, tail="single", varlen=varlen)
                if varlen:
                    assert torch.equal(got.tokens, want.tokens) and torch.equal(got.cu_seqlens, want.cu_seqlens)
                    assert got.max_seqlen == want.max_seqlen
                else:
                    assert torch.equal(got, want)
        # a row longer than padlen still raises after the flip
        with pytest.raises((ValueError, RuntimeError)):
            batch_tokenize_revcomp(tok, batch, int(np.diff(offs).max()) + k - 1, rc="always")


@pytest.mark.parametrize("flags", [(True, True, True), (False, False, False)])
def test_varlen_seqpack_and_crop_order(flags, tmp_path):
    bos, eos, pad = flags
    tok = cbioseq.Tokenizer("DNA", bos=bos, eos=eos, padchar=pad)
    orc = OracleTokenizer("DNA", bos=bos, eos=eos, padchar=pad)
    k = int(bos) + int(eos)
    buf, offs = gen(12, 900, 0, 400, DNA)
    W, L = 150, 256
    for name, batch, base in forms(buf, offs, tmp_path, "v"):
        for mode, rc_prob in MODES:
            kw = dict(rc=mode, rc_prob=rc_prob, seed=6, seq_index_base=base)
            p = 0.5 if rc_prob is None else rc_prob
            ref = cuda(*reference_revcomp(buf, offs, mode, p, 6, base)[:2])
            got = batch_tokenize_varlen(tok, batch, "l", **kw)
            want = batch_tokenize_varlen(tok, ref, "l")
            assert torch.equal(got.tokens, want.tokens) and torch.equal(got.cu_seqlens, want.cu_seqlens)
            assert got.max_seqlen == want.max_seqlen
            # crop first, then flip: the flipped window of the crop drawn with the same seed
            cb, co, _ = reference_crop(buf, offs, W, True, 6, base)
            cref = reference_revcomp(cb, co, mode, p, 6, base)[:2]
            got = batch_tokenize_cropped(tok, batch, W + k, crop_len=W, **kw)
            torch.cuda.synchronize()
            assert_same_bits(orc.batch_tokenize(cref, padlen=W + k, destchar="B", batch_first=True), got.cpu().numpy())
            got = batch_tokenize_varlen(tok, batch, "B", crop="random", crop_len=W, **kw)
            want = batch_tokenize_varlen(tok, cuda(*cref), "B")
            assert torch.equal(got.tokens, want.tokens) and torch.equal(got.cu_seqlens, want.cu_seqlens)
            got = batch_tokenize_seqpack(tok, batch, L, crop="random", crop_len=W, **kw)
            want = batch_tokenize_seqpack(tok, cuda(*cref), L)
            for g_, w_ in zip(got[:5], want[:5]):
                assert (g_ == w_) if isinstance(g_, int) else torch.equal(g_, w_)
            if mode != "both":
                # MLM positions are positions in the flipped window
                got = batch_tokenize_mlm(tok, batch, varlen=True, crop="random", crop_len=W, **kw)
                want = batch_tokenize_mlm(tok, cuda(*cref), varlen=True, seed=6, seq_index_base=base)
                assert torch.equal(got.inputs.tokens, want.inputs.tokens) and torch.equal(got.labels, want.labels)
                got = batch_tokenize_seqpack(tok, batch, L, crop="random", crop_len=W, mlm=True, **kw)
                want = batch_tokenize_seqpack(tok, cuda(*cref), L, mlm=True, seed=6, seq_index_base=base)
                assert torch.equal(got.tokens, want.tokens) and torch.equal(got.labels, want.labels)
                assert torch.equal(got.starts, want.starts)


def test_both_layout_and_flipped():
    tok = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
    seqs = ["ACGTN", "GATTACA", "", "acgRYkmBDHVswn-*"]
    rb = revcomp_packed(*cuda(*consumers_pack(seqs)), rc="both")
    torch.cuda.synchronize()
    o = rb.offsets.tolist()
    out = [rb.bytes[o[i]:o[i + 1]].cpu().numpy().tobytes().decode() for i in range(8)]
    assert out == seqs + ["NACGT", "TGTAATC", "", "*-nwsBDHVkmRYcgt"]
    assert rb.flipped.tolist() == [False] * 4 + [True] * 4
    t = batch_tokenize_revcomp(tok, seqs, 32, rc="both")
    assert t.shape == (8, 32) and torch.equal(t[:4], tok.batch_tokenize(seqs, padlen=32, batch_first=True))
    assert torch.equal(t[4:], tok.batch_tokenize(out[4:], padlen=32, batch_first=True))


def consumers_pack(seqs):
    enc = [s.encode() for s in seqs]
    offs = np.zeros(len(enc) + 1, np.int64)
    np.cumsum([len(s) for s in enc], out=offs[1:])
    return np.frombuffer(b"".join(enc) or b"\0", np.uint8)[:int(offs[-1])].copy(), offs


def test_bad_offsets_are_rejected():
    buf, offs = gen(3, 500, 0, 300, DNA)
    b, o = cuda(buf, offs)
    bad = o.clone()
    bad[10] = bad[11] + 1
    tok = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
    for call in (lambda: revcomp_packed(b, bad), lambda: revcomp_packed(b[:-1], o),
                 lambda: batch_tokenize_revcomp(tok, (b, bad), 512), lambda: batch_tokenize_varlen(tok, (b, bad), rc="both"),
                 lambda: batch_tokenize_kmer(tok, (b, bad), 3, 512, rc="always")):
        with pytest.raises(ValueError):
            call()


# ------------------------------------------------------------------------------------------------------------------
def test_dataset_draws_anew_and_reproducibly(tmp_path):
    tok = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
    rng = np.random.default_rng(77)
    lens = rng.integers(1, 300, size=1200)
    table = np.frombuffer(b"ACGT", np.uint8)
    seqs = [table[rng.integers(0, 4, size=int(n))].tobytes() for n in lens]
    path = tmp_path / "dna.ff"
    path.write_bytes(flatfile_image(seqs))
    ff = cbioseq.FlatFile(str(path))
    L = 128

    def seed_of(draw, base=13):
        return (base & 0xFFFFFFFF) | (draw << 32)

    ds = FlatFileDataset(ff, tok, max_seq_len=L, rc="random")
    a, b = ds[0:1200], ds[0:1200]
    assert a.shape == (1200, L) and not torch.equal(a, b)
    assert torch.equal(a, batch_tokenize_cropped(tok, (ff, 0, 1200), L, seed=seed_of(1), rc="random").to(torch.long))
    assert torch.equal(b, batch_tokenize_cropped(tok, (ff, 0, 1200), L, seed=seed_of(2), rc="random").to(torch.long))
    assert torch.equal(FlatFileDataset(ff, tok, max_seq_len=L, rc="random")[0:1200], a)
    # a single index is that sequence's row of a slice fetched with the same draw
    one = FlatFileDataset(ff, tok, max_seq_len=L, rc="random")[7]
    assert torch.equal(one, batch_tokenize_cropped(tok, (ff, 7, 8), L, seed=seed_of(1), seq_index_base=7, rc="random")[0].to(torch.long))
    item, raw = ds.fetch(5, return_items=True)
    assert bytes(raw) == seqs[5]  # the stored, unflipped item
    # without a crop, and in every other output form
    ds = FlatFileDataset(ff, tok, rc="random", rc_prob=0.3)
    got = ds[0:1200]
    want = batch_tokenize_revcomp(tok, (ff, 0, 1200), ff.maxseqlen + 2, rc_prob=0.3, seed=seed_of(1)).to(torch.long)
    assert torch.equal(got, want)
    vb = FlatFileDataset(ff, tok, varlen=True, rc="random")[0:1200]
    want = batch_tokenize_varlen(tok, (ff, 0, 1200), "l", rc="random", seed=seed_of(1))
    assert torch.equal(vb.tokens, want.tokens)
    mb = FlatFileDataset(ff, tok, max_seq_len=L, mlm=True, rc="random")[0:1200]
    want = batch_tokenize_mlm(tok, (ff, 0, 1200), L, "l", crop="random", rc="random", seed=seed_of(1),
                              mask_token=tok.alphabet_size())
    assert torch.equal(mb.inputs, want.inputs) and torch.equal(mb.labels, want.labels)
    sp = FlatFileDataset(ff, tok, max_seq_len=L, seqpack=True, rc="random")[0:1200]
    want = batch_tokenize_seqpack(tok, (ff, 0, 1200), L, "l", crop="random", rc="random", seed=seed_of(1))
    assert torch.equal(sp.tokens, want.tokens)
    cnn = FlatFileDataset(ff, tok, max_seq_len=L, cnn=True, rc="random")
    got = cnn[0:64]
    want = batch_onehot_encode_bcl(tok, (ff, 0, 64), L, "f", crop="random", rc="random", seed=seed_of(1))
    assert torch.equal(got, want)
    assert cnn[3].shape == (L, tok.alphabet_size())
