"""Sequence packing (batch_tokenize_seqpack / bsq_tokenize_seqpack, kernel K10), bit for bit against the rule of
include/bsq.h: the plan of tests/seqpack_reference.py filled with the rows of batch_tokenize_varlen (itself checked
against the oracle elsewhere, and here against the oracle's padded rows too), the padding value and position ids that
restart per segment.

K10 runs one warp per row: 16-element chunks of the flat output, 16-byte stores of residues realigned from the source,
pattern-filled padding, computed position ids, element stores at segment edges.  The cases cover all six element kinds
and eight bos/eos/padchar combinations, every source alignment with offsets[0] != 0, row widths whose bytes are not a
multiple of 16, a 16 384-wide row, empty batches and sequences, spare rows, MLM, crop and augmentation, every batch
form, a side stream, back-to-back launches, a CUDA graph captured through the C ABI, and the dataset."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from bioseq_b200 import capi, cbioseq, consumers, batch_tokenize_seqpack, SeqPackBatch  # noqa: E402
from bioseq_b200 import batch_tokenize_varlen, batch_tokenize_mlm  # noqa: E402
from bioseq_b200.loaders import FlatFileDataset  # noqa: E402
from oracle.oracle import OracleTokenizer, flatfile_image  # noqa: E402
from helpers import gen  # noqa: E402
from crop_reference import crop as reference_crop  # noqa: E402
from seqpack_reference import plan as reference_plan, pack as reference_pack  # noqa: E402

AA = b"ACDEFGHIKLMNPQRSTVWY"
MIX = b"ACDEFGHIKLMNPQRSTVWYacdefghiklmnpqrstvwyXBZOUJ*-NnUu .\x00\x7f\x80\xc3\xff"
FLAGS = [(b, e, p) for b in (False, True) for e in (False, True) for p in (False, True)]
KINDS = ("B", "b", "h", "i", "l", "f", "d")


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests selected but no CUDA device is visible")


def cuda(buf, offs):
    return torch.from_numpy(np.ascontiguousarray(buf)).cuda(), torch.from_numpy(np.ascontiguousarray(offs)).cuda()


def batch_of(lens, seed, alphabet=MIX, lead=0):
    offs = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    rng = np.random.default_rng(seed)
    table = np.frombuffer(alphabet, np.uint8)
    buf = table[rng.integers(0, table.size, size=int(offs[-1]) + lead)]
    return buf, offs + lead


def pad_value(tok):
    return tok.pad() if tok.is_padded() else 0


def expect(tok, batch, L, destchar, lens, rows=None, **kw):
    """(plan, tokens, position_ids) the rule gives: the reference plan of the (cropped) lengths, filled with the rows of
    batch_tokenize_varlen on the same batch and arguments."""
    k = int(tok.includes_bos()) + int(tok.includes_eos())
    vb = batch_tokenize_varlen(tok, batch, destchar, **kw)
    cu = vb.cu_seqlens.cpu().numpy()
    flat = vb.tokens.cpu().numpy()
    seq_rows = [flat[cu[i]:cu[i + 1]] for i in range(cu.size - 1)]
    p = reference_plan(np.diff(cu) - k, k, L, rows)
    tokens, pos = reference_pack(p, seq_rows, L, pad_value(tok), flat.dtype)
    return p, tokens, pos, seq_rows


def check(sb, p, tokens, pos):
    torch.cuda.synchronize()
    assert isinstance(sb, SeqPackBatch)
    assert sb.tokens.shape == tokens.shape and sb.position_ids.dtype == torch.int32
    assert np.array_equal(sb.starts.cpu().numpy(), p["starts"])
    assert np.array_equal(sb.cu_seqlens.cpu().numpy(), p["cu_seqlens"])
    assert sb.max_seqlen == p["max_seqlen"]
    got = sb.tokens.cpu().numpy()
    assert got.tobytes() == tokens.tobytes(), np.flatnonzero(got.reshape(-1) != tokens.reshape(-1))[:8]
    assert np.array_equal(sb.position_ids.cpu().numpy(), pos)


@pytest.mark.parametrize("flags", FLAGS)
def test_every_kind_and_flag_combination(flags):
    bos, eos, pad = flags
    tok = cbioseq.Tokenizer("PROTEIN", bos=bos, eos=eos, padchar=pad)
    orc = OracleTokenizer("PROTEIN", bos=bos, eos=eos, padchar=pad)
    k = int(bos) + int(eos)
    L = 128
    lens = np.random.default_rng(sum(flags)).integers(0, L - k + 1, size=700)
    lens[:4] = [0, L - k, 1, 17]
    buf, offs = batch_of(lens, 3, lead=5)
    d = cuda(buf, offs)
    padded = orc.batch_tokenize((buf, offs), padlen=L, destchar="B", batch_first=True)
    for destchar in KINDS:
        p, tokens, pos, seq_rows = expect(tok, d, L, destchar, lens)
        sb = batch_tokenize_seqpack(tok, d, L, destchar)
        check(sb, p, tokens, pos)
        if destchar == "B":  # the oracle's padded rows, cut to the sequence
            flat = sb.tokens.view(-1).cpu().numpy()
            for i in range(0, lens.size, 7):
                s = p["starts"][i]
                if s >= 0:
                    assert np.array_equal(flat[s:s + lens[i] + k], padded[i, :lens[i] + k])


@pytest.mark.parametrize("shift", range(16))
def test_every_source_alignment(shift):
    tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    lens = np.random.default_rng(100 + shift).integers(0, 300, size=900)
    buf, offs = batch_of(lens, shift, lead=shift)
    d = cuda(buf, offs)
    for destchar in ("B", "l"):
        p, tokens, pos, _ = expect(tok, d, 512, destchar, lens)
        check(batch_tokenize_seqpack(tok, d, 512, destchar), p, tokens, pos)


@pytest.mark.parametrize("L", [1, 3, 37, 1021, 1023, 16384])
def test_row_widths(L):
    # byte widths that are not a multiple of 16 (rows start at every alignment), and a wide row
    for flags in ((True, True, False), (False, False, True)):
        tok = cbioseq.Tokenizer("DNA", bos=flags[0], eos=flags[1], padchar=flags[2])
        k = int(flags[0]) + int(flags[1])
        if L <= k:
            continue
        n = 3000 if L < 16384 else 400
        lens = np.random.default_rng(L).integers(0, min(L - k, 3000) + 1, size=n)
        buf, offs = batch_of(lens, L, alphabet=b"ACGTNacgtn")
        d = cuda(buf, offs)
        for destchar in ("B", "h", "f"):
            p, tokens, pos, _ = expect(tok, d, L, destchar, lens)
            check(batch_tokenize_seqpack(tok, d, L, destchar), p, tokens, pos)


def test_empty_batches_empty_sequences_and_spare_rows():
    for flags in ((True, True, True), (False, False, False)):
        tok = cbioseq.Tokenizer("PROTEIN", bos=flags[0], eos=flags[1], padchar=flags[2])
        e = cuda(np.zeros(0, np.uint8), np.zeros(1, np.int64))
        sb = batch_tokenize_seqpack(tok, e, 64)
        assert sb.tokens.shape == (0, 64) and sb.cu_seqlens.tolist() == [0] and sb.max_seqlen == 0 and sb.starts.numel() == 0
        sb = batch_tokenize_seqpack(tok, e, 64, rows=3)
        torch.cuda.synchronize()
        assert sb.tokens.shape == (3, 64) and (sb.tokens == pad_value(tok)).all()
        assert sb.cu_seqlens.tolist() == [0, 64, 128, 192] and sb.position_ids[1].tolist() == list(range(64))
        for lens in ([0, 0, 0], [0, 5, 0, 0, 9, 0]):
            buf, offs = batch_of(lens, 1)
            for batch in (cuda(buf, offs), (buf, offs)):
                for rows in (None, 4):
                    p, tokens, pos, _ = expect(tok, batch, 16, "B", lens, rows)
                    check(batch_tokenize_seqpack(tok, batch, 16, rows=rows), p, tokens, pos)
        with pytest.raises(ValueError):
            batch_tokenize_seqpack(tok, cuda(*batch_of([60] * 5, 2)), 64, rows=2)


def test_mlm_matches_varlen_mlm_per_sequence():
    for flags in ((True, True, True), (False, True, False), (False, False, False)):
        tok = cbioseq.Tokenizer("PROTEIN", bos=flags[0], eos=flags[1], padchar=flags[2])
        k = int(flags[0]) + int(flags[1])
        L = 256
        lens = np.random.default_rng(7).integers(0, L - k + 1, size=1500)
        buf, offs = batch_of(lens, 8, alphabet=AA + b"xz")
        for batch in (cuda(buf, offs), (buf, offs)):
            for destchar in ("B", "i", "l", "d"):
                kw = dict(maskfrac=0.3, mask_token=30, ignore_index=-7, seed=99, seq_index_base=1000)
                sb = batch_tokenize_seqpack(tok, batch, L, destchar, mlm=True, **kw)
                mb = batch_tokenize_mlm(tok, batch, destchar=destchar, varlen=True, **kw)
                cu = mb.inputs.cu_seqlens.cpu().numpy()
                p = reference_plan(np.diff(cu) - k, k, L)
                inp = mb.inputs.tokens.cpu().numpy()
                lab = mb.labels.cpu().numpy()
                rows_i = [inp[cu[i]:cu[i + 1]] for i in range(cu.size - 1)]
                rows_l = [lab[cu[i]:cu[i + 1]] for i in range(cu.size - 1)]
                tokens, pos, labels = reference_pack(p, rows_i, L, pad_value(tok), inp.dtype, -7, rows_l)
                check(sb, p, tokens, pos)
                assert sb.labels.dtype == torch.int64 and np.array_equal(sb.labels.cpu().numpy(), labels)
                assert (sb.labels != -7).any()


def test_crop_and_augment_match_varlen():
    tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    buf, offs = gen(21, 2000, 0, 3000, AA)
    L = 1024
    for batch in (cuda(buf, offs), (buf, offs)):
        for mode in ("head", "random"):
            kw = dict(crop=mode, crop_len=L - 2, seed=4, seq_index_base=9)
            lens = np.minimum(np.diff(offs), L - 2)
            p, tokens, pos, _ = expect(tok, batch, L, "B", lens, **kw)
            check(batch_tokenize_seqpack(tok, batch, L, crop=mode, seed=4, seq_index_base=9), p, tokens, pos)
            # augmentation after the crop: the packed sequences are the cropped, mutated ones
            sb = batch_tokenize_seqpack(tok, batch, L, crop=mode, crop_len=300, augment=2, augment_frac=0.7, seed=4)
            cb, co, _ = reference_crop(buf, offs, 300, mode == "random", 4, 0)
            mut = cuda(cb, co)
            consumers.augment_packed(mut[0], mut[1], 2, 0.7, 4, 0)
            p, tokens, pos, _ = expect(tok, mut, L, "B", np.diff(co))
            check(sb, p, tokens, pos)


def test_batch_forms(tmp_path):
    tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=False, padchar=True)
    buf, offs = gen(5, 800, 0, 400, AA + b"*x")
    seqs = [buf[offs[i]:offs[i + 1]].tobytes() for i in range(offs.size - 1)]
    path = tmp_path / "f.ff"
    path.write_bytes(flatfile_image([b"MKV"] + seqs))
    ff = cbioseq.FlatFile(str(path))
    L = 700
    p, tokens, pos, _ = expect(tok, cuda(buf, offs), L, "i", np.diff(offs))
    forms = [seqs, (buf, offs), (torch.from_numpy(buf).pin_memory(), torch.from_numpy(offs).pin_memory()),
             (torch.from_numpy(buf), torch.from_numpy(offs)), cuda(buf, offs), (ff, 1, 1 + len(seqs))]
    for batch in forms:
        check(batch_tokenize_seqpack(tok, batch, L, "i"), p, tokens, pos)


def test_side_stream_back_to_back_and_graph():
    tok_py = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    tok = consumers.descriptor(tok_py)
    lens = np.random.default_rng(5).integers(1, 1000, size=3000)
    buf_a, offs = batch_of(lens, 50, alphabet=AA)
    buf_b, _ = batch_of(lens, 51, alphabet=AA)
    L = 1024
    da, db = cuda(buf_a, offs), cuda(buf_b, offs)
    want = {name: expect(tok_py, d, L, "B", lens) for name, d in (("a", da), ("b", db))}
    # a side stream, back to back
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        outs = [batch_tokenize_seqpack(tok_py, da if i % 2 == 0 else db, L) for i in range(6)]
    s.synchronize()
    for i, sb in enumerate(outs):
        check(sb, *want["a" if i % 2 == 0 else "b"][:3])
    # a CUDA graph captured through the C ABI with a precomputed plan, replayed bit-exact
    p = want["a"][0]
    R, n = p["R"], lens.size
    d_row_ptr = torch.from_numpy(p["row_ptr"]).cuda()
    d_row_seq = torch.from_numpy(p["row_seq"]).cuda()
    out = torch.zeros((R, L), dtype=torch.uint8, device="cuda")
    posd = torch.zeros((R, L), dtype=torch.int32, device="cuda")
    lab = torch.zeros((R, L), dtype=torch.int64, device="cuda")
    mlm = consumers._mlm_desc(tok, "B", 0.15, 0.8, 0.1, None, -100, 3, 0)
    mb = batch_tokenize_seqpack(tok_py, db, L, mlm=True, seed=3)

    def launch(st, d, with_mlm):
        if with_mlm:
            capi.tokenize_seqpack_mlm(0, st, d[0], d[1], tok, capi.I8, mlm, L, R, d_row_ptr, d_row_seq, out, posd, lab)
        else:
            capi.tokenize_seqpack(0, st, d[0], d[1], tok, capi.I8, L, R, d_row_ptr, d_row_seq, out, posd)

    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch(torch.cuda.current_stream().cuda_stream, da, False)
        launch(torch.cuda.current_stream().cuda_stream, db, False)
    for _ in range(2):
        out.zero_()
        posd.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), want["b"][1]) and np.array_equal(posd.cpu().numpy(), want["b"][2])
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2):
        launch(torch.cuda.current_stream().cuda_stream, db, True)
    lab.zero_()
    g2.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, mb.tokens) and torch.equal(lab, mb.labels) and torch.equal(posd, mb.position_ids)


def test_dataset(tmp_path):
    tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    rng = np.random.default_rng(77)
    lens = rng.integers(0, 400, size=1200)
    lens[[3, 500]] = [5000, 1023]
    table = np.frombuffer(AA, np.uint8)
    seqs = [table[rng.integers(0, 20, size=int(n))].tobytes() for n in lens]
    path = tmp_path / "ds.ff"
    path.write_bytes(flatfile_image(seqs))
    ff = cbioseq.FlatFile(str(path))
    L = 1024

    def seed_of(draw, base=13):
        return (base & 0xFFFFFFFF) | (draw << 32)

    ds = FlatFileDataset(ff, tok, max_seq_len=L, seqpack=True, crop="head")
    sb = ds[0:600]
    assert isinstance(sb, SeqPackBatch) and sb.tokens.dtype == torch.long and sb.labels is None
    want = batch_tokenize_seqpack(tok, (ff, 0, 600), L, "l", crop="head", seed=seed_of(1))
    assert torch.equal(sb.tokens, want.tokens) and torch.equal(sb.position_ids, want.position_ids)
    one = ds[3]
    assert one.tokens.shape == (1, L) and one.starts.tolist() == [0]
    assert one.cu_seqlens.tolist() == [0, L] and one.max_seqlen == L  # the 5000-residue sequence cropped to fill the row
    ds = FlatFileDataset(ff, tok, max_seq_len=L, seqpack=True, mlm=True)
    a = ds[0:600]
    want = batch_tokenize_seqpack(tok, (ff, 0, 600), L, "l", mlm=True, mask_token=tok.alphabet_size(), crop="random",
                                  seed=seed_of(1))
    assert torch.equal(a.tokens, want.tokens) and torch.equal(a.labels, want.labels)
    assert not torch.equal(a.labels, ds[0:600].labels)  # a new draw every fetch
    # max_seq_len through batches(prefetch=2): every batch ready on the caller's stream
    ds = FlatFileDataset(ff, tok, max_seq_len=L, seqpack=True, mlm=True, crop="head")
    got = list(ds.batches(300, prefetch=2))
    assert len(got) == 4
    for j, b in enumerate(got):
        want = batch_tokenize_seqpack(tok, (ff, 300 * j, 300 * j + 300), L, "l", mlm=True, mask_token=tok.alphabet_size(),
                                      crop="head", seed=seed_of(j + 1), seq_index_base=300 * j)
        assert torch.equal(b.tokens, want.tokens) and torch.equal(b.labels, want.labels)
        assert torch.equal(b.cu_seqlens, want.cu_seqlens) and b.max_seqlen == want.max_seqlen
