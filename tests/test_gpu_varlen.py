"""Padding-free tokens (batch_tokenize_varlen / bsq_tokenize_varlen, kernel K1v), bit for bit against the oracle's padded
batch-first tokens cut to len + bos + eos per row and concatenated.

K1v deals output tiles of 16384 elements round-robin to a persistent grid of SMs x 4 CTAs (k = bos + eos >= 1); k = 0
is a row-free byte map.  The cases cover every flag combination and element kind, rows that are shorter than a 16-byte
vector (several rows per vector and up to thousands per tile), a sequence longer than several tiles, every source
alignment, the schedule's round edges, back-to-back launches, a replayed CUDA graph, concurrent streams, every batch
form, and the errors."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import bioseq_b200  # noqa: E402
from bioseq_b200 import capi, cbioseq, batch_tokenize_varlen, VarlenBatch  # noqa: E402
from bioseq_b200.loaders import FlatFileDataset  # noqa: E402
from oracle.oracle import OracleTokenizer, flatfile_image  # noqa: E402
from helpers import assert_same_bits, gen  # noqa: E402
from test_varlen_host import oracle_varlen  # noqa: E402

MIX = b"ACDEFGHIKLMNPQRSTVWYacdefghiklmnpqrstvwyXBZOUJ*-NnUu .\x00\x7f\x80\xc3\xff"
FLAGS = [(b, e, p) for b in (False, True) for e in (False, True) for p in (False, True)]
DESTCHARS = ["B", "b", "h", "i", "l", "f", "d"]
TILE = 16384
CTAS_PER_SM = 4


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests selected but no CUDA device is visible")


def toks(key, flags):
    bos, eos, pad = flags
    return cbioseq.Tokenizer(key, bos=bos, eos=eos, padchar=pad), OracleTokenizer(key, bos=bos, eos=eos, padchar=pad)


def cuda(buf, offs):
    return torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda()


def check(vb, orc, buf, offs, destchar="B"):
    assert isinstance(vb, VarlenBatch)
    want_t, want_cu = oracle_varlen(orc, buf, offs, destchar)
    k = int(orc.bos() >= 0) + int(orc.eos() >= 0)
    lens = np.diff(offs)
    torch.cuda.synchronize()
    assert vb.tokens.dim() == 1 and vb.cu_seqlens.dtype == torch.int32
    assert_same_bits(want_t, vb.tokens.cpu().numpy())
    assert_same_bits(want_cu, vb.cu_seqlens.cpu().numpy())
    assert vb.max_seqlen == (int(lens.max()) + k if lens.size else 0)


@pytest.mark.parametrize("key", ["PROTEIN", "DNA", "BYTES"])
@pytest.mark.parametrize("destchar", DESTCHARS)
@pytest.mark.parametrize("flags", FLAGS)
def test_flags_and_kinds(key, destchar, flags):
    tok, orc = toks(key, flags)
    buf, offs = gen(1000 * DESTCHARS.index(destchar) + 10 * FLAGS.index(flags) + len(key), 3000, 0, 300, MIX)
    check(batch_tokenize_varlen(tok, cuda(buf, offs), destchar), orc, buf, offs, destchar)


def test_empty_batch():
    tok, orc = toks("PROTEIN", (True, True, True))
    buf, offs = np.zeros(0, np.uint8), np.zeros(1, np.int64)
    for batch in ((buf, offs), cuda(buf, offs), []):
        vb = batch_tokenize_varlen(tok, batch)
        torch.cuda.synchronize()
        assert tuple(vb.tokens.shape) == (0,) and vb.cu_seqlens.cpu().tolist() == [0] and vb.max_seqlen == 0


@pytest.mark.parametrize("flags", [(False, False, True), (True, False, False), (False, True, True), (True, True, False)])
@pytest.mark.parametrize("n", [1, 17, 5000, 40000])
def test_all_empty_sequences(flags, n):
    # k = 0: T = 0; k = 1, 2: every row is only its specials (up to 16 rows per vector, 8192 per tile: over-full tiles)
    tok, orc = toks("DNA", flags)
    buf, offs = np.zeros(0, np.uint8), np.zeros(n + 1, np.int64)
    for batch in ((buf, offs), cuda(buf, offs)):
        check(batch_tokenize_varlen(tok, batch), orc, buf, offs)


@pytest.mark.parametrize("destchar", ["B", "i"])
@pytest.mark.parametrize("flags", [(True, True, True), (False, True, False), (True, False, True), (False, False, False)])
def test_short_rows(flags, destchar):
    # lengths 0..40: many rows per vector and per tile, tiles with and without room in the row table
    tok, orc = toks("PROTEIN", flags)
    for seed, n, hi in ((1, 20000, 40), (2, 300000, 8), (3, 50000, 3)):
        buf, offs = gen(seed, n, 0, hi, MIX)
        check(batch_tokenize_varlen(tok, cuda(buf, offs), destchar), orc, buf, offs, destchar)


@pytest.mark.parametrize("flags", [(True, True, True), (False, False, False), (False, True, False)])
def test_sequence_longer_than_several_tiles(flags):
    tok, orc = toks("PROTEIN", flags)
    parts = [gen(s, 1, n, n, MIX)[0] for s, n in ((4, 5), (5, 5 * TILE + 123), (6, 0), (7, 3 * TILE), (8, 9))]
    buf = np.concatenate(parts)
    offs = np.zeros(len(parts) + 1, np.int64)
    np.cumsum([p.size for p in parts], out=offs[1:])
    for destchar in ("B", "l"):
        check(batch_tokenize_varlen(tok, cuda(buf, offs), destchar), orc, buf, offs, destchar)


@pytest.mark.parametrize("flags", [(True, True, True), (False, False, False), (True, False, False)])
@pytest.mark.parametrize("shift", range(16))
def test_source_alignment(flags, shift):
    # offsets[0] = shift (mod 16): the packed residues start anywhere in a 16-byte word
    tok, orc = toks("PROTEIN", flags)
    buf, offs = gen(100 + shift, 4000, 0, 700, MIX)
    buf = np.concatenate([np.full(shift + 32, ord("W"), np.uint8), buf])
    offs = offs + shift + 32
    check(batch_tokenize_varlen(tok, cuda(buf, offs)), orc, buf, offs)
    check(batch_tokenize_varlen(tok, (buf, offs), "h"), orc, buf, offs, "h")


def grid():
    return torch.cuda.get_device_properties(0).multi_processor_count * CTAS_PER_SM


@pytest.mark.parametrize("case", ["fewer_tiles_than_ctas", "one_round", "one_round_plus_one", "two_rounds_plus_one",
                                  "ragged_past_two_rounds"])
def test_round_edges(case):
    tok, orc = toks("PROTEIN", (True, True, True))  # k = 2: rows of 1022 residues are 1024 tokens
    per_round = grid() * TILE // 1024
    n = {"fewer_tiles_than_ctas": 100, "one_round": per_round, "one_round_plus_one": per_round + 1,
         "two_rounds_plus_one": 2 * per_round + 1}.get(case)
    if n is None:
        buf, offs = gen(77, 2 * per_round * 2 + 999, 0, 1022, MIX)
    else:
        buf, offs = gen(78, n, 1022, 1022, MIX)
    check(batch_tokenize_varlen(tok, cuda(buf, offs)), orc, buf, offs)


def _launch(st, tok, d_b, d_o, n, out, cu):
    capi.tokenize_varlen(0, st, d_b, d_o, n, tok, capi.I8, out, cu)


def _same_shape_pair(seed, n):
    # two batches with the same offsets and different residues
    buf_a, offs = gen(seed, n, 50, 1022, MIX)
    buf_b = gen(seed + 1, 1, buf_a.size, buf_a.size, MIX)[0]
    return (buf_a, offs), (buf_b, offs)


@pytest.mark.parametrize("flags", [(True, True, True), (False, False, False)])
def test_back_to_back_launches_into_one_buffer(flags):
    tok_py, orc = toks("PROTEIN", flags)
    tok = consumers_desc(tok_py)
    a, b = _same_shape_pair(90, 30000)
    want_a, want_cu = oracle_varlen(orc, *a)
    want_b, _ = oracle_varlen(orc, *b)
    da, db = cuda(*a), cuda(*b)
    n = a[1].size - 1
    out = torch.zeros(want_a.size, dtype=torch.uint8, device="cuda")
    cu = torch.zeros(n + 1, dtype=torch.int32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    for i in range(50):
        _launch(st, tok, *(da if i % 2 == 0 else db), n, out, cu)
    torch.cuda.synchronize()
    assert_same_bits(want_b, out.cpu().numpy())
    assert_same_bits(want_cu, cu.cpu().numpy())
    # inside a CUDA graph: 49 launches end on input a; replayed twice, each time followed by a direct launch of b
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(49):
            _launch(torch.cuda.current_stream().cuda_stream, tok, *(da if i % 2 == 0 else db), n, out, cu)
    for _ in range(2):
        out.zero_()
        cu.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert_same_bits(want_a, out.cpu().numpy())
        assert_same_bits(want_cu, cu.cpu().numpy())
        _launch(torch.cuda.current_stream().cuda_stream, tok, *db, n, out, cu)
        torch.cuda.synchronize()
        assert_same_bits(want_b, out.cpu().numpy())


def consumers_desc(tok):
    return bioseq_b200.consumers.descriptor(tok)


def test_concurrent_streams():
    streams = [torch.cuda.Stream() for _ in range(4)]
    work = []
    for s, flags in enumerate([(True, True, True), (False, False, False), (True, False, True), (False, True, False)]):
        tok_py, orc = toks("PROTEIN", flags)
        buf, offs = gen(200 + s, 20000 + 1000 * s, 0, 1022, MIX)
        want, want_cu = oracle_varlen(orc, buf, offs)
        outs = [(torch.zeros(want.size, dtype=torch.uint8, device="cuda"), torch.zeros(offs.size, dtype=torch.int32, device="cuda"))
                for _ in range(6)]
        work.append((consumers_desc(tok_py), cuda(buf, offs), offs.size - 1, want, want_cu, outs))
    torch.cuda.synchronize()
    for rep in range(6):
        for st, (tok, (d_b, d_o), n, _, _, outs) in zip(streams, work):
            _launch(st.cuda_stream, tok, d_b, d_o, n, *outs[rep])
    torch.cuda.synchronize()
    for _, _, _, want, want_cu, outs in work:
        for out, cu in outs:
            assert_same_bits(want, out.cpu().numpy())
            assert_same_bits(want_cu, cu.cpu().numpy())


def test_input_forms(tmp_path):
    tok, orc = toks("PROTEIN", (True, True, True))
    buf, offs = gen(300, 2000, 0, 900, MIX)
    seqs = [buf[offs[i]:offs[i + 1]].tobytes() for i in range(offs.size - 1)]
    check(batch_tokenize_varlen(tok, seqs), orc, buf, offs)                                          # list of bytes
    check(batch_tokenize_varlen(tok, [s.decode("latin-1") if max(s, default=0) < 0x80 else s for s in seqs]), orc, buf, offs)
    check(batch_tokenize_varlen(tok, [bytearray(s) for s in seqs]), orc, buf, offs)
    check(batch_tokenize_varlen(tok, (buf, offs)), orc, buf, offs)                                   # host numpy
    tb, to = torch.from_numpy(buf).pin_memory(), torch.from_numpy(offs).pin_memory()
    check(batch_tokenize_varlen(tok, (tb, to)), orc, buf, offs)                                      # pinned torch CPU
    check(batch_tokenize_varlen(tok, cuda(buf, offs)), orc, buf, offs)                               # CUDA tensors
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):                                                                    # non-default stream
        vb = batch_tokenize_varlen(tok, cuda(buf, offs))
        vh = batch_tokenize_varlen(tok, (buf, offs))
    side.synchronize()
    check(vb, orc, buf, offs)
    check(vh, orc, buf, offs)
    check(batch_tokenize_varlen(tok, (buf, offs), device="cuda:0"), orc, buf, offs)                 # device=
    check(batch_tokenize_varlen(tok, seqs, device=torch.device("cuda", 0)), orc, buf, offs)
    # a FlatFile range (offsets[0] != 0)
    ascii_seqs = [bytes(c if c < 0x80 and c not in (10, 13, 62, 64) else 65 for c in s) for s in seqs]
    path = tmp_path / "v.ff"
    path.write_bytes(flatfile_image(ascii_seqs))
    ff = cbioseq.FlatFile(str(path))
    fb, fo = ff.packed(0, len(ascii_seqs))
    fb, fo = np.asarray(fb), np.asarray(fo)
    lo, hi = 123, 1789
    sub_o = fo[lo:hi + 1]
    check(batch_tokenize_varlen(tok, (ff, lo, hi)), orc, fb, sub_o)


def test_decode_and_dataset(tmp_path):
    tok, orc = toks("PROTEIN", (True, True, True))
    buf, offs = gen(400, 3000, 0, 600, b"ACDEFGHIKLMNPQRSTVWY")
    vb = batch_tokenize_varlen(tok, cuda(buf, offs))
    want, _ = oracle_varlen(orc, buf, offs)
    cu = vb.cu_seqlens.cpu().numpy()
    for i in (0, 1, 17, 1500, 2999):
        row = vb.tokens[int(cu[i]):int(cu[i + 1])]
        assert tok.decode_tokens(row) == orc.decode_tokens(want[cu[i]:cu[i + 1]])
    seqs = [buf[offs[i]:offs[i + 1]].tobytes() for i in range(offs.size - 1)]
    path = tmp_path / "d.ff"
    path.write_bytes(flatfile_image(seqs))
    ff = cbioseq.FlatFile(str(path))
    ds = FlatFileDataset(ff, tok, varlen=True)
    part = ds[100:2100]
    ref = batch_tokenize_varlen(tok, (ff, 100, 2100), "l")
    torch.cuda.synchronize()
    assert part.tokens.dtype == torch.long and torch.equal(part.tokens, ref.tokens)
    assert torch.equal(part.cu_seqlens, ref.cu_seqlens) and part.max_seqlen == ref.max_seqlen
    one = ds[5]
    assert torch.equal(one, ref.tokens[:0].new_tensor(want[int(cu[5]):int(cu[6])].astype(np.int64)))
    for prefetch in (0, 2):
        got = list(ds.batches(700, prefetch=prefetch))
        assert len(got) == 5
        for j, vbj in enumerate(got):
            r = batch_tokenize_varlen(tok, (ff, 700 * j, min(700 * (j + 1), 3000)), "l")
            assert torch.equal(vbj.tokens, r.tokens) and torch.equal(vbj.cu_seqlens, r.cu_seqlens)
    with pytest.raises(ValueError):
        FlatFileDataset(ff, tok, varlen=True, cnn=True)


def test_errors():
    tok, _ = toks("PROTEIN", (True, True, True))
    buf, offs = gen(500, 100, 0, 50, MIX)
    with pytest.raises(ValueError, match="Unsupported dtype"):
        batch_tokenize_varlen(tok, (buf, offs), destchar="z")
    with pytest.raises(ValueError, match="item was none of"):
        batch_tokenize_varlen(tok, ["ACGT", 5])
    with pytest.raises(ValueError, match="past the end"):
        batch_tokenize_varlen(tok, (buf[:-1], offs))
    with pytest.raises(ValueError, match="past the end"):
        batch_tokenize_varlen(tok, cuda(buf[:-1], offs))
    bad = offs.copy()
    bad[50] = bad[51] + 1  # a negative length
    with pytest.raises(ValueError, match="non-decreasing"):
        batch_tokenize_varlen(tok, cuda(buf, bad))
    with pytest.raises(ValueError, match="non-decreasing"):
        batch_tokenize_varlen(tok, (buf, bad))
    # T = 2^31 tokens (one sequence of 2^31 - 2 residues + BOS + EOS): refused from the host offsets before any copy or
    # launch (the residues are a lazily zero-filled host buffer; nothing of that size reaches the device)
    big = np.zeros(2 ** 31 - 2, np.uint8)
    capi.lib().bsq_launch_count_reset()
    with pytest.raises(ValueError, match="2\\^31 - 1"):
        batch_tokenize_varlen(tok, (big, np.array([0, big.size], np.int64)))
    assert capi.lib().bsq_launch_count() == 0
    del big
