"""Masked-language-model batches (batch_tokenize_mlm / bsq_tokenize_mlm / bsq_tokenize_varlen_mlm, kernel K8), bit for
bit against the rule of include/bsq.h (tests/mlm_reference.py) applied to the oracle's padded batch-first tokens, and
for the padding-free form the same rows cut to len + bos + eos and concatenated.

The padded kernel takes 16 columns of one row per thread (vector stores when a row's bytes are a multiple of 16,
scalar stores otherwise); the padding-free kernel takes 16 elements of the packed stream per thread, with a vector
path for 16 residues of one row and an element-by-element path for row boundaries.  The cases cover every flag
combination and element kind, both forms, aligned and unaligned padlen, every source alignment, empty batches and
rows, a sequence longer than many blocks, every batch form, augmentation, back-to-back launches, a replayed CUDA graph,
concurrent streams, the dataset and the errors."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import bioseq_b200  # noqa: E402
from bioseq_b200 import capi, cbioseq, consumers, batch_tokenize_mlm, batch_tokenize_varlen, MLMBatch, VarlenBatch  # noqa: E402
from bioseq_b200.loaders import FlatFileDataset  # noqa: E402
from oracle import oracle  # noqa: E402
from oracle.oracle import OracleTokenizer, flatfile_image  # noqa: E402
from helpers import assert_same_bits, gen  # noqa: E402
from mlm_reference import mlm as reference_mlm  # noqa: E402

MIX = b"ACDEFGHIKLMNPQRSTVWYacdefghiklmnpqrstvwyXBZOUJ*-NnUu .\x00\x7f\x80\xc3\xff"
FLAGS = [(b, e, p) for b in (False, True) for e in (False, True) for p in (False, True)]
DESTCHARS = ["B", "b", "h", "i", "l", "f", "d"]
TH = consumers._mlm_thresholds(0.3, 0.6, 0.3)  # a large random share: both Philox streams are exercised


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests selected but no CUDA device is visible")


def toks(key, flags):
    bos, eos, pad = flags
    return cbioseq.Tokenizer(key, bos=bos, eos=eos, padchar=pad), OracleTokenizer(key, bos=bos, eos=eos, padchar=pad)


def cuda(buf, offs):
    return torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda()


def default_mask_token(tok, destchar):
    return tok.alphabet_size() if tok.alphabet_size() <= consumers._mask_token_limit(destchar) else 7


def want_padded(orc, buf, offs, padlen, destchar, mask_token, seed=0, base=0, th=TH, ignore=-100):
    t = orc.batch_tokenize((buf, offs), padlen=padlen, destchar=destchar, batch_first=True)
    return reference_mlm(t, offs, int(orc.bos() >= 0), orc.nchars(), th, mask_token, ignore, seed, base)


def cut(orc, offs, a):
    k = int(orc.bos() >= 0) + int(orc.eos() >= 0)
    lens = np.diff(offs)
    rows = [a[i, :int(lens[i]) + k] for i in range(lens.size)]
    return np.concatenate(rows) if rows else a.reshape(-1)[:0]


def want_varlen(orc, buf, offs, destchar, mask_token, seed=0, base=0, th=TH, ignore=-100):
    k = int(orc.bos() >= 0) + int(orc.eos() >= 0)
    lens = np.diff(offs)
    padlen = max(int(lens.max()) + k if lens.size else 1, 1)
    i, l = want_padded(orc, buf, offs, padlen, destchar, mask_token, seed, base, th, ignore)
    cu = np.zeros(lens.size + 1, np.int64)
    np.cumsum(lens + k, out=cu[1:])
    return cut(orc, offs, i), cut(orc, offs, l), cu.astype(np.int32)


def check_padded(mb, orc, buf, offs, padlen, destchar, mask_token, **kw):
    assert isinstance(mb, MLMBatch)
    wi, wl = want_padded(orc, buf, offs, padlen, destchar, mask_token, **kw)
    torch.cuda.synchronize()
    assert mb.labels.dtype == torch.int64 and tuple(mb.inputs.shape) == tuple(mb.labels.shape) == wi.shape
    assert_same_bits(wi, mb.inputs.cpu().numpy())
    assert_same_bits(wl, mb.labels.cpu().numpy())


def check_varlen(mb, orc, buf, offs, destchar, mask_token, **kw):
    assert isinstance(mb, MLMBatch) and isinstance(mb.inputs, VarlenBatch)
    wi, wl, wcu = want_varlen(orc, buf, offs, destchar, mask_token, **kw)
    torch.cuda.synchronize()
    assert mb.labels.dtype == torch.int64 and mb.labels.dim() == 1
    assert_same_bits(wi, mb.inputs.tokens.cpu().numpy())
    assert_same_bits(wl, mb.labels.cpu().numpy())
    assert_same_bits(wcu, mb.inputs.cu_seqlens.cpu().numpy())


def mlm_kw(mask_token, seed=0, base=0):
    """batch_tokenize_mlm arguments whose thresholds are TH."""
    return dict(maskfrac=0.3, mask_prob=0.6, random_prob=0.3, mask_token=mask_token, seed=seed, seq_index_base=base)


@pytest.mark.parametrize("key", ["PROTEIN", "DNA", "BYTES"])
@pytest.mark.parametrize("destchar", DESTCHARS)
@pytest.mark.parametrize("flags", FLAGS)
def test_flags_and_kinds(key, destchar, flags):
    tok, orc = toks(key, flags)
    buf, offs = gen(1000 * DESTCHARS.index(destchar) + 10 * FLAGS.index(flags) + len(key), 1500, 0, 300, MIX)
    mt = default_mask_token(tok, destchar)
    seed = 12345 + FLAGS.index(flags)
    kw = mlm_kw(None if mt == tok.alphabet_size() else mt, seed=seed, base=3)
    check_padded(batch_tokenize_mlm(tok, cuda(buf, offs), padlen=320, destchar=destchar, **kw), orc, buf, offs, 320, destchar, mt,
                 seed=seed, base=3)
    check_varlen(batch_tokenize_mlm(tok, cuda(buf, offs), destchar=destchar, varlen=True, **kw), orc, buf, offs, destchar, mt,
                 seed=seed, base=3)


@pytest.mark.parametrize("flags", [(True, True, True), (False, False, False), (True, False, False), (False, True, True)])
@pytest.mark.parametrize("destchar", ["B", "l"])
def test_padded_rows_cut_equal_varlen(flags, destchar):
    tok, orc = toks("PROTEIN", flags)
    buf, offs = gen(31 + FLAGS.index(flags), 4000, 0, 1000, MIX)
    k = sum(flags[:2])
    p = batch_tokenize_mlm(tok, cuda(buf, offs), padlen=1024, destchar=destchar, seed=9)
    v = batch_tokenize_mlm(tok, cuda(buf, offs), destchar=destchar, varlen=True, seed=9)
    lens = np.diff(offs)
    cu = v.inputs.cu_seqlens.cpu().numpy()
    pi, pl, vi, vl = (x.cpu().numpy() for x in (p.inputs, p.labels, v.inputs.tokens, v.labels))
    for i in range(lens.size):
        n = int(lens[i]) + k
        assert np.array_equal(pi[i, :n], vi[cu[i]:cu[i + 1]]) and np.array_equal(pl[i, :n], vl[cu[i]:cu[i + 1]])
        assert (pl[i, n:] == -100).all()


@pytest.mark.parametrize("flags", [(True, True, True), (False, False, False)])
def test_maskfrac_zero_and_all_masked(flags):
    tok, orc = toks("PROTEIN", flags)
    buf, offs = gen(41, 3000, 0, 700, MIX)
    d = cuda(buf, offs)
    k = sum(flags[:2])
    for destchar in ("B", "i", "d"):
        p = batch_tokenize_mlm(tok, d, padlen=704, destchar=destchar, maskfrac=0.0)
        assert torch.equal(p.inputs, tok.batch_tokenize_packed(*d, padlen=704, batch_first=True, destchar=destchar))
        assert (p.labels == -100).all()
        v = batch_tokenize_mlm(tok, d, destchar=destchar, varlen=True, maskfrac=0.0, ignore_index=-1)
        ref = batch_tokenize_varlen(tok, d, destchar)
        assert torch.equal(v.inputs.tokens, ref.tokens) and torch.equal(v.inputs.cu_seqlens, ref.cu_seqlens)
        assert v.inputs.max_seqlen == ref.max_seqlen and (v.labels == -1).all()
    # every residue masked, specials kept
    p = batch_tokenize_mlm(tok, d, padlen=704, maskfrac=1.0, mask_prob=1.0, random_prob=0.0)
    plain = tok.batch_tokenize_packed(*d, padlen=704, batch_first=True).cpu().numpy()
    lens = np.diff(offs)
    cols = np.arange(704)[None, :]
    res = (cols >= flags[0]) & (cols < flags[0] + lens[:, None])
    pi, pl = p.inputs.cpu().numpy(), p.labels.cpu().numpy()
    assert (pi[res] == tok.alphabet_size()).all() and np.array_equal(pi[~res], plain[~res])
    assert np.array_equal(pl[res], plain[res].astype(np.int64)) and (pl[~res] == -100).all()
    v = batch_tokenize_mlm(tok, d, varlen=True, maskfrac=1.0, mask_prob=1.0, random_prob=0.0)
    assert int((v.inputs.tokens == tok.alphabet_size()).sum()) == int(lens.sum())
    assert int((v.labels != -100).sum()) == int(lens.sum()) and v.labels.numel() == int(lens.sum()) + k * lens.size


def test_seq_index_base_slicing():
    tok, orc = toks("PROTEIN", (True, True, True))
    buf, offs = gen(51, 5000, 0, 500, MIX)
    full = batch_tokenize_mlm(tok, cuda(buf, offs), padlen=512, seed=3)
    fv = batch_tokenize_mlm(tok, cuda(buf, offs), varlen=True, seed=3)
    for a, b in ((0, 1), (17, 2000), (4321, 5000)):
        part = batch_tokenize_mlm(tok, cuda(buf, offs[a:b + 1].copy()), padlen=512, seed=3, seq_index_base=a)
        assert torch.equal(part.inputs, full.inputs[a:b]) and torch.equal(part.labels, full.labels[a:b])
        pv = batch_tokenize_mlm(tok, cuda(buf, offs[a:b + 1].copy()), varlen=True, seed=3, seq_index_base=a)
        cu = fv.inputs.cu_seqlens
        lo, hi = int(cu[a]), int(cu[b])
        assert torch.equal(pv.inputs.tokens, fv.inputs.tokens[lo:hi]) and torch.equal(pv.labels, fv.labels[lo:hi])
    other = batch_tokenize_mlm(tok, cuda(buf, offs), padlen=512, seed=3, seq_index_base=1)
    assert not torch.equal(other.labels, full.labels)


@pytest.mark.parametrize("padlen", [1026, 1023, 601, 16, 17])
@pytest.mark.parametrize("destchar", ["B", "h", "l"])
def test_unaligned_padlen(padlen, destchar):
    tok, orc = toks("PROTEIN", (True, True, True))
    buf, offs = gen(61 + padlen, 2000, 0, padlen - 2, MIX)
    check_padded(batch_tokenize_mlm(tok, cuda(buf, offs), padlen=padlen, destchar=destchar, **mlm_kw(None)), orc, buf, offs,
                 padlen, destchar, tok.alphabet_size())


@pytest.mark.parametrize("flags", [(True, True, True), (False, False, False), (True, False, False)])
@pytest.mark.parametrize("shift", range(16))
def test_source_alignment(flags, shift):
    tok, orc = toks("PROTEIN", flags)
    buf, offs = gen(100 + shift, 1500, 0, 700, MIX)
    buf = np.concatenate([np.full(shift + 32, ord("W"), np.uint8), buf])
    offs = offs + shift + 32
    mt = tok.alphabet_size()
    check_padded(batch_tokenize_mlm(tok, cuda(buf, offs), padlen=704, **mlm_kw(None)), orc, buf, offs, 704, "B", mt)
    check_varlen(batch_tokenize_mlm(tok, cuda(buf, offs), varlen=True, **mlm_kw(None)), orc, buf, offs, "B", mt)
    check_varlen(batch_tokenize_mlm(tok, (buf, offs), destchar="h", varlen=True, **mlm_kw(None)), orc, buf, offs, "h", mt)


def test_empty_batch_and_empty_rows():
    tok, orc = toks("PROTEIN", (True, True, True))
    buf, offs = np.zeros(0, np.uint8), np.zeros(1, np.int64)
    for batch in ((buf, offs), cuda(buf, offs)):
        p = batch_tokenize_mlm(tok, batch, padlen=8)
        v = batch_tokenize_mlm(tok, batch, varlen=True)
        torch.cuda.synchronize()
        assert tuple(p.inputs.shape) == tuple(p.labels.shape) == (0, 8)
        assert tuple(v.inputs.tokens.shape) == tuple(v.labels.shape) == (0,) and v.inputs.cu_seqlens.cpu().tolist() == [0]
    for flags in ((True, True, True), (False, False, False), (False, True, False)):
        tok, orc = toks("DNA", flags)
        for n in (1, 17, 40000):
            buf, offs = np.zeros(0, np.uint8), np.zeros(n + 1, np.int64)
            check_padded(batch_tokenize_mlm(tok, cuda(buf, offs), padlen=4, **mlm_kw(None)), orc, buf, offs, 4, "B",
                         tok.alphabet_size())
            check_varlen(batch_tokenize_mlm(tok, cuda(buf, offs), varlen=True, **mlm_kw(None)), orc, buf, offs, "B",
                         tok.alphabet_size())


@pytest.mark.parametrize("flags", [(True, True, True), (False, True, False), (False, False, False)])
def test_short_rows_and_one_long_row(flags):
    tok, orc = toks("PROTEIN", flags)
    mt = tok.alphabet_size()
    for seed, n, hi in ((1, 20000, 40), (2, 100000, 8), (3, 30000, 3)):
        buf, offs = gen(seed, n, 0, hi, MIX)
        check_padded(batch_tokenize_mlm(tok, cuda(buf, offs), padlen=hi + 2, **mlm_kw(None)), orc, buf, offs, hi + 2, "B", mt)
        check_varlen(batch_tokenize_mlm(tok, cuda(buf, offs), destchar="i", varlen=True, **mlm_kw(None)), orc, buf, offs, "i", mt)
    parts = [gen(s, 1, n, n, MIX)[0] for s, n in ((4, 5), (5, 5 * 16384 + 123), (6, 0), (7, 3 * 16384), (8, 9))]
    buf = np.concatenate(parts)
    offs = np.zeros(len(parts) + 1, np.int64)
    np.cumsum([p.size for p in parts], out=offs[1:])
    check_padded(batch_tokenize_mlm(tok, cuda(buf, offs), padlen=5 * 16384 + 126, destchar="l", **mlm_kw(None)), orc, buf, offs,
                 5 * 16384 + 126, "l", mt)
    check_varlen(batch_tokenize_mlm(tok, cuda(buf, offs), destchar="B", varlen=True, **mlm_kw(None)), orc, buf, offs, "B", mt)


def test_input_forms_and_augment(tmp_path):
    tok, orc = toks("PROTEIN", (True, True, True))
    mt = tok.alphabet_size()
    buf, offs = gen(300, 2000, 0, 900, MIX)
    seqs = [buf[offs[i]:offs[i + 1]].tobytes() for i in range(offs.size - 1)]
    kw = mlm_kw(None, seed=5)
    for batch in (seqs, [bytearray(s) for s in seqs], (buf, offs), (torch.from_numpy(buf).pin_memory(), torch.from_numpy(offs).pin_memory()),
                  cuda(buf, offs)):
        check_padded(batch_tokenize_mlm(tok, batch, padlen=902, **kw), orc, buf, offs, 902, "B", mt, seed=5)
        check_varlen(batch_tokenize_mlm(tok, batch, varlen=True, **kw), orc, buf, offs, "B", mt, seed=5)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        a = batch_tokenize_mlm(tok, cuda(buf, offs), padlen=902, **kw)
        b = batch_tokenize_mlm(tok, (buf, offs), varlen=True, **kw)
    side.synchronize()
    check_padded(a, orc, buf, offs, 902, "B", mt, seed=5)
    check_varlen(b, orc, buf, offs, "B", mt, seed=5)
    # a FlatFile range (offsets[0] != 0); padlen defaults to maxseqlen + bos + eos
    ascii_seqs = [bytes(c if c < 0x80 and c not in (10, 13, 62, 64) else 65 for c in s) for s in seqs]
    path = tmp_path / "m.ff"
    path.write_bytes(flatfile_image(ascii_seqs))
    ff = cbioseq.FlatFile(str(path))
    fb, fo = (np.asarray(x) for x in ff.packed(0, len(ascii_seqs)))
    sub = fo[123:1790]
    P = ff.maxseqlen + 2
    check_padded(batch_tokenize_mlm(tok, (ff, 123, 1789), **mlm_kw(None, seed=5, base=123)), orc, fb, sub, P, "B", mt, seed=5, base=123)
    check_varlen(batch_tokenize_mlm(tok, (ff, 123, 1789), varlen=True, **mlm_kw(None, seed=5, base=123)), orc, fb, sub, "B", mt,
                 seed=5, base=123)
    # augmentation first (the oracle's bsqo_augment), then the mask (the reference rule), one seed for both
    pbuf, poffs = gen(301, 1500, 1, 600, b"ACDEFGHIKLMNPQRSTVWY")
    mut = oracle.augment(pbuf, poffs, chain_len=2, augment_frac=0.7, seed=11, seq_index_base=40)
    for batch in ((pbuf, poffs), cuda(pbuf, poffs)):
        check_padded(batch_tokenize_mlm(tok, batch, padlen=602, augment=2, augment_frac=0.7, **mlm_kw(None, seed=11, base=40)),
                     orc, mut, poffs, 602, "B", mt, seed=11, base=40)
        check_varlen(batch_tokenize_mlm(tok, batch, varlen=True, augment=2, augment_frac=0.7, **mlm_kw(None, seed=11, base=40)),
                     orc, mut, poffs, "B", mt, seed=11, base=40)
    d = cuda(pbuf, poffs)
    batch_tokenize_mlm(tok, d, padlen=602, augment=2, seed=11)
    torch.cuda.synchronize()
    assert np.array_equal(d[0].cpu().numpy(), pbuf)  # the caller's residues are not mutated


def _desc(tok):
    return consumers.descriptor(tok)


def test_back_to_back_graph_and_streams():
    tok_py, orc = toks("PROTEIN", (True, True, True))
    tok = _desc(tok_py)
    buf_a, offs = gen(90, 20000, 50, 1022, MIX)
    buf_b = gen(91, 1, buf_a.size, buf_a.size, MIX)[0]
    mt = tok_py.alphabet_size()
    m = capi.mlm_desc(7, 0, TH, mt, -100)
    pa = want_padded(orc, buf_a, offs, 1024, "B", mt, seed=7)
    pb = want_padded(orc, buf_b, offs, 1024, "B", mt, seed=7)
    va = want_varlen(orc, buf_a, offs, "B", mt, seed=7)
    vb = want_varlen(orc, buf_b, offs, "B", mt, seed=7)
    da, db = cuda(buf_a, offs), cuda(buf_b, offs)
    n = offs.size - 1
    pin, plab = torch.zeros((n, 1024), dtype=torch.uint8, device="cuda"), torch.zeros((n, 1024), dtype=torch.int64, device="cuda")
    T = va[0].size
    vin, vlab = torch.zeros(T, dtype=torch.uint8, device="cuda"), torch.zeros(T, dtype=torch.int64, device="cuda")
    cu = torch.zeros(n + 1, dtype=torch.int32, device="cuda")

    def launch(st, d):
        capi.tokenize_mlm(0, st, d[0], d[1], n, 1024, tok, capi.I8, m, pin, plab)
        capi.tokenize_varlen_mlm(0, st, d[0], d[1], n, tok, capi.I8, m, vin, vlab, cu)

    def expect(p, v):
        torch.cuda.synchronize()
        assert_same_bits(p[0], pin.cpu().numpy())
        assert_same_bits(p[1], plab.cpu().numpy())
        assert_same_bits(v[0], vin.cpu().numpy())
        assert_same_bits(v[1], vlab.cpu().numpy())
        assert_same_bits(v[2], cu.cpu().numpy())

    st = torch.cuda.current_stream().cuda_stream
    for i in range(20):
        launch(st, da if i % 2 == 0 else db)
    expect(pb, vb)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(9):
            launch(torch.cuda.current_stream().cuda_stream, da if i % 2 == 0 else db)
    for _ in range(2):
        for t in (pin, plab, vin, vlab, cu):
            t.zero_()
        g.replay()
        expect(pa, va)
        launch(torch.cuda.current_stream().cuda_stream, db)
        expect(pb, vb)
    # concurrent streams, each with its own outputs
    streams = [torch.cuda.Stream() for _ in range(4)]
    outs = [(torch.zeros((n, 1024), dtype=torch.uint8, device="cuda"), torch.zeros((n, 1024), dtype=torch.int64, device="cuda"),
             torch.zeros(T, dtype=torch.uint8, device="cuda"), torch.zeros(T, dtype=torch.int64, device="cuda"),
             torch.zeros(n + 1, dtype=torch.int32, device="cuda")) for _ in streams]
    torch.cuda.synchronize()
    for rep in range(3):
        for s, (a, b, c, e, f) in zip(streams, outs):
            capi.tokenize_mlm(0, s.cuda_stream, da[0], da[1], n, 1024, tok, capi.I8, m, a, b)
            capi.tokenize_varlen_mlm(0, s.cuda_stream, da[0], da[1], n, tok, capi.I8, m, c, e, f)
    torch.cuda.synchronize()
    for a, b, c, e, f in outs:
        for want, got in zip(pa + va, (a, b, c, e, f)):
            assert_same_bits(want, got.cpu().numpy())


def test_dataset(tmp_path):
    tok, orc = toks("PROTEIN", (True, True, True))
    buf, offs = gen(400, 3000, 0, 600, b"ACDEFGHIKLMNPQRSTVWY")
    seqs = [buf[offs[i]:offs[i + 1]].tobytes() for i in range(offs.size - 1)]
    path = tmp_path / "d.ff"
    path.write_bytes(flatfile_image(seqs))
    ff = cbioseq.FlatFile(str(path))
    P = ff.maxseqlen + 2

    def seed_of(draw, base=13):
        return (base & 0xFFFFFFFF) | (draw << 32)

    for varlen in (False, True):
        ds = FlatFileDataset(ff, tok, mlm=True, varlen=varlen, maskfrac=0.2)
        part = ds[100:2100]                                                     # draw 1
        ref = batch_tokenize_mlm(tok, (ff, 100, 2100), destchar="l", varlen=varlen, padlen=-1 if varlen else P, maskfrac=0.2,
                                 seed=seed_of(1), seq_index_base=100)
        assert isinstance(part, MLMBatch) and part.labels.dtype == torch.long
        if varlen:
            assert part.inputs.tokens.dtype == torch.long and torch.equal(part.inputs.tokens, ref.inputs.tokens)
            assert torch.equal(part.inputs.cu_seqlens, ref.inputs.cu_seqlens)
        else:
            assert part.inputs.dtype == torch.long and part.inputs.shape == (2000, P) and torch.equal(part.inputs, ref.inputs)
        assert torch.equal(part.labels, ref.labels)
        again = ds[100:2100]                                                    # draw 2: a different mask
        assert not torch.equal(again.labels, part.labels)
        one = ds[5]                                                             # draw 3
        r1 = batch_tokenize_mlm(tok, (ff, 5, 6), destchar="l", varlen=varlen, padlen=-1 if varlen else P, maskfrac=0.2,
                                seed=seed_of(3), seq_index_base=5)
        assert one.inputs.dim() == 1 and one.labels.dim() == 1
        if varlen:
            assert torch.equal(one.inputs, r1.inputs.tokens) and torch.equal(one.labels, r1.labels)
        else:
            assert torch.equal(one.inputs, r1.inputs[0]) and torch.equal(one.labels, r1.labels[0])
        for prefetch in (0, 2):
            ds = FlatFileDataset(ff, tok, mlm=True, varlen=varlen, seed=21)
            got = list(ds.batches(700, prefetch=prefetch))
            assert len(got) == 5
            for j, mb in enumerate(got):
                r = batch_tokenize_mlm(tok, (ff, 700 * j, min(700 * (j + 1), 3000)), destchar="l", varlen=varlen,
                                       padlen=-1 if varlen else P, maskfrac=0.15, seed=seed_of(j + 1, 21), seq_index_base=700 * j)
                gi, ri = (mb.inputs.tokens, r.inputs.tokens) if varlen else (mb.inputs, r.inputs)
                assert torch.equal(gi, ri) and torch.equal(mb.labels, r.labels)
    # augmentation and the mask share the per-fetch seed
    ds = FlatFileDataset(ff, tok, mlm=True, augment=1, augment_frac=1.0)
    got = ds[0:500]
    r = batch_tokenize_mlm(tok, (ff, 0, 500), padlen=P, destchar="l", augment=1, augment_frac=1.0, seed=seed_of(1))
    assert torch.equal(got.inputs, r.inputs) and torch.equal(got.labels, r.labels)
    with pytest.raises(ValueError):
        FlatFileDataset(ff, tok, mlm=True, cnn=True)


def test_errors():
    tok, _ = toks("PROTEIN", (True, True, True))
    buf, offs = gen(500, 100, 0, 50, MIX)
    with pytest.raises(RuntimeError, match="seq len"):
        batch_tokenize_mlm(tok, (buf, offs), padlen=20)
    with pytest.raises(ValueError, match="provded"):
        batch_tokenize_mlm(tok, [b"ACD"])
    with pytest.raises(ValueError, match="padlen"):
        batch_tokenize_mlm(tok, (buf, offs), padlen=64, varlen=True)
    with pytest.raises(ValueError, match="item was none of"):
        batch_tokenize_mlm(tok, ["ACGT", 5], padlen=64)
    with pytest.raises(ValueError, match="past the end"):
        batch_tokenize_mlm(tok, cuda(buf[:-1], offs), varlen=True)
    with pytest.raises(ValueError, match="mask_token"):
        batch_tokenize_mlm(cbioseq.Tokenizer("BYTES"), cuda(buf, offs), padlen=64)
    with pytest.raises(ValueError, match="mask_token"):
        batch_tokenize_mlm(tok, cuda(buf, offs), padlen=64, destchar="b", mask_token=200)
    for kw in (dict(maskfrac=-0.5), dict(maskfrac=2.0), dict(mask_prob=0.9, random_prob=0.2), dict(random_prob=-0.1),
               dict(ignore_index=2 ** 63)):
        with pytest.raises(ValueError):
            batch_tokenize_mlm(tok, cuda(buf, offs), padlen=64, **kw)
    big = np.zeros(2 ** 31 - 2, np.uint8)
    capi.lib().bsq_launch_count_reset()
    with pytest.raises(ValueError, match="2\\^31 - 1"):
        batch_tokenize_mlm(tok, (big, np.array([0, big.size], np.int64)), varlen=True)
    assert capi.lib().bsq_launch_count() == 0
    del big
