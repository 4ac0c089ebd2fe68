"""Translation into protein reading frames (translate_packed / batch_tokenize_translated / translate= / bsq_translate,
kernel K14), bit for bit against the rule of include/bsq.h (tests/translate_reference.py).

K14a scans each sequence's output bytes (the sum of its frame lengths); K14b writes the n F + 1 output offsets and then
translates as a flat map over 16-byte output vectors in 64 KiB tiles, each vector decoding 16 codons of a 48-byte
source span per (sequence, frame) piece.  The cases cover lengths 0-5, around 48 nucleotides (one output vector) and
around the 64 KiB tile, every source (offsets[0] % 16) and output alignment, all 256 byte values, every ordered frame set,
every built-in code and a custom one, over-full tiles of empty and short rows, an output past 2^31 bytes, the caller's
tensors left unchanged, a side stream, a CUDA graph captured through the C ABI, every consumer with translate= against
the same consumer on the reference-translated batch (crop, MLM and augmentation draws keyed by the output index and
the same across slicings), every batch form, the dataset, and one read-back for a CUDA batch with translate and crop."""
import itertools

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from bioseq_b200 import capi, cbioseq, consumers, translate_packed, batch_tokenize_translated, TranslatedBatch  # noqa: E402
from bioseq_b200 import batch_tokenize_cropped, batch_tokenize_varlen, batch_tokenize_mlm, batch_tokenize_seqpack  # noqa: E402
from bioseq_b200 import batch_tokenize_kmer, batch_onehot_encode_bcl, batch_embed, VarlenBatch  # noqa: E402
from bioseq_b200.loaders import FlatFileDataset  # noqa: E402
from oracle.oracle import flatfile_image  # noqa: E402
from helpers import assert_same_bits, table_cap_lens  # noqa: E402
import translate_reference as ref  # noqa: E402

SIX = (1, 2, 3, -1, -2, -3)
DNA = b"ACGTACGTACGTNacgtuRYSWKMBDHVn-*"


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests selected but no CUDA device is visible")


def cuda(buf, offs):
    return torch.from_numpy(np.ascontiguousarray(buf)).cuda(), torch.from_numpy(np.ascontiguousarray(offs)).cuda()


def batch_of(lens, seed, lead=0, table=DNA):
    offs = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    rng = np.random.default_rng(seed)
    t = np.frombuffer(table, np.uint8) if isinstance(table, bytes) else table
    buf = t[rng.integers(0, t.size, size=int(offs[-1]) + lead)]
    return buf, offs + lead


def check(tb, buf, offs, frames, code=1):
    wb, wo = ref.translate(buf, offs, frames, code)
    torch.cuda.synchronize()
    n, F = len(offs) - 1, len(frames)
    assert isinstance(tb, TranslatedBatch) and tb.frames == tuple(frames)
    assert_same_bits(wo, tb.offsets.cpu().numpy())
    assert_same_bits(wb, tb.bytes.cpu().numpy())
    assert_same_bits(np.repeat(np.arange(n, dtype=np.int64), F), tb.seq_index.cpu().numpy())
    assert_same_bits(np.tile(np.array(frames, np.int8), n), tb.frame.cpu().numpy())


def test_worked_answers():
    seqs = ["ATGGCCATTGTAATGGGCCGCTGAAAGGGTGCCCGATAG", "ATGA", "ATGAA", "", "A", "AT"]
    buf, offs = capi.Pack(pinned=False).gather([s.encode() for s in seqs]).to_numpy()
    tb = translate_packed(*cuda(buf, offs), frames="six")
    o = tb.offsets.tolist()
    got = [tb.bytes[o[w]:o[w + 1]].cpu().numpy().tobytes().decode() for w in range(len(seqs) * 6)]
    assert got[:6] == ["MAIVMGR*KGAR*", "WPL*WAAERVPD", "GHCNGPLKGCPI", "LSGTLSAAHYNGH", "YRAPFQRPITMA", "IGHPFSGPLQWP"]
    assert got[6:18] == ["M", "*", "", "S", "H", "", "M", "*", "E", "F", "S", "H"] and got[18:] == [""] * 18
    codons = ["GCN", "TAR", "TRA", "YTG", "atg", "AUG", "A-G", "TGA", "AGA"]
    buf, offs = capi.Pack(pinned=False).gather([c.encode() for c in codons]).to_numpy()
    for code, frame, want in ((1, 1, "A**LMMX*R"), (2, 1, "A*XLMMXW*"), (1, -1, "XLXQHHXSS")):
        tb = translate_packed(*cuda(buf, offs), frames=frame, genetic_code=code)
        assert tb.bytes.cpu().numpy().tobytes().decode() == want
    for seq, code, want in (("ATAAGATGA", 1, "IR*"), ("ATAAGATGA", 2, "M*W"), ("TAATAG", 6, "QQ")):
        tb = translate_packed(*cuda(np.frombuffer(seq.encode(), np.uint8).copy(), np.array([0, len(seq)])), genetic_code=code)
        assert tb.bytes.cpu().numpy().tobytes().decode() == want


@pytest.mark.parametrize("frames", [SIX, (1,), (-1,), (2, -3), (-3, -2, -1, 3, 2, 1)])
def test_edge_lengths_every_source_alignment(frames):
    lens = list(range(0, 6)) + list(range(44, 54)) + [143, 144, 145, 146, 147, 148, 149, 150, 1000, 3 * 21845, 3 * 21845 + 2,
                                                       65536 * 3 // len(frames) + 7, 200003]
    for lead in range(16):
        buf, offs = batch_of(lens + lens[::-1], 13 + lead, lead)
        b, o = cuda(buf, offs)
        keep_b, keep_o = b.clone(), o.clone()
        check(translate_packed(b, o, frames=frames), buf, offs, frames)
        assert torch.equal(b, keep_b) and torch.equal(o, keep_o)  # the caller's tensors are unchanged


# (sequence lengths, frames): mixed lengths; the same ending in a run of empty sequences (every alignment but one leaves
# the last vector partial); sequences whose frame +1 fills tiles to the row table's cap and one past it
ALIGN_CASES = [([0, 5, 40, 3, 129, 77, 1, 300, 48, 49, 50], SIX), ([0, 5, 40, 3, 129, 77, 1, 300, 48, 49, 50] + [0] * 40, SIX),
               ([3 * n for n in table_cap_lens()], (1,))]


def test_every_output_alignment():
    for lens, frames in ALIGN_CASES:
        buf, offs = batch_of(lens, 3)
        wb, wo = ref.translate(buf, offs, frames)
        b, o = cuda(buf, offs)
        st = torch.cuda.current_stream().cuda_stream
        code = capi.genetic_code(1)
        for a in range(16):
            out = torch.full((wb.size + 32,), 0xEE, dtype=torch.uint8, device="cuda")
            oo = torch.empty(wo.size, dtype=torch.int64, device="cuda")
            capi.translate(0, st, b, o, len(offs) - 1, frames, code, out[a:].data_ptr(), oo)
            torch.cuda.synchronize()
            h = out.cpu().numpy()
            assert_same_bits(wb, h[a:a + wb.size])
            assert (h[:a] == 0xEE).all() and (h[a + wb.size:] == 0xEE).all()
            assert_same_bits(wo, oo.cpu().numpy())


@pytest.mark.parametrize("code", [1, 2, 4, 5, 6, 11, "custom"])
def test_all_byte_values_every_code(code):
    if code == "custom":
        code = "".join(chr(0x21 + (11 * i + 5) % 94) for i in range(64))
    for table in (np.arange(256, dtype=np.uint8), np.frombuffer(DNA, np.uint8)):
        buf, offs = batch_of([0, 1, 2, 3, 7, 48, 100, 1000, 5000, 31], 5, lead=7, table=table)
        check(translate_packed(*cuda(buf, offs), frames="six", genetic_code=code), buf, offs, SIX, code)


def test_every_ordered_frame_set():
    buf, offs = batch_of([0, 2, 3, 4, 5, 17, 48, 49, 50, 64, 151, 333], 17, lead=9)
    b, o = cuda(buf, offs)
    for k in range(1, 7):
        for frames in itertools.permutations(SIX, k):
            check(translate_packed(b, o, frames=list(frames)), buf, offs, frames)


def test_over_full_tiles_and_many_sequences():
    rng = np.random.default_rng(4)  # thousands of empty and short rows per 64 KiB tile, past 1024 (scan CTAs)
    for lens in (rng.integers(0, 6, 300_000), np.zeros(5000, np.int64), rng.integers(0, 60, 100_000)):
        buf, offs = batch_of(lens, 5, lead=3)
        check(translate_packed(*cuda(buf, offs), frames="six"), buf, offs, SIX)
    b, o = cuda(np.zeros(0, np.uint8), np.array([0], np.int64))
    tb = translate_packed(b, o, frames="six")
    assert tb.offsets.tolist() == [0] and tb.bytes.numel() == 0 and tb.seq_index.numel() == 0


def test_output_past_2_pow_31_bytes():
    # 1 200 000 x 1 000 DNA (1.2 GB), six frames: 333 + 333 + 332 amino acids a strand, 2.4 GB of output; checked by samples
    n, L = 1_200_000, 1_000
    per = np.cumsum([0] + [(L - (abs(f) - 1)) // 3 for f in SIX])
    R = int(per[-1])
    g = torch.Generator("cuda").manual_seed(6)
    b = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")[torch.randint(0, 4, (n * L,), device="cuda", generator=g)]
    o = torch.arange(n + 1, dtype=torch.int64, device="cuda") * L
    tb = translate_packed(b, o, frames="six")
    assert R == 1996 and tb.bytes.numel() == n * R > 2 ** 31
    for i in (0, 1, 1_075_000, n // 2 + 7, n - 1):
        assert tb.offsets[i * 6:i * 6 + 6].cpu().numpy().tolist() == (i * R + per[:6]).tolist()
        src = b[i * L:(i + 1) * L].cpu().numpy()
        wb, _ = ref.translate(src, [0, L], SIX)
        assert_same_bits(wb, tb.bytes[i * R:(i + 1) * R].cpu().numpy())
    assert int(tb.offsets[-1]) == n * R
    del b, tb
    torch.cuda.empty_cache()


def test_side_stream_graph_and_bad_offsets():
    buf, offs = batch_of([3, 100, 0, 517, 64, 48], 8)
    frames = (2, -1, 3)
    wb, wo = ref.translate(buf, offs, frames, 2)
    b, o = cuda(buf, offs)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        tb = translate_packed(b, o, frames=frames, genetic_code=2)
    s.synchronize()
    check(tb, buf, offs, frames, 2)
    out_b = torch.empty(wb.size, dtype=torch.uint8, device="cuda")
    out_o = torch.empty(wo.size, dtype=torch.int64, device="cuda")
    code = capi.genetic_code(2)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        capi.translate(0, torch.cuda.current_stream().cuda_stream, b, o, len(offs) - 1, frames, code, out_b, out_o)
    out_b.zero_()
    out_o.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert_same_bits(wb, out_b.cpu().numpy())
    assert_same_bits(wo, out_o.cpu().numpy())
    for bad in ([0, 5, 3], [-1, 5], [0, 10 ** 6]):
        with pytest.raises(ValueError):
            translate_packed(b, torch.tensor(bad, dtype=torch.int64, device="cuda"))


# ---- consumers -------------------------------------------------------------------------------------------------------
def reference_batch(buf, offs, frames, code=1):
    wb, wo = ref.translate(buf, offs, frames, code)
    return cuda(wb, wo)


def forms(buf, offs, tmp_path):
    seqs = [bytes(buf[offs[i]:offs[i + 1]]) for i in range(len(offs) - 1)]
    path = tmp_path / "t.ff"
    path.write_bytes(flatfile_image(seqs))
    ff = cbioseq.FlatFile(str(path))
    host = (buf[offs[0]:].copy(), offs - offs[0])
    return [seqs, host, cuda(*host), (ff, 0, len(seqs))]


PROT = None


def prot():
    global PROT
    if PROT is None:
        PROT = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    return PROT


@pytest.mark.parametrize("frames", [1, "six", (-2, 3)])
def test_every_consumer_equals_the_reference_translated_batch(frames, tmp_path):
    buf, offs = batch_of([0, 7, 300, 45, 1001, 2, 150, 151], 9, lead=3, table=b"ACGTACGTNRY")
    fr = consumers._frames(frames)
    F = len(fr)
    rb = reference_batch(buf, offs, fr, 4)
    tok, seb = prot(), cbioseq.Tokenizer("SEB8", bos=True, eos=True)
    w = torch.randn(tok.alphabet_size(), 64, device="cuda")
    base, seed = 5, 21
    kw = dict(translate=frames, genetic_code=4)
    cases = [
        (lambda x, **t: batch_tokenize_cropped(tok, x, 130, crop="random", seed=seed, seq_index_base=base * (F if not t else 1), **t)),
        (lambda x, **t: batch_tokenize_cropped(seb, x, 40, crop="head", **t)),
        (lambda x, **t: batch_tokenize_varlen(tok, x, crop="random", crop_len=50, seed=seed, seq_index_base=base * (F if not t else 1),
                                              **t).tokens),
        (lambda x, **t: batch_tokenize_mlm(tok, x, 340, seed=seed, seq_index_base=base * (F if not t else 1), **t).labels),
        (lambda x, **t: batch_tokenize_mlm(tok, x, varlen=True, seed=seed, seq_index_base=base * (F if not t else 1), augment=2,
                                           crop="random", crop_len=30, **t).inputs.tokens),
        (lambda x, **t: batch_tokenize_seqpack(tok, x, 400, seed=seed, seq_index_base=base * (F if not t else 1), mlm=True,
                                               augment=1, **t).labels),
        (lambda x, **t: batch_tokenize_kmer(tok, x, 2, 400, stride=2, tail="single", **t)),
        (lambda x, **t: batch_tokenize_kmer(tok, x, 3, varlen=True, crop="head", crop_len=20, **t).tokens),
        (lambda x, **t: batch_onehot_encode_bcl(tok, x, 340, augment=3, seed=seed, seq_index_base=base * (F if not t else 1), **t)),
        (lambda x, **t: batch_embed(tok, x, w, 340, crop="random", crop_len=100, seed=seed, seq_index_base=base * (F if not t else 1),
                                    **t)),
    ]
    for k, f in enumerate(cases):
        want = f(rb)
        for form in forms(buf, offs, tmp_path):
            got = f(form, **kw)
            assert torch.equal(got.cpu(), want.cpu()), (k, type(form))


def test_batch_tokenize_translated_across_forms(tmp_path):
    tok = prot()
    buf, offs = batch_of([0, 9, 130, 64, 65, 33, 2], 11)
    for frames, code in ((1, 1), ("six", 2), ([-3, 1], 11)):
        fr = consumers._frames(frames)
        wb, wo = ref.translate(buf, offs, fr, code)
        rows = [bytes(wb[wo[i]:wo[i + 1]]) for i in range(len(wo) - 1)]
        P = max(len(r) for r in rows) + 2
        want = tok.batch_tokenize(rows, padlen=P, batch_first=True)
        want_v = batch_tokenize_varlen(tok, cuda(wb, wo))
        for form in forms(buf, offs, tmp_path):
            got = batch_tokenize_translated(tok, form, frames=frames, genetic_code=code)
            assert tuple(got.shape) == (len(rows), P) and torch.equal(got.cpu(), want.cpu())
            got = batch_tokenize_translated(tok, form, 300, "l", frames=frames, genetic_code=code)
            assert torch.equal(got[:, :P].cpu(), want.long().cpu())
            vb = batch_tokenize_translated(tok, form, frames=frames, genetic_code=code, varlen=True)
            assert isinstance(vb, VarlenBatch) and torch.equal(vb.tokens.cpu(), want_v.tokens.cpu())
            assert torch.equal(vb.cu_seqlens.cpu(), want_v.cu_seqlens.cpu()) and vb.max_seqlen == want_v.max_seqlen
    # BYTES keeps the letters: '*' and 'X' tokenize as themselves, PROTEIN as invalid bytes (0)
    byts = cbioseq.Tokenizer("BYTES")
    got = batch_tokenize_translated(byts, ["TAATAGNNN"])
    assert got[0].tolist() == list(b"**X")
    assert batch_tokenize_translated(cbioseq.Tokenizer("PROTEIN"), ["TAANNNATG"])[0].tolist() == [0, 0, tok.batch_tokenize(["M"], padlen=3,
                                                                                                                        batch_first=True)[0, 1].item()]


def test_draws_keyed_by_output_index_and_same_across_slicings():
    tok = prot()
    buf, offs = batch_of([400, 20, 333, 151, 90, 600, 3, 301], 2, table=b"ACGT")
    host = (buf, offs)
    full = batch_tokenize_mlm(tok, host, 210, seed=9, translate="six", crop="random", augment=2)
    for lo, hi in ((0, 3), (3, 8), (5, 6)):
        part = (buf, offs[lo:hi + 1])
        got = batch_tokenize_mlm(tok, part, 210, seed=9, seq_index_base=lo, translate="six", crop="random", augment=2)
        assert torch.equal(got.inputs, full.inputs[6 * lo:6 * hi]) and torch.equal(got.labels, full.labels[6 * lo:6 * hi])
        got = batch_tokenize_mlm(tok, cuda(*part), 210, seed=9, seq_index_base=lo, translate="six", crop="random", augment=2)
        assert torch.equal(got.inputs, full.inputs[6 * lo:6 * hi])


def test_one_read_back_for_a_cuda_batch_with_translate_and_crop(monkeypatch):
    tok = prot()
    buf, offs = batch_of([0, 500, 31, 2000, 47], 1)
    b, o = cuda(buf, offs)
    syncs = []
    for name in ("crop_extent_device", "translate_extent_device", "varlen_extent_device", "check_lengths_device",
                 "kmer_extent_device", "tile_extent_device"):
        real = getattr(capi, name)
        monkeypatch.setattr(capi, name, lambda *a, _real=real, _name=name, **k: syncs.append(_name) or _real(*a, **k))
    real_cpu = torch.Tensor.cpu
    monkeypatch.setattr(torch.Tensor, "cpu", lambda self, *a, **k: syncs.append("cpu") or real_cpu(self, *a, **k))
    batch_tokenize_cropped(tok, (b, o), 100, crop="random", translate="six")
    assert syncs == ["translate_extent_device"]
    syncs.clear()
    batch_tokenize_varlen(tok, (b, o), crop="head", crop_len=64, translate=(1, -1))
    assert syncs == ["translate_extent_device"]
    syncs.clear()
    batch_tokenize_translated(tok, (b, o), frames="six", crop="random", crop_len=64)
    assert syncs == ["translate_extent_device"]
    syncs.clear()
    batch_tokenize_translated(tok, (buf, offs), frames="six")  # a host batch: sized in numpy
    assert syncs == []


def test_dataset(tmp_path):
    tok = prot()
    buf, offs = batch_of([30, 7, 300, 45, 100, 2, 151, 90, 64], 9, table=b"ACGT")
    seqs = [bytes(buf[offs[i]:offs[i + 1]]) for i in range(len(offs) - 1)]
    path = tmp_path / "d.ff"
    path.write_bytes(flatfile_image(seqs))
    ff = cbioseq.FlatFile(str(path))
    ds = FlatFileDataset(ff, tok, translate="six")
    assert ds.max_seq_len == 300 // 3 + 2
    wb, wo = ref.translate(buf, offs, SIX)
    rows = [bytes(wb[wo[i]:wo[i + 1]]) for i in range(len(wo) - 1)]
    want = tok.batch_tokenize(rows, padlen=ds.max_seq_len, batch_first=True).long()
    got = ds[2:5]
    assert tuple(got.shape) == (18, ds.max_seq_len) and torch.equal(got, want[12:30])
    assert torch.equal(ds[3], want[18:24])
    one = FlatFileDataset(ff, tok, translate=-1)
    w1b, w1o = ref.translate(buf, offs, (-1,))
    r1 = tok.batch_tokenize([bytes(w1b[w1o[i]:w1o[i + 1]]) for i in range(len(w1o) - 1)], padlen=one.max_seq_len, batch_first=True)
    assert one[4].dim() == 1 and torch.equal(one[4], r1[4].long()) and torch.equal(one[1:3], r1[1:3].long())
    ds = FlatFileDataset(ff, tok, translate="forward", max_seq_len=22, crop="head")
    wfb, wfo = ref.translate(buf, offs, (1, 2, 3))
    want = tok.batch_tokenize([bytes(wfb[wfo[i]:wfo[i] + min(20, wfo[i + 1] - wfo[i])]) for i in range(len(wfo) - 1)], padlen=22,
                              batch_first=True).long()
    assert torch.equal(ds[0:9], want)
    vds = FlatFileDataset(ff, tok, translate="forward", varlen=True)
    assert torch.equal(vds[0:9].tokens.long().cpu(), batch_tokenize_varlen(tok, cuda(wfb, wfo), "l").tokens.cpu())
    mds = FlatFileDataset(ff, tok, translate="six", mlm=True, max_seq_len=40)
    mb = mds[1:4]
    assert tuple(mb.inputs.shape) == (18, 40)
    cds = FlatFileDataset(ff, tok, translate=1, cnn=True)
    assert tuple(cds[0:3].shape) == (3, tok.alphabet_size(), cds.max_seq_len)
    assert tuple(cds[2].shape) == (cds.max_seq_len, tok.alphabet_size())
    with pytest.raises(ValueError):
        FlatFileDataset(ff, tok, translate="six", rc="random")
    with pytest.raises(ValueError):
        FlatFileDataset(ff, cbioseq.Tokenizer("DNA"), translate=1)
