"""Sliding-window tiling and stitching (tile_packed / batch_tokenize_tiled / untile / bsq_tile / bsq_untile_mean, kernel
K13), bit for bit against the rule of include/bsq.h (tests/tile_reference.py).

K13a scans window counts and window bytes per sequence, then writes the window table and gathers the windows' bytes as a
flat map over 16-byte output vectors (each tile searching its first sequence, every window found by a division by W).
The cases cover lengths around W, S and the 16-byte vector, every source and output alignment, every tail, heavy overlap
(S = 1, W = 64) and S = W, a row of 2^24 + 3 bytes, empty batches and all-empty sequences, an output past 2^31 bytes,
NULL optional outputs, a side stream, a CUDA graph captured through the C ABI, every consumer on the tiled batch against
the same consumer on the reference-tiled batch, and batch_tokenize_tiled across batch forms.  K13b (untile) is checked
for three dtypes, several channel counts, padded and padding-free outputs, one and two strands, random flips, DROP tails
and the worked answers, and by a round trip that must give every residue its own position."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from bioseq_b200 import capi, cbioseq, tile_packed, batch_tokenize_tiled, untile, TiledTokens  # noqa: E402
from bioseq_b200 import batch_tokenize_varlen, batch_tokenize_mlm, batch_tokenize_kmer, revcomp_packed  # noqa: E402
from bioseq_b200 import VarlenBatch  # noqa: E402
from oracle.oracle import flatfile_image  # noqa: E402
from helpers import assert_same_bits, table_cap_lens  # noqa: E402
import tile_reference as ref  # noqa: E402
from revcomp_reference import revcomp as reference_revcomp  # noqa: E402

DNA = b"ACGTNacgtn"
TAILS = {"short": capi.TILE_SHORT, "end": capi.TILE_END, "drop": capi.TILE_DROP}


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests selected but no CUDA device is visible")


def cuda(buf, offs):
    return torch.from_numpy(np.ascontiguousarray(buf)).cuda(), torch.from_numpy(np.ascontiguousarray(offs)).cuda()


def batch_of(lens, seed, lead=0):
    offs = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    rng = np.random.default_rng(seed)
    table = np.frombuffer(DNA, np.uint8)
    buf = table[rng.integers(0, table.size, size=int(offs[-1]) + lead)]
    return buf, offs + lead


def check(tb, buf, offs, W, S, tail):
    wb, wo, wsp, wsi, wst = ref.tile(buf, offs, W, S, tail)
    torch.cuda.synchronize()
    assert_same_bits(wo, tb.offsets.cpu().numpy())
    assert_same_bits(wsp, tb.seq_ptr.cpu().numpy())
    assert_same_bits(wsi, tb.seq_index.cpu().numpy())
    assert_same_bits(wst, tb.starts.cpu().numpy())
    assert_same_bits(wb, tb.bytes.cpu().numpy())
    assert_same_bits(offs - offs[0], tb.seq_offsets.cpu().numpy())


@pytest.mark.parametrize("tail", ["short", "end", "drop"])
@pytest.mark.parametrize("W,S", [(4, 3), (16, 16), (17, 5), (64, 1), (100, 100), (33, 32)])
def test_edge_lengths_every_source_alignment(tail, W, S):
    lens = sorted({0, 1, 15, 16, 17, W - 1, W, W + 1, W + S - 1, W + S, W + S + 1, 2 * W + 7, 5 * W + 3, 1000} - {-1})
    for lead in range(16):
        buf, offs = batch_of(lens + lens[::-1], 13 + lead, lead)
        check(tile_packed(*cuda(buf, offs), W, stride=S, tail=tail), buf, offs, W, S, tail)


# (sequence lengths, W, S): mixed lengths; the same ending in a run of empty sequences (every alignment but one leaves the
# last vector partial); one window per sequence that fills tiles to the row table's cap and one past it
ALIGN_CASES = [([0, 5, 40, 3, 129, 77, 1, 300], 24, 10), ([0, 5, 40, 3, 129, 77, 1, 300] + [0] * 40, 24, 10),
               (table_cap_lens(), 65536, 65536)]


@pytest.mark.parametrize("tail", ["short", "end", "drop"])
def test_every_output_alignment_and_null_outputs(tail):
    for lens, W, S in ALIGN_CASES:
        buf, offs = batch_of(lens, 3)
        wb, wo, wsp, wsi, wst = ref.tile(buf, offs, W, S, tail)
        b, o = cuda(buf, offs)
        st = torch.cuda.current_stream().cuda_stream
        for a in range(16):
            out = torch.full((wb.size + 32,), 0xEE, dtype=torch.uint8, device="cuda")
            oo = torch.empty(wo.size, dtype=torch.int64, device="cuda")
            capi.tile(0, st, b, o, len(offs) - 1, W, S, TAILS[tail], out[a:].data_ptr(), oo)  # every optional output NULL
            torch.cuda.synchronize()
            h = out.cpu().numpy()
            assert_same_bits(wb, h[a:a + wb.size])
            assert (h[:a] == 0xEE).all() and (h[a + wb.size:] == 0xEE).all()
            assert_same_bits(wo, oo.cpu().numpy())


def test_empty_batches_huge_row_and_many_sequences():
    b, o = cuda(np.zeros(0, np.uint8), np.array([0], np.int64))
    tb = tile_packed(b, o, 8)
    assert tb.offsets.tolist() == [0] and tb.seq_ptr.tolist() == [0] and tb.bytes.numel() == 0
    buf, offs = batch_of([0] * 5000, 1)
    tb = tile_packed(*cuda(buf, offs), 8, stride=3)
    check(tb, buf, offs, 8, 3, "short")
    for tail in ("short", "end", "drop"):
        buf, offs = batch_of([2 ** 24 + 3], 2, lead=5)
        check(tile_packed(*cuda(buf, offs), 1000, stride=333, tail=tail), buf, offs, 1000, 333, tail)
    rng = np.random.default_rng(4)  # over-full tiles: thousands of short sequences per 64 KiB tile, past 1024 (scan CTAs)
    lens = rng.integers(0, 12, 300_000)
    buf, offs = batch_of(lens, 5, lead=3)
    check(tile_packed(*cuda(buf, offs), 7, stride=2, tail="end"), buf, offs, 7, 2, "end")


def test_output_past_2_pow_31_bytes():
    # 600 000 x 4 000 DNA (2.4 GB), W = 2 000, S = 1 000: 3 windows each, 3.6 GB of output; checked by samples
    n, L, W, S = 600_000, 4_000, 2_000, 1_000
    b = torch.randint(65, 91, (n * L,), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(6))
    o = torch.arange(n + 1, dtype=torch.int64, device="cuda") * L
    tb = tile_packed(b, o, W, stride=S)
    assert tb.bytes.numel() == 3 * n * W > 2 ** 31
    assert torch.equal(tb.offsets[::97], torch.arange(0, 3 * n + 1, 97, device="cuda") * W)
    for w in (0, 1, 2, 1_073_741 // 2, 3 * n // 2 + 1, 3 * n - 1):
        i, j = w // 3, w % 3
        assert torch.equal(tb.bytes[w * W:(w + 1) * W], b[i * L + j * S:i * L + j * S + W]), w
    assert torch.equal(tb.bytes[-W:], b[-W:])
    del b, tb
    torch.cuda.empty_cache()


def test_side_stream_graph_and_bad_offsets():
    buf, offs = batch_of([3, 100, 0, 517, 64], 8)
    W, S = 32, 7
    wb, wo, wsp, wsi, wst = ref.tile(buf, offs, W, S, "end")
    b, o = cuda(buf, offs)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        tb = tile_packed(b, o, W, stride=S, tail="end")
    s.synchronize()
    check(tb, buf, offs, W, S, "end")
    out_b = torch.empty(wb.size, dtype=torch.uint8, device="cuda")
    out_o = torch.empty(wo.size, dtype=torch.int64, device="cuda")
    sp, si, st = (torch.empty(k, dtype=torch.int64, device="cuda") for k in (wsp.size, wsi.size, wst.size))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        capi.tile(0, torch.cuda.current_stream().cuda_stream, b, o, len(offs) - 1, W, S, capi.TILE_END, out_b, out_o, sp, si, st)
    for x in (out_b, out_o, sp, si, st):
        x.zero_()
    g.replay()
    torch.cuda.synchronize()
    for want, got in ((wb, out_b), (wo, out_o), (wsp, sp), (wsi, si), (wst, st)):
        assert_same_bits(want, got.cpu().numpy())
    for bad in ([0, 5, 3], [-1, 5], [0, 10 ** 6]):
        with pytest.raises(ValueError):
            tile_packed(b, torch.tensor(bad, dtype=torch.int64, device="cuda"), 8)


def test_consumers_on_the_tiled_batch():
    dna = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
    buf, offs = batch_of([0, 7, 300, 45, 1001], 9, lead=3)
    W, S = 40, 25
    tb = tile_packed(*cuda(buf, offs), W, stride=S, tail="end")
    wb, wo, _, _, _ = ref.tile(buf, offs, W, S, "end")
    rb = cuda(wb, wo)
    t = (tb.bytes, tb.offsets)
    for f in (lambda x: batch_tokenize_varlen(dna, x),
              lambda x: batch_tokenize_mlm(dna, x, 64, seed=3).labels,
              lambda x: batch_tokenize_kmer(dna, x, 3, 64, stride=2),
              lambda x: revcomp_packed(*x, rc="both").bytes):
        a, r = f(t), f(rb)
        a, r = (a.tokens, r.tokens) if isinstance(a, VarlenBatch) else (a, r)
        assert torch.equal(a, r)


def forms(buf, offs, tmp_path):
    seqs = [bytes(buf[offs[i]:offs[i + 1]]) for i in range(len(offs) - 1)]
    path = tmp_path / "t.ff"
    path.write_bytes(flatfile_image(seqs))
    ff = cbioseq.FlatFile(str(path))
    host = (buf[offs[0]:].copy(), offs - offs[0])
    return [seqs, host, cuda(*host), (ff, 0, len(seqs))]


@pytest.mark.parametrize("rc", [None, "always", "both"])
@pytest.mark.parametrize("varlen", [False, True])
def test_batch_tokenize_tiled_across_forms(rc, varlen, tmp_path):
    dna = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
    buf, offs = batch_of([0, 9, 130, 64, 65, 33], 11)
    W, S = 64, 48
    wb, wo, wsp, wsi, wst = ref.tile(buf, offs, W, S, "short")
    fb, fo = wb, wo
    if rc is not None:
        fb, fo, _ = reference_revcomp(wb, wo, rc, 0.5, 0, 0)
    rows = len(fo) - 1
    if varlen:
        want = batch_tokenize_varlen(dna, cuda(fb, fo)).tokens
    else:
        want = dna.batch_tokenize([bytes(fb[fo[i]:fo[i + 1]]) for i in range(rows)], padlen=W + 2, batch_first=True)
    for form in forms(buf, offs, tmp_path):
        tt = batch_tokenize_tiled(dna, form, W, S, varlen=varlen, rc=rc)
        assert isinstance(tt, TiledTokens) and tt.strands == (2 if rc == "both" else 1) and tt.bos == 1
        got = tt.tokens.tokens if varlen else tt.tokens
        assert torch.equal(got.cpu(), want.cpu())
        assert_same_bits(wsp, tt.seq_ptr.cpu().numpy())
        assert_same_bits(wsi, tt.seq_index.cpu().numpy())
        assert_same_bits(wst, tt.starts.cpu().numpy())
        assert_same_bits(offs - offs[0], tt.seq_offsets.cpu().numpy())
        assert (tt.flipped is None) == (rc is None)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("C", [1, 3, 8, 64, 257])
@pytest.mark.parametrize("varlen", [False, True])
@pytest.mark.parametrize("strands", [1, 2])
def test_untile_against_reference(dtype, C, varlen, strands):
    dna = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
    buf, offs = batch_of([0, 5, 61, 200, 16, 17], 21)
    lens = np.diff(offs)
    for tail in ("short", "end", "drop"):
        W, S = 16, 5
        tt = batch_tokenize_tiled(dna, cuda(buf, offs), W, S, tail=tail, varlen=varlen, rc="both" if strands == 2 else "random",
                                  seed=4)
        rows = tt.seq_index.numel() * strands
        g = torch.Generator(device="cuda").manual_seed(C)
        if varlen:
            y = torch.randn((tt.tokens.tokens.numel(), C), generator=g, device="cuda").to(dtype)
            cu = tt.tokens.cu_seqlens.cpu().numpy().astype(np.int64)
            base = lambda w: int(cu[w])  # noqa: E731
        else:
            y = torch.randn((rows, W + 2, C), generator=g, device="cuda").to(dtype)
            base = lambda w: w * (W + 2)  # noqa: E731
        ub = untile(y if C > 1 else y[..., 0].contiguous(), tt)  # C = 1: the (rows, P) and (T,) forms
        want = ref.untile(y.float().cpu().numpy().reshape(-1, C), lens, W, S, tail, base, 1, strands,
                          tt.flipped.cpu().numpy())
        torch.cuda.synchronize()
        assert ub.values.dtype == torch.float32 and tuple(ub.values.shape) == (int(lens.sum()), C)
        assert_same_bits(want, ub.values.cpu().numpy())
        assert_same_bits(offs - offs[0], ub.offsets.cpu().numpy())


@pytest.mark.parametrize("tail,want", [
    ("short", [0, 0, 0, 0.5, 1, 1, 1.5, 2, 2, 2.5, 3]),
    ("end", [0, 0, 0, 0.5, 1, 1, 1.5, 2.5, 2.5, 2.5, 3]),
    ("drop", [0, 0, 0, 0.5, 1, 1, 1.5, 2, 2, 2, float("nan")]),
])
def test_untile_worked_answers(tail, want):
    dna = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
    tt = batch_tokenize_tiled(dna, ["ACGTACGTACG"], 4, 3, tail=tail)
    M = tt.tokens.shape[0]
    y = torch.arange(M, dtype=torch.float32, device="cuda")[:, None].expand(M, 6).contiguous()
    got = untile(y, tt).values[:, 0].cpu().numpy()
    assert_same_bits(np.array(want, np.float32), got)
    assert_same_bits(np.array(want, np.float32), untile(y, tt, col0=1).values[:, 0].cpu().numpy())


@pytest.mark.parametrize("varlen", [False, True])
def test_round_trip_positions_with_both_strands(varlen):
    # every window's "model output" at each residue is that residue's source position: untile gives every position back
    dna = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
    buf, offs = batch_of([1, 0, 999, 4096, 37, 1500], 31)
    W, S = 256, 100
    tt = batch_tokenize_tiled(dna, cuda(buf, offs), W, S, tail="end", varlen=varlen, rc="both")
    M = tt.seq_index.numel()
    st = torch.cat([tt.starts, tt.starts])
    lens = torch.from_numpy(np.diff(offs)).cuda()
    wl = torch.minimum(lens[torch.cat([tt.seq_index, tt.seq_index])], torch.tensor(W, device="cuda"))
    t = torch.arange(W, device="cuda")[None, :]
    pos = torch.where(tt.flipped[:, None], st[:, None] + wl[:, None] - 1 - t, st[:, None] + t).float()
    if varlen:
        cu = tt.tokens.cu_seqlens.long()
        y = torch.zeros(tt.tokens.tokens.numel(), dtype=torch.float32, device="cuda")
        for w in range(2 * M):
            n = int(wl[w])
            y[cu[w] + 1:cu[w] + 1 + n] = pos[w, :n]
    else:
        y = torch.zeros((2 * M, W + 2), dtype=torch.float32, device="cuda")
        y[:, 1:W + 1] = pos
    got = untile(y, tt).values[:, 0]
    want = torch.cat([torch.arange(int(n), dtype=torch.float32) for n in np.diff(offs)]).cuda()
    assert torch.equal(got, want)


def test_untile_rejects_bad_values():
    dna = cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)
    tt = batch_tokenize_tiled(dna, ["ACGTACGTACG", "AC"], 4, 3)
    M = tt.tokens.shape[0]
    for bad in (torch.zeros((M, 6), dtype=torch.float64, device="cuda"), torch.zeros((M + 1, 6), device="cuda"),
                torch.zeros((M, 4), device="cuda"), torch.zeros((M, 6, 2), device="cuda")[:, :, :1],
                torch.zeros((M, 6)), torch.zeros(M * 6, device="cuda")):
        with pytest.raises(ValueError):
            untile(bad, tt)
    with pytest.raises(ValueError):
        untile(torch.zeros((M, 6), device="cuda"), tt, col0=-1)
