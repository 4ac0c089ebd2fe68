"""The span kernel's tile schedule at its edges, bit for bit against the oracle.

Every CTA of the span kernel (tokenize_span_kernel, padlen >= 257) takes two static tiles, blockIdx.x and
blockIdx.x + G (G = gridDim.x = SMs x 4 CTAs of tiles of at most 1536 16-byte vectors), before it asks the
per-stream atomic counter for more; the host sizes the tiles so that the tile count fills whole rounds of G.  The cases
below sit on the boundaries of that schedule: fewer tiles than CTAs, exactly one round, between one and two rounds, just
past two, several batches in one launch, launches that overwrite one buffer back to back (also inside a CUDA graph, where
the kernel uses its static order), and concurrent streams that all reach their counters."""
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from bioseq_b200 import capi  # noqa: E402
from oracle.oracle import OracleTokenizer  # noqa: E402
from helpers import assert_same_bits, gen  # noqa: E402

MIX = b"ACDEFGHIKLMNPQRSTVWYacdefghiklmnpqrstvwyXBZOUJ*-NnUu .\x00\x7f\x80\xc3\xff"
VT = 1536             # vectors of a full tile (kSpanTileVecs in bsq_span.cu)
CTAS_PER_SM = 4      # span kernel CTAs per SM at that tile size


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests selected but no CUDA device is visible")


def grid():
    return torch.cuda.get_device_properties(0).multi_processor_count * CTAS_PER_SM


def round_rows(padlen, rounds=1):
    """Rows whose output is `rounds` whole rounds of full tiles."""
    return rounds * grid() * VT * 16 // padlen


def toks(flags):
    bos, eos, pad = flags
    return (capi.tokenizer("PROTEIN", bos=bos, eos=eos, padchar=pad),
            OracleTokenizer("PROTEIN", bos=bos, eos=eos, padchar=pad))


def batch(seed, n, padlen):
    buf, offs = gen(seed, n, 0, padlen - 2, MIX)
    return buf, offs, torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda()


def run_one(n, padlen, flags=(True, True, True), seed=0):
    tok, orc = toks(flags)
    buf, offs, d_b, d_o = batch(seed, n, padlen)
    out = torch.full((n, padlen), 0xAB, dtype=torch.uint8, device="cuda")
    capi.tokenize(0, torch.cuda.current_stream().cuda_stream, d_b, d_o, n, padlen, tok, True, 0, out)
    torch.cuda.synchronize()
    assert_same_bits(orc.batch_tokenize((buf, offs), padlen=padlen, destchar="B", batch_first=True), out.cpu().numpy())


def test_fewer_tiles_than_ctas():
    # 100 rows: a few 256-vector tiles, no second static tile and no counter tile for any CTA
    run_one(100, 1024, seed=1)
    run_one(7, 1024, seed=2)


@pytest.mark.parametrize("rounds,extra", [(1, 0), (1, 500), (2, 0), (2, 100), (3, 0)])
def test_round_boundaries(rounds, extra):
    # (1, 0): exactly G tiles, no second static tile; (1, 500): between one and two rounds, some CTAs take a second static
    # tile and none reaches the counter; (2, 0): both static tiles everywhere; (2, 100): just past two rounds, the first
    # counter tiles; (3, 0): a whole round from the counter
    run_one(round_rows(1024, rounds) + extra, 1024, seed=10 * rounds + extra)


@pytest.mark.parametrize("padlen", [1024, 1026, 652])
@pytest.mark.parametrize("flags", [(True, True, True), (False, False, False), (True, False, True), (False, True, False)])
def test_padlens_and_specials(padlen, flags):
    # several rounds: both static tiles and counter tiles
    run_one(round_rows(padlen, 3) + 12345, padlen, flags, seed=padlen)


@pytest.mark.parametrize("first", [300, "round"])
def test_many_batches(first):
    # bsq_tokenize_many numbers the tiles one batch after the other: static and counter tiles fall across batch edges
    tok, orc = toks((True, True, True))
    padlen = 1024
    n0 = first if first != "round" else round_rows(padlen) + 777
    sizes = [n0, 5000, 1, 30000, 2500]
    work, calls = [], []
    for k, n in enumerate(sizes):
        buf, offs, d_b, d_o = batch(50 + k, n, padlen)
        out = torch.full((n, padlen), 0xCD, dtype=torch.uint8, device="cuda")
        work.append((buf, offs, out))
        calls.append((d_b, d_o, n, out))
    capi.tokenize_many(0, torch.cuda.current_stream().cuda_stream, calls, padlen, tok, True, 0)
    torch.cuda.synchronize()
    for buf, offs, out in work:
        assert_same_bits(orc.batch_tokenize((buf, offs), padlen=padlen, destchar="B", batch_first=True), out.cpu().numpy())


def _alternating_launches(st, tok, inputs, out, n, padlen, count):
    for i in range(count):
        d_b, d_o = inputs[i % 2]
        capi.tokenize(0, st, d_b, d_o, n, padlen, tok, True, 0, out)


def test_back_to_back_launches_into_one_buffer_last_wins():
    # 50 dependent launches on one stream write the same output; each must start its stores only after the previous
    # one has finished, so the last input's tokens are what remains
    tok, orc = toks((True, True, True))
    n, padlen = 20000, 1024
    a = batch(60, n, padlen)
    b = batch(61, n, padlen)
    out = torch.zeros((n, padlen), dtype=torch.uint8, device="cuda")
    _alternating_launches(torch.cuda.current_stream().cuda_stream, tok, [(a[2], a[3]), (b[2], b[3])], out, n, padlen, 50)
    torch.cuda.synchronize()
    assert_same_bits(orc.batch_tokenize((b[0], b[1]), padlen=padlen, destchar="B", batch_first=True), out.cpu().numpy())


def test_back_to_back_launches_into_one_buffer_in_a_cuda_graph():
    # the same 50 launches captured once (the kernel uses its static tile order under capture) and replayed twice
    tok, orc = toks((True, True, True))
    n, padlen = 20000, 1024
    a = batch(62, n, padlen)
    b = batch(63, n, padlen)
    out = torch.zeros((n, padlen), dtype=torch.uint8, device="cuda")
    want_a = orc.batch_tokenize((a[0], a[1]), padlen=padlen, destchar="B", batch_first=True)
    want_b = orc.batch_tokenize((b[0], b[1]), padlen=padlen, destchar="B", batch_first=True)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        # 49 launches: the capture ends on input a, so a replay is told apart from the direct launch below
        _alternating_launches(torch.cuda.current_stream().cuda_stream, tok, [(a[2], a[3]), (b[2], b[3])], out, n, padlen, 49)
    for _ in range(2):
        out.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert_same_bits(want_a, out.cpu().numpy())
        capi.tokenize(0, torch.cuda.current_stream().cuda_stream, b[2], b[3], n, padlen, tok, True, 0, out)
        torch.cuda.synchronize()
        assert_same_bits(want_b, out.cpu().numpy())


def test_concurrent_streams_past_the_static_tiles():
    # four streams, six launches back to back on each, every batch large enough that its CTAs take counter tiles
    tok, orc = toks((True, True, True))
    streams = [torch.cuda.Stream() for _ in range(4)]
    work = []
    for k, padlen in enumerate((1024, 1026, 652, 2048)):
        n = round_rows(padlen, 2) + 1000 * (k + 1)
        buf, offs, d_b, d_o = batch(7800 + k, n, padlen)
        want = orc.batch_tokenize((buf, offs), padlen=padlen, destchar="B", batch_first=True)
        work.append((d_b, d_o, n, padlen, want, [torch.zeros((n, padlen), dtype=torch.uint8, device="cuda") for _ in range(6)]))
    torch.cuda.synchronize()
    for rep in range(6):
        for s, (d_b, d_o, n, padlen, _, outs) in zip(streams, work):
            capi.tokenize(0, s.cuda_stream, d_b, d_o, n, padlen, tok, True, 0, outs[rep])
    torch.cuda.synchronize()
    for d_b, d_o, n, padlen, want, outs in work:
        for o in outs:
            assert_same_bits(want, o.cpu().numpy())
