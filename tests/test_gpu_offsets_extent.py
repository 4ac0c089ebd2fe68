"""The offsets reductions of libbsq: the length check, the varlen, crop, k-mer, tile and translate extents.

Each device entry point validates a device-resident offsets array and sizes an output from it in one launch and one
synchronise; the k-mer, tile and translate extents also have a host form.  On the same seeded offsets (empty rows,
one row, just past the 1024 rows of a scan CTA, and more rows than the reduction grid has threads) every host extent
must equal its device extent and the Python reference.  Each validation error is checked alone on the device with its
message, and the totals near and past INT64_MAX (offsets without a residue buffer) with the overflow error of each
extent."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from bioseq_b200 import capi  # noqa: E402
import kmer_reference  # noqa: E402
import tile_reference  # noqa: E402
import translate_reference  # noqa: E402

I64_MAX = 2 ** 63 - 1
SIZES = [1, 1025, 400_000]
SIX = (1, 2, 3, -1, -2, -3)


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests selected but no CUDA device is visible")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _offsets(n, seed, maxlen=300, lead=3):
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, maxlen, n).astype(np.int64)
    lens[rng.random(n) < 0.1] = 0
    return lens, np.concatenate([[lead], lead + np.cumsum(lens)]).astype(np.int64)


def _tok():
    return capi.tokenizer("DNA", bos=True, eos=True)


def _tile_ref(lens, W, S, tail):
    wins = [tile_reference.windows(int(n), W, S, tail) for n in lens]
    return sum(len(w) for w in wins), sum(ln for w in wins for _, ln in w), max((min(int(n), W) for n in lens), default=0)


def _translate_ref(lens, frames, crop_len=I64_MAX):
    L = [translate_reference.frame_len(int(n), f) for n in lens for f in frames]
    return sum(L), sum(min(x, crop_len) for x in L), max((min(x, crop_len) for x in L), default=0)


# name -> (device call (offsets tensor, n, nbytes) -> extent, host call (offsets array, n) -> extent or None, reference(lens))
KM = dict(k=3, stride=2, tail=capi.KMER_SINGLE)
EXTENTS = {
    "varlen": (lambda o, n, nb: capi.varlen_extent_device(0, _stream(), o, n, _tok(), nbytes=nb), None,
               lambda lens: (int(lens.sum()) + 2 * lens.size, int(lens.max()) + 2)),
    "crop": (lambda o, n, nb: capi.crop_extent_device(0, _stream(), o, n, 100, nbytes=nb), None,
             lambda lens: (int(np.minimum(lens, 100).sum()), int(np.minimum(lens, 100).max()))),
    "kmer": (lambda o, n, nb: capi.kmer_extent_device(0, _stream(), o, n, capi.kmer_desc(_tok(), **KM), nbytes=nb),
             lambda h, n: capi.kmer_extent_host(h, n, capi.kmer_desc(_tok(), **KM)),
             lambda lens: (int(kmer_reference.count(lens, 3, 2, True, 1, 1).sum()), int(kmer_reference.count(lens, 3, 2, True, 1, 1).max()))),
    "tile": (lambda o, n, nb: capi.tile_extent_device(0, _stream(), o, n, 64, 24, capi.TILE_SHORT, nbytes=nb),
             lambda h, n: capi.tile_extent_host(h, n, 64, 24, capi.TILE_SHORT),
             lambda lens: _tile_ref(lens, 64, 24, "short")),
    "translate": (lambda o, n, nb: capi.translate_extent_device(0, _stream(), o, n, SIX, 40, nbytes=nb),
                  lambda h, n: capi.translate_extent_host(h, n, SIX, 40),
                  lambda lens: _translate_ref(lens, SIX, 40)),
}


def _check_lengths(o, n, nb, padlen):
    capi.check_lengths_device(0, _stream(), o, n, padlen, _tok(), nbytes=nb)


def _launches(fn):
    capi.lib().bsq_launch_count_reset()
    out = fn()
    return out, capi.lib().bsq_launch_count()


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("name", sorted(EXTENTS))
def test_extent_matches_host_and_reference(name, n):
    device, host, reference = EXTENTS[name]
    lens, offs = _offsets(n, seed=n + len(name))
    o = torch.from_numpy(offs).cuda()
    got, launches = _launches(lambda: device(o, n, int(offs[-1])))
    assert launches == 1
    assert got == reference(lens)
    if host is not None:
        assert host(offs, n) == got


@pytest.mark.parametrize("n", SIZES)
def test_check_lengths_finds_the_longest_row(n):
    lens, offs = _offsets(n, seed=n)
    o = torch.from_numpy(offs).cuda()
    longest = int(lens.max()) + 2  # with BOS and EOS
    _, launches = _launches(lambda: _check_lengths(o, n, int(offs[-1]), longest))
    assert launches == 1
    with pytest.raises(RuntimeError, match=f"seq len \\+ bos \\+ eos > padlen: {longest}, vs padlen {longest - 1}"):
        _check_lengths(o, n, int(offs[-1]), longest - 1)


def _bad(kind, n):
    """(offsets, nbytes) wrong in one way only."""
    _, offs = _offsets(n, seed=5)
    nbytes = int(offs[-1])
    if kind == "decreasing":
        i = n // 2
        offs[i] = offs[i + 1] + 1
    elif kind == "negative start":
        offs[0] = -1
    else:
        nbytes -= 1
    return offs, nbytes


MESSAGES = {"decreasing": "offsets must be non-decreasing", "negative start": "offsets must start at or after 0",
            "past the end": "offsets run past the end of bytes"}


@pytest.mark.parametrize("n", [3, 400_000])
@pytest.mark.parametrize("kind", sorted(MESSAGES))
@pytest.mark.parametrize("name", sorted(EXTENTS) + ["check_lengths"])
def test_each_error_alone(name, kind, n):
    offs, nbytes = _bad(kind, n)
    o = torch.from_numpy(offs).cuda()
    call = (lambda: _check_lengths(o, n, nbytes, 1 << 30)) if name == "check_lengths" else (lambda: EXTENTS[name][0](o, n, nbytes))
    capi.lib().bsq_launch_count_reset()
    with pytest.raises(ValueError, match=MESSAGES[kind]):
        call()
    assert capi.lib().bsq_launch_count() == 1


def _spread(lens, n, stride):
    """offsets of n rows, all empty but rows 0, stride, 2 * stride, ... which take `lens` in turn."""
    full = np.zeros(n, np.int64)
    full[np.arange(len(lens)) * stride] = lens
    return np.concatenate([[0], np.cumsum(full)]).astype(np.int64)


def _grid_threads():
    return torch.cuda.get_device_properties(0).multi_processor_count * 8 * 256


def _placements():
    """(n, stride): big rows in one warp, in different warps, in different CTAs, and in the same thread of the grid."""
    g = _grid_threads()
    return [(2, 1), (200, 100), (6000, 3000), (g + 10, g)]


def _device(o, n, name, *args):
    return getattr(capi, name + "_extent_device")(0, _stream(), torch.from_numpy(o).cuda(), n, *args)


@pytest.mark.parametrize("place", range(4))
def test_tile_near_and_past_int64_max(place):
    n, stride = _placements()[place]
    one = _spread([2 ** 62 + 12345], n, stride)
    for S in (1000, 999, 600):
        for tail in (capi.TILE_SHORT, capi.TILE_END, capi.TILE_DROP):
            assert _device(one, n, "tile", 1000, S, tail) == capi.tile_extent_host(one, n, 1000, S, tail)
    for tail in (capi.TILE_SHORT, capi.TILE_END, capi.TILE_DROP):
        with pytest.raises(ValueError, match="the windows' count or bytes exceed INT64_MAX"):
            _device(one, n, "tile", 1000, 7, tail)
    # an empty sequence is one window of no bytes: exactly INT64_MAX windows fit
    big = _spread([2 ** 62, 2 ** 62 - 1 - (n - 2)], n, stride)
    want = (I64_MAX, I64_MAX - (n - 2), 1)
    assert _device(big, n, "tile", 1, 1, capi.TILE_SHORT) == want == capi.tile_extent_host(big, n, 1, 1, capi.TILE_SHORT)
    with pytest.raises(ValueError, match="the windows' count or bytes exceed INT64_MAX"):
        _device(big, n, "tile", 2, 1, capi.TILE_SHORT)


@pytest.mark.parametrize("place", range(4))
def test_translate_near_and_past_int64_max(place):
    n, stride = _placements()[place]
    big = _spread([2 ** 62, 2 ** 62 - 1], n, stride)
    want = ((2 ** 62) // 3 + (2 ** 62 - 1) // 3,) * 2 + ((2 ** 62) // 3,)
    assert _device(big, n, "translate", (1,)) == want == capi.translate_extent_host(big, n, (1,))
    with pytest.raises(ValueError, match="the translated batch exceeds INT64_MAX bytes"):
        _device(big, n, "translate", SIX)


@pytest.mark.parametrize("place", range(4))
def test_kmer_near_int64_max(place):
    n, stride = _placements()[place]
    km = capi.kmer_desc(_tok(), 1)  # T(len) = len + 2, so an empty row is BOS and EOS
    fits = _spread([2 ** 62, 2 ** 62 - 5 - 2 * (n - 2)], n, stride)  # exactly INT64_MAX tokens
    assert _device(fits, n, "kmer", km) == (I64_MAX, 2 ** 62 + 2) == capi.kmer_extent_host(fits, n, km)


@pytest.mark.parametrize("place", range(4))
def test_kmer_past_int64_max(place):
    """A k-mer total past INT64_MAX is an error, as the tile and translate extents' are."""
    n, stride = _placements()[place]
    km = capi.kmer_desc(_tok(), 1)
    for lens in ([2 ** 62, 2 ** 62 - 1], [I64_MAX]):  # 2^63 + 3 tokens; one row of 2^63 + 1
        over = _spread(lens, n, stride)
        for call in (lambda: _device(over, n, "kmer", km), lambda: capi.kmer_extent_host(over, n, km)):
            with pytest.raises(ValueError, match="the k-mer tokens exceed INT64_MAX"):
                call()
