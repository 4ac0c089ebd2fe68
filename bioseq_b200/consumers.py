"""Consumers fused onto the tokeniser and on-device BLOSUM62 augmentation (SURVEY.md 8(f) rows 3-4).

Reference counterparts:

* ``batch_onehot_encode_bcl`` -- ``einops.rearrange(torch.from_numpy(tok.batch_onehot_encode(seqs, padlen)).to(dev),
  "length batch emb -> batch emb length").float()`` (bioseq/loaders.py:74-75, :93-94): one kernel writes the
  ``(batch, emb, length)`` tensor directly instead of one-hot + transpose + cast (three full-tensor passes).
* ``batch_embed`` -- ``embedding(torch.from_numpy(tok.batch_tokenize(seqs, padlen, batch_first=...)).to(dev).long())``
  with ``embedding = bioseq.make_embedding(tok, dim)`` (bioseq/__init__.py:171-188): the token tensor is never
  materialised, the kernel writes embedding rows.
* ``augment_packed`` -- ``bioseq.blosum.augment_seq`` (bioseq/blosum.py:63-87) applied to each sequence of a packed
  batch on the device (the reference mutates Python strings one by one, bioseq/loaders.py:71-73).
* ``batch_tokenize_varlen`` -- the tokens of ``batch_tokenize(..., batch_first=True)`` without their padding, as one
  packed stream plus int32 ``cu_seqlens`` (what varlen attention takes), written by one kernel instead of padded
  tokenize + mask + ``out[mask]``.
* ``batch_tokenize_mlm`` -- a masked-language-model batch (the objective of ``training/cnnpretrain.py:119-125``; BERT /
  ESM pretraining): masked input tokens and ``cross_entropy``-ready int64 labels, padded or padding-free, written by
  one kernel instead of tokenize + the HuggingFace-collator recipe in torch (rand, where, index_put, casts).
* ``batch_tokenize_seqpack`` -- sequence packing: whole sequences best-fit into fixed-width ``(rows, L)`` rows with
  position ids that restart per sequence and ``cu_seqlens`` (optionally MLM inputs and labels), written by one kernel
  from a host plan instead of varlen tokenize + a torch scatter + ``repeat_interleave`` position ids.
* ``crop_packed`` / ``crop=`` -- every sequence cropped to a window of the model's context on the device (ESM-style
  seeded random windows, or the heads as HF ``truncation=True`` does) instead of slicing Python strings or gathering
  in torch; the consumers above take ``crop=`` and ``crop_len=`` and run unchanged on the cropped batch.
* ``revcomp_packed`` / ``rc=`` -- the reverse complement of every DNA / RNA sequence on the device (seeded strand flips
  for training, both strands for test-time averaging) instead of flipping Python strings or gathering in torch; every
  consumer takes ``rc=`` and ``rc_prob=`` and runs unchanged on the flipped batch.
* ``tile_packed`` / ``batch_tokenize_tiled`` / ``untile`` -- every window of every sequence at a stride (inference over
  whole long sequences, chunked datasets) on the device instead of slicing Python strings or a ragged gather in torch,
  and the per-residue mean of the model's window outputs stitched back deterministically instead of ``index_add_`` and
  counts.

All of these call the C ABI (``include/bsq.h``) through ``capi``; torch supplies memory and the stream.
A *batch* is one of

* ``(bytes, offsets)`` -- uint8 residues + int64 offsets, both torch CUDA tensors (used in place) or both host
  arrays (numpy / torch CPU, pinned or pageable: staged to the device by the stager),
* ``(flatfile, start, stop)`` -- a range of a ``cbioseq.FlatFile`` (its packed form goes to the device as is),
* a list/tuple of ``str`` / ``bytes`` / ``bytearray`` (packed into pinned memory first, like ``batch_tokenize``).
"""
import collections
import math
import operator
import threading

import numpy as np

from . import capi
from . import cbioseq

_DTYPES = None
_ctx = {}
_ctx_lock = threading.Lock()
_desc_cache = {}


def _torch():
    import torch
    return torch


def _dtype_of(destchar):
    global _DTYPES
    torch = _torch()
    if _DTYPES is None:
        _DTYPES = {"B": torch.uint8, "b": torch.int8, "h": torch.int16, "i": torch.int32, "l": torch.int64, "q": torch.int64,
                   "f": torch.float32, "d": torch.float64}
    kind = capi.kind_of(destchar)
    c = destchar[0]
    return kind, _DTYPES[c if c in ("B", "b") else c.lower()]


def descriptor(tokenizer):
    """``struct bsq_tokenizer`` of a ``cbioseq.Tokenizer`` (cached)."""
    if isinstance(tokenizer, capi.TokenizerDesc):
        return tokenizer
    key = (tokenizer.key, bool(tokenizer.includes_eos()), bool(tokenizer.includes_bos()), bool(tokenizer.is_padded()))
    d = _desc_cache.get(key)
    if d is None:
        d = _desc_cache[key] = capi.tokenizer(key[0], eos=key[1], bos=key[2], padchar=key[3])
    return d


class _DeviceCtx:
    def __init__(self, device):
        self.lock = threading.Lock()
        self.stager = capi.Stager(device)
        self.pack = None


def _device_ctx(device):
    with _ctx_lock:
        c = _ctx.get(device)
        if c is None:
            c = _ctx[device] = _DeviceCtx(device)
        return c


def _resolve_device(device):
    torch = _torch()
    if not torch.cuda.is_available():
        raise RuntimeError("bioseq_b200: no CUDA device -- there is no CPU fallback")
    if device is None:
        return torch.cuda.current_device()
    d = torch.device(device)
    if d.type != "cuda":
        raise ValueError("bioseq_b200 produces CUDA tensors; device must be a CUDA device")
    return torch.cuda.current_device() if d.index is None else d.index


class _Resolved:
    """Device pointers of a batch plus what is needed to validate and release it."""
    __slots__ = ("device", "stream", "d_bytes", "d_offs", "nseq", "h_offs", "keep", "ctx", "base", "extent")

    def release(self):
        if self.ctx is not None:
            self.ctx.stager.release(self.stream)
            self.ctx.lock.release()
            self.ctx = None


_Batch = collections.namedtuple("_Batch", ["bytes", "offsets", "keep"])


def _parse(batch):
    """-> _Batch: checked CUDA tensors (``offsets`` is a torch tensor), checked host numpy arrays (``keep``: the FlatFile
    they view), or ``bytes`` None and ``offsets`` the items as ``bytes``, gathered when the batch is staged.  The
    offsets of a CUDA batch are validated on the device, by the reduction that sizes or checks it."""
    torch = _torch()
    keep = None
    if isinstance(batch, tuple) and len(batch) == 3 and isinstance(batch[0], cbioseq.FlatFile):
        keep = batch[0]
        b, o = keep.packed(batch[1], batch[2])
    elif isinstance(batch, tuple) and len(batch) == 2 and hasattr(batch[0], "dtype"):
        b, o = batch
        if isinstance(b, torch.Tensor) and b.is_cuda:
            if not (isinstance(o, torch.Tensor) and o.is_cuda and o.device == b.device):
                raise ValueError("bytes and offsets must live on the same side (all host or all CUDA)")
            ok = b.dtype == torch.uint8 and o.dtype == torch.int64 and b.is_contiguous() and o.is_contiguous()
        else:
            b = b.numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
            o = o.numpy() if isinstance(o, torch.Tensor) else np.asarray(o)
            ok = b.dtype == np.uint8 and o.dtype == np.int64 and b.flags.c_contiguous and o.flags.c_contiguous
        if not ok:
            raise ValueError("packed batch: contiguous uint8 bytes and int64 offsets expected")
        if isinstance(o, torch.Tensor):
            return _Batch(b, o, None)
    else:  # list of str / bytes / bytearray (any other batch fails as an item)
        items = []
        for s in (batch if isinstance(batch, (list, tuple)) else [None]):
            if isinstance(s, str):
                s = s.encode("utf-8")
            elif not isinstance(s, (bytes, bytearray)):
                raise ValueError("item was none of string, bytes, or numpy array of 8-bit integers. ")
            items.append(s)
        return _Batch(None, items, None)
    _nseq(o, b.size)
    return _Batch(b, o, keep)


def _nseq(offsets, nbytes=None):
    """The number of sequences ``offsets`` (numpy or torch) delimit; with ``nbytes`` (host offsets), they must end
    within that many bytes."""
    n = (offsets.numel() if isinstance(offsets, _torch().Tensor) else offsets.size) - 1
    if n < 0:
        raise ValueError("offsets needs at least one entry")
    if nbytes is not None and n > 0 and int(offsets[n]) > nbytes:
        raise ValueError("offsets run past the end of bytes")
    return n


def _packed_cuda(name, bytes_cuda, offsets_cuda):
    """Check the packed CUDA batch of entry point ``name``."""
    torch = _torch()
    if not (isinstance(bytes_cuda, torch.Tensor) and bytes_cuda.is_cuda and bytes_cuda.dtype == torch.uint8 and
            isinstance(offsets_cuda, torch.Tensor) and offsets_cuda.is_cuda and offsets_cuda.dtype == torch.int64 and
            bytes_cuda.device == offsets_cuda.device and bytes_cuda.is_contiguous() and offsets_cuda.is_contiguous()):
        raise ValueError(f"{name}: contiguous uint8 bytes and int64 offsets CUDA tensors on one device expected")


def _resolve(batch, device, augment=None, before_stage=None, crop=None, rc=None, checked=None, translate=None):
    """-> _Resolved of a batch (or of its ``_parse``), in these steps: size the translation, crop and flip,
    ``before_stage``, stage (or use in place), translate, crop, augment, flip.

    Host batches are staged; CUDA batches are used in place (with ``augment`` and no crop or translation: a clone).
    ``before_stage(host_offsets, n)`` checks a host batch before anything is copied to the device.  ``translate`` (from
    ``_translate_spec``): the batch is translated into fresh device buffers, n F protein sequences.  ``crop`` (from
    ``_crop_spec``): the batch is cropped into fresh device buffers.  ``augment``: BLOSUM62 mutations, by the stager's
    copy of an uncropped, untranslated host batch, else in place on the device.  ``rc`` (from ``_rc_spec``): the batch is
    then flipped into fresh device buffers (``_apply_rc``); ``"both"`` doubles it.

    With a translation, crop or flip the result has ``extent = (sum, max)`` of its lengths, and ``before_stage`` and
    ``h_offs`` see the translated, cropped and flipped offsets from 0.  Host batches are sized from their host offsets;
    CUDA batches pay one ``bsq_crop_extent_device`` or ``bsq_translate_extent_device`` (which also validates their
    offsets), unless ``checked`` says the caller has validated them already: it is then their ``(sum, max)`` after the
    crop (``(sum, max, translated bytes)`` with ``translate``), or True when the caller has no such extent."""
    torch = _torch()
    p = batch if isinstance(batch, _Batch) else _parse(batch)
    cuda = isinstance(p.offsets, torch.Tensor)
    sized = crop is not None or rc is not None or translate is not None
    crop_len = crop[1] if crop is not None else _UNCROPPED
    r = _Resolved()
    r.ctx, r.keep, r.h_offs, r.base, r.extent = None, [p], None, 0, None
    tr_total = None
    ctx = None
    if cuda:
        b, o = p.bytes, p.offsets
        r.device = b.device.index
        r.stream = torch.cuda.current_stream(r.device).cuda_stream
        if sized and checked is None and translate is not None:
            tr_total, kept, longest = capi.translate_extent_device(r.device, r.stream, o, o.numel() - 1, translate[0], crop_len,
                                                                   nbytes=b.numel())
            r.extent = (kept, longest)
        elif sized and checked is None:
            r.extent = capi.crop_extent_device(r.device, r.stream, o, o.numel() - 1, crop_len, nbytes=b.numel())
        elif sized and checked is not True:
            r.extent = tuple(checked[:2])
            tr_total = checked[2] if translate is not None else None
        if augment and crop is None and translate is None:
            with torch.cuda.device(r.device):
                b = b.clone()  # never mutate the caller's residues
            r.keep.append(b)
        r.d_bytes, r.d_offs, r.nseq = b.data_ptr(), o.data_ptr(), o.numel() - 1
    else:
        r.device = _resolve_device(device)
        r.stream = torch.cuda.current_stream(r.device).cuda_stream
        ctx = _device_ctx(r.device)
        ctx.lock.acquire()
    try:
        if not cuda:
            if p.bytes is None:
                if ctx.pack is None:
                    ctx.pack = capi.Pack(pinned=True)
                ctx.stager.sync_copies()  # the pinned pack buffer may still be in flight
                ctx.pack.gather(p.offsets, nthreads=4)
                n = ctx.pack.nseq
                hb_ptr = ctx.pack.bytes_ptr or 0
                h = np.ctypeslib.as_array(capi.C.cast(ctx.pack.offsets_ptr, capi.C.POINTER(capi.C.c_int64)), shape=(n + 1,))
            else:
                n, hb_ptr, h = p.offsets.size - 1, p.bytes.ctypes.data, p.offsets
            if sized:
                r.h_offs, r.extent, tr_total = _sized_host(h, n, crop_len, translate)
            else:
                r.h_offs, r.base = h, int(h[0])
            if before_stage is not None:
                before_stage(*_rc_host_offsets(r.h_offs, n * len(translate[0]) if translate is not None else n, rc))
            stager_augment = augment and crop is None and translate is None
            if stager_augment:
                ctx.stager.set_augment(*augment)
            try:
                r.d_bytes, r.d_offs = ctx.stager.stage(r.stream, hb_ptr, h.ctypes.data, n)
            finally:
                if stager_augment:
                    ctx.stager.set_augment(0)
            r.nseq, r.ctx = n, ctx
        if translate is not None:
            _apply_translate(r, translate, tr_total)
        if crop is not None:
            _apply_crop(r, crop)
        if augment and (cuda or crop is not None or translate is not None):
            capi.augment_blosum62(r.device, r.stream, r.d_bytes, r.d_offs, r.nseq, *augment)
        if rc is not None:
            _apply_rc(r, rc, r.extent[0] if r.extent is not None else p.bytes.numel())
    except BaseException:
        if ctx is not None:
            ctx.lock.release()
        raise
    return r


def _check_lengths(r, padlen, tok, onehot):
    if r.extent is not None:  # cropped or flipped: the offsets are validated and the longest length is known
        capi.check_lengths_host(np.array([0, r.extent[1]], np.int64), 1, padlen, tok, onehot=onehot)
        return
    if r.h_offs is not None:
        capi.check_lengths_host(r.h_offs, r.nseq, padlen, tok, onehot=onehot)
    else:
        capi.check_lengths_device(r.device, r.stream, r.d_offs, r.nseq, padlen, tok, onehot=onehot)


def _default_padlen(batch, tokenizer, padlen):
    if padlen is not None and padlen > 0:
        return int(padlen)
    if isinstance(batch, tuple) and len(batch) == 3 and isinstance(batch[0], cbioseq.FlatFile):
        return int(batch[0].maxseqlen + tokenizer.includes_bos() + tokenizer.includes_eos())
    raise ValueError("batch tokenize requires padlen is provded.")  # src/tokenize.h:383


def _padlen(name, padlen, varlen, default=None):
    """``padlen`` of a consumer that writes padded or padding-free output: None or -1 give ``default``, anything else
    must be an integer; with ``varlen`` (no padding is written) None, and giving one is an error."""
    if varlen:
        if padlen is not None and padlen != -1:
            raise ValueError(f"{name}(varlen=True) writes no padding: padlen must not be given")
        return None
    if padlen is None or padlen == -1:
        return default
    try:
        return operator.index(padlen)
    except TypeError:
        raise ValueError("padlen must be an integer") from None


def _augment_args(augment, augment_frac, seed, seq_index_base):
    if not augment:
        return None
    return (int(augment), float(augment_frac), int(seed), int(seq_index_base))


_CROP_MODES = (None, "head", "random")


def _crop_spec(crop, crop_len, seed, seq_index_base, max_len=None):
    """Validate the crop arguments (ValueError before anything is staged) -> None (no crop) or
    ``(random, crop_len, seed, seq_index_base)``.  ``max_len``: the residues a padded row holds (``padlen - bos -
    eos``), which is also the default ``crop_len``; None for padding-free output, where ``crop_len`` is required."""
    if crop not in _CROP_MODES:
        raise ValueError(f"crop must be one of None, 'head', 'random', got {crop!r}")
    if crop is None:
        if crop_len is not None:
            raise ValueError("crop_len is given without crop: pass crop='head' or crop='random'")
        return None
    if crop_len is None:
        if max_len is None:
            raise ValueError("padding-free output needs an explicit crop_len")
        crop_len = max_len
    try:
        crop_len = operator.index(crop_len)
    except TypeError:
        raise ValueError("crop_len must be an integer") from None
    if crop_len < 1:
        raise ValueError(f"crop_len must be >= 1, got {crop_len}")
    if max_len is not None and crop_len > max_len:
        raise ValueError(f"crop_len {crop_len} does not fit a row: padlen - bos - eos = {max_len}")
    return (crop == "random", int(crop_len), int(seed), int(seq_index_base))


def _crop_host_extent(h_offs, n, crop_len):
    """-> (cropped offsets from 0, (sum, max) of the cropped lengths) of host offsets, in numpy; ValueError on offsets
    the crop must not index with."""
    o = np.asarray(h_offs[:n + 1], dtype=np.int64)
    lens = np.diff(o)
    if n > 0 and (int(o[0]) < 0 or int(lens.min()) < 0):
        raise ValueError("offsets must start at or after 0 and be non-decreasing")
    kept = np.minimum(lens, crop_len)
    out = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(kept, out=out[1:])
    return out, (int(out[n]), int(kept.max()) if n > 0 else 0)


def _apply_crop(r, crop):
    """Crop the resolved batch into fresh device buffers (r.extent already holds their size); r then describes the
    cropped batch."""
    torch = _torch()
    random, crop_len, seed, base = crop
    dev = torch.device("cuda", r.device)
    out_b = torch.empty(max(r.extent[0], 1), dtype=torch.uint8, device=dev)  # (never a null pointer)
    out_o = torch.empty(r.nseq + 1, dtype=torch.int64, device=dev)
    # an all-empty batch may have no residue buffer at all; nothing is read from it then
    capi.crop(r.device, r.stream, r.d_bytes or out_b, r.d_offs, r.nseq, crop_len, random, seed, base, out_b, out_o)
    r.keep += [out_b, out_o]
    r.d_bytes, r.d_offs, r.base = out_b.data_ptr(), out_o.data_ptr(), 0


_RC_MODES = {None: None, "always": capi.RC_ALWAYS, "random": capi.RC_RANDOM, "both": capi.RC_BOTH}
# the nucleotide alphabets: the complement table is meaningless for protein codes and raw bytes
_RC_KEYS = ("DNA", "DNA4", "DNA5", "DNAMETH", "C", "KETO", "PURPYR")
_UNCROPPED = (1 << 63) - 1  # a window no sequence exceeds: bsq_crop_extent_device then only validates and measures


def _rc_spec(rc, rc_prob, seed, seq_index_base, tokenizer=None, augment=None, mlm=False):
    """Validate the reverse-complement arguments (ValueError before anything is staged) -> None (no flip) or
    ``(mode, rc_prob, seed, seq_index_base)``.  ``tokenizer`` (None for ``revcomp_packed``) must be nucleotide; ``augment``
    (BLOSUM62, for proteins) and ``rc="both"`` with ``mlm`` are rejected."""
    if not isinstance(rc, (str, type(None))) or rc not in _RC_MODES:
        raise ValueError(f"rc must be one of None, 'always', 'random', 'both', got {rc!r}")
    if rc_prob is not None and rc != "random":
        raise ValueError("rc_prob is given without rc='random'")
    if rc is None:
        return None
    if rc == "random":
        try:
            rc_prob = float(0.5 if rc_prob is None else rc_prob)
        except (TypeError, ValueError):
            raise ValueError(f"rc_prob must be a number in [0, 1], got {rc_prob!r}") from None
        if not 0.0 <= rc_prob <= 1.0:
            raise ValueError(f"rc_prob must lie in [0, 1], got {rc_prob}")
    if tokenizer is not None:
        key = descriptor(tokenizer).key.decode("latin-1").upper()
        if key not in _RC_KEYS:
            raise ValueError(f"rc needs a nucleotide tokenizer ({', '.join(_RC_KEYS)}), got {key}")
    if augment:
        raise ValueError("rc cannot be combined with augment: BLOSUM62 substitutions are for proteins")
    if mlm and rc == "both":
        raise ValueError("rc='both' doubles the batch for inference; it cannot be combined with mlm")
    return (_RC_MODES[rc], rc_prob or 0.0, int(seed), int(seq_index_base))


def _rc_host_offsets(h_offs, n, rc):
    """-> (offsets, n) of the batch ``rc`` makes from host offsets that start at 0: the same, or doubled for "both"."""
    if rc is None or rc[0] != capi.RC_BOTH:
        return h_offs, n
    h = np.asarray(h_offs[:n + 1], dtype=np.int64)
    return np.concatenate([h, h[n] + h[1:]]), 2 * n


def _apply_rc(r, rc, nbytes, flipped=False):
    """Flip the resolved batch (validated offsets, ``nbytes`` >= its residues) into fresh device buffers; r then
    describes the flipped batch (doubled for "both").  ``flipped``: return the bool mask of the flipped sequences."""
    torch = _torch()
    mode, rc_prob, seed, base = rc
    m = 2 if mode == capi.RC_BOTH else 1
    dev = torch.device("cuda", r.device)
    out_b = torch.empty(max(nbytes * m, 1), dtype=torch.uint8, device=dev)  # (never a null pointer)
    out_o = torch.empty(r.nseq * m + 1, dtype=torch.int64, device=dev)
    flipped = torch.empty(r.nseq * m, dtype=torch.uint8, device=dev) if flipped else None
    capi.revcomp(r.device, r.stream, r.d_bytes or out_b, r.d_offs, r.nseq, mode, rc_prob, seed, base, out_b, out_o, flipped)
    r.keep += [out_b, out_o]
    if r.h_offs is not None:
        r.h_offs = _rc_host_offsets(np.asarray(r.h_offs, np.int64) - int(r.h_offs[0]), r.nseq, rc)[0]
    r.d_bytes, r.d_offs, r.base, r.nseq = out_b.data_ptr(), out_o.data_ptr(), 0, out_o.numel() - 1
    if m == 2 and r.extent is not None:
        r.extent = (2 * r.extent[0], r.extent[1])
    return None if flipped is None else flipped.view(torch.bool)


_FRAME_SETS = {"forward": (1, 2, 3), "six": (1, 2, 3, -1, -2, -3)}
_GENETIC_CODES = (1, 2, 4, 5, 6, 11)
# the alphabets a translated batch can be tokenized with: the protein and reduced protein codes, and raw bytes
_TRANSLATE_KEYS = ("AMINO", "AMINO20", "PROTEIN", "DAYHOFF", "LIA10", "LIB10", "MURPHY", "SEB6", "SEB8", "SEB10", "SEB14", "SEV10",
                   "BYTES")


def _frames(frames):
    """-> tuple of 1..6 distinct frames from ``frames`` (one of +-1, +-2, +-3, a list / tuple of them, "forward", "six")."""
    if isinstance(frames, str):
        if frames not in _FRAME_SETS:
            raise ValueError(f"frames must be 'forward', 'six', one of +-1, +-2, +-3 or a list of them, got {frames!r}")
        return _FRAME_SETS[frames]
    items = list(frames) if isinstance(frames, (list, tuple)) else [frames]
    out = []
    for f in items:
        try:
            f = operator.index(f)
        except TypeError:
            raise ValueError(f"frames must be integers among +-1, +-2, +-3, got {f!r}") from None
        if f not in (1, 2, 3, -1, -2, -3):
            raise ValueError(f"frames must lie among +-1, +-2, +-3, got {f}")
        if f in out:
            raise ValueError(f"frame {f} is given twice")
        out.append(int(f))
    if not 1 <= len(out) <= 6:
        raise ValueError("frames: 1 to 6 frames expected")
    return tuple(out)


def _genetic_code(code):
    """-> the 64 bytes of a built-in NCBI table id or of a 64-character code string (TCAG order)."""
    if isinstance(code, (str, bytes)):
        b = code.encode("latin-1") if isinstance(code, str) else code
        if len(b) != 64 or not all(0x21 <= x <= 0x7E for x in b):
            raise ValueError("genetic_code: a string of 64 printable ASCII characters (TCAG order) expected")
        return b
    try:
        code = operator.index(code)
    except TypeError:
        raise ValueError(f"genetic_code must be one of {_GENETIC_CODES} or a 64-character string, got {code!r}") from None
    if code not in _GENETIC_CODES:
        raise ValueError(f"genetic_code must be one of {_GENETIC_CODES} or a 64-character string, got {code}")
    return capi.genetic_code(code)


def _translate_spec(translate, genetic_code, tokenizer=None, rc=None, seq_index_base=0):
    """Validate the translation arguments (ValueError before anything is staged) -> None (no translation) or ``(frames,
    code64)``.  ``tokenizer`` (None for ``translate_packed``) must be a protein alphabet or BYTES; ``rc`` must be None (the
    reverse frames are the other strand); ``seq_index_base * F`` must fit int64 (seeded draws use the output index)."""
    if translate is None:
        if not (isinstance(genetic_code, int) and genetic_code == 1):
            raise ValueError("genetic_code is given without translate=")
        return None
    frames, code = _frames(translate), _genetic_code(genetic_code)
    if tokenizer is not None:
        key = descriptor(tokenizer).key.decode("latin-1").upper()
        if key not in _TRANSLATE_KEYS:
            raise ValueError(f"translate= gives proteins: it needs a protein tokenizer or BYTES ({', '.join(_TRANSLATE_KEYS)}), "
                             f"got {key}")
    if rc is not None:
        raise ValueError("rc cannot be combined with translate=: the reverse frames (-1, -2, -3) are the other strand")
    if not _INT64_MIN <= int(seq_index_base) * len(frames) <= _INT64_MAX:
        raise ValueError(f"seq_index_base * frames = {int(seq_index_base) * len(frames)} overflows int64")
    return frames, code


def _out_base(seq_index_base, tr):
    """The global index of a consumer's first output sequence: seeded draws of a translated batch are keyed by
    (seq_index_base + i) * F + f."""
    return seq_index_base if tr is None else int(seq_index_base) * len(tr[0])


def _translate_host_offsets(h_offs, n, frames):
    """-> the translated batch's offsets (n F + 1, from 0) of host offsets, in numpy; ValueError on offsets the kernels
    must not index with."""
    o = np.asarray(h_offs[:n + 1], dtype=np.int64)
    lens = np.diff(o)
    if n > 0 and (int(o[0]) < 0 or int(lens.min()) < 0):
        raise ValueError("offsets must start at or after 0 and be non-decreasing")
    L = np.stack([np.maximum(lens - (abs(f) - 1), 0) // 3 for f in frames], 1)
    out = np.zeros(n * len(frames) + 1, dtype=np.int64)
    np.cumsum(L.reshape(-1), out=out[1:])
    return out


def _sized_host(h_offs, n, crop_len, tr):
    """-> (offsets from 0 of the batch after translation and crop, (sum, max) of its lengths, translated bytes or None) of
    host offsets."""
    if tr is None:
        return (*_crop_host_extent(h_offs, n, crop_len), None)
    t = _translate_host_offsets(h_offs, n, tr[0])
    return (*_crop_host_extent(t, n * len(tr[0]), crop_len), int(t[-1]))


def _apply_translate(r, tr, total):
    """Translate the resolved batch (validated offsets, ``total`` output bytes) into fresh device buffers; r then
    describes the n F protein sequences."""
    torch = _torch()
    frames, code = tr
    dev = torch.device("cuda", r.device)
    out_b = torch.empty(max(total, 1), dtype=torch.uint8, device=dev)  # (never a null pointer)
    out_o = torch.empty(r.nseq * len(frames) + 1, dtype=torch.int64, device=dev)
    # an all-empty batch may have no residue buffer at all; nothing is read from it then
    capi.translate(r.device, r.stream, r.d_bytes or out_b, r.d_offs, r.nseq, frames, code, out_b, out_o)
    r.keep += [out_b, out_o]
    r.d_bytes, r.d_offs, r.base, r.nseq = out_b.data_ptr(), out_o.data_ptr(), 0, out_o.numel() - 1


def _row_residues(tokenizer, padlen):
    return padlen - int(tokenizer.includes_bos()) - int(tokenizer.includes_eos())


def batch_onehot_encode_bcl(tokenizer, batch, padlen=-1, destchar="f", mask=None, device=None, *, augment=0, augment_frac=1.0,
                            seed=0, seq_index_base=0, crop=None, crop_len=None, rc=None, rc_prob=None, translate=None, genetic_code=1):
    """One-hot ``(batch, alphabet_size, padlen)`` tensor (CNN layout), default float32.

    Element ``[i, c, p]`` equals ``batch_onehot_encode(...)[p, i, c]`` (src/tokenize.h:345-368), i.e. the result of the
    reference's rearrange + float (bioseq/loaders.py:74-75).  ``mask``: uint8, one entry per residue of ``bytes``
    (packed batches only, not with ``crop``, ``rc`` or ``translate``).  ``crop``: as ``batch_tokenize_cropped``; ``rc`` /
    ``rc_prob``: as ``batch_tokenize_revcomp``; ``translate`` / ``genetic_code``: as ``batch_tokenize_translated``."""
    torch = _torch()
    tok = descriptor(tokenizer)
    padlen = _default_padlen(batch, tokenizer, padlen)
    kind, dtype = _dtype_of(destchar)
    tr = _translate_spec(translate, genetic_code, tokenizer, rc, seq_index_base)
    if tr is not None and mask is not None:
        raise ValueError("mask covers the nucleotides: it cannot be combined with translate")
    seq_index_base = _out_base(seq_index_base, tr)
    crop = _crop_spec(crop, crop_len, seed, seq_index_base, _row_residues(tokenizer, padlen))
    if crop is not None and mask is not None:
        raise ValueError("mask covers the uncropped residues: it cannot be combined with crop")
    rc = _rc_spec(rc, rc_prob, seed, seq_index_base, tokenizer, augment)
    if rc is not None and mask is not None:
        raise ValueError("mask covers the unflipped residues: it cannot be combined with rc")
    r = _resolve(batch, device, _augment_args(augment, augment_frac, seed, seq_index_base), crop=crop, rc=rc, translate=tr)
    try:
        _check_lengths(r, padlen, tok, onehot=True)
        d_mask = None
        if mask is not None:
            if (isinstance(mask, torch.Tensor) and mask.is_cuda) != (r.h_offs is None):
                raise ValueError("bytes, offsets and mask must live on the same side (all host or all CUDA)")
            if r.h_offs is None:
                m = mask
                d_mask = m.data_ptr()
            else:
                hm = mask.numpy() if isinstance(mask, torch.Tensor) else np.asarray(mask, dtype=np.uint8)
                end = int(r.h_offs[r.nseq])
                if hm.size < end:
                    raise ValueError("mask shorter than bytes")
                m = torch.from_numpy(np.ascontiguousarray(hm[r.base:end])).to(torch.device("cuda", r.device))
                d_mask = m.data_ptr() - r.base
            if m.dtype != torch.uint8:
                raise ValueError("mask must be uint8")
            r.keep.append(m)
        out = torch.empty((r.nseq, tok.alphabet_size, padlen), dtype=dtype, device=torch.device("cuda", r.device))
        capi.onehot_bcl(r.device, r.stream, r.d_bytes, r.d_offs, d_mask, r.nseq, padlen, tok, kind, out)
        return out
    finally:
        r.release()


def batch_embed(tokenizer, batch, weight, padlen=-1, batch_first=True, device=None, *, augment=0, augment_frac=1.0, seed=0,
                seq_index_base=0, crop=None, crop_len=None, rc=None, rc_prob=None, translate=None, genetic_code=1):
    """``weight[tokens]`` for the tokens of ``batch_tokenize(batch, padlen, batch_first=batch_first)`` without
    materialising them: ``(batch, padlen, dim)`` or ``(padlen, batch, dim)``, dtype and device of ``weight``.

    ``weight``: ``(rows >= alphabet_size, dim)`` CUDA tensor (an ``nn.Embedding.weight``); ``dim * itemsize`` must be
    a multiple of 16 bytes.  Forward only (no autograd graph is recorded).  ``crop``: as ``batch_tokenize_cropped``; ``rc`` /
    ``rc_prob``: as ``batch_tokenize_revcomp``; ``translate`` / ``genetic_code``: as ``batch_tokenize_translated``."""
    torch = _torch()
    tok = descriptor(tokenizer)
    padlen = _default_padlen(batch, tokenizer, padlen)
    tr = _translate_spec(translate, genetic_code, tokenizer, rc, seq_index_base)
    seq_index_base = _out_base(seq_index_base, tr)
    crop = _crop_spec(crop, crop_len, seed, seq_index_base, _row_residues(tokenizer, padlen))
    rc = _rc_spec(rc, rc_prob, seed, seq_index_base, tokenizer, augment)
    w = weight.detach()
    if not w.is_cuda or w.dim() != 2:
        raise ValueError("weight must be a 2-D CUDA tensor")
    if not w.is_contiguous():
        w = w.contiguous()
    row_bytes = w.shape[1] * w.element_size()
    r = _resolve(batch, w.device if device is None else device, _augment_args(augment, augment_frac, seed, seq_index_base),
                 crop=crop, rc=rc, translate=tr)
    try:
        if r.device != w.device.index:
            raise ValueError("weight and batch live on different devices")
        _check_lengths(r, padlen, tok, onehot=False)
        shape = (r.nseq, padlen, w.shape[1]) if batch_first else (padlen, r.nseq, w.shape[1])
        out = torch.empty(shape, dtype=w.dtype, device=w.device)
        capi.embed(r.device, r.stream, r.d_bytes, r.d_offs, r.nseq, padlen, tok, batch_first, w, w.shape[0], row_bytes, out)
        r.keep.append(w)
        return out
    finally:
        r.release()


def augment_packed(bytes_cuda, offsets_cuda, augment=1, augment_frac=1.0, seed=0, seq_index_base=0):
    """BLOSUM62 point mutations of a packed CUDA batch, in place (bioseq/blosum.py:63-87 per sequence).
    Returns ``bytes_cuda``."""
    torch = _torch()
    if not (isinstance(bytes_cuda, torch.Tensor) and bytes_cuda.is_cuda and bytes_cuda.dtype == torch.uint8 and
            isinstance(offsets_cuda, torch.Tensor) and offsets_cuda.is_cuda and offsets_cuda.dtype == torch.int64):
        raise ValueError("augment_packed: uint8 bytes and int64 offsets CUDA tensors expected")
    dev = bytes_cuda.device.index
    capi.augment_blosum62(dev, torch.cuda.current_stream(dev).cuda_stream, bytes_cuda, offsets_cuda, offsets_cuda.numel() - 1,
                          int(augment), float(augment_frac), int(seed), int(seq_index_base))
    return bytes_cuda


CroppedBatch = collections.namedtuple("CroppedBatch", ["bytes", "offsets", "starts"])
CroppedBatch.__doc__ = """A cropped packed batch: ``bytes`` (uint8) and ``offsets`` (int64, from 0) of the windows, and ``starts``
(int64, one per sequence: where its window begins in the sequence -- what a caller needs to crop per-residue labels or
coordinates the same way)."""


def crop_packed(bytes_cuda, offsets_cuda, crop_len, *, crop="random", seed=0, seq_index_base=0):
    """Every sequence of a packed CUDA batch cropped to at most ``crop_len`` residues: a :class:`CroppedBatch`.

    ``crop="random"``: a window drawn from Philox4x32-10 keyed by ``seed`` at sequence ``seq_index_base + i`` (the same
    window whatever the batch's slicing; redraw with another seed); ``crop="head"``: the first ``crop_len`` residues.
    A sequence no longer than ``crop_len`` is kept whole.  The exact rule is documented with ``bsq_crop`` in
    include/bsq.h.  One synchronisation: the output's size is read back, and the offsets are validated."""
    torch = _torch()
    _packed_cuda("crop_packed", bytes_cuda, offsets_cuda)
    if crop is None:
        raise ValueError("crop_packed: crop must be 'head' or 'random'")
    random, crop_len, seed, base = _crop_spec(crop, crop_len, seed, seq_index_base)
    n = _nseq(offsets_cuda)
    dev = bytes_cuda.device
    stream = torch.cuda.current_stream(dev.index).cuda_stream
    total, _ = capi.crop_extent_device(dev.index, stream, offsets_cuda, n, crop_len, nbytes=bytes_cuda.numel())
    out_b = torch.empty(max(total, 1), dtype=torch.uint8, device=dev)
    out_o = torch.empty(n + 1, dtype=torch.int64, device=dev)
    starts = torch.empty(n, dtype=torch.int64, device=dev)
    src = bytes_cuda if bytes_cuda.numel() > 0 else out_b  # (an all-empty batch: nothing is read)
    capi.crop(dev.index, stream, src, offsets_cuda, n, crop_len, random, seed, base, out_b, out_o, starts)
    return CroppedBatch(out_b[:total], out_o, starts)


def batch_tokenize_cropped(tokenizer, batch, padlen, destchar="B", batch_first=True, device=None, *, crop="random", crop_len=None,
                           seed=0, seq_index_base=0, augment=0, augment_frac=1.0, rc=None, rc_prob=None, translate=None,
                           genetic_code=1):
    """``batch_tokenize`` of the batch with every sequence cropped to ``crop_len`` residues on the device (default and
    maximum: ``padlen - bos - eos``): stage -> crop -> augment -> tokenize.  ``crop``: ``"random"`` or ``"head"``, as
    :func:`crop_packed` (same ``seed`` / ``seq_index_base``).  ``rc`` / ``rc_prob``: the windows are then flipped, as
    :func:`batch_tokenize_revcomp` does.  ``translate`` / ``genetic_code``: the DNA is first translated, as
    :func:`batch_tokenize_translated` does, and the proteins are cropped (``crop_len`` in amino acids)."""
    if crop is None:
        raise ValueError("batch_tokenize_cropped: crop must be 'head' or 'random'")
    return _tokenize_padded(tokenizer, batch, padlen, destchar, batch_first, device, crop, crop_len, seed, seq_index_base,
                            augment, augment_frac, rc, rc_prob, translate, genetic_code)


def batch_tokenize_revcomp(tokenizer, batch, padlen, destchar="B", batch_first=True, device=None, *, rc="random", rc_prob=None,
                           seed=0, seq_index_base=0, crop=None, crop_len=None):
    """``batch_tokenize`` of the batch's reverse complements, flipped on the device: stage -> crop -> flip -> tokenize.

    ``rc="random"``: each sequence is flipped with probability ``rc_prob`` (default 0.5) by a coin drawn from
    Philox4x32-10 keyed by ``seed`` at sequence ``seq_index_base + i`` (the same coin whatever the slicing); ``"always"``:
    every sequence; ``"both"``: ``2n`` rows, the batch as is and then its reverse complements (average the model's outputs
    over ``y[:n]`` and the flipped ``y[n:]``).  The complement keeps case and maps IUPAC codes (U -> A); the exact rule is
    documented with ``bsq_revcomp`` in include/bsq.h.  Nucleotide tokenizers only (DNA, DNA4, DNA5, DNAMETH, C, KETO,
    PURPYR).  ``crop`` / ``crop_len``: as :func:`batch_tokenize_cropped`, applied before the flip.  CUDA batches pay one
    read-back, which validates their offsets and replaces the length check."""
    if rc is None:
        raise ValueError("batch_tokenize_revcomp: rc must be 'always', 'random' or 'both'")
    return _tokenize_padded(tokenizer, batch, padlen, destchar, batch_first, device, crop, crop_len, seed, seq_index_base, 0, 1.0,
                            rc, rc_prob)


def _tokenize_padded(tokenizer, batch, padlen, destchar, batch_first, device, crop, crop_len, seed, seq_index_base, augment,
                     augment_frac, rc, rc_prob, translate=None, genetic_code=1):
    torch = _torch()
    tok = descriptor(tokenizer)
    padlen = _default_padlen(batch, tokenizer, padlen)
    kind, dtype = _dtype_of(destchar)
    tr = _translate_spec(translate, genetic_code, tokenizer, rc, seq_index_base)
    seq_index_base = _out_base(seq_index_base, tr)
    crop = _crop_spec(crop, crop_len, seed, seq_index_base, _row_residues(tokenizer, padlen))
    rc = _rc_spec(rc, rc_prob, seed, seq_index_base, tokenizer, augment)
    r = _resolve(batch, device, _augment_args(augment, augment_frac, seed, seq_index_base), crop=crop, rc=rc, translate=tr)
    try:
        _check_lengths(r, padlen, tok, onehot=False)
        shape = (r.nseq, padlen) if batch_first else (padlen, r.nseq)
        out = torch.empty(shape, dtype=dtype, device=torch.device("cuda", r.device))
        capi.tokenize(r.device, r.stream, r.d_bytes, r.d_offs, r.nseq, padlen, tok, batch_first, kind, out)
        return out
    finally:
        r.release()


RevCompBatch = collections.namedtuple("RevCompBatch", ["bytes", "offsets", "flipped"])
RevCompBatch.__doc__ = """A reverse-complemented packed batch: ``bytes`` (uint8) and ``offsets`` (int64, from 0) of the output
sequences, and ``flipped`` (bool, one per output sequence: whether it is a reverse complement -- what a caller needs to
flip per-position labels the same way)."""


def revcomp_packed(bytes_cuda, offsets_cuda, *, rc="always", rc_prob=None, seed=0, seq_index_base=0):
    """The reverse complement of a packed CUDA batch: a :class:`RevCompBatch`; the input is not modified.

    ``rc="always"``: every sequence is flipped; ``"random"``: each with probability ``rc_prob`` (default 0.5), the coin
    drawn from Philox4x32-10 keyed by ``seed`` at sequence ``seq_index_base + i``; ``"both"``: ``2n`` sequences, the batch
    unchanged and then flipped.  The exact rule is documented with ``bsq_revcomp`` in include/bsq.h.  For per-position
    labels: crop with :func:`crop_packed`, flip with this, then reverse the labels of the rows ``flipped`` marks.  One
    synchronisation: the offsets are validated and the output's size is read back."""
    torch = _torch()
    _packed_cuda("revcomp_packed", bytes_cuda, offsets_cuda)
    if rc is None:
        raise ValueError("revcomp_packed: rc must be 'always', 'random' or 'both'")
    mode, rc_prob, seed, base = _rc_spec(rc, rc_prob, seed, seq_index_base)
    n = _nseq(offsets_cuda)
    dev = bytes_cuda.device
    stream = torch.cuda.current_stream(dev.index).cuda_stream
    total, _ = capi.crop_extent_device(dev.index, stream, offsets_cuda, n, _UNCROPPED, nbytes=bytes_cuda.numel())
    m = 2 if mode == capi.RC_BOTH else 1
    out_b = torch.empty(max(m * total, 1), dtype=torch.uint8, device=dev)
    out_o = torch.empty(m * n + 1, dtype=torch.int64, device=dev)
    flipped = torch.empty(m * n, dtype=torch.uint8, device=dev)
    src = bytes_cuda if bytes_cuda.numel() > 0 else out_b  # (an all-empty batch: nothing is read)
    capi.revcomp(dev.index, stream, src, offsets_cuda, n, mode, rc_prob, seed, base, out_b, out_o, flipped)
    return RevCompBatch(out_b[:m * total], out_o, flipped.view(torch.bool))


def batch_tokenize_augmented(tokenizer, batch, padlen=-1, destchar="B", batch_first=False, device=None, *, augment=1,
                             augment_frac=1.0, seed=0, seq_index_base=0):
    """``batch_tokenize`` of the BLOSUM62-augmented batch: copy -> mutate on the device -> tokenize
    (what FlatFileDataset does per item with Python strings, bioseq/loaders.py:99-101)."""
    return _tokenize_padded(tokenizer, batch, padlen, destchar, batch_first, device, None, None, seed, seq_index_base, augment,
                            augment_frac, None, None)


VarlenBatch = collections.namedtuple("VarlenBatch", ["tokens", "cu_seqlens", "max_seqlen"])
VarlenBatch.__doc__ = """A padding-free token batch: ``tokens`` (1-D, all rows back to back), ``cu_seqlens`` (int32, ``n + 1``
entries: row ``i`` is ``tokens[cu_seqlens[i]:cu_seqlens[i + 1]]``) and ``max_seqlen`` (int) -- the arguments of varlen
attention (``flash_attn_varlen_func(q, k, v, cu_seqlens, cu_seqlens, max_seqlen, max_seqlen)``)."""

_INT32_MAX = 2 ** 31 - 1


def _check_cu_seqlens(total, what="varlen"):
    """ValueError unless ``total`` tokens of a ``what`` batch can be indexed by int32 ``cu_seqlens``."""
    if total > _INT32_MAX:
        raise ValueError(f"{what} batch of {total} tokens: cu_seqlens is int32, so at most 2^31 - 1 tokens fit one batch; "
                         "split the batch")


def _varlen_extent_host(h_offs, n, k):
    """(T, max_seqlen) of host offsets; ValueError on offsets the kernels must not index with, or T > 2^31 - 1."""
    if n == 0:
        return 0, 0
    o = np.asarray(h_offs[:n + 1], dtype=np.int64)
    lens = np.diff(o)
    if int(o[0]) < 0:
        raise ValueError("offsets must start at or after 0")
    if lens.size and int(lens.min()) < 0:
        raise ValueError("offsets must be non-decreasing")
    total = int(o[n]) - int(o[0]) + n * k
    _check_cu_seqlens(total)
    return total, int(lens.max()) + k


def batch_tokenize_varlen(tokenizer, batch, destchar="B", device=None, *, crop=None, crop_len=None, seed=0, seq_index_base=0,
                          rc=None, rc_prob=None, translate=None, genetic_code=1):
    """Tokens of every sequence of ``batch`` back to back, without padding: a :class:`VarlenBatch`.

    Row ``i`` (``tokens[cu_seqlens[i]:cu_seqlens[i + 1]]``) equals ``batch_tokenize(batch, padlen=P, batch_first=True,
    destchar=destchar)[i, :len_i + bos + eos]`` for any large enough ``P``: ``[BOS] residues [EOS]``, no PAD token
    whatever ``padchar`` is.  ``cu_seqlens[i] = (offsets[i] - offsets[0]) + i * (bos + eos)`` as int32; a batch of more
    than 2^31 - 1 tokens raises ``ValueError``.  Host batches are sized from their host offsets without synchronising;
    CUDA batches pay one synchronisation (the extent is read back).  ``crop`` / ``crop_len`` (required with ``crop``):
    every sequence is cropped first, as :func:`crop_packed` does.  ``rc`` / ``rc_prob``: then flipped, as
    :func:`batch_tokenize_revcomp` does (``"both"`` gives ``2n`` rows).  ``translate`` / ``genetic_code``: the DNA is
    first translated, as :func:`batch_tokenize_translated` does (``crop_len`` then counts amino acids)."""
    tr = _translate_spec(translate, genetic_code, tokenizer, rc, seq_index_base)
    seq_index_base = _out_base(seq_index_base, tr)
    return _tokenize_varlen(tokenizer, batch, destchar, device, crop=_crop_spec(crop, crop_len, seed, seq_index_base),
                            rc=_rc_spec(rc, rc_prob, seed, seq_index_base, tokenizer), translate=tr)


def _tokenize_varlen(tokenizer, batch, destchar, device, augment=None, mlm=None, crop=None, rc=None, translate=None):
    """batch_tokenize_varlen; ``augment``: BLOSUM62 arguments as ``_augment_args`` makes them (FlatFileDataset);
    ``mlm``: a ``capi.MLMDesc`` -- then ``(VarlenBatch, labels)`` is returned; ``crop``: from ``_crop_spec``; ``rc``: from
    ``_rc_spec``; ``translate``: from ``_translate_spec``."""
    torch = _torch()
    tok = descriptor(tokenizer)
    kind, dtype = _dtype_of(destchar)
    k = int(tokenizer.includes_bos()) + int(tokenizer.includes_eos())
    extent = []
    r = _resolve(batch, device, augment, before_stage=lambda h_offs, n: extent.extend(_varlen_extent_host(h_offs, n, k)),
                 crop=crop, rc=rc, translate=translate)
    try:
        if r.h_offs is not None:
            total, max_seqlen = extent
        else:
            if r.extent is not None:  # a cropped or flipped CUDA batch: sized by its one read-back
                total, max_seqlen = r.extent[0] + r.nseq * k, (r.extent[1] + k if r.nseq > 0 else 0)
            else:
                total, max_seqlen = capi.varlen_extent_device(r.device, r.stream, r.d_offs, r.nseq, tok, nbytes=batch[0].numel())
            _check_cu_seqlens(total)
        dev = torch.device("cuda", r.device)
        tokens = torch.empty(total, dtype=dtype, device=dev)
        cu_seqlens = torch.empty(r.nseq + 1, dtype=torch.int32, device=dev)
        if mlm is not None:
            labels = torch.empty(total, dtype=torch.int64, device=dev)
            capi.tokenize_varlen_mlm(r.device, r.stream, r.d_bytes, r.d_offs, r.nseq, tok, kind, mlm, tokens, labels, cu_seqlens)
            return VarlenBatch(tokens, cu_seqlens, max_seqlen), labels
        capi.tokenize_varlen(r.device, r.stream, r.d_bytes, r.d_offs, r.nseq, tok, kind, tokens, cu_seqlens)
        return VarlenBatch(tokens, cu_seqlens, max_seqlen)
    finally:
        r.release()


MLMBatch = collections.namedtuple("MLMBatch", ["inputs", "labels"])
MLMBatch.__doc__ = """A masked-language-model batch: ``inputs`` (the model's input tokens: a padded ``(n, padlen)`` tensor or a
:class:`VarlenBatch`) and ``labels`` (int64, the same shape as the tokens: the original token where a position was
selected, ``ignore_index`` elsewhere) -- ``F.cross_entropy(logits.view(-1, V), labels.view(-1), ignore_index=...)``."""

_TWO32 = 1 << 32
_INT64_MIN, _INT64_MAX = -(1 << 63), (1 << 63) - 1


def _mlm_thresholds(maskfrac=0.15, mask_prob=0.8, random_prob=0.1):
    """The integer thresholds ``(t_select, t_mask, t_random)`` the kernel compares 32-bit draws with (include/bsq.h,
    bsq_mlm), computed once in float64.  ValueError unless 0 <= maskfrac <= 1, mask_prob, random_prob >= 0 and
    mask_prob + random_prob <= 1."""
    maskfrac, mask_prob, random_prob = float(maskfrac), float(mask_prob), float(random_prob)
    if not 0.0 <= maskfrac <= 1.0:
        raise ValueError(f"maskfrac must lie in [0, 1], got {maskfrac}")
    if not (mask_prob >= 0.0 and random_prob >= 0.0):
        raise ValueError(f"mask_prob and random_prob must be >= 0, got {mask_prob} and {random_prob}")
    if not mask_prob + random_prob <= 1.0:
        raise ValueError(f"mask_prob + random_prob must be <= 1, got {mask_prob + random_prob}")
    t_select = _TWO32 if maskfrac >= 1.0 else math.floor(maskfrac * _TWO32)
    t_mask = math.floor(t_select * mask_prob)
    t_random = min(t_select, math.floor(t_select * (mask_prob + random_prob)))
    return t_select, t_mask, t_random


def _mask_token_limit(destchar):
    c = destchar[0]
    if c == "B":
        return 255
    return {"b": 127, "h": 32767, "f": 1 << 24}.get(c.lower(), (1 << 31) - 1)


def _mlm_desc(tok, destchar, maskfrac, mask_prob, random_prob, mask_token, ignore_index, seed, seq_index_base):
    """Validate everything and build the capi.MLMDesc (ValueError before anything is staged or launched)."""
    thresholds = _mlm_thresholds(maskfrac, mask_prob, random_prob)
    if mask_token is None:
        mask_token = int(tok.alphabet_size)
    try:
        mask_token = operator.index(mask_token)
        ignore_index = operator.index(ignore_index)
    except TypeError:
        raise ValueError("mask_token and ignore_index must be integers") from None
    limit = _mask_token_limit(destchar)
    if not 0 <= mask_token <= limit:
        raise ValueError(f"mask_token {mask_token} is not representable in destchar {destchar!r} (0..{limit}); "
                         "pass mask_token= explicitly")
    if not _INT64_MIN <= ignore_index <= _INT64_MAX:
        raise ValueError(f"ignore_index {ignore_index} does not fit int64")
    return capi.mlm_desc(int(seed), int(seq_index_base), thresholds, mask_token, ignore_index)


def batch_tokenize_mlm(tokenizer, batch, padlen=-1, destchar="B", device=None, *, varlen=False, maskfrac=0.15, mask_prob=0.8,
                       random_prob=0.1, mask_token=None, ignore_index=-100, seed=0, seq_index_base=0, augment=0,
                       augment_frac=1.0, crop=None, crop_len=None, rc=None, rc_prob=None, translate=None, genetic_code=1):
    """A masked-language-model batch in one launch: :class:`MLMBatch` ``(inputs, labels)``.

    ``inputs`` start from ``batch_tokenize(batch, padlen, batch_first=True, destchar=destchar)`` (``varlen=False``:
    ``(n, padlen)``) or ``batch_tokenize_varlen(batch, destchar)`` (``varlen=True``: a :class:`VarlenBatch`; passing
    ``padlen`` is then an error).  ``labels`` are int64, shaped like the tokens.  Only residue positions are eligible
    (never BOS / EOS / PAD).  A residue is selected with probability ``maskfrac``; a selected residue's label is its
    token, and its input becomes ``mask_token`` (default ``alphabet_size()``, the first id the tokenizer does not
    use) with probability ``mask_prob``, a uniformly random residue id with probability ``random_prob``, and stays
    otherwise.  Every other label is ``ignore_index``.

    The draw is Philox4x32-10 keyed by ``seed`` at (``seq_index_base + i``, residue position): the same sequence gets
    the same mask padded or padding-free, in any slice (the exact rule is documented with ``bsq_tokenize_mlm`` in
    include/bsq.h).  ``augment``: BLOSUM62 point mutations first (as ``batch_tokenize_augmented``, same seed), then the
    mask.  ``crop`` / ``crop_len``: every sequence is cropped before both (as :func:`batch_tokenize_cropped`, same seed;
    ``varlen=True`` needs an explicit ``crop_len``); residue positions are then positions within the window.  ``rc`` /
    ``rc_prob``: "always" or "random" (not "both"), after the crop and before the mask, as :func:`batch_tokenize_revcomp`
    does; residue positions are then positions in the flipped window.  ``translate`` / ``genetic_code``: the DNA is first
    translated, as :func:`batch_tokenize_translated` does; positions are then amino acids and the draw for output row
    ``(i, f)`` is keyed by ``(seq_index_base + i) * F + f``."""
    torch = _torch()
    tok = descriptor(tokenizer)
    kind, dtype = _dtype_of(destchar)
    tr = _translate_spec(translate, genetic_code, tokenizer, rc, seq_index_base)
    seq_index_base = _out_base(seq_index_base, tr)
    mlm = _mlm_desc(tok, destchar, maskfrac, mask_prob, random_prob, mask_token, ignore_index, seed, seq_index_base)
    rc = _rc_spec(rc, rc_prob, seed, seq_index_base, tokenizer, augment, mlm=True)
    augment = _augment_args(augment, augment_frac, seed, seq_index_base)
    if varlen:
        _padlen("batch_tokenize_mlm", padlen, varlen)
        crop = _crop_spec(crop, crop_len, seed, seq_index_base)
        vb, labels = _tokenize_varlen(tokenizer, batch, destchar, device, augment, mlm, crop, rc, tr)
        return MLMBatch(vb, labels)
    padlen = _default_padlen(batch, tokenizer, padlen)
    crop = _crop_spec(crop, crop_len, seed, seq_index_base, _row_residues(tokenizer, padlen))
    r = _resolve(batch, device, augment, crop=crop, rc=rc, translate=tr)
    try:
        _check_lengths(r, padlen, tok, onehot=False)
        dev = torch.device("cuda", r.device)
        inputs = torch.empty((r.nseq, padlen), dtype=dtype, device=dev)
        labels = torch.empty((r.nseq, padlen), dtype=torch.int64, device=dev)
        capi.tokenize_mlm(r.device, r.stream, r.d_bytes, r.d_offs, r.nseq, padlen, tok, kind, mlm, inputs, labels)
        return MLMBatch(inputs, labels)
    finally:
        r.release()


SeqPackBatch = collections.namedtuple("SeqPackBatch", ["tokens", "position_ids", "cu_seqlens", "max_seqlen", "starts", "labels"])
SeqPackBatch.__doc__ = """Whole sequences packed into fixed-width rows: ``tokens`` ``(rows, L)`` (MLM inputs with ``mlm=True``),
``position_ids`` int32 ``(rows, L)`` (0 at the start of every sequence and of every row's padding run), ``cu_seqlens`` (int32:
the flat start of every segment -- a sequence or a padding run -- then ``rows * L``), ``max_seqlen`` (int, the longest
segment), ``starts`` (int64, one per sequence: its flat position in ``tokens.view(-1)``, -1 for a sequence that occupies
nothing) and ``labels`` (int64 ``(rows, L)`` with ``mlm=True``, else None)."""


class _SeqPackPlan:
    """The host plan (bsq_seqpack_plan) in one pinned int64 buffer: row_ptr | row_seq | starts | cu_seqlens (int32)."""

    def __init__(self, h_offs, n, k, row_len, rows):
        torch = _torch()
        h_offs = np.ascontiguousarray(h_offs[:n + 1], dtype=np.int64)
        R, nseg, self.max_seqlen = capi.seqpack_plan(h_offs, n, k, row_len, rows)  # (sizes; ValueError on a bad layout)
        self.R, self.nseg, self.n = R, nseg, n
        self.o_seq, self.o_starts, self.o_cu = R + 1, R + 1 + n, R + 1 + 2 * n
        self.buf = torch.empty(self.o_cu + (nseg + 2) // 2, dtype=torch.int64, pin_memory=True)
        a = self.buf.numpy()
        capi.seqpack_plan(h_offs, n, k, row_len, rows, a[self.o_starts:], a, a[self.o_seq:], a[self.o_cu:])

    def to_device(self, dev):
        """One cudaMemcpyAsync from pinned memory on the current stream."""
        self.dbuf = self.buf.to(dev, non_blocking=True)
        d = self.dbuf
        return (d[:self.o_seq], d[self.o_seq:self.o_starts], d[self.o_starts:self.o_cu],
                d[self.o_cu:].view(_torch().int32)[:self.nseg + 1])


def batch_tokenize_seqpack(tokenizer, batch, row_len, destchar="B", device=None, *, rows=None, mlm=False, maskfrac=0.15,
                           mask_prob=0.8, random_prob=0.1, mask_token=None, ignore_index=-100, crop=None, crop_len=None,
                           augment=0, augment_frac=1.0, seed=0, seq_index_base=0, rc=None, rc_prob=None, translate=None,
                           genetic_code=1):
    """Sequence packing: every sequence of ``batch`` whole, laid end to end in rows of ``row_len`` tokens -- a
    :class:`SeqPackBatch` of fixed shape ``(rows, row_len)`` with almost no padding.

    Placement is best-fit decreasing (longest first, each into the fullest row that still fits it; the exact,
    deterministic rule is documented with ``bsq_seqpack_plan`` in include/bsq.h).  The tokens of sequence ``i`` at
    ``starts[i]`` equal row ``i`` of :func:`batch_tokenize_varlen`: ``[BOS] residues [EOS]``; the rest of a row is what
    ``batch_tokenize`` writes after EOS.  ``position_ids`` restart at 0 for every sequence and padding run, and
    ``cu_seqlens`` lists them all, so the batch feeds ``flash_attn_varlen_func`` (flattened), SDPA with a block mask
    (``(position_ids == 0).cumsum(-1)``) or models that find packed sequences from position ids.

    ``rows``: exactly that many rows (extra rows are padding; ValueError if the batch needs more), else as many as
    needed.  ``mlm=True``: inputs and int64 labels as :func:`batch_tokenize_mlm` (``varlen=True``, same seed and
    ``seq_index_base``) writes them per sequence, padding labels ``ignore_index``.  ``crop`` / ``crop_len`` (default
    ``row_len - bos - eos``) and ``augment`` as for the other consumers: stage -> crop -> augment -> pack.  Every
    sequence must fit a row (ValueError otherwise).  ``rc`` / ``rc_prob``: sequences are flipped after the crop, as
    :func:`batch_tokenize_revcomp` does (``"both"``, not with ``mlm``, packs ``2n`` sequences).  ``translate`` /
    ``genetic_code``: the DNA is first translated, as :func:`batch_tokenize_translated` does, and the ``n F`` proteins are
    packed.  Host batches are planned from their host offsets without synchronising; CUDA batches pay one read-back of
    their offsets, which also validates them."""
    torch = _torch()
    tok = descriptor(tokenizer)
    kind, dtype = _dtype_of(destchar)
    tr = _translate_spec(translate, genetic_code, tokenizer, rc, seq_index_base)
    seq_index_base = _out_base(seq_index_base, tr)
    k = int(tokenizer.includes_bos()) + int(tokenizer.includes_eos())
    try:
        row_len = operator.index(row_len)
        rows = None if rows is None else operator.index(rows)
    except TypeError:
        raise ValueError("row_len and rows must be integers") from None
    if row_len < 1:
        raise ValueError(f"row_len must be >= 1, got {row_len}")
    if rows is not None and rows < 1:
        raise ValueError(f"rows must be >= 1, got {rows}")
    rows = rows or 0  # (the planner's "as many as needed")
    mlm = _mlm_desc(tok, destchar, maskfrac, mask_prob, random_prob, mask_token, ignore_index, seed, seq_index_base) if mlm else None
    crop = _crop_spec(crop, crop_len, seed, seq_index_base, row_len - k)
    rc = _rc_spec(rc, rc_prob, seed, seq_index_base, tokenizer, augment, mlm=mlm is not None)
    augment = _augment_args(augment, augment_frac, seed, seq_index_base)
    plan = []

    def make_plan(h_offs, n):
        plan.append(_SeqPackPlan(h_offs, n, k, row_len, rows))

    p = _parse(batch)
    checked = None
    if p.bytes is not None:  # planned before anything is staged (a CUDA batch: from its offsets, read back once)
        cuda, sized, h = isinstance(p.offsets, torch.Tensor), crop is not None or rc is not None or tr is not None, p.offsets
        if cuda:
            h = h.cpu().numpy()
            _nseq(h, p.bytes.numel())
        n = h.size - 1
        if cuda or sized:  # (this also validates the offsets)
            cropped, checked, tr_total = _sized_host(h, n, crop[1] if crop is not None else _UNCROPPED, tr)
            if tr is not None:
                checked = (*checked, tr_total)
        make_plan(*_rc_host_offsets(cropped if sized else h, n * len(tr[0]) if tr is not None else n, rc))
    r = _resolve(p, device, augment, before_stage=None if plan else make_plan, crop=crop, rc=rc, checked=checked, translate=tr)
    try:
        p = plan[0]
        dev = torch.device("cuda", r.device)
        with torch.cuda.device(r.device):
            d_row_ptr, d_row_seq, starts, cu_seqlens = p.to_device(dev)
        tokens = torch.empty((p.R, row_len), dtype=dtype, device=dev)
        position_ids = torch.empty((p.R, row_len), dtype=torch.int32, device=dev)
        labels = None
        if mlm is not None:
            labels = torch.empty((p.R, row_len), dtype=torch.int64, device=dev)
            capi.tokenize_seqpack_mlm(r.device, r.stream, r.d_bytes, r.d_offs, tok, kind, mlm, row_len, p.R, d_row_ptr, d_row_seq,
                                      tokens, position_ids, labels)
        else:
            capi.tokenize_seqpack(r.device, r.stream, r.d_bytes, r.d_offs, tok, kind, row_len, p.R, d_row_ptr, d_row_seq, tokens,
                                  position_ids)
        r.keep.append(p)
        return SeqPackBatch(tokens, position_ids, cu_seqlens, p.max_seqlen, starts, labels)
    finally:
        r.release()


KmerIds = collections.namedtuple("KmerIds", ["nkmers", "single_base", "unk", "bos", "eos", "pad", "vocab_size"])
KmerIds.__doc__ = """The ids of a k-mer vocabulary (include/bsq.h, bsq_kmer): k-mers are ``0 .. nkmers - 1`` (``nkmers = b^k``),
the single residue of code ``c`` is ``single_base + c``, ``unk`` stands for anything with an invalid byte, then ``bos`` /
``eos`` (None when the tokenizer has none) and ``pad``; ``vocab_size`` ids in all -- the size of an ``nn.Embedding``."""

_KMER_TAILS = {"drop": capi.KMER_DROP, "single": capi.KMER_SINGLE}


def _kmer_desc(tokenizer, k, stride=1, tail="drop"):
    """capi.KmerDesc of (tokenizer, k, stride, tail); ValueError on anything bsq_kmer_init rejects."""
    if tail not in _KMER_TAILS:
        raise ValueError(f"tail must be 'drop' or 'single', got {tail!r}")
    try:
        k, stride = operator.index(k), operator.index(stride)
    except TypeError:
        raise ValueError("k and stride must be integers") from None
    if not (-2 ** 31 <= k < 2 ** 31 and -2 ** 31 <= stride < 2 ** 31):
        raise ValueError(f"k = {k} or stride = {stride} out of range")
    return capi.kmer_desc(descriptor(tokenizer), k, stride, _KMER_TAILS[tail])


def kmer_ids(tokenizer, k):
    """The ids of ``tokenizer``'s k-mer vocabulary: a :class:`KmerIds`.  They depend on the tokenizer and ``k`` only (not on
    the stride or the tail mode), so one embedding serves every way of cutting the sequences."""
    km = _kmer_desc(tokenizer, k)
    return KmerIds(km.nkmers, km.nkmers, km.unk_id, km.bos_id if km.bos else None, km.eos_id if km.eos else None, km.pad_id,
                   km.vocab_size)


def kmer_vocab(tokenizer, k):
    """The string of every id of ``tokenizer``'s k-mer vocabulary, in id order (for HF vocab files and for inspection).

    K-mers and single residues are spelled with the letter ``decode_tokens`` prints for each residue code (so a k-mer is
    its k letters, first residue first); the specials are ``"<UNK>"``, ``"<BOS>"``, ``"<EOS>"`` and ``"<PAD>"`` (those the
    tokenizer has).  Its length is ``vocab_size = b^k + b + 1 + bos + eos + padchar``: it grows as b^k (4 096 k-mers for
    DNA with k = 6, about 10^9 with k = 15), so build it only for the k a model uses."""
    import itertools
    tok = descriptor(tokenizer)
    ids = kmer_ids(tokenizer, k)
    buf = capi.C.create_string_buffer(8)
    letters = []
    for c in range(int(tok.nchars)):
        n = capi.lib().bsq_tokenizer_lookup(capi.C.byref(tok), c, buf, 8)
        letters.append(buf.value.decode("latin-1") if n else "?")
    vocab = ["".join(p) for p in itertools.product(letters, repeat=int(k))]
    vocab += letters + ["<UNK>"]
    vocab += ["<BOS>"] * (ids.bos is not None) + ["<EOS>"] * (ids.eos is not None) + ["<PAD>"] * bool(tok.padchar)
    assert len(vocab) == ids.vocab_size
    return vocab


def _kmer_check_extent(extent, padlen, varlen):
    total, longest = extent
    if varlen:
        _check_cu_seqlens(total, "k-mer")
    elif longest > padlen:
        raise ValueError(f"k-mer tokens + bos + eos > padlen: {longest}, vs padlen {padlen}")


def batch_tokenize_kmer(tokenizer, batch, k, padlen=-1, destchar="i", device=None, *, stride=1, tail="drop", varlen=False,
                        crop=None, crop_len=None, seed=0, seq_index_base=0, rc=None, rc_prob=None, translate=None, genetic_code=1):
    """K-mer tokens of every sequence of ``batch``, written by one kernel (padding-free: three small ones).

    Sequence ``i`` of ``n`` residues gives ``[BOS] k-mer ids [single-residue ids] [EOS]``: ``m = (n - k) // stride + 1``
    k-mers (none when ``n < k``) starting at residues ``0, stride, 2 * stride, ...``; with ``tail="single"`` the residues
    after the last k-mer follow one token each, with ``tail="drop"`` they are dropped.  ``stride=1`` gives DNABERT's
    overlapping k-mers, ``stride=k, tail="single"`` Nucleotide Transformer's.  Ids are those of :func:`kmer_ids`: a k-mer is
    its codes read as a base-``b`` number, first residue most significant; anything holding an invalid byte is ``unk``.
    The exact rule is documented with ``bsq_kmer`` in include/bsq.h.

    ``varlen=False``: a padded ``(n, padlen)`` tensor (``padlen`` required), after EOS ``pad`` with ``padchar`` and 0
    without; a row longer than ``padlen`` raises ValueError.  ``varlen=True``: a :class:`VarlenBatch` (``padlen`` must not
    be given); more than 2^31 - 1 tokens raise ValueError.  ``destchar`` defaults to int32 (``"i"``), which holds every
    vocabulary the rule allows; a kind too narrow for ``vocab_size`` raises ValueError.  ``crop`` / ``crop_len`` (required
    with ``crop``, in residues): every sequence is cropped first, as :func:`crop_packed` does.  ``rc`` / ``rc_prob``: then
    flipped, as :func:`batch_tokenize_revcomp` does, so the k-mers are those of the reverse complement.  ``translate`` /
    ``genetic_code``: the DNA is first translated, as :func:`batch_tokenize_translated` does, and the k-mers are those of
    the proteins (a protein tokenizer).  Host batches are sized from their host offsets without synchronising; CUDA
    batches pay one read-back (two when cropped or translated)."""
    torch = _torch()
    tok = descriptor(tokenizer)
    kind, dtype = _dtype_of(destchar)
    tr = _translate_spec(translate, genetic_code, tokenizer, rc, seq_index_base)
    seq_index_base = _out_base(seq_index_base, tr)
    km = _kmer_desc(tokenizer, k, stride, tail)
    limit = _mask_token_limit(destchar)
    if km.vocab_size - 1 > limit:
        raise ValueError(f"k-mer ids up to {km.vocab_size - 1} do not fit destchar {destchar!r} (0..{limit})")
    padlen = _padlen("batch_tokenize_kmer", padlen, varlen, -1)
    if not varlen and padlen <= 0:
        raise ValueError("batch_tokenize_kmer requires padlen (or varlen=True)")
    crop = _crop_spec(crop, crop_len, seed, seq_index_base)
    rc = _rc_spec(rc, rc_prob, seed, seq_index_base, tokenizer)
    extent = []

    def before_stage(h_offs, n):
        e = capi.kmer_extent_host(np.ascontiguousarray(h_offs[:n + 1], dtype=np.int64), n, km)
        _kmer_check_extent(e, padlen, varlen)
        extent.extend(e)

    p = _parse(batch)
    checked = None
    if rc is not None and crop is None and isinstance(p.offsets, torch.Tensor):
        # the extent of the unflipped offsets is the flipped batch's (doubled by "both"), and reading it validates them:
        # the flip needs no read-back of its own
        d = p.bytes.device.index
        total, longest = capi.kmer_extent_device(d, torch.cuda.current_stream(d).cuda_stream, p.offsets, _nseq(p.offsets), km,
                                                 nbytes=p.bytes.numel())
        extent = [total * (2 if rc[0] == capi.RC_BOTH else 1), longest]
        _kmer_check_extent(extent, padlen, varlen)
        checked = True
    r = _resolve(p, device, before_stage=before_stage, crop=crop, rc=rc, checked=checked, translate=tr)
    try:
        if r.h_offs is None and checked is None:  # a CUDA batch: one reduction and read-back, which also validates its offsets
            fresh = crop is not None or tr is not None  # (offsets of buffers _resolve wrote)
            extent = capi.kmer_extent_device(r.device, r.stream, r.d_offs, r.nseq, km, nbytes=-1 if fresh else p.bytes.numel())
            _kmer_check_extent(extent, padlen, varlen)
        dev = torch.device("cuda", r.device)
        if varlen:
            tokens = torch.empty(extent[0], dtype=dtype, device=dev)
            cu_seqlens = torch.empty(r.nseq + 1, dtype=torch.int32, device=dev)
            # an all-empty batch may have no residue buffer at all; nothing is read from it then
            capi.tokenize_kmer_varlen(r.device, r.stream, r.d_bytes or cu_seqlens, r.d_offs, r.nseq, tok, km, kind, tokens,
                                      cu_seqlens)
            return VarlenBatch(tokens, cu_seqlens, extent[1])
        out = torch.empty((r.nseq, padlen), dtype=dtype, device=dev)
        capi.tokenize_kmer(r.device, r.stream, r.d_bytes or out, r.d_offs, r.nseq, padlen, tok, km, kind, out)
        return out
    finally:
        r.release()


_TILE_TAILS = {"short": capi.TILE_SHORT, "end": capi.TILE_END, "drop": capi.TILE_DROP}


def _tile_spec(window, stride, tail):
    """Validate the tiling arguments (ValueError before anything is staged) -> ``(window, stride, tail code)``; ``stride``
    defaults to ``window`` (windows side by side)."""
    if not isinstance(tail, str) or tail not in _TILE_TAILS:
        raise ValueError(f"tail must be 'short', 'end' or 'drop', got {tail!r}")
    try:
        window = operator.index(window)
        stride = window if stride is None else operator.index(stride)
    except TypeError:
        raise ValueError("window and stride must be integers") from None
    if not 1 <= window <= _INT64_MAX:
        raise ValueError(f"window must be >= 1, got {window}")
    if not 1 <= stride <= window:
        raise ValueError(f"stride must lie in 1..window = {window}, got {stride}")
    return int(window), int(stride), _TILE_TAILS[tail]


TiledBatch = collections.namedtuple("TiledBatch", ["bytes", "offsets", "seq_index", "starts", "seq_ptr", "seq_offsets"])
TiledBatch.__doc__ = """Every window of a packed batch, as a packed batch: ``bytes`` (uint8) and ``offsets`` (int64, from 0) of the
windows; ``seq_index`` (int64, one per window: its sequence -- HF's ``overflow_to_sample_mapping``); ``starts`` (int64, one
per window: where it begins in its sequence); ``seq_ptr`` (int64, ``n + 1``: sequence ``i``'s windows are
``seq_ptr[i] .. seq_ptr[i + 1] - 1``); ``seq_offsets`` (int64, ``n + 1``: the source offsets from 0, the layout
:func:`untile` writes)."""


def tile_packed(bytes_cuda, offsets_cuda, window, *, stride=None, tail="short"):
    """Every window of ``window`` residues, every ``stride`` residues (default ``window``), of every sequence of a packed
    CUDA batch: a :class:`TiledBatch`; the input is not modified.

    A sequence of at most ``window`` residues is one window (an empty sequence one empty window).  A longer one gives
    windows at ``0, stride, 2 * stride, ...``; ``tail`` decides the last: ``"short"`` keeps a shorter last window,
    ``"end"`` ends the last window at the sequence's end (every window is ``window`` long), ``"drop"`` drops the residues
    after the last full window.  The exact rule is documented with ``bsq_tile`` in include/bsq.h.  ``(tb.bytes,
    tb.offsets)`` is a packed CUDA batch that every consumer takes, ``rc=`` included; their seeded draws are then keyed by
    window index (``seq_index_base + w``).  One synchronisation: the offsets are validated and the output's size is read
    back."""
    torch = _torch()
    _packed_cuda("tile_packed", bytes_cuda, offsets_cuda)
    window, stride, tail = _tile_spec(window, stride, tail)
    n = _nseq(offsets_cuda)
    dev = bytes_cuda.device
    stream = torch.cuda.current_stream(dev.index).cuda_stream
    M, nbytes, _ = capi.tile_extent_device(dev.index, stream, offsets_cuda, n, window, stride, tail, nbytes=bytes_cuda.numel())
    out = _tile_into(dev, stream, bytes_cuda.data_ptr(), offsets_cuda, n, window, stride, tail, M, nbytes)
    return out._replace(seq_offsets=offsets_cuda - offsets_cuda[:1])


def _tile_into(dev, stream, d_bytes, d_offs, n, window, stride, tail, M, nbytes):
    """bsq_tile into fresh buffers (a TiledBatch without seq_offsets)."""
    torch = _torch()
    out_b = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)  # (never a null pointer)
    out_o = torch.empty(M + 1, dtype=torch.int64, device=dev)
    seq_ptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
    seq_index = torch.empty(M, dtype=torch.int64, device=dev)
    starts = torch.empty(M, dtype=torch.int64, device=dev)
    # an all-empty batch may have no residue buffer at all; nothing is read from it then
    capi.tile(dev.index, stream, d_bytes or out_b, d_offs, n, window, stride, tail, out_b, out_o, seq_ptr, seq_index, starts)
    return TiledBatch(out_b[:nbytes], out_o, seq_index, starts, seq_ptr, None)


TiledTokens = collections.namedtuple("TiledTokens", ["tokens", "seq_index", "starts", "seq_ptr", "seq_offsets", "flipped", "strands",
                                                     "window", "stride", "tail", "bos"])
TiledTokens.__doc__ = """Tokens of every window of a batch: ``tokens`` (padded ``(strands * M, padlen)`` or a :class:`VarlenBatch`),
``seq_index`` / ``starts`` / ``seq_ptr`` / ``seq_offsets`` as in :class:`TiledBatch` (for the ``M`` windows of one strand:
with ``strands == 2`` rows ``M .. 2M - 1`` are rows ``0 .. M - 1`` reverse-complemented), ``flipped`` (bool, one per row,
or None without ``rc``), ``strands`` (1, or 2 for ``rc="both"``), ``window`` / ``stride`` / ``tail`` (the tiling) and
``bos`` (leading special tokens per row: :func:`untile`'s default ``col0``)."""

UntiledBatch = collections.namedtuple("UntiledBatch", ["values", "offsets"])
UntiledBatch.__doc__ = """Per-residue values stitched back onto the sequences: ``values`` (float32 ``(sum len_i, C)``, sequence
``i``'s residues in rows ``offsets[i] .. offsets[i + 1] - 1``) and ``offsets`` (int64, from 0)."""


def batch_tokenize_tiled(tokenizer, batch, window, stride=None, padlen=None, destchar="B", device=None, *, tail="short",
                         varlen=False, rc=None, rc_prob=None, seed=0, crop=None):
    """Tokens of every window of every sequence of ``batch``: stage -> tile -> reverse complement -> tokenize, on the
    device.  A :class:`TiledTokens`.

    Windows as :func:`tile_packed` cuts them (``stride`` defaults to ``window``; ``tail`` ``"short"``, ``"end"`` or
    ``"drop"``).  ``varlen=False``: a padded ``(rows, padlen)`` tensor, one row per window as ``batch_tokenize(...,
    batch_first=True)`` writes it; ``padlen`` defaults to ``window + bos + eos`` and may not be smaller.  ``varlen=True``:
    a :class:`VarlenBatch` (``padlen`` must not be given).  ``rc`` / ``rc_prob`` / ``seed``: the windows are flipped as
    :func:`batch_tokenize_revcomp` does, with the coins keyed by window index; ``"both"`` gives ``2M`` rows, the windows
    and then their reverse complements -- the layout :func:`untile` averages over.  A tile is a crop, so ``crop`` is
    rejected.  Host batches are sized from their host offsets without synchronising; CUDA batches pay one read-back,
    which also validates their offsets."""
    torch = _torch()
    if crop is not None:
        raise ValueError("batch_tokenize_tiled: a tile is already a crop of the sequence; crop cannot be combined with it")
    tok = descriptor(tokenizer)
    kind, dtype = _dtype_of(destchar)
    window, stride, tail_code = _tile_spec(window, stride, tail)
    k = int(tokenizer.includes_bos()) + int(tokenizer.includes_eos())
    padlen = _padlen("batch_tokenize_tiled", padlen, varlen, window + k)
    if not varlen and padlen < window + k:
        raise ValueError(f"padlen {padlen} is shorter than window + bos + eos = {window + k}")
    rc = _rc_spec(rc, rc_prob, seed, 0, tokenizer)
    strands = 2 if rc is not None and rc[0] == capi.RC_BOTH else 1
    extent = []
    seq_offsets = []

    def checked(e):
        if varlen:
            _check_cu_seqlens(strands * (e[1] + e[0] * k))
        return e

    def before_stage(h_offs, n):
        h = np.ascontiguousarray(h_offs[:n + 1], dtype=np.int64)
        extent.extend(checked(capi.tile_extent_host(h, n, window, stride, tail_code)))
        seq_offsets.append(h - h[0] if n >= 0 else h)

    r = _resolve(batch, device, before_stage=before_stage)
    try:
        dev = torch.device("cuda", r.device)
        if r.h_offs is None:  # a CUDA batch: one reduction and read-back, which also validates its offsets
            b, o = batch
            extent = checked(capi.tile_extent_device(r.device, r.stream, o, r.nseq, window, stride, tail_code, nbytes=b.numel()))
            so = o - o[:1]
        else:
            so = torch.from_numpy(seq_offsets[0]).to(dev)
        M, nbytes, longest = extent
        tb = _tile_into(dev, r.stream, r.d_bytes, r.d_offs, r.nseq, window, stride, tail_code, M, nbytes)
        r.d_bytes, r.d_offs, r.nseq, r.h_offs = tb.bytes.data_ptr(), tb.offsets.data_ptr(), M, None  # r: the windows
        flipped = None if rc is None else _apply_rc(r, rc, nbytes, flipped=True)
        if varlen:
            tokens = torch.empty(strands * nbytes + r.nseq * k, dtype=dtype, device=dev)
            cu_seqlens = torch.empty(r.nseq + 1, dtype=torch.int32, device=dev)
            capi.tokenize_varlen(r.device, r.stream, r.d_bytes, r.d_offs, r.nseq, tok, kind, tokens, cu_seqlens)
            tokens = VarlenBatch(tokens, cu_seqlens, longest + k if r.nseq > 0 else 0)
        else:
            tokens = torch.empty((r.nseq, padlen), dtype=dtype, device=dev)
            if r.nseq > 0:
                capi.tokenize(r.device, r.stream, r.d_bytes, r.d_offs, r.nseq, padlen, tok, True, kind, tokens)
        return TiledTokens(tokens, tb.seq_index, tb.starts, tb.seq_ptr, so, flipped, strands, window, stride, tail,
                           int(tokenizer.includes_bos()))
    finally:
        r.release()


_UNTILE_DTYPES = None


def untile(values, tiled, *, col0=None):
    """The per-residue mean of model outputs over every window (and strand) that covers each residue: an
    :class:`UntiledBatch`.

    ``values``: the outputs for ``tiled.tokens`` (a :class:`TiledTokens`), float32, bfloat16 or float16, contiguous, on the
    tokens' device: ``(rows, P, C)`` or ``(rows, P)`` (C = 1) for padded tokens (``P >= col0 + window``), ``(T, C)`` or
    ``(T,)`` for a :class:`VarlenBatch` of ``T`` tokens.  Position ``col0 + t`` of a window's row (``col0`` defaults to
    ``tiled.bos``) is its residue ``t``; in a flipped window that is residue ``len - 1 - t`` of the window's span.  The sum
    runs in float32 in a fixed order (strand 0 before strand 1, windows in ascending order), so the result is
    deterministic; a residue no window covers (``tail="drop"``) gets NaN.  The exact rule is documented with
    ``bsq_untile_mean`` in include/bsq.h.  One synchronisation: the residue count is read back."""
    global _UNTILE_DTYPES
    torch = _torch()
    if _UNTILE_DTYPES is None:
        _UNTILE_DTYPES = {torch.float32: capi.UNTILE_F32, torch.bfloat16: capi.UNTILE_BF16, torch.float16: capi.UNTILE_F16}
    if not isinstance(tiled, TiledTokens):
        raise ValueError("untile: tiled must be the TiledTokens of batch_tokenize_tiled")
    if not isinstance(values, torch.Tensor) or values.dtype not in _UNTILE_DTYPES:
        raise ValueError("untile: values must be a float32, bfloat16 or float16 tensor")
    if not values.is_contiguous():
        raise ValueError("untile: values must be contiguous")
    varlen = isinstance(tiled.tokens, VarlenBatch)
    tokens = tiled.tokens.tokens if varlen else tiled.tokens
    if values.device != tokens.device:
        raise ValueError("untile: values must live on the tokens' device")
    try:
        col0 = tiled.bos if col0 is None else operator.index(col0)
    except TypeError:
        raise ValueError("col0 must be an integer") from None
    if col0 < 0:
        raise ValueError(f"col0 must be >= 0, got {col0}")
    rows = tiled.seq_index.numel() * tiled.strands
    if varlen:
        if values.dim() not in (1, 2) or values.shape[0] != tokens.numel():
            raise ValueError(f"untile: padding-free values must be (T,) or (T, C) with T = {tokens.numel()}, got {tuple(values.shape)}")
        C, stride, cu = (values.shape[1] if values.dim() == 2 else 1), 0, tiled.tokens.cu_seqlens
    else:
        if values.dim() not in (2, 3) or values.shape[0] != rows:
            raise ValueError(f"untile: padded values must be (rows, P) or (rows, P, C) with rows = {rows}, got {tuple(values.shape)}")
        C, stride, cu = (values.shape[2] if values.dim() == 3 else 1), values.shape[1], None
        if stride < col0 + tiled.window:
            raise ValueError(f"untile: P = {stride} is shorter than col0 + window = {col0 + tiled.window}")
    if C < 1:
        raise ValueError("untile: values have no channels")
    dev = values.device
    n = tiled.seq_ptr.numel() - 1
    R = int(tiled.seq_offsets[-1].item()) if n > 0 else 0
    out = torch.empty((R, C), dtype=torch.float32, device=dev)
    if n > 0 and R > 0:
        flipped = tiled.flipped.view(torch.uint8) if tiled.flipped is not None else None
        capi.untile_mean(dev.index, torch.cuda.current_stream(dev.index).cuda_stream, _UNTILE_DTYPES[values.dtype], values, C,
                         stride, cu, col0, tiled.seq_offsets, n, tiled.window, tiled.stride, _TILE_TAILS[tiled.tail], tiled.seq_ptr,
                         tiled.seq_index.numel(), tiled.strands, flipped, out)
    return UntiledBatch(out, tiled.seq_offsets)


TranslatedBatch = collections.namedtuple("TranslatedBatch", ["bytes", "offsets", "seq_index", "frame", "frames"])
TranslatedBatch.__doc__ = """The reading frames of a packed DNA batch, as a packed protein batch: ``bytes`` (uint8 amino-acid letters,
``*`` for stops, ``X`` where a codon is ambiguous or holds an invalid byte) and ``offsets`` (int64, from 0) of the ``n F``
output sequences, sequence-major; ``seq_index`` (int64, one per output sequence: ``w // F``, its input sequence); ``frame``
(int8, one per output sequence: ``frames[w % F]``); ``frames`` (the tuple of the F frames)."""


def translate_packed(bytes_cuda, offsets_cuda, *, frames=1, genetic_code=1):
    """Translate every sequence of a packed CUDA DNA / RNA batch into the reading frames ``frames``: a
    :class:`TranslatedBatch`; the input is not modified.

    ``frames``: one of 1, 2, 3, -1, -2, -3 (frame +k reads from offset k - 1, frame -k the reverse complement from offset
    k - 1), a list or tuple of distinct ones (kept in that order), ``"forward"`` = (1, 2, 3) or ``"six"`` = (1, 2, 3, -1,
    -2, -3).  Output sequence ``w = i * F + f`` is frame ``frames[f]`` of sequence ``i``, ``(len - k + 1) // 3`` amino acids
    long (a trailing partial codon is dropped; sequences shorter than 3 give empty rows).  ``genetic_code``: an NCBI
    table id (1 standard, 2 vertebrate mitochondrial, 4 mold / protozoan mitochondrial, 5 invertebrate mitochondrial, 6
    ciliate, 11 bacterial) or 64 letters in TCAG order.  Residues are case-insensitive IUPAC codes (U = T); a codon whose
    expansions all give one amino acid gives it, any other gives ``X``.  The exact rule is documented with
    ``bsq_translate`` in include/bsq.h.  ``(tb.bytes, tb.offsets)`` is a packed CUDA batch that every consumer takes with a
    protein tokenizer.  One synchronisation: the offsets are validated and the output's size is read back."""
    torch = _torch()
    _packed_cuda("translate_packed", bytes_cuda, offsets_cuda)
    fr, code = _translate_spec(frames, genetic_code)
    n, F = _nseq(offsets_cuda), len(fr)
    dev = bytes_cuda.device
    stream = torch.cuda.current_stream(dev.index).cuda_stream
    total, _, _ = capi.translate_extent_device(dev.index, stream, offsets_cuda, n, fr, nbytes=bytes_cuda.numel())
    out_b = torch.empty(max(total, 1), dtype=torch.uint8, device=dev)
    out_o = torch.empty(n * F + 1, dtype=torch.int64, device=dev)
    src = bytes_cuda if bytes_cuda.numel() > 0 else out_b  # (an all-empty batch: nothing is read)
    capi.translate(dev.index, stream, src, offsets_cuda, n, fr, code, out_b, out_o)
    seq_index = torch.arange(n, dtype=torch.int64, device=dev).repeat_interleave(F)
    frame = torch.tensor(fr, dtype=torch.int8, device=dev).repeat(n)
    return TranslatedBatch(out_b[:total], out_o, seq_index, frame, fr)


def batch_tokenize_translated(tokenizer, batch, padlen=None, destchar="B", device=None, *, frames=1, genetic_code=1, varlen=False,
                              crop=None, crop_len=None, seed=0, seq_index_base=0, augment=0, augment_frac=1.0):
    """Tokens of the reading frames of every DNA / RNA sequence of ``batch``: stage -> translate -> crop -> augment ->
    tokenize, on the device.

    ``frames`` / ``genetic_code``: as :func:`translate_packed`; row ``w = i * F + f`` is frame ``frames[f]`` of sequence
    ``i``.  ``tokenizer``: a protein alphabet (PROTEIN, AMINO20 and the reduced ones) or BYTES.  PROTEIN / AMINO20 have no
    ``*`` or ``X``, so stops and ambiguous codons tokenize as every invalid byte does (id 0).  ``varlen=False``: a padded
    ``(n F, padlen)`` tensor as ``batch_tokenize(..., batch_first=True)`` writes it; ``padlen`` defaults to the longest
    translated (and cropped) row + bos + eos.  ``varlen=True``: a :class:`VarlenBatch` (``padlen`` must not be given).
    ``crop`` / ``crop_len`` (in amino acids; default ``padlen - bos - eos``, required without ``padlen``) and ``augment``
    (BLOSUM62, on the proteins) as for the other consumers, with seeded draws keyed by the output index
    ``(seq_index_base + i) * F + f``.  Host batches are sized from their host offsets without synchronising; CUDA batches
    pay one read-back, which also validates their offsets."""
    torch = _torch()
    tok = descriptor(tokenizer)
    kind, dtype = _dtype_of(destchar)
    tr = _translate_spec(frames, genetic_code, tokenizer, None, seq_index_base)
    base = _out_base(seq_index_base, tr)
    augment = _augment_args(augment, augment_frac, seed, base)
    padlen = _padlen("batch_tokenize_translated", padlen, varlen)
    if padlen is not None and padlen < 1:
        raise ValueError(f"padlen must be >= 1, got {padlen}")
    if varlen or padlen is None:
        if crop is not None and crop_len is None:
            raise ValueError("batch_tokenize_translated: crop without padlen needs an explicit crop_len")
        crop = _crop_spec(crop, crop_len, seed, base)
    else:
        crop = _crop_spec(crop, crop_len, seed, base, _row_residues(tokenizer, padlen))
    if varlen:
        return _tokenize_varlen(tokenizer, batch, destchar, device, augment, crop=crop, translate=tr)
    r = _resolve(batch, device, augment, crop=crop, translate=tr)
    try:
        k = int(tokenizer.includes_bos()) + int(tokenizer.includes_eos())
        if padlen is None:
            padlen = r.extent[1] + k
        out = torch.empty((r.nseq, padlen), dtype=dtype, device=torch.device("cuda", r.device))
        if r.nseq > 0 and padlen > 0:
            _check_lengths(r, padlen, tok, onehot=False)
            capi.tokenize(r.device, r.stream, r.d_bytes, r.d_offs, r.nseq, padlen, tok, True, kind, out)
        return out
    finally:
        r.release()
