"""FlatFile callers of the tokenizer, GPU-fed (reference: bioseq/loaders.py:11-115, bioseq/__init__.py:198-219).

The reference's loaders pull one Python ``bytearray`` per sequence out of the FlatFile, tokenise
on the CPU and move the numpy result to the device.  Here a range of the file goes to the GPU as
packed bytes + offsets (``Tokenizer.batch_tokenize_flatfile``), so no per-sequence host work is
left.  BLOSUM62 augmentation (``augment=``; bioseq/blosum.py:63-87) runs on the device between the copy and
the tokeniser (``consumers``; Philox streams keyed by the dataset seed, the draw number and the sequence index),
and ``cnn=True`` batches are written directly in the ``(batch, emb, length)`` float layout.  ``max_seq_len=`` crops
over-long sequences on the device (``consumers.crop_packed``) so that a file with a few very long sequences still
yields batches of the model's context, and ``rc="random"`` flips DNA sequences to their reverse complement on the device
(``consumers.revcomp_packed``).  ``translate=`` reads protein rows out of a DNA file: each sequence's reading frames
are translated on the device (``consumers.translate_packed``) before the crop.
"""
import numpy as np

from . import cbioseq
from . import consumers


def FF2NP(x, tokenizer, destfile, *, batch_size=8192, device=None):
    """Tokenise a whole FlatFile into an ``np.memmap`` of shape (nseqs, maxseqlen + bos + eos), uint8
    (bioseq/loaders.py:11-26).  Rows are produced on the GPU ``batch_size`` sequences at a time.

    The reference passes ``padlen=maxseqlen`` while sizing rows ``maxseqlen + bos + eos``, which only
    works without BOS/EOS; the row width is used as padlen here."""
    assert isinstance(x, cbioseq.FlatFile)
    assert isinstance(tokenizer, cbioseq.Tokenizer)
    total_msl = x.maxseqlen + tokenizer.includes_bos() + tokenizer.includes_eos()
    nseqs = x.nseqs()
    retmat = np.memmap(destfile, mode='w+', dtype=np.uint8, shape=(nseqs, total_msl))
    for start in range(0, nseqs, batch_size):
        stop = min(start + batch_size, nseqs)
        toks = tokenizer.batch_tokenize_flatfile(x, start, stop, padlen=total_msl, batch_first=True, destchar='B',
                                                 device=device)
        retmat[start:stop] = toks.cpu().numpy()
    return (retmat, destfile)


def FF2Tensor(x, tokenizer, *, batch_first=True, destchar='B', device=None):
    """The whole FlatFile as one token tensor resident on the GPU (one staged pass over the file)."""
    return tokenizer.batch_tokenize_flatfile(x, 0, None, batch_first=batch_first, destchar=destchar, device=device)


def _dataset_base():
    import torch.utils.data
    return torch.utils.data.Dataset


class FlatFileDataset(_dataset_base()):
    """Map-style ``torch.utils.data.Dataset`` over a FlatFile and a Tokenizer (bioseq/loaders.py:29-115).

    ``ds[i]`` -> 1-D ``long`` token tensor of length ``max_seq_len``; ``ds[a:b]`` -> ``(b-a, max_seq_len)``.
    With ``cnn=True`` a slice is a one-hot ``float`` tensor laid out ``(batch, emb, length)`` and a single index is
    what ``Tokenizer.onehot_encode(seq, padlen=max_seq_len)`` gives the reference (bioseq/loaders.py:101-103):
    ``(max_seq_len + bos + eos, emb)`` -- the single-sequence encoder adds BOS/EOS rows ON TOP of padlen
    (src/tokenize.h:195), so with a BOS/EOS tokenizer a single item is longer than a slice's rows, as in the reference.
    Tensors live on ``device``.

    With ``varlen=True`` a slice is a ``consumers.VarlenBatch`` -- the ``long`` tokens of its sequences back to back,
    without padding, plus ``cu_seqlens`` and ``max_seqlen`` (what varlen attention takes) -- and a single index is that
    sequence's unpadded 1-D ``long`` tokens.

    With ``mlm=True`` items are masked-language-model batches (``consumers.MLMBatch(inputs, labels)``, one kernel per
    fetch): a slice gives ``long`` inputs padded to ``max_seq_len`` (or a ``VarlenBatch`` with ``varlen=True``) and int64
    labels of the same shape, a single index the 1-D pair.  ``maskfrac`` of the residues are selected, 80 / 10 / 10
    masked (id ``alphabet_size()``) / randomised / kept, labels ``-100`` elsewhere.  Like augmentation, every fetch is a
    new draw: the mask is keyed by the dataset seed, the draw number and the sequence's index in the file.

    ``max_seq_len=L`` makes rows ``L`` wide whatever the file holds: every sequence is cropped on the device to a window of
    at most ``L - bos - eos`` residues before augmentation, masking or tokenization (the padding-free forms use the same
    window length).  ``crop="random"`` (the default) draws a new window every fetch from the same per-fetch seed as
    augmentation and masking (ESM-style); ``crop="head"`` keeps the first residues (truncation).  Without
    ``max_seq_len`` rows are as wide as the file's longest sequence and nothing is cropped.

    With ``seqpack=True`` a slice is a ``consumers.SeqPackBatch``: its sequences packed whole, best-fit, into as few rows of
    ``max_seq_len`` as they need, with ``long`` tokens, position ids that restart per sequence and ``cu_seqlens`` (and
    labels with ``mlm=True``); a single index is the same with one row.  Crop, augmentation and masking draw from the
    per-fetch seed as above.  ``seqpack=True`` cannot be combined with ``varlen=True`` or ``cnn=True``.

    ``rc="random"`` (nucleotide tokenizers, not with ``augment``) flips each sequence to its reverse complement with
    probability ``rc_prob`` after the crop and before masking or tokenization: strand augmentation, usually together with
    ``crop="random"`` as the random shift.  Like the crop, every fetch is a new draw from the per-fetch seed.  Datasets
    are for training, so the inference modes (``"always"``, ``"both"``) are rejected: call the consumers directly.

    ``translate=frames`` (with ``genetic_code``, as ``consumers.batch_tokenize_translated``; a protein tokenizer) turns a
    DNA file into protein rows: F frames per sequence, so a slice ``[start, stop)`` yields ``(stop - start) * F`` rows, and a
    single index F rows (a 1-D row when F = 1, as without translation).  The default ``max_seq_len`` is then
    ``maxseqlen // 3 + bos + eos``; ``max_seq_len`` crops the proteins, and every seeded draw is keyed by the output row
    ``(index * F + f)``.  Not with ``rc`` (the reverse frames are the other strand).

    ``fetch(index, return_items=True)`` also hands back the raw sequence(s) (bioseq/loaders.py:60-84), as stored in the
    file: uncropped and unflipped, like they are unaugmented.  Two quirks of
    the reference's ``fetch`` are NOT reproduced: with ``cnn=True`` and ``return_items=False`` it falls off the end and
    returns ``None``, and without ``cnn`` it ignores ``return_items``; here both modes honour the flag.
    """

    def __init__(self, ff, tokenizer, *, augment=0, augment_frac=0.5, cnn=False, device=None, maskfrac=0.15, seed=13,
                 varlen=False, mlm=False, max_seq_len=None, crop="random", seqpack=False, rc=None, rc_prob=0.5, translate=None, genetic_code=1):
        super().__init__()
        assert isinstance(ff, cbioseq.FlatFile)
        assert isinstance(tokenizer, cbioseq.Tokenizer)
        if varlen and cnn:
            raise ValueError("FlatFileDataset: varlen=True yields tokens, cnn=True one-hot; choose one")
        if mlm and cnn:
            raise ValueError("FlatFileDataset: mlm=True yields masked tokens and labels, cnn=True one-hot; choose one")
        if seqpack and (varlen or cnn):
            raise ValueError("FlatFileDataset: seqpack=True yields packed fixed-width rows; it cannot be combined with varlen=True "
                             "or cnn=True")
        self.varlen, self.mlm, self.seqpack = bool(varlen), bool(mlm), bool(seqpack)
        self.ff, self.tokenizer = ff, tokenizer
        self.seed, self._draw = int(seed), 0  # the reference seeds its generator with 13 (bioseq/loaders.py:49-50)
        self.maskfrac, self.augment, self.augment_frac, self.cnn, self.device = maskfrac, augment, augment_frac, cnn, device
        k = tokenizer.includes_bos() + tokenizer.includes_eos()
        self.tr = consumers._translate_spec(translate, genetic_code, tokenizer, rc)  # ValueError now rather than per fetch
        self.translate, self.genetic_code = translate, genetic_code
        self.crop, self.crop_len = None, None
        if max_seq_len is None:
            self.max_seq_len = (ff.maxseqlen // 3 if self.tr else ff.maxseqlen) + k
        else:
            if crop not in ("head", "random"):
                raise ValueError(f"FlatFileDataset: crop must be 'head' or 'random', got {crop!r}")
            if max_seq_len < k + 1:
                raise ValueError(f"FlatFileDataset: max_seq_len {max_seq_len} leaves no room for a residue next to bos + eos")
            self.max_seq_len, self.crop, self.crop_len = int(max_seq_len), crop, int(max_seq_len) - k
        self.maxseqlen = self.max_seq_len
        if rc not in (None, "random"):
            raise ValueError(f"FlatFileDataset: rc must be None or 'random' (a dataset is for training), got {rc!r}")
        consumers._rc_spec(rc, rc_prob if rc else None, 0, 0, tokenizer, augment)  # ValueError now rather than per fetch
        self.rc, self.rc_prob = rc, rc_prob

    def _range(self, index):
        n = len(self)
        if isinstance(index, slice):
            start, stop, step = index.indices(n)
            if step != 1:
                raise IndexError("FlatFileDataset: only contiguous slices go to the GPU as one range")
            return start, max(start, stop), True
        index = int(index)
        if index < 0:
            index += n
        if not 0 <= index < n:
            raise IndexError("Accessing sequence out of range")
        return index, index + 1, False

    def _augment_kwargs(self, start):
        """Every fetch is a new draw (the reference's generator advances per item, bioseq/loaders.py:71-73);
        within a draw a sequence's stream depends on its index in the file only."""
        self._draw += 1
        return dict(augment=self.augment, augment_frac=self.augment_frac, seq_index_base=start,
                    seed=(self.seed & 0xFFFFFFFF) | ((self._draw & 0xFFFFFFFF) << 32))

    def __getitem__(self, index):
        import torch
        start, stop, many = self._range(index)
        crop = dict(crop=self.crop, crop_len=self.crop_len) if self.crop else {}
        rc = dict(rc=self.rc, rc_prob=self.rc_prob) if self.rc else {}
        tr = dict(translate=self.translate, genetic_code=self.genetic_code) if self.tr else {}
        F = len(self.tr[0]) if self.tr else 1
        if self.seqpack:
            kw = self._augment_kwargs(start) if self.mlm or self.augment or self.crop or self.rc else {}
            mlm = dict(mlm=True, maskfrac=self.maskfrac, mask_token=self.tokenizer.alphabet_size()) if self.mlm else {}
            return consumers.batch_tokenize_seqpack(self.tokenizer, (self.ff, start, stop), self.max_seq_len, "l", self.device,
                                                    rows=None if many or F > 1 else 1, **mlm, **kw, **crop, **rc, **tr)
        if self.mlm:
            # one draw per fetch, shared by the augmentation (counter word 3 = 0), the mask (words 1, 2), the crop (3) and the
            # strand flip (4)
            kw = self._augment_kwargs(start)
            mb = consumers.batch_tokenize_mlm(self.tokenizer, (self.ff, start, stop),
                                              padlen=-1 if self.varlen else self.max_seq_len, destchar="l",
                                              device=self.device, varlen=self.varlen, maskfrac=self.maskfrac,
                                              mask_token=self.tokenizer.alphabet_size(), **kw, **crop, **rc, **tr)
            if many or (F > 1 and not self.varlen):
                return mb
            return consumers.MLMBatch(mb.inputs.tokens if self.varlen else mb.inputs[0], mb.labels if self.varlen else mb.labels[0])
        aug = self._augment_kwargs(start) if self.augment or self.crop or self.rc else {}
        if self.cnn:
            if many:  # (batch, emb, length) float, written in that layout by one kernel
                return consumers.batch_onehot_encode_bcl(self.tokenizer, (self.ff, start, stop), padlen=self.max_seq_len,
                                                         destchar='f', device=self.device, **aug, **crop, **rc, **tr)
            if tr:  # F (length, emb) items
                oh = consumers.batch_onehot_encode_bcl(self.tokenizer, (self.ff, start, stop), padlen=self.max_seq_len,
                                                       destchar='f', device=self.device, **aug, **crop, **tr).transpose(1, 2)
                return oh[0] if F == 1 else oh
            if aug:
                # (mutated, cropped or flipped on the device: the batched path at padlen = max_seq_len; such a sequence is no
                # longer than before, so only the reference's extra bos + eos pad rows of the single-sequence encoder are
                # missing here)
                return consumers.batch_onehot_encode_bcl(self.tokenizer, (self.ff, start, stop), padlen=self.max_seq_len,
                                                         destchar='f', device=self.device, **aug, **crop, **rc)[0].t()
            return self.tokenizer.onehot_encode(bytes(self.ff[start]), padlen=self.max_seq_len, destchar='f', device=self.device)
        if self.varlen:
            base = consumers._out_base(start, self.tr)  # (the global index of the first output row)
            vb = consumers._tokenize_varlen(self.tokenizer, (self.ff, start, stop), "l", self.device,
                                            consumers._augment_args(**dict(aug, seq_index_base=base)) if aug else None,
                                            crop=consumers._crop_spec(self.crop, self.crop_len, aug.get("seed", 0), base)
                                            if crop else None,
                                            rc=consumers._rc_spec(self.rc, self.rc_prob, aug.get("seed", 0), start) if rc else None,
                                            translate=self.tr)
            return vb if many else vb.tokens
        if tr:
            kw = dict(seed=aug.get("seed", 0), seq_index_base=start, augment=self.augment, augment_frac=self.augment_frac)
            toks = consumers.batch_tokenize_translated(self.tokenizer, (self.ff, start, stop), self.max_seq_len, 'B', self.device,
                                                       frames=self.translate, genetic_code=self.genetic_code, **kw,
                                                       **crop).to(torch.long)
            return toks if many or F > 1 else toks[0]
        if crop:
            toks = consumers.batch_tokenize_cropped(self.tokenizer, (self.ff, start, stop), self.max_seq_len, batch_first=True,
                                                    destchar='B', device=self.device, **aug, **crop, **rc).to(torch.long)
            return toks if many else toks[0]
        if rc:
            seed = dict(seed=aug["seed"], seq_index_base=start)
            toks = consumers.batch_tokenize_revcomp(self.tokenizer, (self.ff, start, stop), self.max_seq_len, batch_first=True,
                                                    destchar='B', device=self.device, **seed, **rc).to(torch.long)
            return toks if many else toks[0]
        if aug:
            toks = consumers.batch_tokenize_augmented(self.tokenizer, (self.ff, start, stop), padlen=self.max_seq_len,
                                                      batch_first=True, destchar='B', device=self.device, **aug).to(torch.long)
        else:
            toks = self.tokenizer.batch_tokenize_flatfile(self.ff, start, stop, padlen=self.max_seq_len, batch_first=True,
                                                          destchar='B', device=self.device).to(torch.long)
        return toks if many else toks[0]

    def fetch(self, index, return_items=False):
        """``ds[index]``, and with ``return_items`` the sequence(s) it was made from (bioseq/loaders.py:60-84): the
        ``bytearray`` of a single index, a list of them for a slice -- what ``FlatFile.__getitem__`` returns.  With
        augmentation the items are the sequences as stored in the file (mutation happens on the device)."""
        ret = self[index]
        if not return_items:
            return ret
        start, stop, many = self._range(index)
        return ret, (self.ff[start:stop] if many else self.ff[start])

    def access(self, slc, stop=None, step=None):
        if isinstance(slc, int):
            slc = slice(slc, stop, step)
        return self[slc]

    def batches(self, batch_size, prefetch=0):
        """Consecutive ``(batch, max_seq_len)`` token batches (``VarlenBatch``es with ``varlen=True``, ``MLMBatch``es with
        ``mlm=True``, ``SeqPackBatch``es of ``batch_size`` sequences with ``seqpack=True``) covering the file.

        ``prefetch=k`` (k > 0) keeps k batches ahead of the consumer on a side stream: the host-to-device copy and the
        tokeniser of batch i+1 .. i+k run while the caller's stream is still busy with batch i (the reference's
        training loops, training/cnnpretrain.py:119-128, tokenise on the CPU between optimizer steps).  Every yielded
        tensor is ready on the caller's current stream."""
        if prefetch <= 0:
            for start in range(0, len(self), batch_size):
                yield self[start:start + batch_size]
            return
        import collections
        import torch
        dev = torch.device("cuda", torch.cuda.current_device()) if self.device is None else torch.device(self.device)
        if dev.type != "cuda":
            raise ValueError("FlatFileDataset.batches(prefetch=...): a CUDA device is needed")
        side = torch.cuda.Stream(device=dev)
        ahead = collections.deque()

        def record(x, cur):
            if isinstance(x, torch.Tensor):
                x.record_stream(cur)  # (allocated on the side stream, used on the caller's)
            elif isinstance(x, tuple):  # VarlenBatch, MLMBatch(VarlenBatch, labels), SeqPackBatch (int / None fields skipped)
                for y in x:
                    record(y, cur)

        def hand_over(item):
            t, ev = item
            cur = torch.cuda.current_stream(dev)
            cur.wait_event(ev)
            record(t, cur)
            return t

        for start in range(0, len(self), batch_size):
            side.wait_stream(torch.cuda.current_stream(dev))  # nothing the caller enqueued so far is overtaken
            with torch.cuda.stream(side):
                t = self[start:start + batch_size]
                ev = torch.cuda.Event()
                ev.record(side)
            ahead.append((t, ev))
            if len(ahead) > prefetch:
                yield hand_over(ahead.popleft())
        while ahead:
            yield hand_over(ahead.popleft())

    def __len__(self):
        return self.ff.nseqs()

    def cleanup(self):
        pass


class AugmentedSeqDataset(FlatFileDataset):
    """bioseq/loaders.py:117-119."""

    def __init__(self, ff, tokenizer, augment=1, augment_frac=.5, **kw):
        super().__init__(ff, tokenizer, augment=augment, augment_frac=augment_frac, **kw)


class PyViewFF:
    """Pure-numpy view of a FlatFile (bioseq/__init__.py:198-219)."""

    def __init__(self, path):
        fp = np.memmap(path, mode='r', dtype=np.uint8)
        self.nseqs = int(fp[:8].view(np.uint64)[0])
        self.offsets = fp[8:8 * (2 + self.nseqs)].view(np.uint64)
        self.seqs = fp[8 * (2 + self.nseqs):]
        self.fp = fp

    def access(self, idx):
        return bytes(self.seqs[int(self.offsets[idx]):int(self.offsets[idx + 1])])

    def __getitem__(self, idx):
        if isinstance(idx, int):
            return self.access(idx)
        if isinstance(idx, slice):
            return [self.access(i) for i in range(*idx.indices(self.nseqs))]
        raise ValueError("PyViewFF can only support slices and integers.")

    def __len__(self):
        return self.nseqs
