"""bioseq_b200 -- B200-native batch tokenisation with the Python surface of dnbaker/bioseq.

Mirrors the tokenizer part of ``bioseq/__init__.py`` of the reference (lines 36-168): the
compiled ``cbioseq.Tokenizer`` class, the pre-made tokenizers, the
``bos/eos/beos/pbos/peos/pos/pbeos_tokenizers`` dictionaries keyed by alphabet name (upper- and
lower-case), ``total_tokenizer_dict``, ``get_tokenizer_dict``, ``onehot_encode``, ``f_encode``,
``make_embedding`` and ``torchify`` keep their names, arguments and defaults.  What changes is
where the work happens: ``batch_tokenize`` / ``batch_onehot_encode`` / ``decode_tokens`` run as
hand-written sm_100a CUDA kernels and hand back torch CUDA tensors.

There is no CPU fallback: importing this package needs the compiled extension
(``python -m bioseq_b200.build``) and calling a batch method needs a CUDA device.
"""
import os as _os
import sys as _sys

try:
    from . import cbioseq
except ImportError as _e:  # pragma: no cover - exercised only on a broken checkout
    if "bioseq_b200.build" in getattr(_sys, "orig_argv", ()):
        # `python -m bioseq_b200.build` on a checkout whose extension is missing or stale: let the build script run
        _sys.exit(__import__("runpy").run_path(_os.path.join(_os.path.dirname(_os.path.abspath(__file__)), "build.py"),
                                               run_name="__main__") and 0)
    raise ImportError(
        "bioseq_b200: the compiled extension is missing (%s). Build it with "
        "`python -m bioseq_b200.build`; there is no pure-Python or CPU fallback." % (_e,)) from _e

from .cbioseq import Tokenizer, Threading, set_num_threads, get_num_threads  # noqa: F401
from .cbioseq import FlatFile, FlatFileIterator, getstats  # noqa: F401

LIBBSQ_PATH = _os.path.join(_os.path.dirname(_os.path.abspath(__file__)), "libbsq.so")


def onehot_encode(tokenizer, seqbatch, padlen=-1, destchar='B', batch_first=False, to_pytorch=False, device=None):
    """One-hot encode one sequence or a batch (reference: bioseq/__init__.py:36-66).

    A str/bytes ``seqbatch`` goes to ``Tokenizer.onehot_encode``; anything else is a batch for
    ``Tokenizer.batch_onehot_encode`` whose ``(seq, batch, base)`` result is returned as a
    ``(batch, seq, base)`` view when ``batch_first``.  Results already are torch CUDA tensors, so
    ``to_pytorch`` is accepted for compatibility and ``device`` selects the CUDA device.
    """
    if isinstance(seqbatch, (str, bytes)):
        res = tokenizer.onehot_encode(seqbatch, padlen, destchar, device=device)
    else:
        res = tokenizer.batch_onehot_encode(seqbatch, padlen, destchar, device=device)
        if batch_first:
            res = res.permute(1, 0, 2)
    return res


def f_encode(seqbatch, key="DNA", bos=False, eos=False, padchar=False, padlen=-1, destchar='B', batch_first=False,
             to_pytorch=False, device=None):
    """Functional form: build a Tokenizer for ``key`` and one-hot encode with it
    (reference: bioseq/__init__.py:69-116)."""
    tokenizer = Tokenizer(key, bos=bos, eos=eos, padchar=padchar)
    return onehot_encode(tokenizer, seqbatch, padlen=padlen, destchar=destchar, batch_first=batch_first,
                         to_pytorch=to_pytorch, device=device)


# reference: bioseq/__init__.py:119-120 (SEB6 is listed twice there as well)
keys = ("SEB6", "SEB8", "SEB10", "SEV10", "MURPHY", "LIA10", "LIB10", "SEB6", "DAYHOFF", "DNA4", "DNA", "DNA5",
        "KETO", "PURPYR", "BYTES", "AMINO20", "PROTEIN")
bkeys = keys + tuple(k.lower() for k in keys)

DNATokenizer = Tokenizer("DNA")
AmineTokenizer = Tokenizer("AMINO20")
Reduced6Tokenizer = Tokenizer("SEB6")
Reduced8Tokenizer = Tokenizer("SEB8")
Reduced10Tokenizer = Tokenizer("SEB10")
Reduced14Tokenizer = Tokenizer("SEB14")
DayhoffTokenizer = Tokenizer("DAYHOFF")
LIATokenizer = Tokenizer("LIA10")
LIBTokenizer = Tokenizer("LIB10")
default_tokenizers = {
    "DNA": DNATokenizer, "AMINO20": AmineTokenizer, "AMINE": AmineTokenizer, "PROTEIN": AmineTokenizer,
    "SEB6": Reduced6Tokenizer, "SEB8": Reduced8Tokenizer, "SEB10": Reduced10Tokenizer, "SEB14": Reduced14Tokenizer,
    "LIA10": LIATokenizer, "LIA": LIATokenizer, "LIB10": LIBTokenizer, "LIB": LIBTokenizer,
}


def _family(bos, eos, padchar):
    return {k: Tokenizer(k, bos=bos, eos=eos, padchar=padchar) for k in bkeys}


pbeos_tokenizers = _family(True, True, True)
beos_tokenizers = _family(True, True, False)
pbos_tokenizers = _family(True, False, True)
bos_tokenizers = _family(True, False, False)
peos_tokenizers = _family(False, True, True)
eos_tokenizers = _family(False, True, False)
pos_tokenizers = _family(False, False, True)
total_tokenizer_dict = {(b, e, p, k): Tokenizer(k.upper(), bos=b, eos=e, padchar=p)
                        for b in (0, 1) for e in (0, 1) for p in (0, 1) for k in bkeys}


def get_tokenizer_dict(bos, eos, padchar):
    """The pre-made dictionary for a (bos, eos, padchar) combination (bioseq/__init__.py:159-168)."""
    if bos:
        if eos:
            return pbeos_tokenizers if padchar else beos_tokenizers
        return pbos_tokenizers if padchar else bos_tokenizers
    if eos:
        return peos_tokenizers if padchar else eos_tokenizers
    return pos_tokenizers if padchar else default_tokenizers


def make_embedding(tok, embdim, maxnorm=None, norm_type=2.0, scale_grad_by_freq=False, sparse=False, _weight=None):
    """``nn.Embedding`` sized for a tokenizer, pad id as ``padding_idx`` (bioseq/__init__.py:171-188)."""
    assert norm_type >= 1., f"{norm_type} is not >= 1., so it is not a norm."
    import torch.nn as nn
    return nn.Embedding(tok.alphabet_size(), embdim, padding_idx=tok.pad() if tok.is_padded() else None,
                        scale_grad_by_freq=scale_grad_by_freq, sparse=sparse, _weight=_weight)


def torchify(arr):
    """numpy -> torch (bioseq/__init__.py:191-195); tensors pass through unchanged."""
    import torch
    return arr if isinstance(arr, torch.Tensor) else torch.from_numpy(arr)


from . import consumers  # noqa: E402
from . import loaders  # noqa: E402
from .loaders import PyViewFF  # noqa: E402
from .consumers import batch_onehot_encode_bcl, batch_embed, augment_packed, batch_tokenize_augmented  # noqa: E402
from .consumers import batch_tokenize_varlen, VarlenBatch  # noqa: E402
from .consumers import batch_tokenize_mlm, MLMBatch  # noqa: E402
from .consumers import crop_packed, batch_tokenize_cropped, CroppedBatch  # noqa: E402
from .consumers import batch_tokenize_seqpack, SeqPackBatch  # noqa: E402
from .consumers import batch_tokenize_kmer, kmer_ids, kmer_vocab, KmerIds  # noqa: E402
from .consumers import revcomp_packed, batch_tokenize_revcomp, RevCompBatch  # noqa: E402
from .consumers import tile_packed, batch_tokenize_tiled, untile, TiledBatch, TiledTokens, UntiledBatch  # noqa: E402
from .consumers import translate_packed, batch_tokenize_translated, TranslatedBatch  # noqa: E402


def __getattr__(name):
    # nn.Module front ends import torch.nn; keep `import bioseq_b200` light
    if name in ("TokenizerLayer", "EmbeddingTokenizerLayer", "layers"):
        import importlib
        layers = importlib.import_module(".layers", __name__)
        return layers if name == "layers" else getattr(layers, name)
    raise AttributeError(name)


__all__ = ["onehot_encode", "cbioseq", "f_encode", "Tokenizer", "make_embedding",
           "bos_tokenizers", "eos_tokenizers", "beos_tokenizers", "pbeos_tokenizers", "peos_tokenizers",
           "pbos_tokenizers", "pos_tokenizers", "default_tokenizers", "total_tokenizer_dict", "get_tokenizer_dict",
           "DNATokenizer", "AmineTokenizer", "Reduced6Tokenizer", "Reduced8Tokenizer", "Reduced10Tokenizer",
           "Reduced14Tokenizer", "DayhoffTokenizer", "LIATokenizer", "LIBTokenizer", "torchify",
           "set_num_threads", "get_num_threads", "Threading", "keys", "bkeys", "FlatFile", "FlatFileIterator", "getstats",
           "PyViewFF", "loaders", "consumers", "batch_onehot_encode_bcl", "batch_embed", "augment_packed",
           "batch_tokenize_augmented", "batch_tokenize_varlen", "VarlenBatch", "batch_tokenize_mlm", "MLMBatch", "crop_packed",
           "batch_tokenize_cropped", "CroppedBatch", "batch_tokenize_seqpack", "SeqPackBatch", "batch_tokenize_kmer", "kmer_ids", "kmer_vocab", "KmerIds",
           "revcomp_packed", "batch_tokenize_revcomp", "RevCompBatch",
           "tile_packed", "batch_tokenize_tiled", "untile", "TiledBatch", "TiledTokens", "UntiledBatch",
           "translate_packed", "batch_tokenize_translated", "TranslatedBatch",
           "TokenizerLayer", "EmbeddingTokenizerLayer"]
