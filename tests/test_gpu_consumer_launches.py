"""Kernel launches and outputs of every public consumer, per batch form and option, pinned to integer literals.

Every offset reduction in libbsq (the length check, the crop, k-mer, tile and varlen extents) is one launch that ends
in one stream synchronise, so the launch count of a call pins its read-backs: host batches (numpy arrays, FlatFile
ranges, lists of items) never synchronise, and a CUDA batch pays exactly one read-back (two for cropped k-mers; sequence
packing reads CUDA offsets back through torch, which launches nothing of libbsq's).  The output of every form must be
the same, and equal to the digest recorded here."""
import hashlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from bioseq_b200 import capi, cbioseq, consumers  # noqa: E402
from oracle.oracle import flatfile_image  # noqa: E402

SEQS = [b"ACGTACGTNNACGTTGCA", b"", b"GATTACA" * 10, b"acgtRYKMSWbdhvN", b"T"]
P = 80  # padlen and seqpack's row_len: every sequence fits uncropped
NONE = {}
CROP = dict(crop="random", crop_len=12, seed=3)
RC = dict(rc="random", seed=5)
CROP_RC = dict(crop="random", crop_len=12, rc="random", seed=7)
AUG = dict(augment=2, augment_frac=0.5, seed=9)
BOTH = dict(rc="both")
OPTS = {"none": NONE, "crop": CROP, "rc": RC, "crop+rc": CROP_RC, "augment": AUG, "both": BOTH}


def _tok():
    return cbioseq.Tokenizer("DNA", bos=True, eos=True, padchar=True)


def _weight():
    return torch.arange(_tok().alphabet_size() * 4, dtype=torch.float32, device="cuda").reshape(-1, 4)


CONSUMERS = {
    "onehot": (lambda b, **o: consumers.batch_onehot_encode_bcl(_tok(), b, P, "B", **o),
               ["none", "crop", "rc", "crop+rc", "augment", "both"]),
    "embed": (lambda b, **o: consumers.batch_embed(_tok(), b, _weight(), P, **o), ["none", "crop", "rc", "crop+rc", "augment", "both"]),
    "augmented": (lambda b, **o: consumers.batch_tokenize_augmented(_tok(), b, P, **o), ["augment"]),
    "cropped": (lambda b, **o: consumers.batch_tokenize_cropped(_tok(), b, P, **o), ["none", "crop", "crop+rc"]),
    "revcomp": (lambda b, **o: consumers.batch_tokenize_revcomp(_tok(), b, P, **o), ["none", "rc", "crop+rc", "both"]),
    "varlen": (lambda b, **o: consumers.batch_tokenize_varlen(_tok(), b, **o), ["none", "crop", "rc", "crop+rc", "both"]),
    "mlm": (lambda b, **o: consumers.batch_tokenize_mlm(_tok(), b, P, **o), ["none", "crop", "rc", "crop+rc", "augment"]),
    "mlm_varlen": (lambda b, **o: consumers.batch_tokenize_mlm(_tok(), b, varlen=True, **o), ["none", "crop", "rc", "crop+rc", "augment"]),
    "seqpack": (lambda b, **o: consumers.batch_tokenize_seqpack(_tok(), b, P, **o), ["none", "crop", "rc", "crop+rc", "augment", "both"]),
    "seqpack_mlm": (lambda b, **o: consumers.batch_tokenize_seqpack(_tok(), b, P, mlm=True, **o),
                    ["none", "crop", "rc", "crop+rc", "augment"]),
    "kmer": (lambda b, **o: consumers.batch_tokenize_kmer(_tok(), b, 3, P, **o), ["none", "crop", "rc", "crop+rc", "both"]),
    "kmer_varlen": (lambda b, **o: consumers.batch_tokenize_kmer(_tok(), b, 3, varlen=True, **o), ["none", "crop", "rc", "crop+rc", "both"]),
    "tiled": (lambda b, **o: consumers.batch_tokenize_tiled(_tok(), b, 16, 8, **o), ["none", "rc", "both"]),
    "tiled_varlen": (lambda b, **o: consumers.batch_tokenize_tiled(_tok(), b, 16, 8, varlen=True, **o), ["none", "rc", "both"]),
}
# the packed entry points take CUDA tensors only
PACKED = {
    "crop_packed-head": lambda b, o: consumers.crop_packed(b, o, 12, crop="head"),
    "crop_packed-random": lambda b, o: consumers.crop_packed(b, o, 12, seed=3),
    "revcomp_packed-always": lambda b, o: consumers.revcomp_packed(b, o),
    "revcomp_packed-random": lambda b, o: consumers.revcomp_packed(b, o, rc="random", seed=5),
    "revcomp_packed-both": lambda b, o: consumers.revcomp_packed(b, o, rc="both"),
    "tile_packed": lambda b, o: consumers.tile_packed(b, o, 16, stride=8, tail="end"),
}
CASES = [f"{name}-{opt}" for name, (_, opts) in CONSUMERS.items() for opt in opts] + list(PACKED)

# case -> (launches with a CUDA batch, launches with each host form (None: CUDA only), digest of the output), measured
# once on a B200: a change to any of them changes what a call launches, synchronises or computes
EXPECTED = {
    "onehot-none": (2, 1, "08f1c5d1f9a21d8b"),
    "onehot-crop": (4, 3, "1ab64c6ec7e22743"),
    "onehot-rc": (3, 2, "746ec744287fa8b1"),
    "onehot-crop+rc": (5, 4, "7acf627bc9b427ff"),
    "onehot-augment": (3, 2, "f2645d3caf8a9f11"),
    "onehot-both": (3, 2, "93b432b197ef2a85"),
    "embed-none": (2, 1, "20f59286cbab9873"),
    "embed-crop": (4, 3, "c1e7270f946d0ca0"),
    "embed-rc": (3, 2, "a440ca94aec5f8bd"),
    "embed-crop+rc": (5, 4, "209a31acd388f7d2"),
    "embed-augment": (3, 2, "68403b531be84f03"),
    "embed-both": (3, 2, "d4a5bbb8ee95e2d9"),
    "augmented-augment": (3, 2, "1772080b1ab09771"),
    "cropped-none": (4, 3, "bb620c7628f6447a"),
    "cropped-crop": (4, 3, "3ffd0be4dab6b556"),
    "cropped-crop+rc": (5, 4, "3e627092cb0149b1"),
    "revcomp-none": (3, 2, "718df636a740e6e1"),
    "revcomp-rc": (3, 2, "3e818b263e619cc2"),
    "revcomp-crop+rc": (5, 4, "3e627092cb0149b1"),
    "revcomp-both": (3, 2, "341318c4af715688"),
    "varlen-none": (2, 1, "a82ed8cbf0899f41"),
    "varlen-crop": (4, 3, "4756d092b1593197"),
    "varlen-rc": (3, 2, "69d84d630d2e331b"),
    "varlen-crop+rc": (5, 4, "19a81a77d77daef1"),
    "varlen-both": (3, 2, "3ca1f5bd051b4dc6"),
    "mlm-none": (2, 1, "639355c7d3c271be"),
    "mlm-crop": (4, 3, "6c1c3eb24c340fdf"),
    "mlm-rc": (3, 2, "9bd937cc12ffb9a8"),
    "mlm-crop+rc": (5, 4, "fd4d2eed6ed605bd"),
    "mlm-augment": (3, 2, "04d746508805e283"),
    "mlm_varlen-none": (2, 1, "f1337f4961f5b450"),
    "mlm_varlen-crop": (4, 3, "918f327abcd0ce87"),
    "mlm_varlen-rc": (3, 2, "37d246c13b9929bf"),
    "mlm_varlen-crop+rc": (5, 4, "37df1b106f73dcd1"),
    "mlm_varlen-augment": (3, 2, "78d8e65c19f05f72"),
    "seqpack-none": (1, 1, "e63083329e64adbd"),
    "seqpack-crop": (3, 3, "bf14e74f7d2cc7b6"),
    "seqpack-rc": (2, 2, "37928396b3f0b5cf"),
    "seqpack-crop+rc": (4, 4, "8cd81f74d4b6060f"),
    "seqpack-augment": (2, 2, "e2aabd137f5d276e"),
    "seqpack-both": (2, 2, "a666870f7dfca824"),
    "seqpack_mlm-none": (1, 1, "a44be09947114606"),
    "seqpack_mlm-crop": (3, 3, "b72cca36557288ec"),
    "seqpack_mlm-rc": (2, 2, "c93d4b92428b4678"),
    "seqpack_mlm-crop+rc": (4, 4, "991a299e79fb7bfa"),
    "seqpack_mlm-augment": (2, 2, "df3797aedac5e511"),
    "kmer-none": (2, 1, "383760fcf04dc374"),
    "kmer-crop": (5, 3, "93c2542d364cfa84"),
    "kmer-rc": (3, 2, "23037948ff14bc4e"),
    "kmer-crop+rc": (6, 4, "6a3c1fc3cb49238e"),
    "kmer-both": (3, 2, "2bc92d681e4f8450"),
    "kmer_varlen-none": (3, 2, "cbf54fdd747d6fd5"),
    "kmer_varlen-crop": (6, 4, "9b83d569c5d7b605"),
    "kmer_varlen-rc": (4, 3, "6b2d1070e8d90e44"),
    "kmer_varlen-crop+rc": (7, 5, "533b0b7abfeb4431"),
    "kmer_varlen-both": (4, 3, "60497343a2b5c3cf"),
    "tiled-none": (5, 4, "74bda253abb0f8a6"),
    "tiled-rc": (6, 5, "90ee5637572624ee"),
    "tiled-both": (6, 5, "dd0c590a7021a938"),
    "tiled_varlen-none": (5, 4, "ee08a78fbb397e9b"),
    "tiled_varlen-rc": (6, 5, "f3986018ded0c1f9"),
    "tiled_varlen-both": (6, 5, "4a57d3086a755482"),
    "crop_packed-head": (3, None, "cc7fdc7ea9c6acae"),
    "crop_packed-random": (3, None, "509a1314e77103ad"),
    "revcomp_packed-always": (2, None, "8e3d975f2f29992f"),
    "revcomp_packed-random": (2, None, "62b55395ca16bf40"),
    "revcomp_packed-both": (2, None, "66fc649e92936833"),
    "tile_packed": (4, None, "365fbe4594953d1f"),
}


def batches(tmp_dir):
    """The batch in every form: CUDA tensors, host numpy, a FlatFile range (offsets[0] != 0) and a list of bytes."""
    offs = np.zeros(len(SEQS) + 1, np.int64)
    np.cumsum([len(s) for s in SEQS], out=offs[1:])
    buf = np.frombuffer(b"".join(SEQS), np.uint8).copy()
    path = tmp_dir / "launches.ff"
    path.write_bytes(flatfile_image([b"GGGCCC"] + SEQS))
    ff = cbioseq.FlatFile(str(path))
    return {"cuda": (torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda()), "host": (buf, offs),
            "flatfile": (ff, 1, 1 + len(SEQS)), "list": list(SEQS)}


def digest(out):
    """SHA-256 over every tensor (dtype, shape, bytes) and every other field (repr) of a consumer's output."""
    h = hashlib.sha256()

    def feed(x):
        if isinstance(x, torch.Tensor):
            a = x.detach().cpu().contiguous()
            h.update(f"{a.dtype}{tuple(a.shape)}".encode())
            h.update(a.numpy().tobytes())
        elif isinstance(x, tuple):
            for v in x:
                feed(v)
        else:
            h.update(repr(x).encode())

    feed(out)
    return h.hexdigest()[:16]


def measure(case, forms):
    """-> {form: (launch count of one call, digest of its output)} for every form the case takes."""
    lib = capi.lib()
    res = {}
    if case in PACKED:
        calls = {"cuda": lambda: PACKED[case](*forms["cuda"])}
    else:
        name, opt = case.split("-", 1)
        fn, _ = CONSUMERS[name]
        calls = {form: (lambda b=b: fn(b, **OPTS[opt])) for form, b in forms.items()}
    for form, call in calls.items():
        before = lib.bsq_launch_count()
        out = call()
        launches = lib.bsq_launch_count() - before
        torch.cuda.synchronize()
        res[form] = (launches, digest(out))
    return res


@pytest.fixture(scope="module")
def forms(tmp_path_factory):
    if not torch.cuda.is_available():
        pytest.fail("GPU tests selected but no CUDA device is visible")
    return batches(tmp_path_factory.mktemp("launches"))


def test_every_case_is_pinned():
    assert sorted(EXPECTED) == sorted(CASES)


@pytest.mark.parametrize("case", CASES)
def test_launches_and_output(case, forms):
    cuda_launches, host_launches, want = EXPECTED[case]
    got = measure(case, forms)
    assert got.pop("cuda") == (cuda_launches, want)
    for form, (launches, d) in got.items():
        assert (form, launches, d) == (form, host_launches, want)
