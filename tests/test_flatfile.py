"""FlatFile (SURVEY 8f row 1): the on-disk packed store that feeds the path.

CPU: the file writer/reader of libbsq (bsq_flatfile_*) and the `cbioseq.FlatFile` class against
(1) tests/golden/flatfile.json -- exact bytes the reference's FlatFile wrote for each input,
(2) the Python restatement in oracle/oracle.py, (3) on random inputs, the reference's outputs
recorded in tests/golden/reference.json, and the compiled reference itself when oracle/_ref is
present.  GPU: batches taken straight from a FlatFile (mapped and pinned) against the oracle
tokenizer on the same sequences.
"""
import gzip
import json
import os
import random

import numpy as np
import pytest

from bioseq_b200 import cbioseq
from oracle.oracle import parse_fastx, flatfile_image, load_ref, OracleTokenizer, pack
from oracle.fastx_cases import cases, random_fastx
from helpers import Reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ff_golden():
    with open(os.path.join(ROOT, "tests", "golden", "flatfile.json")) as f:
        return json.load(f)


def write_input(tmp_path, name, data, gz=False):
    p = str(tmp_path / (name + (".gz" if gz else "")))
    with (gzip.open if gz else open)(p, "wb") as f:
        f.write(data)
    return p


def test_restatement_matches_golden(ff_golden):
    assert [c["input"].encode("latin-1") for c in ff_golden] == cases(), "case generator drifted"
    for c in ff_golden:
        seqs = parse_fastx(c["input"].encode("latin-1"))
        assert [s.decode("latin-1") for s in seqs] == c["seqs"], c["input"]
        assert flatfile_image(seqs).hex() == c["ff_hex"], c["input"]


def test_writer_and_reader_match_golden(ff_golden, tmp_path):
    for i, c in enumerate(ff_golden):
        src = write_input(tmp_path, f"c{i}.fa", c["input"].encode("latin-1"), c["gz"])
        dst = str(tmp_path / f"c{i}.ff")
        ff = cbioseq.FlatFile(src, dst)
        assert open(dst, "rb").read().hex() == c["ff_hex"], c["input"]
        assert (ff.nseqs(), len(ff), ff.size(), ff.seq_offset(), ff.maxseqlen, ff.max_seq_len, ff.path) == \
            (c["nseqs"], c["nseqs"], c["nseqs"], c["seq_offset"], c["maxseqlen"], c["maxseqlen"], dst)
        assert [bytes(x).decode("latin-1") for x in ff.access(0, ff.nseqs())] == c["seqs"]
        assert cbioseq.getstats([src])[0].tolist() == c["lens"]
        assert cbioseq.getstats([src])[0].dtype == np.uint64
        re = cbioseq.FlatFile(dst)           # reopen: maxseqlen from a scan of the offsets
        assert re.maxseqlen == c["maxseqlen"] and re.nseqs() == c["nseqs"]
        assert re.indptr().dtype == np.uint64
        assert re.indptr().tolist() == np.concatenate([[0], np.cumsum(c["lens"])]).astype(int).tolist()


def test_default_output_path_and_errors(tmp_path):
    src = write_input(tmp_path, "x.fa", b">a\nACGT\n>b\nGG\n")
    ff = cbioseq.FlatFile(src, "")
    assert ff.path == src + ".ff" and os.path.exists(src + ".ff")
    with pytest.raises(RuntimeError, match="No such file or directory"):
        cbioseq.FlatFile(str(tmp_path / "missing.ff"))
    with pytest.raises(RuntimeError, match="missing.fa failed to open"):
        cbioseq.FlatFile(str(tmp_path / "missing.fa"), str(tmp_path / "o.ff"))
    with pytest.raises(RuntimeError, match="could not be opened for writing"):
        cbioseq.FlatFile(src, str(tmp_path / "no_such_dir" / "o.ff"))
    with pytest.raises(IndexError, match="Accessing sequence out of range"):
        ff.access(2)
    with pytest.raises(IndexError, match="For a negative index"):
        ff[-3]
    with pytest.raises(ValueError, match="step must be nonzero"):
        ff.access(0, 2, 0)
    # a file that is not a FlatFile is rejected instead of read out of bounds
    bad = write_input(tmp_path, "bad.ff", np.uint64(1 << 40).tobytes() + b"\0" * 64)
    with pytest.raises(RuntimeError, match="not a FlatFile"):
        cbioseq.FlatFile(bad)
    short = write_input(tmp_path, "short.ff", b"\1\0\0")
    with pytest.raises(RuntimeError, match="not a FlatFile"):
        cbioseq.FlatFile(short)
    # maxseqlen given by the caller is trusted (src/fxstats.cpp:69)
    assert cbioseq.FlatFile(src + ".ff", 99).maxseqlen == 99
    assert cbioseq.FlatFile(src + ".ff", maxseqlen=-1).maxseqlen == 4


def test_access_forms(tmp_path):
    seqs = [b"ACGT", b"", b"GGA", b"T", b"CCCCCC"]
    src = write_input(tmp_path, "y.fa", b"".join(b">s\n" + s + b"\n" for s in seqs))
    ff = cbioseq.FlatFile(src, str(tmp_path / "y.ff"))
    assert [bytes(ff[i]) for i in range(5)] == seqs
    assert isinstance(ff[0], bytearray)
    assert bytes(ff[-1]) == seqs[-1] and bytes(ff[-5]) == seqs[0]
    assert [bytes(x) for x in ff[1:4]] == seqs[1:4]
    assert [bytes(x) for x in ff[::2]] == seqs[::2]
    assert [bytes(x) for x in ff.access(slice(0, 5, 2))] == seqs[::2]
    assert [bytes(x) for x in ff.access(4, 0, -2)] == [seqs[4], seqs[2]]
    assert [bytes(x) for x in ff.access(start=1, stop=3)] == seqs[1:3]
    assert [bytes(x) for x in ff[np.array([3, 0, 3])]] == [seqs[3], seqs[0], seqs[3]]
    # iteration protocol of the reference: __next__ advances first and yields the iterator itself
    it = iter(ff)
    assert isinstance(it, cbioseq.FlatFileIterator)
    assert [bytes(x.seq) for x in ff] == seqs[1:]
    assert [bytes(x.sequence) for x in ff] == seqs[1:]
    # zero-copy packed views
    b, o = ff.packed()
    assert b.dtype == np.uint8 and o.dtype == np.int64 and not b.flags.writeable
    assert b.tobytes() == b"".join(seqs) and o.tolist() == [0, 4, 4, 7, 8, 14]
    b2, o2 = ff.packed(2, 4)
    assert o2.tolist() == [4, 7, 8] and b2.tobytes() == b.tobytes()
    with pytest.raises(IndexError):
        ff.packed(3, 9)


def test_against_compiled_reference(tmp_path):
    R = load_ref()
    rec = Reference("test_flatfile::test_against_compiled_reference", R)
    rng = random.Random(7)

    def walk(f):
        try:
            return [bytes(x.seq) for x in f]
        except IndexError:   # the reference's iterator never meets its end on an empty file; mirrored
            return "IndexError"

    for i in range(300):
        data = random_fastx(rng)
        gz = i % 7 == 0
        src = write_input(tmp_path, "r.fa", data, gz)
        a, b = str(tmp_path / "ref.ff"), str(tmp_path / "our.ff")

        def ref_file():
            R.FlatFile(src, a)   # written out when the object goes
            return open(a, "rb").read()

        ours = cbioseq.FlatFile(src, b)
        rec.check(open(b, "rb").read(), ref_file)
        assert open(b, "rb").read() == flatfile_image(parse_fastx(data)), data
        ref = R and R.FlatFile(a)
        rec.check((ours.nseqs(), ours.seq_offset(), ours.maxseqlen), lambda: (ref.nseqs(), ref.seq_offset(), ref.maxseqlen))
        rec.check(ours.access(0, ours.nseqs()), lambda: ref.access(0, ref.nseqs()))
        rec.check(walk(ours), lambda: walk(ref))
        rec.check(cbioseq.getstats([src])[0].tolist(), lambda: R.getstats([src])[0].tolist())
        if gz:
            os.remove(src)
    rec.done()


# ------------------------------------------------------------------------------------------ GPU
def _protein_file(tmp_path, n=3000, lo=0, hi=700, seed=11):
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWYacdxXBZ*", dtype=np.uint8)
    seqs = [alpha[rng.integers(0, alpha.size, size=int(l))].tobytes() for l in rng.integers(lo, hi, size=n, endpoint=True)]
    lines = []
    for i, s in enumerate(seqs):
        lines.append(b">sp|%d| some protein\n" % i)
        lines += [s[k:k + 60] + b"\n" for k in range(0, len(s), 60)]
    src = write_input(tmp_path, "prot.fa", b"".join(lines))
    return src, seqs


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True])
def test_gpu_flatfile_batches(tmp_path, pinned):
    import torch
    import bioseq_b200
    src, seqs = _protein_file(tmp_path)
    ff = cbioseq.FlatFile(src, str(tmp_path / "prot.ff"), pinned=pinned)
    assert ff.pinned == pinned and ff.nseqs() == len(seqs)
    tok = bioseq_b200.pbeos_tokenizers["PROTEIN"]
    ora = OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    P = ff.maxseqlen + 2

    def same(want, got):
        got = got.cpu().numpy()
        assert want.shape == got.shape and want.tobytes() == got.tobytes()

    # whole file, default padlen = longest + bos + eos
    same(ora.batch_tokenize(pack(seqs), padlen=P, batch_first=True), tok.batch_tokenize_flatfile(ff, batch_first=True))
    same(ora.batch_tokenize(pack(seqs), padlen=P, batch_first=True), tok.batch_tokenize(ff, batch_first=True))
    same(ora.batch_tokenize(pack(seqs), padlen=P), tok.batch_tokenize_flatfile(ff))
    # ranges, including empty and unaligned starts, explicit padlen and wide dtypes
    for a, b in ((0, 0), (0, 1), (1, 130), (777, 2049), (2999, 3000), (128, 3000)):
        same(ora.batch_tokenize(pack(seqs[a:b]), padlen=P + 5, batch_first=True),
             tok.batch_tokenize_flatfile(ff, a, b, padlen=P + 5, batch_first=True))
        same(ora.batch_tokenize(pack(seqs[a:b]), padlen=P, destchar="i"),
             tok.batch_tokenize_flatfile(ff, start=a, stop=b, destchar="i"))
    same(ora.batch_onehot_encode(pack(seqs[5:300]), padlen=P), tok.batch_onehot_encode_flatfile(ff, 5, 300))
    # mask covers the whole file's residues
    total = sum(len(s) for s in seqs)
    m = (np.random.default_rng(3).random(total) < 0.8).astype(np.uint8)
    offs = np.concatenate([[0], np.cumsum([len(s) for s in seqs])])
    want = ora.batch_onehot_encode(pack(seqs[40:400]), padlen=P, destchar="f",
                                   mask=[m[offs[i]:offs[i + 1]] for i in range(40, 400)])
    same(want, tok.batch_onehot_encode_flatfile(ff, 40, 400, destchar="f", mask=m))
    # the packed views feed the packed entry point as well
    b, o = ff.packed(100, 900)
    same(ora.batch_tokenize(pack(seqs[100:900]), padlen=P, batch_first=True),
         tok.batch_tokenize_packed(b, o, padlen=P, batch_first=True))
    # errors keep the reference's text
    with pytest.raises(RuntimeError, match="seq len \\+ bos \\+ eos > padlen"):
        tok.batch_tokenize_flatfile(ff, padlen=ff.maxseqlen + 1)
    with pytest.raises(IndexError):
        tok.batch_tokenize_flatfile(ff, 10, 5)
    torch.cuda.synchronize()


def test_pyviewff(tmp_path):
    from bioseq_b200 import PyViewFF
    seqs = [b"ACGT", b"", b"GGA", b"T"]
    src = write_input(tmp_path, "v.fa", b"".join(b">s\n" + s + b"\n" for s in seqs))
    cbioseq.FlatFile(src, str(tmp_path / "v.ff"))
    v = PyViewFF(str(tmp_path / "v.ff"))
    assert len(v) == 4 and [v[i] for i in range(4)] == seqs and v[1:3] == seqs[1:3]


@pytest.mark.gpu
def test_gpu_flatfile_open_modes_give_the_same_tokens(tmp_path):
    # plain mapping, prefaulted mapping, mapping page-locked in place (cudaHostRegister; falls back to prefaulted where
    # the platform cannot register file pages) and the pinned copy: same tokens, and `pinned` tells which path was taken
    import torch
    import bioseq_b200
    src, seqs = _protein_file(tmp_path, n=900, hi=300, seed=9)
    cbioseq.FlatFile(src, str(tmp_path / "m.ff"))
    tok = bioseq_b200.pbeos_tokenizers["PROTEIN"]
    outs = []
    for kw in (dict(), dict(prefault=1), dict(prefault=2), dict(pinned=True)):
        ff = cbioseq.FlatFile(str(tmp_path / "m.ff"), **kw)
        assert ff.nseqs() == 900
        if kw.get("pinned"):
            assert ff.pinned
        if not kw or kw.get("prefault") == 1:
            assert not ff.pinned
        outs.append(tok.batch_tokenize_flatfile(ff, 0, None, batch_first=True, destchar="B"))
        assert [bytes(b) for b in ff[3:6]] == seqs[3:6]
        del ff
    for o in outs[1:]:
        assert torch.equal(o, outs[0])


@pytest.mark.gpu
def test_gpu_loaders(tmp_path):
    import torch
    import bioseq_b200
    from bioseq_b200.loaders import FF2NP, FF2Tensor, FlatFileDataset
    src, seqs = _protein_file(tmp_path, n=700, hi=200, seed=5)
    ff = cbioseq.FlatFile(src, str(tmp_path / "l.ff"))
    tok = bioseq_b200.pbeos_tokenizers["PROTEIN"]
    ora = OracleTokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    P = ff.maxseqlen + 2
    want = ora.batch_tokenize(pack(seqs), padlen=P, batch_first=True).view(np.uint8)
    mm, path = FF2NP(ff, tok, str(tmp_path / "toks.u8"), batch_size=256)
    assert mm.shape == (700, P) and np.array_equal(np.asarray(mm), want)
    assert np.array_equal(FF2Tensor(ff, tok).cpu().numpy(), want)
    ds = FlatFileDataset(ff, tok)
    assert len(ds) == 700 and ds.max_seq_len == P
    assert ds[3].dtype == torch.long and ds[3].shape == (P,) and np.array_equal(ds[3].cpu().numpy(), want[3])
    assert np.array_equal(ds[-1].cpu().numpy(), want[-1])
    assert np.array_equal(ds[10:300].cpu().numpy(), want[10:300])
    assert np.array_equal(torch.cat(list(ds.batches(128))).cpu().numpy(), want)
    # ... with the next two batches tokenised on a side stream while this one is consumed
    got = [b.clone() for b in ds.batches(100, prefetch=2)]
    assert len(got) == 7 and np.array_equal(torch.cat(got).cpu().numpy(), want)
    cnn = FlatFileDataset(ff, tok, cnn=True)
    oh = ora.batch_onehot_encode(pack(seqs[5:9]), padlen=P, destchar="f")        # (P, 4, C)
    got = cnn[5:9]
    assert got.dtype == torch.float32 and got.shape == (4, 23, P)
    assert np.array_equal(got.cpu().numpy(), np.transpose(oh, (1, 2, 0)))
    # a single index is Tokenizer.onehot_encode(seq, padlen=P): bos + eos zero rows on top of padlen (src/tokenize.h:195)
    one = cnn[5].cpu().numpy()
    assert one.shape == (P + 2, 23) and np.array_equal(one[:P], oh[:, 0, :]) and not one[P:].any()
    assert isinstance(cnn, torch.utils.data.Dataset)
    t, items = cnn.fetch(slice(5, 9), return_items=True)             # bioseq/loaders.py:60-84
    assert torch.equal(t, got) and [bytes(b) for b in items] == seqs[5:9]
    t, item = ds.fetch(3, return_items=True)
    assert torch.equal(t, ds[3]) and bytes(item) == seqs[3] and torch.equal(ds.fetch(3), ds[3])
    assert got.is_contiguous()          # written in (batch, emb, length) layout, not a permuted view
    aug = FlatFileDataset(ff, tok, augment=2, augment_frac=1.0)      # on-device BLOSUM62 augmentation (test_gpu_consumers.py)
    a = aug[0:700].cpu().numpy()
    nd = (a != want).sum(1)
    assert a.shape == want.shape and nd.max() <= 2 and nd.mean() > 1.8
