"""ctypes binding of the C ABI in include/bsq.h (libbsq.so).

This is the same boundary the ``cbioseq`` extension sits on; bench.py and the GPU parity tests
use it to drive the kernels with raw device pointers (torch supplies the memory and the stream).
Every wrapper raises the exception type the reference would (ValueError for
``std::invalid_argument``, RuntimeError otherwise) with libbsq's message.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libbsq.so")

OK, ERR_ARG, ERR_TOO_LONG, ERR_BAD_TOKEN, ERR_KEY, ERR_CUDA, ERR_NOMEM, ERR_IO, ERR_RANGE = 0, -1, -2, -3, -4, -5, -6, -7, -8
I8, I16, I32, I64, F32, F64 = range(6)


class MLMDesc(C.Structure):
    """struct bsq_mlm"""
    _fields_ = [("seed", C.c_uint64), ("seq_index_base", C.c_int64), ("t_select", C.c_uint64), ("t_mask", C.c_uint64),
                ("t_random", C.c_uint64), ("mask_id", C.c_int64), ("ignore_index", C.c_int64)]


class KmerDesc(C.Structure):
    """struct bsq_kmer"""
    _fields_ = [("k", C.c_int32), ("stride", C.c_int32), ("tail", C.c_int32), ("nchars", C.c_int32), ("bos", C.c_int32),
                ("eos", C.c_int32), ("padchar", C.c_int32), ("nkmers", C.c_int64), ("unk_id", C.c_int64), ("bos_id", C.c_int64),
                ("eos_id", C.c_int64), ("pad_id", C.c_int64), ("vocab_size", C.c_int64)]


KMER_DROP, KMER_SINGLE = 0, 1
RC_ALWAYS, RC_RANDOM, RC_BOTH = 0, 1, 2
TILE_SHORT, TILE_END, TILE_DROP = 0, 1, 2
UNTILE_F32, UNTILE_BF16, UNTILE_F16 = 0, 1, 2


class TokenizerDesc(C.Structure):
    """struct bsq_tokenizer"""
    _fields_ = [("lut", C.c_int8 * 256), ("nchars", C.c_int32), ("bos_id", C.c_int32), ("eos_id", C.c_int32),
                ("pad_id", C.c_int32), ("padchar", C.c_int32), ("alphabet_size", C.c_int32), ("key", C.c_char * 16)]


_lib = None


def lib():
    """Load libbsq.so (fails loudly: there is no fallback implementation)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -m bioseq_b200.build`")
    L = C.CDLL(LIB_PATH)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int
    tokp = C.POINTER(TokenizerDesc)
    sigs = {
        "bsq_abi_version": (i32, []),
        "bsq_last_error": (C.c_char_p, []),
        "bsq_launch_count": (i64, []),
        "bsq_launch_count_reset": (None, []),
        "bsq_kind_of_destchar": (i32, [C.c_char]),
        "bsq_kind_size": (C.c_size_t, [i32]),
        "bsq_alphabet_count": (i32, []),
        "bsq_alphabet_key": (C.c_char_p, [i32]),
        "bsq_tokenizer_init": (i32, [tokp, C.c_char_p, i32, i32, i32]),
        "bsq_tokenizer_lookup": (i32, [tokp, C.c_int32, C.c_char_p, C.c_size_t]),
        "bsq_pack_create": (i32, [C.POINTER(vp), i32]),
        "bsq_pack_destroy": (None, [vp]),
        "bsq_pack_gather": (i32, [vp, C.POINTER(vp), C.POINTER(i64), i64, i32]),
        "bsq_pack_bytes": (vp, [vp]),
        "bsq_pack_offsets": (vp, [vp]),
        "bsq_pack_nseq": (i64, [vp]),
        "bsq_pack_nbytes": (i64, [vp]),
        "bsq_pack_maxlen": (i64, [vp]),
        "bsq_check_lengths_host": (i32, [vp, i64, i64, tokp]),
        "bsq_check_lengths_device": (i32, [i32, vp, vp, i64, i64, tokp]),
        "bsq_check_offsets_device": (i32, [i32, vp, vp, i64, i64, i64, tokp]),
        "bsq_tokenize": (i32, [i32, vp, vp, vp, i64, i64, tokp, i32, i32, vp]),
        "bsq_onehot": (i32, [i32, vp, vp, vp, vp, i64, i64, tokp, i32, vp]),
        "bsq_decode_lengths": (i32, [i32, vp, vp, i32, i64, i64, i64, i64, tokp, vp, vp, C.POINTER(i64)]),
        "bsq_decode_chars": (i32, [i32, vp, vp, i32, i64, i64, i64, i64, tokp, vp, vp, vp]),
        "bsq_decode_text": (i32, [i32, vp, vp, i32, i64, i64, i64, i64, tokp, vp, vp, vp, i64, C.POINTER(i64)]),
        "bsq_stager_create": (i32, [C.POINTER(vp), i32]),
        "bsq_stager_destroy": (None, [vp]),
        "bsq_stager_sync_copies": (i32, [vp]),
        "bsq_tokenize_host": (i32, [vp, vp, vp, vp, i64, i64, tokp, i32, i32, vp]),
        "bsq_onehot_host": (i32, [vp, vp, vp, vp, vp, i64, i64, tokp, i32, vp]),
        "bsq_tokenize_items": (i32, [vp, vp, vp, C.POINTER(vp), C.POINTER(i64), i64, i64, tokp, i32, i32, vp, i32]),
        "bsq_onehot_items": (i32, [vp, vp, vp, C.POINTER(vp), C.POINTER(i64), i64, i64, tokp, i32, vp, i32]),
        "bsq_parallel_for": (i32, [i32, vp, vp]),
        "bsq_fetch_rows": (i32, [vp, vp, vp, vp, i64, C.POINTER(vp), i32]),
        "bsq_stage_host": (i32, [vp, vp, vp, vp, i64, C.POINTER(vp), C.POINTER(vp)]),
        "bsq_stage_release": (i32, [vp, vp]),
        "bsq_stager_set_augment": (i32, [vp, i32, C.c_double, C.c_uint64, i64]),
        "bsq_onehot_bcl": (i32, [i32, vp, vp, vp, vp, i64, i64, tokp, i32, vp]),
        "bsq_embed": (i32, [i32, vp, vp, vp, i64, i64, tokp, i32, vp, i64, i64, vp]),
        "bsq_augment_blosum62": (i32, [i32, vp, vp, vp, i64, i32, C.c_double, C.c_uint64, i64]),
        "bsq_blosum62_thresholds": (i32, [vp, vp, vp]),
        "bsq_flatfile_make": (i32, [C.c_char_p, C.c_char_p, C.POINTER(i64), C.POINTER(i64)]),
        "bsq_flatfile_open": (i32, [C.POINTER(vp), C.c_char_p, i64, i32]),
        "bsq_flatfile_close": (None, [vp]),
        "bsq_flatfile_nseqs": (i64, [vp]),
        "bsq_flatfile_seq_offset": (i64, [vp]),
        "bsq_flatfile_max_seq_len": (i64, [vp]),
        "bsq_flatfile_offsets": (vp, [vp]),
        "bsq_flatfile_bytes": (vp, [vp]),
        "bsq_flatfile_is_pinned": (i32, [vp]),
        "bsq_fastx_lengths": (i32, [C.c_char_p, C.POINTER(C.POINTER(i64)), C.POINTER(i64)]),
        "bsq_free": (None, [vp]),
        "bsq_tokenize_stream_items": (i32, [vp, vp, i64, vp, vp, vp, i64, tokp, i32, i32, vp, i32]),
        "bsq_onehot_stream_items": (i32, [vp, vp, i64, vp, vp, vp, i64, tokp, i32, vp, i32]),
        "bsq_shard_bounds": (i32, [vp, i64, i32, vp]),
        "bsq_tokenize_host_sharded": (i32, [vp, vp, i32, vp, vp, i64, i64, tokp, i32, i32, i32, vp, vp]),
        "bsq_memcpy_d2d": (i32, [i32, vp, vp, vp, C.c_size_t]),
        "bsq_tokenize_many": (i32, [i32, vp, i32, vp, vp, vp, i64, tokp, i32, i32, vp]),
        "bsq_tokenize_varlen": (i32, [i32, vp, vp, vp, i64, tokp, i32, vp, vp]),
        "bsq_varlen_extent_device": (i32, [i32, vp, vp, i64, i64, tokp, C.POINTER(i64), C.POINTER(i64)]),
        "bsq_tokenize_mlm": (i32, [i32, vp, vp, vp, i64, i64, tokp, i32, C.POINTER(MLMDesc), vp, vp]),
        "bsq_tokenize_varlen_mlm": (i32, [i32, vp, vp, vp, i64, tokp, i32, C.POINTER(MLMDesc), vp, vp, vp]),
        "bsq_crop": (i32, [i32, vp, vp, vp, i64, i64, i32, C.c_uint64, i64, vp, vp, vp]),
        "bsq_crop_extent_device": (i32, [i32, vp, vp, i64, i64, i64, C.POINTER(i64), C.POINTER(i64)]),
        "bsq_seqpack_plan": (i32, [vp, i64, i32, i64, i64, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), vp, vp, vp, vp]),
        "bsq_tokenize_seqpack": (i32, [i32, vp, vp, vp, tokp, i32, i64, i64, vp, vp, vp, vp]),
        "bsq_tokenize_seqpack_mlm": (i32, [i32, vp, vp, vp, tokp, i32, C.POINTER(MLMDesc), i64, i64, vp, vp, vp, vp, vp]),
        "bsq_kmer_init": (i32, [C.POINTER(KmerDesc), tokp, i32, i32, i32]),
        "bsq_tokenize_kmer": (i32, [i32, vp, vp, vp, i64, i64, tokp, C.POINTER(KmerDesc), i32, vp]),
        "bsq_tokenize_kmer_varlen": (i32, [i32, vp, vp, vp, i64, tokp, C.POINTER(KmerDesc), i32, vp, vp]),
        "bsq_kmer_extent_host": (i32, [vp, i64, C.POINTER(KmerDesc), C.POINTER(i64), C.POINTER(i64)]),
        "bsq_kmer_extent_device": (i32, [i32, vp, vp, i64, i64, C.POINTER(KmerDesc), C.POINTER(i64), C.POINTER(i64)]),
        "bsq_revcomp": (i32, [i32, vp, vp, vp, i64, i32, C.c_double, C.c_uint64, i64, vp, vp, vp]),
        "bsq_revcomp_table": (i32, [vp]),
        "bsq_tile_extent_host": (i32, [vp, i64, i64, i64, i32, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
        "bsq_tile_extent_device": (i32, [i32, vp, vp, i64, i64, i64, i64, i32, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
        "bsq_tile": (i32, [i32, vp, vp, vp, i64, i64, i64, i32, vp, vp, vp, vp, vp]),
        "bsq_untile_mean": (i32, [i32, vp, i32, vp, i64, i64, vp, i64, vp, i64, i64, i64, i32, vp, i64, i32, vp, vp]),
        "bsq_genetic_code": (i32, [i32, vp]),
        "bsq_translate_table": (i32, [C.c_char_p, vp, vp]),
        "bsq_translate_extent_host": (i32, [vp, i64, vp, i32, i64, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
        "bsq_translate_extent_device": (i32, [i32, vp, vp, i64, i64, vp, i32, i64, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
        "bsq_translate": (i32, [i32, vp, vp, vp, i64, vp, i32, C.c_char_p, vp, vp]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


EXPORTS = ("bsq_abi_version bsq_last_error bsq_launch_count bsq_launch_count_reset bsq_kind_of_destchar bsq_kind_size "
           "bsq_alphabet_count bsq_alphabet_key bsq_tokenizer_init bsq_tokenizer_lookup bsq_pack_create bsq_pack_destroy "
           "bsq_pack_gather bsq_pack_bytes bsq_pack_offsets bsq_pack_nseq bsq_pack_nbytes bsq_pack_maxlen "
           "bsq_check_lengths_host bsq_check_lengths_device bsq_check_offsets_device bsq_tokenize bsq_onehot bsq_decode_lengths bsq_decode_chars bsq_decode_text "
           "bsq_stager_create bsq_stager_destroy bsq_stager_sync_copies bsq_tokenize_host bsq_onehot_host "
           "bsq_flatfile_make bsq_flatfile_open bsq_flatfile_close bsq_flatfile_nseqs bsq_flatfile_seq_offset "
           "bsq_flatfile_max_seq_len bsq_flatfile_offsets bsq_flatfile_bytes bsq_flatfile_is_pinned bsq_fastx_lengths "
           "bsq_free bsq_stage_host bsq_stage_release bsq_stager_set_augment bsq_onehot_bcl bsq_embed bsq_augment_blosum62 "
           "bsq_blosum62_thresholds bsq_tokenize_items bsq_onehot_items bsq_fetch_rows bsq_parallel_for "
           "bsq_tokenize_stream_items bsq_onehot_stream_items bsq_shard_bounds bsq_tokenize_host_sharded bsq_memcpy_d2d bsq_tokenize_many "
           "bsq_tokenize_varlen bsq_varlen_extent_device bsq_tokenize_mlm bsq_tokenize_varlen_mlm bsq_crop bsq_crop_extent_device "
           "bsq_seqpack_plan bsq_tokenize_seqpack bsq_tokenize_seqpack_mlm bsq_kmer_init bsq_tokenize_kmer bsq_tokenize_kmer_varlen "
           "bsq_kmer_extent_host bsq_kmer_extent_device bsq_revcomp bsq_revcomp_table bsq_tile_extent_host bsq_tile_extent_device "
           "bsq_tile bsq_untile_mean bsq_genetic_code bsq_translate_table bsq_translate_extent_host bsq_translate_extent_device "
           "bsq_translate").split()


def last_error():
    return lib().bsq_last_error().decode("latin-1")


def check(rc, onehot=False):
    if rc == OK:
        return
    msg = last_error()
    if rc == ERR_ARG or (rc == ERR_TOO_LONG and onehot):
        raise ValueError(msg)
    if rc == ERR_RANGE:
        raise IndexError(msg)
    raise RuntimeError(msg)


def tokenizer(key, eos=False, bos=False, padchar=False):
    t = TokenizerDesc()
    check(lib().bsq_tokenizer_init(C.byref(t), key.encode(), int(eos), int(bos), int(padchar)))
    return t


def kind_of(destchar):
    k = lib().bsq_kind_of_destchar(destchar[:1].encode("latin-1") if destchar else b"\0")
    check(min(k, 0))
    return k


def _ptr(x):
    """Raw address of a torch tensor / numpy array / int / None."""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if hasattr(x, "data_ptr"):
        return x.data_ptr()
    return x.ctypes.data


def tokenize(device, stream, d_bytes, d_offsets, nseq, padlen, tok, batch_first, kind, d_out):
    check(lib().bsq_tokenize(device, stream, _ptr(d_bytes), _ptr(d_offsets), nseq, padlen, C.byref(tok),
                             int(batch_first), kind, _ptr(d_out)))


def tokenize_many(device, stream, batches, padlen, tok, batch_first, kind):
    """batches: list of (d_bytes, d_offsets, nseq, d_out).  One launch per group of up to 32 batches (bsq_tokenize_many)."""
    n = len(batches)
    pb = (C.c_void_p * n)(*[_ptr(b[0]) for b in batches])
    po = (C.c_void_p * n)(*[_ptr(b[1]) for b in batches])
    ns = (C.c_int64 * n)(*[int(b[2]) for b in batches])
    pd = (C.c_void_p * n)(*[_ptr(b[3]) for b in batches])
    check(lib().bsq_tokenize_many(device, stream, n, pb, po, ns, padlen, C.byref(tok), int(batch_first), kind, pd))


def tokenize_varlen(device, stream, d_bytes, d_offsets, nseq, tok, kind, d_out, d_cu_seqlens):
    """Packed tokens + int32 cu_seqlens (bsq_tokenize_varlen); d_out holds exactly T elements."""
    check(lib().bsq_tokenize_varlen(device, stream, _ptr(d_bytes), _ptr(d_offsets), nseq, C.byref(tok), kind, _ptr(d_out),
                                    _ptr(d_cu_seqlens)))


def mlm_desc(seed, seq_index_base, thresholds, mask_id, ignore_index):
    """struct bsq_mlm from the integer thresholds (t_select, t_mask, t_random)."""
    ts, tm, tr = thresholds
    return MLMDesc(seed & 0xFFFFFFFFFFFFFFFF, seq_index_base, ts, tm, tr, mask_id, ignore_index)


def tokenize_mlm(device, stream, d_bytes, d_offsets, nseq, padlen, tok, kind, mlm, d_inputs, d_labels):
    """Masked inputs + int64 labels, padded batch-first (bsq_tokenize_mlm); ``mlm``: an MLMDesc."""
    check(lib().bsq_tokenize_mlm(device, stream, _ptr(d_bytes), _ptr(d_offsets), nseq, padlen, C.byref(tok), kind, C.byref(mlm),
                                 _ptr(d_inputs), _ptr(d_labels)))


def tokenize_varlen_mlm(device, stream, d_bytes, d_offsets, nseq, tok, kind, mlm, d_inputs, d_labels, d_cu_seqlens):
    """Masked inputs + int64 labels, padding-free, + int32 cu_seqlens (bsq_tokenize_varlen_mlm)."""
    check(lib().bsq_tokenize_varlen_mlm(device, stream, _ptr(d_bytes), _ptr(d_offsets), nseq, C.byref(tok), kind, C.byref(mlm),
                                        _ptr(d_inputs), _ptr(d_labels), _ptr(d_cu_seqlens)))


def varlen_extent_device(device, stream, d_offsets, nseq, tok, nbytes=-1):
    """-> (T, max_seqlen) of device-resident offsets (bsq_varlen_extent_device: validates them; synchronises)."""
    total, maxlen = C.c_int64(), C.c_int64()
    check(lib().bsq_varlen_extent_device(device, stream, _ptr(d_offsets), nseq, nbytes, C.byref(tok), C.byref(total),
                                         C.byref(maxlen)))
    return total.value, maxlen.value


def crop(device, stream, d_bytes, d_offsets, nseq, crop_len, random, seed, seq_index_base, d_out_bytes, d_out_offsets,
         d_starts=None):
    """Windows of at most crop_len residues per sequence (bsq_crop); ``random``: seeded windows, else the heads."""
    check(lib().bsq_crop(device, stream, _ptr(d_bytes), _ptr(d_offsets), nseq, crop_len, int(bool(random)),
                         seed & 0xFFFFFFFFFFFFFFFF, seq_index_base, _ptr(d_out_bytes), _ptr(d_out_offsets), _ptr(d_starts)))


def crop_extent_device(device, stream, d_offsets, nseq, crop_len, nbytes=-1):
    """-> (sum, max) of min(len_i, crop_len) over device-resident offsets (bsq_crop_extent_device: validates them;
    synchronises)."""
    total, maxlen = C.c_int64(), C.c_int64()
    check(lib().bsq_crop_extent_device(device, stream, _ptr(d_offsets), nseq, nbytes, crop_len, C.byref(total),
                                       C.byref(maxlen)))
    return total.value, maxlen.value


def revcomp(device, stream, d_bytes, d_offsets, nseq, mode, rc_prob, seed, seq_index_base, d_out_bytes, d_out_offsets,
            d_flipped=None):
    """Reverse complement of a packed batch (bsq_revcomp); ``mode``: RC_ALWAYS, RC_RANDOM or RC_BOTH."""
    check(lib().bsq_revcomp(device, stream, _ptr(d_bytes), _ptr(d_offsets), nseq, mode, float(rc_prob), seed & 0xFFFFFFFFFFFFFFFF,
                            seq_index_base, _ptr(d_out_bytes), _ptr(d_out_offsets), _ptr(d_flipped)))


def revcomp_table():
    """The complement table of bsq_revcomp: a uint8 numpy array of 256 entries (no device call)."""
    import numpy as np
    t = np.zeros(256, np.uint8)
    check(lib().bsq_revcomp_table(t.ctypes.data))
    return t


def tile_extent_host(h_offsets, nseq, window, stride, tail):
    """-> (windows, bytes, longest window) of host offsets (bsq_tile_extent_host; no device call)."""
    w, b, m = C.c_int64(), C.c_int64(), C.c_int64()
    check(lib().bsq_tile_extent_host(_ptr(h_offsets), nseq, window, stride, tail, C.byref(w), C.byref(b), C.byref(m)))
    return w.value, b.value, m.value


def tile_extent_device(device, stream, d_offsets, nseq, window, stride, tail, nbytes=-1):
    """-> (windows, bytes, longest window) of device-resident offsets (bsq_tile_extent_device: validates them;
    synchronises)."""
    w, b, m = C.c_int64(), C.c_int64(), C.c_int64()
    check(lib().bsq_tile_extent_device(device, stream, _ptr(d_offsets), nseq, nbytes, window, stride, tail, C.byref(w), C.byref(b),
                                       C.byref(m)))
    return w.value, b.value, m.value


def tile(device, stream, d_bytes, d_offsets, nseq, window, stride, tail, d_out_bytes, d_out_offsets, d_seq_ptr=None,
         d_seq_index=None, d_starts=None):
    """Every window of every sequence (bsq_tile); ``tail``: TILE_SHORT, TILE_END or TILE_DROP."""
    check(lib().bsq_tile(device, stream, _ptr(d_bytes), _ptr(d_offsets), nseq, window, stride, tail, _ptr(d_out_bytes),
                         _ptr(d_out_offsets), _ptr(d_seq_ptr), _ptr(d_seq_index), _ptr(d_starts)))


def untile_mean(device, stream, dtype, d_y, channels, row_stride, d_cu, col0, d_src_offsets, nseq, window, stride, tail, d_seq_ptr,
                nwin, strands, d_flipped, d_out):
    """Per-residue mean of window outputs (bsq_untile_mean); ``dtype``: UNTILE_F32, UNTILE_BF16 or UNTILE_F16."""
    check(lib().bsq_untile_mean(device, stream, dtype, _ptr(d_y), channels, row_stride, _ptr(d_cu), col0, _ptr(d_src_offsets), nseq,
                                window, stride, tail, _ptr(d_seq_ptr), nwin, strands, _ptr(d_flipped), _ptr(d_out)))


def genetic_code(code_id):
    """The built-in genetic code ``code_id`` as 64 bytes in TCAG order (bsq_genetic_code; no device call)."""
    buf = C.create_string_buffer(64)
    check(lib().bsq_genetic_code(code_id, buf))
    return buf.raw


def translate_table(code64):
    """-> (masks, codons): uint8 numpy arrays of 256 and 4096 entries, the rule of bsq_translate (no device call)."""
    import numpy as np
    masks, codons = np.zeros(256, np.uint8), np.zeros(4096, np.uint8)
    check(lib().bsq_translate_table(code64, masks.ctypes.data, codons.ctypes.data))
    return masks, codons


def _frames_arg(frames):
    return (C.c_int8 * max(len(frames), 1))(*frames), len(frames)


_NO_CROP = (1 << 63) - 1


def translate_extent_host(h_offsets, nseq, frames, crop_len=_NO_CROP):
    """-> (total, total after the crop, longest kept row) of host offsets (bsq_translate_extent_host; no device call)."""
    t, c, m = C.c_int64(), C.c_int64(), C.c_int64()
    fa, nf = _frames_arg(frames)
    check(lib().bsq_translate_extent_host(_ptr(h_offsets), nseq, fa, nf, crop_len, C.byref(t), C.byref(c), C.byref(m)))
    return t.value, c.value, m.value


def translate_extent_device(device, stream, d_offsets, nseq, frames, crop_len=_NO_CROP, nbytes=-1):
    """The same of device-resident offsets (bsq_translate_extent_device: validates them; synchronises)."""
    t, c, m = C.c_int64(), C.c_int64(), C.c_int64()
    fa, nf = _frames_arg(frames)
    check(lib().bsq_translate_extent_device(device, stream, _ptr(d_offsets), nseq, nbytes, fa, nf, crop_len, C.byref(t), C.byref(c),
                                            C.byref(m)))
    return t.value, c.value, m.value


def translate(device, stream, d_bytes, d_offsets, nseq, frames, code64, d_out_bytes, d_out_offsets):
    """Reading frames ``frames`` of every sequence under the 64-letter genetic code ``code64`` (bsq_translate)."""
    fa, nf = _frames_arg(frames)
    check(lib().bsq_translate(device, stream, _ptr(d_bytes), _ptr(d_offsets), nseq, fa, nf, code64, _ptr(d_out_bytes),
                              _ptr(d_out_offsets)))


def seqpack_plan(h_offsets, nseq, k, row_len, rows=0, starts=None, row_ptr=None, row_seq=None, cu_seqlens=None):
    """Best-fit-decreasing layout of host offsets in rows of row_len (bsq_seqpack_plan) -> (R, nsegments, max_seqlen).
    Without the four arrays only the sizes are computed; with them (host pointers or arrays: starts[nseq],
    row_ptr[R + 1], row_seq[nseq] int64, cu_seqlens[nsegments + 1] int32) the layout is written as well."""
    R, nseg, mx = C.c_int64(), C.c_int64(), C.c_int64()
    check(lib().bsq_seqpack_plan(_ptr(h_offsets), nseq, k, row_len, rows, C.byref(R), C.byref(nseg), C.byref(mx), _ptr(starts),
                                 _ptr(row_ptr), _ptr(row_seq), _ptr(cu_seqlens)))
    return R.value, nseg.value, mx.value


def tokenize_seqpack(device, stream, d_bytes, d_offsets, tok, kind, row_len, nrows, d_row_ptr, d_row_seq, d_tokens,
                     d_position_ids):
    """(nrows, row_len) tokens + int32 position ids of a plan (bsq_tokenize_seqpack)."""
    check(lib().bsq_tokenize_seqpack(device, stream, _ptr(d_bytes), _ptr(d_offsets), C.byref(tok), kind, row_len, nrows,
                                     _ptr(d_row_ptr), _ptr(d_row_seq), _ptr(d_tokens), _ptr(d_position_ids)))


def tokenize_seqpack_mlm(device, stream, d_bytes, d_offsets, tok, kind, mlm, row_len, nrows, d_row_ptr, d_row_seq, d_inputs,
                         d_position_ids, d_labels):
    """The same with masked inputs + int64 labels (bsq_tokenize_seqpack_mlm); ``mlm``: an MLMDesc."""
    check(lib().bsq_tokenize_seqpack_mlm(device, stream, _ptr(d_bytes), _ptr(d_offsets), C.byref(tok), kind, C.byref(mlm), row_len,
                                         nrows, _ptr(d_row_ptr), _ptr(d_row_seq), _ptr(d_inputs), _ptr(d_position_ids),
                                         _ptr(d_labels)))


def kmer_desc(tok, k, stride=1, tail=KMER_DROP):
    """struct bsq_kmer of a tokenizer descriptor (bsq_kmer_init: ValueError on a bad k, stride, tail or alphabet)."""
    km = KmerDesc()
    check(lib().bsq_kmer_init(C.byref(km), C.byref(tok), k, stride, tail))
    return km


def tokenize_kmer(device, stream, d_bytes, d_offsets, nseq, padlen, tok, km, kind, d_out):
    """(nseq, padlen) k-mer tokens, batch-first (bsq_tokenize_kmer); ``km``: a KmerDesc."""
    check(lib().bsq_tokenize_kmer(device, stream, _ptr(d_bytes), _ptr(d_offsets), nseq, padlen, C.byref(tok), C.byref(km), kind,
                                  _ptr(d_out)))


def tokenize_kmer_varlen(device, stream, d_bytes, d_offsets, nseq, tok, km, kind, d_out, d_cu_seqlens):
    """Padding-free k-mer tokens + int32 cu_seqlens (bsq_tokenize_kmer_varlen)."""
    check(lib().bsq_tokenize_kmer_varlen(device, stream, _ptr(d_bytes), _ptr(d_offsets), nseq, C.byref(tok), C.byref(km), kind,
                                         _ptr(d_out), _ptr(d_cu_seqlens)))


def kmer_extent_host(h_offsets, nseq, km):
    """-> (sum, max) of the k-mer row lengths T(len_i) of host offsets (bsq_kmer_extent_host; no device call)."""
    total, mx = C.c_int64(), C.c_int64()
    check(lib().bsq_kmer_extent_host(_ptr(h_offsets), nseq, C.byref(km), C.byref(total), C.byref(mx)))
    return total.value, mx.value


def kmer_extent_device(device, stream, d_offsets, nseq, km, nbytes=-1):
    """-> (sum, max) of T(len_i) over device-resident offsets (bsq_kmer_extent_device: validates them; synchronises)."""
    total, mx = C.c_int64(), C.c_int64()
    check(lib().bsq_kmer_extent_device(device, stream, _ptr(d_offsets), nseq, nbytes, C.byref(km), C.byref(total), C.byref(mx)))
    return total.value, mx.value


def onehot(device, stream, d_bytes, d_offsets, d_mask, nseq, padlen, tok, kind, d_out):
    check(lib().bsq_onehot(device, stream, _ptr(d_bytes), _ptr(d_offsets), _ptr(d_mask), nseq, padlen, C.byref(tok),
                           kind, _ptr(d_out)), onehot=True)


def onehot_bcl(device, stream, d_bytes, d_offsets, d_mask, nseq, padlen, tok, kind, d_out):
    check(lib().bsq_onehot_bcl(device, stream, _ptr(d_bytes), _ptr(d_offsets), _ptr(d_mask), nseq, padlen, C.byref(tok),
                               kind, _ptr(d_out)), onehot=True)


def embed(device, stream, d_bytes, d_offsets, nseq, padlen, tok, batch_first, d_weight, nrows, row_bytes, d_out):
    check(lib().bsq_embed(device, stream, _ptr(d_bytes), _ptr(d_offsets), nseq, padlen, C.byref(tok), int(batch_first),
                          _ptr(d_weight), nrows, row_bytes, _ptr(d_out)))


def augment_blosum62(device, stream, d_bytes, d_offsets, nseq, chain_len, augment_frac, seed, seq_index_base=0):
    check(lib().bsq_augment_blosum62(device, stream, _ptr(d_bytes), _ptr(d_offsets), nseq, chain_len, float(augment_frac),
                                     seed & 0xFFFFFFFFFFFFFFFF, seq_index_base))


def blosum62_thresholds():
    import numpy as np
    thr, row_of, aa = np.zeros((21, 19), np.uint32), np.zeros(256, np.uint8), np.zeros(20, np.uint8)
    check(lib().bsq_blosum62_thresholds(thr.ctypes.data, row_of.ctypes.data, aa.ctypes.data))
    return thr, row_of, aa


def check_lengths_host(h_offsets, nseq, padlen, tok, onehot=False):
    check(lib().bsq_check_lengths_host(_ptr(h_offsets), nseq, padlen, C.byref(tok)), onehot)


def check_lengths_device(device, stream, d_offsets, nseq, padlen, tok, onehot=False, nbytes=-1):
    check(lib().bsq_check_offsets_device(device, stream, _ptr(d_offsets), nseq, nbytes, padlen, C.byref(tok)), onehot)


def decode_lengths(device, stream, d_tokens, itemsize, rows, cols, row_stride, col_stride, tok, d_row_offsets, d_row_tail=None):
    total = C.c_int64()
    check(lib().bsq_decode_lengths(device, stream, _ptr(d_tokens), itemsize, rows, cols, row_stride, col_stride,
                                   C.byref(tok), _ptr(d_row_offsets), _ptr(d_row_tail), C.byref(total)))
    return total.value


def decode_chars(device, stream, d_tokens, itemsize, rows, cols, row_stride, col_stride, tok, d_row_offsets, d_chars, d_row_tail=None):
    check(lib().bsq_decode_chars(device, stream, _ptr(d_tokens), itemsize, rows, cols, row_stride, col_stride,
                                 C.byref(tok), _ptr(d_row_offsets), _ptr(d_row_tail), _ptr(d_chars)))


def decode_text(device, stream, d_tokens, itemsize, rows, cols, row_stride, col_stride, tok, d_row_offsets, d_row_tail, d_chars, capacity):
    """Both decode passes in one call; returns the total (> capacity: nothing was written, call decode_chars)."""
    total = C.c_int64()
    check(lib().bsq_decode_text(device, stream, _ptr(d_tokens), itemsize, rows, cols, row_stride, col_stride,
                                C.byref(tok), _ptr(d_row_offsets), _ptr(d_row_tail), _ptr(d_chars), capacity, C.byref(total)))
    return total.value


class Stager:
    """bsq_stager: per-device copy stream + staging buffers for the host-staged entry points."""

    def __init__(self, device):
        self.h = C.c_void_p()
        check(lib().bsq_stager_create(C.byref(self.h), device))

    def tokenize_host(self, stream, h_bytes, h_offsets, nseq, padlen, tok, batch_first, kind, d_out):
        check(lib().bsq_tokenize_host(self.h, stream, _ptr(h_bytes), _ptr(h_offsets), nseq, padlen, C.byref(tok),
                                      int(batch_first), kind, _ptr(d_out)))

    def onehot_host(self, stream, h_bytes, h_offsets, h_mask, nseq, padlen, tok, kind, d_out):
        check(lib().bsq_onehot_host(self.h, stream, _ptr(h_bytes), _ptr(h_offsets), _ptr(h_mask), nseq, padlen,
                                    C.byref(tok), kind, _ptr(d_out)), onehot=True)

    def sync_copies(self):
        check(lib().bsq_stager_sync_copies(self.h))

    def stage(self, stream, h_bytes, h_offsets, nseq):
        """-> (biased device residue pointer, device offsets pointer); see bsq_stage_host."""
        db, do = C.c_void_p(), C.c_void_p()
        check(lib().bsq_stage_host(self.h, stream, _ptr(h_bytes), _ptr(h_offsets), nseq, C.byref(db), C.byref(do)))
        return db.value or 0, do.value or 0

    def release(self, stream):
        check(lib().bsq_stage_release(self.h, stream))

    def set_augment(self, chain_len, augment_frac=1.0, seed=0, seq_index_base=0):
        check(lib().bsq_stager_set_augment(self.h, chain_len, float(augment_frac), seed & 0xFFFFFFFFFFFFFFFF, seq_index_base))

    def close(self):
        if self.h:
            lib().bsq_stager_destroy(self.h)
            self.h = C.c_void_p()


class Pack:
    """bsq_pack: gather ragged host sequences into (pinned) bytes + offsets."""

    def __init__(self, pinned=True):
        self.h = C.c_void_p()
        check(lib().bsq_pack_create(C.byref(self.h), int(pinned)))

    def gather(self, seqs, nthreads=1):
        n = len(seqs)
        bufs = [bytes(s) if not isinstance(s, bytes) else s for s in seqs]
        ptrs = (C.c_void_p * n)(*[C.cast(C.c_char_p(b), C.c_void_p) for b in bufs])
        lens = (C.c_int64 * n)(*[len(b) for b in bufs])
        check(lib().bsq_pack_gather(self.h, ptrs, lens, n, nthreads))
        return self

    @property
    def nseq(self): return lib().bsq_pack_nseq(self.h)
    @property
    def nbytes(self): return lib().bsq_pack_nbytes(self.h)
    @property
    def maxlen(self): return lib().bsq_pack_maxlen(self.h)
    @property
    def bytes_ptr(self): return lib().bsq_pack_bytes(self.h)
    @property
    def offsets_ptr(self): return lib().bsq_pack_offsets(self.h)

    def to_numpy(self):
        import numpy as np
        b = np.ctypeslib.as_array(C.cast(self.bytes_ptr, C.POINTER(C.c_uint8)), shape=(max(self.nbytes, 1),))[:self.nbytes]
        o = np.ctypeslib.as_array(C.cast(self.offsets_ptr, C.POINTER(C.c_int64)), shape=(self.nseq + 1,))
        return b.copy(), o.copy()

    def close(self):
        if self.h:
            lib().bsq_pack_destroy(self.h)
            self.h = C.c_void_p()


class FlatFile:
    """bsq_flatfile through the C ABI: what a non-Python host binds (the Python class lives in cbioseq)."""

    def __init__(self, path, maxseqlen=-1, pinned=False, prefault=False):
        self.h = C.c_void_p()
        # BSQ_FF_PINNED / BSQ_FF_MMAP_REGISTERED (prefault=2: populated and page-locked in place) / BSQ_FF_MMAP_PREFAULT / BSQ_FF_MMAP
        mode = 1 if pinned else (3 if int(prefault) >= 2 else (2 if prefault else 0))
        check(lib().bsq_flatfile_open(C.byref(self.h), os.fsencode(path), maxseqlen, mode))

    @staticmethod
    def make(inpath, outpath=""):
        n, m = C.c_int64(), C.c_int64()
        check(lib().bsq_flatfile_make(os.fsencode(inpath), os.fsencode(outpath), C.byref(n), C.byref(m)))
        return n.value, m.value

    @property
    def nseqs(self): return lib().bsq_flatfile_nseqs(self.h)
    @property
    def maxseqlen(self): return lib().bsq_flatfile_max_seq_len(self.h)
    @property
    def bytes_ptr(self): return lib().bsq_flatfile_bytes(self.h)

    @property
    def pinned(self): return bool(lib().bsq_flatfile_is_pinned(self.h))
    @property
    def offsets_ptr(self): return lib().bsq_flatfile_offsets(self.h)

    def close(self):
        if self.h:
            lib().bsq_flatfile_close(self.h)
            self.h = C.c_void_p()
