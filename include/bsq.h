/*
 * bsq.h -- C ABI of the B200-native batch tokeniser (libbsq.so).
 *
 * This is the drop-in boundary for the hot path of dnbaker/bioseq: everything the
 * reference's pybind11 class `cbioseq.Tokenizer` (src/tokenize.cpp:21-113) computes for
 *     batch_tokenize       (src/tokenize.cpp:82-98  -> Tokenizer::transencode<T>, src/tokenize.h:381-485)
 *     batch_onehot_encode  (src/tokenize.cpp:65-81  -> Tokenizer::tokenize<T>,    src/tokenize.h:283-371)
 *     decode_tokens        (src/tokenize.cpp:49-51  -> Tokenizer::decode_tokens,  src/tokenize.h:131-179)
 * is reachable through the plain-C entry points below.  The reference has no FFI of its
 * own (the Python class *is* its interface); these are the functions a maintainer's
 * pybind11 shim binds instead of the CPU loops (see INTEGRATION.md), and they are what
 * bioseq_b200's own `cbioseq` module, the GPU parity tests and bench.py call.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch/Python types cross the boundary;
 *   - every function returns 0 (BSQ_OK) or a negative BSQ_ERR_* code and never throws;
 *     bsq_last_error() returns the message of the calling thread's last failure -- where
 *     the reference raises, the text is the reference's text (file:line cited per code);
 *   - "d_" pointers are device memory on `device`, "h_" pointers are host memory;
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream);
 *     device entry points only enqueue work, they do not synchronise unless stated;
 *   - sequences travel packed: one byte buffer + int64 offsets, offsets[i]..offsets[i+1]
 *     delimiting sequence i (nseq+1 entries).  This is what the pack layer produces from
 *     the Python str/bytes/bytearray items the reference unpacks at src/tokenize.h:389-419;
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails
 *     with BSQ_ERR_CUDA.
 */
#ifndef BSQ_H_
#define BSQ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSQ_ABI_VERSION 5

/* ---- status codes ---------------------------------------------------------------- */
#define BSQ_OK 0
#define BSQ_ERR_ARG (-1)       /* std::invalid_argument in the reference -> ValueError          */
#define BSQ_ERR_TOO_LONG (-2)  /* "seq len + bos + eos > padlen: N, vs padlen P" (tokenize.h:458 runtime_error, :361 invalid_argument) */
#define BSQ_ERR_BAD_TOKEN (-3) /* "Unexpected/invalid token N" (tokenize.h:148,170) -> RuntimeError */
#define BSQ_ERR_KEY (-4)       /* "Invalid tokenizer type; select one from..." (tokenize.h:78) -> RuntimeError */
#define BSQ_ERR_CUDA (-5)      /* CUDA runtime failure / no device -> RuntimeError              */
#define BSQ_ERR_NOMEM (-6)
#define BSQ_ERR_IO (-7)        /* file could not be opened / read / written -> RuntimeError     */
#define BSQ_ERR_RANGE (-8)     /* std::out_of_range in the reference -> IndexError              */

/* ---- element kinds of the output array (src/tokenize.cpp:66-79, :83-96) ------------ */
typedef enum bsq_kind {
    BSQ_I8 = 0,  /* destchar b/B : 1-byte integer (reference: int8)            */
    BSQ_I16 = 1, /* destchar h/H */
    BSQ_I32 = 2, /* destchar i/I */
    BSQ_I64 = 3, /* destchar l/L/q/Q : 8-byte integer (reference: uint64)      */
    BSQ_F32 = 4, /* destchar f/F */
    BSQ_F64 = 5  /* destchar d/D */
} bsq_kind;

/* tolower(destchar) dispatch of src/tokenize.cpp:66,83.  Returns a bsq_kind, or
 * BSQ_ERR_ARG ("Unsupported dtype: X", tokenize.cpp:80,97). */
int bsq_kind_of_destchar(char destchar);
/* bytes per element of a kind (1,2,4,8,4,8); 0 for an invalid kind. */
size_t bsq_kind_size(int kind);

/* ---- tokenizer descriptor ---------------------------------------------------------- */
/* Plain data; filled by bsq_tokenizer_init and passed by pointer to the compute calls.
 * Mirrors struct Tokenizer's state (src/tokenize.h:10-38). */
typedef struct bsq_tokenizer {
    int8_t lut[256];        /* alphabet.h:32-61 make_lut: byte -> id, -1 = invalid            */
    int32_t nchars;         /* alphabet.h:27   number of groups                                */
    int32_t bos_id;         /* tokenize.h:23-26  nchars, or -1 when BOS is not included        */
    int32_t eos_id;         /* tokenize.h:27-30  nchars + bos, or -1                           */
    int32_t pad_id;         /* tokenize.h:31-33  nchars + bos + eos (defined even if !padchar) */
    int32_t padchar;        /* tokenize.h:13   zero_onehot_pad_: pad id is a real symbol       */
    int32_t alphabet_size;  /* tokenize.h:22   nchars + eos + bos + padchar                    */
    char key[16];           /* upper-cased key (tokenize.h:73)                                 */
} bsq_tokenizer;

/* Registry of alphabet keys (CAMAP, src/alphabet.h:198-222), in map order. */
int bsq_alphabet_count(void);
const char *bsq_alphabet_key(int index);

/* Tokenizer(key, eos, bos, padchar) -- src/tokenize.h:72-106.  Key lookup is
 * case-insensitive.  BSQ_ERR_KEY on an unknown key. */
int bsq_tokenizer_init(bsq_tokenizer *tok, const char *key, int eos, int bos, int padchar);

/* id -> decoded text, the reference's `lookup` map (src/tokenize.h:83-99): for ids
 * -128..127 the first byte value whose LUT entry is that id; "<BOS>", "<EOS>", "<PAD>"
 * for the specials.  Writes up to cap-1 chars + NUL to buf and returns the length
 * (1 or 5), or 0 when the id has no entry. */
int bsq_tokenizer_lookup(const bsq_tokenizer *tok, int32_t id, char *buf, size_t cap);

/* ---- pack layer (host) -------------------------------------------------------------- */
/* Gathers ragged host sequences into one pinned byte buffer + int64 offsets: the form
 * the kernels read and the form cudaMemcpyAsync can stage without a bounce.  Replaces
 * the reference's vector<pair<const char*, size_t>> of borrowed pointers
 * (src/tokenize.h:386-419). */
typedef struct bsq_pack bsq_pack;

/* pinned != 0: cudaHostAlloc'ed storage (needs a CUDA device); 0: pageable (malloc). */
int bsq_pack_create(bsq_pack **out, int pinned);
void bsq_pack_destroy(bsq_pack *p);
/* Replace the contents with n sequences given as pointer/length arrays; the copy is
 * split over up to nthreads host threads.  Also records the longest length. */
int bsq_pack_gather(bsq_pack *p, const void *const *ptrs, const int64_t *lens, int64_t n, int nthreads);
const uint8_t *bsq_pack_bytes(const bsq_pack *p);
const int64_t *bsq_pack_offsets(const bsq_pack *p); /* n+1 entries */
int64_t bsq_pack_nseq(const bsq_pack *p);
int64_t bsq_pack_nbytes(const bsq_pack *p);
int64_t bsq_pack_maxlen(const bsq_pack *p);

/* Host-side length check done before any launch: the reference aborts the process when
 * len + bos + eos > padlen (exception inside an OpenMP region, src/tokenize.h:456-459);
 * here the call fails with BSQ_ERR_TOO_LONG and the reference's message.
 * padlen <= 0 -> BSQ_ERR_ARG "batch tokenize requires padlen is provded." (tokenize.h:383). */
int bsq_check_lengths_host(const int64_t *h_offsets, int64_t nseq, int64_t padlen, const bsq_tokenizer *tok);
/* Same check for device-resident offsets: one reduction kernel + an 8-byte read-back
 * (synchronises `stream`). */
int bsq_check_lengths_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq,
                             int64_t padlen, const bsq_tokenizer *tok);
/* The same reduction, also validating the offsets themselves before a kernel indexes `d_bytes` with them: every
 * length >= 0, offsets[0] >= 0 and offsets[nseq] <= nbytes (the byte buffer's size; < 0 = unknown, not checked)
 * -> BSQ_ERR_ARG otherwise.  What cbioseq's batch_tokenize_packed / batch_onehot_encode_packed call for
 * device-resident inputs. */
int bsq_check_offsets_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t nbytes,
                             int64_t padlen, const bsq_tokenizer *tok);

/* ---- device compute ------------------------------------------------------------------ */
/* batch_tokenize: tokens with BOS/EOS/PAD fused in one pass.
 *   d_out: (nseq, padlen) if batch_first else (padlen, nseq), C-contiguous, `kind`
 *   elements, 16-byte aligned; every element is written exactly once (no memset).
 *   Row i = [bos?] lut[residues] (invalid -> 0) [eos?] then pad_id if padchar else 0
 *   (src/tokenize.h:460-478).  Lengths must already have been checked. */
int bsq_tokenize(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets,
                 int64_t nseq, int64_t padlen, const bsq_tokenizer *tok, int batch_first,
                 int kind, void *d_out);

/* Padding-free tokens: one packed token stream plus int32 cu_seqlens -- the input of varlen attention
 * (FlashAttention's *_varlen_func), nested / jagged tensors and sequence-packing loaders.  With k = bos + eos:
 *   d_cu_seqlens[i] = (d_offsets[i] - d_offsets[0]) + i * k for i = 0 .. nseq  (nseq + 1 int32 entries), T = d_cu_seqlens[nseq];
 *   d_out[cu[i] .. cu[i+1]) = row i of bsq_tokenize (batch-first, any padlen >= its length) without its padding:
 *   [bos?] lut[residues] (invalid -> 0) [eos?].  No pad id is emitted, whatever tok->padchar says.
 * d_out holds exactly T `kind` elements and is 16-byte aligned (it may be NULL when T == 0); every element is written
 * once.  The caller sizes d_out from T, which it knows from host offsets or from bsq_varlen_extent_device, and has
 * checked that T <= 2^31 - 1 and that the offsets are valid.  Enqueues only (one kernel; nseq == 0: a 4-byte memset).
 * Capturable into a CUDA graph: the kernel keeps a static tile order and no state between launches. */
int bsq_tokenize_varlen(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq,
                        const bsq_tokenizer *tok, int kind, void *d_out, int32_t *d_cu_seqlens);
/* The extent of that output for device-resident offsets: *total = T and *max_seqlen = longest sequence + k (0 for
 * nseq == 0), from one reduction kernel and one read-back (synchronises `stream`).  Validates the offsets like
 * bsq_check_offsets_device (BSQ_ERR_ARG: negative length, offsets[0] < 0, offsets[nseq] > nbytes when nbytes >= 0). */
int bsq_varlen_extent_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t nbytes,
                             const bsq_tokenizer *tok, int64_t *total, int64_t *max_seqlen);

/* Masked-language-model batches (BERT / ESM pretraining): the tokens of bsq_tokenize (batch-first) or
 * bsq_tokenize_varlen with BERT-style corruption, plus int64 labels, written by one kernel.  Call the unmasked
 * tokens `tok`.  Only residue positions are eligible -- residue j (0 <= j < len_i) of row i, at column bos + j; BOS, EOS
 * and PAD are never selected -- and eligibility depends on the position only (an invalid byte is a residue whose token
 * and label are 0).  With g = seq_index_base + i and u = word (j & 3) of Philox4x32-10 with counter
 * (g_lo, g_hi, j >> 2, 1) and key (seed_lo, seed_hi):
 *   u >= t_select              input = tok        label = ignore_index
 *   u <  t_mask                input = mask_id    label = tok
 *   t_mask <= u < t_random     input = (w * nchars) >> 32, w = word (j & 3) of the block with counter (g_lo, g_hi,
 *                              j >> 2, 2)         label = tok
 *   otherwise                  input = tok        label = tok
 * Non-residue positions: input = tok, label = ignore_index.  The counters' word 3 (1 and 2) keeps these draws disjoint
 * from bsq_augment_blosum62's (word 3 = 0) under the same seed, and the mask depends only on (seed, global sequence
 * index, residue position): not on padlen, the padded or padding-free form, or how the data is sliced.
 * The thresholds are integers in [0, 2^32] with t_mask <= t_random <= t_select; a caller with fractions computes
 *   t_select = maskfrac >= 1 ? 2^32 : floor(maskfrac * 2^32),  t_mask = floor(t_select * mask_prob),
 *   t_random = min(t_select, floor(t_select * (mask_prob + random_prob)))     (in double precision)
 * so that the rule never depends on floating-point arithmetic on the device.  mask_id must be >= 0 and representable in
 * `kind`: <= 255 for BSQ_I8 (the byte is written as is), <= 32767 for BSQ_I16, <= 2^24 for BSQ_F32, <= 2^31 - 1
 * otherwise.  BSQ_ERR_ARG otherwise, or for thresholds out of order. */
typedef struct bsq_mlm {
    uint64_t seed;
    int64_t seq_index_base;
    uint64_t t_select, t_mask, t_random;
    int64_t mask_id, ignore_index;
} bsq_mlm;
/* Padded: d_inputs is (nseq, padlen) `kind` elements and d_labels (nseq, padlen) int64, batch-first, both 16-byte
 * aligned; every element is written once.  Lengths must already have been checked, as for bsq_tokenize. */
int bsq_tokenize_mlm(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int64_t padlen,
                     const bsq_tokenizer *tok, int kind, const bsq_mlm *mlm, void *d_inputs, int64_t *d_labels);
/* Padding-free: d_inputs and d_labels hold exactly T elements each (T and the caller's checks as for
 * bsq_tokenize_varlen), aligned element for element; d_cu_seqlens as there.  Both entry points only enqueue work (one
 * kernel; nseq == 0: nothing, or a 4-byte memset of cu_seqlens), keep no state between launches and are capturable
 * into a CUDA graph. */
int bsq_tokenize_varlen_mlm(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq,
                            const bsq_tokenizer *tok, int kind, const bsq_mlm *mlm, void *d_inputs, int64_t *d_labels,
                            int32_t *d_cu_seqlens);

/* Cropping over-long sequences (protein / DNA language-model training crops each sequence to the model's context):
 * a packed batch in, a packed batch of windows out, which every entry point above then takes unchanged.
 * Let W = crop_len >= 1, len_i = offsets[i+1] - offsets[i] and len'_i = min(len_i, W).
 *   - start_i = 0 if len_i <= W or the mode is head (random == 0).
 *   - Random mode: with span = len_i - W + 1, g = seq_index_base + i, and (x0, x1, x2, x3) = Philox4x32-10 at counter
 *     (g_lo, g_hi, 0, 3) under key (seed_lo, seed_hi):
 *       start_i = floor(d * span / 2^64) with d = x0 | x1 << 32 (__umul64hi; exact integers, nothing in floating point).
 *   - Output: out_offsets[0] = 0, out_offsets[i+1] = out_offsets[i] + len'_i, and
 *     out_bytes[out_offsets[i] + j] = bytes[offsets[i] + start_i + j] for j < len'_i.  Optionally, starts[i] = start_i
 *     (int64).
 *   - Counter word 3 = 3 keeps these draws disjoint from augmentation (0) and MLM (1, 2) under the same seed.  The window
 *     depends only on (seed, global sequence index, length, W).  It does not depend on padlen, on the padded or
 *     padding-free form, or on how the data is sliced.
 *   - A sequence no longer than W is copied unchanged, and no draw is used for it.
 * Order inside a consumer: stage -> crop -> augment -> tokenize / mask.  For augmentation and MLM, "residue position"
 * then means position within the window, and the sequence index is unchanged.
 *
 * bsq_crop enqueues only (at most three kernels; nseq == 0: an 8-byte memset of out_offsets), keeps no state between
 * launches and is capturable into a CUDA graph.  The caller has validated the offsets (bsq_crop_extent_device does) and
 * sized d_out_bytes to at least sum(len'_i) bytes (any alignment); d_out_offsets has nseq + 1 entries; d_starts (nseq
 * entries) may be NULL.  BSQ_ERR_ARG for crop_len < 1, nseq < 0, or NULL pointers with nseq > 0, before any device call.
 * The output must not overlap the input. */
int bsq_crop(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int64_t crop_len,
             int random, uint64_t seed, int64_t seq_index_base, uint8_t *d_out_bytes, int64_t *d_out_offsets, int64_t *d_starts);
/* The extent of that output for device-resident offsets: *total = sum(len'_i) and *max_len = max(len'_i) (0 for
 * nseq == 0), from one reduction kernel and one read-back (synchronises `stream`).  Validates the offsets like
 * bsq_check_offsets_device, with no padlen limit (BSQ_ERR_ARG: negative length, offsets[0] < 0, offsets[nseq] > nbytes
 * when nbytes >= 0); BSQ_ERR_ARG for crop_len < 1. */
int bsq_crop_extent_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t nbytes, int64_t crop_len,
                           int64_t *total, int64_t *max_len);

/* Reverse complement (strand augmentation for DNA / RNA models in training, both-strand averaging at inference): a
 * packed batch in, a packed batch out, which every entry point above then takes unchanged.
 *   Complement table comp[256], defined on every byte value and case-preserving: A<->T, C<->G, R<->Y, K<->M, B<->V, D<->H;
 *   S, W and N map to themselves; U -> A (RNA gives its DNA reverse complement); the same pairs in lower case.  Every
 *   other byte maps to itself (gaps, '*', digits, bytes >= 0x80), so a byte a tokenizer rejects is still rejected after
 *   the flip.  bsq_revcomp_table copies it out.
 *   Flip of a sequence of len bytes: out[j] = comp[in[len - 1 - j]].
 *   Modes:
 *     BSQ_RC_ALWAYS  every sequence is flipped;
 *     BSQ_RC_RANDOM  sequence i is flipped iff x0 < gate, with x0 = word 0 of Philox4x32-10 at counter (g_lo, g_hi, 0, 4)
 *                    under key (seed_lo, seed_hi), g = seq_index_base + i, and gate = rc_prob >= 1 ? 2^32 :
 *                    floor(rc_prob * 2^32) (in double precision, on the host).  Counter word 3 = 4 keeps the draw
 *                    disjoint from augmentation (0), MLM (1, 2) and crop (3) under the same seed: the flip depends only on
 *                    (seed, global sequence index), not on the length, padlen, the padded or padding-free form or slicing;
 *     BSQ_RC_BOTH    2n output sequences: sequence i is input sequence i unchanged, sequence n + i its reverse complement
 *                    (the torch.cat([x, x_rc]) layout that both-strand inference averages over).
 *   Output: out_offsets start at 0; out_offsets[i] = offsets[i] - offsets[0] for i = 0 .. n, and in BOTH mode, with
 *   T = offsets[n] - offsets[0], out_offsets[n + i] = T + offsets[i] - offsets[0].  d_flipped (optional, may be NULL): one
 *   byte (0 / 1) per output sequence.
 *   Order inside a consumer: stage -> crop -> reverse complement -> tokenize / mask / pack / k-mer.  MLM positions are
 *   positions in the flipped window; the sequence index is unchanged.
 * Worked answers: "ACGTN" -> "NACGT", "GATTACA" -> "TGTAATC", "ACGU" -> "ACGT", "acgRYkmBDHVswn-*" -> "*-nwsBDHVkmRYcgt",
 * "" -> "".  RANDOM, rc_prob 0.5, sequences 0 .. 7: seed 7, seq_index_base 0 flips [1,0,1,1,1,1,1,1] (x0 = 407685168,
 * 3339964855, 305774060, ...); seed 0x123456789ABCDEF0, seq_index_base 2^32 + 11 flips [1,0,0,0,1,0,1,1].
 *
 * bsq_revcomp enqueues only (one kernel; nseq == 0: an 8-byte memset of out_offsets), uses no scratch memory, keeps no
 * state between launches and is capturable into a CUDA graph.  The caller has validated the offsets (as for bsq_crop).
 * d_out_bytes (any alignment, not overlapping the input) holds at least T bytes, 2T in BOTH mode -- a caller with a
 * device batch can size it from the byte buffer's size, with no read-back; BOTH writes its forward half too.
 * d_out_offsets has n + 1 entries (2n + 1 in BOTH mode).  BSQ_ERR_ARG, before any device call, for a bad mode, rc_prob
 * NaN or < 0 (read in RANDOM mode only, checked in every mode), nseq < 0, a NULL d_out_offsets, or NULL bytes, offsets or
 * output bytes with nseq > 0. */
#define BSQ_RC_ALWAYS 0
#define BSQ_RC_RANDOM 1
#define BSQ_RC_BOTH 2
int bsq_revcomp(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int mode, double rc_prob,
                uint64_t seed, int64_t seq_index_base, uint8_t *d_out_bytes, int64_t *d_out_offsets, uint8_t *d_flipped);
/* Host only, no device call: out[b] = comp[b] for every byte value b.  BSQ_ERR_ARG for a NULL out. */
int bsq_revcomp_table(uint8_t out[256]);

/* Sliding-window tiling (inference over whole long sequences, dataset construction by chunking -- HF's
 * return_overflowing_tokens=True with stride=): a packed batch in, a packed batch of all its windows out, which every
 * entry point above then takes unchanged, with the maps that connect the two.  Nothing is drawn at random: the windows
 * depend only on (len_i, W, S, tail).
 * Let W = window >= 1, S = stride with 1 <= S <= W, len_i = offsets[i+1] - offsets[i] and tail one of BSQ_TILE_*:
 *   - len_i <= W (0 included): one window, the whole sequence (start 0, length len_i), under every tail.  An empty
 *     sequence gives one empty window, so every sequence has at least one window.
 *   - len_i > W:
 *       SHORT  m_i = ceil((len_i - W) / S) + 1 windows; window j starts at j*S and has length min(W, len_i - j*S) (only
 *              the last can be shorter than W);
 *       END    the same m_i; windows j < m_i - 1 start at j*S, the last at len_i - W; every window is W long (the last
 *              overlaps its predecessor by more than W - S; identical to SHORT when S divides len_i - W);
 *       DROP   m_i = floor((len_i - W) / S) + 1 windows at j*S, all W long; the last len_i - ((m_i - 1)*S + W) residues
 *              are in no window.
 *   - Output order: the windows of sequence 0 by start, then those of sequence 1, ...; M = sum m_i.
 *     seq_ptr[i] (int64, n + 1 entries, seq_ptr[0] = 0): index of sequence i's first window;
 *     seq_index[w] (int64, M): the sequence of window w (HF's overflow_to_sample_mapping);
 *     starts[w] (int64, M): where window w begins in its sequence;
 *     out_offsets (int64, M + 1, from 0) and out_bytes[out_offsets[w] + t] = bytes[offsets[seq_index[w]] + starts[w] + t].
 * Worked answers, W = 4, S = 3: "ACGTACGTACG" (11) -> SHORT starts 0, 3, 6, 9: ACGT, TACG, GTAC, CG; END 0, 3, 6, 7: ACGT,
 * TACG, GTAC, TACG; DROP 0, 3, 6: ACGT, TACG, GTAC.  Length 5: SHORT (0, 4), (3, 2); END (0, 4), (1, 4); DROP (0, 4).
 * Lengths 4 and 0: one window each, under every tail.
 *
 * bsq_tile_extent_host (no device call): *nwin = M, *nbytes = sum of the window lengths, *max_len = the longest window
 * (all 0 for nseq == 0).  BSQ_ERR_ARG for W < 1, S < 1, S > W, a bad tail, NULL outputs, negative lengths, offsets[0] < 0,
 * and a window count or byte total past INT64_MAX (the arithmetic does not overflow for any int64 lengths). */
#define BSQ_TILE_SHORT 0
#define BSQ_TILE_END 1
#define BSQ_TILE_DROP 2
int bsq_tile_extent_host(const int64_t *h_offsets, int64_t nseq, int64_t window, int64_t stride, int tail, int64_t *nwin,
                         int64_t *nbytes, int64_t *max_len);
/* The same for device-resident offsets, from one reduction kernel and one read-back (synchronises `stream`); it validates
 * the offsets like bsq_crop_extent_device (BSQ_ERR_ARG: negative length, offsets[0] < 0, offsets[nseq] > nbytes when
 * nbytes >= 0). */
int bsq_tile_extent_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t nbytes, int64_t window,
                           int64_t stride, int tail, int64_t *nwin, int64_t *out_nbytes, int64_t *max_len);
/* bsq_tile enqueues only (nseq == 0: out_offsets[0] = 0 and seq_ptr[0] = 0 by 8-byte memsets), keeps no state between
 * launches and is capturable into a CUDA graph.  Scratch: 8 (n + 1) bytes, 16 (n + 1) when d_seq_ptr is NULL, allocated
 * and freed in stream order (cudaMallocAsync / cudaFreeAsync from the device's default memory pool).  The caller has
 * validated the offsets (bsq_tile_extent_device does) and sized d_out_bytes (any alignment, not overlapping the input) to
 * the extent's nbytes and d_out_offsets to nwin + 1 entries; d_seq_ptr (n + 1), d_seq_index and d_starts (nwin each) may
 * be NULL.  BSQ_ERR_ARG, before any device call, for a bad W, S or tail, nseq < 0, a NULL d_out_offsets, or NULL bytes,
 * offsets or output bytes with nseq > 0. */
int bsq_tile(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int64_t window, int64_t stride,
             int tail, uint8_t *d_out_bytes, int64_t *d_out_offsets, int64_t *d_seq_ptr, int64_t *d_seq_index, int64_t *d_starts);

/* Stitching per-residue model outputs of the windows back onto the sequences: the mean over every covering window.
 *   d_y: the outputs, C channels per position of element type dtype (BSQ_UNTILE_*), channels contiguous.  Window w's
 *   residue t is row base_w + col0 + t of the 2-D (rows, C) view: base_w = w * row_stride for padded batch-first outputs
 *   (M', P, C) (d_cu NULL, row_stride = P > col0), base_w = d_cu[w] for padding-free outputs (T, C) (d_cu: int32 window starts,
 *   a padding-free token batch's cu_seqlens); col0 is the number of leading special tokens (BOS).
 *   strands 1 or 2: with 2 (the layout BSQ_RC_BOTH makes), windows M .. 2M - 1 are windows 0 .. M - 1 again.
 *   d_flipped (strands * M bytes, or NULL): windows that were reverse-complemented; in a flipped window of length l,
 *   residue t is source position starts + l - 1 - t.
 *   Output d_out: float32 (offsets[n] - offsets[0], C), row offsets[i] - offsets[0] + p for residue p of sequence i: the
 *   sum over every covering window (of every strand) in float32 -- strand 0 before strand 1, windows in ascending order
 *   within a strand -- divided by their count; a residue no window covers (DROP) gets a quiet NaN.  Channels are averaged
 *   as they are (swapping strand-specific channels of a flipped window is the caller's business).
 * Worked answer: "ACGTACGTACG", W = 4, S = 3, C = 1, every window reporting its index w at every position: SHORT gives
 * [0, 0, 0, 0.5, 1, 1, 1.5, 2, 2, 2.5, 3], END [0, 0, 0, 0.5, 1, 1, 1.5, 2.5, 2.5, 2.5, 3], DROP [0, 0, 0, 0.5, 1, 1, 1.5,
 * 2, 2, 2, NaN].
 * Enqueues one kernel, keeps no state between launches and is capturable into a CUDA graph.  d_seq_ptr is bsq_tile's
 * (n + 1 entries), nwin = M.  BSQ_ERR_ARG, before any device call, for a bad W, S, tail or dtype, C < 1, col0 < 0,
 * strands not 1 or 2, nseq < 0, nwin < nseq, row_stride <= col0 without d_cu, or NULL pointers with nseq > 0. */
#define BSQ_UNTILE_F32 0
#define BSQ_UNTILE_BF16 1
#define BSQ_UNTILE_F16 2
int bsq_untile_mean(int device, void *stream, int dtype, const void *d_y, int64_t channels, int64_t row_stride, const int32_t *d_cu,
                    int64_t col0, const int64_t *d_src_offsets, int64_t nseq, int64_t window, int64_t stride, int tail,
                    const int64_t *d_seq_ptr, int64_t nwin, int strands, const uint8_t *d_flipped, float *d_out);

/* Translation (protein language models on coding sequences, six-frame searches over reads, gene calls into a protein
 * model): a packed DNA / RNA batch in, a packed protein batch of its reading frames out, which every entry point above
 * then takes unchanged.
 *   Residues -> base sets, case-insensitive IUPAC: A, C, G, T (U = T) stand for themselves; R = AG, Y = CT, S = CG,
 *   W = AT, K = GT, M = AC, B = CGT, D = AGT, H = ACT, V = ACG, N = ACGT.  Every other byte is invalid (gaps, '*', digits,
 *   bytes >= 0x80).  As a 4-bit mask: A = 1, C = 2, G = 4, T = 8, invalid = 0; the complement (A <-> T, C <-> G, K12's
 *   pairs applied to base sets) is then the reversal of the 4 bits.
 *   Codon -> amino acid: every expansion of the three base sets is looked up in the genetic code; if all give the same
 *   letter that letter is the result, otherwise -- or if a byte is invalid -- 'X'.  Stops are the code's '*'.  (Biopython's
 *   B / Z / J ambiguity letters are not produced.)
 *   Genetic code: 64 characters in TCAG order, codon index 16 b1 + 4 b2 + b3 with T = 0, C = 1, A = 2, G = 3.  Any 64
 *   printable ASCII characters (0x21..0x7E) are accepted, so a custom table's letters come out as written; the built-in
 *   NCBI tables (bsq_genetic_code) are upper case.  Every codon translates to its table letter, the first included
 *   (alternative start codons are not applied).
 *   Frames: frame +k (k = 1, 2, 3) reads the sequence from offset k - 1, frame -k its reverse complement from offset
 *   k - 1 (so frame -1 starts at the last base).  Each has max(0, floor((len - (k - 1)) / 3)) amino acids; a trailing
 *   partial codon is dropped.  Amino acid t of frame +k comes from nucleotides k - 1 + 3t .. k + 1 + 3t, of frame -k from
 *   len - k - 3t - 2 .. len - k - 3t, read right to left on the complement.
 *   Output: the caller gives F frames, 1 to 6 distinct values in any order; output sequence w = i F + f is frame frames[f]
 *   of input sequence i (sequence-major, n F sequences).  out_offsets (int64, n F + 1 entries) start at 0.  Sequences
 *   shorter than 3 give empty rows, which are kept.
 *   Order inside a consumer: stage -> translate -> crop -> augment -> tokenize / mask / pack / k-mer.  Crop lengths,
 *   padlen and MLM positions count amino acids; a seeded draw for output sequence (i, f) is keyed by the global output
 *   index (seq_index_base + i) F + f, so slicing a batch changes no draw.
 * Worked answers, standard code, frames +1, +2, +3, -1, -2, -3:
 *   "ATGGCCATTGTAATGGGCCGCTGAAAGGGTGCCCGATAG" (39 nt) -> "MAIVMGR*KGAR*", "WPL*WAAERVPD", "GHCNGPLKGCPI", "LSGTLSAAHYNGH",
 *   "YRAPFQRPITMA", "IGHPFSGPLQWP";  "ATGA" -> "M", "*", "", "S", "H", "";  "ATGAA" -> "M", "*", "E", "F", "S", "H";
 *   "", "A" and "AT" -> six empty rows each.
 *   Frame +1 under codes 1 / 2, and frame -1 under code 1: GCN A / A, X; TAR * / *, L; TRA * / X, X; YTG L / L, Q;
 *   atg and AUG M / M, H; A-G X / X, X; TGA * / W, S; AGA R / *, S.  "ATAAGATGA" frame +1: "IR*" (code 1), "M*W" (code 2);
 *   "TAATAG" frame +1 under code 6: "QQ".
 *
 * bsq_genetic_code (host only): the built-in tables -- 1 standard and 11 bacterial (the same amino acids), 2 vertebrate
 * mitochondrial, 4 mold / protozoan mitochondrial and Mycoplasma, 5 invertebrate mitochondrial, 6 ciliate -- as 64
 * characters (no terminating NUL).  BSQ_ERR_ARG for any other id.
 * bsq_translate_table (host only): masks[b] = the base set of byte b, codons[m0 << 8 | m1 << 4 | m2] = the letter of
 * that triple of base sets (or 'X').  The only place the rule is built in the library; the kernels get these tables.
 * BSQ_ERR_ARG for a NULL or non-printable code or NULL outputs. */
int bsq_genetic_code(int id, char out[64]);
int bsq_translate_table(const char *code64, uint8_t masks[256], uint8_t codons[4096]);
/* The output's size before a crop (*total bytes) and after a crop of every output row to crop_len amino acids
 * (*crop_total, *max_len = the longest kept row); crop_len = INT64_MAX means no crop.  All 0 for nseq == 0.  The host
 * form makes no device call; BSQ_ERR_ARG for bad frames (as bsq_translate), crop_len < 1, NULL outputs, negative lengths,
 * offsets[0] < 0 or a total past INT64_MAX.  The device form runs one reduction and one read-back (synchronises `stream`)
 * and validates the offsets like bsq_crop_extent_device (BSQ_ERR_ARG: negative length, offsets[0] < 0, offsets[nseq] >
 * nbytes when nbytes >= 0). */
int bsq_translate_extent_host(const int64_t *h_offsets, int64_t nseq, const int8_t *frames, int nframes, int64_t crop_len,
                              int64_t *total, int64_t *crop_total, int64_t *max_len);
int bsq_translate_extent_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t nbytes, const int8_t *frames,
                                int nframes, int64_t crop_len, int64_t *total, int64_t *crop_total, int64_t *max_len);
/* bsq_translate enqueues only (two or three kernels; nseq == 0: an 8-byte memset of out_offsets), keeps no state between
 * launches and is capturable into a CUDA graph.  Scratch: 8 (n + 1) bytes, allocated and freed in stream order
 * (cudaMallocAsync / cudaFreeAsync from the device's default memory pool).  `frames` (nframes entries) and `code64` are
 * host memory, read before the call returns.  The caller has validated the offsets (bsq_translate_extent_device does) and
 * sized d_out_bytes (any alignment, not overlapping the input) to the extent's total and d_out_offsets to n F + 1 entries.
 * BSQ_ERR_ARG, before any device call, for bad, duplicate, zero or more than six frames, a NULL or non-printable code,
 * nseq < 0 (or n F + 1 past INT64_MAX), a NULL d_out_offsets, or NULL bytes, offsets or output bytes with nseq > 0. */
int bsq_translate(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, const int8_t *frames,
                  int nframes, const char *code64, uint8_t *d_out_bytes, int64_t *d_out_offsets);

/* Sequence packing (padding-free batches of a fixed shape: SDPA with a block-diagonal mask, position-id packing as in
 * HF's DataCollatorWithFlattening, CUDA graphs, torch.compile): whole sequences laid end to end in R rows of L tokens.
 * With k = bos + eos and the (already cropped) lengths len_i, sequence i occupies need_i = len_i + k tokens; every
 * need_i must be <= L (BSQ_ERR_ARG "seq len + bos + eos > padlen: N, vs padlen L" otherwise).
 *   Placement is best-fit decreasing, fully deterministic:
 *     1. sequences with need_i > 0 are placed in order of decreasing need_i, ties to the lower index (a stable sort);
 *     2. each goes into the open row with the least remaining space that still fits it, ties to the lowest row index;
 *     3. if no open row fits, a new row is opened with the next row index;
 *     4. within a row, sequences lie in placement order from column 0 without gaps: a sequence's column is the row's
 *        fill when it is placed;
 *     5. sequences with need_i == 0 (empty, k = 0) occupy nothing: starts[i] = -1.
 *   Layout: R rows are used; with rows = R0 > 0 exactly R0 (the extra rows are padding), BSQ_ERR_ARG if the layout needs
 *   more.  R * L must be <= 2^31 - 1 (cu_seqlens is int32), BSQ_ERR_ARG otherwise.
 *   Output: a placed sequence starts at flat position s = starts[i] = row * L + column of the (R, L) tokens;
 *   tokens[s .. s + need_i) = row i of bsq_tokenize_varlen on the same batch ([BOS] lut(residues) [EOS]) and
 *   position_ids over that span are 0 .. need_i - 1.  A segment is a placed sequence or the non-empty padding run at the
 *   end of a row; a padding run holds what bsq_tokenize writes after EOS (pad_id with padchar, else 0) and its position
 *   ids restart at 0 too.  cu_seqlens (int32) lists the flat start of every segment in order, then R * L; max_seqlen is
 *   the longest segment.  So varlen attention runs on the flattened tokens as they are, and a block mask is
 *   (position_ids == 0).cumsum(-1) compared within a row.
 *   MLM: inputs and int64 labels of a placed sequence equal bsq_tokenize_varlen_mlm's under the same bsq_mlm -- the draw
 *   is keyed by the global sequence index, not by the placement; padding labels are ignore_index.
 *   Crop and augmentation: stage -> crop -> augment -> pack, as for the other consumers.
 *
 * bsq_seqpack_plan (host only, no device call) computes that layout from host offsets (the cropped ones when a crop
 * applies): O(n log L).  *nrows = R, *nsegments = the number of segments, *max_seqlen.  A first call with starts,
 * row_ptr, row_seq and cu_seqlens all NULL only sizes; otherwise all four are written: starts[nseq] (int64), row_ptr[R + 1]
 * and row_seq[row_ptr[R]] (at most nseq entries: the sequences of each row in column order, the CSR the kernel walks),
 * cu_seqlens[nsegments + 1].  rows <= 0: as many rows as the layout needs.  BSQ_ERR_ARG for nseq < 0, k outside 0..2,
 * row_len < 1, NULL offsets with nseq > 0, NULL size outputs, only some of the four arrays, negative lengths, and the
 * cases above. */
int bsq_seqpack_plan(const int64_t *h_offsets, int64_t nseq, int k, int64_t row_len, int64_t rows, int64_t *nrows,
                     int64_t *nsegments, int64_t *max_seqlen, int64_t *starts, int64_t *row_ptr, int64_t *row_seq,
                     int32_t *cu_seqlens);
/* The packed rows of a plan: d_tokens (nrows, row_len) `kind` elements and d_position_ids (nrows, row_len) int32, both
 * 16-byte aligned (any row_len); every element is written once (no memset).  d_row_ptr / d_row_seq: the plan's CSR on
 * the device, for the batch given by d_bytes / d_offsets (the offsets the plan was made from, up to a constant shift;
 * d_bytes, d_offsets and d_row_seq are only read for placed sequences, so a plan of padding rows alone may pass NULL).
 * One kernel (nrows == 0: nothing); enqueues only, keeps no state between launches, capturable into a CUDA graph.
 * BSQ_ERR_ARG for a NULL d_row_ptr, NULL or misaligned outputs, row_len < 1, nrows < 0 or nrows * row_len > 2^31 - 1. */
int bsq_tokenize_seqpack(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, const bsq_tokenizer *tok,
                         int kind, int64_t row_len, int64_t nrows, const int64_t *d_row_ptr, const int64_t *d_row_seq,
                         void *d_tokens, int32_t *d_position_ids);
/* The same rows with the masked-language-model rule of bsq_tokenize_mlm: d_inputs as d_tokens, plus d_labels
 * (nrows, row_len) int64, 16-byte aligned.  BSQ_ERR_ARG also for a bsq_mlm bsq_tokenize_mlm rejects. */
int bsq_tokenize_seqpack_mlm(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, const bsq_tokenizer *tok,
                             int kind, const bsq_mlm *mlm, int64_t row_len, int64_t nrows, const int64_t *d_row_ptr,
                             const int64_t *d_row_seq, void *d_inputs, int32_t *d_position_ids, int64_t *d_labels);

/* K-mer tokens (DNABERT's overlapping k-mers, Nucleotide Transformer's non-overlapping 6-mers with single-residue
 * tails, reduced-alphabet protein k-mers).  Take a tokenizer with b = nchars codes, its LUT (byte -> code, -1 invalid;
 * bytes >= 0x80 are invalid) and its bos / eos / padchar flags; choose k >= 1, a stride 1 <= s <= k and a tail mode.
 *   Ids depend on (tokenizer, k) only, not on the stride or tail mode:
 *     0 .. b^k - 1      k-mer c_0 ... c_{k-1} -> sum_t c_t * b^(k-1-t)   (the first residue is the most significant)
 *     b^k + c           single residue of code c (tail mode BSQ_KMER_SINGLE)
 *     unk = b^k + b     any k-mer or single residue that contains an invalid byte
 *     unk + 1, ...      BOS (if bos), EOS (if eos), PAD = unk + 1 + bos + eos (always defined, written only with padchar)
 *   vocab_size = b^k + b + 1 + bos + eos + padchar.  BSQ_ERR_ARG when vocab_size - 1 > 2^31 - 1, for the BYTES alphabet
 *   (nchars == 256: its LUT is not a code table), k < 1 or s outside 1..k; the compute calls also reject an output kind
 *   that cannot hold vocab_size - 1 (255 for BSQ_I8, 32767 for BSQ_I16, 2^24 for BSQ_F32, 2^31 - 1 otherwise, as for
 *   bsq_mlm's mask_id).  So DNA allows k <= 15, PROTEIN k <= 7 and the two-letter alphabets k <= 30.
 *   Tokens of one sequence of n residues, before the specials:
 *     m = n >= k ? (n - k) / s + 1 : 0 k-mers, starting at residues 0, s, 2s, ...;
 *     covered = m > 0 ? (m - 1) * s + k : 0 and r = n - covered;
 *     BSQ_KMER_SINGLE: the r residues after `covered` follow, one token each; BSQ_KMER_DROP: they are dropped;
 *     T(n) = m + (single ? r : 0) + bos + eos.
 *   Padded, batch-first (nseq, padlen): row i = [BOS] tokens [EOS], then pad_id with padchar and 0 without (as
 *   bsq_tokenize); T(len_i) <= padlen is the caller's check ("k-mer tokens + bos + eos > padlen: N, vs padlen P").
 *   Padding-free: the rows back to back, int32 cu_seqlens with cu[0] = 0 and cu[i+1] - cu[i] = T(len_i); no PAD.  The
 *   caller has checked that the total is <= 2^31 - 1.
 *   Crop: stage -> crop -> k-mer, with crop_len counted in residues, as for the other consumers.
 * Worked answers: Tokenizer("DNA", bos, eos, padchar) with k = 3: b^k = 64, singles 64..67, unk 68, BOS 69, EOS 70,
 * PAD 71, vocab_size 72 (N is invalid in DNA):
 *     "ACGTNAG"  s = 1, either tail  [69, 6, 27, 68, 68, 68, 70]
 *     "ACGTNAG"  s = 3, single       [69, 6, 68, 66, 70]
 *     "ACGTNAG"  s = 3, drop         [69, 6, 68, 70]
 *     "AC"       any s, single       [69, 64, 65, 70]
 *     "AC"       any s, drop         [69, 70]
 *     ""         any s, either tail  [69, 70]
 */
#define BSQ_KMER_DROP 0
#define BSQ_KMER_SINGLE 1
typedef struct bsq_kmer {
    int32_t k, stride, tail; /* tail: BSQ_KMER_DROP or BSQ_KMER_SINGLE                                        */
    int32_t nchars;          /* b                                                                             */
    int32_t bos, eos, padchar;
    int64_t nkmers;          /* b^k, also the id of the single residue of code 0                            */
    int64_t unk_id;          /* b^k + b                                                                       */
    int64_t bos_id, eos_id;  /* -1 when absent                                                                */
    int64_t pad_id;          /* unk + 1 + bos + eos                                                           */
    int64_t vocab_size;
} bsq_kmer;
/* Host only, no device call: validates (tok, k, stride, tail) as above and fills *km.  The only place the ids are
 * computed. */
int bsq_kmer_init(bsq_kmer *km, const bsq_tokenizer *tok, int k, int stride, int tail);
/* Padded tokens: d_out (nseq, padlen) `kind` elements, batch-first, 16-byte aligned; every element is written once (no
 * memset).  `km` must come from bsq_kmer_init with `tok`.  Enqueues only (one kernel); keeps no state between launches and
 * is capturable into a CUDA graph.  BSQ_ERR_ARG for NULL or misaligned pointers, padlen < 1, nseq < 0 or a kind too
 * narrow for the vocabulary, before any device call. */
int bsq_tokenize_kmer(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int64_t padlen,
                      const bsq_tokenizer *tok, const bsq_kmer *km, int kind, void *d_out);
/* Padding-free tokens: d_out holds exactly the total (16-byte aligned; may be NULL when it is 0) and d_cu_seqlens nseq + 1
 * int32 entries, both written by this call (at most three kernels; nseq == 0: a 4-byte memset of cu_seqlens).  Enqueues
 * only, keeps no state between launches, capturable into a CUDA graph. */
int bsq_tokenize_kmer_varlen(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq,
                             const bsq_tokenizer *tok, const bsq_kmer *km, int kind, void *d_out, int32_t *d_cu_seqlens);
/* *total = sum of T(len_i) and *max_tokens = max T(len_i) (both 0 for nseq == 0) of host offsets, with no device call.
 * BSQ_ERR_ARG for a negative length or offsets[0] < 0. */
int bsq_kmer_extent_host(const int64_t *h_offsets, int64_t nseq, const bsq_kmer *km, int64_t *total, int64_t *max_tokens);
/* The same for device-resident offsets, from one reduction kernel and one read-back (synchronises `stream`); validates
 * the offsets like bsq_crop_extent_device (BSQ_ERR_ARG: negative length, offsets[0] < 0, offsets[nseq] > nbytes when
 * nbytes >= 0). */
int bsq_kmer_extent_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t nbytes, const bsq_kmer *km,
                           int64_t *total, int64_t *max_tokens);

/* Several batches that share padlen and tokenizer in one launch (batch-first one-byte tokens; other layouts / element
 * types fall back to one launch per batch): batch k = (d_bytes[k], d_offsets[k], nseq[k]) -> d_out[k].  The reference's
 * per-step callers tokenise small batches (training/cnnpretrain.py:123-125,145, bioseq/decoders.py:505): a 4096 x 1000
 * batch is 8 MB of traffic, 1.3 us at the HBM roofline and launch-latency-bound when launched alone; up to 32 of them
 * share one persistent grid here.  The pointer arrays are host arrays and are not referenced after the return.
 * (Single launches are also capturable into a CUDA graph: the kernel then uses its static tile order.) */
int bsq_tokenize_many(int device, void *stream, int nbatch, const uint8_t *const *d_bytes, const int64_t *const *d_offsets,
                      const int64_t *nseq, int64_t padlen, const bsq_tokenizer *tok, int batch_first, int kind,
                      void *const *d_out);

/* batch_onehot_encode: d_out is (padlen, nseq, alphabet_size), always sequence-first
 * (src/tokenize.h:323-326); one 1 per position, all-zero rows for invalid or masked-out
 * residues and -- unless padchar -- for the tail (src/tokenize.h:345-368).
 * d_mask: optional, packed like d_bytes (one uint8 per residue, 0 = zero row). */
int bsq_onehot(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets,
               const uint8_t *d_mask, int64_t nseq, int64_t padlen, const bsq_tokenizer *tok,
               int kind, void *d_out);

/* decode_tokens on a (rows, cols) device array of `itemsize`-byte integers with byte
 * strides (a 1-D array is rows = 1).  Two steps so the caller can size the output:
 *   bsq_decode_lengths: validates every token, fills d_row_offsets[rows+1] (exclusive
 *     prefix sum of the decoded row lengths) and returns the total through *total_chars
 *     (synchronises `stream`).  BSQ_ERR_BAD_TOKEN carries the reference's message with
 *     the first offending value in row-major order (src/tokenize.h:148,170).
 *   bsq_decode_chars: writes the decoded characters of row r to
 *     d_chars[d_row_offsets[r] .. d_row_offsets[r+1]).
 * d_row_tail (optional, `rows` int32 entries of device scratch, the same buffer for both calls): the first step
 * records where each row's trailing run of one repeated special begins (the <PAD>s behind a sequence are 4/5 of
 * the decoded text of a padded batch); the second then writes that run as a pattern fill without reading its
 * tokens again.  NULL for either call: every token is decoded one by one. */
int bsq_decode_lengths(int device, void *stream, const void *d_tokens, int itemsize, int64_t rows,
                       int64_t cols, int64_t row_stride, int64_t col_stride, const bsq_tokenizer *tok,
                       int64_t *d_row_offsets, int32_t *d_row_tail, int64_t *total_chars);
int bsq_decode_chars(int device, void *stream, const void *d_tokens, int itemsize, int64_t rows,
                     int64_t cols, int64_t row_stride, int64_t col_stride, const bsq_tokenizer *tok,
                     const int64_t *d_row_offsets, const int32_t *d_row_tail, uint8_t *d_chars);

/* Both passes in ONE call and one host synchronisation (ABI v5): pass 2 is enqueued right behind pass 1 and reads the
 * total on the device, so the GPU does not idle while the host learns the size and allocates.  The caller provides
 * `capacity` bytes at d_chars (a guess: 3 bytes per token covers batches that are up to half <PAD>; 5 per token
 * always suffices).  Returns like bsq_decode_lengths (*total_chars, d_row_offsets, BSQ_ERR_BAD_TOKEN).  If
 * *total_chars > capacity NOTHING was written to d_chars: allocate *total_chars and call bsq_decode_chars with the
 * offsets and hint this call produced. */
int bsq_decode_text(int device, void *stream, const void *d_tokens, int itemsize, int64_t rows, int64_t cols,
                    int64_t row_stride, int64_t col_stride, const bsq_tokenizer *tok, int64_t *d_row_offsets,
                    int32_t *d_row_tail, uint8_t *d_chars, int64_t capacity, int64_t *total_chars);

/* ---- host-staged entry points (the end-to-end path) ------------------------------------ */
/* A stager owns, for one device: a copy stream, device staging buffers for residues /
 * offsets / mask, and a pinned bounce ring for pageable sources.  The *_host calls split
 * the batch into sequence ranges, cudaMemcpyAsync each range host->device on the copy
 * stream and launch its kernel on `stream` as soon as it lands, so the transfer of
 * range k+1 overlaps the compute of range k.  Inputs may be pinned (copied directly) or
 * pageable (bounced through the ring).  Lengths are checked first (bsq_check_lengths_host).
 * The calls return once all work is enqueued.  Pageable sources have been fully read when
 * the call returns; pinned sources are read asynchronously (cudaMemcpyAsync semantics: do
 * not overwrite them until `stream` reaches this point, or call bsq_stager_sync_copies).
 * The staging buffers stay owned by the stager; two sets alternate call by call, so the
 * copies of a call never wait for the kernels of the call before it. */
typedef struct bsq_stager bsq_stager;
int bsq_stager_create(bsq_stager **out, int device);
void bsq_stager_destroy(bsq_stager *s);
/* Block the host until every host->device copy enqueued by earlier *_host calls on this
 * stager has finished, i.e. until the caller may overwrite the host buffers it passed. */
int bsq_stager_sync_copies(bsq_stager *s);
int bsq_tokenize_host(bsq_stager *s, void *stream, const uint8_t *h_bytes, const int64_t *h_offsets,
                      int64_t nseq, int64_t padlen, const bsq_tokenizer *tok, int batch_first,
                      int kind, void *d_out);
int bsq_onehot_host(bsq_stager *s, void *stream, const uint8_t *h_bytes, const int64_t *h_offsets,
                    const uint8_t *h_mask, int64_t nseq, int64_t padlen, const bsq_tokenizer *tok,
                    int kind, void *d_out);

/* The reference's own calling convention (src/tokenize.h:389-419 / :289-322: a sequence of str / bytes / bytearray
 * items, unpacked into borrowed pointers + lengths) as ONE pass over the items, range by range (~4 MiB of
 * residues each): pool threads walk a range's items, gather exactly the items they walked into a pinned pack
 * and write the offsets as they go; the caller's thread enqueues the range's host->device copies and its kernel
 * as soon as it is gathered.  The DMA of range k overlaps the gather of range k+1 and the walk of range k+2;
 * nothing is walked twice, and back-to-back calls do not synchronise with the copy stream (two pinned packs,
 * owned by the stager, alternate).
 *
 * The items stay with their owner:
 *   resolve(ctx, lo, hi, ptrs, lens)   called from pool threads; fills ptrs[i], lens[i] for lo <= i < hi.  It must
 *                                      only read (no allocation, no interpreter calls); lens[i] = -1 defers item i to
 *   fixup(ctx, i, &ptr, &len)          called on the calling thread (may use the interpreter: the caller holds its
 *                                      lock for the whole call, which is also what keeps the items unchanged while the
 *                                      pool reads them -- the reference holds the GIL throughout as well); non-zero =
 *                                      not an accepted item -> BSQ_ERR_ARG "item was none of string, bytes, ..." (:412).
 * Over-long items -> BSQ_ERR_TOO_LONG with the reference's text (:458), found while streaming: ranges enqueued before
 * the offending one have run, the output is to be discarded.  Returns once all work is enqueued; the items are not
 * referenced after the return. */
typedef void (*bsq_resolve_fn)(void *ctx, int64_t lo, int64_t hi, const void **ptrs, int64_t *lens);
typedef int (*bsq_fixup_fn)(void *ctx, int64_t i, const void **ptr, int64_t *len);
int bsq_tokenize_stream_items(bsq_stager *s, void *stream, int64_t n, bsq_resolve_fn resolve, bsq_fixup_fn fixup, void *ctx,
                              int64_t padlen, const bsq_tokenizer *tok, int batch_first, int kind, void *d_out, int nthreads);
int bsq_onehot_stream_items(bsq_stager *s, void *stream, int64_t n, bsq_resolve_fn resolve, bsq_fixup_fn fixup, void *ctx,
                            int64_t padlen, const bsq_tokenizer *tok, int kind, void *d_out, int nthreads);

/* Same pipeline for items that have already been unpacked into pointer / length arrays.  `p` is not used any more
 * (the stager owns its pinned packs) and may be NULL; ptrs/lens are not referenced after the return. */
int bsq_tokenize_items(bsq_stager *s, bsq_pack *p, void *stream, const void *const *ptrs, const int64_t *lens,
                       int64_t n, int64_t padlen, const bsq_tokenizer *tok, int batch_first, int kind,
                       void *d_out, int nthreads);
int bsq_onehot_items(bsq_stager *s, bsq_pack *p, void *stream, const void *const *ptrs, const int64_t *lens,
                     int64_t n, int64_t padlen, const bsq_tokenizer *tok, int kind, void *d_out, int nthreads);

/* ---- one process, several devices (SURVEY.md 8(e): "one host thread per GPU") ------------------------ */
/* The path shards by sequence index with no exchange step: every output row depends on one input sequence.
 * bsq_shard_bounds splits a packed batch into `nshards` contiguous sequence ranges holding equal shares of the
 * RESIDUES (ragged lengths: equal counts would not balance): bounds[0] = 0 <= ... <= bounds[nshards] = nseq.
 * bsq_tokenize_host_sharded runs shard g (sequences bounds[g] .. bounds[g+1]) through stagers[g] / streams[g]
 * into d_outs[g] -- that device's own (n_g, padlen) / (padlen, n_g) / (padlen, n_g, C) array -- with one pool
 * thread per device enqueuing its copies and kernels concurrently; the host source is shared, nothing is
 * gathered between devices.  onehot != 0 selects batch_onehot_encode (batch_first ignored).  The reference's
 * only multi-GPU construct is nn.DataParallel around the model (training/cnnpretrain.py:86), fed by exactly
 * such per-device batches. */
int bsq_shard_bounds(const int64_t *h_offsets, int64_t nseq, int nshards, int64_t *bounds);
int bsq_tokenize_host_sharded(bsq_stager *const *stagers, void *const *streams, int ndev, const uint8_t *h_bytes,
                              const int64_t *h_offsets, int64_t nseq, int64_t padlen, const bsq_tokenizer *tok, int onehot,
                              int batch_first, int kind, void *const *d_outs, const int64_t *bounds);

/* Run fn(t, nthreads, ctx) for t = 0 .. nthreads-1 on the library's persistent host worker pool (the one the
 * gather / scatter loops above use) and return when all have finished.  The reference's counterpart is its
 * OpenMP team (`#pragma omp parallel for num_threads(nthreads)`, src/tokenize.h:340,452); the Python shim uses
 * this for the per-item pointer/length walk of large batches.  fn must not call back into the pool. */
int bsq_parallel_for(int nthreads, void (*fn)(int t, int nthreads, void *ctx), void *ctx);

/* Second half of decode_tokens (src/tokenize.h:131-179 builds one std::string per row): row r of the
 * decoded characters, d_chars[h_offsets[r] .. h_offsets[r+1]), is delivered to host address dst[r] (the body
 * of the string object the caller created for it).  Device->host copies go through a pinned ring in 8 MiB
 * stages on `stream`; `nthreads` pool threads scatter stage k into the rows while stage k+1 is in flight.
 * h_offsets (rows+1 entries) is on the host.  Blocks until every row has arrived. */
int bsq_fetch_rows(bsq_stager *s, void *stream, const uint8_t *d_chars, const int64_t *h_offsets, int64_t rows,
                   void *const *dst, int nthreads);

/* Stage a packed host batch into the stager's device buffers without running a kernel, for the
 * device entry points that have no *_host twin (bsq_embed, bsq_onehot_bcl, ...).  `stream` is made
 * to wait for the copy.  *d_bytes is biased so that residue k of h_bytes is (*d_bytes)[k], i.e. it
 * pairs with the unrebased *d_offsets exactly like h_bytes pairs with h_offsets.  The buffers stay
 * valid until the next *_host / *_items / bsq_stage_host call on this stager; call bsq_stage_release after
 * enqueuing the kernels that read them so that the next staging waits for those kernels. */
int bsq_stage_host(bsq_stager *s, void *stream, const uint8_t *h_bytes, const int64_t *h_offsets, int64_t nseq,
                   const uint8_t **d_bytes, const int64_t **d_offsets);
int bsq_stage_release(bsq_stager *s, void *stream);

/* ---- consumers fused onto the tokeniser (SURVEY.md 8(f) row 4) ------------------------------ */
/* One-hot in (nseq, alphabet_size, padlen) layout: what the reference's CNN path builds from
 * batch_onehot_encode with einops.rearrange("length batch emb -> batch emb length") and .float()
 * (bioseq/loaders.py:74-75, :93-94) -- two extra full-tensor passes -- written here in one pass.
 * Element semantics are bsq_onehot's (src/tokenize.h:345-368); d_mask as there. */
int bsq_onehot_bcl(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, const uint8_t *d_mask,
                   int64_t nseq, int64_t padlen, const bsq_tokenizer *tok, int kind, void *d_out);
/* tokenize -> embedding gather: d_out[(i, p), :] = d_weight[token(i, p), :] with the tokens of
 * bsq_tokenize (never materialised); d_out is (nseq, padlen, row) if batch_first else
 * (padlen, nseq, row).  Replaces batch_tokenize -> torch.from_numpy -> .to(device) -> nn.Embedding
 * (bioseq/__init__.py:171-188 make_embedding and its callers).  Rows are opaque: row_bytes (a
 * multiple of 16) of any element type; nrows >= alphabet_size; d_weight 16-byte aligned. */
int bsq_embed(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int64_t padlen,
              const bsq_tokenizer *tok, int batch_first, const void *d_weight, int64_t nrows, int64_t row_bytes, void *d_out);

/* ---- BLOSUM62 augmentation on the device (SURVEY.md 8(f) row 3) ------------------------------ */
/* augment_seq(seq, chain_len) of bioseq/blosum.py:63-87 applied in place to the packed residues of
 * every selected sequence: chain_len times, draw a position and a substitute from the BLOSUM62
 * row of the residue there (probabilities 2^score / row sum, blosum.py:41-43; anything that is not
 * an upper-case amino acid uses the X row, :60) until the substitute differs, and write it.  A
 * sequence is selected with probability augment_frac (always when >= 1), bioseq/loaders.py:71-73.
 * Randomness is Philox4x32-10 keyed by `seed`, counter (seq_index_base + i, block): the result
 * depends only on (seed, global sequence index), not on batching -- and not on numpy's generator,
 * so it matches the reference in distribution, not draw for draw (oracle/bsq_oracle.c restates the
 * exact procedure).  Empty sequences are left alone. */
int bsq_augment_blosum62(int device, void *stream, uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int chain_len,
                         double augment_frac, uint64_t seed, int64_t seq_index_base);
/* The integer substitution table the kernel samples from: thr[21][19] (rows ARNDCQEGHILKMFPSTWYV + X;
 * floor(2^32 * cumulative probability)), row_of[256] (residue byte -> row), aa[20].  NULLs skipped. */
int bsq_blosum62_thresholds(uint32_t *thr, uint8_t *row_of, uint8_t *aa);
/* Apply bsq_augment_blosum62 to every range the *_host / bsq_stage_host calls of this stager stage,
 * between the copy and the kernel (sequence i of a call has index seq_index_base + i).
 * chain_len 0 switches it off. */
int bsq_stager_set_augment(bsq_stager *s, int chain_len, double augment_frac, uint64_t seed, int64_t seq_index_base);

/* ---- FlatFile: the on-disk packed-sequence store that feeds the path -------------------- */
/* The reference's FlatFile (src/fxstats.cpp:26-134) stores a FASTA/FASTQ collection as
 *     uint64 nseqs | uint64 offsets[nseqs+1] | residue bytes          (src/fxstats.cpp:50-59)
 * which is exactly the packed bytes + offsets form the kernels read: a range of sequences
 * [start, stop) of an open file goes to the GPU as
 *     bsq_tokenize_host(stager, stream, bsq_flatfile_bytes(f), bsq_flatfile_offsets(f) + start,
 *                       stop - start, padlen, tok, batch_first, kind, d_out)
 * with no per-sequence host work (the reference materialises one Python bytearray per
 * sequence, src/fxstats.cpp:128-133, and walks them again in src/tokenize.h:389-419). */
typedef struct bsq_flatfile bsq_flatfile;

#define BSQ_FF_MMAP 0   /* map the file read-only (pageable: staged through the pinned ring)        */
#define BSQ_FF_PINNED 1 /* read the file into cudaHostAlloc'ed memory once (direct DMA afterwards) */
#define BSQ_FF_MMAP_PREFAULT 2 /* BSQ_FF_MMAP with the page tables populated at open (MAP_POPULATE): a streamed first
                                  pass over a page-cache-resident file then runs at copy speed instead of fault speed */
#define BSQ_FF_MMAP_REGISTERED 3 /* BSQ_FF_MMAP_PREFAULT, and the mapping is page-locked IN PLACE (cudaHostRegister):
                                    ranges go to the device by direct DMA like BSQ_FF_PINNED, without a second copy of
                                    the file in memory.  Registered read-only where the platform can; else through a
                                    shared writable mapping of the file (never written) when the file may be opened for
                                    writing; else the file stays BSQ_FF_MMAP_PREFAULT (bsq_flatfile_is_pinned tells). */

/* FlatFile::make (src/fxstats.cpp:33-64): parse a FASTA/FASTQ file (plain or gzip; kseq.h
 * record rules) and write the flat file.  outpath NULL or "" -> inpath + ".ff".  Returns the
 * number of sequences and the longest length through the out-pointers (either may be NULL).
 * BSQ_ERR_IO "<path> failed to open" / "<path> could not be opened for writing" (:41,:53),
 * BSQ_ERR_ARG "Cannot handle sequences longer than 2^32 - 1" (:46). */
int bsq_flatfile_make(const char *inpath, const char *outpath, int64_t *nseqs, int64_t *max_seq_len);
/* FlatFile(path, maxseqlen) (src/fxstats.cpp:66-75).  maxseqlen < 0: computed by a scan of
 * the offsets.  Unlike the reference the header is validated against the file size. */
int bsq_flatfile_open(bsq_flatfile **out, const char *path, int64_t maxseqlen, int mode);
void bsq_flatfile_close(bsq_flatfile *f);
int64_t bsq_flatfile_nseqs(const bsq_flatfile *f);
int64_t bsq_flatfile_seq_offset(const bsq_flatfile *f);  /* (nseqs + 2) * 8, src/fxstats.cpp:67 */
int64_t bsq_flatfile_max_seq_len(const bsq_flatfile *f);
const int64_t *bsq_flatfile_offsets(const bsq_flatfile *f); /* nseqs+1 entries, relative to bsq_flatfile_bytes */
const uint8_t *bsq_flatfile_bytes(const bsq_flatfile *f);   /* sequence i = bytes[offsets[i] .. offsets[i+1]) */
int bsq_flatfile_is_pinned(const bsq_flatfile *f);
/* getstats / getlens (src/fxstats.cpp:12-23, :202-219): sequence lengths of a FASTA/FASTQ
 * file.  *lens is malloc'ed by the callee (free it with bsq_free). */
int bsq_fastx_lengths(const char *path, int64_t **lens, int64_t *n);
void bsq_free(void *p);

/* ---- misc -------------------------------------------------------------------------- */
/* Measurement aid: a plain cudaMemcpyAsync device->device on `stream` (bench.py times it on the same rotating
 * buffers as the tokeniser to put a copy of the same HBM traffic next to the kernel's number). */
int bsq_memcpy_d2d(int device, void *stream, void *d_dst, const void *d_src, size_t nbytes);
int bsq_abi_version(void);
const char *bsq_last_error(void);
/* number of kernel launches issued by this library on the calling thread since the last
 * reset (bench.py's gpu_launches counter). */
int64_t bsq_launch_count(void);
void bsq_launch_count_reset(void);

#ifdef __cplusplus
}
#endif
#endif /* BSQ_H_ */
