// K11: k-mer tokens, padded or padding-free (sm_100a).
//
// Semantics (include/bsq.h, bsq_kmer): row i = [BOS] m_i k-mer ids (residues 0, s, 2s, ...) [single-residue tail]
// [EOS]; a k-mer or single residue with an invalid byte is unk.  T(n) is kmer_tokens (bsq_kernels.cuh).
//
// Every thread fills 16 consecutive output elements at a time (kmer_fill): for the k-mers among them it reads its residue
// window once, in order, through the LUT in shared memory.  The first k-mer of the 16 costs k residues; each next one
// rolls the previous id, id = (id mod b^(k-s)) * b^s + the s new digits, so s residues (a FastDiv, no division).  The last
// invalid residue seen decides which of them are unk.
//   kmer_padded_kernel   flat over the (nseq, padlen) output: thread q takes elements [16q, 16q + 16), so the lanes of a
//                        warp write 512 contiguous elements with 16-byte stores whatever padlen is.  Row and column are
//                        plain arithmetic (a FastDiv by padlen); a 16-element chunk that crosses a row end is filled one
//                        row segment at a time.  Only the batch's last, partial chunk uses element stores.
//   padding-free         K9's scan and carry (bsq_kernels.cuh) write cu_seqlens from T(len_i); then kmer_varlen_kernel,
//                        one warp per row, finishes the row's cu entry as K9's gather does and writes the row's 16-element
//                        chunks of the flat output: 16-byte stores inside the row, element stores in the (at most two)
//                        chunks it shares with its neighbours, so a vector shared by two rows keeps both rows' tokens.
// No scratch memory, no state between launches (capturable into a CUDA graph).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <string>

#include "bsq_internal.h"
#include "bsq_kernels.cuh"

namespace bsq {

namespace {

constexpr int kKThreads = 256;
constexpr uint32_t kKInvalid = 0xFF;  // LUT code of an invalid byte

struct KmerParam {
    KmerShape ks;
    FastDiv keep;    // divides by b^(k - s): id mod b^(k-s) keeps the digits the next k-mer shares
    uint32_t b;      // nchars
    uint32_t nk;     // b^k: first single-residue id
    uint32_t unk, bos_id, eos_id;
    uint32_t pad;    // what follows EOS in a padded row: pad_id with padchar, else 0
};

// the per-row count of the cu_seqlens scan, and the extents' measure: the sum and the max of T(len_i)
struct KmerCountFn {
    KmerShape ks;
    __host__ __device__ __forceinline__ int64_t operator()(int64_t len) const { return kmer_tokens(len, ks); }
    __host__ __device__ __forceinline__ Extent extent(int64_t len) const {
        const int64_t t = kmer_tokens(len, ks);
        return t < 0 ? Extent{kI64Max, 0, kI64Max, true} : Extent{t, 0, t, false};
    }
};

// Ids of columns c_lo + (t - tlo), t in [tlo, thi), of a row of n residues at src, into tok[t].
__device__ __forceinline__ void kmer_fill(uint32_t tok[16], int tlo, int thi, int64_t c_lo, const uint8_t *__restrict__ src,
                                          int64_t n, const KmerParam &p, const uint8_t *lut) {
    const KmerCount kc = kmer_count(n, p.ks);
    const int64_t ntok = kc.m + kc.tail;  // tokens between BOS and EOS
    uint32_t id = 0;
    int64_t lastbad = -1;  // the last invalid residue read
    bool have = false;     // id holds the previous column's k-mer
#pragma unroll
    for (int t = 0; t < 16; ++t) {
        if (t < tlo || t >= thi) continue;
        const int64_t j = c_lo + (t - tlo) - p.ks.bos;
        uint32_t v;
        if (j < 0) {
            v = p.bos_id;
        } else if (j < kc.m) {
            const int64_t p0 = j * p.ks.s;
            int u = 0;
            if (have) {
                id -= fd_div(id, p.keep) * p.keep.d;
                u = p.ks.k - p.ks.s;
            } else {
                id = 0;
            }
            have = true;
            for (; u < p.ks.k; ++u) {
                const uint32_t c = lut[__ldg(src + p0 + u)];
                if (c == kKInvalid) lastbad = p0 + u;
                id = id * p.b + (c == kKInvalid ? 0u : c);
            }
            v = lastbad >= p0 ? p.unk : id;
        } else if (j < ntok) {
            const uint32_t c = lut[__ldg(src + kc.covered + (j - kc.m))];
            v = c == kKInvalid ? p.unk : p.nk + c;
        } else {
            v = (j == ntok && p.ks.eos) ? p.eos_id : p.pad;
        }
        tok[t] = v;
    }
}

template <typename T>
__device__ __forceinline__ T id_value(uint32_t v) {
    if (sizeof(T) == 1) return static_cast<T>(static_cast<uint8_t>(v));  // ids up to 255: the byte as is
    return static_cast<T>(static_cast<int32_t>(v));
}

// tok[t] -> dst[t] for t in [tlo, thi); dst is 16-element aligned in the output (so 16-byte aligned): one or more
// 16-byte stores for a whole chunk, element stores otherwise.
template <typename T>
__device__ __forceinline__ void kmer_store(T *dst, const uint32_t tok[16], int tlo, int thi) {
    if (tlo == 0 && thi == 16) {
        constexpr int EPV = 16 / sizeof(T);
#pragma unroll
        for (int s = 0; s < 16 / EPV; ++s) {
            T vals[EPV];
#pragma unroll
            for (int e = 0; e < EPV; ++e) vals[e] = id_value<T>(tok[s * EPV + e]);
            __stcs(reinterpret_cast<uint4 *>(dst) + s, *reinterpret_cast<const uint4 *>(vals));
        }
    } else {
#pragma unroll
        for (int t = 0; t < 16; ++t)
            if (t >= tlo && t < thi) dst[t] = id_value<T>(tok[t]);
    }
}

__device__ __forceinline__ void kmer_load_lut(uint8_t *lut, const LutParam &lutp) {
    load_lut(lut, lutp);
    __syncthreads();
}

template <typename T>
__global__ void __launch_bounds__(kKThreads)
kmer_padded_kernel(const uint8_t *__restrict__ bytes, const int64_t *__restrict__ offs, int64_t nseq, int64_t padlen,
                   FastDiv pdiv, KmerParam p, LutParam lutp, T *__restrict__ out) {
    __shared__ uint8_t lut[256];
    kmer_load_lut(lut, lutp);
    const int64_t total = nseq * padlen;
    const int64_t nchunks = (total + 15) >> 4;
    const bool small = total < (int64_t(1) << 31);  // row = e0 / padlen by FastDiv
    for (int64_t q = static_cast<int64_t>(blockIdx.x) * kKThreads + threadIdx.x; q < nchunks;
         q += static_cast<int64_t>(gridDim.x) * kKThreads) {
        const int64_t e0 = q << 4;
        const int cnt = static_cast<int>(min(int64_t(16), total - e0));
        int64_t row = small ? static_cast<int64_t>(fd_div(static_cast<uint32_t>(e0), pdiv)) : e0 / padlen;
        int64_t c = e0 - row * padlen;
        uint32_t tok[16];
        int t0 = 0;
        while (t0 < cnt) {  // one pass per row the chunk touches
            const int t1 = static_cast<int>(min(static_cast<int64_t>(cnt), t0 + (padlen - c)));
            const int64_t s0 = __ldg(offs + row);
            kmer_fill(tok, t0, t1, c, bytes + s0, __ldg(offs + row + 1) - s0, p, lut);
            t0 = t1;
            ++row;
            c = 0;
        }
        kmer_store<T>(out + e0, tok, 0, cnt);
    }
}

template <typename T>
__global__ void __launch_bounds__(kKThreads)
kmer_varlen_kernel(const uint8_t *__restrict__ bytes, const int64_t *__restrict__ offs, int64_t n, KmerParam p, LutParam lutp,
                   T *__restrict__ out, int32_t *__restrict__ cu) {
    __shared__ uint8_t lut[256];
    kmer_load_lut(lut, lutp);
    const int lane = threadIdx.x & 31;
    const int64_t i = static_cast<int64_t>(blockIdx.x) * (kKThreads / 32) + (threadIdx.x >> 5);
    if (i >= n) return;
    const int64_t s0 = __ldg(offs + i), len = __ldg(offs + i + 1) - s0;
    const int64_t ntok = kmer_tokens(len, p.ks);
    // the row's end entry: its CTA-local inclusive prefix plus the carry it still lacks
    const int64_t carry = row_scan_carry(cu, i + 1, n);
    const int64_t e = cu[i + 1] + carry;
    __syncwarp();
    if (lane == 0 && carry != 0) cu[i + 1] = static_cast<int32_t>(e);
    const int64_t f0 = e - ntok;
    if (ntok <= 0) return;
    const int64_t q0 = f0 >> 4, q1 = (e - 1) >> 4;
    for (int64_t q = q0 + lane; q <= q1; q += 32) {
        const int tlo = static_cast<int>(max(f0 - 16 * q, int64_t(0)));
        const int thi = static_cast<int>(min(e - 16 * q, int64_t(16)));
        uint32_t tok[16];
        kmer_fill(tok, tlo, thi, 16 * q + tlo - f0, bytes + s0, len, p, lut);
        kmer_store<T>(out + 16 * q, tok, tlo, thi);
    }
}

KmerShape shape_of(const bsq_kmer &km) {
    return KmerShape{km.k, km.stride, km.tail == BSQ_KMER_SINGLE, km.bos, km.eos, make_fastdiv(static_cast<uint32_t>(km.stride))};
}

int64_t kind_limit(int kind) {
    switch (kind) {
        case BSQ_I8: return 255;
        case BSQ_I16: return 32767;
        case BSQ_F32: return int64_t(1) << 24;
        default: return (int64_t(1) << 31) - 1;
    }
}

// A descriptor the caller passes back must be the one bsq_kmer_init makes for this tokenizer.
int check_kmer(const bsq_tokenizer *tok, const bsq_kmer *km, int kind) {
    if (tok == nullptr || km == nullptr) return fail(BSQ_ERR_ARG, "null tokenizer or k-mer descriptor");
    bsq_kmer ref;
    if (int rc = bsq_kmer_init(&ref, tok, km->k, km->stride, km->tail)) return rc;
    if (ref.nchars != km->nchars || ref.bos != km->bos || ref.eos != km->eos || ref.padchar != km->padchar ||
        ref.nkmers != km->nkmers || ref.unk_id != km->unk_id || ref.bos_id != km->bos_id || ref.eos_id != km->eos_id ||
        ref.pad_id != km->pad_id || ref.vocab_size != km->vocab_size)
        return fail(BSQ_ERR_ARG, "k-mer descriptor does not belong to this tokenizer (make it with bsq_kmer_init)");
    if (bsq_kind_size(kind) == 0) return fail(BSQ_ERR_ARG, "invalid element kind");
    if (km->vocab_size - 1 > kind_limit(kind))
        return fail(BSQ_ERR_ARG, "k-mer ids up to " + std::to_string(km->vocab_size - 1) + " do not fit the output kind (at most " +
                                     std::to_string(kind_limit(kind)) + ")");
    return BSQ_OK;
}

void make_param(const bsq_tokenizer &tok, const bsq_kmer &km, KmerParam *p, LutParam *lutp) {
    p->ks = shape_of(km);
    uint32_t keep = 1;
    for (int t = 0; t < km.k - km.stride; ++t) keep *= static_cast<uint32_t>(km.nchars);
    p->keep = make_fastdiv(keep);
    p->b = static_cast<uint32_t>(km.nchars);
    p->nk = static_cast<uint32_t>(km.nkmers);
    p->unk = static_cast<uint32_t>(km.unk_id);
    p->bos_id = static_cast<uint32_t>(km.bos_id);
    p->eos_id = static_cast<uint32_t>(km.eos_id);
    p->pad = km.padchar ? static_cast<uint32_t>(km.pad_id) : 0u;
    uint8_t codes[256];
    for (int b = 0; b < 256; ++b) codes[b] = (b < 0x80 && tok.lut[b] >= 0) ? static_cast<uint8_t>(tok.lut[b]) : kKInvalid;
    std::memcpy(lutp->w, codes, 256);
}

template <typename T>
int launch_kmer(cudaStream_t st, const uint8_t *d_bytes, const int64_t *d_offs, int64_t nseq, int64_t padlen, const KmerParam &p,
                const LutParam &lutp, void *d_out, int32_t *d_cu) {
    T *o = static_cast<T *>(d_out);
    if (d_cu == nullptr) {
        const int64_t nchunks = (nseq * padlen + 15) / 16;
        const int64_t blocks = std::min<int64_t>((nchunks + kKThreads - 1) / kKThreads, static_cast<int64_t>(cur_sms()) * 16);
        const FastDiv pdiv = make_fastdiv(static_cast<uint32_t>(std::min<int64_t>(padlen, (int64_t(1) << 31) - 1)));
        kmer_padded_kernel<T><<<static_cast<unsigned>(blocks), kKThreads, 0, st>>>(d_bytes, d_offs, nseq, padlen, pdiv, p, lutp, o);
        count_launch();
        BSQ_CUDA_TRY(cudaGetLastError());
        return BSQ_OK;
    }
    if (int rc = launch_row_scan(st, d_offs, nseq, KmerCountFn{p.ks}, d_cu)) return rc;
    const int64_t rows_per_cta = kKThreads / 32;
    kmer_varlen_kernel<T><<<static_cast<unsigned>((nseq + rows_per_cta - 1) / rows_per_cta), kKThreads, 0, st>>>(
        d_bytes, d_offs, nseq, p, lutp, o, d_cu);
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}

int dispatch(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int64_t padlen,
             const bsq_tokenizer *tok, const bsq_kmer *km, int kind, void *d_out, int32_t *d_cu) {
    KmerParam p;
    LutParam lutp;
    make_param(*tok, *km, &p, &lutp);
    BSQ_CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (kind) {
        case BSQ_I8: return launch_kmer<int8_t>(st, d_bytes, d_offsets, nseq, padlen, p, lutp, d_out, d_cu);
        case BSQ_I16: return launch_kmer<int16_t>(st, d_bytes, d_offsets, nseq, padlen, p, lutp, d_out, d_cu);
        case BSQ_I32: return launch_kmer<int32_t>(st, d_bytes, d_offsets, nseq, padlen, p, lutp, d_out, d_cu);
        case BSQ_I64: return launch_kmer<int64_t>(st, d_bytes, d_offsets, nseq, padlen, p, lutp, d_out, d_cu);
        case BSQ_F32: return launch_kmer<float>(st, d_bytes, d_offsets, nseq, padlen, p, lutp, d_out, d_cu);
        default: return launch_kmer<double>(st, d_bytes, d_offsets, nseq, padlen, p, lutp, d_out, d_cu);
    }
}

}  // namespace

}  // namespace bsq

using namespace bsq;

extern "C" int bsq_kmer_init(bsq_kmer *km, const bsq_tokenizer *tok, int k, int stride, int tail) {
    if (km == nullptr || tok == nullptr) return fail(BSQ_ERR_ARG, "null k-mer descriptor or tokenizer");
    const int64_t b = tok->nchars;
    if (b >= 256) return fail(BSQ_ERR_ARG, "k-mer tokens need a residue alphabet: BYTES has no code table");
    if (b < 1) return fail(BSQ_ERR_ARG, "tokenizer has no residue codes");
    if (k < 1) return fail(BSQ_ERR_ARG, "k must be >= 1, got " + std::to_string(k));
    if (stride < 1 || stride > k)
        return fail(BSQ_ERR_ARG, "stride must lie in 1..k = " + std::to_string(k) + ", got " + std::to_string(stride));
    if (tail != BSQ_KMER_DROP && tail != BSQ_KMER_SINGLE) return fail(BSQ_ERR_ARG, "tail must be drop (0) or single (1)");
    for (int c = 0; c < 256; ++c)
        if (tok->lut[c] >= b) return fail(BSQ_ERR_ARG, "tokenizer LUT holds a code >= nchars");
    const int64_t kLimit = (int64_t(1) << 31) - 1;
    const int bos = tok->bos_id >= 0, eos = tok->eos_id >= 0, padchar = tok->padchar != 0;
    int64_t nk = 1;
    for (int t = 0; t < k && nk <= kLimit; ++t) nk *= b;
    const int64_t vocab = nk + b + 1 + bos + eos + padchar;  // (nk <= 2^31 * 255: no overflow)
    if (vocab - 1 > kLimit)
        return fail(BSQ_ERR_ARG, "k-mer vocabulary of " + std::string(tok->key) + " with k = " + std::to_string(k) +
                                     " has more than 2^31 ids: choose a smaller k");
    km->k = k;
    km->stride = stride;
    km->tail = tail;
    km->nchars = static_cast<int32_t>(b);
    km->bos = bos;
    km->eos = eos;
    km->padchar = padchar;
    km->nkmers = nk;
    km->unk_id = nk + b;
    km->bos_id = bos ? km->unk_id + 1 : -1;
    km->eos_id = eos ? km->unk_id + 1 + bos : -1;
    km->pad_id = km->unk_id + 1 + bos + eos;
    km->vocab_size = vocab;
    return BSQ_OK;
}

extern "C" int bsq_kmer_extent_host(const int64_t *h_offsets, int64_t nseq, const bsq_kmer *km, int64_t *total,
                                    int64_t *max_tokens) {
    if (km == nullptr || total == nullptr || max_tokens == nullptr) return fail(BSQ_ERR_ARG, "null argument");
    if (nseq < 0 || (nseq > 0 && h_offsets == nullptr)) return fail(BSQ_ERR_ARG, "bad offsets");
    if (km->k < 1 || km->stride < 1 || km->stride > km->k) return fail(BSQ_ERR_ARG, "bad k-mer descriptor");
    *total = *max_tokens = 0;
    if (nseq == 0) return BSQ_OK;
    Extent e{};
    if (int rc = reduce_offsets_host(h_offsets, nseq, KmerCountFn{shape_of(*km)}, &e)) return rc;
    if (e.over) return fail(BSQ_ERR_ARG, "the k-mer tokens exceed INT64_MAX");
    *total = e.sum0;
    *max_tokens = e.max;
    return BSQ_OK;
}

extern "C" int bsq_kmer_extent_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t nbytes,
                                      const bsq_kmer *km, int64_t *total, int64_t *max_tokens) {
    bsq::DeviceRestore restore_device;
    if (km == nullptr || total == nullptr || max_tokens == nullptr) return fail(BSQ_ERR_ARG, "null argument");
    if (nseq < 0 || (nseq > 0 && d_offsets == nullptr)) return fail(BSQ_ERR_ARG, "bad offsets");
    if (km->k < 1 || km->stride < 1 || km->stride > km->k) return fail(BSQ_ERR_ARG, "bad k-mer descriptor");
    *total = *max_tokens = 0;
    if (nseq == 0) return BSQ_OK;
    Extent e{};
    if (int rc = reduce_offsets_device(device, static_cast<cudaStream_t>(stream), d_offsets, nseq, nbytes, KmerCountFn{shape_of(*km)}, &e))
        return rc;
    if (e.over) return fail(BSQ_ERR_ARG, "the k-mer tokens exceed INT64_MAX");
    *total = e.sum0;
    *max_tokens = e.max;
    return BSQ_OK;
}

extern "C" int bsq_tokenize_kmer(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq,
                                 int64_t padlen, const bsq_tokenizer *tok, const bsq_kmer *km, int kind, void *d_out) {
    bsq::DeviceRestore restore_device;
    if (int rc = check_kmer(tok, km, kind)) return rc;
    if (nseq < 0) return fail(BSQ_ERR_ARG, "negative batch size");
    if (padlen < 1) return fail(BSQ_ERR_ARG, "batch tokenize requires padlen is provded.");
    if (nseq == 0) return BSQ_OK;
    if (d_bytes == nullptr || d_offsets == nullptr || d_out == nullptr) return fail(BSQ_ERR_ARG, "null bytes, offsets or output");
    if (reinterpret_cast<uintptr_t>(d_out) & 15u) return fail(BSQ_ERR_ARG, "output pointer must be 16-byte aligned");
    return dispatch(device, stream, d_bytes, d_offsets, nseq, padlen, tok, km, kind, d_out, nullptr);
}

extern "C" int bsq_tokenize_kmer_varlen(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq,
                                        const bsq_tokenizer *tok, const bsq_kmer *km, int kind, void *d_out, int32_t *d_cu_seqlens) {
    bsq::DeviceRestore restore_device;
    if (int rc = check_kmer(tok, km, kind)) return rc;
    if (nseq < 0) return fail(BSQ_ERR_ARG, "negative batch size");
    if (d_cu_seqlens == nullptr) return fail(BSQ_ERR_ARG, "null cu_seqlens");
    if (reinterpret_cast<uintptr_t>(d_out) & 15u) return fail(BSQ_ERR_ARG, "output pointer must be 16-byte aligned");
    if (nseq == 0) {
        BSQ_CUDA_TRY(cudaSetDevice(device));
        BSQ_CUDA_TRY(cudaMemsetAsync(d_cu_seqlens, 0, sizeof(int32_t), static_cast<cudaStream_t>(stream)));
        return BSQ_OK;
    }
    if (d_bytes == nullptr || d_offsets == nullptr) return fail(BSQ_ERR_ARG, "null bytes or offsets");
    return dispatch(device, stream, d_bytes, d_offsets, nseq, 0, tok, km, kind, d_out, d_cu_seqlens);
}
