// K8: masked-language-model batches -- tokens, BERT-style corruption and int64 labels in one pass (sm_100a).
//
// Semantics (include/bsq.h, bsq_tokenize_mlm): start from what bsq_tokenize (batch-first) or bsq_tokenize_varlen writes,
// `tok`.  Only residue positions are eligible: residue j (0 <= j < len_i) of row i, at column bos + j.  With
// g = seq_index_base + i, u = word (j & 3) of Philox4x32-10, counter (g_lo, g_hi, j >> 2, 1), key = seed:
//   u >= t_select          input = tok,        label = ignore_index     (BOS / EOS / PAD are never selected either)
//   u <  t_mask            input = mask_id,    label = tok
//   t_mask <= u < t_random input = random id,  label = tok              random id = (w * nchars) >> 32, w = word (j & 3)
//                                                                       of the block with counter word 3 = 2
//   otherwise              input = tok,        label = tok
// Counter word 3 = 1 and 2 keep these streams disjoint from K7's augmentation stream (word 3 = 0) under one seed.  The
// mask depends on (seed, global sequence index, residue position) only: the same sequence gets the same mask padded
// and padding-free, in any slice of the data.
//
// Labels dominate the bytes (8 per position against 1 of input at kind I8), so both forms are HBM-write-bound maps:
//   mlm_padded_kernel  one thread per 16 columns of one row: 16 codes from tokens16 (bsq_kernels.cuh), the 4-5 Philox
//                      blocks that hold the chunk's residues (none for padding), one st.global.cs.v4 per 16 bytes of
//                      inputs (wide kinds through Expand) and eight for the labels.  Rows whose byte size is not a
//                      multiple of 16 take scalar stores.
//   mlm_varlen_kernel  one thread per 16 output elements of the packed stream: a binary search of cu (computed from the
//                      offsets on the fly) for the vector's row; a vector made of 16 residues of one row takes the same
//                      path as the padded kernel, one that crosses a row boundary or holds BOS / EOS goes element by
//                      element.  The same launch writes cu_seqlens, as K1v does.
// Neither keeps state between launches: both are capturable into a CUDA graph.
#include <cuda_runtime.h>

#include <algorithm>

#include "bsq_internal.h"
#include "bsq_kernels.cuh"

namespace bsq {

namespace {

constexpr int kMThreads = 256;

// ------------------------------------------------------------------------------------------------------------------
// padded, batch-first: item = (row, 16-column chunk); `items` < 2^31 (the host splits larger batches by rows)
template <typename T, bool VEC>
__global__ void __launch_bounds__(kMThreads)
mlm_padded_kernel(SeqView v, uint32_t items, FastDiv cpr, int padlen, LutParam lutp, Specials sp, Expand ex, MlmParam m,
                  T *__restrict__ in, int64_t *__restrict__ lab) {
    __shared__ __align__(16) uint8_t lut[256];
    __shared__ TailTab tab;
    load_lut(lut, lutp);
    init_tailtab(tab, sp);
    __syncthreads();
    for (uint32_t it = blockIdx.x * kMThreads + threadIdx.x; it < items; it += gridDim.x * kMThreads) {
        const uint32_t row = fd_div(it, cpr);
        const int c0 = static_cast<int>(it - row * cpr.d) * 16;
        const int64_t start = __ldg(v.offs + row);
        const int len = static_cast<int>(__ldg(v.offs + row + 1) - start);
        uint32_t t[4];
        if (c0 >= sp.bos + len + sp.eos) {
            t[0] = t[1] = t[2] = t[3] = sp.pad_w;
        } else {
            const RowSrc rs = make_rowsrc(v.bytes, start, sp.bos, len);
            const uint4 c = tokens16<false>(rs, nullptr, len, c0, sp, lut, tab);
            t[0] = c.x; t[1] = c.y; t[2] = c.z; t[3] = c.w;
        }
        const Mlm16 d = mlm_decide16(c0 - sp.bos, len, static_cast<uint64_t>(m.base + row), m);
        const size_t o = static_cast<size_t>(row) * padlen + c0;
        const int cnt = min(16, padlen - c0);
        if (VEC && cnt == 16) mlm_emit16<T, true>(in + o, lab + o, t, d, 16, m, ex);
        else mlm_emit16<T, false>(in + o, lab + o, t, d, cnt, m, ex);  // (VEC: the row's last, partial chunk)
    }
}

// ------------------------------------------------------------------------------------------------------------------
// padding-free: cu[i] = offsets[i] - offsets[0] + i * k, tokens[cu[i] .. cu[i+1]) = row i of the padded form, unpadded
template <typename T>
__global__ void __launch_bounds__(kMThreads)
mlm_varlen_kernel(const uint8_t *__restrict__ bytes, const int64_t *__restrict__ offs, int64_t n, LutParam lutp, Specials sp,
                  Expand ex, MlmParam m, T *__restrict__ in, int64_t *__restrict__ lab, int32_t *__restrict__ cu) {
    __shared__ __align__(16) uint8_t lut[256];
    load_lut(lut, lutp);
    const int k = sp.bos + sp.eos;
    const int64_t off0 = __ldg(offs), total = __ldg(offs + n) - off0 + n * k;
    for (int64_t i = blockIdx.x * static_cast<int64_t>(kMThreads) + threadIdx.x; i <= n; i += static_cast<int64_t>(gridDim.x) * kMThreads)
        cu[i] = static_cast<int32_t>(__ldg(offs + i) - off0 + i * k);
    __syncthreads();
    auto cu_g = [&](int64_t i) { return __ldg(offs + i) - off0 + i * k; };
    const int64_t nvec = (total + 15) / 16;
    for (int64_t vi = blockIdx.x * static_cast<int64_t>(kMThreads) + threadIdx.x; vi < nvec; vi += static_cast<int64_t>(gridDim.x) * kMThreads) {
        const int64_t f0 = 16 * vi;
        const int cnt = static_cast<int>(min(int64_t(16), total - f0));
        // the row of element f0: the largest r < n with cu[r] <= f0 (empty rows before it are skipped)
        int64_t lo = 0, hi = n;
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if (cu_g(mid) <= f0) lo = mid;
            else hi = mid;
        }
        int64_t row = lo, cs = cu_g(row), ce = cu_g(row + 1);
        const int c = static_cast<int>(f0 - cs);
        if (cnt == 16 && c >= sp.bos && c + 16 <= static_cast<int>(ce - cs) - sp.eos) {
            // 16 residues of one row: the padded kernel's path
            const int64_t start = __ldg(offs + row);
            const int len = static_cast<int>(ce - cs) - k;
            const RowSrc rs = make_rowsrc(bytes, start, sp.bos, len);
            uint32_t raw[4], t[4];
            fetch16(rs, c, raw);
#pragma unroll
            for (int w = 0; w < 4; ++w) t[w] = translate4(raw[w], lut);
            const Mlm16 d = mlm_decide16(c - sp.bos, len, static_cast<uint64_t>(m.base + row), m);
            mlm_emit16<T, true>(in + f0, lab + f0, t, d, 16, m, ex);
            continue;
        }
        // row boundaries, BOS / EOS or the batch's last vector: element by element
        uint64_t cached_g = ~0ull;
        uint32_t cached_blk = ~0u;
        Philox cp;
        cp.c[0] = cp.c[1] = cp.c[2] = cp.c[3] = 0u;
#pragma unroll 1
        for (int p = 0; p < cnt; ++p) {
            const int64_t e = f0 + p;
            while (ce <= e) {  // the next row starts here (empty rows emit k elements each, or none when k = 0)
                ++row;
                cs = ce;
                ce = cu_g(row + 1);
            }
            const int cc = static_cast<int>(e - cs), len = static_cast<int>(ce - cs) - k;
            uint32_t code;
            bool res = false;
            if (cc < sp.bos) {
                code = sp.bos_w & 0xffu;
            } else if (cc - sp.bos < len) {
                code = lut[__ldg(bytes + off0 + e - row * k - sp.bos)];
                res = true;
            } else {
                code = sp.eos_w & 0xffu;
            }
            T val = code_value<T>(code, ex);
            int64_t label = m.ignore;
            if (res) {
                const uint32_t j = static_cast<uint32_t>(cc - sp.bos);
                const uint64_t g = static_cast<uint64_t>(m.base + row);
                if (g != cached_g || (j >> 2) != cached_blk) {
                    cp = mlm_block(g, j >> 2, 1u, m);
                    cached_g = g;
                    cached_blk = j >> 2;
                }
                const uint64_t u = pick4(cp, j & 3u);
                if (u < m.ts) {
                    label = code;
                    if (u < m.tm) val = static_cast<T>(m.mask_id);
                    else if (u < m.tr) val = static_cast<T>(static_cast<int32_t>(mlm_random_id(g, j, m)));
                }
            }
            in[e] = val;
            lab[e] = label;
        }
    }
}

// Persistent grids are sized to the CTAs that are resident at once: every CTA strides over an equal share, so a CTA
// that had to wait for a free slot would double the launch's time.
template <typename K>
int resident_grid(K kern, int64_t work, int64_t per_cta) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kMThreads, 0) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        per_sm = 1;
    }
    const int64_t want = std::max<int64_t>(1, (work + per_cta - 1) / per_cta);
    return static_cast<int>(std::min<int64_t>(want, static_cast<int64_t>(cur_sms()) * per_sm));
}

template <typename T>
int launch_mlm_padded(cudaStream_t st, const uint8_t *d_bytes, const int64_t *d_offs, int64_t nseq, int64_t padlen,
                      const bsq_tokenizer &tok, MlmParam m, void *d_in, int64_t *d_lab) {
    const Prepared p = prepare(tok, sizeof(T) == 1 ? 0 : 1);
    const int64_t cpr = (padlen + 15) / 16;
    const bool vec = (padlen * static_cast<int64_t>(sizeof(T))) % 16 == 0 && padlen % 2 == 0;
    const int64_t rows_per_launch = std::max<int64_t>(1, 0x7fffffffll / cpr);
    for (int64_t r0 = 0; r0 < nseq; r0 += rows_per_launch) {
        const int64_t nr = std::min(rows_per_launch, nseq - r0);
        const uint32_t items = static_cast<uint32_t>(nr * cpr);
        const SeqView v{d_bytes, d_offs + r0, nullptr};
        T *in = static_cast<T *>(d_in) + r0 * padlen;
        int64_t *lab = d_lab + r0 * padlen;
        MlmParam mr = m;
        mr.base = m.base + r0;
        const FastDiv fd = make_fastdiv(static_cast<uint32_t>(cpr));
        const int pl = static_cast<int>(padlen);
        auto kern = vec ? mlm_padded_kernel<T, true> : mlm_padded_kernel<T, false>;
        kern<<<resident_grid(kern, items, kMThreads), kMThreads, 0, st>>>(v, items, fd, pl, p.lut, p.sp, p.ex, mr, in, lab);
        count_launch();
        BSQ_CUDA_TRY(cudaGetLastError());
    }
    return BSQ_OK;
}

template <typename T>
int launch_mlm_varlen(cudaStream_t st, const uint8_t *d_bytes, const int64_t *d_offs, int64_t nseq, const bsq_tokenizer &tok,
                      MlmParam m, void *d_in, int64_t *d_lab, int32_t *d_cu) {
    const Prepared p = prepare(tok, sizeof(T) == 1 ? 0 : 1);
    // the output's extent lives on the device: a persistent grid strides over whatever it is
    const int grid = resident_grid(mlm_varlen_kernel<T>, int64_t(1) << 40, kMThreads);
    mlm_varlen_kernel<T><<<grid, kMThreads, 0, st>>>(d_bytes, d_offs, nseq, p.lut, p.sp, p.ex, m, static_cast<T *>(d_in), d_lab, d_cu);
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}

}  // namespace

// BSQ_ERR_ARG cases shared by K8's and K10's MLM entry points
int check_mlm_param(const bsq_tokenizer *tok, int kind, const bsq_mlm *mlm, MlmParam *m) {
    if (tok == nullptr) return fail(BSQ_ERR_ARG, "null tokenizer");
    if (bsq_kind_size(kind) == 0) return fail(BSQ_ERR_ARG, "invalid element kind");
    if (mlm == nullptr) return fail(BSQ_ERR_ARG, "null bsq_mlm");
    if (!(mlm->t_mask <= mlm->t_random && mlm->t_random <= mlm->t_select && mlm->t_select <= (1ull << 32)))
        return fail(BSQ_ERR_ARG, "MLM thresholds must satisfy t_mask <= t_random <= t_select <= 2^32");
    int64_t max_id = 0x7fffffffll;
    if (kind == BSQ_I8) max_id = 255;
    else if (kind == BSQ_I16) max_id = 32767;
    else if (kind == BSQ_F32) max_id = 1ll << 24;
    if (mlm->mask_id < 0 || mlm->mask_id > max_id)
        return fail(BSQ_ERR_ARG, "mask_id " + std::to_string(mlm->mask_id) + " is not representable in the output kind (0.." +
                                     std::to_string(max_id) + ")");
    m->k0 = static_cast<uint32_t>(mlm->seed);
    m->k1 = static_cast<uint32_t>(mlm->seed >> 32);
    m->ts = mlm->t_select;
    m->tm = mlm->t_mask;
    m->tr = mlm->t_random;
    m->base = mlm->seq_index_base;
    m->ignore = mlm->ignore_index;
    m->mask_id = static_cast<int32_t>(mlm->mask_id);
    m->nchars = static_cast<uint32_t>(tok->nchars);
    return BSQ_OK;
}

}  // namespace bsq

using namespace bsq;

#define BSQ_MLM_DISPATCH(FN, ...)                                    \
    switch (kind) {                                                  \
        case BSQ_I8: return FN<int8_t>(__VA_ARGS__);                 \
        case BSQ_I16: return FN<int16_t>(__VA_ARGS__);               \
        case BSQ_I32: return FN<int32_t>(__VA_ARGS__);               \
        case BSQ_I64: return FN<int64_t>(__VA_ARGS__);               \
        case BSQ_F32: return FN<float>(__VA_ARGS__);                 \
        default: return FN<double>(__VA_ARGS__);                     \
    }

extern "C" int bsq_tokenize_mlm(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq,
                                int64_t padlen, const bsq_tokenizer *tok, int kind, const bsq_mlm *mlm, void *d_inputs,
                                int64_t *d_labels) {
    bsq::DeviceRestore restore_device;
    MlmParam m;
    if (int rc = check_mlm_param(tok, kind, mlm, &m)) return rc;
    if (int rc = check_launch_args(device, nseq, padlen, tok, kind, d_inputs)) return rc;
    if (nseq == 0) return BSQ_OK;
    if (d_offsets == nullptr) return fail(BSQ_ERR_ARG, "null offsets");
    if (d_labels == nullptr || (reinterpret_cast<uintptr_t>(d_labels) & 15u))
        return fail(BSQ_ERR_ARG, "labels pointer must be non-null and 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    BSQ_MLM_DISPATCH(launch_mlm_padded, st, d_bytes, d_offsets, nseq, padlen, *tok, m, d_inputs, d_labels)
}

extern "C" int bsq_tokenize_varlen_mlm(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq,
                                       const bsq_tokenizer *tok, int kind, const bsq_mlm *mlm, void *d_inputs, int64_t *d_labels,
                                       int32_t *d_cu_seqlens) {
    bsq::DeviceRestore restore_device;
    MlmParam m;
    if (int rc = check_mlm_param(tok, kind, mlm, &m)) return rc;
    if (nseq < 0) return fail(BSQ_ERR_ARG, "negative batch size");
    if (d_offsets == nullptr || d_cu_seqlens == nullptr) return fail(BSQ_ERR_ARG, "null offsets or cu_seqlens");
    if ((reinterpret_cast<uintptr_t>(d_inputs) & 15u) || (reinterpret_cast<uintptr_t>(d_labels) & 15u))
        return fail(BSQ_ERR_ARG, "inputs and labels pointers must be 16-byte aligned");
    BSQ_CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nseq == 0) {
        BSQ_CUDA_TRY(cudaMemsetAsync(d_cu_seqlens, 0, sizeof(int32_t), st));
        return BSQ_OK;
    }
    BSQ_MLM_DISPATCH(launch_mlm_varlen, st, d_bytes, d_offsets, nseq, *tok, m, d_inputs, d_labels, d_cu_seqlens)
}
