// K10: sequence packing -- whole sequences best-fit into fixed-width rows, with position ids and optional MLM labels
// (sm_100a), and the host planner that lays them out.
//
// Semantics (include/bsq.h, bsq_seqpack_plan / bsq_tokenize_seqpack): sequence i occupies need_i = len_i + k tokens
// (k = bos + eos) of one row of width L: [BOS] lut(residues) [EOS], exactly row i of bsq_tokenize_varlen.  The rest of a
// row is padding, written as bsq_tokenize writes it after EOS.  Position ids restart at 0 in every segment (a placed
// sequence or a row's padding run).
//
// The planner (host) is best-fit decreasing in O(n log L): a stable counting sort by need (a stable sort of indices when
// L is large next to n), then, for each sequence, the open row with the least remaining space that still fits it, ties
// to the lowest row index.  Open rows are kept in buckets by remaining space, each a min-heap of row indices; a two-level
// bitset over the buckets finds the first non-empty bucket at or above `need` in a few word scans.  Very wide rows
// (L > kDenseMax) key the buckets in an ordered map instead: the same rule, O(n log n).
//
// The kernel (seqpack_kernel) is output-driven: one warp per row walks the row's sequences (row_ptr / row_seq, the
// plan's CSR) and then its padding run; every element of tokens, position ids and labels is written exactly once, so no
// memset precedes it.  Inside a segment the warp's lanes take the 16-element chunks of the flat output (chunk q =
// elements 16q .. 16q + 15, so every chunk is 16-byte aligned whatever the row width):
//   - a chunk of 16 residues: two aligned 16-byte loads of the source realigned by funnel shifts (the shift is the same
//     for the whole segment: K9's scheme), 16 LUT look-ups, one st.global.cs.v4 per 16 bytes of tokens; with MLM the
//     16 decisions and the stores of K8 (mlm_decide16 / mlm_emit16, bsq_kernels.cuh);
//   - a chunk of padding: the pad vector, a pattern fill;
//   - position ids of a whole chunk: four 16-byte stores of c0 .. c0 + 15, computed, not loaded;
//   - chunks that hold a segment edge, BOS or EOS: element stores.
// Nothing is kept between launches: the kernel is capturable into a CUDA graph.
#include <cuda_runtime.h>

#include <algorithm>
#include <map>
#include <numeric>
#include <vector>

#include "bsq_internal.h"
#include "bsq_kernels.cuh"

namespace bsq {

namespace {

constexpr int kPThreads = 256;              // 8 warps, one row each
constexpr int64_t kDenseMax = 1 << 18;      // row widths up to this use dense buckets (a bitset of 2^18 bits: 32 KiB)

// ------------------------------------------------------------------------------------------------------------------
// host planner

// Buckets of open rows by remaining space 1 .. L, each a min-heap of row indices.
class DenseBuckets {
public:
    explicit DenseBuckets(int64_t L) : heaps_(L + 1), lo_((L + 64) / 64, 0), hi_((lo_.size() + 63) / 64, 0) {}
    void push(int64_t cap, int64_t row) {
        auto &h = heaps_[cap];
        h.push_back(row);
        std::push_heap(h.begin(), h.end(), std::greater<int64_t>());
        lo_[cap >> 6] |= 1ull << (cap & 63);
        hi_[cap >> 12] |= 1ull << ((cap >> 6) & 63);
    }
    // the lowest row of the smallest non-empty bucket >= need, removed; -1 if none
    int64_t pop_fit(int64_t need, int64_t *cap) {
        const int64_t c = next_set(need);
        if (c < 0) return -1;
        auto &h = heaps_[c];
        std::pop_heap(h.begin(), h.end(), std::greater<int64_t>());
        const int64_t row = h.back();
        h.pop_back();
        if (h.empty()) {
            lo_[c >> 6] &= ~(1ull << (c & 63));
            if (lo_[c >> 6] == 0) hi_[c >> 12] &= ~(1ull << ((c >> 6) & 63));
        }
        *cap = c;
        return row;
    }

private:
    int64_t next_set(int64_t x) const {
        int64_t w = x >> 6;
        if (w >= static_cast<int64_t>(lo_.size())) return -1;
        uint64_t bits = lo_[w] & (~0ull << (x & 63));
        if (bits) return (w << 6) + __builtin_ctzll(bits);
        // the next non-empty word after w, from the summary
        int64_t s = (w + 1) >> 6;
        if (s >= static_cast<int64_t>(hi_.size())) return -1;
        uint64_t sb = ((w + 1) & 63) ? hi_[s] & (~0ull << ((w + 1) & 63)) : hi_[s];
        while (!sb) {
            if (++s >= static_cast<int64_t>(hi_.size())) return -1;
            sb = hi_[s];
        }
        w = (s << 6) + __builtin_ctzll(sb);
        return (w << 6) + __builtin_ctzll(lo_[w]);
    }
    std::vector<std::vector<int64_t>> heaps_;
    std::vector<uint64_t> lo_, hi_;
};

class SparseBuckets {
public:
    void push(int64_t cap, int64_t row) {
        auto &h = m_[cap];
        h.push_back(row);
        std::push_heap(h.begin(), h.end(), std::greater<int64_t>());
    }
    int64_t pop_fit(int64_t need, int64_t *cap) {
        auto it = m_.lower_bound(need);
        if (it == m_.end()) return -1;
        auto &h = it->second;
        std::pop_heap(h.begin(), h.end(), std::greater<int64_t>());
        const int64_t row = h.back();
        h.pop_back();
        *cap = it->first;
        if (h.empty()) m_.erase(it);
        return row;
    }

private:
    std::map<int64_t, std::vector<int64_t>> m_;
};

// Best-fit decreasing: row_of[i] and col[i] of every sequence with need > 0 (row -1 otherwise); returns the rows used.
template <typename Buckets>
int64_t best_fit(Buckets &b, const std::vector<int64_t> &order, const std::vector<int64_t> &need, int64_t L,
                 std::vector<int64_t> &row_of, std::vector<int64_t> &col) {
    int64_t nrows = 0;
    for (const int64_t i : order) {
        const int64_t w = need[i];
        int64_t cap = 0;
        int64_t r = b.pop_fit(w, &cap);
        if (r < 0) {
            r = nrows++;
            cap = L;
        }
        row_of[i] = r;
        col[i] = L - cap;
        if (cap - w > 0) b.push(cap - w, r);
    }
    return nrows;
}

}  // namespace

}  // namespace bsq

using namespace bsq;

extern "C" int bsq_seqpack_plan(const int64_t *h_offsets, int64_t nseq, int k, int64_t row_len, int64_t rows, int64_t *nrows,
                                int64_t *nsegments, int64_t *max_seqlen, int64_t *starts, int64_t *row_ptr, int64_t *row_seq,
                                int32_t *cu_seqlens) {
    if (nseq < 0) return fail(BSQ_ERR_ARG, "negative batch size");
    if (k < 0 || k > 2) return fail(BSQ_ERR_ARG, "k = bos + eos must be 0, 1 or 2");
    if (row_len < 1) return fail(BSQ_ERR_ARG, "row_len must be >= 1");
    if (nseq > 0 && h_offsets == nullptr) return fail(BSQ_ERR_ARG, "null offsets");
    if (nrows == nullptr || nsegments == nullptr || max_seqlen == nullptr) return fail(BSQ_ERR_ARG, "null nrows, nsegments or max_seqlen");
    const bool sizing = starts == nullptr && row_ptr == nullptr && row_seq == nullptr && cu_seqlens == nullptr;
    if (!sizing && (starts == nullptr || row_ptr == nullptr || row_seq == nullptr || cu_seqlens == nullptr))
        return fail(BSQ_ERR_ARG, "starts, row_ptr, row_seq and cu_seqlens must all be given, or none (sizing call)");
    const int64_t L = row_len;
    std::vector<int64_t> need(static_cast<size_t>(nseq));
    int64_t placed = 0;
    for (int64_t i = 0; i < nseq; ++i) {
        const int64_t len = h_offsets[i + 1] - h_offsets[i];
        if (len < 0 || (i == 0 && h_offsets[0] < 0)) return fail(BSQ_ERR_ARG, "offsets must start at or after 0 and be non-decreasing");
        need[i] = len + k;
        if (need[i] > L)
            return fail(BSQ_ERR_ARG, "seq len + bos + eos > padlen: " + std::to_string(need[i]) + ", vs padlen " + std::to_string(L));
        placed += need[i] > 0;
    }
    // placement order: decreasing need, ties to the lower index (stable)
    std::vector<int64_t> order(static_cast<size_t>(placed));
    if (L <= std::max<int64_t>(kDenseMax, 4 * nseq) && L <= kDenseMax * 64) {
        std::vector<int64_t> cnt(static_cast<size_t>(L + 2), 0);  // counting sort on L - need
        for (int64_t i = 0; i < nseq; ++i)
            if (need[i] > 0) ++cnt[L - need[i] + 1];
        for (int64_t v = 1; v <= L + 1; ++v) cnt[v] += cnt[v - 1];
        for (int64_t i = 0; i < nseq; ++i)
            if (need[i] > 0) order[cnt[L - need[i]]++] = i;
    } else {
        int64_t j = 0;
        for (int64_t i = 0; i < nseq; ++i)
            if (need[i] > 0) order[j++] = i;
        std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) { return need[a] > need[b]; });
    }
    std::vector<int64_t> row_of(static_cast<size_t>(nseq), -1), col(static_cast<size_t>(nseq), 0);
    int64_t R;
    if (L <= kDenseMax) {
        DenseBuckets b(L);
        R = best_fit(b, order, need, L, row_of, col);
    } else {
        SparseBuckets b;
        R = best_fit(b, order, need, L, row_of, col);
    }
    if (rows > 0) {
        if (R > rows)
            return fail(BSQ_ERR_ARG, "the batch needs " + std::to_string(R) + " rows of " + std::to_string(L) + ", more than rows = " +
                                         std::to_string(rows));
        R = rows;
    }
    if (R > 0 && R > 0x7fffffffll / L)
        return fail(BSQ_ERR_ARG, std::to_string(R) + " rows of " + std::to_string(L) + " tokens exceed 2^31 - 1 tokens: cu_seqlens is int32; "
                                     "split the batch");
    // per-row fill, and the CSR in column order (placement order within a row is increasing column)
    std::vector<int64_t> fill(static_cast<size_t>(R), 0), rp(static_cast<size_t>(R + 1), 0);
    int64_t mx = 0;
    for (const int64_t i : order) {
        fill[row_of[i]] += need[i];
        ++rp[row_of[i] + 1];
        mx = std::max(mx, need[i]);
    }
    int64_t nseg = placed;
    for (int64_t r = 0; r < R; ++r) {
        rp[r + 1] += rp[r];
        if (fill[r] < L) {
            ++nseg;
            mx = std::max(mx, L - fill[r]);
        }
    }
    *nrows = R;
    *nsegments = nseg;
    *max_seqlen = mx;
    if (sizing) return BSQ_OK;
    std::copy(rp.begin(), rp.end(), row_ptr);
    {
        std::vector<int64_t> next(rp.begin(), rp.end() - 1);
        for (const int64_t i : order) row_seq[next[row_of[i]]++] = i;
    }
    for (int64_t i = 0; i < nseq; ++i) starts[i] = row_of[i] < 0 ? -1 : row_of[i] * L + col[i];
    int64_t s = 0;
    for (int64_t r = 0; r < R; ++r) {
        for (int64_t p = rp[r]; p < rp[r + 1]; ++p) cu_seqlens[s++] = static_cast<int32_t>(starts[row_seq[p]]);
        if (fill[r] < L) cu_seqlens[s++] = static_cast<int32_t>(r * L + fill[r]);
    }
    cu_seqlens[s] = static_cast<int32_t>(R * L);
    return BSQ_OK;
}

namespace bsq {

namespace {

// ------------------------------------------------------------------------------------------------------------------
// device

// the bits of one element, zero-extended
__device__ __forceinline__ uint64_t sp_bits(int8_t v) { return static_cast<uint8_t>(v); }
__device__ __forceinline__ uint64_t sp_bits(int16_t v) { return static_cast<uint16_t>(v); }
__device__ __forceinline__ uint64_t sp_bits(int32_t v) { return static_cast<uint32_t>(v); }
__device__ __forceinline__ uint64_t sp_bits(int64_t v) { return static_cast<uint64_t>(v); }
__device__ __forceinline__ uint64_t sp_bits(float v) { return __float_as_uint(v); }
__device__ __forceinline__ uint64_t sp_bits(double v) { return static_cast<uint64_t>(__double_as_longlong(v)); }

// 16 codes (bytes) -> 16 elements at the 16-byte aligned `out`
template <typename T>
__device__ __forceinline__ void sp_store16(T *out, const uint32_t t[4], const Expand &ex) {
    if (sizeof(T) == 1) {
        __stcs(reinterpret_cast<uint4 *>(out), make_uint4(t[0], t[1], t[2], t[3]));
        return;
    }
    // the element bits packed into words with shifts (an array reinterpreted as uint4 would live in local memory)
    constexpr int EPV = 16 / sizeof(T), B = 8 * sizeof(T);
#pragma unroll
    for (int s = 0; s < 16 / EPV; ++s) {
        uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int j = 0; j < EPV; ++j) {
            const int e = s * EPV + j;
            const uint64_t b = sp_bits(code_value<T>((t[e >> 2] >> (8 * (e & 3))) & 0xffu, ex));
            if (B == 64) {
                w[2 * j] = static_cast<uint32_t>(b);
                w[2 * j + 1] = static_cast<uint32_t>(b >> 32);
            } else {
                w[(j * B) >> 5] |= static_cast<uint32_t>(b) << ((j * B) & 31);
            }
        }
        __stcs(reinterpret_cast<uint4 *>(out) + s, make_uint4(w[0], w[1], w[2], w[3]));
    }
}

// position ids c0 .. c0 + 15 at the 16-byte aligned `pos`
__device__ __forceinline__ void sp_pos16(int32_t *pos, int c0) {
#pragma unroll
    for (int s = 0; s < 4; ++s)
        __stcs(reinterpret_cast<int4 *>(pos) + s, make_int4(c0 + 4 * s, c0 + 4 * s + 1, c0 + 4 * s + 2, c0 + 4 * s + 3));
}

// One segment of a row: flat elements [fa, fa + w).  seq: a sequence of `len` residues at src (global index g for MLM;
// src may be null when len == 0: an all-empty batch has no residue buffer); otherwise the row's padding run.
template <typename T, bool MLM>
__device__ __forceinline__ void sp_segment(int64_t fa, int w, bool seq, const uint8_t *src, int len, uint64_t g, const Specials &sp,
                                           const uint8_t *lut, const Expand &ex, const MlmParam &m, T *__restrict__ out,
                                           int32_t *__restrict__ pos, int64_t *__restrict__ lab, int lane) {
    const int64_t fb = fa + w;
    const int64_t q_end = (fb + 15) >> 4;
    // the source shift of a chunk's first residue is the same for every chunk of the segment
    const uintptr_t sbase = reinterpret_cast<uintptr_t>(src);
    for (int64_t q = (fa >> 4) + lane; q < q_end; q += 32) {
        const int64_t f0 = q << 4;
        const int c0 = static_cast<int>(f0 - fa);  // column in the segment of the chunk's element 0 (may be < 0)
        const bool full = c0 >= 0 && c0 + 16 <= w;
        if (full && !seq) {
            const uint32_t pw = sp.pad_w;
            const uint32_t t[4] = {pw, pw, pw, pw};
            sp_store16<T>(out + f0, t, ex);
            sp_pos16(pos + f0, c0);
            if (MLM) {
                const longlong2 ig = make_longlong2(m.ignore, m.ignore);
#pragma unroll
                for (int s = 0; s < 8; ++s) __stcs(reinterpret_cast<longlong2 *>(lab + f0) + s, ig);
            }
            continue;
        }
        const int j0 = c0 - sp.bos;  // residue index of the chunk's element 0
        if (full && j0 >= 0 && j0 + 16 <= len) {
            const uintptr_t a = sbase + static_cast<uint32_t>(j0);
            const uint32_t shift = static_cast<uint32_t>(a & 15u);
            Fetched fe;
            fe.v0 = ldg16(a - shift);
            fe.v1 = shift != 0 ? ldg16(a - shift + 16) : make_uint4(0u, 0u, 0u, 0u);
            RowSrc rs;
            rs.off = static_cast<int>(shift);
            uint32_t t[4];
            fetch_align(fe, rs, 0, t);
#pragma unroll
            for (int i = 0; i < 4; ++i) t[i] = translate4(t[i], lut);
            if (MLM) {
                const Mlm16 d = mlm_decide16(j0, len, g, m);
                mlm_emit16<T, true>(out + f0, lab + f0, t, d, 16, m, ex);
            } else {
                sp_store16<T>(out + f0, t, ex);
            }
            sp_pos16(pos + f0, c0);
            continue;
        }
        // segment edges, BOS / EOS: element by element
        const int e_lo = max(c0, 0), e_hi = min(c0 + 16, w);
#pragma unroll 1
        for (int c = e_lo; c < e_hi; ++c) {
            const int64_t f = fa + c;
            const int j = c - sp.bos;
            uint32_t code;
            bool res = false;
            if (!seq) code = sp.pad_w & 0xffu;
            else if (j < 0) code = sp.bos_w & 0xffu;
            else if (j < len) {
                code = lut[__ldg(src + j)];
                res = true;
            } else code = sp.eos_w & 0xffu;
            T val = code_value<T>(code, ex);
            if (MLM) {
                int64_t label = m.ignore;
                if (res) {
                    const uint64_t u = pick4(mlm_block(g, static_cast<uint32_t>(j) >> 2, 1u, m), static_cast<uint32_t>(j) & 3u);
                    if (u < m.ts) {
                        label = code;
                        if (u < m.tm) val = static_cast<T>(m.mask_id);
                        else if (u < m.tr) val = static_cast<T>(static_cast<int32_t>(mlm_random_id(g, static_cast<uint32_t>(j), m)));
                    }
                }
                lab[f] = label;
            }
            out[f] = val;
            pos[f] = c;
        }
    }
}

template <typename T, bool MLM>
__global__ void __launch_bounds__(kPThreads, MLM ? 2 : 4)
seqpack_kernel(const uint8_t *__restrict__ bytes, const int64_t *__restrict__ offs, const int64_t *__restrict__ row_ptr,
               const int64_t *__restrict__ row_seq, int64_t nrows, int L, LutParam lutp, Specials sp, Expand ex, MlmParam m,
               T *__restrict__ out, int32_t *__restrict__ pos, int64_t *__restrict__ lab) {
    __shared__ __align__(16) uint8_t lut[256];
    load_lut(lut, lutp);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t r = static_cast<int64_t>(blockIdx.x) * (kPThreads / 32) + (threadIdx.x >> 5);
    if (r >= nrows) return;
    const int k = sp.bos + sp.eos;
    const int64_t rb = r * L;
    const int64_t p1 = __ldg(row_ptr + r + 1);
    int col = 0;
    // the row's sequences, then (p == p1) its padding run, through one copy of the segment code
    for (int64_t p = __ldg(row_ptr + r);; ++p) {
        const uint8_t *src = nullptr;
        int len = 0, w = L - col;
        int64_t s = 0;
        if (p < p1) {
            s = __ldg(row_seq + p);
            const int64_t st = __ldg(offs + s);
            len = static_cast<int>(__ldg(offs + s + 1) - st);
            src = bytes + st;
            w = len + k;
        } else if (w == 0) {
            break;
        }
        sp_segment<T, MLM>(rb + col, w, p < p1, src, len, static_cast<uint64_t>(m.base + s), sp, lut, ex, m, out, pos, lab, lane);
        if (p >= p1) break;
        col += w;
    }
}

template <typename T>
int launch_seqpack(cudaStream_t st, const uint8_t *d_bytes, const int64_t *d_offs, const int64_t *d_row_ptr, const int64_t *d_row_seq,
                   int64_t nrows, int64_t L, const bsq_tokenizer &tok, const MlmParam *m, void *d_out, int32_t *d_pos, int64_t *d_lab) {
    const Prepared p = prepare(tok, sizeof(T) == 1 ? 0 : 1);
    const int64_t rows_per_cta = kPThreads / 32;
    const unsigned grid = static_cast<unsigned>((nrows + rows_per_cta - 1) / rows_per_cta);
    if (m != nullptr) {
        seqpack_kernel<T, true><<<grid, kPThreads, 0, st>>>(d_bytes, d_offs, d_row_ptr, d_row_seq, nrows, static_cast<int>(L), p.lut,
                                                          p.sp, p.ex, *m, static_cast<T *>(d_out), d_pos, d_lab);
    } else {
        MlmParam none{};
        seqpack_kernel<T, false><<<grid, kPThreads, 0, st>>>(d_bytes, d_offs, d_row_ptr, d_row_seq, nrows, static_cast<int>(L), p.lut,
                                                           p.sp, p.ex, none, static_cast<T *>(d_out), d_pos, nullptr);
    }
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}

int seqpack_entry(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, const bsq_tokenizer *tok, int kind,
                  int64_t row_len, int64_t nrows, const int64_t *d_row_ptr, const int64_t *d_row_seq, const MlmParam *m,
                  void *d_tokens, int32_t *d_position_ids, int64_t *d_labels) {
    if (tok == nullptr) return fail(BSQ_ERR_ARG, "null tokenizer");
    if (bsq_kind_size(kind) == 0) return fail(BSQ_ERR_ARG, "invalid element kind");
    if (row_len < 1 || nrows < 0) return fail(BSQ_ERR_ARG, "row_len must be >= 1 and nrows >= 0");
    if (nrows > 0 && nrows > 0x7fffffffll / row_len) return fail(BSQ_ERR_ARG, "nrows * row_len exceeds 2^31 - 1");
    if (nrows == 0) return BSQ_OK;
    if (d_row_ptr == nullptr) return fail(BSQ_ERR_ARG, "null row_ptr");  // (bytes, offsets, row_seq: only read for placed sequences)
    const auto misaligned = [](const void *q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15u) != 0; };
    if (misaligned(d_tokens) || misaligned(d_position_ids) || (m != nullptr && misaligned(d_labels)))
        return fail(BSQ_ERR_ARG, "tokens, position_ids and labels pointers must be non-null and 16-byte aligned");
    BSQ_CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (kind) {
        case BSQ_I8: return launch_seqpack<int8_t>(st, d_bytes, d_offsets, d_row_ptr, d_row_seq, nrows, row_len, *tok, m, d_tokens, d_position_ids, d_labels);
        case BSQ_I16: return launch_seqpack<int16_t>(st, d_bytes, d_offsets, d_row_ptr, d_row_seq, nrows, row_len, *tok, m, d_tokens, d_position_ids, d_labels);
        case BSQ_I32: return launch_seqpack<int32_t>(st, d_bytes, d_offsets, d_row_ptr, d_row_seq, nrows, row_len, *tok, m, d_tokens, d_position_ids, d_labels);
        case BSQ_I64: return launch_seqpack<int64_t>(st, d_bytes, d_offsets, d_row_ptr, d_row_seq, nrows, row_len, *tok, m, d_tokens, d_position_ids, d_labels);
        case BSQ_F32: return launch_seqpack<float>(st, d_bytes, d_offsets, d_row_ptr, d_row_seq, nrows, row_len, *tok, m, d_tokens, d_position_ids, d_labels);
        default: return launch_seqpack<double>(st, d_bytes, d_offsets, d_row_ptr, d_row_seq, nrows, row_len, *tok, m, d_tokens, d_position_ids, d_labels);
    }
}

}  // namespace

}  // namespace bsq

extern "C" int bsq_tokenize_seqpack(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, const bsq_tokenizer *tok,
                                    int kind, int64_t row_len, int64_t nrows, const int64_t *d_row_ptr, const int64_t *d_row_seq,
                                    void *d_tokens, int32_t *d_position_ids) {
    bsq::DeviceRestore restore_device;
    return seqpack_entry(device, stream, d_bytes, d_offsets, tok, kind, row_len, nrows, d_row_ptr, d_row_seq, nullptr, d_tokens,
                         d_position_ids, nullptr);
}

extern "C" int bsq_tokenize_seqpack_mlm(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets,
                                        const bsq_tokenizer *tok, int kind, const bsq_mlm *mlm, int64_t row_len, int64_t nrows,
                                        const int64_t *d_row_ptr, const int64_t *d_row_seq, void *d_inputs, int32_t *d_position_ids,
                                        int64_t *d_labels) {
    bsq::DeviceRestore restore_device;
    MlmParam m;
    if (int rc = check_mlm_param(tok, kind, mlm, &m)) return rc;
    return seqpack_entry(device, stream, d_bytes, d_offsets, tok, kind, row_len, nrows, d_row_ptr, d_row_seq, &m, d_inputs,
                         d_position_ids, d_labels);
}
