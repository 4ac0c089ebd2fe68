// Consumers fused onto the tokeniser, and the on-device augmentation that precedes it
// (SURVEY.md section 8(f) rows 3 and 4).  Elementwise byte maps like the rest of libbsq:
// HBM-write-bound, no tensor cores.
//
//   K5  onehot_bcl_kernel   one-hot emitted directly in the (batch, channel, length) layout the
//       reference's CNN path builds with two extra full-tensor passes: batch_onehot_encode ->
//       einops.rearrange("length batch emb -> batch emb length") -> .float()
//       (bioseq/loaders.py:74-75, :93-94).
//   K6  embed_kernel        tokenize -> nn.Embedding row gather in one pass: the (B,P) / (P,B)
//       token tensor is never materialised (bioseq/__init__.py:171-188 make_embedding and its
//       callers, e.g. bioseq/decoders.py SeqEncoder: embedding(tokens)).
//   K7  augment_kernel      BLOSUM62 point mutations of the packed residues on the device before
//       they are tokenised (bioseq/blosum.py:36-87 substitute/augment_seq, applied per sequence
//       by FlatFileDataset, bioseq/loaders.py:71-73, :99-100), Philox4x32-10 counter-based so
//       that the result depends only on (seed, sequence index).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>

#include "bsq_internal.h"
#include "bsq_kernels.cuh"

namespace bsq {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

__device__ __forceinline__ void stcs16(void *p, const uint4 &v) { __stcs(reinterpret_cast<uint4 *>(p), v); }

// Codes of columns c0..c0+15 of one row, pad vector beyond the row's last symbol.
__device__ __forceinline__ uint4 row_codes16(const RowSrc &rs, const RowSrc *ms, int len, int c0, const Specials &sp,
                                             const uint8_t *lut, const TailTab &tab) {
    if (c0 >= sp.bos + len + sp.eos) return make_uint4(sp.pad_w, sp.pad_w, sp.pad_w, sp.pad_w);
    return tokens16<false>(rs, ms, len, c0, sp, lut, tab);
}

// ---------------------------------------------------------------------------------------
// K5: one-hot, (B, C, L) layout
// ---------------------------------------------------------------------------------------
// S = element size; a 16-byte vector holds V = 16 / S consecutive positions of one channel.
// `code` bytes are compared with channel c; WIDE routes codes >= 0x80 through Expand (ids that do
// not fit a byte and the "leave zero" sentinel), otherwise the byte compare is exact because
// channel numbers stay below 0x80 and every code >= 0x80 is the sentinel.
template <bool WIDE>
__device__ __forceinline__ bool code_is(uint32_t code, int c, const Expand &ex) {
    if (WIDE) return expand_code(code, ex) == c;
    return code == static_cast<uint32_t>(c);
}

// Build the 16-byte vector for V codes held in the low V bytes of (w0, w1, w2, w3).
template <int S, bool WIDE>
__device__ __forceinline__ uint4 match_vec(const uint32_t w[4], int c, uint32_t one_lo, uint32_t one_hi, const Expand &ex) {
    uint4 r;
    if (S == 1) {
        if (!WIDE) {
            const uint32_t cc = static_cast<uint32_t>(c) * 0x01010101u;
            r.x = __vcmpeq4(w[0], cc) & 0x01010101u; r.y = __vcmpeq4(w[1], cc) & 0x01010101u;
            r.z = __vcmpeq4(w[2], cc) & 0x01010101u; r.w = __vcmpeq4(w[3], cc) & 0x01010101u;
        } else {
            uint32_t o[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                o[k] = 0;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (code_is<true>((w[k] >> (8 * i)) & 0xffu, c, ex)) o[k] |= 1u << (8 * i);
            }
            r = make_uint4(o[0], o[1], o[2], o[3]);
        }
    } else if (S == 2) {  // 8 codes in w[0], w[1]
        uint32_t o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t src = w[k >> 1] >> (16 * (k & 1));
            o[k] = (code_is<WIDE>(src & 0xffu, c, ex) ? one_lo : 0u) | (code_is<WIDE>((src >> 8) & 0xffu, c, ex) ? one_lo << 16 : 0u);
        }
        r = make_uint4(o[0], o[1], o[2], o[3]);
    } else if (S == 4) {  // 4 codes in w[0]
        r.x = code_is<WIDE>(w[0] & 0xffu, c, ex) ? one_lo : 0u;
        r.y = code_is<WIDE>((w[0] >> 8) & 0xffu, c, ex) ? one_lo : 0u;
        r.z = code_is<WIDE>((w[0] >> 16) & 0xffu, c, ex) ? one_lo : 0u;
        r.w = code_is<WIDE>(w[0] >> 24, c, ex) ? one_lo : 0u;
    } else {  // S == 8: 2 codes in the low half of w[0]
        const bool a = code_is<WIDE>(w[0] & 0xffu, c, ex), b = code_is<WIDE>((w[0] >> 8) & 0xffu, c, ex);
        r.x = a ? one_lo : 0u; r.y = a ? one_hi : 0u;
        r.z = b ? one_lo : 0u; r.w = b ? one_hi : 0u;
    }
    return r;
}

// One warp per (sequence, 512-position span).  The 16 codes each lane computes go through a
// 512-byte per-warp stage so that in the store loop lane l owns the V positions l*V.. of every
// 32*V-position group: each store instruction writes 512 contiguous bytes of one channel row.
template <int S, bool WIDE>
__global__ void __launch_bounds__(kThreads)
onehot_bcl_kernel(SeqView v, int64_t nseq, int padlen, int ncols, LutParam lutp, Specials sp, Expand ex, uint32_t one_lo,
                  uint32_t one_hi, uint8_t *__restrict__ out) {
    constexpr int V = 16 / S;          // positions per 16-byte vector
    constexpr int NIT = S;             // 512 / (32 * V) store groups per span
    __shared__ __align__(16) uint8_t lut[256];
    __shared__ TailTab tab;
    __shared__ __align__(16) uint8_t stage[kWarps][512];
    load_lut(lut, lutp);
    init_tailtab(tab, sp);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int spans = (padlen + 511) >> 9;
    const int64_t items = nseq * spans;
    for (int64_t it = static_cast<int64_t>(blockIdx.x) * kWarps + warp; it < items; it += static_cast<int64_t>(gridDim.x) * kWarps) {
        const int64_t b = it / spans;
        const int p0 = static_cast<int>(it - b * spans) << 9;
        const int64_t start = __ldg(v.offs + b);
        const int len = static_cast<int>(__ldg(v.offs + b + 1) - start);
        const RowSrc rs = make_rowsrc(v.bytes, start, sp.bos, len);
        RowSrc msrc;
        const RowSrc *ms = nullptr;
        if (v.mask != nullptr) {
            msrc = make_rowsrc(v.mask, start, sp.bos, len);
            ms = &msrc;
        }
        const int c0 = p0 + lane * 16;
        uint4 codes = make_uint4(0u, 0u, 0u, 0u);
        if (c0 < padlen) codes = row_codes16(rs, ms, len, c0, sp, lut, tab);
        *reinterpret_cast<uint4 *>(&stage[warp][lane * 16]) = codes;
        __syncwarp();
        // this lane's codes for store group j: bytes [j*32*V + lane*V, +V) of the stage
        uint32_t w[NIT][4];
#pragma unroll
        for (int j = 0; j < NIT; ++j) {
            const uint8_t *src = &stage[warp][j * 32 * V + lane * V];
            w[j][0] = w[j][1] = w[j][2] = w[j][3] = 0u;
            if (V == 16) {
                const uint4 t = *reinterpret_cast<const uint4 *>(src);
                w[j][0] = t.x; w[j][1] = t.y; w[j][2] = t.z; w[j][3] = t.w;
            } else if (V == 8) {
                const uint2 t = *reinterpret_cast<const uint2 *>(src);
                w[j][0] = t.x; w[j][1] = t.y;
            } else if (V == 4) {
                w[j][0] = *reinterpret_cast<const uint32_t *>(src);
            } else {
                w[j][0] = *reinterpret_cast<const uint16_t *>(src);
            }
        }
        __syncwarp();
        uint8_t *row = out + (static_cast<size_t>(b) * ncols * padlen + p0 + lane * V) * S;
        for (int c = 0; c < ncols; ++c) {
#pragma unroll
            for (int j = 0; j < NIT; ++j) {
                if (p0 + j * 32 * V + lane * V < padlen) stcs16(row + static_cast<size_t>(j) * 32 * V * S, match_vec<S, WIDE>(w[j], c, one_lo, one_hi, ex));
            }
            row += static_cast<size_t>(padlen) * S;
        }
    }
}

// Any padlen / element size: one element per thread, coalesced along the length.
template <int S>
__global__ void __launch_bounds__(kThreads)
onehot_bcl_scalar_kernel(SeqView v, int64_t nseq, int padlen, int ncols, LutParam lutp, Specials sp, Expand ex, uint32_t one_lo,
                         uint32_t one_hi, uint8_t *__restrict__ out) {
    __shared__ __align__(16) uint8_t lut[256];
    load_lut(lut, lutp);
    __syncthreads();
    const int64_t total = nseq * ncols * static_cast<int64_t>(padlen);
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x; i < total; i += static_cast<int64_t>(gridDim.x) * kThreads) {
        const int pos = static_cast<int>(i % padlen);
        const int64_t bc = i / padlen;
        const int c = static_cast<int>(bc % ncols);
        const int64_t b = bc / ncols;
        const int64_t start = __ldg(v.offs + b);
        const int len = static_cast<int>(__ldg(v.offs + b + 1) - start);
        const bool hit = expand_code(token_at(v, start, len, pos, sp, lut), ex) == c;
        uint8_t *dst = out + static_cast<size_t>(i) * S;
        if (S == 1) *dst = hit ? static_cast<uint8_t>(one_lo) : 0;
        else if (S == 2) *reinterpret_cast<uint16_t *>(dst) = hit ? static_cast<uint16_t>(one_lo) : 0;
        else if (S == 4) *reinterpret_cast<uint32_t *>(dst) = hit ? one_lo : 0u;
        else *reinterpret_cast<uint2 *>(dst) = hit ? make_uint2(one_lo, one_hi) : make_uint2(0u, 0u);
    }
}

// ---------------------------------------------------------------------------------------
// K6: tokenize -> embedding rows
// ---------------------------------------------------------------------------------------
constexpr int kETileSeqs = 32;
constexpr int kETilePos = 128;
constexpr int kEPitch = kETilePos + 16;

// A CTA takes a 32-sequence x 128-position tile: phase 1 computes the tile's codes (each thread one
// 16-column chunk, 8 threads reading 128 consecutive residues of a sequence), phase 2 streams the
// embedding rows out: the flat index over (token, 16-byte vector of the row) is contiguous in the
// output for 128 tokens of a sequence (batch-first) or 32 sequences of a position (seq-first), so
// every store instruction writes 512 contiguous bytes.  The table lives in shared memory when it
// fits (TABLE_SMEM), else it is read through L1/L2 (it is a few hundred KB at most and hot).
template <bool SEQ_FIRST, bool TABLE_SMEM>
__global__ void __launch_bounds__(kThreads)
embed_kernel(SeqView v, int64_t nseq, int64_t ld, int padlen, LutParam lutp, Specials sp, Expand ex,
             const uint4 *__restrict__ weight, int nrows, FastDiv rv, int tiles_pos, int64_t ntiles, uint4 *__restrict__ out) {
    extern __shared__ __align__(16) uint8_t dyn[];
    __shared__ __align__(16) uint8_t lut[256];
    __shared__ TailTab tab;
    __shared__ __align__(16) uint8_t codes[kETileSeqs][kEPitch];
    const int row_vecs = static_cast<int>(rv.d);
    uint4 *table = reinterpret_cast<uint4 *>(dyn);
    load_lut(lut, lutp);
    init_tailtab(tab, sp);
    if (TABLE_SMEM)
        for (int i = threadIdx.x; i < nrows * row_vecs; i += kThreads) table[i] = __ldg(weight + i);
    __syncthreads();
    const int s1 = threadIdx.x >> 3, ch = threadIdx.x & 7;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t tb = tile / tiles_pos;
        const int p0 = static_cast<int>(tile - tb * tiles_pos) * kETilePos;
        const int64_t b0 = tb * kETileSeqs;
        const int nb = static_cast<int>(min(static_cast<int64_t>(kETileSeqs), nseq - b0));
        const int np = min(kETilePos, padlen - p0);
        {
            const int c0 = p0 + ch * 16;
            if (s1 < nb && c0 < padlen) {
                const int64_t start = __ldg(v.offs + b0 + s1);
                const int len = static_cast<int>(__ldg(v.offs + b0 + s1 + 1) - start);
                const RowSrc rs = make_rowsrc(v.bytes, start, sp.bos, len);
                *reinterpret_cast<uint4 *>(&codes[s1][ch * 16]) = row_codes16(rs, nullptr, len, c0, sp, lut, tab);
            }
        }
        __syncthreads();
        const uint32_t total = static_cast<uint32_t>(nb) * np * row_vecs;
        const FastDiv inner = make_fastdiv(SEQ_FIRST ? nb : np);
        for (uint32_t idx = threadIdx.x; idx < total; idx += kThreads) {
            const uint32_t k = fd_div(idx, rv), vec = idx - k * row_vecs;
            const uint32_t hi = fd_div(k, inner), lo = k - hi * inner.d;
            const uint32_t s = SEQ_FIRST ? lo : hi, p = SEQ_FIRST ? hi : lo;
            const int id = expand_code(codes[s][p], ex);
            const uint4 val = TABLE_SMEM ? table[id * row_vecs + vec] : __ldg(weight + static_cast<size_t>(id) * row_vecs + vec);
            const size_t orow = SEQ_FIRST ? static_cast<size_t>(p0 + p) * ld + b0 + s : static_cast<size_t>(b0 + s) * padlen + p0 + p;
            __stcs(out + orow * row_vecs + vec, val);
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------
// K7: BLOSUM62 point mutations (Philox4x32-10)
// ---------------------------------------------------------------------------------------
// BLOSUM62 log-odds scores (NCBI), rows and columns in the order ARNDCQEGHILKMFPSTWYV, plus the
// row of X (unknown residue) -- the 21 x 20 block the reference selects (bioseq/blosum.py:36-40).
constexpr char kAA[21] = "ARNDCQEGHILKMFPSTWYV";
constexpr int8_t kBlosum62[21][20] = {
    /*A*/ {4, -1, -2, -2, 0, -1, -1, 0, -2, -1, -1, -1, -1, -2, -1, 1, 0, -3, -2, 0},
    /*R*/ {-1, 5, 0, -2, -3, 1, 0, -2, 0, -3, -2, 2, -1, -3, -2, -1, -1, -3, -2, -3},
    /*N*/ {-2, 0, 6, 1, -3, 0, 0, 0, 1, -3, -3, 0, -2, -3, -2, 1, 0, -4, -2, -3},
    /*D*/ {-2, -2, 1, 6, -3, 0, 2, -1, -1, -3, -4, -1, -3, -3, -1, 0, -1, -4, -3, -3},
    /*C*/ {0, -3, -3, -3, 9, -3, -4, -3, -3, -1, -1, -3, -1, -2, -3, -1, -1, -2, -2, -1},
    /*Q*/ {-1, 1, 0, 0, -3, 5, 2, -2, 0, -3, -2, 1, 0, -3, -1, 0, -1, -2, -1, -2},
    /*E*/ {-1, 0, 0, 2, -4, 2, 5, -2, 0, -3, -3, 1, -2, -3, -1, 0, -1, -3, -2, -2},
    /*G*/ {0, -2, 0, -1, -3, -2, -2, 6, -2, -4, -4, -2, -3, -3, -2, 0, -2, -2, -3, -3},
    /*H*/ {-2, 0, 1, -1, -3, 0, 0, -2, 8, -3, -3, -1, -2, -1, -2, -1, -2, -2, 2, -3},
    /*I*/ {-1, -3, -3, -3, -1, -3, -3, -4, -3, 4, 2, -3, 1, 0, -3, -2, -1, -3, -1, 3},
    /*L*/ {-1, -2, -3, -4, -1, -2, -3, -4, -3, 2, 4, -2, 2, 0, -3, -2, -1, -2, -1, 1},
    /*K*/ {-1, 2, 0, -1, -3, 1, 1, -2, -1, -3, -2, 5, -1, -3, -1, 0, -1, -3, -2, -2},
    /*M*/ {-1, -1, -2, -3, -1, 0, -2, -3, -2, 1, 2, -1, 5, 0, -2, -1, -1, -1, -1, 1},
    /*F*/ {-2, -3, -3, -3, -2, -3, -3, -3, -1, 0, 0, -3, 0, 6, -4, -2, -2, 1, 3, -1},
    /*P*/ {-1, -2, -2, -1, -3, -1, -1, -2, -2, -3, -3, -1, -2, -4, 7, -1, -1, -4, -3, -2},
    /*S*/ {1, -1, 1, 0, -1, 0, 0, 0, -1, -2, -2, 0, -1, -2, -1, 4, 1, -3, -2, -2},
    /*T*/ {0, -1, 0, -1, -1, -1, -1, -2, -2, -1, -1, -1, -1, -2, -1, 1, 5, -2, -2, 0},
    /*W*/ {-3, -3, -4, -4, -2, -2, -3, -2, -2, -3, -2, -3, -1, 1, -4, -3, -2, 11, 2, -3},
    /*Y*/ {-2, -2, -2, -3, -2, -1, -2, -3, 2, -1, -1, -2, -1, 3, -3, -2, -2, 2, 7, -1},
    /*V*/ {0, -3, -3, -3, -1, -2, -2, -3, -3, 3, 1, -2, 1, -1, -2, -2, 0, -3, -1, 4},
    /*X*/ {0, -1, -1, -1, -2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -2, 0, 0, -2, -1, -1},
};

// Substitution table in integer form.  probability(row -> j) = 2^score / sum_j 2^score
// (bioseq/blosum.py:41-43); thr[row][j] = floor(2^32 * cumulative probability through j) for
// j = 0..18 (the 20th cumulative value is 2^32).  A 32-bit uniform r selects the number of
// thresholds that are <= r.  Exact integer arithmetic: 2^(score+4) are integers.
struct BlosumTab {
    uint32_t thr[21][19];
    uint8_t row_of[256];  // residue byte -> row (20 = X for anything that is not an upper-case amino acid)
    uint8_t aa[20];
};

const BlosumTab &blosum_tab() {
    static const BlosumTab t = [] {
        BlosumTab b;
        for (int r = 0; r < 21; ++r) {
            uint64_t sum = 0;
            for (int j = 0; j < 20; ++j) sum += 1ull << (kBlosum62[r][j] + 4);
            uint64_t cum = 0;
            for (int j = 0; j < 19; ++j) {
                cum += 1ull << (kBlosum62[r][j] + 4);
                b.thr[r][j] = static_cast<uint32_t>((cum << 32) / sum);
            }
        }
        std::memset(b.row_of, 20, sizeof(b.row_of));
        for (int j = 0; j < 20; ++j) {
            b.row_of[static_cast<uint8_t>(kAA[j])] = static_cast<uint8_t>(j);
            b.aa[j] = static_cast<uint8_t>(kAA[j]);
        }
        return b;
    }();
    return t;
}

constexpr int kMaxTries = 4096;  // the reference retries until the substitution differs (blosum.py:79-82)

// One thread per sequence.  Counter = (sequence index lo, hi, block number, 0), key = seed.
// Block 0, word 0 gates the sequence (applied iff word < gate, gate = floor(augment_frac * 2^32), or
// always when augment_frac >= 1).  Blocks 1, 2, ... feed the tries, two per block: (position word,
// substitution word).  position = mulhi(word, len); substitution = #thresholds <= word.
__global__ void __launch_bounds__(kThreads)
augment_kernel(uint8_t *__restrict__ bytes, const int64_t *__restrict__ offs, int64_t nseq, int chain_len, uint64_t gate,
               uint32_t k0, uint32_t k1, int64_t seq_base, BlosumTab tabp) {
    __shared__ BlosumTab tab;
    for (int i = threadIdx.x; i < static_cast<int>(sizeof(BlosumTab) / 4); i += kThreads)
        reinterpret_cast<uint32_t *>(&tab)[i] = reinterpret_cast<const uint32_t *>(&tabp)[i];
    __syncthreads();
    const int64_t i = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x;
    if (i >= nseq) return;
    const int64_t start = offs[i];
    const uint64_t len64 = static_cast<uint64_t>(offs[i + 1] - start);
    if (len64 == 0) return;
    const uint32_t len = static_cast<uint32_t>(min(len64, static_cast<uint64_t>(0xffffffffu)));
    const uint64_t g = static_cast<uint64_t>(seq_base + i);
    const uint32_t g0 = static_cast<uint32_t>(g), g1 = static_cast<uint32_t>(g >> 32);
    if (gate < (1ull << 32)) {
        const Philox p = philox4x32_10(g0, g1, 0u, 0u, k0, k1);
        if (static_cast<uint64_t>(p.c[0]) >= gate) return;
    }
    uint8_t *seq = bytes + start;
    uint32_t blk = 1;
    for (int m = 0; m < chain_len; ++m) {
        bool done = false;
        for (int t = 0; t < kMaxTries && !done; t += 2) {
            const Philox p = philox4x32_10(g0, g1, blk++, 0u, k0, k1);
#pragma unroll
            for (int h = 0; h < 2 && !done; ++h) {
                const uint32_t idx = __umulhi(p.c[2 * h], len);
                const uint8_t cur = seq[idx];
                const uint32_t *thr = tab.thr[tab.row_of[cur]];
                const uint32_t r = p.c[2 * h + 1];
                int j = 0;
#pragma unroll
                for (int q = 0; q < 19; ++q) j += thr[q] <= r;
                const uint8_t sub = tab.aa[j];
                if (sub != cur) {
                    seq[idx] = sub;
                    done = true;
                }
            }
        }
    }
}

int grid_for(int64_t work_items, int per_cta, int ctas_per_sm) {
    const int64_t want = (work_items + per_cta - 1) / per_cta;
    return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(want, static_cast<int64_t>(cur_sms()) * ctas_per_sm)));
}

void one_pattern(int kind, uint32_t *lo, uint32_t *hi) {
    *lo = 1u;
    *hi = 0u;
    if (kind == BSQ_F32) *lo = 0x3f800000u;
    if (kind == BSQ_F64) {
        *lo = 0u;
        *hi = 0x3ff00000u;
    }
}

}  // namespace
}  // namespace bsq

using bsq::fail;

extern "C" {

int bsq_onehot_bcl(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, const uint8_t *d_mask,
                   int64_t nseq, int64_t padlen, const bsq_tokenizer *tok, int kind, void *d_out) {
    bsq::DeviceRestore restore_device;
    using namespace bsq;
    if (int rc = check_launch_args(device, nseq, padlen, tok, kind, d_out)) return rc;
    if (nseq == 0) return BSQ_OK;
    if (d_offsets == nullptr) return fail(BSQ_ERR_ARG, "null offsets");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Prepared p = prepare(*tok, 2);
    const SeqView v{d_bytes, d_offsets, d_mask};
    const int S = static_cast<int>(bsq_kind_size(kind));
    const int ncols = tok->alphabet_size;
    const bool wide = tok->pad_id >= 0x80;
    uint32_t lo, hi;
    one_pattern(kind, &lo, &hi);
    uint8_t *out = static_cast<uint8_t *>(d_out);
    const int P = static_cast<int>(padlen);
    if ((padlen * S) % 16 == 0) {
        const int64_t items = nseq * ((padlen + 511) / 512);
        const int grid = grid_for(items, kWarps, 8);
#define BSQ_BCL(SZ)                                                                                                      \
    do {                                                                                                                 \
        if (wide) onehot_bcl_kernel<SZ, true><<<grid, kThreads, 0, st>>>(v, nseq, P, ncols, p.lut, p.sp, p.ex, lo, hi, out); \
        else onehot_bcl_kernel<SZ, false><<<grid, kThreads, 0, st>>>(v, nseq, P, ncols, p.lut, p.sp, p.ex, lo, hi, out);   \
    } while (0)
        switch (S) {
            case 1: BSQ_BCL(1); break;
            case 2: BSQ_BCL(2); break;
            case 4: BSQ_BCL(4); break;
            default: BSQ_BCL(8); break;
        }
#undef BSQ_BCL
    } else {
        const int grid = grid_for(nseq * ncols * padlen, kThreads * 4, 8);
        switch (S) {
            case 1: onehot_bcl_scalar_kernel<1><<<grid, kThreads, 0, st>>>(v, nseq, P, ncols, p.lut, p.sp, p.ex, lo, hi, out); break;
            case 2: onehot_bcl_scalar_kernel<2><<<grid, kThreads, 0, st>>>(v, nseq, P, ncols, p.lut, p.sp, p.ex, lo, hi, out); break;
            case 4: onehot_bcl_scalar_kernel<4><<<grid, kThreads, 0, st>>>(v, nseq, P, ncols, p.lut, p.sp, p.ex, lo, hi, out); break;
            default: onehot_bcl_scalar_kernel<8><<<grid, kThreads, 0, st>>>(v, nseq, P, ncols, p.lut, p.sp, p.ex, lo, hi, out); break;
        }
    }
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}

int bsq_embed(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int64_t padlen,
              const bsq_tokenizer *tok, int batch_first, const void *d_weight, int64_t nrows, int64_t row_bytes, void *d_out) {
    bsq::DeviceRestore restore_device;
    using namespace bsq;
    if (int rc = check_launch_args(device, nseq, padlen, tok, BSQ_I8, d_out)) return rc;
    if (d_weight == nullptr || (reinterpret_cast<uintptr_t>(d_weight) & 15u))
        return fail(BSQ_ERR_ARG, "embedding table must be non-null and 16-byte aligned");
    if (row_bytes <= 0 || row_bytes % 16 != 0) return fail(BSQ_ERR_ARG, "embedding rows must be a multiple of 16 bytes");
    if (row_bytes / 16 > (1 << 18)) return fail(BSQ_ERR_ARG, "embedding rows above 4 MiB are not supported");
    if (nrows < tok->alphabet_size)
        return fail(BSQ_ERR_ARG, "embedding table has " + std::to_string(nrows) + " rows, the tokenizer's alphabet_size is " +
                                     std::to_string(tok->alphabet_size));
    if (nseq == 0) return BSQ_OK;
    if (d_offsets == nullptr) return fail(BSQ_ERR_ARG, "null offsets");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Prepared p = prepare(*tok, 1);
    const SeqView v{d_bytes, d_offsets, nullptr};
    const int P = static_cast<int>(padlen);
    const int tiles_pos = (P + kETilePos - 1) / kETilePos;
    const int64_t ntiles = ((nseq + kETileSeqs - 1) / kETileSeqs) * tiles_pos;
    const FastDiv rv = make_fastdiv(static_cast<uint32_t>(row_bytes / 16));
    // rows the kernel can index: every id of the tokenizer (alphabet_size covers bos/eos/pad when present;
    // pad_id is also the fill of an unpadded tokenizer's tail when padchar is off -> code 0 there)
    const int used_rows = tok->alphabet_size;
    const size_t table_bytes = static_cast<size_t>(used_rows) * row_bytes;
    const bool in_smem = table_bytes <= (96u << 10);
    const int grid = static_cast<int>(std::min<int64_t>(ntiles, static_cast<int64_t>(cur_sms()) * (in_smem && table_bytes > (40u << 10) ? 2 : 4)));
    const uint4 *w = static_cast<const uint4 *>(d_weight);
    uint4 *out = static_cast<uint4 *>(d_out);
#define BSQ_EMB(SF, TS)                                                                                              \
    do {                                                                                                             \
        const size_t dyn = TS ? table_bytes : 0;                                                                     \
        if (dyn > (40u << 10))                                                                                       \
            BSQ_CUDA_TRY(cudaFuncSetAttribute(embed_kernel<SF, TS>, cudaFuncAttributeMaxDynamicSharedMemorySize,   \
                                              static_cast<int>(dyn)));                                              \
        embed_kernel<SF, TS><<<grid, kThreads, dyn, st>>>(v, nseq, nseq, P, p.lut, p.sp, p.ex, w, used_rows, rv, tiles_pos, \
                                                          ntiles, out);                                              \
    } while (0)
    if (batch_first) {
        if (in_smem) BSQ_EMB(false, true);
        else BSQ_EMB(false, false);
    } else {
        if (in_smem) BSQ_EMB(true, true);
        else BSQ_EMB(true, false);
    }
#undef BSQ_EMB
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}

int bsq_blosum62_thresholds(uint32_t *out, uint8_t *row_of, uint8_t *aa) {
    const bsq::BlosumTab &t = bsq::blosum_tab();
    if (out) std::memcpy(out, t.thr, sizeof(t.thr));
    if (row_of) std::memcpy(row_of, t.row_of, sizeof(t.row_of));
    if (aa) std::memcpy(aa, t.aa, sizeof(t.aa));
    return BSQ_OK;
}

int bsq_augment_blosum62(int device, void *stream, uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int chain_len,
                         double augment_frac, uint64_t seed, int64_t seq_index_base) {
    bsq::DeviceRestore restore_device;
    using namespace bsq;
    if (nseq < 0 || chain_len < 0) return fail(BSQ_ERR_ARG, "negative count");
    if (!(augment_frac >= 0.0)) return fail(BSQ_ERR_ARG, "augment_frac must be >= 0");
    if (nseq == 0 || chain_len == 0 || augment_frac == 0.0) return BSQ_OK;
    if (d_bytes == nullptr || d_offsets == nullptr) return fail(BSQ_ERR_ARG, "null argument");
    BSQ_CUDA_TRY(cudaSetDevice(device));
    const uint64_t gate = augment_frac >= 1.0 ? (1ull << 32) : static_cast<uint64_t>(std::floor(augment_frac * 4294967296.0));
    const int grid = static_cast<int>((nseq + kThreads - 1) / kThreads);
    augment_kernel<<<grid, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        d_bytes, d_offsets, nseq, chain_len, gate, static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), seq_index_base,
        blosum_tab());
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}

}  // extern "C"
