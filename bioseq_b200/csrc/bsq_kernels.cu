// sm_100a kernels + launchers for batch_tokenize / batch_onehot_encode / decode_tokens.
//
//   K1 tokenize_rows_kernel (nseq, padlen) batch-first tokens.  One warp per row, one lane =
//                           16 output bytes = one st.global.v4 per iteration; BOS/EOS/PAD fused;
//                           ragged tails skip all loads.
//   K2 seqfirst_kernel<..,kTokGeneric>  (padlen, nseq) tokens of any element type: 128 seq x 128 pos
//                           shared-memory tile, coalesced reads along each sequence, one element per
//                           lane along the batch.
//   K3 seqfirst_kernel<..,kOneHot> (padlen, nseq, C) one-hot: same tile, then every (pos, seq)
//                           row is written with one 4/8/16-byte store when C*sizeof(T) allows,
//                           else the run is zero-filled with 16-byte stores and the ones are
//                           scattered after a barrier (no separate memset pass).
//   K2t seqfirst_tok8_kernel  the instruction-lean form of K2 for one-byte tokens (what batch_first=False runs).
//   K4 decode_*             tokens -> characters: pass 1 decode_len16p_kernel (lengths, validation, where each row's
//                           trailing <PAD> run starts) + scan, pass 2 decode_chars_kernel (text); bsq_decode_text
//                           enqueues both behind one another.
//   K0 offsets_extent_kernel<CropCount>  length and offsets validation for device-resident packed input, and the crop's
//                           and varlen's extents (the template and its launcher are in bsq_kernels.cuh).
//   (K1s, the batch-first one-byte kernel for padlen >= 257 -- the headline path -- lives in bsq_span.cu.)
//
// Reference semantics: src/tokenize.h:381-485 (K1/K2), :283-371 (K3), :131-179 (K4).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <mutex>
#include <string>

#include "bsq_internal.h"
#include "bsq_kernels.cuh"

namespace bsq {

constexpr int kThreads = 256;
constexpr int kTileSeqs = 128;
constexpr int kTilePos = 128;
constexpr int kTilePitch = kTilePos + 4;  // 33 words: conflict-free column reads

template <typename T>
__device__ __forceinline__ T cast_id(int32_t v) {
    return static_cast<T>(v);
}

// ------------------------------------------------------------------------------------------
// K1: batch-first tokens, one warp per row (or per group of rows when padlen < 512).
//
// Lane `sub` of a row owns the 16-byte output chunks sub, sub+L, sub+2L, ... of that row
// (L = lanes per row), so a warp streams 512 contiguous output bytes per iteration.  All
// per-row state -- offsets, length, source alignment -- is loaded/derived once per row and is
// warp-uniform when L = 32, which keeps the realignment switch and the pad-only shortcut
// free of divergence.  Chunks are aligned to 16 bytes in the *flat* output, so rows whose
// padlen is not a multiple of 16 still use vector stores; only the (at most two) partial
// chunks at the ends of such a row fall back to byte stores.
//
// Element types wider than a byte go through a per-warp 512-byte shared-memory stage so that
// every st.global.v4 of the expanded values is contiguous across the warp.
// ------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ uint4 expand_vec(const uint8_t *codes, const Expand &ex) {
    constexpr int EPV = 16 / sizeof(T);
    T vals[EPV];
#pragma unroll
    for (int j = 0; j < EPV; ++j) vals[j] = cast_id<T>(expand_code(codes[j], ex));
    return *reinterpret_cast<const uint4 *>(vals);
}

// ROWWARP: a whole warp works on one row (padlen > 256): the row index is warp-uniform, and the
//          row's offsets are broadcast from lane 0 so that the per-row arithmetic can live in the
//          uniform datapath.  Otherwise 32 >> lanes_log2 rows share a warp.
// ALIGNED: padlen % 16 == 0, i.e. every row starts 16-byte aligned in the output and has no
//          partial chunk (always true for the wide element types handled here).
struct RowInfo {  // what a warp needs to know about its row, published through shared memory
    const uint8_t *al;
    int off, len;
};

template <typename T, bool ROWWARP, bool ALIGNED>
__global__ void __launch_bounds__(kThreads)
tokenize_rows_kernel(SeqView v, int64_t nseq, int padlen, int lanes_log2, LutParam lutp, Specials sp, Expand ex,
                     T *__restrict__ out) {
    constexpr int S = sizeof(T);
    constexpr int WARPS = kThreads / 32;
    __shared__ __align__(16) uint8_t lut[256];
    __shared__ TailTab tab;
    __shared__ __align__(16) RowInfo rinfo[WARPS];
    __shared__ __align__(16) uint8_t stage[S == 1 ? 16 : WARPS * 512];
    load_lut(lut, lutp);    // threads 0..63
    init_tailtab(tab, sp);  // threads 64..80
    if (ROWWARP && threadIdx.x >= 96 && threadIdx.x < 96 + WARPS) {
        // one thread per row of this CTA resolves the row's offsets and source alignment, so the
        // 8 warps do not each repeat that (dependent-load + 64-bit) arithmetic in all 32 lanes
        const int w = threadIdx.x - 96;
        const int64_t row = static_cast<int64_t>(blockIdx.x) * WARPS + w;
        if (row < nseq) {
            const int64_t start = __ldg(v.offs + row);
            const int len = static_cast<int>(__ldg(v.offs + row + 1) - start);
            const RowSrc r0 = make_rowsrc(v.bytes, start, sp.bos, len);
            rinfo[w].al = r0.al;
            rinfo[w].off = r0.off;
            rinfo[w].len = len;
        }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);  // tell the compiler it is uniform
    if (ROWWARP) lanes_log2 = 5;
    const int L = 1 << lanes_log2;
    const int64_t row0 = (static_cast<int64_t>(blockIdx.x) * WARPS + warp) * (32 >> lanes_log2);
    const int64_t row = ROWWARP ? row0 : row0 + (lane >> lanes_log2);
    const int sub = lane & (L - 1);
    const bool row_ok = row < nseq;
    RowSrc rs;
    int len = 0;
    if (ROWWARP) {
        if (!row_ok) return;  // whole warp
        const RowInfo ri = rinfo[warp];
        len = ri.len;
        rs.al = ri.al;
        rs.off = ri.off;
        rs.fw = (ri.off + sp.bos) & ~15;
        rs.lw = (ri.off + sp.bos + len - 1) & ~15;
    } else {
        int64_t start = 0;
        if (row_ok) {
            start = __ldg(v.offs + row);
            len = static_cast<int>(__ldg(v.offs + row + 1) - start);
        }
        rs = make_rowsrc(v.bytes, start, sp.bos, len);
    }
    const int npos = sp.bos + len + sp.eos;
    const int64_t rowbase = row * padlen;  // flat element index of column 0
    const uint4 padv = make_uint4(sp.pad_w, sp.pad_w, sp.pad_w, sp.pad_w);

    if (S == 1) {
        const int r = ALIGNED ? 0 : static_cast<int>(rowbase & 15);  // misalignment of the row in the flat output
        if (!row_ok) return;
        uint8_t *orow = reinterpret_cast<uint8_t *>(out) + rowbase;
        auto store = [&](int c0, const uint4 &codes) {
            if (ALIGNED || (c0 >= 0 && c0 + 16 <= padlen)) {
                __stcs(reinterpret_cast<uint4 *>(orow + c0), codes);
            } else {  // partial chunk at either end of an unaligned row
                const uint32_t w[4] = {codes.x, codes.y, codes.z, codes.w};
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (c0 + j >= 0 && c0 + j < padlen) orow[c0 + j] = static_cast<uint8_t>(w[j >> 2] >> (8 * (j & 3)));
            }
        };
        // two chunks (16*L columns apart) per iteration: both chunks' loads are in flight before
        // either is translated
        for (int c0 = 16 * sub - r; c0 < padlen; c0 += 32 * L) {
            const int c1 = c0 + 16 * L;
            const bool ld0 = c0 < npos && has_residues(c0, sp.bos, len);
            const bool ld1 = c1 < padlen && c1 < npos && has_residues(c1, sp.bos, len);
            Fetched f0, f1;
            if (ld0) f0 = fetch_issue(rs, c0);
            if (ld1) f1 = fetch_issue(rs, c1);
            store(c0, c0 >= npos ? padv : tokens16_from<!ALIGNED>(f0, ld0, rs, len, c0, sp, lut, tab));
            if (c1 < padlen) store(c1, c1 >= npos ? padv : tokens16_from<!ALIGNED>(f1, ld1, rs, len, c1, sp, lut, tab));
        }
    } else {
        // rows are 16-byte aligned here (the host checked padlen * sizeof(T) % 16 == 0)
        constexpr int EPV = 16 / S;
        uint8_t *wstage = stage + warp * 512;
        for (int cb = 0; cb < padlen; cb += 16 * L) {  // warp-uniform trip count
            const int c0 = cb + 16 * sub;
            uint4 codes = padv;
            if (row_ok && c0 < padlen && c0 < npos) codes = tokens16<false>(rs, nullptr, len, c0, sp, lut, tab);
            *reinterpret_cast<uint4 *>(wstage + 16 * lane) = codes;
            __syncwarp();
#pragma unroll
            for (int q = 0; q < S; ++q) {
                const int e = EPV * (lane + 32 * q);  // first of this lane's EPV codes within the 512 staged
                const int src_lane = e >> 4;
                const int64_t srow = row0 + (src_lane >> lanes_log2);
                const int scol = cb + 16 * (src_lane & (L - 1)) + (e & 15);
                if (srow < nseq && scol < padlen)
                    __stcs(reinterpret_cast<uint4 *>(out + srow * padlen + scol), expand_vec<T>(wstage + e, ex));
            }
            __syncwarp();
        }
    }
}

// ---- PTX helpers: mbarrier + 1-D bulk asynchronous copy (TMA unit, SASS UBLKCP) ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar_smem, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "BSQ_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@!p bra BSQ_WAIT_%=;\n"
        "}\n" ::"r"(bar_smem),
        "r"(parity)
        : "memory");
}

// Fallback for wide element types whose rows are not 16-byte aligned (padlen * sizeof(T) % 16
// != 0): flat element indexing, one 16-byte output vector per thread, per-element tokens.
template <typename T>
__global__ void __launch_bounds__(kThreads)
tokenize_flat_kernel(SeqView v, int64_t nseq, int padlen, FastDiv div_padlen, LutParam lutp, Specials sp,
                     Expand ex, T *__restrict__ out) {
    constexpr int TPT = 16 / sizeof(T);
    __shared__ __align__(16) uint8_t lut[256];
    __shared__ int64_t s_row0;
    __shared__ uint32_t s_col0;
    load_lut(lut, lutp);
    if (threadIdx.x == 0) {
        const int64_t f0 = static_cast<int64_t>(blockIdx.x) * (kThreads * TPT);
        const int64_t r0 = f0 / padlen;
        s_row0 = r0;
        s_col0 = static_cast<uint32_t>(f0 - r0 * padlen);
    }
    __syncthreads();
    const uint32_t x = s_col0 + threadIdx.x * TPT;  // < padlen + 4096
    const uint32_t dr = fd_div(x, div_padlen);
    int64_t row = s_row0 + dr;
    int c = static_cast<int>(x - dr * static_cast<uint32_t>(padlen));
    const int64_t total = nseq * static_cast<int64_t>(padlen);
    const int64_t f = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) * TPT;
    if (f >= total) return;
    int64_t start = __ldg(v.offs + row);
    int len = static_cast<int>(__ldg(v.offs + row + 1) - start);
    T vals[TPT];
    int nvalid = TPT;
#pragma unroll
    for (int j = 0; j < TPT; ++j) {
        if (c >= padlen) {  // crossed into the next row
            c = 0;
            ++row;
            if (row < nseq) {
                start = __ldg(v.offs + row);
                len = static_cast<int>(__ldg(v.offs + row + 1) - start);
            } else if (nvalid == TPT) {
                nvalid = j;
            }
        }
        const uint32_t code = row < nseq ? token_at(v, start, len, c, sp, lut) : 0u;
        vals[j] = cast_id<T>(expand_code(code, ex));
        ++c;
    }
    if (nvalid == TPT) {
        __stcs(reinterpret_cast<uint4 *>(out + f), *reinterpret_cast<const uint4 *>(vals));
    } else {
#pragma unroll
        for (int j = 0; j < TPT; ++j)
            if (j < nvalid) out[f + j] = vals[j];
    }
}

// ------------------------------------------------------------------------------------------
// K2 / K3: sequence-first layouts through a shared-memory tile of byte codes.
//   phase 1: tile[seq][pos] <- tokens16 (lanes run along the positions of a sequence, so the
//            residue reads are coalesced); 4-byte shared stores, row pitch 33 words.
//   phase 2: lanes run along the batch (tokens) or along the expanded C*sizeof(T) run
//            (one-hot), so global stores are coalesced / 16-byte vectorised.
// ------------------------------------------------------------------------------------------
template <typename T>
struct OneVal;  // bit pattern of T(1) as two 32-bit halves
template <> struct OneVal<int8_t> { static constexpr uint32_t lo = 1u, hi = 0u; };
template <> struct OneVal<int16_t> { static constexpr uint32_t lo = 1u, hi = 0u; };
template <> struct OneVal<int32_t> { static constexpr uint32_t lo = 1u, hi = 0u; };
template <> struct OneVal<int64_t> { static constexpr uint32_t lo = 1u, hi = 0u; };
template <> struct OneVal<float> { static constexpr uint32_t lo = 0x3f800000u, hi = 0u; };
template <> struct OneVal<double> { static constexpr uint32_t lo = 0u, hi = 0x3ff00000u; };

// Set element `e` (0 <= e < 16/sizeof(T)) of a 16-byte vector held in w[4] to T(1).
template <typename T>
__device__ __forceinline__ void set_one(uint32_t w[4], int e) {
    if (sizeof(T) == 8) {
#pragma unroll
        for (int k = 0; k < 2; ++k)
            if (e == k) { w[2 * k] = OneVal<T>::lo; w[2 * k + 1] = OneVal<T>::hi; }
    } else {
        const int byte = e * static_cast<int>(sizeof(T));
        const uint32_t pat = OneVal<T>::lo << (8 * (byte & 3));
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if ((byte >> 2) == k) w[k] |= pat;
    }
}

// 4x4 byte transpose: x[r] holds 4 consecutive positions of sequence r; y[j] gets position j of
// the 4 sequences.  8 PRMT.
__device__ __forceinline__ void transpose4x4(const uint32_t x[4], uint32_t y[4]) {
    const uint32_t t0 = __byte_perm(x[0], x[1], 0x5140), t1 = __byte_perm(x[2], x[3], 0x5140);
    const uint32_t t2 = __byte_perm(x[0], x[1], 0x7362), t3 = __byte_perm(x[2], x[3], 0x7362);
    y[0] = __byte_perm(t0, t1, 0x5410);
    y[1] = __byte_perm(t0, t1, 0x7632);
    y[2] = __byte_perm(t2, t3, 0x5410);
    y[3] = __byte_perm(t2, t3, 0x7632);
}

// MODE: how phase 2 leaves the tile (a template parameter, so every variant gets its own register budget).  The
// values appear in the kernels' names, which the profiles under profiles/ quote.
constexpr int kTokGeneric = 1;  // any element type / alignment: one element per lane, coalesced along the batch
constexpr int kOhRow = 2;       // one-hot, C*sizeof(T) is 4, 8 or 16: one store writes the whole one-hot row of a (pos, seq)
constexpr int kOhVec = 3;       // one-hot, aligned runs, any C*sizeof(T): 16-byte vectors assembled in registers (zeros included)
constexpr int kOhScalar = 4;    // one-hot, unaligned runs: one element per lane

// Phase 0 stages, for each of the tile's 128 sequences, the 16-byte aligned window of packed residues
// that holds the tile's 128 columns: one 1-D bulk asynchronous copy (TMA unit) per sequence, issued by
// the thread that resolved the sequence's offsets, completion counted on one mbarrier.  The window of
// sequence il lands at stage + il * kStagePitch so that column p0 + j sits at byte (A & 15) + j, A being
// the global address of column p0 (at most 15 + 127 < 144).  Phase 1 then needs no clamping and no
// data-dependent select tree: five 4-byte aligned LDS.32 at the lane's own word offset and four funnel
// shifts realign any source alignment, whatever mix of sequences a warp holds.  Bytes of the pitch that
// no copy wrote are stale; they only ever reach columns that the BOS / tail fix-ups overwrite.
constexpr int kStagePitch = kTilePos + 16;

__device__ __forceinline__ void staged16(const uint8_t *srow, uint32_t o, uint32_t out[4]) {
    const uint32_t *wp = reinterpret_cast<const uint32_t *>(srow + (o & ~3u));
    const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2], w3 = wp[3], w4 = wp[4];
    const uint32_t sh = (o & 3u) * 8u;
    out[0] = __funnelshift_r(w0, w1, sh); out[1] = __funnelshift_r(w1, w2, sh);
    out[2] = __funnelshift_r(w2, w3, sh); out[3] = __funnelshift_r(w3, w4, sh);
}

template <typename T, int MODE>
__global__ void __launch_bounds__(kThreads)
seqfirst_kernel(SeqView v, int64_t nseq, int64_t ld, int padlen, LutParam lutp, Specials sp, Expand ex, int ncols,
                FastDiv div_ncols, FastDiv div_rowbytes, T *__restrict__ out) {
    // nseq sequences are processed; ld (>= nseq) is the batch extent of the output array, so a
    // sub-range of a larger batch can be written in place (out already points at its first column).
    constexpr bool ONEHOT = MODE >= kOhRow;
    extern __shared__ __align__(128) uint8_t stage[];  // kTileSeqs * kStagePitch residues (+ as much again for a mask)
    __shared__ __align__(16) uint8_t lut[256];
    __shared__ __align__(16) uint8_t tile[kTileSeqs * kTilePitch];
    __shared__ TailTab tab;
    __shared__ uint4 ohtab[MODE == kOhVec ? 17 : 1];  // [b] = 16-byte vector with T(1) at byte b (b % sizeof(T) == 0); [16] = zero
    __shared__ __align__(16) int4 rinfo[kTileSeqs];   // per sequence: len, (A & 15) of the residues, of the mask
    __shared__ __align__(8) uint64_t bar;
    load_lut(lut, lutp);
    init_tailtab(tab, sp);
    if (MODE == kOhVec && threadIdx.x >= 96 && threadIdx.x < 96 + 17) {
        const int b = threadIdx.x - 96;
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        if (b < 16 && b % static_cast<int>(sizeof(T)) == 0) set_one<T>(w, b / static_cast<int>(sizeof(T)));
        ohtab[b] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    if (threadIdx.x == 128) {
        mbar_init(&bar, kTileSeqs);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int64_t i0 = static_cast<int64_t>(blockIdx.x) * kTileSeqs;
    const int p0 = blockIdx.y * kTilePos;
    const int nseq_tile = static_cast<int>(min(static_cast<int64_t>(kTileSeqs), nseq - i0));
    const int npos_tile = min(kTilePos, padlen - p0);
    const bool masked = ONEHOT && v.mask != nullptr;
    uint8_t *mstage = stage + kTileSeqs * kStagePitch;

    // ---- phase 0: one thread per sequence resolves it and issues its bulk copy ----
    if (threadIdx.x < kTileSeqs) {
        const int il = threadIdx.x;
        int len = 0;
        uint32_t shb = 0, shm = 0, nb = 0;
        if (il < nseq_tile) {
            const int64_t start = __ldg(v.offs + i0 + il);
            len = static_cast<int>(__ldg(v.offs + i0 + il + 1) - start);
            const int r0 = max(p0 - sp.bos, 0), r1 = min(p0 + kTilePos - sp.bos, len);  // residues under this tile
            const int64_t col0 = start - sp.bos + p0;                                     // packed index of column p0
            shb = static_cast<uint32_t>(reinterpret_cast<uintptr_t>(v.bytes + col0) & 15u);
            if (masked) shm = static_cast<uint32_t>(reinterpret_cast<uintptr_t>(v.mask + col0) & 15u);
            if (r1 > r0) {
                const uintptr_t a = reinterpret_cast<uintptr_t>(v.bytes + col0) & ~static_cast<uintptr_t>(15);
                const uintptr_t w0 = reinterpret_cast<uintptr_t>(v.bytes + start + r0) & ~static_cast<uintptr_t>(15);
                const uintptr_t w1 = (reinterpret_cast<uintptr_t>(v.bytes + start + r1 - 1) & ~static_cast<uintptr_t>(15)) + 16;
                nb = static_cast<uint32_t>(w1 - w0);
                uint32_t nm = 0;
                uintptr_t m0 = 0, ma = 0;
                if (masked) {
                    ma = reinterpret_cast<uintptr_t>(v.mask + col0) & ~static_cast<uintptr_t>(15);
                    m0 = reinterpret_cast<uintptr_t>(v.mask + start + r0) & ~static_cast<uintptr_t>(15);
                    nm = static_cast<uint32_t>((reinterpret_cast<uintptr_t>(v.mask + start + r1 - 1) & ~static_cast<uintptr_t>(15)) + 16 - m0);
                }
                mbar_expect_tx(&bar, nb + nm);
                bulk_g2s(stage + il * kStagePitch + (w0 - a), reinterpret_cast<const void *>(w0), nb, &bar);
                if (masked) bulk_g2s(mstage + il * kStagePitch + (m0 - ma), reinterpret_cast<const void *>(m0), nm, &bar);
            }
        }
        if (nb == 0u) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&bar)) : "memory");
        rinfo[il] = make_int4(len, static_cast<int>(shb), static_cast<int>(shm), 0);
    }
    __syncthreads();  // rinfo
    mbar_wait_u32(smem_u32(&bar), 0u);

    // ---- phase 1: tile[seq][pos] <- codes; lanes run along the positions of a sequence ----
    const uint4 padv = make_uint4(sp.pad_w, sp.pad_w, sp.pad_w, sp.pad_w);
#pragma unroll
    for (int u = 0; u < (kTileSeqs * kTilePos / 16) / kThreads; ++u) {
        const int ch = threadIdx.x + u * kThreads;
        const int q = ch & 7, il = ch >> 3;
        const int c0 = p0 + 16 * q;
        if (il < nseq_tile && c0 < padlen) {
            const int4 ri = rinfo[il];
            const int len = ri.x;
            uint4 codes = padv;
            if (c0 < sp.bos + len + sp.eos) {
                uint32_t t[4] = {0u, 0u, 0u, 0u};
                if (has_residues(c0, sp.bos, len)) {
                    uint32_t raw[4];
                    staged16(stage + il * kStagePitch, static_cast<uint32_t>(ri.y) + 16u * q, raw);
#pragma unroll
                    for (int w = 0; w < 4; ++w) t[w] = translate4(raw[w], lut);
                    if (masked) {  // masked-out residues become kCodeInvalid (0xFF)
                        staged16(mstage + il * kStagePitch, static_cast<uint32_t>(ri.z) + 16u * q, raw);
#pragma unroll
                        for (int w = 0; w < 4; ++w) t[w] |= __vcmpeq4(raw[w], 0u);
                    }
                }
                codes = tokens16_finish<false>(t, len, c0, sp, tab);
            }
            uint32_t *dst = reinterpret_cast<uint32_t *>(tile + il * kTilePitch + 16 * q);
            dst[0] = codes.x; dst[1] = codes.y; dst[2] = codes.z; dst[3] = codes.w;
        }
    }
    __syncthreads();

    // ---- phase 2 ----
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (MODE == kTokGeneric) {
        for (int pp = warp; pp < npos_tile; pp += kThreads / 32) {
            T *orow = out + (static_cast<int64_t>(p0 + pp) * ld + i0);
#pragma unroll
            for (int m = 0; m < kTileSeqs / 32; ++m) {
                const int il = lane + 32 * m;
                if (il < nseq_tile) {
                    const uint32_t code = tile[il * kTilePitch + pp];
                    __stcs(orow + il, cast_id<T>(expand_code(code, ex)));
                }
            }
        }
    } else if (MODE == kOhRow) {
        const int row_bytes = ncols * static_cast<int>(sizeof(T));
        for (int pp = warp; pp < npos_tile; pp += kThreads / 32) {
            uint8_t *orow = reinterpret_cast<uint8_t *>(out + (static_cast<int64_t>(p0 + pp) * ld + i0) * ncols);
#pragma unroll
            for (int m = 0; m < kTileSeqs / 32; ++m) {
                const int il = lane + 32 * m;
                if (il < nseq_tile) {
                    const int col = expand_code(tile[il * kTilePitch + pp], ex);
                    uint32_t w[4] = {0u, 0u, 0u, 0u};
                    if (col >= 0) set_one<T>(w, col);
                    uint8_t *o = orow + il * row_bytes;
                    if (row_bytes == 16) __stcs(reinterpret_cast<uint4 *>(o), make_uint4(w[0], w[1], w[2], w[3]));
                    else if (row_bytes == 8) __stcs(reinterpret_cast<uint2 *>(o), make_uint2(w[0], w[1]));
                    else __stcs(reinterpret_cast<uint32_t *>(o), w[0]);
                }
            }
        }
    } else if (MODE == kOhVec) {
        // Any C * sizeof(T) (codes are direct column ids here; 0xFF = all-zero row): every 16-byte vector of
        // the (pos, seq-run, C) output is assembled in registers from the `nover` sequences whose one-hot
        // rows can overlap it -- a table look-up (the vector with T(1) at byte b) and four ORs each -- and
        // stored once, zeros included: no fill pass, no partial-sector traffic, only st.global.v4.
        constexpr int S = static_cast<int>(sizeof(T));
        const int row_bytes = ncols * S;
        const int nvec = (nseq_tile * row_bytes) >> 4;
        const int nover = (16 + row_bytes - 1) / row_bytes + ((16 % row_bytes) != 0);  // warp-uniform trip count
        for (int pp = warp; pp < npos_tile; pp += kThreads / 32) {
            uint8_t *orow = reinterpret_cast<uint8_t *>(out + (static_cast<int64_t>(p0 + pp) * ld + i0) * ncols);
            const uint8_t *tcol = tile + pp;
            for (int vec = lane; vec < nvec; vec += 32) {
                const int b0 = 16 * vec;
                int il = static_cast<int>(fd_div(static_cast<uint32_t>(b0), div_rowbytes));
                int rel = il * row_bytes - b0;  // byte offset of sequence il's row inside this vector (<= 0)
                uint4 w = make_uint4(0u, 0u, 0u, 0u);
                for (int k = 0; k < nover; ++k, ++il, rel += row_bytes) {
                    const uint32_t code = il < nseq_tile ? tcol[il * kTilePitch] : 0xffu;
                    const uint32_t b = min(static_cast<uint32_t>(rel + static_cast<int>(code) * S), 16u);  // 16 = not in this vector
                    const uint4 o = ohtab[b];
                    w.x |= o.x; w.y |= o.y; w.z |= o.z; w.w |= o.w;
                }
                __stcs(reinterpret_cast<uint4 *>(orow + b0), w);
            }
            // elements after the last whole vector (partial last tile only)
            T *erow = reinterpret_cast<T *>(orow);
            for (int e = (nvec << 4) / S + lane; e < nseq_tile * ncols; e += 32) {
                const int il = static_cast<int>(fd_div(static_cast<uint32_t>(e), div_ncols));
                erow[e] = static_cast<int>(tcol[il * kTilePitch]) == e - il * ncols ? cast_id<T>(1) : cast_id<T>(0);
            }
        }
    } else {
        const int run_elems = nseq_tile * ncols;
        for (int pp = warp; pp < npos_tile; pp += kThreads / 32) {
            T *orow = out + (static_cast<int64_t>(p0 + pp) * ld + i0) * ncols;
            for (int e = lane; e < run_elems; e += 32) {
                const int il = static_cast<int>(fd_div(static_cast<uint32_t>(e), div_ncols));
                const int col = e - il * ncols;
                const int hot = expand_code(tile[il * kTilePitch + pp], ex);
                orow[e] = hot == col ? cast_id<T>(1) : cast_id<T>(0);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// K2t: (padlen, nseq) one-byte tokens -- the reference's default layout (batch_first=False) -- as a
// dedicated, instruction-lean kernel (the tile kernel above, with register 4x4 transposes for one-byte
// tokens, was issue-bound: 700 instructions per warp per 16 KB tile, profiles/r01d_seqfirst_*).  Same
// 128 x 128 tile, but
//   * the sequences' windows are staged with per-lane 16-byte cp.async (LDGSTS): the eight lanes that
//     will translate a sequence's eight chunks copy them, so the hand-over needs cp.async.wait_all +
//     __syncwarp only -- no mbarrier, no block barrier, no per-copy uniform-datapath loop;
//   * everything a thread needs per chunk is either thread-constant (chunk column, BOS predicate,
//     shared-memory addresses) or one LDS.128 of per-sequence data resolved once per CTA;
//   * phase 2 runs unguarded on full tiles (the common case) and keeps its addresses in registers.
// A persistent, software-pipelined form of this kernel (offsets of tile k+2 and windows of tile k+1 prefetched,
// double-buffered code tile, one block barrier per tile; 58 KB and 70 registers -> 3 CTAs per SM) was measured
// and rejected: C2x4 118 us vs 101 us, C1x64 124 us vs 112 us (132 / 138 us at 2 CTAs per SM).  The kernel is
// bound by shared-memory wavefronts and dependent LDS chains (profiles/r01e: LSU data pipe 65 % busy, issue-active
// 63 %), which 48 resident warps of independent one-shot CTAs cover better than 24 pipelined ones.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src) : "memory");
}

// TPC: position tiles per CTA (1, or 2 neighbouring ones): the second tile reuses the LUT, the tail table and the
// resolved sequences (its windows start 128 bytes further), so the prologue and its offsets round trip are paid once.
template <int TPC>
__global__ void __launch_bounds__(kThreads, 6)
seqfirst_tok8_kernel(SeqView v, int64_t nseq, int64_t ld, int padlen, FastDiv div_ptiles, LutParam lutp, Specials sp,
                     uint8_t *__restrict__ out) {
    __shared__ __align__(16) uint8_t lut[256];
    __shared__ TailTab tab;
    __shared__ __align__(16) int4 rinfo[kTileSeqs];  // n = bos + len, A & 15, A & ~15 (A = global address of column p0)
    __shared__ __align__(128) uint8_t stage[kTileSeqs * kStagePitch];
    __shared__ __align__(128) uint8_t tile[kTileSeqs * kTilePos];
    const int tid = threadIdx.x;
    // 1-D grid, position tiles fastest: the tiles of one group of sequences run back to back, so the
    // 32-byte sectors that two neighbouring windows share are still in L2 when the second one asks
    const uint32_t st = fd_div(blockIdx.x, div_ptiles);
    const int64_t i0 = static_cast<int64_t>(st) * kTileSeqs;
    const int p00 = static_cast<int>(blockIdx.x - st * div_ptiles.d) * (TPC * kTilePos);  // div_ptiles: groups of TPC position tiles
    const int nseq_tile = static_cast<int>(min(static_cast<int64_t>(kTileSeqs), nseq - i0));
    load_lut(lut, lutp);
    init_tailtab(tab, sp);
    if (tid >= 128) {  // warps 4..7 resolve the tile's sequences
        const int il = tid - 128;
        int n = 0;
        uintptr_t a = 0;
        if (il < nseq_tile) {
            const int64_t start = __ldg(v.offs + i0 + il);
            n = sp.bos + static_cast<int>(__ldg(v.offs + i0 + il + 1) - start);
            a = reinterpret_cast<uintptr_t>(v.bytes + (start - sp.bos + p00));
        }
        rinfo[il] = make_int4(n, static_cast<int>(a & 15u), static_cast<int>(static_cast<uint32_t>(a & ~static_cast<uintptr_t>(15))),
                              static_cast<int>(static_cast<uint32_t>(a >> 32)));
    }
    __syncthreads();

    const int q = tid & 7;
    const uint32_t stage_s = smem_u32(stage) + static_cast<uint32_t>(tid >> 3) * kStagePitch;
#pragma unroll 1
    for (int tp = 0; tp < TPC; ++tp) {
    const int p0 = p00 + tp * kTilePos;
    if (TPC > 1 && p0 >= padlen) break;
    // ---- phase 0: lane (il, q) copies 16-byte word q (and lane q == 0 word 8) of sequence il's window ----
    const int c0 = p0 + 16 * q;  // first column of this thread's chunks
    int nn[4], sh[4];
    int4 ris[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) ris[u] = rinfo[(tid >> 3) + 32 * u];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int4 ri = ris[u];
        nn[u] = ri.x;
        sh[u] = ri.y;
        // stage offsets [olo, ohi) hold the residues under this tile (columns max(bos, p0) .. min(n, p0 + 128))
        const int olo = ri.y + max(sp.bos - p0, 0), ohi = ri.y + min(ri.x - p0, kTilePos);
        const uint8_t *src = reinterpret_cast<const uint8_t *>((static_cast<uint64_t>(static_cast<uint32_t>(ri.w)) << 32) |
                                                               static_cast<uint32_t>(ri.z)) + tp * kTilePos;
        const uint32_t dst = stage_s + static_cast<uint32_t>(32 * u) * kStagePitch + 16u * q;
        if (16 * q < ohi && 16 * q + 16 > olo) cp_async16(dst, src + 16 * q);
        if (q == 0 && ohi > kTilePos) cp_async16(dst + kTilePos, src + kTilePos);
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncwarp();

    // ---- phase 1: tile[seq][pos] <- codes ----
    const uint4 padv = make_uint4(sp.pad_w, sp.pad_w, sp.pad_w, sp.pad_w);
    const bool bos_here = sp.bos && c0 == 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int il = (tid >> 3) + 32 * u;
        const int n = nn[u];
        uint4 codes = padv;
        if (c0 < n + sp.eos) {
            uint32_t t[4] = {0u, 0u, 0u, 0u};
            if (c0 < n) {
                uint32_t raw[4];
                staged16(stage + il * kStagePitch, static_cast<uint32_t>(sh[u]) + 16u * q, raw);
#pragma unroll
                for (int w = 0; w < 4; ++w) t[w] = translate4(raw[w], lut);
            }
            if (bos_here) t[0] = __byte_perm(t[0], sp.bos_w, 0x3214);
            if (c0 + 16 > n) {  // the row ends inside this chunk
                const uint4 m = tab.m[n - c0], f = tab.f[n - c0];
                t[0] = (t[0] & m.x) | f.x; t[1] = (t[1] & m.y) | f.y;
                t[2] = (t[2] & m.z) | f.z; t[3] = (t[3] & m.w) | f.w;
            }
            codes = make_uint4(t[0], t[1], t[2], t[3]);
        }
        // 16-byte chunks XOR-swizzled by the sequence group, so that phase 2's column-of-words reads
        // (16 sequences apart) hit 32 distinct banks
        *reinterpret_cast<uint4 *>(tile + il * kTilePos + 16 * (q ^ ((il >> 4) & 7))) = codes;
    }
    __syncthreads();

    // ---- phase 2: thread = 16 sequences (group A) x 4 positions (word pw): 16 LDS.32, four 4x4 byte
    // transposes, one 16-byte store per position; lanes A = 0..7 make 128 contiguous bytes per row ----
    const int warp = tid >> 5, lane = tid & 31;
    const int A = lane & 7, pw = 4 * warp + (lane >> 3);
    const uint32_t *t32 = reinterpret_cast<const uint32_t *>(tile) + 16 * A * (kTilePos / 4) + (pw ^ (4 * A));
    uint32_t y[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        uint32_t x[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) x[k] = t32[(4 * a + k) * (kTilePos / 4)];
        transpose4x4(x, y[a]);
    }
    const int pos = p0 + 4 * pw;
    uint8_t *o = out + (static_cast<int64_t>(pos) * ld + i0 + 16 * A);
    if (nseq_tile == kTileSeqs && p0 + kTilePos <= padlen) {
#pragma unroll
        for (int j = 0; j < 4; ++j, o += ld) __stcs(reinterpret_cast<uint4 *>(o), make_uint4(y[0][j], y[1][j], y[2][j], y[3][j]));
    } else {
        const int nvalid = nseq_tile - 16 * A;  // sequences of this group that exist
#pragma unroll
        for (int j = 0; j < 4; ++j, o += ld) {
            if (pos + j >= padlen || nvalid <= 0) continue;
            if (nvalid >= 16) {
                __stcs(reinterpret_cast<uint4 *>(o), make_uint4(y[0][j], y[1][j], y[2][j], y[3][j]));
            } else {
#pragma unroll
                for (int k = 0; k < 16; ++k)
                    if (k < nvalid) o[k] = static_cast<uint8_t>(y[k >> 2][j] >> (8 * (k & 3)));
            }
        }
    }
    if (TPC > 1 && tp + 1 < TPC) __syncthreads();  // the tile is rewritten by the next position tile
    }
}

// ------------------------------------------------------------------------------------------
// K4: decode.  inv[key + 128] for key in [-128, 384): 0..255 = character, 0x100 + k = the
// 5-character special k (0 <BOS>, 1 <EOS>, 2 <PAD>), 0xFFFF = no entry.
// ------------------------------------------------------------------------------------------
struct InvParam {
    uint16_t e[512];
};
constexpr uint16_t kInvNone = 0xFFFF;

__device__ __forceinline__ int32_t load_key(const uint8_t *p, int itemsize) {
    switch (itemsize) {  // src/tokenize.h:107-124 + the uint32 truncation at :145/:167
        case 1: return static_cast<int32_t>(*p);
        case 2: return static_cast<int32_t>(*reinterpret_cast<const uint16_t *>(p));
        case 4: return *reinterpret_cast<const int32_t *>(p);
        default: return static_cast<int32_t>(*reinterpret_cast<const uint64_t *>(p));
    }
}

__device__ __forceinline__ uint32_t inv_lookup(const uint16_t *inv, int32_t key) {
    return (key >= -128 && key < 384) ? inv[key + 128] : kInvNone;
}

// pass 1: one warp per row, persistent grid (rows dealt round-robin to the warps).  row_len[r] =
// decoded length; first_bad = min flat index of a token without an entry.  FAST: one-byte tokens,
// contiguous along the row, every row 4-byte aligned -> four tokens per 32-bit load.
constexpr int kDecWarps = 8;

// character j of the text of special k: <BOS> <EOS> <PAD> (src/tokenize.h:92-100)
__device__ __forceinline__ uint8_t special_char(int k, int j) {
    const uint32_t mid = k == 0 ? 0x00534f42u : (k == 1 ? 0x00534f45u : 0x00444150u);  // "BOS" "EOS" "PAD", little-endian
    return j == 0 ? '<' : (j == 4 ? '>' : static_cast<uint8_t>(mid >> (8 * (j - 1))));
}

__device__ __forceinline__ void decode_fetch4(const uint8_t *rp, int itemsize, int64_t col_stride, int64_t c, int64_t cols,
                                              const uint16_t *inv, bool fast, uint32_t e[4]) {
    // entries of tokens c .. c+3 of a row (kInvNone beyond the row end is reported as 0xFFFE = "absent")
    if (fast) {
        const uint32_t x = c < cols ? *reinterpret_cast<const uint32_t *>(rp + c) : 0u;
#pragma unroll
        for (int k = 0; k < 4; ++k) e[k] = c + k < cols ? inv[((x >> (8 * k)) & 0xffu) + 128] : 0xFFFEu;
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) e[k] = c + k < cols ? inv_lookup(inv, load_key(rp + (c + k) * col_stride, itemsize)) : 0xFFFEu;
    }
}

__global__ void __launch_bounds__(kDecWarps * 32)
decode_len_kernel(const uint8_t *__restrict__ tokens, int itemsize, int64_t rows, int64_t cols, int64_t row_stride,
                  int64_t col_stride, int fast, InvParam invp, int64_t *__restrict__ row_len,
                  unsigned long long *first_bad) {
    __shared__ uint16_t inv[512];
    for (int i = threadIdx.x; i < 512; i += kDecWarps * 32) inv[i] = invp.e[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t gw = static_cast<int64_t>(blockIdx.x) * kDecWarps + (threadIdx.x >> 5);
    const int64_t GW = static_cast<int64_t>(gridDim.x) * kDecWarps;
    for (int64_t r = gw; r < rows; r += GW) {
        const uint8_t *rp = tokens + r * row_stride;
        int specials = 0;
        unsigned long long bad = ~0ull;
        for (int64_t c0 = 0; c0 < cols; c0 += 128) {
            const int64_t c = c0 + 4 * lane;
            uint32_t e[4];
            decode_fetch4(rp, itemsize, col_stride, c, cols, inv, fast != 0, e);
#pragma unroll
            for (int k = 3; k >= 0; --k) {
                if (e[k] == kInvNone) bad = static_cast<unsigned long long>(r * cols + c + k);  // lowest k wins
                else if (e[k] != 0xFFFEu) specials += (e[k] >> 8) & 1;
            }
            if (bad != ~0ull) break;  // this lane's first bad token is its lowest; later chunks cannot beat it
        }
        for (int o = 16; o > 0; o >>= 1) {
            specials += __shfl_xor_sync(0xffffffffu, specials, o);
            bad = min(bad, __shfl_xor_sync(0xffffffffu, bad, o));
        }
        if (lane == 0) {
            row_len[r] = cols + 4ll * specials;
            if (bad != ~0ull) atomicMin(first_bad, bad);
        }
    }
}

// pass 1, lean form for one-byte tokens that are contiguous along the row (any row alignment, any length): 16
// tokens per lane and load over the aligned 16-byte vectors that cover the row, a 256-entry class table (0 = one
// character, 1 = five-character special, 0x100 = no entry) summed per vector -- 2.5 instructions per token instead
// of 31 (profiles/r01e: the general kernel was issue-bound at 0.78 TB/s).  Bytes of the first / last vector that lie
// outside the row are replaced by token 0, which is a plain character in every alphabet.  A row that holds a token
// without an entry (the error path) is rescanned for the exact position.
// ANYALIGN = false: rows are 16-byte aligned and a multiple of 16 long (what batch_tokenize produces for such padlens):
// the shifts and masks fold away.
template <bool ANYALIGN>
__global__ void __launch_bounds__(kDecWarps * 32)
decode_len16_kernel(const uint8_t *__restrict__ tokens, int64_t rows, int64_t cols, int64_t row_stride, InvParam invp,
                    int64_t *__restrict__ row_len, int32_t *__restrict__ row_tail, unsigned long long *first_bad) {
    __shared__ uint16_t cls[256];
    __shared__ uint8_t knd[256];  // which special (0 <BOS>, 1 <EOS>, 2 <PAD>)
    for (int i = threadIdx.x; i < 256; i += kDecWarps * 32) {
        const uint16_t e = invp.e[i + 128];
        cls[i] = e == kInvNone ? 0x100 : ((e >> 8) & 1);
        knd[i] = static_cast<uint8_t>(e & 3u);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t gw = static_cast<int64_t>(blockIdx.x) * kDecWarps + (threadIdx.x >> 5);
    const int64_t GW = static_cast<int64_t>(gridDim.x) * kDecWarps;
    for (int64_t r = gw; r < rows; r += GW) {
        const uint8_t *rb = tokens + r * row_stride;
        const int a = ANYALIGN ? static_cast<int>(reinterpret_cast<uintptr_t>(rb) & 15u) : 0;
        const uint4 *rp = reinterpret_cast<const uint4 *>(rb - a);
        const int64_t nvec = (a + cols + 15) >> 4;
        const int ktail = ANYALIGN ? static_cast<int>(a + cols - 16 * (nvec - 1)) : 16;  // bytes of the last vector that belong to the row
        uint32_t specials = 0, bad = 0;
        // the run of one repeated five-character special that ends the row (the <PAD>s behind a sequence: 4/5 of the
        // decoded text of a padded batch): pass 2 writes it as a pattern fill without reading those tokens again.
        // T: the row's last token; tail_vec: first vector from which every byte equals T (vector granularity).
        const uint32_t T = (row_tail != nullptr && cols > 0) ? rb[cols - 1] : 0u;
        const uint32_t T4 = T * 0x01010101u;
        int tail_vec = 0;
#pragma unroll 2
        for (int64_t v = lane; v < nvec; v += 32) {
            const uint4 x = __ldcs(rp + v);
            uint32_t w[4] = {x.x, x.y, x.z, x.w};
            uint32_t d[4] = {x.x ^ T4, x.y ^ T4, x.z ^ T4, x.w ^ T4};  // non-zero bytes: tokens other than T
            if (v == 0 && a != 0) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    w[k] &= ~lt_mask(a, k);
                    d[k] &= ~lt_mask(a, k);
                }
            }
            if (v == nvec - 1 && ktail != 16) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    w[k] &= lt_mask(ktail, k);
                    d[k] &= lt_mask(ktail, k);
                }
            }
            uint32_t sum = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                sum += cls[w[k] & 0xffu] + cls[__byte_perm(w[k], 0, 0x4441)] + cls[__byte_perm(w[k], 0, 0x4442)] + cls[w[k] >> 24];
            specials += sum & 0xffu;
            bad |= sum >> 8;
            if (d[0] | d[1] | d[2] | d[3]) tail_vec = static_cast<int>(v) + 1;
        }
        for (int o = 16; o > 0; o >>= 1) specials += __shfl_xor_sync(0xffffffffu, specials, o);
        if (row_tail != nullptr) {
            for (int o = 16; o > 0; o >>= 1) tail_vec = max(tail_vec, __shfl_xor_sync(0xffffffffu, tail_vec, o));
            // columns [16 tail_vec - a, cols) all hold T; only a special's run is worth a separate path
            const int64_t ts = min(max(static_cast<int64_t>(16) * tail_vec - a, static_cast<int64_t>(0)), cols);
            if (lane == 0)
                row_tail[r] = (cls[T] & 1) ? static_cast<int32_t>(static_cast<uint32_t>(ts) | (static_cast<uint32_t>(knd[T]) << 30)) : static_cast<int32_t>(cols);
        }
        if (__any_sync(0xffffffffu, bad != 0)) {
            unsigned long long b = ~0ull;
            for (int64_t c = lane; c < cols; c += 32)
                if (cls[rb[c]] & 0x100) {
                    b = static_cast<unsigned long long>(r * cols + c);
                    break;
                }
            for (int o = 16; o > 0; o >>= 1) b = min(b, __shfl_xor_sync(0xffffffffu, b, o));
            if (lane == 0) atomicMin(first_bad, b);
        }
        if (lane == 0) row_len[r] = cols + 4ll * specials;
    }
}

// The same pass for rows of at most 32 * VPL vectors (padlen up to 1024 / 2048), software-pipelined: a warp holds
// its whole row in registers -- VPL vectors per lane -- and the NEXT row's vectors and last token are in flight while
// the current one is counted.  The loop above takes one row at a time through the chain last token -> vectors ->
// reduction per warp and ran at 2.8 TB/s (ncu r02r: 95 us for 268 MB); vectors wholly inside the trailing run skip
// the class look-ups; the three warp reductions are single REDUX instructions.
// THR: the token ids are laid out [0, a) characters, [a, b) five-character specials, [b, 256) nothing, b <= 128 (every
// tokenizer of the reference: the specials follow the alphabet) -- the class of four tokens is then two SIMD-in-a-word
// comparisons ((w | 0x80808080) - a x 0x01010101 has bit 7 of a byte set iff that byte >= a) instead of four table
// look-ups: 8 instructions per word instead of 16 (ncu r02s: the look-ups were 99 of the kernel's 227 instructions
// per row, issue-active 79 %).
template <bool ANYALIGN, int VPL, bool THR>
__global__ void __launch_bounds__(kDecWarps * 32)
decode_len16p_kernel(const uint8_t *__restrict__ tokens, int64_t rows, int64_t cols, int64_t row_stride, InvParam invp,
                     int64_t *__restrict__ row_len, int32_t *__restrict__ row_tail, unsigned long long *first_bad,
                     uint32_t thr_lo4, uint32_t thr_hi4) {
    __shared__ uint16_t cls[256];
    __shared__ uint8_t knd[256];  // which special (0 <BOS>, 1 <EOS>, 2 <PAD>)
    for (int i = threadIdx.x; i < 256; i += kDecWarps * 32) {
        const uint16_t e = invp.e[i + 128];
        cls[i] = e == kInvNone ? 0x100 : ((e >> 8) & 1);
        knd[i] = static_cast<uint8_t>(e & 3u);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t gw = static_cast<int64_t>(blockIdx.x) * kDecWarps + (threadIdx.x >> 5);
    const int64_t GW = static_cast<int64_t>(gridDim.x) * kDecWarps;
    const bool want_tail = row_tail != nullptr && cols > 0;
    uint4 xn[VPL];
    uint32_t Tn = 0;
    auto load_row = [&](int64_t r) {
        const uint8_t *rb = tokens + r * row_stride;
        const int a = ANYALIGN ? static_cast<int>(reinterpret_cast<uintptr_t>(rb) & 15u) : 0;
        const uint4 *rp = reinterpret_cast<const uint4 *>(rb - a);
        const int nvec = static_cast<int>((a + cols + 15) >> 4);
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
            xn[i] = make_uint4(0u, 0u, 0u, 0u);
            if (lane + 32 * i < nvec) xn[i] = __ldcs(rp + lane + 32 * i);
        }
        if (want_tail) Tn = rb[cols - 1];
    };
    if (gw < rows) load_row(gw);
    for (int64_t r = gw; r < rows; r += GW) {
        uint4 x[VPL];
#pragma unroll
        for (int i = 0; i < VPL; ++i) x[i] = xn[i];
        const uint32_t T = Tn;
        if (r + GW < rows) load_row(r + GW);
        const uint8_t *rb = tokens + r * row_stride;
        const int a = ANYALIGN ? static_cast<int>(reinterpret_cast<uintptr_t>(rb) & 15u) : 0;
        const int nvec = static_cast<int>((a + cols + 15) >> 4);
        const int ktail = ANYALIGN ? static_cast<int>(a + cols - 16 * (static_cast<int64_t>(nvec) - 1)) : 16;
        const uint32_t T4 = T * 0x01010101u;
        const uint32_t clsT = cls[T];
        uint32_t specials = 0, bad = 0;
        int tail_vec = 0;
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
            const int v = lane + 32 * i;
            if (v < nvec) {
                uint32_t w[4] = {x[i].x, x[i].y, x[i].z, x[i].w};
                uint32_t d[4] = {w[0] ^ T4, w[1] ^ T4, w[2] ^ T4, w[3] ^ T4};  // non-zero bytes: tokens other than T
                int inrow = 16;
                if (ANYALIGN && v == 0 && a != 0) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        w[k] &= ~lt_mask(a, k);
                        d[k] &= ~lt_mask(a, k);
                    }
                    inrow -= a;
                }
                if (ANYALIGN && v == nvec - 1 && ktail != 16) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        w[k] &= lt_mask(ktail, k);
                        d[k] &= lt_mask(ktail, k);
                    }
                    inrow -= 16 - ktail;
                }
                if (want_tail && (d[0] | d[1] | d[2] | d[3]) == 0) {  // every token of the row in this vector is T
                    specials += static_cast<uint32_t>(inrow) * (clsT & 1u);
                    bad |= clsT >> 8;
                } else if (THR) {
                    constexpr uint32_t H = 0x80808080u;
                    uint32_t ge = 0, over = 0;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint32_t wh = w[k] | H;
                        ge += __popc((wh - thr_lo4) & H);
                        over |= ((wh - thr_hi4) | w[k]) & H;  // a byte >= b, or >= 128
                    }
                    specials += ge;
                    bad |= over;
                    tail_vec = v + 1;
                } else {
                    uint32_t sum = 0;
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        sum += cls[w[k] & 0xffu] + cls[__byte_perm(w[k], 0, 0x4441)] + cls[__byte_perm(w[k], 0, 0x4442)] + cls[w[k] >> 24];
                    specials += sum & 0xffu;
                    bad |= sum >> 8;
                    tail_vec = v + 1;
                }
            }
        }
        specials = __reduce_add_sync(0xffffffffu, specials);
        if (want_tail) {
            tail_vec = __reduce_max_sync(0xffffffffu, tail_vec);
            // columns [16 tail_vec - a, cols) all hold T; only a special's run is worth a separate path
            const int64_t ts = min(max(static_cast<int64_t>(16) * tail_vec - a, static_cast<int64_t>(0)), cols);
            if (lane == 0)
                row_tail[r] = (clsT & 1) ? static_cast<int32_t>(static_cast<uint32_t>(ts) | (static_cast<uint32_t>(knd[T]) << 30)) : static_cast<int32_t>(cols);
        }
        if (__reduce_or_sync(0xffffffffu, bad) != 0) {
            unsigned long long b = ~0ull;
            for (int64_t c = lane; c < cols; c += 32)
                if (cls[rb[c]] & 0x100) {
                    b = static_cast<unsigned long long>(r * cols + c);
                    break;
                }
            for (int o = 16; o > 0; o >>= 1) b = min(b, __shfl_xor_sync(0xffffffffu, b, o));
            if (lane == 0) atomicMin(first_bad, b);
        }
        if (lane == 0) row_len[r] = cols + 4ll * specials;
    }
}

__global__ void fill_i32_kernel(int32_t *p, int64_t n, int32_t v) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// exclusive scan of row_len (three small kernels; rows can be millions)
constexpr int kScanBlock = 1024;
__global__ void __launch_bounds__(kScanBlock)
scan_local_kernel(int64_t *__restrict__ data, int64_t n, int64_t *__restrict__ block_tot) {
    __shared__ int64_t s_warp[32];
    __shared__ int64_t s_total;
    const int64_t i = static_cast<int64_t>(blockIdx.x) * kScanBlock + threadIdx.x;
    const int64_t x = i < n ? data[i] : 0;
    const int64_t ex = block_exclusive_scan(x, s_warp, &s_total);
    if (i < n) data[i] = ex;
    if (threadIdx.x == 0) block_tot[blockIdx.x] = s_total;
}

__global__ void __launch_bounds__(kScanBlock)
scan_totals_kernel(int64_t *__restrict__ block_tot, int64_t nblocks, int64_t *__restrict__ grand_total) {
    __shared__ int64_t s_warp[32];
    __shared__ int64_t s_total;
    int64_t carry = 0;
    for (int64_t base = 0; base < nblocks; base += kScanBlock) {
        const int64_t i = base + threadIdx.x;
        const int64_t x = i < nblocks ? block_tot[i] : 0;
        const int64_t ex = block_exclusive_scan(x, s_warp, &s_total);
        if (i < nblocks) block_tot[i] = carry + ex;
        carry += s_total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *grand_total = carry;
}

// The second and third step in one for up to a few thousand blocks: every block sums the totals of the blocks in front
// of it itself (nblocks loads spread over its threads) instead of waiting for a one-block scan of the totals.
__global__ void __launch_bounds__(kScanBlock)
scan_add_direct_kernel(int64_t *__restrict__ data, int64_t n, const int64_t *__restrict__ block_tot, const int64_t *__restrict__ first_bad,
                       int64_t *__restrict__ host_out) {
    __shared__ int64_t s_warp[32];
    __shared__ int64_t s_pre;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t part = 0;
    for (int64_t j = threadIdx.x; j < blockIdx.x; j += kScanBlock) part += block_tot[j];
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) s_warp[warp] = part;
    __syncthreads();
    if (warp == 0) {
        int64_t v = s_warp[lane];  // (kScanBlock / 32 = 32 warps)
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) s_pre = v;
    }
    __syncthreads();
    const int64_t pre = s_pre;
    const int64_t i = static_cast<int64_t>(blockIdx.x) * kScanBlock + threadIdx.x;
    if (i < n) data[i] += pre;
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) {
        const int64_t total = pre + block_tot[blockIdx.x];
        data[n] = total;
        host_out[0] = *first_bad;
        host_out[1] = total;
    }
}

// (host_out: two words of pinned host memory the caller polls after its stream synchronize -- {first bad token, total}
// leave with the last kernel instead of a separate device-to-host copy)
__global__ void __launch_bounds__(kScanBlock)
scan_add_kernel(int64_t *__restrict__ data, int64_t n, const int64_t *__restrict__ block_pre,
                const int64_t *__restrict__ grand_total, const int64_t *__restrict__ first_bad, int64_t *__restrict__ host_out) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * kScanBlock + threadIdx.x;
    if (i < n) data[i] += block_pre[blockIdx.x];
    if (i == 0) {
        data[n] = *grand_total;
        host_out[0] = *first_bad;
        host_out[1] = *grand_total;
    }
}

// pass 2: one warp per row, persistent grid.  Per step a warp takes 128 tokens (four per lane), a warp
// scan of the decoded lengths gives every lane its position, and the characters are first laid out in
// a per-warp shared-memory stage that carries the same 16-byte misalignment as the row's place in
// the output buffer: whole 16-byte vectors then leave with st.global.v4, only the row's first and
// last partial vectors (shared with the neighbouring rows) are written byte-wise.
constexpr int kDecStage = 16 + 512 * 5 + 48;  // carry + the longest step (512 specials) + slack, a multiple of 16

// One decode step as a stream of whole 32-bit words.  A lane's TPL (4 or 16) tokens expand to TPL + 4 * (#specials)
// bytes -- whole words -- so the text moves as words: token k sits at byte k & 3 of the lane's current word; a special
// closes that word with its first 4 - (k & 3) characters and opens the next one with the remaining (k & 3) + 1; a
// plain character at byte 3 closes the word.  Word offsets come from one warp scan; the stream is shifted by the
// carry (fill & 3 bytes) with one funnel shift per word.  Returns the number of bytes appended to the stage.
// bytes [a, a + 16) of the 32 bytes v:n (a = 1..15, warp-uniform)
__device__ __forceinline__ uint4 shift16(const uint4 &v, const uint4 &n, int a) {
    const uint32_t sh = static_cast<uint32_t>(a & 3) * 8u;
    switch (a >> 2) {
        case 0: return make_uint4(__funnelshift_r(v.x, v.y, sh), __funnelshift_r(v.y, v.z, sh), __funnelshift_r(v.z, v.w, sh), __funnelshift_r(v.w, n.x, sh));
        case 1: return make_uint4(__funnelshift_r(v.y, v.z, sh), __funnelshift_r(v.z, v.w, sh), __funnelshift_r(v.w, n.x, sh), __funnelshift_r(n.x, n.y, sh));
        case 2: return make_uint4(__funnelshift_r(v.z, v.w, sh), __funnelshift_r(v.w, n.x, sh), __funnelshift_r(n.x, n.y, sh), __funnelshift_r(n.y, n.z, sh));
        default: return make_uint4(__funnelshift_r(v.w, n.x, sh), __funnelshift_r(n.x, n.y, sh), __funnelshift_r(n.y, n.z, sh), __funnelshift_r(n.z, n.w, sh));
    }
}

// "<BOS" / "<EOS" / "<PAD" as a little-endian word (registers, no table look-up)
__device__ __forceinline__ uint32_t special_word(uint32_t entry) {
    const uint32_t k = entry & 3u;
    return k == 0 ? 0x534f423cu : (k == 1 ? 0x534f453cu : 0x4441503cu);
}
__device__ __forceinline__ uint32_t pack4(uint32_t e0, uint32_t e1, uint32_t e2, uint32_t e3) {
    return __byte_perm(__byte_perm(e0, e1, 0x0040), __byte_perm(e2, e3, 0x0040), 0x5410);
}

// Four one-byte tokens -> four bytes of a 256-byte shared-memory table whose address has a zero low byte: one PRMT
// forms each address (the token replaces the low byte), one LDS.U8 reads it, three PRMTs pack the word.
__device__ __forceinline__ uint32_t dec_lds_u8(uint32_t addr) {
    uint32_t v;
    asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t dec_lut4(uint32_t lutbase, uint32_t x) {
    const uint32_t b0 = dec_lds_u8(__byte_perm(lutbase, x, 0x3214)), b1 = dec_lds_u8(__byte_perm(lutbase, x, 0x3215));
    const uint32_t b2 = dec_lds_u8(__byte_perm(lutbase, x, 0x3216)), b3 = dec_lds_u8(__byte_perm(lutbase, x, 0x3217));
    return __byte_perm(__byte_perm(b0, b1, 0x0040), __byte_perm(b2, b3, 0x0040), 0x5410);
}

// nact: lanes 0 .. nact-1 hold tokens (a row's last step may be partial); the others contribute nothing.
template <int TPL>
__device__ __forceinline__ int decode_word_step(const uint32_t (&ee)[TPL], uint32_t *stage_w, int fill, int lane, int nact = 32) {
    constexpr int G = TPL / 4;
    // groups of four tokens without a special are one packed word; only the others are walked token by token
    uint32_t gm[G];
    int nw = G;
#pragma unroll
    for (int g = 0; g < G; ++g) {
        gm[g] = (ee[4 * g] | ee[4 * g + 1] | ee[4 * g + 2] | ee[4 * g + 3]) & 0x100u;
        if (gm[g]) nw += static_cast<int>(((ee[4 * g] >> 8) & 1u) + ((ee[4 * g + 1] >> 8) & 1u) + ((ee[4 * g + 2] >> 8) & 1u) + ((ee[4 * g + 3] >> 8) & 1u));
    }
    const bool act = lane < nact;
    if (!act) nw = 0;
    int incl = nw;
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += y;
    }
    const int nwords = __shfl_sync(0xffffffffu, incl, 31);
    uint32_t last;  // this lane's final word: decided by its last four tokens
    if (!gm[G - 1]) {
        last = pack4(ee[TPL - 4], ee[TPL - 3], ee[TPL - 2], ee[TPL - 1]);
    } else if (ee[TPL - 4] == ee[TPL - 3] && ee[TPL - 4] == ee[TPL - 2] && ee[TPL - 4] == ee[TPL - 1]) {
        last = __byte_perm(special_word(ee[TPL - 1]), 0x3eu, 0x4321);  // "XYZ>"
    } else {
        last = 0;
#pragma unroll
        for (int k = TPL - 4; k < TPL; ++k)
            last = (ee[k] & 0x100u) ? __funnelshift_rc(special_word(ee[k]), 0x3eu, 32 - 8 * (k & 3)) : (last | ((ee[k] & 0xffu) << (8 * (k & 3))));
    }
    const int r8 = (fill & 3) * 8, kw = fill >> 2;
    uint32_t pw = __shfl_up_sync(0xffffffffu, last, 1);
    if (lane == 0) pw = r8 ? stage_w[kw] << (32 - r8) : 0u;
    uint32_t *d = stage_w + kw + incl - nw;
    if (!act) return 4 * nwords;
#pragma unroll
    for (int g = 0; g < G; ++g) {
        if (!gm[g]) {
            const uint32_t w = pack4(ee[4 * g], ee[4 * g + 1], ee[4 * g + 2], ee[4 * g + 3]);
            *d++ = __funnelshift_l(pw, w, r8);
            pw = w;
        } else if (ee[4 * g] == ee[4 * g + 1] && ee[4 * g] == ee[4 * g + 2] && ee[4 * g] == ee[4 * g + 3]) {
            // four times the same special (the <PAD> run behind a sequence): 20 characters = five constant words
            const uint32_t P = special_word(ee[4 * g]);  // "<XYZ"; the other four words are byte rotations of it with '>'
            const uint32_t w1 = __byte_perm(P, 0x3eu, 0x2104), w2 = __byte_perm(P, 0x3eu, 0x1043);
            const uint32_t w3 = __byte_perm(P, 0x3eu, 0x0432), w4 = __byte_perm(P, 0x3eu, 0x4321);
            d[0] = __funnelshift_l(pw, P, r8); d[1] = __funnelshift_l(P, w1, r8); d[2] = __funnelshift_l(w1, w2, r8);
            d[3] = __funnelshift_l(w2, w3, r8); d[4] = __funnelshift_l(w3, w4, r8);
            d += 5;
            pw = w4;
        } else {
            uint32_t cur = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const uint32_t e = ee[4 * g + b];
                const bool sp = (e & 0x100u) != 0;
                const uint32_t P = special_word(e);
                cur |= (sp ? P : (e & 0xffu)) << (8 * b);
                if (sp) {
                    *d++ = __funnelshift_l(pw, cur, r8);
                    pw = cur;
                    cur = __funnelshift_rc(P, 0x3eu, 32 - 8 * b);
                }
            }
            *d++ = __funnelshift_l(pw, cur, r8);  // byte 3 closes the word either way
            pw = cur;
        }
    }
    if (lane == nact - 1 && r8) *d = pw >> (32 - r8);
    return 4 * nwords;
}

// `n` tokens of special k appended to the stage: bytes fill .. fill + 5 n repeat its five characters.
__device__ __forceinline__ void decode_fill_special(int k, int n, const uint32_t (*patw)[8], uint8_t *stage, int fill, int lane) {
    uint32_t *stage_w = reinterpret_cast<uint32_t *>(stage);
    const int k0 = (fill + 3) >> 2, kend = (fill + 5 * n) >> 2;
    if (lane < 4 * k0 - fill) stage[fill + lane] = special_char(k, lane);
    int ph = (4 * (k0 + lane) - fill) % 5;  // the phase advances by 128 % 5 = 3 from one of a lane's words to the next
    for (int q = k0 + lane; q < kend; q += 32) {
        stage_w[q] = patw[k][ph];
        ph = ph >= 2 ? ph - 2 : ph + 3;
    }
    if (lane < ((fill + 5 * n) & 3)) stage[4 * kend + lane] = special_char(k, (4 * kend + lane - fill) % 5);
}

// STAGED: a warp's next row of tokens is fetched into a two-slot shared-memory ring by one 1-D bulk asynchronous copy
// (TMA unit) while the current row is decoded, together with the row's output offset: the kernel used to be bound by
// the chain row offset -> tokens -> text of one row at a time per warp (ncu r02q: long-scoreboard 4.9 per issue,
// half of the warps' time).  Needs one-byte contiguous tokens and rows that fit the ring.
#ifndef BSQ_DEC_MINB
#define BSQ_DEC_MINB 4
#endif
template <bool ANYALIGN, bool STAGED>  // ANYALIGN = false: every row is 16-byte aligned (the realignment folds away)
__global__ void __launch_bounds__(kDecWarps * 32, BSQ_DEC_MINB)
decode_chars_kernel(const uint8_t *__restrict__ tokens, int itemsize, int64_t rows, int64_t cols, int64_t row_stride,
                    int64_t col_stride, int fast, InvParam invp, const int64_t *__restrict__ row_offs,
                    const int32_t *__restrict__ row_tail, uint8_t *__restrict__ chars, int64_t capacity,
                    const unsigned long long *__restrict__ first_bad) {
    // (bsq_decode_text launches this pass before the host knows pass 1's verdict: a text that does not fit is not
    // written, and neither is one with a token that has no entry -- its row lengths are not what this pass would write)
    if (capacity >= 0 && (row_offs[rows] > capacity || *first_bad != ~0ull)) return;
    extern __shared__ __align__(128) uint8_t rowring[];  // STAGED: kDecWarps x 2 slots of slot_bytes
    __shared__ __align__(8) uint64_t rowbar[kDecWarps][2];
    __shared__ uint16_t inv[512];
    __shared__ __align__(16) uint8_t pat16[3][5][16];  // pat16[k][ph]: 16 bytes of special k's text repeated, starting at phase ph
    __shared__ __align__(16) uint8_t stage_all[kDecWarps][kDecStage];
    __shared__ uint32_t patw[4][8];  // patw[k][ph]: four bytes of special k's text repeated, starting at phase ph
    // one-byte tokens -> one byte: the character, or 0x80 | kind for a five-character special (characters are ASCII;
    // an alphabet with a character >= 0x80 keeps to the 16-bit table)
    __shared__ __align__(256) uint8_t lutb[256];
    __shared__ int lutb_bad;
    if (threadIdx.x == 0) lutb_bad = 0;
    for (int i = threadIdx.x; i < 512; i += kDecWarps * 32) inv[i] = invp.e[i];
    __syncthreads();
    {
        const uint16_t e = invp.e[threadIdx.x + 128];  // (kDecWarps * 32 = 256 threads)
        lutb[threadIdx.x] = (e & 0x100u) ? static_cast<uint8_t>(0x80u | (e & 3u)) : static_cast<uint8_t>(e);
        if (e != kInvNone && !(e & 0x100u) && (e & 0x80u)) lutb_bad = 1;
    }
    if (threadIdx.x >= 32 && threadIdx.x < 40) patw[3][threadIdx.x - 32] = 0u;  // (kind 3 does not exist; keeps stray look-ups defined)
    if (threadIdx.x < 240) {
        const int i = threadIdx.x;
        pat16[i / 80][(i / 16) % 5][i % 16] = special_char(i / 80, ((i / 16) % 5 + i % 16) % 5);
    }
    if (threadIdx.x < 15) {
        const int k = threadIdx.x / 5, ph = threadIdx.x % 5;
        uint32_t w = 0;
        for (int j = 0; j < 4; ++j) w |= static_cast<uint32_t>(special_char(k, (ph + j) % 5)) << (8 * j);
        patw[k][ph] = w;
    }
    if (STAGED && threadIdx.x < 2 * kDecWarps) {
        mbar_init(&rowbar[threadIdx.x >> 1][threadIdx.x & 1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *stage = stage_all[warp];
    uint32_t *stage_w = reinterpret_cast<uint32_t *>(stage);
    const uint32_t lutbase = smem_u32(lutb);
    const bool bytelut = fast && lutb_bad == 0;
    const int lane5 = lane % 5;
    const int64_t gw = static_cast<int64_t>(blockIdx.x) * kDecWarps + warp;
    const int64_t GW = static_cast<int64_t>(gridDim.x) * kDecWarps;
    const int slot_bytes = STAGED ? static_cast<int>((cols + 15 + 16) / 16 * 16 + 16) : 0;
    uint8_t *myring = rowring + static_cast<size_t>(warp) * 2 * slot_bytes;
    // lane 0 fetches row rr into slot `sl`: the 16-byte aligned window that holds its tokens
    auto fetch_row = [&](int64_t rr, int sl) {
        if (lane == 0) {
            const uint8_t *g = tokens + rr * row_stride;
            const int a = ANYALIGN ? static_cast<int>(reinterpret_cast<uintptr_t>(g) & 15u) : 0;
            const uint32_t nb = static_cast<uint32_t>((a + cols + 15) / 16 * 16);
            mbar_expect_tx(&rowbar[warp][sl], nb);
            bulk_g2s(myring + sl * slot_bytes, g - a, nb, &rowbar[warp][sl]);
        }
    };
    if (STAGED && gw < rows) fetch_row(gw, 0);
    int64_t off_next = gw < rows ? row_offs[gw] : 0;
    // (row_tail[r]: where the row's trailing run starts, with the run's kind -- <BOS> <EOS> <PAD> -- in bits 30..31)
    int32_t tail_next = (row_tail != nullptr && gw < rows) ? row_tail[gw] : 0;
    uint32_t it = 0;
    for (int64_t r = gw; r < rows; r += GW, ++it) {
        const int64_t off_r = off_next;
        const int32_t tail_r = tail_next;
        if (r + GW < rows) {  // the next row's output offset, hint and tokens: in flight while this row is decoded
            off_next = row_offs[r + GW];
            if (row_tail != nullptr) tail_next = row_tail[r + GW];
            if (STAGED) fetch_row(r + GW, (it + 1) & 1);
        }
        const uint8_t *gp = tokens + r * row_stride;
        const int ra = ANYALIGN ? static_cast<int>(reinterpret_cast<uintptr_t>(gp) & 15u) : 0;  // the row's misalignment: loads are aligned, tokens are shifted into place
        if (STAGED) mbar_wait_u32(smem_u32(&rowbar[warp][it & 1]), (it >> 1) & 1u);
        const uint8_t *rp = STAGED ? myring + (it & 1) * slot_bytes + ra : gp;  // (rp - ra is 16-byte aligned either way)
        uint8_t *dst = chars + off_r;
        int fill = static_cast<int>(reinterpret_cast<uintptr_t>(dst) & 15u);  // bytes of the stage in front of the data
        uint8_t *gal = dst - fill;                                             // aligned address of stage[0]
        int head = fill;                                                       // > 0: stage[0 .. head) is not ours
        int step = 128;
        // columns [cols_head, cols) are one repeated special (found by pass 1): written below as a pattern fill
        const int64_t cols_all = cols;
        const int64_t cols = row_tail != nullptr ? static_cast<int64_t>(tail_r & 0x3fffffff) : cols_all;
        // One 16-tokens-per-lane step in its byte-table form (tokens [c0, c0 + min(left, 512)) of the row, appended to the
        // stage at `fill`): false = the step does not have the shape this form handles, nothing was written.
        auto step16 = [&](int c0, int left, int &total) -> bool {
            const bool ragged = left < 512 && (left & 15) != 0;
            const int nact = min(32, (left + 15) >> 4);
            const int nlast = ragged ? (left & 15) : 16;  // tokens of the last active vector
            const bool act = lane < nact;
            uint4 x = make_uint4(0u, 0u, 0u, 0u);
            if (act) x = *reinterpret_cast<const uint4 *>(rp - ra + c0 + 16 * lane);
            if (ra != 0) {  // (warp-uniform) tokens of this lane: bytes [ra, ra + 16) of its vector and the next one
                uint4 nx;
                nx.x = __shfl_down_sync(0xffffffffu, x.x, 1); nx.y = __shfl_down_sync(0xffffffffu, x.y, 1);
                nx.z = __shfl_down_sync(0xffffffffu, x.z, 1); nx.w = __shfl_down_sync(0xffffffffu, x.w, 1);
                if (lane == nact - 1) {  // (the vector behind the last one is read only if the row reaches into it)
                    nx = make_uint4(0u, 0u, 0u, 0u);
                    if (c0 + 16 * nact < ra + cols_all) nx = *reinterpret_cast<const uint4 *>(rp - ra + c0 + 16 * nact);
                }
                x = shift16(x, nx, ra);
            }
            // The shape of nearly every step of a tokenised batch: plain text, possibly behind ONE special in the
            // very first position (the BOS that opens a row: one extra word "<BOS" in front, its '>' takes the
            // first byte of lane 0's first word), possibly with specials in the LAST active vector only (the EOS and
            // the first <PAD>s in front of the trailing run).  Lanes in front of that vector store four words each;
            // the last vector's 16 tokens are then laid down byte-wise by 16 lanes.  No scan.
            uint32_t w[4];
            w[0] = dec_lut4(lutbase, x.x); w[1] = dec_lut4(lutbase, x.y); w[2] = dec_lut4(lutbase, x.z); w[3] = dec_lut4(lutbase, x.w);
            const uint32_t spm = (w[0] | w[1] | w[2] | w[3]) & 0x80808080u;
            const uint32_t spb = __ballot_sync(0xffffffffu, act && spm != 0);
            const bool tail_emit = ragged || ((spb >> (nact - 1)) & 1u) != 0;  // warp-uniform
            // (ragged: the EOS sits in the last 16 BYTES of the head, which straddle the last two token vectors)
            const int nev = !tail_emit ? 0 : ((ragged && nact > 1) ? 2 : 1);  // vectors laid down byte-wise
            const int nwl = nact - nev;                                        // lanes that store whole words
            const uint32_t w00 = __shfl_sync(0xffffffffu, w[0], 0);
            const int lead = (nwl > 0 && (w00 & 0x80u)) ? 1 : 0;
            uint32_t rest = spm;
            if (lane == 0) rest = ((w[0] & 0xffffff00u) | w[1] | w[2] | w[3]) & 0x80808080u;
            if (__any_sync(0xffffffffu, lane < nwl && rest != 0)) return false;
            const int r8 = (fill & 3) * 8, kw = fill >> 2;
            uint32_t lo = __shfl_up_sync(0xffffffffu, w[3], 1);
            uint32_t w0 = w[0];
            if (lane == 0) {
                lo = r8 ? stage_w[kw] << (32 - r8) : 0u;
                if (lead) {
                    const uint32_t P = special_word(w00);
                    stage_w[kw] = __funnelshift_l(lo, P, r8);
                    lo = P;
                    w0 = (w0 & 0xffffff00u) | 0x3eu;
                }
            }
            uint32_t *d = stage_w + kw + lead + 4 * lane;
            if (lane < nwl) {
                d[0] = __funnelshift_l(lo, w0, r8);
                d[1] = __funnelshift_l(w0, w[1], r8);
                d[2] = __funnelshift_l(w[1], w[2], r8);
                d[3] = __funnelshift_l(w[2], w[3], r8);
                if (lane == nwl - 1 && r8) d[4] = w[3] >> (32 - r8);
            }
            total = 16 * nwl + 4 * lead;
            if (tail_emit) {
                __syncwarp();  // (the carry word above covers the first bytes written here)
                // lane t owns token t of the last vector(s)
                const int q = (lane >> 2) & 3, src = nwl + (lane >> 4);
                const uint32_t t0 = __shfl_sync(0xffffffffu, w[0], src), t1 = __shfl_sync(0xffffffffu, w[1], src);
                const uint32_t t2 = __shfl_sync(0xffffffffu, w[2], src), t3 = __shfl_sync(0xffffffffu, w[3], src);
                const uint32_t tw = q == 0 ? t0 : (q == 1 ? t1 : (q == 2 ? t2 : t3));
                const uint32_t c = (tw >> (8 * (lane & 3))) & 0xffu;
                const int nem = 16 * (nev - 1) + nlast;  // tokens laid down here
                const bool mine = lane < nem;
                const uint32_t sm = __ballot_sync(0xffffffffu, mine && (c & 0x80u));
                uint8_t *o = stage + fill + total + lane + 4 * __popc(sm & ((1u << lane) - 1u));
                if (mine) {
                    if (c & 0x80u) {
                        const int sp = static_cast<int>(c & 3u);
#pragma unroll
                        for (int j = 0; j < 5; ++j) o[j] = special_char(sp, j);
                    } else {
                        *o = static_cast<uint8_t>(c);
                    }
                }
                total += nem + 4 * __popc(sm);
            }
            return true;
        };
        // the stage's whole 16-byte vectors leave for global memory; what is left moves to its front
        auto flush = [&]() {
            const int nfull = fill >> 4;
            int vfirst = lane;
            if (head > 0 && nfull > 0) {  // first vector of the row: bytes [0, head) belong to the previous row
                if (lane >= head && lane < 16) gal[lane] = stage[lane];
                if (lane == 0) vfirst = 32;
            }
            {
                const uint4 *sv = reinterpret_cast<const uint4 *>(stage) + vfirst;
                uint4 *gv = reinterpret_cast<uint4 *>(gal) + vfirst;
                int left_v = nfull - vfirst;  // (a handful of trips: no unrolling, no remainder code)
#pragma unroll 1
                for (; left_v > 0; left_v -= 32, sv += 32, gv += 32) *gv = *sv;
            }
            if (nfull > 0) head = 0;
            const int rest = fill & 15;
            uint8_t keep = 0;
            if (lane < rest) keep = stage[16 * nfull + lane];
            __syncwarp();
            if (nfull > 0 && lane < rest) stage[lane] = keep;
            __syncwarp();
            gal += 16 * nfull;
            fill = rest;
        };
        // A row of a tokenised batch -- its head in front of the trailing run is at most two such steps -- goes into the
        // stage in one piece and is flushed once (the stage holds 2 x (512 + 4 + 5 x 32) bytes and the carry).
        int64_t c_begin = 0;
        bool try16 = bytelut;  // (a row whose step did not have the shape stops asking: rows without the hint hold <PAD> runs)
        if (bytelut && cols <= 1024) {
            const int h = static_cast<int>(cols);
            int c = 0, total = 0;
            while (c < h && step16(c, h - c, total)) {
                __syncwarp();
                fill += total;
                c += 512;
            }
            c_begin = min(c, h);
            try16 = c_begin >= h;
            if (c_begin > 0) flush();
        }
        for (int64_t c0 = c_begin; c0 < cols; c0 += step) {
            step = 128;
            int total;
            bool done = false;
            // Steps of plain text or of one repeated special (the <PAD> run behind a sequence) -- nearly all of
            // them -- are laid into the stage as whole 32-bit words shifted by the carry (fill & 3 bytes):
            // one shuffle and one funnel shift per word instead of a scan and a byte store per character.
            // 16 tokens per lane: a full step of 512, or the row's last step when what is left is a whole number of
            // 16-token vectors (always the case in front of a trailing run found by pass 1): lanes >= nact hold nothing
            // A ragged last vector (rows that are not 16-byte aligned: the head in front of the trailing run ends
            // where an ALIGNED vector ends) is taken by the byte-wise tail of the byte-table path only.
            const int64_t left = cols - c0;
            const bool ragged = left < 512 && (left & 15) != 0;
            if (fast && (!ragged || bytelut)) {
                if (try16 && left < (1ll << 30) && c0 < (1ll << 30) && step16(static_cast<int>(c0), static_cast<int>(min(left, static_cast<int64_t>(512))), total)) {
                    step = 512;
                    done = true;
                } else {
                    try16 = false;
                }
                if (!done && !ragged) {
                const int nact = static_cast<int>(min(static_cast<int64_t>(32), (left + 15) >> 4));
                const bool act = lane < nact;
                uint4 x = make_uint4(0u, 0u, 0u, 0u);
                if (act) x = *reinterpret_cast<const uint4 *>(rp - ra + c0 + 16 * lane);
                if (ra != 0) {  // (warp-uniform) tokens of this lane: bytes [ra, ra + 16) of its vector and the next one
                    uint4 nx;
                    nx.x = __shfl_down_sync(0xffffffffu, x.x, 1); nx.y = __shfl_down_sync(0xffffffffu, x.y, 1);
                    nx.z = __shfl_down_sync(0xffffffffu, x.z, 1); nx.w = __shfl_down_sync(0xffffffffu, x.w, 1);
                    if (lane == nact - 1) {
                        nx = make_uint4(0u, 0u, 0u, 0u);
                        if (c0 + 16 * nact < ra + cols_all) nx = *reinterpret_cast<const uint4 *>(rp - ra + c0 + 16 * nact);
                    }
                    x = shift16(x, nx, ra);
                }
                const uint32_t xs[4] = {x.x, x.y, x.z, x.w};
                uint32_t ee[16], any = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    ee[4 * k + 0] = inv[(xs[k] & 0xffu) + 128];
                    ee[4 * k + 1] = inv[__byte_perm(xs[k], 0, 0x4441) + 128];
                    ee[4 * k + 2] = inv[__byte_perm(xs[k], 0, 0x4442) + 128];
                    ee[4 * k + 3] = inv[(xs[k] >> 24) + 128];
                    any |= ee[4 * k] | ee[4 * k + 1] | ee[4 * k + 2] | ee[4 * k + 3];
                }
                if (!act) {  // nothing here: neither a special nor a different token for the votes below
                    any = 0;
#pragma unroll
                    for (int k = 0; k < 16; ++k) ee[k] = 0;
                }
                const uint32_t x0 = __shfl_sync(0xffffffffu, x.x, 0);
                // plain text, possibly behind ONE special in the very first position (the BOS that opens a row): that
                // special is one extra word in front ("<BOS") and its '>' takes the first byte of lane 0's first word
                uint32_t any_rest = any;
                if (lane == 0)
                    any_rest = ee[1] | ee[2] | ee[3] | ee[4] | ee[5] | ee[6] | ee[7] | ee[8] | ee[9] | ee[10] | ee[11] | ee[12] | ee[13] | ee[14] | ee[15];
                if (!__any_sync(0xffffffffu, (any_rest & 0x100u) != 0)) {
                    const uint32_t e00 = __shfl_sync(0xffffffffu, ee[0], 0);
                    const int lead = (e00 & 0x100u) ? 1 : 0;  // warp-uniform
                    uint32_t w[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        w[k] = pack4(ee[4 * k], ee[4 * k + 1], ee[4 * k + 2], ee[4 * k + 3]);
                    const int r8 = (fill & 3) * 8, kw = fill >> 2;
                    uint32_t lo = __shfl_up_sync(0xffffffffu, w[3], 1);
                    if (lane == 0) {
                        lo = r8 ? stage_w[kw] << (32 - r8) : 0u;
                        if (lead) {
                            const uint32_t P = special_word(e00);
                            stage_w[kw] = __funnelshift_l(lo, P, r8);
                            lo = P;
                            w[0] = (w[0] & 0xffffff00u) | 0x3eu;
                        }
                    }
                    uint32_t *d = stage_w + kw + lead + 4 * lane;
                    if (act) {
                        d[0] = __funnelshift_l(lo, w[0], r8);
                        d[1] = __funnelshift_l(w[0], w[1], r8);
                        d[2] = __funnelshift_l(w[1], w[2], r8);
                        d[3] = __funnelshift_l(w[2], w[3], r8);
                    }
                    if (lane == nact - 1 && r8) d[4] = w[3] >> (32 - r8);
                    total = 16 * nact + 4 * lead;
                } else if (__all_sync(0xffffffffu, !act || (x.x == x0 && x.x == __byte_perm(x.x, 0, 0x0000) && x.y == x.x && x.z == x.x && x.w == x.x))) {
                    const uint32_t e00 = __shfl_sync(0xffffffffu, ee[0], 0);
                    decode_fill_special(static_cast<int>(e00 & 3u), 16 * nact, patw, stage, fill, lane);
                    total = 80 * nact;
                } else {
                    total = decode_word_step<16>(ee, stage_w, fill, lane, nact);
                }
                step = 512;
                done = true;
                }
            }
            if (!done && fast && c0 + 128 <= cols) {
                uint32_t x = *reinterpret_cast<const uint32_t *>(rp - (ra & 3) + c0 + 4 * lane);
                if (ra & 3) {
                    uint32_t nx = __shfl_down_sync(0xffffffffu, x, 1);
                    if (lane == 31) nx = *reinterpret_cast<const uint32_t *>(rp - (ra & 3) + c0 + 128);
                    x = __funnelshift_r(x, nx, 8 * (ra & 3));
                }
                const uint32_t e0 = inv[(x & 0xffu) + 128], e1 = inv[__byte_perm(x, 0, 0x4441) + 128],
                               e2 = inv[__byte_perm(x, 0, 0x4442) + 128], e3 = inv[(x >> 24) + 128];
                const bool sp_here = ((e0 | e1 | e2 | e3) & 0x100u) != 0;
                const uint32_t x0 = __shfl_sync(0xffffffffu, x, 0);
                if (!__any_sync(0xffffffffu, sp_here)) {
                    const uint32_t w = pack4(e0, e1, e2, e3);
                    const int r8 = (fill & 3) * 8, kw = fill >> 2;
                    uint32_t lo = __shfl_up_sync(0xffffffffu, w, 1);
                    if (lane == 0) lo = r8 ? stage_w[kw] << (32 - r8) : 0u;
                    stage_w[kw + lane] = __funnelshift_l(lo, w, r8);
                    if (lane == 31 && r8) stage_w[kw + 32] = w >> (32 - r8);
                    total = 128;
                    done = true;
                } else if (__all_sync(0xffffffffu, x == x0 && x == __byte_perm(x, 0, 0x0000))) {
                    decode_fill_special(static_cast<int>(e0 & 3u), 128, patw, stage, fill, lane);
                    total = 640;
                    done = true;
                } else {
                    const uint32_t ee[4] = {e0, e1, e2, e3};
                    total = decode_word_step<4>(ee, stage_w, fill, lane);
                    done = true;
                }
            }
            if (!done) {
                uint32_t e[4];
                decode_fetch4(rp, itemsize, col_stride, c0 + 4 * lane, cols, inv, fast != 0 && (ra & 3) == 0, e);
                int mylen = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) mylen += e[k] >= 0xFFFEu ? 0 : ((e[k] & 0x100u) ? 5 : 1);
                int incl = mylen;
                for (int o = 1; o < 32; o <<= 1) {
                    const int y = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += y;
                }
                total = __shfl_sync(0xffffffffu, incl, 31);
                uint8_t *w = stage + fill + incl - mylen;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (e[k] >= 0xFFFEu) continue;
                    if (e[k] & 0x100u) {
                        const int sp = static_cast<int>(e[k] & 3u);  // <BOS> <EOS> <PAD>
#pragma unroll
                        for (int j = 0; j < 5; ++j) w[j] = special_char(sp, j);
                        w += 5;
                    } else {
                        *w++ = static_cast<uint8_t>(e[k]);
                    }
                }
            }
            __syncwarp();
            fill += total;
            flush();
        }
        if (cols < cols_all) {
            // The trailing run: 5 (cols_all - cols) bytes "<PAD><PAD>..." starting at gal[fill].  Period 5 against 16-byte
            // vectors: vector v of the run starts at phase (phase0 + v) % 5 (16 = 1 mod 5) -- one LDS.128 of the pattern
            // table and one st.global.v4 per 16 bytes, no token is read, nothing goes through the stage.
            const int k = static_cast<int>(static_cast<uint32_t>(tail_r) >> 30);  // (only rows with a hint get here)
            const int run = 5 * static_cast<int>(cols_all - cols);  // (cols <= 2^28 on this path)
            int done = 0;  // bytes of the run written so far
            if (fill > 0 || head > 0) {  // the vector that holds the staged bytes [head, fill): completed with the run's first bytes
                done = min(16 - fill, run);
                // (pat16[k][0][i] = character i % 5 of the special's text)
                if (lane >= head && lane < fill + done) gal[lane] = lane < fill ? stage[lane] : pat16[k][0][lane - fill];
                gal += 16;  // (if the run ended inside this vector there is nothing left to write)
            }
            const int left = run - done;
            const int nvec = left >> 4;
            const int phase0 = done >= 10 ? done - 10 : (done >= 5 ? done - 5 : done);  // done % 5, done <= 16
            const uint4 *pk = reinterpret_cast<const uint4 *>(&pat16[k][0][0]);
            // vector v starts at phase (phase0 + v) % 5: 30 lanes stride the run by 30 vectors, so a lane's phase -- its
            // 16 bytes -- never changes: one LDS.128 per row, then bare stores
            if (lane < 30) {
                const int phl = phase0 + lane5;  // lane5 = lane % 5
                const uint4 pv = pk[phl >= 5 ? phl - 5 : phl];
                uint4 *gv = reinterpret_cast<uint4 *>(gal) + lane;
                int left_v = nvec - lane;
#pragma unroll 1
                for (; left_v > 90; left_v -= 120, gv += 120) {
                    __stcs(gv, pv);
                    __stcs(gv + 30, pv);
                    __stcs(gv + 60, pv);
                    __stcs(gv + 90, pv);
                }
                if (left_v > 0) __stcs(gv, pv);
                if (left_v > 30) __stcs(gv + 30, pv);
                if (left_v > 60) __stcs(gv + 60, pv);
            }
            const int rest = left & 15;
            if (lane < rest) gal[16 * static_cast<int64_t>(nvec) + lane] = pat16[k][(phase0 + nvec) % 5][lane];
            fill = 0;
            head = 0;
        }
        // the row's last partial vector
        for (int i = head + lane; i < fill; i += 32) gal[i] = stage[i];
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// host-side launch helpers
// ------------------------------------------------------------------------------------------
namespace {

inline uint32_t rep4(uint32_t b) { return (b & 0xffu) * 0x01010101u; }

}  // namespace

// mode 0: batch-first one-byte tokens (codes are the output bytes: ids wrap to 8 bits like
//         the reference's int -> int8 store);
// mode 1: tokens through Expand (wide element types / tile kernels);
// mode 2: one-hot columns through Expand.
Prepared prepare(const bsq_tokenizer &tok, int mode) {
    Prepared p;
    uint8_t codes[256];
    const bool onehot = mode == 2;
    for (int b = 0; b < 256; ++b) {
        const int id = b < 0x80 ? tok.lut[b] : -1;  // bytes >= 0x80: undefined in the reference, invalid here
        codes[b] = id >= 0 ? static_cast<uint8_t>(id) : (onehot ? kCodeInvalid : 0);
    }
    std::memcpy(p.lut.w, codes, 256);
    p.sp.bos = tok.bos_id >= 0;
    p.sp.eos = tok.eos_id >= 0;
    const bool fits = tok.pad_id < 0x80;  // every special id is a valid direct code
    uint32_t bos_c, eos_c, pad_c;
    if (mode == 0) {
        bos_c = static_cast<uint32_t>(tok.bos_id);
        eos_c = static_cast<uint32_t>(tok.eos_id);
        pad_c = tok.padchar ? static_cast<uint32_t>(tok.pad_id) : 0u;
    } else {
        bos_c = fits ? static_cast<uint32_t>(tok.bos_id) : kCodeBos;
        eos_c = fits ? static_cast<uint32_t>(tok.eos_id) : kCodeEos;
        if (tok.padchar) pad_c = fits ? static_cast<uint32_t>(tok.pad_id) : kCodePad;
        else pad_c = onehot ? kCodeInvalid : 0u;
    }
    p.sp.bos_w = rep4(bos_c);
    p.sp.eos_w = rep4(eos_c);
    p.sp.pad_w = rep4(pad_c);
    p.ex.map[0] = tok.padchar ? tok.pad_id : (onehot ? -1 : 0);
    p.ex.map[1] = tok.eos_id;
    p.ex.map[2] = tok.bos_id;
    p.ex.map[3] = onehot ? -1 : 0;
    return p;
}

namespace {

int check_common(int device, int64_t nseq, int64_t padlen, const bsq_tokenizer *tok, int kind, const void *d_out) {
    if (tok == nullptr) return fail(BSQ_ERR_ARG, "null tokenizer");
    if (padlen <= 0) return fail(BSQ_ERR_ARG, "batch tokenize requires padlen is provded.");  // src/tokenize.h:383
    if (padlen > (1ll << 30)) return fail(BSQ_ERR_ARG, "padlen above 2^30 is not supported");
    if (nseq < 0) return fail(BSQ_ERR_ARG, "negative batch size");
    if (bsq_kind_size(kind) == 0) return fail(BSQ_ERR_ARG, "invalid element kind");
    if (nseq > 0 && (d_out == nullptr || (reinterpret_cast<uintptr_t>(d_out) & 15u)))
        return fail(BSQ_ERR_ARG, "output pointer must be non-null and 16-byte aligned");
    BSQ_CUDA_TRY(cudaSetDevice(device));
    return BSQ_OK;
}

template <typename T>
int launch_bf(cudaStream_t st, const SeqView &v, int64_t nseq, int64_t /*ld*/, int64_t padlen, const bsq_tokenizer &tok, void *d_out,
              int64_t first_off) {
    // one-byte tokens: the codes are the output bytes (ids wrap to 8 bits like the reference's
    // int -> int8 store); wider types expand codes through Expand.
    const Prepared p = prepare(tok, sizeof(T) == 1 ? 0 : 1);
    if (sizeof(T) == 1 && span_kernel_applicable(padlen)) {
        int dev = 0;
        BSQ_CUDA_TRY(cudaGetDevice(&dev));
        return launch_tokenize_span(dev, st, v, nseq, padlen, p, static_cast<uint8_t *>(d_out));
    }
    if (sizeof(T) == 1 || (padlen * sizeof(T)) % 16 == 0) {
        int lanes_log2 = 0;  // lanes per row: smallest power of two covering the row, at most a warp
        while (lanes_log2 < 5 && (16ll << lanes_log2) < padlen + (sizeof(T) == 1 ? 15 : 0)) ++lanes_log2;
        const int64_t rows_per_block = static_cast<int64_t>(kThreads / 32) * (32 >> lanes_log2);
        const int64_t blocks = (nseq + rows_per_block - 1) / rows_per_block;
        if (blocks > 0x7fffffffll) return fail(BSQ_ERR_ARG, "batch too large for one launch");
        const bool aligned = sizeof(T) != 1 || padlen % 16 == 0;
        const unsigned nb = static_cast<unsigned>(blocks);
        T *o = static_cast<T *>(d_out);
        const int pl = static_cast<int>(padlen);
        if (lanes_log2 == 5 && aligned)
            tokenize_rows_kernel<T, true, true><<<nb, kThreads, 0, st>>>(v, nseq, pl, lanes_log2, p.lut, p.sp, p.ex, o);
        else if (lanes_log2 == 5)
            tokenize_rows_kernel<T, true, false><<<nb, kThreads, 0, st>>>(v, nseq, pl, lanes_log2, p.lut, p.sp, p.ex, o);
        else if (aligned)
            tokenize_rows_kernel<T, false, true><<<nb, kThreads, 0, st>>>(v, nseq, pl, lanes_log2, p.lut, p.sp, p.ex, o);
        else
            tokenize_rows_kernel<T, false, false><<<nb, kThreads, 0, st>>>(v, nseq, pl, lanes_log2, p.lut, p.sp, p.ex, o);
    } else {
        constexpr int TPT = 16 / sizeof(T);
        const int64_t total = nseq * padlen;
        const int64_t per_block = static_cast<int64_t>(kThreads) * TPT;
        const int64_t blocks = (total + per_block - 1) / per_block;
        if (blocks > 0x7fffffffll) return fail(BSQ_ERR_ARG, "batch too large for one launch");
        tokenize_flat_kernel<T><<<static_cast<unsigned>(blocks), kThreads, 0, st>>>(
            v, nseq, static_cast<int>(padlen), make_fastdiv(static_cast<uint32_t>(padlen)), p.lut, p.sp, p.ex,
            static_cast<T *>(d_out));
    }
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}

template <typename T, bool ONEHOT>
int launch_sf(cudaStream_t st, const SeqView &v, int64_t nseq, int64_t ld, int64_t padlen, const bsq_tokenizer &tok, void *d_out,
              int64_t /*first_off*/) {
    const Prepared p = prepare(tok, ONEHOT ? 2 : 1);
    const int64_t gx = (nseq + kTileSeqs - 1) / kTileSeqs, gy = (padlen + kTilePos - 1) / kTilePos;
    if (gx > 0x7fffffffll || gy > 65535) return fail(BSQ_ERR_ARG, "batch too large for one launch");
    const dim3 grid(static_cast<unsigned>(gx), static_cast<unsigned>(gy));
    const int ncols = ONEHOT ? tok.alphabet_size : 1;
    const FastDiv dc = make_fastdiv(static_cast<uint32_t>(ncols));
    const bool aligned = (reinterpret_cast<uintptr_t>(d_out) & 15u) == 0;
    T *o = static_cast<T *>(d_out);
    const int pl = static_cast<int>(padlen);
    const size_t smem = static_cast<size_t>(kTileSeqs) * kStagePitch * (v.mask != nullptr ? 2 : 1);  // staged residues (+ mask)
    const int64_t row_bytes = static_cast<int64_t>(ncols) * sizeof(T);
    const FastDiv drb = make_fastdiv(static_cast<uint32_t>(row_bytes));
    // (with a mask the two staging areas + the static tile exceed the 48 KB a kernel gets without opting in)
#define BSQ_SF(MODE)                                                                                                        \
    do {                                                                                                                    \
        if (v.mask != nullptr)                                                                                              \
            BSQ_CUDA_TRY(cudaFuncSetAttribute(seqfirst_kernel<T, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,        \
                                              static_cast<int>(smem)));                                                     \
        seqfirst_kernel<T, MODE><<<grid, kThreads, smem, st>>>(v, nseq, ld, pl, p.lut, p.sp, p.ex, ncols, dc, drb, o);      \
    } while (0)
    if (!ONEHOT) {
        // the register-transpose path needs one-byte elements whose rows start 16-byte aligned and
        // codes that are the output bytes (every alphabet but BYTES, whose special ids exceed 8 bits)
        if (sizeof(T) == 1 && aligned && ld % 16 == 0 && tok.pad_id < 0x80) {
            if (gx * gy > 0x7fffffffll) return fail(BSQ_ERR_ARG, "batch too large for one launch");
            else if (gy % 2 == 0 && gx * gy / 2 >= 8ll * cur_sms() * 6)  // enough CTAs left to balance the resident slots (6 per SM)
                seqfirst_tok8_kernel<2><<<static_cast<unsigned>(gx * gy / 2), kThreads, 0, st>>>(
                    v, nseq, ld, pl, make_fastdiv(static_cast<uint32_t>(gy / 2)), p.lut, p.sp, reinterpret_cast<uint8_t *>(o));
            else seqfirst_tok8_kernel<1><<<static_cast<unsigned>(gx * gy), kThreads, 0, st>>>(
                    v, nseq, ld, pl, make_fastdiv(static_cast<uint32_t>(gy)), p.lut, p.sp, reinterpret_cast<uint8_t *>(o));
        }
        else BSQ_SF(kTokGeneric);
    } else {
        // 16-byte stores need every row of the (padlen, ld, ncols) array and this launch's first
        // column to start on a 16-byte boundary (tiles are 128 sequences wide, so then every run does)
        const bool vec_ok = aligned && (ld * row_bytes) % 16 == 0;  // every tile's run starts on a 16-byte boundary
        if (aligned && row_bytes == 16) BSQ_SF(kOhRow);
        else if (vec_ok && tok.pad_id < 0x80) BSQ_SF(kOhVec);  // (BYTES alphabet: ids need the Expand table)
        else if (aligned && (row_bytes == 4 || row_bytes == 8)) BSQ_SF(kOhRow);
        else BSQ_SF(kOhScalar);
    }
#undef BSQ_SF
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}

// one-byte tokens, contiguous along the row (any alignment: the kernels load aligned words and shift)
int decode_fast_path(const void * /*d_tokens*/, int itemsize, int64_t /*row_stride*/, int64_t col_stride) {
    return itemsize == 1 && col_stride == 1;
}
unsigned decode_grid(int64_t rows, int ctas_per_sm = 8) {  // persistent: one warp per row, rows dealt round-robin
    return static_cast<unsigned>(std::min<int64_t>((rows + kDecWarps - 1) / kDecWarps, static_cast<int64_t>(cur_sms()) * ctas_per_sm));
}

InvParam make_inv(const bsq_tokenizer &tok) {
    InvParam inv;
    for (int i = 0; i < 512; ++i) inv.e[i] = kInvNone;
    for (int b = 255; b >= 0; --b) inv.e[static_cast<int>(tok.lut[b]) + 128] = static_cast<uint16_t>(b);  // lowest byte wins
    if (tok.bos_id >= 0) inv.e[tok.bos_id + 128] = 0x100;
    if (tok.eos_id >= 0) inv.e[tok.eos_id + 128] = 0x101;
    if (tok.padchar) inv.e[tok.pad_id + 128] = 0x102;
    // Negative ids of the BYTES alphabet would decode to single bytes >= 0x80, which the
    // reference then fails to turn into a Python str (invalid UTF-8); treated as invalid.
    if (tok.nchars == 256)
        for (int i = 0; i < 128; ++i) inv.e[i] = kInvNone;
    return inv;
}

}  // namespace

#define BSQ_DISPATCH(FN, ...)                                                               \
    switch (kind) {                                                                         \
        case BSQ_I8: return FN<int8_t __VA_ARGS__>(st, v, nseq, ld, padlen, tok, d_out, first_off);    \
        case BSQ_I16: return FN<int16_t __VA_ARGS__>(st, v, nseq, ld, padlen, tok, d_out, first_off);  \
        case BSQ_I32: return FN<int32_t __VA_ARGS__>(st, v, nseq, ld, padlen, tok, d_out, first_off);  \
        case BSQ_I64: return FN<int64_t __VA_ARGS__>(st, v, nseq, ld, padlen, tok, d_out, first_off);  \
        case BSQ_F32: return FN<float __VA_ARGS__>(st, v, nseq, ld, padlen, tok, d_out, first_off);    \
        default: return FN<double __VA_ARGS__>(st, v, nseq, ld, padlen, tok, d_out, first_off);        \
    }
#define BSQ_COMMA_FALSE , false
#define BSQ_COMMA_TRUE , true

int launch_tokenize(cudaStream_t st, const uint8_t *d_bytes, const int64_t *d_offs, int64_t nseq, int64_t ld,
                    int64_t padlen, const bsq_tokenizer &tok, int batch_first, int kind, void *d_out, int64_t first_off) {
    if (nseq <= 0) return BSQ_OK;
    const SeqView v{d_bytes, d_offs, nullptr};
    if (batch_first) {
        BSQ_DISPATCH(launch_bf)
    } else {
        BSQ_DISPATCH(launch_sf, BSQ_COMMA_FALSE)
    }
}

int launch_onehot(cudaStream_t st, const uint8_t *d_bytes, const int64_t *d_offs, const uint8_t *d_mask, int64_t nseq,
                  int64_t ld, int64_t padlen, const bsq_tokenizer &tok, int kind, void *d_out) {
    if (nseq <= 0) return BSQ_OK;
    if (static_cast<int64_t>(kTileSeqs) * tok.alphabet_size > 0x7fffffffll) return fail(BSQ_ERR_ARG, "alphabet too large");
    const SeqView v{d_bytes, d_offs, d_mask};
    const int64_t first_off = -1;
    BSQ_DISPATCH(launch_sf, BSQ_COMMA_TRUE)
}

int check_launch_args(int device, int64_t nseq, int64_t padlen, const bsq_tokenizer *tok, int kind, const void *d_out) {
    return check_common(device, nseq, padlen, tok, kind, d_out);
}

}  // namespace bsq

using namespace bsq;

extern "C" {

int bsq_tokenize(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq,
                 int64_t padlen, const bsq_tokenizer *tok, int batch_first, int kind, void *d_out) {
    bsq::DeviceRestore restore_device;
    if (int rc = check_common(device, nseq, padlen, tok, kind, d_out)) return rc;
    if (nseq == 0) return BSQ_OK;
    if (d_offsets == nullptr) return fail(BSQ_ERR_ARG, "null offsets");
    return launch_tokenize(static_cast<cudaStream_t>(stream), d_bytes, d_offsets, nseq, nseq, padlen, *tok, batch_first,
                           kind, d_out, /*first_off=*/-1);
}

int bsq_tokenize_many(int device, void *stream, int nbatch, const uint8_t *const *d_bytes, const int64_t *const *d_offsets,
                      const int64_t *nseq, int64_t padlen, const bsq_tokenizer *tok, int batch_first, int kind, void *const *d_out) {
    bsq::DeviceRestore restore_device;
    if (nbatch < 0 || (nbatch > 0 && (d_bytes == nullptr || d_offsets == nullptr || nseq == nullptr || d_out == nullptr)))
        return fail(BSQ_ERR_ARG, "bad batch arguments");
    for (int k = 0; k < nbatch; ++k) {
        if (int rc = check_common(device, nseq[k], padlen, tok, kind, d_out[k])) return rc;
        if (nseq[k] > 0 && d_offsets[k] == nullptr) return fail(BSQ_ERR_ARG, "null offsets");
    }
    if (nbatch == 0) return BSQ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (batch_first && bsq_kind_size(kind) == 1 && span_kernel_applicable(padlen)) {
        const Prepared p = prepare(*tok, 0);
        for (int k0 = 0; k0 < nbatch; k0 += kSpanManyMax) {  // one launch per group of up to 32 batches
            const int nb = std::min(kSpanManyMax, nbatch - k0);
            if (int rc = launch_tokenize_span_many(device, st, nb, d_bytes + k0, d_offsets + k0, nseq + k0, padlen, p,
                                                   reinterpret_cast<uint8_t *const *>(d_out + k0)))
                return rc;
        }
        return BSQ_OK;
    }
    for (int k = 0; k < nbatch; ++k)  // layouts / element types without a multi-batch kernel: one launch each
        if (int rc = launch_tokenize(st, d_bytes[k], d_offsets[k], nseq[k], nseq[k], padlen, *tok, batch_first, kind, d_out[k], -1)) return rc;
    return BSQ_OK;
}

int bsq_onehot(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, const uint8_t *d_mask,
               int64_t nseq, int64_t padlen, const bsq_tokenizer *tok, int kind, void *d_out) {
    bsq::DeviceRestore restore_device;
    if (int rc = check_common(device, nseq, padlen, tok, kind, d_out)) return rc;
    if (nseq == 0) return BSQ_OK;
    if (d_offsets == nullptr) return fail(BSQ_ERR_ARG, "null offsets");
    return launch_onehot(static_cast<cudaStream_t>(stream), d_bytes, d_offsets, d_mask, nseq, nseq, padlen, *tok, kind,
                         d_out);
}

}  // extern "C"

namespace bsq {

// Scratch for the entry points that need a few words of device workspace (offsets reductions, decode
// scan).  A library-owned memory pool per device with an unbounded release threshold: the default
// pool hands its memory back to the driver at every synchronisation that finds it empty, which made
// each of these calls pay a fresh physical allocation (measured: decode 1.07 ms -> 11.6 ms per call).
int scratch_alloc(int device, void **p, size_t bytes, cudaStream_t st) {
    static std::mutex mu;
    static cudaMemPool_t pools[64] = {};
    if (device < 0 || device >= 64) return fail(BSQ_ERR_ARG, "bad device index");
    cudaMemPool_t pool;
    {
        std::lock_guard<std::mutex> g(mu);
        if (pools[device] == nullptr) {
            cudaMemPoolProps props = {};
            props.allocType = cudaMemAllocationTypePinned;
            props.handleTypes = cudaMemHandleTypeNone;
            props.location.type = cudaMemLocationTypeDevice;
            props.location.id = device;
            BSQ_CUDA_TRY(cudaMemPoolCreate(&pools[device], &props));
            uint64_t keep = ~0ull;
            BSQ_CUDA_TRY(cudaMemPoolSetAttribute(pools[device], cudaMemPoolAttrReleaseThreshold, &keep));
        }
        pool = pools[device];
    }
    BSQ_CUDA_TRY(cudaMallocFromPoolAsync(p, bytes, pool, st));
    return BSQ_OK;
}

int offsets_error(unsigned long long bits) {
    if (bits & 1u) return fail(BSQ_ERR_ARG, "offsets must be non-decreasing");
    if (bits & 2u) return fail(BSQ_ERR_ARG, "offsets must start at or after 0");
    if (bits & 4u) return fail(BSQ_ERR_ARG, "offsets run past the end of bytes");
    return BSQ_OK;
}

}  // namespace bsq

extern "C" {

int bsq_check_offsets_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t nbytes, int64_t padlen,
                             const bsq_tokenizer *tok) {
    bsq::DeviceRestore restore_device;
    if (tok == nullptr) return fail(BSQ_ERR_ARG, "null tokenizer");
    if (padlen <= 0) return fail(BSQ_ERR_ARG, "batch tokenize requires padlen is provded.");
    if (nseq <= 0) return BSQ_OK;
    Extent e{};
    if (int rc = reduce_offsets_device(device, static_cast<cudaStream_t>(stream), d_offsets, nseq, nbytes, CropCount{kI64Max}, &e)) return rc;
    const int64_t tl = e.max + (tok->bos_id >= 0) + (tok->eos_id >= 0);
    if (tl > padlen)
        return fail(BSQ_ERR_TOO_LONG, "seq len + bos + eos > padlen: " + std::to_string(tl) + ", vs padlen " + std::to_string(padlen));
    return BSQ_OK;
}

int bsq_varlen_extent_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t nbytes,
                             const bsq_tokenizer *tok, int64_t *total, int64_t *max_seqlen) {
    bsq::DeviceRestore restore_device;
    if (tok == nullptr || total == nullptr || max_seqlen == nullptr) return fail(BSQ_ERR_ARG, "null argument");
    if (nseq < 0 || (nseq > 0 && d_offsets == nullptr)) return fail(BSQ_ERR_ARG, "bad offsets");
    *total = *max_seqlen = 0;
    if (nseq == 0) return BSQ_OK;
    Extent e{};
    if (int rc = reduce_offsets_device(device, static_cast<cudaStream_t>(stream), d_offsets, nseq, nbytes, CropCount{kI64Max}, &e)) return rc;
    const int64_t k = (tok->bos_id >= 0) + (tok->eos_id >= 0);
    *total = e.sum0 + nseq * k;
    *max_seqlen = e.max + k;
    return BSQ_OK;
}

int bsq_crop_extent_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t nbytes, int64_t crop_len,
                           int64_t *total, int64_t *max_len) {
    bsq::DeviceRestore restore_device;
    if (total == nullptr || max_len == nullptr) return fail(BSQ_ERR_ARG, "null argument");
    if (crop_len < 1) return fail(BSQ_ERR_ARG, "crop_len must be >= 1");
    if (nseq < 0 || (nseq > 0 && d_offsets == nullptr)) return fail(BSQ_ERR_ARG, "bad offsets");
    *total = *max_len = 0;
    if (nseq == 0) return BSQ_OK;
    Extent e{};
    if (int rc = reduce_offsets_device(device, static_cast<cudaStream_t>(stream), d_offsets, nseq, nbytes, CropCount{crop_len}, &e)) return rc;
    *total = e.sum0;
    *max_len = e.max;
    return BSQ_OK;
}

int bsq_check_lengths_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t padlen,
                             const bsq_tokenizer *tok) {
    return bsq_check_offsets_device(device, stream, d_offsets, nseq, -1, padlen, tok);
}

}  // extern "C"

namespace {

// pass 1 + scan, enqueued on `st`: d_row_offsets[0 .. rows] and d_row_tail are final when the stream gets there;
// {first bad token, total} land in *host_pair (pinned) with the last kernel.  *d_work_out is to be freed by the caller.
int decode_lengths_enqueue(int device, cudaStream_t st, const void *d_tokens, int itemsize, int64_t rows, int64_t cols,
                           int64_t row_stride, int64_t col_stride, const bsq_tokenizer *tok, int64_t *d_row_offsets,
                           int32_t *d_row_tail, int64_t **host_pair, int64_t **d_work_out) {
    const int64_t nblocks = (rows + kScanBlock - 1) / kScanBlock;
    int64_t *d_work = nullptr;  // [0] first_bad, [1] grand total, [2..] block totals
    if (int rc = scratch_alloc(device, reinterpret_cast<void **>(&d_work), sizeof(int64_t) * (2 + nblocks), st)) return rc;
    *d_work_out = d_work;
    BSQ_CUDA_TRY(cudaMemsetAsync(d_work, 0xff, sizeof(int64_t), st));
    const InvParam inv = make_inv(*tok);
    const int fast = decode_fast_path(d_tokens, itemsize, row_stride, col_stride);
    const bool rows16 = (reinterpret_cast<uintptr_t>(d_tokens) & 15u) == 0 && row_stride % 16 == 0;
    const bool al = rows16 && cols % 16 == 0;
    const int64_t maxvec = al ? cols / 16 : (15 + cols + 15) / 16;  // vectors that cover a row, at the worst alignment
    if (fast && cols > 0) {
        const uint8_t *tk = static_cast<const uint8_t *>(d_tokens);
        unsigned long long *fb = reinterpret_cast<unsigned long long *>(d_work);
        const unsigned grid = decode_grid(rows);
        // ids laid out [0, a) characters, [a, b) specials, [b, 256) nothing with b <= 128: classes by comparison
        int a = 0, b = 0;
        while (a < 256 && inv.e[a + 128] != kInvNone && !(inv.e[a + 128] & 0x100u)) ++a;
        b = a;
        while (b < 256 && inv.e[b + 128] != kInvNone && (inv.e[b + 128] & 0x100u)) ++b;
        bool thr = b >= 1 && b <= 128;
        for (int t = b; t < 256 && thr; ++t) thr = inv.e[t + 128] == kInvNone;
        const uint32_t lo4 = static_cast<uint32_t>(a) * 0x01010101u, hi4 = static_cast<uint32_t>(b) * 0x01010101u;
#define BSQ_LEN16P(AL, V)                                                                                                                      \
    do {                                                                                                                                       \
        if (thr) decode_len16p_kernel<AL, V, true><<<grid, kDecWarps * 32, 0, st>>>(tk, rows, cols, row_stride, inv, d_row_offsets, d_row_tail, fb, lo4, hi4);  \
        else decode_len16p_kernel<AL, V, false><<<grid, kDecWarps * 32, 0, st>>>(tk, rows, cols, row_stride, inv, d_row_offsets, d_row_tail, fb, lo4, hi4); \
    } while (0)
        if (maxvec <= 64) {
            if (al) BSQ_LEN16P(false, 2);
            else BSQ_LEN16P(true, 2);
        } else if (maxvec <= 96) {  // (padlen 1026, rows at any alignment: 66 vectors)
            if (al) BSQ_LEN16P(false, 3);
            else BSQ_LEN16P(true, 3);
        } else if (maxvec <= 128) {
            if (al) BSQ_LEN16P(false, 4);
            else BSQ_LEN16P(true, 4);
#undef BSQ_LEN16P
        } else if (al) {
            decode_len16_kernel<false><<<grid, kDecWarps * 32, 0, st>>>(tk, rows, cols, row_stride, inv, d_row_offsets, d_row_tail, fb);
        } else {
            decode_len16_kernel<true><<<grid, kDecWarps * 32, 0, st>>>(tk, rows, cols, row_stride, inv, d_row_offsets, d_row_tail, fb);
        }
    } else if (fast) {
        decode_len16_kernel<true><<<decode_grid(rows), kDecWarps * 32, 0, st>>>(
            static_cast<const uint8_t *>(d_tokens), rows, cols, row_stride, inv, d_row_offsets, d_row_tail, reinterpret_cast<unsigned long long *>(d_work));
    } else {
        // (wide / strided tokens: no trailing-run hint; "cols" = nothing to fill)
        if (d_row_tail != nullptr) fill_i32_kernel<<<static_cast<unsigned>((rows + 255) / 256), 256, 0, st>>>(d_row_tail, rows, static_cast<int32_t>(cols));
        decode_len_kernel<<<decode_grid(rows), kDecWarps * 32, 0, st>>>(
            static_cast<const uint8_t *>(d_tokens), itemsize, rows, cols, row_stride, col_stride, fast, inv, d_row_offsets,
            reinterpret_cast<unsigned long long *>(d_work));
    }
    // one pinned result slot per host thread (the calls are synchronous)
    // (16 bytes, never freed: a destructor would run at thread exit, possibly after the CUDA runtime is torn down)
    struct PinnedPair {
        int64_t *p = nullptr;
    };
    static thread_local PinnedPair pinned;
    if (pinned.p == nullptr) BSQ_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&pinned.p), 2 * sizeof(int64_t), cudaHostAllocPortable));
    *host_pair = pinned.p;
    scan_local_kernel<<<static_cast<unsigned>(nblocks), kScanBlock, 0, st>>>(d_row_offsets, rows, d_work + 2);
    if (nblocks <= 4096) {  // (up to 4 M rows: two kernels instead of three)
        scan_add_direct_kernel<<<static_cast<unsigned>(nblocks), kScanBlock, 0, st>>>(d_row_offsets, rows, d_work + 2, d_work, pinned.p);
        count_launch(3);
        BSQ_CUDA_TRY(cudaGetLastError());
        return BSQ_OK;
    }
    scan_totals_kernel<<<1, kScanBlock, 0, st>>>(d_work + 2, nblocks, d_work + 1);
    scan_add_kernel<<<static_cast<unsigned>(nblocks), kScanBlock, 0, st>>>(d_row_offsets, rows, d_work + 2, d_work + 1, d_work, pinned.p);
    count_launch(4);
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}

// after the stream synchronize: the reference's error for a token without an entry, or the total
int decode_lengths_finish(cudaStream_t st, const void *d_tokens, int itemsize, int64_t cols, int64_t row_stride, int64_t col_stride,
                          const int64_t *host_pair, int64_t *d_work, int64_t *total_chars) {
    const int64_t h[2] = {host_pair[0], host_pair[1]};
    if (h[0] != -1) {  // fetch the offending value for the reference's message
        const int64_t r = h[0] / cols, c = h[0] % cols;
        uint64_t raw = 0;
        BSQ_CUDA_TRY(cudaMemcpy(&raw, static_cast<const uint8_t *>(d_tokens) + r * row_stride + c * col_stride, itemsize,
                                cudaMemcpyDeviceToHost));
        BSQ_CUDA_TRY(cudaFreeAsync(d_work, st));
        return fail(BSQ_ERR_BAD_TOKEN, "Unexpected/invalid token " + std::to_string(static_cast<uint32_t>(raw)));
    }
    BSQ_CUDA_TRY(cudaFreeAsync(d_work, st));
    *total_chars = h[1];
    return BSQ_OK;
}

int decode_chars_enqueue(cudaStream_t st, const void *d_tokens, int itemsize, int64_t rows, int64_t cols, int64_t row_stride,
                         int64_t col_stride, const bsq_tokenizer *tok, const int64_t *d_row_offsets, const int32_t *d_row_tail,
                         uint8_t *d_chars, int64_t capacity, const unsigned long long *d_first_bad) {
    const InvParam inv = make_inv(*tok);
    const int fast = decode_fast_path(d_tokens, itemsize, row_stride, col_stride);
    const bool rows16 = (reinterpret_cast<uintptr_t>(d_tokens) & 15u) == 0 && row_stride % 16 == 0;
    // (a grid of only the 4 resident CTAs per SM measured slower: 470 vs 442 us)
    const int32_t *tail = (fast && cols <= (1 << 28)) ? d_row_tail : nullptr;  // (the run's byte count is an int in the kernel)
    const uint8_t *tk = static_cast<const uint8_t *>(d_tokens);
    const size_t ring = static_cast<size_t>(kDecWarps) * 2 * ((cols + 15 + 16) / 16 * 16 + 16);
    if (fast && ring <= 96 * 1024) {  // rows up to ~6 K tokens ride the ring
        auto kern = rows16 ? decode_chars_kernel<false, true> : decode_chars_kernel<true, true>;
        if (ring > 24 * 1024) BSQ_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        kern<<<decode_grid(rows), kDecWarps * 32, ring, st>>>(tk, itemsize, rows, cols, row_stride, col_stride, fast, inv, d_row_offsets, tail, d_chars, capacity, d_first_bad);
    } else if (fast && rows16) {
        decode_chars_kernel<false, false><<<decode_grid(rows), kDecWarps * 32, 0, st>>>(tk, itemsize, rows, cols, row_stride, col_stride, fast, inv,
                                                                                         d_row_offsets, tail, d_chars, capacity, d_first_bad);
    } else {
        decode_chars_kernel<true, false><<<decode_grid(rows), kDecWarps * 32, 0, st>>>(tk, itemsize, rows, cols, row_stride, col_stride, fast, inv,
                                                                                        d_row_offsets, tail, d_chars, capacity, d_first_bad);
    }
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}

int decode_args_check(const bsq_tokenizer *tok, int itemsize, int64_t rows, int64_t cols) {
    if (tok == nullptr) return fail(BSQ_ERR_ARG, "null argument");
    if (itemsize != 1 && itemsize != 2 && itemsize != 4 && itemsize != 8)
        return fail(BSQ_ERR_ARG, "Unexpected itemsize: expected 1, 2, 4, or 8. Found " + std::to_string(itemsize));  // src/tokenize.h:123
    if (rows < 0 || cols < 0 || rows > 0x7fffffffll) return fail(BSQ_ERR_ARG, "bad decode shape");
    return BSQ_OK;
}

}  // namespace

extern "C" {

int bsq_decode_lengths(int device, void *stream, const void *d_tokens, int itemsize, int64_t rows, int64_t cols,
                       int64_t row_stride, int64_t col_stride, const bsq_tokenizer *tok, int64_t *d_row_offsets,
                       int32_t *d_row_tail, int64_t *total_chars) {
    bsq::DeviceRestore restore_device;
    if (total_chars == nullptr) return fail(BSQ_ERR_ARG, "null argument");
    if (int rc = decode_args_check(tok, itemsize, rows, cols)) return rc;
    *total_chars = 0;
    BSQ_CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (rows == 0) {
        BSQ_CUDA_TRY(cudaMemsetAsync(d_row_offsets, 0, sizeof(int64_t), st));
        return BSQ_OK;
    }
    if (d_tokens == nullptr && cols > 0) return fail(BSQ_ERR_ARG, "Empty array cannot yield a decoded string");  // src/tokenize.h:133
    int64_t *host_pair = nullptr, *d_work = nullptr;
    if (int rc = decode_lengths_enqueue(device, st, d_tokens, itemsize, rows, cols, row_stride, col_stride, tok, d_row_offsets, d_row_tail,
                                        &host_pair, &d_work))
        return rc;
    BSQ_CUDA_TRY(cudaStreamSynchronize(st));
    return decode_lengths_finish(st, d_tokens, itemsize, cols, row_stride, col_stride, host_pair, d_work, total_chars);
}

int bsq_decode_chars(int device, void *stream, const void *d_tokens, int itemsize, int64_t rows, int64_t cols,
                     int64_t row_stride, int64_t col_stride, const bsq_tokenizer *tok, const int64_t *d_row_offsets,
                     const int32_t *d_row_tail, uint8_t *d_chars) {
    bsq::DeviceRestore restore_device;
    if (tok == nullptr) return fail(BSQ_ERR_ARG, "null tokenizer");
    if (itemsize != 1 && itemsize != 2 && itemsize != 4 && itemsize != 8) return fail(BSQ_ERR_ARG, "bad itemsize");
    if (rows <= 0 || cols <= 0) return BSQ_OK;
    if (rows > 0x7fffffffll) return fail(BSQ_ERR_ARG, "bad decode shape");
    BSQ_CUDA_TRY(cudaSetDevice(device));
    return decode_chars_enqueue(static_cast<cudaStream_t>(stream), d_tokens, itemsize, rows, cols, row_stride, col_stride, tok, d_row_offsets,
                                d_row_tail, d_chars, -1, nullptr);
}

int bsq_decode_text(int device, void *stream, const void *d_tokens, int itemsize, int64_t rows, int64_t cols, int64_t row_stride,
                    int64_t col_stride, const bsq_tokenizer *tok, int64_t *d_row_offsets, int32_t *d_row_tail, uint8_t *d_chars,
                    int64_t capacity, int64_t *total_chars) {
    bsq::DeviceRestore restore_device;
    if (total_chars == nullptr || capacity < 0) return fail(BSQ_ERR_ARG, "null argument");
    if (int rc = decode_args_check(tok, itemsize, rows, cols)) return rc;
    *total_chars = 0;
    BSQ_CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (rows == 0) {
        BSQ_CUDA_TRY(cudaMemsetAsync(d_row_offsets, 0, sizeof(int64_t), st));
        return BSQ_OK;
    }
    if (d_tokens == nullptr && cols > 0) return fail(BSQ_ERR_ARG, "Empty array cannot yield a decoded string");  // src/tokenize.h:133
    int64_t *host_pair = nullptr, *d_work = nullptr;
    if (int rc = decode_lengths_enqueue(device, st, d_tokens, itemsize, rows, cols, row_stride, col_stride, tok, d_row_offsets, d_row_tail,
                                        &host_pair, &d_work))
        return rc;
    // pass 2 follows pass 1 on the stream without a host round trip; it reads the total on the device and writes
    // nothing when the text does not fit `capacity` (or when a token had no entry: the offsets are then meaningless
    // but bounded by 5 x tokens, and the call fails below)
    if (cols > 0 && d_chars != nullptr && capacity > 0) {
        if (int rc = decode_chars_enqueue(st, d_tokens, itemsize, rows, cols, row_stride, col_stride, tok, d_row_offsets, d_row_tail,
                                          d_chars, capacity, reinterpret_cast<const unsigned long long *>(d_work))) {
            cudaStreamSynchronize(st);
            cudaFreeAsync(d_work, st);
            return rc;
        }
    }
    BSQ_CUDA_TRY(cudaStreamSynchronize(st));
    return decode_lengths_finish(st, d_tokens, itemsize, cols, row_stride, col_stride, host_pair, d_work, total_chars);
}

}  // extern "C"
