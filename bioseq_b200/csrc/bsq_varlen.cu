// K1v: padding-free tokens -- one packed token stream plus int32 cu_seqlens (sm_100a).
//
// Semantics (batch_tokenize's rows with the padding cut off, src/tokenize.h:460-478):
//   cu[i] = (offsets[i] - offsets[0]) + i * k,  k = bos + eos,  T = cu[n];
//   tokens[cu[i] .. cu[i+1]) = [BOS] lut(residues of sequence i) [EOS].
// Row i's residue column c (c >= bos) comes from source byte offsets[0] + f - i * k - bos, f = cu[i] + c: inside one
// row the output is the input shifted by a constant, and the shift grows by k from one row to the next.  So the
// residues an output tile needs are ONE contiguous span of the packed input, no longer than the tile.
//
//   k = 0   varlen_map_kernel: a pure byte map over [offsets[0], offsets[n]) -- no rows at all.  Each thread takes 16
//           output elements: one or two aligned 16-byte loads (the source shift offsets[0] % 16 is the same for the
//           whole launch: the realignment switch is uniform), 16 LUT look-ups, one 16-byte store per 16 output bytes.
//   k >= 1  varlen_tile_kernel: tiles of kVTile output elements, dealt round-robin to a persistent grid (a static
//           order: no tile counter, so every launch is capturable and may be replayed concurrently with itself).
//           Per tile the CTA
//             1. finds the tile's first row with a 256-ary search over cu (computed from offsets on the fly; two
//                rounds up to 66 049 rows, three up to 17 million): each thread probes one point, __syncthreads_count
//                of "cu <= f0" is where the answer lies;
//             2. loads the row table -- cu of the tile's rows, relative to the tile -- into shared memory, 256 rows a
//                round, until a row reaches past the tile's end.  Rows per tile are unbounded (an empty sequence still
//                emits k tokens): a tile with more than kVRowCap - 1 rows is "over-full" and takes step 4b;
//             3. copies the residue span, rounded out to 16 bytes, into shared memory with one 1-D bulk asynchronous
//                copy (cp.async.bulk, completion on an mbarrier) -- the global reads are exactly what the padded
//                kernel K1s reads for the same residues;
//             4a. one 16-byte output vector per thread and step: a binary search of the row table for the row of the
//                vector's first element, then, when all 16 elements are residues of that row, two LDS.128 of the
//                staged span, word select + funnel shifts, 16 look-ups and one st.global.cs.v4 -- otherwise element
//                by element (row boundaries, BOS / EOS, several rows per vector);
//             4b. over-full tiles: element by element, rows searched and residues read in global memory.
// Wide element kinds run the same kernels: codes go through the Expand table (as in K1f) and every 16 codes leave as
// sizeof(T) 16-byte stores.
//
// cu_seqlens is written by the same launch (a grid-stride pass over the offsets it reads anyway): no extra launch and
// no host round trip.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>

#include "bsq_internal.h"
#include "bsq_kernels.cuh"

namespace bsq {

namespace {

constexpr int kVThreads = 256;
constexpr int kVTile = 16384;             // output elements per tile: 1024 vectors, 4 per thread
constexpr int kVRowCap = 1024;            // row-table entries: tiles of up to kVRowCap - 1 rows use the table
constexpr int kVStage = kVTile + 64;      // staged span: <= kVTile + 32 bytes after rounding, + 32 for the second LDS.128
constexpr int kVMinBlocks = 4;            // CTAs per SM

__device__ __forceinline__ uint32_t v_s_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ uint4 v_lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t v_ldsu8(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void v_bar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "BSQ_VARLEN_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@!p bra BSQ_VARLEN_WAIT_%=;\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}

// Four LUT look-ups; `lutb` is the LUT's shared address, 256-byte aligned (one PRMT forms each address).
__device__ __forceinline__ uint32_t v_translate4(uint32_t x, uint32_t lutb) {
    const uint32_t b0 = v_ldsu8(__byte_perm(x, lutb, 0x7650));
    const uint32_t b1 = v_ldsu8(__byte_perm(x, lutb, 0x7651));
    const uint32_t b2 = v_ldsu8(__byte_perm(x, lutb, 0x7652));
    const uint32_t b3 = v_ldsu8(__byte_perm(x, lutb, 0x7653));
    return b0 + b1 * 0x100u + b2 * 0x10000u + b3 * 0x1000000u;
}

// 16 codes from the 16 source bytes at shared address S (any alignment; the shift varies from lane to lane, so the
// words are picked with selects instead of a switch).
__device__ __forceinline__ void v_window16(uint32_t S, uint32_t lutb, uint32_t t[4]) {
    const uint4 v0 = v_lds128(S & ~15u), v1 = v_lds128((S & ~15u) + 16u);
    const uint32_t sh = S << 3;
    const bool q2 = (S & 8u) != 0, q1 = (S & 4u) != 0;
    const uint32_t a0 = q2 ? v0.z : v0.x, a1 = q2 ? v0.w : v0.y, a2 = q2 ? v1.x : v0.z, a3 = q2 ? v1.y : v0.w;
    const uint32_t a4 = q2 ? v1.z : v1.x, a5 = q2 ? v1.w : v1.y;
    const uint32_t x[5] = {q1 ? a1 : a0, q1 ? a2 : a1, q1 ? a3 : a2, q1 ? a4 : a3, q1 ? a5 : a4};
#pragma unroll
    for (int k = 0; k < 4; ++k) t[k] = v_translate4(__funnelshift_r(x[k], x[k + 1], sh), lutb);
}

// 16 codes -> 16 output elements at out (cnt < 16: only the first cnt exist -- the batch's last vector).
template <typename T>
__device__ __forceinline__ void v_store16(T *out, const uint32_t t[4], int cnt, const Expand &ex) {
    if (sizeof(T) == 1) {
        if (cnt == 16) {
            __stcs(reinterpret_cast<uint4 *>(out), make_uint4(t[0], t[1], t[2], t[3]));
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
                if (j < cnt) reinterpret_cast<uint8_t *>(out)[j] = static_cast<uint8_t>(t[j >> 2] >> (8 * (j & 3)));
        }
        return;
    }
    constexpr int EPV = 16 / sizeof(T);  // elements per 16-byte store
    if (cnt == 16) {
#pragma unroll
        for (int s = 0; s < 16 / EPV; ++s) {
            T vals[EPV];
#pragma unroll
            for (int j = 0; j < EPV; ++j) {
                const int e = s * EPV + j;
                vals[j] = static_cast<T>(expand_code((t[e >> 2] >> (8 * (e & 3))) & 0xffu, ex));
            }
            __stcs(reinterpret_cast<uint4 *>(out) + s, *reinterpret_cast<const uint4 *>(vals));
        }
    } else {
#pragma unroll
        for (int e = 0; e < 16; ++e)
            if (e < cnt) out[e] = static_cast<T>(expand_code((t[e >> 2] >> (8 * (e & 3))) & 0xffu, ex));
    }
}

// cu[i] = offsets[i] - offsets[0] + i * k for i = 0 .. n, grid-stride.
__device__ __forceinline__ void v_write_cu(const int64_t *__restrict__ offs, int64_t n, int k, int64_t off0, int32_t *__restrict__ cu) {
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i <= n; i += static_cast<int64_t>(gridDim.x) * blockDim.x)
        cu[i] = static_cast<int32_t>(__ldg(offs + i) - off0 + i * k);
}

// ------------------------------------------------------------------------------------------------------------------
// k = 0: tokens[f] = lut[bytes[offsets[0] + f]].
template <typename T>
__global__ void __launch_bounds__(kVThreads)
varlen_map_kernel(const uint8_t *__restrict__ bytes, const int64_t *__restrict__ offs, int64_t n, LutParam lutp, Expand ex,
                  T *__restrict__ out, int32_t *__restrict__ cu) {
    __shared__ __align__(256) uint8_t lut[256];
    load_lut(lut, lutp);
    const int64_t off0 = __ldg(offs), total = __ldg(offs + n) - off0;
    v_write_cu(offs, n, 0, off0, cu);
    __syncthreads();
    const uint32_t lutb = v_s_u32(lut);
    const uintptr_t src = reinterpret_cast<uintptr_t>(bytes + off0);
    const uint32_t shift = static_cast<uint32_t>(src & 15u);
    const uintptr_t al = src - shift;
    const int64_t nvec = (total + 15) / 16;
    for (int64_t v = blockIdx.x * static_cast<int64_t>(kVThreads) + threadIdx.x; v < nvec; v += static_cast<int64_t>(gridDim.x) * kVThreads) {
        const int cnt = static_cast<int>(min(int64_t(16), total - 16 * v));
        Fetched fe;
        fe.v0 = ldg16(al + 16 * v);
        // the second word holds residues only when the vector's bytes run past the first: never outside the span
        fe.v1 = shift + cnt > 16 ? ldg16(al + 16 * v + 16) : make_uint4(0u, 0u, 0u, 0u);
        RowSrc rs;
        rs.off = static_cast<int>(shift);
        uint32_t t[4];
        fetch_align(fe, rs, 0, t);
#pragma unroll
        for (int w = 0; w < 4; ++w) t[w] = v_translate4(t[w], lutb);
        v_store16<T>(out + 16 * v, t, cnt, ex);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// k >= 1: output tiles over a persistent grid.

// Codes of output elements [f, f + cnt) one by one.  `row` is the row of element f; cu_of(i) is cu[i] (absolute),
// src_of(g) the code of source byte g (bytes[g] through the LUT).
template <typename CU, typename SRC>
__device__ __forceinline__ void v_codes_bytewise(int64_t f, int cnt, int64_t row, int64_t off0, int k, const Specials &sp,
                                                 const CU &cu_of, const SRC &src_of, uint32_t t[4]) {
    t[0] = t[1] = t[2] = t[3] = 0u;
    int64_t c0 = cu_of(row), c1 = cu_of(row + 1);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        if (j >= cnt) break;
        const int64_t e = f + j;
        while (c1 <= e) {  // the next row starts here (empty sequences: several rows per element run)
            ++row;
            c0 = c1;
            c1 = cu_of(row + 1);
        }
        const int64_t c = e - c0;                  // column in the row
        const int64_t len = c1 - c0 - k;
        uint32_t code;
        if (c < sp.bos) code = sp.bos_w & 0xffu;
        else if (c - sp.bos < len) code = src_of(off0 + e - row * k - sp.bos);
        else code = sp.eos_w & 0xffu;
        t[j >> 2] |= code << (8 * (j & 3));
    }
}

// largest i in [lo, hi) with cu_of(i) <= x, given cu_of(lo) <= x
template <typename CU>
__device__ __forceinline__ int64_t v_row_of(int64_t x, int64_t lo, int64_t hi, const CU &cu_of) {
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (cu_of(mid) <= x) lo = mid;
        else hi = mid;
    }
    return lo;
}

template <typename T>
__global__ void __launch_bounds__(kVThreads, kVMinBlocks)
varlen_tile_kernel(const uint8_t *__restrict__ bytes, const int64_t *__restrict__ offs, int64_t n, LutParam lutp, Specials sp,
                   Expand ex, T *__restrict__ out, int32_t *__restrict__ cu) {
    __shared__ __align__(128) uint8_t stage[kVStage];
    __shared__ __align__(256) uint8_t lut[256];
    __shared__ int32_t rowtab[kVRowCap];  // cu[r0 + j] - f0
    __shared__ __align__(8) uint64_t full;
    __shared__ int64_t s_alo;             // global index of the first staged byte
    __shared__ int s_nrows;               // rows of the tile, -1: over-full
    __shared__ uint32_t s_copied;         // staged bytes

    load_lut(lut, lutp);
    if (threadIdx.x == 96) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(v_s_u32(&full)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const int k = sp.bos + sp.eos;
    const int64_t off0 = __ldg(offs), total = __ldg(offs + n) - off0 + n * k;
    v_write_cu(offs, n, k, off0, cu);
    __syncthreads();
    const uint32_t lutb = v_s_u32(lut), stage_a = v_s_u32(stage), full_a = v_s_u32(&full);
    const int tid = threadIdx.x;
    auto cu_g = [&](int64_t i) { return __ldg(offs + i) - off0 + i * k; };
    const int64_t ntiles = (total + kVTile - 1) / kVTile;
    uint32_t phase = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t f0 = tile * kVTile;
        const int tl = static_cast<int>(min(static_cast<int64_t>(kVTile), total - f0));  // elements of this tile
        // 1. first row: the largest r with cu[r] <= f0
        const int64_t r0 = block_search_le<kVThreads>(0, n, f0, cu_g);
        // 2. row table: cu[r0 + j] - f0 up to the first row that starts at or after the tile's end
        int nrows = block_row_table<kVThreads, kVRowCap>(r0, n, tl, [&](int j, int64_t r) {
            const int64_t c = cu_g(r) - f0;
            rowtab[j] = static_cast<int32_t>(c);
            return c;
        });
        // 3. the residue span, rounded out to 16 bytes, into shared memory
        if (tid == 0) {
            uint32_t copied = 0;
            int64_t alo = 0;
            if (nrows > 0) {
                const int64_t r1 = r0 + nrows - 1;  // last row touched
                const int64_t a0 = __ldg(offs + r0), a1 = __ldg(offs + r0 + 1), b0 = __ldg(offs + r1), b1 = __ldg(offs + r1 + 1);
                const int64_t slo = a0 + min(max(f0 - (static_cast<int64_t>(rowtab[0]) + f0) - sp.bos, int64_t(0)), a1 - a0);
                const int64_t shi = b0 + min(max(f0 + tl - (static_cast<int64_t>(rowtab[nrows - 1]) + f0) - sp.bos, int64_t(0)), b1 - b0);
                if (shi > slo) {
                    const uintptr_t A_lo = reinterpret_cast<uintptr_t>(bytes + slo) & ~uintptr_t(15);
                    const uintptr_t A_hi = (reinterpret_cast<uintptr_t>(bytes + shi) + 15) & ~uintptr_t(15);
                    copied = static_cast<uint32_t>(A_hi - A_lo);
                    alo = static_cast<int64_t>(A_lo - reinterpret_cast<uintptr_t>(bytes));
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full_a), "r"(copied) : "memory");
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(stage_a),
                                 "l"(reinterpret_cast<const void *>(A_lo)), "r"(copied), "r"(full_a)
                                 : "memory");
                }
            }
            s_nrows = nrows;
            s_alo = alo;
            s_copied = copied;
        }
        __syncthreads();
        nrows = s_nrows;
        const int64_t alo = s_alo;
        if (s_copied) {
            v_bar_wait(full_a, phase);
            phase ^= 1u;
        }
        T *const otile = out + f0;
        const int nv = (tl + 15) >> 4;
        if (nrows > 0) {
            // 4a. rows from the table, residues from the stage
            auto cu_t = [&](int64_t i) { return static_cast<int64_t>(rowtab[i - r0]) + f0; };
            auto src_t = [&](int64_t g) { return v_ldsu8(lutb + v_ldsu8(stage_a + static_cast<uint32_t>(g - alo))); };
            for (int v = tid; v < nv; v += kVThreads) {
                const int e0 = 16 * v;  // relative to f0
                const int cnt = min(16, tl - e0);
                int a = 0, b = nrows;  // largest j < nrows with rowtab[j] <= e0
                while (b - a > 1) {
                    const int mid = (a + b) >> 1;
                    if (rowtab[mid] <= e0) a = mid;
                    else b = mid;
                }
                const int c = e0 - rowtab[a];
                const int len = rowtab[a + 1] - rowtab[a] - k;
                uint32_t t[4];
                if (cnt == 16 && c >= sp.bos && c + 16 <= sp.bos + len) {
                    const int64_t g = off0 + f0 + e0 - (r0 + a) * k - sp.bos;
                    v_window16(stage_a + static_cast<uint32_t>(g - alo), lutb, t);
                } else {
                    v_codes_bytewise(f0 + e0, cnt, r0 + a, off0, k, sp, cu_t, src_t, t);
                }
                v_store16<T>(otile + e0, t, cnt, ex);
            }
        } else {
            // 4b. over-full tile (more rows than the table holds): rows and residues from global memory
            auto src_g = [&](int64_t g) { return v_ldsu8(lutb + __ldg(bytes + g)); };
            for (int v = tid; v < nv; v += kVThreads) {
                const int e0 = 16 * v;
                const int cnt = min(16, tl - e0);
                const int64_t row = v_row_of(f0 + e0, r0, min(n, r0 + e0 + 1 + (f0 - cu_g(r0))), cu_g);
                uint32_t t[4];
                v_codes_bytewise(f0 + e0, cnt, row, off0, k, sp, cu_g, src_g, t);
                v_store16<T>(otile + e0, t, cnt, ex);
            }
        }
        __syncthreads();  // the stage and the row table are refilled by the next tile
    }
}

template <typename T>
int launch_varlen(cudaStream_t st, const uint8_t *d_bytes, const int64_t *d_offs, int64_t nseq, const bsq_tokenizer &tok, void *d_out,
                  int32_t *d_cu) {
    const Prepared p = prepare(tok, sizeof(T) == 1 ? 0 : 1);
    T *o = static_cast<T *>(d_out);
    if (p.sp.bos + p.sp.eos == 0) {
        varlen_map_kernel<T><<<cur_sms() * 8, kVThreads, 0, st>>>(d_bytes, d_offs, nseq, p.lut, p.ex, o, d_cu);
    } else {
        varlen_tile_kernel<T><<<cur_sms() * kVMinBlocks, kVThreads, 0, st>>>(d_bytes, d_offs, nseq, p.lut, p.sp, p.ex, o, d_cu);
    }
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}

}  // namespace

}  // namespace bsq

using namespace bsq;

extern "C" int bsq_tokenize_varlen(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq,
                                   const bsq_tokenizer *tok, int kind, void *d_out, int32_t *d_cu_seqlens) {
    bsq::DeviceRestore restore_device;
    if (tok == nullptr) return fail(BSQ_ERR_ARG, "null tokenizer");
    if (nseq < 0) return fail(BSQ_ERR_ARG, "negative batch size");
    if (bsq_kind_size(kind) == 0) return fail(BSQ_ERR_ARG, "invalid element kind");
    if (d_offsets == nullptr || d_cu_seqlens == nullptr) return fail(BSQ_ERR_ARG, "null offsets or cu_seqlens");
    if (reinterpret_cast<uintptr_t>(d_out) & 15u) return fail(BSQ_ERR_ARG, "output pointer must be 16-byte aligned");
    BSQ_CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nseq == 0) {
        BSQ_CUDA_TRY(cudaMemsetAsync(d_cu_seqlens, 0, sizeof(int32_t), st));
        return BSQ_OK;
    }
    switch (kind) {
        case BSQ_I8: return launch_varlen<int8_t>(st, d_bytes, d_offsets, nseq, *tok, d_out, d_cu_seqlens);
        case BSQ_I16: return launch_varlen<int16_t>(st, d_bytes, d_offsets, nseq, *tok, d_out, d_cu_seqlens);
        case BSQ_I32: return launch_varlen<int32_t>(st, d_bytes, d_offsets, nseq, *tok, d_out, d_cu_seqlens);
        case BSQ_I64: return launch_varlen<int64_t>(st, d_bytes, d_offsets, nseq, *tok, d_out, d_cu_seqlens);
        case BSQ_F32: return launch_varlen<float>(st, d_bytes, d_offsets, nseq, *tok, d_out, d_cu_seqlens);
        default: return launch_varlen<double>(st, d_bytes, d_offsets, nseq, *tok, d_out, d_cu_seqlens);
    }
}
