// K13: sliding-window tiling of a packed batch and per-residue stitching of model outputs (sm_100a).
//
// Semantics (include/bsq.h, bsq_tile / bsq_untile_mean): sequence i of len_i residues gives m_i windows of at most W
// residues starting every S residues (W >= S >= 1); the tail mode decides the last one.  Everything about one sequence's
// windows -- count, starts, lengths, byte total -- is the arithmetic of tile_count / tile_start / tile_len below, the only
// statement of the rule in the library (host extent, device extent and both kernels use it).
//
// K13a, bsq_tile (no state between launches, capturable into a CUDA graph):
//   row_scan_kernel + row_carry_kernel, twice (the carry only past 1024 sequences, bsq_kernels.cuh): the per-sequence
//                       window counts into seq_ptr, then the per-sequence output byte totals (closed form: (m - 1) W +
//                       len_last for SHORT, m W otherwise) into byte_ptr.  byte_ptr, and seq_ptr when the caller passes
//                       none, live in stream-ordered scratch (cudaMallocAsync / cudaFreeAsync on the call's stream).
//   tile_fix_kernel     one thread per sequence adds the carry of its scan CTA (row_scan_carry) to both entries.
//   tile_gather_kernel  a grid-stride pass over the windows writes out_offsets, seq_index and starts (a binary search of
//                       seq_ptr per window), then the bytes: bsq_kernels.cuh's flat map with the sequences as rows and
//                       byte_ptr as their starts (no row data of its own).  Its piece of a sequence: a FastDiv by W gives
//                       the first window the vector touches (every window but a sequence's last is exactly W bytes of
//                       output), and each window piece is two aligned ld.global.nc loads of its source, realigned with
//                       funnel shifts and merged in with a byte mask.
//   With S < W, overlapping windows re-read their shared source bytes; those re-reads hit L2 (a tile's source span is
//   about 64 KiB * S / W + W bytes).
//
// K13b, bsq_untile_mean: one thread per (residue, channel vector): the residue's sequence by a binary search of the
// source offsets, then the covering windows by arithmetic -- j from ceil((p - W + 1) / S) to floor(p / S), and END's last
// window -- strand 0 before strand 1, ascending within a strand; a float32 sum divided by the count (NaN for none).
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <string>
#include <type_traits>

#include "bsq_internal.h"
#include "bsq_kernels.cuh"

namespace bsq {

namespace {

struct TileShape {
    int64_t W, S;
    int tail;
};

// windows of a sequence of len >= 0 residues
__host__ __device__ __forceinline__ int64_t tile_count(int64_t len, const TileShape &t) {
    if (len <= t.W) return 1;
    const int64_t d = len - t.W;
    return (t.tail == BSQ_TILE_DROP ? d : d + t.S - 1) / t.S + 1;
}
// output bytes of those windows (I: int64_t in the kernels, whose totals are validated; __int128 in the extents)
template <typename I>
__host__ __device__ __forceinline__ I tile_bytes(int64_t len, int64_t m, const TileShape &t) {
    if (len <= t.W) return static_cast<I>(len);
    if (t.tail == BSQ_TILE_SHORT) return static_cast<I>(m - 1) * t.W + (len - (m - 1) * t.S);
    return static_cast<I>(m) * t.W;
}
__host__ __device__ __forceinline__ int64_t tile_start(int64_t j, int64_t m, int64_t len, const TileShape &t) {
    return (t.tail == BSQ_TILE_END && j == m - 1 && len > t.W) ? len - t.W : j * t.S;
}
__host__ __device__ __forceinline__ int64_t tile_len(int64_t j, int64_t len, const TileShape &t) {
    if (len <= t.W) return len;
    return t.tail == BSQ_TILE_SHORT ? min(t.W, len - j * t.S) : t.W;
}

struct WinCount {
    TileShape t;
    __device__ __forceinline__ int64_t operator()(int64_t len) const { return tile_count(len, t); }
};
struct ByteCount {
    TileShape t;
    __device__ __forceinline__ int64_t operator()(int64_t len) const { return tile_bytes<int64_t>(len, tile_count(len, t), t); }
};
// the extents' measure: windows, their bytes, and the longest window
struct TileMeasure {
    TileShape t;
    __host__ __device__ __forceinline__ Extent extent(int64_t len) const {
        const int64_t m = tile_count(len, t);
        bool over = false;
        const int64_t nb = clamp_sat(tile_bytes<__int128>(len, m, t), &over);
        return {m, nb, len < t.W ? len : t.W, over};
    }
};

// the scan entries that lack their scan CTA's carry get it (the others are final and only read here, so no thread reads
// an entry another thread writes)
__global__ void tile_fix_kernel(int64_t n, int64_t *__restrict__ seq_ptr, int64_t *__restrict__ byte_ptr) {
    const int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x + 1;
    if (e > n) return;
    const int64_t cs = row_scan_carry(seq_ptr, e, n), cb = row_scan_carry(byte_ptr, e, n);
    if (cs != 0) seq_ptr[e] += cs;
    if (cb != 0) byte_ptr[e] += cb;
}

struct TileArgs {
    const uint8_t *bytes;
    const int64_t *offs;
    const int64_t *seq_ptr;
    const int64_t *byte_ptr;
    int64_t n, total;
    TileShape t;
    FastDiv wdiv;  // W, when W < 2^31
};

__device__ __forceinline__ int64_t div_w(int64_t x, const TileArgs &a) {
    return (x < (int64_t(1) << 31) && a.t.W < (int64_t(1) << 31)) ? static_cast<int64_t>(fd_div(static_cast<uint32_t>(x), a.wdiv))
                                                                   : x / a.t.W;
}

// K13a's rows for flat_map: the sequences, starting at byte_ptr
struct TileMap {
    TileArgs a;
    struct None {};

    __device__ __forceinline__ int64_t start(int64_t i) const { return __ldg(a.byte_ptr + i); }
    __device__ __forceinline__ void stage(int, int64_t) const {}
    __device__ __forceinline__ None row_t(int) const { return {}; }
    __device__ __forceinline__ None row_g(int64_t) const { return {}; }
    // the windows of sequence i (output bytes from b) that output bytes [q, q + 16) touch
    __device__ __forceinline__ void piece(int64_t q, int64_t i, int64_t b, int64_t, None, uint32_t res[4]) const {
        const uintptr_t src0 = reinterpret_cast<uintptr_t>(a.bytes);
        const int64_t s = __ldg(a.offs + i), len = __ldg(a.offs + i + 1) - s;
        const int64_t m = tile_count(len, a.t);
        for (int64_t j = div_w(max(q, b) - b, a); j < m; ++j) {
            const int64_t ws = b + j * a.t.W;  // the window's first output byte
            if (ws >= q + 16) break;
            const int64_t wl = tile_len(j, len, a.t);
            const int64_t src = s + tile_start(j, m, len, a.t);  // its first source byte
            const uintptr_t lo = (src0 + static_cast<uintptr_t>(src)) & ~uintptr_t(15);
            const uintptr_t hi = (src0 + static_cast<uintptr_t>(src + wl - 1)) & ~uintptr_t(15);
            uint32_t t[4];
            fetch_clamped<4>(src0 + static_cast<uintptr_t>(src + (q - ws)), lo, hi, t);
            merge16(res, t, ws - q, ws + wl - q);
        }
    }
};

__global__ void __launch_bounds__(kFlatThreads, kFlatMinBlocks)
tile_gather_kernel(TileArgs a, uint8_t *__restrict__ out, int64_t *__restrict__ out_offs, int64_t *__restrict__ seq_index,
                   int64_t *__restrict__ starts) {
    a.total = __ldg(a.byte_ptr + a.n);
    // window table: out_offsets, seq_index, starts
    const int64_t M = __ldg(a.seq_ptr + a.n);
    for (int64_t w = blockIdx.x * static_cast<int64_t>(kFlatThreads) + threadIdx.x; w <= M; w += static_cast<int64_t>(gridDim.x) * kFlatThreads) {
        if (w == M) {
            out_offs[M] = a.total;
            break;
        }
        int64_t lo = 0, hi = a.n;  // the largest i with seq_ptr[i] <= w
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if (__ldg(a.seq_ptr + mid) <= w) lo = mid;
            else hi = mid;
        }
        const int64_t j = w - __ldg(a.seq_ptr + lo);
        out_offs[w] = __ldg(a.byte_ptr + lo) + j * a.t.W;
        if (seq_index != nullptr) seq_index[w] = lo;
        if (starts != nullptr) {
            const int64_t len = __ldg(a.offs + lo + 1) - __ldg(a.offs + lo);
            starts[w] = tile_start(j, tile_count(len, a.t), len, a.t);
        }
    }
    flat_map(out, a.n, a.total, TileMap{a});
}

// ---- K13b -------------------------------------------------------------------------------------------------------------

struct UntileArgs {
    const void *y;
    const int32_t *cu;   // per-window first row, or nullptr: w * stride
    int64_t stride, col0, C;
    const int64_t *offs;  // source offsets
    int64_t n;
    const int64_t *seq_ptr;
    int64_t nwin;
    int strands;
    const uint8_t *flipped;
    TileShape t;
    int64_t nc;  // channel vectors per row
    FastDiv ncdiv;
};

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <>
__device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }

// V consecutive elements of type T (V * sizeof(T) is 4, 8 or 16 bytes with V > 1: one load, aligned by the host's checks)
template <typename T, int V>
__device__ __forceinline__ void load_v(const T *p, float f[V]) {
    if constexpr (V == 1) {
        f[0] = to_f32<T>(p[0]);
    } else {
        constexpr int kBytes = V * sizeof(T);
        using L = typename std::conditional<kBytes == 16, uint4, typename std::conditional<kBytes == 8, uint2, uint32_t>::type>::type;
        const L raw = __ldg(reinterpret_cast<const L *>(p));
        const T *e = reinterpret_cast<const T *>(&raw);
#pragma unroll
        for (int k = 0; k < V; ++k) f[k] = to_f32<T>(e[k]);
    }
}

template <typename T, int V>
__global__ void __launch_bounds__(256) untile_kernel(UntileArgs a, float *__restrict__ out) {
    const int64_t R = __ldg(a.offs + a.n) - __ldg(a.offs);
    const int64_t items = R * a.nc;
    const int64_t M = a.nwin;
    for (int64_t it = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; it < items;
         it += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t row = it < (int64_t(1) << 31) ? static_cast<int64_t>(fd_div(static_cast<uint32_t>(it), a.ncdiv)) : it / a.nc;
        const int64_t c = (it - row * a.nc) * V;
        const int64_t gpos = row + __ldg(a.offs);
        int64_t lo = 0, hi = a.n;  // the largest i with offs[i] <= gpos (the first of equal offsets is an empty sequence)
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if (__ldg(a.offs + mid) <= gpos) lo = mid;
            else hi = mid;
        }
        const int64_t s = __ldg(a.offs + lo), len = __ldg(a.offs + lo + 1) - s, p = gpos - s;
        const int64_t m = tile_count(len, a.t), w0 = __ldg(a.seq_ptr + lo);
        // regular windows (all but END's last) cover p for j in [jlo, jhi]
        const int64_t mreg = (a.t.tail == BSQ_TILE_END && len > a.t.W) ? m - 1 : m;
        const int64_t jlo = p >= a.t.W ? (p - a.t.W) / a.t.S + 1 : 0;
        const int64_t jhi = min(p / a.t.S, mreg - 1);
        const bool last = mreg < m && p >= len - a.t.W;  // END's last window
        float acc[V];
#pragma unroll
        for (int k = 0; k < V; ++k) acc[k] = 0.0f;
        int cnt = 0;
        for (int strand = 0; strand < a.strands; ++strand) {
            auto add = [&](int64_t j) {
                const int64_t w = w0 + j + strand * M;
                const int64_t st = tile_start(j, m, len, a.t), wl = tile_len(j, len, a.t);
                const bool fl = a.flipped != nullptr && a.flipped[w] != 0;
                const int64_t tpos = fl ? wl - 1 - (p - st) : p - st;
                const int64_t yrow = (a.cu != nullptr ? __ldg(a.cu + w) : w * a.stride) + a.col0 + tpos;
                float f[V];
                load_v<T, V>(static_cast<const T *>(a.y) + yrow * a.C + c, f);
#pragma unroll
                for (int k = 0; k < V; ++k) acc[k] += f[k];
                ++cnt;
            };
            for (int64_t j = jlo; j <= jhi; ++j) add(j);
            if (last) add(m - 1);
        }
        float *o = out + row * a.C + c;
#pragma unroll
        for (int k = 0; k < V; ++k) o[k] = cnt > 0 ? acc[k] / static_cast<float>(cnt) : __int_as_float(0x7fc00000);
    }
}

// a persistent grid: the row count lives on the device, and the kernel strides over whatever it is
template <typename T, int V>
int launch_untile(cudaStream_t st, const UntileArgs &a, float *out) {
    untile_kernel<T, V><<<cur_sms() * 8, 256, 0, st>>>(a, out);
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}

int check_shape(int64_t W, int64_t S, int tail) {
    if (W < 1) return fail(BSQ_ERR_ARG, "window must be >= 1, got " + std::to_string(W));
    if (S < 1 || S > W) return fail(BSQ_ERR_ARG, "stride must lie in 1..window = " + std::to_string(W) + ", got " + std::to_string(S));
    if (tail != BSQ_TILE_SHORT && tail != BSQ_TILE_END && tail != BSQ_TILE_DROP)
        return fail(BSQ_ERR_ARG, "tail must be BSQ_TILE_SHORT, BSQ_TILE_END or BSQ_TILE_DROP");
    return BSQ_OK;
}

}  // namespace

}  // namespace bsq

using namespace bsq;

extern "C" int bsq_tile_extent_host(const int64_t *h_offsets, int64_t nseq, int64_t window, int64_t stride, int tail, int64_t *nwin,
                                    int64_t *nbytes, int64_t *max_len) {
    if (int rc = check_shape(window, stride, tail)) return rc;
    if (nwin == nullptr || nbytes == nullptr || max_len == nullptr) return fail(BSQ_ERR_ARG, "null output");
    if (nseq < 0 || (nseq > 0 && h_offsets == nullptr)) return fail(BSQ_ERR_ARG, "bad offsets");
    *nwin = *nbytes = *max_len = 0;
    if (nseq == 0) return BSQ_OK;
    Extent e{};
    if (int rc = reduce_offsets_host(h_offsets, nseq, TileMeasure{{window, stride, tail}}, &e)) return rc;
    if (e.over) return fail(BSQ_ERR_ARG, "the windows' count or bytes exceed INT64_MAX");
    *nwin = e.sum0;
    *nbytes = e.sum1;
    *max_len = e.max;
    return BSQ_OK;
}

extern "C" int bsq_tile_extent_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t nbytes, int64_t window,
                                      int64_t stride, int tail, int64_t *nwin, int64_t *out_nbytes, int64_t *max_len) {
    bsq::DeviceRestore restore_device;
    if (int rc = check_shape(window, stride, tail)) return rc;
    if (nwin == nullptr || out_nbytes == nullptr || max_len == nullptr) return fail(BSQ_ERR_ARG, "null output");
    if (nseq < 0 || (nseq > 0 && d_offsets == nullptr)) return fail(BSQ_ERR_ARG, "bad offsets");
    *nwin = *out_nbytes = *max_len = 0;
    if (nseq == 0) return BSQ_OK;
    Extent e{};
    if (int rc = reduce_offsets_device(device, static_cast<cudaStream_t>(stream), d_offsets, nseq, nbytes, TileMeasure{{window, stride, tail}},
                                       &e))
        return rc;
    if (e.over) return fail(BSQ_ERR_ARG, "the windows' count or bytes exceed INT64_MAX");
    *nwin = e.sum0;
    *out_nbytes = e.sum1;
    *max_len = e.max;
    return BSQ_OK;
}

extern "C" int bsq_tile(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int64_t window,
                        int64_t stride, int tail, uint8_t *d_out_bytes, int64_t *d_out_offsets, int64_t *d_seq_ptr,
                        int64_t *d_seq_index, int64_t *d_starts) {
    bsq::DeviceRestore restore_device;
    if (int rc = check_shape(window, stride, tail)) return rc;
    if (nseq < 0) return fail(BSQ_ERR_ARG, "negative batch size");
    if (d_out_offsets == nullptr) return fail(BSQ_ERR_ARG, "null output offsets");
    if (nseq > 0 && (d_bytes == nullptr || d_offsets == nullptr || d_out_bytes == nullptr))
        return fail(BSQ_ERR_ARG, "null bytes, offsets or output bytes");
    BSQ_CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nseq == 0) {
        BSQ_CUDA_TRY(cudaMemsetAsync(d_out_offsets, 0, sizeof(int64_t), st));
        if (d_seq_ptr != nullptr) BSQ_CUDA_TRY(cudaMemsetAsync(d_seq_ptr, 0, sizeof(int64_t), st));
        return BSQ_OK;
    }
    const TileShape t{window, stride, tail};
    int64_t *scratch = nullptr;
    const size_t ns = static_cast<size_t>(nseq + 1) * (d_seq_ptr != nullptr ? 1 : 2);
    BSQ_CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&scratch), ns * sizeof(int64_t), st));
    int64_t *byte_ptr = scratch, *seq_ptr = d_seq_ptr != nullptr ? d_seq_ptr : scratch + nseq + 1;
    if (int rc = launch_row_scan(st, d_offsets, nseq, WinCount{t}, seq_ptr)) return rc;
    if (int rc = launch_row_scan(st, d_offsets, nseq, ByteCount{t}, byte_ptr)) return rc;
    if (nseq > kRowScan) {
        tile_fix_kernel<<<static_cast<unsigned>((nseq + 255) / 256), 256, 0, st>>>(nseq, seq_ptr, byte_ptr);
        count_launch();
        BSQ_CUDA_TRY(cudaGetLastError());
    }
    TileArgs a;
    a.bytes = d_bytes;
    a.offs = d_offsets;
    a.seq_ptr = seq_ptr;
    a.byte_ptr = byte_ptr;
    a.n = nseq;
    a.total = 0;  // (byte_ptr[n]: read by the kernel)
    a.t = t;
    a.wdiv = make_fastdiv(static_cast<uint32_t>(std::min<int64_t>(window, (int64_t(1) << 31) - 1)));
    tile_gather_kernel<<<cur_sms() * kFlatMinBlocks, kFlatThreads, 0, st>>>(a, d_out_bytes, d_out_offsets, d_seq_index, d_starts);
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    BSQ_CUDA_TRY(cudaFreeAsync(scratch, st));
    return BSQ_OK;
}

extern "C" int bsq_untile_mean(int device, void *stream, int dtype, const void *d_y, int64_t channels, int64_t row_stride,
                               const int32_t *d_cu, int64_t col0, const int64_t *d_src_offsets, int64_t nseq, int64_t window,
                               int64_t stride, int tail, const int64_t *d_seq_ptr, int64_t nwin, int strands,
                               const uint8_t *d_flipped, float *d_out) {
    bsq::DeviceRestore restore_device;
    if (int rc = check_shape(window, stride, tail)) return rc;
    if (dtype != BSQ_UNTILE_F32 && dtype != BSQ_UNTILE_BF16 && dtype != BSQ_UNTILE_F16)
        return fail(BSQ_ERR_ARG, "dtype must be BSQ_UNTILE_F32, BSQ_UNTILE_BF16 or BSQ_UNTILE_F16");
    if (channels < 1) return fail(BSQ_ERR_ARG, "channels must be >= 1");
    if (col0 < 0) return fail(BSQ_ERR_ARG, "col0 must be >= 0");
    if (strands != 1 && strands != 2) return fail(BSQ_ERR_ARG, "strands must be 1 or 2");
    if (nseq < 0 || nwin < nseq) return fail(BSQ_ERR_ARG, "negative batch size, or fewer windows than sequences");
    if (d_cu == nullptr && row_stride <= col0) return fail(BSQ_ERR_ARG, "row_stride must exceed col0 without cu_seqlens");
    if (nseq == 0) return BSQ_OK;
    if (d_y == nullptr || d_src_offsets == nullptr || d_seq_ptr == nullptr || d_out == nullptr)
        return fail(BSQ_ERR_ARG, "null values, offsets, seq_ptr or output");
    const size_t es = dtype == BSQ_UNTILE_F32 ? 4 : 2;
    UntileArgs a;
    a.y = d_y;
    a.cu = d_cu;
    a.stride = row_stride;
    a.col0 = col0;
    a.C = channels;
    a.offs = d_src_offsets;
    a.n = nseq;
    a.seq_ptr = d_seq_ptr;
    a.nwin = nwin;
    a.strands = strands;
    a.flipped = d_flipped;
    a.t = TileShape{window, stride, tail};
    // channel vectors: 16 bytes of input when every row and both pointers allow it, else one element
    const bool al16 = ((reinterpret_cast<uintptr_t>(d_y) | reinterpret_cast<uintptr_t>(d_out)) & 15u) == 0;
    const int V = (al16 && (channels * static_cast<int64_t>(es)) % 16 == 0) ? static_cast<int>(16 / es) : 1;
    a.nc = channels / V;
    a.ncdiv = make_fastdiv(static_cast<uint32_t>(std::min<int64_t>(a.nc, (int64_t(1) << 31) - 1)));
    BSQ_CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == BSQ_UNTILE_F32) return V == 4 ? launch_untile<float, 4>(st, a, d_out) : launch_untile<float, 1>(st, a, d_out);
    if (dtype == BSQ_UNTILE_BF16) return V == 8 ? launch_untile<__nv_bfloat16, 8>(st, a, d_out) : launch_untile<__nv_bfloat16, 1>(st, a, d_out);
    return V == 8 ? launch_untile<__half, 8>(st, a, d_out) : launch_untile<__half, 1>(st, a, d_out);
}
