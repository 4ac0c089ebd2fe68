// K9: crop every sequence of a packed batch to a window of at most W residues (sm_100a).
//
// Semantics (include/bsq.h, bsq_crop): len'_i = min(len_i, W); the window starts at 0 (head mode, or len_i <= W) or,
// in random mode, at floor(d * (len_i - W + 1) / 2^64) with d = x0 | x1 << 32 of Philox4x32-10 at counter
// (g_lo, g_hi, 0, 3), g = seq_index_base + i.  out_offsets is the exclusive scan of len'_i (out_offsets[0] = 0).
//
// Three launches, no scratch memory and no state between launches (capturable into a CUDA graph):
//   row_scan_kernel     one thread per row, kRowScan rows per CTA: len'_i (CropCount), the CTA's inclusive scan of them
//                       (block_exclusive_scan) written to out_offsets[i + 1].  The entry at the end of each CTA's rows
//                       is then that CTA's total.  (Shared with K11's cu_seqlens, bsq_kernels.cuh.)
//   row_carry_kernel    one CTA (only when there is more than one scan CTA): scans the CTA totals in place, so every
//                       entry at the end of a scan CTA's rows becomes final.
//   crop_gather_kernel  one warp per row: adds the carry (the final entry at the end of the previous scan CTA, never
//                       written by this kernel) to the row's own entry, draws the start (one Philox block, cropped
//                       random rows only) and copies the window.  Destination-aligned 16-byte stores, each from two
//                       aligned 16-byte loads of the source realigned by funnel shifts (the shift is the same for the
//                       whole row); the up to 15 bytes at either end of a row are byte stores, so a 16-byte vector
//                       shared by two rows keeps both rows' bytes.  A row's end offset is its own entry, and its start
//                       is that minus len'_i: no warp reads an entry another warp writes.
// The kept bytes are read once and written once: the kernel is HBM-bound by design.
#include <cuda_runtime.h>

#include <algorithm>

#include "bsq_internal.h"
#include "bsq_kernels.cuh"

namespace bsq {

namespace {

constexpr int kCThreads = 256;  // crop_gather_kernel: 8 warps, one row each

struct CropParam {
    int64_t W;
    int64_t base;  // global index of this launch's sequence 0
    uint32_t k0, k1;
    int random;
};

__device__ __forceinline__ int64_t crop_start(int64_t len, int64_t i, const CropParam &c) {
    if (!c.random || len <= c.W) return 0;
    const uint64_t g = static_cast<uint64_t>(c.base + i);
    const Philox p = philox4x32_10(static_cast<uint32_t>(g), static_cast<uint32_t>(g >> 32), 0u, 3u, c.k0, c.k1);
    const uint64_t d = static_cast<uint64_t>(p.c[0]) | (static_cast<uint64_t>(p.c[1]) << 32);
    return static_cast<int64_t>(__umul64hi(d, static_cast<uint64_t>(len - c.W + 1)));
}

__global__ void __launch_bounds__(kCThreads)
crop_gather_kernel(const uint8_t *__restrict__ bytes, const int64_t *__restrict__ offs, int64_t n, CropParam c,
                   int64_t *__restrict__ out_offs, uint8_t *__restrict__ out, int64_t *__restrict__ starts) {
    const int lane = threadIdx.x & 31;
    const int64_t i = static_cast<int64_t>(blockIdx.x) * (kCThreads / 32) + (threadIdx.x >> 5);
    if (i >= n) return;
    const int64_t s = __ldg(offs + i), len = __ldg(offs + i + 1) - s;
    const int64_t kept = min(len, c.W);
    const int64_t st = crop_start(len, i, c);
    // the row's end offset: its CTA-local inclusive prefix plus the carry it still lacks
    const int64_t carry = row_scan_carry(out_offs, i + 1, n);
    const int64_t e = out_offs[i + 1] + carry;
    __syncwarp();
    if (lane == 0) {
        if (carry != 0) out_offs[i + 1] = e;
        if (starts != nullptr) starts[i] = st;
    }
    if (kept <= 0) return;
    uint8_t *dst = out + (e - kept);
    const uint8_t *src = bytes + s + st;
    const int64_t head = min(static_cast<int64_t>((16u - (reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u), kept);
    const int64_t nvec = (kept - head) >> 4;
    const int64_t body_end = head + 16 * nvec;
    const int tail = static_cast<int>(kept - body_end);
    if (lane < head) dst[lane] = __ldg(src + lane);
    if (lane < tail) dst[body_end + lane] = __ldg(src + body_end + lane);
    // body: every vector lies inside the window, so both aligned source words hold window bytes
    const uintptr_t sa = reinterpret_cast<uintptr_t>(src + head);
    const uint32_t shift = static_cast<uint32_t>(sa & 15u);
    const uintptr_t al = sa - shift;
    RowSrc rs;
    rs.off = static_cast<int>(shift);
    uint4 *d4 = reinterpret_cast<uint4 *>(dst + head);
    for (int64_t v = lane; v < nvec; v += 32) {
        Fetched fe;
        fe.v0 = ldg16(al + 16 * v);
        fe.v1 = shift != 0 ? ldg16(al + 16 * v + 16) : make_uint4(0u, 0u, 0u, 0u);
        uint32_t t[4];
        fetch_align(fe, rs, 0, t);
        d4[v] = make_uint4(t[0], t[1], t[2], t[3]);
    }
}

}  // namespace

}  // namespace bsq

using namespace bsq;

extern "C" int bsq_crop(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int64_t crop_len,
                        int random, uint64_t seed, int64_t seq_index_base, uint8_t *d_out_bytes, int64_t *d_out_offsets,
                        int64_t *d_starts) {
    bsq::DeviceRestore restore_device;
    if (crop_len < 1) return fail(BSQ_ERR_ARG, "crop_len must be >= 1");
    if (nseq < 0) return fail(BSQ_ERR_ARG, "negative batch size");
    if (d_out_offsets == nullptr) return fail(BSQ_ERR_ARG, "null output offsets");
    if (nseq > 0 && (d_bytes == nullptr || d_offsets == nullptr || d_out_bytes == nullptr))
        return fail(BSQ_ERR_ARG, "null bytes, offsets or output bytes");
    BSQ_CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nseq == 0) {
        BSQ_CUDA_TRY(cudaMemsetAsync(d_out_offsets, 0, sizeof(int64_t), st));
        return BSQ_OK;
    }
    if (int rc = launch_row_scan(st, d_offsets, nseq, CropCount{crop_len}, d_out_offsets)) return rc;
    const CropParam c{crop_len, seq_index_base, static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), random != 0};
    const int64_t rows_per_cta = kCThreads / 32;
    crop_gather_kernel<<<static_cast<unsigned>((nseq + rows_per_cta - 1) / rows_per_cta), kCThreads, 0, st>>>(
        d_bytes, d_offsets, nseq, c, d_out_offsets, d_out_bytes, d_starts);
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}
