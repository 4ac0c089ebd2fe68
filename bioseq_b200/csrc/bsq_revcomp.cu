// K12: reverse complement of a packed batch (sm_100a).
//
// Semantics (include/bsq.h, bsq_revcomp): out[j] = comp[in[len - 1 - j]] for a flipped sequence, a copy otherwise.
// ALWAYS flips every sequence, RANDOM sequence i iff x0 < gate (x0 = word 0 of Philox4x32-10 at counter (g_lo, g_hi, 0, 4),
// g = seq_index_base + i), BOTH writes the batch unchanged and then flipped: 2n sequences.
//
// Flips stay inside their rows, so the output has the input's flat layout -- shifted to start at 0, and in BOTH mode
// followed by a second copy of it.  The kernel therefore never walks rows: it is a flat map over the 16-byte aligned
// output vectors of a "virtual" batch of nv rows (n, or 2n in BOTH mode, where row n + i is input row i flipped), with
// virtual row starts start(r) = offsets[r] - offsets[0] (r <= n) and T + offsets[r - n] - offsets[0] (r > n).  Vectors are
// dealt in tiles of kRTile to a persistent grid in a static order (no tile counter, nothing survives a launch: the launch
// is capturable and may run concurrently with itself).  Per tile the CTA
//   1. finds the row of the tile's first byte with a 256-ary search over the virtual starts (K1v's search: two rounds up
//      to 66 049 rows, three up to 17 million);
//   2. loads the row table -- the tile's row starts and flip bits -- into shared memory, 256 rows a round, until a row
//      starts at or after the tile's end.  A tile with more than kRRowCap - 1 rows (rows shorter than 32 bytes on
//      average, or many empty ones) is "over-full" and reads starts and draws coins in global memory instead (step 3b);
//   3. per output vector: a binary search of the table for the row of its first byte, then for each row the vector
//      touches one whole-vector result merged in with a byte mask -- never element by element:
//        unflipped   two aligned 16-byte loads of the source (the shift is bytes + offsets[0] - out, launch-uniform
//                    outside BOTH's second half) and a funnel-shift realignment;
//        flipped     two aligned 16-byte loads of the mirrored source span (one contiguous range: a row's piece of any
//                    length mirrors to a piece of the same row), realignment, a byte reversal with PRMT and 16
//                    complement look-ups in shared memory.
//      Loads are clamped to the 16-byte words that hold a byte of the row, so nothing outside the input is touched.  A
//      vector inside [0, total) leaves as one st.global.cs.v4; the at most two partial vectors at the ends of the
//      output (d_out_bytes may have any alignment) are byte stores.
// out_offsets and the flip flags are written by the same launch (a grid-stride pass over the offsets it reads anyway).
// Every byte is read once and written once (twice in BOTH mode): the kernel is HBM-bound by design.
#include <cuda_runtime.h>

#include <cmath>

#include "bsq_internal.h"
#include "bsq_kernels.cuh"

namespace bsq {

namespace {

constexpr int kRThreads = 256;
constexpr int kRVecs = 16;                     // output vectors per thread and tile
constexpr int kRTile = kRThreads * kRVecs;     // 4096 vectors: 64 KiB of output per tile
constexpr int kRRowCap = 2048;                 // row-table entries: tiles of up to kRRowCap - 1 rows use the table
constexpr int kRMinBlocks = 4;                 // CTAs per SM

// The complement table of include/bsq.h: A<->T, C<->G, R<->Y, K<->M, B<->V, D<->H, U->A, the same in lower case; every
// other byte (S, W, N, gaps, '*', digits, bytes >= 0x80) maps to itself.  The only statement of it in the library.
struct CompTable {
    uint8_t c[256];
};
CompTable comp_table() {
    CompTable t;
    for (int b = 0; b < 256; ++b) t.c[b] = static_cast<uint8_t>(b);
    const char pairs[] = "ATCGRYKMBVDH";
    for (int i = 0; pairs[i] != 0; i += 2) {
        for (int lower = 0; lower < 2; ++lower) {
            const uint8_t x = static_cast<uint8_t>(pairs[i] | (lower << 5)), y = static_cast<uint8_t>(pairs[i + 1] | (lower << 5));
            t.c[x] = y;
            t.c[y] = x;
        }
    }
    t.c['U'] = 'A';
    t.c['u'] = 'a';
    return t;
}

struct RcParam {
    uint64_t gate;  // RANDOM: flip iff x0 < gate, gate in [0, 2^32]
    int64_t base;   // global index of this launch's sequence 0
    uint32_t k0, k1;
    int mode;
};

// flip of virtual row r (r < nv)
__device__ __forceinline__ bool rc_flip(int64_t r, int64_t n, const RcParam &p) {
    if (p.mode == BSQ_RC_BOTH) return r >= n;
    if (p.mode == BSQ_RC_ALWAYS) return true;
    const uint64_t g = static_cast<uint64_t>(p.base + r);
    const Philox x = philox4x32_10(static_cast<uint32_t>(g), static_cast<uint32_t>(g >> 32), 0u, 4u, p.k0, p.k1);
    return x.c[0] < p.gate;
}

struct RcBatch {
    const uint8_t *bytes;
    const uint8_t *comp;  // complement table in shared memory
    int64_t n, T, Tv, off0;
};

// Output bytes [q, q + 16) (out + q is 16-byte aligned), whose first byte in [0, Tv) lies in virtual row r.
// start_of(r) is the virtual start of row r (r <= nv), flip_of(r) its flip bit.
template <typename START, typename FLIP>
__device__ __forceinline__ void rc_vector(int64_t q, int64_t r, const RcBatch &b, const START &start_of, const FLIP &flip_of,
                                          uint8_t *dst) {
    uint32_t res[4] = {0u, 0u, 0u, 0u};
    const uintptr_t base = reinterpret_cast<uintptr_t>(b.bytes);
    int64_t s = start_of(r);
    for (;;) {
        const int64_t e = start_of(r + 1);
        if (e > s) {
            const int64_t sb = b.off0 - (r >= b.n ? b.T : 0);  // source index = virtual position + sb
            const uintptr_t lo = (base + static_cast<uintptr_t>(s + sb)) & ~uintptr_t(15);
            const uintptr_t hi = (base + static_cast<uintptr_t>(e - 1 + sb)) & ~uintptr_t(15);
            // unflipped: output position p reads source index p + sb; flipped: s + e - 1 + sb - p, so bytes q .. q + 15
            // mirror the 16 source bytes that end at s + e - 1 + sb - q
            const bool flip = flip_of(r);
            uint32_t t[4];
            fetch16_clamped(base + static_cast<uintptr_t>(flip ? s + e - 16 + sb - q : q + sb), lo, hi, t);
            if (flip) {
                const uint32_t w0 = t[0], w1 = t[1];
                t[0] = translate4(__byte_perm(t[3], 0u, 0x0123), b.comp);
                t[1] = translate4(__byte_perm(t[2], 0u, 0x0123), b.comp);
                t[2] = translate4(__byte_perm(w1, 0u, 0x0123), b.comp);
                t[3] = translate4(__byte_perm(w0, 0u, 0x0123), b.comp);
            }
            const int k0 = static_cast<int>(min(max(s - q, int64_t(0)), int64_t(16)));
            const int k1 = static_cast<int>(min(max(e - q, int64_t(0)), int64_t(16)));
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                const uint32_t m = lt_mask(k1, w) & ~lt_mask(k0, w);
                res[w] = (res[w] & ~m) | (t[w] & m);
            }
        }
        if (e >= q + 16 || e >= b.Tv) break;
        ++r;
        s = e;
    }
    if (q >= 0 && q + 16 <= b.Tv) {
        __stcs(reinterpret_cast<uint4 *>(dst), make_uint4(res[0], res[1], res[2], res[3]));
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (q + j >= 0 && q + j < b.Tv) dst[j] = static_cast<uint8_t>(res[j >> 2] >> (8 * (j & 3)));
    }
}

__global__ void __launch_bounds__(kRThreads, kRMinBlocks)
revcomp_kernel(const uint8_t *__restrict__ bytes, const int64_t *__restrict__ offs, int64_t n, LutParam lutp, RcParam p,
               uint8_t *__restrict__ out, int64_t *__restrict__ out_offs, uint8_t *__restrict__ flipped) {
    __shared__ __align__(256) uint8_t comp[256];
    __shared__ int64_t tab[kRRowCap];  // virtual starts of rows r0, r0 + 1, ...
    __shared__ uint8_t tflip[kRRowCap];
    load_lut(comp, lutp);
    RcBatch b;
    b.bytes = bytes;
    b.comp = comp;
    b.n = n;
    b.off0 = __ldg(offs);
    b.T = __ldg(offs + n) - b.off0;
    const bool both = p.mode == BSQ_RC_BOTH;
    const int64_t nv = both ? 2 * n : n;
    b.Tv = both ? 2 * b.T : b.T;
    auto start_g = [&](int64_t r) { return r <= n ? __ldg(offs + r) - b.off0 : b.T + __ldg(offs + r - n) - b.off0; };
    auto flip_g = [&](int64_t r) { return rc_flip(r, n, p); };
    for (int64_t i = blockIdx.x * static_cast<int64_t>(kRThreads) + threadIdx.x; i <= nv; i += static_cast<int64_t>(gridDim.x) * kRThreads) {
        out_offs[i] = start_g(i);
        if (flipped != nullptr && i < nv) flipped[i] = flip_g(i);
    }
    __syncthreads();
    const int a = static_cast<int>(reinterpret_cast<uintptr_t>(out) & 15u);  // out - a is 16-byte aligned
    const int64_t nvec = b.Tv > 0 ? (b.Tv - 1 + a) / 16 + 1 : 0;             // vector v holds bytes [16v - a, 16v - a + 16)
    const int64_t ntiles = (nvec + kRTile - 1) / kRTile;
    const int tid = threadIdx.x;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t v0 = tile * kRTile;
        const int64_t p0 = max(16 * v0 - a, int64_t(0)), p1 = min(16 * (v0 + kRTile) - a, b.Tv);
        // 1. first row: the largest r in [0, nv) with start(r) <= p0
        int64_t lo = 0, hi = nv;
        while (hi - lo > 1) {
            const int64_t w = hi - lo;
            const int64_t pr = lo + (static_cast<int64_t>(tid) + 1) * w / (kRThreads + 1);
            const int cnt = __syncthreads_count(start_g(pr) <= p0);  // a prefix of the probes (starts are non-decreasing)
            const int64_t nlo = cnt > 0 ? lo + static_cast<int64_t>(cnt) * w / (kRThreads + 1) : lo;
            const int64_t nhi = cnt < kRThreads ? lo + (static_cast<int64_t>(cnt) + 1) * w / (kRThreads + 1) : hi;
            lo = nlo;
            hi = nhi;
        }
        const int64_t r0 = lo;
        // 2. row table up to the first row that starts at or after the tile's end (row nv starts at Tv >= p1, so that
        //    entry exists and closes the table)
        int nrows = -1;
        for (int base = 0; base < kRRowCap; base += kRThreads) {
            const int j = base + tid;
            const int64_t r = r0 + j;
            bool past = true;
            if (r <= nv) {
                const int64_t s = start_g(r);
                tab[j] = s;
                tflip[j] = r < nv && flip_g(r);
                past = s >= p1;
            }
            const int cnt = __syncthreads_count(past);  // a suffix of the chunk
            if (cnt > 0) {
                nrows = base + kRThreads - cnt;
                break;
            }
        }
        if (nrows > 0) {
            // 3a. rows from the table
            auto start_t = [&](int64_t r) { return tab[r - r0]; };
            auto flip_t = [&](int64_t r) { return tflip[r - r0] != 0; };
            for (int k = 0; k < kRVecs; ++k) {
                const int64_t v = v0 + k * kRThreads + tid;
                if (v >= nvec) break;
                const int64_t q = 16 * v - a, x = max(q, int64_t(0));
                int l = 0, h = nrows;  // largest j < nrows with tab[j] <= x
                while (h - l > 1) {
                    const int mid = (l + h) >> 1;
                    if (tab[mid] <= x) l = mid;
                    else h = mid;
                }
                rc_vector(q, r0 + l, b, start_t, flip_t, out + q);
            }
        } else {
            // 3b. over-full tile: rows searched and coins drawn in global memory
            for (int k = 0; k < kRVecs; ++k) {
                const int64_t v = v0 + k * kRThreads + tid;
                if (v >= nvec) break;
                const int64_t q = 16 * v - a, x = max(q, int64_t(0));
                int64_t l = r0, h = nv;
                while (h - l > 1) {
                    const int64_t mid = (l + h) >> 1;
                    if (start_g(mid) <= x) l = mid;
                    else h = mid;
                }
                rc_vector(q, l, b, start_g, flip_g, out + q);
            }
        }
        __syncthreads();  // the table is refilled by the next tile
    }
}

}  // namespace

}  // namespace bsq

using namespace bsq;

extern "C" int bsq_revcomp_table(uint8_t out[256]) {
    if (out == nullptr) return fail(BSQ_ERR_ARG, "null output table");
    const CompTable t = comp_table();
    for (int i = 0; i < 256; ++i) out[i] = t.c[i];
    return BSQ_OK;
}

extern "C" int bsq_revcomp(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq, int mode,
                           double rc_prob, uint64_t seed, int64_t seq_index_base, uint8_t *d_out_bytes, int64_t *d_out_offsets,
                           uint8_t *d_flipped) {
    bsq::DeviceRestore restore_device;
    if (mode != BSQ_RC_ALWAYS && mode != BSQ_RC_RANDOM && mode != BSQ_RC_BOTH)
        return fail(BSQ_ERR_ARG, "mode must be BSQ_RC_ALWAYS, BSQ_RC_RANDOM or BSQ_RC_BOTH");
    if (std::isnan(rc_prob) || rc_prob < 0.0) return fail(BSQ_ERR_ARG, "rc_prob must be >= 0");
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
    const CompTable t = comp_table();
    LutParam lut;
    for (int w = 0; w < 64; ++w)
        lut.w[w] = t.c[4 * w] | (t.c[4 * w + 1] << 8) | (t.c[4 * w + 2] << 16) | (static_cast<uint32_t>(t.c[4 * w + 3]) << 24);
    RcParam p;
    p.gate = rc_prob >= 1.0 ? (uint64_t(1) << 32) : static_cast<uint64_t>(std::floor(rc_prob * 4294967296.0));
    p.base = seq_index_base;
    p.k0 = static_cast<uint32_t>(seed);
    p.k1 = static_cast<uint32_t>(seed >> 32);
    p.mode = mode;
    revcomp_kernel<<<cur_sms() * kRMinBlocks, kRThreads, 0, st>>>(d_bytes, d_offsets, nseq, lut, p, d_out_bytes, d_out_offsets,
                                                                  d_flipped);
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}
