// K12: reverse complement of a packed batch (sm_100a).
//
// Semantics (include/bsq.h, bsq_revcomp): out[j] = comp[in[len - 1 - j]] for a flipped sequence, a copy otherwise.
// ALWAYS flips every sequence, RANDOM sequence i iff x0 < gate (x0 = word 0 of Philox4x32-10 at counter (g_lo, g_hi, 0, 4),
// g = seq_index_base + i), BOTH writes the batch unchanged and then flipped: 2n sequences.
//
// Flips stay inside their rows, so the output has the input's flat layout -- shifted to start at 0, and in BOTH mode
// followed by a second copy of it.  The kernel is therefore bsq_kernels.cuh's flat map over a "virtual" batch of nv rows
// (n, or 2n in BOTH mode, where row n + i is input row i flipped), with virtual row starts start(r) = offsets[r] -
// offsets[0] (r <= n) and T + offsets[r - n] - offsets[0] (r > n).  Its row data is the flip bit (one Philox block per
// row, staged in the table; over-full tiles draw coins in global memory), and its piece of a row is one whole-vector
// result:
//   unflipped   two aligned 16-byte loads of the source (the shift is bytes + offsets[0] - out, launch-uniform outside
//               BOTH's second half) and a funnel-shift realignment;
//   flipped     two aligned 16-byte loads of the mirrored source span (one contiguous range: a row's piece of any length
//               mirrors to a piece of the same row), realignment, a byte reversal with PRMT and 16 complement look-ups
//               in shared memory.
// Loads are clamped to the 16-byte words that hold a byte of the row, so nothing outside the input is touched.
// out_offsets and the flip flags are written by the same launch (a grid-stride pass over the offsets it reads anyway).
// Every byte is read once and written once (twice in BOTH mode): the kernel is HBM-bound by design.
#include <cuda_runtime.h>

#include <cmath>

#include "bsq_internal.h"
#include "bsq_kernels.cuh"

namespace bsq {

namespace {

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

// K12's rows for flat_map: the nv virtual rows, and their flip bits as row data
struct RcMap {
    const uint8_t *bytes;
    const int64_t *offs;
    const uint8_t *comp;  // complement table in shared memory
    uint8_t *tflip;       // flip bits of the tile's rows, in shared memory
    int64_t n, nv, T, off0;
    RcParam p;

    __device__ __forceinline__ int64_t start(int64_t r) const {
        return r <= n ? __ldg(offs + r) - off0 : T + __ldg(offs + r - n) - off0;
    }
    __device__ __forceinline__ bool row_g(int64_t r) const { return rc_flip(r, n, p); }
    __device__ __forceinline__ void stage(int j, int64_t r) const { tflip[j] = r < nv && row_g(r); }
    __device__ __forceinline__ bool row_t(int j) const { return tflip[j] != 0; }
    __device__ __forceinline__ void piece(int64_t q, int64_t r, int64_t s, int64_t e, bool flip, uint32_t res[4]) const {
        const uintptr_t base = reinterpret_cast<uintptr_t>(bytes);
        const int64_t sb = off0 - (r >= n ? T : 0);  // source index = virtual position + sb
        const uintptr_t lo = (base + static_cast<uintptr_t>(s + sb)) & ~uintptr_t(15);
        const uintptr_t hi = (base + static_cast<uintptr_t>(e - 1 + sb)) & ~uintptr_t(15);
        // unflipped: output position p reads source index p + sb; flipped: s + e - 1 + sb - p, so bytes q .. q + 15
        // mirror the 16 source bytes that end at s + e - 1 + sb - q
        uint32_t t[4];
        fetch_clamped<4>(base + static_cast<uintptr_t>(flip ? s + e - 16 + sb - q : q + sb), lo, hi, t);
        if (flip) {
            const uint32_t w0 = t[0], w1 = t[1];
            t[0] = translate4(__byte_perm(t[3], 0u, 0x0123), comp);
            t[1] = translate4(__byte_perm(t[2], 0u, 0x0123), comp);
            t[2] = translate4(__byte_perm(w1, 0u, 0x0123), comp);
            t[3] = translate4(__byte_perm(w0, 0u, 0x0123), comp);
        }
        merge16(res, t, s - q, e - q);
    }
};

__global__ void __launch_bounds__(kFlatThreads, kFlatMinBlocks)
revcomp_kernel(const uint8_t *__restrict__ bytes, const int64_t *__restrict__ offs, int64_t n, LutParam lutp, RcParam p,
               uint8_t *__restrict__ out, int64_t *__restrict__ out_offs, uint8_t *__restrict__ flipped) {
    __shared__ __align__(256) uint8_t comp[256];
    __shared__ uint8_t tflip[kFlatRowCap];
    load_lut(comp, lutp);
    RcMap m;
    m.bytes = bytes;
    m.offs = offs;
    m.comp = comp;
    m.tflip = tflip;
    m.n = n;
    m.p = p;
    m.off0 = __ldg(offs);
    m.T = __ldg(offs + n) - m.off0;
    const bool both = p.mode == BSQ_RC_BOTH;
    m.nv = both ? 2 * n : n;
    for (int64_t i = blockIdx.x * static_cast<int64_t>(kFlatThreads) + threadIdx.x; i <= m.nv; i += static_cast<int64_t>(gridDim.x) * kFlatThreads) {
        out_offs[i] = m.start(i);
        if (flipped != nullptr && i < m.nv) flipped[i] = m.row_g(i);
    }
    __syncthreads();
    flat_map(out, m.nv, both ? 2 * m.T : m.T, m);
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
    revcomp_kernel<<<cur_sms() * kFlatMinBlocks, kFlatThreads, 0, st>>>(d_bytes, d_offsets, nseq, lut, p, d_out_bytes,
                                                                        d_out_offsets, d_flipped);
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    return BSQ_OK;
}
