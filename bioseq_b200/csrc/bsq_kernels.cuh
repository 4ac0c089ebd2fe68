// Device-side building blocks of the sm_100a tokeniser kernels (see DESIGN.md section 3).
//
// Everything here is an elementwise byte map bounded by HBM bandwidth; no tensor cores.
// The shared pieces are
//   * a 256-entry byte LUT staged in shared memory (ASCII inputs never bank-conflict:
//     bytes 0..127 live in 32 distinct 4-byte words),
//   * `tokens16`: 16 consecutive output codes of one row -- two 16-byte aligned
//     ld.global.nc loads of the packed residues (clamped to the words that hold the row),
//     an in-register realignment (sequence starts are arbitrary byte offsets and BOS shifts
//     the row by one), 16 LUT look-ups, and BOS / EOS / PAD synthesised by byte masks on the
//     boundary chunks only,
//   * a scalar `token_at` for ragged edges and multi-byte element types.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "bsq_internal.h"

struct bsq_tokenizer;
struct bsq_mlm;

namespace bsq {

struct LutParam {
    uint32_t w[64];  // 256 byte codes, passed by value in kernel parameter space
};

struct SeqView {
    const uint8_t *bytes;  // packed residues
    const int64_t *offs;   // nseq + 1 offsets into bytes
    const uint8_t *mask;   // optional (one-hot only), indexed like bytes
};

// Byte codes (replicated into all four bytes of a word) for the non-residue columns.
struct Specials {
    uint32_t bos_w, eos_w, pad_w;
    int bos, eos;  // 0/1: symbol present
};

// Tile kernels keep one byte per token in shared memory.  Codes < 0x80 are ids; codes
// 0xFC..0xFF index this 4-entry table (ids that do not fit a byte -- BYTES alphabet --
// and "leave the one-hot row zero").
struct Expand {
    int32_t map[4];  // [0]=pad  [1]=eos  [2]=bos  [3]=invalid
};
constexpr uint32_t kCodePad = 0xFC, kCodeEos = 0xFD, kCodeBos = 0xFE, kCodeInvalid = 0xFF;

// n / d for 0 <= n < 2^31, 1 <= d < 2^31 (Granlund-Montgomery round-up multiplier).
struct FastDiv {
    uint32_t mul, shift, d;
};
__host__ __device__ inline FastDiv make_fastdiv(uint32_t d) {
    FastDiv f;
    f.d = d;
    uint32_t l = 0;
    while ((1ull << l) < d) ++l;
    f.shift = l;
    f.mul = static_cast<uint32_t>((((1ull << l) - d) << 32) / d + 1);
    return f;
}
__host__ __device__ __forceinline__ uint32_t fd_div(uint32_t n, const FastDiv &f) {
    const uint32_t t = static_cast<uint32_t>((static_cast<uint64_t>(n) * f.mul) >> 32);
    return (t + n) >> f.shift;
}

// Kernel-side form of a tokenizer (built on the host by prepare(), bsq_kernels.cu):
// mode 0: batch-first one-byte tokens (codes are the output bytes), mode 1: tokens through Expand
// (wide element types, tile kernels, embedding gather), mode 2: one-hot columns through Expand.
struct Prepared {
    LutParam lut;
    Specials sp;
    Expand ex;
};
Prepared prepare(const bsq_tokenizer &tok, int mode);

// K1s (bsq_span.cu): batch-first one-byte tokens, tile-staged and warp-specialised.  It runs every padlen above
// kSpanMinPadlen (up to the 2^30 every entry point allows); shorter rows share warps in K1.
constexpr int64_t kSpanMinPadlen = 256;
inline bool span_kernel_applicable(int64_t padlen) { return padlen > kSpanMinPadlen; }
int sm_count(int device);  // SMs of the device (cached per device)
inline int cur_sms() {     // ... of the current device (the entry points have made the call's device current)
    int d = 0;
    cudaGetDevice(&d);
    return sm_count(d);
}
int launch_tokenize_span(int device, cudaStream_t st, const SeqView &v, int64_t nseq, int64_t padlen, const Prepared &p,
                         uint8_t *out);
// A slot of the per-stream tile counters of the dynamic schedulers (bsq_span.cu), or nullptr when none can be used
// (stream capture in progress, out of memory): the kernels then keep their static tile order.
unsigned int *tile_counter_slot(int device, cudaStream_t st);
// n / d = umulhi(n, mul) >> shift for 0 <= n < 2^31, 2 <= d <= 2^30.
void span_magic(uint32_t d, uint32_t *mul, uint32_t *shift);
constexpr int kSpanManyMax = 32;  // batches per launch of launch_tokenize_span_many
int launch_tokenize_span_many(int device, cudaStream_t st, int nbatch, const uint8_t *const *d_bytes, const int64_t *const *d_offs,
                              const int64_t *nseqs, int64_t padlen, const Prepared &p, uint8_t *const *outs);

// Masked-language-model parameters (include/bsq.h, bsq_mlm) in kernel form, and below the per-residue selection and
// corruption shared by K8 (bsq_mlm.cu) and K10 (bsq_seqpack.cu).
struct MlmParam {
    uint32_t k0, k1;      // Philox key (seed)
    uint64_t ts, tm, tr;  // t_select, t_mask, t_random, each in [0, 2^32]
    int64_t base;         // global index of this launch's sequence 0
    int64_t ignore;       // label of positions that are not selected
    int32_t mask_id;
    uint32_t nchars;
};
// Validates a bsq_mlm for `kind` (BSQ_ERR_ARG with the message of include/bsq.h) and fills *m (bsq_mlm.cu).
int check_mlm_param(const bsq_tokenizer *tok, int kind, const bsq_mlm *mlm, MlmParam *m);

// The token count of one k-mer row (include/bsq.h, bsq_kmer): the only statement of T(n), used by the host extent, the
// device extent and K11 (bsq_kmer.cu).  sdiv divides by the stride.
struct KmerShape {
    int32_t k, s, single, bos, eos;
    FastDiv sdiv;
};
struct KmerCount {
    int64_t m;        // k-mers, starting at residues 0, s, 2s, ...
    int64_t covered;  // residues they cover
    int64_t tail;     // residues after them that become single tokens (0 when dropped)
};
__host__ __device__ inline KmerCount kmer_count(int64_t n, const KmerShape &ks) {
    KmerCount c;
    const int64_t d = n - ks.k;
    c.m = d < 0 ? 0 : (d < (int64_t(1) << 31) ? static_cast<int64_t>(fd_div(static_cast<uint32_t>(d), ks.sdiv)) : d / ks.s) + 1;
    c.covered = c.m > 0 ? (c.m - 1) * ks.s + ks.k : 0;
    c.tail = ks.single ? n - c.covered : 0;
    return c;
}
// T(n) = m + (single ? r : 0) + bos + eos.  m + r <= n, so only the specials can take T past INT64_MAX (n within two of
// it): the sum wraps to a negative value then, which KmerCountFn::extent reports.
__host__ __device__ inline int64_t kmer_tokens(int64_t n, const KmerShape &ks) {
    const KmerCount c = kmer_count(n, ks);
    return static_cast<int64_t>(static_cast<uint64_t>(c.m + c.tail) + ks.bos + ks.eos);
}

// ---- offsets reductions: validate a packed batch's offsets and size an output from them ------------------------------
// Each feature states its per-row share as a measure, m.extent(len) for a row of len >= 0: two sums and a max, each in
// [0, INT64_MAX], and whether one had to be clamped.  reduce_offsets_host and reduce_offsets_device (below) add the rows
// up with the same measure, so host and device extents cannot disagree.
constexpr int64_t kI64Max = INT64_MAX;
struct Extent {
    int64_t sum0, sum1, max;
    bool over;  // a value passed INT64_MAX (it is clamped there)
};
// a + b for a, b in [0, INT64_MAX], clamped to INT64_MAX
__host__ __device__ __forceinline__ int64_t add_sat(int64_t a, int64_t b, bool *over) {
    if (a > kI64Max - b) {
        *over = true;
        return kI64Max;
    }
    return a + b;
}
// v >= 0 clamped to INT64_MAX
__host__ __device__ __forceinline__ int64_t clamp_sat(__int128 v, bool *over) {
    if (v > kI64Max) {
        *over = true;
        return kI64Max;
    }
    return static_cast<int64_t>(v);
}

// The kept length min(len, W) of a crop (K9's scan, K0c), and with W = INT64_MAX the length itself (K0): the sum and the
// max of the kept lengths.
struct CropCount {
    int64_t W;
    __host__ __device__ __forceinline__ int64_t operator()(int64_t len) const { return len < W ? len : W; }
    __host__ __device__ __forceinline__ Extent extent(int64_t len) const { return {(*this)(len), 0, (*this)(len), false}; }
};

#ifdef __CUDACC__

__device__ __forceinline__ uint4 ldg16(uintptr_t addr) {
    return __ldg(reinterpret_cast<const uint4 *>(addr));
}

__device__ __forceinline__ uintptr_t clamp_word(uintptr_t a, uintptr_t lo, uintptr_t hi) { return a < lo ? lo : (a > hi ? hi : a); }

// The 4 * kWords bytes at address X (any alignment) as kWords little-endian words (kWords a multiple of 4), from the
// aligned 16-byte words at X & ~15 and the kWords / 4 after it (the last only when X is not aligned), each clamped to
// [lo, hi] (16-byte aligned).  The shift may vary from thread to thread, so the words are picked with selects.  K12 and
// K13a read 16 bytes, K14b 48.
template <int kWords>
__device__ __forceinline__ void fetch_clamped(uintptr_t X, uintptr_t lo, uintptr_t hi, uint32_t t[kWords]) {
    const uintptr_t a0 = X & ~uintptr_t(15);
    const uint32_t s = static_cast<uint32_t>(X) & 15u;
    uint32_t w[kWords + 4];
#pragma unroll
    for (int k = 0; k <= kWords / 4; ++k) {
        const uint4 v = k < kWords / 4 || s != 0 ? ldg16(clamp_word(a0 + 16 * k, lo, hi)) : make_uint4(0u, 0u, 0u, 0u);
        w[4 * k] = v.x;
        w[4 * k + 1] = v.y;
        w[4 * k + 2] = v.z;
        w[4 * k + 3] = v.w;
    }
    const bool q2 = (s & 8u) != 0, q1 = (s & 4u) != 0;
    uint32_t a[kWords + 2], b[kWords + 1];
#pragma unroll
    for (int k = 0; k < kWords + 2; ++k) a[k] = q2 ? w[k + 2] : w[k];
#pragma unroll
    for (int k = 0; k < kWords + 1; ++k) b[k] = q1 ? a[k + 1] : a[k];
    const uint32_t sh = (s & 3u) * 8u;
#pragma unroll
    for (int k = 0; k < kWords; ++k) t[k] = __funnelshift_r(b[k], b[k + 1], sh);
}

__device__ __forceinline__ void load_lut(uint8_t *lut_smem, const LutParam &p) {
    if (threadIdx.x < 64) reinterpret_cast<uint32_t *>(lut_smem)[threadIdx.x] = p.w[threadIdx.x];
}

// Mask of the bytes j < k of a 16-byte chunk that fall in 32-bit word `w` (j = 4w..4w+3):
// the high word of (0:ffffffff) << clamp(8*(k-4w), 0, 32) -- one VIADDMNMX + one SHF.L.W.
// k must already be clamped to [0, 16].
__device__ __forceinline__ uint32_t lt_mask(int k, int w) {
    return __funnelshift_lc(0xffffffffu, 0u, static_cast<uint32_t>(max(8 * k - 32 * w, 0)));
}
__device__ __forceinline__ int clamp16(int k) { return min(max(k, 0), 16); }

// Four LUT look-ups: byte extraction with PRMT (one ALU op each), LDS.U8, and the re-packing as
// integer multiply-adds so it lands on the FMA pipe instead of the (half-rate) ALU pipe.
__device__ __forceinline__ uint32_t translate4(uint32_t x, const uint8_t *lut) {
    const uint32_t b0 = lut[__byte_perm(x, 0u, 0x4440)];
    const uint32_t b1 = lut[__byte_perm(x, 0u, 0x4441)];
    const uint32_t b2 = lut[__byte_perm(x, 0u, 0x4442)];
    const uint32_t b3 = lut[__byte_perm(x, 0u, 0x4443)];
    return b0 + b1 * 0x100u + b2 * 0x10000u + b3 * 0x1000000u;
}

// Where the bytes of one row live: column c of the row (BOS shift included) is al[off + c].
// `al` is 16-byte aligned; fw/lw are the byte offsets (multiples of 16, relative to al) of the
// first and last aligned 16-byte words that hold a residue of this row.  Loads are clamped to
// [fw, lw], so nothing outside words containing valid residues is ever touched, whatever
// column range is asked for (a clamped word only ever replaces bytes that are masked out).
struct RowSrc {
    const uint8_t *al;
    int off, fw, lw;
};
__device__ __forceinline__ RowSrc make_rowsrc(const uint8_t *base, int64_t start, int bos, int len) {
    const uint8_t *src = base + start - bos;
    RowSrc r;
    r.off = static_cast<int>(reinterpret_cast<uintptr_t>(src) & 15u);
    r.al = src - r.off;
    r.fw = (r.off + bos) & ~15;
    r.lw = (r.off + bos + len - 1) & ~15;
    return r;
}

// The 16 bytes of columns c0 .. c0+15, in two steps so that callers can issue the loads of
// several chunks before consuming any of them:
//   fetch_issue   two aligned 16-byte ld.global.nc loads (the second only when the chunk is not
//                 16-byte aligned in the source),
//   fetch_align   funnel-shift realignment into four little-endian words.
// The byte shift (off + c0) & 15 is the same for every chunk of a row, so when a warp works on
// one row the switch is warp-uniform.
struct Fetched {
    uint4 v0, v1;
};
__device__ __forceinline__ Fetched fetch_issue(const RowSrc &rs, int c0) {
    const int a = rs.off + c0;
    const int a0 = a & ~15;
    Fetched f;
    f.v0 = ldg16(reinterpret_cast<uintptr_t>(rs.al) + static_cast<uint32_t>(min(max(a0, rs.fw), rs.lw)));
    f.v1 = make_uint4(0u, 0u, 0u, 0u);
    if ((a & 15) != 0)
        f.v1 = ldg16(reinterpret_cast<uintptr_t>(rs.al) + static_cast<uint32_t>(min(max(a0 + 16, rs.fw), rs.lw)));
    return f;
}
__device__ __forceinline__ void fetch_align(const Fetched &f, const RowSrc &rs, int c0, uint32_t out[4]) {
    const uint32_t s = static_cast<uint32_t>(rs.off + c0) & 15u;
    const uint32_t sh = (s & 3u) * 8u;
    const uint4 &v0 = f.v0, &v1 = f.v1;
    switch (s >> 2) {
        case 0:
            out[0] = __funnelshift_r(v0.x, v0.y, sh); out[1] = __funnelshift_r(v0.y, v0.z, sh);
            out[2] = __funnelshift_r(v0.z, v0.w, sh); out[3] = __funnelshift_r(v0.w, v1.x, sh);
            break;
        case 1:
            out[0] = __funnelshift_r(v0.y, v0.z, sh); out[1] = __funnelshift_r(v0.z, v0.w, sh);
            out[2] = __funnelshift_r(v0.w, v1.x, sh); out[3] = __funnelshift_r(v1.x, v1.y, sh);
            break;
        case 2:
            out[0] = __funnelshift_r(v0.z, v0.w, sh); out[1] = __funnelshift_r(v0.w, v1.x, sh);
            out[2] = __funnelshift_r(v1.x, v1.y, sh); out[3] = __funnelshift_r(v1.y, v1.z, sh);
            break;
        default:
            out[0] = __funnelshift_r(v0.w, v1.x, sh); out[1] = __funnelshift_r(v1.x, v1.y, sh);
            out[2] = __funnelshift_r(v1.y, v1.z, sh); out[3] = __funnelshift_r(v1.z, v1.w, sh);
            break;
    }
}
__device__ __forceinline__ void fetch16(const RowSrc &rs, int c0, uint32_t out[4]) {
    const Fetched f = fetch_issue(rs, c0);
    fetch_align(f, rs, c0, out);
}
// does the chunk starting at column c0 hold at least one residue?
__device__ __forceinline__ bool has_residues(int c0, int bos, int len) {
    const int r0 = c0 - bos;
    return min(r0 + 16, len) > max(r0, 0);
}

// Per-CTA shared-memory tables for the chunk that holds the end of a row: for k = 0..16 leading
// bytes that are still BOS/residues, m[k] keeps those bytes and f[k] supplies the rest (EOS at
// byte k when the tokenizer has one, the pad code after it).  Two LDS.128 + four LOP3 replace
// ~70 mask-building instructions per tail chunk.
struct TailTab {
    uint4 m[17];
    uint4 f[17];
};
__device__ __forceinline__ void init_tailtab(TailTab &tab, const Specials &sp) {
    const int k = static_cast<int>(threadIdx.x) - 64;  // threads 64..80 (0..63 load the LUT)
    if (k >= 0 && k <= 16) {
        uint32_t m[4], f[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            m[w] = lt_mask(k, w);
            const uint32_t m_eos = lt_mask(clamp16(k + sp.eos), w);
            f[w] = (sp.eos_w & m_eos & ~m[w]) | (sp.pad_w & ~m_eos);
        }
        tab.m[k] = make_uint4(m[0], m[1], m[2], m[3]);
        tab.f[k] = make_uint4(f[0], f[1], f[2], f[3]);
    }
}

// Codes of columns c0 .. c0+15 of a row with `len` residues, for c0 < bos + len + eos (the
// caller emits the constant pad vector beyond that).  Column layout (src/tokenize.h:460-478):
//   [0, bos)            BOS
//   [bos, bos+len)      lut[residue]
//   bos+len             EOS (if eos)
//   beyond              pad code
// With MAYBE_NEG, c0 may be negative (rows that do not start 16-byte aligned in the output);
// bytes left of column 0 are don't-care.  `ms` is the row's mask source (one-hot only) or nullptr.
template <bool MAYBE_NEG>
__device__ __forceinline__ uint4 tokens16_finish(uint32_t t[4], int len, int c0, const Specials &sp, const TailTab &tab) {
    const int n = sp.bos + len;  // column of EOS
    if (MAYBE_NEG && c0 < 0) {
        const int kr0 = clamp16(sp.bos - c0), kr1 = clamp16(n - c0), kr2 = clamp16(n + sp.eos - c0);
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const uint32_t m_bos = lt_mask(kr0, w);
            const uint32_t m_res = lt_mask(kr1, w);
            const uint32_t m_eos = lt_mask(kr2, w);
            t[w] = (sp.bos_w & m_bos) | (t[w] & m_res & ~m_bos) | (sp.eos_w & m_eos & ~m_res) | (sp.pad_w & ~m_eos);
        }
    } else {
        if (c0 < sp.bos) t[0] = __byte_perm(t[0], sp.bos_w, 0x3214);  // c0 == 0: column 0 is BOS
        if (c0 + 16 > n) {                                           // the row ends inside this chunk
            const uint4 m = tab.m[n - c0], f = tab.f[n - c0];
            t[0] = (t[0] & m.x) | f.x; t[1] = (t[1] & m.y) | f.y;
            t[2] = (t[2] & m.z) | f.z; t[3] = (t[3] & m.w) | f.w;
        }
    }
    return make_uint4(t[0], t[1], t[2], t[3]);
}

template <bool MAYBE_NEG>
__device__ __forceinline__ uint4 tokens16(const RowSrc &rs, const RowSrc *ms, int len, int c0,
                                          const Specials &sp, const uint8_t *lut, const TailTab &tab) {
    uint32_t t[4] = {0u, 0u, 0u, 0u};
    if (has_residues(c0, sp.bos, len)) {
        uint32_t raw[4];
        fetch16(rs, c0, raw);
#pragma unroll
        for (int w = 0; w < 4; ++w) t[w] = translate4(raw[w], lut);
        if (ms != nullptr) {  // masked-out residues become kCodeInvalid (0xFF)
            uint32_t m[4];
            fetch16(*ms, c0, m);
#pragma unroll
            for (int w = 0; w < 4; ++w) t[w] |= __vcmpeq4(m[w], 0u);
        }
    }
    return tokens16_finish<MAYBE_NEG>(t, len, c0, sp, tab);
}

// Same result as tokens16 (no mask) from loads issued earlier with fetch_issue.
template <bool MAYBE_NEG>
__device__ __forceinline__ uint4 tokens16_from(const Fetched &f, bool loaded, const RowSrc &rs, int len, int c0,
                                               const Specials &sp, const uint8_t *lut, const TailTab &tab) {
    uint32_t t[4] = {0u, 0u, 0u, 0u};
    if (loaded) {
        uint32_t raw[4];
        fetch_align(f, rs, c0, raw);
#pragma unroll
        for (int w = 0; w < 4; ++w) t[w] = translate4(raw[w], lut);
    }
    return tokens16_finish<MAYBE_NEG>(t, len, c0, sp, tab);
}

// One code, any column: the scalar twin of tokens16.
__device__ __forceinline__ uint32_t token_at(const SeqView &v, int64_t start, int len, int c,
                                             const Specials &sp, const uint8_t *lut) {
    const int r = c - sp.bos;
    if (r < 0) return sp.bos_w & 0xffu;
    if (r < len) {
        uint32_t code = lut[__ldg(v.bytes + start + r)];
        if (v.mask != nullptr && __ldg(v.mask + start + r) == 0) code = kCodeInvalid;
        return code;
    }
    if (r == len && sp.eos) return sp.eos_w & 0xffu;
    return sp.pad_w & 0xffu;
}

__device__ __forceinline__ int32_t expand_code(uint32_t code, const Expand &ex) {
    return code < 0x80u ? static_cast<int32_t>(code) : ex.map[code & 3u];
}

// Philox4x32-10 (Salmon et al., SC'11), the counter-based generator of K7 (BLOSUM62 augmentation, counter word 3 = 0)
// and K8 (masked-language-model batches, counter word 3 = 1 and 2): one block of four 32-bit words per counter.
struct Philox {
    uint32_t c[4];
};
__device__ __forceinline__ Philox philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    Philox p;
    p.c[0] = c0; p.c[1] = c1; p.c[2] = c2; p.c[3] = c3;
    return p;
}

// Exclusive prefix sum of one int64 per thread over the whole block (blockDim.x a multiple of 32, at most 1024);
// *total receives the block's sum.  s_warp: 32 entries of shared memory.  Every thread of the block must call it.
// Used by the decode scan (K4) and the crop's output offsets (K9).
__device__ __forceinline__ int64_t block_exclusive_scan(int64_t x, int64_t *s_warp, int64_t *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t incl = x;
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t y = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += y;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int64_t wv = lane < (blockDim.x >> 5) ? s_warp[lane] : 0;
        int64_t wi = wv;
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t y = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += y;
        }
        s_warp[lane] = wi - wv;  // exclusive prefix of the warp totals
        if (lane == 31) *total = wi;
    }
    __syncthreads();
    return s_warp[warp] + incl - x;
}

// Exclusive scan of a per-row count over a packed batch, in two launches without scratch memory (K9's crop offsets, K11's
// cu_seqlens).  count(len) is the row's count from its length; Out the element type of the offsets array.
//   row_scan_kernel   one thread per row, kRowScan rows per CTA: the CTA's inclusive scan of count(len_i) goes to
//                     out[i + 1] (and out[0] = 0), so the entry at the end of each CTA's rows is that CTA's total.
//   row_carry_kernel  one CTA, only when there is more than one scan CTA: scans the CTA totals in place, so every entry
//                     at the end of a scan CTA's rows becomes final.
// The consumer then finishes entry e itself by adding row_scan_carry (below).
constexpr int kRowScan = 1024;  // block_exclusive_scan handles up to 1024 threads

template <typename Count, typename Out>
__global__ void __launch_bounds__(kRowScan)
row_scan_kernel(const int64_t *__restrict__ offs, int64_t n, Count count, Out *__restrict__ out_offs) {
    __shared__ int64_t s_warp[32];
    __shared__ int64_t s_total;
    const int64_t i = static_cast<int64_t>(blockIdx.x) * kRowScan + threadIdx.x;
    const int64_t kept = i < n ? count(__ldg(offs + i + 1) - __ldg(offs + i)) : 0;
    const int64_t ex = block_exclusive_scan(kept, s_warp, &s_total);
    if (i < n) out_offs[i + 1] = static_cast<Out>(ex + kept);
    if (i == 0) out_offs[0] = 0;
}

// entry e = min((b + 1) * kRowScan, n) holds scan CTA b's total; it becomes the inclusive prefix over CTAs 0 .. b
template <typename Out>
__global__ void __launch_bounds__(kRowScan)
row_carry_kernel(Out *__restrict__ out_offs, int64_t n, int64_t nblocks) {
    __shared__ int64_t s_warp[32];
    __shared__ int64_t s_total;
    int64_t carry = 0;
    for (int64_t base = 0; base < nblocks; base += kRowScan) {
        const int64_t b = base + threadIdx.x;
        const int64_t e = min((b + 1) * kRowScan, n);
        const int64_t x = b < nblocks ? static_cast<int64_t>(out_offs[e]) : 0;
        const int64_t ex = block_exclusive_scan(x, s_warp, &s_total);
        if (b < nblocks) out_offs[e] = static_cast<Out>(carry + ex + x);
        carry += s_total;
        __syncthreads();
    }
}

// row_scan_kernel, and row_carry_kernel past kRowScan rows, enqueued on st
template <typename Count, typename Out>
int launch_row_scan(cudaStream_t st, const int64_t *d_offs, int64_t n, Count count, Out *out_offs) {
    const int64_t nblocks = (n + kRowScan - 1) / kRowScan;
    row_scan_kernel<<<static_cast<unsigned>(nblocks), kRowScan, 0, st>>>(d_offs, n, count, out_offs);
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    if (nblocks > 1) {
        row_carry_kernel<<<1, kRowScan, 0, st>>>(out_offs, n, nblocks);
        count_launch();
        BSQ_CUDA_TRY(cudaGetLastError());
    }
    return BSQ_OK;
}

// What entry e of launch_row_scan's n + 1 entries still lacks: the entry that closes the previous scan CTA, or 0 when e
// lies in the first scan CTA or closes a scan CTA or the batch (those entries are final, and never written by a
// consumer, so every thread may read them).
template <typename Out>
__device__ __forceinline__ int64_t row_scan_carry(const Out *out_offs, int64_t e, int64_t n) {
    const int64_t blk = (e - 1) / kRowScan;  // the scan CTA of row e - 1
    if (e % kRowScan == 0 || e == n || blk == 0) return 0;
    return static_cast<int64_t>(out_offs[blk * kRowScan]);
}

// ---- row searches over a tile of a packed output (K1v, K12, K13a, K14b) ----------------------------------------------

// The largest r in [lo, hi) with key(r) <= x, for a non-decreasing key with key(lo) <= x: a (kThreads + 1)-ary search,
// one probe per thread and one __syncthreads_count a round (two rounds up to 66 049 rows at 256 threads, three up to
// 17 million).  Every thread of the block must call it; all get the answer.
template <int kThreads, typename Key>
__device__ __forceinline__ int64_t block_search_le(int64_t lo, int64_t hi, int64_t x, const Key &key) {
    while (hi - lo > 1) {
        const int64_t w = hi - lo;
        const int64_t pr = lo + (static_cast<int64_t>(threadIdx.x) + 1) * w / (kThreads + 1);
        const int cnt = __syncthreads_count(key(pr) <= x);  // a prefix of the probes
        const int64_t nlo = cnt > 0 ? lo + static_cast<int64_t>(cnt) * w / (kThreads + 1) : lo;
        const int64_t nhi = cnt < kThreads ? lo + (static_cast<int64_t>(cnt) + 1) * w / (kThreads + 1) : hi;
        lo = nlo;
        hi = nhi;
    }
    return lo;
}

// A tile's row table: stage(j, r) for the rows r = r0 + j <= last, kThreads a round, until a row starts at or after p1.
// stage writes the caller's shared arrays for entry j and returns row r's start.  Returns the number of rows before
// that first one (which the table holds as well), or -1 when the kCap entries run out first: an over-full tile.  Every
// thread of the block must call it.
template <int kThreads, int kCap, typename Stage>
__device__ __forceinline__ int block_row_table(int64_t r0, int64_t last, int64_t p1, const Stage &stage) {
    for (int base = 0; base < kCap; base += kThreads) {
        const int j = base + static_cast<int>(threadIdx.x);
        bool past = true;
        if (r0 + j <= last) past = stage(j, r0 + j) >= p1;
        const int cnt = __syncthreads_count(past);  // a suffix of the round
        if (cnt > 0) return base + kThreads - cnt;
    }
    return -1;
}

// ---- the flat map over a packed output's 16-byte vectors (K12, K13a, K14b) -------------------------------------------
// The output is n rows laid end to end from byte 0: row r covers [start(r), start(r + 1)), start(n) = total, and out may
// have any alignment.  Its 16-byte aligned vectors are dealt in tiles of kFlatTile to a persistent grid of kFlatMinBlocks
// CTAs per SM in a static order (no tile counter: a launch is capturable and may run concurrently with itself).  Per tile
// the CTA
//   1. finds the row of the tile's first byte with block_search_le over start;
//   2. stages the tile's row starts, and the kernel's own row data, with block_row_table, up to the first row that starts
//      at or after the tile's end (row n starts at total, so that entry exists and closes the table).  A tile of more
//      than kFlatRowCap - 1 rows (rows shorter than 32 bytes on average, or many empty ones) is over-full and reads
//      everything from global memory instead;
//   3. per vector of output bytes [q, q + 16): a binary search of the table (or of global memory) for the row of its
//      first byte, then a walk over the rows it touches up to the first whose end is at or past min(q + 16, total) -- in
//      the table never past its closing entry.  Each non-empty row adds its bytes with the kernel's piece, merged by
//      byte mask; a vector inside the output leaves as one st.global.cs.v4, the at most two partial vectors at the ends
//      as byte stores.
// The kernel supplies a Map m with
//   int64_t start(int64_t r)          row r's start, from global memory (r <= n);
//   void stage(int j, int64_t r)      its own row data of row r into table entry j;
//   Row row_t(int j), row_g(int64_t r)   that data from entry j, or from global memory;
//   void piece(q, r, s, e, row, res)  merge16 of row r (output span [s, e), data row) into bytes [q, q + 16) of res.
constexpr int kFlatThreads = 256;
constexpr int kFlatVecs = 16;                         // output vectors per thread and tile
constexpr int kFlatTile = kFlatThreads * kFlatVecs;   // 4096 vectors: 64 KiB of output per tile
constexpr int kFlatRowCap = 2048;                     // row-table entries: tiles of up to kFlatRowCap - 1 rows use the table
constexpr int kFlatMinBlocks = 4;                     // CTAs per SM

// Output bytes [k0, k1) of t into res (k0, k1 relative to the vector's first byte, any values)
__device__ __forceinline__ void merge16(uint32_t res[4], const uint32_t t[4], int64_t k0, int64_t k1) {
    const int m0 = static_cast<int>(min(max(k0, int64_t(0)), int64_t(16)));
    const int m1 = static_cast<int>(min(max(k1, int64_t(0)), int64_t(16)));
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        const uint32_t mk = lt_mask(m1, w) & ~lt_mask(m0, w);
        res[w] = (res[w] & ~mk) | (t[w] & mk);
    }
}

// One vector: output bytes [q, q + 16) at dst (16-byte aligned), whose first byte in [0, total) lies in row r
template <typename Map, typename StartOf, typename RowOf>
__device__ __forceinline__ void flat_vector(int64_t q, int64_t r, int64_t total, const Map &m, const StartOf &start_of,
                                            const RowOf &row_of, uint8_t *dst) {
    uint32_t res[4] = {0u, 0u, 0u, 0u};
    const int64_t stop = min(q + 16, total);
    int64_t s = start_of(r);
    for (;;) {
        const int64_t e = start_of(r + 1);
        if (e > s) m.piece(q, r, s, e, row_of(r), res);
        if (e >= stop) break;
        ++r;
        s = e;
    }
    if (q >= 0 && q + 16 <= total) {
        __stcs(reinterpret_cast<uint4 *>(dst), make_uint4(res[0], res[1], res[2], res[3]));
    } else {
#pragma unroll
        for (int k = 0; k < 16; ++k)
            if (q + k >= 0 && q + k < total) dst[k] = static_cast<uint8_t>(res[k >> 2] >> (8 * (k & 3)));
    }
}

// The output's bytes; every thread of the block must call it (blockDim.x = kFlatThreads).
template <typename Map>
__device__ __forceinline__ void flat_map(uint8_t *out, int64_t n, int64_t total, const Map &m) {
    __shared__ int64_t tab[kFlatRowCap];  // starts of rows r0, r0 + 1, ...
    const int a = static_cast<int>(reinterpret_cast<uintptr_t>(out) & 15u);  // out - a is 16-byte aligned
    const int64_t nvec = total > 0 ? (total - 1 + a) / 16 + 1 : 0;         // vector v holds bytes [16v - a, 16v - a + 16)
    const int64_t ntiles = (nvec + kFlatTile - 1) / kFlatTile;
    auto start_g = [&](int64_t r) { return m.start(r); };
    auto row_g = [&](int64_t r) { return m.row_g(r); };
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t v0 = tile * kFlatTile;
        const int64_t p0 = max(16 * v0 - a, int64_t(0)), p1 = min(16 * (v0 + kFlatTile) - a, total);
        const int64_t r0 = block_search_le<kFlatThreads>(0, n, p0, start_g);
        const int nrows = block_row_table<kFlatThreads, kFlatRowCap>(r0, n, p1, [&](int j, int64_t r) {
            const int64_t s = m.start(r);
            tab[j] = s;
            m.stage(j, r);
            return s;
        });
        if (nrows > 0) {
            for (int k = 0; k < kFlatVecs; ++k) {
                const int64_t v = v0 + k * kFlatThreads + threadIdx.x;
                if (v >= nvec) break;
                const int64_t q = 16 * v - a, x = max(q, int64_t(0));
                int l = 0, h = nrows;  // the largest j < nrows with tab[j] <= x
                while (h - l > 1) {
                    const int mid = (l + h) >> 1;
                    if (tab[mid] <= x) l = mid;
                    else h = mid;
                }
                flat_vector(q, r0 + l, total, m, [&](int64_t r) { return tab[r - r0]; }, [&](int64_t r) { return m.row_t(r - r0); },
                            out + q);
            }
        } else {
            for (int k = 0; k < kFlatVecs; ++k) {
                const int64_t v = v0 + k * kFlatThreads + threadIdx.x;
                if (v >= nvec) break;
                const int64_t q = 16 * v - a, x = max(q, int64_t(0));
                int64_t l = r0, h = n;
                while (h - l > 1) {
                    const int64_t mid = (l + h) >> 1;
                    if (m.start(mid) <= x) l = mid;
                    else h = mid;
                }
                flat_vector(q, l, total, m, start_g, row_g, out + q);
            }
        }
        __syncthreads();  // the table is refilled by the next tile
    }
}

// K0: the device offsets reduction.  out = {sum0, sum1, max, what is wrong}: 1 a negative length, 2 offsets[0] < 0,
// 4 offsets[n] > nbytes (nbytes < 0: the size of the byte buffer is not known), 8 a sum or a row's value past INT64_MAX.
// The kernels index the byte buffer with these offsets, so a bad array must fail here and not read out of bounds.  Sums
// saturate per thread, warp and CTA; each CTA's atomicAdd then sees in the old value whether the total passed INT64_MAX
// (the counter only rises, so the CTA whose add crosses 2^63 sees it before any add could wrap 2^64).  One atomic per
// CTA and word, not per warp: with per-warp atomics a call on a million rows took 45 us instead of 34 us (B200, 1000 W).
constexpr int kExtentThreads = 256;

template <typename Measure>
__global__ void __launch_bounds__(kExtentThreads)
offsets_extent_kernel(const int64_t *__restrict__ offs, int64_t n, int64_t nbytes, Measure m, unsigned long long *out) {
    constexpr int kWarps = kExtentThreads / 32;
    __shared__ int64_t s_part[3][kWarps];
    __shared__ unsigned s_bad[kWarps];
    int64_t s0 = 0, s1 = 0, best = 0;
    unsigned bad = 0;
    bool over = false;
    for (int64_t i = blockIdx.x * static_cast<int64_t>(kExtentThreads) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * kExtentThreads) {
        const int64_t a = offs[i], b = offs[i + 1];
        if (b < a) bad |= 1u;
        if (i == 0 && a < 0) bad |= 2u;
        if (i == n - 1 && nbytes >= 0 && b > nbytes) bad |= 4u;
        // negative: b < a, or a < 0 with more than INT64_MAX after it (flagged at offsets[0] or an earlier decrease)
        const int64_t len = static_cast<int64_t>(static_cast<uint64_t>(b) - static_cast<uint64_t>(a));
        if (len < 0) continue;
        const Extent e = m.extent(len);
        over |= e.over;
        s0 = add_sat(s0, e.sum0, &over);
        s1 = add_sat(s1, e.sum1, &over);
        best = max(best, e.max);
    }
    for (int o = 16; o > 0; o >>= 1) {
        best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
        s0 = add_sat(s0, __shfl_xor_sync(0xffffffffu, s0, o), &over);
        s1 = add_sat(s1, __shfl_xor_sync(0xffffffffu, s1, o), &over);
    }
    bad = __reduce_or_sync(0xffffffffu, bad | (over ? 8u : 0u));
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        s_part[0][warp] = s0;
        s_part[1][warp] = s1;
        s_part[2][warp] = best;
        s_bad[warp] = bad;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    for (int w = 1; w < kWarps; ++w) {
        s0 = add_sat(s0, s_part[0][w], &over);
        s1 = add_sat(s1, s_part[1][w], &over);
        best = max(best, s_part[2][w]);
        bad |= s_bad[w];
    }
    const unsigned long long kMax = static_cast<unsigned long long>(kI64Max);
    if (s0 > 0) {
        const unsigned long long old = atomicAdd(out, static_cast<unsigned long long>(s0));
        over |= old > kMax || old + s0 > kMax;
    }
    if (s1 > 0) {
        const unsigned long long old = atomicAdd(out + 1, static_cast<unsigned long long>(s1));
        over |= old > kMax || old + s1 > kMax;
    }
    if (best > 0) atomicMax(out + 2, static_cast<unsigned long long>(best));
    if (over) bad |= 8u;
    if (bad) atomicOr(out + 3, static_cast<unsigned long long>(bad));
}

// BSQ_ERR_ARG for the first of offsets_extent_kernel's validation bits that is set (BSQ_OK when none is)
int offsets_error(unsigned long long bits);

// The offsets reduction of n rows of device offsets on st: one launch, one read-back, one synchronise.  Fails on bad
// offsets; a total past INT64_MAX is left to the caller (e->over), whose output it sizes.
template <typename Measure>
int reduce_offsets_device(int device, cudaStream_t st, const int64_t *d_offs, int64_t n, int64_t nbytes, const Measure &m, Extent *e) {
    BSQ_CUDA_TRY(cudaSetDevice(device));
    unsigned long long *d_res = nullptr, h_res[4] = {0, 0, 0, 0};
    if (int rc = scratch_alloc(device, reinterpret_cast<void **>(&d_res), sizeof(h_res), st)) return rc;
    BSQ_CUDA_TRY(cudaMemsetAsync(d_res, 0, sizeof(h_res), st));
    const int blocks = static_cast<int>(std::min<int64_t>((n + kExtentThreads - 1) / kExtentThreads, static_cast<int64_t>(cur_sms()) * 8));
    offsets_extent_kernel<<<blocks, kExtentThreads, 0, st>>>(d_offs, n, nbytes, m, d_res);
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    BSQ_CUDA_TRY(cudaMemcpyAsync(h_res, d_res, sizeof(h_res), cudaMemcpyDeviceToHost, st));
    BSQ_CUDA_TRY(cudaFreeAsync(d_res, st));
    BSQ_CUDA_TRY(cudaStreamSynchronize(st));
    if (int rc = offsets_error(h_res[3] & 7u)) return rc;
    *e = Extent{static_cast<int64_t>(h_res[0]), static_cast<int64_t>(h_res[1]), static_cast<int64_t>(h_res[2]), (h_res[3] & 8u) != 0};
    return BSQ_OK;
}

// The same of host offsets: offsets[0] < 0 first, then row by row up to the first negative length (an error) or the
// first row that takes a total past INT64_MAX (e->over).
template <typename Measure>
int reduce_offsets_host(const int64_t *h_offs, int64_t n, const Measure &m, Extent *e) {
    if (h_offs[0] < 0) return offsets_error(2u);
    *e = Extent{0, 0, 0, false};
    for (int64_t i = 0; i < n && !e->over; ++i) {
        const int64_t len = h_offs[i + 1] - h_offs[i];  // (both >= offsets[0] >= 0 so far: no overflow)
        if (len < 0) return offsets_error(1u);
        const Extent r = m.extent(len);
        e->over |= r.over;
        e->sum0 = add_sat(e->sum0, r.sum0, &e->over);
        e->sum1 = add_sat(e->sum1, r.sum1, &e->over);
        e->max = r.max > e->max ? r.max : e->max;
    }
    return BSQ_OK;
}

// word w (0..3) of a block, with selects (a run-time index into the block would put it in local memory)
__device__ __forceinline__ uint32_t pick4(const Philox &p, uint32_t w) {
    const uint32_t lo = (w & 1u) ? p.c[1] : p.c[0], hi = (w & 1u) ? p.c[3] : p.c[2];
    return (w & 2u) ? hi : lo;
}

__device__ __forceinline__ Philox mlm_block(uint64_t g, uint32_t blk, uint32_t stream, const MlmParam &m) {
    return philox4x32_10(static_cast<uint32_t>(g), static_cast<uint32_t>(g >> 32), blk, stream, m.k0, m.k1);
}

__device__ __forceinline__ uint32_t mlm_random_id(uint64_t g, uint32_t j, const MlmParam &m) {
    return __umulhi(pick4(mlm_block(g, j >> 2, 2u, m), j & 3u), m.nchars);
}

template <typename T>
__device__ __forceinline__ T code_value(uint32_t code, const Expand &ex) {
    // one-byte kinds: codes are the output bytes; wider kinds: ids through Expand
    if (sizeof(T) == 1) return static_cast<T>(static_cast<uint8_t>(code));
    return static_cast<T>(expand_code(code, ex));
}

// The decisions for 16 consecutive positions p of one row whose position 0 is residue j0 (position p is a residue
// iff 0 <= j0 + p < len): bit p of sel (selected), msk (-> mask_id) and rnd (-> random id), the random ids one per
// byte of rid.
struct Mlm16 {
    uint32_t sel, msk, rnd;
    uint32_t rid[4];
};

__device__ __forceinline__ Mlm16 mlm_decide16(int j0, int len, uint64_t g, const MlmParam &m) {
    Mlm16 d;
    d.sel = d.msk = d.rnd = 0u;
    d.rid[0] = d.rid[1] = d.rid[2] = d.rid[3] = 0u;
    const int lo = max(-j0, 0), hi = min(len - j0, 16);
    if (hi <= lo) return d;  // no residue (padding, or only BOS / EOS)
    // selection words of blocks j0 >> 2 .. +4 that hold a residue of the chunk (j0 = -1: block -1 holds none)
    const int b0 = j0 >> 2, jlo = j0 + lo, jhi = j0 + hi - 1;
    uint32_t W[20];
#pragma unroll
    for (int b = 0; b < 5; ++b) {
        const int blk = b0 + b;
        W[4 * b] = W[4 * b + 1] = W[4 * b + 2] = W[4 * b + 3] = 0u;
        if (4 * blk + 3 >= jlo && 4 * blk <= jhi) {
            const Philox p = mlm_block(g, static_cast<uint32_t>(blk), 1u, m);
            W[4 * b] = p.c[0]; W[4 * b + 1] = p.c[1]; W[4 * b + 2] = p.c[2]; W[4 * b + 3] = p.c[3];
        }
    }
    // u[p] = W[(j0 & 3) + p]: a two-step shift with selects
    const uint32_t a = static_cast<uint32_t>(j0) & 3u;
    uint32_t X[18];
#pragma unroll
    for (int q = 0; q < 18; ++q) X[q] = (a & 2u) ? W[q + 2] : W[q];
#pragma unroll
    for (int p = 0; p < 16; ++p) {
        const uint64_t u = (a & 1u) ? X[p + 1] : X[p];
        if (p >= lo && p < hi && u < m.ts) {
            d.sel |= 1u << p;
            if (u < m.tm) d.msk |= 1u << p;
            else if (u < m.tr) d.rnd |= 1u << p;
        }
    }
    // random ids: rare (random_prob of the selected share), one block each, only where needed
    uint32_t need = d.rnd;
    while (need) {
        const int p = __ffs(need) - 1;
        need &= need - 1u;
        const uint32_t v = mlm_random_id(g, static_cast<uint32_t>(j0 + p), m) << (8 * (p & 3));
        const int w = p >> 2;
        d.rid[0] |= w == 0 ? v : 0u;
        d.rid[1] |= w == 1 ? v : 0u;
        d.rid[2] |= w == 2 ? v : 0u;
        d.rid[3] |= w == 3 ? v : 0u;
    }
    return d;
}

// bits 0..3 of x -> 0x000000ff / 0x0000ff00 / 0x00ff0000 / 0xff000000
__device__ __forceinline__ uint32_t byte_mask4(uint32_t x) { return (((x & 0xfu) * 0x00204081u) & 0x01010101u) * 0xffu; }

// 16 codes t (bytes) + decisions -> inputs at `in` and labels at `lab`.  VEC: 16 elements, both pointers 16-byte
// aligned; otherwise the first cnt elements, one by one.
template <typename T, bool VEC>
__device__ __forceinline__ void mlm_emit16(T *in, int64_t *lab, const uint32_t t[4], const Mlm16 &d, int cnt, const MlmParam &m,
                                           const Expand &ex) {
    if (sizeof(T) == 1) {
        const uint32_t mrep = (static_cast<uint32_t>(m.mask_id) & 0xffu) * 0x01010101u;
        uint32_t o[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const uint32_t mm = byte_mask4(d.msk >> (4 * w)), rm = byte_mask4(d.rnd >> (4 * w));
            o[w] = (t[w] & ~(mm | rm)) | (mrep & mm) | (d.rid[w] & rm);
        }
        if (VEC) {
            __stcs(reinterpret_cast<uint4 *>(in), make_uint4(o[0], o[1], o[2], o[3]));
        } else {
#pragma unroll
            for (int p = 0; p < 16; ++p)
                if (p < cnt) reinterpret_cast<uint8_t *>(in)[p] = static_cast<uint8_t>(o[p >> 2] >> (8 * (p & 3)));
        }
    } else {
        constexpr int EPV = 16 / sizeof(T);
#pragma unroll
        for (int s = 0; s < 16 / EPV; ++s) {
            T vals[EPV];
#pragma unroll
            for (int j = 0; j < EPV; ++j) {
                const int p = s * EPV + j;
                const uint32_t code = (t[p >> 2] >> (8 * (p & 3))) & 0xffu;
                const uint32_t rid = (d.rid[p >> 2] >> (8 * (p & 3))) & 0xffu;
                vals[j] = (d.msk >> p) & 1u ? static_cast<T>(m.mask_id)
                                            : ((d.rnd >> p) & 1u ? static_cast<T>(static_cast<int32_t>(rid)) : code_value<T>(code, ex));
            }
            if (VEC) {
                __stcs(reinterpret_cast<uint4 *>(in) + s, *reinterpret_cast<const uint4 *>(vals));
            } else {
#pragma unroll
                for (int j = 0; j < EPV; ++j)
                    if (s * EPV + j < cnt) in[s * EPV + j] = vals[j];
            }
        }
    }
    // labels: the residue's code (< 0x80 in every mode) where selected
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        int64_t l[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int p = 2 * q + h;
            l[h] = (d.sel >> p) & 1u ? static_cast<int64_t>((t[p >> 2] >> (8 * (p & 3))) & 0xffu) : m.ignore;
        }
        if (VEC) {
            __stcs(reinterpret_cast<uint4 *>(lab) + q,
                   make_uint4(static_cast<uint32_t>(l[0]), static_cast<uint32_t>(static_cast<uint64_t>(l[0]) >> 32),
                              static_cast<uint32_t>(l[1]), static_cast<uint32_t>(static_cast<uint64_t>(l[1]) >> 32)));
        } else {
            if (2 * q < cnt) lab[2 * q] = l[0];
            if (2 * q + 1 < cnt) lab[2 * q + 1] = l[1];
        }
    }
}

#endif  // __CUDACC__

}  // namespace bsq
