// K14: translation of a packed DNA / RNA batch into protein reading frames under a genetic code (sm_100a).
//
// Semantics (include/bsq.h, bsq_translate): every byte is an IUPAC base set (a 4-bit mask, A = 1, C = 2, G = 4, T = 8,
// invalid = 0) and every codon the one letter all expansions of its three base sets agree on, else 'X'.  Both rules are
// tables built once on the host by bsq_translate_table -- the only statement of them in the library -- and handed to the
// kernel as parameters: masks[256] (and their complements, the 4-bit reversals) and codons[4096] indexed by
// m0 << 8 | m1 << 4 | m2.  Output sequence w = i * F + f is frame frames[f] of input sequence i; frame +k has
// max(0, (len - k + 1) / 3) amino acids read from offset k - 1, frame -k as many read from the reverse complement.
// tr_len below is the only statement of that length (host extent, device extent and both kernels use it).
//
// K14a: row_scan_kernel (+ row_carry_kernel past 1024 sequences, bsq_kernels.cuh) scans the per-sequence output bytes
//       (the sum of its F frame lengths, TranslateCount) into stream-ordered scratch S[n + 1].  seq_base adds the carry
//       an entry still lacks (row_scan_carry) where it is read, so no fix-up pass runs.
// K14b: translate_kernel -- a grid-stride pass over the n * F + 1 output offsets (each sequence's base plus the lengths of
//       its earlier frames), then the bytes: bsq_kernels.cuh's flat map with the sequences as rows, seq_base as their
//       starts and their source offsets as row data.  Its piece of a sequence: every frame the vector touches costs
//         - one 48-byte source span (16 codons) as four clamped aligned 16-byte loads realigned with selects and funnel
//           shifts; a reverse frame reads the mirrored span and reverses its bytes with PRMT, as K12 does;
//         - 48 mask look-ups (the complemented mask table for a reverse frame) and 16 codon look-ups in shared memory;
//         - a merge into the output vector by byte mask.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <string>

#include "bsq_internal.h"
#include "bsq_kernels.cuh"

namespace bsq {

namespace {

// A frame in 4 bits: k - 1 in bits 0-1, bit 3 set for the reverse strand.  F frames are packed 4 bits each, so the kernels
// index them with shifts instead of a run-time index into a parameter array.
__host__ __device__ __forceinline__ uint32_t frame_code(uint32_t fcode, int f) { return (fcode >> (4 * f)) & 15u; }

// amino acids of one frame of a sequence of len >= 0 nucleotides
__host__ __device__ __forceinline__ int64_t tr_len(int64_t len, uint32_t fr) {
    const int64_t skip = fr & 3u;
    return len > skip ? (len - skip) / 3 : 0;
}

struct FrameSet {
    uint32_t fcode;
    int F;
};

__host__ __device__ __forceinline__ int64_t tr_row_total(int64_t len, const FrameSet &fs) {
    int64_t t = 0;
    for (int f = 0; f < fs.F; ++f) t += tr_len(len, frame_code(fs.fcode, f));
    return t;
}

struct TranslateCount {
    FrameSet fs;
    __device__ __forceinline__ int64_t operator()(int64_t len) const { return tr_row_total(len, fs); }
};
// the extents' measure: the row's amino acids, the same after a crop to crop_len, and its longest cropped frame (a row
// has at most 2 len amino acids, so the 128-bit sums cannot wrap)
struct TranslateMeasure {
    FrameSet fs;
    int64_t crop_len;
    __host__ __device__ __forceinline__ Extent extent(int64_t len) const {
        __int128 t = 0, c = 0;
        int64_t best = 0;
        for (int f = 0; f < fs.F; ++f) {
            const int64_t L = tr_len(len, frame_code(fs.fcode, f)), k = L < crop_len ? L : crop_len;
            t += L;
            c += k;
            best = k > best ? k : best;
        }
        bool over = false;
        const int64_t st = clamp_sat(t, &over), sc = clamp_sat(c, &over);
        return {st, sc, best, over};
    }
};

// BSQ_ERR_ARG unless frames holds 1..6 distinct values of +-1, +-2, +-3; fills *fs
int check_frames(const int8_t *frames, int nframes, FrameSet *fs) {
    if (frames == nullptr || nframes < 1 || nframes > 6) return fail(BSQ_ERR_ARG, "frames: 1 to 6 distinct values of +-1, +-2, +-3 expected");
    fs->fcode = 0;
    fs->F = nframes;
    for (int f = 0; f < nframes; ++f) {
        const int v = frames[f];
        if (v == 0 || v < -3 || v > 3) return fail(BSQ_ERR_ARG, "frames must be +-1, +-2 or +-3, got " + std::to_string(v));
        for (int g = 0; g < f; ++g)
            if (frames[g] == v) return fail(BSQ_ERR_ARG, "frame " + std::to_string(v) + " is given twice");
        const uint32_t c = static_cast<uint32_t>((v > 0 ? v : -v) - 1) | (v < 0 ? 8u : 0u);
        fs->fcode |= c << (4 * f);
    }
    return BSQ_OK;
}

int check_code(const char *code64) {
    if (code64 == nullptr) return fail(BSQ_ERR_ARG, "null genetic code");
    for (int c = 0; c < 64; ++c) {
        const unsigned char b = static_cast<unsigned char>(code64[c]);
        if (b < 0x21 || b > 0x7E)
            return fail(BSQ_ERR_ARG, "genetic code: 64 printable ASCII characters (0x21..0x7E) expected; byte " + std::to_string(c) +
                                         " is " + std::to_string(static_cast<int>(b)));
    }
    return BSQ_OK;
}

// The rule of include/bsq.h, built once: base sets of every byte and the letter of every triple of base sets.
struct Tables {
    uint8_t mask[256];
    uint8_t codon[4096];
};
void build_tables(const char *code64, Tables *t) {
    // each code, then the bases it stands for (upper and lower case alike)
    static const char *const kSets[] = {"AA", "CC", "GG", "TT", "UT", "RAG", "YCT", "SCG", "WAT", "KGT", "MAC", "BCGT", "DAGT", "HACT",
                                        "VACG", "NACGT"};
    std::memset(t->mask, 0, sizeof(t->mask));
    auto bit = [](char b) -> uint8_t { return b == 'A' ? 1 : b == 'C' ? 2 : b == 'G' ? 4 : 8; };
    for (const char *s : kSets) {
        uint8_t m = 0;
        for (const char *p = s + 1; *p; ++p) m |= bit(*p);
        t->mask[static_cast<uint8_t>(s[0])] = m;
        t->mask[static_cast<uint8_t>(s[0] | 0x20)] = m;
    }
    static const int kTcag[4] = {2, 1, 3, 0};  // mask bit (A, C, G, T) -> index in TCAG order
    for (int m0 = 0; m0 < 16; ++m0)
        for (int m1 = 0; m1 < 16; ++m1)
            for (int m2 = 0; m2 < 16; ++m2) {
                char letter = 0;
                bool agree = m0 && m1 && m2;
                for (int b0 = 0; agree && b0 < 4; ++b0)
                    for (int b1 = 0; agree && b1 < 4; ++b1)
                        for (int b2 = 0; agree && b2 < 4; ++b2) {
                            if (!((m0 >> b0) & 1) || !((m1 >> b1) & 1) || !((m2 >> b2) & 1)) continue;
                            const char c = code64[16 * kTcag[b0] + 4 * kTcag[b1] + kTcag[b2]];
                            if (letter == 0) letter = c;
                            else if (letter != c) agree = false;
                        }
                t->codon[m0 << 8 | m1 << 4 | m2] = static_cast<uint8_t>(agree ? letter : 'X');
            }
}

__host__ __device__ __forceinline__ uint8_t bitrev4(uint8_t m) {
    return static_cast<uint8_t>(((m & 1) << 3) | ((m & 2) << 1) | ((m & 4) >> 1) | ((m & 8) >> 3));
}

struct TrTables {
    uint32_t mask[64], cmask[64];  // 256 masks and their complements, 4 per word
    uint32_t codon[1024];          // 4096 letters, 4 per word
};

struct TrArgs {
    const uint8_t *bytes;
    const int64_t *offs;
    const int64_t *S;  // K14a's scan (see seq_base)
    int64_t n, total;
    FrameSet fs;
};

// S[e] with its scan CTA's carry: the global exclusive prefix of the per-sequence output bytes (seq_base(n) = total)
__device__ __forceinline__ int64_t seq_base(const TrArgs &a, int64_t e) { return __ldg(a.S + e) + row_scan_carry(a.S, e, a.n); }

// The 16 letters of one (sequence, frame) piece for output bytes [q, q + 16): amino acid t0 + j of the frame lands in
// byte j.  s / len: the sequence's source start and length; fr: the frame's code.
__device__ __forceinline__ void tr_piece(int64_t q, int64_t ws, int64_t s, int64_t len, uint32_t fr, const TrArgs &a,
                                         const uint8_t *mask, const uint8_t *cmask, const uint8_t *codon, uint32_t t[4]) {
    const uintptr_t src0 = reinterpret_cast<uintptr_t>(a.bytes);
    const int64_t t0 = q - ws, skip = fr & 3u;
    const bool rev = (fr & 8u) != 0;
    // forward: codon j is nucleotides skip + 3 (t0 + j) .. + 2; reverse: len - skip - 3 (t0 + j) - 3 .. - 1, read right to
    // left -- byte 47 - 3j .. 45 - 3j of the 48 that end at len - skip - 3 t0
    const int64_t X = rev ? s + len - skip - 3 * t0 - 48 : s + skip + 3 * t0;
    const uintptr_t lo = (src0 + static_cast<uintptr_t>(s)) & ~uintptr_t(15);
    const uintptr_t hi = (src0 + static_cast<uintptr_t>(s + len - 1)) & ~uintptr_t(15);
    uint32_t w[12];
    fetch_clamped<12>(src0 + static_cast<uintptr_t>(X), lo, hi, w);
    if (rev) {
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            const uint32_t x = w[k];
            w[k] = __byte_perm(w[11 - k], 0u, 0x0123);
            w[11 - k] = __byte_perm(x, 0u, 0x0123);
        }
    }
    const uint8_t *m = rev ? cmask : mask;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        uint32_t word = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int p = 3 * (4 * k + j);
            const uint32_t m0 = m[__byte_perm(w[p >> 2], 0u, 0x4440 + (p & 3))];
            const uint32_t m1 = m[__byte_perm(w[(p + 1) >> 2], 0u, 0x4440 + ((p + 1) & 3))];
            const uint32_t m2 = m[__byte_perm(w[(p + 2) >> 2], 0u, 0x4440 + ((p + 2) & 3))];
            word += static_cast<uint32_t>(codon[m0 << 8 | m1 << 4 | m2]) << (8 * j);
        }
        t[k] = word;
    }
}

struct SrcRow {
    int64_t start, end;  // a sequence's source offsets
};

// K14b's rows for flat_map: the sequences, starting at seq_base, with their source offsets as row data
struct TrMap {
    TrArgs a;
    const uint8_t *mask, *cmask, *codon;  // tables in shared memory
    int64_t *src;                         // source starts of the tile's rows, in shared memory

    __device__ __forceinline__ int64_t start(int64_t i) const { return seq_base(a, i); }
    __device__ __forceinline__ void stage(int j, int64_t i) const { src[j] = __ldg(a.offs + i); }
    __device__ __forceinline__ SrcRow row_t(int j) const { return {src[j], src[j + 1]}; }
    __device__ __forceinline__ SrcRow row_g(int64_t i) const { return {__ldg(a.offs + i), __ldg(a.offs + i + 1)}; }
    // the frames of a sequence (output bytes from b) that output bytes [q, q + 16) touch
    __device__ __forceinline__ void piece(int64_t q, int64_t, int64_t b, int64_t, SrcRow r, uint32_t res[4]) const {
        const int64_t len = r.end - r.start;
        int64_t ws = b;
        for (int f = 0; f < a.fs.F && ws < q + 16; ++f) {
            const uint32_t fr = frame_code(a.fs.fcode, f);
            const int64_t L = tr_len(len, fr);
            if (L > 0 && ws + L > q) {
                uint32_t t[4];
                tr_piece(q, ws, r.start, len, fr, a, mask, cmask, codon, t);
                merge16(res, t, ws - q, ws + L - q);
            }
            ws += L;
        }
    }
};

__global__ void __launch_bounds__(kFlatThreads, kFlatMinBlocks)
translate_kernel(TrArgs a, const __grid_constant__ TrTables tbl, uint8_t *__restrict__ out, int64_t *__restrict__ out_offs) {
    __shared__ __align__(16) uint8_t s_mask[256];
    __shared__ __align__(16) uint8_t s_cmask[256];
    __shared__ __align__(16) uint8_t s_codon[4096];
    __shared__ int64_t s_src[kFlatRowCap];
    const int tid = threadIdx.x;
    if (tid < 64) {
        reinterpret_cast<uint32_t *>(s_mask)[tid] = tbl.mask[tid];
        reinterpret_cast<uint32_t *>(s_cmask)[tid] = tbl.cmask[tid];
    }
    for (int k = tid; k < 1024; k += kFlatThreads) reinterpret_cast<uint32_t *>(s_codon)[k] = tbl.codon[k];
    a.total = seq_base(a, a.n);
    // output offsets: sequence i's base, then each frame's length
    const int64_t nw = a.n * a.fs.F;
    for (int64_t w = blockIdx.x * static_cast<int64_t>(kFlatThreads) + tid; w <= nw; w += static_cast<int64_t>(gridDim.x) * kFlatThreads) {
        if (w == nw) {
            out_offs[nw] = a.total;
            break;
        }
        const int64_t i = w / a.fs.F;
        const int f = static_cast<int>(w - i * a.fs.F);
        const int64_t len = __ldg(a.offs + i + 1) - __ldg(a.offs + i);
        int64_t o = seq_base(a, i);
        for (int g = 0; g < f; ++g) o += tr_len(len, frame_code(a.fs.fcode, g));
        out_offs[w] = o;
    }
    __syncthreads();  // the tables are in shared memory
    flat_map(out, a.n, a.total, TrMap{a, s_mask, s_cmask, s_codon, s_src});
}

}  // namespace

}  // namespace bsq

using namespace bsq;

extern "C" int bsq_genetic_code(int id, char out[64]) {
    if (out == nullptr) return fail(BSQ_ERR_ARG, "null output");
    const char *s = nullptr;
    switch (id) {
        case 1:
        case 11: s = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"; break;
        case 2: s = "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIMMTTTTNNKKSS**VVVVAAAADDEEGGGG"; break;
        case 4: s = "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"; break;
        case 5: s = "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIMMTTTTNNKKSSSSVVVVAAAADDEEGGGG"; break;
        case 6: s = "FFLLSSSSYYQQCC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"; break;
        default: return fail(BSQ_ERR_ARG, "no built-in genetic code " + std::to_string(id) + " (built in: 1, 2, 4, 5, 6, 11)");
    }
    std::memcpy(out, s, 64);
    return BSQ_OK;
}

extern "C" int bsq_translate_table(const char *code64, uint8_t masks[256], uint8_t codons[4096]) {
    if (int rc = check_code(code64)) return rc;
    if (masks == nullptr || codons == nullptr) return fail(BSQ_ERR_ARG, "null output table");
    Tables t;
    build_tables(code64, &t);
    std::memcpy(masks, t.mask, 256);
    std::memcpy(codons, t.codon, 4096);
    return BSQ_OK;
}

extern "C" int bsq_translate_extent_host(const int64_t *h_offsets, int64_t nseq, const int8_t *frames, int nframes, int64_t crop_len,
                                         int64_t *total, int64_t *crop_total, int64_t *max_len) {
    FrameSet fs;
    if (int rc = check_frames(frames, nframes, &fs)) return rc;
    if (crop_len < 1) return fail(BSQ_ERR_ARG, "crop_len must be >= 1");
    if (total == nullptr || crop_total == nullptr || max_len == nullptr) return fail(BSQ_ERR_ARG, "null output");
    if (nseq < 0 || (nseq > 0 && h_offsets == nullptr)) return fail(BSQ_ERR_ARG, "bad offsets");
    *total = *crop_total = *max_len = 0;
    if (nseq == 0) return BSQ_OK;
    Extent e{};
    if (int rc = reduce_offsets_host(h_offsets, nseq, TranslateMeasure{fs, crop_len}, &e)) return rc;
    if (e.over) return fail(BSQ_ERR_ARG, "the translated batch exceeds INT64_MAX bytes");
    *total = e.sum0;
    *crop_total = e.sum1;
    *max_len = e.max;
    return BSQ_OK;
}

extern "C" int bsq_translate_extent_device(int device, void *stream, const int64_t *d_offsets, int64_t nseq, int64_t nbytes,
                                           const int8_t *frames, int nframes, int64_t crop_len, int64_t *total, int64_t *crop_total,
                                           int64_t *max_len) {
    bsq::DeviceRestore restore_device;
    FrameSet fs;
    if (int rc = check_frames(frames, nframes, &fs)) return rc;
    if (crop_len < 1) return fail(BSQ_ERR_ARG, "crop_len must be >= 1");
    if (total == nullptr || crop_total == nullptr || max_len == nullptr) return fail(BSQ_ERR_ARG, "null output");
    if (nseq < 0 || (nseq > 0 && d_offsets == nullptr)) return fail(BSQ_ERR_ARG, "bad offsets");
    *total = *crop_total = *max_len = 0;
    if (nseq == 0) return BSQ_OK;
    Extent e{};
    if (int rc = reduce_offsets_device(device, static_cast<cudaStream_t>(stream), d_offsets, nseq, nbytes, TranslateMeasure{fs, crop_len}, &e))
        return rc;
    if (e.over) return fail(BSQ_ERR_ARG, "the translated batch exceeds INT64_MAX bytes");
    *total = e.sum0;
    *crop_total = e.sum1;
    *max_len = e.max;
    return BSQ_OK;
}

extern "C" int bsq_translate(int device, void *stream, const uint8_t *d_bytes, const int64_t *d_offsets, int64_t nseq,
                             const int8_t *frames, int nframes, const char *code64, uint8_t *d_out_bytes, int64_t *d_out_offsets) {
    bsq::DeviceRestore restore_device;
    FrameSet fs;
    if (int rc = check_frames(frames, nframes, &fs)) return rc;
    if (int rc = check_code(code64)) return rc;
    if (nseq < 0 || nseq > kI64Max / 6 - 1) return fail(BSQ_ERR_ARG, "bad batch size");
    if (d_out_offsets == nullptr) return fail(BSQ_ERR_ARG, "null output offsets");
    if (nseq > 0 && (d_bytes == nullptr || d_offsets == nullptr || d_out_bytes == nullptr))
        return fail(BSQ_ERR_ARG, "null bytes, offsets or output bytes");
    BSQ_CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nseq == 0) {
        BSQ_CUDA_TRY(cudaMemsetAsync(d_out_offsets, 0, sizeof(int64_t), st));
        return BSQ_OK;
    }
    Tables t;
    build_tables(code64, &t);
    TrTables tt;
    for (int w = 0; w < 64; ++w) {
        const uint8_t *m = t.mask + 4 * w;
        tt.mask[w] = m[0] | (m[1] << 8) | (m[2] << 16) | (static_cast<uint32_t>(m[3]) << 24);
        tt.cmask[w] = bitrev4(m[0]) | (bitrev4(m[1]) << 8) | (bitrev4(m[2]) << 16) | (static_cast<uint32_t>(bitrev4(m[3])) << 24);
    }
    std::memcpy(tt.codon, t.codon, sizeof(tt.codon));
    int64_t *S = nullptr;
    BSQ_CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&S), static_cast<size_t>(nseq + 1) * sizeof(int64_t), st));
    if (int rc = launch_row_scan(st, d_offsets, nseq, TranslateCount{fs}, S)) return rc;
    TrArgs a;
    a.bytes = d_bytes;
    a.offs = d_offsets;
    a.S = S;
    a.n = nseq;
    a.total = 0;  // (S's last entry: read by the kernel)
    a.fs = fs;
    translate_kernel<<<cur_sms() * kFlatMinBlocks, kFlatThreads, 0, st>>>(a, tt, d_out_bytes, d_out_offsets);
    count_launch();
    BSQ_CUDA_TRY(cudaGetLastError());
    BSQ_CUDA_TRY(cudaFreeAsync(S, st));
    return BSQ_OK;
}
