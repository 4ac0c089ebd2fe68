// K1s: batch-first one-byte tokens, tile-staged and warp-specialised (sm_100a).
//
// Reference semantics: Tokenizer::transencode<T>, batch_first branch (src/tokenize.h:430-434, :451-479).
//
// The (nseq, padlen) output is one flat byte array; a *tile* is a run of `vt` 16-byte output vectors of
// it (whole rows when padlen divides the tile, otherwise it starts and ends inside rows).  The residues
// that a tile needs are ONE contiguous span of the packed input (rows are consecutive sequences), so a
// tile costs one 1-D bulk asynchronous copy (cp.async.bulk global -> shared, SASS UBLKCP, the TMA unit)
// instead of one copy, one barrier wait and one slot computation per row:
//
//   producer warp   per tile: divides the tile's flat range into rows, loads the rows' offsets
//                   (coalesced), issues the span copy into the next free stage of a ring of kSpanStages
//                   shared-memory buffers (completion counted on the stage's `full` mbarrier) and
//                   writes the per-row table {source position in the stage, length} next to it;
//   8 consumer warps per tile: one 16-byte output vector per lane and step, vectors dealt flat
//                   (consecutive lanes = consecutive vectors, a warp stores 512 contiguous bytes).
//                   A lane finds its row with one multiply-shift division and one LDS.64 of the row
//                   table, then: two LDS.128 of the staged residues, word select + four funnel
//                   shifts (source-to-output byte shift), 16 LUT look-ups, BOS / EOS / PAD from the
//                   17-entry mask tables on boundary vectors only, one st.global.cs.v4.  Vectors
//                   beyond a row's EOS are the constant pad vector and skip all loads.
//
// Rows whose padlen is not a multiple of 16 use the same code: vectors stay aligned in the flat
// output, a vector that straddles two rows is assembled from both and stored whole, and only the
// batch's final partial vector (nseq * padlen % 16 != 0) is stored bytewise.
//
// Nothing per row is left in the instruction stream of the consumers except the row-table load: the
// warp-per-row ring kernel it replaced (K1r, since removed) spent 236 warp-instructions per 1 KiB row, 128 of
// them on per-row bookkeeping (slot arithmetic, elect loops around each row's bulk copy, barrier waits,
// uniform-datapath shuffling); see profiles/ r01x vs r02.
#include <cuda_runtime.h>

#include <algorithm>
#include <mutex>
#include <unordered_map>

#include "bsq_internal.h"
#include "bsq_kernels.cuh"

namespace bsq {

namespace {

constexpr unsigned kWaitBackoffNs = 64;

constexpr int kSpanConsumerWarps = 8;
constexpr int kSpanConsumers = kSpanConsumerWarps * 32;
constexpr int kSpanThreads = kSpanConsumers + 32;
constexpr int kSpanSlack = 32;  // bytes in front of the staged span (two LDS.128 never leave the stage)
constexpr int kSpanTail = 64;   // and behind it
// Stages of the ring: 3 and 4 were measured no faster than 2 (profiles/r02_sweep_span.txt).
constexpr int kSpanStages = 2;
// Tile size in 16-byte output vectors (24 KB), and resident CTAs per SM; both from the r02 sweep (DESIGN §3).
constexpr int kSpanTileVecs = 1536;
constexpr int kSpanCtasPerSm = 4;

__device__ __forceinline__ uint32_t s_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void bar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s_u32(bar)), "r"(count));
}
__device__ __forceinline__ void bar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void bar_wait(uint32_t bar, uint32_t parity) {
    // A warp that polls in a tight loop takes issue slots from the warps that have work (ncu r02n: 40 % of the
    // executed instructions were polls); after a failed first try it backs off with nanosleep between tries.
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra BSQ_SPAN_WAIT_DONE_%=;\n"
        "BSQ_SPAN_WAIT_%=:\n"
        "nanosleep.u32 %2;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@!p bra BSQ_SPAN_WAIT_%=;\n"
        "BSQ_SPAN_WAIT_DONE_%=:\n"
        "}\n" ::"r"(bar),
        "r"(parity), "r"(kWaitBackoffNs)
        : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}

// One launch can serve several batches that share padlen and tokenizer (bsq_tokenize_many: the small per-step batches of
// the reference's training loops, training/cnnpretrain.py:123-125,145): their tiles are numbered one batch after the other.
struct SpanBatch {
    const uint8_t *bytes;
    const int64_t *offs;
    uint8_t *out;
    int64_t nseq;
    int64_t total;       // nseq * padlen output bytes
    int64_t first_tile;  // index of the batch's first tile
};
struct SpanBatches {
    SpanBatch b[kSpanManyMax];
};

struct SpanParams {
    int64_t ntiles;
    int nbatch;
    // A CTA's first two tiles are static, blockIdx.x and blockIdx.x + gridDim.x (no atomic result is waited on before
    // both copies are in flight); the rest are handed out by an atomic counter, 2 * gridDim.x + atomicAdd(ctr, 1):
    // whatever the placement and start time of the CTAs (a programmatically launched grid gets its SM slots as the
    // previous grid drains), the work stays balanced.  ctr[0] = tiles handed out, ctr[1] = CTAs that have seen the end;
    // the last of those resets both for the slot's next launch.  nullptr: static round-robin (tile += gridDim.x).
    unsigned int *ctr;
    int padlen;
    int vt;           // 16-byte vectors per tile (a multiple of kSpanConsumers)
    int stage_bytes;  // data area of a stage
    int max_rows;     // row-table entries of a stage
    uint32_t div_mul, div_shift;  // n / padlen = umulhi(n, div_mul) >> div_shift for 0 <= n < 2^31 (span_magic)
    int straddle;     // != 0: a warp's 32 vectors can lie in two rows (padlen % 512 != 0)
#ifdef BSQ_SPAN_TRACE
    unsigned long long *trace;  // kSpanTraceWords per CTA (bsq_span_trace_arm), nullptr: not recorded
#endif
};

#ifdef BSQ_SPAN_TRACE
// Timeline probe (tools/span_timeline.py builds the library with -DBSQ_SPAN_TRACE; the shipped build has none of it).
// Per CTA: words 0-5 %globaltimer at the events below, word 6 %smid, word 7 tiles the CTA took, words 8-13 clock64 at
// the same events (SM-local: intervals inside one CTA only).  The exit words are maxima over the consumer warps.
constexpr int kSpanTraceWords = 16;
enum SpanTraceEvent { kTrEntry = 0, kTrWait = 1, kTrCopy0 = 2, kTrFull0 = 3, kTrStore0 = 4, kTrExit = 5 };
__device__ __forceinline__ unsigned long long span_globaltimer() {
    unsigned long long g;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
    return g;
}
__device__ __forceinline__ unsigned span_smid() {
    unsigned v;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(v));
    return v;
}
__device__ __forceinline__ void span_trace(const SpanParams &q, int ev) {
    if (q.trace == nullptr) return;
    unsigned long long *r = q.trace + kSpanTraceWords * blockIdx.x;
    const unsigned long long g = span_globaltimer(), c = clock64();
    if (ev == kTrExit) {
        atomicMax(r + ev, g);
        atomicMax(r + 8 + ev, c);
    } else {
        r[ev] = g;
        r[8 + ev] = c;
    }
}
__device__ __forceinline__ void span_trace_word(const SpanParams &q, int w, unsigned long long v) {
    if (q.trace != nullptr) q.trace[kSpanTraceWords * blockIdx.x + w] = v;
}
#define BSQ_SPAN_MARK(cond, ev) \
    do {                        \
        if (cond) span_trace(q, ev); \
    } while (0)
#else
#define BSQ_SPAN_MARK(cond, ev) \
    do {                        \
    } while (0)
#endif

// Shared-memory loads by 32-bit shared address (the addresses are formed once per tile, outside the vector loop).
__device__ __forceinline__ uint4 lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ int4 lds128i(uint32_t a) {
    int4 v;
    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t ldsu8(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}

// Four LUT look-ups.  `lutb` is the LUT's shared address, 256-byte aligned: one PRMT per byte builds the
// whole address (byte k of x under the upper three bytes of lutb), then LDS.U8; the codes are re-packed
// with integer multiply-adds (FMA pipe; the PRMTs sit on the ALU pipe).
__device__ __forceinline__ uint32_t span_translate4(uint32_t x, uint32_t lutb) {
    const uint32_t b0 = ldsu8(__byte_perm(x, lutb, 0x7650));
    const uint32_t b1 = ldsu8(__byte_perm(x, lutb, 0x7651));
    const uint32_t b2 = ldsu8(__byte_perm(x, lutb, 0x7652));
    const uint32_t b3 = ldsu8(__byte_perm(x, lutb, 0x7653));
    return b0 + b1 * 0x100u + b2 * 0x10000u + b3 * 0x1000000u;
}

// 16 codes from the 32-byte window {v0, v1}: word shift Q (compile time), bit shift sh (taken mod 32).
template <int Q>
__device__ __forceinline__ void span_translate16(const uint4 &v0, const uint4 &v1, uint32_t sh, uint32_t lutb, uint32_t t[4]) {
    const uint32_t w[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t x = __funnelshift_r(w[Q + k], w[Q + k + 1], sh);
        t[k] = span_translate4(x, lutb);
    }
}
__device__ __forceinline__ void span_window16(uint32_t S, uint32_t lutb, int straddle, uint32_t t[4]) {
    const uint4 v0 = lds128(S & ~15u), v1 = lds128((S & ~15u) + 16u);
    const uint32_t sh = S << 3;
    // One whole specialised body per word shift, entered by a branch that is warp-uniform whenever the warp's 32
    // vectors lie in one row.  A warp that holds two rows with different shifts (padlen % 512 != 0: most warps at
    // padlen 656) would run two of the 50-instruction bodies one after the other: such a warp takes a fifth body,
    // which picks its words with 11 selects instead (padlen 656: 0.755 -> 0.807 of the HBM peak, 652: 0.665 -> 0.691).
    // Rows of whole 512-byte windows never straddle and skip the vote (it costs 0.4 us of C2's 20.4).
    const uint32_t q = S & 12u;
    int uni = 1;
    if (straddle) __match_all_sync(__activemask(), q, &uni);
    if (uni) {
        switch (q) {
            case 0: span_translate16<0>(v0, v1, sh, lutb, t); break;
            case 4: span_translate16<1>(v0, v1, sh, lutb, t); break;
            case 8: span_translate16<2>(v0, v1, sh, lutb, t); break;
            default: span_translate16<3>(v0, v1, sh, lutb, t); break;
        }
    } else {
        const bool q2 = (S & 8u) != 0, q1 = (S & 4u) != 0;
        const uint32_t a0 = q2 ? v0.z : v0.x, a1 = q2 ? v0.w : v0.y, a2 = q2 ? v1.x : v0.z, a3 = q2 ? v1.y : v0.w;
        const uint32_t a4 = q2 ? v1.z : v1.x, a5 = q2 ? v1.w : v1.y;
        const uint32_t x[5] = {q1 ? a1 : a0, q1 ? a2 : a1, q1 ? a3 : a2, q1 ? a4 : a3, q1 ? a5 : a4};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t y = __funnelshift_r(x[k], x[k + 1], sh);
            t[k] = span_translate4(y, lutb);
        }
    }
}

// Loop invariants of the consumers, kept in registers.  They are read back from shared memory (cst[]) rather than
// taken from the kernel parameters: ptxas re-materialises parameter values with constant-bank loads (and shared
// addresses with window arithmetic) inside the vector loop -- 6 to 10 extra instructions per vector -- which it
// cannot do with the result of a shared-memory load.
struct SpanRegs {
    uint32_t lutb;   // shared address of the LUT (256-byte aligned)
    uint32_t tab_m;  // shared address of TailTab::m[0]; TailTab::f[k] is 17 * 16 bytes further on
    uint32_t tab_h;  // shared address of the head table: entry j = j pad codes, then BOS (if any), then zeros
    uint32_t bos_w, bos_sel;  // BOS byte and the PRMT selector that puts it into byte 0 (identity without BOS)
    uint4 padq;               // the constant pad vector
    int bos, eos, padlen, neg_padlen;
    uint32_t mul, shift;  // multiply-shift division by padlen
    int straddle;         // a warp's 32 vectors can lie in two rows
};
constexpr int kCstWords = 16;

// Codes of columns c0 .. c0+15 of one row (src/tokenize.h:460-478), for c0 < n + eos: `srow` is the shared
// address of the byte that column 0 would come from (first residue - bos), n = bos + len.  Columns >= padlen are
// don't-care.  The residue window is loaded and translated unconditionally: whatever lies left of the first
// residue or right of the last is replaced by the BOS / tail fix-ups (for c0 == n the whole vector is).
__device__ __forceinline__ uint4 span_row_codes(uint32_t srow, int n, int c0, const SpanRegs &g) {
    uint32_t t[4];
    span_window16(srow + static_cast<uint32_t>(c0), g.lutb, g.straddle, t);
    if (c0 == 0) t[0] = __byte_perm(t[0], g.bos_w, g.bos_sel);
    if (c0 + 16 > n) {  // the row's residues end inside this vector: keep n - c0 bytes, then EOS / pad
        const uint32_t a = g.tab_m + 16u * static_cast<uint32_t>(n - c0);
        const uint4 m = lds128(a), f = lds128(a + 17u * 16u);
        t[0] = (t[0] & m.x) | f.x; t[1] = (t[1] & m.y) | f.y;
        t[2] = (t[2] & m.z) | f.z; t[3] = (t[3] & m.w) | f.w;
    }
    return make_uint4(t[0], t[1], t[2], t[3]);
}

// Unaligned rows: columns c0 .. c0+15 with -16 < c0 <= padlen - 16; for c0 < 0 the bytes left of column 0 are the
// previous row's tail and are set to the pad code (the caller has checked that the previous row ends before them).
__device__ __forceinline__ uint4 span_row_codes_u(uint32_t srow, int n, int c0, const SpanRegs &g) {
    uint32_t t[4];
    span_window16(srow + static_cast<uint32_t>(c0), g.lutb, g.straddle, t);
    if (c0 <= 0) {  // bytes [0, -c0): pad; byte -c0: BOS when the tokenizer has one -- a ready-made vector per -c0
        const uint32_t j16 = 16u * static_cast<uint32_t>(-c0);
        const uint4 mb = lds128(g.tab_m + j16 + 16u * static_cast<uint32_t>(g.bos)), hh = lds128(g.tab_h + j16);
        t[0] = (t[0] & ~mb.x) | hh.x;
        t[1] = (t[1] & ~mb.y) | hh.y;
        t[2] = (t[2] & ~mb.z) | hh.z;
        t[3] = (t[3] & ~mb.w) | hh.w;
    }
    if (c0 + 16 > n) {  // the row's residues end inside this vector: keep n - c0 bytes, then EOS / pad
        const uint32_t a = g.tab_m + 16u * static_cast<uint32_t>(n - c0);
        const uint4 m = lds128(a), f = lds128(a + 17u * 16u);
        t[0] = (t[0] & m.x) | f.x; t[1] = (t[1] & m.y) | f.y;
        t[2] = (t[2] & m.z) | f.z; t[3] = (t[3] & m.w) | f.w;
    }
    return make_uint4(t[0], t[1], t[2], t[3]);
}

// The rare straddling vector whose first bytes are NOT pad: the previous row (rl - 1) is so long that its residues /
// EOS reach into them.  Both rows' codes are built and merged.  Kept out of line: it must not cost the hot loop registers.
__device__ __noinline__ uint4 span_straddle_general(uint32_t rows_a, uint32_t rl, int col, const SpanRegs &g) {
    const int4 rp = lds128i(rows_a + 16u * rl - 16u), ri = lds128i(rows_a + 16u * rl);
    const int cp = col + g.padlen;  // the vector's first column in the previous row (> padlen - 16)
    uint4 prev = g.padq;
    if (cp < rp.z) prev = span_row_codes_u(static_cast<uint32_t>(rp.x), rp.y, cp, g);
    const uint4 cur = span_row_codes_u(static_cast<uint32_t>(ri.x), ri.y, col, g);
    const uint4 m = lds128(g.tab_m - 16u * static_cast<uint32_t>(col));  // bytes [0, -col) come from the previous row
    return make_uint4((prev.x & m.x) | (cur.x & ~m.x), (prev.y & m.y) | (cur.y & ~m.y), (prev.z & m.z) | (cur.z & ~m.z),
                      (prev.w & m.w) | (cur.w & ~m.w));
}

// The four offsets that delimit a tile's span: rows r0 and r1 (first and last row the tile touches).
struct SpanEdges {
    int64_t a0, a1, b0, b1;
};

// 4 CTAs per SM leave 56 registers per thread; 5 and 6 (40 and 32 registers) were measured slower (r02 sweep, DESIGN §3).
template <bool ALIGNED>
__global__ void __launch_bounds__(kSpanThreads, kSpanCtasPerSm)
tokenize_span_kernel(const SpanParams q, const __grid_constant__ SpanBatches mb, const LutParam lutp, const Specials sp) {
    extern __shared__ __align__(128) uint8_t dyn[];  // kSpanStages x { data[stage_bytes], rows[max_rows] x 16 B }
    __shared__ __align__(256) uint8_t lut[256];
    __shared__ TailTab tab;
    __shared__ uint4 headtab[16];
    __shared__ __align__(8) uint64_t full[kSpanStages], empty[kSpanStages];
    __shared__ __align__(16) int4 hdr[kSpanStages];      // c_first, nrows, nvec, -
    __shared__ __align__(16) uint32_t cst[kCstWords];    // loop invariants of the consumers (see SpanRegs)
    __shared__ uint8_t *tile_out[kSpanStages];           // where the stage's tile starts in its batch's output

    // Programmatic dependent launch: the next kernel of the stream may start its prologue now; ours (LUT, mask
    // tables, barriers: no global memory) runs before the previous kernel of the stream has finished.
    BSQ_SPAN_MARK(threadIdx.x == kSpanConsumers, kTrEntry);
    asm volatile("griddepcontrol.launch_dependents;");
    load_lut(lut, lutp);
    init_tailtab(tab, sp);
    if (threadIdx.x >= 160 && threadIdx.x < 176) {
        const int j = static_cast<int>(threadIdx.x) - 160;
        uint32_t hw[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const uint32_t mj = lt_mask(j, w), mjb = lt_mask(clamp16(j + sp.bos), w);
            hw[w] = (sp.pad_w & mj) | (sp.bos_w & mjb & ~mj);
        }
        headtab[j] = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    }
    if (threadIdx.x == 96) {
        cst[0] = static_cast<uint32_t>(q.padlen); cst[1] = q.div_mul; cst[2] = q.div_shift;
        cst[3] = static_cast<uint32_t>(sp.eos); cst[4] = sp.bos ? sp.bos_w : 0u; cst[5] = sp.bos ? 0x3214u : 0x3210u;
        cst[6] = static_cast<uint32_t>(-q.padlen); cst[7] = static_cast<uint32_t>(sp.bos);
        cst[8] = s_u32(lut); cst[9] = s_u32(&tab.m[0]); cst[10] = static_cast<uint32_t>(q.straddle); cst[11] = s_u32(&headtab[0]);
        cst[12] = cst[13] = cst[14] = cst[15] = sp.pad_w;
    }
    if (threadIdx.x == 128) {
#pragma unroll
        for (int s = 0; s < kSpanStages; ++s) {
            bar_init(full + s, 1);
            bar_init(empty + s, kSpanConsumerWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int stage_stride = q.stage_bytes + 16 * q.max_rows;
    const int tile_bytes = q.vt * 16;

    if (warp == kSpanConsumerWarps) {
        // ------------------------------- producer -------------------------------
        // Tile coordinates: first row r0 and column c_first of the tile's first byte, last row r1 / column c_last.
        struct Coord {
            int64_t r0, r1, f0;
            int c_first, c_last, batch, len;  // len: bytes of the tile (the batch's last tile may be short)
        };
        auto coord_of = [&](int64_t tt) {
            Coord c;
            int bi = 0;
            while (bi + 1 < q.nbatch && tt >= mb.b[bi + 1].first_tile) ++bi;
            c.batch = bi;
            c.f0 = (tt - mb.b[bi].first_tile) * tile_bytes;
            c.len = static_cast<int>(min(static_cast<int64_t>(tile_bytes), mb.b[bi].total - c.f0));
            c.r0 = c.f0 / q.padlen;
            c.c_first = static_cast<int>(c.f0 - c.r0 * q.padlen);
            const uint32_t e = static_cast<uint32_t>(c.c_first) + static_cast<uint32_t>(c.len) - 1u;
            const uint32_t dr = __umulhi(e, q.div_mul) >> q.div_shift;
            c.c_last = static_cast<int>(e - dr * static_cast<uint32_t>(q.padlen));
            c.r1 = c.r0 + dr;
            return c;
        };
        auto load_edges = [&](const Coord &c) {
            const int64_t *offs = mb.b[c.batch].offs;
            SpanEdges e;
            e.a0 = __ldg(offs + c.r0); e.a1 = __ldg(offs + c.r0 + 1);
            e.b0 = __ldg(offs + c.r1); e.b1 = __ldg(offs + c.r1 + 1);
            return e;
        };
        int64_t t = blockIdx.x;  // < ntiles (the grid is never larger)
        Coord cc = coord_of(t);
        const int maxlen = max(q.padlen - sp.bos - sp.eos, 0);
        {
            // Both static tiles go into L2 while the previous kernel drains (a prefetch is only a hint, the real loads
            // come after the wait): their offsets, and their residues from the offsets as they read NOW.  The previous
            // kernel of the stream may still be producing them, so these values are hints only: they go through L2
            // (ld.global.cg: nothing stale can stay in L1), address nothing but an L2 prefetch -- which is dropped when
            // its address is not mapped (tools/probes/prefetch_probe.cu) -- and are read again for real after the wait.
            const int64_t t1 = t + gridDim.x;
            const Coord pc[2] = {cc, t1 < q.ntiles ? coord_of(t1) : cc};
            const int npf = t1 < q.ntiles ? 2 : 1;
            int64_t sa[2] = {0, 0}, sb[2] = {0, 0};
            for (int k = 0; k < npf; ++k) {
                const int64_t *o = mb.b[pc[k].batch].offs;
                if (16 * lane <= pc[k].len / q.padlen + 2 && pc[k].r0 + 16 * lane <= mb.b[pc[k].batch].nseq)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(o + pc[k].r0 + 16 * lane));
                asm volatile("ld.global.cg.s64 %0, [%1];" : "=l"(sa[k]) : "l"(o + pc[k].r0));
                asm volatile("ld.global.cg.s64 %0, [%1];" : "=l"(sb[k]) : "l"(o + pc[k].r1 + 1));
            }
            for (int k = 0; k < npf; ++k) {
                const int64_t span = min(max(sb[k] - sa[k], int64_t(0)), static_cast<int64_t>(q.stage_bytes));
                const uintptr_t pa = reinterpret_cast<uintptr_t>(mb.b[pc[k].batch].bytes + sa[k]) & ~uintptr_t(15);
                const uint32_t pn = static_cast<uint32_t>((span + 31) & ~int64_t(15));
                if (lane == 0 && pn > 0) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(pa), "r"(pn) : "memory");
            }
        }
        asm volatile("griddepcontrol.wait;" ::: "memory");
        BSQ_SPAN_MARK(lane == 0, kTrWait);
        SpanEdges cur = load_edges(cc);
        unsigned int ask = 0;  // lane 0: the counter's answer for the tile after the next one, read one iteration later
        uint32_t it = 0;
        for (;; ++it) {
            const int s = static_cast<int>(it % kSpanStages);
            const uint32_t ph = (it / kSpanStages) & 1u;
            const uint8_t *bytes = mb.b[cc.batch].bytes;
            const int64_t *offs = mb.b[cc.batch].offs;
            const int nrows = static_cast<int>(cc.r1 - cc.r0) + 1;
            // the span: residues of columns [c_first, padlen) of row r0 ... [0, c_last] of row r1
            const int len0 = static_cast<int>(min(max(cur.a1 - cur.a0, int64_t(0)), static_cast<int64_t>(maxlen)));
            const int len1 = static_cast<int>(min(max(cur.b1 - cur.b0, int64_t(0)), static_cast<int64_t>(maxlen)));
            const int64_t lo = cur.a0 + min(max(cc.c_first - sp.bos, 0), len0);
            const int64_t hi = cur.b0 + min(max(cc.c_last + 1 - sp.bos, 0), len1);
            const uintptr_t A_lo = reinterpret_cast<uintptr_t>(bytes + lo) & ~uintptr_t(15);
            const uintptr_t A_hi = (reinterpret_cast<uintptr_t>(bytes + hi) + 15) & ~uintptr_t(15);
            const uint32_t nbytes = hi > lo ? static_cast<uint32_t>(min(static_cast<int64_t>(A_hi - A_lo),
                                                                         static_cast<int64_t>(q.stage_bytes - kSpanSlack - kSpanTail)))
                                            : 0u;
            uint8_t *stage = dyn + static_cast<size_t>(s) * stage_stride;
            int4 *rows = reinterpret_cast<int4 *>(stage + q.stage_bytes);
            // shared address of the byte that column 0 of row r0 + i comes from
            const int64_t base = static_cast<int64_t>(reinterpret_cast<uintptr_t>(bytes)) - static_cast<int64_t>(A_lo) + kSpanSlack - sp.bos +
                                 static_cast<int64_t>(s_u32(stage));
            auto row_entry = [&](int i) {  // {source address of column 0, bos + len, bos + len + eos, the previous row's bos + len + eos}
                const int64_t o0 = __ldg(offs + cc.r0 + i), o1 = __ldg(offs + cc.r0 + i + 1);
                const int n = sp.bos + static_cast<int>(min(max(o1 - o0, int64_t(0)), static_cast<int64_t>(maxlen)));
                int pn = 0;
                if (!ALIGNED && i > 0) pn = sp.bos + sp.eos + static_cast<int>(min(max(o0 - __ldg(offs + cc.r0 + i - 1), int64_t(0)), static_cast<int64_t>(maxlen)));
                return make_int4(static_cast<int>(o0 + base), n, n + sp.eos, pn);
            };
            // the first 32 rows' entries are formed before the barrier wait (their offsets are in flight meanwhile)
            int4 e0 = make_int4(0, 0, 0, 0);
            if (lane < nrows) e0 = row_entry(lane);
            if (it >= kSpanStages) bar_wait(s_u32(empty + s), ph ^ 1u);  // the consumers are done with this stage
            if (lane == 0) {
                if (nbytes) {
                    bar_expect_tx(s_u32(full + s), nbytes);
                    bulk_load(s_u32(stage + kSpanSlack), reinterpret_cast<const void *>(A_lo), nbytes, s_u32(full + s));
                }
                BSQ_SPAN_MARK(it == 0, kTrCopy0);
                // {first column, bytes to keep of a final partial vector (0: none), vectors, staged bytes}
                hdr[s] = make_int4(cc.c_first, cc.len & 15, (cc.len + 15) >> 4, static_cast<int>(nbytes));
                tile_out[s] = mb.b[cc.batch].out + cc.f0;
            }
            if (lane < nrows) rows[lane] = e0;
            for (int i = lane + 32; i < nrows; i += 32) rows[i] = row_entry(i);
            __syncwarp();
            if (lane == 0) bar_arrive(s_u32(full + s));  // release: row table + header visible to whoever sees the phase flip
            // The next tile: static for the first two, then the counter's answer to the request made one iteration ago,
            // so no atomic result is waited on before both static copies are in flight.  The counter is asked for the
            // tile after it now, and its edge offsets are loaded for the next iteration.
            const int64_t tn = (q.ctr == nullptr || it == 0) ? t + gridDim.x
                                                             : 2 * static_cast<int64_t>(gridDim.x) + __shfl_sync(0xffffffffu, ask, 0);
            if (tn >= q.ntiles) break;
            if (q.ctr != nullptr && lane == 0) ask = atomicAdd(q.ctr, 1u);
            t = tn;
            cc = coord_of(t);
            cur = load_edges(cc);
        }
        // end of work for this CTA: a stage whose header says so
        {
            ++it;
            const int s = static_cast<int>(it % kSpanStages);
            const uint32_t ph = (it / kSpanStages) & 1u;
            if (it >= kSpanStages) bar_wait(s_u32(empty + s), ph ^ 1u);
            if (lane == 0) {
                hdr[s] = make_int4(0, 0, -1, 0);
                bar_arrive(s_u32(full + s));
            }
#ifdef BSQ_SPAN_TRACE
            if (lane == 0) span_trace_word(q, 6, span_smid()), span_trace_word(q, 7, it);
#endif
        }
        // the last CTA to see the end of the tiles re-arms the counter for the next launch that uses this slot
        if (q.ctr != nullptr && lane == 0) {
            __threadfence();
            if (atomicAdd(q.ctr + 1, 1u) == gridDim.x - 1) {
                q.ctr[0] = 0u;
                q.ctr[1] = 0u;
                __threadfence();
            }
        }
        return;
    }

    // ------------------------------- consumers -------------------------------
    const int ctid = threadIdx.x;  // 0 .. kSpanConsumers-1
    SpanRegs g;
    const uint32_t cst_a = s_u32(cst);
    g.padlen = static_cast<int>(lds32(cst_a));
    g.mul = lds32(cst_a + 4u);
    g.shift = lds32(cst_a + 8u);
    g.eos = static_cast<int>(lds32(cst_a + 12u));
    g.bos_w = lds32(cst_a + 16u);
    g.bos_sel = lds32(cst_a + 20u);
    g.neg_padlen = static_cast<int>(lds32(cst_a + 24u));
    g.bos = static_cast<int>(lds32(cst_a + 28u));
    g.lutb = lds32(cst_a + 32u);
    g.tab_m = lds32(cst_a + 36u);
    g.straddle = static_cast<int>(lds32(cst_a + 40u));
    g.tab_h = lds32(cst_a + 44u);
    g.padq = lds128(cst_a + 48u);
    const uint32_t dyn_a = s_u32(dyn);
    for (uint32_t it = 0;; ++it) {
        const int s = static_cast<int>(it % kSpanStages);
        const uint32_t ph = (it / kSpanStages) & 1u;
        const uint32_t rows_a = dyn_a + static_cast<uint32_t>(s * stage_stride + q.stage_bytes);
        bar_wait(s_u32(full + s), ph);
        BSQ_SPAN_MARK(it == 0 && ctid == 0, kTrFull0);
        const int4 h = hdr[s];
        if (h.z < 0) break;  // no more tiles for this CTA
        uint8_t *const otile = tile_out[s];
        // F: column-space offset of the lane's vector from column 0 of the tile's first row
        uint32_t F = static_cast<uint32_t>(h.x) + 16u * static_cast<uint32_t>(ctid);
        const uint32_t Fend = static_cast<uint32_t>(h.x) + 16u * static_cast<uint32_t>(h.z);
        uint8_t *dst = otile + 16 * ctid;
        if (ALIGNED) {
            for (; F < Fend; F += 16u * kSpanConsumers, dst += 16 * kSpanConsumers) {
                const uint32_t rl = __umulhi(F, g.mul) >> g.shift;
                const int col = static_cast<int>(rl * static_cast<uint32_t>(g.neg_padlen) + F);
                const int4 ri = lds128i(rows_a + 16u * rl);  // {shared address of column 0's source byte, bos + len, bos + len + eos, -}
                if (col >= ri.z) __stcs(reinterpret_cast<uint4 *>(dst), g.padq);
                else __stcs(reinterpret_cast<uint4 *>(dst), span_row_codes(static_cast<uint32_t>(ri.x), ri.y, col, g));
                BSQ_SPAN_MARK(it == 0 && ctid == 0 && dst == otile, kTrStore0);
            }
        } else {
            // padlen % 16 != 0: vectors stay 16-byte aligned in the flat output, so one vector per row straddles two rows.
            // A vector belongs to the row that holds its LAST byte: its columns run from col in [-15, padlen - 16], the
            // bytes left of column 0 are the previous row's tail -- pad, unless that row is nearly full (rare: the general
            // path).  So the straddling vector costs one translation like any other, in the same instruction stream.
            const bool partial_tail = h.y != 0;  // the batch's final vector is cut short
            const uint32_t Fsafe = partial_tail ? Fend - 16u : Fend;
            for (; F < Fsafe; F += 16u * kSpanConsumers, dst += 16 * kSpanConsumers) {
                const uint32_t rl = __umulhi(F + 15u, g.mul) >> g.shift;
                const int col = static_cast<int>(rl * static_cast<uint32_t>(g.neg_padlen) + F);
                const int4 ri = lds128i(rows_a + 16u * rl);  // {source address of column 0, bos + len, bos + len + eos, the previous row's bos + len + eos}
                if (col >= ri.z) {
                    __stcs(reinterpret_cast<uint4 *>(dst), g.padq);
                } else if (col >= 0 || ri.w <= g.padlen + col) {
                    __stcs(reinterpret_cast<uint4 *>(dst), span_row_codes_u(static_cast<uint32_t>(ri.x), ri.y, col, g));
                } else {
                    __stcs(reinterpret_cast<uint4 *>(dst), span_straddle_general(rows_a, rl, col, g));
                }
                BSQ_SPAN_MARK(it == 0 && ctid == 0 && dst == otile, kTrStore0);
            }
            if (partial_tail && F == Fsafe) {  // exactly one lane of the CTA: the final vector, bytewise
                const uint32_t rl = __umulhi(F, g.mul) >> g.shift;  // the row of its first byte (the batch's last row)
                const int col = static_cast<int>(rl * static_cast<uint32_t>(g.neg_padlen) + F);
                const int4 ri = lds128i(rows_a + 16u * rl);
                uint4 codes = g.padq;
                if (col < ri.z) codes = span_row_codes_u(static_cast<uint32_t>(ri.x), ri.y, col, g);
                const int keep = h.y;
                const uint32_t w[4] = {codes.x, codes.y, codes.z, codes.w};
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (j < keep) dst[j] = static_cast<uint8_t>(w[j >> 2] >> (8 * (j & 3)));
            }
        }
        __syncwarp();
        if (lane == 0) bar_arrive(s_u32(empty + s));
    }
    BSQ_SPAN_MARK(lane == 0, kTrExit);
}

struct DevInfo {
    int sms = 0;
    bool attr_set[2] = {};  // per ALIGNED: the kernel's shared-memory limit has been raised
    // tile counters of the dynamic scheduler: kCtrPairs x 2 slots x {handed out, CTAs done}, zero when idle (the
    // kernel re-arms its slot itself).  A stream owns a pair of slots and alternates between them: kernels of one
    // stream touch their counter only after the previous kernel of the stream has completed (griddepcontrol.wait /
    // stream order), so two slots per stream can never be in use by more than their own launch.
    unsigned int *ctr = nullptr;
    bool ctr_failed = false;
    std::unordered_map<cudaStream_t, int> pair_of;  // stream -> 2 * pair index + flip
};
constexpr int kCtrPairs = 1024;

#ifdef BSQ_SPAN_TRACE
unsigned long long *g_span_trace = nullptr;  // where the next launches record their timeline (bsq_span_trace_arm)
#endif

std::mutex g_dev_mu;
DevInfo &dev_info(int dev) {
    static DevInfo info[64];
    DevInfo &d = info[dev & 63];
    if (d.sms == 0) cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, dev);
    return d;
}

// Counter slot for a launch on `st`, or nullptr (stream capture in progress, no memory, more than kCtrPairs streams):
// the kernel then falls back to the static tile order.
unsigned int *span_counter(DevInfo &d, cudaStream_t st) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (cap != cudaStreamCaptureStatusNone) return nullptr;  // a captured launch may be replayed concurrently with itself
    if (d.ctr == nullptr) {
        if (d.ctr_failed) return nullptr;
        if (cudaMalloc(reinterpret_cast<void **>(&d.ctr), sizeof(unsigned int) * 4 * kCtrPairs) != cudaSuccess ||
            cudaMemset(d.ctr, 0, sizeof(unsigned int) * 4 * kCtrPairs) != cudaSuccess) {
            cudaGetLastError();
            d.ctr = nullptr;
            d.ctr_failed = true;
            return nullptr;
        }
    }
    auto it = d.pair_of.find(st);
    if (it == d.pair_of.end()) {
        if (static_cast<int>(d.pair_of.size()) >= kCtrPairs) return nullptr;
        it = d.pair_of.emplace(st, 2 * static_cast<int>(d.pair_of.size())).first;
    }
    it->second ^= 1;
    return d.ctr + 2 * it->second;  // slot index = 2 * pair + flip, two words per slot
}

}  // namespace

// n / d = umulhi(n, mul) >> shift for every 0 <= n < 2^31 and 2 <= d <= 2^30 (round-up magic number with one
// bit of headroom: no add-back step, two instructions per division).
void span_magic(uint32_t d, uint32_t *mul, uint32_t *shift) {
    uint32_t s = 0;
    while ((1ull << s) < d) ++s;
    *mul = static_cast<uint32_t>((1ull << (31 + s)) / d + 1);
    *shift = s - 1;
}

// SMs of a device (cached): grids are sized from this, never from a constant
int sm_count(int device) {
    std::lock_guard<std::mutex> g(g_dev_mu);
    const int n = dev_info(device).sms;
    return n > 0 ? n : 148;
}

unsigned int *tile_counter_slot(int device, cudaStream_t st) {
    std::lock_guard<std::mutex> dev_lock(g_dev_mu);
    return span_counter(dev_info(device), st);
}

// Launches K1s over `nbatch` (<= kSpanManyMax) batches that share padlen and tokenizer; `device` is the current device.
int launch_tokenize_span_many(int device, cudaStream_t st, int nbatch, const uint8_t *const *d_bytes, const int64_t *const *d_offs,
                              const int64_t *nseqs, int64_t padlen, const Prepared &p, uint8_t *const *outs) {
    if (nbatch <= 0 || nbatch > kSpanManyMax) return fail(BSQ_ERR_ARG, "bad batch count");
    std::lock_guard<std::mutex> dev_lock(g_dev_mu);
    DevInfo &di = dev_info(device);
    const int sms = di.sms > 0 ? di.sms : 148;
    int64_t V = 0, max_nseq = 0;  // 16-byte output vectors of all batches
    for (int k = 0; k < nbatch; ++k) {
        V += (nseqs[k] * padlen + 15) / 16;
        max_nseq = std::max(max_nseq, nseqs[k]);
    }
    if (V == 0) return BSQ_OK;
    // stage: slack + span (<= tile bytes + 32) + tail, plus the row table
    auto smem_for = [&](int vt) {
        const int stage_bytes = (kSpanSlack + vt * 16 + 32 + kSpanTail + 127) / 128 * 128;
        const int max_rows = static_cast<int>(std::min<int64_t>(vt * 16 / padlen + 3, max_nseq + 1));
        return static_cast<size_t>(kSpanStages) * (stage_bytes + 16 * ((max_rows + 7) / 8 * 8));
    };
    const size_t static_smem = 256 + sizeof(TailTab) + 16 * kSpanStages * 2 + 1024;
    int per_sm = static_cast<int>((227 * 1024) / (smem_for(kSpanTileVecs) + static_smem));
    per_sm = std::max(1, std::min(std::min(per_sm, 2048 / kSpanThreads), kSpanCtasPerSm));
    const int64_t grid_full = static_cast<int64_t>(sms) * per_sm;
    // tiles: at most kSpanTileVecs vectors, and a count that fills whole rounds of the persistent grid
    const int64_t rounds = std::max<int64_t>(1, (V + grid_full * kSpanTileVecs - 1) / (grid_full * kSpanTileVecs));
    int64_t vt = (V + grid_full * rounds - 1) / (grid_full * rounds);
    vt = std::min<int64_t>(kSpanTileVecs, (vt + kSpanConsumers - 1) / kSpanConsumers * kSpanConsumers);
    SpanBatches mb = {};
    int64_t ntiles = 0;
    int nb = 0;
    for (int k = 0; k < nbatch; ++k) {
        if (nseqs[k] <= 0) continue;
        SpanBatch &b = mb.b[nb++];
        b.bytes = d_bytes[k];
        b.offs = d_offs[k];
        b.out = outs[k];
        b.nseq = nseqs[k];
        b.total = nseqs[k] * padlen;
        b.first_tile = ntiles;
        ntiles += ((b.total + 15) / 16 + vt - 1) / vt;
    }
    SpanParams q;
    q.ntiles = ntiles;
    q.nbatch = nb;
    q.padlen = static_cast<int>(padlen);
    q.vt = static_cast<int>(vt);
    q.stage_bytes = (kSpanSlack + static_cast<int>(vt) * 16 + 32 + kSpanTail + 127) / 128 * 128;
    q.max_rows = (static_cast<int>(std::min<int64_t>(vt * 16 / padlen + 3, max_nseq + 1)) + 7) / 8 * 8;
    span_magic(static_cast<uint32_t>(padlen), &q.div_mul, &q.div_shift);
#ifdef BSQ_SPAN_TRACE
    q.trace = g_span_trace;
#endif
    q.straddle = padlen % 512 != 0;
    const size_t smem = static_cast<size_t>(kSpanStages) * (q.stage_bytes + 16 * q.max_rows);
    const bool aligned = padlen % 16 == 0;

    const int64_t blocks = std::min<int64_t>(ntiles, grid_full);
    q.ctr = ntiles < 0x7fffffffll ? span_counter(di, st) : nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(blocks));
    cfg.blockDim = dim3(kSpanThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    // Programmatic dependent launch hides this launch's ramp behind the previous kernel's tail.  With the dynamic tile
    // order any co-residency is fine; with the static order two whole persistent grids must fit on the SMs at once
    // (otherwise the late CTAs pile up on the first SMs to drain and the fixed partition becomes unbalanced).
    const bool pdl = q.ctr != nullptr || (2 * per_sm * (smem + static_smem) <= 227 * 1024 && 2 * per_sm * kSpanThreads <= 2048);
    cfg.numAttrs = pdl ? 1 : 0;

    const auto kern = aligned ? tokenize_span_kernel<true> : tokenize_span_kernel<false>;
    if (!di.attr_set[aligned]) {
        BSQ_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        di.attr_set[aligned] = true;
    }
    BSQ_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, q, mb, p.lut, p.sp));
    count_launch();
    return BSQ_OK;
}

int launch_tokenize_span(int device, cudaStream_t st, const SeqView &v, int64_t nseq, int64_t padlen, const Prepared &p, uint8_t *out) {
    return launch_tokenize_span_many(device, st, 1, &v.bytes, &v.offs, &nseq, padlen, p, &out);
}

}  // namespace bsq

#ifdef BSQ_SPAN_TRACE
// Traced builds only (not part of include/bsq.h): K1s launches from now on record their per-CTA timeline into `buf`
// (kSpanTraceWords 64-bit words per CTA, zeroed by the caller); nullptr stops recording.
extern "C" void bsq_span_trace_arm(void *buf) {
    std::lock_guard<std::mutex> g(bsq::g_dev_mu);
    bsq::g_span_trace = static_cast<unsigned long long *>(buf);
}
#endif
