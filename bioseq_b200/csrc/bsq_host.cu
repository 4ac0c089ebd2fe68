// Host side of libbsq.so: error state, launch counter, the pack layer (ragged host
// sequences -> pinned bytes + int64 offsets) and the host-staged pipeline that overlaps
// host->device copies with the kernels.
//
// Reference counterpart: the serial unpack loop and borrowed-pointer vector of
// src/tokenize.h:386-419 (transencode) / :289-322 (one-hot); the caller-side
// `torch.from_numpy(arr).to(device)` (bioseq/loaders.py:84) is what the staging replaces.
#include <cuda_runtime.h>
#if defined(__x86_64__)
#include <cpuid.h>
#include <immintrin.h>  // _mm_sfence
#endif

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <pthread.h>
#include <sched.h>
#include <string>
#include <thread>
#include <vector>

#include "bsq_internal.h"

namespace bsq {

namespace {
thread_local std::string g_last_error;
thread_local int64_t g_launches = 0;
}  // namespace

int fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}
void count_launch(int n) { g_launches += n; }

}  // namespace bsq

using bsq::fail;

// ---------------------------------------------------------------------------------------
// worker pool: persistent host threads for the gather (items -> pinned pack) and scatter
// (pinned ring -> Python string bodies) loops.  The submitting thread keeps running (it issues the CUDA
// copies and launches) and joins with wait().  A team of threads runs one job at a time; callers that
// arrive while a team is busy (other Python threads, other devices) get another team -- up to kTeams --
// instead of queueing behind it.
// ---------------------------------------------------------------------------------------
namespace {

thread_local bool t_in_pool_worker = false;  // set on pool threads: a nested parallel section runs inline instead

class Team {
public:
    bool try_claim() { return job_mu_.try_lock(); }
    void claim() { job_mu_.lock(); }
    // run fn(t) for t in [0, nt) on the team's threads; returns at once.  The team is claimed; wait() releases it.
    void start(int nt, std::function<void(int)> fn) {
        std::unique_lock<std::mutex> lk(mu_);
        while (static_cast<int>(threads_.size()) < nt) {
            const int id = static_cast<int>(threads_.size());
            threads_.emplace_back([this, id] { loop(id); });
            threads_.back().detach();
        }
        fn_ = std::move(fn);
        nt_ = nt;
        pending_ = nt;
        ++generation_;
        lk.unlock();
        cv_.notify_all();
    }
    void wait() {
        std::unique_lock<std::mutex> lk(mu_);
        done_cv_.wait(lk, [this] { return pending_ == 0; });
        fn_ = nullptr;
        lk.unlock();
        job_mu_.unlock();
    }

private:
    void loop(int id) {
        uint64_t seen = 0;
        for (;;) {
            std::function<void(int)> fn;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return generation_ != seen; });
                seen = generation_;
                if (id >= nt_) continue;
                fn = fn_;
            }
            t_in_pool_worker = true;
            fn(id);
            t_in_pool_worker = false;
            std::lock_guard<std::mutex> lk(mu_);
            if (--pending_ == 0) done_cv_.notify_all();
        }
    }
    std::mutex job_mu_, mu_;
    std::condition_variable cv_, done_cv_;
    std::vector<std::thread> threads_;
    std::function<void(int)> fn_;
    int nt_ = 0, pending_ = 0;
    uint64_t generation_ = 0;
};

class Pool {
public:
    static constexpr int kTeams = 4;
    static Pool &get() {
        // leaked: worker threads must not be torn down under a running job at exit.  After fork() the child has
        // none of the parent's threads, so it starts over with empty teams (a forked DataLoader worker that only
        // walks items would otherwise wait for workers that do not exist).
        static std::once_flag once;
        std::call_once(once, [] {
            instance() = new Pool();
            pthread_atfork(nullptr, nullptr, [] { instance() = new Pool(); });
        });
        return *instance();
    }
    // run fn(t) for t in [0, nt) on a free team (the first team when all are busy: queue there); returns at once.
    // Pair with wait() on the same thread.
    void start(int nt, std::function<void(int)> fn) {
        Team *team = nullptr;
        for (int k = 0; k < kTeams && team == nullptr; ++k)
            if (teams_[k].try_claim()) team = &teams_[k];
        if (team == nullptr) {
            team = &teams_[0];
            team->claim();
        }
        mine() = team;
        team->start(nt, std::move(fn));
    }
    void wait() {
        Team *team = mine();
        mine() = nullptr;
        if (team != nullptr) team->wait();
    }

private:
    static Pool *&instance() {
        static Pool *p = nullptr;
        return p;
    }
    static Team *&mine() {  // the team this thread's job in flight runs on
        static thread_local Team *t = nullptr;
        return t;
    }
    Team teams_[kTeams];
};

// Pool threads worth using for a memory-bound host loop: the caller's wish, capped at three quarters of the CPUs
// this process may use (16-core B200 host, streamed item pipeline, 35 MB batch: 8 workers 1.18 ms, 12 workers
// 0.875 ms, 15 workers 0.878 ms -- the submitting thread needs a core of its own and the host memory system is
// saturated by then).  BSQ_POOL_CAP overrides the cap.
inline int pool_threads(int wanted) {
    static const int cap = [] {
        cpu_set_t set;  // the CPUs this process may run on (a container's cpuset), not the machine's
        CPU_ZERO(&set);
        const int n = sched_getaffinity(0, sizeof(set), &set) == 0 ? CPU_COUNT(&set) : static_cast<int>(std::thread::hardware_concurrency());
        if (const char *e = std::getenv("BSQ_POOL_CAP")) return std::max(1, std::atoi(e));
        return std::max(1, n * 3 / 4);
    }();
    if (t_in_pool_worker) return 1;  // the pool runs one job at a time: a worker must not wait for it
    return std::max(1, std::min(std::min(wanted, cap), 64));
}

// Write the cache lines of [p, p + n) back to memory (clwb keeps them valid in the cache); no-op without clwb.
// The gathered bytes are read next by the DMA engine, and lines still dirty in the cores' caches slow that read
// down: without the write-back the last copy of a gathered 35 MB batch finished ~1 ms after it was issued (device done
// 2.0 ms after the call started, vs 1.45 ms with it; non-temporal stores also fix the lag but make the gather 2x slower).
inline bool have_clwb() {
#if defined(__x86_64__)
    static const bool ok = [] {
        unsigned a, b, c, d;
        if (!__get_cpuid_count(7, 0, &a, &b, &c, &d)) return false;
        return ((b >> 24) & 1u) != 0;
    }();
    return ok;
#else
    return false;
#endif
}
inline void writeback_lines(const uint8_t *p, size_t n) {
#if defined(__x86_64__)
    if (n == 0 || !have_clwb()) return;
    const uintptr_t lo = reinterpret_cast<uintptr_t>(p) & ~uintptr_t(63), hi = reinterpret_cast<uintptr_t>(p) + n;
    for (uintptr_t a = lo; a < hi; a += 64) asm volatile("clwb (%0)" ::"r"(a) : "memory");
#endif
}
inline void copy_fence() {
#if defined(__x86_64__)
    _mm_sfence();
#endif
}

inline void spin_until(const std::function<bool()> &ready) {
    for (int i = 0; !ready(); ++i) {
        if (i < 64) std::this_thread::yield();
        else std::this_thread::sleep_for(std::chrono::microseconds(20));
    }
}

}  // namespace

// ---------------------------------------------------------------------------------------
// pack layer
// ---------------------------------------------------------------------------------------
struct bsq_pack {
    int pinned = 0;
    uint8_t *bytes = nullptr;
    size_t cap_bytes = 0;
    int64_t *offs = nullptr;
    size_t cap_offs = 0;  // entries
    int64_t nseq = 0, nbytes = 0, maxlen = 0;
};

namespace {

int host_alloc(void **p, size_t n, int pinned) {
    if (pinned) {
        BSQ_CUDA_TRY(cudaHostAlloc(p, n, cudaHostAllocPortable));
    } else {
        *p = std::malloc(n);
        if (*p == nullptr) return fail(BSQ_ERR_NOMEM, "out of host memory");
    }
    return BSQ_OK;
}
void host_free(void *p, int pinned) {
    if (p == nullptr) return;
    if (pinned) cudaFreeHost(p);
    else std::free(p);
}

int pack_reserve(bsq_pack *p, int64_t nbytes, int64_t nseq) {
    // +32: the kernels read whole aligned 16-byte words around the residues
    const size_t want_b = static_cast<size_t>(nbytes) + 32, want_o = static_cast<size_t>(nseq) + 1;
    if (want_b > p->cap_bytes) {
        host_free(p->bytes, p->pinned);
        p->bytes = nullptr;
        p->cap_bytes = 0;
        const size_t cap = std::max(want_b + want_b / 4, size_t(1) << 16);
        if (int rc = host_alloc(reinterpret_cast<void **>(&p->bytes), cap, p->pinned)) return rc;
        p->cap_bytes = cap;
    }
    if (want_o > p->cap_offs) {
        host_free(p->offs, p->pinned);
        p->offs = nullptr;
        p->cap_offs = 0;
        const size_t cap = std::max(want_o + want_o / 4, size_t(1) << 10);
        if (int rc = host_alloc(reinterpret_cast<void **>(&p->offs), cap * sizeof(int64_t), p->pinned)) return rc;
        p->cap_offs = cap;
    }
    return BSQ_OK;
}

}  // namespace

extern "C" {

int bsq_pack_create(bsq_pack **out, int pinned) {
    if (out == nullptr) return fail(BSQ_ERR_ARG, "null argument");
    *out = new bsq_pack();
    (*out)->pinned = pinned != 0;
    return BSQ_OK;
}

void bsq_pack_destroy(bsq_pack *p) {
    if (p == nullptr) return;
    host_free(p->bytes, p->pinned);
    host_free(p->offs, p->pinned);
    delete p;
}

int bsq_pack_gather(bsq_pack *p, const void *const *ptrs, const int64_t *lens, int64_t n, int nthreads) {
    if (p == nullptr || n < 0 || (n > 0 && (ptrs == nullptr || lens == nullptr))) return fail(BSQ_ERR_ARG, "bad pack arguments");
    int64_t total = 0, maxlen = 0;
    for (int64_t i = 0; i < n; ++i) {
        if (lens[i] < 0) return fail(BSQ_ERR_ARG, "negative sequence length");
        total += lens[i];
        maxlen = std::max(maxlen, lens[i]);
    }
    if (int rc = pack_reserve(p, total, n)) return rc;
    int64_t acc = 0;
    for (int64_t i = 0; i < n; ++i) {
        p->offs[i] = acc;
        acc += lens[i];
    }
    p->offs[n] = acc;
    p->nseq = n;
    p->nbytes = total;
    p->maxlen = maxlen;

    const bool pinned = p->pinned != 0;
    auto copy_range = [&](int64_t lo, int64_t hi) {
        if (hi <= lo) return;
        for (int64_t i = lo; i < hi; ++i)
            if (lens[i] > 0) std::memcpy(p->bytes + p->offs[i], ptrs[i], static_cast<size_t>(lens[i]));
        if (pinned) {  // read next by the DMA engine: see writeback_lines
            writeback_lines(p->bytes + p->offs[lo], static_cast<size_t>(p->offs[hi] - p->offs[lo]));
            copy_fence();
        }
    };
    int nt = pool_threads(nthreads);
    nt = static_cast<int>(std::min<int64_t>(nt, std::max<int64_t>(1, total >> 20)));  // >= 1 MiB per thread
    if (nt <= 1) {
        copy_range(0, n);
    } else {
        // shares split by bytes, not by count, so ragged batches stay balanced
        Pool &pool = Pool::get();
        pool.start(nt, [&, nt](int t) {
            auto cut = [&](int u) {
                if (u <= 0) return int64_t(0);
                if (u >= nt) return n;
                return static_cast<int64_t>(std::lower_bound(p->offs, p->offs + n, total * u / nt) - p->offs);
            };
            copy_range(cut(t), cut(t + 1));
        });
        pool.wait();
    }
    std::memset(p->bytes + total, 0, 32);
    return BSQ_OK;
}

const uint8_t *bsq_pack_bytes(const bsq_pack *p) { return p ? p->bytes : nullptr; }
const int64_t *bsq_pack_offsets(const bsq_pack *p) { return p ? p->offs : nullptr; }
int64_t bsq_pack_nseq(const bsq_pack *p) { return p ? p->nseq : 0; }
int64_t bsq_pack_nbytes(const bsq_pack *p) { return p ? p->nbytes : 0; }
int64_t bsq_pack_maxlen(const bsq_pack *p) { return p ? p->maxlen : 0; }

int bsq_check_lengths_host(const int64_t *h_offsets, int64_t nseq, int64_t padlen, const bsq_tokenizer *tok) {
    if (tok == nullptr) return fail(BSQ_ERR_ARG, "null tokenizer");
    if (padlen <= 0) return fail(BSQ_ERR_ARG, "batch tokenize requires padlen is provded.");  // src/tokenize.h:383
    if (nseq < 0 || (nseq > 0 && h_offsets == nullptr)) return fail(BSQ_ERR_ARG, "bad offsets");
    const int64_t extra = (tok->bos_id >= 0) + (tok->eos_id >= 0);
    if (nseq > 0 && h_offsets[0] < 0) return fail(BSQ_ERR_ARG, "offsets must start at or after 0");
    for (int64_t i = 0; i < nseq; ++i) {
        const int64_t len = h_offsets[i + 1] - h_offsets[i];
        if (len < 0) return fail(BSQ_ERR_ARG, "offsets must be non-decreasing");
        if (len + extra > padlen)  // src/tokenize.h:456-459
            return fail(BSQ_ERR_TOO_LONG, "seq len + bos + eos > padlen: " + std::to_string(len + extra) + ", vs padlen " +
                                              std::to_string(padlen));
    }
    return BSQ_OK;
}

const char *bsq_last_error(void) { return bsq::g_last_error.c_str(); }
int64_t bsq_launch_count(void) { return bsq::g_launches; }
void bsq_launch_count_reset(void) { bsq::g_launches = 0; }

}  // extern "C"

// ---------------------------------------------------------------------------------------
// host-staged pipeline
// ---------------------------------------------------------------------------------------
namespace {
constexpr int kRingSlots = 4;
constexpr size_t kChunkBytes = size_t(4) << 20;  // residues per pipeline stage
constexpr int64_t kSeqAlign = 128;               // chunk boundaries: whole tiles / 16-byte aligned rows
constexpr size_t kFetchBytes = size_t(8) << 20;  // decoded characters per device -> host stage
}  // namespace

// Device-side staging of one batch in flight: residues (+ mask) and offsets, and the event that says the kernels
// reading them have finished.  Two slots alternate call by call, so the copies of call k+1 never wait for the
// kernels of call k (they used to: one buffer, stream-wait on `done` before the first copy).
struct DevSlot {
    uint8_t *d_bytes = nullptr, *d_mask = nullptr;
    int64_t *d_offs = nullptr;
    size_t cap_bytes = 0, cap_mask = 0, cap_offs = 0;
    cudaEvent_t done = nullptr;  // completion of the kernels of the call that used this slot last
    bool busy = false;
};
constexpr int kDevSlots = 2;

struct bsq_stager {
    int device = 0;
    cudaStream_t copy_stream = nullptr;
    DevSlot slot[kDevSlots];
    int cur = 0;  // slot of the call in progress / of the last call
    uint8_t *ring[kRingSlots] = {};
    cudaEvent_t ring_free[kRingSlots] = {};
    bool ring_used[kRingSlots] = {};
    int ring_next = 0;
    std::vector<cudaEvent_t> events;  // one per chunk in flight
    cudaEvent_t grow_ev = nullptr;    // orders a staging buffer's release behind the kernels that still read it
    // device -> host ring of bsq_fetch_rows
    uint8_t *fetch_ring[kRingSlots] = {};
    cudaEvent_t fetch_ev[kRingSlots] = {};
    // BLOSUM62 augmentation applied to every staged range before it is tokenised (chain_len 0 = off)
    int aug_chain = 0;
    double aug_frac = 0.0;
    uint64_t aug_seed = 0;
    int64_t aug_base = 0;
    // pinned-ness of host buffers seen before (cudaPointerGetAttributes is a driver call; callers hand the same
    // pinned buffers over again and again)
    const void *pin_key[8] = {};
    size_t pin_len[8] = {};
    bool pin_val[8] = {};
    int pin_next = 0;
    // streamed item batches (bsq_*_stream_items): two pinned packs alternate call by call, each with the event of
    // the last copy that read it, plus the per-item scratch arrays
    bsq_pack ipack[2];
    cudaEvent_t ipack_ev[2] = {nullptr, nullptr};
    bool ipack_used[2] = {false, false};
    int ipack_next = 0;
    std::vector<const void *> it_ptrs;
    std::vector<int64_t> it_lens;
    int64_t avg_len_hint = 512;
};

namespace {

// Grows a device staging buffer, stream-ordered on the stager's copy stream (cudaFreeAsync / cudaMallocAsync): no
// device-wide synchronisation, other streams of the device keep running.  The copy stream already waits for the kernels
// that read the slot's previous contents (slot_begin); `reader`, if given, is a stream with kernels of the CURRENT call
// that still read the old buffer.
int dev_reserve(bsq_stager *s, void **p, size_t *cap, size_t want, cudaStream_t reader = nullptr, bool have_reader = false) {
    if (want <= *cap) return BSQ_OK;
    if (*p != nullptr) {
        if (have_reader) {
            if (s->grow_ev == nullptr) BSQ_CUDA_TRY(cudaEventCreateWithFlags(&s->grow_ev, cudaEventDisableTiming));
            BSQ_CUDA_TRY(cudaEventRecord(s->grow_ev, reader));
            BSQ_CUDA_TRY(cudaStreamWaitEvent(s->copy_stream, s->grow_ev, 0));
        }
        BSQ_CUDA_TRY(cudaFreeAsync(*p, s->copy_stream));
    }
    *p = nullptr;
    *cap = 0;
    const size_t n = want + want / 4 + 256;
    BSQ_CUDA_TRY(cudaMallocAsync(p, n, s->copy_stream));
    *cap = n;
    return BSQ_OK;
}

bool is_pinned(const void *p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost;
}
// Cached form for the [p, p + n) ranges a stager is handed: a hit needs the same start and a length the earlier
// answer covered (a pinned registration covers whole allocations, so a shorter range of one is pinned too; a buffer
// that was freed and re-allocated pageable at the same address with a larger size is asked about again).
bool is_pinned_cached(bsq_stager *s, const void *p, size_t n) {
    if (p == nullptr) return false;
    for (int i = 0; i < 8; ++i)
        if (s->pin_key[i] == p && n <= s->pin_len[i] && s->pin_val[i]) return true;
    const bool v = is_pinned(p);
    if (v) {  // only positive answers are cached: "pageable" must stay safe if the caller pins the buffer later
        const int k = s->pin_next;
        s->pin_next = (k + 1) % 8;
        s->pin_key[k] = p;
        s->pin_len[k] = n;
        s->pin_val[k] = true;
    }
    return v;
}

// Software write-combining for the host copies into pinned memory (the gather of item batches, the bounce of pageable
// sources).  In the gather a thread's share of a range lands in ONE contiguous run of the pinned pack, so the ~0.5 KB items are first appended to a 4 KiB line-aligned buffer in L1 and leave as whole 64-byte lines
// with non-temporal stores.  Against memcpy + clwb this removes the read-for-ownership of every destination line and the
// separate write-back pass: per batch the host memory system moves source read + pack write + DMA read instead of
// those plus a second read of the pack -- and the host memory bandwidth is what bounds the drop-in call on the 16-core
// B200 host (12 threads: 0.875 ms per 35 MB batch with memcpy + clwb).
struct WcStream {
    alignas(64) uint8_t buf[4096];
    uint8_t *dst;   // next line-aligned destination address
    size_t fill = 0;
    explicit WcStream(uint8_t *aligned_dst) : dst(aligned_dst) {}
    void flush_lines(size_t nbytes) {  // nbytes: a multiple of 64, <= fill
#if defined(__x86_64__)
        for (size_t o = 0; o < nbytes; o += 64) {
            const __m128i a = _mm_load_si128(reinterpret_cast<const __m128i *>(buf + o)), b = _mm_load_si128(reinterpret_cast<const __m128i *>(buf + o + 16));
            const __m128i c = _mm_load_si128(reinterpret_cast<const __m128i *>(buf + o + 32)), d = _mm_load_si128(reinterpret_cast<const __m128i *>(buf + o + 48));
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + o), a);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + o + 16), b);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + o + 32), c);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + o + 48), d);
        }
#else
        std::memcpy(dst, buf, nbytes);
#endif
        dst += nbytes;
    }
    void append(const uint8_t *p, size_t n) {
        while (n > 0) {
            const size_t m = std::min(n, sizeof(buf) - fill);
            std::memcpy(buf + fill, p, m);
            fill += m; p += m; n -= m;
            if (fill == sizeof(buf)) {
                flush_lines(sizeof(buf));
                fill = 0;
            }
        }
    }
    // whole lines out; the trailing partial line (shared with the next thread's run) goes with ordinary stores
    void finish() {
        const size_t whole = fill & ~size_t(63);
        flush_lines(whole);
        if (fill > whole) {
            std::memcpy(dst, buf + whole, fill - whole);
            writeback_lines(dst, fill - whole);
        }
        fill = 0;
    }
};

// host -> device copy of n bytes on the copy stream.  Pinned sources go as one cudaMemcpyAsync.  Pageable sources
// (plain numpy arrays, a mapped FlatFile) bounce through a ring of pinned 4 MiB slots: pool threads fill slot after slot
// (write-combining non-temporal stores, each thread a contiguous share of the slot) and run up to kRingSlots - 1 slots
// ahead of the DMA engine, while this thread enqueues the copy of every slot as soon as it is full.  One pool job per
// transfer: no per-slot dispatch (it cost ~50 us of condition-variable wake-ups per 75 us of DMA).
struct BounceShared {
    const uint8_t *src;
    size_t n, nchunks;
    int nt;
    uint8_t *ring[kRingSlots];
    std::vector<std::atomic<int>> filled;  // per chunk: threads done
    std::atomic<int64_t> released{0};      // chunks whose DMA has completed + kRingSlots = chunks that may be filled
    std::atomic<bool> abort{false};
};
void bounce_worker(BounceShared &b, int t) {
    for (size_t k = 0; k < b.nchunks; ++k) {
        spin_until([&] { return b.released.load(std::memory_order_acquire) > static_cast<int64_t>(k) || b.abort.load(std::memory_order_relaxed); });
        if (b.abort.load(std::memory_order_relaxed)) return;
        const size_t c0 = k * kChunkBytes, m = std::min(kChunkBytes, b.n - c0);
        // shares on 64-byte boundaries of the slot: whole lines per thread
        const size_t lines = (m + 63) / 64;
        const size_t lo = std::min(m, lines * t / b.nt * 64), hi = std::min(m, lines * (t + 1) / b.nt * 64);
        if (hi > lo) {
            WcStream wc(b.ring[k % kRingSlots] + lo);
            wc.append(b.src + c0 + lo, hi - lo);
            wc.finish();
            copy_fence();
        }
        b.filled[k].fetch_add(1, std::memory_order_release);
    }
}

int stage_copy(bsq_stager *s, void *dst, const void *src, size_t n, bool src_pinned) {
    if (n == 0) return BSQ_OK;
    if (src_pinned) {
        BSQ_CUDA_TRY(cudaMemcpyAsync(dst, src, n, cudaMemcpyHostToDevice, s->copy_stream));
        return BSQ_OK;
    }
    for (int k = 0; k < kRingSlots; ++k)
        if (s->ring[k] == nullptr) {
            BSQ_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&s->ring[k]), kChunkBytes, cudaHostAllocDefault));
            BSQ_CUDA_TRY(cudaEventCreateWithFlags(&s->ring_free[k], cudaEventDisableTiming));
        }
    // slots still being read by the DMA of an earlier call
    for (int k = 0; k < kRingSlots; ++k)
        if (s->ring_used[k]) {
            BSQ_CUDA_TRY(cudaEventSynchronize(s->ring_free[k]));
            s->ring_used[k] = false;
        }
    BounceShared b;
    b.src = static_cast<const uint8_t *>(src);
    b.n = n;
    b.nchunks = (n + kChunkBytes - 1) / kChunkBytes;
    for (int k = 0; k < kRingSlots; ++k) b.ring[k] = s->ring[k];
    b.filled = std::vector<std::atomic<int>>(b.nchunks);
    for (auto &f : b.filled) f.store(0, std::memory_order_relaxed);
    b.released.store(kRingSlots, std::memory_order_relaxed);
    int nt = static_cast<int>(std::min<size_t>(static_cast<size_t>(pool_threads(1 << 20)), std::max<size_t>(1, n >> 19)));  // >= 512 KiB per thread
    b.nt = nt;
    Pool &pool = Pool::get();
    const bool pooled = nt > 1;
    if (pooled) pool.start(nt, [&b](int t) { bounce_worker(b, t); });
    int rc = BSQ_OK;
    for (size_t k = 0; k < b.nchunks && rc == BSQ_OK; ++k) {
        const int slot = static_cast<int>(k % kRingSlots);
        const size_t c0 = k * kChunkBytes, m = std::min(kChunkBytes, n - c0);
        if (pooled) {
            spin_until([&] { return b.filled[k].load(std::memory_order_acquire) == nt; });
        } else {
            if (k >= static_cast<size_t>(kRingSlots) && cudaEventSynchronize(s->ring_free[slot]) != cudaSuccess) {
                rc = fail(BSQ_ERR_CUDA, "bounce copy failed");
                break;
            }
            WcStream wc(s->ring[slot]);
            wc.append(b.src + c0, m);
            wc.finish();
            copy_fence();
        }
        if (rc == BSQ_OK && cudaMemcpyAsync(static_cast<uint8_t *>(dst) + c0, s->ring[slot], m, cudaMemcpyHostToDevice, s->copy_stream) != cudaSuccess)
            rc = fail(BSQ_ERR_CUDA, "cudaMemcpyAsync failed in the bounce ring");
        if (rc == BSQ_OK && cudaEventRecord(s->ring_free[slot], s->copy_stream) != cudaSuccess) rc = fail(BSQ_ERR_CUDA, "cudaEventRecord failed");
        s->ring_used[slot] = true;
        // the slot of chunk k + 1 - kRingSlots ... is free again once ITS copy has completed: release the next chunk
        if (pooled && rc == BSQ_OK && k + 1 >= static_cast<size_t>(kRingSlots) && k + 1 < b.nchunks) {
            const int nslot = static_cast<int>((k + 1) % kRingSlots);
            if (cudaEventSynchronize(s->ring_free[nslot]) != cudaSuccess) rc = fail(BSQ_ERR_CUDA, "bounce copy failed");
            b.released.store(static_cast<int64_t>(k) + 2, std::memory_order_release);
        }
    }
    if (rc) b.abort.store(true);
    if (pooled) pool.wait();
    return rc;
}

struct RunArgs {
    cudaStream_t st;
    const uint8_t *h_bytes;  // indexed by the offsets' own values (h_bytes + offs[i] = sequence i)
    const int64_t *h_offs;
    const uint8_t *h_mask;
    int64_t nseq, padlen, base;
    const bsq_tokenizer *tok;
    int onehot, batch_first, kind;
    void *d_out;
    bool pin_b, pin_m;
};

// Takes the next device slot, reserves its staging buffers for `nbytes` residues and nseq + 1 offsets.
int slot_begin(bsq_stager *s, int64_t nbytes, int64_t nseq, bool with_mask) {
    s->cur = (s->cur + 1) % kDevSlots;
    DevSlot &d = s->slot[s->cur];
    if (d.busy) BSQ_CUDA_TRY(cudaStreamWaitEvent(s->copy_stream, d.done, 0));  // the kernels that read this slot two calls ago
    if (int rc = dev_reserve(s, reinterpret_cast<void **>(&d.d_bytes), &d.cap_bytes, static_cast<size_t>(nbytes) + 32)) return rc;
    if (int rc = dev_reserve(s, reinterpret_cast<void **>(&d.d_offs), &d.cap_offs, sizeof(int64_t) * (nseq + 1))) return rc;
    if (with_mask)
        if (int rc = dev_reserve(s, reinterpret_cast<void **>(&d.d_mask), &d.cap_mask, static_cast<size_t>(nbytes) + 32)) return rc;
    return BSQ_OK;
}

// Reserves the device-side staging buffers of a batch and copies its offsets.
int stage_begin(bsq_stager *s, const RunArgs &a) {
    const int64_t nbytes = a.h_offs[a.nseq] - a.base;
    if (int rc = slot_begin(s, nbytes, a.nseq, a.h_mask != nullptr)) return rc;
    // offsets first (small); the kernels index d_bytes with (offset - base) via a shifted pointer
    return stage_copy(s, s->slot[s->cur].d_offs, a.h_offs, sizeof(int64_t) * (a.nseq + 1),
                      is_pinned_cached(s, a.h_offs, sizeof(int64_t) * (a.nseq + 1)));
}

// End of the staged range that starts at sequence i0: whole 128-sequence groups holding ~kChunkBytes of residues.
int64_t range_end(const int64_t *h_offs, int64_t nseq, int64_t i0, size_t chunk = kChunkBytes) {
    const int64_t want = h_offs[i0] + static_cast<int64_t>(chunk);
    int64_t i1 = std::upper_bound(h_offs + i0, h_offs + nseq + 1, want) - h_offs - 1;
    i1 = std::max(i1, i0 + 1);
    return std::min(nseq, (i1 + kSeqAlign - 1) / kSeqAlign * kSeqAlign);
}

// Copies the residues (and mask) of sequences [i0, i1) and launches their kernel behind the copy.
int stage_range(bsq_stager *s, const RunArgs &a, int64_t i0, int64_t i1, size_t nchunk) {
    DevSlot &d = s->slot[s->cur];
    const int64_t base = a.base;
    const int64_t b0 = a.h_offs[i0] - base, b1 = a.h_offs[i1] - base;
    if (int rc = stage_copy(s, d.d_bytes + b0, a.h_bytes + base + b0, static_cast<size_t>(b1 - b0), a.pin_b)) return rc;
    if (a.h_mask)
        if (int rc = stage_copy(s, d.d_mask + b0, a.h_mask + base + b0, static_cast<size_t>(b1 - b0), a.pin_m)) return rc;
    while (nchunk >= s->events.size()) {
        cudaEvent_t e;
        BSQ_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        s->events.push_back(e);
    }
    BSQ_CUDA_TRY(cudaEventRecord(s->events[nchunk], s->copy_stream));
    BSQ_CUDA_TRY(cudaStreamWaitEvent(a.st, s->events[nchunk], 0));
    const uint8_t *d_bytes_shifted = d.d_bytes - base;
    const uint8_t *d_mask_shifted = a.h_mask ? d.d_mask - base : nullptr;
    const size_t esize = bsq_kind_size(a.kind);
    const int64_t ncols = a.onehot ? a.tok->alphabet_size : 1;
    if (s->aug_chain > 0)
        if (int rc = bsq_augment_blosum62(s->device, a.st, d.d_bytes - base, d.d_offs + i0, i1 - i0, s->aug_chain, s->aug_frac,
                                          s->aug_seed, s->aug_base + i0))
            return rc;
    if (a.onehot)
        return bsq::launch_onehot(a.st, d_bytes_shifted, d.d_offs + i0, d_mask_shifted, i1 - i0, a.nseq, a.padlen, *a.tok, a.kind,
                                  static_cast<uint8_t *>(a.d_out) + static_cast<size_t>(i0) * ncols * esize);
    const size_t off = a.batch_first ? static_cast<size_t>(i0) * a.padlen * esize : static_cast<size_t>(i0) * esize;
    return bsq::launch_tokenize(a.st, d_bytes_shifted, d.d_offs + i0, i1 - i0, a.nseq, a.padlen, *a.tok, a.batch_first, a.kind,
                                static_cast<uint8_t *>(a.d_out) + off, /*first_off=*/a.h_offs[i0]);
}

// Marks the current slot as in use by whatever `st` holds now.  Also called on the error paths: kernels of earlier
// ranges may already be reading the slot.
int stage_end(bsq_stager *s, cudaStream_t st) {
    DevSlot &d = s->slot[s->cur];
    BSQ_CUDA_TRY(cudaEventRecord(d.done, st));
    d.busy = true;
    return BSQ_OK;
}

int staged_run(bsq_stager *s, cudaStream_t st, const uint8_t *h_bytes, const int64_t *h_offs, const uint8_t *h_mask,
               int64_t nseq, int64_t padlen, const bsq_tokenizer *tok, int onehot, int batch_first, int kind, void *d_out) {
    if (s == nullptr) return fail(BSQ_ERR_ARG, "null stager");
    if (int rc = bsq::check_launch_args(s->device, nseq, padlen, tok, kind, d_out)) return rc;
    if (int rc = bsq_check_lengths_host(h_offs, nseq, padlen, tok)) {
        // the reference raises invalid_argument for one-hot (:361) and runtime_error for tokens (:458);
        // both map to BSQ_ERR_TOO_LONG here, the Python shim picks the exception type.
        return rc;
    }
    if (nseq == 0) return BSQ_OK;
    RunArgs a{st, h_bytes, h_offs, h_mask, nseq, padlen, h_offs[0], tok, onehot, batch_first, kind, d_out, false, false};
    const int64_t nbytes = h_offs[nseq] - a.base;
    if (nbytes > 0 && h_bytes == nullptr) return fail(BSQ_ERR_ARG, "null residue buffer");
    a.pin_b = nbytes > 0 && is_pinned_cached(s, h_bytes + a.base, static_cast<size_t>(nbytes));
    a.pin_m = h_mask && nbytes > 0 && is_pinned_cached(s, h_mask + a.base, static_cast<size_t>(nbytes));
    if (int rc = stage_begin(s, a)) return rc;
    // Range size.  The call costs copy time + the kernel of the last range + a few microseconds per copy: small
    // outputs (narrow tokens: the whole batch's kernel is a few % of its copy) do best with few large ranges from a
    // pinned source, expanding outputs (one-hot, wide types) and bounced pageable sources with 4 MiB ones.
    size_t chunk = kChunkBytes;
    if (a.pin_b && !h_mask && !onehot && bsq_kind_size(kind) <= 2) chunk = size_t(32) << 20;  // 35 MB batch, pipelined calls: 4 MiB 0.707 ms, 16 MiB 0.689, 32 MiB 0.674, one range 0.681 (raw copy 0.650)
    size_t nchunk = 0;
    int rc = BSQ_OK;
    for (int64_t i0 = 0; i0 < nseq && rc == BSQ_OK;) {
        const int64_t i1 = range_end(h_offs, nseq, i0, chunk);
        rc = stage_range(s, a, i0, i1, nchunk++);
        i0 = i1;
    }
    const int rc2 = stage_end(s, st);  // also after a failure: earlier ranges' kernels may be reading the slot
    return rc ? rc : rc2;
}

// ------------------------------------------------------------------------------------------------------------------
// Streamed item batches: the reference's unpacked batch (src/tokenize.h:389-419: a Python list of str / bytes /
// bytearray) -> pinned pack -> device -> kernels in ONE pass over the items, range by range.
//
// The items stay with their owner; `resolve(ctx, lo, hi, ptrs, lens)` is called from pool threads and fills pointer
// and length of items [lo, hi) (length -1 = "needs the owner's thread", e.g. a Python str whose UTF-8 form has to be
// created), `fixup(ctx, i, &ptr, &len)` is then called on the calling thread for those.
//
// Per range of R items (a multiple of 128, ~4 MiB of residues going by the previous call's mean length):
//   workers   walk their share of the range (prefetching the item headers ahead), publish its byte sum / maximum,
//             walk their share of the NEXT range, wait for the range's base offsets, then copy exactly the items they
//             walked (their header lines are still in that core's cache) into the pinned pack, writing the offsets as
//             they go, and write the lines back (clwb) for the DMA engine;
//   caller    as soon as a range is walked: fixes up what the workers could not resolve, checks the lengths, turns the
//             byte sums into base offsets; as soon as the previous range is gathered: enqueues its two copies (offsets,
//             residues) on the copy stream and its kernel behind them.
// The DMA of range k overlaps the gather of range k+1 and the walk of range k+2; nothing is walked twice and the
// call returns when the last range has been enqueued.  Two pinned packs alternate call by call (each with the event
// of the last copy that read it), so back-to-back calls do not synchronise with the copy stream.
// ------------------------------------------------------------------------------------------------------------------
struct ItemsShared {
    int nt = 1;
    int64_t n = 0, R = 0, nranges = 0;
    const void **ptrs = nullptr;
    int64_t *lens = nullptr;
    bsq_resolve_fn resolve = nullptr;
    void *ctx = nullptr;
    bsq_pack *pack = nullptr;
    std::vector<int64_t> sum, mx, special, base;  // [range * nt + thread]
    std::vector<std::atomic<int>> walked, gathered, go;  // per range
    std::atomic<bool> abort{false};
    int64_t lo(int64_t k) const { return k * R; }
    int64_t hi(int64_t k) const { return std::min(n, (k + 1) * R); }
    // thread t's share of range k: items [cut(k, t), cut(k, t + 1))
    int64_t cut(int64_t k, int t) const { return lo(k) + (hi(k) - lo(k)) * t / nt; }
};

void items_walk(ItemsShared &sh, int64_t k, int t) {
    const int64_t a = sh.cut(k, t), b = sh.cut(k, t + 1);
    if (b > a) sh.resolve(sh.ctx, a, b, sh.ptrs, sh.lens);
    int64_t sum = 0, mx = 0, special = 0;
    for (int64_t i = a; i < b; ++i) {
        const int64_t l = sh.lens[i];
        if (l < 0) ++special;
        else { sum += l; mx = std::max(mx, l); }
    }
    const size_t j = static_cast<size_t>(k) * sh.nt + t;
    sh.sum[j] = sum; sh.mx[j] = mx; sh.special[j] = special;
    sh.walked[static_cast<size_t>(k)].fetch_add(1, std::memory_order_release);
}

void items_gather(ItemsShared &sh, int64_t k, int t) {
    const int64_t a = sh.cut(k, t), b = sh.cut(k, t + 1);
    uint8_t *bytes = sh.pack->bytes;
    int64_t *offs = sh.pack->offs;
    int64_t pos = sh.base[static_cast<size_t>(k) * sh.nt + t];
    // the items are separate heap objects: every one starts with a miss that the hardware prefetcher cannot
    // anticipate, so the bodies are requested a few items ahead
    constexpr int64_t kAhead = 4;
    auto prefetch_body = [&](int64_t j) {
        const char *p = static_cast<const char *>(sh.ptrs[j]);
        const int64_t l = std::min<int64_t>(sh.lens[j], 2048);
        for (int64_t o = 0; o < l; o += 64) __builtin_prefetch(p + o, 0, 0);
    };
    for (int64_t j = a; j < std::min(b, a + kAhead); ++j) prefetch_body(j);
    // leading partial line of this run (shared with the previous thread's run): ordinary stores + write-back
    int64_t i = a;
    int64_t head_left = (64 - (reinterpret_cast<uintptr_t>(bytes + pos) & 63)) & 63;  // bytes until the first line boundary
    const uint8_t *carry_p = nullptr;  // rest of the item that straddles the boundary
    int64_t carry_n = 0;
    uint8_t *head_at = bytes + pos;
    const int64_t head_total = head_left;
    for (; i < b && head_left > 0; ++i) {
        if (i != sh.lo(k)) offs[i] = pos;  // (the range's first offset was written by the caller)
        const int64_t l = sh.lens[i];
        const int64_t m = std::min(l, head_left);
        if (m > 0) std::memcpy(bytes + pos, sh.ptrs[i], static_cast<size_t>(m));
        pos += l;
        head_left -= m;
        if (m < l) {
            carry_p = static_cast<const uint8_t *>(sh.ptrs[i]) + m;
            carry_n = l - m;
        }
    }
    if (head_total > head_left) writeback_lines(head_at, static_cast<size_t>(head_total - head_left));
    if (head_left == 0) {
        WcStream wc(bytes + (pos - carry_n));  // line-aligned by construction
        if (carry_n > 0) wc.append(carry_p, static_cast<size_t>(carry_n));
        for (; i < b; ++i) {
            if (i + kAhead < b) prefetch_body(i + kAhead);
            if (i != sh.lo(k)) offs[i] = pos;
            const int64_t l = sh.lens[i];
            if (l > 0) wc.append(static_cast<const uint8_t *>(sh.ptrs[i]), static_cast<size_t>(l));
            pos += l;
        }
        wc.finish();
    }
    writeback_lines(reinterpret_cast<const uint8_t *>(offs + a), static_cast<size_t>(b - a) * sizeof(int64_t));
    copy_fence();
    sh.gathered[static_cast<size_t>(k)].fetch_add(1, std::memory_order_release);
}

void items_worker(ItemsShared &sh, int t) {
    items_walk(sh, 0, t);
    for (int64_t k = 0; k < sh.nranges; ++k) {
        if (k + 1 < sh.nranges) items_walk(sh, k + 1, t);
        spin_until([&] { return sh.go[static_cast<size_t>(k)].load(std::memory_order_acquire) != 0 || sh.abort.load(std::memory_order_relaxed); });
        if (sh.abort.load(std::memory_order_relaxed)) return;
        items_gather(sh, k, t);
    }
}

int pack_event(bsq_stager *s, int k) {
    if (s->ipack_ev[k] == nullptr) BSQ_CUDA_TRY(cudaEventCreateWithFlags(&s->ipack_ev[k], cudaEventDisableTiming));
    return BSQ_OK;
}

int items_stream_run(bsq_stager *s, cudaStream_t st, int64_t n, bsq_resolve_fn resolve, bsq_fixup_fn fixup, void *ctx, int64_t padlen,
                     const bsq_tokenizer *tok, int onehot, int batch_first, int kind, void *d_out, int nthreads) {
    if (s == nullptr) return fail(BSQ_ERR_ARG, "null stager");
    if (n < 0 || (n > 0 && resolve == nullptr)) return fail(BSQ_ERR_ARG, "bad item arguments");
    if (int rc = bsq::check_launch_args(s->device, n, padlen, tok, kind, d_out)) return rc;
    if (n == 0) return BSQ_OK;
    const int64_t extra = (tok->bos_id >= 0) + (tok->eos_id >= 0);

    // the pack this call gathers into: wait for the last copy that read it (two calls ago: long done in steady state)
    const int pk = s->ipack_next;
    s->ipack_next ^= 1;
    bsq_pack *pack = &s->ipack[pk];
    pack->pinned = 1;
    if (int rc = pack_event(s, pk)) return rc;
    if (s->ipack_used[pk]) BSQ_CUDA_TRY(cudaEventSynchronize(s->ipack_ev[pk]));

    ItemsShared sh;
    sh.n = n;
    const int64_t want_items = std::max<int64_t>(1, static_cast<int64_t>(kChunkBytes) / std::max<int64_t>(s->avg_len_hint, 1));
    sh.R = std::max<int64_t>(kSeqAlign, std::min<int64_t>(int64_t(1) << 20, (want_items + kSeqAlign - 1) / kSeqAlign * kSeqAlign));
    sh.nranges = (n + sh.R - 1) / sh.R;
    int nt = pool_threads(nthreads);
    nt = static_cast<int>(std::min<int64_t>(nt, std::max<int64_t>(1, std::min(n, sh.R) / 256)));  // >= 256 items per share
    sh.nt = nt;
    s->it_ptrs.resize(static_cast<size_t>(n));
    s->it_lens.resize(static_cast<size_t>(n));
    sh.ptrs = s->it_ptrs.data();
    sh.lens = s->it_lens.data();
    sh.resolve = resolve;
    sh.ctx = ctx;
    sh.pack = pack;
    const size_t cells = static_cast<size_t>(sh.nranges) * nt;
    sh.sum.assign(cells, 0); sh.mx.assign(cells, 0); sh.special.assign(cells, 0); sh.base.assign(cells, 0);
    sh.walked = std::vector<std::atomic<int>>(static_cast<size_t>(sh.nranges));
    sh.gathered = std::vector<std::atomic<int>>(static_cast<size_t>(sh.nranges));
    sh.go = std::vector<std::atomic<int>>(static_cast<size_t>(sh.nranges));
    for (int64_t k = 0; k < sh.nranges; ++k) { sh.walked[k].store(0); sh.gathered[k].store(0); sh.go[k].store(0); }

    if (int rc = pack_reserve(pack, 0, n)) return rc;  // offsets: n + 1 entries, known up front
    if (int rc = slot_begin(s, static_cast<int64_t>(pack->cap_bytes), n, false)) return rc;  // device buffers follow the pack's capacity
    RunArgs a{st, pack->bytes, pack->offs, nullptr, n, padlen, 0, tok, onehot, batch_first, kind, d_out, true, false};

    Pool &pool = Pool::get();
    const bool pooled = nt > 1;
    if (pooled) pool.start(nt, [&sh](int t) { items_worker(sh, t); });

    int rc = BSQ_OK;
    int64_t running = 0, issued = 0;  // bytes placed so far; ranges enqueued so far
    auto issue = [&](int64_t k) -> int {  // copies + kernel of range k (gathered)
        DevSlot &d = s->slot[s->cur];
        const int64_t i0 = sh.lo(k), i1 = sh.hi(k);
        BSQ_CUDA_TRY(cudaMemcpyAsync(d.d_offs + i0, pack->offs + i0, sizeof(int64_t) * static_cast<size_t>(i1 - i0 + 1), cudaMemcpyHostToDevice,
                                     s->copy_stream));
        a.h_bytes = pack->bytes;
        return stage_range(s, a, i0, i1, static_cast<size_t>(k));
    };
    auto wait_gathered = [&](int64_t k) {
        if (pooled) spin_until([&] { return sh.gathered[static_cast<size_t>(k)].load(std::memory_order_acquire) == nt; });
    };
    for (int64_t k = 0; k < sh.nranges && rc == BSQ_OK; ++k) {
        if (pooled) spin_until([&] { return sh.walked[static_cast<size_t>(k)].load(std::memory_order_acquire) == nt; });
        else items_walk(sh, k, 0);
        // items the workers could not resolve (Python str) or that are of no accepted type
        int64_t special = 0;
        for (int t = 0; t < nt; ++t) special += sh.special[static_cast<size_t>(k) * nt + t];
        if (special > 0) {
            for (int t = 0; t < nt && rc == BSQ_OK; ++t) {
                const size_t j = static_cast<size_t>(k) * nt + t;
                if (sh.special[j] == 0) continue;
                int64_t sum = 0, mx = 0;
                for (int64_t i = sh.cut(k, t); i < sh.cut(k, t + 1); ++i) {
                    if (sh.lens[i] < 0 && (fixup == nullptr || fixup(ctx, i, &sh.ptrs[i], &sh.lens[i]) != 0 || sh.lens[i] < 0)) {
                        rc = fail(BSQ_ERR_ARG, "item was none of string, bytes, or numpy array of 8-bit integers. ");  // src/tokenize.h:412
                        break;
                    }
                    sum += sh.lens[i];
                    mx = std::max(mx, sh.lens[i]);
                }
                sh.sum[j] = sum; sh.mx[j] = mx;
            }
            if (rc) break;
        }
        int64_t total_k = 0, mx = 0;
        for (int t = 0; t < nt; ++t) {
            const size_t j = static_cast<size_t>(k) * nt + t;
            sh.base[j] = running + total_k;
            total_k += sh.sum[j];
            mx = std::max(mx, sh.mx[j]);
        }
        if (mx + extra > padlen) {  // src/tokenize.h:456-459
            rc = fail(BSQ_ERR_TOO_LONG, "seq len + bos + eos > padlen: " + std::to_string(mx + extra) + ", vs padlen " + std::to_string(padlen));
            break;
        }
        // capacity: the pinned pack and the device slot grow together (rare after the first calls: both keep their size)
        if (static_cast<size_t>(running + total_k) + 32 > pack->cap_bytes) {
            // everything gathered so far has to leave the old buffers first
            while (issued < k && rc == BSQ_OK) { wait_gathered(issued); rc = issue(issued++); }
            if (rc) break;
            BSQ_CUDA_TRY(cudaStreamSynchronize(s->copy_stream));
            const int64_t seen = sh.hi(k);
            const int64_t est = static_cast<int64_t>(static_cast<double>(running + total_k) * static_cast<double>(n) / static_cast<double>(seen) * 1.15) + 4096;
            if ((rc = pack_reserve(pack, est, n)) != BSQ_OK) break;  // (offsets keep their buffer: capacity n + 1 already)
            DevSlot &d = s->slot[s->cur];
            // (kernels of this call's earlier ranges, on `stream`, may still read the old device buffer)
            if ((rc = dev_reserve(s, reinterpret_cast<void **>(&d.d_bytes), &d.cap_bytes, pack->cap_bytes, st, true)) != BSQ_OK) break;
        }
        pack->offs[sh.lo(k)] = running;
        running += total_k;
        pack->offs[sh.hi(k)] = running;
        if (pooled) sh.go[static_cast<size_t>(k)].store(1, std::memory_order_release);
        else items_gather(sh, k, 0);
        // enqueue whatever is gathered by now, but never wait for the range that was only just released
        while (issued < k && rc == BSQ_OK) { wait_gathered(issued); rc = issue(issued++); }
    }
    while (issued < sh.nranges && rc == BSQ_OK) { wait_gathered(issued); rc = issue(issued++); }
    if (rc) {
        sh.abort.store(true);
        for (auto &g : sh.go) g.store(1, std::memory_order_release);
    }
    if (pooled) pool.wait();  // also on error: the workers borrow this frame
    pack->nseq = n;
    pack->nbytes = running;
    if (rc == BSQ_OK && n > 0) s->avg_len_hint = std::max<int64_t>(1, running / n);
    // the pack is free again when the copies enqueued so far have been made
    if (cudaEventRecord(s->ipack_ev[pk], s->copy_stream) == cudaSuccess) s->ipack_used[pk] = true;
    const int rc2 = stage_end(s, st);
    return rc ? rc : rc2;
}

// Items given as pointer / length arrays (already walked): the streamed pipeline with a resolver that copies from them.
struct ArrayItems {
    const void *const *ptrs;
    const int64_t *lens;
};
void array_resolve(void *ctx, int64_t lo, int64_t hi, const void **ptrs, int64_t *lens) {
    const ArrayItems &it = *static_cast<const ArrayItems *>(ctx);
    for (int64_t i = lo; i < hi; ++i) {
        ptrs[i] = it.ptrs[i];
        lens[i] = it.lens[i];
    }
}
int items_run(bsq_stager *s, bsq_pack * /*unused: the stager owns the pinned packs*/, cudaStream_t st, const void *const *ptrs, const int64_t *lens,
              int64_t n, int64_t padlen, const bsq_tokenizer *tok, int onehot, int batch_first, int kind, void *d_out, int nthreads) {
    if (n < 0 || (n > 0 && (ptrs == nullptr || lens == nullptr))) return fail(BSQ_ERR_ARG, "bad pack arguments");
    for (int64_t i = 0; i < n; ++i)
        if (lens[i] < 0) return fail(BSQ_ERR_ARG, "negative sequence length");
    ArrayItems it{ptrs, lens};
    return items_stream_run(s, st, n, array_resolve, nullptr, &it, padlen, tok, onehot, batch_first, kind, d_out, nthreads);
}

// Rows of a device byte buffer -> separate host destinations (the bodies of the Python strings that
// decode_tokens returns): device -> pinned ring in ~8 MiB stages on `st`, host threads scatter stage k
// while stage k+1 is in flight.  Returns when every row has arrived.
int fetch_rows(bsq_stager *s, cudaStream_t st, const uint8_t *d_chars, const int64_t *h_offs, int64_t rows, void *const *dst,
               int nthreads) {
    if (s == nullptr) return fail(BSQ_ERR_ARG, "null stager");
    if (rows < 0 || (rows > 0 && (h_offs == nullptr || dst == nullptr))) return fail(BSQ_ERR_ARG, "bad fetch arguments");
    if (rows == 0) return BSQ_OK;
    BSQ_CUDA_TRY(cudaSetDevice(s->device));
    const int64_t base = h_offs[0], total = h_offs[rows] - base;
    if (total < 0) return fail(BSQ_ERR_ARG, "offsets must be non-decreasing");
    if (total == 0) return BSQ_OK;
    if (d_chars == nullptr) return fail(BSQ_ERR_ARG, "null character buffer");
    for (int k = 0; k < kRingSlots; ++k)
        if (s->fetch_ring[k] == nullptr) {
            BSQ_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&s->fetch_ring[k]), kFetchBytes, cudaHostAllocDefault));
            BSQ_CUDA_TRY(cudaEventCreateWithFlags(&s->fetch_ev[k], cudaEventDisableTiming));
        }
    const int64_t S = static_cast<int64_t>(kFetchBytes);
    const int64_t nstages = (total + S - 1) / S;
    int nt = pool_threads(nthreads);
    nt = static_cast<int>(std::min<int64_t>(nt, std::max<int64_t>(1, total >> 19)));

    // bytes [lo, hi) of the character stream (relative to base), now in `src` (src[0] = byte stage_lo), go to their rows
    auto scatter = [&](const uint8_t *src, int64_t stage_lo, int64_t lo, int64_t hi) {
        if (lo >= hi) return;
        int64_t r = std::upper_bound(h_offs, h_offs + rows + 1, base + lo) - h_offs - 1;  // row holding byte lo
        for (; r < rows && h_offs[r] - base < hi; ++r) {
            const int64_t r0 = h_offs[r] - base, r1 = h_offs[r + 1] - base;
            const int64_t c0 = std::max(r0, lo), c1 = std::min(r1, hi);
            if (c1 > c0) std::memcpy(static_cast<uint8_t *>(dst[r]) + (c0 - r0), src + (c0 - stage_lo), static_cast<size_t>(c1 - c0));
        }
    };
    auto issue = [&](int64_t k) -> int {
        const int64_t lo = k * S, m = std::min(S, total - lo);
        BSQ_CUDA_TRY(cudaMemcpyAsync(s->fetch_ring[k % kRingSlots], d_chars + base + lo, static_cast<size_t>(m), cudaMemcpyDeviceToHost, st));
        BSQ_CUDA_TRY(cudaEventRecord(s->fetch_ev[k % kRingSlots], st));
        return BSQ_OK;
    };
    if (nt <= 1) {
        for (int64_t k = 0; k < std::min<int64_t>(nstages, kRingSlots); ++k)
            if (int rc = issue(k)) return rc;
        for (int64_t k = 0; k < nstages; ++k) {
            BSQ_CUDA_TRY(cudaEventSynchronize(s->fetch_ev[k % kRingSlots]));
            scatter(s->fetch_ring[k % kRingSlots], k * S, k * S, std::min(total, (k + 1) * S));
            if (k + kRingSlots < nstages)
                if (int rc = issue(k + kRingSlots)) return rc;
        }
        return BSQ_OK;
    }
    std::atomic<int64_t> ready{0};
    std::atomic<bool> abort{false};
    std::vector<std::atomic<int>> done(static_cast<size_t>(nstages));
    for (auto &d : done) d.store(0, std::memory_order_relaxed);
    Pool &pool = Pool::get();
    pool.start(nt, [&, nt](int t) {
        for (int64_t k = 0; k < nstages; ++k) {
            spin_until([&] { return ready.load(std::memory_order_acquire) > k || abort.load(std::memory_order_relaxed); });
            if (abort.load(std::memory_order_relaxed)) return;
            const int64_t lo = k * S, m = std::min(S, total - lo);
            scatter(s->fetch_ring[k % kRingSlots], lo, lo + m * t / nt, lo + m * (t + 1) / nt);
            done[static_cast<size_t>(k)].fetch_add(1, std::memory_order_release);
        }
    });
    int rc = BSQ_OK;
    for (int64_t k = 0; k < std::min<int64_t>(nstages, kRingSlots) && rc == BSQ_OK; ++k) rc = issue(k);
    for (int64_t k = 0; k < nstages && rc == BSQ_OK; ++k) {
        if (cudaEventSynchronize(s->fetch_ev[k % kRingSlots]) != cudaSuccess) {
            rc = fail(BSQ_ERR_CUDA, "bsq_fetch_rows: device -> host copy failed");
            break;
        }
        ready.store(k + 1, std::memory_order_release);
        if (k + kRingSlots < nstages) {  // slot k is needed again: wait until it has been scattered
            spin_until([&] { return done[static_cast<size_t>(k)].load(std::memory_order_acquire) == nt; });
            rc = issue(k + kRingSlots);
        }
    }
    if (rc) abort.store(true);
    pool.wait();
    return rc;
}

}  // namespace

extern "C" {

int bsq_stager_create(bsq_stager **out, int device) {
    bsq::DeviceRestore restore_device;
    if (out == nullptr) return fail(BSQ_ERR_ARG, "null argument");
    BSQ_CUDA_TRY(cudaSetDevice(device));
    bsq_stager *s = new bsq_stager();
    s->device = device;
    cudaError_t e = cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking);
    for (int k = 0; k < kDevSlots && e == cudaSuccess; ++k) e = cudaEventCreateWithFlags(&s->slot[k].done, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        delete s;
        return fail(BSQ_ERR_CUDA, std::string("bsq_stager_create: ") + cudaGetErrorString(e));
    }
    *out = s;
    return BSQ_OK;
}

void bsq_stager_destroy(bsq_stager *s) {
    bsq::DeviceRestore restore_device;
    if (s == nullptr) return;
    cudaSetDevice(s->device);
    cudaDeviceSynchronize();
    for (int k = 0; k < kDevSlots; ++k) {
        cudaFree(s->slot[k].d_bytes);
        cudaFree(s->slot[k].d_mask);
        cudaFree(s->slot[k].d_offs);
        if (s->slot[k].done) cudaEventDestroy(s->slot[k].done);
    }
    for (int k = 0; k < 2; ++k) {
        host_free(s->ipack[k].bytes, 1);
        host_free(s->ipack[k].offs, 1);
        if (s->ipack_ev[k]) cudaEventDestroy(s->ipack_ev[k]);
    }
    for (int k = 0; k < kRingSlots; ++k) {
        if (s->ring[k]) cudaFreeHost(s->ring[k]);
        if (s->ring_free[k]) cudaEventDestroy(s->ring_free[k]);
    }
    for (cudaEvent_t e : s->events) cudaEventDestroy(e);
    if (s->grow_ev) cudaEventDestroy(s->grow_ev);
    for (int k = 0; k < kRingSlots; ++k) {
        if (s->fetch_ring[k]) cudaFreeHost(s->fetch_ring[k]);
        if (s->fetch_ev[k]) cudaEventDestroy(s->fetch_ev[k]);
    }
    if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
    delete s;
}

int bsq_stager_sync_copies(bsq_stager *s) {
    if (s == nullptr) return fail(BSQ_ERR_ARG, "null stager");
    BSQ_CUDA_TRY(cudaStreamSynchronize(s->copy_stream));
    return BSQ_OK;
}

int bsq_stager_set_augment(bsq_stager *s, int chain_len, double augment_frac, uint64_t seed, int64_t seq_index_base) {
    if (s == nullptr) return fail(BSQ_ERR_ARG, "null stager");
    if (chain_len < 0 || !(augment_frac >= 0.0)) return fail(BSQ_ERR_ARG, "bad augmentation parameters");
    s->aug_chain = chain_len;
    s->aug_frac = augment_frac;
    s->aug_seed = seed;
    s->aug_base = seq_index_base;
    return BSQ_OK;
}

int bsq_stage_host(bsq_stager *s, void *stream, const uint8_t *h_bytes, const int64_t *h_offsets, int64_t nseq,
                   const uint8_t **d_bytes, const int64_t **d_offsets) {
    bsq::DeviceRestore restore_device;
    if (s == nullptr || d_bytes == nullptr || d_offsets == nullptr) return fail(BSQ_ERR_ARG, "null argument");
    if (nseq < 0 || h_offsets == nullptr) return fail(BSQ_ERR_ARG, "bad offsets");
    BSQ_CUDA_TRY(cudaSetDevice(s->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t base = h_offsets[0], nbytes = h_offsets[nseq] - base;
    if (nbytes < 0) return fail(BSQ_ERR_ARG, "offsets must be non-decreasing");
    if (nbytes > 0 && h_bytes == nullptr) return fail(BSQ_ERR_ARG, "null residue buffer");
    if (int rc = slot_begin(s, nbytes, nseq, false)) return rc;
    DevSlot &d = s->slot[s->cur];
    if (int rc = stage_copy(s, d.d_offs, h_offsets, sizeof(int64_t) * (nseq + 1), is_pinned_cached(s, h_offsets, sizeof(int64_t) * (nseq + 1)))) return rc;
    if (int rc = stage_copy(s, d.d_bytes, h_bytes + base, static_cast<size_t>(nbytes),
                            nbytes > 0 && is_pinned_cached(s, h_bytes + base, static_cast<size_t>(nbytes))))
        return rc;
    if (s->events.empty()) {
        cudaEvent_t e;
        BSQ_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        s->events.push_back(e);
    }
    BSQ_CUDA_TRY(cudaEventRecord(s->events[0], s->copy_stream));
    BSQ_CUDA_TRY(cudaStreamWaitEvent(st, s->events[0], 0));
    if (s->aug_chain > 0 && nseq > 0)
        if (int rc = bsq_augment_blosum62(s->device, st, d.d_bytes - base, d.d_offs, nseq, s->aug_chain, s->aug_frac, s->aug_seed,
                                          s->aug_base))
            return rc;
    // until bsq_stage_release the buffers count as in use by `stream`
    if (int rc = stage_end(s, st)) return rc;
    *d_bytes = d.d_bytes - base;
    *d_offsets = d.d_offs;
    return BSQ_OK;
}

int bsq_stage_release(bsq_stager *s, void *stream) {
    bsq::DeviceRestore restore_device;
    if (s == nullptr) return fail(BSQ_ERR_ARG, "null stager");
    BSQ_CUDA_TRY(cudaSetDevice(s->device));
    return stage_end(s, static_cast<cudaStream_t>(stream));
}

int bsq_tokenize_host(bsq_stager *s, void *stream, const uint8_t *h_bytes, const int64_t *h_offsets, int64_t nseq,
                      int64_t padlen, const bsq_tokenizer *tok, int batch_first, int kind, void *d_out) {
    bsq::DeviceRestore restore_device;
    return staged_run(s, static_cast<cudaStream_t>(stream), h_bytes, h_offsets, nullptr, nseq, padlen, tok, 0, batch_first,
                      kind, d_out);
}

int bsq_onehot_host(bsq_stager *s, void *stream, const uint8_t *h_bytes, const int64_t *h_offsets, const uint8_t *h_mask,
                    int64_t nseq, int64_t padlen, const bsq_tokenizer *tok, int kind, void *d_out) {
    bsq::DeviceRestore restore_device;
    return staged_run(s, static_cast<cudaStream_t>(stream), h_bytes, h_offsets, h_mask, nseq, padlen, tok, 1, 0, kind, d_out);
}

int bsq_tokenize_items(bsq_stager *s, bsq_pack *p, void *stream, const void *const *ptrs, const int64_t *lens, int64_t n,
                       int64_t padlen, const bsq_tokenizer *tok, int batch_first, int kind, void *d_out, int nthreads) {
    bsq::DeviceRestore restore_device;
    return items_run(s, p, static_cast<cudaStream_t>(stream), ptrs, lens, n, padlen, tok, 0, batch_first, kind, d_out, nthreads);
}

int bsq_onehot_items(bsq_stager *s, bsq_pack *p, void *stream, const void *const *ptrs, const int64_t *lens, int64_t n,
                     int64_t padlen, const bsq_tokenizer *tok, int kind, void *d_out, int nthreads) {
    bsq::DeviceRestore restore_device;
    return items_run(s, p, static_cast<cudaStream_t>(stream), ptrs, lens, n, padlen, tok, 1, 0, kind, d_out, nthreads);
}

int bsq_tokenize_stream_items(bsq_stager *s, void *stream, int64_t n, bsq_resolve_fn resolve, bsq_fixup_fn fixup, void *ctx,
                              int64_t padlen, const bsq_tokenizer *tok, int batch_first, int kind, void *d_out, int nthreads) {
    bsq::DeviceRestore restore_device;
    return items_stream_run(s, static_cast<cudaStream_t>(stream), n, resolve, fixup, ctx, padlen, tok, 0, batch_first, kind, d_out, nthreads);
}

int bsq_onehot_stream_items(bsq_stager *s, void *stream, int64_t n, bsq_resolve_fn resolve, bsq_fixup_fn fixup, void *ctx,
                            int64_t padlen, const bsq_tokenizer *tok, int kind, void *d_out, int nthreads) {
    bsq::DeviceRestore restore_device;
    return items_stream_run(s, static_cast<cudaStream_t>(stream), n, resolve, fixup, ctx, padlen, tok, 1, 0, kind, d_out, nthreads);
}

int bsq_shard_bounds(const int64_t *h_offsets, int64_t nseq, int nshards, int64_t *bounds) {
    if (nseq < 0 || nshards <= 0 || bounds == nullptr || (nseq > 0 && h_offsets == nullptr)) return fail(BSQ_ERR_ARG, "bad shard arguments");
    bounds[0] = 0;
    bounds[nshards] = nseq;
    if (nseq == 0) {
        for (int g = 1; g < nshards; ++g) bounds[g] = 0;
        return BSQ_OK;
    }
    const int64_t base = h_offsets[0], total = h_offsets[nseq] - base;
    for (int g = 1; g < nshards; ++g) {
        // first sequence whose start is at or beyond g/nshards of the residues (ties and empty batches: by count)
        int64_t i = total > 0 ? static_cast<int64_t>(std::lower_bound(h_offsets, h_offsets + nseq, base + static_cast<int64_t>((static_cast<__int128>(total) * g) / nshards)) - h_offsets)
                              : nseq * g / nshards;
        bounds[g] = std::max(bounds[g - 1], std::min(i, nseq));
    }
    return BSQ_OK;
}

int bsq_tokenize_host_sharded(bsq_stager *const *stagers, void *const *streams, int ndev, const uint8_t *h_bytes, const int64_t *h_offsets,
                              int64_t nseq, int64_t padlen, const bsq_tokenizer *tok, int onehot, int batch_first, int kind,
                              void *const *d_outs, const int64_t *bounds) {
    bsq::DeviceRestore restore_device;
    if (stagers == nullptr || streams == nullptr || d_outs == nullptr || bounds == nullptr || ndev <= 0) return fail(BSQ_ERR_ARG, "bad shard arguments");
    if (int rc = bsq_check_lengths_host(h_offsets, nseq, padlen, tok)) return rc;
    std::vector<int> rcs(static_cast<size_t>(ndev), BSQ_OK);
    std::vector<std::string> msgs(static_cast<size_t>(ndev));
    auto run = [&](int g) {
        const int64_t i0 = bounds[g], i1 = bounds[g + 1];
        if (i1 <= i0) return;
        rcs[g] = staged_run(stagers[g], static_cast<cudaStream_t>(streams[g]), h_bytes, h_offsets + i0, nullptr, i1 - i0, padlen, tok, onehot,
                            batch_first, kind, d_outs[g]);
        if (rcs[g] != BSQ_OK) msgs[g] = bsq_last_error();
    };
    if (ndev == 1 || t_in_pool_worker) {
        for (int g = 0; g < ndev; ++g) run(g);
    } else {
        // one host thread per device (each keeps its own current device and enqueues its shard's copies and kernels)
        Pool &pool = Pool::get();
        pool.start(ndev, run);
        pool.wait();
    }
    for (int g = 0; g < ndev; ++g)
        if (rcs[g] != BSQ_OK) return fail(rcs[g], msgs[g]);
    return BSQ_OK;
}

int bsq_memcpy_d2d(int device, void *stream, void *d_dst, const void *d_src, size_t nbytes) {
    bsq::DeviceRestore restore_device;
    BSQ_CUDA_TRY(cudaSetDevice(device));
    BSQ_CUDA_TRY(cudaMemcpyAsync(d_dst, d_src, nbytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
    return BSQ_OK;
}

int bsq_parallel_for(int nthreads, void (*fn)(int, int, void *), void *ctx) {
    if (fn == nullptr) return fail(BSQ_ERR_ARG, "null function");
    const int nt = pool_threads(nthreads);
    if (nt == 1) {
        fn(0, 1, ctx);
        return BSQ_OK;
    }
    Pool &pool = Pool::get();
    pool.start(nt, [fn, nt, ctx](int t) { fn(t, nt, ctx); });
    pool.wait();
    return BSQ_OK;
}

int bsq_fetch_rows(bsq_stager *s, void *stream, const uint8_t *d_chars, const int64_t *h_offsets, int64_t rows, void *const *dst,
                   int nthreads) {
    bsq::DeviceRestore restore_device;
    return fetch_rows(s, static_cast<cudaStream_t>(stream), d_chars, h_offsets, rows, dst, nthreads);
}

}  // extern "C"
