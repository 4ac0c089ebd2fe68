// Internal helpers shared by the translation units of libbsq.so (not installed).
#pragma once
#include <cstdint>
#include <string>

#include "../../include/bsq.h"

namespace bsq {

// Records `msg` as the calling thread's last error and returns `code`.
int fail(int code, const std::string &msg);
// Kernel-launch bookkeeping for bsq_launch_count().
void count_launch(int n = 1);


#ifdef __CUDACC__
// Launchers shared by the device entry points and the host-staged pipeline.  `nseq`
// sequences starting at d_offs[0] are processed; `ld` is the batch extent of the whole
// output array and d_out points at this range's first row (batch-first) / column.  first_off is
// d_offs[0] when the host knows it (-1 otherwise): it lets the TMA-fed kernel anchor its tensor map
// at the range's first residue so that coordinates stay small for sub-ranges of huge buffers.
int launch_tokenize(cudaStream_t st, const uint8_t *d_bytes, const int64_t *d_offs, int64_t nseq, int64_t ld,
                    int64_t padlen, const bsq_tokenizer &tok, int batch_first, int kind, void *d_out, int64_t first_off);
int launch_onehot(cudaStream_t st, const uint8_t *d_bytes, const int64_t *d_offs, const uint8_t *d_mask, int64_t nseq,
                  int64_t ld, int64_t padlen, const bsq_tokenizer &tok, int kind, void *d_out);
int check_launch_args(int device, int64_t nseq, int64_t padlen, const bsq_tokenizer *tok, int kind, const void *d_out);
// A few bytes of device workspace for an entry point that synchronises before it returns, from a library-owned
// stream-ordered pool of `device` (bsq_kernels.cu); free it with cudaFreeAsync on st.
int scratch_alloc(int device, void **p, size_t bytes, cudaStream_t st);
#endif

}  // namespace bsq

#ifdef __CUDACC__
namespace bsq {
// Entry points take their device explicitly and switch to it; the caller's current device is put back on return
// (a host that drives several devices from one thread -- torch does -- must not find it changed behind its back).
struct DeviceRestore {
    int prev = -1;
    DeviceRestore() {
        if (cudaGetDevice(&prev) != cudaSuccess) {
            cudaGetLastError();
            prev = -1;
        }
    }
    ~DeviceRestore() {
        int now = -1;
        if (prev >= 0 && cudaGetDevice(&now) == cudaSuccess && now != prev) cudaSetDevice(prev);
    }
    DeviceRestore(const DeviceRestore &) = delete;
    DeviceRestore &operator=(const DeviceRestore &) = delete;
};
}  // namespace bsq
#endif

#define BSQ_CUDA_TRY(expr)                                                                       \
    do {                                                                                         \
        cudaError_t err__ = (expr);                                                              \
        if (err__ != cudaSuccess)                                                                \
            return bsq::fail(BSQ_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(err__)); \
    } while (0)
