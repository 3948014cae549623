// Host toolkit of the C ABI (include/vgsim_b200.h), shared by every file that implements an entry point: error
// reporting, checked CUDA calls and device buffers owned by a handle or by a single call.  An entry point that fails
// sets the message vgsim_last_error() returns and returns non-zero.
#pragma once
#include <cuda_runtime.h>
#include <algorithm>
#include <string>
#include "handle.h"

struct vgsim_handle_s : public vg::Handle {};

namespace vg {

// Sets the calling thread's vgsim_last_error() message (the string lives in capi.cu); returns 1.
int fail(const std::string &m);

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) return vg::fail(std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)
#define HOST_SYNC(h)                                                    \
    do {                                                                \
        if (!(h)->async_host) CK(cudaStreamSynchronize((h)->stream));   \
    } while (0)

inline int check_replicate(const Handle *h, int r) { return r < 0 || r >= h->R ? fail("replicate out of range") : 0; }

// Device buffer of n (at least one) zero-filled elements, owned by the handle until dfree or vgsim_destroy.
template <class T>
int dalloc(Handle *h, T **p, size_t n) {
    void *q = nullptr;
    if (n == 0) n = 1;
    cudaError_t e = cudaMalloc(&q, n * sizeof(T));
    if (e != cudaSuccess) return fail(std::string("cudaMalloc: ") + cudaGetErrorString(e));
    h->allocs.push_back(q);
    *p = (T *)q;
    e = cudaMemsetAsync(q, 0, n * sizeof(T), h->stream);
    if (e != cudaSuccess) return fail(std::string("cudaMemset: ") + cudaGetErrorString(e));
    return 0;
}
inline void dfree(Handle *h, void *p) {  // best-effort, like vgsim_destroy
    if (!p) return;
    auto it = std::find(h->allocs.begin(), h->allocs.end(), p);
    if (it != h->allocs.end()) h->allocs.erase(it);
    cudaFree(p);
}

// Device temporaries of one call (not zero-filled): freed when the buffer goes out of scope, on every return path.
template <class T>
struct Scratch {
    T *p = nullptr;
    Scratch() = default;
    Scratch(const Scratch &) = delete;
    Scratch &operator=(const Scratch &) = delete;
    ~Scratch() {
        if (p) cudaFree(p);  // best-effort, like dfree
    }
    int alloc(size_t n) {
        void *q = nullptr;
        cudaError_t e = cudaMalloc(&q, std::max<size_t>(n, 1) * sizeof(T));
        if (e != cudaSuccess) return fail(std::string("cudaMalloc: ") + cudaGetErrorString(e));
        p = (T *)q;
        return 0;
    }
    operator T *() const { return p; }
};

}  // namespace vg
