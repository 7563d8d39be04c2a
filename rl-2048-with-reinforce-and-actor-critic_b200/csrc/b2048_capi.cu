// b2048_capi.cu — error reporting, version and debug switches of the C ABI (include/b2048.h).
#include "b2048_internal.h"

namespace b2 {

static thread_local std::string g_last_error;

void set_error(const std::string& msg) { g_last_error = msg; }

int fail(b2048_status st, const std::string& msg) {
    set_error(msg);
    return (int)st;
}

int check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return B2048_OK;
    set_error(std::string(what) + ": " + cudaGetErrorString(e));
    return (int)B2048_ERR_CUDA;
}

long long* debug_clock_begin(const b2048_handle* h, int option, cudaStream_t stream) {
    if (!(h->debug & (1u << option))) return nullptr;
    cudaMemsetAsync(h->dbg_clock, 0, DBG_CLOCK_SLOTS * sizeof(long long), stream);
    return h->dbg_clock;
}

int debug_clock_read(const b2048_handle* h, long long* host, int count, cudaStream_t stream) {
    B2_CUDA(cudaStreamSynchronize(stream));
    B2_CUDA(cudaMemcpy(host, h->dbg_clock, count * sizeof(long long), cudaMemcpyDeviceToHost));
    return B2048_OK;
}

// The clock buffer and the pipeline's progress words, allocated on the handle's device (b2048_destroy frees them).
static int alloc_debug_buffers(b2048_handle* h) {
    int cur = 0;
    B2_CUDA(cudaGetDevice(&cur));
    B2_CUDA(cudaSetDevice(h->device));
    cudaError_t e = cudaMalloc(&h->dbg_clock, DBG_CLOCK_SLOTS * sizeof(long long));
    if (e == cudaSuccess) e = cudaHostAlloc(&h->dbg_progress, DBG_PROGRESS_WORDS * sizeof(int), cudaHostAllocMapped);
    cudaSetDevice(cur);
    if (e == cudaSuccess) return B2048_OK;
    cudaFree(h->dbg_clock);
    h->dbg_clock = nullptr;
    h->dbg_progress = nullptr;
    return check_cuda(e, "b2048_debug_set: clock buffers");
}

}  // namespace b2

extern "C" const char* b2048_last_error(void) { return b2::g_last_error.c_str(); }

extern "C" int b2048_version(void) { return 100; }

extern "C" int b2048_debug_set(b2048_handle* h, int32_t option, int32_t value) {
    B2_REQUIRE(h != nullptr, "b2048_debug_set: handle is NULL");
    if (option == B2048_DBG_PARAM_PIPE_SPLIT) {
        h->pipe_split = (unsigned)value;
        return B2048_OK;
    }
    B2_REQUIRE(option >= 0 && option < B2048_DBG_COUNT, "b2048_debug_set: unknown option");
    if (value && (option == B2048_DBG_TC_CLOCKS || option == B2048_DBG_STEP_CLOCKS) && !h->dbg_clock) {
        const int st = b2::alloc_debug_buffers(h);
        if (st != B2048_OK) return st;
    }
    if (value) h->debug |= 1u << option;
    else h->debug &= ~(1u << option);
    return B2048_OK;
}
