// quantum_basis_b200/csrc/context.cu -- per-thread context, error reporting, device-memory helpers of libqbgpu.
#include "internal.hpp"
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>

namespace qb {

static thread_local std::string g_err;
static thread_local Context g_ctx;

void set_error(const std::string &msg) { g_err = msg; }
int fail(int code, const std::string &msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const char *what, const char *file, int line)
{
    char buf[1024];
    snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
    g_err = buf;
    (void)cudaGetLastError();
    return QBGPU_ERR_CUDA;
}
Context &ctx() { return g_ctx; }

int ensure_init()
{
    if (g_ctx.device >= 0) return QBGPU_OK;
    return qbgpu_init(0);
}

}  // namespace qb

using namespace qb;

extern "C" {

const char *qbgpu_last_error(void) { return g_err.c_str(); }
const char *qbgpu_version(void) { return "qbgpu 0.1 (sm_100a)"; }

int qbgpu_device_count(int *count)
{
    if (!count) return fail(QBGPU_ERR_ARG, "count is null");
    QB_CUDA(cudaGetDeviceCount(count));
    return QBGPU_OK;
}

int qbgpu_init(int device)
{
    Context &c = g_ctx;
    if (c.device == device) { QB_CUDA(cudaSetDevice(device)); return QBGPU_OK; }
    if (c.device >= 0) QB_TRY(qbgpu_finalize());
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(QBGPU_ERR_CUDA, std::string("no CUDA device available (libqbgpu has no CPU fallback): ") +
                                        cudaGetErrorString(e));
    if (device < 0 || device >= count) return fail(QBGPU_ERR_ARG, "device index out of range");
    QB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    QB_CUDA(cudaGetDeviceProperties(&prop, device));
    c.num_sms = prop.multiProcessorCount;
    // No L2 limit is set.  L2 evict_last / persisting accesses only take effect inside the persisting set-aside, which
    // defaults to 0 bytes; measured, a set-aside does not help the products and the maximum one costs 7-13 %
    // (profiles/r01_kbench_sweep3_l2_persist.txt).  An L2 fetch granularity hint had no effect at all
    // (profiles/r01_kbench_l2_fetch_granularity.txt).
    QB_CUDA(cudaStreamCreateWithFlags(&c.own_stream, cudaStreamNonBlocking));
    QB_CUDA(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
    c.stream = c.own_stream;
    QB_CUDA(cudaMalloc(&c.partials, sizeof(double) * kMaxPartialBlocks * kDotSlots));
    QB_CUDA(cudaMalloc(&c.ticket, sizeof(unsigned)));
    QB_CUDA(cudaMemset(c.ticket, 0, sizeof(unsigned)));
    QB_CUDA(cudaMalloc(&c.scal_dev, sizeof(double) * 64));
    QB_CUDA(cudaMemset(c.scal_dev, 0, sizeof(double) * 64));
    QB_CUDA(cudaMallocHost(&c.scal_host, sizeof(double) * 64));
    c.device = device;
    return QBGPU_OK;
}

int qbgpu_finalize(void)
{
    Context &c = g_ctx;
    if (c.device < 0) return QBGPU_OK;
    cudaSetDevice(c.device);
    cudaDeviceSynchronize();
    if (c.partials) cudaFree(c.partials);
    if (c.ticket) cudaFree(c.ticket);
    if (c.scal_dev) cudaFree(c.scal_dev);
    if (c.scal_host) cudaFreeHost(c.scal_host);
    if (c.stage_x) cudaFree(c.stage_x);
    if (c.stage_y) cudaFree(c.stage_y);
    if (c.own_stream) cudaStreamDestroy(c.own_stream);
    if (c.copy_stream) cudaStreamDestroy(c.copy_stream);
    c = Context();
    return QBGPU_OK;
}

int qbgpu_set_stream(void *s)
{
    QB_TRY(ensure_init());
    g_ctx.stream = s ? (cudaStream_t)s : g_ctx.own_stream;
    return QBGPU_OK;
}

int qbgpu_synchronize(void)
{
    QB_TRY(ensure_init());
    QB_CUDA(cudaStreamSynchronize(g_ctx.stream));
    return QBGPU_OK;
}

int qbgpu_malloc(void **p, size_t bytes)
{
    QB_TRY(ensure_init());
    if (!p) return fail(QBGPU_ERR_ARG, "null out pointer");
    cudaError_t e = cudaMalloc(p, bytes ? bytes : 1);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(QBGPU_ERR_ALLOC, std::string("cudaMalloc failed: ") + cudaGetErrorString(e)); }
    return QBGPU_OK;
}
int qbgpu_free(void *p) { if (p) QB_CUDA(cudaFree(p)); return QBGPU_OK; }
int qbgpu_memcpy_h2d(void *dst, const void *src, size_t bytes)
{
    QB_TRY(ensure_init());
    QB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, g_ctx.stream));
    QB_CUDA(cudaStreamSynchronize(g_ctx.stream));
    return QBGPU_OK;
}
int qbgpu_memcpy_d2d(void *dst, const void *src, size_t bytes)
{
    QB_TRY(ensure_init());
    QB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, g_ctx.stream));
    return QBGPU_OK;
}
int qbgpu_memcpy_d2h(void *dst, const void *src, size_t bytes)
{
    QB_TRY(ensure_init());
    QB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, g_ctx.stream));
    QB_CUDA(cudaStreamSynchronize(g_ctx.stream));
    return QBGPU_OK;
}
int qbgpu_memset0(void *p, size_t bytes)
{
    QB_TRY(ensure_init());
    QB_CUDA(cudaMemsetAsync(p, 0, bytes, g_ctx.stream));
    return QBGPU_OK;
}

// host ranges pinned for asynchronous copies (ARPACK's workd, src/lanczos.cc:417,464)
static std::mutex g_reg_mu;
static std::map<void *, size_t> g_registered;

int qbgpu_host_register(void *ptr, size_t bytes)
{
    QB_TRY(ensure_init());
    std::lock_guard<std::mutex> lk(g_reg_mu);
    if (g_registered.count(ptr)) return QBGPU_OK;
    QB_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterDefault));
    g_registered[ptr] = bytes;
    return QBGPU_OK;
}
int qbgpu_host_unregister(void *ptr)
{
    std::lock_guard<std::mutex> lk(g_reg_mu);
    auto it = g_registered.find(ptr);
    if (it == g_registered.end()) return QBGPU_OK;
    QB_CUDA(cudaHostUnregister(ptr));
    g_registered.erase(it);
    return QBGPU_OK;
}

int qbgpu_debug_set_variant(int id)
{
    if (id < 1000 || id > 1002) return fail(QBGPU_ERR_ARG, "debug_set_variant: unknown id " + std::to_string(id) + " (1000, 1001 or 1002)");
    qb::set_kron_local_variant(id - 1000);
    return QBGPU_OK;
}

int64_t qbgpu_kernel_launches(int reset)
{
    long long v = g_ctx.launches;
    if (reset) g_ctx.launches = 0;
    return v;
}

}  // extern "C"
