// OFFLINE VERIFICATION TOOL (not part of the repo): a libcudart stand-in that keeps "device" memory on the host, runs no
// kernel and logs every host-to-device copy (size + FNV-1a hash), so that two builds of the library's HOST logic can be
// compared upload for upload on a machine without a GPU.
#include <cuda_runtime_api.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <mutex>
static std::mutex g_mu;
static std::vector<unsigned long long> g_log;
static unsigned long long fnv(const void* p, size_t n) { const unsigned char* b = (const unsigned char*)p; unsigned long long h = 1469598103934665603ull; for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 1099511628211ull; } return h; }
static void log_copy(const void* src, size_t n, int kind) { if (kind != cudaMemcpyHostToDevice) return; std::lock_guard<std::mutex> lk(g_mu); g_log.push_back(n); g_log.push_back(fnv(src, n)); }
extern "C" {
size_t fake_log_size() { return g_log.size(); }
void fake_log_copy(unsigned long long* out) { memcpy(out, g_log.data(), 8 * g_log.size()); }
void fake_log_clear() { g_log.clear(); }
void** __cudaRegisterFatBinary(void*) { static void* h; return &h; }
void __cudaRegisterFatBinaryEnd(void**) {}
void __cudaUnregisterFatBinary(void**) {}
void __cudaRegisterFunction(void**, const char*, char*, const char*, int, uint3*, uint3*, dim3*, dim3*, int*) {}
unsigned __cudaPushCallConfiguration(dim3, dim3, size_t, cudaStream_t) { return 0; }
cudaError_t __cudaPopCallConfiguration(dim3*, dim3*, size_t*, void*) { return cudaSuccess; }
cudaError_t cudaLaunchKernel(const void*, dim3, dim3, void**, size_t, cudaStream_t) { return cudaSuccess; }
cudaError_t cudaDeviceSynchronize() { return cudaSuccess; }
cudaError_t cudaDeviceGetAttribute(int* v, cudaDeviceAttr a, int) {
    switch (a) {
        case cudaDevAttrComputeCapabilityMajor: *v = 10; break;
        case cudaDevAttrComputeCapabilityMinor: *v = 0; break;
        case cudaDevAttrMultiProcessorCount: *v = 148; break;
        case cudaDevAttrMaxSharedMemoryPerBlock: *v = 49152; break;
        case cudaDevAttrMaxSharedMemoryPerBlockOptin: *v = 232448; break;
        case cudaDevAttrMaxSharedMemoryPerMultiprocessor: *v = 233472; break;
        default: *v = 1;
    }
    return cudaSuccess;
}
cudaError_t cudaFuncGetAttributes(cudaFuncAttributes* a, const void*) { memset(a, 0, sizeof *a); a->ptxVersion = a->binaryVersion = 100; a->maxThreadsPerBlock = 1024; return cudaSuccess; }
cudaError_t cudaPeekAtLastError() { return cudaSuccess; }
void __cudaRegisterVar(void**, char*, char*, const char*, int, size_t, int, int) {}
cudaError_t cudaEventCreate(cudaEvent_t* e) { *e = (cudaEvent_t)malloc(8); return cudaSuccess; }
cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { *e = (cudaEvent_t)malloc(8); return cudaSuccess; }
cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t, cudaEvent_t) { *ms = 0.f; return cudaSuccess; }
cudaError_t cudaEventDestroy(cudaEvent_t e) { free(e); return cudaSuccess; }
cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t) { return cudaSuccess; }
cudaError_t cudaEventSynchronize(cudaEvent_t) { return cudaSuccess; }
cudaError_t cudaFree(void* p) { free(p); return cudaSuccess; }
cudaError_t cudaFreeHost(void* p) { free(p); return cudaSuccess; }
cudaError_t cudaFuncSetAttribute(const void*, cudaFuncAttribute, int) { return cudaSuccess; }
cudaError_t cudaGetDevice(int* d) { *d = 0; return cudaSuccess; }
cudaError_t cudaGetDeviceCount(int* n) { *n = 1; return cudaSuccess; }
cudaError_t cudaGetDeviceProperties_v2(cudaDeviceProp* p, int) { memset(p, 0, sizeof *p); strcpy(p->name, "stub B200"); p->major = 10; p->minor = 0; p->multiProcessorCount = 148; p->sharedMemPerBlockOptin = 232448; p->totalGlobalMem = 180ull << 30; p->l2CacheSize = 126 << 20; return cudaSuccess; }
const char* cudaGetErrorString(cudaError_t) { return "stub"; }
cudaError_t cudaGetLastError() { return cudaSuccess; }
cudaError_t cudaHostAlloc(void** p, size_t n, unsigned) { *p = malloc(n ? n : 1); return cudaSuccess; }
cudaError_t cudaMalloc(void** p, size_t n) { *p = calloc(n ? n : 1, 1); return *p ? cudaSuccess : cudaErrorMemoryAllocation; }
cudaError_t cudaMemcpy(void* d, const void* s, size_t n, cudaMemcpyKind k) { log_copy(s, n, k); memcpy(d, s, n); return cudaSuccess; }
cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, cudaMemcpyKind k, cudaStream_t) { log_copy(s, n, k); memcpy(d, s, n); return cudaSuccess; }
cudaError_t cudaMemset(void* d, int v, size_t n) { memset(d, v, n); return cudaSuccess; }
cudaError_t cudaMemsetAsync(void* d, int v, size_t n, cudaStream_t) { memset(d, v, n); return cudaSuccess; }
cudaError_t cudaOccupancyMaxActiveBlocksPerMultiprocessorWithFlags(int* n, const void*, int, size_t, unsigned) { *n = 1; return cudaSuccess; }
cudaError_t cudaSetDevice(int) { return cudaSuccess; }
cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { *s = (cudaStream_t)malloc(8); return cudaSuccess; }
cudaError_t cudaStreamDestroy(cudaStream_t s) { free(s); return cudaSuccess; }
cudaError_t cudaStreamSynchronize(cudaStream_t) { return cudaSuccess; }
cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned) { return cudaSuccess; }
}
