// Host emulation of the small part of CUDA that the decode kernels use (tools/emu: development tooling, never
// loaded by the package).  Compiling csrc/*.cu{,h} with g++ against this header instead of the real
// <cuda_runtime.h> turns every kernel into a plain C++ function; a launch runs the thread blocks one after the
// other, every CUDA thread as a fiber, with warp collectives (__shfl_sync, __syncwarp, ballots) and __syncthreads
// implemented as fiber barriers.  Purpose: check bit-exactness of kernel changes against the oracle on the
// CPU-only build box before spending GPU time.  Nothing here is a decode path of the product.
#pragma once
#define PB_HOST_EMU 1
#include <algorithm>
#include <cassert>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <type_traits>
#include <utility>
#include <vector>

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __noinline__
#define __launch_bounds__(...)
#define __grid_constant__
#define __shared__ static
#define __align__(x) alignas(x)

struct uint2 { unsigned x, y; };
struct uint4 { unsigned x, y, z, w; };
struct int2 { int x, y; };
struct int4 { int x, y, z, w; };
struct alignas(16) double2 { double x, y; };
struct float2 { float x, y; };
static inline uint2 make_uint2(unsigned x, unsigned y) { return uint2{x, y}; }
static inline uint4 make_uint4(unsigned x, unsigned y, unsigned z, unsigned w) { return uint4{x, y, z, w}; }
static inline int2 make_int2(int x, int y) { return int2{x, y}; }
static inline double2 make_double2(double x, double y) { return double2{x, y}; }
struct dim3 {
    unsigned x, y, z;
    dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};

// ------------------------------------------------------------------------------------------------ host runtime
typedef int cudaError_t;
enum { cudaSuccess = 0, cudaErrorInvalidValue = 1, cudaErrorMemoryAllocation = 2 };
typedef void *cudaStream_t;
typedef void *cudaEvent_t;
enum cudaMemcpyKind { cudaMemcpyHostToDevice = 1, cudaMemcpyDeviceToHost = 2, cudaMemcpyDeviceToDevice = 3, cudaMemcpyDefault = 4 };
enum { cudaHostAllocMapped = 2, cudaHostAllocDefault = 0, cudaHostAllocPortable = 1, cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2 };
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize = 8 };
enum cudaDeviceAttr { cudaDevAttrMultiProcessorCount = 16 };
struct cudaDeviceProp { int major = 10, minor = 0, multiProcessorCount = 2; char name[64] = "emulated sm_100"; };

namespace pb_emu {
inline int sm_count() { const char *e = getenv("PB_EMU_SMS"); return e ? atoi(e) : 2; }
}
static inline const char *cudaGetErrorString(cudaError_t e) { return e == cudaSuccess ? "no error" : "emulated CUDA error"; }
static inline cudaError_t cudaGetLastError() { return cudaSuccess; }
static inline cudaError_t cudaGetDevice(int *d) { *d = 0; return cudaSuccess; }
static inline cudaError_t cudaSetDevice(int) { return cudaSuccess; }
static inline cudaError_t cudaGetDeviceCount(int *n) { *n = 1; return cudaSuccess; }
static inline cudaError_t cudaDeviceGetAttribute(int *v, cudaDeviceAttr, int) { *v = pb_emu::sm_count(); return cudaSuccess; }
static inline cudaError_t cudaGetDeviceProperties(cudaDeviceProp *p, int) { *p = cudaDeviceProp(); p->multiProcessorCount = pb_emu::sm_count(); return cudaSuccess; }
static inline cudaError_t cudaMalloc(void **p, size_t n) { *p = aligned_alloc(256, (n + 255) & ~(size_t)255); return *p ? cudaSuccess : cudaErrorMemoryAllocation; }
template <class T> static inline cudaError_t cudaMalloc(T **p, size_t n) { return cudaMalloc((void **)p, n); }
static inline cudaError_t cudaFree(void *p) { free(p); return cudaSuccess; }
static inline cudaError_t cudaHostAlloc(void **p, size_t n, unsigned) { return cudaMalloc(p, n); }
static inline cudaError_t cudaFreeHost(void *p) { free(p); return cudaSuccess; }
static inline cudaError_t cudaHostGetDevicePointer(void **d, void *h, unsigned) { *d = h; return cudaSuccess; }
static inline cudaError_t cudaMemcpy(void *d, const void *s, size_t n, cudaMemcpyKind) { memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemcpyAsync(void *d, const void *s, size_t n, cudaMemcpyKind, cudaStream_t = nullptr) { memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemset(void *d, int v, size_t n) { memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaMemsetAsync(void *d, int v, size_t n, cudaStream_t = nullptr) { memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t *s, unsigned) { *s = (void *)1; return cudaSuccess; }
static inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaStreamDestroy(cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaDeviceSynchronize() { return cudaSuccess; }
static inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t *e, unsigned) { *e = (void *)1; return cudaSuccess; }
static inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaEventDestroy(cudaEvent_t) { return cudaSuccess; }
static inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return cudaSuccess; }
enum cudaMemoryType { cudaMemoryTypeUnregistered = 0, cudaMemoryTypeHost = 1, cudaMemoryTypeDevice = 2 };
struct cudaPointerAttributes { cudaMemoryType type = cudaMemoryTypeUnregistered; };
static inline cudaError_t cudaPointerGetAttributes(cudaPointerAttributes *a, const void *) { a->type = cudaMemoryTypeUnregistered; return cudaSuccess; }
static inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned) { return cudaSuccess; }
static inline cudaError_t cudaFuncSetAttribute(const void *, cudaFuncAttribute, int) { return cudaSuccess; }
static inline cudaError_t cudaOccupancyMaxActiveBlocksPerMultiprocessor(int *n, const void *, int threads, size_t smem) {
    long v = 233472 / (long)(smem + 1024);
    long w = 64 / std::max(1, threads / 32);
    *n = (int)std::max(0l, std::min(std::min(v, w), 32l));
    return cudaSuccess;
}

// ------------------------------------------------------------------------------------------------ fibers
namespace pb_emu {
struct Idx { unsigned x = 0, y = 0, z = 0; };
struct WarpState {
    int arrived = 0, gen = 0;
    unsigned long long xchg[2][32];
};
struct State {
    Idx tid, bid, bdim, gdim;
    int nthreads = 0, cur = 0;
    std::vector<void *> sp;
    std::vector<char> done;
    void *main_sp = nullptr;
    std::vector<WarpState> warps;
    std::vector<unsigned> ncoll;   // per thread: collectives executed so far (selects the exchange buffer)
    int blk_arrived = 0, blk_gen = 0;
    int blk_or[2] = {0, 0};        // __syncthreads_or: one accumulator per barrier generation parity
    char *smem = nullptr;
    std::function<void()> body;
    int live = 0;
};
State &st();
void yield();
void launch(const std::function<void()> &body, dim3 grid, dim3 block, size_t smem);
inline int lane() { return (int)(st().cur & 31); }
inline WarpState &warp() { return st().warps[st().cur >> 5]; }
inline int warp_threads() { State &s = st(); return std::min(32, s.nthreads - (s.cur & ~31)); }
inline void warp_barrier() {
    WarpState &w = warp();
    const int g = w.gen;
    if (++w.arrived == warp_threads()) { w.arrived = 0; w.gen++; }
    else while (w.gen == g) yield();
}
inline void block_barrier() {
    State &s = st();
    const int g = s.blk_gen;
    if (++s.blk_arrived == s.nthreads) { s.blk_arrived = 0; s.blk_gen++; }
    else while (s.blk_gen == g) yield();
}
// generation g accumulates into blk_or[g & 1]; it is cleared by the first arrival at generation g + 2, which no thread
// reaches before every thread has passed generation g + 1, i.e. has read the result of g
inline int block_barrier_or(int pred) {
    State &s = st();
    const int g = s.blk_gen;
    if (s.blk_arrived == 0) s.blk_or[g & 1] = 0;
    s.blk_or[g & 1] |= pred ? 1 : 0;
    block_barrier();
    return s.blk_or[g & 1];
}
template <class T> inline T exchange(T v, int src) {   // one barrier per collective: double-buffered slots
    static_assert(sizeof(T) <= 8, "shuffle of > 8 bytes");
    // buffer k of collective c is only rewritten by collective c+2, which no lane reaches before every lane has passed
    // the barrier of c+1, i.e. has finished reading c
    const unsigned k = st().ncoll[st().cur]++ & 1u;
    unsigned long long bits = 0;
    memcpy(&bits, &v, sizeof(T));
    warp().xchg[k][lane()] = bits;
    warp_barrier();
    T r;
    memcpy(&r, &warp().xchg[k][src & 31], sizeof(T));
    return r;
}
// kernel registry: cudaLaunchKernel gets a const void* and an argument array
std::map<const void *, std::function<void(void **)>> &registry();
template <class... A, size_t... I>
inline void call_kernel(void (*k)(A...), void **args, std::index_sequence<I...>) { k(*(std::remove_reference_t<A> *)args[I]...); }
template <class... A>
inline const void *reg(void (*k)(A...)) {
    const void *key = (const void *)k;
    registry()[key] = [k](void **args) { call_kernel(k, args, std::index_sequence_for<A...>{}); };
    return key;
}
inline char *dyn_smem() { return st().smem; }
}  // namespace pb_emu

#define threadIdx (pb_emu::st().tid)
#define blockIdx (pb_emu::st().bid)
#define blockDim (pb_emu::st().bdim)
#define gridDim (pb_emu::st().gdim)

static inline cudaError_t cudaLaunchKernel(const void *fn, dim3 grid, dim3 block, void **args, size_t smem, cudaStream_t) {
    auto it = pb_emu::registry().find(fn);
    if (it == pb_emu::registry().end()) { fprintf(stderr, "pb_emu: launch of an unregistered kernel\n"); abort(); }
    auto f = it->second;
    pb_emu::launch([f, args]() { f(args); }, grid, block, smem);
    return cudaSuccess;
}

// ------------------------------------------------------------------------------------------------ device intrinsics
static inline void __syncwarp(unsigned = 0xffffffffu) { pb_emu::warp_barrier(); }
static inline void __syncthreads() { pb_emu::block_barrier(); }
static inline int __syncthreads_or(int pred) { return pb_emu::block_barrier_or(pred); }
template <class T> static inline T __shfl_sync(unsigned, T v, int src, int width = 32) {
    const int l = pb_emu::lane();
    return pb_emu::exchange(v, (l & ~(width - 1)) | (src & (width - 1)));
}
template <class T> static inline T __shfl_xor_sync(unsigned, T v, int m, int width = 32) { (void)width; return pb_emu::exchange(v, pb_emu::lane() ^ m); }
template <class T> static inline T __shfl_down_sync(unsigned, T v, unsigned d, int width = 32) {
    const int l = pb_emu::lane();
    const int s = ((l & (width - 1)) + (int)d < width) ? l + (int)d : l;
    return pb_emu::exchange(v, s);
}
template <class T> static inline T __shfl_up_sync(unsigned, T v, unsigned d, int width = 32) {
    const int l = pb_emu::lane();
    const int s = ((l & (width - 1)) >= (int)d) ? l - (int)d : l;
    return pb_emu::exchange(v, s);
}
static inline unsigned __ballot_sync(unsigned, int pred) {
    unsigned r = 0;
    const int n = pb_emu::warp_threads();
    // gather every lane's predicate with one exchange per source lane would be slow: exchange once, then read all slots
    const unsigned k = pb_emu::st().ncoll[pb_emu::st().cur]++ & 1u;
    pb_emu::warp().xchg[k][pb_emu::lane()] = pred ? 1ull : 0ull;
    pb_emu::warp_barrier();
    for (int i = 0; i < n; ++i) r |= (unsigned)(pb_emu::warp().xchg[k][i] & 1ull) << i;
    return r;
}
static inline int __all_sync(unsigned m, int pred) { const unsigned b = __ballot_sync(m, pred); const int n = pb_emu::warp_threads(); return b == (n == 32 ? 0xffffffffu : ((1u << n) - 1u)); }
static inline int __any_sync(unsigned m, int pred) { return __ballot_sync(m, pred) != 0; }
template <class T> static inline T __ldg(const T *p) { return *p; }
template <class T> static inline T __ldcs(const T *p) { return *p; }
template <class T> static inline T __ldcg(const T *p) { return *p; }
template <class T> static inline void __stcs(T *p, T v) { *p = v; }
template <class T> static inline void __stcg(T *p, T v) { *p = v; }
static inline unsigned __byte_perm(unsigned x, unsigned y, unsigned s) {
    const unsigned long long v = ((unsigned long long)y << 32) | x;
    unsigned r = 0;
    for (int i = 0; i < 4; ++i) {
        const unsigned sel = (s >> (4 * i)) & 0xfu;
        unsigned b = (unsigned)(v >> (8 * (sel & 7u))) & 0xffu;
        if (sel & 8u) b = (b & 0x80u) ? 0xffu : 0u;
        r |= b << (8 * i);
    }
    return r;
}
static inline unsigned __funnelshift_r(unsigned lo, unsigned hi, unsigned sh) { return (unsigned)(((((unsigned long long)hi) << 32) | lo) >> (sh & 31u)); }
static inline unsigned __funnelshift_l(unsigned lo, unsigned hi, unsigned sh) { return (unsigned)((((((unsigned long long)hi) << 32) | lo) << (sh & 31u)) >> 32); }
static inline int __popc(unsigned x) { return __builtin_popcount(x); }
static inline int __popcll(unsigned long long x) { return __builtin_popcountll(x); }
static inline int __clz(int x) { return x ? __builtin_clz((unsigned)x) : 32; }
static inline int __ffs(int x) { return __builtin_ffs(x); }
static inline unsigned __brev(unsigned x) { unsigned r = 0; for (int i = 0; i < 32; ++i) r |= ((x >> i) & 1u) << (31 - i); return r; }
static inline double __hiloint2double(int hi, int lo) { unsigned long long b = ((unsigned long long)(unsigned)hi << 32) | (unsigned)lo; double d; memcpy(&d, &b, 8); return d; }
static inline int __double2hiint(double d) { unsigned long long b; memcpy(&b, &d, 8); return (int)(b >> 32); }
static inline int __double2loint(double d) { unsigned long long b; memcpy(&b, &d, 8); return (int)(b & 0xffffffffu); }
static inline long long __double_as_longlong(double d) { long long b; memcpy(&b, &d, 8); return b; }
static inline double __longlong_as_double(long long b) { double d; memcpy(&d, &b, 8); return d; }
static inline size_t __cvta_generic_to_shared(const void *p) { return (size_t)p; }
template <class T> static inline T atomicAdd(T *p, T v) { T o = *p; *p = o + v; return o; }
template <class T> static inline T atomicExch(T *p, T v) { T o = *p; *p = v; return o; }
template <class T> static inline T atomicCAS(T *p, T c, T v) { T o = *p; if (o == c) *p = v; return o; }
template <class T> static inline T atomicOr(T *p, T v) { T o = *p; *p = o | v; return o; }
template <class T> static inline T atomicMax(T *p, T v) { T o = *p; if (v > o) *p = v; return o; }
static inline void __nanosleep(unsigned) {}
static inline void __threadfence() {}
static inline void __threadfence_block() {}
