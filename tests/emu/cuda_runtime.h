/* TEST INFRASTRUCTURE ONLY — never part of the product build.
 *
 * A stand-in for <cuda_runtime.h> that lets g++ compile the product's CUDA sources (csrc/mcb_api.cu + mcb_kernels.cuh)
 * into tests/emu/_build/libmcb200_emu.so, so that the CPU test tier can EXECUTE THE KERNELS' SOURCE on the host, at small
 * grid sizes, against the oracle (there is no GPU in the build container; a kernel bug found here costs seconds, on
 * the GPU box a queue slot).  The product library (libmcb200.so) is built by nvcc from the same sources without any
 * of this; nothing in the package, bench.py or __graft_entry__ loads the emulated library.
 *
 * How device code runs here: one thread block at a time, every CUDA thread of the block a ucontext fiber on one OS
 * thread, scheduled round-robin.  __syncthreads and the warp collectives (__shfl_*_sync, __ballot_sync, __any_sync,
 * __syncwarp) are rendezvous points: a fiber yields until every live thread of the block / warp has arrived.  Exited
 * threads stop counting, as in CUDA.  Atomics are plain read-modify-writes (one OS thread).  __shared__ becomes
 * `static` (blocks run one after the other); dynamic shared memory comes from emu::dyn_smem().
 * The runtime API is backed by malloc/memcpy; streams and events are no-ops (everything is synchronous).
 */
#pragma once
#include <math.h>
#include <signal.h>
#include <stdio.h>
#include <sys/mman.h>
#include <unistd.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <ucontext.h>

#include <cmath>
#include <functional>
#include <map>
#include <mutex>
#include <vector>

#define MCB_EMULATED_DEVICE 1
#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __noinline__ /* libstdc++ spells __attribute__((__noinline__)): must expand to nothing */
#define __launch_bounds__(...)
#define __grid_constant__
#define __shared__ static
#define __constant__ static

using std::isinf;
using std::isnan;

struct uint3 { unsigned x, y, z; };
struct dim3 {
    unsigned x, y, z;
    dim3(unsigned a = 1, unsigned b = 1, unsigned c = 1) : x(a), y(b), z(c) {}
};
struct alignas(16) float4 { float x, y, z, w; };
struct alignas(16) uint4 { unsigned x, y, z, w; };
struct alignas(8) float2 { float x, y; };
struct alignas(8) uint2 { unsigned x, y; };
static inline float4 make_float4(float a, float b, float c, float d) { return float4{a, b, c, d}; }
static inline uint4 make_uint4(unsigned a, unsigned b, unsigned c, unsigned d) { return uint4{a, b, c, d}; }
static inline float2 make_float2(float a, float b) { return float2{a, b}; }
static inline uint2 make_uint2(unsigned a, unsigned b) { return uint2{a, b}; }

inline uint3 threadIdx, blockIdx;
inline dim3 blockDim, gridDim;

/* ---- fiber engine ------------------------------------------------------------------------------------------- */
namespace emu {
struct Barrier { unsigned alive = 0, arrived = 0, gen = 0; };
struct Fiber {
    ucontext_t ctx;
    bool done = false;
    unsigned tid = 0;
};
struct State {
    ucontext_t sched;
    std::vector<Fiber> fibers;
    std::vector<char> stacks;
    Barrier block_bar;
    std::vector<Barrier> warp_bar;
    std::vector<unsigned long long> slots; /* 32 exchange slots per warp */
    int current = -1;
    const std::function<void()>* body = nullptr;
    std::vector<char> dyn;
    unsigned long long launches = 0;
};
inline State& S() { static State s; return s; }
constexpr size_t kStack = 192 * 1024;

inline void yield() {
    State& s = S();
    swapcontext(&s.fibers[s.current].ctx, &s.sched);
}
inline void arrive_and_wait(Barrier& b) {
    const unsigned g = b.gen;
    if (++b.arrived >= b.alive) { b.arrived = 0; b.gen++; return; }
    while (b.gen == g) yield();
}
inline void thread_exit(Barrier& b) {
    if (b.alive) b.alive--;
    if (b.alive && b.arrived >= b.alive) { b.arrived = 0; b.gen++; }
}
inline void trampoline() {
    State& s = S();
    Fiber& f = s.fibers[s.current];
    (*s.body)();
    f.done = true;
    thread_exit(s.block_bar);
    thread_exit(s.warp_bar[f.tid >> 5]);
    swapcontext(&f.ctx, &s.sched);
}
inline void* dyn_smem() { return S().dyn.data(); }

inline void launch(dim3 grid, dim3 block, size_t smem, const std::function<void()>& body) {
    State& s = S();
    const unsigned nt = block.x * block.y * block.z;
    if (nt == 0 || grid.x == 0 || grid.y == 0 || grid.z == 0) return;
    s.launches++;
    if (s.dyn.size() < smem + 64) s.dyn.resize(smem + 64);
    if (s.stacks.size() < (size_t)nt * kStack) s.stacks.resize((size_t)nt * kStack);
    s.fibers.resize(nt);
    s.body = &body;
    gridDim = grid;
    blockDim = block;
    const unsigned nw = (nt + 31) / 32;
    for (unsigned bz = 0; bz < grid.z; bz++)
        for (unsigned by = 0; by < grid.y; by++)
            for (unsigned bx = 0; bx < grid.x; bx++) {
                blockIdx = uint3{bx, by, bz};
                s.block_bar = Barrier{nt, 0, 0};
                s.warp_bar.assign(nw, Barrier{});
                s.slots.assign((size_t)nw * 32, 0ull);
                for (unsigned w = 0; w < nw; w++) s.warp_bar[w].alive = (w + 1) * 32 <= nt ? 32 : nt - w * 32;
                for (unsigned t = 0; t < nt; t++) {
                    Fiber& f = s.fibers[t];
                    f.done = false;
                    f.tid = t;
                    getcontext(&f.ctx);
                    f.ctx.uc_stack.ss_sp = s.stacks.data() + (size_t)t * kStack;
                    f.ctx.uc_stack.ss_size = kStack;
                    f.ctx.uc_link = &s.sched;
                    makecontext(&f.ctx, (void (*)())trampoline, 0);
                }
                unsigned remaining = nt;
                while (remaining) {
                    for (unsigned t = 0; t < nt; t++) {
                        Fiber& f = s.fibers[t];
                        if (f.done) continue;
                        s.current = (int)t;
                        threadIdx = uint3{t % block.x, (t / block.x) % block.y, t / (block.x * block.y)};
                        swapcontext(&s.sched, &f.ctx);
                        if (f.done) remaining--;
                    }
                }
            }
    s.current = -1;
}

inline unsigned lane_id() { return S().fibers[S().current].tid & 31u; }
inline unsigned warp_id() { return S().fibers[S().current].tid >> 5; }
template <class T>
inline unsigned long long to_bits(T v) { unsigned long long b = 0; memcpy(&b, &v, sizeof(T)); return b; }
template <class T>
inline T from_bits(unsigned long long b) { T v; memcpy(&v, &b, sizeof(T)); return v; }
/* exchange: every live lane publishes a value, then reads lane `src` (its own when src is out of range or exited) */
template <class T>
inline T exchange(T v, int src) {
    State& s = S();
    const unsigned w = warp_id(), l = lane_id();
    s.slots[(size_t)w * 32 + l] = to_bits(v);
    arrive_and_wait(s.warp_bar[w]);
    T r = v;
    if (src >= 0 && src < 32) {
        const unsigned t = w * 32 + (unsigned)src;
        if (t < s.fibers.size() && !s.fibers[t].done) r = from_bits<T>(s.slots[(size_t)w * 32 + src]);
    }
    arrive_and_wait(s.warp_bar[w]);
    return r;
}
inline unsigned ballot(bool p) {
    State& s = S();
    const unsigned w = warp_id(), l = lane_id();
    s.slots[(size_t)w * 32 + l] = p ? 1ull : 0ull;
    arrive_and_wait(s.warp_bar[w]);
    unsigned m = 0;
    for (unsigned q = 0; q < 32; q++) {
        const unsigned t = w * 32 + q;
        if (t < s.fibers.size() && !s.fibers[t].done && s.slots[(size_t)w * 32 + q]) m |= 1u << q;
    }
    arrive_and_wait(s.warp_bar[w]);
    return m;
}
}  // namespace emu

static inline void __syncthreads() { emu::arrive_and_wait(emu::S().block_bar); }
static inline void __syncwarp(unsigned = 0xffffffffu) { emu::arrive_and_wait(emu::S().warp_bar[emu::warp_id()]); }
template <class T> static inline T __shfl_sync(unsigned, T v, int src) { return emu::exchange(v, src & 31); }
template <class T> static inline T __shfl_up_sync(unsigned, T v, unsigned d) { return emu::exchange(v, (int)emu::lane_id() - (int)d); }
template <class T> static inline T __shfl_down_sync(unsigned, T v, unsigned d) { return emu::exchange(v, (int)emu::lane_id() + (int)d); }
template <class T> static inline T __shfl_xor_sync(unsigned, T v, int m) { return emu::exchange(v, (int)(emu::lane_id() ^ (unsigned)m)); }
static inline unsigned __ballot_sync(unsigned, bool p) { return emu::ballot(p); }
static inline bool __any_sync(unsigned, bool p) { return emu::ballot(p) != 0u; }
static inline bool __all_sync(unsigned, bool p) { return emu::ballot(!p) == 0u; }

template <class T> static inline T __ldg(const T* p) { return *p; }
template <class T> static inline T __ldcs(const T* p) { return *p; }
template <class T> static inline void __stcs(T* p, T v) { *p = v; }
template <class T> static inline void __stcg(T* p, T v) { *p = v; }
static inline int __popc(unsigned x) { return __builtin_popcount(x); }
static inline int __popcll(unsigned long long x) { return __builtin_popcountll(x); }
static inline int __ffs(int x) { return __builtin_ffs(x); }
static inline int __ffsll(long long x) { return __builtin_ffsll(x); }
static inline int __clz(int x) { return x ? __builtin_clz((unsigned)x) : 32; }
static inline unsigned __funnelshift_r(unsigned lo, unsigned hi, unsigned sh) {
    return (unsigned)(((((unsigned long long)hi) << 32) | lo) >> (sh & 31u));
}
static inline unsigned __funnelshift_l(unsigned lo, unsigned hi, unsigned sh) {
    return (unsigned)((((((unsigned long long)hi) << 32) | lo) << (sh & 31u)) >> 32);
}
static inline unsigned __umulhi(unsigned a, unsigned b) { return (unsigned)(((unsigned long long)a * b) >> 32); }
static inline unsigned __float_as_uint(float f) { unsigned u; memcpy(&u, &f, 4); return u; }
static inline int __float_as_int(float f) { int u; memcpy(&u, &f, 4); return u; }
static inline float __uint_as_float(unsigned u) { float f; memcpy(&f, &u, 4); return f; }
static inline float __int_as_float(int u) { float f; memcpy(&f, &u, 4); return f; }
static inline long long __double_as_longlong(double d) { long long u; memcpy(&u, &d, 8); return u; }
static inline double __longlong_as_double(long long u) { double d; memcpy(&d, &u, 8); return d; }
static inline float __fadd_rn(float a, float b) { return a + b; }
static inline float __fsub_rn(float a, float b) { return a - b; }
static inline float __fmul_rn(float a, float b) { return a * b; }
static inline float __fdiv_rn(float a, float b) { return a / b; }
static inline float __fmaf_rn(float a, float b, float c) { return fmaf(a, b, c); }
static inline float rsqrtf(float x) { return 1.0f / sqrtf(x); }
static inline float __frcp_rn(float x) { return 1.0f / x; }
static inline float __fsqrt_rn(float x) { return sqrtf(x); }
template <class T> static inline T min(T a, T b) { return b < a ? b : a; }
template <class T> static inline T max(T a, T b) { return a < b ? b : a; }

template <class T> static inline T atomicAdd(T* p, T v) { T o = *p; *p = o + v; return o; }
static inline unsigned atomicOr(unsigned* p, unsigned v) { unsigned o = *p; *p = o | v; return o; }
static inline unsigned long long atomicOr(unsigned long long* p, unsigned long long v) { unsigned long long o = *p; *p = o | v; return o; }
static inline unsigned atomicAnd(unsigned* p, unsigned v) { unsigned o = *p; *p = o & v; return o; }
template <class T> static inline T atomicExch(T* p, T v) { T o = *p; *p = v; return o; }
template <class T> static inline T atomicMax(T* p, T v) { T o = *p; if (v > o) *p = v; return o; }
template <class T> static inline T atomicMin(T* p, T v) { T o = *p; if (v < o) *p = v; return o; }
template <class T> static inline T atomicCAS(T* p, T cmp, T v) { T o = *p; if (o == cmp) *p = v; return o; }
static inline void __threadfence() {}
static inline void __threadfence_block() {}

/* ---- runtime API, host memory behind it ---------------------------------------------------------------------- */
typedef int cudaError_t;
enum { cudaSuccess = 0, cudaErrorMemoryAllocation = 2, cudaErrorNotSupported = 801 };
typedef struct emuStream* cudaStream_t;
typedef struct emuEvent* cudaEvent_t;
typedef struct emuLibrary* cudaLibrary_t;
typedef struct emuKernel* cudaKernel_t;
enum cudaMemcpyKind { cudaMemcpyHostToHost = 0, cudaMemcpyHostToDevice = 1, cudaMemcpyDeviceToHost = 2, cudaMemcpyDeviceToDevice = 3, cudaMemcpyDefault = 4 };
enum { cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2, cudaHostRegisterDefault = 0, cudaHostRegisterPortable = 1 };
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize = 8, cudaFuncAttributePreferredSharedMemoryCarveout = 9 };
struct cudaDeviceProp { int multiProcessorCount; char name[256]; size_t totalGlobalMem; };
struct cudaPitchedPtr { void* ptr; size_t pitch, xsize, ysize; };
struct cudaPos { size_t x, y, z; };
struct cudaExtent { size_t width, height, depth; };
struct cudaMemcpy3DParms { cudaPitchedPtr srcPtr; cudaPos srcPos; cudaPitchedPtr dstPtr; cudaPos dstPos; cudaExtent extent; cudaMemcpyKind kind; };
static inline cudaPitchedPtr make_cudaPitchedPtr(void* p, size_t pitch, size_t xs, size_t ys) { return cudaPitchedPtr{p, pitch, xs, ys}; }
static inline cudaPos make_cudaPos(size_t x, size_t y, size_t z) { return cudaPos{x, y, z}; }
static inline cudaExtent make_cudaExtent(size_t w, size_t h, size_t d) { return cudaExtent{w, h, d}; }

static inline const char* cudaGetErrorString(cudaError_t e) { return e == cudaSuccess ? "no error" : e == cudaErrorMemoryAllocation ? "out of memory" : "emulated runtime: not supported"; }
static inline cudaError_t cudaGetLastError() { return cudaSuccess; }
static inline cudaError_t cudaGetDeviceCount(int* n) { *n = 1; return cudaSuccess; }
static inline cudaError_t cudaSetDevice(int) { return cudaSuccess; }
static inline cudaError_t cudaGetDeviceProperties(cudaDeviceProp* p, int) {
    memset(p, 0, sizeof *p);
    const char* e = getenv("MCB_EMU_SMS");
    p->multiProcessorCount = e ? atoi(e) : 2;
    strcpy(p->name, "host emulation (tests/emu)");
    return cudaSuccess;
}
/* $MCB_EMU_FENCE=1: every device allocation ends right before an inaccessible page (the end rounded up to 16 bytes only), so
 * that a kernel reading or writing past its buffer faults at the instruction that does it; the handler names the kernel. */
namespace emu {
inline bool fence_on() { static const bool on = [] { const char* e = getenv("MCB_EMU_FENCE"); return e && e[0] == '1'; }(); return on; }
inline const char*& current_kernel() { static const char* k = "(host)"; return k; }
inline std::map<void*, std::pair<void*, size_t>>& fence_map() { static std::map<void*, std::pair<void*, size_t>> m; return m; }
inline std::mutex& fence_mutex() { static std::mutex m; return m; }
inline void fence_handler(int, siginfo_t* si, void*) {
    char b[256];
    const int n = snprintf(b, sizeof b, "\nemulator fence: invalid access at %p in kernel %s\n", si->si_addr, current_kernel());
    if (n > 0) (void)!write(2, b, (size_t)n);
    _exit(99);
}
inline void* fence_alloc(size_t n) {
    static const bool installed = [] {
        static char altstack[1 << 16];
        stack_t ss; ss.ss_sp = altstack; ss.ss_size = sizeof altstack; ss.ss_flags = 0; sigaltstack(&ss, nullptr);
        struct sigaction sa; memset(&sa, 0, sizeof sa); sa.sa_sigaction = fence_handler; sa.sa_flags = SA_SIGINFO | SA_ONSTACK;
        sigaction(SIGSEGV, &sa, nullptr); sigaction(SIGBUS, &sa, nullptr);
        return true; }();
    (void)installed;
    const size_t page = 4096, used = (n + 15) / 16 * 16, body = (used + page - 1) / page * page;
    char* base = (char*)mmap(nullptr, body + page, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (base == (char*)MAP_FAILED) return nullptr;
    mprotect(base + body, page, PROT_NONE);
    void* p = base + (body - used);
    memset(base, 0xA5, body); /* cudaMalloc does not clear: whoever reads before writing gets a wild index, not a convenient zero */
    std::lock_guard<std::mutex> lk(fence_mutex());
    fence_map()[p] = std::make_pair((void*)base, body + page);
    return p;
}
inline bool fence_free(void* p) {
    std::lock_guard<std::mutex> lk(fence_mutex());
    auto it = fence_map().find(p);
    if (it == fence_map().end()) return false;
    munmap(it->second.first, it->second.second);
    fence_map().erase(it);
    return true;
}
/* Allocation accounting for the tests (tests/test_emu_buffers.py): the live allocations, the number of cudaMalloc /
 * cudaMallocHost calls, and a switch that makes the n-th following call fail with cudaErrorMemoryAllocation. */
struct Allocs {
    std::mutex m;
    std::map<void*, size_t> live;
    long long calls = 0, fail_in = 0;
};
inline Allocs& allocs() { static Allocs a; return a; }
} /* namespace emu */
extern "C" __attribute__((used, visibility("default"))) inline void mcb_emu_alloc_stats(long long* live, long long* calls) {
    std::lock_guard<std::mutex> lk(emu::allocs().m);
    *live = (long long)emu::allocs().live.size();
    *calls = emu::allocs().calls;
}
/* n > 0: the n-th cudaMalloc / cudaMallocHost from now on fails (once); 0: none does */
extern "C" __attribute__((used, visibility("default"))) inline void mcb_emu_fail_alloc(long long n) {
    std::lock_guard<std::mutex> lk(emu::allocs().m);
    emu::allocs().fail_in = n;
}
template <class T> static inline cudaError_t cudaMalloc(T** p, size_t n) {
    emu::Allocs& a = emu::allocs();
    std::lock_guard<std::mutex> lk(a.m);
    a.calls++;
    if (a.fail_in > 0 && --a.fail_in == 0) { *p = nullptr; return cudaErrorMemoryAllocation; }
    *p = emu::fence_on() ? (T*)emu::fence_alloc(n) : (T*)aligned_alloc(256, (n + 255) / 256 * 256 + 256);
    if (!*p) return cudaErrorMemoryAllocation;
    a.live[(void*)*p] = n;
    return cudaSuccess;
}
template <class T> static inline cudaError_t cudaMallocHost(T** p, size_t n) { return cudaMalloc(p, n); }
static inline cudaError_t cudaFree(void* p) {
    if (!p) return cudaSuccess;
    {
        std::lock_guard<std::mutex> lk(emu::allocs().m);
        emu::allocs().live.erase(p);
    }
    if (!emu::fence_free(p)) free(p);
    return cudaSuccess;
}
static inline cudaError_t cudaFreeHost(void* p) { return cudaFree(p); }
static inline cudaError_t cudaHostRegister(void*, size_t, unsigned) { return cudaSuccess; }
static inline cudaError_t cudaHostUnregister(void*) { return cudaSuccess; }
static inline cudaError_t cudaMemcpy(void* d, const void* s, size_t n, cudaMemcpyKind) { memmove(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, cudaMemcpyKind, cudaStream_t = nullptr) { memmove(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemsetAsync(void* d, int v, size_t n, cudaStream_t = nullptr) { memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaMemset(void* d, int v, size_t n) { memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaMemcpy3DAsync(const cudaMemcpy3DParms* p, cudaStream_t = nullptr) {
    for (size_t z = 0; z < p->extent.depth; z++)
        for (size_t y = 0; y < p->extent.height; y++) {
            const char* s = (const char*)p->srcPtr.ptr + ((p->srcPos.z + z) * p->srcPtr.ysize + (p->srcPos.y + y)) * p->srcPtr.pitch + p->srcPos.x;
            char* d = (char*)p->dstPtr.ptr + ((p->dstPos.z + z) * p->dstPtr.ysize + (p->dstPos.y + y)) * p->dstPtr.pitch + p->dstPos.x;
            memcpy(d, s, p->extent.width);
        }
    return cudaSuccess;
}
static inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { *s = (cudaStream_t)malloc(8); return cudaSuccess; }
static inline cudaError_t cudaStreamDestroy(cudaStream_t s) { free(s); return cudaSuccess; }
static inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaDeviceSynchronize() { return cudaSuccess; }
static inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned) { return cudaSuccess; }
static inline cudaError_t cudaEventCreate(cudaEvent_t* e) { *e = (cudaEvent_t)malloc(8); return cudaSuccess; }
static inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { return cudaEventCreate(e); }
static inline cudaError_t cudaEventDestroy(cudaEvent_t e) { free(e); return cudaSuccess; }
static inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t = nullptr) { return cudaSuccess; }
static inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return cudaSuccess; }
static inline cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t, cudaEvent_t) { *ms = 0.001f; return cudaSuccess; }
template <class F> static inline cudaError_t cudaFuncSetAttribute(F, cudaFuncAttribute, int) { return cudaSuccess; }
/* run-time compiled kernels need a device: the library falls back to its interpreter kernels (MCB_JIT_AUTO) */
static inline cudaError_t cudaLibraryLoadData(cudaLibrary_t*, const void*, void*, void*, unsigned, void*, void*, unsigned) { return cudaErrorNotSupported; }
static inline cudaError_t cudaLibraryGetKernel(cudaKernel_t*, cudaLibrary_t, const char*) { return cudaErrorNotSupported; }
static inline cudaError_t cudaLibraryUnload(cudaLibrary_t) { return cudaSuccess; }
static inline cudaError_t cudaLaunchKernel(const void*, dim3, dim3, void**, size_t, cudaStream_t) { return cudaErrorNotSupported; }

/* launcher and dynamic shared memory as the product sources spell them (csrc/mcb_launch.h keeps the CUDA forms) */
#define MCB_UNPAREN(...) __VA_ARGS__
#define MCB_LAUNCH(kern, grid, block, smem, stream, ...) \
    do { emu::current_kernel() = #kern; emu::launch(dim3(grid), dim3(block), (size_t)(smem), [&]() { MCB_UNPAREN kern(__VA_ARGS__); }); \
         emu::current_kernel() = "(host)"; } while (0)
#define MCB_DYNAMIC_SMEM(type, name) type* name = reinterpret_cast<type*>(emu::dyn_smem())
