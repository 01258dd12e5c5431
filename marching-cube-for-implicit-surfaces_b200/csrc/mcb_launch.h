/* How the host code launches a kernel and how a kernel names its dynamic shared memory.
 * The product build (nvcc) uses the CUDA forms below.  A test harness may define both before this header is seen
 * (tests/emu/cuda_runtime.h executes the kernels' source on the host for the CPU test tier); nothing in the product
 * build does. */
#ifndef MCB_LAUNCH
#include <cstdio>
#include <cstdlib>
/* $MCB_DEBUG_SYNC=1 (debugging aid, read once): wait for every kernel right after its launch and name the one that
 * failed on stderr — an asynchronous fault is otherwise reported by whatever call synchronises next. */
inline bool mcb_debug_sync_on() {
    static const bool on = [] { const char* e = std::getenv("MCB_DEBUG_SYNC"); return e && e[0] == '1'; }();
    return on;
}
inline void mcb_debug_sync_check(const char* kernel, cudaStream_t stream) {
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) std::fprintf(stderr, "MCB_DEBUG_SYNC: kernel %s: %s\n", kernel, cudaGetErrorString(e));
}
#define MCB_UNPAREN(...) __VA_ARGS__
#define MCB_LAUNCH(kern, grid, block, smem, stream, ...)                                  \
    do {                                                                                  \
        MCB_UNPAREN kern<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);             \
        if (mcb_debug_sync_on()) mcb_debug_sync_check(#kern, (stream));                   \
    } while (0)
/* Programmatic dependent launch: the kernel may be placed on the SMs while its predecessor on the stream is still
 * finishing.  Only for kernels that run MCB_GRID_WAIT() before they touch global memory written earlier in the call
 * (DESIGN.md §5, "The wait rule"); a launch error is left to cudaGetLastError, like that of MCB_LAUNCH. */
#define MCB_LAUNCH_PDL(kern, grid, block, smem, strm, ...)                                \
    do {                                                                                  \
        cudaLaunchAttribute attr_[1];                                                     \
        attr_[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                 \
        attr_[0].val.programmaticStreamSerializationAllowed = 1;                          \
        cudaLaunchConfig_t cfg_ = {};                                                     \
        cfg_.gridDim = dim3(grid);                                                        \
        cfg_.blockDim = dim3(block);                                                      \
        cfg_.dynamicSmemBytes = (smem);                                                   \
        cfg_.stream = (strm);                                                             \
        cfg_.attrs = attr_;                                                               \
        cfg_.numAttrs = 1;                                                                \
        (void)cudaLaunchKernelEx(&cfg_, MCB_UNPAREN kern, __VA_ARGS__);                   \
        if (mcb_debug_sync_on()) mcb_debug_sync_check(#kern, (strm));                     \
    } while (0)
/* griddepcontrol.wait: returns once every grid this one depends on has completed and its memory is visible (at once
 * for a kernel launched without the attribute).  griddepcontrol.launch_dependents: the next grid's blocks may be
 * placed from now on; its own wait still covers this grid's completion. */
#define MCB_GRID_WAIT() asm volatile("griddepcontrol.wait;" ::: "memory")
#define MCB_GRID_DEPENDENTS() asm volatile("griddepcontrol.launch_dependents;" ::: "memory")
#define MCB_DYNAMIC_SMEM(type, name) extern __shared__ type name[]
#endif
/* a harness that brings its own MCB_LAUNCH runs every launch to completion before the next: no overlap to control */
#ifndef MCB_LAUNCH_PDL
#define MCB_LAUNCH_PDL MCB_LAUNCH
#endif
#ifndef MCB_GRID_WAIT
#define MCB_GRID_WAIT() ((void)0)
#endif
#ifndef MCB_GRID_DEPENDENTS
#define MCB_GRID_DEPENDENTS() ((void)0)
#endif
