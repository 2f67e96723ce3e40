// Programmatic dependent launch (PDL) for the training path.  Every kernel of the step is launched with
// cudaLaunchAttributeProgrammaticStreamSerialization: the next kernel's CTAs may become resident and run their
// prologue (mbarrier init, TMEM allocation, descriptor prefetch, index math) while the previous kernel drains, and
// block in pdl_wait() until the previous grid has completed and its writes are visible.  In the captured step graph
// the kernel -> kernel edges become programmatic edges, which removes the ~1-2 us launch gap between the ~500 small
// kernels of a step.
//
// Rules every kernel follows: (1) pdl_trigger() then pdl_wait() are executed by EVERY thread before its first access
// to global memory that an earlier kernel may have written, and before any early return; (2) nothing before
// pdl_wait() touches such memory (kernel parameters, including __grid_constant__ tensor maps, are fine).
// Launched without the attribute (layer API, tools) both instructions are no-ops.
#pragma once
#include <cuda_runtime.h>

#include <cstdlib>
#include <utility>

namespace ub {

__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// Measured (bench.py, B=32): no PDL 6.87 ms/step, implicit trigger 6.62, early trigger in every kernel 7.30, early
// trigger only in the forward-pass convs 6.01 vs 5.93 without -- early-resident CTAs of the next kernel take SM slots,
// TMEM and shared memory from the kernel that is still draining and from the weight-gradient branch.
#ifndef UB_PDL_EARLY_TRIGGER
#define UB_PDL_EARLY_TRIGGER 0
#endif
__device__ __forceinline__ void pdl_trigger() {
#if UB_PDL_EARLY_TRIGGER
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}
// Late trigger (GEMM-shaped kernels): issued by a CTA once its main loop is complete, so the next kernel's CTAs become
// resident and run their prologue (barrier init, TMEM allocation, descriptor prefetch) under this kernel's epilogue
// and teardown only -- they cannot take resources from a main loop that is still running.
#ifndef UB_PDL_LATE_TRIGGER
#define UB_PDL_LATE_TRIGGER 1
#endif
__device__ __forceinline__ void pdl_trigger_late() {
#if UB_PDL_LATE_TRIGGER
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}
// the usual kernel entry: let the dependent grid start early, then wait for our own prerequisite
// (UB_PDL_ELT_EARLY: entry trigger only in the elementwise / normalisation kernels, whose CTAs hold no shared memory
//  or TMEM that an early-resident dependent could be starved of.  Measured round 2, bench.py B = 32: 5.09 ms/step with,
//  5.18 without -- the launch latency of every kernel that follows a GroupNorm / data-movement kernel was exposed.)
#ifndef UB_PDL_ELT_EARLY
#define UB_PDL_ELT_EARLY 1
#endif
__device__ __forceinline__ void pdl_entry() {
#if UB_PDL_ELT_EARLY
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#else
    pdl_trigger();
#endif
    pdl_wait();
}

// SMs of the current device (148 on a B200), queried once: grid-size heuristics only, never correctness
inline int sm_count() {
    static const int n = [] {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0)
            v = 148;
        return v;
    }();
    return n;
}

inline bool pdl_enabled() {
    static const bool on = !(getenv("UB_NO_PDL") && atoi(getenv("UB_NO_PDL")) != 0);
    return on;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at, cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

}  // namespace ub
