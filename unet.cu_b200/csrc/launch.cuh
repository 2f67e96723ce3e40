// Programmatic dependent launch (PDL) for the training path.  Every kernel of the step is launched with
// cudaLaunchAttributeProgrammaticStreamSerialization: the next kernel's CTAs may become resident and run their
// prologue (mbarrier init, TMEM allocation, descriptor prefetch, index math) while the previous kernel drains, and
// block in pdl_wait() until the previous grid has completed and its writes are visible.  In the captured step graph
// the kernel -> kernel edges become programmatic edges, which removes the ~1-2 us launch gap between the ~500 small
// kernels of a step.
//
// Rules every kernel follows: (1) pdl_wait() is executed by EVERY thread before its first access to global memory that
// an earlier kernel may have written, and before any early return; (2) nothing before pdl_wait() touches such memory
// (kernel parameters, including __grid_constant__ tensor maps, are fine).  Launched without the attribute (layer API,
// tools) the griddepcontrol instructions are no-ops.
#pragma once
#include <cuda_runtime.h>

#include <cstdlib>
#include <utility>

namespace ub {

// Where the dependent grid is released (griddepcontrol.launch_dependents), measured with bench.py at B = 32:
// - no PDL 6.87 ms/step, the implicit trigger at grid end 6.62, an entry trigger in every kernel 7.30, an entry
//   trigger only in the forward-pass convs 6.01 against 5.93 without: early-resident CTAs of the next kernel take SM
//   slots, TMEM and shared memory from the kernel that is still draining and from the weight-gradient branch.  The
//   GEMM-shaped kernels therefore trigger late (pdl_trigger_late), the others at entry (pdl_entry).
// - round 2: the entry trigger in the elementwise / normalisation kernels gave 5.09 ms/step against 5.18 without --
//   the launch latency of every kernel that follows a GroupNorm / data-movement kernel was exposed.
// The early-trigger, no-late-trigger and no-entry-trigger variants were measured and removed.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// Late trigger (GEMM-shaped kernels): issued by a CTA once its main loop is complete, so the next kernel's CTAs become
// resident and run their prologue (barrier init, TMEM allocation, descriptor prefetch) under this kernel's epilogue
// and teardown only -- they cannot take resources from a main loop that is still running.
__device__ __forceinline__ void pdl_trigger_late() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// the usual kernel entry (elementwise / normalisation kernels, whose CTAs hold no shared memory or TMEM that an
// early-resident dependent could be starved of): let the dependent grid start early, then wait for our own prerequisite
__device__ __forceinline__ void pdl_entry() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
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
