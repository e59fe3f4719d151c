// Programmatic dependent launch for the chains of short dependent kernels of this library.
#pragma once
#include <cuda_runtime.h>

namespace pnode {
namespace pdl {

// Programmatic dependent launch (griddepcontrol): a kernel launched through launch_pdl may start -- be scheduled, set up its
// barriers / tensor memory / shared memory -- while its predecessor in the stream is still running; it must execute pdl_wait()
// before touching global memory (the predecessor's writes are complete and visible after it).  Every kernel calls
// pdl_launch_dependents() first thing so that ITS successor can do the same.  The SINODE pass is ~250 short dependent launches
// (products of 70-130 us, slicings of 2-20 us): the overlap of each launch's ramp-up with its predecessor's tail is what this
// buys.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr, cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

}  // namespace pdl
}  // namespace pnode
