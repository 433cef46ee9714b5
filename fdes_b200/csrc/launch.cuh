// fdes_b200 -- the one way the library checks a CUDA call and launches a kernel.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <stdexcept>
#include <string>
#include <utility>

namespace fdes {

// CUDA errors become exceptions (capi.cu turns them into return codes / fdes_b200_last_error())
#define CK(x)                                                                                    \
    do {                                                                                         \
        const cudaError_t e_ = (x);                                                              \
        if (e_ != cudaSuccess)                                                                   \
            throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(e_) +      \
                                     " at " + __FILE__ + ":" + std::to_string(__LINE__));        \
    } while (0)

// Kernels this host thread has launched through launch() / launch_pdl() (defined in sweeps.cu).  The engine reports
// its growth over each of its calls as EngineTimings::kernel_launches; the launches it captures into a CUDA graph it
// takes back out and counts at every launch of the graph (Engine::slice_loop).
extern thread_local long long launch_tally;

// Launches kernel(args) and adds 1 to launch_tally.  Dynamic shared memory beyond the 48 KB default is opted in
// first, per kernel and device, up to the largest size requested so far.  A launch the driver refuses throws,
// naming the kernel.  pdl: programmatic stream serialisation (launch_pdl).
void launch_args(const void* kernel, dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, void** args);

template <class... KArgs, class... Args>
void launch_as(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args)
{
    // the arguments converted to the kernel's parameter types, as a triple-chevron launch converts them
    [&](KArgs... a) {
        void* p[] = {&a..., nullptr};
        launch_args(reinterpret_cast<const void*>(kernel), grid, block, smem, st, pdl, p);
    }(std::forward<Args>(args)...);
}

// A plain launch: the kernel starts after everything queued before it on st has finished.
template <class... KArgs, class... Args>
void launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args)
{
    launch_as(false, kernel, grid, block, smem, st, std::forward<Args>(args)...);
}

// Programmatic dependent launch, for the sweeps of the slice loop (about sixty dependent launches per batch): the
// sweep is launched with programmatic stream serialisation, signals at its very start that its dependents may be
// scheduled, and waits for its own prerequisites before it touches memory (pdl_prologue, sweep_kernels.cuh).  The
// CTAs of sweep i+1 are then resident (index arithmetic, barrier set-up done) when the last CTAs of sweep i drain,
// instead of being launched after the grid has completed.  Only for kernels that begin with pdl_prologue(): any
// other kernel would read its inputs before the previous one has finished.
template <class... KArgs, class... Args>
void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args)
{
    launch_as(true, kernel, grid, block, smem, st, std::forward<Args>(args)...);
}

}  // namespace fdes
