// Host-side helpers shared by the C-ABI translation units: thread-local error state, the
// cuTensorMapEncodeTiled entry point (resolved at run time so the library links without
// libcuda), and a small cache of encoded TMA descriptors.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>

#include "../../include/cesm_b200.h"

namespace cesm {

int set_error(int code, const char* fmt, ...);
#define CESM_CHECK_CUDA(expr)                                                                  \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess)                                                                 \
            return ::cesm::set_error(CESM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,            \
                                     cudaGetErrorString(_e), __FILE__, __LINE__);              \
    } while (0)
// Every kernel launch goes through this: counts it (cesm_launch_count) and checks the launch.
void note_launch();
#define CESM_CHECK_LAUNCH()            \
    do {                               \
        ::cesm::note_launch();         \
        CESM_CHECK_CUDA(cudaGetLastError()); \
    } while (0)
// Zero a caller-provided scratch / statistics buffer before the kernels that accumulate into it --
// unless the caller has promised (cesm_set_prezeroed_scratch) that such buffers arrive zeroed: the
// training engine carves them from one arena cleared by a single memset per step instead of ~70.
bool scratch_prezeroed();
#define CESM_ZERO_SCRATCH(ptr, bytes, st)                                               \
    do {                                                                                \
        if (!::cesm::scratch_prezeroed()) CESM_CHECK_CUDA(cudaMemsetAsync((ptr), 0, (bytes), (st))); \
    } while (0)
#define CESM_REQUIRE(cond, ...)                                                 \
    do {                                                                        \
        if (!(cond)) return ::cesm::set_error(CESM_ERR_INVALID, __VA_ARGS__);   \
    } while (0)

// Every kernel is launched with the programmatic-stream-serialization attribute: its CTAs may be scheduled
// while the preceding kernel of the stream drains (they park in griddepcontrol.wait, see pdl_wait() in
// common.cuh), which hides launch latency and the CTA ramp between the ~480 back-to-back kernels of a step.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// Same, as thread-block clusters of `cluster_x` CTAs along x (1 = no cluster attribute).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl_cluster(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                      int cluster_x, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    int n = 1;
    if (cluster_x > 1) {
        attr[n].id = cudaLaunchAttributeClusterDimension;
        attr[n].val.clusterDim.x = (unsigned)cluster_x;
        attr[n].val.clusterDim.y = 1;
        attr[n].val.clusterDim.z = 1;
        ++n;
    }
    cfg.attrs = attr;
    cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// Encode (or fetch from the cache) a fp16 tiled tensor map with SWIZZLE_128B.
// dims/strides/box follow cuTensorMapEncodeTiled (dim 0 innermost, strides in bytes for dims >= 1).
int get_tensor_map_h16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                        const uint64_t* strides_bytes, const uint32_t* box);

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

}  // namespace cesm
