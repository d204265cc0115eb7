// gw-b200: the CUDA helpers that callers of the kept API use next to Batch / Aligner
// (common/base/include/claraparabricks/genomeworks/utils/cudautils.hpp:40-54,153,196-261; common/base/src/cudautils.cpp:28-100):
// GW_CU_CHECK_ERR / GW_CU_ABORT_ON_ERR, cudautils::find_largest_contiguous_device_memory_section, get_value_from_device,
// set_device_value_async, device_copy_n_async, CudaStream + make_cuda_stream, scoped_device_switch. Header-only, CUDA runtime API only.
#pragma once

#include <cuda_runtime_api.h>

#include <cassert>
#include <cstddef>
#include <cstdint>
#include <cstdlib>
#include <iostream>
#include <limits>
#include <memory>
#include <type_traits>

namespace claraparabricks
{
namespace genomeworks
{
namespace cudautils
{

/// Reports a CUDA runtime error with its location and terminates, as the reference does (cudautils.cpp:75-100).
inline void gpu_assert(cudaError_t code, const char* file, int line)
{
    if (code == cudaSuccess)
        return;
    std::cerr << "GPU Error:: " << cudaGetErrorString(code) << " " << file << " " << line << std::endl;
    std::abort();
}

/// Largest single device allocation that currently succeeds: trial allocations from 99 % of the free memory downwards in 1 %
/// steps (cudautils.cpp:28-73). Returns 0 if nothing can be allocated.
inline std::size_t find_largest_contiguous_device_memory_section()
{
    std::size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess)
    {
        cudaGetLastError();
        return 0;
    }
    for (int percent = 99; percent > 0; percent--)
    {
        const std::size_t bytes = free_b / 100 * static_cast<std::size_t>(percent);
        void* p                 = nullptr;
        if (cudaMalloc(&p, bytes) == cudaSuccess)
        {
            cudaFree(p);
            return bytes;
        }
        cudaGetLastError();
    }
    return 0;
}

/// Copies one value from the device (or any address cudaMemcpy accepts) and waits for the stream (cudautils.hpp:115-121).
template <typename Type>
Type get_value_from_device(const Type* d_ptr, cudaStream_t stream = 0);

/// Copies one value to dst on the stream; src must stay valid until the stream reaches the copy (cudautils.hpp:125-128).
template <typename Type>
void set_device_value_async(Type* dst, const Type* src, cudaStream_t stream);

/// Copies n elements between any two addresses on the stream (cudautils.hpp:139-142).
template <typename Type>
void device_copy_n_async(const Type* src, std::size_t n, Type* dst, cudaStream_t stream);

/// Rounds value up to a multiple of the (power of two) alignment.
template <typename T, int alignment>
inline T align(const T& value)
{
    static_assert(alignment > 0 && (alignment & (alignment - 1)) == 0, "alignment has to be a power of two");
    return (value + static_cast<T>(alignment - 1)) & ~static_cast<T>(alignment - 1);
}

} // namespace cudautils
} // namespace genomeworks
} // namespace claraparabricks

#define GW_CU_CHECK_ERR(ans)                                                            \
    {                                                                                   \
        claraparabricks::genomeworks::cudautils::gpu_assert((ans), __FILE__, __LINE__); \
    }
#define GW_CU_ABORT_ON_ERR(ans)                                                         \
    {                                                                                   \
        claraparabricks::genomeworks::cudautils::gpu_assert((ans), __FILE__, __LINE__); \
    }
// GW_NVTX_RANGE (reference cudautils.hpp:155-184): a scoped NVTX range when the including build defines GW_PROFILING (the
// header-only NVTX v3 that ships with the CUDA toolkit: no extra library to link), otherwise nothing.
#if defined(GW_PROFILING) && defined(__has_include)
#if __has_include(<nvtx3/nvToolsExt.h>)
#include <nvtx3/nvToolsExt.h>
namespace claraparabricks
{
namespace genomeworks
{
namespace cudautils
{
class nvtx_range
{
public:
    explicit nvtx_range(char const* name) { nvtxRangePushA(name); }
    ~nvtx_range() { nvtxRangePop(); }
    nvtx_range(const nvtx_range&) = delete;
    nvtx_range& operator=(const nvtx_range&) = delete;
};
} // namespace cudautils
} // namespace genomeworks
} // namespace claraparabricks
#define GW_NVTX_RANGE(varname, label) ::claraparabricks::genomeworks::cudautils::nvtx_range varname(label)
#endif
#endif
#ifndef GW_NVTX_RANGE
#define GW_NVTX_RANGE(varname, label)
#endif

namespace claraparabricks
{
namespace genomeworks
{
namespace detail
{
struct CudaStreamDeleter
{
    void operator()(cudaStream_t s) const
    {
        if (s)
            GW_CU_ABORT_ON_ERR(cudaStreamDestroy(s));
    }
};
} // namespace detail

namespace cudautils
{
template <typename Type>
Type get_value_from_device(const Type* d_ptr, cudaStream_t stream)
{
    Type val;
    GW_CU_CHECK_ERR(cudaMemcpyAsync(&val, d_ptr, sizeof(Type), cudaMemcpyDefault, stream));
    GW_CU_CHECK_ERR(cudaStreamSynchronize(stream));
    return val;
}

template <typename Type>
void set_device_value_async(Type* dst, const Type* src, cudaStream_t stream)
{
    GW_CU_CHECK_ERR(cudaMemcpyAsync(dst, src, sizeof(Type), cudaMemcpyDefault, stream));
}

template <typename Type>
void device_copy_n_async(const Type* src, std::size_t n, Type* dst, cudaStream_t stream)
{
    GW_CU_CHECK_ERR(cudaMemcpyAsync(dst, src, n * sizeof(Type), cudaMemcpyDefault, stream));
}
} // namespace cudautils

/// Owning handle of a cudaStream_t; create with make_cuda_stream(), pass `.get()` to create_batch / create_aligner.
using CudaStream = std::unique_ptr<std::remove_pointer<cudaStream_t>::type, detail::CudaStreamDeleter>;

inline CudaStream make_cuda_stream()
{
    cudaStream_t native = nullptr;
    GW_CU_CHECK_ERR(cudaStreamCreateWithFlags(&native, cudaStreamNonBlocking));
    return CudaStream(native);
}

/// Makes `device_id` the current device for the enclosing scope and restores the previous one afterwards.
class scoped_device_switch
{
public:
    explicit scoped_device_switch(int32_t device_id)
    {
        GW_CU_CHECK_ERR(cudaGetDevice(&previous_));
        if (previous_ != device_id)
            GW_CU_CHECK_ERR(cudaSetDevice(device_id))
        else
            previous_ = kNoSwitch;
    }
    ~scoped_device_switch()
    {
        if (previous_ != kNoSwitch)
            cudaSetDevice(previous_);
    }
    scoped_device_switch()                            = delete;
    scoped_device_switch(const scoped_device_switch&) = delete;
    scoped_device_switch& operator=(const scoped_device_switch&) = delete;

private:
    static constexpr int32_t kNoSwitch = std::numeric_limits<int32_t>::max();
    int32_t previous_;
};

} // namespace genomeworks
} // namespace claraparabricks
