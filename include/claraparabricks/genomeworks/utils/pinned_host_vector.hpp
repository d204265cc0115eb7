// gw-b200: pinned_host_vector<T> (common/base/include/claraparabricks/genomeworks/utils/pinned_host_vector.hpp:37-38): a
// std::vector whose storage is page-locked host memory (cudaMallocHost), so copies to and from the device can run async.
#pragma once

#include <cuda_runtime_api.h>

#include <cstddef>
#include <new>
#include <vector>

namespace claraparabricks
{
namespace genomeworks
{
namespace details
{

template <typename T>
struct PinnedAllocator
{
    using value_type = T;
    PinnedAllocator() = default;
    template <typename U>
    PinnedAllocator(const PinnedAllocator<U>&)
    {
    }
    T* allocate(std::size_t n)
    {
        void* p = nullptr;
        if (n > 0 && cudaMallocHost(&p, n * sizeof(T)) != cudaSuccess)
        {
            cudaGetLastError();
            throw std::bad_alloc();
        }
        return static_cast<T*>(p);
    }
    void deallocate(T* p, std::size_t)
    {
        if (p)
            cudaFreeHost(p);
    }
    template <typename U>
    bool operator==(const PinnedAllocator<U>&) const
    {
        return true;
    }
    template <typename U>
    bool operator!=(const PinnedAllocator<U>&) const
    {
        return false;
    }
};

} // namespace details

template <typename T>
using pinned_host_vector = std::vector<T, details::PinnedAllocator<T>>;

} // namespace genomeworks
} // namespace claraparabricks
