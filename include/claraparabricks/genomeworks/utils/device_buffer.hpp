// gw-b200: device_buffer<T> (common/base/include/claraparabricks/genomeworks/utils/device_buffer.hpp:37-224): an owning,
// movable array of trivially copyable T in device memory, taken from a DefaultDeviceAllocator and given back on destruction.
#pragma once

#include "allocator.hpp"

#include <cstddef>
#include <type_traits>
#include <utility>
#include <vector>

namespace claraparabricks
{
namespace genomeworks
{

template <typename T>
class device_buffer
{
    static_assert(std::is_trivially_copyable<T>::value, "device_buffer only holds trivially copyable types");

public:
    using value_type     = T;
    using size_type      = std::ptrdiff_t;
    using iterator       = T*;
    using const_iterator = const T*;
    using allocator_type = DefaultDeviceAllocator;

    /// n elements from `allocator`; the block is associated with `streams` (the allocator's default stream if none)
    template <typename... Streams>
    explicit device_buffer(size_type n = 0, DefaultDeviceAllocator allocator = DefaultDeviceAllocator(), Streams... streams)
        : size_(n)
        , allocator_(allocator)
        , streams_{streams...}
    {
        if (size_ > 0)
            data_ = reinterpret_cast<T*>(allocator_.allocate(static_cast<std::size_t>(size_) * sizeof(T), streams_));
    }
    template <typename... Streams>
    explicit device_buffer(DefaultDeviceAllocator allocator, Streams... streams)
        : device_buffer(0, allocator, streams...)
    {
    }
    device_buffer(const device_buffer&) = delete;
    device_buffer& operator=(const device_buffer&) = delete;
    device_buffer(device_buffer&& rhs) noexcept
        : data_(std::exchange(rhs.data_, nullptr))
        , size_(std::exchange(rhs.size_, 0))
        , allocator_(rhs.allocator_)
        , streams_(std::move(rhs.streams_))
    {
    }
    device_buffer& operator=(device_buffer&& rhs) noexcept
    {
        if (this != &rhs)
        {
            free();
            data_      = std::exchange(rhs.data_, nullptr);
            size_      = std::exchange(rhs.size_, 0);
            allocator_ = rhs.allocator_;
            streams_   = std::move(rhs.streams_);
        }
        return *this;
    }
    ~device_buffer() { free(); }

    T* data() { return data_; }
    const T* data() const { return data_; }
    size_type size() const { return size_; }
    iterator begin() { return data_; }
    const_iterator begin() const { return data_; }
    iterator end() { return data_ + size_; }
    const_iterator end() const { return data_ + size_; }
    allocator_type get_allocator() const { return allocator_; }

    /// Gives the memory back to the allocator.
    void free()
    {
        if (data_)
            allocator_.deallocate(reinterpret_cast<char*>(data_), static_cast<std::size_t>(size_) * sizeof(T));
        data_ = nullptr;
        size_ = 0;
    }
    /// Drops the contents and holds new_size elements.
    void clear_and_resize(size_type new_size)
    {
        if (new_size == size_)
            return;
        free();
        size_ = new_size;
        if (size_ > 0)
            data_ = reinterpret_cast<T*>(allocator_.allocate(static_cast<std::size_t>(size_) * sizeof(T), streams_));
    }

private:
    T* data_   = nullptr;
    size_type size_ = 0;
    DefaultDeviceAllocator allocator_;
    std::vector<cudaStream_t> streams_;
};

} // namespace genomeworks
} // namespace claraparabricks
