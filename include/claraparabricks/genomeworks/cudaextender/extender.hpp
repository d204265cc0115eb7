// gw-b200: cudaextender::SeedPair / ScoredSegmentPair / Extender / create_extender with the reference's signatures
// (cudaextender/include/claraparabricks/genomeworks/cudaextender/extender.hpp:36-154), as a header-only adapter over the C ABI
// of libgwb200.so. Every device buffer of the extender is a block of the caller's allocator.
#pragma once

#include "cudaextender.hpp"
#include "../types.hpp"
#include "../utils/allocator.hpp"

#include <cuda_runtime_api.h>

#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

namespace claraparabricks
{
namespace genomeworks
{
namespace cudaextender
{

/// Seed positions in target and query reads (the layout is ABI: device-API callers pass arrays of these)
struct SeedPair
{
    /// position of first sketch element in query_read_id_
    position_in_read_t query_position_in_read;
    /// position of second sketch element in target_read_id_
    position_in_read_t target_position_in_read;
};

/// Segment pairs in target & query reads with associated length & score
struct ScoredSegmentPair
{
    /// leftmost coordinate for the segment
    SeedPair start_coord;
    /// length of the segment (one less than the number of bases it covers)
    int32_t length;
    /// score of the segment
    int32_t score;
};

static_assert(sizeof(SeedPair) == sizeof(gwb200_seed_pair), "SeedPair layout");
static_assert(sizeof(ScoredSegmentPair) == sizeof(gwb200_scored_segment_pair), "ScoredSegmentPair layout");

/// Equality operator for ScoredSegmentPair
inline bool operator==(const ScoredSegmentPair& x, const ScoredSegmentPair& y)
{
    return x.start_coord.target_position_in_read == y.start_coord.target_position_in_read &&
           x.start_coord.query_position_in_read == y.start_coord.query_position_in_read && x.length == y.length && x.score == y.score;
}

/// CUDA Extender Class
class Extender
{
public:
    virtual ~Extender() = default;

    /// Host pointer API: copies the encoded sequences and the seeds to the device and extends them on the extender's stream.
    virtual StatusType extend_async(const int8_t* h_query, int32_t query_length, const int8_t* h_target, int32_t target_length,
                                    int32_t score_threshold, const std::vector<SeedPair>& h_seed_pairs) = 0;

    /// Device pointer API: inputs resident on the device, d_scored_segment_pairs holds num_seed_pairs entries.
    virtual StatusType extend_async(const int8_t* d_query, int32_t query_length, const int8_t* d_target, int32_t target_length,
                                    int32_t score_threshold, const SeedPair* d_seed_pairs, int32_t num_seed_pairs,
                                    ScoredSegmentPair* d_scored_segment_pairs, int32_t* d_num_scored_segment_pairs) = 0;

    /// Waits for the host pointer API call and fetches its results; invalid_operation without one.
    virtual StatusType sync() = 0;

    /// Results of the last host pointer API call (after sync()); std::runtime_error without one.
    virtual const std::vector<ScoredSegmentPair>& get_scored_segment_pairs() const = 0;

    /// Forgets the results of the host pointer API.
    virtual void reset() = 0;
};

namespace detail
{

inline int check(int rc)
{
    if (rc >= 0)
        return rc;
    const std::string msg = gwb200_last_error();
    if (rc == GWB200_E_BAD_ALLOC)
        throw device_memory_allocation_exception();
    if (rc == GWB200_E_INVALID_ARGUMENT)
        throw std::invalid_argument(msg);
    throw std::runtime_error(msg);
}

class UngappedXDropB200 : public Extender
{
public:
    UngappedXDropB200(const int32_t* h_score_mat, int32_t score_mat_dim, int32_t xdrop_threshold, bool no_entropy, cudaStream_t stream,
                      int32_t device_id, DefaultDeviceAllocator allocator, ExtensionType type)
        : stream_(stream)
        , allocator_(allocator)
    {
        check(gwb200_extender_create(&h_, h_score_mat, score_mat_dim, xdrop_threshold, no_entropy ? 1 : 0, stream, device_id,
                                     static_cast<int32_t>(type), &UngappedXDropB200::pool_alloc, &UngappedXDropB200::pool_free, this));
    }
    ~UngappedXDropB200() override { gwb200_extender_destroy(h_); }
    UngappedXDropB200(const UngappedXDropB200&) = delete;
    UngappedXDropB200& operator=(const UngappedXDropB200&) = delete;

    StatusType extend_async(const int8_t* h_query, int32_t query_length, const int8_t* h_target, int32_t target_length, int32_t score_threshold,
                            const std::vector<SeedPair>& h_seed_pairs) override
    {
        results_.clear();
        return static_cast<StatusType>(check(gwb200_extender_extend_host(h_, h_query, query_length, h_target, target_length, score_threshold,
                                                                         reinterpret_cast<const gwb200_seed_pair*>(h_seed_pairs.data()),
                                                                         static_cast<int32_t>(h_seed_pairs.size()))));
    }

    StatusType extend_async(const int8_t* d_query, int32_t query_length, const int8_t* d_target, int32_t target_length, int32_t score_threshold,
                            const SeedPair* d_seed_pairs, int32_t num_seed_pairs, ScoredSegmentPair* d_scored_segment_pairs,
                            int32_t* d_num_scored_segment_pairs) override
    {
        return static_cast<StatusType>(check(gwb200_extender_extend_device(
            h_, d_query, query_length, d_target, target_length, score_threshold, reinterpret_cast<const gwb200_seed_pair*>(d_seed_pairs),
            num_seed_pairs, reinterpret_cast<gwb200_scored_segment_pair*>(d_scored_segment_pairs), d_num_scored_segment_pairs)));
    }

    StatusType sync() override
    {
        const int rc = check(gwb200_extender_sync(h_));
        if (rc == success)
        {
            results_.resize(static_cast<std::size_t>(check(static_cast<int>(gwb200_extender_num_results(h_)))));
            if (!results_.empty())
                gwb200_extender_get_results(h_, reinterpret_cast<gwb200_scored_segment_pair*>(results_.data()),
                                            static_cast<int64_t>(results_.size()));
        }
        return static_cast<StatusType>(rc);
    }

    const std::vector<ScoredSegmentPair>& get_scored_segment_pairs() const override
    {
        if (gwb200_extender_num_results(h_) < 0)
            throw std::runtime_error("Invalid API call. Getting scored segment pairs without calling extend_async host ptr API");
        return results_;
    }

    void reset() override
    {
        results_.clear();
        check(gwb200_extender_reset(h_));
    }

private:
    static void* pool_alloc(void* user, int64_t bytes)
    {
        UngappedXDropB200* self = static_cast<UngappedXDropB200*>(user);
        try
        {
            return self->allocator_.allocate(static_cast<std::size_t>(bytes), {self->stream_});
        }
        catch (const device_memory_allocation_exception&)
        {
            return nullptr;
        }
    }
    static void pool_free(void* user, void* ptr, int64_t bytes)
    {
        static_cast<UngappedXDropB200*>(user)->allocator_.deallocate(static_cast<char*>(ptr), static_cast<std::size_t>(bytes));
    }

    gwb200_extender* h_ = nullptr;
    cudaStream_t stream_;
    DefaultDeviceAllocator allocator_;
    std::vector<ScoredSegmentPair> results_;
};

} // namespace detail

/// Create Extender object (extender.hpp:147-154). Another ExtensionType throws std::runtime_error; a score matrix of fewer than
/// 64 entries throws std::invalid_argument.
inline std::unique_ptr<Extender> create_extender(const int32_t* h_score_mat, int32_t score_mat_dim, int32_t xdrop_threshold, bool no_entropy,
                                                 cudaStream_t stream, int32_t device_id, DefaultDeviceAllocator allocator,
                                                 ExtensionType type = ExtensionType::ungapped_xdrop)
{
    return std::unique_ptr<Extender>(
        new detail::UngappedXDropB200(h_score_mat, score_mat_dim, xdrop_threshold, no_entropy, stream, device_id, allocator, type));
}

} // namespace cudaextender
} // namespace genomeworks
} // namespace claraparabricks
