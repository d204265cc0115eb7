// gw-b200: host engine + C ABI for the ungapped X-drop extender (include/gwb200.h names the reference interface each entry
// replaces). Host behaviour follows cudaextender/src/ungapped_xdrop.cu:50-253 (status codes, host/device API modes, reset);
// scratch memory is sized per call from the caller's allocator instead of a fixed share of the device memory.
// The extension is this repo's kernel (extender_kernels.cuh); the kept segments are ordered with CUB radix sort passes and
// compacted with CUB's flagged select, all stream ordered. No CPU fallback.

#include "../../include/gwb200.h"
#include "common.cuh"
#include "extender_kernels.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>

#include <algorithm>
#include <vector>

using namespace gwb200;
using namespace gwb200::extender;

static_assert(sizeof(gwb200_seed_pair) == 8 && sizeof(Seed) == 8, "SeedPair is 8 bytes");
static_assert(sizeof(gwb200_scored_segment_pair) == 16 && sizeof(Segment) == 16, "ScoredSegmentPair is 16 bytes");

namespace
{

// One device block, from cudaMalloc or from the caller's allocator; grows to the largest call seen.
struct Block
{
    void* p       = nullptr;
    int64_t bytes = 0;
};

} // namespace

struct gwb200_extender
{
    int32_t device_id   = 0;
    cudaStream_t stream = nullptr;
    int32_t xdrop       = 0;
    int32_t no_entropy  = 0;
    int32_t n_sms       = 0;
    gwb200_device_alloc_fn alloc_fn = nullptr;
    gwb200_device_free_fn free_fn   = nullptr;
    void* user                      = nullptr;

    Block score_mat;            // 64 x int32
    Block scratch;              // per-call working memory
    Block h_query, h_target, h_seeds, h_out; // device copies for the host pointer API
    int32_t* pinned   = nullptr; // [0] kept count, [1] result count
    unsigned long long* pinned_positions = nullptr;

    bool host_mode = false;
    int32_t h_num_seeds = 0;
    std::vector<gwb200_scored_segment_pair> results;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timed      = false;
    unsigned long long* d_positions = nullptr; // inside scratch
};

namespace
{

void release(gwb200_extender* e, Block& b)
{
    if (b.p)
    {
        if (e->free_fn)
            e->free_fn(e->user, b.p, b.bytes);
        else
            cudaFree(b.p);
    }
    b.p     = nullptr;
    b.bytes = 0;
}

// Makes b hold at least `bytes`; false when the allocator (or the device) cannot serve it.
bool ensure(gwb200_extender* e, Block& b, int64_t bytes)
{
    bytes = std::max<int64_t>(bytes, 256);
    if (b.bytes >= bytes)
        return true;
    cudaStreamSynchronize(e->stream); // earlier work of this extender may still use the old block
    release(e, b);
    void* p = nullptr;
    if (e->alloc_fn)
        p = e->alloc_fn(e->user, bytes);
    else if (cudaMalloc(&p, bytes) != cudaSuccess)
    {
        cudaGetLastError();
        p = nullptr;
    }
    if (!p)
        return false;
    b.p     = p;
    b.bytes = bytes;
    return true;
}

int64_t align256(int64_t x) { return (x + 255) & ~int64_t(255); }

int grid_for(int64_t n, int threads, int n_sms)
{
    const int64_t blocks = (n + threads - 1) / threads;
    return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(blocks, int64_t(n_sms) * 8)));
}

int extend_device(gwb200_extender* e, const int8_t* d_query, int32_t query_length, const int8_t* d_target, int32_t target_length,
                  int32_t score_threshold, const gwb200_seed_pair* d_seed_pairs, int32_t num_seed_pairs,
                  gwb200_scored_segment_pair* d_out, int32_t* d_num_out)
{
    if (d_query == nullptr || d_target == nullptr || d_seed_pairs == nullptr)
        return set_error(GWB200_EXT_INVALID_INPUT, "Invalid input pointers");
    if (d_out == nullptr || d_num_out == nullptr)
        return set_error(GWB200_EXT_INVALID_INPUT, "Invalid output pointers");
    DeviceGuard guard(e->device_id);
    const int64_t n = std::max<int32_t>(num_seed_pairs, 0);
    e->timed        = false;
    e->pinned_positions[0] = 0;
    if (n == 0)
    {
        GWB200_CUDA_TRY(cudaMemsetAsync(d_num_out, 0, sizeof(int32_t), e->stream));
        return GWB200_EXT_SUCCESS;
    }
    // scratch: counters | kept segments | sorted segments | keys in / out | head flags | CUB temporary storage
    Segment* segs = static_cast<Segment*>(nullptr);
    size_t sort_bytes = 0, select_bytes = 0;
    GWB200_CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, static_cast<const uint64_t*>(nullptr), static_cast<uint64_t*>(nullptr),
                                                    static_cast<const Segment*>(nullptr), segs, static_cast<int>(n), 0, 64, e->stream));
    GWB200_CUDA_TRY(cub::DeviceSelect::Flagged(nullptr, select_bytes, static_cast<const Segment*>(nullptr), static_cast<const uint8_t*>(nullptr),
                                               reinterpret_cast<Segment*>(d_out), d_num_out, static_cast<int>(n), e->stream));
    const int64_t off_kept  = 256;
    const int64_t off_alt   = off_kept + align256(n * 16);
    const int64_t off_k0    = off_alt + align256(n * 16);
    const int64_t off_k1    = off_k0 + align256(n * 8);
    const int64_t off_flags = off_k1 + align256(n * 8);
    const int64_t off_temp  = off_flags + align256(n);
    const int64_t total     = off_temp + align256(static_cast<int64_t>(std::max(sort_bytes, select_bytes)));
    if (!ensure(e, e->scratch, total))
        return set_error(GWB200_E_BAD_ALLOC, "Could not allocate device memory for the extension scratch space");
    char* base          = static_cast<char*>(e->scratch.p);
    int32_t* counters   = reinterpret_cast<int32_t*>(base);                      // [0] kept, [1] next seed
    e->d_positions      = reinterpret_cast<unsigned long long*>(base + 64);
    Segment* kept       = reinterpret_cast<Segment*>(base + off_kept);
    Segment* alt        = reinterpret_cast<Segment*>(base + off_alt);
    uint64_t* k0        = reinterpret_cast<uint64_t*>(base + off_k0);
    uint64_t* k1        = reinterpret_cast<uint64_t*>(base + off_k1);
    uint8_t* flags      = reinterpret_cast<uint8_t*>(base + off_flags);
    void* temp          = base + off_temp;

    GWB200_CUDA_TRY(cudaMemsetAsync(base, 0, 128, e->stream));
    GWB200_CUDA_TRY(cudaEventRecord(e->ev0, e->stream));
    ExtendParams P;
    P.target          = d_target;
    P.target_length   = target_length;
    P.query           = d_query;
    P.query_length    = query_length;
    P.score_mat       = static_cast<const int32_t*>(e->score_mat.p);
    P.xdrop           = e->xdrop;
    P.score_threshold = score_threshold;
    P.no_entropy      = e->no_entropy;
    P.seeds           = reinterpret_cast<const Seed*>(d_seed_pairs);
    P.num_seeds       = static_cast<int32_t>(n);
    P.kept            = kept;
    P.num_kept        = counters;
    P.next_seed       = counters + 1;
    P.positions       = e->d_positions;
    const int warps_needed = static_cast<int>((n + kSeedsPerGrab - 1) / kSeedsPerGrab);
    int blocks_per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, ungapped_xdrop_kernel, kWarpsPerBlock * 32, 0);
    const int grid = std::max(1, std::min(e->n_sms * std::max(blocks_per_sm, 1), (warps_needed + kWarpsPerBlock - 1) / kWarpsPerBlock));
    ungapped_xdrop_kernel<<<grid, kWarpsPerBlock * 32, 0, e->stream>>>(P);
    count_launch();
    GWB200_CUDA_TRY(cudaGetLastError());
    // the one read-back of the call (the reference reads its inclusive-scan total at the same point, ungapped_xdrop.cu:146)
    GWB200_CUDA_TRY(cudaMemcpyAsync(e->pinned, counters, sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    GWB200_CUDA_TRY(cudaMemcpyAsync(e->pinned_positions, e->d_positions, sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->stream));
    GWB200_CUDA_TRY(cudaStreamSynchronize(e->stream));
    const int32_t k = e->pinned[0];
    if (k > 0)
    {
        const int threads = 256;
        const int g       = grid_for(k, threads, e->n_sms);
        minor_keys_kernel<<<g, threads, 0, e->stream>>>(kept, k, k0);
        count_launch();
        size_t tb = sort_bytes;
        GWB200_CUDA_TRY(cub::DeviceRadixSort::SortPairs(temp, tb, k0, k1, kept, alt, k, 0, 64, e->stream));
        count_launch();
        major_keys_kernel<<<g, threads, 0, e->stream>>>(alt, k, k0);
        count_launch();
        tb = sort_bytes;
        GWB200_CUDA_TRY(cub::DeviceRadixSort::SortPairs(temp, tb, k0, k1, alt, kept, k, 0, 64, e->stream));
        count_launch();
        head_flags_kernel<<<g, threads, 0, e->stream>>>(kept, k, flags);
        count_launch();
        size_t sb = select_bytes;
        GWB200_CUDA_TRY(cub::DeviceSelect::Flagged(temp, sb, kept, flags, reinterpret_cast<Segment*>(d_out), d_num_out, k, e->stream));
        count_launch();
        GWB200_CUDA_TRY(cudaGetLastError());
    }
    else
    {
        GWB200_CUDA_TRY(cudaMemsetAsync(d_num_out, 0, sizeof(int32_t), e->stream));
    }
    GWB200_CUDA_TRY(cudaEventRecord(e->ev1, e->stream));
    e->timed = true;
    return GWB200_EXT_SUCCESS;
}

} // namespace

extern "C" {

int gwb200_extender_create(gwb200_extender** out, const int32_t* h_score_mat, int32_t score_mat_dim, int32_t xdrop_threshold,
                           int32_t no_entropy, void* stream, int32_t device_id, int32_t type, gwb200_device_alloc_fn alloc_fn,
                           gwb200_device_free_fn free_fn, void* user)
{
    if (!out)
        return set_error(GWB200_E_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    if (type != GWB200_EXT_UNGAPPED_XDROP)
        return set_error(GWB200_E_RUNTIME, "Extender for specified type not implemented yet.");
    if (!h_score_mat || score_mat_dim < 64)
        return set_error(GWB200_E_INVALID_ARGUMENT, "the score matrix must hold 8 x 8 = 64 entries");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device_id < 0 || ndev <= device_id)
    {
        cudaGetLastError();
        return set_error(GWB200_E_CUDA, "no usable CUDA device: this engine has no CPU fallback");
    }
    DeviceGuard guard(device_id);
    gwb200_extender* e = new gwb200_extender;
    e->device_id       = device_id;
    e->stream          = static_cast<cudaStream_t>(stream);
    e->xdrop           = xdrop_threshold;
    e->no_entropy      = no_entropy ? 1 : 0;
    if (alloc_fn && free_fn)
    {
        e->alloc_fn = alloc_fn;
        e->free_fn  = free_fn;
        e->user     = user;
    }
    cudaDeviceGetAttribute(&e->n_sms, cudaDevAttrMultiProcessorCount, device_id);
    if (cudaEventCreate(&e->ev0) != cudaSuccess || cudaEventCreate(&e->ev1) != cudaSuccess ||
        cudaHostAlloc(reinterpret_cast<void**>(&e->pinned), 2 * sizeof(int32_t), cudaHostAllocDefault) != cudaSuccess ||
        cudaHostAlloc(reinterpret_cast<void**>(&e->pinned_positions), sizeof(unsigned long long), cudaHostAllocDefault) != cudaSuccess)
    {
        cudaGetLastError();
        gwb200_extender_destroy(e);
        return set_error(GWB200_E_CUDA, "CUDA initialisation of the extender failed");
    }
    e->pinned_positions[0] = 0;
    if (!ensure(e, e->score_mat, 64 * sizeof(int32_t)))
    {
        gwb200_extender_destroy(e);
        return set_error(GWB200_E_BAD_ALLOC, "Could not allocate device memory for the score matrix");
    }
    if (cudaMemcpyAsync(e->score_mat.p, h_score_mat, 64 * sizeof(int32_t), cudaMemcpyHostToDevice, e->stream) != cudaSuccess ||
        cudaStreamSynchronize(e->stream) != cudaSuccess)
    {
        cudaGetLastError();
        gwb200_extender_destroy(e);
        return set_error(GWB200_E_CUDA, "copying the score matrix failed");
    }
    *out = e;
    return 0;
}

void gwb200_extender_destroy(gwb200_extender* e)
{
    if (!e)
        return;
    DeviceGuard guard(e->device_id);
    cudaStreamSynchronize(e->stream);
    for (Block* b : {&e->score_mat, &e->scratch, &e->h_query, &e->h_target, &e->h_seeds, &e->h_out})
        release(e, *b);
    if (e->pinned)
        cudaFreeHost(e->pinned);
    if (e->pinned_positions)
        cudaFreeHost(e->pinned_positions);
    if (e->ev0)
        cudaEventDestroy(e->ev0);
    if (e->ev1)
        cudaEventDestroy(e->ev1);
    delete e;
}

int gwb200_extender_extend_device(gwb200_extender* e, const int8_t* d_query, int32_t query_length, const int8_t* d_target,
                                  int32_t target_length, int32_t score_threshold, const gwb200_seed_pair* d_seed_pairs,
                                  int32_t num_seed_pairs, gwb200_scored_segment_pair* d_out, int32_t* d_num_out)
{
    if (!e)
        return set_error(GWB200_E_INVALID_ARGUMENT, "null extender");
    return extend_device(e, d_query, query_length, d_target, target_length, score_threshold, d_seed_pairs, num_seed_pairs, d_out, d_num_out);
}

int gwb200_extender_extend_host(gwb200_extender* e, const int8_t* h_query, int32_t query_length, const int8_t* h_target,
                                int32_t target_length, int32_t score_threshold, const gwb200_seed_pair* h_seed_pairs,
                                int32_t num_seed_pairs)
{
    if (!e)
        return set_error(GWB200_E_INVALID_ARGUMENT, "null extender");
    if ((query_length > 0 && !h_query) || (target_length > 0 && !h_target) || (num_seed_pairs > 0 && !h_seed_pairs) || query_length < 0 ||
        target_length < 0)
        return set_error(GWB200_E_INVALID_ARGUMENT, "null host input");
    gwb200_extender_reset(e);
    e->host_mode   = true;
    e->h_num_seeds = std::max<int32_t>(num_seed_pairs, 0);
    DeviceGuard guard(e->device_id);
    const int64_t n = e->h_num_seeds;
    if (!ensure(e, e->h_query, query_length) || !ensure(e, e->h_target, target_length) || !ensure(e, e->h_seeds, n * 8) ||
        !ensure(e, e->h_out, n * 16 + 256))
        return set_error(GWB200_E_BAD_ALLOC, "Could not allocate device memory for the extension inputs");
    if (query_length > 0)
        GWB200_CUDA_TRY(cudaMemcpyAsync(e->h_query.p, h_query, query_length, cudaMemcpyHostToDevice, e->stream));
    if (target_length > 0)
        GWB200_CUDA_TRY(cudaMemcpyAsync(e->h_target.p, h_target, target_length, cudaMemcpyHostToDevice, e->stream));
    if (n > 0)
        GWB200_CUDA_TRY(cudaMemcpyAsync(e->h_seeds.p, h_seed_pairs, n * 8, cudaMemcpyHostToDevice, e->stream));
    char* out = static_cast<char*>(e->h_out.p);
    return extend_device(e, static_cast<const int8_t*>(e->h_query.p), query_length, static_cast<const int8_t*>(e->h_target.p), target_length,
                         score_threshold, static_cast<const gwb200_seed_pair*>(e->h_seeds.p), num_seed_pairs,
                         reinterpret_cast<gwb200_scored_segment_pair*>(out + 256), reinterpret_cast<int32_t*>(out));
}

int gwb200_extender_sync(gwb200_extender* e)
{
    if (!e)
        return set_error(GWB200_E_INVALID_ARGUMENT, "null extender");
    if (!e->host_mode)
        return GWB200_EXT_INVALID_OPERATION;
    DeviceGuard guard(e->device_id);
    char* out = static_cast<char*>(e->h_out.p);
    GWB200_CUDA_TRY(cudaMemcpyAsync(e->pinned + 1, out, sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    GWB200_CUDA_TRY(cudaStreamSynchronize(e->stream));
    const int32_t k = e->pinned[1];
    e->results.resize(std::max(k, 0));
    if (k > 0)
    {
        GWB200_CUDA_TRY(cudaMemcpyAsync(e->results.data(), out + 256, static_cast<size_t>(k) * 16, cudaMemcpyDeviceToHost, e->stream));
        GWB200_CUDA_TRY(cudaStreamSynchronize(e->stream));
    }
    return GWB200_EXT_SUCCESS;
}

int64_t gwb200_extender_num_results(const gwb200_extender* e)
{
    if (!e || !e->host_mode)
        return set_error(GWB200_E_RUNTIME, "Invalid API call. Getting scored segment pairs without calling extend_async host ptr API");
    return static_cast<int64_t>(e->results.size());
}

int64_t gwb200_extender_get_results(const gwb200_extender* e, gwb200_scored_segment_pair* out, int64_t capacity)
{
    if (!e || !e->host_mode)
        return set_error(GWB200_E_RUNTIME, "Invalid API call. Getting scored segment pairs without calling extend_async host ptr API");
    const int64_t n = std::min<int64_t>(capacity, static_cast<int64_t>(e->results.size()));
    if (n > 0)
        std::copy(e->results.begin(), e->results.begin() + n, out);
    return n;
}

int gwb200_extender_reset(gwb200_extender* e)
{
    if (!e)
        return set_error(GWB200_E_INVALID_ARGUMENT, "null extender");
    if (e->host_mode)
    {
        e->results.clear();
        e->host_mode = false;
    }
    return 0;
}

float gwb200_extender_last_kernel_ms(gwb200_extender* e)
{
    if (!e || !e->timed)
        return 0.f;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, e->ev0, e->ev1) != cudaSuccess)
    {
        cudaGetLastError();
        return 0.f;
    }
    return ms;
}

int64_t gwb200_extender_last_positions(gwb200_extender* e) { return e ? static_cast<int64_t>(e->pinned_positions[0]) : 0; }

} // extern "C"
