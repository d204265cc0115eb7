// gw-b200: ungapped X-drop seed extension (the cudaextender module; the reference's kernel is
// cudaextender/src/ungapped_xdrop_kernels.cu:37-505, the algorithm is SegAlign's ungapped extender).
//
// One warp per seed, seeds pulled from an atomic counter by a persistent grid. Per-seed state lives in registers; the only
// shared memory is the 8x8 score matrix. Each step scores kPerLane consecutive positions per lane (32 * kPerLane per warp):
//   lane-local prefix sum and prefix max -> one warp sum scan + one warp max scan -> first drop or edge by ballot + __ffs ->
//   the best score before it by __reduce_max_sync and the earliest position holding it by a ballot.
// A second pass over the final segment counts the matching A/C/G/T bases for the entropy correction, only for seeds whose total
// score falls in [threshold, 3 * threshold]. Kept segments are appended (unordered) to a compact array; the host engine sorts
// and deduplicates them on the device (extender_capi.cu).
//
// Rules (DESIGN.md section 4, restated literally by oracle/extender_oracle.cpp):
//   right extension over p = 0, 1, ...: (T[t+p], Q[q+p]); best starts at (0, -1);
//   left extension over p = 1, 2, ...:  (T[t-p], Q[q-p]); best starts at (0, 0);
//   the running sum S(p) moves the best only when strictly larger (earliest maximum wins); the extension stops at the first p
//   where max(best, max S up to p) - S(p) > xdrop (that position does not count) or at the first position outside a sequence.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace gwb200
{
namespace extender
{

// == cudaextender::SeedPair / ScoredSegmentPair (extender.hpp:36-53); the layouts are ABI
struct Seed
{
    uint32_t query;
    uint32_t target;
};

struct Segment
{
    uint32_t query;
    uint32_t target;
    int32_t length;
    int32_t score;
};

constexpr int kWarpsPerBlock = 8;
constexpr int kSeedsPerGrab  = 4;   // seeds a warp takes from the counter at a time
constexpr int kPerLane       = 4;   // positions per lane per step: 128 positions per warp step

struct ExtendParams
{
    const int8_t* target;
    int64_t target_length;
    const int8_t* query;
    int64_t query_length;
    const int32_t* score_mat; // 64 entries, row = target code, column = query code
    int32_t xdrop;
    int32_t score_threshold;
    int32_t no_entropy;
    const Seed* seeds;
    int32_t num_seeds;
    Segment* kept;                  // [num_seeds], kept segments in no particular order
    int32_t* num_kept;              // zeroed before the launch
    int32_t* next_seed;             // zeroed before the launch
    unsigned long long* positions;  // evaluated positions (summed), zeroed before the launch
};

__device__ __forceinline__ int32_t warp_inclusive_sum(int32_t v, int lane)
{
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const int32_t u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o)
            v += u;
    }
    return v;
}

__device__ __forceinline__ int32_t warp_inclusive_max(int32_t v, int lane)
{
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const int32_t u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o)
            v = max(v, u);
    }
    return v;
}

// One direction of the extension. Position index i = 0, 1, ... maps to sequence offsets base_t + dir * i, base_q + dir * i;
// the first n_valid indices lie inside both sequences. Returns the best score (>= 0) and its index in *best_i (-1: none).
__device__ __forceinline__ int32_t extend_one_side(const ExtendParams& P, const int32_t* smat, int64_t base_t, int64_t base_q, int dir,
                                                   int64_t n_valid, int lane, int64_t* best_i_out, unsigned long long* evaluated)
{
    int32_t run_sum = 0; // S at the end of the previous step
    int32_t best    = 0;
    int64_t best_i  = -1;
    for (int64_t base = 0;; base += 32 * kPerLane)
    {
        const int64_t left_in_seq = n_valid - base;
        *evaluated += static_cast<unsigned long long>(left_in_seq <= 0 ? 0 : (left_in_seq < 32 * kPerLane ? left_in_seq : 32 * kPerLane));
        int32_t s[kPerLane];
        int32_t m[kPerLane];
        bool valid[kPerLane];
        int32_t acc = 0;
#pragma unroll
        for (int k = 0; k < kPerLane; k++)
        {
            const int64_t i = base + lane * kPerLane + k;
            valid[k]        = i < n_valid;
            int32_t sc      = 0;
            if (valid[k])
            {
                const int tc = __ldg(P.target + (base_t + dir * i)) & 7;
                const int qc = __ldg(P.query + (base_q + dir * i)) & 7;
                sc           = smat[tc * 8 + qc];
            }
            acc += sc;
            s[k] = acc; // lane-local inclusive prefix
        }
        const int32_t incl = warp_inclusive_sum(acc, lane);
        const int32_t off  = run_sum + incl - acc;
        int32_t lmax       = INT32_MIN;
#pragma unroll
        for (int k = 0; k < kPerLane; k++)
        {
            s[k] += off;
            lmax = max(lmax, s[k]);
            m[k] = lmax; // lane-local prefix max
        }
        const int32_t incl_max = warp_inclusive_max(lmax, lane);
        int32_t prev_max       = __shfl_up_sync(0xffffffffu, incl_max, 1);
        prev_max               = max(best, lane == 0 ? best : prev_max);
        int first_k            = kPerLane; // first stopping position of this lane
#pragma unroll
        for (int k = kPerLane - 1; k >= 0; k--)
        {
            if (!valid[k] || max(prev_max, m[k]) - s[k] > P.xdrop)
                first_k = k;
        }
        const unsigned stop_mask = __ballot_sync(0xffffffffu, first_k < kPerLane);
        const int stop_lane      = stop_mask ? __ffs(stop_mask) - 1 : 32;
        // positions before the stop: all of the lanes before stop_lane, first_k of stop_lane
        const int lim = lane < stop_lane ? kPerLane : (lane == stop_lane ? first_k : 0);
        int32_t cand  = INT32_MIN;
        int cand_k    = -1;
#pragma unroll
        for (int k = 0; k < kPerLane; k++)
        {
            if (k < lim && s[k] > cand)
            {
                cand   = s[k];
                cand_k = k;
            }
        }
        const int32_t step_best = __reduce_max_sync(0xffffffffu, cand);
        if (step_best > best)
        {
            const unsigned who = __ballot_sync(0xffffffffu, cand_k >= 0 && cand == step_best);
            const int w        = __ffs(who) - 1;
            const int wk       = __shfl_sync(0xffffffffu, cand_k, w);
            best               = step_best;
            best_i             = base + w * kPerLane + wk;
        }
        if (stop_mask)
            break;
        run_sum = __shfl_sync(0xffffffffu, incl, 31) + run_sum;
    }
    *best_i_out = best_i;
    return best;
}

// ln(4) as the reference computes it in f32 under -use_fast_math: lg2.approx(4) * 0.693147182f = 2 * 0.693147182f
__device__ __forceinline__ double ln4_f32() { return static_cast<double>(__int_as_float(0x3FB17218)); }

__global__ void __launch_bounds__(kWarpsPerBlock * 32) ungapped_xdrop_kernel(ExtendParams P)
{
    __shared__ int32_t smat[64];
    if (threadIdx.x < 64)
        smat[threadIdx.x] = P.score_mat[threadIdx.x];
    __syncthreads();
    const int lane                = threadIdx.x & 31;
    unsigned long long evaluated  = 0;
    const int64_t tlen            = P.target_length;
    const int64_t qlen            = P.query_length;
    const uint32_t thr3           = 3u * static_cast<uint32_t>(P.score_threshold);
    for (;;)
    {
        int32_t first = 0;
        if (lane == 0)
            first = atomicAdd(P.next_seed, kSeedsPerGrab);
        first = __shfl_sync(0xffffffffu, first, 0);
        if (first >= P.num_seeds)
            break;
        const int32_t last = min(P.num_seeds, first + kSeedsPerGrab);
        for (int32_t sid = first; sid < last; sid++)
        {
            const Seed seed = P.seeds[sid];
            const int64_t t = seed.target;
            const int64_t q = seed.query;
            // right: indices 0.. while t + i < |T| and q + i < |Q|
            int64_t n_right = min(tlen - t, qlen - q);
            n_right         = n_right < 0 ? 0 : n_right;
            // left: p = i + 1 <= min(t, q); a seed beyond the end of a sequence reads nothing outside it
            const int64_t n_left = (t > tlen || q > qlen) ? 0 : min(t, q);
            int64_t ri, li;
            const int32_t rs = extend_one_side(P, smat, t, q, 1, n_right, lane, &ri, &evaluated);
            const int32_t ls = extend_one_side(P, smat, t - 1, q - 1, -1, n_left, lane, &li, &evaluated);
            const int64_t rp    = ri;      // -1: right side empty
            const int64_t lp    = li + 1;  // 0: left side empty
            const int32_t total = rs + ls;
            double entropy      = 1.0;
            if (!P.no_entropy && total >= P.score_threshold && total <= static_cast<int32_t>(thr3))
            {
                // matching A/C/G/T over offsets [-lp, rp] of the final segment
                const int64_t len = rp + lp + 1;
                const int8_t* tp  = P.target + (t - lp);
                const int8_t* qp  = P.query + (q - lp);
                uint32_t c0 = 0, c1 = 0, c2 = 0, c3 = 0;
                for (int64_t j = lane; j < len; j += 32)
                {
                    const int tc = __ldg(tp + j);
                    const int qc = __ldg(qp + j);
                    const bool same = tc == qc;
                    c0 += same && tc == 0;
                    c1 += same && tc == 1;
                    c2 += same && tc == 2;
                    c3 += same && tc == 3;
                }
                c0 = __reduce_add_sync(0xffffffffu, c0);
                c1 = __reduce_add_sync(0xffffffffu, c1);
                c2 = __reduce_add_sync(0xffffffffu, c2);
                c3 = __reduce_add_sync(0xffffffffu, c3);
                if (c0 + c1 + c2 + c3 >= 20)
                {
                    const double denom = static_cast<double>(static_cast<int32_t>(len));
                    const uint32_t c[4] = {c0, c1, c2, c3};
                    double acc          = 0.0;
#pragma unroll
                    for (int i = 0; i < 4; i++)
                    {
                        if (c[i] != 0)
                        {
                            const double p = static_cast<double>(c[i]) / denom;
                            acc            = fma(p, log(p), acc);
                        }
                    }
                    entropy = -acc / ln4_f32();
                }
            }
            const int32_t score = static_cast<int32_t>(static_cast<double>(total) * entropy);
            if (lane == 0 && score >= P.score_threshold)
            {
                const int32_t slot = atomicAdd(P.num_kept, 1);
                Segment out;
                out.target      = static_cast<uint32_t>(t - lp);
                out.query       = static_cast<uint32_t>(q - lp);
                out.length      = static_cast<int32_t>(rp + lp);
                out.score       = score;
                P.kept[slot]    = out;
            }
        }
    }
    if (lane == 0 && evaluated)
        atomicAdd(P.positions, evaluated);
}

// Sort keys of the kept segments. The order is (uint32)(target - query) ascending, target ascending, length descending,
// score descending (scored_segment_pair_comp, ungapped_xdrop_kernels.cuh:85-134); two stable radix passes: minor key first.
__device__ __forceinline__ uint32_t descending_key(int32_t v) { return ~(static_cast<uint32_t>(v) ^ 0x80000000u); }

__global__ void minor_keys_kernel(const Segment* __restrict__ segs, int32_t n, uint64_t* __restrict__ keys)
{
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        const Segment s = segs[i];
        keys[i]         = (static_cast<uint64_t>(descending_key(s.length)) << 32) | descending_key(s.score);
    }
}

__global__ void major_keys_kernel(const Segment* __restrict__ segs, int32_t n, uint64_t* __restrict__ keys)
{
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        const Segment s = segs[i];
        keys[i]         = (static_cast<uint64_t>(s.target - s.query) << 32) | s.target;
    }
}

// scored_segment_pair_diagonal_overlap (ungapped_xdrop_kernels.cuh:65-83): same diagonal and one contains the other, the
// ends summed in uint32
__device__ __forceinline__ bool diagonal_overlap(const Segment& x, const Segment& y)
{
    if (x.target - x.query != y.target - y.query)
        return false;
    const uint32_t xe = x.target + static_cast<uint32_t>(x.length);
    const uint32_t ye = y.target + static_cast<uint32_t>(y.length);
    return (x.target >= y.target && xe <= ye) || (y.target >= x.target && ye <= xe);
}

// thrust::unique_copy semantics: an element is kept unless it overlaps its immediate predecessor in sorted order
__global__ void head_flags_kernel(const Segment* __restrict__ segs, int32_t n, uint8_t* __restrict__ flags)
{
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        flags[i] = (i == 0 || !diagonal_overlap(segs[i - 1], segs[i])) ? 1 : 0;
}

} // namespace extender
} // namespace gwb200
