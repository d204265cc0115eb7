// TEST / BASELINE INFRASTRUCTURE ONLY: a flat C entry over the UNMODIFIED reference cudaextender (built from the reference
// sources into oracle/_ref/libgwref_ext.so by oracle/Makefile). Runs one extension through the host pointer API or the device
// pointer API, the way cudaextender/samples/sample_cudaextender.cpp does, and times it.
#include <claraparabricks/genomeworks/cudaextender/extender.hpp>
#include <claraparabricks/genomeworks/utils/cudautils.hpp>
#include <claraparabricks/genomeworks/utils/device_buffer.hpp>

#include <chrono>
#include <cstdio>
#include <cstring>
#include <exception>
#include <vector>

using namespace claraparabricks::genomeworks;
using namespace claraparabricks::genomeworks::cudaextender;

extern "C" {

// seeds: n pairs {query, target}; out: n records {query, target, length, score}; *n_out: records written.
// timings[0]: device ms of the device-API extend_async (CUDA events; device_api only), timings[1]: host ms of extend_async + sync
// (+ result copy), timings[2]: host ms of create_extender.
int ref_extender_run(const int8_t* query, int32_t query_length, const int8_t* target, int32_t target_length, const int32_t* score_mat,
                     int32_t xdrop, int32_t no_entropy, int32_t score_threshold, const uint32_t* seeds, int32_t n, int32_t device_api,
                     int32_t* out, int32_t* n_out, double* timings, char* err, int32_t err_len)
{
    try
    {
        static_assert(sizeof(SeedPair) == 8 && sizeof(ScoredSegmentPair) == 16, "layout");
        std::vector<SeedPair> h_seeds(n);
        if (n > 0)
            std::memcpy(h_seeds.data(), seeds, static_cast<size_t>(n) * 8);
        cudaDeviceProp prop;
        GW_CU_CHECK_ERR(cudaGetDeviceProperties(&prop, 0));
        // the reference's own scratch (ungapped_xdrop.cu:75-92) plus inputs, outputs and thrust's temporary storage
        const size_t batch = static_cast<size_t>(static_cast<int32_t>(static_cast<float>(prop.totalGlobalMem) / 1073741824.0f)) * 4194304;
        const size_t pool  = batch * 20 + static_cast<size_t>(n) * 96 + 2 * (static_cast<size_t>(query_length) + target_length) + (1ull << 30);
        DefaultDeviceAllocator allocator = create_default_device_allocator(pool);
        CudaStream stream                = make_cuda_stream();
        const auto c0                    = std::chrono::steady_clock::now();
        std::unique_ptr<Extender> ext    = create_extender(score_mat, 64, xdrop, no_entropy != 0, stream.get(), 0, allocator);
        GW_CU_CHECK_ERR(cudaStreamSynchronize(stream.get()));
        const auto c1 = std::chrono::steady_clock::now();
        timings[2]    = std::chrono::duration<double, std::milli>(c1 - c0).count();
        std::vector<ScoredSegmentPair> res;
        if (!device_api)
        {
            const auto t0 = std::chrono::steady_clock::now();
            ext->extend_async(query, query_length, target, target_length, score_threshold, h_seeds);
            ext->sync();
            res           = ext->get_scored_segment_pairs();
            const auto t1 = std::chrono::steady_clock::now();
            timings[0]    = 0;
            timings[1]    = std::chrono::duration<double, std::milli>(t1 - t0).count();
        }
        else
        {
            device_buffer<int8_t> d_query(query_length, allocator, stream.get());
            device_buffer<int8_t> d_target(target_length, allocator, stream.get());
            device_buffer<SeedPair> d_seeds(n, allocator, stream.get());
            device_buffer<ScoredSegmentPair> d_ssp(n, allocator, stream.get());
            device_buffer<int32_t> d_num(1, allocator, stream.get());
            cudautils::device_copy_n_async(query, query_length, d_query.data(), stream.get());
            cudautils::device_copy_n_async(target, target_length, d_target.data(), stream.get());
            cudautils::device_copy_n_async(h_seeds.data(), n, d_seeds.data(), stream.get());
            GW_CU_CHECK_ERR(cudaStreamSynchronize(stream.get()));
            cudaEvent_t e0, e1;
            cudaEventCreate(&e0);
            cudaEventCreate(&e1);
            const auto t0 = std::chrono::steady_clock::now();
            cudaEventRecord(e0, stream.get());
            ext->extend_async(d_query.data(), query_length, d_target.data(), target_length, score_threshold, d_seeds.data(), n, d_ssp.data(),
                              d_num.data());
            cudaEventRecord(e1, stream.get());
            GW_CU_CHECK_ERR(cudaStreamSynchronize(stream.get()));
            const auto t1 = std::chrono::steady_clock::now();
            float ms      = 0;
            cudaEventElapsedTime(&ms, e0, e1);
            cudaEventDestroy(e0);
            cudaEventDestroy(e1);
            timings[0]      = ms;
            timings[1]      = std::chrono::duration<double, std::milli>(t1 - t0).count();
            const int32_t k = cudautils::get_value_from_device(d_num.data(), stream.get());
            res.resize(k);
            if (k > 0)
                cudautils::device_copy_n_async(d_ssp.data(), k, res.data(), stream.get());
            GW_CU_CHECK_ERR(cudaStreamSynchronize(stream.get()));
        }
        *n_out = static_cast<int32_t>(res.size());
        if (!res.empty())
            std::memcpy(out, res.data(), res.size() * 16);
        ext.reset();
        return 0;
    }
    catch (const std::exception& e)
    {
        std::snprintf(err, err_len, "%s", e.what());
        return -1;
    }
}

} // extern "C"
