/*
 * gwb200.h -- C ABI of the B200-native POA / banded-alignment / seed-extension engine (libgwb200.so).
 *
 * This is the drop-in boundary: plain C, opaque handles, host pointers and sizes, no C++/torch types.
 * Every entry point names the reference interface it replaces (paths relative to the GenomeWorks tree):
 *
 *   cudapoa     cudapoa/include/claraparabricks/genomeworks/cudapoa/batch.hpp     (BatchConfig, Batch, create_batch)
 *               cudapoa/include/claraparabricks/genomeworks/cudapoa/cudapoa.hpp   (StatusType, BandMode, OutputType, Init)
 *   cudaaligner cudaaligner/include/claraparabricks/genomeworks/cudaaligner/aligner.hpp   (Aligner, FixedBandAligner, create_aligner)
 *               cudaaligner/include/claraparabricks/genomeworks/cudaaligner/alignment.hpp (Alignment)
 *   cudaextender cudaextender/include/claraparabricks/genomeworks/cudaextender/extender.hpp (Extender, create_extender)
 *
 * The C++ classes with the reference's names (include/claraparabricks/genomeworks/...) and the Python mirror of
 * pygenomeworks (genomeworks_b200/) are thin wrappers over exactly these functions.
 *
 * Error convention (mirrors the reference's three tiers, SURVEY.md 8b):
 *   - functions that return a StatusType in the reference return that StatusType value (>= 0);
 *   - what the reference reports by throwing is returned as a negative GWB200_E_* code, message via gwb200_last_error();
 *   - there is NO CPU fallback: without a CUDA device every create call fails with GWB200_E_CUDA.
 */
#ifndef GWB200_H
#define GWB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GWB200_E_INVALID_ARGUMENT (-1) /* std::invalid_argument in the reference */
#define GWB200_E_RUNTIME (-2)          /* std::runtime_error in the reference */
#define GWB200_E_CUDA (-3)             /* CUDA runtime failure (the reference logs + aborts) */
#define GWB200_E_BAD_ALLOC (-4)        /* device_memory_allocation_exception in the reference */

/* Thread-local text of the last negative return. */
const char* gwb200_last_error(void);
/* Library version string. */
const char* gwb200_version(void);
/* Number of kernel launches issued by this library since load (all handles); used by bench.py's gpu_launches. */
int64_t gwb200_kernel_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * cudapoa
 * ---------------------------------------------------------------------------------------------- */

/* cudapoa::StatusType, cudapoa.hpp:34-49 (values are ABI: they cross the device boundary as a byte) */
enum gwb200_poa_status
{
    GWB200_POA_SUCCESS = 0,
    GWB200_POA_EXCEEDED_MAXIMUM_POAS,
    GWB200_POA_EXCEEDED_MAXIMUM_SEQUENCE_SIZE,
    GWB200_POA_EXCEEDED_MAXIMUM_SEQUENCES_PER_POA,
    GWB200_POA_NODE_COUNT_EXCEEDED_MAXIMUM_GRAPH_SIZE,
    GWB200_POA_EDGE_COUNT_EXCEEDED_MAXIMUM_GRAPH_SIZE,
    GWB200_POA_EXCEEDED_ADAPTIVE_BANDED_MATRIX_SIZE,
    GWB200_POA_EXCEEDED_MAXIMUM_PREDECESSOR_DISTANCE,
    GWB200_POA_LOOP_COUNT_EXCEEDED_UPPER_BOUND,
    GWB200_POA_OUTPUT_TYPE_UNAVAILABLE,
    GWB200_POA_ZERO_WEIGHTED_POA_SEQUENCE,
    GWB200_POA_EMPTY_POA_GROUP,
    GWB200_POA_GENERIC_ERROR
};

/* cudapoa::BandMode, cudapoa.hpp:62-69 */
enum gwb200_poa_band_mode
{
    GWB200_POA_FULL_BAND = 0,
    GWB200_POA_STATIC_BAND,
    GWB200_POA_ADAPTIVE_BAND,
    GWB200_POA_STATIC_BAND_TRACEBACK,
    GWB200_POA_ADAPTIVE_BAND_TRACEBACK
};

/* cudapoa::OutputType, cudapoa.hpp:75-79 */
enum gwb200_poa_output_type
{
    GWB200_POA_OUTPUT_CONSENSUS = 0x1,
    GWB200_POA_OUTPUT_MSA       = 0x2
};

/* cudapoa::BatchConfig, batch.hpp:60-86 -- same 8 fields, same order. */
typedef struct gwb200_poa_config
{
    int32_t max_sequence_size;
    int32_t max_consensus_size;
    int32_t max_nodes_per_graph;
    int32_t matrix_sequence_dimension;
    int32_t alignment_band_width;
    int32_t max_sequences_per_poa;
    int32_t band_mode;
    int32_t max_banded_pred_distance;
} gwb200_poa_config;

/* BatchConfig(max_seq_sz, max_seq_per_poa, band_width, banding, adaptive_storage_factor, graph_length_factor, max_pred_dist)
 * -- batch.hpp:80-81, cudapoa/src/batch.cu:34-71. Negative sizes -> GWB200_E_INVALID_ARGUMENT. */
int gwb200_poa_config_init(gwb200_poa_config* cfg, int32_t max_seq_sz, int32_t max_seq_per_poa, int32_t band_width, int32_t band_mode,
                           float adaptive_storage_factor, float graph_length_factor, int32_t max_pred_dist);
/* BatchConfig(max_seq_sz, max_consensus_sz, max_nodes_per_poa, band_width, max_seq_per_poa, matrix_seq_dim, banding, max_pred_dist)
 * -- batch.hpp:84-85, batch.cu:73-104. */
int gwb200_poa_config_init_explicit(gwb200_poa_config* cfg, int32_t max_seq_sz, int32_t max_consensus_sz, int32_t max_nodes_per_poa,
                                    int32_t band_width, int32_t max_seq_per_poa, int32_t matrix_seq_dim, int32_t band_mode, int32_t max_pred_dist);

/* cudapoa::Init(), cudapoa.hpp:72 */
int gwb200_poa_init(void);
/* cudapoa::decode_error(), cudapoa.hpp:55 -- writes NUL-terminated strings; unknown status -> GWB200_E_RUNTIME */
int gwb200_poa_decode_error(int32_t status, char* message, int32_t message_len, char* hint, int32_t hint_len);

/* SPOA_ACCURATE (cudapoa/src/cudapoa_kernels.cuh:508-530: a build flag of the reference that swaps the per-read topological sort
 * for racon's, which makes the graphs -- and MSAs -- identical to 3rdparty/spoa's). Here a library-wide run-time switch, also settable
 * with the environment variable GWB200_SPOA_ACCURATE=1 before the first batch; it applies to batches created afterwards. The C++
 * headers turn it on when the including translation unit defines SPOA_ACCURATE. */
void gwb200_poa_set_spoa_accurate(int32_t on);
int32_t gwb200_poa_get_spoa_accurate(void);

/* BatchBlock::estimate_max_poas(batch_size, msa_flag, memory_usage_quota, mismatch, gap, match) -- allocate_block.hpp:403-449:
 * how many windows of this configuration one batch holds when it may use `gpu_memory_usage_quota` of the currently free memory
 * of the current device (this engine's own arena layout). Used by get_multi_batch_sizes (utils.hpp:55-68). < 0 on error. */
int64_t gwb200_poa_estimate_max_poas(const gwb200_poa_config* cfg, int32_t msa_flag, float gpu_memory_usage_quota, int16_t mismatch_score,
                                     int16_t gap_score, int16_t match_score);

typedef struct gwb200_poa_batch gwb200_poa_batch; /* opaque: one cudapoa::Batch */

/* create_batch(device_id, stream, max_gpu_mem, output_mask, batch_size, gap_score, mismatch_score, match_score)
 * -- batch.hpp:191-204 (note the reference's argument order: gap, mismatch, match). `stream` is a cudaStream_t.
 * max_gpu_mem: bytes the batch may use; -1 => largest free block; < -1 => GWB200_E_INVALID_ARGUMENT.
 * Too little memory for one window => GWB200_E_RUNTIME (allocate_block.hpp:67-73). */
int gwb200_poa_batch_create(gwb200_poa_batch** out, int32_t device_id, void* stream, int64_t max_gpu_mem, int8_t output_mask,
                            const gwb200_poa_config* cfg, int16_t gap_score, int16_t mismatch_score, int16_t match_score);
/* create_batch(device_id, stream, DefaultDeviceAllocator allocator, max_gpu_mem, ...) -- batch.hpp:176-189, batch.cu:106-232,
 * allocate_block.hpp:48-100: the batch lives entirely inside `device_block` (a 256-byte aligned block of device_block_bytes
 * bytes the caller took from its allocator and releases after gwb200_poa_batch_destroy); nothing else is allocated on the device. */
int gwb200_poa_batch_create_in_block(gwb200_poa_batch** out, int32_t device_id, void* stream, void* device_block, int64_t device_block_bytes,
                                     int8_t output_mask, const gwb200_poa_config* cfg, int16_t gap_score, int16_t mismatch_score,
                                     int16_t match_score);
void gwb200_poa_batch_destroy(gwb200_poa_batch* batch);

/* Batch::add_poa_group(per_seq_status, poa_group) -- batch.hpp:100-111, cudapoa_batch.cuh:103-151.
 * One Entry per i: {seqs[i], weights ? weights[i] : NULL, lengths[i]}. weights may be NULL (all entries unweighted).
 * per_seq_status (n entries, may be NULL) receives one StatusType per entry; *n_per_seq the number written
 * (0 when the group itself is rejected). Returns the group's StatusType; negative weight => GWB200_E_INVALID_ARGUMENT. */
int gwb200_poa_batch_add_group(gwb200_poa_batch* batch, int32_t n, const char* const* seqs, const int8_t* const* weights,
                               const int32_t* lengths, int32_t* per_seq_status, int32_t* n_per_seq);
/* Bulk form of the same call for flat callers (Python): windows [first, first+count) of a flat window list
 * (win_nseq[], seq_len[], concatenated seq_data, optional concatenated weights). Stops at the first window that is not taken
 * into the batch; *n_added = windows consumed; returns that window's StatusType (success if all were added). A window whose reads
 * were all rejected is consumed like in the reference (it stays in the batch as an empty window): the call goes on and returns
 * empty_poa_group at the end if no later window stopped it. */
int gwb200_poa_batch_add_groups_flat(gwb200_poa_batch* batch, int32_t n_windows, const int32_t* win_nseq, const int32_t* seq_len,
                                     const char* seq_data, const int8_t* weights, int32_t* n_added);

/* Batch::get_total_poas(), batch.hpp:114 */
int32_t gwb200_poa_batch_total_poas(const gwb200_poa_batch* batch);
/* Capacity the batch was sized for (max_poas_, cudapoa_batch.cuh:77). */
int32_t gwb200_poa_batch_max_poas(const gwb200_poa_batch* batch);
/* Batch::generate_poa(), batch.hpp:117 -- async on the batch's stream: H2D of the packed inputs, then the kernels. */
int gwb200_poa_batch_generate(gwb200_poa_batch* batch);
/* The two halves of generate_poa, for callers that want inputs resident before timing (bench.py `value`). */
int gwb200_poa_batch_upload(gwb200_poa_batch* batch);
int gwb200_poa_batch_launch(gwb200_poa_batch* batch);
/* cudaStreamSynchronize on the batch's stream. */
int gwb200_poa_batch_sync(gwb200_poa_batch* batch);

/* Batch::get_consensus(consensus, coverage, output_status) -- batch.hpp:124-131, cudapoa_batch.cuh:202-258. Blocking.
 * consensus: [total_poas * max_consensus_size] forward-oriented NUL-terminated strings ("" on error);
 * coverage:  [total_poas * max_consensus_size]; lengths/status: [total_poas]. Returns success or output_type_unavailable. */
int gwb200_poa_batch_get_consensus(gwb200_poa_batch* batch, char* consensus, uint16_t* coverage, int32_t* lengths, int32_t* status);
/* Batch::get_msa(msa, output_status) -- batch.hpp:137-139, cudapoa_batch.cuh:261-313. Blocking.
 * msa: [total_poas * max_sequences_per_poa * max_consensus_size]; row r of window w at (w*max_seqs + r)*max_consensus.
 * num_rows[w] = number of sequences in window w (0 on error). */
int gwb200_poa_batch_get_msa(gwb200_poa_batch* batch, char* msa, int32_t* num_rows, int32_t* status);
/* Batch::get_graphs(graphs, output_status) -- batch.hpp:145-147, cudapoa_batch.cuh:315-393. Two-call protocol:
 * first call with edge_src == NULL fills node_counts[w], edge_counts[w], status[w]; second call fills
 * node_labels (concatenated per window), edge_src / edge_dst / edge_weight (concatenated, in the reference's
 * insertion order: for each sink node n ascending, its incoming edges in slot order). */
int gwb200_poa_batch_get_graphs(gwb200_poa_batch* batch, int32_t* node_counts, int32_t* edge_counts, int32_t* status,
                                uint8_t* node_labels, int32_t* edge_src, int32_t* edge_dst, int32_t* edge_weight);
/* Batch::batch_id(), batch.hpp:150 ; Batch::reset(), batch.hpp:153 */
int32_t gwb200_poa_batch_id(const gwb200_poa_batch* batch);
int gwb200_poa_batch_reset(gwb200_poa_batch* batch);

/* Measurement helpers (not in the reference API): executed DP cells of the last generate (sum over windows of
 * graph_count x band_width per alignment pass incl. adaptive reruns, SURVEY.md 8d), and device time of the last
 * launch measured with CUDA events on the batch's stream (ms; requires gwb200_poa_batch_sync first). */
int64_t gwb200_poa_batch_last_cells(gwb200_poa_batch* batch);
float gwb200_poa_batch_last_kernel_ms(gwb200_poa_batch* batch);
/* Optional per-phase cycle counters of the POA kernel (development / profiling aid): enable before generate, read after
 * sync. out8[0..5] = DP rows, end-cell search, traceback, add-alignment, topological sort, consensus/MSA; summed over windows. */
int gwb200_poa_batch_enable_timers(gwb200_poa_batch* batch, int32_t on);
int gwb200_poa_batch_get_timers(gwb200_poa_batch* batch, uint64_t* out8);
/* Windows the device can keep resident at once for this batch's kernel (SMs x CTAs per SM): a batch of at most this many
 * windows runs as a single wave. */
int32_t gwb200_poa_batch_resident_windows(gwb200_poa_batch* batch);
/* sizeof(ScoreT) chosen for this batch (2 or 4), cudapoa_limits.hpp:34-44. */
int32_t gwb200_poa_batch_score_bytes(const gwb200_poa_batch* batch);

/* Evaluates __fdividef(a, b) on the device (the fast-math division the reference's band geometry uses,
 * cudapoa_nw_banded.cuh:207). Exists so tests can give the CPU oracle bit-identical band placement. */
int gwb200_device_fdividef(int32_t n, const float* a, const float* b, float* out);

/* ------------------------------------------------------------------------------------------------
 * cudaaligner (banded Myers global aligner)
 * ---------------------------------------------------------------------------------------------- */

/* cudaaligner::StatusType, cudaaligner.hpp:34-42 */
enum gwb200_aligner_status
{
    GWB200_ALN_SUCCESS = 0,
    GWB200_ALN_UNINITIALIZED,
    GWB200_ALN_EXCEEDED_MAX_ALIGNMENTS,
    GWB200_ALN_EXCEEDED_MAX_LENGTH,
    GWB200_ALN_EXCEEDED_MAX_ALIGNMENT_DIFFERENCE,
    GWB200_ALN_GENERIC_ERROR
};

/* cudaaligner::AlignmentState, cudaaligner.hpp:51-57 (the bytes in device results) */
enum gwb200_alignment_state
{
    GWB200_ALN_MATCH = 0,
    GWB200_ALN_MISMATCH,
    GWB200_ALN_INSERTION,
    GWB200_ALN_DELETION
};

typedef struct gwb200_aligner gwb200_aligner; /* opaque: one cudaaligner::FixedBandAligner */

/* cudaaligner::Init(), cudaaligner.hpp:66 */
int gwb200_aligner_init(void);
/* create_aligner(AlignmentType::global_alignment, max_bandwidth, stream, device_id, max_device_memory)
 * -- aligner.hpp:208-219, cudaaligner/src/aligner.cpp:76-124. max_device_memory: -1 => largest free block,
 * < -1 => GWB200_E_INVALID_ARGUMENT; max_bandwidth % 32 == 1 => GWB200_E_INVALID_ARGUMENT
 * (aligner_global_myers_banded.cpp:470-473). */
int gwb200_aligner_create(gwb200_aligner** out, int32_t max_bandwidth, void* stream, int32_t device_id, int64_t max_device_memory);
/* create_aligner(..., DefaultDeviceAllocator allocator, max_device_memory) -- aligner.hpp:183-219, cudaaligner/src/aligner.cpp:76-124:
 * every device buffer of the aligner is a block of the caller's allocator (allocator.hpp:322-358). alloc_fn returns NULL when
 * the pool cannot serve the request (the alignment call then fails the way an out-of-memory does); free_fn gets the size back. */
typedef void* (*gwb200_device_alloc_fn)(void* user, int64_t bytes);
typedef void (*gwb200_device_free_fn)(void* user, void* ptr, int64_t bytes);
int gwb200_aligner_create_with_allocator(gwb200_aligner** out, int32_t max_bandwidth, void* stream, int32_t device_id, int64_t max_device_memory,
                                         gwb200_device_alloc_fn alloc_fn, gwb200_device_free_fn free_fn, void* user);
void gwb200_aligner_destroy(gwb200_aligner* aligner);
/* FixedBandAligner::add_alignment([max_bandwidth,] query, query_length, target, target_length, rc_query, rc_target)
 * -- aligner.hpp:96-97,158-170; aligner_global_myers_banded.cpp:155-258. max_bandwidth == GWB200_ALN_DEFAULT_BANDWIDTH => the aligner's
 * own (the overload without a bandwidth); any other value is taken as given: 0 is honoured (such a pair is skipped on the device
 * and stays uninitialized, myers_gpu.cu:903-912), other negative values return generic_error, as in the reference. */
#define GWB200_ALN_DEFAULT_BANDWIDTH (-2147483647 - 1)
int gwb200_aligner_add_alignment(gwb200_aligner* aligner, int32_t max_bandwidth, const char* query, int32_t query_length,
                                 const char* target, int32_t target_length, int32_t reverse_complement_query,
                                 int32_t reverse_complement_target);
/* Aligner::align_all(), aligner.hpp:82 -- async. Aligner::sync_alignments(), aligner.hpp:87 -- blocking. */
int gwb200_aligner_align_all(gwb200_aligner* aligner);
int gwb200_aligner_sync_alignments(gwb200_aligner* aligner);
/* Aligner::num_alignments(), aligner.hpp:128 */
int32_t gwb200_aligner_num_alignments(const gwb200_aligner* aligner);
/* number of results the last sync_alignments() produced (what get_alignments() can be filled from) */
int32_t gwb200_aligner_num_results(const gwb200_aligner* aligner);
/* Results of alignment i after sync (what Alignment::get_status / is_optimal / get_actions / get_runlengths expose,
 * alignment.hpp:55-111): status, is_optimal, number of run-length entries; then the entries themselves
 * (actions: AlignmentState bytes, runlengths), query-start to query-end order. */
int gwb200_aligner_result_info(const gwb200_aligner* aligner, int32_t i, int32_t* status, int32_t* is_optimal, int32_t* n_runs);
int gwb200_aligner_result_runs(const gwb200_aligner* aligner, int32_t i, int8_t* actions, int32_t* runlengths);
/* Aligner::reset(), aligner.hpp:112 ; FixedBandAligner::reset_max_bandwidth(), aligner.hpp:153 ;
 * Aligner::free_temporary_device_buffers(), aligner.hpp:124 */
/* Convenience for FFI callers (not part of the reference surface): the loop a C++ caller writes around add_alignment(), and all
 * results of the last sync_alignments() in one call (run_offsets[n + 1]; entries of alignment i at [run_offsets[i], run_offsets[i + 1])). */
int gwb200_aligner_add_alignments(gwb200_aligner* aligner, int32_t n, const char* const* queries, const int32_t* query_lengths,
                                  const char* const* targets, const int32_t* target_lengths, int32_t* n_added);
int gwb200_aligner_results_flat(const gwb200_aligner* aligner, int32_t* status, int32_t* is_optimal, int64_t* run_offsets, int8_t* actions,
                                int32_t* runlengths, int64_t capacity);
int gwb200_aligner_reset(gwb200_aligner* aligner);
int gwb200_aligner_reset_max_bandwidth(gwb200_aligner* aligner, int32_t max_bandwidth);
int gwb200_aligner_free_temporary_device_buffers(gwb200_aligner* aligner);
/* Aligner::get_alignments_device(), aligner.hpp:107 -- DeviceAlignmentsPtrs (aligner.hpp:62-72): device pointers
 * borrowed until reset()/destroy. */
int gwb200_aligner_get_alignments_device(const gwb200_aligner* aligner, const int8_t** cigar_operations, const int32_t** cigar_runlengths,
                                         const int32_t** cigar_offsets, const uint32_t** metadata, int64_t* total_length,
                                         int32_t* n_alignments);
/* Measurement helpers: executed DP cells (sum over Ukkonen passes of band_width x target_length) and device ms of the
 * last align_all. */
int64_t gwb200_aligner_last_cells(gwb200_aligner* aligner);
float gwb200_aligner_last_kernel_ms(gwb200_aligner* aligner);

/* ------------------------------------------------------------------------------------------------
 * cudaaligner, fixed-size global aligners: what the deprecated factory create_aligner(max_query_length, max_target_length,
 * max_alignments, type, [allocator,] stream, device) builds (cudaaligner/include/.../aligner.hpp:183,196; src/aligner.cpp:31-74
 * -> AlignerGlobalHirschbergMyers) and the in-library AlignerGlobalMyers / AlignerGlobalUkkonen (cudaaligner/src/aligner_global_{myers,
 * ukkonen}.cpp).
 * Host behaviour = AlignerGlobal (cudaaligner/src/aligner_global.cpp:50-197): fixed-stride sequence and result slots,
 * results as one AlignmentState byte per alignment column in forward order.
 * ---------------------------------------------------------------------------------------------- */
enum gwb200_global_algorithm
{
    GWB200_GLOBAL_HIRSCHBERG_MYERS = 0, /* aligner_global_hirschberg_myers.cpp:32-75, hirschberg_myers_gpu.cu:575-699 */
    GWB200_GLOBAL_MYERS            = 1, /* aligner_global_myers.cpp:40-70, myers_gpu.cu:256-442,1117-1139 */
    GWB200_GLOBAL_UKKONEN          = 2  /* aligner_global_ukkonen.cpp:30-81, ukkonen_gpu.cu:62-262 (band p = 100, int16 scores) */
};
typedef struct gwb200_global_aligner gwb200_global_aligner; /* opaque: one cudaaligner::AlignerGlobal */

/* AlignerGlobal::AlignerGlobal (aligner_global.cpp:50-76): negative sizes -> GWB200_E_INVALID_ARGUMENT, max_alignments < 1 ->
 * GWB200_E_RUNTIME ("Max alignments must be at least 1."). alloc/release may be NULL (cudaMalloc / cudaFree). */
int gwb200_global_aligner_create(gwb200_global_aligner** out, int32_t algorithm, int32_t max_query_length, int32_t max_target_length,
                                 int32_t max_alignments, void* stream, int32_t device_id, gwb200_device_alloc_fn alloc,
                                 gwb200_device_free_fn release, void* user);
void gwb200_global_aligner_destroy(gwb200_global_aligner* aligner);
/* AlignerGlobal::add_alignment (aligner_global.cpp:78-141): returns a gwb200_aligner_status */
int gwb200_global_aligner_add_alignment(gwb200_global_aligner* aligner, const char* query, int32_t query_length, const char* target,
                                        int32_t target_length, int32_t reverse_complement_query, int32_t reverse_complement_target);
int gwb200_global_aligner_align_all(gwb200_global_aligner* aligner);      /* aligner_global.cpp:143-160 */
int gwb200_global_aligner_sync_alignments(gwb200_global_aligner* aligner); /* aligner_global.cpp:162-190 */
int32_t gwb200_global_aligner_num_alignments(const gwb200_global_aligner* aligner);
/* Result i after sync: *length = number of alignment columns (0 with *has_result == 0: the alignment failed and the reference
 * leaves its Alignment untouched); *is_optimal as AlignmentImpl::set_alignment receives it. */
int gwb200_global_aligner_result_info(const gwb200_global_aligner* aligner, int32_t i, int32_t* has_result, int32_t* is_optimal, int32_t* length);
/* The alignment columns of result i in forward order (gwb200_alignment_state bytes); states must hold *length entries. */
int gwb200_global_aligner_result_states(const gwb200_global_aligner* aligner, int32_t i, int8_t* states);
int gwb200_global_aligner_reset(gwb200_global_aligner* aligner);           /* aligner_global.cpp:192-195 */
int64_t gwb200_global_aligner_last_cells(gwb200_global_aligner* aligner);
float gwb200_global_aligner_last_kernel_ms(gwb200_global_aligner* aligner);

/* ------------------------------------------------------------------------------------------------
 * cudaextender (ungapped X-drop seed extension)
 *   cudaextender/include/claraparabricks/genomeworks/cudaextender/cudaextender.hpp (StatusType, ExtensionType)
 *   cudaextender/include/claraparabricks/genomeworks/cudaextender/extender.hpp     (SeedPair, ScoredSegmentPair, Extender,
 *                                                                                   create_extender)
 *   cudaextender/src/ungapped_xdrop.cu:50-253                                      (UngappedXDrop)
 * ---------------------------------------------------------------------------------------------- */

/* cudaextender::StatusType, cudaextender.hpp:34-40 */
enum gwb200_extender_status
{
    GWB200_EXT_SUCCESS           = 0,
    GWB200_EXT_INVALID_OPERATION = 1,
    GWB200_EXT_INVALID_INPUT     = 2,
    GWB200_EXT_GENERIC_ERROR     = 3
};

/* cudaextender::ExtensionType, cudaextender.hpp:44-47 */
enum gwb200_extension_type
{
    GWB200_EXT_UNGAPPED_XDROP = 0
};

/* cudaextender::SeedPair, extender.hpp:36-42: {query, target}, 8 bytes (device-API callers pass arrays of these) */
typedef struct gwb200_seed_pair
{
    uint32_t query_position_in_read;
    uint32_t target_position_in_read;
} gwb200_seed_pair;

/* cudaextender::ScoredSegmentPair, extender.hpp:45-53: {SeedPair start_coord, length, score}, 16 bytes. length is one less than
 * the number of bases the segment covers. */
typedef struct gwb200_scored_segment_pair
{
    gwb200_seed_pair start_coord;
    int32_t length;
    int32_t score;
} gwb200_scored_segment_pair;

typedef struct gwb200_extender gwb200_extender; /* opaque: one cudaextender::Extender (UngappedXDrop) */

/* create_extender(h_score_mat, score_mat_dim, xdrop_threshold, no_entropy, stream, device_id, allocator, type) -- extender.hpp:147-154,
 * cudaextender/src/extender.cpp:27-43, ungapped_xdrop.cu:50-94. h_score_mat is 8 x 8, row = target code, column = query code
 * (codes of utils.hpp:36-44); score_mat_dim < 64 or a NULL matrix -> GWB200_E_INVALID_ARGUMENT; type other than
 * GWB200_EXT_UNGAPPED_XDROP -> GWB200_E_RUNTIME. Device memory comes from alloc_fn / free_fn (NULL: cudaMalloc / cudaFree) and
 * is sized per call. */
int gwb200_extender_create(gwb200_extender** out, const int32_t* h_score_mat, int32_t score_mat_dim, int32_t xdrop_threshold,
                           int32_t no_entropy, void* stream, int32_t device_id, int32_t type, gwb200_device_alloc_fn alloc_fn,
                           gwb200_device_free_fn free_fn, void* user);
void gwb200_extender_destroy(gwb200_extender* ext);
/* Extender::extend_async, host pointer API (extender.hpp:82-85, ungapped_xdrop.cu:181-210): copies the encoded sequences and
 * the seeds to the device and extends them on the extender's stream. Resets the results of the previous host call. Returns a
 * gwb200_extender_status; a pool too small for the call -> GWB200_E_BAD_ALLOC. */
int gwb200_extender_extend_host(gwb200_extender* ext, const int8_t* h_query, int32_t query_length, const int8_t* h_target,
                                int32_t target_length, int32_t score_threshold, const gwb200_seed_pair* h_seed_pairs,
                                int32_t num_seed_pairs);
/* Extender::extend_async, device pointer API (extender.hpp:108-112, ungapped_xdrop.cu:96-179). d_scored_segment_pairs holds
 * num_seed_pairs entries; *d_num_scored_segment_pairs receives the number written. NULL input or output pointers ->
 * GWB200_EXT_INVALID_INPUT. Stream ordered; the call waits once for the number of segments that pass the threshold. */
int gwb200_extender_extend_device(gwb200_extender* ext, const int8_t* d_query, int32_t query_length, const int8_t* d_target,
                                  int32_t target_length, int32_t score_threshold, const gwb200_seed_pair* d_seed_pairs,
                                  int32_t num_seed_pairs, gwb200_scored_segment_pair* d_scored_segment_pairs,
                                  int32_t* d_num_scored_segment_pairs);
/* Extender::sync(), extender.hpp:121, ungapped_xdrop.cu:212-228: waits and fetches the results of the last host call;
 * GWB200_EXT_INVALID_OPERATION without one. */
int gwb200_extender_sync(gwb200_extender* ext);
/* Extender::get_scored_segment_pairs(), extender.hpp:130, ungapped_xdrop.cu:230-238: the number of results after sync, and a flat
 * copy of them (capacity entries at most). Without a preceding host call both return GWB200_E_RUNTIME. */
int64_t gwb200_extender_num_results(const gwb200_extender* ext);
int64_t gwb200_extender_get_results(const gwb200_extender* ext, gwb200_scored_segment_pair* out, int64_t capacity);
/* Extender::reset(), extender.hpp:133, ungapped_xdrop.cu:240-248 */
int gwb200_extender_reset(gwb200_extender* ext);
/* Measurement helpers (not in the reference API): device ms of the last extension call, from the extension kernel to the last
 * deduplication kernel (requires the stream to have finished it), and the positions the last call scored (each reads one byte
 * of each sequence). */
float gwb200_extender_last_kernel_ms(gwb200_extender* ext);
int64_t gwb200_extender_last_positions(gwb200_extender* ext);

/* ------------------------------------------------------------------------------------------------
 * Synthetic workloads (SURVEY.md 8d): the reference's own generators
 * (common/base/include/claraparabricks/genomeworks/utils/genomeutils.hpp:33-142, std::minstd_rand).
 * ---------------------------------------------------------------------------------------------- */

/* Window w: rng(seed0 + w); backbone = generate_random_genome(backbone_len); reads = generate_random_sequences(backbone,
 * n_reads, rng, max_mut, max_ins, max_del) (read 0 is the backbone); reads longer than max_read_len (> 0) are truncated.
 * seq_len[n_windows * n_reads]; seq_data receives the reads concatenated. Returns bytes written, -1 if capacity is too small. */
int64_t gwb200_synth_poa_windows(int32_t n_windows, uint32_t seed0, int32_t backbone_len, int32_t n_reads, int32_t max_mut, int32_t max_ins,
                                 int32_t max_del, int32_t max_read_len, int32_t* seq_len, char* seq_data, int64_t capacity);
/* Pairs exactly as cudaaligner/benchmarks/main.cpp:116-129: one rng(seed); g1 = generate_random_genome(genome_size);
 * g2 = generate_random_sequence(g1, rng, L/30, L/30, L/30) truncated to genome_size. query = g1, target = g2. */
int64_t gwb200_synth_aligner_pairs(int32_t n_pairs, uint32_t seed, int32_t genome_size, int32_t* q_len, char* q_data, int64_t q_capacity,
                                   int32_t* t_len, char* t_data, int64_t t_capacity);

#ifdef __cplusplus
}
#endif
#endif /* GWB200_H */
