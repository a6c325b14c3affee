// dfd_internal.h — host-side objects behind the opaque C ABI handles.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "dfd_b200.h"
#include "dfd_hash.cuh"
#include "dfd_types.cuh"

namespace dfd {

int set_error(int code, const char* fmt, ...);
int cuda_error(cudaError_t e, const char* what);

struct Scratch {
    void* ptr = nullptr;
    size_t bytes = 0;
    int ensure(size_t need, int device);
};

}  // namespace dfd

// One worker == one GPU (reference `Worker`, src/worker/worker_service.rs:39-49).
struct dfd_ctx {
    int device = 0;
    int sm_count = 148;
    size_t l2_bytes = 0;
    cudaStream_t stream = nullptr;  // compute stream: K1/K1b/K2 launch here
    // profiling: ring of event quads recorded without syncing; drained lazily
    std::vector<cudaEvent_t> ev_ring;  // 4 events per call
    size_t ev_pending = 0;             // calls recorded, not yet accumulated
    static constexpr size_t EV_RING_CALLS = 64;
    int drain_events();                // sync + accumulate into metrics
    cudaEvent_t timer_a = nullptr, timer_b = nullptr;
    bool profiling = false;
    dfd::Scratch scratch;  // tile histograms / cursors
    void* scratch_done = nullptr;  // zero-initialised "blocks done" counter inside scratch
    dfd::Scratch flush;    // L2 flush buffer
    dfd::Scratch var_scratch;  // K4: iota | src row ids | block sums
    dfd::Scratch lb;           // single-pass mode: [ticket, done | 256 B] [look-back descriptors u64 [N][n_tiles]]
    uint32_t lb_epoch = 0;     // epoch of the last single-pass launch (30 bits; descriptors of older epochs are stale)
    dfd_metrics metrics = {};
    std::shared_ptr<void> pinned_cache;  // host operator: pinned output chunks of finished operators (dfd_exec.cu: PinnedCache)
    std::mutex mu;
};

// ≙ DataFusion BatchPartitioner::Hash { exprs, num_partitions, hash_buffer, random_state }
struct dfd_partitioner {
    dfd_ctx* ctx = nullptr;
    uint32_t N = 0;
    std::vector<int32_t> key_cols;
    std::vector<int32_t> key_modes;  // dfd_key_hash_mode per key column
    struct KeyDict { const uint64_t* hashes = nullptr; const uint8_t* validity = nullptr; };
    std::vector<KeyDict> key_dicts;  // DFD_KEY_HASH_DICTIONARY: device hashes / validity of the dictionary values
    dfd::HashState st{};
    dfd::ModN mod{};
    int64_t* d_part_starts = nullptr;  // [N+1]
    size_t smem_configured = 0;
    // single-pass (region layout) state: results of the last dfd_partition_device_onepass
    int64_t* d_counts = nullptr;       // [N] rows per destination | [N] dest_base | [N] dest_cap (exact re-run) | overflow flag
    int64_t* h_pin = nullptr;          // pinned: [N] counts, then the overflow flag
    enum { LAST_NONE = 0, LAST_DENSE = 1, LAST_REGIONS = 2 } last = LAST_NONE;
    std::vector<dfd_column> last_in, last_out;
    int64_t last_rows = 0, last_stride = 0;
};

namespace dfd {
using Ctx = ::dfd_ctx;
using Partitioner = ::dfd_partitioner;

// One partition call split into its stages so the exchange can put the count
// all-gather between K1b and K2.  Caller holds ctx->mu and has set the device.
struct PartitionJob {
    Partitioner* p = nullptr;
    cudaStream_t stream = nullptr;
    bool peer = false;
    KeySet ks{};
    std::vector<PayloadCol> passes;
    struct VarCol { dfd_column in, out; };
    std::vector<VarCol> var_cols;        // K4: variable-width payload columns
    uint32_t* d_src = nullptr;            // K4: input row of every output row (scattered iota)
    unsigned long long* d_block_sums = nullptr;
    uint64_t bytes = 0;
    int64_t n_rows = 0, n_tiles = 0;
    bool var_bytes_known = false;        // set before prepare(): in_cols[i].values_bytes IS the byte count of a var-width input (no D2H read + sync)
    bool onepass_tiling = false;         // set before prepare(): tile the rows for the single-pass kernel (ONEPASS_K rows per thread)
    int64_t out_rows = -1;               // rows of the OUTPUT row space (-1: n_rows; single-pass regions: N * region_rows)
    uint32_t* d_hist = nullptr;
    uint32_t* d_base = nullptr;
    int64_t* d_totals = nullptr;  // [N] rows per destination (after run_hist_scan)
    unsigned* d_done = nullptr;
    uint16_t* d_dest_cache = nullptr;  // two-pass, non-trivial keys: destination of every row (written by K1, read by every K2 launch)
    cudaEvent_t* ev = nullptr;
    int prepare(Partitioner* part, const dfd_column* in_cols, int n_cols, int64_t rows, const dfd_column* out_cols,
                bool peer_mode, cudaStream_t st);
    int run_hist_scan();
    int run_scatter(const int64_t* dest_base, void* const* peer_base, int world, uint32_t parts_per_rank,
                    const int32_t* abort_flag);
    int run_varwidth();  // called by run_scatter after the fixed-width launches
    // Single-pass K2 (no K1/K1b): destinations live in fixed regions; see k_scatter<..., ONEPASS>.
    struct OnePassLayout {
        const int64_t* d_dest_base = nullptr;  // device [N] region starts (rows); nullptr: region_stride formula
        const int64_t* d_dest_cap = nullptr;   // device [N] region capacities; nullptr: region_stride
        int64_t region_stride = 0;
        void* const* peer_base = nullptr;      // peer mode: every rank's window slot
        int world = 1, rank = 0;
        uint32_t parts_per_rank = 1;
        int64_t* d_totals = nullptr;           // device [N] out: rows per destination
        int32_t* d_overflow = nullptr;         // device out: set to 1 if a region is too small (caller zeroes it)
        const unsigned long long* ready_flags = nullptr;  // peer mode: "window free" flags in my header (see ExchangeHeader)
        unsigned long long ready_epoch = 0;
    };
    int run_onepass(const OnePassLayout& L);
};

constexpr uint32_t ONEPASS_MAX_N = 256;  // above this the per-tile look-back costs more than the K1 pass it replaces

// Small conversion kernels the exchange uses for bit-packed / variable-width columns (defined in dfd_api.cu).
int launch_bits_to_bytes(const uint8_t* bits, int64_t bit_offset, int64_t n, uint8_t* out, cudaStream_t s);
int launch_bytes_to_bits(const uint8_t* in, int64_t n, void* out_words, cudaStream_t s);
int launch_offsets_to_lengths(const void* off, int ow, int64_t n, void* len, cudaStream_t s);
int launch_var_dest_bytes(const void* off, int ow, const int64_t* part_starts, uint32_t N, int64_t* bytes, int64_t* first, cudaStream_t s);
int launch_lengths_to_offsets(const void* len, int ow, int64_t n, unsigned long long* block_sums /*[n/2048 + 2]*/, void* out_off, cudaStream_t s);
// out_data[out_off[j], out_off[j+1]) <- in_data at input row src[j] (+ in_offset), n output rows: k_var_copy_bytes with the
// lengths taken from the output offsets (a row may be shorter in the output than in the input, e.g. a null written as "").
int launch_var_gather(const void* in_off, int ow, int64_t in_offset, const uint8_t* in_data, const uint32_t* src, const void* out_off,
                      uint8_t* out_data, int64_t n, cudaStream_t s);

// Aligned write-out (k_scatter KV > K) is used for the peer-store exchange at small N (measured: +15% over NVLink, -5% local).
bool use_aligned(uint32_t N, bool peer);
// Kernel launch dispatch, one translation unit each (dfd_scatter_*.cu, templates in dfd_launch.cuh)
int launch_scatter_twopass_local(const ScatterParams& sp, int width, bool fast, int sm_count, size_t smem, cudaStream_t stream);
int launch_scatter_twopass_peer(const ScatterParams& sp, int width, bool fast, int sm_count, size_t smem, cudaStream_t stream);
int launch_scatter_onepass_local(const ScatterParams& sp, int width, bool fast, int sm_count, size_t smem, cudaStream_t stream);
int launch_scatter_onepass_peer(const ScatterParams& sp, int width, bool fast, int sm_count, size_t smem, cudaStream_t stream);
int launch_scatter_follow_local(const ScatterParams& sp, int width, bool fast, int sm_count, size_t smem, cudaStream_t stream);
int launch_scatter_follow_peer(const ScatterParams& sp, int width, bool fast, int sm_count, size_t smem, cudaStream_t stream);

// create_hashes over device columns -> raw u64 row hashes (dictionary values, parity hook).  Caller holds ctx->mu.
int hash_columns_locked(Ctx* c, const dfd_column* cols, int n_cols, int64_t n_rows, const uint64_t* seeds, uint64_t* hashes_device, cudaStream_t stream);

// Launches K1 -> K1b -> K2 on `stream`; caller holds ctx->mu and has set the device.
int partition_device_locked(Partitioner* p, const dfd_column* in_cols, int n_cols, int64_t n_rows,
                            const dfd_column* out_cols, cudaStream_t stream, bool var_bytes_known = false);

}  // namespace dfd
