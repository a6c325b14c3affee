// dfd_reduce.cu — device-side PartialReduce ahead of the shuffle.
//
// The reference inserts AggregateExec(mode = PartialReduce) ABOVE the producers' hash RepartitionExec
// (src/distributed_planner/partial_reduce_below_network_shuffles.rs:17-100; plan shape tests/distributed_aggregation.rs:63-67):
// after hash repartitioning, rows with equal group keys sit in the same destination partition, so merging their
// aggregate states there shrinks what crosses the network.  Here the partitioned table is already on the GPU
// (output of dfd_partition_device), so the merge runs on it in place of a PCIe round trip:
//   k_group_insert   open-addressing table of REPRESENTATIVE ROW indices (one u32 per slot): a row claims an empty slot
//                    with atomicCAS or joins the group whose representative has equal key bytes AND lies in the same
//                    input partition (any number / width of fixed-width keys — the keys themselves are never copied into
//                    the table).  Groups never cross partitions: the caller's part_starts need not follow the group keys.
//   k_group_count    groups per destination partition (representatives only)      -> exclusive scan (host, N+1 values)
//   k_group_place    every group gets an output row inside its partition; key columns copied, states initialised
//   k_group_combine  every input row folds its states into its group's output row with atomics
//                    (SUM i64 / f64 / i128 (two 64-bit adds with carry), MIN / MAX i64, MIN / MAX f64 in the integer
//                    image of IEEE-754 totalOrder, so the result is the same whatever order the atomics land in)
//   k_group_finish   only with a float MIN / MAX column: maps those states back from the totalOrder image to doubles
// Integer / byte work; random access into an L2-resident table for the cardinalities PartialReduce is used for.
#include <cuda_runtime.h>

#include <cstdint>
#include <mutex>
#include <vector>

#include "dfd_b200.h"
#include "dfd_internal.h"

using namespace dfd;

namespace {

constexpr int MAX_REDUCE_COLS = 32;
constexpr uint32_t SLOT_EMPTY = 0xffffffffu;

struct ReduceCol {
    const char* in;
    char* out;
    int32_t width;
    int32_t op;  // dfd_agg_op, or -1 for a group key
};

struct ReduceParams {
    ReduceCol col[MAX_REDUCE_COLS];
    int32_t n_cols;
    int32_t key_idx[MAX_KEYS];
    int32_t n_keys;
    int64_t n_rows;
    uint32_t N;
    uint32_t table_mask;
    uint32_t* table;        // [table_mask + 1] representative row of every slot
    uint32_t* row_slot;     // [n_rows] slot of every row's group
    uint32_t* slot_out;     // [table_mask + 1] output row of the slot's group
    const int64_t* part_starts;  // [N+1] input partition boundaries (device)
    unsigned long long* group_count;  // [N]
    int64_t* out_starts;    // [N+1] (device)
    unsigned long long* cursor;  // [N]
};

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x;
}

__device__ __forceinline__ uint64_t key_hash(const ReduceParams& P, int64_t row) {
    uint64_t h = 0x9e3779b97f4a7c15ULL;
    for (int k = 0; k < P.n_keys; ++k) {
        const ReduceCol& c = P.col[P.key_idx[k]];
        const char* p = c.in + row * (int64_t)c.width;
        switch (c.width) {
            case 8: h = mix64(h ^ *(const uint64_t*)p); break;
            case 4: h = mix64(h ^ *(const uint32_t*)p); break;
            case 2: h = mix64(h ^ *(const uint16_t*)p); break;
            case 1: h = mix64(h ^ *(const uint8_t*)p); break;
            default: h = mix64(mix64(h ^ ((const uint64_t*)p)[0]) ^ ((const uint64_t*)p)[1]); break;
        }
    }
    return h;
}

__device__ __forceinline__ bool keys_equal(const ReduceParams& P, int64_t a, int64_t b) {
    for (int k = 0; k < P.n_keys; ++k) {
        const ReduceCol& c = P.col[P.key_idx[k]];
        const char* pa = c.in + a * (int64_t)c.width;
        const char* pb = c.in + b * (int64_t)c.width;
        bool eq;
        switch (c.width) {
            case 8: eq = *(const uint64_t*)pa == *(const uint64_t*)pb; break;
            case 4: eq = *(const uint32_t*)pa == *(const uint32_t*)pb; break;
            case 2: eq = *(const uint16_t*)pa == *(const uint16_t*)pb; break;
            case 1: eq = *pa == *pb; break;
            default: eq = ((const uint64_t*)pa)[0] == ((const uint64_t*)pb)[0] && ((const uint64_t*)pa)[1] == ((const uint64_t*)pb)[1]; break;
        }
        if (!eq) return false;
    }
    return true;
}

__device__ __forceinline__ uint32_t partition_of(const int64_t* starts, uint32_t N, int64_t row) {
    uint32_t lo = 0, hi = N;  // last p with starts[p] <= row
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (starts[mid] <= row) lo = mid; else hi = mid;
    }
    return lo;
}

// Bit pattern of a double <-> an int64 whose signed order is IEEE-754 totalOrder (Rust's f64::total_cmp):
// -NaN < -inf < ... < -0.0 < +0.0 < ... < +inf < +NaN.  Negative values get their 63 low bits flipped; the map is its own
// inverse.  MIN / MAX of these integers is an exact fold, so float MIN / MAX states do not depend on the atomics' order.
__device__ __forceinline__ long long f64_total_order(long long b) {
    return b ^ (long long)((unsigned long long)(b >> 63) >> 1);
}

__global__ void __launch_bounds__(256) k_group_insert(const __grid_constant__ ReduceParams P) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < P.n_rows; row += (int64_t)gridDim.x * blockDim.x) {
        // the row's input partition is [lo, hi): only a representative inside it can be the row's group
        const uint32_t p = partition_of(P.part_starts, P.N, row);
        const int64_t lo = p == 0 ? 0 : P.part_starts[p];
        const int64_t hi = p + 1 == P.N ? P.n_rows : P.part_starts[p + 1];
        // the partition shifts the start slot, so equal keys of different partitions do not share a probe chain
        uint32_t s = (uint32_t)(key_hash(P, row) + (uint64_t)p * 0x9e3779b97f4a7c15ULL) & P.table_mask;
        for (;;) {
            uint32_t rep = P.table[s];
            if (rep == SLOT_EMPTY) {
                rep = atomicCAS(P.table + s, SLOT_EMPTY, (uint32_t)row);
                if (rep == SLOT_EMPTY) break;  // this row represents a new group
            }
            if ((int64_t)rep >= lo && (int64_t)rep < hi && keys_equal(P, (int64_t)rep, row)) break;
            s = (s + 1) & P.table_mask;
        }
        P.row_slot[row] = s;
    }
}

__global__ void __launch_bounds__(256) k_group_count(const __grid_constant__ ReduceParams P) {
    for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s <= (int64_t)P.table_mask; s += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t rep = P.table[s];
        if (rep != SLOT_EMPTY) atomicAdd(P.group_count + partition_of(P.part_starts, P.N, (int64_t)rep), 1ULL);
    }
}

__device__ __forceinline__ void state_init(const ReduceCol& c, char* dst) {
    switch (c.op) {
        case DFD_AGG_SUM_I64: case DFD_AGG_SUM_F64: *(uint64_t*)dst = 0; break;
        case DFD_AGG_SUM_I128: ((uint64_t*)dst)[0] = 0; ((uint64_t*)dst)[1] = 0; break;
        case DFD_AGG_MIN_I64: *(long long*)dst = 0x7fffffffffffffffLL; break;
        case DFD_AGG_MAX_I64: *(long long*)dst = (long long)0x8000000000000000ULL; break;
        // float MIN / MAX states live in the totalOrder image until k_group_finish
        case DFD_AGG_MIN_F64: *(long long*)dst = 0x7fffffffffffffffLL; break;
        case DFD_AGG_MAX_F64: *(long long*)dst = (long long)0x8000000000000000ULL; break;
    }
}

__global__ void __launch_bounds__(256) k_group_place(const __grid_constant__ ReduceParams P) {
    for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s <= (int64_t)P.table_mask; s += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t rep = P.table[s];
        if (rep == SLOT_EMPTY) continue;
        const uint32_t p = partition_of(P.part_starts, P.N, (int64_t)rep);
        const int64_t o = P.out_starts[p] + (int64_t)atomicAdd(P.cursor + p, 1ULL);
        P.slot_out[s] = (uint32_t)o;
        for (int c = 0; c < P.n_cols; ++c) {
            const ReduceCol& col = P.col[c];
            char* dst = col.out + o * (int64_t)col.width;
            if (col.op < 0) {
                const char* src = col.in + (int64_t)rep * col.width;
                for (int b = 0; b < col.width; ++b) dst[b] = src[b];
            } else {
                state_init(col, dst);
            }
        }
    }
}

__global__ void __launch_bounds__(256) k_group_combine(const __grid_constant__ ReduceParams P) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < P.n_rows; row += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o = (int64_t)P.slot_out[P.row_slot[row]];
        for (int c = 0; c < P.n_cols; ++c) {
            const ReduceCol& col = P.col[c];
            if (col.op < 0) continue;
            const char* src = col.in + row * (int64_t)col.width;
            char* dst = col.out + o * (int64_t)col.width;
            switch (col.op) {
                case DFD_AGG_SUM_I64: atomicAdd((unsigned long long*)dst, *(const unsigned long long*)src); break;
                case DFD_AGG_SUM_F64: atomicAdd((double*)dst, *(const double*)src); break;
                case DFD_AGG_MIN_I64: atomicMin((long long*)dst, *(const long long*)src); break;
                case DFD_AGG_MAX_I64: atomicMax((long long*)dst, *(const long long*)src); break;
                case DFD_AGG_MIN_F64: atomicMin((long long*)dst, f64_total_order(*(const long long*)src)); break;
                case DFD_AGG_MAX_F64: atomicMax((long long*)dst, f64_total_order(*(const long long*)src)); break;
                case DFD_AGG_SUM_I128: {
                    // two's complement 128-bit add as two 64-bit atomics: each add propagates its OWN carry exactly once
                    const unsigned long long lo = ((const unsigned long long*)src)[0], hi = ((const unsigned long long*)src)[1];
                    const unsigned long long old = atomicAdd((unsigned long long*)dst, lo);
                    const unsigned long long carry = (old + lo) < old ? 1ULL : 0ULL;
                    atomicAdd((unsigned long long*)dst + 1, hi + carry);
                    break;
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256) k_group_finish(const __grid_constant__ ReduceParams P, int64_t n_out) {
    for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < n_out; o += (int64_t)gridDim.x * blockDim.x) {
        for (int c = 0; c < P.n_cols; ++c) {
            const ReduceCol& col = P.col[c];
            if (col.op != DFD_AGG_MIN_F64 && col.op != DFD_AGG_MAX_F64) continue;
            long long* dst = (long long*)(col.out + o * 8);
            *dst = f64_total_order(*dst);
        }
    }
}

}  // namespace

extern "C" int dfd_partial_reduce_device(dfd_ctx* c, const dfd_column* in_cols, int n_cols, int64_t n_rows, const int32_t* key_cols, int n_keys,
                                         const int32_t* agg_ops, const int64_t* part_starts_device, uint32_t num_partitions,
                                         const dfd_column* out_cols, int64_t* out_part_starts_host, int64_t* out_part_starts_device) {
    if (!c || !in_cols || !out_cols || !key_cols || !agg_ops || !part_starts_device || !out_part_starts_host)
        return set_error(DFD_ERR_INVALID_ARGUMENT, "dfd_partial_reduce_device: NULL argument");
    if (n_cols < 1 || n_cols > MAX_REDUCE_COLS || n_keys < 1 || n_keys > MAX_KEYS || n_rows < 0 || n_rows >= 0xffffffffLL || num_partitions < 1)
        return set_error(DFD_ERR_INVALID_ARGUMENT, "dfd_partial_reduce_device: bad sizes (columns <= %d, keys <= %d, rows < 2^32)", MAX_REDUCE_COLS, MAX_KEYS);
    ReduceParams P{};
    P.n_cols = n_cols;
    P.n_keys = n_keys;
    P.n_rows = n_rows;
    P.N = num_partitions;
    for (int k = 0; k < n_keys; ++k) {
        if (key_cols[k] < 0 || key_cols[k] >= n_cols || agg_ops[key_cols[k]] >= 0)
            return set_error(DFD_ERR_INVALID_ARGUMENT, "key column %d out of range or carries an aggregate", key_cols[k]);
        P.key_idx[k] = key_cols[k];
    }
    for (int i = 0; i < n_cols; ++i) {
        const dfd_column& ic = in_cols[i];
        if (ic.kind != DFD_COL_FIXED || ic.validity || out_cols[i].kind != DFD_COL_FIXED || out_cols[i].width != ic.width)
            return set_error(DFD_ERR_UNSUPPORTED, "column %d: partial reduce moves fixed-width non-null columns (keys and aggregate states)", i);
        const int op = agg_ops[i];
        bool is_key = false;
        for (int k = 0; k < n_keys; ++k) is_key |= key_cols[k] == i;
        if (op < 0 && !is_key) return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d is neither a group key nor an aggregate state", i);
        const int need = op < 0 ? ic.width : (op == DFD_AGG_SUM_I128 ? 16 : 8);
        if (op > DFD_AGG_MAX_F64 || ic.width != need || (op < 0 && ic.width != 1 && ic.width != 2 && ic.width != 4 && ic.width != 8 && ic.width != 16))
            return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: aggregate op %d does not match value width %d", i, op, ic.width);
        P.col[i] = ReduceCol{(const char*)ic.values + ic.offset * (int64_t)ic.width, (char*)out_cols[i].values, ic.width, op};
        if (!ic.values || !out_cols[i].values) return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: values is NULL", i);
    }
    std::lock_guard<std::mutex> lk(c->mu);
    cudaError_t e = cudaSetDevice(c->device);
    if (e != cudaSuccess) return cuda_error(e, "cudaSetDevice");
    cudaStream_t s = c->stream;
    const uint32_t N = num_partitions;
    if (n_rows == 0) {
        for (uint32_t p = 0; p <= N; ++p) out_part_starts_host[p] = 0;
        if (out_part_starts_device && (e = cudaMemsetAsync(out_part_starts_device, 0, sizeof(int64_t) * (N + 1), s)) != cudaSuccess)
            return cuda_error(e, "cudaMemsetAsync");
        return DFD_OK;
    }
    uint64_t slots = 64;
    while (slots < (uint64_t)n_rows * 2) slots <<= 1;  // load factor <= 0.5
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t table_b = al(slots * 4), rowslot_b = al((size_t)n_rows * 4), small_b = al((size_t)(3 * N + 2) * 8);
    int rc = c->var_scratch.ensure(2 * table_b + rowslot_b + small_b + 256, c->device);
    if (rc) return rc;
    char* base = (char*)c->var_scratch.ptr;
    P.table = (uint32_t*)base;
    P.slot_out = (uint32_t*)(base + table_b);
    P.row_slot = (uint32_t*)(base + 2 * table_b);
    P.group_count = (unsigned long long*)(base + 2 * table_b + rowslot_b);
    P.cursor = P.group_count + N;
    P.out_starts = (int64_t*)(P.cursor + N);
    P.part_starts = part_starts_device;
    P.table_mask = (uint32_t)(slots - 1);
    if ((e = cudaMemsetAsync(P.table, 0xff, slots * 4, s)) != cudaSuccess) return cuda_error(e, "cudaMemsetAsync(table)");
    if ((e = cudaMemsetAsync(P.group_count, 0, small_b, s)) != cudaSuccess) return cuda_error(e, "cudaMemsetAsync(counters)");
    const unsigned grid = (unsigned)(c->sm_count * 8);
    k_group_insert<<<grid, 256, 0, s>>>(P);
    k_group_count<<<grid, 256, 0, s>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_error(e, "k_group_insert / k_group_count");
    std::vector<unsigned long long> counts(N);
    if ((e = cudaMemcpyAsync(counts.data(), P.group_count, sizeof(unsigned long long) * N, cudaMemcpyDeviceToHost, s)) != cudaSuccess ||
        (e = cudaStreamSynchronize(s)) != cudaSuccess)
        return cuda_error(e, "partial reduce: group counts");
    out_part_starts_host[0] = 0;
    for (uint32_t p = 0; p < N; ++p) out_part_starts_host[p + 1] = out_part_starts_host[p] + (int64_t)counts[p];
    if ((e = cudaMemcpyAsync(P.out_starts, out_part_starts_host, sizeof(int64_t) * (N + 1), cudaMemcpyHostToDevice, s)) != cudaSuccess)
        return cuda_error(e, "H2D out_starts");
    if (out_part_starts_device &&
        (e = cudaMemcpyAsync(out_part_starts_device, out_part_starts_host, sizeof(int64_t) * (N + 1), cudaMemcpyHostToDevice, s)) != cudaSuccess)
        return cuda_error(e, "H2D out_starts");
    k_group_place<<<grid, 256, 0, s>>>(P);
    k_group_combine<<<grid, 256, 0, s>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_error(e, "k_group_place / k_group_combine");
    c->metrics.kernel_launches += 4;
    bool float_min_max = false;
    for (int i = 0; i < n_cols; ++i) float_min_max |= agg_ops[i] == DFD_AGG_MIN_F64 || agg_ops[i] == DFD_AGG_MAX_F64;
    if (float_min_max) {
        k_group_finish<<<grid, 256, 0, s>>>(P, out_part_starts_host[N]);
        if ((e = cudaGetLastError()) != cudaSuccess) return cuda_error(e, "k_group_finish");
        c->metrics.kernel_launches += 1;
    }
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return cuda_error(e, "partial reduce");  // (out_part_starts_host is caller memory)
    return DFD_OK;
}
