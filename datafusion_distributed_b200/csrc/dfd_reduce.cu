// dfd_reduce.cu — device-side PartialReduce ahead of the shuffle.
//
// The reference inserts AggregateExec(mode = PartialReduce) ABOVE the producers' hash RepartitionExec
// (src/distributed_planner/partial_reduce_below_network_shuffles.rs:17-100; plan shape tests/distributed_aggregation.rs:63-67):
// after hash repartitioning, rows with equal group keys sit in the same destination partition, so merging their
// aggregate states there shrinks what crosses the network.  Here the partitioned table is already on the GPU
// (output of dfd_partition_device), so the merge runs on it in place of a PCIe round trip:
//   k_group_insert   open-addressing table of REPRESENTATIVE ROW indices (one u32 per slot): a row claims an empty slot
//                    with atomicCAS or joins the group whose representative has equal keys AND lies in the same input
//                    partition (any number / width of keys — the keys themselves are never copied into the table).
//                    Groups never cross partitions: the caller's part_starts need not follow the group keys.
//   k_group_count    groups per destination partition (representatives only), and the bytes of the string keys the
//                    representatives carry                                          -> exclusive scan (host, N+1 values)
//   k_group_place    every group gets an output row inside its partition; key columns copied, states initialised
//   k_group_combine  every input row folds its non-null states into its group's output row with atomics
//                    (SUM i64 / f64 / i128 (two 64-bit adds with carry), MIN / MAX i64, MIN / MAX f64 in the integer
//                    image of IEEE-754 totalOrder, so the result is the same whatever order the atomics land in)
//   k_group_finish   only with a float MIN / MAX column or a nullable MIN / MAX column: maps float states back from the
//                    totalOrder image to doubles and writes 0 under null MIN / MAX states
//   string keys      K4's lengths -> offsets scan and gather (k_var_copy_bytes, lengths from the output offsets)
// Every kernel has two instantiations: GENERAL = false for fixed-width non-null columns only (the original kernels), and
// GENERAL = true once any column is nullable, Boolean or variable-width (validity bits, bit-packed values, strings).
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
constexpr uint64_t NULL_KEY_TAG = 0x6c62272e07bb0142ULL;  // hashed in place of a null key's value

struct ReduceCol {
    const char* in;            // FIXED: values already advanced by the Arrow offset; BOOL: bitmap; strings: byte buffer
    char* out;                 // FIXED: values; BOOL: bitmap (words); strings: byte buffer
    const uint8_t* in_valid;   // input validity bitmap (bit offset = `offset`) or NULL
    uint32_t* out_valid;       // output validity bitmap (offset 0, 32-bit words) or NULL
    const void* in_off;        // strings: input offsets (index offset + row)
    void* out_off;             // strings: output offsets
    void* out_len;             // strings: [n_rows] output length of every output row (offset width), from var_scratch
    int64_t offset;            // Arrow logical offset of the input (rows / bits)
    int32_t width;             // FIXED: bytes per value
    int32_t op;                // dfd_agg_op, or -1 for a group key
    int32_t kind;              // dfd_col_kind
    int32_t ow;                // strings: offset width (4 / 8)
    int32_t var_slot;          // strings: index into ReduceParams::key_bytes, else -1
    int32_t pad;
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
    // GENERAL only
    unsigned long long* key_bytes;  // [string keys][N] bytes of the representatives' strings per partition
    uint32_t* out_src;      // [n_rows] representative row of every output row (string keys: source of the gather)
    int32_t n_var;          // string key columns
};

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x;
}

__device__ __forceinline__ bool bit_at(const uint8_t* bits, int64_t i) { return (bits[i >> 3] >> (i & 7)) & 1; }

__device__ __forceinline__ bool is_valid(const ReduceCol& c, int64_t row) { return !c.in_valid || bit_at(c.in_valid, c.offset + row); }

__device__ __forceinline__ void set_bit(uint32_t* words, int64_t i) { atomicOr(words + (i >> 5), 1u << (i & 31)); }

__device__ __forceinline__ void var_span(const ReduceCol& c, int64_t row, int64_t& start, int64_t& len) {
    const int64_t j = c.offset + row;
    if (c.ow == 8) {
        const long long* o = (const long long*)c.in_off;
        start = o[j];
        len = o[j + 1] - start;
    } else {
        const int* o = (const int*)c.in_off;
        start = o[j];
        len = (int64_t)o[j + 1] - start;
    }
}

// 8 bytes at an arbitrary address, little endian, from the two aligned words that hold them (a string starts anywhere:
// a 64-bit load at its address would be misaligned).  Both words hold a byte of [p, p + 8), so neither leaves the buffer.
__device__ __forceinline__ uint64_t load8_any(const uint8_t* p) {
    const uintptr_t a = (uintptr_t)p;
    const uint64_t* w = (const uint64_t*)(a & ~(uintptr_t)7);
    const unsigned sh = (unsigned)(a & 7) * 8;
    return sh == 0 ? w[0] : (w[0] >> sh) | (w[1] << (64 - sh));
}

// the last n < 8 bytes, byte by byte (zero-padded)
__device__ __forceinline__ uint64_t load_tail(const uint8_t* p, int n) {
    uint64_t v = 0;
    for (int i = 0; i < n; ++i) v |= (uint64_t)p[i] << (8 * i);
    return v;
}

__device__ __forceinline__ uint64_t hash_fixed(uint64_t h, const char* p, int width) {
    switch (width) {
        case 8: return mix64(h ^ *(const uint64_t*)p);
        case 4: return mix64(h ^ *(const uint32_t*)p);
        case 2: return mix64(h ^ *(const uint16_t*)p);
        case 1: return mix64(h ^ *(const uint8_t*)p);
        default: return mix64(mix64(h ^ ((const uint64_t*)p)[0]) ^ ((const uint64_t*)p)[1]);
    }
}

__device__ __forceinline__ bool fixed_equal(const char* pa, const char* pb, int width) {
    switch (width) {
        case 8: return *(const uint64_t*)pa == *(const uint64_t*)pb;
        case 4: return *(const uint32_t*)pa == *(const uint32_t*)pb;
        case 2: return *(const uint16_t*)pa == *(const uint16_t*)pb;
        case 1: return *pa == *pb;
        default: return ((const uint64_t*)pa)[0] == ((const uint64_t*)pb)[0] && ((const uint64_t*)pa)[1] == ((const uint64_t*)pb)[1];
    }
}

template <bool GENERAL>
__device__ __forceinline__ uint64_t key_hash(const ReduceParams& P, int64_t row) {
    uint64_t h = 0x9e3779b97f4a7c15ULL;
    for (int k = 0; k < P.n_keys; ++k) {
        const ReduceCol& c = P.col[P.key_idx[k]];
        if constexpr (GENERAL) {
            if (!is_valid(c, row)) {  // the bytes under a null are never read
                h = mix64(h ^ NULL_KEY_TAG);
                continue;
            }
            if (c.kind == DFD_COL_BOOL) {
                h = mix64(h ^ (bit_at((const uint8_t*)c.in, c.offset + row) ? 2u : 1u));
                continue;
            }
            if (c.kind != DFD_COL_FIXED) {
                int64_t s, len;
                var_span(c, row, s, len);
                const uint8_t* p = (const uint8_t*)c.in + s;
                h = mix64(h ^ (uint64_t)len);
                int64_t i = 0;
                for (; i + 8 <= len; i += 8) h = mix64(h ^ load8_any(p + i));
                if (i < len) h = mix64(h ^ load_tail(p + i, (int)(len - i)));
                continue;
            }
        }
        h = hash_fixed(h, c.in + row * (int64_t)c.width, c.width);
    }
    return h;
}

template <bool GENERAL>
__device__ __forceinline__ bool keys_equal(const ReduceParams& P, int64_t a, int64_t b) {
    for (int k = 0; k < P.n_keys; ++k) {
        const ReduceCol& c = P.col[P.key_idx[k]];
        if constexpr (GENERAL) {
            const bool va = is_valid(c, a);
            if (va != is_valid(c, b)) return false;
            if (!va) continue;  // NULL == NULL
            if (c.kind == DFD_COL_BOOL) {
                if (bit_at((const uint8_t*)c.in, c.offset + a) != bit_at((const uint8_t*)c.in, c.offset + b)) return false;
                continue;
            }
            if (c.kind != DFD_COL_FIXED) {
                int64_t sa, la, sb, lb;
                var_span(c, a, sa, la);
                var_span(c, b, sb, lb);
                if (la != lb) return false;
                const uint8_t* pa = (const uint8_t*)c.in + sa;
                const uint8_t* pb = (const uint8_t*)c.in + sb;
                int64_t i = 0;
                for (; i + 8 <= la; i += 8)
                    if (load8_any(pa + i) != load8_any(pb + i)) return false;
                if (i < la && load_tail(pa + i, (int)(la - i)) != load_tail(pb + i, (int)(la - i))) return false;
                continue;
            }
        }
        if (!fixed_equal(c.in + a * (int64_t)c.width, c.in + b * (int64_t)c.width, c.width)) return false;
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

template <bool GENERAL>
__global__ void __launch_bounds__(256) k_group_insert(const __grid_constant__ ReduceParams P) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < P.n_rows; row += (int64_t)gridDim.x * blockDim.x) {
        // the row's input partition is [lo, hi): only a representative inside it can be the row's group
        const uint32_t p = partition_of(P.part_starts, P.N, row);
        const int64_t lo = p == 0 ? 0 : P.part_starts[p];
        const int64_t hi = p + 1 == P.N ? P.n_rows : P.part_starts[p + 1];
        // the partition shifts the start slot, so equal keys of different partitions do not share a probe chain
        uint32_t s = (uint32_t)(key_hash<GENERAL>(P, row) + (uint64_t)p * 0x9e3779b97f4a7c15ULL) & P.table_mask;
        for (;;) {
            uint32_t rep = P.table[s];
            if (rep == SLOT_EMPTY) {
                rep = atomicCAS(P.table + s, SLOT_EMPTY, (uint32_t)row);
                if (rep == SLOT_EMPTY) break;  // this row represents a new group
            }
            if ((int64_t)rep >= lo && (int64_t)rep < hi && keys_equal<GENERAL>(P, (int64_t)rep, row)) break;
            s = (s + 1) & P.table_mask;
        }
        P.row_slot[row] = s;
    }
}

template <bool GENERAL>
__global__ void __launch_bounds__(256) k_group_count(const __grid_constant__ ReduceParams P) {
    for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s <= (int64_t)P.table_mask; s += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t rep = P.table[s];
        if (rep == SLOT_EMPTY) continue;
        const uint32_t p = partition_of(P.part_starts, P.N, (int64_t)rep);
        atomicAdd(P.group_count + p, 1ULL);
        if constexpr (GENERAL) {
            for (int k = 0; k < P.n_keys; ++k) {
                const ReduceCol& c = P.col[P.key_idx[k]];
                if (c.var_slot < 0 || !is_valid(c, rep)) continue;
                int64_t st, len;
                var_span(c, rep, st, len);
                if (len > 0) atomicAdd(P.key_bytes + (size_t)c.var_slot * P.N + p, (unsigned long long)len);
            }
        }
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

template <bool GENERAL>
__global__ void __launch_bounds__(256) k_group_place(const __grid_constant__ ReduceParams P) {
    for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s <= (int64_t)P.table_mask; s += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t rep = P.table[s];
        if (rep == SLOT_EMPTY) continue;
        const uint32_t p = partition_of(P.part_starts, P.N, (int64_t)rep);
        const int64_t o = P.out_starts[p] + (int64_t)atomicAdd(P.cursor + p, 1ULL);
        P.slot_out[s] = (uint32_t)o;
        if constexpr (GENERAL) {
            if (P.n_var) P.out_src[o] = rep;
        }
        for (int c = 0; c < P.n_cols; ++c) {
            const ReduceCol& col = P.col[c];
            if constexpr (GENERAL) {
                if (col.op >= 0) {
                    // a state whose input has no validity is never null; one with validity is set by k_group_combine
                    if (col.out_valid && !col.in_valid) set_bit(col.out_valid, o);
                    state_init(col, col.out + o * (int64_t)col.width);
                    continue;
                }
                const bool valid = is_valid(col, rep);
                if (valid && col.out_valid) set_bit(col.out_valid, o);
                if (col.kind == DFD_COL_BOOL) {
                    if (valid && bit_at((const uint8_t*)col.in, col.offset + rep)) set_bit((uint32_t*)col.out, o);
                    continue;
                }
                if (col.kind != DFD_COL_FIXED) {
                    int64_t st = 0, len = 0;
                    if (valid) var_span(col, rep, st, len);
                    if (col.ow == 8) ((long long*)col.out_len)[o] = len;
                    else ((int*)col.out_len)[o] = (int)len;
                    continue;
                }
                char* dst = col.out + o * (int64_t)col.width;
                const char* src = col.in + (int64_t)rep * col.width;
                for (int b = 0; b < col.width; ++b) dst[b] = valid ? src[b] : 0;
            } else {
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
}

template <bool GENERAL>
__global__ void __launch_bounds__(256) k_group_combine(const __grid_constant__ ReduceParams P) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < P.n_rows; row += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o = (int64_t)P.slot_out[P.row_slot[row]];
        for (int c = 0; c < P.n_cols; ++c) {
            const ReduceCol& col = P.col[c];
            if (col.op < 0) continue;
            if constexpr (GENERAL) {
                if (col.in_valid) {
                    if (!bit_at(col.in_valid, col.offset + row)) continue;  // null states are skipped
                    uint32_t* w = col.out_valid + (o >> 5);
                    const uint32_t m = 1u << (o & 31);
                    if (!(*(volatile uint32_t*)w & m)) atomicOr(w, m);  // (most rows find the bit already set)
                }
            }
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

__device__ __forceinline__ bool is_min_max(int op) {
    return op == DFD_AGG_MIN_I64 || op == DFD_AGG_MAX_I64 || op == DFD_AGG_MIN_F64 || op == DFD_AGG_MAX_F64;
}

template <bool GENERAL>
__global__ void __launch_bounds__(256) k_group_finish(const __grid_constant__ ReduceParams P, int64_t n_out) {
    for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < n_out; o += (int64_t)gridDim.x * blockDim.x) {
        for (int c = 0; c < P.n_cols; ++c) {
            const ReduceCol& col = P.col[c];
            long long* dst = (long long*)(col.out + o * 8);
            if constexpr (GENERAL) {
                // a null MIN / MAX state still holds its initial sentinel: write 0 there
                if (is_min_max(col.op) && col.in_valid && !((col.out_valid[o >> 5] >> (o & 31)) & 1)) {
                    *dst = 0;
                    continue;
                }
            }
            if (col.op != DFD_AGG_MIN_F64 && col.op != DFD_AGG_MAX_F64) continue;
            *dst = f64_total_order(*dst);
        }
    }
}

template <bool GENERAL>
void launch_group_kernels(const ReduceParams& P, int phase, unsigned grid, cudaStream_t s, int64_t n_out) {
    if (phase == 0) {
        k_group_insert<GENERAL><<<grid, 256, 0, s>>>(P);
        k_group_count<GENERAL><<<grid, 256, 0, s>>>(P);
    } else if (phase == 1) {
        k_group_place<GENERAL><<<grid, 256, 0, s>>>(P);
        k_group_combine<GENERAL><<<grid, 256, 0, s>>>(P);
    } else {
        k_group_finish<GENERAL><<<grid, 256, 0, s>>>(P, n_out);
    }
}

bool is_var_kind(int kind) { return kind == DFD_COL_UTF8 || kind == DFD_COL_LARGE_UTF8 || kind == DFD_COL_BINARY; }

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
    bool general = false;
    std::vector<int> var_cols;  // string key columns, in var_slot order
    for (int i = 0; i < n_cols; ++i) {
        const dfd_column& ic = in_cols[i];
        const dfd_column& oc = out_cols[i];
        const int op = agg_ops[i];
        const bool var = is_var_kind(ic.kind);
        if (ic.kind != DFD_COL_FIXED && ic.kind != DFD_COL_BOOL && !var)
            return set_error(DFD_ERR_UNSUPPORTED, "column %d: partial reduce takes fixed-width, Boolean and Utf8 / LargeUtf8 / Binary columns", i);
        if (oc.kind != ic.kind || (ic.kind == DFD_COL_FIXED && oc.width != ic.width))
            return set_error(DFD_ERR_UNSUPPORTED, "column %d: output kind / width differs from the input's", i);
        if (ic.validity && !oc.validity)
            return set_error(DFD_ERR_UNSUPPORTED, "column %d: a nullable input needs an output validity bitmap", i);
        if (op >= 0 && ic.kind != DFD_COL_FIXED)
            return set_error(DFD_ERR_UNSUPPORTED, "column %d: aggregate states are fixed-width (no op on Boolean or string columns)", i);
        bool is_key = false;
        for (int k = 0; k < n_keys; ++k) is_key |= key_cols[k] == i;
        if (op < 0 && !is_key) return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d is neither a group key nor an aggregate state", i);
        if (ic.kind == DFD_COL_FIXED) {
            const int need = op < 0 ? ic.width : (op == DFD_AGG_SUM_I128 ? 16 : 8);
            if (op > DFD_AGG_MAX_F64 || ic.width != need || (op < 0 && ic.width != 1 && ic.width != 2 && ic.width != 4 && ic.width != 8 && ic.width != 16))
                return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: aggregate op %d does not match value width %d", i, op, ic.width);
        }
        if (!ic.values || !oc.values) return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: values is NULL", i);
        if (var && (!ic.offsets || !oc.offsets)) return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: offsets is NULL", i);
        if (((uintptr_t)oc.validity & 3) || (ic.kind == DFD_COL_BOOL && ((uintptr_t)oc.values & 3)))
            return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: output bitmaps must be 4-byte aligned", i);
        ReduceCol& rc = P.col[i];
        rc.in = ic.kind == DFD_COL_FIXED ? (const char*)ic.values + ic.offset * (int64_t)ic.width : (const char*)ic.values;
        rc.out = (char*)oc.values;
        rc.in_valid = ic.validity;
        rc.out_valid = (uint32_t*)oc.validity;
        rc.in_off = ic.offsets;
        rc.out_off = oc.offsets;
        rc.offset = ic.offset;
        rc.width = ic.kind == DFD_COL_FIXED ? ic.width : 0;
        rc.op = op;
        rc.kind = ic.kind;
        rc.ow = ic.kind == DFD_COL_LARGE_UTF8 ? 8 : 4;
        rc.var_slot = -1;
        if (var) {
            rc.var_slot = (int32_t)var_cols.size();
            var_cols.push_back(i);
        }
        general |= ic.validity || oc.validity || ic.kind != DFD_COL_FIXED;
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
        for (int i : var_cols)
            if ((e = cudaMemsetAsync(out_cols[i].offsets, 0, (size_t)P.col[i].ow, s)) != cudaSuccess) return cuda_error(e, "cudaMemsetAsync(offsets)");
        return DFD_OK;
    }
    const int V = (int)var_cols.size();
    uint64_t slots = 64;
    while (slots < (uint64_t)n_rows * 2) slots <<= 1;  // load factor <= 0.5
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t table_b = al(slots * 4), rowslot_b = al((size_t)n_rows * 4), small_b = al((size_t)(3 * N + 2 + (size_t)V * N) * 8);
    // string keys: out_src [n_rows] u32 | one length array [n_rows] of the offset width per column | K4 scan block sums
    const size_t src_b = V ? al((size_t)n_rows * 4) : 0;
    const size_t sums_b = V ? al((size_t)(n_rows / 2048 + 2) * 8) : 0;  // (launch_lengths_to_offsets: 2048 rows per block)
    size_t len_b = 0;
    for (int i : var_cols) len_b += al((size_t)n_rows * P.col[i].ow);
    int rc = c->var_scratch.ensure(2 * table_b + rowslot_b + small_b + src_b + len_b + sums_b + 256, c->device);
    if (rc) return rc;
    char* base = (char*)c->var_scratch.ptr;
    P.table = (uint32_t*)base;
    P.slot_out = (uint32_t*)(base + table_b);
    P.row_slot = (uint32_t*)(base + 2 * table_b);
    P.group_count = (unsigned long long*)(base + 2 * table_b + rowslot_b);
    P.cursor = P.group_count + N;
    P.out_starts = (int64_t*)(P.cursor + N);
    P.key_bytes = (unsigned long long*)(P.out_starts + N + 2);
    char* vbase = base + 2 * table_b + rowslot_b + small_b;
    P.out_src = V ? (uint32_t*)vbase : nullptr;
    vbase += src_b;
    for (int i : var_cols) {
        P.col[i].out_len = vbase;
        vbase += al((size_t)n_rows * P.col[i].ow);
    }
    unsigned long long* block_sums = (unsigned long long*)vbase;
    P.n_var = V;
    P.part_starts = part_starts_device;
    P.table_mask = (uint32_t)(slots - 1);
    if ((e = cudaMemsetAsync(P.table, 0xff, slots * 4, s)) != cudaSuccess) return cuda_error(e, "cudaMemsetAsync(table)");
    if ((e = cudaMemsetAsync(P.group_count, 0, small_b, s)) != cudaSuccess) return cuda_error(e, "cudaMemsetAsync(counters)");
    const unsigned grid = (unsigned)(c->sm_count * 8);
    if (general) launch_group_kernels<true>(P, 0, grid, s, 0);
    else launch_group_kernels<false>(P, 0, grid, s, 0);
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_error(e, "k_group_insert / k_group_count");
    // group counts and, for string keys, the representatives' bytes per partition: one copy, one sync
    std::vector<unsigned long long> counts((size_t)N * (1 + V));
    if ((e = cudaMemcpyAsync(counts.data(), P.group_count, sizeof(unsigned long long) * N, cudaMemcpyDeviceToHost, s)) != cudaSuccess ||
        (V && (e = cudaMemcpyAsync(counts.data() + N, P.key_bytes, sizeof(unsigned long long) * N * V, cudaMemcpyDeviceToHost, s)) != cudaSuccess) ||
        (e = cudaStreamSynchronize(s)) != cudaSuccess)
        return cuda_error(e, "partial reduce: group counts");
    for (int v = 0; v < V; ++v) {
        unsigned long long need = 0;
        for (uint32_t p = 0; p < N; ++p) need += counts[(size_t)(1 + v) * N + p];
        const dfd_column& oc = out_cols[var_cols[v]];
        if ((unsigned long long)oc.values_bytes < need)
            return set_error(DFD_ERR_CAPACITY, "column %d: out values_bytes %lld < %llu bytes of group-key strings", var_cols[v],
                             (long long)oc.values_bytes, need);
    }
    out_part_starts_host[0] = 0;
    for (uint32_t p = 0; p < N; ++p) out_part_starts_host[p + 1] = out_part_starts_host[p] + (int64_t)counts[p];
    const int64_t n_out = out_part_starts_host[N];
    if ((e = cudaMemcpyAsync(P.out_starts, out_part_starts_host, sizeof(int64_t) * (N + 1), cudaMemcpyHostToDevice, s)) != cudaSuccess)
        return cuda_error(e, "H2D out_starts");
    if (out_part_starts_device &&
        (e = cudaMemcpyAsync(out_part_starts_device, out_part_starts_host, sizeof(int64_t) * (N + 1), cudaMemcpyHostToDevice, s)) != cudaSuccess)
        return cuda_error(e, "H2D out_starts");
    // bit-packed outputs are written with 32-bit atomic ORs: zero the words of the output rows first
    for (int i = 0; i < n_cols; ++i) {
        const size_t words_b = (size_t)((n_out + 31) / 32) * 4;
        if (out_cols[i].validity && (e = cudaMemsetAsync(out_cols[i].validity, 0, words_b, s)) != cudaSuccess)
            return cuda_error(e, "cudaMemsetAsync(validity)");
        if (in_cols[i].kind == DFD_COL_BOOL && (e = cudaMemsetAsync(out_cols[i].values, 0, words_b, s)) != cudaSuccess)
            return cuda_error(e, "cudaMemsetAsync(boolean values)");
    }
    if (general) launch_group_kernels<true>(P, 1, grid, s, n_out);
    else launch_group_kernels<false>(P, 1, grid, s, n_out);
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_error(e, "k_group_place / k_group_combine");
    c->metrics.kernel_launches += 4;
    bool finish = false;
    for (int i = 0; i < n_cols; ++i)
        finish |= agg_ops[i] == DFD_AGG_MIN_F64 || agg_ops[i] == DFD_AGG_MAX_F64 ||
                  ((agg_ops[i] == DFD_AGG_MIN_I64 || agg_ops[i] == DFD_AGG_MAX_I64) && in_cols[i].validity);
    if (finish) {
        if (general) launch_group_kernels<true>(P, 2, grid, s, n_out);
        else launch_group_kernels<false>(P, 2, grid, s, n_out);
        if ((e = cudaGetLastError()) != cudaSuccess) return cuda_error(e, "k_group_finish");
        c->metrics.kernel_launches += 1;
    }
    // string keys: lengths -> offsets (K4 scan, 3 launches), then the representatives' bytes (1 launch)
    for (int i : var_cols) {
        const ReduceCol& col = P.col[i];
        if ((rc = launch_lengths_to_offsets(col.out_len, col.ow, n_out, block_sums, col.out_off, s))) return rc;
        if ((rc = launch_var_gather(col.in_off, col.ow, col.offset, (const uint8_t*)col.in, P.out_src, col.out_off, (uint8_t*)col.out, n_out, s)))
            return rc;
        c->metrics.kernel_launches += 4;
    }
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return cuda_error(e, "partial reduce");  // (out_part_starts_host is caller memory)
    return DFD_OK;
}
