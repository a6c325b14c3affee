// dfd_kernels.cuh — sm_100a kernels of the hash-repartition hot path.
//
// Replaces the CPU inner loop of DataFusion's RepartitionExec(Hash) that the
// reference runs on every producer worker (src/worker/impl_execute_task.rs:77-86):
//   create_hashes -> `hash % N` -> per-destination index vectors -> take per column
// with three device passes over Arrow columnar buffers:
//   K1 k_tile_hist     hash(keys) -> destination -> per-tile radix histogram
//   K1b k_scan_tiles                   exclusive scans -> per-(tile,destination) write cursors
//   K2 k_scatter       fused hash -> stable rank (warp match/ballot) -> shared-memory
//                      staging of each column in destination order -> coalesced run writes
// Integer / byte work bounded by HBM bandwidth; no tensor cores.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <type_traits>

#include "dfd_hash.cuh"
#include "dfd_types.cuh"

namespace dfd {

// ---------------------------------------------------------------------------
// small block-scan helper: exclusive scan of one value per thread
// ---------------------------------------------------------------------------
// BAR == 0: __syncthreads(); BAR > 0: named barrier BAR over the first THREADS threads of the CTA (the
// consumer warps of a warp-specialised kernel; the producer warp never joins it)
template <int THREADS, int BAR>
__device__ __forceinline__ void block_sync() {
    if constexpr (BAR == 0) __syncthreads();
    else asm volatile("bar.sync %0, %1;" ::"n"(BAR), "n"(THREADS) : "memory");
}

template <int THREADS, int BAR = 0>
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* s_warp /*[THREADS/32 + 1]*/,
                                                         uint32_t& block_total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) s_warp[w] = inc;
    block_sync<THREADS, BAR>();
    if (w == 0) {
        uint32_t x = lane < THREADS / 32 ? s_warp[lane] : 0;
        uint32_t xi = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, xi, d);
            if (lane >= d) xi += t;
        }
        if (lane < THREADS / 32) s_warp[lane] = xi - x;
        if (lane == 31) s_warp[THREADS / 32] = xi;
    }
    block_sync<THREADS, BAR>();
    uint32_t res = s_warp[w] + inc - v;
    block_total = s_warp[THREADS / 32];
    block_sync<THREADS, BAR>();
    return res;
}

// Lanes of the warp holding the same destination id `d` (d < 2^nbits), from
// nbits ballots (fully unrolled per bit count; nbits is warp-uniform).
template <int NB>
__device__ __forceinline__ unsigned peers_of_t(uint32_t d) {
    unsigned peers = 0xffffffffu;
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        unsigned bit = (d >> b) & 1u;
        unsigned bal = __ballot_sync(0xffffffffu, bit);
        peers &= bal ^ (bit - 1u);  // bit ? bal : ~bal
    }
    return peers;
}

__device__ __forceinline__ unsigned peers_of(uint32_t d, int nbits) {
    switch (nbits) {
        case 1: return peers_of_t<1>(d);
        case 2: return peers_of_t<2>(d);
        case 3: return peers_of_t<3>(d);
        case 4: return peers_of_t<4>(d);
        case 5: return peers_of_t<5>(d);
        case 6: return peers_of_t<6>(d);
        case 7: return peers_of_t<7>(d);
        case 8: return peers_of_t<8>(d);
        default: return __match_any_sync(0xffffffffu, d);
    }
}

// ---------------------------------------------------------------------------
// K0 (debug / parity): destination id per row
// ---------------------------------------------------------------------------
static __global__ void k_partition_ids(KeySet keys, HashState st, ModN mod, int64_t n_rows, uint32_t* __restrict__ dest) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += (int64_t)gridDim.x * blockDim.x)
        dest[r] = mod_n(row_hash<false>(keys, r, st), mod);
}

// create_hashes over the given key columns, raw 64-bit hashes (used for dictionary VALUES: DataFusion's hash_dictionary
// hashes the values array once and rows pick dict_hashes[index]; also a parity hook for create_hashes itself)
static __global__ void k_row_hashes(KeySet keys, HashState st, int64_t n_rows, uint64_t* __restrict__ out) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += (int64_t)gridDim.x * blockDim.x)
        out[r] = row_hash<false>(keys, r, st);
}

// ---------------------------------------------------------------------------
// K1: per-tile destination histogram.  Tile t covers rows [t*T, (t+1)*T) —
// the same tiling K2 uses.  hist is destination-major ([N][n_tiles]) so the
// tile scan reads contiguously.
//   NF > 0 : N <= 4*NF.  Each thread counts its K rows into NF packed u64
//            accumulators (four 16-bit fields each), one xor-shuffle tree per
//            warp adds them up and lanes 0..N-1 publish the fields: ~6
//            integer instructions per row instead of a ballot cascade.
//   NF == 0: any N.  Warp-aggregated shared-memory atomics (ballot peers).
// ---------------------------------------------------------------------------
template <int THREADS, int K, bool FAST_I64, int NF>
__global__ void __launch_bounds__(THREADS) k_tile_hist(KeySet keys, HashState st, ModN mod, int64_t n_rows,
                                                        int64_t n_tiles, uint32_t N, uint32_t* __restrict__ hist,
                                                        uint16_t* __restrict__ dest_cache /* nullptr: do not cache */) {
    constexpr int T = THREADS * K;
    static_assert(K * 32 < 65536, "16-bit packed counters");
    extern __shared__ uint32_t s_hist[];
    const int lane = threadIdx.x & 31;
    const int nbits = 32 - __clz(N);  // ids 0..N (N = "no row")
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        for (uint32_t p = threadIdx.x; p < N; p += THREADS) s_hist[p] = 0;
        __syncthreads();
        const int64_t row0 = tile * T;
        const int tile_rows = (int)((n_rows - row0) < T ? (n_rows - row0) : T);
        uint32_t d[K];
        if (tile_rows == T) {  // full tile (all but the last): no per-row bounds predicates
#pragma unroll
            for (int j = 0; j < K; ++j) d[j] = mod_n(row_hash<FAST_I64>(keys, row0 + j * THREADS + (int)threadIdx.x, st), mod);
        } else {
#pragma unroll
            for (int j = 0; j < K; ++j) {
                int t = j * THREADS + (int)threadIdx.x;
                d[j] = t < tile_rows ? mod_n(row_hash<FAST_I64>(keys, row0 + t, st), mod) : N;
            }
        }
        if (!FAST_I64 && dest_cache) {
#pragma unroll
            for (int j = 0; j < K; ++j) {
                int t = j * THREADS + (int)threadIdx.x;
                if (t < tile_rows) dest_cache[row0 + t] = (uint16_t)d[j];
            }
        }
        if constexpr (NF > 0) {
            unsigned long long acc[NF];
#pragma unroll
            for (int q = 0; q < NF; ++q) acc[q] = 0;
#pragma unroll
            for (int j = 0; j < K; ++j) {
                unsigned long long inc = d[j] < N ? 1ULL << ((d[j] & 3u) * 16u) : 0ULL;
#pragma unroll
                for (int q = 0; q < NF; ++q) acc[q] += ((d[j] >> 2) == (uint32_t)q) ? inc : 0ULL;
            }
#pragma unroll
            for (int q = 0; q < NF; ++q) {
#pragma unroll
                for (int sh = 16; sh >= 1; sh >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], sh);
            }
            if ((uint32_t)lane < N) {
                unsigned long long a = acc[0];
#pragma unroll
                for (int q = 1; q < NF; ++q) a = ((lane >> 2) == q) ? acc[q] : a;
                uint32_t c = (uint32_t)(a >> ((lane & 3) * 16)) & 0xffffu;
                if (c) atomicAdd(&s_hist[lane], c);
            }
        } else {
#pragma unroll
            for (int j = 0; j < K; ++j) {
                unsigned peers = peers_of(d[j], nbits);
                if (d[j] < N && (peers & ((1u << lane) - 1)) == 0) atomicAdd(&s_hist[d[j]], __popc(peers));
            }
        }
        __syncthreads();
        for (uint32_t p = threadIdx.x; p < N; p += THREADS) hist[(int64_t)p * n_tiles + tile] = s_hist[p];
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------
// K1b: one block per destination: exclusive scan of its tile counts
// (tile_base, relative to the destination's start), then the LAST block to
// finish turns the N totals into part_starts[N+1].  `done` is a zeroed
// counter the kernel resets for the next call.
// ---------------------------------------------------------------------------
template <int THREADS>
__device__ __forceinline__ unsigned long long block_exclusive_scan_u64(unsigned long long v, unsigned long long* s_warp,
                                                                       unsigned long long& total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned long long inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned long long t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) s_warp[w] = inc;
    __syncthreads();
    if (w == 0) {
        unsigned long long x = lane < THREADS / 32 ? s_warp[lane] : 0;
        unsigned long long xi = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, xi, d);
            if (lane >= d) xi += t;
        }
        if (lane < THREADS / 32) s_warp[lane] = xi - x;
        if (lane == 31) s_warp[32] = xi;
    }
    __syncthreads();
    unsigned long long res = s_warp[w] + inc - v;
    total = s_warp[32];
    __syncthreads();
    return res;
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS) k_scan_tiles(const uint32_t* __restrict__ hist, uint32_t* __restrict__ tile_base,
                                                         int64_t* __restrict__ totals, int64_t* __restrict__ part_starts,
                                                         unsigned* __restrict__ done, int64_t n_tiles, uint32_t N) {
    constexpr int W = THREADS / 32;
    __shared__ unsigned long long s_warp[33];
    __shared__ unsigned long long s_wsum[W];
    __shared__ bool s_last;
    const uint32_t p = blockIdx.x;
    const uint32_t* h = hist + (int64_t)p * n_tiles;
    uint32_t* b = tile_base + (int64_t)p * n_tiles;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    // warp w owns the contiguous tiles [lo, hi); every access is a coalesced 32-wide row
    const int64_t per = ((n_tiles + W - 1) / W + 31) & ~(int64_t)31;
    const int64_t lo = (int64_t)w * per;
    const int64_t hi = lo + per < n_tiles ? lo + per : n_tiles;
    unsigned long long sum = 0;
    for (int64_t i = lo + lane; i < hi; i += 32) sum += h[i];
#pragma unroll
    for (int sh = 16; sh >= 1; sh >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, sh);
    if (lane == 0) s_wsum[w] = sum;
    __syncthreads();
    unsigned long long total = 0, base = 0;
#pragma unroll
    for (int ww = 0; ww < W; ++ww) {
        unsigned long long v = s_wsum[ww];
        if (ww < w) base += v;
        total += v;
    }
    unsigned long long run = base;
    for (int64_t i0 = lo; i0 < hi; i0 += 32) {
        const int64_t i = i0 + lane;
        const uint32_t v = i < hi ? h[i] : 0;
        uint32_t inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += t;
        }
        if (i < hi) b[i] = (uint32_t)(run + inc - v);
        run += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (threadIdx.x == 0) {
        totals[p] = (int64_t)total;
        __threadfence();
        s_last = atomicAdd(done, 1u) == N - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // last block: part_starts[q] = sum(totals[0..q)), part_starts[N] = n_rows
    unsigned long long carry = 0;
    for (uint32_t q0 = 0; q0 < N; q0 += THREADS) {
        uint32_t q = q0 + threadIdx.x;
        unsigned long long v = q < N ? (unsigned long long)((volatile int64_t*)totals)[q] : 0;
        unsigned long long tot;
        unsigned long long ex = block_exclusive_scan_u64<THREADS>(v, s_warp, tot);
        if (q < N) part_starts[q] = (int64_t)(carry + ex);
        carry += tot;
    }
    if (threadIdx.x == 0) {
        part_starts[N] = (int64_t)carry;
        *done = 0;
    }
}

// ---------------------------------------------------------------------------
// K2: fused hash -> stable rank -> staged scatter of every column.
//
// One CTA owns one tile of T = THREADS*K rows.  Warp w owns the contiguous
// rows [w*32K, (w+1)*32K) of the tile and walks them in K rounds of 32, so
// every global load is one fully coalesced 32-lane request.  Ranks come from
// __match_any_sync + running per-warp counters in shared memory (stable: rank
// order == row order), a block scan turns them into positions in a tile-local
// staging buffer sorted by destination, and each column is then (a) scattered
// into the staging buffer and (b) streamed out so that every destination's
// run is written as consecutive, coalesced global stores.
// ---------------------------------------------------------------------------
template <typename V>
struct StageIO {
    static __device__ __forceinline__ V ld(const void* base, int64_t i) { return ((const V*)base)[i]; }
};

constexpr uint32_t SLOT_NONE = 0xffffffffu;

// Payload columns are streamed exactly once: evict-first loads / stores keep the L2 for what is reused
// (the key tiles between phase 1 and the scatter of the same tile, the look-back descriptors).
template <typename V> __device__ __forceinline__ V ld_stream(const V* p) { return __ldcs(p); }
template <typename V> __device__ __forceinline__ void st_stream(V* p, V v) { __stcs(p, v); }

// ROWS == false: slot[k] = (destination << 16 | staging index) for write-out iteration k (or SLOT_NONE)
// ROWS == true : slot[k] = absolute output row of staging index k*THREADS + threadIdx.x (or SLOT_NONE) — local
//                mode with KV == K: no per-store delta lookup, 4 instructions per stored element
template <int THREADS, int K, int KV, typename V, int CHUNK = K, bool ROWS = false>
__device__ __forceinline__ void scatter_fixed_column(const PayloadCol& c, void* stage_raw, int64_t row0, int tile_rows,
                                                     const uint32_t (&ps)[K], const uint32_t (&slot)[KV], const int64_t* delta,
                                                     int t0, void* const* out_base /* per destination (peer mode) or nullptr */) {
    static_assert(K % CHUNK == 0, "CHUNK must divide K");
    V* stage = (V*)stage_raw;
    const V* in = (const V*)c.in + (c.in_offset + row0);  // tile-relative indexing below is 32-bit
    V* out = (V*)c.out;                                    // local mode: delta[] holds absolute output rows
    V v[CHUNK];
#pragma unroll
    for (int j = 0; j < CHUNK; ++j) {
        int t = t0 + j * 32;
        if (t < tile_rows) v[j] = ld_stream(in + t);
    }
    __syncthreads();  // staging buffer free (previous column fully written out)
#pragma unroll
    for (int ch = 0; ch < K / CHUNK; ++ch) {
        if (ch > 0) {
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) {
                int t = t0 + (ch * CHUNK + j) * 32;
                if (t < tile_rows) v[j] = ld_stream(in + t);
            }
        }
#pragma unroll
        for (int j = 0; j < CHUNK; ++j) {
            int t = t0 + (ch * CHUNK + j) * 32;
            if (t < tile_rows) stage[ps[ch * CHUNK + j]] = v[j];
        }
    }
    __syncthreads();  // staging buffer holds the tile in destination order
    if constexpr (ROWS) {
        static_assert(KV == K, "row mode walks the staging buffer linearly");
#pragma unroll
        for (int k = 0; k < K; ++k)
            if (slot[k] != SLOT_NONE) st_stream(out + slot[k], stage[k * THREADS + (int)threadIdx.x]);
    } else {
#pragma unroll
        for (int k = 0; k < KV; ++k) {
            if (slot[k] != SLOT_NONE) {
                const uint32_t i = slot[k] & 0xffffu, p = slot[k] >> 16;
                V* o = out_base ? (V*)out_base[p] : out;  // peer mode: the owner rank's receive window (NVLink store)
                st_stream(o + ((int64_t)i + delta[p]), stage[i]);
            }
        }
    }
}

// bit column (boolean values or a validity bitmap): staged as one byte per row,
// written back with warp-aggregated atomicOr on 32-bit output words.
template <int THREADS, int K, int KV>
__device__ __forceinline__ void scatter_bit_column(const PayloadCol& c, void* stage_raw, int64_t row0, int tile_rows,
                                                   const uint32_t (&ps)[K], const uint32_t (&slot)[KV], const int64_t* delta, int t0) {
    uint8_t* stage = (uint8_t*)stage_raw;
    const uint8_t* in = (const uint8_t*)c.in;
    unsigned* out = (unsigned*)c.out;
    const int lane = threadIdx.x & 31;
    uint8_t v[K];
#pragma unroll
    for (int j = 0; j < K; ++j) {
        int t = t0 + j * 32;
        v[j] = (t < tile_rows) ? (uint8_t)bit_is_set(in, row0 + t + c.in_offset) : 0;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < K; ++j) {
        int t = t0 + j * 32;
        if (t < tile_rows) stage[ps[j]] = v[j];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < KV; ++k) {
        const bool active = slot[k] != SLOT_NONE;
        const uint32_t i = slot[k] & 0xffffu;
        int64_t d = active ? (int64_t)i + delta[slot[k] >> 16] : -1;
        unsigned bit = (active && stage[i]) ? (1u << (d & 31)) : 0u;
        int64_t word = active ? (d >> 5) : -1;
        unsigned peers = __match_any_sync(0xffffffffu, word);
        unsigned merged = __reduce_or_sync(peers, bit);
        if (active && merged && (peers & ((1u << lane) - 1)) == 0) atomicOr(out + word, merged);
    }
}

struct BitColumn {};  // tag: bit-packed column (boolean values / validity bitmap)

// ---- decoupled look-back descriptors (single-pass mode) --------------------
// One 64-bit word per (destination, tile): high half = (call epoch << 2) | state, low half = rows.
// Status and value travel in ONE word, so relaxed loads/stores suffice (Merrill & Garland's
// single-word trick); a word whose epoch is not the current call's reads as "not published", so
// the table never needs clearing between calls.
constexpr uint32_t LB_AGG = 1u;     // value = rows of this tile for the destination
constexpr uint32_t LB_PREFIX = 2u;  // value = rows of tiles 0..this for the destination (inclusive)

__device__ __forceinline__ unsigned long long lb_pack(uint32_t epoch, uint32_t state, uint32_t value) {
    return ((unsigned long long)((epoch << 2) | state) << 32) | value;
}
__device__ __forceinline__ void lb_store(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long lb_load(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// first output row of destination p's region (single-pass mode without an explicit dest_base[])
template <bool PEER>
__device__ __forceinline__ int64_t region_base_of(const ScatterParams& P, uint32_t p) {
    if (P.dest_base) return P.dest_base[p];
    if (PEER) return ((int64_t)(p % P.parts_per_rank) * P.world + P.rank) * P.region_stride;
    return (int64_t)p * P.region_stride;
}

// One instantiation per element type V: a launch moves all columns of one
// width (the host groups them), so the hot instantiation (8-byte values)
// carries no code or registers for the other widths.
// KV: write-out iterations per thread.  KV == K: staging slots are written out
// linearly.  KV > K ("aligned" mode, small N): the write-out walks a virtual slot
// space in which every destination's run is shifted so that each warp's 32 rows
// start on a 32-row (256 B for 8-byte values) boundary of the OUTPUT buffer —
// full-line stores to HBM and full-size write packets over NVLink.
struct ScatterSmem {
    // layout: stage | delta[N] | warp_cnt[W][N] | tile_start[2][N+1] | scan scratch | misc[4] | pos16[2][T] | dest8[2][T] | out_base[N] | vstart[N+1]
    uint32_t off_delta, off_wc, off_ts, off_scan, off_misc, off_pos, off_d8, off_ob, off_vs;
};
template <int THREADS, int K>
__host__ __device__ __forceinline__ ScatterSmem scatter_smem_layout(uint32_t N, uint32_t stage_width, bool onepass) {
    constexpr uint32_t T = THREADS * K, W = THREADS / 32;
    ScatterSmem L;
    L.off_delta = (T * stage_width + 15u) & ~15u;
    L.off_wc = L.off_delta + N * 8u;
    L.off_ts = L.off_wc + W * N * 4u;
    L.off_scan = L.off_ts + (onepass ? 2u : 1u) * (N + 1u) * 4u;
    L.off_misc = L.off_scan + (W + 1u) * 4u;
    L.off_pos = (L.off_misc + 4u * 4u + 3u) & ~3u;
    L.off_d8 = L.off_pos + (onepass ? 2u * T * 2u : 0u);                  // single-pass mode: destination of every staging slot
    L.off_ob = (L.off_d8 + (onepass ? 2u * T : 0u) + 7u) & ~7u;            // peer mode only: per-destination bases
    L.off_vs = L.off_ob + N * 8u;                                          // aligned mode only: virtual run starts
    return L;
}

// which staging slot (and destination) each of this thread's write-out iterations handles
template <int THREADS, int K, int KV, int BAR = 0>
__device__ __forceinline__ void compute_slots(uint32_t (&slot)[KV], uint32_t N, int tile_rows, const uint32_t* tile_start,
                                              const int64_t* delta, uint32_t* vstart, uint32_t* s_scan) {
    if constexpr (KV == K) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            uint32_t i = k * THREADS + threadIdx.x;
            uint32_t lo = 0, hi = N;  // last p with tile_start[p] <= i
            while (hi - lo > 1) {
                uint32_t mid = (lo + hi) >> 1;
                if (tile_start[mid] <= i) lo = mid; else hi = mid;
            }
            slot[k] = i < (uint32_t)tile_rows ? (i | (lo << 16)) : SLOT_NONE;
        }
    } else {
        // virtual run of destination p: [vstart[p], vstart[p+1]) = m_p leading pad + its rows, rounded up to 32,
        // where m_p = (first output row of the run) mod 32
        {
            uint32_t carry = 0;
            for (uint32_t p0 = 0; p0 < N; p0 += THREADS) {
                uint32_t p = p0 + threadIdx.x;
                uint32_t len = 0;
                if (p < N) {
                    uint32_t ts = tile_start[p], cnt = tile_start[p + 1] - ts;
                    uint32_t m = (uint32_t)((int64_t)ts + delta[p]) & 31u;
                    len = cnt ? (m + cnt + 31u) & ~31u : 0u;
                }
                uint32_t tot;
                uint32_t ex = block_exclusive_scan<THREADS, BAR>(len, s_scan, tot);
                if (p < N) vstart[p] = carry + ex;
                carry += tot;
            }
            if (threadIdx.x == 0) vstart[N] = carry;
            block_sync<THREADS, BAR>();
        }
        const uint32_t vtotal = vstart[N];
#pragma unroll
        for (int k = 0; k < KV; ++k) {
            uint32_t vs = k * THREADS + threadIdx.x;
            slot[k] = SLOT_NONE;
            if (vs < vtotal) {
                uint32_t lo = 0, hi = N;  // last p with vstart[p] <= vs
                while (hi - lo > 1) {
                    uint32_t mid = (lo + hi) >> 1;
                    if (vstart[mid] <= vs) lo = mid; else hi = mid;
                }
                uint32_t ts = tile_start[lo], cnt = tile_start[lo + 1] - ts;
                uint32_t m = (uint32_t)((int64_t)ts + delta[lo]) & 31u;
                uint32_t off = vs - vstart[lo] - m;  // wraps for the leading pad
                if (off < cnt) slot[k] = (ts + off) | (lo << 16);
            }
        }
    }
}

// phase 2: every column of the launch through the staging buffer
template <int THREADS, int K, int KV, typename V, bool PEER, bool ROWS = false>
__device__ __forceinline__ void scatter_all_columns(const ScatterParams& P, unsigned char* stage, int64_t row0, int tile_rows,
                                                    const uint32_t (&pos)[K], const uint32_t (&slot)[KV], const int64_t* delta, int t0,
                                                    void** out_base) {
#pragma unroll 1
    for (int c = 0; c < P.n_cols; ++c) {
        const PayloadCol& col = P.cols[c];
        if constexpr (std::is_same<V, BitColumn>::value) {
            scatter_bit_column<THREADS, K, KV>(col, stage, row0, tile_rows, pos, slot, delta, t0);
        } else {
            if (PEER) {
                // (the previous column's write-out reads out_base: the barrier inside
                //  scatter_fixed_column orders this rewrite after it only for the staging
                //  buffer, so fence explicitly)
                __syncthreads();
                for (uint32_t p = threadIdx.x; p < P.N; p += THREADS)
                    out_base[p] = (char*)P.peer_base[p / P.parts_per_rank] + (size_t)col.out;
            }
            scatter_fixed_column<THREADS, K, KV, V, (sizeof(V) == 16 && K % 2 == 0 ? K / 2 : K), ROWS>(col, stage, row0, tile_rows, pos, slot, delta,
                                                                                                 t0, PEER ? out_base : nullptr);
        }
    }
}

// phase 1 of one tile: destination + stable rank of every row.  Returns (dest << 16 | rank in (warp, dest)) per row
// and leaves the per-(warp, destination) counts in warp_cnt[W][N].
template <int THREADS, int K, bool FAST_I64>
__device__ __forceinline__ void rank_rows(const ScatterParams& P, int64_t row0, int tile_rows, int t0, uint32_t* warp_cnt, uint32_t (&pos)[K]) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t N = P.N;
    uint32_t* wc = warp_cnt + (uint32_t)w * N;
    for (uint32_t p = lane; p < N; p += 32) wc[p] = 0;
    __syncwarp();
    const int nbits = 32 - __clz(N);
#pragma unroll
    for (int j = 0; j < K; ++j) {
        int t = t0 + j * 32;
        bool valid = t < tile_rows;
        uint32_t d = N;
        if (valid) d = (!FAST_I64 && P.dest_cache) ? (uint32_t)P.dest_cache[row0 + t] : mod_n(row_hash<FAST_I64>(P.keys, row0 + t, P.st), P.mod);
        unsigned peers = peers_of(d, nbits);
        uint32_t rank = __popc(peers & ((1u << lane) - 1));
        uint32_t base = valid ? wc[d] : 0;
        __syncwarp();
        if (valid && rank == 0) wc[d] = base + __popc(peers);
        __syncwarp();
        pos[j] = (d << 16) | (base + rank);
    }
}

template <int THREADS, int K, int KV, int MIN_CTAS, bool FAST_I64, typename V, bool PEER>
__global__ void __launch_bounds__(THREADS, MIN_CTAS) k_scatter(const __grid_constant__ ScatterParams P) {
    constexpr int T = THREADS * K;
    constexpr int W = THREADS / 32;
    extern __shared__ __align__(128) unsigned char smem[];
    const uint32_t N = P.N;
    const ScatterSmem L = scatter_smem_layout<THREADS, K>(N, (uint32_t)P.stage_width, false);
    unsigned char* stage = smem;
    int64_t* const DELTA = (int64_t*)(smem + L.off_delta);
    uint32_t* const WARP_CNT = (uint32_t*)(smem + L.off_wc);
    uint32_t* const TILE_START = (uint32_t*)(smem + L.off_ts);
    uint32_t* const S_SCAN = (uint32_t*)(smem + L.off_scan);
    if (P.abort_flag && *P.abort_flag) return;  // a receive window / region overflowed: write nothing

    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t tile = blockIdx.x;
    const int64_t row0 = tile * T;
    const int tile_rows = (int)((P.n_rows - row0) < T ? (P.n_rows - row0) : T);
    const int t0 = w * (K * 32) + lane;  // this thread's first tile-relative row; rows t0 + 32*j

    // ---- tile_start / delta from the K1 histogram (independent of phase 1).
    // delta[p] maps a staging slot i to its absolute output row: out_row = i + delta[p]
    {
        uint32_t carry = 0;
        for (uint32_t p0 = 0; p0 < N; p0 += THREADS) {
            uint32_t p = p0 + threadIdx.x;
            uint32_t c = p < N ? P.hist[(int64_t)p * P.n_tiles + tile] : 0;
            uint32_t tot;
            uint32_t ex = block_exclusive_scan<THREADS>(c, S_SCAN, tot);
            if (p < N) {
                uint32_t ts = carry + ex;
                TILE_START[p] = ts;
                DELTA[p] = region_base_of<PEER>(P, p) + (int64_t)P.tile_base[(int64_t)p * P.n_tiles + tile] - (int64_t)ts;
            }
            carry += tot;
        }
        if (threadIdx.x == 0) TILE_START[N] = carry;
    }

    // ---- phase 1: destination + stable rank of every row of the tile
    uint32_t pos[K];  // first: (dest << 16 | rank) ; later: staging position
    rank_rows<THREADS, K, FAST_I64>(P, row0, tile_rows, t0, WARP_CNT, pos);
    __syncthreads();
    // warp_cnt[w][p] -> staging base of (warp w, destination p)
    for (uint32_t p = threadIdx.x; p < N; p += THREADS) {
        uint32_t run = TILE_START[p];
#pragma unroll
        for (int ww = 0; ww < W; ++ww) {
            uint32_t c = WARP_CNT[(uint32_t)ww * N + p];
            WARP_CNT[(uint32_t)ww * N + p] = run;
            run += c;
        }
    }
    __syncthreads();
    {
        const uint32_t* wc = WARP_CNT + (uint32_t)w * N;
#pragma unroll
        for (int j = 0; j < K; ++j) {
            uint32_t d = pos[j] >> 16;
            pos[j] = d < N ? wc[d] + (pos[j] & 0xffffu) : 0;
        }
    }
    uint32_t slot[KV];
    compute_slots<THREADS, K, KV>(slot, N, tile_rows, TILE_START, DELTA, (uint32_t*)(smem + L.off_vs), S_SCAN);
    scatter_all_columns<THREADS, K, KV, V, PEER>(P, stage, row0, tile_rows, pos, slot, DELTA, t0, (void**)(smem + L.off_ob));
}

// ---------------------------------------------------------------------------
// mbarrier + TMA bulk-copy primitives (sm_90+/sm_100a): the producer warp of the single-pass kernel
// streams contiguous column tiles global -> shared with cp.async.bulk (UBLKCP in SASS); completion is
// signalled on an mbarrier by transaction bytes, so no register ever stages a payload load.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* b, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* b, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(b)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must fail the launch (trap -> CUDA error), never hang the GPU.
__device__ __forceinline__ void mbar_wait(unsigned long long* b, uint32_t parity) {
    if (mbar_try_wait(b, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(b, parity)) {
        if (clock64() - t0 > (1LL << 33)) __trap();  // ~4 s at 2 GHz
    }
}
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, unsigned long long* bar, unsigned long long pol,
                                         bool hint) {
    if (hint)
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                         smem_u32(dst_smem)),
                     "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
                     : "memory");
    else
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)), "l"(src),
                     "r"(bytes), "r"(smem_u32(bar))
                     : "memory");
}

// shared-memory layout of k_scatter_onepass
struct OnePassSmem {
    uint32_t off_bars, off_tix, off_delta, off_ob, off_wc, off_ts, off_scan, off_misc, off_vs, off_src, off_d8, total;
};
template <int THREADS, int K, int NB>
__host__ __device__ __forceinline__ OnePassSmem onepass_smem_layout(uint32_t N, uint32_t width, bool peer, bool aligned) {
    constexpr uint32_t T = THREADS * K, W = THREADS / 32;
    OnePassSmem L;
    const uint32_t slot_bytes = (T * width + 127u) & ~127u;  // ring of NB input tiles first (128-B aligned bulk-copy destinations)
    L.off_bars = NB * slot_bytes;                             // full[NB] | empty[NB]
    L.off_tix = L.off_bars + 2u * NB * 8u;                    // tile of the header item in each slot (int64)
    L.off_delta = L.off_tix + NB * 8u;
    L.off_ob = L.off_delta + N * 8u;                          // peer mode: window of every destination's owner
    L.off_wc = L.off_ob + (peer ? N * 8u : 0u);
    L.off_ts = L.off_wc + W * N * 4u;
    L.off_scan = L.off_ts + 2u * (N + 1u) * 4u;
    L.off_misc = L.off_scan + (W + 1u) * 4u;
    L.off_vs = L.off_misc + 4u * 4u;                          // aligned mode: virtual run starts
    L.off_src = (L.off_vs + (aligned ? (N + 1u) * 4u : 0u) + 3u) & ~3u;
    L.off_d8 = L.off_src + 2u * T * 2u;
    L.total = L.off_d8 + 2u * T;
    return L;
}

// ---------------------------------------------------------------------------
// K2', single pass: no K1/K1b; every row is hashed once and every column read once.
//
// Warp-specialised persistent kernel (one CTA per resident slot): THREADS consumer threads + one producer warp.
//  * producer warp: draws tile tickets (atomic, launch order) and streams, per tile, a header item (the key
//    tile when the key is a single non-null 8-byte column) and one item per payload column into a ring of NB
//    shared-memory slots with TMA bulk copies; per-slot full/empty mbarriers — loads run NB-1 items ahead of
//    their use and never occupy registers.
//  * consumers, per tile:
//      phase 1 (on the header item of the NEXT tile): hash -> destination -> stable rank (ballot peers +
//        per-warp counters); the tile's per-destination counts are published as look-back aggregates and
//        the inverse permutation (source row of every destination-ordered slot) is left in shared memory;
//      look-back (current tile): warp w resolves destinations w, w+W, ...: exclusive prefix over the lower
//        tiles' descriptors, 32 predecessors per step.  Because phase 1 of a tile runs a whole tile-time
//        before its look-back, the aggregates below it are always published already;
//      scatter: per column item, slot i of the destination order is gathered from the ring (src row) and
//        stored to its output row — consecutive threads write consecutive rows of a destination's run.
// Order is stable (cursor = sum over lower tiles).  Destinations live in fixed regions (dest_base /
// region_stride); a tile that would overflow a region sets overflow_out and writes nothing — the counts stay
// exact and the host re-runs with exact regions.
// ---------------------------------------------------------------------------
template <int THREADS, int K, int KV, int NB, int MIN_CTAS, bool FAST_I64, typename V, bool PEER>
__global__ void __launch_bounds__(THREADS + 32, MIN_CTAS) k_scatter_onepass(const __grid_constant__ ScatterParams P) {
    constexpr int T = THREADS * K;
    constexpr int W = THREADS / 32;
    constexpr int BAR = 1;  // named barrier of the consumer warps
    constexpr bool ROWS = (KV == K) && !PEER;
    static_assert(!std::is_same<V, BitColumn>::value, "bit columns take the two-pass kernel");
    extern __shared__ __align__(128) unsigned char smem[];
    const uint32_t N = P.N;
    const OnePassSmem L = onepass_smem_layout<THREADS, K, NB>(N, (uint32_t)sizeof(V), PEER, KV != K);
    const uint32_t slot_bytes = ((uint32_t)T * (uint32_t)sizeof(V) + 127u) & ~127u;
    unsigned long long* const FULL = (unsigned long long*)(smem + L.off_bars);
    unsigned long long* const EMPTY = FULL + NB;
    long long* const TIX = (long long*)(smem + L.off_tix);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;

    if (threadIdx.x == 0) {
        for (int i = 0; i < NB; ++i) {
            mbar_init(FULL + i, 1);   // the producer's arrive (+ the bulk copy's transaction bytes)
            mbar_init(EMPTY + i, W);  // one arrive per consumer warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    if (w == W) {
        // =========================== producer warp ===========================
        const unsigned long long pol = l2_policy_evict_first();
        uint32_t seq = 0;
        auto acquire_slot = [&]() -> int {
            const int slot = (int)(seq % NB);
            if (lane == 0) mbar_wait(EMPTY + slot, ((seq / NB) & 1u) ^ 1u);
            __syncwarp();
            return slot;
        };
        // rows [row0, row0 + rows) of a column of `width`-byte values -> ring slot
        auto fill = [&](int slot, const void* base, int64_t first_row, int rows, uint32_t width, bool stream) {
            const char* src = (const char*)base + first_row * (int64_t)width;
            const uint32_t bytes = (uint32_t)rows * width;
            unsigned char* dst = smem + (uint32_t)slot * slot_bytes;
            if ((((uintptr_t)src | (uintptr_t)bytes) & 15u) == 0) {
                if (lane == 0) {
                    mbar_arrive_expect_tx(FULL + slot, bytes);
                    bulk_g2s(dst, src, bytes, FULL + slot, pol, stream);
                }
            } else {  // unaligned Arrow offset / ragged last tile: element-wise copy by the producer lanes
                if (width == 8) for (int e = lane; e < rows; e += 32) ((uint64_t*)dst)[e] = ((const uint64_t*)src)[e];
                else if (width == 4) for (int e = lane; e < rows; e += 32) ((uint32_t*)dst)[e] = ((const uint32_t*)src)[e];
                else if (width == 16) for (int e = lane; e < 2 * rows; e += 32) ((uint64_t*)dst)[e] = ((const uint64_t*)src)[e];
                else for (uint32_t e = lane; e < bytes; e += 32) dst[e] = ((const unsigned char*)src)[e];
                __syncwarp();
                if (lane == 0) mbar_arrive(FULL + slot);
            }
            ++seq;
        };
        auto draw = [&]() -> int64_t {
            unsigned t = 0;
            if (lane == 0) t = atomicAdd(P.lb_ticket, 1u);
            t = __shfl_sync(0xffffffffu, t, 0);
            return (int64_t)t < P.n_tiles ? (int64_t)t : -1;
        };
        auto emit_header = [&](int64_t tile) {
            const int slot = acquire_slot();
            if (lane == 0) TIX[slot] = tile;
            if (FAST_I64 && tile >= 0) {
                const int64_t row0 = tile * T;
                const int rows = (int)((P.n_rows - row0) < T ? (P.n_rows - row0) : T);
                fill(slot, P.keys.col[0].values, row0, rows, 8, false);  // key tile: default L2 policy (re-read as a payload column)
            } else {
                __syncwarp();
                if (lane == 0) mbar_arrive(FULL + slot);
                ++seq;
            }
        };
        int64_t cur = draw();
        emit_header(cur);
        while (cur >= 0) {
            const int64_t nxt = draw();
            emit_header(nxt);
            const int64_t row0 = cur * T;
            const int rows = (int)((P.n_rows - row0) < T ? (P.n_rows - row0) : T);
            for (int c = 0; c < P.n_cols; ++c) {
                // a column wider than the ring's element type (16-byte values in an 8-byte ring) arrives as width / sizeof(V)
                // items of T * sizeof(V) bytes each: consecutive ROW RANGES of the tile — the ring slots stay small enough for
                // 4 resident CTAs whatever the schema
                const uint32_t cw = (uint32_t)P.cols[c].width;
                const int parts = cw > (uint32_t)sizeof(V) ? (int)(cw / (uint32_t)sizeof(V)) : 1;
                const int rows_per = T / parts;
                for (int h = 0; h < parts; ++h) {
                    const int slot = acquire_slot();
                    int rr = rows - h * rows_per;
                    rr = rr < 0 ? 0 : (rr > rows_per ? rows_per : rr);
                    if (rr > 0) {
                        fill(slot, P.cols[c].in, P.cols[c].in_offset + row0 + h * rows_per, rr, cw, true);
                    } else {  // ragged last tile: nothing in this range
                        __syncwarp();
                        if (lane == 0) mbar_arrive(FULL + slot);
                        ++seq;
                    }
                }
            }
            cur = nxt;
        }
        return;
    }

    // ============================== consumer warps ==============================
    int64_t* const DELTA = (int64_t*)(smem + L.off_delta);
    void** const OUT_BASE = (void**)(smem + L.off_ob);
    uint32_t* const WARP_CNT = (uint32_t*)(smem + L.off_wc);
    uint32_t* const S_SCAN = (uint32_t*)(smem + L.off_scan);
    uint32_t* const S_MISC = (uint32_t*)(smem + L.off_misc);  // [0] tile overflow
    const int t0 = w * (K * 32) + lane;  // this thread's first tile-relative row; rows t0 + 32*j
    if (PEER)
        for (uint32_t p = threadIdx.x; p < N; p += THREADS) OUT_BASE[p] = P.peer_base[p / P.parts_per_rank];
    uint32_t cseq = 0;
    auto wait_item = [&]() -> int {
        const int slot = (int)(cseq % NB);
        mbar_wait(FULL + slot, (cseq / NB) & 1u);
        return slot;
    };
    auto release_item = [&](int slot) {
        __syncwarp();
        if (lane == 0) mbar_arrive(EMPTY + slot);
        ++cseq;
    };

    // phase 1 of the tile announced by the next header item, into buffer `buf`; returns the tile (or -1: end of stream)
    auto rank_tile = [&](int buf) -> int64_t {
        const int slot = wait_item();
        const int64_t tile = TIX[slot];
        if (tile < 0) {
            release_item(slot);
            return -1;
        }
        const int64_t row0 = tile * T;
        const int tile_rows = (int)((P.n_rows - row0) < T ? (P.n_rows - row0) : T);
        uint32_t* const TS = (uint32_t*)(smem + L.off_ts) + (uint32_t)buf * (N + 1u);
        uint16_t* const SRC16 = (uint16_t*)(smem + L.off_src) + (uint32_t)buf * T;
        uint8_t* const DEST8 = smem + L.off_d8 + (uint32_t)buf * T;
        uint32_t* wc = WARP_CNT + (uint32_t)w * N;
        for (uint32_t p = lane; p < N; p += 32) wc[p] = 0;
        __syncwarp();
        const int nbits = 32 - __clz(N);
        const uint64_t* keys = (const uint64_t*)(smem + (uint32_t)slot * slot_bytes);
        uint32_t pos[K];  // (dest << 16 | rank within (warp, dest))
#pragma unroll
        for (int j = 0; j < K; ++j) {
            const int t = t0 + j * 32;
            const bool valid = t < tile_rows;
            uint32_t d = N;
            if (valid) {
                const uint64_t h = FAST_I64 ? hash_one_u64(P.st, keys[t]) : row_hash<false>(P.keys, row0 + t, P.st);
                d = mod_n(h, P.mod);
            }
            const unsigned peers = peers_of(d, nbits);
            const uint32_t rank = __popc(peers & ((1u << lane) - 1));
            const uint32_t base = valid ? wc[d] : 0;
            __syncwarp();
            if (valid && rank == 0) wc[d] = base + __popc(peers);
            __syncwarp();
            pos[j] = (d << 16) | (base + rank);
        }
        release_item(slot);  // key tile consumed
        block_sync<THREADS, BAR>();
        // tile counts = sum of the warps' counts; publish them, then turn warp_cnt into staging bases
        uint32_t carry = 0;
        for (uint32_t p0 = 0; p0 < N; p0 += THREADS) {
            const uint32_t p = p0 + threadIdx.x;
            uint32_t c = 0;
            if (p < N) {
#pragma unroll
                for (int ww = 0; ww < W; ++ww) c += WARP_CNT[(uint32_t)ww * N + p];
                // tile 0 has no predecessor: its aggregate IS its inclusive prefix
                lb_store(P.lb_desc + (int64_t)p * P.n_tiles + tile, lb_pack(P.lb_epoch, tile == 0 ? LB_PREFIX : LB_AGG, c));
            }
            uint32_t tot;
            const uint32_t ex = block_exclusive_scan<THREADS, BAR>(c, S_SCAN, tot);
            if (p < N) {
                uint32_t run = carry + ex;
                TS[p] = run;
#pragma unroll
                for (int ww = 0; ww < W; ++ww) {
                    const uint32_t cc = WARP_CNT[(uint32_t)ww * N + p];
                    WARP_CNT[(uint32_t)ww * N + p] = run;
                    run += cc;
                }
            }
            carry += tot;
        }
        if (threadIdx.x == 0) TS[N] = carry;
        block_sync<THREADS, BAR>();
#pragma unroll
        for (int j = 0; j < K; ++j) {
            const uint32_t d = pos[j] >> 16;
            if (d < N) {
                const uint32_t sp = wc[d] + (pos[j] & 0xffffu);  // slot of this row in destination order
                SRC16[sp] = (uint16_t)(t0 + j * 32);
                DEST8[sp] = (uint8_t)d;  // N <= 256 in single-pass mode
            }
        }
        return tile;
    };

    int buf = 0;
    int64_t tile = rank_tile(0);
    if (PEER && P.ready_flags) {
        // every consumer must have released its window (previous shuffle fully read) before the first peer store;
        // the flags were signalled before this kernel started, so this normally falls through — after phase 1 of
        // the first tile, i.e. off the critical path
        if ((int)threadIdx.x < P.world) {
            const long long t_start = clock64();
            unsigned long long v;
            do {
                asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(P.ready_flags + threadIdx.x) : "memory");
                if (v < P.ready_epoch && clock64() - t_start > (1LL << 33)) __trap();
            } while (v < P.ready_epoch);
        }
        block_sync<THREADS, BAR>();
    }
    while (tile >= 0) {
        const int64_t next = rank_tile(buf ^ 1);
        const uint32_t* const TS = (const uint32_t*)(smem + L.off_ts) + (uint32_t)buf * (N + 1u);
        const int64_t row0 = tile * T;
        const int tile_rows = (int)((P.n_rows - row0) < T ? (P.n_rows - row0) : T);
        if (threadIdx.x == 0) S_MISC[0] = 0;
        block_sync<THREADS, BAR>();  // (also: SRC16 / DEST8 of this tile are visible, DELTA is free)
        // ---- decoupled look-back: exclusive prefix of every destination over the lower tiles
        // (a warp owns destinations w, w+W, ...: the first window of predecessor descriptors is loaded for LBQ of them at once,
        //  so their L2 round trips overlap instead of queueing behind each other — with N = 48 that is 6 per warp)
        constexpr int LBQ = 8;
        for (uint32_t p0 = (uint32_t)w; p0 < N; p0 += W * LBQ) {
            unsigned long long first[LBQ];
#pragma unroll
            for (int q = 0; q < LBQ; ++q) {
                const uint32_t p = p0 + (uint32_t)q * W;
                const int64_t idx = tile - 1 - lane;
                first[q] = (p < N && idx >= 0) ? lb_load(P.lb_desc + (int64_t)p * P.n_tiles + idx) : 0ull;
            }
#pragma unroll
            for (int q = 0; q < LBQ; ++q) {
                const uint32_t p = p0 + (uint32_t)q * W;
                if (p >= N) break;
                const uint32_t cnt = TS[p + 1] - TS[p];
                uint32_t excl = 0;
                if (tile > 0) {
                    const unsigned long long* d = P.lb_desc + (int64_t)p * P.n_tiles;
                    int64_t j = tile - 1;  // lane 0 looks at the nearest predecessor
                    unsigned long long v = first[q];
                    for (;;) {
                        const int64_t idx = j - lane;
                        uint32_t st = LB_PREFIX, val = 0;
                        if (idx >= 0) {
                            uint32_t hi = (uint32_t)(v >> 32);
                            while ((hi >> 2) != P.lb_epoch || (hi & 3u) == 0u) {
                                v = lb_load(d + idx);
                                hi = (uint32_t)(v >> 32);
                            }
                            st = hi & 3u;
                            val = (uint32_t)v;
                        }
                        const unsigned pm = __ballot_sync(0xffffffffu, st == LB_PREFIX);
                        const int firstp = __ffs(pm) - 1;  // nearest predecessor with an inclusive prefix (-1: none)
                        excl += __reduce_add_sync(0xffffffffu, (firstp < 0 || lane <= firstp) ? val : 0u);
                        if (pm) break;
                        j -= 32;
                        v = (j - lane) >= 0 ? lb_load(d + (j - lane)) : 0ull;
                    }
                    if (lane == 0) lb_store(P.lb_desc + (int64_t)p * P.n_tiles + tile, lb_pack(P.lb_epoch, LB_PREFIX, excl + cnt));
                }
                if (lane == 0) {
                    const int64_t cap = P.dest_cap ? P.dest_cap[p] : P.region_stride;
                    if ((int64_t)excl + (int64_t)cnt > cap) S_MISC[0] = 1;
                    DELTA[p] = region_base_of<PEER>(P, p) + (int64_t)excl - (int64_t)TS[p];
                    if (P.hist_out) {
                        P.hist_out[(int64_t)p * P.n_tiles + tile] = cnt;
                        P.base_out[(int64_t)p * P.n_tiles + tile] = excl;
                    }
                    if (tile == P.n_tiles - 1) P.totals_out[p] = (int64_t)excl + (int64_t)cnt;
                }
            }
        }
        block_sync<THREADS, BAR>();
        const bool overflow = S_MISC[0] != 0;
        if (overflow && threadIdx.x == 0) *P.overflow_out = 1;  // a region is too small: this tile writes nothing
        const uint16_t* const SRC16 = (const uint16_t*)(smem + L.off_src) + (uint32_t)buf * T;
        const uint8_t* const DEST8 = smem + L.off_d8 + (uint32_t)buf * T;
        if constexpr (ROWS) {
            // absolute output row (< 2^32: host-checked) and source row of every slot this thread writes
            uint32_t orow[K], src[K];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const uint32_t i = k * THREADS + threadIdx.x;
                const bool on = i < (uint32_t)tile_rows && !overflow;
                orow[k] = on ? i + (uint32_t)DELTA[DEST8[i]] : SLOT_NONE;
                src[k] = on ? SRC16[i] : 0;
            }
#pragma unroll 1
            for (int c = 0; c < P.n_cols; ++c) {
                void* out_raw = P.cols[c].out;
                const int cw = P.cols[c].width;
                const int parts = cw > (int)sizeof(V) ? cw / (int)sizeof(V) : 1;  // (see the producer: wide columns come in row ranges)
                for (int h = 0; h < parts; ++h) {
                    const int slot = wait_item();
                    const unsigned char* in_raw = smem + (uint32_t)slot * slot_bytes;
                    // one launch moves columns of every width (the rows were ranked once): the element type is per column
                    auto copy_col = [&](auto tag, auto split) {
                        using E = decltype(tag);
                        const E* in = (const E*)in_raw;
                        E* out = (E*)out_raw;
                        if constexpr (decltype(split)::value) {
                            const uint32_t rows_per = (uint32_t)T / (uint32_t)parts, lo = (uint32_t)h * rows_per;
#pragma unroll
                            for (int k = 0; k < K; ++k) {
                                const uint32_t sr = src[k] - lo;  // source row relative to this range (wraps when below it)
                                if (orow[k] != SLOT_NONE && sr < rows_per) st_stream(out + orow[k], in[sr]);
                            }
                        } else {
#pragma unroll
                            for (int k = 0; k < K; ++k)
                                if (orow[k] != SLOT_NONE) st_stream(out + orow[k], in[src[k]]);
                        }
                    };
                    if (parts > 1) {
                        if constexpr (sizeof(V) == 8) copy_col(uint4{}, std::true_type{});  // (the host only sends 16-byte columns this way)
                    } else {
                        switch (cw) {
                            case 16: if constexpr (sizeof(V) >= 16) copy_col(uint4{}, std::false_type{}); break;
                            case 8: if constexpr (sizeof(V) >= 8) copy_col((unsigned long long)0, std::false_type{}); break;
                            case 4: if constexpr (sizeof(V) >= 4) copy_col((unsigned)0, std::false_type{}); break;
                            case 2: if constexpr (sizeof(V) >= 2) copy_col((unsigned short)0, std::false_type{}); break;
                            default: copy_col((unsigned char)0, std::false_type{}); break;
                        }
                    }
                    release_item(slot);
                }
            }
        } else {
            uint32_t slot_of[KV];
            compute_slots<THREADS, K, KV, BAR>(slot_of, N, tile_rows, TS, DELTA, (uint32_t*)(smem + L.off_vs), S_SCAN);
#pragma unroll 1
            for (int c = 0; c < P.n_cols; ++c) {
                const size_t col_out = (size_t)P.cols[c].out;  // local: pointer; peer: byte offset into every window
                const int cw = P.cols[c].width;
                const int parts = cw > (int)sizeof(V) ? cw / (int)sizeof(V) : 1;
                for (int h = 0; h < parts; ++h) {
                    const int slot = wait_item();
                    const unsigned char* in_raw = smem + (uint32_t)slot * slot_bytes;
                    auto copy_col = [&](auto tag, auto split) {
                        using E = decltype(tag);
                        const E* in = (const E*)in_raw;
                        const uint32_t rows_per = (uint32_t)T / (uint32_t)parts, lo = (uint32_t)h * rows_per;
#pragma unroll
                        for (int k = 0; k < KV; ++k) {
                            if (slot_of[k] != SLOT_NONE && !overflow) {
                                const uint32_t i = slot_of[k] & 0xffffu, p = slot_of[k] >> 16;
                                uint32_t sr = SRC16[i];
                                if constexpr (decltype(split)::value) {
                                    sr -= lo;
                                    if (sr >= rows_per) continue;
                                }
                                E* o = PEER ? (E*)((char*)OUT_BASE[p] + col_out) : (E*)col_out;  // peer: the owner's window (NVLink store)
                                st_stream(o + ((int64_t)i + DELTA[p]), in[sr]);
                            }
                        }
                    };
                    if (parts > 1) {
                        if constexpr (sizeof(V) == 8) copy_col(uint4{}, std::true_type{});
                    } else {
                        switch (cw) {
                            case 16: if constexpr (sizeof(V) >= 16) copy_col(uint4{}, std::false_type{}); break;
                            case 8: if constexpr (sizeof(V) >= 8) copy_col((unsigned long long)0, std::false_type{}); break;
                            case 4: if constexpr (sizeof(V) >= 4) copy_col((unsigned)0, std::false_type{}); break;
                            case 2: if constexpr (sizeof(V) >= 2) copy_col((unsigned short)0, std::false_type{}); break;
                            default: copy_col((unsigned char)0, std::false_type{}); break;
                        }
                    }
                    release_item(slot);
                }
            }
        }
        tile = next;
        buf ^= 1;
    }
    // every CTA draws exactly one ticket >= n_tiles; the last CTA out re-arms the counters for the next launch
    if (threadIdx.x == 0 && atomicAdd(P.lb_ticket + 1, 1u) == gridDim.x - 1) {
        P.lb_ticket[0] = 0;
        P.lb_ticket[1] = 0;
    }
}

// ---------------------------------------------------------------------------
// K4: variable-width payload columns (Utf8 / LargeUtf8 / Binary).
// K2 scatters an iota column, giving src[j] = input row of output row j.  Per
// var-width column: gather the string lengths in output order, exclusive-scan
// them into the output offsets (3-phase device scan), then copy the bytes.
// ---------------------------------------------------------------------------
constexpr int VAR_BLOCK = 256;
constexpr int VAR_ITEMS = 8;  // rows per thread in the scan kernels (block = 2048 rows)

static __global__ void k_iota_u32(uint32_t* __restrict__ out, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = (uint32_t)i;
}

template <typename OFF>
__device__ __forceinline__ unsigned long long var_len(const OFF* __restrict__ in_off, int64_t in_offset, uint32_t src) {
    const int64_t j = (int64_t)src + in_offset;
    return (unsigned long long)(in_off[j + 1] - in_off[j]);
}

// phase a: per-block sum of the gathered lengths
template <typename OFF>
__global__ void __launch_bounds__(VAR_BLOCK) k_var_block_sums(const OFF* __restrict__ in_off, int64_t in_offset,
                                                               const uint32_t* __restrict__ src, int64_t n,
                                                               unsigned long long* __restrict__ block_sums) {
    __shared__ unsigned long long s_warp[VAR_BLOCK / 32];
    const int64_t base = (int64_t)blockIdx.x * (VAR_BLOCK * VAR_ITEMS) + (int64_t)threadIdx.x * VAR_ITEMS;
    unsigned long long sum = 0;
#pragma unroll
    for (int k = 0; k < VAR_ITEMS; ++k)
        if (base + k < n) sum += var_len(in_off, in_offset, src[base + k]);
#pragma unroll
    for (int sh = 16; sh >= 1; sh >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, sh);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < VAR_BLOCK / 32; ++w) t += s_warp[w];
        block_sums[blockIdx.x] = t;
    }
}

// phase b: exclusive scan of the block sums in place (single CTA), total -> block_sums[n_blocks]
static __global__ void __launch_bounds__(1024) k_var_scan_block_sums(unsigned long long* __restrict__ block_sums, int64_t n_blocks) {
    __shared__ unsigned long long s_warp[33];
    unsigned long long carry = 0;
    for (int64_t b0 = 0; b0 < n_blocks; b0 += 1024) {
        int64_t b = b0 + threadIdx.x;
        unsigned long long v = b < n_blocks ? block_sums[b] : 0, tot;
        unsigned long long ex = block_exclusive_scan_u64<1024>(v, s_warp, tot);
        if (b < n_blocks) block_sums[b] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) block_sums[n_blocks] = carry;
}

// phase c: output offsets = block base + block-local exclusive scan of the lengths
template <typename OFF>
__global__ void __launch_bounds__(VAR_BLOCK) k_var_write_offsets(const OFF* __restrict__ in_off, int64_t in_offset,
                                                                  const uint32_t* __restrict__ src, int64_t n,
                                                                  const unsigned long long* __restrict__ block_sums,
                                                                  OFF* __restrict__ out_off) {
    __shared__ unsigned long long s_warp[33];
    const int64_t base = (int64_t)blockIdx.x * (VAR_BLOCK * VAR_ITEMS) + (int64_t)threadIdx.x * VAR_ITEMS;
    unsigned long long len[VAR_ITEMS], sum = 0;
#pragma unroll
    for (int k = 0; k < VAR_ITEMS; ++k) {
        len[k] = base + k < n ? var_len(in_off, in_offset, src[base + k]) : 0;
        sum += len[k];
    }
    unsigned long long tot;
    unsigned long long run = block_sums[blockIdx.x] + block_exclusive_scan_u64<VAR_BLOCK>(sum, s_warp, tot);
#pragma unroll
    for (int k = 0; k < VAR_ITEMS; ++k) {
        if (base + k < n) out_off[base + k] = (OFF)run;
        run += len[k];
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) out_off[n] = (OFF)block_sums[gridDim.x];
}

// bytes of output row j <- bytes of input row src[j].  A warp takes 32 consecutive output rows: every lane resolves its
// row's (source offset, length, destination offset) — the three dependent loads src -> offsets -> bytes, 32 rows in flight
// per warp — then the warp copies the non-empty rows one after the other with all 32 lanes on consecutive bytes, so both
// the loads and the stores of a string are coalesced whatever its length (a thread-per-row byte loop is neither, and a
// warp runs as long as its longest string).  LEN_FROM_OUT takes each row's length from the OUTPUT offsets instead, so that a
// row whose output slot is shorter than its source (PartialReduce: a null key written as length 0) copies only that many.
template <typename OFF, bool LEN_FROM_OUT = false>
__global__ void __launch_bounds__(256) k_var_copy_bytes(const OFF* __restrict__ in_off, int64_t in_offset,
                                                         const uint8_t* __restrict__ in_data, const uint32_t* __restrict__ src,
                                                         const OFF* __restrict__ out_off, uint8_t* __restrict__ out_data, int64_t n) {
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t base = ((((int64_t)blockIdx.x * blockDim.x) + threadIdx.x) >> 5) << 5; base < n; base += n_warps << 5) {
        const int64_t j = base + lane;
        int64_t so = 0, dof = 0, len = 0;
        if (j < n) {
            const int64_t r = (int64_t)src[j] + in_offset;
            so = (int64_t)in_off[r];
            dof = (int64_t)out_off[j];
            len = LEN_FROM_OUT ? (int64_t)out_off[j + 1] - dof : (int64_t)in_off[r + 1] - so;
        }
        unsigned todo = __ballot_sync(0xffffffffu, len > 0);
        while (todo) {
            const int l = __ffs(todo) - 1;
            todo &= todo - 1;
            const uint8_t* s = in_data + __shfl_sync(0xffffffffu, so, l);
            uint8_t* d = out_data + __shfl_sync(0xffffffffu, dof, l);
            const int64_t L = __shfl_sync(0xffffffffu, len, l);
            if (L >= 256 && (((uintptr_t)s ^ (uintptr_t)d) & 7) == 0) {  // long, co-aligned: byte head, 8-byte body
                const int64_t head = (int64_t)((8 - ((uintptr_t)d & 7)) & 7);
                if (lane < head) d[lane] = s[lane];
                const int64_t words = (L - head) >> 3;
                const uint64_t* s8 = (const uint64_t*)(s + head);
                uint64_t* d8 = (uint64_t*)(d + head);
                for (int64_t i = lane; i < words; i += 32) d8[i] = s8[i];
                for (int64_t i = head + (words << 3) + lane; i < L; i += 32) d[i] = s[i];
            } else {
                for (int64_t i = lane; i < L; i += 32) d[i] = s[i];
            }
        }
    }
}

// (the peer / aligned tables are last in scatter_smem_layout, so launches that do not use them do not allocate them)
// ---------------------------------------------------------------------------
// Exchange helpers for bit-packed and variable-width columns (NCCL mode): bitmaps travel as one
// byte per row, strings as (lengths, bytes); the receiver rebuilds bitmaps and offsets.
// ---------------------------------------------------------------------------
static __global__ void k_bits_to_bytes(const uint8_t* __restrict__ bits, int64_t bit_offset, int64_t n, uint8_t* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = bit_is_set(bits, i + bit_offset) ? 1 : 0;
}

// out bitmap words are fully written (n rounded up to 32 rows per warp): no pre-zeroing, no atomics
static __global__ void k_bytes_to_bits(const uint8_t* __restrict__ in, int64_t n, unsigned* __restrict__ out_words) {
    const int64_t n32 = (n + 31) & ~(int64_t)31;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n32; i += (int64_t)gridDim.x * blockDim.x) {
        unsigned b = __ballot_sync(0xffffffffu, i < n && in[i] != 0);
        if ((threadIdx.x & 31) == 0) out_words[i >> 5] = b;
    }
}

template <typename OFF>
__global__ void k_offsets_to_lengths(const OFF* __restrict__ off, int64_t n, OFF* __restrict__ len) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) len[i] = off[i + 1] - off[i];
}

// bytes[g] / first[g] of every destination's run of a destination-sorted var-width column
template <typename OFF>
__global__ void k_var_dest_bytes(const OFF* __restrict__ off, const int64_t* __restrict__ part_starts, uint32_t N,
                                 int64_t* __restrict__ bytes, int64_t* __restrict__ first) {
    for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < N; g += gridDim.x * blockDim.x) {
        const int64_t a = (int64_t)off[part_starts[g]], b = (int64_t)off[part_starts[g + 1]];
        bytes[g] = b - a;
        first[g] = a;
    }
}

// lengths -> exclusive offsets, same 3-phase scan as K4 (phase b is k_var_scan_block_sums)
template <typename OFF>
__global__ void __launch_bounds__(VAR_BLOCK) k_len_block_sums(const OFF* __restrict__ len, int64_t n, unsigned long long* __restrict__ block_sums) {
    __shared__ unsigned long long s_warp[VAR_BLOCK / 32];
    const int64_t base = (int64_t)blockIdx.x * (VAR_BLOCK * VAR_ITEMS) + (int64_t)threadIdx.x * VAR_ITEMS;
    unsigned long long sum = 0;
#pragma unroll
    for (int k = 0; k < VAR_ITEMS; ++k)
        if (base + k < n) sum += (unsigned long long)len[base + k];
#pragma unroll
    for (int sh = 16; sh >= 1; sh >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, sh);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < VAR_BLOCK / 32; ++w) t += s_warp[w];
        block_sums[blockIdx.x] = t;
    }
}

template <typename OFF>
__global__ void __launch_bounds__(VAR_BLOCK) k_len_write_offsets(const OFF* __restrict__ len, int64_t n,
                                                                  const unsigned long long* __restrict__ block_sums, OFF* __restrict__ out_off) {
    __shared__ unsigned long long s_warp[33];
    const int64_t base = (int64_t)blockIdx.x * (VAR_BLOCK * VAR_ITEMS) + (int64_t)threadIdx.x * VAR_ITEMS;
    unsigned long long l[VAR_ITEMS], sum = 0;
#pragma unroll
    for (int k = 0; k < VAR_ITEMS; ++k) {
        l[k] = base + k < n ? (unsigned long long)len[base + k] : 0;
        sum += l[k];
    }
    unsigned long long tot;
    unsigned long long run = block_sums[blockIdx.x] + block_exclusive_scan_u64<VAR_BLOCK>(sum, s_warp, tot);
#pragma unroll
    for (int k = 0; k < VAR_ITEMS; ++k) {
        if (base + k < n) out_off[base + k] = (OFF)run;
        run += l[k];
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) out_off[n] = (OFF)block_sums[gridDim.x];
}

template <int THREADS, int K>
inline size_t scatter_smem_bytes(uint32_t N, int stage_width, bool peer, bool aligned, bool onepass = false) {
    const ScatterSmem L = scatter_smem_layout<THREADS, K>(N, (uint32_t)stage_width, onepass);
    size_t off = L.off_ob;
    if (peer || aligned) off += (size_t)N * 8;  // per-destination output bases (peer mode)
    if (aligned) off += (size_t)(N + 1) * 4;    // virtual run starts (aligned mode)
    return off;
}

template <int THREADS, int K, int NB>
inline size_t onepass_smem_bytes(uint32_t N, int width, bool peer, bool aligned) {
    return onepass_smem_layout<THREADS, K, NB>(N, (uint32_t)width, peer, aligned).total;
}

}  // namespace dfd
