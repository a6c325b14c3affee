// dfd_api.cu — C ABI (include/dfd_b200.h) over the sm_100a kernels.
// Host side of the producer half of the shuffle: what DataFusion's
// RepartitionExec(Hash) does inside `plan.execute(partition)` on a worker
// (reference: src/worker/impl_execute_task.rs:77-86), re-designed as
// whole-table device passes instead of per-8192-row-batch CPU gathers.
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "dfd_b200.h"
#include "dfd_internal.h"
#include "dfd_kernels.cuh"
#include "dfd_launch.cuh"

namespace dfd {

thread_local std::string g_last_error;

int set_error(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

int cuda_error(cudaError_t e, const char* what) {
    int code = (e == cudaErrorMemoryAllocation) ? DFD_ERR_OOM : DFD_ERR_CUDA;
    return set_error(code, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
}

int Scratch::ensure(size_t need, int device) {
    if (need <= bytes) return DFD_OK;
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    bytes = 0;
    size_t want = need + need / 4;
    cudaError_t e = cudaMalloc(&ptr, want);
    if (e != cudaSuccess) return cuda_error(e, "cudaMalloc(scratch)");
    bytes = want;
    (void)device;
    return DFD_OK;
}

}  // namespace dfd

int dfd_ctx::drain_events() {
    if (ev_pending == 0) return DFD_OK;
    cudaError_t e = cudaEventSynchronize(ev_ring[4 * (ev_pending - 1) + 3]);
    if (e != cudaSuccess) return dfd::cuda_error(e, "partition kernels");
    for (size_t i = 0; i < ev_pending; ++i) {
        cudaEvent_t* ev = &ev_ring[4 * i];
        float a = 0, b = 0, d = 0;
        cudaEventElapsedTime(&a, ev[0], ev[1]);
        cudaEventElapsedTime(&b, ev[1], ev[2]);
        cudaEventElapsedTime(&d, ev[2], ev[3]);
        metrics.hist_ms += a;
        metrics.scan_ms += b;
        metrics.scatter_ms += d;
    }
    ev_pending = 0;
    return DFD_OK;
}

using namespace dfd;

static int build_keyset(const dfd_partitioner* p, const dfd_column* cols, int n_cols, KeySet* ks) {
    memset(ks, 0, sizeof *ks);
    ks->n = (int32_t)p->key_cols.size();
    for (int k = 0; k < ks->n; ++k) {
        int ci = p->key_cols[k];
        if (ci >= n_cols) return set_error(DFD_ERR_INVALID_ARGUMENT, "key column %d out of range (n_cols=%d)", ci, n_cols);
        const dfd_column& c = cols[ci];
        KeyCol& kc = ks->col[k];
        kc.values = c.values;
        kc.offsets = c.offsets;
        kc.validity = c.validity;
        kc.offset = c.offset;
        kc.kind = c.kind;
        kc.width = (int16_t)c.width;
        kc.mode = (int16_t)p->key_modes[k];
        if (kc.mode == KEY_HASH_DICTIONARY) {
            if (c.kind != DFD_COL_FIXED || (c.width != 1 && c.width != 2 && c.width != 4 && c.width != 8))
                return set_error(DFD_ERR_INVALID_ARGUMENT, "key column %d: dictionary indices must be a fixed-width integer column", ci);
            if (!p->key_dicts[k].hashes) return set_error(DFD_ERR_INVALID_ARGUMENT, "key column %d: no dictionary set (dfd_partitioner_set_key_dictionary)", ci);
            kc.offsets = p->key_dicts[k].hashes;
            kc.dict_validity = p->key_dicts[k].validity;
        }
        switch (c.kind) {
            case DFD_COL_FIXED:
                if (c.width != 1 && c.width != 2 && c.width != 4 && c.width != 8 && c.width != 16)
                    return set_error(DFD_ERR_UNSUPPORTED, "key column %d: fixed width %d not in {1,2,4,8,16}", ci, c.width);
                if ((kc.mode == KEY_HASH_INTERVAL_DAY_TIME && c.width != 8) || (kc.mode == KEY_HASH_INTERVAL_MONTH_DAY_NANO && c.width != 16))
                    return set_error(DFD_ERR_INVALID_ARGUMENT, "key column %d: key hash mode %d does not match value width %d", ci, kc.mode, c.width);
                if (!c.values) return set_error(DFD_ERR_INVALID_ARGUMENT, "key column %d: values is NULL", ci);
                break;
            case DFD_COL_BOOL:
                if (!c.values) return set_error(DFD_ERR_INVALID_ARGUMENT, "key column %d: values is NULL", ci);
                break;
            case DFD_COL_UTF8:
            case DFD_COL_LARGE_UTF8:
            case DFD_COL_BINARY:
                if (!c.offsets) return set_error(DFD_ERR_INVALID_ARGUMENT, "key column %d: offsets is NULL", ci);
                break;
            default: return set_error(DFD_ERR_UNSUPPORTED, "key column %d: unknown kind %d", ci, c.kind);
        }
    }
    ks->fast_i64 = (ks->n == 1 && ks->col[0].kind == COL_FIXED && ks->col[0].width == 8 && !ks->col[0].validity &&
                    ks->col[0].offset == 0 && ks->col[0].mode == KEY_HASH_PLAIN)
                       ? 1
                       : 0;
    return DFD_OK;
}

#define LAUNCH_CHECK(what)                                             \
    {                                                                  \
        cudaError_t _e = cudaGetLastError();                           \
        if (_e != cudaSuccess) return cuda_error(_e, what);            \
    }

// Measured on B200 (profiles/): aligned write-out costs ~5% on local HBM stores (more write-out
// iterations, L2 already merges partial lines) but gains ~15% on NVLink peer stores (full-size
// write packets), so it is on for the fused exchange only.  DFD_ALIGNED_WRITEOUT=0/1 forces it.
bool dfd::use_aligned(uint32_t N, bool peer) {
    static const int forced = [] { const char* e = getenv("DFD_ALIGNED_WRITEOUT"); return e ? (atoi(e) != 0 ? 1 : 0) : -1; }();
    if (N > ALIGNED_MAX_N) return false;
    return forced >= 0 ? forced == 1 : peer;
}

// mode: 0 two-pass, 1 single-pass, 2 follow-up of a single-pass launch (see dfd_launch.cuh)
static int launch_scatter(const ScatterParams& sp, int width, bool fast, bool peer, int mode, int sm_count, size_t smem,
                          cudaStream_t stream) {
    if (mode == 1) return peer ? launch_scatter_onepass_peer(sp, width, fast, sm_count, smem, stream)
                               : launch_scatter_onepass_local(sp, width, fast, sm_count, smem, stream);
    if (mode == 2) return peer ? launch_scatter_follow_peer(sp, width, fast, sm_count, smem, stream)
                               : launch_scatter_follow_local(sp, width, fast, sm_count, smem, stream);
    return peer ? launch_scatter_twopass_peer(sp, width, fast, sm_count, smem, stream)
                : launch_scatter_twopass_local(sp, width, fast, sm_count, smem, stream);
}

// ---- PartitionJob: validation -> K1/K1b -> K2, reusable by the local path and the exchange ----

int dfd::PartitionJob::prepare(Partitioner* part, const dfd_column* in_cols, int n_cols, int64_t rows,
                               const dfd_column* out_cols, bool peer_mode, cudaStream_t st) {
    p = part;
    stream = st;
    peer = peer_mode;
    n_rows = rows;
    passes.clear();
    var_cols.clear();
    d_src = nullptr;
    bytes = 0;
    Ctx* c = p->ctx;
    const uint32_t N = p->N;
    if (n_rows < 0 || n_cols < 0 || (n_cols > 0 && (!in_cols || !out_cols)))
        return set_error(DFD_ERR_INVALID_ARGUMENT, "partition: bad arguments");
    if (n_rows > 0xffffffffLL) return set_error(DFD_ERR_UNSUPPORTED, "n_rows must be < 2^32 per call");
    int rc = build_keyset(p, in_cols, n_cols, &ks);
    if (rc) return rc;
    // payload passes: every column's values, plus a bit pass per validity bitmap
    for (int i = 0; i < n_cols; ++i) {
        const dfd_column& ic = in_cols[i];
        const dfd_column& oc = out_cols[i];
        if (ic.kind != oc.kind || ic.width != oc.width)
            return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: in/out layout mismatch", i);
        const bool var_kind = ic.kind == DFD_COL_UTF8 || ic.kind == DFD_COL_LARGE_UTF8 || ic.kind == DFD_COL_BINARY;
        if (!var_kind && (!ic.values || (!peer && !oc.values))) return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: values is NULL", i);
        PayloadCol pc{};
        if (ic.kind == DFD_COL_FIXED) {
            if (ic.width != 1 && ic.width != 2 && ic.width != 4 && ic.width != 8 && ic.width != 16)
                return set_error(DFD_ERR_UNSUPPORTED, "column %d: fixed width %d not in {1,2,4,8,16}", i, ic.width);
            if (((uintptr_t)ic.values | (uintptr_t)oc.values) & (uintptr_t)(ic.width - 1))
                return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: buffers must be aligned to the value width", i);
            pc.in = ic.values;
            pc.out = oc.values;
            pc.in_offset = ic.offset;
            pc.width = ic.width;
            bytes += (uint64_t)n_rows * ic.width;
        } else if (ic.kind == DFD_COL_BOOL) {
            if (peer) return set_error(DFD_ERR_UNSUPPORTED, "column %d: bit-packed columns need the NCCL exchange mode", i);
            if ((uintptr_t)oc.values & 3) return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: output bitmap must be 4-byte aligned", i);
            pc.in = ic.values;
            pc.out = oc.values;
            pc.in_offset = ic.offset;
            pc.width = 0;
            bytes += (uint64_t)(n_rows + 7) / 8;
        } else if (ic.kind == DFD_COL_UTF8 || ic.kind == DFD_COL_LARGE_UTF8 || ic.kind == DFD_COL_BINARY) {
            if (peer) return set_error(DFD_ERR_UNSUPPORTED, "column %d: variable-width columns need the NCCL exchange mode", i);
            if (!ic.offsets || !oc.offsets) return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: offsets is NULL", i);
            // capacity check needs the input's byte count: two small D2H reads and a stream sync — unless the caller built
            // the offsets itself and vouches for in_cols[i].values_bytes (the host operator: a sync here would hold its
            // producer thread until the chunk's H2D has landed, serialising staging with the copies)
            const size_t ow = ic.kind == DFD_COL_LARGE_UTF8 ? 8 : 4;
            int64_t first = 0, last = 0;
            if (var_bytes_known) {
                last = ic.values_bytes;
            } else {
                cudaError_t e = cudaMemcpyAsync(&first, (const char*)ic.offsets + (size_t)ic.offset * ow, ow, cudaMemcpyDeviceToHost, stream);
                if (e == cudaSuccess) e = cudaMemcpyAsync(&last, (const char*)ic.offsets + (size_t)(ic.offset + n_rows) * ow, ow, cudaMemcpyDeviceToHost, stream);
                if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
                if (e != cudaSuccess) return cuda_error(e, "reading variable-width offsets");
                if (ow == 4) { first = (int32_t)first; last = (int32_t)last; }
            }
            const int64_t nbytes = last - first;
            if (nbytes < 0) return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: offsets are not monotonic", i);
            if (oc.values_bytes < nbytes)
                return set_error(DFD_ERR_CAPACITY, "column %d: out values_bytes %lld < %lld bytes of input data", i,
                                 (long long)oc.values_bytes, (long long)nbytes);
            if (nbytes > 0 && (!ic.values || !oc.values)) return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: values is NULL", i);
            var_cols.push_back(VarCol{ic, oc});
            bytes += (uint64_t)nbytes + (uint64_t)(n_rows + 1) * ow;
        } else {
            return set_error(DFD_ERR_UNSUPPORTED, "column %d: unknown column kind %d", i, ic.kind);
        }
        if (ic.kind == DFD_COL_FIXED || ic.kind == DFD_COL_BOOL) passes.push_back(pc);
        if (ic.validity) {
            if (peer) return set_error(DFD_ERR_UNSUPPORTED, "column %d: nullable columns need the NCCL exchange mode", i);
            if (!oc.validity) return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: input has a validity bitmap but out validity is NULL", i);
            if ((uintptr_t)oc.validity & 3) return set_error(DFD_ERR_INVALID_ARGUMENT, "column %d: output validity must be 4-byte aligned", i);
            PayloadCol vc{};
            vc.in = ic.validity;
            vc.out = oc.validity;
            vc.in_offset = ic.offset;
            vc.width = 0;
            passes.push_back(vc);
            bytes += (uint64_t)(n_rows + 7) / 8;
        }
    }
    // bit-packed outputs (boolean values, validity bitmaps) are produced with 32-bit atomicOr: zero them here, in whole
    // words (the header requires capacities of ceil(rows / 32) * 4 bytes), so callers need not pre-clear them
    if (!peer) {
        const int64_t orows = out_rows >= 0 ? out_rows : n_rows;
        for (const PayloadCol& pc : passes)
            if (pc.width == 0 && orows > 0) {
                cudaError_t e = cudaMemsetAsync(pc.out, 0, (size_t)((orows + 31) / 32) * 4, stream);
                if (e != cudaSuccess) return cuda_error(e, "cudaMemsetAsync(bit-packed output)");
            }
    }
    if (!var_cols.empty() && n_rows > 0) {
        // K4 needs the input row of every output row: scatter an iota column with the rest
        const size_t nb = (((size_t)n_rows * 4) + 255) & ~(size_t)255;
        const int64_t n_blocks = (n_rows + VAR_BLOCK * VAR_ITEMS - 1) / (VAR_BLOCK * VAR_ITEMS);
        rc = c->var_scratch.ensure(2 * nb + (size_t)(n_blocks + 1) * 8 + 256, c->device);
        if (rc) return rc;
        uint32_t* d_iota = (uint32_t*)c->var_scratch.ptr;
        d_src = (uint32_t*)((char*)c->var_scratch.ptr + nb);
        d_block_sums = (unsigned long long*)((char*)c->var_scratch.ptr + 2 * nb);
        k_iota_u32<<<(unsigned)(c->sm_count * 8), 256, 0, stream>>>(d_iota, n_rows);
        LAUNCH_CHECK("k_iota_u32");
        c->metrics.kernel_launches++;
        PayloadCol ip{};
        ip.in = d_iota;
        ip.out = d_src;
        ip.in_offset = 0;
        ip.width = 4;
        passes.push_back(ip);
    }
    const int64_t tile_rows = onepass_tiling ? ONEPASS_ROWS : TILE_ROWS;
    n_tiles = n_rows > 0 ? (n_rows + tile_rows - 1) / tile_rows : 1;
    // scratch: hist u32 [N][n_tiles] | tile_base u32 [N][n_tiles] | totals i64 [N] | done u32
    size_t hist_bytes = (((size_t)N * n_tiles * 4) + 255) & ~(size_t)255;
    size_t tot_bytes = (((size_t)N * 8) + 255) & ~(size_t)255;
    // (+ 2 B per row of destination ids when the keys are not the trivial single-i64 case and the launch is two-pass)
    const size_t cache_bytes = (!ks.fast_i64 && !onepass_tiling) ? ((((size_t)n_rows * 2) + 255) & ~(size_t)255) : 0;
    size_t need = 2 * hist_bytes + tot_bytes + 256 + cache_bytes;
    bool fresh = need > c->scratch.bytes;
    rc = c->scratch.ensure(need, c->device);
    if (rc) return rc;
    d_hist = (uint32_t*)c->scratch.ptr;
    d_base = (uint32_t*)((char*)c->scratch.ptr + hist_bytes);
    d_totals = (int64_t*)((char*)c->scratch.ptr + 2 * hist_bytes);
    d_done = (unsigned*)((char*)c->scratch.ptr + 2 * hist_bytes + tot_bytes);
    d_dest_cache = cache_bytes ? (uint16_t*)((char*)c->scratch.ptr + 2 * hist_bytes + tot_bytes + 256) : nullptr;
    if (fresh || c->scratch_done != d_done) {
        cudaError_t e = cudaMemsetAsync(d_done, 0, 256, stream);
        if (e != cudaSuccess) return cuda_error(e, "cudaMemsetAsync(done)");
        c->scratch_done = d_done;
    }
    ev = nullptr;
    if (c->profiling) {
        if (c->ev_ring.empty()) {
            c->ev_ring.resize(4 * dfd_ctx::EV_RING_CALLS);
            for (auto& e : c->ev_ring) cudaEventCreate(&e);
        }
        if (c->ev_pending == dfd_ctx::EV_RING_CALLS) {
            rc = c->drain_events();
            if (rc) return rc;
        }
        ev = &c->ev_ring[4 * c->ev_pending];
    }
    return DFD_OK;
}

// K1 + K1b: d_hist, d_base (tile cursors), d_totals[N] and p->d_part_starts[N+1]
int dfd::PartitionJob::run_hist_scan() {
    Ctx* c = p->ctx;
    const uint32_t N = p->N;
    if (ev) cudaEventRecord(ev[0], stream);
    if (n_rows == 0) {
        cudaError_t e = cudaMemsetAsync(d_totals, 0, sizeof(int64_t) * (size_t)N, stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(p->d_part_starts, 0, sizeof(int64_t) * (size_t)(N + 1), stream);
        if (ev) { cudaEventRecord(ev[1], stream); cudaEventRecord(ev[2], stream); }
        return e == cudaSuccess ? DFD_OK : cuda_error(e, "cudaMemsetAsync");
    }
    {
        size_t smem = (size_t)N * 4;
        const int nf = N <= 4 ? 1 : N <= 8 ? 2 : N <= 16 ? 4 : 0;
        const unsigned grid = (unsigned)n_tiles;
#define HIST(FAST, NF) k_tile_hist<TILE_THREADS, TILE_K, FAST, NF><<<grid, TILE_THREADS, smem, stream>>>(ks, p->st, p->mod, n_rows, n_tiles, N, d_hist, d_dest_cache)
        if (ks.fast_i64) {
            switch (nf) { case 1: HIST(true, 1); break; case 2: HIST(true, 2); break; case 4: HIST(true, 4); break; default: HIST(true, 0); }
        } else {
            switch (nf) { case 1: HIST(false, 1); break; case 2: HIST(false, 2); break; case 4: HIST(false, 4); break; default: HIST(false, 0); }
        }
#undef HIST
        LAUNCH_CHECK("k_tile_hist");
    }
    if (ev) cudaEventRecord(ev[1], stream);
    k_scan_tiles<1024><<<N, 1024, 0, stream>>>(d_hist, d_base, d_totals, p->d_part_starts, d_done, n_tiles, N);
    LAUNCH_CHECK("k_scan_tiles");
    if (ev) cudaEventRecord(ev[2], stream);
    c->metrics.kernel_launches += 2;
    return DFD_OK;
}

// K2.  dest_base[N]: first output row of each destination (p->d_part_starts in local mode).
int dfd::PartitionJob::run_scatter(const int64_t* dest_base, void* const* peer_base, int world, uint32_t parts_per_rank,
                                   const int32_t* abort_flag) {
    Ctx* c = p->ctx;
    const uint32_t N = p->N;
    int launches = 0;
    if (n_rows > 0) {
        ScatterParams sp{};
        sp.keys = ks;
        sp.st = p->st;
        sp.mod = p->mod;
        sp.n_rows = n_rows;
        sp.n_tiles = n_tiles;
        sp.hist = d_hist;
        sp.tile_base = d_base;
        sp.dest_base = dest_base;
        sp.N = N;
        sp.parts_per_rank = parts_per_rank ? parts_per_rank : 1;
        sp.abort_flag = abort_flag;
        sp.dest_cache = d_dest_cache;
        if (peer) {
            if (world > MAX_RANKS) return set_error(DFD_ERR_UNSUPPORTED, "world size %d > %d", world, MAX_RANKS);
            for (int r = 0; r < world; ++r) sp.peer_base[r] = peer_base[r];
        }
        // one launch per element width (0 = bit columns), columns of that width batched
        static const int kWidths[6] = {8, 4, 16, 2, 1, 0};
        for (int wi = 0; wi < 6; ++wi) {
            const int width = kWidths[wi];
            std::vector<PayloadCol> group;
            for (const PayloadCol& pc : passes)
                if (pc.width == width) group.push_back(pc);
            if (group.empty()) continue;
            sp.stage_width = width ? width : 1;
            size_t smem = scatter_smem_bytes<TILE_THREADS, TILE_K>(N, sp.stage_width, peer, use_aligned(N, peer));
            if (smem > 227 * 1024)
                return set_error(DFD_ERR_UNSUPPORTED, "num_partitions %u needs %zu B of shared memory per CTA", N, smem);
            for (size_t first = 0; first < group.size(); first += MAX_COLS_PER_LAUNCH) {
                size_t n = group.size() - first < (size_t)MAX_COLS_PER_LAUNCH ? group.size() - first : (size_t)MAX_COLS_PER_LAUNCH;
                for (size_t i = 0; i < n; ++i) sp.cols[i] = group[first + i];
                sp.n_cols = (int32_t)n;
                int rc = launch_scatter(sp, width, ks.fast_i64 != 0, peer, 0, c->sm_count, smem, stream);
                if (rc) return rc;
                ++launches;
            }
        }
    }
    if (!var_cols.empty()) {
        int rc = run_varwidth();
        if (rc) return rc;
    }
    if (ev) {
        cudaEventRecord(ev[3], stream);
        c->ev_pending++;
        ev = nullptr;
    }
    c->metrics.kernel_launches += launches;
    c->metrics.scatter_launches += launches;
    c->metrics.calls++;
    c->metrics.rows += (uint64_t)n_rows;
    c->metrics.bytes_in += bytes;
    c->metrics.bytes_out += bytes;
    return DFD_OK;
}

// Single-pass partition: ONE k_scatter<ONEPASS> launch hashes, ranks, resolves the tile cursors by
// decoupled look-back and scatters the first width group; further width groups (and bit columns) reuse
// the per-tile counts / cursors it leaves in d_hist / d_base through the two-pass code path.
int dfd::PartitionJob::run_onepass(const OnePassLayout& L) {
    Ctx* c = p->ctx;
    const uint32_t N = p->N;
    if (ev) { cudaEventRecord(ev[0], stream); cudaEventRecord(ev[1], stream); cudaEventRecord(ev[2], stream); }
    if (!var_cols.empty()) return set_error(DFD_ERR_INTERNAL, "single-pass mode does not move variable-width columns");
    int launches = 0;
    if (n_rows == 0) {
        cudaError_t e = cudaMemsetAsync(L.d_totals, 0, sizeof(int64_t) * (size_t)N, stream);
        if (e != cudaSuccess) return cuda_error(e, "cudaMemsetAsync");
    } else {
        const size_t need = 256 + (size_t)N * (size_t)n_tiles * 8;
        bool clear = false;
        if (need > c->lb.bytes) {
            int rc = c->lb.ensure(need, c->device);
            if (rc) return rc;
            clear = true;
        }
        if (++c->lb_epoch >= (1u << 30)) { c->lb_epoch = 1; clear = true; }
        if (clear) {
            cudaError_t e = cudaMemsetAsync(c->lb.ptr, 0, c->lb.bytes, stream);
            if (e != cudaSuccess) return cuda_error(e, "cudaMemsetAsync(look-back table)");
        }
        ScatterParams sp{};
        sp.keys = ks;
        sp.st = p->st;
        sp.mod = p->mod;
        sp.n_rows = n_rows;
        sp.n_tiles = n_tiles;
        sp.N = N;
        sp.parts_per_rank = L.parts_per_rank ? L.parts_per_rank : 1;
        sp.dest_base = L.d_dest_base;
        sp.dest_cap = L.d_dest_cap;
        sp.region_stride = L.region_stride;
        sp.rank = L.rank;
        sp.world = L.world;
        sp.lb_ticket = (unsigned*)c->lb.ptr;
        sp.lb_desc = (unsigned long long*)((char*)c->lb.ptr + 256);
        sp.lb_epoch = c->lb_epoch;
        sp.totals_out = L.d_totals;
        sp.overflow_out = L.d_overflow;
        sp.ready_flags = L.ready_flags;
        sp.ready_epoch = L.ready_epoch;
        if (peer) {
            if (L.world > MAX_RANKS) return set_error(DFD_ERR_UNSUPPORTED, "world size %d > %d", L.world, MAX_RANKS);
            for (int r = 0; r < L.world; ++r) sp.peer_base[r] = L.peer_base[r];
        }
        // ONE single-pass launch moves every fixed-width column (any mix of widths up to the widest, per-column element type
        // inside the kernel): the rows are hashed and ranked once.  Bit columns (validity / booleans) and columns beyond the
        // per-launch limit follow through k_scatter on the same tiling, driven by the counts / cursors the first launch leaves.
        std::vector<PayloadCol> fixed, rest;
        int maxw = 0;
        for (const PayloadCol& pc : passes) {
            if (pc.width > 0 && fixed.size() < (size_t)MAX_COLS_PER_LAUNCH) { fixed.push_back(pc); if (pc.width > maxw) maxw = pc.width; }
            else rest.push_back(pc);
        }
        if (fixed.empty()) return set_error(DFD_ERR_INTERNAL, "single-pass mode needs a fixed-width column");
        {
            for (size_t i = 0; i < fixed.size(); ++i) sp.cols[i] = fixed[i];
            sp.n_cols = (int32_t)fixed.size();
            sp.stage_width = maxw;
            sp.hist_out = rest.empty() ? nullptr : d_hist;
            sp.base_out = rest.empty() ? nullptr : d_base;
            // the ring's element type is at most 8 bytes: 16-byte columns travel as two row-range items per tile (see the kernel),
            // which keeps the slots at tile x 8 bytes and the CTA count per SM independent of the schema
            const int ring_w = maxw > 8 ? 8 : maxw;
            int rc = launch_scatter(sp, ring_w, ks.fast_i64 != 0 && ring_w >= 8, peer, 1, c->sm_count, 0, stream);
            if (rc) return rc;
            ++launches;
            // the follow-up launches take the two-pass code path over the counts / cursors just written
            sp.hist = d_hist;
            sp.tile_base = d_base;
            sp.abort_flag = L.d_overflow;
        }
        static const int kWidths[6] = {8, 4, 16, 2, 1, 0};
        for (int wi = 0; wi < 6 && !rest.empty(); ++wi) {
            const int width = kWidths[wi];
            std::vector<PayloadCol> group;
            for (const PayloadCol& pc : rest)
                if (pc.width == width) group.push_back(pc);
            if (group.empty()) continue;
            sp.stage_width = width ? width : 1;
            for (size_t f0 = 0; f0 < group.size(); f0 += MAX_COLS_PER_LAUNCH) {
                size_t n = group.size() - f0 < (size_t)MAX_COLS_PER_LAUNCH ? group.size() - f0 : (size_t)MAX_COLS_PER_LAUNCH;
                for (size_t i = 0; i < n; ++i) sp.cols[i] = group[f0 + i];
                sp.n_cols = (int32_t)n;
                int rc = launch_scatter(sp, width, ks.fast_i64 != 0, peer, 2, c->sm_count, 0, stream);
                if (rc) return rc;
                ++launches;
            }
        }
    }
    if (ev) {
        cudaEventRecord(ev[3], stream);
        c->ev_pending++;
        ev = nullptr;
    }
    c->metrics.kernel_launches += launches;
    c->metrics.scatter_launches += launches;
    c->metrics.calls++;
    c->metrics.rows += (uint64_t)n_rows;
    c->metrics.bytes_in += bytes;
    c->metrics.bytes_out += bytes;
    return DFD_OK;
}

template <typename OFF>
static int launch_varwidth(const dfd::PartitionJob::VarCol& vc, const uint32_t* d_src, unsigned long long* d_block_sums,
                           int64_t n_rows, int sm_count, cudaStream_t stream) {
    const int64_t n_blocks = (n_rows + VAR_BLOCK * VAR_ITEMS - 1) / (VAR_BLOCK * VAR_ITEMS);
    const OFF* in_off = (const OFF*)vc.in.offsets;
    OFF* out_off = (OFF*)vc.out.offsets;
    k_var_block_sums<OFF><<<(unsigned)n_blocks, VAR_BLOCK, 0, stream>>>(in_off, vc.in.offset, d_src, n_rows, d_block_sums);
    LAUNCH_CHECK("k_var_block_sums");
    k_var_scan_block_sums<<<1, 1024, 0, stream>>>(d_block_sums, n_blocks);
    LAUNCH_CHECK("k_var_scan_block_sums");
    k_var_write_offsets<OFF><<<(unsigned)n_blocks, VAR_BLOCK, 0, stream>>>(in_off, vc.in.offset, d_src, n_rows, d_block_sums, out_off);
    LAUNCH_CHECK("k_var_write_offsets");
    const int64_t copy_blocks = (n_rows + 255) / 256;
    (void)sm_count;
    k_var_copy_bytes<OFF><<<(unsigned)(copy_blocks > 0x7fffffffLL ? 0x7fffffffLL : copy_blocks), 256, 0, stream>>>(in_off, vc.in.offset, (const uint8_t*)vc.in.values, d_src, out_off,
                                                                       (uint8_t*)vc.out.values, n_rows);
    LAUNCH_CHECK("k_var_copy_bytes");
    return DFD_OK;
}

int dfd::PartitionJob::run_varwidth() {
    Ctx* c = p->ctx;
    for (const VarCol& vc : var_cols) {
        if (n_rows == 0) {
            const size_t ow = vc.in.kind == DFD_COL_LARGE_UTF8 ? 8 : 4;
            cudaError_t e = cudaMemsetAsync(vc.out.offsets, 0, ow, stream);
            if (e != cudaSuccess) return cuda_error(e, "cudaMemsetAsync");
            continue;
        }
        int rc = vc.in.kind == DFD_COL_LARGE_UTF8 ? launch_varwidth<int64_t>(vc, d_src, d_block_sums, n_rows, c->sm_count, stream)
                                                  : launch_varwidth<int32_t>(vc, d_src, d_block_sums, n_rows, c->sm_count, stream);
        if (rc) return rc;
        c->metrics.kernel_launches += 4;
    }
    return DFD_OK;
}

int dfd::launch_bits_to_bytes(const uint8_t* bits, int64_t bit_offset, int64_t n, uint8_t* out, cudaStream_t s) {
    if (n <= 0) return DFD_OK;
    k_bits_to_bytes<<<(unsigned)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(bits, bit_offset, n, out);
    LAUNCH_CHECK("k_bits_to_bytes");
    return DFD_OK;
}

int dfd::launch_bytes_to_bits(const uint8_t* in, int64_t n, void* out_words, cudaStream_t s) {
    if (n <= 0) return DFD_OK;
    k_bytes_to_bits<<<(unsigned)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(in, n, (unsigned*)out_words);
    LAUNCH_CHECK("k_bytes_to_bits");
    return DFD_OK;
}

int dfd::launch_offsets_to_lengths(const void* off, int ow, int64_t n, void* len, cudaStream_t s) {
    if (n <= 0) return DFD_OK;
    const unsigned grid = (unsigned)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256);
    if (ow == 8) k_offsets_to_lengths<int64_t><<<grid, 256, 0, s>>>((const int64_t*)off, n, (int64_t*)len);
    else k_offsets_to_lengths<int32_t><<<grid, 256, 0, s>>>((const int32_t*)off, n, (int32_t*)len);
    LAUNCH_CHECK("k_offsets_to_lengths");
    return DFD_OK;
}

int dfd::launch_var_dest_bytes(const void* off, int ow, const int64_t* part_starts, uint32_t N, int64_t* bytes, int64_t* first, cudaStream_t s) {
    const unsigned grid = (N + 255) / 256;
    if (ow == 8) k_var_dest_bytes<int64_t><<<grid, 256, 0, s>>>((const int64_t*)off, part_starts, N, bytes, first);
    else k_var_dest_bytes<int32_t><<<grid, 256, 0, s>>>((const int32_t*)off, part_starts, N, bytes, first);
    LAUNCH_CHECK("k_var_dest_bytes");
    return DFD_OK;
}

int dfd::launch_lengths_to_offsets(const void* len, int ow, int64_t n, unsigned long long* block_sums, void* out_off, cudaStream_t s) {
    if (n <= 0) {
        cudaError_t e = cudaMemsetAsync(out_off, 0, (size_t)ow, s);
        return e == cudaSuccess ? DFD_OK : cuda_error(e, "cudaMemsetAsync");
    }
    const int64_t n_blocks = (n + VAR_BLOCK * VAR_ITEMS - 1) / (VAR_BLOCK * VAR_ITEMS);
    if (ow == 8) k_len_block_sums<int64_t><<<(unsigned)n_blocks, VAR_BLOCK, 0, s>>>((const int64_t*)len, n, block_sums);
    else k_len_block_sums<int32_t><<<(unsigned)n_blocks, VAR_BLOCK, 0, s>>>((const int32_t*)len, n, block_sums);
    LAUNCH_CHECK("k_len_block_sums");
    k_var_scan_block_sums<<<1, 1024, 0, s>>>(block_sums, n_blocks);
    LAUNCH_CHECK("k_var_scan_block_sums");
    if (ow == 8) k_len_write_offsets<int64_t><<<(unsigned)n_blocks, VAR_BLOCK, 0, s>>>((const int64_t*)len, n, block_sums, (int64_t*)out_off);
    else k_len_write_offsets<int32_t><<<(unsigned)n_blocks, VAR_BLOCK, 0, s>>>((const int32_t*)len, n, block_sums, (int32_t*)out_off);
    LAUNCH_CHECK("k_len_write_offsets");
    return DFD_OK;
}

int dfd::launch_var_gather(const void* in_off, int ow, int64_t in_offset, const uint8_t* in_data, const uint32_t* src, const void* out_off,
                           uint8_t* out_data, int64_t n, cudaStream_t s) {
    if (n <= 0) return DFD_OK;
    const int64_t blocks = (n + 255) / 256;
    const unsigned grid = (unsigned)(blocks > 0x7fffffffLL ? 0x7fffffffLL : blocks);
    if (ow == 8) k_var_copy_bytes<int64_t, true><<<grid, 256, 0, s>>>((const int64_t*)in_off, in_offset, in_data, src, (const int64_t*)out_off, out_data, n);
    else k_var_copy_bytes<int32_t, true><<<grid, 256, 0, s>>>((const int32_t*)in_off, in_offset, in_data, src, (const int32_t*)out_off, out_data, n);
    LAUNCH_CHECK("k_var_copy_bytes");
    return DFD_OK;
}

int dfd::partition_device_locked(Partitioner* p, const dfd_column* in_cols, int n_cols, int64_t n_rows,
                                 const dfd_column* out_cols, cudaStream_t stream, bool var_bytes_known) {
    PartitionJob job;
    job.var_bytes_known = var_bytes_known;
    int rc = job.prepare(p, in_cols, n_cols, n_rows, out_cols, false, stream);
    if (rc) return rc;
    if ((rc = job.run_hist_scan())) return rc;
    return job.run_scatter(p->d_part_starts, nullptr, 1, 1, nullptr);
}

int dfd::hash_columns_locked(Ctx* c, const dfd_column* cols, int n_cols, int64_t n_rows, const uint64_t* seeds, uint64_t* hashes_device,
                             cudaStream_t stream) {
    if (!cols || n_cols < 1 || n_cols > MAX_KEYS || n_rows < 0 || !hashes_device)
        return set_error(DFD_ERR_INVALID_ARGUMENT, "hash_columns: bad arguments");
    dfd_partitioner tmp;
    tmp.ctx = c;
    tmp.N = 1;
    for (int i = 0; i < n_cols; ++i) tmp.key_cols.push_back(i);
    tmp.key_modes.assign((size_t)n_cols, DFD_KEY_HASH_PLAIN);
    tmp.key_dicts.assign((size_t)n_cols, dfd_partitioner::KeyDict{});
    static const uint64_t PI2[4] = {0x452821e638d01377ULL, 0xbe5466cf34e90c6cULL, 0xc0ac29b7c97c50ddULL, 0x3f84d5b5b5470917ULL};
    uint64_t sd[4] = {0, 0, 0, 0};
    if (seeds) memcpy(sd, seeds, sizeof sd);
    tmp.st = HashState{sd[0] ^ PI2[0], sd[1] ^ PI2[1], sd[2] ^ PI2[2], sd[3] ^ PI2[3]};
    if (n_rows == 0) return DFD_OK;
    KeySet ks;
    int rc = build_keyset(&tmp, cols, n_cols, &ks);
    if (rc) return rc;
    int64_t blocks = (n_rows + 255) / 256;
    if (blocks > (int64_t)c->sm_count * 32) blocks = (int64_t)c->sm_count * 32;
    k_row_hashes<<<(unsigned)blocks, 256, 0, stream>>>(ks, tmp.st, n_rows, hashes_device);
    LAUNCH_CHECK("k_row_hashes");
    c->metrics.kernel_launches++;
    return DFD_OK;
}

extern "C" {

int dfd_abi_version(void) { return DFD_ABI_VERSION; }
const char* dfd_last_error(void) { return g_last_error.c_str(); }

const char* dfd_status_name(int s) {
    switch (s) {
        case DFD_OK: return "DFD_OK";
        case DFD_ERR_INVALID_ARGUMENT: return "DFD_ERR_INVALID_ARGUMENT";
        case DFD_ERR_OOM: return "DFD_ERR_OOM";
        case DFD_ERR_CUDA: return "DFD_ERR_CUDA";
        case DFD_ERR_NCCL: return "DFD_ERR_NCCL";
        case DFD_ERR_INTERNAL: return "DFD_ERR_INTERNAL";
        case DFD_ERR_UNSUPPORTED: return "DFD_ERR_UNSUPPORTED";
        case DFD_ERR_CAPACITY: return "DFD_ERR_CAPACITY";
    }
    return "DFD_ERR_UNKNOWN";
}

int dfd_device_count(int* out) {
    if (!out) return set_error(DFD_ERR_INVALID_ARGUMENT, "dfd_device_count: out is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *out = 0;
        return cuda_error(e, "cudaGetDeviceCount");
    }
    *out = n;
    return DFD_OK;
}

int dfd_ctx_create(int device, dfd_ctx** out) {
    if (!out) return set_error(DFD_ERR_INVALID_ARGUMENT, "dfd_ctx_create: out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return cuda_error(e, "cudaGetDeviceCount (no CUDA device: this library has no CPU fallback)");
    if (device < 0 || device >= n) return set_error(DFD_ERR_INVALID_ARGUMENT, "device %d out of range [0,%d)", device, n);
    if ((e = cudaSetDevice(device)) != cudaSuccess) return cuda_error(e, "cudaSetDevice");
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return cuda_error(e, "cudaGetDeviceProperties");
    if (prop.major < 10)
        return set_error(DFD_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                         prop.major, prop.minor);
    dfd_ctx* c = new (std::nothrow) dfd_ctx();
    if (!c) return set_error(DFD_ERR_OOM, "out of host memory");
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->l2_bytes = (size_t)prop.l2CacheSize;
    if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        delete c;
        return cuda_error(e, "cudaStreamCreate");
    }
    cudaEventCreate(&c->timer_a);
    cudaEventCreate(&c->timer_b);
    *out = c;
    return DFD_OK;
}

void dfd_ctx_destroy(dfd_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    c->pinned_cache.reset();  // unpins the cached output chunks of finished host operators
    if (c->scratch.ptr) cudaFree(c->scratch.ptr);
    if (c->flush.ptr) cudaFree(c->flush.ptr);
    if (c->var_scratch.ptr) cudaFree(c->var_scratch.ptr);
    if (c->lb.ptr) cudaFree(c->lb.ptr);
    for (auto& ev : c->ev_ring) cudaEventDestroy(ev);
    cudaEventDestroy(c->timer_a);
    cudaEventDestroy(c->timer_b);
    cudaStreamDestroy(c->stream);
    delete c;
}

void* dfd_ctx_stream(dfd_ctx* c) { return c ? (void*)c->stream : nullptr; }

#define CTX_GUARD(c)                                                            \
    if (!(c)) return set_error(DFD_ERR_INVALID_ARGUMENT, "%s: ctx is NULL", __func__); \
    std::lock_guard<std::mutex> _lk((c)->mu);                                   \
    {                                                                           \
        cudaError_t _e = cudaSetDevice((c)->device);                            \
        if (_e != cudaSuccess) return cuda_error(_e, "cudaSetDevice");          \
    }

int dfd_ctx_synchronize(dfd_ctx* c) {
    CTX_GUARD(c);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "cudaStreamSynchronize");
}

int dfd_ctx_set_profiling(dfd_ctx* c, int on) {
    CTX_GUARD(c);
    c->profiling = on != 0;
    return DFD_OK;
}

int dfd_device_alloc(dfd_ctx* c, size_t bytes, void** out) {
    CTX_GUARD(c);
    if (!out) return set_error(DFD_ERR_INVALID_ARGUMENT, "out is NULL");
    *out = nullptr;
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMalloc(out, bytes);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "cudaMalloc");
}

int dfd_device_free(dfd_ctx* c, void* p) {
    CTX_GUARD(c);
    cudaError_t e = cudaFree(p);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "cudaFree");
}

int dfd_host_alloc(dfd_ctx* c, size_t bytes, void** out) {
    CTX_GUARD(c);
    if (!out) return set_error(DFD_ERR_INVALID_ARGUMENT, "out is NULL");
    *out = nullptr;
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaHostAlloc(out, bytes, cudaHostAllocPortable);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "cudaHostAlloc");
}

int dfd_host_free(dfd_ctx* c, void* p) {
    CTX_GUARD(c);
    cudaError_t e = cudaFreeHost(p);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "cudaFreeHost");
}

int dfd_memcpy_h2d(dfd_ctx* c, void* dst, const void* src, size_t bytes) {
    CTX_GUARD(c);
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "cudaMemcpy H2D");
}

int dfd_memcpy_d2h(dfd_ctx* c, void* dst, const void* src, size_t bytes) {
    CTX_GUARD(c);
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "cudaMemcpy D2H");
}

int dfd_memset_device(dfd_ctx* c, void* dst, int value, size_t bytes) {
    CTX_GUARD(c);
    cudaError_t e = cudaMemsetAsync(dst, value, bytes, c->stream);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "cudaMemsetAsync");
}

int dfd_flush_l2(dfd_ctx* c) {
    CTX_GUARD(c);
    size_t need = c->l2_bytes * 2 > (size_t)(256u << 20) ? c->l2_bytes * 2 : (size_t)(256u << 20);
    int rc = c->flush.ensure(need, c->device);
    if (rc) return rc;
    cudaError_t e = cudaMemsetAsync(c->flush.ptr, 0x5a, need, c->stream);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "cudaMemsetAsync(flush)");
}

int dfd_timer_start(dfd_ctx* c) {
    CTX_GUARD(c);
    cudaError_t e = cudaEventRecord(c->timer_a, c->stream);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "cudaEventRecord");
}

int dfd_timer_stop(dfd_ctx* c, float* out_ms) {
    CTX_GUARD(c);
    cudaError_t e = cudaEventRecord(c->timer_b, c->stream);
    if (e == cudaSuccess) e = cudaEventSynchronize(c->timer_b);
    if (e == cudaSuccess && out_ms) e = cudaEventElapsedTime(out_ms, c->timer_a, c->timer_b);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "timer_stop");
}

int dfd_metrics_get(dfd_ctx* c, dfd_metrics* out) {
    CTX_GUARD(c);
    if (!out) return set_error(DFD_ERR_INVALID_ARGUMENT, "out is NULL");
    int rc = c->drain_events();
    if (rc) return rc;
    *out = c->metrics;
    return DFD_OK;
}

int dfd_metrics_reset(dfd_ctx* c) {
    CTX_GUARD(c);
    c->drain_events();
    memset(&c->metrics, 0, sizeof c->metrics);
    return DFD_OK;
}

/* ---- partitioner ------------------------------------------------------ */

int dfd_partitioner_create(dfd_ctx* c, uint32_t num_partitions, const int32_t* key_cols, int n_keys,
                           const uint64_t* seeds, dfd_partitioner** out) {
    if (!c) return set_error(DFD_ERR_INVALID_ARGUMENT, "ctx is NULL");
    if (!out) return set_error(DFD_ERR_INVALID_ARGUMENT, "out is NULL");
    *out = nullptr;
    if (num_partitions < 1 || num_partitions > MAX_PARTITIONS)
        return set_error(DFD_ERR_INVALID_ARGUMENT, "num_partitions %u not in [1, %u]", num_partitions, MAX_PARTITIONS);
    if (n_keys < 1 || n_keys > MAX_KEYS || !key_cols)
        return set_error(DFD_ERR_INVALID_ARGUMENT, "n_keys %d not in [1, %d]", n_keys, MAX_KEYS);
    // worst-case shared memory of the two-pass scatter (16-byte values) must fit one CTA: fail here, not at the first launch
    if (scatter_smem_bytes<TILE_THREADS, TILE_K>(num_partitions, 16, false, false) > 227 * 1024)
        return set_error(DFD_ERR_UNSUPPORTED, "num_partitions %u needs more than 227 KB of shared memory per CTA", num_partitions);
    for (int k = 0; k < n_keys; ++k)
        if (key_cols[k] < 0) return set_error(DFD_ERR_INVALID_ARGUMENT, "key_cols[%d] is negative", k);
    dfd_partitioner* p = new (std::nothrow) dfd_partitioner();
    if (!p) return set_error(DFD_ERR_OOM, "out of host memory");
    p->ctx = c;
    p->N = num_partitions;
    p->key_cols.assign(key_cols, key_cols + n_keys);
    p->key_modes.assign((size_t)n_keys, DFD_KEY_HASH_PLAIN);
    p->key_dicts.assign((size_t)n_keys, dfd_partitioner::KeyDict{});
    // ahash RandomState::with_seeds: seed ^ PI2 (random_state.rs); DataFusion's
    // REPARTITION_RANDOM_STATE uses seeds (0,0,0,0).
    static const uint64_t PI2[4] = {0x452821e638d01377ULL, 0xbe5466cf34e90c6cULL, 0xc0ac29b7c97c50ddULL,
                                    0x3f84d5b5b5470917ULL};
    uint64_t s[4] = {0, 0, 0, 0};
    if (seeds) memcpy(s, seeds, sizeof s);
    p->st = HashState{s[0] ^ PI2[0], s[1] ^ PI2[1], s[2] ^ PI2[2], s[3] ^ PI2[3]};
    p->mod = make_modn(num_partitions);
    {
        CTX_GUARD(c);
        cudaError_t e = cudaMalloc((void**)&p->d_part_starts, sizeof(int64_t) * (size_t)(num_partitions + 1));
        if (e == cudaSuccess) e = cudaMalloc((void**)&p->d_counts, sizeof(int64_t) * (size_t)(3 * num_partitions + 1));
        if (e == cudaSuccess) e = cudaMemset(p->d_counts, 0, sizeof(int64_t) * (size_t)(3 * num_partitions + 1));
        if (e == cudaSuccess) e = cudaHostAlloc((void**)&p->h_pin, sizeof(int64_t) * (size_t)(num_partitions + 1), cudaHostAllocPortable);
        if (e != cudaSuccess) {
            cudaFree(p->d_part_starts);
            cudaFree(p->d_counts);
            delete p;
            return cuda_error(e, "cudaMalloc(part_starts)");
        }
    }
    *out = p;
    return DFD_OK;
}

void dfd_partitioner_destroy(dfd_partitioner* p) {
    if (!p) return;
    {
        std::lock_guard<std::mutex> lk(p->ctx->mu);
        cudaSetDevice(p->ctx->device);
        cudaStreamSynchronize(p->ctx->stream);
        cudaFree(p->d_part_starts);
        cudaFree(p->d_counts);
        cudaFreeHost(p->h_pin);
    }
    delete p;
}

uint32_t dfd_partitioner_num_partitions(const dfd_partitioner* p) { return p ? p->N : 0; }

int dfd_partitioner_set_key_dictionary(dfd_partitioner* p, int key_index, const uint64_t* dict_hashes_device, const uint8_t* dict_validity_device) {
    if (!p) return set_error(DFD_ERR_INVALID_ARGUMENT, "partitioner is NULL");
    if (key_index < 0 || key_index >= (int)p->key_cols.size()) return set_error(DFD_ERR_INVALID_ARGUMENT, "key index %d out of range", key_index);
    std::lock_guard<std::mutex> lk(p->ctx->mu);
    if (!dict_hashes_device) {  // back to a plain key
        p->key_modes[(size_t)key_index] = DFD_KEY_HASH_PLAIN;
        p->key_dicts[(size_t)key_index] = dfd_partitioner::KeyDict{};
        return DFD_OK;
    }
    p->key_modes[(size_t)key_index] = KEY_HASH_DICTIONARY;
    p->key_dicts[(size_t)key_index] = dfd_partitioner::KeyDict{dict_hashes_device, dict_validity_device};
    return DFD_OK;
}

int dfd_hash_columns_device(dfd_ctx* c, const dfd_column* cols, int n_cols, int64_t n_rows, const uint64_t* seeds, uint64_t* hashes_device) {
    if (!c) return set_error(DFD_ERR_INVALID_ARGUMENT, "dfd_hash_columns_device: ctx is NULL");
    CTX_GUARD(c);
    return hash_columns_locked(c, cols, n_cols, n_rows, seeds, hashes_device, c->stream);
}

int dfd_partitioner_set_key_hash_mode(dfd_partitioner* p, int key_index, int mode) {
    if (!p) return set_error(DFD_ERR_INVALID_ARGUMENT, "partitioner is NULL");
    if (key_index < 0 || key_index >= (int)p->key_cols.size()) return set_error(DFD_ERR_INVALID_ARGUMENT, "key index %d out of range", key_index);
    if (mode != DFD_KEY_HASH_PLAIN && mode != DFD_KEY_HASH_INTERVAL_DAY_TIME && mode != DFD_KEY_HASH_INTERVAL_MONTH_DAY_NANO)
        return set_error(DFD_ERR_INVALID_ARGUMENT, "unknown key hash mode %d (dictionary keys: dfd_partitioner_set_key_dictionary)", mode);
    std::lock_guard<std::mutex> lk(p->ctx->mu);
    p->key_modes[(size_t)key_index] = mode;
    return DFD_OK;
}
const int64_t* dfd_partitioner_part_starts_device(const dfd_partitioner* p) { return p ? p->d_part_starts : nullptr; }

int dfd_partition_ids_device(dfd_partitioner* p, const dfd_column* cols, int n_cols, int64_t n_rows,
                             uint32_t* dest_device) {
    if (!p) return set_error(DFD_ERR_INVALID_ARGUMENT, "partitioner is NULL");
    dfd_ctx* c = p->ctx;
    CTX_GUARD(c);
    if (n_rows < 0 || !cols || !dest_device) return set_error(DFD_ERR_INVALID_ARGUMENT, "bad arguments");
    if (n_rows == 0) return DFD_OK;
    KeySet ks;
    int rc = build_keyset(p, cols, n_cols, &ks);
    if (rc) return rc;
    int64_t blocks = (n_rows + 255) / 256;
    int64_t cap = (int64_t)c->sm_count * 32;
    if (blocks > cap) blocks = cap;
    k_partition_ids<<<(unsigned)blocks, 256, 0, c->stream>>>(ks, p->st, p->mod, n_rows, dest_device);
    LAUNCH_CHECK("k_partition_ids");
    c->metrics.kernel_launches++;
    cudaError_t e = cudaStreamSynchronize(c->stream);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "k_partition_ids");
}

int dfd_partition_device(dfd_partitioner* p, const dfd_column* in_cols, int n_cols, int64_t n_rows,
                         const dfd_column* out_cols, int64_t* part_starts_host) {
    if (!p) return set_error(DFD_ERR_INVALID_ARGUMENT, "partitioner is NULL");
    dfd_ctx* c = p->ctx;
    CTX_GUARD(c);
    int rc = partition_device_locked(p, in_cols, n_cols, n_rows, out_cols, c->stream);
    if (rc) return rc;
    if (part_starts_host) {
        cudaError_t e = cudaMemcpyAsync(part_starts_host, p->d_part_starts, sizeof(int64_t) * (size_t)(p->N + 1),
                                        cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) return cuda_error(e, "dfd_partition_device");
    }
    return DFD_OK;
}

/* ---- single-pass partition (region layout) ---------------------------------- */

static int onepass_launch_locked(dfd_partitioner* p, const int64_t* d_base, const int64_t* d_cap, int64_t stride) {
    dfd_ctx* c = p->ctx;
    const uint32_t N = p->N;
    int32_t* d_flag = (int32_t*)(p->d_counts + 3 * (size_t)N);
    cudaError_t e = cudaMemsetAsync(d_flag, 0, sizeof(int64_t), c->stream);
    if (e != cudaSuccess) return cuda_error(e, "cudaMemsetAsync(overflow flag)");
    PartitionJob job;
    job.onepass_tiling = true;
    job.out_rows = stride > 0 ? stride * (int64_t)N : p->last_rows;  // region layout spans N * region_rows output rows
    int rc = job.prepare(p, p->last_in.data(), (int)p->last_in.size(), p->last_rows, p->last_out.data(), false, c->stream);
    if (rc) return rc;
    PartitionJob::OnePassLayout L;
    L.d_dest_base = d_base;
    L.d_dest_cap = d_cap;
    L.region_stride = stride;
    L.d_totals = p->d_counts;
    L.d_overflow = d_flag;
    if ((rc = job.run_onepass(L))) return rc;
    e = cudaMemcpyAsync(p->h_pin, p->d_counts, sizeof(int64_t) * (size_t)N, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(p->h_pin + N, d_flag, sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream);
    return e == cudaSuccess ? DFD_OK : cuda_error(e, "D2H counts");
}

static int collect_locked(dfd_partitioner* p, int64_t* starts, int64_t* counts) {
    dfd_ctx* c = p->ctx;
    const uint32_t N = p->N;
    if (p->last == dfd_partitioner::LAST_NONE) return set_error(DFD_ERR_INVALID_ARGUMENT, "no partition call to collect");
    if (p->last == dfd_partitioner::LAST_DENSE) {
        std::vector<int64_t> ps(N + 1);
        cudaError_t e = cudaMemcpyAsync(ps.data(), p->d_part_starts, sizeof(int64_t) * (size_t)(N + 1), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) return cuda_error(e, "dfd_partitioner_collect");
        for (uint32_t q = 0; q < N; ++q) {
            if (starts) starts[q] = ps[q];
            if (counts) counts[q] = ps[q + 1] - ps[q];
        }
        return DFD_OK;
    }
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return cuda_error(e, "single-pass partition");
    if (p->h_pin[N] != 0) {
        // a destination outgrew its region (skewed keys): the counts are exact, so re-run with exact,
        // dense regions (dest_base = prefix of the counts) — always fits in N * region_rows >= n_rows rows
        std::vector<int64_t> reg(2 * (size_t)N);
        int64_t run = 0;
        for (uint32_t q = 0; q < N; ++q) {
            reg[q] = run;
            reg[N + q] = p->h_pin[q];
            run += p->h_pin[q];
        }
        e = cudaMemcpyAsync(p->d_counts + N, reg.data(), sizeof(int64_t) * 2 * (size_t)N, cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);  // `reg` is pageable
        if (e != cudaSuccess) return cuda_error(e, "H2D exact regions");
        int rc = onepass_launch_locked(p, p->d_counts + N, p->d_counts + 2 * (size_t)N, 0);
        if (rc) return rc;
        e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) return cuda_error(e, "single-pass partition (exact re-run)");
        if (p->h_pin[N] != 0) return set_error(DFD_ERR_INTERNAL, "exact re-run overflowed");
        c->metrics.onepass_reruns++;
        for (uint32_t q = 0; q < N; ++q) {
            if (starts) starts[q] = reg[q];
            if (counts) counts[q] = p->h_pin[q];
        }
        p->last_stride = -1;  // dense now
        return DFD_OK;
    }
    for (uint32_t q = 0; q < N; ++q) {
        if (starts) starts[q] = (int64_t)q * p->last_stride;
        if (counts) counts[q] = p->h_pin[q];
    }
    return DFD_OK;
}

int dfd_partition_device_onepass(dfd_partitioner* p, const dfd_column* in_cols, int n_cols, int64_t n_rows,
                                 const dfd_column* out_cols, int64_t region_rows, int64_t* part_starts_host,
                                 int64_t* part_counts_host) {
    if (!p) return set_error(DFD_ERR_INVALID_ARGUMENT, "partitioner is NULL");
    dfd_ctx* c = p->ctx;
    CTX_GUARD(c);
    if (n_rows < 0 || n_cols < 0 || (n_cols > 0 && (!in_cols || !out_cols)))
        return set_error(DFD_ERR_INVALID_ARGUMENT, "partition: bad arguments");
    const uint32_t N = p->N;
    bool has_fixed = false, has_var = false;
    for (int i = 0; i < n_cols; ++i) {
        has_fixed |= in_cols[i].kind == DFD_COL_FIXED;
        has_var |= in_cols[i].kind == DFD_COL_UTF8 || in_cols[i].kind == DFD_COL_LARGE_UTF8 || in_cols[i].kind == DFD_COL_BINARY;
    }
    p->last_in.assign(in_cols, in_cols + n_cols);
    p->last_out.assign(out_cols, out_cols + n_cols);
    p->last_rows = n_rows;
    int rc;
    if (!has_fixed || has_var || N > ONEPASS_MAX_N) {
        // dense two-pass path (K1 -> K1b -> K2 [-> K4]); same (start, count) contract
        if ((rc = partition_device_locked(p, in_cols, n_cols, n_rows, out_cols, c->stream))) return rc;
        p->last = dfd_partitioner::LAST_DENSE;
    } else {
        if (region_rows < 1 || (__int128)region_rows * N < n_rows)
            return set_error(DFD_ERR_INVALID_ARGUMENT, "region_rows %lld x %u partitions < n_rows %lld", (long long)region_rows, N,
                             (long long)n_rows);
        if ((__int128)region_rows * N >= 0xffffffffLL)
            return set_error(DFD_ERR_UNSUPPORTED, "region_rows x partitions must be < 2^32 - 1 rows per call (32-bit output rows)");
        p->last_stride = region_rows;
        if ((rc = onepass_launch_locked(p, nullptr, nullptr, region_rows))) return rc;
        p->last = dfd_partitioner::LAST_REGIONS;
    }
    if (part_starts_host || part_counts_host) return collect_locked(p, part_starts_host, part_counts_host);
    return DFD_OK;
}

int dfd_partitioner_collect(dfd_partitioner* p, int64_t* part_starts_host, int64_t* part_counts_host) {
    if (!p) return set_error(DFD_ERR_INVALID_ARGUMENT, "partitioner is NULL");
    dfd_ctx* c = p->ctx;
    CTX_GUARD(c);
    return collect_locked(p, part_starts_host, part_counts_host);
}

}  // extern "C"
