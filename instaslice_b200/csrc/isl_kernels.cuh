// isl_kernels.cuh — sm_100a kernels of the MIG-slot placement engine.
//
// Replaces, for a whole batch of pending pods at once, the reference's per-pod scan
//   Reconcile node loop            internal/controller/instaslice_controller.go:190
//   findDeviceForASlice GPU loop   :240-262
//   getStartIndexFromPreparedState :303-384
// Pure integer / bitmask work: no tensor cores, nothing to reshape into a GEMM.
//
// Pipeline per batch (DESIGN.md "Kernels"):
//   k_prepare            frees (atomicAnd on packed occupancy words), default results, per-tile
//                        per-profile histogram of the ALLOC requests
//   per chunk of <= 65536 requests:
//     k_partition        stable P-way partition of the chunk's ALLOC requests into per-profile queues
//     k_sweep_count/_scatter   vectorised sweep over the occupancy bytes: feasibility bitmask via a
//                        256-entry shared-memory table, ordered compaction of the candidate GPUs
//     k_chain<K>         exact first-fit commit: GPU-major stream filtering with one lane per
//                        (profile, start) candidate and a warp min-reduction per accepted placement
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/islplace.h"

namespace isl {

constexpr uint32_t kChunk = 65536;         // requests per commit chunk: in-chunk request index fits 16 bits
constexpr uint32_t kTile = 1024;           // requests per partition tile (256 threads x 4 rounds)
constexpr uint32_t kTileThreads = 256;
constexpr uint32_t kTilesPerChunk = kChunk / kTile;
constexpr uint32_t kQPad = 32;             // per-profile queue segments start on 32-entry boundaries
constexpr uint32_t kQCap = kChunk + kQPad * ISL_MAX_PROFILES;
constexpr uint32_t kSweepThreads = 256;
constexpr uint32_t kSweepPerThread = 16;   // one 16-byte vector load = 16 GPUs
constexpr uint32_t kSweepBlock = kSweepThreads * kSweepPerThread;   // 4096 GPUs per CTA
constexpr uint32_t kSkip = 0xFFu;          // partition key of a request that is not a valid ALLOC
constexpr uint32_t kInf = 0xFFFFFFFFu;
constexpr uint32_t kMaxCand = ISL_MAX_PROFILES * ISL_MAX_STARTS;   // 128 (profile,start) candidates
constexpr uint32_t kChainThreads = 256;
constexpr uint32_t kMaxTables = ISL_MAX_TABLES;   // per-node profile tables (heterogeneous clusters)

// The chain's occupancy word is 16 bits: the busy slices in the low byte and, in the high byte, every table bit set EXCEPT
// the one of the table the GPU's node publishes.  A candidate of table t carries bit (8 + t) in its mask, so `(occ16 & mask) == 0`
// holds only on GPUs of its own table — no extra instruction per decision.
// A/B switches of the decision loop (tools/ab_build.sh builds the variants; the defaults are what measured fastest)
#ifndef ISL_UNIFORM_WARP
#define ISL_UNIFORM_WARP 1      // the chain warp is selected by a warp-UNIFORM predicate (redux of the warp index): ptxas then knows the warp
#endif                          // is converged and drops the BRA.DIV / UMOV guard in front of every redux of the loop
#ifndef ISL_DEFER_INF
#define ISL_DEFER_INF 1         // the "nothing fits" test runs once per unrolled group instead of once per decision
#endif
// true for every lane of warp 0 and only there; with ISL_UNIFORM_WARP the predicate comes out of a redux (a uniform register)
__device__ __forceinline__ bool is_chain_warp(uint32_t warp) {
#if ISL_UNIFORM_WARP
    return __reduce_or_sync(0xFFFFFFFFu, warp) == 0;
#else
    return warp == 0;
#endif
}

__host__ __device__ inline uint32_t table_tag(uint32_t table) { return ((~(1u << table)) & 0xFFu) << 8; }

struct DevProfiles {            // kernel parameter (by value)
    uint32_t n;
    uint32_t quirks;
    isl_profile rows[ISL_MAX_PROFILES];
    uint32_t flip;              // ISL_POLICY_RIGHT_TO_LEFT: G (the inventory is stored in REVERSE canonical order), else 0
};

// ISL_POLICY_RIGHT_TO_LEFT walks the GPUs in descending canonical order.  The engine stores such an inventory reversed (internal index
// i = G - 1 - canonical) so that every scan stays an ascending sweep; only the two edges translate: the GPU a FREE names, and the GPU a
// PLACED record reports.
__host__ __device__ inline uint32_t flip_gpu(uint32_t g, uint32_t flip) { return flip ? flip - 1u - g : g; }

// One (profile, start) candidate of the chain: bits  [3:0] profile | [6:4] order in the row |
// [10:7] start | [14:11] size | [23:16] slot mask | [26:24] table | [31] valid
struct CandTab {                // kernel parameter (by value): slot k of lane l is desc[k][l]
    uint32_t desc[4][32];
};

struct Ctrl {                   // device-resident control block, rewritten per chunk
    uint32_t qoff[ISL_MAX_PROFILES + 1];   // queue segment offsets (entries) inside the chunk's queue buffer
    uint32_t qcnt[ISL_MAX_PROFILES];       // requests of profile p in this chunk
    uint32_t active;                       // profiles with requests in this chunk AND >= 1 valid candidate
    uint32_t n_cand;                       // candidate GPUs found by the sweep
    uint32_t heads_out[ISL_MAX_PROFILES];  // queue heads after the chain (token for the next rank)
    uint32_t n_log;                        // decisions logged by the chain of this chunk
    unsigned long long placed, freed, bad, steps, visited, allocs, jumps, scanned;
    unsigned long long spec_sims, spec_rounds, spec_cells;   // speculative rounds: segment simulations run (all stages), rounds until the last stage was certified summed over chunks, chunks
};

// The one rule both the device table and the chain candidates come from: slot mask of placing a
// `size`-slice profile at start v, or 0 when getStartIndexFromPreparedState can never return v
//   size 1            -> only busy[v] is tested (:346-349)
//   size 2/4/8        -> needs v+size < 8 (strict, Q1) and all slots free (:350-378)
//   any other size    -> never placed under Q2; with the quirk off, any size 2..8 with v+size <= 8
__host__ __device__ inline uint32_t candidate_mask(uint32_t size, uint32_t v, uint32_t quirks) {
    if (v >= ISL_SLOTS || size == 0 || size > ISL_SLOTS) return 0;
    if (size == 1) return 1u << v;
    const bool pow2_only = quirks & ISL_QUIRK_POW2_ONLY;
    if (pow2_only && !(size == 2 || size == 4 || size == 8)) return 0;
    const bool strict = quirks & ISL_QUIRK_STRICT_BOUND;
    if (strict ? !(v + size < ISL_SLOTS) : !(v + size <= ISL_SLOTS)) return 0;
    return (((1u << size) - 1u) << v) & 0xFFu;
}

// ---------------------------------------------------------------------------------------------
// Device table: lut[p][occ] = first legal start of profile p on a GPU with occupancy byte occ
// (or 9), feas[occ] = bitmask of profiles that have a legal start.  256 threads, one per byte.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_build_lut(DevProfiles prof, uint32_t table, uint8_t* __restrict__ lut, uint16_t* __restrict__ feas,
                                                   uint8_t* __restrict__ capn, uint32_t* __restrict__ seq) {
    lut += (size_t)table * ISL_MAX_PROFILES * 256; feas += (size_t)table * 256;        // lut[table][profile][occ], feas[table][occ]
    capn += (size_t)table * ISL_MAX_PROFILES * 256; seq += (size_t)table * ISL_MAX_PROFILES * 256;
    const uint32_t occ = threadIdx.x;
    uint32_t fmask = 0;
    for (uint32_t p = 0; p < ISL_MAX_PROFILES; ++p) {
        uint32_t found = ISL_START_NONE;
        if (p < prof.n) {
            const isl_profile& row = prof.rows[p];
            for (uint32_t k = 0; k < row.n_starts; ++k) {                        // CRD order (:344)
                const uint32_t m = candidate_mask(row.size, row.starts[k], prof.quirks);
                if (m != 0 && (occ & m) == 0) { found = row.starts[k]; break; }
            }
        }
        lut[p * 256 + occ] = (uint8_t)found;
        if (found != ISL_START_NONE) fmask |= 1u << p;
        // how many requests of this profile the GPU takes IN A ROW from this occupancy, and at which starts (4 bits each):
        // the single-profile scan commit (k_sweep_* in scan mode) places whole GPUs at once from these two tables
        uint32_t o = occ, cnt = 0, packed = 0;
        if (p < prof.n) {
            const isl_profile& row = prof.rows[p];
            while (cnt < 8) {
                uint32_t st = ISL_START_NONE, mk = 0;
                for (uint32_t k = 0; k < row.n_starts; ++k) {
                    const uint32_t m = candidate_mask(row.size, row.starts[k], prof.quirks);
                    if (m != 0 && (o & m) == 0) { st = row.starts[k]; mk = m; break; }
                }
                if (st == ISL_START_NONE) break;
                packed |= st << (4 * cnt); o |= mk; ++cnt;
            }
        }
        capn[p * 256 + occ] = (uint8_t)cnt;
        seq[p * 256 + occ] = packed;
    }
    feas[occ] = (uint16_t)fmask;
}

__global__ void k_eval_starts(const uint8_t* __restrict__ lut, uint32_t profile, uint32_t n,
                              const uint8_t* __restrict__ occ, uint8_t* __restrict__ out) {
    __shared__ uint8_t s_lut[256];
    if (threadIdx.x < 256) s_lut[threadIdx.x] = lut[profile * 256 + threadIdx.x];
    __syncthreads();
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = s_lut[occ[i]];
}

__global__ void k_free_spans(uint32_t n, const isl_span* __restrict__ spans, uint32_t* __restrict__ occ32,
                             uint32_t G, uint32_t lo, uint32_t hi, Ctrl* ctrl, uint32_t flip) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    isl_span s = spans[i];
    if (s.gpu >= G || s.size == 0 || (uint32_t)s.start + s.size > ISL_SLOTS) { atomicAdd(&ctrl->bad, 1ull); return; }
    s.gpu = flip_gpu(s.gpu, flip);
    if (s.gpu < lo || s.gpu >= hi) return;
    const uint32_t m = (((1u << s.size) - 1u) << s.start) << ((s.gpu & 3u) * 8u);
    atomicAnd(&occ32[s.gpu >> 2], ~m);
    atomicAdd(&ctrl->freed, 1ull);
}

// ---------------------------------------------------------------------------------------------
// k_prepare: one pass over the request stream (8 B coalesced loads, 8 B coalesced stores).
//   FREE  -> clear the span in the packed occupancy word, result FREED / BAD_SPAN
//   ALLOC -> default result (gpu NONE, start 9, NO_CAPACITY); the chain overwrites what it places
//   per-tile histogram of ALLOC requests by profile (warp match + one shared atomic per group)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint2 pack_result(uint32_t gpu, uint32_t start, uint32_t size, uint32_t status) {
    return make_uint2(gpu, start | (size << 8) | (status << 16));
}

// One tile of 1024 requests of a stream: which batch / pipeline chunk it belongs to (host-built table, one launch
// of k_prepare and one of k_partition cover every batch and chunk of a stream call).
struct TileDesc {
    uint32_t batch_off, batch_n, batch, batch_first_tile;      // batch: request offset in the stream, size, index, first global tile
    uint32_t chunk, chunk_first_tile, chunk_tiles, chunk_off;  // chunk: index, first global tile, tiles, request offset in the stream
    uint32_t chunk_n, pad0, pad1, pad2;
};

__global__ void __launch_bounds__(kTileThreads) k_prepare(uint32_t n, const uint2* __restrict__ in, uint2* __restrict__ out,
                                                           uint32_t* __restrict__ occ32, uint32_t G, uint32_t lo, uint32_t hi,
                                                           DevProfiles prof, uint32_t* __restrict__ tile_counts, Ctrl* ctrl,
                                                           const TileDesc* __restrict__ descs, uint32_t* __restrict__ free_acc, uint32_t free_stride,
                                                           uint32_t tile_base) {
    // descs != nullptr (stream mode): the tile's batch comes from the table, and FREEs are not applied here but ORed
    // into the batch's free-mask array (one byte per GPU); the segment pipeline clears them in batch order inside the
    // segment that owns the GPU.  tile_base: first global tile of this launch (a stream may be fed batch by batch).
    const uint32_t bid = blockIdx.x + tile_base;
    uint32_t tile = bid;
    if (descs) {
        const TileDesc d = descs[bid];
        n = d.batch_n; in += d.batch_off; out += d.batch_off; tile = bid - d.batch_first_tile;
        free_acc += (size_t)d.batch * free_stride;
    }
    __shared__ uint32_t s_cnt[ISL_MAX_PROFILES];
    __shared__ uint32_t s_freed;
    if (threadIdx.x < ISL_MAX_PROFILES) s_cnt[threadIdx.x] = 0;
    if (threadIdx.x == 0) s_freed = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u;
#pragma unroll
    for (uint32_t r = 0; r < kTile / kTileThreads; ++r) {
        const uint32_t i = tile * kTile + r * kTileThreads + threadIdx.x;
        uint32_t key = kSkip;
        if (i < n) {
            const uint2 rq = in[i];
            const uint32_t handle = rq.x, profile = rq.y & 0xFFu, op = (rq.y >> 8) & 0xFFu;
            const uint32_t start = (rq.y >> 16) & 0xFFu, size = rq.y >> 24;
            if (op == ISL_OP_ALLOC) {
                if (profile < prof.n) { key = profile; out[i] = pack_result(ISL_GPU_NONE, ISL_START_NONE, prof.rows[profile].size, ISL_ST_NO_CAPACITY); }
                else out[i] = pack_result(ISL_GPU_NONE, ISL_START_NONE, 0, ISL_ST_BAD_PROFILE);
            } else if (op == ISL_OP_FREE) {
                if (handle >= G || size == 0 || start + size > ISL_SLOTS) out[i] = pack_result(handle, start, size, ISL_ST_BAD_SPAN);
                else {
                    const uint32_t gi = flip_gpu(handle, prof.flip);       // where the engine keeps that GPU
                    if (gi >= lo && gi < hi) {
                        const uint32_t span = (((1u << size) - 1u) << start) << ((gi & 3u) * 8u);
                        if (descs) atomicOr(&free_acc[gi >> 2], span);
                        else atomicAnd(&occ32[gi >> 2], ~span);
                        atomicAdd(&s_freed, 1u);
                    }
                    out[i] = pack_result(handle, start, size, ISL_ST_FREED);
                }
            } else out[i] = pack_result(ISL_GPU_NONE, ISL_START_NONE, 0, ISL_ST_NOOP);
        }
        const uint32_t peers = __match_any_sync(0xFFFFFFFFu, key);
        if (key != kSkip && lane == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&s_cnt[key], (uint32_t)__popc(peers));
    }
    __syncthreads();
    if (threadIdx.x < ISL_MAX_PROFILES) tile_counts[bid * ISL_MAX_PROFILES + threadIdx.x] = s_cnt[threadIdx.x];
    if (threadIdx.x == 0) {
        if (s_freed) atomicAdd(&ctrl->freed, (unsigned long long)s_freed);
        uint32_t allocs = 0;
        for (uint32_t p = 0; p < ISL_MAX_PROFILES; ++p) allocs += s_cnt[p];
        if (allocs) atomicAdd(&ctrl->allocs, (unsigned long long)allocs);
    }
}

// ---------------------------------------------------------------------------------------------
// k_partition: stable P-way partition of one chunk's ALLOC requests.  Queue p receives the
// in-chunk indices (16 bit) of the requests for profile p, in request order.
// grid = tiles of the chunk; every CTA re-derives the chunk-wide offsets from tile_counts
// (<= 64 tiles x 16 counters), so no inter-CTA communication is needed.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kTileThreads) k_partition(uint32_t n_chunk, const uint2* __restrict__ in_chunk, uint32_t n_profiles,
                                                             const uint32_t* __restrict__ tile_counts_chunk, uint32_t n_tiles,
                                                             uint32_t cand_profiles, uint16_t* __restrict__ q, Ctrl* ctrl,
                                                             const TileDesc* __restrict__ descs, uint32_t q_stride, uint32_t tile_base) {
    // descs != nullptr (stream mode): in_chunk / tile_counts_chunk / q / ctrl are the bases of the whole stream and
    // the tile's chunk comes from the table.
    const uint32_t bid = blockIdx.x + tile_base;
    uint32_t tile = bid;
    if (descs) {
        const TileDesc d = descs[bid];
        n_chunk = d.chunk_n; in_chunk += d.chunk_off; tile_counts_chunk += (size_t)d.chunk_first_tile * ISL_MAX_PROFILES;
        n_tiles = d.chunk_tiles; tile = bid - d.chunk_first_tile; q += (size_t)d.chunk * q_stride; ctrl += d.chunk;
    }
    __shared__ uint32_t s_part[16][ISL_MAX_PROFILES][2];   // [j][p][0]=total, [1]=prefix before this tile
    __shared__ uint32_t s_base[ISL_MAX_PROFILES];
    __shared__ uint32_t s_seg[32][ISL_MAX_PROFILES];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    {   // chunk-wide per-profile totals and the prefix of the tiles before this one
        const uint32_t p = tid & 15u, j = tid >> 4;
        uint32_t tot = 0, pre = 0;
        for (uint32_t t = j; t < n_tiles; t += 16) {
            const uint32_t c = tile_counts_chunk[t * ISL_MAX_PROFILES + p];
            tot += c;
            if (t < tile) pre += c;
        }
        s_part[j][p][0] = tot; s_part[j][p][1] = pre;
    }
    for (uint32_t k = tid; k < 32 * ISL_MAX_PROFILES; k += kTileThreads) (&s_seg[0][0])[k] = 0;
    __syncthreads();
    if (tid == 0) {
        uint32_t off = 0, active = 0;
        for (uint32_t p = 0; p < ISL_MAX_PROFILES; ++p) {
            uint32_t tot = 0, pre = 0;
            for (uint32_t j = 0; j < 16; ++j) { tot += s_part[j][p][0]; pre += s_part[j][p][1]; }
            s_base[p] = off + pre;
            if (tile == 0) {
                ctrl->qoff[p] = off; ctrl->qcnt[p] = tot;
                if (tot && ((cand_profiles >> p) & 1u)) active |= 1u << p;
            }
            off += (tot + kQPad - 1) & ~(kQPad - 1);
        }
        if (tile == 0) { ctrl->qoff[ISL_MAX_PROFILES] = off; ctrl->active = active; ctrl->n_cand = 0; }
    }
    uint32_t key[4], rank[4];
#pragma unroll
    for (uint32_t r = 0; r < 4; ++r) {
        const uint32_t i = tile * kTile + r * kTileThreads + tid;
        key[r] = kSkip;
        if (i < n_chunk) {
            const uint32_t w = in_chunk[i].y;
            const uint32_t profile = w & 0xFFu, op = (w >> 8) & 0xFFu;
            if (op == ISL_OP_ALLOC && profile < n_profiles) key[r] = profile;
        }
        const uint32_t peers = __match_any_sync(0xFFFFFFFFu, key[r]);
        rank[r] = __popc(peers & ((1u << lane) - 1u));
        if (key[r] != kSkip && lane == (uint32_t)(__ffs(peers) - 1)) s_seg[r * 8 + warp][key[r]] = __popc(peers);
    }
    __syncthreads();
    if (tid < ISL_MAX_PROFILES) {           // exclusive scan over the 32 (round, warp) segments, in request order
        uint32_t run = 0;
        for (uint32_t s = 0; s < 32; ++s) { const uint32_t c = s_seg[s][tid]; s_seg[s][tid] = run; run += c; }
    }
    __syncthreads();
#pragma unroll
    for (uint32_t r = 0; r < 4; ++r) {
        if (key[r] == kSkip) continue;
        const uint32_t i = tile * kTile + r * kTileThreads + tid;
        q[s_base[key[r]] + s_seg[r * 8 + warp][key[r]] + rank[r]] = (uint16_t)i;
    }
}

// one word, stream-ordered: "the pre-pass of this batch is complete" for a segment pipeline that is already running
__global__ void k_set_flag(uint32_t* flag, uint32_t value) {
    __threadfence();
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(flag), "r"(value) : "memory");
}

// ---------------------------------------------------------------------------------------------
// Sweep: every thread loads 16 occupancy bytes with one 128-bit read-only load, looks each byte
// up in the 256-entry feasibility table staged in shared memory, and keeps the GPUs on which at
// least one profile that is pending in this chunk has a legal start.  Two passes (count, then
// ordered scatter) keep the candidate list in canonical GPU order without inter-CTA spinning.
// Candidate record = (gpu << 8) | occupancy byte.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ld_nc_v4(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

__device__ __forceinline__ uint32_t sweep_mask16(const uint4 v, const uint4 tv, const uint16_t* s_feas, uint32_t active, uint32_t g0, uint32_t lo, uint32_t hi) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w}, tw[4] = {tv.x, tv.y, tv.z, tv.w};
    uint32_t mask = 0;
#pragma unroll
    for (uint32_t j = 0; j < 16; ++j) {
        const uint32_t o = (w[j >> 2] >> ((j & 3u) * 8u)) & 0xFFu, t = (tw[j >> 2] >> ((j & 3u) * 8u)) & (kMaxTables - 1);
        const uint32_t g = g0 + j;
        if ((s_feas[t * 256 + o] & active) && g >= lo && g < hi) mask |= 1u << j;
    }
    return mask;
}

// Scan mode (exactly ONE placeable profile in the chunk, e.g. a burst of replicas of one Deployment): there is nothing
// to interleave, GPU g simply takes the next capn[occ_g] requests of the queue.  The two sweep passes then compute the
// device-wide exclusive scan of those capacities and commit results and occupancy directly — fully parallel, no chain.
__device__ __forceinline__ uint32_t scan_capacity16(const uint4 v, const uint4 tv, const uint8_t* __restrict__ capn, uint32_t p, uint32_t g0, uint32_t lo, uint32_t hi) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w}, tw[4] = {tv.x, tv.y, tv.z, tv.w};
    uint32_t c = 0;
#pragma unroll
    for (uint32_t j = 0; j < 16; ++j) {
        const uint32_t o = (w[j >> 2] >> ((j & 3u) * 8u)) & 0xFFu, t = (tw[j >> 2] >> ((j & 3u) * 8u)) & (kMaxTables - 1);
        const uint32_t g = g0 + j;
        if (g >= lo && g < hi) c += capn[(t * ISL_MAX_PROFILES + p) * 256 + o];
    }
    return c;
}

__global__ void __launch_bounds__(kSweepThreads) k_sweep_count(const uint4* __restrict__ occ16, const uint4* __restrict__ gtab16, const uint16_t* __restrict__ feas,
                                                                uint32_t first_block, uint32_t lo, uint32_t hi,
                                                                const Ctrl* __restrict__ ctrl, uint32_t* __restrict__ counts, const uint8_t* __restrict__ capn) {
    __shared__ uint16_t s_feas[kMaxTables * 256];
    __shared__ uint32_t s_warp[kSweepThreads / 32];
    for (uint32_t i = threadIdx.x; i < kMaxTables * 256; i += kSweepThreads) s_feas[i] = feas[i];
    __syncthreads();
    const uint32_t active = ctrl->active;
    const uint32_t g0 = (first_block + blockIdx.x) * kSweepBlock + threadIdx.x * kSweepPerThread;
    uint32_t c = 0;
    if (active && g0 < hi && g0 + kSweepPerThread > lo) {
        const uint4 v = ld_nc_v4(&occ16[g0 >> 4]), tv = ld_nc_v4(&gtab16[g0 >> 4]);
        c = __popc(active) == 1 ? scan_capacity16(v, tv, capn, __ffs(active) - 1, g0, lo, hi) : __popc(sweep_mask16(v, tv, s_feas, active, g0, lo, hi));
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, d);
    if ((threadIdx.x & 31u) == 0) s_warp[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (uint32_t w = 0; w < kSweepThreads / 32; ++w) t += s_warp[w];
        counts[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(kSweepThreads) k_sweep_scatter(const uint4* __restrict__ occ16, const uint4* __restrict__ gtab16, const uint16_t* __restrict__ feas,
                                                                  uint32_t first_block, uint32_t lo, uint32_t hi, Ctrl* ctrl,
                                                                  const uint32_t* __restrict__ counts, uint32_t* __restrict__ cand,
                                                                  uint16_t* __restrict__ cand_o16, const uint8_t* __restrict__ capn, const uint32_t* __restrict__ seq,
                                                                  const uint16_t* __restrict__ q, uint8_t* __restrict__ occ8, uint2* __restrict__ out_chunk,
                                                                  const uint32_t* __restrict__ heads_in, uint32_t* __restrict__ heads_out, const uint8_t* __restrict__ sizes, uint32_t flip) {
    __shared__ uint16_t s_feas[kMaxTables * 256];
    __shared__ uint32_t s_warp[kSweepThreads / 32];
    __shared__ uint32_t s_red[kSweepThreads / 32];
    __shared__ uint32_t s_base;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    for (uint32_t i = tid; i < kMaxTables * 256; i += kSweepThreads) s_feas[i] = feas[i];
    // base = number of candidates in the CTAs before this one (and the grand total for the last CTA)
    uint32_t pre = 0;
    for (uint32_t b = tid; b < blockIdx.x; b += kSweepThreads) pre += counts[b];
#pragma unroll
    for (int d = 16; d; d >>= 1) pre += __shfl_xor_sync(0xFFFFFFFFu, pre, d);
    if (lane == 0) s_red[warp] = pre;
    __syncthreads();
    if (tid == 0) { uint32_t t = 0; for (uint32_t w = 0; w < kSweepThreads / 32; ++w) t += s_red[w]; s_base = t; }
    const uint32_t active = ctrl->active;
    const uint32_t g0 = (first_block + blockIdx.x) * kSweepBlock + tid * kSweepPerThread;
    uint4 v = make_uint4(0, 0, 0, 0), tv = make_uint4(0, 0, 0, 0);
    uint32_t mask = 0;
    const bool scan_mode = __popc(active) == 1;
    const uint32_t sp = scan_mode ? __ffs(active) - 1 : 0u;
    uint32_t cap_sum = 0;
    if (active && g0 < hi && g0 + kSweepPerThread > lo) {
        v = ld_nc_v4(&occ16[g0 >> 4]); tv = ld_nc_v4(&gtab16[g0 >> 4]);
        if (scan_mode) cap_sum = scan_capacity16(v, tv, capn, sp, g0, lo, hi);
        else mask = sweep_mask16(v, tv, s_feas, active, g0, lo, hi);
    }
    const uint32_t c = scan_mode ? cap_sum : __popc(mask);
    uint32_t incl = c;                                  // inclusive warp scan of the per-thread counts
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d); if ((int)lane >= d) incl += t; }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t off = s_base + incl - c;
    for (uint32_t w = 0; w < warp; ++w) off += s_warp[w];
    const uint32_t wv[4] = {v.x, v.y, v.z, v.w}, twv[4] = {tv.x, tv.y, tv.z, tv.w};
    if (scan_mode) {        // `off` is the exclusive scan of the capacities = queue position this thread's first GPU starts at
        const uint32_t h0 = heads_in ? heads_in[sp] : 0u, n_p = ctrl->qcnt[sp];
        const uint16_t* qp = q + ctrl->qoff[sp];
        uint32_t pos = h0 + off;
        if (cap_sum && pos < n_p) {
#pragma unroll 1
            for (uint32_t j = 0; j < 16 && pos < n_p; ++j) {
                const uint32_t g = g0 + j;
                if (g < lo || g >= hi) continue;
                const uint32_t o = (wv[j >> 2] >> ((j & 3u) * 8u)) & 0xFFu, t = (twv[j >> 2] >> ((j & 3u) * 8u)) & (kMaxTables - 1);
                const uint32_t row = (t * ISL_MAX_PROFILES + sp) * 256 + o;
                const uint32_t cg = capn[row], size = sizes[t * ISL_MAX_PROFILES + sp];
                if (!cg) continue;
                uint32_t starts = seq[row], o2 = o;
                for (uint32_t k = 0; k < cg && pos < n_p; ++k, ++pos) {
                    const uint32_t st = (starts >> (4 * k)) & 15u;
                    out_chunk[qp[pos]] = pack_result(flip_gpu(g, flip), st, size, ISL_ST_PLACED);
                    o2 |= (((1u << size) - 1u) << st) & 0xFFu;
                }
                occ8[g] = (uint8_t)o2;
            }
        }
        if (blockIdx.x == gridDim.x - 1 && tid == kSweepThreads - 1) {      // `off + cap_sum` = total capacity of the range
            const uint32_t total = off + cap_sum, left = n_p > h0 ? n_p - h0 : 0u, placed = min(total, left);
            ctrl->n_cand = 0; ctrl->n_log = 0;                              // the chain and k_commit have nothing to do
            if (heads_out) heads_out[sp] = h0 + placed;
            if (placed) { atomicAdd(&ctrl->placed, (unsigned long long)placed); atomicAdd(&ctrl->scanned, (unsigned long long)placed); }
        }
        return;
    }
    uint32_t m = mask;
    while (m) {
        const uint32_t j = __ffs(m) - 1; m &= m - 1;
        const uint32_t o = (wv[j >> 2] >> ((j & 3u) * 8u)) & 0xFFu, t = (twv[j >> 2] >> ((j & 3u) * 8u)) & (kMaxTables - 1);
        cand_o16[off] = (uint16_t)(o | table_tag(t));          // what the chain needs: occupancy + table tag
        cand[off++] = ((g0 + j) << 8) | o;                       // what the commit needs: the GPU
    }
    if (blockIdx.x == gridDim.x - 1 && tid == kSweepThreads - 1) ctrl->n_cand = off;
}

// ---------------------------------------------------------------------------------------------
// k_chain<K>: the exact commit decision chain.
//
// First-fit in canonical GPU order is GPU-major stream filtering: GPU g accepts, in request
// order, a prefix of each profile's remaining queue (occupancy only grows inside an alloc phase, so
// a profile that stopped fitting on g never fits again).  The state between GPUs is one queue head
// per profile.  The chain is a latency-bound sequential recurrence, so ONE warp walks the candidate
// GPUs and does nothing but decide; lane l owns up to K (profile, start) candidates with their slot
// masks in registers.  One warp min-reduction per accepted placement answers "which pending
// request is next and where does it start", looking at the current candidate GPU and the one after
// it at once:
//     key = sel << 31 | t << 15 | profile << 11 | order << 8 | mask
//       sel  0 = the candidate's mask is free on the current GPU, 1 = only on the next GPU
//       t    in-chunk index of the next pending request of the candidate's profile
//     m = warp-min(key):  lowest GPU first, then earliest request, then first legal start in row order
//     occupancy |= m & 0xFF; the lanes of the winning profile pop their queue head.
// Every decision is appended to a log (8 B: m, candidate index); k_commit turns the log into result
// records and occupancy updates with full parallelism afterwards.
// m == INF means neither GPU can take anything: a ballot over the feasibility table jumps straight to
// the next candidate GPU on which a profile that still has pending requests fits.
// The queues (16-bit in-chunk indices) are staged once in shared memory; the candidate list streams
// through a 256-entry shared ring refilled one 32-entry block ahead from a register-held load.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kRing = 256;

// The chain itself, run by ONE warp (shared by k_chain and k_small).  qoff / qcnt: queue layout of the chunk; s_q: the
// queues in shared memory; cand_o16: occupancy + table tag of every candidate GPU in canonical order (global memory,
// streamed through s_ring); log: one (key, candidate index) record per decision.  Returns the number of decisions.
template <int K>
__device__ __forceinline__ uint32_t chain_warp(const CandTab& tab, const uint32_t* qoff, const uint32_t* qcnt, const uint16_t* s_q, uint32_t* s_ring,
                                               const uint16_t* s_feas, const uint16_t* __restrict__ cand_o16, uint32_t n_cand, uint2* log,
                                               const uint32_t* __restrict__ heads_in, uint32_t* __restrict__ heads_out, uint32_t lane,
                                               uint32_t* visited_out, uint32_t* jumps_out) {
    uint32_t cmask[K], keylow[K], pbit[K], head[K], left[K], qa[K], tcur[K], tnext[K];
    bool reports[K];
    uint32_t rem = 0;                       // requests still pending over all profiles that have a candidate (warp-uniform)
    {
        uint32_t seen = 0;
        for (uint32_t k = 0; k < 4; ++k)
            for (uint32_t l = 0; l < 32; ++l) {
                const uint32_t d = tab.desc[k][l];
                if (!(d >> 31)) continue;
                const uint32_t p = d & 15u;
                if ((seen >> p) & 1u) continue;
                seen |= 1u << p;
                const uint32_t h = heads_in ? heads_in[p] : 0u, e = qcnt[p];
                rem += e > h ? e - h : 0u;
            }
    }
    const uint32_t rem0 = rem;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const uint32_t d = tab.desc[k][lane];
        const bool valid = d >> 31;
        const uint32_t p = d & 15u;
        cmask[k] = valid ? ((d >> 16) & 0xFFu) | (1u << (8 + ((d >> 24) & 7u))) : 0xFFFFu;      // slot mask + own-table bit
        keylow[k] = (p << 11) | (((d >> 4) & 7u) << 8) | (cmask[k] & 0xFFu);
        pbit[k] = valid ? 1u << p : 0u;
        reports[k] = valid && ((d >> 4) & 7u) == 0;       // first candidate of the row reports the head
        const uint32_t qb = qoff[p], end = valid ? qcnt[p] : 0u;
        head[k] = heads_in ? heads_in[p] : 0u;
        left[k] = end > head[k] ? end - head[k] : 0u;      // requests of this profile not yet popped
        qa[k] = qb + head[k];                              // shared-memory index of the current head entry
        tcur[k] = left[k] > 0 ? ((uint32_t)s_q[qa[k]] << 15) | keylow[k] : kInf;
        tnext[k] = left[k] > 1 ? ((uint32_t)s_q[qa[k] + 1] << 15) | keylow[k] : kInf;
    }
    auto ldc = [&](uint32_t idx) -> uint32_t { return idx < n_cand ? (uint32_t)__ldcg(cand_o16 + idx) : 0xFFFFu; };   // past the end: nothing fits
    uint32_t fill = 0, pending;
    auto reload = [&](uint32_t at) {       // synchronous (re)fill of 5 blocks starting at the block that holds `at`
        __syncwarp();                          // every lane is done reading the slots that are about to be overwritten
        fill = at & ~31u;
        for (int b = 0; b < 5; ++b) { s_ring[(fill + lane) & (kRing - 1)] = ldc(fill + lane); fill += 32; }
        pending = ldc(fill + lane);
        __syncwarp();
    };
    reload(0);
    uint32_t i0 = 0;
    uint32_t o0 = s_ring[0], o1 = s_ring[1], o2 = s_ring[2];
    uint32_t jumps = 0;
    uint2* lp = log;
    while (rem) {
        uint32_t key = kInf;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const uint32_t kk = (o0 & cmask[k]) == 0 ? tcur[k] : ((o1 & cmask[k]) == 0 ? tcur[k] | 0x80000000u : kInf);
            key = min(key, kk);
        }
        const uint32_t m = __reduce_min_sync(0xFFFFFFFFu, key);
        if (m == kInf) {
            // Neither GPU takes anything.  Ballot over the next candidates for one on which a profile that still has
            // pending requests fits (the list was built for every profile pending at chunk start).
            uint32_t alive = 0;
#pragma unroll
            for (int k = 0; k < K; ++k) alive |= tcur[k] != kInf ? pbit[k] : 0u;
            alive = __reduce_or_sync(0xFFFFFFFFu, alive);
            uint32_t j = i0 + 2;
            bool found = false;
            while (j < n_cand) {
                const uint32_t c = ldc(j + lane);                 // table = the one cleared bit of the tag
                const uint32_t b = __ballot_sync(0xFFFFFFFFu, c != 0xFFFFu && (s_feas[(__ffs(~(c >> 8) & 0xFFu) - 1) * 256 + (c & 0xFFu)] & alive) != 0);
                if (b) { j += __ffs(b) - 1; found = true; break; }
                j += 32;
            }
            ++jumps;
            if (!found) break;
            i0 = j;
            if (i0 + 64 > fill) reload(i0);
            o0 = s_ring[i0 & (kRing - 1)]; o1 = s_ring[(i0 + 1) & (kRing - 1)]; o2 = s_ring[(i0 + 2) & (kRing - 1)];
            continue;
        }
        const uint32_t sel = m >> 31;
        if (lane == 0) *lp = make_uint2(m, i0 + sel);     // decision log: (key, candidate index it landed on)
        ++lp;
        if (sel) {      // warp-uniform: the current GPU is finished, the next one becomes current
            o0 = o1 | (m & 0xFFu); o1 = o2;
            ++i0;
            o2 = s_ring[(i0 + 2) & (kRing - 1)];
            if ((i0 & 31u) == 0 && fill < i0 + 224) {
                __syncwarp();
                s_ring[(fill + lane) & (kRing - 1)] = pending;
                fill += 32;
                pending = ldc(fill + lane);
                __syncwarp();
            }
        } else {
            o0 |= m & 0xFFu;
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {       // lanes of the winning profile (same t, same profile field) pop their queue
            // branch-free: the shared-memory read is unconditional (index 0 when there is nothing to read)
            const bool adv = ((m ^ tcur[k]) & 0x7FFFF800u) == 0 && tcur[k] != kInf;
            left[k] -= adv ? 1u : 0u;
            qa[k] += adv ? 1u : 0u;
            const bool more = left[k] > 1;
            const uint32_t v = s_q[more ? qa[k] + 1 : 0u];
            const uint32_t tn = more ? (v << 15) | keylow[k] : kInf;
            tcur[k] = adv ? tnext[k] : tcur[k];
            tnext[k] = adv ? tn : tnext[k];
        }
        --rem;
    }
#pragma unroll
    for (int k = 0; k < K; ++k)
        if (reports[k] && heads_out) heads_out[(keylow[k] >> 11) & 15u] = qcnt[(keylow[k] >> 11) & 15u] - left[k];
    *visited_out = i0; *jumps_out = jumps;
    return rem0 - rem;
}

template <int K>
__global__ void __launch_bounds__(kChainThreads, 1) k_chain(CandTab tab, Ctrl* ctrl, const uint16_t* __restrict__ q_global,
                                                             const uint16_t* __restrict__ cand_o16, const uint16_t* __restrict__ feas,
                                                             uint2* __restrict__ log, const uint32_t* __restrict__ heads_in,
                                                             uint32_t* __restrict__ heads_out) {
    extern __shared__ __align__(16) uint16_t s_q[];
    __shared__ uint32_t s_ring[kRing];
    __shared__ uint16_t s_feas[kMaxTables * 256];
    if (__popc(ctrl->active) == 1) {        // single-profile chunk: the sweep kernels committed it in scan mode, nothing to chain
        if (threadIdx.x == 0) ctrl->n_log = 0;
        return;
    }
    const uint32_t q_total = ctrl->qoff[ISL_MAX_PROFILES];
    {   // stage every queue of the chunk: <= 129 KB, 16-byte vector copies
        const uint4* src = reinterpret_cast<const uint4*>(q_global);
        uint4* dst = reinterpret_cast<uint4*>(s_q);
        for (uint32_t i = threadIdx.x; i < (q_total + 7) / 8; i += kChainThreads) dst[i] = src[i];
        for (uint32_t i = threadIdx.x; i < kMaxTables * 256; i += kChainThreads) s_feas[i] = feas[i];
    }
    __syncthreads();
    if (!is_chain_warp(threadIdx.x >> 5)) return;
    uint32_t visited, jumps;
    const uint32_t steps = chain_warp<K>(tab, ctrl->qoff, ctrl->qcnt, s_q, s_ring, s_feas, cand_o16, ctrl->n_cand, log, heads_in, heads_out, threadIdx.x,
                                         &visited, &jumps);
    if (threadIdx.x == 0) {
        ctrl->n_log = steps;
        atomicAdd(&ctrl->placed, (unsigned long long)steps);
        atomicAdd(&ctrl->steps, (unsigned long long)steps);
        atomicAdd(&ctrl->visited, (unsigned long long)visited);
        atomicAdd(&ctrl->jumps, (unsigned long long)jumps);
    }
}

// ---------------------------------------------------------------------------------------------
// k_small<K>: the whole hot path of ONE small batch (<= 1024 requests) in ONE launch of ONE CTA — the latency path
// (BASELINE config 5: a reconciler handing over one or two pods at a time).  Same steps as the big path:
//   A  frees / default results / stable partition of the ALLOC requests into per-profile queues (shared memory)
//   B  vectorised sweep of the inventory with ordered compaction of the candidate GPUs (16 GPUs per thread and round)
//   C  the decision chain (warp 0)
//   D  commit of the logged decisions
// Tiny batches (<= 64 requests) arrive as kernel parameters and their results go straight to mapped pinned host memory,
// so the call is one launch and one stream synchronisation.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kSmallThreads = 1024;
constexpr uint32_t kSmallMax = 1024;              // requests: one per thread in phase A
constexpr uint32_t kSmallInline = 64;             // requests that travel as kernel parameters
struct SmallReqs { uint2 r[kSmallInline]; };

template <int K>
__global__ void __launch_bounds__(kSmallThreads, 1) k_small(CandTab tab, DevProfiles prof, uint32_t n, const uint2* __restrict__ in, SmallReqs inl,
                                                             uint2* __restrict__ out, uint8_t* __restrict__ occ, const uint8_t* __restrict__ gtab,
                                                             const uint16_t* __restrict__ feas, uint32_t G, uint32_t lo, uint32_t hi,
                                                             uint32_t cand_profiles, uint32_t* __restrict__ cand, uint16_t* __restrict__ cand_o16, Ctrl* stats) {
    __shared__ uint16_t s_q[kSmallMax + kQPad * ISL_MAX_PROFILES];
    __shared__ uint32_t s_ring[kRing];
    __shared__ uint16_t s_feas[kMaxTables * 256];
    __shared__ uint32_t s_seg[32][ISL_MAX_PROFILES];
    __shared__ uint32_t s_qoff[ISL_MAX_PROFILES + 1], s_qcnt[ISL_MAX_PROFILES], s_scan[32], s_active, s_base, s_nlog, s_freed;
    __shared__ uint2 s_log[kSmallMax];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    uint32_t* occ32 = reinterpret_cast<uint32_t*>(occ);
    for (uint32_t i = tid; i < kMaxTables * 256; i += kSmallThreads) s_feas[i] = feas[i];
    if (tid < 32 * ISL_MAX_PROFILES) (&s_seg[0][0])[tid] = 0;
    if (tid == 0) { s_base = 0; s_freed = 0; }
    __syncthreads();
    // ---- A: one request per thread
    uint32_t key = kSkip, rank = 0;
    if (tid < n) {
        const uint2 rq = in ? in[tid] : inl.r[tid];
        const uint32_t handle = rq.x, profile = rq.y & 0xFFu, op = (rq.y >> 8) & 0xFFu, start = (rq.y >> 16) & 0xFFu, size = rq.y >> 24;
        if (op == ISL_OP_ALLOC) {
            if (profile < prof.n) { key = profile; out[tid] = pack_result(ISL_GPU_NONE, ISL_START_NONE, prof.rows[profile].size, ISL_ST_NO_CAPACITY); }
            else out[tid] = pack_result(ISL_GPU_NONE, ISL_START_NONE, 0, ISL_ST_BAD_PROFILE);
        } else if (op == ISL_OP_FREE) {
            if (handle >= G || size == 0 || start + size > ISL_SLOTS) out[tid] = pack_result(handle, start, size, ISL_ST_BAD_SPAN);
            else {
                const uint32_t gi = flip_gpu(handle, prof.flip);
                if (gi >= lo && gi < hi) { atomicAnd(&occ32[gi >> 2], ~((((1u << size) - 1u) << start) << ((gi & 3u) * 8u))); atomicAdd(&s_freed, 1u); }
                out[tid] = pack_result(handle, start, size, ISL_ST_FREED);
            }
        } else out[tid] = pack_result(ISL_GPU_NONE, ISL_START_NONE, 0, ISL_ST_NOOP);
    }
    {
        const uint32_t peers = __match_any_sync(0xFFFFFFFFu, key);
        rank = __popc(peers & ((1u << lane) - 1u));
        if (key != kSkip && lane == (uint32_t)(__ffs(peers) - 1)) s_seg[warp][key] = __popc(peers);
    }
    __syncthreads();
    if (tid < ISL_MAX_PROFILES) {           // exclusive scan over the 32 warps, in request order
        uint32_t run = 0;
        for (uint32_t w = 0; w < 32; ++w) { const uint32_t c = s_seg[w][tid]; s_seg[w][tid] = run; run += c; }
        s_qcnt[tid] = run;
    }
    __syncthreads();
    if (tid == 0) {
        uint32_t off = 0, active = 0, allocs = 0;
        for (uint32_t p = 0; p < ISL_MAX_PROFILES; ++p) {
            s_qoff[p] = off;
            if (s_qcnt[p] && ((cand_profiles >> p) & 1u)) active |= 1u << p;
            allocs += s_qcnt[p];
            off += (s_qcnt[p] + kQPad - 1) & ~(kQPad - 1);
        }
        s_qoff[ISL_MAX_PROFILES] = off; s_active = active;
        if (allocs) atomicAdd(&stats->allocs, (unsigned long long)allocs);
        if (s_freed) atomicAdd(&stats->freed, (unsigned long long)s_freed);
    }
    __threadfence();                        // the frees must be visible to the sweep's loads
    __syncthreads();
    if (key != kSkip) s_q[s_qoff[key] + s_seg[warp][key] + rank] = (uint16_t)tid;
    // ---- B: sweep, 16 GPUs per thread and round, ordered compaction into cand / cand_o16
    const uint32_t active = s_active;
    if (active) {
        for (uint32_t base = lo / (kSmallThreads * 16u) * (kSmallThreads * 16u); base < hi; base += kSmallThreads * 16u) {
            const uint32_t g0 = base + tid * 16u;
            uint4 v = make_uint4(0, 0, 0, 0), tv = make_uint4(0, 0, 0, 0);
            uint32_t mask = 0;
            if (g0 < hi && g0 + 16u > lo) {
                v = __ldcg(reinterpret_cast<const uint4*>(occ) + (g0 >> 4)); tv = __ldcg(reinterpret_cast<const uint4*>(gtab) + (g0 >> 4));
                mask = sweep_mask16(v, tv, s_feas, active, g0, lo, hi);
            }
            const uint32_t c = __popc(mask);
            uint32_t incl = c;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d); if ((int)lane >= d) incl += t; }
            if (lane == 31) s_scan[warp] = incl;
            __syncthreads();
            if (warp == 0) {                    // exclusive scan of the 32 warp totals
                const uint32_t t = s_scan[lane];
                uint32_t x = t;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, d); if ((int)lane >= d) x += y; }
                s_scan[lane] = x - t;
                if (lane == 31) s_nlog = x;     // round total (s_nlog is reused as scratch here)
            }
            __syncthreads();
            uint32_t off = s_base + s_scan[warp] + incl - c;
            const uint32_t wv[4] = {v.x, v.y, v.z, v.w}, twv[4] = {tv.x, tv.y, tv.z, tv.w};
            uint32_t m = mask;
            while (m) {
                const uint32_t j = __ffs(m) - 1; m &= m - 1;
                const uint32_t o = (wv[j >> 2] >> ((j & 3u) * 8u)) & 0xFFu, t = (twv[j >> 2] >> ((j & 3u) * 8u)) & (kMaxTables - 1);
                cand_o16[off] = (uint16_t)(o | table_tag(t));
                cand[off++] = ((g0 + j) << 8) | o;
            }
            __syncthreads();
            if (tid == 0) s_base += s_nlog;
            __syncthreads();
        }
    }
    __threadfence();
    __syncthreads();
    // ---- C: the chain
    if (is_chain_warp(warp)) {
        uint32_t visited = 0, jumps = 0;
        const uint32_t steps = active ? chain_warp<K>(tab, s_qoff, s_qcnt, s_q, s_ring, s_feas, cand_o16, s_base, s_log, nullptr, nullptr, lane, &visited, &jumps) : 0u;
        if (lane == 0) {
            s_nlog = steps;
            if (steps) { atomicAdd(&stats->placed, (unsigned long long)steps); atomicAdd(&stats->steps, (unsigned long long)steps); }
            if (visited) atomicAdd(&stats->visited, (unsigned long long)visited);
            if (jumps) atomicAdd(&stats->jumps, (unsigned long long)jumps);
        }
    }
    __syncthreads();
    // ---- D: commit
    for (uint32_t j = tid; j < s_nlog; j += kSmallThreads) {
        const uint2 e = s_log[j];
        const uint32_t g = __ldcg(cand + e.y) >> 8, mask = e.x & 0xFFu, t = (e.x >> 15) & 0xFFFFu;
        out[t] = pack_result(flip_gpu(g, prof.flip), __ffs(mask) - 1, __popc(mask), ISL_ST_PLACED);
        atomicOr(&occ32[g >> 2], mask << ((g & 3u) * 8u));
    }
}

// ---------------------------------------------------------------------------------------------
// k_few: the latency path of a reconciler that hands over one or two pods at a time (BASELINE configs 1 and 5): at most
// kFewMax requests, an inventory range of at most kFewGpus GPUs, first-fit.  Request-major on purpose — with a handful of
// requests there is nothing to amortise a partition / sweep / chain over: ONE CTA holds 16 occupancy bytes per thread in
// registers, the first-start tables in shared memory, and for every ALLOC in order finds the first feasible GPU with a
// block-wide min (redux + one shared-memory hop) — exactly the reference's scan order (:240-262, :303-384).  Requests travel as
// kernel parameters, results go straight to mapped pinned host memory: one launch, one stream synchronisation.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kFewThreads = 1024;
constexpr uint32_t kFewMax = 8;
constexpr uint32_t kFewGpus = kFewThreads * 16;

__global__ void __launch_bounds__(kFewThreads, 1) k_few(DevProfiles prof, uint32_t n, SmallReqs inl, uint2* __restrict__ out, uint8_t* __restrict__ occ,
                                                         const uint8_t* __restrict__ gtab, const uint8_t* __restrict__ lut, const uint8_t* __restrict__ sizes,
                                                         uint32_t n_tables, uint32_t G, uint32_t lo, uint32_t hi, Ctrl* stats) {
    __shared__ __align__(16) uint8_t s_lut[kMaxTables * ISL_MAX_PROFILES * 256];
    __shared__ uint8_t s_sizes[kMaxTables * ISL_MAX_PROFILES];
    __shared__ uint32_t s_red[32], s_win;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    uint32_t* occ32 = reinterpret_cast<uint32_t*>(occ);
    for (uint32_t i = tid; i < n_tables * ISL_MAX_PROFILES * 64; i += kFewThreads) reinterpret_cast<uint32_t*>(s_lut)[i] = reinterpret_cast<const uint32_t*>(lut)[i];
    if (tid < n_tables * ISL_MAX_PROFILES) s_sizes[tid] = sizes[tid];
    uint32_t freed = 0, allocs = 0;
    if (tid < n) {          // defaults and FREEs, one request per thread (as k_prepare / k_small phase A)
        const uint2 rq = inl.r[tid];
        const uint32_t handle = rq.x, profile = rq.y & 0xFFu, op = (rq.y >> 8) & 0xFFu, start = (rq.y >> 16) & 0xFFu, size = rq.y >> 24;
        if (op == ISL_OP_ALLOC) {
            if (profile < prof.n) { out[tid] = pack_result(ISL_GPU_NONE, ISL_START_NONE, prof.rows[profile].size, ISL_ST_NO_CAPACITY); allocs = 1; }
            else out[tid] = pack_result(ISL_GPU_NONE, ISL_START_NONE, 0, ISL_ST_BAD_PROFILE);
        } else if (op == ISL_OP_FREE) {
            if (handle >= G || size == 0 || start + size > ISL_SLOTS) out[tid] = pack_result(handle, start, size, ISL_ST_BAD_SPAN);
            else {
                const uint32_t gi = flip_gpu(handle, prof.flip);
                if (gi >= lo && gi < hi) { atomicAnd(&occ32[gi >> 2], ~((((1u << size) - 1u) << start) << ((gi & 3u) * 8u))); freed = 1; }
                out[tid] = pack_result(handle, start, size, ISL_ST_FREED);
            }
        } else out[tid] = pack_result(ISL_GPU_NONE, ISL_START_NONE, 0, ISL_ST_NOOP);
    }
    __threadfence();                        // the frees must be visible to the loads below
    __syncthreads();
    // 16 GPUs per thread, aligned to 16: the byte of a GPU outside [lo, hi) reads as full
    const uint32_t g0 = (lo & ~15u) + tid * 16u;
    uint4 v = make_uint4(~0u, ~0u, ~0u, ~0u), tv = make_uint4(0, 0, 0, 0);
    if (g0 < hi) { v = __ldcg(reinterpret_cast<const uint4*>(occ) + (g0 >> 4)); if (n_tables > 1) tv = __ldcg(reinterpret_cast<const uint4*>(gtab) + (g0 >> 4)); }
    uint32_t wv[4] = {v.x, v.y, v.z, v.w};
    const uint32_t twv[4] = {tv.x, tv.y, tv.z, tv.w};
    for (uint32_t r = 0; r < n; ++r) {      // the ALLOCs strictly in request order, each seeing all earlier commits
        const uint32_t w = inl.r[r].y, p = w & 0xFFu, op = (w >> 8) & 0xFFu;
        if (op != ISL_OP_ALLOC || p >= prof.n) continue;        // uniform
        uint32_t best = kInf;
#pragma unroll
        for (int j = 15; j >= 0; --j) {     // descending, so the lowest feasible GPU of the thread is what remains
            const uint32_t g = g0 + j, o = (wv[j >> 2] >> ((j & 3) * 8)) & 0xFFu, t = (twv[j >> 2] >> ((j & 3) * 8)) & (kMaxTables - 1);
            if (g >= lo && g < hi && s_lut[(t * ISL_MAX_PROFILES + p) * 256 + o] != ISL_START_NONE) best = g;
        }
        const uint32_t wm = __reduce_min_sync(0xFFFFFFFFu, best);
        if (lane == 0) s_red[warp] = wm;
        __syncthreads();
        if (warp == 0) { const uint32_t m = __reduce_min_sync(0xFFFFFFFFu, s_red[lane]); if (lane == 0) s_win = m; }
        __syncthreads();
        const uint32_t g = s_win;
        if (g != kInf && g >= g0 && g < g0 + 16u) {             // the owner commits
            const uint32_t j = g - g0, sh = (j & 3u) * 8u, o = (wv[j >> 2] >> sh) & 0xFFu, t = (twv[j >> 2] >> sh) & (kMaxTables - 1);
            const uint32_t st = s_lut[(t * ISL_MAX_PROFILES + p) * 256 + o], size = s_sizes[t * ISL_MAX_PROFILES + p];
            const uint32_t o2 = o | ((((1u << size) - 1u) << st) & 0xFFu);
            wv[j >> 2] = (wv[j >> 2] & ~(0xFFu << sh)) | (o2 << sh);
            occ[g] = (uint8_t)o2;
            out[r] = pack_result(flip_gpu(g, prof.flip), st, size, ISL_ST_PLACED);
            atomicAdd(&stats->placed, 1ull); atomicAdd(&stats->steps, 1ull);
        }
        // s_red / s_win are rewritten only after the next request's first barrier has been passed by everybody who read them
    }
    // statistics (off the caller's critical path: the results are already on their way)
    if (freed) atomicAdd(&stats->freed, 1ull);
    if (allocs) atomicAdd(&stats->allocs, 1ull);
}

// ---------------------------------------------------------------------------------------------
// k_commit: one thread per logged decision.  Writes the result record of the request (the fields of
// AllocationDetails the allocator decides) and ORs the slot mask into the packed occupancy word.
// Distinct decisions on one GPU have disjoint masks (the chain only accepts free masks): no double
// booking; the atomics only serialise neighbours that share a 32-bit word.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_commit(const Ctrl* __restrict__ ctrl, const uint2* __restrict__ log, const uint32_t* __restrict__ cand,
                                                 uint32_t* __restrict__ occ32, uint2* __restrict__ out_chunk, uint32_t flip) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= ctrl->n_log) return;
    const uint2 e = log[j];
    const uint32_t g = cand[e.y] >> 8, mask = e.x & 0xFFu, t = (e.x >> 15) & 0xFFFFu;
    out_chunk[t] = pack_result(flip_gpu(g, flip), __ffs(mask) - 1, __popc(mask), ISL_ST_PLACED);
    atomicOr(&occ32[g >> 2], mask << ((g & 3u) * 8u));
}

// ---------------------------------------------------------------------------------------------
// k_pipeline<K>: the segment pipeline for STREAMS of batches (BASELINE config 4's shape).
//
// The commit chain of one chunk is sequential, but chunks of a stream pipeline exactly over
// inventory segments: segment s may work on chunk c+1 while segment s+1 is still on chunk c, because
//   * inside a segment everything happens in stream order: allocs of chunk c, then the frees of the
//     next batch, then its allocs (occupancy of the segment lives in this CTA's shared memory), and
//   * the only state that crosses a segment boundary is the per-profile queue-head token (16 counters).
// One persistent CTA per segment (cooperative launch, all co-resident; one CTA fills an SM's shared memory).  Per chunk a CTA
//   0. has the chunk's queues (uint16 request indices) copied into shared memory by cp.async, issued when the previous
//      chunk's chain ended: they do not depend on the token
//   1. applies the batch's frees that fall into its range                      (all threads)
//   2. sweeps its occupancy bytes into an ordered candidate list               (all threads, before the token arrives)
//   3. waits for the token of segment s-1 (self-validating words: epoch tag + head, polled by 16 lanes), converts the queue
//      windows it may pop into ready-made 32-bit keys (shared -> shared)
//   4. runs the decision chain on its candidates                               (warp 0; DESIGN.md 4.1)
//   5. publishes the token for segment s+1 and only then
//   6. commits the logged decisions: result records + occupancy bits           (all threads)
// Host-buffer streams: the batches are fed by a second stream while this kernel runs (ready flags), an extra CTA delivers
// finished chunks into the caller's pinned result array (done counters).
// Results are bit-identical to resolving the batches one after the other.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kSegMax = 512;                   // GPUs per (sub-)segment (2 per thread in the local sweep)
constexpr uint32_t kSubMax = 8;                     // sub-segments one CTA walks per chunk: inventories beyond 148 x 512 GPUs stay on the pipeline
#ifndef ISL_PIPE_THREADS
#define ISL_PIPE_THREADS 256
#endif
constexpr uint32_t kPipeThreads = ISL_PIPE_THREADS;     // 1 or 2 GPUs per thread in the local sweep
static_assert(kPipeThreads == kSegMax || 2 * kPipeThreads == kSegMax, "sweep layout");
constexpr uint32_t kLogCap = 8 * kSegMax;           // a GPU accepts at most 8 placements
constexpr uint32_t kTokStride = 32;                 // uint32 per token: 16 tagged head words inside a GPU; raw heads[16] + flag at [16] across GPUs
// shared memory: occupancy bytes | candidate records (+8 sentinels) | decision log (+1 pseudo-decision) | the chunk's queues (uint16) | queue-window keys
constexpr uint32_t kPipeOffCand = kSegMax * kSubMax;      // occupancy bytes of the whole stage (all its sub-segments)
constexpr uint32_t kCandPad = 16;                   // INF records behind a segment's candidates: a group of pseudo-decisions may walk that far
constexpr uint32_t kWinPad = 10;                    // INF keys behind every queue window: an exhausted lane is popped at most once per decision of a group
constexpr uint32_t kPipeOffLog = kPipeOffCand + 4 * (kSegMax + kCandPad);
constexpr uint32_t kPipeOffQ = (kPipeOffLog + 8 * (kLogCap + 1) + 15u) & ~15u;
constexpr uint32_t kPipeOffWin = kPipeOffQ + 2 * kQCap + 16;
constexpr uint32_t kWinTotal = 12288;               // 32-bit queue-window keys a segment can stage for all profiles together
constexpr uint32_t kPipeSmem = kPipeOffWin + 4 * (kWinTotal + 4 * ISL_MAX_PROFILES);

// largest segment whose worst-case queue windows (every candidate GPU accepting every legal start of every
// profile) fit: n_cand * total_candidates + 2 sentinels per profile <= kWinTotal
constexpr uint32_t kWinMargin = 32;                 // speculative rounds: queue entries staged on either side of a window, so that a corrected entry nearby re-uses it
__host__ __device__ inline uint32_t max_segment_for(uint32_t total_candidates) {
    const uint32_t s = (kWinTotal - (kWinPad + 2 * kWinMargin + 2) * ISL_MAX_PROFILES) / (total_candidates ? total_candidates : 1u);
    return s >= kSegMax ? kSegMax : s / 64u * 64u;
}

struct ChunkDesc {
    uint32_t req_off, n, batch, first_of_batch;
    uint2* host_out;                // open streams: mapped pinned destination of this chunk's results (nullptr: PipeArgs.host_out + req_off)
    uint64_t pad;
};

struct PipeArgs {
    uint32_t n_chunks, n_seg, seg, lo, hi, epoch;     // seg: GPUs per pipeline stage (CTA) = sub x sub-segments
    uint32_t sub;                                     // GPUs per sub-segment (<= kSegMax): what one sweep / chain / commit round covers
    const ChunkDesc* chunks;
    const Ctrl* cctl;               // per chunk: qoff / qcnt / active (written by k_partition)
    const uint16_t* q_all;          // per chunk queues, stride q_stride entries
    const uint8_t* free_acc;        // per batch one byte per GPU: OR of the slot masks its FREEs release (stride free_stride bytes)
    uint32_t q_stride, free_stride;
    uint32_t* tokens;               // [chunk][segment + 1][kTokStride] of (epoch tag << 17 | head); slot n_seg = 'everything placeable is placed' broadcast
    uint8_t* occ;
    const uint8_t* gtab;            // table id of every GPU's node
    uint2* out;
    const uint16_t* feas;
    Ctrl* stats;
    const uint32_t* heads_in;       // [chunk][16] token entering the first segment (nullptr = zeros)
    uint32_t* heads_out;            // [chunk][16] token leaving the last segment (may be nullptr)
    // partitioned inventory: the token crosses GPUs through peer-mapped memory (NVLink), system-scope release/acquire
    const uint32_t* inbox;          // local [chunk][kTokStride] of tagged head words, written by the previous rank's last segment (nullptr = first rank); cleared by the reader
    uint32_t* outbox;               // the next rank's inbox, peer-mapped (nullptr = last rank)
    uint32_t xepoch;                // stream id shared by all ranks
    // host-buffer streams (isl_place_stream): the batches are fed while the pipeline runs, the results leave chunk by chunk
    const uint32_t* ready;          // [batch] == epoch once the batch's requests are in HBM and its pre-pass is done (nullptr = all ready)
    uint32_t* done_cnt;             // [chunk] segments that have committed the chunk (zeroed per call; nullptr = no copier CTA)
    uint2* host_out;                // mapped pinned result array of the caller: CTA n_seg copies every complete chunk there
    // open streams (isl_stream_open / _submit / _wait / _close): batches arrive while the kernel runs, one chunk per batch, n_chunks is
    // the capacity; ready[b] == ~epoch closes the stream.  host_done[c] = epoch (mapped pinned) tells the host that chunk c is delivered.
    uint32_t open, copier;          // copier: an extra CTA (index n_seg) delivers finished chunks to host memory
    uint32_t* host_done;
    // causal window: chunk c may start only after chunk c - window has been committed by every segment (0 = no constraint)
    uint32_t window;
    unsigned long long wait_ns;     // a starved wait traps after this long instead of hanging the GPU
    // partitioned inventory, results gathered on the owner rank: peer-mapped result array of rank 0 (nullptr = keep results local)
    uint2* owner_out;
    // causal window across ranks: the CTA that completes a chunk on its rank adds 1 to ring_done[chunk] on the owner rank (peer atomic);
    // the owner starts chunk c only when ring_done[c - window] == world
    uint32_t* ring_done; uint32_t world;
    uint32_t flip;                  // ISL_POLICY_RIGHT_TO_LEFT: G, the reported GPU is G - 1 - internal index
    unsigned long long* trace;      // optional [chunk][segment][kTraceWords]: globaltimer ns of sweep done, token in, token out, commit done, chain start, chain end; decisions; jumps | visited << 32; ns of heads done, windows staged; 2 spare
    // speculative rounds (below): every stage simulates its segment from PREDICTED queue heads at once, the predictions are corrected round
    // by round and a stage commits once its entry heads are certified to be the true ones.  Record memory: spec_mem(), kSpecWordsPerChunk per chunk.
    uint32_t spec;
    unsigned long long* spec_mem;
    // partitioned inventory: the stages of all ranks form ONE sequence (global index spec_base + stage); every rank keeps the whole record
    // memory and a stage stores what later ranks read straight into their copies (peer stores over NVLink, system scope)
    uint32_t spec_world, spec_rank, spec_base, spec_total;
    unsigned long long* spec_peer[8];
    unsigned long long* spec_dbg;   // optional [kSpecRounds][8] globaltimer stamps of the rounds of ONE (chunk, stage) cell (ISL_SPEC_DBG=chunk,stage; tools/spec_trace.py)
    uint32_t spec_dbg_cell;         // chunk << 16 | stage
};

// ---------------------------------------------------------------------------------------------
// Speculative rounds over the stages of ONE chunk (DESIGN.md 4.5) — exact, only faster.
// A chunk's decisions are one recurrence over the inventory: stage s needs the queue heads stage s-1 leaves (the token).  Instead of
// idling until the token has travelled, every stage simulates its segment at once from a PREDICTED token:
//   round 0   every stage publishes what its occupancy can take (per contention group: placements of the size >= 4 profiles, slices left
//             for the size 1/2 profiles); stage s predicts its entry heads from the sums over the stages in front of it
//   round r   stage s simulates from its predicted entry H (the exact chain of 4.1, log kept in shared memory), publishes its exit heads
//             X (to s+1) and the group masses it consumed D (to every later stage), reads X of s-1 and D of all j < s, and corrects:
//             H' = X(s-1) shifted, per group, to the mass sum of D(j), j < s   (a Newton step: a shift of the entry by conserved
//             quantities passes through a segment unchanged; the split inside a group heals by itself within a few hundred GPUs)
//   stage s is CERTIFIED in round r when H(j) of round r-1 equalled X(j-1) of round r-1 for every j <= s: by induction from stage 0
//             (whose entry is the true one) every such entry is the true token; it commits its log and publishes final records.
// Every round certifies at least one more stage, so the worst case is the token travelling stage by stage as before; predictions that
// hold certify whole runs of stages at once.  Words are self-validating (call epoch and round above the payload): no flags, no fences.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kSpecStride = 160;               // stage slots per row (>= 148 stages)
constexpr uint32_t kSpecRounds = 160;               // rounds <= stages + 2
constexpr uint32_t kSpecWordsPerChunk = kSpecStride * (32 + 16 + kSpecRounds + 1 + 2 + 1);
struct SpecMem {
    unsigned long long* x;          // [stage][round & 1][16]   tag(round) << 32 | exit head
    unsigned long long* xf;         // [stage][16]              final: tagF << 32 | certified-in-round << 24 | exit head
    unsigned long long* d;          // [round][stage]           tag(round) << 32 | c << 31 | dq << 13 | dr   (c: entry equalled the predecessor's exit one round earlier)
    unsigned long long* df;         // [stage]                  final: tagF << 32 | certified-in-round << 24 | dq << 13 | dr
    unsigned long long* m;          // [stage][2]               round 0: tag(0) << 32 | placements of the big group ; tag(0) << 32 | slices with << 16 | slices without them
    unsigned long long* ack;        // [stage]                  epoch << 32 | last round whose X(stage - 1) this stage has read
};
__host__ __device__ inline SpecMem spec_mem(unsigned long long* base, uint32_t chunk) {
    unsigned long long* p = base + (size_t)chunk * kSpecWordsPerChunk;
    SpecMem s;
    s.x = p; p += kSpecStride * 32; s.xf = p; p += kSpecStride * 16; s.d = p; p += (size_t)kSpecStride * kSpecRounds;
    s.df = p; p += kSpecStride; s.m = p; p += kSpecStride * 2; s.ack = p;
    return s;
}

constexpr uint32_t kTraceWords = 12;
#ifndef ISL_UNROLL
#define ISL_UNROLL 8
#endif
constexpr int kUnroll = ISL_UNROLL;          // decisions per trip of the decision loop
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// Trace stamp without a branch: a divergent `if (lane == 0)` in front of the decision loop can leave warp 0 split for good, and
// every redux of the loop then takes the BRA.DIV emulation path (measured: 4x slower decisions).  `p` may be any address when !pred.
__device__ __forceinline__ void stamp_if(bool pred, unsigned long long* p) {
    asm volatile("{ .reg .pred q; .reg .u64 t; setp.ne.u32 q, %0, 0; mov.u64 t, %%globaltimer; @q st.global.u64 [%1], t; }" ::"r"((uint32_t)pred), "l"(p) : "memory");
}
__device__ __forceinline__ void store_if(bool pred, unsigned long long* p, unsigned long long v) {
    asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q st.global.u64 [%1], %2; }" ::"r"((uint32_t)pred), "l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed_gpu(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_gpu(uint32_t* p, uint32_t v) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_gpu_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_gpu_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Speculative rounds: move the heads of the profiles in `members` so that their mass (sum of weight x head) changes by d.
// By a whole warp: lane p < 16 holds head h of profile p and returns the moved head.  Shares proportional to the queue lengths; the single-slice profile with the highest index (a group without one:
// its highest member) takes the remainder, so that the mass is met exactly whenever the weights allow it.  |d| <= 2^13: float shares.
__device__ __forceinline__ uint32_t spec_spread_warp(uint32_t h, uint32_t qc, uint32_t w, uint32_t members, int d, bool weighted, uint32_t lane) {
    const bool in = (members >> lane) & 1u;
    if (!weighted) w = 1;
    const uint32_t light = __ballot_sync(0xFFFFFFFFu, in && w <= 1), heavy = __ballot_sync(0xFFFFFFFFu, in && w > 1);
    const uint32_t tot = __reduce_add_sync(0xFFFFFFFFu, in ? qc * w : 0u);
    if (d == 0 || members == 0) return h;
    const uint32_t last = 31u - __clz(light ? light : heavy);
    int dp = in && lane != last && tot ? __float2int_rn((float)d * (float)qc / (float)tot) : 0;
    const int used = __reduce_add_sync(0xFFFFFFFFu, dp * (int)w);
    const int wl = (int)__shfl_sync(0xFFFFFFFFu, w, last);
    if (lane == last) dp = (d - used) / wl;
    if (!in) return h;
    const int v = (int)h + dp;
    return (uint32_t)(v < 0 ? 0 : (v > (int)qc ? (int)qc : v));
}

__device__ __forceinline__ uint32_t lds_u32(uint32_t sa) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(sa)); return v; }
__device__ __forceinline__ uint32_t lds_u16(uint32_t sa) { uint32_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(sa)); return v; }
__device__ __forceinline__ void sts_v2_if(bool pred, uint32_t sa, uint32_t x, uint32_t y) {
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %0, 0; @p st.shared.v2.u32 [%1], {%2, %3}; }" ::"r"((uint32_t)pred), "r"(sa), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ uint32_t add_if(bool pred, uint32_t x, uint32_t inc) {         // one predicated add instead of select + move
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %1, 0; @p add.u32 %0, %0, %2; }" : "+r"(x) : "r"((uint32_t)pred), "r"(inc));
    return x;
}
__device__ __forceinline__ uint32_t redux_min_u32(uint32_t v) {
    uint32_t r;
    asm volatile("redux.sync.min.u32 %0, %1, 0xffffffff;" : "=r"(r) : "r"(v));
    return r;
}
__device__ __forceinline__ uint32_t lds_u32_if(bool pred, uint32_t sa, uint32_t keep) {   // predicated load: keeps `keep` when !pred
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %1, 0; @p ld.shared.u32 %0, [%2]; }" : "+r"(keep) : "r"((uint32_t)pred), "r"(sa));
    return keep;
}

// Rare path of the decision chain, kept out of line so that the hot loop stays free of divergence-capable constructs:
// first candidate index >= from + 2 on which a profile of `alive` fits, or kInf.
__device__ __noinline__ uint32_t pipeline_skip(uint32_t sa_cand, const uint16_t* s_feas, uint32_t n_cand, uint32_t cur_plus2, uint32_t alive, uint32_t lane) {
    alive = __reduce_or_sync(0xFFFFFFFFu, alive);
    uint32_t j = cur_plus2;                      // record index of (current + 2)
    while (alive && j < n_cand) {
        const uint32_t cr = j + lane < n_cand ? lds_u32(sa_cand + 4 * (j + lane)) : kInf;
        const uint32_t b = __ballot_sync(0xFFFFFFFFu, cr != kInf && (s_feas[(__ffs(~(cr >> 8) & 0xFFu) - 1) * 256 + (cr & 0xFFu)] & alive) != 0);
        if (b) return j + __ffs(b) - 1;
        j += 32;
    }
    return kInf;
}

template <int K, bool kP15, bool kSpec>
__global__ void __launch_bounds__(kPipeThreads, 1) k_pipeline(CandTab tab, PipeArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint32_t* s_occ32 = reinterpret_cast<uint32_t*>(smem);                       // kSegMax occupancy bytes
    uint32_t* s_cand = reinterpret_cast<uint32_t*>(smem + kPipeOffCand);         // records (local gpu << 16 | table tag | occ) + sentinels
    uint2* s_log = reinterpret_cast<uint2*>(smem + kPipeOffLog);                 // (key, candidate index) per decision
    __shared__ uint16_t s_feas[kMaxTables * 256];
    __shared__ uint8_t s_tab[kSegMax * kSubMax];                                 // table of every local GPU
    __shared__ uint32_t s_heads[ISL_MAX_PROFILES], s_wn[ISL_MAX_PROFILES], s_wbase[ISL_MAX_PROFILES], s_qbeg[ISL_MAX_PROFILES], s_pop[ISL_MAX_PROFILES];
    __shared__ uint32_t s_maxacc[ISL_MAX_PROFILES], s_minsize[ISL_MAX_PROFILES], s_usable[kMaxTables], s_plist[ISL_MAX_PROFILES], s_nplist;
    __shared__ uint32_t s_warp[kPipeThreads / 32], s_ncand, s_nfree, s_nlog, s_idle, s_closed;
    // speculative rounds: predicted entry heads, own / predecessor's exit heads, queue lengths, gathered sums, contention groups
    __shared__ uint32_t s_specH[ISL_MAX_PROFILES], s_specX[ISL_MAX_PROFILES], s_specXp[ISL_MAX_PROFILES], s_qc[ISL_MAX_PROFILES];
    __shared__ uint32_t s_acc[4], s_grp_big, s_grp_small, s_specflag, s_bigd[32], s_nbigd, s_dqr[2], s_us[kMaxTables], s_qo[ISL_MAX_PROFILES];
    __shared__ uint8_t s_smallm[kMaxTables][ISL_MAX_PROFILES];
    // speculative rounds, bounded simulations: entry / exit heads of the stage's last COMPLETE simulation; {decisions of the largest complete one,
    // have one, the log in shared memory is a complete simulation of the current entry}; decisions this simulation may take; it was cut off
    // speculative rounds: the staged key windows outlive a simulation — per profile the queue position of the first staged entry, the number
    // of staged entries, where the current entry sits inside them; the windows are valid for this chunk; this simulation must stage anew
    __shared__ uint32_t s_wlo[ISL_MAX_PROFILES], s_wlen[ISL_MAX_PROFILES], s_woff[ISL_MAX_PROFILES], s_wvalid, s_restage;
    __shared__ uint32_t s_predc, s_predA[ISL_MAX_PROFILES], s_predB[ISL_MAX_PROFILES], s_havepred;
    __shared__ uint32_t s_Hc[ISL_MAX_PROFILES], s_Xc[ISL_MAX_PROFILES], s_capst[3], s_cap, s_capped;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5, seg = blockIdx.x;
    if (seg == a.n_seg) {       // the extra CTA of a host-buffer stream: every chunk all segments have committed goes to the caller's
                                // (mapped, pinned) result array right away, so the D2H of the results hides behind the rest of the stream
        __shared__ uint32_t s_stop;
        for (uint32_t c = 0; c < a.n_chunks; ++c) {
            if (tid == 0) {
                uint32_t stop = 0;
                const unsigned long long t0 = globaltimer_ns();
                while (ld_acquire_gpu(a.done_cnt + c) < a.n_seg) {
                    // a closed (or aborted) stream never commits this chunk: ready[batch] holds ~epoch
                    if (a.ready && ld_acquire_gpu(a.ready + (a.open ? c : a.chunks[c].batch)) == ~a.epoch) { stop = 1; break; }
                    __nanosleep(256);
                    if (globaltimer_ns() - t0 > a.wait_ns + 5000000000ull) __trap();
                }
                s_stop = stop;
            }
            __syncthreads();
            if (s_stop) break;
            const ChunkDesc cd = a.chunks[c];
            const uint2* __restrict__ src = a.out + cd.req_off;
            uint2* __restrict__ dst = cd.host_out ? cd.host_out : a.host_out + cd.req_off;
            // 16-byte body between an 8-byte head / tail when source and destination are 16-byte aligned at the same records;
            // otherwise (a destination that is only 8-byte aligned relative to the staging buffer) plain 8-byte stores
            const bool same = ((reinterpret_cast<uintptr_t>(src) ^ reinterpret_cast<uintptr_t>(dst)) & 8u) == 0;
            if (same) {
                const uint32_t head = min(cd.n, (uint32_t)((reinterpret_cast<uintptr_t>(dst) >> 3) & 1u)), pairs = (cd.n - head) >> 1;
                if (tid == 0 && head) dst[0] = __ldcg(src);
                const uint4* __restrict__ s4 = reinterpret_cast<const uint4*>(src + head);
                uint4* __restrict__ d4 = reinterpret_cast<uint4*>(dst + head);
#pragma unroll 4
                for (uint32_t i = tid; i < pairs; i += kPipeThreads) d4[i] = __ldcg(s4 + i);
                if (tid == 0 && ((cd.n - head) & 1u)) dst[cd.n - 1] = __ldcg(src + cd.n - 1);
            } else {
#pragma unroll 4
                for (uint32_t i = tid; i < cd.n; i += kPipeThreads) dst[i] = __ldcg(src + i);
            }
            if (a.host_done) {          // the host may read the chunk's results as soon as it sees this word
                __threadfence_system();
                __syncthreads();
                if (tid == 0) st_release_sys(a.host_done + c, a.epoch);
            }
        }
        __threadfence_system();
        return;
    }
    const uint32_t lo_s = min(a.hi, a.lo + seg * a.seg), hi_s = min(a.hi, lo_s + a.seg), n_g = hi_s - lo_s;
    const uint32_t sa_cand = (uint32_t)__cvta_generic_to_shared(s_cand), sa_log = (uint32_t)__cvta_generic_to_shared(s_log);
    const uint32_t sa_q = (uint32_t)__cvta_generic_to_shared(smem + kPipeOffQ);     // the chunk's queues: uint16 in-chunk request indices
    uint32_t* s_wkey = reinterpret_cast<uint32_t*>(smem + kPipeOffWin);          // per-profile windows of ready-made keys t<<15 | p<<11
    const uint32_t sa_wkey = (uint32_t)__cvta_generic_to_shared(s_wkey);

    for (uint32_t i = tid; i < kSegMax * kSubMax / 4; i += kPipeThreads) s_occ32[i] = 0xFFFFFFFFu;
    for (uint32_t i = tid; i < kMaxTables * 256; i += kPipeThreads) s_feas[i] = a.feas[i];
    for (uint32_t i = tid; i < kSegMax * kSubMax; i += kPipeThreads) s_tab[i] = i < n_g ? a.gtab[lo_s + i] & (kMaxTables - 1) : 0;
    if (tid < ISL_MAX_PROFILES) {
        uint32_t n = 0, sz = 8;
        for (uint32_t k = 0; k < 4; ++k) for (uint32_t l = 0; l < 32; ++l) {
            const uint32_t d = tab.desc[k][l];
            if ((d >> 31) && (d & 15u) == tid) { ++n; sz = min(sz, (uint32_t)__popc((d >> 16) & 0xFFu)); }
        }
        s_maxacc[tid] = n;
        s_minsize[tid] = max(sz, 1u);           // smallest span of the profile over all tables
        const uint32_t have = __ballot_sync(0xFFFFu, n != 0);      // profiles that own at least one candidate: only these get a window
        if (n) s_plist[__popc(have & ((1u << tid) - 1u))] = tid;
        if (tid == 0) s_nplist = __popc(have);
    }
    if (tid >= 32 && tid < 32 + kMaxTables) {   // slices any candidate of the table can ever cover (REF_EXACT 80GB-class tables: 0x7F)
        uint32_t u = 0;
        for (uint32_t k = 0; k < 4; ++k) for (uint32_t l = 0; l < 32; ++l) {
            const uint32_t d = tab.desc[k][l];
            if ((d >> 31) && ((d >> 24) & 7u) == tid - 32) u |= (d >> 16) & 0xFFu;
        }
        s_usable[tid - 32] = u;
    }
    if (kSpec && tid >= 64 && tid < 96) {      // speculative rounds: the (profile, start) candidates of >= 4 slices as a list; per (table, profile) the slices of its smaller spans
        const uint32_t l = tid - 64;
        uint32_t n = 0;
        for (uint32_t k = 0; k < 4; ++k) {
            const uint32_t d = tab.desc[k][l];
            const bool big = (d >> 31) && __popc((d >> 16) & 0xFFu) >= 4;
            const uint32_t b = __ballot_sync(0xFFFFFFFFu, big);
            if (big) { const uint32_t at = n + __popc(b & ((1u << l) - 1u)); if (at < 32) s_bigd[at] = d; }
            n += __popc(b);
        }
        if (l == 0) s_nbigd = min(n, 32u);
        for (uint32_t i = l; i < kMaxTables * ISL_MAX_PROFILES; i += 32) {
            const uint32_t t = i / ISL_MAX_PROFILES, pp = i % ISL_MAX_PROFILES;
            uint32_t u = 0;
            for (uint32_t k = 0; k < 4; ++k) for (uint32_t x = 0; x < 32; ++x) {
                const uint32_t d = tab.desc[k][x];
                if ((d >> 31) && ((d >> 24) & 7u) == t && (d & 15u) == pp && __popc((d >> 16) & 0xFFu) < 4) u |= (d >> 16) & 0xFFu;
            }
            s_smallm[t][pp] = (uint8_t)u;
        }
    }
    __syncthreads();
    for (uint32_t i = tid; i < n_g; i += kPipeThreads) reinterpret_cast<uint8_t*>(s_occ32)[i] = a.occ[lo_s + i];
    __syncthreads();

    // chain-warp constants: one (profile, start) candidate per slot
    uint32_t cmask[K], klow[K], cprof[K];
    bool valid[K], reports[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const uint32_t d = tab.desc[k][lane];
        valid[k] = d >> 31;
        cprof[k] = d & 15u;
        cmask[k] = valid[k] ? ((d >> 16) & 0xFFu) | (1u << (8 + ((d >> 24) & 7u))) : 0xFFFFu;   // slot mask + own-table bit
        klow[k] = (((d >> 4) & 7u) << 8) | (cmask[k] & 0xFFu);            // order-in-row and slot mask; t and profile come from the window key
        reports[k] = valid[k] && ((d >> 4) & 7u) == 0;
    }
    unsigned long long st_steps = 0, st_jumps = 0, st_visited = 0, st_sims = 0, st_rounds_sum = 0, st_cells = 0, spec_steps = 0, spec_visited = 0;

    // The queues of a chunk (k_partition wrote them before this kernel started) are copied into shared memory with cp.async
    // while the segment still waits for the chunk's token: they do not depend on the heads, so nothing is staged on the
    // critical path between 'token in' and the first decision.  Offset -> thread mapping is the same for every chunk, so a
    // thread's own wait_group orders its copies of consecutive chunks.
    auto queue_load_async = [&](uint32_t chunk) {
        const char* src = reinterpret_cast<const char*>(a.q_all + (size_t)chunk * a.q_stride);
        const uint32_t bytes = (a.cctl[chunk].qoff[ISL_MAX_PROFILES] * 2u + 15u) & ~15u;
        for (uint32_t off = tid * 16u; off < bytes; off += kPipeThreads * 16u)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa_q + off), "l"(src + off) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // fed streams: the requests of a batch may still be on their way (H2D + pre-pass on the feed stream) when the pipeline gets there.
    // Returns true when the stream ends in front of this chunk (an open stream was closed, or the host aborted a feed).
    // Causal window: chunk c additionally waits until every segment has committed chunk c - window.
    auto wait_ready = [&](uint32_t chunk) -> bool {
        if (!a.ready && !a.window) return false;
        const bool gate_ring = a.ring_done && !a.inbox;          // ranks behind the owner are gated by the token itself
        if (tid == 0) {
            uint32_t closed = 0;
            const unsigned long long t0 = globaltimer_ns();
            if (a.ready) {
                const uint32_t* f = a.ready + (a.open ? chunk : a.chunks[chunk].batch);
                // the feed kernels are launched AFTER this one; a tool that serialises kernels would starve the wait (the host side switches
                // feeding off when it detects one, ISL_NO_FEED=1 forces it) — fail loudly instead of hanging the GPU
                while (true) {
                    const uint32_t v = ld_acquire_gpu(f);
                    if (v == a.epoch) break;
                    if (v == ~a.epoch) { closed = 1; break; }
                    __nanosleep(128);
                    if (globaltimer_ns() - t0 > a.wait_ns) __trap();
                }
            }
            if (!closed && a.window && chunk >= a.window) {
                if (gate_ring) while (ld_acquire_sys(a.ring_done + chunk - a.window) < a.world) { __nanosleep(64); if (globaltimer_ns() - t0 > a.wait_ns) __trap(); }
                else if (!a.ring_done) while (ld_acquire_gpu(a.done_cnt + chunk - a.window) < a.n_seg) { __nanosleep(64); if (globaltimer_ns() - t0 > a.wait_ns) __trap(); }
            }
            s_closed = closed;
        }
        __syncthreads();
        return s_closed != 0;
    };
    auto chunk_done = [&](uint32_t chunk) {     // after the barrier that ends the chunk's commit
        if (a.done_cnt && tid == 0) {
            if (a.ring_done) __threadfence_system(); else __threadfence();
            const uint32_t before = atomicAdd(a.done_cnt + chunk, 1u);
            if (a.ring_done && before + 1 == a.n_seg) atomicAdd_system(a.ring_done + chunk, 1u);     // this rank is through with the chunk
        }
    };
    bool closed = wait_ready(0);
    if (!closed) queue_load_async(0);

    for (uint32_t c = 0; c < a.n_chunks && !closed; ++c) {
        const ChunkDesc cd = a.chunks[c];
        const Ctrl* cc = a.cctl + c;
        if (cd.first_of_batch) {            // 1. frees of this batch inside my range: one byte per GPU
            const uint8_t* fa = a.free_acc + (size_t)cd.batch * a.free_stride + lo_s;
            for (uint32_t i = tid; i < n_g; i += kPipeThreads) {
                const uint32_t f = fa[i];
                if (f) atomicAnd(&s_occ32[i >> 2], ~(f << ((i & 3u) * 8u)));
            }
            __syncthreads();
        }
        const uint32_t active = cc->active;
        // A stage is walked sub-segment by sub-segment (one for inventories up to 148 x 512 GPUs): sweep, heads, windows, chain, commit per
        // sub-segment; the token is awaited in front of the first and published behind the last one (or as soon as nothing is pending).
        const uint32_t n_sub = max(1u, (n_g + a.sub - 1) / a.sub);
        bool prefetched = false;            // the next chunk's queues are on their way (they may only overwrite this chunk's after its last chain)
        for (uint32_t sb = 0; sb < n_sub; ++sb) {
        const uint32_t sb_base = sb * a.sub, n_sb = min(a.sub, n_g - min(n_g, sb_base));
        const bool last_sub = sb + 1 == n_sub;
        {   // 2. local sweep: thread t owns kSegMax / kPipeThreads consecutive local GPUs; ordered compaction
            constexpr uint32_t kGpt = kSegMax / kPipeThreads;
            uint32_t og[kGpt], tg[kGpt];
            bool fg[kGpt];
            // one scan carries both counts: candidates (low half) and free usable slices on the candidates (high half) — the latter
            // bounds what the segment can accept: a profile of span z pops at most free / z requests here
            uint32_t cnt = 0;
#pragma unroll
            for (uint32_t x = 0; x < kGpt; ++x) {
                const uint32_t g = kGpt * tid + x;
                og[x] = reinterpret_cast<const uint8_t*>(s_occ32)[sb_base + g]; tg[x] = s_tab[sb_base + g];
                fg[x] = g < n_sb && (s_feas[tg[x] * 256 + og[x]] & active);
                if (fg[x]) cnt += 1u | ((uint32_t)__popc(~og[x] & s_usable[tg[x]]) << 16);
            }
            uint32_t incl = cnt;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d); if ((int)lane >= d) incl += t; }
            if (lane == 31) s_warp[warp] = incl;
            __syncthreads();
            uint32_t off = incl - cnt;
            for (uint32_t x = 0; x < warp; ++x) off += s_warp[x];
            const uint32_t nfree = (off + cnt) >> 16;
            off &= 0xFFFFu;
#pragma unroll
            for (uint32_t x = 0; x < kGpt; ++x) if (fg[x]) s_cand[off++] = ((kGpt * tid + x) << 16) | table_tag(tg[x]) | og[x];
            if (tid == kPipeThreads - 1) { s_ncand = off; s_nfree = nfree; for (uint32_t x = 0; x < kCandPad; ++x) s_cand[off + x] = kInf; }   // sentinels: nothing fits
        }
        __syncthreads();                    // s_ncand / s_nfree of the sweep are visible to warp 0
        // 3. token of the previous segment
        unsigned long long* tr = a.trace ? a.trace + ((size_t)c * a.n_seg + seg) * kTraceWords : nullptr;
        const size_t tok_chunk = (size_t)c * (a.n_seg + 1);
        constexpr bool spec = kSpec;        // host: only with one sub-segment per stage (a.spec); a separate instantiation, so that the plain pipeline's code is untouched by the rounds' machinery
        const SpecMem sm = spec_mem(a.spec_mem, spec ? c : 0);
        // a partitioned inventory tags with the stream id all ranks share
        const uint32_t tage = a.spec_world > 1 ? a.xepoch : a.epoch;
        const unsigned long long tagb = (unsigned long long)((tage & 0xFFFFFFu) << 8) << 32, tagF = tagb | (0xFFull << 32);
        const bool xr = a.spec_world > 1;                                  // records cross ranks
        const uint32_t gseg = a.spec_base + seg, gtot = a.spec_total;      // my place in the sequence of all stages of all ranks
        auto sld = [&](const unsigned long long* p) { return xr ? ld_relaxed_sys_u64(p) : ld_relaxed_gpu_u64(p); };
        // a word every LATER stage reads: my copy and the copies of the ranks behind me
        auto pub_down = [&](unsigned long long* p, unsigned long long v) {
            st_relaxed_gpu_u64(p, v);
            if (xr) for (uint32_t r = a.spec_rank + 1; r < a.spec_world; ++r) st_relaxed_sys_u64(a.spec_peer[r] + (p - a.spec_mem), v);
        };
        // a word only the next (prev = false) / the previous (prev = true) stage reads
        auto pub_nb = [&](unsigned long long* p, unsigned long long v, bool prev) {
            const bool remote = xr && (prev ? (seg == 0 && a.spec_rank > 0) : (seg + 1 == a.n_seg && a.spec_rank + 1 < a.spec_world));
            if (remote) st_relaxed_sys_u64(a.spec_peer[prev ? a.spec_rank - 1 : a.spec_rank + 1] + (p - a.spec_mem), v);
            else st_relaxed_gpu_u64(p, v);
        };
        if (spec) {     // round 0: what this stage's occupancy can take, per contention group -> predicted entry heads
            uint16_t* s_mj = reinterpret_cast<uint16_t*>(s_wkey);               // scratch (the windows are staged later): [3][kSpecStride] gathered masses of the stages in front
            if (tid < ISL_MAX_PROFILES) {
                const bool on = ((active >> tid) & 1u) && s_maxacc[tid] != 0 && cc->qcnt[tid] != 0;
                s_qc[tid] = on ? cc->qcnt[tid] : 0u; s_qo[tid] = cc->qoff[tid];
                const uint32_t big = __ballot_sync(0xFFFFu, on && s_minsize[tid] >= 4), small = __ballot_sync(0xFFFFu, on && s_minsize[tid] < 4);
                if (tid == 0) { s_grp_big = big; s_grp_small = small; s_acc[0] = 0; s_acc[1] = 0; s_acc[2] = 0; }
                if (tid < kMaxTables) { uint32_t us = 0; for (uint32_t m = small; m; m &= m - 1) us |= s_smallm[tid][__ffs(m) - 1]; s_us[tid] = us; }   // slices the small group can use, per table
            }
            __syncthreads();
            {   // per GPU: the big group takes the widest span that still fits, twice at most (two quads); the small group fills the usable rest
                constexpr uint32_t kGpt = kSegMax / kPipeThreads;
                const uint32_t gb = s_grp_big, nb = s_nbigd;
                uint32_t mq = 0, mw = 0, mo = 0;
#pragma unroll
                for (uint32_t x = 0; x < kGpt; ++x) {
                    const uint32_t g = kGpt * tid + x;
                    if (g < n_sb) {
                        const uint32_t t = s_tab[sb_base + g], o0 = reinterpret_cast<const uint8_t*>(s_occ32)[sb_base + g], us = s_us[t];
                        uint32_t o = o0;
                        for (uint32_t it = 0; it < 2; ++it) {
                            uint32_t best = 0;
                            for (uint32_t y = 0; y < nb; ++y) {
                                const uint32_t d = s_bigd[y], mk = (d >> 16) & 0xFFu;
                                if (((d >> 24) & 7u) == t && ((gb >> (d & 15u)) & 1u) && (o & mk) == 0 && __popc(mk) > __popc(best)) best = mk;
                            }
                            if (!best) break;
                            o |= best; ++mq;
                        }
                        mw += __popc(~o & us); mo += __popc(~o0 & us);
                    }
                }
                mq = __reduce_add_sync(0xFFFFFFFFu, mq); mw = __reduce_add_sync(0xFFFFFFFFu, mw); mo = __reduce_add_sync(0xFFFFFFFFu, mo);
                if (lane == 0) { atomicAdd(&s_acc[0], mq); atomicAdd(&s_acc[1], mw); atomicAdd(&s_acc[2], mo); }
            }
            __syncthreads();
            if (tid == 0) {
                pub_down(sm.m + gseg * 2, tagb | s_acc[0]);
                pub_down(sm.m + gseg * 2 + 1, tagb | (min(s_acc[1], 0xFFFFu) << 16) | min(s_acc[2], 0xFFFFu));
            }
            if (tid < gseg) {       // masses of every stage in front of this one
                const unsigned long long t0 = globaltimer_ns();
                unsigned long long w0, w1;
                uint32_t spins = 0;
                while (true) {
                    w0 = sld(sm.m + tid * 2); w1 = sld(sm.m + tid * 2 + 1);
                    if ((w0 >> 32) == (tagb >> 32) && (w1 >> 32) == (tagb >> 32)) break;
                    if ((++spins & 255u) == 0 && globaltimer_ns() - t0 > a.wait_ns) __trap();
                }
                s_mj[tid] = (uint16_t)w0; s_mj[kSpecStride + tid] = (uint16_t)(w1 >> 16); s_mj[2 * kSpecStride + tid] = (uint16_t)w1;
            }
            __syncthreads();
            if (tid < 32) {         // the big group takes its placements until its queues run dry; the small group fills what is left
                uint32_t totb = 0, tots = 0;
                for (uint32_t m = s_grp_big; m; m &= m - 1) totb += s_qc[__ffs(m) - 1];
                for (uint32_t m = s_grp_small; m; m &= m - 1) { const uint32_t pp = __ffs(m) - 1; tots += s_qc[pp] * s_minsize[pp]; }
                constexpr uint32_t kPer = (kSpecStride + 31) / 32;
                uint32_t ql = 0;
                for (uint32_t x = 0; x < kPer; ++x) { const uint32_t j = lane * kPer + x; if (j < gseg) ql += s_mj[j]; }
                uint32_t incl = ql;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d); if ((int)lane >= d) incl += t; }
                uint32_t run = incl - ql, r = 0;
                for (uint32_t x = 0; x < kPer; ++x) {
                    const uint32_t j = lane * kPer + x;
                    if (j < gseg) { r += run < totb ? s_mj[kSpecStride + j] : s_mj[2 * kSpecStride + j]; run += s_mj[j]; }
                }
                r = __reduce_add_sync(0xFFFFFFFFu, r);
                const uint32_t Q = min(__shfl_sync(0xFFFFFFFFu, incl, 31), totb), R = min(r, tots);
                {
                    const uint32_t qcl = lane < ISL_MAX_PROFILES ? s_qc[lane] : 0u, wl = lane < ISL_MAX_PROFILES ? s_minsize[lane] : 1u;
                    uint32_t hg = lane < ISL_MAX_PROFILES && gseg == 0 && a.heads_in ? a.heads_in[(size_t)c * ISL_MAX_PROFILES + lane] : 0u;
                    if (gseg > 0) {
                        hg = spec_spread_warp(hg, qcl, wl, s_grp_big, (int)Q, false, lane);
                        hg = spec_spread_warp(hg, qcl, wl, s_grp_small, (int)R, true, lane);
                    }
                    if (lane < ISL_MAX_PROFILES) s_specH[lane] = hg;
                }
            }
            __syncthreads();
        }
        uint32_t rnd = 1;
        bool c_prev = spec ? gseg == 0 : seg == 0, need_sim = true, idle_break = false;
        bool known_exact = gseg == 0;       // everything in front of the stage right in front of me was consistent one round ago: my next entry may be the true one
        if (tid == 0) { s_capst[0] = 0; s_capst[1] = 0; s_capst[2] = 0; s_cap = kLogCap + 1; s_capped = 0; s_wvalid = 0; s_havepred = 0; }
        bool p_final = false; unsigned long long p_word = 0;      // pollers: a certified stage's final record is read once and kept
        const unsigned long long t_cell = tr && spec ? globaltimer_ns() : 0ull, sims_cell = st_sims;   // spec trace: [0] sweep + prediction done, [2] certified, [7] simulations, [11] rounds
#ifdef ISL_SPEC_DBG_STAMPS      // per-round stamps of one cell (tools/spec_trace.py): a debugging build — the extra live pointer around the decision loop costs ~14 %
        unsigned long long* dbg = a.spec_dbg && a.spec_dbg_cell == ((c << 16) | seg) ? a.spec_dbg : nullptr;
#else
        constexpr unsigned long long* dbg = nullptr;
#endif
        while (true) {      // one pass unless the stage speculates
        stamp_if(dbg && tid == 0, dbg + rnd * 8 + 0);
        if (need_sim) {
        // Inside a GPU a token is self-validating: every head word carries the call's 15-bit epoch tag above its 17 bits of payload
        // (heads <= 65 536), so there is no separate flag, no fence on the producer side and no second round trip on this side —
        // lanes 0..15 of warp 0 each poll their own word of the previous segment's token or of the chunk's 'done' record (whichever
        // is valid first: when both are, they hold the same heads).  Across GPUs (inbox) the flag + system-scope release stays.
        asm volatile("cp.async.wait_group 0;" ::: "memory");       // my share of the chunk's queues has landed (long ago, as a rule)
        if (tid < 32) {     // heads, window sizes and the compact window layout (exclusive scan over the 16 profiles)
            uint32_t h = 0, wn = 0, left = 0;
            bool from_done = false;
            const uint32_t tag = a.epoch & 0x7FFFu;
            stamp_if(tr && tid == 0, tr + 0);
            if (spec) {                 // the predicted (or, at stage 0, the true) token
                if (tid < ISL_MAX_PROFILES) h = s_specH[tid];
            } else if (sb > 0) {        // behind the first sub-segment the heads are the ones its chain left
                if (tid < ISL_MAX_PROFILES) h = s_heads[tid] + s_pop[tid];
            } else if (seg > 0) {
                const uint32_t* pt = a.tokens + (tok_chunk + seg - 1) * kTokStride + (tid & 15u);
                const uint32_t* pd = a.tokens + (tok_chunk + a.n_seg) * kTokStride + (tid & 15u);
                bool ok = tid >= ISL_MAX_PROFILES;
                while (!__all_sync(0xFFFFFFFFu, ok)) {
                    if (!ok) {
                        uint32_t v = ld_relaxed_gpu(pt);
                        if ((v >> 17) == tag) { h = v & 0x1FFFFu; ok = true; }
                        else { v = ld_relaxed_gpu(pd); if ((v >> 17) == tag) { h = v & 0x1FFFFu; ok = true; from_done = true; } }
                    }
                }
            } else if (a.inbox) {       // first segment of a rank that has a predecessor: the token comes over NVLink
                // Self-validating words across GPUs as well: every head word carries the low 15 bits of the stream id above its 17 bits of
                // payload, written with ONE relaxed system-scope store each (4-byte stores are single-copy atomic) — no fence and no flag on
                // the sender's side, one NVLink write latency per hop instead of fence + flag.  The consumer clears its slot after reading,
                // so a tag can never be mistaken for one of 32 768 streams ago.  A dead or stuck predecessor must not hang this GPU for
                // good: the wait traps like wait_ready does.
                uint32_t* slot = const_cast<uint32_t*>(a.inbox) + (size_t)c * kTokStride + (tid & 15u);
                const uint32_t xtag = a.xepoch % 32767u + 1u;      // never 0: a cleared slot is never valid
                bool ok = tid >= ISL_MAX_PROFILES;
                const unsigned long long t0 = globaltimer_ns();
                while (!__all_sync(0xFFFFFFFFu, ok)) {
                    if (!ok) {
                        const uint32_t v = ld_relaxed_sys(slot);
                        if ((v >> 17) == xtag) { h = v & 0x1FFFFu; ok = true; }
                        else if (globaltimer_ns() - t0 > a.wait_ns) __trap();
                    }
                }
                if (tid < ISL_MAX_PROFILES) st_relaxed_sys(slot, 0u);
            } else if (tid < ISL_MAX_PROFILES) h = a.heads_in ? a.heads_in[(size_t)c * ISL_MAX_PROFILES + tid] : 0u;
            stamp_if(tr && tid == 0, tr + 1);
            const bool all_done = sb == 0 && __all_sync(0xFFFFFFFFu, from_done || tid >= ISL_MAX_PROFILES);
            if (tid < ISL_MAX_PROFILES) {
                const uint32_t qc = spec ? s_qc[tid] : cc->qcnt[tid], qo = spec ? s_qo[tid] : cc->qoff[tid];     // re-simulations: no trip to L2
                left = ((active >> tid) & 1u) && qc > h ? qc - h : 0u;
                wn = min(left, min(s_ncand * s_maxacc[tid], s_nfree / s_minsize[tid]));   // no more pops than that are possible here
                s_heads[tid] = h; s_pop[tid] = 0;
                if (!kSpec) {
                    s_wn[tid] = wn;
                    s_qbeg[tid] = qo + h;                                       // first pending entry in the shared copy of the queues
                }
            }
            bool win_keep = true;
            if (kSpec) {
                // A corrected entry usually sits a few requests from the one simulated before: the windows are staged with kWinMargin entries on
                // either side and stay for the next simulation when every profile's new window [h, h + wn + 2) lies inside what is staged (real
                // keys behind the first wn entries are as good as the INF sentinels there: capacity, not the window, ends a profile's pops)
                uint32_t lo = 0, len = 0, woff = 0;
                bool ok = true;
                const uint32_t qc = tid < ISL_MAX_PROFILES ? s_qc[tid] : 0u;
                if (tid < ISL_MAX_PROFILES) {
                    lo = s_wlo[tid]; len = s_wlen[tid];
                    if (left == 0) woff = len;                                  // nothing pending: straight onto the sentinels
                    else { ok = s_wvalid && h >= lo && (h + wn + 2 <= lo + len || lo + len >= qc); woff = h - lo; }
                }
                const bool keep = __all_sync(0xFFFFFFFFu, ok) && !(a.spec & 2u);      // (bit 1 of PipeArgs.spec: stage anew every time — a debugging switch, ISL_SPEC_NOREUSE)
                if (!keep && tid < ISL_MAX_PROFILES) {
                    if (left == 0) { lo = h; len = 0; woff = 0; }
                    else { lo = h - min(h, kWinMargin); len = min(qc - lo, (h - lo) + wn + kWinMargin + 2); woff = h - lo; }
                    s_wlo[tid] = lo; s_wlen[tid] = len;
                    s_qbeg[tid] = s_qo[tid] + lo;
                }
                if (tid < ISL_MAX_PROFILES) { s_woff[tid] = woff; s_wn[tid] = len - woff; }     // real entries from the entry to the staged end
                win_keep = keep;
                wn = len;                                                       // the layout below counts the staged entries
            }
            // nothing placeable is pending any more: tell every later segment at once instead of relaying hop by hop
            const bool idle = __ballot_sync(0xFFFFFFFFu, left != 0) == 0;
            if (idle && !all_done && !spec && tid < ISL_MAX_PROFILES) st_relaxed_gpu(a.tokens + (tok_chunk + a.n_seg) * kTokStride + tid, (tag << 17) | h);
            if (tid == 0) {
                s_idle = idle ? 1u : 0u;
                if (kSpec) {        // an idle simulation stages nothing: a new layout that was never filled must not be kept by the next one
                    s_restage = win_keep ? 0u : 1u;
                    if (!win_keep) s_wvalid = idle ? 0u : 1u;
                }
                // A speculative simulation from an entry that is far off can run several times longer than the segment's true work (everything the
                // stages in front are wrongly believed to have left over lands here) and would hold up the whole round.  Unless the entry is known
                // to be the true one, the simulation is cut off at 1.3 x the largest complete one so far; a cut-off round publishes the exit
                // extrapolated from the last complete simulation instead (what the stages behind would assume anyway).
                s_cap = spec && s_capst[1] && !known_exact ? min(kLogCap + 1, ((s_capst[0] * 21u) >> 4) + 64u) : kLogCap + 1;
                s_capped = 0;
            }
            uint32_t incl = wn + kWinPad;                       // INF sentinels close every window
#pragma unroll
            for (int d = 1; d < 16; d <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d); if ((int)lane >= d) incl += t; }
            if (tid < ISL_MAX_PROFILES) s_wbase[tid] = incl - (wn + kWinPad);
        }
        __syncthreads();
        stamp_if(tr && tid == 0, tr + 8);
        stamp_if(dbg && tid == 0, dbg + rnd * 8 + 1);
        if (s_idle && spec) { if (tid == 0) { s_nlog = 0; spec_steps = 0; spec_visited = 0; } }      // nothing pending at these heads: the exit equals the entry
        else if (s_idle) {  // pass-through: the token (unchanged heads) still reaches the next rank / the caller from the last segment
            if (warp == 0) {
                const bool last = seg == a.n_seg - 1;
                uint32_t* tok = a.tokens + (tok_chunk + seg) * kTokStride;
                uint32_t* peer = last && a.outbox ? a.outbox + (size_t)c * kTokStride : nullptr;
                if (lane < ISL_MAX_PROFILES) {
                    const uint32_t h = s_heads[lane];
                    st_relaxed_gpu(tok + lane, ((a.epoch & 0x7FFFu) << 17) | h);
                    if (last && a.heads_out) a.heads_out[(size_t)c * ISL_MAX_PROFILES + lane] = h;
                    if (peer) st_relaxed_sys(peer + lane, ((a.xepoch % 32767u + 1u) << 17) | h);
                }
                __syncwarp();
                if (lane == 0) {
                    if (tr) { tr[2] = globaltimer_ns(); tr[3] = tr[2]; }
                }
            }
            __syncthreads();
            idle_break = true;
            break;              // the remaining sub-segments have nothing to take either
        }
        if (!s_idle) {
        {   // windows of ready-made keys t << 15 | profile << 11, each closed by two INF sentinels — converted from the shared copy of
            // the queues (a shared-memory round trip per round instead of an L2 one), only for profiles that own candidates
            const uint32_t npl = kSpec && !s_restage ? 0u : s_nplist;
            const uint16_t* __restrict__ sq = reinterpret_cast<const uint16_t*>(smem + kPipeOffQ);
            for (uint32_t x = 0; x < npl; ++x) {
                const uint32_t p = s_plist[x], wn = kSpec ? s_wlen[p] : s_wn[p], pk = p << 11, qb = s_qbeg[p];
                uint32_t* __restrict__ dst = s_wkey + s_wbase[p];
                // plain, unconditional (clamped) accesses: the loads of a round overlap instead of queueing behind each other
                for (uint32_t i = tid; i < wn + kWinPad; i += kPipeThreads) { const uint32_t v = sq[qb + min(i, wn)]; dst[i] = i < wn ? (v << 15) | pk : kInf; }
            }
            stamp_if(tr && tid == 0, tr + 10);
            store_if(tr && tid == 0, tr + 11, s_wn[s_plist[0]] | ((unsigned long long)s_nfree << 32));
        }
        __syncthreads();
        stamp_if(tr && tid == 0, tr + 9);
        if (is_chain_warp(warp)) {          // 4. the decision chain (see k_chain), tuned for the shortest loop-carried path
            const uint32_t n_cand = s_ncand;
            uint32_t tcur[K], tnext[K], tnn[K], wa[K], wa0[K];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                wa0[k] = sa_wkey + 4 * (s_wbase[cprof[k]] + (kSpec ? s_woff[cprof[k]] : 0u));
                const bool has = valid[k];
                tcur[k] = has ? lds_u32(wa0[k]) | klow[k] : kInf;               // INF | anything = INF
                tnext[k] = has ? lds_u32(wa0[k] + 4) | klow[k] : kInf;
                const bool two = has && s_wn[cprof[k]] >= 1;                    // a third entry exists only behind >= 1 real one
                tnn[k] = two ? lds_u32(wa0[k] + 8) : kInf;
                wa[k] = wa0[k] + 12;                                            // next entry to load on a pop
            }
            uint32_t la = sa_log, ca = sa_cand + 8;                             // ca: shared address of candidate record (current + 2)
            // Per slot the loop carries conflict words z = occupancy & candidate mask of the current / next / next-but-one candidate GPU
            // and g = "fits on that GPU ? sel bit : nothing" as a ready OR mask; the key of the NEXT decision is formed at the end of the
            // body.  Loop-carried path behind the redux: sign mask of `sel` -> bitwise mux of z -> fold the winner's slices in and test
            // (one LOP3 with a predicate output) -> pick the key: four ALU levels (a freshly updated occupancy register tested through
            // ISETP / SEL needs five; measured 41 -> 35 ns per decision, and ISETP + SEL behind the redux costs ~10 cycles more than
            // shift + LOP3 mux: tools/microbench_pred.cu).
            // The updates are issued unconditionally and the "nothing fits" test comes LAST: a branch is not speculated, so a test in
            // front of the updates would put its resolution on the loop-carried path of every decision.  m == INF behaves like a decision
            // that lands on the next GPU and pops only exhausted lanes (no real key has all-ones t / profile fields unless profile 15
            // is in use, kP15); the rare path rewinds the cursors and reloads the conflict words after the jump.
            uint32_t z0[K], z1[K], z2[K], g1[K], g2[K], cm8[K];
            auto reload_z = [&]() {
                const uint32_t a0 = lds_u16(ca - 8), a1 = lds_u16(ca - 4), a2 = lds_u16(ca);
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    z0[k] = a0 & cmask[k]; z1[k] = a1 & cmask[k]; z2[k] = a2 & cmask[k];
                    g1[k] = z1[k] == 0 ? 0x80000000u : kInf; g2[k] = z2[k] == 0 ? 0x80000000u : kInf;
                }
            };
#pragma unroll
            for (int k = 0; k < K; ++k) cm8[k] = cmask[k] & 0xFFu;
            reload_z();
            uint32_t key = kInf, a2 = lds_u16(ca);
            auto first_key = [&]() {
                key = kInf;
#pragma unroll
                for (int k = 0; k < K; ++k) key = min(key, z0[k] == 0 ? tcur[k] : (tcur[k] | g1[k]));
            };
            first_key();
            const unsigned long long jumps0 = st_jumps;
            // (trace stamps next to the decision loop perturb its schedule in the instantiation with the rounds — measured 9 % of a round; that
            // instantiation records its cell at certification instead)
            if (!kSpec) stamp_if(tr && lane == 0, tr + 4);
            stamp_if(dbg && lane == 0, dbg + rnd * 8 + 2);
            constexpr bool kDefer = ISL_DEFER_INF && !kP15;     // see the rare path below
            const uint32_t la_cap = sa_log + 8u * s_cap;
            bool cut = false;
            while (true) {
                if (!kDefer && la >= la_cap) { cut = true; break; }     // once per group of decisions, off the loop-carried path
                bool none = false;
                uint32_t m = 0, mmax = 0;
#pragma unroll
                for (int u = 0; u < kUnroll; ++u) {     // unrolled: one taken branch per kUnroll decisions
                    m = redux_min_u32(key);
#pragma unroll
                    for (int k = 0; k < K; ++k) {       // in the shadow of the redux: the record fetched by the previous decision (the same one again if it did not advance)
                        z2[k] = a2 & cmask[k];
                        g2[k] = z2[k] == 0 ? 0x80000000u : kInf;
                    }
                    if (kP15) { none = m == kInf; if (none) break; }
                    uint32_t ks;
                    asm("shr.s32 %0, %1, 31;" : "=r"(ks) : "r"(m));                                            // all ones: landed on the next GPU
                    asm("mad.lo.s32 %0, %1, -4, %0;" : "+r"(ca) : "r"(ks));                                     // ca += sel * 4
                    if (kDefer) {       // a pseudo-decision (m == INF: nothing fits here or on the next GPU, move on by one) leaves no log record
                        const bool real = m != kInf;
                        sts_v2_if(lane == 0 && real, la, m, ca);
                        la = add_if(real, la, 8u);
                        mmax = max(mmax, m);
                    } else {
                        sts_v2_if(lane == 0, la, m, ca);                // decision log: (key, address of the record two past the GPU it landed on)
                        la += 8;
                    }
                    a2 = lds_u16(ca);
                    key = kInf;
#pragma unroll
                    for (int k = 0; k < K; ++k) {
                        const bool adv = kP15 ? (((m & 0x7FFFF800u) ^ tcur[k]) & 0xFFFFF800u) == 0 : ((m ^ tcur[k]) & 0x7FFFF800u) == 0;
                        const uint32_t tn = adv ? tnext[k] : tcur[k];
                        uint32_t zs, gn, kk;
                        asm("lop3.b32 %0, %1, %2, %3, 0xca;" : "=r"(zs) : "r"(ks), "r"(z1[k]), "r"(z0[k]));       // sel ? z1 : z0
                        asm("lop3.b32 %0, %1, %2, %3, 0xca;" : "=r"(gn) : "r"(ks), "r"(g2[k]), "r"(g1[k]));       // sel ? g2 : g1
                        asm("{ .reg .pred p; .reg .b32 t; lop3.b32 t, %1, %2, %3, 0xF8; setp.eq.u32 p, t, 0; selp.b32 %0, %4, %5, p; }"
                            : "=r"(kk) : "r"(zs), "r"(m), "r"(cm8[k]), "r"(tn), "r"(tn | gn));
                        key = min(key, kk);
                        z0[k] = zs | (m & cm8[k]);
                        g1[k] = gn;
                        asm("lop3.b32 %0, %1, %2, %3, 0xca;" : "=r"(z1[k]) : "r"(ks), "r"(z2[k]), "r"(z1[k]));    // sel ? z2 : z1
                        tcur[k] = tn;
                        tnext[k] = adv ? (tnn[k] | klow[k]) : tnext[k];
                        tnn[k] = lds_u32_if(adv, wa[k], tnn[k]);        // consumed at the earliest one pop later
                        wa[k] = add_if(adv, wa[k], 4u);
                    }
                    if (!kP15 && !kDefer) {
                        none = m == kInf;
                        if (__builtin_expect(none, 0)) {
                            ca -= 4; la -= 8;                           // rewind the pseudo-decision
#pragma unroll
                            for (int k = 0; k < K; ++k)
                                if (tcur[k] == kInf) { tnext[k] = kInf; wa[k] -= 4; }
                            break;
                        }
                    }
                }
                uint32_t from = (ca - sa_cand) >> 2;        // record index of (current + 2)
                if (kDefer) {
                    // m == INF is a legitimate step of the recurrence ("neither this GPU nor the next takes anything: the next one becomes
                    // current"; it pops only lanes whose window is exhausted, into their INF sentinels), so the loop body needs no exit
                    // test per decision — one test per group: did ANY decision of the group find nothing?
                    if (__builtin_expect(mmax != kInf && la < la_cap, 1)) continue;     // (the cut-off test rides on the group's one branch)
                    if (la >= la_cap) { cut = true; break; }
                    // exhausted lanes were popped past the end of their windows: back onto the sentinels (at most kUnroll pops since the last time)
#pragma unroll
                    for (int k = 0; k < K; ++k)
                        if (tcur[k] == kInf) { tnext[k] = kInf; tnn[k] = kInf; wa[k] = wa0[k] + 12 + 4 * s_wn[cprof[k]]; }
                    if (m != kInf) continue;                // the group ended on a real decision: carry on
                    from -= 1;                              // the pseudo-decision already moved on by one GPU: the new 'next' is still unexamined
                } else if (__builtin_expect(!none, 1)) continue;
                uint32_t alive = 0;
#pragma unroll
                for (int k = 0; k < K; ++k) alive |= tcur[k] != kInf ? 1u << cprof[k] : 0u;
                const uint32_t j = pipeline_skip(sa_cand, s_feas, n_cand, from, alive, lane);
                ++st_jumps;
                if (j == kInf) break;
                ca = sa_cand + 4 * (j + 2);
                reload_z();
                a2 = lds_u16(ca);
                first_key();
            }
            const uint32_t nlog = (la - sa_log) >> 3;
            if (!kSpec) {
            stamp_if(tr && lane == 0, tr + 5);
            stamp_if(dbg && lane == 0, dbg + rnd * 8 + 3);
            store_if(tr && lane == 0, tr + 6, nlog);
            store_if(tr && lane == 0, tr + 7, (st_jumps - jumps0) | ((unsigned long long)(((ca - sa_cand) >> 2) - 2) << 32));
            }
            if (!spec) { st_steps += nlog; st_visited += ((ca - sa_cand) >> 2) - 2; }
            else { spec_steps = nlog; spec_visited = ((ca - sa_cand) >> 2) - 2; ++st_sims; }
#pragma unroll
            for (int k = 0; k < K; ++k) if (reports[k]) s_pop[cprof[k]] = min((wa[k] - wa0[k] - 12) >> 2, s_wn[cprof[k]]);
            __syncwarp();
            // 5. token for the next segment: heads first, then the flag (release) — behind the stage's last sub-segment
            uint32_t* tok = a.tokens + (tok_chunk + seg) * kTokStride;
            const bool last = seg == a.n_seg - 1;
            uint32_t* peer = last && a.outbox ? a.outbox + (size_t)c * kTokStride : nullptr;
            if (last_sub && lane < ISL_MAX_PROFILES && !spec) {
                const uint32_t h = s_heads[lane] + s_pop[lane];
                st_relaxed_gpu(tok + lane, ((a.epoch & 0x7FFFu) << 17) | h);       // the next segment starts
                if (last && a.heads_out) a.heads_out[(size_t)c * ISL_MAX_PROFILES + lane] = h;
                if (peer) st_relaxed_sys(peer + lane, ((a.xepoch % 32767u + 1u) << 17) | h);
            }
            __syncwarp();
            if (lane == 0) {
                s_nlog = nlog;
                s_capped = cut ? 1u : 0u;
                if (tr) tr[2] = globaltimer_ns();
            }
        }
        else if (spec && tid == kPipeThreads - 32 && rnd >= 3 && gseg + 1 < gtot) {
            // in the shadow of the chain: the slot of round rnd - 2 is about to be overwritten — the successor must have read it (it has, as a rule)
            const unsigned long long t0 = globaltimer_ns();
            uint32_t spins = 0;
            while (true) {
                const unsigned long long w = sld(sm.ack + gseg + 1);
                if ((uint32_t)(w >> 32) == tage && (uint32_t)w + 2u >= rnd) break;
                if ((++spins & 255u) == 0 && globaltimer_ns() - t0 > a.wait_ns) __trap();
            }
        }
        }   // !s_idle
        __syncthreads();
        }   // need_sim
        if (!spec) break;
        {   // ---- the round's exchange: publish exit heads and consumed masses, read the predecessor's exit and every earlier stage's masses
            const unsigned long long tagr = tagb | ((unsigned long long)rnd << 32);
            if (tid < 32) {
                uint32_t X = 0, dq = 0, dr = 0, pop = 0;
                const bool was_cut = s_capped != 0;
                if (tid < ISL_MAX_PROFILES) { pop = s_pop[tid]; X = s_heads[tid] + pop; }
                if (was_cut) {      // exit of the last complete simulation, moved by what the entry has moved since (per group, shares as always)
                    int eq = 0, er = 0;
                    uint32_t xe = 0;
                    const uint32_t qcl = tid < ISL_MAX_PROFILES ? s_qc[tid] : 0u, wl = tid < ISL_MAX_PROFILES ? s_minsize[tid] : 1u;
                    if (tid < ISL_MAX_PROFILES) {
                        const int d = (int)s_heads[tid] - (int)s_Hc[tid];
                        if ((s_grp_big >> tid) & 1u) eq = d;
                        if ((s_grp_small >> tid) & 1u) er = d * (int)s_minsize[tid];
                        xe = s_Xc[tid];
                    }
                    eq = __reduce_add_sync(0xFFFFFFFFu, eq); er = __reduce_add_sync(0xFFFFFFFFu, er);
                    xe = spec_spread_warp(xe, qcl, wl, s_grp_big, eq, false, lane);
                    xe = spec_spread_warp(xe, qcl, wl, s_grp_small, er, true, lane);
                    if (tid < ISL_MAX_PROFILES) { X = max(xe, s_heads[tid]); pop = X - s_heads[tid]; }
                }
                if (tid < ISL_MAX_PROFILES) {
                    s_specX[tid] = X;
                    if (!was_cut) { s_Hc[tid] = s_heads[tid]; s_Xc[tid] = X; }
                    if ((s_grp_big >> tid) & 1u) dq = pop;
                    if ((s_grp_small >> tid) & 1u) dr = pop * s_minsize[tid];
                }
                if (tid == 0) { if (was_cut) s_capst[2] = 0; else { s_capst[0] = max(s_capst[0], s_nlog); s_capst[1] = 1; s_capst[2] = 1; } }
                dq = __reduce_add_sync(0xFFFFFFFFu, dq); dr = __reduce_add_sync(0xFFFFFFFFu, dr);
                if (rnd >= 3 && gseg + 1 < gtot && !(need_sim && !s_idle)) {      // the slot of round rnd - 2 is overwritten: the successor must have read it (checked behind the chain when one ran)
                    const unsigned long long t0 = globaltimer_ns();
                    uint32_t spins = 0;
                    while (true) {
                        const unsigned long long w = sld(sm.ack + gseg + 1);
                        if ((uint32_t)(w >> 32) == tage && (uint32_t)w + 2u >= rnd) break;
                        if ((++spins & 255u) == 0 && globaltimer_ns() - t0 > a.wait_ns) __trap();
                    }
                }
                if (tid < ISL_MAX_PROFILES) pub_nb(sm.x + ((size_t)gseg * 2 + (rnd & 1u)) * 16 + tid, tagr | X, false);
                if (tid == 16) pub_down(sm.d + (size_t)rnd * kSpecStride + gseg, tagr | ((c_prev ? 1u : 0u) << 31) | (dq << 13) | dr);
                if (tid == 0) { s_dqr[0] = dq; s_dqr[1] = dr; s_acc[0] = 0; s_acc[1] = 0; }
                stamp_if(dbg && tid == 0, dbg + rnd * 8 + 4);
            }
            __syncthreads();
            bool cbit = true;
            if (tid < gseg) {
                unsigned long long w = p_word;
                if (!p_final) {
                    const unsigned long long t0 = globaltimer_ns();
                    uint32_t spins = 0;
                    while (true) {
                        w = sld(sm.d + (size_t)rnd * kSpecStride + tid);
                        if ((w >> 32) == (tagr >> 32)) { cbit = (w >> 31) & 1u; break; }
                        if ((spins++ & 3u) == 0) {      // a certified stage no longer publishes rounds: its final record stands for every round from then on
                            w = sld(sm.df + tid);
                            if ((w >> 32) == (tagF >> 32) && ((w >> 24) & 0xFFu) <= rnd) { p_final = true; p_word = w; break; }
                        }
                        if ((spins & 255u) == 0 && globaltimer_ns() - t0 > a.wait_ns) __trap();
                    }
                }
                atomicAdd(&s_acc[0], (uint32_t)(w >> 13) & 0x7FFu);
                atomicAdd(&s_acc[1], (uint32_t)w & 0x1FFFu);
            }
            if (gseg > 0 && tid >= 192 && tid < 192 + ISL_MAX_PROFILES) {
                const uint32_t i = tid - 192;
                unsigned long long w = p_word;
                if (!p_final) {
                    const unsigned long long t0 = globaltimer_ns();
                    uint32_t spins = 0;
                    while (true) {
                        w = sld(sm.x + ((size_t)(gseg - 1) * 2 + (rnd & 1u)) * 16 + i);
                        if ((w >> 32) == (tagr >> 32)) break;
                        if ((spins++ & 3u) == 0) {
                            w = sld(sm.xf + (size_t)(gseg - 1) * 16 + i);
                            if ((w >> 32) == (tagF >> 32) && ((w >> 24) & 0xFFu) <= rnd) { p_final = true; p_word = w; break; }
                        }
                        if ((spins & 255u) == 0 && globaltimer_ns() - t0 > a.wait_ns) __trap();
                    }
                }
                s_specXp[i] = (uint32_t)w & 0x1FFFFu;
            }
            if (tid + 1 == gseg) s_predc = cbit ? 1u : 0u;         // the bit of the stage right in front of me
            const int unset = __syncthreads_count(!cbit);
            const bool allc = unset == 0;
            // Knowledge lags a round: the stage whose entry becomes the true one NEXT round sits behind a consistent prefix whose last member's
            // bit is not set yet (that member's own entry became the true one only this round).  So "everything in front but the stage right
            // in front of me is consistent" already exempts the next simulation from the cut-off — otherwise the frontier itself could be cut
            // off and every step of it would cost a second round (tests/spec_rounds_model.cpp).
            const bool near = allc || (unset == 1 && !s_predc);
            const bool certified = allc && c_prev;
            stamp_if(dbg && tid == 0, dbg + rnd * 8 + 5);
            store_if(dbg && tid == 0, dbg + rnd * 8 + 7, s_nlog | ((unsigned long long)need_sim << 32));
            if (gseg > 0 && tid == 192) pub_nb(sm.ack + gseg, ((unsigned long long)tage << 32) | (certified ? 0xFFFFu : rnd), true);
            if (certified) {    // every entry up to mine was the true token one round ago and has not moved since: the log in shared memory is THE log
                if (tid < ISL_MAX_PROFILES) {
                    pub_nb(sm.xf + (size_t)gseg * 16 + tid, tagF | (rnd << 24) | s_specX[tid], false);
                    if (gseg == gtot - 1 && a.heads_out) a.heads_out[(size_t)c * ISL_MAX_PROFILES + tid] = s_specX[tid];
                }
                if (tid == 16) pub_down(sm.df + gseg, tagF | (rnd << 24) | (s_dqr[0] << 13) | s_dqr[1]);
                if (tid == 0) { st_steps += spec_steps; st_visited += spec_visited; if (gseg == gtot - 1) { st_rounds_sum += rnd; ++st_cells; } if (tr) { tr[0] = t_cell; tr[2] = globaltimer_ns(); tr[6] = s_nlog; tr[7] = st_sims - sims_cell; tr[11] = rnd; } }
                break;
            }
            if (tid < 32) {     // c for the next round; the corrected prediction
                const bool same = tid >= ISL_MAX_PROFILES || s_specH[tid] == s_specXp[tid];
                const bool cnow = __all_sync(0xFFFFFFFFu, same);
                uint32_t mq = 0, mr = 0, hold = 0, hn = 0;
                const uint32_t qcl = tid < ISL_MAX_PROFILES ? s_qc[tid] : 0u, wl = tid < ISL_MAX_PROFILES ? s_minsize[tid] : 1u;
                if (tid < ISL_MAX_PROFILES) {
                    hold = s_specH[tid];
                    hn = s_specXp[tid];
                    if ((s_grp_big >> tid) & 1u) mq = hn;
                    if ((s_grp_small >> tid) & 1u) mr = hn * s_minsize[tid];
                }
                mq = __reduce_add_sync(0xFFFFFFFFu, mq); mr = __reduce_add_sync(0xFFFFFFFFu, mr);
                hn = spec_spread_warp(hn, qcl, wl, s_grp_big, (int)s_acc[0] - (int)mq, false, lane);
                hn = spec_spread_warp(hn, qcl, wl, s_grp_small, (int)s_acc[1] - (int)mr, true, lane);
                {   // Two candidates for the next entry: the Newton step (hn) and plain chaining (the exit of the stage in front as it is).  Where a
                    // batch's contested front reaches far the Newton step over-corrects round after round; each stage uses the rule whose
                    // candidate of the PREVIOUS round came closer to what the stage in front has published now (study, section 8).
                    // The candidates of round 1 are not scored: they come from the occupancy guess, and judging the rules by them sends
                    // stages to plain chaining too early (batch 8 of config 4: 24 -> 19 rounds).
                    const uint32_t xp = tid < ISL_MAX_PROFILES ? s_specXp[tid] : 0u;
                    uint32_t ea = 0, eb = 0;
                    if (tid < ISL_MAX_PROFILES && s_havepred) { ea = (uint32_t)abs((int)s_predA[tid] - (int)xp); eb = (uint32_t)abs((int)s_predB[tid] - (int)xp); }
                    ea = __reduce_add_sync(0xFFFFFFFFu, ea); eb = __reduce_add_sync(0xFFFFFFFFu, eb);
                    __syncwarp();
                    if (tid < ISL_MAX_PROFILES) { s_predA[tid] = hn; s_predB[tid] = xp; }
                    if (tid == 0 && rnd >= 2) s_havepred = 1;
                    if (eb < ea) hn = xp;
                }
                if (tid < ISL_MAX_PROFILES) s_specH[tid] = hn;
                const bool moved = tid < ISL_MAX_PROFILES && hn != hold;
                const bool changed = __any_sync(0xFFFFFFFFu, moved);
                // a cut-off simulation left no usable log: the entry is simulated again (in full once it is known to be the true one) and counts as
                // inconsistent until then
                if (tid == 0) s_specflag = (cnow && s_capst[2] ? 1u : 0u) | (changed || !s_capst[2] ? 2u : 0u);
                stamp_if(dbg && tid == 0, dbg + rnd * 8 + 6);
            }
            __syncthreads();
            c_prev = s_specflag & 1u; need_sim = s_specflag & 2u; known_exact = near;
            if (++rnd >= kSpecRounds - 1) __trap();      // cannot happen: every round certifies at least one more stage
        }
        }   // rounds
        if (idle_break) break;
        if (last_sub && c + 1 < a.n_chunks && !a.ready && !a.window) { queue_load_async(c + 1); prefetched = true; }   // the chain is done with the queues: fetch the next chunk's behind the commit
        {   // 6. commit
            const uint32_t nlog = s_nlog;
            for (uint32_t j = tid; j < nlog; j += kPipeThreads) {
                const uint2 e = s_log[j];
                const uint32_t l = sb_base + (s_cand[((e.y - sa_cand) >> 2) - 2] >> 16), mask = e.x & 0xFFu, t = (e.x >> 15) & 0xFFFFu;
                const uint2 rec = pack_result(flip_gpu(lo_s + l, a.flip), __ffs(mask) - 1, __popc(mask), ISL_ST_PLACED);
                a.out[cd.req_off + t] = rec;
                if (a.owner_out) a.owner_out[cd.req_off + t] = rec;         // partitioned inventory: straight into the owner rank's result array (peer store over NVLink)
                atomicOr(&s_occ32[l >> 2], mask << ((l & 3u) * 8u));
            }
        }
        __syncthreads();
        if (tr && tid == 0) tr[3] = globaltimer_ns();
        }   // sub-segments
        chunk_done(c);
        if (c + 1 < a.n_chunks && !prefetched) { closed = wait_ready(c + 1); if (!closed) queue_load_async(c + 1); }   // fed / windowed stream: the next batch may not be due yet
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    for (uint32_t i = tid; i < n_g; i += kPipeThreads) a.occ[lo_s + i] = reinterpret_cast<uint8_t*>(s_occ32)[i];
    if (a.owner_out) __threadfence_system();        // the peer stores of this CTA are performed before the grid is seen as complete
    if (tid == 0 && st_steps + st_jumps) {
        atomicAdd(&a.stats->placed, st_steps);
        atomicAdd(&a.stats->steps, st_steps);
        atomicAdd(&a.stats->visited, st_visited);
        atomicAdd(&a.stats->jumps, st_jumps);
    }
    if (kSpec && tid == 0) {
        atomicAdd(&a.stats->spec_sims, st_sims);
        atomicAdd(&a.stats->spec_rounds, st_rounds_sum);
        atomicAdd(&a.stats->spec_cells, (unsigned long long)st_cells);
    }
}

// ---------------------------------------------------------------------------------------------
// k_capacity: the what-if / defragmentation query (SURVEY 8f-4).  cap[p] = how many more pods of profile p ALONE the GPUs of [lo, hi)
// could still take = sum over GPUs of capn[table][p][occupancy] (the same per-byte table the scan-mode commit places from).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_capacity(const uint8_t* __restrict__ occ, const uint8_t* __restrict__ gtab, const uint8_t* __restrict__ capn,
                                                   uint32_t n_profiles, uint32_t lo, uint32_t hi, unsigned long long* __restrict__ cap) {
    __shared__ unsigned long long s_cap[ISL_MAX_PROFILES];
    if (threadIdx.x < ISL_MAX_PROFILES) s_cap[threadIdx.x] = 0;
    __syncthreads();
    uint32_t acc[ISL_MAX_PROFILES];
#pragma unroll
    for (uint32_t p = 0; p < ISL_MAX_PROFILES; ++p) acc[p] = 0;
    for (uint32_t g = lo + blockIdx.x * blockDim.x + threadIdx.x; g < hi; g += gridDim.x * blockDim.x) {
        const uint32_t o = occ[g], t = gtab[g] & (kMaxTables - 1);
#pragma unroll
        for (uint32_t p = 0; p < ISL_MAX_PROFILES; ++p) if (p < n_profiles) acc[p] += capn[(t * ISL_MAX_PROFILES + p) * 256 + o];
    }
#pragma unroll
    for (uint32_t p = 0; p < ISL_MAX_PROFILES; ++p) {
        uint32_t v = acc[p];
#pragma unroll
        for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, d);
        if ((threadIdx.x & 31u) == 0 && v) atomicAdd(&s_cap[p], (unsigned long long)v);
    }
    __syncthreads();
    if (threadIdx.x < ISL_MAX_PROFILES && s_cap[threadIdx.x]) atomicAdd(&cap[threadIdx.x], s_cap[threadIdx.x]);
}

// ---------------------------------------------------------------------------------------------
// k_bestfit: ISL_POLICY_BEST_FIT (extension, SURVEY 8a-ext — no reference counterpart, parity is against
// oracle/ref_fast.cpp's best-fit).  Among the GPUs on which the profile has a legal start, take the one with the
// fewest free slices after the placement = the highest popcount of the occupancy byte, ties to the lowest canonical
// index; the start is the reference's first legal start.  Requests are resolved strictly in order (request-major: a
// placement can make a GPU the best fit of the very next request, so there is no GPU-major shortcut).
// State: GPUs grouped by occupancy byte (256 classes); per class a two-level bitmap (32 GPUs per word, 1024 per
// summary bit) and its minimum member.  One warp: lane = a few classes, key = (8 - popcount) << 24 | class minimum,
// redux.min picks the GPU; lane 0 moves it to its new class.  One CTA; all threads build the class structure.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kBfThreads = 1024;
constexpr uint32_t kBfMaxGpus = 1u << 20;           // class bitmaps: G / 32 words + G / 1024 summary words per (table, occupancy byte) class
constexpr uint32_t kBfSmemGpus = 4096;              // up to here the class bitmaps live in shared memory (132 KiB)

template <bool kMulti>
__global__ void __launch_bounds__(kBfThreads, 1) k_bestfit(uint32_t n, const uint2* __restrict__ in, uint2* __restrict__ out, uint8_t* __restrict__ occ,
                                                           uint32_t lo, uint32_t hi, const uint8_t* __restrict__ lut, DevProfiles prof,
                                                           uint32_t* __restrict__ g_bitmaps, Ctrl* ctrl, const uint8_t* __restrict__ score,
                                                           const uint8_t* __restrict__ gtab, const uint8_t* __restrict__ sizes, uint32_t n_tables) {
    extern __shared__ __align__(16) uint32_t s_dyn[];
    // a class = (table of the GPU's node, occupancy byte): every GPU of a class behaves the same for every profile
    __shared__ uint32_t s_min[kMaxTables * 256];
    __shared__ uint8_t s_lut[ISL_MAX_PROFILES * 256];
    // what the policy minimises, per (table, profile, occupancy byte): ISL_POLICY_BEST_FIT = free slices (8 - popcount), ISL_POLICY_MIN_FRAG =
    // (profile, start) pairs of the table that stop being feasible when the profile takes its first legal start there (host-built)
    __shared__ uint8_t s_score[ISL_MAX_PROFILES * 256];
    __shared__ uint8_t s_sizes[kMaxTables * ISL_MAX_PROFILES];
    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    const uint32_t Gr = hi - lo, W0 = (Gr + 31) / 32, W1 = (W0 + 31) / 32, stride = W0 + W1;   // words per class
    const uint32_t n_cls = n_tables * 256;
    const bool small = n_tables == 1 && Gr <= kBfSmemGpus;      // bitmaps in shared memory; otherwise in global memory, zeroed by the host
    uint32_t* bm = small ? s_dyn : g_bitmaps;
    if (small) for (uint32_t i = tid; i < 256 * stride; i += kBfThreads) bm[i] = 0;
    // one table (kMulti == false): the per-byte tables sit in shared memory; several: they are read from global memory (L1-resident,
    // 8 KiB per table)
    if (!kMulti) for (uint32_t i = tid; i < ISL_MAX_PROFILES * 256; i += kBfThreads) { s_lut[i] = lut[i]; s_score[i] = score[i]; }
    auto lut_at = [&](uint32_t idx) -> uint32_t { return kMulti ? (uint32_t)__ldg(lut + idx) : (uint32_t)s_lut[idx]; };
    auto score_at = [&](uint32_t idx) -> uint32_t { return kMulti ? (uint32_t)__ldg(score + idx) : (uint32_t)s_score[idx]; };
    if (tid < kMaxTables * ISL_MAX_PROFILES) s_sizes[tid] = sizes[tid];
    for (uint32_t i = tid; i < n_cls; i += kBfThreads) s_min[i] = kInf;
    __syncthreads();
    for (uint32_t g = tid; g < Gr; g += kBfThreads) {           // build: every GPU joins its class
        const uint32_t c = (kMulti ? (uint32_t)(gtab[lo + g] & (kMaxTables - 1)) * 256u : 0u) + occ[lo + g];
        atomicOr(&bm[c * stride + (g >> 5)], 1u << (g & 31u));
        atomicOr(&bm[c * stride + W0 + (g >> 10)], 1u << ((g >> 5) & 31u));
        atomicMin(&s_min[c], g);
    }
    __syncthreads();
    if (!is_chain_warp(tid >> 5)) return;
    uint32_t placed = 0;
    uint32_t dead = 0;              // profiles that found no GPU: occupancy only grows inside a batch's ALLOC phase, so they never will again
    uint2 ahead = lane < n ? in[lane] : make_uint2(0, (uint32_t)ISL_OP_NOOP << 8);
    for (uint32_t base = 0; base < n; base += 32) {
        const uint2 mine = ahead;                               // the next block's requests are fetched while this one is resolved
        ahead = base + 32 + lane < n ? in[base + 32 + lane] : make_uint2(0, (uint32_t)ISL_OP_NOOP << 8);
        // only the live ALLOCs of the block are looked at (frees, unknown or dead profiles: defaults were written by k_prepare)
        uint32_t live;
        {
            const uint32_t wp = mine.y & 0xFFu, wop = (mine.y >> 8) & 0xFFu;
            live = __ballot_sync(0xFFFFFFFFu, wop == ISL_OP_ALLOC && wp < prof.n && !((dead >> wp) & 1u));
        }
        while (live) {
            const uint32_t j = __ffs(live) - 1;
            live &= live - 1;
            const uint32_t p = __shfl_sync(0xFFFFFFFFu, mine.y, j) & 0xFFu;
            if ((dead >> p) & 1u) continue;                     // died inside this block
            uint32_t key = kInf, kc = 0;
#pragma unroll 8
            for (uint32_t c = lane; c < n_cls; c += 32) {       // lane l looks at classes l, l+32, ...
                const uint32_t mn = s_min[c];
                const uint32_t idx = ((c >> 8) * ISL_MAX_PROFILES + p) * 256 + (c & 255u);
                if (mn != kInf && lut_at(idx) != ISL_START_NONE) {
                    const uint32_t k2 = (score_at(idx) << 24) | mn;
                    if (k2 < key) { key = k2; kc = c; }
                }
            }
            const uint32_t m = __reduce_min_sync(0xFFFFFFFFu, key);
            if (m == kInf) { dead |= 1u << p; continue; }      // stays NO_CAPACITY, and so does every later request of the profile
            const uint32_t g = m & 0xFFFFFFu;
            const uint32_t cw = __shfl_sync(0xFFFFFFFFu, kc, __ffs(__ballot_sync(0xFFFFFFFFu, key == m)) - 1);   // the class IS (table, occupancy byte)
            const uint32_t t = cw >> 8, o = cw & 255u;
            const uint32_t start = lut_at((t * ISL_MAX_PROFILES + p) * 256 + o), size = s_sizes[t * ISL_MAX_PROFILES + p];
            const uint32_t o2 = o | ((((1u << size) - 1u) << start) & 0xFFu), cw2 = (t << 8) | o2;
            uint32_t* c0 = bm + cw * stride;
            uint32_t* c1 = bm + cw2 * stride;
            __syncwarp();                                       // all lanes have read the class minima before they are rewritten
            if (lane == 0) {                                    // the GPU leaves class o and joins class o2: independent words, loads first
                const uint32_t w0 = c0[g >> 5] & ~(1u << (g & 31u)), w1 = c1[g >> 5] | (1u << (g & 31u));
                const uint32_t s1 = c1[W0 + (g >> 10)] | (1u << ((g >> 5) & 31u));
                c0[g >> 5] = w0; c1[g >> 5] = w1; c1[W0 + (g >> 10)] = s1;
                if (w0 == 0) c0[W0 + (g >> 10)] &= ~(1u << ((g >> 5) & 31u));
                occ[lo + g] = (uint8_t)o2;
                out[base + j] = pack_result(flip_gpu(lo + g, prof.flip), start, size, ISL_ST_PLACED);
                if (g < s_min[cw2]) s_min[cw2] = g;
                ++placed;
            }
            __syncwarp();
            // new minimum of the class (g was its minimum: nothing below it).  Usually it sits under the summary word that held g: every
            // lane reads that word (one broadcast); only when it is empty do the lanes look at the further summary words, 32 at a time
            uint32_t mn = kInf;
            {
                const uint32_t k = g >> 10, sw = c0[W0 + k];
                if (sw) { const uint32_t wi = k * 32 + __ffs(sw) - 1; mn = wi * 32 + __ffs(c0[wi]) - 1; }
                else
                    for (uint32_t k0 = k + 1; k0 < W1; k0 += 32) {
                        const uint32_t s2 = k0 + lane < W1 ? c0[W0 + k0 + lane] : 0u;
                        const uint32_t b = __ballot_sync(0xFFFFFFFFu, s2 != 0);
                        if (b) {
                            const uint32_t src = __ffs(b) - 1;
                            const uint32_t wi = (k0 + src) * 32 + __ffs(__shfl_sync(0xFFFFFFFFu, s2, src)) - 1;
                            mn = wi * 32 + __ffs(c0[wi]) - 1;
                            break;
                        }
                    }
            }
            if (lane == 0) s_min[cw] = mn;
            __syncwarp();
        }
    }
    if (lane == 0) { atomicAdd(&ctrl->placed, (unsigned long long)placed); atomicAdd(&ctrl->steps, (unsigned long long)placed); }
}

}  // namespace isl
