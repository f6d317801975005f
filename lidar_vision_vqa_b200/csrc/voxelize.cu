// Point -> pillar grouping on the GPU with the hard voxeliser's deterministic semantics
// (replaces the spconv CPU call behind src/lidar-encoder/pcdet/datasets/processor/data_processor.py:16-61,133-180):
//
//   k_quantize_insert   coalesced float4 tile loads -> fp32 sub/div/floor -> cell key -> open-addressing hash insert
//                       (one 64-bit atomicCAS on {key, first index}: claims the slot and records the first point at
//                       once; an atomicMin follows only if a later-arriving point has a smaller index) and
//                       atomicAdd(count).  __match_any_sync merges the lanes of a warp that hit
//                       the same cell so one lane talks to HBM for the whole group.  One point per thread: the kernel
//                       is a chain of L2 round trips, so it wants as many warps in flight as the SMs hold.
//   k_scan_assign       single-pass scan over points in index order of [point is the first of its cell] and of the
//                       cell counts: gives every pillar its id in first-appearance order and the start of its point
//                       list, with no sort.  Tiles publish their aggregate at once; a tile sums the aggregates of the
//                       tiles of its 256-tile group in ONE parallel read plus the published prefix of the previous
//                       group, so the dependency chain is n_tiles/256 long instead of n_tiles.
//   k_place             moves each point into its pillar's list (index list and/or 32-byte point records); block 0
//                       also turns the per-frame first-appearance counts into output rows under the max_voxels cap.
//
// The per-pillar "first P points in index order" rule is applied by the consumers (pfn.cu) with a radix select over
// the list, so nothing here depends on the order in which atomics land.
#include "group_common.cuh"

namespace pillars {

namespace {

constexpr int kThreads = 256;
constexpr int kPerThread = kTile / kThreads;  // 4 (scan kernel); must stay a multiple of 4 (int4 slot loads)
constexpr int kGroup = kLookGroup;            // tiles per look-back group

__device__ __forceinline__ uint32_t hash_key(uint32_t k)
{
    k *= 0x9E3779B1u;
    k ^= k >> 15;
    k *= 0x85EBCA77u;
    k ^= k >> 13;
    return k;
}

// ---------------------------------------------------------------------------------------------
// frame offsets from the batch-index column (datasets/dataset.py:237-244 writes that column)
// ---------------------------------------------------------------------------------------------
__global__ void k_frame_offsets(const float *__restrict__ pts, int64_t n, int stride, int nb, int32_t *__restrict__ offs)
{
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i > n) return;
    // frame of row i-1 and of row i; offsets[f] = i for every f in (prev, cur]
    int prev = (i == 0) ? -1 : static_cast<int>(pts[(i - 1) * stride]);
    int cur = (i == n) ? nb : static_cast<int>(pts[i * stride]);
    prev = max(-1, min(prev, nb));
    cur = max(0, min(cur, nb));
    for (int f = prev + 1; f <= cur; ++f) offs[f] = static_cast<int32_t>(i);
}

// ---------------------------------------------------------------------------------------------
// K1: one point per thread, 256 points per CTA
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 8)
k_quantize_insert(const float *__restrict__ points, int64_t n, int stride, int col0,
                  const int32_t *__restrict__ frame_offsets, int nb, GridDev gd, HashEntry *__restrict__ table,
                  uint32_t cap, int32_t *__restrict__ point_slot, uint32_t *__restrict__ point_arrival, int vec_ok,
                  uint4 *__restrict__ zero_region, uint32_t zero_vecs, uint4 *__restrict__ ff_region, uint32_t ff_vecs)
{
    // Scratch that only the LATER kernels of the call read is initialised here, in the shadow of this kernel's atomic round
    // trips, instead of by separate memsets: the scan's header / tile descriptors (zero) and the BEV index map (-1).
    {
        const uint32_t gtid = blockIdx.x * kThreads + threadIdx.x, gsz = gridDim.x * kThreads;
        if (gtid < zero_vecs) zero_region[gtid] = make_uint4(0u, 0u, 0u, 0u);
        for (uint32_t v = gtid; v < ff_vecs; v += gsz) ff_region[v] = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
    }
    extern __shared__ __align__(16) float s_pts[];  // [kThreads * stride]
    __shared__ uint32_t s_cnt[2];

    pdl_trigger();
    const int tid = threadIdx.x;
    const int64_t tile_start = static_cast<int64_t>(blockIdx.x) * kThreads;
    const int count = static_cast<int>(tmin<int64_t>(kThreads, n - tile_start));
    if (tid < 2) s_cnt[tid] = 0u;
    __syncthreads();
    load_point_tile(points + tile_start * stride, count, stride, vec_ok, s_pts, tid, kThreads);
    {  // frames touched by this tile: [b0, b1] = (frame starts <= first / last point of the tile) - 1; independent loads
        uint32_t c_lo, c_hi;
        count_frame_starts(frame_offsets, nb, tile_start, tile_start + count - 1, tid, kThreads, c_lo, c_hi);
        if (c_lo) atomicAdd(&s_cnt[0], c_lo);
        if (c_hi) atomicAdd(&s_cnt[1], c_hi);
    }
    __syncthreads();
    const int s_b0 = static_cast<int>(s_cnt[0]) - 1, s_b1 = static_cast<int>(s_cnt[1]) - 1;

    const int64_t i = tile_start + tid;
    bool valid = false;
    uint32_t key = 0;
    if (tid < count) {
        uint32_t cell = 0;
        valid = quantize_point(s_pts + tid * stride + col0, gd, cell);
        if (valid) {
            int b = s_b0;  // almost always the only frame of the tile
            const int b1 = s_b1;
            while (b < b1 && __ldg(frame_offsets + b + 1) <= i) ++b;
            key = static_cast<uint32_t>(b) * gd.cells + cell;
        }
    }
    const unsigned active = __ballot_sync(0xffffffffu, valid);
    int32_t slot_out = -1;
    uint32_t arrival = 0;
    if (valid) {
        const int lane = tid & 31;
        const unsigned peers = __match_any_sync(active, key);
        const int leader = __ffs(peers) - 1;  // lowest lane == smallest point index of the group
        uint32_t slot = 0, base = 0;
        if (lane == leader) {
            slot = static_cast<uint32_t>((static_cast<uint64_t>(hash_key(key)) * cap) >> 32);
            const unsigned long long mine = (static_cast<unsigned long long>(key) << 32) | static_cast<uint32_t>(i);
            while (true) {
                unsigned long long *word = reinterpret_cast<unsigned long long *>(&table[slot]);
                const unsigned long long cur = atomicCAS(word, 0xFFFFFFFFFFFFFFFFull, mine);
                if (cur == 0xFFFFFFFFFFFFFFFFull) break;  // claimed: key and first index set by the same atomic
                if (static_cast<uint32_t>(cur >> 32) == key) {
                    if (mine < cur) atomicMin(word, mine);  // same key in the high half: orders by point index
                    break;
                }
                slot = (slot + 1 == cap) ? 0u : slot + 1;
            }
            base = atomicAdd(&table[slot].cnt, static_cast<uint32_t>(__popc(peers))) + 1u;
        }
        slot = __shfl_sync(peers, slot, leader);
        base = __shfl_sync(peers, base, leader);
        slot_out = static_cast<int32_t>(slot);
        arrival = base + static_cast<uint32_t>(__popc(peers & lanemask_lt()));
    }
    if (tid < count) {
        point_slot[i] = slot_out;
        point_arrival[i] = arrival;
    }
}

// ---------------------------------------------------------------------------------------------
// K2: scan.  Descriptor = valid(1) | pillars(31) | listed points(31); running sums travel as (pillars << 32 | listed)
// ---------------------------------------------------------------------------------------------
constexpr unsigned long long kValid = 1ull << 63;

__device__ __forceinline__ unsigned long long pack_desc(unsigned long long v)
{
    return kValid | ((v >> 32) << 31) | (v & 0x7FFFFFFFull);
}
__device__ __forceinline__ unsigned long long unpack_desc(unsigned long long d)
{
    d &= ~kValid;
    return ((d >> 31) << 32) | (d & 0x7FFFFFFFull);
}
__device__ __forceinline__ unsigned long long wait_desc(const unsigned long long *p)
{
    unsigned long long d;
    do {
        d = ld_relaxed_u64(p);
    } while (!(d & kValid));
    return unpack_desc(d);
}

__global__ void __launch_bounds__(kThreads)
k_scan_assign(int64_t n, uint32_t n_tiles, const int32_t *__restrict__ point_slot, HashEntry *__restrict__ table,
              Header *__restrict__ hdr, unsigned long long *__restrict__ tile_agg, unsigned long long *__restrict__ tile_prefix,
              uint32_t *__restrict__ pillar_key, uint32_t *__restrict__ pillar_list,
              uint32_t *__restrict__ pillar_cnt, const int32_t *__restrict__ frame_offsets, int nb,
              uint32_t *__restrict__ frame_gstart, int dynamic_ids, int max_voxels, uint32_t *__restrict__ frame_rowbase,
              int32_t *__restrict__ pillar_count)
{
    __shared__ uint32_t s_tile;
    __shared__ unsigned long long s_warp[kThreads / 32];
    __shared__ unsigned long long s_look[kThreads / 32];
    __shared__ uint32_t s_thr_excl[kThreads];
    __shared__ uint8_t s_thr_flags[kThreads];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    pdl_wait();
    pdl_trigger();
    // A tile spins on its predecessors, so they must be running: guaranteed when the whole grid is co-resident
    // (blockIdx is then the tile id), otherwise ids are handed out in scheduling order.
    if (dynamic_ids) {
        if (tid == 0) s_tile = atomicAdd(&hdr->tile_counter, 1u);
        __syncthreads();
    }
    const uint32_t tile = dynamic_ids ? s_tile : blockIdx.x;
    const int64_t tile_start = static_cast<int64_t>(tile) * kTile;
    const int64_t i0 = tile_start + tid * kPerThread;

    int32_t slot[kPerThread];
    if (i0 + kPerThread <= n) {
#pragma unroll
        for (int k = 0; k < kPerThread; k += 4) {
            const int4 v = *reinterpret_cast<const int4 *>(point_slot + i0 + k);
            slot[k] = v.x; slot[k + 1] = v.y; slot[k + 2] = v.z; slot[k + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int k = 0; k < kPerThread; ++k) slot[k] = (i0 + k < n) ? point_slot[i0 + k] : -1;
    }
    uint4 ent[kPerThread];
#pragma unroll
    for (int k = 0; k < kPerThread; ++k)  // all gathers in flight before the first use
        ent[k] = slot[k] >= 0 ? *reinterpret_cast<const uint4 *>(&table[slot[k]]) : make_uint4(0xFFFFFFFFu, 0, 0, 0);
    unsigned long long val[kPerThread];
    unsigned flags = 0;
    unsigned long long tsum = 0;
#pragma unroll
    for (int k = 0; k < kPerThread; ++k) {
        val[k] = 0;
        if (slot[k] >= 0 && ent[k].x == static_cast<uint32_t>(i0 + k)) {  // this point opened the pillar
            val[k] = (1ull << 32) | static_cast<unsigned long long>(ent[k].z + 1u);
            flags |= 1u << k;
        }
        tsum += val[k];
    }
    // block-wide exclusive scan of tsum
    unsigned long long incl = tsum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    unsigned long long warp_excl = 0, tile_sum = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) {
        const unsigned long long s = s_warp[w];
        if (w < warp) warp_excl += s;
        tile_sum += s;
    }
    const unsigned long long thr_excl = warp_excl + incl - tsum;
    if (tid == 0) st_relaxed_u64(&tile_agg[tile], pack_desc(tile_sum));  // visible to the successors at once

    // look-back: aggregates of the tiles of my group that precede me (one parallel read) + prefix of the previous group
    const uint32_t group_first = tile & ~static_cast<uint32_t>(kGroup - 1);
    unsigned long long look = 0;
    if (group_first + tid < tile) look = wait_desc(&tile_agg[group_first + tid]);
    if (tid == kThreads - 1 && group_first > 0) look += wait_desc(&tile_prefix[group_first - 1]);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) look += __shfl_xor_sync(0xffffffffu, look, s);
    if (lane == 0) s_look[warp] = look;
    s_thr_excl[tid] = static_cast<uint32_t>(thr_excl >> 32);
    s_thr_flags[tid] = static_cast<uint8_t>(flags);
    __syncthreads();
    unsigned long long tile_excl = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) tile_excl += s_look[w];
    if (tid == 0 && (tile & (kGroup - 1)) == kGroup - 1) st_relaxed_u64(&tile_prefix[tile], pack_desc(tile_excl + tile_sum));

    unsigned long long run = tile_excl + thr_excl;
#pragma unroll
    for (int k = 0; k < kPerThread; ++k) {
        if (flags & (1u << k)) {
            const uint32_t g = static_cast<uint32_t>(run >> 32);
            // cnt was only needed by this (owning) thread: the entry now carries the list base and the pillar id, so
            // k_place resolves a point with one 16-byte load
            *reinterpret_cast<uint2 *>(&table[slot[k]].cnt) = make_uint2(static_cast<uint32_t>(run & 0xFFFFFFFFull), g);
            pillar_key[g] = ent[k].y;
            pillar_list[g] = static_cast<uint32_t>(run & 0xFFFFFFFFull);
            pillar_cnt[g] = static_cast<uint32_t>(val[k] & 0xFFFFFFFFull);
            run += val[k];
        }
    }

    // first-appearance id at every frame start that falls into this tile
    const bool last_tile = (tile == n_tiles - 1);
    const uint32_t tile_total = static_cast<uint32_t>((tile_excl + tile_sum) >> 32);
    for (int f = tid; f <= nb; f += kThreads) {
        const int64_t pos = frame_offsets[f];
        if (pos >= tile_start && pos < tile_start + kTile && pos < n) {
            const int rel = static_cast<int>(pos - tile_start);
            const int t = rel / kPerThread, k = rel % kPerThread;
            frame_gstart[f] = static_cast<uint32_t>(tile_excl >> 32) + s_thr_excl[t] +
                              __popc(static_cast<unsigned>(s_thr_flags[t]) & ((1u << k) - 1u));
        } else if (pos >= n && last_tile) {
            frame_gstart[f] = tile_total;
        }
    }
    if (last_tile && tid == 0) {
        hdr->total_pillars = tile_total;
        hdr->total_listed = static_cast<uint32_t>((tile_excl + tile_sum) & 0xFFFFFFFFull);
    }

    // The tile that finishes last turns the per-frame first-appearance counts into output rows under the max_voxels cap
    // (every frame start has been published by then).
    __shared__ uint32_t s_done;
    __threadfence();
    __syncthreads();
    if (tid == 0) s_done = atomicAdd(&hdr->tiles_done, 1u);
    __syncthreads();
    if (s_done == n_tiles - 1 && warp == 0) {
        uint32_t carry = 0;
        for (int f0 = 0; f0 < nb; f0 += 32) {
            const int f = f0 + lane;
            uint32_t m = 0;
            if (f < nb) m = min(__ldcg(frame_gstart + f + 1) - __ldcg(frame_gstart + f), static_cast<uint32_t>(max_voxels));
            uint32_t incl = m;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += o;
            }
            if (f < nb) {
                frame_rowbase[f] = carry + incl - m;
                if (pillar_count) pillar_count[f] = static_cast<int32_t>(m);
            }
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) {
            frame_rowbase[nb] = carry;
            if (pillar_count) pillar_count[nb] = static_cast<int32_t>(carry);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K3: lists.  For the streaming feature kernel it also resolves everything about a pillar that needs no feature
// arithmetic: the point's coordinates relative to the pillar centre go into its record, and the thread of the point that
// opened the pillar writes the pillar's constants (centre, row, count) plus voxel_coords / voxel_num_points / the BEV index
// map.  This kernel waits on L2 round trips, so the extra integer work is free; in the feature kernel it was not.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_place(const __grid_constant__ PlaceParams p)
{
    pdl_wait();
    pdl_trigger();
    const int64_t i = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x;
    if (i >= p.n) return;
    const int32_t s = p.point_slot[i];
    if (s < 0) return;
    const uint4 e = *reinterpret_cast<const uint4 *>(&p.table[s]);  // {first, key, list base, pillar id}
    const uint32_t g = e.w;
    const uint32_t arrival = p.point_arrival[i];
    const uint32_t pos = e.z + arrival;
    if (p.sorted_idx) p.sorted_idx[pos] = static_cast<uint32_t>(i);
    if (!p.records) return;

    const CellCoord c = decode_key(p, e.y);
    write_record(p, i, c, pos, arrival);

    if (e.x == static_cast<uint32_t>(i)) {  // this point opened the pillar
        const uint32_t n = p.pillar_cnt[g];
        const uint32_t local = g - p.frame_gstart[c.b];
        const int64_t row = static_cast<int64_t>(p.frame_rowbase[c.b]) + local;
        const bool live = local < static_cast<uint32_t>(p.gd.max_voxels) && row < p.capacity;
        const uint32_t P = static_cast<uint32_t>(p.gd.max_points);
        // indexed by the list START POSITION, so the consumer needs nothing but its own position to find it
        publish_pillar(p.pillar_meta, p.long_list, p.long_count, e.z, c, live ? static_cast<uint32_t>(row) : 0xFFFFFFFFu, n);
        if (live) {
            if (p.voxel_coords)
                *reinterpret_cast<int4 *>(p.voxel_coords + row * 4) =
                    make_int4(static_cast<int>(c.b), static_cast<int>(c.z), static_cast<int>(c.y), static_cast<int>(c.x));
            if (p.voxel_num_points) p.voxel_num_points[row] = static_cast<int32_t>(min(n, P));
            if (p.cell_row)
                p.cell_row[static_cast<int64_t>(c.b) * p.gd.cells_xy + static_cast<int64_t>(c.y) * p.gd.g[0] + c.x] =
                    static_cast<int32_t>(row);
        }
    }
}

}  // namespace

cudaError_t launch_frame_offsets(const float *points_b, int64_t n, int stride, int nb, int32_t *offs, cudaStream_t st)
{
    const int threads = 256;
    const int64_t blocks = (n + 1 + threads - 1) / threads;
    k_frame_offsets<<<static_cast<unsigned>(blocks), threads, 0, st>>>(points_b, n, stride, nb, offs);
    note_launch();
    return cudaGetLastError();
}

cudaError_t launch_group_points(const float *points, int64_t n, int stride, int col0, int c_point,
                                const int32_t *frame_offsets, int nb, const GridDev &gd, const Workspace &ws,
                                int32_t *pillar_count, bool want_index_lists, const PlaceExtras &extras, cudaStream_t st)
{
    if (ws.mode == kGroupDense)
        return launch_group_points_dense(points, n, stride, col0, c_point, frame_offsets, nb, gd, ws, pillar_count,
                                         want_index_lists, extras, st);
    cudaError_t err;
    // One memset per call: the hash table must be empty before the first insert.  The rest of the scratch (scan header and
    // tile descriptors: zero; BEV index map: -1) is initialised by the insert kernel itself, unless there is no point at all.
    // The index map sits at the end of the 0xFF region; a call that reads no map leaves it alone.
    const size_t table_bytes = reinterpret_cast<char *>(ws.cell_row) - ws.ff_begin;
    const size_t map_bytes = extras.skip_index_map ? 0 : ws.ff_bytes - table_bytes;
    const bool in_kernel_init = n > 0 && static_cast<int64_t>(ws.zero_bytes / 16) <= n && ws.zero_bytes % 16 == 0 &&
                                map_bytes % 16 == 0;
    if (!in_kernel_init) {
        if ((err = cudaMemsetAsync(ws.zero_begin, 0, ws.zero_bytes, st)) != cudaSuccess) return err;
        note_launch();
    }
    if ((err = cudaMemsetAsync(ws.ff_begin, 0xFF, in_kernel_init ? table_bytes : table_bytes + map_bytes, st)) != cudaSuccess)
        return err;
    note_launch();
    if (n == 0) {
        if (pillar_count) {
            if ((err = cudaMemsetAsync(pillar_count, 0, sizeof(int32_t) * (nb + 1), st)) != cudaSuccess) return err;
            note_launch();
        }
        return cudaSuccess;
    }
    const size_t smem = sizeof(float) * kThreads * stride;
    const int vec_ok = (reinterpret_cast<uintptr_t>(points) % 16 == 0) ? 1 : 0;  // tile starts are 256 rows apart
    const unsigned pb = static_cast<unsigned>((n + kThreads - 1) / kThreads);
    k_quantize_insert<<<pb, kThreads, smem, st>>>(points, n, stride, col0, frame_offsets, nb, gd, ws.table, ws.cap,
                                                  ws.point_slot, ws.point_arrival, vec_ok,
                                                  reinterpret_cast<uint4 *>(ws.zero_begin),
                                                  in_kernel_init ? static_cast<uint32_t>(ws.zero_bytes / 16) : 0u,
                                                  reinterpret_cast<uint4 *>(ws.cell_row),
                                                  in_kernel_init ? static_cast<uint32_t>(map_bytes / 16) : 0u);
    // Tile ids are always handed out in scheduling order (one atomic per CTA): with other streams sharing the GPU nothing
    // guarantees that blockIdx order is dispatch order, and a tile spins on its predecessors.
    const int dynamic_ids = 1;
    if ((err = launch_pdl(k_scan_assign, dim3(ws.n_tiles), dim3(kThreads), 0, st, n, ws.n_tiles,
                          static_cast<const int32_t *>(ws.point_slot), ws.table, ws.hdr, ws.tile_desc, ws.tile_prefix,
                          ws.pillar_key, ws.pillar_list, ws.pillar_cnt, frame_offsets, nb, ws.frame_gstart, dynamic_ids,
                          gd.max_voxels, ws.frame_rowbase, pillar_count)) != cudaSuccess)
        return err;
    note_launch(2);
    if (want_index_lists || extras.records) {
        const PlaceParams pp = make_place_params(points, n, stride, col0, c_point, gd, ws, want_index_lists, extras);
        if ((err = launch_pdl(k_place, dim3(pb), dim3(kThreads), 0, st, pp)) != cudaSuccess) return err;
        note_launch();
    }
    return cudaGetLastError();
}

}  // namespace pillars
