// Dense BEV canvas in "gather form" (replaces PointPillarScatter.forward,
// src/lidar-encoder/pcdet/models/backbones_2d/map_to_bev/pointpillar_scatter.py:14-37).
//
// The reference zero-fills a [F, ny*nx] canvas per frame, index-assigns F strided 4-byte columns per pillar and then
// stacks the frames (a third full pass).  Here a dense index map cell -> pillar row (4 B per cell, written by the
// grouping stage or by k_build_cell_row) turns the scatter inside out: every output element is written exactly once,
// in NCHW order, with full-line stores, zero-fill included, no atomics.
//
// On a canvas the library wrote before, most of those stores put zeros over zeros.  The caller then passes two occupancy
// bitmaps (layout in include/pillars_b200.h, pillars_set_canvas_occupancy): bit = "these 8 cells of the frame may be
// non-zero".  With the previous bitmap, k_scatter_sparse reads the index map once and writes only the 8-cell groups that
// are occupied now or were last time (zeros where only the old bit is set); every other canvas element already holds its
// zero.  The store unit stays one 32-byte sector, so no sector is ever written in part.  Without it (fresh or invalidated
// canvas) the full-write kernels run and record the next bitmap.
//
// Full writes: the channel-group 256-bit store kernel (k_scatter_wide, 99 % of the measured copy peak) and a plain
// kernel for shapes it does not cover (odd plane sizes, unaligned canvases, F not a multiple of 8).  The other store paths
// that were measured and lost (bulk 1-D copies, TMA tile stores, persistent warps, zero-fill + patches) are kept as
// evidence, out of the product library: profiles/micro/r01_scatter_variants.cu.txt, numbers in
// profiles/r01_scatter_variants.md.
#include <cuda_fp16.h>

#include "common.cuh"

namespace pillars {

namespace {

constexpr int kThreads = 256;

__global__ void k_build_cell_row(const void *__restrict__ coords, int coords_float, int64_t m,
                                 const int32_t *__restrict__ m_dev, int nb, int nx, int ny, int nz,
                                 int32_t *__restrict__ cell_row)
{
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    int64_t live = m;
    if (m_dev) live = tmin<int64_t>(m, static_cast<int64_t>(*m_dev));
    if (i >= live) return;
    int b, z, y, x;
    if (coords_float) {
        const float4 c = *reinterpret_cast<const float4 *>(static_cast<const float *>(coords) + i * 4);
        b = static_cast<int>(c.x); z = static_cast<int>(c.y); y = static_cast<int>(c.z); x = static_cast<int>(c.w);
    } else {
        const int4 c = *reinterpret_cast<const int4 *>(static_cast<const int32_t *>(coords) + i * 4);
        b = c.x; z = c.y; y = c.z; x = c.w;
    }
    // pointpillar_scatter.py:27  index = z + y*nx + x (nz == 1, so z == 0);  :63  index = z*ny*nx + y*nx + x (3-D variant)
    const int64_t plane = static_cast<int64_t>(nx) * ny * nz;
    const int64_t cell = nz > 1 ? (static_cast<int64_t>(z) * ny + y) * nx + x : static_cast<int64_t>(z) + static_cast<int64_t>(y) * nx + x;
    if (b < 0 || b >= nb || cell < 0 || cell >= plane || x < 0 || x >= nx) return;
    atomicMax(cell_row + static_cast<int64_t>(b) * plane + cell, static_cast<int32_t>(i));  // later row wins
}

// Gathered compact BEV tokens of several ranks lie in equal-sized segments of `rows_per_seg` rows (segment s starts
// `seg_stride` int32 elements after segment s - 1); segment s holds seg_counts[s * count_stride] live rows whose frame
// indices are local to its rank.  Live rows get the segment's frame base added, the padding rows get frame -1 (every
// consumer of voxel_coords skips those).  A count beyond the segment's capacity raises *overflow.
__global__ void k_rebase_segments(int32_t *__restrict__ coords, int n_seg, int64_t rows_per_seg, int64_t seg_stride,
                                  const int32_t *__restrict__ seg_counts, int64_t count_stride, int frames_per_seg,
                                  int32_t *__restrict__ overflow)
{
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= rows_per_seg * n_seg) return;
    const int seg = static_cast<int>(i / rows_per_seg);
    const int64_t r = i - seg * rows_per_seg;
    const int32_t cnt = __ldg(seg_counts + static_cast<int64_t>(seg) * count_stride);
    int32_t *b = coords + seg * seg_stride + r * 4;
    if (r < cnt) *b += seg * frames_per_seg;
    else *b = -1;
    if (r == 0 && cnt > rows_per_seg && overflow) *overflow = 1;
}

// ---- variant 1 ----------------------------------------------------------------------------------
// Warp-autonomous direct stores: a warp owns 128 consecutive cells (4 per lane) x all channels = 32 KB of the canvas and
// never waits for another warp.  A warp whose 128 cells are empty streams zeros; otherwise each lane fetches, 8 channels
// at a time, the feature rows of its occupied cells with two 16-byte loads per row and composes one float4 per channel.
// Eight passes of one L2 round trip each per 32 KB keep the SM far above its share of HBM write bandwidth with a handful
// of resident warps, so the kernel runs at the speed of the write stream.
template <bool VEC>
__global__ void __launch_bounds__(kThreads)
k_scatter_plain(const float *__restrict__ feats, const int32_t *__restrict__ cell_row, int f, int64_t plane,
                int tiles_per_plane, float *__restrict__ bev)
{
    constexpr int kPer = VEC ? 4 : 1;
    const int b = blockIdx.x / tiles_per_plane;
    const int64_t cell0 = static_cast<int64_t>(blockIdx.x % tiles_per_plane) * (blockDim.x * kPer) + threadIdx.x * kPer;
    const bool inb = cell0 < plane;
    int32_t r[kPer];
#pragma unroll
    for (int k = 0; k < kPer; ++k) r[k] = -1;
    if (inb) {
        if (VEC) {
            const int4 v = __ldg(reinterpret_cast<const int4 *>(cell_row + b * plane + cell0));
            r[0] = v.x; r[1 % kPer] = v.y; r[2 % kPer] = v.z; r[3 % kPer] = v.w;
        } else {
            r[0] = __ldg(cell_row + b * plane + cell0);
        }
    }
    bool any = false;
#pragma unroll
    for (int k = 0; k < kPer; ++k) any |= r[k] >= 0;
    float *dst = bev + (static_cast<int64_t>(b) * f) * plane + cell0;
    if (!__any_sync(0xffffffffu, any)) {
        if (inb) {
            if (VEC) {
#pragma unroll 8
                for (int c = 0; c < f; ++c) __stcs(reinterpret_cast<float4 *>(dst + c * plane), make_float4(0.f, 0.f, 0.f, 0.f));
            } else {
                for (int c = 0; c < f; ++c) __stcs(dst + c * plane, 0.f);
            }
        }
        return;
    }
    if (!inb) return;
    if (VEC) {
        constexpr int kV = 2;  // 16-byte loads per row and pass of 8 channels
        float4 cur[4][kV];
        auto fetch = [&](float4 (&dstv)[4][kV], int c0) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
#pragma unroll
                for (int q = 0; q < kV; ++q) dstv[k][q] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r[k % kPer] >= 0) {
                    const float4 *row = reinterpret_cast<const float4 *>(feats + static_cast<int64_t>(r[k % kPer]) * f + c0);
#pragma unroll
                    for (int q = 0; q < kV; ++q) dstv[k][q] = __ldg(row + q);
                }
            }
        };
        fetch(cur, 0);
        for (int c0 = 0; c0 < f; c0 += 8) {
#pragma unroll
            for (int q = 0; q < kV; ++q) {
                __stcs(reinterpret_cast<float4 *>(dst + (c0 + 4 * q + 0) * plane), make_float4(cur[0][q].x, cur[1][q].x, cur[2][q].x, cur[3][q].x));
                __stcs(reinterpret_cast<float4 *>(dst + (c0 + 4 * q + 1) * plane), make_float4(cur[0][q].y, cur[1][q].y, cur[2][q].y, cur[3][q].y));
                __stcs(reinterpret_cast<float4 *>(dst + (c0 + 4 * q + 2) * plane), make_float4(cur[0][q].z, cur[1][q].z, cur[2][q].z, cur[3][q].z));
                __stcs(reinterpret_cast<float4 *>(dst + (c0 + 4 * q + 3) * plane), make_float4(cur[0][q].w, cur[1][q].w, cur[2][q].w, cur[3][q].w));
            }
            if (c0 + 8 < f) fetch(cur, c0 + 8);
        }
    } else {
        for (int c = 0; c < f; ++c) __stcs(dst + c * plane, r[0] >= 0 ? __ldg(feats + static_cast<int64_t>(r[0]) * f + c) : 0.f);
    }
}

// ---- occupancy bitmaps ------------------------------------------------------------------------------
// One bit per 8 cells, one word per 256 cells (a warp of the wide kernels), words_per_frame = ceil(plane / 256).
__host__ __device__ __forceinline__ int64_t occ_words(int64_t plane) { return (plane + 255) >> 8; }

// ---- variant 4 ----------------------------------------------------------------------------------
// Same warp-autonomous scheme with 256-bit accesses (sm_100: LDG.256 / STG.256): a lane owns 8 consecutive cells, a warp
// 256 cells x all channels = 64 KB of the canvas, and every store instruction of the warp writes 1 KB contiguous.  Half the
// LSU instructions of variant 1 for the same bytes.
__device__ __forceinline__ void stg256(float *p, float a, float b, float c, float d, float e, float f, float g, float h)
{
    asm volatile("st.global.L1::no_allocate.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(a), "f"(b), "f"(c),
                 "f"(d), "f"(e), "f"(f), "f"(g), "f"(h)
                 : "memory");
}

// Work split: a CTA owns blockDim.x * 8 consecutive cells x `chan_per_cta` channels (a multiple of 8; every launch uses 8).
// With 8 channels per CTA the canvas is written as few long sequential streams (measured with
// profiles/micro/fill_patterns.cu on B200: 64 channel-strided streams per thread 164 us for the 1 GiB canvas, 8 channels x
// 8 KB runs per CTA 149 us, linear fill 146 us); the CTAs of one cell tile then each read one 32-byte sector of every
// pillar row, so no feature byte is fetched twice.
// tile_major != 0: consecutive CTAs are the channel groups of one cell tile (index map and feature rows are shared by CTAs
// that run together); 0: consecutive CTAs walk the plane for one channel group.
// occ_next != NULL: the channel group 0 CTAs record each lane's "any cell occupied" test into occ_next.
// chan_per_cta and tile_major stay runtime parameters: with both folded to constants (8, 0) the invalidated cfg2 canvas
// took 173.1 us against 171.0-171.1 us, in 4 alternated rounds on one B200 at 1000 W (same loads and stores, scheduled
// differently); cfg4 was unchanged.
__global__ void __launch_bounds__(kThreads)
k_scatter_wide(const float *__restrict__ feats, const int32_t *__restrict__ cell_row, int f, int64_t plane,
               int tiles_per_plane, int chan_per_cta, int tile_major, float *__restrict__ bev, uint32_t *__restrict__ occ_next)
{
    pdl_wait();  // feature rows and index map come from the kernels before this one
    const int groups = f / chan_per_cta;
    int b, tile, cg;
    if (tile_major) {
        cg = blockIdx.x % groups;
        tile = (blockIdx.x / groups) % tiles_per_plane;
        b = blockIdx.x / (groups * tiles_per_plane);
    } else {
        tile = blockIdx.x % tiles_per_plane;
        cg = (blockIdx.x / tiles_per_plane) % groups;
        b = blockIdx.x / (groups * tiles_per_plane);
    }
    const int64_t cell0 = static_cast<int64_t>(tile) * (blockDim.x * 8) + threadIdx.x * 8;
    const bool inb = cell0 < plane;  // plane % 8 == 0: a lane is entirely inside or outside
    int32_t r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = -1;
    if (inb) {
        const int4 *src = reinterpret_cast<const int4 *>(cell_row + b * plane + cell0);
        const int4 v = __ldg(src), w = __ldg(src + 1);
        r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
        r[4] = w.x; r[5] = w.y; r[6] = w.z; r[7] = w.w;
    }
    bool any = false;
#pragma unroll
    for (int k = 0; k < 8; ++k) any |= r[k] >= 0;
    const int c_begin = cg * chan_per_cta, c_end = c_begin + chan_per_cta;
    float *dst = bev + (static_cast<int64_t>(b) * f) * plane + cell0;
    const uint32_t now = __ballot_sync(0xffffffffu, any);
    if (occ_next && cg == 0 && (threadIdx.x & 31) == 0 && inb) occ_next[b * occ_words(plane) + (cell0 >> 8)] = now;
    if (!inb) return;
    if (now == 0) {
#pragma unroll 8
        for (int c = c_begin; c < c_end; ++c) stg256(dst + c * plane, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f);
        return;
    }
    constexpr int kV = 2;  // 16-byte loads per row and pass of 8 channels
    for (int c0 = c_begin; c0 < c_end; c0 += 8) {
        float4 v[8][kV];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
#pragma unroll
            for (int q = 0; q < kV; ++q) v[k][q] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r[k] >= 0) {
                const float4 *row = reinterpret_cast<const float4 *>(feats + static_cast<int64_t>(r[k]) * f + c0);
#pragma unroll
                for (int q = 0; q < kV; ++q) v[k][q] = __ldg(row + q);
            }
        }
#pragma unroll
        for (int q = 0; q < kV; ++q) {
            float *d = dst + (c0 + 4 * q) * plane;
            stg256(d, v[0][q].x, v[1][q].x, v[2][q].x, v[3][q].x, v[4][q].x, v[5][q].x, v[6][q].x, v[7][q].x);
            stg256(d + plane, v[0][q].y, v[1][q].y, v[2][q].y, v[3][q].y, v[4][q].y, v[5][q].y, v[6][q].y, v[7][q].y);
            stg256(d + 2 * plane, v[0][q].z, v[1][q].z, v[2][q].z, v[3][q].z, v[4][q].z, v[5][q].z, v[6][q].z, v[7][q].z);
            stg256(d + 3 * plane, v[0][q].w, v[1][q].w, v[2][q].w, v[3][q].w, v[4][q].w, v[5][q].w, v[6][q].w, v[7][q].w);
        }
    }
}

__device__ __forceinline__ void ldg256_stream(const float *p, float (&v)[8])
{
    asm volatile("ld.global.nc.L1::no_allocate.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                 : "l"(p));
}

// ---- fp16 canvas ---------------------------------------------------------------------------------
// The product's caller stores the BEV map as float16 (src/get-data/precompute_bev_features.py:394: bev.astype(np.float16));
// converting in the scatter halves the dominant write.  Same work split as variant 4: a lane owns 8 cells = one 16-byte
// store per channel, round-to-nearest-even like numpy / torch.
__global__ void __launch_bounds__(kThreads)
k_scatter_wide_half(const float *__restrict__ feats, const int32_t *__restrict__ cell_row, int f, int64_t plane,
                    int tiles_per_plane, __half *__restrict__ bev, uint32_t *__restrict__ occ_next)
{
    const int groups = f >> 3;
    const int tile = blockIdx.x % tiles_per_plane;
    const int cg = (blockIdx.x / tiles_per_plane) % groups;
    const int b = blockIdx.x / (groups * tiles_per_plane);
    const int64_t cell0 = static_cast<int64_t>(tile) * (blockDim.x * 8) + threadIdx.x * 8;
    const bool inb = cell0 < plane;
    int32_t r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = -1;
    if (inb) {
        const int4 *src = reinterpret_cast<const int4 *>(cell_row + b * plane + cell0);
        const int4 v = __ldg(src), w = __ldg(src + 1);
        r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
        r[4] = w.x; r[5] = w.y; r[6] = w.z; r[7] = w.w;
    }
    bool any = false;
#pragma unroll
    for (int k = 0; k < 8; ++k) any |= r[k] >= 0;
    const int c0 = cg * 8;
    __half *dst = bev + (static_cast<int64_t>(b) * f + c0) * plane + cell0;
    const uint32_t now = __ballot_sync(0xffffffffu, any);
    if (occ_next && cg == 0 && (threadIdx.x & 31) == 0 && inb) occ_next[b * occ_words(plane) + (cell0 >> 8)] = now;
    if (!inb) return;
    if (now == 0) {
#pragma unroll
        for (int c = 0; c < 8; ++c) __stcs(reinterpret_cast<uint4 *>(dst + c * plane), make_uint4(0u, 0u, 0u, 0u));
        return;
    }
    float v[8][8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
#pragma unroll
        for (int c = 0; c < 8; ++c) v[k][c] = 0.f;
        if (r[k] >= 0) ldg256_stream(feats + static_cast<int64_t>(r[k]) * f + c0, v[k]);
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        uint4 o;
        __half2 h;
        h = __floats2half2_rn(v[0][c], v[1][c]); o.x = *reinterpret_cast<uint32_t *>(&h);
        h = __floats2half2_rn(v[2][c], v[3][c]); o.y = *reinterpret_cast<uint32_t *>(&h);
        h = __floats2half2_rn(v[4][c], v[5][c]); o.z = *reinterpret_cast<uint32_t *>(&h);
        h = __floats2half2_rn(v[6][c], v[7][c]); o.w = *reinterpret_cast<uint32_t *>(&h);
        *reinterpret_cast<uint4 *>(dst + c * plane) = o;
    }
}

// ---- reused canvas: dirty groups only -------------------------------------------------------------
// With occ_prev, every canvas element outside prev's groups already holds its zero, so only the 8-cell groups of
// prev | now need stores.  A CTA owns a span of kSparseWarps bitmap words (256 cells each) of one frame, all channels:
//  1. each warp takes one word: prev (loaded before pdl_wait), the index map of its 256 cells (a lane = one group, two
//     16-byte loads), now = ballot of "any cell occupied", recorded into occ_next.  The groups of now | prev store their
//     8 row indices (-1 = empty cell) and position, in cell order, in the warp's part of a shared list;
//  2. the CTA walks the items (dirty group, 8-channel chunk), chunk by chunk, so that a warp's stores go to one channel
//     plane, close together.  A lane loads the group's rows (one 32-byte sector each, nothing for an empty cell) and
//     stores 8 channels x 8 cells: 8 STG.256, or 8 16-byte stores on the float16 canvas.
// The index map is read once, not once per channel group, and a clean empty group costs nothing more.  On the float16
// canvas a lane's 16 bytes are half a sector: the lane pairs are dirty together (pair-closed masks keep both halves in
// adjacent list slots at even offsets, so one warp store instruction writes both).  A pair is one 32-byte sector when
// the canvas is 32-byte aligned and the plane a multiple of 16 cells (the bench's shapes); otherwise pairs straddle
// sectors, which costs speed, not correctness.  Both canvases launch it with PDL (the float16 full-write kernel keeps
// its plain launch).
// Span: 1024 cells.  The dirty groups are unevenly spread over the plane; short CTAs balance them over the SMs, and the
// grid (cfg1: 256 CTAs, cfg2: 4096, cfg4: 8192; 5 fit on an SM at 96 registers x 128 threads, 4 of the float16 kernel at
// 98) leaves SMs free for a concurrent stream's grouping as it drains.  Longer spans (2, 4 or 8 words per warp) were
// measured and are slower: cfg2 105k / 101k sweeps/s at 2 / 4 words against 107k; cfg4 cycling batches 243 us at 2 words
// against 229 us (B200; profiles/r04_ab.txt, r04_scatter_sparse.json).
constexpr int kSparseWarps = 4;

template <bool HALF>
__global__ void __launch_bounds__(kSparseWarps * 32)
k_scatter_sparse(const float *__restrict__ feats, const int32_t *__restrict__ cell_row, int f, int64_t plane,
                 int spans_per_plane, void *__restrict__ bev, const uint32_t *__restrict__ occ_prev,
                 uint32_t *__restrict__ occ_next)
{
    constexpr int kGroups = kSparseWarps * 32;
    __shared__ int4 s_rows[2 * kGroups];
    __shared__ int32_t s_cell[kGroups];  // the group's first cell, relative to the span
    __shared__ int s_count[kSparseWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.x / spans_per_plane;
    const int64_t words = occ_words(plane);
    const int64_t span_word = static_cast<int64_t>(blockIdx.x % spans_per_plane) * kSparseWarps;
    const int64_t word = span_word + warp;
    // the previous call on this canvas wrote occ_prev and finished before this call's first (non-PDL) launch
    const uint32_t prev = word < words ? __ldg(occ_prev + b * words + word) : 0u;
    pdl_wait();  // feature rows and index map come from the kernels before this one
    const int64_t cell0 = word * 256 + lane * 8;
    const bool inb = cell0 < plane;  // plane % 8 == 0: a lane is entirely inside or outside
    int4 v = make_int4(-1, -1, -1, -1), w = v;
    if (inb) {
        const int4 *src = reinterpret_cast<const int4 *>(cell_row + b * plane + cell0);
        v = __ldg(src);
        w = __ldg(src + 1);
    }
    const bool any = (v.x & v.y & v.z & v.w & w.x & w.y & w.z & w.w) >= 0;  // some row index is not -1
    const uint32_t now = __ballot_sync(0xffffffffu, any);
    if (lane == 0 && word < words) occ_next[b * words + word] = now;
    uint32_t dirty = now | prev;
    if (HALF) dirty |= ((dirty >> 1) & 0x55555555u) | ((dirty & 0x55555555u) << 1);
    dirty &= __ballot_sync(0xffffffffu, inb);
    if ((dirty >> lane) & 1u) {
        const int s = warp * 32 + __popc(dirty & ((1u << lane) - 1u));
        s_rows[2 * s] = v;
        s_rows[2 * s + 1] = w;
        s_cell[s] = static_cast<int>(cell0 - span_word * 256);
    }
    const int n = __popc(dirty);
    if (lane == 0) s_count[warp] = n;
    __syncthreads();
    int off[kSparseWarps];  // list position of each warp's first group
    off[0] = 0;
#pragma unroll
    for (int k = 1; k < kSparseWarps; ++k) off[k] = off[k - 1] + s_count[k - 1];
    const int total = off[kSparseWarps - 1] + s_count[kSparseWarps - 1];
    const int items = total * (f >> 3);
    const int64_t span_base = static_cast<int64_t>(b) * f * plane + span_word * 256;
    for (int i = threadIdx.x; i < items; i += blockDim.x) {
        const int chunk = i / total, g = i - chunk * total;
        int s = g;
#pragma unroll
        for (int k = 1; k < kSparseWarps; ++k)
            if (g >= off[k]) s = k * 32 + g - off[k];
        const int4 v = s_rows[2 * s], w = s_rows[2 * s + 1];
        const int r[8] = {v.x, v.y, v.z, v.w, w.x, w.y, w.z, w.w};
        const int c0 = chunk * 8;
        float x[8][8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
#pragma unroll
            for (int c = 0; c < 8; ++c) x[k][c] = 0.f;
            if (r[k] >= 0) ldg256_stream(feats + static_cast<int64_t>(r[k]) * f + c0, x[k]);
        }
        const int64_t at = span_base + static_cast<int64_t>(c0) * plane + s_cell[s];
        if (HALF) {
            __half *dst = static_cast<__half *>(bev) + at;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                uint4 o;
                __half2 h;
                h = __floats2half2_rn(x[0][c], x[1][c]); o.x = *reinterpret_cast<uint32_t *>(&h);
                h = __floats2half2_rn(x[2][c], x[3][c]); o.y = *reinterpret_cast<uint32_t *>(&h);
                h = __floats2half2_rn(x[4][c], x[5][c]); o.z = *reinterpret_cast<uint32_t *>(&h);
                h = __floats2half2_rn(x[6][c], x[7][c]); o.w = *reinterpret_cast<uint32_t *>(&h);
                *reinterpret_cast<uint4 *>(dst + c * plane) = o;
            }
        } else {
            float *dst = static_cast<float *>(bev) + at;
#pragma unroll
            for (int c = 0; c < 8; ++c)
                stg256(dst + c * plane, x[0][c], x[1][c], x[2][c], x[3][c], x[4][c], x[5][c], x[6][c], x[7][c]);
        }
    }
}

}  // namespace

cudaError_t launch_build_cell_row(const void *coords, bool coords_float, int64_t m, const int32_t *m_dev, int nb, int nx,
                                  int ny, int nz, int32_t *cell_row, cudaStream_t st)
{
    cudaError_t err = cudaMemsetAsync(cell_row, 0xFF, sizeof(int32_t) * static_cast<size_t>(nb) * nx * ny * nz, st);
    note_launch();
    if (err != cudaSuccess || m == 0) return err;
    const unsigned blocks = static_cast<unsigned>((m + kThreads - 1) / kThreads);
    k_build_cell_row<<<blocks, kThreads, 0, st>>>(coords, coords_float ? 1 : 0, m, m_dev, nb, nx, ny, nz, cell_row);
    note_launch();
    return cudaGetLastError();
}

cudaError_t launch_rebase_segments(int32_t *coords, int n_seg, int64_t rows_per_seg, int64_t seg_stride,
                                   const int32_t *seg_counts, int64_t count_stride, int frames_per_seg, int32_t *overflow,
                                   cudaStream_t st)
{
    const int64_t total = rows_per_seg * n_seg;
    if (total == 0) return cudaSuccess;
    k_rebase_segments<<<static_cast<unsigned>((total + kThreads - 1) / kThreads), kThreads, 0, st>>>(
        coords, n_seg, rows_per_seg, seg_stride, seg_counts, count_stride, frames_per_seg, overflow);
    note_launch();
    return cudaGetLastError();
}

// k_scatter_sparse for a canvas with a previous bitmap (needs plane % 8 == 0, f % 8 == 0, 32-byte aligned feature rows
// and a canvas aligned to its store unit).
template <bool HALF>
cudaError_t launch_scatter_sparse(const float *feats, const int32_t *cell_row, int nb, int f, int64_t plane, void *bev,
                                  cudaStream_t st, const uint32_t *occ_prev, uint32_t *occ_next)
{
    const int spp = static_cast<int>((occ_words(plane) + kSparseWarps - 1) / kSparseWarps);
    const cudaError_t err = launch_pdl(k_scatter_sparse<HALF>, dim3(static_cast<unsigned>(nb) * spp), dim3(kSparseWarps * 32),
                                       0, st, feats, cell_row, f, plane, spp, bev, occ_prev, occ_next);
    if (err != cudaSuccess) return err;
    note_launch();
    return cudaGetLastError();
}

cudaError_t launch_scatter_half(const float *feats, const int32_t *cell_row, int nb, int f, int nx, int ny, void *bev,
                                cudaStream_t st, const uint32_t *occ_prev, uint32_t *occ_next)
{
    const int64_t plane = static_cast<int64_t>(nx) * ny;
    if (nb == 0 || plane == 0 || f == 0) return cudaSuccess;
    if (plane % 8 != 0 || f % 8 != 0 || reinterpret_cast<uintptr_t>(bev) % 16 != 0 ||
        reinterpret_cast<uintptr_t>(feats) % 32 != 0)
        return cudaErrorInvalidValue;
    if (occ_prev) return launch_scatter_sparse<true>(feats, cell_row, nb, f, plane, bev, st, occ_prev, occ_next);
    const int bs = 128;
    const int tpp = static_cast<int>((plane + bs * 8 - 1) / (bs * 8));
    const unsigned grid = static_cast<unsigned>(nb) * tpp * (f / 8);
    k_scatter_wide_half<<<grid, bs, 0, st>>>(feats, cell_row, f, plane, tpp, static_cast<__half *>(bev), occ_next);
    note_launch();
    return cudaGetLastError();
}
cudaError_t launch_scatter(const float *feats, const int32_t *cell_row, int nb, int f, int nx, int ny, float *bev,
                           int variant, cudaStream_t st, const uint32_t *occ_prev, uint32_t *occ_next)
{
    const int64_t plane = static_cast<int64_t>(nx) * ny;
    if (nb == 0 || plane == 0 || f == 0) return cudaSuccess;
    const bool vec_ok = (plane % 4 == 0) && (reinterpret_cast<uintptr_t>(bev) % 16 == 0) &&
                        (reinterpret_cast<uintptr_t>(feats) % 16 == 0) && (f % 8 == 0);
    const bool wide_ok = vec_ok && (plane % 8 == 0) && (reinterpret_cast<uintptr_t>(bev) % 32 == 0);
    // measured on B200, cfg2 (profiles/r01_scatter_variants.md): channel-group 256-bit stores 172 us, direct stores with all
    // channels per warp 203 us
    if (variant != 1 && wide_ok && occ_prev && reinterpret_cast<uintptr_t>(feats) % 32 == 0)
        return launch_scatter_sparse<false>(feats, cell_row, nb, f, plane, bev, st, occ_prev, occ_next);
    if (variant != 1 && wide_ok) {
        // a CTA owns 128 lanes x 8 cells x 8 channels: few long sequential write streams per CTA
        constexpr int bs = 128, chan = 8;
        const int tpp = static_cast<int>((plane + bs * 8 - 1) / (bs * 8));
        const unsigned grid = static_cast<unsigned>(nb) * tpp * (f / chan);
        const cudaError_t err = launch_pdl(k_scatter_wide, dim3(grid), dim3(bs), 0, st, feats, cell_row, f, plane, tpp, chan,
                                           0, bev, occ_next);
        if (err != cudaSuccess) return err;
        note_launch();
        return cudaGetLastError();
    }
    // the plain kernel writes the whole canvas: the next call on it must not skip anything ("all dirty")
    if (occ_next) {
        const cudaError_t err = cudaMemsetAsync(occ_next, 0xFF, sizeof(uint32_t) * nb * occ_words(plane), st);
        if (err != cudaSuccess) return err;
        note_launch();
    }
    if (vec_ok) {
        const int tpp = static_cast<int>((plane + kThreads * 4 - 1) / (kThreads * 4));
        k_scatter_plain<true><<<static_cast<unsigned>(nb) * tpp, kThreads, 0, st>>>(feats, cell_row, f, plane, tpp, bev);
    } else {
        const int tpp = static_cast<int>((plane + kThreads - 1) / kThreads);
        k_scatter_plain<false><<<static_cast<unsigned>(nb) * tpp, kThreads, 0, st>>>(feats, cell_row, f, plane, tpp, bev);
    }
    note_launch();
    return cudaGetLastError();
}

}  // namespace pillars
