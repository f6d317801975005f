// Shared definitions for libpillars_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <utility>

#include "../../include/pillars_b200.h"

namespace pillars {

// ------------------------------------------------------------------------------------------------
// Pillar hash table (open addressing, linear probing, HBM resident; 16 B entries = half a sector).  Initialised by a single
// 0xFF memset.  The first eight bytes are ONE 64-bit word (key << 32 | first): a point claims an empty slot and records
// itself as the pillar's first point with a single 64-bit atomicCAS; later points of the same cell only issue a 64-bit
// atomicMin when their index is smaller than the one the CAS returned (rare: blocks run roughly in index order).
//   first = 0xFFFFFFFF  -> smallest point index that hit the cell          (low half of the word)
//   key   = 0xFFFFFFFF  -> empty                                           (high half of the word)
//   cnt   = 0xFFFFFFFF  -> "count - 1": atomicAdd(cnt, k) returns old; old + 1 is the arrival rank base;
//                          the scan kernel later replaces it by the start of the pillar's point list
//   gid   = pillar id in first-appearance order over the whole batch (written by the scan kernel)
// ------------------------------------------------------------------------------------------------
struct __align__(16) HashEntry {
    uint32_t first;
    uint32_t key;
    uint32_t cnt;
    uint32_t gid;
};
static constexpr uint32_t kEmptyKey = 0xFFFFFFFFu;

// small zero-initialised header at the start of the workspace
struct Header {
    uint32_t tile_counter;   // dynamic tile ids of the chained scan
    uint32_t total_pillars;  // G: distinct occupied cells over the batch, before the max_voxels cap
    uint32_t total_listed;   // points that fell into some cell (sum of all counts)
    uint32_t tiles_done;     // scan tiles that have finished (the last one turns frame starts into output rows)
    uint32_t ticket_seq;     // dense: tile tickets of the scan kernel; only ever counts up (any start value, wraps)
    uint32_t ticket_base;    // dense: ticket_seq when this call's insert kernel started => tile id = ticket - ticket_base
    uint32_t pad[10];
};

// One point, moved next to the other points of its pillar (32 B = one DRAM sector).
struct __align__(32) PointRecord {
    float x, y, z, intensity, time;  // x,y,z RELATIVE TO THE PILLAR CENTRE (pillar_vfe.py:100-103); missing channels are 0
    uint32_t flags;                  // 0; walk control in the feature kernel's staged copy
    uint32_t idx;                    // index of the point in the input batch
    uint32_t arrival;                // position inside the pillar's list; 0 marks the start of a list
};

static constexpr int kMaxFrames = 1024;  // frame_offsets are staged in shared memory
static constexpr int kTile = 1024;       // points per CTA tile of the scan kernel

// Two grouping implementations fill the same workspace products:
//   kGroupHash   open-addressing hash table keyed by the 32-bit cell key (any grid, voxelize.cu)
//   kGroupDense  direct-mapped table with one entry per (frame, cell) (group_dense.cu); chosen when n_frames * cells is of
//                the order of the point count, which is the case for every pillar grid of the reference's configs
enum GroupMode { kGroupHash = 0, kGroupDense = 1 };

struct Workspace {
    int mode;
    // hash: zero-initialised region.  dense: hdr / frame tables need no initialisation, the tile descriptors live in the
    // 0xFF region (a descriptor is ready when bit 63 is clear)
    Header *hdr;
    unsigned long long *tile_desc;  // [n_tiles] scan: per-tile aggregates (valid bit | pillars | listed points)
    unsigned long long *tile_prefix;// [n_tiles] scan: inclusive prefixes published by the last tile of each group
    uint32_t *frame_gstart;         // [B+1] first-appearance id at each frame start (uncapped, batch-global)
    uint32_t *frame_rowbase;        // [B+1] output row at each frame start (after the max_voxels cap)
    size_t zero_bytes;
    // 0xFF-initialised region
    uint32_t *long_count;           // pillars of more than 32 points listed so far, minus one (counts up from 0xFFFFFFFF)
    uint32_t *long_cursor;          // next entry of that list to be processed by the feature kernel, minus one
    HashEntry *table;               // hash: [cap]
    uint32_t *frame_new;            // dense: [B] pillars opened in each frame, minus one
    uint32_t *cell_first;           // dense: [B * cells] smallest point index of the cell; after the scan 0x80000000 | list base
    int32_t *cell_row;              // BEV index map, -1 = empty.  hash: [B * ny * nx].  dense: [B * cells], holds
                                    // "points in the cell - 1" between the insert and the scan kernel
    size_t ff_bytes;
    // no init needed
    int32_t *point_slot;            // [n] hash: slot of each point; dense: its key b * cells + cell; -1 = rejected
    uint32_t *point_arrival;        // [n] arrival rank inside the cell (arbitrary order, only a bijection)
    uint32_t *pillar_key;           // [n] cell key of pillar g
    uint32_t *pillar_list;          // [n] start of pillar g's point list
    uint32_t *pillar_cnt;           // [n] points that fell into pillar g (uncapped)
    uint32_t *sorted_idx;           // [n] point indices grouped by pillar
    PointRecord *records;           // [n] point records grouped by pillar
    uint4 *pillar_meta;             // [n] per pillar, at its list start position: {x | y << 16, row (-1: dropped), n, z}
    uint4 *long_list;               // [2 * (n / 32 + 2)] pillars of more than 32 points: {list start, n, row, x | y << 16} {z, -, -, -}
    float *folded;                  // [PILLARS_FOLDED_FLOATS] folded PFN table when the caller did not prepare one
    float *folded2;                 // [kFolded2Floats] layer 1 of a two-layer stack, folded
    uint32_t *scan_scratch;         // [B * ny * nx / 2048 + 2] block sums of the cell-rank scan (dynamic variant)
    uint32_t cap;                   // hash slots
    uint32_t n_tiles;
    size_t total_bytes;
    char *zero_begin;
    char *ff_begin;
};

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

template <typename T>
__host__ __device__ __forceinline__ T tmin(T a, T b)
{
    return a < b ? a : b;
}

// The dense table needs n_frames * cells entries: worth it while that stays within a small multiple of the point count
// (16 x 512^2 cells for 0.5 M points at cfg2) and below 2^31 (the base tag bit).
inline bool dense_possible(int64_t n, int nb, int64_t cells)
{
    const int64_t total = static_cast<int64_t>(nb) * cells;
    return n > 0 && total > 0 && total < (1ll << 31);
}
inline bool dense_preferred(int64_t n, int nb, int64_t cells)
{
    return dense_possible(n, nb, cells) && static_cast<int64_t>(nb) * cells <= 16 * n + (1ll << 22);
}

// Carves `base` (may be nullptr to only size it).  n = total points, nb = frames, cells_xy = ny*nx, cells = nz*ny*nx.
inline Workspace carve_workspace(void *base, int64_t n, int nb, int64_t cells_xy, int64_t cells, int mode)
{
    Workspace w{};
    w.mode = mode;
    char *p = reinterpret_cast<char *>(base);
    size_t off = 0;
    auto take = [&](size_t bytes) {
        char *r = p ? p + off : nullptr;
        off += align_up(bytes, 256);
        return r;
    };
    w.n_tiles = static_cast<uint32_t>((n + kTile - 1) / kTile);
    uint64_t cap = static_cast<uint64_t>(n) + static_cast<uint64_t>(n) / 2 + 64;  // load factor <= 2/3 worst case
    w.cap = static_cast<uint32_t>(cap);
    w.zero_begin = p ? p : nullptr;
    if (mode == kGroupHash) {
        w.hdr = reinterpret_cast<Header *>(take(sizeof(Header)));
        w.tile_desc = reinterpret_cast<unsigned long long *>(take(sizeof(unsigned long long) * (w.n_tiles + 1)));
        w.tile_prefix = reinterpret_cast<unsigned long long *>(take(sizeof(unsigned long long) * (w.n_tiles + 1)));
        w.frame_gstart = reinterpret_cast<uint32_t *>(take(sizeof(uint32_t) * (nb + 1)));
        w.frame_rowbase = reinterpret_cast<uint32_t *>(take(sizeof(uint32_t) * (nb + 1)));
        w.zero_bytes = off;
        w.ff_begin = p ? p + off : nullptr;
        const size_t ff0 = off;
        w.long_count = reinterpret_cast<uint32_t *>(take(256));
        w.long_cursor = w.long_count ? w.long_count + 16 : nullptr;
        w.table = reinterpret_cast<HashEntry *>(take(n > 0 ? sizeof(HashEntry) * cap : 0));
        w.cell_row = reinterpret_cast<int32_t *>(take(sizeof(int32_t) * static_cast<size_t>(nb) * cells_xy));
        w.ff_bytes = off - ff0;
    } else {
        w.zero_bytes = 0;
        w.ff_begin = p ? p : nullptr;
        w.long_count = reinterpret_cast<uint32_t *>(take(256));
        w.long_cursor = w.long_count ? w.long_count + 16 : nullptr;
        w.frame_new = reinterpret_cast<uint32_t *>(take(sizeof(uint32_t) * (nb + 1)));
        w.tile_desc = reinterpret_cast<unsigned long long *>(take(sizeof(unsigned long long) * (w.n_tiles + 1)));
        w.tile_prefix = reinterpret_cast<unsigned long long *>(take(sizeof(unsigned long long) * (w.n_tiles + 1)));
        w.cell_first = reinterpret_cast<uint32_t *>(take(sizeof(uint32_t) * static_cast<size_t>(nb) * cells));
        w.cell_row = reinterpret_cast<int32_t *>(take(sizeof(int32_t) * static_cast<size_t>(nb) * cells));
        w.ff_bytes = off;
        w.hdr = reinterpret_cast<Header *>(take(sizeof(Header)));
        w.frame_gstart = reinterpret_cast<uint32_t *>(take(sizeof(uint32_t) * (nb + 1)));
        w.frame_rowbase = reinterpret_cast<uint32_t *>(take(sizeof(uint32_t) * (nb + 1)));
    }
    w.point_slot = reinterpret_cast<int32_t *>(take(sizeof(int32_t) * n));
    w.point_arrival = reinterpret_cast<uint32_t *>(take(sizeof(uint32_t) * n));
    w.pillar_key = reinterpret_cast<uint32_t *>(take(sizeof(uint32_t) * n));
    w.pillar_list = reinterpret_cast<uint32_t *>(take(sizeof(uint32_t) * n));
    w.pillar_cnt = reinterpret_cast<uint32_t *>(take(sizeof(uint32_t) * n));
    w.sorted_idx = reinterpret_cast<uint32_t *>(take(sizeof(uint32_t) * n));
    w.records = reinterpret_cast<PointRecord *>(take(sizeof(PointRecord) * (n + 64)));  // + a look-ahead chunk of slack
    w.pillar_meta = reinterpret_cast<uint4 *>(take(sizeof(uint4) * (n + 64)));
    w.long_list = reinterpret_cast<uint4 *>(take(sizeof(uint4) * 2 * (n / 32 + 2)));
    w.folded = reinterpret_cast<float *>(take(sizeof(float) * PILLARS_FOLDED_FLOATS));
    w.folded2 = reinterpret_cast<float *>(take(sizeof(float) * (2 * 32 * 64 + 64)));
    w.scan_scratch = reinterpret_cast<uint32_t *>(take(sizeof(uint32_t) * (static_cast<size_t>(nb) * cells_xy / 2048 + 2)));
    w.total_bytes = off;
    return w;
}

// bytes that fit either layout (what pillars_workspace_bytes reports)
inline size_t workspace_bytes_any(int64_t n, int nb, int64_t cells_xy, int64_t cells)
{
    size_t b = carve_workspace(nullptr, n, nb, cells_xy, cells, kGroupHash).total_bytes;
    if (dense_possible(n, nb, cells)) {
        const size_t d = carve_workspace(nullptr, n, nb, cells_xy, cells, kGroupDense).total_bytes;
        if (d > b) b = d;
    }
    return b;
}

// Device-side copy of pillars_grid_t plus derived integers.
struct GridDev {
    float rmin[3];
    float vsz[3];
    int32_t g[3];       // nx ny nz
    int32_t max_points;
    int32_t max_voxels;
    uint32_t cells;     // nx*ny*nz
    uint32_t cells_xy;  // nx*ny
    int32_t ignore_z;   // dynamic pillar variant: z is neither range checked nor part of the key (dynamic_pillar_vfe.py:93-96)
};

inline GridDev make_grid_dev(const pillars_grid_t &g)
{
    GridDev d;
    for (int i = 0; i < 3; ++i) {
        d.rmin[i] = g.range[i];
        d.vsz[i] = g.voxel[i];
        d.g[i] = g.grid[i];
    }
    d.max_points = g.max_points;
    d.max_voxels = g.max_voxels;
    d.cells_xy = static_cast<uint32_t>(g.grid[0]) * static_cast<uint32_t>(g.grid[1]);
    d.cells = d.cells_xy * static_cast<uint32_t>(g.grid[2]);
    d.ignore_z = 0;
    return d;
}

struct PfnDev {
    const float *weight;  // [F, C_in]
    const float *scale;   // [F]
    const float *shift;   // [F]
    float off[3];
    float vsz[3];
};

// ---- programmatic dependent launch (sm_90+): the kernels of one call form a chain on one stream; each is launched with
// the attribute below, so its CTAs may be scheduled while the previous kernel drains, and executes pdl_wait() before it
// touches anything a predecessor wrote (griddepcontrol.wait returns once ALL prerequisite grids have completed and their
// writes are visible).  pdl_trigger() lets the next kernel's CTAs start occupying SMs as this grid's CTAs retire.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args)
{
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// ---- measurement hook: nanosecond stamps of kernel phases (pillars_set_debug_times) --------------------------------------
// `dbg` is NULL in normal operation.  Even slots keep the EARLIEST stamp of a phase (stored complemented, so that a zeroed
// buffer works with atomicMax), odd slots the LATEST.
#ifdef __CUDACC__
__device__ __forceinline__ void dbg_stamp(unsigned long long *dbg, int slot)
{
    if (!dbg) return;
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    atomicMax(dbg + slot, (slot & 1) ? t : ~t);
}
#endif
unsigned long long *debug_times_ptr();

// launch bookkeeping (api.cu)
void note_launch(int n = 1);
// SM count of the calling thread's current device (cached per device)
int current_sm_count();

// ---- launchers implemented in the kernel translation units ---------------------------------------
cudaError_t launch_frame_offsets(const float *points_b, int64_t n, int stride, int nb, int32_t *offs, cudaStream_t st);

// What k_place additionally emits for the streaming feature kernel (records == true): point records relative to the pillar
// centre, the per-pillar constants, and the per-pillar outputs that need no feature arithmetic.
struct PlaceExtras {
    bool records;
    float vsz[3], off[3];      // pillar centre = coord * vsz + off (pillar_vfe.py:79-81,101-103)
    int32_t *voxel_coords;     // [capacity,4] or NULL
    int32_t *voxel_num_points; // [capacity] or NULL
    bool write_cell_row;       // fill ws.cell_row for the BEV scatter
    int64_t capacity;
};
cudaError_t launch_group_points(const float *points, int64_t n, int stride, int col0, int c_point,
                                const int32_t *frame_offsets, int nb, const GridDev &gd, const Workspace &ws,
                                int32_t *pillar_count, bool want_index_lists, const PlaceExtras &extras, cudaStream_t st);

// the direct-mapped implementation (group_dense.cu); same products as launch_group_points, chosen by ws.mode
cudaError_t launch_group_points_dense(const float *points, int64_t n, int stride, int col0, int c_point,
                                      const int32_t *frame_offsets, int nb, const GridDev &gd, const Workspace &ws,
                                      int32_t *pillar_count, bool want_index_lists, const PlaceExtras &extras,
                                      cudaStream_t st);

struct FeatureJob {
    const float *points;
    int64_t n;
    int stride;
    int col0;
    int c_point;
    int nb;
    int idx_bits;              // bits needed to hold a point index
    bool use_abs;
    bool with_dist;
    bool do_features;          // run the PFN (needs pfn + pillar_features)
    PfnDev pfn;
    pillars_outputs_t out;     // by value; NULL members are skipped
    bool write_cell_row;       // fill ws.cell_row for the BEV scatter
};
cudaError_t launch_pillar_features(const FeatureJob &job, const GridDev &gd, const Workspace &ws, cudaStream_t st);

struct FastJob {
    int64_t n;  // upper bound of listed points (the input point count)
    int idx_bits;
    float *pillar_features;
    float vsz[3], off[3];  // pillar centre = coord * vsz + off (pillar_vfe.py:79-81,101-103)
    const float *folded2;  // two-layer stack [64, 64]: launch_fold_pfn2's table, else NULL
    bool dynamic;          // DynamicPillarVFE semantics (rows patched into the pillar entries by launch_dynamic_rows)
};
// The streaming feature kernel (pfn_stream.cu) and the folding of one PFN layer into its table:
//   rows 0-4   per point   scale * (W_p + W_cluster + W_centre) for x,y,z;  scale * W for intensity, time
//   rows 5-10  per pillar  scale * W_p (x,y,z) applied to the centre;  -scale * W_cluster applied to (mean - centre)
//   row  11    shift       row 12  relu(shift)
cudaError_t launch_fold_pfn(const PfnDev &pfn, int c_point, int c_in, float *folded, cudaStream_t st, int f_out = 64);
constexpr int kFolded2Floats = 2 * 32 * 64 + 64;
cudaError_t launch_fold_pfn2(const float *weight, const float *scale, const float *shift, float *folded2, cudaStream_t st);
// PillarVFE.forward on padded voxels in the streaming kernel's folded form (configurations stream_kernel_covers accepts)
cudaError_t launch_pfn_padded(const float *voxels, const void *num_points, bool np_float, const void *coords, bool coords_float,
                              int64_t m, int max_points, int c_point, const PfnDev &pfn, const float *folded, float *out,
                              cudaStream_t st);
cudaError_t launch_pillar_features_stream(const FastJob &job, const float *folded, const GridDev &gd, const Workspace &ws,
                                          cudaStream_t st);

cudaError_t launch_pfn_dense(const float *voxels, const void *num_points, bool np_float, const void *coords,
                             bool coords_float, int64_t m, int max_points, int c_point, bool use_abs, bool with_dist,
                             const PfnDev &pfn, float *out, cudaStream_t st);

// ---- general feature stack (pfn_multi.cu) -----------------------------------------------------
struct StackDev {
    int n_layers;          // 1 or 2
    int out[2];            // outputs of each layer's linear
    int use_abs, with_dist;
    int layout;            // 0: [point, cluster, centre(, dist)]   1: [centre, point(, dist)] (DynamicPillarVFESimple2D)
    const float *weight[2], *scale[2], *shift[2];
    float off[3], vsz[3];
};
struct MultiJob {
    const float *points;
    int64_t n;
    int stride, col0, c_point, nb, idx_bits;
    bool dynamic;          // DynamicPillarVFE semantics (rows by sorted key, no caps)
    bool write_cell_row;
    float *pillar_features;
    int32_t *voxel_coords, *voxel_num_points;
    int coords_cols;
    int64_t capacity;
};
int stack_c_in(const StackDev &sd, int c_point);
bool stack_supported(const StackDev &sd, int c_point);
// Dynamic variant, after the grouping: ranks every occupied cell in (b, ix, iy) order (the order torch.unique gives the merged
// key, dynamic_pillar_vfe.py:99-103) into the index-map region of the workspace (entry = rank | occupied << 31).
cudaError_t launch_dynamic_ranks(const GridDev &gd, const Workspace &ws, int nb, int64_t n, cudaStream_t st);
// ... and, for the streaming feature kernel, writes that rank as the row of every pillar entry (0xFFFFFFFF beyond `capacity`)
// together with voxel_coords (b, 0, y, x) and the uncapped voxel_num_points of the row.
cudaError_t launch_dynamic_rows(const GridDev &gd, const Workspace &ws, int nb, int64_t n, int64_t capacity,
                                int32_t *voxel_coords, int32_t *voxel_num_points, cudaStream_t st);
cudaError_t launch_pfn_multi_lists(const MultiJob &job, const StackDev &sd, const GridDev &gd, const Workspace &ws,
                                   cudaStream_t st);
cudaError_t launch_pfn_multi_dense(const float *voxels, const void *num_points, bool np_float, const void *coords,
                                   bool coords_float, int64_t m, int max_points, int c_point, const StackDev &sd,
                                   float *out, cudaStream_t st);

cudaError_t launch_build_cell_row(const void *coords, bool coords_float, int64_t m, const int32_t *m_dev, int nb, int nx,
                                  int ny, int nz, int32_t *cell_row, cudaStream_t st);
// occ_prev / occ_next: the canvas occupancy bitmaps of pillars_set_canvas_occupancy (NULL: none); only the wide kernels
// skip stores, the plain kernel writes everything and sets occ_next to all ones
cudaError_t launch_scatter(const float *feats, const int32_t *cell_row, int nb, int f, int nx, int ny, float *bev,
                           int variant, cudaStream_t st, const uint32_t *occ_prev = nullptr, uint32_t *occ_next = nullptr);
cudaError_t launch_rebase_segments(int32_t *coords, int n_seg, int64_t rows_per_seg, int64_t seg_stride,
                                   const int32_t *seg_counts, int64_t count_stride, int frames_per_seg, int32_t *overflow,
                                   cudaStream_t st);
// float16 canvas (plane % 8 == 0, f % 8 == 0)
cudaError_t launch_scatter_half(const float *feats, const int32_t *cell_row, int nb, int f, int nx, int ny, void *bev,
                                cudaStream_t st, const uint32_t *occ_prev = nullptr, uint32_t *occ_next = nullptr);

// ---- BEV tokeniser (tokens.cu): head of VATLiDAR.forward, src/encoder-decoder/training/models/vat_lidar.py:206-253 ----
struct TokenizerDev {
    int c, d;
    const float *dw_w, *dw_b;  // [c, 9], [c]
    const float *wt, *pb;      // [c, d] (transposed projection), [d]
    const float *gamma, *beta; // LayerNorm
    float eps;
    const float *pe, *bg;      // [h*w, d], [d]
    const float *wimg;         // [2 * c * d] projection as the tcgen05 shared-memory image (tf32 hi | lo, swizzled), or NULL
};
bool tokens_shape_supported(int c, int d);
bool tokens_umma_supported(int c, int d);
cudaError_t launch_tokens_wimg(const float *wt, int c, int d, float *img, cudaStream_t st);
cudaError_t launch_bev_tokens_umma(const TokenizerDev &tk, const float *feats, const int32_t *cell_row, int nb, int h, int w,
                                   float *out, uint32_t *list, uint32_t *count, cudaStream_t st);
cudaError_t launch_tokens_prepare(const TokenizerDev &tk, const float *geom, const int32_t *sid, int h, int w, const float *w1,
                                  const float *b1, const float *w2t, const float *b2, const float *view, float *pe, float *bg,
                                  cudaStream_t st);
// One convolution layer of the BEV backbone (conv_umma.cu)
struct ConvJob {
    const float *in;           // NHWC [nb, h_in, w_in, c_in], or NULL when the input is gathered:
    const float *rows;         // [M, c_in] pillar rows + cell_row [nb, h_in, w_in] (-1 = empty cell)
    const int32_t *cell_row;
    const void *wimg;          // launch_conv_wimg's image
    const float *shift;        // [c_out]
    float *out;
    int nb, h_in, w_in, c_in, c_out;
    int k, stride, pad;        // (3,1,1) (3,2,1) (2,2,0) (1,1,0) (1,2,0)
    int up;                    // 1, or 2 = transposed convolution with kernel = stride = 2 (k = 1 per phase)
    int out_c_total, out_c_off, out_nchw;
    int relu, round_out;       // round_out: store tf32-rounded values (the next layer's tensor cores would truncate them)
    uint32_t *error;
    const float *res;          // NULL, or the residual added before the ReLU: NHWC fp32 laid out like out (out_nchw == 0, up == 1)
};
cudaError_t launch_conv_wimg(const float *weight, const float *scale, int c_in, int c_out, int k, int up, float *img, cudaStream_t st);
cudaError_t launch_conv_umma(const ConvJob &job, cudaStream_t st);
cudaError_t launch_canvas_to_rows(const float *bev, int nb, int c, int h, int w, int32_t *cell_row, float *rows,
                                  uint32_t *counter, cudaStream_t st);
cudaError_t launch_bev_tokens(const TokenizerDev &tk, const float *feats, const int32_t *cell_row, int nb, int h, int w,
                              float *out, cudaStream_t st);

}  // namespace pillars
