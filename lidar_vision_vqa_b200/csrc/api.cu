// extern "C" surface of libpillars_b200.so (see include/pillars_b200.h for the contract and the reference lines each
// entry point replaces).  Argument checking, workspace carving and kernel sequencing only -- no compute on the host.
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "common.cuh"

namespace pillars {

static thread_local char g_err[512] = "";
static thread_local int g_launches = 0;
static thread_local int g_launches_last = 0;
static thread_local cudaEvent_t g_stage_ev[4] = {nullptr, nullptr, nullptr, nullptr};
static thread_local bool g_stage_on = false;

// canvas occupancy bitmaps for the next pillars_encode_bev / pillars_encode_stack on this thread (one-shot)
struct CanvasOccupancy {
    const uint32_t *prev = nullptr;
    uint32_t *next = nullptr;
};
static thread_local CanvasOccupancy g_occ;

static CanvasOccupancy take_canvas_occupancy()
{
    const CanvasOccupancy o = g_occ;
    g_occ = CanvasOccupancy{};
    return o;
}

static void stage_mark(int i, cudaStream_t st)
{
    if (g_stage_on && g_stage_ev[i]) cudaEventRecord(g_stage_ev[i], st);
}

void note_launch(int n) { g_launches += n; }

static thread_local unsigned long long *g_dbg_times = nullptr;
unsigned long long *debug_times_ptr() { return g_dbg_times; }

int current_sm_count()
{
    static thread_local int cache[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev >= 0 && dev < 64 && cache[dev]) return cache[dev];
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    if (dev >= 0 && dev < 64) cache[dev] = sms;
    return sms;
}

// grouping implementation: 0 = automatic, 1 = hash table, 2 = direct-mapped table whenever it is possible
static thread_local int g_grouping = 0;

static int resolve_group_mode(bool allow_dense, int64_t n, int nb, int64_t cells)
{
    if (!allow_dense || g_grouping == 1) return kGroupHash;
    if (g_grouping == 2) return dense_possible(n, nb, cells) ? kGroupDense : kGroupHash;
    return dense_preferred(n, nb, cells) ? kGroupDense : kGroupHash;
}

static int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

static int cuda_fail(cudaError_t e, const char *where)
{
    snprintf(g_err, sizeof(g_err), "%s: %s (%s)", where, cudaGetErrorName(e), cudaGetErrorString(e));
    return static_cast<int>(e);
}

static int check_grid(const pillars_grid_t *g, int nb)
{
    if (!g) return fail(PILLARS_E_BADARG, "grid is NULL");
    for (int i = 0; i < 3; ++i) {
        if (g->grid[i] < 1) return fail(PILLARS_E_BADARG, "grid[%d] = %d", i, g->grid[i]);
        if (!(g->voxel[i] > 0.f)) return fail(PILLARS_E_BADARG, "voxel[%d] must be > 0", i);
    }
    if (g->max_points < 1) return fail(PILLARS_E_BADARG, "max_points = %d", g->max_points);
    if (g->max_voxels < 0) return fail(PILLARS_E_BADARG, "max_voxels = %d", g->max_voxels);
    if (nb < 0 || nb > kMaxFrames) return fail(PILLARS_E_UNSUPPORTED, "n_frames = %d (max %d)", nb, kMaxFrames);
    const unsigned long long cells =
        static_cast<unsigned long long>(g->grid[0]) * g->grid[1] * static_cast<unsigned long long>(g->grid[2]);
    if (cells * static_cast<unsigned long long>(nb > 0 ? nb : 1) >= 0xFFFFFFFFull)
        return fail(PILLARS_E_UNSUPPORTED, "n_frames * cells does not fit a 32-bit pillar key");
    return 0;
}

static int check_points(const float *points, int64_t n, int stride, int col0, int c_point)
{
    if (n < 0 || n >= (1ll << 31) - kTile) return fail(PILLARS_E_UNSUPPORTED, "n_points = %lld", (long long)n);
    if (n > 0 && !points) return fail(PILLARS_E_BADARG, "points is NULL");
    if (stride < 3 || stride > 16) return fail(PILLARS_E_UNSUPPORTED, "row_stride = %d (3..16)", stride);
    if (col0 < 0 || c_point < 3 || col0 + c_point > stride)
        return fail(PILLARS_E_BADARG, "col0 = %d, c_point = %d do not fit row_stride = %d", col0, c_point, stride);
    return 0;
}

static int idx_bits_for(int64_t n)
{
    int bits = 1;
    while ((1ll << bits) < n) ++bits;
    return bits;
}

static int check_pfn(const pillars_pfn_t *pfn)
{
    if (!pfn || !pfn->weight || !pfn->scale || !pfn->shift) return fail(PILLARS_E_BADARG, "pfn / weights NULL");
    if (pfn->f_out != 64) return fail(PILLARS_E_UNSUPPORTED, "f_out = %d (only 64 is instantiated)", pfn->f_out);
    if (pfn->c_point < 3 || pfn->c_point > 6)
        return fail(PILLARS_E_UNSUPPORTED, "c_point = %d (3..6 are instantiated)", pfn->c_point);
    const int want = (pfn->use_absolute_xyz ? pfn->c_point : pfn->c_point - 3) + 6 + (pfn->with_distance ? 1 : 0);
    if (pfn->c_in != want) return fail(PILLARS_E_BADARG, "c_in = %d, expected %d", pfn->c_in, want);
    return 0;
}

static thread_local bool g_force_generic = false;

// what pfn_stream.cu is written for: absolute xyz + cluster + centre features of a <= 5-channel point, 64 outputs
static bool stream_kernel_covers(const pillars_pfn_t &pfn)
{
    return pfn.use_absolute_xyz && !pfn.with_distance && pfn.c_point <= 5 && pfn.f_out == 64;
}

static PfnDev make_pfn_dev(const float *weight, const float *scale, const float *shift, const float offset[3],
                           const float voxel[3])
{
    PfnDev d;
    d.weight = weight;
    d.scale = scale;
    d.shift = shift;
    for (int i = 0; i < 3; ++i) {
        d.off[i] = offset[i];
        d.vsz[i] = voxel[i];
    }
    return d;
}

static PfnDev make_pfn_dev(const pillars_pfn_t &pfn, const float voxel[3])
{
    return make_pfn_dev(pfn.weight, pfn.scale, pfn.shift, pfn.offset, voxel);
}

}  // namespace pillars

using namespace pillars;

extern "C" {

int pillars_abi_version(void) { return PILLARS_ABI_VERSION; }
const char *pillars_last_error(void) { return g_err; }
int pillars_last_launch_count(void) { return g_launches_last; }

int pillars_set_stage_events(void *const *events4)
{
    g_stage_on = events4 != nullptr;
    for (int i = 0; i < 4; ++i) g_stage_ev[i] = events4 ? static_cast<cudaEvent_t>(events4[i]) : nullptr;
    return 0;
}

int pillars_set_canvas_occupancy(const uint32_t *prev, uint32_t *next)
{
    g_occ = CanvasOccupancy{};
    if (prev && !next) return fail(PILLARS_E_BADARG, "canvas occupancy: prev without next");
    g_occ.prev = prev;
    g_occ.next = next;
    return 0;
}

int pillars_set_debug_times(void *buffer32)
{
    g_dbg_times = static_cast<unsigned long long *>(buffer32);
    return 0;
}

int pillars_set_grouping(int mode)
{
    if (mode < 0 || mode > 2) return fail(PILLARS_E_BADARG, "grouping mode = %d (0 auto, 1 hash, 2 dense)", mode);
    g_grouping = mode;
    return 0;
}

int pillars_force_generic_features(int on)
{
    g_force_generic = on != 0;
    return 0;
}

int pillars_device_ok(int device)
{
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) return fail(PILLARS_E_NODEVICE, "no CUDA device (%s)", cudaGetErrorName(e));
    if (device < 0 && (e = cudaGetDevice(&device)) != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
    int major = 0;
    if ((e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device)) != cudaSuccess)
        return cuda_fail(e, "cudaDeviceGetAttribute");
    if (major != 10) return fail(PILLARS_E_NODEVICE, "device %d has compute capability %d.x; this library is sm_100a only", device, major);
    return 0;
}

size_t pillars_workspace_bytes(int64_t n_points, int32_t n_frames, const pillars_grid_t *grid)
{
    if (!grid || n_points < 0 || n_frames < 0) return 0;
    const int64_t cells_xy = static_cast<int64_t>(grid->grid[0]) * grid->grid[1];
    const int64_t cells = cells_xy * grid->grid[2];
    // A pillar grid (nz == 1) is charged for the dense layout wherever it is possible, whatever the grouping mode: its
    // table is at most 8 bytes per BEV cell, and a workspace sized once fits every mode.  A voxel grid is charged only where
    // a call on this thread resolves to it: 16 x 1440 x 1440 x 40 cells would otherwise cost 10.7 GB that its calls never use.
    const bool dense = grid->grid[2] == 1 ? dense_possible(n_points, n_frames, cells)
                                          : resolve_group_mode(true, n_points, n_frames, cells) == kGroupDense;
    return workspace_bytes_for(n_points, n_frames, cells_xy, cells, dense);
}

int pillars_frame_offsets(const float *points_b, int64_t n, int32_t row_stride, int32_t n_frames,
                          int32_t *frame_offsets, void *stream)
{
    g_launches = 0;
    if (!frame_offsets || n < 0 || (n > 0 && !points_b) || row_stride < 1 || n_frames < 0)
        return fail(PILLARS_E_BADARG, "pillars_frame_offsets: bad argument");
    cudaError_t e = launch_frame_offsets(points_b, n, row_stride, n_frames, frame_offsets, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "pillars_frame_offsets");
    g_launches_last = g_launches;
    return 0;
}

// One call of the fused encoder, as its entry point normalised it.  The features are those of `pfn`
// (pillars_encode_bev), of `stack` (pillars_encode_stack), the voxel mean (pillars_voxelize_mean) or none
// (pillars_voxelize).
struct EncodeCall {
    const float *points;
    int64_t n;
    int stride, col0, c_point;
    const int32_t *frame_offsets;
    int nb;
    const pillars_grid_t *grid;
    const pillars_outputs_t *out;
    void *workspace;
    size_t workspace_bytes;
    int scatter_variant;
    void *stream;
    CanvasOccupancy occ;
    const pillars_pfn_t *pfn;  // checked by check_pfn
    const StackDev *stack;     // checked by check_stack
    bool dynamic;              // PILLARS_MODE_DYNAMIC
    int coords_cols;
    float *voxel_mean;         // [capacity, c_point] (pillars_voxelize_mean)
};

// Which kernels compute the per-pillar outputs of a call
enum FeatureRoute {
    kRouteEmit,    // k_emit_voxels only (pillars_voxelize)
    kRoutePfn,     // the general one-layer kernel (pfn.cu)
    kRouteMulti,   // the general stack kernel (pfn_multi.cu)
    kRouteStream,  // the streaming kernel (pfn_stream.cu), on the point records the grouping emits
    kRouteMean,    // k_voxel_mean (pfn.cu, pillars_voxelize_mean)
};

// The streaming kernel covers the mainstream configurations; everything else runs a general kernel.  For stacks these are
// Waymo's own PFN, NUM_FILTERS [64, 64] (waymo_models/pointpillar_1x.yaml:34), and DynamicPillarVFE
// (dynamic_pillar_vfe.py:14-142) with NUM_FILTERS [64] or [64, 64], in the standard feature layout.  A hard one-layer stack
// and an empty batch stay on the general kernel.
static FeatureRoute pick_route(const EncodeCall &c)
{
    if (c.voxel_mean) return kRouteMean;
    if (!c.pfn && !c.stack) return kRouteEmit;
    // (the streaming kernel's per-pillar record packs x and y into 16 bits each)
    const bool stream_ok = !g_force_generic && c.grid->grid[0] <= 0xFFFF && c.grid->grid[1] <= 0xFFFF;
    if (c.pfn) return stream_ok && stream_kernel_covers(*c.pfn) ? kRouteStream : kRoutePfn;
    const StackDev &s = *c.stack;
    const bool layers = s.n_layers == 2 ? s.out[0] == 32 && s.out[1] == 64 : c.dynamic && s.out[0] == 64;
    const bool covered = layers && s.layout == PILLARS_LAYOUT_PILLAR_VFE && s.use_abs && !s.with_dist && c.c_point <= 5 &&
                         c.coords_cols == 4 && c.n > 0;
    return stream_ok && covered ? kRouteStream : kRouteMulti;
}

// What the three entry points share: the common checks, then grouping -> (dynamic rows) -> (fold) -> features -> scatter.
static int encode(const EncodeCall &c)
{
    g_launches = 0;
    const pillars_grid_t *grid = c.grid;
    const pillars_outputs_t *out = c.out;
    int rc;
    if ((rc = check_grid(grid, c.nb))) return rc;
    if ((rc = check_points(c.points, c.n, c.stride, c.col0, c.c_point))) return rc;
    if (!c.frame_offsets || !out) return fail(PILLARS_E_BADARG, "frame_offsets / out is NULL");
    if (c.n > 0 && c.nb == 0) return fail(PILLARS_E_BADARG, "n_points = %lld with n_frames = 0", (long long)c.n);
    const bool features = c.pfn || c.stack;
    if (features && !out->pillar_features) return fail(PILLARS_E_BADARG, "pillar_features output is required");
    if (out->pillar_capacity < 0) return fail(PILLARS_E_BADARG, "pillar_capacity < 0");
    if (c.occ.next && out->bev && out->bev_half)
        return fail(PILLARS_E_BADARG, "canvas occupancy is set but the call writes both bev and bev_half");
    const bool want_bev = features && (out->bev || out->bev_half);
    const bool want_map = want_bev || out->want_index_map;
    if (want_map && grid->grid[2] != 1) return fail(PILLARS_E_UNSUPPORTED, "BEV scatter / index map needs nz == 1");
    if (!c.workspace || reinterpret_cast<uintptr_t>(c.workspace) % 256 != 0)
        return fail(PILLARS_E_WORKSPACE, "workspace NULL or not 256-byte aligned");
    const int64_t cells_xy = static_cast<int64_t>(grid->grid[0]) * grid->grid[1];
    const int64_t cells = cells_xy * grid->grid[2];
    // the dynamic variant ranks the cells of the dense index-map region itself: it keeps the hash table
    const Workspace ws = carve_workspace(c.workspace, c.n, c.nb, cells_xy, cells,
                                         resolve_group_mode(!c.dynamic, c.n, c.nb, cells));
    if (ws.total_bytes > c.workspace_bytes)
        return fail(PILLARS_E_WORKSPACE, "workspace has %zu bytes, %zu needed", c.workspace_bytes, ws.total_bytes);

    cudaStream_t st = static_cast<cudaStream_t>(c.stream);
    GridDev gd = make_grid_dev(*grid);
    if (c.dynamic) {
        gd.ignore_z = 1;
        gd.max_points = 0x7FFFFFFF;
        gd.max_voxels = 0x7FFFFFFF;
    }
    const FeatureRoute route = pick_route(c);
    const bool membership = out->voxels || out->point_pillar || out->point_slot;
    const int idx_bits = idx_bits_for(c.n > 1 ? c.n : 2);
    // layer 0; its offset and voxel size also place the pillar centres for the grouping and the streaming kernel
    PfnDev l0{};
    if (c.pfn) l0 = make_pfn_dev(*c.pfn, grid->voxel);
    if (c.stack) l0 = make_pfn_dev(c.stack->weight[0], c.stack->scale[0], c.stack->shift[0], c.stack->off, c.stack->vsz);
    cudaError_t e;
    stage_mark(0, st);

    if (out->point_pillar && c.n > 0) {
        if ((e = cudaMemsetAsync(out->point_pillar, 0xFF, sizeof(int32_t) * c.n, st)) != cudaSuccess) return cuda_fail(e, "memset");
        note_launch();
    }
    if (out->point_slot && c.n > 0) {
        if ((e = cudaMemsetAsync(out->point_slot, 0xFF, sizeof(int32_t) * c.n, st)) != cudaSuccess) return cuda_fail(e, "memset");
        note_launch();
    }
    PlaceExtras px{};
    px.records = route == kRouteStream;
    px.capacity = out->pillar_capacity;
    px.skip_index_map = route == kRouteMean;
    if (px.records) {
        for (int i = 0; i < 3; ++i) {
            px.vsz[i] = l0.vsz[i];
            px.off[i] = l0.off[i];
        }
        if (!c.dynamic) {  // (launch_dynamic_rows writes these for the dynamic variant)
            px.voxel_coords = out->voxel_coords;
            px.voxel_num_points = out->voxel_num_points;
            px.write_cell_row = want_map;
        }
    }
    if ((e = launch_group_points(c.points, c.n, c.stride, c.col0, c.c_point, c.frame_offsets, c.nb, gd, ws, out->pillar_count,
                                 /*want_index_lists=*/membership || route != kRouteStream, px, st)) != cudaSuccess)
        return cuda_fail(e, "group_points");
    stage_mark(1, st);

    // membership outputs (pillars_voxelize, pillars_encode_bev) come from k_emit_voxels, whatever computes the features;
    // the voxel mean walks the same lists
    if (route == kRouteEmit || route == kRoutePfn || route == kRouteMean || membership) {
        FeatureJob job{};
        job.points = c.points;
        job.n = c.n;
        job.stride = c.stride;
        job.col0 = c.col0;
        job.c_point = c.c_point;
        job.nb = c.nb;
        job.idx_bits = idx_bits;
        job.do_features = route == kRoutePfn;
        if (c.pfn) {
            job.use_abs = c.pfn->use_absolute_xyz != 0;
            job.with_dist = c.pfn->with_distance != 0;
        }
        job.pfn = l0;
        job.out = *out;
        job.write_cell_row = want_map && route != kRouteStream;
        if (route == kRouteMean) {
            if ((e = launch_voxel_mean(job, c.voxel_mean, gd, ws, st)) != cudaSuccess) return cuda_fail(e, "voxel_mean");
        } else if ((e = launch_pillar_features(job, gd, ws, st)) != cudaSuccess) {
            return cuda_fail(e, "pillar_features");
        }
    }
    if (route == kRouteStream) {
        // the dynamic variant's pillar entries get their rows (sorted-key order) between the grouping and the feature kernel
        if (c.dynamic &&
            (e = launch_dynamic_rows(gd, ws, c.nb, c.n, out->pillar_capacity, out->voxel_coords, out->voxel_num_points, st)) != cudaSuccess)
            return cuda_fail(e, "dynamic_rows");
        const bool two = c.stack && c.stack->n_layers == 2;
        const float *folded = c.pfn ? c.pfn->folded : nullptr;
        if (!folded) {  // the caller did not prepare the table: fold into the workspace (one more single-block launch)
            const int c_in = c.pfn ? c.pfn->c_in : stack_c_in(*c.stack, c.c_point);
            if ((e = launch_fold_pfn(l0, c.c_point, c_in, ws.folded, st, two ? 32 : 64)) != cudaSuccess)
                return cuda_fail(e, "fold_pfn");
            folded = ws.folded;
        }
        if (two && (e = launch_fold_pfn2(c.stack->weight[1], c.stack->scale[1], c.stack->shift[1], ws.folded2, st)) != cudaSuccess)
            return cuda_fail(e, "fold_pfn2");
        FastJob fj{};
        fj.dynamic = c.dynamic;
        fj.n = c.n;
        fj.idx_bits = idx_bits;
        fj.pillar_features = out->pillar_features;
        fj.folded2 = two ? ws.folded2 : nullptr;
        for (int i = 0; i < 3; ++i) {
            fj.vsz[i] = l0.vsz[i];
            fj.off[i] = l0.off[i];
        }
        if ((e = launch_pillar_features_stream(fj, folded, gd, ws, st)) != cudaSuccess)
            return cuda_fail(e, "pillar_features_stream");
    }
    if (route == kRouteMulti) {
        MultiJob job{};
        job.points = c.points;
        job.n = c.n;
        job.stride = c.stride;
        job.col0 = c.col0;
        job.c_point = c.c_point;
        job.nb = c.nb;
        job.idx_bits = idx_bits;
        job.dynamic = c.dynamic;
        job.write_cell_row = want_map;
        job.pillar_features = out->pillar_features;
        job.voxel_coords = out->voxel_coords;
        job.voxel_num_points = out->voxel_num_points;
        job.coords_cols = c.coords_cols;
        job.capacity = out->pillar_capacity;
        if ((e = launch_pfn_multi_lists(job, *c.stack, gd, ws, st)) != cudaSuccess) return cuda_fail(e, "pfn_multi");
    }
    stage_mark(2, st);

    if (want_bev) {
        const int f = c.pfn ? c.pfn->f_out : c.stack->out[c.stack->n_layers - 1];
        if (out->bev && (e = launch_scatter(out->pillar_features, ws.cell_row, c.nb, f, grid->grid[0], grid->grid[1], out->bev,
                                            c.scatter_variant, st, c.occ.prev, c.occ.next)) != cudaSuccess)
            return cuda_fail(e, "scatter");
        if (out->bev_half && (e = launch_scatter_half(out->pillar_features, ws.cell_row, c.nb, f, grid->grid[0], grid->grid[1],
                                                      out->bev_half, st, c.occ.prev, c.occ.next)) != cudaSuccess)
            return cuda_fail(e, "scatter (float16 canvas: needs nx*ny % 8 == 0, f % 8 == 0)");
    }
    stage_mark(3, st);
    g_launches_last = g_launches;
    return 0;
}

int pillars_fold_pfn(const pillars_pfn_t *pfn, float *folded, void *stream)
{
    g_launches = 0;
    int rc;
    if ((rc = check_pfn(pfn))) return rc;
    if (!folded) return fail(PILLARS_E_BADARG, "folded is NULL");
    if (!stream_kernel_covers(*pfn)) return fail(PILLARS_E_UNSUPPORTED, "layer is outside what the streaming feature kernel covers");
    const float unit[3] = {1.f, 1.f, 1.f};
    cudaError_t e = launch_fold_pfn(make_pfn_dev(*pfn, unit), pfn->c_point, pfn->c_in, folded, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "fold_pfn");
    g_launches_last = g_launches;
    return 0;
}

int pillars_voxelize(const float *points, int64_t n, int32_t row_stride, int32_t col0, int32_t c_point,
                     const int32_t *frame_offsets, int32_t n_frames, const pillars_grid_t *grid,
                     const pillars_outputs_t *out, void *workspace, size_t workspace_bytes, void *stream)
{
    return encode({points, n, row_stride, col0, c_point, frame_offsets, n_frames, grid, out, workspace, workspace_bytes, 0,
                   stream});
}

int pillars_voxelize_mean(const float *points, int64_t n, int32_t row_stride, int32_t col0, int32_t c_point,
                          const int32_t *frame_offsets, int32_t n_frames, const pillars_grid_t *grid,
                          const pillars_outputs_t *out, float *voxel_mean, void *workspace, size_t workspace_bytes,
                          void *stream)
{
    g_launches = 0;
    if (!voxel_mean) return fail(PILLARS_E_BADARG, "voxel_mean is NULL");
    if (out && (out->pillar_features || out->voxels || out->point_pillar || out->point_slot || out->bev || out->bev_half ||
                out->want_index_map))
        return fail(PILLARS_E_UNSUPPORTED, "pillars_voxelize_mean writes voxel_coords, voxel_num_points and pillar_count "
                                           "only; the other outputs come from pillars_voxelize");
    if (grid && grid->max_points > kMeanMaxPoints)
        return fail(PILLARS_E_UNSUPPORTED, "max_points = %d (the voxel mean is built for up to %d)", grid->max_points,
                    kMeanMaxPoints);
    EncodeCall c{points, n, row_stride, col0, c_point, frame_offsets, n_frames, grid, out, workspace, workspace_bytes, 0, stream};
    c.voxel_mean = voxel_mean;
    return encode(c);
}

int pillars_encode_bev(const float *points, int64_t n, int32_t row_stride, int32_t col0, const int32_t *frame_offsets,
                       int32_t n_frames, const pillars_grid_t *grid, const pillars_pfn_t *pfn,
                       const pillars_outputs_t *out, void *workspace, size_t workspace_bytes, int32_t scatter_variant,
                       void *stream)
{
    const CanvasOccupancy occ = take_canvas_occupancy();
    int rc;
    if ((rc = check_pfn(pfn))) return rc;
    return encode({points, n, row_stride, col0, pfn->c_point, frame_offsets, n_frames, grid, out, workspace, workspace_bytes,
                   scatter_variant, stream, occ, pfn});
}

int pillars_pfn_dense(const float *voxels, const void *num_points, int32_t num_points_is_float, const void *coords,
                      int32_t coords_is_float, int64_t m, int32_t max_points, const pillars_pfn_t *pfn,
                      const float voxel_size[3], float *out, void *stream)
{
    g_launches = 0;
    int rc;
    if ((rc = check_pfn(pfn))) return rc;
    if (m < 0 || max_points < 1 || !voxel_size) return fail(PILLARS_E_BADARG, "pillars_pfn_dense: bad size");
    if (m > 0 && (!voxels || !num_points || !coords || !out)) return fail(PILLARS_E_BADARG, "pillars_pfn_dense: NULL pointer");
    if (reinterpret_cast<uintptr_t>(coords) % 16 != 0 || reinterpret_cast<uintptr_t>(out) % 16 != 0)
        return fail(PILLARS_E_BADARG, "coords / out must be 16-byte aligned");
    const PfnDev pd = make_pfn_dev(*pfn, voxel_size);
    // the folded form (table prepared by pillars_fold_pfn) where it applies, else the faithful 11-feature kernel
    const bool folded_ok = pfn->folded && stream_kernel_covers(*pfn) && !g_force_generic && m < (int64_t(1) << 31) &&
                           max_points <= 32;  // one slot per lane
    cudaError_t e = folded_ok
                        ? launch_pfn_padded(voxels, num_points, num_points_is_float != 0, coords, coords_is_float != 0, m,
                                            max_points, pfn->c_point, pd, pfn->folded, out, static_cast<cudaStream_t>(stream))
                        : launch_pfn_dense(voxels, num_points, num_points_is_float != 0, coords, coords_is_float != 0, m,
                                           max_points, pfn->c_point, pfn->use_absolute_xyz != 0, pfn->with_distance != 0, pd,
                                           out, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "pillars_pfn_dense");
    g_launches_last = g_launches;
    return 0;
}

static int check_stack(const pillars_pfn_stack_t *sk, StackDev *sd, const float voxel[3])
{
    if (!sk) return fail(PILLARS_E_BADARG, "stack is NULL");
    if (sk->n_layers < 1 || sk->n_layers > 2)
        return fail(PILLARS_E_UNSUPPORTED, "n_layers = %d (1 or 2 are built)", sk->n_layers);
    if (sk->c_point < 3 || sk->c_point > 8) return fail(PILLARS_E_UNSUPPORTED, "c_point = %d (3..8)", sk->c_point);
    if (sk->layout != PILLARS_LAYOUT_PILLAR_VFE && sk->layout != PILLARS_LAYOUT_SIMPLE2D)
        return fail(PILLARS_E_BADARG, "layout = %d", sk->layout);
    sd->n_layers = sk->n_layers;
    sd->use_abs = sk->use_absolute_xyz != 0;
    sd->with_dist = sk->with_distance != 0;
    sd->layout = sk->layout;
    for (int l = 0; l < 2; ++l) {
        sd->out[l] = l < sk->n_layers ? sk->out_features[l] : 0;
        sd->weight[l] = l < sk->n_layers ? sk->weight[l] : nullptr;
        sd->scale[l] = l < sk->n_layers ? sk->scale[l] : nullptr;
        sd->shift[l] = l < sk->n_layers ? sk->shift[l] : nullptr;
        if (l < sk->n_layers && (!sk->weight[l] || !sk->scale[l] || !sk->shift[l]))
            return fail(PILLARS_E_BADARG, "stack layer %d: weight / scale / shift NULL", l);
    }
    for (int i = 0; i < 3; ++i) {
        sd->off[i] = sk->offset[i];
        sd->vsz[i] = voxel ? voxel[i] : 1.f;
    }
    if (!stack_supported(*sd, sk->c_point))
        return fail(PILLARS_E_UNSUPPORTED, "feature stack outside the built shapes (layer 0 in <= 16, out <= 64; two layers: "
                                           "out[0] <= 32)");
    return 0;
}

int pillars_pfn_stack_in_features(const pillars_pfn_stack_t *stack)
{
    if (!stack) return fail(PILLARS_E_BADARG, "stack is NULL");
    StackDev sd{};
    sd.use_abs = stack->use_absolute_xyz != 0;
    sd.with_dist = stack->with_distance != 0;
    sd.layout = stack->layout;
    return stack_c_in(sd, stack->c_point);
}

int pillars_pfn_dense_stack(const float *voxels, const void *num_points, int32_t num_points_is_float, const void *coords,
                            int32_t coords_is_float, int64_t m, int32_t max_points, const pillars_pfn_stack_t *stack,
                            const float voxel_size[3], float *out, void *stream)
{
    g_launches = 0;
    StackDev sd{};
    int rc;
    if (!voxel_size) return fail(PILLARS_E_BADARG, "voxel_size is NULL");
    if ((rc = check_stack(stack, &sd, voxel_size))) return rc;
    if (stack->layout != PILLARS_LAYOUT_PILLAR_VFE) return fail(PILLARS_E_BADARG, "padded voxels only exist for PillarVFE");
    if (m < 0 || max_points < 1) return fail(PILLARS_E_BADARG, "pillars_pfn_dense_stack: bad size");
    if (m > 0 && (!voxels || !num_points || !coords || !out)) return fail(PILLARS_E_BADARG, "pillars_pfn_dense_stack: NULL pointer");
    if (reinterpret_cast<uintptr_t>(coords) % 16 != 0) return fail(PILLARS_E_BADARG, "coords must be 16-byte aligned");
    cudaError_t e = launch_pfn_multi_dense(voxels, num_points, num_points_is_float != 0, coords, coords_is_float != 0, m,
                                           max_points, stack->c_point, sd, out, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "pillars_pfn_dense_stack");
    g_launches_last = g_launches;
    return 0;
}

int pillars_encode_stack(const float *points, int64_t n, int32_t row_stride, int32_t col0, const int32_t *frame_offsets,
                         int32_t n_frames, const pillars_grid_t *grid, const pillars_pfn_stack_t *stack, int32_t mode,
                         int32_t coords_cols, const pillars_outputs_t *out, void *workspace, size_t workspace_bytes,
                         int32_t scatter_variant, void *stream)
{
    const CanvasOccupancy occ = take_canvas_occupancy();
    StackDev sd{};
    int rc;
    if ((rc = check_stack(stack, &sd, grid ? grid->voxel : nullptr))) return rc;
    if (mode != PILLARS_MODE_HARD && mode != PILLARS_MODE_DYNAMIC) return fail(PILLARS_E_BADARG, "mode = %d", mode);
    if (coords_cols != 3 && coords_cols != 4) return fail(PILLARS_E_BADARG, "coords_cols = %d", coords_cols);
    const bool dynamic = mode == PILLARS_MODE_DYNAMIC;
    if (out && (out->voxels || out->point_pillar || out->point_slot))
        return fail(PILLARS_E_UNSUPPORTED, "membership outputs come from pillars_voxelize");
    if (out && (out->bev || out->bev_half || out->want_index_map) && (dynamic || coords_cols != 4))
        return fail(PILLARS_E_UNSUPPORTED, "the fused BEV canvas / index map needs mode HARD and 4-column coords");
    return encode({points, n, row_stride, col0, stack->c_point, frame_offsets, n_frames, grid, out, workspace, workspace_bytes,
                   scatter_variant, stream, occ, nullptr, &sd, dynamic, coords_cols});
}

// What pillars_scatter_bev and pillars_scatter_bev_half share: the argument checks and the index map, built in the
// workspace.  *cell_row stays NULL when there is nothing to scatter (n_frames == 0).
static int scatter_cell_row(bool half, const float *feats, const void *coords, int32_t coords_is_float, int64_t m,
                            const int32_t *m_dev, int32_t n_frames, int32_t f, int32_t nx, int32_t ny, int32_t nz,
                            const void *canvas, void *workspace, size_t workspace_bytes, cudaStream_t st, int32_t **cell_row)
{
    g_launches = 0;
    *cell_row = nullptr;
    const char *what = half ? "pillars_scatter_bev_half" : "pillars_scatter_bev";
    if (m < 0 || n_frames < 0 || f < 1 || nx < 1 || ny < 1 || nz < 1) return fail(PILLARS_E_BADARG, "%s: bad size", what);
    if (n_frames > 0 && !canvas) return fail(PILLARS_E_BADARG, "%s: canvas is NULL", what);
    if (m > 0 && (!feats || !coords)) return fail(PILLARS_E_BADARG, "feats / coords NULL");
    if (m > 0 && reinterpret_cast<uintptr_t>(coords) % 16 != 0) return fail(PILLARS_E_BADARG, "coords must be 16-byte aligned");
    if (half && ((static_cast<int64_t>(nx) * ny * nz) % 8 != 0 || f % 8 != 0))
        return fail(PILLARS_E_UNSUPPORTED, "float16 canvas needs nx*ny*nz %% 8 == 0 and f %% 8 == 0");
    const size_t need = sizeof(int32_t) * static_cast<size_t>(n_frames) * nx * ny * nz;
    if (need > 0 && (!workspace || workspace_bytes < need || reinterpret_cast<uintptr_t>(workspace) % 16 != 0))
        return fail(PILLARS_E_WORKSPACE, "workspace has %zu bytes, %zu needed", workspace_bytes, need);
    if (n_frames == 0) return 0;
    *cell_row = static_cast<int32_t *>(workspace);
    const cudaError_t e = launch_build_cell_row(coords, coords_is_float != 0, m, m_dev, n_frames, nx, ny, nz, *cell_row, st);
    return e == cudaSuccess ? 0 : cuda_fail(e, "build_cell_row");
}

int pillars_scatter_bev(const float *feats, const void *coords, int32_t coords_is_float, int64_t m, const int32_t *m_dev,
                        int32_t n_frames, int32_t f, int32_t nx, int32_t ny, int32_t nz, float *bev, void *workspace,
                        size_t workspace_bytes, int32_t variant, void *stream)
{
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int32_t *cell_row;
    const int rc = scatter_cell_row(false, feats, coords, coords_is_float, m, m_dev, n_frames, f, nx, ny, nz, bev, workspace,
                                    workspace_bytes, st, &cell_row);
    if (rc || !cell_row) return rc;
    // the canvas of the 3-D variant is the 2-D one with nz*ny rows per channel
    const cudaError_t e = launch_scatter(feats, cell_row, n_frames, f, nx, ny * nz, bev, variant, st);
    if (e != cudaSuccess) return cuda_fail(e, "scatter");
    g_launches_last = g_launches;
    return 0;
}

int pillars_rebase_segments(int32_t *coords, int32_t n_segments, int64_t rows_per_segment, int64_t segment_stride,
                            const int32_t *segment_counts, int64_t count_stride, int32_t frames_per_segment,
                            int32_t *overflow, void *stream)
{
    g_launches = 0;
    if (n_segments < 0 || rows_per_segment < 0 || count_stride < 1 || frames_per_segment < 0 ||
        segment_stride < rows_per_segment * 4)
        return fail(PILLARS_E_BADARG, "pillars_rebase_segments: bad size");
    if (static_cast<int64_t>(n_segments) * rows_per_segment > 0 && (!coords || !segment_counts))
        return fail(PILLARS_E_BADARG, "pillars_rebase_segments: NULL pointer");
    cudaError_t e = launch_rebase_segments(coords, n_segments, rows_per_segment, segment_stride, segment_counts,
                                           count_stride, frames_per_segment, overflow, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "rebase_segments");
    g_launches_last = g_launches;
    return 0;
}

int pillars_scatter_bev_half(const float *feats, const void *coords, int32_t coords_is_float, int64_t m,
                             const int32_t *m_dev, int32_t n_frames, int32_t f, int32_t nx, int32_t ny, int32_t nz,
                             void *bev_half, void *workspace, size_t workspace_bytes, void *stream)
{
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int32_t *cell_row;
    const int rc = scatter_cell_row(true, feats, coords, coords_is_float, m, m_dev, n_frames, f, nx, ny, nz, bev_half,
                                    workspace, workspace_bytes, st, &cell_row);
    if (rc || !cell_row) return rc;
    const cudaError_t e = launch_scatter_half(feats, cell_row, n_frames, f, nx, ny * nz, bev_half, st);
    if (e != cudaSuccess) return cuda_fail(e, "scatter (float16 canvas)");
    g_launches_last = g_launches;
    return 0;
}

// ---- BEV tokeniser ------------------------------------------------------------------------------------------------------
static int check_tokenizer(const pillars_tokenizer_t *tk, bool need_tables, TokenizerDev *td)
{
    if (!tk) return fail(PILLARS_E_BADARG, "tokenizer is NULL");
    if (!tokens_shape_supported(tk->c_in, tk->d_model))
        return fail(PILLARS_E_UNSUPPORTED, "tokeniser needs c_in %% 4 == 0 (<= 512) and d_model %% 128 == 0 (<= 1024), got %d / %d",
                    tk->c_in, tk->d_model);
    const void *ptrs[] = {tk->dw_weight, tk->dw_bias, tk->proj_weight_t, tk->proj_bias, tk->ln_weight, tk->ln_bias,
                          need_tables ? tk->pe : tk->dw_bias, need_tables ? tk->background : tk->dw_bias};
    for (const void *q : ptrs)
        if (!q || reinterpret_cast<uintptr_t>(q) % 16 != 0) return fail(PILLARS_E_BADARG, "tokenizer pointer NULL or not 16-byte aligned");
    td->c = tk->c_in; td->d = tk->d_model;
    td->dw_w = tk->dw_weight; td->dw_b = tk->dw_bias; td->wt = tk->proj_weight_t; td->pb = tk->proj_bias;
    td->gamma = tk->ln_weight; td->beta = tk->ln_bias; td->eps = tk->ln_eps; td->pe = tk->pe; td->bg = tk->background;
    td->wimg = need_tables ? tk->proj_umma : nullptr;
    if (td->wimg && reinterpret_cast<uintptr_t>(td->wimg) % 16 != 0) return fail(PILLARS_E_BADARG, "proj_umma not 16-byte aligned");
    return 0;
}

int pillars_tokens_prepare(const pillars_tokenizer_t *tk, const float *geom, const int32_t *sector, int32_t h, int32_t w,
                           const float *geo_w1, const float *geo_b1, const float *geo_w2_t, const float *geo_b2,
                           const float *view_embed, float *pe_out, float *background_out, float *proj_umma_out, void *stream)
{
    g_launches = 0;
    TokenizerDev td{};
    int rc;
    if ((rc = check_tokenizer(tk, false, &td))) return rc;
    if (h < 0 || w < 0) return fail(PILLARS_E_BADARG, "pillars_tokens_prepare: bad size");
    if (!background_out || !geo_w1 || !geo_b1 || !geo_w2_t || !geo_b2 || !view_embed)
        return fail(PILLARS_E_BADARG, "pillars_tokens_prepare: NULL pointer");
    if (static_cast<int64_t>(h) * w > 0 && (!geom || !sector || !pe_out))
        return fail(PILLARS_E_BADARG, "pillars_tokens_prepare: geom / sector / pe_out NULL");
    cudaError_t e = launch_tokens_prepare(td, geom, sector, h, w, geo_w1, geo_b1, geo_w2_t, geo_b2, view_embed, pe_out,
                                          background_out, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "tokens_prepare");
    if (proj_umma_out && tokens_umma_supported(td.c, td.d) &&
        (e = launch_tokens_wimg(td.wt, td.c, td.d, proj_umma_out, static_cast<cudaStream_t>(stream))) != cudaSuccess)
        return cuda_fail(e, "tokens_wimg");
    g_launches_last = g_launches;
    return 0;
}

static size_t tokens_map_bytes(int32_t n_frames, int32_t h, int32_t w)
{
    return align_up(sizeof(int32_t) * static_cast<size_t>(n_frames) * h * w, 256);
}

// pair list of the tcgen05 variant: a counter (256 B) + one 32-bit entry per (frame, cell)
static size_t tokens_list_bytes(int32_t n_frames, int32_t h, int32_t w) { return 256 + tokens_map_bytes(n_frames, h, w); }

// runs the tokeniser on rows + index map; `scratch` (tokens_list_bytes, 256-byte aligned) enables the tcgen05 variant
static cudaError_t run_tokens(const TokenizerDev &td, const float *feats, const int32_t *cell_row, int32_t n_frames, int32_t h,
                              int32_t w, float *tokens, void *scratch, size_t scratch_bytes, cudaStream_t st)
{
    if (td.wimg && tokens_umma_supported(td.c, td.d) && scratch && reinterpret_cast<uintptr_t>(scratch) % 256 == 0 &&
        scratch_bytes >= tokens_list_bytes(n_frames, h, w)) {
        uint32_t *count = static_cast<uint32_t *>(scratch);
        uint32_t *list = reinterpret_cast<uint32_t *>(static_cast<char *>(scratch) + 256);
        return launch_bev_tokens_umma(td, feats, cell_row, n_frames, h, w, tokens, list, count, st);
    }
    return launch_bev_tokens(td, feats, cell_row, n_frames, h, w, tokens, st);
}

size_t pillars_tokens_workspace_bytes(int32_t n_frames, int32_t c_in, int32_t h, int32_t w, int32_t dense)
{
    if (n_frames < 0 || c_in < 0 || h < 0 || w < 0) return 0;
    size_t b = tokens_map_bytes(n_frames, h, w) + tokens_list_bytes(n_frames, h, w);
    if (dense) b += 256 + align_up(sizeof(float) * static_cast<size_t>(n_frames) * h * w * c_in, 256);
    return b;
}

static int check_tokens_call(const pillars_tokenizer_t *tk, int32_t n_frames, int32_t h, int32_t w, const float *tokens,
                             TokenizerDev *td)
{
    int rc;
    if ((rc = check_tokenizer(tk, true, td))) return rc;
    if (n_frames < 0 || h < 0 || w < 0) return fail(PILLARS_E_BADARG, "tokens: bad size");
    if (static_cast<int64_t>(n_frames) * h * w > 0 && (!tokens || reinterpret_cast<uintptr_t>(tokens) % 16 != 0))
        return fail(PILLARS_E_BADARG, "tokens output NULL or not 16-byte aligned");
    return 0;
}

int pillars_bev_tokens_map(const float *feats, const int32_t *cell_row, int32_t n_frames, int32_t h, int32_t w,
                           const pillars_tokenizer_t *tk, float *tokens, void *workspace, size_t workspace_bytes, void *stream)
{
    g_launches = 0;
    TokenizerDev td{};
    int rc;
    if ((rc = check_tokens_call(tk, n_frames, h, w, tokens, &td))) return rc;
    if (static_cast<int64_t>(n_frames) * h * w == 0) return 0;
    if (!cell_row) return fail(PILLARS_E_BADARG, "cell_row is NULL");
    // the pair list sits behind the (unused here) index-map part of a pillars_tokens_workspace_bytes(..., 0) workspace
    char *scratch = workspace ? static_cast<char *>(workspace) + tokens_map_bytes(n_frames, h, w) : nullptr;
    const size_t scratch_bytes = workspace && workspace_bytes > tokens_map_bytes(n_frames, h, w) ? workspace_bytes - tokens_map_bytes(n_frames, h, w) : 0;
    cudaError_t e = run_tokens(td, feats, cell_row, n_frames, h, w, tokens, scratch, scratch_bytes, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "bev_tokens");
    g_launches_last = g_launches;
    return 0;
}

int pillars_bev_tokens(const float *feats, const void *coords, int32_t coords_is_float, int64_t m, const int32_t *m_dev,
                       int32_t n_frames, int32_t h, int32_t w, const pillars_tokenizer_t *tk, float *tokens,
                       void *workspace, size_t workspace_bytes, void *stream)
{
    g_launches = 0;
    TokenizerDev td{};
    int rc;
    if ((rc = check_tokens_call(tk, n_frames, h, w, tokens, &td))) return rc;
    if (m < 0 || (m > 0 && (!feats || !coords))) return fail(PILLARS_E_BADARG, "feats / coords NULL");
    if (m > 0 && reinterpret_cast<uintptr_t>(coords) % 16 != 0) return fail(PILLARS_E_BADARG, "coords must be 16-byte aligned");
    if (static_cast<int64_t>(n_frames) * h * w == 0) return 0;
    const size_t need = tokens_map_bytes(n_frames, h, w);
    if (!workspace || workspace_bytes < need || reinterpret_cast<uintptr_t>(workspace) % 16 != 0)
        return fail(PILLARS_E_WORKSPACE, "workspace has %zu bytes, %zu needed", workspace_bytes, need);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int32_t *cell_row = static_cast<int32_t *>(workspace);
    cudaError_t e;
    if ((e = launch_build_cell_row(coords, coords_is_float != 0, m, m_dev, n_frames, w, h, 1, cell_row, st)) != cudaSuccess)
        return cuda_fail(e, "build_cell_row");
    char *scratch = static_cast<char *>(workspace) + need;
    if ((e = run_tokens(td, feats, cell_row, n_frames, h, w, tokens, scratch, workspace_bytes - need, st)) != cudaSuccess)
        return cuda_fail(e, "bev_tokens");
    g_launches_last = g_launches;
    return 0;
}

int pillars_bev_tokens_dense(const float *bev, int32_t n_frames, int32_t h, int32_t w, const pillars_tokenizer_t *tk,
                             float *tokens, void *workspace, size_t workspace_bytes, void *stream)
{
    g_launches = 0;
    TokenizerDev td{};
    int rc;
    if ((rc = check_tokens_call(tk, n_frames, h, w, tokens, &td))) return rc;
    if (static_cast<int64_t>(n_frames) * h * w == 0) return 0;
    if (!bev) return fail(PILLARS_E_BADARG, "bev is NULL");
    const size_t need = pillars_tokens_workspace_bytes(n_frames, tk->c_in, h, w, 1);
    if (!workspace || workspace_bytes < need || reinterpret_cast<uintptr_t>(workspace) % 256 != 0)
        return fail(PILLARS_E_WORKSPACE, "workspace has %zu bytes (256-byte aligned), %zu needed", workspace_bytes, need);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char *base = static_cast<char *>(workspace);
    int32_t *cell_row = reinterpret_cast<int32_t *>(base);
    char *scratch = base + tokens_map_bytes(n_frames, h, w);
    const size_t scratch_bytes = tokens_list_bytes(n_frames, h, w);
    uint32_t *counter = reinterpret_cast<uint32_t *>(scratch + scratch_bytes);
    float *rows = reinterpret_cast<float *>(scratch + scratch_bytes + 256);
    cudaError_t e;
    if ((e = launch_canvas_to_rows(bev, n_frames, tk->c_in, h, w, cell_row, rows, counter, st)) != cudaSuccess)
        return cuda_fail(e, "canvas_to_rows");
    if ((e = run_tokens(td, rows, cell_row, n_frames, h, w, tokens, scratch, scratch_bytes, st)) != cudaSuccess)
        return cuda_fail(e, "bev_tokens");
    g_launches_last = g_launches;
    return 0;
}

// ---- BEV backbone convolutions ------------------------------------------------------------------------------------------
static bool conv_ok(const pillars_conv_t *cv)
{
    if (!cv || cv->c_in < 32 || cv->c_in % 32 != 0 || (cv->c_out != 64 && cv->c_out != 128 && cv->c_out != 256)) return false;
    // transposed: the two dx phases share one accumulator of 2 * c_out columns, and no kernel is instantiated for 512
    if (cv->up == 2 || cv->up == 4) return cv->c_out != 256 && cv->k == 1 && cv->stride == 1 && cv->pad == 0;
    if (cv->up != 1) return false;
    return (cv->k == 3 && cv->stride == 1 && cv->pad == 1) || (cv->k == 1 && cv->stride == 1 && cv->pad == 0) ||
           (cv->k == 3 && cv->stride == 2 && cv->pad == 1) || (cv->k == 2 && cv->stride == 2 && cv->pad == 0) ||
           (cv->k == 1 && cv->stride == 2 && cv->pad == 0);
}

size_t pillars_conv_weight_bytes(const pillars_conv_t *cv)
{
    if (!conv_ok(cv)) return 0;
    const size_t taps = cv->up > 1 ? 1 : static_cast<size_t>(cv->k) * cv->k;
    return static_cast<size_t>(cv->up) * cv->up * (cv->c_in / 32) * taps * cv->c_out * 128;
}

int pillars_conv_prepare(const pillars_conv_t *cv, const float *weight, const float *bn_scale, void *image, void *stream)
{
    if (!conv_ok(cv)) return fail(PILLARS_E_UNSUPPORTED, "convolution shape outside the instantiated set");
    if (!weight || !image) return fail(PILLARS_E_BADARG, "NULL weight / image");
    g_launches = 0;
    cudaError_t e = launch_conv_wimg(weight, bn_scale, cv->c_in, cv->c_out, cv->k, cv->up, static_cast<float *>(image),
                                     static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "conv_prepare");
    g_launches_last = g_launches;
    return 0;
}

static int conv_forward(const pillars_conv_t *cv, const void *image, const float *bn_shift, const float *in_nhwc,
                        const float *rows, const int32_t *cell_row, int32_t n_frames, int32_t h_in, int32_t w_in, float *out,
                        int32_t out_c_total, int32_t out_c_off, int32_t out_nchw, const float *residual_nhwc, uint32_t *error_word,
                        void *stream)
{
    if (!conv_ok(cv)) return fail(PILLARS_E_UNSUPPORTED, "convolution shape outside the instantiated set");
    if (!image || !bn_shift || !out) return fail(PILLARS_E_BADARG, "NULL image / shift / out");
    if (!in_nhwc && !(rows && cell_row)) return fail(PILLARS_E_BADARG, "neither a dense input nor (rows, cell_row)");
    if (n_frames < 0 || h_in < 1 || w_in < 1) return fail(PILLARS_E_BADARG, "bad image shape");
    if (static_cast<int64_t>(n_frames) * h_in * w_in >= (1ll << 31)) return fail(PILLARS_E_UNSUPPORTED, "more than 2^31 input pixels");
    const auto misaligned = [](const void *q) { return q && reinterpret_cast<uintptr_t>(q) % 16 != 0; };
    if (misaligned(image) || misaligned(in_nhwc) || misaligned(rows) || misaligned(out) || misaligned(residual_nhwc))
        return fail(PILLARS_E_BADARG, "image / activations / rows / out / residual must be 16-byte aligned");
    if (out_c_off < 0 || out_c_off + cv->c_out > out_c_total || (out_nchw == 0 && (out_c_total % 4 != 0 || out_c_off % 4 != 0)))
        return fail(PILLARS_E_BADARG, "bad output channel window");
    g_launches = 0;
    if (n_frames == 0) {
        g_launches_last = 0;
        return 0;
    }
    ConvJob j{};
    j.in = in_nhwc;
    j.rows = in_nhwc ? nullptr : rows;
    j.cell_row = in_nhwc ? nullptr : cell_row;
    j.wimg = image;
    j.shift = bn_shift;
    j.out = out;
    j.nb = n_frames;
    j.h_in = h_in;
    j.w_in = w_in;
    j.c_in = cv->c_in;
    j.c_out = cv->c_out;
    j.k = cv->k;
    j.stride = cv->stride;
    j.pad = cv->pad;
    j.up = cv->up;
    j.out_c_total = out_c_total;
    j.out_c_off = out_c_off;
    j.out_nchw = out_nchw;
    j.relu = cv->relu;
    j.round_out = cv->round_out;
    j.error = error_word;
    j.res = residual_nhwc;
    cudaError_t e = launch_conv_umma(j, static_cast<cudaStream_t>(stream));
    if (e == cudaErrorInvalidValue) return fail(PILLARS_E_UNSUPPORTED, "convolution geometry not instantiated");
    if (e != cudaSuccess) return cuda_fail(e, "conv_forward");
    g_launches_last = g_launches;
    return 0;
}

int pillars_conv_forward(const pillars_conv_t *cv, const void *image, const float *bn_shift, const float *in_nhwc,
                         const float *rows, const int32_t *cell_row, int32_t n_frames, int32_t h_in, int32_t w_in, float *out,
                         int32_t out_c_total, int32_t out_c_off, int32_t out_nchw, uint32_t *error_word, void *stream)
{
    return conv_forward(cv, image, bn_shift, in_nhwc, rows, cell_row, n_frames, h_in, w_in, out, out_c_total, out_c_off, out_nchw,
                        nullptr, error_word, stream);
}

int pillars_conv_forward_residual(const pillars_conv_t *cv, const void *image, const float *bn_shift, const float *in_nhwc,
                                  const float *rows, const int32_t *cell_row, int32_t n_frames, int32_t h_in, int32_t w_in,
                                  float *out, int32_t out_c_total, int32_t out_c_off, int32_t out_nchw, const float *residual_nhwc,
                                  uint32_t *error_word, void *stream)
{
    if (!residual_nhwc) return fail(PILLARS_E_BADARG, "NULL residual");
    if (cv && (cv->up != 1 || out_nchw != 0))
        return fail(PILLARS_E_UNSUPPORTED, "a residual is added only by a plain (not transposed) convolution with NHWC output");
    return conv_forward(cv, image, bn_shift, in_nhwc, rows, cell_row, n_frames, h_in, w_in, out, out_c_total, out_c_off, out_nchw,
                        residual_nhwc, error_word, stream);
}

int pillars_canvas_to_rows(const float *bev, int32_t n_frames, int32_t c, int32_t h, int32_t w, int32_t *cell_row, float *rows,
                           uint32_t *counter, void *stream)
{
    if (!bev || !cell_row || !rows || !counter) return fail(PILLARS_E_BADARG, "NULL argument");
    if (n_frames < 0 || c < 1 || h < 1 || w < 1) return fail(PILLARS_E_BADARG, "bad canvas shape");
    g_launches = 0;
    cudaError_t e = launch_canvas_to_rows(bev, n_frames, c, h, w, cell_row, rows, counter, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "canvas_to_rows");
    g_launches_last = g_launches;
    return 0;
}

size_t pillars_workspace_cell_row_offset(int64_t n_points, int32_t n_frames, const pillars_grid_t *grid)
{
    if (!grid || n_points < 0 || n_frames < 0) return 0;
    const int64_t cells_xy = static_cast<int64_t>(grid->grid[0]) * grid->grid[1];
    char *base = reinterpret_cast<char *>(static_cast<uintptr_t>(4096));  // any non-null base: only the offset is wanted
    const int64_t cells = cells_xy * grid->grid[2];
    const Workspace ws = carve_workspace(base, n_points, n_frames, cells_xy, cells,
                                         resolve_group_mode(true, n_points, n_frames, cells));
    return static_cast<size_t>(reinterpret_cast<char *>(ws.cell_row) - base);
}

}  // extern "C"
