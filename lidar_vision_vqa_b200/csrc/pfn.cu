// Per-pillar feature stage: augmentation + Linear + folded BatchNorm + ReLU + max over the pillar's points
// (replaces PillarVFE.forward / PFNLayer.forward, src/lidar-encoder/pcdet/models/backbones_3d/vfe/pillar_vfe.py:29-49,94-123).
//
// Work decomposition: 16 lanes own one pillar, each lane 4 of the 64 output channels with its 4 x C_in weights in
// registers; a warp therefore carries two pillars.  Points are never materialised as a padded [M,P,C] tensor: the
// fused path walks the pillar's index list straight into the raw point array; padded slots contribute the closed
// form relu(shift) (pillar_vfe.py:116-118 zeroes them BEFORE the linear, :39-42 lets them take part in the max).
// The 11 -> 64 contraction stays on the FMA pipes (memory/latency bound, no tensor cores).
// The same walk over the lists also serves the reference's padded outputs (k_emit_voxels) and MeanVFE (k_voxel_mean).
#include "common.cuh"

namespace pillars {

namespace {

constexpr int kThreads = 256;
constexpr int kLpp = 16;  // lanes per pillar
constexpr int kCpl = 4;   // channels per lane (F = 64)
constexpr unsigned kFull = 0xffffffffu;

struct FeatParams {
    const float *points;
    int stride, col0, idx_bits, c_point;
    GridDev gd;
    const Header *hdr;
    const uint32_t *pillar_key, *pillar_list, *pillar_cnt, *sorted_idx, *frame_gstart, *frame_rowbase;
    int32_t *cell_row;
    PfnDev pfn;
    float *pillar_features;
    int32_t *voxel_coords, *voxel_num_points, *point_pillar, *point_slot;
    float *voxels;
    int64_t capacity;
};

__device__ __forceinline__ uint32_t group_sum_u32(uint32_t v)
{
#pragma unroll
    for (int s = kLpp / 2; s > 0; s >>= 1) v += __shfl_xor_sync(kFull, v, s);
    return v;
}
__device__ __forceinline__ double group_sum_f64(double v)
{
#pragma unroll
    for (int s = kLpp / 2; s > 0; s >>= 1) v += __shfl_xor_sync(kFull, v, s);
    return v;
}

// Everything a consumer needs to know about pillar g.  Uniform inside a 16-lane group.
struct PillarInfo {
    bool live;       // in range and under the max_voxels cap (and the caller's capacity)
    uint32_t list;   // start of the point list
    uint32_t n;      // points that fell into the cell
    uint32_t thr;    // keep list entries with point index <= thr  (first-P rule)
    int32_t b, z, y, x;
    int64_t row;     // output row
};

// P-th smallest point index of a list by MSB-first radix select; all 32 lanes must call (shuffles inside).
__device__ __forceinline__ uint32_t select_threshold(const uint32_t *__restrict__ sorted_idx, uint32_t list, uint32_t n,
                                                     uint32_t want, bool need, int idx_bits, int sub)
{
    uint32_t prefix = 0, kk = want;
    for (int bit = idx_bits - 1; bit >= 0; --bit) {
        const uint32_t himask = 0xFFFFFFFFu << (bit + 1);  // bit <= 30
        uint32_t cnt0 = 0;
        if (need)
            for (uint32_t j = sub; j < n; j += kLpp) {
                const uint32_t v = sorted_idx[list + j];
                cnt0 += ((v & himask) == prefix && ((v >> bit) & 1u) == 0u) ? 1u : 0u;
            }
        cnt0 = group_sum_u32(cnt0);
        if (kk > cnt0) {
            prefix |= 1u << bit;
            kk -= cnt0;
        }
    }
    return need ? prefix : 0xFFFFFFFFu;
}

__device__ __forceinline__ PillarInfo resolve_pillar(const FeatParams &p, uint32_t g, uint32_t total, int sub)
{
    PillarInfo pi;
    const bool act = g < total;
    uint32_t key = 0;
    pi.list = 0;
    pi.n = 0;
    if (act) {
        key = p.pillar_key[g];
        pi.list = p.pillar_list[g];
        pi.n = p.pillar_cnt[g];
    }
    const uint32_t b = key / p.gd.cells;
    const uint32_t cell = key - b * p.gd.cells;
    const uint32_t z = cell / p.gd.cells_xy;
    const uint32_t rem = cell - z * p.gd.cells_xy;
    const uint32_t y = rem / static_cast<uint32_t>(p.gd.g[0]);
    pi.b = static_cast<int32_t>(b);
    pi.z = static_cast<int32_t>(z);
    pi.y = static_cast<int32_t>(y);
    pi.x = static_cast<int32_t>(rem - y * static_cast<uint32_t>(p.gd.g[0]));
    uint32_t local = 0;
    pi.row = 0;
    if (act) {
        local = g - p.frame_gstart[b];
        pi.row = static_cast<int64_t>(p.frame_rowbase[b]) + local;
    }
    pi.live = act && local < static_cast<uint32_t>(p.gd.max_voxels) && pi.row < p.capacity;
    const bool need = pi.live && pi.n > static_cast<uint32_t>(p.gd.max_points);
    pi.thr = 0xFFFFFFFFu;
    if (__any_sync(kFull, need))
        pi.thr = select_threshold(p.sorted_idx, pi.list, pi.n, static_cast<uint32_t>(p.gd.max_points), need,
                                  p.idx_bits, sub);
    return pi;
}

template <int C, bool ABS, bool DIST>
struct FeatDims {
    static constexpr int kCin = (ABS ? C : C - 3) + 6 + (DIST ? 1 : 0);
};

// one point through augmentation + linear + BN + ReLU, folded into the running max
template <int C, bool ABS, bool DIST>
__device__ __forceinline__ void accumulate_point(const float (&pt)[C], float mx, float my, float mz, float cx, float cy,
                                                 float cz, const float (&w)[FeatDims<C, ABS, DIST>::kCin][kCpl],
                                                 const float (&scale)[kCpl], const float (&shift)[kCpl],
                                                 float (&best)[kCpl])
{
    constexpr int kCin = FeatDims<C, ABS, DIST>::kCin;
    float f[kCin];
    int q = 0;
#pragma unroll
    for (int c = (ABS ? 0 : 3); c < C; ++c) f[q++] = pt[c];
    f[q++] = __fsub_rn(pt[0], mx);  // f_cluster  (pillar_vfe.py:98)
    f[q++] = __fsub_rn(pt[1], my);
    f[q++] = __fsub_rn(pt[2], mz);
    f[q++] = __fsub_rn(pt[0], cx);  // f_center   (pillar_vfe.py:100-103)
    f[q++] = __fsub_rn(pt[1], cy);
    f[q++] = __fsub_rn(pt[2], cz);
    if (DIST) f[q++] = sqrtf(pt[0] * pt[0] + pt[1] * pt[1] + pt[2] * pt[2]);  // pillar_vfe.py:110-112
#pragma unroll
    for (int o = 0; o < kCpl; ++o) {
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < kCin; ++k) acc = fmaf(f[k], w[k][o], acc);
        const float yv = fmaxf(fmaf(acc, scale[o], shift[o]), 0.f);
        best[o] = fmaxf(best[o], yv);
    }
}

template <int C, bool ABS, bool DIST>
__device__ __forceinline__ void load_weights(const PfnDev &pfn, int sub, float (&w)[FeatDims<C, ABS, DIST>::kCin][kCpl],
                                             float (&scale)[kCpl], float (&shift)[kCpl])
{
    constexpr int kCin = FeatDims<C, ABS, DIST>::kCin;
#pragma unroll
    for (int o = 0; o < kCpl; ++o) {
        const int ch = sub * kCpl + o;
#pragma unroll
        for (int k = 0; k < kCin; ++k) w[k][o] = __ldg(pfn.weight + ch * kCin + k);
        scale[o] = __ldg(pfn.scale + ch);
        shift[o] = __ldg(pfn.shift + ch);
    }
}

// ---------------------------------------------------------------------------------------------
// fused path: pillar lists over raw points
// ---------------------------------------------------------------------------------------------
template <int C, bool ABS, bool DIST>
__global__ void __launch_bounds__(kThreads, 2) k_pillar_features(const FeatParams p)
{
    constexpr int kCin = FeatDims<C, ABS, DIST>::kCin;
    const int lane = threadIdx.x & 31, sub = lane & (kLpp - 1), grp = lane / kLpp;
    const int warp = threadIdx.x >> 5;
    constexpr int kGroupsPerWarp = 32 / kLpp;

    float w[kCin][kCpl], scale[kCpl], shift[kCpl];
    load_weights<C, ABS, DIST>(p.pfn, sub, w, scale, shift);

    const uint32_t total = p.hdr->total_pillars;
    const uint32_t warp_stride = gridDim.x * (kThreads / 32) * kGroupsPerWarp;
    for (uint32_t gbase = (blockIdx.x * (kThreads / 32) + warp) * kGroupsPerWarp; gbase < total; gbase += warp_stride) {
        const uint32_t g = gbase + grp;
        const PillarInfo pi = resolve_pillar(p, g, total, sub);
        const uint32_t n_eff = pi.live ? pi.n : 0u;
        const uint32_t n_keep = min(n_eff, static_cast<uint32_t>(p.gd.max_points));

        // pass 1: mean of the kept points (double accumulation => independent of list order)
        double sx = 0.0, sy = 0.0, sz = 0.0;
        for (uint32_t j = sub; j < n_eff; j += kLpp) {
            const uint32_t idx = p.sorted_idx[pi.list + j];
            if (idx <= pi.thr) {
                const float *pt = p.points + static_cast<int64_t>(idx) * p.stride + p.col0;
                sx += static_cast<double>(__ldg(pt));
                sy += static_cast<double>(__ldg(pt + 1));
                sz += static_cast<double>(__ldg(pt + 2));
            }
        }
        sx = group_sum_f64(sx);
        sy = group_sum_f64(sy);
        sz = group_sum_f64(sz);
        const float nf = static_cast<float>(n_keep);
        const float mx = __fdiv_rn(static_cast<float>(sx), nf);  // pillar_vfe.py:97
        const float my = __fdiv_rn(static_cast<float>(sy), nf);
        const float mz = __fdiv_rn(static_cast<float>(sz), nf);
        // pillar centre: coord * voxel + offset, two roundings as in the reference (no FMA)
        const float cx = __fadd_rn(__fmul_rn(static_cast<float>(pi.x), p.pfn.vsz[0]), p.pfn.off[0]);
        const float cy = __fadd_rn(__fmul_rn(static_cast<float>(pi.y), p.pfn.vsz[1]), p.pfn.off[1]);
        const float cz = __fadd_rn(__fmul_rn(static_cast<float>(pi.z), p.pfn.vsz[2]), p.pfn.off[2]);

        float best[kCpl];
#pragma unroll
        for (int o = 0; o < kCpl; ++o)
            best[o] = (n_keep < static_cast<uint32_t>(p.gd.max_points)) ? fmaxf(shift[o], 0.f) : 0.f;

        // pass 2: 16 list entries at a time, one per lane, then broadcast point by point inside the group
        uint32_t n_warp = max(n_eff, __shfl_xor_sync(kFull, n_eff, kLpp));
        for (uint32_t c0 = 0; c0 < n_warp; c0 += kLpp) {
            const uint32_t j = c0 + sub;
            bool mine = false;
            float pr[C];
#pragma unroll
            for (int c = 0; c < C; ++c) pr[c] = 0.f;
            if (j < n_eff) {
                const uint32_t idx = p.sorted_idx[pi.list + j];
                if (idx <= pi.thr) {
                    mine = true;
                    const float *pt = p.points + static_cast<int64_t>(idx) * p.stride + p.col0;
#pragma unroll
                    for (int c = 0; c < C; ++c) pr[c] = __ldg(pt + c);
                }
            }
            const int lim = static_cast<int>(min(static_cast<uint32_t>(kLpp), n_warp - c0));
            for (int jj = 0; jj < lim; ++jj) {
                const bool has = __shfl_sync(kFull, mine, jj, kLpp);
                float pt[C];
#pragma unroll
                for (int c = 0; c < C; ++c) pt[c] = __shfl_sync(kFull, pr[c], jj, kLpp);
                if (has) accumulate_point<C, ABS, DIST>(pt, mx, my, mz, cx, cy, cz, w, scale, shift, best);
            }
        }

        if (pi.live) {
            float4 o4 = make_float4(best[0], best[1], best[2], best[3]);
            *reinterpret_cast<float4 *>(p.pillar_features + pi.row * (kLpp * kCpl) + sub * kCpl) = o4;
            if (sub == 0) {
                if (p.voxel_coords)
                    *reinterpret_cast<int4 *>(p.voxel_coords + pi.row * 4) = make_int4(pi.b, pi.z, pi.y, pi.x);
                if (p.voxel_num_points) p.voxel_num_points[pi.row] = static_cast<int32_t>(n_keep);
                if (p.cell_row)
                    p.cell_row[static_cast<int64_t>(pi.b) * p.gd.cells_xy + static_cast<int64_t>(pi.y) * p.gd.g[0] +
                               pi.x] = static_cast<int32_t>(pi.row);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// grouping outputs in the reference's own format: voxels [M,P,C] zero padded, coords, counts, membership
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_emit_voxels(const FeatParams p)
{
    const int lane = threadIdx.x & 31, sub = lane & (kLpp - 1), grp = lane / kLpp;
    const int warp = threadIdx.x >> 5;
    constexpr int kGroupsPerWarp = 32 / kLpp;
    const uint32_t total = p.hdr->total_pillars;
    const uint32_t warp_stride = gridDim.x * (kThreads / 32) * kGroupsPerWarp;
    const int P = p.gd.max_points, C = p.c_point;
    for (uint32_t gbase = (blockIdx.x * (kThreads / 32) + warp) * kGroupsPerWarp; gbase < total; gbase += warp_stride) {
        const uint32_t g = gbase + grp;
        const PillarInfo pi = resolve_pillar(p, g, total, sub);
        if (!pi.live) continue;  // no shuffles below
        const uint32_t n_keep = min(pi.n, static_cast<uint32_t>(P));
        for (uint32_t j = sub; j < pi.n; j += kLpp) {
            const uint32_t idx = p.sorted_idx[pi.list + j];
            int32_t slot = -1;
            if (idx <= pi.thr) {
                uint32_t rank = 0;  // kept entries are exactly the n_keep smallest: rank among all == rank among kept
                for (uint32_t t = 0; t < pi.n; ++t) rank += (p.sorted_idx[pi.list + t] < idx) ? 1u : 0u;
                slot = static_cast<int32_t>(rank);
                if (p.voxels) {
                    const float *src = p.points + static_cast<int64_t>(idx) * p.stride + p.col0;
                    float *dst = p.voxels + (pi.row * P + rank) * C;
                    for (int c = 0; c < C; ++c) dst[c] = __ldg(src + c);
                }
            }
            if (p.point_pillar) p.point_pillar[idx] = static_cast<int32_t>(pi.row);
            if (p.point_slot) p.point_slot[idx] = slot;
        }
        if (p.voxels) {
            float *dst = p.voxels + (pi.row * P + n_keep) * C;
            const uint32_t pad = (static_cast<uint32_t>(P) - n_keep) * C;
            for (uint32_t t = sub; t < pad; t += kLpp) dst[t] = 0.f;
        }
        if (sub == 0) {
            if (p.voxel_coords) *reinterpret_cast<int4 *>(p.voxel_coords + pi.row * 4) = make_int4(pi.b, pi.z, pi.y, pi.x);
            if (p.voxel_num_points) p.voxel_num_points[pi.row] = static_cast<int32_t>(n_keep);
            if (p.cell_row)
                p.cell_row[static_cast<int64_t>(pi.b) * p.gd.cells_xy + static_cast<int64_t>(pi.y) * p.gd.g[0] + pi.x] =
                    static_cast<int32_t>(pi.row);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// MeanVFE (models/backbones_3d/vfe/mean_vfe.py:14-31) straight from the lists, without the padded [M,P,C] tensor:
//   voxel_mean[row][c] = (sequential fp32 sum of the reference's P slots of channel c) / max(n_keep, 1)
// Slot s holds the kept point of rank s (kept = the n_keep smallest indices of the list, the hard voxeliser's first-P rule),
// and the padding slots hold +0.0.  So the sum adds the kept points in increasing point index, then one +0.0 when padding
// follows: that changes nothing but the sign of a -0.0 sum, exactly as the padding does.  A 16-lane group ranks its kept
// entries (atomic arrival order is no order at all), puts their point indices into shared memory by rank, and lane c then
// adds channel c slot after slot.  No atomics: the result depends on the points alone.
// ---------------------------------------------------------------------------------------------
struct MeanParams {
    FeatParams f;  // pillar_features, voxels and the membership outputs are not used
    float *mean;   // [capacity, c_point]
};

__global__ void __launch_bounds__(kThreads) k_voxel_mean(const __grid_constant__ MeanParams mp)
{
    extern __shared__ uint32_t s_slot[];  // [kThreads / kLpp][P]: point index in each kept slot of the group's voxel
    const FeatParams &p = mp.f;
    const int lane = threadIdx.x & 31, sub = lane & (kLpp - 1), grp = lane / kLpp;
    const int warp = threadIdx.x >> 5;
    constexpr int kGroupsPerWarp = 32 / kLpp;
    const int P = p.gd.max_points, C = p.c_point;
    uint32_t *slot = s_slot + (warp * kGroupsPerWarp + grp) * P;
    pdl_wait();
    pdl_trigger();
    const uint32_t total = p.hdr->total_pillars;
    const uint32_t warp_stride = gridDim.x * (kThreads / 32) * kGroupsPerWarp;
    for (uint32_t gbase = (blockIdx.x * (kThreads / 32) + warp) * kGroupsPerWarp; gbase < total; gbase += warp_stride) {
        const uint32_t g = gbase + grp;
        const PillarInfo pi = resolve_pillar(p, g, total, sub);
        const uint32_t n_eff = pi.live ? pi.n : 0u;
        const uint32_t n_keep = min(n_eff, static_cast<uint32_t>(P));
        for (uint32_t j = sub; j < n_eff; j += kLpp) {
            const uint32_t idx = p.sorted_idx[pi.list + j];
            if (idx <= pi.thr) {
                uint32_t rank = 0;  // kept entries are exactly the n_keep smallest: rank among all == rank among kept
                for (uint32_t t = 0; t < n_eff; ++t) rank += (p.sorted_idx[pi.list + t] < idx) ? 1u : 0u;
                slot[rank] = idx;
            }
        }
        __syncwarp();
        if (pi.live) {
            // (check_points caps row_stride at 16, so one pass covers every channel; the loop keeps any C correct)
            for (int c = sub; c < C; c += kLpp) {
                const float *col = p.points + p.col0 + c;
                float acc = __ldg(col + static_cast<int64_t>(slot[0]) * p.stride);
#pragma unroll 4
                for (uint32_t r = 1; r < n_keep; ++r) acc = __fadd_rn(acc, __ldg(col + static_cast<int64_t>(slot[r]) * p.stride));
                if (n_keep < static_cast<uint32_t>(P)) acc = __fadd_rn(acc, 0.f);  // the padding slots
                mp.mean[pi.row * C + c] = __fdiv_rn(acc, static_cast<float>(max(n_keep, 1u)));
            }
            if (sub == 0) {
                if (p.voxel_coords) *reinterpret_cast<int4 *>(p.voxel_coords + pi.row * 4) = make_int4(pi.b, pi.z, pi.y, pi.x);
                if (p.voxel_num_points) p.voxel_num_points[pi.row] = static_cast<int32_t>(n_keep);
            }
        }
        __syncwarp();  // the slots are rewritten by the next voxel
    }
}

// ---------------------------------------------------------------------------------------------
// hard variant: the reference's own padded input  voxels [M,P,C], num_points [M], coords [M,4] (b,z,y,x)
// ---------------------------------------------------------------------------------------------
struct DenseParams {
    const float *voxels;
    const void *num_points;
    const void *coords;
    int np_float, coords_float;
    int64_t m;
    int max_points;
    PfnDev pfn;
    float *out;
};

template <int C, bool ABS, bool DIST>
__global__ void __launch_bounds__(kThreads, 2) k_pfn_dense(const DenseParams p)
{
    constexpr int kCin = FeatDims<C, ABS, DIST>::kCin;
    const int lane = threadIdx.x & 31, sub = lane & (kLpp - 1), grp = lane / kLpp;
    const int warp = threadIdx.x >> 5;
    constexpr int kGroupsPerWarp = 32 / kLpp;
    float w[kCin][kCpl], scale[kCpl], shift[kCpl];
    load_weights<C, ABS, DIST>(p.pfn, sub, w, scale, shift);
    const int P = p.max_points;
    const int64_t warp_stride = static_cast<int64_t>(gridDim.x) * (kThreads / 32) * kGroupsPerWarp;
    for (int64_t gbase = (static_cast<int64_t>(blockIdx.x) * (kThreads / 32) + warp) * kGroupsPerWarp; gbase < p.m;
         gbase += warp_stride) {
        const int64_t g = gbase + grp;
        const bool act = g < p.m;
        int n = 0;
        float nf = 1.f, fx = 0.f, fy = 0.f, fz = 0.f;
        if (act) {
            if (p.np_float) {
                nf = static_cast<const float *>(p.num_points)[g];
                n = static_cast<int>(nf);  // .int() in get_paddings_indicator (pillar_vfe.py:91)
            } else {
                n = static_cast<const int32_t *>(p.num_points)[g];
                nf = static_cast<float>(n);  // .type_as(voxel_features) (pillar_vfe.py:97)
            }
            if (p.coords_float) {
                const float4 c4 = *reinterpret_cast<const float4 *>(static_cast<const float *>(p.coords) + g * 4);
                fz = c4.y; fy = c4.z; fx = c4.w;
            } else {
                const int4 c4 = *reinterpret_cast<const int4 *>(static_cast<const int32_t *>(p.coords) + g * 4);
                fz = static_cast<float>(c4.y); fy = static_cast<float>(c4.z); fx = static_cast<float>(c4.w);
            }
        }
        const int n_valid = act ? max(0, min(n, P)) : 0;
        const float *vox = p.voxels + g * P * C;
        // pass 1: the reference sums ALL P slots (pillar_vfe.py:97), whatever the padding holds
        float sx = 0.f, sy = 0.f, sz = 0.f;
        if (act)
            for (int j = sub; j < P; j += kLpp) {
                sx += __ldg(vox + j * C);
                sy += __ldg(vox + j * C + 1);
                sz += __ldg(vox + j * C + 2);
            }
#pragma unroll
        for (int s = kLpp / 2; s > 0; s >>= 1) {
            sx += __shfl_xor_sync(kFull, sx, s);
            sy += __shfl_xor_sync(kFull, sy, s);
            sz += __shfl_xor_sync(kFull, sz, s);
        }
        const float mx = __fdiv_rn(sx, nf), my = __fdiv_rn(sy, nf), mz = __fdiv_rn(sz, nf);
        const float cx = __fadd_rn(__fmul_rn(fx, p.pfn.vsz[0]), p.pfn.off[0]);
        const float cy = __fadd_rn(__fmul_rn(fy, p.pfn.vsz[1]), p.pfn.off[1]);
        const float cz = __fadd_rn(__fmul_rn(fz, p.pfn.vsz[2]), p.pfn.off[2]);
        float best[kCpl];
#pragma unroll
        for (int o = 0; o < kCpl; ++o) best[o] = (n_valid < P) ? fmaxf(shift[o], 0.f) : 0.f;

        const int n_warp = max(n_valid, __shfl_xor_sync(kFull, n_valid, kLpp));
        for (int c0 = 0; c0 < n_warp; c0 += kLpp) {
            const int j = c0 + sub;
            float pr[C];
#pragma unroll
            for (int c = 0; c < C; ++c) pr[c] = 0.f;
            const bool mine = j < n_valid;
            if (mine) {
#pragma unroll
                for (int c = 0; c < C; ++c) pr[c] = __ldg(vox + j * C + c);
            }
            const int lim = min(kLpp, n_warp - c0);
            for (int jj = 0; jj < lim; ++jj) {
                const bool has = __shfl_sync(kFull, mine, jj, kLpp);
                float pt[C];
#pragma unroll
                for (int c = 0; c < C; ++c) pt[c] = __shfl_sync(kFull, pr[c], jj, kLpp);
                if (has) accumulate_point<C, ABS, DIST>(pt, mx, my, mz, cx, cy, cz, w, scale, shift, best);
            }
        }
        if (act)
            *reinterpret_cast<float4 *>(p.out + g * (kLpp * kCpl) + sub * kCpl) =
                make_float4(best[0], best[1], best[2], best[3]);
    }
}

int grid_for(int64_t groups, int sms_x)
{
    const int64_t groups_per_block = (kThreads / kLpp);
    int64_t blocks = (groups + groups_per_block - 1) / groups_per_block;
    const int64_t cap = static_cast<int64_t>(sms_x);
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return static_cast<int>(blocks);
}

int num_sms() { return current_sm_count(); }  // per device (a process may drive more than one)

template <int C>
cudaError_t dispatch_features(const FeatParams &p, bool abs_xyz, bool dist, int grid, cudaStream_t st)
{
    if (abs_xyz && !dist) k_pillar_features<C, true, false><<<grid, kThreads, 0, st>>>(p);
    else if (abs_xyz && dist) k_pillar_features<C, true, true><<<grid, kThreads, 0, st>>>(p);
    else if (!abs_xyz && !dist) k_pillar_features<C, false, false><<<grid, kThreads, 0, st>>>(p);
    else k_pillar_features<C, false, true><<<grid, kThreads, 0, st>>>(p);
    return cudaGetLastError();
}

template <int C>
cudaError_t dispatch_dense(const DenseParams &p, bool abs_xyz, bool dist, int grid, cudaStream_t st)
{
    if (abs_xyz && !dist) k_pfn_dense<C, true, false><<<grid, kThreads, 0, st>>>(p);
    else if (abs_xyz && dist) k_pfn_dense<C, true, true><<<grid, kThreads, 0, st>>>(p);
    else if (!abs_xyz && !dist) k_pfn_dense<C, false, false><<<grid, kThreads, 0, st>>>(p);
    else k_pfn_dense<C, false, true><<<grid, kThreads, 0, st>>>(p);
    return cudaGetLastError();
}

FeatParams make_feat_params(const FeatureJob &job, const GridDev &gd, const Workspace &ws)
{
    FeatParams p{};
    p.points = job.points;
    p.stride = job.stride;
    p.col0 = job.col0;
    p.idx_bits = job.idx_bits;
    p.c_point = job.c_point;
    p.gd = gd;
    p.hdr = ws.hdr;
    p.pillar_key = ws.pillar_key;
    p.pillar_list = ws.pillar_list;
    p.pillar_cnt = ws.pillar_cnt;
    p.sorted_idx = ws.sorted_idx;
    p.frame_gstart = ws.frame_gstart;
    p.frame_rowbase = ws.frame_rowbase;
    p.cell_row = job.write_cell_row ? ws.cell_row : nullptr;
    p.pfn = job.pfn;
    p.pillar_features = job.out.pillar_features;
    p.voxel_coords = job.out.voxel_coords;
    p.voxel_num_points = job.out.voxel_num_points;
    p.point_pillar = job.out.point_pillar;
    p.point_slot = job.out.point_slot;
    p.voxels = job.out.voxels;
    p.capacity = job.out.pillar_capacity;
    return p;
}

}  // namespace

cudaError_t launch_pillar_features(const FeatureJob &job, const GridDev &gd, const Workspace &ws, cudaStream_t st)
{
    const FeatParams p = make_feat_params(job, gd, ws);
    if (job.n == 0) return cudaSuccess;

    // persistent grids: the pillar count lives on the device, so size for the SM count and stride
    const int grid = grid_for(job.n, num_sms() * 8);
    cudaError_t err = cudaSuccess;
    const bool membership = job.out.voxels || job.out.point_pillar || job.out.point_slot;
    if (membership || !job.do_features) {
        FeatParams pe = p;
        if (job.do_features) pe.cell_row = nullptr;  // written once, by the feature kernel
        k_emit_voxels<<<grid, kThreads, 0, st>>>(pe);
        note_launch();
        if ((err = cudaGetLastError()) != cudaSuccess) return err;
    }
    if (job.do_features) {
        switch (job.c_point) {
            case 3: err = dispatch_features<3>(p, job.use_abs, job.with_dist, grid, st); break;
            case 4: err = dispatch_features<4>(p, job.use_abs, job.with_dist, grid, st); break;
            case 5: err = dispatch_features<5>(p, job.use_abs, job.with_dist, grid, st); break;
            case 6: err = dispatch_features<6>(p, job.use_abs, job.with_dist, grid, st); break;
            default: return cudaErrorInvalidValue;
        }
        note_launch();
    }
    return err;
}

cudaError_t launch_voxel_mean(const FeatureJob &job, float *voxel_mean, const GridDev &gd, const Workspace &ws,
                              cudaStream_t st)
{
    if (job.n == 0) return cudaSuccess;
    if (gd.max_points > kMeanMaxPoints) return cudaErrorInvalidValue;
    const MeanParams mp{make_feat_params(job, gd, ws), voxel_mean};
    const size_t smem = sizeof(uint32_t) * (kThreads / kLpp) * gd.max_points;
    const cudaError_t err = launch_pdl(k_voxel_mean, dim3(grid_for(job.n, num_sms() * 8)), dim3(kThreads), smem, st, mp);
    note_launch();
    return err;
}

cudaError_t launch_pfn_dense(const float *voxels, const void *num_points, bool np_float, const void *coords,
                             bool coords_float, int64_t m, int max_points, int c_point, bool use_abs, bool with_dist,
                             const PfnDev &pfn, float *out, cudaStream_t st)
{
    if (m == 0) return cudaSuccess;
    DenseParams p{};
    p.voxels = voxels;
    p.num_points = num_points;
    p.coords = coords;
    p.np_float = np_float;
    p.coords_float = coords_float;
    p.m = m;
    p.max_points = max_points;
    p.pfn = pfn;
    p.out = out;
    const int grid = grid_for(m, num_sms() * 8);
    cudaError_t err;
    switch (c_point) {
        case 3: err = dispatch_dense<3>(p, use_abs, with_dist, grid, st); break;
        case 4: err = dispatch_dense<4>(p, use_abs, with_dist, grid, st); break;
        case 5: err = dispatch_dense<5>(p, use_abs, with_dist, grid, st); break;
        case 6: err = dispatch_dense<6>(p, use_abs, with_dist, grid, st); break;
        default: return cudaErrorInvalidValue;
    }
    note_launch();
    return err;
}

}  // namespace pillars
