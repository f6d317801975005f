// General pillar feature stack: every PFN configuration of the reference that the streaming kernel (pfn_stream.cu) does not
// cover, behind one kernel.
//
//   * PillarVFE with NUM_FILTERS of two entries, e.g. [64, 64] (waymo_models/pointpillar_1x.yaml:34): layer 0 has
//     NUM_FILTERS[0] / 2 outputs, its per-point output is concatenated with the pillar-wise max and fed to layer 1
//     (src/lidar-encoder/pcdet/models/backbones_3d/vfe/pillar_vfe.py:18-19,44-49,119-120).  Padded slots are zeroed once,
//     before layer 0 (:115-118), and are NOT re-masked between layers, so a pillar with n < P points carries one more row
//     whose augmented features are all zero through the whole stack, max included.
//   * DynamicPillarVFE / PFNLayerV2 (models/backbones_3d/vfe/dynamic_pillar_vfe.py:14-142): no per-pillar cap, no padded
//     rows, z is not range checked, f_center_z = z - z_offset, rows ordered by the merged key b*nx*ny + ix*ny + iy,
//     voxel_coords = (b, 0, iy, ix).
//   * DynamicPillarVFESimple2D (:145-240): features [f_center, point channels (, distance)], no cluster offset,
//     NUM_FILTERS [32], pillar_coords = (b, iy, ix).
//   * PillarVFE on the reference's padded `voxels [M,P,C]` input with two layers.
//
// Mapping: one warp per pillar.  A lane owns output channel `lane` (and `lane + 32` when a layer has more than 32 outputs);
// weights live in shared memory, transposed to [input][output] so the lanes of a warp read consecutive words.  The
// augmented feature vector of a point is built by the first C_in lanes (one feature each) and exchanged through a small
// per-warp shared buffer; layer 0 outputs reach layer 1 the same way.  For two layers the pillar is walked twice (first
// the max of layer 0, then layer 1 on [x, max]) and layer 0 is recomputed instead of stored, so pillars of any length
// (the dynamic variant has no cap) need no scratch.  Not the headline kernel: it exists for coverage and is bound by
// shared-memory traffic; the mainstream single-layer configuration runs pfn_stream.cu.
#include "common.cuh"

namespace pillars {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kMaxIn0 = 16;   // C_in of layer 0
constexpr int kMaxOut = 64;   // outputs of any layer
constexpr int kMaxIn1 = 64;   // inputs of layer 1 = 2 * outputs of layer 0
constexpr int kKeepMax = 128; // kept point indices compacted per warp when a capped pillar is longer than that

enum FeatKind : int { kPoint = 0, kCluster = 1, kCentre = 2, kDist = 3 };

struct MultiParams {
    // source A: pillar lists over raw points (grouping workspace)
    const float *points;
    int stride, col0, c_point, idx_bits;
    GridDev gd;
    const Header *hdr;
    const uint32_t *pillar_key, *pillar_list, *pillar_cnt, *sorted_idx, *frame_gstart, *frame_rowbase;
    const uint32_t *rank_xmajor;  // dynamic: [B * nx * ny] exclusive rank of the cell in (b, ix, iy) order; else NULL
    // source B: the reference's padded voxels
    const float *voxels;
    const void *num_points, *coords;
    int np_float, coords_float;
    int64_t m;
    int dense;    // 1: source B
    int dynamic;  // 1: DynamicPillarVFE semantics
    // feature layout of layer 0 and the stack
    int c_in, n_layers, out0, out1;
    int kind[kMaxIn0], arg[kMaxIn0];
    const float *w0, *s0, *h0, *w1, *s1, *h1;
    float vsz[3], off[3];
    int max_points;
    // outputs
    float *pillar_features;
    int32_t *voxel_coords, *voxel_num_points, *cell_row;
    int coords_cols;  // 4: (b,z,y,x)   3: (b,y,x)
    int64_t capacity;
};

struct Pillar {
    bool live;
    uint32_t list, n_all, n_keep, thr;
    int32_t b, z, y, x;
    int64_t row;
    float nf;  // divisor of the mean
};

__device__ __forceinline__ uint32_t warp_sum_u32(uint32_t v)
{
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(kFull, v, s);
    return v;
}
__device__ __forceinline__ double warp_sum_f64(double v)
{
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(kFull, v, s);
    return v;
}
__device__ __forceinline__ float warp_sum_f32(float v)
{
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(kFull, v, s);
    return v;
}

struct PillarCtx {
    Pillar pi;
    const float *vox;   // dense source: the pillar's padded rows
    bool compact;       // kept point indices were compacted into the warp's shared list
    uint32_t n_iter;    // list entries (or rows) to visit
    float mx, my, mz;   // mean of the kept points
    float cx, cy, cz;   // pillar centre
};

// t-th list entry of the pillar -> pointer to the point's channels, or NULL when the entry is beyond the first-P cap
__device__ __forceinline__ const float *pillar_point(const MultiParams &p, const PillarCtx &c, const uint32_t *keep, uint32_t t)
{
    if (p.dense) return c.vox + static_cast<int64_t>(t) * p.c_point;
    const uint32_t idx = c.compact ? keep[t] : p.sorted_idx[c.pi.list + t];
    if (idx > c.pi.thr) return nullptr;
    return p.points + static_cast<int64_t>(idx) * p.stride + p.col0;
}

// Everything about pillar g that does not depend on the feature stack (warp-uniform): row, coordinates, the kept subset
// under the first-P rule, mean, centre.  Returns false for a pillar that produces no output.  All 32 lanes must call.
__device__ __forceinline__ bool prepare_pillar(const MultiParams &p, int64_t g, int lane, uint32_t *keep, PillarCtx &c)
{
    const uint32_t P = static_cast<uint32_t>(p.max_points);
    {
        // ---- resolve the pillar (warp-uniform) -----------------------------------------------------------------------
        Pillar &pi = c.pi;
        pi = Pillar{};
        pi.thr = 0xFFFFFFFFu;
        c.vox = nullptr;
        if (p.dense) {
            int n;
            if (p.np_float) {
                pi.nf = static_cast<const float *>(p.num_points)[g];
                n = static_cast<int>(pi.nf);  // .int() in get_paddings_indicator (pillar_vfe.py:91)
            } else {
                n = static_cast<const int32_t *>(p.num_points)[g];
                pi.nf = static_cast<float>(n);
            }
            float fz, fy, fx;
            if (p.coords_float) {
                const float4 c4 = *reinterpret_cast<const float4 *>(static_cast<const float *>(p.coords) + g * 4);
                fz = c4.y; fy = c4.z; fx = c4.w;
            } else {
                const int4 c4 = *reinterpret_cast<const int4 *>(static_cast<const int32_t *>(p.coords) + g * 4);
                fz = static_cast<float>(c4.y); fy = static_cast<float>(c4.z); fx = static_cast<float>(c4.w);
            }
            pi.z = static_cast<int32_t>(fz); pi.y = static_cast<int32_t>(fy); pi.x = static_cast<int32_t>(fx);
            pi.n_keep = static_cast<uint32_t>(max(0, min(n, static_cast<int>(P))));
            pi.n_all = pi.n_keep;
            pi.row = g;
            pi.live = true;
            c.vox = p.voxels + g * static_cast<int64_t>(P) * p.c_point;
        } else {
            const uint32_t key = p.pillar_key[g];
            pi.list = p.pillar_list[g];
            pi.n_all = p.pillar_cnt[g];
            const uint32_t b = key / p.gd.cells;
            const uint32_t cell = key - b * p.gd.cells;
            const uint32_t z = cell / p.gd.cells_xy;
            const uint32_t rem = cell - z * p.gd.cells_xy;
            const uint32_t y = rem / static_cast<uint32_t>(p.gd.g[0]);
            const uint32_t x = rem - y * static_cast<uint32_t>(p.gd.g[0]);
            pi.b = static_cast<int32_t>(b); pi.z = static_cast<int32_t>(z);
            pi.y = static_cast<int32_t>(y); pi.x = static_cast<int32_t>(x);
            if (p.dynamic) {
                // rows in the order torch.unique gives the merged key b*nx*ny + ix*ny + iy (dynamic_pillar_vfe.py:99-103)
                pi.row = p.rank_xmajor[static_cast<size_t>(b) * p.gd.cells_xy + static_cast<size_t>(x) * p.gd.g[1] + y] & 0x7FFFFFFFu;
                pi.live = pi.row < p.capacity;
                pi.n_keep = pi.n_all;
            } else {
                const uint32_t local = static_cast<uint32_t>(g) - p.frame_gstart[b];
                pi.row = static_cast<int64_t>(p.frame_rowbase[b]) + local;
                pi.live = local < static_cast<uint32_t>(p.gd.max_voxels) && pi.row < p.capacity;
                pi.n_keep = min(pi.n_all, P);
                if (pi.live && pi.n_all > P) {  // first-P rule: P-th smallest point index by radix select
                    uint32_t prefix = 0, kk = P;
                    for (int bit = p.idx_bits - 1; bit >= 0; --bit) {
                        const uint32_t himask = 0xFFFFFFFFu << (bit + 1);
                        uint32_t c0 = 0;
                        for (uint32_t j = lane; j < pi.n_all; j += 32) {
                            const uint32_t v = p.sorted_idx[pi.list + j];
                            c0 += ((v & himask) == prefix && ((v >> bit) & 1u) == 0u) ? 1u : 0u;
                        }
                        c0 = warp_sum_u32(c0);
                        if (kk > c0) {
                            prefix |= 1u << bit;
                            kk -= c0;
                        }
                    }
                    pi.thr = prefix;
                }
            }
            pi.nf = static_cast<float>(pi.n_keep);
        }
        if (!pi.live) return false;

        // a capped pillar much longer than the cap: compact the kept indices once instead of filtering in every pass
        c.compact = false;
        if (!p.dense && !p.dynamic && pi.n_all > P && pi.n_all > 64 && P <= static_cast<uint32_t>(kKeepMax)) {
            uint32_t base = 0;
            for (uint32_t j0 = 0; j0 < pi.n_all; j0 += 32) {
                const uint32_t j = j0 + lane;
                uint32_t idx = 0xFFFFFFFFu;
                if (j < pi.n_all) idx = p.sorted_idx[pi.list + j];
                const bool k = j < pi.n_all && idx <= pi.thr;
                const unsigned bal = __ballot_sync(kFull, k);
                if (k) keep[base + __popc(bal & ((1u << lane) - 1u))] = idx;
                base += __popc(bal);
            }
            __syncwarp();
            c.compact = true;
        }
        c.n_iter = p.dense ? pi.n_keep : (c.compact ? pi.n_keep : pi.n_all);
        const uint32_t n_iter = c.n_iter;
        const float *vox = c.vox;
        auto point_at = [&](uint32_t t) -> const float * { return pillar_point(p, c, keep, t); };

        // ---- mean of the pillar (pillar_vfe.py:97 / scatter_mean, dynamic_pillar_vfe.py:105) --------------------------
        float &mx = c.mx, &my = c.my, &mz = c.mz;
        mx = my = mz = 0.f;
        {
            if (p.dense) {  // the reference sums ALL P slots in fp32, whatever the padding holds
                float sx = 0.f, sy = 0.f, sz = 0.f;
                for (uint32_t j = lane; j < P; j += 32) {
                    const float *q = vox + static_cast<int64_t>(j) * p.c_point;
                    sx += __ldg(q); sy += __ldg(q + 1); sz += __ldg(q + 2);
                }
                mx = __fdiv_rn(warp_sum_f32(sx), pi.nf);
                my = __fdiv_rn(warp_sum_f32(sy), pi.nf);
                mz = __fdiv_rn(warp_sum_f32(sz), pi.nf);
            } else {  // double accumulation: independent of the order in which the list was filled
                double sx = 0.0, sy = 0.0, sz = 0.0;
                for (uint32_t j = lane; j < n_iter; j += 32) {
                    const float *q = point_at(j);
                    if (q) {
                        sx += static_cast<double>(__ldg(q));
                        sy += static_cast<double>(__ldg(q + 1));
                        sz += static_cast<double>(__ldg(q + 2));
                    }
                }
                mx = __fdiv_rn(static_cast<float>(warp_sum_f64(sx)), pi.nf);
                my = __fdiv_rn(static_cast<float>(warp_sum_f64(sy)), pi.nf);
                mz = __fdiv_rn(static_cast<float>(warp_sum_f64(sz)), pi.nf);
            }
        }
        // pillar centre: coord * voxel + offset, two roundings (pillar_vfe.py:100-103; dynamic_pillar_vfe.py:109-111)
        c.cx = __fadd_rn(__fmul_rn(static_cast<float>(pi.x), p.vsz[0]), p.off[0]);
        c.cy = __fadd_rn(__fmul_rn(static_cast<float>(pi.y), p.vsz[1]), p.off[1]);
        c.cz = p.dynamic ? p.off[2] : __fadd_rn(__fmul_rn(static_cast<float>(pi.z), p.vsz[2]), p.off[2]);

    }
    return true;
}

__global__ void __launch_bounds__(kThreads) k_pfn_multi(const __grid_constant__ MultiParams p)
{
    __shared__ float s_w0[kMaxIn0][kMaxOut];
    __shared__ float s_w1[kMaxIn1][kMaxOut];
    __shared__ float s_sc[2][kMaxOut], s_sh[2][kMaxOut];
    __shared__ float s_f[kWarps][kMaxOut];          // feature / activation exchange of a warp
    __shared__ uint32_t s_keep[kWarps][kKeepMax];   // kept point indices of a long capped pillar

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int in1 = 2 * p.out0;
    for (int i = tid; i < kMaxIn0 * kMaxOut; i += kThreads) {
        const int k = i / kMaxOut, o = i % kMaxOut;
        s_w0[k][o] = (k < p.c_in && o < p.out0) ? p.w0[o * p.c_in + k] : 0.f;
    }
    for (int i = tid; i < kMaxIn1 * kMaxOut; i += kThreads) {
        const int k = i / kMaxOut, o = i % kMaxOut;
        s_w1[k][o] = (p.n_layers > 1 && k < in1 && o < p.out1) ? p.w1[o * in1 + k] : 0.f;
    }
    for (int o = tid; o < kMaxOut; o += kThreads) {
        s_sc[0][o] = o < p.out0 ? p.s0[o] : 0.f;
        s_sh[0][o] = o < p.out0 ? p.h0[o] : 0.f;
        s_sc[1][o] = (p.n_layers > 1 && o < p.out1) ? p.s1[o] : 0.f;
        s_sh[1][o] = (p.n_layers > 1 && o < p.out1) ? p.h1[o] : 0.f;
    }
    __syncthreads();

    const int f_last = p.n_layers > 1 ? p.out1 : p.out0;
    const int my_kind = lane < p.c_in ? p.kind[lane < kMaxIn0 ? lane : 0] : -1;
    const int my_arg = lane < p.c_in ? p.arg[lane < kMaxIn0 ? lane : 0] : 0;
    float *const fbuf = s_f[warp];
    uint32_t *const keep = s_keep[warp];
    const int64_t total = p.dense ? p.m : static_cast<int64_t>(p.hdr->total_pillars);
    const int64_t warp_stride = static_cast<int64_t>(gridDim.x) * kWarps;
    const uint32_t P = static_cast<uint32_t>(p.max_points);

    for (int64_t g = static_cast<int64_t>(blockIdx.x) * kWarps + warp; g < total; g += warp_stride) {
        PillarCtx ctx;
        if (!prepare_pillar(p, g, lane, keep, ctx)) continue;
        const Pillar &pi = ctx.pi;
        const uint32_t n_iter = ctx.n_iter;
        const float mx = ctx.mx, my = ctx.my, mz = ctx.mz, cx = ctx.cx, cy = ctx.cy, cz = ctx.cz;
        auto point_at = [&](uint32_t t) -> const float * { return pillar_point(p, ctx, keep, t); };

        // the first C_in lanes build one augmented feature each; every lane then reads all of them
        auto features_to_buf = [&](const float *q) {
            if (my_kind >= 0) {
                float v;
                if (my_kind == kPoint) v = __ldg(q + my_arg);
                else if (my_kind == kCluster) v = __fsub_rn(__ldg(q + my_arg), my_arg == 0 ? mx : (my_arg == 1 ? my : mz));
                else if (my_kind == kCentre) v = __fsub_rn(__ldg(q + my_arg), my_arg == 0 ? cx : (my_arg == 1 ? cy : cz));
                else {
                    const float a = __ldg(q), b2 = __ldg(q + 1), c2 = __ldg(q + 2);
                    v = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b2, b2)), __fmul_rn(c2, c2)));
                }
                fbuf[lane] = v;
            }
            __syncwarp();
        };
        // layer 0 for channels lane and lane + 32 (the buffer holds the features, or zeros for the padded row)
        auto layer0 = [&](bool zero_row, float &ya, float &yb) {
            float a = 0.f, b2 = 0.f;
            if (!zero_row) {
                for (int k = 0; k < p.c_in; ++k) {
                    const float f = fbuf[k];
                    a = fmaf(f, s_w0[k][lane], a);
                    b2 = fmaf(f, s_w0[k][lane + 32], b2);
                }
            }
            ya = fmaxf(fmaf(a, s_sc[0][lane], s_sh[0][lane]), 0.f);
            yb = fmaxf(fmaf(b2, s_sc[0][lane + 32], s_sh[0][lane + 32]), 0.f);
            __syncwarp();  // everyone has read the buffer
        };
        const bool pad_row = !p.dynamic && pi.n_keep < P;  // one all-zero row stands for every padded slot

        float out_a, out_b;
        if (p.n_layers == 1) {
            float best_a = -INFINITY, best_b = -INFINITY;
            for (uint32_t t = 0; t < n_iter; ++t) {
                const float *q = point_at(t);
                if (!q) continue;
                features_to_buf(q);
                float ya, yb;
                layer0(false, ya, yb);
                best_a = fmaxf(best_a, ya);
                best_b = fmaxf(best_b, yb);
            }
            if (pad_row) {
                float ya, yb;
                layer0(true, ya, yb);
                best_a = fmaxf(best_a, ya);
                best_b = fmaxf(best_b, yb);
            }
            out_a = best_a;
            out_b = best_b;
        } else {
            // pass A: pillar-wise max of layer 0 (out0 <= 32: channel `lane`)
            float xmax = -INFINITY;
            for (uint32_t t = 0; t < n_iter; ++t) {
                const float *q = point_at(t);
                if (!q) continue;
                features_to_buf(q);
                float ya, yb;
                layer0(false, ya, yb);
                xmax = fmaxf(xmax, ya);
            }
            float xpad = 0.f, dummy;
            if (pad_row) {
                layer0(true, xpad, dummy);
                xmax = fmaxf(xmax, xpad);
            }
            // constant half of layer 1's input: W1[:, out0:] . xmax
            if (lane < p.out0) fbuf[lane] = xmax;
            __syncwarp();
            float ka = 0.f, kb = 0.f;
            for (int k = 0; k < p.out0; ++k) {
                const float f = fbuf[k];
                ka = fmaf(f, s_w1[p.out0 + k][lane], ka);
                kb = fmaf(f, s_w1[p.out0 + k][lane + 32], kb);
            }
            __syncwarp();
            auto layer1 = [&](float x, float &ya, float &yb) {
                if (lane < p.out0) fbuf[lane] = x;
                __syncwarp();
                float a = ka, b2 = kb;
                for (int k = 0; k < p.out0; ++k) {
                    const float f = fbuf[k];
                    a = fmaf(f, s_w1[k][lane], a);
                    b2 = fmaf(f, s_w1[k][lane + 32], b2);
                }
                ya = fmaxf(fmaf(a, s_sc[1][lane], s_sh[1][lane]), 0.f);
                yb = fmaxf(fmaf(b2, s_sc[1][lane + 32], s_sh[1][lane + 32]), 0.f);
                __syncwarp();
            };
            // pass B: layer 0 again, then layer 1 on [x, xmax]
            float best_a = -INFINITY, best_b = -INFINITY;
            for (uint32_t t = 0; t < n_iter; ++t) {
                const float *q = point_at(t);
                if (!q) continue;
                features_to_buf(q);
                float xa, xb, ya, yb;
                layer0(false, xa, xb);
                layer1(xa, ya, yb);
                best_a = fmaxf(best_a, ya);
                best_b = fmaxf(best_b, yb);
            }
            if (pad_row) {
                float ya, yb;
                layer1(xpad, ya, yb);
                best_a = fmaxf(best_a, ya);
                best_b = fmaxf(best_b, yb);
            }
            out_a = best_a;
            out_b = best_b;
        }

        float *dst = p.pillar_features + pi.row * f_last;
        if (lane < f_last) dst[lane] = out_a;
        if (lane + 32 < f_last) dst[lane + 32] = out_b;
        if (lane == 0 && !p.dense) {
            if (p.voxel_coords) {
                if (p.coords_cols == 3) {
                    int32_t *c = p.voxel_coords + pi.row * 3;
                    c[0] = pi.b; c[1] = pi.y; c[2] = pi.x;
                } else {
                    *reinterpret_cast<int4 *>(p.voxel_coords + pi.row * 4) = make_int4(pi.b, p.dynamic ? 0 : pi.z, pi.y, pi.x);
                }
            }
            if (p.voxel_num_points) p.voxel_num_points[pi.row] = static_cast<int32_t>(pi.n_keep);
            if (p.cell_row)
                p.cell_row[static_cast<int64_t>(pi.b) * p.gd.cells_xy + static_cast<int64_t>(pi.y) * p.gd.g[0] + pi.x] =
                    static_cast<int32_t>(pi.row);
        }
    }
}

// ---- the common shapes, register resident -------------------------------------------------------------------------------
// USE_ABSLOTE_XYZ, no WITH_DISTANCE, C point channels known at compile time: every lane builds the whole augmented feature
// vector itself from one broadcast load of the point (no exchange), layer 0's weights for the lane's channels sit in
// registers, and so do layer 1's (32 inputs x the channel pair {lane, lane + 32} = 64 registers, consumed by packed
// FFMA2).  Layer 0's outputs travel to layer 1 through a 128-byte per-warp buffer read back as eight 16-byte broadcasts.
//   LAYOUT 0: [point, point_xyz - mean, point_xyz - centre]     LAYOUT 1 (Simple2D): [point_xyz - centre, point]
__device__ __forceinline__ unsigned long long pk2(float a, float b)
{
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void ffma2_bcast(unsigned long long &acc, unsigned long long w, float x)
{
    unsigned long long rx;
    asm("mov.b64 %0, {%1, %1};" : "=l"(rx) : "f"(x));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(w), "l"(rx));
}

template <int C, int LAYOUT, bool TWO>
__global__ void __launch_bounds__(kThreads, 2) k_pfn_multi_reg(const __grid_constant__ MultiParams p)
{
    constexpr int kCin = LAYOUT == 1 ? C + 3 : C + 6;
    __shared__ float s_w1k[32][kMaxOut];             // layer 1, inputs out0..2*out0-1 (the pillar-max half), [k][channel]
    __shared__ __align__(16) float s_x[kWarps][32];  // layer 0 outputs of the current point
    __shared__ uint32_t s_keep[kWarps][kKeepMax];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int out0 = p.out0, out1 = p.out1;
    if (TWO) {
        for (int i = tid; i < 32 * kMaxOut; i += kThreads) {
            const int k = i / kMaxOut, o = i % kMaxOut;
            s_w1k[k][o] = (k < out0 && o < out1) ? p.w1[o * (2 * out0) + out0 + k] : 0.f;
        }
    }
    // layer 0: channels lane (a) and lane + 32 (b; only single-layer stacks are wider than 32)
    float w0a[kCin], w0b[kCin];
#pragma unroll
    for (int k = 0; k < kCin; ++k) {
        w0a[k] = lane < out0 ? __ldg(p.w0 + lane * kCin + k) : 0.f;
        w0b[k] = (!TWO && lane + 32 < out0) ? __ldg(p.w0 + (lane + 32) * kCin + k) : 0.f;
    }
    const float s0a = lane < out0 ? __ldg(p.s0 + lane) : 0.f, h0a = lane < out0 ? __ldg(p.h0 + lane) : 0.f;
    const float s0b = (!TWO && lane + 32 < out0) ? __ldg(p.s0 + lane + 32) : 0.f;
    const float h0b = (!TWO && lane + 32 < out0) ? __ldg(p.h0 + lane + 32) : 0.f;
    // layer 1: inputs 0..out0-1 (the per-point half) for the channel pair {lane, lane + 32}
    unsigned long long w1[TWO ? 32 : 1];
    float s1a = 0.f, h1a = 0.f, s1b = 0.f, h1b = 0.f;
    if (TWO) {
#pragma unroll
        for (int k = 0; k < 32; ++k) {
            const float a = (k < out0 && lane < out1) ? __ldg(p.w1 + lane * (2 * out0) + k) : 0.f;
            const float b = (k < out0 && lane + 32 < out1) ? __ldg(p.w1 + (lane + 32) * (2 * out0) + k) : 0.f;
            w1[k] = pk2(a, b);
        }
        if (lane < out1) { s1a = __ldg(p.s1 + lane); h1a = __ldg(p.h1 + lane); }
        if (lane + 32 < out1) { s1b = __ldg(p.s1 + lane + 32); h1b = __ldg(p.h1 + lane + 32); }
    }
    __syncthreads();

    const int f_last = TWO ? out1 : out0;
    float *const xbuf = s_x[warp];
    uint32_t *const keep = s_keep[warp];
    const int64_t total = p.dense ? p.m : static_cast<int64_t>(p.hdr->total_pillars);
    const int64_t warp_stride = static_cast<int64_t>(gridDim.x) * kWarps;
    const uint32_t P = static_cast<uint32_t>(p.max_points);

    for (int64_t g = static_cast<int64_t>(blockIdx.x) * kWarps + warp; g < total; g += warp_stride) {
        PillarCtx ctx;
        if (!prepare_pillar(p, g, lane, keep, ctx)) continue;
        const Pillar &pi = ctx.pi;
        const uint32_t n_iter = ctx.n_iter;
        const bool pad_row = !p.dynamic && pi.n_keep < P;  // one all-zero row stands for every padded slot

        // layer 0 of one point for the lane's channels (pre-activation sums)
        auto layer0 = [&](const float *q, float &ya, float &yb) {
            float pt[C];
#pragma unroll
            for (int c = 0; c < C; ++c) pt[c] = __ldg(q + c);
            float f[kCin];
            if (LAYOUT == 1) {
                f[0] = __fsub_rn(pt[0], ctx.cx); f[1] = __fsub_rn(pt[1], ctx.cy); f[2] = __fsub_rn(pt[2], ctx.cz);
#pragma unroll
                for (int c = 0; c < C; ++c) f[3 + c] = pt[c];
            } else {
#pragma unroll
                for (int c = 0; c < C; ++c) f[c] = pt[c];
                f[C + 0] = __fsub_rn(pt[0], ctx.mx); f[C + 1] = __fsub_rn(pt[1], ctx.my); f[C + 2] = __fsub_rn(pt[2], ctx.mz);
                f[C + 3] = __fsub_rn(pt[0], ctx.cx); f[C + 4] = __fsub_rn(pt[1], ctx.cy); f[C + 5] = __fsub_rn(pt[2], ctx.cz);
            }
            float a = 0.f, b = 0.f;
#pragma unroll
            for (int k = 0; k < kCin; ++k) {
                a = fmaf(f[k], w0a[k], a);
                if (!TWO) b = fmaf(f[k], w0b[k], b);
            }
            ya = fmaxf(fmaf(a, s0a, h0a), 0.f);
            yb = fmaxf(fmaf(b, s0b, h0b), 0.f);
        };

        float out_a, out_b;
        if (!TWO) {
            float best_a = -INFINITY, best_b = -INFINITY;
            for (uint32_t t = 0; t < n_iter; ++t) {
                const float *q = pillar_point(p, ctx, keep, t);
                if (!q) continue;
                float ya, yb;
                layer0(q, ya, yb);
                best_a = fmaxf(best_a, ya);
                best_b = fmaxf(best_b, yb);
            }
            if (pad_row) {
                best_a = fmaxf(best_a, fmaxf(h0a, 0.f));
                best_b = fmaxf(best_b, fmaxf(h0b, 0.f));
            }
            out_a = best_a;
            out_b = best_b;
        } else {
            // pass A: pillar-wise max of layer 0
            float xmax = -INFINITY;
            for (uint32_t t = 0; t < n_iter; ++t) {
                const float *q = pillar_point(p, ctx, keep, t);
                if (!q) continue;
                float ya, yb;
                layer0(q, ya, yb);
                xmax = fmaxf(xmax, ya);
            }
            const float xpad = fmaxf(h0a, 0.f);
            if (pad_row) xmax = fmaxf(xmax, xpad);
            // constant half of layer 1's input: W1[:, out0:] . xmax
            xbuf[lane] = lane < out0 ? xmax : 0.f;
            __syncwarp();
            float ka = 0.f, kb = 0.f;
            for (int k = 0; k < out0; ++k) {
                const float f = xbuf[k];
                ka = fmaf(f, s_w1k[k][lane], ka);
                kb = fmaf(f, s_w1k[k][lane + 32], kb);
            }
            __syncwarp();
            const unsigned long long kacc = pk2(ka, kb);
            auto layer1 = [&](float x, float &ya, float &yb) {
                xbuf[lane] = x;  // lanes >= out0 carry 0 (zero weights, zero scale and shift)
                __syncwarp();
                unsigned long long acc = kacc;
#pragma unroll
                for (int k4 = 0; k4 < 8; ++k4) {
                    const float4 xv = *reinterpret_cast<const float4 *>(xbuf + 4 * k4);
                    ffma2_bcast(acc, w1[4 * k4 + 0], xv.x);
                    ffma2_bcast(acc, w1[4 * k4 + 1], xv.y);
                    ffma2_bcast(acc, w1[4 * k4 + 2], xv.z);
                    ffma2_bcast(acc, w1[4 * k4 + 3], xv.w);
                }
                float a, b;
                asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(acc));
                ya = fmaxf(fmaf(a, s1a, h1a), 0.f);
                yb = fmaxf(fmaf(b, s1b, h1b), 0.f);
                __syncwarp();
            };
            // pass B: layer 0 again, then layer 1 on [x, xmax]
            float best_a = -INFINITY, best_b = -INFINITY;
            for (uint32_t t = 0; t < n_iter; ++t) {
                const float *q = pillar_point(p, ctx, keep, t);
                if (!q) continue;
                float xa, xb, ya, yb;
                layer0(q, xa, xb);
                layer1(xa, ya, yb);
                best_a = fmaxf(best_a, ya);
                best_b = fmaxf(best_b, yb);
            }
            if (pad_row) {
                float ya, yb;
                layer1(xpad, ya, yb);
                best_a = fmaxf(best_a, ya);
                best_b = fmaxf(best_b, yb);
            }
            out_a = best_a;
            out_b = best_b;
        }

        float *dst = p.pillar_features + pi.row * f_last;
        if (lane < f_last) dst[lane] = out_a;
        if (lane + 32 < f_last) dst[lane + 32] = out_b;
        if (lane == 0 && !p.dense) {
            if (p.voxel_coords) {
                if (p.coords_cols == 3) {
                    int32_t *c = p.voxel_coords + pi.row * 3;
                    c[0] = pi.b; c[1] = pi.y; c[2] = pi.x;
                } else {
                    *reinterpret_cast<int4 *>(p.voxel_coords + pi.row * 4) = make_int4(pi.b, p.dynamic ? 0 : pi.z, pi.y, pi.x);
                }
            }
            if (p.voxel_num_points) p.voxel_num_points[pi.row] = static_cast<int32_t>(pi.n_keep);
            if (p.cell_row)
                p.cell_row[static_cast<int64_t>(pi.b) * p.gd.cells_xy + static_cast<int64_t>(pi.y) * p.gd.g[0] + pi.x] =
                    static_cast<int32_t>(pi.row);
        }
    }
}

// picks the register-resident kernel when the configuration is one of its instantiations, else the general one
bool launch_reg_variant(const MultiParams &p, const StackDev &sd, unsigned blocks, cudaStream_t st)
{
    if (!sd.use_abs || sd.with_dist) return false;
    if (reinterpret_cast<uintptr_t>(p.points) % 4 != 0) return false;
    const bool two = sd.n_layers == 2;
    if (two && (sd.out[0] > 32 || sd.out[1] > 64)) return false;
    if (!two && sd.out[0] > 64) return false;
#define PILLARS_REG_CASE(CC, LL)                                                              \
    if (p.c_point == CC && sd.layout == LL) {                                                 \
        if (two) k_pfn_multi_reg<CC, LL, true><<<blocks, kThreads, 0, st>>>(p);               \
        else k_pfn_multi_reg<CC, LL, false><<<blocks, kThreads, 0, st>>>(p);                  \
        return true;                                                                          \
    }
    PILLARS_REG_CASE(4, 0)
    PILLARS_REG_CASE(5, 0)
    PILLARS_REG_CASE(4, 1)
    PILLARS_REG_CASE(5, 1)
#undef PILLARS_REG_CASE
    return false;
}

// ---- rows of the dynamic variant: rank of every occupied cell in (b, ix, iy) order -----------------------------------------
constexpr int kScanBlock = 2048;  // cells per CTA (256 threads x 8)

__global__ void k_mark_cells(const Header *__restrict__ hdr, const uint32_t *__restrict__ pillar_key, GridDev gd,
                             uint32_t *__restrict__ occ)
{
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= hdr->total_pillars) return;
    const uint32_t key = pillar_key[g];
    const uint32_t b = key / gd.cells, cell = key - b * gd.cells;  // nz == 1 in this mode
    const uint32_t y = cell / static_cast<uint32_t>(gd.g[0]), x = cell - y * static_cast<uint32_t>(gd.g[0]);
    occ[static_cast<size_t>(b) * gd.cells_xy + static_cast<size_t>(x) * gd.g[1] + y] = 1u;
}

__global__ void __launch_bounds__(256) k_block_counts(const uint32_t *__restrict__ occ, int64_t n, uint32_t *__restrict__ block_sum)
{
    __shared__ uint32_t s_w[8];
    const int64_t i0 = static_cast<int64_t>(blockIdx.x) * kScanBlock + threadIdx.x * 8;
    uint32_t c = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) c += (i0 + k < n) ? (occ[i0 + k] & 1u) : 0u;
    c = warp_sum_u32(c);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < 8; ++w) t += s_w[w];
        block_sum[blockIdx.x] = t;
    }
}

// single CTA: exclusive scan of the block sums in place; block_sum[n_blocks] = total
__global__ void __launch_bounds__(1024) k_scan_block_sums(uint32_t *__restrict__ block_sum, int n_blocks)
{
    __shared__ uint32_t s_w[32];
    __shared__ uint32_t s_carry;
    pdl_wait();  // (a no-op in a plain launch)
    pdl_trigger();
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < n_blocks; base += 1024) {
        const int i = base + threadIdx.x;
        const uint32_t v = i < n_blocks ? block_sum[i] : 0u;
        uint32_t incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(kFull, incl, d);
            if ((threadIdx.x & 31) >= d) incl += o;
        }
        if ((threadIdx.x & 31) == 31) s_w[threadIdx.x >> 5] = incl;
        __syncthreads();
        uint32_t wex = 0;
        for (int w = 0; w < static_cast<int>(threadIdx.x >> 5); ++w) wex += s_w[w];
        const uint32_t carry = s_carry;
        if (i < n_blocks) block_sum[i] = carry + wex + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + wex + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) block_sum[n_blocks] = s_carry;
}

// occ[i] <- exclusive rank | occupied << 31
__global__ void __launch_bounds__(256) k_apply_ranks(uint32_t *__restrict__ occ, int64_t n, const uint32_t *__restrict__ block_sum)
{
    __shared__ uint32_t s_w[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i0 = static_cast<int64_t>(blockIdx.x) * kScanBlock + threadIdx.x * 8;
    uint32_t o[8], c = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        o[k] = (i0 + k < n) ? (occ[i0 + k] & 1u) : 0u;
        c += o[k];
    }
    uint32_t incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(kFull, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    uint32_t run = block_sum[blockIdx.x] + incl - c;
    for (int w = 0; w < warp; ++w) run += s_w[w];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if (i0 + k < n) occ[i0 + k] = run | (o[k] << 31);
        run += o[k];
    }
}

int num_sms() { return current_sm_count(); }  // per device (a process may drive more than one)

void fill_layout(MultiParams &p, const StackDev &sd, int c_point)
{
    int q = 0;
    auto push = [&](int kind, int arg) {
        if (q < kMaxIn0) {
            p.kind[q] = kind;
            p.arg[q] = arg;
        }
        ++q;
    };
    if (sd.layout == 1) {  // DynamicPillarVFESimple2D: [f_center, point channels, distance]  (dynamic_pillar_vfe.py:209-224)
        for (int a = 0; a < 3; ++a) push(kCentre, a);
        for (int c = sd.use_abs ? 0 : 3; c < c_point; ++c) push(kPoint, c);
    } else {  // PillarVFE / DynamicPillarVFE: [point channels, f_cluster, f_center, distance]  (pillar_vfe.py:105-113)
        for (int c = sd.use_abs ? 0 : 3; c < c_point; ++c) push(kPoint, c);
        for (int a = 0; a < 3; ++a) push(kCluster, a);
        for (int a = 0; a < 3; ++a) push(kCentre, a);
    }
    if (sd.with_dist) push(kDist, 0);
    p.c_in = q;
}

void fill_stack(MultiParams &p, const StackDev &sd)
{
    p.n_layers = sd.n_layers;
    p.out0 = sd.out[0];
    p.out1 = sd.n_layers > 1 ? sd.out[1] : 0;
    p.w0 = sd.weight[0]; p.s0 = sd.scale[0]; p.h0 = sd.shift[0];
    p.w1 = sd.weight[1]; p.s1 = sd.scale[1]; p.h1 = sd.shift[1];
    for (int i = 0; i < 3; ++i) {
        p.vsz[i] = sd.vsz[i];
        p.off[i] = sd.off[i];
    }
}

}  // namespace

int stack_c_in(const StackDev &sd, int c_point)
{
    MultiParams p{};
    fill_layout(p, sd, c_point);
    return p.c_in;
}

bool stack_supported(const StackDev &sd, int c_point)
{
    if (sd.n_layers < 1 || sd.n_layers > 2) return false;
    const int c_in = stack_c_in(sd, c_point);
    if (c_in > kMaxIn0) return false;
    if (sd.n_layers == 1) return sd.out[0] >= 1 && sd.out[0] <= kMaxOut;
    return sd.out[0] >= 1 && sd.out[0] <= 32 && sd.out[1] >= 1 && sd.out[1] <= kMaxOut;
}

cudaError_t launch_dynamic_ranks(const GridDev &gd, const Workspace &ws, int nb, int64_t n, cudaStream_t st)
{
    // the index-map region of the workspace holds the (b, ix, iy)-ordered occupancy, then the ranks
    uint32_t *occ = reinterpret_cast<uint32_t *>(ws.cell_row);
    const int64_t n_cells = static_cast<int64_t>(nb) * gd.cells_xy;
    const int n_blocks = static_cast<int>((n_cells + kScanBlock - 1) / kScanBlock);
    uint32_t *block_sum = ws.scan_scratch;
    cudaError_t e = cudaMemsetAsync(occ, 0, sizeof(uint32_t) * n_cells, st);
    if (e != cudaSuccess) return e;
    note_launch();
    const unsigned mb = static_cast<unsigned>((n + 255) / 256);
    k_mark_cells<<<mb, 256, 0, st>>>(ws.hdr, ws.pillar_key, gd, occ);
    k_block_counts<<<n_blocks, 256, 0, st>>>(occ, n_cells, block_sum);
    k_scan_block_sums<<<1, 1024, 0, st>>>(block_sum, n_blocks);
    k_apply_ranks<<<n_blocks, 256, 0, st>>>(occ, n_cells, block_sum);
    note_launch(4);
    return cudaGetLastError();
}

// ---- the same ranks for the streaming kernel, from a BITMAP of the occupied cells (1 bit per cell in (b, ix, iy) order: 0.5 MB
//      at cfg2 instead of the 16.7 MB word-per-cell array above): mark, prefix of the word popcounts, one thread per pillar
__device__ __forceinline__ uint32_t dyn_bit_index(const GridDev &gd, uint32_t key)
{
    const uint32_t b = key / gd.cells, cell = key - b * gd.cells;  // nz == 1 in this mode
    const uint32_t y = cell / static_cast<uint32_t>(gd.g[0]), x = cell - y * static_cast<uint32_t>(gd.g[0]);
    return b * static_cast<uint32_t>(gd.cells_xy) + x * static_cast<uint32_t>(gd.g[1]) + y;
}

__global__ void k_dyn_mark_bits(const Header *__restrict__ hdr, const uint32_t *__restrict__ pillar_key, GridDev gd,
                                uint32_t *__restrict__ bm)
{
    pdl_wait();
    pdl_trigger();
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= hdr->total_pillars) return;
    const uint32_t idx = dyn_bit_index(gd, pillar_key[g]);
    atomicOr(bm + (idx >> 5), 1u << (idx & 31u));
}

// pre[w] <- occupied cells before word w inside its 2048-word block; block_sum[blk] <- occupied cells of the block
__global__ void __launch_bounds__(256) k_dyn_word_prefix(const uint32_t *__restrict__ bm, int64_t n_words, uint32_t *__restrict__ pre,
                                                         uint32_t *__restrict__ block_sum)
{
    __shared__ uint32_t s_w[8];
    pdl_wait();
    pdl_trigger();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i0 = static_cast<int64_t>(blockIdx.x) * kScanBlock + threadIdx.x * 8;
    uint32_t o[8], c = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        o[k] = (i0 + k < n_words) ? __popc(bm[i0 + k]) : 0u;
        c += o[k];
    }
    uint32_t incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(kFull, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    uint32_t run = incl - c;
    for (int w = 0; w < warp; ++w) run += s_w[w];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if (i0 + k < n_words) pre[i0 + k] = run;
        run += o[k];
    }
    if (threadIdx.x == 255) block_sum[blockIdx.x] = run;
}

// one thread per pillar (grouping order): row = rank of its cell; patches the pillar entry the streaming kernel reads
__global__ void k_dynamic_rows(const Header *__restrict__ hdr, const uint32_t *__restrict__ pillar_key,
                               const uint32_t *__restrict__ pillar_list, const uint32_t *__restrict__ pillar_cnt, GridDev gd,
                               const uint32_t *__restrict__ bm, const uint32_t *__restrict__ pre,
                               const uint32_t *__restrict__ block_sum, int64_t capacity, uint4 *__restrict__ pillar_meta,
                               int32_t *__restrict__ voxel_coords, int32_t *__restrict__ voxel_num_points)
{
    pdl_wait();
    pdl_trigger();
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= hdr->total_pillars) return;
    const uint32_t key = pillar_key[g];
    const uint32_t b = key / gd.cells, cell = key - b * gd.cells;  // nz == 1 in this mode
    const uint32_t y = cell / static_cast<uint32_t>(gd.g[0]), x = cell - y * static_cast<uint32_t>(gd.g[0]);
    const uint32_t idx = b * static_cast<uint32_t>(gd.cells_xy) + x * static_cast<uint32_t>(gd.g[1]) + y, w = idx >> 5;
    const uint32_t row = block_sum[w / kScanBlock] + pre[w] + __popc(bm[w] & ((1u << (idx & 31u)) - 1u));
    const bool live = static_cast<int64_t>(row) < capacity;
    reinterpret_cast<uint32_t *>(pillar_meta + pillar_list[g])[1] = live ? row : 0xFFFFFFFFu;
    if (!live) return;
    if (voxel_coords)
        *reinterpret_cast<int4 *>(voxel_coords + static_cast<size_t>(row) * 4) =
            make_int4(static_cast<int>(b), 0, static_cast<int>(y), static_cast<int>(x));
    if (voxel_num_points) voxel_num_points[row] = static_cast<int32_t>(pillar_cnt[g]);
}

cudaError_t launch_dynamic_rows(const GridDev &gd, const Workspace &ws, int nb, int64_t n, int64_t capacity,
                                int32_t *voxel_coords, int32_t *voxel_num_points, cudaStream_t st)
{
    // scratch in the index-map region of the workspace (4 bytes per cell; the bitmap and its prefix need 1/4 of a byte)
    const int64_t n_cells = static_cast<int64_t>(nb) * gd.cells_xy;
    if (n_cells >= (int64_t(1) << 32)) return cudaErrorInvalidValue;
    const int64_t n_words = (n_cells + 31) / 32;
    uint32_t *bm = reinterpret_cast<uint32_t *>(ws.cell_row);
    uint32_t *pre = bm + ((n_words + 3) & ~int64_t(3));
    uint32_t *block_sum = ws.scan_scratch;
    const int n_blocks = static_cast<int>((n_words + kScanBlock - 1) / kScanBlock);
    cudaError_t e = cudaMemsetAsync(bm, 0, sizeof(uint32_t) * n_words, st);
    if (e != cudaSuccess) return e;
    note_launch();
    const unsigned mb = static_cast<unsigned>((n + 255) / 256);
    // chained by programmatic dependent launch: every kernel waits for its predecessor at its first instruction, so the
    // chain stays transitive, and its CTAs are resident before the predecessor has drained
    const uint32_t *c_bm = bm, *c_pre = pre, *c_bs = block_sum;
    const Header *c_hdr = ws.hdr;
    const uint32_t *c_key = ws.pillar_key, *c_list = ws.pillar_list, *c_cnt = ws.pillar_cnt;
    if ((e = launch_pdl(k_dyn_mark_bits, dim3(mb), dim3(256), 0, st, c_hdr, c_key, gd, bm)) != cudaSuccess) return e;
    if ((e = launch_pdl(k_dyn_word_prefix, dim3(n_blocks), dim3(256), 0, st, c_bm, n_words, pre, block_sum)) != cudaSuccess) return e;
    if ((e = launch_pdl(k_scan_block_sums, dim3(1), dim3(1024), 0, st, block_sum, n_blocks)) != cudaSuccess) return e;
    if ((e = launch_pdl(k_dynamic_rows, dim3(mb), dim3(256), 0, st, c_hdr, c_key, c_list, c_cnt, gd, c_bm, c_pre, c_bs, capacity,
                        ws.pillar_meta, voxel_coords, voxel_num_points)) != cudaSuccess)
        return e;
    note_launch(4);
    return cudaGetLastError();
}

cudaError_t launch_pfn_multi_lists(const MultiJob &job, const StackDev &sd, const GridDev &gd, const Workspace &ws,
                                   cudaStream_t st)
{
    if (job.n == 0) return cudaSuccess;
    MultiParams p{};
    p.points = job.points;
    p.stride = job.stride;
    p.col0 = job.col0;
    p.c_point = job.c_point;
    p.idx_bits = job.idx_bits;
    p.gd = gd;
    p.hdr = ws.hdr;
    p.pillar_key = ws.pillar_key;
    p.pillar_list = ws.pillar_list;
    p.pillar_cnt = ws.pillar_cnt;
    p.sorted_idx = ws.sorted_idx;
    p.frame_gstart = ws.frame_gstart;
    p.frame_rowbase = ws.frame_rowbase;
    p.dynamic = job.dynamic ? 1 : 0;
    p.max_points = gd.max_points;
    fill_layout(p, sd, job.c_point);
    fill_stack(p, sd);
    p.pillar_features = job.pillar_features;
    p.voxel_coords = job.voxel_coords;
    p.voxel_num_points = job.voxel_num_points;
    p.coords_cols = job.coords_cols;
    p.capacity = job.capacity;
    p.cell_row = (!job.dynamic && job.write_cell_row) ? ws.cell_row : nullptr;

    if (job.dynamic) {
        cudaError_t e = launch_dynamic_ranks(gd, ws, job.nb, job.n, st);
        if (e != cudaSuccess) return e;
        p.rank_xmajor = reinterpret_cast<uint32_t *>(ws.cell_row);
    }
    int64_t blocks = (job.n + kWarps - 1) / kWarps;
    const int64_t cap = static_cast<int64_t>(num_sms()) * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    if (!launch_reg_variant(p, sd, static_cast<unsigned>(blocks), st))
        k_pfn_multi<<<static_cast<unsigned>(blocks), kThreads, 0, st>>>(p);
    note_launch();
    return cudaGetLastError();
}

cudaError_t launch_pfn_multi_dense(const float *voxels, const void *num_points, bool np_float, const void *coords,
                                   bool coords_float, int64_t m, int max_points, int c_point, const StackDev &sd,
                                   float *out, cudaStream_t st)
{
    if (m == 0) return cudaSuccess;
    MultiParams p{};
    p.voxels = voxels;
    p.num_points = num_points;
    p.coords = coords;
    p.np_float = np_float ? 1 : 0;
    p.coords_float = coords_float ? 1 : 0;
    p.m = m;
    p.dense = 1;
    p.c_point = c_point;
    p.max_points = max_points;
    fill_layout(p, sd, c_point);
    fill_stack(p, sd);
    p.pillar_features = out;
    p.capacity = m;
    int64_t blocks = (m + kWarps - 1) / kWarps;
    const int64_t cap = static_cast<int64_t>(num_sms()) * 8;
    if (blocks > cap) blocks = cap;
    if (!launch_reg_variant(p, sd, static_cast<unsigned>(blocks), st))
        k_pfn_multi<<<static_cast<unsigned>(blocks), kThreads, 0, st>>>(p);
    note_launch();
    return cudaGetLastError();
}

}  // namespace pillars
