// Per-pillar feature stage for the mainstream configuration (USE_ABSLOTE_XYZ, no WITH_DISTANCE, C <= 5 point channels,
// one PFN layer, F = 64): pillar_vfe.py:94-123 (augment) + :29-49 (Linear + BatchNorm(eval) + ReLU + max over the pillar).
//
// Shape of the work.  The points arrive as 32-byte records grouped by pillar (place kernel), ~2 points per pillar, and one
// 16-byte {cell key, row, n} record per pillar at the pillar's list start position (scan / place kernel).  The layer is
// regrouped around the pillar centre c (x' = x - c, m' = mean - c):
//       W.[p, p_xyz - mean, p_xyz - c] = (W_p + W_cl + W_ce).x' + W_it.(i,t)  +  [ W_p.c - W_cl.m' ]
// i.e. 5 FMAs per (point, channel) plus one 6-FMA constant per (pillar, channel); every per-point term is a small number, so
// nothing cancels.  BatchNorm's scale is folded into W, and since "+ constant" and ReLU are monotone the max over the
// pillar's points is taken before them.
//
// Mapping.  The kernel is bound by instruction issue, not by HBM, so everything is arranged to issue few instructions and
// to never wait for memory:
//   * persistent warps: a warp owns a contiguous range of 32-position chunks of the record list.  A chunk's window is 64
//     positions (32 own + 32 look-ahead); records and pillar entries are brought in by cp.async (LDGSTS, no registers)
//     into the warp's second buffer while the current chunk is processed;
//   * phase 1, one lane per list position, no loops: the per-pillar sums for the mean are accumulated with shared-memory
//     integer atomics on fixed-point coordinates relative to the pillar centre (order independent => bit-reproducible,
//     resolution 2^-29 of a metre at 0.2 m pillars, far below the fp32 rounding of the reference's own absolute-coordinate
//     sum); points beyond the first-P cap are found by rank counting inside the window and become NaN (fmaxf ignores
//     NaN, so the walk needs no branch); the lane on a list start turns the sums into the pillar's constants and flags
//     the pillar's final point;
//   * phase 2, ONE LANE PER CHANNEL PAIR: the warp walks its points in list order, each point is two broadcast
//     shared-memory loads + 5 packed FFMA2 (fma.rn.f32x2: two channels per instruction) + 2 FMNMX with the running max in
//     registers; at a pillar end the lanes add the per-pillar constant (6 FFMA2), apply ReLU / the padded-slot term and
//     store the 256-byte output row with one coalesced 8-byte store per lane.
// A chunk owns the pillars whose list STARTS inside it.  A pillar of more than 32 points cannot fit the window: the grouping
// stage lists those, and every warp that runs out of chunks takes entries from that list (warp-cooperative path reading the
// records from global memory; 8-bit radix select of the P-th smallest point index when n > P).
#include <cmath>

#include "group_common.cuh"

namespace pillars {

namespace {

constexpr unsigned kFull = 0xffffffffu;

// per-warp shared memory (bytes): two chunk buffers (the chunk being processed, the chunk in flight), each holding the 64
// records of the window (32 own positions + 32 look-ahead) and the 32 pillar entries of the own positions
constexpr uint32_t kRecBytes = 64 * 32;
constexpr uint32_t kMetaBytes = 32 * 16;
constexpr uint32_t kBufBytes = kRecBytes + kMetaBytes;  // 2560
constexpr uint32_t kPlBytes = 32 * 32;                  // pillar constants of the chunk being walked
constexpr uint32_t kSumBytes = 3 * 32 * 4;
constexpr uint32_t kOffPl = 2 * kBufBytes;
constexpr uint32_t kOffSum = kOffPl + kPlBytes;
constexpr uint32_t kWarpSmem = kOffSum + kSumBytes;     // 6528
// two-layer stacks: layer 0's outputs of two points (or of the pillar-wise max), double buffered: 4 x [64] floats
constexpr uint32_t kOffX = kWarpSmem;
constexpr uint32_t kXBytes = 256;
constexpr uint32_t kWarpSmemTwo = kOffX + 4 * kXBytes;  // 7552

struct WalkParams {
    const PointRecord *records;   // grouped by pillar, x,y,z relative to the pillar centre (place kernel)
    const Header *hdr;
    const uint4 *pillar_meta;     // by list start position: {x | y << 16, row, n, z}
    const uint4 *long_list;       // pillars of more than 32 points: {list start, n, row, x | y << 16} {z, -, -, -}
    const uint32_t *long_count;   // entries - 1
    uint32_t *long_cursor;        // next entry to process - 1 (shared by all warps of the grid)
    uint32_t *chunk_cursor;       // two-layer stacks: next chunk - 1 (chunks are handed out one at a time)
    int idx_bits;                 // bits of a point index; in the pad before `folded`, so that the fields below keep the
                                  // 16-byte alignment that lets ptxas fetch them with 128-bit constant loads
    const float *folded;          // [PILLARS_FOLDED_FLOATS], see launch_fold_pfn
    float *pillar_features;
    const float *folded2;         // two-layer stacks: [32][64] per-point half of layer 1 | [32][64] pillar-max half | [64] shift
    GridDev gd;
    int sh_cells, sh_cells_xy, sh_nx;
    float vsz[3], off[3];
    float fx_scale[3], fx_inv[3];  // fixed-point scale of the mean sums per axis (a power of two) and its inverse
    unsigned long long *dbg;
};

// ---- packed fp32 pairs (Blackwell FFMA2 / FMUL2 / FADD2) ------------------------------------------------------------
__device__ __forceinline__ unsigned long long pack2(float2 v)
{
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(v.x), "f"(v.y));
    return r;
}
__device__ __forceinline__ float2 unpack2(unsigned long long r)
{
    float2 v;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(v.x), "=f"(v.y) : "l"(r));
    return v;
}
// w * (x, x) + c : ptxas turns the duplicated half into FFMA2's scalar-broadcast operand
__device__ __forceinline__ float2 fma2s(float2 w, float x, float2 c)
{
    unsigned long long rx, rd;
    asm("mov.b64 %0, {%1, %1};" : "=l"(rx) : "f"(x));
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(pack2(w)), "l"(rx), "l"(pack2(c)));
    return unpack2(rd);
}
__device__ __forceinline__ float2 mul2s(float2 w, float x)
{
    unsigned long long rx, rd;
    asm("mov.b64 %0, {%1, %1};" : "=l"(rx) : "f"(x));
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(pack2(w)), "l"(rx));
    return unpack2(rd);
}
__device__ __forceinline__ float2 add2(float2 a, float2 b)
{
    unsigned long long rd;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(pack2(a)), "l"(pack2(b)));
    return unpack2(rd);
}

// shared-memory accesses by 32-bit address: the walk carries one address register and no generic-pointer arithmetic
__device__ __forceinline__ float4 lds4(uint32_t addr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint4 lds4u(uint32_t addr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds1u(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts4(uint32_t addr, float4 v)
{
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts1(uint32_t addr, uint32_t v)
{
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void atoms_add(uint32_t addr, int v)
{
    asm volatile("red.shared.add.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
// 16 bytes global -> shared without registers; src_bytes = 0 writes zeros
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, int src_bytes)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// 1 / n for the window sizes (n <= 32); index 0 unused
__constant__ float kRcp[33] = {0.f, 1.f / 1, 1.f / 2, 1.f / 3, 1.f / 4, 1.f / 5, 1.f / 6, 1.f / 7, 1.f / 8, 1.f / 9, 1.f / 10,
                               1.f / 11, 1.f / 12, 1.f / 13, 1.f / 14, 1.f / 15, 1.f / 16, 1.f / 17, 1.f / 18, 1.f / 19,
                               1.f / 20, 1.f / 21, 1.f / 22, 1.f / 23, 1.f / 24, 1.f / 25, 1.f / 26, 1.f / 27, 1.f / 28,
                               1.f / 29, 1.f / 30, 1.f / 31, 1.f / 32};

struct LaneWeights {
    float2 w0, w1, w2, w3, w4;        // per point: x', y', z', intensity, time
    float2 k0, k1, k2, k3, k4, k5;    // per pillar: centre xyz, -(cluster weights) on (mean - centre)
    float2 sh, rsh;                   // BatchNorm shift, relu(shift)
};

// the lane's two channels of one staged point (before the per-pillar constant); NaN for a point beyond the first-P cap
__device__ __forceinline__ float2 point_eval(const LaneWeights &w, uint32_t addr)
{
    const float4 a = lds4(addr);
    const float t = __uint_as_float(lds1u(addr + 16));
    float2 y = mul2s(w.w0, a.x);
    y = fma2s(w.w1, a.y, y);
    y = fma2s(w.w2, a.z, y);
    y = fma2s(w.w3, a.w, y);
    return fma2s(w.w4, t, y);
}
// fmaxf ignores NaN operands, so dropped points vanish
__device__ __forceinline__ float2 max2(float2 a, float2 b) { return make_float2(fmaxf(a.x, b.x), fmaxf(a.y, b.y)); }
__device__ __forceinline__ float2 max3(float2 a, float2 b, float2 c)
{
    return make_float2(fmaxf(a.x, fmaxf(b.x, c.x)), fmaxf(a.y, fmaxf(b.y, c.y)));
}

// points 1..n-1 of a pillar: two at a time (independent chains), the running max combined with a 3-input max
__device__ __forceinline__ float2 more_points(const LaneWeights &w, uint32_t pa, uint32_t n, float2 acc)
{
    uint32_t k = 1;
    for (; k + 1 < n; k += 2) {
        const float2 ya = point_eval(w, pa + k * 32u), yb = point_eval(w, pa + k * 32u + 32u);
        acc = max3(acc, ya, yb);
    }
    if (k < n) acc = max2(acc, point_eval(w, pa + k * 32u));
    return acc;
}

// the per-pillar constant  W_p.c - W_cl.(mean - c) + shift  for the lane's two channels
__device__ __forceinline__ float2 pillar_const(const LaneWeights &w, const float4 c4, const float4 m4)
{
    float2 kc = fma2s(w.k0, c4.x, w.sh);
    kc = fma2s(w.k1, c4.y, kc);
    kc = fma2s(w.k2, c4.z, kc);
    kc = fma2s(w.k3, m4.x, kc);
    kc = fma2s(w.k4, m4.y, kc);
    return fma2s(w.k5, m4.z, kc);
}
// + constant, ReLU / padded-slot term, one coalesced 256-byte row (row < 0: pillar not emitted)
__device__ __forceinline__ void pillar_store(const LaneWeights &w, const float2 kc, const int row, const bool padded,
                                             const float2 acc, unsigned long long out_lane)
{
    const float2 v = add2(acc, kc);
    const float2 fl2 = mul2s(w.rsh, padded ? 1.f : 0.f);  // relu(shift) when the pillar has padded slots, else 0
    if (row >= 0)
        asm volatile("st.global.v2.f32 [%0], {%1, %2};" ::"l"(out_lane + static_cast<unsigned long long>(static_cast<uint32_t>(row)) * 256ull),
                     "f"(fmaxf(v.x, fl2.x)), "f"(fmaxf(v.y, fl2.y))
                     : "memory");
}

// per-pillar constant, ReLU, padded-slot term, one 256-byte row.  c4 = centre xyz + (1.0 when the pillar has empty slots),
// m4 = mean - centre xyz + row as int bits (-1: pillar not emitted)
__device__ __forceinline__ void pillar_finish(const LaneWeights &w, const float4 c4, const float4 m4, const bool padded,
                                              const float2 acc, unsigned long long out_lane)
{
    float2 kc = fma2s(w.k0, c4.x, w.sh);
    kc = fma2s(w.k1, c4.y, kc);
    kc = fma2s(w.k2, c4.z, kc);
    kc = fma2s(w.k3, m4.x, kc);
    kc = fma2s(w.k4, m4.y, kc);
    kc = fma2s(w.k5, m4.z, kc);
    const float2 v = add2(acc, kc);
    const float2 fl2 = mul2s(w.rsh, padded ? 1.f : 0.f);  // relu(shift) when the pillar has padded slots, else 0
    const int row = __float_as_int(m4.w);
    if (row >= 0)
        asm volatile("st.global.v2.f32 [%0], {%1, %2};" ::"l"(out_lane + static_cast<unsigned long long>(static_cast<uint32_t>(row)) * 256ull),
                     "f"(fmaxf(v.x, fl2.x)), "f"(fmaxf(v.y, fl2.y))
                     : "memory");
}

// mean - centre with the reference's rounding of the ABSOLUTE mean to fp32 (pillar_vfe.py:97-98)
__device__ __forceinline__ float rel_mean(float c, float s_rel_mean) { return __fsub_rn(__fadd_rn(c, s_rel_mean), c); }

__device__ __forceinline__ LaneWeights load_lane_weights(const float *folded, int lane)
{
    LaneWeights w;
    const float2 *fw = reinterpret_cast<const float2 *>(folded) + lane;
    w.w0 = __ldg(fw + 0 * 32); w.w1 = __ldg(fw + 1 * 32); w.w2 = __ldg(fw + 2 * 32); w.w3 = __ldg(fw + 3 * 32);
    w.w4 = __ldg(fw + 4 * 32);
    w.k0 = __ldg(fw + 5 * 32); w.k1 = __ldg(fw + 6 * 32); w.k2 = __ldg(fw + 7 * 32); w.k3 = __ldg(fw + 8 * 32);
    w.k4 = __ldg(fw + 9 * 32); w.k5 = __ldg(fw + 10 * 32);
    w.sh = __ldg(fw + 11 * 32); w.rsh = __ldg(fw + 12 * 32);
    return w;
}

// ---- second layer of a [64, 64] stack (pillar_vfe.py:18-19,44-49: layer 1 sees [x_p, max over the pillar of x]) ------------
struct Layer1 {
    float2 wa[32];    // the lane's two output channels of scale1 * W1[:, k], per-point inputs k = 0..31
    float2 sh, upad;  // shift1;  W1a . relu(shift0): the per-point half of the row that stands for the padded slots
};
__device__ __forceinline__ Layer1 load_layer1(const float *folded, const float *folded2, int lane)
{
    Layer1 l;
    const float2 *f2 = reinterpret_cast<const float2 *>(folded2) + lane;
    l.sh = __ldg(reinterpret_cast<const float2 *>(folded2 + 4096) + lane);
    float2 u0 = make_float2(0.f, 0.f), u1 = u0;
#pragma unroll
    for (int k = 0; k < 32; k += 2) {
        l.wa[k] = __ldg(f2 + k * 32);
        l.wa[k + 1] = __ldg(f2 + (k + 1) * 32);
        u0 = fma2s(l.wa[k], __ldg(folded + 12 * 64 + k), u0);
        u1 = fma2s(l.wa[k + 1], __ldg(folded + 12 * 64 + k + 1), u1);
    }
    l.upad = add2(u0, u1);
    return l;
}
__device__ __forceinline__ void sts2(uint32_t addr, float2 v)
{
    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(v.x), "f"(v.y) : "memory");
}
// cst = shift1 + (scale1 W1[:, 32:]) . m  for the lane's two channels: m = 32 floats at shared address xs, weights [32][64]
// (shared memory in the walk, global memory on the long-pillar path); four independent chains
__device__ __forceinline__ float2 layer1_const(const float *w1b, uint32_t xs, float2 sh1, int lane)
{
    float2 y0 = sh1, y1 = make_float2(0.f, 0.f), y2 = y1, y3 = y1;
#pragma unroll
    for (int k4 = 0; k4 < 8; ++k4) {
        const float4 mv = lds4(xs + k4 * 16u);
        const float2 *wb = reinterpret_cast<const float2 *>(w1b + (4 * k4) * 64) + lane;
        y0 = fma2s(wb[0], mv.x, y0);
        y1 = fma2s(wb[32], mv.y, y1);
        y2 = fma2s(wb[64], mv.z, y2);
        y3 = fma2s(wb[96], mv.w, y3);
    }
    return add2(add2(y0, y1), add2(y2, y3));
}
// Layer 1 over the n staged points at shared address pa (32-byte records, NaN x = beyond the first-P cap), two points per
// trip: x = relu(layer 0) of both goes through the warp's x buffers (double buffered: one __syncwarp per trip), then four
// independent FFMA2 chains (two per point) of 16; an odd last point takes a trip of its own (the same two chains).  Returns the
// running max of  W1a . x + cst  over the kept points.  The caller guarantees a __syncwarp() between the last read of the x
// buffers and this call.
__device__ __forceinline__ float2 point_lin(const LaneWeights &w, const float4 a, const float t)
{
    float2 y = mul2s(w.w0, a.x);
    y = fma2s(w.w1, a.y, y);
    y = fma2s(w.w2, a.z, y);
    y = fma2s(w.w3, a.w, y);
    return fma2s(w.w4, t, y);
}
__device__ __forceinline__ float2 relu2(float2 v) { return make_float2(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f)); }
__device__ __forceinline__ float2 layer1_points(const LaneWeights &w, const float2 (&wa)[32], const float2 kc, const float2 cst,
                                                uint32_t pa, uint32_t n, uint32_t s_x, int lane, float2 best)
{
    const uint32_t qnan_bits = 0x7fc00000u;
    const float2 zero = make_float2(0.f, 0.f);
    uint32_t half = 0, j = 0;
    for (; j + 1u < n; j += 2) {
        const uint32_t qa = pa + j * 32u;
        const float4 a0 = lds4(qa), a1 = lds4(qa + 32u);
        const float t0 = __uint_as_float(lds1u(qa + 16u)), t1 = __uint_as_float(lds1u(qa + 48u));
        const bool ok0 = __float_as_uint(a0.x) != qnan_bits, ok1 = __float_as_uint(a1.x) != qnan_bits;
        const float2 x0 = relu2(add2(point_lin(w, a0, t0), kc)), x1 = relu2(add2(point_lin(w, a1, t1), kc));
        const uint32_t xs = s_x + half;
        half ^= 2u * kXBytes;
        sts2(xs + lane * 8u, x0);
        sts2(xs + kXBytes + lane * 8u, x1);
        __syncwarp();
        float2 ya = cst, yb = zero, yc = cst, yd = zero;
#pragma unroll
        for (int k4 = 0; k4 < 8; ++k4) {
            const float4 u = lds4(xs + k4 * 16u), v = lds4(xs + kXBytes + k4 * 16u);
            ya = fma2s(wa[4 * k4 + 0], u.x, ya);
            yc = fma2s(wa[4 * k4 + 0], v.x, yc);
            yb = fma2s(wa[4 * k4 + 1], u.y, yb);
            yd = fma2s(wa[4 * k4 + 1], v.y, yd);
            ya = fma2s(wa[4 * k4 + 2], u.z, ya);
            yc = fma2s(wa[4 * k4 + 2], v.z, yc);
            yb = fma2s(wa[4 * k4 + 3], u.w, yb);
            yd = fma2s(wa[4 * k4 + 3], v.w, yd);
        }
        if (ok0) best = max2(best, add2(ya, yb));
        if (ok1) best = max2(best, add2(yc, yd));
    }
    if (j < n) {
        const uint32_t qa = pa + j * 32u;
        const float4 a0 = lds4(qa);
        const float t0 = __uint_as_float(lds1u(qa + 16u));
        if (__float_as_uint(a0.x) != qnan_bits) {  // warp-uniform
            const uint32_t xs = s_x + half;
            sts2(xs + lane * 8u, relu2(add2(point_lin(w, a0, t0), kc)));
            __syncwarp();
            // the same two chains and summation order as in a pair: a point's value must not depend on where the
            // (unordered) list placed it, or the output would not be bit-reproducible from run to run
            float2 ya = cst, yb = zero;
#pragma unroll
            for (int k4 = 0; k4 < 8; ++k4) {
                const float4 u = lds4(xs + k4 * 16u);
                ya = fma2s(wa[4 * k4 + 0], u.x, ya);
                yb = fma2s(wa[4 * k4 + 1], u.y, yb);
                ya = fma2s(wa[4 * k4 + 2], u.z, ya);
                yb = fma2s(wa[4 * k4 + 3], u.w, yb);
            }
            best = max2(best, add2(ya, yb));
        }
    }
    return best;
}

// A pillar of more than 32 points: straight from global memory, the whole warp on one pillar (rare: it reloads the lane's
// weights instead of taking them from the caller, so that the caller's copy never needs an address).
template <bool kTwo, bool kDyn>
__device__ __noinline__ void long_pillar(const WalkParams &p, uint32_t s_hist, uint32_t s_x, uint32_t p0, uint32_t n, int row,
                                         float cx, float cy, float cz, unsigned long long out_lane, int lane)
{
    const LaneWeights w = load_lane_weights(p.folded, lane);
    const uint32_t P = static_cast<uint32_t>(p.gd.max_points);  // 0x7FFFFFFF in the dynamic variant: nothing is dropped
    // dynamic variant: the row (rank of the cell in sorted-key order) was patched into the pillar's entry after the grouping
    if constexpr (kDyn) row = static_cast<int>(__ldcg(reinterpret_cast<const uint32_t *>(p.pillar_meta + p0) + 1));
    const bool has_pad = !kDyn && n < P;  // the dynamic variant has no padded slots (dynamic_pillar_vfe.py:48-53)
    // Pillars of up to 128 points (nearly all of them) keep their point indices in registers, 4 per lane: the radix select
    // and both passes then run without touching the index column again (one round trip instead of one per digit and pass).
    const bool small = n <= 128u;
    uint32_t id0[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint32_t j = q * 32u + lane;
        id0[q] = (small && j < n) ? __ldg(&p.records[p0 + j].idx) : 0xFFFFFFFFu;
    }
    uint32_t thr = 0xFFFFFFFFu;
    if (n > P) {
        // threshold = P-th smallest point index: the first P points in index order are kept.  Radix select with 8-bit digits:
        // one streaming pass over the pillar's indices per digit (3 passes for up to 16 M points), a 256-bin histogram in
        // shared memory (s_hist: 1 KB of the warp's region that is free after the walk).
        uint32_t prefix = 0, himask = 0, kk = P;
        for (int shift = ((p.idx_bits + 7) / 8) * 8 - 8; shift >= 0; shift -= 8) {
            sts4(s_hist + lane * 32u, make_float4(0.f, 0.f, 0.f, 0.f));
            sts4(s_hist + lane * 32u + 16, make_float4(0.f, 0.f, 0.f, 0.f));
            __syncwarp();
            if (small) {
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (q * 32u + lane < n && (id0[q] & himask) == prefix) atoms_add(s_hist + ((id0[q] >> shift) & 255u) * 4u, 1);
            } else {
                for (uint32_t j = lane; j < n; j += 32) {
                    const uint32_t v = __ldg(&p.records[p0 + j].idx);
                    if ((v & himask) == prefix) atoms_add(s_hist + ((v >> shift) & 255u) * 4u, 1);
                }
            }
            __syncwarp();
            const uint4 h0 = lds4u(s_hist + lane * 32u), h1 = lds4u(s_hist + lane * 32u + 16);  // bins 8*lane .. 8*lane+7
            const uint32_t bins[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
            uint32_t mine = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) mine += bins[k];
            uint32_t incl = mine;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t o = __shfl_up_sync(kFull, incl, d);
                if (lane >= d) incl += o;
            }
            const uint32_t excl = incl - mine;
            const bool owner = excl < kk && kk <= incl;  // exactly one lane: the matching indices number at least kk
            uint32_t digit = 0, before = excl;
            if (owner) {
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    if (before + bins[k] < kk) {
                        before += bins[k];
                        digit = k + 1;
                    } else {
                        break;
                    }
                }
                digit += 8u * lane;
            }
            const int src = __ffs(__ballot_sync(kFull, owner)) - 1;
            digit = __shfl_sync(kFull, digit, src);
            before = __shfl_sync(kFull, before, src);
            prefix |= digit << shift;
            himask |= 255u << shift;
            kk -= before;
            __syncwarp();
        }
        thr = prefix;
    }
    // The KEPT records (index <= thr; at most P of them when the cap binds, however long the pillar) are compacted into the
    // warp's 32-record scratch and handed to `body` 32 at a time.  The scan reads only the 4-byte indices, 128 per round
    // trip (4 independent loads per lane); the 32-byte records are fetched for kept points only.  (Before: every record of
    // the pillar went through both layers and the dropped ones were discarded at the max -- a 1000-point pillar with
    // P = 32 did 30x the work, and the drain of such pillars was the last 70-140 us of the two-layer kernel at cfg4 / cfg3.)
    auto for_kept = [&](auto &&body) {
        uint32_t fill = 0;
        for (uint32_t k0 = 0; k0 < n; k0 += 128u) {
            uint32_t id[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t j = k0 + q * 32u + lane;
                id[q] = small ? id0[q] : (j < n ? __ldg(&p.records[p0 + j].idx) : 0xFFFFFFFFu);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t j = k0 + q * 32u + lane;
                const bool keep = j < n && id[q] <= thr;
                const unsigned kb = __ballot_sync(kFull, keep);
                if (kb == 0u) continue;
                const uint32_t k = __popc(kb);
                if (fill + k > 32u) {
                    cp_async_commit();
                    cp_async_wait_all();
                    __syncwarp();
                    body(fill);
                    __syncwarp();
                    fill = 0;
                }
                if (keep) {  // global -> shared without registers: the kept records of a batch are all in flight together
                    const float4 *src = reinterpret_cast<const float4 *>(p.records + p0 + j);
                    const uint32_t dst = s_hist + (fill + __popc(kb & ((1u << lane) - 1u))) * 32u;
                    cp_async16(dst, src, 16);
                    cp_async16(dst + 16, src + 1, 16);
                }
                fill += k;
            }
        }
        if (fill) {
            cp_async_commit();
            cp_async_wait_all();
            __syncwarp();
            body(fill);
            __syncwarp();
        }
    };
    // pass 1: sums for the mean of the kept points (double: independent of the list order) and the running max of layer 0,
    // two records at a time (independent FFMA2 chains)
    double sx = 0.0, sy = 0.0, sz = 0.0;
    float2 acc = make_float2(-INFINITY, -INFINITY);
    for_kept([&](uint32_t cnt) {
        if (lane < cnt) {
            const float4 a = lds4(s_hist + lane * 32u);
            sx += static_cast<double>(a.x);
            sy += static_cast<double>(a.y);
            sz += static_cast<double>(a.z);
        }
        uint32_t k = 0;
        for (; k + 1u < cnt; k += 2) {
            const float2 ya = point_eval(w, s_hist + k * 32u), yb = point_eval(w, s_hist + k * 32u + 32u);
            acc = max3(acc, ya, yb);
        }
        if (k < cnt) acc = max2(acc, point_eval(w, s_hist + k * 32u));
    });
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        sx += __shfl_xor_sync(kFull, sx, s);
        sy += __shfl_xor_sync(kFull, sy, s);
        sz += __shfl_xor_sync(kFull, sz, s);
    }
    const float rn = __frcp_rn(static_cast<float>(min(n, P)));
    const float4 c4 = make_float4(cx, cy, cz, 0.f);
    const float4 m4 = make_float4(rel_mean(cx, static_cast<float>(sx) * rn), rel_mean(cy, static_cast<float>(sy) * rn),
                                  rel_mean(cz, static_cast<float>(sz) * rn), __int_as_float(row));
    if constexpr (!kTwo) {
        pillar_finish(w, c4, m4, has_pad, acc, out_lane);
    } else {
        // two layers: the pillar-wise max of layer 0 -> layer 1's constant, then a second pass over the records
        const Layer1 l1 = load_layer1(p.folded, p.folded2, lane);
        const bool padded = has_pad;
        const float2 kc = pillar_const(w, c4, m4);
        float2 m = add2(acc, kc);
        m.x = fmaxf(m.x, padded ? w.rsh.x : 0.f);
        m.y = fmaxf(m.y, padded ? w.rsh.y : 0.f);
        __syncwarp();
        sts2(s_x + 3u * kXBytes + lane * 8u, m);
        __syncwarp();
        const float2 cst = layer1_const(p.folded2 + 2048, s_x + 3u * kXBytes, l1.sh, lane);
        float2 best = make_float2(-INFINITY, -INFINITY);
        if (min(n, P) <= 32u)  // the kept records are still in the scratch, compacted by pass 1
            best = layer1_points(w, l1.wa, kc, cst, s_hist, min(n, P), s_x, lane, best);
        else
            for_kept([&](uint32_t cnt) { best = layer1_points(w, l1.wa, kc, cst, s_hist, cnt, s_x, lane, best); });
        if (padded) best = max2(best, add2(l1.upad, cst));
        if (row >= 0)
            asm volatile("st.global.v2.f32 [%0], {%1, %2};" ::"l"(out_lane + static_cast<unsigned long long>(static_cast<uint32_t>(row)) * 256ull),
                         "f"(fmaxf(best.x, 0.f)), "f"(fmaxf(best.y, 0.f))
                         : "memory");
    }
}

// Pillars of more than 32 points, listed by the grouping stage: every warp, once its own chunks are done, takes entries
// from the list through one grid-wide cursor, so the long tail is spread over the whole machine instead of serialising the
// warps whose chunks happen to contain it.
template <bool kTwo, bool kDyn>
__device__ __forceinline__ void drain_long_pillars(const WalkParams &p, uint32_t s_hist, uint32_t s_x, unsigned long long out_lane,
                                                   int lane)
{
    const uint32_t n_long = __ldcg(p.long_count) + 1u;
    if (n_long == 0u) return;
    while (true) {
        uint32_t i = 0;
        if (lane == 0) i = atomicAdd(p.long_cursor, 1u) + 1u;  // the cursor starts at 0xFFFFFFFF
        i = __shfl_sync(kFull, i, 0);
        if (i >= n_long) break;
        const uint4 e0 = __ldcg(p.long_list + 2 * i), e1 = __ldcg(p.long_list + 2 * i + 1);
        const float cx = __fadd_rn(__fmul_rn(static_cast<float>(e0.w & 0xFFFFu), p.vsz[0]), p.off[0]);
        const float cy = __fadd_rn(__fmul_rn(static_cast<float>(e0.w >> 16), p.vsz[1]), p.off[1]);
        const float cz = __fadd_rn(__fmul_rn(static_cast<float>(e1.x), p.vsz[2]), p.off[2]);
        long_pillar<kTwo, kDyn>(p, s_hist, s_x, e0.x, e0.y, static_cast<int>(e0.z), cx, cy, cz, out_lane, lane);
    }
}

// kTwo: a two-layer stack NUM_FILTERS [64, 64] (waymo_models/pointpillar_1x.yaml:34; pillar_vfe.py:18-19,44-49,119-120).
// Layer 0 (32 outputs: lanes 0-15 carry them, the folded table holds zeros for channels 32-63) is evaluated exactly like the
// single layer; its pillar-wise max m goes through shared memory into  cst = shift1 + (scale1 W1[:, 32:]) m  (weights in
// shared memory, once per pillar), then every kept point is evaluated again:  y = relu((scale1 W1[:, :32]) x_p + cst)  with
// the lane's 2 x 32 weights in registers, x_p broadcast from shared memory; padded slots contribute one row with
// x = relu(shift0) (NOT re-masked between the layers, as in the reference).  Pillars of more than 32 points: long_pillar<true>
// makes a second pass over the records.
// kDyn: DynamicPillarVFE / PFNLayerV2 semantics (dynamic_pillar_vfe.py:14-142): no cap and no padded slots, z neither range
// checked nor part of the cell, so z - z_offset is unbounded: its sum for the mean is a 64-bit fixed-point shared-memory
// atomic (2^-20 m); rows come from the pillar entries as patched by launch_dynamic_rows (sorted-key order).
template <int kWarps, int kMinBlocks, bool kTwo = false, bool kDyn = false>
__global__ void __launch_bounds__(32 * kWarps, kMinBlocks)
k_pillar_walk(const __grid_constant__ WalkParams p)
{
    constexpr uint32_t kOffZ64 = kTwo ? kWarpSmemTwo : kWarpSmem;  // dynamic variant: 32 x 8 bytes of z sums
    constexpr uint32_t kStride = kOffZ64 + (kDyn ? 256u : 0u);
    __shared__ __align__(16) unsigned char s_all[kWarps * kStride];
    __shared__ __align__(16) float s_w1b[kTwo ? 32 * 64 : 4];

    const int lane = threadIdx.x & 31;
    // (a shuffle result is warp-uniform by construction: the compiler then treats the chunk loop as convergent)
    const int warp = __shfl_sync(kFull, static_cast<int>(threadIdx.x >> 5), 0);
    if (threadIdx.x == 0) dbg_stamp(p.dbg, 18);
    pdl_wait();  // records, pillar entries and the list header come from the grouping kernels
    pdl_trigger();
    if (threadIdx.x == 0) dbg_stamp(p.dbg, 20);
    const uint32_t total = __ldcg(&p.hdr->total_listed);
    const uint32_t n_chunks = (total + 31u) >> 5;
    const uint32_t s_warp = static_cast<uint32_t>(__cvta_generic_to_shared(s_all)) + warp * kStride;
    const uint32_t s_pl = s_warp + kOffPl, s_sum = s_warp + kOffSum;
    const float qnan = __int_as_float(0x7fc00000);
    const uint32_t P = static_cast<uint32_t>(p.gd.max_points);
    // the lane's output base as a global-space address kept in registers (not recomputed per pillar)
    unsigned long long out_lane = static_cast<unsigned long long>(__cvta_generic_to_global(p.pillar_features + 2 * lane));
    asm volatile("" : "+l"(out_lane));

    // A warp owns a contiguous range of chunks.  (Handing chunks out one at a time through a grid-wide cursor was measured
    // SLOWER, 37-39 us against 33 us on cfg2, although per-warp times vary by +-40 %: neighbouring chunks then run on different
    // SMs and every window is fetched twice.)
    // Leaving the last chunks unassigned, for warps that finish their range to take one at a time from a grid-wide cursor,
    // was measured without gain for one layer (cfg2 34.8 us static, 36.9 us with 19-62 % pooled, 38.9 us all pooled; cfg3
    // 120.8 / 114.9 / 123.9 us; profiles/r02_walk_pool.txt) -- the late warps are not short of chunks, the SM is short of
    // issue slots -- so one layer uses static ranges only.  Two-layer stacks are the opposite case (a chunk costs 5-10x more
    // arithmetic, and 2.5x more when its pillars hold one point each; static ranges left the last warp running at 196 us when
    // the first was done at 18 us): there every chunk comes from the cursor.
    const uint32_t gw = blockIdx.x * kWarps + warp, n_warps = gridDim.x * kWarps;
    // Bulk phase: the cursor is read one chunk ahead (lane 0 keeps the reply of the atomic issued a chunk earlier) and the
    // next window is fetched during the current chunk, so a warp never waits for either round trip.  Tail phase (the last
    // 3 chunks per warp of the grid, two-layer stacks only): a chunk reserved ahead would sit idle behind a 16 us chunk while
    // other warps run dry -- with read-ahead everywhere the last warp finished at 142 us when the cursor ran out at 96 us --
    // so there a warp asks for its next chunk only when it is done with the current one.
    // A warp leaves only on an index >= n_chunks, and what it holds ahead is larger still.
    const uint32_t bulk_end = kTwo ? (n_chunks > 3u * n_warps ? n_chunks - 3u * n_warps : 0u) : 0xFFFFFFFFu;
    uint32_t ahead = 0;
    bool primed = false;
    auto grab = [&]() {
        if (!kTwo) return 0x7FFFFFFFu;  // one layer: no pool, nothing to wait for
        if (!primed && lane == 0) ahead = atomicAdd(p.chunk_cursor, 1u) + 1u;  // the cursor starts at 0xFFFFFFFF
        const uint32_t i = __shfl_sync(kFull, ahead, 0);
        primed = i < bulk_end;
        if (primed && lane == 0) ahead = atomicAdd(p.chunk_cursor, 1u) + 1u;
        return i;
    };
    const uint32_t n_static = kTwo ? 0u : n_chunks;
    uint32_t cur = static_cast<uint32_t>(static_cast<unsigned long long>(n_static) * gw / n_warps);
    const uint32_t c_end = static_cast<uint32_t>(static_cast<unsigned long long>(n_static) * (gw + 1) / n_warps);
    bool pooled = false;
    if (cur >= c_end) {
        pooled = true;
        cur = n_static + grab();
    }
    // chunk k -> buffer b: own records, look-ahead records, pillar entries (zero-filled beyond the end of the list)
    auto fetch = [&](uint32_t k, uint32_t b) {
        const uint32_t pos = (k << 5) + lane;
        const uint32_t dst = s_warp + b * kBufBytes + lane * 32u;
        const bool ok = pos < total, ok2 = pos + 32u < total;
        const float4 *src = reinterpret_cast<const float4 *>(p.records + (ok ? pos : 0u));
        cp_async16(dst, src, ok ? 16 : 0);
        cp_async16(dst + 16, src + 1, ok ? 16 : 0);
        const float4 *src2 = reinterpret_cast<const float4 *>(p.records + (ok2 ? pos + 32u : 0u));
        cp_async16(dst + 1024, src2, ok2 ? 16 : 0);
        cp_async16(dst + 1024 + 16, src2 + 1, ok2 ? 16 : 0);
        cp_async16(s_warp + b * kBufBytes + kRecBytes + lane * 16u, p.pillar_meta + (ok ? pos : 0u), ok ? 16 : 0);
    };

    const uint32_t s_x = s_warp + kOffX;
    Layer1 l1;
    if constexpr (kTwo) {
        for (int i = threadIdx.x; i < 32 * 64 / 4; i += 32 * kWarps)
            reinterpret_cast<float4 *>(s_w1b)[i] = __ldg(reinterpret_cast<const float4 *>(p.folded2 + 2048) + i);
        __syncthreads();
        l1 = load_layer1(p.folded, p.folded2, lane);
    }
    if (cur >= n_chunks) {
        drain_long_pillars<kTwo, kDyn>(p, s_pl, s_x, out_lane, lane);
        return;
    }
    fetch(cur, 0);
    cp_async_commit();
    const LaneWeights w = load_lane_weights(p.folded, lane);
    uint32_t buf = 0;
    cp_async_wait_all();
    __syncwarp();

    while (true) {
        // the next chunk's loads fly during this chunk's arithmetic
        uint32_t nxt = cur + 1u;
        const bool lazy = kTwo && cur >= bulk_end;  // tail phase: ask for the next chunk after this one
        if (!lazy) {
            if (pooled || nxt >= c_end) {
                pooled = true;
                nxt = n_static + grab();
            }
            if (nxt < n_chunks) fetch(nxt, buf ^ 1u);
        }
        cp_async_commit();
        const uint32_t rs = s_warp + buf * kBufBytes;  // window: 64 consecutive positions starting at chunk cur
        const uint32_t ms = rs + kRecBytes;
        const uint32_t pos = (cur << 5) + lane;

        // ---- phase 1 -----------------------------------------------------------------------------------------------------
        const uint4 rb = lds4u(rs + lane * 32u + 16);          // {time, flags, idx, arrival} of my own position
        const uint4 tb = lds4u(rs + (32u + lane) * 32u + 16);  // ... and of my look-ahead position
        const bool own_ok = pos < total, la_ok = pos + 32u < total;
        const bool is_start = own_ok && rb.w == 0u;
        const unsigned bal = __ballot_sync(kFull, is_start);
        if (bal != 0u) {
            sts1(s_sum + lane * 4u, 0u);
            sts1(s_sum + 128u + lane * 4u, 0u);
            sts1(s_sum + 256u + lane * 4u, 0u);
            if constexpr (kDyn) asm volatile("st.shared.u64 [%0], %1;" ::"r"(s_warp + kOffZ64 + lane * 8u), "l"(0ull) : "memory");
            __syncwarp();
            // every position adds itself to the sums of its pillar (when that pillar starts in this chunk and fits the
            // window); positions beyond the first-P cap are found by rank counting and become NaN
            auto contribute = [&](uint32_t j, uint32_t arrival, uint32_t idx) {
                if (arrival > j) return;  // the pillar started in an earlier chunk
                const uint32_t slot = j - arrival;
                if (slot >= 32u) return;  // starts in the next chunk
                const uint32_t np = lds1u(ms + slot * 16u + 8u);
                if (np > 32u) return;     // long pillar: taken from the long-pillar list
                bool keep = true;
                if (np > P) {
                    uint32_t rank = 0;
                    for (uint32_t k = 0; k < np; ++k) rank += lds1u(rs + (slot + k) * 32u + 24u) < idx ? 1u : 0u;
                    keep = rank < P;
                }
                if (keep) {
                    const float4 q = lds4(rs + j * 32u);
                    atoms_add(s_sum + slot * 4u, __float2int_rn(q.x * p.fx_scale[0]));
                    atoms_add(s_sum + 128u + slot * 4u, __float2int_rn(q.y * p.fx_scale[1]));
                    if constexpr (kDyn)
                        asm volatile("red.shared.add.u64 [%0], %1;" ::"r"(s_warp + kOffZ64 + slot * 8u),
                                     "l"(static_cast<unsigned long long>(__float2ll_rn(q.z * 1048576.f)))
                                     : "memory");
                    else
                        atoms_add(s_sum + 256u + slot * 4u, __float2int_rn(q.z * p.fx_scale[2]));
                } else {
                    sts1(rs + j * 32u, __float_as_uint(qnan));
                }
            };
            if (own_ok) contribute(lane, rb.w, rb.z);
            if (la_ok) contribute(32u + lane, tb.w, tb.z);
            __syncwarp();

            // the lane on a list start publishes the pillar's constants.  A pillar of more than 32 points does not fit the window
            // (it can only be the last start of the chunk): it is skipped here and taken from the long-pillar list later.
            unsigned rem = bal;
            {
                const uint4 me = lds4u(ms + lane * 16u);  // {x | y << 16, row, n, z}: valid on start lanes
                const uint32_t n = me.z;
                const bool is_long = is_start && n > 32u;
                if (is_start && !is_long) {
                    const float cx = __fadd_rn(__fmul_rn(static_cast<float>(me.x & 0xFFFFu), p.vsz[0]), p.off[0]);
                    const float cy = __fadd_rn(__fmul_rn(static_cast<float>(me.x >> 16), p.vsz[1]), p.off[1]);
                    const float cz = __fadd_rn(__fmul_rn(static_cast<float>(me.w), p.vsz[2]), p.off[2]);
                    const float rn = kRcp[min(n, P)];
                    const float mx = static_cast<float>(static_cast<int>(lds1u(s_sum + lane * 4u))) * p.fx_inv[0] * rn;
                    const float my = static_cast<float>(static_cast<int>(lds1u(s_sum + 128u + lane * 4u))) * p.fx_inv[1] * rn;
                    float mz;
                    if constexpr (kDyn) {
                        long long zs;
                        asm volatile("ld.shared.u64 %0, [%1];" : "=l"(zs) : "r"(s_warp + kOffZ64 + lane * 8u));
                        mz = __ll2float_rn(zs) * 9.5367431640625e-07f * rn;  // 2^-20
                    } else {
                        mz = static_cast<float>(static_cast<int>(lds1u(s_sum + 256u + lane * 4u))) * p.fx_inv[2] * rn;
                    }
                    // n with bit 31 set when the pillar has empty (padded) slots
                    sts4(s_pl + lane * 32u, make_float4(cx, cy, cz, __uint_as_float(n | (!kDyn && n < P ? 0x80000000u : 0u))));
                    sts4(s_pl + lane * 32u + 16, make_float4(rel_mean(cx, mx), rel_mean(cy, my), rel_mean(cz, mz),
                                                             __uint_as_float(me.y)));
                }
                rem &= ~__ballot_sync(kFull, is_long);
                __syncwarp();
            }

            // ---- phase 2: the warp walks the pillars that start among its 32 positions; lane = channel pair.  TWO pillars per
            //      trip: their first-point chains and constant chains are four independent FFMA2 chains in one straight-line
            //      block; further points of a pillar are evaluated two at a time.
            if constexpr (kTwo) {
                while (rem) {
                    const uint32_t slot = __ffs(rem) - 1;
                    rem &= rem - 1;
                    const uint32_t pa = rs + slot * 32u;
                    const float4 c4 = lds4(s_pl + slot * 32u), m4 = lds4(s_pl + slot * 32u + 16);
                    const float2 kc = pillar_const(w, c4, m4);
                    const uint32_t nbits = __float_as_uint(c4.w), n = nbits & 0x7FFFFFFFu;
                    const bool padded = static_cast<int>(nbits) < 0;
                    const int row = __float_as_int(m4.w);
                    // pass A: pillar-wise max of layer 0 (ReLU and the constant commute with the max; dropped points are NaN)
                    float2 acc = point_eval(w, pa);
                    if (n > 1u) acc = more_points(w, pa, n, acc);
                    float2 m = add2(acc, kc);
                    m.x = fmaxf(m.x, padded ? w.rsh.x : 0.f);
                    m.y = fmaxf(m.y, padded ? w.rsh.y : 0.f);
                    __syncwarp();  // the previous pillar's reads of the x buffers
                    sts2(s_x + 3u * kXBytes + lane * 8u, m);
                    __syncwarp();
                    const float2 cst = layer1_const(s_w1b, s_x + 3u * kXBytes, l1.sh, lane);
                    // pass B: layer 1 on [x_p, m] for every kept point
                    float2 best = layer1_points(w, l1.wa, kc, cst, pa, n, s_x, lane, make_float2(-INFINITY, -INFINITY));
                    if (padded) best = max2(best, add2(l1.upad, cst));
                    if (row >= 0)
                        asm volatile("st.global.v2.f32 [%0], {%1, %2};" ::"l"(out_lane + static_cast<unsigned long long>(static_cast<uint32_t>(row)) * 256ull),
                                     "f"(fmaxf(best.x, 0.f)), "f"(fmaxf(best.y, 0.f))
                                     : "memory");
                }
            }
            while (!kTwo && rem) {
                const uint32_t slot_a = __ffs(rem) - 1;
                rem &= rem - 1;
                const bool has_b = rem != 0u;
                const uint32_t slot_b = has_b ? static_cast<uint32_t>(__ffs(rem) - 1) : slot_a;
                rem &= rem - 1;  // (0 & anything stays 0)
                const uint32_t pa = rs + slot_a * 32u, pb = rs + slot_b * 32u;
                const float4 c4a = lds4(s_pl + slot_a * 32u), m4a = lds4(s_pl + slot_a * 32u + 16);
                const float4 c4b = lds4(s_pl + slot_b * 32u), m4b = lds4(s_pl + slot_b * 32u + 16);
                float2 acc_a = point_eval(w, pa), acc_b = point_eval(w, pb);
                const float2 kc_a = pillar_const(w, c4a, m4a), kc_b = pillar_const(w, c4b, m4b);
                const uint32_t nba = __float_as_uint(c4a.w), nbb = __float_as_uint(c4b.w);
                const uint32_t na = nba & 0x7FFFFFFFu, nb2 = nbb & 0x7FFFFFFFu;
                if ((na | nb2) > 1u) {  // some pillar of the pair has more points
                    if (na > 1u) acc_a = more_points(w, pa, na, acc_a);
                    if (nb2 > 1u && has_b) acc_b = more_points(w, pb, nb2, acc_b);
                }
                pillar_store(w, kc_a, __float_as_int(m4a.w), static_cast<int>(nba) < 0, acc_a, out_lane);
                if (has_b) pillar_store(w, kc_b, __float_as_int(m4b.w), static_cast<int>(nbb) < 0, acc_b, out_lane);
            }
        }
        if (lazy) {
            nxt = n_static + grab();
            if (nxt < n_chunks) fetch(nxt, buf ^ 1u);
            cp_async_commit();
        }
        cp_async_wait_all();
        __syncwarp();
        cur = nxt;
        if (cur >= n_chunks) break;
        buf ^= 1u;
    }
    if (lane == 0) {
        dbg_stamp(p.dbg, 21);  // chunks done (latest warp)
        dbg_stamp(p.dbg, 22);  // (earliest warp)
    }
    drain_long_pillars<kTwo, kDyn>(p, s_pl, s_x, out_lane, lane);
    if (lane == 0) {
        dbg_stamp(p.dbg, 23);
        dbg_stamp(p.dbg, 24);
    }
}

// ---- the reference's own padded input: voxels [M, P, C], num_points [M], coords [M, 4] (b, z, y, x) ----------------------
// PillarVFE.forward on what the data processor's voxeliser hands over (pillar_vfe.py:86-123), in the same folded form as the
// walk above: a warp takes one pillar at a time (pillars strided over the persistent warps), lane = slot while the pillar
// is loaded -- 20-byte slots, 640 contiguous bytes per pillar at P = 32 -- and turned into the 32-byte records point_eval
// reads, lane = channel pair while the valid points are evaluated.  The mean is the reference's: the sum over ALL P slots,
// whatever the padding holds, divided by num_points (:97), in a fixed shuffle order (bit-reproducible).
struct PaddedParams {
    const float *voxels;
    const void *num_points, *coords;
    int np_float, coords_float;
    int64_t m;
    int P, C;
    const float *folded;
    float vsz[3], off[3];
    float fx_scale[3], fx_inv[3], extent[3];  // fixed-point sums of the valid slots: scale, inverse, |x - centre| bound
    float *out;
};

// what a warp needs of a pillar before it can start: the header and its slot (one per lane, P <= 32)
struct PaddedHead {
    float nf, fx, fy, fz, x, y, z, a, t;
    int n;
};

__device__ __forceinline__ PaddedHead padded_fetch(const PaddedParams &p, int64_t g, int lane)
{
    PaddedHead h;
    if (p.np_float) {
        h.nf = __ldg(static_cast<const float *>(p.num_points) + g);
        h.n = static_cast<int>(h.nf);  // .int() in get_paddings_indicator (pillar_vfe.py:91)
    } else {
        h.n = __ldg(static_cast<const int32_t *>(p.num_points) + g);
        h.nf = static_cast<float>(h.n);  // .type_as(voxel_features) (pillar_vfe.py:97)
    }
    if (p.coords_float) {
        const float4 c4 = __ldg(reinterpret_cast<const float4 *>(static_cast<const float *>(p.coords) + g * 4));
        h.fz = c4.y; h.fy = c4.z; h.fx = c4.w;
    } else {
        const int4 c4 = __ldg(reinterpret_cast<const int4 *>(static_cast<const int32_t *>(p.coords) + g * 4));
        h.fz = static_cast<float>(c4.y); h.fy = static_cast<float>(c4.z); h.fx = static_cast<float>(c4.w);
    }
    h.x = h.y = h.z = h.a = h.t = 0.f;
    if (lane < p.P) {
        const float *q = p.voxels + (g * p.P + lane) * p.C;
        h.x = __ldg(q);
        h.y = __ldg(q + 1);
        h.z = __ldg(q + 2);
        if (p.C > 3) h.a = __ldg(q + 3);
        if (p.C > 4) h.t = __ldg(q + 4);
    }
    return h;
}

__device__ __forceinline__ void padded_pillar(const PaddedParams &p, const LaneWeights &w, const PaddedHead &h, int64_t g,
                                              uint32_t s_rec, unsigned long long out_lane, int lane)
{
    const float cx = __fadd_rn(__fmul_rn(h.fx, p.vsz[0]), p.off[0]);
    const float cy = __fadd_rn(__fmul_rn(h.fy, p.vsz[1]), p.off[1]);
    const float cz = __fadd_rn(__fmul_rn(h.fz, p.vsz[2]), p.off[2]);
    const int n_valid = __shfl_sync(kFull, max(0, min(h.n, p.P)), 0);  // (uniform anyway; the shuffle tells the compiler)
    const float rx = __fsub_rn(h.x, cx), ry = __fsub_rn(h.y, cy), rz = __fsub_rn(h.z, cz);
    // Sum over ALL P slots (pillar_vfe.py:97).  What a voxeliser hands over -- valid points inside their pillar, zeros in
    // the padding -- is summed exactly: fixed-point integers relative to the pillar centre, one redux.sync per axis.
    // Anything else (non-zero padding, a "valid" point outside its pillar, num_points outside 1..P) takes the float path.
    int ix = 0, iy = 0, iz = 0;
    bool odd;
    if (lane < n_valid) {
        odd = !(fabsf(rx) <= p.extent[0] && fabsf(ry) <= p.extent[1] && fabsf(rz) <= p.extent[2]);
        ix = __float2int_rn(rx * p.fx_scale[0]);
        iy = __float2int_rn(ry * p.fx_scale[1]);
        iz = __float2int_rn(rz * p.fx_scale[2]);
    } else {
        odd = h.x != 0.f || h.y != 0.f || h.z != 0.f;  // (lanes beyond P hold zeros)
    }
    odd |= h.n != n_valid || h.n < 1;
    __syncwarp();  // the previous pillar's records have been read
    sts4(s_rec + lane * 32u, make_float4(rx, ry, rz, h.a));
    sts1(s_rec + lane * 32u + 16u, __float_as_uint(h.t));
    __syncwarp();
    float2 acc = make_float2(-INFINITY, -INFINITY);
    int k = 0;
    for (; k + 1 < n_valid; k += 2) {
        const float2 ya = point_eval(w, s_rec + k * 32u), yb = point_eval(w, s_rec + k * 32u + 32u);
        acc = max3(acc, ya, yb);
    }
    if (k < n_valid) acc = max2(acc, point_eval(w, s_rec + k * 32u));
    float mrx, mry, mrz;  // mean - centre
    if (!__any_sync(kFull, odd)) {
        const float rn = __frcp_rn(h.nf);
        mrx = rel_mean(cx, static_cast<float>(__reduce_add_sync(kFull, ix)) * p.fx_inv[0] * rn);
        mry = rel_mean(cy, static_cast<float>(__reduce_add_sync(kFull, iy)) * p.fx_inv[1] * rn);
        mrz = rel_mean(cz, static_cast<float>(__reduce_add_sync(kFull, iz)) * p.fx_inv[2] * rn);
    } else {
        float sx = h.x, sy = h.y, sz = h.z;
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
            sx = __fadd_rn(sx, __shfl_xor_sync(kFull, sx, s));
            sy = __fadd_rn(sy, __shfl_xor_sync(kFull, sy, s));
            sz = __fadd_rn(sz, __shfl_xor_sync(kFull, sz, s));
        }
        mrx = __fsub_rn(__fdiv_rn(sx, h.nf), cx);
        mry = __fsub_rn(__fdiv_rn(sy, h.nf), cy);
        mrz = __fsub_rn(__fdiv_rn(sz, h.nf), cz);
    }
    const float4 c4 = make_float4(cx, cy, cz, 0.f);
    const float4 m4 = make_float4(mrx, mry, mrz, __int_as_float(static_cast<int>(g)));
    pillar_finish(w, c4, m4, n_valid < p.P, acc, out_lane);
}

// P <= 32 (every pillar configuration of the reference: 20 / 32): one slot per lane.  The NEXT pillar's loads are issued
// before the current one is processed (two heads in ping-pong, the loop unrolled by two so that neither is copied).
template <int kWarps>
__global__ void __launch_bounds__(32 * kWarps, 6) k_pfn_padded(const __grid_constant__ PaddedParams p)
{
    __shared__ __align__(16) unsigned char s_all[kWarps * 1024];
    const int lane = threadIdx.x & 31;
    // warp-uniform by construction (a shuffle result), so the compiler sees the pillar loop as convergent and the *_sync
    // operations inside it stay single instructions instead of convergence-barrier sequences
    const int warp = __shfl_sync(kFull, static_cast<int>(threadIdx.x >> 5), 0);
    const uint32_t s_rec = static_cast<uint32_t>(__cvta_generic_to_shared(s_all)) + warp * 1024u;
    const LaneWeights w = load_lane_weights(p.folded, lane);
    const unsigned long long out_lane = static_cast<unsigned long long>(__cvta_generic_to_global(p.out + 2 * lane));
    const int64_t n_warps = static_cast<int64_t>(gridDim.x) * kWarps;
    int64_t g = static_cast<int64_t>(blockIdx.x) * kWarps + warp;
    if (g >= p.m) return;
    PaddedHead a = padded_fetch(p, g, lane), b = a;
    while (true) {
        const bool has_b = g + n_warps < p.m;
        if (has_b) b = padded_fetch(p, g + n_warps, lane);
        padded_pillar(p, w, a, g, s_rec, out_lane, lane);
        if (!has_b) break;
        g += n_warps;
        const bool has_a = g + n_warps < p.m;
        if (has_a) a = padded_fetch(p, g + n_warps, lane);
        padded_pillar(p, w, b, g, s_rec, out_lane, lane);
        if (!has_a) break;
        g += n_warps;
    }
}

// ---- folding of the layer's weights (once per model: pillars_fold_pfn) ------------------------------------------------
__global__ void k_fold_pfn(const float *__restrict__ weight, const float *__restrict__ scale,
                           const float *__restrict__ shift, int c_point, int c_in, int f_out, float *__restrict__ folded)
{
    pdl_wait();  // a link of the stack paths' launch chain (a no-op in a plain launch)
    pdl_trigger();
    const int o = threadIdx.x;
    if (o >= 64) return;
    if (o >= f_out) {  // a 32-output layer 0 of a two-layer stack: the upper channels are zeros throughout
        for (int r = 0; r < 13; ++r) folded[r * 64 + o] = 0.f;
        return;
    }
    const float *w = weight + static_cast<size_t>(o) * c_in;  // feature order: p[0..c), cluster xyz, centre xyz
    const double s = scale[o];
    const int c = c_point;
    for (int a = 0; a < 3; ++a) {
        folded[a * 64 + o] = static_cast<float>(s * (static_cast<double>(w[a]) + w[c + a] + w[c + 3 + a]));
        folded[(5 + a) * 64 + o] = static_cast<float>(s * w[a]);
        folded[(8 + a) * 64 + o] = -static_cast<float>(s * w[c + a]);
    }
    folded[3 * 64 + o] = c > 3 ? static_cast<float>(s * w[3]) : 0.f;
    folded[4 * 64 + o] = c > 4 ? static_cast<float>(s * w[4]) : 0.f;
    const float sh = shift[o];
    folded[11 * 64 + o] = sh;
    folded[12 * 64 + o] = fmaxf(sh, 0.f);
}

}  // namespace

cudaError_t launch_fold_pfn(const PfnDev &pfn, int c_point, int c_in, float *folded, cudaStream_t st, int f_out)
{
    const cudaError_t e = launch_pdl(k_fold_pfn, dim3(1), dim3(64), 0, st, pfn.weight, pfn.scale, pfn.shift, c_point, c_in, f_out, folded);
    if (e != cudaSuccess) return e;
    note_launch();
    return cudaGetLastError();
}

// layer 1 of a [64, 64] stack: weight [64][64] (inputs 0-31 per point, 32-63 the pillar-wise max), BatchNorm scale folded in
__global__ void k_fold_pfn2(const float *__restrict__ weight, const float *__restrict__ scale, const float *__restrict__ shift,
                            float *__restrict__ folded2)
{
    pdl_wait();
    pdl_trigger();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;  // (k, j): input k of both halves, output j
    if (i >= 32 * 64) return;
    const int k = i >> 6, j = i & 63;
    const float s = scale[j];
    folded2[k * 64 + j] = s * weight[j * 64 + k];
    folded2[2048 + k * 64 + j] = s * weight[j * 64 + 32 + k];
    if (k == 0) folded2[4096 + j] = shift[j];
}

cudaError_t launch_fold_pfn2(const float *weight, const float *scale, const float *shift, float *folded2, cudaStream_t st)
{
    const cudaError_t e = launch_pdl(k_fold_pfn2, dim3(8), dim3(256), 0, st, weight, scale, shift, folded2);
    if (e != cudaSuccess) return e;
    note_launch();
    return cudaGetLastError();
}

cudaError_t launch_pfn_padded(const float *voxels, const void *num_points, bool np_float, const void *coords, bool coords_float,
                              int64_t m, int max_points, int c_point, const PfnDev &pfn, const float *folded, float *out,
                              cudaStream_t st)
{
    if (m == 0) return cudaSuccess;
    PaddedParams p{};
    p.voxels = voxels;
    p.num_points = num_points;
    p.coords = coords;
    p.np_float = np_float ? 1 : 0;
    p.coords_float = coords_float ? 1 : 0;
    p.m = m;
    p.P = max_points;
    p.C = c_point;
    p.folded = folded;
    for (int k = 0; k < 3; ++k) {
        p.vsz[k] = pfn.vsz[k];
        p.off[k] = pfn.off[k];
    }
    p.out = out;
    for (int k = 0; k < 3; ++k) {
        // |x - centre| <= voxel / 2 (+ rounding) for a point inside its pillar; the sum of P such values stays below 2^31
        const double extent = 0.5 * static_cast<double>(pfn.vsz[k]) * 1.01 + 1e-6;
        int sc = static_cast<int>(std::floor(std::log2(2147483647.0 / (static_cast<double>(max_points) * extent))));
        sc = sc < -60 ? -60 : (sc > 60 ? 60 : sc);
        p.fx_scale[k] = static_cast<float>(std::ldexp(1.0, sc));
        p.fx_inv[k] = static_cast<float>(std::ldexp(1.0, -sc));
        p.extent[k] = static_cast<float>(extent);
    }
    constexpr int kWarps = 4;
    const int64_t wave = static_cast<int64_t>(current_sm_count()) * 6;
    const int64_t blocks = tmin<int64_t>((m + kWarps - 1) / kWarps, wave);
    k_pfn_padded<kWarps><<<static_cast<unsigned>(blocks), 32 * kWarps, 0, st>>>(p);
    note_launch();
    return cudaGetLastError();
}

cudaError_t launch_pillar_features_stream(const FastJob &job, const float *folded, const GridDev &gd, const Workspace &ws,
                                          cudaStream_t st)
{
    if (job.n == 0) return cudaSuccess;
    WalkParams p{};
    p.records = ws.records;
    p.hdr = ws.hdr;
    p.pillar_meta = ws.pillar_meta;
    p.long_list = ws.long_list;
    p.long_count = ws.long_count;
    p.long_cursor = ws.long_cursor;
    p.chunk_cursor = ws.long_cursor ? ws.long_cursor + 16 : nullptr;  // same 0xFF-filled 256-byte block, own 64-byte line
    p.folded = folded;
    p.folded2 = job.folded2;
    p.pillar_features = job.pillar_features;
    p.gd = gd;
    p.sh_cells = log2_exact(gd.cells);
    p.sh_cells_xy = log2_exact(gd.cells_xy);
    p.sh_nx = log2_exact(static_cast<uint32_t>(gd.g[0]));
    p.idx_bits = job.idx_bits;
    p.dbg = debug_times_ptr();
    const int window = gd.max_points < 32 ? gd.max_points : 32;  // points that can enter one sum
    for (int k = 0; k < 3; ++k) {
        p.vsz[k] = job.vsz[k];
        p.off[k] = job.off[k];
        // |x'| <= voxel / 2 (+ rounding); the sum of `window` fixed-point values must stay below 2^31
        const double extent = 0.5 * static_cast<double>(gd.vsz[k]) * 1.01 + 1e-6;
        int s = static_cast<int>(std::floor(std::log2(2147483647.0 / (window * extent))));
        s = s < -60 ? -60 : (s > 60 ? 60 : s);
        p.fx_scale[k] = static_cast<float>(std::ldexp(1.0, s));
        p.fx_inv[k] = static_cast<float>(std::ldexp(1.0, -s));
    }
    // Persistent warps, one per two chunks, at most one full wave of `occ` CTAs per SM (the kernel's minimum-blocks bound).
    const int sms = current_sm_count();
    constexpr int kWarps = 4;
    const int64_t chunks = (job.n + 31) / 32;  // upper bound: listed points <= n
    auto grid = [&](int occ) {
        return dim3(static_cast<unsigned>((tmin<int64_t>((chunks + 1) / 2, static_cast<int64_t>(sms) * occ * kWarps) + kWarps - 1) / kWarps));
    };
    cudaError_t err;
    if (job.dynamic)  // DynamicPillarVFE (one or two layers)
        err = job.folded2 ? launch_pdl(k_pillar_walk<kWarps, 3, true, true>, grid(3), dim3(32 * kWarps), 0, st, p)
                          : launch_pdl(k_pillar_walk<kWarps, 5, false, true>, grid(5), dim3(32 * kWarps), 0, st, p);
    else  // PillarVFE; a two-layer stack has 64 more weight registers per lane: 3 CTAs per SM
        err = job.folded2 ? launch_pdl(k_pillar_walk<kWarps, 3, true>, grid(3), dim3(32 * kWarps), 0, st, p)
                          : launch_pdl(k_pillar_walk<kWarps, 5>, grid(5), dim3(32 * kWarps), 0, st, p);
    if (err != cudaSuccess) return err;
    note_launch();
    return cudaGetLastError();
}

}  // namespace pillars
