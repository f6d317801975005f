// 2-D convolutions of the BEV backbone (base_bev_backbone.py:29-69) as implicit GEMMs on the 5th-generation tensor cores.
//
//   out[b, oy, ox, n] = relu( shift[n] + sum_{ky, kx, c} in[b, oy * s + ky - pad, ox * s + kx - pad, c] * w'[n, c, ky, kx] )
//
// with w' = bn_scale[n] * w (eval-mode BatchNorm folded into the weights, base_bev_backbone.py:36 eps = 1e-3) and tf32 operands /
// fp32 accumulation (what the reference's own nn.Conv2d does on this GPU under torch.backends.cudnn.allow_tf32 = True).
//
// One CTA computes T stacked 16 x 8 patches of output pixels (M = 128 rows of the MMA each) for ALL output channels
// (N = 64 / 128 / 256 accumulator columns each, T * N <= 512 columns of tensor memory).  Activations are NHWC, so the 32
// channels of one pixel are one 128-byte row of a K-major, 128-byte-swizzled operand tile.  The point of the design:
//
//   * ONE halo tile per 32-channel block serves all k x k taps.  The tensor core applies the 128-byte swizzle to ABSOLUTE
//     shared-memory address bits (profiles/micro/umma_shifted_desc.cu: any start row, any 16-byte-multiple group stride,
//     base offset 0), so tap (ky, kx) is the same buffer behind a descriptor that starts (ky * pitch + kx) pixel rows further
//     and strides `pitch` rows between its 8-row groups.  Activation traffic from L2 is (halo / patch) ~ 1.3x instead of 9x.
//   * stride-2 layers store the halo as four parity planes (even/odd row x even/odd column); every tap is again a shifted
//     view of one plane.  The first layer can gather its pixels from the PILLAR ROWS through the BEV index map: the dense
//     canvas (1 GiB at 16 x 64 x 512^2) is never read -- or written, if nothing else wants it.
//   * weights arrive as a ready-made shared-memory image (K-major, swizzled, BN scale folded, rounded to tf32), one bulk
//     copy per (channel block, tap), shared by the T patches.
//
// Warp roles (192 threads): warps 0-3 load the halo with cp.async (zero fill = padding) and later run the epilogue out of
// tensor memory (thread = accumulator lane = output pixel); warp 4 issues the MMAs; warp 5 issues the weight copies.
#include "common.cuh"

namespace pillars {

namespace {

constexpr int kConvThreads = 352;  // 4 loader warps, 2 MMA-issue warps (the second only when MW == 2), 1 weight warp, 4 epilogue warps
constexpr int kLoaders = 128;
constexpr int kPatchW = 8, kPatchH = 16;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
// K-major, 128-byte swizzle; sbo = bytes between 8-row groups (any multiple of 16: the swizzle follows the absolute address)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t sbo)
{
    return static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4) | (static_cast<uint64_t>(sbo >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ uint32_t umma_idesc_tf32(int n)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | ((128u >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0), "r"(0), "r"(0), "r"(0)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t mbar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t mbar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mbar) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
// bounded: a set-up mistake becomes an error code, not a hung GPU
__device__ __forceinline__ bool mbar_wait(uint32_t mbar, uint32_t parity, volatile uint32_t *abort_flag)
{
    for (uint32_t spin = 0; spin < (1u << 15); ++spin) {
        uint32_t ok;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(ok)
                     : "r"(mbar), "r"(parity)
                     : "memory");
        if (ok) return true;
        if (*abort_flag) return false;
    }
    *abort_flag = 1u;
    return false;
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t mbar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(mbar)
                 : "memory");
}
__device__ __forceinline__ void cp_async16_zfill(uint32_t dst, const void *src, bool valid)
{
    const uint32_t n = valid ? 16u : 0u;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32])
{
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, "
        "%18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n\ttcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
}
// the same load without the wait, and the wait as a separate statement that "produces" the registers (so that no use of
// them can be scheduled above it): the next chunk's load runs under this chunk's arithmetic and stores
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, "
        "%18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                   "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                   "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                   "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :
                 : "memory");
}
__device__ __forceinline__ float round_tf32(float x)
{
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

struct ConvParams {
    const float *in;          // NHWC [nb, h_in, w_in, c_in] (dense input)
    const float *rows;        // [M, c_in] pillar rows (gathered input), with cell_row [nb, h_in, w_in]
    const int32_t *cell_row;
    const uint8_t *wimg;      // [phase][c_in / 32][taps][N x 128 B] shared-memory images
    const float *shift;       // [N]
    float *out;
    int nb, h_in, w_in, c_in;
    int h_out, w_out;         // output pixels of the convolution proper
    int stride, pad, taps;
    int plane_rows;           // stride 2: pixel rows of one parity plane
    int pitch;                // pixel rows between vertically adjacent pixels of the halo (or of a plane)
    int stage_rows;           // pixel rows (128 B each) of one halo stage
    int tap_off[9];           // start of each tap's view, in pixel rows
    int tiles_x, tiles_y;
    // where an output pixel goes: (oy * out_mul + ph_y, ox * out_mul + ph_x) of a [nb, out_h, out_w] image with out_c_total
    // channels, this layer's starting at out_c_off; phases (transposed convolution) are blockIdx.z
    int out_mul, out_h, out_w, out_c_total, out_c_off, out_nchw;
    int relu, round_out;
    int pair;                 // transposed convolution: two dx phases per accumulator (N = 2 * c_out)
    uint32_t *error;          // device word: nonzero when a bounded wait expired
    unsigned long long *timeline;  // measurement hook (pillars_set_debug_times): one CTA's phase stamps, %globaltimer ns
    // residual kernels (RES): NHWC fp32, laid out exactly like `out` (same pixel pitch, same channel window), added before the
    // ReLU.  (last, so that the kernels without it keep every parameter offset)
    const float *res;
};

__device__ __forceinline__ void tl_stamp(const ConvParams &p, int slot)
{
    if (p.timeline && blockIdx.x == 100 && blockIdx.z == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        p.timeline[slot] = t;
    }
}

// Persistent: a CTA walks over tile sets (tile = blockIdx.x, += gridDim.x).  With NB = 2 the accumulator is double buffered in
// tensor memory, so the epilogue of tile set i (warps 6-9) runs under the MMAs of tile set i + 1, and the loaders (warps 0-3)
// run ahead into the next tile set's halo as soon as a stage is released -- no prologue or epilogue is exposed after the first.
// RES: the residual epilogue (ResNet BasicBlock, y = relu(acc + shift + residual)); only the NHWC epilogue of a plain
// convolution reads it (the host refuses a residual with NCHW output or a transposed convolution).
template <int N, int T, int SA, int SB, int NB, int MW = 1, int MB = 1, bool RES = false>
__global__ void __launch_bounds__(kConvThreads, MB) k_conv_umma(const __grid_constant__ ConvParams p)
{
    extern __shared__ __align__(1024) uint8_t s_raw[];
    __shared__ uint64_t s_bar[2 * SA + 2 * SB + 2 * NB];
    __shared__ uint32_t s_tmem;
    __shared__ uint32_t s_abort_word;
    __shared__ float s_shift[N];
    volatile uint32_t *const s_abort = &s_abort_word;

    const int tid = threadIdx.x, lane = tid & 31;
    // (the shuffle tells the compiler that the role branches below are warp-uniform: the MMA warp then runs converged and its
    // tcgen05 instructions are issued under one elected lane instead of a per-instruction election loop)
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    if (tid == 0) tl_stamp(p, 0);  // CTA start
    uint8_t *const s_al = s_raw + ((1024u - (smem_u32(s_raw) & 1023u)) & 1023u);
    const uint32_t a_bytes = (static_cast<uint32_t>(p.stage_rows) * 128u + 1023u) & ~1023u;
    constexpr uint32_t b_bytes = static_cast<uint32_t>(N) * 128u;
    const uint32_t a0 = smem_u32(s_al), b0 = a0 + SA * a_bytes;
    uint8_t *const s_stage = s_al + SA * a_bytes + SB * b_bytes;  // 4 x 4 KB: the epilogue warps' transposition buffers
    int32_t *const s_src = reinterpret_cast<int32_t *>(s_stage + 4 * 4096);  // [stage_rows] source of each pixel row
    const int occ_cap = ((p.stage_rows + 15) >> 4) * 4 + 8;  // pixel rows one loader warp owns (+ slack)
    // gathered input: per loader warp, the occupied pixel rows of this and of the previous tile set
    uint16_t *const s_occ = reinterpret_cast<uint16_t *>(s_src + ((p.stage_rows + 15) & ~15));
    const uint32_t bar0 = smem_u32(s_bar);
    const uint32_t a_full = bar0, a_empty = bar0 + 8u * SA, b_full = bar0 + 16u * SA, b_empty = b_full + 8u * SB,
                   acc_full = b_empty + 8u * SB, acc_empty = acc_full + 8u * NB;
    constexpr uint32_t acc_cols = T * N;
    constexpr uint32_t tmem_cols = (NB * acc_cols <= 32) ? 32u : (NB * acc_cols <= 64) ? 64u : (NB * acc_cols <= 128) ? 128u
                                   : (NB * acc_cols <= 256) ? 256u : 512u;
    static_assert(NB * acc_cols <= 512, "tensor memory has 512 columns");

    const int tiles_per_frame = p.tiles_x * p.tiles_y;
    const int total_tiles = p.nb * tiles_per_frame;
    const int phase = blockIdx.z;
    const int cbn = p.c_in >> 5;
    const auto tile_origin = [&](int tile, int &b, int &y0, int &x0) {
        b = tile / tiles_per_frame;
        const int tr = tile - b * tiles_per_frame, ty = tr / p.tiles_x;
        y0 = ty * (kPatchH * T);
        x0 = (tr - ty * p.tiles_x) * kPatchW;
    };

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "r"(tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
        for (int i = 0; i < SA; ++i) {
            mbar_init(a_full + 8u * i, kLoaders);
            mbar_init(a_empty + 8u * i, MW);
        }
        for (int i = 0; i < SB; ++i) {
            mbar_init(b_full + 8u * i, 1);
            mbar_init(b_empty + 8u * i, MW);
        }
        for (int i = 0; i < NB; ++i) {
            mbar_init(acc_full + 8u * i, MW);
            mbar_init(acc_empty + 8u * i, kLoaders);  // the 128 epilogue threads
        }
        s_abort_word = 0u;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < (p.pair ? N / 2 : N); i += kConvThreads) s_shift[i] = __ldg(p.shift + i);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    if (tid == 0) tl_stamp(p, 1);  // set-up done
    // Programmatic dependent launch: the next layer's CTAs may take an SM as soon as one of this grid's CTAs retires, and do
    // their own set-up (tensor-memory allocation, barriers, the first weight copies: weights are not produced by a
    // predecessor) while the tail of this grid is still working; whatever reads or writes activations waits below.
    pdl_trigger();

    if (warp < 4) {
        // ================================ halo loaders ===========================================================================
        // A thread loads chunk ch of the pixel rows px = (tid >> 3) + 16 j; a WARP therefore owns the rows with
        // (px mod 16) / 4 == warp, fills exactly those entries of the source table and needs no barrier wider than itself.
        // The table says where each pixel row comes from (the pixel's index in the source array, -1 = zero fill: padding,
        // empty cell, outside the image): divisions, bounds and -- for a gathered input -- the index-map lookups are done once
        // per tile set, not once per channel block.
        const int ch = tid & 7;
        const float *const base = (p.rows ? p.rows : p.in) + ch * 4;
        const uint32_t dst0 = static_cast<uint32_t>(tid >> 3) * 128u + (static_cast<uint32_t>(ch ^ ((tid >> 3) & 7)) << 4);
        int ia = 0;
        bool ok = true;
        // (a stage's previous content must stem from this or the previous tile set: it is reused every SA channel blocks)
        const bool sparse = p.rows != nullptr && cbn >= SA;
        int n_prev = 0, n_tiles_done = 0;
        pdl_wait();  // the activations / pillar rows / index map are the predecessor's output
        if (sparse) {  // every pixel row of every stage starts as zeros; only occupied cells are ever written
            for (uint32_t i = tid; i < (SA * a_bytes) >> 4; i += kLoaders)
                asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(a0 + (i << 4)), "r"(0) : "memory");
            asm volatile("bar.sync 1, %0;" ::"n"(kLoaders) : "memory");  // (before any wait that could fail: all 128 get here)
        }
        for (int tile = blockIdx.x; tile < total_tiles && ok; tile += gridDim.x) {
            int b, y0, x0;
            tile_origin(tile, b, y0, x0);
            __syncwarp();
            for (int e = lane; e < ((p.stage_rows + 15) >> 4) * 4; e += 32) {
                const int px = (e >> 2) * 16 + warp * 4 + (e & 3);
                if (px >= p.stage_rows) continue;
                int iy, ix;
                if (p.stride == 1) {
                    const int hy = px / p.pitch, hx = px - hy * p.pitch;
                    iy = y0 - p.pad + hy;
                    ix = x0 - p.pad + hx;
                } else {
                    const int plane = px / p.plane_rows, rem = px - plane * p.plane_rows;
                    const int q = rem / p.pitch, qx = rem - q * p.pitch;
                    iy = 2 * (y0 + q - 1) + (plane >> 1);
                    ix = 2 * (x0 + qx - 1) + (plane & 1);
                }
                int32_t src = -1;
                if (iy >= 0 && iy < p.h_in && ix >= 0 && ix < p.w_in) {
                    src = (b * p.h_in + iy) * p.w_in + ix;
                    if (p.rows) src = __ldg(p.cell_row + src);  // the pixel's channels are a pillar row, or the cell is empty
                }
                s_src[px] = src;
            }
            __syncwarp();
            if (tid == 0 && tile == blockIdx.x) tl_stamp(p, 2);  // first source table done
            if (sparse) {
                // Gathered input (pillar rows through the index map): ~95 % of the halo is empty cells.  The stages were zeroed
                // once; per tile set a warp lists its occupied pixel rows, un-writes the ones the PREVIOUS tile set left in
                // this stage and copies only the occupied ones -- a handful of cp.async per lane instead of one per pixel.
                uint16_t *const cur = s_occ + (warp * 2 + (n_tiles_done & 1)) * occ_cap;
                const uint16_t *const prev = s_occ + (warp * 2 + ((n_tiles_done & 1) ^ 1)) * occ_cap;
                int n_cur = 0;
                for (int e0 = 0; e0 < ((p.stage_rows + 15) >> 4) * 4; e0 += 32) {
                    const int e = e0 + lane;
                    const int px = (e >> 2) * 16 + warp * 4 + (e & 3);
                    const bool occ = px < p.stage_rows && s_src[px] >= 0;
                    const unsigned m = __ballot_sync(0xffffffffu, occ);
                    if (occ) cur[n_cur + __popc(m & ((1u << lane) - 1u))] = static_cast<uint16_t>(px);
                    n_cur += __popc(m);
                }
                __syncwarp();
                for (int cb = 0; cb < cbn; ++cb, ++ia) {
                    const int sa = ia % SA;
                    if (ia >= SA && !mbar_wait(a_empty + 8u * sa, ((ia / SA) - 1) & 1u, s_abort)) {
                        ok = false;
                        break;
                    }
                    const uint32_t stage = a0 + sa * a_bytes;
                    // (with one stage the second channel block of a tile set finds its own pixels there: nothing to undo)
                    for (int e = lane; e < ((SA == 1 && cb > 0) ? 0 : n_prev * 8); e += 32) {
                        const int px = prev[e >> 3], c8 = e & 7;
                        if (s_src[px] < 0)  // (a pixel occupied again is overwritten whole by the copy below)
                            asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(stage + px * 128u + ((c8 ^ (px & 7)) << 4)), "r"(0) : "memory");
                    }
                    for (int e = lane; e < n_cur * 8; e += 32) {
                        const int px = cur[e >> 3], c8 = e & 7;
                        cp_async16_zfill(stage + px * 128u + ((c8 ^ (px & 7)) << 4),
                                         p.rows + static_cast<size_t>(s_src[px]) * p.c_in + cb * 32 + c8 * 4, true);
                    }
                    asm volatile("cp.async.commit_group;" ::: "memory");
                    asm volatile("cp.async.wait_group 0;" ::: "memory");
                    fence_async_smem();
                    mbar_arrive(a_full + 8u * sa);
                }
                n_prev = n_cur;
                ++n_tiles_done;
                continue;
            }
            for (int cb = 0; cb < cbn; ++cb, ++ia) {
                const int sa = ia % SA;
                if (ia >= SA && !mbar_wait(a_empty + 8u * sa, ((ia / SA) - 1) & 1u, s_abort)) {
                    ok = false;
                    break;
                }
                const uint32_t stage = a0 + sa * a_bytes + dst0;
                const float *const src_cb = base + cb * 32;
#pragma unroll 4
                for (int px = tid >> 3; px < p.stage_rows; px += kLoaders / 8) {
                    const int32_t src = s_src[px];
                    cp_async16_zfill(stage + static_cast<uint32_t>(px - (tid >> 3)) * 128u,
                                     src_cb + static_cast<size_t>(src < 0 ? 0 : src) * p.c_in, src >= 0);
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                fence_async_smem();  // this thread's writes are in shared memory: make them visible to the tensor core's proxy
                mbar_arrive(a_full + 8u * sa);
                if (tid == 0 && ia < 8) tl_stamp(p, 8 + ia);  // halo stage landed
            }
        }
    } else if (warp == 4 || warp == 5) {
        // ================================ MMA issue ==============================================================================
        // One thread issues; with MW == 2 a second warp's thread issues the other half of the patches (64-column MMAs last
        // ~34 cycles, about what one thread needs to issue one: the stage barriers then count two commits).
        const int mw = warp - 4;
        if (mw < MW) {  // the whole warp walks the loop (waits included); one elected lane issues
            const bool leader = elect_one();
            const uint32_t idesc = umma_idesc_tf32(N);
            const uint32_t sbo = static_cast<uint32_t>(p.pitch) * 128u;
            const uint32_t tile_step = static_cast<uint32_t>(kPatchH * p.pitch) * 128u;
            bool ok = true;
            int ia = 0, ib = 0, it = 0;
            for (int tile = blockIdx.x; tile < total_tiles && ok; tile += gridDim.x, ++it) {
                const int buf = it % NB;
                if (it >= NB) ok = mbar_wait(acc_empty + 8u * buf, ((it / NB) - 1) & 1u, s_abort);  // drained by the epilogue
                if (!ok) break;
                tc_fence_after();
                const uint32_t acc = tmem + static_cast<uint32_t>(buf) * acc_cols;
                uint32_t accumulate = 0;
                for (int cb = 0; cb < cbn && ok; ++cb, ++ia) {
                    const int sa = ia % SA;
                    ok = mbar_wait(a_full + 8u * sa, (ia / SA) & 1u, s_abort);
                    if (ia < 8 && mw == 0 && lane == 0) tl_stamp(p, 16 + ia);  // MMA warp: halo stage available
                    const uint32_t stage = a0 + sa * a_bytes;
                    for (int tap = 0; tap < p.taps && ok; ++tap, ++ib) {
                        const int sb = ib % SB;
                        ok = mbar_wait(b_full + 8u * sb, (ib / SB) & 1u, s_abort);
                        if (!ok) break;
                        tc_fence_after();
                        const uint64_t ad = umma_desc(stage + static_cast<uint32_t>(p.tap_off[tap]) * 128u, sbo);
                        const uint64_t bd = umma_desc(b0 + sb * b_bytes, 1024u);
                        if (leader) {
#pragma unroll
                            for (int t = 0; t < T; ++t) {
                                if (MW == 2 && (t & 1) != mw) continue;
#pragma unroll
                                for (int k = 0; k < 4; ++k)  // (+2 in the address field = +32 bytes = the next 8 channels)
                                    umma_tf32(acc + static_cast<uint32_t>(t * N), ad + ((t * tile_step + k * 32u) >> 4), bd + 2u * k, idesc,
                                              k == 0 ? accumulate : 1u);
                            }
                            umma_commit(b_empty + 8u * sb);
                        }
                        accumulate = 1u;
                        __syncwarp();
                    }
                    if (leader) umma_commit(a_empty + 8u * sa);
                }
                if (leader) umma_commit(acc_full + 8u * buf);
                if (it == 0 && mw == 0 && lane == 0) tl_stamp(p, 4);  // last MMA of the first tile set issued
            }
        }
    } else if (warp == 6) {
        // ================================ weight copies ==========================================================================
        if (lane == 0) {
            const uint8_t *src = p.wimg + static_cast<size_t>(phase) * cbn * p.taps * b_bytes;
            const int per_tile = cbn * p.taps;
            int ib = 0;
            bool ok = true;
            for (int tile = blockIdx.x; tile < total_tiles && ok; tile += gridDim.x) {
                for (int i = 0; i < per_tile; ++i, ++ib) {
                    const int sb = ib % SB;
                    if (ib >= SB && !mbar_wait(b_empty + 8u * sb, ((ib / SB) - 1) & 1u, s_abort)) {
                        ok = false;
                        break;
                    }
                    mbar_expect_tx(b_full + 8u * sb, b_bytes);
                    bulk_g2s(b0 + sb * b_bytes, src + static_cast<size_t>(i) * b_bytes, b_bytes, b_full + 8u * sb);
                }
            }
        }
    } else {
        // ================================ epilogue (warps 7-10) ==================================================================
        const int q = warp & 3;                    // TMEM lane quarter this warp may read
        const int r = 4 * q + (lane >> 3), c = lane & 7;  // accumulator lane = MMA row = patch pixel (r, c)
        // transposed convolutions: the accumulator holds TWO horizontally adjacent output phases side by side (columns
        // [0, cw) and [cw, 2 cw)), so a thread stores pairs of neighbouring pixels: full sectors, not every other float
        const int cw = p.pair ? N / 2 : N;
        const int half = p.out_mul >> 1;  // phase = dy * half + g;  output column = ox * up + 2 g + {0, 1}
        uint8_t *const stg = s_stage + q * 4096;
        int it = 0;
        pdl_wait();  // the output buffer may be memory an earlier layer is still reading
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
            const int buf = it % NB;
            if (!mbar_wait(acc_full + 8u * buf, (it / NB) & 1u, s_abort)) break;
            tc_fence_after();
            if (it == 0 && tid == 224) tl_stamp(p, 3);  // first accumulators complete
            int b, y0, x0;
            tile_origin(tile, b, y0, x0);
            const uint32_t lane_base = tmem + (static_cast<uint32_t>(32 * q) << 16) + static_cast<uint32_t>(buf) * acc_cols;
            if (!p.out_nchw && !p.pair) {
                // ---- the common case (NHWC between layers): chunks of 32 columns, the next chunk's tensor-memory load in flight
                // while this one is shifted, clamped, rounded, transposed through shared memory (a thread owns one pixel, eight
                // lanes then write one pixel's full 128-byte line) and stored; all addresses are increments of one base
                constexpr int kChunks = T * (N / 32);  // even (N >= 64)
                const int pl = lane >> 3, ch4 = (lane & 7) * 4;
                const size_t row_stride = static_cast<size_t>(p.out_w) * p.out_c_total;
                const bool col_ok0 = x0 + pl < p.w_out, col_ok1 = x0 + pl + 4 < p.w_out;
                uint32_t va[32], vb[32];
                const auto chunk = [&](uint32_t (&vr)[32], int ci) {
                    const int t = ci / (N / 32), n0 = (ci - t * (N / 32)) * 32;
                    float f[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        float x = __uint_as_float(vr[j]) + s_shift[n0 + j];
                        if (!RES) {  // (with a residual: after the addition, below)
                            if (p.relu) x = fmaxf(x, 0.f);
                            if (p.round_out) x = round_tf32(x);
                        }
                        f[j] = x;
                    }
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<float4 *>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) =
                            make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
                    __syncwarp();
                    const int oyb = y0 + kPatchH * t + 4 * q;
                    float *dst = p.out + (static_cast<size_t>(b) * p.out_h + oyb) * row_stride +
                                 static_cast<size_t>(x0 + pl) * p.out_c_total + p.out_c_off + n0 + ch4;
                    // residual: the same eight 128-byte pixel lines the stores write, read the same way (eight lanes per
                    // line), all eight loads in flight together
                    float4 rv[RES ? 8 : 1];
                    if (RES) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            rv[RES ? i : 0] = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (oyb + (i >> 1) < p.h_out && ((i & 1) ? col_ok1 : col_ok0))
                                rv[RES ? i : 0] = __ldcs(reinterpret_cast<const float4 *>(
                                    p.res + (dst - p.out) + (i >> 1) * row_stride + (i & 1) * 4 * p.out_c_total));
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) {  // pixel 4 i + pl of the warp's 32 = patch row 4 q + i / 2, column pl + 4 (i & 1)
                        const int rr = 4 * i + pl;
                        float4 val = *reinterpret_cast<const float4 *>(stg + rr * 128 + (((lane & 7) ^ (rr & 7)) << 4));
                        if (RES) {
                            float *const e = reinterpret_cast<float *>(&val);
                            const float *const r = reinterpret_cast<const float *>(&rv[RES ? i : 0]);
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                float x = e[u] + r[u];
                                if (p.relu) x = fmaxf(x, 0.f);
                                if (p.round_out) x = round_tf32(x);
                                e[u] = x;
                            }
                        }
                        if (oyb + (i >> 1) < p.h_out && ((i & 1) ? col_ok1 : col_ok0))
                            *reinterpret_cast<float4 *>(dst + (i >> 1) * row_stride + (i & 1) * 4 * p.out_c_total) = val;
                    }
                };
                if (RES) {  // (no next-chunk load in flight: its 32 registers hold the residual lines instead)
#pragma unroll 1
                    for (int ci = 0; ci < kChunks; ++ci) {
                        tmem_ld32_issue(lane_base + static_cast<uint32_t>(ci * 32), va);
                        tmem_ld_wait(va);
                        chunk(va, ci);
                    }
                } else {
                    tmem_ld32_issue(lane_base, va);
#pragma unroll 1
                    for (int ci = 0; ci < kChunks; ci += 2) {
                        tmem_ld_wait(va);
                        tmem_ld32_issue(lane_base + static_cast<uint32_t>((ci + 1) * 32), vb);
                        chunk(va, ci);
                        tmem_ld_wait(vb);
                        if (ci + 2 < kChunks) tmem_ld32_issue(lane_base + static_cast<uint32_t>((ci + 2) * 32), va);
                        chunk(vb, ci + 1);
                    }
                }
                tc_fence_before();
                mbar_arrive(acc_empty + 8u * buf);
                if (it == 0 && tid == 224) tl_stamp(p, 5);  // first epilogue done
                continue;
            }
#pragma unroll 1
            for (int t = 0; t < T; ++t) {
                const int oy = y0 + kPatchH * t + r, ox = x0 + c;
                const bool live = oy < p.h_out && ox < p.w_out;
                const int py = p.pair ? oy * p.out_mul + phase / half : oy;
                const int pxo = p.pair ? ox * p.out_mul + 2 * (phase % half) : ox;
#pragma unroll 1
                for (int n0 = 0; n0 < cw; n0 += 32) {
                    float v[32], u[32];
                    tmem_ld32(lane_base + static_cast<uint32_t>(t * N + n0), v);
                    if (p.pair) tmem_ld32(lane_base + static_cast<uint32_t>(t * N + cw + n0), u);
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float sh = s_shift[n0 + j];
                        float x = v[j] + sh, y = u[j] + sh;
                        if (p.relu) { x = fmaxf(x, 0.f); y = fmaxf(y, 0.f); }
                        if (p.round_out) { x = round_tf32(x); y = round_tf32(y); }
                        v[j] = x;
                        u[j] = y;
                    }
                    if (p.out_nchw) {
                        if (!live) continue;
                        float *dst = p.out + ((static_cast<size_t>(b) * p.out_c_total + p.out_c_off + n0) * p.out_h + py) * p.out_w + pxo;
                        const size_t cs = static_cast<size_t>(p.out_h) * p.out_w;
                        if (p.pair) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) *reinterpret_cast<float2 *>(dst + j * cs) = make_float2(v[j], u[j]);
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j) dst[j * cs] = v[j];
                        }
                    } else if (p.pair) {
                        if (!live) continue;
                        float4 *dst = reinterpret_cast<float4 *>(
                            p.out + ((static_cast<size_t>(b) * p.out_h + py) * p.out_w + pxo) * p.out_c_total + p.out_c_off + n0);
#pragma unroll
                        for (int j = 0; j < 8; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                        dst += p.out_c_total >> 2;
#pragma unroll
                        for (int j = 0; j < 8; ++j) dst[j] = make_float4(u[4 * j], u[4 * j + 1], u[4 * j + 2], u[4 * j + 3]);
                    } else {
                        // NHWC: a thread owns one pixel, so its 128 bytes of this chunk are contiguous but the warp's 32 pixels
                        // are not: the 32 x 32 tile goes through shared memory so that eight lanes write one pixel's full
                        // 128-byte line.
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            *reinterpret_cast<float4 *>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) =
                                make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                        __syncwarp();
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int rr = 4 * i + (lane >> 3);  // pixel of the warp's 32 (= 4 patch rows x 8 columns)
                            const int oy2 = y0 + kPatchH * t + 4 * q + (rr >> 3), ox2 = x0 + (rr & 7);
                            const float4 val = *reinterpret_cast<const float4 *>(stg + rr * 128 + (((lane & 7) ^ (rr & 7)) << 4));
                            if (oy2 < p.h_out && ox2 < p.w_out)
                                *reinterpret_cast<float4 *>(p.out + ((static_cast<size_t>(b) * p.out_h + oy2) * p.out_w + ox2) * p.out_c_total +
                                                            p.out_c_off + n0 + (lane & 7) * 4) = val;
                        }
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(acc_empty + 8u * buf);  // this thread has read its part of the accumulator
            if (it == 0 && tid == 224) tl_stamp(p, 5);  // first epilogue done
        }
    }
    if (*s_abort && tid == 0 && p.error) {
        pdl_wait();
        atomicExch(p.error, 0xC0DE0000u | static_cast<uint32_t>(blockIdx.x & 0xFFFF));
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(tmem_cols) : "memory");
}

// Shared-memory image of the weights: [phase][c_in / 32][tap][n][128 B], chunk c of row n at (c ^ (n & 7)) * 16 -- exactly what
// one bulk copy per (channel block, tap) must put behind the B descriptor.  BN scale folded in, rounded to nearest tf32.
//   conv:            weight [c_out, c_in, k, k]   (nn.Conv2d)
//   transposed (up): weight [c_in, c_out, up, up] (nn.ConvTranspose2d with kernel = stride = up): phase = (dy, dx)
__global__ void k_conv_wimg(const float *__restrict__ weight, const float *__restrict__ scale, int c_in, int c_out, int k, int up,
                            float *__restrict__ img)
{
    const int taps = up > 1 ? 1 : k * k, phases = up > 1 ? up * up / 2 : 1, cbn = c_in >> 5;
    const int rows = up > 1 ? 2 * c_out : c_out;  // transposed: the dx pair (2 g, 2 g + 1) side by side
    const int64_t total = static_cast<int64_t>(phases) * cbn * taps * rows * 8;
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = static_cast<int>(i & 7);
    int64_t r = i >> 3;
    const int row = static_cast<int>(r % rows); r /= rows;
    const int tap = static_cast<int>(r % taps); r /= taps;
    const int cb = static_cast<int>(r % cbn);
    const int phase = static_cast<int>(r / cbn);
    const int n = row % c_out;
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int ci = cb * 32 + c * 4 + e;
        float w;
        if (up > 1) {
            const int half = up / 2, dy = phase / half, dx = 2 * (phase % half) + row / c_out;
            w = weight[((static_cast<int64_t>(ci) * c_out + n) * up + dy) * up + dx];
        } else {
            w = weight[(static_cast<int64_t>(n) * c_in + ci) * taps + tap];
        }
        v[e] = round_tf32(scale ? w * scale[n] : w);
    }
    const int64_t block = (static_cast<int64_t>(phase) * cbn + cb) * taps + tap;
    float *dst = img + block * rows * 32 + static_cast<int64_t>(row) * 32 + ((c ^ (row & 7)) << 2);
    *reinterpret_cast<float4 *>(dst) = make_float4(v[0], v[1], v[2], v[3]);
}

template <int N, int T, int SA, int SB, int NB, int MW, int MB = 1, bool RES = false>
cudaError_t launch_one(const ConvParams &p, int phases, cudaStream_t st)
{
    const size_t a_bytes = (static_cast<size_t>(p.stage_rows) * 128 + 1023) & ~static_cast<size_t>(1023);
    const size_t occ_cap = ((static_cast<size_t>(p.stage_rows) + 15) / 16) * 4 + 8;
    const size_t smem = SA * a_bytes + static_cast<size_t>(SB) * N * 128 + 4 * 4096 + 1024 +
                        4 * ((static_cast<size_t>(p.stage_rows) + 15) & ~static_cast<size_t>(15)) + (p.rows ? 16 * occ_cap : 0) + 64;
    if (smem > 225 * 1024) return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(k_conv_umma<N, T, SA, SB, NB, MW, MB, RES>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    const int tiles = p.nb * p.tiles_x * p.tiles_y;
    const int ctas = current_sm_count() * MB;
    const dim3 grid(static_cast<unsigned>(tiles < ctas ? tiles : ctas), 1, static_cast<unsigned>(phases));
    e = launch_pdl(k_conv_umma<N, T, SA, SB, NB, MW, MB, RES>, grid, dim3(kConvThreads), smem, st, p);
    note_launch();
    return e != cudaSuccess ? e : cudaGetLastError();
}

}  // namespace

cudaError_t launch_conv_wimg(const float *weight, const float *scale, int c_in, int c_out, int k, int up, float *img, cudaStream_t st)
{
    const int taps = up > 1 ? 1 : k * k;
    const int64_t total = static_cast<int64_t>(up) * up * (c_in >> 5) * taps * c_out * 8;  // (= phases * rows, either way)
    k_conv_wimg<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(weight, scale, c_in, c_out, k, up, img);
    note_launch();
    return cudaGetLastError();
}

// Geometry of one layer -> kernel parameters.  Returns cudaErrorInvalidValue for shapes outside the instantiated set.
cudaError_t launch_conv_umma(const ConvJob &j, cudaStream_t st)
{
    ConvParams p{};
    p.in = j.in;
    p.rows = j.rows;
    p.cell_row = j.cell_row;
    p.wimg = static_cast<const uint8_t *>(j.wimg);
    p.shift = j.shift;
    p.out = j.out;
    p.nb = j.nb;
    p.h_in = j.h_in;
    p.w_in = j.w_in;
    p.c_in = j.c_in;
    p.stride = j.stride;
    p.pad = j.pad;
    p.taps = j.k * j.k;
    p.relu = j.relu;
    p.round_out = j.round_out;
    p.error = j.error;
    p.timeline = debug_times_ptr();
    p.res = j.res;
    p.h_out = (j.h_in + 2 * j.pad - j.k) / j.stride + 1;
    p.w_out = (j.w_in + 2 * j.pad - j.k) / j.stride + 1;
    p.out_mul = j.up;
    p.out_h = p.h_out * j.up;
    p.out_w = p.w_out * j.up;
    p.out_c_total = j.out_c_total;
    p.out_c_off = j.out_c_off;
    p.out_nchw = j.out_nchw;
    const int phases = j.up > 1 ? j.up * j.up / 2 : 1;
    const int n_eff = j.up > 1 ? 2 * j.c_out : j.c_out;
    p.pair = j.up > 1;
    if (j.c_in % 32 != 0 || j.c_in < 32 || (j.stride != 1 && j.stride != 2) || j.k < 1 || j.k > 3 || (j.up != 1 && j.up != 2 && j.up != 4) ||
        (j.up > 1 && (j.k != 1 || j.stride != 1)) || (j.rows && !j.cell_row) || (!j.rows && !j.in) || p.h_out < 1 || p.w_out < 1)
        return cudaErrorInvalidValue;
    if (j.res && (j.up > 1 || j.out_nchw)) return cudaErrorInvalidValue;  // only the plain NHWC epilogue reads a residual
    // (1x1 stride 2: the one tap of the even/even parity plane; the odd planes are loaded and not read)
    if (j.stride == 2 && !((j.k == 3 && j.pad == 1) || (j.k == 2 && j.pad == 0) || (j.k == 1 && j.pad == 0))) return cudaErrorInvalidValue;
    if (j.stride == 1 && j.pad != (j.k - 1) / 2) return cudaErrorInvalidValue;

    // patches per tile set: two accumulator buffers of T * N columns must fit the 512 columns of tensor memory
    int T;
    if (n_eff > 256) return cudaErrorInvalidValue;
    if (j.stride == 1) T = n_eff == 64 ? 4 : n_eff == 128 ? 2 : 1;
    else T = 1;  // (two patches on ONE halo stage measured slower on the gathered first layer: 0.43 vs 0.38 ms)
    while (T > 1 && kPatchH * (T / 2) >= p.h_out) T /= 2;  // small images: do not pad the patch stack past the image
    if (j.stride == 1) {
        p.pitch = kPatchW + j.k - 1;
        p.stage_rows = (kPatchH * T + j.k - 1) * p.pitch;
        for (int ky = 0; ky < j.k; ++ky)
            for (int kx = 0; kx < j.k; ++kx) p.tap_off[ky * j.k + kx] = ky * p.pitch + kx;
    } else {
        p.pitch = kPatchW + 1;
        p.plane_rows = (kPatchH * T + 1) * p.pitch;
        p.stage_rows = 4 * p.plane_rows;
        for (int ky = 0; ky < j.k; ++ky)
            for (int kx = 0; kx < j.k; ++kx) {
                const int dy = ky - j.pad, dx = kx - j.pad;  // -1, 0, 1 (3x3 pad 1) or 0, 1 (2x2 pad 0)
                const int py = dy & 1, px = dx & 1;
                const int qy = (dy < 0 ? -1 : 0) + 1, qx = (dx < 0 ? -1 : 0) + 1;  // floor(d / 2) + 1: planes keep one leading row / column
                p.tap_off[ky * j.k + kx] = (py * 2 + px) * p.plane_rows + qy * p.pitch + qx;
            }
    }
    p.tiles_y = (p.h_out + kPatchH * T - 1) / (kPatchH * T);
    p.tiles_x = (p.w_out + kPatchW - 1) / kPatchW;

#define CONV_CASE(n, t, sa, sb, nb, mw) \
    if (n_eff == n && T == t)              \
    return j.res ? launch_one<n, t, sa, sb, nb, mw, 1, true>(p, phases, st) : launch_one<n, t, sa, sb, nb, mw>(p, phases, st)
    if (j.stride == 1) {
        CONV_CASE(64, 4, 2, 4, 2, 2);
        CONV_CASE(64, 2, 2, 4, 2, 2);
        CONV_CASE(64, 1, 2, 4, 2, 1);
        CONV_CASE(128, 2, 2, 4, 2, 1);
        CONV_CASE(128, 1, 2, 4, 2, 1);
        CONV_CASE(256, 1, 2, 4, 2, 1);
    } else {
        CONV_CASE(64, 1, 2, 4, 2, 1);
        CONV_CASE(128, 1, 2, 3, 2, 1);
        CONV_CASE(256, 1, 1, 3, 2, 1);
    }
#undef CONV_CASE
    return cudaErrorInvalidValue;
}

}  // namespace pillars
