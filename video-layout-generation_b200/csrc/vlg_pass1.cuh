// vlg_pass1.cuh -- pass 1 of the fused op: warp + every per-pixel loss term + d(loss)/d(warped)
// + d(loss)/d(coords) in ONE kernel, one CTA per 32x8 output tile (grid = tiles_x x tiles_y x N).
// It evaluates the un-warped criteria (vlg_pixel_loss_*, rgb and layout) and, for a warped step, the layout
// and TV terms when lay_tile_kernel cannot take them; the rgb terms of a warped step run in rgb_strip_kernel.
//
// Loss definitions followed (reference gongaa/video-layout-generation):
//   L1          src/trainer.py:130,248      mean |a-b| over N*3*H*W, sign(0)=0
//   GD          src/loss.py:20-25           sum||da|-|db|| along H and along W, / (N*C*H*W)
//   SSIM        src/loss.py:68-91           3x3 valid avg-pool stats, C1=1e-4, C2=9e-4,
//                                           clamp((1-SSIM)/2,0,1).mean() summed over channels
//   CE          src/trainer.py:124,250      mean over labels != ignore_index of -log_softmax[label]
//   TV          (absent upstream)           mean|d_H flow| + mean|d_W flow|, stencils of loss.py:22,24
//   composition src/trainer.py:248-251      w_l1*L1 + w_gd*GD + w_ssim*SSIM + w_ce*CE (+ w_tv*TV)
//
// The kernel is issue-bound, not HBM-bound (profiles/): everything below is organised to spend
// few instructions per pixel.  Phases of one CTA (256 threads, tile 32x8, rgb halo 2):
//   0a  base-grid coordinates of the tile's rows/columns -> smem (one IEEE division each)
//   0b  over tile+halo: rgb (given) and target -> smem, or (WARP) the coordinates -> smem and the
//       bounding box of the layout taps of the tile's own pixels (integer smem atomics)
//   1   cp.async the source-layout bounding box into smem row by row (zero-filled outside the
//       image), and meanwhile evaluate the 3x3 SSIM windows (runs of 5 share their column sums,
//       packed fp32x2 math on the (x,y) pairs)
//   2   own pixel: L1 / GD / SSIM-adjoint, layout gather from smem with FFMA2 on channel pairs,
//       softmax-CE with ex2/lg2.approx, coordinate gradient, TV, stores
//   3   block reduction -> one row of partial sums, per-tile displacement maxima
#pragma once
#include <cuda.h>   // CUtensorMap (type only; the encoder is resolved at run time, libcuda is not linked)

#include "vlg_device.cuh"

namespace vlg {

struct Pass1Params {
    CoordCfg cc;
    int N;
    int tiles_x, tiles_y;
    const void *src_rgb, *src_layout;  // WARP: source layout (src_rgb unused).  !WARP: `output` rgb / logits themselves
    const float *coords;
    const void *tgt_rgb;
    const int64_t *label;
    int64_t ignore_index;
    const float *class_weight;   // per-class CE weights (K floats) or NULL
    TermCoeffs tc;
    int need_grad;          // compute gradients at all
    // outputs
    float *d_coords;        // WARP && need_grad
    void *d_out_rgb;        // !WARP: user tensor of type T (nullable)
    void *d_out_lay;
    int64_t *out_argmax;    // nullable
    float *partials;        // [n_blocks][kPartialSlots]
    float *tile_disp;       // [n_blocks] max displacement among the tile's NEAR output pixels (WARP)
    int4 *far_list;         // [P] queue of FAR output pixels: {pixel index, tap cell, fractional weights} (nullable: no source gradient / no far path)
    uint32_t *seg_cnt;      // [n_blocks][kTH] far output pixels per row of a SOURCE tile (zeroed with the header)
    uint32_t *tile_flags;   // [n_blocks] != 0 where a far pixel lands in that SOURCE tile (zeroed with the header)
    int *flagged_list;      // [n_blocks] compacted ids of the flagged source tiles
    ReduceParams red;       // red.out != NULL: the last CTA also performs the final reduction
    WsHeader *hdr;
    int accum_dcoords;      // d_coords already holds the rgb part (written by rgb_strip_kernel): add to it
};

#ifndef VLG_P1_MIN_BLOCKS
#define VLG_P1_MIN_BLOCKS 3   // resident CTAs per SM the register / shared-memory budget targets
#endif
// staged source-layout window (pixels); covers the tile's taps for displacement spreads of a few
// pixels around the tile's mean motion; pixels whose taps fall outside use the global path
#if VLG_P1_MIN_BLOCKS >= 4
constexpr int kSW = 36, kSH = 10;   // 28.8 KB (K=20 fp32): 4 CTAs of <= 56 KB fit one SM
#define VLG_P1_FLOW_IN_SMEM 0
#else
constexpr int kSW = 40, kSH = 12;
#define VLG_P1_FLOW_IN_SMEM 1
#endif
constexpr int kSegW = 5;                               // SSIM windows per run
constexpr int kSegs = (kWW + kSegW - 1) / kSegW;       // 7 runs per window row
static_assert(kSegs * kWH * 3 <= kThreads, "one SSIM run per thread");

template <typename T, int K>
struct Pass1Smem {
    float2 ab[3][kRN];      // (warped-or-given rgb, target rgb) over the tile + halo 2
#if VLG_P1_FLOW_IN_SMEM
    float2 flow[kRN];       // raw coords (TV stencil, tap recomputation)
#endif
    float2 kab[3][kWN];     // per-window SSIM adjoint coefficients (A,B) ...
    float kc[3][kWN];       // ... and C (12 bytes per window: fewer smem wavefronts than a padded float4)
    float bx[kRW], by[kRH]; // base-grid coordinates of the region's columns / rows
    float red[kThreads / 32][kPartialSlots];
    float redmax[kThreads / 32][4];
    int bbox[4];            // min x0, min y0, max x0, max y0 of the tile's own taps
    alignas(128) T stage[kSH * kSW * K];   // staged source-layout window
};
static_assert(sizeof(float2) * 3 * kRN + sizeof(float) * 9 * kWN >= 6 * 256 * sizeof(double),
              "ab (+flow) + k must hold the final-reduction scratch");

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async4(void *smem, const void *gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
}

// ---- TMA (cp.async.bulk.tensor) + mbarrier: one instruction per CTA stages the whole layout window,
// out-of-image elements are zero-filled by the hardware (exactly the padding the gather wants)
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // init visible to the async (TMA) proxy
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
    const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"   // suspend-time hint: the warp sleeps in hardware
        "@p bra WAIT_DONE;\n"                                             // instead of burning issue slots on a spin loop
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(a), "r"(parity), "r"(0x989680u)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void *smem_dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n" ::"r"(
            (unsigned)__cvta_generic_to_shared(smem_dst)),
        "l"(map), "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

__device__ __forceinline__ void tma_load_3d(void *smem_dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n" ::"r"(
            (unsigned)__cvta_generic_to_shared(smem_dst)),
        "l"(map), "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

// prefetch of a tensor-map descriptor (hides its fetch behind the barrier set-up)
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *map) {
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(map) : "memory");
}

// bulk shared -> global store (one instruction per contiguous run) and its bookkeeping
__device__ __forceinline__ void bulk_store(void *gdst, const void *ssrc, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(gdst),
                 "r"((unsigned)__cvta_generic_to_shared(ssrc)), "r"(bytes)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
__device__ __forceinline__ void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// sampling coordinates from raw coords + the smem base-grid table
__device__ __forceinline__ float2 source_xy(const CoordCfg &cc, float2 c, float bx, float by, float &mx, float &my) {
    float gx = c.x, gy = c.y;
    if (cc.coord_mode == VLG_COORD_FLOW) {
        gx = __fadd_rn(bx, __fmul_rn(c.x, cc.sx));
        gy = __fadd_rn(by, __fmul_rn(c.y, cc.sy));
    }
    float ux = __fmul_rn(__fmul_rn(__fadd_rn(gx, 1.0f), 0.5f), cc.Wm1);
    float uy = __fmul_rn(__fmul_rn(__fadd_rn(gy, 1.0f), 0.5f), cc.Hm1);
    mx = __fmul_rn(cc.Wm1, 0.5f);
    my = __fmul_rn(cc.Hm1, 0.5f);
    if (cc.padding == VLG_PAD_BORDER) {
        if (ux <= 0.0f || ux >= cc.Wm1) mx = 0.0f;
        if (uy <= 0.0f || uy >= cc.Hm1) my = 0.0f;
        ux = fminf(cc.Wm1, fmaxf(ux, 0.0f));
        uy = fminf(cc.Hm1, fmaxf(uy, 0.0f));
    }
    if (cc.coord_mode == VLG_COORD_FLOW) {
        mx *= cc.sx;
        my *= cc.sy;
    }
    return make_float2(ux, uy);
}

__device__ __forceinline__ Taps taps_from_xy(const CoordCfg &cc, float2 xy, float mx, float my) {
    Taps t;
    t.ix = xy.x; t.iy = xy.y; t.mx = mx; t.my = my;
    t.fx0 = floorf(xy.x);
    t.fy0 = floorf(xy.y);
    const float fx1 = __fadd_rn(t.fx0, 1.0f), fy1 = __fadd_rn(t.fy0, 1.0f);
    const float wx1 = __fsub_rn(xy.x, t.fx0), wx0 = __fsub_rn(fx1, xy.x);
    const float wy1 = __fsub_rn(xy.y, t.fy0), wy0 = __fsub_rn(fy1, xy.y);
    t.nw = __fmul_rn(wx0, wy0);
    t.ne = __fmul_rn(wx1, wy0);
    t.sw = __fmul_rn(wx0, wy1);
    t.se = __fmul_rn(wx1, wy1);
    t.x0 = (int)fminf(fmaxf(t.fx0, -4.0f), (float)cc.W + 4.0f);
    t.y0 = (int)fminf(fmaxf(t.fy0, -4.0f), (float)cc.H + 4.0f);
    return t;
}

// +-c with the sign of (u*v), 0 if either is 0  (c >= 0)
__device__ __forceinline__ float signed_c(float c, float u, float v) {
    const unsigned s = (__float_as_uint(u) ^ __float_as_uint(v)) & 0x80000000u;
    return (u == 0.0f || v == 0.0f) ? 0.0f : __uint_as_float(__float_as_uint(c) | s);
}
// +-c with the sign of u, 0 if u is 0
__device__ __forceinline__ float signed_c1(float c, float u) {
    return u == 0.0f ? 0.0f : __uint_as_float(__float_as_uint(c) | (__float_as_uint(u) & 0x80000000u));
}

// one channel of one tap read straight from global memory (zero outside the image)
template <typename T>
__device__ __forceinline__ float tap_global(const T *img, int C, int c, int y, int x, int H, int W) {
    return (y >= 0 && y < H && x >= 0 && x < W) ? to_f<T>(__ldg(img + ((int64_t)y * W + x) * C + c)) : 0.0f;
}

template <typename T, int K, bool WARP>
__global__ void __launch_bounds__(kThreads, VLG_P1_MIN_BLOCKS) pass1_kernel(const Pass1Params p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Pass1Smem<T, K> &sm = *reinterpret_cast<Pass1Smem<T, K> *>(smem_raw);
    const CoordCfg &cc = p.cc;
    const int H = cc.H, W = cc.W;
    const int tid = threadIdx.x;
    const int lane = tid & 31, wid = tid >> 5;
    const int n = blockIdx.z;
    const int bt = (n * p.tiles_y + blockIdx.y) * p.tiles_x + blockIdx.x;
    const int ty0 = blockIdx.y * kTH, tx0 = blockIdx.x * kTW;
    const int64_t img_px = (int64_t)n * H * W;

    // a warped step evaluates its rgb terms in rgb_strip_kernel
    const bool has_rgb = !WARP && p.src_rgb != nullptr && p.tgt_rgb != nullptr;
    const bool has_lay = p.src_layout != nullptr && p.label != nullptr;
    const T *src_rgb = has_rgb ? reinterpret_cast<const T *>(p.src_rgb) + img_px * 3 : nullptr;
    const T *tgt_rgb = has_rgb ? reinterpret_cast<const T *>(p.tgt_rgb) + img_px * 3 : nullptr;
    const T *src_lay = has_lay ? reinterpret_cast<const T *>(p.src_layout) + img_px * K : nullptr;
    const float2 *coords = WARP ? reinterpret_cast<const float2 *>(p.coords) + img_px : nullptr;

    float s_l1 = 0.f, s_gd = 0.f, s_ssim = 0.f, s_ce = 0.f, s_tvh = 0.f, s_tvw = 0.f;
    float m_disp = 0.f, m_near = 0.f, m_grad = 0.f;

    // Loads whose consumers sit in phase 2 are issued now, so that their (L2/DRAM) latency is
    // hidden behind phases 0-1 instead of stalling the longest phase.
    int64_t lab_pre = 0;
    float denom_pre = 1.0f, wl_pre = 1.0f;
    float2 dc_pre = make_float2(0.f, 0.f);
    {
        const int py = ty0 + tid / kTW, px = tx0 + (tid & (kTW - 1));
        if (WARP && p.accum_dcoords && p.need_grad && p.d_coords && py < H && px < W)
            dc_pre = __ldcg(reinterpret_cast<const float2 *>(p.d_coords) + img_px + (int64_t)py * W + px);
        if (has_lay && py < H && px < W) {
            lab_pre = __ldg(p.label + img_px + (int64_t)py * W + px);
            if (p.class_weight && lab_pre >= 0 && lab_pre < K) wl_pre = __ldg(p.class_weight + lab_pre);
        }
        if (has_lay && p.need_grad)
            denom_pre = ce_divisor(p.tc, p.hdr);
    }

    // ---------------- phase 0a: base grid of the region's rows / columns ----------------
    if (WARP) {
        if (tid < kRW) sm.bx[tid] = base_coord(tx0 - kHalo + tid, cc.Wm1);
        else if (tid >= 64 && tid < 64 + kRH) sm.by[tid - 64] = base_coord(ty0 - kHalo + tid - 64, cc.Hm1);
        if (tid == 128) { sm.bbox[0] = 1 << 30; sm.bbox[1] = 1 << 30; sm.bbox[2] = -(1 << 30); sm.bbox[3] = -(1 << 30); }
        // (the barrier that publishes the table sits in phase 0b, after the coords loads were issued)
    }

    // ---------------- phase 0b: coordinates + rgb over the tile + halo ----------------
    {
        int bx0 = 1 << 30, by0 = 1 << 30, bx1 = -(1 << 30), by1 = -(1 << 30);
        if (WARP) __syncthreads();   // base-grid table ready
#pragma unroll
        for (int it = 0; it < (kRN + kThreads - 1) / kThreads; ++it) {
            const int q = tid + it * kThreads;
            if (q < kRN) {
                const int ry = q / kRW, rx = q - ry * kRW;
                const int y = ty0 - kHalo + ry, x = tx0 - kHalo + rx;
                float a[3] = {0.f, 0.f, 0.f}, b[3] = {0.f, 0.f, 0.f};
                float2 fl = make_float2(0.f, 0.f);
                if (y >= 0 && y < H && x >= 0 && x < W) {
                    const int64_t o = (int64_t)y * W + x;
                    if (WARP) {
                        float mx, my;
                        fl = __ldg(coords + o);
                        const float2 xy = source_xy(cc, fl, sm.bx[rx], sm.by[ry], mx, my);
                        const bool own = ry >= kHalo && ry < kHalo + kTH && rx >= kHalo && rx < kHalo + kTW;
                        if (own && has_lay) {
                            const int x0 = (int)fminf(fmaxf(floorf(xy.x), -4.0f), (float)W + 4.0f);
                            const int y0 = (int)fminf(fmaxf(floorf(xy.y), -4.0f), (float)H + 4.0f);
                            bx0 = min(bx0, x0); bx1 = max(bx1, x0);
                            by0 = min(by0, y0); by1 = max(by1, y0);
                        }
                    } else if (has_rgb) {
                        load_px<T, 3>(src_rgb + o * 3, a);
                    }
                    if (has_rgb) load_px<T, 3>(tgt_rgb + o * 3, b);
                }
                if (has_rgb) {
#pragma unroll
                    for (int c = 0; c < 3; ++c) sm.ab[c][q] = make_float2(a[c], b[c]);
                }
#if VLG_P1_FLOW_IN_SMEM
                if (WARP) sm.flow[q] = fl;
#endif
            }
        }
        if (WARP && has_lay) {
            bx0 = __reduce_min_sync(0xffffffffu, bx0); by0 = __reduce_min_sync(0xffffffffu, by0);
            bx1 = __reduce_max_sync(0xffffffffu, bx1); by1 = __reduce_max_sync(0xffffffffu, by1);
            if (lane == 0) {
                atomicMin(&sm.bbox[0], bx0); atomicMin(&sm.bbox[1], by0);
                atomicMax(&sm.bbox[2], bx1); atomicMax(&sm.bbox[3], by1);
            }
        }
        __syncthreads();
    }

    // ---------------- phase 1a: stage the source-layout window (async, one warp per row) --------
    // window origin = min tap; extent clipped to the stage capacity.  Cells outside the image are
    // zero-filled, so in-window taps need no bounds predicate (torch skips out-of-image taps).
    int ox = 0, oy = 0, sw = 0, sh = 0;
    if (WARP && has_lay) {
        ox = sm.bbox[0]; oy = sm.bbox[1];
        sw = min(kSW, sm.bbox[2] + 2 - ox);
        sh = min(kSH, sm.bbox[3] + 2 - oy);
        constexpr int PXB = K * (int)sizeof(T);
        constexpr int VB = vec_bytes(PXB);
        if (sw > 0 && sh > 0) {
            const int xa = min(max(0, ox), ox + sw), xb = max(min(ox + sw, W), xa);   // in-image columns [xa, xb)
            for (int ry = wid; ry < sh; ry += kThreads / 32) {
                const int y = oy + ry;
                char *drow = reinterpret_cast<char *>(sm.stage) + (size_t)ry * kSW * PXB;
                T *zrow = reinterpret_cast<T *>(drow);
                const T zero = from_f<T>(0.0f);
                if (y < 0 || y >= H) {
                    for (int i = lane; i < sw * K; i += 32) zrow[i] = zero;
                    continue;
                }
                for (int i = lane; i < (xa - ox) * K; i += 32) zrow[i] = zero;
                for (int i = lane; i < (ox + sw - xb) * K; i += 32) zrow[(size_t)(xb - ox) * K + i] = zero;
                const char *srow = reinterpret_cast<const char *>(src_lay) + ((int64_t)y * W + xa) * PXB;
                char *d = drow + (size_t)(xa - ox) * PXB;
                const int nbytes = (xb - xa) * PXB;
                if constexpr (VB == 16) {
                    for (int i = lane * 16; i < nbytes; i += 32 * 16) cp_async16(d + i, srow + i);
                } else {
                    const T *sp = reinterpret_cast<const T *>(srow);
                    T *dp = reinterpret_cast<T *>(d);
                    for (int i = lane; i < (xb - xa) * K; i += 32) dp[i] = __ldg(sp + i);
                }
            }
        }
    }

    // ---------------- phase 1b: SSIM windows, runs of kSegW along x ----------------
    if (has_rgb && (p.tc.terms & VLG_TERM_SSIM)) {
        if (tid < kSegs * kWH * 3) {
            const int c = tid / (kSegs * kWH);
            const int r2 = tid - c * (kSegs * kWH);
            const int wy = r2 / kSegs, seg = r2 - wy * kSegs;
            const int wx0 = seg * kSegW;
            const int nwin = min(kSegW, kWW - wx0);
            // column sums over the 3 rows: (sum x, sum y), (sum x^2, sum y^2), sum xy
            float2 cs[kSegW + 2], cq[kSegW + 2];
            float cxy[kSegW + 2];
            const float2 *row0 = &sm.ab[c][wy * kRW + wx0];
#pragma unroll
            for (int j = 0; j < kSegW + 2; ++j) {
                if (j < nwin + 2) {
                    const float2 v0 = row0[j], v1 = row0[kRW + j], v2 = row0[2 * kRW + j];
                    cs[j] = __fadd2_rn(__fadd2_rn(v0, v1), v2);
                    cq[j] = __ffma2_rn(v2, v2, __ffma2_rn(v1, v1, __fmul2_rn(v0, v0)));
                    cxy[j] = fmaf(v2.x, v2.y, fmaf(v1.x, v1.y, v0.x * v0.y));
                } else {
                    cs[j] = cq[j] = make_float2(0.f, 0.f);
                    cxy[j] = 0.f;
                }
            }
            const int i = ty0 - kHalo + wy;
            const bool row_ok = i >= 0 && i + 2 < H;
            const float inv9 = 1.0f / 9.0f, C1 = 1e-4f, C2 = 9e-4f;
            const float2 inv9_2 = make_float2(inv9, inv9);
            const float kk = -p.tc.c_ssim * (2.0f / 9.0f);
#pragma unroll
            for (int w = 0; w < kSegW; ++w) {
                if (w < nwin) {
                    const int wx = wx0 + w;
                    const int j = tx0 - kHalo + wx;
                    float4 kk4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (row_ok && j >= 0 && j + 2 < W) {
                        const float2 m2 = __fmul2_rn(__fadd2_rn(__fadd2_rn(cs[w], cs[w + 1]), cs[w + 2]), inv9_2);   // (mx, my)
                        const float2 mm = __fmul2_rn(m2, m2);
                        const float2 q2 = __fadd2_rn(__fadd2_rn(cq[w], cq[w + 1]), cq[w + 2]);
                        const float2 var = __ffma2_rn(q2, inv9_2, make_float2(-mm.x, -mm.y));                        // (vx, vy)
                        const float mxy = m2.x * m2.y;
                        const float vxy = fmaf(cxy[w] + cxy[w + 1] + cxy[w + 2], inv9, -mxy);
                        const float n1 = fmaf(2.f, mxy, C1), n2 = fmaf(2.f, vxy, C2);
                        const float d1 = mm.x + mm.y + C1, d2 = var.x + var.y + C2;
                        const float inv_d1 = rcp_approx(d1), inv_d2 = rcp_approx(d2);
                        const float r = inv_d1 * inv_d2;
                        const float S = (n1 * n2) * r;
                        const float v = fmaf(-0.5f, S, 0.5f);
                        if (wy >= kHalo && wx >= kHalo) s_ssim += __saturatef(v);
                        if (p.need_grad && v >= 0.0f && v <= 1.0f) {
                            // dS/dx_p = A + B x_p + C y_p (DESIGN.md section 4); loss = (1-S)/2 / M
                            kk4.y = kk * (-S * inv_d2);
                            kk4.z = kk * (n1 * r);
                            kk4.x = kk * (m2.y * (n2 - n1) * r + S * m2.x * (inv_d2 - inv_d1));
                        }
                    }
                    sm.kab[c][wy * kWW + wx] = make_float2(kk4.x, kk4.y);
                    sm.kc[c][wy * kWW + wx] = kk4.z;
                }
            }
        }
    }
    if (WARP && has_lay) cp_async_commit_wait_all();
    __syncthreads();

    // ---------------- phase 2: own pixel ----------------
    const int ty = tid / kTW, tx = tid - ty * kTW;
    const int y = ty0 + ty, x = tx0 + tx;
    const bool inside = y < H && x < W;
    if (inside) {
        const int64_t o = (int64_t)y * W + x;
        const int q0 = (ty + kHalo) * kRW + tx + kHalo;
        Taps t;
        if (WARP) {
            float mx, my;
#if VLG_P1_FLOW_IN_SMEM
#define VLG_FLOW_AT(dq, doff) sm.flow[q0 + (dq)]
#else
#define VLG_FLOW_AT(dq, doff) __ldg(coords + o + (doff))
#endif
            const float2 xy = source_xy(cc, VLG_FLOW_AT(0, 0), sm.bx[tx + kHalo], sm.by[ty + kHalo], mx, my);
            t = taps_from_xy(cc, xy, mx, my);
            m_disp = tap_displacement(cc, t, y, x);
            m_near = m_disp < (float)VLG_NEAR_RADIUS ? m_disp : 0.0f;
            if (m_disp >= (float)VLG_NEAR_RADIUS && p.d_out_lay != nullptr) {
                // far pixel (rare): queue it for the fixed-point scatter and flag the source tiles it hits
                if (p.far_list) {
                    p.far_list[atomicAdd(&p.hdr->far_count, 1u)] = make_int4((int)(img_px + o), (t.x0 + 8) | ((t.y0 + 8) << 16),
                                                                              __float_as_int(t.ix - t.fx0), __float_as_int(t.iy - t.fy0));
                    far_announce(p.tile_flags, p.flagged_list, p.seg_cnt, p.hdr, n, p.tiles_x, p.tiles_y, t.x0, t.y0, W, H, nullptr);
                } else {
                    atomicOr(&p.hdr->status, VLG_STATUS_FAR_TAPS);
                }
            }
        }
        float gix = 0.f, giy = 0.f;

        if (has_rgb) {
            float dr[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float2 ab0 = sm.ab[c][q0];
                const float a = ab0.x, b = ab0.y;
                const float d = a - b;
                float g = 0.f;
                if (p.tc.terms & VLG_TERM_L1) {
                    s_l1 += fabsf(d);
                    g = signed_c1(p.tc.c_l1, d);
                }
                if (p.tc.terms & VLG_TERM_GD) {
                    // vertical pairs (reference `xloss`, src/loss.py:21-22): (y -> y+1) owned here
                    if (y + 1 < H) {
                        const float2 dv = __fadd2_rn(sm.ab[c][q0 + kRW], make_float2(-a, -b));
                        const float tt = fabsf(dv.x) - fabsf(dv.y);
                        s_gd += fabsf(tt);
                        g -= signed_c(p.tc.c_gd, tt, dv.x);
                    }
                    if (y >= 1) {
                        const float2 v = sm.ab[c][q0 - kRW];
                        const float da = a - v.x;
                        g += signed_c(p.tc.c_gd, fabsf(da) - fabsf(b - v.y), da);
                    }
                    // horizontal pairs (reference `yloss`, src/loss.py:23-24)
                    if (x + 1 < W) {
                        const float2 dv = __fadd2_rn(sm.ab[c][q0 + 1], make_float2(-a, -b));
                        const float tt = fabsf(dv.x) - fabsf(dv.y);
                        s_gd += fabsf(tt);
                        g -= signed_c(p.tc.c_gd, tt, dv.x);
                    }
                    if (x >= 1) {
                        const float2 v = sm.ab[c][q0 - 1];
                        const float da = a - v.x;
                        g += signed_c(p.tc.c_gd, fabsf(da) - fabsf(b - v.y), da);
                    }
                }
                if (p.need_grad && (p.tc.terms & VLG_TERM_SSIM)) {
                    // SSIM adjoint: the <=9 windows whose footprint contains this pixel
                    float2 sAB = make_float2(0.f, 0.f);
                    float sC = 0.f;
                    const float2 *kab = &sm.kab[c][ty * kWW + tx];
                    const float *kc = &sm.kc[c][ty * kWW + tx];
#pragma unroll
                    for (int di = 0; di < 3; ++di)
#pragma unroll
                        for (int dj = 0; dj < 3; ++dj) {
                            sAB = __fadd2_rn(sAB, kab[di * kWW + dj]);
                            sC += kc[di * kWW + dj];
                        }
                    g += fmaf(sC, b, fmaf(sAB.y, a, sAB.x));
                }
                dr[c] = g;
                m_grad = fmaxf(m_grad, fabsf(g));
            }
            if (p.need_grad && p.d_out_rgb) {
                store_px<T, 3>(reinterpret_cast<T *>(p.d_out_rgb) + (img_px + o) * 3, dr);
            }
        }

        if (has_lay) {
            const int64_t lab = lab_pre;
            const bool lab_ok = lab >= 0 && lab < K;
            if (!lab_ok && lab != p.ignore_index) atomicOr(&p.hdr->status, VLG_STATUS_BAD_LABEL);
            const int il = lab_ok ? (int)lab : 0;
            float z[K], v[K];
            float vl[4] = {0.f, 0.f, 0.f, 0.f};   // label channel of the four taps
            float zl;
            const T *st00 = nullptr;   // smem address of the nw tap when all four taps are staged
            if (WARP) {
                const int rx = t.x0 - ox, ry = t.y0 - oy;
                if (rx >= 0 && rx + 1 < sw && ry >= 0 && ry + 1 < sh) {
                    st00 = sm.stage + (size_t)(ry * kSW + rx) * K;
                    load_px_smem<T, K>(st00, v);                 mul2_bcast<K>(z, v, t.nw);
                    load_px_smem<T, K>(st00 + K, v);             fma2_bcast<K>(z, v, t.ne);
                    load_px_smem<T, K>(st00 + kSW * K, v);       fma2_bcast<K>(z, v, t.sw);
                    load_px_smem<T, K>(st00 + kSW * K + K, v);   fma2_bcast<K>(z, v, t.se);
                    vl[0] = to_f<T>(st00[il]);            vl[1] = to_f<T>(st00[K + il]);
                    vl[2] = to_f<T>(st00[kSW * K + il]);  vl[3] = to_f<T>(st00[kSW * K + K + il]);
                } else {
                    gather_px<T, K>(src_lay, cc, t, z);   // taps outside the staged window: global path
                    vl[0] = tap_global<T>(src_lay, K, il, t.y0, t.x0, H, W);
                    vl[1] = tap_global<T>(src_lay, K, il, t.y0, t.x0 + 1, H, W);
                    vl[2] = tap_global<T>(src_lay, K, il, t.y0 + 1, t.x0, H, W);
                    vl[3] = tap_global<T>(src_lay, K, il, t.y0 + 1, t.x0 + 1, H, W);
                }
                // same FMA chain as z[il], so zl == z[il] bit for bit without indexing registers
                zl = __fmaf_rn(vl[3], t.se, __fmaf_rn(vl[2], t.sw, __fmaf_rn(vl[1], t.ne, __fmul_rn(vl[0], t.nw))));
            } else {
                load_px<T, K>(src_lay + o * K, z);
                zl = to_f<T>(__ldg(src_lay + o * K + il));
            }
            float m = z[0];
#pragma unroll
            for (int k = 1; k < K; ++k) m = fmaxf(m, z[k]);
            if (p.out_argmax) {
                int best = K - 1;
#pragma unroll
                for (int k = K - 2; k >= 0; --k) best = (z[k] == m) ? k : best;   // first maximal index (src/trainer.py:342)
                p.out_argmax[img_px + o] = best;
            }
            // softmax in base 2: e_k = 2^((z_k - m) * log2(e))
            const float L2E = 1.4426950408889634f;
            const float ml2 = m * L2E;
            float se = 0.f;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                z[k] = ex2_approx(fmaf(z[k], L2E, -ml2));
                se += z[k];
            }
            if (lab_ok) s_ce += wl_pre * (fmaf(lg2_approx(se), 0.6931471805599453f, m) - zl);
            if (p.need_grad) {
                const float cce = lab_ok ? p.tc.w_ce_over_scale * wl_pre / denom_pre : 0.0f;
                const float inv = cce / se;
                // d/dz_k = cce * (softmax_k - [k == label]); the one-hot part is applied to the label
                // channel alone (a scalar fix-up store / a rank-1 term of the coordinate gradient)
                mul2_bcast<K>(z, z, inv);
                const float gl = fmaf(ex2_approx(fmaf(zl, L2E, -ml2)), inv, -cce);
                m_grad = fmaxf(m_grad, cce);   // |softmax - onehot| <= 1: an upper bound is all the far path needs
                if (WARP) {
                    float dnw, dne, dsw, dse;
                    if (st00) {
                        load_px_smem<T, K>(st00, v);                 dnw = dot2<K>(z, v);
                        load_px_smem<T, K>(st00 + K, v);             dne = dot2<K>(z, v);
                        load_px_smem<T, K>(st00 + kSW * K, v);       dsw = dot2<K>(z, v);
                        load_px_smem<T, K>(st00 + kSW * K + K, v);   dse = dot2<K>(z, v);
                        dnw = fmaf(-cce, vl[0], dnw); dne = fmaf(-cce, vl[1], dne);
                        dsw = fmaf(-cce, vl[2], dsw); dse = fmaf(-cce, vl[3], dse);
                        const float wx1 = t.ix - t.fx0, wx0 = (t.fx0 + 1.0f) - t.ix;
                        const float wy1 = t.iy - t.fy0, wy0 = (t.fy0 + 1.0f) - t.iy;
                        gix += (dne - dnw) * wy0 + (dse - dsw) * wy1;
                        giy += (dsw - dnw) * wx0 + (dse - dne) * wx1;
                    } else {
                        float gfull[K];
#pragma unroll
                        for (int k = 0; k < K; ++k) gfull[k] = z[k] - (k == il ? cce : 0.0f);
                        coord_grad_px<T, K>(src_lay, cc, t, gfull, gix, giy);
                    }
                    if (p.d_out_lay) {
                        // (a chunk-planar staging layout makes these stores coalesced, -10 us here, but
                        // costs pass 2 +27 us in strided cp.async runs: measured, rejected)
                        float *dst = reinterpret_cast<float *>(p.d_out_lay) + (img_px + o) * K;
                        store_px<float, K>(dst, z);
                        if (lab_ok) dst[il] = gl;
                    }
                } else if (p.d_out_lay) {
                    T *dst = reinterpret_cast<T *>(p.d_out_lay) + (img_px + o) * K;
                    store_px<T, K>(dst, z);
                    if (lab_ok) dst[il] = from_f<T>(gl);
                }
            }
        }

        if (WARP) {
            float gx = fmaf(t.mx, gix, dc_pre.x), gy = fmaf(t.my, giy, dc_pre.y);
            if (p.tc.terms & VLG_TERM_TV) {
                const float2 f = VLG_FLOW_AT(0, 0);
                if (y + 1 < H) {
                    const float2 df = __fadd2_rn(VLG_FLOW_AT(kRW, W), make_float2(-f.x, -f.y));
                    s_tvh += fabsf(df.x) + fabsf(df.y);
                    gx -= signed_c1(p.tc.c_tvh, df.x);
                    gy -= signed_c1(p.tc.c_tvh, df.y);
                }
                if (y >= 1) {
                    const float2 f1 = VLG_FLOW_AT(-kRW, -W);
                    gx += signed_c1(p.tc.c_tvh, f.x - f1.x);
                    gy += signed_c1(p.tc.c_tvh, f.y - f1.y);
                }
                if (x + 1 < W) {
                    const float2 df = __fadd2_rn(VLG_FLOW_AT(1, 1), make_float2(-f.x, -f.y));
                    s_tvw += fabsf(df.x) + fabsf(df.y);
                    gx -= signed_c1(p.tc.c_tvw, df.x);
                    gy -= signed_c1(p.tc.c_tvw, df.y);
                }
                if (x >= 1) {
                    const float2 f1 = VLG_FLOW_AT(-1, -1);
                    gx += signed_c1(p.tc.c_tvw, f.x - f1.x);
                    gy += signed_c1(p.tc.c_tvw, f.y - f1.y);
                }
            }
            if (p.need_grad && p.d_coords)
                reinterpret_cast<float2 *>(p.d_coords)[img_px + o] = make_float2(gx, gy);
        }
    }

    // ---------------- phase 3: block reduction -> one partial row per CTA ----------------
    float vals[6] = {s_l1, s_gd, s_ssim, s_ce, s_tvh, s_tvw};
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        const float r = warp_sum(vals[i]);
        if (lane == 0) sm.red[wid][i] = r;
    }
    m_disp = warp_max(m_disp);
    m_grad = warp_max(m_grad);
    m_near = warp_max(m_near);
    if (lane == 0) {
        sm.redmax[wid][0] = m_disp;
        sm.redmax[wid][1] = m_grad;
        sm.redmax[wid][2] = m_near;
    }
    __syncthreads();
    if (tid < kPartialSlots) {
        float r = 0.f;
        if (tid < 6)
#pragma unroll
            for (int w = 0; w < kThreads / 32; ++w) r += sm.red[w][tid];
        p.partials[(int64_t)bt * kPartialSlots + tid] = r;
        if (bt == 0 && tid == 0) p.hdr->n_tile = gridDim.x * gridDim.y * gridDim.z;
    }
    if (tid == 32) {
        float d = 0.f, g = 0.f, nr = 0.f;
#pragma unroll
        for (int w = 0; w < kThreads / 32; ++w) {
            d = fmaxf(d, sm.redmax[w][0]);
            g = fmaxf(g, sm.redmax[w][1]);
            nr = fmaxf(nr, sm.redmax[w][2]);
        }
        if (WARP && p.tile_disp) p.tile_disp[bt] = nr;
        if (d > 0.f) atomicMax(&p.hdr->maxdisp_bits, __float_as_uint(d));
        if (g > 0.f) {   // this organisation keeps one maximum over all channels: a valid (looser) bound for either group
            atomicMax(&p.hdr->maxgrad_rgb_bits, __float_as_uint(g));
            atomicMax(&p.hdr->maxgrad_lay_bits, __float_as_uint(g));
        }
    }

    // ---------------- phase 4: the last CTA to finish reduces all partial rows ----------------
    // (replaces a separate 1-CTA reduction launch; the summation order is fixed by row index, so
    // the result does not depend on which CTA happens to be last)
    if (p.red.out != nullptr) {
        __shared__ int s_last;
        if (tid < kPartialSlots || tid == 32) __threadfence();   // only the threads that wrote partials / maxima
        __syncthreads();
        if (tid == 0) s_last = atomicAdd(&p.hdr->blocks_done, 1u) == gridDim.x * gridDim.y * gridDim.z - 1;
        __syncthreads();
        if (s_last) {
            __threadfence();
            reduce_partials_block<kThreads>(p.red, reinterpret_cast<double *>(smem_raw));   // reuses sm.ab/flow (>= 12 KB)
        }
    }
}

}  // namespace vlg
