// vlg_device.cuh -- device-side building blocks shared by the sm_100a kernels.
//
// Coordinate arithmetic is written with explicit round-to-nearest intrinsics so that nvcc's FMA
// contraction cannot change a single bit relative to the oracle (SURVEY.md Appendix A):
//   base grid   reference src/models/modules.py:69-70      arange(S)/(S-1)*2-1
//   unnormalise torch ATen/native/GridSampler.h:31         ((g+1)/2)*(S-1)
//   clip        GridSampler.h:58-60
//   weights     Appendix A.5, accumulation Appendix A.6    fma(se, fma(sw, fma(ne, nw*)))
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/vlg_b200.h"

namespace vlg {

// ---------------------------------------------------------------- workspace layout
struct WsHeader {
    uint32_t status;        // VLG_STATUS_* bits (sticky until the next pass-1 launch)
    uint32_t maxdisp_bits;  // float bits of max |displacement| (non-negative => uint order == float order)
    uint32_t reserved0;
    uint32_t far_count;     // number of far output pixels
    unsigned long long n_valid;  // labels != ignore_index
    uint32_t blocks_done;   // pass-1 CTAs that have published their partial sums (last one reduces)
    uint32_t n_flagged;     // source tiles that receive far contributions (length of the flagged list)
    uint32_t count_done;    // label-count CTAs finished (the last one derives ce_denom)
    uint32_t n_rgb;         // per-warp partial rows written by rgb_strip_kernel (0: it did not run)
    double ce_denom;        // divisor of the weighted CE sum: sum_k w_k * hist_k (VLG_CE_NORM_TORCH with weights)
    uint32_t n_tile;        // partial rows written by the tile kernel (pass1_kernel), 0: it did not run
    uint32_t n_lay;         // per-CTA partial rows written by lay_tile_kernel
    uint32_t maxgrad_rgb_bits;  // float bits of max |d_out| over the rgb channels    } scales of the fixed-point far path, which treats
    uint32_t maxgrad_lay_bits;  // ... over the layout channels                       } the two groups separately (vlg_pass2.cuh)
    unsigned long long prof[8];   // spare (tuning builds: per-section cycle counters)
    unsigned long long hist[32];  // labels per class (only filled when class weights are given)
};
static_assert(sizeof(WsHeader) == 384, "header size");

constexpr int kPartialSlots = 8;  // l1, gd, ssim, ce, tv_h, tv_w, n_valid(unused), spare

// Final reduction of the partial sums: fixed summation order (row index, then a fixed tree), fp64
// accumulation -> bitwise reproducible loss vector whatever the CTA / warp schedule was.  Three
// producers: the tile kernel (one row of 8 per CTA), the rgb strip kernel (l1, gd, ssim per warp)
// and the layout strip kernel (ce, tv_h, tv_w per warp); each publishes its row count in the header.
struct ReduceParams {
    const float *partials;       // [hdr->n_tile][kPartialSlots]
    const float *partials_rgb;   // [hdr->n_rgb][4]  (l1, gd, ssim, -)
    const float *partials_lay;   // [hdr->n_lay][4]  (ce, tv_h, tv_w, -)
    const WsHeader *hdr;
    double inv_numel_rgb;   // 1/(Ng*3*H*W)
    double inv_ssim;        // 1/(Ng*(H-2)*(W-2))
    double inv_tvh, inv_tvw;
    double ce_scale;        // N_local/N_global
    float w_l1, w_gd, w_ssim, w_ce, w_tv;
    int weighted_denom;     // 1: CE divisor = hdr->ce_denom (class-weighted torch mean), 0: n_valid
    uint32_t terms;         // TermCoeffs::terms: the slot of a term whose bit is clear reads 0 and stays out of the total
    float *out;
};

// The loss terms a call evaluates and their gradient scales (upstream gradient 1.0), derived once on the host from the
// problem (make_terms).  A coefficient is 0 when its term is off.
struct TermCoeffs {
    uint32_t terms;              // VLG_TERM_* bits in effect: term_mask (0 = all), SSIM cleared below 3x3, TV only for pixel flow
    float c_l1, c_gd, c_ssim, c_tvh, c_tvw;
    float w_ce_over_scale;       // w_ce * (N_local/N_global); divided by the CE divisor on the device
    int weighted_denom;          // 1: CE divisor = hdr->ce_denom (class-weighted torch mean), 0: number of valid labels
};

// The CE divisor counted by count_valid_kernel, as the pass-1 kernels scale their CE gradient with it.
__device__ __forceinline__ float ce_divisor(const TermCoeffs &tc, const WsHeader *hdr) {
    return tc.weighted_denom ? (float)__ldcg(&hdr->ce_denom) : (float)__ldcg(&hdr->n_valid);
}

// Called by all NT threads of one CTA; `s` is 6*NT doubles of shared memory.
template <int NT>
__device__ __forceinline__ void reduce_partials_block(const ReduceParams &p, double *s) {
    double acc[6] = {0, 0, 0, 0, 0, 0};
    const int64_t n_tile = __ldcg(&p.hdr->n_tile), n_rgb = __ldcg(&p.hdr->n_rgb), n_lay = __ldcg(&p.hdr->n_lay);
    for (int64_t b = threadIdx.x; b < n_tile; b += NT) {
        const float4 lo = __ldcg(reinterpret_cast<const float4 *>(p.partials + b * kPartialSlots));
        const float2 hi = __ldcg(reinterpret_cast<const float2 *>(p.partials + b * kPartialSlots + 4));
        acc[0] += lo.x; acc[1] += lo.y; acc[2] += lo.z; acc[3] += lo.w; acc[4] += hi.x; acc[5] += hi.y;
    }
    for (int64_t b = threadIdx.x; b < n_rgb; b += NT) {
        const float4 v = __ldcg(reinterpret_cast<const float4 *>(p.partials_rgb) + b);
        acc[0] += v.x; acc[1] += v.y; acc[2] += v.z;
    }
    for (int64_t b = threadIdx.x; b < n_lay; b += NT) {
        const float4 v = __ldcg(reinterpret_cast<const float4 *>(p.partials_lay) + b);
        acc[3] += v.x; acc[4] += v.y; acc[5] += v.z;
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) s[i * NT + threadIdx.x] = acc[i];
    __syncthreads();
    for (int o = NT / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o)
#pragma unroll
            for (int i = 0; i < 6; ++i) s[i * NT + threadIdx.x] += s[i * NT + threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double nv = (double)__ldcg(&p.hdr->n_valid);
        const double l1 = (p.terms & VLG_TERM_L1) ? s[0] * p.inv_numel_rgb : 0.0;
        const double gd = (p.terms & VLG_TERM_GD) ? s[NT] * p.inv_numel_rgb : 0.0;
        const double ssim = (p.terms & VLG_TERM_SSIM) ? s[2 * NT] * p.inv_ssim : 0.0;
        const double cd = p.weighted_denom ? __ldcg(&p.hdr->ce_denom) : nv;
        const double ce = ((p.terms & VLG_TERM_CE) && cd > 0) ? s[3 * NT] / cd * p.ce_scale : 0.0;
        const double tv = (p.terms & VLG_TERM_TV) ? s[4 * NT] * p.inv_tvh + s[5 * NT] * p.inv_tvw : 0.0;
        p.out[VLG_LOSS_L1] = (float)l1;
        p.out[VLG_LOSS_GD] = (float)gd;
        p.out[VLG_LOSS_SSIM] = (float)ssim;
        p.out[VLG_LOSS_CE] = (float)ce;
        p.out[VLG_LOSS_TV] = (float)tv;
        const double tot = (double)p.w_l1 * l1 + (double)p.w_gd * gd + (double)p.w_ssim * ssim +
                           (double)p.w_ce * ce + (double)p.w_tv * tv;
        p.out[VLG_LOSS_TOTAL] = (float)tot;
        p.out[VLG_LOSS_NVALID] = (float)nv;
        p.out[VLG_LOSS_MAXDISP] = __uint_as_float(__ldcg(&p.hdr->maxdisp_bits));
    }
}

// The arrays of a workspace (ws_layout); NULL where the problem allocates none.
struct WsLayout {
    WsHeader *hdr;
    uint32_t *tile_flags;
    float *tile_disp;
    uint32_t *seg_cnt;           // NULL under VLG_FLAG_FAR_WIDE (its space stays reserved)
    float *partials, *partials_rgb, *partials_lay;
    int *flagged;
    // with a source gradient only
    float *dout_rgb, *dout_lay;
    uint32_t *rec_code;          // tap records of pass 1 for pass 2 (pitched rows)
    float2 *rec_frac;
    long long *far_acc;          // far_acc / far_list: NULL under VLG_FLAG_NO_FAR_PATH
    int4 *far_list;
    int64_t pitch;               // row pitch (pixels) of dout_rgb / rec_code / rec_frac: W rounded up to 4, so that every
                                 // row starts on a 16-byte boundary and the arrays can be described by TMA tensor maps
    size_t zero_bytes;           // header .. seg_cnt: what pass 1 resets with one memset
    size_t total;
};

// ---------------------------------------------------------------- tiling of pass 1
constexpr int kTW = 32, kTH = 8;          // output tile (one thread per pixel)
constexpr int kHalo = 2;                  // SSIM adjoint reaches 2 pixels
constexpr int kRW = kTW + 2 * kHalo, kRH = kTH + 2 * kHalo, kRN = kRW * kRH;  // rgb region
constexpr int kWW = kTW + 2, kWH = kTH + 2, kWN = kWW * kWH;                  // 3x3 windows
constexpr int kThreads = kTW * kTH;

__host__ __device__ inline int64_t tiles_x(int64_t W) { return (W + kTW - 1) / kTW; }
__host__ __device__ inline int64_t tiles_y(int64_t H) { return (H + kTH - 1) / kTH; }

// A far output pixel (vlg_pass2.cuh) announces itself to the source tiles its four taps (x0 | x0+1, y0 | y0+1) land in: the
// tile is flagged (once: an L2 load first, the returning atomic only while the flag still reads 0 -- with rough flow every
// tile is hit hundreds of times) and the row of the tile counts one more far pixel (a RED, no round trip).  The two taps
// of a row share a segment unless they straddle a tile border.
// `seen` (nullable): a CTA's direct-mapped memory (kFarSeen ints of shared memory, initialised to -1) of tiles it has already
// flagged -- rough flow lands in the same few tiles around the CTA's own again and again, and the L2 round trip of the
// flag load was 18 % of the layout kernel's stall samples on BASELINE config 5.
constexpr int kFarSeen = 256;
__device__ __forceinline__ void far_announce(uint32_t *tile_flags, int *flagged_list, uint32_t *seg_cnt, WsHeader *hdr,
                                             int n, int tiles_x_, int tiles_y_, int x0, int y0, int W, int H, int *seen) {
    int flagged = -1;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int yy = y0 + r;
        if (yy < 0 || yy >= H) continue;
        int last = -1;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const int xx = x0 + c;
            if (xx < 0 || xx >= W) continue;
            const int tl = (n * tiles_y_ + yy / kTH) * tiles_x_ + xx / kTW;
            if (tl == last) continue;
            last = tl;
            if (seg_cnt) atomicAdd(&seg_cnt[(int64_t)tl * kTH + (yy & (kTH - 1))], 1u);
            if (tl != flagged) {
                flagged = tl;
                if (seen == nullptr || seen[tl & (kFarSeen - 1)] != tl) {
                    if (__ldcg(&tile_flags[tl]) == 0u && atomicOr(&tile_flags[tl], 1u) == 0u)
                        flagged_list[atomicAdd(&hdr->n_flagged, 1u)] = tl;
                    if (seen) seen[tl & (kFarSeen - 1)] = tl;      // after the flag is set; a lost race costs one more look
                }
            }
        }
    }
}

// ---------------------------------------------------------------- typed loads / stores
template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

__host__ __device__ constexpr int vec_bytes(int pixel_bytes) {
    return pixel_bytes % 16 == 0 ? 16 : pixel_bytes % 8 == 0 ? 8 : pixel_bytes % 4 == 0 ? 4 : 2;
}

// Load C consecutive channels of one pixel (read-only path) into fp32 registers.
template <typename T, int C>
__device__ __forceinline__ void load_px(const T *__restrict__ p, float (&v)[C]) {
    constexpr int VB = vec_bytes(C * (int)sizeof(T));
    constexpr int EPV = VB / (int)sizeof(T);  // elements per vector
    static_assert(EPV >= 1, "vector narrower than an element");
    if constexpr (VB == 16) {
        const uint4 *q = reinterpret_cast<const uint4 *>(p);
#pragma unroll
        for (int i = 0; i < C / EPV; ++i) {
            uint4 r = __ldg(q + i);
            const T *e = reinterpret_cast<const T *>(&r);
#pragma unroll
            for (int j = 0; j < EPV; ++j) v[i * EPV + j] = to_f<T>(e[j]);
        }
    } else if constexpr (VB == 8) {
        const uint2 *q = reinterpret_cast<const uint2 *>(p);
#pragma unroll
        for (int i = 0; i < C / EPV; ++i) {
            uint2 r = __ldg(q + i);
            const T *e = reinterpret_cast<const T *>(&r);
#pragma unroll
            for (int j = 0; j < EPV; ++j) v[i * EPV + j] = to_f<T>(e[j]);
        }
    } else if constexpr (VB == 4 && sizeof(T) == 2) {
        const uint32_t *q = reinterpret_cast<const uint32_t *>(p);
#pragma unroll
        for (int i = 0; i < C / 2; ++i) {
            uint32_t r = __ldg(q + i);
            const T *e = reinterpret_cast<const T *>(&r);
            v[2 * i] = to_f<T>(e[0]);
            v[2 * i + 1] = to_f<T>(e[1]);
        }
    } else {
#pragma unroll
        for (int i = 0; i < C; ++i) v[i] = to_f<T>(__ldg(p + i));
    }
}

// argmax over the K channels of one pixel as torch.argmax takes it (src/trainer.py:342,467): the first maximal index,
// strict `>` in channel order.  `z` holds the values as stored in the layout's dtype.
template <int K>
__device__ __forceinline__ int first_max_index(const float (&z)[K]) {
    float m = z[0];
    int best = 0;
#pragma unroll
    for (int k = 1; k < K; ++k)
        if (z[k] > m) { m = z[k]; best = k; }
    return best;
}

template <typename T, int C>
__device__ __forceinline__ void store_px(T *__restrict__ p, const float (&v)[C]) {
    constexpr int VB = vec_bytes(C * (int)sizeof(T));
    constexpr int EPV = VB / (int)sizeof(T);
    if constexpr (VB == 16) {
        uint4 *q = reinterpret_cast<uint4 *>(p);
#pragma unroll
        for (int i = 0; i < C / EPV; ++i) {
            uint4 r;
            T *e = reinterpret_cast<T *>(&r);
#pragma unroll
            for (int j = 0; j < EPV; ++j) e[j] = from_f<T>(v[i * EPV + j]);
            q[i] = r;
        }
    } else if constexpr (VB == 8) {
        uint2 *q = reinterpret_cast<uint2 *>(p);
#pragma unroll
        for (int i = 0; i < C / EPV; ++i) {
            uint2 r;
            T *e = reinterpret_cast<T *>(&r);
#pragma unroll
            for (int j = 0; j < EPV; ++j) e[j] = from_f<T>(v[i * EPV + j]);
            q[i] = r;
        }
    } else {
#pragma unroll
        for (int i = 0; i < C; ++i) p[i] = from_f<T>(v[i]);
    }
}

// ---------------------------------------------------------------- sampling coordinates
struct CoordCfg {
    int H, W;
    int padding, coord_mode;
    float Wm1, Hm1;  // (float)(W-1), (float)(H-1)
    float sx, sy;    // fp32(2/(W-1)), fp32(2/(H-1)) rounded once from double on the host
};

struct Taps {
    float ix, iy;     // source coordinates after padding treatment
    float fx0, fy0;   // floor
    float nw, ne, sw, se;
    int x0, y0;
    float mx, my;     // d(ix)/d(coord) incl. border mask and (flow mode) the pixel->grid scale
};

__device__ __forceinline__ float base_coord(int i, float Sm1) {
    // reference src/models/modules.py:69: (i / (S-1)) * 2 - 1, one rounding per op
    return __fsub_rn(__fmul_rn(__fdiv_rn((float)i, Sm1), 2.0f), 1.0f);
}

// c = raw coords of output pixel (y,x): flow in pixels or normalised grid value.
__device__ __forceinline__ Taps make_taps(const CoordCfg &cc, float2 c, int y, int x) {
    float gx, gy;
    if (cc.coord_mode == VLG_COORD_FLOW) {
        gx = __fadd_rn(base_coord(x, cc.Wm1), __fmul_rn(c.x, cc.sx));
        gy = __fadd_rn(base_coord(y, cc.Hm1), __fmul_rn(c.y, cc.sy));
    } else {
        gx = c.x;
        gy = c.y;
    }
    // GridSampler.h:31 -- (g+1)/2 is exact, so one rounding after the add and one after the mul
    float ux = __fmul_rn(__fmul_rn(__fadd_rn(gx, 1.0f), 0.5f), cc.Wm1);
    float uy = __fmul_rn(__fmul_rn(__fadd_rn(gy, 1.0f), 0.5f), cc.Hm1);
    Taps t;
    // GridSampler.h:47 and :70-81 (border positions count as clipped for the gradient)
    t.mx = __fmul_rn(cc.Wm1, 0.5f);
    t.my = __fmul_rn(cc.Hm1, 0.5f);
    if (cc.padding == VLG_PAD_BORDER) {
        if (ux <= 0.0f || ux >= cc.Wm1) t.mx = 0.0f;
        if (uy <= 0.0f || uy >= cc.Hm1) t.my = 0.0f;
        ux = fminf(cc.Wm1, fmaxf(ux, 0.0f));
        uy = fminf(cc.Hm1, fmaxf(uy, 0.0f));
    }
    if (cc.coord_mode == VLG_COORD_FLOW) {
        t.mx *= cc.sx;
        t.my *= cc.sy;
    }
    t.ix = ux;
    t.iy = uy;
    t.fx0 = floorf(ux);
    t.fy0 = floorf(uy);
    const float fx1 = __fadd_rn(t.fx0, 1.0f), fy1 = __fadd_rn(t.fy0, 1.0f);
    const float wx1 = __fsub_rn(ux, t.fx0), wx0 = __fsub_rn(fx1, ux);
    const float wy1 = __fsub_rn(uy, t.fy0), wy0 = __fsub_rn(fy1, uy);
    t.nw = __fmul_rn(wx0, wy0);
    t.ne = __fmul_rn(wx1, wy0);
    t.sw = __fmul_rn(wx0, wy1);
    t.se = __fmul_rn(wx1, wy1);
    // Saturating conversion keeps far-out-of-range zeros-mode coordinates harmless.
    t.x0 = (int)fminf(fmaxf(t.fx0, -4.0f), (float)cc.W + 4.0f);
    t.y0 = (int)fminf(fmaxf(t.fy0, -4.0f), (float)cc.H + 4.0f);
    return t;
}

// Chebyshev displacement of the sampling position from its own output pixel, in source pixels.
// Output pixels whose four taps all fall outside the image contribute nothing and report 0.
__device__ __forceinline__ float tap_displacement(const CoordCfg &cc, const Taps &t, int y, int x) {
    if (t.x0 < -1 || t.x0 >= cc.W || t.y0 < -1 || t.y0 >= cc.H) return 0.0f;
    return fmaxf(fabsf(t.ix - (float)x), fabsf(t.iy - (float)y));
}

// Tap record of one output pixel, written by pass 1 and consumed by pass 2 (the transpose of the gather):
// the cell of the NW tap relative to the pixel itself, packed as (x0 - x + 8) | (y0 - y + 8) << 16, or 0
// when the pixel contributes nothing through the near path (all taps outside the image, or displaced by
// >= VLG_NEAR_RADIUS: those travel through the fixed-point far path).  A valid code is never 0 -- which
// is also what the TMA zero-fill hands pass 2 for cells outside the image.
__device__ __forceinline__ uint32_t tap_cell_code(const CoordCfg &cc, const Taps &t, int y, int x) {
    const bool dead = t.x0 < -1 || t.x0 >= cc.W || t.y0 < -1 || t.y0 >= cc.H;
    const bool far = fmaxf(fabsf(t.ix - (float)x), fabsf(t.iy - (float)y)) >= (float)VLG_NEAR_RADIUS;
    return (dead || far) ? 0u : ((uint32_t)(t.x0 - x + 8) | ((uint32_t)(t.y0 - y + 8) << 16));
}

// Bilinear gather of C channels at one output pixel from an NHWC image plane `img` (batch n
// already applied).  Bit-exact FMA chain of Appendix A.6; out-of-image taps read 0.
template <typename T, int C>
__device__ __forceinline__ void gather_px(const T *__restrict__ img, const CoordCfg &cc, const Taps &t,
                                          float (&out)[C]) {
    const bool xin0 = t.x0 >= 0 && t.x0 < cc.W, xin1 = t.x0 + 1 >= 0 && t.x0 + 1 < cc.W;
    const bool yin0 = t.y0 >= 0 && t.y0 < cc.H, yin1 = t.y0 + 1 >= 0 && t.y0 + 1 < cc.H;
    const T *p00 = img + ((int64_t)t.y0 * cc.W + t.x0) * C;
    float v[C];
    if (yin0 && xin0) {
        load_px<T, C>(p00, v);
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = __fmul_rn(v[c], t.nw);
    } else {
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = __fmul_rn(0.0f, t.nw);
    }
    if (yin0 && xin1) {
        load_px<T, C>(p00 + C, v);
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = __fmaf_rn(v[c], t.ne, out[c]);
    }
    if (yin1 && xin0) {
        load_px<T, C>(p00 + (int64_t)cc.W * C, v);
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = __fmaf_rn(v[c], t.sw, out[c]);
    }
    if (yin1 && xin1) {
        load_px<T, C>(p00 + (int64_t)cc.W * C + C, v);
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = __fmaf_rn(v[c], t.se, out[c]);
    }
}

// d(out)/d(ix), d(out)/d(iy) contracted with the per-channel upstream gradient g[C]
// (GridSampler.h backward: gix = sum_c g_c * [(v_ne-v_nw)(y1-iy) + (v_se-v_sw)(iy-y0)]).
template <typename T, int C>
__device__ __forceinline__ void coord_grad_px(const T *__restrict__ img, const CoordCfg &cc, const Taps &t,
                                              const float (&g)[C], float &gix, float &giy) {
    const bool xin0 = t.x0 >= 0 && t.x0 < cc.W, xin1 = t.x0 + 1 >= 0 && t.x0 + 1 < cc.W;
    const bool yin0 = t.y0 >= 0 && t.y0 < cc.H, yin1 = t.y0 + 1 >= 0 && t.y0 + 1 < cc.H;
    const T *p00 = img + ((int64_t)t.y0 * cc.W + t.x0) * C;
    float a[C], b[C];  // a = sum_c g_c v_nw.. handled tap by tap to keep registers low
    const float wx1 = t.ix - t.fx0, wx0 = (t.fx0 + 1.0f) - t.ix;
    const float wy1 = t.iy - t.fy0, wy0 = (t.fy0 + 1.0f) - t.iy;
    float dnw = 0.f, dne = 0.f, dsw = 0.f, dse = 0.f;  // sum_c g_c * v_tap
    if (yin0 && xin0) {
        load_px<T, C>(p00, a);
#pragma unroll
        for (int c = 0; c < C; ++c) dnw = fmaf(g[c], a[c], dnw);
    }
    if (yin0 && xin1) {
        load_px<T, C>(p00 + C, b);
#pragma unroll
        for (int c = 0; c < C; ++c) dne = fmaf(g[c], b[c], dne);
    }
    if (yin1 && xin0) {
        load_px<T, C>(p00 + (int64_t)cc.W * C, a);
#pragma unroll
        for (int c = 0; c < C; ++c) dsw = fmaf(g[c], a[c], dsw);
    }
    if (yin1 && xin1) {
        load_px<T, C>(p00 + (int64_t)cc.W * C + C, b);
#pragma unroll
        for (int c = 0; c < C; ++c) dse = fmaf(g[c], b[c], dse);
    }
    gix += (dne - dnw) * wy0 + (dse - dsw) * wy1;
    giy += (dsw - dnw) * wx0 + (dse - dne) * wx1;
}

// Shared-memory variants (plain loads, no read-only path) used on the staged source window.
template <typename T, int C>
__device__ __forceinline__ void load_px_smem(const T *p, float (&v)[C]) {
    constexpr int VB = vec_bytes(C * (int)sizeof(T));
    constexpr int EPV = VB / (int)sizeof(T);
    if constexpr (VB == 16) {
#pragma unroll
        for (int i = 0; i < C / EPV; ++i) {
            const uint4 r = reinterpret_cast<const uint4 *>(p)[i];
            const T *e = reinterpret_cast<const T *>(&r);
#pragma unroll
            for (int j = 0; j < EPV; ++j) v[i * EPV + j] = to_f<T>(e[j]);
        }
    } else if constexpr (VB == 8) {
#pragma unroll
        for (int i = 0; i < C / EPV; ++i) {
            const uint2 r = reinterpret_cast<const uint2 *>(p)[i];
            const T *e = reinterpret_cast<const T *>(&r);
#pragma unroll
            for (int j = 0; j < EPV; ++j) v[i * EPV + j] = to_f<T>(e[j]);
        }
    } else {
#pragma unroll
        for (int i = 0; i < C; ++i) v[i] = to_f<T>(p[i]);
    }
}

// coord_grad_px on a staged window: all four taps are present (out-of-image cells hold zeros).
template <typename T, int C>
__device__ __forceinline__ void coord_grad_smem(const T *p00, int row_stride, const Taps &t, const float (&g)[C],
                                                float &gix, float &giy) {
    const float wx1 = t.ix - t.fx0, wx0 = (t.fx0 + 1.0f) - t.ix;
    const float wy1 = t.iy - t.fy0, wy0 = (t.fy0 + 1.0f) - t.iy;
    float v[C];
    float dnw = 0.f, dne = 0.f, dsw = 0.f, dse = 0.f;
    load_px_smem<T, C>(p00, v);
#pragma unroll
    for (int c = 0; c < C; ++c) dnw = fmaf(g[c], v[c], dnw);
    load_px_smem<T, C>(p00 + C, v);
#pragma unroll
    for (int c = 0; c < C; ++c) dne = fmaf(g[c], v[c], dne);
    load_px_smem<T, C>(p00 + row_stride, v);
#pragma unroll
    for (int c = 0; c < C; ++c) dsw = fmaf(g[c], v[c], dsw);
    load_px_smem<T, C>(p00 + row_stride + C, v);
#pragma unroll
    for (int c = 0; c < C; ++c) dse = fmaf(g[c], v[c], dse);
    gix += (dne - dnw) * wy0 + (dse - dsw) * wy1;
    giy += (dsw - dnw) * wx0 + (dse - dne) * wx1;
}

// ---------------------------------------------------------------- Blackwell packed fp32x2 math
// sm_100 adds FFMA2 / FMUL2 / FADD2 (two IEEE fp32 lanes per instruction, one issue slot): the
// per-channel loops are issue-bound, so they run on channel PAIRS.  Each lane rounds exactly like
// the scalar op, so the bit-exact FMA chain of Appendix A.6 is preserved.
template <int C>
__device__ __forceinline__ void mul2_bcast(float (&z)[C], const float (&v)[C], float w) {
    const float2 w2 = make_float2(w, w);
#pragma unroll
    for (int j = 0; j + 1 < C; j += 2) {
        const float2 r = __fmul2_rn(make_float2(v[j], v[j + 1]), w2);
        z[j] = r.x; z[j + 1] = r.y;
    }
    if (C & 1) z[C - 1] = __fmul_rn(v[C - 1], w);
}
template <int C>
__device__ __forceinline__ void fma2_bcast(float (&z)[C], const float (&v)[C], float w) {
    const float2 w2 = make_float2(w, w);
#pragma unroll
    for (int j = 0; j + 1 < C; j += 2) {
        const float2 r = __ffma2_rn(make_float2(v[j], v[j + 1]), w2, make_float2(z[j], z[j + 1]));
        z[j] = r.x; z[j + 1] = r.y;
    }
    if (C & 1) z[C - 1] = __fmaf_rn(v[C - 1], w, z[C - 1]);
}
template <int C>
__device__ __forceinline__ float dot2(const float (&g)[C], const float (&v)[C]) {
    float2 acc = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j + 1 < C; j += 2) acc = __ffma2_rn(make_float2(g[j], g[j + 1]), make_float2(v[j], v[j + 1]), acc);
    float r = acc.x + acc.y;
    if (C & 1) r = fmaf(g[C - 1], v[C - 1], r);
    return r;
}

__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lg2_approx(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// ---------------------------------------------------------------- tuning builds: when do the units of a persistent kernel finish?
// (tools/tail_prof.py; -DVLG_PROFILE_TAIL)
#ifdef VLG_PROFILE_TAIL
__device__ __forceinline__ unsigned long long global_ns() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
// (SM id << 24) | (ns timer / 16, 24 bits): where and when a unit of work finished
__device__ __forceinline__ unsigned prof_stamp() {
    unsigned sm; asm volatile("mov.u32 %0, %smid;" : "=r"(sm));
    return (sm << 24) | (unsigned)((global_ns() >> 4) & 0xFFFFFFull);
}
// slots (zero-initialised with the header): [0] ~(first start), [1] last start, [2] ~(first end), [3] last end
__device__ __forceinline__ void prof_mark(unsigned long long *slot4, bool end) {
    const unsigned long long t = global_ns();
    atomicMax(slot4 + (end ? 2 : 0), ~t);
    atomicMax(slot4 + (end ? 3 : 1), t);
}
#endif

// ---------------------------------------------------------------- reductions
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__device__ __forceinline__ float sgn(float v) { return (float)((v > 0.0f) - (v < 0.0f)); }

}  // namespace vlg
