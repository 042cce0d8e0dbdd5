// vlg_rgb.cuh -- the RGB half of pass 1 as a register-resident column-strip pipeline.
//
// What it computes (reference gongaa/video-layout-generation):
//   warp        (absent upstream) F.grid_sample(bilinear, align_corners=True) on the
//               src/models/modules.py:69 grid -- same bit-exact tap arithmetic as vlg_device.cuh
//   L1          src/trainer.py:130,248      mean |a-b|, sign(0)=0
//   GD          src/loss.py:20-25           sum||da|-|db|| along H and along W, / (N*C*H*W)
//   SSIM        src/loss.py:68-91           3x3 valid avg-pool stats, clamp((1-SSIM)/2,0,1).mean()
// and their gradients w.r.t. the warped image (d_out_rgb) and, through the sampler, w.r.t. the
// coordinates (rgb part of d_coords; the layout kernel adds its own part and the TV term).
//
// Organisation.  The tile kernel spends most of its instructions on shared-memory stencil traffic,
// halo recomputation (1.69x) and barriers.  Here ONE WARP owns a strip of 28 output columns (+2 halo
// lanes on each side) and walks down the rows:
//   * vertical neighbours (GD pairs, the three rows of an SSIM window, the 3x3 adjoint box) live in
//     REGISTERS as a sliding window over the last three rows -- no shared memory, no halo rows
//     except 4 per segment;
//   * horizontal neighbours come from warp shuffles (4 per channel for the pixel values, 6 for the
//     SSIM adjoint coefficients);
//   * no __syncthreads anywhere: warps are independent, work is split into equal contiguous runs
//     of (image, strip, row) so that a single wave of persistent warps finishes together;
//   * the loads of row t+1 (taps + target) and the flow of row t+2 are issued before row t is
//     processed (software pipeline), so the dependent flow -> taps round trips overlap compute.
// Per row t the warp: warps row t, forms the horizontal 3-sums of (a, b, a^2, b^2, ab), completes the
// SSIM windows centred on row t-1, and finalises the gradient of row t-2.
#pragma once
#include <type_traits>
#include "vlg_device.cuh"
#include "vlg_pass1.cuh"   // source_xy, taps_from_xy, signed_c

namespace vlg {

constexpr int kRS = 28;             // output columns per strip (32 lanes - 2x2 halo)
constexpr int kRgbThreads = 128;    // 4 independent warps per CTA
#ifndef VLG_RGB_MIN_BLOCKS
#define VLG_RGB_MIN_BLOCKS 3
#endif
constexpr int kRgbSlots = 4;        // partial sums per warp: l1, gd, ssim, spare
constexpr int kRgbMaxWarps = 8192;  // rows reserved in the workspace

struct RgbParams {
    CoordCfg cc;
    int N, strips;                  // strips = ceil(W / kRS)
    int64_t total_rows;             // N * strips * H
    int64_t chunk;                  // rows per warp (contiguous in (n, strip, y) order)
    const void *src_rgb, *tgt_rgb;
    const float *coords;
    TermCoeffs tc;                  // c_l1, c_gd, c_ssim: the rgb gradient scales
    float *d_coords;                // [P][2] rgb part of d(loss)/d(coords); the layout kernel that follows adds its own (nullable)
    float *d_out_rgb;               // [N][H][pitch][3] fp32 staging for pass 2 (nullable)
    int pitch;
    float *partials;                // [n_warps][kRgbSlots]
    WsHeader *hdr;
};

struct RgbRow {                     // one row in flight: raw taps, target, weights
    float v[4][3];
    float b[3];
    float nw, ne, sw, se, wx1, wy1, mx, my;
    unsigned tin;                   // bit k: tap k lies inside the image
};

// BORDER: taps are clamped into the image, so the only out-of-image tap is x0+1 == W (or y0+1 == H) and it
// carries weight exactly 0 and a coordinate-gradient mask of exactly 0: the clamped load stands in for
// the zero torch substitutes and no per-tap select is needed (finite inputs).
template <typename T, bool BORDER>
__device__ __forceinline__ void rgb_issue_row(RgbRow &r, const CoordCfg &cc, float2 fl, float bxv, int t, int xc,
                                              const T *__restrict__ src, const T *__restrict__ tgt, bool row_ok) {
    const int H = cc.H, W = cc.W;
    if (row_ok) {
        float mx, my;
        const float2 xy = source_xy(cc, fl, bxv, base_coord(t, cc.Hm1), mx, my);
        const Taps tp = taps_from_xy(cc, xy, mx, my);
        // border padding: the position was clipped into [0, S-1] before the floor, so only the far taps need a clamp
        const int x0c = BORDER ? tp.x0 : min(max(tp.x0, 0), W - 1), x1c = BORDER ? min(tp.x0 + 1, W - 1) : min(max(tp.x0 + 1, 0), W - 1);
        const int y0c = BORDER ? tp.y0 : min(max(tp.y0, 0), H - 1), y1c = BORDER ? min(tp.y0 + 1, H - 1) : min(max(tp.y0 + 1, 0), H - 1);
        load_px<T, 3>(src + (int64_t)(y0c * W + x0c) * 3, r.v[0]);
        load_px<T, 3>(src + (int64_t)(y0c * W + x1c) * 3, r.v[1]);
        load_px<T, 3>(src + (int64_t)(y1c * W + x0c) * 3, r.v[2]);
        load_px<T, 3>(src + (int64_t)(y1c * W + x1c) * 3, r.v[3]);
        load_px<T, 3>(tgt + (int64_t)(t * W + xc) * 3, r.b);
        if (!BORDER) {
            const bool xin0 = tp.x0 >= 0 && tp.x0 < W, xin1 = tp.x0 + 1 >= 0 && tp.x0 + 1 < W;
            const bool yin0 = tp.y0 >= 0 && tp.y0 < H, yin1 = tp.y0 + 1 >= 0 && tp.y0 + 1 < H;
            r.tin = (unsigned)(yin0 && xin0) | ((unsigned)(yin0 && xin1) << 1) | ((unsigned)(yin1 && xin0) << 2) |
                    ((unsigned)(yin1 && xin1) << 3);
        } else {
            r.tin = 15u;
        }
        r.nw = tp.nw; r.ne = tp.ne; r.sw = tp.sw; r.se = tp.se;
        r.wx1 = tp.ix - tp.fx0; r.wy1 = tp.iy - tp.fy0;
        r.mx = mx; r.my = my;
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int c = 0; c < 3; ++c) r.v[k][c] = 0.f;
#pragma unroll
        for (int c = 0; c < 3; ++c) r.b[c] = 0.f;
        r.nw = r.ne = r.sw = r.se = r.wx1 = r.wy1 = r.mx = r.my = 0.f;
        r.tin = 0u;
    }
}

template <typename T, bool GRAD, bool BORDER>
__global__ void __launch_bounds__(kRgbThreads, VLG_RGB_MIN_BLOCKS) rgb_strip_kernel(const RgbParams p) {
    const CoordCfg &cc = p.cc;
    const int H = cc.H, W = cc.W;
    const int lane = threadIdx.x & 31;
    // broadcast from lane 0: tells the compiler the warp index (hence all loop control) is warp-uniform
    const int gw = blockIdx.x * (kRgbThreads / 32) + __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    int64_t rho = (int64_t)gw * p.chunk;
    const int64_t rho_end = min(rho + p.chunk, p.total_rows);
    const unsigned FULL = 0xffffffffu;

    float s_l1 = 0.f, s_gd = 0.f, s_ssim = 0.f, m_grad = 0.f;
#ifdef VLG_PROFILE_TAIL
    if (lane == 0) prof_mark(p.hdr->prof, false);
#endif

    const float inv9 = 1.0f / 9.0f, C1 = 1e-4f, C2 = 9e-4f;
    const float kk = -p.tc.c_ssim * (2.0f / 9.0f);

    while (rho < rho_end) {
        // ---- one segment: rows [ya, yb) of strip s of image n ----
        const int colid = (int)(rho / H);
        const int ya = (int)(rho - (int64_t)colid * H);
        const int yb = (int)min((int64_t)H, (int64_t)ya + (rho_end - rho));
        rho += yb - ya;
        const int n = colid / p.strips, s = colid - n * p.strips;

        const int x = s * kRS - 2 + lane;
        const bool col_ok = x >= 0 && x < W;
        const bool out_lane = lane >= 2 && lane < 30 && x < W;
        const int xc = min(max(x, 0), W - 1);
        const float bxv = base_coord(xc, cc.Wm1);
        const float cR = (col_ok && x + 1 < W) ? p.tc.c_gd : 0.f;   // pair (x, x+1) exists
        const float cV = col_ok ? p.tc.c_gd : 0.f;
        const float mR = (out_lane && x + 1 < W) ? 1.f : 0.f;       // this lane counts the pair (x, x+1)
        const bool win_x = x >= 1 && x <= W - 2;                    // a 3x3 window can be centred on column x
        const int64_t img = (int64_t)n * H * W;
        const T *src = reinterpret_cast<const T *>(p.src_rgb) + img * 3;
        const T *tgt = reinterpret_cast<const T *>(p.tgt_rgb) + img * 3;
        const float2 *coords = reinterpret_cast<const float2 *>(p.coords) + img;
        const int t_last = yb + 1;

        // sliding state: index 1 = row t-1, index 2 = row t-2
        float a1[3] = {0.f, 0.f, 0.f}, b1[3] = {0.f, 0.f, 0.f}, a2[3] = {0.f, 0.f, 0.f}, b2[3] = {0.f, 0.f, 0.f};
        // vertical 3-sums are formed as (row t-2 + row t-1) + row t: the pair sum of the two previous rows is carried
        // instead of row t-2 itself (same association, one register move less per quantity and row)
        float2 hs1[3], hsP[3], hq1[3], hqP[3];     // horizontal 3-sums of (a,b) and (a^2,b^2): row t-1, rows (t-2) + (t-1)
        float hx1[3], hxP[3];                       // ... and of a*b
        float QA1[3], QB1[3], QC1[3], QAP[3], QBP[3], QCP[3];   // horizontal 3-sums of the window coefficients
        float G1[3], G2[3];                         // partial d(loss)/d(a) of rows t-1, t-2
        float Dx1[3], Dy1[3], Dx2[3], Dy2[3];       // d(a)/d(coord) of rows t-1, t-2 (mask and scale folded in)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            hs1[c] = hsP[c] = hq1[c] = hqP[c] = make_float2(0.f, 0.f);
            hx1[c] = hxP[c] = 0.f;
            QA1[c] = QB1[c] = QC1[c] = QAP[c] = QBP[c] = QCP[c] = 0.f;
            G1[c] = G2[c] = 0.f;
            Dx1[c] = Dy1[c] = Dx2[c] = Dy2[c] = 0.f;
        }

        auto load_flow = [&](int t) -> float2 {
            return (t >= 0 && t < H && t <= t_last) ? __ldg(coords + (t * W + xc)) : make_float2(0.f, 0.f);
        };

        int t = ya - 2;
        float2 fl_next = load_flow(t + 1);
        RgbRow cur;
        rgb_issue_row<T, BORDER>(cur, cc, load_flow(t), bxv, t, xc, src, tgt, t >= 0 && t < H);

        // One row of the pipeline.  STEADY rows are those for which every ownership / image-border condition below holds
        // (rows t-2 .. t owned, t-2 .. t+2 inside the image and the segment): ~87 % of the rows of a 44-row segment run
        // the instantiation in which these conditions are compile-time constants; the first and last rows of a segment
        // run the general one.
        auto row_step = [&](auto steady_tag, const int t) {
            constexpr bool ST = decltype(steady_tag)::value;
            // ---- row t ----
            const bool row_ok = ST || (t >= 0 && t < H);
            const bool live = row_ok && col_ok;
            const bool own0 = ST || (t >= ya && t < yb), own1 = ST || (t - 1 >= ya && t - 1 < yb), own2 = ST || (t - 2 >= ya && t - 2 < yb);
            const bool vpair = ST || (t >= 1 && t < H);              // rows t-1 and t are both image rows
            const bool win_y = ST || (t >= 2 && t <= H - 1);         // a window can be centred on row t-1
            const float mo0 = (own0 && out_lane) ? 1.f : 0.f, mo1 = (own1 && out_lane) ? 1.f : 0.f;
            const float mR0 = own0 ? mR : 0.f;
            const bool winv = win_x && win_y;
            const float mw1 = winv ? mo1 : 0.f;       // this lane counts the window centred on (x, t-1)

            float a0[3], b0[3], G0[3], Dx0[3], Dy0[3];
            float QA0[3], QB0[3], QC0[3];
            float2 hs0[3], hq0[3];
            float hx0[3];
            {
                const float wx1 = cur.wx1, wy1 = cur.wy1, wx0 = 1.0f - wx1, wy0 = 1.0f - wy1;
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float v0 = (BORDER || (cur.tin & 1u)) ? cur.v[0][c] : 0.f, v1 = (BORDER || (cur.tin & 2u)) ? cur.v[1][c] : 0.f;
                    const float v2 = (BORDER || (cur.tin & 4u)) ? cur.v[2][c] : 0.f, v3 = (BORDER || (cur.tin & 8u)) ? cur.v[3][c] : 0.f;
                    float acc = __fmul_rn(v0, cur.nw);
                    acc = __fmaf_rn(v1, cur.ne, acc);
                    acc = __fmaf_rn(v2, cur.sw, acc);
                    acc = __fmaf_rn(v3, cur.se, acc);
                    a0[c] = live ? acc : 0.f;
                    b0[c] = live ? cur.b[c] : 0.f;
                    if (GRAD) {
                        Dx0[c] = live ? cur.mx * ((v1 - v0) * wy0 + (v3 - v2) * wy1) : 0.f;
                        Dy0[c] = live ? cur.my * ((v2 - v0) * wx0 + (v3 - v1) * wx1) : 0.f;
                    }
                }
            }
            // ---- software pipeline: the raw taps of row t are consumed -- the taps + target of row t+1 are loaded into the
            // same registers (no second row buffer, no copy) and travel while the rest of this iteration computes; the flow of
            // row t+2 follows ----
            rgb_issue_row<T, BORDER>(cur, cc, fl_next, bxv, t + 1, xc, src, tgt, ST || (t + 1 >= 0 && t + 1 < H && t + 1 <= t_last));
            fl_next = ST ? __ldg(coords + ((t + 2) * W + xc)) : load_flow(t + 2);

#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float a = a0[c], b = b0[c];
                const float al = __shfl_up_sync(FULL, a, 1), ar = __shfl_down_sync(FULL, a, 1);
                const float bl = __shfl_up_sync(FULL, b, 1), br = __shfl_down_sync(FULL, b, 1);
                // L1
                const float d = a - b;
                s_l1 = fmaf(fabsf(d), mo0, s_l1);
                float g = signed_c1(p.tc.c_l1, d);
                // GD along W (reference `yloss`, src/loss.py:23-24): pairs (x, x+1) and (x-1, x)
                {   // each lane evaluates its pair (x, x+1) once; the right neighbour receives the gradient by a shuffle
                    const float da = ar - a, tt = fabsf(da) - fabsf(br - b);
                    s_gd = fmaf(fabsf(tt), mR0, s_gd);
                    const float gr = signed_c(cR, tt, da);
                    g += __shfl_up_sync(FULL, gr, 1) - gr;
                }
                // GD along H (reference `xloss`, src/loss.py:21-22): pair (t-1, t), counted by the owner of row t-1
                if (vpair) {
                    const float da = a - a1[c], tt = fabsf(da) - fabsf(b - b1[c]);
                    s_gd = fmaf(fabsf(tt), mo1, s_gd);
                    const float gv = signed_c(cV, tt, da);
                    g += gv;
                    G1[c] -= gv;
                }
                G0[c] = g;
                // horizontal 3-sums of row t
                const float2 pl = make_float2(al, bl), pc = make_float2(a, b), pr = make_float2(ar, br);
                hs0[c] = __fadd2_rn(__fadd2_rn(pl, pc), pr);
                hq0[c] = __ffma2_rn(pr, pr, __ffma2_rn(pc, pc, __fmul2_rn(pl, pl)));
                hx0[c] = fmaf(ar, br, fmaf(a, b, al * bl));
                // SSIM window centred on (x, t-1): rows t-2, t-1, t
                const float2 S1 = __fadd2_rn(hsP[c], hs0[c]);
                const float2 S2 = __fadd2_rn(hqP[c], hq0[c]);
                const float Sxy = hxP[c] + hx0[c];
                const float2 inv9_2 = make_float2(inv9, inv9);
                const float2 m2 = __fmul2_rn(S1, inv9_2);                           // (mu_x, mu_y)
                const float2 mm = __fmul2_rn(m2, m2);
                const float2 var = __ffma2_rn(S2, inv9_2, make_float2(-mm.x, -mm.y));
                const float mxy = m2.x * m2.y;
                const float vxy = fmaf(Sxy, inv9, -mxy);
                const float n1 = fmaf(2.f, mxy, C1), n2 = fmaf(2.f, vxy, C2);
                const float d1 = mm.x + mm.y + C1, d2 = var.x + var.y + C2;
                const float inv_d1 = rcp_approx(d1), inv_d2 = rcp_approx(d2);
                const float r = inv_d1 * inv_d2;
                const float S = (n1 * n2) * r;
                const float v = fmaf(-0.5f, S, 0.5f);
                s_ssim = fmaf(__saturatef(v), mw1, s_ssim);
                if (GRAD) {
                    // dS/dx_p = A + B x_p + C y_p (DESIGN.md section 4); the clamp passes gradient on [0, 1]
                    const float kke = (winv && v >= 0.0f && v <= 1.0f) ? kk : 0.f;
                    const float kA = kke * (m2.y * (n2 - n1) * r + S * m2.x * (inv_d2 - inv_d1));
                    const float kB = kke * (-S * inv_d2);
                    const float kC = kke * (n1 * r);
                    QA0[c] = (__shfl_up_sync(FULL, kA, 1) + kA) + __shfl_down_sync(FULL, kA, 1);
                    QB0[c] = (__shfl_up_sync(FULL, kB, 1) + kB) + __shfl_down_sync(FULL, kB, 1);
                    QC0[c] = (__shfl_up_sync(FULL, kC, 1) + kC) + __shfl_down_sync(FULL, kC, 1);
                }
            }

            // ---- gradient of row t-2 is complete ----
            if (GRAD && own2) {
                float dr[3];
                float gx = 0.f, gy = 0.f;
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float sA = QAP[c] + QA0[c], sB = QBP[c] + QB0[c];
                    const float sC = QCP[c] + QC0[c];
                    dr[c] = G2[c] + fmaf(sC, b2[c], fmaf(sB, a2[c], sA));
                    gx = fmaf(dr[c], Dx2[c], gx);
                    gy = fmaf(dr[c], Dy2[c], gy);
                    m_grad = fmaxf(m_grad, out_lane ? fabsf(dr[c]) : 0.f);
                }
                if (out_lane) {
                    const int64_t o = img + (int64_t)(t - 2) * W + x;
                    if (p.d_out_rgb) store_px<float, 3>(p.d_out_rgb + (((int64_t)n * H + (t - 2)) * p.pitch + x) * 3, dr);
                    if (p.d_coords) reinterpret_cast<float2 *>(p.d_coords)[o] = make_float2(gx, gy);
                }
            }

            // ---- slide ----
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                a2[c] = a1[c]; b2[c] = b1[c]; a1[c] = a0[c]; b1[c] = b0[c];
                hsP[c] = __fadd2_rn(hs1[c], hs0[c]); hs1[c] = hs0[c];
                hqP[c] = __fadd2_rn(hq1[c], hq0[c]); hq1[c] = hq0[c];
                hxP[c] = hx1[c] + hx0[c]; hx1[c] = hx0[c];
                if (GRAD) {
                    QAP[c] = QA1[c] + QA0[c]; QA1[c] = QA0[c];
                    QBP[c] = QB1[c] + QB0[c]; QB1[c] = QB0[c];
                    QCP[c] = QC1[c] + QC0[c]; QC1[c] = QC0[c];
                    G2[c] = G1[c]; G1[c] = G0[c];
                    Dx2[c] = Dx1[c]; Dx1[c] = Dx0[c]; Dy2[c] = Dy1[c]; Dy1[c] = Dy0[c];
                }
            }
        };
        // steady rows: t-2 >= ya, t < yb, t >= 2, t+2 < H (then t+2 <= t_last = yb+1 holds too)
        const int steady_begin = max(ya + 2, 2), steady_end = min(yb, H - 2);
#pragma unroll 1
        for (; t <= t_last && t < steady_begin; ++t) row_step(std::false_type{}, t);
#pragma unroll 1
        for (; t < steady_end; ++t) row_step(std::true_type{}, t);
#pragma unroll 1
        for (; t <= t_last; ++t) row_step(std::false_type{}, t);
    }

    // ---- per-warp partial sums (fixed order: the final reduction walks the rows by index; it also reads the slot of a
    // masked-off term as 0) ----
    s_l1 = warp_sum(s_l1);
    s_gd = warp_sum(s_gd);
    s_ssim = warp_sum(s_ssim);
    m_grad = warp_max(m_grad);
    if (lane == 0) {
        float4 o;
        o.x = s_l1;
        o.y = s_gd;
        o.z = s_ssim;
        o.w = 0.f;
#ifdef VLG_PROFILE_TAIL
        o.w = __uint_as_float(prof_stamp());     // where and when this warp finished
#endif
        reinterpret_cast<float4 *>(p.partials)[gw] = o;
        if (m_grad > 0.f) atomicMax(&p.hdr->maxgrad_rgb_bits, __float_as_uint(m_grad));
        if (gw == 0) p.hdr->n_rgb = gridDim.x * (kRgbThreads / 32);
    }

}

}  // namespace vlg
