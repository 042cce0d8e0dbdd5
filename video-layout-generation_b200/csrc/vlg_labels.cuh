// vlg_labels.cuh -- the layout half of pass 1 when the layout SOURCE is a label map (SURVEY 8f-2).
//
// In the reference the layout fed to the generator is always one_hot(label): `transform_seg_one_hot`
// (src/models/net_utils.py:14-24), the rollout feedback `argmax -> next input` (src/trainer.py:461,467),
// and the sources are DATA (frames and class maps from the dataset, src/folder.py:85-104): no gradient
// flows to them.  For a 0/1 source the K-channel bilinear gather collapses: the warped layout is
//     z_c = sum of the tap weights whose tap carries class c          (at most 4 non-zero channels)
// through the same chain as the dense path (fmul for the nw tap, then three fmas, Appendix A.6), so
//   argmax        bit-exact with argmax(warp(one_hot(label)))  (src/trainer.py:342; first maximal index)
//   CE            log(sum_c e^{z_c}) - z_label with (K - #distinct) channels at exactly 0  (src/trainer.py:124,250)
//   d CE / d z_c  cce * (softmax_c - [c == label]); the coordinate gradient only needs it at the four
//                 tap classes:  sum_c g_c v_tap,c = g_{label(tap)}
// Per pixel: 8 B of source labels' worth of gathers instead of an 80-byte pixel x 4 taps from shared memory,
// ~150 instructions instead of ~870, no d_src_layout (labels are not differentiable) and no pass 2.
// TV on the flow (absent upstream; stencils of src/loss.py:22,24) and the sum with the rgb part of
// d(loss)/d(coords) written by rgb_strip_kernel are as in lay_tile_kernel.
#pragma once
#include "vlg_device.cuh"
#include "vlg_pass1.cuh"   // signed_c1

namespace vlg {

struct LabParams {
    CoordCfg cc;
    int K;
    int64_t P, HW;
    const int64_t *src_label;      // [N,H,W] class ids of the source layout (values outside [0,K) warp as an all-zero pixel)
    const float2 *coords;
    const int64_t *tgt_label;
    int64_t ignore_index;
    const float *class_weight;
    TermCoeffs tc;                 // w_ce_over_scale, weighted_denom, c_tvh, c_tvw; TV runs when terms has VLG_TERM_TV
    int accum_dcoords;             // d_coords already holds the rgb part (the rgb strip kernel ran before): add to it
    float *d_coords;               // nullable (validation)
    int64_t *out_argmax;           // nullable
    float *partials;               // [gridDim.x][4]: ce, tv_h, tv_w, -
    ReduceParams red;
    WsHeader *hdr;
};

constexpr int kLabThreads = 256;

template <bool GRAD>
__global__ void __launch_bounds__(kLabThreads) lab_pix_kernel(const LabParams p) {
    __shared__ double s_red[6 * kLabThreads];
    __shared__ float s_part[kLabThreads / 32][4];
    __shared__ int s_last;
    const CoordCfg &cc = p.cc;
    const int H = cc.H, W = cc.W, K = p.K;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const float L2E = 1.4426950408889634f;
    const float denom = GRAD ? ce_divisor(p.tc, p.hdr) : 1.0f;
    const float ce_unit = GRAD ? p.tc.w_ce_over_scale / denom : 0.f;
    float s_ce = 0.f, s_tvh = 0.f, s_tvw = 0.f, m_disp = 0.f;
    bool bad = false;

    // contiguous run of pixels per CTA, consecutive threads on consecutive pixels (coalesced flow / label / d_coords)
    const int64_t per_cta = (p.P + gridDim.x - 1) / gridDim.x;
    const int64_t i0 = (int64_t)blockIdx.x * per_cta, i1 = min(p.P, i0 + per_cta);
    for (int64_t i = i0 + threadIdx.x; i < i1; i += kLabThreads) {
        // N*H*W < 2^31 (check_problem): 32-bit divisions (a 64-bit division by a run-time value costs ~60 instructions)
        const unsigned nu = (unsigned)i / (unsigned)p.HW, rem = (unsigned)i - nu * (unsigned)p.HW;
        const int64_t n = nu;
        const int y = (int)(rem / (unsigned)W), x = (int)(rem - (unsigned)y * (unsigned)W);
        const float2 f = __ldg(p.coords + i);
        const Taps t = make_taps(cc, f, y, x);
        const int64_t lb = __ldg(p.tgt_label + i);
        const float2 dc = (GRAD && p.accum_dcoords) ? __ldcg(reinterpret_cast<const float2 *>(p.d_coords) + i) : make_float2(0.f, 0.f);
        m_disp = fmaxf(m_disp, tap_displacement(cc, t, y, x));

        // the four taps' classes (-1: tap outside the image or class id outside [0,K): contributes nothing)
        const int64_t *lab_img = p.src_label + n * p.HW;
        int lab[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int xs = t.x0 + (k & 1), ys = t.y0 + (k >> 1);
            int64_t l = -1;
            if (xs >= 0 && xs < W && ys >= 0 && ys < H) l = __ldg(lab_img + (int64_t)ys * W + xs);
            lab[k] = (l >= 0 && l < K) ? (int)l : -1;
        }
        const float ws[4] = {t.nw, t.ne, t.sw, t.se};
        // z of class c through the dense path's chain (fmul for the nw tap, then three fmas)
        auto z_of = [&](int c) -> float {
            float z = __fmul_rn(lab[0] == c ? 1.0f : 0.0f, ws[0]);
            z = __fmaf_rn(lab[1] == c ? 1.0f : 0.0f, ws[1], z);
            z = __fmaf_rn(lab[2] == c ? 1.0f : 0.0f, ws[2], z);
            z = __fmaf_rn(lab[3] == c ? 1.0f : 0.0f, ws[3], z);
            return z;
        };
        float zt[4];
        bool first[4];
        int nd = 0;
        float m = 0.0f;                                // the absent classes sit at exactly 0 and nd <= 4 < K
        float best_z = 0.0f;
        int best_c = 0;                                // all-zero pixel: first maximal index is class 0
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c = lab[k];
            bool fst = c >= 0;
#pragma unroll
            for (int j = 0; j < k; ++j) fst = fst && lab[j] != c;
            first[k] = fst;
            zt[k] = c >= 0 ? z_of(c) : 0.0f;
            if (fst) {
                ++nd;
                m = fmaxf(m, zt[k]);
                if (zt[k] > best_z || (zt[k] == best_z && c < best_c)) { best_z = zt[k]; best_c = c; }
            }
        }
        if (p.out_argmax) p.out_argmax[i] = best_c;

        const bool lab_ok = lb >= 0 && lb < K;
        if (!lab_ok && lb != p.ignore_index) bad = true;
        const int il = lab_ok ? (int)lb : -2;
        const float wl = (lab_ok && p.class_weight) ? __ldg(p.class_weight + il) : 1.0f;
        const float ml2 = m * L2E;
        float et[4];
        float se = (float)(K - nd) * ex2_approx(-ml2);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            et[k] = ex2_approx(fmaf(zt[k], L2E, -ml2));
            if (first[k]) se += et[k];
        }
        const float zl = lab_ok ? z_of(il) : 0.0f;
        if (lab_ok) s_ce += wl * (fmaf(lg2_approx(se), 0.6931471805599453f, m) - zl);

        float gx = dc.x, gy = dc.y;
        if (GRAD) {
            const float cce = lab_ok ? ce_unit * wl : 0.0f;
            const float inv = cce * rcp_approx(se);
            float d4[4];                                 // sum_c g_c v_tap,c = g at the tap's class (0 for a tap that carries nothing)
#pragma unroll
            for (int k = 0; k < 4; ++k) d4[k] = lab[k] >= 0 ? fmaf(et[k], inv, lab[k] == il ? -cce : 0.0f) : 0.0f;
            const float wx1 = t.ix - t.fx0, wx0 = (t.fx0 + 1.0f) - t.ix;
            const float wy1 = t.iy - t.fy0, wy0 = (t.fy0 + 1.0f) - t.iy;
            const float gix = (d4[1] - d4[0]) * wy0 + (d4[3] - d4[2]) * wy1;
            const float giy = (d4[2] - d4[0]) * wx0 + (d4[3] - d4[1]) * wx1;
            gx = fmaf(t.mx, gix, gx);
            gy = fmaf(t.my, giy, gy);
        }
        if (p.tc.terms & VLG_TERM_TV) {
            const float2 *ci = p.coords + i;
            const bool hD = y + 1 < H, hU = y >= 1, hR = x + 1 < W, hL = x >= 1;
            const float2 fdn = hD ? __ldg(ci + W) : f, fup = hU ? __ldg(ci - W) : f;
            const float2 frt = hR ? __ldg(ci + 1) : f, flt = hL ? __ldg(ci - 1) : f;
            const float cD = hD ? p.tc.c_tvh : 0.f, cU = hU ? p.tc.c_tvh : 0.f, cR = hR ? p.tc.c_tvw : 0.f, cL = hL ? p.tc.c_tvw : 0.f;
            const float2 dd = make_float2(fdn.x - f.x, fdn.y - f.y), du = make_float2(f.x - fup.x, f.y - fup.y);
            const float2 dr = make_float2(frt.x - f.x, frt.y - f.y), dl = make_float2(f.x - flt.x, f.y - flt.y);
            s_tvh = fmaf(fabsf(dd.x) + fabsf(dd.y), hD ? 1.f : 0.f, s_tvh);
            s_tvw = fmaf(fabsf(dr.x) + fabsf(dr.y), hR ? 1.f : 0.f, s_tvw);
            gx += (signed_c1(cU, du.x) - signed_c1(cD, dd.x)) + (signed_c1(cL, dl.x) - signed_c1(cR, dr.x));
            gy += (signed_c1(cU, du.y) - signed_c1(cD, dd.y)) + (signed_c1(cL, dl.y) - signed_c1(cR, dr.y));
        }
        if (GRAD && p.d_coords) reinterpret_cast<float2 *>(p.d_coords)[i] = make_float2(gx, gy);
    }

    // ---- per-CTA partial sums (fixed order: lanes by shuffle tree, warps by index) ----
    s_ce = warp_sum(s_ce); s_tvh = warp_sum(s_tvh); s_tvw = warp_sum(s_tvw);
    m_disp = warp_max(m_disp);
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(&p.hdr->status, VLG_STATUS_BAD_LABEL);
    if (lane == 0) {
        s_part[wid][0] = s_ce; s_part[wid][1] = s_tvh; s_part[wid][2] = s_tvw;
        if (m_disp > 0.f) atomicMax(&p.hdr->maxdisp_bits, __float_as_uint(m_disp));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int w = 0; w < kLabThreads / 32; ++w) { o.x += s_part[w][0]; o.y += s_part[w][1]; o.z += s_part[w][2]; }
        reinterpret_cast<float4 *>(p.partials)[blockIdx.x] = o;
        if (blockIdx.x == 0) p.hdr->n_lay = gridDim.x;
        __threadfence();
    }
    if (p.red.out != nullptr) {
        __syncthreads();
        if (threadIdx.x == 0) s_last = atomicAdd(&p.hdr->blocks_done, 1u) == gridDim.x - 1;
        __syncthreads();
        if (s_last) {
            __threadfence();
            reduce_partials_block<kLabThreads>(p.red, s_red);
        }
    }
}

}  // namespace vlg
