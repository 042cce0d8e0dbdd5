// vlg_laytile.cuh -- the layout half of pass 1 as a PERSISTENT, double-buffered tile kernel.
//
// What it computes (reference gongaa/video-layout-generation):
//   warp of the K-channel layout  (absent upstream) F.grid_sample(bilinear, align_corners=True) on
//                                 the src/models/modules.py:69 grid, bit-exact FMA chain (App. A.6)
//   argmax layouts                src/trainer.py:342,423,467 (first maximal index)
//   CE                            src/trainer.py:124,250
//   TV on the flow                (absent upstream) stencils of src/loss.py:22,24
// plus d(loss)/d(warped layout), the layout + TV part of d(loss)/d(coords) and pass 2's bookkeeping.
//
// Why this organisation.  Measured on B200 (profiles/): a warp of this path runs at ~6 cycles per
// instruction whatever else the SM does (in-order issue, LDS / MUFU / integer chains), so throughput
// is (resident warps) / (instructions per pixel).  A per-warp strip kernel with a TMA row ring (round 1,
// dropped) paid ~250 instructions of ring bookkeeping per 32 pixels and its 16 KB ring per warp capped the
// SM at 12 warps; the first tile kernel (vlg_pass1.cuh) amortised the bookkeeping over 256 pixels but
// exposed three dependent global round trips per CTA.  This kernel keeps the tile (one TMA window per
// 32x8 pixels, 4.8 KB per warp) and removes the exposed latency with a software pipeline over the CTA's tiles:
//   iteration i:  issue the TMA window of tile i+1 (origin from sums accumulated during iteration i-1)
//                 issue the loads of tile i+3's coordinates / tile i+1's labels
//                 wait for tile i's window, compute tile i
//                 accumulate the window origin of tile i+2, publish tile i+1's flow block for the TV stencil
//                 ONE __syncthreads
// Loaded values are only ever consumed one iteration after their load was issued.
#pragma once
#include <cuda.h>

#include "vlg_device.cuh"
#include "vlg_pass1.cuh"   // mbarrier / TMA helpers, source_xy, taps_from_xy

namespace vlg {

// four consecutive channels from shared memory as fp32 (one 128-bit / 64-bit load)
template <typename T> __device__ __forceinline__ float4 load4_smem(const T *p);
template <> __device__ __forceinline__ float4 load4_smem<float>(const float *p) { return *reinterpret_cast<const float4 *>(p); }
template <> __device__ __forceinline__ float4 load4_smem<__nv_bfloat16>(const __nv_bfloat16 *p) {
    const uint2 r = *reinterpret_cast<const uint2 *>(p);
    const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162 *>(&r.x), hi = *reinterpret_cast<const __nv_bfloat162 *>(&r.y);
    const float2 a = __bfloat1622float2(lo), b = __bfloat1622float2(hi);
    return make_float4(a.x, a.y, b.x, b.y);
}

// four consecutive channels from global memory (read-only path) as fp32
template <typename T> __device__ __forceinline__ float4 load4_global(const T *p);
template <> __device__ __forceinline__ float4 load4_global<float>(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }
template <> __device__ __forceinline__ float4 load4_global<__nv_bfloat16>(const __nv_bfloat16 *p) {
    const uint2 r = __ldg(reinterpret_cast<const uint2 *>(p));
    const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162 *>(&r.x), hi = *reinterpret_cast<const __nv_bfloat162 *>(&r.y);
    const float2 a = __bfloat1622float2(lo), b = __bfloat1622float2(hi);
    return make_float4(a.x, a.y, b.x, b.y);
}

constexpr int kLayMaxWarps = 8192;    // partial-sum rows reserved in the workspace (one per CTA of the persistent grid)

struct LayParams {
    CoordCfg cc;
    int N, strips;                 // strips = ceil(W / kTW)
    int tiles_y;                   // ceil(H / kTH) (tile geometry of pass 2)
    int64_t total_rows, chunk;
    const void *src_layout;
    const float *coords;
    const int64_t *label;
    int64_t ignore_index;
    const float *class_weight;
    TermCoeffs tc;                 // w_ce_over_scale, weighted_denom, c_tvh, c_tvw; TV runs when terms has VLG_TERM_TV
    int accum_dcoords;             // d_coords already holds the rgb part (the rgb strip kernel ran before): add to it
    float *d_coords;               // nullable (validation)
    float *d_out_lay;              // [P][K] fp32 staging, nullable
    uint32_t *rec_code;            // [N][H][pitch] tap records for pass 2 (tap_cell_code), nullable
    float2 *rec_frac;              // [N][H][pitch] fractional tap weights (ix - x0, iy - y0)
    int pitch;
    int64_t *out_argmax;           // nullable
    float *partials;               // [n_ctas][4]: ce, tv_h, tv_w, -
    float *tile_disp;              // [n_tiles] max NEAR displacement per 32x8 tile (zero-initialised, atomicMax)
    int4 *far_list;                // queue of far output pixels (see Pass2Params::far_list)
    uint32_t *tile_flags;
    uint32_t *seg_cnt;             // [n_tiles][kTH] far output pixels per row of a SOURCE tile (zeroed with the header)
    int *flagged_list;
    ReduceParams red;
    WsHeader *hdr;
};

constexpr int kTSW = 40, kTSH = 12;   // staged window (pixels)
constexpr int kFW = kTW + 2, kFH = kTH + 2;   // flow block with a halo of one pixel (TV stencil)
#ifndef VLG_LAYTILE_MIN_BLOCKS
#define VLG_LAYTILE_MIN_BLOCKS 2
#endif

template <typename T, int K>
struct LayTileSmem {
    alignas(128) T win[2][kTSH * kTSW * K];
    alignas(128) float obuf[kTH][kTW * K];     // one output row of d(loss)/d(warped layout) per warp
    float2 flow[4][kFH * kFW];                  // tile i lives in flow[i & 3]: published two tiles ahead, no CTA barrier
    alignas(8) uint64_t bar[2];
    int acc[2][4];                              // sum of (x0 - x), sum of (y0 - y), pixels counted
    int org[2][2];                              // window origin (ox, oy)
    unsigned cnt[2];                            // warps that have finished the tile using window buffer b
    float red[kTH][4];
    int last;
    int seen[kFarSeen];                         // tiles this CTA has already flagged as far targets (far_announce)
};

// PX8: the tensor map describes rows of 8-byte units (pixels whose byte size is not a multiple of 16, e.g.
// 20 bf16 channels = 40 B): 3-D map {W*PXB/8, H, N}, window origin scaled by PXB/8.
template <typename T, int K, bool GRAD, bool PX8>
__global__ void __launch_bounds__(kThreads, VLG_LAYTILE_MIN_BLOCKS) lay_tile_kernel(const LayParams p,
                                                                                   const __grid_constant__ CUtensorMap win_map) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    LayTileSmem<T, K> &sm = *reinterpret_cast<LayTileSmem<T, K> *>(smem_raw);
    const CoordCfg &cc = p.cc;
    const int H = cc.H, W = cc.W;
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31;
    const int wid = __shfl_sync(FULL, tid >> 5, 0);
    constexpr unsigned kWinBytes = (unsigned)(kTSH * kTSW * K * sizeof(T));
    constexpr int PXB = K * (int)sizeof(T);
    const int tiles_x = p.strips, tiles_y = p.tiles_y;
    const int tiles_img = tiles_x * tiles_y;

    // contiguous run of tiles (column-major inside an image) per CTA
    const int64_t n_tiles = (int64_t)p.N * tiles_img;
    const int64_t per_cta = (n_tiles + gridDim.x - 1) / gridDim.x;
    const int64_t tau0 = (int64_t)blockIdx.x * per_cta;
    const int nt = (int)max((int64_t)0, min(per_cta, n_tiles - tau0));

    const float mx_c = (cc.coord_mode == VLG_COORD_FLOW) ? __fmul_rn(cc.Wm1, 0.5f) * cc.sx : __fmul_rn(cc.Wm1, 0.5f);
    const float my_c = (cc.coord_mode == VLG_COORD_FLOW) ? __fmul_rn(cc.Hm1, 0.5f) * cc.sy : __fmul_rn(cc.Hm1, 0.5f);
    const bool border = cc.padding == VLG_PAD_BORDER;
    const float denom = GRAD ? ce_divisor(p.tc, p.hdr) : 1.0f;
    const float ce_unit = GRAD ? p.tc.w_ce_over_scale / denom : 0.f;
    const float2 *coords_all = reinterpret_cast<const float2 *>(p.coords);
    const T *src_all = reinterpret_cast<const T *>(p.src_layout);

    float s_ce = 0.f, s_tvh = 0.f, s_tvw = 0.f, m_disp = 0.f, m_grad = 0.f;
    const float wreg = (p.class_weight && lane < K) ? __ldg(p.class_weight + lane) : 1.0f;   // class weights need K <= 32

    // Geometry of a tile, advanced incrementally: no divisions in the loop.  A CTA walks DOWN a column of
    // tiles (column-major inside an image): consecutive windows then share 4 of their 12 rows, which the
    // second fetch finds in L2 -- in row-major order those rows came from DRAM again (1.875x read
    // amplification measured as 306 MB of DRAM reads for 201 MB of inputs).
    struct TileGeo { int n, ty0, tx0; };
    auto advance = [&](TileGeo g) -> TileGeo {
        g.ty0 += kTH;
        if (g.ty0 >= tiles_y * kTH) { g.ty0 = 0; g.tx0 += kTW; if (g.tx0 >= tiles_x * kTW) { g.tx0 = 0; ++g.n; } }
        return g;
    };
    TileGeo g0;
    {
        g0.n = (int)(tau0 / tiles_img);
        const int rem = (int)(tau0 - (int64_t)g0.n * tiles_img);
        const int txi = rem / tiles_y;
        g0.tx0 = txi * kTW; g0.ty0 = (rem - txi * tiles_y) * kTH;
    }
    TileGeo g1 = advance(g0), g2 = advance(g1), g3 = advance(g2);

    // this thread's pixel of a tile (clamped into the image for the loads)
    auto px_index = [&](const TileGeo &g, int dy, int dx) -> int64_t {
        const int y = min(max(g.ty0 + dy, 0), H - 1), x = min(max(g.tx0 + dx, 0), W - 1);
        return (int64_t)g.n * H * W + (int64_t)y * W + x;
    };
    auto load_coords = [&](int i, const TileGeo &g) -> float2 {
        return i < nt ? __ldg(coords_all + px_index(g, wid, lane)) : make_float2(0.f, 0.f);
    };
    auto load_label = [&](int i, const TileGeo &g) -> int64_t { return i < nt ? __ldg(p.label + px_index(g, wid, lane)) : (int64_t)0; };
    // halo of the flow block (TV only): threads 0..83 own one halo cell each (top row, bottom row, left / right column)
    int hy = 0, hx = 0;                 // halo cell of this thread, relative to the tile origin
    const bool has_halo = tid < 2 * kFW + 2 * kTH;
    if (tid < kFW) { hy = -1; hx = tid - 1; }
    else if (tid < 2 * kFW) { hy = kTH; hx = tid - kFW - 1; }
    else if (tid < 2 * kFW + kTH) { hy = tid - 2 * kFW; hx = -1; }
    else { hy = tid - 2 * kFW - kTH; hx = kTW; }
    auto load_halo = [&](int i, const TileGeo &g) -> float2 {
        return (i < nt && has_halo && (p.tc.terms & VLG_TERM_TV)) ? __ldg(coords_all + px_index(g, hy, hx)) : make_float2(0.f, 0.f);
    };
    // sampling position of this thread's pixel + its contribution to the tile's window origin
    // (mean tap displacement of the tile: robust against a few outliers)
    auto sample_and_accumulate = [&](int i, const TileGeo &g, float2 fl, int buf) -> float2 {
        if (i >= nt) return make_float2(0.f, 0.f);
        const int y = g.ty0 + wid, x = g.tx0 + lane;
        const bool inside = y < H && x < W;
        float mx, my;
        const float2 xy = source_xy(cc, fl, base_coord(min(x, W - 1), cc.Wm1), base_coord(min(y, H - 1), cc.Hm1), mx, my);
        const int x0 = (int)fminf(fmaxf(floorf(xy.x), -4.0f), (float)W + 4.0f);
        const int y0 = (int)fminf(fmaxf(floorf(xy.y), -4.0f), (float)H + 4.0f);
        const int sdx = __reduce_add_sync(FULL, inside ? x0 - x : 0), sdy = __reduce_add_sync(FULL, inside ? y0 - y : 0);
        const int cnt = __popc(__ballot_sync(FULL, inside));
        if (lane == 0 && cnt) { atomicAdd(&sm.acc[buf][0], sdx); atomicAdd(&sm.acc[buf][1], sdy); atomicAdd(&sm.acc[buf][2], cnt); }
        return xy;
    };
    auto publish_flow = [&](int i, float2 fl, float2 fh, int buf) {
        if (i >= nt || !(p.tc.terms & VLG_TERM_TV)) return;
        sm.flow[buf][(wid + 1) * kFW + lane + 1] = fl;
        if (has_halo) sm.flow[buf][(hy + 1) * kFW + hx + 1] = fh;
    };
    // thread 0: origin of a tile's window from the accumulated sums, then its TMA load
    auto issue_window = [&](const TileGeo &g, int buf) {
        const int cnt = max(sm.acc[buf][2], 1);
        const int sx_ = sm.acc[buf][0], sy_ = sm.acc[buf][1];
        // floor division of the sums (C division truncates towards zero)
        const int mdx = (sx_ >= 0 ? sx_ : sx_ - cnt + 1) / cnt, mdy = (sy_ >= 0 ? sy_ : sy_ - cnt + 1) / cnt;
        int ox = g.tx0 + mdx - (kTSW - kTW - 2) / 2;
        const int oy = g.ty0 + mdy - (kTSH - kTH - 2) / 2;
        if (PX8 && (PXB % 16) != 0) ox &= ~1;   // TMA needs a 16-byte aligned start: 40-byte pixels -> even column
        sm.org[buf][0] = ox; sm.org[buf][1] = oy;
        sm.acc[buf][0] = 0; sm.acc[buf][1] = 0; sm.acc[buf][2] = 0;
        mbar_expect_tx(&sm.bar[buf], kWinBytes);
        if (PX8) tma_load_3d(sm.win[buf], &win_map, &sm.bar[buf], ox * (PXB / 8), oy, g.n);
        else tma_load_4d(sm.win[buf], &win_map, &sm.bar[buf], 0, ox, oy, g.n);
    };

    // ---------------- prologue ----------------
#ifdef VLG_PROFILE_TAIL
    if (tid == 0) prof_mark(p.hdr->prof + 4, false);
#endif
    if (tid < 2) { mbar_init(&sm.bar[tid], 1); sm.cnt[tid] = 0u; }
    if (tid < 8) sm.acc[tid >> 2][tid & 3] = 0;
    static_assert(kFarSeen == kThreads, "one entry per thread");
    sm.seen[tid] = -1;
    float2 f0 = load_coords(0, g0), f1 = load_coords(1, g1);
    float2 xy0, xy1;
    {
        const float2 h0 = load_halo(0, g0), h1 = load_halo(1, g1);
        __syncthreads();
        xy0 = sample_and_accumulate(0, g0, f0, 0);
        xy1 = sample_and_accumulate(1, g1, f1, 1);
        publish_flow(0, f0, h0, 0);
        publish_flow(1, f1, h1, 1);
    }
    __syncthreads();
    if (tid == 0 && nt > 0) issue_window(g0, 0);
    if (tid == 0 && nt > 1) issue_window(g1, 1);
    __syncthreads();
    float2 pend_f = load_coords(2, g2), pend_h = load_halo(2, g2);
    int64_t pend_lab = load_label(0, g0);
    // rgb part of d(loss)/d(coords), written by the rgb strip kernel that ran before: loaded one tile ahead
    auto load_dc = [&](int i, const TileGeo &g) -> float2 {
        const int y = g.ty0 + wid, x = g.tx0 + lane;
        return (GRAD && p.accum_dcoords && i < nt && y < H && x < W)
                   ? __ldcg(reinterpret_cast<const float2 *>(p.d_coords) + ((int64_t)g.n * H * W + (int64_t)y * W + x)) : make_float2(0.f, 0.f);
    };
    float2 pend_dc = load_dc(0, g0);

#pragma unroll 1
    for (int i = 0; i < nt; ++i) {
        const int b = i & 1;
        // ---- take over last iteration's loads, issue this iteration's ----
        const float2 f2 = pend_f, h2 = pend_h;   // coordinates / flow halo of tile i+2
        const int64_t lb = pend_lab;
        const float2 dc = pend_dc;
        pend_dc = load_dc(i + 1, g1);
        pend_f = load_coords(i + 3, g3);
        pend_h = load_halo(i + 3, g3);
        pend_lab = load_label(i + 1, g1);
        // ---- tile i ----
        const TileGeo g = g0;
        const int y = g.ty0 + wid, x = g.tx0 + lane;
        const bool inside = y < H && x < W;
        const int64_t img = (int64_t)g.n * H * W;
        const T *src_lay = src_all + img * K;
        const float2 xy = xy0;
        float mx = mx_c, my = my_c;
        if (border) {   // the clipped position tells whether the border clip was active
            mx = (xy.x <= 0.0f || xy.x >= cc.Wm1) ? 0.0f : mx;
            my = (xy.y <= 0.0f || xy.y >= cc.Hm1) ? 0.0f : my;
        }
        const Taps tp = taps_from_xy(cc, xy, mx, my);
        const int npx = min(kTW, W - g.tx0);

        // displacement bookkeeping for pass 2
        const float disp = inside ? tap_displacement(cc, tp, y, x) : 0.f;
        const bool is_far = disp >= (float)VLG_NEAR_RADIUS;
        m_disp = fmaxf(m_disp, disp);
        {
            const unsigned nmax = __reduce_max_sync(FULL, __float_as_uint(is_far ? 0.f : disp));
            if (lane == 0 && nmax != 0u) atomicMax(reinterpret_cast<unsigned *>(p.tile_disp) + ((g.n * tiles_y + g.ty0 / kTH) * tiles_x + g.tx0 / kTW), nmax);
        }
        if (is_far && p.d_out_lay != nullptr) {
            if (p.far_list) {
                p.far_list[atomicAdd(&p.hdr->far_count, 1u)] = make_int4((int)(img + (int64_t)y * W + x), (tp.x0 + 8) | ((tp.y0 + 8) << 16),
                                                                          __float_as_int(tp.ix - tp.fx0), __float_as_int(tp.iy - tp.fy0));
                far_announce(p.tile_flags, p.flagged_list, p.seg_cnt, p.hdr, g.n, tiles_x, tiles_y, tp.x0, tp.y0, W, H, sm.seen);
            } else {
                atomicOr(&p.hdr->status, VLG_STATUS_FAR_TAPS);
            }
        }

        if (GRAD && p.rec_code && inside) {   // tap record for pass 2: which source cell this pixel feeds, with which weights
            const int64_t ro = ((int64_t)g.n * H + y) * p.pitch + x;
            p.rec_code[ro] = tap_cell_code(cc, tp, y, x);
            p.rec_frac[ro] = make_float2(tp.ix - tp.fx0, tp.iy - tp.fy0);
        }

        const bool lab_ok = lb >= 0 && lb < K;
        if (inside && !lab_ok && lb != p.ignore_index) atomicOr(&p.hdr->status, VLG_STATUS_BAD_LABEL);
        const int il = lab_ok ? (int)lb : 0;
        // class weight of this pixel's label: lane k keeps weight k in a register (loaded once), so the loop has no
        // dependent global load -- a predicated-off LDG here still cost a long-scoreboard round trip (14 % of stalls)
        const float wl = __shfl_sync(FULL, wreg, il);

        mbar_wait(&sm.bar[b], (unsigned)((i >> 1) & 1));     // window of tile i has landed

        // Shared-memory bandwidth bounds this kernel (every organisation of the path tried ran at
        // ~2 cycles per shared-memory wavefront), so every tap is read ONCE: the channels are walked
        // in chunks of four with an online softmax (running maximum + rescaled accumulators), and the
        // sums sum_k e_k * v_tap,k the coordinate gradient needs are accumulated in the same sweep.
        float z[K];      // on exit: softmax part of d(loss)/d(warped layout) (cce * softmax_k)
        float vl[4];     // label channel of the four taps
        float zl, m, se, gix = 0.f, giy = 0.f, gl = 0.f;
        const float L2E = 1.4426950408889634f;
        const float cce = (GRAD && lab_ok && inside) ? ce_unit * wl : 0.0f;
        const T *st0 = nullptr;
        (void)src_lay;
        {
            const unsigned rx = (unsigned)(tp.x0 - sm.org[b][0]), ry = (unsigned)(tp.y0 - sm.org[b][1]);
            if (inside && rx < (unsigned)(kTSW - 1) && ry < (unsigned)(kTSH - 1)) st0 = sm.win[b] + (ry * kTSW + rx) * K;
        }
        // One sweep for both sources of the taps: ld4(tap, c) hands channels 4c .. 4c+3 of tap 0..3 (nw, ne, sw, se),
        // ld1(tap) its label channel.  Staged window: plain shared-memory loads (out-of-image cells hold the TMA's zeros).
        // Taps outside the window (rare for smooth flow, the rule for rough flow such as BASELINE config 5): the same
        // sweep on global loads, out-of-image taps read as zeros -- every tap is still fetched once.
        auto sweep = [&](auto ld4, auto ld1) {
            vl[0] = ld1(0); vl[1] = ld1(1); vl[2] = ld1(2); vl[3] = ld1(3);
            const float2 nw2 = make_float2(tp.nw, tp.nw), ne2 = make_float2(tp.ne, tp.ne);
            const float2 sw2 = make_float2(tp.sw, tp.sw), se2 = make_float2(tp.se, tp.se);
            float m_run = -3.0e38f;
            float mcs[K / 4];
            float2 Snw = make_float2(0.f, 0.f), Sne = Snw, Ssw = Snw, Sse = Snw;
            float bestv = -3.0e38f;
            int best = 0;
            se = 0.f;
#pragma unroll
            for (int c = 0; c < K / 4; ++c) {
                const float4 a = ld4(0, c), bq = ld4(1, c), cq = ld4(2, c), dq = ld4(3, c);
                // bit-exact FMA chain of Appendix A.6 on channel pairs
                float2 z01 = __fmul2_rn(make_float2(a.x, a.y), nw2), z23 = __fmul2_rn(make_float2(a.z, a.w), nw2);
                z01 = __ffma2_rn(make_float2(bq.x, bq.y), ne2, z01); z23 = __ffma2_rn(make_float2(bq.z, bq.w), ne2, z23);
                z01 = __ffma2_rn(make_float2(cq.x, cq.y), sw2, z01); z23 = __ffma2_rn(make_float2(cq.z, cq.w), sw2, z23);
                z01 = __ffma2_rn(make_float2(dq.x, dq.y), se2, z01); z23 = __ffma2_rn(make_float2(dq.z, dq.w), se2, z23);
                if (p.out_argmax) {   // first maximal index (src/trainer.py:342): strict comparisons in channel order
                    if (z01.x > bestv) { bestv = z01.x; best = 4 * c; }
                    if (z01.y > bestv) { bestv = z01.y; best = 4 * c + 1; }
                    if (z23.x > bestv) { bestv = z23.x; best = 4 * c + 2; }
                    if (z23.y > bestv) { bestv = z23.y; best = 4 * c + 3; }
                }
                const float m_new = fmaxf(fmaxf(m_run, fmaxf(z01.x, z01.y)), fmaxf(z23.x, z23.y));
                const float sc = ex2_approx((m_run - m_new) * L2E);     // 1 when the maximum did not move
                m_run = m_new; mcs[c] = m_new;
                const float ml2 = m_new * L2E;
                const float e0 = ex2_approx(fmaf(z01.x, L2E, -ml2)), e1 = ex2_approx(fmaf(z01.y, L2E, -ml2));
                const float e2 = ex2_approx(fmaf(z23.x, L2E, -ml2)), e3 = ex2_approx(fmaf(z23.y, L2E, -ml2));
                se = fmaf(se, sc, (e0 + e1) + (e2 + e3));
                z[4 * c] = e0; z[4 * c + 1] = e1; z[4 * c + 2] = e2; z[4 * c + 3] = e3;
                if (GRAD) {
                    const float2 sc2 = make_float2(sc, sc), e01 = make_float2(e0, e1), e23 = make_float2(e2, e3);
                    Snw = __ffma2_rn(make_float2(a.z, a.w), e23, __ffma2_rn(make_float2(a.x, a.y), e01, __fmul2_rn(Snw, sc2)));
                    Sne = __ffma2_rn(make_float2(bq.z, bq.w), e23, __ffma2_rn(make_float2(bq.x, bq.y), e01, __fmul2_rn(Sne, sc2)));
                    Ssw = __ffma2_rn(make_float2(cq.z, cq.w), e23, __ffma2_rn(make_float2(cq.x, cq.y), e01, __fmul2_rn(Ssw, sc2)));
                    Sse = __ffma2_rn(make_float2(dq.z, dq.w), e23, __ffma2_rn(make_float2(dq.x, dq.y), e01, __fmul2_rn(Sse, sc2)));
                }
            }
            m = m_run;
            zl = __fmaf_rn(vl[3], tp.se, __fmaf_rn(vl[2], tp.sw, __fmaf_rn(vl[1], tp.ne, __fmul_rn(vl[0], tp.nw))));
            if (p.out_argmax && inside) p.out_argmax[img + (int64_t)y * W + x] = best;
            if (GRAD) {
                const float inv = cce * rcp_approx(se);
#pragma unroll
                for (int c = 0; c < K / 4; ++c) {
                    const float fc = ex2_approx((mcs[c] - m) * L2E) * inv;   // brings the chunk to the final maximum
                    const float2 fc2 = make_float2(fc, fc);
                    const float2 r01 = __fmul2_rn(make_float2(z[4 * c], z[4 * c + 1]), fc2), r23 = __fmul2_rn(make_float2(z[4 * c + 2], z[4 * c + 3]), fc2);
                    z[4 * c] = r01.x; z[4 * c + 1] = r01.y; z[4 * c + 2] = r23.x; z[4 * c + 3] = r23.y;
                }
                gl = fmaf(ex2_approx((zl - m) * L2E), inv, -cce);
                const float dnw = fmaf(inv, Snw.x + Snw.y, -cce * vl[0]), dne = fmaf(inv, Sne.x + Sne.y, -cce * vl[1]);
                const float dsw = fmaf(inv, Ssw.x + Ssw.y, -cce * vl[2]), dse = fmaf(inv, Sse.x + Sse.y, -cce * vl[3]);
                const float wx1 = tp.ix - tp.fx0, wx0 = (tp.fx0 + 1.0f) - tp.ix;
                const float wy1 = tp.iy - tp.fy0, wy0 = (tp.fy0 + 1.0f) - tp.iy;
                gix = (dne - dnw) * wy0 + (dse - dsw) * wy1;
                giy = (dsw - dnw) * wx0 + (dse - dne) * wx1;
            }
        };
        if (st0) {
            const T *st1 = st0 + kTSW * K;
            sweep([&](int tap, int c) { return load4_smem<T>((tap & 2 ? st1 : st0) + (tap & 1) * K + 4 * c); },
                  [&](int tap) { return to_f<T>(((tap & 2) ? st1 : st0)[(tap & 1) * K + il]); });
        } else {
            const T *q0 = src_lay + ((int64_t)tp.y0 * W + tp.x0) * K, *q1 = q0 + (int64_t)W * K;
            const bool xin0 = tp.x0 >= 0 && tp.x0 < W, xin1 = tp.x0 + 1 >= 0 && tp.x0 + 1 < W;
            const bool yin0 = tp.y0 >= 0 && tp.y0 < H, yin1 = tp.y0 + 1 >= 0 && tp.y0 + 1 < H;
            const unsigned tin = (unsigned)(inside && yin0 && xin0) | ((unsigned)(inside && yin0 && xin1) << 1) |
                                 ((unsigned)(inside && yin1 && xin0) << 2) | ((unsigned)(inside && yin1 && xin1) << 3);
            sweep([&](int tap, int c) { return (tin >> tap) & 1u ? load4_global<T>((tap & 2 ? q1 : q0) + (tap & 1) * K + 4 * c) : make_float4(0.f, 0.f, 0.f, 0.f); },
                  [&](int tap) { return (tin >> tap) & 1u ? to_f<T>(__ldg(((tap & 2) ? q1 : q0) + (tap & 1) * K + il)) : 0.0f; });
        }
        if (lab_ok && inside) s_ce += wl * (fmaf(lg2_approx(se), 0.6931471805599453f, m) - zl);
        if (GRAD) {
            m_grad = fmaxf(m_grad, cce);
            if (p.d_out_lay && y < H) {   // warp-uniform: one contiguous row of d_out leaves through shared memory
                if (lane == 0) bulk_store_wait_read();
                __syncwarp();
                float *ob = sm.obuf[wid] + lane * K;
#pragma unroll
                for (int k = 0; k < K; k += 4) *reinterpret_cast<float4 *>(ob + k) = make_float4(z[k], z[k + 1], z[k + 2], z[k + 3]);
                if (lab_ok) ob[il] = gl;
                fence_async_smem();
                __syncwarp();
                if (lane == 0) bulk_store(p.d_out_lay + (img + (int64_t)y * W + g.tx0) * K, sm.obuf[wid], (unsigned)(npx * K * 4));
            }
        }

        // ---- coordinate gradient: layout part + TV ----
        float gx = fmaf(tp.mx, gix, dc.x), gy = fmaf(tp.my, giy, dc.y);
        if (p.tc.terms & VLG_TERM_TV) {
            const float2 *fc = &sm.flow[i & 3][(wid + 1) * kFW + lane + 1];
            const float2 f = f0, fdn = fc[kFW], fup = fc[-kFW], frt = fc[1], flt = fc[-1];
            const float cD = (inside && y + 1 < H) ? p.tc.c_tvh : 0.f, cU = (inside && y >= 1) ? p.tc.c_tvh : 0.f;
            const float cR = (inside && x + 1 < W) ? p.tc.c_tvw : 0.f, cL = (inside && x >= 1) ? p.tc.c_tvw : 0.f;
            const float2 dd = make_float2(fdn.x - f.x, fdn.y - f.y), du = make_float2(f.x - fup.x, f.y - fup.y);
            const float2 dr = make_float2(frt.x - f.x, frt.y - f.y), dl = make_float2(f.x - flt.x, f.y - flt.y);
            s_tvh = fmaf(fabsf(dd.x) + fabsf(dd.y), (inside && y + 1 < H) ? 1.f : 0.f, s_tvh);
            s_tvw = fmaf(fabsf(dr.x) + fabsf(dr.y), (inside && x + 1 < W) ? 1.f : 0.f, s_tvw);
            gx += (signed_c1(cU, du.x) - signed_c1(cD, dd.x)) + (signed_c1(cL, dl.x) - signed_c1(cR, dr.x));
            gy += (signed_c1(cU, du.y) - signed_c1(cD, dd.y)) + (signed_c1(cL, dl.y) - signed_c1(cR, dr.y));
        }
        if (GRAD && p.d_coords && inside) reinterpret_cast<float2 *>(p.d_coords)[img + (int64_t)y * W + x] = make_float2(gx, gy);

        // ---- prepare tile i+2: sampling positions, window origin sums, flow block ----
        const float2 xy2 = sample_and_accumulate(i + 2, g2, f2, b);
        publish_flow(i + 2, f2, h2, (i + 2) & 3);
        // No CTA barrier: the LAST warp to finish tile i (which used window buffer b) issues the window of
        // tile i+2 into that buffer.  Everything the other warps wrote for tile i+2 (origin sums, flow block)
        // is ordered before that TMA by their fence + the counter, and every reader of tile i+2 waits for
        // the TMA -- so warps may drift up to one tile apart instead of meeting at a barrier every tile.
        __syncwarp();
        if (lane == 0) {
            __threadfence_block();
            if (atomicAdd(&sm.cnt[b], 1u) == (unsigned)(kTH - 1)) {
                sm.cnt[b] = 0u;
                __threadfence_block();
                if (i + 2 < nt) issue_window(g2, b);
            }
        }
        f0 = f1; f1 = f2;
        xy0 = xy1; xy1 = xy2;
        g0 = g1; g1 = g2; g2 = g3; g3 = advance(g3);
    }
    if (GRAD && p.d_out_lay && lane == 0) bulk_store_wait_read();

    // ---- per-CTA partial sums ----
    s_ce = warp_sum(s_ce); s_tvh = warp_sum(s_tvh); s_tvw = warp_sum(s_tvw);
    m_grad = warp_max(m_grad); m_disp = warp_max(m_disp);
    if (lane == 0) {
        sm.red[wid][0] = s_ce; sm.red[wid][1] = s_tvh; sm.red[wid][2] = s_tvw;
        if (m_disp > 0.f) atomicMax(&p.hdr->maxdisp_bits, __float_as_uint(m_disp));
        if (m_grad > 0.f) atomicMax(&p.hdr->maxgrad_lay_bits, __float_as_uint(m_grad));
    }
    __syncthreads();
    if (tid == 0) {
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int w = 0; w < kTH; ++w) { o.x += sm.red[w][0]; o.y += sm.red[w][1]; o.z += sm.red[w][2]; }
#ifdef VLG_PROFILE_TAIL
        o.w = __uint_as_float(prof_stamp());     // where and when this CTA finished
#endif
        reinterpret_cast<float4 *>(p.partials)[blockIdx.x] = o;
        if (blockIdx.x == 0) p.hdr->n_lay = gridDim.x;
        __threadfence();
    }
    if (p.red.out != nullptr) {
        __syncthreads();
        if (tid == 0) sm.last = atomicAdd(&p.hdr->blocks_done, 1u) == gridDim.x - 1;
        __syncthreads();
        if (sm.last) {
            __threadfence();
            reduce_partials_block<kThreads>(p.red, reinterpret_cast<double *>(smem_raw));
        }
    }
}

}  // namespace vlg
