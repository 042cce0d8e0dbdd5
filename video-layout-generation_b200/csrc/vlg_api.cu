// vlg_api.cu -- the C ABI declared in include/vlg_b200.h: argument checks, workspace carving,
// kernel launches.  No allocation, no host synchronisation (except vlg_read_status), no torch.
#include <atomic>
#include <climits>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <type_traits>

#include "vlg_pass1.cuh"
#include "vlg_pass2.cuh"
#include "vlg_rgb.cuh"
#include "vlg_laytile.cuh"
#include "vlg_frames.cuh"
#include "vlg_ingest.cuh"
#include "vlg_labels.cuh"
#include "vlg_metrics.cuh"

using namespace vlg;

// Layout class counts compiled in: 20 = Cityscapes trainer head (src/models/gridnet.py:9), 19 = its
// train ids without "None", 30 = the 29+1 classes of the earlier head (src/models/simple.py:19,42),
// 5 = small-K parity fixture.
#ifdef VLG_FAST_BUILD   // kernel-tuning builds: the benchmark head only
#define VLG_FOR_EACH_K(X) X(20)
#else
#define VLG_FOR_EACH_K(X) X(20) X(19) X(30) X(5)
#endif

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

static int check_launch(const char *what) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(VLG_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
    return VLG_OK;
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---- kernel timeline (measurement aid behind vlg_timeline_arm / vlg_timeline_read) ----
// While armed on the calling thread, the fused entry points record CUDA events on their launch stream right before
// and after the three main kernels, so that a benchmark can time each kernel inside the real launch sequence.
enum { kTlRgb0, kTlRgb1, kTlLay0, kTlLay1, kTlP2a, kTlP2b, kTlCount };
struct Timeline {
    bool armed = false;
    int dev = -1;
    unsigned seen = 0;
    cudaEvent_t ev[kTlCount] = {};
};
static thread_local Timeline g_tl;
static void tl_mark(int i, cudaStream_t st) {
    if (!g_tl.armed) return;
    if (cudaEventRecord(g_tl.ev[i], st) == cudaSuccess) g_tl.seen |= 1u << i;
    else (void)cudaGetLastError();
}

// ---- per-device launch state ----
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) and occupancy-derived grid sizes belong to a DEVICE, not to the
// process: a process that drives several GPUs (nn.DataParallel at src/val.py:131, one thread per device, ...) must
// opt every device in.  Each launcher keeps one slot per device ordinal; the slots are atomics, and setting an
// attribute twice is harmless, so concurrent first calls need no lock.
constexpr int kMaxDevices = 64;
struct PerDevice {
    std::atomic<int> v[kMaxDevices];
    int get(int dev) const { return v[dev].load(std::memory_order_acquire); }
    void set(int dev, int x) { v[dev].store(x, std::memory_order_release); }
};
static int current_device(int *dev) {
    cudaError_t e = cudaGetDevice(dev);
    if (e != cudaSuccess) return fail(VLG_ERR_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
    if (*dev < 0 || *dev >= kMaxDevices) return fail(VLG_ERR_UNSUPPORTED, "device ordinal %d >= %d", *dev, kMaxDevices);
    return VLG_OK;
}
// number of SMs of the current device (148 on a B200; queried, never assumed)
static int sm_count() {
    static PerDevice sms;
    int dev = 0;
    if (current_device(&dev)) return 148;
    int n = sms.get(dev);
    if (!n) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n < 1) n = 148;
        sms.set(dev, n);
    }
    return n;
}
// opt a kernel in to `smem` bytes of dynamic shared memory on the current device (once per device and instantiation)
template <typename Kern>
static int ensure_smem(PerDevice &done, Kern kern, size_t smem, const char *what) {
    int dev = 0;
    if (int rc = current_device(&dev)) return rc;
    if (done.get(dev)) return VLG_OK;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail(VLG_ERR_CUDA, "cudaFuncSetAttribute(%s): %s", what, cudaGetErrorString(e));
    done.set(dev, 1);
    return VLG_OK;
}
// *ctas = CTAs of `kern` (`threads` threads, `smem` bytes of dynamic shared memory) resident at once on the current
// device, at most `max_per_sm` per SM: one wave of a persistent grid.  Queried once per device into `cache`, which the
// caller keeps per instantiation.
template <typename Kern>
static int resident_ctas(PerDevice &cache, Kern kern, int threads, size_t smem, int max_per_sm, const char *what, int *ctas) {
    int dev = 0;
    if (int rc = current_device(&dev)) return rc;
    *ctas = cache.get(dev);
    if (*ctas) return VLG_OK;
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem);
    if (e != cudaSuccess || per_sm < 1) return fail(VLG_ERR_CUDA, "%s occupancy query: %s", what, cudaGetErrorString(e));
    *ctas = sm_count() * (per_sm < max_per_sm ? per_sm : max_per_sm);
    cache.set(dev, *ctas);
    return VLG_OK;
}

// Calls f(std::integral_constant<int, K>{}) for a K compiled in, fails for any other.
template <typename F>
static int with_k(int64_t K, F &&f) {
#define X(k) if (K == k) return f(std::integral_constant<int, k>{});
    VLG_FOR_EACH_K(X)
#undef X
    return fail(VLG_ERR_UNSUPPORTED, "K=%lld not compiled in (see VLG_FOR_EACH_K)", (long long)K);
}
// Calls f(type_tag<T>{}) with the element type of a checked dtype.
template <typename T> struct type_tag { using type = T; };
template <typename F>
static int with_type(int dtype, F &&f) {
    return dtype == VLG_F32 ? f(type_tag<float>{}) : f(type_tag<__nv_bfloat16>{});
}
// Calls f(type_tag<T>{}, std::integral_constant<int, K>{}) for the problem's dtype and K.
template <typename F>
static int with_type_k(const vlg_problem_t *p, F &&f) {
    return with_k(p->K, [&](auto k) { return with_type(p->dtype, [&](auto t) { return f(t, k); }); });
}

static int check_problem(const vlg_problem_t *p) {
    if (!p) return fail(VLG_ERR_ARG, "problem is NULL");
    if (p->struct_size != sizeof(vlg_problem_t))
        return fail(VLG_ERR_ARG, "vlg_problem_t.struct_size is %u, this library was built with %zu: stale binding of include/vlg_b200.h?",
                    p->struct_size, sizeof(vlg_problem_t));
    if (p->abi_version / 100 != VLG_VERSION / 100)
        return fail(VLG_ERR_ARG, "vlg_problem_t.abi_version %u does not match the library's %d (major versions differ)", p->abi_version, VLG_VERSION);
    if (p->N < 1 || p->H < 2 || p->W < 2) return fail(VLG_ERR_ARG, "need N>=1, H>=2, W>=2 (got %lld,%lld,%lld)", (long long)p->N, (long long)p->H, (long long)p->W);
    if (p->N * p->H * p->W >= (1ll << 31)) return fail(VLG_ERR_UNSUPPORTED, "N*H*W must be < 2^31");
    if (p->N > 65535 || (p->H + 7) / 8 > 65535) return fail(VLG_ERR_UNSUPPORTED, "N and H/8 must fit a CUDA grid dimension (65535)");
    if (p->H > 65000 || p->W > 65000) return fail(VLG_ERR_UNSUPPORTED, "H and W must be <= 65000 (16-bit tap cells in the far-pixel queue)");
    if (int rc = with_k(p->K, [](auto) { return VLG_OK; })) return rc;
    if (p->dtype != VLG_F32 && p->dtype != VLG_BF16) return fail(VLG_ERR_ARG, "bad dtype %d", p->dtype);
    if (p->padding != VLG_PAD_ZEROS && p->padding != VLG_PAD_BORDER) return fail(VLG_ERR_ARG, "bad padding %d", p->padding);
    if (p->coord_mode != VLG_COORD_FLOW && p->coord_mode != VLG_COORD_GRID) return fail(VLG_ERR_ARG, "bad coord_mode %d", p->coord_mode);
    if (p->global_N != 0 && p->global_N < p->N) return fail(VLG_ERR_ARG, "global_N < N");
    if (p->ce_norm != VLG_CE_NORM_TORCH && p->ce_norm != VLG_CE_NORM_COUNT) return fail(VLG_ERR_ARG, "bad ce_norm %u", p->ce_norm);
    if (p->ce_class_weight && p->K > 32) return fail(VLG_ERR_UNSUPPORTED, "class weights need K <= 32");
    constexpr uint32_t known_flags = VLG_FLAG_NO_FAR_PATH | VLG_FLAG_NO_TMA | VLG_FLAG_PASS2_COORDS | VLG_FLAG_FAR_WIDE;
    if (p->flags & ~known_flags)
        return fail(VLG_ERR_ARG, "unknown flag bits 0x%x (4 and 8 were VLG_FLAG_TILE_RGB and VLG_FLAG_TILE_LAYOUT, which are retired)",
                    p->flags & ~known_flags);
    return VLG_OK;
}

// The workspace of a problem: its size, and its arrays for a workspace at `base` (all NULL when `base` is).
static WsLayout ws_layout(const vlg_problem_t *p, int with_src_grad, void *base = nullptr) {
    WsLayout L{};
    const size_t P = (size_t)p->N * p->H * p->W;
    const size_t n_blocks = (size_t)(p->N * tiles_x(p->W) * tiles_y(p->H));
    size_t off = 0;
    auto take = [&](auto *&array, size_t count) {   // `count` elements, 256-byte aligned
        array = base ? reinterpret_cast<std::remove_reference_t<decltype(array)>>((char *)base + off) : nullptr;
        off = align_up(off + count * sizeof(*array), 256);
    };
    // header, per-tile far flags, per-tile displacement maxima and the far-pixel counts per tile row are contiguous: one memset
    // resets them all
    take(L.hdr, 1);
    take(L.tile_flags, n_blocks);
    take(L.tile_disp, n_blocks);
    take(L.seg_cnt, n_blocks * kTH);   // far pixels per SOURCE tile row
    L.zero_bytes = off;
    take(L.partials, n_blocks * kPartialSlots);
    take(L.partials_rgb, (size_t)kRgbMaxWarps * kRgbSlots);
    take(L.partials_lay, (size_t)kLayMaxWarps * 4);
    take(L.flagged, n_blocks);
    L.pitch = (int64_t)align_up((size_t)p->W, 4);
    if (with_src_grad) {
        const size_t Pp = (size_t)p->N * p->H * (size_t)L.pitch;   // pitched rows: TMA-describable (16-byte row starts)
        take(L.dout_rgb, Pp * 3);
        take(L.dout_lay, P * p->K);
        take(L.rec_code, Pp);
        take(L.rec_frac, Pp);
        if (!(p->flags & VLG_FLAG_NO_FAR_PATH)) {
            take(L.far_acc, P * (3 + p->K));
            take(L.far_list, P);
        }
    }
    if (p->flags & VLG_FLAG_FAR_WIDE) L.seg_cnt = nullptr;   // without per-row counts pass 2 packs no row
    L.total = off;
    return L;
}

// The workspace of a checked problem at `workspace`, which must hold at least its total.
static int workspace_at(const vlg_problem_t *p, int with_src_grad, void *workspace, size_t workspace_bytes, WsLayout *L) {
    *L = ws_layout(p, with_src_grad, workspace);
    if (!workspace || workspace_bytes < L->total) return fail(VLG_ERR_WORKSPACE, "workspace too small: need %zu bytes", L->total);
    return VLG_OK;
}

static CoordCfg make_cc(const vlg_problem_t *p) {
    CoordCfg cc;
    cc.H = (int)p->H; cc.W = (int)p->W;
    cc.padding = p->padding; cc.coord_mode = p->coord_mode;
    cc.Wm1 = (float)(p->W - 1); cc.Hm1 = (float)(p->H - 1);
    cc.sx = (float)(2.0 / (double)(p->W - 1));
    cc.sy = (float)(2.0 / (double)(p->H - 1));
    return cc;
}

// ------------------------------------------------------------------ small kernels
// Counts the labels != ignore_index (CE divisor).  With class weights it also builds the per-class
// histogram with INTEGER atomics, and the last CTA (ticket) derives sum_k w_k * hist_k in a fixed
// order: the weighted divisor is bitwise reproducible.
__global__ void count_valid_kernel(const int64_t *__restrict__ label, int64_t P, int64_t ignore_index, int K,
                                   const float *__restrict__ class_weight, WsHeader *hdr) {
    __shared__ unsigned int s[32];
    __shared__ unsigned int sh[32];
    __shared__ int s_last;
    if (threadIdx.x < 32) sh[threadIdx.x] = 0u;
    __syncthreads();
    unsigned int cnt = 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if (!class_weight && (reinterpret_cast<uintptr_t>(label) & 15) == 0) {
        // unweighted: two labels per 128-bit load, four loads in flight per thread
        const longlong2 *l2 = reinterpret_cast<const longlong2 *>(label);
        const int64_t P2 = P >> 1;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P2; i += stride) {
            const longlong2 v = __ldg(l2 + i);
            cnt += (v.x != ignore_index) + (v.y != ignore_index);
        }
        if ((P & 1) && blockIdx.x == 0 && threadIdx.x == 0) cnt += __ldg(label + P - 1) != ignore_index;
    } else
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += stride) {
        const int64_t l = __ldg(label + i);
        cnt += l != ignore_index;
        if (class_weight && l >= 0 && l < K) {
            const unsigned peers = __match_any_sync(__activemask(), (int)l);   // one smem atomic per distinct class
            if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&sh[l], (unsigned)__popc(peers));
        }
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) s[wid] = cnt;
    __syncthreads();
    if (wid == 0) {
        unsigned int v = lane < (blockDim.x >> 5) ? s[lane] : 0u;
        v = __reduce_add_sync(0xffffffffu, v);
        if (lane == 0 && v) atomicAdd(&hdr->n_valid, (unsigned long long)v);
    }
    if (class_weight) {
        if (threadIdx.x < K && sh[threadIdx.x]) atomicAdd(&hdr->hist[threadIdx.x], (unsigned long long)sh[threadIdx.x]);
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) s_last = atomicAdd(&hdr->count_done, 1u) == gridDim.x - 1;
        __syncthreads();
        if (s_last && threadIdx.x == 0) {
            __threadfence();
            double d = 0.0;
            for (int k = 0; k < K; ++k) d += (double)__ldg(class_weight + k) * (double)__ldcg(&hdr->hist[k]);
            hdr->ce_denom = d;
        }
    }
}

__global__ void __launch_bounds__(256) reduce_partials_kernel(const ReduceParams p) {
    __shared__ double s[6 * 256];
    reduce_partials_block<256>(p, s);
}

// The loss terms in effect and their coefficients.  `warp`: a warped step (TV is a term of the pixel flow only).
static TermCoeffs make_terms(const vlg_problem_t *prob, bool warp) {
    const double Ng = (double)(prob->global_N ? prob->global_N : prob->N);
    const double H = (double)prob->H, W = (double)prob->W;
    TermCoeffs tc{};
    tc.terms = prob->term_mask ? prob->term_mask : VLG_TERM_ALL;
    if (!(prob->H > 2 && prob->W > 2)) tc.terms &= ~VLG_TERM_SSIM;
    if (!(warp && prob->coord_mode == VLG_COORD_FLOW)) tc.terms &= ~VLG_TERM_TV;
    tc.c_l1 = (tc.terms & VLG_TERM_L1) ? (float)(prob->w_l1 / (Ng * 3 * H * W)) : 0.f;
    tc.c_gd = (tc.terms & VLG_TERM_GD) ? (float)(prob->w_gd / (Ng * 3 * H * W)) : 0.f;
    tc.c_ssim = (tc.terms & VLG_TERM_SSIM) ? (float)(prob->w_ssim / (2.0 * Ng * (H - 2) * (W - 2))) : 0.f;
    tc.c_tvh = (tc.terms & VLG_TERM_TV) ? (float)(prob->w_tv / (Ng * (H - 1) * W * 2)) : 0.f;
    tc.c_tvw = (tc.terms & VLG_TERM_TV) ? (float)(prob->w_tv / (Ng * H * (W - 1) * 2)) : 0.f;
    // a masked-out CE still runs its forward sum (the reduction drops it) but sends no gradient anywhere
    tc.w_ce_over_scale = (tc.terms & VLG_TERM_CE) ? (float)(prob->w_ce * (double)prob->N / Ng) : 0.f;
    tc.weighted_denom = prob->ce_class_weight != nullptr && prob->ce_norm == VLG_CE_NORM_TORCH;
    return tc;
}

static ReduceParams make_reduce_params(const vlg_problem_t *prob, const TermCoeffs &tc, const WsLayout &L, float *loss_out) {
    const double Ng = (double)(prob->global_N ? prob->global_N : prob->N);
    const double H = (double)prob->H, W = (double)prob->W;
    ReduceParams rp{};
    rp.partials = L.partials;
    rp.partials_rgb = L.partials_rgb;
    rp.partials_lay = L.partials_lay;
    rp.hdr = L.hdr;
    rp.inv_numel_rgb = 1.0 / (Ng * 3 * H * W);
    rp.inv_ssim = (prob->H > 2 && prob->W > 2) ? 1.0 / (Ng * (H - 2) * (W - 2)) : 0.0;
    rp.inv_tvh = 1.0 / (Ng * (H - 1) * W * 2);
    rp.inv_tvw = 1.0 / (Ng * H * (W - 1) * 2);
    rp.ce_scale = (double)prob->N / Ng;
    rp.w_l1 = prob->w_l1; rp.w_gd = prob->w_gd; rp.w_ssim = prob->w_ssim; rp.w_ce = prob->w_ce; rp.w_tv = prob->w_tv;
    rp.weighted_denom = tc.weighted_denom;
    rp.terms = tc.terms;
    rp.out = loss_out;   // NULL: pass 1 does not fuse the final reduction
    return rp;
}

template <typename T>
__global__ void scale_kernel(T *g, int64_t n, const float *scale) {
    const float s = __ldg(scale);
    if (s == 1.0f) return;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        g[i] = from_f<T>(to_f<T>(g[i]) * s);
}

// The same for up to four buffers in ONE launch (autograd's backward of the fused op rescales d_src_rgb, d_src_layout and
// d_coords: three launches that almost always find *scale == 1 and exit).
struct ScaleSet { void *g[4]; int64_t n[4]; int dtype[4]; int count; };
__global__ void scale_multi_kernel(ScaleSet s, const float *scale) {
    const float f = __ldg(scale);
    if (f == 1.0f) return;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int b = 0; b < s.count; ++b) {
        if (s.dtype[b] == VLG_F32) {
            float *g = (float *)s.g[b];
            for (int64_t i = t0; i < s.n[b]; i += stride) g[i] = g[i] * f;
        } else {
            __nv_bfloat16 *g = (__nv_bfloat16 *)s.g[b];
            for (int64_t i = t0; i < s.n[b]; i += stride) g[i] = from_f<__nv_bfloat16>(to_f<__nv_bfloat16>(g[i]) * f);
        }
    }
}

// Rollout warp with LABEL sources (SURVEY 8f-2): the layout fed back between rollout steps is
// argmax -> one-hot (src/trainer.py:467), so the 20-channel gather collapses to four int64 taps.
// out_label == argmax_c warp(one_hot(src_label))_c bit for bit: for a 0/1 source the dense FMA
// chain reduces to adding the weights of the taps that carry class c, in tap order nw,ne,sw,se.
template <typename T>
__global__ void __launch_bounds__(256) warp_fwd_labels_kernel(CoordCfg cc, int64_t P, int64_t HW, const T *__restrict__ src_rgb,
                                                              const int64_t *__restrict__ src_label,
                                                              const float2 *__restrict__ coords, T *out_rgb,
                                                              int64_t *out_label) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    // N*H*W < 2^31 (check_problem): 32-bit divisions (a 64-bit division by a run-time value costs ~60 instructions)
    const unsigned nu = (unsigned)i / (unsigned)HW, rem = (unsigned)i - nu * (unsigned)HW;
    const int64_t n = nu;
    const int y = (int)(rem / (unsigned)cc.W), x = (int)(rem - (unsigned)y * (unsigned)cc.W);
    const Taps t = make_taps(cc, __ldg(coords + i), y, x);
    if (src_rgb && out_rgb) {
        float a[3];
        gather_px<T, 3>(src_rgb + n * HW * 3, cc, t, a);
        store_px<T, 3>(out_rgb + i * 3, a);
    }
    if (src_label && out_label) {
        const int xs[4] = {t.x0, t.x0 + 1, t.x0, t.x0 + 1};
        const int ys[4] = {t.y0, t.y0, t.y0 + 1, t.y0 + 1};
        const float ws[4] = {t.nw, t.ne, t.sw, t.se};
        int64_t lab[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const bool in = xs[k] >= 0 && xs[k] < cc.W && ys[k] >= 0 && ys[k] < cc.H;
            lab[k] = in ? __ldg(src_label + n * HW + (int64_t)ys[k] * cc.W + xs[k]) : (int64_t)-1;   // -1: contributes nothing
        }
        float best_z = 0.0f;          // classes carried by no tap have z == 0; the first of them is class 0
        int64_t best_c = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int64_t c = lab[k];
            if (c < 0) continue;
            // z_c through the same chain as the dense path: fmul for the nw tap, then three fmas
            float z = __fmul_rn(lab[0] == c ? 1.0f : 0.0f, ws[0]);
            z = __fmaf_rn(lab[1] == c ? 1.0f : 0.0f, ws[1], z);
            z = __fmaf_rn(lab[2] == c ? 1.0f : 0.0f, ws[2], z);
            z = __fmaf_rn(lab[3] == c ? 1.0f : 0.0f, ws[3], z);
            if (z > best_z || (z == best_z && c < best_c)) { best_z = z; best_c = c; }
        }
        out_label[i] = best_c;
    }
}

// Visualisation of a layout (src/trainer.py:416-427 vis_seg_mask, src/val.py:178): optional argmax
// over K channels, then a K-entry colour LUT, output rgb = lut / 255 as NHWC T.
template <typename T, int K>
__global__ void __launch_bounds__(256) colorize_kernel(int64_t P, const T *__restrict__ layout, const int64_t *__restrict__ label,
                                                       const uint8_t *__restrict__ lut, T *out_rgb, int64_t *out_label,
                                                       WsHeader *hdr_or_null) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    int64_t l;
    if (layout) {
        float z[K];
        load_px<T, K>(layout + i * K, z);
        l = first_max_index<K>(z);
        if (out_label) out_label[i] = l;
    } else {
        l = __ldg(label + i);
    }
    float rgb[3] = {0.f, 0.f, 0.f};
    if (l >= 0 && l < K) {
#pragma unroll
        for (int c = 0; c < 3; ++c) rgb[c] = __fdiv_rn((float)__ldg(lut + l * 3 + c), 255.0f);
    } else if (hdr_or_null) {
        atomicOr(&hdr_or_null->status, VLG_STATUS_BAD_LABEL);
    }
    store_px<T, 3>(out_rgb + i * 3, rgb);
}

// One-hot layout encoding (src/models/net_utils.py:14-24).  Whole 16-byte chunks per pixel: one WARP per 32 consecutive
// pixels -- every lane reads one class id, the 32 * CPP chunks leave in CPP coalesced rounds, the id of a chunk's pixel
// comes by shuffle (same scheme as ingest_seg_kernel: a thread per chunk spent its time dividing 64-bit indices).
// Otherwise one thread per pixel.
template <typename T, int K>
__global__ void __launch_bounds__(256) one_hot_kernel(int64_t P, const int64_t *__restrict__ lab_i, const float *__restrict__ lab_f,
                                                      T *__restrict__ out, WsHeader *hdr_or_null) {
    constexpr int EPC = 16 / (int)sizeof(T);                    // elements per 16-byte chunk
    constexpr bool kVec = (K % EPC) == 0;
    if constexpr (kVec) {
        constexpr int CPP = K / EPC;                            // chunks per pixel
        const unsigned lane = threadIdx.x & 31;
        const int64_t px0 = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32;
        if (px0 >= P) return;                                   // warp-uniform
        const int64_t px = px0 + lane;
        int l = -1;
        if (px < P) {
            const int64_t l64 = lab_i ? __ldg(lab_i + px) : (int64_t)__ldg(lab_f + px);   // .long() truncation
            const bool bad = l64 < 0 || l64 >= K;
            if (bad && hdr_or_null) atomicOr(&hdr_or_null->status, VLG_STATUS_BAD_LABEL);
            l = bad ? -1 : (int)l64;                            // out-of-range ids encode as an all-zero pixel
        }
        const int npx = (int)min((int64_t)32, P - px0);
        uint4 *dst = reinterpret_cast<uint4 *>(out) + px0 * CPP;
#pragma unroll
        for (int it = 0; it < CPP; ++it) {
            const int e = it * 32 + (int)lane, q = e / CPP, chunk = e - q * CPP;
            const int lq = __shfl_sync(0xffffffffu, l, q);
            if (q < npx) {
                uint4 r = make_uint4(0u, 0u, 0u, 0u);
                T *v = reinterpret_cast<T *>(&r);
                const int rel = lq - chunk * EPC;
                if (lq >= 0 && rel >= 0 && rel < EPC) v[rel] = from_f<T>(1.0f);
                dst[e] = r;
            }
        }
    } else {
        const int64_t px = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (px >= P) return;
        const int64_t l = lab_i ? __ldg(lab_i + px) : (int64_t)__ldg(lab_f + px);
        if ((l < 0 || l >= K) && hdr_or_null) atomicOr(&hdr_or_null->status, VLG_STATUS_BAD_LABEL);
#pragma unroll
        for (int k = 0; k < K; ++k) out[px * K + k] = from_f<T>(l == k ? 1.0f : 0.0f);
    }
}

// forward-only warp (validation / rollout): one thread per output pixel.  A CTA owns 256 CONSECUTIVE pixels, i.e.
// 256 * K contiguous elements of the warped layout: with BULK they are staged in shared memory and every warp
// sends its 32 pixels as one bulk shared->global copy -- a thread-per-pixel store of 80-byte pixels costs 20 L1
// wavefronts per 128-bit store instruction, and the kernel is bound by the LSU data pipe (70 %).
template <typename T, int K, bool BULK>
__global__ void __launch_bounds__(256) warp_fwd_kernel(CoordCfg cc, int64_t P, int64_t HW, const T *__restrict__ src_rgb,
                                                       const T *__restrict__ src_lay, const float2 *__restrict__ coords,
                                                       T *out_rgb, T *out_lay, int64_t *out_argmax, int2 *dbg) {
    __shared__ __align__(128) T s_out[BULK ? 256 * K : 1];
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < P;
    const int64_t ic = live ? i : P - 1;
    const unsigned nu = (unsigned)ic / (unsigned)HW, rem = (unsigned)ic - nu * (unsigned)HW;   // N*H*W < 2^31: 32-bit divisions
    const int64_t n = nu;
    const int y = (int)(rem / (unsigned)cc.W), x = (int)(rem - (unsigned)y * (unsigned)cc.W);
    const Taps t = make_taps(cc, __ldg(coords + ic), y, x);
    if (dbg && live) dbg[i] = make_int2((int)t.fx0, (int)t.fy0);
    if (src_rgb && out_rgb && live) {
        float a[3];
        gather_px<T, 3>(src_rgb + n * HW * 3, cc, t, a);
        store_px<T, 3>(out_rgb + i * 3, a);
    }
    if (src_lay && (out_lay || out_argmax)) {
        float z[K];
        gather_px<T, K>(src_lay + n * HW * K, cc, t, z);
        if (out_lay) {
            if constexpr (BULK) {
                const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
                store_px<T, K>(s_out + (size_t)threadIdx.x * K, z);
                fence_async_smem();
                __syncwarp();
                const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + w * 32;     // first pixel of this warp
                const int64_t npx = P - i0 < 32 ? P - i0 : 32;
                if (lane == 0 && npx > 0) {
                    bulk_store(out_lay + i0 * K, s_out + (size_t)w * 32 * K, (unsigned)(npx * K * (int64_t)sizeof(T)));
                    bulk_store_wait_read();
                }
            } else if (live) {
                store_px<T, K>(out_lay + i * K, z);
            }
        }
        if (out_argmax && live) {
            // argmax is taken on the values as STORED (rounded to T), like torch.argmax on the output
#pragma unroll
            for (int k = 0; k < K; ++k) z[k] = to_f<T>(from_f<T>(z[k]));
            out_argmax[i] = first_max_index<K>(z);
        }
    }
}

// ------------------------------------------------------------------ dispatch helpers
// cuTensorMapEncodeTiled is fetched through the runtime (no -lcuda): NULL if the driver lacks it
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder() {
    static EncodeTiledFn fn = [] {
        void *f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            f = nullptr;
        (void)cudaGetLastError();
        return (EncodeTiledFn)f;
    }();
    return fn;
}

// Tiled tensor map of a `rank`-D array at `base` (global dims innermost first, the rank-1 byte strides of the outer dims,
// the box): unit element strides, no interleave, swizzle or out-of-bounds fill.  False when the driver has no encoder or
// refuses the description.
static bool encode_map(CUtensorMap *map, CUtensorMapDataType dt, int rank, const void *base, const cuuint64_t *gdim,
                       const cuuint64_t *gstr, const cuuint32_t *box) {
    memset(map, 0, sizeof(*map));
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return false;
    const cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
    return enc(map, dt, (cuuint32_t)rank, const_cast<void *>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Tensor map of an NHWC layout [N][H][W][K] with a box_w x box_h x K box.  Returns false when TMA cannot be used
// (bf16 K=20 rows are not 16-byte multiples, odd K, ...).
static bool make_layout_map(const vlg_problem_t *prob, const void *src_layout, CUtensorMap *map, int box_w, int box_h,
                            bool fp32_storage = false) {
    const size_t es = 4;
    if ((prob->dtype != VLG_F32 && !fp32_storage) || (prob->K * es) % 16 != 0 || prob->K > 256) return false;
    if (((uintptr_t)src_layout) % 16 != 0) return false;
    const cuuint64_t gdim[4] = {(cuuint64_t)prob->K, (cuuint64_t)prob->W, (cuuint64_t)prob->H, (cuuint64_t)prob->N};
    const cuuint64_t gstr[3] = {(cuuint64_t)prob->K * es, (cuuint64_t)prob->W * prob->K * es,
                                (cuuint64_t)prob->H * prob->W * prob->K * es};
    const cuuint32_t box[4] = {(cuuint32_t)prob->K, (cuuint32_t)box_w, (cuuint32_t)box_h, 1u};
    return encode_map(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, src_layout, gdim, gstr, box);
}

// Tensor map of an NHWC layout for the persistent tile kernel.  Pixels whose byte size is a multiple of 16
// use the 4-D element-typed map above; 8-byte-multiple pixels (20 bf16 channels = 40 B) are described as
// rows of 8-byte units: 3-D {W*PXB/8, H, N}, box {box_w*PXB/8, box_h, 1}.  *px8 tells which one was built.
static bool make_window_map(const vlg_problem_t *prob, const void *src_layout, CUtensorMap *map, int box_w, int box_h, bool *px8) {
    *px8 = false;
    if (prob->dtype == VLG_F32) return make_layout_map(prob, src_layout, map, box_w, box_h);
    const size_t pxb = (size_t)prob->K * 2;
    if (pxb % 8 != 0 || ((size_t)prob->W * pxb) % 16 != 0 || ((uintptr_t)src_layout) % 16 != 0) return false;
    const size_t upp = pxb / 8;   // 8-byte units per pixel
    if ((size_t)box_w * upp > 256) return false;
    const cuuint64_t gdim[3] = {(cuuint64_t)prob->W * upp, (cuuint64_t)prob->H, (cuuint64_t)prob->N};
    const cuuint64_t gstr[2] = {(cuuint64_t)prob->W * pxb, (cuuint64_t)prob->H * prob->W * pxb};
    const cuuint32_t box[3] = {(cuuint32_t)(box_w * upp), (cuuint32_t)box_h, 1u};
    *px8 = encode_map(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, src_layout, gdim, gstr, box);
    return *px8;
}

// Pass 2 gathers from the tap records pass 1 wrote (pass2_rec_kernel: all staging by TMA) when the d_out
// windows can be described by tensor maps; otherwise, or on request, it re-derives the records from the
// coordinates (pass2_kernel).  Both calls of a step evaluate this with the same problem descriptor.
static bool pass2_from_records(const vlg_problem_t *prob) {
    return prob->K % 4 == 0 && prob->K <= 64 && !(prob->flags & (VLG_FLAG_NO_TMA | VLG_FLAG_PASS2_COORDS)) && tensor_map_encoder() != nullptr;
}

// Tensor map of a pitched workspace array [N][H][pitch * epp] of 4-byte elements (epp elements per pixel) with a
// window of kQW2 x kQH pixels.  The tensor's extent along x is W (not the pitch): the padding columns of a row are
// never written by pass 1, so they must arrive as the TMA's out-of-bounds zeros like every other cell outside the image.
static bool make_pitched_map(const vlg_problem_t *prob, const void *base, int64_t pitch, int epp, CUtensorMapDataType dt, CUtensorMap *map) {
    if (((uintptr_t)base) % 16 != 0 || (pitch * epp * 4) % 16 != 0) return false;
    const cuuint64_t gdim[3] = {(cuuint64_t)(prob->W * epp), (cuuint64_t)prob->H, (cuuint64_t)prob->N};
    const cuuint64_t gstr[2] = {(cuuint64_t)(pitch * epp * 4), (cuuint64_t)(prob->H * pitch * epp * 4)};
    const cuuint32_t box[3] = {(cuuint32_t)(kQW2 * epp), (cuuint32_t)kQH, 1u};
    return encode_map(map, dt, 3, base, gdim, gstr, box);
}

template <typename T, int K>
static int launch_pass1(bool warp, const Pass1Params &pp, cudaStream_t st) {
    // the staged source window is the last member: the un-warped criteria do not allocate it
    using Smem = Pass1Smem<T, K>;
    const size_t smem_warp = sizeof(Smem), smem_plain = offsetof(Smem, stage);
    static PerDevice attr_warp, attr_plain;  // per instantiation
    if (int rc = ensure_smem(attr_warp, pass1_kernel<T, K, true>, smem_warp, "pass1")) return rc;
    if (int rc = ensure_smem(attr_plain, pass1_kernel<T, K, false>, smem_plain, "pass1")) return rc;
    const dim3 grid((unsigned)pp.tiles_x, (unsigned)pp.tiles_y, (unsigned)pp.N);
    if (warp) pass1_kernel<T, K, true><<<grid, kThreads, smem_warp, st>>>(pp);
    else pass1_kernel<T, K, false><<<grid, kThreads, smem_plain, st>>>(pp);
    return check_launch("pass1_kernel");
}

template <typename T, int K>
static int launch_pass2(Pass2Params pp, const vlg_problem_t *prob, cudaStream_t st) {
    if (pp.far_acc) {   // both exit at once unless pass 1 queued far pixels
        const int sms = sm_count();
        far_zero_kernel<K><<<sms * 2, kThreads, 0, st>>>(pp);
        int rc = check_launch("far_zero_kernel");
        if (rc) return rc;
        far_scatter_kernel<K><<<sms * VLG_FAR_CTAS, kThreads, 0, st>>>(pp);
        rc = check_launch("far_scatter_kernel");
        if (rc) return rc;
    }
    if constexpr (K % 4 == 0 && K <= 64) {
        CUtensorMap lay_map, rgb_map, frac_map, code_map;
        if (pass2_from_records(prob) && pp.rec_code && pp.rec_frac &&
            make_layout_map(prob, pp.d_out_lay, &lay_map, kQW, kQH, true) &&
            make_pitched_map(prob, pp.d_out_rgb, pp.pitch, 3, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, &rgb_map) &&
            make_pitched_map(prob, pp.rec_frac, pp.pitch, 2, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, &frac_map) &&
            make_pitched_map(prob, pp.rec_code, pp.pitch, 1, CU_TENSOR_MAP_DATA_TYPE_UINT32, &code_map)) {
            constexpr size_t smem_rec = sizeof(Pass2RecSmem<K>);
            static PerDevice rec_attr;  // per instantiation
            if (int rc = ensure_smem(rec_attr, pass2_rec_kernel<T, K>, smem_rec, "pass2_rec")) return rc;
            tl_mark(kTlP2a, st);
            pass2_rec_kernel<T, K><<<dim3((unsigned)pp.tiles_x, (unsigned)pp.tiles_y, (unsigned)pp.N), kThreads, smem_rec, st>>>(
                pp, lay_map, rgb_map, frac_map, code_map);
            tl_mark(kTlP2b, st);
            return check_launch("pass2_rec_kernel");
        }
    }
    constexpr size_t smem = pass2_smem_bytes<K>();
    static PerDevice attr;  // per instantiation
    if (int rc = ensure_smem(attr, pass2_kernel<T, K>, smem, "pass2")) return rc;
    // the fp32 d_out staging buffer as a [N][H][W][K] tensor with a kQW x kQH window box
    CUtensorMap dout_map;
    pp.use_tma = (pp.d_src_lay && pp.d_out_lay && !(prob->flags & VLG_FLAG_NO_TMA) &&
                  make_layout_map(prob, pp.d_out_lay, &dout_map, kQW, kQH, true)) ? 1 : 0;
    if (!pp.use_tma) memset(&dout_map, 0, sizeof(dout_map));
    tl_mark(kTlP2a, st);
    pass2_kernel<T, K><<<dim3((unsigned)pp.tiles_x, (unsigned)pp.tiles_y, (unsigned)pp.N), kThreads, smem, st>>>(pp, dout_map);
    tl_mark(kTlP2b, st);
    return check_launch("pass2_kernel");
}

template <typename T, int K>
static int launch_fwd(const vlg_problem_t *prob, const void *src_rgb, const void *src_layout, const float *coords,
                      void *out_rgb, void *out_layout, int64_t *out_argmax, int32_t *dbg, cudaStream_t st) {
    const int64_t HW = prob->H * prob->W, P = prob->N * HW;
    // bulk shared->global copies need 16-byte multiples: 32-pixel runs of K*sizeof(T) bytes on a 16-byte aligned base
    const bool bulk = out_layout && (32 * K * sizeof(T)) % 16 == 0 && (K * sizeof(T)) % 8 == 0 && ((uintptr_t)out_layout & 15) == 0 &&
                      (P % 32 == 0 || (P % 32) * K * sizeof(T) % 16 == 0);
    if (bulk)
        warp_fwd_kernel<T, K, true><<<(unsigned)((P + 255) / 256), 256, 0, st>>>(
            make_cc(prob), P, HW, (const T *)src_rgb, (const T *)src_layout, (const float2 *)coords, (T *)out_rgb,
            (T *)out_layout, out_argmax, (int2 *)dbg);
    else
        warp_fwd_kernel<T, K, false><<<(unsigned)((P + 255) / 256), 256, 0, st>>>(
            make_cc(prob), P, HW, (const T *)src_rgb, (const T *)src_layout, (const float2 *)coords, (T *)out_rgb,
            (T *)out_layout, out_argmax, (int2 *)dbg);
    return check_launch("warp_fwd_kernel");
}

// Persistent-warp launch of the rgb strip kernel: one wave of resident warps, each with an equal
// contiguous run of (image, strip, row).
template <typename T>
static int launch_rgb(RgbParams rp, bool grad, cudaStream_t st) {
    static PerDevice resident;   // per instantiation (T); GRAD variants share the register budget
    int ctas = 0;
    if (int rc = resident_ctas(resident, rgb_strip_kernel<T, true, false>, kRgbThreads, 0, INT_MAX, "rgb_strip_kernel", &ctas)) return rc;
    const int warps_resident = ctas * (kRgbThreads / 32);
    int64_t warps = warps_resident < kRgbMaxWarps ? warps_resident : kRgbMaxWarps;
    const int64_t min_rows = 12;   // shorter runs are dominated by the 4 warm-up rows of a segment
    if (warps * min_rows > rp.total_rows) warps = (rp.total_rows + min_rows - 1) / min_rows;
    const int64_t blocks = (warps + kRgbThreads / 32 - 1) / (kRgbThreads / 32);
    rp.chunk = (rp.total_rows + blocks * (kRgbThreads / 32) - 1) / (blocks * (kRgbThreads / 32));
    const bool brd = rp.cc.padding == VLG_PAD_BORDER;
    if (grad && brd) rgb_strip_kernel<T, true, true><<<(unsigned)blocks, kRgbThreads, 0, st>>>(rp);
    else if (grad) rgb_strip_kernel<T, true, false><<<(unsigned)blocks, kRgbThreads, 0, st>>>(rp);
    else if (brd) rgb_strip_kernel<T, false, true><<<(unsigned)blocks, kRgbThreads, 0, st>>>(rp);
    else rgb_strip_kernel<T, false, false><<<(unsigned)blocks, kRgbThreads, 0, st>>>(rp);
    return check_launch("rgb_strip_kernel");
}

// Persistent launch of the double-buffered layout tile kernel: one wave of resident CTAs.
template <typename T, int K, bool PX8>
static int launch_laytile(const LayParams &lp, const CUtensorMap &map, bool grad, cudaStream_t st) {
    const size_t smem = sizeof(LayTileSmem<T, K>);
    static PerDevice resident, attr_g, attr_n;
    if (int rc = ensure_smem(attr_g, lay_tile_kernel<T, K, true, PX8>, smem, "lay_tile")) return rc;
    if (int rc = ensure_smem(attr_n, lay_tile_kernel<T, K, false, PX8>, smem, "lay_tile")) return rc;
    int ctas_resident = 0;
    if (int rc = resident_ctas(resident, lay_tile_kernel<T, K, true, PX8>, kThreads, smem, INT_MAX, "lay_tile_kernel", &ctas_resident))
        return rc;
    const int64_t n_tiles = (int64_t)lp.N * lp.strips * lp.tiles_y;
    int64_t blocks = ctas_resident < kLayMaxWarps ? ctas_resident : kLayMaxWarps;
    if (blocks * 2 > n_tiles) blocks = (n_tiles + 1) / 2;    // at least two tiles per CTA keeps the pipeline meaningful
    if (blocks < 1) blocks = 1;
    if (grad) lay_tile_kernel<T, K, true, PX8><<<(unsigned)blocks, kThreads, smem, st>>>(lp, map);
    else lay_tile_kernel<T, K, false, PX8><<<(unsigned)blocks, kThreads, smem, st>>>(lp, map);
    return check_launch("lay_tile_kernel");
}

// The rgb strip kernel with the gradient scales of `tc`: d(loss)/d(coords) (rgb part, nullable), the d(loss)/d(warped rgb)
// staging for pass 2 (nullable) and one partial row per warp.
static int launch_rgb_strips(const vlg_problem_t *prob, const TermCoeffs &tc, const void *src_rgb, const void *tgt_rgb,
                             const float *coords, float *d_coords, float *d_out_rgb, bool need_grad, const WsLayout &L,
                             cudaStream_t st) {
    RgbParams rp{};
    rp.cc = make_cc(prob);
    rp.N = (int)prob->N;
    rp.strips = (int)((prob->W + kRS - 1) / kRS);
    rp.total_rows = prob->N * rp.strips * prob->H;
    rp.src_rgb = src_rgb; rp.tgt_rgb = tgt_rgb; rp.coords = coords;
    rp.tc = tc;
    rp.d_coords = d_coords;
    rp.d_out_rgb = d_out_rgb;
    rp.pitch = (int)L.pitch;
    rp.partials = L.partials_rgb;
    rp.hdr = L.hdr;
    return with_type(prob->dtype, [&](auto t) { return launch_rgb<typename decltype(t)::type>(rp, need_grad, st); });
}

// Side stream + fork/join events of the calling thread, one lane per device (created on first use).  Used to run the
// label count next to the rgb strip kernel, which does not need it; works under stream capture too (the side stream
// joins the capture through the fork event and is joined back before the layout kernel).
struct SideLane {
    cudaStream_t s = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
static SideLane *side_lane() {
    static thread_local SideLane lanes[kMaxDevices];
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) {
        (void)cudaGetLastError();
        return nullptr;
    }
    SideLane &lane = lanes[dev];
    if (!lane.s) {
        SideLane nl;
        if (cudaStreamCreateWithFlags(&nl.s, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&nl.fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&nl.join, cudaEventDisableTiming) != cudaSuccess) {
            if (nl.join) cudaEventDestroy(nl.join);
            if (nl.fork) cudaEventDestroy(nl.fork);
            if (nl.s) cudaStreamDestroy(nl.s);
            (void)cudaGetLastError();
            return nullptr;
        }
        lane = nl;
    }
    return &lane;
}

// The first launches of pass 1: count_valid_kernel (the CE divisor; when `count`) and `rgb()` (the rgb strip kernel;
// when `has_rgb`).  The rgb kernel does not need the count, so the count runs beside it on the side lane, forked from
// `st` and joined back into it on every path, before the layout kernel that `st` runs next.
template <typename RgbLaunch>
static int count_beside_rgb(const vlg_problem_t *prob, bool count, const int64_t *tgt_label, WsHeader *hdr, bool has_rgb,
                            RgbLaunch rgb, cudaStream_t st) {
    SideLane *lane = nullptr;
    cudaStream_t cst = st;
    if (count && has_rgb && (lane = side_lane()) != nullptr) {
        if (cudaEventRecord(lane->fork, st) == cudaSuccess && cudaStreamWaitEvent(lane->s, lane->fork, 0) == cudaSuccess) cst = lane->s;
        else lane = nullptr;
    }
    int rc = VLG_OK;
    if (count) {
        const int64_t P = prob->N * prob->H * prob->W;
        const int blocks = (int)((P + 256 * 16 - 1) / (256 * 16));
        count_valid_kernel<<<blocks < 1 ? 1 : blocks, 256, 0, cst>>>(tgt_label, P, prob->ignore_index, (int)prob->K,
                                                                      prob->ce_class_weight, hdr);
        rc = check_launch("count_valid_kernel");
    }
    const bool join_recorded = lane && cudaEventRecord(lane->join, lane->s) == cudaSuccess;
    if (!rc && has_rgb) rc = rgb();
    if (lane) {
        if (!join_recorded) return rc ? rc : fail(VLG_ERR_CUDA, "side stream join record failed");
        if (cudaStreamWaitEvent(st, lane->join, 0) != cudaSuccess && !rc) rc = fail(VLG_ERR_CUDA, "side stream join failed");
    }
    return rc;
}

static int run_pass1(const vlg_problem_t *prob, bool warp, const void *src_rgb, const void *src_layout,
                     const float *coords, const void *tgt_rgb, const int64_t *tgt_label, float *d_coords,
                     void *d_out_rgb, void *d_out_lay, bool need_grad, int64_t *out_argmax, float *fused_loss_out,
                     const WsLayout &L, cudaStream_t st) {
    WsHeader *hdr = L.hdr;
    // header + per-tile far flags + per-tile displacement maxima are contiguous: one memset node resets them
    cudaError_t e = cudaMemsetAsync(hdr, 0, L.zero_bytes, st);
    if (e != cudaSuccess) return fail(VLG_ERR_CUDA, "memset header: %s", cudaGetErrorString(e));
    const int64_t P = prob->N * prob->H * prob->W;
    const bool has_lay = src_layout && tgt_label;
    const bool rgb_strips = warp && src_rgb && tgt_rgb;
    const TermCoeffs tc = make_terms(prob, warp);
    // The rgb terms of a warped step run in the column-strip kernel, launched BEFORE the kernel that owns the layout / TV
    // terms: it stores its part of d(loss)/d(coords); the layout kernel, which has issue slots to spare, loads that part
    // one tile ahead, adds its own and performs the final reduction.
    int rc = count_beside_rgb(prob, has_lay, tgt_label, hdr, rgb_strips, [&] {
        tl_mark(kTlRgb0, st);
        const int r = launch_rgb_strips(prob, tc, src_rgb, tgt_rgb, coords, need_grad ? d_coords : nullptr,
                                        need_grad ? (float *)d_out_rgb : nullptr, need_grad, L, st);
        tl_mark(kTlRgb1, st);
        return r;
    }, st);
    if (rc) return rc;
    Pass1Params pp{};
    pp.cc = make_cc(prob);
    pp.N = (int)prob->N;
    pp.tiles_x = (int)tiles_x(prob->W);
    pp.tiles_y = (int)tiles_y(prob->H);
    pp.src_rgb = src_rgb; pp.src_layout = src_layout; pp.coords = coords;
    pp.tgt_rgb = tgt_rgb; pp.label = tgt_label; pp.ignore_index = prob->ignore_index;
    pp.class_weight = prob->ce_class_weight;
    pp.tc = tc;
    pp.need_grad = need_grad;
    pp.d_coords = d_coords; pp.d_out_rgb = d_out_rgb; pp.d_out_lay = d_out_lay;
    pp.out_argmax = out_argmax;
    pp.partials = L.partials;
    pp.tile_disp = L.tile_disp;
    pp.tile_flags = L.tile_flags;
    pp.seg_cnt = L.seg_cnt;
    pp.far_list = (warp && d_out_lay) ? L.far_list : nullptr;
    pp.flagged_list = L.flagged;
    pp.red = make_reduce_params(prob, tc, L, fused_loss_out);
    pp.hdr = hdr;
    pp.accum_dcoords = rgb_strips ? 1 : 0;
    // tap records for pass 2: written by lay_tile_kernel on its way, by tap_records_kernel after pass1_kernel
    const bool want_records = warp && need_grad && d_out_lay != nullptr && L.rec_code && pass2_from_records(prob);
    bool records_done = false;
    bool lay_done = false;
    if (warp && has_lay && prob->K % 4 == 0 && !(prob->flags & VLG_FLAG_NO_TMA)) {
        CUtensorMap row_map;
        bool px8 = false;
        if (make_window_map(prob, src_layout, &row_map, kTSW, kTSH, &px8)) {
            LayParams lp{};
            lp.cc = pp.cc;
            lp.N = pp.N; lp.strips = pp.tiles_x; lp.tiles_y = pp.tiles_y;
            lp.total_rows = prob->N * (int64_t)lp.strips * prob->H;
            lp.src_layout = src_layout; lp.coords = coords; lp.label = tgt_label; lp.ignore_index = prob->ignore_index;
            lp.class_weight = pp.class_weight;
            lp.tc = tc;
            lp.accum_dcoords = pp.accum_dcoords;
            lp.d_coords = need_grad ? d_coords : nullptr;
            lp.d_out_lay = need_grad ? (float *)d_out_lay : nullptr;
            if (want_records) {
                lp.rec_code = L.rec_code; lp.rec_frac = L.rec_frac; lp.pitch = (int)L.pitch;
                records_done = true;
            }
            lp.out_argmax = out_argmax;
            lp.partials = L.partials_lay;
            lp.tile_disp = pp.tile_disp; lp.far_list = pp.far_list; lp.tile_flags = pp.tile_flags; lp.seg_cnt = pp.seg_cnt; lp.flagged_list = pp.flagged_list;
            lp.red = pp.red; lp.hdr = hdr;
            tl_mark(kTlLay0, st);
            // lay_tile_kernel is compiled for K % 4 == 0: fp32, and bf16 in 8-byte units (PX8) or with K % 8 == 0
            rc = with_type_k(prob, [&](auto t, auto k) {
                using T = typename decltype(t)::type;
                constexpr int K = decltype(k)::value;
                constexpr bool f32 = std::is_same<T, float>::value;
                if constexpr (K % 4 == 0 && !f32) {
                    if (px8) return launch_laytile<T, K, true>(lp, row_map, need_grad, st);
                }
                if constexpr (K % 4 == 0 && (f32 || K % 8 == 0)) {
                    if (!px8) return launch_laytile<T, K, false>(lp, row_map, need_grad, st);
                }
                return fail(VLG_ERR_UNSUPPORTED, "layout tile kernel: K / dtype not compiled in");
            });
            tl_mark(kTlLay1, st);
            if (rc) return rc;
            lay_done = true;
        }
    }
    if (!lay_done) {
        rc = with_type_k(prob, [&](auto t, auto k) { return launch_pass1<typename decltype(t)::type, decltype(k)::value>(warp, pp, st); });
        if (rc) return rc;
    }
    if (want_records && !records_done) {
        tap_records_kernel<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(pp.cc, P, prob->H * prob->W, (int)L.pitch, (const float2 *)coords,
                                                                        L.rec_code, L.rec_frac);
        rc = check_launch("tap_records_kernel");
    }
    return rc;
}

// Pass 1 with a LABEL layout source: memset(header) -> (count_valid on the side stream, next to) rgb_strip_kernel ->
// join -> lab_pix_kernel (layout terms from four label taps, TV, sum of d_coords, final reduction).
static int run_pass1_labels(const vlg_problem_t *prob, const void *src_rgb, const int64_t *src_label, const float *coords,
                            const void *tgt_rgb, const int64_t *tgt_label, float *d_coords, int64_t *out_argmax, float *loss_out,
                            const WsLayout &L, cudaStream_t st) {
    WsHeader *hdr = L.hdr;
    const int64_t P = prob->N * prob->H * prob->W;
    const bool has_rgb = src_rgb && tgt_rgb;
    if (!(src_label && tgt_label)) return fail(VLG_ERR_UNSUPPORTED, "the label-source op needs src_label / tgt_label (use vlg_pixel_loss_* for rgb-only criteria)");
    cudaError_t e = cudaMemsetAsync(hdr, 0, L.zero_bytes, st);
    if (e != cudaSuccess) return fail(VLG_ERR_CUDA, "memset header: %s", cudaGetErrorString(e));
    const bool need_grad = d_coords != nullptr;
    const TermCoeffs tc = make_terms(prob, true);
    // sources are data: no pass 2, no d(loss)/d(warped rgb) staging
    int rc = count_beside_rgb(prob, true, tgt_label, hdr, has_rgb, [&] {
        return launch_rgb_strips(prob, tc, src_rgb, tgt_rgb, coords, d_coords, nullptr, need_grad, L, st);
    }, st);
    if (rc) return rc;
    LabParams lp{};
    lp.cc = make_cc(prob); lp.K = (int)prob->K; lp.P = P; lp.HW = prob->H * prob->W;
    lp.src_label = src_label; lp.coords = (const float2 *)coords; lp.tgt_label = tgt_label; lp.ignore_index = prob->ignore_index;
    lp.class_weight = prob->ce_class_weight;
    lp.tc = tc;
    lp.accum_dcoords = has_rgb ? 1 : 0;
    lp.d_coords = d_coords; lp.out_argmax = out_argmax;
    lp.partials = L.partials_lay;
    lp.red = make_reduce_params(prob, tc, L, loss_out);
    lp.hdr = hdr;
    int64_t blocks = (int64_t)sm_count() * 8;
    const int64_t max_blocks = (P + kLabThreads - 1) / kLabThreads;
    if (blocks > max_blocks) blocks = max_blocks;
    if (blocks > kLayMaxWarps) blocks = kLayMaxWarps;
    if (need_grad) lab_pix_kernel<true><<<(unsigned)blocks, kLabThreads, 0, st>>>(lp);
    else lab_pix_kernel<false><<<(unsigned)blocks, kLabThreads, 0, st>>>(lp);
    return check_launch("lab_pix_kernel");
}

// Persistent launch of the confusion-matrix kernel.  Every CTA flushes up to K*K+1 bins with global atomics once, so the
// grid is one wave of at most kConfMaxCtasPerSm CTAs per SM (4 x 256 threads keep enough 16-byte loads in flight to
// stream HBM), and no larger than gives every thread kConfMinPxPerThread pixels.
constexpr int kConfMaxCtasPerSm = 4, kConfMinPxPerThread = 16;
template <typename T, int K, int MODE>
static int launch_confusion(const ConfParams &cp, cudaStream_t st) {
    static PerDevice resident;   // per instantiation
    int ctas = 0;
    if (int rc = resident_ctas(resident, confusion_kernel<T, K, MODE>, kConfThreads, 0, kConfMaxCtasPerSm, "confusion_kernel", &ctas))
        return rc;
    const int64_t by_work = (cp.P + (int64_t)kConfThreads * kConfMinPxPerThread - 1) / ((int64_t)kConfThreads * kConfMinPxPerThread);
    const int64_t blocks = by_work < ctas ? by_work : ctas;
    confusion_kernel<T, K, MODE><<<(unsigned)blocks, kConfThreads, 0, st>>>(cp);
    return check_launch("confusion_kernel");
}

template <typename T>
static int launch_frame_affine(const vlg_problem_t *prob, const FrameAffine &fa, const float *in, bool nchw, int flip, void *out, cudaStream_t st) {
    const int64_t P = prob->N * prob->H * prob->W;
    const int H = (int)prob->H, W = (int)prob->W;
    const bool vec = W % 4 == 0 && ((uintptr_t)in) % 16 == 0 && ((uintptr_t)out) % 16 == 0;
    if (vec) {
        const int64_t groups = P / 4;
        const unsigned blocks = (unsigned)((groups + 255) / 256);
        if (nchw) frame_affine_vec4_kernel<T, true><<<blocks, 256, 0, st>>>(fa, groups, H, W, flip, in, (T *)out);
        else frame_affine_vec4_kernel<T, false><<<blocks, 256, 0, st>>>(fa, groups, H, W, flip, in, (T *)out);
    } else {
        const unsigned blocks = (unsigned)((P + 255) / 256);
        if (nchw) frame_affine_px_kernel<T, true><<<blocks, 256, 0, st>>>(fa, P, H, W, flip, in, (T *)out);
        else frame_affine_px_kernel<T, false><<<blocks, 256, 0, st>>>(fa, P, H, W, flip, in, (T *)out);
    }
    return check_launch("frame_affine_kernel");
}

// ------------------------------------------------------------------ exported C ABI
template <typename T, int K>
static int launch_ingest_seg(int64_t P, int W, int flip, const uint8_t *seg_u8, int64_t *out_label, float *out_seg_f32, void *out_onehot,
                             void *workspace, cudaStream_t st) {
    constexpr int EPC = 16 / (int)sizeof(T);
    if constexpr (K % EPC == 0) {
        if (out_onehot) {     // one thread per 16-byte chunk of the one-hot layout
            const int64_t n = ((P + 31) / 32) * 32;      // one warp per 32 pixels
            ingest_seg_kernel<T, K, true><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(P, W, flip, seg_u8, out_label, out_seg_f32, (T *)out_onehot,
                                                                                       (WsHeader *)workspace);
            return check_launch("ingest_seg_kernel");
        }
    }
    ingest_seg_kernel<T, K, false><<<(unsigned)((P + 255) / 256), 256, 0, st>>>(P, W, flip, seg_u8, out_label, out_seg_f32, (T *)out_onehot,
                                                                                (WsHeader *)workspace);
    return check_launch("ingest_seg_kernel");
}

extern "C" {

int vlg_version(void) { return VLG_VERSION; }
const char *vlg_last_error(void) { return g_err; }
int64_t vlg_launch_count(void) { return g_launches.load(); }

size_t vlg_workspace_bytes(const vlg_problem_t *prob, int with_src_grad) {
    if (check_problem(prob)) return 0;
    return ws_layout(prob, with_src_grad).total;
}

int vlg_timeline_arm(int on) {
    int dev = -1;
    if (int rc = current_device(&dev)) return rc;
    if (on && g_tl.dev != dev) {
        for (int i = 0; i < kTlCount; ++i)
            if (cudaEventCreate(&g_tl.ev[i]) != cudaSuccess) return fail(VLG_ERR_CUDA, "cudaEventCreate failed");
        g_tl.dev = dev;
    }
    g_tl.armed = on != 0;
    if (on) g_tl.seen = 0;
    return VLG_OK;
}

int vlg_timeline_read(float *ms4) {
    if (!ms4) return fail(VLG_ERR_ARG, "ms4 is NULL");
    if (g_tl.dev < 0) return fail(VLG_ERR_ARG, "vlg_timeline_arm was never called on this thread");
    const int pairs[3][2] = {{kTlRgb0, kTlRgb1}, {kTlLay0, kTlLay1}, {kTlP2a, kTlP2b}};
    int first = -1, last = -1;
    for (int i = 0; i < kTlCount; ++i)
        if (g_tl.seen & (1u << i)) { if (first < 0) first = i; last = i; }
    if (last >= 0 && cudaEventSynchronize(g_tl.ev[last]) != cudaSuccess) return fail(VLG_ERR_CUDA, "timeline: event synchronize failed");
    for (int k = 0; k < 3; ++k) {
        ms4[k] = -1.0f;
        const unsigned need = (1u << pairs[k][0]) | (1u << pairs[k][1]);
        if ((g_tl.seen & need) == need && cudaEventElapsedTime(&ms4[k], g_tl.ev[pairs[k][0]], g_tl.ev[pairs[k][1]]) != cudaSuccess) {
            (void)cudaGetLastError();
            ms4[k] = -1.0f;
        }
    }
    ms4[3] = -1.0f;
    if (first >= 0 && last > first && cudaEventElapsedTime(&ms4[3], g_tl.ev[first], g_tl.ev[last]) != cudaSuccess) {
        (void)cudaGetLastError();
        ms4[3] = -1.0f;
    }
    return VLG_OK;
}

int vlg_warp_fwd(const vlg_problem_t *prob, const void *src_rgb, const void *src_layout, const float *coords,
                 void *out_rgb, void *out_layout, int64_t *out_argmax, int32_t *dbg_x0y0, void *stream) {
    int rc = check_problem(prob);
    if (rc) return rc;
    if (!coords) return fail(VLG_ERR_ARG, "coords is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    return with_type_k(prob, [&](auto t, auto k) {
        return launch_fwd<typename decltype(t)::type, decltype(k)::value>(prob, src_rgb, src_layout, coords, out_rgb, out_layout,
                                                                          out_argmax, dbg_x0y0, st);
    });
}

int vlg_warp_fwd_labels(const vlg_problem_t *prob, const void *src_rgb, const int64_t *src_label, const float *coords,
                        void *out_rgb, int64_t *out_label, void *stream) {
    int rc = check_problem(prob);
    if (rc) return rc;
    if (!coords) return fail(VLG_ERR_ARG, "coords is NULL");
    if ((src_label == nullptr) != (out_label == nullptr)) return fail(VLG_ERR_ARG, "src_label and out_label go together");
    const int64_t HW = prob->H * prob->W, P = prob->N * HW;
    cudaStream_t st = (cudaStream_t)stream;
    return with_type(prob->dtype, [&](auto t) {
        using T = typename decltype(t)::type;
        warp_fwd_labels_kernel<T><<<(unsigned)((P + 255) / 256), 256, 0, st>>>(make_cc(prob), P, HW, (const T *)src_rgb, src_label,
                                                                               (const float2 *)coords, (T *)out_rgb, out_label);
        return check_launch("warp_fwd_labels_kernel");
    });
}

int vlg_colorize(const vlg_problem_t *prob, const void *layout, const int64_t *label, const uint8_t *lut_rgb,
                 void *out_rgb, int64_t *out_label, void *stream) {
    int rc = check_problem(prob);
    if (rc) return rc;
    if ((layout == nullptr) == (label == nullptr)) return fail(VLG_ERR_ARG, "give exactly one of layout / label");
    if (!lut_rgb || !out_rgb) return fail(VLG_ERR_ARG, "lut_rgb and out_rgb are required");
    const int64_t P = prob->N * prob->H * prob->W;
    cudaStream_t st = (cudaStream_t)stream;
    return with_type_k(prob, [&](auto t, auto k) {
        using T = typename decltype(t)::type;
        colorize_kernel<T, decltype(k)::value><<<(unsigned)((P + 255) / 256), 256, 0, st>>>(P, (const T *)layout, label, lut_rgb,
                                                                                         (T *)out_rgb, out_label, nullptr);
        return check_launch("colorize_kernel");
    });
}

int vlg_confusion(const vlg_problem_t *prob, const void *layout, int32_t layout_is_nchw, const int64_t *pred_label,
                  const int64_t *tgt_label, uint64_t *counts, void *stream) {
    int rc = check_problem(prob);
    if (rc) return rc;
    if ((layout == nullptr) == (pred_label == nullptr)) return fail(VLG_ERR_ARG, "give exactly one of layout / pred_label");
    if (!tgt_label || !counts) return fail(VLG_ERR_ARG, "tgt_label and counts are required");
    if (layout && !layout_is_nchw && ((uintptr_t)layout & 15)) return fail(VLG_ERR_ARG, "an NHWC layout must be 16-byte aligned");
    ConfParams cp{};
    cp.layout = layout;
    cp.pred = pred_label;
    cp.tgt = tgt_label;
    cp.counts = reinterpret_cast<unsigned long long *>(counts);
    cp.P = prob->N * prob->H * prob->W;
    cp.ignore_index = prob->ignore_index;
    cp.HW = (unsigned)(prob->H * prob->W);
    cp.vec = (((uintptr_t)pred_label | (uintptr_t)tgt_label) & 15) == 0;
    cudaStream_t st = (cudaStream_t)stream;
    return with_k(prob->K, [&](auto k) {
        constexpr int K = decltype(k)::value;
        if (!layout) return launch_confusion<float, K, kConfLabels>(cp, st);   // labels: the problem's dtype plays no part
        return with_type(prob->dtype, [&](auto t) {
            using T = typename decltype(t)::type;
            return layout_is_nchw ? launch_confusion<T, K, kConfNchw>(cp, st) : launch_confusion<T, K, kConfNhwc>(cp, st);
        });
    });
}

int vlg_one_hot(const vlg_problem_t *prob, const int64_t *label_i64, const float *label_f32, void *out_layout,
                void *workspace, void *stream) {
    int rc = check_problem(prob);
    if (rc) return rc;
    if ((label_i64 == nullptr) == (label_f32 == nullptr)) return fail(VLG_ERR_ARG, "give exactly one of label_i64 / label_f32");
    if (!out_layout) return fail(VLG_ERR_ARG, "out_layout is NULL");
    const int64_t P = prob->N * prob->H * prob->W;
    cudaStream_t st = (cudaStream_t)stream;
    return with_type_k(prob, [&](auto t, auto k) {
        using T = typename decltype(t)::type;
        constexpr int K = decltype(k)::value, EPC = 16 / (int)sizeof(T);
        const int64_t n = (K % EPC) == 0 ? ((P + 31) / 32) * 32 : P;     // a warp per 32 pixels / a thread per pixel
        one_hot_kernel<T, K><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(P, label_i64, label_f32, (T *)out_layout, (WsHeader *)workspace);
        return check_launch("one_hot_kernel");
    });
}

static int warp_loss_pass1(const vlg_problem_t *prob, const void *src_rgb, const void *src_layout, const float *coords,
                           const void *tgt_rgb, const int64_t *tgt_label, float *d_coords, int64_t *out_argmax,
                           int with_src_grad, float *fused_loss_out, void *workspace, size_t workspace_bytes,
                           void *stream) {
    if (int rc = check_problem(prob)) return rc;
    if (!coords) return fail(VLG_ERR_ARG, "coords is NULL");
    if (with_src_grad && !d_coords) return fail(VLG_ERR_ARG, "with_src_grad needs d_coords (gradient pass)");
    WsLayout L;
    if (int rc = workspace_at(prob, with_src_grad, workspace, workspace_bytes, &L)) return rc;
    return run_pass1(prob, true, src_rgb, src_layout, coords, tgt_rgb, tgt_label, d_coords, L.dout_rgb, L.dout_lay,
                     d_coords != nullptr, out_argmax, fused_loss_out, L, (cudaStream_t)stream);
}

int vlg_warp_loss_bwd_out(const vlg_problem_t *prob, const void *src_rgb, const void *src_layout, const float *coords,
                          const void *tgt_rgb, const int64_t *tgt_label, float *d_coords, int64_t *out_argmax,
                          int with_src_grad, void *workspace, size_t workspace_bytes, void *stream) {
    return warp_loss_pass1(prob, src_rgb, src_layout, coords, tgt_rgb, tgt_label, d_coords, out_argmax, with_src_grad,
                           nullptr, workspace, workspace_bytes, stream);
}

int vlg_warp_loss_pass1(const vlg_problem_t *prob, const void *src_rgb, const void *src_layout, const float *coords,
                        const void *tgt_rgb, const int64_t *tgt_label, float *loss_out, float *d_coords, int64_t *out_argmax,
                        int with_src_grad, void *workspace, size_t workspace_bytes, void *stream) {
    return warp_loss_pass1(prob, src_rgb, src_layout, coords, tgt_rgb, tgt_label, d_coords, out_argmax, with_src_grad,
                           loss_out, workspace, workspace_bytes, stream);
}

int vlg_warp_bwd_src(const vlg_problem_t *prob, const float *coords, void *d_src_rgb, void *d_src_layout,
                     void *workspace, size_t workspace_bytes, void *stream) {
    if (int rc = check_problem(prob)) return rc;
    if (!coords) return fail(VLG_ERR_ARG, "coords is NULL");
    WsLayout L;
    if (int rc = workspace_at(prob, 1, workspace, workspace_bytes, &L)) return rc;
    Pass2Params pp{};
    pp.cc = make_cc(prob);
    pp.N = (int)prob->N; pp.tiles_x = (int)tiles_x(prob->W); pp.tiles_y = (int)tiles_y(prob->H);
    pp.coords = coords;
    pp.d_out_rgb = L.dout_rgb;
    pp.d_out_lay = L.dout_lay;
    pp.rec_code = L.rec_code;
    pp.rec_frac = L.rec_frac;
    pp.pitch = (int)L.pitch;
    pp.d_src_rgb = d_src_rgb; pp.d_src_lay = d_src_layout;
    pp.far_acc = L.far_acc;
    pp.far_list = L.far_list;
    pp.tile_flags = L.tile_flags;
    pp.seg_cnt = L.seg_cnt;
    pp.flagged_list = L.flagged;
    pp.hdr = L.hdr;
    pp.tile_disp = L.tile_disp;
    pp.HW = prob->H * prob->W;
    cudaStream_t st = (cudaStream_t)stream;
    return with_type_k(prob, [&](auto t, auto k) { return launch_pass2<typename decltype(t)::type, decltype(k)::value>(pp, prob, st); });
}

int vlg_reduce_partials(const vlg_problem_t *prob, float *loss_out, void *workspace, size_t workspace_bytes, void *stream) {
    if (int rc = check_problem(prob)) return rc;
    if (!loss_out) return fail(VLG_ERR_ARG, "loss_out is NULL");
    WsLayout L;
    if (int rc = workspace_at(prob, 0, workspace, workspace_bytes, &L)) return rc;
    const ReduceParams rp = make_reduce_params(prob, make_terms(prob, true), L, loss_out);
    reduce_partials_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(rp);
    return check_launch("reduce_partials_kernel");
}

int vlg_warp_loss_fwd_bwd(const vlg_problem_t *prob, const void *src_rgb, const void *src_layout, const float *coords,
                          const void *tgt_rgb, const int64_t *tgt_label, float *loss_out, float *d_coords,
                          void *d_src_rgb, void *d_src_layout, int64_t *out_argmax, void *workspace,
                          size_t workspace_bytes, void *stream) {
    const int with_src = (d_src_rgb || d_src_layout) ? 1 : 0;
    // the last pass-1 CTA performs the final reduction into loss_out: no separate reduce launch
    int rc = warp_loss_pass1(prob, src_rgb, src_layout, coords, tgt_rgb, tgt_label, d_coords, out_argmax, with_src,
                             loss_out, workspace, workspace_bytes, stream);
    if (rc) return rc;
    if (with_src) rc = vlg_warp_bwd_src(prob, coords, d_src_rgb, d_src_layout, workspace, workspace_bytes, stream);
    return rc;
}

int vlg_warp_loss_labels_fwd_bwd(const vlg_problem_t *prob, const void *src_rgb, const int64_t *src_label, const float *coords,
                                 const void *tgt_rgb, const int64_t *tgt_label, float *loss_out, float *d_coords,
                                 int64_t *out_argmax, void *workspace, size_t workspace_bytes, void *stream) {
    if (int rc = check_problem(prob)) return rc;
    if (!coords) return fail(VLG_ERR_ARG, "coords is NULL");
    if ((src_rgb == nullptr) != (tgt_rgb == nullptr)) return fail(VLG_ERR_ARG, "src_rgb and tgt_rgb go together");
    if ((src_label == nullptr) != (tgt_label == nullptr)) return fail(VLG_ERR_ARG, "src_label and tgt_label go together");
    if (!src_rgb && !src_label) return fail(VLG_ERR_ARG, "nothing to evaluate");
    WsLayout L;
    if (int rc = workspace_at(prob, 0, workspace, workspace_bytes, &L)) return rc;
    return run_pass1_labels(prob, src_rgb, src_label, coords, tgt_rgb, tgt_label, d_coords, out_argmax, loss_out, L, (cudaStream_t)stream);
}

int vlg_ingest(const vlg_problem_t *prob, const uint8_t *frames_u8, const float *mean3, const float *std3, int32_t flip_w,
               void *out_frames, const uint8_t *seg_u8, int64_t *out_label, float *out_seg_f32, void *out_onehot,
               void *workspace, void *stream) {
    int rc = check_problem(prob);
    if (rc) return rc;
    if ((frames_u8 == nullptr) != (out_frames == nullptr)) return fail(VLG_ERR_ARG, "frames_u8 and out_frames go together");
    if ((mean3 == nullptr) != (std3 == nullptr)) return fail(VLG_ERR_ARG, "mean3 and std3 go together");
    if (seg_u8 && !out_label && !out_seg_f32 && !out_onehot) return fail(VLG_ERR_ARG, "seg_u8 given but no output for it");
    if (!seg_u8 && (out_label || out_seg_f32 || out_onehot)) return fail(VLG_ERR_ARG, "segmentation outputs need seg_u8");
    if (!frames_u8 && !seg_u8) return fail(VLG_ERR_ARG, "nothing to ingest");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t P = prob->N * prob->H * prob->W;
    const int W = (int)prob->W, flip = flip_w ? 1 : 0;
    if (frames_u8) {
        IngestNorm nm{};
        nm.normalize = mean3 != nullptr;
        for (int c = 0; c < 3; ++c) { nm.mean[c] = mean3 ? mean3[c] : 0.f; nm.std[c] = std3 ? std3[c] : 1.f; }
        const bool vec = W % 4 == 0 && ((uintptr_t)frames_u8) % 4 == 0 && ((uintptr_t)out_frames) % 16 == 0;
        rc = with_type(prob->dtype, [&](auto t) {
            using T = typename decltype(t)::type;
            if (vec) ingest_frames_vec4_kernel<T><<<(unsigned)((P / 4 + 255) / 256), 256, 0, st>>>(nm, P / 4, W, flip, frames_u8, (T *)out_frames);
            else ingest_frames_px_kernel<T><<<(unsigned)((P + 255) / 256), 256, 0, st>>>(nm, P, W, flip, frames_u8, (T *)out_frames);
            return check_launch("ingest_frames_kernel");
        });
        if (rc) return rc;
    }
    if (seg_u8) {
        return with_type_k(prob, [&](auto t, auto k) {
            return launch_ingest_seg<typename decltype(t)::type, decltype(k)::value>(P, W, flip, seg_u8, out_label, out_seg_f32,
                                                                                     out_onehot, workspace, st);
        });
    }
    return rc;
}

int vlg_pixel_loss_fwd_bwd(const vlg_problem_t *prob, const void *out_rgb, const void *tgt_rgb, const void *logits,
                           const int64_t *tgt_label, float *loss_out, void *d_out_rgb, void *d_logits,
                           int64_t *out_argmax, void *workspace, size_t workspace_bytes, void *stream) {
    if (int rc = check_problem(prob)) return rc;
    WsLayout L;
    if (int rc = workspace_at(prob, 0, workspace, workspace_bytes, &L)) return rc;
    if ((out_rgb == nullptr) != (tgt_rgb == nullptr)) return fail(VLG_ERR_ARG, "out_rgb and tgt_rgb go together");
    if ((logits == nullptr) != (tgt_label == nullptr)) return fail(VLG_ERR_ARG, "logits and tgt_label go together");
    return run_pass1(prob, false, out_rgb, logits, nullptr, tgt_rgb, tgt_label, nullptr, d_out_rgb, d_logits,
                     d_out_rgb != nullptr || d_logits != nullptr, out_argmax, loss_out, L, (cudaStream_t)stream);
}

int vlg_frame_affine(const vlg_problem_t *prob, const float *in_rgb, int32_t in_is_nchw, const float *a3, const float *b3,
                     int32_t denormalize, int32_t flip_w, void *out_rgb, const int64_t *label_in, int64_t *label_out,
                     void *stream) {
    int rc = check_problem(prob);
    if (rc) return rc;
    if ((in_rgb == nullptr) != (out_rgb == nullptr)) return fail(VLG_ERR_ARG, "in_rgb and out_rgb go together");
    if ((label_in == nullptr) != (label_out == nullptr)) return fail(VLG_ERR_ARG, "label_in and label_out go together");
    if (in_rgb && (!a3 || !b3)) return fail(VLG_ERR_ARG, "a3 / b3 (3 host floats each) are required");
    if (in_rgb && (const void *)in_rgb == (const void *)out_rgb && (flip_w || in_is_nchw))
        return fail(VLG_ERR_ARG, "in-place only without flip and re-layout");
    if (label_in && label_in == label_out) return fail(VLG_ERR_ARG, "labels cannot be flipped in place");
    cudaStream_t st = (cudaStream_t)stream;
    if (in_rgb) {
        FrameAffine fa;
        for (int c = 0; c < 3; ++c) { fa.a[c] = a3[c]; fa.b[c] = b3[c]; }
        fa.denorm = denormalize ? 1 : 0;
        rc = with_type(prob->dtype, [&](auto t) {
            return launch_frame_affine<typename decltype(t)::type>(prob, fa, in_rgb, in_is_nchw != 0, flip_w ? 1 : 0, out_rgb, st);
        });
        if (rc) return rc;
    }
    if (label_in) {
        const int64_t P = prob->N * prob->H * prob->W;
        if (flip_w) {
            flip_labels_kernel<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(P, (int)prob->W, label_in, label_out);
            rc = check_launch("flip_labels_kernel");
        } else {
            cudaError_t e = cudaMemcpyAsync(label_out, label_in, (size_t)P * sizeof(int64_t), cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) rc = fail(VLG_ERR_CUDA, "label copy: %s", cudaGetErrorString(e));
        }
    }
    return rc;
}

int vlg_scale_grads(void *g, int64_t n, int32_t dtype, const float *scale, void *stream) {
    if (!g || !scale || n < 0) return fail(VLG_ERR_ARG, "bad arguments to vlg_scale_grads");
    if (n == 0) return VLG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == VLG_F32) scale_kernel<float><<<sm_count() * 8, 256, 0, st>>>((float *)g, n, scale);
    else if (dtype == VLG_BF16) scale_kernel<__nv_bfloat16><<<sm_count() * 8, 256, 0, st>>>((__nv_bfloat16 *)g, n, scale);
    else return fail(VLG_ERR_ARG, "bad dtype");
    return check_launch("scale_kernel");
}

int vlg_scale_grads_multi(int32_t count, void *const *g, const int64_t *n, const int32_t *dtype, const float *scale, void *stream) {
    if (count < 0 || count > 4 || !scale || (count && (!g || !n || !dtype))) return fail(VLG_ERR_ARG, "bad arguments to vlg_scale_grads_multi");
    ScaleSet s{};
    for (int b = 0; b < count; ++b) {
        if (!g[b] || n[b] < 0 || (dtype[b] != VLG_F32 && dtype[b] != VLG_BF16)) return fail(VLG_ERR_ARG, "vlg_scale_grads_multi: bad buffer %d", b);
        if (n[b] == 0) continue;
        s.g[s.count] = g[b]; s.n[s.count] = n[b]; s.dtype[s.count] = dtype[b]; ++s.count;
    }
    if (s.count == 0) return VLG_OK;
    scale_multi_kernel<<<sm_count() * 8, 256, 0, (cudaStream_t)stream>>>(s, scale);
    return check_launch("scale_multi_kernel");
}

int vlg_read_status(void *workspace, size_t workspace_bytes, uint32_t *host_status, void *stream) {
    if (!workspace || workspace_bytes < sizeof(WsHeader) || !host_status) return fail(VLG_ERR_ARG, "bad arguments");
    cudaError_t e = cudaMemcpyAsync(host_status, workspace, sizeof(uint32_t), cudaMemcpyDeviceToHost, (cudaStream_t)stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);
    if (e != cudaSuccess) return fail(VLG_ERR_CUDA, "read status: %s", cudaGetErrorString(e));
    return VLG_OK;
}

}  // extern "C"
