// vlg_metrics.cuh -- confusion matrix of predicted layouts against target labels (vlg_confusion).
//
// The reference's validation and rollout only dump torch.argmax(seg, 1) (src/trainer.py:342,467); per-class IoU, mIoU
// and pixel accuracy all follow from the K x K confusion matrix counted here.  Memory-bound by design: one pass over
// the prediction (int64 labels, or the K scores of a pixel and their argmax) and the int64 target.
//
//   labels          8 + 8 = 16 B/px   two labels per 128-bit load, kConfUnroll loads in flight per thread and array
//   layout NHWC     K*sizeof(T) + 8   thread per pixel, load_px<T,K>
//   layout NCHW     K*sizeof(T) + 8   thread per pixel, k at stride H*W: a warp reads 32 consecutive values per k, so
//                                     the network's plain-contiguous logits are read coalesced without a permute-copy
//
// Persistent grid; every CTA owns one contiguous run of pixels and keeps one uint32 histogram of K*K+1 bins per warp in
// shared memory (no contention between warps).  Updates are warp-aggregated: __match_any_sync on the bin, the first lane
// of each group adds its popcount -- real layouts are piecewise constant, so most lanes of a warp share a bin.  At the
// end the warps' histograms are summed and every non-zero bin goes to `counts` as one 64-bit integer atomicAdd: the
// result does not depend on the launch configuration or the schedule.
#pragma once
#include "vlg_device.cuh"

namespace vlg {

enum { kConfLabels = 0, kConfNhwc = 1, kConfNchw = 2 };
constexpr int kConfThreads = 256, kConfWarps = kConfThreads / 32;
constexpr int kConfUnroll = 4;   // label mode: 128-bit loads in flight per thread and label array

struct ConfParams {
    const void *layout;           // [N,H,W,K] (kConfNhwc) or [N,K,H,W] (kConfNchw) of T
    const int64_t *pred;          // [N,H,W] (kConfLabels)
    const int64_t *tgt;           // [N,H,W]
    unsigned long long *counts;   // K*K + 1: rows = target, columns = prediction, then the skipped pixels
    int64_t P;                    // N*H*W < 2^31 (check_problem)
    int64_t ignore_index;
    unsigned HW;
    int vec;                      // kConfLabels: both label arrays 16-byte aligned
};

// Adds one pixel (target t, prediction p) to the warp's histogram.  Called by all 32 lanes together; `live` == false
// lanes take part in the match only.
template <int K>
__device__ __forceinline__ void conf_count(unsigned *hist, bool live, int64_t t, int64_t p, int64_t ignore_index) {
    int bin = -1;
    if (live && t != ignore_index) bin = (t >= 0 && t < K && p >= 0 && p < K) ? (int)t * K + (int)p : K * K;
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(hist + bin, (unsigned)__popc(peers));
}

template <typename T, int K, int MODE>
__global__ void __launch_bounds__(kConfThreads) confusion_kernel(const ConfParams p) {
    constexpr int NB = K * K + 1;
    __shared__ unsigned s_hist[kConfWarps][NB];
    for (int b = threadIdx.x; b < kConfWarps * NB; b += kConfThreads) (&s_hist[0][0])[b] = 0u;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned *hist = s_hist[w];
    // every loop below advances by a warp-uniform base, so all 32 lanes reach each __match_any_sync
    if constexpr (MODE == kConfLabels) {
        if (p.vec) {
            const longlong2 *t2 = reinterpret_cast<const longlong2 *>(p.tgt);
            const longlong2 *p2 = reinterpret_cast<const longlong2 *>(p.pred);
            const int64_t units = p.P >> 1, chunk = (units + gridDim.x - 1) / gridDim.x;
            const int64_t lo = (int64_t)blockIdx.x * chunk, hi = min(lo + chunk, units);
            for (int64_t base = lo + w * 32 * kConfUnroll; base < hi; base += kConfThreads * kConfUnroll) {
                longlong2 tv[kConfUnroll], pv[kConfUnroll];
#pragma unroll
                for (int j = 0; j < kConfUnroll; ++j) {
                    const int64_t u = base + j * 32 + lane;
                    tv[j] = pv[j] = make_longlong2(0, 0);
                    if (u < hi) { tv[j] = __ldg(t2 + u); pv[j] = __ldg(p2 + u); }
                }
#pragma unroll
                for (int j = 0; j < kConfUnroll; ++j) {
                    const bool live = base + j * 32 + lane < hi;
                    conf_count<K>(hist, live, tv[j].x, pv[j].x, p.ignore_index);
                    conf_count<K>(hist, live, tv[j].y, pv[j].y, p.ignore_index);
                }
            }
            if ((p.P & 1) && blockIdx.x == 0 && w == 0)   // the odd last pixel
                conf_count<K>(hist, lane == 0, __ldg(p.tgt + p.P - 1), __ldg(p.pred + p.P - 1), p.ignore_index);
        } else {
            const int64_t chunk = (p.P + gridDim.x - 1) / gridDim.x;
            const int64_t lo = (int64_t)blockIdx.x * chunk, hi = min(lo + chunk, p.P);
            for (int64_t base = lo + w * 32 * kConfUnroll; base < hi; base += kConfThreads * kConfUnroll) {
                int64_t tv[kConfUnroll], pv[kConfUnroll];
#pragma unroll
                for (int j = 0; j < kConfUnroll; ++j) {
                    const int64_t i = base + j * 32 + lane;
                    tv[j] = pv[j] = 0;
                    if (i < hi) { tv[j] = __ldg(p.tgt + i); pv[j] = __ldg(p.pred + i); }
                }
#pragma unroll
                for (int j = 0; j < kConfUnroll; ++j)
                    conf_count<K>(hist, base + j * 32 + lane < hi, tv[j], pv[j], p.ignore_index);
            }
        }
    } else {
        const T *lay = static_cast<const T *>(p.layout);
        const int64_t chunk = (p.P + gridDim.x - 1) / gridDim.x;
        const int64_t lo = (int64_t)blockIdx.x * chunk, hi = min(lo + chunk, p.P);
        for (int64_t base = lo + w * 32; base < hi; base += kConfThreads) {
            const int64_t i = base + lane;
            const bool live = i < hi;
            int64_t t = 0, pr = 0;
            if (live) {
                float z[K];
                if constexpr (MODE == kConfNhwc) {
                    load_px<T, K>(lay + i * K, z);
                } else {
                    // N*H*W < 2^31: 32-bit divisions
                    const unsigned n = (unsigned)i / p.HW, r = (unsigned)i - n * p.HW;
                    const T *src = lay + (int64_t)n * K * p.HW + r;
#pragma unroll
                    for (int k = 0; k < K; ++k) z[k] = to_f<T>(__ldg(src + (int64_t)k * p.HW));
                }
                pr = first_max_index<K>(z);
                t = __ldg(p.tgt + i);
            }
            conf_count<K>(hist, live, t, pr, p.ignore_index);
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < NB; b += kConfThreads) {
        unsigned s = 0;
#pragma unroll
        for (int r = 0; r < kConfWarps; ++r) s += s_hist[r][b];
        if (s) atomicAdd(p.counts + b, (unsigned long long)s);
    }
}

}  // namespace vlg
