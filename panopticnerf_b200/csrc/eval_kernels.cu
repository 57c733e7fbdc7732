// eval_kernels.cu — on-device evaluation of rendered frames (the reference's `run.py --type evaluate`): semantic
// confusion matrix, panoptic quality, PSNR / SSIM and depth error, accumulated frame by frame into a caller-owned
// statistics buffer (layout in include/pnr.h).  Integer statistics are added with integer atomics (exact); every
// floating-point sum is formed from per-block partials added in a fixed order by one thread, so the statistics are
// bit-identical from run to run and depend only on the frames and the order they are passed in.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include "../../include/pnr.h"
#include "common.cuh"

namespace pnr {
namespace {

constexpr int kThreads = 256;
constexpr int kMaxPartials = 1024;          // per-block partials of each floating-point sum (fixed grid, fixed order)
constexpr int kSegCap = PNR_EVAL_MAX_SEGMENTS;
constexpr int kVoidCol = kSegCap;           // joint histogram column of GT-void pixels
constexpr int kJointLd = kSegCap + 1;
constexpr int kSsimTw = 32, kSsimTh = 16, kSsimR = 5;   // SSIM output tile and window radius (11 x 11)

enum { P_PSNR = 0, P_SSIM, P_ABS_REL, P_SQ_REL, P_SQ_ERR, P_SQ_LOG, P_NUM };

__host__ __device__ inline size_t align256(size_t b) { return (b + 255) & ~size_t(255); }
inline int partial_blocks(int64_t R) { return (int)(R / kThreads + 1 < kMaxPartials ? R / kThreads + 1 : kMaxPartials); }

// Workspace layout: the PQ region is contiguous so that one memset clears it per frame.
struct Ws {
  double* partials;              // [P_NUM][kMaxPartials]
  int32_t* idx[2];               // [C * div] per side: presence flag, then (after the scan) the segment's index
  int32_t* keys[2];              // [kSegCap] per side: segment key, ascending
  int32_t* counts;               // [2] distinct segments per side (may exceed kSegCap: overflow)
  int32_t* p_area;               // [kSegCap]
  int32_t* g_area;               // [kSegCap + 1]
  int32_t* g_matched;            // [kSegCap]
  int32_t* p_state;              // [kSegCap] 0 = TP, 1 = FP, 2 = unmatched but ignored (void / crowd)
  int32_t* joint;                // [kSegCap][kJointLd] |p ∩ g|, column kVoidCol = |p ∩ GT-void|
  double* p_iou;                 // [kSegCap]
  char* pq_begin; size_t pq_bytes;
  size_t total;
};

Ws carve(char* base, int32_t C, int32_t div) {
  Ws w{};
  size_t o = 0;
  auto take = [&](size_t b) { char* p = base ? base + o : nullptr; o += align256(b); return p; };
  w.partials = (double*)take(sizeof(double) * P_NUM * kMaxPartials);
  if (C > 0 && div > 0) {
    const size_t n = (size_t)C * (size_t)div;
    w.pq_begin = base ? base + o : nullptr;
    const size_t o0 = o;
    w.idx[0] = (int32_t*)take(4 * n);
    w.idx[1] = (int32_t*)take(4 * n);
    w.keys[0] = (int32_t*)take(4 * kSegCap);
    w.keys[1] = (int32_t*)take(4 * kSegCap);
    w.counts = (int32_t*)take(4 * 2);
    w.p_area = (int32_t*)take(4 * kSegCap);
    w.g_area = (int32_t*)take(4 * (kSegCap + 1));
    w.g_matched = (int32_t*)take(4 * kSegCap);
    w.p_state = (int32_t*)take(4 * kSegCap);
    w.joint = (int32_t*)take(4 * (size_t)kSegCap * kJointLd);
    w.pq_bytes = o - o0;
    w.p_iou = (double*)take(8 * kSegCap);
  }
  w.total = o;
  return w;
}

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// arr[key] += number of lanes holding `key` (one atomic per distinct key in the warp; key < 0 adds nothing).
// Every lane of the warp must call it.
__device__ __forceinline__ void warp_count(int32_t* arr, int key) {
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  if (key >= 0 && lane_id() == __ffs(peers) - 1) atomicAdd(arr + key, (int32_t)__popc(peers));
}

// Fixed-order tree sum over the block (blockDim.x == kThreads); the result is valid in thread 0.
__device__ double block_sum(double v, double* sh) {
  sh[threadIdx.x] = v;
  __syncthreads();
  for (int s = kThreads / 2; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  const double r = sh[0];
  __syncthreads();
  return r;
}

__device__ __forceinline__ int64_t* stat_i64(void* stats, int word) { return reinterpret_cast<int64_t*>(stats) + word; }
__device__ __forceinline__ double* stat_f64(void* stats, int word) { return reinterpret_cast<double*>(stats) + word; }
__device__ __forceinline__ void add_i64(void* stats, int word, int64_t v) {
  if (v) atomicAdd(reinterpret_cast<unsigned long long*>(stats) + word, (unsigned long long)v);
}

// ------------------------------------------------------------------------------------------------ confusion matrix
// Per-CTA shared histogram (C <= 64: 16 KB), warp-aggregated shared atomics, flushed with one 64-bit integer atomic per
// non-zero bin.
__global__ void __launch_bounds__(kThreads) confusion_kernel(const int16_t* __restrict__ pred,
                                                             const int32_t* __restrict__ gt, int64_t R, int C,
                                                             void* stats) {
  __shared__ int32_t hist[PNR_EVAL_MAX_CLASSES * PNR_EVAL_MAX_CLASSES];
  for (int i = threadIdx.x; i < C * C; i += kThreads) hist[i] = 0;
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  for (int64_t base = (int64_t)blockIdx.x * kThreads + (threadIdx.x & ~31); base < R; base += stride) {
    const int64_t r = base + lane_id();
    int key = -1;
    if (r < R) {
      const int g = gt[r], p = pred[r];
      if (g >= 0 && g < C && p >= 0 && p < C) key = g * C + p;
    }
    warp_count(hist, key);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C * C; i += kThreads) add_i64(stats, PNR_EVAL_HEADER_WORDS + i, hist[i]);
}

// ------------------------------------------------------------------------------------------------ panoptic quality
// Segment key of a panoptic id: -1 = void; stuff categories drop the instance part (one segment per category).
__device__ __forceinline__ int seg_key(int id, int C, int div, const uint8_t* is_thing) {
  if (id < 0) return -1;
  const int cat = id / div;
  if (cat >= C) return -1;
  return is_thing[cat] ? id : cat * div;
}

__global__ void __launch_bounds__(kThreads) pq_mark_kernel(const int32_t* __restrict__ pred,
                                                           const int32_t* __restrict__ gt, int64_t R, int C, int div,
                                                           const uint8_t* __restrict__ is_thing, int32_t* fp,
                                                           int32_t* fg) {
  const int64_t r = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (r >= R) return;
  const int kp = seg_key(pred[r], C, div, is_thing), kg = seg_key(gt[r], C, div, is_thing);
  if (kp >= 0) fp[kp] = 1;
  if (kg >= 0) fg[kg] = 1;
}

// One block per side: exclusive scan of the presence flags over the n = C * div keys, in place (flag -> index of the
// segment in ascending key order), the ascending key list (first kSegCap) and the number of distinct segments.
__global__ void __launch_bounds__(1024) pq_scan_kernel(int32_t* idx0, int32_t* idx1, int n, int32_t* keys0,
                                                       int32_t* keys1, int32_t* counts) {
  __shared__ int32_t sh[1024];
  int32_t* f = blockIdx.x ? idx1 : idx0;
  int32_t* keys = blockIdx.x ? keys1 : keys0;
  const int t = threadIdx.x;
  const int chunk = (n + 1023) / 1024;
  const int lo = min(n, t * chunk), hi = min(n, lo + chunk);
  int s = 0;
  for (int i = lo; i < hi; ++i) s += f[i];
  sh[t] = s;
  __syncthreads();
  for (int d = 1; d < 1024; d <<= 1) {         // inclusive Hillis-Steele scan
    const int v = t >= d ? sh[t - d] : 0;
    __syncthreads();
    sh[t] += v;
    __syncthreads();
  }
  int run = sh[t] - s;
  for (int i = lo; i < hi; ++i) {
    if (f[i]) {
      f[i] = run;
      if (run < kSegCap) keys[run] = i;
      ++run;
    }
  }
  if (t == 1023) counts[blockIdx.x] = sh[1023];
}

// Areas and the joint intersection histogram; a road segment puts ~1e5 pixels on one bin, so every count is
// warp-aggregated.  Skipped when a side has more than kSegCap segments (the finalize kernel records the overflow).
__global__ void __launch_bounds__(kThreads) pq_hist_kernel(const int32_t* __restrict__ pred,
                                                           const int32_t* __restrict__ gt, int64_t R, int C, int div,
                                                           const uint8_t* __restrict__ is_thing, Ws w) {
  if (w.counts[0] > kSegCap || w.counts[1] > kSegCap) return;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  for (int64_t base = (int64_t)blockIdx.x * kThreads + (threadIdx.x & ~31); base < R; base += stride) {
    const int64_t r = base + lane_id();
    int pi = -1, gi = -1;
    if (r < R) {
      const int kp = seg_key(pred[r], C, div, is_thing), kg = seg_key(gt[r], C, div, is_thing);
      pi = kp >= 0 ? w.idx[0][kp] : -1;
      gi = kg >= 0 ? w.idx[1][kg] : kVoidCol;
    }
    warp_count(w.g_area, gi);
    warp_count(w.p_area, pi);
    warp_count(w.joint, pi >= 0 ? pi * kJointLd + gi : -1);
  }
}

__device__ __forceinline__ int lower_bound(const int32_t* a, int n, int v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int m = (lo + hi) >> 1;
    if (a[m] < v) lo = m + 1; else hi = m;
  }
  return lo;
}

// One thread per predicted segment: its match among the non-crowd GT segments of its category (IoU > 0.5, strict; at
// most one can pass, segments of one side being disjoint) or, unmatched, whether it lies mostly on GT void / crowd.
__global__ void __launch_bounds__(kThreads) pq_match_kernel(int C, int div, const uint8_t* __restrict__ is_thing, Ws w) {
  const int np = w.counts[0], ng = w.counts[1];
  const int p = blockIdx.x * kThreads + threadIdx.x;
  if (np > kSegCap || ng > kSegCap || p >= np) return;
  const int cat = w.keys[0][p] / div;
  const bool thing = is_thing[cat] != 0;
  const int32_t* row = w.joint + (size_t)p * kJointLd;
  const int64_t ap = w.p_area[p], on_void = row[kVoidCol];
  const int g0 = lower_bound(w.keys[1], ng, cat * div), g1 = lower_bound(w.keys[1], ng, (cat + 1) * div);
  int state = 1;
  double iou = 0.0;
  int64_t on_crowd = 0;
  for (int g = g0; g < g1; ++g) {
    const int64_t inter = row[g];
    if (thing && w.keys[1][g] == cat * div) { on_crowd = inter; continue; }   // crowd region: never matched
    if (inter == 0) continue;
    const int64_t denom = ap + w.g_area[g] - inter - on_void;
    if (2 * inter > denom) {
      state = 0;
      iou = (double)inter / (double)denom;
      w.g_matched[g] = 1;
    }
  }
  if (state != 0 && 2 * (on_void + on_crowd) > ap) state = 2;
  w.p_state[p] = state;
  w.p_iou[p] = iou;
}

// ------------------------------------------------------------------------------------------------ image metrics
struct PixelArgs {
  const float* rgb_pred; const float* rgb_gt;
  const float* depth_pred; const float* depth_gt;
  float min_depth, max_depth;
  int64_t R;
  double* partials;
  void* stats;
};

// Squared colour error and the depth sums of the pixels of the block's grid-stride share, reduced in a fixed order
// per block; the depth counts go to the statistics with integer atomics.
__global__ void __launch_bounds__(kThreads) pixel_kernel(PixelArgs a) {
  __shared__ double sh[kThreads];
  double se = 0.0, abs_rel = 0.0, sq_rel = 0.0, sq_err = 0.0, sq_log = 0.0;
  int64_t n_valid = 0, n_d1 = 0, n_d2 = 0, n_d3 = 0;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  for (int64_t r = (int64_t)blockIdx.x * kThreads + threadIdx.x; r < a.R; r += stride) {
    if (a.rgb_pred) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const double d = (double)a.rgb_pred[r * 3 + c] - (double)a.rgb_gt[r * 3 + c];
        se += d * d;
      }
    }
    if (a.depth_pred) {
      const float gf = a.depth_gt[r];
      if (gf > 0.f && gf <= a.max_depth) {
        const double g = gf, p = fminf(fmaxf(a.depth_pred[r], a.min_depth), a.max_depth);
        const double d = p - g, dl = log(p) - log(g), ratio = fmax(p / g, g / p);
        abs_rel += fabs(d) / g;
        sq_rel += d * d / g;
        sq_err += d * d;
        sq_log += dl * dl;
        ++n_valid;
        n_d1 += ratio < 1.25;
        n_d2 += ratio < 1.25 * 1.25;
        n_d3 += ratio < 1.25 * 1.25 * 1.25;
      }
    }
  }
  const int b = blockIdx.x;
  if (a.rgb_pred) {
    const double s = block_sum(se, sh);
    if (threadIdx.x == 0) a.partials[P_PSNR * kMaxPartials + b] = s;
  }
  if (a.depth_pred) {
    const double v[4] = {abs_rel, sq_rel, sq_err, sq_log};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const double s = block_sum(v[k], sh);
      if (threadIdx.x == 0) a.partials[(P_ABS_REL + k) * kMaxPartials + b] = s;
    }
    const int64_t cnt[4] = {n_valid, n_d1, n_d2, n_d3};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const double s = block_sum((double)cnt[k], sh);   // exact: counts < 2^53
      if (threadIdx.x == 0) add_i64(a.stats, PNR_EVAL_DEPTH_VALID + k, (int64_t)s);
    }
  }
}

struct SsimArgs {
  const float* x; const float* y;   // [H*W, 3]
  int H, W;
  double g[2 * kSsimR + 1];         // normalised 1-D Gaussian
  double* partials;
};

// SSIM over the valid region, one 32 x 16 tile of outputs per step (grid-stride over tiles, fixed grid): the window
// moments are separable, a horizontal pass into shared memory then a vertical one, all in fp64.
__global__ void __launch_bounds__(kThreads) ssim_kernel(SsimArgs a) {
  constexpr int IH = kSsimTh + 2 * kSsimR, IW = kSsimTw + 2 * kSsimR;
  __shared__ float sx[IH][IW], sy[IH][IW];
  __shared__ double hm[5][IH][kSsimTw];
  __shared__ double red[kThreads];
  const int Ho = a.H - 2 * kSsimR, Wo = a.W - 2 * kSsimR;
  const int tx_n = (Wo + kSsimTw - 1) / kSsimTw, tiles = tx_n * ((Ho + kSsimTh - 1) / kSsimTh);
  const double c1 = 0.01 * 0.01, c2 = 0.03 * 0.03;
  double acc = 0.0;
  for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int oy0 = (tile / tx_n) * kSsimTh, ox0 = (tile % tx_n) * kSsimTw;
    for (int c = 0; c < 3; ++c) {
      for (int i = threadIdx.x; i < IH * IW; i += kThreads) {
        const int iy = i / IW, ix = i % IW, yy = oy0 + iy, xx = ox0 + ix;
        const bool in = yy < a.H && xx < a.W;
        const int64_t o = ((int64_t)yy * a.W + xx) * 3 + c;
        sx[iy][ix] = in ? a.x[o] : 0.f;
        sy[iy][ix] = in ? a.y[o] : 0.f;
      }
      __syncthreads();
      for (int i = threadIdx.x; i < IH * kSsimTw; i += kThreads) {
        const int iy = i / kSsimTw, ix = i % kSsimTw;
        double m0 = 0, m1 = 0, m2 = 0, m3 = 0, m4 = 0;
#pragma unroll
        for (int k = 0; k <= 2 * kSsimR; ++k) {
          const double u = sx[iy][ix + k], v = sy[iy][ix + k], g = a.g[k];
          m0 += g * u; m1 += g * v; m2 += g * (u * u); m3 += g * (v * v); m4 += g * (u * v);
        }
        hm[0][iy][ix] = m0; hm[1][iy][ix] = m1; hm[2][iy][ix] = m2; hm[3][iy][ix] = m3; hm[4][iy][ix] = m4;
      }
      __syncthreads();
      for (int i = threadIdx.x; i < kSsimTh * kSsimTw; i += kThreads) {
        const int oy = i / kSsimTw, ox = i % kSsimTw;
        if (oy0 + oy >= Ho || ox0 + ox >= Wo) continue;
        double m[5] = {0, 0, 0, 0, 0};
#pragma unroll
        for (int k = 0; k <= 2 * kSsimR; ++k) {
          const double g = a.g[k];
#pragma unroll
          for (int j = 0; j < 5; ++j) m[j] += g * hm[j][oy + k][ox];
        }
        const double mx = m[0], my = m[1];
        const double vx = fmax(m[2] - mx * mx, 0.0), vy = fmax(m[3] - my * my, 0.0), cxy = m[4] - mx * my;
        acc += ((2.0 * mx * my + c1) * (2.0 * cxy + c2)) / ((mx * mx + my * my + c1) * (vx + vy + c2));
      }
      __syncthreads();
    }
  }
  const double s = block_sum(acc, red);
  if (threadIdx.x == 0) a.partials[P_SSIM * kMaxPartials + blockIdx.x] = s;
}

// ------------------------------------------------------------------------------------------------ finalize
struct FinalArgs {
  int C, div;
  const uint8_t* is_thing;
  Ws w;
  int pq;                // panoptic inputs given
  int n_pixel, n_ssim;   // partial counts (0: family absent)
  int depth;
  double inv_rgb, inv_ssim;   // 1 / (3 R), 1 / (3 (H-10) (W-10))
  void* stats;
};

// One block: thread c < C adds category c's PQ terms (its segments in ascending key order), thread 64 + k sums the
// partials of family k in block order.  One thread owns every floating-point statistic it writes.
__global__ void __launch_bounds__(128) finalize_kernel(FinalArgs a) {
  const int t = threadIdx.x;
  if (a.pq && t < a.C) {
    const Ws& w = a.w;
    const int np = w.counts[0], ng = w.counts[1];
    if (np > kSegCap || ng > kSegCap) {
      if (t == 0) *stat_i64(a.stats, PNR_EVAL_OVERFLOW) += 1;
    } else {
      if (t == 0) *stat_i64(a.stats, PNR_EVAL_PQ_FRAMES) += 1;
      const int lo = t * a.div, hi = (t + 1) * a.div;
      int64_t tp = 0, fp = 0, fn = 0;
      double iou = 0.0;
      for (int p = lower_bound(w.keys[0], np, lo); p < np && w.keys[0][p] < hi; ++p) {
        tp += w.p_state[p] == 0;
        fp += w.p_state[p] == 1;
        iou += w.p_iou[p];
      }
      const bool thing = a.is_thing[t] != 0;
      for (int g = lower_bound(w.keys[1], ng, lo); g < ng && w.keys[1][g] < hi; ++g)
        fn += !w.g_matched[g] && !(thing && w.keys[1][g] == lo);
      const int base = PNR_EVAL_HEADER_WORDS + a.C * a.C;
      *stat_i64(a.stats, base + t) += tp;
      *stat_i64(a.stats, base + a.C + t) += fp;
      *stat_i64(a.stats, base + 2 * a.C + t) += fn;
      *stat_f64(a.stats, base + 3 * a.C + t) += iou;
    }
  }
  const int k = t - 64;
  if (k < 0 || k >= P_NUM) return;
  const bool depth_fam = k >= P_ABS_REL;
  const int n = k == P_SSIM ? a.n_ssim : (k == P_PSNR || a.depth ? a.n_pixel : 0);
  if (n == 0 || (k == P_PSNR && a.inv_rgb == 0.0) || (depth_fam && !a.depth)) return;
  const double* part = a.w.partials + k * kMaxPartials;
  double s = 0.0;
  for (int b = 0; b < n; ++b) s += part[b];
  if (k == P_PSNR) {
    *stat_f64(a.stats, PNR_EVAL_PSNR_SUM) += -10.0 * log10(s * a.inv_rgb);
    *stat_i64(a.stats, PNR_EVAL_PSNR_FRAMES) += 1;
  } else if (k == P_SSIM) {
    *stat_f64(a.stats, PNR_EVAL_SSIM_SUM) += s * a.inv_ssim;
    *stat_i64(a.stats, PNR_EVAL_SSIM_FRAMES) += 1;
  } else {
    *stat_f64(a.stats, PNR_EVAL_ABS_REL_SUM + (k - P_ABS_REL)) += s;
  }
}

}  // namespace
}  // namespace pnr

using namespace pnr;

extern "C" size_t pnr_eval_stats_bytes(int32_t C) {
  if (C < 0 || C > PNR_EVAL_MAX_CLASSES) return 0;
  return sizeof(int64_t) * ((size_t)PNR_EVAL_HEADER_WORDS + (size_t)C * C + 4 * (size_t)C);
}

extern "C" size_t pnr_eval_workspace_bytes(int64_t R, int32_t C, int32_t label_divisor) {
  (void)R;
  if (C < 0 || C > PNR_EVAL_MAX_CLASSES) return 0;
  if (label_divisor > 0 && (int64_t)C * label_divisor > PNR_EVAL_MAX_KEYS) return 0;
  return carve(nullptr, C, label_divisor > 0 ? label_divisor : 0).total;
}

extern "C" int pnr_eval_frame(const pnr_eval_args* args, void* stream) {
  PNR_CHECK_ARG(args, "pnr_eval_frame: null args");
  const pnr_eval_args& a = *args;
  PNR_CHECK_ARG(a.R >= 0 && a.R < INT32_MAX, "pnr_eval_frame: R=%lld outside [0, 2^31)", (long long)a.R);
  PNR_CHECK_ARG(a.C >= 0 && a.C <= PNR_EVAL_MAX_CLASSES, "pnr_eval_frame: C=%d outside [0, %d]", a.C,
                PNR_EVAL_MAX_CLASSES);
  PNR_CHECK_ARG(a.stats, "pnr_eval_frame: missing stats buffer (pnr_eval_stats_bytes(C) bytes, zeroed once)");
  const bool sem = a.sem_pred || a.sem_gt, pan = a.pan_pred || a.pan_gt, rgb = a.rgb_pred || a.rgb_gt,
             depth = a.depth_pred || a.depth_gt;
  PNR_CHECK_ARG(!sem || (a.sem_pred && a.sem_gt), "pnr_eval_frame: sem_pred and sem_gt go together");
  PNR_CHECK_ARG(!pan || (a.pan_pred && a.pan_gt), "pnr_eval_frame: pan_pred and pan_gt go together");
  PNR_CHECK_ARG(!rgb || (a.rgb_pred && a.rgb_gt), "pnr_eval_frame: rgb_pred and rgb_gt go together");
  PNR_CHECK_ARG(!depth || (a.depth_pred && a.depth_gt), "pnr_eval_frame: depth_pred and depth_gt go together");
  PNR_CHECK_ARG(!(sem || pan) || a.C > 0, "pnr_eval_frame: semantic / panoptic metrics need C > 0");
  if (pan) {
    PNR_CHECK_ARG(a.is_thing, "pnr_eval_frame: panoptic metrics need is_thing [C]");
    PNR_CHECK_ARG(a.label_divisor > 0, "pnr_eval_frame: label_divisor=%d must be positive", a.label_divisor);
    PNR_CHECK_ARG((int64_t)a.C * a.label_divisor <= PNR_EVAL_MAX_KEYS,
                  "pnr_eval_frame: C * label_divisor = %lld exceeds %d", (long long)a.C * a.label_divisor,
                  PNR_EVAL_MAX_KEYS);
  }
  const bool ssim = a.H != 0 || a.W != 0;
  if (ssim) {
    PNR_CHECK_ARG((int64_t)a.H * a.W == a.R, "pnr_eval_frame: H*W = %d*%d != R=%lld (pass H = W = 0 to skip SSIM)",
                  a.H, a.W, (long long)a.R);
    PNR_CHECK_ARG(a.H > 2 * kSsimR && a.W > 2 * kSsimR, "pnr_eval_frame: SSIM needs H, W >= 11 (got %d x %d)", a.H, a.W);
    PNR_CHECK_ARG(rgb, "pnr_eval_frame: SSIM (H, W given) needs rgb_pred / rgb_gt");
  }
  if (depth)
    PNR_CHECK_ARG(a.min_depth > 0.f && a.max_depth >= a.min_depth, "pnr_eval_frame: need 0 < min_depth <= max_depth");
  const size_t need = pnr_eval_workspace_bytes(a.R, a.C, pan ? a.label_divisor : 0);
  PNR_CHECK_ARG(a.workspace && a.workspace_bytes >= need,
                "pnr_eval_frame: workspace of %zu bytes, pnr_eval_workspace_bytes gives %zu", a.workspace_bytes, need);
  PNR_CHECK_ARG(((uintptr_t)a.workspace & 255) == 0 && ((uintptr_t)a.stats & 7) == 0,
                "pnr_eval_frame: workspace must be 256-byte and stats 8-byte aligned");
  if (a.R == 0) return PNR_OK;

  cudaStream_t st = (cudaStream_t)stream;
  const Ws w = carve((char*)a.workspace, a.C, pan ? a.label_divisor : 0);
  const int nb = partial_blocks(a.R);
  if (sem) {
    confusion_kernel<<<nb < 296 ? nb : 296, kThreads, 0, st>>>(a.sem_pred, a.sem_gt, a.R, a.C, a.stats);
    PNR_LAUNCH_CHECK("confusion_kernel");
  }
  if (pan) {
    PNR_CUDA(cudaMemsetAsync(w.pq_begin, 0, w.pq_bytes, st));
    pq_mark_kernel<<<(unsigned)((a.R + kThreads - 1) / kThreads), kThreads, 0, st>>>(
        a.pan_pred, a.pan_gt, a.R, a.C, a.label_divisor, a.is_thing, w.idx[0], w.idx[1]);
    PNR_LAUNCH_CHECK("pq_mark_kernel");
    pq_scan_kernel<<<2, 1024, 0, st>>>(w.idx[0], w.idx[1], a.C * a.label_divisor, w.keys[0], w.keys[1], w.counts);
    PNR_LAUNCH_CHECK("pq_scan_kernel");
    pq_hist_kernel<<<nb, kThreads, 0, st>>>(a.pan_pred, a.pan_gt, a.R, a.C, a.label_divisor, a.is_thing, w);
    PNR_LAUNCH_CHECK("pq_hist_kernel");
    pq_match_kernel<<<kSegCap / kThreads, kThreads, 0, st>>>(a.C, a.label_divisor, a.is_thing, w);
    PNR_LAUNCH_CHECK("pq_match_kernel");
  }
  if (rgb || depth) {
    PixelArgs p{rgb ? a.rgb_pred : nullptr, a.rgb_gt, depth ? a.depth_pred : nullptr, a.depth_gt, a.min_depth,
                a.max_depth, a.R, w.partials, a.stats};
    pixel_kernel<<<nb, kThreads, 0, st>>>(p);
    PNR_LAUNCH_CHECK("pixel_kernel");
  }
  int n_ssim = 0;
  if (ssim) {
    SsimArgs s{a.rgb_pred, a.rgb_gt, a.H, a.W, {}, w.partials};
    double gs = 0.0;
    for (int k = 0; k <= 2 * kSsimR; ++k) {
      const double f = (k - kSsimR) / 1.5;
      s.g[k] = exp(-0.5 * f * f);
      gs += s.g[k];
    }
    for (int k = 0; k <= 2 * kSsimR; ++k) s.g[k] /= gs;
    const int Ho = a.H - 2 * kSsimR, Wo = a.W - 2 * kSsimR;
    const int tiles = ((Wo + kSsimTw - 1) / kSsimTw) * ((Ho + kSsimTh - 1) / kSsimTh);
    n_ssim = tiles < kMaxPartials ? tiles : kMaxPartials;
    ssim_kernel<<<n_ssim, kThreads, 0, st>>>(s);
    PNR_LAUNCH_CHECK("ssim_kernel");
  }
  FinalArgs f{a.C, pan ? a.label_divisor : 1, a.is_thing, w, pan ? 1 : 0, (rgb || depth) ? nb : 0, n_ssim,
              depth ? 1 : 0, rgb ? 1.0 / (3.0 * (double)a.R) : 0.0,
              ssim ? 1.0 / (3.0 * (double)(a.H - 2 * kSsimR) * (double)(a.W - 2 * kSsimR)) : 0.0, a.stats};
  finalize_kernel<<<1, 128, 0, st>>>(f);
  PNR_LAUNCH_CHECK("finalize_kernel");
  return PNR_OK;
}
