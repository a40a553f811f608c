// lm_train.cuh -- template extraction on the GPU (Detector::addTemplate after quantization), batched over views.
//
// Reference being replaced (linemodLevelup/linemodLevelup.cpp of meiqua/6DPose @ 619be57, "LL.cpp"; the host
// restatement is 6dpose_b200/training.py):
//   k_tr_prep       <- ColorGradientPyramid::extractTemplate's candidate scan (mask border, magnitude gate)
//                      and DepthNormalPyramid::extractTemplate's local mask + area             LL.cpp:589-620, 888-900, 956
//   k_tr_coldist    \
//   k_tr_normcand    > cv::distanceTransform(DIST_C, 3) per label + the candidate scan          LL.cpp:900-945
//   k_tr_normscore  /  score = distance / (candidates of that label)                             LL.cpp:946-950
//   (CUB)           <- std::stable_sort(candidates) by score, descending                        LL.cpp:625, 952
//   k_tr_select     <- QuantizedPyramid::selectScatteredFeatures                                 LL.cpp:279-318
// cropTemplates (LL.cpp:234-277) runs on the host after the copy back (lm_extract_templates).
//
// Every kernel takes one view per blockIdx.z (k_tr_normscore: one (view, level) per blockIdx.y, k_tr_select: one
// (view, level, modality) segment per block).  Candidates of a segment are appended in any order as 64-bit keys
//   (~score bits) << 32 | scan index << 3 | label
// Colour scores are integers and normal scores non-negative floats, whose bit patterns order like unsigned
// integers, so ascending keys = score descending, ties in row-major scan order: the order std::stable_sort gives
// the reference's scan-ordered list.  The key is unique, so any sort reproduces it.
#pragma once

#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#define TR_INF 0x3fffffff  // "no zero pixel in that direction" for the column pass of the distance transform

// Warp-aggregated append: one atomic per warp; every lane of the warp must call it (pred may be false).
__device__ __forceinline__ int tr_append(int* counter, bool pred) {
  const unsigned ball = __ballot_sync(0xffffffffu, pred);
  const int lane = threadIdx.x & 31;
  const int leader = ball ? __ffs(ball) - 1 : 0;
  int base = 0;
  if (ball && lane == leader) base = atomicAdd(counter, __popc(ball));
  base = __shfl_sync(0xffffffffu, base, leader);
  return base + __popc(ball & ((1u << lane) - 1u));
}

// Per pixel of one level: colour candidates (appended to segment (v, level, 0)), the normals' "foreground" label
// image (label where the eroded mask is set) and the eroded mask's area.
//   colour  (LL.cpp:596-620): label = hysteresis output without the mask, != 0; magnitude > 55^2; pixel in
//           mask - erode(mask, 3x3, BORDER_REPLICATE) (u8 values: nonzero <=> mask > min of its 3x3 neighbourhood)
//   normals (LL.cpp:893-900): local mask = erode(mask, 3x3, 2 iterations, BORDER_REPLICATE) = min over the 5x5
//           neighbourhood, coordinates clamped
// blocks of 32 x 8 pixels, blockIdx.z = view; per-view buffers are `fs` (angle, mag, nfg) / `ns` (normal, mask) apart.
__global__ void __launch_bounds__(256) k_tr_prep(int H, int W, int level, int L, const uint8_t* __restrict__ angle,
                                                const int32_t* __restrict__ mag, size_t fs, const uint8_t* __restrict__ normal,
                                                const uint8_t* __restrict__ mask, size_t ns, const uint8_t* __restrict__ has_mask,
                                                unsigned long long* __restrict__ keys, int* __restrict__ seg_end,
                                                uint8_t* __restrict__ nfg, int* __restrict__ area) {
  lm_pdl_wait();
  const int v = blockIdx.z;
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  const bool valid = x < W && y < H;
  const size_t p = valid ? (size_t)y * W + x : 0;
  const uint8_t* mk = has_mask[v] ? mask + v * ns : nullptr;
  bool in_c = valid, in_n = valid;
  if (valid && mk) {
    int m3 = 255, m5 = 255;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
      const int yy = min(max(y + dy, 0), H - 1);
#pragma unroll
      for (int dx = -2; dx <= 2; ++dx) {
        const int val = mk[(size_t)yy * W + min(max(x + dx, 0), W - 1)];
        m5 = min(m5, val);
        if (dy >= -1 && dy <= 1 && dx >= -1 && dx <= 1) m3 = min(m3, val);
      }
    }
    in_c = mk[p] > m3;
    in_n = m5 != 0;
  }
  const int seg = (v * L + level) * 2;
  const uint8_t a = valid ? angle[v * fs + p] : 0;
  const int mg = valid ? mag[v * fs + p] : 0;
  const bool cand = in_c && a != 0 && mg > 3025;  // squared magnitude > float(55) * float(55), exact as an integer
  const int pos = tr_append(&seg_end[seg], cand);
  if (cand) keys[pos] = ((unsigned long long)(~(uint32_t)mg) << 32) | ((unsigned long long)p << 3) | (unsigned)(__ffs(a) - 1);
  if (valid) nfg[v * fs + p] = in_n ? normal[v * ns + p] : 0;
  const unsigned inside = __ballot_sync(0xffffffffu, mk != nullptr && in_n);
  if (inside && (threadIdx.x & 31) == 0) atomicAdd(&area[v * L + level], __popc(inside));
}

// Column pass of the chessboard distance transform: per pixel of label c (nfg != 0), the distance along its column
// to the nearest pixel that is not c; beyond the image is far away (TR_INF), not zero.  Thread per column.
__global__ void __launch_bounds__(128) k_tr_coldist(int H, int W, const uint8_t* __restrict__ nfg, size_t fs, int* __restrict__ g) {
  lm_pdl_wait();
  const int x = blockIdx.x * 128 + threadIdx.x;
  if (x >= W) return;
  const uint8_t* f = nfg + blockIdx.z * fs + x;
  int* o = g + blockIdx.z * fs + x;
  int run = 0;
  uint8_t prev = 0;
  for (int y = 0; y < H; ++y) {
    const uint8_t c = f[(size_t)y * W];
    if (!c) run = 0;
    else if (y == 0) run = TR_INF;
    else run = prev == c ? (run >= TR_INF ? TR_INF : run + 1) : 1;
    o[(size_t)y * W] = run;
    prev = c;
  }
  run = 0;
  prev = 0;
  for (int y = H - 1; y >= 0; --y) {
    const uint8_t c = f[(size_t)y * W];
    if (!c) run = 0;
    else if (y == H - 1) run = TR_INF;
    else run = prev == c ? (run >= TR_INF ? TR_INF : run + 1) : 1;
    if (c) o[(size_t)y * W] = min(o[(size_t)y * W], run);
    prev = c;
  }
}

// Row pass + candidate scan of DepthNormalPyramid::extractTemplate (LL.cpp:900-945).  The L-infinity distance of a
// label-c pixel (x, y) is min over x' of max(|x - x'|, col(x', y)), where col is the column distance of a label-c
// pixel and 0 for any other pixel; the scan walks outwards and stops once |x - x'| reaches the best so far.  No
// pixel that is not c anywhere: FLT_MAX, as cv::distanceTransform returns.  Candidates (distance >= the level's
// extract threshold) go to segment (v, level, 1) with the integer distance in the high word (k_tr_normscore
// replaces it by the score); lcount counts them per label.
__global__ void __launch_bounds__(256) k_tr_normcand(int H, int W, int level, int L, int extract_threshold,
                                                    const uint8_t* __restrict__ nfg, const int* __restrict__ g, size_t fs,
                                                    unsigned long long* __restrict__ keys, int* __restrict__ seg_end,
                                                    int* __restrict__ lcount) {
  lm_pdl_wait();
  const int v = blockIdx.z;
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  const bool valid = x < W && y < H;
  const size_t p = valid ? (size_t)y * W + x : 0;
  const uint8_t* f = nfg + v * fs;
  const int* gc = g + v * fs;
  const uint8_t c = valid ? f[p] : 0;
  int best = TR_INF;
  if (c) {
    best = gc[p];
    for (int d = 1; d < best; ++d) {
      const bool lin = x - d >= 0, rin = x + d < W;
      if (!lin && !rin) break;
      if (lin) best = min(best, f[p - d] == c ? max(d, gc[p - d]) : d);
      if (rin) best = min(best, f[p + d] == c ? max(d, gc[p + d]) : d);
    }
  }
  const bool cand = c != 0 && best >= extract_threshold;
  const int seg = (v * L + level) * 2 + 1;
  const int pos = tr_append(&seg_end[seg], cand);
  const int label = c ? __ffs(c) - 1 : 0;
  if (cand) {
    const uint32_t hi = best >= TR_INF ? 0xffffffffu : (uint32_t)best;
    keys[pos] = ((unsigned long long)hi << 32) | ((unsigned long long)p << 3) | (unsigned)label;
  }
  const unsigned same = __match_any_sync(0xffffffffu, cand ? label : -1);
  if (cand && (threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(&lcount[(v * L + level) * 8 + label], __popc(same));
}

// score = float(distance) / float(candidates with that label), correctly rounded (LL.cpp:946-950).
// blockIdx.y = view * L + level.
__global__ void __launch_bounds__(256) k_tr_normscore(unsigned long long* __restrict__ keys, const int* __restrict__ seg_begin,
                                                     const int* __restrict__ seg_end, const int* __restrict__ lcount) {
  lm_pdl_wait();
  const int vl = blockIdx.y, seg = vl * 2 + 1;
  const int end = seg_end[seg];
  for (int i = seg_begin[seg] + blockIdx.x * 256 + threadIdx.x; i < end; i += gridDim.x * 256) {
    const unsigned long long k = keys[i];
    const uint32_t hi = (uint32_t)(k >> 32), lo = (uint32_t)k;
    const float dist = hi == 0xffffffffu ? FLT_MAX : __int2float_rn((int)hi);
    const float score = __fdiv_rn(dist, __int2float_rn(lcount[vl * 8 + (lo & 7)]));
    keys[i] = ((unsigned long long)(~__float_as_uint(score)) << 32) | lo;
  }
}

struct TrainSelect {
  int L, nf0;
  int cols[4], npix[4];
  int first[8];  // slot offset (in features) inside a view's output, slot = level * 2 + modality
  int F;         // features per view
};

// a squared integer distance d passes `d >= float32(distance * distance)` (LL.cpp:300) iff d >= ceil of that float
__device__ __forceinline__ long long tr_need(float distance) { return (long long)ceilf(__fmul_rn(distance, distance)); }

// selectScatteredFeatures (LL.cpp:279-318), one warp per (view, level, modality) segment of sorted candidates.
// Within one pass the distance is fixed and the kept set only grows, so a rejection is final for that pass: the
// warp tests 32 consecutive candidates against the kept set at once, keeps the first that passes and re-tests only
// the lanes after it against that one new feature.  A pass that keeps nothing only lowers the distance; the warp
// then skips straight to the first distance at which the farthest candidate passes (the passes in between keep
// nothing either).  Fewer candidates than features: seg_fail = 1 (addTemplate returns -1, LL.cpp:1956-1960).
// Dynamic shared memory: nf0 x 2 ints (the kept coordinates).
__global__ void __launch_bounds__(32) k_tr_select(TrainSelect s, const unsigned long long* __restrict__ keys,
                                                 const int* __restrict__ seg_begin, const int* __restrict__ seg_end,
                                                 const uint8_t* __restrict__ has_mask, const int* __restrict__ area,
                                                 int32_t* __restrict__ feats, uint8_t* __restrict__ seg_fail) {
  lm_pdl_wait();
  extern __shared__ int s_kept[];
  int* s_kx = s_kept;
  int* s_ky = s_kept + s.nf0;
  const int seg = blockIdx.x, lane = threadIdx.x;
  const int slots = 2 * s.L, v = seg / slots, slot = seg - v * slots, l = slot >> 1, m = slot & 1;
  const int nf = s.nf0 >> l, W = s.cols[l];
  const int begin = seg_begin[seg], n = seg_end[seg] - begin;
  if (n < nf) {
    if (lane == 0) seg_fail[seg] = 1;
    return;
  }
  if (lane == 0) seg_fail[seg] = 0;
  float dist;
  if (m == 0) {
    dist = (float)(n / nf + 1);  // LL.cpp:627
  } else {                       // LL.cpp:953-956
    const int a = has_mask[v] ? area[v * s.L + l] : s.npix[l];
    dist = __fadd_rn(__fdiv_rn(__fsqrt_rn((float)a), __fsqrt_rn((float)nf)), 1.5f);
  }
  long long need = tr_need(dist);
  int32_t* out = feats + ((size_t)v * s.F + s.first[slot]) * 3;
  int k = 0, i = 0, lane_max = -1;
  bool kept_any = false;
  while (k < nf) {
    const int cnt = min(32, n - i);
    const bool valid = lane < cnt;
    int cx = 0, cy = 0, cl = 0;
    if (valid) {
      const uint32_t lo = (uint32_t)keys[begin + i + lane];
      const int p = (int)(lo >> 3);
      cl = (int)(lo & 7);
      cy = p / W;
      cx = p - cy * W;
    }
    int md = 0x7fffffff;
    if (valid)
      for (int j = 0; j < k; ++j) {
        const int dx = cx - s_kx[j], dy = cy - s_ky[j];
        md = min(md, dx * dx + dy * dy);
      }
    unsigned ball = __ballot_sync(0xffffffffu, valid && (long long)md >= need);
    while (ball && k < nf) {
      const int j = __ffs(ball) - 1;
      const int nx = __shfl_sync(0xffffffffu, cx, j), ny = __shfl_sync(0xffffffffu, cy, j), nl = __shfl_sync(0xffffffffu, cl, j);
      if (lane == 0) {
        s_kx[k] = nx; s_ky[k] = ny;
        out[k * 3 + 0] = nx; out[k * 3 + 1] = ny; out[k * 3 + 2] = nl;
      }
      ++k;
      kept_any = true;
      const int dx = cx - nx, dy = cy - ny;
      md = min(md, dx * dx + dy * dy);
      ball &= j == 31 ? 0u : (~0u << (j + 1));
      ball &= __ballot_sync(0xffffffffu, (long long)md >= need);
    }
    __syncwarp();
    if (valid) lane_max = max(lane_max, md);
    i += cnt;
    if (i == n) {  // LL.cpp:309-314
      i = 0;
      dist = __fsub_rn(dist, 1.0f);
      need = tr_need(dist);
      if (!kept_any) {
        const int far = __reduce_max_sync(0xffffffffu, lane_max);
        while (need > far) {
          dist = __fsub_rn(dist, 1.0f);
          need = tr_need(dist);
        }
      }
      kept_any = false;
      lane_max = -1;
    }
  }
}
