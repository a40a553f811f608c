// lm_kernels.cuh -- device code of the LINEMOD match path (sm_100a).
//
// Reference functions replaced (linemodLevelup/linemodLevelup.cpp of meiqua/6DPose @ 619be57, "LL.cpp"):
//   k_linear_memories(_band) <- spread + computeResponseMaps + linearize    LL.cpp:1094-1243
//                         (bit-planes for the coarse scan, column-major H-planes for the refinement, byte linear
//                          memories where something still reads them)
//   k_coarse_packed    <- similarity(_64) + addSimilarities(_64) + threshold loop (bit-sliced)
//   k_coarse_bytes     <- the same, byte-wise (templates the bit-sliced kernel does not take)
//                                                                           LL.cpp:1284-1354, 1435-1534, 1836-1852
//   k_scan_counts      <- candidates.push_back ordering (deterministic offsets)
//   k_refine_prep      <- the candidate list in the reference's pre-sort order
//   k_refine_filter_w + k_refine_bits <- similarityLocal(_64) + best-cell search + remove_if, bit-sliced: an exact
//                         upper-bound filter, then exact scoring of its survivors      LL.cpp:1366-1428, 1855-1938
//   k_refine<split>    <- the same, byte-wise (templates / pyramids the bit-sliced path does not take)
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "linemod_b200.h"

#define LM_SKIP_BIT 0x80000000u  // feature lies outside the image at its own level (LL.cpp:1330)

struct LevelDev {
  const uint8_t* lm;  // [M][8][T*T][plane] response bytes, contiguous, zero pad after the end
  int T, rows, cols, Wd, Hd, plane;
  int off;              // T/2 + (T%2 - 1), LL.cpp:1846/1862
  uint32_t mod_stride;  // 8*T*T*plane
};

// Per (template, slot): x = first feature, y = feature count, z = template_positions P at the
// slot's level (LL.cpp:1309), w = width | height << 16.
typedef int4 TSlot;

__device__ __forceinline__ float lm_score(int raw, int nfeat) {
  // (raw_score * 100.f) / (4 * num_features), LL.cpp:1842 / 1918 -- two correctly rounded float ops
  return __fdiv_rn(__fmul_rn((float)raw, 100.f), (float)(4 * nfeat));
}

// Smallest raw score whose similarity exceeds the threshold (the float compare of LL.cpp:1842-1844
// is monotone in raw).  Returns 4*nfeat + 1 when nothing can pass.
__device__ __forceinline__ int lm_min_passing_raw(float threshold, int nfeat) {
  int lo = 0, hi = 4 * nfeat + 1;  // invariant: everything >= hi passes (hi = max+1 is "nothing")
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (lm_score(mid, nfeat) > threshold) hi = mid; else lo = mid + 1;
  }
  return lo;
}

// Smallest raw score that survives remove_if(similarity < threshold) (LL.cpp:1935-1937); 4*nfeat + 1
// when nothing can.
__device__ __forceinline__ int lm_min_kept_raw(float threshold, int nfeat) {
  int lo = 0, hi = 4 * nfeat + 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (!(lm_score(mid, nfeat) < threshold)) hi = mid; else lo = mid + 1;
  }
  return lo;
}

// response of orientation o against spread mask v: the active SIMILARITY_LUT (LL.cpp:1121) is
// 4 if bit o is set, else 1 if a neighbouring orientation bit is set, else 0 (checked against the
// table in tests/test_oracle_cpu.py).
__device__ __forceinline__ uint32_t lm_response(uint32_t v, int o) {
  const uint32_t hit = (v >> o) & 1u;
  const uint32_t nb = ((v >> ((o + 1) & 7)) | (v >> ((o + 7) & 7))) & 1u;
  return hit ? 4u : nb;
}

// Programmatic dependent launch: every kernel of the per-frame chain is launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, so its launch latency overlaps the tail of its
// predecessor; it must not touch the predecessor's results before this wait returns.
__device__ __forceinline__ void lm_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// --------------------------------------------------------------------------------------------
// K1: spread (OR over the forward TxT window) -> response maps -> linear memories
//     (+ for the lowest level: the same spread masks as bit-planes, one bit per position and label)
// --------------------------------------------------------------------------------------------
struct LinMemLevel {
  const uint8_t* q[LM_MAX_MODALITIES];  // quantized u8 rows x cols
  uint8_t* lm;
  uint32_t* bp;  // optional: [M][8][lbw] words, bit (grid*plane + pos) of block (m, o) = spread bit o
  int lbw;
  int T, rows, cols, Wd, Hd, plane;
  uint32_t mod_stride;
  int block_end;  // blocks [previous end, block_end) of the launch belong to this level (per modality)
  int nseg;       // band kernel: column segments per row of positions (Wd / nseg is a multiple of 4)
  // planes mode (band kernel): instead of the byte linear memories the level gets ONLY the column-major H-planes the
  // bit-sliced refinement reads (k_refine_filter_w / k_refine_bits), straight from the spread masks
  uint32_t* rp;   // non-null: planes mode
  int nyb;        // words per column: word yb = rows 16*yb .. 16*yb + 31
  int pseg;       // positions per column segment of a planes-mode CTA
};

struct LinMemParams {
  LinMemLevel lv[LM_MAX_LEVELS];
  int L, M;
  int block_offset;  // added to blockIdx.x: a launch may cover only the lowest level, or only the levels above it
};

// OR of the forward TxT window at (x, y), clipped at the bottom/right image edge (LL.cpp:1094-1109).
template <int T>
__device__ __forceinline__ uint32_t spread_window(const uint8_t* __restrict__ q, int cols, int rows, int x, int y, int Trt) {
  uint32_t v = 0;
  const uint8_t* __restrict__ p0 = q + (size_t)y * cols + x;
  if (T > 0 && x + T <= cols && y + T <= rows) {
    // interior: T*T independent loads, fully unrolled (the dependent OR chain comes after the loads)
    uint32_t t[T > 0 ? T * T : 1];
#pragma unroll
    for (int dy = 0; dy < T; ++dy)
#pragma unroll
      for (int dx = 0; dx < T; ++dx) t[dy * T + dx] = __ldg(p0 + dy * cols + dx);
#pragma unroll
    for (int k = 0; k < T * T; ++k) v |= t[k];
    return v;
  }
  const int y1 = min(y + Trt, rows), x1 = min(x + Trt, cols);
  for (int yy = y; yy < y1; ++yy)
    for (int xx = x; xx < x1; ++xx) v |= __ldg(q + (size_t)yy * cols + xx);
  return v;
}

__global__ void __launch_bounds__(256) k_linear_memories(LinMemParams p) {
  lm_pdl_wait();
  // which level does this block serve (<= 4 levels: linear search over the uniform block index)
  // which level does this block serve: blocks are numbered lowest level first (<= 4 levels: linear search)
  const int bx = (int)blockIdx.x + p.block_offset;
  int l = p.L - 1, first = 0;
  while (l > 0 && bx >= p.lv[l].block_end) { first = p.lv[l].block_end; --l; }
  const LinMemLevel& lv = p.lv[l];
  const int m = blockIdx.y;
  const int n = lv.T * lv.T * lv.plane;
  const uint8_t* __restrict__ q = (m == 0) ? lv.q[0] : lv.q[1];
  uint8_t* __restrict__ out = lv.lm + (size_t)m * lv.mod_stride;
  const int i = (bx - first) * 256 + (int)threadIdx.x;  // 32-aligned across a warp
  uint32_t v = 0;
  if (i < n) {
    const int g = i / lv.plane, pos = i - g * lv.plane;
    const int gy = g / lv.T, gx = g - gy * lv.T;
    const int py = pos / lv.Wd, px = pos - py * lv.Wd;
    const int y = py * lv.T + gy, x = px * lv.T + gx;
    switch (lv.T) {
      case 2: v = spread_window<2>(q, lv.cols, lv.rows, x, y, 2); break;
      case 4: v = spread_window<4>(q, lv.cols, lv.rows, x, y, 4); break;
      case 5: v = spread_window<5>(q, lv.cols, lv.rows, x, y, 5); break;
      case 8: v = spread_window<8>(q, lv.cols, lv.rows, x, y, 8); break;
      default: v = spread_window<0>(q, lv.cols, lv.rows, x, y, lv.T); break;
    }
#pragma unroll
    for (int o = 0; o < 8; ++o) out[(size_t)o * n + i] = (uint8_t)lm_response(v, o);
  }
  if (lv.bp) {  // block-uniform
#pragma unroll
    for (int o = 0; o < 8; ++o) {
      const uint32_t b = __ballot_sync(0xffffffffu, (v >> o) & 1u);
      if ((threadIdx.x & 31) == 0 && i < n) lv.bp[(size_t)(m * 8 + o) * lv.lbw + (i >> 5)] = b;
    }
  }
}

// K1 (band version): one CTA per (level, modality, row of sampled positions).  The band of T image rows
// (+ T-1 rows below for the forward window) is staged in shared memory, the TxT OR is done separably
// (horizontal then vertical, 4 pixels per 32-bit op), and the responses of 4 consecutive positions of
// one (label, grid) plane are computed SIMD-in-register and written with one 32-bit store.  Needs
// cols % 4 == 0 and Wd % 4 == 0 (every BASELINE size); other sizes use k_linear_memories above.
// Bit-planes are OR-ed in with atomics (the caller zeroes them first).
// (row, column) of flat index i in a [rows][width] grid, advanced by `step` without a division
struct RowCol {
  int r, c;
  __device__ __forceinline__ RowCol(int i, int width) : r(i / width), c(i - (i / width) * width) {}
  __device__ __forceinline__ void advance(int step, int width) {
    c += step;
    while (c >= width) { c -= width; ++r; }
  }
};

// TT = the level's sampling step at compile time (4 and 8 are the reference's defaults: window loops unroll and
// the grid arithmetic is shifts), 0 = any T at run time.
template <int TT>
__device__ __forceinline__ void linear_memories_band_level(const LinMemLevel& lv, int m, int bi, uint8_t* s_band) {
  const int T = TT > 0 ? TT : lv.T;
  const int py = bi / lv.nseg, seg = bi - py * lv.nseg;  // row of sampled positions, column segment
  const int cols = lv.cols, rows = lv.rows, Wd = lv.Wd;
  const int Wseg = Wd / lv.nseg;        // positions in this segment (multiple of 4)
  const int x0 = seg * Wseg * T;        // first image column of the segment
  const int cseg = Wseg * T;            // image columns that produce this segment's positions
  const int Wp = (cseg + T + 3 + 4) & ~3;  // padded row pitch: the forward window needs T-1 more columns
  const int nin = 2 * T - 1;
  uint8_t* s_in = s_band;               // [nin][Wp]
  uint8_t* s_h = s_in + nin * Wp;       // [nin][Wp] horizontal OR
  uint8_t* s_sp = s_h + nin * Wp;       // [T][Wp]   spread mask of the band
  const uint8_t* __restrict__ q = (m == 0) ? lv.q[0] : lv.q[1];
  const int y0 = py * T;
  const int wpr = Wp >> 2, cw = cseg >> 2;
  const int nthr = blockDim.x;
  // A: stage the input rows (zero beyond the image = clipping at the bottom/right edge)
  {
    RowCol rc(threadIdx.x, wpr);
    for (int i = threadIdx.x; i < nin * wpr; i += nthr, rc.advance(nthr, wpr)) {
      uint32_t v = 0;
      if (x0 + 4 * rc.c < cols && y0 + rc.r < rows)
        v = __ldg(reinterpret_cast<const uint32_t*>(q + (size_t)(y0 + rc.r) * cols + x0) + rc.c);
      reinterpret_cast<uint32_t*>(s_in)[i] = v;
    }
  }
  __syncthreads();
  // B: horizontal OR over dx < T, 4 pixels at a time
  {
    RowCol rc(threadIdx.x, cw);
    for (int i = threadIdx.x; i < nin * cw; i += nthr, rc.advance(nthr, cw)) {
      const uint32_t* row = reinterpret_cast<const uint32_t*>(s_in + rc.r * Wp) + rc.c;
      uint32_t acc = row[0];
      if (TT == 4) {
        const uint32_t n1 = row[1];
        acc |= __funnelshift_r(row[0], n1, 8) | __funnelshift_r(row[0], n1, 16) | __funnelshift_r(row[0], n1, 24);
      } else if (TT == 8) {
        const uint32_t n1 = row[1], n2 = row[2];
        acc |= __funnelshift_r(row[0], n1, 8) | __funnelshift_r(row[0], n1, 16) | __funnelshift_r(row[0], n1, 24) | n1 |
               __funnelshift_r(n1, n2, 8) | __funnelshift_r(n1, n2, 16) | __funnelshift_r(n1, n2, 24);
      } else {
        for (int dx = 1; dx < T; ++dx) acc |= __funnelshift_r(row[dx >> 2], row[(dx >> 2) + 1], (dx & 3) << 3);
      }
      reinterpret_cast<uint32_t*>(s_h + rc.r * Wp)[rc.c] = acc;
    }
  }
  __syncthreads();
  // C: vertical OR over dy < T
  {
    RowCol rc(threadIdx.x, cw);
    for (int i = threadIdx.x; i < T * cw; i += nthr, rc.advance(nthr, cw)) {
      uint32_t acc = 0;
#pragma unroll
      for (int dy = 0; dy < (TT > 0 ? TT : 1); ++dy) acc |= reinterpret_cast<const uint32_t*>(s_h + (rc.r + dy) * Wp)[rc.c];
      if (TT == 0)
        for (int dy = 1; dy < T; ++dy) acc |= reinterpret_cast<const uint32_t*>(s_h + (rc.r + dy) * Wp)[rc.c];
      reinterpret_cast<uint32_t*>(s_sp + rc.r * Wp)[rc.c] = acc;
    }
  }
  __syncthreads();
  // D: responses in linear-memory order, 4 positions per store
  const int T2 = T * T, q4 = Wseg >> 2;
  const int n = T2 * lv.plane;
  uint8_t* __restrict__ out = lv.lm + (size_t)m * lv.mod_stride;
  const int pos_row = py * Wd + seg * Wseg;
  RowCol gk(threadIdx.x, q4);  // r = grid g, c = group of 4 positions k
  for (int i = threadIdx.x; i < T2 * q4; i += nthr, gk.advance(nthr, q4)) {
    const int g = gk.r, k = gk.c;
    const int gy = TT > 0 ? g / TT : g / T, gx = g - gy * T;
    const uint8_t* sp = s_sp + gy * Wp + (4 * k) * T + gx;
    const uint32_t V = (uint32_t)sp[0] | ((uint32_t)sp[T] << 8) | ((uint32_t)sp[2 * T] << 16) | ((uint32_t)sp[3 * T] << 24);
    const int pos = g * lv.plane + pos_row + 4 * k;  // multiple of 4
    uint8_t* __restrict__ o0 = out + pos;
#pragma unroll
    for (int o = 0; o < 8; ++o) {
      const uint32_t hit = (V >> o) & 0x01010101u;
      const uint32_t nb = ((V >> ((o + 1) & 7)) | (V >> ((o + 7) & 7))) & 0x01010101u;
      *reinterpret_cast<uint32_t*>(o0 + (size_t)o * n) = (hit << 2) | (nb & ~hit);
      if (lv.bp) {
        const uint32_t nib = ((hit * 0x01020408u) >> 24) & 0xFu;  // the 4 hit bits, position order
        if (nib) atomicOr(lv.bp + (size_t)(m * 8 + o) * lv.lbw + (pos >> 5), nib << (pos & 31));
      }
    }
  }
}

// K1, planes mode: one CTA per (level, modality, block of 16 rows of positions, column segment).  The 16*T (+ T-1) image
// rows are staged and OR-spread exactly as in the band version; then thread (grid, column) walks its 16 positions down the
// block and packs, per label, their H bits into a 16-bit half: the low half of word yb = block and the high half of word
// yb - 1 (words overlap by 16 rows, see k_refine_prep) -- plain 16-bit stores, no atomics, nothing to clear.
template <int TT>
__device__ __forceinline__ void spread_planes_block(const LinMemLevel& lv, int m, int bi, uint8_t* s_band) {
  const int T = TT > 0 ? TT : lv.T;
  const int nsegp = lv.Wd / lv.pseg;
  const int rb = bi / nsegp, seg = bi - rb * nsegp;
  const int cols = lv.cols, rows = lv.rows;
  const int Wseg = lv.pseg;
  const int x0 = seg * Wseg * T;
  const int cseg = Wseg * T;
  const int Wp = (cseg + T + 3 + 4) & ~3;
  const int nrow = 16 * T;         // image rows that hold the block's positions
  const int nin = nrow + T - 1;    // + the forward window
  uint8_t* s_in = s_band;          // [nin][Wp]
  uint8_t* s_h = s_in + nin * Wp;  // [nin][Wp] horizontal OR
  uint8_t* s_sp = s_h + nin * Wp;  // [nrow][Wp] spread masks
  const uint8_t* __restrict__ q = (m == 0) ? lv.q[0] : lv.q[1];
  const int y0 = rb * nrow;
  const int wpr = Wp >> 2, cw = cseg >> 2;
  const int nthr = blockDim.x;
  {
    // 16*T + T-1 rows: eight loads in flight per thread (one round trip to the frame, not one per row)
    const int n = nin * wpr;
    for (int i0 = threadIdx.x; i0 < n; i0 += 8 * nthr) {
      uint32_t v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int i = i0 + k * nthr;
        const int r = i / wpr, c = i - r * wpr;
        v[k] = 0u;
        if (i < n && x0 + 4 * c < cols && y0 + r < rows)
          v[k] = __ldg(reinterpret_cast<const uint32_t*>(q + (size_t)(y0 + r) * cols + x0) + c);
      }
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (i0 + k * nthr < n) reinterpret_cast<uint32_t*>(s_in)[i0 + k * nthr] = v[k];
    }
  }
  __syncthreads();
  {
    RowCol rc(threadIdx.x, cw);
    for (int i = threadIdx.x; i < nin * cw; i += nthr, rc.advance(nthr, cw)) {
      const uint32_t* row = reinterpret_cast<const uint32_t*>(s_in + rc.r * Wp) + rc.c;
      uint32_t acc = row[0];
      if (TT == 4) {
        const uint32_t n1 = row[1];
        acc |= __funnelshift_r(row[0], n1, 8) | __funnelshift_r(row[0], n1, 16) | __funnelshift_r(row[0], n1, 24);
      } else if (TT == 8) {
        const uint32_t n1 = row[1], n2 = row[2];
        acc |= __funnelshift_r(row[0], n1, 8) | __funnelshift_r(row[0], n1, 16) | __funnelshift_r(row[0], n1, 24) | n1 |
               __funnelshift_r(n1, n2, 8) | __funnelshift_r(n1, n2, 16) | __funnelshift_r(n1, n2, 24);
      } else {
        for (int dx = 1; dx < T; ++dx) acc |= __funnelshift_r(row[dx >> 2], row[(dx >> 2) + 1], (dx & 3) << 3);
      }
      reinterpret_cast<uint32_t*>(s_h + rc.r * Wp)[rc.c] = acc;
    }
  }
  __syncthreads();
  {
    RowCol rc(threadIdx.x, cw);
    for (int i = threadIdx.x; i < nrow * cw; i += nthr, rc.advance(nthr, cw)) {
      uint32_t acc = 0;
#pragma unroll
      for (int dy = 0; dy < (TT > 0 ? TT : 1); ++dy) acc |= reinterpret_cast<const uint32_t*>(s_h + (rc.r + dy) * Wp)[rc.c];
      if (TT == 0)
        for (int dy = 1; dy < T; ++dy) acc |= reinterpret_cast<const uint32_t*>(s_h + (rc.r + dy) * Wp)[rc.c];
      reinterpret_cast<uint32_t*>(s_sp + rc.r * Wp)[rc.c] = acc;
    }
  }
  __syncthreads();
  const int T2 = T * T;
  uint16_t* __restrict__ rp16 = reinterpret_cast<uint16_t*>(lv.rp);
  RowCol gk(threadIdx.x, Wseg);  // r = grid, c = column of the segment
  for (int i = threadIdx.x; i < T2 * Wseg; i += nthr, gk.advance(nthr, Wseg)) {
    const int g = gk.r, k = gk.c;
    const int gy = TT > 0 ? g / TT : g / T, gx = g - gy * T;
    const uint8_t* sp = s_sp + gy * Wp + k * T + gx;
    uint32_t half[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) half[o] = 0u;
#pragma unroll 4
    for (int b = 0; b < 16; ++b) {
      const uint32_t v = sp[(size_t)b * T * Wp];
#pragma unroll
      for (int o = 0; o < 8; ++o) half[o] |= ((v >> o) & 1u) << b;
    }
    const int x = seg * Wseg + k;
#pragma unroll
    for (int o = 0; o < 8; ++o) {
      const size_t pb = (size_t)((m * 8 + o) * T2 + g);
      if (rb < lv.nyb) rp16[((pb * lv.nyb + rb) * lv.Wd + x) * 2] = (uint16_t)half[o];
      if (rb >= 1 && rb - 1 < lv.nyb) rp16[((pb * lv.nyb + rb - 1) * lv.Wd + x) * 2 + 1] = (uint16_t)half[o];
    }
  }
}

__global__ void __launch_bounds__(256) k_linear_memories_band(LinMemParams p) {
  lm_pdl_wait();
  extern __shared__ __align__(16) uint8_t s_band[];
  // which level does this block serve: blocks are numbered lowest level first (<= 4 levels: linear search)
  const int bx = (int)blockIdx.x + p.block_offset;
  int l = p.L - 1, first = 0;
  while (l > 0 && bx >= p.lv[l].block_end) { first = p.lv[l].block_end; --l; }
  const LinMemLevel& lv = p.lv[l];
  const int bi = bx - first;
  if (lv.rp) {  // planes mode
    switch (lv.T) {
      case 4: spread_planes_block<4>(lv, blockIdx.y, bi, s_band); break;
      case 8: spread_planes_block<8>(lv, blockIdx.y, bi, s_band); break;
      default: spread_planes_block<0>(lv, blockIdx.y, bi, s_band); break;
    }
    return;
  }
  switch (lv.T) {  // block-uniform
    case 4: linear_memories_band_level<4>(lv, blockIdx.y, bi, s_band); break;
    case 8: linear_memories_band_level<8>(lv, blockIdx.y, bi, s_band); break;
    default: linear_memories_band_level<0>(lv, blockIdx.y, bi, s_band); break;
  }
}

// --------------------------------------------------------------------------------------------
// warp / block helpers
// --------------------------------------------------------------------------------------------
__device__ __forceinline__ int block_exclusive_scan(int v, int* s_warp, int* total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  int inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += t;
  }
  __syncthreads();  // protect s_warp reuse
  if (lane == 31) s_warp[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    int t = lane < nw ? s_warp[lane] : 0;
    int ti = t;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      int u = __shfl_up_sync(0xffffffffu, ti, d);
      if (lane >= d) ti += u;
    }
    if (lane < nw) s_warp[lane] = ti - t;
    if (lane == 31) s_warp[32] = ti;
  }
  __syncthreads();
  *total = s_warp[32];
  return s_warp[wid] + inc - v;
}

// --------------------------------------------------------------------------------------------
// K2 (bit-sliced): coarse similarity scan over the lowest pyramid level.
//
// The response of a feature with orientation o at a position is 4*H + N with H = spread bit o and
// N = (spread bit o-1 | spread bit o+1) & ~H.  The spread bits are kept as bit-planes over the
// linear-memory positions (same flat order as the byte linear memories, so reads that run past a
// grid row continue into the next one exactly as the reference's do).  One warp owns one template:
// lane i holds positions 32*(i + 32 r) ... +31 of round r, and adds the H and N planes of every
// feature into two vertical (bit-sliced) counters with carry-save adders; the score 4*CH + CN, the
// threshold compare and the candidate mask are evaluated bit-sliced as well.  All bit-planes of the
// level (153.6 KB at 640x480) sit in shared memory, staged by one bulk (TMA) copy per CTA.
// --------------------------------------------------------------------------------------------
struct BitScanParams {
  const uint32_t* bp;   // [M*8][lbw]
  uint32_t bp_words;    // M*8*lbw
  int lbw, plane, nwords;
  const TSlot* tslot;
  const uint4* fdesc4;  // per feature: byte offsets (inside bp) of the window start of its label's plane (x) and of the two
                        // neighbouring labels' planes (y, z), bit shift (w); skipped features and the padding to a multiple
                        // of 8 per (template, modality) point at the zero words behind the planes
  const int2* k2info;   // [G][M]: first descriptor, padded count
  uint32_t zero_off;    // byte offset of the zero words
  const int32_t* work;  // template id per work item
  const int32_t* items; // work items taken by this kernel
  int n_items;
  int S, M, slot_low;
  float threshold;
  uint32_t* mask;  // [n_work][nwords] pass bits, position order
  uint16_t* raw;   // [n_work][plane] raw score, written at passing positions only
  int32_t* cnt;    // [n_work]
  // candidate-offset scan fused behind the scan (the last CTA to finish does what k_scan_counts does); off == null:
  // a separate k_scan_counts launch follows (banks that also need k_coarse_bytes)
  int32_t* off;
  int n_work;
  lm_result_header* hdr;
  int capacity, shard;
  unsigned long long* counters;
  int* queue;      // work / survivor counters of the refinement filter, reset with the header
  int* ticket;     // zero between launches
  int split;       // warps per team (1, 2, 4 or 8): a task's features are dealt over the team (see k_coarse_packed)
};

#define CSA(sum, carry, a, b, c)                 \
  {                                              \
    const uint32_t a_ = (a), b_ = (b), c_ = (c); \
    carry = (a_ & b_) | (c_ & (a_ ^ b_));        \
    sum = a_ ^ b_ ^ c_;                          \
  }

// add eight 1-bit planes x[0..7] into the 8-bit vertical counter c[0..7]
__device__ __forceinline__ void vc_add8(uint32_t (&c)[8], const uint32_t (&x)[8]) {
  uint32_t t1a, t1b, t1c, t1d, t2a, t2b, t3;
  CSA(c[0], t1a, c[0], x[0], x[1]);
  CSA(c[0], t1b, c[0], x[2], x[3]);
  CSA(c[1], t2a, c[1], t1a, t1b);
  CSA(c[0], t1c, c[0], x[4], x[5]);
  CSA(c[0], t1d, c[0], x[6], x[7]);
  CSA(c[1], t2b, c[1], t1c, t1d);
  CSA(c[2], t3, c[2], t2a, t2b);
#pragma unroll
  for (int b = 3; b < 8; ++b) {  // ripple the weight-8 carry
    const uint32_t k = c[b] & t3;
    c[b] ^= t3;
    t3 = k;
  }
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

#define LM_PACK_THREADS 768

// exclusive scan of the per-template candidate counts -> off[], result header and counters reset for k_refine,
// counts re-zeroed for the next frame's atomics.  Whole CTA.
__device__ __forceinline__ void scan_counts_block(int32_t* __restrict__ cnt, int32_t* __restrict__ off, int n,
                                                  lm_result_header* __restrict__ hdr, int capacity, int shard,
                                                  unsigned long long* __restrict__ counters, int* __restrict__ queue, int* s_warp) {
  const int per = (n + blockDim.x - 1) / blockDim.x;
  const int b = min((int)threadIdx.x * per, n), e = min(b + per, n);
  int sum = 0;
  for (int i = b; i < e; ++i) sum += __ldcg(cnt + i);
  int total;
  int run = block_exclusive_scan(sum, s_warp, &total);
  for (int i = b; i < e; ++i) {
    off[i] = run;
    run += __ldcg(cnt + i);
    cnt[i] = 0;  // k_coarse_packed accumulates the next frame's counts with atomics
  }
  if (threadIdx.x == 0) {
    off[n] = total;
    hdr->count = 0;  // k_refine appends kept records behind the header
    hdr->coarse_candidates = total;
    hdr->capacity = capacity;
    hdr->shard = shard;
    counters[0] = 0ull;  // k_refine accumulates into them
    counters[1] = 0ull;
    counters[4] = 0ull;  // k_refine_filter_w: features x candidates it dropped, plane words it read
    counters[5] = 0ull;
    queue[0] = 0;        // k_refine_filter_w: next candidate, survivors appended (two lists)
    queue[1] = 0;
    queue[2] = 0;
  }
}

__global__ void __launch_bounds__(1024) k_scan_counts(int32_t* __restrict__ cnt, int32_t* __restrict__ off, int n,
                                                     lm_result_header* __restrict__ hdr, int capacity, int shard,
                                                     unsigned long long* __restrict__ counters, int* __restrict__ queue) {
  lm_pdl_wait();
  __shared__ int s_warp[33];
  scan_counts_block(cnt, off, n, hdr, capacity, shard, counters, queue, s_warp);
}

// K2 work decomposition.  A template only has ceil(P / 32) position words that can hold a score (P = its
// template_positions, LL.cpp:1309; 33 of the 38 words of the level for the bench bank).  Giving a warp a
// whole template in rounds of 32 words leaves 31 of 32 lanes idle in the last round, so the words of a
// template are split in two kinds of tasks:
//   * FULL rounds (32 consecutive words of one template): the feature descriptors are warp-uniform, so the
//     plane addressing lives in the uniform datapath -- 15 instructions per feature;
//   * the REMAINDERS (P/32 mod 32 words per template) of all templates of the CTA, laid end to end and cut
//     into tasks of 32 entries: lane k owns one (template, word) and walks its own template's descriptors
//     (lanes of 2-3 templates share a warp; 26 instructions per feature, but 32 busy lanes).
// Both kinds sit in one dynamic queue per CTA (full rounds first).  Either way a lane owns ONE word: two 8-bit
// vertical counters (H and N planes), the bit-sliced score 4*CH + CN, threshold compare and pass mask.
#define LM_PACK_CHUNK 512  // templates whose task offsets are tabulated in shared memory at a time

// score = 4*CH + CN (bit-sliced ripple add), positions >= P are zero (LL.cpp:1314), compare with the
// smallest passing raw score, emit the pass mask and the raw scores of the passing positions
__device__ __forceinline__ void coarse_emit(const BitScanParams& p, int w, int idx, int P, int nfeat, int words,
                                            const uint32_t (&ch)[8], const uint32_t (&cn)[8]) {
  const int raw_min = lm_min_passing_raw(p.threshold, nfeat);
  const int j0 = idx * 32;
  uint32_t live = 0xffffffffu;   // positions < P carry a score
  uint32_t valid = 0xffffffffu;  // positions < plane exist
  if (P - j0 < 32) live = (P - j0 <= 0) ? 0u : (0xffffffffu >> (32 - (P - j0)));
  if (p.plane - j0 < 32) valid = 0xffffffffu >> (32 - (p.plane - j0));
  uint32_t sc[11];
  sc[0] = cn[0] & live;
  sc[1] = cn[1] & live;
  uint32_t carry = 0u;
#pragma unroll
  for (int b = 2; b < 10; ++b) {
    const uint32_t a = (b < 8) ? cn[b] : 0u;
    const uint32_t h = ch[b - 2];
    sc[b] = (a ^ h ^ carry) & live;
    carry = (a & h) | (carry & (a ^ h));
  }
  sc[10] = carry & live;
  uint32_t pass;
  if (raw_min > 2047) {
    pass = 0u;
  } else {
    uint32_t gt = 0u, eq = 0xffffffffu;
#pragma unroll
    for (int b = 10; b >= 0; --b) {
      if ((raw_min >> b) & 1) {
        eq &= sc[b];
      } else {
        gt |= eq & sc[b];
        eq &= ~sc[b];
      }
    }
    pass = (gt | eq) & valid;
  }
  p.mask[(size_t)w * p.nwords + idx] = pass;
  int my_count = __popc(pass);
  while (pass) {
    const int b = __ffs(pass) - 1;
    pass &= pass - 1;
    uint32_t v = 0;
#pragma unroll
    for (int k = 0; k < 11; ++k) v |= ((sc[k] >> b) & 1u) << k;
    p.raw[(size_t)w * p.plane + j0 + b] = (uint16_t)v;
  }
  if (idx == words - 1) {
    // words beyond the useful ones: every position is >= P, i.e. raw 0 (passes only if 0 does)
    for (int x = words; x < p.nwords; ++x) {
      const int q0 = x * 32;
      uint32_t ps = 0u;
      if (raw_min == 0) {
        ps = (p.plane - q0 < 32) ? (0xffffffffu >> (32 - (p.plane - q0))) : 0xffffffffu;
        for (int b = 0; b < 32; ++b)
          if ((ps >> b) & 1u) p.raw[(size_t)w * p.plane + q0 + b] = 0;
      }
      p.mask[(size_t)w * p.nwords + x] = ps;
      my_count += __popc(ps);
    }
  }
  if (my_count) atomicAdd(p.cnt + w, my_count);  // zero before the frame (k_scan_counts re-zeroes)
}

// bit-sliced add of two 8-bit vertical counters
__device__ __forceinline__ void vc8_add(uint32_t (&c)[8], const uint32_t (&o)[8]) {
  uint32_t carry = 0u;
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    const uint32_t a = c[b], x = o[b];
    c[b] = a ^ x ^ carry;
    carry = (a & x) | (carry & (a ^ x));
  }
}

// barrier over the `nthreads` threads of one team of warps (named barrier `id`, 1..15)
__device__ __forceinline__ void team_bar(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Feature split (p.split = S > 1, small shards): S warps form a team that owns a task together; warp q of the team adds
// the 8-feature steps q, q + S, ... of every modality, the partial counters meet in shared memory and warp 0 of the team
// emits.  A task is then a chain S times shorter -- the latency of the kernel follows the shard instead of staying one
// whole task (what keeps a 1/8 shard from being 8 times faster, and what holds an SM's shared memory for the duration).
template <bool kSmem>
__global__ void __launch_bounds__(LM_PACK_THREADS, 1) k_coarse_packed(BitScanParams p) {
  lm_pdl_wait();
  extern __shared__ __align__(128) uint32_t s_bp[];
  __shared__ __align__(8) unsigned long long s_bar;
  __shared__ int s_full[LM_PACK_CHUNK + 1];  // full rounds before template i
  __shared__ int s_rem[LM_PACK_CHUNK + 1];   // remainder words before template i
  __shared__ int s_warp[33];
  __shared__ int s_next;
  __shared__ int s_team_task[LM_PACK_THREADS / 64];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int t0 = (int)(((long long)p.n_items * blockIdx.x) / gridDim.x);
  const int t1 = (int)(((long long)p.n_items * (blockIdx.x + 1)) / gridDim.x);

  const uint32_t* __restrict__ bp = p.bp;
  if (kSmem) {
    // one elected thread stages every bit-plane with bulk async copies (TMA, 1-D) onto an mbarrier
    const uint32_t bar = smem_u32(&s_bar);
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      const uint32_t bytes = p.bp_words * 4u;  // multiple of 16 (lbw is a multiple of 4)
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
      const char* src = reinterpret_cast<const char*>(p.bp);
      uint32_t dst = smem_u32(s_bp);
      for (uint32_t done = 0; done < bytes;) {
        const uint32_t n = min(bytes - done, 32768u);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst + done),
                     "l"(src + done), "r"(n), "r"(bar)
                     : "memory");
        done += n;
      }
    }
    bp = s_bp;
  }

  bool staged = !kSmem;
  for (int c0 = t0; c0 < t1; c0 += LM_PACK_CHUNK) {
    const int nt = min(LM_PACK_CHUNK, t1 - c0);
    // task offsets of the chunk's templates (while the bit-planes are still in flight the first time)
    {
      const int per = (nt + blockDim.x - 1) / blockDim.x;
      const int b = min((int)threadIdx.x * per, nt), e = min(b + per, nt);
      int sum_f = 0, sum_r = 0;
      for (int i = b; i < e; ++i) {
        const int g = p.work[p.items[c0 + i]];
        const int words = min(max((p.tslot[(size_t)g * p.S + p.slot_low].z + 31) >> 5, 1), p.nwords);
        sum_f += words >> 5;
        sum_r += words & 31;
      }
      int tot_f, tot_r;
      int run_f = block_exclusive_scan(sum_f, s_warp, &tot_f);
      int run_r = block_exclusive_scan(sum_r, s_warp, &tot_r);
      for (int i = b; i < e; ++i) {
        const int g = p.work[p.items[c0 + i]];
        const int words = min(max((p.tslot[(size_t)g * p.S + p.slot_low].z + 31) >> 5, 1), p.nwords);
        s_full[i] = run_f;
        s_rem[i] = run_r;
        run_f += words >> 5;
        run_r += words & 31;
      }
      if (threadIdx.x == 0) {
        s_full[nt] = tot_f;
        s_rem[nt] = tot_r;
        s_next = nwarps / p.split;  // one task per team to start with
      }
    }
    __syncthreads();
    if (!staged) {  // everyone waits for phase 0 of the barrier
      asm volatile(
          "{\n"
          ".reg .pred p;\n"
          "WAIT_%=:\n"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n"
          "@p bra DONE_%=;\n"
          "bra WAIT_%=;\n"
          "DONE_%=:\n"
          "}\n" ::"r"(smem_u32(&s_bar))
          : "memory");
      staged = true;
    }
    const int n_full = s_full[nt], rem_words = s_rem[nt];
    const int n_tasks = n_full + ((rem_words + 31) >> 5);
    const int S = p.split, q = warp & (S - 1), team = warp / S;
    uint32_t* s_part = s_bp + (kSmem ? ((p.bp_words + 3u) & ~3u) : 0u) + (size_t)team * (S - 1) * 16 * 32;
    int task = team;
    while (task < n_tasks) {
      if (task < n_full) {
        // ---- a full round: 32 consecutive words of ONE template, warp-uniform descriptors ----
        int lo = 0, hi = nt;  // last i with s_full[i] <= task
        while (hi - lo > 1) {
          const int mid = (lo + hi) >> 1;
          if (s_full[mid] <= task) lo = mid; else hi = mid;
        }
        const int r = task - s_full[lo];
        const int w = p.items[c0 + lo];
        const int g = p.work[w];
        const int P = p.tslot[(size_t)g * p.S + p.slot_low].z;  // equal for all modalities (host checked)
        const int words = min(max((P + 31) >> 5, 1), p.nwords);
        const int idx = 32 * r + lane;
        int nfeat = 0;
        uint32_t ch[8], cn[8];
#pragma unroll
        for (int b = 0; b < 8; ++b) ch[b] = cn[b] = 0u;
        const char* __restrict__ lane_base = reinterpret_cast<const char*>(bp + idx);  // this lane's word of every window
        for (int m = 0; m < p.M; ++m) {
          nfeat += p.tslot[(size_t)g * p.S + p.slot_low + m].y;
          const int2 k2 = p.k2info[(size_t)g * p.M + m];
          const uint4* __restrict__ fd = p.fdesc4 + k2.x;
          for (int f0 = q * 8; f0 < k2.y; f0 += 8 * S) {  // padded to a multiple of 8: no bounds check, no skip branch
            uint32_t xh[8], xn[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const uint4 d = __ldg(fd + f0 + u);  // warp-uniform
              const uint32_t* __restrict__ ph = reinterpret_cast<const uint32_t*>(lane_base + d.x);
              const uint32_t* __restrict__ pm = reinterpret_cast<const uint32_t*>(lane_base + d.y);
              const uint32_t* __restrict__ pp = reinterpret_cast<const uint32_t*>(lane_base + d.z);
              const uint32_t h = __funnelshift_r(ph[0], ph[1], d.w);
              const uint32_t a = __funnelshift_r(pm[0], pm[1], d.w);
              const uint32_t b = __funnelshift_r(pp[0], pp[1], d.w);
              xh[u] = h;
              xn[u] = (a | b) & ~h;
            }
            vc_add8(ch, xh);
            vc_add8(cn, xn);
          }
        }
        if (S > 1) {  // the team's partial counters meet
          if (q > 0) {
#pragma unroll
            for (int b = 0; b < 8; ++b) {
              s_part[((q - 1) * 16 + b) * 32 + lane] = ch[b];
              s_part[((q - 1) * 16 + 8 + b) * 32 + lane] = cn[b];
            }
          }
          team_bar(team + 1, S * 32);
          if (q == 0) {
            for (int k = 0; k < S - 1; ++k) {
              uint32_t oh[8], on[8];
#pragma unroll
              for (int b = 0; b < 8; ++b) {
                oh[b] = s_part[(k * 16 + b) * 32 + lane];
                on[b] = s_part[(k * 16 + 8 + b) * 32 + lane];
              }
              vc8_add(ch, oh);
              vc8_add(cn, on);
            }
          }
          team_bar(team + 1, S * 32);  // the partials are in registers: the others may overwrite them
        }
        if (q == 0) coarse_emit(p, w, idx, P, nfeat, words, ch, cn);
      } else {
        // ---- remainders: lane k owns entry e of the chunk's remainder words ----
        const int e = (task - n_full) * 32 + lane;
        const bool active = e < rem_words;
        const int ee = active ? e : rem_words - 1;
        int lo = 0, hi = nt;  // last i with s_rem[i] <= ee
        while (hi - lo > 1) {
          const int mid = (lo + hi) >> 1;
          if (s_rem[mid] <= ee) lo = mid; else hi = mid;
        }
        const int w = p.items[c0 + lo];
        const int g = p.work[w];
        const int P = p.tslot[(size_t)g * p.S + p.slot_low].z;
        const int words = min(max((P + 31) >> 5, 1), p.nwords);
        const int idx = (words & ~31) + (ee - s_rem[lo]);  // behind the template's full rounds
        int nfeat = 0;
        uint32_t ch[8], cn[8];
#pragma unroll
        for (int b = 0; b < 8; ++b) ch[b] = cn[b] = 0u;
        const char* __restrict__ lane_base = reinterpret_cast<const char*>(bp + idx);
        const uint4 zdesc = make_uint4(p.zero_off, p.zero_off, p.zero_off, 0u);
        for (int m = 0; m < p.M; ++m) {
          nfeat += p.tslot[(size_t)g * p.S + p.slot_low + m].y;
          const int2 k2 = p.k2info[(size_t)g * p.M + m];
          const uint4* __restrict__ fd = p.fdesc4 + k2.x;
          const int maxn = __reduce_max_sync(0xffffffffu, k2.y);
          for (int f0 = q * 8; f0 < maxn; f0 += 8 * S) {
            uint32_t xh[8], xn[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const uint4 d = (f0 < k2.y) ? __ldg(fd + f0 + u) : zdesc;  // lanes of a shorter template read zeros
              const uint32_t* __restrict__ ph = reinterpret_cast<const uint32_t*>(lane_base + d.x);
              const uint32_t* __restrict__ pm = reinterpret_cast<const uint32_t*>(lane_base + d.y);
              const uint32_t* __restrict__ pp = reinterpret_cast<const uint32_t*>(lane_base + d.z);
              const uint32_t h = __funnelshift_r(ph[0], ph[1], d.w);
              const uint32_t a = __funnelshift_r(pm[0], pm[1], d.w);
              const uint32_t b = __funnelshift_r(pp[0], pp[1], d.w);
              xh[u] = h;
              xn[u] = (a | b) & ~h;
            }
            vc_add8(ch, xh);
            vc_add8(cn, xn);
          }
        }
        if (S > 1) {  // the team's partial counters meet
          if (q > 0) {
#pragma unroll
            for (int b = 0; b < 8; ++b) {
              s_part[((q - 1) * 16 + b) * 32 + lane] = ch[b];
              s_part[((q - 1) * 16 + 8 + b) * 32 + lane] = cn[b];
            }
          }
          team_bar(team + 1, S * 32);
          if (q == 0) {
            for (int k = 0; k < S - 1; ++k) {
              uint32_t oh[8], on[8];
#pragma unroll
              for (int b = 0; b < 8; ++b) {
                oh[b] = s_part[(k * 16 + b) * 32 + lane];
                on[b] = s_part[(k * 16 + 8 + b) * 32 + lane];
              }
              vc8_add(ch, oh);
              vc8_add(cn, on);
            }
          }
          team_bar(team + 1, S * 32);  // the partials are in registers: the others may overwrite them
        }
        if (active && q == 0) coarse_emit(p, w, idx, P, nfeat, words, ch, cn);
      }
      if (S == 1) {
        int nxt = 0;
        if (lane == 0) nxt = atomicAdd(&s_next, 1);
        task = __shfl_sync(0xffffffffu, nxt, 0);
      } else {
        if (q == 0 && lane == 0) s_team_task[team] = atomicAdd(&s_next, 1);
        team_bar(team + 1, S * 32);
        task = s_team_task[team];
      }
    }
    __syncthreads();  // the offset tables and s_next are rebuilt for the next chunk
  }
  if (p.off) {
    // the last CTA to get here owns the scan: every other CTA's masks / counts are fenced before its ticket
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(p.ticket, 1) == (int)gridDim.x - 1);
    __syncthreads();
    if (s_last) {
      __threadfence();
      scan_counts_block(p.cnt, p.off, p.n_work, p.hdr, p.capacity, p.shard, p.counters, p.queue, s_warp);
      if (threadIdx.x == 0) *p.ticket = 0;
    }
  }
  if (kSmem && !staged) {  // a CTA without templates still has to see its copy land before it exits
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(&s_bar))
        : "memory");
  }
}


// --------------------------------------------------------------------------------------------
// K2 (byte-wise): same result for templates the bit-sliced kernel does not take (more than 255
// features in total, modalities with different template_positions, very large frames).  One CTA per
// template, packed-byte accumulation of the response bytes straight from the linear memories.
// --------------------------------------------------------------------------------------------
struct ByteScanParams {
  LevelDev lv;
  const TSlot* tslot;
  const uint32_t* fbase;
  const uint32_t* fxy;
  const int32_t* work;
  const int32_t* items;
  int S, M, slot_low, nwords;
  float threshold;
  uint32_t* mask;
  uint16_t* raw;
  int32_t* cnt;
};

#define SCAN_FEAT_TILE 512

__global__ void __launch_bounds__(1024) k_coarse_bytes(ByteScanParams p) {
  lm_pdl_wait();
  __shared__ uint32_t s_base[SCAN_FEAT_TILE];
  __shared__ int s_count;
  const int w = p.items[blockIdx.x];
  const int g = p.work[w];
  const int plane = p.lv.plane;
  const int lane = threadIdx.x & 31;
  const uint32_t* __restrict__ lm32 = reinterpret_cast<const uint32_t*>(p.lv.lm);
  if (threadIdx.x == 0) s_count = 0;

  int nfeat = 0;
  for (int m = 0; m < p.M; ++m) nfeat += p.tslot[(size_t)g * p.S + p.slot_low + m].y;

  int counted = 0;
  // every thread owns 4 consecutive positions; a warp therefore owns 4 mask words per pass
  const int span = blockDim.x * 4;
  const int plane_up = (plane + 127) & ~127;
  for (int j0 = 0; j0 < plane_up; j0 += span) {
    const int j = j0 + threadIdx.x * 4;
    uint32_t s01 = 0, s23 = 0;  // u16 pairs: positions (j, j+1) and (j+2, j+3)
    for (int m = 0; m < p.M; ++m) {
      const TSlot ts = p.tslot[(size_t)g * p.S + p.slot_low + m];
      const int P = ts.z;
      uint32_t pm = 0;  // positions >= P stay zero ("dst zero elsewhere", LL.cpp:1314)
#pragma unroll
      for (int k = 0; k < 4; ++k) pm |= (j + k < P) ? (0xFFu << (8 * k)) : 0u;
      for (int f0 = 0; f0 < ts.y; f0 += SCAN_FEAT_TILE) {
        const int nt = min(SCAN_FEAT_TILE, ts.y - f0);
        __syncthreads();
        for (int i = threadIdx.x; i < nt; i += blockDim.x) {
          const uint32_t xy = p.fxy[ts.x + f0 + i];
          s_base[i] = (xy & LM_SKIP_BIT) ? 0xFFFFFFFFu : p.fbase[ts.x + f0 + i];
        }
        __syncthreads();
        if (pm) {
          uint32_t a8 = 0;
          int pend = 0;
          for (int i = 0; i < nt; ++i) {
            const uint32_t b = s_base[i];
            if (b == 0xFFFFFFFFu) continue;
            const uint32_t a = b + (uint32_t)j;
            const uint32_t lo = __ldg(lm32 + (a >> 2));
            const uint32_t hi = __ldg(lm32 + (a >> 2) + 1);
            a8 += __funnelshift_r(lo, hi, (a & 3u) << 3) & pm;
            if (++pend == 63) {  // 63 * 4 = 252 < 256: no carry between packed bytes
              s01 += __byte_perm(a8, 0, 0x4140);
              s23 += __byte_perm(a8, 0, 0x4342);
              a8 = 0;
              pend = 0;
            }
          }
          s01 += __byte_perm(a8, 0, 0x4140);
          s23 += __byte_perm(a8, 0, 0x4342);
        }
      }
    }
    // threshold (LL.cpp:1836-1852)
    const int raw[4] = {(int)(s01 & 0xFFFF), (int)(s01 >> 16), (int)(s23 & 0xFFFF), (int)(s23 >> 16)};
    uint32_t pass = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (j + k < plane && lm_score(raw[k], nfeat) > p.threshold) {
        pass |= 1u << k;
        p.raw[(size_t)w * plane + j + k] = (uint16_t)raw[k];
      }
    // 8 lanes -> one 32-bit mask word
    uint32_t word = pass << (4 * (lane & 7));
    word |= __shfl_xor_sync(0xffffffffu, word, 1);
    word |= __shfl_xor_sync(0xffffffffu, word, 2);
    word |= __shfl_xor_sync(0xffffffffu, word, 4);
    if ((lane & 7) == 0 && (j >> 5) < p.nwords) p.mask[(size_t)w * p.nwords + (j >> 5)] = word;
    counted += __popc(pass);
  }
  counted = __reduce_add_sync(0xffffffffu, counted);
  __syncthreads();
  if (lane == 0 && counted) atomicAdd(&s_count, counted);
  __syncthreads();
  if (threadIdx.x == 0) p.cnt[w] = s_count;
}

// --------------------------------------------------------------------------------------------
// k_refine_prep: (a) the ordered candidate list, (b) the refinement bit-planes of the first refined level
//
// (a) The coarse scan leaves a pass mask, raw scores and (after the scan) an offset per template.  The refinement used to
//     decode "candidate c" from them with a binary search + a select-bit walk per candidate; here one warp per template
//     writes cand[off[w] + k] = (w, j) for the k-th set bit j once, in the reference's pre-sort order
//     (template order, then ascending cell; LL.cpp:1797-1852), so c stays the record's `seq`.
// (b) H-planes for the refinement filter: bit = (response == 4) = spread bit of the label (the SIMILARITY_LUT rule, see
//     lm_response).  COLUMN-major and overlapping: word (x, yb) of block (modality, label, grid) holds rows
//     16*yb .. 16*yb + 31 of column x, so the 16 rows of ANY 16x16 patch column are bits s .. s+15 of ONE word, and the 16
//     columns of a patch are 16 consecutive words (64 contiguous bytes) -- against 16 rows x 16 bytes in 16 different
//     128-byte lines of the byte linear memories.
// --------------------------------------------------------------------------------------------
struct PrepParams {
  const int32_t* off;    // [n_work + 1]
  const uint32_t* mask;  // [n_work][nwords]
  int n_work, nwords;
  uint2* cand;
  int cand_cap;
  int expand_blocks;     // blocks [0, expand_blocks) expand, the others build planes
  const uint8_t* lm;     // byte linear memories of the filtered level, [M*8*T*T][plane]
  uint32_t* rp;          // [M*8*T*T][nyb][Wd], null: no planes
  int Wd, Hd, plane, nyb, n_pb;
};

__global__ void __launch_bounds__(256) k_refine_prep(PrepParams p) {
  lm_pdl_wait();
  const int lane = threadIdx.x & 31;
  if ((int)blockIdx.x < p.expand_blocks) {
    const int nw = (p.expand_blocks * 256) >> 5;
    for (int w = (blockIdx.x * 256 + threadIdx.x) >> 5; w < p.n_work; w += nw) {
      const int base = p.off[w];
      if (p.off[w + 1] == base) continue;
      const uint32_t* __restrict__ mk = p.mask + (size_t)w * p.nwords;
      int run = 0;
      for (int b0 = 0; b0 < p.nwords; b0 += 32) {
        uint32_t word = (b0 + lane < p.nwords) ? mk[b0 + lane] : 0u;
        const int pc = __popc(word);
        int inc = pc;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const int t = __shfl_up_sync(0xffffffffu, inc, d);
          if (lane >= d) inc += t;
        }
        int idx = base + run + inc - pc;
        while (word) {
          const int j = (b0 + lane) * 32 + __ffs(word) - 1;
          word &= word - 1;
          if (idx < p.cand_cap) p.cand[idx] = make_uint2((uint32_t)w, (uint32_t)j);  // stores only: nothing to wait for
          ++idx;
        }
        run += __shfl_sync(0xffffffffu, inc, 31);
      }
    }
    return;
  }
  if (!p.rp) return;
  // planes: one thread = 4 neighbouring columns of one word row (32-bit loads of 4 response bytes, one 128-bit store)
  const int wq = p.Wd >> 2;
  const int n = p.n_pb * p.nyb * wq;
  const int t = ((int)blockIdx.x - p.expand_blocks) * 256 + (int)threadIdx.x;
  if (t >= n) return;
  const int x4 = t % wq, yb = (t / wq) % p.nyb, pb = t / (wq * p.nyb);
  const uint32_t* __restrict__ src = reinterpret_cast<const uint32_t*>(p.lm + (size_t)pb * p.plane) + x4;
  uint32_t o0 = 0, o1 = 0, o2 = 0, o3 = 0;
  const int r0 = 16 * yb;
#pragma unroll
  for (int k = 0; k < 4; ++k) {  // 8 rows at a time: byte c of t collects the 8 row bits of column c
    uint32_t v[8];
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int r = r0 + 8 * k + b;
      v[b] = (r < p.Hd) ? __ldg(src + (size_t)r * wq) : 0u;
    }
    uint32_t t = 0u;
#pragma unroll
    for (int b = 0; b < 8; ++b) t += ((v[b] >> 2) & 0x01010101u) << b;  // response 4 <=> bit 2; the bits never meet
    o0 |= (t & 0xFFu) << (8 * k);
    o1 |= ((t >> 8) & 0xFFu) << (8 * k);
    o2 |= ((t >> 16) & 0xFFu) << (8 * k);
    o3 |= (t >> 24) << (8 * k);
  }
  *reinterpret_cast<uint4*>(p.rp + ((size_t)pb * p.nyb + yb) * p.Wd + 4 * x4) = make_uint4(o0, o1, o2, o3);
}

// --------------------------------------------------------------------------------------------
// k_refine_filter_w: exact upper-bound test in front of the refinement, bit-sliced.
//
// similarityLocal adds, per feature, 4 where the feature's label bit is set in the spread mask (H), else at most 1
// (LL.cpp:1121 table; lm_response).  So for every cell of the 16x16 patch  raw <= 4*CH + (nf - CH) = 3*CH + nf  with CH =
// number of features whose H bit is set at that cell.  A candidate survives remove_if (LL.cpp:1935-1937) only if its best
// cell reaches raw_keep, i.e. only if SOME cell has CH >= need = ceil((raw_keep - nf) / 3).  Candidates without such a cell
// are dropped here without ever touching the byte linear memories; the others (a few percent) go on to the exact
// refinement (k_refine_bits / k_refine) -- the filter never changes a result, it only removes work.
// --------------------------------------------------------------------------------------------
struct FilterParams {
  const uint32_t* rp;      // H-planes of the filtered level
  int Wd;
  const uint32_t* rdesc;   // per feature (own order, grouped per template): plane word offset incl. x / T : 23 | y / T : 9
  const int4* finfo;       // per WORK ITEM of the shard (layout below); flags bit 1 = the filter may take the template
  LevelDev low, ref;       // lowest level (cell -> pixel), filtered level (clamp, patch origin)
  const uint2* cand;
  const int32_t* off;
  int n_work, cand_cap;
  uint32_t* surv;          // survivors (candidate indices), unordered
  uint32_t* surv2;         // optional second list: candidates of templates the filter does not take
  int* queue;              // [0] next candidate, [1] survivors, [2] entries of surv2
  unsigned long long* counters;  // [4] features x candidates dropped here, [5] plane words read
};

// add eight 1-bit planes into an NB-bit vertical counter
template <int NB>
__device__ __forceinline__ void vc_add8n(uint32_t (&c)[NB], const uint32_t (&x)[8]) {
  uint32_t t1a, t1b, t1c, t1d, t2a, t2b, t3;
  CSA(c[0], t1a, c[0], x[0], x[1]);
  CSA(c[0], t1b, c[0], x[2], x[3]);
  CSA(c[1], t2a, c[1], t1a, t1b);
  CSA(c[0], t1c, c[0], x[4], x[5]);
  CSA(c[0], t1d, c[0], x[6], x[7]);
  CSA(c[1], t2b, c[1], t1c, t1d);
  CSA(c[2], t3, c[2], t2a, t2b);
#pragma unroll
  for (int b = 3; b < NB; ++b) {
    const uint32_t k = c[b] & t3;
    c[b] ^= t3;
    t3 = k;
  }
}

#define LM_FILTER_BITS 9   // CH <= 511 features of the filtered level

// One warp per candidate.  Lane k of an 8-lane group holds patch columns k and k + 8 as the two halves of a 32-bit word (16
// rows each) and counts CH for its 32 cells in a 9-bit vertical counter (carry-save adders, 8 features per step).  The
// four 8-lane groups of the warp work on the SAME 16x16 patch and deal the features between them: of every 32 consecutive
// features group q adds features 8q .. 8q+7 into its own partial counter, so a candidate is a chain of nf / 32 steps
// (what matters when the candidates are fewer than the machine has lanes, e.g. a 1/8 template shard).  Lane L decodes
// descriptor L of the step once (word offset and shift packed in one register) and the lanes of group q pick theirs up by
// shuffle; control flow is warp-uniform.  The partial counters meet (bit-sliced adds across the groups, two butterfly
// steps) at two check points -- after about half and three quarters of the features -- where cells, lanes and whole
// candidates that can no longer reach `need` are dropped, and at the end.
__device__ __forceinline__ void vc_allreduce_groups(uint32_t (&c)[LM_FILTER_BITS]) {
#pragma unroll
  for (int step = 8; step <= 16; step <<= 1) {
    uint32_t carry = 0u;
#pragma unroll
    for (int b = 0; b < LM_FILTER_BITS; ++b) {
      const uint32_t o = __shfl_xor_sync(0xffffffffu, c[b], step);
      const uint32_t a = c[b];
      c[b] = a ^ o ^ carry;
      carry = (a & o) | (carry & (a ^ o));
    }
  }
}

__device__ __forceinline__ uint32_t vc_ge(const uint32_t (&c)[LM_FILTER_BITS], int thr) {
  if (thr <= 0) return 0xffffffffu;
  uint32_t gt = 0u, eq = 0xffffffffu;
#pragma unroll
  for (int b = LM_FILTER_BITS - 1; b >= 0; --b) {
    const uint32_t tb = 0u - (((uint32_t)thr >> b) & 1u);
    gt |= eq & c[b] & ~tb;
    eq &= ~(c[b] ^ tb);
  }
  return gt | eq;
}

// base + 32-bit byte offset as ONE wide multiply-add (FMA pipe) instead of a shift-mask-add-carry chain on the ALU pipe
__device__ __forceinline__ const uint32_t* lm_ptr_add(const char* base, uint32_t byte_off) {
  unsigned long long r;
  asm("mad.wide.u32 %0, %1, 1, %2;" : "=l"(r) : "r"(byte_off), "l"(reinterpret_cast<unsigned long long>(base)));
  return reinterpret_cast<const uint32_t*>(r);
}

#define LM_FILTER_MIN_CTAS 5
// Layout contract with the host (prepare_bank / prepare_work): every template's descriptors are padded to a multiple of
// 32 with descriptors that point into an all-zero tail of the plane buffer (so the loop needs no bounds predicate), and
// finfo[w] = {first descriptor, features of the level, width | height << 16, flags | need << 8} with `need` computed on
// the host for the call's threshold with the same two IEEE float operations (lm_min_kept_raw).
__global__ void __launch_bounds__(256, LM_FILTER_MIN_CTAS) k_refine_filter_w(FilterParams p) {
  lm_pdl_wait();
  const int lane = threadIdx.x & 31, grp = lane >> 3, gl = lane & 7;
  const int total = min(p.off[p.n_work], p.cand_cap);
  const int T = p.ref.T, border = 8 * T;
  const int Wd = p.Wd;
  unsigned words_read = 0, dropped_feats = 0;
  // A warp takes one candidate at a time from the queue (taking 2..16 consecutive ones, for L1 reuse between neighbouring
  // cells, was measured slower: the tail imbalance costs more).  The NEXT candidate's cell and per-work-item record are
  // fetched while the current one is being counted.
  int c_next = 0;
  if (lane == 0) c_next = atomicAdd(p.queue, 1);
  c_next = __shfl_sync(0xffffffffu, c_next, 0);
  uint2 e_next = make_uint2(0u, 0u);
  int4 fi_next = make_int4(0, 0, 0, 0);
  if (c_next < total) {
    e_next = __ldcg(p.cand + c_next);
    fi_next = __ldg(p.finfo + e_next.x);
  }
  for (;;) {
    const int c = c_next;
    if (c >= total) break;
    const uint2 e = e_next;
    const int4 fi = fi_next;
    if (lane == 0) c_next = atomicAdd(p.queue, 1);
    c_next = __shfl_sync(0xffffffffu, c_next, 0);
    if (c_next < total) {
      e_next = __ldcg(p.cand + c_next);
      fi_next = __ldg(p.finfo + e_next.x);
    }
    const int j = (int)e.y;
    bool pass = true;
    if (fi.w & 2) {
      const int nf = fi.y;
      const int need = (int)((unsigned)fi.w >> 8);
      if (need > nf) {  // nothing can be kept (LL.cpp:1935-1937 would drop whatever the patch holds)
        if (lane == 0) dropped_feats += (unsigned)nf;
        pass = false;
      } else if (need > 0) {
        // patch origin of the candidate at the filtered level (LL.cpp:1871-1880, 1380-1381)
        int x = (j % p.low.Wd) * p.low.T + p.low.off;
        int y = (j / p.low.Wd) * p.low.T + p.low.off;
        x = x * 2 + 1;
        y = y * 2 + 1;
        x = max(x, border); y = max(y, border);
        x = min(x, p.ref.cols - (fi.z & 0xFFFF) - border);
        y = min(y, p.ref.rows - (int)((unsigned)fi.z >> 16) - border);
        const char* __restrict__ col = reinterpret_cast<const char*>(p.rp + (x / T - 8 + gl));  // this lane's first column
        const int cy = y / T - 8;
        const uint32_t* __restrict__ fd = p.rdesc + fi.x;
        const int nfp = (nf + 31) & ~31;  // descriptors are padded with zero-plane entries
        // check points: multiples of 32 features nearest to 1/2 and 3/4 of the template
        const int chk1 = ((nf / 2 + 31) & ~31), chk2 = ((nf * 3 / 4 + 31) & ~31);
        uint32_t ch[LM_FILTER_BITS];
#pragma unroll
        for (int b = 0; b < LM_FILTER_BITS; ++b) ch[b] = 0u;
        bool lane_alive = true, dead = false;
        uint32_t d_next = __ldg(fd + lane);
        for (int i = 0; i < nfp; i += 32) {
          // lane L decodes feature i + L: plane BYTE offset (incl. the row block of this candidate) : 27 | shift : 5
          const uint32_t d = d_next;
          if (i + 32 < nfp) d_next = __ldg(fd + i + 32 + lane);  // one step ahead
          const int py0 = cy + (int)(d >> 23);
          const uint32_t v = (((d & 0x7FFFFFu) + (uint32_t)((py0 >> 4) * Wd)) << 7) | ((uint32_t)py0 & 15u);
          uint32_t xh[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const uint32_t vu = __shfl_sync(0xffffffffu, v, u, 8);  // lane u of this lane's group
            const uint32_t* __restrict__ ptr = lm_ptr_add(col, vu >> 5);
            uint32_t w0 = 0u, w1 = 0u;
            if (lane_alive) {
              w0 = __ldg(ptr);
              w1 = __ldg(ptr + 8);
            }
            // funnel shift = shift by the low 5 bits of vu (the row offset inside the word)
            xh[u] = __byte_perm(__funnelshift_r(w0, 0u, vu), __funnelshift_r(w1, 0u, vu), 0x5410);
          }
          if (lane_alive) words_read += 16;
          vc_add8n<LM_FILTER_BITS>(ch, xh);
          const int done = i + 32;
          if ((done == chk1 || done == chk2) && done < nf) {
            vc_allreduce_groups(ch);  // every group now holds the totals of its 32 cells
            const uint32_t alive_cells = vc_ge(ch, need - (nf - done));
            lane_alive = alive_cells != 0u;
            if (!__any_sync(0xffffffffu, lane_alive)) { dead = true; break; }
            if (grp) {  // the totals live on in group 0; the others start their partial counts again
#pragma unroll
              for (int b = 0; b < LM_FILTER_BITS; ++b) ch[b] = 0u;
            }
          }
        }
        if (!dead) {
          vc_allreduce_groups(ch);
          dead = !__any_sync(0xffffffffu, vc_ge(ch, need) != 0u);
        }
        if (dead) {
          if (lane == 0) dropped_feats += (unsigned)nf;  // the reference's work for it (algorithmic bytes / 256)
          pass = false;
        }
      }
    }
    if (pass && lane == 0) {
      if (p.surv2 && !(fi.w & 2)) p.surv2[atomicAdd(p.queue + 2, 1)] = (uint32_t)c;  // byte-wise refinement (k_refine)
      else p.surv[atomicAdd(p.queue + 1, 1)] = (uint32_t)c;
    }
  }
  words_read = __reduce_add_sync(0xffffffffu, words_read);
  if (lane == 0 && (words_read | dropped_feats)) {
    atomicAdd(p.counters + 4, (unsigned long long)dropped_feats);
    atomicAdd(p.counters + 5, (unsigned long long)words_read);
  }
}

// --------------------------------------------------------------------------------------------
// K3: local refinement, one warp per coarse candidate, all upper pyramid levels
// --------------------------------------------------------------------------------------------
// Multi-GPU exchange fused into k_refine (include/linemod_b200.h, lm_peer_*): every rank's buffer is
//   [2 frame slots][world result blocks of block_bytes] [2][LM_MAX_PEERS] int32 frame flags | int32 ticket
// base[r] is rank r's buffer (a peer mapping over NVLink for r != rank).
struct PeerExchange {
  uint8_t* base[LM_MAX_PEERS];
  int world, rank;         // world == 0: no exchange
  uint32_t block_bytes;    // sizeof(lm_result_header) + capacity records
  uint32_t slot_bytes;     // world * block_bytes
  uint32_t flags_offset;   // byte offset of the flags
};                         // frames carry a sequence number seq >= 1; frame slot = seq & 1

// the exchange, record by record: the same slot of block [frame slot][rank] in every peer's buffer
// (out of line: the rare path must not cost the scoring loop registers)
static __device__ __noinline__ void peer_store_record(const PeerExchange* px, int seq, int slot, int4 r) {
  const int world = px->world, rank = px->rank;
  const size_t at = (size_t)(seq & 1) * px->slot_bytes + (size_t)rank * px->block_bytes + sizeof(lm_result_header) +
                    (size_t)slot * sizeof(lm_record);
  for (int q = 0; q < world; ++q)
    if (q != rank) *reinterpret_cast<int4*>(px->base[q] + at) = r;
}

// publish: the last CTA to finish copies the header to every peer and raises this rank's frame flag there
// (release: every CTA fences its peer stores before taking a ticket)
static __device__ __noinline__ void peer_publish(const PeerExchange* px, int seq, const lm_result_header* hdr) {
  const int world = px->world, rank = px->rank;
  __threadfence_system();
  int* ticket = reinterpret_cast<int*>(px->base[rank] + px->flags_offset) + 2 * LM_MAX_PEERS;
  if (atomicAdd(ticket, 1) != (int)gridDim.x - 1) return;
  *ticket = 0;
  __threadfence();
  const int4 h = __ldcg(reinterpret_cast<const int4*>(hdr));
  const size_t blk = (size_t)(seq & 1) * px->slot_bytes + (size_t)rank * px->block_bytes;
  for (int q = 0; q < world; ++q)
    if (q != rank) *reinterpret_cast<int4*>(px->base[q] + blk) = h;
  __threadfence_system();
  for (int q = 0; q < world; ++q) {
    volatile int32_t* flag =
        reinterpret_cast<volatile int32_t*>(px->base[q] + px->flags_offset) + (seq & 1) * LM_MAX_PEERS + rank;
    *flag = seq;
  }
}

// kept record -> result block (unordered append; (work, seq) restores the reference's pre-sort order on the host) and, in
// multi-GPU mode, the same slot of this rank's block in every peer's buffer
__device__ __forceinline__ void append_record(lm_result_header* hdr, int32_t capacity, const PeerExchange* px, int32_t px_seq,
                                              int x, int y, float sim, int work, int seq) {
  const int slot = atomicAdd(&hdr->count, 1);
  if (slot < capacity) {
    lm_record r;
    r.x = (int16_t)x; r.y = (int16_t)y; r.similarity = sim;
    r.work = work;
    r.seq = seq;
    reinterpret_cast<lm_record*>(hdr + 1)[slot] = r;
    if (px) peer_store_record(px, px_seq, slot, *reinterpret_cast<const int4*>(&r));
  }
}

struct RefineParams {
  const PeerExchange* px;  // device-resident descriptor of the fused multi-GPU exchange, or null
  int32_t px_seq;          // this frame's sequence number
  LevelDev lv[LM_MAX_LEVELS];
  const TSlot* tslot;
  const uint32_t* fbase;
  const uint32_t* fxy;
  const int32_t* work;
  const int32_t* off;    // [n_work + 1]
  const uint2* cand;     // ordered candidate list (k_refine_prep)
  int cand_cap;
  const uint16_t* raw;   // [n_work][plane_low] coarse raw scores (read when there is no level to refine)
  const uint32_t* surv;  // work items: a list of candidate indices written by k_refine_filter_w, or null: every candidate
  const int* queue;      // queue[surv_slot] = length of that list
  int surv_slot;
  int publish;           // multi-GPU: this is the last kernel of the frame that appends records
  int n_work, L, S, M;
  int work_begin, work_stride;  // entry w of this shard is element work_begin + w * work_stride of the selected sequence
  float threshold;
  lm_result_header* hdr;  // result block: header, then `capacity` records
  int32_t capacity;
  unsigned long long* counters;  // [0] features x candidates of the reference's refinement (x256 = algorithmic
                                 // bytes), [1] feature x patch rows actually read (row-wise early exit; x16 bytes)
  const uint8_t* safe;           // per template, bit 0: no feature can leave the image once a clamped patch
                                 // offset is applied (LL.cpp:1394 never skips) -> 128-bit row loads
  const uint16_t* galign;        // [G][S][16]: features per (fbase & 15) group (refined levels are stored
                                 // grouped by it)
  uint32_t* bp_clear;            // lowest level's bit-planes: consumed by the coarse scan of this frame,
  uint32_t bp_words;             // cleared here for the next frame's K1 (which ORs its bits in)
};

// One lane pair = one row of the 16x16 patch: lane `half` loads the aligned 16-byte chunk (a >> 4) +
// half; K = word offset of the row start inside the first chunk.  The lane then needs the words
// K + 2*half .. K + 2*half + 2 of the 8-word pair and gets the ones it lacks from its partner.
#define LM_REFINE_CHECK 21  // features between two early-exit tests of the refinement (<= 63)

template <int K>
__device__ __forceinline__ void refine_rows(const uint4* __restrict__ lm128, const uint32_t* __restrict__ fb, int n,
                                            uint32_t shift_row, int half, uint32_t sh, bool alive, uint32_t& a8,
                                            uint32_t& b8) {
  const bool hi = half != 0;
#pragma unroll 4
  for (int i = 0; i < n; ++i) {
    const uint32_t a = __ldg(fb + i) + shift_row;
    // a row none of whose 16 cells can still reach the keep threshold stops loading (see the row test below)
    const uint4 v = alive ? __ldg(lm128 + (a >> 4) + half) : make_uint4(0u, 0u, 0u, 0u);
    uint32_t w0, w1, w2;
    if (K == 0) {
      const uint32_t p2 = __shfl_xor_sync(0xffffffffu, v.z, 1);
      const uint32_t p3 = __shfl_xor_sync(0xffffffffu, v.w, 1);
      w0 = hi ? p2 : v.x; w1 = hi ? p3 : v.y; w2 = hi ? v.x : v.z;
    } else if (K == 1) {
      const uint32_t p3 = __shfl_xor_sync(0xffffffffu, v.w, 1);
      w0 = hi ? p3 : v.y; w1 = hi ? v.x : v.z; w2 = hi ? v.y : v.w;
    } else if (K == 2) {
      const uint32_t p0 = __shfl_xor_sync(0xffffffffu, v.x, 1);
      w0 = hi ? v.x : v.z; w1 = hi ? v.y : v.w; w2 = hi ? v.z : p0;
    } else {
      const uint32_t p0 = __shfl_xor_sync(0xffffffffu, v.x, 1);
      const uint32_t p1 = __shfl_xor_sync(0xffffffffu, v.y, 1);
      w0 = hi ? v.y : v.w; w1 = hi ? v.z : p0; w2 = hi ? v.w : p1;
    }
    a8 += __funnelshift_r(w0, w1, sh);
    b8 += __funnelshift_r(w1, w2, sh);
  }
}

#define LM_REFINE_MIN_CTAS 4
// kSplit = false: one warp per candidate, exact row-wise early exit (every coarse candidate comes here: no filter).
// kSplit = true : the work items are the filter's survivors -- few (a few percent of the candidates) and nearly all of
//   them kept, so the early exit has nothing to skip and ONE warp per candidate would leave the kernel waiting on a
//   single warp's chain of 300 dependent row loads.  Four warps share a candidate instead: warp q adds the features of the
//   alignment groups q, q + 4, q + 8, q + 12 (the features of a refined level are stored grouped by address & 15), the
//   partial 16x16 sums meet in shared memory, every warp of the quad finishes the candidate redundantly (same best cell,
//   same position for the next level) and warp 0 of the quad appends the record.
template <bool kSplit>
__global__ void __launch_bounds__(256, LM_REFINE_MIN_CTAS) k_refine(RefineParams p) {
  lm_pdl_wait();
  constexpr int Q = kSplit ? 4 : 1;
  __shared__ uint4 s_part[kSplit ? 8 : 1][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = kSplit ? (warp & 3) : 0;
  const int per_cta = kSplit ? 2 : 8;  // candidates in flight per CTA
  const int total = min(p.off[p.n_work], p.cand_cap);
  const LevelDev low = p.lv[p.L - 1];
  const int row = lane >> 1, half = lane & 1;
  unsigned feats_done = 0, rows_read = 0;  // per warp: a few candidates x (features x 16 rows)
  if (p.bp_clear)
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < p.bp_words; i += gridDim.x * blockDim.x) p.bp_clear[i] = 0u;

  // work items: the survivors of k_refine_filter_w (unordered candidate indices), or every candidate
  const int n_items = p.surv ? min(__ldcg(p.queue + p.surv_slot), total) : total;
  for (int base = blockIdx.x * per_cta; base < n_items; base += gridDim.x * per_cta) {
    const int it = base + (kSplit ? (warp >> 2) : warp);
    const bool valid = it < n_items;
    if (!kSplit && !valid) break;
    int c = 0, w = 0, g = 0, x = 0, y = 0;
    float sim = 0.f;
    if (valid) {
      c = p.surv ? (int)__ldcg(p.surv + it) : it;
      const uint2 ce = __ldcg(p.cand + c);  // (work item, cell), written in pre-sort order by k_refine_prep
      w = (int)ce.x;
      const int j = (int)ce.y;
      g = p.work[w];
      x = (j % low.Wd) * low.T + low.off;
      y = (j / low.Wd) * low.T + low.off;
      if (p.L == 1) {  // the coarse similarity is the result only when nothing is refined (one pyramid level)
        int nfeat = 0;
        for (int m = 0; m < p.M; ++m) nfeat += p.tslot[(size_t)g * p.S + (p.L - 1) * p.M + m].y;
        sim = lm_score((int)p.raw[(size_t)w * low.plane + j], nfeat);
      }
    }
    bool kept = valid;

    for (int l = p.L - 2; l >= 0 && (kSplit || kept); --l) {
      const LevelDev lv = p.lv[l];
      const int T = lv.T;
      uint32_t s01 = 0, s23 = 0, s45 = 0, s67 = 0;
      int nf_level = 0;
      bool pruned = false;
      if (kept) {
        const uint32_t* __restrict__ lm32 = reinterpret_cast<const uint32_t*>(lv.lm);
        const TSlot t0 = p.tslot[(size_t)g * p.S + l * p.M];
        const int border = 8 * T;
        const int max_x = lv.cols - (t0.w & 0xFFFF) - border;
        const int max_y = lv.rows - (int)((unsigned)t0.w >> 16) - border;
        x = x * 2 + 1;
        y = y * 2 + 1;
        x = max(x, border); y = max(y, border);  // LL.cpp:1875-1880 (max first, then min)
        x = min(x, max_x);  y = min(y, max_y);
        const int cx = x / T - 8, cy = y / T - 8;  // truncating division, LL.cpp:1380-1381
        const int ox = cx * T, oy = cy * T;
        const int shift = cy * lv.Wd + cx + row * lv.Wd + half * 8;
        for (int m = 0; m < p.M; ++m) nf_level += p.tslot[(size_t)g * p.S + l * p.M + m].y;  // all features, skipped or not (LL.cpp:1888)

        if ((p.safe[g] & 1) && (lv.Wd & 15) == 0) {
          // Fast path.  Every row of the 16x16 patch starts at the same offset inside its 16-byte
          // chunk (Wd is a multiple of 16), so the two lanes of a row fetch the two aligned chunks that
          // hold the row's 16 bytes with ONE 128-bit load each and trade the words they are missing.
          // The features of a template are stored grouped by (address & 15), so the word offset of the
          // row start (which decides who trades what) is constant over a whole group of features.
          const uint4* __restrict__ lm128 = reinterpret_cast<const uint4*>(lv.lm);
          const uint32_t shift_row = (uint32_t)(cy * lv.Wd + cx + row * lv.Wd);
          // Early exit (exact, kSplit = false only), per patch row: a candidate only produces output if its best cell
          // reaches raw_keep.  Every remaining feature adds at most 4 to any cell, so a ROW whose best cell so far +
          // 4 * remaining falls short can never hold the best cell of a kept candidate: its lane pair stops loading (its
          // stale sums stay below raw_keep, so they can neither win nor tie).  When no row is left the candidate is
          // dropped (LL.cpp:1935-1937) whatever the rest adds.  Tested every LM_REFINE_CHECK features.
          const int raw_keep = lm_min_kept_raw(p.threshold, nf_level);
          int done = 0, since = 0;
          bool alive = true;
          unsigned rows_alive = 16;
          if (q == 0) feats_done += nf_level;  // the reference's work for this candidate (algorithmic bytes / 256)
          for (int m = 0; m < p.M && !pruned; ++m) {
            const TSlot ts = p.tslot[(size_t)g * p.S + l * p.M + m];
            const uint32_t* __restrict__ fb = p.fbase + ts.x;
            const uint16_t* __restrict__ ga = p.galign + ((size_t)g * p.S + l * p.M + m) * 16;
            uint32_t a8 = 0, b8 = 0;
            int pend = 0;
            for (int grp = 0; grp < 16 && !pruned; ++grp) {
              int n = ga[grp];
              if (kSplit && (grp & (Q - 1)) != q) {  // another warp of the quad owns this alignment group
                fb += n;
                continue;
              }
              const uint32_t o = ((uint32_t)grp + shift_row) & 15u;
              const uint32_t sh = (o & 3u) << 3;
              while (n > 0) {
                const int take = min(n, LM_REFINE_CHECK - pend);
                switch (o >> 2) {
                  case 0: refine_rows<0>(lm128, fb, take, shift_row, half, sh, alive, a8, b8); break;
                  case 1: refine_rows<1>(lm128, fb, take, shift_row, half, sh, alive, a8, b8); break;
                  case 2: refine_rows<2>(lm128, fb, take, shift_row, half, sh, alive, a8, b8); break;
                  default: refine_rows<3>(lm128, fb, take, shift_row, half, sh, alive, a8, b8); break;
                }
                fb += take;
                n -= take;
                pend += take;
                done += take;
                since += take;
                if (pend == LM_REFINE_CHECK) {  // <= 63: 63 * 4 = 252, no carry between packed bytes
                  s01 += __byte_perm(a8, 0, 0x4140); s23 += __byte_perm(a8, 0, 0x4342);
                  s45 += __byte_perm(b8, 0, 0x4140); s67 += __byte_perm(b8, 0, 0x4342);
                  a8 = b8 = 0;
                  pend = 0;
                  if (!kSplit) {
                    uint32_t mx = max(max(max(s01 & 0xFFFF, s01 >> 16), max(s23 & 0xFFFF, s23 >> 16)),
                                      max(max(s45 & 0xFFFF, s45 >> 16), max(s67 & 0xFFFF, s67 >> 16)));
                    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, 1));  // the row's 16 cells
                    rows_read += (unsigned)since * rows_alive;
                    since = 0;
                    alive = alive && ((int)mx + 4 * (nf_level - done) >= raw_keep);
                    const unsigned live = __ballot_sync(0xffffffffu, alive);
                    rows_alive = (unsigned)__popc(live) >> 1;
                    if (live == 0u) { pruned = true; break; }
                  }
                }
              }
            }
            s01 += __byte_perm(a8, 0, 0x4140); s23 += __byte_perm(a8, 0, 0x4342);
            s45 += __byte_perm(b8, 0, 0x4140); s67 += __byte_perm(b8, 0, 0x4342);
          }
          rows_read += (unsigned)since * rows_alive;
        } else {
          for (int m = 0; m < p.M; ++m) {
            const TSlot ts = p.tslot[(size_t)g * p.S + l * p.M + m];
            uint32_t a8 = 0, b8 = 0;
            int pend = 0;
            for (int i = q; i < ts.y; i += Q) {
              const uint32_t xy = __ldg(p.fxy + ts.x + i);
              const int fx = (int)(xy & 0x7FFFu) + ox, fy = (int)((xy >> 16) & 0x7FFFu) + oy;
              if (fx < 0 || fy < 0 || fx >= lv.cols || fy >= lv.rows) continue;  // LL.cpp:1394
              const uint32_t a = __ldg(p.fbase + ts.x + i) + (uint32_t)shift;
              const uint32_t w0 = __ldg(lm32 + (a >> 2));
              const uint32_t w1 = __ldg(lm32 + (a >> 2) + 1);
              const uint32_t w2 = __ldg(lm32 + (a >> 2) + 2);
              const uint32_t sh = (a & 3u) << 3;
              a8 += __funnelshift_r(w0, w1, sh);
              b8 += __funnelshift_r(w1, w2, sh);
              ++feats_done;
              rows_read += 16;
              if (++pend == 63) {
                s01 += __byte_perm(a8, 0, 0x4140); s23 += __byte_perm(a8, 0, 0x4342);
                s45 += __byte_perm(b8, 0, 0x4140); s67 += __byte_perm(b8, 0, 0x4342);
                a8 = b8 = 0;
                pend = 0;
              }
            }
            s01 += __byte_perm(a8, 0, 0x4140); s23 += __byte_perm(a8, 0, 0x4342);
            s45 += __byte_perm(b8, 0, 0x4140); s67 += __byte_perm(b8, 0, 0x4342);
          }
        }
      }
      if (kSplit) {
        // the quad's partial sums meet: u16 pairs, at most 4 * 8191 per cell in total -> no carry between the halves
        s_part[warp][lane] = make_uint4(s01, s23, s45, s67);
        __syncthreads();
        const int w0 = warp & ~3;
        const uint4 a = s_part[w0][lane], b = s_part[w0 + 1][lane], cc = s_part[w0 + 2][lane], dd = s_part[w0 + 3][lane];
        s01 = a.x + b.x + cc.x + dd.x; s23 = a.y + b.y + cc.y + dd.y;
        s45 = a.z + b.z + cc.z + dd.z; s67 = a.w + b.w + cc.w + dd.w;
        __syncthreads();  // before the next level / candidate overwrites the partials
      }
      if (kept) {
        // best cell: strict > in row-major order == max raw, lowest cell index (LL.cpp:1910-1927)
        const uint32_t v[8] = {s01 & 0xFFFF, s01 >> 16, s23 & 0xFFFF, s23 >> 16,
                               s45 & 0xFFFF, s45 >> 16, s67 & 0xFFFF, s67 >> 16};
        uint32_t key = 0;
        const int cell0 = row * 16 + half * 8;
#pragma unroll
        for (int k = 0; k < 8; ++k) key = max(key, (v[k] << 8) | (uint32_t)(255 - (cell0 + k)));
        key = __reduce_max_sync(0xffffffffu, key);
        const int best_raw = (int)(key >> 8);
        int br = -1, bc = -1;
        if (best_raw > 0) {
          const int cell = 255 - (int)(key & 255u);
          br = cell >> 4;
          bc = cell & 15;
        }
        sim = lm_score(best_raw, nf_level);
        x = (x / T - 8 + bc) * T + lv.off;  // LL.cpp:1930-1931
        y = (y / T - 8 + br) * T + lv.off;
        kept = !pruned && !(sim < p.threshold);  // remove_if(similarity < threshold), LL.cpp:1935-1937
      }
    }
    if (lane == 0 && kept && q == 0)
      append_record(p.hdr, p.capacity, p.px, p.px_seq, x, y, sim, p.work_begin + w * p.work_stride, c);
  }
  if (lane == 0 && (feats_done | rows_read)) {
    atomicAdd(p.counters + 0, (unsigned long long)feats_done);
    atomicAdd(p.counters + 1, (unsigned long long)rows_read);
  }
  if (p.px && p.publish) {
    __syncthreads();
    if (threadIdx.x == 0) peer_publish(p.px, p.px_seq, p.hdr);
  }
}

// --------------------------------------------------------------------------------------------
// k_refine_bits: the exact refinement of the filter's survivors, bit-sliced (two pyramid levels, i.e. the refined level
// is level 0: the reference's default; deeper pyramids and the templates the filter does not take go to k_refine).
//
// similarityLocal's response is 4*H + N with H = the feature's label bit in the spread mask and N = (either neighbouring
// label bit) & ~H (lm_response), so the exact 16x16 sums are raw = 4*CH + CN.  Same warp layout as k_refine_filter_w
// (four 8-lane groups deal the features of the candidate between them, lane k of a group holds patch columns k and k + 8),
// but three H-plane windows per feature (labels o - 1, o, o + 1) and two vertical counters.  The partial counters meet
// once, at the end; the score 4*CH + CN, the best cell (max raw, lowest cell index = first maximum in row-major order,
// LL.cpp:1910-1927) and the keep test (LL.cpp:1935-1937) are evaluated bit-sliced.  The byte linear memories are never
// touched.
// --------------------------------------------------------------------------------------------
struct RefineBitsParams {
  const uint32_t* rp;      // H-planes of level 0 (k_refine_prep), zero tail behind
  int Wd;
  int label_stride;        // words between the planes of consecutive labels: T*T * nyb * Wd
  const uint32_t* rdesc;   // as FilterParams (padded to multiples of 32 per template)
  const uint8_t* rlab;     // per descriptor: the feature's label 0..7, 8 = padding
  const int4* finfo;
  LevelDev low, ref;
  const uint2* cand;
  const int32_t* off;
  int n_work, cand_cap;
  const uint32_t* surv;
  const int* queue;        // [1] survivors
  float threshold;
  int work_begin, work_stride;
  lm_result_header* hdr;
  int32_t capacity;
  const PeerExchange* px;
  int32_t px_seq;
  int publish;
  unsigned long long* counters;  // [0] features x candidates refined here, [5] plane words read
  uint32_t* bp_clear;
  uint32_t bp_words;
};

// bit-sliced add of two vertical counters
__device__ __forceinline__ void vc_add(uint32_t (&c)[LM_FILTER_BITS], const uint32_t (&o)[LM_FILTER_BITS]) {
  uint32_t carry = 0u;
#pragma unroll
  for (int b = 0; b < LM_FILTER_BITS; ++b) {
    const uint32_t a = c[b], x = o[b];
    c[b] = a ^ x ^ carry;
    carry = (a & x) | (carry & (a ^ x));
  }
}

// Four warps share a survivor (a candidate is a chain of nf / 32 dependent steps, and the survivors are too few to hide
// it with other warps): warp q of the quad takes the 32-feature steps q, q + 4, ..., the partial counters meet in shared
// memory and warp 0 of the quad finishes the candidate.
__global__ void __launch_bounds__(256, 4) k_refine_bits(RefineBitsParams p) {
  lm_pdl_wait();
  __shared__ uint32_t s_part[8][2 * LM_FILTER_BITS][32];
  const int lane = threadIdx.x & 31, gl = lane & 7, warp = threadIdx.x >> 5;
  const int quad = warp >> 2, q = warp & 3;
  const int total = min(p.off[p.n_work], p.cand_cap);
  const int n_items = min(__ldcg(p.queue + 1), total);
  const int T = p.ref.T, border = 8 * T;
  const int Wd = p.Wd;
  unsigned feats_done = 0, words_read = 0;
  if (p.bp_clear)
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < p.bp_words; i += gridDim.x * blockDim.x) p.bp_clear[i] = 0u;

  for (int base = blockIdx.x * 2; base < n_items; base += gridDim.x * 2) {
    const int it = base + quad;
    const bool valid = it < n_items;
    int c = 0, w = 0, x = 0, y = 0, nf = 0;
    uint32_t ch[LM_FILTER_BITS], cn[LM_FILTER_BITS];
#pragma unroll
    for (int b = 0; b < LM_FILTER_BITS; ++b) ch[b] = cn[b] = 0u;
    if (valid) {
      c = (int)__ldcg(p.surv + it);
      const uint2 e = __ldcg(p.cand + c);
      w = (int)e.x;
      const int j = (int)e.y;
      const int4 fi = __ldg(p.finfo + w);
      nf = fi.y;
      x = (j % p.low.Wd) * p.low.T + p.low.off;
      y = (j / p.low.Wd) * p.low.T + p.low.off;
      x = x * 2 + 1;
      y = y * 2 + 1;
      x = max(x, border); y = max(y, border);  // LL.cpp:1875-1880 (max first, then min)
      x = min(x, p.ref.cols - (fi.z & 0xFFFF) - border);
      y = min(y, p.ref.rows - (int)((unsigned)fi.z >> 16) - border);
      const char* __restrict__ col = reinterpret_cast<const char*>(p.rp + (x / T - 8 + gl));
      const int cy = y / T - 8;
      const uint32_t* __restrict__ fd = p.rdesc + fi.x;
      const uint8_t* __restrict__ fl = p.rlab + fi.x;
      const int nfp = (nf + 31) & ~31;
      if (q == 0) feats_done += (unsigned)nf;

      for (int i = q * 32; i < nfp; i += 128) {
        // lane L decodes feature i + L: word offsets of the three label planes (row block of this candidate included)
        // : 27 | row shift : 5
        const uint32_t d = __ldg(fd + i + lane);
        const int o = (int)__ldg(fl + i + lane);
        const int py0 = cy + (int)(d >> 23);
        const uint32_t idx = (d & 0x7FFFFFu) + (uint32_t)((py0 >> 4) * Wd);
        const uint32_t sft = (uint32_t)py0 & 15u;
        const int dm = o >= 8 ? 0 : (o == 0 ? 7 * p.label_stride : -p.label_stride);
        const int dp = o >= 7 ? (o == 7 ? -7 * p.label_stride : 0) : p.label_stride;
        const uint32_t v0 = (idx << 7) | sft;  // byte offset : 27 | row shift : 5
        const uint32_t vm = ((uint32_t)((int)idx + dm) << 7) | sft;
        const uint32_t vp = ((uint32_t)((int)idx + dp) << 7) | sft;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          uint32_t xh[4], xn[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int src = half * 4 + u;  // lane `src` of this lane's group
            const uint32_t a0 = __shfl_sync(0xffffffffu, v0, src, 8);
            const uint32_t am = __shfl_sync(0xffffffffu, vm, src, 8);
            const uint32_t ap = __shfl_sync(0xffffffffu, vp, src, 8);
            const uint32_t* __restrict__ p0 = lm_ptr_add(col, a0 >> 5);
            const uint32_t* __restrict__ pm = lm_ptr_add(col, am >> 5);
            const uint32_t* __restrict__ pp = lm_ptr_add(col, ap >> 5);
            const uint32_t h = __byte_perm(__funnelshift_r(__ldg(p0), 0u, a0), __funnelshift_r(__ldg(p0 + 8), 0u, a0), 0x5410);
            const uint32_t a = __byte_perm(__funnelshift_r(__ldg(pm), 0u, a0), __funnelshift_r(__ldg(pm + 8), 0u, a0), 0x5410);
            const uint32_t b = __byte_perm(__funnelshift_r(__ldg(pp), 0u, a0), __funnelshift_r(__ldg(pp + 8), 0u, a0), 0x5410);
            xh[u] = h;
            xn[u] = (a | b) & ~h;
          }
          // four 1-bit planes into each vertical counter
          uint32_t t1a, t1b, t2;
          CSA(ch[0], t1a, ch[0], xh[0], xh[1]);
          CSA(ch[0], t1b, ch[0], xh[2], xh[3]);
          CSA(ch[1], t2, ch[1], t1a, t1b);
#pragma unroll
          for (int b = 2; b < LM_FILTER_BITS; ++b) { const uint32_t k = ch[b] & t2; ch[b] ^= t2; t2 = k; }
          CSA(cn[0], t1a, cn[0], xn[0], xn[1]);
          CSA(cn[0], t1b, cn[0], xn[2], xn[3]);
          CSA(cn[1], t2, cn[1], t1a, t1b);
#pragma unroll
          for (int b = 2; b < LM_FILTER_BITS; ++b) { const uint32_t k = cn[b] & t2; cn[b] ^= t2; t2 = k; }
        }
        words_read += 48;
      }
    }
    // the quad's partial counters meet
    if (q != 0) {
#pragma unroll
      for (int b = 0; b < LM_FILTER_BITS; ++b) {
        s_part[warp][b][lane] = ch[b];
        s_part[warp][LM_FILTER_BITS + b][lane] = cn[b];
      }
    }
    __syncthreads();
    if (q == 0 && valid) {
#pragma unroll
      for (int k = 1; k < 4; ++k) {
        uint32_t oh[LM_FILTER_BITS], on[LM_FILTER_BITS];
#pragma unroll
        for (int b = 0; b < LM_FILTER_BITS; ++b) {
          oh[b] = s_part[warp + k][b][lane];
          on[b] = s_part[warp + k][LM_FILTER_BITS + b][lane];
        }
        vc_add(ch, oh);
        vc_add(cn, on);
      }
      vc_allreduce_groups(ch);
      vc_allreduce_groups(cn);
      // raw = 4*CH + CN, 11 bits (4 * 511 < 2048)
      uint32_t sc[11];
      sc[0] = cn[0];
      sc[1] = cn[1];
      uint32_t carry = 0u;
#pragma unroll
      for (int b = 2; b < 11; ++b) {
        const uint32_t a = (b < LM_FILTER_BITS) ? cn[b] : 0u;
        const uint32_t h = ch[b - 2];
        sc[b] = a ^ h ^ carry;
        carry = (a & h) | (carry & (a ^ h));
      }
      // best raw score: highest bit first, keep the cells that still tie for the maximum
      uint32_t cells = 0xffffffffu;
      int best_raw = 0;
#pragma unroll
      for (int b = 10; b >= 0; --b) {
        const uint32_t t = cells & sc[b];
        if (__any_sync(0xffffffffu, t != 0u)) {
          cells = t;
          best_raw |= 1 << b;
        }
      }
      // first maximum in row-major order: lowest row, then lowest column (bits 0..15 = rows of column gl, 16..31 = of
      // gl + 8)
      int cell = 0x7fffffff;
      if (cells & 0xFFFFu) cell = (__ffs(cells & 0xFFFFu) - 1) * 16 + gl;
      if (cells >> 16) cell = min(cell, (__ffs(cells >> 16) - 1) * 16 + gl + 8);
      cell = __reduce_min_sync(0xffffffffu, cell);
      int br = -1, bc = -1;
      if (best_raw > 0) {
        br = cell >> 4;
        bc = cell & 15;
      }
      const float sim = lm_score(best_raw, nf);
      x = (x / T - 8 + bc) * T + p.ref.off;  // LL.cpp:1930-1931
      y = (y / T - 8 + br) * T + p.ref.off;
      if (lane == 0 && !(sim < p.threshold))  // remove_if(similarity < threshold), LL.cpp:1935-1937
        append_record(p.hdr, p.capacity, p.px, p.px_seq, x, y, sim, p.work_begin + w * p.work_stride, c);
    }
    __syncthreads();  // before the next candidate's partials overwrite these
  }
  words_read = __reduce_add_sync(0xffffffffu, words_read);
  if (lane == 0 && (feats_done | words_read)) {
    atomicAdd(p.counters + 0, (unsigned long long)feats_done);
    atomicAdd(p.counters + 5, (unsigned long long)words_read);
  }
  if (p.px && p.publish) {
    __syncthreads();
    if (threadIdx.x == 0) peer_publish(p.px, p.px_seq, p.hdr);
  }
}

// Abort flag of the fused exchange, one per device (module-scope variable): the first collector that gives up on a peer
// raises it and every later collector of ANY handle / lane on this device returns at once instead of spinning through
// its own timeout -- one stalled rank costs one timeout, not lanes x frames of them.  Cleared by lm_peer_export.
__device__ int g_px_abort = 0;

// Collector of the fused exchange: waits until every rank's frame flag for `seq` has arrived in THIS rank's
// buffer, then packs the `world` blocks of the frame slot into one ordinary result block (header.count =
// all shards' kept records).  status: 0 ok, 1 a peer did not publish within the timeout (or an earlier collector
// on this device already gave up), 2 a block overflowed its capacity.  One CTA.
__global__ void __launch_bounds__(1024) k_peer_collect(PeerExchange px, int32_t seq, int32_t block_capacity, lm_result_header* out_hdr,
                                                       int32_t out_capacity, unsigned long long* status,
                                                       unsigned long long timeout_ns) {
  lm_pdl_wait();
  __shared__ int s_cnt[LM_MAX_PEERS + 1];
  __shared__ int s_coarse[LM_MAX_PEERS];
  __shared__ int s_status;
  const int tid = threadIdx.x;
  if (tid == 0) s_status = 0;
  __syncthreads();
  const uint8_t* mine = px.base[px.rank];
  if (tid < px.world) {
    const volatile int32_t* flag = reinterpret_cast<const volatile int32_t*>(mine + px.flags_offset) +
                                   (seq & 1) * LM_MAX_PEERS + tid;
    const volatile int* abort_flag = &g_px_abort;
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    bool ok = true;
    while ((int32_t)(*flag - seq) < 0) {
      if (*abort_flag) { ok = false; break; }
      __nanosleep(200);
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > timeout_ns) {  // a peer never enqueued this frame (or died)
        atomicExch(&g_px_abort, 1);
        ok = false;
        break;
      }
    }
    __threadfence_system();  // acquire: the block contents were fenced before the flag
    const lm_result_header* h = reinterpret_cast<const lm_result_header*>(
        mine + (size_t)(seq & 1) * px.slot_bytes + (size_t)tid * px.block_bytes);
    const int4 hv = ok ? __ldcv(reinterpret_cast<const int4*>(h)) : make_int4(0, 0, 0, 0);
    if (!ok) atomicMax(&s_status, 1);
    if (hv.x > block_capacity) atomicMax(&s_status, 2);
    s_cnt[tid] = min(hv.x, block_capacity);
    s_coarse[tid] = hv.y;
  }
  __syncthreads();
  if (tid == 0) {
    int run = 0, coarse = 0;
    for (int r = 0; r < px.world; ++r) {
      const int c = s_cnt[r];
      s_cnt[r] = run;
      run += c;
      coarse += s_coarse[r];
    }
    s_cnt[px.world] = run;
    out_hdr->count = run;
    out_hdr->coarse_candidates = coarse;
    out_hdr->capacity = out_capacity;
    out_hdr->shard = -1;  // all shards
    status[0] = (unsigned long long)s_status;
  }
  __syncthreads();
  int4* out = reinterpret_cast<int4*>(out_hdr + 1);
  for (int r = 0; r < px.world; ++r) {
    const int4* src = reinterpret_cast<const int4*>(mine + (size_t)(seq & 1) * px.slot_bytes +
                                                    (size_t)r * px.block_bytes + sizeof(lm_result_header));
    const int b = s_cnt[r], n = s_cnt[r + 1] - b;
    for (int i = tid; i < n; i += blockDim.x)
      if (b + i < out_capacity) out[b + i] = __ldcv(src + i);  // peers wrote them: never from a stale L1 line
  }
}
