// lm_frontend.cuh -- quantization front-end on the GPU (SURVEY.md section 8 row f-1).
//
// Reference being replaced (linemodLevelup/linemodLevelup.cpp of meiqua/6DPose @ 619be57, "LL.cpp"):
//   k_fe_gradient    <- quantizedOrientations: GaussianBlur 7x7 + Sobel + strongest channel + cv::phase +
//                       16-bin quantisation, border zeroing, &7                       LL.cpp:350-455
//   k_fe_hysteresis  <- hysteresisGradient: 3x3 vote, magnitude gate, mask (quantize)   LL.cpp:457-505, 583-587
//   k_fe_pyrdown     <- cv::pyrDown of the colour image                                 LL.cpp:557-567
//   k_fe_normals     <- quantizedNormals (before the median)                            LL.cpp:729-817
//   k_fe_median      <- medianBlur(dst, dst, 5) + mask (quantize)                       LL.cpp:818, 882-886
//   k_fe_decimate    <- resize(..., INTER_NEAREST) of labels / masks                    LL.cpp:865-879
//
// The OpenCV calls are restated in the arithmetic OpenCV itself uses for these types, each verified
// bit-exact against cv2 4.13 (tests/test_gpu_frontend.py; models in tests/test_frontend_models.py):
//   * GaussianBlur(7x7, sigma 0) on u8: fixed-point, kernel {8,28,56,72,56,28,8}/256 per axis (OpenCV's
//     small_gaussian_tab for ksize 7), result (sum + 2^15) >> 16, BORDER_REPLICATE;
//   * Sobel 3x3 -> s16, BORDER_REPLICATE on the blurred image;
//   * cv::phase(degrees) = fastAtan2's 7th-order polynomial in float; only the 16-bin quantisation
//     of the angle is kept, and with separately rounded float operations that bin equals OpenCV's for
//     every (dx, dy) in the Sobel range [-1020, 1020]^2 (exhaustively checked);
//   * pyrDown: separable {1,4,6,4,1}, BORDER_REFLECT_101, (sum + 128) >> 8;
//   * medianBlur 5x5 with BORDER_REPLICATE (labels are one-hot: a 9-bin counting median).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

__device__ __forceinline__ void lm_pdl_wait();

// ---- colour: blur + sobel + channel pick + phase bin -----------------------------------------------
#define FE_TW 32
#define FE_TH 8

__device__ __forceinline__ int fe_phase_bin(float x, float y) {
  // cv::fastAtan2 (degrees) with separately rounded operations, then Mat::convertTo(CV_8U, 16/360)
  const float p1 = __fmul_rn(0.9997878412794807f, 57.29577951308232f);
  const float p3 = __fmul_rn(-0.3258083974640975f, 57.29577951308232f);
  const float p5 = __fmul_rn(0.1555786518463281f, 57.29577951308232f);
  const float p7 = __fmul_rn(-0.04432655554792128f, 57.29577951308232f);
  const float ax = fabsf(x), ay = fabsf(y);
  const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
  const float c = __fdiv_rn(mn, __fadd_rn(mx, 2.220446049250313e-16f));
  const float c2 = __fmul_rn(c, c);
  float a = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c);
  if (ay > ax) a = __fsub_rn(90.f, a);
  if (x < 0.f) a = __fsub_rn(180.f, a);
  if (y < 0.f) a = __fsub_rn(360.f, a);
  return __float2int_rn(__fmul_rn(a, 0.044444445f));  // 16/360 as float, round half to even
}

// src u8 [H][W][3]; out: qun u8 [H][W] = (bin & 7) in the interior, 0 on the border; strong u8 = mag > thr_sq;
// mag (nullable, template extraction only): the squared magnitude of the picked channel, an exact integer <= 2 * 1020^2
__global__ void __launch_bounds__(FE_TW * FE_TH) k_fe_gradient(const uint8_t* __restrict__ src, int H, int W, int thr_sq,
                                                              uint8_t* __restrict__ qun, uint8_t* __restrict__ strong,
                                                              int32_t* __restrict__ mag) {
  lm_pdl_wait();
  __shared__ uint8_t s_in[FE_TH + 8][FE_TW + 8][3];
  __shared__ uint16_t s_h[FE_TH + 8][FE_TW + 2][3];
  __shared__ uint8_t s_b[FE_TH + 2][FE_TW + 2][3];
  const int x0 = blockIdx.x * FE_TW, y0 = blockIdx.y * FE_TH;
  const int tid = threadIdx.y * FE_TW + threadIdx.x, nthr = FE_TW * FE_TH;
  // input tile with a halo of 4 (3 for the blur + 1 for the Sobel), coordinates clamped = BORDER_REPLICATE
  for (int i = tid; i < (FE_TH + 8) * (FE_TW + 8); i += nthr) {
    const int r = i / (FE_TW + 8), c = i - r * (FE_TW + 8);
    const int y = min(max(y0 + r - 4, 0), H - 1), x = min(max(x0 + c - 4, 0), W - 1);
    const uint8_t* p = src + ((size_t)y * W + x) * 3;
    s_in[r][c][0] = p[0]; s_in[r][c][1] = p[1]; s_in[r][c][2] = p[2];
  }
  __syncthreads();
  // The Sobel replicates the border of the BLURRED image, so the blurred value is needed at the clamped
  // coordinates (clamp(x0+c-1), clamp(y0+r-1)); every blur tap is clamped to the image on its own.
  // s_in row r holds image row clamp(y0+r-4), column c holds image column clamp(x0+c-4).
  for (int i = tid; i < (FE_TH + 8) * (FE_TW + 2); i += nthr) {
    const int r = i / (FE_TW + 2), c = i - r * (FE_TW + 2);
    const int xc = min(max(x0 + c - 1, 0), W - 1);  // clamped centre
    const int k[7] = {8, 28, 56, 72, 56, 28, 8};
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      int acc = 0;
#pragma unroll
      for (int t = 0; t < 7; ++t) {
        const int xt = min(max(xc + t - 3, 0), W - 1);
        acc += k[t] * (int)s_in[r][xt - x0 + 4][ch];
      }
      s_h[r][c][ch] = (uint16_t)acc;
    }
  }
  __syncthreads();
  for (int i = tid; i < (FE_TH + 2) * (FE_TW + 2); i += nthr) {
    const int r = i / (FE_TW + 2), c = i - r * (FE_TW + 2);  // row r <-> image y = y0 + r - 1
    const int yc = min(max(y0 + r - 1, 0), H - 1);
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      unsigned acc = 0;
      const unsigned k[7] = {8, 28, 56, 72, 56, 28, 8};
#pragma unroll
      for (int t = 0; t < 7; ++t) {
        const int yt = min(max(yc + t - 3, 0), H - 1);
        acc += k[t] * (unsigned)s_h[yt - y0 + 4][c][ch];
      }
      s_b[r][c][ch] = (uint8_t)((acc + 32768u) >> 16);
    }
  }
  __syncthreads();
  const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
  if (x >= W || y >= H) return;
  const int r = threadIdx.y + 1, c = threadIdx.x + 1;
  int dxs[3], dys[3], mags[3];
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) {
    const int a00 = s_b[r - 1][c - 1][ch], a01 = s_b[r - 1][c][ch], a02 = s_b[r - 1][c + 1][ch];
    const int a10 = s_b[r][c - 1][ch], a12 = s_b[r][c + 1][ch];
    const int a20 = s_b[r + 1][c - 1][ch], a21 = s_b[r + 1][c][ch], a22 = s_b[r + 1][c + 1][ch];
    dxs[ch] = (a02 + 2 * a12 + a22) - (a00 + 2 * a10 + a20);
    dys[ch] = (a20 + 2 * a21 + a22) - (a00 + 2 * a01 + a02);
    mags[ch] = dxs[ch] * dxs[ch] + dys[ch] * dys[ch];
  }
  // strongest channel, tie order of LL.cpp:395-412
  int pick = 2;
  if (mags[0] >= mags[1] && mags[0] >= mags[2]) pick = 0;
  else if (mags[1] >= mags[0] && mags[1] >= mags[2]) pick = 1;
  const int bdx = pick == 0 ? dxs[0] : (pick == 1 ? dxs[1] : dxs[2]);
  const int bdy = pick == 0 ? dys[0] : (pick == 1 ? dys[1] : dys[2]);
  const int bm = pick == 0 ? mags[0] : (pick == 1 ? mags[1] : mags[2]);
  int bin = 0;
  if (!(x == 0 || y == 0 || x == W - 1 || y == H - 1)) bin = fe_phase_bin((float)bdx, (float)bdy) & 7;
  qun[(size_t)y * W + x] = (uint8_t)bin;
  strong[(size_t)y * W + x] = bm > thr_sq ? 1 : 0;
  if (mag) mag[(size_t)y * W + x] = bm;
}

// 3x3 vote among the 8 bins, gate on the magnitude, >= 5 votes, optional mask (LL.cpp:457-505, 583-587)
__global__ void __launch_bounds__(256) k_fe_hysteresis(const uint8_t* __restrict__ qun, const uint8_t* __restrict__ strong,
                                                      const uint8_t* __restrict__ mask, int H, int W, uint8_t* __restrict__ out) {
  lm_pdl_wait();
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= W || y >= H) return;
  uint8_t res = 0;
  if (x > 0 && y > 0 && x < W - 1 && y < H - 1 && strong[(size_t)y * W + x]) {
    uint32_t lo = 0, hi = 0;  // 8 nibble counters (max 9 fits in 4 bits)
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
      for (int dx = -1; dx <= 1; ++dx) {
        const int b = qun[(size_t)(y + dy) * W + x + dx];
        if (b < 4) lo += 1u << (8 * b); else hi += 1u << (8 * (b - 4));
      }
    int best = 0, idx = -1;
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int v = (int)(((b < 4 ? lo : hi) >> (8 * (b & 3))) & 0xFFu);
      if (best < v) { best = v; idx = b; }
    }
    if (best >= 5) res = (uint8_t)(1u << idx);
  }
  if (mask && mask[(size_t)y * W + x] == 0) res = 0;
  out[(size_t)y * W + x] = res;
}

// cv::pyrDown on u8 x 3: {1,4,6,4,1} separable, BORDER_REFLECT_101, (sum + 128) >> 8; dst = (W/2, H/2)
__device__ __forceinline__ int fe_reflect101(int p, int n) {
  if (p < 0) p = -p;
  if (p >= n) p = 2 * n - 2 - p;
  return min(max(p, 0), n - 1);
}

__global__ void __launch_bounds__(256) k_fe_pyrdown(const uint8_t* __restrict__ src, int H, int W, uint8_t* __restrict__ dst, int Hd, int Wd) {
  lm_pdl_wait();
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= Wd || y >= Hd) return;
  const int k[5] = {1, 4, 6, 4, 1};
  int acc[3] = {0, 0, 0};
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    const int yy = fe_reflect101(2 * y + j - 2, H);
    int row[3] = {0, 0, 0};
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const int xx = fe_reflect101(2 * x + i - 2, W);
      const uint8_t* p = src + ((size_t)yy * W + xx) * 3;
      row[0] += k[i] * p[0]; row[1] += k[i] * p[1]; row[2] += k[i] * p[2];
    }
    acc[0] += k[j] * row[0]; acc[1] += k[j] * row[1]; acc[2] += k[j] * row[2];
  }
  uint8_t* o = dst + ((size_t)y * Wd + x) * 3;
  o[0] = (uint8_t)((acc[0] + 128) >> 8); o[1] = (uint8_t)((acc[1] + 128) >> 8); o[2] = (uint8_t)((acc[2] + 128) >> 8);
}

// ---- depth: quantized surface normals ----------------------------------------------------------------
__constant__ uint8_t c_normal_lut[400];  // NORMAL_LUT[.][vy][vx] of normal_lut.i (independent of the first index)

__global__ void __launch_bounds__(256) k_fe_normals(const uint16_t* __restrict__ depth, int H, int W, int distance_threshold,
                                                   int difference_threshold, uint8_t* __restrict__ out) {
  lm_pdl_wait();
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= W || y >= H) return;
  uint8_t res = 0;
  const int r = 5;
  if (y >= r && y < H - r - 1 && x >= r && x < W - r - 1) {  // note the extra -1 (LL.cpp:753, 758)
    const long long d = depth[(size_t)y * W + x];
    if (d < distance_threshold) {
      long long A0 = 0, A1 = 0, A3 = 0, b0 = 0, b1 = 0;
#pragma unroll
      for (int j = -1; j <= 1; ++j)
#pragma unroll
        for (int i = -1; i <= 1; ++i) {
          if (i == 0 && j == 0) continue;
          const long long delta = (long long)depth[(size_t)(y + j * r) * W + x + i * r] - d;
          const long long f = (delta < 0 ? -delta : delta) < difference_threshold ? 1 : 0;
          const long long fi = f * (i * r), fj = f * (j * r);
          A0 += fi * (i * r); A1 += fi * (j * r); A3 += fj * (j * r);
          b0 += fi * delta; b1 += fj * delta;
        }
      const long long det = A0 * A3 - A1 * A1;
      const long long ddx = A3 * b0 - A1 * b1;
      const long long ddy = -A1 * b0 + A0 * b1;
      float nx = __ll2float_rn(1150 * ddx), ny = __ll2float_rn(1150 * ddy), nz = __ll2float_rn(-det * d);
      const float s = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(nx, nx), __fmul_rn(ny, ny)), __fmul_rn(nz, nz)));
      if (s > 0.f) {
        const float inv = __fdiv_rn(1.0f, s);
        nx = __fmul_rn(nx, inv); ny = __fmul_rn(ny, inv); nz = __fmul_rn(nz, inv);
        int v1 = __float2int_rz(__fadd_rn(__fmul_rn(nx, 10.f), 10.f));
        int v2 = __float2int_rz(__fadd_rn(__fmul_rn(ny, 10.f), 10.f));
        v1 = min(max(v1, 0), 19); v2 = min(max(v2, 0), 19);  // vz does not select anything (table independent of it)
        res = c_normal_lut[v2 * 20 + v1];
      }
    }
  }
  out[(size_t)y * W + x] = res;
}

// medianBlur 5x5 (BORDER_REPLICATE) of one-hot labels: counting median over the 9 possible values
__global__ void __launch_bounds__(256) k_fe_median(const uint8_t* __restrict__ in, const uint8_t* __restrict__ mask, int H, int W,
                                                  uint8_t* __restrict__ normal, uint8_t* __restrict__ quantized) {
  lm_pdl_wait();
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= W || y >= H) return;
  uint32_t c0 = 0, c1 = 0, c2 = 0;  // nine 5-bit counters would do; use 8-bit lanes: [0,1,2,4] [8,16,32,64] [128]
#pragma unroll
  for (int j = -2; j <= 2; ++j) {
    const int yy = min(max(y + j, 0), H - 1);
#pragma unroll
    for (int i = -2; i <= 2; ++i) {
      const int xx = min(max(x + i, 0), W - 1);
      const uint32_t v = in[(size_t)yy * W + xx];
      const int slot = v ? 32 - __clz(v) : 0;  // 0 -> 0, 1 -> 1, 2 -> 2, 4 -> 3, ..., 128 -> 8
      if (slot < 4) c0 += 1u << (8 * slot); else if (slot < 8) c1 += 1u << (8 * (slot - 4)); else c2 += 1u;
    }
  }
  int cum = 0, med = 0;
#pragma unroll
  for (int s = 0; s < 9; ++s) {
    const int cnt = (int)(((s < 4 ? c0 : (s < 8 ? c1 : c2)) >> (8 * (s & 3))) & 0xFFu);
    if (cum < 13 && cum + cnt >= 13) med = s;
    cum += cnt;
  }
  const uint8_t val = med ? (uint8_t)(1u << (med - 1)) : 0;
  normal[(size_t)y * W + x] = val;
  quantized[(size_t)y * W + x] = (mask && mask[(size_t)y * W + x] == 0) ? 0 : val;
}

// resize(INTER_NEAREST) to half size (labels and masks); optional mask applied to a second output
__global__ void __launch_bounds__(256) k_fe_decimate(const uint8_t* __restrict__ in, int W, uint8_t* __restrict__ out, int Hd, int Wd,
                                                    const uint8_t* __restrict__ mask, uint8_t* __restrict__ quantized) {
  lm_pdl_wait();
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= Wd || y >= Hd) return;
  const uint8_t v = in[(size_t)(2 * y) * W + 2 * x];
  out[(size_t)y * Wd + x] = v;
  if (quantized) quantized[(size_t)y * Wd + x] = (mask && mask[(size_t)y * Wd + x] == 0) ? 0 : v;
}
