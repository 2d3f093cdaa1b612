// Fused training loss (SURVEY 8f row N2): gau_loss = (1-l) mean|img - gt| + l (1 - mean SSIM),
// replacing the reference's five depthwise 11x11 F.conv2d + elementwise chain and its autograd
// backward (gsplat/pytorch_ssim.py:26-67) with two HBM-bound kernels:
//   k_ssim_fwd : separable 11-tap Gaussian (sigma 1.5, zero padding) of img, gt, img^2, gt^2,
//                img*gt in shared memory -> SSIM map, L1 and SSIM sums (one double atomicAdd
//                per CTA), and the three partial-derivative maps dSSIM/d{mu1, E11, E12};
//   k_ssim_bwd : the same separable filter over the three maps, combined with img / gt and the
//                L1 sign into dloss/dimg -- exactly what loss.backward() hands to splatB --
//                and the final loss scalar.
// Algorithmic bytes: 24 (read img, gt) + 36 (write maps) + 36 + 24 (read) + 12 (write grad)
// = 132 B per pixel (x3 channels already counted) -> HBM roofline.
#include "common.cuh"
#include "kernels.h"

#ifndef GSB_LOSS_FWD_MINB  // resident CTAs (of 4 warps) the row kernels are compiled for
#define GSB_LOSS_FWD_MINB 4
#endif
#ifndef GSB_LOSS_BWD_MINB
#define GSB_LOSS_BWD_MINB 4
#endif

namespace gsb {

constexpr int LW = 32, LH = 16, LR = 5;              // output tile, filter radius
constexpr int LIW = LW + 2 * LR, LIH = LH + 2 * LR;  // 42 x 26 input region
struct Win11 { float w[11]; };

__global__ void __launch_bounds__(256) k_ssim_fwd(int W, int H, const float *__restrict__ img,
                                                  const float *__restrict__ gt, Win11 win,
                                                  float *__restrict__ maps /* [3 maps][3][H][W] */,
                                                  double *__restrict__ acc /* [l1 sum, ssim sum] */) {
  __shared__ float s1[LIH][LIW + 1], s2[LIH][LIW + 1];
  __shared__ float hs[5][LIH][LW + 1];
  __shared__ float red[2][8];
  const int tid = threadIdx.x;
  const int x0 = blockIdx.x * LW, y0 = blockIdx.y * LH, c = blockIdx.z;
  const size_t HW = (size_t)H * W;
  const float *a = img + (size_t)c * HW, *b = gt + (size_t)c * HW;
  for (int i = tid; i < LIH * LIW; i += 256) {
    const int r = i / LIW, q = i % LIW;
    const int y = y0 + r - LR, x = x0 + q - LR;
    const bool in = (x >= 0) && (x < W) && (y >= 0) && (y < H);
    s1[r][q] = in ? __ldg(a + (size_t)y * W + x) : 0.f;
    s2[r][q] = in ? __ldg(b + (size_t)y * W + x) : 0.f;
  }
  __syncthreads();
  // horizontal pass, register blocked: one thread = 4 consecutive outputs of a row, so the 14
  // inputs they share are read from shared memory once (the kernel is LDS-bound otherwise)
  for (int i = tid; i < LIH * (LW / 4); i += 256) {
    const int r = i / (LW / 4), q0 = 4 * (i % (LW / 4));
    // (img, gt) travel as one f32x2: the five filtered quantities cost two FFMA2 + one FMUL2 +
    // one FFMA per tap instead of five FFMA + two FMUL (same IEEE operations, same results)
    float2 pg[14];
#pragma unroll
    for (int k = 0; k < 14; k++) pg[k] = make_float2(s1[r][q0 + k], s2[r][q0 + k]);
#pragma unroll
    for (int m = 0; m < 4; m++) {
      float2 mm = make_float2(0.f, 0.f), ee = make_float2(0.f, 0.f);
      float e12 = 0.f;
#pragma unroll
      for (int k = 0; k < 11; k++) {
        const float2 w2 = make_float2(win.w[k], win.w[k]), ab = pg[m + k];
        mm = __ffma2_rn(w2, ab, mm);            // (m1, m2) += w (a, b)
        const float2 wab = __fmul2_rn(w2, ab);  // (w a, w b)
        ee = __ffma2_rn(wab, ab, ee);           // (e11, e22) += (w a a, w b b)
        e12 = fmaf(wab.x, ab.y, e12);
      }
      hs[0][r][q0 + m] = mm.x; hs[1][r][q0 + m] = mm.y; hs[2][r][q0 + m] = ee.x; hs[3][r][q0 + m] = ee.y;
      hs[4][r][q0 + m] = e12;
    }
  }
  __syncthreads();
  const float C1 = 0.01f * 0.01f, C2 = 0.03f * 0.03f;
  float l1 = 0.f, ss = 0.f;
  // vertical pass, register blocked: one thread = 2 consecutive rows of a column
  for (int i = tid; i < (LH / 2) * LW; i += 256) {
    const int r0 = 2 * (i / LW), q = i % LW;
    const int x = x0 + q;
    float2 c01[12], c23[12];
    float c4[12];
#pragma unroll
    for (int k = 0; k < 12; k++) {
      c01[k] = make_float2(hs[0][r0 + k][q], hs[1][r0 + k][q]);
      c23[k] = make_float2(hs[2][r0 + k][q], hs[3][r0 + k][q]);
      c4[k] = hs[4][r0 + k][q];
    }
#pragma unroll
    for (int m = 0; m < 2; m++) {
      const int r = r0 + m, y = y0 + r;
      if (x >= W || y >= H) continue;
      float2 v01 = make_float2(0.f, 0.f), v23 = make_float2(0.f, 0.f);
      float v4 = 0.f;
#pragma unroll
      for (int k = 0; k < 11; k++) {
        const float2 w2 = make_float2(win.w[k], win.w[k]);
        v01 = __ffma2_rn(w2, c01[m + k], v01);
        v23 = __ffma2_rn(w2, c23[m + k], v23);
        v4 = fmaf(win.w[k], c4[m + k], v4);
      }
      const float mu1 = v01.x, mu2 = v01.y;
      const float s11 = v23.x - mu1 * mu1, s22 = v23.y - mu2 * mu2, s12 = v4 - mu1 * mu2;
      const float A1 = 2.f * mu1 * mu2 + C1, A2 = 2.f * s12 + C2;
      const float B1 = mu1 * mu1 + mu2 * mu2 + C1, B2 = s11 + s22 + C2;
      const float inv = 1.0f / (B1 * B2);
      const float ssim = A1 * A2 * inv;
      ss += ssim;
      l1 += fabsf(s1[r + LR][q + LR] - s2[r + LR][q + LR]);
      const size_t o = (size_t)c * HW + (size_t)y * W + x;
      maps[o] = (2.f * mu2 * (A2 - A1)) * inv - ssim * (2.f * mu1 * (B2 - B1)) * inv;  // dSSIM/dmu1
      maps[3 * HW + o] = -ssim / B2;                                                    // dSSIM/dE11
      maps[6 * HW + o] = 2.f * A1 * inv;                                                // dSSIM/dE12
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    l1 += __shfl_xor_sync(0xffffffffu, l1, o);
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
  }
  if ((tid & 31) == 0) { red[0][tid >> 5] = l1; red[1][tid >> 5] = ss; }
  __syncthreads();
  if (tid == 0) {
    double a0 = 0.0, a1 = 0.0;
#pragma unroll
    for (int w = 0; w < 8; w++) { a0 += (double)red[0][w]; a1 += (double)red[1][w]; }
    atomicAdd(acc + 0, a0);
    atomicAdd(acc + 1, a1);
  }
}

__global__ void __launch_bounds__(256) k_ssim_bwd(int W, int H, const float *__restrict__ img,
                                                  const float *__restrict__ gt, Win11 win,
                                                  const float *__restrict__ maps, const double *__restrict__ acc,
                                                  float lambda, float *__restrict__ loss_out,
                                                  float *__restrict__ grad /* [3,H,W] or nullptr */) {
  __shared__ float sm[3][LIH][LIW + 1];
  __shared__ float hs[3][LIH][LW + 1];
  const int tid = threadIdx.x;
  const int x0 = blockIdx.x * LW, y0 = blockIdx.y * LH, c = blockIdx.z;
  const size_t HW = (size_t)H * W;
  const double n = 3.0 * (double)HW;
  if (blockIdx.x == 0 && blockIdx.y == 0 && c == 0 && tid == 0)
    *loss_out = (float)((1.0 - (double)lambda) * (acc[0] / n) + (double)lambda * (1.0 - acc[1] / n));
  if (grad == nullptr) return;
  for (int i = tid; i < LIH * LIW; i += 256) {
    const int r = i / LIW, q = i % LIW;
    const int y = y0 + r - LR, x = x0 + q - LR;
    const bool in = (x >= 0) && (x < W) && (y >= 0) && (y < H);
    const size_t o = (size_t)c * HW + (size_t)(in ? y : 0) * W + (in ? x : 0);
#pragma unroll
    for (int m = 0; m < 3; m++) sm[m][r][q] = in ? __ldg(maps + 3 * m * HW + o) : 0.f;
  }
  __syncthreads();
  for (int i = tid; i < LIH * (LW / 4); i += 256) {  // 4 outputs per thread (see k_ssim_fwd)
    const int r = i / (LW / 4), q0 = 4 * (i % (LW / 4));
    float2 in01[14];
    float in2[14];
#pragma unroll
    for (int k = 0; k < 14; k++) {
      in01[k] = make_float2(sm[0][r][q0 + k], sm[1][r][q0 + k]);
      in2[k] = sm[2][r][q0 + k];
    }
#pragma unroll
    for (int t = 0; t < 4; t++) {
      float2 v01 = make_float2(0.f, 0.f);
      float v2 = 0.f;
#pragma unroll
      for (int k = 0; k < 11; k++) {
        v01 = __ffma2_rn(make_float2(win.w[k], win.w[k]), in01[t + k], v01);
        v2 = fmaf(win.w[k], in2[t + k], v2);
      }
      hs[0][r][q0 + t] = v01.x; hs[1][r][q0 + t] = v01.y; hs[2][r][q0 + t] = v2;
    }
  }
  __syncthreads();
  const float inv_n = (float)(1.0 / n);
  for (int i = tid; i < (LH / 2) * LW; i += 256) {  // 2 rows per thread
    const int r0 = 2 * (i / LW), q = i % LW;
    const int x = x0 + q;
    float2 col01[12];
    float col2[12];
#pragma unroll
    for (int k = 0; k < 12; k++) {
      col01[k] = make_float2(hs[0][r0 + k][q], hs[1][r0 + k][q]);
      col2[k] = hs[2][r0 + k][q];
    }
#pragma unroll
    for (int t = 0; t < 2; t++) {
      const int y = y0 + r0 + t;
      if (x >= W || y >= H) continue;
      float2 v01 = make_float2(0.f, 0.f);
      float v2 = 0.f;
#pragma unroll
      for (int k = 0; k < 11; k++) {
        v01 = __ffma2_rn(make_float2(win.w[k], win.w[k]), col01[t + k], v01);
        v2 = fmaf(win.w[k], col2[t + k], v2);
      }
      const float v[3] = {v01.x, v01.y, v2};
      const size_t o = (size_t)c * HW + (size_t)y * W + x;
      const float p = __ldg(img + o), g = __ldg(gt + o);
      const float sgn = (p > g) ? 1.f : ((p < g) ? -1.f : 0.f);
      grad[o] = (1.f - lambda) * sgn * inv_n - lambda * inv_n * (v[0] + 2.f * p * v[1] + g * v[2]);
    }
  }
}

// ---------------------------------------------------------------------------------------
// Row streaming: k_ssim_fwd_rows / k_ssim_bwd_rows, the path for every image below 2^31 / 9
// pixels (they use 32-bit element offsets; larger images take the tiled kernels above).  The
// tiled kernels spend 70 % of their instructions on staging (index arithmetic, shared-memory
// traffic for both passes); here one lane owns one image COLUMN and walks down a strip of rows:
//   * a row of img and gt goes through a 48-column per-warp shared-memory line (the warp's 32
//     columns + 8 either side, so that with W % 4 == 0 the line is 12 aligned float4 per image:
//     ONE 16-byte load per lane and row); 22 LDS feed the 11 horizontal taps;
//   * the vertical pass never touches shared memory: the last 11 horizontally filtered rows
//     live in registers (the row loop is unrolled so that the ring is statically indexed).
// ~215 instructions per (pixel, channel) instead of ~500 (ncu: 42 M + 35 M warp instructions at
// 1080p against 98 M + 66 M), same IEEE operations in the same order as the tiled kernels
// (bit-identical maps and gradient).  Warps are independent (one __syncwarp per row, no block
// barrier); the loads of the next two rows are in flight while the current row is filtered.
constexpr int SWARPS = 4;  // warps per CTA, side by side: 128 columns
constexpr int SLINE = 48;  // columns x0-8 .. x0+39 of a warp whose first column is x0
constexpr int SPAD = 8;

// The ring of horizontally filtered rows has 12 slots (11 live): the row loop is unrolled by 12,
// an EVEN count, so that besides the ring slots the parity of the row (line buffer, register
// set of the rows in flight) is static in every unrolled copy.
constexpr int RING = 12;
__device__ __forceinline__ int ring_slot(int i, int k) { return (i + 2 + k) % RING; }  // row t - 10 + k, t % 12 == i

// One row of NIMG images into the warp's lines.  VEC: lane l < 12 * NIMG loads chunk l % 12 of image
// l / 12 (a second round covers NIMG = 3); otherwise every lane loads columns lane and lane + 32.
template <int NIMG, bool VEC>
struct RowFetch {
  static constexpr int ROUNDS = VEC ? (12 * NIMG + 31) / 32 : 1;
  const float *src[VEC ? ROUNDS : 2 * NIMG];  // per-lane source pointers at row 0 (column folded in)
  float *dst[VEC ? ROUNDS : 2 * NIMG];        // per-lane destinations in line buffer 0
  bool ok[VEC ? ROUNDS : 2 * NIMG];
  struct Row {  // one row in flight
    float4 v4[VEC ? ROUNDS : 1];
    float v1[VEC ? 1 : 2 * NIMG];
  };

  // img0..2: row 0 of the (up to three) planes; line: this warp's [NIMG][2][SLINE] buffers
  __device__ __forceinline__ void init(int lane, int x0, int W, const float *img0, const float *img1,
                                       const float *img2, float (*line)[2][SLINE]) {
    if constexpr (VEC) {
#pragma unroll
      for (int r = 0; r < ROUNDS; r++) {
        const int q = lane + 32 * r, im = q / 12, ch = q - 12 * im, col = x0 - SPAD + 4 * ch;
        ok[r] = q < 12 * NIMG && col >= 0 && col < W;
        const int imc = im < NIMG ? im : 0;
        src[r] = (imc == 0 ? img0 : (imc == 1 ? img1 : img2)) + col;
        dst[r] = &line[imc][0][4 * ch];
      }
    } else {
#pragma unroll
      for (int m = 0; m < NIMG; m++)
#pragma unroll
        for (int h = 0; h < 2; h++) {
          const int j = lane + 32 * h, col = x0 - SPAD + j;
          ok[2 * m + h] = j < SLINE && col >= 0 && col < W;
          src[2 * m + h] = (m == 0 ? img0 : (m == 1 ? img1 : img2)) + col;
          dst[2 * m + h] = &line[m][0][j < SLINE ? j : 0];
        }
    }
  }
  __device__ __forceinline__ Row fetch(int yy, int W, int H) const {
    Row row;
    const bool yin = yy >= 0 && yy < H;
    const int o = yy * W;
    if constexpr (VEC) {
#pragma unroll
      for (int r = 0; r < ROUNDS; r++) {
        row.v4[r] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (yin && ok[r]) row.v4[r] = __ldg(reinterpret_cast<const float4 *>(src[r] + o));
      }
    } else {
#pragma unroll
      for (int e = 0; e < 2 * NIMG; e++) {
        row.v1[e] = 0.f;
        if (yin && ok[e]) row.v1[e] = __ldg(src[e] + o);
      }
    }
    return row;
  }
  __device__ __forceinline__ void stage(int buf, int lane, const Row &row) const {  // buf: 0 / 1
    const int off = buf * SLINE;
    if constexpr (VEC) {
#pragma unroll
      for (int r = 0; r < ROUNDS; r++)
        if (lane + 32 * r < 12 * NIMG) *reinterpret_cast<float4 *>(dst[r] + off) = row.v4[r];
    } else {
#pragma unroll
      for (int e = 0; e < 2 * NIMG; e++)
        if ((e & 1) == 0 || lane + 32 < SLINE) dst[e][off] = row.v1[e];
    }
  }
};

template <bool VEC>
__global__ void __launch_bounds__(32 * SWARPS, GSB_LOSS_FWD_MINB) k_ssim_fwd_rows(int W, int H, int SH, const float *__restrict__ img,
                                                                  const float *__restrict__ gt, Win11 win,
                                                                  float *__restrict__ maps,
                                                                  double *__restrict__ acc) {
  __shared__ __align__(16) float line[SWARPS][2][2][SLINE];  // [warp][img | gt][buffer][column]
  __shared__ float red[2][SWARPS];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int x0 = (blockIdx.x * SWARPS + wid) * 32, x = x0 + lane;
  const int yb = blockIdx.y * SH, ye = min(yb + SH, H), c = blockIdx.z;
  const int HW = H * W;  // (the host takes this kernel only for H * W < 2^31 / 9)
  float *__restrict__ mp0 = maps + (size_t)c * HW, *__restrict__ mp1 = mp0 + (size_t)3 * HW,
                      *__restrict__ mp2 = mp0 + (size_t)6 * HW;
  const bool xin = x < W;
  const int n = ye - yb + 2 * LR;  // input rows yb-5 .. ye+4
  float l1 = 0.f, ss = 0.f;
  const float C1 = 0.01f * 0.01f, C2 = 0.03f * 0.03f;
  if (x0 < W) {  // (whole warps beyond the right edge only take part in the final reduction)
    RowFetch<2, VEC> rf;
    rf.init(lane, x0, W, img + (size_t)c * HW, gt + (size_t)c * HW, nullptr, line[wid]);
    float2 r01[RING], r23[RING];
    float r4[RING];
    // Software pipeline over rows: row t is filtered out of line buffer t & 1 while row t + 1
    // (loaded two iterations ago) is stored into the other buffer and the load of row t + 3 is
    // issued into the register set that just emptied: two rows are in flight per lane, a load
    // has ~1.7 iterations (~400 instructions) to arrive.  (One row ahead left 60-110 instructions: 68 % of the backward kernel's warp
    // time was spent waiting for it, profiles/r2_ncu_loss_density_summary.txt.)
    rf.stage(0, lane, rf.fetch(yb - LR, W, H));
    __syncwarp();
    typename RowFetch<2, VEC>::Row rows[2];  // row r in flight lives in rows[r & 1]
    rows[1] = rf.fetch(yb - LR + 1, W, H);
    rows[0] = rf.fetch(yb - LR + 2, W, H);
    for (int t0 = 0; t0 < n; t0 += RING) {
#pragma unroll
      for (int i = 0; i < RING; i++) {
        const int t = t0 + i;
        if (t < n) {
          const int yy = yb - LR + t;
          rf.stage((i + 1) & 1, lane, rows[(i + 1) & 1]);  // row t + 1 (past the strip's last input row: never used)
          rows[(i + 1) & 1] = rf.fetch(yy + 3, W, H);
          const float *ra = &line[wid][0][i & 1][lane + SPAD - LR], *rb = &line[wid][1][i & 1][lane + SPAD - LR];
          float2 mm = make_float2(0.f, 0.f), ee = make_float2(0.f, 0.f);
          float e12 = 0.f;
#pragma unroll
          for (int k = 0; k < 11; k++) {
            const float2 w2 = make_float2(win.w[k], win.w[k]), ab = make_float2(ra[k], rb[k]);
            if (k == LR && t >= LR && t < n - LR) l1 += fabsf(ab.x - ab.y);  // the strip's own rows
            mm = __ffma2_rn(w2, ab, mm);
            const float2 wab = __fmul2_rn(w2, ab);
            ee = __ffma2_rn(wab, ab, ee);
            e12 = fmaf(wab.x, ab.y, e12);
          }
          r01[i] = mm, r23[i] = ee, r4[i] = e12;
          if (t >= 2 * LR && xin) {  // output row yy - 5 = yb + t - 10: its 11 rows are in the ring
            float2 v01 = make_float2(0.f, 0.f), v23 = make_float2(0.f, 0.f);
            float v4 = 0.f;
#pragma unroll
            for (int k = 0; k < 11; k++) {
              const float2 w2 = make_float2(win.w[k], win.w[k]);
              v01 = __ffma2_rn(w2, r01[ring_slot(i, k)], v01);
              v23 = __ffma2_rn(w2, r23[ring_slot(i, k)], v23);
              v4 = fmaf(win.w[k], r4[ring_slot(i, k)], v4);
            }
            const float mu1 = v01.x, mu2 = v01.y;
            const float s11 = v23.x - mu1 * mu1, s22 = v23.y - mu2 * mu2, s12 = v4 - mu1 * mu2;
            const float A1 = 2.f * mu1 * mu2 + C1, A2 = 2.f * s12 + C2;
            const float B1 = mu1 * mu1 + mu2 * mu2 + C1, B2 = s11 + s22 + C2;
            const float inv = 1.0f / (B1 * B2);
            const float ssim = A1 * A2 * inv;
            ss += ssim;
            const int o = (yy - LR) * W + x;
            mp0[o] = (2.f * mu2 * (A2 - A1)) * inv - ssim * (2.f * mu1 * (B2 - B1)) * inv;  // dSSIM/dmu1
            mp1[o] = -ssim / B2;                                                            // dSSIM/dE11
            mp2[o] = 2.f * A1 * inv;                                                        // dSSIM/dE12
          }
          __syncwarp();
        }
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    l1 += __shfl_xor_sync(0xffffffffu, l1, o);
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
  }
  if (lane == 0) { red[0][wid] = l1; red[1][wid] = ss; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a0 = 0.0, a1 = 0.0;
#pragma unroll
    for (int w = 0; w < SWARPS; w++) { a0 += (double)red[0][w]; a1 += (double)red[1][w]; }
    atomicAdd(acc + 0, a0);
    atomicAdd(acc + 1, a1);
  }
}

template <bool VEC>
__global__ void __launch_bounds__(32 * SWARPS, GSB_LOSS_BWD_MINB) k_ssim_bwd_rows(int W, int H, int SH, const float *__restrict__ img,
                                                                  const float *__restrict__ gt, Win11 win,
                                                                  const float *__restrict__ maps,
                                                                  const double *__restrict__ acc, float lambda,
                                                                  float *__restrict__ loss_out,
                                                                  float *__restrict__ grad) {
  __shared__ __align__(16) float line[SWARPS][3][2][SLINE];  // [warp][map][buffer][column]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int x0 = (blockIdx.x * SWARPS + wid) * 32, x = x0 + lane;
  const int yb = blockIdx.y * SH, ye = min(yb + SH, H), c = blockIdx.z;
  const int HW = H * W;
  const double npix = 3.0 * (double)HW;
  if (blockIdx.x == 0 && blockIdx.y == 0 && c == 0 && threadIdx.x == 0)
    *loss_out = (float)((1.0 - (double)lambda) * (acc[0] / npix) + (double)lambda * (1.0 - acc[1] / npix));
  if (grad == nullptr || x0 >= W) return;
  const float *__restrict__ a = img + (size_t)c * HW, *__restrict__ b = gt + (size_t)c * HW;
  float *__restrict__ gr = grad + (size_t)c * HW;
  // (the maps are zero outside the image: conv2d's zero padding, transposed)
  RowFetch<3, VEC> rf;
  rf.init(lane, x0, W, maps + (size_t)c * HW, maps + (size_t)(3 + c) * HW, maps + (size_t)(6 + c) * HW, line[wid]);
  const bool xin = x < W;
  const int n = ye - yb + 2 * LR;
  const float inv_n = (float)(1.0 / npix);
  float2 r01[RING];
  float r2[RING];
  rf.stage(0, lane, rf.fetch(yb - LR, W, H));  // (software pipeline over rows: see k_ssim_fwd_rows)
  __syncwarp();
  typename RowFetch<3, VEC>::Row rows[2];
  rows[1] = rf.fetch(yb - LR + 1, W, H);
  rows[0] = rf.fetch(yb - LR + 2, W, H);
  float pq[2] = {0.f, 0.f}, gq[2] = {0.f, 0.f};  // img / gt of the output pixel of iteration t in [t & 1]
  for (int t0 = 0; t0 < n; t0 += RING) {
#pragma unroll
    for (int i = 0; i < RING; i++) {
      const int t = t0 + i;
      if (t < n) {
        const int yy = yb - LR + t;
        rf.stage((i + 1) & 1, lane, rows[(i + 1) & 1]);
        rows[(i + 1) & 1] = rf.fetch(yy + 3, W, H);
        const bool emit = t >= 2 * LR && xin;
        const int o = (yy - LR) * W + x;
        const float p = pq[i & 1], g = gq[i & 1];
        if (t + 2 >= 2 * LR && t + 2 < n && xin) pq[i & 1] = __ldg(a + o + 2 * W), gq[i & 1] = __ldg(b + o + 2 * W);
        const float *q0 = &line[wid][0][i & 1][lane + SPAD - LR], *q1 = &line[wid][1][i & 1][lane + SPAD - LR],
                    *q2 = &line[wid][2][i & 1][lane + SPAD - LR];
        float2 h01 = make_float2(0.f, 0.f);
        float h2 = 0.f;
#pragma unroll
        for (int k = 0; k < 11; k++) {
          h01 = __ffma2_rn(make_float2(win.w[k], win.w[k]), make_float2(q0[k], q1[k]), h01);
          h2 = fmaf(win.w[k], q2[k], h2);
        }
        r01[i] = h01, r2[i] = h2;
        if (emit) {
          float2 v01 = make_float2(0.f, 0.f);
          float v2 = 0.f;
#pragma unroll
          for (int k = 0; k < 11; k++) {
            v01 = __ffma2_rn(make_float2(win.w[k], win.w[k]), r01[ring_slot(i, k)], v01);
            v2 = fmaf(win.w[k], r2[ring_slot(i, k)], v2);
          }
          const float sgn = (p > g) ? 1.f : ((p < g) ? -1.f : 0.f);
          gr[o] = (1.f - lambda) * sgn * inv_n - lambda * inv_n * (v01.x + 2.f * p * v01.y + g * v2);
        }
        __syncwarp();
      }
    }
  }
}

// rows per strip: about one resident wave of warps (a strip pays 10 halo rows, so the longer the
// better, but every SM needs its share)
static int strip_rows(int H, int W) {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int xblocks = (W + 32 * SWARPS - 1) / (32 * SWARPS);
  const int ctas_wanted = sms * 4;  // 4 CTAs of 4 warps per SM at ~110 registers
  int strips = ctas_wanted / (3 * xblocks);
  if (strips < 1) strips = 1;
  int sh = (H + strips - 1) / strips;
  return sh < 16 ? 16 : sh;
}

size_t gau_loss_workspace_bytes(int H, int W) {
  return 256 + (size_t)9 * H * W * sizeof(float);  // [2 doubles, padded] [3 maps x 3 channels]
}

int launch_gau_loss(int H, int W, const float *img, const float *gt, float lambda, float *loss_out,
                    float *grad, void *ws, cudaStream_t st) {
  if (H <= 0 || W <= 0) return set_arg_error("gau_loss: bad image size");
  Win11 win;
  {  // gsplat/pytorch_ssim.py:12-15: float32 taps, float32 normalisation
    float s = 0.f;
    for (int x = 0; x < 11; x++) {
      win.w[x] = (float)exp(-(double)((x - 5) * (x - 5)) / (2.0 * 1.5 * 1.5));
      s += win.w[x];
    }
    for (int x = 0; x < 11; x++) win.w[x] /= s;
  }
  double *acc = static_cast<double *>(ws);
  float *maps = reinterpret_cast<float *>(static_cast<char *>(ws) + 256);
  GSB_CUDA_TRY(cudaMemsetAsync(acc, 0, 2 * sizeof(double), st));
  // the row kernels address the maps with 32-bit offsets; larger images take the tiled kernels
  if ((long long)H * W < (1ll << 31) / 9) {
    const int SH = strip_rows(H, W);
    const dim3 grid((W + 32 * SWARPS - 1) / (32 * SWARPS), (H + SH - 1) / SH, 3);
    // 16-byte row loads need every row (and plane) of all five arrays 16-byte aligned
    const bool vec = W % 4 == 0 && ((reinterpret_cast<uintptr_t>(img) | reinterpret_cast<uintptr_t>(gt) |
                                     reinterpret_cast<uintptr_t>(maps)) & 15) == 0;
    {
      ProfScope ps(K_LOSS_FWD, st);
      if (vec)
        k_ssim_fwd_rows<true><<<grid, 32 * SWARPS, 0, st>>>(W, H, SH, img, gt, win, maps, acc);
      else
        k_ssim_fwd_rows<false><<<grid, 32 * SWARPS, 0, st>>>(W, H, SH, img, gt, win, maps, acc);
    }
    GSB_CUDA_TRY(cudaGetLastError());
    {
      ProfScope ps(K_LOSS_BWD, st);
      if (vec)
        k_ssim_bwd_rows<true><<<grid, 32 * SWARPS, 0, st>>>(W, H, SH, img, gt, win, maps, acc, lambda, loss_out, grad);
      else
        k_ssim_bwd_rows<false><<<grid, 32 * SWARPS, 0, st>>>(W, H, SH, img, gt, win, maps, acc, lambda, loss_out, grad);
    }
    GSB_CUDA_TRY(cudaGetLastError());
    return 0;
  }
  const dim3 grid((W + LW - 1) / LW, (H + LH - 1) / LH, 3);
  {
    ProfScope ps(K_LOSS_FWD, st);
    k_ssim_fwd<<<grid, 256, 0, st>>>(W, H, img, gt, win, maps, acc);
  }
  GSB_CUDA_TRY(cudaGetLastError());
  {
    ProfScope ps(K_LOSS_BWD, st);
    k_ssim_bwd<<<grid, 256, 0, st>>>(W, H, img, gt, win, maps, acc, lambda, loss_out, grad);
  }
  GSB_CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // namespace gsb
