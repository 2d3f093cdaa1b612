// Density control (prune / clone / split with the Adam moments carried along) and Gaussian
// record conversion (PLY rows <-> .npy rows <-> the six training tensors).  SURVEY 8f row N3.
//
// Reference: gsplat/gsmodel.py:132-166 (update_params / prune_params), :219-234
// (update_density_info), :236-318 (update_gaussian_density), :320-331 (reset_alpha);
// gsplat/gau_io.py:60-107 (load_ply), :138-153 (save_training_params); gsmodel.py:95-113
// (get_training_params).
//
// The reference rebuilds all 18 tensors (6 parameters + exp_avg + exp_avg_sq) with boolean
// indexing and torch.cat, one tensor at a time, plus ~20 temporaries.  Here it is three
// streaming passes: classify (one byte per Gaussian) + per-CTA counts, a two-kernel exclusive
// scan of the three class counters (the output slot of every survivor / clone / split), and one
// apply kernel that moves every surviving row once and writes the new rows at the tail.  All of it is HBM-bound:
// algorithmic bytes = 24 N (classify + scan) + 2 * 708 * K + 708 * (C + S) for the full state
// (59 floats x 3 sets = 708 B per Gaussian).
//
// Transcendentals are the accurate expf / logf / sqrtf / IEEE division (no fast-math here):
// torch's CUDA kernels use the same libdevice routines, which keeps the clone / split values
// within an ulp of the reference's.
#include "common.cuh"
#include "kernels.h"

namespace gsb {

namespace {

constexpr int kWidth[6] = {3, 3, 45, 1, 3, 4};  // pws, low_shs, high_shs, alphas_raw, scales_raw, rots_raw
enum : uint8_t { CLS_KEEP = 0, CLS_CLONE = 1, CLS_SPLIT = 2, CLS_PRUNE = 3 };

struct Slot3 {  // exclusive counts of survivors / clones / splits before this Gaussian
  int k, c, s;
};
// gsmodel.py:219-234.  init != 0 is the first call after a density update: the norm of every
// Gaussian is stored and the counter starts from the mask (:228-229).
__global__ void k_density_accumulate(int64_t N, const float2 *__restrict__ dus, const uint8_t *__restrict__ mask,
                                     float *__restrict__ acc, int32_t *__restrict__ cnt, int init) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const float2 d = dus[i];
  const float g = sqrtf(d.x * d.x + d.y * d.y);
  const bool m = mask[i] != 0;
  if (init) {
    acc[i] = g;
    cnt[i] = m;
  } else if (m) {
    acc[i] += g;
    cnt[i] += 1;
  }
}

// gsmodel.py:238-262
__device__ __forceinline__ uint8_t classify_row(int64_t i, const float *__restrict__ alphas_raw,
                                                const float *__restrict__ scales_raw, const float *__restrict__ acc,
                                                const int32_t *__restrict__ cnt, float alpha_raw_min,
                                                float scale_raw_max, float grad_min, float scale_clone_max) {
  const float a = alphas_raw[i];
  const float s0 = scales_raw[3 * i], s1 = scales_raw[3 * i + 1], s2 = scales_raw[3 * i + 2];
  const float smax = fmaxf(s0, fmaxf(s1, s2));
  uint8_t c;
  if (a < alpha_raw_min || smax > scale_raw_max) {
    c = CLS_PRUNE;
  } else {
    float g = acc[i] / (float)cnt[i];
    if (isnan(g)) g = 0.f;
    // max over exp(s) (the reference compares the activated scales, :257)
    const float big = fmaxf(expf(s0), fmaxf(expf(s1), expf(s2)));
    c = g >= grad_min ? (big <= scale_clone_max ? CLS_CLONE : CLS_SPLIT) : CLS_KEEP;
  }
  return c;
}

// ---- the slots (exclusive scan of the three class counters in row order), hand-written:
//   k_density_classify_count  classify 1024 rows per CTA and leave the CTA's three counts;
//   k_density_scan_blocks     one CTA turns the per-CTA counts into exclusive offsets + totals;
//   k_density_slots           every CTA re-reads its 1024 class bytes (4 consecutive rows per
//                             thread), scans them locally and writes the 12-byte slots.
// 25 B per Gaussian in total; three launches (round 1 used a library scan over the 12-byte struct: 0.034 ms against 0.023).
constexpr int SC_THREADS = 256, SC_PER = 4, SC_ROWS = SC_THREADS * SC_PER;

__global__ void __launch_bounds__(SC_THREADS) k_density_classify_count(
    int64_t N, const float *__restrict__ alphas_raw, const float *__restrict__ scales_raw,
    const float *__restrict__ acc, const int32_t *__restrict__ cnt, float alpha_raw_min, float scale_raw_max,
    float grad_min, float scale_clone_max, uint8_t *__restrict__ cls, int32_t *__restrict__ block_counts) {
  __shared__ uint32_t red[2][SC_THREADS / 32];
  uint32_t kc = 0, sp = 0;  // (survivors | clones << 16), splits: at most SC_ROWS each per CTA
#pragma unroll
  for (int j = 0; j < SC_PER; j++) {
    const int64_t i = (int64_t)blockIdx.x * SC_ROWS + j * SC_THREADS + threadIdx.x;
    if (i < N) {
      const uint8_t c =
          classify_row(i, alphas_raw, scales_raw, acc, cnt, alpha_raw_min, scale_raw_max, grad_min, scale_clone_max);
      cls[i] = c;
      kc += (c != CLS_PRUNE) + ((uint32_t)(c == CLS_CLONE) << 16);
      sp += c == CLS_SPLIT;
    }
  }
  kc = __reduce_add_sync(0xffffffffu, kc);
  sp = __reduce_add_sync(0xffffffffu, sp);
  if ((threadIdx.x & 31) == 0) red[0][threadIdx.x >> 5] = kc, red[1][threadIdx.x >> 5] = sp;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t a = 0, b = 0;
#pragma unroll
    for (int w = 0; w < SC_THREADS / 32; w++) a += red[0][w], b += red[1][w];
    block_counts[3 * blockIdx.x + 0] = (int32_t)(a & 0xffffu);
    block_counts[3 * blockIdx.x + 1] = (int32_t)(a >> 16);
    block_counts[3 * blockIdx.x + 2] = (int32_t)b;
  }
}

// in place: block_counts[b] -> the counts before CTA b; totals = the three sums
__global__ void __launch_bounds__(1024) k_density_scan_blocks(int nb, int32_t *__restrict__ block_counts,
                                                              int64_t *__restrict__ totals) {
  __shared__ int warp_tot[3][32];
  __shared__ int carry[3];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x < 3) carry[threadIdx.x] = 0;
  __syncthreads();
  for (int base = 0; base < nb; base += 1024) {
    const int b = base + threadIdx.x;
    int v[3] = {0, 0, 0}, inc[3];
    if (b < nb) v[0] = block_counts[3 * b], v[1] = block_counts[3 * b + 1], v[2] = block_counts[3 * b + 2];
#pragma unroll
    for (int q = 0; q < 3; q++) {
      int x = v[q];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
      }
      inc[q] = x;
      if (lane == 31) warp_tot[q][wid] = x;
    }
    __syncthreads();
    int c0[3];
#pragma unroll
    for (int q = 0; q < 3; q++) {
      int before = carry[q];
      for (int w = 0; w < wid; w++) before += warp_tot[q][w];
      c0[q] = before + inc[q] - v[q];
    }
    if (b < nb) block_counts[3 * b] = c0[0], block_counts[3 * b + 1] = c0[1], block_counts[3 * b + 2] = c0[2];
    __syncthreads();
    if (threadIdx.x == 1023) {
#pragma unroll
      for (int q = 0; q < 3; q++) carry[q] = c0[q] + v[q];
    }
    __syncthreads();
  }
  if (threadIdx.x < 3) totals[threadIdx.x] = carry[threadIdx.x];
}

__global__ void __launch_bounds__(SC_THREADS) k_density_slots(int64_t N, const uint8_t *__restrict__ cls,
                                                              const int32_t *__restrict__ block_offsets,
                                                              Slot3 *__restrict__ slots) {
  __shared__ uint32_t warp_tot[2][SC_THREADS / 32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t row0 = (int64_t)blockIdx.x * SC_ROWS + (int64_t)threadIdx.x * SC_PER;
  uint8_t c[SC_PER];
  uint32_t kc = 0, sp = 0;
#pragma unroll
  for (int j = 0; j < SC_PER; j++) {
    c[j] = row0 + j < N ? cls[row0 + j] : (uint8_t)CLS_PRUNE;
    kc += (c[j] != CLS_PRUNE) + ((uint32_t)(c[j] == CLS_CLONE) << 16);
    sp += c[j] == CLS_SPLIT;
  }
  uint32_t ikc = kc, isp = sp;  // inclusive over the warp
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t a = __shfl_up_sync(0xffffffffu, ikc, o), b = __shfl_up_sync(0xffffffffu, isp, o);
    if (lane >= o) ikc += a, isp += b;
  }
  if (lane == 31) warp_tot[0][wid] = ikc, warp_tot[1][wid] = isp;
  __syncthreads();
  uint32_t bkc = ikc - kc, bsp = isp - sp;  // exclusive within the CTA
  for (int w = 0; w < wid; w++) bkc += warp_tot[0][w], bsp += warp_tot[1][w];
  Slot3 run{block_offsets[3 * blockIdx.x] + (int)(bkc & 0xffffu), block_offsets[3 * blockIdx.x + 1] + (int)(bkc >> 16),
            block_offsets[3 * blockIdx.x + 2] + (int)bsp};
#pragma unroll
  for (int j = 0; j < SC_PER; j++) {
    if (row0 + j < N) slots[row0 + j] = run;
    run.k += c[j] != CLS_PRUNE, run.c += c[j] == CLS_CLONE, run.s += c[j] == CLS_SPLIT;
  }
}

struct Sets {
  const float *p[6], *m[6], *v[6];  // m / v entries may be null (no optimizer state yet)
  float *dp[6], *dm[6], *dv[6];
};

__device__ __forceinline__ float logit_of_sigmoid(float x) {
  const float a = 1.f / (1.f + expf(-x));  // get_alphas
  return logf(a / (1.f - a));              // get_alphas_raw
}

// utils.py:46-54 on the normalised quaternion, v = z * exp(scales_raw)
__device__ __forceinline__ float split_offset(const float *__restrict__ q4, const float *__restrict__ s3,
                                              const float *__restrict__ z3, int comp) {
  float w = q4[0], x = q4[1], y = q4[2], z = q4[3];
  float n = fmaxf(sqrtf(w * w + x * x + y * y + z * z), 1e-12f);  // get_rots
  w /= n, x /= n, y /= n, z /= n;
  n = fmaxf(sqrtf(w * w + x * x + y * y + z * z), 1e-12f);        // normalize() inside rotate_vector
  w /= n, x /= n, y /= n, z /= n;
  const float v0 = z3[0] * expf(s3[0]), v1 = z3[1] * expf(s3[1]), v2 = z3[2] * expf(s3[2]);
  const float uv = x * v0 + y * v1 + z * v2, uu = x * x + y * y + z * z;
  const float c0 = y * v2 - z * v1, c1 = z * v0 - x * v2, c2 = x * v1 - y * v0;
  const float u = comp == 0 ? x : (comp == 1 ? y : z);
  const float v = comp == 0 ? v0 : (comp == 1 ? v1 : v2);
  const float c = comp == 0 ? c0 : (comp == 1 ? c1 : c2);
  return 2.f * u * uv + v * (w * w - uu) + 2.f * c * w;
}

// One "job" per (tensor, set) pair -- 6 tensors x {parameter, exp_avg, exp_avg_sq} = 18 jobs on
// blockIdx.y, grid-stride over the job's N*w elements, four independent elements in flight
// per thread (loads first, then stores).  Survivors move to their compacted row; clones /
// splits additionally produce a new row at K + slot (clones) or K + C + slot (splits): the
// recomputed value for a parameter, zero for an Adam moment.  64-bit element indices: this
// kernel is the path for N >= 23 M, where N * 45 overflows 32 bits (k_density_apply_rows below).
template <int A, int SET>
__device__ __forceinline__ void apply_job(int64_t N, const uint8_t *__restrict__ cls, const Slot3 *__restrict__ slots,
                                          int64_t K, int64_t C, const Sets &S, const float *__restrict__ z) {
  constexpr int w = kWidth[A];
  constexpr int U = 4;
  const float *__restrict__ src = SET == 0 ? S.p[A] : (SET == 1 ? S.m[A] : S.v[A]);
  float *__restrict__ dst = SET == 0 ? S.dp[A] : (SET == 1 ? S.dm[A] : S.dv[A]);
  if (src == nullptr) return;
  const int64_t total = N * w;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e0 < total; e0 += stride * U) {
    int64_t row[U];
    uint8_t cl[U];
    float val[U];
    Slot3 sl[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int64_t e = e0 + (int64_t)u * stride;
      row[u] = e < total ? e / w : 0;
      cl[u] = e < total ? cls[row[u]] : (uint8_t)CLS_PRUNE;
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      if (cl[u] == CLS_PRUNE) continue;
      val[u] = src[e0 + (int64_t)u * stride];
      sl[u] = slots[row[u]];
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      if (cl[u] == CLS_PRUNE) continue;
      const int64_t i = row[u];
      const int c = (int)(e0 + (int64_t)u * stride - i * w);
      dst[(int64_t)sl[u].k * w + c] = val[u];
      if (cl[u] == CLS_KEEP) continue;
      const bool split = cl[u] == CLS_SPLIT;
      const int64_t r = (split ? K + C + (int64_t)sl[u].s : K + (int64_t)sl[u].c) * w + c;
      float nv = 0.f;
      if (SET == 0) {
        nv = val[u];
        if (A == 0) {
          if (split) nv += split_offset(S.p[5] + 4 * (int64_t)i, S.p[4] + 3 * (int64_t)i, z + 3 * (int64_t)sl[u].s, c);
        } else if (A == 3) {
          nv = logit_of_sigmoid(nv);
        } else if (A == 4) {
          const float s = expf(nv);               // get_scales
          nv = logf(split ? s * 0.6f : s);        // gsmodel.py:281 then get_scales_raw
        } else if (A == 5) {
          const float *q = src + 4 * (int64_t)i;
          nv = nv / fmaxf(sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]), 1e-12f);
        }
      }
      dst[r] = nv;
    }
  }
}

__global__ void __launch_bounds__(256) k_density_apply(int64_t N, const uint8_t *__restrict__ cls,
                                                       const Slot3 *__restrict__ slots, int64_t K, int64_t C, Sets S,
                                                       const float *__restrict__ z) {
#define GSB_JOB(a, s) \
  case 3 * a + s: apply_job<a, s>(N, cls, slots, K, C, S, z); break;
  switch (blockIdx.y) {
    GSB_JOB(0, 0) GSB_JOB(0, 1) GSB_JOB(0, 2) GSB_JOB(1, 0) GSB_JOB(1, 1) GSB_JOB(1, 2)
    GSB_JOB(2, 0) GSB_JOB(2, 1) GSB_JOB(2, 2) GSB_JOB(3, 0) GSB_JOB(3, 1) GSB_JOB(3, 2)
    GSB_JOB(4, 0) GSB_JOB(4, 1) GSB_JOB(4, 2) GSB_JOB(5, 0) GSB_JOB(5, 1) GSB_JOB(5, 2)
  }
#undef GSB_JOB
}

// ---- row groups (the path for N < 23 M): a warp moves 32 consecutive Gaussians of one array.
// The per-Gaussian plan (class, survivor slot, new-row slot) is read once per group into a
// 32-entry shared-memory table instead of once per element (13 B per 4-byte element in the
// kernel above).  Loads and stores are 4-byte but fully coalesced: lane l handles elements
// l, l + 32, ... of the group's contiguous source span, 8 loads in flight per lane for the wide
// arrays; consecutive survivors are consecutive in the destination too, so a store instruction
// writes whole 32-byte sectors.  (A first version read the span with float4 loads and wrote the
// four components with stride-16-byte stores: quarter-filled sectors, 0.57 ms against the 0.45 ms
// of the kernel above.)  Elements of pruned Gaussians are not loaded.
constexpr int DG_WARPS = 8;
constexpr int DG_PAIRS = 4;  // row pairs of a [*, 45] array in flight per lane (12 loads)

// the value a clone / split writes at its new row (parameters; Adam moments start at 0)
template <int A>
__device__ __forceinline__ float new_row_value(float val, bool split, int64_t i, int s, int c, const Sets &S,
                                               const float *__restrict__ z) {
  float nv = val;
  if (A == 0) {
    if (split) nv += split_offset(S.p[5] + 4 * i, S.p[4] + 3 * i, z + 3 * (int64_t)s, c);
  } else if (A == 3) {
    nv = logit_of_sigmoid(nv);
  } else if (A == 4) {
    const float e = expf(nv);          // get_scales
    nv = logf(split ? e * 0.6f : e);   // gsmodel.py:281 then get_scales_raw
  } else if (A == 5) {
    const float *q = S.p[5] + 4 * i;
    nv = nv / fmaxf(sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]), 1e-12f);
  }
  return nv;
}

template <int A, int SET>
__device__ __forceinline__ void rows_job(int row0, const int2 *__restrict__ tab, int K, int C, const Sets &S,
                                         const float *__restrict__ z, int lane) {
  constexpr int w = kWidth[A];
  const float *__restrict__ src = SET == 0 ? S.p[A] : (SET == 1 ? S.m[A] : S.v[A]);
  float *__restrict__ dst = SET == 0 ? S.dp[A] : (SET == 1 ? S.dm[A] : S.dv[A]);
  if (src == nullptr) return;
  const float *__restrict__ gsrc = src + (size_t)row0 * w;
  // element (row r of the group, column col) with plan entry `info`
  auto emit = [&](int r, int col, int2 info, float val) {
    const unsigned cl = (unsigned)info.x >> 30;
    if (cl == CLS_PRUNE) return;
    dst[(size_t)(info.x & 0x3fffffff) * w + col] = val;
    if (cl == CLS_KEEP) return;
    float nv = 0.f;
    if (SET == 0) nv = new_row_value<A>(val, cl == CLS_SPLIT, (int64_t)row0 + r, info.y - K - C, col, S, z);
    dst[(size_t)info.y * w + col] = nv;
  };
  // table entries of rows past the end of the array are CLS_PRUNE, so no row bound is checked;
  // destination element indices fit 32 bits (2 N * 45 < 2^32 for N < 23 M)
  constexpr bool plain = SET != 0 || A == 1 || A == 2;  // the new row is a copy (parameters) or zero (moments)
  auto emit_fixed = [&](int r, int col, int2 info, float val) {
    if constexpr (plain) {  // two predicated stores, no branches
      const unsigned cl = (unsigned)info.x >> 30;
      if (cl != CLS_PRUNE) dst[(unsigned)(info.x & 0x3fffffff) * w + col] = val;
      if (cl == CLS_CLONE || cl == CLS_SPLIT) dst[(unsigned)info.y * w + col] = SET == 0 ? val : 0.f;
    } else {
      emit(r, col, info, val);
    }
  };
  if constexpr (w == 45) {
    // Two rows = 90 elements = three rounds of 32 lanes (94 % of the lanes busy): which of the two
    // rows and which column a lane handles in each round does not depend on the pair, so no
    // element index is divided by 45; DG_PAIRS pairs (3 DG_PAIRS loads) in flight per lane.
    const int2 pruned = make_int2((int)((unsigned)CLS_PRUNE << 30), 0);
    const int rsel[3] = {0, lane >= 13, 1};
    const int col[3] = {lane, lane < 13 ? 32 + lane : lane - 13, 19 + lane};
#pragma unroll 1
    for (int p0 = 0; p0 < 16; p0 += DG_PAIRS) {
      float v[DG_PAIRS][3];
      int2 info[DG_PAIRS][3];
#pragma unroll
      for (int q = 0; q < DG_PAIRS; q++)
#pragma unroll
        for (int rd = 0; rd < 3; rd++) {
          info[q][rd] = tab[2 * (p0 + q) + rsel[rd]];
          if (rd == 2 && lane >= 26) info[q][rd] = pruned;  // 90 elements: the third round has 26
        }
#pragma unroll
      for (int q = 0; q < DG_PAIRS; q++)
#pragma unroll
        for (int rd = 0; rd < 3; rd++) {  // all loads are issued before any is consumed
          v[q][rd] = 0.f;
          if (((unsigned)info[q][rd].x >> 30) != CLS_PRUNE)
            v[q][rd] = __ldg(gsrc + (2 * (p0 + q) + rsel[rd]) * w + col[rd]);
        }
#pragma unroll
      for (int q = 0; q < DG_PAIRS; q++)
#pragma unroll
        for (int rd = 0; rd < 3; rd++) emit_fixed(2 * (p0 + q) + rsel[rd], col[rd], info[q][rd], v[q][rd]);
    }
  } else {
    // w = 1, 3, 4: the whole group is w rounds of 32 lanes, row and column of a lane's element in
    // round u are the same for every group (hoisted out of the group loop by the compiler)
    float v[w];
    int2 info[w];
#pragma unroll
    for (int u = 0; u < w; u++) info[u] = tab[(32 * u + lane) / w];
#pragma unroll
    for (int u = 0; u < w; u++) {
      v[u] = 0.f;
      if (((unsigned)info[u].x >> 30) != CLS_PRUNE) v[u] = __ldg(gsrc + 32 * u + lane);
    }
#pragma unroll
    for (int u = 0; u < w; u++) {
      const int e = 32 * u + lane, r = e / w;
      emit_fixed(r, e - r * w, info[u], v[u]);
    }
  }
}

template <int A, int SET>
__device__ __noinline__ void rows_loop(int N, const uint8_t *__restrict__ cls, const Slot3 *__restrict__ slots, int K,
                                       int C, const Sets &S, const float *__restrict__ z, int2 *tab) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int groups = (N + 31) / 32;
  for (int g = blockIdx.x * DG_WARPS + wid; g < groups; g += gridDim.x * DG_WARPS) {
    const int row0 = g * 32, row = row0 + lane;
    uint8_t c = CLS_PRUNE;
    Slot3 sl{0, 0, 0};
    if (row < N) {
      c = cls[row];
      sl = slots[row];
    }
    // (class | survivor slot, new-row slot); slots < N < 2^30
    tab[lane] = make_int2((int)((unsigned)c << 30) | sl.k, c == CLS_SPLIT ? K + C + sl.s : K + sl.c);
    __syncwarp();
    rows_job<A, SET>(row0, tab, K, C, S, z, lane);
    __syncwarp();  // the table is rewritten for the next group
  }
}

__global__ void __launch_bounds__(32 * DG_WARPS) k_density_apply_rows(int N, const uint8_t *__restrict__ cls,
                                                                       const Slot3 *__restrict__ slots, int K, int C,
                                                                       const __grid_constant__ Sets S,
                                                                       const float *__restrict__ z) {
  __shared__ int2 tabs[DG_WARPS][32];
  int2 *tab = tabs[threadIdx.x >> 5];
#define GSB_JOB(y, a, s) \
  case y: rows_loop<a, s>(N, cls, slots, K, C, S, z, tab); break;
  switch (blockIdx.y) {
    GSB_JOB(0, 2, 0) GSB_JOB(1, 2, 1) GSB_JOB(2, 2, 2) GSB_JOB(3, 0, 0) GSB_JOB(4, 0, 1) GSB_JOB(5, 0, 2)
    GSB_JOB(6, 1, 0) GSB_JOB(7, 1, 1) GSB_JOB(8, 1, 2) GSB_JOB(9, 3, 0) GSB_JOB(10, 3, 1) GSB_JOB(11, 3, 2)
    GSB_JOB(12, 4, 0) GSB_JOB(13, 4, 1) GSB_JOB(14, 4, 2) GSB_JOB(15, 5, 0) GSB_JOB(16, 5, 1) GSB_JOB(17, 5, 2)
  }
#undef GSB_JOB
}

// gsmodel.py:320-331
__global__ void k_reset_alpha(int64_t N, float *__restrict__ alphas_raw, float *__restrict__ m,
                              float *__restrict__ v, float val) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  if (alphas_raw[i] > val) alphas_raw[i] = val;
  if (m) m[i] = 0.f;
  if (v) v[i] = 0.f;
}

// ---- record conversion.  A "gs row" is the reference's .npy record (gau_io.py:7-12):
// pw[3] rot[4] scale[3] alpha sh[sh_dim], 11 + sh_dim floats, activated values.

// gau_io.py:60-107.  rows: the PLY vertex block [N, stride] f32; colmap[j] = source column of
// output column j (the f_rest channel-major -> coefficient-major transpose of :91 is folded
// into the map by the host).  rot is divided by its norm (no epsilon, :80), scale -> exp,
// opacity -> sigmoid.
__global__ void k_ply_rows_to_gs(int64_t N, int stride, int J, const float *__restrict__ rows,
                                 const int32_t *__restrict__ colmap, float *__restrict__ out) {
  const int64_t total = N * J;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / J;
    const int j = (int)(e - i * J);
    const float *__restrict__ row = rows + i * stride;
    float v = row[colmap[j]];
    if (j >= 3 && j < 7) {
      const float a = row[colmap[3]], b = row[colmap[4]], c = row[colmap[5]], d = row[colmap[6]];
      v = v / sqrtf(a * a + b * b + c * c + d * d);
    } else if (j >= 7 && j < 10) {
      v = expf(v);
    } else if (j == 10) {
      v = 1.f / (1.f + expf(-v));
    }
    out[e] = v;
  }
}

// gsmodel.py:95-113: gs rows -> raw training tensors; high_shs padded with 0.001 up to 45
__global__ void k_gs_to_params(int64_t N, int sh_dim, const float *__restrict__ gs, float *__restrict__ pws,
                               float *__restrict__ low, float *__restrict__ high, float *__restrict__ alphas_raw,
                               float *__restrict__ scales_raw, float *__restrict__ rots_raw) {
  const int J = 11 + sh_dim;
  const int64_t total = N * 59;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / 59;
    const int c = (int)(e - i * 59);
    const float *__restrict__ row = gs + i * J;
    if (c < 3) {
      pws[3 * i + c] = row[c];
    } else if (c < 7) {
      rots_raw[4 * i + c - 3] = row[c];
    } else if (c < 10) {
      scales_raw[3 * i + c - 7] = logf(row[c]);
    } else if (c == 10) {
      const float a = row[10];
      alphas_raw[i] = logf(a / (1.f - a));
    } else if (c < 14) {
      low[3 * i + c - 11] = row[c];
    } else {
      const int h = c - 14;
      high[45 * i + h] = (h + 3 < sh_dim) ? row[c] : 0.001f;
    }
  }
}

// gau_io.py:138-153: training tensors -> gs rows with sh_dim = 48
__global__ void k_params_to_gs(int64_t N, const float *__restrict__ pws, const float *__restrict__ low,
                               const float *__restrict__ high, const float *__restrict__ alphas_raw,
                               const float *__restrict__ scales_raw, const float *__restrict__ rots_raw,
                               float *__restrict__ gs) {
  const int64_t total = N * 59;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / 59;
    const int c = (int)(e - i * 59);
    float v;
    if (c < 3) {
      v = pws[3 * i + c];
    } else if (c < 7) {
      const float *q = rots_raw + 4 * i;
      v = q[c - 3] / fmaxf(sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]), 1e-12f);
    } else if (c < 10) {
      v = expf(scales_raw[3 * i + c - 7]);
    } else if (c == 10) {
      v = 1.f / (1.f + expf(-alphas_raw[i]));
    } else if (c < 14) {
      v = low[3 * i + c - 11];
    } else {
      v = high[45 * i + c - 14];
    }
    gs[e] = v;
  }
}

inline int stream_grid(int64_t total, int block) {
  int64_t b = (total + block - 1) / block;
  const int64_t cap = 148 * 16;  // grid-stride: a few waves of the 148 SMs
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace

size_t density_workspace_bytes(int64_t N) {
  // [three int64 totals, padded to 256 B][three counts per 1024-row CTA]
  return 256 + (size_t)((N + SC_ROWS - 1) / SC_ROWS + 1) * 3 * sizeof(int32_t);
}

int launch_density_accumulate(int64_t N, const float *dloss_dus, const uint8_t *mask, float *grad_accum,
                              int32_t *cunt, int init, cudaStream_t st) {
  if (N == 0) return 0;
  ProfScope ps(K_DENSITY_ACC, st);
  k_density_accumulate<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(N, reinterpret_cast<const float2 *>(dloss_dus),
                                                                     mask, grad_accum, cunt, init);
  GSB_CUDA_TRY(cudaGetLastError());
  return 0;
}

int launch_density_plan(int64_t N, const float *alphas_raw, const float *scales_raw, const float *grad_accum,
                        const int32_t *cunt, float alpha_raw_min, float scale_raw_max, float grad_min,
                        float scale_clone_max, void *ws, size_t ws_bytes, uint8_t *cls, int32_t *slots,
                        int64_t *counts_host, cudaStream_t st) {
  counts_host[0] = counts_host[1] = counts_host[2] = 0;
  if (N == 0) return 0;
  int64_t *totals = static_cast<int64_t *>(ws);
  int32_t *block_counts = reinterpret_cast<int32_t *>(static_cast<char *>(ws) + 256);
  const int nb = (int)((N + SC_ROWS - 1) / SC_ROWS);
  {
    ProfScope ps(K_DENSITY_CLASSIFY, st);
    k_density_classify_count<<<nb, SC_THREADS, 0, st>>>(N, alphas_raw, scales_raw, grad_accum, cunt, alpha_raw_min,
                                                       scale_raw_max, grad_min, scale_clone_max, cls, block_counts);
    GSB_CUDA_TRY(cudaGetLastError());
  }
  {
    ProfScope ps(K_DENSITY_SCAN, st);
    k_density_scan_blocks<<<1, 1024, 0, st>>>(nb, block_counts, totals);
    k_density_slots<<<nb, SC_THREADS, 0, st>>>(N, cls, block_counts, reinterpret_cast<Slot3 *>(slots));
    GSB_CUDA_TRY(cudaGetLastError());
  }
  GSB_CUDA_TRY(cudaMemcpyAsync(counts_host, totals, 3 * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  GSB_CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}

int launch_density_apply(int64_t N, const uint8_t *cls, const int32_t *slots, int64_t K, int64_t C,
                         float *const *src, float *const *src_m, float *const *src_v, const float *z,
                         float *const *dst, float *const *dst_m, float *const *dst_v, cudaStream_t st) {
  if (N == 0) return 0;
  Sets S;
  for (int a = 0; a < 6; a++) {
    S.p[a] = src[a];
    S.m[a] = src_m ? src_m[a] : nullptr;
    S.v[a] = src_v ? src_v[a] : nullptr;
    S.dp[a] = dst[a];
    S.dm[a] = dst_m ? dst_m[a] : nullptr;
    S.dv[a] = dst_v ? dst_v[a] : nullptr;
  }
  ProfScope ps(K_DENSITY_APPLY, st);
  if (N < 23000000) {
    int dev = 0, sms = 148;
    GSB_CUDA_TRY(cudaGetDevice(&dev));
    GSB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int64_t blocks = (N + 32 * DG_WARPS - 1) / (32 * DG_WARPS);
    const int grid_x = (int)(blocks < (int64_t)sms * 8 ? blocks : (int64_t)sms * 8);
    const dim3 grid(grid_x, 18);
    k_density_apply_rows<<<grid, 32 * DG_WARPS, 0, st>>>((int)N, cls, reinterpret_cast<const Slot3 *>(slots), (int)K,
                                                         (int)C, S, z);
    GSB_CUDA_TRY(cudaGetLastError());
    return 0;
  }
  dim3 grid(stream_grid((N * 45 + 3) / 4, 256), 18);
  k_density_apply<<<grid, 256, 0, st>>>(N, cls, reinterpret_cast<const Slot3 *>(slots), K, C, S, z);
  GSB_CUDA_TRY(cudaGetLastError());
  return 0;
}

int launch_reset_alpha(int64_t N, float *alphas_raw, float *m, float *v, float val, cudaStream_t st) {
  if (N == 0) return 0;
  ProfScope ps(K_RESET_ALPHA, st);
  k_reset_alpha<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(N, alphas_raw, m, v, val);
  GSB_CUDA_TRY(cudaGetLastError());
  return 0;
}

int launch_ply_rows_to_gs(int64_t N, int stride, int sh_dim, const float *rows, const int32_t *colmap, float *gs,
                          cudaStream_t st) {
  if (N == 0) return 0;
  ProfScope ps(K_GS_DECODE, st);
  const int J = 11 + sh_dim;
  k_ply_rows_to_gs<<<stream_grid(N * J, 256), 256, 0, st>>>(N, stride, J, rows, colmap, gs);
  GSB_CUDA_TRY(cudaGetLastError());
  return 0;
}

int launch_gs_to_params(int64_t N, int sh_dim, const float *gs, float *const *dst, cudaStream_t st) {
  if (N == 0) return 0;
  ProfScope ps(K_GS_TO_PARAMS, st);
  k_gs_to_params<<<stream_grid(N * 59, 256), 256, 0, st>>>(N, sh_dim, gs, dst[0], dst[1], dst[2], dst[3], dst[4],
                                                          dst[5]);
  GSB_CUDA_TRY(cudaGetLastError());
  return 0;
}

int launch_params_to_gs(int64_t N, float *const *src, float *gs, cudaStream_t st) {
  if (N == 0) return 0;
  ProfScope ps(K_PARAMS_TO_GS, st);
  k_params_to_gs<<<stream_grid(N * 59, 256), 256, 0, st>>>(N, src[0], src[1], src[2], src[3], src[4], src[5], gs);
  GSB_CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // namespace gsb
