// Backward tile rasterizer ("drawB").  Replaces reference kernel.cu:809-950.
//
// This file holds the moment finalisation and the launcher; the kernel and its algorithm notes
// are k_draw_bwd4 in raster_bwd4.cu.  Each pixel replays its saved (final_tau, contrib) state back
// to front: tau <- tau / (1 - alpha'), dL/dalpha' = tau (c - gamma_next) . dL/dgamma, with
// gamma_next kept as the scalar s = dL/dgamma . gamma_next (s <- alpha' (dL/dgamma . c) + (1 - alpha') s).
// Geometry gradients are linear in per-pixel moments, so the kernel accumulates per Gaussian one
// contiguous 9-float moment row
//   w dx, w dy, w dx^2, w dx dy, w dy^2   (w = dL/dalpha' * alpha'),  dL/dalpha' * g,  alpha' tau dL/dgamma_rgb
// and finalize_splat_grads() turns the rows into the four gradient tensors:
//   dL/du = -(A Sx + B Sy, B Sx + C Sy),  dL/dconic = (-Sxx/2, -Sxy, -Syy/2).
#include "common.cuh"
#include "kernels.h"
#include "tile_io.cuh"

namespace gsb {

constexpr int MOM = 9;  // floats per moment row

// moment rows [N,9] -> dloss_dus[N,2], dloss_dcinv2ds[N,3], dloss_dalphas[N], dloss_dcolors[N,3]
__global__ void __launch_bounds__(PG) k_finalize_grads(int N, const float *__restrict__ moments,
                                                       const float *__restrict__ cinv2ds,
                                                       float *__restrict__ dus, float *__restrict__ dcinv,
                                                       float *__restrict__ dalphas, float *__restrict__ dcolors) {
  __shared__ float sm[TileT<MOM>::FLOATS];
  const int tid = threadIdx.x;
  const long long base = (long long)blockIdx.x * PG;
  const int nv = min(PG, (int)(N - base));
  const bool valid = tid < nv;
  float A = 0.f, B = 0.f, Cc = 0.f, m[MOM];
  tile_fetch<3>(cinv2ds, base, nv, sm, tid);
  __syncthreads();
  if (valid) { const float *r = sm + tid * TileT<3>::S; A = r[0]; B = r[1]; Cc = r[2]; }
  __syncthreads();
  tile_fetch<MOM>(moments, base, nv, sm, tid);
  __syncthreads();
#pragma unroll
  for (int i = 0; i < MOM; i++) m[i] = valid ? sm[tid * TileT<MOM>::S + i] : 0.f;
  __syncthreads();
  {
    // untouched Gaussians stay exactly 0 even if their conic is inf/NaN (reference: no atomics ran)
    const bool none = (m[0] == 0.f) && (m[1] == 0.f);
    float *o = sm + tid * TileT<2>::S;
    o[0] = none ? 0.f : -(A * m[0] + B * m[1]);
    o[1] = none ? 0.f : -(B * m[0] + Cc * m[1]);
  }
  __syncthreads();
  tile_flush<2>(dus, base, nv, sm, tid);
  __syncthreads();
  { float *o = sm + tid * TileT<3>::S; o[0] = -0.5f * m[2]; o[1] = -m[3]; o[2] = -0.5f * m[4]; }
  __syncthreads();
  tile_flush<3>(dcinv, base, nv, sm, tid);
  __syncthreads();
  { float *o = sm + tid * TileT<3>::S; o[0] = m[6]; o[1] = m[7]; o[2] = m[8]; }
  __syncthreads();
  tile_flush<3>(dcolors, base, nv, sm, tid);
  if (valid) dalphas[base + tid] = m[5];
}

int launch_draw_backward(int H, int W, int N, const int32_t *ranges, const Rec *recs, const int32_t *gsid,
                         const int32_t *contrib,
                         const float *final_tau, const float *dloss_dgammas, const float *cinv2ds,
                         float *moments, int *work_counter, float *dloss_dus,
                         float *dloss_dcinv2ds, float *dloss_dalphas, float *dloss_dcolors, bool finalize,
                         cudaStream_t st) {
  const int gx = (W + TILE - 1) / TILE, gy = (H + TILE - 1) / TILE;
  if (gx <= 0 || gy <= 0 || N <= 0) return 0;
  GSB_CUDA_TRY(cudaMemsetAsync(moments, 0, sizeof(float) * MOM * (size_t)N, st));
  if (recs != nullptr) {
    int rc = launch_draw_bwd4_kernel(H, W, ranges, recs, gsid, contrib, final_tau, dloss_dgammas, moments,
                                     work_counter, st);
    if (rc) return rc;
  }
  GSB_CUDA_TRY(cudaGetLastError());
  if (finalize) {  // otherwise the caller consumes the moment rows (gsb_preprocess_backward)
    ProfScope ps(K_FINALIZE, st);
    k_finalize_grads<<<(N + PG - 1) / PG, PG, 0, st>>>(N, moments, cinv2ds, dloss_dus, dloss_dcinv2ds,
                                                       dloss_dalphas, dloss_dcolors);
  }
  GSB_CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // namespace gsb
