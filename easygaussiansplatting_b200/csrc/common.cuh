// Shared device helpers for the sm_100a kernels: constants fixed by the reference, the packed
// record, fast math, PTX wrappers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gsb {

constexpr int TILE = 16;              // reference common.cuh:13
constexpr float MIN_DEPTH = 0.2f;     // kernel.cu:10: (float)z < 0.2 (double)  <=>  z < 0.2f
constexpr float BAD_MARKER = -1.0f;   // kernel.cu:11
constexpr float ALPHA_CLAMP = 0.99f;  // kernel.cu:245
constexpr float ALPHA_SKIP = 0.002f;  // kernel.cu:246
constexpr float TAU_STOP = 0.0001f;   // kernel.cu:256
constexpr float LOG2E = 1.4426950408889634f;

// Packed per-Gaussian record, 48 B (build_record below), 16-B aligned: the rasterizers gather it
// with three 16-byte cp.async.
//   q0 = (ux, uy, gsid bits, alpha)   mean in pixels, Gaussian id, opacity -- exactly the four
//                              words the backward's moment phase needs per record (one 16-byte copy)
//   q1 = (a, b, c, thr)        log2(g) = a dx^2 + b dx dy + c dy^2  (conic pre-scaled by
//                              -0.5*log2e, -log2e, -0.5*log2e); thr = log2(alpha / 0.002) (+margin):
//                              a pixel can reach alpha' >= 0.002 only where -log2(g) <= thr
//                              (+inf: never cull, -inf: never contributes)
//   q2 = (r, g, b, 0)
struct __align__(16) Rec {
  float4 q0, q1, q2;
};
static_assert(sizeof(Rec) == 48, "record must be 48 bytes");

// GSB_EXACT_MATH=1 (variant builds only, benchmarks/compare_ref_gpu.py --three-way): IEEE reciprocal
// and an exp2 evaluated in double precision instead of the MUFU approximations, to show how much
// of the distance to the fp64 oracle comes from them (CUDA's own exp2f is MUFU.EX2 plus range
// scaling, i.e. the same 2-ulp function).
#ifndef GSB_EXACT_MATH
#define GSB_EXACT_MATH 0
#endif
__device__ __forceinline__ float rcp_approx(float x) {
#if GSB_EXACT_MATH
  return __frcp_rn(x);
#else
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#endif
}
__device__ __forceinline__ float ex2_approx(float x) {
#if GSB_EXACT_MATH
  return (float)exp2((double)x);
#else
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#endif
}

// alpha' of one record at one pixel -- THE single definition used by forward and backward
// so both take identical skip decisions (kernel.cu:243-246 / :909-913).
// Returns g = exp(-maha/2) through *g.
__device__ __forceinline__ float alpha_prime(const float4 &q1, float alpha, float dx, float dy, float *g) {
  float t = fmaf(q1.y, dy, q1.x * dx);
  float p = fmaf(t, dx, (q1.z * dy) * dy);
  p = fminf(p, 0.0f);  // max(0, maha)
  float gg = ex2_approx(p);
  *g = gg;
  return fminf(ALPHA_CLAMP, alpha * gg);
}

// Can this record reach alpha' >= 0.002 anywhere in the pixel rectangle [bx0,bx1] x [by0,by1]?
// Exact minimum of the (positive definite) quadratic Q = -log2(g) over the continuous
// rectangle: 0 if the mean lies inside, otherwise the smallest of the four edge minima (each a
// clamped 1-D parabola).  Conservative by construction (continuous rectangle >= pixel centres)
// plus an fp32 error allowance proportional to the largest term magnitude, so a record is only
// dropped when every pixel of the rectangle would take the reference's `continue`
// (kernel.cu:246) -- image, contrib and final_tau are unaffected.
__device__ __forceinline__ bool rec_can_touch(const float4 &q0, const float4 &q1, float bx0, float bx1,
                                              float by0, float by1) {
  const float A = -q1.x, B = -q1.y, C = -q1.z;
  const float dxl = q0.x - bx1, dxh = q0.x - bx0, dyl = q0.y - by1, dyh = q0.y - by0;
  const bool inside = (dxl <= 0.f) && (dxh >= 0.f) && (dyl <= 0.f) && (dyh >= 0.f);
  const float kx = __fdividef(-0.5f * B, C), ky = __fdividef(-0.5f * B, A);
  float qmin = 3.0e38f;
#pragma unroll
  for (int e = 0; e < 2; e++) {
    const float ex = e ? dxh : dxl;
    const float dy = fminf(fmaxf(kx * ex, dyl), dyh);
    qmin = fminf(qmin, fmaf(fmaf(B, ex, C * dy), dy, A * ex * ex));
    const float ey = e ? dyh : dyl;
    const float dx = fminf(fmaxf(ky * ey, dxl), dxh);
    qmin = fminf(qmin, fmaf(fmaf(B, ey, A * dx), dx, C * ey * ey));
  }
  if (inside) qmin = 0.f;
  const float X = fmaxf(fabsf(dxl), fabsf(dxh)), Y = fmaxf(fabsf(dyl), fabsf(dyh));
  const float S = fmaf(A * X, X, fmaf(fabsf(B) * X, Y, C * Y * Y));
  return !(qmin > q1.w + fmaf(2.0e-6f, S, 1.0e-5f));  // NaN anywhere keeps the record
}

// The 48-byte record the rasterizers work from (one per Gaussian).
// thr = log2(alpha / 0.002): -log2(g) <= thr is necessary for alpha' >= 0.002 -- the bound of the
// warp-level culling test (rec_can_touch); the positive-definiteness check carries a safety
// factor against fp32 cancellation in A C - B^2.
__device__ __forceinline__ Rec build_record(float ux, float uy, float A, float B, float C, float al, float cr,
                                            float cg, float cb, int id) {
  float thr = INFINITY;  // never cull unless the conic is a proper positive definite form
  if (al < ALPHA_SKIP) {
    thr = -INFINITY;  // alpha * g < 0.002 everywhere: never contributes
  } else {
    const float ac = A * C;
    const float det = fmaf(A, C, -B * B);
    if (A > 0.f && C > 0.f && det > 1e-4f * ac && ac < 3.0e38f) {
      const float t = __log2f(al * 500.0f) + 1e-4f;  // log2(alpha / 0.002), lg2.approx error << margin
      if (t < 3.0e38f) thr = t;
    }
  }
  Rec r;
  r.q0 = make_float4(ux, uy, __int_as_float(id), al);
  r.q1 = make_float4(-0.5f * LOG2E * A, -LOG2E * B, -0.5f * LOG2E * C, thr);
  r.q2 = make_float4(cr, cg, cb, 0.f);
  return r;
}

// ---- system-scope flags for the multi-GPU gradient exchange (peer memory over NVLink)
__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ---- shared-memory address of a generic pointer (the operand of ld/st.shared and cp.async)
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

}  // namespace gsb

#define GSB_CUDA_TRY(expr)                                 \
  do {                                                     \
    cudaError_t _e = (expr);                               \
    if (_e != cudaSuccess) return gsb::set_cuda_error(_e, #expr, __FILE__, __LINE__); \
  } while (0)

namespace gsb {
int set_cuda_error(cudaError_t e, const char *what, const char *file, int line);
int set_arg_error(const char *msg);
}  // namespace gsb
