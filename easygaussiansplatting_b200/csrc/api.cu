// extern "C" entry points declared in include/gsplat_b200.h.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "../../include/gsplat_b200.h"
#include "common.cuh"
#include "kernels.h"

namespace gsb {

static thread_local char g_err[512] = "";

int set_cuda_error(cudaError_t e, const char *what, const char *file, int line) {
  snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) in %s at %s:%d", (int)e, cudaGetErrorString(e), what,
           file, line);
  return (int)e;
}
int set_arg_error(const char *msg) {
  snprintf(g_err, sizeof(g_err), "argument error: %s", msg);
  return -1;
}

// ---- profiling
static bool g_prof_on = false;
static long long g_launches[K_COUNT] = {0};
struct EvPair { cudaEvent_t a, b; };
static std::vector<EvPair> g_events[K_COUNT];
static std::mutex g_prof_mu;
static const char *const g_names[K_COUNT] = {"project", "computeCov3D", "computeCov2D", "sh2Color",
                                             "inverseCov2D", "rects+scan", "scan(unused)", "keys", "sort",
                                             "ranges", "pack_records", "draw", "draw_backward",
                                             "preprocess_forward", "preprocess_backward",
                                             "finalize_splat_grads", "gau_loss_forward", "gau_loss_backward",
                                             "small_bmm", "density_accumulate", "density_classify",
                                             "density_scan", "density_apply", "reset_alpha",
                                             "ply_rows_to_gs", "gs_to_params", "params_to_gs",
                                             "grad_reduce_broadcast", "sh_grad_expand"};

ProfScope::ProfScope(int id, cudaStream_t st) : id_(id), st_(st), stop_(nullptr) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_launches[id]++;
  if (g_prof_on) {
    EvPair e;
    if (cudaEventCreate(&e.a) == cudaSuccess && cudaEventCreate(&e.b) == cudaSuccess) {
      cudaEventRecord(e.a, st);
      stop_ = e.b;
      g_events[id].push_back(e);
    }
  }
}
ProfScope::~ProfScope() {
  if (stop_) cudaEventRecord(stop_, st_);
}

}  // namespace gsb

using namespace gsb;

#define GSB_REQUIRE(cond, msg) \
  do {                         \
    if (!(cond)) return set_arg_error(msg); \
  } while (0)

extern "C" {

int gsb_abi_version(void) { return GSB_ABI_VERSION; }
const char *gsb_last_error(void) { return g_err; }

int gsb_project(int N, const float *pws, const float *Rcw, const float *tcw, float fx, float fy,
                float cx, float cy, float *us, float *pcs, float *depths, float *du_dpcs,
                gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0, "project: N < 0");
  GSB_REQUIRE(N == 0 || (pws && Rcw && tcw && us && pcs && depths), "project: null pointer");
  return launch_project(N, pws, Rcw, tcw, fx, fy, cx, cy, us, pcs, depths, du_dpcs, (cudaStream_t)stream);
}

int gsb_compute_cov3d(int N, const float *rots, const float *scales, const float *depths,
                      float *cov3ds, float *dcov3d_drots, float *dcov3d_dscales, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0, "computeCov3D: N < 0");
  GSB_REQUIRE(N == 0 || (rots && scales && depths && cov3ds), "computeCov3D: null pointer");
  GSB_REQUIRE((dcov3d_drots == nullptr) == (dcov3d_dscales == nullptr),
              "computeCov3D: Jacobian outputs must be both set or both null");
  return launch_cov3d(N, rots, scales, depths, cov3ds, dcov3d_drots, dcov3d_dscales, (cudaStream_t)stream);
}

int gsb_compute_cov2d(int N, const float *cov3ds, const float *pcs, const float *Rcw,
                      const float *depths, float fx, float fy, float width, float height,
                      float *cov2ds, float *dcov2d_dcov3ds, float *dcov2d_dpcs, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0, "computeCov2D: N < 0");
  GSB_REQUIRE(N == 0 || (cov3ds && pcs && Rcw && depths && cov2ds), "computeCov2D: null pointer");
  GSB_REQUIRE((dcov2d_dcov3ds == nullptr) == (dcov2d_dpcs == nullptr),
              "computeCov2D: Jacobian outputs must be both set or both null");
  return launch_cov2d(N, cov3ds, pcs, Rcw, depths, fx, fy, width, height, cov2ds, dcov2d_dcov3ds,
                      dcov2d_dpcs, (cudaStream_t)stream);
}

int gsb_sh2color(int N, int sh_dim3, const float *shs, const float *pws, const float *twc,
                 float *colors, float *dcolor_dshs, float *dcolor_dpws, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0, "sh2Color: N < 0");
  GSB_REQUIRE(sh_dim3 == 1 || sh_dim3 == 4 || sh_dim3 == 9 || sh_dim3 == 16,
              "sh2Color: shs.shape[1]/3 must be 1, 4, 9 or 16");
  GSB_REQUIRE(N == 0 || (shs && pws && twc && colors), "sh2Color: null pointer");
  GSB_REQUIRE((dcolor_dshs == nullptr) == (dcolor_dpws == nullptr),
              "sh2Color: Jacobian outputs must be both set or both null");
  return launch_sh2color(N, sh_dim3, shs, pws, twc, colors, dcolor_dshs, dcolor_dpws, (cudaStream_t)stream);
}

int gsb_inverse_cov2d(int N, const float *cov2ds, float *depths, float *cinv2ds, int32_t *areas,
                      float *dcinv2d_dcov2ds, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0, "inverseCov2D: N < 0");
  GSB_REQUIRE(N == 0 || (cov2ds && depths && cinv2ds && areas), "inverseCov2D: null pointer");
  return launch_inv_cov2d(N, cov2ds, depths, cinv2ds, areas, dcinv2d_dcov2ds, (cudaStream_t)stream);
}

void gsb_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_on = on != 0;
}
int gsb_profile_kernels(void) { return (int)K_COUNT; }
const char *gsb_profile_kernel_name(int id) { return (id >= 0 && id < K_COUNT) ? g_names[id] : ""; }
long long gsb_profile_launches(int id) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (id >= 0 && id < K_COUNT) return g_launches[id];
  long long t = 0;
  for (int i = 0; i < K_COUNT; i++) t += g_launches[i];
  return t;
}
int gsb_profile_read(int id, double *ms_total, long long *timed_launches) {
  GSB_REQUIRE(id >= 0 && id < K_COUNT && ms_total && timed_launches, "profile_read: bad arguments");
  std::lock_guard<std::mutex> lk(g_prof_mu);
  double tot = 0.0;
  long long cnt = 0;
  for (auto &e : g_events[id]) {
    float ms = 0.f;
    if (cudaEventSynchronize(e.b) == cudaSuccess && cudaEventElapsedTime(&ms, e.a, e.b) == cudaSuccess) {
      tot += ms;
      cnt++;
    }
    cudaEventDestroy(e.a);
    cudaEventDestroy(e.b);
  }
  g_events[id].clear();
  *ms_total = tot;
  *timed_launches = cnt;
  return 0;
}

int gsb_preprocess_forward(int N, int sh_dim3, const float *pws, const float *rots, const float *scales,
                           const float *shs, const float *Rcw, const float *tcw, const float *twc, float fx,
                           float fy, float cx, float cy, float width, float height, float *us,
                           float *cinv2ds, float *colors, float *depths, int32_t *areas, const float *alphas,
                           void *records, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0, "preprocess: N < 0");
  GSB_REQUIRE((alphas == nullptr) == (records == nullptr), "preprocess: alphas and records go together");
  GSB_REQUIRE((reinterpret_cast<uintptr_t>(records) & 15) == 0, "preprocess: records misaligned");
  GSB_REQUIRE(sh_dim3 == 1 || sh_dim3 == 4 || sh_dim3 == 9 || sh_dim3 == 16,
              "preprocess: shs.shape[1]/3 must be 1, 4, 9 or 16");
  GSB_REQUIRE(N == 0 || (pws && rots && scales && shs && Rcw && tcw && twc && us && cinv2ds && colors &&
                         depths && areas),
              "preprocess: null pointer");
  return launch_preprocess_fwd(N, sh_dim3, pws, rots, scales, shs, Rcw, tcw, twc, fx, fy, cx, cy, width, height,
                               us, cinv2ds, colors, depths, areas, alphas, static_cast<Rec *>(records),
                               (cudaStream_t)stream);
}

int gsb_preprocess_backward(int N, int sh_dim3, const float *pws, const float *rots, const float *scales,
                            const float *shs, const float *Rcw, const float *tcw, const float *twc, float fx,
                            float fy, float cx, float cy, float width, float height, const float *dloss_dus,
                            const float *dloss_dcinv2ds, const float *dloss_dcolors, float *dloss_dpws,
                            float *dloss_dshs, float *dloss_dscales, float *dloss_drots, const float *moments,
                            const float *cinv2ds, float *dloss_dus_out, float *dloss_dalphas_out,
                            gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0, "preprocessB: N < 0");
  if (moments != nullptr) {  // upstream gradients as moment rows (gsb_splat_backward with moments_out)
    GSB_REQUIRE(sh_dim3 == 1 || sh_dim3 == 4 || sh_dim3 == 9 || sh_dim3 == 16,
                "preprocessB: shs.shape[1]/3 must be 1, 4, 9 or 16");
    GSB_REQUIRE(N == 0 || (pws && rots && scales && shs && Rcw && tcw && twc && cinv2ds && dloss_dus_out &&
                           dloss_dalphas_out && dloss_dpws && dloss_dscales && dloss_drots),
                "preprocessB: null pointer");  // (dloss_dshs may be NULL: see gsb_sh_grad_expand)
    const MomentsIn mi{moments, cinv2ds, dloss_dus_out, dloss_dalphas_out};
    return launch_preprocess_bwd(N, sh_dim3, pws, rots, scales, shs, Rcw, tcw, twc, fx, fy, cx, cy, width, height,
                                 nullptr, nullptr, nullptr, dloss_dpws, dloss_dshs, dloss_dscales, dloss_drots, &mi,
                                 (cudaStream_t)stream);
  }
  GSB_REQUIRE(sh_dim3 == 1 || sh_dim3 == 4 || sh_dim3 == 9 || sh_dim3 == 16,
              "preprocessB: shs.shape[1]/3 must be 1, 4, 9 or 16");
  GSB_REQUIRE(N == 0 || (pws && rots && scales && shs && Rcw && tcw && twc && dloss_dus && dloss_dcinv2ds &&
                         dloss_dcolors && dloss_dpws && dloss_dshs && dloss_dscales && dloss_drots),
              "preprocessB: null pointer");
  return launch_preprocess_bwd(N, sh_dim3, pws, rots, scales, shs, Rcw, tcw, twc, fx, fy, cx, cy, width, height,
                               dloss_dus, dloss_dcinv2ds, dloss_dcolors, dloss_dpws, dloss_dshs, dloss_dscales,
                               dloss_drots, nullptr, (cudaStream_t)stream);
}

int gsb_sh_grad_expand(int N, int sh_dim3, int V, const float *pws, const float *twcs, const float *dloss_dcolors,
                       float *dloss_dshs, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0 && V >= 1, "sh_grad_expand: bad N / V");
  GSB_REQUIRE(sh_dim3 == 1 || sh_dim3 == 4 || sh_dim3 == 9 || sh_dim3 == 16,
              "sh_grad_expand: sh_dim3 must be 1, 4, 9 or 16");
  GSB_REQUIRE(N == 0 || (pws && twcs && dloss_dcolors && dloss_dshs), "sh_grad_expand: null pointer");
  return launch_sh_expand(N, sh_dim3, V, pws, twcs, dloss_dcolors, dloss_dshs, (cudaStream_t)stream);
}

int gsb_small_bmm(long long batch, int m, int k, int n, const float *A, const float *B, int b_shared, float *C,
                  gsb_stream_t stream) {
  GSB_REQUIRE(batch >= 0 && m > 0 && k > 0 && n > 0, "small_bmm: bad shape");
  GSB_REQUIRE(batch == 0 || (A && B && C), "small_bmm: null pointer");
  return launch_small_bmm(batch, m, k, n, A, B, b_shared, C, (cudaStream_t)stream);
}

size_t gsb_gau_loss_workspace_bytes(int H, int W) { return gau_loss_workspace_bytes(H, W); }

int gsb_gau_loss(int H, int W, const float *image, const float *gt_image, float loss_lambda, float *loss_out,
                 float *dloss_dimage, void *ws, size_t ws_bytes, gsb_stream_t stream) {
  GSB_REQUIRE(H > 0 && W > 0, "gau_loss: bad H/W");
  GSB_REQUIRE(image && gt_image && loss_out && ws, "gau_loss: null pointer");
  GSB_REQUIRE(ws_bytes >= gau_loss_workspace_bytes(H, W), "gau_loss: workspace too small");
  return launch_gau_loss(H, W, image, gt_image, loss_lambda, loss_out, dloss_dimage, ws, (cudaStream_t)stream);
}

size_t gsb_splat_bin_workspace_bytes(int N) { return bin_layout(N).bytes; }

int gsb_splat_bin(int H, int W, int N, const float *us, float *depths, int32_t *areas, void *bin_ws,
                  size_t bin_ws_bytes, int64_t *P_host, uint32_t *depth_key_max_host, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0 && H > 0 && W > 0, "splat: bad N/H/W");
  GSB_REQUIRE(P_host != nullptr && bin_ws != nullptr, "splat: null workspace / P_host");
  GSB_REQUIRE(N == 0 || (us && depths && areas), "splat: null pointer");
  const BinLayout L = bin_layout(N);
  GSB_REQUIRE(bin_ws_bytes >= L.bytes, "splat: bin workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  int rc = launch_bin(H, W, N, us, depths, areas, bin_ws, L, st);
  if (rc) return rc;
  uint32_t total[3] = {0, 0, 0};  // [patch count, largest depth key, flags]
  GSB_CUDA_TRY(cudaMemcpyAsync(total, static_cast<char *>(bin_ws) + L.total, 3 * sizeof(uint32_t),
                               cudaMemcpyDeviceToHost, st));
  GSB_CUDA_TRY(cudaStreamSynchronize(st));
  GSB_REQUIRE((total[2] & 1u) == 0 && total[0] < (1u << 30), "splat: more than 2^30 patches");
  *P_host = (int64_t)total[0];
  if (depth_key_max_host) *depth_key_max_host = total[1];
  return 0;
}

size_t gsb_splat_records_offset(int N, int H, int W, int64_t P) {
  SortLayout L;
  if (sort_layout(N, H, W, P, &L)) return 0;
  return L.recs;
}

size_t gsb_splat_workspace_bytes(int N, int H, int W, int64_t P) {
  SortLayout L;
  if (sort_layout(N, H, W, P, &L)) return 0;
  return L.bytes;
}

int gsb_splat_render(int H, int W, int N, int64_t P, uint32_t depth_key_max, const float *us,
                     const float *cinv2ds, const float *alphas, const float *depths, const float *colors,
                     const void *packed_records, const void *bin_ws,
                     void *ws, size_t ws_bytes, float *image, int32_t *contrib, float *final_tau,
                     int32_t *patch_range_per_tile, int32_t *gsid_per_patch, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0 && H > 0 && W > 0 && P >= 0, "splat: bad N/H/W/P");
  GSB_REQUIRE(image && contrib && final_tau && patch_range_per_tile, "splat: null output");
  GSB_REQUIRE(P == 0 || (us && cinv2ds && alphas && depths && colors && bin_ws && ws && gsid_per_patch),
              "splat: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  SortLayout SL{};
  {
    int rc = sort_layout(N, H, W, P, &SL);
    if (rc) return rc;
    GSB_REQUIRE(ws != nullptr && ws_bytes >= SL.bytes, "splat: workspace too small");
  }
  const BinLayout BL = bin_layout(N);
  GSB_REQUIRE((reinterpret_cast<uintptr_t>(packed_records) & 15) == 0, "splat: packed_records misaligned");
  int rc = launch_sort_and_pack(H, W, N, P, depth_key_max, us, cinv2ds, alphas, depths, colors, bin_ws, BL, ws, SL,
                                patch_range_per_tile, gsid_per_patch, packed_records == nullptr, nullptr, st);
  if (rc) return rc;
  const Rec *recs = P > 0 ? reinterpret_cast<const Rec *>(static_cast<char *>(ws) + SL.recs) : nullptr;
  if (P > 0 && packed_records != nullptr) recs = static_cast<const Rec *>(packed_records);
  // with P == 0 every tile is empty: the rasterizer only writes zeros
  int *work = reinterpret_cast<int *>(static_cast<char *>(ws) + SL.counters);
  return launch_draw(H, W, patch_range_per_tile, recs, gsid_per_patch, image, contrib, final_tau, work, st);
}

static int splat_forward_impl(int H, int W, int N, const float *us, const float *cinv2ds, const float *alphas,
                              float *depths, const float *colors, int32_t *areas, const void *packed_records,
                              int64_t P_cap, uint32_t depth_key_cap, void *bin_ws, size_t bin_ws_bytes, void *ws,
                              size_t ws_bytes, float *image, int32_t *contrib, float *final_tau,
                              int32_t *patch_range_per_tile, int32_t *gsid_per_patch, uint32_t *status_host,
                              gsb_stream_t stream, bool wait) {
  GSB_REQUIRE(N >= 0 && H > 0 && W > 0 && P_cap > 0 && P_cap < ((int64_t)1 << 30), "splat_forward: bad N/H/W/P_cap");
  GSB_REQUIRE(image && contrib && final_tau && patch_range_per_tile && gsid_per_patch && status_host && bin_ws && ws,
              "splat_forward: null pointer");
  GSB_REQUIRE(N == 0 || (us && cinv2ds && alphas && depths && colors && areas), "splat_forward: null pointer");
  GSB_REQUIRE((reinterpret_cast<uintptr_t>(packed_records) & 15) == 0, "splat_forward: packed_records misaligned");
  cudaStream_t st = (cudaStream_t)stream;
  const BinLayout BL = bin_layout(N);
  GSB_REQUIRE(bin_ws_bytes >= BL.bytes, "splat_forward: bin workspace too small");
  SortLayout SL{};
  int rc = sort_layout(N, H, W, P_cap, &SL);
  if (rc) return rc;
  GSB_REQUIRE(ws_bytes >= SL.bytes, "splat_forward: workspace too small");
  static thread_local cudaEvent_t ready_ev = nullptr;
  if (wait && ready_ev == nullptr) GSB_CUDA_TRY(cudaEventCreateWithFlags(&ready_ev, cudaEventDisableTiming));
  cudaEvent_t ready = wait ? ready_ev : nullptr;
  const StatusRead sr{status_host, ready};
  if (wait) status_host[0] = status_host[1] = status_host[2] = 0;
  rc = launch_bin(H, W, N, us, depths, areas, bin_ws, BL, st);
  if (rc) return rc;
  int *work = reinterpret_cast<int *>(static_cast<char *>(ws) + SL.counters);
  if (N == 0) {  // nothing to bin: every tile is empty
    GSB_CUDA_TRY(cudaMemsetAsync(patch_range_per_tile, 0,
                                 sizeof(int32_t) * 2 * (size_t)((W + GSB_TILE - 1) / GSB_TILE) * ((H + GSB_TILE - 1) / GSB_TILE), st));
    return launch_draw(H, W, patch_range_per_tile, nullptr, gsid_per_patch, image, contrib, final_tau, work, st);
  }
  rc = launch_sort_and_pack(H, W, N, P_cap, depth_key_cap, us, cinv2ds, alphas, depths, colors, bin_ws, BL, ws, SL,
                            patch_range_per_tile, gsid_per_patch, packed_records == nullptr, &sr, st);
  if (rc) return rc;
  const Rec *recs = packed_records != nullptr ? static_cast<const Rec *>(packed_records)
                                              : reinterpret_cast<const Rec *>(static_cast<char *>(ws) + SL.recs);
  rc = launch_draw(H, W, patch_range_per_tile, recs, gsid_per_patch, image, contrib, final_tau, work, st);
  if (rc) return rc;
  if (!wait) return 0;  // enqueue-only (CUDA graph capture): the caller inspects status_host later
  // the sort and the rasterizer are queued; now look at what the binning found
  GSB_CUDA_TRY(cudaEventSynchronize(ready));
  if ((status_host[2] & 1u) != 0 || status_host[0] >= (1u << 30)) return set_arg_error("splat: more than 2^30 patches");
  if ((status_host[2] & 6u) != 0 || (int64_t)status_host[0] > P_cap) {
    snprintf(g_err, sizeof(g_err), "splat_forward: capacity exceeded (P = %u of %lld, flags %u)", status_host[0],
             (long long)P_cap, status_host[2]);
    return GSB_CAPACITY_EXCEEDED;
  }
  return 0;
}

int gsb_splat_forward(int H, int W, int N, const float *us, const float *cinv2ds, const float *alphas,
                      float *depths, const float *colors, int32_t *areas, const void *packed_records,
                      int64_t P_cap, uint32_t depth_key_cap, void *bin_ws, size_t bin_ws_bytes, void *ws,
                      size_t ws_bytes, float *image, int32_t *contrib, float *final_tau,
                      int32_t *patch_range_per_tile, int32_t *gsid_per_patch, uint32_t *status_host,
                      gsb_stream_t stream) {
  return splat_forward_impl(H, W, N, us, cinv2ds, alphas, depths, colors, areas, packed_records, P_cap, depth_key_cap,
                            bin_ws, bin_ws_bytes, ws, ws_bytes, image, contrib, final_tau, patch_range_per_tile,
                            gsid_per_patch, status_host, stream, true);
}

int gsb_splat_forward_enqueue(int H, int W, int N, const float *us, const float *cinv2ds, const float *alphas,
                              float *depths, const float *colors, int32_t *areas, const void *packed_records,
                              int64_t P_cap, uint32_t depth_key_cap, void *bin_ws, size_t bin_ws_bytes, void *ws,
                              size_t ws_bytes, float *image, int32_t *contrib, float *final_tau,
                              int32_t *patch_range_per_tile, int32_t *gsid_per_patch, uint32_t *status_host,
                              gsb_stream_t stream) {
  return splat_forward_impl(H, W, N, us, cinv2ds, alphas, depths, colors, areas, packed_records, P_cap, depth_key_cap,
                            bin_ws, bin_ws_bytes, ws, ws_bytes, image, contrib, final_tau, patch_range_per_tile,
                            gsid_per_patch, status_host, stream, false);
}

size_t gsb_splat_backward_workspace_bytes(int N, int H, int W, int64_t P) {
  // per-Gaussian records (256-B aligned; only when they have to be rebuilt, P > 0) + the [N,9]
  // moment accumulators
  const size_t T = (size_t)((W + GSB_TILE - 1) / GSB_TILE) * (size_t)((H + GSB_TILE - 1) / GSB_TILE);
  return (size_t)(P > 0 && N > 0 ? N : 1) * sizeof(Rec) + 512 + (size_t)(N > 0 ? N : 1) * 9 * sizeof(float) + 512 +
         (4 * T + 2) * sizeof(int);  // + the rasterizer's work area
}

int gsb_splat_backward(int H, int W, int N, int64_t P, const float *us, const float *cinv2ds,
                       const float *alphas, const float *colors, const int32_t *contrib,
                       const float *final_tau, const int32_t *patch_range_per_tile,
                       const int32_t *gsid_per_patch, const float *dloss_dgammas,
                       const void *packed_records, void *ws, size_t ws_bytes, float *dloss_dus, float *dloss_dcinv2ds, float *dloss_dalphas,
                       float *dloss_dcolors, float *moments_out, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0 && H > 0 && W > 0 && P >= 0, "splatB: bad N/H/W/P");
  GSB_REQUIRE(N == 0 || moments_out || (dloss_dus && dloss_dcinv2ds && dloss_dalphas && dloss_dcolors),
              "splatB: null output");
  cudaStream_t st = (cudaStream_t)stream;
  if (N == 0) return 0;
  GSB_REQUIRE(cinv2ds && ws, "splatB: null pointer");
  // with the forward's records handed in, the workspace only has to hold the moment rows
  const int64_t P_ws = packed_records != nullptr ? 0 : P;
  GSB_REQUIRE(ws_bytes >= gsb_splat_backward_workspace_bytes(N, H, W, P_ws), "splatB: workspace too small");
  // workspace: [records, 256-B aligned (cp.async.bulk needs 16 B)] [moment rows]
  uintptr_t base = (reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255;
  Rec *recs = reinterpret_cast<Rec *>(base);
  uintptr_t mbase = (base + (size_t)(P_ws > 0 ? N : 1) * sizeof(Rec) + 255) & ~(uintptr_t)255;
  float *moments = moments_out != nullptr ? moments_out : reinterpret_cast<float *>(mbase);
  int *work = reinterpret_cast<int *>((mbase + (size_t)N * 9 * sizeof(float) + 255) & ~(uintptr_t)255);
  if (P > 0) {
    GSB_REQUIRE(us && alphas && colors && contrib && final_tau && patch_range_per_tile && gsid_per_patch &&
                    dloss_dgammas,
                "splatB: null pointer");
    if (packed_records != nullptr) {  // the forward's record stream is still valid: skip the re-pack
      GSB_REQUIRE((reinterpret_cast<uintptr_t>(packed_records) & 15) == 0, "splatB: packed_records misaligned");
      recs = const_cast<Rec *>(static_cast<const Rec *>(packed_records));
    } else {
      int rc = launch_pack_only(N, nullptr, us, cinv2ds, alphas, colors, recs, st);
      if (rc) return rc;
    }
  }
  // P == 0: nothing was drawn; the zeroed moment rows finalise to all-zero gradients
  return launch_draw_backward(H, W, N, patch_range_per_tile, P > 0 ? recs : nullptr, gsid_per_patch, contrib, final_tau,
                              dloss_dgammas, cinv2ds, moments, work, dloss_dus, dloss_dcinv2ds, dloss_dalphas,
                              dloss_dcolors, moments_out == nullptr, st);
}

// ---- density control + record conversion (density.cu)

static bool gau_complete(const gsb_gaussians *g) {
  return g && g->pws && g->low_shs && g->high_shs && g->alphas_raw && g->scales_raw && g->rots_raw;
}
static float *const *gau_ptrs(const gsb_gaussians *g) {
  // six consecutive float* members: the struct IS the pointer table the launchers index
  static_assert(sizeof(gsb_gaussians) == 6 * sizeof(float *), "gsb_gaussians layout");
  return reinterpret_cast<float *const *>(g);
}

int gsb_density_accumulate(int64_t N, const float *dloss_dus, const uint8_t *mask, float *grad_accum,
                           int32_t *cunt, int first, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0, "density_accumulate: N < 0");
  GSB_REQUIRE(N == 0 || (dloss_dus && mask && grad_accum && cunt), "density_accumulate: null pointer");
  return launch_density_accumulate(N, dloss_dus, mask, grad_accum, cunt, first, (cudaStream_t)stream);
}

size_t gsb_density_workspace_bytes(int64_t N) { return density_workspace_bytes(N); }

int gsb_density_plan(int64_t N, const float *alphas_raw, const float *scales_raw, const float *grad_accum,
                     const int32_t *cunt, float alpha_raw_min, float scale_raw_max, float grad_min,
                     float scale_clone_max, void *ws, size_t ws_bytes, uint8_t *cls, int32_t *slots,
                     int64_t *counts_host, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0 && N < ((int64_t)1 << 31), "density_plan: N out of range");
  GSB_REQUIRE(counts_host != nullptr, "density_plan: counts_host is null");
  GSB_REQUIRE(N == 0 || (alphas_raw && scales_raw && grad_accum && cunt && ws && cls && slots),
              "density_plan: null pointer");
  GSB_REQUIRE(N == 0 || ws_bytes >= density_workspace_bytes(N), "density_plan: workspace too small");
  return launch_density_plan(N, alphas_raw, scales_raw, grad_accum, cunt, alpha_raw_min, scale_raw_max, grad_min,
                             scale_clone_max, ws, ws_bytes, cls, slots, counts_host, (cudaStream_t)stream);
}

int gsb_density_apply(int64_t N, const uint8_t *cls, const int32_t *slots, int64_t K, int64_t C, int64_t S,
                      const gsb_gaussians *src, const gsb_gaussians *src_m, const gsb_gaussians *src_v,
                      const float *z, const gsb_gaussians *dst, const gsb_gaussians *dst_m,
                      const gsb_gaussians *dst_v, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0 && K >= 0 && C >= 0 && S >= 0 && K <= N && C + S <= K, "density_apply: bad counts");
  if (N == 0) return 0;
  GSB_REQUIRE(cls && slots, "density_apply: null plan");
  GSB_REQUIRE(gau_complete(src), "density_apply: src has a null tensor");
  GSB_REQUIRE(K + C + S == 0 || gau_complete(dst), "density_apply: dst has a null tensor");
  const bool state = src_m != nullptr;
  GSB_REQUIRE((src_v != nullptr) == state && (dst_m != nullptr) == state && (dst_v != nullptr) == state,
              "density_apply: Adam moments must be all given or all NULL");
  if (state)
    GSB_REQUIRE(gau_complete(src_m) && gau_complete(src_v) && (K + C + S == 0 || (gau_complete(dst_m) && gau_complete(dst_v))),
                "density_apply: a moment tensor is null");
  GSB_REQUIRE(S == 0 || z != nullptr, "density_apply: z is null");
  if (K + C + S == 0) return 0;
  return launch_density_apply(N, cls, slots, K, C, gau_ptrs(src), state ? gau_ptrs(src_m) : nullptr,
                              state ? gau_ptrs(src_v) : nullptr, z, gau_ptrs(dst), state ? gau_ptrs(dst_m) : nullptr,
                              state ? gau_ptrs(dst_v) : nullptr, (cudaStream_t)stream);
}

int gsb_reset_alpha(int64_t N, float *alphas_raw, float *exp_avg, float *exp_avg_sq, float reset_raw,
                    gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0, "reset_alpha: N < 0");
  GSB_REQUIRE(N == 0 || alphas_raw, "reset_alpha: null pointer");
  return launch_reset_alpha(N, alphas_raw, exp_avg, exp_avg_sq, reset_raw, (cudaStream_t)stream);
}

static bool sh_dim_ok(int d) { return d == 3 || d == 12 || d == 27 || d == 48; }

int gsb_ply_rows_to_gs(int64_t N, int stride, int sh_dim, const float *rows, const int32_t *colmap,
                       float *gs_rows, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0 && sh_dim_ok(sh_dim), "ply_rows_to_gs: sh_dim must be 3, 12, 27 or 48");
  GSB_REQUIRE(stride >= 11 + sh_dim, "ply_rows_to_gs: row stride smaller than 11 + sh_dim");
  GSB_REQUIRE(N == 0 || (rows && colmap && gs_rows), "ply_rows_to_gs: null pointer");
  return launch_ply_rows_to_gs(N, stride, sh_dim, rows, colmap, gs_rows, (cudaStream_t)stream);
}

int gsb_gs_to_params(int64_t N, int sh_dim, const float *gs_rows, const gsb_gaussians *dst, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0 && sh_dim_ok(sh_dim), "gs_to_params: sh_dim must be 3, 12, 27 or 48");
  GSB_REQUIRE(N == 0 || (gs_rows && gau_complete(dst)), "gs_to_params: null pointer");
  if (N == 0) return 0;
  return launch_gs_to_params(N, sh_dim, gs_rows, gau_ptrs(dst), (cudaStream_t)stream);
}

int gsb_params_to_gs(int64_t N, const gsb_gaussians *src, float *gs_rows, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0, "params_to_gs: N < 0");
  GSB_REQUIRE(N == 0 || (gs_rows && gau_complete(src)), "params_to_gs: null pointer");
  if (N == 0) return 0;
  return launch_params_to_gs(N, gau_ptrs(src), gs_rows, (cudaStream_t)stream);
}

// ---- multi-GPU gradient exchange (comm.cu, fused.cu PUSH variant)

size_t gsb_exchange_region_bytes(int N, int sh_dim3, int world) {
  if (N < 0 || world < 1 || world > kMaxWorld) return 0;
  return exchange_geom(N, sh_dim3, world).bytes;
}

size_t gsb_exchange_result_offset(int N, int sh_dim3, int world, int segment) {
  if (segment < 0 || segment > 4 || world < 1 || world > kMaxWorld) return 0;
  const ExchangeGeom G = exchange_geom(N, sh_dim3, world);
  return G.result_base + (size_t)G.result_off[segment] * sizeof(float);
}

int gsb_comm_alloc(size_t bytes, void **ptr, void *handle_out) {
  GSB_REQUIRE(ptr && handle_out && bytes > 0, "comm_alloc: bad arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) == GSB_COMM_HANDLE_BYTES, "IPC handle size");
  GSB_CUDA_TRY(cudaMalloc(ptr, bytes));
  GSB_CUDA_TRY(cudaMemset(*ptr, 0, bytes));
  GSB_CUDA_TRY(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  GSB_CUDA_TRY(cudaIpcGetMemHandle(&h, *ptr));
  memcpy(handle_out, &h, sizeof(h));
  return 0;
}

int gsb_comm_open(const void *handle, void **peer_ptr) {
  GSB_REQUIRE(handle && peer_ptr, "comm_open: bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  GSB_CUDA_TRY(cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}

int gsb_comm_close(void *peer_ptr) {
  if (peer_ptr) GSB_CUDA_TRY(cudaIpcCloseMemHandle(peer_ptr));
  return 0;
}

int gsb_comm_free(void *ptr) {
  if (ptr) GSB_CUDA_TRY(cudaFree(ptr));
  return 0;
}

int gsb_exchange_status(const void *region, int *status_host) {
  GSB_REQUIRE(region && status_host, "exchange_status: bad arguments");
  uint32_t v = 0;
  GSB_CUDA_TRY(cudaMemcpy(&v, static_cast<const char *>(region) + 136, sizeof(v), cudaMemcpyDeviceToHost));
  *status_host = (int)v;
  return 0;
}

int gsb_preprocess_backward_push(int N, int sh_dim3, const float *pws, const float *rots, const float *scales,
                                 const float *shs, const float *Rcw, const float *tcw, const float *twc,
                                 float fx, float fy, float cx, float cy, float width, float height,
                                 const float *dloss_dus, const float *dloss_dcinv2ds, const float *dloss_dcolors,
                                 const float *dloss_dalphas, const float *moments, const float *cinv2ds,
                                 float *dloss_dus_out, int world, int rank, void *const *regions_host,
                                 uint32_t epoch, gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0, "preprocess_backward_push: N < 0");
  GSB_REQUIRE(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world && regions_host && epoch != 0,
              "preprocess_backward_push: bad world / rank / regions / epoch");
  GSB_REQUIRE(N == 0 || (pws && rots && scales && shs && Rcw && tcw && twc), "preprocess_backward_push: null pointer");
  GSB_REQUIRE(N == 0 || (moments ? (cinv2ds && dloss_dus_out)
                                 : (dloss_dus && dloss_dcinv2ds && dloss_dcolors && dloss_dalphas)),
              "preprocess_backward_push: null upstream gradient");
  const ExchangeGeom G = exchange_geom(N, sh_dim3, world);
  GradPush gp{};
  for (int p = 0; p < world; p++) {
    GSB_REQUIRE(regions_host[p] != nullptr, "preprocess_backward_push: null region");
    char *r = static_cast<char *>(regions_host[p]);
    gp.slot[p] = reinterpret_cast<float *>(r + G.staging_off) + (size_t)rank * G.slot_floats;
    gp.flags[p] = reinterpret_cast<uint32_t *>(r);
  }
  gp.counter = reinterpret_cast<uint32_t *>(static_cast<char *>(regions_host[rank]) + 128);
  gp.g_alphas = dloss_dalphas;
  gp.off_rots = G.slot_off[1];
  gp.off_pws = G.slot_off[2];
  gp.off_scales = G.slot_off[3];
  gp.off_alphas = G.slot_off[4];
  gp.world = world;
  gp.rank = rank;
  gp.epoch = epoch;
  const MomentsIn mi{moments, cinv2ds, dloss_dus_out, nullptr};
  return launch_preprocess_bwd_push(N, sh_dim3, pws, rots, scales, shs, Rcw, tcw, twc, fx, fy, cx, cy, width, height,
                                    dloss_dus, dloss_dcinv2ds, dloss_dcolors, gp, moments ? &mi : nullptr,
                                    (cudaStream_t)stream);
}

int gsb_grad_reduce_broadcast(int N, int sh_dim3, int world, int rank, void *const *regions_host, uint32_t epoch,
                              gsb_stream_t stream) {
  GSB_REQUIRE(N >= 0 && world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world && regions_host && epoch != 0,
              "grad_reduce_broadcast: bad arguments");
  for (int p = 0; p < world; p++) GSB_REQUIRE(regions_host[p] != nullptr, "grad_reduce_broadcast: null region");
  const ExchangeGeom G = exchange_geom(N, sh_dim3, world);
  return launch_grad_reduce_bcast(G, rank, regions_host, epoch, (cudaStream_t)stream);
}

}  // extern "C"
