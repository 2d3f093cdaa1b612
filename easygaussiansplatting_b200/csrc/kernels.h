// Internal launcher prototypes (host side, C++).  The public surface is include/gsplat_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace gsb {

struct Rec;

// ---- launch accounting / optional per-kernel CUDA-event timing (api.cu).  Every launcher
// opens a ProfScope; the launch counter always runs, events are recorded only while
// gsb_profile_enable(1) is in effect (bench.py's roofline leg).
enum KernelId {
  K_PROJECT = 0, K_COV3D, K_COV2D, K_SH2COLOR, K_INVCOV, K_RECTS, K_SCAN, K_KEYS, K_SORT, K_RANGES,
  K_PACK, K_DRAW, K_DRAW_BWD, K_PRE_FWD, K_PRE_BWD, K_FINALIZE, K_LOSS_FWD, K_LOSS_BWD, K_BMM,
  K_DENSITY_ACC, K_DENSITY_CLASSIFY, K_DENSITY_SCAN, K_DENSITY_APPLY, K_RESET_ALPHA, K_GS_DECODE,
  K_GS_TO_PARAMS, K_PARAMS_TO_GS, K_GRAD_EXCHANGE, K_SH_EXPAND, K_COUNT
};
struct ProfScope {
  ProfScope(int id, cudaStream_t st);
  ~ProfScope();
  int id_;
  cudaStream_t st_;
  cudaEvent_t stop_;
};

int launch_project(int N, const float *pws, const float *Rcw, const float *tcw, float fx, float fy,
                   float cx, float cy, float *us, float *pcs, float *depths, float *du_dpcs,
                   cudaStream_t st);
int launch_cov3d(int N, const float *rots, const float *scales, const float *depths, float *cov3ds,
                 float *Jr, float *Js, cudaStream_t st);
int launch_cov2d(int N, const float *cov3ds, const float *pcs, const float *Rcw, const float *depths,
                 float fx, float fy, float width, float height, float *cov2ds, float *Jc, float *Jp,
                 cudaStream_t st);
int launch_sh2color(int N, int k3, const float *shs, const float *pws, const float *twc, float *colors,
                    float *Js, float *Jp, cudaStream_t st);
int launch_inv_cov2d(int N, const float *cov2ds, float *depths, float *cinv2ds, int32_t *areas,
                     float *J, cudaStream_t st);

// ---- fused per-Gaussian path (fused.cu)
int launch_preprocess_fwd(int N, int k3, const float *pws, const float *rots, const float *scales,
                          const float *shs, const float *Rcw, const float *tcw, const float *twc, float fx,
                          float fy, float cx, float cy, float width, float height, float *us, float *cinv2ds,
                          float *colors, float *depths, int32_t *areas, const float *alphas, Rec *recs,
                          cudaStream_t st);
// upstream gradients given as the rasterizer backward's moment rows (fused.cu, MOM variants)
struct MomentsIn {
  const float *moments;  // [N,9]
  const float *cinv2ds;  // [N,3]
  float *dus_out;        // [N,2]  dL/du, still needed by the caller
  float *dalphas_out;    // [N]    dL/dalpha (nullable: the push variant forwards it instead)
};
int launch_preprocess_bwd(int N, int k3, const float *pws, const float *rots, const float *scales,
                          const float *shs, const float *Rcw, const float *tcw, const float *twc, float fx,
                          float fy, float cx, float cy, float width, float height, const float *g_us,
                          const float *g_cinv2ds, const float *g_colors, float *g_pws, float *g_shs,
                          float *g_scales, float *g_rots, const MomentsIn *mi, cudaStream_t st);

// dL/dsh[N,3k] = sum over V views of Y(dir_v) (x) dL/dcolor_v  (fused.cu k_sh_expand)
int launch_sh_expand(int N, int k3, int V, const float *pws, const float *twcs, const float *gcols, float *g_shs,
                     cudaStream_t st);

// ---- multi-GPU gradient exchange (comm.cu; the producer is the PUSH variant in fused.cu).
// Every rank owns one region of peer-mapped memory:
//   [control 4 KiB: arrive[8] u32 @0, done[8] u32 @64, counters @128/@132, status @136]
//   [staging: world slots x (rpr rows x (ks+11) floats), slot s = what rank s pushed here]
//   [result:  world*rpr rows x (ks+11) floats, the summed gradients, identical on every rank]
// Tiles of 128 Gaussians are dealt round-robin: rank r owns global tiles r, r + world, ...
// (local tile lt <-> global tile lt * world + r), rpr = tiles_per_rank * 128 rows per rank;
// slot and result keep the SoA segment order shs | rots | pws | scales | alphas.
constexpr int kMaxWorld = 8;
constexpr size_t kCtrlBytes = 4096;
struct ExchangeGeom {
  int world, ks, tiles_per_rank;
  long long rpr, rows_total, slot_floats;
  long long slot_off[5], result_off[5];  // float offsets of the 5 segments inside a slot / the result
  int seg_k[5];
  size_t staging_off, result_base, bytes;  // byte offsets inside the region
};
ExchangeGeom exchange_geom(int N, int k3, int world);
struct GradPush {
  float *slot[kMaxWorld];      // staging slot `rank` on each owner
  uint32_t *flags[kMaxWorld];  // arrive[] array of each rank
  uint32_t *counter;
  const float *g_alphas;       // dL/dalpha of this view (unused when the moment rows are given)
  long long off_rots, off_pws, off_scales, off_alphas;  // float offsets of the segments inside a slot
  int world, rank;
  uint32_t epoch;
};
int launch_preprocess_bwd_push(int N, int k3, const float *pws, const float *rots, const float *scales,
                               const float *shs, const float *Rcw, const float *tcw, const float *twc, float fx,
                               float fy, float cx, float cy, float width, float height, const float *g_us,
                               const float *g_cinv2ds, const float *g_colors, const GradPush &gp,
                               const MomentsIn *mi, cudaStream_t st);
int launch_grad_reduce_bcast(const ExchangeGeom &G, int rank, void *const *regions, uint32_t epoch,
                             cudaStream_t st);

// ---- batched tiny matmul for the reference's Jacobian chain (smallbmm.cu)
int launch_small_bmm(long long batch, int M, int K, int NN, const float *A, const float *B, int b_shared,
                     float *C, cudaStream_t st);

// ---- fused training loss (loss.cu)
size_t gau_loss_workspace_bytes(int H, int W);
int launch_gau_loss(int H, int W, const float *img, const float *gt, float lambda, float *loss_out,
                    float *grad, void *ws, cudaStream_t st);

// ---- density control + Gaussian record conversion (density.cu).  Tensor order everywhere:
// pws, low_shs, high_shs, alphas_raw, scales_raw, rots_raw (widths 3, 3, 45, 1, 3, 4).
size_t density_workspace_bytes(int64_t N);
int launch_density_accumulate(int64_t N, const float *dloss_dus, const uint8_t *mask, float *grad_accum,
                              int32_t *cunt, int init, cudaStream_t st);
int launch_density_plan(int64_t N, const float *alphas_raw, const float *scales_raw, const float *grad_accum,
                        const int32_t *cunt, float alpha_raw_min, float scale_raw_max, float grad_min,
                        float scale_clone_max, void *ws, size_t ws_bytes, uint8_t *cls, int32_t *slots,
                        int64_t *counts_host, cudaStream_t st);
int launch_density_apply(int64_t N, const uint8_t *cls, const int32_t *slots, int64_t K, int64_t C,
                         float *const *src, float *const *src_m, float *const *src_v, const float *z,
                         float *const *dst, float *const *dst_m, float *const *dst_v, cudaStream_t st);
int launch_reset_alpha(int64_t N, float *alphas_raw, float *m, float *v, float val, cudaStream_t st);
int launch_ply_rows_to_gs(int64_t N, int stride, int sh_dim, const float *rows, const int32_t *colmap, float *gs,
                          cudaStream_t st);
int launch_gs_to_params(int64_t N, int sh_dim, const float *gs, float *const *dst, cudaStream_t st);
int launch_params_to_gs(int64_t N, float *const *src, float *gs, cudaStream_t st);

// ---- binning (binning.cu)
struct BinLayout {  // carve-up of the phase-1 workspace
  size_t rects, offsets, total, scan_desc, bytes;  // total: [P, max depth key, flags, scan claim] u32
};
BinLayout bin_layout(int N);
int launch_bin(int H, int W, int N, const float *us, float *depths, int32_t *areas, void *ws,
               const BinLayout &L, cudaStream_t st);

struct SortLayout {  // carve-up of the phase-2 workspace
  size_t keys_a, keys_b, vals_a, vals_b, recs, counters;
  size_t sort_state, sort_state_bytes, hist, desc, desc_stride;  // radix-sort state, zeroed per call
  size_t bytes;
};
int sort_layout(int N, int H, int W, int64_t P, SortLayout *out);
// capacity-based path: where to copy [P, max depth key, flags] for the host, and the event that
// tells it the copy has landed (recorded right after the key kernel)
struct StatusRead {
  uint32_t *host;
  cudaEvent_t ready;
};
int launch_sort_and_pack(int H, int W, int N, int64_t P, uint32_t depth_key_max, const float *us,
                         const float *cinv2ds, const float *alphas, const float *depths, const float *colors,
                         const void *bin_ws, const BinLayout &BL, void *ws, const SortLayout &SL,
                         int32_t *ranges, int32_t *gsid_per_patch, bool pack, const StatusRead *sr,
                         cudaStream_t st);
int launch_pack_only(int64_t P, const int32_t *gsid_per_patch, const float *us, const float *cinv2ds,
                     const float *alphas, const float *colors, Rec *recs, cudaStream_t st);

// ---- rasterizer (raster_fwd3.cu, raster_bwd4.cu + raster_bwd.cu).  recs: one 48-byte record per
// Gaussian; gsid: the sorted patch list -- every warp gathers the records of its tile's list itself.
// work_counter: the work area of k_tile_list (below), which both rasterizers pull their items from.
int launch_draw_bwd4_kernel(int H, int W, const int32_t *ranges, const Rec *recs, const int32_t *gsid,
                            const int32_t *contrib, const float *final_tau, const float *dloss_dgammas,
                            float *moments, int *work_counter, cudaStream_t st);
// work = [item counter, #entries, entries ...] (2 + 4 * tiles ints, see k_tile_list); with outputs given the
// empty tiles are zero-filled here
int launch_tile_list(int H, int W, const int32_t *ranges, float *image, int32_t *contrib, float *final_tau,
                     int *work, cudaStream_t st);
int launch_draw(int H, int W, const int32_t *ranges, const Rec *recs, const int32_t *gsid, float *image,
                int32_t *contrib, float *final_tau, int *work_counter, cudaStream_t st);
int launch_draw_backward(int H, int W, int N, const int32_t *ranges, const Rec *recs, const int32_t *gsid,
                         const int32_t *contrib,
                         const float *final_tau, const float *dloss_dgammas, const float *cinv2ds,
                         float *moments, int *work_counter, float *dloss_dus,
                         float *dloss_dcinv2ds, float *dloss_dalphas, float *dloss_dcolors, bool finalize,
                         cudaStream_t st);

}  // namespace gsb
