// Forward tile rasterizer, variant 3: warp-autonomous blocks + list-driven two-record loop (the
// structure of the backward kernel, raster_bwd4.cu).
//
// A work item is one 8x8 pixel block of a 16x16 tile (reference BLOCK); every warp of the
// persistent grid pulls items from a global counter and streams the tile's record list itself:
// 32-record chunks, lane j gathers the 48-byte record of patch 32 c + j with three 16-byte
// cp.async (double buffered, cp.async groups + __syncwarp -- no CTA barrier anywhere), tests it
// against the block (rec_can_touch: exact, so image / contrib / final_tau are unaffected), and the
// surviving records go into a small shared-memory list that the compositing loop walks two at a
// time (two independent alpha' chains in flight per warp).  A lane owns two horizontally adjacent
// pixels; the quadratic form, the alpha multiply and the compositing update are packed f32x2.
// f3_alpha is the operation sequence of the backward's b4_eval (raster_bwd4.cu), so forward and
// backward compute bit-identical alpha' and take the same skip decisions.
// Replaces reference kernel.cu:152-271 (draw).
#include "common.cuh"
#include "kernels.h"

namespace gsb {

constexpr int F3_RING = 2;  // 32-record chunks in flight per warp
constexpr int F3_CHUNK_BYTES = 32 * 48;
#ifndef FWD3_MINBLOCKS
#define FWD3_MINBLOCKS 8
#endif

namespace {
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ uint4 lds128u(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts64u(uint32_t a, uint32_t x, uint32_t y) {
  asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void cp_async16_sa(uint32_t dst, const void *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ uint32_t opaque_u32(uint32_t x) {  // keep an address in a register
  uint32_t y;
  asm volatile("mov.u32 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}
__device__ __forceinline__ float2 p2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 p2s(float a) { return make_float2(a, a); }

// alpha' = min(0.99, alpha * exp2(a dx^2 + b dx dy + c dy^2)) at the lane's two pixels
// (kernel.cu:236-245; same operation sequence as alpha_prime() in common.cuh)
__device__ __forceinline__ float2 f3_alpha(const float4 &q0, const float4 &q1, const float2 &npx, float fpy) {
  const float2 dx = __fadd2_rn(p2s(q0.x), npx);
  const float dy = q0.y - fpy;
  const float cdy2 = (q1.z * dy) * dy;
  const float2 t = __ffma2_rn(p2s(q1.y), p2s(dy), __fmul2_rn(p2s(q1.x), dx));
  const float2 p = __ffma2_rn(t, dx, p2s(cdy2));
  const float2 ag = __fmul2_rn(p2s(q0.w), p2(ex2_approx(fminf(p.x, 0.0f)), ex2_approx(fminf(p.y, 0.0f))));
  return p2(fminf(ALPHA_CLAMP, ag.x), fminf(ALPHA_CLAMP, ag.y));
}
}  // namespace

// Work list of the two rasterizers (work[0] = the kernels' item counter, work[1] = number of
// entries, work[2..] = entries): a tile with more than 32 patches contributes four entries
// `tile * 8 + block` (one 8x8 block each), a tile with 1..32 patches ONE entry `tile * 8 + 4` --
// the warp that pulls it gathers the tile's single chunk of records once and renders all four
// blocks from it (a block of a sparse tile is bounded by the latency of its queue pull, range
// load, id load and gather, not by work: this quarters them).  A tile without patches keeps
// image 0, contrib 0, tau 0 (kernel.cu:182-183): when outputs are given this pass writes those
// zeros itself with 16-byte stores -- one warp per empty tile -- so the sparse corner of BASELINE config 4
// (50k Gaussians at 4K: 32 400 tiles, most of them empty) costs one streaming pass over the
// frame instead of one queue item per 8x8 block.
__global__ void __launch_bounds__(256) k_tile_list(int W, int H, int gx, int T, const int2 *__restrict__ ranges,
                                                   float *__restrict__ image, int32_t *__restrict__ contrib,
                                                   float *__restrict__ final_tau, int *__restrict__ work) {
  __shared__ unsigned s_empty[8];  // per warp: which of its 32 tiles have no patches
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tile = blockIdx.x * 256 + threadIdx.x;  // phase 1: one thread per tile
  int len = 0;
  if (tile < T) {
    const int2 r = __ldg(ranges + tile);
    len = r.y - r.x;
  }
  const bool has = len > 0;
  const int n_ent = !has ? 0 : (len <= 32 ? 1 : 4);
  int incl = n_ent;  // warp prefix sum of the entry counts -> one atomic per 32 tiles
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const unsigned m = __ballot_sync(0xffffffffu, has);
  int base = 0;
  if (lane == 31 && incl) base = atomicAdd(work + 1, incl);
  base = __shfl_sync(0xffffffffu, base, 31) + incl - n_ent;
  if (n_ent == 1) work[2 + base] = tile * 8 + 4;
  if (n_ent == 4) {
#pragma unroll
    for (int b = 0; b < 4; b++) work[2 + base + b] = tile * 8 + b;
  }
  if (image == nullptr) return;
  if (lane == 0) s_empty[warp] = ~m;
  __syncthreads();
  // phase 2: the CTA's empty tiles, one warp per tile, 16-byte stores
  const size_t HW = (size_t)H * W;
  for (int w = 0; w < 8; w++) {
    unsigned e = s_empty[w];
    // warp `warp` takes every 8th empty tile of the CTA's list; simple static split
    for (int k = 0; e; k++) {
      const int bit = __ffs(e) - 1;
      e &= e - 1;
      if ((k & 7) != warp) continue;
      const int t = blockIdx.x * 256 + w * 32 + bit;
      if (t >= T) break;
      const int x0 = (t % gx) * TILE + (lane & 1) * 8, y = (t / gx) * TILE + (lane >> 1);
      if (y >= H || x0 >= W) continue;
      const size_t pix = (size_t)y * W + x0;
      if ((W & 3) == 0 && x0 + 8 <= W) {  // 8 pixels = two 16-byte stores per plane
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int h = 0; h < 2; h++) {
          *reinterpret_cast<float4 *>(image + pix + 4 * h) = z;
          *reinterpret_cast<float4 *>(image + HW + pix + 4 * h) = z;
          *reinterpret_cast<float4 *>(image + 2 * HW + pix + 4 * h) = z;
          *reinterpret_cast<int4 *>(contrib + pix + 4 * h) = make_int4(0, 0, 0, 0);
          *reinterpret_cast<float4 *>(final_tau + pix + 4 * h) = z;
        }
      } else {
        for (int x = x0; x < min(x0 + 8, W); x++) {
          const size_t q = (size_t)y * W + x;
          image[q] = 0.f; image[HW + q] = 0.f; image[2 * HW + q] = 0.f;
          contrib[q] = 0; final_tau[q] = 0.f;
        }
      }
    }
  }
}

int launch_tile_list(int H, int W, const int32_t *ranges, float *image, int32_t *contrib, float *final_tau,
                     int *work, cudaStream_t st) {
  const int gx = (W + TILE - 1) / TILE, gy = (H + TILE - 1) / TILE;
  const int T = gx * gy;
  GSB_CUDA_TRY(cudaMemsetAsync(work, 0, 2 * sizeof(int), st));
  k_tile_list<<<(T + 255) / 256, 256, 0, st>>>(W, H, gx, T, reinterpret_cast<const int2 *>(ranges), image, contrib,
                                           final_tau, work);
  GSB_CUDA_TRY(cudaGetLastError());
  return 0;
}

__global__ void __launch_bounds__(128, FWD3_MINBLOCKS) k_draw3(int W, int H, int gx, int T,
                                                               const int2 *__restrict__ ranges,
                                                               const Rec *__restrict__ recs,
                                                               const int32_t *__restrict__ gsid,
                                                               float *__restrict__ image,
                                                               int32_t *__restrict__ contrib,
                                                               float *__restrict__ final_tau,
                                                               int *__restrict__ work) {
  __shared__ __align__(16) unsigned char s_ring[4][F3_RING * F3_CHUNK_BYTES];  // gathered records, per warp
  __shared__ __align__(16) uint2 s_list[4][34];  // (record address, patch index + 1) of a chunk's survivors
  __shared__ __align__(16) Rec s_dummy;          // all-zero record (alpha = 0): pads an odd survivor count

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t HW = (size_t)H * W;
  const bool vec2 = (W & 1) == 0;  // pixel pairs are 8-byte aligned in every plane
  const uint32_t ring_addr = opaque_u32(smem_u32(&s_ring[warp][0]));
  const uint32_t list_addr = opaque_u32(smem_u32(&s_list[warp][0]));
  const uint32_t dummy_addr = smem_u32(&s_dummy);
  if (threadIdx.x < 12) reinterpret_cast<float *>(&s_dummy)[threadIdx.x] = 0.0f;
  __syncthreads();  // (the only CTA-wide barrier: start-up)
  (void)T;
  const int items = work[1];  // entries of the work list (k_tile_list)
  const int *__restrict__ entries = work + 2;

  for (;;) {
    int item = 0;
    if (lane == 0) item = atomicAdd(work, 1);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= items) break;
    const int ent = __ldg(entries + item);
    const int tile = ent >> 3, code = ent & 7;
    const bool whole_tile = code == 4;  // <= 32 patches: this warp renders all four blocks from one gather
    const int2 range = __ldg(ranges + tile);
    const int len = range.y - range.x;
    if (whole_tile) {  // the tile's single chunk, gathered once (two groups: see the wait below)
      if (lane < len) {
        const char *src = reinterpret_cast<const char *>(recs + __ldg(gsid + range.x + lane));
        const uint32_t dst = ring_addr + lane * 48;
        cp_async16_sa(dst, src);
        cp_async16_sa(dst + 16, src + 16);
        cp_async16_sa(dst + 32, src + 32);
      }
      cp_async_commit();
      cp_async_commit();
    }
   for (int blk = whole_tile ? 0 : code; blk < (whole_tile ? 4 : code + 1); blk++) {
    const int tx = tile % gx, ty = tile / gx;
    const int rx0 = tx * TILE + (blk & 1) * 8, ry0 = ty * TILE + (blk >> 1) * 8;
    if (rx0 >= W || ry0 >= H) continue;  // block entirely outside the image
    const int px = rx0 + 2 * (lane & 3), py = ry0 + (lane >> 2);
    const bool in0 = px < W && py < H, in1 = px + 1 < W && py < H;
    const size_t pix = (size_t)py * W + px;

    float2 tau = p2s(0.f), cr = p2s(0.f), cg = p2s(0.f), cb = p2s(0.f);
    int cont0 = 0, cont1 = 0;
    if (len > 0) {  // (a tile without patches keeps image 0, contrib 0, tau 0: kernel.cu:182-183)
      const int nch = (len + 31) >> 5;
      const int32_t *ids = gsid + range.x;
      auto issue = [&](int c, int id) {
        if (c < nch && c * 32 + lane < len) {
          const char *src = reinterpret_cast<const char *>(recs + id);
          const uint32_t dst = ring_addr + (c & (F3_RING - 1)) * F3_CHUNK_BYTES + lane * 48;
          cp_async16_sa(dst, src);
          cp_async16_sa(dst + 16, src + 16);
          cp_async16_sa(dst + 32, src + 32);
        }
        cp_async_commit();
      };
      auto load_id = [&](int c) { return (c < nch && c * 32 + lane < len) ? __ldg(ids + c * 32 + lane) : 0; };
      int id_next = 0;
      if (!whole_tile) {
#pragma unroll
        for (int r = 0; r < F3_RING; r++) issue(r, load_id(r));
        id_next = load_id(F3_RING);
      }

      const float2 npx = p2(-(float)px, -(float)(px + 1));
      const float fpy = (float)py;
      const float bx0 = (float)rx0, bx1 = (float)(rx0 + 7), by0 = (float)ry0, by1 = (float)(ry0 + 7);
      // a pixel is finished exactly when tau < 1e-4; pixels outside the image start finished
      tau = p2(in0 ? 1.0f : 0.0f, in1 ? 1.0f : 0.0f);

      for (int c = 0; c < nch; c++) {
        cp_async_wait<F3_RING - 1>();  // this lane's copy of chunk c has landed ...
        __syncwarp();                  // ... and so have the other lanes'
        const uint32_t my_rec = ring_addr + (c & (F3_RING - 1)) * F3_CHUNK_BYTES + lane * 48;
        const int my_idx = c * 32 + lane;
        bool hit = false;
        if (my_idx < len) hit = rec_can_touch(lds128(my_rec), lds128(my_rec + 16), bx0, bx1, by0, by1);
        // survivors of the chunk, front to back, as a list of (record address, patch index + 1)
        const unsigned mask = __ballot_sync(0xffffffffu, hit);
        const int n = __popc(mask);
        if (hit) sts64u(list_addr + __popc(mask & ((1u << lane) - 1u)) * 8, my_rec, (uint32_t)my_idx + 1u);
        if (lane == 0) sts64u(list_addr + n * 8, dummy_addr, 0u);  // pad (alpha = 0: never contributes)
        __syncwarp();
        for (int i = 0; i < n; i += 2) {
          const uint4 ent = lds128u(list_addr + i * 8);
          const float4 q0a = lds128(ent.x), q0b = lds128(ent.z);
          const float4 q1a = lds128(ent.x + 16), q1b = lds128(ent.z + 16);
          const float4 q2a = lds128(ent.x + 32), q2b = lds128(ent.z + 32);
          const float2 apa = f3_alpha(q0a, q1a, npx, fpy), apb = f3_alpha(q0b, q1b, npx, fpy);
          {  // first record; a pixel that skips it composites alpha' = 0: w = 0, tau unchanged
            const bool c0 = (tau.x >= TAU_STOP) && (apa.x >= ALPHA_SKIP);
            const bool c1 = (tau.y >= TAU_STOP) && (apa.y >= ALPHA_SKIP);
            const float2 e = p2(c0 ? apa.x : 0.0f, c1 ? apa.y : 0.0f);
            const float2 w = __fmul2_rn(tau, e);
            cr = __ffma2_rn(w, p2s(q2a.x), cr);
            cg = __ffma2_rn(w, p2s(q2a.y), cg);
            cb = __ffma2_rn(w, p2s(q2a.z), cb);
            tau = __fmul2_rn(tau, __fadd2_rn(p2s(1.0f), p2(-e.x, -e.y)));
            if (c0) cont0 = (int)ent.y;
            if (c1) cont1 = (int)ent.y;
          }
          {  // second record (the pad record when the count is odd)
            const bool c0 = (tau.x >= TAU_STOP) && (apb.x >= ALPHA_SKIP);
            const bool c1 = (tau.y >= TAU_STOP) && (apb.y >= ALPHA_SKIP);
            const float2 e = p2(c0 ? apb.x : 0.0f, c1 ? apb.y : 0.0f);
            const float2 w = __fmul2_rn(tau, e);
            cr = __ffma2_rn(w, p2s(q2b.x), cr);
            cg = __ffma2_rn(w, p2s(q2b.y), cg);
            cb = __ffma2_rn(w, p2s(q2b.z), cb);
            tau = __fmul2_rn(tau, __fadd2_rn(p2s(1.0f), p2(-e.x, -e.y)));
            if (c0) cont0 = (int)ent.w;
            if (c1) cont1 = (int)ent.w;
          }
        }
        // per-warp early out: every pixel of the block has reached tau < 1e-4 (kernel.cu:256)
        const bool done = __all_sync(0xffffffffu, tau.x < TAU_STOP && tau.y < TAU_STOP);
        if (done) break;
        __syncwarp();  // every lane is done with this ring slot and with the list
        issue(c + F3_RING, id_next);
        id_next = load_id(c + F3_RING + 1);
      }
      cp_async_wait<0>();
      __syncwarp();
    }
    if (in0 && in1 && vec2) {
      *reinterpret_cast<float2 *>(image + pix) = cr;
      *reinterpret_cast<float2 *>(image + HW + pix) = cg;
      *reinterpret_cast<float2 *>(image + 2 * HW + pix) = cb;
      *reinterpret_cast<int2 *>(contrib + pix) = make_int2(cont0, cont1);
      *reinterpret_cast<float2 *>(final_tau + pix) = tau;
    } else {
      if (in0) {
        image[pix] = cr.x; image[HW + pix] = cg.x; image[2 * HW + pix] = cb.x;
        contrib[pix] = cont0; final_tau[pix] = tau.x;
      }
      if (in1) {
        image[pix + 1] = cr.y; image[HW + pix + 1] = cg.y; image[2 * HW + pix + 1] = cb.y;
        contrib[pix + 1] = cont1; final_tau[pix + 1] = tau.y;
      }
    }
   }  // blocks of the entry
  }
}

int launch_draw(int H, int W, const int32_t *ranges, const Rec *recs, const int32_t *gsid, float *image,
                 int32_t *contrib, float *final_tau, int *work_counter, cudaStream_t st) {
  const int gx = (W + TILE - 1) / TILE, gy = (H + TILE - 1) / TILE;
  if (gx <= 0 || gy <= 0) return 0;
  const int T = gx * gy;
  if (work_counter == nullptr) return set_arg_error("draw: work area missing");
  // work list (and the zeros of the empty tiles) first; it also clears the item counter
  int rc = launch_tile_list(H, W, ranges, image, contrib, final_tau, work_counter, st);
  if (rc) return rc;
  int dev = 0, sms = 148;
  GSB_CUDA_TRY(cudaGetDevice(&dev));
  GSB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const long long want = (long long)sms * FWD3_MINBLOCKS;
  const int grid = (int)(T < want ? T : want);
  ProfScope ps(K_DRAW, st);
  k_draw3<<<grid, 128, 0, st>>>(W, H, gx, T, reinterpret_cast<const int2 *>(ranges), recs, gsid, image, contrib,
                                final_tau, work_counter);
  GSB_CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // namespace gsb
