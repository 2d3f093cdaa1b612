// Backward tile rasterizer, variant 4: a two-phase scheme (pixel-parallel replay, then
// record-parallel moment sums through shared memory -- notes at b4_flush below) with
//   * warp-autonomous work: a work item is one 8x8 pixel block of a tile; every warp of the
//     persistent grid pulls items from a global counter and streams the tile's record list
//     itself (32-record chunks, one cp.async gather of 48 bytes per lane, double buffered with
//     cp.async groups + __syncwarp).  No __syncthreads anywhere: in variants 2/3 a tenth of
//     all warp time was spent at the per-stage CTA barrier (ncu: stall_barrier), and a warp
//     stops at ITS last contributing record instead of the tile's;
//   * two records per iteration of the replay loop: the alpha' evaluations of two consecutive
//     surviving records are independent chains (LDS -> FFMA2 -> ex2 -> min -> rcp), only the
//     short tau / s recurrences are sequential, so an in-order warp overlaps their latencies.
// The records are read 4x (once per block) instead of once per tile; they come from L2.
// Replaces reference kernel.cu:809-950 (drawB).
#include "common.cuh"
#include "kernels.h"

namespace gsb {

constexpr int B4_SLOTS = 8;
// slot = 2 weight rows of 64 floats + 16 floats of padding: a stride of 16 (mod 32) floats makes the
// phase-B 128-bit reads (2 slots x 4 parts per 8-lane wavefront) conflict-free
constexpr int B4_SLOT_BYTES = (2 * 64 + 16) * 4;       // 576
constexpr int B4_W_BYTES = B4_SLOTS * B4_SLOT_BYTES;   // 4608
constexpr int B4_RING = 2;                             // 32-record chunks in flight per warp
constexpr int B4_CHUNK_BYTES = 32 * 48;
#ifndef BWD4_MINBLOCKS
#define BWD4_MINBLOCKS 6
#endif

namespace {
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ float2 lds64(uint32_t a) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts64(uint32_t a, float2 v) {
  asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t a, float x, float y, float z, float w) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
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
__device__ __forceinline__ float2 lo(const float4 &v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ float2 hi(const float4 &v) { return make_float2(v.z, v.w); }

// Phase B: moment sums of up to 8 records over the warp's 8x8 block.
//   lane = slot * 4 + part; part covers x in [4 (part & 1), +4) of rows (part >> 1) + {0, 2, 4, 6}.
//   inf = record word q0 = (u_x, u_y, gaussian id, alpha) of the lane's slot.  It travels in registers:
//   the kernel is bound by shared-memory wavefronts (ncu: LSU data pipe 89 %), and a 16-byte
//   shared store costs 4 of them even from one lane (benchmarks/micro/redux_bench.cu).
__device__ __forceinline__ void b4_flush(uint32_t w_addr, const float4 &inf, uint32_t dl_addr, int nslots,
                                         float fbx0, float fby0, float *__restrict__ moments, int lane) {
  const int slot = lane >> 2, part = lane & 3;
  const float U = inf.x - (fbx0 + (float)((part & 1) * 4));
  const float V = inf.y - (fby0 + (float)(part >> 1));
  const float2 dx01 = p2(U, U - 1.0f), dx23 = p2(U - 2.0f, U - 3.0f);
  const uint32_t a = w_addr + slot * B4_SLOT_BYTES + part * 16;
  const uint32_t d = dl_addr + part * 16;
  float2 m0 = p2s(0.f), m1 = p2s(0.f), m2 = p2s(0.f), m3 = p2s(0.f), m4 = p2s(0.f), m5 = p2s(0.f),
         m6 = p2s(0.f), m7 = p2s(0.f), m8 = p2s(0.f);
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const float dy = V - (float)(2 * j);
    const float dy2 = dy * dy;
    const float4 w = lds128(a + j * 64);
    const float4 wc = lds128(a + 256 + j * 64);
    const float4 dr = lds128(d + j * 64);
    const float4 dg = lds128(d + 256 + j * 64);
    const float4 db = lds128(d + 512 + j * 64);
    const float2 t01 = __fmul2_rn(lo(w), dx01), t23 = __fmul2_rn(hi(w), dx23);
    const float2 r1 = __fadd2_rn(t01, t23), r0 = __fadd2_rn(lo(w), hi(w));
    m0 = __fadd2_rn(m0, r1);
    m2 = __ffma2_rn(t01, dx01, m2);
    m2 = __ffma2_rn(t23, dx23, m2);
    m1 = __ffma2_rn(p2s(dy), r0, m1);
    m3 = __ffma2_rn(p2s(dy), r1, m3);
    m4 = __ffma2_rn(p2s(dy2), r0, m4);
    m5 = __fadd2_rn(m5, r0);
    m6 = __ffma2_rn(lo(wc), lo(dr), m6);
    m6 = __ffma2_rn(hi(wc), hi(dr), m6);
    m7 = __ffma2_rn(lo(wc), lo(dg), m7);
    m7 = __ffma2_rn(hi(wc), hi(dg), m7);
    m8 = __ffma2_rn(lo(wc), lo(db), m8);
    m8 = __ffma2_rn(hi(wc), hi(db), m8);
  }
  // sum dL/dalpha' g = (sum w) / alpha; records above the clamp were reduced in phase A
  const float inv_alpha = inf.w <= ALPHA_CLAMP ? __fdividef(1.0f, inf.w) : 0.0f;
  const float v[9] = {m0.x + m0.y, m1.x + m1.y, m2.x + m2.y, m3.x + m3.y, m4.x + m4.y,
                      (m5.x + m5.y) * inv_alpha, m6.x + m6.y, m7.x + m7.y, m8.x + m8.y};
  // split exchange between the four parts of a slot: part 0 -> v0 v1 v2, part 2 -> v3 v4,
  // part 1 -> v5 v6 v7, part 3 -> v8
  const unsigned F = 0xffffffffu;
  const bool u1 = part & 1, u2 = part & 2;
  float s[5], b[3];
#pragma unroll
  for (int i = 0; i < 4; i++) s[i] = (u1 ? v[i + 5] : v[i]) + __shfl_xor_sync(F, u1 ? v[i] : v[i + 5], 1);
  s[4] = (u1 ? 0.f : v[4]) + __shfl_xor_sync(F, u1 ? v[4] : 0.f, 1);
  b[0] = (u2 ? s[3] : s[0]) + __shfl_xor_sync(F, u2 ? s[0] : s[3], 2);
  b[1] = (u2 ? s[4] : s[1]) + __shfl_xor_sync(F, u2 ? s[1] : s[4], 2);
  b[2] = (u2 ? 0.f : s[2]) + __shfl_xor_sync(F, u2 ? s[2] : 0.f, 2);
  if (slot < nslots) {
    const int first = u1 ? (u2 ? 8 : 5) : (u2 ? 3 : 0);
    float *row = moments + (size_t)__float_as_int(inf.z) * 9 + first;
    atomicAdd(row, b[0]);
    if (part != 3) atomicAdd(row + 1, b[1]);
    if (!u2) atomicAdd(row + 2, b[2]);
  }
}

// alpha' of one record at the lane's pixel pair, with the skip decisions of kernel.cu:909-913.
// e = alpha' where the pixel replays the record, else 0.  An inactive pixel needs no further
// predication: 1 - 0 = 1 and MUFU.RCP(1) = 1 exactly, so tau stays bit-identical, and both
// weights are (finite) * 0 = 0.
struct B4Eval {
  float2 dx, gg, e, rc;  // rc = 1 / (1 - e)
  float dy;
};
__device__ __forceinline__ B4Eval b4_eval(const float4 &q0, const float4 &q1, const float2 &npx, float fpy, int idx,
                                          int cont0, int cont1) {
  B4Eval r;
  r.dx = __fadd2_rn(p2s(q0.x), npx);
  r.dy = q0.y - fpy;
  const float cdy2 = (q1.z * r.dy) * r.dy;
  const float2 t = __ffma2_rn(p2s(q1.y), p2s(r.dy), __fmul2_rn(p2s(q1.x), r.dx));
  const float2 p = __ffma2_rn(t, r.dx, p2s(cdy2));
  r.gg = p2(ex2_approx(fminf(p.x, 0.0f)), ex2_approx(fminf(p.y, 0.0f)));
  const float2 ag = __fmul2_rn(p2s(q0.w), r.gg);
  const float ap0 = fminf(ALPHA_CLAMP, ag.x), ap1 = fminf(ALPHA_CLAMP, ag.y);
  r.e = p2(((idx < cont0) && (ap0 >= ALPHA_SKIP)) ? ap0 : 0.0f, ((idx < cont1) && (ap1 >= ALPHA_SKIP)) ? ap1 : 0.0f);
  const float2 om = __fadd2_rn(p2s(1.0f), p2(-r.e.x, -r.e.y));
  r.rc = p2(rcp_approx(om.x), rcp_approx(om.y));
  return r;
}
__device__ __forceinline__ uint4 lds128u(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts64u(uint32_t a, uint32_t x, uint32_t y) {
  asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
}  // namespace

__global__ void __launch_bounds__(128, BWD4_MINBLOCKS) k_draw_bwd4(
    int W, int H, int gx, int T, const int2 *__restrict__ ranges, const Rec *__restrict__ recs,
    const int32_t *__restrict__ gsid, const int32_t *__restrict__ contrib, const float *__restrict__ final_tau,
    const float *__restrict__ dloss_dgammas, float *__restrict__ moments, int *__restrict__ work) {
  __shared__ __align__(16) unsigned char s_ring[4][B4_RING * B4_CHUNK_BYTES];  // gathered records, per warp
  __shared__ __align__(16) unsigned char s_w[4][B4_W_BYTES];                   // weight rows, per warp
  __shared__ __align__(16) float s_dl[4][3][64];                               // dL/dgamma of the block
  __shared__ __align__(16) uint2 s_list[4][34];  // (record address, patch index) of a chunk's survivors
  __shared__ __align__(16) Rec s_dummy;          // all-zero record: pads an odd survivor count

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t HW = (size_t)H * W;
  const uint32_t ring_addr = opaque_u32(smem_u32(&s_ring[warp][0]));
  const uint32_t w_addr = opaque_u32(smem_u32(&s_w[warp][0]));
  const uint32_t dl_addr = opaque_u32(smem_u32(&s_dl[warp][0][0]));
  const uint32_t list_addr = opaque_u32(smem_u32(&s_list[warp][0]));
  const uint32_t dummy_addr = smem_u32(&s_dummy);
  if (threadIdx.x < 12) reinterpret_cast<float *>(&s_dummy)[threadIdx.x] = 0.0f;
  __syncthreads();  // (the only CTA-wide barrier: start-up)
  (void)T;
  const int items = work[1];  // entries of the work list (k_tile_list, raster_fwd3.cu)
  const int *__restrict__ entries = work + 2;

  // One flat loop over 8x8 blocks: a new work-list entry is pulled when the current one is used up
  // (an entry is one block of a dense tile, or all four blocks of a tile with <= 32 patches).
  int tile = 0, len = 0, blk = 0, blk_end = 0;
  bool whole_tile = false;
  int2 range = make_int2(0, 0);
  for (;;) {
    if (blk == blk_end) {
      int item = 0;
      if (lane == 0) item = atomicAdd(work, 1);
      item = __shfl_sync(0xffffffffu, item, 0);
      if (item >= items) break;
      const int ent = __ldg(entries + item);
      const int code = ent & 7;
      tile = ent >> 3;
      whole_tile = code == 4;  // <= 32 patches: all four blocks from one gather
      range = __ldg(ranges + tile);
      len = range.y - range.x;
      if (len <= 0) continue;
      blk = whole_tile ? 0 : code;
      blk_end = whole_tile ? 4 : code + 1;
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
    }
    const int cur = blk++;
    const int tx = tile % gx, ty = tile / gx;
    const int rx0 = tx * TILE + (cur & 1) * 8, ry0 = ty * TILE + (cur >> 1) * 8;
    if (rx0 >= W || ry0 >= H) continue;  // block entirely outside the image
    const int px = rx0 + 2 * (lane & 3), py = ry0 + (lane >> 2);
    const bool in0 = px < W && py < H, in1 = px + 1 < W && py < H;
    const size_t pix = (size_t)py * W + px;

    int cont0 = 0, cont1 = 0;
    float2 tau = p2s(0.f), dlr = p2s(0.f), dlg = p2s(0.f), dlb = p2s(0.f);
    if (in0) {
      cont0 = min(__ldg(contrib + pix), len);
      tau.x = __ldg(final_tau + pix);
      dlr.x = __ldg(dloss_dgammas + pix);
      dlg.x = __ldg(dloss_dgammas + HW + pix);
      dlb.x = __ldg(dloss_dgammas + 2 * HW + pix);
    }
    if (in1) {
      cont1 = min(__ldg(contrib + pix + 1), len);
      tau.y = __ldg(final_tau + pix + 1);
      dlr.y = __ldg(dloss_dgammas + pix + 1);
      dlg.y = __ldg(dloss_dgammas + HW + pix + 1);
      dlb.y = __ldg(dloss_dgammas + 2 * HW + pix + 1);
    }
    int wmax = max(cont0, cont1);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wmax = max(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
    if (wmax <= 0) continue;
    // the block's dL/dgamma table for phase B (pixel p = 8 row + x = 2 lane + {0, 1}); the
    // __syncwarp before the first flush orders it
    sts64(dl_addr + lane * 8, dlr);
    sts64(dl_addr + 256 + lane * 8, dlg);
    sts64(dl_addr + 512 + lane * 8, dlb);

    const int nch = (wmax + 31) >> 5;  // chunks [0, nch) hold the records any pixel replays
    const int32_t *ids = gsid + range.x;
    // gather of chunk c: lane j copies the record of patch 32 c + j (if below wmax) into ring slot c & 1
    auto issue = [&](int c, int id) {
      if (c >= 0 && c * 32 + lane < wmax) {
        const char *src = reinterpret_cast<const char *>(recs + id);
        const uint32_t dst = ring_addr + (c & (B4_RING - 1)) * B4_CHUNK_BYTES + lane * 48;
        cp_async16_sa(dst, src);
        cp_async16_sa(dst + 16, src + 16);
        cp_async16_sa(dst + 32, src + 32);
      }
      cp_async_commit();
    };
    auto load_id = [&](int c) { return (c >= 0 && c * 32 + lane < wmax) ? __ldg(ids + c * 32 + lane) : 0; };
    int id_next = 0;
    if (!whole_tile) {
#pragma unroll
      for (int r = 0; r < B4_RING; r++) issue(nch - 1 - r, load_id(nch - 1 - r));
      id_next = load_id(nch - 1 - B4_RING);  // id of the chunk the first refill gathers
    }

    const float2 npx = p2(-(float)px, -(float)(px + 1));
    const float fpy = (float)py;
    const float bx0 = (float)rx0, bx1 = (float)(rx0 + 7), by0 = (float)ry0, by1 = (float)(ry0 + 7);
    float2 sdot = p2s(0.f);  // dL/dgamma . gamma_next, per pixel
    uint32_t wa = w_addr + lane * 8;  // where the next record's weight rows go
    const uint32_t wa_pair_limit = w_addr + lane * 8 + (B4_SLOTS - 2) * B4_SLOT_BYTES;
    int to_my_slot = lane >> 2;  // free slots before the one whose moments this lane sums in phase B
    float4 inf = make_float4(0.f, 0.f, 0.f, 1.f);

    for (int c = nch - 1; c >= 0; c--) {
      cp_async_wait<B4_RING - 1>();  // this lane's copy of chunk c has landed ...
      __syncwarp();                  // ... and so have the other lanes'
      const uint32_t my_rec = ring_addr + (c & (B4_RING - 1)) * B4_CHUNK_BYTES + lane * 48;
      const int my_idx = c * 32 + lane;
      bool hit = false;
      if (my_idx < wmax) hit = rec_can_touch(lds128(my_rec), lds128(my_rec + 16), bx0, bx1, by0, by1);
      // survivors of the chunk, back to front, as a list of (record address, patch index)
      const unsigned mask = __ballot_sync(0xffffffffu, hit);
      const int n = __popc(mask);
      if (hit) sts64u(list_addr + __popc(mask & ~((2u << lane) - 1u)) * 8, my_rec, (uint32_t)my_idx);
      if (lane == 0) sts64u(list_addr + n * 8, dummy_addr, 0x7fffffffu);  // pad: index beyond every contrib
      __syncwarp();
      for (int i = 0; i < n; i += 2) {
        if (wa > wa_pair_limit) {  // no room for a pair
          __syncwarp();
          b4_flush(w_addr, inf, dl_addr, (lane >> 2) - to_my_slot, bx0, by0, moments, lane);
          __syncwarp();
          wa = w_addr + lane * 8;
          to_my_slot = lane >> 2;
        }
        const uint4 ent = lds128u(list_addr + i * 8);  // two records: ent.x / ent.z further back first
        const float4 q0a = lds128(ent.x), q0b = lds128(ent.z);
        const float4 q1a = lds128(ent.x + 16), q1b = lds128(ent.z + 16);
        const float4 q2a = lds128(ent.x + 32), q2b = lds128(ent.z + 32);
        const B4Eval A = b4_eval(q0a, q1a, npx, fpy, (int)ent.y, cont0, cont1);
        const B4Eval B = b4_eval(q0b, q1b, npx, fpy, (int)ent.w, cont0, cont1);
        const float2 dca = __ffma2_rn(dlr, p2s(q2a.x), __ffma2_rn(dlg, p2s(q2a.y), __fmul2_rn(dlb, p2s(q2a.z))));
        const float2 dcb = __ffma2_rn(dlr, p2s(q2b.x), __ffma2_rn(dlg, p2s(q2b.y), __fmul2_rn(dlb, p2s(q2b.z))));
        // first record
        tau = __fmul2_rn(tau, A.rc);
        const float2 diffa = __fadd2_rn(dca, p2(-sdot.x, -sdot.y));
        sdot = __ffma2_rn(A.e, diffa, sdot);
        const float2 dapa = __fmul2_rn(tau, diffa);  // dL/dalpha' (where active; times e = 0 elsewhere)
        sts64(wa, __fmul2_rn(dapa, A.e));        // w
        sts64(wa + 256, __fmul2_rn(A.e, tau));   // wc
        if (to_my_slot == 0) inf = q0a;
        // second record (the all-zero pad record when the count is odd: e = 0, weights 0)
        tau = __fmul2_rn(tau, B.rc);
        const float2 diffb = __fadd2_rn(dcb, p2(-sdot.x, -sdot.y));
        sdot = __ffma2_rn(B.e, diffb, sdot);
        const float2 dapb = __fmul2_rn(tau, diffb);
        sts64(wa + B4_SLOT_BYTES, __fmul2_rn(dapb, B.e));
        sts64(wa + B4_SLOT_BYTES + 256, __fmul2_rn(B.e, tau));
        if (to_my_slot == 1) inf = q0b;
        if (fmaxf(q0a.w, q0b.w) > ALPHA_CLAMP) {  // opacity above the clamp (rare):
          // sum dL/dalpha' g is not (sum w) / alpha on clamped pixels -- reduce it with shuffles
          float va = q0a.w > ALPHA_CLAMP ? fmaf(A.e.x > 0.f ? dapa.x : 0.f, A.gg.x, (A.e.y > 0.f ? dapa.y : 0.f) * A.gg.y) : 0.0f;
          float vb = q0b.w > ALPHA_CLAMP ? fmaf(B.e.x > 0.f ? dapb.x : 0.f, B.gg.x, (B.e.y > 0.f ? dapb.y : 0.f) * B.gg.y) : 0.0f;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            va += __shfl_xor_sync(0xffffffffu, va, o);
            vb += __shfl_xor_sync(0xffffffffu, vb, o);
          }
          if (lane == 0 && va != 0.0f) atomicAdd(moments + (size_t)__float_as_int(q0a.z) * 9 + 5, va);
          if (lane == 0 && vb != 0.0f) atomicAdd(moments + (size_t)__float_as_int(q0b.z) * 9 + 5, vb);
        }
        const bool pair = i + 2 <= n;  // false: the second record was the pad, its slot is reused
        wa += pair ? 2 * B4_SLOT_BYTES : B4_SLOT_BYTES;
        to_my_slot -= pair ? 2 : 1;
      }
      __syncwarp();  // every lane is done with this ring slot and with the list
      issue(c - B4_RING, id_next);
      id_next = load_id(c - B4_RING - 1);
    }
    cp_async_wait<0>();
    if (wa != w_addr + lane * 8) {
      __syncwarp();
      b4_flush(w_addr, inf, dl_addr, (lane >> 2) - to_my_slot, bx0, by0, moments, lane);
    }
    __syncwarp();  // the flush has read s_dl / s_w before the next block rewrites them
  }
}

int launch_draw_bwd4_kernel(int H, int W, const int32_t *ranges, const Rec *recs, const int32_t *gsid,
                            const int32_t *contrib, const float *final_tau, const float *dloss_dgammas,
                            float *moments, int *work_counter, cudaStream_t st) {
  const int gx = (W + TILE - 1) / TILE, gy = (H + TILE - 1) / TILE;
  const int T = gx * gy;
  if (work_counter == nullptr) return set_arg_error("drawB: work area missing");
  int rc = launch_tile_list(H, W, ranges, nullptr, nullptr, nullptr, work_counter, st);  // tiles with patches
  if (rc) return rc;
  int dev = 0, sms = 148;
  GSB_CUDA_TRY(cudaGetDevice(&dev));
  GSB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const long long want = (long long)sms * BWD4_MINBLOCKS;
  const int grid = (int)(T < want ? T : want);
  ProfScope ps(K_DRAW_BWD, st);
  k_draw_bwd4<<<grid, 128, 0, st>>>(W, H, gx, T, reinterpret_cast<const int2 *>(ranges), recs, gsid, contrib,
                                    final_tau, dloss_dgammas, moments, work_counter);
  GSB_CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // namespace gsb
