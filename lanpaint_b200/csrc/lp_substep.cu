// lanpaint_b200: the fused Langevin sub-step (everything between two model calls) and its C ABI.
//
// Reference being replaced: src/LanPaint/lanpaint.py:113-142 -> langevin_dynamics :192-293 -> score_model
// :159-184, Coef_C :217-220, advance_time_overdamped :232-254, run_overdamped :274-286.
//
// Kernels (all templated on the element type H of the model's heads: fp32 / bf16 / fp16)
//   substep_kernel            one float4 per thread, LDG.128; TAPE and PHILOX streams; small or ragged launches
//   substep_tma_kernel        PHILOX: persistent grid, cp.async.bulk ring of 2048-element tiles (HBM-bound sizes)
//   substep_torch_tma_kernel  TORCH (torch.randn_like's exact stream): persistent grid, producer warp + 8
//                             consumer warps, 4 plane-slots of 1024 elements, one Philox call per 4 elements
//   substep_torchvec_kernel   TORCH, LDG.128 + quad transpose (launches the TMA variant cannot take)
//   substep_torch_kernel      TORCH, scalar (odd sizes)
#include "lp_common.cuh"

namespace lp {

struct SubstepArgs {
  float* x;
  const void* x0;
  const void* x0b;
  const float* y;
  const uint8_t* mask;
  float* c;
  float* x_copy;
  float* x0e;
  const float* table;
  const float* tape0;
  const float* tape1;
  const uint64_t* rng_state;
  uint64_t seed, draw0, draw1;
  Geometry g;
  uint32_t torch_T;  // threads of torch's randn grid (LP_RNG_TORCH)
  int store_c;       // write C even when the next half-advance is not fused
  int use_cfg;       // x0/x0b hold raw cond/uncond predictions: combine them here
  float cfg, cfg_big;
};

// ---- the memory side of a fused launch: one N-wide vector per thread ------------
template <int N, typename H, bool kFirst, bool kNext, bool kMerge>
__device__ __forceinline__ void substep_vector(const SubstepArgs& a, uint32_t i, const float (&xi1)[N],
                                               const float (&xi2)[N]) {
  uint32_t row, mi;
  locate(a.g, i, row, mi);
  float x[N], x0[N], x0b[N], y[N], cp[N], cn[N], te[N];
  bool known[N];
  // The mask decides which operands this vector needs: free positions use only x0, known positions only
  // x0_big and y (score_model, lanpaint.py:182-184).  Inpainting masks are spatially coherent, so most
  // vectors are all-free or all-known and skip 4-8 of their 20 input bytes per element.
  load_m<N>(a.mask, mi, known);
  load_f<N>(a.x, i, x);
  if (!kFirst) {
    load_f<N>(a.c, i, cp);
  } else {
#pragma unroll
    for (int j = 0; j < N; ++j) cp[j] = 0.f;
  }
  bool any_known = false, any_free = false;
#pragma unroll
  for (int j = 0; j < N; ++j) {
    any_known |= known[j];
    any_free |= !known[j];
  }
  const bool aliased = a.x0b == a.x0;
  const bool need_x0 = any_free || aliased || a.use_cfg;
  const bool need_x0b = (any_known || a.use_cfg) && !aliased;
#pragma unroll
  for (int j = 0; j < N; ++j) x0[j] = x0b[j] = y[j] = 0.f;
  if (need_x0) load_head_ro<N, H>(static_cast<const H*>(a.x0), i, x0);
  if (need_x0b) {
    load_head_ro<N, H>(static_cast<const H*>(a.x0b), i, x0b);
  } else if (aliased) {
#pragma unroll
    for (int j = 0; j < N; ++j) x0b[j] = x0[j];
  }
  if (a.use_cfg) {  // x0 = cond, x0b = uncond: u + (c-u)*s with the eager path's three roundings
#pragma unroll
    for (int j = 0; j < N; ++j) cfg_combine(x0[j], x0b[j], a.cfg, a.cfg_big);
  }
  if (any_known) load_f_ro<N>(a.y, i, y);
  RowCoef<kFirst, kNext> t;
  t.load(a.table + (size_t)row * LP_TABLE_STRIDE);
#pragma unroll
  for (int j = 0; j < N; ++j)
    substep_element<kFirst, kNext, kMerge>(x[j], x0[j], x0b[j], y[j], cp[j], known[j], xi1[j], xi2[j], t, cn[j],
                                           te[j]);
  store_f<N>(a.x, i, x);
  if (kNext || a.store_c) store_f<N>(a.c, i, cn);
  if (a.x_copy) store_f<N>(a.x_copy, i, x);
  if (a.x0e) store_f<N>(a.x0e, i, te);
}

// ---- TAPE / PHILOX ------------------------------------------------------------
template <int N, typename H, int kRng, bool kFirst, bool kNext, bool kMerge = false>
__global__ void __launch_bounds__(kBlock, 5) substep_kernel(const SubstepArgs a) {
  pdl_prologue();
  const uint32_t v = blockIdx.x * kBlock + threadIdx.x;
  const uint32_t i = v * N;
  if (i >= a.g.total) return;
  float xi1[N], xi2[N];
  if (kRng == LP_RNG_TAPE) {
    load_f_ro<N>(a.tape0, i, xi1);
    if (kNext) {
      load_f_ro<N>(a.tape1, i, xi2);
    } else {
#pragma unroll
      for (int j = 0; j < N; ++j) xi2[j] = 0.f;
    }
  } else {
    uint64_t seed = a.seed, d0 = a.draw0, d1 = a.draw1;
    if (a.rng_state) {
      seed = a.rng_state[0];
      d0 += a.rng_state[1];
      d1 += a.rng_state[1];
    }
    const float4 n1 = philox_normal4(seed, d0, i >> 2);
    float4 n2 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (kNext && !kMerge) n2 = philox_normal4(seed, d1, i >> 2);
    if (N == 4) {
      xi1[0] = n1.x; xi1[1 % N] = n1.y; xi1[2 % N] = n1.z; xi1[3 % N] = n1.w;
      xi2[0] = n2.x; xi2[1 % N] = n2.y; xi2[2 % N] = n2.z; xi2[3 % N] = n2.w;
    } else {
      xi1[0] = pick(n1, i & 3);
      xi2[0] = pick(n2, i & 3);
    }
  }
  substep_vector<N, H, kFirst, kNext, kMerge>(a, i, xi1, xi2);
}

// ---- PHILOX, TMA-staged persistent variant of the fused sub-step ---------------------------
// Same arithmetic and the same Philox stream as substep_kernel (results are bit-identical); different data
// movement: a persistent grid (2 CTAs per SM) walks tiles of kTile consecutive elements of one (row, channel),
// one elected thread streams each tile's five operand slices + mask slice into shared memory with
// cp.async.bulk (the TMA unit, completion counted on an mbarrier), kStages tiles ahead, and the 256 threads
// consume them with LDS.128 and write x / C back with STG.128.  Registers hold no loads in flight, so
// bytes-in-flight per SM is set by kStages * 42 KB instead of by occupancy.
template <typename H, int kTile>
struct __align__(128) TmaStage {
  float x[kTile];
  H x0[kTile], x0b[kTile];
  float y[kTile], c[kTile];
  uint8_t m[kTile];
};

struct TileGeom {
  uint32_t tiles_per_channel, n_tiles, channels;
};

template <typename H, bool kFirst, bool kNext, bool kMerge, int kTile, int kStages, int kMinBlocks>
__global__ void __launch_bounds__(kBlock, kMinBlocks) substep_tma_kernel(const SubstepArgs a, const TileGeom tg) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  using Stage = TmaStage<H, kTile>;
  Stage* stage = reinterpret_cast<Stage*>(smem_raw);
  __shared__ __align__(8) uint64_t full[kStages];
  pdl_prologue();
  const uint32_t S = a.g.spatial.d;
  const bool aliased = a.x0b == a.x0;
  const H* x0p = static_cast<const H*>(a.x0);
  const H* x0bp = static_cast<const H*>(a.x0b);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) mbar_init(&full[s], 1);
    mbar_fence_init();
  }
  __syncthreads();

  auto tile_origin = [&](uint32_t tile, uint32_t& e0, uint32_t& len, uint32_t& row, uint32_t& mi0) {
    const uint32_t rc = tile / tg.tiles_per_channel;          // row * channels + channel
    const uint32_t s0 = (tile - rc * tg.tiles_per_channel) * kTile;
    len = S - s0 < (uint32_t)kTile ? S - s0 : (uint32_t)kTile;
    e0 = rc * S + s0;
    row = rc / tg.channels;
    mi0 = row * a.g.mask_row_stride + (rc - row * tg.channels) * a.g.mask_channel_stride + s0;
  };
  auto issue = [&](uint32_t tile, int s) {  // one thread
    uint32_t e0, len, row, mi0;
    tile_origin(tile, e0, len, row, mi0);
    const uint32_t fb = len * 4u, hb = len * (uint32_t)sizeof(H);
    const uint32_t total = fb * (2u + (kFirst ? 0u : 1u)) + hb * (1u + (aliased ? 0u : 1u)) + len;
    mbar_expect_tx(&full[s], total);
    Stage& t = stage[s];
    tma_load_1d(t.x, a.x + e0, fb, &full[s]);
    tma_load_1d(t.x0, x0p + e0, hb, &full[s]);
    if (!aliased) tma_load_1d(t.x0b, x0bp + e0, hb, &full[s]);
    tma_load_1d(t.y, a.y + e0, fb, &full[s]);
    if (!kFirst) tma_load_1d(t.c, a.c + e0, fb, &full[s]);
    tma_load_1d(t.m, a.mask + mi0, len, &full[s]);
  };

  uint64_t seed = a.seed, d0 = a.draw0, d1 = a.draw1;
  if (a.rng_state) {
    seed = a.rng_state[0];
    d0 += a.rng_state[1];
    d1 += a.rng_state[1];
  }
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
      const uint32_t tile = blockIdx.x + (uint32_t)s * gridDim.x;
      if (tile < tg.n_tiles) issue(tile, s);
    }
  }
  uint32_t k = 0;
  for (uint32_t tile = blockIdx.x; tile < tg.n_tiles; tile += gridDim.x, ++k) {
    const int s = (int)(k % kStages);
    mbar_wait(&full[s], (k / kStages) & 1u);
    uint32_t e0, len, row, mi0;
    tile_origin(tile, e0, len, row, mi0);
    const Stage& t = stage[s];
    RowCoef<kFirst, kNext> rc;
    rc.load(a.table + (size_t)row * LP_TABLE_STRIDE);
#pragma unroll
    for (int pass = 0; pass < kTile / (4 * kBlock); ++pass) {
      const uint32_t v = threadIdx.x + pass * kBlock;  // vector inside the tile
      if (4 * v < len) {
        const float4 xv = reinterpret_cast<const float4*>(t.x)[v];
        float x0[4], x0b[4];
        lds_head4<H>(t.x0, v, x0);
        if (aliased) {
#pragma unroll
          for (int j = 0; j < 4; ++j) x0b[j] = x0[j];
        } else {
          lds_head4<H>(t.x0b, v, x0b);
        }
        const float4 yv = reinterpret_cast<const float4*>(t.y)[v];
        const float4 cv = kFirst ? make_float4(0.f, 0.f, 0.f, 0.f) : reinterpret_cast<const float4*>(t.c)[v];
        const uchar4 mv = reinterpret_cast<const uchar4*>(t.m)[v];
        float x[4] = {xv.x, xv.y, xv.z, xv.w}, y[4] = {yv.x, yv.y, yv.z, yv.w};
        float cp[4] = {cv.x, cv.y, cv.z, cv.w}, cn[4], te[4];
        const bool known[4] = {mv.x != 0, mv.y != 0, mv.z != 0, mv.w != 0};
        if (a.use_cfg) {
#pragma unroll
          for (int j = 0; j < 4; ++j) cfg_combine(x0[j], x0b[j], a.cfg, a.cfg_big);
        }
        const uint32_t i = e0 + 4 * v;
        const float4 n1 = philox_normal4(seed, d0, i >> 2);
        float4 n2 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (kNext && !kMerge) n2 = philox_normal4(seed, d1, i >> 2);
        const float xi1[4] = {n1.x, n1.y, n1.z, n1.w}, xi2[4] = {n2.x, n2.y, n2.z, n2.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
          substep_element<kFirst, kNext, kMerge>(x[j], x0[j], x0b[j], y[j], cp[j], known[j], xi1[j], xi2[j], rc, cn[j],
                                                te[j]);
        *reinterpret_cast<float4*>(a.x + i) = make_float4(x[0], x[1], x[2], x[3]);
        if (kNext || a.store_c) *reinterpret_cast<float4*>(a.c + i) = make_float4(cn[0], cn[1], cn[2], cn[3]);
      }
    }
    __syncthreads();  // every thread is done reading stage s
    const uint32_t next = tile + (uint32_t)kStages * gridDim.x;
    if (threadIdx.x == 0 && next < tg.n_tiles) issue(next, s);
  }
}

// ---- TORCH, TMA-staged persistent variant --------------------------------------------------------
// torch.randn_like gives element li the component ((li div T) mod 4) of the (li div 4T)-th curand_normal4 of
// Philox subsequence (li mod T), T = 256 * grid of torch's own kernel.  So ONE Philox call yields the normals of
// four elements that lie T apart ("planes" 4k..4k+3 of call k).  A work group is (call k, block b of kTorchG
// consecutive subsequences): four sub-tiles of kTorchG consecutive elements, T apart.  Per CTA:
//   * a producer warp streams the four sub-tiles' operand slices into four shared-memory slots with
//     cp.async.bulk, each slot guarded by a full/empty mbarrier pair, refilling a slot as soon as the eight
//     consumer warps have drained it -- so loads of the next group are in flight during the whole RNG phase;
//   * consumer thread c owns subsequences 4c..4c+3 of the block: 4 Philox calls per draw, cuRAND's exact
//     Box-Muller, and its four normals per plane are one float4 of that plane's sub-tile -- no shuffles.
// Same Philox stream, same arithmetic as the LDG kernels: bit-identical results.
template <typename H, int kG>
struct __align__(128) TorchSlot {
  float x[kG];
  H x0[kG], x0b[kG];
  float y[kG], c[kG];
  uint8_t m[kG];
};

struct TorchTmaGeom {
  uint32_t groups_per_call;  // T / kG
  uint32_t n_groups;         // calls * groups_per_call
};

// kG subsequences per group = 4 per consumer thread; one extra warp produces.
template <typename H, bool kFirst, bool kNext, int kG>
__device__ __forceinline__ void torch_tma_body(const SubstepArgs& a, const TorchTmaGeom& tg, unsigned char* smem_raw,
                                               uint64_t* full, uint64_t* empty) {
  constexpr int kConsumers = kG / 4;
  using Slot = TorchSlot<H, kG>;
  Slot* slot = reinterpret_cast<Slot*>(smem_raw);
  pdl_prologue();
  const uint32_t T = a.torch_T, total = a.g.total;
  const bool aliased = a.x0b == a.x0;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      mbar_init(&full[j], 1);
      mbar_init(&empty[j], kConsumers);
    }
    mbar_fence_init();
  }
  __syncthreads();
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // first element / length of sub-tile j of group (k, b)
  auto subtile = [&](uint32_t k, uint32_t b, int j, uint32_t& e0, uint32_t& len) {
    const uint64_t e = (uint64_t)(4u * k + (uint32_t)j) * T + (uint64_t)b * kG;
    if (e >= total) {
      e0 = 0;
      len = 0;
    } else {
      e0 = (uint32_t)e;
      len = total - e0 < (uint32_t)kG ? total - e0 : (uint32_t)kG;
    }
  };

  if (warp == kConsumers / 32) {  // ---------------- producer ----------------
    if (lane == 0) {
      const H* x0p = static_cast<const H*>(a.x0);
      const H* x0bp = static_cast<const H*>(a.x0b);
      uint32_t it = 0;
      for (uint32_t grp = blockIdx.x; grp < tg.n_groups; grp += gridDim.x, ++it) {
        const uint32_t k = grp / tg.groups_per_call, b = grp - k * tg.groups_per_call;
#pragma unroll 1
        for (int j = 0; j < 4; ++j) {
          mbar_wait_relaxed(&empty[j], (it & 1u) ^ 1u);  // consumers have drained this slot (passes at once the first time)
          uint32_t e0, len;
          subtile(k, b, j, e0, len);
          const uint32_t fb = len * 4u, hb = len * (uint32_t)sizeof(H);
          // an empty sub-tile (past the end of the tensor) still completes its phase: expect 0 bytes
          mbar_expect_tx(&full[j], fb * (2u + (kFirst ? 0u : 1u)) + hb * (1u + (aliased ? 0u : 1u)) + len);
          if (len == 0) continue;
          Slot& t = slot[j];
          tma_load_1d(t.x, a.x + e0, fb, &full[j]);
          tma_load_1d(t.x0, x0p + e0, hb, &full[j]);
          if (!aliased) tma_load_1d(t.x0b, x0bp + e0, hb, &full[j]);
          tma_load_1d(t.y, a.y + e0, fb, &full[j]);
          if (!kFirst) tma_load_1d(t.c, a.c + e0, fb, &full[j]);
          // the mask is indexed per (row, channel): one slice per channel segment the sub-tile touches
          uint32_t e = e0, off = 0, rem = len;
          while (rem) {
            const uint32_t row = a.g.per_row.div(e);
            const uint32_t r = e - row * a.g.per_row.d;
            const uint32_t ch = a.g.spatial.div(r);
            const uint32_t s = r - ch * a.g.spatial.d;
            const uint32_t seg = rem < a.g.spatial.d - s ? rem : a.g.spatial.d - s;
            tma_load_1d(t.m + off, a.mask + row * a.g.mask_row_stride + ch * a.g.mask_channel_stride + s, seg,
                        &full[j]);
            e += seg;
            off += seg;
            rem -= seg;
          }
        }
      }
    }
    return;
  }

  // ---------------- consumers ----------------
  uint64_t seed = a.seed, o0 = a.draw0, o1 = a.draw1;
  if (a.rng_state) {
    seed = a.rng_state[0];
    o0 += a.rng_state[1];
    o1 += a.rng_state[1];
  }
  const uint32_t tid = threadIdx.x;  // vector index inside every sub-tile
  // everything a thread does with one sub-tile once its data is in registers
  auto finish = [&](uint32_t i, float (&x)[4], float (&x0)[4], float (&x0b)[4], const float (&y)[4],
                    const float (&cp)[4], uchar4 mv, const float2 (&p1)[4], const float2 (&p2)[4], int jj) {
    const uint32_t row = a.g.per_row.div(i);
    RowCoef<kFirst, kNext> rc;
    rc.load(a.table + (size_t)row * LP_TABLE_STRIDE);
    if (a.use_cfg) {
#pragma unroll
      for (int q = 0; q < 4; ++q) cfg_combine(x0[q], x0b[q], a.cfg, a.cfg_big);
    }
    const bool known[4] = {mv.x != 0, mv.y != 0, mv.z != 0, mv.w != 0};
    float cn[4];
#pragma unroll
    for (int q = 0; q < 4; q += 2) {   // two elements per FP32x2 op; bit-identical to substep_element
      float xx[2] = {x[q], x[q + 1]}, h0[2] = {x0[q], x0[q + 1]}, h1[2] = {x0b[q], x0b[q + 1]}, cc[2];
      const float yy[2] = {y[q], y[q + 1]}, pp[2] = {cp[q], cp[q + 1]};
      const bool kk[2] = {known[q], known[q + 1]};
      const float n1[2] = {jj ? p1[q].y : p1[q].x, jj ? p1[q + 1].y : p1[q + 1].x};
      const float n2[2] = {jj ? p2[q].y : p2[q].x, jj ? p2[q + 1].y : p2[q + 1].x};
      substep_element_x2<kFirst, kNext>(xx, h0, h1, yy, pp, kk, n1, n2, rc, cc);
      x[q] = xx[0]; x[q + 1] = xx[1];
      cn[q] = cc[0]; cn[q + 1] = cc[1];
    }
    *reinterpret_cast<float4*>(a.x + i) = make_float4(x[0], x[1], x[2], x[3]);
    if (kNext || a.store_c) *reinterpret_cast<float4*>(a.c + i) = make_float4(cn[0], cn[1], cn[2], cn[3]);
  };
  auto fetch = [&](const Slot& t, float (&x)[4], float (&x0)[4], float (&x0b)[4], float (&y)[4], float (&cp)[4],
                   uchar4& mv) {
    const float4 xv = reinterpret_cast<const float4*>(t.x)[tid];
    lds_head4<H>(t.x0, tid, x0);
    if (aliased) {
#pragma unroll
      for (int q = 0; q < 4; ++q) x0b[q] = x0[q];
    } else {
      lds_head4<H>(t.x0b, tid, x0b);
    }
    const float4 yv = reinterpret_cast<const float4*>(t.y)[tid];
    const float4 cv = kFirst ? make_float4(0.f, 0.f, 0.f, 0.f) : reinterpret_cast<const float4*>(t.c)[tid];
    mv = reinterpret_cast<const uchar4*>(t.m)[tid];
    x[0] = xv.x; x[1] = xv.y; x[2] = xv.z; x[3] = xv.w;
    y[0] = yv.x; y[1] = yv.y; y[2] = yv.z; y[3] = yv.w;
    cp[0] = cv.x; cp[1] = cv.y; cp[2] = cv.z; cp[3] = cv.w;
  };
  // every consumer THREAD releases the slot itself once its reads are in registers.  (One arrive per warp after a
  // __syncwarp() measured the same 44 us, but compute-sanitizer's racecheck cannot follow that form: 11 hazards
  // against the producer's next cp.async.bulk; with per-thread arrives it reports none -- profiles/r02_sanitizer_*.)
  auto release = [&](int j) { mbar_arrive(&empty[j]); };
  uint32_t it = 0;
  for (uint32_t grp = blockIdx.x; grp < tg.n_groups; grp += gridDim.x, ++it) {
    const uint32_t k = grp / tg.groups_per_call, b = grp - k * tg.groups_per_call;
    const uint32_t t0 = b * kG + 4u * tid;  // my four Philox subsequences (torch threads)
    // all four planes complete (every group but those at the very end of the tensor): no per-thread predicates
    const bool whole = (uint64_t)(4u * k + 3u) * T + (uint64_t)(b + 1u) * kG <= total;
    uint4 r1[4], r2[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      r1[i] = torch_philox(seed, o0, t0 + i, k);
      r2[i] = kNext ? torch_philox(seed, o1, t0 + i, k) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {  // curand_normal4: planes 0,1 <- (x,y), planes 2,3 <- (z,w)
      float2 p1[4], p2[4];
#pragma unroll
      for (int i = 0; i < 4; i += 2) {   // two transforms per call: FP32x2 arithmetic, bit-identical to the scalar form
        box_muller_curand_x2(h ? r1[i].z : r1[i].x, h ? r1[i].w : r1[i].y, h ? r1[i + 1].z : r1[i + 1].x,
                             h ? r1[i + 1].w : r1[i + 1].y, p1[i], p1[i + 1]);
        if (kNext) {
          box_muller_curand_x2(h ? r2[i].z : r2[i].x, h ? r2[i].w : r2[i].y, h ? r2[i + 1].z : r2[i + 1].x,
                               h ? r2[i + 1].w : r2[i + 1].y, p2[i], p2[i + 1]);
        } else {
          p2[i] = p2[i + 1] = make_float2(0.f, 0.f);
        }
      }
#pragma unroll
      for (int jj = 0; jj < 2; ++jj) {
        const int j = 2 * h + jj;
        float x[4], x0[4], x0b[4], y[4], cp[4];
        uchar4 mv = make_uchar4(0, 0, 0, 0);
        mbar_wait(&full[j], it & 1u);
        if (whole) {
          fetch(slot[j], x, x0, x0b, y, cp, mv);
          release(j);  // this warp's reads of slot j are in registers: let it refill
          finish((4u * k + (uint32_t)j) * T + t0, x, x0, x0b, y, cp, mv, p1, p2, jj);
        } else {
          uint32_t e0, len;
          subtile(k, b, j, e0, len);
          const bool active = 4u * tid < len;
          if (active) fetch(slot[j], x, x0, x0b, y, cp, mv);
          release(j);
          if (active) finish(e0 + 4u * tid, x, x0, x0b, y, cp, mv, p1, p2, jj);
        }
      }
    }
  }
}

// <1024 subsequences per group, 256 consumer threads + producer warp, 2 CTAs per SM, 96 registers>.  Measured and
// dropped: a 112-register ceiling (one CTA per SM, 70 us), 2048-subsequence groups with 17 warps (does not launch) and
// two subsequences per thread in groups of 448 (48.7 vs 43.6 us per launch at R=128).
template <typename H, bool kFirst, bool kNext>
__global__ void __launch_bounds__(1024 / 4 + 32, 2) substep_torch_tma_kernel(const SubstepArgs a, const TorchTmaGeom tg) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t full[4], empty[4];
  torch_tma_body<H, kFirst, kNext, 1024>(a, tg, smem_raw, full, empty);
}

// ---- TORCH, 128-bit LDG path ----------------------------------------------------------------------
// Thread (t, k) of this kernel IS torch's thread t at its k-th call: it generates that call's four normals
// (planes 4k..4k+3), then the four lanes of a quad transpose them with shuffles so that lane q ends up with
// plane 4k+q of torch threads t0..t0+3 -- four CONSECUTIVE elements, i.e. one float4 -- and runs the same
// vector body as the other modes.
// 4x4 transpose across the 4 lanes of a quad, two butterfly stages, register indices all static:
// in: v[j] = my normal for plane j;  out: v[i] = plane q's normal of quad lane i.
__device__ __forceinline__ void quad_transpose(float (&v)[4], uint32_t q) {
  const bool b0 = (q & 1u) != 0, b1 = (q & 2u) != 0;
  // stage 1: 2x2 blocks between lanes q and q^1
  float s0 = b0 ? v[0] : v[1], s1 = b0 ? v[2] : v[3];
  s0 = __shfl_xor_sync(0xffffffffu, s0, 1);
  s1 = __shfl_xor_sync(0xffffffffu, s1, 1);
  v[0] = b0 ? s0 : v[0]; v[1] = b0 ? v[1] : s0;
  v[2] = b0 ? s1 : v[2]; v[3] = b0 ? v[3] : s1;
  // stage 2: 2x2 blocks of pairs between lanes q and q^2
  float u0 = b1 ? v[0] : v[2], u1 = b1 ? v[1] : v[3];
  u0 = __shfl_xor_sync(0xffffffffu, u0, 2);
  u1 = __shfl_xor_sync(0xffffffffu, u1, 2);
  v[0] = b1 ? u0 : v[0]; v[2] = b1 ? v[2] : u0;
  v[1] = b1 ? u1 : v[1]; v[3] = b1 ? v[3] : u1;
}

template <typename H, bool kFirst, bool kNext>
__global__ void __launch_bounds__(kBlock) substep_torchvec_kernel(const SubstepArgs a) {
  pdl_prologue();
  const uint32_t T = a.torch_T;
  const uint32_t t = blockIdx.x * kBlock + threadIdx.x;  // torch thread == Philox subsequence (grid.x*256 == T)
  const uint32_t k = blockIdx.y;                          // index of the curand_normal4 call
  const uint32_t q = t & 3u;
  uint64_t seed = a.seed, o0 = a.draw0, o1 = a.draw1;
  if (a.rng_state) {
    seed = a.rng_state[0];
    o0 += a.rng_state[1];
    o1 += a.rng_state[1];
  }
  const float4 n1 = torch_normal4(seed, o0, t, k);
  float4 n2 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (kNext) n2 = torch_normal4(seed, o1, t, k);
  float xi1[4] = {n1.x, n1.y, n1.z, n1.w};
  float xi2[4] = {n2.x, n2.y, n2.z, n2.w};
  quad_transpose(xi1, q);
  if (kNext) quad_transpose(xi2, q);
  const uint64_t e = (uint64_t)(t - q) + (uint64_t)(4u * k + q) * T;  // first of my 4 consecutive elements
  if (e >= a.g.total) return;
  substep_vector<4, H, kFirst, kNext, false>(a, (uint32_t)e, xi1, xi2);
}

// ---- TORCH, scalar fallback: torch.randn_like's own thread<->element mapping ---
// thread t of T handles elements t, t+T, t+2T, t+3T (one curand_normal4) per
// 4T-stride iteration, exactly like distribution_elementwise_grid_stride_kernel
// (ATen/native/cuda/DistributionTemplates.h), so one Philox call feeds 4
// elements and the stream matches the eager reference on the same generator.
template <typename H, bool kFirst, bool kNext>
__global__ void __launch_bounds__(kBlock) substep_torch_kernel(const SubstepArgs a) {
  pdl_prologue();
  const uint32_t T = a.torch_T;
  const uint32_t tid = blockIdx.x * kBlock + threadIdx.x;
  if (tid >= T) return;
  uint64_t seed = a.seed, o0 = a.draw0, o1 = a.draw1;
  if (a.rng_state) {
    seed = a.rng_state[0];
    o0 += a.rng_state[1];
    o1 += a.rng_state[1];
  }
  const H* x0p = static_cast<const H*>(a.x0);
  const H* x0bp = static_cast<const H*>(a.x0b);
  uint32_t call = 0;
  for (uint64_t base = tid; base < a.g.total; base += 4ull * T, ++call) {
    const float4 n1 = torch_normal4(seed, o0, tid, call);
    float4 n2 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (kNext) n2 = torch_normal4(seed, o1, tid, call);
#pragma unroll
    for (int ii = 0; ii < 4; ++ii) {
      const uint64_t li = base + (uint64_t)ii * T;
      if (li >= a.g.total) break;
      const uint32_t i = (uint32_t)li;
      uint32_t row, mi;
      locate(a.g, i, row, mi);
      RowCoef<kFirst, kNext> t;
      t.load(a.table + (size_t)row * LP_TABLE_STRIDE);
      float x = a.x[i];
      float x0 = widen(x0p[i]);
      float x0b = widen(x0bp[i]);
      if (a.use_cfg) cfg_combine(x0, x0b, a.cfg, a.cfg_big);
      const float y = __ldg(a.y + i);
      const bool known = __ldg(a.mask + mi) != 0;
      const float cp = kFirst ? 0.f : a.c[i];
      float cn, te;
      substep_element<kFirst, kNext>(x, x0, x0b, y, cp, known, pick(n1, ii), pick(n2, ii), t, cn, te);
      a.x[i] = x;
      if (kNext || a.store_c) a.c[i] = cn;
      if (a.x_copy) a.x_copy[i] = x;
      if (a.x0e) a.x0e[i] = te;
    }
  }
}

// ----------------------------------------------------------------------------
// launchers
// ----------------------------------------------------------------------------
// 2048-element tiles, 2 stages, 2 CTAs per SM: the fastest of the (tile, stages, CTAs per SM) geometries measured on the
// steady fp32 kernel; 1024x4x2, 4096x2x1, 2048x4x1 and 1024x3x3 lost
template <typename H, bool kFirst, bool kNext, bool kMerge>
int launch_substep_tma(const SubstepArgs& a, cudaStream_t s) {
  constexpr int kTile = 2048, kStages = 2, kMinBlocks = 2;
  const int dev = current_device();
  const size_t smem = sizeof(TmaStage<H, kTile>) * kStages;
  static bool configured[kMaxDevices] = {};  // per instantiation of this launcher
  ensure_dynamic_smem(substep_tma_kernel<H, kFirst, kNext, kMerge, kTile, kStages, kMinBlocks>, smem, dev, configured);
  TileGeom tg;
  tg.channels = a.g.per_row.d / a.g.spatial.d;
  tg.tiles_per_channel = (a.g.spatial.d + kTile - 1) / kTile;
  tg.n_tiles = (a.g.total / a.g.spatial.d) * tg.tiles_per_channel;
  unsigned grid = (unsigned)device_info(dev).sms * (unsigned)kMinBlocks;
  if (grid > tg.n_tiles) grid = tg.n_tiles;
  launch_kernel_smem(substep_tma_kernel<H, kFirst, kNext, kMerge, kTile, kStages, kMinBlocks>, dim3(grid), smem, s, a, tg);
  return check_launch();
}

// The TMA-staged variants need 16-byte aligned slices (spatial a multiple of 16), no side outputs, no row split;
// only worth it when there are enough tiles to keep a persistent grid busy.
inline bool tma_eligible(const SubstepArgs& a) {
  return g_opt_tma != 0 && geometry_tma(a.g, a.mask) && !a.x_copy && !a.x0e && a.g.total >= kTmaMinElements &&
         aligned16(a.x) && aligned16(a.x0) && aligned16(a.x0b) && aligned16(a.y) && (!a.c || aligned16(a.c));
}

template <int N, typename H, int kRng>
int launch_substep_vec(const SubstepArgs& a, bool first, bool next, bool merge, cudaStream_t s) {
  const unsigned grid = blocks_for((a.g.total + N - 1) / N);
  if constexpr (N == 4 && kRng == LP_RNG_PHILOX) {
    if (tma_eligible(a)) {
      if (first && next && merge) return launch_substep_tma<H, true, true, true>(a, s);
      if (first && next) return launch_substep_tma<H, true, true, false>(a, s);
      if (next && merge) return launch_substep_tma<H, false, true, true>(a, s);
      if (next) return launch_substep_tma<H, false, true, false>(a, s);
      if (first) return launch_substep_tma<H, true, false, false>(a, s);
      return launch_substep_tma<H, false, false, false>(a, s);
    }
  }
  if constexpr (kRng == LP_RNG_PHILOX) {
    if (merge) {
      if (first) launch_kernel(substep_kernel<N, H, LP_RNG_PHILOX, true, true, true>, dim3(grid), s, a);
      else launch_kernel(substep_kernel<N, H, LP_RNG_PHILOX, false, true, true>, dim3(grid), s, a);
      return check_launch();
    }
  }
  if (first && next) launch_kernel(substep_kernel<N, H, kRng, true, true>, dim3(grid), s, a);
  else if (first) launch_kernel(substep_kernel<N, H, kRng, true, false>, dim3(grid), s, a);
  else if (next) launch_kernel(substep_kernel<N, H, kRng, false, true>, dim3(grid), s, a);
  else launch_kernel(substep_kernel<N, H, kRng, false, false>, dim3(grid), s, a);
  return check_launch();
}

template <typename H, bool kFirst, bool kNext>
int launch_torch_tma(const SubstepArgs& a, uint32_t calls, cudaStream_t s) {
  const int dev = current_device();
  const size_t smem = sizeof(TorchSlot<H, 1024>) * 4;
  TorchTmaGeom tg;
  tg.groups_per_call = a.torch_T / 1024;
  tg.n_groups = calls * tg.groups_per_call;
  unsigned grid = (unsigned)device_info(dev).sms * 2u;
  if (grid > tg.n_groups) grid = tg.n_groups;
  static bool configured[kMaxDevices] = {};
  ensure_dynamic_smem(substep_torch_tma_kernel<H, kFirst, kNext>, smem, dev, configured);
  launch_kernel_ex(substep_torch_tma_kernel<H, kFirst, kNext>, dim3(grid), dim3(1024 / 4 + 32), smem, s, a, tg);
  return check_launch();
}

template <typename H>
int substep_dispatch(SubstepArgs& a, const lp_rng* rng, bool f, bool n, bool merge, bool v4, cudaStream_t s) {
  if (rng->mode == LP_RNG_TORCH) {
    int64_t grid = 0;
    if (int rc = torch_grid(a.g.total, -1, &grid, nullptr)) return rc;
    a.torch_T = (uint32_t)(grid * 256);
    const unsigned gb = (unsigned)grid;
    const uint64_t calls = ((uint64_t)a.g.total + 4ull * a.torch_T - 1) / (4ull * a.torch_T);
    if (v4 && tma_eligible(a) && a.torch_T % 1024 == 0 && a.g.spatial.d >= 64 && calls <= 0xffffffffull / 4) {
      if (f && n) return launch_torch_tma<H, true, true>(a, (uint32_t)calls, s);
      if (f) return launch_torch_tma<H, true, false>(a, (uint32_t)calls, s);
      if (n) return launch_torch_tma<H, false, true>(a, (uint32_t)calls, s);
      return launch_torch_tma<H, false, false>(a, (uint32_t)calls, s);
    }
    if (v4 && calls <= 65535) {
      const dim3 g2(gb, (unsigned)calls);
      if (f && n) launch_kernel(substep_torchvec_kernel<H, true, true>, dim3(g2), s, a);
      else if (f) launch_kernel(substep_torchvec_kernel<H, true, false>, dim3(g2), s, a);
      else if (n) launch_kernel(substep_torchvec_kernel<H, false, true>, dim3(g2), s, a);
      else launch_kernel(substep_torchvec_kernel<H, false, false>, dim3(g2), s, a);
      return check_launch();
    }
    if (f && n) launch_kernel(substep_torch_kernel<H, true, true>, dim3(gb), s, a);
    else if (f) launch_kernel(substep_torch_kernel<H, true, false>, dim3(gb), s, a);
    else if (n) launch_kernel(substep_torch_kernel<H, false, true>, dim3(gb), s, a);
    else launch_kernel(substep_torch_kernel<H, false, false>, dim3(gb), s, a);
    return check_launch();
  }
  if (rng->mode == LP_RNG_TAPE) {
    if (!rng->tape0 || (n && !rng->tape1)) return LP_ERR_INVALID;
    v4 = v4 && aligned16(rng->tape0) && (!n || aligned16(rng->tape1));
    return v4 ? launch_substep_vec<4, H, LP_RNG_TAPE>(a, f, n, false, s) : launch_substep_vec<1, H, LP_RNG_TAPE>(a, f, n, false, s);
  }
  if (rng->mode == LP_RNG_PHILOX) {
    return v4 ? launch_substep_vec<4, H, LP_RNG_PHILOX>(a, f, n, merge, s)
              : launch_substep_vec<1, H, LP_RNG_PHILOX>(a, f, n, merge, s);
  }
  return LP_ERR_INVALID;
}

static int substep_impl(float* x_model, const lp_heads* heads, const float* y, const uint8_t* mask, float* c_state,
                        float* x_copy, float* x0e_out, const float* table, const lp_dims* dims, const lp_rng* rng,
                        int flags, lp_stream_t stream) {
  if (!x_model || !heads || !heads->a || !y || !mask || !table || !rng) return LP_ERR_INVALID;
  if (flags & ~(LP_SUBSTEP_FIRST | LP_SUBSTEP_FUSE_NEXT | LP_SUBSTEP_STORE_C | LP_SUBSTEP_MERGE_NOISE))
    return LP_ERR_INVALID;
  const int dtype = heads->dtype;
  if (dtype != LP_DTYPE_F32 && dtype != LP_DTYPE_BF16 && dtype != LP_DTYPE_F16) return LP_ERR_INVALID;
  if (heads->combine && (dtype != LP_DTYPE_F32 || !heads->b || heads->b == heads->a)) return LP_ERR_INVALID;
  const bool merge = (flags & LP_SUBSTEP_MERGE_NOISE) != 0;
  if (merge && (!(flags & LP_SUBSTEP_FUSE_NEXT) || rng->mode != LP_RNG_PHILOX)) return LP_ERR_INVALID;
  const bool first = (flags & LP_SUBSTEP_FIRST) != 0;
  const bool has_next = (flags & LP_SUBSTEP_FUSE_NEXT) != 0;
  const void* x0 = heads->a;
  const void* x0_big = heads->b ? heads->b : heads->a;
  if ((!first || has_next || (flags & LP_SUBSTEP_STORE_C)) && !c_state) return LP_ERR_INVALID;
  SubstepArgs a;
  if (int rc = make_geometry(dims, a.g)) return rc;
  if (a.g.total == 0) return LP_OK;
  a.x = x_model; a.x0 = x0; a.x0b = x0_big; a.y = y; a.mask = mask; a.c = c_state;
  a.x_copy = x_copy; a.x0e = x0e_out; a.table = table;
  a.tape0 = rng->tape0; a.tape1 = rng->tape1; a.rng_state = rng->state;
  a.seed = rng->seed; a.draw0 = rng->draw0; a.draw1 = rng->draw1; a.torch_T = 0;
  a.store_c = (flags & LP_SUBSTEP_STORE_C) != 0;
  a.use_cfg = heads->combine != 0; a.cfg = heads->cfg; a.cfg_big = heads->cfg_big;
  cudaStream_t s = (cudaStream_t)stream;
  const bool v4 = geometry_vec4(a.g, mask) && aligned16(x_model) && head_aligned(x0, dtype) &&
                  head_aligned(x0_big, dtype) && aligned16(y) && (!c_state || aligned16(c_state)) &&
                  (!x_copy || aligned16(x_copy)) && (!x0e_out || aligned16(x0e_out));
  switch (dtype) {
    case LP_DTYPE_F32: return substep_dispatch<float>(a, rng, first, has_next, merge, v4, s);
    case LP_DTYPE_BF16: return substep_dispatch<__nv_bfloat16>(a, rng, first, has_next, merge, v4, s);
    default: return substep_dispatch<__half>(a, rng, first, has_next, merge, v4, s);
  }
}

}  // namespace lp

using namespace lp;

extern "C" int lp_substep(float* x_model, const lp_heads* heads, const float* y, const uint8_t* mask, float* c_state,
                          float* x_copy, float* x0e_out, const float* table, const lp_dims* dims, const lp_rng* rng,
                          int flags, lp_stream_t stream) {
  return substep_impl(x_model, heads, y, mask, c_state, x_copy, x0e_out, table, dims, rng, flags, stream);
}

extern "C" int lp_substep_f32(float* x_model, const float* x0, const float* x0_big, const float* y,
                              const uint8_t* mask, float* c_state, float* x_copy, float* x0e_out,
                              const float* table, const lp_dims* dims, const lp_rng* rng, int flags,
                              lp_stream_t stream) {
  lp_heads h = {x0, x0_big, LP_DTYPE_F32, 0, 0.f, 0.f};
  return substep_impl(x_model, &h, y, mask, c_state, x_copy, x0e_out, table, dims, rng, flags, stream);
}

extern "C" int lp_substep_cfg_f32(float* x_model, const float* cond, const float* uncond, float cfg, float cfg_big,
                                  const float* y, const uint8_t* mask, float* c_state, float* x_copy,
                                  float* x0e_out, const float* table, const lp_dims* dims, const lp_rng* rng,
                                  int flags, lp_stream_t stream) {
  lp_heads h = {cond, uncond, LP_DTYPE_F32, 1, cfg, cfg_big};
  return substep_impl(x_model, &h, y, mask, c_state, x_copy, x0e_out, table, dims, rng, flags, stream);
}
