// lanpaint_b200: everything of an outer step that is not the fused sub-step.
//   prologue_kernel     replace step + change of variables              lanpaint.py:85-99
//   boundary_kernel     final paste [+ CFG combine] [+ k-diffusion Euler update] [+ next replace step]
//                       lanpaint.py:151-157, sample_euler, lanpaint.py:85-94
//   advance_kernel      one un-fused advance_time_overdamped             lanpaint.py:232-254
//   stop_stats_kernel   early-stop masked reductions                     earlystop.py:32-55,238-313
#include "lp_common.cuh"

namespace lp {

// ---- prologue ----------------------------------------------------------------
template <int N>
__global__ void __launch_bounds__(kBlock) prologue_kernel(const float* x, const float* __restrict__ y,
                                                          const float* __restrict__ noise,
                                                          const uint8_t* __restrict__ mask, float* x_model,
                                                          float* x_copy, const float* __restrict__ table,
                                                          Geometry g) {
  pdl_prologue();
  const uint32_t i = (blockIdx.x * kBlock + threadIdx.x) * N;
  if (i >= g.total) return;
  uint32_t row, mi;
  locate(g, i, row, mi);
  const float rn = __ldg(table + (size_t)row * LP_TABLE_STRIDE + LP_T_REPN);
  const float ry = __ldg(table + (size_t)row * LP_TABLE_STRIDE + LP_T_REPY);
  float xv[N], yv[N], nv[N];
  bool known[N];
  load_f<N>(x, i, xv);
  load_f_ro<N>(y, i, yv);
  load_f_ro<N>(noise, i, nv);
  load_m<N>(mask, mi, known);
#pragma unroll
  for (int j = 0; j < N; ++j) xv[j] = known[j] ? fmaf(rn, nv[j], ry * yv[j]) : xv[j];
  store_f<N>(x_model, i, xv);
  if (x_copy) store_f<N>(x_copy, i, xv);
}

// ---- the boundary of an outer step ----------------------------------------------------
struct BoundaryArgs {
  const void* a;   // model_out (or cond)
  const void* b;   // uncond when combine
  const float* y;
  const float* noise;
  const uint8_t* mask;
  float* x;        // NULL: no Euler update
  float* out;      // NULL: nobody reads the denoised latent
  const float* next_table;  // NULL: no replace step of the next outer step
  float cfg, coef;
  int combine;
  Geometry g;
};

// per element: d = combine ? b + (a-b) cfg : a ; o = known ? y : d ; x += (x - o) coef ; x = known ? rn n + ry y : x
__device__ __forceinline__ void boundary_element(float a, float b, float y, float nz, bool known, float& x, float& o,
                                                 bool combine, float cfg, float coef, bool euler, bool next, float rn,
                                                 float ry) {
  const float d = combine ? __fadd_rn(b, __fmul_rn(__fsub_rn(a, b), cfg)) : a;
  o = known ? y : d;
  if (euler) x = fmaf(x - o, coef, x);
  if (next) x = known ? fmaf(rn, nz, ry * y) : x;
}

template <int N, typename H>
__global__ void __launch_bounds__(kBlock) boundary_kernel(const BoundaryArgs p) {
  pdl_prologue();
  const uint32_t i = (blockIdx.x * kBlock + threadIdx.x) * N;
  if (i >= p.g.total) return;
  uint32_t row, mi;
  locate(p.g, i, row, mi);
  bool known[N];
  load_m<N>(p.mask, mi, known);
  bool any_known = false, any_free = false;
#pragma unroll
  for (int j = 0; j < N; ++j) {
    any_known |= known[j];
    any_free |= !known[j];
  }
  const bool euler = p.x != nullptr, next = p.next_table != nullptr;
  float av[N], bv[N], yv[N], xv[N], nv[N], ov[N];
#pragma unroll
  for (int j = 0; j < N; ++j) av[j] = bv[j] = xv[j] = nv[j] = 0.f;
  load_f_ro<N>(p.y, i, yv);
  // free positions: the denoised output and the running state; known positions: the re-noised clean latent
  if (any_free) {
    load_head_ro<N, H>(static_cast<const H*>(p.a), i, av);
    if (p.combine) load_head_ro<N, H>(static_cast<const H*>(p.b), i, bv);
  }
  if (euler && (any_free || !next)) load_f<N>(p.x, i, xv);
  float rn = 0.f, ry = 0.f;
  if (next) {
    if (any_known) load_f_ro<N>(p.noise, i, nv);
    rn = __ldg(p.next_table + (size_t)row * LP_TABLE_STRIDE + LP_T_REPN);
    ry = __ldg(p.next_table + (size_t)row * LP_TABLE_STRIDE + LP_T_REPY);
  }
#pragma unroll
  for (int j = 0; j < N; ++j)
    boundary_element(av[j], bv[j], yv[j], nv[j], known[j], xv[j], ov[j], p.combine != 0, p.cfg, p.coef, euler, next, rn,
                     ry);
  if (p.out) store_f<N>(p.out, i, ov);
  if (euler) store_f<N>(p.x, i, xv);
}

template <typename H>
int boundary_dispatch(const BoundaryArgs& p, bool v4, cudaStream_t s) {
  if (v4) launch_kernel(boundary_kernel<4, H>, dim3(blocks_for(p.g.total / 4)), s, p);
  else launch_kernel(boundary_kernel<1, H>, dim3(blocks_for(p.g.total)), s, p);
  return check_launch();
}

static int boundary_impl(const lp_heads* mo, const float* y, const float* noise, const uint8_t* mask, float* x_inout,
                         float* out, float euler_coef, const float* next_table, const lp_dims* dims,
                         lp_stream_t stream) {
  if (!mo || !mo->a || !y || !mask) return LP_ERR_INVALID;
  if (!x_inout && !out) return LP_ERR_INVALID;
  if (next_table && (!noise || !x_inout)) return LP_ERR_INVALID;
  const int dtype = mo->dtype;
  if (dtype != LP_DTYPE_F32 && dtype != LP_DTYPE_BF16 && dtype != LP_DTYPE_F16) return LP_ERR_INVALID;
  if (mo->combine && (dtype != LP_DTYPE_F32 || !mo->b || mo->b == mo->a)) return LP_ERR_INVALID;
  BoundaryArgs p;
  if (int rc = make_geometry(dims, p.g)) return rc;
  if (p.g.total == 0) return LP_OK;
  p.a = mo->a; p.b = mo->combine ? mo->b : nullptr; p.y = y; p.noise = noise; p.mask = mask; p.x = x_inout; p.out = out;
  p.next_table = next_table; p.cfg = mo->cfg; p.coef = euler_coef; p.combine = mo->combine != 0;
  const bool v4 = geometry_vec4(p.g, mask) && head_aligned(p.a, dtype) && (!p.b || head_aligned(p.b, dtype)) &&
                  aligned16(y) && (!noise || aligned16(noise)) && (!x_inout || aligned16(x_inout)) &&
                  (!out || aligned16(out));
  cudaStream_t s = (cudaStream_t)stream;
  switch (dtype) {
    case LP_DTYPE_F32: return boundary_dispatch<float>(p, v4, s);
    case LP_DTYPE_BF16: return boundary_dispatch<__nv_bfloat16>(p, v4, s);
    default: return boundary_dispatch<__half>(p, v4, s);
  }
}

// ---- un-fused OU advance (advance_time_overdamped, lanpaint.py:232-254) --------
struct AdvanceArgs {
  float* x;
  const float* c;
  const uint8_t* mask;
  const float* table;
  const float* tape0;
  const uint64_t* rng_state;
  uint64_t seed, draw0;
  Geometry g;
  uint32_t torch_T;
  int half;
};

__device__ __forceinline__ float advance_element(float x, float c, bool known, float xi,
                                                 const float* __restrict__ t, int half) {
  const float* k = t + (known ? LP_T_CLS1 : LP_T_CLS0);
  const float e = __ldg(k + (half ? LP_C_EH : LP_C_EF));
  const float kk = __ldg(k + (half ? LP_C_KH : LP_C_KF));
  const float sd = __ldg(k + (half ? LP_C_SH : LP_C_SF));
  const float xt = x * __ldg(t + LP_T_INVS);
  return fmaf(e, xt, fmaf(kk, c, sd * xi)) * __ldg(t + LP_T_S);
}

template <int kRng>
__global__ void __launch_bounds__(kBlock) advance_kernel(const AdvanceArgs a) {
  pdl_prologue();
  const uint32_t i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= a.g.total) return;
  uint32_t row, mi;
  locate(a.g, i, row, mi);
  float xi;
  if (kRng == LP_RNG_TAPE) {
    xi = __ldg(a.tape0 + i);
  } else {
    uint64_t seed = a.seed, d0 = a.draw0;
    if (a.rng_state) {
      seed = a.rng_state[0];
      d0 += a.rng_state[1];
    }
    xi = pick(philox_normal4(seed, d0, i >> 2), i & 3);
  }
  a.x[i] = advance_element(a.x[i], __ldg(a.c + i), __ldg(a.mask + mi) != 0, xi,
                           a.table + (size_t)row * LP_TABLE_STRIDE, a.half);
}

__global__ void __launch_bounds__(kBlock) advance_torch_kernel(const AdvanceArgs a) {
  pdl_prologue();
  const uint32_t T = a.torch_T;
  const uint32_t tid = blockIdx.x * kBlock + threadIdx.x;
  if (tid >= T) return;
  uint64_t seed = a.seed, o0 = a.draw0;
  if (a.rng_state) {
    seed = a.rng_state[0];
    o0 += a.rng_state[1];
  }
  uint32_t call = 0;
  for (uint64_t base = tid; base < a.g.total; base += 4ull * T, ++call) {
    const float4 n1 = torch_normal4(seed, o0, tid, call);
#pragma unroll
    for (int ii = 0; ii < 4; ++ii) {
      const uint64_t li = base + (uint64_t)ii * T;
      if (li >= a.g.total) break;
      const uint32_t i = (uint32_t)li;
      uint32_t row, mi;
      locate(a.g, i, row, mi);
      a.x[i] = advance_element(a.x[i], __ldg(a.c + i), __ldg(a.mask + mi) != 0, pick(n1, ii),
                               a.table + (size_t)row * LP_TABLE_STRIDE, a.half);
    }
  }
}

// ---- early-stop statistics: two masked sums of squared differences ---------------
// Grid-stride over float4 groups; per-thread partials -> warp shuffle -> one smem slot per warp ->
// one atomicAdd(double) per block per sum (earlystop.py:51-55 _weighted_mse numerators).
struct StatsArgs {
  const float* a;
  const float* b;
  const uint8_t* mask;
  const uint8_t* ring;
  const float* table;
  double* sums;
  Geometry g;
};

template <int N>
__global__ void __launch_bounds__(kBlock) stop_stats_kernel(const StatsArgs s) {
  pdl_prologue();
  float acc_in = 0.f, acc_ring = 0.f;
  const uint32_t stride = gridDim.x * kBlock * N;
  for (uint32_t i = (blockIdx.x * kBlock + threadIdx.x) * N; i < s.g.total; i += stride) {
    uint32_t row, mi;
    locate(s.g, i, row, mi);
    float av[N], bv[N];
    bool known[N], on_ring[N];
    load_f_ro<N>(s.a, i, av);
    load_f_ro<N>(s.b, i, bv);
    load_m<N>(s.mask, mi, known);
    if (s.ring) {
      load_m<N>(s.ring, mi, on_ring);
    } else {
#pragma unroll
      for (int j = 0; j < N; ++j) on_ring[j] = false;
    }
    const float scale = s.table ? __ldg(s.table + (size_t)row * LP_TABLE_STRIDE + LP_T_INVS) : 1.f;
#pragma unroll
    for (int j = 0; j < N; ++j) {
      const float d = (av[j] - bv[j]) * scale;
      const float d2 = d * d;
      acc_in += known[j] ? 0.f : d2;
      acc_ring += on_ring[j] ? d2 : 0.f;
    }
  }
  __shared__ float part[2][kBlock / 32];
  acc_in = warp_sum(acc_in);
  acc_ring = warp_sum(acc_ring);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) {
    part[0][w] = acc_in;
    part[1][w] = acc_ring;
  }
  __syncthreads();
  if (w == 0) {
    float u = lane < kBlock / 32 ? part[0][lane] : 0.f;
    float v = lane < kBlock / 32 ? part[1][lane] : 0.f;
    u = warp_sum(u);
    v = warp_sum(v);
    if (lane == 0) {
      atomicAdd(s.sums + 0, (double)u);
      atomicAdd(s.sums + 1, (double)v);
    }
  }
}

}  // namespace lp

using namespace lp;

extern "C" int lp_prologue_f32(const float* x, const float* y, const float* noise, const uint8_t* mask,
                               float* x_model, float* x_copy, const float* table, const lp_dims* dims,
                               lp_stream_t stream) {
  if (!x || !y || !noise || !mask || !x_model || !table) return LP_ERR_INVALID;
  Geometry g;
  if (int rc = make_geometry(dims, g)) return rc;
  if (g.total == 0) return LP_OK;
  cudaStream_t s = (cudaStream_t)stream;
  const bool v4 = geometry_vec4(g, mask) && aligned16(x) && aligned16(y) && aligned16(noise) &&
                  aligned16(x_model) && (!x_copy || aligned16(x_copy));
  if (v4) launch_kernel(prologue_kernel<4>, dim3(blocks_for(g.total / 4)), s, x, y, noise, mask, x_model, x_copy, table, g);
  else launch_kernel(prologue_kernel<1>, dim3(blocks_for(g.total)), s, x, y, noise, mask, x_model, x_copy, table, g);
  return check_launch();
}

extern "C" int lp_boundary(const lp_heads* model_out, const float* y, const float* noise, const uint8_t* mask,
                           float* x_inout, float* out, float euler_coef, const float* next_table, const lp_dims* dims,
                           lp_stream_t stream) {
  return boundary_impl(model_out, y, noise, mask, x_inout, out, euler_coef, next_table, dims, stream);
}

extern "C" int lp_epilogue_f32(const float* model_out, const float* y, const uint8_t* mask, float* out,
                               const lp_dims* dims, lp_stream_t stream) {
  if (!out) return LP_ERR_INVALID;
  lp_heads h = {model_out, nullptr, LP_DTYPE_F32, 0, 0.f, 0.f};
  return boundary_impl(&h, y, nullptr, mask, nullptr, out, 0.f, nullptr, dims, stream);
}

extern "C" int lp_epilogue_euler_f32(const float* model_out, const float* y, const uint8_t* mask, float* x_inout,
                                     float* out, float euler_coef, const lp_dims* dims, lp_stream_t stream) {
  if (!x_inout) return LP_ERR_INVALID;
  lp_heads h = {model_out, nullptr, LP_DTYPE_F32, 0, 0.f, 0.f};
  return boundary_impl(&h, y, nullptr, mask, x_inout, out, euler_coef, nullptr, dims, stream);
}

extern "C" int lp_step_boundary_f32(const float* model_out, const float* y, const float* noise, const uint8_t* mask,
                                    float* x_inout, float* out, float euler_coef, const float* next_table,
                                    const lp_dims* dims, lp_stream_t stream) {
  if (!noise || !x_inout || !next_table) return LP_ERR_INVALID;
  lp_heads h = {model_out, nullptr, LP_DTYPE_F32, 0, 0.f, 0.f};
  return boundary_impl(&h, y, noise, mask, x_inout, out, euler_coef, next_table, dims, stream);
}

extern "C" int lp_epilogue_cfg_f32(const float* cond, const float* uncond, float cfg, const float* y,
                                   const uint8_t* mask, float* x_inout, float* out, float euler_coef,
                                   const lp_dims* dims, lp_stream_t stream) {
  if (!cond || !uncond || !out) return LP_ERR_INVALID;
  lp_heads h = {cond, uncond, LP_DTYPE_F32, 1, cfg, cfg};
  return boundary_impl(&h, y, nullptr, mask, x_inout, out, euler_coef, nullptr, dims, stream);
}

extern "C" int lp_advance_f32(float* x_model, const float* c_state, const uint8_t* mask, const float* table,
                              const lp_dims* dims, const lp_rng* rng, int half, lp_stream_t stream) {
  if (!x_model || !c_state || !mask || !table || !rng) return LP_ERR_INVALID;
  AdvanceArgs a;
  if (int rc = make_geometry(dims, a.g)) return rc;
  if (a.g.total == 0) return LP_OK;
  a.x = x_model; a.c = c_state; a.mask = mask; a.table = table; a.tape0 = rng->tape0;
  a.rng_state = rng->state; a.seed = rng->seed; a.draw0 = rng->draw0; a.torch_T = 0; a.half = half != 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (rng->mode == LP_RNG_TORCH) {
    int64_t grid = 0;
    if (int rc = torch_grid(a.g.total, -1, &grid, nullptr)) return rc;
    a.torch_T = (uint32_t)(grid * 256);
    launch_kernel(advance_torch_kernel, dim3((unsigned)grid), s, a);
  } else if (rng->mode == LP_RNG_TAPE) {
    if (!rng->tape0) return LP_ERR_INVALID;
    launch_kernel(advance_kernel<LP_RNG_TAPE>, dim3(blocks_for(a.g.total)), s, a);
  } else if (rng->mode == LP_RNG_PHILOX) {
    launch_kernel(advance_kernel<LP_RNG_PHILOX>, dim3(blocks_for(a.g.total)), s, a);
  } else {
    return LP_ERR_INVALID;
  }
  return check_launch();
}

extern "C" int lp_stop_stats_f32(const float* a, const float* b, const uint8_t* mask, const uint8_t* ring,
                                 const float* table, const lp_dims* dims, double* sums, lp_stream_t stream) {
  if (!a || !b || !mask || !sums) return LP_ERR_INVALID;
  StatsArgs s;
  if (int rc = make_geometry(dims, s.g)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(sums, 0, 2 * sizeof(double), st) != cudaSuccess) {
    check_launch();
    return LP_ERR_CUDA;
  }
  if (s.g.total == 0) return LP_OK;
  s.a = a; s.b = b; s.mask = mask; s.ring = ring; s.table = table; s.sums = sums;
  const int sms = device_info(current_device()).sms;
  const bool v4 = geometry_vec4(s.g, mask) && aligned16(a) && aligned16(b) && (!ring || aligned4(ring));
  const uint32_t groups = v4 ? s.g.total / 4 : s.g.total;
  unsigned grid = blocks_for(groups);
  const unsigned cap = (unsigned)sms * 8;  // persistent-sized: 8 CTAs of 256 threads per SM
  if (grid > cap) grid = cap;
  if (v4) launch_kernel(stop_stats_kernel<4>, dim3(grid), st, s);
  else launch_kernel(stop_stats_kernel<1>, dim3(grid), st, s);
  return check_launch();
}
