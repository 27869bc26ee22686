// lanpaint_b200: library plumbing (options, status, per-device facts, geometry) and the small utility kernels.
#include "lp_common.cuh"

namespace lp {

thread_local int g_last_cuda_error = 0;

// process-wide switches, initialised from the environment, adjustable through lp_set_option()
int g_opt_pdl = [] {
  const char* e = getenv("LANPAINT_B200_PDL");
  return (e && e[0] == '0') ? 0 : 1;
}();
int g_opt_tma = [] {
  const char* e = getenv("LANPAINT_B200_TMA");
  return e ? atoi(e) : 1;
}();

int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  return dev;
}

const DeviceInfo& device_info(int device) {
  static DeviceInfo info[kMaxDevices] = {};
  static DeviceInfo fallback = {148, 2048};
  if (device < 0 || device >= kMaxDevices) return fallback;
  DeviceInfo& d = info[device];
  if (d.sms == 0) {  // benign race: every thread writes the same values
    int sms = 0, tpsm = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess ||
        cudaDeviceGetAttribute(&tpsm, cudaDevAttrMaxThreadsPerMultiProcessor, device) != cudaSuccess) {
      g_last_cuda_error = static_cast<int>(cudaGetLastError());
      return fallback;
    }
    d.threads_per_sm = tpsm;
    d.sms = sms;
  }
  return d;
}

// Exact for every n < 2^31: with l = ceil(log2 d), mul = floor(2^(31+l)/d) + 1 < 2^32 and the error
// n * eps / 2^(31+l) stays below 1/d.  d == 1 is flagged with mul == 0.
FastDiv make_fastdiv(uint32_t d) {
  FastDiv f{d, 0u, 0u};
  if (d <= 1) return f;
  uint32_t l = 0;
  while ((1ull << l) < d) ++l;
  const unsigned shift = 31 + l;
  f.mul = static_cast<uint32_t>(((1ull << shift) / d) + 1);
  f.shift = l - 1;
  return f;
}

int make_geometry(const lp_dims* d, Geometry& g) {
  if (!d || d->n_rows < 0 || d->per_row <= 0 || d->spatial <= 0) return LP_ERR_INVALID;
  if (d->per_row % d->spatial != 0) return LP_ERR_INVALID;
  if (d->mask_row_stride < 0 || d->mask_channel_stride < 0) return LP_ERR_INVALID;
  const int64_t total = d->n_rows * d->per_row;
  const int64_t mask_extent = d->n_rows * d->mask_row_stride + d->per_row;  // loose upper bound
  if (total >= (int64_t(1) << 31) || mask_extent >= (int64_t(1) << 31)) return LP_ERR_UNSUPPORTED;
  g.total = static_cast<uint32_t>(total);
  g.per_row = make_fastdiv(static_cast<uint32_t>(d->per_row));
  g.spatial = make_fastdiv(static_cast<uint32_t>(d->spatial));
  g.mask_row_stride = static_cast<uint32_t>(d->mask_row_stride);
  g.mask_channel_stride = static_cast<uint32_t>(d->mask_channel_stride);
  if (d->row_split < 0 || d->row_split > d->per_row) return LP_ERR_INVALID;
  g.n_rows = static_cast<uint32_t>(d->n_rows);
  g.row_split = static_cast<uint32_t>(d->row_split);
  return LP_OK;
}

// Geometry of torch's own randn kernel (ATen/native/cuda/DistributionTemplates.h: calc_execution_policy).
int torch_grid(int64_t numel, int device, int64_t* grid, uint64_t* inc) {
  if (numel <= 0) return LP_ERR_INVALID;
  if (device < 0) device = current_device();
  if (device < 0) return LP_ERR_CUDA;
  const DeviceInfo& d = device_info(device);
  int64_t g = (numel + 255) / 256;
  const int64_t cap = int64_t(d.sms) * (d.threads_per_sm / 256);
  if (g > cap) g = cap;
  if (grid) *grid = g;
  if (inc) *inc = (uint64_t)(((numel - 1) / (256 * g * 4) + 1) * 4);
  return LP_OK;
}

__global__ void __launch_bounds__(kBlock) pack_mask_kernel(const float* __restrict__ m, uint8_t* out,
                                                           uint32_t n, int invert) {
  pdl_prologue();
  const uint32_t i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  const bool hi = __ldg(m + i) > 0.5f;
  out[i] = (hi != (invert != 0)) ? 1 : 0;
}

__global__ void __launch_bounds__(kBlock) fill_normal_philox_kernel(float* out, uint32_t n, uint64_t seed,
                                                                    uint64_t draw, const uint64_t* st) {
  pdl_prologue();
  const uint32_t i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  if (st) {
    seed = st[0];
    draw += st[1];
  }
  out[i] = pick(philox_normal4(seed, draw, i >> 2), i & 3);
}

__global__ void __launch_bounds__(kBlock) fill_normal_torch_kernel(float* out, uint32_t n, uint64_t seed,
                                                                   uint64_t offset, const uint64_t* st,
                                                                   uint32_t T) {
  pdl_prologue();
  const uint32_t tid = blockIdx.x * kBlock + threadIdx.x;
  if (tid >= T) return;
  if (st) {
    seed = st[0];
    offset += st[1];
  }
  uint32_t call = 0;
  for (uint64_t base = tid; base < n; base += 4ull * T, ++call) {
    const float4 r = torch_normal4(seed, offset, tid, call);
#pragma unroll
    for (int ii = 0; ii < 4; ++ii) {
      const uint64_t li = base + (uint64_t)ii * T;
      if (li < n) out[li] = pick(r, ii);
    }
  }
}

// bitwise comparison of the FP32x2 Box-Muller with the scalar cuRAND form over pseudo-random and edge-case inputs
__global__ void __launch_bounds__(kBlock) selftest_box_muller_kernel(uint64_t n, uint64_t seed, unsigned long long* bad) {
  const uint64_t gid = (uint64_t)blockIdx.x * kBlock + threadIdx.x;
  const uint64_t stride = (uint64_t)gridDim.x * kBlock;
  unsigned long long mine = 0;
  for (uint64_t i = gid; i < n; i += stride) {
    uint4 r = philox4x32_10(make_uint4((uint32_t)i, (uint32_t)(i >> 32), 0x5eedu, 0u),
                            make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    if (i < 4096) {  // edge cases: the extremes of u and v in every combination, u == 1 (log = 0), smallest u
      const uint32_t edge[8] = {0u, 1u, 0x7fffffffu, 0x80000000u, 0xffffff00u, 0xffffff7fu, 0xffffff80u, 0xffffffffu};
      r.x = edge[i & 7];
      r.y = edge[(i >> 3) & 7];
      r.z = edge[(i >> 6) & 7];
      r.w = edge[(i >> 9) & 7];
    }
    const float2 a = box_muller_curand(r.x, r.y), b = box_muller_curand(r.z, r.w);
    float2 c, d;
    box_muller_curand_x2(r.x, r.y, r.z, r.w, c, d);
    mine += (__float_as_uint(a.x) != __float_as_uint(c.x)) + (__float_as_uint(a.y) != __float_as_uint(c.y)) +
            (__float_as_uint(b.x) != __float_as_uint(d.x)) + (__float_as_uint(b.y) != __float_as_uint(d.y));
  }
  if (mine) atomicAdd(bad, mine);
}

template <int N, typename H>
__global__ void __launch_bounds__(kBlock) synth_denoiser_kernel(const float* __restrict__ x, H* h0, H* h1, uint32_t n,
                                                                float a0, float b0, float c0, float a1, float c1) {
  pdl_prologue();
  const uint32_t i = (blockIdx.x * kBlock + threadIdx.x) * N;
  if (i >= n) return;
  float xv[N], u[N], w[N];
  load_f_ro<N>(x, i, xv);
#pragma unroll
  for (int j = 0; j < N; ++j) {
    u[j] = fmaf(a0, xv[j], fmaf(b0, tanhf(xv[j]), c0));
    w[j] = fmaf(a1, xv[j], c1);
  }
  if constexpr (sizeof(H) == 4) {
    store_f<N>(reinterpret_cast<float*>(h0), i, u);
    if (h1) store_f<N>(reinterpret_cast<float*>(h1), i, w);
  } else {
#pragma unroll
    for (int j = 0; j < N; ++j) {   // narrow stores of N consecutive 16-bit values
      if constexpr (sizeof(H) == 2) {
        h0[i + j] = H(u[j]);
        if (h1) h1[i + j] = H(w[j]);
      }
    }
  }
}

template <typename H>
int launch_synth(const float* x, void* h0, void* h1, int64_t n, const float* coef, cudaStream_t s) {
  const bool v4 = n % 4 == 0 && aligned16(x) && aligned16(h0) && (!h1 || aligned16(h1));
  if (v4)
    launch_kernel(synth_denoiser_kernel<4, H>, dim3(blocks_for((uint32_t)n / 4)), s, x, static_cast<H*>(h0),
                  static_cast<H*>(h1), (uint32_t)n, coef[0], coef[1], coef[2], coef[3], coef[4]);
  else
    launch_kernel(synth_denoiser_kernel<1, H>, dim3(blocks_for((uint32_t)n)), s, x, static_cast<H*>(h0),
                  static_cast<H*>(h1), (uint32_t)n, coef[0], coef[1], coef[2], coef[3], coef[4]);
  return check_launch();
}

}  // namespace lp

// ============================================================================
// C ABI
// ============================================================================
using namespace lp;

extern "C" int lp_abi_version(void) { return LP_ABI_VERSION; }

extern "C" const char* lp_status_string(int status) {
  switch (status) {
    case LP_OK: return "ok";
    case LP_ERR_INVALID: return "invalid argument";
    case LP_ERR_ALIGNMENT: return "misaligned pointer";
    case LP_ERR_CUDA: return "CUDA launch failed (see lp_last_cuda_error)";
    case LP_ERR_UNSUPPORTED: return "unsupported size (>= 2^31 elements)";
    default: return "unknown status";
  }
}

extern "C" int lp_last_cuda_error(void) { return g_last_cuda_error; }

extern "C" int lp_set_option(const char* name, int value) {
  if (!name) return LP_ERR_INVALID;
  const auto eq = [&](const char* k) { int i = 0; while (k[i] && name[i] == k[i]) ++i; return !k[i] && !name[i]; };
  if (eq("pdl")) { g_opt_pdl = value; return LP_OK; }
  if (eq("tma")) { g_opt_tma = value; return LP_OK; }
  return LP_ERR_INVALID;
}

extern "C" int64_t lp_selftest_index_math(int64_t samples) {
  int64_t bad = 0;
  auto check = [&](uint32_t n, uint32_t d) {
    const FastDiv f = make_fastdiv(d);
    const uint32_t q = f.mul ? (uint32_t)((((uint64_t)n * f.mul) >> 32) >> f.shift) : n;  // == FastDiv::div
    if (q != n / d) ++bad;
  };
  const uint32_t ds[] = {1u, 2u, 3u, 4u, 5u, 7u, 35u, 105u, 1024u, 3600u, 16384u, 65536u, 75600u, 1209600u,
                         (1u << 30), (1u << 31) - 1u, 0x7fffffffu, 1000003u};
  const uint32_t ns[] = {0u, 1u, 2u, 3u, 1023u, 65535u, 65536u, (1u << 31) - 1u, (1u << 31) - 2u, 0x40000000u};
  for (uint32_t d : ds)
    for (uint32_t n : ns) {
      check(n, d);
      if (d > 1 && n >= d) { check(n - n % d, d); check(n - n % d - 1, d); }
    }
  uint64_t st = 0x9E3779B97F4A7C15ull;
  for (int64_t k = 0; k < samples; ++k) {
    st = st * 6364136223846793005ull + 1442695040888963407ull;
    const uint32_t n = (uint32_t)(st >> 33);                       // < 2^31
    st = st * 6364136223846793005ull + 1442695040888963407ull;
    uint32_t d = (uint32_t)(st >> 33) >> ((st >> 20) & 31);        // all magnitudes
    if (d == 0) d = 1;
    check(n, d);
  }
  return bad;
}

extern "C" int lp_selftest_box_muller(int64_t n, uint64_t seed, unsigned long long* mismatches_dev, lp_stream_t stream) {
  if (n < 0 || !mismatches_dev) return LP_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaMemsetAsync(mismatches_dev, 0, sizeof(unsigned long long), s) != cudaSuccess) return (check_launch(), LP_ERR_CUDA);
  if (n == 0) return LP_OK;
  const unsigned grid = (unsigned)device_info(current_device()).sms * 8u;
  launch_kernel(selftest_box_muller_kernel, dim3(grid), s, (uint64_t)n, seed, mismatches_dev);
  return check_launch();
}

extern "C" int lp_torch_randn_geometry(int64_t numel, int device, int64_t* grid_out, uint64_t* increment_out) {
  return torch_grid(numel, device, grid_out, increment_out);
}

extern "C" int lp_pack_mask_f32(const float* mask_f32, uint8_t* mask_u8, int64_t n, int invert,
                                lp_stream_t stream) {
  if (!mask_f32 || !mask_u8 || n < 0) return LP_ERR_INVALID;
  if (n >= (int64_t(1) << 31)) return LP_ERR_UNSUPPORTED;
  if (n == 0) return LP_OK;
  launch_kernel(pack_mask_kernel, dim3(blocks_for((uint32_t)n)), (cudaStream_t)stream, mask_f32, mask_u8,
                                                                                 (uint32_t)n, invert);
  return check_launch();
}

extern "C" int lp_fill_normal_f32(float* out, int64_t n, const lp_rng* rng, lp_stream_t stream) {
  if (!out || !rng || n < 0) return LP_ERR_INVALID;
  if (n >= (int64_t(1) << 31)) return LP_ERR_UNSUPPORTED;
  if (n == 0) return LP_OK;
  cudaStream_t s = (cudaStream_t)stream;
  if (rng->mode == LP_RNG_PHILOX) {
    launch_kernel(fill_normal_philox_kernel, dim3(blocks_for((uint32_t)n)), s, out, (uint32_t)n, rng->seed,
                                                                        rng->draw0, rng->state);
    return check_launch();
  }
  if (rng->mode == LP_RNG_TORCH) {
    int64_t grid = 0;
    if (int rc = torch_grid(n, -1, &grid, nullptr)) return rc;
    launch_kernel(fill_normal_torch_kernel, dim3((unsigned)grid), s, out, (uint32_t)n, rng->seed, rng->draw0,
                                                              rng->state, (uint32_t)(grid * 256));
    return check_launch();
  }
  return LP_ERR_INVALID;
}

extern "C" int lp_synth_denoiser(const float* x, void* h0, void* h1, int dtype, int64_t n, const float* coef,
                                 lp_stream_t stream) {
  if (!x || !h0 || !coef || n < 0) return LP_ERR_INVALID;
  if (n >= (int64_t(1) << 31)) return LP_ERR_UNSUPPORTED;
  if (n == 0) return LP_OK;
  cudaStream_t s = (cudaStream_t)stream;
  switch (dtype) {
    case LP_DTYPE_F32: return launch_synth<float>(x, h0, h1, n, coef, s);
    case LP_DTYPE_BF16: return launch_synth<__nv_bfloat16>(x, h0, h1, n, coef, s);
    case LP_DTYPE_F16: return launch_synth<__half>(x, h0, h1, n, coef, s);
    default: return LP_ERR_INVALID;
  }
}

extern "C" int lp_synth_denoiser_f32(const float* x, float* h0, float* h1, int64_t n, const float* coef,
                                     lp_stream_t stream) {
  return lp_synth_denoiser(x, h0, h1, LP_DTYPE_F32, n, coef, stream);
}
