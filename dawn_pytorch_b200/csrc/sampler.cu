// DDIM and ancestral DDPM updates around the denoising UNet (reference U:1169-1205 and U:1072-1121): x0 prediction, dynamic
// thresholding with the exact 0.9-quantile of |x0| over the whole clip (torch.quantile semantics, linear interpolation), and
// the eta-noise (DDIM) or posterior-mean + sigma-noise (DDPM) update.  Both steps share the same select chain.
// Everything stays on the device: no host synchronisation inside a sampling step.
#include "common.cuh"
#include "sampler.cuh"
#include "../../include/dawn_unet.h"

#define DAWN_TRY(expr)         \
  do {                         \
    int _rc = (expr);          \
    if (_rc != 0) return _rc;  \
  } while (0)

namespace dawn {
namespace {

// keys[i] = |ca * x - cb * eps|  (x0 magnitude; non-negative floats order like their bit patterns).  kDevCoef: ca, cb are
// read from cab[0..1] in device memory (the DDPM step, whose per-step scalars a replayed graph cannot bake).
template <bool kDevCoef>
__global__ void x0_abs_kernel(const float* __restrict__ x, const float* __restrict__ eps, float ca, float cb,
                              const float* __restrict__ cab, long long n, uint32_t* __restrict__ keys) {
  if (kDevCoef) { ca = cab[0]; cb = cab[1]; }
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    keys[i] = __float_as_uint(fabsf(ca * x[i] - cb * eps[i]));
}

// one launch instead of a pageable-host memcpy + three memsets (keeps the step capturable in a CUDA graph)
__global__ void select_init_kernel(uint32_t* state, unsigned int* hist, unsigned long long* count_le, unsigned int* min_gt,
                                   unsigned long long lo) {
  hist[threadIdx.x] = 0;
  if (threadIdx.x == 0) {
    state[0] = 0u; state[1] = 0u; state[2] = (uint32_t)(lo & 0xFFFFFFFFull); state[3] = (uint32_t)(lo >> 32);
    *count_le = 0ull; *min_gt = 0xFFFFFFFFu;
  }
}

// state[0] = prefix value, state[1] = prefix mask, state[2..3] = remaining rank (64-bit), hist[256]
__global__ void radix_hist_kernel(const uint32_t* __restrict__ keys, long long n, const uint32_t* __restrict__ state, int shift,
                                  unsigned int* __restrict__ hist) {
  __shared__ unsigned int sh[256];
  sh[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t pv = state[0], pm = state[1];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t k = keys[i];
    if ((k & pm) == pv) atomicAdd(&sh[(k >> shift) & 255u], 1u);
  }
  __syncthreads();
  if (sh[threadIdx.x]) atomicAdd(&hist[threadIdx.x], sh[threadIdx.x]);
}

__global__ void radix_pick_kernel(uint32_t* state, int shift, unsigned int* hist) {
  if (threadIdx.x != 0) return;
  unsigned long long rank = ((unsigned long long)state[3] << 32) | state[2];
  unsigned long long cum = 0;
  int b = 0;
  for (; b < 256; ++b) {
    if (cum + hist[b] > rank) break;
    cum += hist[b];
  }
  if (b > 255) b = 255;
  rank -= cum;
  state[0] |= (uint32_t)b << shift;
  state[1] |= 255u << shift;
  state[2] = (uint32_t)rank; state[3] = (uint32_t)(rank >> 32);
  for (int i = 0; i < 256; ++i) hist[i] = 0;
}

// after the 4 digit passes state[0] is the key of order statistic `lo`.  next[0] = #keys <= it, next[1] = min key above it
__global__ void next_stat_kernel(const uint32_t* __restrict__ keys, long long n, const uint32_t* __restrict__ state,
                                 unsigned long long* __restrict__ count_le, unsigned int* __restrict__ min_gt) {
  const uint32_t v = state[0];
  unsigned long long c = 0;
  unsigned int m = 0xFFFFFFFFu;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t k = keys[i];
    if (k <= v) ++c; else m = min(m, k);
  }
  for (int o = 16; o > 0; o >>= 1) {
    c += __shfl_xor_sync(0xffffffffu, c, o);
    m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(count_le, c);
    atomicMin(min_gt, m);
  }
}

// s = max(1, lerp(v[lo], v[hi], w)) exactly as torch.quantile + clamp_(min=1)  (U:1186-1193)
__global__ void threshold_kernel(const uint32_t* state, const unsigned long long* count_le, const unsigned int* min_gt,
                                 long long lo, long long hi, float w, float* s_out) {
  const float vlo = __uint_as_float(state[0]);
  float vhi = vlo;
  if (hi > lo && *count_le < (unsigned long long)(lo + 2)) vhi = __uint_as_float(*min_gt);
  const float d = vhi - vlo;
  const float q = (w < 0.5f) ? (vlo + w * d) : (vhi - d * (1.0f - w));     // at::lerp
  *s_out = fmaxf(q, 1.0f);
}

// img = clamp(x0, -s, s)/s * sqrt(a_next) + c * eps + sigma * noise;  clamp == 0: x0 is used as predicted (clip_denoised=False, U:1183)
__global__ void ddim_update_kernel(float* __restrict__ x, const float* __restrict__ eps, const float* __restrict__ noise,
                                   const float* __restrict__ s_ptr, float ca, float cb, float sqrt_an, float c, float sigma,
                                   long long n, int clamp) {
  const float s = s_ptr ? *s_ptr : 1.0f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float e = eps[i];
    float x0 = ca * x[i] - cb * e;
    if (clamp) x0 = fminf(fmaxf(x0, -s), s) / s;
    float v = x0 * sqrt_an + c * e;
    if (noise) v += sigma * noise[i];
    x[i] = v;
  }
}

// x = c1 * clamp(x0, -s, s)/s + c2 * x + sigma * noise with x0 = ca*x - cb*eps  (U:1072-1085, 1113-1121); coef = {ca, cb, c1,
// c2, sigma} in device memory.  sigma is 0 at t = 0 (the reference's nonzero_mask), where the noise is not read at all.
__global__ void ddpm_update_kernel(float* __restrict__ x, const float* __restrict__ eps, const float* __restrict__ noise,
                                   const float* __restrict__ s_ptr, const float* __restrict__ coef, long long n, int clamp) {
  const float s = s_ptr ? *s_ptr : 1.0f;
  const float ca = coef[0], cb = coef[1], c1 = coef[2], c2 = coef[3], sigma = coef[4];
  const bool add_noise = noise != nullptr && sigma != 0.0f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float xi = x[i];
    float x0 = ca * xi - cb * eps[i];
    if (clamp) x0 = fminf(fmaxf(x0, -s), s) / s;
    float v = c1 * x0 + c2 * xi;
    if (add_noise) v += sigma * noise[i];
    x[i] = v;
  }
}

// slot <- table row *cursor, ++*cursor: one step of a replayed DDPM segment picks up its time index and coefficients
__global__ void ddpm_advance_kernel(const uint32_t* __restrict__ table, int* __restrict__ cursor, uint32_t* __restrict__ slot) {
  const int r = *cursor;
  for (int i = 0; i < kDdpmRowWords; ++i) slot[i] = table[(size_t)r * kDdpmRowWords + i];
  *cursor = r + 1;
}

int grid_blocks(long long n, int threads) { return (int)std::min<long long>((n + threads - 1) / threads, 148LL * 8); }

// The threshold s of one step: the q-quantile of |x0| over the n_global values of the WHOLE clip.  With a frame-sharded clip
// every rank histograms its own keys and the 256-bin digit histograms (4 passes), the count <= v and the min key above v are
// all-reduced through `red`, so every rank walks the identical radix-select and ends with the bit-identical threshold
// (SURVEY 8e-iii).  ca, cb by value, or (cab != nullptr) from device memory.  Writes *s_ptr = the device address of s, or
// nullptr when q <= 0 (no dynamic threshold).
int select_threshold(const float* x, const float* eps, float ca, float cb, const float* cab, int64_t n_local, int64_t n_global,
                     float q, void* scratch, cudaStream_t st, const DdimReduce* red, const float** s_ptr) {
  *s_ptr = nullptr;
  if (!(q > 0.f)) return 0;
  const long long n = n_local;
  const int threads = 256;
  const int blocks = grid_blocks(n, threads);
  // scratch layout (32-bit words): [0,4) select state | [4,260) histogram | [260,262) count_le (u64) | 262 min_gt | 263 s | [512, 512+n) keys
  uint32_t* base = (uint32_t*)scratch;
  uint32_t* state = base;
  unsigned int* hist = base + 4;
  unsigned long long* count_le = (unsigned long long*)(base + 260);
  unsigned int* min_gt = base + 262;
  float* s_out = (float*)(base + 263);
  uint32_t* keys = base + 512;
  // torch.quantile: ranks = q * (n - 1) evaluated in fp32 (ATen quantile_compute), lerp between floor and ceil
  const float rank_f = q * (float)(n_global - 1);
  const long long lo = (long long)floorf(rank_f), hi = (long long)ceilf(rank_f);
  const float w = rank_f - floorf(rank_f);
  select_init_kernel<<<1, 256, 0, st>>>(state, hist, count_le, min_gt, (unsigned long long)lo);
  if (cab) x0_abs_kernel<true><<<blocks, threads, 0, st>>>(x, eps, 0.f, 0.f, cab, n, keys);
  else x0_abs_kernel<false><<<blocks, threads, 0, st>>>(x, eps, ca, cb, nullptr, n, keys);
  for (int shift = 24; shift >= 0; shift -= 8) {
    radix_hist_kernel<<<blocks, 256, 0, st>>>(keys, n, state, shift, hist);
    if (red) DAWN_TRY(red->sum_u32(red->ctx, hist, 256, st));
    radix_pick_kernel<<<1, 32, 0, st>>>(state, shift, hist);
  }
  next_stat_kernel<<<blocks, threads, 0, st>>>(keys, n, state, count_le, min_gt);
  if (red) {
    DAWN_TRY(red->sum_u64(red->ctx, count_le, 1, st));
    DAWN_TRY(red->min_u32(red->ctx, min_gt, 1, st));
  }
  threshold_kernel<<<1, 1, 0, st>>>(state, count_le, min_gt, lo, hi, w, s_out);
  *s_ptr = s_out;
  return 0;
}

}  // namespace

// One DDIM update in place on x (n_local floats of this rank's frames of the (3, F, h, w) latent); the threshold is
// select_threshold's clip-wide quantile.
int ddim_step_impl(float* x, const float* eps, const float* noise, int64_t n_local, int64_t n_global, float ca, float cb,
                   float sqrt_an, float c, float sigma, float q, void* scratch, cudaStream_t st, const DdimReduce* red) {
  if (!x || !eps || !scratch || n_local <= 0 || n_global < n_local) { set_last_error("dawn_ddim_step: bad argument"); return -1; }
  const float* s_ptr = nullptr;
  DAWN_TRY(select_threshold(x, eps, ca, cb, nullptr, n_local, n_global, q, scratch, st, red, &s_ptr));
  ddim_update_kernel<<<grid_blocks(n_local, 256), 256, 0, st>>>(x, eps, noise, s_ptr, ca, cb, sqrt_an, c, sigma, n_local,
                                                                q < 0.f ? 0 : 1);
  DAWN_LAUNCH_OK();
  return 0;
}

// One ancestral DDPM update in place on x: the same select as the DDIM step, then the posterior update with the five
// coefficients {ca, cb, c1, c2, sigma} read from coef (device memory).
int ddpm_step_impl(float* x, const float* eps, const float* noise, int64_t n_local, int64_t n_global, const float* coef, float q,
                   void* scratch, cudaStream_t st, const DdimReduce* red) {
  if (!x || !eps || !coef || !scratch || n_local <= 0 || n_global < n_local) { set_last_error("dawn_ddpm_step: bad argument"); return -1; }
  const float* s_ptr = nullptr;
  DAWN_TRY(select_threshold(x, eps, 0.f, 0.f, coef, n_local, n_global, q, scratch, st, red, &s_ptr));
  ddpm_update_kernel<<<grid_blocks(n_local, 256), 256, 0, st>>>(x, eps, noise, s_ptr, coef, n_local, q < 0.f ? 0 : 1);
  DAWN_LAUNCH_OK();
  return 0;
}

int launch_ddpm_advance(const void* table, int* cursor, void* slot, cudaStream_t st) {
  ddpm_advance_kernel<<<1, 1, 0, st>>>((const uint32_t*)table, cursor, (uint32_t*)slot);
  DAWN_LAUNCH_OK();
  return 0;
}

}  // namespace dawn

using namespace dawn;

extern "C" {

// single-GPU entry (see include/dawn_unet.h); dawn_unet_ddim_step in unet.cu is the frame-sharded one
int dawn_ddim_step(float* x, const float* eps, const float* noise, int64_t n, float ca, float cb, float sqrt_an, float c,
                   float sigma, float q, void* scratch, void* stream) {
  return ddim_step_impl(x, eps, noise, n, n, ca, cb, sqrt_an, c, sigma, q, scratch, (cudaStream_t)stream, nullptr);
}

}  // extern "C"
