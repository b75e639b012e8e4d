// DDIM / DDPM updates around the UNet (sampler.cu): shared between the single-GPU C entry and the frame-sharded one in unet.cu.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

namespace dawn {

// cross-rank reductions of the exact radix-select (in place, stream-ordered); ctx is the caller's communicator
struct DdimReduce {
  void* ctx;
  int (*sum_u32)(void* ctx, unsigned int* buf, size_t n, cudaStream_t st);
  int (*sum_u64)(void* ctx, unsigned long long* buf, size_t n, cudaStream_t st);
  int (*min_u32)(void* ctx, unsigned int* buf, size_t n, cudaStream_t st);
};

int ddim_step_impl(float* x, const float* eps, const float* noise, int64_t n_local, int64_t n_global, float ca, float cb,
                   float sqrt_an, float c, float sigma, float q, void* scratch, cudaStream_t st, const DdimReduce* red);

// coef: device {ca, cb, c1, c2, sigma} of this step (see dawn_unet_ddpm_step)
int ddpm_step_impl(float* x, const float* eps, const float* noise, int64_t n_local, int64_t n_global, const float* coef, float q,
                   void* scratch, cudaStream_t st, const DdimReduce* red);

// One row of the per-loop DDPM table, 32-bit words: [0,2) t (int64) | 2 ca | 3 cb | 4 c1 | 5 c2 | 6 sigma | 7 unused
constexpr int kDdpmRowWords = 8;
constexpr int kDdpmCoefWord = 2;
// slot <- table[*cursor], ++*cursor (one thread; the first node of every step of a replayed segment)
int launch_ddpm_advance(const void* table, int* cursor, void* slot, cudaStream_t st);

}  // namespace dawn
