/* dawn_unet.h — C-ABI of the B200-native DAWN denoising UNet (one "denoising step").
 *
 * The reference has no FFI layer: its seam is the Python nn.Module `DynamicNfUnet3D`
 * (DM_3/modules/video_flow_diffusion_multiGPU_v0_crema_plus_faceemb_ca_multi_test.py:728-965) held by
 * `GaussianDiffusion.denoise_fn` (same file :1010) and `FlowDiffusion.unet`
 * (..._flow_fast_init_cond_test.py:140).  The entry points below are what a binding for that seam needs;
 * dawn_pytorch_b200/unet.py is the ctypes binding that keeps the reference's Python signature on top of them.
 * Plain pointers and sizes only; no torch types.  One handle per GPU, not thread-safe, stream-ordered,
 * no hidden host synchronisation inside forward calls.  All tensors are fp32; one clip (batch element) per call.
 *
 * Return value: 0 ok; -1 bad argument / unsupported configuration / wrong call order; -2 CUDA error.
 * dawn_last_error() returns a human-readable description of the last failure on this thread.
 */
#ifndef DAWN_UNET_H_
#define DAWN_UNET_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dawn_unet dawn_unet;

/* Constructor arguments of Unet3D.__init__ (reference :729-753) that change the network's shape. */
typedef struct {
  int dim;              /* 64 */
  int n_levels;         /* len(dim_mults) = 4 */
  int dim_mults[8];     /* (1,2,4,8) */
  int channels;         /* 275 = 3 + 256 + 16 */
  int cond_aud;         /* 1024 */
  int cond_pose;        /* 6 */
  int cond_eye;         /* 2 */
  int out_grid_dim;     /* 2 */
  int out_conf_dim;     /* 1 */
  int attn_heads;       /* 8  (only 8 supported) */
  int attn_dim_head;    /* 32 (only 32 supported) */
  int resnet_groups;    /* 8  (only 8 supported) */
  int init_kernel_size; /* 7 */
  int win_width;        /* 40: temporal attention attends |i-j| <= win_width (reference :117) */
} dawn_unet_cfg;

/* replaces Unet3D.__init__ / DynamicNfUnet3D.__init__ (reference :728-877, 959-963) */
int dawn_unet_create(const dawn_unet_cfg* cfg, dawn_unet** out);
void dawn_unet_destroy(dawn_unet* h);

/* replaces nn.Module.load_state_dict (unified_video_generator.py:527-528): `name` is the reference
 * state_dict key (SURVEY Appendix B), `host` a host pointer to the fp32 values, row-major in `shape`.
 * Two auxiliary host-computed tables use the same call:
 *   "aux.time_freqs"  (dim/2,)      SinusoidalPosEmb frequencies (reference :157-159)
 *   "aux.rel_bias"    (heads, 2w+1) RelativePositionBias values for rel = -w..w (reference :111-119)  */
int dawn_unet_set_param(dawn_unet* h, const char* name, const float* host, const int64_t* shape, int ndim);
/* repack all parameters into kernel layouts and upload; must follow the last set_param */
int dawn_unet_commit_params(dawn_unet* h);

/* replaces DynamicNfUnet3D.update_num_frames (reference :964-965) and fixes the latent size.
 * For a frame-sharded clip F is the LOCAL frame count of this rank. */
int dawn_unet_set_num_frames(dawn_unet* h, int F, int height, int width);

/* Exact frame sharding of ONE clip over `nranks` GPUs (no reference counterpart; SURVEY 8e): rank r owns the contiguous
 * global frames [r*F, (r+1)*F).  Every temporal attention exchanges its +-win_width boundary frames with the adjacent
 * ranks (ncclSend/ncclRecv) and every GroupNorm all-reduces its 16 partial sums (fp64), so the sharded forward equals the
 * single-GPU forward.  dawn_nccl_unique_id: call on one rank, broadcast the 128 bytes, then init_shard on every rank
 * (after set_num_frames with the local F).  All inputs/outputs of forward* are then the LOCAL frames. */
int dawn_nccl_unique_id(char* out128);
int dawn_unet_init_shard(dawn_unet* h, const char* id128, int nranks, int rank, int F_global);
/* Optional, after init_shard (one process per GPU on ONE node, 2..8 ranks): GroupNorm statistics are then all-reduced by a single
 * kernel over NVLink peer memory (every rank stores its 16 partial sums into every peer's mailbox and adds the mailboxes in rank
 * order: bit-identical on all ranks) instead of ncclAllReduce.  export: this rank's mailbox as a 64-byte cudaIpc handle; exchange the
 * handles (any host channel), then import all of them (nranks x 64 bytes, rank order) and put a barrier before the next forward. */
int dawn_unet_shard_ipc_export(dawn_unet* h, char* out64);
int dawn_unet_shard_ipc_import(dawn_unet* h, const char* handles);

/* Clip invariants (SURVEY §8 a2/a5): the 272 feature channels are identical for every frame and every
 * DDIM step (reference :1167 `fea.repeat`), and cross-attention keys/values depend only on `cond`.
 * fea: device (channels-3, height, width); cond: device (F, cond_dim).  Needed by dawn_unet_forward_x3. */
int dawn_unet_set_clip_invariants(dawn_unet* h, const float* fea, const float* cond, void* stream);

/* replaces Unet3D.forward / forward_with_cond_scale(cond_scale=1) (reference :879-956) for one clip:
 * x: device (channels, F, height, width); t: device int64[1]; cond: device (F, cond_dim);
 * out: device (out_grid_dim + out_conf_dim, F, height, width). */
int dawn_unet_forward(dawn_unet* h, const float* x, const int64_t* t, const float* cond, float* out, void* stream);

/* same function when the caller knows the clip invariants: x_t: device (3, F, height, width) */
int dawn_unet_forward_x3(dawn_unet* h, const float* x_t, const int64_t* t, float* out, void* stream);

/* end-to-end entry with HOST buffers (pinned recommended): copies x_t, fea, cond, t to the device,
 * runs set_clip_invariants + forward_x3 and copies the result back; returns after the stream is synchronised. */
int dawn_unet_forward_host(dawn_unet* h, const float* x_t, const float* fea, const float* cond, int64_t t, float* out);

/* debugging / sub-module parity: request a copy of an internal activation (names as in oracle/unet_oracle.py
 * taps, e.g. "downs.1.0") into dst (device, (C, F, h_l, w_l)) during the next forward calls; dst = NULL clears. */
int dawn_unet_set_tap(dawn_unet* h, const char* name, float* dst);
/* channels and spatial size of a tap for the current set_num_frames: writes C, h_l, w_l */
int dawn_unet_tap_shape(dawn_unet* h, const char* name, int* C, int* hl, int* wl);

/* Per-kernel-category timing with CUDA events on the launching stream (bench.py's roofline object).
 * enable(1) clears the counters and brackets every launch of the following forward calls with events;
 * read() synchronises on the last event and returns, per category, accumulated milliseconds, algorithmic
 * flops (2*MAC, counted once — not the 3 split-precision passes), algorithmic bytes and launch counts.
 * Arrays must hold DAWN_PROF_NCAT entries.  Category order: conv3x3, conv_other, qkv_proj, out_proj,
 * ca_gate, gn_hcond, attn_core, sla_context, gn_apply, rowstats, ca_rstd, misc, prep, temporal_fused_l0 (the fused
 * temporal attention launches at level 0, not counted in attn_core), conv3x3_l0 (dim -> dim 3x3 convs at level 0, not
 * counted in conv3x3). */
#define DAWN_PROF_NCAT 20
int dawn_unet_profile_enable(dawn_unet* h, int on);
int dawn_unet_profile_read(dawn_unet* h, double* ms, double* flops, double* bytes, int64_t* count);

/* number of kernels launched by the last forward on this handle (bench.py's gpu_launches); after a sampler launch, the
 * forward launches of the DDIM graph or the node count of the DDPM segment graph */
int64_t dawn_unet_last_launch_count(dawn_unet* h);
/* bytes of device workspace currently held */
int64_t dawn_unet_workspace_bytes(dawn_unet* h);

/* One DDIM update around the UNet (reference GaussianDiffusion.ddim_sample :1169-1205), in place on x (device, n floats):
 *   x0 = ca*x - cb*eps;  s = max(1, quantile_q(|x0|)) over all n values (torch.quantile semantics) if q > 0, else 1;
 *   q < 0: x0 is neither clamped nor divided (the reference's clip_denoised=False, U:1183);
 *   x = clamp(x0,-s,s)/s * sqrt_an + c*eps + sigma*noise      (noise = NULL for the last step)
 * scratch: device buffer of n + 512 32-bit words.  No host synchronisation. */
int dawn_ddim_step(float* x, const float* eps, const float* noise, int64_t n, float ca, float cb, float sqrt_an, float c,
                   float sigma, float q, void* scratch, void* stream);

/* The same update for the frames a handle owns.  Unsharded handle: identical to dawn_ddim_step.  After dawn_unet_init_shard
 * the quantile spans the whole clip (n_local * nranks values): the radix-select's four 256-bin histograms and its two tail
 * statistics are all-reduced (NCCL, on `stream`), so every rank applies the bit-identical threshold.  Every rank must call
 * it with the same coefficients; `noise` is this rank's slice of the clip's noise. */
int dawn_unet_ddim_step(dawn_unet* h, float* x, const float* eps, const float* noise, int64_t n_local, float ca, float cb,
                        float sqrt_an, float c, float sigma, float q, void* scratch, void* stream);

/* The whole sampling loop of one clip (reference ddim_sample :1156-1208: 20 x [UNet forward + DDIM update]) captured
 * once into ONE CUDA graph and replayed per clip with a single launch: no host work between steps.  All addresses are
 * fixed at capture: x (3,F,h,w) start noise in / sample out, eps (3,F,h,w) scratch, noise_all ((nsteps-1) x 3*F*h*w,
 * slice k feeds step k; the last step adds none), t_all (nsteps int64, device), scratch (as dawn_ddim_step).
 * coef (host): nsteps x {ca, cb, sqrt_alpha_next, c, sigma}.  Per clip: fill x / noise_all, call
 * dawn_unet_set_clip_invariants (rewrites the same tables), then dawn_unet_sampler_launch(stream).
 * set_num_frames / commit_params / init_shard drop the graph. */
int dawn_unet_sampler_capture(dawn_unet* h, float* x, float* eps, const float* noise_all, const int64_t* t_all,
                              const float* coef, int nsteps, float q, void* scratch);
int dawn_unet_sampler_launch(dawn_unet* h, void* stream);

/* One ancestral DDPM update (reference p_sample :1113-1121 over p_mean_variance / q_posterior :1072-1107), in place on x:
 *   x0 = ca*x - cb*eps;  s as in dawn_ddim_step (q > 0: max(1, quantile_q(|x0|)), q = 0: 1, q < 0: no clamp);
 *   x = c1 * clamp(x0,-s,s)/s + c2*x + sigma*noise
 * coef: DEVICE pointer to {ca, cb, c1, c2, sigma} (sqrt_recip_alphas_cumprod[t], sqrt_recipm1_alphas_cumprod[t],
 * posterior_mean_coef1[t], posterior_mean_coef2[t], (t > 0) * exp(0.5 * posterior_log_variance_clipped[t])), so a loop
 * keeps its whole table on the device.  sigma == 0 (t = 0) reads no noise; noise may then be NULL.  Unsharded handle: the
 * plain step; after dawn_unet_init_shard the quantile spans the whole clip exactly as in dawn_unet_ddim_step.
 * scratch as dawn_ddim_step.  No host synchronisation. */
int dawn_unet_ddpm_step(dawn_unet* h, float* x, const float* eps, const float* noise, int64_t n_local, const float* coef, float q,
                        void* scratch, void* stream);

/* A segment of the ancestral loop captured as the handle's sampler graph (replaces any captured DDIM loop; replay it with
 * dawn_unet_sampler_launch).  The graph holds ksteps x [advance, forward_x3, dawn_unet_ddpm_step] and bakes no per-step value:
 * table (device) holds one row of 8 32-bit words per loop step, {t (int64), ca, cb, c1, c2, sigma, unused}; each step copies
 * row *cursor (device int) into slot (device, 8 words), increments *cursor, and runs the forward at slot's t and the update
 * with slot's coefficients.  Step j of a segment adds noise_ring slice j (ksteps x 3*F*h*w floats).  Per clip: set
 * *cursor = 0, then per segment refill noise_ring and launch; launch m runs table rows [m*ksteps, (m+1)*ksteps).  x, eps,
 * scratch as dawn_unet_sampler_capture.  set_num_frames / commit_params / init_shard drop the graph. */
int dawn_unet_ddpm_capture(dawn_unet* h, float* x, float* eps, const float* noise_ring, const void* table, int* cursor, void* slot,
                           int ksteps, float q, void* scratch);

/* self-test of the tcgen05 contraction kernel against the mma.sync kernel on a random k x k convolution
 * (F frames of H x W, Cin -> N channels); reports max |difference| (outputs and, if requested, GroupNorm sums). */
int dawn_selftest_tc_gemm(int F, int H, int W, int Cin, int N, int ksize, int with_stats, float* max_abs_diff, float* max_abs_ref);

/* self-test of the tensor-core attention core against the SIMT fp32 kernel on random q/k/v:
 * temporal != 0: nseq pixel sequences of L frames, band 40 with bias; else nseq frames of L tokens, full attention */
int dawn_selftest_attention(int nseq, int L, int temporal, float* max_abs_diff, float* max_abs_ref);

/* work decomposition of the tcgen05 temporal-attention kernel (host only): out receives 14 ints per segment
 * {w0, wn, qa, qb, tile0{r0, r1, q0, q1, kb}, tile1{r0, r1, q0, q1, kb}} (room for 16 segments); returns the segment count, 0 = unsupported. */
int dawn_temporal_tc_plan(int F, int band, int q_lo, int q_hi, int* out);

/* self-test of the tcgen05 temporal-attention kernel (64-channel levels) on random data: err[0] projection accumulator (relative),
 * err[1] scores, err[2] attention output, err[3] layer output of pixel 0 (all absolute, against a double-precision host computation),
 * err[4] all pixels against the mma.sync kernel (-1 where it does not support the shape), err[5] NaN count.
 * trace48 / ms (optional, both or neither): cycle counters of CTA 0 and the duration of a second, un-instrumented-output run. */
int dawn_selftest_temporal_tc(int F, int P, int band, int q_lo, int q_hi, float* err, float* max_abs_ref, unsigned long long* trace48,
                              float* ms);

const char* dawn_last_error(void);
const char* dawn_build_info(void);

#ifdef __cplusplus
}
#endif
#endif /* DAWN_UNET_H_ */
