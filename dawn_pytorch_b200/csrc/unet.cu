// Host-side orchestration + C-ABI of the DAWN denoising UNet (reference U:728-965; see include/dawn_unet.h).
// One handle = one GPU = one clip at a time.  Weights are repacked once into GEMM-friendly layouts;
// activations live channels-last (F, H, W, C) in a workspace sized by dawn_unet_set_num_frames.
#include <dlfcn.h>
#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/dawn_unet.h"
#include "common.cuh"
#include "gemm.cuh"
#include "kernels.cuh"
#include "tc_gemm.cuh"
#include "temporal_fused.cuh"
#include "temporal_tc.cuh"
#include "sla_fused.cuh"
#include "ca_fused.cuh"
#include "sampler.cuh"

namespace dawn {

static thread_local std::string g_last_error;
void set_last_error(const std::string& s) { g_last_error = s; }

#define DAWN_CHECK(cond, msg)                 \
  do {                                        \
    if (!(cond)) {                            \
      ::dawn::set_last_error(msg);            \
      return -1;                              \
    }                                         \
  } while (0)
#define DAWN_TRY(expr)           \
  do {                           \
    int _rc = (expr);            \
    if (_rc != 0) return _rc;    \
  } while (0)

// ------------------------------------------------------------------ NCCL, resolved at run time (torch ships libnccl.so.2)
typedef struct ncclComm* ncclComm_t;
struct NcclUniqueId { char internal[128]; };
struct NcclApi {
  int (*GetUniqueId)(NcclUniqueId*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, NcclUniqueId, int) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
};
constexpr int kNcclUint32 = 3, kNcclUint64 = 5, kNcclFloat32 = 7, kNcclFloat64 = 8, kNcclSum = 0, kNcclMin = 3;   // nccl.h enums
static NcclApi g_nccl;
static int load_nccl() {
  if (g_nccl.ok) return 0;
  void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) { set_last_error(std::string("cannot load libnccl.so.2: ") + dlerror()); return -1; }
#define DAWN_NCCL_SYM(field, name)                                                        \
  g_nccl.field = reinterpret_cast<decltype(g_nccl.field)>(dlsym(lib, name));              \
  if (!g_nccl.field) { set_last_error(std::string("libnccl lacks ") + name); return -1; }
  DAWN_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
  DAWN_NCCL_SYM(CommInitRank, "ncclCommInitRank")
  DAWN_NCCL_SYM(CommDestroy, "ncclCommDestroy")
  DAWN_NCCL_SYM(AllReduce, "ncclAllReduce")
  DAWN_NCCL_SYM(Send, "ncclSend")
  DAWN_NCCL_SYM(Recv, "ncclRecv")
  DAWN_NCCL_SYM(GroupStart, "ncclGroupStart")
  DAWN_NCCL_SYM(GroupEnd, "ncclGroupEnd")
  DAWN_NCCL_SYM(GetErrorString, "ncclGetErrorString")
#undef DAWN_NCCL_SYM
  g_nccl.ok = true;
  return 0;
}
#define DAWN_NCCL_OK(expr)                                                                                   \
  do {                                                                                                       \
    int _r = (expr);                                                                                         \
    if (_r != 0) { ::dawn::set_last_error(std::string(#expr) + ": " + g_nccl.GetErrorString(_r)); return -2; } \
  } while (0)

struct HostParam {
  std::vector<float> data;
  std::vector<int64_t> shape;
  int64_t numel() const { int64_t n = 1; for (auto s : shape) n *= s; return n; }
};

struct Act {          // channels-last activation view: pixel stride ld, C channels, frame size H x W
  float* p = nullptr; int ld = 0; int C = 0; int H = 0; int W = 0;
};

struct ConvW { float* w = nullptr; float* b = nullptr; float* img = nullptr; float img_scale = 1.f; int K = 0, N = 0, ldb = 0; };

struct CrossAttnW { float *Wkv, *nkv, *qs, *ks, *Wout, *gout; };

struct ResBlockW {
  std::string name;
  int ci = 0, co = 0;
  bool cond = false, res = false;
  ConvW c1, c2, cres;
  float *gn1w = nullptr, *gn1b = nullptr, *gn2w = nullptr, *gn2b = nullptr;
  float *tW = nullptr, *tB = nullptr;
  float *mW[3] = {nullptr, nullptr, nullptr}, *mB[3] = {nullptr, nullptr, nullptr};   // pose, aud, eye MLPs
  float Wq_scale = 1.f;
  float *Wq = nullptr, *wsumq = nullptr, *Wq_img = nullptr;                              // [ci][192], [192]
  uint16_t* fWq = nullptr; float f_inv_wscale = 1.f;                                      // ca_fused.cu image (ci <= 128)
  CrossAttnW ca[3];
  // per-clip (depend on F / cond)
  float *film = nullptr, *kq = nullptr, *nkq = nullptr, *T = nullptr, *G = nullptr;
  int ldbT = 0;
  int st1 = 0, st2 = 0;
};

struct AttnW {     // temporal attention / mid spatial attention (U:648-725)
  int C = 0; float Wqkv_scale = 1.f; float *Wqkv = nullptr, *wsum = nullptr, *Wqkv_img = nullptr; ConvW out;
  // fused per-pixel kernel (temporal_fused.cu), 64-channel levels only
  uint16_t *fq = nullptr, *fo = nullptr; float f_inv_wscale = 1.f, f_inv_oscale = 1.f;
  // tcgen05 kernel (temporal_tc.cu): swizzled shared-memory images per head
  uint8_t *tq = nullptr, *to = nullptr; float t_inv_wscale = 1.f, t_inv_oscale = 1.f;
};
struct SlaW {      // spatial linear attention (U:602-627)
  int C = 0; float Wqkv_scale = 1.f; float *Wqkv = nullptr, *wsum = nullptr, *Wqkv_img = nullptr, *WoutT = nullptr, *bout = nullptr;
  // fused context kernel (sla_fused.cu), 64-channel levels: q-only projection + K/V weights as fp16 hi|lo images
  float *Wq = nullptr, *wsum_q = nullptr, *Wq_img = nullptr; float Wq_scale = 1.f;
  uint16_t* fkv = nullptr; float f_inv_wscale = 1.f;
  uint16_t* fq = nullptr; float fq_inv_wscale = 1.f;
};
struct UpW { ConvW cls[4]; ConvW all; };      // all: the four parity classes as one 3x3 conv with 4*C outputs (C = 64)

}  // namespace dawn

using namespace dawn;

// ---------------------------------------------------------------- GroupNorm all-reduce over peer memory (NVLink)
constexpr int kP2pMaxRanks = 8, kP2pSlots = 4;
struct P2pMail {
  double val[kP2pSlots][kP2pMaxRanks][16];     // [ring slot][source rank][8 groups x {sum, sum of squares}]
  unsigned int flag[kP2pSlots][kP2pMaxRanks];  // sequence number of the data in val[slot][source]
};
struct P2pPeers { P2pMail* m[kP2pMaxRanks]; };

// One warp.  seq = ++*ctr identifies this all-reduce on every rank (all ranks issue the same sequence of calls).  Lanes 0..15 push this
// rank's 16 doubles into every peer's mailbox (plain stores to peer-mapped memory travel over NVLink), a system-scope fence orders them
// before the flag store; then the warp waits for all sources' flags in its own mailbox and adds the 16-vectors in rank order, so every
// rank computes the bit-identical sum.  A rank cannot run more than one all-reduce ahead of the slowest one (it needs everyone's flag
// of the current call), so a ring of 4 slots is never overwritten while still being read.
__global__ void gn_p2p_allreduce_kernel(double* __restrict__ stats, P2pPeers peers, int rank, int nranks, unsigned int* ctr) {
  const int lane = threadIdx.x;
  unsigned int seq = 0;
  if (lane == 0) seq = ++(*ctr);
  seq = __shfl_sync(0xffffffffu, seq, 0);
  const int slot = seq % kP2pSlots;
  if (lane < 16) {
    const double v = stats[lane];
    for (int r = 0; r < nranks; ++r) peers.m[r]->val[slot][rank][lane] = v;
  }
  __threadfence_system();
  __syncwarp();
  if (lane < nranks) {
    volatile unsigned int* f = &peers.m[lane]->flag[slot][rank];
    *f = seq;
  }
  P2pMail* mine = peers.m[rank];
  if (lane < nranks) {
    volatile unsigned int* f = &mine->flag[slot][lane];
    const long long t0 = clock64();
    while (*f != seq) {
      if (clock64() - t0 > 8000000000LL) break;     // ~4 s: a peer never arrived (it failed); do not hang the GPU, the caller's checks report it
    }
  }
  __syncwarp();
  __threadfence_system();
  if (lane < 16) {
    double acc = 0.0;
    for (int r = 0; r < nranks; ++r) acc += *(volatile double*)&mine->val[slot][r][lane];
    stats[lane] = acc;
  }
}

struct dawn_unet {
  dawn_unet_cfg cfg{};
  int nlev = 0;
  std::vector<int> dims;                       // [dim, dim*m0, ...]
  std::vector<std::pair<int, int>> in_out;
  int cond_dim = 0, tdim = 0;
  std::unordered_map<std::string, HostParam> raw;
  bool committed = false;
  bool use_tc = true;                          // tcgen05 contraction path (DAWN_TC=0 falls back to mma.sync)
  bool use_conv3 = true;                       // halo-tile tcgen05 3x3 conv (DAWN_TC_CONV3=0 falls back to the per-tap GEMM)
  bool use_presplit = true;                    // fp16 hi|lo pre-split of A for multi-n-tile 3x3 convs (DAWN_PRESPLIT=0: off)
  bool use_fused_ca = true;                    // fused cross-attention gate kernel for ci <= 128 (DAWN_FUSED_CA=0: unfused)
  bool use_fused_sla = true;                   // fused SLA context on 64-channel levels (DAWN_FUSED_SLA=0: unfused)
  int conv3_tma = 1;                           // halo conv fed by TMA from fp16 hi|lo planes: 1 (default) = second conv of a ResBlock, whose input the
                                               // GroupNorm/cross-attention kernel writes pre-split; 2 = every halo conv through a split pass
                                               // (measurement only); 0 = off (DAWN_CONV3_TMA)
  bool use_ta_tc = true;                       // tcgen05 temporal attention on 64-channel levels (DAWN_TA_TC=0: mma.sync kernel)
  bool use_fused_ta = true;                    // fused per-pixel temporal attention on 64-channel levels (DAWN_FUSED_TA=0: unfused)
  bool use_attn_tc = true;                     // tensor-core attention core (DAWN_ATTN_TC=0 falls back to SIMT)

  // packed weights
  std::vector<void*> owned;                    // weight allocations
  std::vector<void*> ws_owned;                 // workspace allocations
  int64_t ws_bytes = 0;
  ConvW init_full;                             // 7x7 over channels padded to cin_pad
  float* init_w3 = nullptr;                    // [k*k*3][dim] for the 3 noisy channels
  int cin_pad = 0;
  float *time_freqs = nullptr, *tW1 = nullptr, *tb1 = nullptr, *tW2 = nullptr, *tb2 = nullptr;
  float *rel_bias = nullptr, *rot_freqs = nullptr;
  float* ttc_table = nullptr;                  // [8][kTtcTable] bias * log2(e) inside the band, -1e30 outside (temporal_tc.cu)
  std::vector<ResBlockW> rb;                   // all resnet blocks
  std::map<std::string, int> rb_index;
  AttnW init_ta, mid_sa, mid_ta;
  std::vector<AttnW> down_ta, up_ta;
  std::vector<SlaW> down_sla, up_sla;
  std::vector<ConvW> down_conv;
  std::vector<UpW> up_conv;
  float *headW[2] = {nullptr, nullptr}, *headB[2] = {nullptr, nullptr};
  FilmDesc* film_descs = nullptr; int n_film = 0;
  CondDesc* cond_descs = nullptr; int n_cond = 0, cond_max_n1 = 0, cond_max_k = 0, cond_max_co = 0;   // batched per-clip prep

  // workspace (per set_num_frames)
  int F = 0, H = 0, W = 0;
  std::vector<int> lH, lW;
  float* MAPPART = nullptr;                    // k partial maps of the per-clip init conv (one per kernel row)
  int* VARY = nullptr;                         // device flag of the general entry: 1 = feature channels differ between frames
  bool prep_v1 = false;                        // DAWN_PREP_V1=1: the original per-clip table kernels
  float *X288 = nullptr, *FEA288 = nullptr, *MAP = nullptr, *XR = nullptr, *S0 = nullptr;
  std::vector<float*> bufA, bufB, CAT, DS;
  float *Y = nullptr, *A1 = nullptr, *QKV = nullptr, *O = nullptr, *ROWSTATS = nullptr, *GATES = nullptr, *WT = nullptr;
  float *BF = nullptr, *HF = nullptr, *HO = nullptr, *ROT = nullptr, *TSILU = nullptr, *CTX = nullptr, *KV = nullptr;
  double* STATS = nullptr; int n_stats = 0;
  int64_t* T_HOSTSIDE = nullptr;               // device int64 for forward_host
  float *H_XT = nullptr, *H_FEA = nullptr, *H_COND = nullptr, *H_OUT = nullptr;   // device staging for forward_host
  bool have_invariants = false;

  // frame sharding of one clip across ranks (exact: per-layer halo exchange + GroupNorm all-reduce)
  int sh_nranks = 1, sh_rank = 0, sh_Fglobal = 0, sh_halo_l = 0, sh_halo_r = 0;
  ncclComm_t sh_comm = nullptr;
  float* XE = nullptr;                         // (halo_l + F + halo_r) frames of a temporal layer's input, dense
  // GroupNorm all-reduce over NVLink peer memory (one kernel: every rank stores its 16 partial sums into every peer's mailbox, then
  // sums the mailboxes in rank order); set up by dawn_unet_shard_ipc_export / _import, otherwise ncclAllReduce is used
  P2pMail* p2p_own = nullptr;                  // this rank's mailbox (cudaMalloc, exported through cudaIpc)
  P2pMail* p2p_peer[kP2pMaxRanks] = {nullptr}; // every rank's mailbox as mapped into this process ([rank] == own)
  unsigned int* p2p_ctr = nullptr;             // device-side sequence number (graph replays keep counting)
  bool p2p_ready = false;

  std::map<std::string, float*> taps;
  int64_t launches = 0;

  // whole-clip sampling loop captured as one CUDA graph (dawn_unet_sampler_capture); invalidated by any geometry change
  cudaGraphExec_t samp_exec = nullptr;
  cudaStream_t samp_stream = nullptr;          // capture origin (the legacy default stream cannot be captured)
  int64_t samp_launches = 0;

  // per-category kernel timing (CUDA events on the launching stream), see dawn_unet_profile_*
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_ev;
  size_t prof_used = 0;
  struct ProfRec { int cat; double flops; double bytes; };
  std::vector<ProfRec> prof_recs;
  double prof_ms[DAWN_PROF_NCAT] = {0};
  double prof_flops[DAWN_PROF_NCAT] = {0};
  double prof_bytes[DAWN_PROF_NCAT] = {0};
  int64_t prof_cnt[DAWN_PROF_NCAT] = {0};
};

namespace {

// ------------------------------------------------------------------------------------------ allocation helpers
int dev_alloc(std::vector<void*>& owner, size_t nfloats, float** out, int64_t* counter = nullptr) {
  void* p = nullptr;
  size_t bytes = std::max<size_t>(nfloats, 4) * sizeof(float);
  DAWN_CUDA_OK(cudaMalloc(&p, bytes));
  owner.push_back(p);
  if (counter) *counter += (int64_t)bytes;
  *out = (float*)p;
  return 0;
}
int dev_upload(dawn_unet* h, const std::vector<float>& v, float** out) {
  DAWN_TRY(dev_alloc(h->owned, v.size(), out));
  DAWN_CUDA_OK(cudaMemcpy(*out, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}
void free_all(std::vector<void*>& v) {
  for (void* p : v) cudaFree(p);
  v.clear();
}
inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// tcgen05 image of a [K][ldb] weight matrix (only for shapes the tcgen05 kernel accepts)
int upload_tc_image(dawn_unet* h, const std::vector<float>& m, int K, int N, int ldb, float** img, float* scale) {
  *img = nullptr; *scale = 1.f;
  if (!h->use_tc || N % 64 != 0 || K % 64 != 0) return 0;
  std::vector<float> im;
  tc_pack_weights(m.data(), K, N, ldb, im, scale);
  return dev_upload(h, im, img);
}

const HostParam* find(dawn_unet* h, const std::string& name) {
  auto it = h->raw.find(name);
  return it == h->raw.end() ? nullptr : &it->second;
}
int need(dawn_unet* h, const std::string& name, std::vector<int64_t> shape, const HostParam** out) {
  const HostParam* p = find(h, name);
  if (!p) { set_last_error("missing parameter: " + name); return -1; }
  if (p->shape != shape) {
    std::string s = "parameter " + name + " has shape (";
    for (auto d : p->shape) s += std::to_string(d) + ",";
    s += ") expected (";
    for (auto d : shape) s += std::to_string(d) + ",";
    set_last_error(s + ")");
    return -1;
  }
  *out = p;
  return 0;
}

// conv weight (co, ci, 1, kh, kw) -> [ (ky*kw+kx)*ci_pad + c ][ldb]
int pack_conv(dawn_unet* h, const std::string& prefix, int co, int ci, int kh, int kw, int ci_pad, bool bias, ConvW* out) {
  const HostParam* w; const HostParam* b = nullptr;
  DAWN_TRY(need(h, prefix + ".weight", {co, ci, 1, kh, kw}, &w));
  if (bias) DAWN_TRY(need(h, prefix + ".bias", {co}, &b));
  const int ldb = round_up(co, 64);
  const int K = kh * kw * ci_pad;
  std::vector<float> m((size_t)K * ldb, 0.f);
  for (int n = 0; n < co; ++n)
    for (int c = 0; c < ci; ++c)
      for (int t = 0; t < kh * kw; ++t)
        m[((size_t)t * ci_pad + c) * ldb + n] = w->data[((size_t)n * ci + c) * kh * kw + t];
  DAWN_TRY(dev_upload(h, m, &out->w));
  DAWN_TRY(upload_tc_image(h, m, K, co, ldb, &out->img, &out->img_scale));
  out->b = nullptr;
  if (bias) {
    std::vector<float> bb(ldb, 0.f);
    std::copy(b->data.begin(), b->data.end(), bb.begin());
    DAWN_TRY(dev_upload(h, bb, &out->b));
  }
  out->K = K; out->N = co; out->ldb = ldb;
  return 0;
}

// Linear weight (N, K) [+ optional per-input gain, + per-output-row scale for the first `nscale` rows]
// -> [K][ldb], plus column sums for the LayerNorm fold
int pack_linear(dawn_unet* h, const HostParam* w, int N, int K, const float* gain, float qscale, int nscale,
                float** Wout, float** wsum, int* ldb_out, float** img = nullptr, float* img_scale = nullptr) {
  const int ldb = round_up(N, 64);
  std::vector<float> m((size_t)K * ldb, 0.f), s(ldb, 0.f);
  for (int n = 0; n < N; ++n) {
    double acc = 0.0;
    const float sc = (n < nscale) ? qscale : 1.0f;
    for (int k = 0; k < K; ++k) {
      float v = w->data[(size_t)n * K + k];
      if (gain) v *= gain[k];
      v *= sc;
      m[(size_t)k * ldb + n] = v;
      acc += v;
    }
    s[n] = (float)acc;
  }
  DAWN_TRY(dev_upload(h, m, Wout));
  if (img) DAWN_TRY(upload_tc_image(h, m, K, N, ldb, img, img_scale));
  if (wsum) DAWN_TRY(dev_upload(h, s, wsum));
  if (ldb_out) *ldb_out = ldb;
  return 0;
}

int upload_raw(dawn_unet* h, const std::string& name, std::vector<int64_t> shape, float** out) {
  const HostParam* p;
  DAWN_TRY(need(h, name, shape, &p));
  return dev_upload(h, p->data, out);
}

int pack_resblock(dawn_unet* h, const std::string& name, int ci, int co, bool cond, int* stat_counter) {
  ResBlockW r;
  r.name = name; r.ci = ci; r.co = co; r.cond = cond; r.res = (ci != co);
  DAWN_CHECK(ci % 32 == 0 && co % 64 == 0, "channel counts must be multiples of 64 (dim=64 family)");
  DAWN_TRY(pack_conv(h, name + ".block1.proj", co, ci, 3, 3, ci, true, &r.c1));
  DAWN_TRY(pack_conv(h, name + ".block2.proj", co, co, 3, 3, co, true, &r.c2));
  DAWN_TRY(upload_raw(h, name + ".block1.norm.weight", {co}, &r.gn1w));
  DAWN_TRY(upload_raw(h, name + ".block1.norm.bias", {co}, &r.gn1b));
  DAWN_TRY(upload_raw(h, name + ".block2.norm.weight", {co}, &r.gn2w));
  DAWN_TRY(upload_raw(h, name + ".block2.norm.bias", {co}, &r.gn2b));
  if (r.res) DAWN_TRY(pack_conv(h, name + ".res_conv", co, ci, 1, 1, ci, true, &r.cres));
  r.st1 = (*stat_counter)++;
  r.st2 = (*stat_counter)++;
  if (cond) {
    const int tdim = h->tdim;
    DAWN_TRY(upload_raw(h, name + ".time_mlp.1.weight", {2 * co, tdim}, &r.tW));
    DAWN_TRY(upload_raw(h, name + ".time_mlp.1.bias", {2 * co}, &r.tB));
    const char* mlp[3] = {"pose_mlp", "audio_mlp", "eye_mlp"};
    const int kdim[3] = {h->cfg.cond_pose, h->cfg.cond_aud, h->cfg.cond_eye};
    const char* can[3] = {"cross_attn_pose", "cross_attn_aud", "cross_attn_eye"};
    std::vector<float> wq((size_t)ci * 192, 0.f), wsum(192, 0.f);
    for (int a = 0; a < 3; ++a) {
      DAWN_TRY(upload_raw(h, name + "." + mlp[a] + ".1.weight", {2 * co, kdim[a]}, &r.mW[a]));
      DAWN_TRY(upload_raw(h, name + "." + mlp[a] + ".1.bias", {2 * co}, &r.mB[a]));
      const std::string p = name + "." + can[a];
      const HostParam *g, *q;
      DAWN_TRY(need(h, p + ".norm.g", {ci}, &g));
      DAWN_TRY(need(h, p + ".to_q.weight", {64, ci}, &q));
      for (int j = 0; j < 64; ++j) {
        double acc = 0.0;
        for (int k = 0; k < ci; ++k) {
          const float v = q->data[(size_t)j * ci + k] * g->data[k];     // LayerNorm_img gain folded (U:203, 519)
          wq[(size_t)k * 192 + a * 64 + j] = v;
          acc += v;
        }
        wsum[a * 64 + j] = (float)acc;
      }
      DAWN_TRY(upload_raw(h, p + ".to_kv.weight", {128, 2 * co}, &r.ca[a].Wkv));
      DAWN_TRY(upload_raw(h, p + ".null_kv", {2, 8}, &r.ca[a].nkv));
      DAWN_TRY(upload_raw(h, p + ".q_scale", {8}, &r.ca[a].qs));
      DAWN_TRY(upload_raw(h, p + ".k_scale", {8}, &r.ca[a].ks));
      DAWN_TRY(upload_raw(h, p + ".to_out.0.weight", {co, 64}, &r.ca[a].Wout));
      DAWN_TRY(upload_raw(h, p + ".to_out.1.g", {co}, &r.ca[a].gout));
    }
    DAWN_TRY(dev_upload(h, wq, &r.Wq));
    DAWN_TRY(upload_tc_image(h, wq, ci, 192, 192, &r.Wq_img, &r.Wq_scale));
    DAWN_TRY(dev_upload(h, wsum, &r.wsumq));
    if (ci == 64 || ci == 128) {
      std::vector<uint16_t> W;
      ca_fused_pack(wq.data(), ci, W, &r.f_inv_wscale);
      std::vector<float> tmp(W.size() / 2);
      memcpy(tmp.data(), W.data(), W.size() * 2);
      float* d = nullptr;
      DAWN_TRY(dev_upload(h, tmp, &d));
      r.fWq = reinterpret_cast<uint16_t*>(d);
    }
  }
  h->rb_index[name] = (int)h->rb.size();
  h->rb.push_back(r);
  return 0;
}

int pack_attn(dawn_unet* h, const std::string& norm_name, const std::string& fn, int C, AttnW* a) {
  const HostParam *g, *qkv, *o;
  DAWN_TRY(need(h, norm_name + ".gamma", {1, C, 1, 1, 1}, &g));
  DAWN_TRY(need(h, fn + ".to_qkv.weight", {768, C}, &qkv));
  DAWN_TRY(need(h, fn + ".to_out.weight", {C, 256}, &o));
  a->C = C;
  const float scale = 1.0f / sqrtf(32.0f);                                   // q * dim_head^-0.5 (U:657, 687)
  DAWN_TRY(pack_linear(h, qkv, 768, C, g->data.data(), scale, 256, &a->Wqkv, &a->wsum, nullptr, &a->Wqkv_img, &a->Wqkv_scale));
  int ldb = 0;
  DAWN_TRY(pack_linear(h, o, C, 256, nullptr, 1.f, 0, &a->out.w, nullptr, &ldb, &a->out.img, &a->out.img_scale));
  a->out.b = nullptr; a->out.K = 256; a->out.N = C; a->out.ldb = ldb;
  if (C == 64) {
    std::vector<float> wq((size_t)768 * C);
    for (int n = 0; n < 768; ++n)
      for (int k = 0; k < C; ++k) wq[(size_t)n * C + k] = qkv->data[(size_t)n * C + k] * g->data[k] * (n < 256 ? scale : 1.0f);
    std::vector<uint16_t> Wq, Wo;
    temporal_fused_pack(wq.data(), o->data.data(), Wq, Wo, &a->f_inv_wscale, &a->f_inv_oscale);
    float *dq = nullptr, *dout = nullptr;
    std::vector<float> tq(Wq.size() / 2), to(Wo.size() / 2);
    memcpy(tq.data(), Wq.data(), Wq.size() * 2); memcpy(to.data(), Wo.data(), Wo.size() * 2);
    DAWN_TRY(dev_upload(h, tq, &dq)); DAWN_TRY(dev_upload(h, to, &dout));
    a->fq = reinterpret_cast<uint16_t*>(dq); a->fo = reinterpret_cast<uint16_t*>(dout);
    std::vector<uint8_t> Tq, To;
    temporal_tc_pack(wq.data(), o->data.data(), Tq, To, &a->t_inv_wscale, &a->t_inv_oscale);
    std::vector<float> uq(Tq.size() / 4), uo(To.size() / 4);
    memcpy(uq.data(), Tq.data(), Tq.size()); memcpy(uo.data(), To.data(), To.size());
    float *dtq = nullptr, *dto = nullptr;
    DAWN_TRY(dev_upload(h, uq, &dtq)); DAWN_TRY(dev_upload(h, uo, &dto));
    a->tq = reinterpret_cast<uint8_t*>(dtq); a->to = reinterpret_cast<uint8_t*>(dto);
  }
  return 0;
}

int pack_sla(dawn_unet* h, const std::string& p, int C, SlaW* s) {        // p = "downs.L.2.fn"
  const HostParam *g, *qkv, *o, *b;
  DAWN_TRY(need(h, p + ".norm.gamma", {1, C, 1, 1, 1}, &g));
  DAWN_TRY(need(h, p + ".fn.to_qkv.weight", {768, C, 1, 1}, &qkv));
  DAWN_TRY(need(h, p + ".fn.to_out.weight", {C, 256, 1, 1}, &o));
  DAWN_TRY(need(h, p + ".fn.to_out.bias", {C}, &b));
  s->C = C;
  DAWN_TRY(pack_linear(h, qkv, 768, C, g->data.data(), 1.f, 0, &s->Wqkv, &s->wsum, nullptr, &s->Wqkv_img, &s->Wqkv_scale));
  if (C == 64) {
    DAWN_TRY(pack_linear(h, qkv, 256, C, g->data.data(), 1.f, 0, &s->Wq, &s->wsum_q, nullptr, &s->Wq_img, &s->Wq_scale));
    std::vector<float> wf((size_t)768 * C);
    for (int n = 0; n < 768; ++n)
      for (int k = 0; k < C; ++k) wf[(size_t)n * C + k] = qkv->data[(size_t)n * C + k] * g->data[k];
    std::vector<uint16_t> W;
    sla_fused_pack(wf.data(), W, &s->f_inv_wscale);
    std::vector<float> tmp(W.size() / 2);
    memcpy(tmp.data(), W.data(), W.size() * 2);
    float* d = nullptr;
    DAWN_TRY(dev_upload(h, tmp, &d));
    s->fkv = reinterpret_cast<uint16_t*>(d);
    sla_out_pack(wf.data(), W, &s->fq_inv_wscale);
    tmp.assign(W.size() / 2, 0.f);
    memcpy(tmp.data(), W.data(), W.size() * 2);
    DAWN_TRY(dev_upload(h, tmp, &d));
    s->fq = reinterpret_cast<uint16_t*>(d);
  }
  std::vector<float> wt((size_t)256 * C);
  for (int c = 0; c < C; ++c)
    for (int k = 0; k < 256; ++k) wt[(size_t)k * C + c] = o->data[(size_t)c * 256 + k];
  DAWN_TRY(dev_upload(h, wt, &s->WoutT));
  std::vector<float> bb(round_up(C, 64), 0.f);
  std::copy(b->data.begin(), b->data.end(), bb.begin());
  DAWN_TRY(dev_upload(h, bb, &s->bout));
  return 0;
}

// ConvTranspose3d (1,4,4)/(1,2,2)/(0,1,1) weight (ci, co, 1, 4, 4): four output-parity classes, each a 2x2 conv.
// out[y] gets in[(y+1-ky)/2]: y even -> ky in {1 (dy 0), 3 (dy -1)}; y odd -> ky in {0 (dy +1), 2 (dy 0)}.   (U:165-167)
static const int kUpK[2][2] = {{1, 3}, {0, 2}};
static const int kUpD[2][2] = {{0, -1}, {1, 0}};
int pack_up(dawn_unet* h, const std::string& name, int C, UpW* u) {
  const HostParam *w, *b;
  DAWN_TRY(need(h, name + ".weight", {C, C, 1, 4, 4}, &w));
  DAWN_TRY(need(h, name + ".bias", {C}, &b));
  const int ldb = round_up(C, 64);
  std::vector<float> bb(ldb, 0.f);
  std::copy(b->data.begin(), b->data.end(), bb.begin());
  float* bdev;
  DAWN_TRY(dev_upload(h, bb, &bdev));
  for (int py = 0; py < 2; ++py)
    for (int px = 0; px < 2; ++px) {
      std::vector<float> m((size_t)4 * C * ldb, 0.f);
      for (int ty = 0; ty < 2; ++ty)
        for (int tx = 0; tx < 2; ++tx) {
          const int ky = kUpK[py][ty], kx = kUpK[px][tx];
          for (int c = 0; c < C; ++c)
            for (int n = 0; n < C; ++n)
              m[((size_t)(ty * 2 + tx) * C + c) * ldb + n] = w->data[(((size_t)c * C + n) * 4 + ky) * 4 + kx];
        }
      ConvW& cw = u->cls[py * 2 + px];
      DAWN_TRY(dev_upload(h, m, &cw.w));
      DAWN_TRY(upload_tc_image(h, m, 4 * C, C, ldb, &cw.img, &cw.img_scale));
      cw.b = bdev; cw.K = 4 * C; cw.N = C; cw.ldb = ldb;
    }
  if (C == 64) {
    // one 3x3 conv over the input grid producing all four output parities: weight rows (tap, cin), columns (class, cout);
    // taps a class does not touch stay zero (2.25x the MACs, one launch of the halo-tile kernel instead of four gather GEMMs)
    const int N4 = 4 * C;
    std::vector<float> m((size_t)9 * C * N4, 0.f), b4(N4, 0.f);
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px) {
        const int cls = py * 2 + px;
        for (int n = 0; n < C; ++n) b4[cls * C + n] = b->data[n];
        for (int ty = 0; ty < 2; ++ty)
          for (int tx = 0; tx < 2; ++tx) {
            const int ky = kUpK[py][ty], kx = kUpK[px][tx];
            const int tap = (kUpD[py][ty] + 1) * 3 + (kUpD[px][tx] + 1);
            for (int c = 0; c < C; ++c)
              for (int n = 0; n < C; ++n)
                m[((size_t)tap * C + c) * N4 + cls * C + n] = w->data[(((size_t)c * C + n) * 4 + ky) * 4 + kx];
          }
      }
    DAWN_TRY(dev_upload(h, m, &u->all.w));
    DAWN_TRY(upload_tc_image(h, m, 9 * C, N4, N4, &u->all.img, &u->all.img_scale));
    DAWN_TRY(dev_upload(h, b4, &u->all.b));
    u->all.K = 9 * C; u->all.N = N4; u->all.ldb = N4;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------ GEMM wrappers
void base_params(GemmParams& p, const Act& in, int F) {
  memset(&p, 0, sizeof(p));
  p.A = in.p; p.lda = in.ld; p.Cin = in.C;
  p.IH = in.H; p.IW = in.W; p.OHs = in.H; p.OWs = in.W; p.in_stride = 1;
  p.ntaps = 1; p.dy[0] = 0; p.dx[0] = 0;
  p.M = F * in.H * in.W; p.rows_per_batch = p.M;
  p.OH = in.H; p.OW = in.W; p.out_stride = 1; p.oy0 = 0; p.ox0 = 0;
  p.P = in.H * in.W;
  p.q_post_scale = 1.f;
}
void set_weights(GemmParams& p, const ConvW& w) {
  p.B = w.w; p.Bimg = w.img; p.tc_scale = 1.0f / (kTcActScale * w.img_scale); p.ldb = w.ldb; p.b_batch_stride = 0; p.N = w.N; p.K = w.K; p.bias = w.b;
}
void set_square_taps(GemmParams& p, int k, int pad) {
  p.ntaps = k * k;
  for (int ky = 0; ky < k; ++ky)
    for (int kx = 0; kx < k; ++kx) { p.dy[ky * k + kx] = (signed char)(ky - pad); p.dx[ky * k + kx] = (signed char)(kx - pad); }
}


// profile categories (dawn_unet_profile_read)
enum ProfCat : int {
  PC_CONV3 = 0,      // 3x3 conv implicit GEMM (+GroupNorm statistics)
  PC_CONV_OTHER,     // init 7x7, 4x4 down / transposed up, 1x1 residual convs
  PC_QKV,            // LayerNorm-folded qkv projections (temporal / spatial-linear / mid attention)
  PC_OUTPROJ,        // attention output projections (+ residual)
  PC_CA_GATE,        // cross-attention q projection + 2-key softmax gate
  PC_GN_HCOND,       // SiLU(FiLM(GN)) + per-frame cross-attention table GEMM (K=32)
  PC_ATTN_CORE,      // banded temporal / full spatial softmax attention
  PC_SLA_CTX,        // spatial linear attention context + composed projection
  PC_GN_APPLY,       // elementwise SiLU(GN) (+ residual)
  PC_ROWSTATS,       // LayerNorm row statistics
  PC_CA_RSTD,        // cross-attention output LayerNorm via Gram form
  PC_MISC,           // time MLP, FiLM, init conv (3 ch), heads, layout
  PC_PREP,           // per-clip tables
  PC_TEMPORAL_L0,    // fused per-pixel temporal attention at level 0 (the dominant kernel: bench.py's roofline object)
  PC_CONV3_L0,       // halo-tile 3x3 conv, dim -> dim channels at level 0
  PC_COMM_AR,        // frame sharding: GroupNorm statistic all-reduces (stream time, includes waiting for the slowest rank)
  PC_COMM_HALO,      // frame sharding: temporal halo exchange (pack copy + neighbour send/recv)
  PC_COUNT
};
static_assert(PC_COUNT <= DAWN_PROF_NCAT, "increase DAWN_PROF_NCAT");

struct Ctx {
  dawn_unet* h; cudaStream_t st;
  int gemm(const GemmParams& p, int epi, int cat);
};

// one kernel launch: counted, and bracketed by CUDA events when profiling is on
struct ProfScope {
  dawn_unet* h; cudaStream_t st; bool on;
  ProfScope(Ctx& c, int cat, double flops, double bytes) : h(c.h), st(c.st), on(c.h->prof_on) {
    h->launches++;
    if (!on) return;
    while (h->prof_ev.size() < h->prof_used + 2) {
      cudaEvent_t e; cudaEventCreate(&e); h->prof_ev.push_back(e);
    }
    h->prof_recs.push_back({cat, flops, bytes});
    cudaEventRecord(h->prof_ev[h->prof_used], st);
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(h->prof_ev[h->prof_used + 1], st);
    h->prof_used += 2;
  }
};

int Ctx::gemm(const GemmParams& p, int epi, int cat) {
  // algorithmic work: 2*M*N*K flops (1x, not the 3 split passes); bytes: A once + output write (+ residual/Y read)
  const double flops = 2.0 * p.M * (double)p.N * p.K;
  double bytes = 4.0 * p.M * ((double)p.Cin * (p.in_stride == 1 ? 1 : 4) + p.N);
  if (p.Res) bytes += 4.0 * p.M * p.N;
  if (p.Y) bytes += 4.0 * p.M * p.N;
  if (epi == EPI_CA_GATE) bytes = 4.0 * p.M * (p.Cin + 24.0);
  if (h->use_tc && h->use_conv3 && h->conv3_tma == 2 && p.Bimg != nullptr && tc_conv3_supported(p, epi) && p.A16h == nullptr && p.lda == p.Cin) {
    // measurement mode (DAWN_CONV3_TMA=2): every halo conv fed by TMA; the planes come from a stand-alone split pass (timed under "misc")
    GemmParams q = p;
    unsigned short* hi = reinterpret_cast<unsigned short*>(h->O);
    q.A16h = hi; q.A16l = hi + (size_t)p.M * p.Cin;
    {
      ProfScope ps0(*this, PC_MISC, 0, 8.0 * p.M * p.Cin);
      DAWN_TRY(launch_split_rows(p.A, p.lda, p.Cin, p.M, (void*)q.A16h, (void*)q.A16l, st));
    }
    ProfScope ps(*this, cat, flops, bytes);
    return launch_tc_conv3(q, q.Bimg, st);
  }
  ProfScope ps(*this, cat, flops, bytes);
  if (h->use_tc && h->use_conv3 && p.Bimg != nullptr && tc_conv3_supported(p, epi)) return launch_tc_conv3(p, p.Bimg, st);
  if (h->use_tc && p.Bimg != nullptr && tc_gemm_supported(p, epi)) {
    // several n-tiles re-convert the same A panels (per-tap gather of the small levels' 3x3 convolutions): split once instead
    const long long in_rows = (long long)(p.M / (p.OHs * p.OWs)) * p.IH * p.IW;
    const size_t need = (size_t)in_rows * p.Cin * 4;                                   // two fp16 planes
    const size_t have = (size_t)(h->F + 2 * h->cfg.win_width) * h->lH[0] * h->lW[0] * 256 * sizeof(float);
    if (h->use_presplit && ((p.ntaps == 9 && p.N >= 256 && !p.perm_in) || p.want_split) && p.Cin % 64 == 0 && need <= have) {
      GemmParams q = p;
      unsigned short* hi = reinterpret_cast<unsigned short*>(h->O);
      q.A16h = hi; q.A16l = hi + (size_t)in_rows * p.Cin;
      h->launches++;
      DAWN_TRY(launch_split_rows(p.A, p.lda, p.Cin, in_rows, (void*)q.A16h, (void*)q.A16l, st));
      return launch_tc_gemm(q, q.Bimg, epi, st);
    }
    return launch_tc_gemm(p, p.Bimg, epi, st);
  }
  return launch_gemm(p, epi, st);
}

int tap(Ctx& c, const std::string& name, const Act& a);

// LayerNorm-folded 1x1 GEMM: on the tcgen05 path the producers compute the row statistics themselves (no separate
// rowstats launch, no second read of the input); otherwise run rowstats_kernel into the global buffer.
int ln_gemm(Ctx& c, GemmParams& p, int epi, int cat, const float* x, int ldx, int C, int rows) {
  dawn_unet* h = c.h;
  p.ln_inline = 0; p.rowstats = h->ROWSTATS;
  const bool tc_ok = h->use_tc && p.Bimg != nullptr && tc_gemm_supported(p, epi) && p.ntaps == 1;
  if (tc_ok && h->use_presplit && (p.N >= 384 || (p.N == 192 && p.Cin >= 256)) && p.Cin % 64 == 0) {
    // N = 768 is six 128-column tiles, each re-gathering and re-splitting the same A panels: split once (cp.async producers),
    // row statistics from the stand-alone kernel
    p.want_split = 1;
    ProfScope ps(c, PC_ROWSTATS, 0, 4.0 * rows * C);
    DAWN_TRY(launch_rowstats(x, ldx, C, rows, 1e-5f, h->ROWSTATS, c.st));
  } else if (tc_ok) {
    p.ln_inline = 1; p.rowstats = nullptr;
  } else {
    ProfScope ps(c, PC_ROWSTATS, 0, 4.0 * rows * C);
    DAWN_TRY(launch_rowstats(x, ldx, C, rows, 1e-5f, h->ROWSTATS, c.st));
  }
  return c.gemm(p, epi, cat);
}

// conv k x k, stride 1, same padding, + bias, optional GroupNorm statistics slot
int conv_same(Ctx& c, const Act& in, const ConvW& w, int k, const Act& out, int stat_slot, const unsigned short* in16h = nullptr,
              const unsigned short* in16l = nullptr) {
  GemmParams p; base_params(p, in, c.h->F);
  set_weights(p, w); set_square_taps(p, k, k / 2);
  p.Out = out.p; p.ldo = out.ld;
  p.A16h = in16h; p.A16l = in16l;               // the input exists as fp16 hi | lo planes (and NOT as fp32): halo conv by TMA
  if (stat_slot >= 0) { p.stats = c.h->STATS + 16 * stat_slot; p.cpg = w.N / 8; }
  const bool l0 = in.H == c.h->lH[0] && in.C == c.h->cfg.dim && w.N == c.h->cfg.dim;
  return c.gemm(p, EPI_PLAIN, k == 3 ? (l0 ? PC_CONV3_L0 : PC_CONV3) : PC_CONV_OTHER);
}

// GroupNorm statistics span all frames of the clip: with frame sharding the 16 partial sums are all-reduced (fp64)
int gn_allreduce(Ctx& c, int slot) {
  dawn_unet* h = c.h;
  if (h->sh_nranks <= 1) return 0;
  double* st = h->STATS + 16 * slot;
  ProfScope ps(c, PC_COMM_AR, 0, 128.0 * h->sh_nranks);
  if (h->p2p_ready) {
    P2pPeers pp;
    for (int r = 0; r < kP2pMaxRanks; ++r) pp.m[r] = h->p2p_peer[r];
    gn_p2p_allreduce_kernel<<<1, 32, 0, c.st>>>(st, pp, h->sh_rank, h->sh_nranks, h->p2p_ctr);
    DAWN_LAUNCH_OK();
    return 0;
  }
  DAWN_NCCL_OK(g_nccl.AllReduce(st, st, 16, kNcclFloat64, kNcclSum, h->sh_comm, c.st));
  return 0;
}

// ResnetBlock_ca_mul (U:363-479)
int resblock(Ctx& c, const ResBlockW& r, const Act& x, const Act& out) {
  dawn_unet* h = c.h;
  const int F = h->F, M = F * x.H * x.W, P = x.H * x.W;
  DAWN_CHECK(x.C == r.ci && out.C == r.co, "resblock channel mismatch: " + r.name);
  Act y{h->Y, r.co, r.co, x.H, x.W}, a1{h->A1, r.co, r.co, x.H, x.W};
  const double count = (double)h->sh_Fglobal * P * (r.co / 8);     // GroupNorm statistics span the WHOLE clip (U:230)
  if (r.cond && h->use_fused_ca && r.fWq && ca_fused_supported(r.ci, P)) {
    CaFusedArgs a{};
    a.x = x.p; a.ldx = x.ld; a.F = F; a.P = P; a.Wq = r.fWq; a.inv_wscale = r.f_inv_wscale;
    a.kq = r.kq; a.nkq = r.nkq; a.G = r.G; a.Wt = h->WT;
    ProfScope ps(c, PC_CA_GATE, 2.0 * M * r.ci * 192, 4.0 * M * (r.ci + 32));
    DAWN_TRY(launch_ca_fused(a, r.ci, c.st));
  } else if (r.cond) {
    // cross-attention gates from the raw block input (U:454-463): LayerNorm_img folded into the q projection
    GemmParams p; base_params(p, x, F);
    p.B = r.Wq; p.Bimg = r.Wq_img; p.tc_scale = 1.0f / (kTcActScale * r.Wq_scale); p.ldb = 192; p.N = 192; p.K = r.ci;
    p.wsum = r.wsumq; p.kq = r.kq; p.nkq = r.nkq; p.gates = h->GATES;
    DAWN_TRY(ln_gemm(c, p, EPI_CA_GATE, PC_CA_GATE, x.p, x.ld, x.C, M));
    ProfScope ps(c, PC_CA_RSTD, 0, 4.0 * M * 56);
    DAWN_TRY(launch_ca_rstd(h->GATES, r.G, M, P, h->WT, c.st));
  }
  DAWN_TRY(conv_same(c, x, r.c1, 3, y, r.st1));
  DAWN_TRY(gn_allreduce(c, r.st1));
  // a1 is consumed by the second conv only: when that conv runs on the halo-tile tcgen05 kernel, a1 is written as two fp16 planes
  // (hi | lo, the same bytes as the fp32 row) and the conv fetches its tiles by TMA
  const unsigned short *a1h = nullptr, *a1l = nullptr;
  if (r.cond && h->use_fused_ca && gn_hcond_supported(r.co, P) && h->conv3_tma >= 1 && h->use_tc && h->use_conv3 && r.c2.img != nullptr) {
    GemmParams q; base_params(q, a1, F);
    set_weights(q, r.c2); set_square_taps(q, 3, 1);
    q.Out = y.p; q.ldo = y.ld; q.stats = h->STATS + 16 * r.st2; q.cpg = r.co / 8;
    if (tc_conv3_supported(q, EPI_PLAIN)) {
      a1h = reinterpret_cast<const unsigned short*>(h->A1);
      a1l = a1h + (size_t)M * r.co;
    }
  }
  if (r.cond && h->use_fused_ca && gn_hcond_supported(r.co, P)) {
    GnHcondArgs a{};
    a.Wt = h->WT; a.T = r.T; a.ldbT = r.ldbT; a.Y = y.p; a.ldy = y.ld; a.Out = a1.p; a.ldo = a1.ld;
    a.Out16h = const_cast<unsigned short*>(a1h); a.Out16l = const_cast<unsigned short*>(a1l);
    a.F = F; a.P = P; a.co = r.co;
    a.gn_stats = h->STATS + 16 * r.st1; a.gn_count = count; a.cpg = r.co / 8;
    a.gn_w = r.gn1w; a.gn_b = r.gn1b; a.film = r.film;
    ProfScope ps(c, PC_GN_HCOND, 2.0 * M * 32 * r.co, 4.0 * M * (2.0 * r.co + 32));
    DAWN_TRY(launch_gn_hcond(a, c.st));
  } else if (r.cond) {
    // a1 = SiLU(FiLM(GN(y))) + h_cond, h_cond = Wt (M x 32) @ T_f (32 x co) per frame
    Act wt{h->WT, 32, 32, x.H, x.W};
    GemmParams p; base_params(p, wt, F);
    p.B = r.T; p.ldb = r.ldbT; p.b_batch_stride = (long long)32 * r.ldbT; p.N = r.co; p.K = 32;
    p.rows_per_batch = P;
    p.Out = a1.p; p.ldo = a1.ld;
    p.Y = y.p; p.ldy = y.ld; p.gn_stats = h->STATS + 16 * r.st1; p.gn_w = r.gn1w; p.gn_b = r.gn1b;
    p.film = r.film; p.gn_count = count; p.cpg = r.co / 8;
    DAWN_TRY(c.gemm(p, EPI_GN_APPLY, PC_GN_HCOND));
  } else {
    ProfScope ps(c, PC_GN_APPLY, 0, 8.0 * M * r.co);
    DAWN_TRY(launch_gn_apply(y.p, y.ld, r.co, M, h->STATS + 16 * r.st1, count, r.co / 8, r.gn1w, r.gn1b, nullptr,
                             nullptr, 0, a1.p, a1.ld, c.st));
  }
  DAWN_TRY(conv_same(c, a1, r.c2, 3, y, r.st2, a1h, a1l));
  DAWN_TRY(gn_allreduce(c, r.st2));
  const float* res = x.p; int ldr = x.ld;
  if (r.res) {
    GemmParams p; base_params(p, x, F);
    set_weights(p, r.cres);
    p.Out = out.p; p.ldo = out.ld;
    DAWN_TRY(c.gemm(p, EPI_PLAIN, PC_CONV_OTHER));
    res = out.p; ldr = out.ld;
  }
  {
  ProfScope ps(c, PC_GN_APPLY, 0, 12.0 * M * r.co);
  DAWN_TRY(launch_gn_apply(y.p, y.ld, r.co, M, h->STATS + 16 * r.st2, count, r.co / 8, r.gn2w, r.gn2b, nullptr,
                           res, ldr, out.p, out.ld, c.st));
  }
  return tap(c, r.name, out);
}

// largest divisor of P that is <= 16: pixel-block size of the sequence-blocked row order
inline int seq_block(int P) { for (int b = 16; b > 1; --b) if (P % b == 0) return b; return 1; }

// Residual(PreNorm(temporal Attention)) (U:648-725 / LA:275-342): x -> dst = x + to_out(attn(...))
// q/k/v and the attention output live in SEQUENCE-BLOCKED row order (16 adjacent pixels x all frames contiguous):
// with frame-major rows every (pixel, head) sequence touched one 2 MB page per frame and the attention core was
// TLB/latency-bound; the QKV GEMM gathers its A rows through the permutation and the out-projection scatters back.
int temporal_attn(Ctx& c, const AttnW& w, const Act& x, const Act& dst, const std::string& name) {
  dawn_unet* h = c.h;
  const int F = h->F, P = x.H * x.W;
  const int pb = seq_block(P);
  const int hl = h->sh_halo_l, hr = h->sh_halo_r, Fe = hl + F + hr;       // frames incl. neighbours' halos
  const int Me = Fe * P;
  Act xe = x;                                                             // the layer input over Fe frames
  if (h->sh_nranks > 1) {
    // exact frame sharding (SURVEY 8e): the +-win_width neighbour frames of the layer input come from the adjacent ranks;
    // K/V of those frames are re-projected locally.  Own frames are packed densely, boundaries go by NCCL send/recv.
    const size_t rowb = (size_t)x.C * sizeof(float);
    float* mid = h->XE + (size_t)hl * P * x.C;
    ProfScope ps(c, PC_COMM_HALO, 0, 4.0 * (2.0 * F + 2.0 * (hl + hr)) * P * x.C);
    DAWN_CUDA_OK(cudaMemcpy2DAsync(mid, rowb, x.p, (size_t)x.ld * sizeof(float), rowb, (size_t)F * P, cudaMemcpyDeviceToDevice, c.st));
    const size_t hcount = (size_t)h->cfg.win_width * P * x.C;
    DAWN_NCCL_OK(g_nccl.GroupStart());
    if (h->sh_rank > 0) {
      DAWN_NCCL_OK(g_nccl.Send(mid, hcount, kNcclFloat32, h->sh_rank - 1, h->sh_comm, c.st));
      DAWN_NCCL_OK(g_nccl.Recv(h->XE, hcount, kNcclFloat32, h->sh_rank - 1, h->sh_comm, c.st));
    }
    if (h->sh_rank < h->sh_nranks - 1) {
      DAWN_NCCL_OK(g_nccl.Send(mid + (size_t)(F - h->cfg.win_width) * P * x.C, hcount, kNcclFloat32, h->sh_rank + 1, h->sh_comm, c.st));
      DAWN_NCCL_OK(g_nccl.Recv(mid + (size_t)F * P * x.C, hcount, kNcclFloat32, h->sh_rank + 1, h->sh_comm, c.st));
    }
    DAWN_NCCL_OK(g_nccl.GroupEnd());
    xe = Act{h->XE, x.C, x.C, x.H, x.W};
  }
  // tcgen05 kernel: one work unit per pixel while the sequence fits one 240-frame window (a 200-frame shard plus one halo); longer sequences
  // are cut into segments that each pay the full two-tile cost.  Since the issuer warps run warp-uniformly (r2-h) two segments of a
  // 280-frame sequence (a 200-frame shard with both halos) take 3.5 ms at level 0, against ~4.3 ms for the mma.sync kernel that keeps the
  // whole sequence on chip: the tcgen05 kernel is used whenever it supports the shape (DAWN_TA_TC=0 selects the older kernels).
  const bool ttc_ok = h->use_ta_tc && w.tq && h->ttc_table && temporal_tc_supported(x.C, Fe, h->cfg.win_width, hl, hl + F);
  const bool fused_ok = h->use_fused_ta && w.fq && temporal_fused_supported(x.C, Fe, h->cfg.win_width, hl, hl + F);
  if (ttc_ok) {
    // long sequences are cut into segments whose windows overlap: an in-place layer would let one segment read rows another already
    // replaced, so the input is copied aside first (sharded runs already read from the halo-extended copy)
    if (Fe > kTtcWindowMax && xe.p == dst.p) {
      h->launches++;
      DAWN_CUDA_OK(cudaMemcpy2DAsync(h->XE, (size_t)x.C * sizeof(float), x.p, (size_t)x.ld * sizeof(float), (size_t)x.C * sizeof(float),
                                     (size_t)F * P, cudaMemcpyDeviceToDevice, c.st));
      xe = Act{h->XE, x.C, x.C, x.H, x.W};
    }
    TemporalTcArgs a{};
    a.x = xe.p; a.ldx = xe.ld; a.res = x.p; a.ldr = x.ld; a.out = dst.p; a.ldo = dst.ld;
    a.F = Fe; a.P = P; a.q_lo = hl; a.q_hi = hl + F;
    a.Wqkv = w.tq; a.Wout = w.to; a.rot = h->ROT; a.table = h->ttc_table; a.band = h->cfg.win_width;
    a.inv_wscale = w.t_inv_wscale; a.inv_oscale = w.t_inv_oscale;
    double pairs = 0;
    for (int i = hl; i < hl + F; ++i) pairs += std::min(Fe - 1, i + a.band) - std::max(0, i - a.band) + 1;
    ProfScope ps(c, x.H == h->lH[0] ? PC_TEMPORAL_L0 : PC_ATTN_CORE, 2.0 * Me * x.C * 768 + 4.0 * 32 * 8 * P * pairs + 2.0 * F * P * 256 * x.C,
                 4.0 * (Me + 2.0 * F * P) * x.C);
    DAWN_TRY(launch_temporal_tc(a, c.st));
    return tap(c, name, dst);
  }
  if (fused_ok) {
    TemporalFusedArgs a{};
    a.x = xe.p; a.ldx = xe.ld; a.res = x.p; a.ldr = x.ld; a.out = dst.p; a.ldo = dst.ld;
    a.F = Fe; a.P = P; a.q_lo = hl; a.q_hi = hl + F;
    a.Wqkv = w.fq; a.Wout = w.fo; a.wsum = w.wsum; a.rot = h->ROT; a.bias = h->rel_bias; a.band = h->cfg.win_width;
    a.inv_wscale = w.f_inv_wscale; a.inv_oscale = w.f_inv_oscale;
    double pairs = 0;
    for (int i = hl; i < hl + F; ++i) pairs += std::min(Fe - 1, i + a.band) - std::max(0, i - a.band) + 1;
    ProfScope ps(c, x.H == h->lH[0] ? PC_TEMPORAL_L0 : PC_ATTN_CORE, 2.0 * Me * x.C * 768 + 4.0 * 32 * 8 * P * pairs + 2.0 * F * P * 256 * x.C,
                 4.0 * (Me + 2.0 * F * P) * x.C);
    DAWN_TRY(launch_temporal_fused(a, c.st));
    return tap(c, name, dst);
  }
  {
    GemmParams p; base_params(p, xe, Fe);
    p.B = w.Wqkv; p.Bimg = w.Wqkv_img; p.tc_scale = 1.0f / (kTcActScale * w.Wqkv_scale); p.ldb = 768; p.N = 768; p.K = x.C;
    p.wsum = w.wsum; p.rot = h->ROT;
    p.Out = h->QKV; p.ldo = 768;
    p.perm_pb = pb; p.perm_F = Fe; p.perm_in = 1; p.perm_out = 0;
    // output rows are written in plain order m (the permuted enumeration): treat the output as one M x 1 "image"
    p.OH = Me; p.OW = 1; p.OHs = Me; p.OWs = 1; p.IH = Me; p.IW = 1;
    DAWN_TRY(ln_gemm(c, p, EPI_QKV_TEMPORAL, PC_QKV, xe.p, xe.ld, xe.C, Me));
  }
  {
    AttnArgs a{};
    a.qkv = h->QKV; a.ld = 768; a.out = h->O; a.ldo = 256;
    a.nseq = P; a.L = Fe; a.seq_base_stride = 1; a.elem_stride = P; a.pb = pb;
    a.band = h->cfg.win_width; a.bias = h->rel_bias; a.q_lo = hl; a.q_hi = hl + F;
    double pairs = 0;
    for (int i = hl; i < hl + F; ++i) pairs += std::min(Fe - 1, i + a.band) - std::max(0, i - a.band) + 1;
    ProfScope ps(c, PC_ATTN_CORE, 4.0 * 32 * 8 * P * pairs, 4.0 * Me * 1024);
    if (h->use_attn_tc && attention_tc_supported(a)) DAWN_TRY(launch_attention_tc(a, c.st));
    else DAWN_TRY(launch_attention(a, c.st));
  }
  {
    Act o{h->O, 256, 256, Me, 1};
    GemmParams p; base_params(p, o, 1);
    set_weights(p, w.out);
    p.P = P;
    p.perm_pb = pb; p.perm_F = Fe; p.perm_in = 0; p.perm_out = 1; p.perm_f_lo = hl; p.perm_f_hi = hl + F;
    p.Res = x.p; p.ldr = x.ld; p.Out = dst.p; p.ldo = dst.ld;
    DAWN_TRY(c.gemm(p, EPI_PLAIN, PC_OUTPROJ));
  }
  return tap(c, name, dst);
}

// Residual(PreNorm(Attention over the h*w tokens of each frame)) (U:841-843), in place
int mid_spatial_attn(Ctx& c, const AttnW& w, const Act& x, const std::string& name) {
  dawn_unet* h = c.h;
  const int F = h->F, P = x.H * x.W, M = F * P;
  {
    GemmParams p; base_params(p, x, F);
    p.B = w.Wqkv; p.Bimg = w.Wqkv_img; p.tc_scale = 1.0f / (kTcActScale * w.Wqkv_scale); p.ldb = 768; p.N = 768; p.K = x.C;
    p.wsum = w.wsum;
    p.Out = h->QKV; p.ldo = 768;
    DAWN_TRY(ln_gemm(c, p, EPI_QKV_MID, PC_QKV, x.p, x.ld, x.C, M));
  }
  {
    AttnArgs a{};
    a.qkv = h->QKV; a.ld = 768; a.out = h->O; a.ldo = 256;
    a.nseq = F; a.L = P; a.seq_base_stride = P; a.elem_stride = 1;
    a.band = 1 << 30; a.bias = nullptr; a.q_lo = 0; a.q_hi = P;
    ProfScope ps(c, PC_ATTN_CORE, 4.0 * 32 * 8 * (double)F * P * P, 4.0 * M * 1024);
    if (h->use_attn_tc && attention_tc_supported(a)) DAWN_TRY(launch_attention_tc(a, c.st));
    else DAWN_TRY(launch_attention(a, c.st));
  }
  {
    Act o{h->O, 256, 256, x.H, x.W};
    GemmParams p; base_params(p, o, F);
    set_weights(p, w.out);
    p.Res = x.p; p.ldr = x.ld; p.Out = x.p; p.ldo = x.ld;
    DAWN_TRY(c.gemm(p, EPI_PLAIN, PC_OUTPROJ));
  }
  return tap(c, name, x);
}

// Residual(PreNorm(SpatialLinearAttention)) (U:602-627), in place
int sla(Ctx& c, const SlaW& w, const Act& x, const std::string& name) {
  dawn_unet* h = c.h;
  const int F = h->F, P = x.H * x.W, M = F * P;
  const int ldb = round_up(x.C, 64);
  const bool fused = h->use_fused_sla && w.fkv && sla_fused_supported(x.C, P) &&
                     sla_fused_part_floats(F, P) <= (size_t)(F + 2 * h->cfg.win_width) * h->lH[0] * h->lW[0] * 256;
  const int qld = fused ? 256 : 768;
  if (fused) {
    // k, v never leave the context kernel's registers; q never leaves the output kernel's
    SlaCtxArgs a{};
    a.x = x.p; a.ldx = x.ld; a.F = F; a.P = P; a.Wkv = w.fkv; a.inv_wscale = w.f_inv_wscale; a.part = h->O;
    {
      ProfScope ps(c, PC_SLA_CTX, 2.0 * M * x.C * 512 + 2.0 * 8 * 32 * 32 * M + 2.0 * F * 256 * 32 * x.C, 4.0 * M * x.C);
      h->launches++;                                   // context kernel + merge kernel
      DAWN_TRY(launch_sla_ctx_fused(a, w.WoutT, h->BF, ldb, c.st));
    }
    SlaOutArgs o{};
    o.x = x.p; o.ldx = x.ld; o.out = x.p; o.ldo = x.ld; o.F = F; o.P = P; o.Wq = w.fq; o.inv_wscale = w.fq_inv_wscale;
    o.Bf = h->BF; o.ldb = ldb; o.bias = w.bout;
    ProfScope ps2(c, PC_OUTPROJ, 2.0 * M * x.C * 256 + 2.0 * M * 256 * x.C, 8.0 * M * x.C);
    DAWN_TRY(launch_sla_out_fused(o, c.st));
    return tap(c, name, x);
  } else {
    GemmParams p; base_params(p, x, F);
    p.B = w.Wqkv; p.Bimg = w.Wqkv_img; p.tc_scale = 1.0f / (kTcActScale * w.Wqkv_scale); p.ldb = 768; p.N = 768; p.K = x.C;
    p.wsum = w.wsum; p.q_post_scale = 1.0f / sqrtf(32.0f);
    p.Out = h->QKV; p.ldo = 768;
    DAWN_TRY(ln_gemm(c, p, EPI_QKV_SLA, PC_QKV, x.p, x.ld, x.C, M));
  }
  if (!fused) {
    ProfScope ps(c, PC_SLA_CTX, 2.0 * 8 * 32 * 32 * M + 2.0 * F * 256 * 32 * x.C, 4.0 * M * 768);
    DAWN_TRY(launch_sla_context(h->QKV, 768, F, P, w.WoutT, x.C, h->BF, ldb, c.st));
  }
  {
    Act q{h->QKV, qld, 256, x.H, x.W};
    GemmParams p; base_params(p, q, F);
    p.B = h->BF; p.ldb = ldb; p.b_batch_stride = (long long)256 * ldb; p.N = x.C; p.K = 256;
    p.rows_per_batch = P; p.bias = w.bout;
    p.Res = x.p; p.ldr = x.ld; p.Out = x.p; p.ldo = x.ld;
    DAWN_TRY(c.gemm(p, EPI_PLAIN, PC_OUTPROJ));
  }
  return tap(c, name, x);
}

int downsample(Ctx& c, const ConvW& w, const Act& x, const Act& out, const std::string& name) {   // U:175-176
  GemmParams p; base_params(p, x, c.h->F);
  set_weights(p, w);
  p.OHs = out.H; p.OWs = out.W; p.in_stride = 2;
  p.ntaps = 16;
  for (int ky = 0; ky < 4; ++ky)
    for (int kx = 0; kx < 4; ++kx) { p.dy[ky * 4 + kx] = (signed char)(ky - 1); p.dx[ky * 4 + kx] = (signed char)(kx - 1); }
  p.M = c.h->F * out.H * out.W; p.rows_per_batch = p.M;
  p.OH = out.H; p.OW = out.W; p.P = out.H * out.W;
  p.Out = out.p; p.ldo = out.ld;
  DAWN_TRY(c.gemm(p, EPI_PLAIN, PC_CONV_OTHER));
  return tap(c, name, out);
}

int upsample(Ctx& c, const UpW& u, const Act& x, const Act& out, const std::string& name) {       // U:165-167
  if (c.h->use_tc && c.h->use_conv3 && u.all.img != nullptr) {
    GemmParams p; base_params(p, x, c.h->F);
    set_weights(p, u.all); set_square_taps(p, 3, 1);
    p.up2 = 1; p.Out = out.p; p.ldo = out.ld;
    if (tc_conv3_supported(p, EPI_PLAIN)) {
      ProfScope ps(c, PC_CONV_OTHER, 2.0 * p.M * 4.0 * x.C * x.C * 4, 4.0 * p.M * (x.C + 4.0 * x.C));
      DAWN_TRY(launch_tc_conv3(p, p.Bimg, c.st));
      return tap(c, name, out);
    }
  }
  for (int py = 0; py < 2; ++py)
    for (int px = 0; px < 2; ++px) {
      GemmParams p; base_params(p, x, c.h->F);
      set_weights(p, u.cls[py * 2 + px]);
      p.ntaps = 4;
      for (int ty = 0; ty < 2; ++ty)
        for (int tx = 0; tx < 2; ++tx) { p.dy[ty * 2 + tx] = (signed char)kUpD[py][ty]; p.dx[ty * 2 + tx] = (signed char)kUpD[px][tx]; }
      p.OH = out.H; p.OW = out.W; p.out_stride = 2; p.oy0 = py; p.ox0 = px;
      p.Out = out.p; p.ldo = out.ld;
      DAWN_TRY(c.gemm(p, EPI_PLAIN, PC_CONV_OTHER));
    }
  return tap(c, name, out);
}

// (F, P, C) channels-last -> (C, F, P) for taps
__global__ void nhwc_to_ncf_kernel(const float* __restrict__ x, int ld, int C, long long M, float* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * C) return;
  const long long m = idx / C; const int ch = (int)(idx - m * C);
  out[(size_t)ch * M + m] = x[(size_t)m * ld + ch];
}
int tap(Ctx& c, const std::string& name, const Act& a) {
  auto it = c.h->taps.find(name);
  if (it == c.h->taps.end() || it->second == nullptr) return 0;
  const long long M = (long long)c.h->F * a.H * a.W;
  nhwc_to_ncf_kernel<<<(int)((M * a.C + 255) / 256), 256, 0, c.st>>>(a.p, a.ld, a.C, M, it->second);
  DAWN_LAUNCH_OK();
  return 0;
}

// ------------------------------------------------------------------------------------------ per-clip tables
int prep_cond(dawn_unet* h, const float* cond, cudaStream_t st) {
  const int F = h->F;
  Ctx c{h, st};
  if (h->n_cond > 0 && !h->prof_on) {
    // three launches for all (block, cross-attention) pairs; the per-pair path below is kept for profiling
    h->launches += 3;
    return launch_cond_batched(cond, h->cond_dim, h->cond_descs, h->n_cond, h->cond_max_n1, h->cond_max_k, h->cond_max_co, F, st);
  }
  const int off[3] = {h->cfg.cond_aud, 0, h->cfg.cond_aud + h->cfg.cond_pose};          // pose, aud, eye slices (U:425-428)
  const int kd[3] = {h->cfg.cond_pose, h->cfg.cond_aud, h->cfg.cond_eye};
  for (auto& r : h->rb) {
    if (!r.cond) continue;
    for (int a = 0; a < 3; ++a) {
      ProfScope ps(c, PC_PREP, 0, 0);
      h->launches += 2;
      DAWN_TRY(launch_cond_mlp(cond, h->cond_dim, off[a], kd[a], r.mW[a], r.mB[a], 2 * r.co, F, h->CTX, st));
      DAWN_TRY(launch_linear_nobias(h->CTX, 2 * r.co, r.ca[a].Wkv, 128, F, h->KV, st));
      CaTableArgs t{};
      t.kv = h->KV; t.nkv = r.ca[a].nkv; t.qs = r.ca[a].qs; t.ks = r.ca[a].ks; t.Wout = r.ca[a].Wout; t.gout = r.ca[a].gout;
      t.co = r.co; t.ldbT = r.ldbT; t.ca = a; t.kq = r.kq; t.nkq = r.nkq; t.T = r.T; t.G = r.G;
      DAWN_TRY(launch_ca_tables(t, F, st));
    }
  }
  return 0;
}

// Per-clip constant part of the init conv (SURVEY a2) from ONE frame of the feature channels (fea: channel c at
// fea + c * cstride, H0*W0 values): kernel row ky runs as a 1 x k conv over the frame shifted by ky - pad rows ("batch" ky of
// the contraction kernel, weight rows [ky*k*cin_pad, (ky+1)*k*cin_pad) of the packed matrix) -> k x 32 CTAs instead of 32;
// the k partial maps are then added in a fixed order.  skip_flag: device-side path selection of the general entry.
int init_map(dawn_unet* h, const float* fea, long long cstride, cudaStream_t st, const int* skip_flag, int skip_if) {
  Ctx c{h, st};
  const int H0 = h->lH[0], W0 = h->lW[0], dim = h->cfg.dim, k = h->cfg.init_kernel_size;
  {
    ProfScope ps(c, PC_PREP, 0, 0);
    DAWN_TRY(launch_fea_shift_nhwc(fea, cstride, h->cfg.channels - 3, H0, W0, h->cin_pad, 3, k, h->FEA288, st, skip_flag, skip_if));
  }
  {
    Act in{h->FEA288, h->cin_pad, h->cin_pad, H0, W0};
    GemmParams p; base_params(p, in, k);                       // k "frames" = the shifted copies
    set_weights(p, h->init_full);
    p.ntaps = k;
    for (int kx = 0; kx < k; ++kx) { p.dy[kx] = 0; p.dx[kx] = (signed char)(kx - k / 2); }
    p.K = k * h->cin_pad; p.rows_per_batch = H0 * W0; p.b_batch_stride = (long long)k * h->cin_pad * h->init_full.ldb;
    p.bias = nullptr;
    p.Out = h->MAPPART; p.ldo = dim;
    p.skip_flag = skip_flag; p.skip_if = skip_if;
    ProfScope ps(c, PC_PREP, 0, 0);
    DAWN_TRY(launch_gemm(p, EPI_PLAIN, st));
  }
  ProfScope ps(c, PC_PREP, 0, 0);
  return launch_map_reduce(h->MAPPART, k, (long long)H0 * W0 * dim, h->init_full.b, dim, h->MAP, st, skip_flag, skip_if);
}

int forward_core(dawn_unet* h, const int64_t* t_dev, float* out, cudaStream_t st) {
  Ctx c{h, st};
  const int F = h->F, nlev = h->nlev, dim = h->cfg.dim;
  DAWN_CUDA_OK(cudaMemsetAsync(h->STATS, 0, sizeof(double) * 16 * h->n_stats, st));
  {
    ProfScope ps(c, PC_MISC, 0, 0);
    h->launches += 1;
    DAWN_TRY(launch_time_mlp(t_dev, h->time_freqs, dim, h->tW1, h->tb1, h->tW2, h->tb2, h->TSILU, st));
    DAWN_TRY(launch_film(h->film_descs, h->n_film, h->TSILU, h->tdim, st));
  }

  const int H0 = h->lH[0], W0 = h->lW[0];
  Act r{h->XR + dim, 2 * dim, dim, H0, W0};            // init conv output lives in the second half of cat(x, r) (U:911, 955)
  DAWN_TRY(tap(c, "init_conv", r));
  Act s0{h->S0, dim, dim, H0, W0};
  DAWN_TRY(temporal_attn(c, h->init_ta, r, s0, "init_temporal_attn"));

  Act x = s0;
  for (int L = 0; L < nlev; ++L) {
    const int co = h->in_out[L].second;
    Act a{h->bufA[L], co, co, h->lH[L], h->lW[L]}, b{h->bufB[L], co, co, h->lH[L], h->lW[L]};
    Act skip{h->CAT[L] + co, 2 * co, co, h->lH[L], h->lW[L]};
    const std::string pre = "downs." + std::to_string(L);
    DAWN_TRY(resblock(c, h->rb[h->rb_index[pre + ".0"]], x, a));
    DAWN_TRY(resblock(c, h->rb[h->rb_index[pre + ".1"]], a, b));
    DAWN_TRY(sla(c, h->down_sla[L], b, pre + ".2"));
    DAWN_TRY(temporal_attn(c, h->down_ta[L], b, skip, pre + ".3"));
    if (L < nlev - 1) {
      Act d{h->DS[L + 1], co, co, h->lH[L + 1], h->lW[L + 1]};
      DAWN_TRY(downsample(c, h->down_conv[L], skip, d, pre + ".4"));
      x = d;
    } else {
      x = skip;
    }
  }
  {
    const int L = nlev - 1, cm = h->in_out[L].second;
    Act a{h->bufA[L], cm, cm, h->lH[L], h->lW[L]};
    Act xfirst{h->CAT[L], 2 * cm, cm, h->lH[L], h->lW[L]};
    DAWN_TRY(resblock(c, h->rb[h->rb_index["mid_block1"]], x, a));
    DAWN_TRY(mid_spatial_attn(c, h->mid_sa, a, "mid_spatial_attn"));
    DAWN_TRY(temporal_attn(c, h->mid_ta, a, a, "mid_temporal_attn"));
    DAWN_TRY(resblock(c, h->rb[h->rb_index["mid_block2"]], a, xfirst));
  }
  for (int K = 0; K < nlev; ++K) {
    const int l = nlev - 1 - K;
    const int ci = h->in_out[l].first, co = h->in_out[l].second;
    Act cat{h->CAT[l], 2 * co, 2 * co, h->lH[l], h->lW[l]};
    Act a{h->bufA[l], ci, ci, h->lH[l], h->lW[l]}, b{h->bufB[l], ci, ci, h->lH[l], h->lW[l]};
    const std::string pre = "ups." + std::to_string(K);
    DAWN_TRY(resblock(c, h->rb[h->rb_index[pre + ".0"]], cat, a));
    DAWN_TRY(resblock(c, h->rb[h->rb_index[pre + ".1"]], a, b));
    DAWN_TRY(sla(c, h->up_sla[K], b, pre + ".2"));
    if (K < nlev - 1) {
      DAWN_TRY(temporal_attn(c, h->up_ta[K], b, b, pre + ".3"));
      const int cn = h->in_out[l - 1].second;        // == ci
      Act up{h->CAT[l - 1], 2 * cn, cn, h->lH[l - 1], h->lW[l - 1]};
      DAWN_TRY(upsample(c, h->up_conv[K], b, up, pre + ".4"));
    } else {
      Act xf{h->XR, 2 * dim, dim, H0, W0};
      DAWN_TRY(temporal_attn(c, h->up_ta[K], b, xf, pre + ".3"));
    }
  }
  Act xr{h->XR, 2 * dim, 2 * dim, H0, W0};
  Act hf{h->HF, dim, dim, H0, W0}, ho{h->HO, dim, dim, H0, W0};
  DAWN_TRY(resblock(c, h->rb[h->rb_index["final_conv.0"]], xr, hf));
  DAWN_TRY(resblock(c, h->rb[h->rb_index["occlusion_map.0"]], xr, ho));
  ProfScope ps(c, PC_MISC, 0, 4.0 * F * H0 * W0 * (2 * dim + 3));
  DAWN_TRY(launch_heads_out(h->HF, h->HO, dim, F * H0 * W0, h->headW[0], h->headB[0], h->cfg.out_grid_dim,
                            h->headW[1], h->headB[1], h->cfg.out_conf_dim, out, st));
  return 0;
}

}  // namespace

// ============================================================================================== C-ABI
extern "C" {

const char* dawn_last_error(void) { return g_last_error.c_str(); }
const char* dawn_build_info(void) { return "dawn_unet sm_100a; contractions: tcgen05 kind::f16 FP16x3 (TMEM accumulators) + mma.sync m16n8k16 FP16x3 fused attention kernels; fallback mma.sync 3xTF32"; }

// The kernel launchers cache per-function attributes (dynamic shared-memory opt-in, SM count) in process-wide statics: the
// library is built for ONE GPU PER PROCESS (torchrun / one rank per GPU).  A second device in the same process would launch
// with attributes that were never set there, so refuse it loudly instead.
int dawn_check_single_device(void) {
  static int first_dev = -1;
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return 0; }     // no driver / no device here (CPU-only build check)
  if (first_dev < 0) first_dev = dev;
  if (dev != first_dev) {
    set_last_error("this process already uses CUDA device " + std::to_string(first_dev) + "; the library supports one GPU per process "
                   "(launch one rank per GPU), got device " + std::to_string(dev));
    return -1;
  }
  return 0;
}

int dawn_unet_create(const dawn_unet_cfg* cfg, dawn_unet** out) {
  DAWN_CHECK(cfg && out, "null argument");
  DAWN_TRY(dawn_check_single_device());
  DAWN_CHECK(cfg->attn_heads == 8 && cfg->attn_dim_head == 32, "only attn_heads=8, attn_dim_head=32 are supported");
  DAWN_CHECK(cfg->resnet_groups == 8, "only resnet_groups=8 is supported");
  DAWN_CHECK(cfg->dim % 64 == 0 && cfg->dim <= 128, "dim must be 64 or 128");
  DAWN_CHECK(cfg->n_levels >= 2 && cfg->n_levels <= 6, "n_levels out of range");
  DAWN_CHECK(cfg->init_kernel_size == 7 || cfg->init_kernel_size == 5 || cfg->init_kernel_size == 3, "init kernel must be 3, 5 or 7");
  DAWN_CHECK(cfg->win_width >= 1 && cfg->win_width <= 120, "win_width out of range");
  dawn_unet* h = new dawn_unet();
  h->cfg = *cfg;
  { const char* e = getenv("DAWN_TC"); h->use_tc = !(e && e[0] == '0'); }
  { const char* e = getenv("DAWN_ATTN_TC"); h->use_attn_tc = !(e && e[0] == '0'); }
  { const char* e = getenv("DAWN_FUSED_TA"); h->use_fused_ta = !(e && e[0] == '0'); }
  { const char* e = getenv("DAWN_TA_TC"); h->use_ta_tc = !(e && e[0] == '0'); }
  { const char* e = getenv("DAWN_CONV3_TMA"); h->conv3_tma = (e && e[0] >= '0' && e[0] <= '2') ? e[0] - '0' : 1; }
  { const char* e = getenv("DAWN_FUSED_SLA"); h->use_fused_sla = !(e && e[0] == '0'); }
  { const char* e = getenv("DAWN_FUSED_CA"); h->use_fused_ca = !(e && e[0] == '0'); }
  { const char* e = getenv("DAWN_PRESPLIT"); h->use_presplit = !(e && e[0] == '0'); }
  { const char* e = getenv("DAWN_TC_CONV3"); h->use_conv3 = !(e && e[0] == '0'); }
  { const char* e = getenv("DAWN_PREP_V1"); h->prep_v1 = (e && e[0] == '1'); }
  h->nlev = cfg->n_levels;
  h->dims.push_back(cfg->dim);
  for (int i = 0; i < cfg->n_levels; ++i) h->dims.push_back(cfg->dim * cfg->dim_mults[i]);
  for (int i = 0; i < cfg->n_levels; ++i) h->in_out.push_back({h->dims[i], h->dims[i + 1]});
  for (auto& io : h->in_out)
    if (io.second > 1024 || io.second * 2 > 1024 + 1024) { delete h; set_last_error("channel count too large"); return -1; }
  h->cond_dim = cfg->cond_aud + cfg->cond_pose + cfg->cond_eye;
  h->tdim = 4 * cfg->dim;
  h->cin_pad = round_up(cfg->channels, 32);
  *out = h;
  return 0;
}

void dawn_unet_destroy(dawn_unet* h) {
  if (!h) return;
  for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
  if (h->samp_exec) cudaGraphExecDestroy(h->samp_exec);
  if (h->samp_stream) cudaStreamDestroy(h->samp_stream);
  if (h->sh_comm && g_nccl.ok) g_nccl.CommDestroy(h->sh_comm);
  for (int r = 0; r < kP2pMaxRanks; ++r)
    if (h->p2p_peer[r] && h->p2p_peer[r] != h->p2p_own) cudaIpcCloseMemHandle(h->p2p_peer[r]);
  free_all(h->owned);
  free_all(h->ws_owned);
  delete h;
}

int dawn_unet_set_param(dawn_unet* h, const char* name, const float* host, const int64_t* shape, int ndim) {
  DAWN_CHECK(h && name && host && (shape || ndim == 0), "null argument");
  HostParam p;
  p.shape.assign(shape, shape + ndim);
  p.data.assign(host, host + p.numel());
  h->raw[name] = std::move(p);
  h->committed = false;
  return 0;
}

static void drop_sampler_graph(dawn_unet* h) {
  if (h->samp_exec) { cudaGraphExecDestroy(h->samp_exec); h->samp_exec = nullptr; }
}

int dawn_unet_commit_params(dawn_unet* h) {
  DAWN_CHECK(h, "null handle");
  drop_sampler_graph(h);
  free_all(h->owned);
  h->rb.clear(); h->rb_index.clear();
  h->down_ta.clear(); h->up_ta.clear(); h->down_sla.clear(); h->up_sla.clear(); h->down_conv.clear(); h->up_conv.clear();
  const auto& cfg = h->cfg;
  const int dim = cfg.dim, nlev = h->nlev, k = cfg.init_kernel_size;
  // init conv: full (all input channels, padded) and the 3-channel slice for the hoisted path
  DAWN_TRY(pack_conv(h, "init_conv", dim, cfg.channels, k, k, h->cin_pad, true, &h->init_full));
  {
    const HostParam* w;
    DAWN_TRY(need(h, "init_conv.weight", {dim, cfg.channels, 1, k, k}, &w));
    std::vector<float> w3((size_t)k * k * 3 * dim);
    for (int t = 0; t < k * k; ++t)
      for (int c = 0; c < 3; ++c)
        for (int n = 0; n < dim; ++n) w3[((size_t)t * 3 + c) * dim + n] = w->data[((size_t)n * cfg.channels + c) * k * k + t];
    DAWN_TRY(dev_upload(h, w3, &h->init_w3));
  }
  DAWN_TRY(upload_raw(h, "aux.time_freqs", {dim / 2}, &h->time_freqs));
  DAWN_TRY(upload_raw(h, "aux.rel_bias", {8, 2 * cfg.win_width + 1}, &h->rel_bias));
  h->ttc_table = nullptr;
  if (cfg.win_width >= 1 && cfg.win_width <= kTtcBandMax) {
    const HostParam* rb;
    DAWN_TRY(need(h, "aux.rel_bias", {8, 2 * cfg.win_width + 1}, &rb));
    std::vector<float> tab;
    temporal_tc_table(rb->data.data(), cfg.win_width, tab);
    DAWN_TRY(dev_upload(h, tab, &h->ttc_table));
  }
  DAWN_TRY(upload_raw(h, "time_mlp.1.weight", {h->tdim, dim}, &h->tW1));
  DAWN_TRY(upload_raw(h, "time_mlp.1.bias", {h->tdim}, &h->tb1));
  DAWN_TRY(upload_raw(h, "time_mlp.3.weight", {h->tdim, h->tdim}, &h->tW2));
  DAWN_TRY(upload_raw(h, "time_mlp.3.bias", {h->tdim}, &h->tb2));
  DAWN_TRY(upload_raw(h, "init_temporal_attn.fn.fn.fn.rotary_emb.freqs", {16}, &h->rot_freqs));
  DAWN_TRY(pack_attn(h, "init_temporal_attn.fn.norm", "init_temporal_attn.fn.fn.fn", dim, &h->init_ta));
  int stat_counter = 0;
  for (int L = 0; L < nlev; ++L) {
    const int ci = h->in_out[L].first, co = h->in_out[L].second;
    const std::string pre = "downs." + std::to_string(L);
    DAWN_TRY(pack_resblock(h, pre + ".0", ci, co, true, &stat_counter));
    DAWN_TRY(pack_resblock(h, pre + ".1", co, co, true, &stat_counter));
    SlaW s; DAWN_TRY(pack_sla(h, pre + ".2.fn", co, &s)); h->down_sla.push_back(s);
    AttnW a; DAWN_TRY(pack_attn(h, pre + ".3.fn.norm", pre + ".3.fn.fn.fn", co, &a)); h->down_ta.push_back(a);
    if (L < nlev - 1) {
      ConvW d; DAWN_TRY(pack_conv(h, pre + ".4", co, co, 4, 4, co, true, &d)); h->down_conv.push_back(d);
    }
  }
  const int mid = h->dims.back();
  DAWN_TRY(pack_resblock(h, "mid_block1", mid, mid, true, &stat_counter));
  DAWN_TRY(pack_attn(h, "mid_spatial_attn.fn.norm", "mid_spatial_attn.fn.fn.fn", mid, &h->mid_sa));
  DAWN_TRY(pack_attn(h, "mid_temporal_attn.fn.norm", "mid_temporal_attn.fn.fn.fn", mid, &h->mid_ta));
  DAWN_TRY(pack_resblock(h, "mid_block2", mid, mid, true, &stat_counter));
  for (int K = 0; K < nlev; ++K) {
    const int l = nlev - 1 - K;
    const int ci = h->in_out[l].first, co = h->in_out[l].second;
    const std::string pre = "ups." + std::to_string(K);
    DAWN_TRY(pack_resblock(h, pre + ".0", 2 * co, ci, true, &stat_counter));
    DAWN_TRY(pack_resblock(h, pre + ".1", ci, ci, true, &stat_counter));
    SlaW s; DAWN_TRY(pack_sla(h, pre + ".2.fn", ci, &s)); h->up_sla.push_back(s);
    AttnW a; DAWN_TRY(pack_attn(h, pre + ".3.fn.norm", pre + ".3.fn.fn.fn", ci, &a)); h->up_ta.push_back(a);
    if (K < nlev - 1) {
      UpW u; DAWN_TRY(pack_up(h, pre + ".4", ci, &u)); h->up_conv.push_back(u);
    }
  }
  // heads: ResnetBlock_ca_mul without time/cond MLPs (their cross-attention parameters exist but never run, U:862, 875)
  DAWN_TRY(pack_resblock(h, "final_conv.0", 2 * dim, dim, false, &stat_counter));
  DAWN_TRY(pack_resblock(h, "occlusion_map.0", 2 * dim, dim, false, &stat_counter));
  DAWN_TRY(upload_raw(h, "final_conv.1.weight", {cfg.out_grid_dim, dim, 1, 1, 1}, &h->headW[0]));
  DAWN_TRY(upload_raw(h, "final_conv.1.bias", {cfg.out_grid_dim}, &h->headB[0]));
  DAWN_TRY(upload_raw(h, "occlusion_map.1.weight", {cfg.out_conf_dim, dim, 1, 1, 1}, &h->headW[1]));
  DAWN_TRY(upload_raw(h, "occlusion_map.1.bias", {cfg.out_conf_dim}, &h->headB[1]));
  h->n_stats = stat_counter;
  h->committed = true;
  // a changed parameter set invalidates per-clip tables
  h->have_invariants = false;
  if (h->F > 0) return dawn_unet_set_num_frames(h, h->F, h->H, h->W);
  return 0;
}

int dawn_unet_set_num_frames(dawn_unet* h, int F, int height, int width) {
  DAWN_CHECK(h, "null handle");
  drop_sampler_graph(h);
  DAWN_CHECK(h->committed, "commit_params must precede set_num_frames");
  DAWN_CHECK(F >= 1 && F <= 65535, "F out of range");
  const int nlev = h->nlev, dim = h->cfg.dim;
  const int div = 1 << (nlev - 1);
  DAWN_CHECK(height % div == 0 && width % div == 0 && height >= div && width >= div,
             "latent height/width must be divisible by 2^(levels-1)");
  free_all(h->ws_owned);
  h->ws_bytes = 0;
  h->have_invariants = false;
  h->F = F; h->H = height; h->W = width;
  h->lH.assign(nlev, 0); h->lW.assign(nlev, 0);
  for (int l = 0; l < nlev; ++l) { h->lH[l] = height >> l; h->lW[l] = width >> l; }
  auto& own = h->ws_owned;
  const size_t P0 = (size_t)height * width, M0 = (size_t)F * P0;
  int64_t* cnt = &h->ws_bytes;
  DAWN_TRY(dev_alloc(own, M0 * h->cin_pad, &h->X288, cnt));
  DAWN_TRY(dev_alloc(own, P0 * h->cin_pad * h->cfg.init_kernel_size, &h->FEA288, cnt));   // k row-shifted copies
  DAWN_TRY(dev_alloc(own, P0 * dim * h->cfg.init_kernel_size, &h->MAPPART, cnt));
  { float* f; DAWN_TRY(dev_alloc(own, 4, &f, cnt)); h->VARY = (int*)f; }
  DAWN_TRY(dev_alloc(own, P0 * dim, &h->MAP, cnt));
  DAWN_TRY(dev_alloc(own, M0 * 2 * dim, &h->XR, cnt));
  DAWN_TRY(dev_alloc(own, M0 * dim, &h->S0, cnt));
  h->bufA.assign(nlev, nullptr); h->bufB.assign(nlev, nullptr); h->CAT.assign(nlev, nullptr); h->DS.assign(nlev, nullptr);
  size_t max_mc = 0, max_bf = 0;
  for (int l = 0; l < nlev; ++l) {
    const size_t Ml = (size_t)F * h->lH[l] * h->lW[l];
    const int ci = h->in_out[l].first, co = h->in_out[l].second;
    DAWN_TRY(dev_alloc(own, Ml * co, &h->bufA[l], cnt));
    DAWN_TRY(dev_alloc(own, Ml * co, &h->bufB[l], cnt));
    DAWN_TRY(dev_alloc(own, Ml * 2 * co, &h->CAT[l], cnt));
    if (l > 0) DAWN_TRY(dev_alloc(own, Ml * ci, &h->DS[l], cnt));
    max_mc = std::max(max_mc, Ml * co);
    max_bf = std::max(max_bf, (size_t)F * 256 * round_up(co, 64));
  }
  max_mc = std::max(max_mc, M0 * dim);
  DAWN_TRY(dev_alloc(own, max_mc, &h->Y, cnt));
  DAWN_TRY(dev_alloc(own, max_mc, &h->A1, cnt));
  const size_t Mext = (size_t)(F + 2 * h->cfg.win_width) * P0;      // rows incl. temporal halos of a sharded clip
  DAWN_TRY(dev_alloc(own, Mext * 768, &h->QKV, cnt));
  DAWN_TRY(dev_alloc(own, Mext * 256, &h->O, cnt));
  DAWN_TRY(dev_alloc(own, Mext * 2, &h->ROWSTATS, cnt));
  DAWN_TRY(dev_alloc(own, Mext * dim, &h->XE, cnt));
  DAWN_TRY(dev_alloc(own, M0 * 24, &h->GATES, cnt));
  DAWN_TRY(dev_alloc(own, M0 * 32, &h->WT, cnt));
  DAWN_TRY(dev_alloc(own, max_bf, &h->BF, cnt));
  DAWN_TRY(dev_alloc(own, M0 * dim, &h->HF, cnt));
  DAWN_TRY(dev_alloc(own, M0 * dim, &h->HO, cnt));
  DAWN_TRY(dev_alloc(own, (size_t)(F + 2 * h->cfg.win_width) * 32, &h->ROT, cnt));
  DAWN_TRY(dev_alloc(own, h->tdim, &h->TSILU, cnt));
  DAWN_TRY(dev_alloc(own, (size_t)F * 2048, &h->CTX, cnt));
  DAWN_TRY(dev_alloc(own, (size_t)F * 128, &h->KV, cnt));
  {
    float* s; DAWN_TRY(dev_alloc(own, (size_t)h->n_stats * 32, &s, cnt)); h->STATS = (double*)s;
    float* t; DAWN_TRY(dev_alloc(own, 4, &t, cnt)); h->T_HOSTSIDE = (int64_t*)t;
  }
  DAWN_TRY(dev_alloc(own, 3 * M0, &h->H_XT, cnt));
  DAWN_TRY(dev_alloc(own, (size_t)(h->cfg.channels - 3) * P0, &h->H_FEA, cnt));
  DAWN_TRY(dev_alloc(own, (size_t)F * h->cond_dim, &h->H_COND, cnt));
  DAWN_TRY(dev_alloc(own, (size_t)(h->cfg.out_grid_dim + h->cfg.out_conf_dim) * M0, &h->H_OUT, cnt));
  // per-block per-clip tables
  std::vector<FilmDesc> descs;
  for (auto& r : h->rb) {
    if (!r.cond) continue;
    r.ldbT = round_up(r.co, 64);
    DAWN_TRY(dev_alloc(own, 2 * r.co, &r.film, cnt));
    DAWN_TRY(dev_alloc(own, (size_t)F * 3 * 64, &r.kq, cnt));
    DAWN_TRY(dev_alloc(own, 24, &r.nkq, cnt));
    DAWN_TRY(dev_alloc(own, (size_t)F * 32 * r.ldbT, &r.T, cnt));
    DAWN_CUDA_OK(cudaMemset(r.T, 0, (size_t)F * 32 * r.ldbT * sizeof(float)));
    DAWN_TRY(dev_alloc(own, (size_t)F * 3 * 81, &r.G, cnt));
    descs.push_back(FilmDesc{r.tW, r.tB, r.film, 2 * r.co});
  }
  {
    float* d; DAWN_TRY(dev_alloc(own, descs.size() * sizeof(FilmDesc) / sizeof(float) + 4, &d, cnt));
    DAWN_CUDA_OK(cudaMemcpy(d, descs.data(), descs.size() * sizeof(FilmDesc), cudaMemcpyHostToDevice));
    h->film_descs = (FilmDesc*)d; h->n_film = (int)descs.size();
  }
  {
    // descriptors of the per-clip conditioning pipeline: one per (conditioned block, cross-attention), own scratch each
    const int off[3] = {h->cfg.cond_aud, 0, h->cfg.cond_aud + h->cfg.cond_pose};          // pose, aud, eye slices (U:425-428)
    const int kd[3] = {h->cfg.cond_pose, h->cfg.cond_aud, h->cfg.cond_eye};
    std::vector<CondDesc> cd;
    h->cond_max_n1 = h->cond_max_k = h->cond_max_co = 0;
    for (auto& r : h->rb) {
      if (!r.cond) continue;
      for (int a = 0; a < 3; ++a) {
        CondDesc d{};
        d.mW = r.mW[a]; d.mB = r.mB[a]; d.off = off[a]; d.K = kd[a]; d.n1 = 2 * r.co; d.Wkv = r.ca[a].Wkv;
        DAWN_TRY(dev_alloc(own, (size_t)F * d.n1, &d.ctx, cnt));
        DAWN_TRY(dev_alloc(own, (size_t)F * 128, &d.kv, cnt));
        d.t.kv = d.kv; d.t.nkv = r.ca[a].nkv; d.t.qs = r.ca[a].qs; d.t.ks = r.ca[a].ks; d.t.Wout = r.ca[a].Wout; d.t.gout = r.ca[a].gout;
        d.t.co = r.co; d.t.ldbT = r.ldbT; d.t.ca = a; d.t.kq = r.kq; d.t.nkq = r.nkq; d.t.T = r.T; d.t.G = r.G;
        cd.push_back(d);
        h->cond_max_n1 = std::max(h->cond_max_n1, d.n1); h->cond_max_k = std::max(h->cond_max_k, d.K); h->cond_max_co = std::max(h->cond_max_co, r.co);
      }
    }
    float* d; DAWN_TRY(dev_alloc(own, cd.size() * sizeof(CondDesc) / sizeof(float) + 4, &d, cnt));
    DAWN_CUDA_OK(cudaMemcpy(d, cd.data(), cd.size() * sizeof(CondDesc), cudaMemcpyHostToDevice));
    h->cond_descs = (CondDesc*)d; h->n_cond = (int)cd.size();
  }
  h->sh_nranks = 1; h->sh_rank = 0; h->sh_Fglobal = F; h->sh_halo_l = 0; h->sh_halo_r = 0;   // a new geometry is unsharded until init_shard
  h->p2p_ready = false;
  DAWN_TRY(launch_rotary_table(h->rot_freqs, F, 0, h->ROT, 0));
  DAWN_CUDA_OK(cudaDeviceSynchronize());
  return 0;
}

int dawn_unet_set_clip_invariants(dawn_unet* h, const float* fea, const float* cond, void* stream) {
  DAWN_CHECK(h && fea && cond, "null argument");
  DAWN_CHECK(h->F > 0, "set_num_frames must precede set_clip_invariants");
  cudaStream_t st = (cudaStream_t)stream;
  Ctx c{h, st};
  const int H0 = h->lH[0], W0 = h->lW[0], dim = h->cfg.dim, k = h->cfg.init_kernel_size;
  // per-clip constant part of the init conv: conv(cat[0, fea]) + bias  (linearity; SURVEY a2)
  if (!h->prep_v1) {
    DAWN_TRY(init_map(h, fea, (long long)H0 * W0, st, nullptr, 0));
  } else {
  {
    ProfScope ps(c, PC_PREP, 0, 0);
    DAWN_TRY(launch_ncf_to_nhwc(fea, h->cfg.channels - 3, 1, H0 * W0, h->cin_pad, 3, h->FEA288, st));
  }
  {
    Act in{h->FEA288, h->cin_pad, h->cin_pad, H0, W0};
    GemmParams p; base_params(p, in, 1);
    set_weights(p, h->init_full); set_square_taps(p, k, k / 2);
    p.Out = h->MAP; p.ldo = dim;
    DAWN_TRY(c.gemm(p, EPI_PLAIN, PC_PREP));
  }
  }
  DAWN_TRY(prep_cond(h, cond, st));
  h->have_invariants = true;
  return 0;
}

int dawn_unet_forward(dawn_unet* h, const float* x, const int64_t* t, const float* cond, float* out, void* stream) {
  DAWN_CHECK(h && x && t && cond && out, "null argument");
  DAWN_CHECK(h->F > 0, "set_num_frames must precede forward");
  cudaStream_t st = (cudaStream_t)stream;
  h->launches = 0;
  Ctx c{h, st};
  const int H0 = h->lH[0], W0 = h->lW[0], dim = h->cfg.dim, k = h->cfg.init_kernel_size;
  DAWN_TRY(prep_cond(h, cond, st));
  h->have_invariants = false;         // MAP is refreshed by this entry only when the features turn out frame-invariant
  // Path selection on the device, no host synchronisation: one pass over x decides whether channels 3.. are the same in every
  // frame (the reference's sampler tiles them, U:1167); both paths are enqueued and the kernels of the one not taken return
  // at once.  invariant -> hoisted init conv (map from frame 0 + 3 live channels); varying -> full k x k conv over all channels.
  const int* vary = nullptr;
  if (!h->prep_v1) {
    ProfScope ps(c, PC_MISC, 0, 4.0 * h->F * H0 * W0 * h->cfg.channels);
    DAWN_TRY(launch_frame_invariance(x, 3, h->cfg.channels, h->F, H0 * W0, h->VARY, st));
    vary = h->VARY;
  }
  {
    ProfScope ps(c, PC_MISC, 0, 8.0 * h->F * H0 * W0 * h->cin_pad);
    DAWN_TRY(launch_ncf_to_nhwc(x, h->cfg.channels, h->F, H0 * W0, h->cin_pad, 0, h->X288, st, vary, 0));
  }
  {
    Act in{h->X288, h->cin_pad, h->cin_pad, H0, W0};
    GemmParams p; base_params(p, in, h->F);
    set_weights(p, h->init_full); set_square_taps(p, k, k / 2);
    p.Out = h->XR + dim; p.ldo = 2 * dim;
    p.skip_flag = vary; p.skip_if = 0;
    ProfScope ps(c, PC_CONV_OTHER, 2.0 * p.M * (double)p.N * p.K, 4.0 * p.M * ((double)p.Cin + p.N));
    DAWN_TRY(launch_gemm(p, EPI_PLAIN, st));      // Cin = 288 is not a tcgen05 shape: always the mma.sync kernel (it has the skip flag)
  }
  if (vary) {
    DAWN_TRY(init_map(h, x + (size_t)3 * h->F * H0 * W0, (long long)h->F * H0 * W0, st, vary, 1));
    const double k2 = (double)k * k;
    ProfScope ps(c, PC_MISC, 2.0 * h->F * H0 * W0 * dim * 3 * k2, 4.0 * h->F * H0 * W0 * (dim + 3));
    DAWN_TRY(launch_init_conv_x3(x, h->F, H0, W0, h->init_w3, h->MAP, dim, h->XR + dim, 2 * dim, k, st, vary, 1));
  }
  return forward_core(h, t, out, st);
}

int dawn_unet_forward_x3(dawn_unet* h, const float* x_t, const int64_t* t, float* out, void* stream) {
  DAWN_CHECK(h && x_t && t && out, "null argument");
  DAWN_CHECK(h->F > 0 && h->have_invariants, "set_clip_invariants must precede forward_x3");
  cudaStream_t st = (cudaStream_t)stream;
  h->launches = 0;
  const int H0 = h->lH[0], W0 = h->lW[0], dim = h->cfg.dim;
  {
    Ctx c{h, st};
    const double k2 = (double)h->cfg.init_kernel_size * h->cfg.init_kernel_size;
    ProfScope ps(c, PC_MISC, 2.0 * h->F * H0 * W0 * dim * 3 * k2, 4.0 * h->F * H0 * W0 * (dim + 3));
    DAWN_TRY(launch_init_conv_x3(x_t, h->F, H0, W0, h->init_w3, h->MAP, dim, h->XR + dim, 2 * dim,
                                 h->cfg.init_kernel_size, st));
  }
  return forward_core(h, t, out, st);
}

int dawn_unet_forward_host(dawn_unet* h, const float* x_t, const float* fea, const float* cond, int64_t t, float* out) {
  DAWN_CHECK(h && x_t && fea && cond && out, "null argument");
  DAWN_CHECK(h->F > 0, "set_num_frames must precede forward_host");
  cudaStream_t st = 0;
  const size_t M0 = (size_t)h->F * h->H * h->W, P0 = (size_t)h->H * h->W;
  const size_t nout = (size_t)(h->cfg.out_grid_dim + h->cfg.out_conf_dim) * M0;
  DAWN_CUDA_OK(cudaMemcpyAsync(h->H_XT, x_t, 3 * M0 * sizeof(float), cudaMemcpyHostToDevice, st));
  DAWN_CUDA_OK(cudaMemcpyAsync(h->H_FEA, fea, (size_t)(h->cfg.channels - 3) * P0 * sizeof(float), cudaMemcpyHostToDevice, st));
  DAWN_CUDA_OK(cudaMemcpyAsync(h->H_COND, cond, (size_t)h->F * h->cond_dim * sizeof(float), cudaMemcpyHostToDevice, st));
  DAWN_CUDA_OK(cudaMemcpyAsync(h->T_HOSTSIDE, &t, sizeof(int64_t), cudaMemcpyHostToDevice, st));
  DAWN_TRY(dawn_unet_set_clip_invariants(h, h->H_FEA, h->H_COND, st));
  const int64_t prep_launches = h->launches;
  DAWN_TRY(dawn_unet_forward_x3(h, h->H_XT, h->T_HOSTSIDE, h->H_OUT, st));
  h->launches += prep_launches;
  DAWN_CUDA_OK(cudaMemcpyAsync(out, h->H_OUT, nout * sizeof(float), cudaMemcpyDeviceToHost, st));
  DAWN_CUDA_OK(cudaStreamSynchronize(st));
  return 0;
}

int dawn_unet_tap_shape(dawn_unet* h, const char* name, int* C, int* hl, int* wl) {
  DAWN_CHECK(h && name && C && hl && wl && h->F > 0, "bad argument");
  const std::string n(name);
  const int nlev = h->nlev, dim = h->cfg.dim;
  auto set = [&](int c, int l) { *C = c; *hl = h->lH[l]; *wl = h->lW[l]; return 0; };
  if (n == "init_conv" || n == "init_temporal_attn" || n == "final_conv.0" || n == "occlusion_map.0") return set(dim, 0);
  if (n.rfind("mid_", 0) == 0) return set(h->dims.back(), nlev - 1);
  int L = -1, j = -1;
  if (sscanf(name, "downs.%d.%d", &L, &j) == 2 && L >= 0 && L < nlev) {
    if (j == 4) { DAWN_CHECK(L < nlev - 1, "no such tap"); return set(h->in_out[L].second, L + 1); }
    return set(h->in_out[L].second, L);
  }
  if (sscanf(name, "ups.%d.%d", &L, &j) == 2 && L >= 0 && L < nlev) {
    const int l = nlev - 1 - L;
    if (j == 4) { DAWN_CHECK(L < nlev - 1, "no such tap"); return set(h->in_out[l].first, l - 1); }
    return set(h->in_out[l].first, l);
  }
  set_last_error("unknown tap: " + n);
  return -1;
}

int dawn_unet_set_tap(dawn_unet* h, const char* name, float* dst) {
  DAWN_CHECK(h && name, "null argument");
  if (dst) h->taps[name] = dst; else h->taps.erase(name);
  return 0;
}

int dawn_nccl_unique_id(char* out128) {
  DAWN_CHECK(out128, "null argument");
  DAWN_TRY(load_nccl());
  NcclUniqueId id;
  DAWN_NCCL_OK(g_nccl.GetUniqueId(&id));
  memcpy(out128, id.internal, 128);
  return 0;
}

int dawn_unet_init_shard(dawn_unet* h, const char* id128, int nranks, int rank, int F_global) {
  DAWN_CHECK(h && id128, "null argument");
  DAWN_CHECK(h->F > 0, "set_num_frames (with the LOCAL frame count) must precede init_shard");
  DAWN_CHECK(nranks >= 1 && rank >= 0 && rank < nranks, "bad rank");
  DAWN_CHECK(F_global == h->F * nranks, "F_global must equal nranks * local frames (equal contiguous frame ranges)");
  DAWN_CHECK(nranks == 1 || h->F >= h->cfg.win_width, "each rank must own at least win_width frames (only neighbours exchange halos)");
  drop_sampler_graph(h);
  if (nranks > 1) {
    DAWN_TRY(load_nccl());
    if (h->sh_comm) { g_nccl.CommDestroy(h->sh_comm); h->sh_comm = nullptr; }
    NcclUniqueId id;
    memcpy(id.internal, id128, 128);
    DAWN_NCCL_OK(g_nccl.CommInitRank(&h->sh_comm, nranks, id, rank));
  }
  h->sh_nranks = nranks; h->sh_rank = rank; h->sh_Fglobal = F_global;
  h->p2p_ready = false;
  h->sh_halo_l = (rank > 0) ? h->cfg.win_width : 0;
  h->sh_halo_r = (rank < nranks - 1) ? h->cfg.win_width : 0;
  // rotary positions of the halo-extended local sequence are GLOBAL frame indices
  const int pos0 = rank * h->F - h->sh_halo_l;
  DAWN_TRY(launch_rotary_table(h->rot_freqs, h->sh_halo_l + h->F + h->sh_halo_r, pos0, h->ROT, 0));
  DAWN_CUDA_OK(cudaDeviceSynchronize());
  return 0;
}

// Peer-memory mailboxes for the GroupNorm all-reduce: export this rank's mailbox as a cudaIpc handle (64 bytes) ...
int dawn_unet_shard_ipc_export(dawn_unet* h, char* out64) {
  DAWN_CHECK(h && out64, "null argument");
  DAWN_CHECK(h->sh_nranks > 1 && h->sh_nranks <= kP2pMaxRanks, "init_shard (2..8 ranks) must precede shard_ipc_export");
  if (!h->p2p_own) {
    float* p = nullptr;
    DAWN_TRY(dev_alloc(h->owned, (sizeof(P2pMail) + 3) / 4, &p));
    h->p2p_own = reinterpret_cast<P2pMail*>(p);
    DAWN_TRY(dev_alloc(h->owned, 4, &p));
    h->p2p_ctr = reinterpret_cast<unsigned int*>(p);
  }
  DAWN_CUDA_OK(cudaMemset(h->p2p_own, 0, sizeof(P2pMail)));
  DAWN_CUDA_OK(cudaMemset(h->p2p_ctr, 0, 16));
  DAWN_CUDA_OK(cudaDeviceSynchronize());
  cudaIpcMemHandle_t hd;
  DAWN_CUDA_OK(cudaIpcGetMemHandle(&hd, h->p2p_own));
  static_assert(sizeof(hd) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(out64, &hd, 64);
  h->p2p_ready = false;
  return 0;
}
// ... and map every rank's mailbox (handles: nranks x 64 bytes, in rank order; the own entry is not opened).  Collective in the sense
// that every rank must have exported (and zeroed) its mailbox before any rank runs a forward: callers put a barrier after the import.
int dawn_unet_shard_ipc_import(dawn_unet* h, const char* handles) {
  DAWN_CHECK(h && handles, "null argument");
  DAWN_CHECK(h->p2p_own && h->sh_nranks > 1 && h->sh_nranks <= kP2pMaxRanks, "shard_ipc_export must precede shard_ipc_import");
  for (int r = 0; r < h->sh_nranks; ++r) {
    if (r == h->sh_rank) { h->p2p_peer[r] = h->p2p_own; continue; }
    if (h->p2p_peer[r]) { cudaIpcCloseMemHandle(h->p2p_peer[r]); h->p2p_peer[r] = nullptr; }
    cudaIpcMemHandle_t hd;
    memcpy(&hd, handles + 64 * r, 64);
    void* ptr = nullptr;
    DAWN_CUDA_OK(cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess));
    h->p2p_peer[r] = reinterpret_cast<P2pMail*>(ptr);
  }
  h->p2p_ready = true;
  drop_sampler_graph(h);
  return 0;
}

// DDIM update of this handle's frames (see sampler.cu).  Unsharded: identical to dawn_ddim_step.  Frame-sharded: the
// clip-wide quantile (U:1186-1190) is selected over ALL ranks' values by all-reducing the radix-select's histograms
// (4 x 256 u32) and its two tail statistics — 6 tiny collectives per step instead of gathering x0 (4.9 MB per rank).
static int red_sum_u32(void* ctx, unsigned int* b, size_t n, cudaStream_t st) {
  DAWN_NCCL_OK(g_nccl.AllReduce(b, b, n, kNcclUint32, kNcclSum, (ncclComm_t)ctx, st)); return 0;
}
static int red_sum_u64(void* ctx, unsigned long long* b, size_t n, cudaStream_t st) {
  DAWN_NCCL_OK(g_nccl.AllReduce(b, b, n, kNcclUint64, kNcclSum, (ncclComm_t)ctx, st)); return 0;
}
static int red_min_u32(void* ctx, unsigned int* b, size_t n, cudaStream_t st) {
  DAWN_NCCL_OK(g_nccl.AllReduce(b, b, n, kNcclUint32, kNcclMin, (ncclComm_t)ctx, st)); return 0;
}
int dawn_unet_ddim_step(dawn_unet* h, float* x, const float* eps, const float* noise, int64_t n_local, float ca, float cb,
                        float sqrt_an, float c, float sigma, float q, void* scratch, void* stream) {
  DAWN_CHECK(h, "null handle");
  if (h->sh_nranks <= 1 || !h->sh_comm)
    return ddim_step_impl(x, eps, noise, n_local, n_local, ca, cb, sqrt_an, c, sigma, q, scratch, (cudaStream_t)stream, nullptr);
  DdimReduce red{(void*)h->sh_comm, red_sum_u32, red_sum_u64, red_min_u32};
  return ddim_step_impl(x, eps, noise, n_local, n_local * h->sh_nranks, ca, cb, sqrt_an, c, sigma, q, scratch,
                        (cudaStream_t)stream, &red);
}

// The whole sampling loop of one clip as ONE CUDA graph (SURVEY 8f N2): nsteps x (forward_x3 + DDIM update), no host work
// between steps.  Everything the graph touches is fixed at capture time: x (3,F,h,w) in/out, eps scratch, noise_all
// ((nsteps-1) x n floats, step k reads slice k; the last step adds none, U:1201), t_all (nsteps int64 on the device), the
// clip-invariant tables inside the handle (refresh them with set_clip_invariants before each launch: same addresses).
// coef: host array nsteps x 5 = {ca, cb, sqrt_alpha_next, c, sigma} per step.
int dawn_unet_sampler_capture(dawn_unet* h, float* x, float* eps, const float* noise_all, const int64_t* t_all,
                              const float* coef, int nsteps, float q, void* scratch) {
  DAWN_CHECK(h && x && eps && t_all && coef && scratch && nsteps >= 1, "bad argument");
  DAWN_CHECK(noise_all || nsteps == 1, "noise_all is required for more than one step");
  DAWN_CHECK(h->F > 0 && h->have_invariants, "set_clip_invariants must precede sampler_capture");
  DAWN_CHECK(!h->prof_on, "disable profiling before capturing the sampler graph");
  drop_sampler_graph(h);
  if (!h->samp_stream) DAWN_CUDA_OK(cudaStreamCreateWithFlags(&h->samp_stream, cudaStreamNonBlocking));
  const int64_t n = (int64_t)(h->cfg.out_grid_dim + h->cfg.out_conf_dim) * h->F * h->H * h->W;
  cudaStream_t st = h->samp_stream;
  DAWN_CUDA_OK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
  int rc = 0;
  int64_t launches = 0;
  for (int k = 0; k < nsteps && rc == 0; ++k) {
    rc = dawn_unet_forward_x3(h, x, t_all + k, eps, st);
    launches += h->launches;
    const float* cf = coef + 5 * k;
    if (rc == 0)
      rc = dawn_unet_ddim_step(h, x, eps, (k < nsteps - 1) ? noise_all + (size_t)k * n : nullptr, n, cf[0], cf[1], cf[2], cf[3], cf[4],
                               q, scratch, st);
  }
  cudaGraph_t graph = nullptr;
  const cudaError_t e = cudaStreamEndCapture(st, &graph);
  if (rc != 0) { if (graph) cudaGraphDestroy(graph); return rc; }
  DAWN_CUDA_OK(e);
  const cudaError_t ei = cudaGraphInstantiate(&h->samp_exec, graph, 0);
  cudaGraphDestroy(graph);
  DAWN_CUDA_OK(ei);
  h->samp_launches = launches;
  return 0;
}

// Ancestral DDPM update of this handle's frames (reference p_sample U:1113-1121): the DDIM step's select (clip-wide when
// sharded), then the posterior update with {ca, cb, c1, c2, sigma} read from coef (device memory).
int dawn_unet_ddpm_step(dawn_unet* h, float* x, const float* eps, const float* noise, int64_t n_local, const float* coef, float q,
                        void* scratch, void* stream) {
  DAWN_CHECK(h, "null handle");
  if (h->sh_nranks <= 1 || !h->sh_comm)
    return ddpm_step_impl(x, eps, noise, n_local, n_local, coef, q, scratch, (cudaStream_t)stream, nullptr);
  DdimReduce red{(void*)h->sh_comm, red_sum_u32, red_sum_u64, red_min_u32};
  return ddpm_step_impl(x, eps, noise, n_local, n_local * h->sh_nranks, coef, q, scratch, (cudaStream_t)stream, &red);
}

// One SEGMENT of the ancestral loop (ksteps x [advance + forward_x3 + DDPM update]) as the handle's sampler graph.  The graph
// bakes no per-step value: each step first copies table row *cursor into slot and increments *cursor, the forward reads t
// from slot and the update its coefficients, so replaying the segment T / ksteps times walks the whole table.  Step j of a
// segment reads noise slice j of noise_ring (ksteps x n floats), which the caller refills before every launch.
int dawn_unet_ddpm_capture(dawn_unet* h, float* x, float* eps, const float* noise_ring, const void* table, int* cursor, void* slot,
                           int ksteps, float q, void* scratch) {
  DAWN_CHECK(h && x && eps && noise_ring && table && cursor && slot && scratch && ksteps >= 1, "bad argument");
  DAWN_CHECK(h->F > 0 && h->have_invariants, "set_clip_invariants must precede ddpm_capture");
  DAWN_CHECK(!h->prof_on, "disable profiling before capturing the sampler graph");
  drop_sampler_graph(h);
  if (!h->samp_stream) DAWN_CUDA_OK(cudaStreamCreateWithFlags(&h->samp_stream, cudaStreamNonBlocking));
  const int64_t n = (int64_t)(h->cfg.out_grid_dim + h->cfg.out_conf_dim) * h->F * h->H * h->W;
  const int64_t* t_slot = (const int64_t*)slot;
  const float* coef_slot = (const float*)slot + kDdpmCoefWord;
  cudaStream_t st = h->samp_stream;
  DAWN_CUDA_OK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
  int rc = 0;
  for (int k = 0; k < ksteps && rc == 0; ++k) {
    rc = launch_ddpm_advance(table, cursor, slot, st);
    if (rc == 0) rc = dawn_unet_forward_x3(h, x, t_slot, eps, st);
    if (rc == 0) rc = dawn_unet_ddpm_step(h, x, eps, noise_ring + (size_t)k * n, n, coef_slot, q, scratch, st);
  }
  cudaGraph_t graph = nullptr;
  const cudaError_t e = cudaStreamEndCapture(st, &graph);
  if (rc != 0) { if (graph) cudaGraphDestroy(graph); return rc; }
  DAWN_CUDA_OK(e);
  size_t nodes = 0;
  cudaGraphGetNodes(graph, nullptr, &nodes);
  const cudaError_t ei = cudaGraphInstantiate(&h->samp_exec, graph, 0);
  cudaGraphDestroy(graph);
  DAWN_CUDA_OK(ei);
  h->samp_launches = (int64_t)nodes;
  return 0;
}

int dawn_unet_sampler_launch(dawn_unet* h, void* stream) {
  DAWN_CHECK(h && h->samp_exec, "sampler_capture must precede sampler_launch (a geometry change drops the graph)");
  DAWN_CHECK(h->have_invariants, "set_clip_invariants must precede sampler_launch");
  DAWN_CUDA_OK(cudaGraphLaunch(h->samp_exec, (cudaStream_t)stream));
  h->launches = h->samp_launches;
  return 0;
}

int64_t dawn_unet_last_launch_count(dawn_unet* h) { return h ? h->launches : 0; }

int dawn_unet_profile_enable(dawn_unet* h, int on) {
  DAWN_CHECK(h, "null handle");
  h->prof_on = on != 0;
  h->prof_used = 0;
  h->prof_recs.clear();
  for (int i = 0; i < DAWN_PROF_NCAT; ++i) { h->prof_ms[i] = 0; h->prof_flops[i] = 0; h->prof_bytes[i] = 0; h->prof_cnt[i] = 0; }
  return 0;
}

int dawn_unet_profile_read(dawn_unet* h, double* ms, double* flops, double* bytes, int64_t* count) {
  DAWN_CHECK(h && ms && flops && bytes && count, "null argument");
  if (h->prof_used > 0) {
    DAWN_CUDA_OK(cudaEventSynchronize(h->prof_ev[h->prof_used - 1]));
    for (size_t i = 0; i < h->prof_recs.size(); ++i) {
      float t = 0.f;
      DAWN_CUDA_OK(cudaEventElapsedTime(&t, h->prof_ev[2 * i], h->prof_ev[2 * i + 1]));
      const auto& r = h->prof_recs[i];
      h->prof_ms[r.cat] += t; h->prof_flops[r.cat] += r.flops; h->prof_bytes[r.cat] += r.bytes; h->prof_cnt[r.cat]++;
    }
    h->prof_used = 0;
    h->prof_recs.clear();
  }
  for (int i = 0; i < DAWN_PROF_NCAT; ++i) { ms[i] = h->prof_ms[i]; flops[i] = h->prof_flops[i]; bytes[i] = h->prof_bytes[i]; count[i] = h->prof_cnt[i]; }
  return 0;
}
int64_t dawn_unet_workspace_bytes(dawn_unet* h) { return h ? h->ws_bytes : 0; }

// random qkv through both attention kernels (temporal: nseq pixel sequences of L frames, band 40 + bias;
// spatial: nseq frames of L tokens, full attention); reports max |tensor-core - SIMT|
int dawn_selftest_attention(int nseq, int L, int temporal, float* max_abs_diff, float* max_abs_ref) {
  DAWN_CHECK(max_abs_diff && max_abs_ref, "null argument");
  const size_t rows = (size_t)nseq * L;
  std::vector<float> hq(rows * 768), hb(8 * 81);
  uint32_t seed = 777u;
  auto rnd = [&]() { seed = seed * 1664525u + 1013904223u; return ((seed >> 8) & 0xFFFF) / 32768.0f - 1.0f; };
  for (auto& v : hq) v = rnd() * 1.5f;
  for (auto& v : hb) v = rnd() * 2.0f;
  std::vector<void*> own;
  float *dq, *db, *o1, *o2;
  if (dev_alloc(own, hq.size(), &dq) || dev_alloc(own, hb.size(), &db) || dev_alloc(own, rows * 256, &o1) || dev_alloc(own, rows * 256, &o2)) {
    free_all(own); return -2;
  }
  cudaMemcpy(dq, hq.data(), hq.size() * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(db, hb.data(), hb.size() * 4, cudaMemcpyHostToDevice);
  cudaMemset(o1, 0, rows * 256 * 4); cudaMemset(o2, 0, rows * 256 * 4);
  AttnArgs a{};
  a.qkv = dq; a.ld = 768; a.ldo = 256; a.nseq = nseq; a.L = L;
  if (temporal) { a.seq_base_stride = 1; a.elem_stride = nseq; a.band = 40; a.bias = db; }
  else { a.seq_base_stride = L; a.elem_stride = 1; a.band = 1 << 30; a.bias = nullptr; }
  a.q_lo = 0; a.q_hi = L;
  a.out = o1;
  int rc = launch_attention(a, 0);
  a.out = o2;
  if (rc == 0) rc = launch_attention_tc(a, 0);
  if (rc == 0 && cudaDeviceSynchronize() != cudaSuccess) { set_last_error(std::string("selftest: ") + cudaGetErrorString(cudaGetLastError())); rc = -2; }
  if (rc == 0) {
    std::vector<float> r1(rows * 256), r2(rows * 256);
    cudaMemcpy(r1.data(), o1, r1.size() * 4, cudaMemcpyDeviceToHost);
    cudaMemcpy(r2.data(), o2, r2.size() * 4, cudaMemcpyDeviceToHost);
    float md = 0.f, mr = 0.f;
    for (size_t i = 0; i < r1.size(); ++i) {
      const float d = std::fabs(r1[i] - r2[i]);
      md = (d > md || d != d) ? d : md;
      mr = std::max(mr, std::fabs(r1[i]));
    }
    *max_abs_diff = md; *max_abs_ref = mr;
  }
  free_all(own);
  return rc;
}

// random k x k conv through both contraction kernels; reports max |tcgen05 - mma.sync| over outputs and GN statistics
int dawn_selftest_tc_gemm(int F, int H, int W, int Cin, int N, int ksize, int with_stats, float* max_abs_diff, float* max_abs_ref) {
  DAWN_CHECK(max_abs_diff && max_abs_ref, "null argument");
  const int M = F * H * W, K = ksize * ksize * Cin, ldb = round_up(N, 64);
  std::vector<float> hA((size_t)M * Cin), hB((size_t)K * ldb, 0.f), hb(ldb, 0.f);
  uint32_t seed = 12345u;
  auto rnd = [&]() { seed = seed * 1664525u + 1013904223u; return ((seed >> 8) & 0xFFFF) / 32768.0f - 1.0f; };
  for (auto& v : hA) v = rnd();
  for (int k = 0; k < K; ++k) for (int n = 0; n < N; ++n) hB[(size_t)k * ldb + n] = rnd() * 0.05f;
  for (int n = 0; n < N; ++n) hb[n] = rnd();
  std::vector<float> img;
  float img_scale = 1.f;
  tc_pack_weights(hB.data(), K, N, ldb, img, &img_scale);
  std::vector<void*> own;
  float *dA, *dB, *db, *dImg, *dO1, *dO2, *dS;
  auto cleanup = [&]() { free_all(own); };
  if (dev_alloc(own, hA.size(), &dA) || dev_alloc(own, hB.size(), &dB) || dev_alloc(own, hb.size(), &db) ||
      dev_alloc(own, img.size(), &dImg) || dev_alloc(own, (size_t)M * N, &dO1) || dev_alloc(own, (size_t)M * N, &dO2) ||
      dev_alloc(own, 64, &dS)) { cleanup(); return -2; }
  cudaMemcpy(dA, hA.data(), hA.size() * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dB, hB.data(), hB.size() * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(db, hb.data(), hb.size() * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dImg, img.data(), img.size() * 4, cudaMemcpyHostToDevice);
  cudaMemset(dS, 0, 64 * 4);
  Act in{dA, Cin, Cin, H, W};
  GemmParams p; base_params(p, in, F);
  p.B = dB; p.Bimg = dImg; p.tc_scale = 1.0f / (kTcActScale * img_scale); p.ldb = ldb; p.N = N; p.K = K; p.bias = db;
  set_square_taps(p, ksize, ksize / 2);
  if (with_stats) { p.stats = (double*)dS; p.cpg = N / 8; }
  p.Out = dO1; p.ldo = N;
  int rc = launch_gemm(p, EPI_PLAIN, 0);
  if (rc == 0) {
    if (with_stats) p.stats = (double*)dS + 16;
    p.Out = dO2;
    if (!tc_gemm_supported(p, EPI_PLAIN)) { cleanup(); set_last_error("selftest: shape not supported by tc_gemm"); return -1; }
    if (getenv("DAWN_TC_SHIFT")) p.exp_shift = atoi(getenv("DAWN_TC_SHIFT"));
    unsigned long long* dT = nullptr;
    if (getenv("DAWN_TC_TRACE")) {
      float* t; if (dev_alloc(own, 64, &t)) { cleanup(); return -2; }
      cudaMemset(t, 0, 256); dT = (unsigned long long*)t; p.trace = dT;
    }
    if (getenv("DAWN_SELFTEST_CONV3") && tc_conv3_supported(p, EPI_PLAIN)) { rc = launch_tc_conv3(p, dImg, 0); printf("  (halo-tile conv3 kernel)\n"); }
    else rc = launch_tc_gemm(p, dImg, EPI_PLAIN, 0);
    if (rc == 0 && dT) {
      unsigned long long tr[16];
      cudaMemcpy(tr, dT, sizeof(tr), cudaMemcpyDeviceToHost);
      const double n = (double)std::max<unsigned long long>(tr[1], 1);
      printf("  trace (CTA 0, cycles/stage over %llu stages): total %.0f | MMA thread: wait acc_free %.0f, wait A %.0f, wait B %.0f, issue+commit %.0f | "
             "producer t0: load issue %.0f, wait slot %.0f, split+store %.0f | loader wait slot %.0f | epilogue t0: wait acc_full %.0f, drain %.0f, final epilogue %.0f "
             "(scale+bias %.0f, store %.0f)%s\n",
             tr[1], tr[0] / n, tr[2] / n, tr[3] / n, tr[4] / n, tr[5] / n, tr[11] / n, tr[6] / n, tr[7] / n, tr[8] / n, tr[9] / n, tr[12] / n, tr[10] / n,
             tr[13] / n, tr[14] / n, (p.exp_shift & 64) ? "  [stores SKIPPED]" : "");
    }
  }
  if (rc == 0 && cudaDeviceSynchronize() != cudaSuccess) { set_last_error(std::string("selftest: ") + cudaGetErrorString(cudaGetLastError())); rc = -2; }
  if (rc == 0) {
    std::vector<float> o1((size_t)M * N), o2((size_t)M * N);
    cudaMemcpy(o1.data(), dO1, o1.size() * 4, cudaMemcpyDeviceToHost);
    cudaMemcpy(o2.data(), dO2, o2.size() * 4, cudaMemcpyDeviceToHost);
    float md = 0.f, mr = 0.f;
    for (size_t i = 0; i < o1.size(); ++i) { md = std::max(md, std::fabs(o1[i] - o2[i])); mr = std::max(mr, std::fabs(o1[i])); }
    if (with_stats) {
      double st[32];
      cudaMemcpy(st, dS, sizeof(st), cudaMemcpyDeviceToHost);
      for (int i = 0; i < 16; ++i) md = std::max(md, (float)(std::fabs(st[i] - st[16 + i]) / std::max(1.0, std::fabs(st[i]))));
    }
    *max_abs_diff = md; *max_abs_ref = mr;
  }
  cleanup();
  return rc;
}

}  // extern "C"
