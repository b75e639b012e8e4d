"""Drop-in replacement for the reference's `Unet3D` / `DynamicNfUnet3D`
(DM_3/modules/video_flow_diffusion_multiGPU_v0_crema_plus_faceemb_ca_multi_test.py:728-965).

Same constructor keywords, `forward`, `forward_with_cond_scale`, `update_num_frames`, `null_cond_mask`,
`has_cond`, and a state_dict whose 900 keys/shapes equal the reference's (SURVEY Appendix B), so
`diffusion.load_state_dict(checkpoint['diffusion'])` (unified_video_generator.py:527-528) works unchanged.
The sub-modules below only HOLD parameters (names, shapes, default initialisers); all arithmetic runs in
hand-written sm_100a CUDA kernels behind the C-ABI in include/dawn_unet.h.  There is no PyTorch fallback.
"""
import ctypes
import os
import math

import torch
from torch import nn

from . import _lib
from ._lib import DawnUnetCfg, check, lib


# ----------------------------------------------------------------------------- parameter holders
class _Holder(nn.Module):
    """Container whose forward is never called."""

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("parameter holder: the computation runs in the CUDA library")


class _Gain(_Holder):
    def __init__(self, name, shape):
        super().__init__()
        self.register_parameter(name, nn.Parameter(torch.ones(shape)))


class _Rotary(_Holder):
    """rotary-embedding-torch 0.3.5 registers `freqs` as a non-trainable Parameter (reference :761)."""

    def __init__(self, dim, theta=10000):
        super().__init__()
        freqs = 1. / (theta ** (torch.arange(0, dim, 2)[:(dim // 2)].float() / dim))
        self.freqs = nn.Parameter(freqs, requires_grad=False)


def _cross_attn(dim, out_dim, context_dim, dim_head=8, heads=8):           # reference :481-514
    m = _Holder()
    inner = dim_head * heads
    m.norm = _Gain('g', (dim,))
    m.null_kv = nn.Parameter(torch.randn(2, dim_head))
    m.to_q = nn.Linear(dim, inner, bias=False)
    m.to_kv = nn.Linear(context_dim, inner * 2, bias=False)
    m.q_scale = nn.Parameter(torch.ones(dim_head))
    m.k_scale = nn.Parameter(torch.ones(dim_head))
    m.to_out = nn.Sequential(nn.Linear(inner, out_dim, bias=False), _Gain('g', (out_dim,)))
    return m


def _block(dim, dim_out, groups):                                           # reference :226-231
    m = _Holder()
    m.proj = nn.Conv3d(dim, dim_out, (1, 3, 3), padding=(0, 1, 1))
    m.norm = nn.GroupNorm(groups, dim_out)
    return m


def _resnet_block(dim, dim_out, groups, time_dim=None, aud=None, pose=None, eye=None):   # reference :363-417
    m = _Holder()
    if time_dim is not None:
        m.time_mlp = nn.Sequential(nn.SiLU(), nn.Linear(time_dim, dim_out * 2))
    if aud is not None:
        m.audio_mlp = nn.Sequential(nn.SiLU(), nn.Linear(aud, dim_out * 2))
    if pose is not None:
        m.pose_mlp = nn.Sequential(nn.SiLU(), nn.Linear(pose, dim_out * 2))
    if eye is not None:
        m.eye_mlp = nn.Sequential(nn.SiLU(), nn.Linear(eye, dim_out * 2))
    m.cross_attn_aud = _cross_attn(dim, dim_out, dim_out * 2)
    m.cross_attn_pose = _cross_attn(dim, dim_out, dim_out * 2)
    m.cross_attn_eye = _cross_attn(dim, dim_out, dim_out * 2)
    m.block1 = _block(dim, dim_out, groups)
    m.block2 = _block(dim_out, dim_out, groups)
    if dim != dim_out:
        m.res_conv = nn.Conv3d(dim, dim_out, 1)
    return m


def _prenorm_residual(dim, fn):                                             # Residual(PreNorm(dim, fn)) :141-147, 205-213
    pre = _Holder()
    pre.fn = fn
    pre.norm = _Gain('gamma', (1, dim, 1, 1, 1))
    res = _Holder()
    res.fn = pre
    return res


def _attention(dim, heads, dim_head, rotary=None):                          # reference :648-663
    m = _Holder()
    hidden = heads * dim_head
    if rotary is not None:
        m.rotary_emb = rotary
    m.to_qkv = nn.Linear(dim, hidden * 3, bias=False)
    m.to_out = nn.Linear(hidden, dim, bias=False)
    return m


def _einops_wrapped(fn):                                                    # EinopsToAndFrom :632-645
    m = _Holder()
    m.fn = fn
    return m


def _spatial_linear_attention(dim, heads, dim_head=32):                     # reference :602-609
    m = _Holder()
    hidden = heads * dim_head
    m.to_qkv = nn.Conv2d(dim, hidden * 3, 1, bias=False)
    m.to_out = nn.Conv2d(hidden, dim, 1)
    return m


def _rel_bias_table(weight, window, num_buckets=32, max_distance=32):
    """RelativePositionBias values for rel = j - i in [-window, window] (reference :91-119), evaluated with
    the same torch CPU ops as the reference so that the log-spaced bucket edges land identically."""
    rel = torch.arange(-window, window + 1, dtype=torch.long)
    n = -rel
    nb = num_buckets // 2
    bucket = (n < 0).long() * nb
    n = n.abs()
    max_exact = nb // 2
    large = max_exact + (torch.log(n.float() / max_exact) / math.log(max_distance / max_exact)
                         * (nb - max_exact)).long()
    large = torch.min(large, torch.full_like(large, nb - 1))
    bucket = bucket + torch.where(n < max_exact, n, large)
    return weight.detach().float().cpu()[bucket].t().contiguous()           # (heads, 2w+1)


def _time_freqs(dim):
    half = dim // 2                                                         # reference :157-159
    emb = math.log(10000) / (half - 1)
    return torch.exp(torch.arange(half) * -emb).float().contiguous()


# ----------------------------------------------------------------------------- the module
class Unet3D(nn.Module):
    def __init__(self, dim, cond_aud=1024, cond_pose=7, cond_eye=2, cond_dim=None, out_grid_dim=2, out_conf_dim=1,
                 num_frames=40, dim_mults=(1, 2, 4, 8), channels=3, attn_heads=8, attn_dim_head=32,
                 use_hubert_audio_cond=False, init_dim=None, init_kernel_size=7, use_sparse_linear_attn=True,
                 resnet_groups=8, use_final_activation=False, learn_null_cond=False, use_deconv=True,
                 padding_mode="zeros", win_width=20):
        super().__init__()
        if init_dim is not None and init_dim != dim:
            raise NotImplementedError("init_dim != dim is not supported by the CUDA library")
        if not use_sparse_linear_attn or not use_deconv or padding_mode != "zeros" or use_final_activation or learn_null_cond:
            raise NotImplementedError("only the configuration DAWN ships is supported: use_sparse_linear_attn=True, "
                                      "use_deconv=True, padding_mode='zeros', use_final_activation=False, learn_null_cond=False")
        self.null_cond_mask = None
        self.null_cond_emb = None
        self.channels = channels
        self.num_frames = num_frames
        self.HUBERT_MODEL_DIM = 1024
        self.has_cond = (cond_dim is not None) or use_hubert_audio_cond
        self.cond_dim = cond_dim
        self.cond_aud_dim, self.cond_pose_dim, self.cond_eye_dim = cond_aud, cond_pose, cond_eye
        self.learn_null_cond = learn_null_cond
        self.use_final_activation = use_final_activation
        self.win_width = win_width
        self.dim = dim
        self.out_dim = out_grid_dim + out_conf_dim
        if cond_dim is not None and cond_dim != cond_aud + cond_pose + cond_eye:
            raise ValueError("cond_dim must equal cond_aud + cond_pose + cond_eye")

        rotary = _Rotary(min(32, attn_dim_head))

        def temporal(d):
            return _einops_wrapped(_attention(d, attn_heads, attn_dim_head, rotary))

        rpb = _Holder()
        rpb.relative_attention_bias = nn.Embedding(32, attn_heads)
        self.time_rel_pos_bias = rpb
        pad = init_kernel_size // 2
        self.init_conv = nn.Conv3d(channels, dim, (1, init_kernel_size, init_kernel_size), padding=(0, pad, pad))
        self.init_temporal_attn = _prenorm_residual(dim, temporal(dim))
        dims = [dim, *[dim * m for m in dim_mults]]
        in_out = list(zip(dims[:-1], dims[1:]))
        time_dim = dim * 4
        self.time_mlp = nn.Sequential(_Holder(), nn.Linear(dim, time_dim), nn.GELU(), nn.Linear(time_dim, time_dim))

        def cond_block(a, b):
            return _resnet_block(a, b, resnet_groups, time_dim, cond_aud, cond_pose, cond_eye)

        self.downs = nn.ModuleList([])
        self.ups = nn.ModuleList([])
        n_res = len(in_out)
        for ind, (di, do) in enumerate(in_out):
            last = ind >= n_res - 1
            self.downs.append(nn.ModuleList([
                cond_block(di, do), cond_block(do, do),
                _prenorm_residual(do, _spatial_linear_attention(do, attn_heads)),
                _prenorm_residual(do, temporal(do)),
                nn.Conv3d(do, do, (1, 4, 4), (1, 2, 2), (0, 1, 1)) if not last else nn.Identity()]))
        mid = dims[-1]
        self.mid_block1 = cond_block(mid, mid)
        self.mid_spatial_attn = _prenorm_residual(mid, _einops_wrapped(_attention(mid, attn_heads, 32)))
        self.mid_temporal_attn = _prenorm_residual(mid, temporal(mid))
        self.mid_block2 = cond_block(mid, mid)
        for ind, (di, do) in enumerate(reversed(in_out)):
            last = ind >= n_res - 1
            self.ups.append(nn.ModuleList([
                cond_block(do * 2, di), cond_block(di, di),
                _prenorm_residual(di, _spatial_linear_attention(di, attn_heads)),
                _prenorm_residual(di, temporal(di)),
                nn.ConvTranspose3d(di, di, (1, 4, 4), (1, 2, 2), (0, 1, 1)) if not last else nn.Identity()]))
        self.final_conv = nn.Sequential(_resnet_block(dim * 2, dim, resnet_groups), nn.Conv3d(dim, out_grid_dim, 1))
        self.final_activation = nn.Identity()
        self.occlusion_map = nn.Sequential(_resnet_block(dim * 2, dim, resnet_groups), nn.Conv3d(dim, out_conf_dim, 1))

        cfg = DawnUnetCfg()
        cfg.dim, cfg.n_levels = dim, len(dim_mults)
        for i, m in enumerate(dim_mults):
            cfg.dim_mults[i] = m
        cfg.channels, cfg.cond_aud, cfg.cond_pose, cfg.cond_eye = channels, cond_aud, cond_pose, cond_eye
        cfg.out_grid_dim, cfg.out_conf_dim = out_grid_dim, out_conf_dim
        cfg.attn_heads, cfg.attn_dim_head, cfg.resnet_groups = attn_heads, attn_dim_head, resnet_groups
        cfg.init_kernel_size, cfg.win_width = init_kernel_size, win_width
        self._cfg = cfg
        self._handle = None
        self._dirty = True
        self._geom = None
        self._device_index = None
        self.register_load_state_dict_post_hook(lambda module, incompatible: module.mark_dirty())

    # ------------------------------------------------------------------ native handle management
    def mark_dirty(self):
        """Call after mutating parameters in place; load_state_dict / .to() / .cuda() do it automatically."""
        self._dirty = True

    def _apply(self, fn, *a, **k):
        self._dirty = True
        return super()._apply(fn, *a, **k)

    def __del__(self):
        # plain dict access: nn.Module.__setattr__/__getattr__ may already be torn down at interpreter shutdown
        h = self.__dict__.get("_handle")
        self.__dict__["_handle"] = None
        if h is not None:
            try:
                lib.dawn_unet_destroy(h)
            except Exception:
                pass

    def _ensure(self, device, F, h, w):
        if device.type != "cuda":
            raise _lib.DawnError("the DAWN denoising UNet runs on CUDA (sm_100a) only; there is no CPU path")
        idx = device.index if device.index is not None else torch.cuda.current_device()
        if self._handle is not None and self._device_index != idx:
            lib.dawn_unet_destroy(self._handle)
            self._handle, self._dirty, self._geom = None, True, None
        with torch.cuda.device(idx):
            if self._handle is None:
                hd = ctypes.c_void_p()
                check(lib.dawn_unet_create(ctypes.byref(self._cfg), ctypes.byref(hd)), "dawn_unet_create")
                self._handle, self._device_index = hd, idx
            if self._dirty:
                self.sync_parameters()
            if self._geom != (F, h, w):
                check(lib.dawn_unet_set_num_frames(self._handle, F, h, w), "dawn_unet_set_num_frames")
                self._geom = (F, h, w)
                self._gen = getattr(self, "_gen", 0) + 1
            lost = getattr(self, "_shard_lost", None)
            if lost is not None and not getattr(self, "_in_init_shard", False):
                raise _lib.DawnError(f"frame sharding (rank {lost[0]} of {lost[1]}) was dropped by a parameter re-commit "
                                "(.to()/.cuda()/load_state_dict after init_shard): call init_shard again on every rank")

    def sync_parameters(self):
        """Repack the module's parameters into kernel layouts (once per parameter change)."""
        def put(name, t):
            t = t.detach().to(device="cpu", dtype=torch.float32).contiguous()
            shape = (ctypes.c_int64 * max(t.dim(), 1))(*t.shape)
            check(lib.dawn_unet_set_param(self._handle, name.encode(), ctypes.c_void_p(t.data_ptr()), shape, t.dim()),
                  f"dawn_unet_set_param({name})")
        for name, t in self.state_dict().items():
            put(name, t)
        put("aux.time_freqs", _time_freqs(self.dim))
        put("aux.rel_bias", _rel_bias_table(self.time_rel_pos_bias.relative_attention_bias.weight, self.win_width))
        check(lib.dawn_unet_commit_params(self._handle), "dawn_unet_commit_params")
        self._dirty = False
        self._gen = getattr(self, "_gen", 0) + 1
        # commit re-runs set_num_frames in the library, which leaves the handle unsharded: running on would silently drop the
        # temporal halos, the clip-wide GroupNorm statistics and the clip-wide quantile, so the next use raises instead
        if getattr(self, "_shard", None) is not None:
            self._shard_lost = self._shard
        self._shard = None
        if self._geom is not None:
            self._geom = self._geom  # commit re-sized the per-clip tables for the current geometry

    @staticmethod
    def _stream():
        return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    # ------------------------------------------------------------------ reference API
    def forward_with_cond_scale(self, *args, cond_scale=2., **kwargs):      # reference :879-890
        logits = self.forward(*args, null_cond_prob=0., **kwargs)
        if cond_scale == 1 or not self.has_cond:
            return logits
        null_logits = self.forward(*args, null_cond_prob=1., **kwargs)
        return null_logits + (logits - null_logits) * cond_scale

    def forward(self, x, time, cond=None, null_cond_prob=0., focus_present_mask=None, prob_focus_present=0.):
        """reference :892-956.  x (b, channels, F, h, w) fp32; time (b,) int64; cond (b, F, cond_dim)."""
        assert not (self.has_cond and cond is None), 'cond must be passed in if cond_dim specified'
        if focus_present_mask is not None and bool(focus_present_mask.any()) or prob_focus_present != 0:
            raise NotImplementedError("focus_present_mask (training-time arrested attention) is not supported")
        b, ch, F, h, w = x.shape
        if ch != self.channels:
            raise ValueError(f"expected {self.channels} input channels, got {ch}")
        if self.has_cond and (cond.shape[1] != self.num_frames or F != self.num_frames):
            raise ValueError(f"num_frames={self.num_frames} but x has {F} frames and cond {cond.shape[1]}: "
                             "call update_num_frames first (reference :925-926)")
        device = x.device
        self._ensure(device, F, h, w)
        x = x.contiguous().float()
        time = time.to(device=device, dtype=torch.int64).contiguous()
        # classifier-free guidance plumbing (reference :917-926); learn_null_cond=False -> zeros
        self.null_cond_emb = torch.zeros(1, self.num_frames, self.cond_dim or 0) if self.has_cond else None
        if null_cond_prob == 1:
            self.null_cond_mask = torch.ones((b, self.num_frames), device=device, dtype=torch.bool)
        elif null_cond_prob == 0:
            self.null_cond_mask = torch.zeros((b, self.num_frames), device=device, dtype=torch.bool)
        else:
            self.null_cond_mask = torch.zeros((b, self.num_frames), device=device).float().uniform_(0, 1) < null_cond_prob
        cond = cond.to(device=device, dtype=torch.float32)
        if null_cond_prob != 0:
            cond = torch.where(self.null_cond_mask[..., None], torch.zeros((), device=device), cond)
        cond = cond.contiguous()
        out = torch.empty((b, self.out_dim, F, h, w), device=device, dtype=torch.float32)
        st = self._stream()
        with torch.cuda.device(device):
            for i in range(b):
                check(lib.dawn_unet_forward(self._handle, ctypes.c_void_p(x[i].data_ptr()),
                                            ctypes.c_void_p(time[i:i + 1].data_ptr()),
                                            ctypes.c_void_p(cond[i].data_ptr()),
                                            ctypes.c_void_p(out[i].data_ptr()), st), "dawn_unet_forward")
        return out

    # ------------------------------------------------------------------ fast path used by our sampler
    def set_clip_invariants(self, fea, cond):
        """fea (channels-3, h, w) and cond (F, cond_dim) of ONE clip: everything that is constant over the
        DDIM steps (272 of the 275 init-conv input channels, all cross-attention keys/values)."""
        if fea.dim() != 3 or cond.dim() != 2:
            raise ValueError(f"set_clip_invariants: fea must be (channels-3, h, w) and cond (F, cond_dim); got {tuple(fea.shape)}, {tuple(cond.shape)}")
        F, (h, w) = cond.shape[0], fea.shape[-2:]
        if fea.shape[0] != self.channels - 3 or cond.shape[1] != (self.cond_dim or 0):
            raise ValueError(f"set_clip_invariants: expected fea with {self.channels - 3} channels and cond with {self.cond_dim} "
                             f"features; got {tuple(fea.shape)}, {tuple(cond.shape)}")
        if F != self.num_frames:
            raise ValueError(f"num_frames={self.num_frames} but cond has {F} frames: call update_num_frames first (reference :925-926)")
        if not fea.is_cuda or cond.device != fea.device:
            raise _lib.DawnError("set_clip_invariants needs CUDA tensors on one device (no CPU fallback)")
        self._ensure(fea.device, F, h, w)
        self._fea = fea.contiguous().float()
        self._cond = cond.contiguous().float()
        with torch.cuda.device(fea.device):
            check(lib.dawn_unet_set_clip_invariants(self._handle, ctypes.c_void_p(self._fea.data_ptr()),
                                                    ctypes.c_void_p(self._cond.data_ptr()), self._stream()),
                  "dawn_unet_set_clip_invariants")

    def init_shard(self, F_local, h, w, device):
        """Exact frame sharding over the default torch.distributed group: this rank owns global frames
        [rank*F_local, (rank+1)*F_local).  Creates the library's own NCCL communicator (unique id broadcast through
        torch.distributed) and switches the handle to sharded mode for this geometry."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(), dist.get_rank()
        self._shard_lost = None
        self._in_init_shard = True
        try:
            self._ensure(device, F_local, h, w)
        finally:
            self._in_init_shard = False
        buf = ctypes.create_string_buffer(128)
        if rank == 0:
            check(lib.dawn_nccl_unique_id(buf), "dawn_nccl_unique_id")
        box = [bytes(buf.raw)]
        dist.broadcast_object_list(box, src=0)
        with torch.cuda.device(device):
            check(lib.dawn_unet_init_shard(self._handle, box[0], world, rank, F_local * world), "dawn_unet_init_shard")
        # GroupNorm all-reduces over NVLink peer memory (cudaIpc mailboxes) when all ranks sit on one node; DAWN_P2P=0 keeps NCCL
        if 2 <= world <= 8 and os.environ.get("DAWN_P2P", "1") != "0":
            hbuf = ctypes.create_string_buffer(64)
            with torch.cuda.device(device):
                check(lib.dawn_unet_shard_ipc_export(self._handle, hbuf), "dawn_unet_shard_ipc_export")
            allh = [None] * world
            dist.all_gather_object(allh, bytes(hbuf.raw))
            with torch.cuda.device(device):
                check(lib.dawn_unet_shard_ipc_import(self._handle, b"".join(allh)), "dawn_unet_shard_ipc_import")
            dist.barrier()
        self._shard = (rank, world, (F_local, h, w))
        self._gen = getattr(self, "_gen", 0) + 1

    def shard_info(self):
        """(rank, world) of the frame sharding in force for the current geometry; (0, 1) when unsharded."""
        sh = getattr(self, "_shard", None)
        if sh is None or sh[2] != self._geom:
            return 0, 1
        return sh[0], sh[1]

    def graph_generation(self):
        """Changes whenever the native handle dropped a captured sampler graph (new geometry, parameters or sharding)."""
        return (id(self._handle), getattr(self, "_gen", 0))

    def claim_graph_slot(self):
        """Call before capturing a sampler graph: the handle holds ONE (DDIM loop or DDPM segment), so a new capture invalidates
        whatever graph another sampler cached against the previous generation."""
        self._gen = getattr(self, "_gen", 0) + 1

    def forward_x3(self, x_t, time, out=None):
        """x_t (3, F, h, w) of the clip whose invariants were set; time int64 tensor (1,) on the device."""
        if self._geom is None or getattr(self, "_fea", None) is None:
            raise _lib.DawnError("forward_x3: call set_clip_invariants first")
        if tuple(x_t.shape) != (3,) + tuple(self._geom) or x_t.dtype != torch.float32 or x_t.device != self._fea.device:
            raise ValueError(f"forward_x3: x_t must be float32 (3, {self._geom[0]}, {self._geom[1]}, {self._geom[2]}) on "
                             f"{self._fea.device}; got {x_t.dtype} {tuple(x_t.shape)} on {x_t.device}")
        _, F, h, w = x_t.shape
        if out is None:
            out = torch.empty((self.out_dim, F, h, w), device=x_t.device, dtype=torch.float32)
        elif tuple(out.shape) != (self.out_dim, F, h, w) or out.dtype != torch.float32 or not out.is_contiguous() or out.device != x_t.device:
            raise ValueError(f"forward_x3: out must be contiguous float32 ({self.out_dim}, {F}, {h}, {w}) on {x_t.device}")
        x_t = x_t.contiguous()
        with torch.cuda.device(x_t.device):
            check(lib.dawn_unet_forward_x3(self._handle, ctypes.c_void_p(x_t.data_ptr()), ctypes.c_void_p(time.data_ptr()),
                                           ctypes.c_void_p(out.data_ptr()), self._stream()), "dawn_unet_forward_x3")
        return out

    def forward_host(self, x_t, fea, cond, t, out=None):
        """End-to-end step with HOST tensors (pinned recommended): H2D of x_t/fea/cond, compute, D2H of eps."""
        _, F, h, w = x_t.shape
        self._ensure(torch.device("cuda", torch.cuda.current_device()), F, h, w)
        if out is None:
            out = torch.empty((self.out_dim, F, h, w), dtype=torch.float32, pin_memory=True)
        check(lib.dawn_unet_forward_host(self._handle, ctypes.c_void_p(x_t.data_ptr()), ctypes.c_void_p(fea.data_ptr()),
                                         ctypes.c_void_p(cond.data_ptr()), int(t), ctypes.c_void_p(out.data_ptr())),
              "dawn_unet_forward_host")
        return out

    # ------------------------------------------------------------------ debugging taps (sub-module parity tests)
    def request_taps(self, names, F, h, w, device):
        self._ensure(device, F, h, w)
        bufs = {}
        for n in names:
            C, hl, wl = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
            check(lib.dawn_unet_tap_shape(self._handle, n.encode(), ctypes.byref(C), ctypes.byref(hl), ctypes.byref(wl)),
                  f"dawn_unet_tap_shape({n})")
            t = torch.zeros((1, C.value, F, hl.value, wl.value), device=device, dtype=torch.float32)
            check(lib.dawn_unet_set_tap(self._handle, n.encode(), ctypes.c_void_p(t.data_ptr())), "dawn_unet_set_tap")
            bufs[n] = t
        self._tap_bufs = bufs
        return bufs

    def clear_taps(self):
        for n in getattr(self, "_tap_bufs", {}):
            lib.dawn_unet_set_tap(self._handle, n.encode(), None)
        self._tap_bufs = {}

    def profile(self, on=True):
        check(lib.dawn_unet_profile_enable(self._handle, 1 if on else 0), "dawn_unet_profile_enable")

    def profile_read(self):
        """{category: dict(ms, flops, bytes, count)} accumulated since profile(True)."""
        n = _lib.PROF_NCAT
        ms, fl, by = (ctypes.c_double * n)(), (ctypes.c_double * n)(), (ctypes.c_double * n)()
        cnt = (ctypes.c_int64 * n)()
        check(lib.dawn_unet_profile_read(self._handle, ms, fl, by, cnt), "dawn_unet_profile_read")
        return {c: dict(ms=ms[i], flops=fl[i], bytes=by[i], count=int(cnt[i])) for i, c in enumerate(_lib.PROF_CATS)}

    def last_launch_count(self):
        return int(lib.dawn_unet_last_launch_count(self._handle)) if self._handle is not None else 0

    def workspace_bytes(self):
        return int(lib.dawn_unet_workspace_bytes(self._handle)) if self._handle is not None else 0


class DynamicNfUnet3D(Unet3D):
    """reference :959-965 — num_frames can be changed after construction."""

    def __init__(self, default_num_frames=20, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.default_num_frames = default_num_frames
        self.num_frames = default_num_frames

    def update_num_frames(self, new_num_frames):
        self.num_frames = new_num_frames
