"""Inference-side replacement for the reference's `FlowDiffusion` consumer wrapper
(DM_3/modules/video_flow_diffusion_model_multiGPU_v0_crema_vgg_floss_plus_faceemb_flow_fast_init_cond_test.py:97-406, "FD"):
the object `unified_video_generator.py:513-531` builds and calls `update_num_frames` / `sample_one_video` on.

Same attribute names (`generator`, `unet`, `diffusion`, `face_loc_emb`), so `model.diffusion.load_state_dict(checkpoint['diffusion'])`
(UVG:527-528) and `generator.load_state_dict(checkpoint['generator'])` (FD:120) work unchanged; `sample_one_video` keeps its
signature and output dictionary.  Underneath: the source encoder, the DDIM (or ancestral DDPM) loop and the frame decoder are the CUDA paths of
this package (LfgGenerator, DynamicNfGaussianDiffusion over DynamicNfUnet3D) — one batched decode instead of a Python loop over
frames (FD:375-383).  Training-only members (region / background predictors, VGG loss, `forward`) are out of scope and absent.
"""
import ctypes

import torch
from torch import nn

from ._lib import DawnError, check, lib
from .diffusion import DynamicNfGaussianDiffusion
from .lfg import Generator
from .unet import DynamicNfUnet3D


class Face_loc_Encoder(nn.Module):
    """FD:39-50: two 3x3 stride-2 convs + ReLU on the face-box mask.  Parameters are plain nn.Conv2d holders; the arithmetic runs in
    `dawn_conv3x3_s2_relu` (one launch per layer, once per clip)."""

    def __init__(self, dim=1):
        super().__init__()
        self.conv1 = nn.Conv2d(dim, 8, kernel_size=3, stride=2, padding=1)
        self.conv2 = nn.Conv2d(8, 16, kernel_size=3, stride=2, padding=1)

    @torch.no_grad()
    def forward(self, x):
        if x.device.type != "cuda":
            raise DawnError("Face_loc_Encoder runs on CUDA (sm_100a) only; there is no CPU path")
        b, ci, H, W = x.shape
        x = x.contiguous().float()
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        outs = []
        with torch.cuda.device(x.device):
            for i in range(b):
                cur, c_in, h, w = x[i], ci, H, W
                for conv in (self.conv1, self.conv2):
                    co = conv.out_channels
                    out = torch.empty((co, (h + 1) // 2, (w + 1) // 2), device=x.device, dtype=torch.float32)
                    wgt, bias = conv.weight.detach().contiguous().float(), conv.bias.detach().contiguous().float()
                    check(lib.dawn_conv3x3_s2_relu(ctypes.c_void_p(cur.data_ptr()), c_in, h, w, ctypes.c_void_p(wgt.data_ptr()),
                                                   ctypes.c_void_p(bias.data_ptr()), co, ctypes.c_void_p(out.data_ptr()), st),
                          "dawn_conv3x3_s2_relu")
                    cur, c_in, h, w = out, co, (h + 1) // 2, (w + 1) // 2
                outs.append(cur)
        return torch.stack(outs)


class FlowDiffusion(nn.Module):
    def __init__(self, img_size=32, num_frames=40, sampling_timesteps=250, win_width=40, null_cond_prob=0.1, ddim_sampling_eta=1.,
                 pose_dim=7, dim_mults=(1, 2, 4, 8), is_train=False, use_residual_flow=False, learn_null_cond=False, use_deconv=True,
                 padding_mode="zeros", pretrained_pth=None, config_pth=None, generator_params=None):
        """Keywords as FD:98-108.  The reference reads the LFG architecture from `config_pth` (yaml) and its weights from
        `pretrained_pth`; both stay optional here (`generator_params` may be given directly, weights loaded later)."""
        super().__init__()
        if is_train:
            # config/DAWN_128.yaml / DAWN_256.yaml ship is_train: true and UVG:516 passes it straight through; in the reference it only
            # calls .train() on unet/diffusion (FD:171-175) and UVG calls model.eval() right after.  Accept it, stay in eval mode;
            # the training entry points (forward / p_losses) raise.
            import warnings
            warnings.warn("FlowDiffusion(is_train=True): the B200 wrapper is inference-only and stays in eval mode")
        self.use_residual_flow = use_residual_flow
        if generator_params is None:
            if config_pth is not None:
                import yaml
                with open(config_pth) as f:
                    mp = yaml.safe_load(f)['model_params']
                generator_params = dict(num_regions=mp['num_regions'], num_channels=mp['num_channels'],
                                        revert_axis_swap=mp['revert_axis_swap'], **mp['generator_params'])
            else:                                                   # config/hdtf128.yaml == config/hdtf256.yaml generator_params
                generator_params = dict(num_regions=10, num_channels=3, revert_axis_swap=True, block_expansion=64, max_features=512,
                                        num_down_blocks=2, num_bottleneck_blocks=6, skips=True, pixelwise_flow_predictor_params=None)
        self.generator = Generator(**generator_params)                                             # FD:116-121
        if pretrained_pth is not None:
            self.generator.load_state_dict(torch.load(pretrained_pth, map_location="cpu")['generator'])
        self.pose_dim = pose_dim
        self.unet = DynamicNfUnet3D(dim=64, cond_dim=1024 + pose_dim + 2, cond_aud=1024, cond_pose=pose_dim, cond_eye=2,
                                    num_frames=num_frames, channels=3 + 256 + 16, out_grid_dim=2, out_conf_dim=1, dim_mults=dim_mults,
                                    use_hubert_audio_cond=True, learn_null_cond=learn_null_cond, use_final_activation=False,
                                    use_deconv=use_deconv, padding_mode=padding_mode, win_width=win_width)     # FD:140-155
        self.diffusion = DynamicNfGaussianDiffusion(denoise_fn=self.unet, num_frames=num_frames, image_size=img_size,
                                                    sampling_timesteps=sampling_timesteps, timesteps=1000, loss_type='l2',
                                                    use_dynamic_thres=True, null_cond_prob=null_cond_prob,
                                                    ddim_sampling_eta=ddim_sampling_eta)                      # FD:157-167
        self.face_loc_emb = Face_loc_Encoder()                                                                # FD:169
        self.is_train = False
        self.eval()

    def update_num_frames(self, new_num_frames):                                                              # FD:177-180
        self.unet.update_num_frames(new_num_frames)
        self.diffusion.update_num_frames(new_num_frames)

    @staticmethod
    def generate_bbox_mask(bbox, size=32):
        """FD:182-201.  bbox (b, c >= 6, frames): columns [x0, x1, y0, y1, image_w, image_h] of the FIRST frame -> (b, 1, size, size)
        mask of the face box.  Index arithmetic on a handful of integers (torch ops on the caller's device); like the reference
        it compares uint8 row/column indices against int32 box corners (sizes above 255 wrap in the reference too)."""
        b = bbox.shape[0]
        bbox = bbox[:, :, 0].clone().float()
        bbox[:, :2] = (bbox[:, :2] / bbox[:, 4].unsqueeze(1)) * size
        bbox[:, 2:4] = (bbox[:, 2:4] / bbox[:, 5].unsqueeze(1)) * size
        lt = bbox[:, :4:2].to(torch.int32)
        rb = (bbox[:, 1:4:2] + 1).to(torch.int32)
        dev = bbox.device
        rows = torch.arange(size, device=dev).view(1, size, 1).expand(b, size, size).to(torch.uint8)
        cols = torch.arange(size, device=dev).view(1, 1, size).expand(b, size, size).to(torch.uint8)
        mask = (rows >= lt[:, 1].view(b, 1, 1)) & (rows <= rb[:, 1].view(b, 1, 1)) & \
               (cols >= lt[:, 0].view(b, 1, 1)) & (cols <= rb[:, 0].view(b, 1, 1))
        return mask.unsqueeze(1).float()

    @torch.no_grad()
    def sample_one_video(self, sample_img, sample_audio_hubert, sample_pose, sample_eye, sample_bbox, cond_scale, init_pose=None,
                         init_eye=None, real_vid=None, noise_fn=None, use_graph=False):
        """FD:325-406.  sample_img (b, 3, H, W) in [0, 1]; sample_audio_hubert (b, F, 1024); sample_pose (b, >= pose_dim, F);
        sample_eye (b, 2, F); sample_bbox (b, >= 6, F).  Returns the reference's dictionary: sample_vid_grid (b, 2, F, h, w),
        sample_vid_conf (b, 1, F, h, w), sample_out_vid (b, 3, F, H, W), sample_warped_vid (b, 3, F, H, W).
        noise_fn / use_graph are passed to the sampler (tests inject the noise the reference draws with torch.randn)."""
        out = {}
        fea = self.generator.compute_fea(sample_img)                                    # FD:327
        bbox_mask = self.generate_bbox_mask(sample_bbox, size=sample_img.shape[-1])     # FD:328
        bbox_mask = self.face_loc_emb(bbox_mask)                                        # FD:330
        sample_pose = sample_pose[:, :self.pose_dim]
        ref_pose = sample_pose.permute(0, 2, 1)
        ref_eye = sample_eye.permute(0, 2, 1)
        nf = ref_pose.shape[1]
        init_pose = (ref_pose[:, 0] if init_pose is None else init_pose).unsqueeze(1).repeat(1, nf, 1)[:, :, :self.pose_dim]
        init_eye = (ref_eye[:, 0] if init_eye is None else init_eye).unsqueeze(1).repeat(1, nf, 1)
        if ref_pose.shape[-1] != init_pose.shape[-1]:
            ref_pose = torch.cat([ref_pose, init_pose[:, :, -1].unsqueeze(-1)], dim=-1)
        ref_text = torch.cat([sample_audio_hubert, ref_pose - init_pose, ref_eye - init_eye], dim=-1)          # FD:350
        b = fea.shape[0]
        fea272 = torch.cat([fea, bbox_mask], dim=1)                                     # GaussianDiffusion.sample, U:1151
        h, w = fea272.shape[-2:]
        # DDIM when sampling_timesteps < timesteps, else the ancestral loop, as the reference's sample() picks (U:1150)
        sample_fn = self.diffusion.ddim_sample if self.diffusion.is_ddim_sampling else self.diffusion.p_sample_loop
        pred = sample_fn(fea272, (b, self.diffusion.channels, self.diffusion.num_frames, h, w), cond=ref_text,
                         cond_scale=cond_scale, noise_fn=noise_fn, use_graph=use_graph)
        if self.use_residual_flow:
            raise NotImplementedError("use_residual_flow=True is not used by the shipped configs (FD:362-364)")
        out["sample_vid_grid"] = pred[:, :2]                                            # FD:366
        out["sample_vid_conf"] = (pred[:, 2].unsqueeze(1) + 1) * 0.5                    # FD:369
        vids, warped = [], []
        for i in range(b):                                                              # FD:375-383, all frames of a clip at once
            p, d = self.generator.decode_sample(sample_img[i:i + 1], pred[i], need_deformed=True)
            vids.append(p.permute(1, 0, 2, 3))
            warped.append(d.permute(1, 0, 2, 3))
        out["sample_out_vid"] = torch.stack(vids)
        out["sample_warped_vid"] = torch.stack(warped)
        return out

    def forward(self, *a, **k):
        raise NotImplementedError("FlowDiffusion.forward is the training step (FD:203-323): out of scope of the B200 inference path")
