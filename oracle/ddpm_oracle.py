"""Restatement of the reference's ancestral DDPM step (DM_3/modules/video_flow_diffusion_multiGPU_v0_crema_plus_faceemb_ca_multi_test.py,
"U"): predict_start_from_noise U:1072-1076, the clip-denoised x0 of p_mean_variance U:1094-1107, q_posterior U:1078-1085 and the
noise term of p_sample U:1113-1121.  Plain torch on the CPU; the schedule buffers are built exactly as GaussianDiffusion.__init__
builds them (fp64, then registered as fp32, U:1012-1055)."""
import torch
import torch.nn.functional as F


def posterior_buffers(timesteps=1000, s=0.008):
    """U:975-985 + U:1012-1055: {name: fp32 buffer} of the five tables one ancestral step reads."""
    steps = timesteps + 1
    x = torch.linspace(0, timesteps, steps, dtype=torch.float64)
    ac = torch.cos(((x / timesteps) + s) / (1 + s) * torch.pi * 0.5) ** 2
    ac = ac / ac[0]
    betas = torch.clip(1 - (ac[1:] / ac[:-1]), 0, 0.9999)
    alphas = 1. - betas
    acp = torch.cumprod(alphas, dim=0)
    prev = F.pad(acp[:-1], (1, 0), value=1.)
    pv = betas * (1. - prev) / (1. - acp)
    bufs = dict(sqrt_recip_alphas_cumprod=torch.sqrt(1. / acp), sqrt_recipm1_alphas_cumprod=torch.sqrt(1. / acp - 1),
                posterior_mean_coef1=betas * torch.sqrt(prev) / (1. - acp),
                posterior_mean_coef2=(1. - prev) * torch.sqrt(alphas) / (1. - acp),
                posterior_log_variance_clipped=torch.log(pv.clamp(min=1e-20)))
    return {k: v.to(torch.float32) for k, v in bufs.items()}


def ddpm_step(eps, img, t, noise, timesteps=1000, dynamic_thres=True, pct=0.9):
    """One p_sample update (clip_denoised=True) of img (b, ...) given the UNet's eps prediction at time index t (int).
    noise: the tensor the reference draws with randn_like (it is drawn and masked even at t = 0, U:1118-1121)."""
    B = posterior_buffers(timesteps)
    x0 = B['sqrt_recip_alphas_cumprod'][t] * img - B['sqrt_recipm1_alphas_cumprod'][t] * eps                # U:1072-1076
    s = torch.ones(x0.shape[0])
    if dynamic_thres:                                                                                        # U:1096-1104
        s = torch.quantile(x0.reshape(x0.shape[0], -1).abs(), pct, dim=-1).clamp(min=1.)
    s = s.view(-1, *((1,) * (x0.ndim - 1)))
    x0 = x0.clamp(-s, s) / s                                                                                 # U:1107
    mean = B['posterior_mean_coef1'][t] * x0 + B['posterior_mean_coef2'][t] * img                           # U:1078-1085
    nonzero_mask = 1 - (torch.tensor([t]) == 0).float()                                                      # U:1119
    return mean + nonzero_mask * (0.5 * B['posterior_log_variance_clipped'][t:t + 1]).exp() * noise          # U:1121
