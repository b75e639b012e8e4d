"""TEST INFRASTRUCTURE — ancestral DDPM sampling golden from the REAL reference: `GaussianDiffusion.p_sample` / `p_sample_loop`
(U:1087-1135) on the 'odd' clip (23 frames of 16 x 16, synthetic weights), torch.randn / randn_like patched to return
oracle.weights.pseudo_normal draws.  Writes tests/golden/ddpm_odd.npz:
  step_t                   single steps of the T = 1000 schedule at t = 999, 500, 0, each from the 'odd' x_t with noise
                           key ddpm/t{t}/noise0
  step_eps, step_x_after   the reference's eps and the x after each step
  guided_eps, guided_x_after   one cond_scale = 2 step at t = guided_t = 500 (combined eps of forward_with_cond_scale;
                           noise key ddpm/guided500/noise0)
  loop6_sample             the final image of a complete p_sample_loop with timesteps = 6 (sampling_timesteps None -> 6,
                           is_ddim_sampling False); noise key ddpm6/noise{k}: k = -1 start image, k = 0..5 loop step k
  coef1000                 (1000, 5) {ca, cb, c1, c2, sigma} per t from the reference's registered buffers
  oracle_maxabs            max|oracle.ddpm_oracle.ddpm_step - reference| over the three steps and the guided step, given the
                           reference's eps (0 on the last run: the restatement is the same fp32 torch arithmetic)
The archive is written with fixed zip timestamps, so re-running the script reproduces the file byte for byte.

Run in the build container only:    python oracle/make_golden_ddpm.py"""
import importlib
import io
import json
import os
import sys
import warnings
import zipfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import ddpm_oracle as DO     # noqa: E402
from oracle import weights as W          # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')
U_MOD = 'DM_3.modules.video_flow_diffusion_multiGPU_v0_crema_plus_faceemb_ca_multi_test'
CASE = (23, 16, 16)                       # the 'odd' geometry
STEP_T = (999, 500, 0)
GUIDED_T, SCALE = 500, 2.0
LOOP_T = 6


def save_npz(path, **arrays):
    """np.savez_compressed with fixed member timestamps (reproducible bytes); np.load reads it as usual."""
    with zipfile.ZipFile(path, 'w', compression=zipfile.ZIP_DEFLATED) as zf:
        for name in sorted(arrays):
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asarray(arrays[name]), allow_pickle=False)
            info = zipfile.ZipInfo(name + '.npy', date_time=(1980, 1, 1, 0, 0, 0))
            info.compress_type = zipfile.ZIP_DEFLATED
            zf.writestr(info, buf.getvalue())


class Injected:
    """torch.randn / randn_like replacement: draw k of the current key prefix is pseudo_normal(f'{prefix}{k}')."""

    def __init__(self):
        self.prefix, self.k = None, 0

    def start(self, prefix, k0):
        self.prefix, self.k = prefix, k0

    def __call__(self, shape):
        out = torch.from_numpy(W.pseudo_normal(f"{self.prefix}{self.k}", tuple(shape)))
        self.k += 1
        return out


def main():
    sys.path.insert(0, os.path.join(HERE, 'shims'))
    sys.path.insert(0, '/root/reference')
    warnings.filterwarnings("ignore")
    torch.set_num_threads(os.cpu_count())
    U = importlib.import_module(U_MOD)
    with open(os.path.join(GOLD, 'state_dict_schema.json')) as f:
        schema = [(n, tuple(s)) for n, s in json.load(f)['entries']]
    net = U.DynamicNfUnet3D(dim=64, cond_dim=1032, cond_aud=1024, cond_pose=6, cond_eye=2, num_frames=40, channels=275, out_grid_dim=2,
                            out_conf_dim=1, dim_mults=(1, 2, 4, 8), use_hubert_audio_cond=True, learn_null_cond=False,
                            use_final_activation=False, use_deconv=True, padding_mode="zeros", win_width=40).eval()
    net.load_state_dict(W.synth_state_dict(schema), strict=True)

    def diffusion(T):                     # FD:157-167 with sampling_timesteps=None -> the ancestral loop (U:1150)
        return U.DynamicNfGaussianDiffusion(denoise_fn=net, num_frames=40, image_size=32, sampling_timesteps=None, timesteps=T,
                                            loss_type='l2', use_dynamic_thres=True, null_cond_prob=0.1, ddim_sampling_eta=1.0).eval()
    D = diffusion(1000)
    assert not D.is_ddim_sampling
    Fr, h, w = CASE
    x_t, fea, cond = W.synth_inputs('odd', Fr, h, w)
    net.update_num_frames(Fr); D.update_num_frames(Fr)

    # the combined eps the step used (forward_with_cond_scale is what p_mean_variance calls, U:1089)
    seen = []
    fwcs = net.forward_with_cond_scale
    net.forward_with_cond_scale = lambda *a, **k: seen.append(fwcs(*a, **k)) or seen[-1]
    inj = Injected()
    real_randn, real_randn_like = torch.randn, torch.randn_like
    torch.randn = lambda *size, **kw: inj(size[0] if len(size) == 1 and not isinstance(size[0], int) else size)
    torch.randn_like = lambda t, **kw: inj(t.shape)
    out, worst = {}, 0.0
    try:
        def one_step(t, scale, key):
            seen.clear()
            inj.start(key, 0)
            x = D.p_sample(x_t.clone(), torch.full((1,), t, dtype=torch.long), fea, cond=cond, cond_scale=scale)
            assert len(seen) == 1 and inj.k == 1
            eps = seen[0]
            mine = DO.ddpm_step(eps, x_t, t, torch.from_numpy(W.pseudo_normal(f"{key}0", tuple(x_t.shape))))
            d = (mine - x).abs().max().item()
            print(f"p_sample t={t} cond_scale={scale}: |x|max {x.abs().max():.3f}; oracle ddpm_step vs reference max|d| {d:.3e}")
            return eps, x, d

        steps = [one_step(t, 1.0, f"ddpm/t{t}/noise") for t in STEP_T]
        out['step_t'] = np.array(STEP_T, dtype=np.int64)
        out['step_eps'] = np.stack([e[0].numpy() for e, _, _ in steps])
        out['step_x_after'] = np.stack([x[0].numpy() for _, x, _ in steps])
        ge, gx, gd = one_step(GUIDED_T, SCALE, f"ddpm/guided{GUIDED_T}/noise")
        out['guided_eps'], out['guided_x_after'] = ge[0].numpy(), gx[0].numpy()
        out['guided_t'], out['cond_scale'] = np.int64(GUIDED_T), np.float32(SCALE)
        worst = max([d for _, _, d in steps] + [gd])

        D6 = diffusion(LOOP_T)
        D6.update_num_frames(Fr)
        assert D6.sampling_timesteps == LOOP_T and not D6.is_ddim_sampling
        inj.start("ddpm6/noise", -1)
        sample = D6.p_sample_loop(fea, (1, 3, Fr, h, w), cond=cond, cond_scale=1.0)
        assert inj.k == LOOP_T                                # start image + one randn_like per step (t = 0 included)
        out['loop6_sample'], out['loop6_T'] = sample[0].numpy(), np.int64(LOOP_T)
        print(f"p_sample_loop T={LOOP_T}: |x|max {sample.abs().max():.3f} |x|mean {sample.abs().mean():.4f}")
    finally:
        torch.randn, torch.randn_like = real_randn, real_randn_like
        net.forward_with_cond_scale = fwcs

    # the per-step scalars as p_sample evaluates them from the registered buffers (U:1072-1121)
    coef = np.zeros((1000, 5), dtype=np.float32)
    shp = (1, 3, Fr, h, w)
    for t in range(1000):
        tt = torch.full((1,), t, dtype=torch.long)
        lv = U.extract(D.posterior_log_variance_clipped, tt, shp)
        nonzero_mask = (1 - (tt == 0).float()).reshape(1, 1, 1, 1, 1)
        coef[t] = [float(U.extract(D.sqrt_recip_alphas_cumprod, tt, shp)), float(U.extract(D.sqrt_recipm1_alphas_cumprod, tt, shp)),
                   float(U.extract(D.posterior_mean_coef1, tt, shp)), float(U.extract(D.posterior_mean_coef2, tt, shp)),
                   float(nonzero_mask * (0.5 * lv).exp())]
    out['coef1000'] = coef
    out['oracle_maxabs'] = np.float32(worst)
    print(f"oracle ddpm_step vs reference p_sample, worst max|d|: {worst:.3e}")
    path = os.path.join(GOLD, 'ddpm_odd.npz')
    save_npz(path, **out)
    print(f"wrote {path} ({os.path.getsize(path)} bytes)")


if __name__ == "__main__":
    main()
