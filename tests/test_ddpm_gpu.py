"""-m gpu: ancestral DDPM sampling (`p_sample_loop`, reference U:1087-1135) around the CUDA UNet.  Single steps and a guided step
against the REAL reference's p_sample, a complete short-schedule loop against its p_sample_loop (tests/golden/ddpm_odd.npz,
oracle/make_golden_ddpm.py, injected noise), the segmented graph replay against the eager loop, and the FlowDiffusion dispatch."""
import os
import unittest.mock as um

import numpy as np
import pytest
import torch

from oracle import weights as W
from tests import gpu_common as G

pytestmark = pytest.mark.gpu

GOLD = os.path.join(G.ROOT, "tests", "golden", "ddpm_odd.npz")


def _diffusion(timesteps=1000):
    from dawn_pytorch_b200 import DynamicNfGaussianDiffusion
    net = G.cuda_net()
    D = DynamicNfGaussianDiffusion(denoise_fn=net, num_frames=40, image_size=32, sampling_timesteps=None, timesteps=timesteps,
                                   loss_type='l2', use_dynamic_thres=True, null_cond_prob=0.1, ddim_sampling_eta=1.0).cuda()
    F, h, w, _ = G.CASES["odd"]
    x_t, fea, cond = W.synth_inputs("odd", F, h, w)
    D.update_num_frames(F)
    return D, (F, h, w), x_t, fea.cuda(), cond.cuda()


def _injected(prefix, x_t=None):
    """noise_fn with the reference's draws: step -1 is the start image (x_t if given), step k the key {prefix}{k}."""
    def noise_fn(k, shape):
        if k < 0 and x_t is not None:
            return x_t.clone()
        if k < 0:
            return torch.from_numpy(W.pseudo_normal(f"{prefix}{k}", tuple(shape)))
        return torch.from_numpy(W.pseudo_normal(f"{prefix}{k}", (1,) + tuple(shape)))[0]
    return noise_fn


def test_single_steps_match_reference_p_sample():
    """t = 999, 500, 0 (no noise) and a cond_scale = 2 step at t = 500.  Bound: the DDIM step test's 2e-4.  The UNet's eps error
    reaches x through c1 * cb / s, which is below 4e-3 at all four steps (from the golden's coefficients and thresholds), so the
    eps tolerance of the forward tests leaves x far inside it."""
    D, (F, h, w), x_t, fea, cond = _diffusion()
    g = np.load(GOLD)
    for i, t in enumerate(g["step_t"].tolist()):
        img = D.p_sample_loop(fea, (1, 3, F, h, w), cond=cond, noise_fn=_injected(f"ddpm/t{t}/noise", x_t), times=[t])
        d = (img[0].cpu() - torch.from_numpy(g["step_x_after"][i])).abs().max().item()
        print(f"ddpm step t={t}: max|d| vs reference p_sample = {d:.3e}")
        assert d < 2e-4
    t, scale = int(g["guided_t"]), float(g["cond_scale"])
    img = D.p_sample_loop(fea, (1, 3, F, h, w), cond=cond, cond_scale=scale, noise_fn=_injected(f"ddpm/guided{t}/noise", x_t), times=[t])
    d = (img[0].cpu() - torch.from_numpy(g["guided_x_after"])).abs().max().item()
    print(f"ddpm guided step t={t} cond_scale={scale}: max|d| vs reference p_sample = {d:.3e}")
    assert d < 2e-4


def test_short_loop_matches_reference_p_sample_loop_eager_and_graph():
    """A complete timesteps = 6 loop: eagerly, and as 4-step graph segments (one replay, then 2 eager steps)."""
    import dawn_pytorch_b200.diffusion as dd
    g = np.load(GOLD)
    T = int(g["loop6_T"])
    D, (F, h, w), _, fea, cond = _diffusion(T)
    assert not D.is_ddim_sampling and D.num_timesteps == T
    ref = torch.from_numpy(g["loop6_sample"])
    noise_fn = _injected("ddpm6/noise")
    eager = D.p_sample_loop(fea, (1, 3, F, h, w), cond=cond, noise_fn=noise_fn)[0].clone()
    with um.patch.object(dd, "DDPM_SEGMENT_STEPS", 4):
        graph = D.p_sample_loop(fea, (1, 3, F, h, w), cond=cond, noise_fn=noise_fn, use_graph=True)[0].clone()
        assert D._graph["key"][0] == "ddpm" and D._graph["ring"].shape[0] == 4
    torch.cuda.synchronize()
    de, dg, dge = [(a - b).abs().max().item() for a, b in ((eager.cpu(), ref), (graph.cpu(), ref), (graph, eager))]
    print(f"ddpm loop T={T}: eager vs reference {de:.3e}, graph (4-step segments) vs reference {dg:.3e}, graph vs eager {dge:.3e}")
    assert de < 2e-4 and dg < 2e-4
    assert dge < 5e-5


def test_thousand_step_graph_matches_eager_and_replays():
    """T = 1000 on 'odd' with the default noise and a fixed torch seed: 50 replays of one 20-step segment == the eager loop; a
    second clip replays the cached graph without re-capture."""
    D, (F, h, w), _, fea, cond = _diffusion()

    def run(c, use_graph):
        torch.manual_seed(1234)
        return D.p_sample_loop(fea, (1, 3, F, h, w), cond=c, use_graph=use_graph)[0].clone()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eager = run(cond, False)
    e0.record()
    graph = run(cond, True)
    e1.record()
    torch.cuda.synchronize()
    n_nodes = D.denoise_fn.last_launch_count()
    d = (graph - eager).abs().max().item()
    print(f"ddpm T=1000 graph vs eager max|d| {d:.3e}; {n_nodes} graph nodes per 20-step segment; graph loop incl. capture "
          f"{e0.elapsed_time(e1):.0f} ms")
    assert torch.isfinite(graph).all()
    assert d < 5e-5
    gen0 = D._graph["gen"]
    cond2 = cond.flip(1).contiguous()
    e2, g2 = run(cond2, False), run(cond2, True)
    torch.cuda.synchronize()
    assert D._graph["gen"] == gen0                       # no re-capture
    assert (g2 - e2).abs().max().item() < 5e-5
    assert (g2 - graph).abs().max().item() > 1e-3        # and it really is a different clip


def test_sample_one_video_runs_the_ancestral_loop():
    """FlowDiffusion(sampling_timesteps=None): sample_one_video runs p_sample_loop (U:1150) over 1000 steps; its grid equals a
    direct p_sample_loop call with the same arguments and noise_fn."""
    from dawn_pytorch_b200 import FlowDiffusion
    from oracle import lfg_oracle as L
    from oracle.make_golden_e2e import e2e_inputs, face_sd
    m = FlowDiffusion(sampling_timesteps=None, pose_dim=6, win_width=40, ddim_sampling_eta=1.0)
    assert not m.diffusion.is_ddim_sampling
    m.diffusion.load_state_dict({**{"denoise_fn." + k: v for k, v in G.synth_sd().items()},
                                 **{k: v for k, v in m.diffusion.state_dict().items() if not k.startswith("denoise_fn.")}}, strict=True)
    m.generator.load_state_dict(W.lfg_synth_state_dict(L.state_dict_schema()), strict=True)
    m.face_loc_emb.load_state_dict(face_sd(), strict=True)
    m = m.cuda()
    img, hubert, pose, eye, bbox, init_pose, init_eye = [t.cuda() for t in e2e_inputs()]
    nf = hubert.shape[1]
    m.update_num_frames(nf)

    def noise_fn(k, shape):
        return torch.randn(tuple(shape), generator=torch.Generator().manual_seed(1000 + k))
    seen = {}
    loop = m.diffusion.p_sample_loop

    def spy(*a, **k):
        seen["args"] = (a, k)
        return loop(*a, **k)
    with um.patch.object(m.diffusion, "p_sample_loop", spy):
        out = m.sample_one_video(sample_img=img, sample_audio_hubert=hubert, sample_pose=pose, sample_eye=eye, sample_bbox=bbox,
                                 init_pose=init_pose, init_eye=init_eye, cond_scale=1.0, noise_fn=noise_fn)
    a, k = seen["args"]
    assert k["noise_fn"] is noise_fn
    direct = loop(*a, **k)
    torch.cuda.synchronize()
    d = (out["sample_vid_grid"] - direct[:, :2]).abs().max().item()
    print(f"sample_one_video (1000-step DDPM): grid vs direct p_sample_loop max|d| {d:.3e}")
    assert d < 5e-5
    for key in ("sample_vid_grid", "sample_vid_conf", "sample_out_vid", "sample_warped_vid"):
        assert torch.isfinite(out[key]).all(), key
