"""CPU: the ancestral DDPM sampler without a GPU.  The oracle's restated step against the reference's own p_sample (golden eps
given, so no UNet forward runs), the host coefficients against the reference's registered buffers, which native calls one
`p_sample_loop` makes (eager, guided, segmented graph replay with a remainder), and the DDIM / DDPM dispatch of `sample()` and
`sample_one_video()`."""
import contextlib
import os
import unittest.mock as um

import numpy as np
import torch

from oracle import ddpm_oracle as DO
from oracle import weights as W
from tests import gpu_common as G

GOLD = os.path.join(G.ROOT, "tests", "golden", "ddpm_odd.npz")


class _FakeLib:
    def __init__(self, calls):
        self.calls = calls

    def __getattr__(self, name):
        def f(*a):
            self.calls.append(name)
            return 0
        return f


def _diffusion(timesteps=1000, sampling_timesteps=None):
    from dawn_pytorch_b200 import DynamicNfGaussianDiffusion, DynamicNfUnet3D
    net = DynamicNfUnet3D(**G.CTOR).eval()
    D = DynamicNfGaussianDiffusion(denoise_fn=net, num_frames=40, image_size=32, sampling_timesteps=sampling_timesteps, timesteps=timesteps,
                                   loss_type='l2', use_dynamic_thres=True, null_cond_prob=0.1, ddim_sampling_eta=1.0)
    return D, net


def test_oracle_step_reproduces_reference_p_sample():
    g = np.load(GOLD)
    F, h, w, _ = G.CASES["odd"]
    x_t, _, _ = W.synth_inputs("odd", F, h, w)
    for i, t in enumerate(g["step_t"].tolist()):
        noise = torch.from_numpy(W.pseudo_normal(f"ddpm/t{t}/noise0", tuple(x_t.shape)))
        x = DO.ddpm_step(torch.from_numpy(g["step_eps"][i])[None], x_t, t, noise)
        assert torch.equal(x[0], torch.from_numpy(g["step_x_after"][i])), t
    t = int(g["guided_t"])
    noise = torch.from_numpy(W.pseudo_normal(f"ddpm/guided{t}/noise0", tuple(x_t.shape)))
    x = DO.ddpm_step(torch.from_numpy(g["guided_eps"])[None], x_t, t, noise)
    assert torch.equal(x[0], torch.from_numpy(g["guided_x_after"]))
    # t = 0 adds no noise: the step is the clamped posterior mean
    assert torch.equal(DO.ddpm_step(torch.from_numpy(g["step_eps"][2])[None], x_t, 0, noise),
                       DO.ddpm_step(torch.from_numpy(g["step_eps"][2])[None], x_t, 0, torch.zeros_like(noise)))


def test_host_coefficients_equal_reference_buffers():
    D, _ = _diffusion()
    ref = torch.from_numpy(np.load(GOLD)["coef1000"])
    mine = torch.tensor([D.ddpm_coefficients(t) for t in range(1000)], dtype=torch.float32)
    assert torch.equal(mine, ref)
    assert mine[0, 4] == 0 and bool((mine[1:, 4] > 0).all())
    # the device table carries the same values, row k = loop step k, t in the first int64
    times = [999, 500, 0]
    tab = D.ddpm_table(times)
    assert tab.shape == (3, 4) and tab[:, 0].tolist() == times
    assert torch.equal(tab.view(torch.float32)[:, 2:7], ref[times])


def _run(D, net, calls, *, b=1, cond_scale=1.0, use_graph=False, segment=None):
    import dawn_pytorch_b200.diffusion as dd
    D.update_num_frames(4)
    net.set_clip_invariants = lambda f, c: calls.append(("invariants", bool(c.abs().sum() > 0)))
    net.forward_x3 = lambda x, t, e: calls.append(("forward_x3", int(t)))
    net._handle = None
    stream = type("S", (), {"cuda_stream": 0})()

    def noise(k, shp):
        if k >= 0:
            calls.append(("draw", k))
        return torch.zeros(shp)
    with contextlib.ExitStack() as es:
        es.enter_context(um.patch.object(dd, "lib", _FakeLib(calls)))
        es.enter_context(um.patch("torch.cuda.current_stream", lambda: stream))
        es.enter_context(um.patch("torch.cuda.synchronize", lambda *a: None))
        if segment is not None:
            es.enter_context(um.patch.object(dd, "DDPM_SEGMENT_STEPS", segment))
        D.p_sample_loop(torch.rand(b, 272, 8, 8), (b, 3, 4, 8, 8), cond=torch.randn(b, 4, 1032), cond_scale=cond_scale,
                        noise_fn=noise, use_graph=use_graph)


def test_native_call_sequence_eager_and_guided():
    D, net = _diffusion(timesteps=6)
    calls = []
    _run(D, net, calls)
    ts = [5, 4, 3, 2, 1, 0]
    step = lambda k, t: [("forward_x3", t)] + ([("draw", k)] if t > 0 else []) + ["dawn_unet_ddpm_step"]   # noqa: E731
    assert calls == [("invariants", True)] + [c for k, t in enumerate(ts) for c in step(k, t)]
    assert ("draw", 5) not in calls                                     # no draw for t = 0
    calls.clear()
    _run(D, net, calls, cond_scale=2.0)
    guided = lambda k, t: ([("invariants", True), ("forward_x3", t), ("invariants", False), ("forward_x3", t)]    # noqa: E731
                           + ([("draw", k)] if t > 0 else []) + ["dawn_unet_ddpm_step"])
    assert calls == [c for k, t in enumerate(ts) for c in guided(k, t)]


def test_native_call_sequence_segmented_graph():
    """T = 6 with 4-step segments, two clips: one capture, one segment launch per clip whose noise ring holds loop steps 0-3,
    then the remaining 2 steps (t = 1, 0) eagerly; no draw for t = 0."""
    D, net = _diffusion(timesteps=6)
    calls = []
    _run(D, net, calls, b=2, use_graph=True, segment=4)
    assert calls.count("dawn_unet_ddpm_capture") == 1 and calls.count("dawn_unet_sampler_launch") == 2
    per_clip = ([("invariants", True)] + [("draw", k) for k in range(4)] + ["dawn_unet_sampler_launch",
                ("forward_x3", 1), ("draw", 4), "dawn_unet_ddpm_step", ("forward_x3", 0), "dawn_unet_ddpm_step"])
    assert calls == [("invariants", True), "dawn_unet_ddpm_capture"] + per_clip + per_clip
    # the cached capture is reused; the guided loop refuses the graph
    calls.clear()
    _run(D, net, calls, b=1, use_graph=True, segment=4)
    assert "dawn_unet_ddpm_capture" not in calls
    try:
        _run(D, net, [], use_graph=True, cond_scale=2.0, segment=4)
        raise AssertionError("guided graph sampling must raise")
    except NotImplementedError:
        pass


def test_sample_dispatches_ddim_or_ddpm():
    for steps, ddim in ((None, False), (1000, False), (2000, False), (20, True), (999, True)):
        D, _ = _diffusion(sampling_timesteps=steps)
        assert D.is_ddim_sampling == ddim
        picked = []
        with um.patch.object(D, "ddim_sample", lambda *a, **k: picked.append("ddim")), \
                um.patch.object(D, "p_sample_loop", lambda *a, **k: picked.append("ddpm")):
            D.sample(torch.zeros(1, 256, 8, 8), torch.zeros(1, 16, 8, 8), cond=torch.zeros(1, 40, 1032))
        assert picked == ["ddim" if ddim else "ddpm"], steps


def test_sample_one_video_dispatches_ddim_or_ddpm():
    from dawn_pytorch_b200 import FlowDiffusion
    for steps, ddim in ((None, False), (1000, False), (20, True)):
        m = FlowDiffusion(sampling_timesteps=steps, pose_dim=6, win_width=40)
        nf, size = 4, 32
        m.update_num_frames(nf)
        picked = []

        def fake(kind):
            def f(fea, shape, cond=None, cond_scale=1., noise_fn=None, use_graph=False):
                picked.append((kind, noise_fn, use_graph))
                return torch.zeros(shape)
            return f
        with um.patch.object(m.generator, "compute_fea", lambda img: torch.zeros(img.shape[0], 256, size // 4, size // 4)), \
                um.patch.object(m.face_loc_emb, "forward", lambda x: torch.zeros(x.shape[0], 16, size // 4, size // 4)), \
                um.patch.object(m.generator, "decode_sample", lambda s, p, need_deformed: (torch.zeros(nf, 3, size, size),) * 2), \
                um.patch.object(m.diffusion, "ddim_sample", fake("ddim")), um.patch.object(m.diffusion, "p_sample_loop", fake("ddpm")):
            nfn = lambda k, s: torch.zeros(s)      # noqa: E731
            bbox = torch.tensor([[0., 10., 0., 10., 32., 32.]]).unsqueeze(-1).repeat(1, 1, nf)
            out = m.sample_one_video(torch.zeros(1, 3, size, size), torch.zeros(1, nf, 1024), torch.zeros(1, 6, nf), torch.zeros(1, 2, nf),
                                     bbox, cond_scale=1.0, noise_fn=nfn, use_graph=True)
        assert picked == [("ddim" if ddim else "ddpm", nfn, True)], steps
        assert out["sample_vid_grid"].shape == (1, 2, nf, size // 4, size // 4)
