"""-m gpu: parity of the CUDA path (through the reference-facing module API -> C-ABI) against
(1) golden vectors produced by the REAL reference, (2) the CPU oracle on the same seeded inputs,
(3) size-independent properties at sizes the oracle cannot reach in seconds."""
import os

import numpy as np
import pytest
import torch

from oracle import unet_oracle as O
from oracle import weights as W
from tests import gpu_common as G

pytestmark = pytest.mark.gpu


def run(net, x, t, cond, cond_scale=1.0):
    net.update_num_frames(x.shape[2])
    with torch.no_grad():
        out = net.forward_with_cond_scale(x.cuda(), t.cuda(), cond=cond.cuda(), cond_scale=cond_scale)
    torch.cuda.synchronize()
    return out.cpu()


@pytest.mark.parametrize("case", ["band", "odd", "cfg1"])
def test_eps_matches_reference_golden(case):
    net = G.cuda_net()
    x, t, cond, _, _ = G.clip(case)
    out = run(net, x, t, cond)
    ref = torch.from_numpy(G.golden(case)["eps"])
    assert out.shape == ref.shape
    r = G.over_tol(out, ref)
    print(f"{case}: max|d|/(atol+rtol|ref|) = {r:.3f}, max|d| = {(out - ref).abs().max():.3e}")
    assert r <= 1.0
    if case == "band":      # the windowed twin of the reference (`_local_opt` + local_attention.py LA:275-342) on the same clip
        r_ul = G.over_tol(out, torch.from_numpy(G.golden(case)["eps_local_opt"]))
        print(f"band vs the reference's _local_opt UNet: {r_ul:.3f} x tol")
        assert r_ul <= 1.0


def test_every_submodule_boundary_matches_oracle():
    """All 40 sub-module outputs (oracle `taps`) on the banded clip (F=96 > 81: window active)."""
    net = G.cuda_net()
    x, t, cond, _, _ = G.clip("band")
    taps_o = {}
    with torch.no_grad():
        O.unet_forward(G.synth_sd(), O.UnetCfg(), x, t, cond, taps=taps_o)
    bufs = net.request_taps(list(taps_o), x.shape[2], x.shape[3], x.shape[4], torch.device("cuda"))
    try:
        run(net, x, t, cond)
    finally:
        got = {k: v.cpu() for k, v in bufs.items()}
        net.clear_taps()
    worst = {}
    for name, ref in taps_o.items():
        assert got[name].shape == ref.shape, name
        worst[name] = G.over_tol(got[name], ref)
    bad = {k: v for k, v in worst.items() if v > 1.0}
    print("worst taps:", sorted(worst.items(), key=lambda kv: -kv[1])[:5])
    assert not bad, bad


def test_hoisted_fast_path_equals_general_entry():
    """forward_x3 (clip invariants hoisted: SURVEY a2/a5) == forward(x275) on the same clip."""
    net = G.cuda_net()
    x, t, cond, x_t, fea = G.clip("odd")
    ref = run(net, x, t, cond)
    net.set_clip_invariants(fea[0].cuda(), cond[0].cuda())
    out = net.forward_x3(x_t[0].cuda(), t.cuda())
    torch.cuda.synchronize()
    assert G.over_tol(out.cpu()[None], ref) <= 0.25
    assert G.over_tol(out.cpu()[None], torch.from_numpy(G.golden("odd")["eps"])) <= 1.0


def test_cond_scale_two_forwards_golden():
    net = G.cuda_net()
    x, t, cond, _, _ = G.clip("odd")
    out = run(net, x, t, cond, cond_scale=2.0)
    assert G.over_tol(out, torch.from_numpy(G.golden("odd")["eps_cond_scale2"])) <= 1.0


def test_batch_elements_are_independent():
    net = G.cuda_net()
    xa, t, ca, _, _ = G.clip("odd")
    xb, _, cb, _, _ = G.clip("odd_b", 23, 16, 16, 47)
    ya, yb = run(net, xa, t, ca), run(net, xb, t, cb)
    y2 = run(net, torch.cat([xa, xb]), torch.cat([t, t + 100]), torch.cat([ca, cb]))
    assert G.over_tol(y2[0:1], ya) <= 0.05
    # second element used a different timestep: must differ from the t=47 run but match its own oracle
    with torch.no_grad():
        ob = O.unet_forward(G.synth_sd(), O.UnetCfg(), xb, t + 100, cb)
    assert G.over_tol(y2[1:2], ob) <= 1.0
    assert (y2[1:2] - yb).abs().max() > 1e-3


def test_host_buffer_entry_matches():
    net = G.cuda_net()
    x, t, cond, x_t, fea = G.clip("band")
    out = net.forward_host(x_t[0].contiguous().pin_memory(), fea[0].contiguous().pin_memory(),
                           cond[0].contiguous().pin_memory(), int(t))
    assert G.over_tol(out[None], torch.from_numpy(G.golden("band")["eps"])) <= 1.0
    assert net.last_launch_count() > 300


def test_cfg2_shape_against_oracle():
    """BASELINE configs[1] shape: 100 frames, 32x32 latent (window active); oracle takes ~10 s on CPU."""
    net = G.cuda_net()
    x, t, cond, _, _ = G.clip("cfg2", 100, 32, 32, 333)
    out = run(net, x, t, cond)
    with torch.no_grad():
        ref = O.unet_forward(G.synth_sd(), O.UnetCfg(), x, t, cond)
    r = G.over_tol(out, ref)
    print(f"cfg2: {r:.3f}")
    assert r <= 1.0


def test_full_size_properties_cfg3():
    """BASELINE configs[2]: 200 frames, 64x64 latent.  The oracle needs minutes here, so check
    size-independent properties: (a) general entry == hoisted entry (linearity of the init conv),
    (b) run-to-run reproducibility, (c) finite, O(1) outputs, (d) frames far outside every temporal
    window still interact only through GroupNorm statistics: perturbing frame 0 changes frame 199 a little, not a lot."""
    net = G.cuda_net()
    F, h, w = 200, 64, 64
    x_t, fea, cond = W.synth_inputs("cfg3", F, h, w)
    t = torch.full((1,), 500, dtype=torch.long).cuda()
    net.update_num_frames(F)
    net.set_clip_invariants(fea[0].cuda(), cond[0].cuda())
    xt = x_t[0].cuda()
    a = net.forward_x3(xt, t).clone()
    b = net.forward_x3(xt, t).clone()
    torch.cuda.synchronize()
    assert torch.isfinite(a).all() and 0.1 < a.abs().max().item() < 20
    assert G.over_tol(b[None], a[None]) <= 0.05
    x = torch.cat([xt, fea[0].cuda().unsqueeze(1).expand(-1, F, -1, -1)], dim=0)[None].contiguous()
    with torch.no_grad():
        g = net.forward_with_cond_scale(x, t, cond=cond.cuda(), cond_scale=1.0)
    assert G.over_tol(g[0][None], a[None]) <= 0.25
    del x, g
    xt2 = xt.clone()
    xt2[:, 0] += 1.0
    net.set_clip_invariants(fea[0].cuda(), cond[0].cuda())
    c = net.forward_x3(xt2, t)
    d_near = (c[:, 0] - a[:, 0]).abs().max().item()
    d_far = (c[:, 199] - a[:, 199]).abs().max().item()
    assert d_near > 1e-2 and d_far < d_near


def test_cfg3_matches_reference_golden_probes():
    """BASELINE configs[2] (the benchmarked shape: 200 f x 64x64, window active) against the REAL reference
    (oracle/make_golden_cfg3.py: eps on a stride-8 lattice + 65536 eps probes + 2048 probes and abs-mean at each of the 46
    sub-module boundaries).  Exercises the level-0 paths that only exist at full size (persistent halo conv over 148 CTAs,
    4096-pixel temporal attention, spatial-linear-attention splits) through BOTH entries: forward_with_cond_scale(x275) with
    taps, and the hoisted forward_x3."""
    CASE, FR, H, WD, T, SUB = "cfg3", 200, 64, 64, 500, 8

    def probe_idx(name, numel, n=2048):
        return W.probe_indices(name, numel, n)

    g = np.load(os.path.join(G.ROOT, "tests", "golden", "cfg3.npz"))
    net = G.cuda_net()
    x_t, fea, cond = W.synth_inputs(CASE, FR, H, WD)
    t = torch.full((1,), T, dtype=torch.long).cuda()
    names = sorted(k.split("/")[1] for k in g.files if k.startswith("tap/") and k.endswith("/vals"))
    assert len(names) >= 40
    x = torch.cat([x_t, fea.unsqueeze(2).expand(-1, -1, FR, -1, -1)], dim=1).contiguous().cuda()
    bufs = net.request_taps(names, FR, H, WD, torch.device("cuda"))
    try:
        net.update_num_frames(FR)
        with torch.no_grad():
            out = net.forward_with_cond_scale(x, t, cond=cond.cuda(), cond_scale=1.0)
        torch.cuda.synchronize()
        worst = {}
        for n in names:
            flat = bufs[n].reshape(-1)
            assert list(bufs[n].shape) == g[f"tap/{n}/shape"].tolist(), n
            idx = torch.from_numpy(probe_idx(f"{CASE}/{n}", flat.numel())).cuda()
            got = flat[idx].cpu()
            worst[n] = G.over_tol(got, torch.from_numpy(g[f"tap/{n}/vals"]))
            am = flat.double().abs().mean().item()
            assert abs(am - float(g[f"tap/{n}/absmean"])) <= 1e-3 * float(g[f"tap/{n}/absmean"]) + 1e-6, (n, am)
    finally:
        net.clear_taps()
    del x, bufs
    print("cfg3 worst taps:", sorted(worst.items(), key=lambda kv: -kv[1])[:5])
    bad = {k: v for k, v in worst.items() if v > 1.0}
    assert not bad, bad

    def check_eps(o, tag):
        o = o.cpu()
        r_sub = G.over_tol(o[0][:, :, ::SUB, ::SUB], torch.from_numpy(g["eps_sub"]))
        idx = torch.from_numpy(probe_idx(f"{CASE}/eps", o.numel(), 65536))
        r_pr = G.over_tol(o.reshape(-1)[idx], torch.from_numpy(g["eps_probe"]))
        am, sm = o.double().abs().mean().item(), o.double().sum().item()
        print(f"cfg3 {tag}: eps lattice {r_sub:.3f} x tol, probes {r_pr:.3f} x tol, absmean {am:.6f} (ref {g['eps_stats'][0]:.6f})")
        assert r_sub <= 1.0 and r_pr <= 1.0
        assert abs(am - g["eps_stats"][0]) <= 1e-4 and abs(sm - g["eps_stats"][1]) <= 1e-4 * o.numel() ** 0.5 + 1e-3 * abs(g["eps_stats"][1])

    check_eps(out, "general entry")
    net.set_clip_invariants(fea[0].cuda(), cond[0].cuda())
    o3 = net.forward_x3(x_t[0].cuda(), t)
    torch.cuda.synchronize()
    check_eps(o3[None], "hoisted entry")


def test_ddim_sampler_steps_match_reference_golden():
    """Row a16: DDIM update (x0, exact clip-wide 0.9-quantile threshold, eta-noise) around the CUDA UNet, against the
    reference's own arithmetic with injected noise (tests/golden/ddim_odd.npz: steps 952->904, 523->476, 47->0)."""
    from dawn_pytorch_b200 import DynamicNfGaussianDiffusion
    net = G.cuda_net()
    D = DynamicNfGaussianDiffusion(denoise_fn=net, num_frames=40, image_size=32, sampling_timesteps=20, timesteps=1000,
                                   loss_type='l2', use_dynamic_thres=True, null_cond_prob=0.1, ddim_sampling_eta=1.0).cuda()
    assert len(D.state_dict()) == 912                      # 900 UNet entries + 12 schedule buffers (SURVEY App. B)
    g = np.load(__import__("os").path.join(G.ROOT, "tests", "golden", "ddim_odd.npz"))
    F, h, w, _ = G.CASES["odd"]
    x_t, fea, cond = W.synth_inputs("odd", F, h, w)
    steps = [tuple(int(v) for v in p) for p in g["steps"].tolist()]
    assert steps[0] == D.ddim_schedule()[0] and steps[-1] == D.ddim_schedule()[-1]
    D.update_num_frames(F)

    def noise_fn(k, shape):
        if k < 0:
            return x_t.clone()
        return torch.from_numpy(W.pseudo_normal(f"odd/noise{k}", (1,) + tuple(shape)))[0]

    for nsteps in (1, 3):
        img = D.ddim_sample(fea.cuda(), (1, 3, F, h, w), cond=cond.cuda(), noise_fn=noise_fn, pairs=steps[:nsteps])
        torch.cuda.synchronize()
        ref = torch.from_numpy(g["x_after"][nsteps - 1])
        d = (img.cpu() - ref).abs().max().item()
        print(f"ddim {nsteps} step(s): max|d| = {d:.3e}")
        assert d < 2e-4


def _odd_sampler():
    from dawn_pytorch_b200 import DynamicNfGaussianDiffusion
    net = G.cuda_net()
    D = DynamicNfGaussianDiffusion(denoise_fn=net, num_frames=40, image_size=32, sampling_timesteps=20, timesteps=1000,
                                   loss_type='l2', use_dynamic_thres=True, null_cond_prob=0.1, ddim_sampling_eta=1.0).cuda()
    F, h, w, _ = G.CASES["odd"]
    x_t, fea, cond = W.synth_inputs("odd", F, h, w)
    D.update_num_frames(F)

    def noise_fn(k, shape):
        if k < 0:
            return x_t.clone()
        return torch.from_numpy(W.pseudo_normal(f"odd/noise{k}", (1,) + tuple(shape)))[0]
    return D, (F, h, w), fea, cond, noise_fn


def test_graph_captured_sampler_matches_golden_and_eager():
    """Row N2: the whole DDIM loop as ONE CUDA graph (dawn_unet_sampler_capture/launch) == the eager loop == the
    reference's arithmetic (golden, injected noise); a second clip replays the cached graph."""
    D, (F, h, w), fea, cond, noise_fn = _odd_sampler()
    g = np.load(__import__("os").path.join(G.ROOT, "tests", "golden", "ddim_odd.npz"))
    steps = [tuple(int(v) for v in p) for p in g["steps"].tolist()]
    eager = D.ddim_sample(fea.cuda(), (1, 3, F, h, w), cond=cond.cuda(), noise_fn=noise_fn, pairs=steps).clone()
    graph = D.ddim_sample(fea.cuda(), (1, 3, F, h, w), cond=cond.cuda(), noise_fn=noise_fn, pairs=steps, use_graph=True).clone()
    torch.cuda.synchronize()
    n_launch = D.denoise_fn.last_launch_count()
    ref = torch.from_numpy(g["x_after"][len(steps) - 1])
    print(f"graph sampler: vs golden {(graph.cpu() - ref).abs().max():.3e}, vs eager {(graph - eager).abs().max():.3e}, "
          f"{n_launch} kernel launches in one graph")
    assert (graph.cpu() - ref).abs().max().item() < 2e-4
    assert (graph - eager).abs().max().item() < 5e-5
    assert n_launch >= 3 * 200
    # replay on a second clip (other conditioning): the cached graph must pick up the refreshed clip invariants
    gen0 = D._graph["gen"]
    cond2 = cond.flip(1).contiguous()
    e2 = D.ddim_sample(fea.cuda(), (1, 3, F, h, w), cond=cond2.cuda(), noise_fn=noise_fn, pairs=steps).clone()
    g2 = D.ddim_sample(fea.cuda(), (1, 3, F, h, w), cond=cond2.cuda(), noise_fn=noise_fn, pairs=steps, use_graph=True).clone()
    torch.cuda.synchronize()
    assert D._graph["gen"] == gen0                       # no re-capture
    assert (g2 - e2).abs().max().item() < 5e-5
    assert (g2 - graph).abs().max().item() > 1e-3        # and it really is a different clip


def test_handle_ddim_step_equals_plain_entry_unsharded():
    """dawn_unet_ddim_step on an unsharded handle is dawn_ddim_step (same kernels, n_global = n)."""
    import ctypes
    from dawn_pytorch_b200._lib import lib, check
    net = G.cuda_net()
    net.update_num_frames(8)
    x, t, cond, x_t, fea = G.clip("smoke", 8, 8, 8, 500)
    net.set_clip_invariants(fea[0].cuda(), cond[0].cuda())          # makes sure the handle exists
    gen = torch.Generator().manual_seed(5)
    n = 3 * 37 * 16 * 16
    xa = (torch.randn(n, generator=gen) * 1.5).cuda()
    eps, noise = torch.randn(n, generator=gen).cuda(), torch.randn(n, generator=gen).cuda()
    xb = xa.clone()
    scratch = torch.empty(n + 512, dtype=torch.int32, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    args = (n, 1.3, 0.8, 0.9, 0.3, 0.2, 0.9, ctypes.c_void_p(scratch.data_ptr()), st)
    check(lib.dawn_ddim_step(ctypes.c_void_p(xa.data_ptr()), ctypes.c_void_p(eps.data_ptr()), ctypes.c_void_p(noise.data_ptr()), *args), "a")
    check(lib.dawn_unet_ddim_step(net._handle, ctypes.c_void_p(xb.data_ptr()), ctypes.c_void_p(eps.data_ptr()),
                                  ctypes.c_void_p(noise.data_ptr()), *args), "b")
    torch.cuda.synchronize()
    assert torch.equal(xa, xb)
    # against torch's own quantile arithmetic (reference U:1183-1205)
    xr = (torch.randn(n, generator=torch.Generator().manual_seed(5)) * 1.5)
    e, nz = eps.cpu(), noise.cpu()
    x0 = 1.3 * xr - 0.8 * e
    s = torch.quantile(x0.abs(), 0.9).clamp(min=1.0)
    ref = x0.clamp(-s, s) / s * 0.9 + 0.3 * e + 0.2 * nz
    assert (xa.cpu() - ref).abs().max().item() < 2e-6


def test_general_entry_selects_its_init_conv_path_on_the_device():
    """Drop-in entry forward(x275): frame-invariant feature channels (what the reference's sampler passes, U:1167) take the
    hoisted init conv, frame-varying ones the full 7x7 conv over all 275 channels — chosen by a device-side flag, both
    against the oracle on the same inputs."""
    net = G.cuda_net()
    x, t, cond, x_t, fea = G.clip("odd")
    with torch.no_grad():
        ref_inv = O.unet_forward(G.synth_sd(), O.UnetCfg(), x, t, cond)
    out_inv = run(net, x, t, cond)
    assert G.over_tol(out_inv, ref_inv) <= 1.0
    xv = x.clone()
    F = x.shape[2]
    ramp = torch.linspace(-0.5, 0.5, F).view(1, 1, F, 1, 1)
    xv[:, 3:] = torch.relu(xv[:, 3:] + ramp)                  # features now differ from frame to frame
    with torch.no_grad():
        ref_var = O.unet_forward(G.synth_sd(), O.UnetCfg(), xv, t, cond)
    out_var = run(net, xv, t, cond)
    r = G.over_tol(out_var, ref_var)
    print(f"general entry, frame-varying features: {r:.3f} x tol; invariant: {G.over_tol(out_inv, ref_inv):.3f}")
    assert r <= 1.0
    assert (out_var - out_inv).abs().max().item() > 1e-2
    # a single differing value in the last frame must flip the path as well
    x1 = x.clone()
    x1[0, 274, F - 1, -1, -1] += 1.0
    with torch.no_grad():
        ref1 = O.unet_forward(G.synth_sd(), O.UnetCfg(), x1, t, cond)
    assert G.over_tol(run(net, x1, t, cond), ref1) <= 1.0
    # and back: the invariant clip again (the flag is re-evaluated on every call)
    assert G.over_tol(run(net, x, t, cond), ref_inv) <= 1.0


@pytest.mark.parametrize("tag,F,h,w,t", [
    ("edge_f1", 1, 8, 8, 999),          # a single frame: every temporal softmax has one key
    ("edge_f40", 40, 8, 16, 0),         # F == window, non-square latent (w = 2h), t = 0
    ("edge_f41", 41, 16, 8, 523),       # first length at which the band excludes a pair (|i-j| = 41 > 40), h = 2w
    ("edge_f81", 81, 8, 8, 47),         # 2*window + 1: the centre frame sees the whole clip, the ends half of it
    ("edge_f17x24", 17, 24, 24, 300),   # latent side not a power of two (24 = 8*3): level sizes 24, 12, 6, 3
    ("long_f250x8", 250, 8, 8, 640),    # > 240 frames on one GPU: two overlapping on-chip segments per pixel at level 0 (in-place layer: input copied aside)
])
def test_edge_geometries_against_oracle(tag, F, h, w, t):
    """Ragged / extreme geometries the fused kernels special-case (frame counts around the +-40 window and the 16-frame MMA
    tile, non-square and non-power-of-two latents) against the CPU oracle on the same seeded inputs."""
    net = G.cuda_net()
    x, tt, cond, _, _ = G.clip(tag, F, h, w, t)
    out = run(net, x, tt, cond)
    with torch.no_grad():
        ref = O.unet_forward(G.synth_sd(), O.UnetCfg(), x, tt, cond)
    r = G.over_tol(out, ref)
    print(f"{tag}: {r:.3f} x tol, max|d| {(out - ref).abs().max():.2e}")
    assert r <= 1.0


def test_other_window_width_against_oracle():
    """win_width is a constructor argument (FD:155): an 8-frame window on a 23-frame clip."""
    from dawn_pytorch_b200 import DynamicNfUnet3D
    ctor = dict(G.CTOR, win_width=8)
    net = DynamicNfUnet3D(**ctor).eval()
    net.load_state_dict(G.synth_sd(), strict=True)
    net = net.cuda()
    x, t, cond, _, _ = G.clip("odd")
    out = run(net, x, t, cond)
    with torch.no_grad():
        ref = O.unet_forward(G.synth_sd(), O.UnetCfg(win_width=8), x, t, cond)
        ref40 = O.unet_forward(G.synth_sd(), O.UnetCfg(), x, t, cond)
    assert G.over_tol(out, ref) <= 1.0
    assert (ref - ref40).abs().max().item() > 1e-3          # the window really matters on this clip


def test_classifier_free_guidance_sampling_matches_reference_golden():
    """N4: `ddim_sample(cond_scale=2)` — two hoisted UNet forwards per step (conditioning / all-zero null conditioning, U:879-890,
    920) — against the REAL reference's ddim_sample on the 'odd' clip (oracle/make_golden_cfg.py, 3 steps, injected noise)."""
    from dawn_pytorch_b200 import DynamicNfGaussianDiffusion
    g = np.load(os.path.join(G.ROOT, "tests", "golden", "ddim_cfg2_odd.npz"))
    steps, scale = int(g["steps"]), float(g["cond_scale"])
    net = G.cuda_net()
    D = DynamicNfGaussianDiffusion(denoise_fn=net, num_frames=40, image_size=32, sampling_timesteps=steps, timesteps=1000,
                                   loss_type='l2', use_dynamic_thres=True, null_cond_prob=0.1, ddim_sampling_eta=1.0).cuda()
    F, h, w, _ = G.CASES["odd"]
    _, fea, cond = W.synth_inputs("odd", F, h, w)
    D.update_num_frames(F)

    def noise_fn(k, shape):
        return torch.from_numpy(W.pseudo_normal(f"cfg2/noise{k}", tuple(shape)))

    img = D.ddim_sample(fea.cuda(), (1, 3, F, h, w), cond=cond.cuda(), cond_scale=scale, noise_fn=noise_fn)
    torch.cuda.synchronize()
    d = (img.cpu() - torch.from_numpy(g["sample"])).abs().max().item()
    print(f"cfg sampling (cond_scale {scale}, {steps} steps): max|d| = {d:.3e}")
    assert d < 2e-4
