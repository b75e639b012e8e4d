"""Ancestral DDPM sampling (`p_sample_loop`, T = 1000) of one clip at the BASELINE configs[1] shape: 100 frames, 128x128 video
(32x32 latent), synthetic weights and clip.  Times the eager loop and the segmented graph replay (one 20-step graph replayed
50 times) with CUDA events and a final synchronise, and, for scale, 20 DDIM steps at the same shape.  Prints one JSON line
(also written to --out) with seconds per clip, ms per step, kernel launches per step, and the GPU name, power limit and SM
clock read in the same run.

  python tools/bench_ddpm.py [--frames 100] [--latent 32] [--timesteps 1000] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from oracle import weights as W                                     # noqa: E402
from tests import gpu_common as G                                   # noqa: E402


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30)
        name, plim, sm, smax = [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")]
        return dict(gpu=name, power_limit_w=float(plim), sm_clock_mhz=int(sm), sm_clock_max_mhz=int(smax))
    except Exception as e:                                            # noqa: BLE001
        return dict(gpu=torch.cuda.get_device_name(), power_limit_w=None, sm_clock_mhz=None, error=f"nvidia-smi: {e}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--latent", type=int, default=32)
    ap.add_argument("--timesteps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_ddpm measures on a CUDA device"
    import dawn_pytorch_b200.diffusion as dd
    from dawn_pytorch_b200 import DynamicNfGaussianDiffusion
    F, S, T, K = a.frames, a.latent, a.timesteps, dd.DDPM_SEGMENT_STEPS
    net = G.cuda_net()
    x_t, fea, cond = W.synth_inputs("bench_ddpm", F, S, S)
    fea, cond = fea.cuda(), cond.cuda()
    shape = (1, 3, F, S, S)

    def diffusion(sampling_timesteps):
        D = DynamicNfGaussianDiffusion(denoise_fn=net, num_frames=F, image_size=S, sampling_timesteps=sampling_timesteps, timesteps=T,
                                       loss_type='l2', use_dynamic_thres=True, null_cond_prob=0.1, ddim_sampling_eta=1.0).cuda()
        D.update_num_frames(F)
        return D

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    D = diffusion(None)
    seg = list(reversed(range(T)))[:K]
    torch.manual_seed(0)
    D.p_sample_loop(fea, shape, cond=cond, times=seg)                  # warm-up: one segment's worth of eager steps
    fwd_launches = net.last_launch_count()
    torch.manual_seed(0)
    ms_eager, x_eager = timed(lambda: D.p_sample_loop(fea, shape, cond=cond)[0].clone())
    torch.manual_seed(0)
    ms_graph_first, _ = timed(lambda: D.p_sample_loop(fea, shape, cond=cond, use_graph=True))     # includes the capture
    nodes = net.last_launch_count()
    torch.manual_seed(0)
    ms_graph, x_graph = timed(lambda: D.p_sample_loop(fea, shape, cond=cond, use_graph=True)[0].clone())
    state = gpu_state()

    Dd = diffusion(20)
    Dd.ddim_sample(fea, shape, cond=cond)                               # warm-up
    ms_ddim, _ = timed(lambda: Dd.ddim_sample(fea, shape, cond=cond))
    Dd.ddim_sample(fea, shape, cond=cond, use_graph=True)               # capture
    ms_ddim_graph, _ = timed(lambda: Dd.ddim_sample(fea, shape, cond=cond, use_graph=True))

    res = dict(
        workload=f"p_sample_loop T={T}, {F} frames, {S}x{S} latent ({4 * S}x{4 * S} video), 1 clip, synthetic weights",
        eager_s_per_clip=round(ms_eager / 1e3, 3), eager_ms_per_step=round(ms_eager / T, 3),
        graph_s_per_clip=round(ms_graph / 1e3, 3), graph_ms_per_step=round(ms_graph / T, 3),
        graph_first_clip_incl_capture_s=round(ms_graph_first / 1e3, 3), segment_steps=K, graph_replays=T // K, eager_remainder=T % K,
        graph_nodes_per_step=nodes / K, forward_launches_per_step=fwd_launches,
        ddim20_eager_ms_per_step=round(ms_ddim / 20, 3), ddim20_graph_ms_per_step=round(ms_ddim_graph / 20, 3),
        graph_vs_eager_maxabs=float((x_graph - x_eager).abs().max()), sample_finite=bool(torch.isfinite(x_graph).all()),
        **state)
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
