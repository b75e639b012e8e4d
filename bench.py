"""bench.py — denoising-steps/sec of the DAWN denoising UNet on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port) on host cores

A "step" is one UNet forward (`forward_with_cond_scale`, cond_scale=1) over a whole synthetic clip:
BASELINE configs[2] = 200 frames of a 64x64 latent (256x256 video), windowed temporal attention.
N > 1 (torchrun, one rank per GPU): ONE clip of 200*N frames is sharded by contiguous frame range, 200 frames per
GPU (weak scaling), exactly: +-40-frame halo exchange before each of the 10 temporal attentions (ncclSend/Recv) and a
16-double all-reduce per GroupNorm (40 per step) inside the library; `value` counts 200-frame-clip equivalents
(frames denoised per second / 200).  `--replicas` runs one independent 200-frame clip per GPU instead.
`--dump-outputs DIR` writes the eps of the last timed step as DIR/eps.npy (DIR/eps_rank<r>.npy per rank when N > 1); the inputs
are seeded, so two builds run with the same arguments can be compared output for output.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                     # the tree may be read-only: no __pycache__ for the project's modules

F_CLIP, H_LAT, W_LAT = 200, 64, 64
METRIC = "denoising-steps/sec (200-frame 256^2 clip)"
DUMP_BYTES = 64 << 20                              # --dump-outputs: at most this much over all ranks
CTOR = dict(dim=64, cond_dim=1032, cond_aud=1024, cond_pose=6, cond_eye=2, num_frames=40, channels=275,
            out_grid_dim=2, out_conf_dim=1, dim_mults=(1, 2, 4, 8), use_hubert_audio_cond=True,
            learn_null_cond=False, use_final_activation=False, use_deconv=True, padding_mode="zeros", win_width=40)
CPU_SAMPLE_FRAMES = 16


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], tensor=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured (MEASURED_PEAKS.json, bf16 sustained)")
    return dict(hbm=6650.0, tensor=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def log(msg):
    print(f"[bench +{time.perf_counter() - T_START:7.1f}s] {msg}", file=sys.stderr, flush=True)


def dump_output(path, name, t, budget):
    """`t` as path/<name>.npy in float32.  Above `budget` bytes only every k-th element of the flattened tensor is written: a fixed
    sample, the same on every run."""
    a = t.detach().float().cpu().numpy()
    k = -(-a.nbytes // budget)
    if k > 1:
        a = a.reshape(-1)[::k]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, name + ".npy"), a)
    log(f"wrote {os.path.join(path, name + '.npy')}: {a.shape} float32" + (f" (1 in {k} elements)" if k > 1 else ""))


T_START = time.perf_counter()


def host_threads():
    """CPU threads this process may really use: min(affinity, cgroup quota); os.cpu_count() alone can be the
    whole host and oversubscribing a quota-limited container makes OpenMP crawl."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, per = f.read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, min(n, 64))


def synth_clip(seed):
    g = torch.Generator().manual_seed(seed)
    x_t = torch.randn(3, F_CLIP, H_LAT, W_LAT, generator=g)
    fea = torch.relu(torch.randn(272, H_LAT, W_LAT, generator=g))      # post-ReLU LFG / bbox features are non-negative
    cond = torch.randn(F_CLIP, 1032, generator=g)
    return x_t, fea, cond


def synth_state_dict():
    """Deterministic synthetic weights of the reference architecture (oracle/weights.py over the committed 900-key schema):
    the same state_dict feeds the CUDA arm and the CPU arm, and building it does not touch the product package."""
    from oracle import weights as W
    with open(os.path.join(ROOT, "tests", "golden", "state_dict_schema.json")) as f:
        schema = [(n, tuple(sh)) for n, sh in json.load(f)["entries"]]
    return W.synth_state_dict(schema)


def cpu_cfg1_run(state_dict, steps=5, warmup=3):
    """BASELINE.md section 4: BASELINE configs[0] (16 frames, 32x32 latent) on the host cores, NOT extrapolated:
    3 warm-ups + 5 timed forwards of the oracle port, median."""
    from oracle import unet_oracle as O
    from oracle import weights as W
    cores = host_threads()
    torch.set_num_threads(cores)
    x_t, fea, cond = W.synth_inputs("cfg1", 16, 32, 32)
    x = torch.cat([x_t, fea.unsqueeze(2).expand(-1, -1, 16, -1, -1)], dim=1).contiguous()
    t = torch.full((1,), 500, dtype=torch.long)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            O.unet_forward(state_dict, O.UnetCfg(), x, t, cond)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    sec = statistics.median(times)
    return {"workload": "configs[0]: 16 frames, 32x32 latent, one UNet forward", "s_per_step": sec, "steps_per_s": 1.0 / sec,
            "cores": cores, "kind": "port", "timed": steps, "warmup": warmup}


def cpu_baseline_run(state_dict, steps, warmup):
    """The reference's algorithm on the host cores: oracle port (the reference itself is Python and does not
    travel to this box).  Bounded sample: the first CPU_SAMPLE_FRAMES frames of the same 64x64-latent workload;
    per-frame cost is scaled to the 200-frame clip."""
    from oracle import unet_oracle as O
    cores = host_threads()
    torch.set_num_threads(cores)
    log(f"cpu baseline: oracle port on {cores} threads, {CPU_SAMPLE_FRAMES} frames sample")
    x_t, fea, cond = synth_clip(1)
    Fs = CPU_SAMPLE_FRAMES
    x = torch.cat([x_t[:, :Fs], fea.unsqueeze(1).expand(-1, Fs, -1, -1)], dim=0)[None].contiguous()
    c = cond[None, :Fs].contiguous()
    t = torch.full((1,), 500, dtype=torch.long)
    cfg = O.UnetCfg()
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            O.unet_forward(state_dict, cfg, x, t, c)
            log(f"  cpu forward {i}: {time.perf_counter() - t0:.2f} s")
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    sec = statistics.median(times)
    value = (1.0 / sec) * (Fs / F_CLIP)
    return dict(value=value, unit="steps/s", cores=cores, kind="port",
                sample=f"{Fs} of {F_CLIP} frames at 64x64 latent, median of {steps} forwards ({sec:.2f} s each), scaled by {Fs}/{F_CLIP}"), sec


def clip_pipeline(rank, world, dev, dist, clips=2, steps=20, chunk=50):
    """BASELINE configs[4] pipeline, one clip end to end from HOST buffers: source encoder + bbox embedding, `steps` DDIM steps over
    the CUDA UNet replayed as ONE CUDA graph, batched LFG decode of the sampled flow/occlusion maps into frames, D2H of the frames.
    N = 1: a 200-frame 256x256 clip (configs[2]'s clip).  N > 1: 100 frames per GPU as configs[3]/[4] state (400 f on 4, 800 f on 8):
    the sampler runs frame-sharded (halo exchange, GroupNorm and quantile reductions), every rank decodes its own frames (the decoder
    is per-frame: no exchange).  Random-init weights of the reference architecture, synthetic inputs.  Times are CUDA-event /
    wall-clock maxima over ranks; the first clip (graph capture, allocations) is not timed."""
    from dawn_pytorch_b200 import FlowDiffusion
    torch.manual_seed(0)
    Fl, S = (F_CLIP if world == 1 else 100), 4 * H_LAT
    Fg = Fl * world
    m = FlowDiffusion(sampling_timesteps=steps, pose_dim=6, win_width=40).to(dev)
    m.update_num_frames(Fl)
    if world > 1:
        m.unet.init_shard(Fl, H_LAT, W_LAT, dev)
    g = torch.Generator().manual_seed(7)
    img_h = torch.rand(1, 3, S, S, generator=g).pin_memory()
    hub_h = torch.randn(1, Fg, 1024, generator=g)[:, rank * Fl:(rank + 1) * Fl].contiguous().pin_memory()
    pose_h = (torch.randn(1, 6, Fg, generator=g) * 0.2)[:, :, rank * Fl:(rank + 1) * Fl].contiguous().pin_memory()
    eye_h = torch.rand(1, 2, Fg, generator=g)[:, :, rank * Fl:(rank + 1) * Fl].contiguous().pin_memory()
    bbox = torch.tensor([[0.3 * S, 0.7 * S, 0.25 * S, 0.8 * S, S, S]]).unsqueeze(-1).repeat(1, 1, Fl)
    out_h = torch.empty((Fl, 3, S, S), dtype=torch.float32).pin_memory()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    stage, wall = [], []
    for clip in range(clips + 1):
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        img, hub, pose, eye = img_h.to(dev, non_blocking=True), hub_h.to(dev, non_blocking=True), pose_h.to(dev, non_blocking=True), eye_h.to(dev, non_blocking=True)
        ev[0].record()
        fea = m.generator.compute_fea(img)
        mask = m.face_loc_emb(m.generate_bbox_mask(bbox.to(dev), size=S))
        cond = torch.cat([hub, pose.permute(0, 2, 1), eye.permute(0, 2, 1)], dim=-1)      # (1, F, 1024 + 6 + 2), synthetic deltas (FD:350)
        ev[1].record()
        pred = m.diffusion.ddim_sample(torch.cat([fea, mask], dim=1), (1, 3, Fl, H_LAT, W_LAT), cond=cond, use_graph=True, seed=1234 + clip)
        ev[2].record()
        for i in range(0, Fl, chunk):
            out_h[i:i + chunk].copy_(m.generator.decode_sample(img, pred[0][:, i:i + chunk].contiguous()), non_blocking=True)
        ev[3].record()
        torch.cuda.synchronize()
        if clip > 0:
            wall.append(time.perf_counter() - t0)
            stage.append([ev[i].elapsed_time(ev[i + 1]) for i in range(3)])
    t = torch.tensor([statistics.median(wall)] + [statistics.median(x) for x in zip(*stage)], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall_s, prep, samp, dec = [float(v) for v in t]
    finite = bool(torch.isfinite(out_h).all())
    del m
    torch.cuda.empty_cache()
    return {"workload": (f"configs[4] pipeline: one {Fg}-frame 256x256 clip, {steps} DDIM steps (one CUDA graph) + batched LFG decode, "
                         + ("single GPU" if world == 1 else f"{Fl} frames per GPU, sampler frame-sharded x{world}, decode per rank")),
            "clips_per_s": 1.0 / wall_s, "frames_per_s": Fg / wall_s, "ms_per_clip_e2e": wall_s * 1e3,
            "stage_ms": {"source_encoder_and_bbox": prep, "sampling": samp, "sampling_per_step": samp / steps, "lfg_decode_and_d2h": dec},
            "h2d_bytes_per_clip": int(img_h.numel() + hub_h.numel() + pose_h.numel() + eye_h.numel()) * 4, "d2h_bytes_per_clip": int(out_h.numel()) * 4,
            "timed_clips": clips, "finite": finite}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--replicas", action="store_true", help="N > 1: independent clips per GPU instead of one frame-sharded clip")
    ap.add_argument("--no-clip", action="store_true", help="skip the whole-clip pipeline (configs[4]) measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the eps of the last timed step as DIR/eps.npy (float32)")
    ap.add_argument("--cpu-baseline-worker", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the CUDA path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    warmup = max(args.warmup, 3)

    sd_cpu = synth_state_dict()                   # synthetic weights of the reference architecture (no checkpoint is reachable offline)
    config = {"workload": "configs[2]: 256x256 video = 64x64 latent, 200 frames, windowed (+-40) temporal attention, 1 UNet forward per step",
              "frames": F_CLIP * (1 if (args.gpus == 1 or args.replicas) else args.gpus), "latent": [H_LAT, W_LAT],
              "parallelism": ("single GPU" if args.gpus == 1 else
                              f"replicas x{args.gpus} (one 200-frame clip per GPU, no collective)" if args.replicas else
                              f"exact frame sharding x{args.gpus}: one {F_CLIP * args.gpus}-frame clip, {F_CLIP} frames/GPU; per step 10 halo "
                              "exchanges (ncclSend/Recv of 40 boundary frames) + 40 GroupNorm all-reduces (16 fp64) over NVLink"),
              "l2": "per-step working set ~7 GB >> 126 MB L2 (inputs larger than L2, no explicit flush)"}

    if args.cpu_baseline_worker:
        cb, _ = cpu_baseline_run(sd_cpu, 3, 1)
        cb["cfg1"] = cpu_cfg1_run(sd_cpu)
        print(json.dumps(cb))
        return
    if args.impl == "reference":
        # the reference's algorithm on the host cores (oracle port; the product package is never imported on this arm)
        if rank != 0:
            return
        steps, warmup = args.steps, max(1, min(args.warmup, 5))
        cb, sec = cpu_baseline_run(sd_cpu, steps, warmup)
        cb["cfg1"] = cpu_cfg1_run(sd_cpu)
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "steps/s", "n_gpus": args.gpus,
                "steps": steps, "warmup": warmup, "ms_per_step": 1000.0 / cb["value"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    from dawn_pytorch_b200 import DynamicNfUnet3D
    net = DynamicNfUnet3D(**CTOR).eval()
    net.load_state_dict(sd_cpu, strict=True)
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    net = net.to(dev)
    sharded = world > 1 and not args.replicas
    x_t, fea, cond = synth_clip(1 + rank)
    if sharded:                                   # every rank needs the same per-clip features; frames differ per rank
        fea = synth_clip(1)[1]
    net.update_num_frames(F_CLIP)
    if sharded:
        net.init_shard(F_CLIP, H_LAT, W_LAT, dev)
    xt_d, fea_d, cond_d = x_t.to(dev), fea.to(dev), cond.to(dev)
    t_d = torch.full((1,), 500, dtype=torch.long, device=dev)
    out_d = torch.empty((3, F_CLIP, H_LAT, W_LAT), device=dev)
    net.set_clip_invariants(fea_d, cond_d)
    log("module ready, clip invariants set")

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    # ---------------- device-resident throughput (inputs already in HBM)
    for _ in range(warmup):
        net.forward_x3(xt_d, t_d, out_d)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    net.profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        net.forward_x3(xt_d, t_d, out_d)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    prof = net.profile_read()
    net.profile(False)
    launches = net.last_launch_count() * args.steps
    clocks = sampler.stop() if rank == 0 else None
    if dist is not None:
        tt = torch.tensor([ms_total], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total = float(tt.item())
    ms_per_step = ms_total / args.steps
    value = args.gpus * 1000.0 / ms_per_step
    if args.dump_outputs:                         # out_d holds the eps of the last timed step
        dump_output(args.dump_outputs, "eps" if world == 1 else f"eps_rank{rank}", out_d, DUMP_BYTES // world)
    comm = None
    if sharded:
        # stream time spent in the sharding collectives (CUDA events around them on the compute stream: they are serialised with the
        # kernels, so all of it is exposed; includes waiting for the slowest rank), max over ranks
        cm = torch.tensor([prof["comm_allreduce"]["ms"], prof["comm_halo"]["ms"]], device=dev, dtype=torch.float64)
        cmin = cm.clone()
        dist.all_reduce(cm, op=dist.ReduceOp.MAX)
        dist.all_reduce(cmin, op=dist.ReduceOp.MIN)
        # max over ranks includes the time the lightly loaded edge ranks (one halo) wait for the interior ranks (two halos: the critical
        # path); min over ranks is what the collectives cost the slowest rank itself
        comm = {"allreduce_ms": float(cm[0]) / args.steps, "halo_ms": float(cm[1]) / args.steps,
                "exposed_ms": float(cm[0] + cm[1]) / args.steps,
                "allreduce_ms_min_rank": float(cmin[0]) / args.steps, "halo_ms_min_rank": float(cmin[1]) / args.steps,
                "allreduce_calls_per_step": prof["comm_allreduce"]["count"] // args.steps, "halo_exchanges_per_step": prof["comm_halo"]["count"] // args.steps,
                "allreduce_impl": "one kernel over NVLink peer memory (cudaIpc mailboxes)" if os.environ.get("DAWN_P2P", "1") != "0" else "ncclAllReduce",
                "halo_impl": "pack copy + grouped ncclSend/ncclRecv with the two neighbours"}
    log(f"device-resident: {ms_per_step:.2f} ms/step")

    # ---------------- end to end through the C-ABI with HOST buffers (H2D inputs + D2H eps every step)
    xt_h, fea_h, cond_h = x_t.pin_memory(), fea.pin_memory(), cond.pin_memory()
    out_h = torch.empty((3, F_CLIP, H_LAT, W_LAT), dtype=torch.float32).pin_memory()
    for _ in range(2):
        net.forward_host(xt_h, fea_h, cond_h, 500, out_h)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        net.forward_host(xt_h, fea_h, cond_h, 500, out_h)       # returns after the result is on the host
    barrier()
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        tt = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s = float(tt.item())
    log(f"e2e: {e2e_s / args.steps * 1e3:.2f} ms/step")
    h2d = (xt_h.numel() + fea_h.numel() + cond_h.numel()) * 4 + 8
    d2h = out_h.numel() * 4
    e2e = {"value": args.gpus * args.steps / e2e_s, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "note": "dawn_unet_forward_host: per step H2D of x_t+fea+cond+t, clip-invariant tables rebuilt, forward, D2H of eps"}
    clip = None
    if not args.no_clip and not args.replicas:
        try:
            del out_h
            clip = clip_pipeline(rank, world, dev, dist)
            log(f"clip pipeline: {clip['ms_per_clip_e2e']:.1f} ms per clip")
        except Exception as e:  # noqa: BLE001
            clip = {"error": f"{type(e).__name__}: {e}"[:300]}
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---------------- BASELINE configs[0] (16 frames, 32x32 latent), device-resident, for the un-extrapolated CPU comparison
    cfg1_gpu = None
    if world == 1:
        from oracle import weights as W
        x1, f1, c1 = W.synth_inputs("cfg1", 16, 32, 32)
        net.update_num_frames(16)
        net.set_clip_invariants(f1[0].to(dev), c1[0].to(dev))
        x1d, o1d = x1[0].to(dev), torch.empty((3, 16, 32, 32), device=dev)
        for _ in range(5):
            net.forward_x3(x1d, t_d, o1d)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(20):
            net.forward_x3(x1d, t_d, o1d)
        e1.record()
        torch.cuda.synchronize()
        cfg1_gpu = {"workload": "configs[0]: 16 frames, 32x32 latent, one UNet forward (device-resident)",
                    "ms_per_step": e0.elapsed_time(e1) / 20, "steps_per_s": 20e3 / e0.elapsed_time(e1), "timed": 20, "warmup": 5}
        log(f"cfg1 on the GPU: {cfg1_gpu['ms_per_step']:.3f} ms/step")

    # ---------------- roofline of the dominant kernel, live CUDA-event times (category timers inside the library)
    pk = peaks()
    total_kernel_ms = sum(v["ms"] for v in prof.values())
    breakdown = {k: {"ms_per_step": v["ms"] / args.steps, "share": v["ms"] / total_kernel_ms if total_kernel_ms else 0,
                     "launches_per_step": v["count"] // args.steps,
                     "alg_tflops": (v["flops"] / (v["ms"] * 1e-3) / 1e12) if v["ms"] > 0 and v["flops"] > 0 else None,
                     "alg_gbs": (v["bytes"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] > 0 and v["bytes"] > 0 else None}
                 for k, v in prof.items() if v["count"] > 0}
    traffic = {}
    import glob
    tfiles = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
    tpath = tfiles[-1] if tfiles else ""             # newest committed ncu --set full capture (same kernels as this HEAD: profiles/README.md)
    if tpath and os.path.exists(tpath):              # dram bytes per launch of exactly these launches
        with open(tpath) as f:
            traffic = json.load(f)

    def tensor_view(cat, kernel, note):
        v = prof[cat]
        n = max(v["count"], 1)
        tf = v["flops"] / (v["ms"] * 1e-3) / 1e12 if v["ms"] > 0 else 0.0
        return {"kernel": kernel, "bound": "tensor", "achieved": tf, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": tf / pk["tensor"],
                "traffic": traffic.get(cat, {}).get("dram_bytes_per_launch"), "peak_source": pk["src"],
                "alg_flops_per_launch": v["flops"] / n, "alg_bytes_per_launch": v["bytes"] / n, "avg_launch_ms": v["ms"] / n,
                "launches_per_step": v["count"] // args.steps, "share_of_step": v["ms"] / total_kernel_ms if total_kernel_ms else 0,
                "note": note}

    split_note = ("algorithmic flops (2*MAC, counted once); every product is issued as 3 fp16 MMAs (hi*hi + hi*lo + lo*hi) for "
                  "fp32-level parity, so the attainable fraction of the bf16 peak is 1/3")
    # the kernel with the largest share of the step: fused per-pixel temporal attention at level 0 (4096 px x 200 f x 64 ch)
    roofline = tensor_view("temporal_fused_l0",
                           "temporal_tc_kernel @ level 0 (LayerNorm + QKV projection + rotary + banded softmax attention + out-projection "
                           "+ residual per pixel sequence; tcgen05 kind::f16 FP16x3, TMEM accumulators, P from TMEM)",
                           split_note + "; flops = QKV 80.5 + attention 61 + out-proj 26.8 GFLOP per launch")
    # second view: the tcgen05 halo-tile 3x3 conv (64 -> 64 channels, 819 200 px), the largest tcgen05 kernel
    roofline_conv3 = tensor_view("conv3x3_l0", "tc_conv3_kernel<64> @ level 0 (halo-tile tcgen05 3x3 conv 64->64 ch, FP16x3 kind::f16, TMEM accumulators)",
                                 split_note)
    # third view: an HBM-bound kernel of the path — SiLU(GroupNorm(y)) + residual (reads y and the residual, writes the block output)
    gna = prof["gn_apply"]
    gna_gbs = gna["bytes"] / (gna["ms"] * 1e-3) / 1e9 if gna["ms"] > 0 else 0.0
    roofline_hbm = {"kernel": "gn_apply_kernel (SiLU(GroupNorm(y)) + residual, all levels)", "bound": "hbm", "achieved": gna_gbs, "peak": pk["hbm"],
                    "unit": "GB/s", "frac": gna_gbs / pk["hbm"], "traffic": traffic.get("gn_apply_l0", {}).get("dram_bytes_per_launch"),
                    "launches_per_step": gna["count"] // args.steps, "share_of_step": gna["ms"] / total_kernel_ms if total_kernel_ms else 0}
    # whole-step roofline for context (BASELINE.md: F_alg 3834.6 GFLOP, B_alg 22.9 GB per step at this config)
    step_roof = {"F_alg_gflop": 3834.6, "B_alg_gb": 22.9,
                 "t_roof_ms": max(3834.6e9 / (pk["tensor"] * 1e12), 22.9e9 / (pk["hbm"] * 1e9)) * 1e3}
    step_roof["frac"] = step_roof["t_roof_ms"] / ms_per_step

    cpu_baseline = None
    if args.gpus == 1 and not args.no_cpu_baseline:
        # time-boxed child process: a slow or wedged host must not take the GPU numbers down with it
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-baseline-worker"], capture_output=True,
                               text=True, timeout=240)
            cpu_baseline = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:  # noqa: BLE001
            cpu_baseline = {"value": None, "unit": "steps/s", "cores": host_threads(), "kind": "port",
                            "sample": f"not measured: {type(e).__name__}"}
        log(f"cpu baseline: {cpu_baseline}")

    line = {"metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config, "roofline": roofline, "roofline_conv3_view": roofline_conv3, "roofline_hbm_view": roofline_hbm, "step_roofline": step_roof, "cpu_baseline": cpu_baseline,
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "comm": comm, "clip": clip, "cfg1": cfg1_gpu, "breakdown": breakdown}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
