"""2+ GPUs (torchrun): the ancestral DDPM loop (`p_sample_loop`) on one clip frame-sharded over the ranks — clip-wide quantile
through the all-reduced radix select, per-rank slice of one clip-wide noise tensor — eager and as replayed graph segments,
against the single-GPU loop with the same noise (asserts on rank 0).
   torchrun --nproc-per-node 2 tools/shard_ddpm_test.py"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import weights as W            # noqa: E402
from tests import gpu_common as G          # noqa: E402


def ddpm_case(net, rank, world, dev):
    """The ancestral loop under sharding: a complete T = 20 p_sample_loop on a frame-sharded clip, eagerly and as graph segments
    of 8 steps (two replays, then 4 eager steps), vs the single-GPU eager loop with the same noise."""
    import dawn_pytorch_b200.diffusion as dd
    from dawn_pytorch_b200 import DynamicNfGaussianDiffusion, DynamicNfUnet3D
    T = 20
    Fg, h, w = 48 * world, 16, 16
    Fl, lo = Fg // world, rank * (Fg // world)
    x_t, fea, cond = W.synth_inputs("shardddpm", Fg, h, w)

    def make(unet):
        return DynamicNfGaussianDiffusion(denoise_fn=unet, num_frames=40, image_size=32, sampling_timesteps=None, timesteps=T,
                                          loss_type='l2', use_dynamic_thres=True, null_cond_prob=0.1, ddim_sampling_eta=1.0).to(dev)

    def noise_global(k):
        return x_t[0] if k < 0 else torch.from_numpy(W.pseudo_normal(f"shardddpm/noise{k}", (3, Fg, h, w)))

    D = make(net)
    net.update_num_frames(Fl)
    net.init_shard(Fl, h, w, dev)
    assert net.shard_info() == (rank, world)
    D.update_num_frames(Fl)
    one = None
    if rank == 0:
        net1 = DynamicNfUnet3D(**G.CTOR).eval()
        net1.load_state_dict(G.synth_sd(), strict=True)
        D1 = make(net1.to(dev))
        D1.update_num_frames(Fg)
        one = D1.p_sample_loop(fea.to(dev), (1, 3, Fg, h, w), cond=cond.to(dev),
                               noise_fn=lambda k, shp: noise_global(k).reshape(shp).clone())[0].cpu()
        del D1, net1
    dist.barrier()
    for use_graph in (False, True):
        dd.DDPM_SEGMENT_STEPS = 8
        out = D.p_sample_loop(fea.to(dev), (1, 3, Fl, h, w), cond=cond[:, lo:lo + Fl].contiguous().to(dev),
                              noise_fn=lambda k, shp: noise_global(k)[:, lo:lo + Fl].reshape(shp).clone(), use_graph=use_graph)[0].clone()
        parts = [torch.empty_like(out) for _ in range(world)]
        dist.all_gather(parts, out)
        full = torch.cat(parts, dim=1).cpu()
        if rank == 0:
            dmax = (full - one).abs().max().item()
            print(f"[ddpm] F={Fg} sharded x{world} p_sample_loop T={T} ({'graph, 8-step segments' if use_graph else 'eager'}): "
                  f"max|d| vs single-GPU {dmax:.2e}", flush=True)
            assert dmax < 2e-4, "sharded DDPM sampler disagrees with the single-GPU sampler"
        dist.barrier()
    # default noise: one clip-wide stream, sliced per rank
    a = D.p_sample_loop(fea.to(dev), (1, 3, Fl, h, w), cond=cond[:, lo:lo + Fl].contiguous().to(dev), seed=123)
    assert torch.isfinite(a).all()


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=dev)
    from dawn_pytorch_b200 import DynamicNfUnet3D
    net = DynamicNfUnet3D(**G.CTOR).eval()
    net.load_state_dict(G.synth_sd(), strict=True)
    ddpm_case(net.to(dev), rank, world, dev)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
