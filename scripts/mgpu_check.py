"""Multi-GPU parity check (run under torchrun): the CFG/view-sharded forward and sampler against the same rank's
un-sharded run. python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 scripts/mgpu_check.py"""
import os
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from panfusion_b200 import sd2_unet  # noqa: E402
from panfusion_b200.mvgen import MultiViewBaseModel  # noqa: E402
from panfusion_b200.sampler import PanFusionSampler  # noqa: E402

TINY = dict(sd2_unet.SD2_CONFIG, block_out_channels=(64, 128, 128, 128), attention_heads=(1, 2, 2, 2), cross_attention_dim=64)


def build(dev, parallel):
    torch.manual_seed(0)
    u1 = sd2_unet.build_synthetic(TINY, seed=1)
    u2 = sd2_unet.build_synthetic(TINY, seed=2)
    torch.manual_seed(3)
    m = MultiViewBaseModel(u1, u2, compute_dtype=torch.float16)
    g = torch.Generator().manual_seed(4)
    with torch.no_grad():
        for name, p in sorted(m.named_parameters()):
            if "cp_blocks" in name and float(p.abs().sum()) == 0.0:
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
    m = m.to(dev).eval()
    if parallel:
        m.set_view_parallel(dist.group.WORLD)
    m.prepare(dev, torch.float16)
    return m


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    modes = [m == "1" for m in os.environ.get("MGPU_GRAPH_MODES", "0,1").split(",")]

    def log(msg):  # progress on stderr: the last line of each rank shows where a hung or failed run stopped
        print(f"[mgpu rank {rank}] {msg}", file=sys.stderr, flush=True)

    log("init")
    dist.init_process_group("nccl", device_id=dev)
    log("nccl up")
    views = 8
    g = torch.Generator().manual_seed(0)
    import numpy as np
    theta = torch.tensor(np.rad2deg(np.linspace(0, 2 * np.pi, views, endpoint=False)), dtype=torch.float32)[None]
    cams = dict(FoV=torch.full((1, views), 90.0), theta=theta, phi=torch.zeros(1, views))
    pano = torch.randn(1, 1, 4, 16, 32, generator=g).to(dev)
    lat = torch.randn(1, views, 4, 16, 16, generator=g).to(dev)
    null, text = torch.randn(1, 1, 77, 64, generator=g), torch.randn(1, 1, 77, 64, generator=g)
    pano_prompt = torch.cat([null, text]).to(dev)
    prompt = torch.cat([null.repeat(1, views, 1, 1), text.repeat(1, views, 1, 1)]).to(dev)
    ok = True
    for graph in modes:
        outs = []
        for parallel in (False, True):
            log(f"build graph={graph} parallel={parallel}")
            model = build(dev, parallel)
            s = PanFusionSampler(model, use_cuda_graph=graph)
            log("denoise")
            outs.append(s.denoise(lat, pano, prompt, pano_prompt, cams, num_steps=9, rotate_back=False))
            torch.cuda.synchronize()
            log("done, barrier")
            dist.barrier()
        d_lat = (outs[0][0] - outs[1][0]).abs().max().item()
        d_pano = (outs[0][1] - outs[1][1]).abs().max().item()
        scale = outs[0][0].abs().max().item()
        # bit-identical with PF_SPLIT_K=0; the default M-dependent split-K partition changes fp32 summation order only
        from panfusion_b200 import ops
        tol = float(os.environ.get("MGPU_TOL", "2e-3" if ops.SPLIT_K else "0"))
        good = d_lat <= tol * scale and d_pano <= tol * scale
        ok = ok and good
        if rank == 0:
            print(f"[mgpu] world={world} graph={graph}: |sharded - single| latents {d_lat:.3e} pano {d_pano:.3e} "
                  f"(scale {scale:.2f}) {'OK' if good else 'MISMATCH'}", flush=True)
    if rank == 0 and os.environ.get("PF_FORCE_IPC_FAIL", "0") != "0":
        assert model._par.device_gather is False, "the forced IPC failure must have switched the transport to NCCL"
        print("[mgpu] transport fell back to NCCL as requested by PF_FORCE_IPC_FAIL", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
