#!/usr/bin/env python
"""Benchmark of the PanFusion denoise hot path (BASELINE.json metric: denoise-steps/sec, 512x1024 pano + 8x512^2
views, CFG batch 2, bf16, 50-step DDIM schedule).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --steps K --warmup W     # the reference algorithm's CPU path (oracle port)

One "step" = one iteration of the reference loop models/pano/PanFusion.py:146-162: rotate, CFG-batched
MultiViewBaseModel.forward (7 EPPA fusions), CFG combine, two DDIM updates. Prints ONE JSON line (rank 0).
`--dump-outputs DIR` writes the view and panorama latents after the last timed step as DIR/<name>.npy (float32); the
inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

# SURVEY.md App. C (algorithmic, 2*MAC, un-padded widths); c1 here = 2 views WITH CFG (2x the survey's no-CFG C1)
FLOPS_PER_STEP = {"c2": 17.733e12, "c1": 3.669e12, "c4": 64.084e12, "c5": 19.060e12}
METRIC = "denoise-steps/sec (512x1024 pano + 8x512^2 views, 50-step DDIM)"
WORKLOADS = {
    # name: (views m, pano latent HxW, pers latent hxw, CFG)
    "c2": dict(m=8, pano_hw=(64, 128), pers_hw=(64, 64), cfg=True,
               desc="512x1024 pano + 8x512x512 views, CFG batch 2, 50-step DDIM (BASELINE configs[1])"),
    "c1": dict(m=2, pano_hw=(64, 128), pers_hw=(64, 64), cfg=True,
               desc="512x1024 pano + 2x512x512 views, CFG batch 2 (reduced-view parity config)"),
    "c4": dict(m=20, pano_hw=(128, 256), pers_hw=(64, 64), cfg=True, cameras="icosahedron",
               desc="1024x2048 pano + 20x512x512 icosahedron views, CFG batch 2 (BASELINE configs[3])"),
    "c5": dict(m=8, pano_hw=(64, 128), pers_hw=(64, 64), cfg=True, layout_cond=True,
               desc="512x1024 pano + 8x512x512 views + panorama ControlNet (layout condition), CFG batch 2 "
                    "(BASELINE configs[4])"),
}


def icosahedron_cameras():
    """20 face-centre cameras of a regular icosahedron (utils/pano.py:34-71): two rings of 5 at +-phi_a (offset by
    half a step) and two at +-phi_b; degrees."""
    import numpy as np
    r_circ, r_in, r_mid = np.sin(2 * np.pi / 5), np.sqrt(3) / 12 * (3 + np.sqrt(5)), np.cos(np.pi / 5)
    step = 2 * np.pi / 5
    phi_a = np.pi / 2 - np.arccos(r_in / r_circ)
    phi_b = phi_a - 2 * np.arccos(r_in / r_mid)
    theta, phi = [], []
    for ring, (p, off) in enumerate(((phi_a, step / 2), (phi_b, step / 2), (-phi_b, 0.0), (-phi_a, 0.0))):
        for k in range(5):
            theta.append(-np.pi + off + k * step)
            phi.append(p)
    return np.rad2deg(np.array(theta)), np.rad2deg(np.array(phi))


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is None:
            return
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.flush()
        self.f.seek(0)
        self.rows = [l.strip().split(", ") for l in self.f.read().splitlines() if l.strip()]
        self.f.close()
        os.unlink(self.f.name)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(n)
            except (ValueError, IndexError):
                continue
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=mx or None, reasons=sorted(reasons),
                    samples=len(sm))


def synthetic_inputs(wl, ctx_dim, device, sampler, seed=0):
    """SURVEY.md §8(d): seed 0, pano latent N(0,1), view latents = init_noise's e2p-nearest of it, text/null
    embeddings N(0,1), horizon cameras, FoV 90."""
    import numpy as np
    m = wl["m"]
    g = torch.Generator().manual_seed(seed)
    if wl.get("cameras") == "icosahedron":
        theta, phi = icosahedron_cameras()
    else:
        theta = np.rad2deg(np.linspace(0, 2 * np.pi, m, endpoint=False))  # utils/pano.py:28-31
        phi = np.zeros(m)
    cams = dict(FoV=torch.full((1, m), 90.0), theta=torch.tensor(theta, dtype=torch.float32)[None],
                phi=torch.tensor(phi, dtype=torch.float32)[None])
    pano = torch.randn(1, 1, 4, *wl["pano_hw"], generator=g)
    text = torch.randn(1, 1, 77, ctx_dim, generator=g)
    null = torch.randn(1, 1, 77, ctx_dim, generator=g)
    pano_prompt = torch.cat([null, text])                                              # PanFusion.py:135-138
    prompt = torch.cat([null.repeat(1, m, 1, 1), text.repeat(1, m, 1, 1)])             # copy_pano_prompt
    out = dict(cams=cams, pano=pano, prompt=prompt, pano_prompt=pano_prompt)
    if wl.get("layout_cond"):  # layout image at pixel resolution (8x the latent), values in [0, 1]
        out["pano_layout_cond"] = torch.rand(1, 1, 3, wl["pano_hw"][0] * 8, wl["pano_hw"][1] * 8, generator=g)
    return out


def dump_outputs(out_dir, latents, pano_latent):
    """What the caller of the denoise loop receives after the last timed step: the view latents [1, m, 4, h, w] and the
    panorama latent [1, 1, 4, H, W], as float32 .npy files."""
    import numpy as np
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, t in (("latents", latents), ("pano_latent", pano_latent)):
        np.save(d / f"{name}.npy", t.detach().to("cpu", torch.float32).numpy())


# ------------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch.distributed as dist
    from panfusion_b200 import _lib, geometry, ops, sd2_unet
    from panfusion_b200.mvgen import MultiViewBaseModel
    from panfusion_b200.sampler import PanFusionSampler

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.check(_lib.lib().pf_check_device())
    pk = peaks()
    wl = WORKLOADS[args.workload]
    dtype = torch.bfloat16

    # random-init SD-2 architecture, seeded (no checkpoints offline); EPPA zero-init tensors redrawn N(0, 0.02^2)
    unet = sd2_unet.build_synthetic(seed=1, device=dev)
    pano_unet = sd2_unet.build_synthetic(seed=2, device=dev)
    torch.manual_seed(3)
    pano_cn = sd2_unet.build_synthetic_controlnet(seed=5, device=dev) if wl.get("layout_cond") else None
    model = MultiViewBaseModel(unet, pano_unet, pano_cn=pano_cn, compute_dtype=dtype).to(dev).eval()
    g = torch.Generator(device=dev).manual_seed(4)
    with torch.no_grad():
        for name, p in sorted(model.named_parameters()):
            if "cp_blocks" in name and float(p.abs().sum()) == 0.0:
                p.copy_(torch.randn(p.shape, generator=g, device=dev) * 0.02)
    if world > 1:
        model.set_view_parallel(dist.group.WORLD)
    model.prepare(dev, dtype)
    sampler = PanFusionSampler(model, use_cuda_graph=not args.no_graph)
    inp = synthetic_inputs(wl, 1024, dev, sampler)
    pano = inp["pano"].to(dev)
    cams_flat = {k: v.flatten(0, 1) for k, v in inp["cams"].items()}
    lat = geometry.e2p(pano.expand(-1, wl["m"], -1, -1, -1).flatten(0, 1).contiguous(), cams_flat["FoV"],
                       cams_flat["theta"], cams_flat["phi"], wl["pers_hw"], mode="nearest")[None]
    prompt, pano_prompt = inp["prompt"].to(dev), inp["pano_prompt"].to(dev)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n_sched = sampler.diff_timestep
    cond = inp["pano_layout_cond"].to(dev) if "pano_layout_cond" in inp else None
    sampler.start(lat, pano, prompt, pano_prompt, inp["cams"], pano_layout_cond=cond)
    if args.profile_one_step:
        # ncu --profile-from-start off: tables/weights warmed by 4 eager steps, then exactly one step is profiled
        sampler.use_cuda_graph = False
        for i in range(4):
            sampler.step(i)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        sampler.step(4)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        print(json.dumps({"profiled_step_launches": sampler.launches_per_step}))
        return
    # preparation (untimed, not counted as warm-up): build camera tables + capture one CUDA graph per rotation phase
    phases = 4 if sampler.rot_diff % 360 else 1
    l0 = ops.LAUNCHES
    for i in range(phases):
        sampler.step(i % n_sched)
    sync_all()
    launches_per_step = sampler.launches_per_step
    step_idx = phases
    for _ in range(args.warmup):
        sampler.step(step_idx % n_sched)
        step_idx += 1
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        e0.record()
        for _ in range(args.steps):
            sampler.step(step_idx % n_sched)
            step_idx += 1
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *sampler.finish())
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    sync_all()
    steps_per_s = args.steps / (ms / 1e3)

    # ---- end to end through the public API with HOST buffers ---------------------------------------
    # per step: pinned host -> device copies of every input of forward_cls_free (latents, pano latent, timestep,
    # both prompt embeddings), the step, device -> pinned host copy of the updated latents.
    pin = lambda t: t.detach().to("cpu").contiguous().pin_memory()
    h_lat, h_pano = pin(sampler._st["latents"]), pin(sampler._st["pano"])
    h_prompt, h_pano_prompt = pin(prompt), pin(pano_prompt)
    h_ts = pin(sampler._st["timestep"])
    h_out_lat, h_out_pano = torch.empty_like(h_lat).pin_memory(), torch.empty_like(h_pano).pin_memory()
    st = sampler._st
    h2d = sum(t.numel() * t.element_size() for t in (h_lat, h_pano, h_prompt, h_pano_prompt, h_ts))
    d2h = sum(t.numel() * t.element_size() for t in (h_out_lat, h_out_pano))

    def e2e_step(i):
        st["latents"].copy_(h_lat, non_blocking=True)
        st["pano"].copy_(h_pano, non_blocking=True)
        st["prompt"].copy_(h_prompt, non_blocking=True)
        st["pano_prompt"].copy_(h_pano_prompt, non_blocking=True)
        st["timestep"].copy_(h_ts, non_blocking=True)
        model.update_text(st["prompt"], st["pano_prompt"])  # a prompt that arrives from the host is projected again
        sampler.step(i % n_sched)
        h_out_lat.copy_(st["latents"], non_blocking=True)
        h_out_pano.copy_(st["pano"], non_blocking=True)

    for _ in range(max(3, min(args.warmup, 4))):
        e2e_step(step_idx)
        step_idx += 1
    sync_all()
    e0.record()
    for _ in range(args.steps):
        e2e_step(step_idx)
        step_idx += 1
    e1.record()
    torch.cuda.synchronize()
    ms_e2e = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())
    e2e_sps = args.steps / (ms_e2e / 1e3)

    out = None
    if world > 1:
        from panfusion_b200.parallel import pick_layout
        bsh, vsh = pick_layout(world, 2, wl["m"])
        from panfusion_b200.parallel import DEVICE_GATHER
        transport = ("device-initiated (pf_allgather_views: NVLink stores into CUDA-IPC receive buffers, inside the step's "
                     "CUDA graph)" if DEVICE_GATHER else "NCCL between graph segments")
        parallelism = (f"{bsh} CFG shards x {vsh} view shards (one process per GPU; pano branch once per CFG shard; "
                       f"{'one K|V all-gather per EPPA block + ' if vsh > 1 else ''}one eps all-gather per step, {transport})")
    else:
        parallelism = "single GPU"
    if rank == 0:
        flops = FLOPS_PER_STEP[args.workload]
        ach = steps_per_s * flops / 1e12 / world
        out = {
            "metric": METRIC, "value": round(steps_per_s, 4), "unit": "steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": wl["desc"], "views": wl["m"], "cfg_batch": 2, "pano_latent": list(wl["pano_hw"]),
                       "view_latent": list(wl["pers_hw"]), "weights": "random-init SD-2 architecture (seeded)",
                       "parallelism": parallelism,
                       "cuda_graph": not args.no_graph,
                       "l2": "working set (3.4 GB weights + activations per step) exceeds the 126 MB L2; no flush needed"},
            "clocks": clk.summary(),
            "e2e": {"value": round(e2e_sps, 4), "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "eppa_tables_mb": round(model.cp_blocks_mid.tables.nbytes() / 2 ** 20, 1),  # all 4 rotation phases, resident form
            "gpu_launches": int(launches_per_step * args.steps) if launches_per_step else int(ops.LAUNCHES - l0),
            "launches_per_step": launches_per_step,
            "roofline": {"bound": "tensor", "achieved": round(ach, 2), "peak": pk["tf_sust"], "unit": "TFLOP/s",
                         "frac": round(ach / pk["tf_sust"], 4), "traffic": None, "peak_source": pk["src"],
                         "flops_per_step": flops, "scope": "whole denoise step (dense contractions dominate)"},
        }
        if not args.skip_micro:
            out["kernels"] = micro_rooflines(dev, pk)
        if world == 1 and not args.skip_image and not wl.get("layout_cond"):
            out["image_latency"] = image_latency(model, inp, wl, dev)
        if world == 1 and not args.skip_cpu:
            out["cpu_baseline"] = cpu_baseline(args.workload, budget_s=args.cpu_budget)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        print(json.dumps(out))


def _ncu_traffic():
    """DRAM bytes per launch of the resampling kernels from the committed `ncu --set full` captures
    (profiles/resample_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum); absent -> null."""
    f = ROOT / "profiles" / "resample_traffic.json"
    return json.loads(f.read_text()) if f.exists() else {}


def micro_rooflines(dev, pk):
    """Isolated timings of the kernels the north star names. Each kernel is launched 20x inside ONE captured CUDA
    graph (no Python between launches), timed with CUDA events around graph replays; the launches rotate over
    enough distinct input/output buffers that consecutive launches never touch the same bytes within 126 MB of L2."""
    import numpy as np
    from panfusion_b200 import geometry, ops
    from panfusion_b200.engine import taps3x3
    from panfusion_b200.packing import pack_conv3x3
    res = {}
    traffic = _ncu_traffic()
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def timeit(fns, launches=20, reps=5):
        """fns: list of closures over DISTINCT buffers; launch i runs fns[i % len(fns)]. -> ms per launch."""
        for f in fns:
            f()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(launches):
                fns[i % len(fns)]()
        g.replay()
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        for _ in range(reps):
            g.replay()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / (reps * launches)

    def hbm_entry(name, ms, alg, note):
        t = traffic.get(name)
        res[name] = {"bound": "hbm", "ms": round(ms, 4), "algorithmic_bytes": alg, "achieved": round(alg / ms / 1e6, 1),
                     "peak": pk["hbm"], "unit": "GB/s", "frac": round(alg / ms / 1e6 / pk["hbm"], 4),
                     "traffic": t["dram_bytes"] if t else None, "traffic_source": t["source"] if t else None,
                     "shape": note}

    th16 = torch.tensor(np.tile(np.arange(8) * 45.0, 2), dtype=torch.float32)
    fov16, phi16 = torch.full((16,), 90.0), torch.zeros(16)
    # (1) e2p at the reference's own hot-path shape (get_masks, level 32): fp32 (16,2048,32,64) -> (16,2048,32,32)
    xs = [torch.randn(16, 2048, 32, 64, device=dev) for _ in range(2)]      # 268 MB each: > L2
    ms = timeit([(lambda x=x: geometry.e2p(x, fov16, th16, phi16, (32, 32))) for x in xs])
    hbm_entry("e2p_fp32_16x2048x32x64", ms, xs[0].numel() * 4 + 16 * 2048 * 32 * 32 * 4,
              "fp32 (16,2048,32,64) -> (16,2048,32,32), SURVEY 8d (i)")
    del xs
    # (2) p2e at the reference's hot-path shape: fp32 (16,1024,32,32) -> (16,1024,32,64) + 1 B/px mask
    ys = [torch.randn(16, 1024, 32, 32, device=dev) for _ in range(3)]      # 67 MB in + 134 MB out per launch
    ms = timeit([(lambda y=y: geometry.p2e(y, fov16, th16, phi16, (32, 64))) for y in ys])
    hbm_entry("p2e_fp32_16x1024x32x32", ms, ys[0].numel() * 4 + 16 * 1024 * 32 * 64 * 4 + 16 * 32 * 64,
              "fp32 (16,1024,32,32) -> (16,1024,32,64) + mask, SURVEY 8d (i)")
    del ys
    # (3) feature-map warp, bf16: pano (2,320,64,128) -> 16 views (16,320,64,64); the 2 panoramas are each read by their
    # 8 views (algorithmic source bytes = the 2 unique panoramas)
    zs = [torch.randn(2, 320, 64, 128, device=dev).bfloat16() for _ in range(16)]   # 16 x (10.5 MB in + 42 MB out)
    ms = timeit([(lambda z=z: geometry.e2p(z, fov16, th16, phi16, (64, 64), views_per_image=8)) for z in zs], launches=32)
    hbm_entry("e2p_bf16_2x320x64x128_to_16x320x64x64", ms, 2 * 320 * 64 * 128 * 2 + 16 * 320 * 64 * 64 * 2,
              "bf16 (2,320,64,128) -> (16,320,64,64), SURVEY 8d (ii)")
    del zs
    torch.cuda.empty_cache()
    # (4) tap-GEMM as the dominant 3x3 conv: 16 x 64x64 images, 320 -> 320 channels
    N, H, W, Ci, Co = 16, 64, 64, 320, 320
    Hp, Wp = H + 2, W + 2
    As = [torch.randn(N * Hp * Wp, Ci, device=dev).bfloat16() for _ in range(4)]   # 4 x (45 MB in + 42 MB out)
    wgt = pack_conv3x3(torch.randn(Co, Ci, 3, 3) * 0.02).bfloat16().to(dev)
    os_ = [torch.empty(N * H * W, Co, dtype=torch.bfloat16, device=dev) for _ in range(4)]
    ms = timeit([(lambda a=a, o=o: ops.gemm_taps(a, wgt, o, M=N * Hp * Wp, Kc=Ci, taps=taps3x3(Wp),
                                                 image_map=(Hp, Wp, 1, 1, H, W))) for a, o in zip(As, os_)])
    fl = 2.0 * 9 * Ci * Co * N * H * W
    res["conv3x3_320_16x64x64"] = {"bound": "tensor", "ms": round(ms, 4), "algorithmic_flops": fl,
                                   "achieved": round(fl / ms / 1e9, 1), "peak": pk["tf_burst"], "unit": "TFLOP/s",
                                   "frac": round(fl / ms / 1e9 / pk["tf_burst"], 4)}
    del As, os_
    # (5) flash attention, UNet self-attention at 64x64 (16 images, 5 heads, d 64)
    B, Hh, L, d = 16, 5, 4096, 64
    C = Hh * d
    qs = [torch.randn(B, L, 3 * C, device=dev).bfloat16() for _ in range(3)]       # 3 x (126 MB in + 42 MB out)
    oo = [torch.empty(B, L, C, dtype=torch.bfloat16, device=dev) for _ in range(3)]
    ms = timeit([(lambda q=q, o=o: ops.fmha(q[..., :C], q[..., C:2 * C], q[..., 2 * C:], o, heads=Hh, head_dim=d,
                                            scale=d ** -0.5)) for q, o in zip(qs, oo)], launches=12)
    fl = 4.0 * B * Hh * L * L * d
    res["fmha_d64_16x5x4096"] = {"bound": "tensor", "ms": round(ms, 4), "algorithmic_flops": fl,
                                 "achieved": round(fl / ms / 1e9, 1), "peak": pk["tf_burst"], "unit": "TFLOP/s",
                                 "frac": round(fl / ms / 1e9 / pk["tf_burst"], 4)}
    del qs, oo
    torch.cuda.empty_cache()
    return res


def image_latency(model, inp, wl, dev, n_steps=50):
    """What `main.py predict` pays per image (PanFusion.py:125-172 after the text encoder): a FRESH sampler runs
    init_noise -> 50 denoise steps -> rotate back -> VAE decode (views + circularly padded panorama) -> uint8, wall
    clock, including the camera-table builds and the 4 CUDA-graph captures of a first image ("cold"); then a second
    image on the same sampler, which reuses buffers, tables and graphs ("warm")."""
    from panfusion_b200 import sd2_unet, vae as pv
    from panfusion_b200.sampler import PanFusionSampler
    dt = torch.bfloat16
    dec = pv.VAEDecoder(sd2_unet.build_synthetic_vae(seed=9, device=dev), dt).prepare(dev, dt)
    sampler = PanFusionSampler(model)
    prompt, pano_prompt = inp["prompt"].to(dev), inp["pano_prompt"].to(dev)
    out = {}
    for tag, seed in (("cold_first_image_s", 11), ("warm_next_image_s", 12)):
        g = torch.Generator(device=dev).manual_seed(seed)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        images, pano = sampler.inference(inp["cams"], prompt, pano_prompt, dec, wl["pano_hw"], wl["pers_hw"], device=dev,
                                         generator=g, num_steps=n_steps)
        h_img, h_pano = images, pano   # uint8 numpy on the host, like the reference's tensor_to_image
        out[tag] = round(time.perf_counter() - t0, 4)
    out["what"] = (f"sampler.inference: init_noise + {n_steps} denoise steps + rotate back + VAE decode of {wl['m']} views "
                   f"and the padded panorama + tensor_to_image (uint8 images returned on the host)")
    out["image_shapes"] = [list(h_img.shape), list(h_pano.shape)]
    return out


# ------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle (a port of the reference algorithm) on the host cores
# ------------------------------------------------------------------------------------------------------
_ORACLE_MODEL = {}


def host_threads() -> int:
    """Cores this process may actually use: min(cpu_count, affinity mask, cgroup quota), capped at 64 (the oracle's
    fp32 convolutions stop scaling well before that)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, min(n, 64))


def _oracle_model(layout_cond: bool = False):
    """SD-2-size oracle model for TIMING: built on the meta device and filled by tiling one random block (the values
    do not matter for a CPU throughput baseline; PyTorch's seeded default init of 2 x 866 M parameters alone takes
    about a minute of single-threaded RNG). layout_cond adds the panorama ControlNet of BASELINE configs[4]
    (ControlNetModel.from_unet topology, models/pano/PanoGenerator.py:153-157)."""
    if layout_cond not in _ORACLE_MODEL:
        from oracle import controlnet as ocn, mvgen as om, unet as ou
        torch.set_num_threads(host_threads())
        with torch.device("meta"):
            cn = ocn.ControlNetModel(ou.UNet2DConditionModel(**ou.SD2_CONFIG)) if layout_cond else None
            model = om.MultiViewBaseModel(ou.UNet2DConditionModel(**ou.SD2_CONFIG), ou.UNet2DConditionModel(**ou.SD2_CONFIG),
                                          pano_cn=cn)
        model = model.to_empty(device="cpu").eval()
        g = torch.Generator().manual_seed(0)
        block = torch.randn(1 << 20, generator=g) * 0.02
        with torch.no_grad():
            for name, p in model.named_parameters():
                n = p.numel()
                p.view(-1).copy_(block.repeat((n + block.numel() - 1) // block.numel())[:n])
                if name.endswith("weight") and p.dim() == 1:
                    p.add_(1.0)  # norm scales around 1
            for name, b in model.named_buffers():
                if name.endswith("freq_bands"):
                    nf = b.numel()
                    base = 2 if nf <= 80 else 5000 ** (1 / (nf / 2.5))
                    b.copy_(base ** torch.linspace(0, nf - 1, nf))
        _ORACLE_MODEL[layout_cond] = model
    return _ORACLE_MODEL[layout_cond]


class _OracleLoop:
    """The reference's sampling loop (models/pano/PanFusion.py:146-162: rotate -> CFG-batched
    MultiViewBaseModel.forward -> CFG combine -> 2x DDIM update) on the host cores, through the oracle port, on the
    benchmark workload itself (same views / latent sizes / CFG batch / cameras / guidance as the B200 arm)."""

    def __init__(self, workload):
        from oracle import sampler as osamp
        torch.set_num_threads(host_threads())
        wl = WORKLOADS[workload]
        self.osamp, self.model = osamp, _oracle_model(bool(wl.get("layout_cond")))
        inp = synthetic_inputs(wl, 1024, "cpu", None)
        self.cond = inp.get("pano_layout_cond")   # rolled a quarter turn per step, cumulatively (PanFusion.py:152-153)
        self.cams = inp["cams"]
        self.pano = inp["pano"]
        self.lat = osamp.init_noise(self.pano, *wl["pers_hw"], self.cams)
        self.prompt, self.pano_prompt = inp["prompt"], inp["pano_prompt"]
        self.i = 0

    def step(self) -> float:
        """One iteration of the loop; returns its wall time in seconds."""
        t0 = time.perf_counter()
        self.lat, self.pano, self.cams = self.osamp.denoise_steps(
            self.model, self.lat, self.pano, self.prompt, self.pano_prompt, self.cams, num_steps=1,
            start_step=self.i % 50, pano_layout_cond=self.cond)
        if self.cond is not None:  # denoise_steps rolled its own copy for this step: keep the roll for the next call
            self.cond = torch.roll(self.cond, self.cond.shape[-1] // 4, dims=-1)
        self.i += 1
        return time.perf_counter() - t0


def cpu_baseline(workload, budget_s=30.0):
    """ONE real iteration of the reference loop on the benchmark workload (oracle port, fp32, all usable host cores):
    no extrapolation. About a minute of CPU work at C2 — the smallest sample that IS the metric's unit."""
    cores = host_threads()
    loop = _OracleLoop(workload)
    t = loop.step()
    return {"value": round(1.0 / t, 5), "unit": "steps/s", "cores": cores, "kind": "port",
            "sample": f"1 full denoise step of this workload (rotate + CFG-batched forward + combine + 2 DDIM updates, "
                      f"reference algorithm via the oracle port, fp32) = {t:.1f} s on {cores} threads; measured, not scaled"}


def run_reference(args):
    """`--impl reference`: the reference algorithm's own CPU path (oracle port; diffusers/xformers/kornia are not
    installable offline, SURVEY.md §8c) on the usable host cores, REAL steps of the benchmark workload: one warm-up
    step, then --steps timed steps (about a minute each at C2). `steps` / `warmup` in the JSON line are the counts
    actually run. Rank 0 only."""
    if int(os.environ.get("RANK", 0)) != 0:
        return
    wl = WORKLOADS[args.workload]
    cores = host_threads()
    loop = _OracleLoop(args.workload)
    loop.step()
    times = [loop.step() for _ in range(args.steps)]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, loop.lat, loop.pano)
    per = sum(times) / args.steps
    val = round(1.0 / per, 5)
    sample = (f"{args.steps} full denoise steps of this workload after 1 warm-up step (rotate + CFG-batched forward + combine "
              f"+ 2 DDIM updates; reference algorithm via the oracle port, fp32, {cores} threads): "
              f"{', '.join(f'{t:.1f}' for t in times)} s; measured, not scaled")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": 1, "ms_per_step": round(per * 1e3, 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "views": wl["m"], "cfg_batch": 2, "pano_latent": list(wl["pano_hw"]),
                   "view_latent": list(wl["pers_hw"]), "weights": "synthetic SD-2 architecture"},
        "cpu_baseline": {"value": val, "unit": "steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=list(WORKLOADS))
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying CUDA graphs")
    ap.add_argument("--skip-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--skip-micro", action="store_true", help="skip the isolated kernel rooflines")
    ap.add_argument("--skip-image", action="store_true", help="skip the cold / warm whole-image latency leg")
    ap.add_argument("--cpu-budget", type=float, default=30.0)
    ap.add_argument("--profile-one-step", action="store_true", help="for ncu --profile-from-start off: profile one eager step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the latents of the last timed step as DIR/latents.npy and DIR/pano_latent.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
