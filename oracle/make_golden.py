"""Mint tests/golden/*.npz by EXECUTING THE REFERENCE'S OWN FILES (oracle/ref_loader.py) on seeded inputs, and
check the oracle restatement against them. Runs only where /root/reference is mounted (the build container).

    python -m oracle.make_golden [--full]     # --full adds the SD-2-size C1 step (minutes on 8 cores)
    python -m oracle.make_golden --only c2    # BASELINE configs[1]: SD-2 widths, 8 views, CFG pair (b = 2)
    python -m oracle.make_golden --only c4geo # get_masks at config 4's real level size (32x32 views, 64x128 pano)
    python -m oracle.make_golden --only py360 # external/py360convert e2p (dataset convention) on seeded images

Each fixture stores the seeded inputs' identifying parameters and the reference outputs; tests regenerate the
inputs from the seeds (same torch build on both boxes) and compare.
"""
from __future__ import annotations

import argparse
import sys
import time
from pathlib import Path

import numpy as np
import torch

from . import eppa as oe, geometry as og, mvgen as om, ref_loader, synth, unet as ounet

OUT = Path(__file__).resolve().parent.parent / "tests" / "golden"


def _cams3():
    return dict(FoV=torch.tensor([90.0, 75.0, 100.0]), theta=torch.tensor([0.0, 45.0, 200.0]),
                phi=torch.tensor([0.0, 30.0, -60.0]))


def _cams_ico():
    """One camera from each icosahedron ring (utils/pano.py:34-71), degrees."""
    return dict(FoV=torch.full((4,), 90.0), theta=torch.tensor([-144.0, 72.0, -180.0, 36.0]),
                phi=torch.tensor([52.6226, 10.8123, -10.8123, -52.6226]))


def _report(name, ref, mine):
    err = max((a - b).abs().max().item() for a, b in zip(ref, mine))
    print(f"  {name}: max |oracle - reference| = {err:.3e}")
    return err


def round_mantissa(a: np.ndarray, bits: int = 15) -> np.ndarray:
    """float32 rounded to nearest with `bits` of its 23 mantissa bits kept (relative error <= 2**-(bits + 1)). The low
    mantissa bits of model outputs do not compress; dropping 8 of them keeps a fixture under 1 MB at 1.5e-5 of each
    value, far below the 4e-3 / 2.5e-2 parity gates it is compared at."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    drop = 23 - bits
    return ((u + np.uint32(1 << (drop - 1))) >> drop << drop).astype(np.uint32).view(np.float32)


def golden_c2(ref):
    """BASELINE configs[1], the benchmarked configuration: SD-2 widths, 8 horizon views 64x64 + pano 64x128, the CFG
    pair (b = 2, prompts [null; text]) — ONE reference MultiViewBaseModel.forward (MVGenModel.py:38-297) on CPU."""
    cfg = ounet.SD2_CONFIG
    model_r = synth.build_model(ref.MultiViewBaseModel, cfg, seed=0)
    inp = synth.step_inputs_cfg(8, (64, 128), (64, 64), cfg["cross_attention_dim"], seed=0)
    t0 = time.time()
    rs, rp_ = model_r(**inp)
    t1 = time.time()
    print(f"  [c2] reference forward {t1 - t0:.1f}s", flush=True)
    np.savez_compressed(OUT / "mvgen_c2.npz", sample=round_mantissa(rs.numpy()), pano_sample=round_mantissa(rp_.numpy()))
    model_o = synth.build_model(om.MultiViewBaseModel, cfg, seed=0)
    model_o.load_state_dict(model_r.state_dict())
    del model_r
    os_, op_ = model_o(**inp)
    print(f"  [c2] oracle forward {time.time() - t1:.1f}s", flush=True)
    return _report("MultiViewBaseModel c2", [rs, rp_], [os_, op_])


C4GEO_LEVEL = (32, 32, 64, 128)   # config 4's first EPPA level: 512^2 views / 8 / 2, 1024x2048 pano / 8 / 2


def c4geo_subsample(pm, em):
    """The full masks are 2 x 134 MB: the fixture keeps every 7th x 9th panorama query row of pers_masks, every 5th x
    5th view query row of equi_masks (all keys), plus the key-sum of EVERY query row (float64) of both."""
    return dict(pers_rows=pm[:, ::7, ::9].numpy(), equi_rows=em[:, ::5, ::5].numpy(),
                pers_rowsum=pm.double().sum((-1, -2)).numpy(), equi_rowsum=em.double().sum((-1, -2)).numpy())


def golden_c4_geometry(ref):
    """get_masks (models/pano/utils.py:10-84) at config 4's REAL first-level size with one camera per icosahedron
    ring — the sizes at which the circular / replicate blur borders, the pole rows and the per-row normalisation see
    production-size grids."""
    ci = _cams_ico()
    ph, pw, eh, ew = C4GEO_LEVEL
    t0 = time.time()
    pm, em = ref.get_masks(ph, pw, eh, ew, ci, "cpu")
    print(f"  [c4geo] reference get_masks {time.time() - t0:.1f}s", flush=True)
    err = _report("get_masks (ico, 32x32 / 64x128)", [pm, em], oe.get_masks(ph, pw, eh, ew, ci))
    np.savez_compressed(OUT / "eppa_geometry_c4_level.npz", **c4geo_subsample(pm, em))
    return err


PY360_CASES = [  # (fov (h, v), yaw u, pitch v, out_hw, in_rot, mode): poles, the +-180 seam, non-square FoV, roll
    ((90, 90), 30.0, 20.0, (48, 48), 0.0, "bilinear"), ((90, 90), 180.0, -85.0, (40, 56), 10.0, "bilinear"),
    ((70, 100), -170.0, 88.0, (33, 21), 0.0, "nearest"), ((90, 90), 0.0, 0.0, (64, 64), 0.0, "bilinear"),
    ((90, 90), -179.5, 0.0, (32, 32), 0.0, "nearest")]


def py360_images():
    rng = np.random.default_rng(0)
    return rng.integers(0, 256, (64, 128, 3)).astype(np.uint8), rng.random((32, 64, 2)).astype(np.float32)


def golden_py360():
    """external/py360convert/e2p.py executed by path (it imports cleanly: numpy + scipy) on seeded images."""
    import importlib
    from . import py360 as op
    if str(ref_loader.REF) not in sys.path:
        sys.path.insert(0, str(ref_loader.REF))
    ref360 = importlib.import_module("external.py360convert")
    out, worst = {}, 0.0
    for k, (fov, u, v, hw, rot, mode) in enumerate(PY360_CASES):
        for tag, im in zip(("u8", "f32"), py360_images()):
            r = ref360.e2p(im, fov, u, v, hw, in_rot_deg=rot, mode=mode)
            out[f"case{k}_{tag}"] = r
            worst = max(worst, float(np.abs(r.astype(np.float64) - op.e2p(im, fov, u, v, hw, rot, mode).astype(np.float64)).max()))
    print(f"  py360convert.e2p: max |oracle - reference| = {worst:.3e}")
    np.savez_compressed(OUT / "py360_e2p.npz", **out)
    return worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--full", action="store_true")
    ap.add_argument("--only", choices=["c2", "c4geo", "py360"], help="mint just one of the separately kept fixtures")
    args = ap.parse_args()
    ref = ref_loader.load()
    OUT.mkdir(parents=True, exist_ok=True)
    torch.set_grad_enabled(False)
    worst = 0.0
    if args.only == "c2":
        return 0 if golden_c2(ref) < 1e-4 else 1
    if args.only == "c4geo":
        return 0 if golden_c4_geometry(ref) < 1e-5 else 1
    if args.only == "py360":
        return 0 if golden_py360() == 0.0 else 1

    # 1. resampling (e2p.py:54-76, p2e.py:52-77)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(3, 5, 32, 64, generator=g)
    y = torch.randn(3, 5, 16, 24, generator=g)
    c = _cams3()
    out = {}
    for mode in ("bilinear", "nearest"):
        r = ref.e2p(x, c["FoV"], c["theta"], c["phi"], (16, 24), mode=mode)
        out[f"e2p_{mode}"] = r.numpy()
        worst = max(worst, _report(f"e2p {mode}", [r], [og.e2p(x, c["FoV"], c["theta"], c["phi"], (16, 24), mode=mode)]))
        r, rm = ref.p2e(y, c["FoV"], c["theta"], c["phi"], (32, 64), mode=mode)
        out[f"p2e_{mode}"], out[f"p2e_{mode}_mask"] = r.numpy(), rm.numpy()
        mo, mm = og.p2e(y, c["FoV"], c["theta"], c["phi"], (32, 64), mode=mode)
        worst = max(worst, _report(f"p2e {mode}", [r, rm.float()], [mo, mm.float()]))
    r = ref.e2p(x, 90, 10, 5, (16, 16))
    out["e2p_scalar"] = r.numpy()
    np.savez_compressed(OUT / "resample.npz", **out)

    # 2. EPPA geometry (models/pano/utils.py:10-106)
    pm, em = ref.get_masks(8, 8, 8, 16, c, "cpu")
    pc, ec = ref.get_coords(8, 8, 8, 16, c, "cpu")
    worst = max(worst, _report("get_masks", [pm, em], oe.get_masks(8, 8, 8, 16, c)))
    worst = max(worst, _report("get_coords", [pc, ec], oe.get_coords(8, 8, 8, 16, c)))
    np.savez_compressed(OUT / "eppa_geometry.npz", pers_masks=pm.numpy(), equi_masks=em.numpy(),
                        pers_coords=pc.numpy(), equi_coords=ec.numpy())

    # 2b. BASELINE config 4's geometry: pers level smaller than the pano level (ph != eh), icosahedron-ring cameras
    # (utils/pano.py:34-71: phi = +-52.62 / +-10.81 deg, negative thetas)
    ci = _cams_ico()
    pm, em = ref.get_masks(8, 8, 16, 32, ci, "cpu")
    pc, ec = ref.get_coords(8, 8, 16, 32, ci, "cpu")
    worst = max(worst, _report("get_masks (ico, ph != eh)", [pm, em], oe.get_masks(8, 8, 16, 32, ci)))
    worst = max(worst, _report("get_coords (ico, ph != eh)", [pc, ec], oe.get_coords(8, 8, 16, 32, ci)))
    np.savez_compressed(OUT / "eppa_geometry_c4.npz", pers_masks=pm.numpy(), equi_masks=em.numpy(),
                        pers_coords=pc.numpy(), equi_coords=ec.numpy())

    # 3. WarpAttn (models/pano/modules.py:8-59), dim 320, 2 batches x 2 views
    torch.manual_seed(7)
    wr = ref.WarpAttn(320).eval()
    holder = torch.nn.Module()
    holder.cp_blocks = wr
    synth.randomize_zero_init(holder, 11)
    wm = oe.WarpAttn(320).eval()
    wm.load_state_dict(wr.state_dict())
    g = torch.Generator().manual_seed(8)
    px, ex = torch.randn(4, 320, 8, 8, generator=g), torch.randn(2, 320, 8, 16, generator=g)
    c4 = dict(FoV=torch.full((4,), 90.0), theta=torch.tensor([0.0, 180.0, 0.0, 180.0]), phi=torch.zeros(4))
    rp, re = wr(px, ex, c4)
    worst = max(worst, _report("WarpAttn", [rp, re], wm(px, ex, c4)))
    np.savez_compressed(OUT / "warpattn_320.npz", pers_out=rp.numpy(), equi_out=re.numpy())

    # 4. MultiViewBaseModel (models/pano/MVGenModel.py:38-297) with narrow UNets: m=2, pers 16x16, pano 16x32
    def mv(config, pano_hw, pers_hw, tag):
        model_r = synth.build_model(ref.MultiViewBaseModel, config, seed=0)
        model_o = synth.build_model(om.MultiViewBaseModel, config, seed=0)
        model_o.load_state_dict(model_r.state_dict())
        inp = synth.step_inputs(2, pano_hw, pers_hw, config["cross_attention_dim"], seed=0)
        t0 = time.time()
        rs, rp_ = model_r(**inp)
        t1 = time.time()
        os_, op_ = model_o(**inp)
        print(f"  [{tag}] reference {t1 - t0:.1f}s oracle {time.time() - t1:.1f}s")
        np.savez_compressed(OUT / f"mvgen_{tag}.npz", sample=rs.numpy(), pano_sample=rp_.numpy())
        return _report(f"MultiViewBaseModel {tag}", [rs, rp_], [os_, op_])

    worst = max(worst, mv(ounet.TINY_CONFIG, (16, 32), (16, 16), "tiny"))

    # 5. layout-conditioned step (BASELINE config 5): the reference's residual wiring (MVGenModel.py:62-83,154-170,
    # 200-203) executed as-is around the duck-typed ControlNet restatement (oracle/controlnet.py, [3P])
    def mv_cn(config, pano_hw, pers_hw, tag, pers):
        model_r = synth.build_model_cn(ref.MultiViewBaseModel, config, seed=0, pers=pers)
        model_o = synth.build_model_cn(om.MultiViewBaseModel, config, seed=0, pers=pers)
        model_o.load_state_dict(model_r.state_dict())
        inp = synth.step_inputs(2, pano_hw, pers_hw, config["cross_attention_dim"], seed=0)
        inp.update(synth.layout_conds(1, 2, pano_hw, pers_hw, seed=5, pers=pers))
        rs, rp_ = model_r(**inp)
        os_, op_ = model_o(**inp)
        base_s, base_p = model_r(**{**inp, "pano_layout_cond": None, "pers_layout_cond": None})
        print(f"  [{tag}] effect of the layout condition: {(rs - base_s).abs().max():.3e} / {(rp_ - base_p).abs().max():.3e}")
        np.savez_compressed(OUT / f"mvgen_{tag}.npz", sample=rs.numpy(), pano_sample=rp_.numpy())
        return _report(f"MultiViewBaseModel {tag}", [rs, rp_], [os_, op_])

    worst = max(worst, mv_cn(ounet.TINY_CONFIG, (16, 32), (16, 16), "tiny_cn", False))
    worst = max(worst, mv_cn(ounet.TINY_CONFIG, (16, 32), (16, 16), "tiny_cn2", True))
    if args.full:
        worst = max(worst, mv(ounet.SD2_CONFIG, (64, 128), (64, 64), "c1"))
    print(f"worst oracle-vs-reference deviation: {worst:.3e}")
    return 0 if worst < 1e-4 else 1


if __name__ == "__main__":
    sys.exit(main())
