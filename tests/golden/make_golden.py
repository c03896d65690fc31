"""Generate tests/golden/reference_path.pt by running the REFERENCE'S OWN in-tree Python.

Needs a checkout of the reference (Ced-NeRF); the tests only read the file this writes:

    python tests/golden/make_golden.py <reference checkout>

The reference cannot be imported as-is: cednerf/model.py exits without tinycudann, cednerf/utils.py
and cednerf/render.py import nerfacc, cednerf/taichi_kernel/* import taichi (SURVEY.md §8c).  Those
three absent third-party packages are replaced in sys.modules by the oracle's restatements
(oracle.tcnn_ref / oracle.nerfacc_ref) and an inert taichi stub; everything else that executes is the
reference's own code, unmodified, read from the checkout:

    cednerf/encoder.py   SinusoidalEncoder, SinusoidalEncoderWithExp
    cednerf/utils.py     trunc_exp, render_image, render_image_test
    cednerf/render.py    rendering
    cednerf/model.py     DNGPradianceField

The frozen vectors pin (a) oracle.cednerf_ref and (b) cednerf_b200's mirror of the same surface.
`compact` says what of them the file keeps.
"""
import os
import sys
import types
from unittest.mock import MagicMock

import torch

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)

from oracle import nerfacc_ref as nf  # noqa: E402
from oracle import tcnn_ref as tc  # noqa: E402


def install_stubs():
    ti = MagicMock(name="taichi")
    sys.modules["taichi"] = ti
    sys.modules["taichi.math"] = ti.math
    tcnn = types.ModuleType("tinycudann")
    tcnn.Encoding, tcnn.Network, tcnn.NetworkWithInputEncoding = tc.Encoding, tc.Network, tc.NetworkWithInputEncoding
    sys.modules["tinycudann"] = tcnn
    na = types.ModuleType("nerfacc")
    for name in ("traverse_grids", "ray_aabb_intersect", "render_weight_from_density", "accumulate_along_rays",
                 "render_transmittance_from_density", "render_visibility_from_density"):
        setattr(na, name, getattr(nf, name))
    est = types.ModuleType("nerfacc.estimators")
    occ = types.ModuleType("nerfacc.estimators.occ_grid")
    occ.OccGridEstimator = nf.OccGridEstimator
    vol = types.ModuleType("nerfacc.volrend")
    vol.accumulate_along_rays_ = nf.accumulate_along_rays_
    na.estimators, est.occ_grid, na.volrend = est, occ, vol
    sys.modules.update({"nerfacc": na, "nerfacc.estimators": est, "nerfacc.estimators.occ_grid": occ,
                        "nerfacc.volrend": vol})


def synthetic_scene(seed=42, n_rays=96, res=16, levels=2):
    g = torch.Generator().manual_seed(seed)
    est = nf.OccGridEstimator([-1.0, -1.0, -1.0, 1.0, 1.0, 1.0], resolution=res, levels=levels)
    est.binaries = torch.rand(levels, res, res, res, generator=g) < 0.15
    est.occs = est.binaries.flatten().float() * 0.5
    origins = torch.tensor([0.0, 0.0, -3.5]) + (torch.rand(n_rays, 3, generator=g) - 0.5) * 0.6
    target = (torch.rand(n_rays, 3, generator=g) - 0.5) * 1.6
    dirs = torch.nn.functional.normalize(target - origins, dim=-1)
    ts = torch.rand(n_rays, 1, generator=g)
    return est, origins, dirs, ts


FIELD_KW = dict(n_levels=8, log2_hashmap_size=12, dst_resolution=256, moving_step=1.0 / 256)
FLAG_SETS = {
    "plain": dict(),
    "te_ta_df": dict(use_time_embedding=True, use_time_attenuation=True, use_div_offsets=True),
    "te_after": dict(use_time_embedding=True, time_inject_before_sigma=False),
}


def boost_density(field):
    """Random-init sigma is ~exp(-1) everywhere; widen the logits so that alpha_thre keeps samples,
    transmittance decays and early termination triggers (sigma median ~2, max ~60)."""
    with torch.no_grad():
        field.hash_encoder.params.mul_(5000.0)
        field.mlp_base.params.mul_(3.0)


HASH_GRAD_SAMPLE = 4096


def compact(out):
    """What reference_path.pt keeps of `out`, so that it stays under 1 MB:
    - the four tiny-cuda-nn parameter tables of each field's initial state are not stored.  The reference draws them
      with tcnn's default seed and boost_density scales them; tests/conftest.py repeats that and checks the result
      against the float64 sums stored as `<set>.state_sum.<key>`.  `<set>.field_kwargs` holds the field's arguments.
    - each hash-grid gradient keeps the entries at one fixed, seeded sample of HASH_GRAD_SAMPLE positions
      (`grad_sample_index`) and the float64 L2 norm of the whole tensor.
    Everything else is stored as computed."""
    out = dict(out)
    n_table = out["plain.field.grad.hash_encoder.params"].numel()
    idx = torch.randperm(n_table, generator=torch.Generator().manual_seed(0))[:HASH_GRAD_SAMPLE].sort().values
    out["grad_sample_index"] = idx.int()
    for name, flags in FLAG_SETS.items():
        out[f"{name}.field_kwargs"] = dict(FIELD_KW, **flags)
        for mod in ("xyz_wrap", "hash_encoder", "mlp_base", "mlp_head"):
            out[f"{name}.state_sum.{mod}.params"] = out.pop(f"{name}.state.{mod}.params").double().sum()
        for part in ("field", "train"):
            key = f"{name}.{part}.grad.hash_encoder.params"
            g = out.pop(key)
            out[key + ".sample"], out[key + ".norm"] = g[idx].clone(), g.double().norm()
    return out


def main(ref):
    sys.path.insert(0, ref)
    install_stubs()
    from cednerf.encoder import SinusoidalEncoder, SinusoidalEncoderWithExp
    from cednerf.model import DNGPradianceField
    from cednerf.render import rendering
    from cednerf.utils import render_image, render_image_test, trunc_exp
    from datasets.utils import Rays

    out = {}
    g = torch.Generator().manual_seed(7)
    # --- E4 / E5
    t = torch.rand(64, 1, generator=g)
    mv = torch.rand(64, 1, generator=g) * 0.01
    out["enc.t"], out["enc.move"] = t, mv
    out["enc.sin"] = SinusoidalEncoder(1, 0, 4, True)(t)
    out["enc.sinexp"] = SinusoidalEncoderWithExp(1, 0, 4, True)(t, mv)
    # --- trunc_exp
    x = (torch.rand(64, generator=g) * 40 - 20).requires_grad_(True)
    y = trunc_exp(x)
    gy = torch.rand(64, generator=g)
    y.backward(gy)
    out["texp.x"], out["texp.y"], out["texp.gy"], out["texp.gx"] = x.detach(), y.detach(), gy, x.grad

    est, origins, dirs, ts = synthetic_scene()
    out["scene.binaries"], out["scene.occs"], out["scene.aabbs"] = est.binaries, est.occs, est.aabbs
    out["scene.origins"], out["scene.dirs"], out["scene.timestamps"] = origins, dirs, ts
    rays = Rays(origins=origins, viewdirs=dirs)
    opts = dict(near_plane=0.2, render_step_size=2e-2, cone_angle=0.004, alpha_thre=1e-2)

    for name, flags in FLAG_SETS.items():
        field = DNGPradianceField(aabb=est.aabbs[-1], **FIELD_KW, **flags)
        boost_density(field)
        for k, v in field.state_dict().items():
            out[f"{name}.state.{k}"] = v.clone()
        # --- field forward/backward on random points (train mode -> interal_output)
        pts = (torch.rand(160, 3, generator=g) * 2 - 1) * 1.2
        pts.requires_grad_(False)
        tt = torch.rand(160, 1, generator=g)
        dd = torch.nn.functional.normalize(torch.randn(160, 3, generator=g), dim=-1)
        field.train()
        rgb, res = field(pts, tt, dd)
        grgb, gsig = torch.rand(160, 3, generator=g), torch.rand(160, 1, generator=g)
        field.zero_grad()
        ((rgb * grgb).sum() + (res["density"] * gsig).sum()).backward()
        out[f"{name}.field.pts"], out[f"{name}.field.t"], out[f"{name}.field.dirs"] = pts, tt, dd
        out[f"{name}.field.rgb"], out[f"{name}.field.density"] = rgb.detach(), res["density"].detach()
        out[f"{name}.field.base_mlp_out"] = res["base_mlp_out"].detach()
        out[f"{name}.field.move"] = res["interal_output"]["move"].detach()
        out[f"{name}.field.grgb"], out[f"{name}.field.gsig"] = grgb, gsig
        for k, p in field.named_parameters():
            if p.grad is not None:
                out[f"{name}.field.grad.{k}"] = p.grad.clone()
        # --- render_image, train mode (stratified jitter from the global RNG, seeded)
        field.train()
        est.train()
        bkgd = torch.tensor([0.2, 0.5, 0.8])
        torch.manual_seed(123)
        rgb, acc, depth, n_s, extra = render_image(field, est, rays, render_bkgd=bkgd, timestamps=ts, **opts)
        out[f"{name}.train.rgb"], out[f"{name}.train.acc"], out[f"{name}.train.depth"] = rgb.detach(), acc.detach(), depth.detach()
        out[f"{name}.train.n_samples"] = torch.tensor(n_s)
        for k in ("ray_indices", "t_starts", "t_ends", "weights", "trans", "alphas", "sigmas"):
            out[f"{name}.train.{k}"] = extra[0][k].detach()
        # backward of an MSE loss through the reference's rendering()
        pix = torch.rand(rgb.shape, generator=g)
        field.zero_grad()
        loss = torch.nn.functional.mse_loss(rgb, pix)
        (loss * 1024.0).backward()
        out[f"{name}.train.pixels"], out[f"{name}.train.loss"] = pix, loss.detach()
        for k, p in field.named_parameters():
            if p.grad is not None:
                out[f"{name}.train.grad.{k}"] = p.grad.clone()
        # --- eval paths
        field.eval()
        est.eval()
        t_frame = torch.tensor([[0.5]])
        with torch.no_grad():
            rgb, acc, depth, n_s, _ = render_image(field, est, rays, render_bkgd=bkgd, timestamps=t_frame,
                                                   test_chunk_size=40, **opts)
        out[f"{name}.eval.rgb"], out[f"{name}.eval.acc"], out[f"{name}.eval.depth"] = rgb, acc, depth
        out[f"{name}.eval.n_samples"] = torch.tensor(n_s)
        rgb, acc, depth, n_s = render_image_test(64, field, est, rays, render_bkgd=bkgd, timestamps=t_frame, **opts)
        out[f"{name}.test.rgb"], out[f"{name}.test.acc"], out[f"{name}.test.depth"] = rgb, acc, depth
        out[f"{name}.test.n_samples"] = torch.tensor(n_s)

    # --- rendering() alone on hand-made samples and a closed-form field
    ridx = torch.tensor([0, 0, 0, 2, 2, 5])
    t0 = torch.tensor([0.1, 0.2, 0.3, 0.5, 0.6, 1.0])
    t1 = t0 + 0.1
    sig = torch.tensor([0.5, 3.0, 10.0, 0.0, 7.0, 100.0], requires_grad=True)
    col = torch.rand(6, 3, generator=g).requires_grad_(True)
    c, o, d, ex = rendering(t0, t1, ridx, 6, lambda a, b, r: (col, {"density": sig[:, None]}), torch.ones(3))
    gc, go, gd = torch.rand(6, 3, generator=g), torch.rand(6, 1, generator=g), torch.rand(6, 1, generator=g)
    ((c * gc).sum() + (o * go).sum() + (d * gd).sum()).backward()
    out.update({"rend.ridx": ridx, "rend.t0": t0, "rend.t1": t1, "rend.sigma": sig.detach(), "rend.rgb": col.detach(),
                "rend.colors": c.detach(), "rend.opac": o.detach(), "rend.depth": d.detach(),
                "rend.weights": ex["weights"].detach(), "rend.trans": ex["trans"].detach(),
                "rend.gc": gc, "rend.go": go, "rend.gd": gd, "rend.gsigma": sig.grad, "rend.grgb": col.grad})

    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_path.pt")
    out = compact(out)
    torch.save({k: (v.clone() if torch.is_tensor(v) else v) for k, v in out.items()}, path)
    print("wrote", path, f"{os.path.getsize(path) / 1e6:.2f} MB,", len(out), "entries")


if __name__ == "__main__":
    main(sys.argv[1])
