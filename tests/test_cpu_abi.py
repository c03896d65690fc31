"""CPU-side checks (no GPU): the C-ABI library loads, exports every symbol include/cednerf_b200.h declares,
the ctypes signatures agree with the header, host-side descriptors match the oracle's geometry, and the product
refuses to run without CUDA (no CPU fallback)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_decls():
    h = open(os.path.join(ROOT, "include", "cednerf_b200.h")).read()
    h = re.sub(r"/\*.*?\*/", "", h, flags=re.S)
    return re.findall(r"\b(int|int64_t|const char\*)\s+(cednerf_\w+)\s*\(([^;]*?)\)\s*;", h, flags=re.S)


def test_library_exports_every_declared_symbol():
    from cednerf_b200 import _lib

    lib = _lib.load()
    names = [n for _, n, _ in header_decls()]
    assert len(names) >= 28
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"
    assert sorted(names) == _lib.exported_symbols()
    assert lib.cednerf_abi_version() == 4


def test_ctypes_signatures_match_header():
    from cednerf_b200 import _lib

    for _, name, args in header_decls():
        if name not in _lib._SIGNATURES:
            continue
        sig = ""
        for a in [x.strip() for x in args.split(",")]:
            if "CednerfFieldDesc" in a:
                sig += "F"
            elif "CednerfGridLevels" in a:
                sig += "G"
            elif "CednerfMlpDesc" in a:
                sig += "M"
            elif "CednerfAdamTensors" in a:
                sig += "A"
            elif "CednerfDpPeers" in a:
                sig += "P"
            elif "CednerfDpAdam" in a:
                sig += "D"
            elif "CednerfDpSmall" in a:
                sig += "S"
            elif "CednerfRenderRound" in a:
                sig += "R"
            elif a.startswith("uint32_t "):
                sig += "u"
            elif "*" in a:
                sig += "p"
            elif a.startswith("int64_t"):
                sig += "l"
            elif a.startswith("int "):
                sig += "i"
            elif a.startswith("float "):
                sig += "f"
            else:
                raise AssertionError(f"unparsed argument {a!r} in {name}")
        assert sig == _lib._SIGNATURES[name], name


def test_descriptor_structs_match_header_layout():
    from cednerf_b200 import _lib

    assert ctypes.sizeof(_lib.GridLevels) == 4 + 5 * 4 * 32
    assert ctypes.sizeof(_lib.MlpDesc) == 4 + 4 * 4 * 5 + 4
    # n_tensors (+ padding to 8), five pointer arrays, n[8], lr[8], weight_decay[8], chunk_begin[9]
    assert ctypes.sizeof(_lib.AdamTensors) == 8 + 5 * 8 * 8 + 8 * 8 + 2 * 4 * 8 + 9 * 8
    assert ctypes.sizeof(_lib.DpCtrl) == 8 * 4 + 4 + 4 == _lib.load().cednerf_dp_ctrl_bytes()
    assert ctypes.sizeof(_lib.DpPeers) == 8 + 8 * 8
    assert ctypes.sizeof(_lib.RenderRound) == _lib.load().cednerf_render_round_bytes() == 344
    # world, rank, grad[8], n_out (+ padding), p32_out[8], p16_out[8], m, v, lo, hi, lr, weight_decay, grad_div (+ padding),
    # grad_mc, p16_mc
    assert ctypes.sizeof(_lib.DpAdam) == 8 + 64 + 8 + 64 + 64 + 16 + 16 + 16 + 16
    # world, n_tensors, grad[8], p/m/v[8], off[8], n[8], lr[8], weight_decay[8], grad_div (+ padding), chunk_begin[9]
    assert ctypes.sizeof(_lib.DpSmall) == 8 + 64 + 3 * 64 + 64 + 64 + 32 + 32 + 8 + 72
    assert ctypes.sizeof(_lib.FieldDesc) == 6 * 4 + 4 + 3 * 4 + 4 * ctypes.sizeof(_lib.MlpDesc) + ctypes.sizeof(_lib.GridLevels)


def test_level_geometry_matches_oracle_and_survey():
    import math

    from cednerf_b200 import ops
    from oracle import tcnn_ref as tc

    for dst, log2_t in ((8192, 21), (4096, 21), (1024, 21), (256, 12)):
        log_b = math.log(dst / 16) / 15
        g, total, info = ops.grid_levels(16, 16, log_b, 2 ** log2_t)
        scales, ress, sizes, offsets, hashed, tot = tc.grid_levels(16, 16, log_b, 2 ** log2_t)
        assert total == tot and [i[1] for i in info] == ress and [i[2] for i in info] == sizes
        assert [i[3] for i in info] == offsets and [i[4] for i in info] == hashed
        assert [g.scale[l] for l in range(16)] == [float(s) for s in scales]
    _, total, info = ops.grid_levels(16, 16, math.log(8192 / 16) / 15, 2 ** 21)
    assert total == 23928800 and [i[1] for i in info][:6] == [16, 25, 37, 56, 85, 128]  # SURVEY.md E0


def test_mlp_descriptor_matches_oracle_shapes():
    from cednerf_b200 import ops
    from oracle import tcnn_ref as tc

    for n_in, n_out, h in ((32, 6, 3), (41, 16, 1), (19, 3, 2), (32, 32, 1), (32, 1, 1)):
        d, n_params = ops.mlp_desc(n_in, n_out, 64, h)
        shapes = tc.mlp_layer_shapes(n_in, n_out, 64, h)
        assert d.n_layers == len(shapes) and n_params == sum(o * i for o, i in shapes)
        assert [(d.dim_out[l], d.dim_in[l]) for l in range(d.n_layers)] == shapes
        assert d.image_bytes == sum(o for o, _ in shapes) * 128
    with pytest.raises(NotImplementedError):
        ops.mlp_desc(32, 3, 128, 2)


def test_no_cpu_fallback():
    import cednerf_b200 as cb

    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(RuntimeError):
        cb.nerfacc.ray_aabb_intersect(torch.zeros(4, 3), torch.ones(4, 3), torch.zeros(1, 6))
    with pytest.raises(RuntimeError):
        cb.tcnn.Network(32, 16, {"otype": "FullyFusedMLP", "n_neurons": 64, "n_hidden_layers": 1})(torch.zeros(8, 32))
    with pytest.raises(RuntimeError):
        cb.ops.time_embed(torch.zeros(3, 1))
    # optimiser and loss of the training loop: same rule
    p = torch.nn.Parameter(torch.zeros(16))
    p.grad = torch.ones(16)
    with pytest.raises(RuntimeError):
        cb.optim.FusedAdam([p], lr=1e-2, eps=1e-15).step()
    with pytest.raises(RuntimeError):
        cb.optim.FusedAdam([p], amsgrad=True)
    ex = {"rgbs": torch.zeros(5, 3), "weights": torch.zeros(5), "ray_indices": torch.zeros(5, dtype=torch.long),
          "latent_losses": torch.zeros(4, 32)}
    with pytest.raises(RuntimeError):
        cb.losses.training_loss(torch.zeros(4, 3), torch.zeros(4, 1), torch.zeros(4, 3), [ex])
    est = cb.OccGridEstimator([-1, -1, -1, 1, 1, 1], resolution=16, levels=1)
    with pytest.raises(RuntimeError):
        est.mark_invisible_cells(torch.eye(3)[None], torch.eye(4)[None], 8, 8, 0.1)
    # the importance-sampled batch of the DyNeRF loader and the 4-D encoder: same rule
    with pytest.raises(RuntimeError):
        cb.importance.weighted_sample(torch.rand(100), 10)
    with pytest.raises(RuntimeError):   # host tensors are refused when the sampler is built
        cb.importance.ImportanceSampler(torch.zeros(2, 8, 8, 3, dtype=torch.uint8), torch.eye(4)[None, :3].repeat(2, 1, 1),
                                        torch.eye(3), torch.zeros(2, 1), torch.ones(2 * 4 * 4), 2, num_rays=16)
    with pytest.raises(ValueError):   # argument checks come before any launch
        cb.importance.ImportanceSampler(torch.zeros(2, 8, 8, 3), torch.eye(4)[None, :3], torch.eye(3), torch.zeros(2, 1),
                                        torch.ones(32), 2)
    with pytest.raises(RuntimeError):
        cb.hash_encoder.HashEncoder4D(max_params=2 ** 8, levels=4, base_res=4.0, max_res=16.0)(torch.rand(5, 4))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "cednerf_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, os.path.join(dirpath, f)


def test_module_surface_mirrors_reference_names():
    import cednerf_b200 as cb

    for name in ("traverse_grids", "ray_aabb_intersect", "render_weight_from_density", "accumulate_along_rays",
                 "render_transmittance_from_density", "render_visibility_from_density", "OccGridEstimator"):
        assert hasattr(cb.nerfacc, name)
    assert hasattr(cb.nerfacc.volrend, "accumulate_along_rays_")
    from cednerf_b200.nerfacc.estimators.occ_grid import OccGridEstimator  # noqa: F401  (train_real.py:27)

    for name in ("Encoding", "Network", "NetworkWithInputEncoding"):
        assert hasattr(cb.tcnn, name)
    for name in ("render_image", "render_image_test", "trunc_exp", "set_random_seed", "Rays", "namedtuple_map"):
        assert hasattr(cb.utils, name)
    est = cb.OccGridEstimator([-1, -1, -1, 1, 1, 1], resolution=128, levels=4)
    assert est.binaries.shape == (4, 128, 128, 128) and est.occs.numel() == 4 * 128 ** 3
    assert torch.equal(est.aabbs[-1], torch.tensor([-8.0, -8, -8, 8, 8, 8]))
    field = cb.DNGPradianceField(est.aabbs[-1], dst_resolution=8192, log2_hashmap_size=21, use_feat_predict=True,
                                 use_time_embedding=True, use_time_attenuation=True, use_div_offsets=True)
    assert field.hash_encoder.params.numel() == 2 * 23928800
    assert field.mlp_base.n_input_dims == 41 and field.mlp_head.n_input_dims == 19
    assert field.xyz_wrap.n_output_dims == 6 and field.mlp_feat_prediction.n_output_dims == 32


def test_state_dict_has_the_reference_checkpoint_key_set():
    """A `model.pth` written by train_real.py:438 must load with strict=True: tcnn modules save ONE flat `params` each
    (NetworkWithInputEncoding included), the two time encoders save their `scales` buffers (cednerf/encoder.py:18-20,
    :55-60) and both exist whenever -te is on (cednerf/model.py:266-267)."""
    import cednerf_b200 as cb

    field = cb.DNGPradianceField([-1, -1, -1, 1, 1, 1], n_levels=4, log2_hashmap_size=10, dst_resolution=64,
                                 use_feat_predict=True, use_weight_predict=True, use_time_embedding=True,
                                 use_time_attenuation=True, use_div_offsets=True)
    want = {"aabb", "xyz_wrap.params", "direction_encoding.params", "hash_encoder.params", "time_encoder.scales",
            "time_encoder_feat.scales", "time_encoder_feat.scales_move", "mlp_base.params", "mlp_head.params",
            "mlp_feat_prediction.params", "mlp_weight_prediction.params"}
    sd = field.state_dict()
    assert set(sd) == want
    assert sd["time_encoder_feat.scales_move"].tolist() == [0, 2, 8, 24] and sd["time_encoder.scales"].tolist() == [1, 2, 4, 8]
    # what an optimiser sees: each tensor once, the NetworkWithInputEncoding parameters included
    names = [n for n, _ in field.named_parameters()]
    assert len(names) == len(set(names)) == 7 and "xyz_wrap.params" in names
    # round trip through a fresh module, strict
    other = cb.DNGPradianceField([-1, -1, -1, 1, 1, 1], n_levels=4, log2_hashmap_size=10, dst_resolution=64,
                                 use_feat_predict=True, use_weight_predict=True, use_time_embedding=True,
                                 use_time_attenuation=True, use_div_offsets=True, seed=7)
    other.load_state_dict({k: v.clone() for k, v in sd.items()}, strict=True)
    assert torch.equal(other.xyz_wrap.params, field.xyz_wrap.params)
    assert other.xyz_wrap.network.params is other.xyz_wrap.params  # the helper borrows the registered Parameter


def test_workload_initial_state_is_the_module_initialisation():
    """bench.py's two arms start from workload.initial_state (pure torch): it must be bit-identical to what
    DNGPradianceField's own constructors draw, key for key, and the pose generators must give unit directions."""
    import cednerf_b200 as cb
    from cednerf_b200 import workload as w

    for cfg in (w.TINY, w.DNERF):
        est = cb.OccGridEstimator(list(cfg.roi_aabb), resolution=cfg.occ_res, levels=cfg.occ_levels)
        sd, st = cb.DNGPradianceField(est.aabbs[-1], **w.field_kwargs(cfg)).state_dict(), w.initial_state(cfg)
        assert set(sd) == set(st)
        for k in sd:
            assert torch.equal(sd[k].float(), st[k].float()), (cfg.name, k)
    poses = w.spiral_poses(w.DYNERF, 300)
    assert poses.shape == (300, 3, 4) and len({tuple(p[:, 3].tolist()) for p in poses}) == 300  # 300 distinct positions
    r = poses[:, :, :3]
    assert torch.allclose(r @ r.transpose(1, 2), torch.eye(3).expand(300, 3, 3), atol=1e-5)       # rotations
    o, d = w.pose_rays(w.TINY, poses[17])
    assert o.shape == d.shape == (w.TINY.width * w.TINY.height, 3)
    assert torch.allclose(d.norm(dim=-1), torch.ones(d.shape[0]), atol=1e-6) and bool((d[:, 2] > 0.5).all())
    c = w.orbit_pose(4.0, 1.0)
    o, d = w.pose_rays(w.DNERF, c, True)
    centre = d[(w.DNERF.height // 2) * w.DNERF.width + w.DNERF.width // 2]
    assert torch.allclose(centre, -c[:, 3] / 4.0, atol=2e-3)  # the centre pixel looks at the origin
