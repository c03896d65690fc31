"""The device-resident marching rounds of render_image_test (csrc/render_round.cu) against the oracle, exactly.

A round marches the alive rays with a sample limit k, replays the recorded runs of each ray, and sends the rays with more
than RUN_CAP runs through the full-march fallback fill.  Blob scenes never give a ray that many runs; the grids here do
(a checkerboard alternates occupied and empty cells at every cell crossing), and a field whose networks are zeroed has the
same density and colour everywhere, so whole frames can be compared with the oracle without any tolerance for the
network: the sample total exactly, the images to fp32 compositing order.
"""
import dataclasses
import math
import types

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import cednerf_ref as cr  # noqa: E402
from oracle import nerfacc_ref as nf  # noqa: E402

DEV = "cuda:0"
SIGMA = math.exp(-1.0)   # trunc_exp(0 - 1): the density of a field whose density network is zero


@pytest.fixture(scope="module")
def cb():
    import cednerf_b200

    return cednerf_b200


def checkerboard(levels, res):
    i = torch.arange(res)
    one = ((i[:, None, None] + i[None, :, None] + i[None, None, :]) % 2) == 0
    return one[None].expand(levels, res, res, res).contiguous()


def grid_of(kind, levels, res):
    """bool [L,R,R,R] with the outermost shell of cells of the outermost level empty (no sample lies near the box of the
    field, so its in-box selector never decides anything)."""
    if kind == "checker":
        b = checkerboard(levels, res)
    elif kind == "full":
        b = torch.ones(levels, res, res, res, dtype=torch.bool)
    elif kind == "empty":
        b = torch.zeros(levels, res, res, res, dtype=torch.bool)
    else:   # one occupied cell near the centre of level 0
        b = torch.zeros(levels, res, res, res, dtype=torch.bool)
        b[0, res // 2, res // 2 - 1, res // 2] = True
    b = b.clone()
    b[-1, 0], b[-1, -1], b[-1, :, 0], b[-1, :, -1], b[-1, :, :, 0], b[-1, :, :, -1] = (False,) * 6
    return b


# ------------------------------------------------------------------------------------------- one round at the entry points
@pytest.mark.parametrize("run_cap", [1, 3, 16])
def test_one_round_at_the_entry_points_matches_the_oracle(cb, run_cap):
    """The four marching launches of a round (count, capped scan, fill from runs, full-march fallback fill) on a seeded
    alive list: every slot's range holds exactly its ray's oracle samples, nothing is left unwritten, and near_term ends
    as the termination planes.  Launches no field kernel."""
    from cednerf_b200 import ops
    from cednerf_b200._lib import call, ptr, stream

    levels, res, n = 2, 64, 4096
    n_alive = n // 32                                  # k = n // n_alive = 32 samples per ray this round
    step, cone, far = 0.6 * 2.0 / res, 0.004, 1e10     # 1-2 samples per occupied level-0 cell: short runs
    g = torch.Generator().manual_seed(7)
    est = nf.OccGridEstimator([-1.0] * 3 + [1.0] * 3, resolution=res, levels=levels)
    binaries = checkerboard(levels, res)
    o = torch.tensor([0.0, 0.0, -2.5]) + (torch.rand(n, 3, generator=g) - 0.5) * 0.6
    d = torch.nn.functional.normalize((torch.rand(n, 3, generator=g) - 0.5) * 1.2 - o, dim=-1)
    near = 0.2 + torch.rand(n, generator=g) * step
    perm = torch.randperm(n, generator=g)
    mask = torch.zeros(n, dtype=torch.bool)
    mask[perm[:n_alive]] = True
    t_mins, t_maxs, hits = nf.ray_aabb_intersect(o, d, est.aabbs)
    ts, ti = nf.sort_boundaries(t_mins, t_maxs)
    k = n // n_alive
    iv, sm, term = nf.traverse_grids(o, d, binaries, est.aabbs, near, torch.full((n,), far), step, cone, k, True, mask,
                                     ts, ti, hits)
    want_t0, want_t1 = iv.vals[iv.is_left], iv.vals[iv.is_right]
    want_r, want_cnt = sm.ray_indices[sm.is_valid], sm.packed_info[:, 1]
    assert want_t0.numel() == want_r.numel() == int(want_cnt.sum())

    to = lambda t: t.to(DEV).contiguous()
    o_g, d_g, aabbs, ts_g, ti_g, hits_g = to(o), to(d), to(est.aabbs), to(ts), to(ti), to(hits)
    bits = ops.pack_occupancy(to(binaries))
    coarse = ops.occupancy_coarse(bits, levels, res)
    near_term = to(near)
    n_bound = 2 * n_alive                              # the live part of the list is state[0], the launches are larger
    alive = to(perm[:n_bound].to(torch.int32))
    I32, I64 = torch.int32, torch.int64
    state = torch.zeros(8, dtype=I32, device=DEV)
    state[3] = n_alive
    total = torch.zeros(1, dtype=I64, device=DEV)
    n_sm = torch.empty(n_bound, dtype=I32, device=DEV)
    run_t = torch.empty(n_bound, run_cap, device=DEV)
    run_n = torch.empty(n_bound, run_cap, dtype=I32, device=DEV)
    n_runs = torch.empty(n_bound, dtype=I32, device=DEV)
    overflow = torch.empty(n_bound, dtype=torch.bool, device=DEV)
    cap = n_alive * k
    t0 = torch.full((cap,), float("nan"), device=DEV)
    t1 = torch.full((cap,), float("nan"), device=DEV)
    ridx = torch.full((cap,), -1, dtype=I64, device=DEV)
    offsets = torch.empty(n_bound + 1, dtype=I64, device=DEV)
    totals = torch.zeros(2, dtype=I64, device=DEV)
    ws = torch.empty(max(int(cb._lib.load().cednerf_scan_workspace_bytes(n_bound)) // 8, 1), dtype=I64, device=DEV)
    st = stream()
    call("cednerf_render_round_begin", ptr(state), n, 1024, 1, None, ptr(total), st)
    call("cednerf_march_round", 0, ptr(o_g), ptr(d_g), n_bound, ptr(bits), ptr(aabbs), levels, res, ptr(near_term), far,
         step, cone, ptr(ts_g), ptr(ti_g), ptr(hits_g), ptr(alive), ptr(state), None, None, None, None, None, ptr(n_sm),
         ptr(run_t), ptr(run_n), ptr(n_runs), run_cap, ptr(coarse), st)
    call("cednerf_exclusive_scan_capped", ptr(n_sm), n_bound, cap, ptr(offsets), ptr(totals), ptr(ws), st)
    call("cednerf_march_fill_runs_round", n_bound, ptr(offsets), ptr(n_sm), ptr(run_t), ptr(run_n), ptr(n_runs), run_cap,
         step, cone, ptr(alive), ptr(state), ptr(t0), ptr(t1), ptr(ridx), ptr(overflow), st)
    call("cednerf_march_round", 1, ptr(o_g), ptr(d_g), n_bound, ptr(bits), ptr(aabbs), levels, res, ptr(near_term), far,
         step, cone, ptr(ts_g), ptr(ti_g), ptr(hits_g), ptr(alive), ptr(state), ptr(overflow), ptr(offsets), ptr(t0),
         ptr(t1), ptr(ridx), None, None, None, None, run_cap, ptr(coarse), st)
    torch.cuda.synchronize()

    assert state.tolist()[:2] == [n_alive, k]
    assert bool(overflow[:n_alive].any()), "no ray took the full-march fallback"
    assert not bool(overflow[n_alive:].any())
    tot = int(totals[0])
    assert tot == int(totals[1]) == want_r.numel()
    slots_cnt, offs = n_sm.cpu().long(), offsets.cpu()
    assert torch.equal(slots_cnt[n_alive:], torch.zeros(n_bound - n_alive, dtype=I64))
    assert torch.equal(offs[1:] - offs[:-1], slots_cnt) and int(offs[-1]) == tot
    slot_ray = perm[:n_alive]
    assert torch.equal(slots_cnt[:n_alive], want_cnt[slot_ray])
    # every slot's range, taken in ray order, is the oracle's packed sample set (which is sorted by ray)
    by_ray = torch.argsort(slot_ray)
    idx = torch.cat([torch.arange(int(offs[s]), int(offs[s]) + int(slots_cnt[s])) for s in by_ray.tolist()])
    g0, g1, gr = t0.cpu(), t1.cpu(), ridx.cpu()
    assert not bool(torch.isnan(g0[:tot]).any() | torch.isnan(g1[:tot]).any() | (gr[:tot] < 0).any()), "unwritten slots"
    assert torch.equal(gr[idx], want_r)
    assert torch.equal(g0[idx], want_t0) and torch.equal(g1[idx], want_t1)
    # near_term: the termination planes of the alive rays, the start planes of the others
    got_near = near_term.cpu()
    assert torch.equal(got_near[mask], term[mask])
    assert torch.equal(got_near[~mask], near[~mask])


# ------------------------------------------------------------------------------------------- whole frames
class ConstField:
    """The oracle side of a field with zeroed networks: density e^-1 and colour sigmoid(0) = 0.5 at every sample."""

    training = False

    def __init__(self, sigma, rgb):
        self.sigma, self.rgb = float(sigma), float(rgb)

    def query_density(self, x, t):
        return {"density": torch.full((x.shape[0], 1), self.sigma)}

    def __call__(self, x, t, d):
        return torch.full((x.shape[0], 3), self.rgb), self.query_density(x, t)


SCENE = dict(roi_aabb=(-0.5, -0.5, -0.5, 0.5, 0.5, 0.5), near_plane=0.05, render_step_size=0.04, alpha_thre=0.0)
_FIELDS = {}


def const_field(cb, levels):
    """The product's DNGPradianceField (workload.build_scene) with xyz_wrap, mlp_base and mlp_head zeroed: no offset,
    raw density 0, colour logits 0.  Its box is the outermost level's."""
    if levels not in _FIELDS:
        from cednerf_b200 import workload as w

        cfg = dataclasses.replace(w.TINY, occ_levels=levels, occ_res=16, **SCENE)
        est, field = w.build_scene(cfg, DEV, cb, seed=42)
        field.eval()
        with torch.no_grad():
            for m in (field.xyz_wrap, field.mlp_base, field.mlp_head):
                m.params.zero_()
        # the value every sample gets, checked with the fused kernel the rounds use
        g = torch.Generator().manual_seed(3)
        m = 4096
        lo, hi = est.aabbs[-1, :3].cpu() * 0.9, est.aabbs[-1, 3:].cpu() * 0.9
        x = lo + torch.rand(m, 3, generator=g) * (hi - lo)
        dr = torch.nn.functional.normalize(torch.randn(m, 3, generator=g), dim=-1)
        tt = torch.rand(m, generator=g) * 0.1
        packed = (torch.arange(m, device=DEV), (tt - 0.01).to(DEV), (tt + 0.01).to(DEV), (x - dr * tt[:, None]).to(DEV),
                  dr.to(DEV))
        sigma, rgb = field.fused_query(m, packed=packed, timestamps=torch.tensor([[0.4]], device=DEV), t_stride=0,
                                       sigma_only=False)
        torch.testing.assert_close(sigma.cpu(), torch.full((m,), SIGMA), rtol=2e-7, atol=0)
        assert torch.equal(rgb.cpu(), torch.full((m, 3), 0.5))
        _FIELDS[levels] = (field, est.aabbs.clone())
    return _FIELDS[levels]


def ray_set(levels):
    """A 16 x 16 pinhole crop plus rays at the edges of the marcher: exactly-zero direction components of both signs,
    origins inside the grids and on cell planes, rays that miss every box, rays grazing box faces."""
    outer = 0.5 * 2 ** (levels - 1)
    focal = 20.0 / outer                               # the outermost box fills most of the crop, its corners miss
    v, u = torch.meshgrid(torch.arange(16.0), torch.arange(16.0), indexing="ij")
    dc = torch.stack([(u - 7.5) / focal, (v - 7.3) / focal, torch.ones_like(u)], -1).reshape(256, 3)
    dc = torch.nn.functional.normalize(dc, dim=-1)
    oc = torch.tensor([0.05, 0.03, -3.0]).expand(256, 3)
    z = 0.0
    extra = [  # (origin, direction)
        ((0.1, 0.2, -3.0), (z, z, 1.0)), ((0.1, -0.2, -3.0), (-z, -z, 1.0)), ((0.13, -3.0, 0.07), (z, 1.0, -z)),
        ((0.21, -0.17, 3.0), (-z, z, -1.0)), ((-3.0, 0.11, -0.06), (1.0, -z, z)),
        ((0.1, -0.2, 0.05), (0.3, 0.5, 0.81)), ((0.0, 0.0, 0.0), (1.0, 2.0, 3.0)),          # origins inside the grids
        ((0.25, 0.125, 0.0), (z, 0.6, 0.8)), ((0.25, 0.1, -3.0), (z, z, 1.0)),           # on cell planes
        ((0.125, -0.25, 0.375), (-0.4, 0.1, 0.3)),
        ((5.0, 5.0, 5.0), (1.0, z, z)), ((0.0, 0.0, -3.0), (z, 1.0, z)), ((9.0, 0.0, 0.0), (1.0, 0.2, 0.1)),  # misses
        ((-3.0, outer, 0.1), (1.0, z, z)), ((-3.0, 0.5, 0.1), (1.0, z, z)),              # grazing box faces
        ((-3.0, outer - 1e-6, -outer + 1e-6), (1.0, z, z)), ((0.2, -3.0, outer), (z, 1.0, z)),
        ((0.3, -0.2, -3.0), (-0.29, 0.19, 3.01)), ((-2.0, 1.0, 2.0), (2.01, -1.01, -1.99)),  # through grid_of's single cell
    ]
    oe = torch.tensor([e[0] for e in extra])
    de = torch.tensor([e[1] for e in extra])
    de = de / torch.linalg.norm(de, dim=-1, keepdim=True)   # (keeps the sign of the zero components)
    return torch.cat([oc, oe]), torch.cat([dc, de])


def render_ours(cb, monkeypatch, field, aabbs, binaries, o, d, max_samples, cone, path, run_cap, lag):
    from cednerf_b200 import ops, utils as U

    est = types.SimpleNamespace(aabbs=aabbs.to(DEV), binaries=binaries.to(DEV))
    with monkeypatch.context() as mp:
        mp.setattr(ops.MarchInputs, "RUN_CAP", run_cap)
        mp.setattr(U, "_ROUND_LAG", lag)
        mp.setattr(U, "_DEVICE_ROUNDS", path != "host")
        mp.setattr(U, "_ROUND_BY_PARTS", path == "parts")
        out = cb.render_image_test(max_samples, field, est, cb.Rays(o.to(DEV), d.to(DEV)), render_bkgd=BKGD.to(DEV),
                                   timestamps=torch.tensor([[0.4]], device=DEV), cone_angle=cone,
                                   near_plane=SCENE["near_plane"], render_step_size=SCENE["render_step_size"])
    torch.cuda.synchronize()
    return out


def render_oracle(aabbs, binaries, o, d, max_samples, cone):
    est = types.SimpleNamespace(aabbs=aabbs.cpu(), binaries=binaries.cpu())
    return cr.render_image_test(max_samples, ConstField(SIGMA, 0.5), est, cr.Rays(o, d), render_bkgd=BKGD,
                                timestamps=torch.tensor([[0.4]]), cone_angle=cone, near_plane=SCENE["near_plane"],
                                render_step_size=SCENE["render_step_size"])


BKGD = torch.tensor([0.1, 0.6, 0.9])
# (path, RUN_CAP, _ROUND_LAG): one call per round, the eight launches as separate calls, and the host-driven loop (which
# reads every round's alive count, so has no lag)
VARIANTS = ([(path, cap, lag) for path in ("rounds", "parts") for cap in (16, 1) for lag in (4, 0)]
            + [("host", cap, 4) for cap in (16, 1)])


def check_frame(got, want, what):
    assert got[3] == want[3], (what, got[3], want[3])
    for i in range(3):
        assert got[i].shape == want[i].shape, what
        torch.testing.assert_close(got[i].cpu(), want[i], rtol=0, atol=1e-5, msg=lambda m: f"{what} output {i}: {m}")


def run_matrix(cb, monkeypatch, kind, levels, res, cone, sample_limits=(1, 7, 1024)):
    field, aabbs = const_field(cb, levels)
    binaries = grid_of(kind, levels, res)
    o, d = ray_set(levels)
    for max_samples in sample_limits:
        want = render_oracle(aabbs, binaries, o, d, max_samples, cone)
        assert float(want[1].max()) < 0.99   # no ray comes near early termination: the alive set is pure marching
        outs = []
        for path, run_cap, lag in VARIANTS:
            what = (kind, levels, res, cone, max_samples, path, run_cap, lag)
            got = render_ours(cb, monkeypatch, field, aabbs, binaries, o, d, max_samples, cone, path, run_cap, lag)
            check_frame(got, want, what)
            outs.append(got)
        for got in outs[1:]:   # our paths among themselves: up to the order of a ray's sums inside a lane group
            for i in range(3):
                torch.testing.assert_close(got[i], outs[0][i], rtol=0, atol=2e-6)
    if kind != "empty":
        assert want[3] > 0
    # fewer rays: a partial warp, and a single ray
    for m in (129, 1):
        want = render_oracle(aabbs, binaries, o[-m:], d[-m:], 1024, cone)
        got = render_ours(cb, monkeypatch, field, aabbs, binaries, o[-m:], d[-m:], 1024, cone, "rounds", 1, 4)
        check_frame(got, want, (kind, levels, res, cone, m))


@pytest.mark.parametrize("cone", [0.0, 0.004])
@pytest.mark.parametrize("res", [16, 64])
@pytest.mark.parametrize("levels", [1, 3])
@pytest.mark.parametrize("kind", ["checker", "full", "empty", "single"])
def test_whole_frames_with_a_constant_field_match_the_oracle(cb, monkeypatch, kind, levels, res, cone):
    """render_image_test on every path (one call per round, eight calls per round, the host-driven loop) with the
    full-march fallback for every ray with more than one run, against oracle.cednerf_ref.render_image_test."""
    run_matrix(cb, monkeypatch, kind, levels, res, cone)


@pytest.mark.parametrize("res", [18, 30])
def test_resolutions_that_are_not_a_multiple_of_four(cb, monkeypatch, res):
    """No 4^3-block bits at such resolutions: the rounds march every cell (and the bit field has a partial last word)."""
    for levels in (1, 3):
        run_matrix(cb, monkeypatch, "checker", levels, res, 0.004, sample_limits=(7, 1024))


# ------------------------------------------------------------------------------------------- interleaved frames, cold caches
def test_interleaved_frames_build_shared_caches_on_the_callers_stream(cb, monkeypatch):
    """render_images_test after the parameters and the occupancy changed (every eval after training steps): the bit
    field, the 4^3-block bits, the fp16 hash table and the three weight images are built once, on the calling stream,
    before the frames fork onto their own streams - and every frame equals render_image_test bit for bit."""
    from cednerf_b200 import nerfacc, ops, workload as w

    cfg = w.TINY
    rk = w.render_kwargs(cfg)
    est, field = w.build_scene(cfg, DEV, cb, seed=42)
    est.eval(), field.eval()
    poses = w.spiral_poses(cfg, 4)
    K = [[cfg.focal, 0.0, cfg.width / 2], [0.0, cfg.focal, cfg.height / 2], [0.0, 0.0, 1.0]]
    bk = torch.tensor([0.2, 0.4, 0.6], device=DEV)
    ts = [torch.tensor([[k / 4.0]], device=DEV) for k in range(4)]
    rows = [cfg.height, 37, 20, 45]                    # frames of different ray counts

    def rays_of(k):
        r = cb.utils.generate_rays(K, poses[k].to(DEV), cfg.width, cfg.height)
        return cb.Rays(r.origins[:rows[k]].reshape(-1, 3), r.viewdirs[:rows[k]].reshape(-1, 3))

    def cold():
        torch.cuda.synchronize()
        for t in (est.binaries, field.hash_encoder.params, field.xyz_wrap.params, field.mlp_base.params,
                  field.mlp_head.params):
            torch.autograd.graph.increment_version(t)

    produced = []

    def recorder(name, fn):
        def wrapped(*a, **kw):
            produced.append((name, torch.cuda.current_stream()))
            return fn(*a, **kw)
        return wrapped

    def coarse_recorder(fn):
        def wrapped(bits, *a):
            before = getattr(bits, "_cednerf_coarse", None)
            out = fn(bits, *a)
            if out is not None and (before is None or before[1] is not out):
                produced.append(("coarse", torch.cuda.current_stream()))
            return out
        return wrapped

    cold()
    want = [cb.render_image_test(1024, field, est, rays_of(k), render_bkgd=bk, timestamps=ts[k], **rk) for k in range(4)]
    assert len({int(x[0].numel()) for x in want}) == 4 and all(x[3] > 0 for x in want)
    monkeypatch.setattr(ops, "pack_occupancy", recorder("bits", ops.pack_occupancy))
    monkeypatch.setattr(ops, "occupancy_coarse", coarse_recorder(ops.occupancy_coarse))
    monkeypatch.setattr(ops, "cast_f16", recorder("table_f16", ops.cast_f16))
    monkeypatch.setattr(ops, "mlp_pack", recorder("weight_image", ops.mlp_pack))
    assert nerfacc.grid.ops is ops
    for _ in range(2):
        cold()
        produced.clear()
        main = torch.cuda.current_stream()
        got = cb.render_images_test(1024, field, est, [(lambda k=k: rays_of(k)) for k in range(4)], ts, concurrency=3,
                                    render_bkgd=bk, **rk)
        torch.cuda.synchronize()
        names = sorted(name for name, _ in produced)
        assert names == ["bits", "coarse", "table_f16", "weight_image", "weight_image", "weight_image"], names
        assert all(s == main for _, s in produced), [(name, s) for name, s in produced if s != main]
        for k in range(4):
            assert got[k][3] == want[k][3]
            for i in range(3):
                assert torch.equal(got[k][i], want[k][i]), (k, i)
