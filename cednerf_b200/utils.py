"""cednerf/utils.py surface: render_image (:46-150), render_image_test (:153-318), trunc_exp, set_random_seed."""
from __future__ import annotations

import collections
import random

import numpy as np
import torch

from . import nerfacc, ops
from .model import trunc_exp  # noqa: F401  (re-exported like cednerf/utils.py:43)
from .render import rendering

Rays = collections.namedtuple("Rays", ("origins", "viewdirs"))


def namedtuple_map(fn, tup):
    """datasets/utils.py:8-15."""
    return type(tup)(*(None if x is None else fn(x) for x in tup))


def set_random_seed(seed):
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)


def generate_rays(K, c2w, width: int, height: int, opengl: bool = False, x=None, y=None, image_id=None,
                  return_directions: bool = False):
    """Pixel -> ray generation of the reference's datasets (datasets/dnerf_3d_video_IS.py:330-358,
    datasets/dnerf_synthetic.py:196-224, gui.py:43-86) in one launch.  K: 3x3 intrinsics (host tensor / nested list);
    c2w: [n_cams, 3|4, 4] (or one [3|4, 4] pose) on the device.  Without x / y: every pixel of one frame, row-major
    (origins / viewdirs shaped [height, width, 3]); with them: one ray per (x[i], y[i], image_id[i])."""
    import ctypes  # noqa: F401

    from ._lib import call, ptr, stream

    c2w = c2w if c2w.dim() == 3 else c2w[None]
    c2w = ops._f32c(c2w)
    Kh = torch.as_tensor(K, dtype=torch.float32).cpu()
    fx, fy, cx, cy = float(Kh[0, 0]), float(Kh[1, 1]), float(Kh[0, 2]), float(Kh[1, 2])
    dev = c2w.device
    if x is None:
        n = int(width) * int(height)
        px = py = cam = None
    else:
        px, py = x.to(dev, torch.int64).contiguous(), y.to(dev, torch.int64).contiguous()
        cam = None if image_id is None else image_id.to(dev, torch.int64).contiguous()
        n = px.numel()
    o, d = torch.empty(n, 3, device=dev), torch.empty(n, 3, device=dev)
    dirs = torch.empty(n, 3, device=dev) if return_directions else None
    call("cednerf_generate_rays", ptr(px), ptr(py), ptr(cam), ptr(c2w), int(c2w.shape[1]), fx, fy, cx, cy, int(width),
         int(bool(opengl)), n, ptr(o), ptr(d), ptr(dirs), stream())
    if x is None:
        o, d = o.view(height, width, 3), d.view(height, width, 3)
        dirs = None if dirs is None else dirs.view(height, width, 3)
    return (Rays(o, d), dirs) if return_directions else Rays(o, d)


class FieldOccEval:
    """occ_eval_fn of the reference's training loop (train_real.py:324-328) as an object:

        occ_eval_fn = FieldOccEval(radiance_field, render_step_size)
        estimator.update_every_n_steps(step=step, occ_eval_fn=occ_eval_fn, occ_thre=1e-2)

    Called like the reference's closure it returns query_density(x, rand_t)["density"] * render_step_size.  Handed to
    cednerf_b200's OccGridEstimator it additionally lets `_update` run each level as ONE launch (cell -> jittered point
    -> field -> EMA-max, csrc/field.cu::cednerf_occ_update_level) instead of the fused density kernel plus ~10 element-wise
    launches per level.  `rng` (randint(high, n), rand(*shape)): the source of the random timestamps (default torch.rand);
    dp.SharedRng keeps data-parallel replicas identical."""

    def __init__(self, field, render_step_size: float, rng=None):
        self.field, self.step, self.rng = field, float(render_step_size), rng

    def rand_t(self, n: int, device):
        return torch.rand(n, 1, device=device) if self.rng is None else self.rng.rand(n, 1).to(device)

    def __call__(self, x):
        return self.field.query_density(x, self.rand_t(x.shape[0], x.device))["density"] * self.step


def _field_fns(field, rays, timestamps):
    def positions_of(t0, t1, ridx):
        o, d = rays.origins[ridx], rays.viewdirs[ridx]
        x = o + d * (t0 + t1)[:, None] / 2.0
        t = timestamps[ridx] if field.training else timestamps.expand_as(x[:, :1])
        return x, t, d

    def fused(t0, t1, ridx, sigma_only):
        """One launch from packed samples: positions, encodings and networks never leave the SM."""
        per_ray = field.training and timestamps.numel() == rays.origins.shape[0]
        counts = ops.counts_of(ridx)
        return field.fused_query(t0.numel(), packed=(ridx, t0, t1, rays.origins, rays.viewdirs), timestamps=timestamps,
                                 t_stride=1 if per_ray else 0, sigma_only=sigma_only,
                                 n_dev=None if counts is None else counts[1])

    def can_fuse(t0):
        ok = (not torch.is_grad_enabled()) and t0.numel() > 0 and getattr(field, "fused_supported", lambda: False)()
        return ok and (timestamps.numel() == 1 or (field.training and timestamps.numel() == rays.origins.shape[0]))

    def sigma_fn(t0, t1, ridx):
        if can_fuse(t0):
            return fused(t0, t1, ridx, True)[0]
        x, t, _ = positions_of(t0, t1, ridx)
        return field.query_density(x, t)["density"].squeeze(-1)

    def rgb_sigma_fn(t0, t1, ridx):
        if (field.training and torch.is_grad_enabled() and t0.numel() > 0
                and getattr(field, "fused_train_supported", lambda: False)()
                and (timestamps.numel() == 1 or timestamps.numel() == rays.origins.shape[0])):
            return field.fused_train(ridx, t0, t1, rays.origins, rays.viewdirs, timestamps,
                                     1 if timestamps.numel() == rays.origins.shape[0] else 0)
        if can_fuse(t0) and not field.training:
            sigma, rgb = fused(t0, t1, ridx, False)
            return rgb, {"density": sigma[:, None]}
        x, t, d = positions_of(t0, t1, ridx)
        return field(x, t, d)

    return sigma_fn, rgb_sigma_fn


def render_image(radiance_field, estimator, rays, near_plane=0.0, far_plane=1e10, render_step_size=1e-3,
                 render_bkgd=None, cone_angle=0.0, alpha_thre=0.0, test_chunk_size=8192, timestamps=None,
                 jitter=None, device_counts=False):
    """-> (rgb, acc, depth, n_rendering_samples, extras list).  `jitter` (optional, [n_rays] in [0,1)) replaces the
    stratified random draw so that parity tests do not depend on the RNG stream.

    device_counts=True (training, fused field only): nothing is read back by the host during the call.  The packed
    sample tensors in `extras` are then allocated at a capacity derived from earlier batches, only their first
    n_rendering_samples rows are live, and n_rendering_samples is a 0-dim int64 DEVICE tensor (the reference's training
    loop reads it once per step for its ray-count controller, train_real.py:354-360: `int(n)` does that)."""
    shape = rays.origins.shape
    rays = Rays(rays.origins.reshape(-1, 3), rays.viewdirs.reshape(-1, 3))
    n = rays.origins.shape[0]
    chunk = n if radiance_field.training else test_chunk_size
    outs, infos = [], []
    for i in range(0, n, chunk):
        cr = Rays(rays.origins[i:i + chunk], rays.viewdirs[i:i + chunk])
        ts = timestamps[i:i + chunk] if (radiance_field.training and timestamps is not None) else timestamps
        sigma_fn, rgb_sigma_fn = _field_fns(radiance_field, cr, ts)
        ridx, t0, t1 = estimator.sampling(cr.origins, cr.viewdirs, sigma_fn=sigma_fn, near_plane=near_plane,
                                          far_plane=far_plane, render_step_size=render_step_size,
                                          stratified=radiance_field.training, cone_angle=cone_angle,
                                          alpha_thre=alpha_thre, jitter=None if jitter is None else jitter[i:i + chunk],
                                          device_counts=bool(device_counts and radiance_field.training and
                                                             getattr(radiance_field, "fused_train_supported", lambda: False)()
                                                             and timestamps is not None and torch.is_grad_enabled()))
        rgb, opac, depth, extras = rendering(t0, t1, ridx, cr.origins.shape[0], rgb_sigma_fn=rgb_sigma_fn,
                                             render_bkgd=render_bkgd)
        extras.update(ray_indices=ridx, t_starts=t0, t_ends=t1)
        counts = ops.counts_of(ridx)
        outs.append((rgb, opac, depth, len(t0) if counts is None else counts[1].view(())))
        infos.append(extras)
    rgb, opac, depth = (torch.cat([o[k] for o in outs], 0) for k in range(3))
    return (rgb.view(*shape[:-1], -1), opac.view(*shape[:-1], -1), depth.view(*shape[:-1], -1),
            outs[0][3] if len(outs) == 1 else sum(o[3] for o in outs), infos)


_DEVICE_ROUNDS = True   # False: the host-driven rounds below (one host read per round, as the reference does)
_ROUND_LAG = 4          # rounds the host may run ahead of the newest alive count it has seen
_ROUND_BY_PARTS = bool(int(__import__("os").environ.get("CEDNERF_ROUND_BY_PARTS", "0")))  # diagnostic: eight calls per round


def _render_rounds_gen(max_samples, field, rays, bits, aabbs, res, near, far_plane, step, cone, early_stop_eps,
                       timestamps, t_sorted, t_indices, hits, min_samples, rgb, opacity, depth):
    """The marching rounds of cednerf/utils.py:224-304 with the alive-ray list, the per-round k and the termination test
    on the device (csrc/march.cu: cednerf_render_round_begin / cednerf_march_round / cednerf_march_fill_runs_round,
    csrc/composite.cu: cednerf_render_round_composite).  The host enqueues rounds and reads a copy of the round state
    that is up to _ROUND_LAG rounds old: it tells it when every ray is done and how far the launches can shrink
    (the alive count never grows).  Rays are marched in alive-list order; the list is the ORDERED compaction of the
    survivors, so neighbouring lanes keep neighbouring pixels and a round's warps are dense however few rays survive;
    per ray the samples, their order and the arithmetic are those of the host-driven loop.

    A generator: it yields after enqueuing each round (and while it waits for the final total), so that a scheduler can
    interleave the rounds of several frames on several streams (render_images_test); it returns the sample total."""
    from ._lib import call, ptr, stream

    n, dev = rays.origins.shape[0], rays.origins.device
    o, d = ops._f32c(rays.origins), ops._f32c(rays.viewdirs)
    aabbs_c = ops._f32c(aabbs)
    n_levels = aabbs_c.shape[0]
    coarse = ops.occupancy_coarse(bits, n_levels, res)
    I32, I64 = torch.int32, torch.int64
    # n_alive * k <= n when k = n // n_alive, and <= min_samples * n_alive otherwise
    cap = ops._sticky_capacity(n * max(1, min_samples))
    state = torch.zeros(8, dtype=I32, device=dev)
    state[3] = n
    total = torch.zeros(1, dtype=I64, device=dev)
    lists = [torch.arange(n, dtype=I32, device=dev), torch.empty(n, dtype=I32, device=dev)]
    n_sm = torch.empty(n, dtype=I32, device=dev)
    run_cap = ops.MarchInputs.RUN_CAP
    run_t = torch.empty(n, run_cap, device=dev)
    run_n = torch.empty(n, run_cap, dtype=I32, device=dev)
    n_runs = torch.empty(n, dtype=I32, device=dev)
    overflow = torch.empty(n, dtype=torch.bool, device=dev)
    t0, t1 = torch.empty(cap, device=dev), torch.empty(cap, device=dev)
    ridx = torch.empty(cap, dtype=I64, device=dev)
    offsets = torch.empty(n + 1, dtype=I64, device=dev)
    totals = torch.zeros(2, dtype=I64, device=dev)
    flags = torch.empty(n, dtype=I32, device=dev)
    pos, pos_tot = torch.empty(n + 1, dtype=I64, device=dev), torch.empty(2, dtype=I64, device=dev)
    ws = torch.empty(max(int(_lib_scan_ws(n)) // 8, 1), dtype=I64, device=dev)
    ts = ops._f32c(timestamps).view(-1)
    images = (field.xyz_wrap.network.weight_image(), field.mlp_base.weight_image(), field.mlp_head.weight_image())
    desc, table = field._field_desc(), field.hash_encoder.table_f16()
    sigma, rgbs = torch.empty(cap, device=dev), torch.empty(cap, 3, device=dev)
    ring = [torch.empty(8, dtype=I32).pin_memory() for _ in range(_ROUND_LAG + 2)]
    pending = []          # (event, host copy of the state at the START of a round)
    bound, k_hint = n, max(1, min_samples)
    max_rounds = (max_samples + min_samples - 1) // min_samples + 1
    import ctypes as _ct

    # everything that is the same for every round of the frame goes into one struct; a round is then ONE library call
    # (eight launches: count pass, scan, fill from runs, fallback fill, field, compositing, scan, ordered compaction)
    from . import _lib
    from ._lib import RenderRound

    rr = RenderRound()
    for name, t in (("rays_o", o), ("rays_d", d), ("occ_bits", bits), ("aabbs", aabbs_c), ("near_term", near),
                    ("t_sorted", t_sorted), ("t_indices", t_indices), ("hits", hits), ("state", state), ("total", total),
                    ("n_samples", n_sm), ("run_t", run_t), ("run_n", run_n), ("n_runs", n_runs), ("occ_coarse", coarse),
                    ("offsets", offsets), ("totals", totals), ("scan_workspace", ws), ("t_starts", t0), ("t_ends", t1),
                    ("ray_indices", ridx), ("overflow", overflow), ("timestamps", ts), ("image_deform", images[0]),
                    ("image_density", images[1]), ("image_colour", images[2]), ("table_f16", table), ("sigma", sigma),
                    ("rgbs", rgbs), ("colors", rgb), ("opacity", opacity), ("depth", depth), ("alive_flags", flags),
                    ("positions", pos), ("position_totals", pos_tot)):
        setattr(rr, name, ptr(t))
    rr.n_rays, rr.n_levels, rr.resolution, rr.capacity = n, n_levels, res, cap
    rr.far_const, rr.step_size, rr.cone_angle, rr.early_stop_eps = far_plane, float(step), float(cone), float(early_stop_eps)
    rr.desc = _ct.pointer(desc)
    rr.run_cap, rr.k_hint, rr.max_samples, rr.min_samples = run_cap, int(k_hint), int(max_samples), int(min_samples)
    rr_ref = _ct.byref(rr)
    list_ptrs = (ptr(lists[0]), ptr(lists[1]))
    call("cednerf_render_round_begin", ptr(state), n, int(max_samples), int(min_samples), None, ptr(total), stream())
    for rnd in range(max_rounds):   # (every later round is begun by the compaction launch that ends its predecessor)
        host = ring[rnd % len(ring)]
        host.copy_(state, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        pending.append((ev, host))
        if _lib._timers is None and not _ROUND_BY_PARTS:
            call("cednerf_render_round", rr_ref, bound, list_ptrs[rnd & 1], list_ptrs[(rnd + 1) & 1], stream())
        else:   # bench.py's per-entry-point instrumentation: the same eight launches as separate calls
            _round_by_parts(rr, bound, list_ptrs[rnd & 1], list_ptrs[(rnd + 1) & 1], desc)
        # look at the oldest state copies that have arrived; never run more than _ROUND_LAG rounds ahead of one
        stop = False
        while pending and (pending[0][0].query() or len(pending) > _ROUND_LAG):
            ev0, h0 = pending.pop(0)
            ev0.synchronize()
            n_alive, k_seen, over = int(h0[0]), int(h0[1]), int(h0[5])
            if over or n_alive == 0:
                stop = True
                break
            bound = min(bound, n_alive)                    # valid for every later round: the list only shrinks
            # (k_hint stays at min_samples: it picks the lane-group width of the compositing kernel, i.e. the order in
            # which a ray's samples are summed - following the host's LAGGED view of k made the last bits of a frame
            # depend on timing; late rounds with large k have few rays left, so the narrow groups cost nothing)
        if stop:
            break
        yield
    # the rounds still in flight when the host saw the end did nothing (state[0] == 0, totals == 0)
    total_host = torch.empty(1, dtype=I64).pin_memory()
    total_host.copy_(total, non_blocking=True)
    done_ev = torch.cuda.Event()
    done_ev.record()
    while not done_ev.query():
        yield
    return int(total_host[0])


def _round_by_parts(r, bound, cur, nxt, desc):
    """cednerf_render_round spelled out as its eight entry points (csrc/render_round.cu), for per-kernel timing."""
    import ctypes as _ct

    from ._lib import call, stream

    st = stream()
    call("cednerf_march_round", 0, r.rays_o, r.rays_d, bound, r.occ_bits, r.aabbs, r.n_levels, r.resolution, r.near_term,
         r.far_const, r.step_size, r.cone_angle, r.t_sorted, r.t_indices, r.hits, cur, r.state, None, None, None, None, None,
         r.n_samples, r.run_t, r.run_n, r.n_runs, r.run_cap, r.occ_coarse, st)
    call("cednerf_exclusive_scan_capped", r.n_samples, bound, r.capacity, r.offsets, r.totals, r.scan_workspace, st)
    call("cednerf_march_fill_runs_round", bound, r.offsets, r.n_samples, r.run_t, r.run_n, r.n_runs, r.run_cap, r.step_size,
         r.cone_angle, cur, r.state, r.t_starts, r.t_ends, r.ray_indices, r.overflow, st)
    call("cednerf_march_round", 1, r.rays_o, r.rays_d, bound, r.occ_bits, r.aabbs, r.n_levels, r.resolution, r.near_term,
         r.far_const, r.step_size, r.cone_angle, r.t_sorted, r.t_indices, r.hits, cur, r.state, r.overflow, r.offsets,
         r.t_starts, r.t_ends, r.ray_indices, None, None, None, None, r.run_cap, r.occ_coarse, st)
    call("cednerf_field_fwd", r.ray_indices, r.t_starts, r.t_ends, r.rays_o, r.rays_d, None, None, r.timestamps, 0, r.capacity,
         r.image_deform, r.image_density, r.image_colour, r.table_f16, _ct.byref(desc), r.sigma, r.rgbs, r.totals, st)
    call("cednerf_render_round_composite", r.t_starts, r.t_ends, r.sigma, r.rgbs, r.offsets, cur, r.state, r.n_samples, bound,
         r.k_hint, r.early_stop_eps, r.colors, r.opacity, r.depth, r.alive_flags, st)
    call("cednerf_exclusive_scan_capped", r.alive_flags, bound, r.n_rays, r.positions, r.position_totals, r.scan_workspace, st)
    call("cednerf_render_round_compact", r.alive_flags, r.positions, cur, bound, r.state, nxt, r.n_rays, r.max_samples,
         r.min_samples, r.totals, r.total, st)


def _lib_scan_ws(n):
    from . import _lib

    return _lib.load().cednerf_scan_workspace_bytes(n)


@torch.no_grad()
def render_image_test(max_samples, radiance_field, estimator, rays, near_plane=0.0, far_plane=1e10,
                      render_step_size=1e-3, render_bkgd=None, cone_angle=0.0, alpha_thre=0.0, early_stop_eps=1e-4,
                      timestamps=None):
    """Iterative early-terminating marcher of cednerf/utils.py:153-318 -> (rgb, acc, depth, n_samples)."""
    gen = _render_image_test_gen(max_samples, radiance_field, estimator, rays, near_plane, far_plane, render_step_size,
                                 render_bkgd, cone_angle, alpha_thre, early_stop_eps, timestamps)
    while True:
        try:
            next(gen)
        except StopIteration as fin:
            return fin.value


_FRAME_STREAMS = {}


def _frame_streams(k: int):
    """The side streams frames are interleaved on, kept for the life of the process: the caching allocator pools memory per
    stream, so fresh streams on every call would re-allocate every per-frame buffer (and strand the old pools)."""
    dev = torch.cuda.current_device()
    pool = _FRAME_STREAMS.setdefault(dev, [])
    while len(pool) < k:
        pool.append(torch.cuda.Stream(device=dev))
    return pool[:k]


@torch.no_grad()
def render_images_test(max_samples, radiance_field, estimator, rays_list, timestamps_list, concurrency: int = 2,
                       on_frame=None, **kwargs):
    """render_image_test for several independent frames (a video: datasets/utils.py:67-112 poses, one timestamp each),
    with the marching rounds of up to `concurrency` frames interleaved on separate CUDA streams: a round's count pass
    ends with a few rays walking long stretches of empty space while most SMs idle, and the field kernel of another frame
    fills them.  rays_list: Rays, or callables returning Rays (called inside the frame's stream, e.g. generate_rays).
    on_frame(index, (rgb, acc, depth, n_samples)): called as each frame completes (the results are then not kept).
    -> list of (rgb, acc, depth, n_samples), frame by frame identical to render_image_test."""
    n_frames = len(rays_list)
    results = [None] * n_frames
    main = torch.cuda.current_stream()
    # The frames share caches derived from the occupancy grid and the parameters.  Build them here, on the calling
    # stream, which every frame stream waits for: built inside the first frame's stream, they would be read by the
    # other frames' streams with nothing ordering the reads after the writes.
    bits = nerfacc.grid.occupancy_bits(estimator.binaries)
    ops.occupancy_coarse(bits, int(estimator.aabbs.shape[0]), int(estimator.binaries.shape[1]))
    if getattr(radiance_field, "fused_supported", lambda: False)():
        radiance_field.hash_encoder.table_f16()
        for net in (radiance_field.xyz_wrap.network, radiance_field.mlp_base, radiance_field.mlp_head):
            net.weight_image()
    streams = _frame_streams(max(1, min(int(concurrency), n_frames)))
    free, active, nxt = list(streams), [], 0
    while active or nxt < n_frames:
        while free and nxt < n_frames:
            st = free.pop()
            st.wait_stream(main)
            with torch.cuda.stream(st):
                r = rays_list[nxt]
                r = r() if callable(r) else r
                gen = _render_image_test_gen(max_samples, radiance_field, estimator, r, timestamps=timestamps_list[nxt],
                                             **kwargs)
            active.append((gen, st, nxt))
            nxt += 1
        for entry in list(active):
            gen, st, idx = entry
            with torch.cuda.stream(st):
                try:
                    next(gen)
                except StopIteration as fin:
                    main.wait_stream(st)
                    for t in fin.value[:3]:
                        t.record_stream(main)
                    if on_frame is None:
                        results[idx] = fin.value
                    else:
                        with torch.cuda.stream(main):
                            on_frame(idx, fin.value)
                    active.remove(entry)
                    free.append(st)
    return results


def _render_image_test_gen(max_samples, radiance_field, estimator, rays, near_plane=0.0, far_plane=1e10,
                           render_step_size=1e-3, render_bkgd=None, cone_angle=0.0, alpha_thre=0.0, early_stop_eps=1e-4,
                           timestamps=None):
    """render_image_test as a generator (yields between marching rounds on the device-resident path)."""
    shape = rays.origins.shape
    rays = Rays(rays.origins.reshape(-1, 3), rays.viewdirs.reshape(-1, 3))
    n, dev = rays.origins.shape[0], rays.origins.device
    _, rgb_sigma_fn = _field_fns(radiance_field, rays, timestamps)
    opacity, depth, rgb = torch.zeros(n, 1, device=dev), torch.zeros(n, 1, device=dev), torch.zeros(n, 3, device=dev)
    alive = torch.ones(n, dtype=torch.bool, device=dev)
    min_samples = 1 if cone_angle == 0 else 4
    near = torch.full((n,), float(near_plane), device=dev)
    far = torch.full((n,), float(far_plane), device=dev)
    t_mins, t_maxs, hits = nerfacc.ray_aabb_intersect(rays.origins, rays.viewdirs, estimator.aabbs)
    t_sorted, t_indices = ops.sort_boundaries(t_mins, t_maxs)
    bits = nerfacc.grid.occupancy_bits(estimator.binaries)
    res = int(estimator.binaries.shape[1])
    fuse = (getattr(radiance_field, "fused_supported", lambda: False)() and not radiance_field.training
            and timestamps is not None and timestamps.numel() == 1 and render_step_size > 0 and n < 2 ** 31)
    if fuse and _DEVICE_ROUNDS:
        total = yield from _render_rounds_gen(max_samples, radiance_field, rays, bits, estimator.aabbs, res, near,
                                              float(far_plane), render_step_size, cone_angle, early_stop_eps, timestamps,
                                              t_sorted, t_indices, hits, min_samples, rgb, opacity, depth)
        rgb = rgb + render_bkgd * (1.0 - opacity)
        depth = depth / opacity.clamp_min(torch.finfo(torch.float32).eps)
        return rgb.view(*shape[:-1], -1), opacity.view(*shape[:-1], -1), depth.view(*shape[:-1], -1), total
    done = total = 0
    # With the fused field kernel a round needs ONE host read (the reference's `alive.sum()`): the round's sample total
    # stays on the device - outputs are sized for the bound n_alive * k and the kernels read the live count themselves.
    total_dev = torch.zeros(1, dtype=torch.int64, device=dev)
    while done < max_samples:
        n_alive = int(alive.sum())                     # the reference's host read (utils.py:231)
        if n_alive == 0:
            break
        k = max(min(n // n_alive, 64), min_samples)
        done += k
        # traverse_grids(..., k, over_allocate=True, alive, ...) of utils.py:245-264, emitted directly in packed form:
        # same samples, no interval flags to compact afterwards
        mi = ops.MarchInputs(rays.origins, rays.viewdirs, bits, estimator.aabbs, res, near, far, 0.0, float("inf"),
                             render_step_size, cone_angle, k, alive, t_sorted, t_indices, hits)
        _, n_sm, term = mi.count(record_runs=True)
        starts, _, n_tot = ops.exclusive_scan(n_sm, want_packed=False)
        if fuse and mi.runs is not None:
            cap = n_alive * k
            ridx, t0, t1 = mi.fill_packed_from_runs(starts, cap)
            sigma, rgbs = radiance_field.fused_query(cap, packed=(ridx, t0, t1, rays.origins, rays.viewdirs),
                                                     timestamps=timestamps, t_stride=0, sigma_only=False, n_dev=n_tot)
            ops.composite_round_(t0, t1, sigma, rgbs, torch.cat([starts, n_tot]), rgb, opacity, depth)
            total_dev += n_tot
        else:
            n_round = int(n_tot.item())
            if n_round:
                if mi.runs is not None:
                    ridx, t0, t1 = mi.fill_packed_from_runs(starts, n_round)
                else:
                    ridx, t0, t1, _ = mi.fill_packed(starts, n_round)
                rgbs, sres = rgb_sigma_fn(t0, t1, ridx)
                ops.composite_round_(t0, t1, sres["density"].squeeze(-1), rgbs, torch.cat([starts, n_tot]), rgb, opacity,
                                     depth)
            total += n_round
        near = term
        alive = (opacity.view(-1) <= 1 - early_stop_eps) & (n_sm == k)
    total += int(total_dev.item())
    rgb = rgb + render_bkgd * (1.0 - opacity)
    depth = depth / opacity.clamp_min(torch.finfo(torch.float32).eps)
    return rgb.view(*shape[:-1], -1), opacity.view(*shape[:-1], -1), depth.view(*shape[:-1], -1), total
