"""Exact tests for the capacity-mode training step (`render_image(..., device_counts=True)`), the path bench.py times.

In this mode the sample tensors are allocated at a capacity that comes from earlier batches, only a live prefix is
valid, and every kernel reads the live count from the device.  The tests below check the kernels of that path against
exact-size runs and plain references: the capped scans against numpy int64, the capped marched fill against the
oracle (including the drop contract of a batch that outgrows its capacity), visibility and compaction at several
capacities, every consumer of a device-side count with poisoned tails, and the whole step against host-count mode.

Poisoning: `torch.empty` / `torch.empty_like` hand out NaN (floating), True (bool) or 0 (integers) for the duration of
a test, so that a kernel that reads past the live count sees NaN rather than freshly mapped zeros.  Integers get 0 so
that a wrongly read index still lands inside its buffer.  Where a test calls a C entry point directly, every output
and input has a guard band of GUARD rows past the capacity, filled with a sentinel (outputs) or NaN (inputs).
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import nerfacc_ref as nf  # noqa: E402

DEV = "cuda:0"
GUARD = 256
SENT_I = -7
SCAN_TILE = 4096


@pytest.fixture(scope="module")
def cb():
    import cednerf_b200

    return cednerf_b200


def _fill_poison(t):
    if t.numel():
        if t.is_floating_point():
            t.fill_(float("nan"))
        elif t.dtype == torch.bool:
            t.fill_(True)
        else:
            t.fill_(0)
    return t


@pytest.fixture
def poison(monkeypatch):
    real_empty, real_empty_like = torch.empty, torch.empty_like
    monkeypatch.setattr(torch, "empty", lambda *a, **k: _fill_poison(real_empty(*a, **k)))
    monkeypatch.setattr(torch, "empty_like", lambda *a, **k: _fill_poison(real_empty_like(*a, **k)))


@pytest.fixture
def guard_rows(cb, poison, monkeypatch):
    """Sample-sized outputs and workspaces of the wrappers get GUARD spare rows, so that a device count above the
    capacity cannot write outside an allocation even if a kernel failed to clamp it."""
    from cednerf_b200 import losses

    ops = cb.ops
    real_sticky = ops._sticky_capacity

    def sempty(n, *tail, dtype=None, device=None):
        return torch.empty((int(n) + GUARD,) + tuple(tail), dtype=dtype, device=device)[:n]

    monkeypatch.setattr(ops, "_sempty", sempty)
    monkeypatch.setattr(losses, "_sempty", sempty)
    monkeypatch.setattr(ops, "_sticky_capacity", lambda n: real_sticky(n) + GUARD)


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def guarded(n, *tail, dtype=torch.float32, fill=float("nan")):
    """(buffer of n + GUARD rows filled with `fill`, its first n rows)."""
    buf = torch.full((n + GUARD,) + tail, fill, dtype=dtype, device=DEV)
    return buf, buf[:n]


def guard_intact(buf, n, fill=float("nan")):
    g = buf[n:]
    if isinstance(fill, float) and math.isnan(fill):
        return bool(torch.isnan(g).all())
    return bool((g == fill).all())


def p(t):
    from cednerf_b200._lib import ptr

    return ptr(t)


# ------------------------------------------------------------------------------------------------------------- A: scans
SCAN_NS = [0, 1, 4095, 4096, 4097, 3 * SCAN_TILE + 5, 2 ** 22 + 3]


def scan_counts(n, kind, seed=0):
    g = np.random.default_rng(seed + n)
    if kind == "zero":
        return np.zeros(n, np.int32)
    hi = 2001 if kind == "big" else 64
    c = g.integers(0, hi, n, dtype=np.int64).astype(np.int32)
    c[g.random(n) < 0.2] = 0
    return c


@pytest.mark.parametrize("n", SCAN_NS)
@pytest.mark.parametrize("kind", ["random", "zero", "big"])
def test_scans_match_int64_reference(cb, poison, n, kind):
    ops = cb.ops
    c = scan_counts(n, kind)
    ref = np.concatenate([[0], np.cumsum(c, dtype=np.int64)])
    total = int(ref[-1])
    if kind == "big" and n == SCAN_NS[-1]:
        assert total > 2 ** 31
    counts = torch.from_numpy(c).to(DEV)
    starts, packed, tot = ops.exclusive_scan(counts)
    assert int(tot) == total
    assert np.array_equal(starts.cpu().numpy(), ref[:-1])
    assert np.array_equal(packed.cpu().numpy(), np.stack([ref[:-1], c.astype(np.int64)], -1).reshape(n, 2))
    for cap in sorted({0, 1, max(total - 1, 0), total, total + 1, 2 ** 40}):
        off, tots = ops.exclusive_scan_capped(counts, cap)
        assert np.array_equal(off.cpu().numpy(), np.minimum(ref, cap)), cap
        assert tots.cpu().tolist() == [min(total, cap), total], cap


def test_capped_scan_back_to_back_on_one_workspace(cb):
    """Twenty scans of different counts on one stream, reusing one workspace: the look-back's tickets and flag words
    are reset by every call, so every result is exact.  Outputs carry guard bands."""
    ops = cb.ops
    n = 3 * SCAN_TILE + 5 + 50 * SCAN_TILE
    ws = torch.empty(int(cb._lib.load().cednerf_scan_workspace_bytes(n)) // 8, dtype=torch.int64, device=DEV)
    outs = []
    for k in range(20):
        c = scan_counts(n, "big" if k % 3 == 0 else ("zero" if k % 7 == 6 else "random"), seed=100 + k)
        counts = torch.from_numpy(c).to(DEV)
        ref = np.concatenate([[0], np.cumsum(c, dtype=np.int64)])
        cap = [int(ref[-1]), int(ref[-1]) // 2, 2 ** 40, 1][k % 4]
        off_buf, off = guarded(n + 1, dtype=torch.int64, fill=SENT_I)
        tot_buf, tot = guarded(2, dtype=torch.int64, fill=SENT_I)
        ops.call("cednerf_exclusive_scan_capped", p(counts), n, cap, p(off), p(tot), p(ws), ops.stream())
        outs.append((counts, ref, cap, off_buf, tot_buf))
    torch.cuda.synchronize()
    for counts, ref, cap, off_buf, tot_buf in outs:
        assert np.array_equal(off_buf[:n + 1].cpu().numpy(), np.minimum(ref, cap))
        assert tot_buf[:2].cpu().tolist() == [min(int(ref[-1]), cap), int(ref[-1])]
        assert guard_intact(off_buf, n + 1, SENT_I) and guard_intact(tot_buf, 2, SENT_I)


# ---------------------------------------------------------------------------------------- B: marched fill, capped
def march_scene(seed, grid, n_rays=3000, res=16, levels=2):
    g = torch.Generator().manual_seed(seed)
    est = nf.OccGridEstimator([-1.0, -1.0, -1.0, 1.0, 1.0, 1.0], resolution=res, levels=levels)
    if grid == "checker":
        i = torch.arange(res)
        cb3 = (i[:, None, None] + i[None, :, None] + i[None, None, :]) % 2 == 0
        est.binaries = cb3[None].expand(levels, res, res, res).contiguous()
    else:
        est.binaries = torch.rand(levels, res, res, res, generator=g) < 0.25
    origins = torch.tensor([0.0, 0.0, -3.5]) + (torch.rand(n_rays, 3, generator=g) - 0.5) * 0.6
    target = (torch.rand(n_rays, 3, generator=g) - 0.5) * 1.6
    dirs = torch.nn.functional.normalize(target - origins, dim=-1)
    return est, origins, dirs, g


def capped_expectation(ridx, t0, t1, counts, n_runs, run_cap, cap):
    """The drop contract, on the host: rays wholly below the capacity keep the oracle's samples; a ray cut at the
    capacity keeps its first samples if it has at most run_cap runs, else zero-length samples (0, 0, r)."""
    starts = np.concatenate([[0], np.cumsum(counts.numpy().astype(np.int64))])
    k = min(cap, int(starts[-1]))
    e_r, e_a, e_b = ridx[:k].clone(), t0[:k].clone(), t1[:k].clone()
    cut = int(np.searchsorted(starts, k, side="right")) - 1   # the ray whose range holds index k (if any is cut)
    if cut < counts.numel() and starts[cut] < k < starts[cut + 1] and int(n_runs[cut]) > run_cap:
        e_a[starts[cut]:k] = 0.0
        e_b[starts[cut]:k] = 0.0
    return e_r, e_a, e_b, k


def capacities_for(counts, n_runs, run_cap):
    starts = np.concatenate([[0], np.cumsum(counts.numpy().astype(np.int64))])
    total = int(starts[-1])
    long_rays = [r for r in range(counts.numel()) if counts[r] >= 3]
    few = [r for r in long_rays if int(n_runs[r]) <= run_cap]
    many = [r for r in long_rays if int(n_runs[r]) > run_cap]
    caps = {"total": total, "ray_boundary": int(starts[long_rays[len(long_rays) // 3]]), "one": 1, "above": total + 1000}
    if few:
        caps["inside_few_runs"] = int(starts[few[len(few) // 2]]) + 1
    if many:
        caps["inside_many_runs"] = int(starts[many[len(many) // 2]]) + 1
    return caps


@pytest.mark.parametrize("grid", ["checker", "random"])
@pytest.mark.parametrize("cone", [0.0, 0.004])
@pytest.mark.parametrize("run_cap", [1, 3, 16])
def test_capped_marched_fill_follows_the_drop_contract(cb, poison, monkeypatch, grid, cone, run_cap):
    ops = cb.ops
    est, o, d, g = march_scene(31, grid)
    n = o.shape[0]
    step = 2e-2
    near = torch.full((n,), 0.2) + torch.rand(n, generator=g) * step
    far = torch.full((n,), 1e10)
    ridx, t0, t1, packed, _ = nf.traverse_grids(o, d, est.binaries, est.aabbs, near, far, step, cone, packed_only=True)
    monkeypatch.setattr(ops.MarchInputs, "RUN_CAP", run_cap)
    mi = ops.MarchInputs(o.to(DEV), d.to(DEV), ops.pack_occupancy(est.binaries.to(DEV)), est.aabbs.to(DEV), 16,
                         near.to(DEV), far.to(DEV), 0.0, 1e10, step, cone)
    _, n_sm, _ = mi.count(record_runs=True)
    counts, n_runs = n_sm.cpu(), mi.runs[2].cpu()
    assert torch.equal(counts.long(), packed[:, 1])
    caps = capacities_for(counts, n_runs, run_cap)
    assert "inside_few_runs" in caps or grid == "checker"   # checkerboard rays cross a run per cell
    assert "inside_many_runs" in caps or run_cap == 16
    for name, cap in caps.items():
        offsets, totals = ops.exclusive_scan_capped(n_sm, cap)
        a_buf, a = guarded(cap)
        b_buf, b = guarded(cap)
        r_buf, r = guarded(cap, dtype=torch.int64, fill=SENT_I)
        overflow = torch.empty(n, dtype=torch.bool, device=DEV)
        rt, rn, nr = mi.runs
        ops.call("cednerf_march_fill_runs_capped", n, p(offsets), p(n_sm), p(rt), p(rn), p(nr), run_cap, step, cone,
                 p(a), p(b), p(r), p(overflow), ops.stream())
        user_mask, mi.mask = mi.mask, overflow
        ops.call("cednerf_march", *mi._common(1), None, p(offsets), None, None, None, None, None, None, None,
                 p(a), p(b), p(r), None, None, None, None, None, None, 0, None, p(mi.coarse), ops.stream())
        mi.mask = user_mask
        e_r, e_a, e_b, k = capped_expectation(ridx, t0, t1, counts, n_runs, run_cap, cap)
        assert totals.cpu().tolist() == [k, ridx.numel()], name
        assert torch.equal(r[:k].cpu(), e_r), name
        assert torch.equal(a[:k].cpu(), e_a) and torch.equal(b[:k].cpu(), e_b), name
        assert bool((r[k:] == SENT_I).all()) and bool(torch.isnan(a[k:]).all()) and bool(torch.isnan(b[k:]).all()), name
        assert guard_intact(a_buf, cap) and guard_intact(b_buf, cap) and guard_intact(r_buf, cap, SENT_I), name


# --------------------------------------------------------------------------------- C: visibility and compaction
def sample_set(mean, n_rays=4000, seed=5):
    """Packed samples with about `mean` samples per ray, a tenth of the rays empty, densities that make early stopping
    and the alpha threshold both matter."""
    g = torch.Generator().manual_seed(seed + int(mean))
    cnt = torch.poisson(torch.full((n_rays,), float(mean)), generator=g).long()
    cnt[torch.rand(n_rays, generator=g) < 0.1] = 0
    S = int(cnt.sum())
    ridx = torch.repeat_interleave(torch.arange(n_rays), cnt)
    dt = torch.rand(S, generator=g) * 0.05 + 0.005
    off = torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(cnt, 0)])
    cs = torch.cumsum(dt, 0)
    t0 = 0.5 + cs - dt - (cs - dt)[off[:-1].clamp(max=S - 1)].repeat_interleave(cnt)
    t1 = t0 + dt
    sig = torch.exp(torch.randn(S, generator=g) * 2.0) * (4.0 / max(mean, 1))
    return ridx, t0, t1, sig, off, n_rays


def padded(x, cap, fill=float("nan")):
    """x (exact size) in a buffer of cap + GUARD rows: live prefix, then `fill`."""
    buf = torch.full((cap + GUARD,) + tuple(x.shape[1:]), fill, dtype=x.dtype, device=DEV)
    buf[:x.shape[0]] = x.to(DEV)
    return buf, buf[:cap]


MEANS = [3, 10, 20, 90]
EPS, ATHR = 1e-4, 1e-2


@pytest.mark.parametrize("mean", MEANS)
def test_capped_compaction_is_the_truncated_uncapped_compaction(cb, poison, mean):
    ops = cb.ops
    ridx, t0, t1, sig, off, n_rays = sample_set(mean)
    S = t0.numel()
    T0, T1, SG, OFF = (x.to(DEV) for x in (t0, t1, sig, off))
    u_r, u_a, u_b = ops.visible_samples(T0, T1, SG, OFF, n_rays, EPS, ATHR)
    keep, kc = ops.visibility_mask(T0, T1, SG, OFF, n_rays, EPS, ATHR, want_counts=True)
    kept_off = torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(kc.long().cpu(), 0)])
    n_kept = u_r.numel()
    assert int(kept_off[-1]) == n_kept > 0
    for cap in sorted({0, 1, n_kept // 3, n_kept - 1, n_kept, n_kept + 5}):
        out_off, totals = ops.exclusive_scan_capped(kc, cap)
        r_buf, r = guarded(cap, dtype=torch.int64, fill=SENT_I)
        a_buf, a = guarded(cap)
        b_buf, b = guarded(cap)
        ops.call("cednerf_compact_samples_capped", p(keep), p(OFF), p(out_off), p(T0), p(T1), cap, n_rays, p(r), p(a),
                 p(b), ops.stream())
        k = min(cap, n_kept)
        assert totals.cpu().tolist() == [k, n_kept]
        assert torch.equal(out_off.cpu(), torch.clamp(kept_off, max=cap))
        assert torch.equal(r[:k], u_r[:k]) and torch.equal(a[:k], u_a[:k]) and torch.equal(b[:k], u_b[:k]), cap
        assert bool((r[k:] == SENT_I).all()) and bool(torch.isnan(a[k:]).all()), cap
        assert guard_intact(r_buf, cap, SENT_I) and guard_intact(a_buf, cap) and guard_intact(b_buf, cap), cap


def bucket_capacities(S, n_rays):
    """Capacities >= S whose mean per ray falls in each lane-group bucket (<= 6, <= 12, <= 24, > 24) that can hold S."""
    caps = [S, S * 3 // 2 + 1]
    for edge in (6.0, 12.0, 24.0, 40.0):
        c = int(edge * n_rays)
        if c > S:
            caps.append(c)
    return sorted(set(caps))


@pytest.mark.parametrize("mean", MEANS)
def test_per_ray_kernels_do_not_depend_on_the_capacity(cb, poison, mean):
    """The same live samples in buffers of several capacities (tails NaN) give the same visibility, compaction,
    weights, colours and gradients bit for bit: the lane-group width of the per-ray scans follows the live count."""
    ops = cb.ops
    ridx, t0, t1, sig, off, n_rays = sample_set(mean)
    S = t0.numel()
    g = torch.Generator().manual_seed(9)
    rgbs = torch.rand(S, 3, generator=g)
    g_col = torch.rand(n_rays, 3, generator=g).to(DEV)
    OFF = off.to(DEV)
    results = []
    for cap in bucket_capacities(S, n_rays):
        (_, a), (_, b), (_, s), (_, c) = (padded(x, cap) for x in (t0, t1, sig, rgbs))
        keep, kc = ops.visibility_mask(a, b, s, OFF, n_rays, EPS, ATHR, want_counts=True)
        ridx_v, a_v, b_v, off_v, tot_v = ops.visible_samples_capped(a, b, s, OFF, n_rays, EPS, ATHR, cap)
        sg = s.clone().requires_grad_(True)
        cc = c.clone().requires_grad_(True)
        col, opac, dep, w, tr, al = ops.CompositeFunction.apply(a, b, sg, cc, OFF, n_rays, None)
        (col * g_col).sum().add(opac.sum()).add(dep.sum()).backward()
        acc = ops.AccumulateFunction.apply(w.detach(), c, None, OFF, n_rays, None)
        results.append((cap, keep[:S].clone(), kc.clone(), ridx_v[:int(tot_v[0])].clone(), a_v[:int(tot_v[0])].clone(),
                        col.detach(), opac.detach(), dep.detach(), w[:S].detach(), tr[:S].detach(),
                        sg.grad[:S].clone(), cc.grad[:S].clone(), acc.detach()))
    assert len(results) >= 2
    base = results[0]
    for other in results[1:]:
        for i in range(1, len(base)):
            assert torch.equal(other[i], base[i]), (base[0], other[0], i)


@pytest.mark.parametrize("mean", MEANS)
def test_visibility_disagrees_with_fp64_only_at_its_thresholds(cb, mean):
    """Every sample whose keep flag differs from a float64 evaluation of render_visibility_from_density has its
    transmittance or alpha within 1e-4 (relative) of the threshold that decided it."""
    ops = cb.ops
    ridx, t0, t1, sig, off, n_rays = sample_set(mean)
    keep = ops.visibility_mask(t0.to(DEV), t1.to(DEV), sig.to(DEV), off.to(DEV), n_rays, EPS, ATHR)[:t0.numel()].cpu()
    sd = sig.double() * (t1.double() - t0.double())
    cs = torch.cumsum(sd, 0)
    base = (cs - sd)[off[:-1].clamp(max=sd.numel() - 1)].repeat_interleave(off[1:] - off[:-1])
    trans = torch.exp(-(cs - sd - base))
    alpha = 1.0 - torch.exp(-sd)
    ref = (trans >= EPS) & (alpha >= ATHR)
    ref_nf = nf.render_visibility_from_density(t0, t1, sig, ray_indices=ridx, n_rays=n_rays, early_stop_eps=EPS,
                                               alpha_thre=ATHR)
    for r in (ref, ref_nf.bool()):
        bad = keep != r
        near_t = (trans - EPS).abs() <= 1e-4 * EPS
        near_a = (alpha - ATHR).abs() <= 1e-4 * ATHR
        assert not bool((bad & ~(near_t | near_a)).any()), int((bad & ~(near_t | near_a)).sum())


# -------------------------------------------------------------------------------------------- D: n_device consumers
LIVE = [0, 1, 127, 128, 129, 128 * 613 + 37]
REL = ["below", "equal", "above"]


def capacity_and_ndev(live, relation):
    """(buffer capacity, device count): the count is below the capacity, equal to it, or above it (clamped)."""
    if relation == "below":
        return live + 300, live
    if relation == "equal":
        return live, live
    return live, live + 200   # past the capacity but inside the guard band


def packed_inputs(live, n_rays=97, seed=3):
    g = torch.Generator().manual_seed(seed + live)
    ridx = torch.sort(torch.randint(0, n_rays, (live,), generator=g))[0]
    t0 = 1.5 + torch.rand(live, generator=g) * 3
    o = torch.tensor([0.0, 0.0, -3.0]) + (torch.rand(n_rays, 3, generator=g) - 0.5) * 0.4
    d = torch.nn.functional.normalize(torch.randn(n_rays, 3, generator=g) * 0.2 + torch.tensor([0.0, 0.0, 1.0]), dim=-1)
    ts = torch.rand(n_rays, 1, generator=g)
    return ridx, t0, t0 + 0.02, o.to(DEV), d.to(DEV), ts.to(DEV), n_rays


def trained_field(cb, name, extra):
    kw = dict(n_levels=8, log2_hashmap_size=12, dst_resolution=256, moving_step=1.0 / 256)
    if extra.get("use_feat_predict"):
        kw.update(n_levels=16, log2_hashmap_size=14, dst_resolution=512)
    field = cb.DNGPradianceField(torch.tensor([-1.0, -1.0, -1.0, 1.0, 1.0, 1.0]), **kw, **TRAIN_FLAGS[name], **extra)
    with torch.no_grad():
        field.hash_encoder.params.mul_(5000.0)
        field.mlp_base.params.mul_(3.0)
    return field.to(DEV)


@pytest.mark.parametrize("live", LIVE)
@pytest.mark.parametrize("relation", REL)
@pytest.mark.parametrize("t_stride", [0, 1])
def test_fused_query_reads_the_live_count(cb, guard_rows, live, relation, t_stride):
    field = trained_field(cb, "te_ta_df", {}).eval()
    ridx, t0, t1, o, d, ts, _ = packed_inputs(live)
    cap, nd = capacity_and_ndev(live, relation)
    (_, R), (_, A), (_, B) = padded(ridx, cap, 0), padded(t0, cap), padded(t1, cap)
    n_dev = torch.tensor([nd], dtype=torch.int64, device=DEV)
    if cap == 0:   # the entry point refuses buffers of no rows
        with pytest.raises(RuntimeError, match="bad arguments"):
            field.fused_query(0, packed=(R, A, B, o, d), timestamps=ts, t_stride=t_stride, n_dev=n_dev)
        return
    with torch.no_grad():
        s_c, c_c = field.fused_query(cap, packed=(R, A, B, o, d), timestamps=ts, t_stride=t_stride, sigma_only=False,
                                     n_dev=n_dev)
        if live:   # (the entry point refuses n = 0: there is nothing to compare with)
            s_e, c_e = field.fused_query(live, packed=(R[:live], A[:live], B[:live], o, d), timestamps=ts,
                                         t_stride=t_stride, sigma_only=False)
            assert torch.equal(s_c[:live], s_e) and torch.equal(c_c[:live], c_e)
    assert bool(torch.isnan(s_c[live:]).all()) and bool(torch.isnan(c_c[live:]).all())


TRAIN_FLAGS = {
    "plain": dict(),
    "te_ta_df": dict(use_time_embedding=True, use_time_attenuation=True, use_div_offsets=True),
    "te_after": dict(use_time_embedding=True, time_inject_before_sigma=False),
}
TRAIN_SETS = [("plain", {}), ("te_ta_df", {}), ("te_after", {}), ("te_ta_df", {"use_feat_predict": True})]


@pytest.mark.parametrize("name,extra", TRAIN_SETS)
@pytest.mark.parametrize("live", [1, 129, 128 * 613 + 37])
@pytest.mark.parametrize("relation", REL)
@pytest.mark.parametrize("split", [False, True])
def test_fused_training_reads_the_live_count(cb, guard_rows, name, extra, live, relation, split):
    """cednerf_field_train_fwd/bwd with a device count: the live rows and every gradient match the exact-size run;
    upstream gradients of the tail rows are NaN and must not be read.  `split`: the table-gradient hook's two phases."""
    ops = cb.ops
    field = trained_field(cb, name, extra).train()
    ridx, t0, t1, o, d, ts, n_rays = packed_inputs(live)
    cap, nd = capacity_and_ndev(live, relation)
    (_, R), (_, A), (_, B) = padded(ridx, cap, 0), padded(t0, cap), padded(t1, cap)
    R._cednerf_counts = (None, torch.tensor([nd], dtype=torch.int64, device=DEV))
    g = torch.Generator().manual_seed(live)
    g_rgb, g_sig = torch.rand(live, 3, generator=g).to(DEV), torch.rand(live, generator=g).to(DEV)
    g_lat = torch.rand(live, 32, generator=g).to(DEV) * 0.1

    def run(r, a, b, n):
        def pad(x):
            return padded(x, n)[1] if n > live else x

        rgb, res = field.fused_train(r, a, b, o, d, ts, 1)
        for q in field.parameters():
            q.grad = None
        loss = (rgb * pad(g_rgb)).sum() + (res["density"].view(-1) * pad(g_sig)).sum()
        lat = res["interal_output"].get("latent_losses")
        if lat is not None and lat.numel():
            loss = loss + (lat * pad(g_lat)).sum()
        (loss * 64.0).backward()
        return rgb.detach()[:live], res["density"].detach()[:live], {k: q.grad.clone() for k, q in
                                                                  field.named_parameters() if q.grad is not None}

    if split:
        ops.set_table_grad_hook(lambda gt: None)
    try:
        got = run(R, A, B, cap)
        ref = run(R[:live].clone(), A[:live], B[:live], live)
    finally:
        ops.set_table_grad_hook(None)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    assert set(got[2]) == set(ref[2])
    for k, gr in ref[2].items():
        assert bool(torch.isfinite(got[2][k]).all()), k
        assert rel(got[2][k], gr) <= 2e-6, (k, rel(got[2][k], gr))


@pytest.mark.parametrize("live", LIVE)
@pytest.mark.parametrize("relation", REL)
@pytest.mark.parametrize("C", [1, 3, 12, 32])
def test_accumulate_reads_the_live_count(cb, guard_rows, live, relation, C):
    ops = cb.ops
    n_rays = 97
    g = torch.Generator().manual_seed(live + C)
    ridx = torch.sort(torch.randint(0, n_rays, (live,), generator=g))[0]
    off = torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(torch.bincount(ridx, minlength=n_rays), 0)]).to(DEV)
    w, v = torch.rand(live, generator=g), torch.randn(live, C, generator=g)
    cap, nd = capacity_and_ndev(live, relation)
    (_, R), (_, W), (_, V) = padded(ridx, cap, 0), padded(w, cap), padded(v, cap)
    n_dev = torch.tensor([nd], dtype=torch.int64, device=DEV)
    g_out = torch.rand(n_rays, C, generator=g).to(DEV)

    def run(r, ww, vv, nd_):
        ww, vv = ww.clone().requires_grad_(True), vv.clone().requires_grad_(True)
        out = ops.AccumulateFunction.apply(ww, vv, r, off, n_rays, nd_)
        (out * g_out).sum().backward()
        return out.detach(), ww.grad[:live], vv.grad[:live]

    got, ref = run(R, W, V, n_dev), run(R[:live], W[:live], V[:live], None)
    for x, y in zip(got, ref):
        assert torch.equal(x, y)


@pytest.mark.parametrize("live", LIVE)
@pytest.mark.parametrize("relation", REL)
def test_training_loss_reads_the_live_count(cb, guard_rows, live, relation):
    from cednerf_b200.losses import TrainingLossFunction

    n_rays = 97
    g = torch.Generator().manual_seed(live)
    ridx = torch.sort(torch.randint(0, n_rays, (live,), generator=g))[0]
    rgb, acc, pix = (torch.rand(n_rays, k, generator=g).to(DEV) for k in (3, 1, 3))
    rgbs, w = torch.rand(live, 3, generator=g), torch.rand(live, generator=g)
    lat = torch.rand(n_rays, 32, generator=g).to(DEV)
    cap, nd = capacity_and_ndev(live, relation)
    (_, R), (_, RG), (_, W) = padded(ridx, cap, 0), padded(rgbs, cap), padded(w, cap)
    n_dev = torch.tensor([nd], dtype=torch.int64, device=DEV)

    def run(r, rg, ww, nd_):
        xs = [t.clone().requires_grad_(True) for t in (rgb, acc, rg, lat)]
        loss = TrainingLossFunction.apply(xs[0], xs[1], pix, xs[2], ww, r, xs[3], 1e-3, 1e-3, nd_)
        loss.backward()
        return [loss.detach()] + [x.grad for x in xs[:2]] + [xs[2].grad[:live], xs[3].grad]

    got, ref = run(R, RG, W, n_dev), run(R[:live], RG[:live], W[:live], None)
    assert abs(float(got[0]) - float(ref[0])) <= 1e-6 * abs(float(ref[0]))   # fp64 sums, reduced in launch order
    for x, y in zip(got[1:], ref[1:]):
        assert torch.equal(x, y)


@pytest.mark.parametrize("live", LIVE[1:])
@pytest.mark.parametrize("empty_tail", [False, True])
def test_distortion_on_a_capacity_sized_set(cb, poison, live, empty_tail):
    """losses.distortion on counts-carrying inputs equals the exact-size call, including a batch whose last rays have
    no samples (the loss is normalised by the last ray with samples + 1)."""
    n_rays = 97
    g = torch.Generator().manual_seed(live)
    top = n_rays - 20 if empty_tail else n_rays
    ridx = torch.sort(torch.randint(0, top, (live,), generator=g))[0]
    t0 = torch.sort(torch.rand(live, generator=g))[0] + ridx.float()
    t1, w = t0 + 0.01, torch.rand(live, generator=g)
    cap = live + 300
    off = torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(torch.bincount(ridx, minlength=n_rays), 0)]).to(DEV)
    (_, R), (_, A), (_, B), (_, W) = padded(ridx, cap, 0), padded(t0, cap), padded(t1, cap), padded(w, cap)
    R._cednerf_counts = (off, torch.tensor([live], dtype=torch.int64, device=DEV))
    wc, we = W.clone().requires_grad_(True), W[:live].clone().requires_grad_(True)
    lc = cb.losses.distortion(R, wc, A, B, n_rays=n_rays)
    le = cb.losses.distortion(R[:live].clone(), we, A[:live], B[:live])
    lc.backward(), le.backward()
    assert abs(float(lc.detach()) - float(le.detach())) <= 1e-6 * abs(float(le.detach()))
    assert torch.equal(wc.grad[:live], we.grad)


# ------------------------------------------------------------------------ E: the whole step, capacity vs host mode
N_STEP_RAYS = 2 ** 16 + 1234


def step_scene(cb, cfg_name):
    from cednerf_b200 import workload as wl

    cfg = getattr(wl, cfg_name)
    est, field = wl.build_scene(cfg, DEV, cb, seed=42)
    est.train(), field.train()
    b = {k: v.to(DEV) for k, v in wl.draw_batch(cfg, N_STEP_RAYS, torch.Generator().manual_seed(3)).items()}
    return cfg, wl.render_kwargs(cfg), est, field, b


def run_step(cb, cfg, rk, est, field, b, device_counts):
    """render_image + the loss exactly as bench.train_step builds them; -> outputs, loss, gradients."""
    for q in field.parameters():
        q.grad = None
    rgb, acc, depth, n_s, extra = cb.render_image(field, est, cb.Rays(b["origins"], b["viewdirs"]),
                                                  render_bkgd=b["color_bkgd"], timestamps=b["timestamps"],
                                                  jitter=b["jitter"], device_counts=device_counts, **rk)
    loss = cb.losses.training_loss(rgb, acc, b["pixels"], extra, acc_entropy_loss=True, weight_rgbper=True,
                                   use_feat_predict=bool(cfg.flags.get("use_feat_predict")),
                                   distortion_loss=cfg.name.startswith("hypernerf"))
    (loss * 1024.0).backward()
    grads = {k: q.grad.detach().clone() for k, q in field.named_parameters() if q.grad is not None}
    return rgb.detach(), acc.detach(), depth.detach(), n_s, extra[0], float(loss.detach()), grads


def record_visible(cb, monkeypatch):
    rec = []
    real = cb.ops.visible_samples_capped

    def wrapped(t0, t1, sigmas, offsets, n_rays, eps, athr, capacity):
        out = real(t0, t1, sigmas, offsets, n_rays, eps, athr, capacity)
        rec.append(dict(t0=t0.clone(), t1=t1.clone(), sigmas=sigmas.clone(), offsets=offsets.clone(), n_rays=n_rays,
                        eps=eps, athr=athr, cap=capacity, out=[x.clone() for x in out]))
        return out

    monkeypatch.setattr(cb.ops, "visible_samples_capped", wrapped)
    return rec


def assert_step_equal(got, ref, n):
    ex, ex_ref = got[4], ref[4]
    for i in range(3):
        assert torch.equal(got[i], ref[i]), i
    for k in ("ray_indices", "t_starts", "t_ends", "weights", "rgbs"):
        assert torch.equal(ex[k][:n], ex_ref[k]), k
    assert abs(got[5] - ref[5]) <= 1e-6 * abs(ref[5])
    assert set(got[6]) == set(ref[6])
    for k, g in ref[6].items():
        assert bool(torch.isfinite(got[6][k]).all()), k
        assert rel(got[6][k], g) <= 2e-6, (k, rel(got[6][k], g))


CONFIGS = ["TINY", "DNERF", "HYPERNERF", "DYNERF"]


@pytest.mark.parametrize("cfg_name", CONFIGS)
def test_step_without_drops_matches_host_mode_at_every_capacity(cb, poison, monkeypatch, cfg_name):
    cfg, rk, est, field, b = step_scene(cb, cfg_name)
    ref = run_step(cb, cfg, rk, est, field, b, False)
    n_v = ref[3]
    rec = record_visible(cb, monkeypatch)
    raw_m = march_oracle_for(cb, est, b, rk)[0].numel()
    caps = {"marched": raw_m, "visible": n_v}
    for kind in caps:
        est._seed_capacity(kind, 1)   # the totals queue of each kind exists
    monkeypatch.setattr(est, "_capacity", lambda kind: caps[kind])
    tried = 0
    for cap_m in bucket_capacities(raw_m, N_STEP_RAYS):
        for cap_v in bucket_capacities(n_v, N_STEP_RAYS):
            caps.update(marched=cap_m, visible=cap_v)
            rec.clear()
            got = run_step(cb, cfg, rk, est, field, b, True)
            assert int(rec[0]["offsets"][-1]) == raw_m and int(rec[0]["out"][4][1]) == n_v
            assert int(got[3]) == n_v and got[4]["t_starts"].numel() == cap_v
            assert_step_equal(got, ref, n_v)
            tried += 1
    assert tried >= 2


def march_oracle_for(cb, est, b, rk):
    """The host-count marched set of the batch (est.march with the batch's jitter) and its per-ray run counts."""
    ops = cb.ops
    n = b["origins"].shape[0]
    ridx, t0, t1, packed = est.march(b["origins"], b["viewdirs"], rk["near_plane"], 1e10, rk["render_step_size"],
                                     rk["cone_angle"], stratified=True, jitter=b["jitter"])
    near = torch.full((n,), float(rk["near_plane"]), device=DEV) + b["jitter"] * rk["render_step_size"]
    from cednerf_b200.nerfacc.grid import occupancy_bits

    mi = ops.MarchInputs(b["origins"], b["viewdirs"], occupancy_bits(est.binaries), est.aabbs, int(est.binaries.shape[1]),
                         near, torch.full((n,), 1e10, device=DEV), float(rk["near_plane"]), 1e10, rk["render_step_size"],
                         rk["cone_angle"])
    mi.count(record_runs=True)
    return ridx.cpu(), t0.cpu(), t1.cpu(), packed[:, 1].cpu(), mi.runs[2].cpu()


@pytest.mark.parametrize("cfg_name", CONFIGS)
@pytest.mark.parametrize("drop", ["marched", "visible", "both"])
def test_step_with_drops_matches_the_exact_pipeline_on_the_truncated_sets(cb, poison, monkeypatch, cfg_name, drop):
    from cednerf_b200 import utils as cu
    from cednerf_b200.render import rendering

    cfg, rk, est, field, b = step_scene(cb, cfg_name)
    ref = run_step(cb, cfg, rk, est, field, b, False)
    m_ridx, m_t0, m_t1, m_cnt, m_runs = march_oracle_for(cb, est, b, rk)
    raw_m = m_ridx.numel()
    cap_m = int(raw_m * 0.6) if drop in ("marched", "both") else raw_m + 1000
    # the visible total of the marched stage (truncated or not) decides the visible capacity
    caps = {"marched": cap_m, "visible": cap_m}
    for kind in caps:
        est._seed_capacity(kind, 1)   # the totals queue of each kind exists
    monkeypatch.setattr(est, "_capacity", lambda kind: caps[kind])
    rec = record_visible(cb, monkeypatch)
    probe = run_step(cb, cfg, rk, est, field, b, True)
    raw_v = int(rec[-1]["out"][4][1])
    caps["visible"] = int(raw_v * 0.6) if drop in ("visible", "both") else raw_v + 1000
    rec.clear()
    got = run_step(cb, cfg, rk, est, field, b, True)
    r = rec[-1]
    assert int(r["offsets"][-1]) == min(cap_m, raw_m) and r["cap"] == caps["visible"]
    # marched live prefix: the drop contract against the host-count march
    e_r, e_a, e_b, k = capped_expectation(m_ridx, m_t0, m_t1, m_cnt, m_runs, cb.ops.MarchInputs.RUN_CAP, cap_m)
    assert torch.equal(r["t0"][:k].cpu(), e_a) and torch.equal(r["t1"][:k].cpu(), e_b)
    m_off = torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(m_cnt.long(), 0)])
    assert torch.equal(r["offsets"].cpu(), torch.clamp(m_off, max=cap_m))
    # sigmas: sigma_fn on exact-size copies of the marched prefix
    rays = cb.Rays(b["origins"], b["viewdirs"])
    sigma_fn, rgb_sigma_fn = cu._field_fns(field, rays, b["timestamps"])
    with torch.no_grad():
        sig = sigma_fn(e_a.to(DEV), e_b.to(DEV), e_r.to(DEV))
    assert torch.equal(r["sigmas"][:k], sig)
    # visible live prefix: the exact-size compaction of that prefix, truncated to the visible capacity
    off_m = r["offsets"]
    v_r, v_a, v_b = cb.ops.visible_samples(e_a.to(DEV), e_b.to(DEV), sig, off_m, N_STEP_RAYS, r["eps"], r["athr"])
    kv = min(caps["visible"], v_r.numel())
    assert int(got[3]) == kv and int(r["out"][4][0]) == kv and int(r["out"][4][1]) == v_r.numel()
    assert drop == "marched" or kv < v_r.numel()
    ex = got[4]
    v_r, v_a, v_b = v_r[:kv].clone(), v_a[:kv].clone(), v_b[:kv].clone()
    assert torch.equal(ex["ray_indices"][:kv], v_r) and torch.equal(ex["t_starts"][:kv], v_a)
    assert torch.equal(ex["t_ends"][:kv], v_b)
    # render, loss and gradients: the exact-size pipeline on the truncated visible set
    for q in field.parameters():
        q.grad = None
    rgb, acc, depth, extras = rendering(v_a, v_b, v_r, N_STEP_RAYS, rgb_sigma_fn=rgb_sigma_fn,
                                        render_bkgd=b["color_bkgd"])
    extras.update(ray_indices=v_r, t_starts=v_a, t_ends=v_b)
    loss = cb.losses.training_loss(rgb, acc, b["pixels"], [extras], acc_entropy_loss=True, weight_rgbper=True,
                                   use_feat_predict=bool(cfg.flags.get("use_feat_predict")),
                                   distortion_loss=cfg.name.startswith("hypernerf"))
    (loss * 1024.0).backward()
    grads = {kk: q.grad.detach().clone() for kk, q in field.named_parameters() if q.grad is not None}
    assert_step_equal(got, (rgb.detach(), acc.detach(), depth.detach(), kv, extras, float(loss), grads), kv)


@pytest.mark.parametrize("cfg_name", ["TINY", "HYPERNERF"])
def test_dropped_samples_are_counted_and_the_next_step_has_none(cb, poison, monkeypatch, cfg_name):
    cfg, rk, est, field, b = step_scene(cb, cfg_name)
    ref = run_step(cb, cfg, rk, est, field, b, False)
    run_step(cb, cfg, rk, est, field, b, True)          # no capacity known: host-count path, seeds the capacities
    rec = record_visible(cb, monkeypatch)
    for kind in ("marched", "visible"):
        est._cap_state[kind]["last"] = est._cap_state[kind]["last"] // 3
        est._cap_state[kind]["pending"].clear()
    cap_m, cap_v = est._capacity("marched"), est._capacity("visible")
    before = est.dropped_samples
    short = run_step(cb, cfg, rk, est, field, b, True)
    torch.cuda.synchronize()
    est._capacity("marched"), est._capacity("visible")
    r = rec[-1]
    raw_v = int(r["out"][4][1])
    m_tot = est._cap_state["marched"]["last"]
    expect = max(0, m_tot - cap_m) + max(0, raw_v - cap_v)
    assert est.dropped_samples - before == expect > 0
    assert int(short[3]) == min(raw_v, cap_v)
    nxt = run_step(cb, cfg, rk, est, field, b, True)
    torch.cuda.synchronize()
    est._capacity("marched"), est._capacity("visible")
    assert est.dropped_samples - before == expect
    assert_step_equal(nxt, ref, ref[3])
