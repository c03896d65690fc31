"""nerfacc.estimators.occ_grid.OccGridEstimator surface (reference: ctor train_real.py:185-187, .sampling
cednerf/utils.py:115-125, .update_every_n_steps train_real.py:332-336, state_dict train_real.py:438)."""
from __future__ import annotations

import math
from typing import Callable, Optional

import torch

from ... import ops
from ..grid import occupancy_bits, set_occupancy_bits


class OccGridEstimator(torch.nn.Module):
    def __init__(self, roi_aabb, resolution: int = 128, levels: int = 1):
        super().__init__()
        roi = torch.as_tensor(roi_aabb, dtype=torch.float32).flatten()
        centre, half = (roi[:3] + roi[3:]) / 2, (roi[3:] - roi[:3]) / 2
        aabbs = torch.stack([torch.cat([centre - half * 2 ** l, centre + half * 2 ** l]) for l in range(levels)])
        self.levels, self.cells_per_lvl = int(levels), int(resolution) ** 3
        if self.cells_per_lvl % 32:
            raise ValueError("resolution^3 must be a multiple of 32")
        self.register_buffer("resolution", torch.tensor([resolution] * 3, dtype=torch.int32))
        self.register_buffer("aabbs", aabbs)
        self.register_buffer("occs", torch.zeros(self.levels * self.cells_per_lvl))
        self.register_buffer("binaries", torch.zeros(levels, resolution, resolution, resolution, dtype=torch.bool))
        g = torch.arange(resolution)
        coords = torch.stack(torch.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
        self.register_buffer("grid_coords", coords, persistent=False)
        self.register_buffer("grid_indices", torch.arange(self.cells_per_lvl), persistent=False)
        self._occ_mean_key, self._occ_mean = None, 0.0
        self._may_have_invisible, self._occs_seen = False, None  # occs = -1 cells exist (mark_invisible_cells, checkpoints)
        self._cap_state, self.dropped_samples = {}, 0  # sampling(..., device_counts=True)
        self._aabbs_host, self._occ_cand, self._occ_touched = None, None, None  # fused occupancy update

    def aabbs_on_host(self):
        """The level boxes as nested host lists (one host read, repeated only when the buffer changes)."""
        if self._aabbs_host is None or self._aabbs_host[0] != (self.aabbs.data_ptr(), self.aabbs._version):
            self._aabbs_host = ((self.aabbs.data_ptr(), self.aabbs._version), self.aabbs.cpu().tolist())
        return self._aabbs_host[1]

    def _load_from_state_dict(self, *args, **kwargs):
        self._occs_seen = None  # contents replaced in place: look again at the next update
        return super()._load_from_state_dict(*args, **kwargs)

    @property
    def device(self):
        return self.aabbs.device

    def _occs_mean(self) -> float:
        """occs.mean() as nerfacc reads it in .sampling; one host read per occupancy version."""
        key = (self.occs.data_ptr(), self.occs._version)
        if key != self._occ_mean_key:
            self._occ_mean, self._occ_mean_key = float(self.occs.mean().item()), key
        return self._occ_mean

    @torch.no_grad()
    def march(self, rays_o, rays_d, near_plane=0.0, far_plane=1e10, render_step_size=1e-3, cone_angle=0.0,
              stratified=False, jitter: Optional[torch.Tensor] = None, t_min=None, t_max=None):
        """Two-pass marching -> (ray_indices, t_starts, t_ends, packed_info).  One host read (the total)."""
        n = rays_o.shape[0]
        near = far = None
        if stratified or t_min is not None or t_max is not None:
            near = torch.full((n,), float(near_plane), device=rays_o.device)
            far = torch.full((n,), float(far_plane), device=rays_o.device)
            if t_min is not None:
                near = torch.clamp(near, min=t_min)
            if t_max is not None:
                far = torch.clamp(far, max=t_max)
            if stratified:
                u = torch.rand(n, device=rays_o.device) if jitter is None else jitter.to(rays_o.device).float()
                near = near + u * render_step_size
        mi = ops.MarchInputs(rays_o, rays_d, occupancy_bits(self.binaries), self.aabbs, int(self.binaries.shape[1]),
                             near, far, float(near_plane), float(far_plane), render_step_size, cone_angle)
        if stratified and n >= 65536:  # a large batch of (random) training rays
            mi.sort_for_coherence()
        _, n_sm, _ = mi.count(record_runs=True)
        starts, packed, total = ops.exclusive_scan(n_sm)
        if mi.runs is not None:
            ridx, t0, t1 = mi.fill_packed_from_runs(starts, int(total.item()))
        else:
            ridx, t0, t1, _ = mi.fill_packed(starts, int(total.item()))
        return ridx, t0, t1, packed

    # ---- capacities of the sync-free path ------------------------------------------------------------------------
    # The sample totals of a batch are copied to pinned host memory asynchronously and looked at when a LATER batch is
    # sampled: a capacity is 1.25 x the newest total that has arrived.  A batch that outgrows it loses its last samples
    # (totals[1] > totals[0]); `dropped_samples` counts them and the next capacity already covers the new total.
    _HEADROOM = 1.25

    def _capacity(self, kind: str):
        st = self._cap_state.setdefault(kind, {"last": None, "pending": [], "ring": [], "next": 0})
        while st["pending"] and st["pending"][0][0].query():
            _, host, cap, marched = st["pending"].pop(0)
            raw = int(host[1])
            st["last"] = raw
            if raw > cap:
                self.dropped_samples += raw - cap
            if marched is not None and int(marched[1]) > int(marched[0]):
                # the visible samples of a truncated marched set: scaled up to the whole set (and at most all of it),
                # or the next batch would outgrow this capacity as well
                kept_m, raw_m = int(marched[0]), int(marched[1])
                st["last"] = min(-(-raw * raw_m // kept_m), raw_m) if kept_m else raw_m
        if st["last"] is None:
            return None
        return ops._sticky_capacity(max(int(st["last"] * self._HEADROOM), 65536))

    def _note_totals(self, kind: str, totals: torch.Tensor, cap: int, marched: Optional[torch.Tensor] = None):
        """Queue the copy of a batch's totals (and, for the visible ones, the same batch's marched totals) to the host."""
        st = self._cap_state[kind]
        if not st["ring"]:
            st["ring"] = [tuple(torch.empty(2, dtype=torch.int64).pin_memory() for _ in range(2)) for _ in range(32)]
        if len(st["pending"]) >= len(st["ring"]):   # the host ran 32 batches ahead of the device: wait for the oldest
            st["pending"][0][0].synchronize()
            self._capacity(kind)
        host, host_m = st["ring"][st["next"] % len(st["ring"])]
        st["next"] += 1
        host.copy_(totals, non_blocking=True)
        if marched is not None:
            host_m.copy_(marched, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        st["pending"].append((ev, host, cap, None if marched is None else host_m))

    def _seed_capacity(self, kind: str, total: int):
        self._cap_state.setdefault(kind, {"last": None, "pending": [], "ring": [], "next": 0})["last"] = int(total)

    @torch.no_grad()
    def _sampling_device_counts(self, rays_o, rays_d, sigma_fn, near_plane, far_plane, render_step_size, early_stop_eps,
                                alpha_thre, cone_angle, jitter):
        """.sampling for a stratified training batch without any host read: capacity-sized outputs whose ray_indices
        carry (offsets, live count) - see ops.counts_of.  None when no capacity is known yet (first batch)."""
        cap_m, cap_v = self._capacity("marched"), self._capacity("visible")
        if cap_m is None or cap_v is None or render_step_size <= 0:
            return None
        n = rays_o.shape[0]
        u = torch.rand(n, device=rays_o.device) if jitter is None else jitter.to(rays_o.device).float()
        near = torch.full((n,), float(near_plane), device=rays_o.device) + u * render_step_size
        far = torch.full((n,), float(far_plane), device=rays_o.device)
        mi = ops.MarchInputs(rays_o, rays_d, occupancy_bits(self.binaries), self.aabbs, int(self.binaries.shape[1]),
                             near, far, float(near_plane), float(far_plane), render_step_size, cone_angle)
        if n >= 65536:
            mi.sort_for_coherence()
        _, n_sm, _ = mi.count(record_runs=True)
        offsets, totals = ops.exclusive_scan_capped(n_sm, cap_m)
        ridx, t0, t1 = mi.fill_packed_capped(offsets, n_sm, cap_m)
        self._note_totals("marched", totals, cap_m)
        ridx._cednerf_counts = (offsets, totals[0:1])
        sigmas = sigma_fn(t0, t1, ridx)
        assert sigmas.shape == t0.shape, f"sigmas must have shape {tuple(t0.shape)}"
        k_idx, k_t0, k_t1, k_off, k_tot = ops.visible_samples_capped(t0, t1, sigmas, offsets, n, early_stop_eps,
                                                                     min(alpha_thre, self._occs_mean()), cap_v)
        self._note_totals("visible", k_tot, cap_v, totals)
        k_idx._cednerf_counts = (k_off, k_tot[0:1])
        return k_idx, k_t0, k_t1

    @torch.no_grad()
    def sampling(self, rays_o, rays_d, sigma_fn: Optional[Callable] = None, alpha_fn: Optional[Callable] = None,
                 near_plane: float = 0.0, far_plane: float = 1e10, t_min=None, t_max=None,
                 render_step_size: float = 1e-3, early_stop_eps: float = 1e-4, alpha_thre: float = 0.0,
                 stratified: bool = False, cone_angle: float = 0.0, jitter: Optional[torch.Tensor] = None,
                 device_counts: bool = False):
        """device_counts=True (stratified training batches with a sigma_fn): no host read - see render_image."""
        if alpha_fn is not None:
            raise NotImplementedError("alpha_fn is not used by the reference")
        device_counts = (device_counts and stratified and sigma_fn is not None and t_min is None and t_max is None
                         and (alpha_thre > 0 or early_stop_eps > 0))
        if device_counts:
            out = self._sampling_device_counts(rays_o, rays_d, sigma_fn, near_plane, far_plane, render_step_size,
                                               early_stop_eps, alpha_thre, cone_angle, jitter)
            if out is not None:
                return out
        ridx, t0, t1, packed = self.march(rays_o, rays_d, near_plane, far_plane, render_step_size, cone_angle,
                                          stratified, jitter, t_min, t_max)
        if device_counts:
            self._seed_capacity("marched", t0.numel())
        if (alpha_thre > 0 or early_stop_eps > 0) and sigma_fn is not None:
            alpha_thre = min(alpha_thre, self._occs_mean())
            if t0.numel():
                sigmas = sigma_fn(t0, t1, ridx)
                assert sigmas.shape == t0.shape, f"sigmas must have shape {tuple(t0.shape)}"
                ridx, t0, t1 = ops.visible_samples(t0, t1, sigmas, ops.offsets_from_packed(packed), rays_o.shape[0],
                                                   early_stop_eps, alpha_thre)
        if device_counts:
            self._seed_capacity("visible", t0.numel())
        return ridx, t0, t1

    @torch.no_grad()
    def mark_invisible_cells(self, K, c2w, width: int, height: int, near_plane: float = 0.0, chunk: int = 32 ** 3):
        """nerfacc's call of train_real.py:205-211: occs = -1 for cells outside every camera frustum (or closer than
        near_plane to one); `_update` never touches them again.  `chunk` is accepted and ignored (one launch)."""
        assert K.dim() == 3 and K.shape[1:] == (3, 3)
        assert c2w.dim() == 3 and (c2w.shape[1:] == (3, 4) or c2w.shape[1:] == (4, 4))
        assert K.shape[0] == c2w.shape[0] or K.shape[0] == 1
        dev = self.device
        K, c2w = K.to(dev, torch.float32).contiguous(), c2w.to(dev, torch.float32).contiguous()
        ops.call("cednerf_occ_mark_invisible", ops.ptr(K), K.shape[0], ops.ptr(c2w), c2w.shape[0], c2w.shape[1],
                 ops.ptr(self.aabbs), self.levels, int(self.binaries.shape[1]), int(width), int(height), float(near_plane),
                 ops.ptr(self.occs), ops.stream())
        self._may_have_invisible = True
        self.occs.add_(0)  # bump the version: `occs.mean()` is cached per version for `.sampling`

    @torch.no_grad()
    def update_every_n_steps(self, step: int, occ_eval_fn: Callable, occ_thre: float = 1e-2, ema_decay: float = 0.95,
                             warmup_steps: int = 256, n: int = 16, rng=None):
        if not self.training:
            raise RuntimeError("update_every_n_steps() is a training-time call (estimator.train())")
        if step % n == 0:
            self._update(step, occ_eval_fn, occ_thre, ema_decay, warmup_steps, rng)

    def _fused_occ_eval(self, occ_eval_fn):
        """The FieldOccEval behind `occ_eval_fn` when its field can run the fused occupancy update, else None."""
        from ...utils import FieldOccEval

        if not isinstance(occ_eval_fn, FieldOccEval):
            return None
        f = occ_eval_fn.field
        ok = getattr(f, "fused_supported", lambda: False)() and self.occs.is_cuda and self.occs.dtype == torch.float32
        return occ_eval_fn if ok else None

    def _update_level_fused(self, l: int, idx, fn, rand, ema_decay: float, unique: bool):
        """One level of `_update` in one launch (cednerf_occ_update_level); draws in the order of the op-by-op path."""
        import ctypes

        dev, cpl = self.device, self.cells_per_lvl
        n = cpl if idx is None else int(idx.numel())
        if n == 0:
            return
        jitter = rand(n, 3).to(dev).float().contiguous()
        tt = fn.rand_t(n, dev).float().contiguous().view(-1)
        f = fn.field
        box = (ctypes.c_float * 6)(*self.aabbs_on_host()[l])
        cells = None if idx is None else idx.to(torch.int64).contiguous()
        cand = touched = None
        if not unique:
            if self._occ_cand is None or self._occ_cand.device != dev:
                self._occ_cand = torch.zeros(cpl, device=dev)
                self._occ_touched = torch.zeros(cpl, dtype=torch.uint8, device=dev)
            cand, touched = self._occ_cand, self._occ_touched
        lvl = self.occs[l * cpl:(l + 1) * cpl]
        ops.call("cednerf_occ_update_level", ops.ptr(cells), n, ops.ptr(jitter), ops.ptr(tt), box, int(self.binaries.shape[1]),
                 float(fn.step), float(ema_decay), ops.ptr(f.xyz_wrap.network.weight_image()), ops.ptr(f.mlp_base.weight_image()),
                 ops.ptr(f.hash_encoder.table_f16()), ctypes.byref(f._field_desc()), ops.ptr(lvl), ops.ptr(cand),
                 ops.ptr(touched), ops.stream())

    @torch.no_grad()
    def _update(self, step, occ_eval_fn, occ_thre=1e-2, ema_decay=0.95, warmup_steps=256, rng=None):
        """SURVEY.md Appendix A.2.  `rng` (randint(high, n), rand(*shape)) lets parity tests share draws."""
        dev, cpl = self.device, self.cells_per_lvl
        randint = (lambda hi, k: torch.randint(hi, (k,), device=dev)) if rng is None else rng.randint
        rand = (lambda *s: torch.rand(*s, device=dev)) if rng is None else rng.rand
        # `all_valid`: no cell has been marked invisible (occs = -1 comes only from mark_invisible_cells or a loaded
        # checkpoint), so "cells with occs >= 0" is every cell and none of the compactions below - each one a host
        # read - is needed
        if self._occs_seen != self.occs.data_ptr():  # buffer replaced (assignment, .to(), load): look once (one host read)
            self._may_have_invisible = bool((self.occs < 0).any())
            self._occs_seen = self.occs.data_ptr()
        all_valid = not self._may_have_invisible
        lvl_indices = []
        if step < warmup_steps:
            for l in range(self.levels):
                lvl_indices.append(None if all_valid else self.grid_indices[self.occs[l * cpl + self.grid_indices] >= 0])
        else:
            k = cpl // 4
            for l in range(self.levels):
                uni = randint(cpl, k).to(dev)
                if not all_valid:
                    uni = uni[self.occs[l * cpl + uni] >= 0]
                occ_idx = torch.nonzero(self.binaries[l].flatten())[:, 0]
                if k < len(occ_idx):
                    occ_idx = occ_idx[randint(len(occ_idx), k).to(dev)]
                lvl_indices.append(torch.cat([uni, occ_idx]))
        fused = self._fused_occ_eval(occ_eval_fn)
        for l, idx in enumerate(lvl_indices):
            if fused is not None:
                self._update_level_fused(l, idx, fused, rand, ema_decay, unique=step < warmup_steps)
                continue
            coords = self.grid_coords if idx is None else self.grid_coords[idx]
            x = (coords.float() + rand(coords.shape[0], 3).to(dev)) / self.resolution.float()
            x = self.aabbs[l, :3] + x * (self.aabbs[l, 3:] - self.aabbs[l, :3])
            occ = occ_eval_fn(x).squeeze(-1).float()
            if idx is None:  # every cell of the level exactly once: an element-wise maximum, no scatter
                lvl = self.occs[l * cpl:(l + 1) * cpl]
                torch.maximum(lvl * ema_decay, occ, out=lvl)
                continue
            cell = l * cpl + idx
            # nerfacc writes occs[cell] = max(occs[cell]*decay, occ) with an index_put whose winner among duplicate
            # cells (uniform draws that repeat or coincide with occupied cells) is undefined on CUDA; here the
            # largest candidate wins (scatter-amax), which is one of those outcomes and is deterministic.
            self.occs.scatter_reduce_(0, cell, torch.maximum(self.occs[cell] * ema_decay, occ), "amax",
                                      include_self=False)
        if all_valid:
            thre = torch.clamp(self.occs.mean(), max=occ_thre).reshape(1).contiguous()
        else:
            valid = self.occs >= 0
            thre = torch.clamp((self.occs * valid).sum() / valid.sum(), max=occ_thre).reshape(1).contiguous()
        bits = torch.empty(self.occs.numel() // 32, dtype=torch.int32, device=dev)
        ops.occ_threshold_pack(self.occs, thre, self.binaries, bits)
        set_occupancy_bits(self.binaries, bits)
