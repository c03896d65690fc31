"""Thin torch-side wrappers over the C ABI: allocation, autograd.Function glue, nothing else.

Every function here ends in a call into libcednerf_b200.so; none computes on the host or through
PyTorch operators (PyTorch is used for device memory, streams and autograd bookkeeping only).
"""
from __future__ import annotations

import ctypes
import math
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import FieldDesc, GridLevels, MlpDesc, call, ptr, stream

F32, F16, I64, I32, U8 = torch.float32, torch.float16, torch.int64, torch.int32, torch.uint8


def _f32c(t: torch.Tensor) -> torch.Tensor:
    _lib.check_device()
    if not t.is_cuda:
        raise RuntimeError("cednerf_b200 ops need CUDA tensors (no CPU fallback)")
    return t.detach().to(F32).contiguous()


# ------------------------------------------------------------------------------------------------
# K1 marching
# ------------------------------------------------------------------------------------------------
def ray_aabb_intersect(rays_o, rays_d, aabbs, near_plane=-math.inf, far_plane=math.inf, miss_value=math.inf):
    o, d, bx = _f32c(rays_o), _f32c(rays_d), _f32c(aabbs)
    n, nl = o.shape[0], bx.shape[0]
    t_mins = torch.empty(n, nl, device=o.device)
    t_maxs = torch.empty(n, nl, device=o.device)
    hits = torch.empty(n, nl, dtype=torch.bool, device=o.device)
    call("cednerf_ray_aabb_intersect", ptr(o), ptr(d), n, ptr(bx), nl, near_plane, far_plane, miss_value,
         ptr(t_mins), ptr(t_maxs), ptr(hits), stream())
    return t_mins, t_maxs, hits


def sort_boundaries(t_mins, t_maxs):
    a, b = _f32c(t_mins), _f32c(t_maxs)
    n, nl = a.shape
    t_sorted = torch.empty(n, 2 * nl, device=a.device)
    t_indices = torch.empty(n, 2 * nl, dtype=I64, device=a.device)
    call("cednerf_sort_boundaries", ptr(a), ptr(b), n, nl, ptr(t_sorted), ptr(t_indices), stream())
    return t_sorted, t_indices


def pack_occupancy(binaries: torch.Tensor) -> torch.Tensor:
    """bool [L,R,R,R] -> uint32 bit field (int32 storage), 1 bit per cell in the same order, the last word zero-padded."""
    _lib.check_device()
    b = binaries.detach().contiguous()
    if b.dtype != torch.bool and b.dtype != U8:
        b = b.to(torch.bool)
    n_cells = b.numel()
    bits = torch.empty((n_cells + 31) // 32, dtype=I32, device=b.device)
    call("cednerf_occ_pack_bits", ptr(b), n_cells, ptr(bits), stream())
    return bits


def occ_threshold_pack(occs: torch.Tensor, threshold: torch.Tensor, binaries: torch.Tensor, bits: torch.Tensor):
    call("cednerf_occ_threshold_pack", ptr(occs), occs.numel(), ptr(threshold), ptr(binaries), ptr(bits), stream())


def exclusive_scan(counts: torch.Tensor, want_packed: bool = True):
    """int32 counts -> (starts int64, packed_info int64 [n,2] or None, total int64 [1]); all on device."""
    n = counts.numel()
    dev = counts.device
    starts = torch.empty(n, dtype=I64, device=dev)
    packed = torch.empty(n, 2, dtype=I64, device=dev) if want_packed else None
    total = torch.empty(1, dtype=I64, device=dev)
    ws = torch.empty(max(int(_lib.load().cednerf_scan_workspace_bytes(n)) // 8, 1), dtype=I64, device=dev)
    call("cednerf_exclusive_scan", ptr(counts), n, ptr(starts), ptr(packed), ptr(total), ptr(ws), stream())
    return starts, packed, total


def counts_of(t: Optional[torch.Tensor]):
    """(offsets int64 [n_rays + 1], n_dev int64 [1]) attached to the ray_indices of a capacity-sized packed sample set
    (OccGridEstimator.sampling(..., device_counts=True)), else None.  Only the first n_dev[0] rows of such tensors are
    live; every kernel downstream reads the count from the device, so the host never waits for it."""
    return getattr(t, "_cednerf_counts", None) if t is not None else None


def exclusive_scan_capped(counts: torch.Tensor, capacity: int):
    """int32 counts -> (offsets int64 [n + 1] clamped to `capacity`, totals int64 [2] = (clamped, raw)); device only."""
    n, dev = counts.numel(), counts.device
    offsets = torch.empty(n + 1, dtype=I64, device=dev)
    totals = torch.empty(2, dtype=I64, device=dev)
    ws = torch.empty(max(int(_lib.load().cednerf_scan_workspace_bytes(n)) // 8, 1), dtype=I64, device=dev)
    call("cednerf_exclusive_scan_capped", ptr(counts), n, int(capacity), ptr(offsets), ptr(totals), ptr(ws), stream())
    return offsets, totals


def occupancy_coarse(bits: torch.Tensor, n_levels: int, res: int):
    """One bit per 4x4x4 block of cells (cednerf_occ_coarsen), cached on the bit-field tensor it was derived from (a new
    bit field is a new tensor).  None when the resolution is not a multiple of 4."""
    if res % 4 or bits is None:
        return None
    hit = getattr(bits, "_cednerf_coarse", None)
    if hit is not None and hit[0] == bits._version:
        return hit[1]
    words = (n_levels * (res // 4) ** 3 + 31) // 32
    coarse = torch.empty(words, dtype=I32, device=bits.device)
    call("cednerf_occ_coarsen", ptr(bits), n_levels, res, ptr(coarse), stream())
    bits._cednerf_coarse = (bits._version, coarse)
    return coarse


class MarchInputs:
    """Argument bundle shared by the count and fill passes."""

    def __init__(self, rays_o, rays_d, occ_bits, aabbs, resolution, near_planes=None, far_planes=None,
                 near_const=0.0, far_const=math.inf, step_size=1e-3, cone_angle=0.0, limit=-1, rays_mask=None,
                 t_sorted=None, t_indices=None, hits=None):
        self.o, self.d = _f32c(rays_o), _f32c(rays_d)
        self.bits, self.aabbs = occ_bits, _f32c(aabbs)
        self.n, self.nl, self.res = self.o.shape[0], self.aabbs.shape[0], int(resolution)
        self.near = None if near_planes is None else _f32c(near_planes)
        self.far = None if far_planes is None else _f32c(far_planes)
        self.near_const, self.far_const = float(near_const), float(far_const)
        self.step, self.cone, self.limit = float(step_size), float(cone_angle), int(limit)
        self.mask = None if rays_mask is None else rays_mask.detach().to(torch.bool).contiguous()
        self.t_sorted = None if t_sorted is None else _f32c(t_sorted)
        self.t_indices = None if t_indices is None else t_indices.detach().to(I64).contiguous()
        self.hits = None if hits is None else hits.detach().to(torch.bool).contiguous()
        self.order = None  # int32 permutation for the count pass (sort_for_coherence)
        # 4^3-block bits for the marcher's empty-space skip.  Measured: it pays in the marching rounds of render_image_test
        # (dense warps of coherent rays: -7 % per frame) and costs in the two-pass count of a training batch (+18 %: the
        # count pass is bound by the latency of the DDA's dependent chain, which the skipped look-ups are not on), so only
        # the rounds pass it (utils._render_rounds_on_device)
        self.coarse = None

    def sort_for_coherence(self):
        """Random training rays: march them in the order of a direction key so that the lanes of a warp walk
        neighbouring paths (the count pass is instruction-bound and half its lanes idle otherwise).  Outputs stay
        indexed by ray, so nothing downstream sees the permutation."""
        keys = torch.empty(self.n, dtype=I32, device=self.o.device)
        call("cednerf_ray_coherence_keys", ptr(self.d), self.n, ptr(keys), stream())
        self.order = torch.empty(self.n, dtype=I32, device=self.o.device)
        ws = torch.empty(16384, dtype=I32, device=self.o.device)
        call("cednerf_ray_coherence_order", ptr(keys), self.n, ptr(self.order), ptr(ws), stream())

    def _common(self, fill):
        return (fill, ptr(self.o), ptr(self.d), self.n, ptr(self.bits), ptr(self.aabbs), self.nl, self.res,
                ptr(self.near), ptr(self.far), self.near_const, self.far_const, self.step, self.cone, self.limit,
                ptr(self.mask), ptr(self.t_sorted), ptr(self.t_indices), ptr(self.hits))

    RUN_CAP = 16

    def count(self, record_runs: bool = False):
        dev = self.o.device
        n_iv = torch.empty(self.n, dtype=I32, device=dev)
        n_sm = torch.empty(self.n, dtype=I32, device=dev)
        term = torch.empty(self.n, device=dev)
        self.runs = None
        if record_runs and self.step > 0:
            self.runs = (torch.empty(self.n, self.RUN_CAP, device=dev), torch.empty(self.n, self.RUN_CAP, dtype=I32, device=dev),
                         torch.empty(self.n, dtype=I32, device=dev))
        rt, rn, nr = self.runs if self.runs is not None else (None, None, None)
        call("cednerf_march", *self._common(0), None, None, None, None, None, None, None, None, None, None, None,
             None, ptr(n_iv), ptr(n_sm), ptr(term), ptr(rt), ptr(rn), ptr(nr), self.RUN_CAP if rt is not None else 0,
             ptr(self.order), ptr(self.coarse), stream())
        return n_iv, n_sm, term

    def fill_packed_from_runs(self, sm_starts, total):
        """Packed fill replaying the recorded runs; rays with more than RUN_CAP runs take the full-march fill."""
        dev = self.o.device
        t0 = _sempty(total, device=dev)
        t1 = _sempty(total, device=dev)
        ridx = _sempty(total, dtype=I64, device=dev)
        overflow = torch.empty(self.n, dtype=torch.bool, device=dev)
        rt, rn, nr = self.runs
        call("cednerf_march_fill_runs", self.n, ptr(sm_starts), ptr(rt), ptr(rn), ptr(nr), self.RUN_CAP, self.step,
             self.cone, ptr(t0), ptr(t1), ptr(ridx), ptr(overflow), stream())
        # overflow is 0 for rays the caller masked out (their run count is 0), so it can stand in as the ray mask
        user_mask, self.mask = self.mask, overflow
        call("cednerf_march", *self._common(1), None, ptr(sm_starts), None, None, None, None, None, None, None,
             ptr(t0), ptr(t1), ptr(ridx), None, None, None, None, None, None, 0, None, ptr(self.coarse), stream())
        self.mask = user_mask
        return ridx, t0, t1

    def fill_packed_capped(self, offsets, n_sm, capacity):
        """fill_packed_from_runs into buffers of `capacity` samples: no host read of the total (offsets from
        exclusive_scan_capped); samples beyond the capacity are dropped."""
        dev = self.o.device
        t0 = torch.empty(capacity, device=dev)
        t1 = torch.empty(capacity, device=dev)
        ridx = torch.empty(capacity, dtype=I64, device=dev)
        overflow = torch.empty(self.n, dtype=torch.bool, device=dev)
        rt, rn, nr = self.runs
        call("cednerf_march_fill_runs_capped", self.n, ptr(offsets), ptr(n_sm), ptr(rt), ptr(rn), ptr(nr), self.RUN_CAP,
             self.step, self.cone, ptr(t0), ptr(t1), ptr(ridx), ptr(overflow), stream())
        user_mask, self.mask = self.mask, overflow   # rays over the run limit: full-march fill into their (whole) range
        call("cednerf_march", *self._common(1), None, ptr(offsets), None, None, None, None, None, None, None,
             ptr(t0), ptr(t1), ptr(ridx), None, None, None, None, None, None, 0, None, ptr(self.coarse), stream())
        self.mask = user_mask
        return ridx, t0, t1

    def fill_packed(self, sm_starts, total):
        dev = self.o.device
        t0 = _sempty(total, device=dev)
        t1 = _sempty(total, device=dev)
        ridx = _sempty(total, dtype=I64, device=dev)
        term = torch.empty(self.n, device=dev)
        call("cednerf_march", *self._common(1), None, ptr(sm_starts), None, None, None, None, None, None, None,
             ptr(t0), ptr(t1), ptr(ridx), None, None, ptr(term), None, None, None, 0, None, ptr(self.coarse), stream())
        return ridx, t0, t1, term

    def fill_nerfacc(self, iv_starts, sm_starts, n_iv_total, n_sm_total):
        dev = self.o.device
        iv_vals = torch.zeros(n_iv_total, device=dev)
        iv_left = torch.zeros(n_iv_total, dtype=torch.bool, device=dev)
        iv_right = torch.zeros(n_iv_total, dtype=torch.bool, device=dev)
        iv_ray = torch.zeros(n_iv_total, dtype=I64, device=dev)
        sm_vals = torch.zeros(n_sm_total, device=dev)
        sm_ray = torch.zeros(n_sm_total, dtype=I64, device=dev)
        sm_valid = torch.zeros(n_sm_total, dtype=torch.bool, device=dev)
        n_iv = torch.empty(self.n, dtype=I32, device=dev)
        n_sm = torch.empty(self.n, dtype=I32, device=dev)
        term = torch.empty(self.n, device=dev)
        call("cednerf_march", *self._common(1), ptr(iv_starts), ptr(sm_starts), ptr(iv_vals), ptr(iv_left),
             ptr(iv_right), ptr(iv_ray), ptr(sm_vals), ptr(sm_ray), ptr(sm_valid), None, None, None, ptr(n_iv),
             ptr(n_sm), ptr(term), None, None, None, 0, None, ptr(self.coarse), stream())
        return (iv_vals, iv_left, iv_right, iv_ray), (sm_vals, sm_ray, sm_valid), n_iv, n_sm, term


# ------------------------------------------------------------------------------------------------
# K2 hash grids
# ------------------------------------------------------------------------------------------------
def grid_levels(n_levels: int, base_resolution: float, log_per_level_scale: float, max_params: int):
    """Level geometry (cednerf/taichi_kernel/hash_encoder_half.py:12-35, :268-293); host arithmetic only.

    Returns (GridLevels struct, total entries, python lists for introspection)."""
    import numpy as np

    if n_levels > _lib.MAX_LEVELS:
        raise ValueError(f"at most {_lib.MAX_LEVELS} levels")
    g = GridLevels()
    g.n_levels = n_levels
    off = 0
    info = []
    for l in range(n_levels):
        s = float(base_resolution) * math.exp(float(l) * log_per_level_scale) - 1.0
        res = int(math.ceil(s)) + 1
        full = res ** 3
        size = min(int(max_params), (full + 7) // 8 * 8)
        if full > size and size & (size - 1):
            # every kernel reduces a hashed index with `& (size - 1)` (tcnn's and the reference's configurations are
            # 2^log2_hashmap_size); a table of another size would need the reference's `% size` in all of them
            raise ValueError(f"hashed level {l}: max_params must be a power of two, got {max_params}")
        g.scale[l] = float(np.float32(s))
        g.res[l], g.size[l], g.offset[l], g.hashed[l] = res, size, off, int(full > size)
        info.append((float(np.float32(s)), res, size, off, full > size))
        off += size
    return g, off, info


def cast_f16(src: torch.Tensor) -> torch.Tensor:
    s = _f32c(src).view(-1)
    dst = torch.empty(s.numel(), dtype=F16, device=s.device)
    call("cednerf_cast_f32_to_f16", ptr(s), ptr(dst), s.numel(), stream())
    return dst


def _cap(n: int) -> int:
    return (int(n) + 32767) // 32768 * 32768


# Sample-sized buffers: the number of marched / visible samples changes a little with every batch, and a caching
# allocator serves a request that is a few KB larger than last time with fresh cudaMallocs (bursts of 10-100 ms when a
# size class boundary is crossed).  `_sempty` therefore allocates at a sticky capacity - the smallest remembered one in
# [n, 1.3 n], else a new one 10 % above n - and returns the leading n rows: in the steady state of a training loop every
# request repeats the size of the previous step exactly.
_capacities: List[int] = []


def _sticky_capacity(n: int) -> int:
    n = int(n)
    if n < 65536:
        return n
    best = 0
    for c in _capacities:
        if n <= c <= n * 13 // 10 and (best == 0 or c < best):
            best = c
    if best == 0:
        best = (n * 11 // 10 + 65535) // 65536 * 65536
        _capacities.append(best)
        if len(_capacities) > 64:
            del _capacities[0]
    return best


def _sempty(n: int, *tail, dtype=None, device=None) -> torch.Tensor:
    cap = _sticky_capacity(n)
    t = torch.empty((cap,) + tuple(tail), dtype=dtype, device=device)
    return t if cap == n else t[:n]


_param_epoch = 0


def note_parameter_gradient():
    """Called by the backward of every op that produces a parameter gradient: an optimiser step is about to follow, and
    some optimisers (torch's fused Adam) update parameters without bumping their autograd version, so derived fp16
    copies made before this point must not be trusted afterwards."""
    global _param_epoch
    _param_epoch += 1


class _F16Cache:
    """fp16 working copy (or packed weight image) of an fp32 master parameter.  The reference re-casts on every forward
    (hash_encoder_half.py:381-385); here the copy is reused until the parameter may have changed: its version counter
    moved, or a backward pass produced parameter gradients since the copy was made (see note_parameter_gradient).
    optim.FusedAdam writes the copy inside its update pass and re-validates it with `adopt`."""

    def __init__(self):
        self.key, self.val, self.epoch = None, None, -1
        self.version_only = False  # set by an optimiser that maintains the copy itself and always bumps the version

    def get(self, p: torch.Tensor, make):
        key = (p.data_ptr(), p._version, p.numel())
        if key != self.key or (self.epoch != _param_epoch and not self.version_only):
            self.val, self.key, self.epoch = make(p), key, _param_epoch
        return self.val

    def adopt(self, p: torch.Tensor):
        """`val` now holds the copy of the current contents of `p` (written by the optimiser)."""
        self.key, self.epoch = (p.data_ptr(), p._version, p.numel()), _param_epoch


class HashGridFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, table, table_f16, levels: GridLevels, four_d: bool, taichi_compat: bool, dy_f16: bool):
        xs = _f32c(x)
        n, xd = xs.shape
        nf = 2 * levels.n_levels
        out = torch.empty(n, nf, dtype=F16, device=xs.device)
        if four_d:
            call("cednerf_hashgrid4d_fwd", ptr(xs), xd, n, ptr(table_f16), ctypes.byref(levels), ptr(out), nf,
                 int(taichi_compat), stream())
        else:
            call("cednerf_hashgrid_fwd", ptr(xs), xd, n, ptr(table_f16), ctypes.byref(levels), ptr(out), nf, stream())
        ctx.save_for_backward(xs, table_f16)
        ctx.levels, ctx.four_d, ctx.compat = levels, four_d, taichi_compat
        ctx.table_shape, ctx.x_shape, ctx.x_dtype = table.shape, x.shape, x.dtype
        return out

    @staticmethod
    def backward(ctx, g):
        note_parameter_gradient()
        xs, table_f16 = ctx.saved_tensors
        n, xd = xs.shape
        nf = 2 * ctx.levels.n_levels
        if g.dtype == F16:
            dy, is16 = g.contiguous(), 1
        else:
            dy, is16 = g.to(F32).contiguous(), 0
        need_t, need_x = ctx.needs_input_grad[1], ctx.needs_input_grad[0] and not ctx.four_d
        g_table = torch.zeros(ctx.table_shape, dtype=F32, device=xs.device) if need_t else None
        g_x = None
        if ctx.four_d:
            if need_t:
                call("cednerf_hashgrid4d_bwd", ptr(xs), xd, n, ctypes.byref(ctx.levels), ptr(dy), nf, is16,
                     ptr(g_table), int(ctx.compat), stream())
        elif need_t or need_x:
            g_x = torch.empty(n, 3, dtype=F32, device=xs.device) if need_x else None
            if need_x and ctx.levels.n_levels not in (8, 16, 32):
                g_x.zero_()
            call("cednerf_hashgrid_bwd", ptr(xs), xd, n, ptr(table_f16), ctypes.byref(ctx.levels), ptr(dy), nf, is16,
                 ptr(g_table), ptr(g_x), stream())
            if g_x is not None and xd != 3:
                g_x = torch.cat([g_x, torch.zeros(n, xd - 3, device=xs.device)], -1)
        return (None if g_x is None else g_x.to(ctx.x_dtype)), g_table, None, None, None, None, None


# ------------------------------------------------------------------------------------------------
# K3 fused MLP
# ------------------------------------------------------------------------------------------------
def pad16(n: int) -> int:
    return (n + 15) // 16 * 16


def mlp_desc(n_in: int, n_out: int, n_neurons: int, n_hidden: int) -> Tuple[MlpDesc, int]:
    if n_neurons != 64:
        raise NotImplementedError("cednerf_b200 fused MLP is 64 neurons wide (all reference networks are)")
    if pad16(n_in) > 64 or pad16(n_out) > 64:
        raise NotImplementedError("fused MLP input/output width is limited to 64 after padding")
    dims = [pad16(n_in)] + [64] * n_hidden + [pad16(n_out)]
    if len(dims) - 1 > _lib.MLP_MAX_LAYERS:
        raise NotImplementedError(f"at most {_lib.MLP_MAX_LAYERS - 1} hidden layers")
    d = MlpDesc()
    d.n_layers = len(dims) - 1
    p_off = i_off = 0
    for l in range(d.n_layers):
        d.dim_in[l], d.dim_out[l], d.param_off[l], d.image_off[l] = dims[l], dims[l + 1], p_off, i_off
        p_off += dims[l] * dims[l + 1]
        i_off += dims[l + 1] * 128
    d.image_bytes = i_off
    return d, p_off


def mlp_pack(params: torch.Tensor, desc: MlpDesc) -> torch.Tensor:
    p = _f32c(params).view(-1)
    image = torch.empty(desc.image_bytes, dtype=U8, device=p.device)
    call("cednerf_mlp_pack_weights", ptr(p), ctypes.byref(desc), ptr(image), stream())
    return image


class MlpFunction(torch.autograd.Function):
    """x [N, n_in] (any float dtype) -> fp16 [N, n_out].

    The operand handed to the kernel is fp16 [N, pad16(n_in)] with the padding columns set to 1.0 (tcnn's
    input padding); d_x is produced in the network precision (fp16), as tcnn's dL_dinput is."""

    _debug = None  # tests / diagnostics: set to a dict to capture the masked hidden gradients of the next backward

    @staticmethod
    def debug_hidden_grads(n, desc, device):
        if MlpFunction._debug is None or desc.n_layers < 2:
            return None
        t = torch.zeros(desc.n_layers - 1, n, 64, dtype=F16, device=device)
        MlpFunction._debug.setdefault("d_hidden", []).append(t)
        return t

    @staticmethod
    def forward(ctx, x, params, image, desc: MlpDesc, save: bool, n_out: int):
        _lib.check_device()
        n, n_in = x.shape
        k0 = desc.dim_in[0]
        if x.dtype == F16 and n_in == k0 and x.is_contiguous():
            x16 = x.detach()
        else:
            x16 = torch.ones(n, k0, dtype=F16, device=x.device)
            x16[:, :n_in] = x.detach()
        L = desc.n_layers
        out = torch.empty(n, desc.dim_out[L - 1], dtype=F16, device=x.device)
        hidden = torch.empty(L - 1, n, 64, dtype=F16, device=x.device) if (save and L > 1) else None
        call("cednerf_mlp_fwd", ptr(x16), ptr(image), ctypes.byref(desc), n, ptr(out), ptr(hidden), stream())
        if save:
            ctx.save_for_backward(x16, hidden if hidden is not None else x16, image)
        ctx.desc, ctx.n_params, ctx.n_in, ctx.n_out = desc, params.numel(), n_in, n_out
        return out[:, :n_out]

    @staticmethod
    def backward(ctx, g):
        note_parameter_gradient()
        x16, hidden, image = ctx.saved_tensors
        desc = ctx.desc
        n = x16.shape[0]
        out_pad = desc.dim_out[desc.n_layers - 1]
        dy = torch.zeros(n, out_pad, dtype=F16, device=x16.device)
        dy[:, : ctx.n_out] = g
        need_x, need_p = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        d_x = torch.empty(n, desc.dim_in[0], dtype=F16, device=x16.device) if need_x else None
        d_p = torch.zeros(ctx.n_params, dtype=F32, device=x16.device) if need_p else None
        if need_x or need_p:
            call("cednerf_mlp_bwd", ptr(x16), ptr(hidden), ptr(dy), ptr(image), ctypes.byref(desc), n, ptr(d_x), 0,
                 ptr(d_p), ptr(MlpFunction.debug_hidden_grads(n, desc, x16.device)), stream())
        return (None if d_x is None else d_x[:, : ctx.n_in]), d_p, None, None, None, None


# ------------------------------------------------------------------------------------------------
# K4 compositing
# ------------------------------------------------------------------------------------------------
def ray_offsets(ray_indices: torch.Tensor, n_rays: int) -> torch.Tensor:
    _lib.check_device()
    r = ray_indices.detach().to(I64).contiguous()
    off = torch.empty(n_rays + 1, dtype=I64, device=r.device)
    call("cednerf_ray_offsets", ptr(r), r.numel(), n_rays, ptr(off), stream())
    return off


def offsets_from_packed(packed_info: torch.Tensor) -> torch.Tensor:
    """nerfacc packed_info [n,2] = (start, count) with contiguous chunks -> offsets [n+1]."""
    starts, cnts = packed_info[:, 0], packed_info[:, 1]
    return torch.cat([starts, (starts[-1:] + cnts[-1:])]).contiguous()


def visibility_mask(t_starts, t_ends, sigmas, offsets, n_rays, early_stop_eps, alpha_thre, want_counts=False):
    """-> keep bool [S] (and, with want_counts, the per-ray number of kept samples int32 [n_rays])."""
    t0, t1, sg = _f32c(t_starts), _f32c(t_ends), _f32c(sigmas)
    keep = _sempty(t0.numel(), dtype=torch.bool, device=t0.device)
    counts = torch.empty(n_rays, dtype=I32, device=t0.device) if want_counts else None
    call("cednerf_visibility_mask", ptr(t0), ptr(t1), ptr(sg), ptr(offsets), t0.numel(), n_rays,
         float(early_stop_eps), float(alpha_thre), ptr(keep), ptr(counts), stream())
    return (keep, counts) if want_counts else keep


def visible_samples(t_starts, t_ends, sigmas, offsets, n_rays, early_stop_eps, alpha_thre):
    """render_visibility_from_density + the compaction of OccGridEstimator.sampling in three launches (mask + per-ray
    counts, scan, ordered scatter) and one host read (the kept total) -> (ray_indices, t_starts, t_ends)."""
    t0, t1 = _f32c(t_starts), _f32c(t_ends)
    keep, counts = visibility_mask(t0, t1, sigmas, offsets, n_rays, early_stop_eps, alpha_thre, want_counts=True)
    starts, _, total = exclusive_scan(counts, want_packed=False)
    n_kept = int(total.item())
    dev = t0.device
    ridx = _sempty(n_kept, dtype=I64, device=dev)
    o0, o1 = _sempty(n_kept, device=dev), _sempty(n_kept, device=dev)
    if n_kept:
        call("cednerf_compact_samples", ptr(keep), ptr(offsets), ptr(starts), ptr(t0), ptr(t1), t0.numel(), n_rays,
             ptr(ridx), ptr(o0), ptr(o1), stream())
    return ridx, o0, o1


def visible_samples_capped(t_starts, t_ends, sigmas, offsets, n_rays, early_stop_eps, alpha_thre, capacity):
    """visible_samples without the host read: outputs of `capacity` rows + (out_offsets [n_rays + 1], totals [2])."""
    t0, t1 = _f32c(t_starts), _f32c(t_ends)
    keep, counts = visibility_mask(t0, t1, sigmas, offsets, n_rays, early_stop_eps, alpha_thre, want_counts=True)
    out_offsets, totals = exclusive_scan_capped(counts, capacity)
    dev = t0.device
    ridx = torch.empty(capacity, dtype=I64, device=dev)
    o0, o1 = torch.empty(capacity, device=dev), torch.empty(capacity, device=dev)
    call("cednerf_compact_samples_capped", ptr(keep), ptr(offsets), ptr(out_offsets), ptr(t0), ptr(t1), int(capacity),
         n_rays, ptr(ridx), ptr(o0), ptr(o1), stream())
    return ridx, o0, o1, out_offsets, totals


class RenderWeightFunction(torch.autograd.Function):
    """(t_starts, t_ends, sigmas) -> (weights, trans, alphas); gradient flows to sigmas only."""

    @staticmethod
    def forward(ctx, t_starts, t_ends, sigmas, offsets, n_rays, prefix_trans):
        t0, t1, sg = _f32c(t_starts), _f32c(t_ends), _f32c(sigmas)
        pf = None if prefix_trans is None else _f32c(prefix_trans)
        s = t0.numel()
        w, tr, al = (_sempty(s, device=t0.device) for _ in range(3))
        call("cednerf_composite_fwd", ptr(t0), ptr(t1), ptr(sg), None, ptr(pf), ptr(offsets), None, 0, s, n_rays,
             ptr(w), ptr(tr), ptr(al), None, None, None, None, 0, 0.0, stream())
        ctx.save_for_backward(t0, t1, tr, al, offsets)
        ctx.n_rays = n_rays
        ctx.set_materialize_grads(False)
        return w, tr, al

    @staticmethod
    def backward(ctx, gw, gt, ga):
        t0, t1, tr, al, offsets = ctx.saved_tensors
        s = t0.numel()
        gs = _sempty(s, device=t0.device)
        gw, gt, ga = (None if g is None else _f32c(g) for g in (gw, gt, ga))
        call("cednerf_composite_bwd", ptr(t0), ptr(t1), None, ptr(tr), ptr(al), ptr(offsets), None, 0, s, ctx.n_rays,
             None, None, None, None, None, ptr(gw), ptr(gt), ptr(ga), ptr(gs), None, 0.0, stream())
        return None, None, gs, None, None, None


class AccumulateFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, weights, values, ray_indices, offsets, n_rays, n_dev=None):
        w = _f32c(weights)
        v = None if values is None else _f32c(values)
        c = 1 if v is None else v.shape[-1]
        out = torch.empty(n_rays, c, device=w.device)
        call("cednerf_accumulate_fwd", ptr(w), ptr(v), c, ptr(offsets), w.numel(), n_rays, ptr(out), 0, stream())
        ctx.save_for_backward(w, v if v is not None else w, ray_indices)
        ctx.has_v, ctx.c, ctx.n_dev = v is not None, c, n_dev
        ctx.set_materialize_grads(False)
        return out

    @staticmethod
    def backward(ctx, g):
        if g is None:
            return None, None, None, None, None, None
        w, v, ridx = ctx.saved_tensors
        v = v if ctx.has_v else None
        g = _f32c(g)
        gw = _sempty(w.numel(), device=w.device) if ctx.needs_input_grad[0] else None
        gv = _sempty(v.shape[0], v.shape[1], device=v.device) if (ctx.has_v and ctx.needs_input_grad[1]) else None
        if gw is not None or gv is not None:
            call("cednerf_accumulate_bwd", ptr(w), ptr(v), ctx.c, ptr(ridx), w.numel(), ptr(g), ptr(gw), ptr(gv),
                 ptr(ctx.n_dev), stream())
        return gw, gv, None, None, None, None


def accumulate_inplace(weights, values, offsets, outputs):
    w = _f32c(weights)
    v = None if values is None else _f32c(values)
    c = 1 if v is None else v.shape[-1]
    assert outputs.is_contiguous() and outputs.dtype == F32 and outputs.shape[-1] == c
    call("cednerf_accumulate_fwd", ptr(w), ptr(v), c, ptr(offsets), w.numel(), outputs.shape[0], ptr(outputs), 1,
         stream())


def composite_round_(t_starts, t_ends, sigmas, rgbs, offsets, rgb, opacity, depth):
    """One marching round of render_image_test in one launch: weights with prefix transmittance 1 - opacity[ray], then
    rgb / opacity / depth accumulated in place (cednerf/utils.py:274-299)."""
    t0, t1, sg, c = _f32c(t_starts), _f32c(t_ends), _f32c(sigmas), _f32c(rgbs)
    assert rgb.is_contiguous() and opacity.is_contiguous() and depth.is_contiguous()
    call("cednerf_composite_fwd", ptr(t0), ptr(t1), ptr(sg), ptr(c), None, ptr(offsets), None, 0, t0.numel(), rgb.shape[0],
         None, None, None, ptr(rgb), ptr(opacity), ptr(depth), None, 2, 0.0, stream())


class CompositeFunction(torch.autograd.Function):
    """Fused rendering(): (sigmas, rgbs) -> (colors, opacity, depth, weights, trans, alphas).

    cednerf/render.py:81-87 + :158-174 in one launch; backward is one launch as well."""

    @staticmethod
    def forward(ctx, t_starts, t_ends, sigmas, rgbs, offsets, n_rays, bkgd):
        t0, t1, sg, rgb = _f32c(t_starts), _f32c(t_ends), _f32c(sigmas), _f32c(rgbs)
        s, dev = t0.numel(), t0.device
        bk, stride = None, 0
        if bkgd is not None:
            bk = _f32c(bkgd)
            stride = 3 if bk.numel() == 3 * n_rays and bk.dim() == 2 and n_rays > 1 else 0
        w, tr, al = (_sempty(s, device=dev) for _ in range(3))
        colors = torch.empty(n_rays, 3, device=dev)
        opac, depth, draw = (torch.empty(n_rays, 1, device=dev) for _ in range(3))
        eps = float(torch.finfo(torch.float32).eps)
        call("cednerf_composite_fwd", ptr(t0), ptr(t1), ptr(sg), ptr(rgb), None, ptr(offsets), ptr(bk), stride, s,
             n_rays, ptr(w), ptr(tr), ptr(al), ptr(colors), ptr(opac), ptr(depth), ptr(draw), 0, eps, stream())
        ctx.save_for_backward(t0, t1, rgb, tr, al, offsets, opac, draw, bk if bk is not None else t0)
        ctx.has_bk, ctx.stride, ctx.n_rays, ctx.eps = bk is not None, stride, n_rays, eps
        ctx.set_materialize_grads(False)  # unused outputs (weights / trans / alphas ...) arrive as None, not as zero fills
        return colors, opac, depth, w, tr, al

    @staticmethod
    def backward(ctx, gc, go, gd, gw, gt, ga):
        t0, t1, rgb, tr, al, offsets, opac, draw, bk = ctx.saved_tensors
        bk = bk if ctx.has_bk else None
        s = t0.numel()
        gs = _sempty(s, device=t0.device)
        grgb = _sempty(s, 3, device=t0.device) if ctx.needs_input_grad[3] else None
        gc, go, gd, gw, gt, ga = (None if g is None else _f32c(g) for g in (gc, go, gd, gw, gt, ga))
        call("cednerf_composite_bwd", ptr(t0), ptr(t1), ptr(rgb), ptr(tr), ptr(al), ptr(offsets), ptr(bk), ctx.stride,
             s, ctx.n_rays, ptr(opac), ptr(draw), ptr(gc), ptr(go), ptr(gd), ptr(gw), ptr(gt), ptr(ga), ptr(gs),
             ptr(grgb), ctx.eps, stream())
        return None, None, gs, grgb, None, None, None


# ------------------------------------------------------------------------------------------------
# parameter-free encodings
# ------------------------------------------------------------------------------------------------
class FrequencyFunction(torch.autograd.Function):
    """x f32 [N,D] -> fp16 [N, pad16(D*2*n)], padding columns = 1.0 (tcnn MLP-input padding)."""

    @staticmethod
    def forward(ctx, x, n_freq: int, pad_to: int):
        xs = _f32c(x)
        n, d = xs.shape
        width = d * 2 * n_freq
        cols = max(width, pad_to)
        out = torch.empty(n, cols, dtype=F16, device=xs.device)
        call("cednerf_frequency_fwd", ptr(xs), d, n, n_freq, ptr(out), cols, pad_to, 1.0, stream())
        ctx.save_for_backward(xs)
        ctx.n_freq, ctx.x_dtype = n_freq, x.dtype
        return out

    @staticmethod
    def backward(ctx, g):
        (xs,) = ctx.saved_tensors
        n, d = xs.shape
        if g.dtype == F16:
            dy, is16 = g.contiguous(), 1
        else:
            dy, is16 = g.to(F32).contiguous(), 0
        dx = torch.empty(n, d, dtype=F32, device=xs.device)
        call("cednerf_frequency_bwd", ptr(xs), d, n, ctx.n_freq, ptr(dy), dy.shape[1], is16, ptr(dx), stream())
        return dx.to(ctx.x_dtype), None, None


def sh2_encode(d01: torch.Tensor) -> torch.Tensor:
    x = _f32c(d01)
    out = torch.empty(x.shape[0], 4, dtype=F16, device=x.device)
    call("cednerf_sh2_fwd", ptr(x), x.shape[0], ptr(out), 4, stream())
    return out


def time_embed(t: torch.Tensor, move_norm: Optional[torch.Tensor] = None) -> torch.Tensor:
    tt = _f32c(t).view(-1)
    mv = None if move_norm is None else _f32c(move_norm).view(-1)
    out = torch.empty(tt.numel(), 9, device=tt.device)
    call("cednerf_time_embed", ptr(tt), ptr(mv), tt.numel(), ptr(out), stream())
    return out


# ------------------------------------------------------------------------------------------------
# fused field query (inference: density pre-pass of the sampler, occupancy updates, eval rendering)
# ------------------------------------------------------------------------------------------------
def field_fwd(desc: FieldDesc, images, table_f16, n: int, sigma_only: bool, packed=None, points=None,
              timestamps=None, t_stride: int = 1, n_dev: Optional[torch.Tensor] = None):
    """packed = (ray_indices, t_starts, t_ends, rays_o, rays_d) or points = (x, dirs-or-None).
    -> (sigma [n], rgb [n,3] or None).  n_dev (int64 [1] on the device): only the first min(n, n_dev) entries are live
    (computed and written); n is then the capacity of the buffers and no host read of the count is needed."""
    _lib.check_device()
    dev = table_f16.device
    sigma = _sempty(n, device=dev)
    rgb = None if sigma_only else _sempty(n, 3, device=dev)
    ts = _f32c(timestamps).view(-1)
    if packed is not None:
        ridx, t0, t1, o, d = packed
        # converted copies are bound to locals so that they outlive the launch (a temporary freed right after its ptr()
        # would hand its block to the next conversion: two arguments aliasing one buffer)
        ridx_c, t0_c, t1_c, o_c, d_c = ridx.detach().to(I64).contiguous(), _f32c(t0), _f32c(t1), _f32c(o), _f32c(d)
        args = (ptr(ridx_c), ptr(t0_c), ptr(t1_c), ptr(o_c), ptr(d_c), None, None)
    else:
        x, dirs = points
        xs = _f32c(x)
        ds = None if dirs is None else _f32c(dirs)
        args = (None, None, None, None, None, ptr(xs), ptr(ds))
    call("cednerf_field_fwd", *args, ptr(ts), int(t_stride), n, ptr(images[0]), ptr(images[1]), ptr(images[2]),
         ptr(table_f16), ctypes.byref(desc), ptr(sigma), ptr(rgb), ptr(n_dev), stream())
    del args  # (ridx_c ... d_c / xs, ds stay referenced by this frame until here: the launch is enqueued)
    return sigma, rgb


_table_grad_hook = None

def set_table_grad_hook(fn):
    """fn(g_table) is called from the fused training backward as soon as the hash-table gradient is complete, before
    the encoding's dL/dx and the deformation-net backward are launched (dp.GradAllReducer starts its all-reduce there).
    None removes the hook."""
    global _table_grad_hook
    _table_grad_hook = fn


_table_grad_alloc = None


def set_table_grad_alloc(fn):
    """fn(shape, device) -> zero-filled fp32 tensor (or None) that the fused training backward accumulates the hash-table
    gradient into.  dp.DistributedFusedAdam hands out its peer-visible buffer here, so that the other ranks read this
    rank's gradient where the kernel wrote it.  None removes the hook."""
    global _table_grad_alloc
    _table_grad_alloc = fn


class FieldTrainFunction(torch.autograd.Function):
    """Training-mode DNGPradianceField.forward on packed ray samples: one forward launch, backward = one tensor-core
    launch per network + the hash-grid backward.  Returns (sigma [n], rgb [n,3], latent [n,32] | None, selector, move)."""

    @staticmethod
    def forward(ctx, p1, p2, p3, p4, table, desc, images, table_f16, ridx, t0, t1, rays_o, rays_d, ts, t_stride,
                want_latent, n_dev=None):
        _lib.check_device()
        lib = _lib.load()
        n, dev = t0.numel(), t0.device
        ridx = ridx.detach().to(I64).contiguous()
        t0, t1, rays_o, rays_d = _f32c(t0), _f32c(t1), _f32c(rays_o), _f32c(rays_d)
        ts = _f32c(ts).view(-1)
        sigma = _sempty(n, device=dev)
        rgb = _sempty(n, 3, device=dev)
        latent = _sempty(n, 32, device=dev) if want_latent else None
        selector = _sempty(n, dtype=torch.bool, device=dev)
        move = _sempty(n, 3, device=dev)
        # capacity in steps of 32 Ki samples: the visible-sample count changes a little every step, and a 1 GB buffer that
        # grows by a few KB would make the caching allocator cudaMalloc (and sometimes free + retry) in the hot loop
        saved = torch.empty(max(int(lib.cednerf_field_saved_bytes(ctypes.byref(desc), _sticky_capacity(n))), 16), dtype=U8, device=dev)
        call("cednerf_field_train_fwd", ptr(ridx), ptr(t0), ptr(t1), ptr(rays_o), ptr(rays_d), ptr(ts), int(t_stride), n,
             ptr(images[0]), ptr(images[1]), ptr(images[2]), ptr(images[3]), ptr(table_f16), ctypes.byref(desc),
             ptr(sigma), ptr(rgb), ptr(latent), ptr(selector), ptr(move), ptr(saved), ptr(n_dev), stream())
        ctx.save_for_backward(ridx, t0, t1, rays_o, rays_d, ts, sigma, rgb, selector, saved, table_f16, images[0],
                              images[1], images[2], images[3] if images[3] is not None else images[0])
        ctx.desc, ctx.t_stride, ctx.has4 = desc, int(t_stride), images[3] is not None and want_latent
        ctx.n_dev = n_dev
        ctx.shapes = (p1.shape, p2.shape, p3.shape, None if p4 is None else p4.shape, table.shape)
        ctx.mark_non_differentiable(selector, move)
        ctx.set_materialize_grads(False)
        if latent is None:
            latent = torch.zeros(0, device=dev)
        return sigma, rgb, latent, selector, move

    @staticmethod
    def backward(ctx, d_sigma, d_rgb, d_latent, _sel, _mv):
        note_parameter_gradient()
        ridx, t0, t1, rays_o, rays_d, ts, sigma, rgb, selector, saved, table_f16, i1, i2, i3, i4 = ctx.saved_tensors
        lib = _lib.load()
        n, dev = t0.numel(), t0.device
        s1, s2, s3, s4, st = ctx.shapes
        # the MLP weight gradients share one zero-filled buffer (one fill launch instead of four)
        want4 = ctx.has4 and s4 is not None
        sizes = [math.prod(s) for s in (s1, s2, s3)] + ([math.prod(s4)] if want4 else [])
        padded = [(k + 3) // 4 * 4 for k in sizes]  # 16-byte aligned slices
        pool = torch.zeros(sum(padded), dtype=F32, device=dev)
        views, o = [], 0
        for k, kp, shp in zip(sizes, padded, (s1, s2, s3) + ((s4,) if want4 else ())):
            views.append(pool[o:o + k].view(shp))
            o += kp
        g1, g2, g3 = views[:3]
        g4 = views[3] if want4 else None
        gt = _table_grad_alloc(st, dev) if _table_grad_alloc is not None else None
        if gt is None:
            gt = torch.zeros(st, dtype=F32, device=dev)
        d_sigma = torch.zeros(n, device=dev) if d_sigma is None else _f32c(d_sigma)
        d_rgb = torch.zeros(n, 3, device=dev) if d_rgb is None else _f32c(d_rgb)
        dl = None
        if ctx.has4 and d_latent is not None and d_latent.numel():
            dl = _f32c(d_latent)
        work = torch.empty(max(int(lib.cednerf_field_bwd_workspace_bytes(ctypes.byref(ctx.desc), _sticky_capacity(n))), 16), dtype=U8,
                           device=dev)
        hook = _table_grad_hook
        for phase in ((1, 2) if hook is not None else (0,)):
            if n:
                call("cednerf_field_train_bwd", ptr(ridx), ptr(t0), ptr(t1), ptr(rays_o), ptr(rays_d), ptr(ts),
                     ctx.t_stride, n, ptr(i1), ptr(i2), ptr(i3), ptr(i4) if ctx.has4 else None, ptr(table_f16),
                     ctypes.byref(ctx.desc), ptr(sigma), ptr(rgb), ptr(selector), ptr(saved), ptr(d_sigma), ptr(d_rgb),
                     ptr(dl), ptr(work), ptr(g1), ptr(g2), ptr(g3), ptr(g4) if dl is not None else None, ptr(gt), phase,
                     ptr(ctx.n_dev), stream())
            if phase == 1:
                hook(gt)  # the 191 MB table gradient is complete: its all-reduce overlaps the rest of the backward
        return (g1, g2, g3, g4 if dl is not None else None, gt) + (None,) * 12
