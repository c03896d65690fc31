#!/usr/bin/env python
"""Benchmark of the per-ray rendering hot path on the configurations BASELINE.json names.

    python bench.py --gpus N --steps K --warmup W             # this repo's CUDA path (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...   # the CPU restatement of the reference path (oracle/)
    python bench.py --config {dynerf,hypernerf,dnerf} ...     # which configuration is the headline (default dynerf)

Headline (configs[1]): DyNeRF flame_salmon_1-shaped TRAIN STEP, 2^18 rays per GPU.  One step = the body of the
reference's training loop for this path (train_real.py:330-420 without the data loader): estimator.update_every_n_steps
(works every 16th step; on a twin estimator, see OccupancyUpdate), stratified occupancy-grid sampling with the no-grad
density pre-pass and visibility filtering, the field forward on the surviving samples, compositing, the MSE + auxiliary
losses of the canonical flags (-te -ta -df -f -wr -ae), backward, GradScaler (2^10) and fused Adam at the reference
schedule's first-iteration learning rate (see TrainState).  With N > 1 every rank runs the step on its own 2^18 rays
(weak scaling) and the optimiser step is dp.DistributedFusedAdam (fused reduce-scatter + Adam + all-gather over NVLink
peer memory; `--dp nccl` selects the all-reduce path of round 1).

Besides the headline the default run measures, and reports under `configs` / `render` at the END of the JSON line:
  configs[3]  `render`            the 300-pose novel-view video of the DyNeRF-shaped scene (datasets/utils.py:67-112 spiral,
                                  t = i/300), frames interleaved over the ranks, no collective (strong scaling);
  configs[0]  `configs.dnerf`     D-NeRF-shaped 800x800 frames (t = 0.5) through render_image_test;
  configs[2]  `configs.hypernerf` HyperNeRF-shaped train step (536x960 camera, one timestamp per batch);
  configs[4]  `configs.dynerf_2p20` (N > 1 only) the DyNeRF train step with 2^20 rays split over the N ranks.
The reference arm runs the headline configuration on the CPU restatement (oracle/) from the same initial weights, the
same learning rate and the same loss scaling, on a bounded ray sample, without the occupancy update (8.4 M CPU field
queries per update would only flatter the ratio).
Rank 0 prints ONE JSON line.  Synthetic data: seeded rays / pixels / occupancy, random-init weights with a density
boost (cednerf_b200/workload.py)."""
from __future__ import annotations

import argparse
import importlib.util
import json
import os

# Sample-sized buffers change size a little every step (the visible-sample count follows the field, and the named
# configuration sits right at 2^20 samples - a size-class boundary of any power-of-two rounding).  The library allocates
# them at sticky capacities (ops._sempty), so the caching allocator sees the same request sizes step after step; 1/8
# power-of-two rounding keeps the few remaining torch-side temporaries in one class.
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "roundup_power2_divisions:8")
import statistics
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="dynerf", choices=["dynerf", "hypernerf", "dnerf"])
    ap.add_argument("--rays", type=int, default=2 ** 18, help="rays per rank per step (train configurations)")
    ap.add_argument("--cpu-rays", type=int, default=4096, help="rays per step of the bounded CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-steps", type=int, default=3, help="instrumented steps for the per-kernel breakdown")
    ap.add_argument("--render-frames", type=int, default=300,
                    help="frames of the video leg in total (subsampled from the 300-pose spiral; 0 = skip)")
    ap.add_argument("--render-streams", type=int, default=3,
                    help="frames of the video / frame legs whose marching rounds are interleaved on separate streams")
    ap.add_argument("--headline-only", action="store_true", help="skip the other configurations")
    ap.add_argument("--host-counts", action="store_true",
                    help="read the sample totals back to the host inside the step (the reference's behaviour) instead "
                         "of the capacity mode that keeps them on the device")
    ap.add_argument("--dp", default="peer", choices=["peer", "nccl"], help="multi-GPU optimiser step")
    ap.add_argument("--dp-transport", default="auto", choices=["auto", "nvls", "p2p"],
                    help="peer-memory DP: reduce / broadcast inside the NVSwitch (multimem) or by peer loads / stores")
    ap.add_argument("--torch-profile", default="", help="write a torch.profiler kernel table of one step to this file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step of the headline computed to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def load_workload():
    """cednerf_b200/workload.py by path: it needs torch only, and the reference arm must not load the product."""
    spec = importlib.util.spec_from_file_location("cednerf_workload", os.path.join(ROOT, "cednerf_b200", "workload.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["cednerf_workload"] = mod
    spec.loader.exec_module(mod)
    return mod


# --------------------------------------------------------------------------------------------------------------
# the step (shared by both arms: `impl` is cednerf_b200 or the oracle namespace below)
# --------------------------------------------------------------------------------------------------------------
def aux_losses(rgb, acc, pixels, extra, flags):
    """train_real.py:369-409 for the canonical DyNeRF flags (-ae, -wr, -f)."""
    loss = 0.0
    t_last = (1 - acc).clamp(1e-6, 1 - 1e-6)
    loss = loss + (-(t_last * torch.log(t_last) + (1 - t_last) * torch.log(1 - t_last)).mean()) * 1e-3
    for ex in extra:
        rgbper = (ex["rgbs"] - pixels[ex["ray_indices"]]).pow(2).sum(dim=-1)
        loss = loss + (rgbper * ex["weights"].detach()).sum() / pixels.shape[0] * 1e-3
        if flags.get("use_feat_predict"):
            loss = loss + ex["latent_losses"].mean()
    return loss


def make_scheduler(opt, max_steps=20000):
    """train_real.py:276-287: linear warm-up from 0.01 x lr over 100 iterations, then step decay."""
    return torch.optim.lr_scheduler.ChainedScheduler([
        torch.optim.lr_scheduler.LinearLR(opt, start_factor=0.01, total_iters=100),
        torch.optim.lr_scheduler.MultiStepLR(opt, milestones=[max_steps // 2, max_steps * 3 // 4, max_steps * 9 // 10],
                                             gamma=0.33)])


class TrainState:
    """Parameters at iteration 0, so that every timed leg measures the same iterations of training on the same field.
    The learning rate is held at the reference schedule's FIRST-iteration value (LinearLR start_factor 0.01 -> 1e-4):
    random-init weights fitted to random pixels move the density by e-folds within tens of Adam steps at the full rate,
    and the visible-sample count (the work per step) would then be whatever the step count made it - 1.0 M samples at
    step 0, 1.4 M fifteen steps later - instead of the named configuration's 2^20 per 2^18 rays.  Every kernel of the
    step, the optimiser included, does the same work at any learning rate."""

    def __init__(self, field, opt):
        self.field, self.opt = field, opt
        self.params = [p.detach().clone() for p in field.parameters()]
        self.sched = None
        self.restore()

    def restore(self):
        with torch.no_grad():
            for p, q in zip(self.field.parameters(), self.params):
                p.copy_(q)
        self.opt.state.clear()
        if hasattr(self.opt, "_step_t"):
            self.opt._step_t = None
        for g in self.opt.param_groups:
            g["lr"] = g.get("initial_lr", g["lr"])
        make_scheduler(self.opt)  # sets lr to 0.01 x initial_lr (iteration 0 of the reference schedule); never stepped


class OccupancyUpdate:
    """estimator.update_every_n_steps(step, occ_eval_fn, occ_thre) of the reference loop (train_real.py:324-336): every
    16th iteration the field is queried at one jittered point per grid cell (all L x 128^3 cells during the first 256
    iterations) with random timestamps.  It runs on a TWIN of the estimator: the synthetic occupancy is what defines the
    workload (a random field would otherwise mark everything occupied), so the marcher keeps reading the original.
    All draws come from dp.SharedRng, seeded alike on every rank: the replicas stay identical without a collective."""

    def __init__(self, impl, cfg, est, field, step_size, rng):
        self.twin = impl.OccGridEstimator(list(cfg.roi_aabb), resolution=cfg.occ_res, levels=cfg.occ_levels)
        self.twin = self.twin.to(est.aabbs.device)
        self.twin.binaries, self.twin.occs = est.binaries.clone(), est.occs.clone()
        self.twin.train()
        self.field, self.step_size, self.step, self.updates, self.rng = field, step_size, 0, 0, rng
        # the closure of train_real.py:324-328 as an object: called like a function it computes the same thing, and it
        # lets this repo's estimator run each level of the update as one fused launch
        self.occ_eval_fn = impl.utils.FieldOccEval(field, step_size, rng=rng)

    def __call__(self):
        if self.step % 16 == 0:
            self.updates += 1
        self.twin.update_every_n_steps(step=self.step, occ_eval_fn=self.occ_eval_fn, occ_thre=1e-2, rng=self.rng)
        self.step += 1


def train_step(impl, field, est, opt, scaler, batch, cfg, rk, reducer=None, sched=None, occ=None, device_counts=False,
               keep=None):
    """`keep`: a dict that receives this step's rendered rays and loss (for --dump-outputs)."""
    if occ is not None:
        occ()
    rays = impl.Rays(batch["origins"], batch["viewdirs"])
    extra_kw = {"device_counts": True} if device_counts else {}   # this repo only: no host read inside the step
    rgb, acc, depth, n_samples, extra = impl.render_image(field, est, rays, render_bkgd=batch["color_bkgd"],
                                                          timestamps=batch["timestamps"], jitter=batch["jitter"], **rk,
                                                          **extra_kw)
    if keep is not None:
        keep.update(rgb=rgb, acc=acc, depth=depth, n_samples=n_samples)
    if not torch.is_tensor(n_samples) and n_samples == 0:
        return None, 0
    if hasattr(impl, "losses"):  # this repo: the same loss as one fused forward / backward launch
        loss = impl.losses.training_loss(rgb, acc, batch["pixels"], extra, acc_entropy_loss=True, weight_rgbper=True,
                                         use_feat_predict=bool(cfg.flags.get("use_feat_predict")),
                                         distortion_loss=cfg.name.startswith("hypernerf"))   # run_hyper.sh: -d
    else:
        loss = torch.nn.functional.mse_loss(rgb, batch["pixels"]) + aux_losses(rgb, acc, batch["pixels"], extra, cfg.flags)
    if keep is not None:
        keep["loss"] = loss
    opt.zero_grad()
    if scaler is not None:
        scaler.scale(loss).backward()
        if reducer is not None:
            reducer.wait()
        scaler.step(opt)
        scaler.update()
    else:  # CPU arm: the GradScaler(2^10) protocol spelled out (scale, unscale, step)
        (loss * 1024.0).backward()
        for p in field.parameters():
            if p.grad is not None:
                p.grad.div_(1024.0)
        opt.step()
    if sched is not None:
        sched.step()
    return loss, n_samples


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index, self.sm, self.reasons, self.max_mhz, self.run, self.th = index, [], set(), None, False, None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001 - NVML missing: report it, do not fail the benchmark
            return
        names = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        self.run = True

        def loop():
            while self.run:
                try:
                    self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                    mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                    for k, bit in names.items():
                        if mask & bit:
                            self.reasons.add(k)
                except Exception:  # noqa: BLE001
                    pass
                time.sleep(0.02)

        self.th = threading.Thread(target=loop, daemon=True)
        self.th.start()

    def stop(self):
        self.run = False
        if self.th is not None:
            self.th.join(timeout=1.0)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"], "samples": 0}
        return {"sm_mhz": statistics.median(self.sm), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


# algorithmic bytes per launch of each entry point (SURVEY.md §8d per-unit figures x units of the launch)
def algorithmic_bytes(name, args, live=None):
    live = live or {}
    if name == "cednerf_hashgrid_fwd":
        n, L = args[2], args[4]._obj.n_levels
        return n * (L * 8 * 4 + 12 + L * 4)                     # 512 B table + 12 B xyz + 64 B features (L = 16)
    if name == "cednerf_hashgrid_bwd":
        n, L, is16 = args[2], args[4]._obj.n_levels, args[7]
        b = n * (2 * L * (2 if is16 else 4) + 12)               # dy + xyz
        if args[8]:
            b += n * L * 8 * 8                                  # fp32 table-gradient RMW, counted once (1024 B)
        if args[9]:
            b += n * (L * 8 * 4 + 12)                           # table re-read for dL/dx + dx write
        return b
    if name == "cednerf_field_fwd":
        n, L = args[9], args[14]._obj.levels.n_levels
        if args[17] and live.get("marched"):                     # capacity-sized launch: the live count is what moves
            n = min(n, live["marched"])
        return n * (L * 8 * 4 + 16 + 4 + (12 if args[16] else 0))  # 512 B table + packed sample 16 B + sigma (+ rgb)
    if name == "cednerf_field_train_fwd":                       # 512 B table + 16 B sample + sigma / rgb / selector / move
        n, L = args[7], args[13]._obj.levels.n_levels
        if args[-2] and live.get("visible"):
            n = min(n, live["visible"])
        return n * (L * 8 * 4 + 16 + 4 + 12 + 1 + 12)
    if name == "cednerf_field_train_bwd":                       # 1024 B table-gradient RMW + 512 B table re-read + d_sigma / d_rgb
        n, L = args[7], args[13]._obj.levels.n_levels
        if args[-2] and live.get("visible"):
            n = min(n, live["visible"])
        return n * (L * 8 * 8 + L * 8 * 4 + 16 + 16)
    if name == "cednerf_mlp_fwd":
        d, n = args[2]._obj, args[3]
        hid = (d.n_layers - 1) * 128 if args[5] else 0
        return n * (d.dim_in[0] * 2 + d.dim_out[d.n_layers - 1] * 2 + hid)
    if name == "cednerf_mlp_bwd":
        d, n = args[4]._obj, args[5]
        return n * (d.dim_in[0] * 2 + (d.n_layers - 1) * 128 + d.dim_out[d.n_layers - 1] * 2 +
                    (d.dim_in[0] * (4 if args[7] else 2) if args[6] else 0))
    if name == "cednerf_march":
        n = args[3]
        return n * 52                                           # 32 B/ray in + 20 B/ray out (per-sample writes: the fill)
    if name == "cednerf_march_fill_runs":
        return None
    if name == "cednerf_composite_fwd":
        return min(args[8], live.get("visible") or args[8]) * 44 + args[9] * 20
    if name == "cednerf_composite_bwd":
        return min(args[8], live.get("visible") or args[8]) * 60 + args[9] * 20
    if name == "cednerf_adam_step":                             # 16 B read + 12 B written (+ 2 B fp16 copy) per parameter
        t = args[0]._obj
        return sum(t.n[k] * (30 if t.p16[k] else 28) for k in range(t.n_tensors))
    if name == "cednerf_dp_adam":                               # N gradient reads + 12 B state in + 8 B state out + 6 N B replicas
        a = args[0]._obj
        return (a.hi - a.lo) * (4 * a.world + 20 + 6 * a.n_out)
    if name == "cednerf_nonfinite_check":
        t = args[0]._obj
        return sum(t.n[k] * 4 for k in range(t.n_tensors))
    return None


class Instrument:
    """CUDA events around every entry point of the library (same stream), for per-kernel shares and rooflines."""

    def __init__(self, cb, _lib):
        self.mods = (_lib, cb.ops, cb.optim, cb.losses)
        self.real, self.rec = _lib.call, []

    def __enter__(self):
        def recording_call(name, *a):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            self.real(name, *a)
            e.record()
            self.rec.append((name, a, s, e))

        for m in self.mods:
            m.call = recording_call
        return self

    def __exit__(self, *exc):
        for m in self.mods:
            m.call = self.real

    def aggregate(self, live=None):
        agg = {}
        for name, a, s, e in self.rec:
            by = algorithmic_bytes(name, a, live)
            d = agg.setdefault(name, {"ms": 0.0, "launches": 0, "bytes": 0, "has_bytes": by is not None})
            d["ms"] += s.elapsed_time(e)
            d["launches"] += 1
            d["bytes"] += by or 0
        return agg


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured"
    except (OSError, ValueError, KeyError):
        return 6650.0, "fallback"


# entry points that are several kernels behind one call (their time is a sum, not a kernel's duration)
MULTI_KERNEL_ENTRIES = {"cednerf_field_train_bwd"}


def roofline_of(agg, n_iter, total_ms):
    """Dominant kernel (by time, among those with algorithmic bytes) against the HBM copy peak; plus the whole step."""
    hbm_peak, src = peaks()
    # the dominant KERNEL: entry points that are one launch (cednerf_field_train_bwd is seven kernels behind one call, its
    # sum is not a kernel's duration)
    single = [n for n in agg if agg[n]["has_bytes"] and n not in MULTI_KERNEL_ENTRIES]
    top = max(single or [n for n in agg if agg[n]["has_bytes"]], key=lambda n: agg[n]["ms"])
    d = agg[top]
    achieved = d["bytes"] / (d["ms"] * 1e-3) / 1e9
    traffic = None  # dram__bytes_read + dram__bytes_write per launch of that kernel, from the committed ncu capture
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json"))).get(top, {}).get("bytes_per_launch")
    except (OSError, ValueError):
        pass
    step_bytes = sum(v["bytes"] for v in agg.values()) / n_iter
    return {"kernel": top, "bound": "hbm", "achieved": round(achieved, 1), "peak": hbm_peak, "unit": "GB/s",
            "frac": round(achieved / hbm_peak, 4), "traffic": traffic, "peak_source": src,
            "avg_launch_ms": round(d["ms"] / d["launches"], 4), "bytes_per_launch": d["bytes"] // d["launches"],
            "share_of_step": round(d["ms"] / n_iter / total_ms, 3),
            "step_bytes": int(step_bytes), "step_frac": round(step_bytes / (total_ms * 1e-3) / 1e9 / hbm_peak, 4),
            "limiter": ("the 96 MB fp16 table is L2-resident (DRAM 2 %): the kernel is paced by instruction issue and the L1 "
                        "tag stage of its divergent gathers, so the HBM fraction is a lower bound on how well it uses what "
                        "binds it (profiles/r2o_field_fwd_phase_experiments.md)") if top == "cednerf_field_fwd" else None}


class Dist:
    def __init__(self):
        import torch.distributed as dist

        self.dist = dist
        self.rank = int(os.environ.get("RANK", 0))
        self.local_rank = int(os.environ.get("LOCAL_RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py (impl=ours) needs a CUDA device: the product has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()


PARAM_SAMPLE = 2 ** 20        # --dump-outputs: entries kept of a larger parameter tensor
DUMP_LIMIT = 64 * 2 ** 20     # --dump-outputs: bytes in all


def host_outputs(keep, field=None):
    """--dump-outputs: the tensors a caller received from the last timed step, as float32 / float64 host arrays.  A train
    step also hands back the updated parameters: each whole, or its entries at a fixed seeded sample of PARAM_SAMPLE
    positions."""
    out = {}
    for k, v in keep.items():
        v = torch.as_tensor(v).detach()
        out[k] = (v.float() if v.is_floating_point() else v.double()).cpu().numpy()
    for k, p in (field.named_parameters() if field is not None else ()):
        v = p.detach().flatten()
        if v.numel() == 0:   # parameter-free modules (the spherical-harmonics direction encoding) have nothing to compare
            continue
        if v.numel() > PARAM_SAMPLE:
            idx = torch.randint(v.numel(), (PARAM_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            v = v[idx.to(v.device)]
        out["param." + k] = v.float().cpu().numpy()
    return out


def write_outputs(dirname, arrays):
    import numpy as np

    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(dirname, k + ".npy"), a)


# --------------------------------------------------------------------------------------------------------------
# train-step leg
# --------------------------------------------------------------------------------------------------------------
def train_leg(D, cb, workload, cfg, args, n_rays, steps, warmup, full: bool):
    """-> dict.  `full`: also the end-to-end (host batches) leg, the per-kernel breakdown and the clock samples."""
    from cednerf_b200 import _lib, dp

    dev, world, rank = D.dev, D.world, D.rank
    rk = workload.render_kwargs(cfg)
    est, field = workload.build_scene(cfg, dev, cb, seed=42)
    est.train(), field.train()
    scaler = cb.optim.GradScaler(2 ** 10)                              # torch.cuda.amp.GradScaler(2**10), train_real.py:252
    reducer, dp_mode = None, "single"
    if world > 1 and args.dp == "peer":
        opt = dp.DistributedFusedAdam(field.parameters(), lr=1e-2, eps=1e-15)
        ok = torch.ones(1, device=dev)
        try:
            opt.setup()
        except Exception as e:  # noqa: BLE001 - no peer access / IPC on this box: fall back, and say so
            print(f"[bench] rank {rank}: peer-memory setup failed ({e}); using the NCCL all-reduce path", file=sys.stderr)
            ok.zero_()
        D.dist.all_reduce(ok, op=D.dist.ReduceOp.MIN)
        dp_mode = "peer" if float(ok.item()) == 1.0 else "nccl"
        if dp_mode == "peer" and args.dp_transport != "auto":
            opt.nvls = args.dp_transport == "nvls"
    if world > 1 and dp_mode != "peer":
        dp_mode = "nccl"
        opt = cb.optim.FusedAdam(field.parameters(), lr=1e-2, eps=1e-15)
        reducer = dp.GradAllReducer(field.parameters(), world)
    if world == 1:
        opt = cb.optim.FusedAdam(field.parameters(), lr=1e-2, eps=1e-15)  # apex.optimizers.FusedAdam, train_real.py:267-270
    state = TrainState(field, opt)
    occ = OccupancyUpdate(cb, cfg, est, field, rk["render_step_size"], dp.SharedRng(4242, dev))

    gen = torch.Generator().manual_seed(1000 + rank)  # every rank draws its own slice of the global batch
    n_host = 4
    host = [workload.draw_batch(cfg, n_rays, gen, pin=True) for _ in range(n_host)]
    resident = [{k: v.to(dev) for k, v in b.items()} for b in host]
    # allocator warm-up batches: the visible-sample count moves by a few % from step to step.  Untimed forward+backward
    # passes (no optimiser step) on 1.06 x, 1.12 x ... the rays, run after the warm-up steps, leave free blocks of the
    # next size classes in the cache, so the timed step in which the count crosses a boundary does not grow the pool.
    n_classes = max(2, int((0.003 * (steps + max(warmup, 3)) + 0.06) / 0.06) + 1)
    oversized = [{k: v.to(dev) for k, v in workload.draw_batch(cfg, int(n_rays * (1.0 + 0.06 * (j + 1))), gen).items()}
                 for j in range(min(n_classes, 12))]

    def touch_size_classes():
        for b in oversized:
            rays_b = cb.Rays(b["origins"], b["viewdirs"])
            rgb, acc, _, n_s, extra = cb.render_image(field, est, rays_b, render_bkgd=b["color_bkgd"],
                                                      timestamps=b["timestamps"], jitter=b["jitter"], **rk)
            loss = torch.nn.functional.mse_loss(rgb, b["pixels"]) + aux_losses(rgb, acc, b["pixels"], extra, cfg.flags)
            opt.zero_grad()
            scaler.scale(loss).backward()
            if reducer is not None:
                reducer.wait()
            opt.zero_grad()

    keep = {} if (args.dump_outputs and full) else None   # the tensors of the latest resident step, for --dump-outputs

    def step_resident(i):
        return train_step(cb, field, est, opt, scaler, resident[i % n_host], cfg, rk, reducer, state.sched, occ,
                          not args.host_counts, keep)

    # End-to-end leg: every step's inputs come from pinned host memory and every step's loss goes back to the host, both
    # inside the timed region - pipelined the way a data loader and a logger are: batch i + 1 is copied on a side stream
    # while step i computes, and the loss of step i is read (from a pinned buffer, after its own event) while step i + 1
    # is being enqueued; the last loss is read before the clock stops.
    copy_stream = torch.cuda.Stream(device=dev)
    loss_host = [torch.zeros(1).pin_memory() for _ in range(2)]
    pipe = {"next": None, "pending": None, "losses": []}

    def upload(i):
        with torch.cuda.stream(copy_stream):
            b = {k: v.to(dev, non_blocking=True) for k, v in host[i % n_host].items()}
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return b, ev

    def step_e2e(i):
        if pipe["next"] is not None and pipe["next"][2] == i:
            b, ev = pipe["next"][0], pipe["next"][1]
        else:
            b, ev = upload(i)
        torch.cuda.current_stream().wait_event(ev)
        for t in b.values():
            t.record_stream(torch.cuda.current_stream())
        nb, nev = upload(i + 1)
        pipe["next"] = (nb, nev, i + 1)
        loss, n_s = train_step(cb, field, est, opt, scaler, b, cfg, rk, reducer, state.sched, occ, not args.host_counts)
        if pipe["pending"] is not None:                 # device -> host read of the PREVIOUS step's result
            pev, slot = pipe["pending"]
            pev.synchronize()
            pipe["losses"].append(float(loss_host[slot][0]))
        slot = i & 1
        loss_host[slot].copy_(loss.detach().reshape(1), non_blocking=True)
        lev = torch.cuda.Event()
        lev.record()
        pipe["pending"] = (lev, slot)
        return loss, n_s

    def drain_e2e():
        if pipe["pending"] is not None:
            pev, slot = pipe["pending"]
            pev.synchronize()
            pipe["losses"].append(float(loss_host[slot][0]))
            pipe["pending"] = None
        pipe["next"] = None

    def timed(fn, k):
        state.restore()          # iteration 0 again (untimed), then the warm-up steps allocate the optimiser state
        occ.step = 0
        for i in range(max(warmup, 3)):
            fn(i)
        touch_size_classes()
        D.barrier()
        occ.updates = 0
        l0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n_tot = 0
        drain = fn is step_e2e
        if drain:
            drain_e2e()
        for i in range(k):
            if os.environ.get("BENCH_DEBUG_STEPS"):
                torch.cuda.synchronize()
                t_dbg = time.perf_counter()
                n_i = fn(i)[1]
                torch.cuda.synchronize()
                print(f"[debug] step {i}: {(time.perf_counter() - t_dbg) * 1e3:.2f} ms, {n_i} samples", file=sys.stderr)
                n_tot += n_i
                continue
            n_tot += fn(i)[1]
        if drain:
            drain_e2e()   # the last step's loss reaches the host before the clock stops
        e1.record()
        D.barrier()
        ms = dp.max_over_ranks(e0.elapsed_time(e1) / k, dev)
        return ms, float(n_tot) / k, (_lib.launch_count() - l0) // k

    if os.environ.get("BENCH_SYNC_DEBUG"):   # list every host<->device synchronisation of two steady-state steps
        state.restore()
        for i in range(4):
            step_resident(i)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("warn")
        for i in range(2):
            step_resident(4 + i)
        torch.cuda.set_sync_debug_mode("default")
    clocks = ClockSampler(D.local_rank) if (full and rank == 0) else None
    if clocks:
        clocks.start()
    ms, samples, launches = timed(step_resident, steps)
    out = {"ms": ms, "samples": dp.sum_over_ranks(samples, dev), "launches": int(launches), "occ_updates": occ.updates,
           "dp_mode": dp_mode, "rays": n_rays * world, "dropped": int(est.dropped_samples), "clocks": clocks.stop() if clocks else None,
           "h2d": sum(v.numel() * v.element_size() for v in host[0].values())}
    if keep is not None:   # before the legs below run more steps on the same field
        out["outputs"] = host_outputs(keep, field)
        keep = None
    if full:
        out["ms_e2e"] = timed(step_e2e, steps)[0]
    if args.profile_steps > 0 and full:
        # every rank runs the instrumented steps (they contain the cross-rank barriers); rank 0 keeps the records
        state.restore()
        step_resident(0)
        with Instrument(cb, _lib) as ins:
            D.barrier()
            t0 = time.perf_counter()
            for i in range(args.profile_steps):
                step_resident(i)
            torch.cuda.synchronize()
            prof_ms = (time.perf_counter() - t0) * 1e3 / args.profile_steps
        if rank == 0:
            live = {k: v.get("last") for k, v in est._cap_state.items()}   # totals of a recent batch (capacity mode)
            agg = ins.aggregate(live)
            out["breakdown"] = {n: {"ms_per_step": round(d["ms"] / args.profile_steps, 4),
                                    "launches_per_step": d["launches"] // args.profile_steps} for n, d in agg.items()}
            out["breakdown"]["_ours_total_ms"] = round(sum(v["ms"] for v in agg.values()) / args.profile_steps, 3)
            out["breakdown"]["_instrumented_step_ms"] = round(prof_ms, 3)
            out["roofline"] = roofline_of(agg, args.profile_steps, prof_ms)
    if args.torch_profile and full:
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            step_resident(0)
            torch.cuda.synchronize()
        if rank == 0:
            with open(args.torch_profile, "w") as f:
                f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=60, max_name_column_width=70))
    if dp_mode == "peer":
        out["dp_mode"] = "peer/" + opt.transport()
        out["dp_timed_out"] = bool(opt.timed_out())
        opt.close()
    if reducer is not None:
        reducer.remove()
    return out


# --------------------------------------------------------------------------------------------------------------
# render leg: full frames through render_image_test, frames interleaved over the ranks, no collective
# --------------------------------------------------------------------------------------------------------------
def render_leg(D, cb, workload, cfg, args, poses, times, opengl, bkgd, profile: bool, dump: bool = False):
    """poses [F,3,4], times [F]: the whole job; rank r renders frames r, r+W, ... (strong scaling).  `dump`: return the
    last frame of the timed job under "outputs"."""
    from cednerf_b200 import _lib, dp

    dev, world, rank = D.dev, D.world, D.rank
    rk = workload.render_kwargs(cfg)
    est, field = workload.build_scene(cfg, dev, cb, seed=42)
    est.eval(), field.eval()
    mine = dp.shard_interleaved(len(poses), rank, world)
    bk = torch.tensor(bkgd, dtype=torch.float32, device=dev)
    frames = [(poses[i].to(dev), torch.tensor([[float(times[i])]], device=dev)) for i in mine]
    K = [[cfg.focal, 0.0, cfg.width / 2], [0.0, cfg.focal, cfg.height / 2], [0.0, 0.0, 1.0]]

    # the frame goes back to the host as 8-bit RGB (what the reference's video writer consumes, 3 bytes per pixel), through
    # a ring of pinned buffers: the copy of frame k overlaps the rendering of frame k + 1
    ring = [torch.empty(cfg.height, cfg.width, 3, dtype=torch.uint8).pin_memory() for _ in range(3)]
    copies = []

    n_samples_box = [0]
    keep = {} if dump else None

    def to_host(k, res):   # 8-bit frame -> pinned ring; the copy of frame k overlaps the rendering of the next frames
        rgb, _, _, n_s = res
        n_samples_box[0] += n_s
        if keep is not None and k == len(frames) - 1:   # frames complete out of order: keep the job's last frame
            keep.update(rgb=rgb, acc=res[1], depth=res[2], n_samples=n_s)
        if len(copies) >= len(ring):
            copies.pop(0).synchronize()
        ring[k % len(ring)].copy_((rgb.clamp(0.0, 1.0) * 255.0).to(torch.uint8), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        copies.append(ev)

    def render_all(idx):
        """Frames `idx` through render_images_test: pixel -> ray generation (one launch per frame, inside the timed region,
        gui.py:43-86 does it per frame), the marching rounds of `--render-streams` frames interleaved, 8-bit frames to the host."""
        n_samples_box[0] = 0
        rays = [(lambda c=frames[k][0]: cb.utils.generate_rays(K, c, cfg.width, cfg.height, opengl)) for k in idx]
        cb.utils.render_images_test(1024, field, est, rays, [frames[k][1] for k in idx], concurrency=args.render_streams,
                                    on_frame=to_host, render_bkgd=bk, **rk)
        while copies:
            copies.pop(0).synchronize()   # every frame has reached the host before the clock stops
        return n_samples_box[0]

    # warm-up: one frame more than there are frames in flight, so that every stream of render_images_test has run a frame
    # (each stream has its own allocator pool; a cold pool means cudaMallocs of ~1 GB of per-frame buffers inside the clock)
    render_all(list(range(min(max(3, args.render_streams + 1), len(frames)))))
    D.barrier()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = _lib.launch_count()
    r0.record()
    n_samples = render_all(list(range(len(frames))))
    r1.record()
    D.barrier()
    ms = dp.max_over_ranks(r0.elapsed_time(r1), dev)
    n_all = dp.sum_over_ranks(n_samples, dev)
    rays = cfg.width * cfg.height * len(poses)
    hbm_peak, _ = peaks()
    out = {"workload": f"{cfg.name}: {len(poses)} {cfg.width}x{cfg.height} frames, render_image_test(1024), "
                       f"frames interleaved over {world} GPU(s), no collective; {args.render_streams} frame(s) in flight per GPU",
           "frames": len(poses), "scaling": "strong", "d2h_bytes_per_frame": cfg.width * cfg.height * 3, "rays_per_s": round(rays / (ms * 1e-3), 1),
           "samples_per_s": round(n_all / (ms * 1e-3), 1), "ms_per_frame_per_gpu": round(ms / max(len(mine), 1), 3),
           "samples_per_ray": round(n_all / rays, 3), "launches_per_frame": (_lib.launch_count() - l0) // max(len(mine), 1),
           # fused render per sample: 512 B table + ~50 B (SURVEY.md 8d) against the HBM copy peak, whole job
           "pipeline_frac": round(n_all * 562 / (ms * 1e-3) / 1e9 / (hbm_peak * world), 4)}
    if keep:
        out["outputs"] = host_outputs(keep)
    if profile and rank == 0 and frames:
        with Instrument(cb, _lib) as ins:
            cb.render_image_test(1024, field, est, cb.utils.generate_rays(K, frames[0][0], cfg.width, cfg.height, opengl),
                                 render_bkgd=bk, timestamps=frames[0][1], **rk)
            torch.cuda.synchronize()
        agg = ins.aggregate()
        out["breakdown_ms_per_frame"] = {k: [round(v["ms"], 3), v["launches"]] for k, v in
                                         sorted(agg.items(), key=lambda kv: -kv[1]["ms"])}
    return out


def encoder4d_leg(cb, workload, dev, log2_samples=22):
    """North-star kernel (2) on its own: the 4-D (xyz + t key-frame) hash encoder of hash_encoder_inter.py:279-430 at full
    size (16 levels, 2^21 entries x 8 fp16 per hashed level: a 383 MB table, NOT L2-resident) on the packed samples of a
    DyNeRF-shaped batch.  Algorithmic bytes per sample (SURVEY.md 8d): forward 16 x 8 x 16 B + 16 B + 64 B, backward 64 B
    + 16 B + 16 x 8 x 16 B of fp32 gradient; fraction of the measured HBM copy bandwidth."""
    cfg = workload.DYNERF
    rk = workload.render_kwargs(cfg)
    enc = cb.hash_encoder.HashEncoder4D(max_params=2 ** 21, levels=16, base_res=16.0, max_res=2048.0, seed=3).to(dev)
    est, _ = workload.build_scene(cfg, dev, cb, seed=42)
    est.train()
    b = {k: v.to(dev) for k, v in workload.draw_batch(cfg, 262144, torch.Generator().manual_seed(1000)).items()}
    with torch.no_grad():
        ridx, t0, t1 = est.sampling(b["origins"], b["viewdirs"], stratified=True, jitter=b["jitter"], **rk)
    n = min(2 ** log2_samples, ridx.numel())
    x = b["origins"][ridx[:n]] + b["viewdirs"][ridx[:n]] * ((t0[:n] + t1[:n]) / 2)[:, None]
    lo, hi = (torch.tensor(cfg.roi_aabb[k:k + 3], device=dev) for k in (0, 3))
    pts = torch.cat([((x - lo) / (hi - lo)).clamp(0, 1), b["timestamps"][ridx[:n]]], -1).contiguous()
    dy = torch.randn(n, 32, device=dev).half()
    peak = peaks()[0]

    def timed(fn, k):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k

    with torch.no_grad():
        fwd = timed(lambda: enc(pts), 10)
    y = enc(pts)

    def bwd():
        enc.hash_table.grad = None
        y.backward(dy, retain_graph=True)

    zero = timed(lambda: torch.zeros_like(enc.hash_table), 5)
    tot = timed(bwd, 5)
    fb, bb = 2128.0 * n, 2128.0 * n
    return {"workload": "4-D hash encoder, 16 levels x 2^21 x 8 fp16 (383 MB table), packed samples of a DyNeRF-shaped batch",
            "samples": n, "fwd_ms": round(fwd, 4), "fwd_gbs": round(fb / fwd / 1e6, 1), "fwd_frac": round(fb / fwd / 1e6 / peak, 4),
            "bwd_ms": round(tot - zero, 4), "bwd_gbs": round(bb / (tot - zero) / 1e6, 1),
            "bwd_frac": round(bb / (tot - zero) / 1e6 / peak, 4), "bound": "hbm", "peak_gbs": peak,
            "bytes_per_sample": 2128}


def run_ours(args):
    import cednerf_b200 as cb
    from cednerf_b200 import workload

    D = Dist()
    rank, world = D.rank, D.world
    cfgs = {"dynerf": workload.DYNERF, "hypernerf": workload.HYPERNERF, "dnerf": workload.DNERF}
    cfg = cfgs[args.config]

    def video_leg(profile):
        n = max(1, args.render_frames)
        idx = [k * 300 // n for k in range(n)] if n < 300 else list(range(300))
        poses = workload.spiral_poses(workload.DYNERF, 300)
        return render_leg(D, cb, workload, workload.DYNERF, args, poses[idx], [k / 300.0 for k in idx], False,
                          (0.0, 0.0, 0.0), profile)

    def dnerf_leg(n_frames, profile, dump=False):
        poses = torch.stack([workload.orbit_pose(4.0, 2 * 3.14159265 * k / n_frames) for k in range(n_frames)])
        return render_leg(D, cb, workload, workload.DNERF, args, poses, [0.5] * n_frames, True, (1.0, 1.0, 1.0), profile,
                          dump)

    line = {"higher_is_better": True, "vs_baseline": None, "data": "synthetic", "n_gpus": world,
            "dtype": "f16 (MLP, tables) / f32 (marching, compositing, grads)"}
    extra = {}
    if args.config == "dnerf":   # configs[0]: one "step" = one 800x800 frame
        n_frames = max(args.steps, 1) * world
        for _ in range(1):
            r = dnerf_leg(n_frames, args.profile_steps > 0, bool(args.dump_outputs))
        outputs = r.pop("outputs", None)
        line.update({"metric": "render_rays_per_s", "value": r["rays_per_s"], "unit": "rays/s", "steps": args.steps,
                     "warmup": 2, "ms_per_step": r["ms_per_frame_per_gpu"], "scaling": "weak",
                     "config": {"workload": r["workload"], "samples_per_ray": r["samples_per_ray"],
                                "samples_per_s": r["samples_per_s"], "l2": "inputs (800x800 rays x frames) and the 96 MB table exceed L2"},
                     "e2e": {"value": r["rays_per_s"], "unit": "rays/s", "h2d_bytes_per_step": 48,
                             "d2h_bytes_per_step": r["d2h_bytes_per_frame"],
                             "note": "a 3x4 pose goes up, the 8-bit frame comes back (pipelined with the next frame)"},
                     "gpu_launches": r["launches_per_frame"], "clocks": None,
                     "roofline": {"bound": "hbm", "frac": r["pipeline_frac"], "kernel": "render pipeline"}})
        extra["render_breakdown"] = r.get("breakdown_ms_per_frame")
    else:
        t = train_leg(D, cb, workload, cfg, args, args.rays, args.steps, args.warmup, True)
        outputs = t.pop("outputs", None)
        rays_all = t["rays"]
        line.update({
            "metric": "train_step_rays_per_s", "value": round(rays_all / (t["ms"] * 1e-3), 1), "unit": "rays/s",
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(t["ms"], 4), "scaling": "weak",
            "config": {"workload": f"{cfg.name} train step, {args.rays} rays/GPU/step, occgrid sampler "
                                   f"(BASELINE.json configs[{1 if args.config == 'dynerf' else 2}])",
                       "flags": "-te -ta -df -f -wr -ae; GradScaler 2^10 + fused Adam",
                       "rays_per_gpu": args.rays, "samples_per_step": round(t["samples"], 1),
                       "samples_per_ray": round(t["samples"] / rays_all, 3),
                       "samples_per_s": round(t["samples"] / (t["ms"] * 1e-3), 1),
                       "l2": "working set (96 MB fp16 table, 191 MB fp32 master, 383 MB Adam state) exceeds the 126 MB L2; 4 rotating batches",
                       "occ_update": f"every step on a twin estimator; {t['occ_updates']} full update(s) in the timed steps",
                       "sample_counts": ("host reads (reference behaviour)" if args.host_counts else
                                         f"device-side, capacity mode; {t['dropped']} samples dropped"),
                       "parallelism": ("single" if world == 1 else
                                       f"dp{world}, optimiser step: " + (f"fused reduce-scatter+Adam+all-gather over NVLink peer memory ({t['dp_mode']})"
                                                                        if t["dp_mode"].startswith("peer") else "NCCL all-reduce + Adam"))},
            "e2e": {"value": round(rays_all / (t["ms_e2e"] * 1e-3), 1), "unit": "rays/s", "ms_per_step": round(t["ms_e2e"], 4),
                    "h2d_bytes_per_step": t["h2d"], "d2h_bytes_per_step": 4,
                    "pipelining": "batch i+1 is uploaded on a side stream during step i; the loss of step i is read during step i+1"},
            "gpu_launches": t["launches"], "clocks": t["clocks"], "roofline": t.get("roofline")})
        if t.get("dp_timed_out"):
            line["config"]["parallelism"] += " (A BARRIER TIMED OUT)"
        extra["breakdown"] = t.get("breakdown")

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = run_reference_steps(args.config, args.cpu_rays, steps=3, warmup=1)
    line["cpu_baseline"] = cpu
    line.update(extra)   # the long per-kernel tables go before the other configurations: the END of the line is what a
                         # truncated log keeps
    if not args.headline_only and args.config == "dynerf":
        others = {}
        if args.render_frames > 0:
            line["render"] = video_leg(args.profile_steps > 0)
            line["config"]["render"] = {k: line["render"][k] for k in ("frames", "rays_per_s", "samples_per_s",
                                                                       "ms_per_frame_per_gpu", "pipeline_frac")}
        r = dnerf_leg(16 * world, False)
        others["dnerf"] = {k: r[k] for k in ("frames", "rays_per_s", "samples_per_s", "ms_per_frame_per_gpu",
                                             "samples_per_ray", "pipeline_frac")}
        h = train_leg(D, cb, workload, workload.HYPERNERF, args, args.rays, 10, 3, False)
        others["hypernerf"] = {"rays_per_s": round(h["rays"] / (h["ms"] * 1e-3), 1), "ms_per_step": round(h["ms"], 4),
                               "samples_per_s": round(h["samples"] / (h["ms"] * 1e-3), 1),
                               "samples_per_ray": round(h["samples"] / h["rays"], 3), "rays_per_gpu": args.rays}
        if world == 1:  # north-star kernel (2) at full size, on its own (it is not on the canonical recipes' path)
            others["encoder4d"] = encoder4d_leg(cb, workload, D.dev)
        if world > 1:   # configs[4]: 2^20 rays per step split over the ranks
            s = train_leg(D, cb, workload, workload.DYNERF, args, 2 ** 20 // world, 10, 3, False)
            others["dynerf_2p20"] = {"rays_per_s": round(s["rays"] / (s["ms"] * 1e-3), 1), "ms_per_step": round(s["ms"], 4),
                                     "rays_per_gpu": 2 ** 20 // world, "samples_per_s": round(s["samples"] / (s["ms"] * 1e-3), 1),
                                     "dp": s["dp_mode"]}
        line["configs"] = others
        line["config"]["others"] = others
    try:   # the last ~400 characters of the line: what a truncated log keeps of every configuration
        cfgs_ = line.get("configs") or {}
        rnd = line.get("render") or {}
        line["summary"] = {
            "n_gpus": world, "metric": line.get("metric"), "value": line.get("value"), "ms_per_step": line.get("ms_per_step"),
            "e2e": (line.get("e2e") or {}).get("value"), "roofline_frac": (line.get("roofline") or {}).get("frac"),
            "video_rays_per_s": rnd.get("rays_per_s"), "video_ms_per_frame_per_gpu": rnd.get("ms_per_frame_per_gpu"),
            "dnerf_ms_per_frame": (cfgs_.get("dnerf") or {}).get("ms_per_frame_per_gpu"),
            "hypernerf_ms_per_step": (cfgs_.get("hypernerf") or {}).get("ms_per_step"),
            "dynerf_2p20_rays_per_s": (cfgs_.get("dynerf_2p20") or {}).get("rays_per_s"),
            "encoder4d_fwd_bwd_frac": [(cfgs_.get("encoder4d") or {}).get("fwd_frac"), (cfgs_.get("encoder4d") or {}).get("bwd_frac")]}
    except Exception:  # noqa: BLE001 - a summary must never cost the line
        pass
    if rank == 0 and outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        D.dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------------------
# reference arm: the CPU restatement of the reference path (the reference itself cannot run: nerfacc / tiny-cuda-nn /
# Taichi are CUDA-only third-party packages that are not installed and the reference has no CPU path, BASELINE.md §2)
# --------------------------------------------------------------------------------------------------------------
class _OracleImpl:
    def __init__(self):
        from oracle import cednerf_ref as cr
        from oracle import nerfacc_ref as nf

        self.OccGridEstimator, self.DNGPradianceField = nf.OccGridEstimator, cr.DNGPradianceField
        self.Rays, self.render_image, self.render_image_test = cr.Rays, cr.render_image, cr.render_image_test


def run_reference_steps(config, n_rays, steps, warmup):
    """The headline configuration on the CPU restatement: same initial weights (workload.initial_state + density boost),
    same learning rate (iteration 0 of the reference schedule), same loss scaling, a bounded sample of the rays."""
    workload = load_workload()
    torch.set_num_threads(os.cpu_count() or 1)
    impl = _OracleImpl()
    cfg = {"dynerf": workload.DYNERF, "hypernerf": workload.HYPERNERF, "dnerf": workload.DNERF}[config]
    rk = workload.render_kwargs(cfg)
    est, field = workload.build_scene(cfg, "cpu", impl, seed=42)
    if config == "dnerf":   # a square crop of the 800x800 frame (each render marches the crop to the end: ~280 samples
        est.eval(), field.eval()   # per ray through 35 rounds of the oracle's field, ~0.1 s per ray-round batch)
        side = max(8, int(min(n_rays, 256) ** 0.5))
        o, d = workload.pose_rays(cfg, workload.orbit_pose(4.0, 0.0), True)
        lo = (cfg.height - side) // 2
        sel = (torch.arange(lo, lo + side)[:, None] * cfg.width + torch.arange(lo, lo + side)[None, :]).reshape(-1)
        rays = impl.Rays(o[sel], d[sel])
        times, samples = [], 0
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            with torch.no_grad():
                n_s = impl.render_image_test(1024, field, est, rays, render_bkgd=torch.ones(3),
                                             timestamps=torch.tensor([[0.5]]), **rk)[3]
            if i >= warmup:
                times.append(time.perf_counter() - t0)
                samples += n_s
        sec = sum(times) / len(times)
        return {"value": round(side * side / sec, 1), "unit": "rays/s", "cores": torch.get_num_threads(), "kind": "port",
                "sample": f"centre {side}x{side} crop of one 800x800 frame, {steps} timed renders "
                          f"({round(samples / steps / side / side, 2)} samples/ray), oracle/ PyTorch-CPU + OpenMP C marcher",
                "ms_per_step": round(sec * 1e3, 1), "samples_per_s": round(samples / steps / sec, 1)}
    est.train(), field.train()
    opt = torch.optim.Adam(field.parameters(), lr=1e-2, eps=1e-15)
    make_scheduler(opt)   # lr -> 1e-4, as the GPU arm's TrainState
    gen = torch.Generator().manual_seed(1000)
    batches = [workload.draw_batch(cfg, n_rays, gen) for _ in range(2)]
    times, samples = [], 0
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        _, n_s = train_step(impl, field, est, opt, None, batches[i % 2], cfg, rk)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
            samples += n_s
    sec = sum(times) / len(times)
    return {"value": round(n_rays / sec, 1), "unit": "rays/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n_rays} rays/step of the same workload and initial weights, {steps} timed steps after {warmup} "
                      f"warm-up ({round(samples / steps / n_rays, 2)} samples/ray; no occupancy update), oracle/ "
                      f"PyTorch-CPU + OpenMP C marcher",
            "ms_per_step": round(sec * 1e3, 1), "samples_per_s": round(samples / steps / sec, 1),
            "samples_per_ray": round(samples / steps / n_rays, 3)}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 3))
    cpu = run_reference_steps(args.config, args.cpu_rays, steps=steps, warmup=1)
    train = args.config != "dnerf"
    line = {"impl": "reference", "metric": "train_step_rays_per_s" if train else "render_rays_per_s", "value": cpu["value"],
            "unit": "rays/s", "n_gpus": args.gpus, "steps": steps, "warmup": 1, "ms_per_step": cpu["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (CPU), fp16-rounded MLP",
            "data": "synthetic",
            "config": {"workload": f"{args.config}-shaped {'train step' if train else 'frame render'}, bounded sample of "
                                   f"{args.cpu_rays} rays/step on the host CPU, same initial weights / lr / loss scale as the GPU arm"},
            "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
