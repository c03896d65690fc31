"""MS-SSIM of the evaluation after training (cednerf_b200.metrics.ms_ssim, csrc/metrics.cu) against pytorch_msssim's
formulation in torch on the same GPU (oracle/metrics_ref.ms_ssim: what the reference pays), on DyNeRF test frames
(3 x 1014 x 1352 fp32, two images per pair):

  * per-call time, median of 60 calls after warm-up, CUDA events around each call: one pair and a batch of 8, with the
    inputs taken from a pool that is L2-resident (one pair, 33 MB; a batch of 8 pairs is 263 MB and never is) or from
    a pool of more than 200 MB (HBM reads included);
  * launches per call: the library's counter, and CUDA kernels per call under torch.profiler (a separate run);
  * an evaluation run: 96 spiral frames rendered with render_images_test, three in flight, alone and with every frame
    scored in on_frame (against a fixed target), ms per frame.

Prints its numbers as one JSON line at the end, and writes them to OUT.json if given:
    python profiles/tools/exp_metrics.py [OUT.json]"""
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import cednerf_b200 as cb  # noqa: E402
from cednerf_b200 import _lib, workload as w  # noqa: E402
from oracle import metrics_ref as mr  # noqa: E402

DEV = torch.device("cuda:0")
H, W, CALLS, WARMUP = 1014, 1352, 60, 10


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def timed(fn, pool):
    """median / min ms of CALLS calls, input pair i % len(pool), events around each call"""
    for i in range(WARMUP):
        fn(*pool[i % len(pool)])
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(CALLS)]
    for i, (a, b) in enumerate(ev):
        x, y = pool[i % len(pool)]
        a.record()
        fn(x, y)
        b.record()
    torch.cuda.synchronize()
    t = [a.elapsed_time(b) for a, b in ev]
    return round(statistics.median(t), 4), round(min(t), 4)


def kernels_per_call(fn, x, y):
    from torch.profiler import ProfilerActivity, profile

    fn(x, y)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            fn(x, y)
        torch.cuda.synchronize()
    names = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "emcpy" not in e.name
             and "emset" not in e.name]
    return len(names) / 5


def main():
    out = {"card (name, power limit, max SM clock)": card()}
    print(out)
    ours = lambda x, y: cb.metrics.ms_ssim(x, y, data_range=1.0)  # noqa: E731
    ref = lambda x, y: mr.ms_ssim(x, y, data_range=1.0)  # noqa: E731
    g = torch.Generator(device=DEV).manual_seed(0)
    pair_bytes = 2 * 3 * H * W * 4
    for n in (1, 8):
        one = [(torch.rand(n, 3, H, W, device=DEV, generator=g), torch.rand(n, 3, H, W, device=DEV, generator=g))]
        k = max(1, -(-(200 << 20) // (pair_bytes * n)))   # > 126 MB of L2
        big = [(torch.rand(n, 3, H, W, device=DEV, generator=g), torch.rand(n, 3, H, W, device=DEV, generator=g))
               for _ in range(k)]
        x, y = one[0]
        diff = abs(float(ours(x, y)) - float(ref(x, y)))
        l0 = _lib.launch_count()
        ours(x, y)
        launches = _lib.launch_count() - l0
        row = {"n": n, "pool_small_MB": round(pair_bytes * n / 2 ** 20, 1), "pool_large_MB": round(pair_bytes * n * k / 2 ** 20, 1),
               "ours_ms_small_pool (median, min)": timed(ours, one), "ours_ms_large_pool": timed(ours, big),
               "torch_ms_small_pool": timed(ref, one), "torch_ms_large_pool": timed(ref, big),
               "ours_library_launches_per_call": launches, "|ours - torch|": diff}
        print(row)
        out[f"batch{n}"] = row
        del big
    x, y = (torch.rand(1, 3, H, W, device=DEV, generator=g) for _ in range(2))
    out["cuda_kernels_per_call (torch.profiler)"] = {"ours": kernels_per_call(ours, x, y),
                                                     "torch": kernels_per_call(ref, x, y)}
    print(out["cuda_kernels_per_call (torch.profiler)"])

    # evaluation run: 96 spiral frames of the DyNeRF-shaped scene, three in flight
    cfg = w.DYNERF
    rk = w.render_kwargs(cfg)
    est, field = w.build_scene(cfg, DEV, cb, seed=42)
    est.eval(), field.eval()
    poses = [p.to(DEV) for p in w.spiral_poses(cfg, 96)]
    ts = [torch.tensor([[k / 96.0]], device=DEV) for k in range(96)]
    K = [[cfg.focal, 0.0, cfg.width / 2], [0.0, cfg.focal, cfg.height / 2], [0.0, 0.0, 1.0]]
    bk = torch.zeros(3, device=DEV)
    target = torch.rand(cfg.height, cfg.width, 3, device=DEV, generator=g).permute(2, 0, 1)[None]
    scores = []

    def score(k, res):
        scores.append(cb.metrics.ms_ssim(res[0].permute(2, 0, 1)[None], target, data_range=1.0))

    def run(idx, on_frame):
        rays = [(lambda c=poses[k]: cb.utils.generate_rays(K, c, cfg.width, cfg.height)) for k in idx]
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        with torch.no_grad():
            cb.render_images_test(1024, field, est, rays, [ts[k] for k in idx], concurrency=3, on_frame=on_frame,
                                  render_bkgd=bk, **rk)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / len(idx)

    drop = lambda k, res: None  # noqa: E731  (frames are dropped, not kept, in both arms)
    run(list(range(4)), drop), run(list(range(4)), score)   # warm-up of every frame stream
    ev = {"render": [], "render+ms_ssim": []}
    for _ in range(2):   # alternate the two arms
        ev["render"].append(round(run(list(range(96)), drop), 3))
        scores.clear()
        ev["render+ms_ssim"].append(round(run(list(range(96)), score), 3))
    assert len(scores) == 96
    out["eval_96_frames_ms_per_frame (two alternated runs each)"] = ev
    print(ev)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
