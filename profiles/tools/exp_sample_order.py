"""Does the ORDER of the visible samples matter to the gradient-carrying field kernels?  The fused training forward and
backward on the visible samples of a DyNeRF-shaped batch, (a) in ray order (as `render_image` feeds them) and (b) sorted
by a Morton key of their position - same samples, same results up to the permutation; kernel times per entry point.

    python profiles/tools/exp_sample_order.py [bits per axis]"""
import sys, torch
sys.path.insert(0, '/root/repo')
import cednerf_b200 as cb
from cednerf_b200 import workload as w, _lib
import bench
DEV = torch.device('cuda:0')
bits = int(sys.argv[1]) if len(sys.argv) > 1 else 7
cfg = w.DYNERF; rk = w.render_kwargs(cfg)
est, field = w.build_scene(cfg, DEV, cb, seed=42); est.train(); field.train()
b = {k: v.to(DEV) for k, v in w.draw_batch(cfg, 262144, torch.Generator().manual_seed(1000)).items()}
rays = cb.Rays(b['origins'], b['viewdirs'])
with torch.no_grad():
    sigma_fn = cb.utils._field_fns(field, rays, b['timestamps'])[0]
    ridx, t0, t1 = est.sampling(b['origins'], b['viewdirs'], sigma_fn=sigma_fn, stratified=True, jitter=b['jitter'], **rk)
n = ridx.numel()
x = b['origins'][ridx] + b['viewdirs'][ridx] * ((t0 + t1) / 2)[:, None]
lo, hi = torch.tensor(cfg.roi_aabb[:3], device=DEV), torch.tensor(cfg.roi_aabb[3:], device=DEV)
q = (((x - lo) / (hi - lo)).clamp(0, 1 - 1e-6) * (1 << bits)).long()
def spread(v):
    out = torch.zeros_like(v)
    for i in range(bits): out |= ((v >> i) & 1) << (3 * i)
    return out
key = spread(q[:, 0]) | (spread(q[:, 1]) << 1) | (spread(q[:, 2]) << 2)
perm = torch.argsort(key)
gs, gr = torch.randn(n, device=DEV) * 1e-3, torch.randn(n, 3, device=DEV) * 1e-3
def run(order, label):
    ri, a0, a1 = (ridx[order], t0[order], t1[order]) if order is not None else (ridx, t0, t1)
    g0, g1 = (gs[order], gr[order]) if order is not None else (gs, gr)
    def step():
        for p in field.parameters(): p.grad = None
        rgb, out = field.fused_train(ri, a0, a1, b['origins'], b['viewdirs'], b['timestamps'], 1)
        lat = out['interal_output']['latent_losses']
        ((out['density'][:, 0] * g0).sum() + (rgb * g1).sum() + lat.mean()).backward()
        return rgb
    for _ in range(2): step()
    torch.cuda.synchronize()
    with bench.Instrument(cb, _lib) as ins:
        for _ in range(5): rgb = step()
        torch.cuda.synchronize()
    agg = {}
    for name, a, s, e in ins.rec:
        agg.setdefault(name, 0.0); agg[name] += s.elapsed_time(e) / 5
    print(label, {k: round(v, 4) for k, v in agg.items() if v > 0.02})
    return rgb, [p.grad.clone() for p in field.parameters() if p.grad is not None]
r0, g_ray = run(None, f'{n} samples, ray order    ')
r1, g_sorted = run(perm, f'sorted by {3 * bits}-bit Morton key')
# (c) whole RAYS reordered (samples stay packed per ray): key of a ray = Morton code of its point at the depth of the scene
depth = float((lo + hi).norm()) * 0 + 1.6
pr = b['origins'] + b['viewdirs'] * depth
qr = (((pr - lo) / (hi - lo)).clamp(0, 1 - 1e-6) * (1 << bits)).long()
rkey = spread(qr[:, 0]) | (spread(qr[:, 1]) << 1) | (spread(qr[:, 2]) << 2)
rank = torch.empty_like(rkey); rank[torch.argsort(rkey)] = torch.arange(rkey.numel(), device=DEV)
perm_r = torch.argsort(rank[ridx], stable=True)
r2, g_rays = run(perm_r, 'rays sorted (samples packed)  ')
print('max |rgb diff| after un-permuting', float((r1 - r0[perm]).detach().abs().max()), float((r2 - r0[perm_r]).detach().abs().max()))
print('gradient rel diff per tensor', [float((a - c).norm() / (c.norm() + 1e-30)) for a, c in zip(g_sorted, g_ray)])
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(10): p2 = torch.argsort(key)
e1.record(); torch.cuda.synchronize(); print('torch.argsort of the keys', e0.elapsed_time(e1) / 10, 'ms')
