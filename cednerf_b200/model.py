"""cednerf/model.py surface: DNGPradianceField (cednerf/model.py:97-488) on the B200 kernels.

Composition (per sample): deformation MLP F1 on Frequency(x, t) -> x + move -> aabb normalise + selector ->
hash grid -> [hash | time embedding] -> density MLP F2 -> trunc_exp; SH(dir) + geometry feature -> colour MLP F3
-> sigmoid; optional feature / weight predictors F4 / F5 (training only)."""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from . import ops, tcnn
from .encoder import SinusoidalEncoder, SinusoidalEncoderWithExp


class _TruncExp(torch.autograd.Function):
    """cednerf/utils.py:27-43: exp forward in fp32, backward g * exp(clamp(x, max=15))."""

    @staticmethod
    def forward(ctx, x):
        x = x.float()
        ctx.save_for_backward(x)
        return torch.exp(x)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return g * torch.exp(x.clamp(max=15.0))


trunc_exp = _TruncExp.apply


def _mlp_cfg(n_hidden):
    return {"otype": "FullyFusedMLP", "activation": "ReLU", "output_activation": "None", "n_neurons": 64,
            "n_hidden_layers": n_hidden}


class DNGPradianceField(torch.nn.Module):
    def __init__(self, aabb, num_dim: int = 3, use_viewdirs: bool = True, density_activation=None,
                 unbounded: bool = False, geo_feat_dim: int = 15, base_resolution: int = 16, n_levels: int = 16,
                 n_features_per_level: int = 2, dst_resolution: int = 4096, log2_hashmap_size: int = 19,
                 use_feat_predict: bool = False, use_weight_predict: bool = False, moving_step: float = 1 / 4096,
                 use_div_offsets: bool = False, use_time_embedding: bool = False, use_time_attenuation: bool = False,
                 time_inject_before_sigma: bool = True, hash4motion: bool = False, seed: int = 1337):
        super().__init__()
        if unbounded or hash4motion or num_dim != 3:
            raise NotImplementedError("bounded 3-D scenes without hash4motion (the reference's live configuration)")
        self.register_buffer("aabb", torch.as_tensor(aabb, dtype=torch.float32).flatten())
        self.num_dim, self.use_viewdirs, self.geo_feat_dim = num_dim, use_viewdirs, geo_feat_dim
        self.use_feat_predict, self.use_weight_predict = use_feat_predict, use_weight_predict
        self.use_time_embedding, self.use_time_attenuation = use_time_embedding, use_time_attenuation
        self.time_inject_before_sigma, self.use_div_offsets = time_inject_before_sigma, use_div_offsets
        self.MOVING_STEP, self.loose_move = moving_step, False
        self._default_density = density_activation is None
        self.density_activation = density_activation or (lambda x: trunc_exp(x - 1))
        freq = {"otype": "Frequency", "n_frequencies": 4}
        self.xyz_wrap = tcnn.NetworkWithInputEncoding(4, 6 if use_div_offsets else 3, freq, _mlp_cfg(3), seed + 1)
        if use_viewdirs:
            self.direction_encoding = tcnn.Encoding(3, {"otype": "Composite", "nested": [
                {"n_dims_to_encode": 3, "otype": "SphericalHarmonics", "degree": 2}]})
        b = math.exp(math.log(dst_resolution / base_resolution) / (n_levels - 1))
        self.hash_encoder = tcnn.Encoding(num_dim, {
            "otype": "HashGrid", "n_levels": n_levels, "n_features_per_level": n_features_per_level,
            "log2_hashmap_size": log2_hashmap_size, "base_resolution": base_resolution, "per_level_scale": b}, seed + 2)
        base_in, self.geo_feat_dim_head = self.hash_encoder.n_output_dims, geo_feat_dim
        if use_time_embedding:
            self.time_encoder = SinusoidalEncoder(1, 0, 4, True)               # both exist in the reference
            self.time_encoder_feat = SinusoidalEncoderWithExp(1, 0, 4, True)   # (model.py:266-267) and in its checkpoints
            if time_inject_before_sigma:
                base_in += 9
            else:
                self.geo_feat_dim_head += 9
        self.mlp_base = tcnn.Network(base_in, 1 + geo_feat_dim, _mlp_cfg(1), seed + 3)
        self.mlp_head = tcnn.Network((4 if use_viewdirs else 0) + self.geo_feat_dim_head, 3, _mlp_cfg(2), seed + 4)
        if use_feat_predict:
            self.mlp_feat_prediction = tcnn.NetworkWithInputEncoding(4, self.hash_encoder.n_output_dims, freq,
                                                                     _mlp_cfg(1), seed + 5)
        if use_weight_predict:
            self.mlp_weight_prediction = tcnn.NetworkWithInputEncoding(4, 1, freq, _mlp_cfg(1), seed + 6)

    # ---- fused no-grad path (cednerf_field_fwd): sampler pre-pass, occupancy updates, eval rendering ------------
    def fused_supported(self) -> bool:
        return (self.use_viewdirs and self.geo_feat_dim == 15 and not self.loose_move and self._default_density
                and self.hash_encoder.n_levels <= 16 and self.aabb.is_cuda)

    def _field_desc(self):
        key = (self.aabb.data_ptr(), self.aabb._version, self.MOVING_STEP)
        if getattr(self, "_fdesc_key", None) != key:
            from ._lib import FieldDesc

            d = FieldDesc()
            for i, v in enumerate(self.aabb.tolist()):
                d.aabb[i] = v
            d.moving_step = float(self.MOVING_STEP)
            d.use_div_offsets = int(self.use_div_offsets)
            d.time_mode = 0 if not self.use_time_embedding else (2 if self.use_time_attenuation else 1)
            d.time_before_sigma = int(self.time_inject_before_sigma)
            d.f1, d.f2, d.f3 = self.xyz_wrap.network.desc, self.mlp_base.desc, self.mlp_head.desc
            if self.use_feat_predict:
                d.f4 = self.mlp_feat_prediction.network.desc
            d.levels = self.hash_encoder.levels
            self._fdesc, self._fdesc_key = d, key
        return self._fdesc

    @torch.no_grad()
    def fused_query(self, n, packed=None, points=None, timestamps=None, t_stride=1, sigma_only=True, n_dev=None):
        """-> (sigma [n], rgb [n,3] | None) in one kernel; see ops.field_fwd."""
        images = (self.xyz_wrap.network.weight_image(), self.mlp_base.weight_image(), self.mlp_head.weight_image())
        return ops.field_fwd(self._field_desc(), images, self.hash_encoder.table_f16(), n, sigma_only, packed, points,
                             timestamps, t_stride, n_dev)

    def fused_train_supported(self) -> bool:
        return (self.fused_supported() and not self.use_weight_predict
                and (not self.use_feat_predict or self.hash_encoder.n_levels == 16))

    def fused_train(self, ridx, t0, t1, rays_o, rays_d, timestamps, t_stride):
        """Training forward of `forward(positions, t, directions)` on packed samples, differentiable w.r.t. every
        parameter: -> (rgb [n,3], {"density", "base_mlp_out", "interal_output"}) like the op-by-op path."""
        f4 = self.mlp_feat_prediction.network if self.use_feat_predict else None
        images = (self.xyz_wrap.network.weight_image(), self.mlp_base.weight_image(), self.mlp_head.weight_image(),
                  None if f4 is None else f4.weight_image())
        sigma, rgb, latent, selector, move = ops.FieldTrainFunction.apply(
            self.xyz_wrap.network.params, self.mlp_base.params, self.mlp_head.params,
            None if f4 is None else f4.params, self.hash_encoder.params.view(-1, 2), self._field_desc(), images,
            self.hash_encoder.table_f16(), ridx, t0, t1, rays_o, rays_d, timestamps, t_stride, f4 is not None,
            None if ops.counts_of(ridx) is None else ops.counts_of(ridx)[1])
        io = {"move": torch.linalg.norm(move, dim=-1) if (self.use_time_embedding and self.use_time_attenuation) else move}
        if self.use_feat_predict:
            io["selector"], io["latent_losses"] = selector, latent
        return rgb, {"density": sigma[:, None], "interal_output": io}

    def query_move(self, x, t):
        off = self.xyz_wrap(torch.cat([x, t], -1)).float()
        move = off[:, :3] * self.MOVING_STEP
        if self.use_div_offsets:
            move = move + torch.tanh(off[:, 3:]) * self.MOVING_STEP
        return x + move, move

    def query_density(self, x, t, return_feat: bool = False, return_interal: bool = False):
        if (not torch.is_grad_enabled()) and not return_feat and not return_interal and x.shape[0] > 0 \
                and self.fused_supported():
            xs = x.reshape(-1, 3)
            ts = t.reshape(-1)
            sigma, _ = self.fused_query(xs.shape[0], points=(xs, None), timestamps=ts,
                                        t_stride=1 if ts.numel() == xs.shape[0] else 0)
            return {"density": sigma[:, None]}
        if (not self.loose_move) and x.shape[0] > 0:
            x_move, move = self.query_move(x.view(-1, 3), t.view(-1, 1))
        else:
            x_move = x.view(-1, 3)
            move = torch.zeros_like(x_move[:, :1])
        lo, hi = self.aabb[:3], self.aabb[3:]
        x_move = (x_move - lo) / (hi - lo)
        selector = ((x_move > 0.0) & (x_move < 1.0)).all(-1)
        hash_feat = self.hash_encoder(x_move)
        feat = hash_feat
        time_encode = None
        if self.use_time_embedding:
            with torch.no_grad():
                if self.use_time_attenuation:
                    move = torch.linalg.norm(move.detach(), dim=-1)
                    time_encode = self.time_encoder_feat(t.view(-1, 1), move.view(-1, 1))
                else:
                    time_encode = self.time_encoder(t.view(-1, 1))
            if self.time_inject_before_sigma:
                feat = torch.cat([hash_feat, time_encode.to(hash_feat.dtype)], -1)
        h = self.mlp_base(feat).float()
        raw, base_out = h[:, :1], h[:, 1:]
        res = {"density": self.density_activation(raw) * selector[:, None]}
        if return_feat:
            res["base_mlp_out"] = (torch.cat([base_out, time_encode], -1)
                                   if self.use_time_embedding and not self.time_inject_before_sigma else base_out)
        if return_interal:
            io = {"move": move}
            if self.use_feat_predict or self.use_weight_predict:
                tf = torch.cat([x_move, t.view(-1, 1)], -1)
                io["selector"] = selector
                if self.use_feat_predict:
                    io["latent_losses"] = F.huber_loss(self.mlp_feat_prediction(tf).float(), hash_feat.float(),
                                                       reduction="none") * selector[:, None]
                if self.use_weight_predict:
                    io["weight_losses"] = self.mlp_weight_prediction(tf)
            res["interal_output"] = io
        return res

    def _query_rgb(self, dirs, embedding, apply_act: bool = True):
        emb = embedding.reshape(-1, self.geo_feat_dim_head)
        if self.use_viewdirs:
            dirs = dirs / torch.linalg.norm(dirs, dim=-1, keepdims=True)
            d = self.direction_encoding(((dirs + 1.0) / 2.0).reshape(-1, 3))
            h = torch.cat([d, emb.to(d.dtype)], -1)
        else:
            h = emb
        rgb = self.mlp_head(h).float()
        return torch.sigmoid(rgb) if apply_act else rgb

    def forward(self, positions, t, directions=None):
        res = self.query_density(positions, t, return_feat=True, return_interal=self.training)
        return self._query_rgb(directions, res["base_mlp_out"]), res
