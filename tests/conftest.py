import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def reference_tables(aabb, field_kwargs):
    """The four tiny-cuda-nn parameter tables of the reference's initial DNGPradianceField, restated with the oracle's
    initialisers: the reference builds every module with tcnn's default seed, 1337, and make_golden.boost_density scales
    the hash table by 5000 and the density MLP by 3."""
    import torch

    from oracle import cednerf_ref as cr
    from oracle import tcnn_ref as tc

    f = cr.DNGPradianceField(aabb, **field_kwargs)
    mlp = lambda n: tc.mlp_init_params(n.n_input_dims, n.n_output_dims, n.n_neurons, n.n_hidden,
                                       torch.Generator().manual_seed(1337))
    table = tc.Encoding(f.hash_encoder.n_input_dims, f.hash_encoder.cfg, 1337).params.detach()
    return {"xyz_wrap.params": mlp(f.xyz_wrap.network), "hash_encoder.params": table * 5000.0,
            "mlp_base.params": mlp(f.mlp_base) * 3.0, "mlp_head.params": mlp(f.mlp_head)}


class Golden(dict):
    """tests/golden/reference_path.pt with every state dict whole again (see make_golden.compact)."""

    def grads(self, prefix, module):
        """(parameter name, computed, frozen) for every gradient of `module` frozen under `prefix`: whole tensors, and
        for a hash-grid gradient its entries at the stored sample positions plus its L2 norm in float64."""
        for k, p in module.named_parameters():
            key = f"{prefix}.grad.{k}"
            if key in self:
                yield k, p.grad, self[key]
            elif key + ".sample" in self:
                g = p.grad.flatten()
                yield k, g[self["grad_sample_index"].long().to(g.device)], self[key + ".sample"]
                yield k, g.double().norm(), self[key + ".norm"]


@pytest.fixture(scope="session")
def golden():
    import torch

    g = Golden(torch.load(os.path.join(ROOT, "tests", "golden", "reference_path.pt"), map_location="cpu"))
    for name in [k[:-len(".field_kwargs")] for k in g if k.endswith(".field_kwargs")]:
        for k, v in reference_tables(g["scene.aabbs"][-1], g[f"{name}.field_kwargs"]).items():
            assert torch.equal(v.double().sum(), g.pop(f"{name}.state_sum.{k}")), (name, k)
            g[f"{name}.state.{k}"] = v
    return g
