"""The torch restatement of the reference's Net that ModelWrapper serves for geometries the CUDA tower does not compile
(connect4_b200/neural/torch_model.py), and the choice between the two backends.  CPU only."""
import ctypes

import pytest

from conftest import golden


def lively_state(filters, residuals, fc, seed=None):
    """a freshly initialised state dict with weights and batch-norm statistics perturbed so that the activations are far
    from the near-constant outputs of a fresh initialisation (the perturbation of test_gpu_net's geometry test; towers deeper
    than 6 blocks get smaller residual weights, or the value head saturates)"""
    import torch
    from connect4_b200.neural.config import NetConfig
    from connect4_b200.neural.model import _init_state_dict
    torch.manual_seed(filters + residuals if seed is None else seed)
    sd = _init_state_dict(NetConfig(filters=filters, n_fc_layers=fc, n_residuals=residuals))
    gen = torch.Generator().manual_seed(7)
    for k, v in sd.items():
        if k.endswith("running_var"):
            v.copy_(0.5 + torch.rand(v.shape, generator=gen))
        elif k.endswith("running_mean"):
            v.copy_(0.2 * torch.randn(v.shape, generator=gen))
        elif "batch_norm" in k and k.endswith("weight") or (k.startswith("body.0.1") and k.endswith("weight")):
            v.copy_(0.6 + 0.8 * torch.rand(v.shape, generator=gen))
        elif "batch_norm" in k and k.endswith("bias") or (k.startswith("body.0.1") and k.endswith("bias")):
            v.copy_(0.2 * torch.randn(v.shape, generator=gen))
        elif "conv" in k and k.endswith("weight") or k == "body.0.0.weight":
            v.mul_(0.8 if k.startswith("body.1.") and residuals > 6 else 2.0)
        elif ".fc" in k and k.endswith("weight"):
            v.mul_(2.5)
    return sd


@pytest.mark.parametrize("filters,residuals,fc", [(32, 3, 4), (64, 6, 6), (16, 1, 1), (48, 10, 2), (128, 2, 1)])
def test_torch_net_equals_the_fp32_restatement(filters, residuals, fc):
    import torch
    from oracle import net_ref as nr
    from connect4_b200.neural.torch_model import TorchNet
    g = golden("net_outputs.npz")
    sd = lively_state(filters, residuals, fc)
    x = torch.as_tensor(nr.planes_from_bitboards(g["c0"][:512], g["c1"][:512]))
    with torch.no_grad():
        rv, rp = nr.forward_state({k: v.numpy() for k, v in sd.items()}, x)
        v, p = TorchNet(sd)(x)
    assert v.dtype == torch.float32 and p.dtype == torch.float32 and v.shape == (512,) and p.shape == (512, 7)
    assert rv.std() > 0.003 and rp.std() > 0.01                      # the positions really are told apart
    assert (v - rv).abs().max() < 1e-6 and (p - rp).abs().max() < 1e-6


def test_backend_is_cuda_exactly_where_the_library_compiles_the_network():
    """compiled_geometry against c4_net_create itself: the library refuses a geometry before it looks for a device, so this
    runs without a GPU"""
    import torch
    from connect4_b200 import _build, _lib
    from connect4_b200.neural.config import NetConfig
    from connect4_b200.neural.model import _init_state_dict, compiled_geometry
    from connect4_b200.neural.weights import fold_state_dict
    _build.build()
    lib = _lib.load()
    geometry_refusals = ("filters must be 32 or 64", "n_residuals out of range")
    for filters in (16, 32, 48, 64, 128):
        for residuals in (0, 1, 16, 17):
            torch.manual_seed(0)
            blob = fold_state_dict(_init_state_dict(NetConfig(filters=filters, n_fc_layers=1, n_residuals=residuals)))
            h = ctypes.c_void_p()
            rc = lib.c4_net_create(0, blob.ctypes.data_as(ctypes.c_void_p), blob.size, ctypes.byref(h))
            accepted = rc == 0 or not any(m in lib.c4_last_error().decode() for m in geometry_refusals)
            if rc == 0:
                lib.c4_net_destroy(h)
            assert accepted == compiled_geometry(filters, residuals), (filters, residuals)
            assert compiled_geometry(filters, residuals, "mma")          # a requested kernel is never served by torch


def test_flops_per_position_from_the_shapes():
    from connect4_b200.neural.model import flops_per_position
    assert flops_per_position(32, 3, 4) == 4740876.0                  # c4_net_flops_per_position of the same networks
    assert flops_per_position(64, 6, 6) == 37342620.0
    assert flops_per_position(128, 6, 6) == 2.0 * (42 * 27 * 128 + 12 * 42 * 9 * 128 * 128 + 42 * 128 + 6 * 42 * 42 + 42 +
                                                   84 * 128 + 84 * 7)
