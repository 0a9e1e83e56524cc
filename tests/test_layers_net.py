"""Kernel "layers" (connect4_b200/csrc/c4_layers.cu): the geometry check of c4_net_create.  The library checks a blob's
geometry before it looks for a device, so this runs without a GPU."""
import ctypes

import pytest


def _create(filters, residuals, kernel):
    import torch
    from connect4_b200 import _lib
    from connect4_b200.neural.config import NetConfig
    from connect4_b200.neural.model import _init_state_dict
    from connect4_b200.neural.weights import fold_state_dict
    lib = _lib.load()
    torch.manual_seed(0)
    blob = fold_state_dict(_init_state_dict(NetConfig(filters=filters, n_fc_layers=1, n_residuals=residuals)),
                           kernel=kernel)
    h = ctypes.c_void_p()
    rc = lib.c4_net_create(0, blob.ctypes.data_as(ctypes.c_void_p), blob.size, ctypes.byref(h))
    if rc == 0:
        lib.c4_net_destroy(h)
    return rc, lib.c4_last_error().decode()


LAYER_LIMITS = ("the layered kernels need filters a multiple of 16 in 16..256", "the layered kernels need n_residuals in 1..40")


@pytest.fixture(scope="module", autouse=True)
def _built():
    from connect4_b200 import _build
    _build.build()


@pytest.mark.parametrize("filters", [16, 48, 96, 128, 256])
@pytest.mark.parametrize("residuals", [1, 40])
def test_layers_accepts_every_multiple_of_16_up_to_256(filters, residuals):
    rc, err = _create(filters, residuals, "layers")
    assert rc == 0 or not any(m in err for m in LAYER_LIMITS), err


@pytest.mark.parametrize("filters,residuals,message", [(8, 1, 0), (100, 1, 0), (272, 1, 0), (64, 0, 1), (64, 41, 1)])
def test_layers_refuses_other_geometries_before_looking_for_a_device(filters, residuals, message):
    rc, err = _create(filters, residuals, "layers")
    assert rc == -1 and LAYER_LIMITS[message] in err, err


@pytest.mark.parametrize("kernel", ["auto", "mma"])
@pytest.mark.parametrize("filters,residuals,message", [(8, 1, "filters must be 32 or 64"),
                                                        (100, 1, "filters must be 32 or 64"),
                                                        (272, 1, "filters must be 32 or 64"),
                                                        (128, 2, "filters must be 32 or 64"),
                                                        (64, 0, "n_residuals out of range"),
                                                        (64, 17, "n_residuals out of range"),
                                                        (64, 41, "n_residuals out of range")])
def test_tower_kernels_keep_their_refusals(kernel, filters, residuals, message):
    rc, err = _create(filters, residuals, kernel)
    assert rc == -1 and err == "invalid argument: c4_net_create: " + message, err
