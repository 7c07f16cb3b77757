"""Laplacian and energy kernel convolutions for 8 < D <= 64 (tensor-core path), checked without a GPU: the C ABI
accepts them (argument validation runs before any CUDA call), and the CPU oracle reproduces the reference fixtures
tests/golden/hdsqrt_*.npz (make_golden_highdim_sqrt.py) in fp64."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import golden_kwargs, golden_names, load_golden
from geomloss_b200 import _lib
from oracle import geomloss_oracle as O

LAPLACIAN, ENERGY, UNCLAMPED = 1, 2, 0x100


@pytest.fixture(scope="module")
def L():
    return _lib.lib()


@pytest.mark.parametrize("kind", [LAPLACIAN, ENERGY, LAPLACIAN | UNCLAMPED, ENERGY | UNCLAMPED])
def test_sqrt_kernels_are_accepted_above_eight_dimensions(L, kind):
    """D = 16 passes the argument checks and reaches the scratch-size check (ESCRATCH with 16 bytes of scratch)."""
    null, fake = ctypes.c_void_p(None), ctypes.c_void_p(0x1000)
    assert L.b200ot_kernel_conv_fwd(fake, fake, fake, null, fake, 1000, 1000, 16, kind, 0.5, fake, 16, null) == -2
    assert L.b200ot_kernel_conv_bwd_x(fake, fake, fake, null, fake, fake, 1000, 1000, 16, kind, 0.5, fake, 16,
                                      null) == -2
    # D = 65 has no kernel; the one-pass value + gradient entry stays gaussian-only
    assert L.b200ot_kernel_conv_fwd(fake, fake, fake, null, fake, 1000, 1000, 65, kind, 0.5, fake, 1 << 30,
                                    null) == -1
    assert L.b200ot_kernel_conv_bwd_x(fake, fake, fake, null, fake, fake, 1000, 1000, 65, kind, 0.5, fake, 1 << 30,
                                      null) == -1
    assert L.b200ot_kernel_conv_fwd_bwd_x(fake, fake, fake, null, fake, fake, 1000, 1000, 16, kind, 0.5, fake, 1 << 30,
                                          null) == -1


def test_sqrt_kernels_still_validate_blur_and_flags(L):
    null, fake = ctypes.c_void_p(None), ctypes.c_void_p(0x1000)
    assert L.b200ot_kernel_conv_fwd(fake, fake, fake, null, fake, 1000, 1000, 16, LAPLACIAN, 0.0, fake, 16, null) == -1
    assert L.b200ot_kernel_conv_fwd(fake, fake, fake, null, fake, 1000, 1000, 16, ENERGY | 0x200, 0.5, fake, 16,
                                    null) == -1
    # energy has no length scale: any blur
    assert L.b200ot_kernel_conv_fwd(fake, fake, fake, null, fake, 1000, 1000, 16, ENERGY, 0.0, fake, 16, null) == -2


def test_scratch_size_is_kind_independent_above_eight_dimensions(L):
    """One size query serves every kind: the tensor-core plan of the shape (its misc block holds the coordinate scale
    of the laplacian / energy kernels next to max|w|)."""
    for D in (9, 16, 33, 64):
        assert L.b200ot_kernel_conv_scratch_bytes(1000, 1500, D) == L.b200ot_softmin_scratch_bytes(1000, 1500, D) > 0


@pytest.mark.parametrize("name", golden_names("hdsqrt_"))
def test_oracle_reproduces_highdim_sqrt_fixtures(name):
    g = load_golden(name)
    kw = golden_kwargs(g)
    leaves = [torch.from_numpy(g[k]).double().requires_grad_(True) for k in "axby"]
    val = O.samples_loss(*leaves, **kw)
    np.testing.assert_allclose(val.item(), g["value_f64"], rtol=1e-11)
    ga, gx, gb, gy = torch.autograd.grad(val, leaves)
    np.testing.assert_allclose(ga.numpy(), g["grad_a_f64"], rtol=1e-9, atol=1e-14)
    np.testing.assert_allclose(gb.numpy(), g["grad_b_f64"], rtol=1e-9, atol=1e-14)
    # (point gradients are stored as float32)
    for got, key in ((gx, "grad_x_f64"), (gy, "grad_y_f64")):
        np.testing.assert_allclose(got.numpy(), g[key], rtol=2e-6, atol=1e-7 * np.abs(g[key]).max())


def test_fixture_prefix_stays_out_of_the_gaussian_tests():
    assert not set(golden_names("hd_")) & set(golden_names("hdsqrt_"))
