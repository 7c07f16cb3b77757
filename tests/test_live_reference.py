"""The CUDA engine against the unmodified reference on fresh random inputs (not the committed fixtures).

The reference (jeanfeydy/geomloss @ 00e493f) was run on the CPU by ``tests/golden/make_golden_live.py``: its
tensorized backend as is, its pykeops-backed backends (online / multiscale / images) on ``tests/golden/pykeops_shim``.
Its fp64 outputs are stored in ``tests/golden/live_reference.npz``; the inputs are not stored but regenerated here
from their seeds, and checked against stored checksums.  Gradients are stored for a fixed sample of 512 rows per
tensor (in fp32), with the largest entry of the full fp64 gradient as the tolerance scale.  Tolerances as in
tests/test_gpu_reference_goldens.py, against the reference's fp64 run.
"""
import numpy as np
import pytest
import torch

from conftest import load_golden

DEV = "cuda:0"


@pytest.fixture(scope="module")
def ref():
    return load_golden("live_reference")


def _clouds(seed, n, m, d):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, d, generator=g, dtype=torch.float64)
    y = torch.rand(m, d, generator=g, dtype=torch.float64) * 0.8 + 0.2
    a = torch.rand(n, generator=g, dtype=torch.float64) + 0.2
    b = torch.rand(m, generator=g, dtype=torch.float64) + 0.2
    return a / a.sum(), x, b / b.sum(), y


def _image_pair():
    g = torch.Generator().manual_seed(11)
    a = torch.rand(1, 2, 32, 32, generator=g, dtype=torch.float64) ** 2
    b = torch.rand(1, 2, 32, 32, generator=g, dtype=torch.float64) ** 2
    return a / a.sum(), 1.2 * b / b.sum()


def _checksum(tensors):
    return np.array([float(t.sum()) for t in tensors] + [float((t * t).sum()) for t in tensors])


def test_stored_reference_run_reproduces_a_committed_fixture(ref):
    """The stored reference run is the code that generated tests/golden: bit-for-bit on cfg1 (fp32 run)."""
    want = float(load_golden("cfg1_sinkhorn_n1000")["value_f32"])
    assert float(ref["cfg1_value_f32"]) == pytest.approx(want, rel=1e-6)


CASES = [
    ("tensorized", dict(loss="sinkhorn", p=2, blur=0.05), 3),
    ("tensorized", dict(loss="sinkhorn", p=1, blur=0.05, reach=0.4), 2),
    ("online", dict(loss="sinkhorn", p=1, blur=0.05), 3),
    ("multiscale", dict(loss="sinkhorn", p=2, blur=0.03, truncate=1, cluster_scale=0.1), 3),
    ("multiscale", dict(loss="sinkhorn", p=2, blur=0.05, reach=0.5, truncate=3), 2),
    ("tensorized", dict(loss="gaussian", blur=0.2), 3),
    ("online", dict(loss="laplacian", blur=0.2), 3),
    ("multiscale", dict(loss="gaussian", blur=0.1, truncate=2), 3),
    ("tensorized", dict(loss="energy"), 5),
]
IMAGE_KWARGS = (dict(p=2, reach=0.4), dict(p=1, blur=0.06, scaling=0.6))


def case_inputs(backend, kw, d):
    return _clouds(sum(map(ord, backend + kw["loss"])) + d, 1700, 1500, d)


def case_key(backend, kw, d):
    return f"{backend}_{'_'.join(f'{k}{v}' for k, v in kw.items())}_d{d}"


def test_regenerated_inputs_match_the_reference_run(ref):
    for backend, kw, d in CASES:
        key = case_key(backend, kw, d)
        np.testing.assert_allclose(_checksum(case_inputs(backend, kw, d)), ref[key + "_inputs"], rtol=1e-12,
                                   err_msg=key)
    np.testing.assert_allclose(_checksum(_image_pair()), ref["images_inputs"], rtol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("backend,kw,d", CASES)
def test_samples_loss_vs_live_reference(ref, backend, kw, d, sinkhorn_path):
    from geomloss_b200 import SamplesLoss

    key = case_key(backend, kw, d)
    a, x, b, y = case_inputs(backend, kw, d)
    dl = [t.float().to(DEV).requires_grad_(True) for t in (a, x, b, y)]
    got = SamplesLoss(backend=backend, **kw)(*dl)
    got_g = torch.autograd.grad(got.sum(), dl)
    want = ref[key + "_value"]
    assert tuple(got.shape) == want.shape
    slack = 3e-7 * float((a.sum() ** 2 + b.sum() ** 2) / 2) if kw["loss"] != "sinkhorn" else 0.0
    assert abs(got.sum().item() - want.sum()) <= 1e-4 * abs(want.sum()) + slack
    for gg, t, name in zip(got_g, (a, x, b, y), "axby"):
        assert gg.shape == t.shape
        rows = torch.from_numpy(ref[key + ("_rows_x" if name in "ax" else "_rows_y")].astype(np.int64))
        want_rows = torch.from_numpy(ref[f"{key}_grad_{name}_rows"]).double()
        err = (gg.cpu().double()[rows] - want_rows).abs().max().item()
        assert err <= 5e-4 * float(ref[f"{key}_grad_{name}_absmax"]) + 1e-12, name


@pytest.mark.gpu
def test_image_divergence_vs_live_reference(ref):
    from geomloss_b200 import sinkhorn_divergence

    a, b = _image_pair()
    for i, kw in enumerate(IMAGE_KWARGS):
        got = sinkhorn_divergence(a.float().to(DEV), b.float().to(DEV), **kw)
        np.testing.assert_allclose(got.cpu().double().numpy(), ref[f"images_{i}_value"], rtol=1e-4)
