"""One small launch of every kernel family of libb200ot.so, for compute-sanitizer (memcheck / racecheck / synccheck):

    compute-sanitizer --tool memcheck  python tools/sanitize_smoke.py
    compute-sanitizer --tool racecheck python tools/sanitize_smoke.py

Shapes are the smallest that select each code path (big / small tile shapes, ranges mode, tensor-core kernels, 2-D and
3-D grid passes with both tile widths); results are checked against torch so a silent corruption also fails."""
import sys

import torch

sys.path.insert(0, __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__))))
from geomloss_b200 import SamplesLoss, ops, ranges  # noqa: E402
from geomloss_b200.sinkhorn_images import softmin_grid  # noqa: E402

DEV = "cuda:0"
g = torch.Generator().manual_seed(0)


def ref_softmin(eps, x, y, h, p):
    d2 = ((x[:, None, :].double() - y[None, :, :].double()) ** 2).sum(-1)
    C = d2 / 2 if p == 2 else d2.clamp_min(1e-8).sqrt()
    return (-eps * torch.logsumexp(h.double()[None, :] - C / eps, dim=1)).float()


def check(name, got, ref, tol=2e-5):
    err = (got.double().cpu() - ref.double().cpu()).abs().max().item() / max(1.0, ref.abs().max().item())
    print(f"{name}: max err {err:.2e}")
    assert err < tol, name


which = set(sys.argv[1:]) or {"softmin", "ranges", "conv", "tc", "grid", "loss"}
if "ring" in which:
    # the dense kernels with MANY tiles per CTA (B200OT_FORCE_SPLITS=1 in the environment): every stage of the TMA ring
    # is refilled a dozen times — the pattern the N = 1e6 runs live in
    assert __import__("os").environ.get("B200OT_FORCE_SPLITS") == "1", "run with B200OT_FORCE_SPLITS=1"
    x, y, h = torch.rand(4200, 3, generator=g), torch.rand(40000, 3, generator=g), torch.randn(40000, generator=g)
    xg = x.to(DEV).requires_grad_(True)
    out = ops.softmin(0.05, xg, y.to(DEV), h.to(DEV), p=2)
    check("ring_softmin", out, ref_softmin(0.05, x, y, h, 2))
    (gx,) = torch.autograd.grad(out.sum(), xg)
    assert torch.isfinite(gx).all()
    w = torch.rand(40000, generator=g)
    conv = ops.kernel_conv("laplacian", xg, y.to(DEV), w.to(DEV), 0.3)
    assert torch.isfinite(conv).all()
if "softmin" in which:
    for tag, n, m, d, p in (("big", 4200, 4300, 3, 2), ("small", 300, 500, 2, 1), ("big_p1", 4100, 4100, 1, 1),
                            ("d8", 600, 700, 8, 2)):
        x, y, h = torch.rand(n, d, generator=g), torch.rand(m, d, generator=g), torch.randn(m, generator=g)
        xg = x.to(DEV).requires_grad_(True)
        out = ops.softmin(0.05, xg, y.to(DEV), h.to(DEV), p=p)
        check("softmin_" + tag, out, ref_softmin(0.05, x, y, h, p))
        (gx,) = torch.autograd.grad(out.sum(), xg)
        assert torch.isfinite(gx).all()
if "ranges" in which:
    for variant, n, m in ((ranges.SMALL, 900, 700), (ranges.BIG, 2500, 3000)):
        R = 5
        rc = torch.tensor([n // R] * (R - 1) + [n - (R - 1) * (n // R)])
        cc = torch.tensor([m // R] * (R - 1) + [m - (R - 1) * (m // R)])
        keep = torch.rand(R, R, generator=g) < 0.6
        keep[torch.arange(R), torch.arange(R)] = True
        lay = ranges.ColumnLayout(cc.to(DEV))
        prob = ranges.build_problem(keep.to(DEV), rc.to(DEV), lay, variant=variant)
        x, y, h = torch.rand(n, 3, generator=g), torch.rand(m, 3, generator=g), torch.randn(m, generator=g)
        xg = x.to(DEV).requires_grad_(True)
        out = ranges.softmin_ranges(0.05, xg, y.to(DEV), h.to(DEV), None, 0.0, prob)
        mask = keep[torch.repeat_interleave(torch.arange(R), rc)][:, torch.repeat_interleave(torch.arange(R), cc)]
        d2 = ((x[:, None, :].double() - y[None, :, :].double()) ** 2).sum(-1) / 2
        ref = -0.05 * torch.logsumexp((h.double()[None, :] - d2 / 0.05).masked_fill(~mask, -float("inf")), dim=1)
        check(f"ranges_softmin_v{variant}", out, ref.float())
        (gx,) = torch.autograd.grad(out.sum(), xg)
        assert torch.isfinite(gx).all()
        w = torch.rand(m, generator=g)
        conv = ranges.kernel_conv_ranges(0, xg, y.to(DEV), w.to(DEV), 0.2, prob, None)
        refc = ((-d2 / 0.04).exp() * mask) @ w.double()
        check(f"ranges_conv_v{variant}", conv, refc.float())
        (gx,) = torch.autograd.grad(conv.sum(), xg)
        assert torch.isfinite(gx).all()
if "conv" in which:
    for kind in ("gaussian", "laplacian", "energy"):
        x, y, w = torch.rand(4200, 3, generator=g), torch.rand(4100, 3, generator=g), torch.rand(4100, generator=g)
        xg = x.to(DEV).requires_grad_(True)
        out = ops.kernel_conv(kind, xg, y.to(DEV), w.to(DEV), 0.3)
        d2 = ((x[:, None, :].double() - y[None, :, :].double()) ** 2).sum(-1)
        K = {"gaussian": (-d2 / 0.18).exp(), "laplacian": (-(d2 / 0.09).clamp_min(1e-8).sqrt()).exp(),
             "energy": -d2.clamp_min(1e-8).sqrt()}[kind]
        check("conv_" + kind, out, (K @ w.double()).float(), 5e-5)
        (gx,) = torch.autograd.grad(out.sum(), xg)
        assert torch.isfinite(gx).all()
if "tc" in which:
    for d in (16, 64):
        x, y, w = torch.rand(700, d, generator=g), torch.rand(900, d, generator=g), torch.rand(900, generator=g)
        xg = x.to(DEV).requires_grad_(True)
        out = ops.kernel_conv("gaussian", xg, y.to(DEV), w.to(DEV), 2.0)
        d2 = ((x[:, None, :].double() - y[None, :, :].double()) ** 2).sum(-1)
        check(f"tc_conv_d{d}", out, ((-d2 / 8.0).exp() @ w.double()).float(), 1e-4)
        (gx,) = torch.autograd.grad(out.sum(), xg)
        assert torch.isfinite(gx).all()
        h = torch.randn(900, generator=g)
        sm = ops.softmin(1.0, xg, y.to(DEV), h.to(DEV), p=2)
        check(f"tc_softmin_d{d}", sm, ref_softmin(1.0, x, y, h, 2), 1e-4)
        (gx,) = torch.autograd.grad(sm.sum(), xg)
        assert torch.isfinite(gx).all()
        # laplacian / energy (MODE 4 / 5 of the forward and row-gradient kernels), cross and self (x is y)
        for kind in ("laplacian", "energy"):
            K = {"laplacian": (-(d2 / 4.0).clamp_min(1e-8).sqrt()).exp(), "energy": -d2.clamp_min(1e-8).sqrt()}[kind]
            out = ops.kernel_conv(kind, xg, y.to(DEV), w.to(DEV), 2.0)
            check(f"tc_conv_{kind}_d{d}", out, (K @ w.double()).float(), 1e-4)
            (gx,) = torch.autograd.grad(out.sum(), xg)
            assert torch.isfinite(gx).all()
            out = ops.kernel_conv(kind, xg, xg.detach(), w[:700].to(DEV), 2.0)
            (gx,) = torch.autograd.grad(out.sum(), xg)
            assert torch.isfinite(out).all() and torch.isfinite(gx).all()
if "grid" in which:
    for shape in ((1, 2, 32, 32), (1, 1, 16, 16, 16), (1, 1, 1024, 1024)):
        h = torch.randn(*shape, generator=g)
        out = softmin_grid(0.01, 2, h.to(DEV))
        assert torch.isfinite(out).all()
        print("grid", shape, "ok")
if "loss" in which:
    x, y = torch.rand(3, 300, 3, generator=g).to(DEV), torch.rand(3, 200, 3, generator=g).to(DEV)
    v = SamplesLoss("sinkhorn", blur=0.1)(x.requires_grad_(True), y)
    v.sum().backward()
    print("batched sinkhorn", v.tolist())
    v = SamplesLoss("sinkhorn", blur=0.1, reach=0.5, debias=False)(x.detach().requires_grad_(True), y)
    v.sum().backward()
    print("batched unbalanced sinkhorn (small-problem kernels: iteration, cost, backward)", v.tolist())
    v = SamplesLoss("gaussian", blur=0.1)(x.detach().requires_grad_(True), y)
    v.sum().backward()
    print("batched gaussian (fused MMD + value kernel)", v.tolist())
    big = torch.rand(100000, 3, generator=g).to(DEV)
    for _ in range(2):  # many CTAs: partial boxes + last-block fold, ticket counter re-used
        lh = ops.cloud_extent(big, big[:777])
    assert torch.equal(lh[0], big.min(0).values) and torch.equal(lh[1], big.max(0).values)
    print("cloud_extent ok")
    v = SamplesLoss("sinkhorn", blur=0.05, backend="multiscale", cluster_scale=0.2, truncate=2)(x[0], y[0])
    print("multiscale sinkhorn", v.item())
    v = SamplesLoss("gaussian", blur=0.1, backend="multiscale", truncate=2)(x[0], y[0])
    print("multiscale gaussian", v.item())
torch.cuda.synchronize()
print("sanitize_smoke: all launches completed")
