"""Golden fixtures for the laplacian and energy kernel MMDs in dimensions 16 to 64 (the tensor-core kernels) from the
REAL reference's tensorized backend.

    python tests/golden/make_golden_highdim_sqrt.py

Imports geomloss from /root/reference/src (commit 00e493f); fp32 and fp64 runs of
SamplesLoss("energy" | "laplacian", backend="tensorized") with autograd gradients.  The laplacian blur = .3, D = 64
case is dominated by the diagonal of K_xx and K_yy (exp(-|x - y| / blur) ~ e^-10 off the diagonal).  The file prefix
is hdsqrt_: the hd_ fixtures are the gaussian / sinkhorn ones, with their own tests.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.environ.get("GEOMLOSS_REFERENCE", "/root/reference/src"))
from geomloss import SamplesLoss  # noqa: E402

torch.set_num_threads(8)


def npy(t):
    return t.detach().cpu().numpy()


CASES = [
    ("hdsqrt_energy_d16", 61, 700, 600, 16, dict(loss="energy")),
    ("hdsqrt_energy_d33", 62, 500, 450, 33, dict(loss="energy")),
    ("hdsqrt_energy_d64", 63, 600, 650, 64, dict(loss="energy")),
    ("hdsqrt_laplacian_d16_blur1", 64, 700, 600, 16, dict(loss="laplacian", blur=1.0)),
    ("hdsqrt_laplacian_d64_blur2", 65, 600, 650, 64, dict(loss="laplacian", blur=2.0)),
    ("hdsqrt_laplacian_d64_blur03", 66, 600, 650, 64, dict(loss="laplacian", blur=0.3)),
]


def main():
    for name, seed, n, m, d, kw in CASES:
        g = torch.Generator().manual_seed(seed)
        # fp32-representable inputs: the fp64 run of the reference sees exactly the same numbers (x.double())
        x = torch.rand(n, d, generator=g)
        y = torch.rand(m, d, generator=g) * 0.9 + 0.15
        a = torch.rand(n, generator=g) + 0.1
        b = torch.rand(m, generator=g) + 0.1
        a, b = a / a.sum(), b / b.sum()
        arrays = dict(a=npy(a), x=npy(x), b=npy(b), y=npy(y))
        for k, v in kw.items():
            arrays["kw_" + k] = np.array(v)
        for dtype, suf in ((torch.float32, ""), (torch.float64, "_f64")):
            leaves = [t.to(dtype).requires_grad_(True) for t in (a, x, b, y)]
            val = SamplesLoss(backend="tensorized", **kw)(*leaves)
            ga, gx, gb, gy = torch.autograd.grad(val, leaves)
            arrays.update({"value" + suf: npy(val), "grad_a" + suf: npy(ga), "grad_b" + suf: npy(gb)})
            if suf:  # point gradients: the fp64 run only (stored as float32)
                arrays.update({"grad_x" + suf: npy(gx).astype(np.float32), "grad_y" + suf: npy(gy).astype(np.float32)})
            else:
                gx32 = npy(gx)
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **arrays)
        gx_err = np.abs(gx32 - arrays["grad_x_f64"]).max() / np.abs(arrays["grad_x_f64"]).max()
        print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB value fp32 {arrays['value']} fp64 {arrays['value_f64']}"
              f" fp32 run's grad_x error {gx_err:.2e} of max")


if __name__ == "__main__":
    main()
