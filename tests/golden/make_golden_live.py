"""Golden data of tests/test_live_reference.py: the reference's fp64 outputs on the test's seeded inputs.

    python tests/golden/make_golden_live.py <reference source dir, the one that holds geomloss/>

The UNMODIFIED reference (jeanfeydy/geomloss @ 00e493f) is imported with ``tests/golden/pykeops_shim`` first on
``sys.path`` (its pykeops-backed backends run on the shim's dense torch stand-in).  The cases and their input
generators are the test module's own; for each case this stores the value, a fixed sample of 512 gradient rows per
input tensor (rounded to fp32, far below the test's 5e-4 bar) with the largest entry of the full gradient, and input
checksums (the inputs themselves are regenerated from their seeds by the test).  Writes
tests/golden/live_reference.npz.
"""
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
if len(sys.argv) != 2:
    raise SystemExit(__doc__)
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, os.path.join(HERE, "pykeops_shim"))
sys.path.insert(0, os.path.dirname(HERE))
import pykeops  # noqa: E402

assert pykeops.__version__.startswith("shim"), "the dense pykeops shim must shadow any real pykeops"
import geomloss  # noqa: E402
from test_live_reference import CASES, IMAGE_KWARGS, _checksum, _image_pair, case_inputs, case_key  # noqa: E402

ROWS = 512


def main():
    out = {}
    with np.load(os.path.join(HERE, "cfg1_sinkhorn_n1000.npz")) as g:
        x, y = torch.from_numpy(g["x"]), torch.from_numpy(g["y"])
    rng = np.random.default_rng(0)
    out["cfg1_value_f32"] = np.array(geomloss.SamplesLoss("sinkhorn", p=2, blur=0.05, backend="tensorized")(x, y).item())
    for backend, kw, d in CASES:
        key = case_key(backend, kw, d)
        a, x, b, y = case_inputs(backend, kw, d)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            leaves = [t.clone().requires_grad_(True) for t in (a, x, b, y)]
            want = geomloss.SamplesLoss(backend=backend, **kw)(*leaves)
            grads = torch.autograd.grad(want.sum(), leaves)
        rows = {"x": np.sort(rng.choice(x.shape[0], ROWS, replace=False)).astype(np.int16),
                "y": np.sort(rng.choice(y.shape[0], ROWS, replace=False)).astype(np.int16)}
        out[key + "_inputs"] = _checksum((a, x, b, y))
        out[key + "_value"] = want.detach().numpy()
        out[key + "_rows_x"], out[key + "_rows_y"] = rows["x"], rows["y"]
        for name, gr in zip("axby", grads):
            out[f"{key}_grad_{name}_rows"] = gr.numpy()[rows["x" if name in "ax" else "y"]].astype(np.float32)
            out[f"{key}_grad_{name}_absmax"] = np.array(gr.abs().max().item())
        print(f"{key}: value {want.sum().item():.12e}")
    a, b = _image_pair()
    out["images_inputs"] = _checksum((a, b))
    for i, kw in enumerate(IMAGE_KWARGS):
        out[f"images_{i}_value"] = geomloss.sinkhorn_divergence(a, b, **kw).numpy()
        print(f"images {kw}: {out[f'images_{i}_value']}")
    path = os.path.join(HERE, "live_reference.npz")
    np.savez_compressed(path, **out)
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
