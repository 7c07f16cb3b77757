"""Rates of the tensor-core kernel convolutions above eight dimensions: laplacian and energy next to the gaussian
(the baseline, same run), forward and row gradients, plus SamplesLoss("energy") forward + backward and a sampled-row
fp64 check at the timed size.  One JSON object per line on stdout (and in --out).

    python tools/bench_sqrt_conv.py [--n 1000000] [--dims 16 64] [--out FILE]

Timing: CUDA events around each call, best of --reps after one warm-up call; a 256 MB buffer is overwritten
between timed calls so that no operand image is served from the 126 MB L2.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from geomloss_b200 import SamplesLoss, ops  # noqa: E402

DEV = "cuda:0"


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def timed(fn, reps, flush):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / 1e3)
    return min(ts), ts


def sampled_rows_fp64(name, x, y, w, blur, rows, go):
    """(out, grad) in fp64 for the sampled rows, tensorized convention, explicit differences."""
    xs = x[rows].double()
    out = torch.zeros(len(rows), dtype=torch.float64, device=DEV)
    grad = torch.zeros_like(xs)
    for j0 in range(0, y.shape[0], 8192):
        diff = xs[:, None, :] - y[None, j0:j0 + 8192].double()
        d2 = (diff * diff).sum(-1)
        wj = w[j0:j0 + 8192].double()
        if name == "energy":
            r = d2.clamp_min(1e-8).sqrt()
            k, c = -r, torch.where(d2 > 1e-8, -1.0 / r, torch.zeros_like(r))
        else:
            q = d2 / blur**2
            rb = q.clamp_min(1e-8).sqrt()
            k = torch.exp(-rb)
            c = torch.where(q > 1e-8, -k / (blur * blur * rb), torch.zeros_like(rb))
        out += k @ wj
        grad += ((c * wj)[:, :, None] * diff).sum(1)
    return out, grad * go[rows].double()[:, None]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--dims", type=int, nargs="+", default=[16, 64])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def emit(rec):
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    emit({"what": "device", **gpu_info(), "time": time.strftime("%Y-%m-%d %H:%M:%S")})
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    n = args.n
    for D in args.dims:
        g = torch.Generator(device=DEV).manual_seed(D)
        x = torch.rand(n, D, generator=g, device=DEV)
        y = torch.rand(n, D, generator=g, device=DEV) * 0.9 + 0.15
        w = torch.rand(n, generator=g, device=DEV) / n
        go = torch.randn(n, generator=g, device=DEV)
        c = ops.default_center(x, y)
        rows = torch.randint(0, n, (64,), generator=g, device=DEV)
        for kind in ("gaussian", "laplacian", "energy"):
            blur = 2.0
            box = {}

            def fwd():
                box["out"] = ops.kernel_conv_raw(kind, x, y, w, blur, center=c)

            def bwd():
                box["gx"] = ops.kernel_conv_grad_rows(kind, x, y, w, blur, go, center=c)

            tf, tfs = timed(fwd, args.reps, flush)
            tb, tbs = timed(bwd, args.reps, flush)
            rec = {"what": "operator", "kind": kind, "N": n, "M": n, "D": D, "blur": blur,
                   "fwd_s": tf, "fwd_pairs_per_s": n * n / tf, "bwd_s": tb, "bwd_pairs_per_s": n * n / tb,
                   "fwd_all_s": tfs, "bwd_all_s": tbs}
            if kind != "gaussian":
                ref, gref = sampled_rows_fp64(kind, x, y, w, blur, rows, go)
                mag = ref.abs().max().item()
                rec["fwd_rows_max_err_rel"] = (box["out"][rows].double() - ref).abs().max().item() / mag
                rec["bwd_rows_max_err_rel"] = ((box["gx"][rows].double() - gref).abs().max().item()
                                               / gref.abs().max().item())
            emit(rec)
        del x, y, w, go

    # SamplesLoss("energy") forward + backward, N = M = 1e6, D = 64 (BASELINE configs[2] shape), gradient w.r.t. x
    g = torch.Generator(device=DEV).manual_seed(2)
    x = torch.rand(n, 64, generator=g, device=DEV)
    y = torch.rand(n, 64, generator=g, device=DEV)
    L = SamplesLoss("energy")

    def loss_step():
        xg = x.clone().requires_grad_(True)
        v = L(xg, y)
        v.backward()
        return v

    for _ in range(1):
        loss_step()
    torch.cuda.synchronize()
    ts = []
    for _ in range(2):
        t0 = time.perf_counter()
        v = loss_step()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    emit({"what": "samples_loss", "loss": "energy", "N": n, "M": n, "D": 64, "fwd_bwd_s": min(ts), "all_s": ts,
          "value": v.item()})
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
