#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native Sinkhorn engine (contract: see DESIGN.md section 6).

Metric (BASELINE.json): Sinkhorn N x M pair-interactions / second, N = M = 1e6, D = 3, p = 2, blur = .01
(configs[1]).  One pair-interaction = one evaluation of exp(h_j - C(x_i, y_j)/eps) accumulated into row i.

A "step" is ONE symmetric Sinkhorn iteration at the final temperature eps = blur^2 on the full clouds:
the four softmins  xy, yx, xx, yy  with the fused  h = log_w + pot/eps  prologue and  1/2 (f + f~)
epilogue (src/geomloss/_legacy/sinkhorn_divergence.py:468-493 of the reference) = 2NM + N^2 + M^2 pairs.
A full loss of configs[1] is 53 such iteration-equivalents (212 softmins); the instruction stream does
not depend on eps, so the step rate is the loss rate.

    python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA, libb200ot.so)
    python bench.py --impl reference [--steps K] [--warmup W]      the reference's dense CPU algorithm
                                                                   (oracle port) on the host cores

Multi-GPU: one process per GPU (torchrun); the column cloud of every softmin is sharded over the ranks,
one all_gather of (N, 2) partials per softmin (geomloss_b200/distributed.py).  Total work is fixed:
strong scaling.  Timing: CUDA events on the compute stream around every step, L2 flushed between
steps, barrier + synchronize on both sides of the timed region, max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "sinkhorn_pair_interactions_per_second"
UNIT = "pairs/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=1_000_000, help="points per cloud (N = M)")
    ap.add_argument("--blur", type=float, default=0.01)
    ap.add_argument("--e2e-steps", type=int, default=1, help="full SamplesLoss calls timed end to end")
    ap.add_argument("--e2e-scaling", type=float, default=0.9,
                    help="eps-scaling ratio of the end-to-end loss: .9 = BASELINE configs[1]'s '~50 iters' (51 eps values)")
    ap.add_argument("--no-secondary", action="store_true", help="skip BASELINE configs[2..4] (config.secondary)")
    ap.add_argument("--cpu-n", type=int, default=16000, help="cloud size of the bounded CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the potentials of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(out_dir, pots):
    """The four potentials (f_ba, g_ab, f_aa, g_bb) the last timed step returned: 4 (N,) float32 arrays, 16 MB at the
    default N = 1e6.  The inputs are seeded, so two builds run with the same arguments can be compared array by array."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in pots.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy().reshape(-1))


# ----------------------------------------------------------------------------------------------------
# clocks: sample SM clock / throttle reasons DURING the timed region (NVML, 100 ms period)
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int, period: float = 0.1):
        self.period = period
        self.samples, self.reasons, self.power = [], set(), []
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as exc:  # pragma: no cover
            self.nv = None
            self.err = repr(exc)

    _NAMES = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
              0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
              0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self._NAMES.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "no NVML samples"}
        return {"sm_mhz": statistics.median(self.samples), "sm_min_mhz": min(self.samples),
                "sm_max_mhz": self.max_mhz, "power_w_max": round(max(self.power), 1),
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------------
# the reference arm: the reference's dense CPU algorithm (oracle port) on the host cores
# ----------------------------------------------------------------------------------------------------
class _RefOps:
    """softmin_dense / cost_matrix served by the UNMODIFIED reference installed under oracle/_ref (oracle/make_ref.sh):
    softmin_tensorized (sinkhorn_samples.py:32-71) and cost_routines[p] (:26-29)."""

    kind = "reference"

    def __init__(self, ss):
        self.ss = ss

    def cost_matrix(self, x, y, p):
        return self.ss.cost_routines[p](x, y)

    def softmin_dense(self, eps, C, h):
        return self.ss.softmin_tensorized(eps, C, h)


def reference_ops():
    """(ops, kind): the real reference if oracle/_ref is present, else the oracle port."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if os.path.isdir(os.path.join(ref_dir, "geomloss")):
        sys.path.insert(0, ref_dir)
        try:
            from geomloss._legacy import sinkhorn_samples as ss

            if os.path.realpath(ss.__file__).startswith(os.path.realpath(ref_dir)):
                return _RefOps(ss), "reference"
        except Exception:  # pragma: no cover - fall through to the port
            pass
        finally:
            sys.path.remove(ref_dir)
    from oracle import geomloss_oracle as O

    return O, "port"


def dense_iteration_state(n, blur, seed=0):
    import torch

    O, _ = reference_ops()

    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, 3, generator=g)
    y = torch.rand(n, 3, generator=g)
    a_log = torch.full((1, n), -float(torch.log(torch.tensor(float(n)))))
    eps = blur**2
    xb, yb = x[None], y[None]
    C = dict(xy=O.cost_matrix(xb, yb, 2), yx=O.cost_matrix(yb, xb, 2), xx=O.cost_matrix(xb, xb, 2),
             yy=O.cost_matrix(yb, yb, 2))
    pots = {k: O.softmin_dense(eps, C[c], a_log) for k, c in (("f_ba", "xy"), ("g_ab", "yx"), ("f_aa", "xx"),
                                                               ("g_bb", "yy"))}
    return O, eps, a_log, C, pots


def dense_iteration(O, eps, a_log, C, p):
    """One symmetric Sinkhorn iteration of the reference on stored cost matrices (4 dense softmins)."""
    ft_ba = O.softmin_dense(eps, C["xy"], a_log + p["g_ab"] / eps)
    gt_ab = O.softmin_dense(eps, C["yx"], a_log + p["f_ba"] / eps)
    ft_aa = O.softmin_dense(eps, C["xx"], a_log + p["f_aa"] / eps)
    gt_bb = O.softmin_dense(eps, C["yy"], a_log + p["g_bb"] / eps)
    return dict(f_ba=0.5 * (p["f_ba"] + ft_ba), g_ab=0.5 * (p["g_ab"] + gt_ab), f_aa=0.5 * (p["f_aa"] + ft_aa),
                g_bb=0.5 * (p["g_bb"] + gt_bb))


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def run_reference(args):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs and prints the reference line
    # torchrun exports OMP_NUM_THREADS=1 to every rank: the reference arm is entitled to all host threads it can use
    if os.environ.get("OMP_NUM_THREADS") == "1" and "LOCAL_RANK" in os.environ:
        try:
            torch.set_num_threads(len(os.sched_getaffinity(0)))
        except (AttributeError, OSError):
            torch.set_num_threads(os.cpu_count() or 1)
    n = args.cpu_n
    O, eps, a_log, C, pots = dense_iteration_state(n, args.blur)
    with torch.no_grad():
        for _ in range(args.warmup):
            pots = dense_iteration(O, eps, a_log, C, pots)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pots = dense_iteration(O, eps, a_log, C, pots)
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, pots)
    pairs = 4.0 * n * n
    value = pairs * args.steps / dt
    cores = torch.get_num_threads()
    kind = reference_ops()[1]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1] single-scale Sinkhorn, D=3 p=2 blur=%g; step = one symmetric Sinkhorn "
                               "iteration (4 dense softmins on stored N x N cost matrices), bounded sample "
                               "N=M=%d of the N=M=1e6 problem (4 TB per cost matrix at full size)" % (args.blur, n),
                   "N": n, "M": n, "D": 3, "pairs_per_step": pairs},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"N=M={n}, {args.steps} dense Sinkhorn iterations "
                                   f"({'the unmodified reference (oracle/_ref): softmin_tensorized on cost_routines[2] matrices' if kind == 'reference' else 'oracle port of the tensorized path'}), "
                                   f"torch CPU {cores} threads, {cpu_model()}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    from geomloss_b200 import SamplesLoss, _lib, ops
    from geomloss_b200.sinkhorn import epsilon_schedule

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 with torchrun (one rank per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    L = _lib.lib()  # fails loudly if libb200ot.so is missing
    engine = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        from geomloss_b200.distributed import ColumnShardedEngine

        engine = ColumnShardedEngine()
    sm = engine.softmin_raw if engine else ops.softmin_raw

    N = M = args.n
    D, p = 3, 2
    eps = args.blur**2
    g = torch.Generator().manual_seed(0)
    x_h = torch.rand(N, D, generator=g).pin_memory()
    y_h = torch.rand(M, D, generator=g).pin_memory()
    x, y = x_h.to(dev), y_h.to(dev)
    a_log = torch.full((N,), -float(torch.log(torch.tensor(float(N)))), device=dev)
    b_log = torch.full((M,), -float(torch.log(torch.tensor(float(M)))), device=dev)
    center = ops.default_center(x, y)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # potentials: the reference's initialisation at this temperature (sinkhorn_divergence.py:461-465)
    pots = {"f_ba": sm(eps, x, y, b_log, p=p, center=center)[0], "g_ab": sm(eps, y, x, a_log, p=p, center=center)[0],
            "f_aa": sm(eps, x, x, a_log, p=p, center=center)[0], "g_bb": sm(eps, y, y, b_log, p=p, center=center)[0]}
    inv = 1.0 / eps

    from geomloss_b200.sinkhorn import softmin_many

    def step(pt):
        # exactly the body of sinkhorn.sinkhorn_loop_points: four independent (Jacobi) fused updates
        ukw = dict(p=p, center=center, alpha_old=0.5, beta=0.5)
        res = softmin_many(sm, [((eps, x, y, b_log, pt["g_ab"], inv), dict(out_old=pt["f_ba"], **ukw)),
                                ((eps, y, x, a_log, pt["f_ba"], inv), dict(out_old=pt["g_ab"], **ukw)),
                                ((eps, x, x, a_log, pt["f_aa"], inv), dict(out_old=pt["f_aa"], **ukw)),
                                ((eps, y, y, b_log, pt["g_bb"], inv), dict(out_old=pt["g_bb"], **ukw))])
        return {"f_ba": res[0][0], "g_ab": res[1][0], "f_aa": res[2][0], "g_bb": res[3][0]}

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    pairs_per_step = 2.0 * N * M + float(N) * N + float(M) * M
    for _ in range(max(args.warmup, 3)):
        pots = step(pots)
    sync_all()

    # ---- timed region: K steps, per-step CUDA events, L2 flushed between steps ----
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches0 = ops.launches()
    sampler = ClockSampler(local_rank)
    with sampler:
        sync_all()
        for k in range(args.steps):
            flush.zero_()
            ev[k][0].record()
            pots = step(pots)
            ev[k][1].record()
        sync_all()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pots)
    total_ms = torch.tensor([sum(step_ms)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = total_ms.item()
    gpu_launches = ops.launches() - launches0
    value = pairs_per_step * args.steps / (total_ms * 1e-3)
    finite = bool(torch.isfinite(pots["f_ba"]).all().item())

    # ---- dominant kernel alone: staged calls, CUDA events around the partial-reduction launch ----
    kern = kernel_pass(L, ops, torch, dev, x, y, b_log, pots["g_ab"], inv, center, eps, p, flush, reps=max(3, args.steps // 2),
                       world=world, rank=rank)
    # ---- MUFU / FP32 ceilings of this device, measured now ----
    ceil = pipe_ceilings(L, ops, torch, dev)

    # ---- end to end through the public API with host buffers ----
    e2e = None
    if not args.no_e2e:
        # backend="online": the exact, dense reduction — every counted pair-interaction is evaluated
        # (the default "auto" would pick the truncated multiscale scheme at this size, like the reference)
        loss = SamplesLoss("sinkhorn", p=2, blur=args.blur, scaling=args.e2e_scaling, diameter=3**0.5,
                           backend="online")
        if engine:
            engine.attach(loss)
        n_eps = len(epsilon_schedule(2, 3**0.5, args.blur, args.e2e_scaling))
        pairs_loss = (n_eps + 2) * pairs_per_step

        def e2e_call():
            xd = x_h.to(dev, non_blocking=True)
            yd = y_h.to(dev, non_blocking=True)
            return loss(xd, yd).item()  # .item(): device -> host read of the result

        warm = SamplesLoss("sinkhorn", p=2, blur=args.blur, scaling=0.5, diameter=3**0.5, backend="online")
        if engine:
            engine.attach(warm)
        warm(x_h.to(dev, non_blocking=True), y_h.to(dev, non_blocking=True)).item()  # warm-up: the short ladder
        sync_all()
        t0 = time.perf_counter()
        vals = [e2e_call() for _ in range(args.e2e_steps)]
        sync_all()
        dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": pairs_loss * args.e2e_steps / dt.item(), "unit": UNIT,
               "h2d_bytes_per_step": int(x_h.numel() * 4 + y_h.numel() * 4), "d2h_bytes_per_step": 4,
               "call": f"SamplesLoss('sinkhorn', p=2, blur={args.blur}, scaling={args.e2e_scaling}, diameter=sqrt(3), "
                       f"backend='online')"
                       f"(x_host->cuda, y_host->cuda).item(): {n_eps} eps values, {4 * (n_eps + 2)} softmins",
               "s_per_call": dt.item() / args.e2e_steps, "loss_value": vals[-1]}

    # ---- BASELINE configs[2], [3], [4]: own CUDA-event timings + in-run spot parity (config.secondary) ----
    secondary = None
    if not args.no_secondary:
        secondary = secondary_configs(torch, dev, world, rank, engine, peaks_file=os.path.join(ROOT, "MEASURED_PEAKS.json"),
                                      mufu_peak=ceil["mufu_ex2_per_s"])

    # ---- CPU baseline: the oracle port on this box's host cores, bounded sample (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args)

    if rank == 0:
        clocks = sampler.summary()
        mufu_peak = ceil["mufu_ex2_per_s"]
        k_rate = kern["pairs_per_s"]
        traffic = None
        tfile = os.path.join(ROOT, "profiles", "softmin_partial_ncu_summary.json")
        if os.path.exists(tfile):
            try:
                traffic = json.load(open(tfile)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        alg_bytes = 4.0 * ((N + M / world) * (D + 1))  # SURVEY 8(d): compulsory HBM bytes per softmin launch
        peaks = {}
        pfile = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pfile):
            peaks = json.load(open(pfile))
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": "configs[1]: single-scale Sinkhorn N=M=%d D=3 p=2 blur=%g on uniform-in-cube clouds; "
                            "step = one symmetric Sinkhorn iteration = 4 softmins (xy, yx, xx, yy) with fused "
                            "prologue/epilogue" % (N, args.blur),
                "N": N, "M": M, "D": D, "p": p, "blur": args.blur, "pairs_per_step": pairs_per_step,
                "l2": "flushed between timed steps (256 MiB write); inputs (40 MB) are smaller than L2 by nature",
                "parallelism": "single GPU" if world == 1 else f"columns of every softmin sharded x{world}, "
                                                                "1 all_gather of (N,2) fp32 per softmin",
                "finite": finite,
                "secondary": secondary,
            },
            "e2e": e2e,
            "gpu_launches": gpu_launches,
            "clocks": clocks,
            "roofline": {
                "bound": "sfu",
                "kernel": "softmin_partial_kernel (1 MUFU.EX2 per pair, 16-pair chunks between running-max checks, no "
                          "FMA-pipe off-load at D=3; SURVEY.md 8(d): the path is exp-bound, not HBM-bound)",
                "achieved": k_rate / 1e9, "peak": mufu_peak / 1e9, "unit": "Gexp/s", "frac": k_rate / mufu_peak,
                "peak_source": "MUFU.EX2 micro-benchmark (b200ot_ubench) run in this process after the timed region",
                "kernel_ms": kern["ms_per_launch"], "kernel_share_of_step": kern["ms_per_launch"] * 4 / (total_ms / args.steps),
                "fp32": {"achieved_tflops": k_rate * 13 / 1e12, "ffma_peak_tflops": 2 * ceil["ffma_per_s"] / 1e12,
                         "note": "13 flop/pair (SURVEY 8d); FFMA micro-benchmark peak"},
                "hbm": {"algorithmic_bytes_per_launch": alg_bytes, "achieved_gbs": alg_bytes / (kern["ms_per_launch"] * 1e-3) / 1e9,
                        "peak_gbs": hbm_peak, "frac": alg_bytes / (kern["ms_per_launch"] * 1e-3) / 1e9 / hbm_peak,
                        "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"},
                "traffic": traffic,
                "traffic_source": "profiles/softmin_partial_ncu_summary.json (dram__bytes_read.sum + dram__bytes_write.sum "
                                  "of one ncu --set full capture of this kernel at this shape; not re-measured per run)",
            },
            "cpu_baseline": cpu,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()



# ----------------------------------------------------------------------------------------------------
# BASELINE.json configs[2], [3], [4] — reported inside config.secondary of the same JSON line
# ----------------------------------------------------------------------------------------------------
def _ev_time(torch, dev, fn, reps=2, warm=1):
    """Best CUDA-event time (s) of fn over `reps` runs after `warm` warm-ups, plus the last result."""
    out = None
    for _ in range(warm):
        out = fn()
    torch.cuda.synchronize(dev)
    best = None
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize(dev)
        t = e0.elapsed_time(e1) * 1e-3
        best = t if best is None else min(best, t)
    return best, out


def secondary_configs(torch, dev, world, rank, engine, peaks_file, mufu_peak):
    import math

    import torch.distributed as dist

    from geomloss_b200 import SamplesLoss, multiscale, ops, ranges, sinkhorn_divergence
    from geomloss_b200.sinkhorn_images import softmin_grid

    out = {}
    peaks = json.load(open(peaks_file)) if os.path.exists(peaks_file) else {}
    tensor_peak = peaks.get("bf16_tflops_sustained", 1450.0) * 1e12

    if world == 1:
        # ---- configs[2]: SamplesLoss('gaussian') N=M=1e6, D=64 (tensor-core path) ----
        N, D = 1_000_000, 64
        g = torch.Generator().manual_seed(0)
        x = torch.rand(N, D, generator=g).to(dev)
        y = torch.rand(N, D, generator=g).to(dev)
        L = SamplesLoss("gaussian", blur=0.05, backend="online")
        t_fwd, _ = _ev_time(torch, dev, lambda: L(x, y), reps=2)
        xg = x.clone().requires_grad_(True)

        def fwd_bwd():
            v = L(xg, y)
            torch.autograd.grad(v, xg)
            return v

        t_fb, _ = _ev_time(torch, dev, fwd_bwd, reps=2)
        fwd_rate = 3.0 * N * N / t_fwd          # K_xx a, K_yy b, K_xy b
        one_pass = bool(ops.FUSED_CONV_GRAD)
        if one_pass:
            # the two matvecs whose rows need a gradient come out of the row-gradient reduction itself (value + unit
            # gradient in one pass, ops._KernelConv): forward + backward = 1 plain reduction (K_yy b) + 2 such passes
            bwd_rate = 2.0 * N * N / (t_fb - t_fwd / 3.0)
        else:
            bwd_rate = 2.0 * N * N / (t_fb - t_fwd)  # row gradients of the xx and xy terms, after a 3-reduction forward
        # spot parity at blur = 2 (at the config's blur = .05 every off-diagonal kernel value underflows in [0,1]^64:
        # SURVEY.md 8(d)); 128 sampled rows of K_xy @ b against fp64 brute force on the device
        w = torch.full((N,), 1.0 / N, device=dev)
        rows = torch.randint(0, N, (128,), generator=g).to(dev)
        got = ops.kernel_conv_raw("gaussian", x, y, w, 2.0, center=ops.default_center(x, y))[rows].double()
        xr = x[rows].double()
        d2 = (xr * xr).sum(1)[:, None] - 2 * xr @ y.double().t() + (y.double() ** 2).sum(1)[None, :]
        want = (torch.exp(-d2 / 8.0) @ w.double())
        out["cfg3_gaussian_mmd_D64"] = {
            "workload": "SamplesLoss('gaussian', blur=.05) N=M=1e6 D=64, uniform in [0,1]^64",
            "s_fwd": t_fwd, "s_fwd_bwd": t_fb, "fwd_pairs_per_s": fwd_rate, "bwd_pairs_per_s": bwd_rate,
            "reductions_fwd_bwd": 3 if one_pass else 5, "one_pass_value_and_gradient": one_pass,
            "sfu_frac_fwd": fwd_rate / mufu_peak, "sfu_frac_bwd": bwd_rate / mufu_peak,
            "tensor_frac_fwd_algorithmic_128_flop_per_pair": fwd_rate * 128 / tensor_peak,
            "tensor_frac_fwd_issued_416_flop_per_pair": fwd_rate * 416 / tensor_peak,
            "tensor_peak_tflops": tensor_peak / 1e12,
            "spot_parity": {"what": "128 sampled rows of K_xy @ b at blur=2 vs fp64 brute force",
                            "max_rel_err": float(((got - want).abs() / want.abs()).max())},
        }
        del x, y, xg, d2
        torch.cuda.empty_cache()

        # ---- configs[4]: unbalanced Sinkhorn on a 256^3 volume (separable grid softmin) ----
        n = 256
        ax = torch.linspace(0, 1, n, device=dev)
        X, Y, Z = torch.meshgrid(ax, ax, ax, indexing="ij")

        def blobs(seed, mass):
            gg = torch.Generator().manual_seed(seed)
            f = torch.full((n, n, n), 1e-3, device=dev)
            for _ in range(3):
                c = 0.25 + 0.5 * torch.rand(3, generator=gg)
                s = 0.05 + 0.1 * float(torch.rand(1, generator=gg))
                f = f + torch.exp(-((X - c[0]) ** 2 + (Y - c[1]) ** 2 + (Z - c[2]) ** 2) / (2 * s * s))
            return (f * (mass / f.sum()))[None, None].contiguous()

        a, b = blobs(0, 1.0), blobs(1, 1.3)
        h = torch.log(a)
        # a smooth dual potential (a Sinkhorn iterate is smooth at the pixel scale; white noise / eps would make every
        # 8-input chunk re-base the running max and measure the kernel's slow path, not its Sinkhorn-time behaviour)
        pot = (0.02 * (torch.sin(3.0 * X) + torch.cos(2.0 * Y) * Z))[None, None].contiguous()
        eps = (1.0 / n) ** 2
        t_op, res = _ev_time(torch, dev, lambda: softmin_grid(eps, 2, h, pot, 1.0 / eps), reps=5)
        t_div, val = _ev_time(torch, dev, lambda: sinkhorn_divergence(a, b, p=2, blur=1.0 / n, reach=0.3, scaling=0.5), reps=2)
        # spot parity: 64 sampled output lines along the last axis, fp64 on the device, separable form
        hh = (h + pot / eps)[0, 0].double()
        xs = torch.arange(n, device=dev, dtype=torch.float64) / n / math.sqrt(2 * eps)
        k = -(xs[:, None] - xs[None, :]) ** 2
        i0 = torch.randint(0, n, (8,), generator=torch.Generator().manual_seed(3)).to(dev)
        i1 = torch.randint(0, n, (8,), generator=torch.Generator().manual_seed(4)).to(dev)
        t2 = torch.logsumexp(hh[:, :, None, :] + k[None, None, :, :], dim=-1)          # axis 2: (j0, j1, i2)
        t1 = torch.logsumexp(t2[:, None, :, :] + k[i1][None, :, :, None], dim=2)        # axis 1 at i1: (j0, 8, i2)
        t0 = torch.logsumexp(t1[None, :, :, :] + k[i0][:, :, None, None], dim=1)        # axis 0 at i0: (8, 8, i2)
        want = -eps * t0
        got = res[0, 0][i0][:, i1].double()
        out["cfg5_grid_256"] = {
            "workload": "sinkhorn_images.sinkhorn_divergence(a, b, p=2, blur=1/256, reach=.3, scaling=.5) on 256^3",
            "softmin_grid_ms": t_op * 1e3, "softmin_grid_pairs_per_s": 3.0 * n**4 / t_op,
            "sfu_frac": 3.0 * n**4 / t_op / mufu_peak,
            "hbm_GBps_algorithmic": 3 * 8 * n**3 / t_op / 1e9, "divergence_ms": t_div * 1e3, "value": float(val[0]),
            "spot_parity": {"what": "8 x 8 sampled output lines (all 256 entries) of one softmin_grid call vs fp64",
                            "max_abs_err": float((got - want).abs().max()), "scale": float(want.abs().max())},
        }
        del a, b, h, pot, res, hh, t2, t1, t0, X, Y, Z
        torch.cuda.empty_cache()

    if world == 1:
        # ---- small / batched clouds (ADVICE r01: the regime most users live in): B=64 x N=M=500 and one N=M=1000 problem,
        #      reference benchmark protocol = forward + backward, wall clock over 20 calls after a warm-up ----
        small = {}
        g = torch.Generator().manual_seed(0)
        for tag, shape in (("B64_N500", (64, 500, 3)), ("N1000", (1000, 3))):
            xs = torch.rand(*shape, generator=g).to(dev).requires_grad_(True)
            ys = torch.rand(*shape, generator=g).to(dev)
            for loss_name, kw in (("sinkhorn", dict(p=2, blur=0.05, diameter=1.8)), ("gaussian", dict(blur=0.1))):
                Ls = SamplesLoss(loss_name, **kw)

                def call():
                    v = Ls(xs, ys).sum()
                    torch.autograd.grad(v, xs)
                    return v

                call()
                torch.cuda.synchronize(dev)
                l0, t0 = ops.launches(), time.perf_counter()
                for _ in range(20):
                    call()
                torch.cuda.synchronize(dev)
                small[f"{tag}_{loss_name}"] = {"ms_per_call_fwd_bwd": (time.perf_counter() - t0) / 20 * 1e3,
                                              "b200ot_launches_per_call": (ops.launches() - l0) / 20}
        small["workload"] = ("SamplesLoss(loss)(x, y) + autograd.grad w.r.t. x, uniform cube, D=3; batched inputs run as ONE "
                             "launch group per Sinkhorn iteration (csrc/b200ot_small.cu)")
        out["small_and_batched"] = small

    if world == 1:
        # ---- D = 6, 8: the forward operators of large problems run on the tensor-core kernels (DESIGN.md 3.3c; the
        #      CUDA-core rates they replace are in profiles/r02_ab_tc_route.jsonl).  Default routing, nothing forced; a
        #      failure here drops this entry, not the bench line ----
        try:
            dims = {}
            N = 400_000
            for D in (6, 8):
                g = torch.Generator().manual_seed(D)
                x = torch.rand(N, D, generator=g).to(dev)
                y = torch.rand(N, D, generator=g).to(dev)
                h = (torch.rand(N, generator=g) * 0.1).to(dev)
                w = (torch.rand(N, generator=g) / N).to(dev)
                c = ops.default_center(x, y)
                eps, blur = 1e-3, 0.15
                t_s, f = _ev_time(torch, dev, lambda: ops.softmin_raw(eps, x, y, h, p=2, center=c)[0], reps=2)
                t_c, kv = _ev_time(torch, dev, lambda: ops.kernel_conv_raw("gaussian", x, y, w, blur, center=c), reps=2)
                rows = torch.randint(0, N, (64,), generator=g).to(dev)
                xr, yd = x[rows].double(), y.double()
                d2 = ((xr * xr).sum(1)[:, None] - 2 * xr @ yd.t() + (yd * yd).sum(1)[None, :]).clamp_min(0)
                f_ref = -eps * torch.logsumexp(h.double()[None, :] - d2 / (2 * eps), dim=1)
                k_ref = torch.exp(-d2 / (2 * blur * blur)) @ w.double()
                dims[f"D{D}"] = {
                    "softmin_fwd_ms": t_s * 1e3, "softmin_fwd_pairs_per_s": N * N / t_s, "sfu_frac_softmin": N * N / t_s / mufu_peak,
                    "gaussian_fwd_ms": t_c * 1e3, "gaussian_fwd_pairs_per_s": N * N / t_c, "sfu_frac_gaussian": N * N / t_c / mufu_peak,
                    "spot_parity": {"what": "64 sampled rows vs fp64 brute force",
                                    "softmin_max_abs_err": float((f[rows].double() - f_ref).abs().max()),
                                    "softmin_scale": float(f_ref.abs().max()),
                                    "gaussian_max_rel_err": float(((kv[rows].double() - k_ref).abs() / k_ref.abs()).max())},
                }
                del x, y, h, w, d2, xr, yd
            dims["workload"] = ("ops.softmin_raw(eps=1e-3, p=2) and ops.kernel_conv_raw('gaussian', blur=.15), N=M=4e5, uniform cube; "
                                "tensor-core kernels on the zero-padded dk=16 problem (forward softmin from D=6, gaussian from D=5)")
            out["forward_D6_D8"] = dims
        except Exception as exc:  # pragma: no cover
            out["forward_D6_D8"] = {"error": repr(exc)[:300]}
        torch.cuda.empty_cache()

    # ---- configs[3]: multiscale Sinkhorn (eps-scaling .5, truncate 5): N=M=1e6 at every --gpus, 1e7 at --gpus 8 ----
    sizes = [1_000_000] + ([10_000_000] if world >= 8 else [])
    ms = {}
    for N in sizes:
        g = torch.Generator().manual_seed(0)
        x = torch.rand(N, 3, generator=g).to(dev)
        y = torch.rand(N, 3, generator=g).to(dev)
        L = SamplesLoss("sinkhorn", p=2, blur=0.01, scaling=0.5, truncate=5, backend="multiscale")
        if engine:
            engine.attach(L)
        stats = {}
        orig_build = ranges.build_problem

        def spy(*a, **k):
            pr = orig_build(*a, **k)
            stats.setdefault("density", []).append(pr.density)
            return pr

        ranges.build_problem = spy
        try:
            t, v = _ev_time(torch, dev, lambda: L(x, y), reps=1, warm=1)
        finally:
            ranges.build_problem = orig_build
        tt = torch.tensor([t], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms[f"N{N}"] = {"s_fwd": float(tt), "value": float(v),
                       "kept_pair_fraction": (sum(stats["density"]) / len(stats["density"])) if stats.get("density") else None}
        del x, y
        torch.cuda.empty_cache()
    if world == 1:
        # operator-level spot parity of the ranges mode at full size: a geometric cluster mask, 64 sampled rows
        N = 1_000_000
        g = torch.Generator().manual_seed(1)
        x, y = torch.rand(N, 3, generator=g).to(dev), torch.rand(N, 3, generator=g).to(dev)
        w = torch.full((N,), 1.0 / N, device=dev)
        cs = math.sqrt(3) / (math.sqrt(3) * 2000 ** (1 / 3))
        (_, x_c), (_, x_s), lab_x, _, cnt_x = multiscale.clusterize(w, x, scale=cs)
        (_, y_c), (_, y_s), lab_y, _, cnt_y = multiscale.clusterize(w, y, scale=cs)
        keep = ((x_c[:, None, :] - y_c[None, :, :]) ** 2).sum(-1) < 0.2**2
        prob = ranges.build_problem(keep, cnt_x, ranges.ColumnLayout(cnt_y))
        h = torch.randn(N, generator=g).to(dev)
        eps = 1e-3
        t_op, (res, _) = _ev_time(torch, dev, lambda: ranges.softmin_ranges_raw(eps, x_s, y_s, h, None, 0.0, prob, p=2,
                                                                              center=ops.default_center(x, y)), reps=3)
        rows = torch.randint(0, N, (64,), generator=g).to(dev)
        colmask = keep[lab_x[rows]][:, lab_y]
        d2 = ((x_s[rows].double()[:, None, :] - y_s.double()[None, :, :]) ** 2).sum(-1) / 2
        want = -eps * torch.logsumexp((h.double()[None, :] - d2 / eps).masked_fill(~colmask, -float("inf")), dim=1)
        ms["ranges_operator_N1e6"] = {
            "kept_pair_fraction": prob.density, "ms": t_op * 1e3, "pairs_per_s": prob.density * N * N / t_op,
            "sfu_frac": prob.density * N * N / t_op / mufu_peak,
            "spot_parity": {"what": "64 sampled rows of one ranges-mode softmin (cluster mask: centroids closer than .2) vs fp64 "
                                    "brute force over the kept columns", "max_abs_err": float((res[rows].double() - want).abs().max()),
                            "scale": float(want.abs().max())}}
    ms["workload"] = "SamplesLoss('sinkhorn', p=2, blur=.01, scaling=.5, truncate=5, backend='multiscale') on uniform-in-cube clouds"
    out["cfg4_multiscale"] = ms
    return out


def kernel_pass(L, ops, torch, dev, x, y, h_a, h_b, inv, center, eps, p, flush, reps, world, rank):
    """Time the partial-reduction kernel alone (pack and finalize outside the events)."""
    from geomloss_b200.distributed import shard_bounds

    N, D = x.shape
    lo, hi = shard_bounds(y.shape[0], rank, world)
    ys, ha, hb = y[lo:hi], h_a[lo:hi], h_b[lo:hi]
    M = ys.shape[0]
    nsplit = L.b200ot_softmin_num_splits(N, M, D)
    cols = torch.empty(L.b200ot_packed_cols_floats(M, D, 1), dtype=torch.float32, device=dev)
    part = torch.empty(nsplit * N * 2, dtype=torch.float32, device=dev)
    st = ops._stream(dev)
    from geomloss_b200 import _lib

    _lib.check(L.b200ot_softmin_pack(ops._ptr(ys), ops._ptr(ha), ops._ptr(hb), float(inv), ops._ptr(center), M, D, p,
                                     float(eps), ops._ptr(cols), st), "pack")
    times = []
    for r in range(reps + 1):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(L.b200ot_softmin_partial(ops._ptr(x), ops._ptr(center), ops._ptr(cols), ops._ptr(part), nsplit, N, M,
                                            D, p, float(eps), st), "partial")
        e1.record()
        torch.cuda.synchronize(dev)
        if r > 0:
            times.append(e0.elapsed_time(e1))
    ms = sum(times) / len(times)
    return {"ms_per_launch": ms, "pairs_per_s": float(N) * M / (ms * 1e-3)}


def pipe_ceilings(L, ops, torch, dev):
    import ctypes

    from geomloss_b200 import _lib

    sink = torch.zeros(256, dtype=torch.float32, device=dev)
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    out = {}
    for name, which in (("mufu_ex2_per_s", 0), ("ffma_per_s", 1)):
        ops_per = ctypes.c_int32(0)
        iters, blocks = 8192, sms * 8
        best = None
        for r in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(L.b200ot_ubench(which, iters, blocks, ops._ptr(sink), ctypes.byref(ops_per), ops._stream(dev)),
                       "ubench")
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1)
            if r > 0 and (best is None or ms < best):
                best = ms
        out[name] = float(blocks) * 256 * iters * ops_per.value / (best * 1e-3)
    return out


def cpu_baseline(args):
    import torch

    n = args.cpu_n
    O, eps, a_log, C, pots = dense_iteration_state(n, args.blur)
    with torch.no_grad():
        pots = dense_iteration(O, eps, a_log, C, pots)
        t0 = time.perf_counter()
        it = 0
        while True:
            pots = dense_iteration(O, eps, a_log, C, pots)
            it += 1
            dt = time.perf_counter() - t0
            if dt > 10.0 or it >= 50:
                break
    cores = torch.get_num_threads()
    kind = reference_ops()[1]
    what = ("the unmodified reference's softmin_tensorized (oracle/_ref)" if kind == "reference"
            else "oracle port of the reference's tensorized path")
    return {"value": 4.0 * n * n * it / dt, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{it} dense symmetric Sinkhorn iterations (4 softmins each) at N=M={n}, D=3, blur={args.blur}, "
                      f"{what}, torch CPU {cores} threads, {cpu_model()}, {dt:.1f} s"}


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
