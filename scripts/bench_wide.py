"""Wide models (64 < L <= 256 latents) on one GPU: ms per call and latent-steps/s of the fused filter + smoother + NLL pass,
the objective and update(), with the projection kernel's own time, FP64 tensor rate and Y bandwidth.

    python scripts/bench_wide.py [--reps R] [--windows K] [--warmup W] [--out FILE]

Workloads (inputs resident in HBM, each larger than the 126 MB L2):
  W1  N = 1,   T = 10^6,    p = 512, L = 128, Matern-3/2: fused pass and objective; the fused pass once more with Y at an
      8-byte offset, which sends the projection to the scalar k_project (the same pass without the tensor-pipe kernel)
  W2  N = 256, T = 4096,    p = 128, L = 96,  Matern-5/2: fused pass
  W3  N = 1,   T = 2 10^5,  p = 256, L = 256, Matern-3/2 (square U): fused pass
  update() at p = 512, L = 256: a raw block one small step away from the current U (an optimiser's line search), and a
      random block (scaled start)
Times are CUDA events around windows of R calls after W warm-up calls, K windows per measurement: the median window
and the fastest and slowest ones are reported.  update() is a host call, timed with the host clock (it waits for the
device), K x R calls.  The projection's own time comes from the library's per-kernel event records (profile on), in a separate
run of the pass.  One JSON line per measurement, with the GPU name and power limit read in the same process."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)

DMMA_PEAK = 37.0e12          # FP64 tensor-pipe rate the project measured on a B200 (DESIGN 4)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(torch, fn, a):
    """ms per call of each of a.windows windows of a.reps calls"""
    for _ in range(a.warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(a.windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / a.reps)
    return out


def spread(ms):
    return {"ms": float(np.median(ms)), "ms_min": float(np.min(ms)), "ms_max": float(np.max(ms)), "windows": len(ms)}


def kernel_ms(m, fn, name):
    m.profile(True)
    fn()
    rec = m.profile_read()
    m.profile(False)
    return rec[name][0] / rec[name][1] if name in rec else None


def model(torch, kernel, p, L, seed):
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_params
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    m.update(make_params(np.random.default_rng(seed), p, L, kernel))
    return m


def observations(torch, N, T, p, offset=False):
    g = torch.Generator(device="cuda").manual_seed(N * T + p)
    n = N * T * p
    buf = torch.empty(n + 1, dtype=torch.float64, device="cuda")
    buf.normal_(generator=g)
    Y = buf[int(offset):int(offset) + n].view(N, T, p)
    assert (Y.data_ptr() % 16 == 8) == offset
    return Y


def fused(torch, name, kernel, N, T, p, L, a, info, with_objective=False, with_scalar=False):
    m = model(torch, kernel, p, L, 1)
    d = m.igp_dim
    f64 = dict(dtype=torch.float64, device="cuda")
    X, Xs = torch.empty((N, T, L, d), **f64), torch.empty((N, T, L, d), **f64)
    nll, xT = torch.empty(N, **f64), torch.empty((N, L, d), **f64)
    rows = []
    variants = [("aligned Y", False)] + ([("offset Y (scalar k_project)", True)] if with_scalar else [])
    for what, off in variants:
        Y = observations(torch, N, T, p, off)
        run = lambda: m.filter_smoother_nll_device(Y, smoother_mode=1, X=X, Xs=Xs, nll=nll, xT=xT)
        ms = spread(timed(torch, run, a))
        kp = float(np.median([kernel_ms(m, run, "k_project") for _ in range(a.windows)]))
        flop, ybytes = 2.0 * p * L * N * T, 8.0 * p * N * T
        rows.append({"workload": name, "call": "filter_smoother_nll_dev (RTS)", "variant": what, "kernel": kernel, "N": N, "T": T, "p": p,
                     "L": L, **ms, "reps_per_window": a.reps, "latent_steps_per_s": N * T * L / (ms["ms"] * 1e-3), "k_project_ms": kp,
                     "k_project_tflops": flop / (kp * 1e-3) / 1e12 if kp else None,
                     "k_project_share_of_dmma_peak": flop / (kp * 1e-3) / DMMA_PEAK if kp else None,
                     "k_project_Y_GBps": ybytes / (kp * 1e-3) / 1e9 if kp else None, "gpu": info})
        del Y
    if with_objective:
        Y = observations(torch, N, T, p)
        loss, grad = torch.empty(1, **f64), torch.empty(m.num_param, **f64)
        run = lambda: m.objective_device(Y, loss, grad)
        ms = spread(timed(torch, run, a))
        rows.append({"workload": name, "call": "objective_dev", "kernel": kernel, "N": N, "T": T, "p": p, "L": L, **ms, "reps_per_window": a.reps,
                     "latent_steps_per_s": N * T * L / (ms["ms"] * 1e-3), "k_project_ms": kernel_ms(m, run, "k_project"), "gpu": info})
        del Y
    del X, Xs
    torch.cuda.empty_cache()
    return rows


def update_rows(torch, a, info):
    from multioutputihgp_b200 import MOIHGPSequences
    p, L = 512, 256
    rng = np.random.default_rng(4)
    m = MOIHGPSequences(0.1, p, L, "Matern32", True)
    rest = np.concatenate([np.ones(L), [1e-2], np.tile([1.0, 1.0, 0.1], L)])
    m.update(np.concatenate([(np.eye(p, L) + 0.3 * rng.standard_normal((p, L))).ravel(), rest]))
    rows = []
    for what, make in (("small step from the current U", lambda: m.U + 1e-3 * rng.standard_normal((p, L))),
                       ("random block", lambda: rng.standard_normal((p, L)))):
        blocks = [np.concatenate([make().ravel(), rest]) for _ in range(a.warmup + a.reps * a.windows)]
        ts = []
        for i, b in enumerate(blocks):
            m.synchronize()
            t0 = time.perf_counter()
            m.update(b)
            m.synchronize()
            if i >= a.warmup:
                ts.append(1e3 * (time.perf_counter() - t0))
        rows.append({"workload": "update", "variant": what, "p": p, "L": L, "ms_median": float(np.median(ts)), "ms_min": float(np.min(ts)),
                     "ms_max": float(np.max(ts)), "calls": len(ts), "gpu": info})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    info = gpu_info()
    rows = []
    rows += fused(torch, "W1", "Matern32", 1, 1000000, 512, 128, a, info, with_objective=True, with_scalar=True)
    rows += fused(torch, "W2", "Matern52", 256, 4096, 128, 96, a, info)
    rows += fused(torch, "W3", "Matern32", 1, 200000, 256, 256, a, info)
    rows += update_rows(torch, a, info)
    for r in rows:
        print(json.dumps(r))
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in rows) + "\n")


if __name__ == "__main__":
    main()
