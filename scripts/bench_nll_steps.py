"""Device time of the per-step NLL pass (moihgp_cuda_nll_steps_dev) next to the fused pass it extends
(moihgp_cuda_filter_smoother_nll_dev with smoother_mode = NONE, no states, nll only), at the BASELINE config-3 and config-4
shapes.

Inputs are resident in HBM.  Every case runs one warm-up call of each pass, then --rounds rounds that alternate the two
passes, --reps calls each, timed with CUDA events around the calls (the host does not wait between calls).  Reported per
case and pass: ms per call (median over the rounds), the bytes the algorithm must move (read Y; write nll_steps [N][T] for
the per-step pass) and, separately, the bytes of the workspace the chunked scan adds for the per-step terms (v^2 [N][L][T]
written and read, the residual norms written into nll_steps and read back), and the share of the HBM roofline those
algorithmic bytes imply at the device-to-device copy bandwidth measured in the same run.  The algorithmic bytes are the
same on both paths: the scan path's own projected-series workspace u is a cost of that path, not of the algorithm, and is
not counted.  Card name and power limit are read in the same run.  Writes one
JSON document to --out (default: stdout only).

    python scripts/bench_nll_steps.py [--reps 5] [--rounds 5] [--out FILE] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)

DT = 0.1
IGP = {"Matern32": [(1, 1, .1), (.5, .5, .1), (2, .3, .05), (.5, .3, .5)],    # bench.py's latents
       "Matern52": [(1, 1, .1), (.5, .5, .1), (.5, .3, .05), (.5, .5, .5)]}


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        return dict(zip(q.split(","), [s.strip() for s in out.splitlines()[0].split(",")]))
    except Exception as e:      # the figures are still valid, only unlabelled
        return {"error": repr(e)}


def copy_gbs(reps=10):
    """Device-to-device copy bandwidth (read + write bytes) of a 4 GiB fp64 tensor, best of `reps`."""
    import torch
    a = torch.empty(1 << 29, dtype=torch.float64, device="cuda:0")
    b = torch.empty_like(a)
    b.copy_(a)
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2 * 8 * (1 << 29) / (best * 1e-3) / 1e9


def params(p, L, kernel, seed):
    rng = np.random.default_rng(seed)
    tbl = IGP[kernel]
    igp = np.array([tbl[l % len(tbl)] for l in range(L)], dtype=np.float64).ravel()
    return np.concatenate([(rng.standard_normal((p, L)) / np.sqrt(L)).ravel(), np.ones(L), [1e-2], igp])


def run_case(name, kernel, p, L, N, T, path, reps, rounds, hbm_gbs):
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    d = 3 if kernel == "Matern52" else 2
    dev = torch.device("cuda:0")
    m = MOIHGPSequences(DT, p, L, kernel, True)
    m.update(params(p, L, kernel, 1234))
    m.set_path(path)
    g = torch.Generator(device=dev).manual_seed(7)
    Y = torch.randn((N, T, p), dtype=torch.float64, device=dev, generator=g)
    steps = torch.empty((N, T), dtype=torch.float64, device=dev)
    nll_f, nll_s = (torch.empty(N, dtype=torch.float64, device=dev) for _ in range(2))
    xT = torch.empty((N, L, d), dtype=torch.float64, device=dev)
    passes = {"nll_steps": lambda: m.nll_steps_device(Y, steps, nll=nll_s, xT=xT),
              "fused_nll_only": lambda: m.filter_smoother_nll_device(Y, smoother_mode=-1, nll=nll_f)}
    for f in passes.values():
        f()
    torch.cuda.synchronize()
    # which kernels serve the per-step pass (one profiled call, not timed)
    m.profile(True)
    passes["nll_steps"]()
    kernels = sorted(m.profile_read())
    m.profile(False)
    times = {k: [] for k in passes}
    for _ in range(rounds):
        for k, f in passes.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                f()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / reps)
    rel = float((steps.sum(dim=1) - nll_f).abs().max() / nll_f.abs().max())
    scan = "k_nll_steps" in kernels
    y_bytes, out_bytes = 8 * N * T * p, 8 * N * T
    ws_bytes = (2 * 8 * N * L * T + 2 * 8 * N * T) if scan else 0
    res = {"case": name, "kernel": kernel, "p": p, "L": L, "d": d, "N": N, "T": T, "path": "chunked scan" if scan else "many-chains",
           "kernels": kernels, "sum_of_terms_vs_fused_nll_rel": rel, "passes": {}}
    for k, ts in times.items():
        ms = float(np.median(ts))
        alg = y_bytes + (out_bytes if k == "nll_steps" else 0)
        res["passes"][k] = {"ms_per_call": ms, "ms_all_rounds": ts, "alg_bytes": alg,
                            "scan_workspace_bytes": ws_bytes if k == "nll_steps" else 0,
                            "alg_gbs": alg / (ms * 1e-3) / 1e9, "hbm_roofline_share": alg / (hbm_gbs * 1e9) / (ms * 1e-3)}
    res["overhead"] = res["passes"]["nll_steps"]["ms_per_call"] / res["passes"]["fused_nll_only"]["ms_per_call"] - 1.0
    print(json.dumps(res), flush=True)
    del Y, steps, m
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small shapes (a rehearsal of the script, not a measurement)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_nll_steps.py needs a CUDA device")
    n3, t3, t4 = (256, 1024, 100000) if a.quick else (4096, 16384, 10_000_000)
    info = gpu_info()
    hbm = copy_gbs()
    print(json.dumps({"gpu": info, "copy_gbs": hbm}), flush=True)
    cases = [
        ("c3", "Matern52", 16, 8, n3, t3, "auto"),      # many-chains kernels
        ("c3", "Matern52", 16, 8, n3, t3, "scan"),      # the chunked scan forced at the same shape
        ("c4", "Matern32", 64, 32, 1, t4, "auto"),      # chunked scan
    ]
    res = [run_case(*c, reps=a.reps, rounds=a.rounds, hbm_gbs=hbm) for c in cases]
    doc = {"what": "per-step NLL pass vs the fused pass (NONE smoother, nll only): CUDA events around --reps calls, median of "
                   "--rounds alternating rounds, inputs resident in HBM",
           "gpu": info, "gpu_after": gpu_info(), "copy_gbs_measured": hbm, "reps": a.reps, "rounds": a.rounds, "results": res}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
