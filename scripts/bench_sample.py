"""Device time of the posterior sampler (moihgp_cuda_sample_posterior_dev) at the BASELINE config-3 and config-4 shapes.

Each case runs the whole call (RTS mean pass + sampler) with inputs resident in HBM: one warm-up call, then --reps calls
under the library's per-kernel event markers (moihgp_cuda_profile).  Reported per case: the sampler kernels' device time
per call, k_smooth_chain's time in the same calls where the mean pass runs on the many-chains kernels, the algorithmic
bytes of the sampler (read the mean, write the samples) and the rate they imply, and the time the same bytes would take at
the measured copy bandwidth.  A sampler time far above that HBM time means the kernel is bound by its arithmetic
(Philox + fp64 Box-Muller + the backward recursion), not by memory.  Card name, power limit and clocks are read in the
same run.  Writes one JSON document to --out (default: stdout only).

    python scripts/bench_sample.py [--reps 3] [--out FILE] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)

HBM_GBS = 6553.3   # measured device-to-device copy bandwidth of one B200 (DESIGN.md section 4)
DT = 0.1
IGP = {"Matern32": [(1, 1, .1), (.5, .5, .1), (2, .3, .05), (.5, .3, .5)],    # bench.py's latents
       "Matern52": [(1, 1, .1), (.5, .5, .1), (.5, .3, .05), (.5, .5, .5)]}
SAMPLER_KERNELS = ("k_sample", "k_sample_chunks", "k_sample_carry", "k_sample_final")


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        return dict(zip(q.split(","), [s.strip() for s in out.splitlines()[0].split(",")]))
    except Exception as e:      # the figures are still valid, only unlabelled
        return {"error": repr(e)}


def params(p, L, kernel, seed):
    rng = np.random.default_rng(seed)
    tbl = IGP[kernel]
    igp = np.array([tbl[l % len(tbl)] for l in range(L)], dtype=np.float64).ravel()
    return np.concatenate([(rng.standard_normal((p, L)) / np.sqrt(L)).ravel(), np.ones(L), [1e-2], igp])


def run_case(name, kernel, p, L, N, T, S, values_only, path, reps):
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    d = 3 if kernel == "Matern52" else 2
    dev = torch.device("cuda:0")
    m = MOIHGPSequences(DT, p, L, kernel, True)
    m.update(params(p, L, kernel, 1234))
    m.set_path(path)
    g = torch.Generator(device=dev).manual_seed(7)
    Y = torch.randn((N, T, p), dtype=torch.float64, device=dev, generator=g)
    Xs = torch.empty((N, T, L, d), dtype=torch.float64, device=dev)
    X = None if values_only else torch.empty((S, N, T, L, d), dtype=torch.float64, device=dev)
    F = torch.empty((S, N, T, L), dtype=torch.float64, device=dev) if values_only else None
    m.sample_posterior_device(Y, 1, Xs=Xs, X=X, F=F)
    torch.cuda.synchronize()
    m.profile(True)
    for r in range(reps):
        m.sample_posterior_device(Y, 100 + r, Xs=Xs, X=X, F=F)
    prof = m.profile_read()
    m.profile(False)
    steps = S * N * T * L
    # the mean is read once per sample: all d components for full states, component 0 for values only
    nbytes = steps * (8 * 2 * d if not values_only else 8 * 2)
    ms = sum(prof.get(k, (0.0, 0))[0] for k in SAMPLER_KERNELS) / reps
    out = {"case": name, "kernel": kernel, "p": p, "L": L, "d": d, "N": N, "T": T, "S": S,
           "outputs": "values F [S][N][T][L]" if values_only else "states X [S][N][T][L][d]",
           "variant": "time-chunked" if "k_sample_chunks" in prof else "one pass per chain",
           "sampler_ms": ms, "latent_steps_per_s": steps / (ms * 1e-3),
           "alg_bytes": nbytes, "alg_gbs": nbytes / (ms * 1e-3) / 1e9,
           "hbm_time_ms_at_measured_copy_bw": nbytes / (HBM_GBS * 1e9) * 1e3,
           "kernels_ms_per_call": {k: v[0] / reps for k, v in prof.items()}}
    out["hbm_share"] = out["hbm_time_ms_at_measured_copy_bw"] / ms
    if "k_smooth_chain" in prof:
        sm = prof["k_smooth_chain"][0] / reps
        out["k_smooth_chain_ms"] = sm
        out["k_smooth_chain_gbs"] = N * T * L * 16 * d / (sm * 1e-3) / 1e9
    print(json.dumps(out), flush=True)
    del Y, Xs, X, F, m
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small shapes (a rehearsal of the script, not a measurement)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_sample.py needs a CUDA device")
    n3, t3, t4 = (256, 1024, 100000) if a.quick else (4096, 16384, 10_000_000)
    info = gpu_info()
    print(json.dumps({"gpu": info}), flush=True)
    cases = [
        ("c3", "Matern52", 16, 8, n3, t3, 1, False, "auto"),
        ("c3", "Matern52", 16, 8, n3, t3, 1, True, "auto"),
        ("c3", "Matern52", 16, 8, n3, t3, 1, True, "scan"),      # the time-chunked variant forced, for the variant choice
        ("c3", "Matern52", 16, 8, n3, t3, 8, True, "auto"),
        ("c3", "Matern52", 16, 8, n3, t3, 8, False, "auto"),
        ("c4", "Matern32", 64, 32, 1, t4, 4, False, "auto"),
        ("c4", "Matern32", 64, 32, 1, t4, 4, True, "auto"),
    ]
    res = [run_case(*c, reps=a.reps) for c in cases]
    doc = {"what": "posterior sampler device time (moihgp_cuda_sample_posterior_dev), per-kernel CUDA events after one warm-up call",
           "gpu": info, "gpu_after": gpu_info(), "hbm_gbs_reference": HBM_GBS, "reps": a.reps, "results": res}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
