#!/usr/bin/env python
"""bench.py - latent time-steps/s of the fused filter + smoother + NLL pass (fp64) on B200.

Contract (one JSON line on stdout from rank 0):
    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun, one rank per GPU)
    python bench.py --impl reference ...                      (the CPU implementation of the same path, host cores)
    python bench.py ... --dump-outputs DIR                    (also writes what the last timed step computed, DIR/*.npy)

Workload (BASELINE.json configs[2], the configuration its metric and SURVEY 8(d)'s >= 50 % target are
quoted on): 4096 independent sequences x T = 16384, p = 16 outputs, L = 8 latents, Matern-5/2 (state
dim 3), dt = 0.1, synthetic data.  One "step" = one fused pass over the whole batch: projection, steady-state
Kalman filter, RTS smoother and NLL, writing the filtered states X, the smoothed states Xs and nll[n].
Multi-GPU: sequences are sharded over ranks (weak scaling: 4096 sequences PER GPU), no data-path collective;
the only exchange is the fp64 all-reduce of the summed NLL.

  value    : N*T*L / time with Y, X, Xs resident in HBM (CUDA events around K steps, max over ranks)
  e2e      : same metric through the host-buffer C-ABI call (moihgp_cuda_filter_smoother_nll), pinned host
             memory, H2D of Y and D2H of X, Xs, nll inside the timed region
  roofline : algorithmic bytes (SURVEY 8(d): 8*(p/L + 2d) per latent-step) / device time, vs the measured HBM peak
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (kind, kernel, p, L, N per GPU, T)      kind "fsn" = filter + smoother + NLL, "obj" = NLL + gradient
    "c3": ("fsn", "Matern52", 16, 8, 4096, 16384),
    "c4": ("fsn", "Matern32", 64, 32, 1, 10000000),
    "c5": ("obj", "Matern32", 256, 64, 1, 1000000),
}
WORKLOAD_DESC = {
    "c3": "BASELINE configs[2]: batched filter+smoother, 4096 sequences x T=16384, p=16, L=8, Matern-5/2 (d=3), dt=0.1",
    "c4": "BASELINE configs[3]: long-horizon single sequence, p=64, L=32, Matern-3/2 (d=2), T=1e7, dt=0.1 (parallel-scan stress test)",
    "c5": "BASELINE configs[4]: L-BFGS objective (NLL + gradient), p=256, L=64, Matern-3/2 (d=2), T=1e6, dt=0.1",
}
# per-latent (magnitude, lengthscale, noise), cycled; filter- and smoother-stable under the reference's semantics
# (SURVEY 8(d)); checked at setup (rho(AKHA) < 1, rho(G) < 1)
IGP_TABLE = {
    "Matern32": [(1, 1, .1), (.5, .5, .1), (2, .3, .05), (.5, .3, .5)],
    "Matern52": [(1, 1, .1), (.5, .5, .1), (.5, .3, .05), (.5, .5, .5)],
}
DT = 0.1
METRIC = "latent time-steps/sec (filter+smoother+NLL, fp64)"
UNIT = "latent-steps/s"


def model_params(p, L, kernel, seed):
    rng = np.random.default_rng(seed)
    Hmix = rng.standard_normal((p, L)) / np.sqrt(L)
    tbl = IGP_TABLE[kernel]
    igp = np.array([tbl[l % len(tbl)] for l in range(L)], dtype=np.float64).ravel()
    # U = polar(Hmix) is formed by update(); S = 1, sigma = 1e-2 are the reference's defaults (moihgp.h:126-127)
    return np.concatenate([Hmix.ravel(), np.ones(L), [1e-2], igp]), Hmix


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def alg_bytes_per_latent_step(kind, p, L, d):
    if kind == "obj":
        return 8.0 * p / L             # SURVEY 8(d): the objective reads Y once and writes O(num_param)
    return 8.0 * (p / L + 2 * d)       # SURVEY 8(d): read y share, write filtered x (d) and smoothed xs (d)


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def _nvml_loop(self, index):
        # in-process sampling through NVML every 5 ms (nvidia-smi -lms delivers only a handful of samples in a 0.2 s timed
        # region); the nvidia-smi stream stays as the fallback
        try:
            import pynvml as nv
            nv.nvmlInit()
            hd = nv.nvmlDeviceGetHandleByIndex(index)
            mx = float(nv.nvmlDeviceGetMaxClockInfo(hd, nv.NVML_CLOCK_SM))
            bits = (("gpu_idle", 0x1), ("applications_clocks_setting", 0x2), ("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sync_boost", 0x10),
                    ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40), ("hw_power_brake_slowdown", 0x80), ("display_clock_setting", 0x100))
            while not self._nv_stop:
                if self._nv_on:
                    sm = float(nv.nvmlDeviceGetClockInfo(hd, nv.NVML_CLOCK_SM))
                    try:
                        rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(hd))
                    except Exception:
                        rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(hd))
                    try:
                        pw = nv.nvmlDeviceGetPowerUsage(hd) / 1000.0
                    except Exception:
                        pw = None
                    self._nv_rows.append((sm, mx, tuple(n for n, b in bits if rs & b), rs, pw))
                time.sleep(0.005)
        except Exception:
            pass

    def __init__(self, index):
        self._nv_rows, self._nv_stop, self._nv_on = [], False, False
        self._nv_thread = threading.Thread(target=self._nvml_loop, args=(index,), daemon=True)
        self._nv_thread.start()
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def mark_timed_region_start(self):
        """Samples taken before this point (start-up, warm-up) are dropped."""
        self._nv_on = True
        self.f.flush()
        try:
            self.skip = sum(1 for _ in open(self.f.name))
        except Exception:
            self.skip = 0

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        self._nv_on, self._nv_stop = False, True
        if len(self._nv_rows) >= 3:
            if self.p is not None:
                self.p.terminate()
                try:
                    self.p.wait(timeout=5)
                except Exception:
                    self.p.kill()
                try:
                    os.unlink(self.f.name)
                except Exception:
                    pass
            rows = list(self._nv_rows)
            reasons = sorted({r for row in rows for r in row[2]})
            out.update(sm_mhz=float(np.median([r[0] for r in rows])), sm_max_mhz=float(max(r[1] for r in rows)), reasons=reasons,
                       samples=len(rows), source="nvml", sm_mhz_min=float(min(r[0] for r in rows)),
                       reasons_mask="0x%x" % int(np.bitwise_or.reduce([r[3] for r in rows])),
                       power_w=(float(np.median([r[4] for r in rows if r[4] is not None])) if any(r[4] is not None for r in rows) else None))
            return out
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().splitlines() if r.strip()][getattr(self, "skip", 0):]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if val.strip().lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def make_data_device(torch, dev, Hmix, N, T, p, L, seed, rank, t_offset=0):
    """Synthetic observations after example_regression.cpp:18-28: sinusoidal latents sin(w_l t + phi_n), mixed by Hmix,
    plus 0.1 * U(-1, 1) noise.  Built block-wise on the device.  t_offset: first time step (a rank's block of one long
    sequence sharded in time)."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed + 7919 * rank)
    Y = torch.empty((N, T, p), dtype=torch.float64, device=dev)
    t = (torch.arange(T, dtype=torch.float64, device=dev) + float(t_offset)) * DT
    w = 1.0 + 3.0 * torch.arange(L, dtype=torch.float64, device=dev) / max(L - 1, 1)
    H = torch.from_numpy(Hmix).to(dev)
    nb = 128
    for n0 in range(0, N, nb):
        n1 = min(N, n0 + nb)
        phi = 2.0 * np.pi * (torch.arange(n0, n1, dtype=torch.float64, device=dev) + rank * N) / N
        F = torch.sin(t[None, :, None] * w[None, None, :] + phi[:, None, None])
        noise = 0.1 * (2.0 * torch.rand((n1 - n0, T, p), dtype=torch.float64, device=dev, generator=g) - 1.0)
        Y[n0:n1] = F @ H.T + noise
    return Y


def check_stability(model, L):
    worst = {"rho_AKHA": 0.0, "rho_G_rts": 0.0}
    for l in range(L):
        c = model.latent_consts(l)
        G, _ = model.smoother_consts(l, 1)
        worst["rho_AKHA"] = max(worst["rho_AKHA"], float(np.max(np.abs(np.linalg.eigvals(c["AKHA"])))))
        worst["rho_G_rts"] = max(worst["rho_G_rts"], float(np.max(np.abs(np.linalg.eigvals(G)))))
    if worst["rho_AKHA"] >= 1.0 or worst["rho_G_rts"] >= 1.0:
        raise SystemExit("benchmark hyper-parameters are unstable under the reference's semantics: %s" % worst)
    return worst


def cpu_reference_rate(kind, kernel, p, L, N, T, seed, budget_s, nthreads, repeats=1, force_port=False):
    """Time the CPU implementation of the same pass on the host cores, on a bounded sample of the workload: as many
    sequences (full length when the workload has many, a T-prefix when it is one long sequence) as fit in ~budget_s
    seconds.  Filter + smoother + NLL: the reference's OWN classes (MOIHGP::step / negLogLikelihood / IHGP::
    backwardSmoother, compiled -O3 from /root/reference against the Eigen-API shim into oracle/_ref, one model object per
    host thread, threads over sequences) when that build exists, else the oracle port.  Objective: the oracle port (the
    reference's O(p^3 L^2)-per-step gradient loop cannot finish at these sizes).
    `repeats` > 1: the sample is sized once (budget_s seconds each) and timed `repeats` times; the rate and seconds
    returned are then lists.  Returns (latent-steps/s, sample description, seconds, threads used, kind)."""
    from oracle import binding
    from oracle.gen_golden import make_data
    params, Hmix = model_params(p, L, kernel, seed)
    rng = np.random.default_rng(seed)
    many = N >= nthreads
    use_ref = kind == "fsn" and binding.ref_pass_available() and not force_port
    if use_ref:
        Ts = T if many else min(T, 4000)
    else:
        Ts = T if many else min(T, 20000 if kind == "fsn" else 2000)
    base = make_data(rng, p, L, Ts, DT)

    if use_ref:
        import threading
        workers = [binding.RefPass(DT, p, L, kernel, params) for _ in range(nthreads)]

        def run(nseq):
            Y = np.ascontiguousarray(np.broadcast_to(base, (nseq, Ts, p))) + 0.01 * rng.standard_normal((nseq, 1, p))
            d = 3 if kernel == "Matern52" else 2
            outs = [(np.empty((Ts, L, d)), np.empty((Ts, L, d))) for _ in range(nthreads)]

            def work(k):
                for n in range(k, nseq, nthreads):
                    workers[k].run(Y[n], outs[k][0], outs[k][1], smooth=True)
            th = [threading.Thread(target=work, args=(k,)) for k in range(nthreads)]
            t0 = time.perf_counter()
            for t in th:
                t.start()
            for t in th:
                t.join()
            return time.perf_counter() - t0
        n0, used, what_impl = nthreads, nthreads, "reference classes (-O3, Eigen-API shim), one model per thread, threads over sequences"
    else:
        o = binding.OracleMOIHGP(DT, p, L, kernel, threading=True)
        o.update(params)

        def run(nseq):
            Y = np.ascontiguousarray(np.broadcast_to(base, (nseq, Ts, p))) + 0.01 * rng.standard_normal((nseq, 1, p))
            t0 = time.perf_counter()
            if kind == "fsn":
                o.filter_smoother_nll(Y, smoother_mode=1, nthreads=nthreads)
            else:
                o.objective(Y)       # single thread: the reference's objective loop is sequential (moihgp_regression.h:42-50)
            return time.perf_counter() - t0
        n0 = max(nthreads, 1) if kind == "fsn" else 1
        used = nthreads if kind == "fsn" else 1
        what_impl = "oracle/moihgp_oracle.cpp -O3" + (", std::thread over sequences" if used > 1 else ", one thread")

    t_cal = run(n0)
    cap = 4096 if many else 64 * n0
    nseq = int(max(n0, min(cap, n0 * budget_s / max(t_cal, 1e-3))))
    nseq = (nseq // n0) * n0
    times = [run(nseq) for _ in range(repeats)]
    dt_ = times[0] if repeats == 1 else times
    what = ("%d full-length sequences of the workload (T=%d)" % (nseq, Ts)) if many else \
           ("%d copies of a T=%d prefix of the workload's single sequence (T=%d)" % (nseq, Ts, T))
    rate = nseq * Ts * L / dt_ if repeats == 1 else [nseq * Ts * L / t for t in times]
    return rate, what + ", " + what_impl, dt_, used, ("reference" if use_ref else "port")


def workload_setup(name, nseq=0, tlen=0):
    kind, kernel, p, L, N, T = WORKLOADS[name]
    if nseq:
        N = nseq
    if tlen:
        T = tlen
    d = 3 if kernel == "Matern52" else 2
    seed = 1234 + {"c3": 2, "c4": 3, "c5": 4}[name]   # SURVEY 8(d): 1234 + config index
    metric = METRIC if kind == "fsn" else "latent time-steps/sec (NLL+gradient objective, fp64)"
    ybytes = 8.0 * N * T * p
    cfg = {"workload": WORKLOAD_DESC[name], "kernel": kernel, "p": p, "L": L, "d": d, "sequences_per_gpu": N, "T": T,
           "dt": DT, "pass": "filter + RTS smoother + NLL (writes X, Xs, nll); smoother_mode = RTS (this library's extension: the reference's "
                             "literal IHGP::backwardSmoother, which the reference arm runs, does the same work per step but is unstable for "
                             "the default Matern-3/2 latent, SURVEY Q3)" if kind == "fsn" else "NLL + gradient (writes loss, grad[num_param])",
           "sharding": "sequences over ranks, no data-path collective; all-reduce of the summed NLL only" if kind == "fsn"
                       else "independent sequences over ranks; fp64 all-reduce of [loss, grad]",
           "l2": "inputs (%.1f GB/GPU) larger than L2 (126 MB), no flush needed" % (ybytes / 1e9)}
    return kind, kernel, p, L, N, T, d, seed, metric, cfg


def source_hash():
    """sha256 over the CUDA sources: profiles/traffic.json is only quoted while it describes THESE kernels."""
    import glob
    import hashlib
    h = hashlib.sha256()
    for f in sorted(glob.glob(os.path.join(ROOT, "multioutputihgp_b200", "csrc", "*"))):
        if f.endswith((".cu", ".cuh", ".h")):
            h.update(os.path.basename(f).encode())
            h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


FP64_PEAK_TFLOPS = 37.0   # measured here: scripts/microbench/fp64_rate.cu, profiles/r01/fp64_rate_microbench.txt (DMMA m8n8k4)


def objective_flops_per_step(p, L, d):
    """SURVEY 8(d): algorithmic flops of one sequence-step of the NLL + gradient objective"""
    K = 3
    return 6.0 * p * L + L * (2 * d * d + 2 * d + K * (4 * d * d + 2 * d) + 4 * K * d + 30)


def emit(line):
    """The ONE JSON line goes to the process's real stdout; everything else printed while running (NCCL's version
    banner, library chatter) was redirected to stderr by main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1

DUMP_BUDGET = 60 << 20     # bytes of array data --dump-outputs writes: with the .npy headers, under 64 MB


def dump_outputs(torch, path, arrays, seed=0):
    """Write each array (a tensor on any device) as path/<name>.npy in float64.  Together they stay within DUMP_BUDGET: an
    array too large for its share is reduced to a fixed, seeded sample of its rows along the first two axes (the same rows
    on every run of the same workload), in ascending order."""
    os.makedirs(path, exist_ok=True)
    share = DUMP_BUDGET // len(arrays)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() * 8 > share:
            rows = t.reshape(t.shape[0] * t.shape[1], -1) if t.dim() > 1 else t.reshape(-1, 1)
            keep = max(1, share // (8 * rows.shape[1]))
            idx = np.sort(np.random.default_rng(seed).choice(rows.shape[0], size=keep, replace=False))
            t = rows[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.to(torch.float64).cpu().numpy())


def run_ours(a, wl, torch, dist, rank, local_rank, world, steps, warmup, cores, with_e2e, with_cpu, nseq=0, tlen=0, shard="auto"):
    """One workload on this rank's GPU: device-resident timed region (+ e2e through the host-buffer C ABI, + CPU baseline).
    Returns the JSON line (rank 0) or None.
    shard: "sequences" = weak scaling (every rank its own sequences); "time" = STRONG scaling of the objective (BASELINE
    configs[4]: the ONE sequence of T steps is cut into contiguous blocks of time, one per rank; carry exchange by NCCL
    all-gather + a device kernel, [loss, grad] by NCCL all-reduce); "auto" = time for the objective when world > 1."""
    kind, kernel, p, L, N, T, d, seed, metric, cfg = workload_setup(wl, nseq, tlen)
    time_shard = kind == "obj" and world > 1 and shard in ("auto", "time")
    T_total = T
    if time_shard:
        from multioutputihgp_b200.parallel import time_block_bounds_aligned
        bounds = [time_block_bounds_aligned(T_total, world, r) for r in range(world)]
        t_lo, t_hi = bounds[rank]
        T = t_hi - t_lo
        cfg["sharding"] = ("ONE sequence cut into %d contiguous blocks of time (whole 256-step chunks), one per rank: begin -> NCCL all-gather of "
                           "the block ends (L*d*4 doubles per rank) -> carry-in kernel -> finish -> NCCL all-reduce of [loss, grad]; no host "
                           "round trip inside an evaluation" % world)
        cfg["T_per_gpu"] = [b[1] - b[0] for b in bounds]
    dev = torch.device("cuda", local_rank)
    from multioutputihgp_b200 import MOIHGPSequences
    model = MOIHGPSequences(DT, p, L, kernel, threading=True, device=local_rank)
    params, Hmix = model_params(p, L, kernel, seed)
    model.update(params)
    model.set_path(a.path if wl == a.workload else "auto")
    model.set_chain_seqs_per_warp(a.spw if wl == a.workload else 0)
    stab = check_stability(model, L)

    if time_shard:
        # every rank builds the SAME whole sequence (rank 0's seed) and keeps its block: loss_total is then comparable with
        # the one-GPU evaluation of the same workload
        Yfull = make_data_device(torch, dev, Hmix, N, T_total, p, L, seed, 0)
        Y = Yfull[:, t_lo:t_hi].contiguous()
        del Yfull
        torch.cuda.empty_cache()
    else:
        Y = make_data_device(torch, dev, Hmix, N, T, p, L, seed, rank)
    if kind == "fsn":
        X = torch.empty((N, T, L, d), dtype=torch.float64, device=dev)
        Xs = torch.empty_like(X)
        nll = torch.empty(N, dtype=torch.float64, device=dev)
        out = torch.zeros(1, dtype=torch.float64, device=dev)       # summed NLL (all-reduced)

        def device_pass():
            model.filter_smoother_nll_device(Y, smoother_mode=1, X=X, Xs=Xs, nll=nll)

        def step():
            device_pass()
            torch.sum(nll, dim=0, keepdim=True, out=out)
            if world > 1 and not os.environ.get("BENCH_SKIP_ALLREDUCE"):      # (diagnosis only: isolates the collective's cost)
                dist.all_reduce(out)
    elif time_shard:
        from multioutputihgp_b200.parallel import TimeShardedDeviceObjective
        tso = TimeShardedDeviceObjective(model, [b[1] - b[0] for b in bounds], num_sequences=N)
        out = tso.buf                                                              # [loss, pad, grad...] (all-reduced in enqueue)

        def step():
            tso.enqueue(Y)
    else:
        out = torch.zeros(2 + model.num_param, dtype=torch.float64, device=dev)   # [loss, pad, grad...] (all-reduced)

        def device_pass():
            model.objective_device(Y, out[0:1], out[2:])

        def step():
            device_pass()
            if world > 1:
                dist.all_reduce(out)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank) if rank == 0 else None     # started before the warm-up: nvidia-smi needs ~0.3 s to produce its first line
    for _ in range(warmup):
        step()
    sync_all()
    if sampler:
        sampler.mark_timed_region_start()
    l0 = model.launch_count
    model.profile(True)    # one CUDA event after every kernel of the library, on the launching stream, inside the timed region
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    sync_all()
    prof = model.profile_read()
    model.profile(False)
    launches = model.launch_count - l0
    clocks = sampler.stop() if sampler else None
    ms = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(ms.item())
    units = float(N) * T_total * L if time_shard else float(N) * T * L * world
    value = units / (ms_per_step * 1e-3)
    result_scalar = float(out[0].item())
    if a.dump_outputs and wl == a.workload and rank == 0:
        # what the timed path returned in its last step (this rank's share of it)
        if kind == "fsn":
            dump_outputs(torch, a.dump_outputs, {"X": X, "Xs": Xs, "nll": nll}, seed)
        else:
            dump_outputs(torch, a.dump_outputs, {"loss": out[0:1], "grad": out[2:]}, seed)

    # per-kernel device times: the events recorded during the timed steps above.  Event-bracketed kernel times add up
    # to ~5-10 % more than the event-bracketed loop (an event between two kernels costs a drain the plain stream does
    # not pay), so the roofline figure uses the loop time and the per-kernel events only give each kernel's share.
    kern = {k: v[0] / v[1] for k, v in prof.items()}
    ksum = sum(kern.values())
    peak, peak_src = measured_peak()
    balg = alg_bytes_per_latent_step(kind, p, L, d)
    dom = max(kern, key=kern.get)
    # bytes each kernel must move by construction (its own compulsory traffic, per launch)
    NT = float(N) * T
    own = {"k_project": 8.0 * NT * (p + L + 1) if kind == "fsn" else 8.0 * NT * (p + 3 * L + 1),
           "k_scan_summaries": 8.0 * NT * L, "k_scan_final": 8.0 * NT * L * (1 + 2 * d),
           "k_filter_chain": 8.0 * NT * (p + L * d), "k_smooth_chain": 8.0 * NT * 2 * L * d,
           "k_obj_scan_summaries": 8.0 * NT * L, "k_obj_scan_final": 8.0 * NT * 4 * L, "k_gradU": 8.0 * NT * (p + L)}
    pass_ms = ms_per_step       # one step = one fused pass (+ the 32 KB NLL sum / all-reduce)
    roof = {"bound": "hbm", "kernel": "fused pass = " + " + ".join(kern.keys()),
            "achieved": balg * N * T * L / (pass_ms * 1e-3) / 1e9, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
            "traffic": None, "algorithmic_bytes_per_latent_step": balg, "pass_ms": pass_ms,
            "kernels_ms_event_bracketed": {k: round(v, 4) for k, v in kern.items()},
            "kernel_share": {k: round(v / ksum, 4) for k, v in kern.items()},
            "dominant": {"kernel": dom, "share": kern[dom] / ksum, "ms": pass_ms * kern[dom] / ksum, "own_bytes": own.get(dom),
                         "own_GBps": (own[dom] / (pass_ms * kern[dom] / ksum * 1e-3) / 1e9) if dom in own else None}}
    roof["frac"] = roof["achieved"] / peak
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f).get(wl, {})
        # DRAM bytes per step from the ncu --set full capture of this workload; quoted only while the capture describes the
        # kernels that just ran (same source hash, same size) - otherwise null, never a stale constant
        if tj.get("source_hash") == source_hash() and not nseq and not tlen:
            roof["traffic"] = tj.get("fused_pass_dram_bytes_per_step")
            roof["traffic_source"] = tj.get("source")
        else:
            roof["traffic_note"] = "profiles/traffic.json was captured with other kernel sources (hash %s, now %s) or another size" % (tj.get("source_hash"), source_hash())
    except Exception:
        pass
    if kind == "obj":
        fl = objective_flops_per_step(p, L, d) * N * T
        roof["fp64"] = {"flops_per_step": fl, "achieved_tflops": fl / (pass_ms * 1e-3) / 1e12, "peak_tflops": FP64_PEAK_TFLOPS,
                        "frac": fl / (pass_ms * 1e-3) / 1e12 / FP64_PEAK_TFLOPS,
                        "note": "this pass is FP64-compute-bound (48 flop/B), not HBM-bound: SURVEY 8(d)"}

    # ------------------------------------------------------------------ e2e: host buffers through the C ABI
    e2e = None
    if with_e2e and not time_shard:
        import psutil
        lib, h = model._lib, model._h
        model.set_stream(None)
        if kind == "fsn":
            need = 8.0 * N * T * (p + 2 * L * d) * 1.05
            avail = psutil.virtual_memory().available / max(world, 1)
            Ne = N if need < 0.7 * avail else max(1, int(N * 0.7 * avail / need))
            del X, Xs
            torch.cuda.empty_cache()
            Yh = torch.empty((Ne, T, p), dtype=torch.float64, pin_memory=True)
            Yh.copy_(Y[:Ne])
            Xh = torch.empty((Ne, T, L, d), dtype=torch.float64, pin_memory=True)
            Xsh = torch.empty((Ne, T, L, d), dtype=torch.float64, pin_memory=True)
            nllh = torch.empty(Ne, dtype=torch.float64, pin_memory=True)

            def e2e_step():
                rc = lib.moihgp_cuda_filter_smoother_nll(h, Yh.data_ptr(), Ne, T, None, 1, Xh.data_ptr(), Xsh.data_ptr(), None, nllh.data_ptr(), None)
                if rc != 0:
                    raise SystemExit("e2e call failed: " + lib.moihgp_cuda_last_error(h).decode())
            api, h2d, d2h = "moihgp_cuda_filter_smoother_nll (host buffers, pinned)", int(8 * Ne * T * p), int(8 * Ne * (2 * T * L * d + 1))
        else:
            Ne = N
            Yh = torch.empty((Ne, T, p), dtype=torch.float64, pin_memory=True)
            Yh.copy_(Y)
            lossh = torch.zeros(1, dtype=torch.float64, pin_memory=True)
            gradh = torch.zeros(model.num_param, dtype=torch.float64, pin_memory=True)

            def e2e_step():
                rc = lib.moihgp_cuda_objective(h, Yh.data_ptr(), Ne, T, None, None, lossh.data_ptr(), gradh.data_ptr(), None, None)
                if rc != 0:
                    raise SystemExit("e2e call failed: " + lib.moihgp_cuda_last_error(h).decode())
            api, h2d, d2h = "moihgp_cuda_objective (host buffers, pinned)", int(8 * Ne * T * p), int(8 * (1 + model.num_param))

        ke = max(2, min(steps, 3))
        e2e_step()   # warm-up (allocates the call's device buffers)
        sync_all()
        t0 = time.perf_counter()
        for _ in range(ke):
            e2e_step()
        sync_all()
        te = torch.tensor([(time.perf_counter() - t0) / ke], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        if kind == "fsn":
            ref_val, got = float(nll[:Ne].sum().item()), float(nllh.sum().item())
        else:
            model.objective_device(Y, out[0:1], out[2:])      # this rank's own loss (no all-reduce)
            torch.cuda.synchronize(dev)
            ref_val, got = float(out[0].item()), float(lossh.item())
        e2e = {"value": float(Ne) * T * L * world / float(te.item()), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * float(te.item()), "sequences_per_gpu": Ne,
               "api": api, "steps": ke, "result_check": abs(got - ref_val) <= 1e-9 * abs(ref_val)}
        if kind == "fsn":
            # second figure: the same call returning only the function-value component H x of the filtered / smoothed states
            # ([N,T,L]: what predict-style callers consume) - d times fewer bytes from the device to the host
            del Xh, Xsh
            Fh = torch.empty((Ne, T, L), dtype=torch.float64, pin_memory=True)
            Fsh = torch.empty((Ne, T, L), dtype=torch.float64, pin_memory=True)

            def e2e_values_step():
                rc = lib.moihgp_cuda_filter_smoother_nll_values(h, Yh.data_ptr(), Ne, T, None, 1, Fh.data_ptr(), Fsh.data_ptr(), None, nllh.data_ptr(), None)
                if rc != 0:
                    raise SystemExit("e2e (values) call failed: " + lib.moihgp_cuda_last_error(h).decode())
            e2e_values_step()
            sync_all()
            t0 = time.perf_counter()
            for _ in range(ke):
                e2e_values_step()
            sync_all()
            tv = torch.tensor([(time.perf_counter() - t0) / ke], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tv, op=dist.ReduceOp.MAX)
            e2e["function_values_only"] = {"value": float(Ne) * T * L * world / float(tv.item()), "unit": UNIT, "ms_per_step": 1e3 * float(tv.item()),
                                           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(8 * Ne * (2 * T * L + 1)),
                                           "api": "moihgp_cuda_filter_smoother_nll_values (host buffers, pinned): F, Fs [N,T,L] + nll",
                                           "result_check": abs(float(nllh.sum().item()) - ref_val) <= 1e-9 * abs(ref_val)}
            e2e["host_topology_note"] = ("the timed copies run at PCIe speed (D2H of X, Xs dominates); with N ranks the pinned traffic of all "
                                         "ranks shares one host memory system - on this pool every GPU reports CPU affinity 0-31 / NUMA node 0, "
                                         "so there is no second node to bind to")

    # ------------------------------------------------------------------ CPU baseline beside it (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and with_cpu:
        r, what, dt_, used, ckind = cpu_reference_rate(kind, kernel, p, L, N, T, seed, budget_s=a.cpu_seconds, nthreads=cores)
        cpu = {"value": r, "unit": UNIT, "cores": used, "kind": ckind, "sample": "%s, %.1f s" % (what, dt_)}
        if ckind == "reference":
            # next to the reference's own classes (eager Eigen-style temporaries on the shim): the oracle port of the same
            # algorithm (oracle/moihgp_oracle.cpp, plain loops), on one core and on all of them (BASELINE.md section 3)
            port = {}
            for tag, nt in (("1_core", 1), ("all_cores", cores)):
                rp, whatp, dtp, usedp, _ = cpu_reference_rate(kind, kernel, p, L, N, T, seed, budget_s=min(3.0, a.cpu_seconds), nthreads=nt, force_port=True)
                port[tag] = {"value": rp, "unit": UNIT, "cores": usedp, "sample": "%s, %.1f s" % (whatp, dtp)}
            cpu["oracle_port"] = port

    if rank == 0:
        line = {"metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "strong" if time_shard else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": cfg, "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
                "hbm_GBps_alg": balg * units / world / (ms_per_step * 1e-3) / 1e9,
                ("nll_total" if kind == "fsn" else "loss_total"): result_scalar, "stability": stab}
        return line
    return None


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--nseq", type=int, default=0, help="override sequences per GPU (debug only: not the benchmark config)")
    ap.add_argument("--tlen", type=int, default=0, help="override T (debug only)")
    ap.add_argument("--path", default="auto", choices=["auto", "scan", "chain"], help="force a kernel path (debug only)")
    ap.add_argument("--spw", type=int, default=0, help="many-chains kernels: sequences per warp (debug only; 0 = automatic)")
    ap.add_argument("--shard", default="auto", choices=["auto", "time", "sequences"],
                    help="multi-GPU objective (c5): 'time' = one sequence cut into blocks of time (strong scaling, the default for c5), "
                         "'sequences' = independent sequences per rank (weak scaling)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the extra configs[3] / configs[4] device passes of the default run")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy (float64, at most 64 MB in all: "
                         "a fixed, seeded sample of the rows of a larger output); GPU path only, with N > 1 GPUs rank 0's share")
    a = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    steps, warmup = max(a.steps, 1), max(a.warmup, 3)
    cores = len(os.sched_getaffinity(0))
    kind, kernel, p, L, N, T, d, seed, metric, cfg = workload_setup(a.workload, a.nseq, a.tlen)

    # ------------------------------------------------------------------ reference arm (CPU)
    if a.impl == "reference":
        if a.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs writes the GPU path's outputs; --impl reference has none to write")
        if rank != 0:
            return
        t0 = time.perf_counter()
        # every step is the same bounded sample, sized so that warmup + steps of them take about two minutes
        per = max(1.0, min(10.0, 120.0 / (warmup + steps)))
        r, what, dts, used, ckind = cpu_reference_rate(kind, kernel, p, L, N, T, seed, budget_s=per, nthreads=cores, repeats=warmup + steps)
        rates = r[warmup:]
        samples = [(what, t) for t in dts[warmup:]]
        value = float(np.mean(rates))
        sample = samples[-1][0] + " per step"
        line = {"impl": "reference", "metric": metric, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": steps, "warmup": warmup,
                "ms_per_step": 1e3 * float(np.mean([s[1] for s in samples])), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": ckind, "sample": sample},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "kind=reference: the reference's own classes (MOIHGP::step v3 + negLogLikelihood(x,y) per observation, then "
                        "IHGP::backwardSmoother per latent) compiled from /root/reference against the Eigen-API shim (Eigen itself is "
                        "absent from the image), literal smoother; kind=port: oracle/moihgp_oracle.cpp; wall %.0f s" % (time.perf_counter() - t0)}
        emit(line)
        return

    # ------------------------------------------------------------------ our arm (B200)
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    line = run_ours(a, a.workload, torch, dist, rank, local_rank, world, steps, warmup, cores, not a.no_e2e, not a.no_cpu, a.nseq, a.tlen, a.shard)
    # the other single-GPU BASELINE configurations, device-resident passes only (a second or two each), so that the one
    # line the driver records also witnesses configs[3] and configs[4]
    if world == 1 and a.workload == "c3" and not a.no_also and not a.nseq and not a.tlen:
        also = {}
        for wl in ("c4", "c5"):
            torch.cuda.empty_cache()
            sub = run_ours(a, wl, torch, dist, rank, local_rank, world, min(steps, 10), warmup, cores, False, False)
            r = sub["roofline"]
            also[wl] = {"workload": sub["config"]["workload"], "metric": sub["metric"], "value": sub["value"], "unit": sub["unit"],
                        "ms_per_step": sub["ms_per_step"], "steps": sub["steps"], "gpu_launches": sub["gpu_launches"], "clocks": sub["clocks"],
                        "result_total": sub.get("nll_total", sub.get("loss_total")),
                        "roofline": {k: r.get(k) for k in ("bound", "achieved", "peak", "unit", "frac", "traffic", "traffic_note",
                                                           "algorithmic_bytes_per_latent_step", "kernels_ms_event_bracketed", "fp64")}}
        line["also"] = also
    # BASELINE configs[4] as quoted ("NLL+gradient sharded over 8 GPUs with NCCL all-reduce"): the ONE T = 1e6 sequence
    # sharded in TIME over the ranks of this run - strong scaling, next to the weak-scaling headline
    if world > 1 and a.workload == "c3" and not a.no_also and not a.nseq and not a.tlen:
        torch.cuda.empty_cache()
        sub = run_ours(a, "c5", torch, dist, rank, local_rank, world, min(steps, 20), warmup, cores, False, False, shard="time")
        if rank == 0:
            line["also"] = {"c5_time_sharded": {"workload": sub["config"]["workload"], "sharding": sub["config"]["sharding"], "metric": sub["metric"],
                                                "value": sub["value"], "unit": sub["unit"], "ms_per_step": sub["ms_per_step"], "scaling": sub["scaling"],
                                                "n_gpus": world, "steps": sub["steps"], "gpu_launches": sub["gpu_launches"], "clocks": sub["clocks"],
                                                "loss_total": sub.get("loss_total"),
                                                "kernels_ms_event_bracketed": sub["roofline"]["kernels_ms_event_bracketed"]}}
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
