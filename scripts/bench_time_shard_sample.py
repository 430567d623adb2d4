"""Posterior sample paths of one long sequence sharded in time (run under torchrun; one rank = the whole-sequence call).

Config-4 shape (N = 1, p = 64, L = 32, Matern-3/2, d = 2) at TS_T steps (default 8e6), S = TS_S samples (default 4), two
outputs: values only (Fsamp [S][N][T][L]) and full states (Xsamp [S][N][T][L][d]).  With one rank it times
sample_posterior_device on the whole sequence; with G ranks it times TimeShardedPosteriorSampler.enqueue end to end, then the
same steps one by one between CUDA events: the time-sharded RTS mean, sampler phase 1, the all-gather of the starts, the
carry kernel and phase 2.  Medians over TS_REPS calls after one warm-up; the per-rank maximum over ranks.  With full states
the last rank checks its paths against the noise recomputed in NumPy on windows of steps (e at the window's end taken from
the output).  Prints one JSON line per output kind, with the card's name and power limit read in the same run."""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np
import torch
import torch.distributed as dist

from bench import model_params, DT
from multioutputihgp_b200 import MOIHGPSequences
from multioutputihgp_b200.parallel import TimeShardedPosteriorSampler, time_block_bounds_aligned
from test_gpu_sampling import normals

rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
p, L, kernel = 64, 32, "Matern32"
T, S, reps = int(float(os.environ.get("TS_T", 8e6))), int(os.environ.get("TS_S", 4)), int(os.environ.get("TS_REPS", 3))
seed = 0x5A3D_0000_0004
params, Hmix = model_params(p, L, kernel, 4321)
m = MOIHGPSequences(DT, p, L, kernel, threading=True, device=local)
m.update(params)
d = m.igp_dim
bounds = [time_block_bounds_aligned(T, world, r) for r in range(world)]
lengths = [b[1] - b[0] for b in bounds]
t0, t1 = bounds[rank]
n, last = t1 - t0, rank == world - 1
f64 = dict(dtype=torch.float64, device=dev)
# the block of a deterministic sequence, generated on the device from the global step
tt = (t0 + torch.arange(n, device=dev, dtype=torch.float64)) * DT
Fl = torch.sin(tt[:, None] * (1.0 + 3.0 * torch.arange(L, device=dev, dtype=torch.float64) / (L - 1))[None, :])
Yb = (Fl @ torch.from_numpy(Hmix.T.copy()).to(dev) + 0.05 * torch.cos(7.3 * tt[:, None] + torch.arange(p, device=dev)[None, :]))[None].contiguous()
del Fl


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)], capture_output=True, text=True)
    return q.stdout.strip()


def timed(fn):
    """median ms over reps of fn() between CUDA events (after one warm-up), the maximum over ranks"""
    fn()
    ts = []
    for _ in range(reps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    v = torch.tensor([float(np.median(ts))], **f64)
    if world > 1:
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
    return float(v.item())


def steps_timed(sampler, outs):
    """the steps of enqueue one by one between events (median per step over reps, maximum over ranks)"""
    b = sampler._buffers(1, n, S)
    Xs = b._Xs
    steps = [("mean", lambda: sampler.mean.enqueue(Yb, b._X, Xs)),
             ("phase1", lambda: m.sample_block_async(1, Xs, S, seed, t0, last, out=b._e1)),
             ("all_gather", lambda: sampler.mean._all_gather(b._eg, b._e1)),
             ("carry", lambda: m.fsn_carry_device(1, b._eg, lengths, rank, b._eend, smoother_mode=1)),
             ("phase2", lambda: m.sample_block_async(2, Xs, S, seed, t0, last, e_end=None if last else b._eend, **outs))]
    rec = {k: [] for k, _ in steps}
    for it in range(reps + 1):
        dist.barrier()
        torch.cuda.synchronize(dev)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(steps) + 1)]
        ev[0].record()
        for i, (_, fn) in enumerate(steps):
            fn()
            ev[i + 1].record()
        ev[-1].synchronize()
        if it:
            for i, (k, _) in enumerate(steps):
                rec[k].append(ev[i].elapsed_time(ev[i + 1]))
    v = torch.tensor([float(np.median(rec[k])) for k, _ in steps], **f64)
    dist.all_reduce(v, op=dist.ReduceOp.MAX)
    return {k: round(float(x), 3) for (k, _), x in zip(steps, v.tolist())}


def window_check(X, Xs):
    """worst rel. error of X - Xs against the NumPy noise on windows of 64 steps at the block's start, middle and end"""
    G_ = np.stack([m.smoother_consts(l, 1)[0] for l in range(L)])
    LF, LC = (np.stack(f) for f in zip(*[m.sampler_consts(l) for l in range(L)]))
    worst = 0.0
    for a in (0, n // 2, n - 64):
        e = (X[:, 0, a:a + 64] - Xs[0, a:a + 64][None]).cpu().numpy()                       # [S, 64, L, d]
        z = normals(seed, np.arange(S)[:, None, None], 0, np.arange(L)[None, None, :], t0 + a + np.arange(64)[None, :, None], d)
        ref = np.empty_like(e)
        if a + 64 == n and last:
            ref[:, 63] = np.einsum("lij,slj->sli", LF, z[:, 63])
        else:
            nxt = (X[:, 0, a + 64] - Xs[0, a + 64][None]).cpu().numpy() if a + 64 < n else None
            if nxt is None:                                     # a block's last step of a non-final block: e_end from the next
                ref[:, 63] = e[:, 63]
            else:
                ref[:, 63] = np.einsum("lij,slj->sli", G_, nxt) + np.einsum("lij,slj->sli", LC, z[:, 63])
        for j in range(62, -1, -1):
            ref[:, j] = np.einsum("lij,slj->sli", G_, ref[:, j + 1]) + np.einsum("lij,slj->sli", LC, z[:, j])
        worst = max(worst, float(np.max(np.abs(e - ref)) / np.max(np.abs(ref))))
    return worst


for kind in ("values", "states"):
    out = {"Fsamp": torch.zeros((S, 1, n, L), **f64)} if kind == "values" else {"Xsamp": torch.zeros((S, 1, n, L, d), **f64)}
    rec = {"workload": "time-sharded posterior sampling, config-4 shape", "p": p, "L": L, "N": 1, "T": T, "S": S, "output": kind,
           "gpus": world, "reps": reps}
    if world == 1:
        Xs = torch.zeros((1, T, L, d), **f64)
        key = {"Fsamp": "F", "Xsamp": "X"}
        kw = {key[k]: v for k, v in out.items()}
        rec["whole_sequence_ms"] = round(timed(lambda: m.sample_posterior_device(Yb, seed, Xs=Xs, **kw)), 3)
        if kind == "states":
            rec["noise_window_rel_err"] = window_check(out["Xsamp"], Xs)
    else:
        sampler = TimeShardedPosteriorSampler(m, lengths)
        rec["end_to_end_ms"] = round(timed(lambda: sampler.enqueue(Yb, S, seed, **out)), 3)
        rec["steps_ms"] = steps_timed(sampler, out)
        if kind == "states":
            err = torch.tensor([window_check(out["Xsamp"], sampler._Xs)], **f64)
            dist.all_reduce(err, op=dist.ReduceOp.MAX)
            rec["noise_window_rel_err"] = float(err.item())
    rec["card"] = card()
    if rank == 0:
        print(json.dumps(rec), flush=True)
    del out
    torch.cuda.empty_cache()
if world > 1:
    dist.destroy_process_group()
