"""2+ GPU check of the time-sharded filter + smoother + NLL pass (run under torchrun): one long sequence (BASELINE config-4
shape), a block of time per rank, forward carry exchange + mirror-image backward exchange by all-gather, NLL by NCCL
all-reduce; compared with the whole sequence on one GPU.  Prints one summary line."""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from bench import model_params, DT
from multioutputihgp_b200 import MOIHGPSequences
from multioutputihgp_b200.parallel import TimeShardedFilterSmoother, time_block_bounds_aligned

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
# TS_BACKEND=gloo: the ranks share the visible GPUs (rank r on device r % device_count) and exchange through gloo - lets a
# ONE-GPU box run the whole protocol with two ranks (NCCL refuses two ranks on one device)
backend = os.environ.get("TS_BACKEND", "nccl")
local = local % torch.cuda.device_count() if backend == "gloo" else local
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if backend == "gloo":
    dist.init_process_group("gloo")
else:
    dist.init_process_group("nccl", device_id=dev)
p, L, T, kernel = int(os.environ.get("TS_P", 64)), int(os.environ.get("TS_L", 32)), int(os.environ.get("TS_T", 2000000)), "Matern32"
params, Hmix = model_params(p, L, kernel, 4321)
m = MOIHGPSequences(DT, p, L, kernel, threading=True, device=local)
m.update(params)
d = m.igp_dim
rng = np.random.default_rng(99)                      # every rank builds the same sequence and keeps its block
t = np.arange(T) * DT
F = np.sin(t[:, None] * (1.0 + 3.0 * np.arange(L) / max(L - 1, 1))[None, :])
Y = F @ Hmix.T + 0.1 * (2 * rng.random((T, p)) - 1)
bounds = [time_block_bounds_aligned(T, world, r) for r in range(world)]
t0_b, t1_b = bounds[rank]
Yb = torch.from_numpy(np.ascontiguousarray(Y[t0_b:t1_b])).to(dev)[None].contiguous()
X = torch.zeros((1, t1_b - t0_b, L, d), dtype=torch.float64, device=dev)
Xs = torch.zeros_like(X)
fs = TimeShardedFilterSmoother(m, [b[1] - b[0] for b in bounds], 1)
fs(Yb, X, Xs)                                         # warm-up
torch.cuda.synchronize(dev)
dist.barrier()
tic = time.perf_counter()
nll_call = fs(Yb, X, Xs)                              # __call__ = enqueue + synchronise
torch.cuda.synchronize(dev)
dist.barrier()
t_call = time.perf_counter() - tic
Xc, Xsc = X.clone(), Xs.clone()
X.zero_(); Xs.zero_()
for _ in range(2):                                    # device-side exchange: nothing leaves the stream (warm-up, then timed)
    torch.cuda.synchronize(dev)
    dist.barrier()
    tic = time.perf_counter()
    nll = fs.enqueue(Yb, X, Xs)
    torch.cuda.synchronize(dev)
    dist.barrier()
    t_shard = time.perf_counter() - tic
nll = nll.cpu().numpy()
assert torch.equal(X, Xc) and torch.equal(Xs, Xsc) and np.array_equal(nll, nll_call)
# every rank checks its own block against the whole-sequence pass computed on rank 0
if rank == 0:
    Yd = torch.from_numpy(Y).to(dev)[None].contiguous()
    Xw = torch.zeros((1, T, L, d), dtype=torch.float64, device=dev)
    Xsw = torch.zeros_like(Xw)
    nllw = torch.zeros(1, dtype=torch.float64, device=dev)
    m.set_path("scan")
    m.filter_smoother_nll_device(Yd, smoother_mode=1, X=Xw, Xs=Xsw, nll=nllw)
    torch.cuda.synchronize(dev)
    tic = time.perf_counter()
    m.filter_smoother_nll_device(Yd, smoother_mode=1, X=Xw, Xs=Xsw, nll=nllw)
    torch.cuda.synchronize(dev)
    t_one = time.perf_counter() - tic
    scale_x, scale_s = float(Xw.abs().max()), float(Xsw.abs().max())
    e_x = float((X - Xw[:, t0_b:t1_b]).abs().max()) / scale_x
    e_s = float((Xs - Xsw[:, t0_b:t1_b]).abs().max()) / scale_s
    e_n = abs(float(nll[0]) - float(nllw[0])) / abs(float(nllw[0]))
    # the other ranks' blocks: gather their first / last rows through the host is overkill - compare the block borders
    print("time-sharded filter+smoother+NLL: world=%d p=%d L=%d T=%d  rank-0 block rel.err X %.2e Xs %.2e, nll %.2e | wall: sharded %.2f ms (__call__ = enqueue + sync %.2f ms), one GPU %.2f ms"
          % (world, p, L, T, e_x, e_s, e_n, 1e3 * t_shard, 1e3 * t_call, 1e3 * t_one))
    assert e_x < 1e-9 and e_s < 1e-9 and e_n < 1e-9
    ref_tail = (Xw[:, -1].cpu().numpy(), Xsw[:, -1].cpu().numpy(), Xsw[:, bounds[-1][0]].cpu().numpy())
    tail = torch.from_numpy(np.concatenate([a.ravel() for a in ref_tail])).to(dev)
else:
    tail = torch.zeros(3 * L * d, dtype=torch.float64, device=dev)
dist.broadcast(tail, src=0)
if rank == world - 1:                                 # the last rank checks its own block's first and last rows
    rt = tail.cpu().numpy().reshape(3, L, d)
    mine = (X[0, -1].cpu().numpy(), Xs[0, -1].cpu().numpy(), Xs[0, 0].cpu().numpy())
    for a, b in zip(mine, rt):
        assert np.max(np.abs(a - b)) <= 1e-9 * max(np.max(np.abs(b)), 1e-300), "last block differs from the whole-sequence pass"
    print("last rank: block borders agree with the whole-sequence pass")
dist.destroy_process_group()
