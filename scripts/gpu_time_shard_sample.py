"""2+ rank check of the time-sharded posterior sampler (run under torchrun): one long sequence, a block of time per rank,
TimeShardedPosteriorSampler (time-sharded RTS mean, sampler phase 1, all-gather, backward carry kernel, phase 2); every rank
compares its block with the whole-sequence call (sample_posterior_device, same seed) on its own device and prints one line.
TS_BACKEND=gloo lets the ranks share the visible GPUs (rank r on device r % device_count)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from bench import model_params, DT
from multioutputihgp_b200 import MOIHGPSequences
from multioutputihgp_b200.parallel import TimeShardedPosteriorSampler, time_block_bounds_aligned

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
backend = os.environ.get("TS_BACKEND", "nccl")
local = local % torch.cuda.device_count() if backend == "gloo" else local
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if backend == "gloo":
    dist.init_process_group("gloo")
else:
    dist.init_process_group("nccl", device_id=dev)
p, L, T, S, kernel = int(os.environ.get("TS_P", 64)), int(os.environ.get("TS_L", 32)), int(os.environ.get("TS_T", 200000)), int(os.environ.get("TS_S", 2)), "Matern32"
seed = 0x5A3D_0000_0001
params, Hmix = model_params(p, L, kernel, 4321)
m = MOIHGPSequences(DT, p, L, kernel, threading=True, device=local)
m.update(params)
d = m.igp_dim
rng = np.random.default_rng(99)                      # every rank builds the same sequence and keeps its block
t = np.arange(T) * DT
F = np.sin(t[:, None] * (1.0 + 3.0 * np.arange(L) / max(L - 1, 1))[None, :])
Y = F @ Hmix.T + 0.1 * (2 * rng.random((T, p)) - 1)
bounds = [time_block_bounds_aligned(T, world, r) for r in range(world)]
t0, t1 = bounds[rank]
n = t1 - t0
f64 = dict(dtype=torch.float64, device=dev)
Yb = torch.from_numpy(np.ascontiguousarray(Y[t0:t1])).to(dev)[None].contiguous()
X, Fs, Ys = torch.zeros((S, 1, n, L, d), **f64), torch.zeros((S, 1, n, L), **f64), torch.zeros((S, 1, n, p), **f64)
sampler = TimeShardedPosteriorSampler(m, [b[1] - b[0] for b in bounds])
Xs = sampler.enqueue(Yb, S, seed, Xsamp=X, Fsamp=Fs, Ysamp=Ys)
torch.cuda.synchronize(dev)
# the whole sequence on this rank's device, with its own handle
w = MOIHGPSequences(DT, p, L, kernel, threading=True, device=local)
w.update(params)
Yd = torch.from_numpy(Y).to(dev)[None].contiguous()
ref = {"Xs": torch.zeros((1, T, L, d), **f64), "X": torch.zeros((S, 1, T, L, d), **f64), "F": torch.zeros((S, 1, T, L), **f64),
       "Y": torch.zeros((S, 1, T, p), **f64)}
w.sample_posterior_device(Yd, seed, Xs=ref["Xs"], X=ref["X"], F=ref["F"], Ysamp=ref["Y"])
torch.cuda.synchronize(dev)
err = {}
for k, a, b in (("Xs", Xs, ref["Xs"][:, t0:t1]), ("X", X, ref["X"][:, :, t0:t1]), ("F", Fs, ref["F"][:, :, t0:t1]), ("Y", Ys, ref["Y"][:, :, t0:t1])):
    err[k] = float((a - b).abs().max()) / float(b.abs().max())
print("rank %d/%d (%s) steps [%d, %d) of T=%d, p=%d L=%d S=%d: rel.err vs the whole sequence %s"
      % (rank, world, backend, t0, t1, T, p, L, S, " ".join("%s %.1e" % kv for kv in err.items())))
assert max(err.values()) < 1e-9, err
print("rank %d: sampled block agrees with the whole-sequence call" % rank)
dist.barrier()
dist.destroy_process_group()
