"""Posterior sample paths of one sequence sharded in time (moihgp_cuda_sample_block_async, parallel.TimeShardedPosteriorSampler).

A block of n steps starting at global step t0 draws the same normals as the whole-sequence call (the Philox counter is the
global step), and its noise at the first step is what it produces from a zero e_end plus G^n e_end, e_end being the next
block's start: the RTS smoother's backward exchange with N -> S N.  So the concatenated blocks must equal
sample_posterior_dev on the whole sequence with the same seed, and every block's X - Xs must equal the noise recomputed in
NumPy from the global steps.

The CPU test runs TimeShardedPosteriorSampler under gloo on a NumPy stand-in model; the GPU tests (-m gpu) run the library."""
import os

import numpy as np
import pytest

from conftest import TOL, rel_err
from test_gpu_sampling import _factors, _model, _outputs, noise, normals


# ---------------------------------------------------------------------------------------------------------------- CPU
class _NumpyBlockModel(object):
    """CPU stand-in for the interface TimeShardedPosteriorSampler uses (fsn_block_async, fsn_carry_device,
    sample_block_async), in NumPy on CPU tensors.  Its mean is local in time (Xs[n,t,l,k] = Y[n,t,l] + k, so the mean's
    carries are zero); its sampler is the block recursion of sample.cu with random stable factors, and its backward carry
    is parallel.backward_carry_in."""

    def __init__(self, p, L, d, seed=5):
        rng = np.random.default_rng(seed)
        self.num_output, self.num_latent, self.igp_dim = p, L, d
        self.G = 0.4 * rng.standard_normal((L, d, d))
        tri = lambda s: np.tril(s * rng.standard_normal((L, d, d))) + np.eye(d)[None]
        self.LF, self.LC = tri(1.0), tri(0.3)

    def mean(self, Y):
        L, d = self.num_latent, self.igp_dim
        return Y[..., :L, None] + np.arange(d)[None, None, None, :]

    def fsn_block_async(self, phase, Y, seq_end, smoother_mode=1, x0=None, u_after=None, b_end=None, X=None, Xs=None, nll=None, xT=None, out=None):
        import torch
        if phase < 3:
            out.zero_()
            return
        Xs.copy_(torch.from_numpy(self.mean(Y.numpy())))
        X.copy_(Xs)
        nll.zero_()

    def fsn_carry_device(self, direction, gathered, block_lengths, rank, out, smoother_mode=1, x0=None, u_after=None):
        import torch
        from multioutputihgp_b200.parallel import backward_carry_in
        if direction == 0:
            out.zero_()
            return
        power = lambda n_: np.stack([np.linalg.matrix_power(g_, n_) for g_ in self.G])
        be = backward_carry_in(power, block_lengths, list(gathered.numpy()), rank)
        if be is not None:
            out.copy_(torch.from_numpy(be))

    def sample_block_async(self, phase, Xs_mean, num_samples, seed, t0, seq_end, e_end=None, Xsamp=None, Fsamp=None, Ysamp=None, out=None):
        import torch
        Xs = Xs_mean.numpy()
        N, n, L, d = Xs.shape
        S = int(num_samples)
        z = normals(seed, np.arange(S)[:, None, None, None], np.arange(N)[None, :, None, None], np.arange(L)[None, None, None, :],
                    t0 + np.arange(n)[None, None, :, None], d)
        e = np.zeros((S, N, n, L, d))
        if seq_end:
            e[:, :, n - 1] = np.einsum("lij,snlj->snli", self.LF, z[:, :, n - 1])
        else:
            e_in = np.zeros((S, N, L, d)) if phase == 1 else e_end.numpy().reshape(S, N, L, d)
            e[:, :, n - 1] = np.einsum("lij,snlj->snli", self.G, e_in) + np.einsum("lij,snlj->snli", self.LC, z[:, :, n - 1])
        for t in range(n - 2, -1, -1):
            e[:, :, t] = np.einsum("lij,snlj->snli", self.G, e[:, :, t + 1]) + np.einsum("lij,snlj->snli", self.LC, z[:, :, t])
        if phase == 1:
            out.copy_(torch.from_numpy(e[:, :, 0].reshape(out.shape)))
            return
        Xsamp.copy_(torch.from_numpy(Xs[None] + e))
        Fsamp.copy_(Xsamp[..., 0])


def _gloo_worker(rank, world, port, T, out_dir):
    import torch
    import torch.distributed as dist
    from multioutputihgp_b200.parallel import TimeShardedPosteriorSampler, time_block_bounds
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    p, L, d, N, S, seed = 4, 3, 2, 2, 3, 0xABCD_0123_4567
    Y = np.random.default_rng(17).standard_normal((N, T, p))
    bounds = [time_block_bounds(T, world, r) for r in range(world)]
    t0, t1 = bounds[rank]
    sampler = TimeShardedPosteriorSampler(_NumpyBlockModel(p, L, d), [b[1] - b[0] for b in bounds], device=torch.device("cpu"))
    X = torch.zeros((S, N, t1 - t0, L, d), dtype=torch.float64)
    F = torch.zeros((S, N, t1 - t0, L), dtype=torch.float64)
    Xs = sampler.enqueue(torch.from_numpy(np.ascontiguousarray(Y[:, t0:t1])), S, seed, Xsamp=X, Fsamp=F)
    np.savez(os.path.join(out_dir, "srank%d.npz" % rank), X=X.numpy(), F=F.numpy(), Xs=Xs.numpy(), t0=t0, t1=t1)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,T", [(2, 57), (3, 40)])
def test_time_sharded_sampler_gloo(tmp_path, world, T):
    """The exchange of TimeShardedPosteriorSampler (RTS mean, phase 1, all-gather, backward carry, phase 2) under gloo: every
    rank's block of the paths equals the whole sequence's mean plus its noise drawn from the global steps."""
    import torch.multiprocessing as mp
    from test_parallel import _free_port
    mp.spawn(_gloo_worker, args=(world, _free_port(), T, str(tmp_path)), nprocs=world, join=True)
    p, L, d, N, S, seed = 4, 3, 2, 2, 3, 0xABCD_0123_4567
    m = _NumpyBlockModel(p, L, d)
    Xs = m.mean(np.random.default_rng(17).standard_normal((N, T, p)))
    X = Xs[None] + noise(seed, S, N, T, m.G, m.LC, m.LF)
    for r in range(world):
        z = np.load(os.path.join(str(tmp_path), "srank%d.npz" % r))
        t0, t1 = int(z["t0"]), int(z["t1"])
        assert np.array_equal(z["Xs"], Xs[:, t0:t1]), r
        assert rel_err(z["X"], X[:, :, t0:t1]) < 1e-12, r
        assert np.array_equal(z["F"], z["X"][..., 0]), r


# ---------------------------------------------------------------------------------------------------------------- GPU
_PATH_IDS = {"scan": 1, "chain": 2, "auto": 0}


def _whole_and_models(kernel, p, L, N, T, G, S, seed, path, rseed):
    """(whole-sequence outputs as torch tensors, one handle per block with the same parameters, the handles' rng).  The
    reference is sample_posterior_device on one handle with the same path."""
    import torch
    from oracle.gen_golden import make_data
    ref, params, rng = _model(kernel, p, L, rseed)
    models = []
    for _ in range(G):
        m, _, _ = _model(kernel, p, L, rseed)
        m.set_path(path)
        models.append(m)
    ref.set_path(path)
    d = ref.igp_dim
    f64 = dict(dtype=torch.float64, device="cuda")
    Y = torch.from_numpy(np.stack([make_data(rng, p, L, T) for _ in range(N)])).cuda()
    w = {"Xs": torch.zeros((N, T, L, d), **f64), "X": torch.zeros((S, N, T, L, d), **f64), "F": torch.zeros((S, N, T, L), **f64),
         "Y": torch.zeros((S, N, T, p), **f64)}
    ref.sample_posterior_device(Y, seed, Xs=w["Xs"], X=w["X"], F=w["F"], Ysamp=w["Y"])
    torch.cuda.synchronize()
    return w, models, ref


def _sharded(models, Xs, cuts, S, seed):
    """Blocks cut from the mean Xs [N,T,L,d] at `cuts`, one handle per block, one block after another: phase 1 of every
    block, the gathered starts stacked, the backward carry kernel and phase 2.  Returns the concatenated X, F, Y (torch)."""
    import torch
    G = len(cuts) - 1
    lengths = [cuts[g + 1] - cuts[g] for g in range(G)]
    N, _, L, d = Xs.shape
    p = models[0].num_output
    f64 = dict(dtype=torch.float64, device=Xs.device)
    blocks = [Xs[:, cuts[g]:cuts[g + 1]].contiguous() for g in range(G)]
    starts = [torch.zeros((S * N, L, d), **f64) for _ in range(G)]
    for g in range(G):
        models[g].sample_block_async(1, blocks[g], S, seed, cuts[g], g == G - 1, out=starts[g])
    gathered = torch.stack(starts)
    out = {"X": [], "F": [], "Y": []}
    for g in range(G):
        n, last = lengths[g], g == G - 1
        e_end = torch.zeros((S * N, L, d), **f64)
        models[g].fsn_carry_device(1, gathered, lengths, g, e_end, smoother_mode=1)
        X, F, Ys = torch.zeros((S, N, n, L, d), **f64), torch.zeros((S, N, n, L), **f64), torch.zeros((S, N, n, p), **f64)
        models[g].sample_block_async(2, blocks[g], S, seed, cuts[g], last, e_end=None if last else e_end, Xsamp=X, Fsamp=F, Ysamp=Ys)
        for k, v in (("X", X), ("F", F), ("Y", Ys)):
            out[k].append(v)
    return {k: torch.cat(v, dim=2) for k, v in out.items()}


BLOCK_CASES = [
    # kernel, p, L, N, S, cuts, path (set_path: scan = time-chunked sampler, chain = one pass, auto = by the number of chains)
    ("Matern32", 8, 4, 1, 1, (0, 512, 1300), "scan"),
    ("Matern32", 8, 4, 1, 1, (0, 512, 1300), "chain"),
    ("Matern52", 6, 3, 3, 2, (0, 256, 768, 1000), "scan"),
    ("Matern52", 6, 3, 3, 2, (0, 256, 768, 1000), "chain"),
    ("Matern52", 12, 5, 2, 3, (0, 1024, 2560, 4001), "auto"),     # few chains: the time-chunked sampler, chunked-scan mean
    ("Matern32", 16, 8, 600, 8, (0, 256, 600), "auto"),           # S N L = 38400 chains: the one-pass sampler, many-chains mean
]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L,N,S,cuts,path", BLOCK_CASES)
def test_blocks_equal_the_whole_sequence_and_the_recomputed_noise(cuda_lib, kernel, p, L, N, S, cuts, path):
    """G = 2 and 3 blocks (uneven cuts, every block but the last a multiple of 256 steps) on one device: the concatenated
    X, F, Y equal sample_posterior_dev on the whole sequence with the same seed; every block's X - Xs equals e recomputed
    in NumPy from the global steps with the library's factors (below 10^6 draws: the NumPy Philox is slow)."""
    T, G, seed = cuts[-1], len(cuts) - 1, 0x5EED_0000_0000 + sum(cuts)
    w, models, ref = _whole_and_models(kernel, p, L, N, T, G, S, seed, path, 3 * T + N)
    got = _sharded(models, w["Xs"], cuts, S, seed)
    import torch
    torch.cuda.synchronize()
    errs = {k: rel_err(got[k].cpu().numpy(), w[k].cpu().numpy()) for k in ("X", "F", "Y")}
    print("sharded sampler %s p=%d L=%d N=%d S=%d cuts=%s path=%s: worst rel. err vs the whole sequence %s"
          % (kernel, p, L, N, S, cuts, path, {k: "%.1e" % v for k, v in errs.items()}))
    assert max(errs.values()) < TOL, errs
    X, Xs = got["X"].cpu().numpy(), w["Xs"].cpu().numpy()
    assert np.array_equal(got["F"].cpu().numpy(), X[..., 0])
    if S * N * T * L <= 10 ** 6:
        e = noise(seed, S, N, T, *_factors(ref))
        for g in range(G):
            sl = slice(cuts[g], cuts[g + 1])
            assert rel_err(X[:, :, sl] - Xs[None, :, sl], e[:, :, sl]) < TOL, g


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["scan", "chain"])
def test_paths_do_not_depend_on_where_the_sequence_is_cut(cuda_lib, path):
    """Two cut sets give the same paths to rounding, and the last step's draw Xs + LF z bit for bit."""
    kernel, p, L, N, S, T = "Matern32", 8, 4, 2, 3, 1500
    seed = 99
    w, models, _ = _whole_and_models(kernel, p, L, N, T, 4, S, seed, path, 41)
    a = _sharded(models[:2], w["Xs"], (0, 512, T), S, seed)
    b = _sharded(models, w["Xs"], (0, 256, 1024, 1280, T), S, seed)
    for k in ("X", "F", "Y"):
        ak, bk = a[k].cpu().numpy(), b[k].cpu().numpy()
        assert rel_err(ak, bk) < 1e-13, k
        assert np.array_equal(ak[:, :, -1], bk[:, :, -1]), k


@pytest.mark.gpu
def test_sample_block_refuses_bad_requests(cuda_lib):
    import torch
    p, L, N, T, S = 4, 2, 1, 10, 2
    m, _, _ = _model("Matern32", p, L, 1)
    d = m.igp_dim
    f64 = dict(dtype=torch.float64, device="cuda")
    Xs, e, F = torch.zeros((N, T, L, d), **f64), torch.zeros((S, N, L, d), **f64), torch.zeros((S, N, T, L), **f64)
    fn = m._lib.moihgp_cuda_sample_block_async
    x, ep, f = Xs.data_ptr(), e.data_ptr(), F.data_ptr()
    big = 2 ** 32
    cases = [((3, x, N, T, 0, 1, S, 5, None, None, f, None, None), "phase must be 1 or 2"),
             ((1, x, N, T, 0, 1, 0, 5, None, None, None, None, ep), "S must be positive"),
             ((2, x, N, T, 0, 1, S, 5, None, None, None, None, None), "no output requested"),
             ((2, x, N, T, 0, 0, S, 5, None, None, f, None, None), "needs e_end"),
             ((1, x, N, T, big - T + 1, 1, S, 5, None, None, None, None, ep), "t0 \\+ T must not exceed 2\\^32"),
             ((1, x, 2 ** 16, T, 0, 1, 2 ** 16, 5, None, None, None, None, ep), "S \\* N must be below 2\\^32"),
             ((1, x, N, T, 0, 1, S, 5, None, None, None, None, None), "phase 1 needs dev_out"),
             ((2, None, N, T, 0, 1, S, 5, None, None, f, None, None), "phase 2 needs Xs_mean")]
    import re
    for args, msg in cases:
        assert fn(m._h, *args) == -2, msg
        assert re.search(msg, m._lib.moihgp_cuda_last_error(m._h).decode()), msg
    # the last step of the counter's range is accepted
    assert fn(m._h, 1, x, N, T, big - T, 1, S, 5, None, None, None, None, ep) == 0
    with pytest.raises(ValueError, match="out must be %d elements" % (S * N * L * d)):
        m.sample_block_async(1, Xs, S, 5, 0, True, out=torch.zeros((N, L, d), **f64))
    with pytest.raises(ValueError, match="Xs_mean must be a \\[N,T,L,d\\] tensor"):
        m.sample_block_async(1, Xs[0], S, 5, 0, True, out=e)
    with pytest.raises(ValueError, match="e_end must be torch.float64"):
        m.sample_block_async(2, Xs, S, 5, 0, False, e_end=e.float(), Fsamp=F)
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["scan", "chain"])
def test_block_exchange_right_after_update_is_capturable_in_a_cuda_graph(cuda_lib, path):
    """Phase 1 of every block -> the stacked starts -> the carry kernel -> phase 2, captured into a CUDA graph right after
    update(params); replays on new means equal the same calls run directly, and X - Xs is the whole sequence's noise."""
    import torch
    from oracle.gen_golden import make_params
    kernel, p, L, N, S, cuts = "Matern52", 12, 5, 2, 2, (0, 768, 1900)
    T, G, seed = cuts[-1], 2, 1234
    rng = np.random.default_rng(8)
    models = []
    for _ in range(G):
        m, _, _ = _model(kernel, p, L, 8)
        m.set_path(path)
        models.append(m)
    d = models[0].igp_dim
    Xs = torch.zeros((N, T, L, d), dtype=torch.float64, device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        _sharded(models, Xs, cuts, S, seed)                              # warm-up on the capture stream: workspaces
        torch.cuda.synchronize()
        params = make_params(rng, p, L, kernel)
        for m in models:
            m.update(params)                                             # K-setup queued, nothing waits
        with torch.cuda.graph(g, stream=side):
            got = _sharded(models, Xs, cuts, S, seed)
    for rep in range(2):
        Xs.copy_(torch.from_numpy(rng.standard_normal((N, T, L, d))))
        g.replay()
        torch.cuda.synchronize()
        direct = _sharded(models, Xs, cuts, S, seed)
        torch.cuda.synchronize()
        for k in ("X", "F", "Y"):
            assert torch.equal(got[k], direct[k]), (rep, k)
        e = noise(seed, S, N, T, *_factors(models[0]))
        assert rel_err(got["X"].cpu().numpy() - Xs.cpu().numpy()[None], e) < TOL, rep
        assert rel_err(got["Y"].cpu().numpy(), _outputs(models[0], got["F"].cpu().numpy())) < 1e-12, rep


def _torchrun(nproc, port, env):
    import subprocess
    import sys
    from conftest import ROOT
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(ROOT, "scripts", "gpu_time_shard_sample.py")], capture_output=True, text=True,
                       env=dict(os.environ, **env), timeout=600)
    print(r.stdout[-2000:], r.stderr[-2000:])
    return r


@pytest.mark.gpu
def test_time_sharded_sampler_two_ranks_on_one_gpu(cuda_lib):
    """TimeShardedPosteriorSampler end to end with TWO ranks on whatever GPUs are visible (gloo exchange on CUDA tensors):
    every rank's block of the paths equals the whole-sequence call."""
    r = _torchrun(2, 29551, {"TS_BACKEND": "gloo", "TS_T": "70001", "TS_P": "16", "TS_L": "8"})
    assert r.returncode == 0 and r.stdout.count("sampled block agrees") == 2


@pytest.mark.gpu
def test_time_sharded_sampler_two_gpus(cuda_lib):
    """The same over NCCL on two GPUs.  Needs two devices."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = _torchrun(2, 29553, {"TS_T": "70001", "TS_P": "16", "TS_L": "8"})
    assert r.returncode == 0 and r.stdout.count("sampled block agrees") == 2
