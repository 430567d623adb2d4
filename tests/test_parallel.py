"""Host-side multi-GPU logic on CPU: two ranks under gloo, the oracle standing in for the CUDA evaluator.

(The oracle is only the stand-in evaluator and the checker here - test infrastructure, as allowed.)"""
import os
import socket

import numpy as np
import pytest

from conftest import rel_err
from multioutputihgp_b200.parallel import shard_bounds


def test_shard_bounds_cover_everything_once():
    for N in (0, 1, 2, 5, 8, 4096, 4097):
        for world in (1, 2, 3, 4, 8):
            cover = []
            for r in range(world):
                lo, hi = shard_bounds(N, world, r)
                assert 0 <= lo <= hi <= N
                cover += list(range(lo, hi))
            assert cover == list(range(N)), (N, world)
            sizes = [shard_bounds(N, world, r)[1] - shard_bounds(N, world, r)[0] for r in range(world)]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_bounds(4, 2, 2)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, N, out_dir):
    import torch.distributed as dist
    from multioutputihgp_b200.parallel import ShardedObjective, sharded_nll
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(77)
    p, L, T = 6, 3, 40
    params = make_params(rng, p, L, "Matern32")
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)]) if N else np.zeros((0, T, p))
    o = OracleMOIHGP(0.1, p, L, "Matern32", threading=True)
    o.update(params)
    lo, hi = shard_bounds(N, world, rank)
    obj = ShardedObjective(lambda Yl: o.objective(Yl)[:2], o.num_param)
    loss, grad = obj(Y[lo:hi])
    nll_local = o.filter_smoother_nll(Y[lo:hi], smoother_mode=-1, want_states=False)["nll"] if hi > lo else np.zeros(0)
    total = sharded_nll(nll_local)
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), loss=loss, grad=grad, total=total, lo=lo, hi=hi)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("N", [5, 1])
def test_sharded_objective_two_ranks_gloo(tmp_path, N):
    import torch.multiprocessing as mp
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), N, str(tmp_path)), nprocs=world, join=True)
    rng = np.random.default_rng(77)
    p, L, T = 6, 3, 40
    params = make_params(rng, p, L, "Matern32")
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    o = OracleMOIHGP(0.1, p, L, "Matern32", threading=True)
    o.update(params)
    loss, grad = o.objective(Y)[:2]
    nll = o.filter_smoother_nll(Y, smoother_mode=-1, want_states=False)["nll"].sum()
    outs = [np.load(os.path.join(str(tmp_path), "rank%d.npz" % r)) for r in range(world)]
    for z in outs:                                   # every rank holds the identical reduced result
        assert abs(float(z["loss"]) - loss) <= 1e-12 * abs(loss)
        assert rel_err(z["grad"], grad) < 1e-12
        assert abs(float(z["total"]) - nll) <= 1e-12 * abs(nll)
    assert float(outs[0]["loss"]) == float(outs[1]["loss"]) and np.array_equal(outs[0]["grad"], outs[1]["grad"])
    assert int(outs[0]["lo"]) == 0 and int(outs[1]["hi"]) == N


def test_block_transition_matches_the_step_by_step_recursion():
    from multioutputihgp_b200.parallel import block_transition
    rng = np.random.default_rng(3)
    for d in (2, 3):
        M = 0.6 * rng.standard_normal((d, d)) / np.sqrt(d)
        dM = [rng.standard_normal((d, d)) for _ in range(3)]
        for n in (0, 1, 2, 7, 64, 1000):
            P, E = block_transition(M, dM, n)
            Pr, Er = np.eye(d), [np.zeros((d, d)) for _ in range(3)]
            for _ in range(n):
                Er = [M @ e + dm @ Pr for e, dm in zip(Er, dM)]
                Pr = M @ Pr
            assert np.allclose(P, Pr, rtol=1e-12, atol=1e-300)
            for a, b in zip(E, Er):
                assert np.allclose(a, b, rtol=1e-11, atol=1e-300)


def _time_worker(rank, world, port, T, out_dir):
    import torch.distributed as dist
    from multioutputihgp_b200.parallel import TimeShardedObjective, time_block_bounds
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(78)
    p, L = 6, 3
    params = make_params(rng, p, L, "Matern52")
    Y = make_data(rng, p, L, T)
    o = OracleMOIHGP(0.1, p, L, "Matern52", threading=True)
    o.update(params)
    consts = [o.ihgp_consts(l) for l in range(L)]
    bounds = [time_block_bounds(T, world, r) for r in range(world)]

    def evaluate(Yb, x0, dx0):
        loss, grad, xT, dxT = o.objective(Yb[None], x0=x0[None], dx0=dx0[None])
        return loss, grad, xT[0], dxT[0]
    obj = TimeShardedObjective(evaluate, consts, [b[1] - b[0] for b in bounds], o.num_param)
    t0, t1 = bounds[rank]
    loss, grad = obj(Y[t0:t1])
    # an optimiser loop changes the parameters between evaluations: with a provider / a callable the block transitions follow
    params2 = params.copy()
    params2[p * L + L + 1:] *= 1.3
    params2[p * L:p * L + L] *= 0.8
    prov = TimeShardedObjective(evaluate, lambda: [o.ihgp_consts(l) for l in range(L)], [b[1] - b[0] for b in bounds], o.num_param)

    def transition(n):
        from multioutputihgp_b200.parallel import block_transition, stack_consts
        AK, dAK = stack_consts([o.ihgp_consts(l) for l in range(L)])
        return block_transition(AK, dAK, n)
    call = TimeShardedObjective(evaluate, transition, [b[1] - b[0] for b in bounds], o.num_param)
    prov(Y[t0:t1])
    call(Y[t0:t1])
    o.update(params2)
    loss2, grad2 = prov(Y[t0:t1])
    loss3, grad3 = call(Y[t0:t1])
    np.savez(os.path.join(out_dir, "trank%d.npz" % rank), loss=loss, grad=grad, loss2=loss2, grad2=grad2, loss3=loss3, grad3=grad3)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,T", [(2, 301), (3, 100)])
def test_time_sharded_objective_gloo(tmp_path, world, T):
    """One sequence split in time over the ranks (SURVEY 8(e)): carries exchanged by all-gather, [loss, grad] all-reduced;
    equals the single-process evaluation of the whole sequence."""
    import torch.multiprocessing as mp
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    mp.spawn(_time_worker, args=(world, _free_port(), T, str(tmp_path)), nprocs=world, join=True)
    rng = np.random.default_rng(78)
    p, L = 6, 3
    params = make_params(rng, p, L, "Matern52")
    Y = make_data(rng, p, L, T)
    o = OracleMOIHGP(0.1, p, L, "Matern52", threading=True)
    o.update(params)
    loss, grad = o.objective(Y[None])[:2]
    params2 = params.copy()
    params2[p * L + L + 1:] *= 1.3
    params2[p * L:p * L + L] *= 0.8
    o.update(params2)
    loss2, grad2 = o.objective(Y[None])[:2]
    for r in range(world):
        z = np.load(os.path.join(str(tmp_path), "trank%d.npz" % r))
        assert abs(float(z["loss"]) - loss) <= 1e-11 * abs(loss)
        assert rel_err(z["grad"], grad) < 1e-10
        # after update(params2): the provider / callable forms re-derive the block transitions on every call
        for k in ("2", "3"):
            assert abs(float(z["loss" + k]) - loss2) <= 1e-11 * abs(loss2), k
            assert rel_err(z["grad" + k], grad2) < 1e-10, k


class _OracleBlockModel(object):
    """CPU stand-in for MOIHGPSequences' time-sharding interface (fsn_block_async / fsn_carry_device), built on the oracle:
    lets the exchange protocol of TimeShardedFilterSmoother run under gloo without a GPU."""

    def __init__(self, o, params, p, L):
        self.o, self.num_latent, self.igp_dim = o, L, o.ihgp_consts(0)["AKHA"].shape[0]
        c = [o.ihgp_consts(l) for l in range(L)]
        self.M = np.stack([c_["AKHA"] for c_ in c])
        self.K = np.stack([np.asarray(c_["K"]).ravel() for c_ in c])
        self.HA = np.stack([np.asarray(c_["HA"]).ravel() for c_ in c])
        self.G = np.stack([o.smoother_consts(l, 1)[0] for l in range(L)])
        self.U, self.S = o.U, params[p * L:p * L + L]

    def block_transition(self, n):
        return np.stack([np.linalg.matrix_power(m_, n) for m_ in self.M]), None

    def smoother_power(self, n, mode):
        return np.stack([np.linalg.matrix_power(g_, n) for g_ in self.G])

    def fsn_block(self, phase, Y, seq_end, smoother_mode=1, x0=None, u_after=None, b_end=None, X=None, Xs=None, nll=None, xT=None):
        import torch
        Ynp = Y.numpy()
        N, n, _ = Ynp.shape
        L, d = self.num_latent, self.igp_dim
        u = (Ynp @ self.U) / np.sqrt(self.S)
        x_in = np.zeros((N, L, d)) if x0 is None else x0.numpy()
        r = self.o.filter_smoother_nll(Ynp, x0=x_in, smoother_mode=1)
        if phase == 1:
            return r["xT"].copy(), u[:, 0, :].copy()
        Xf = r["X"]
        b = np.zeros((N, L, d)) if b_end is None else b_end.numpy().copy()
        bs = np.zeros((N, n, L, d))
        for j in range(n - 1, -1, -1):
            if j + 1 < n:
                v = u[:, j + 1] - np.einsum("lq,nlq->nl", self.HA, Xf[:, j])
            elif seq_end:
                v = np.zeros((N, L))
            else:
                v = u_after.numpy() - np.einsum("lq,nlq->nl", self.HA, Xf[:, j])
            gk = np.einsum("lij,lj->li", self.G, self.K)
            b = np.einsum("lij,nlj->nli", self.G, b) + gk[None] * v[:, :, None]
            bs[:, j] = b
        if phase == 2:
            return bs[:, 0].copy()
        X.copy_(torch.from_numpy(Xf))
        Xs.copy_(torch.from_numpy(Xf + bs))
        nll.copy_(torch.from_numpy(r["nll"]))
        if xT is not None:
            xT.copy_(torch.from_numpy(r["xT"]))

    def fsn_block_async(self, phase, Y, seq_end, smoother_mode=1, x0=None, u_after=None, b_end=None, X=None, Xs=None, nll=None, xT=None, out=None):
        import torch
        r = self.fsn_block(phase, Y, seq_end, smoother_mode, x0=x0, u_after=u_after, b_end=b_end, X=X, Xs=Xs, nll=nll, xT=xT)
        if phase == 1:
            out.copy_(torch.from_numpy(np.concatenate([r[0], r[1][..., None]], axis=-1)))
        elif phase == 2:
            out.copy_(torch.from_numpy(r))

    def fsn_carry_device(self, direction, gathered, block_lengths, rank, out, smoother_mode=1, x0=None, u_after=None):
        import torch
        from multioutputihgp_b200.parallel import backward_carry_in, forward_carry_in
        g = gathered.numpy()
        d = self.igp_dim
        if direction == 0:
            x0n = np.zeros(g.shape[1:3] + (d,)) if x0 is None else x0.numpy()
            out.copy_(torch.from_numpy(forward_carry_in(self.block_transition, block_lengths, list(g[..., :d]), x0n, rank)))
            if u_after is not None and rank + 1 < len(block_lengths):
                u_after.copy_(torch.from_numpy(g[rank + 1][..., d].copy()))
        else:
            be = backward_carry_in(lambda n_: self.smoother_power(n_, smoother_mode), block_lengths, list(g), rank)
            if be is not None:
                out.copy_(torch.from_numpy(be))


def _fsn_worker(rank, world, port, T, out_dir):
    import torch
    import torch.distributed as dist
    from multioutputihgp_b200.parallel import TimeShardedFilterSmoother, time_block_bounds
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(91)
    p, L, N = 6, 3, 2
    params = make_params(rng, p, L, "Matern32")
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    x0 = 0.2 * rng.standard_normal((N, L, 2))
    o = OracleMOIHGP(0.1, p, L, "Matern32", threading=True)
    o.update(params)
    bounds = [time_block_bounds(T, world, r) for r in range(world)]
    t0, t1 = bounds[rank]
    fs = TimeShardedFilterSmoother(_OracleBlockModel(o, params, p, L), [b[1] - b[0] for b in bounds], 1, device=torch.device("cpu"))
    X = torch.zeros((N, t1 - t0, L, 2), dtype=torch.float64)
    Xs = torch.zeros_like(X)
    Yb = torch.from_numpy(np.ascontiguousarray(Y[:, t0:t1]))
    nll = fs(Yb, X, Xs, x0=x0)
    # the same exchange through enqueue, with x0 as a tensor
    X2, Xs2 = torch.zeros_like(X), torch.zeros_like(Xs)
    nll2 = fs.enqueue(Yb, X2, Xs2, x0=torch.from_numpy(x0)).numpy().copy()
    np.savez(os.path.join(out_dir, "frank%d.npz" % rank), X=X.numpy(), Xs=Xs.numpy(), nll=nll, t0=t0, t1=t1, X2=X2.numpy(), Xs2=Xs2.numpy(), nll2=nll2)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,T", [(2, 151), (3, 90)])
def test_time_sharded_filter_smoother_gloo(tmp_path, world, T):
    """One sequence split in time over the ranks (SURVEY 8(e)): forward carry exchange, mirror-image backward exchange,
    NLL all-reduce; every rank's block of X / Xs and the NLL equal the single-process pass over the whole sequence."""
    import torch.multiprocessing as mp
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    mp.spawn(_fsn_worker, args=(world, _free_port(), T, str(tmp_path)), nprocs=world, join=True)
    rng = np.random.default_rng(91)
    p, L, N = 6, 3, 2
    params = make_params(rng, p, L, "Matern32")
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    x0 = 0.2 * rng.standard_normal((N, L, 2))
    o = OracleMOIHGP(0.1, p, L, "Matern32", threading=True)
    o.update(params)
    ref = o.filter_smoother_nll(Y, x0=x0, smoother_mode=1)
    for r in range(world):
        z = np.load(os.path.join(str(tmp_path), "frank%d.npz" % r))
        t0, t1 = int(z["t0"]), int(z["t1"])
        assert rel_err(z["X"], ref["X"][:, t0:t1]) < 1e-12
        assert rel_err(z["Xs"], ref["Xs"][:, t0:t1]) < 1e-11
        assert rel_err(z["nll"], ref["nll"]) < 1e-11
        # __call__ is enqueue and a synchronise: the same numbers
        assert np.array_equal(z["X2"], z["X"]) and np.array_equal(z["Xs2"], z["Xs"]) and np.array_equal(z["nll2"], z["nll"])


def test_carry_algebra_of_the_time_sharded_smoother():
    """forward_carry_in / backward_carry_in against the plain sequential recursions on random stable systems."""
    from multioutputihgp_b200.parallel import backward_carry_in, forward_carry_in
    rng = np.random.default_rng(12)
    L, d, N = 3, 2, 2
    M = 0.5 * rng.standard_normal((L, d, d)) * 0.6
    Gm = 0.5 * rng.standard_normal((L, d, d)) * 0.6
    lengths = [5, 7, 4]
    T = sum(lengths)
    drive_f = rng.standard_normal((T, N, L, d))
    drive_b = rng.standard_normal((T, N, L, d))
    x0 = rng.standard_normal((N, L, d))
    x, xs = x0.copy(), []
    for t in range(T):
        xs.append(x.copy())                              # state BEFORE step t
        x = np.einsum("lij,nlj->nli", M, x) + drive_f[t]
    b, bs = np.zeros((N, L, d)), [None] * (T + 1)
    bs[T] = b.copy()
    for t in range(T - 1, -1, -1):
        b = np.einsum("lij,nlj->nli", Gm, b) + drive_b[t]
        bs[t] = b.copy()
    cuts = np.concatenate([[0], np.cumsum(lengths)])
    ends, starts = [], []
    for g in range(3):
        z = np.zeros((N, L, d))
        for t in range(cuts[g], cuts[g + 1]):
            z = np.einsum("lij,nlj->nli", M, z) + drive_f[t]
        ends.append(z)
        z = np.zeros((N, L, d))
        for t in range(cuts[g + 1] - 1, cuts[g] - 1, -1):
            z = np.einsum("lij,nlj->nli", Gm, z) + drive_b[t]
        starts.append(z)
    tr = lambda n: (np.stack([np.linalg.matrix_power(m_, n) for m_ in M]), None)
    sp = lambda n: np.stack([np.linalg.matrix_power(g_, n) for g_ in Gm])
    for g in range(3):
        assert rel_err(forward_carry_in(tr, lengths, ends, x0, g), xs[cuts[g]]) < 1e-13
        be = backward_carry_in(sp, lengths, starts, g)
        if g == 2:
            assert be is None
        else:
            assert rel_err(be, bs[cuts[g + 1]]) < 1e-13
