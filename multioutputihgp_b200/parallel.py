"""Multi-GPU use of the hot path: one process per GPU, independent sequences sharded over ranks.

The reference has a single sequence and no communication layer (SURVEY.md 2.2); its objective is a plain sum
over observations (moihgp_regression.h:46-47), so N independent sequences shard over ranks with NO data-path
collective.  The only exchange is one fp64 all-reduce per evaluation of the fused buffer ``[loss, grad]``
(``1 + num_param`` doubles; objective) or of the summed NLL (filter pass) - SURVEY.md 8(e).  Every rank ends up
with the identical reduced result, which is what a replicated L-BFGS loop needs.

``torch.distributed`` is plumbing only: NCCL over NVLink on the GPU box, gloo in the CPU tests
(tests/test_parallel.py, world_size 2, with a stand-in evaluator).
"""
import numpy as np


def shard_bounds(num_sequences, world_size, rank):
    """Contiguous, balanced shard [lo, hi) of ``num_sequences`` for ``rank``: the first ``N % world`` ranks get one more.
    A rank may receive an empty shard (N < world)."""
    if world_size < 1 or not (0 <= rank < world_size):
        raise ValueError("bad rank %r / world_size %r" % (rank, world_size))
    base, extra = divmod(int(num_sequences), world_size)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def _dist():
    import torch.distributed as dist
    return dist


def _ranks(group):
    """(multi, world, rank) of this process in ``group``: (False, 1, 0) without a process group of more than one rank."""
    dist = _dist()
    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1):
        return False, 1, 0
    return True, dist.get_world_size(group), dist.get_rank(group)


def _all_gather_into(out, inp, group):
    """out[G, ...] <- every rank's inp, on the current stream (NCCL); gloo (ranks sharing a GPU, CPU tests) takes the list form"""
    dist = _dist()
    if dist.get_backend(group) == "gloo":
        dist.all_gather(list(out.unbind(0)), inp, group=group)
    else:
        dist.all_gather_into_tensor(out, inp, group=group)


class ShardedObjective(object):
    """loss, grad = sum over ALL ranks' sequences of the objective; call with this rank's shard.

    ``evaluate(Y_local) -> (loss, grad)`` is the local evaluator: ``MOIHGPSequences.objective`` on a GPU box.
    An empty local shard contributes zeros.  The reduction is one all-reduce of a single fp64 buffer."""

    def __init__(self, evaluate, num_param, group=None, device=None):
        self.evaluate = evaluate
        self.num_param = int(num_param)
        self.group = group
        self.device = device

    def __call__(self, Y_local):
        import torch
        buf = np.zeros(1 + self.num_param)
        if Y_local is not None and len(Y_local) > 0:
            loss, grad = self.evaluate(Y_local)
            buf[0] = loss
            buf[1:] = grad
        dist = _dist()
        if _ranks(self.group)[0]:
            t = torch.from_numpy(buf)
            if self.device is not None:
                t = t.to(self.device)
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
            buf = t.cpu().numpy()
        return float(buf[0]), buf[1:].copy()


class ShardedDeviceObjective(object):
    """Device-resident variant for the GPU box: the model writes ``[loss, pad, grad]`` into one torch CUDA buffer and
    NCCL all-reduces it in place on the same stream (no host round trip before the reduction)."""

    def __init__(self, model, group=None):
        import torch
        self.model = model
        self.group = group
        self.buf = torch.zeros(2 + model.num_param, dtype=torch.float64, device=torch.device("cuda", torch.cuda.current_device()))

    def __call__(self, Y_local_device):
        dist = _dist()
        self.buf.zero_()
        if Y_local_device is not None and Y_local_device.shape[0] > 0:
            self.model.objective_device(Y_local_device, self.buf[0:1], self.buf[2:])
        if _ranks(self.group)[0]:
            dist.all_reduce(self.buf, op=dist.ReduceOp.SUM, group=self.group)
        host = self.buf.cpu().numpy()
        return float(host[0]), host[2:].copy()


def sharded_nll(local_nll, group=None, device=None):
    """Total NLL over all ranks' sequences from this rank's per-sequence values (filter + smoother + NLL pass)."""
    import torch
    t = torch.tensor([float(np.sum(local_nll)) if local_nll is not None and len(local_nll) else 0.0], dtype=torch.float64)
    if device is not None:
        t = t.to(device)
    dist = _dist()
    if _ranks(group)[0]:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return float(t.item())


# ------------------------------------------------------------------------------------------------------------------
# One LONG sequence sharded over ranks in TIME (SURVEY.md 8(e), BASELINE configs 4 and 5).
#
# The recursion is LTI-affine (ihgp.h:50,54): over a block of n steps the augmented state z = [x; dx_0; dx_1; dx_2] of a
# latent maps as  z_out = T(n) z_in + z_out(z_in = 0),  with  T(n): x -> M^n x,  dx_k -> M^n dx_k + E_k(n) x,
# M = AKHA, E_k(n) = sum_i M^(n-1-i) dAKHA_k M^i.  So every rank (1) runs its block from a ZERO carry-in, (2) all-gathers
# the L*d*(1+K) end-state doubles, (3) forms its true carry-in from the blocks before it, (4) runs its block again from
# the true carry-in - the loss / gradient are quadratic in the state, so they need the true states - and (5) all-reduces
# [loss, grad].  Two passes per rank, no other exchange: a G-rank job runs G/2 times faster than one GPU.

def block_transition(AKHA, dAKHA, n):
    """(M^n, E_k(n)) by binary powering: doubling (P, E) -> (P P, P E + E P), increment (P, E) -> (M P, M E + dM P).
    Batched over leading axes: AKHA [..., d, d], dAKHA [..., K, d, d] (or a list of K [d, d] matrices for one latent)."""
    AKHA = np.asarray(AKHA, dtype=np.float64)
    as_list = isinstance(dAKHA, (list, tuple))
    dM = np.stack([np.asarray(m_, dtype=np.float64) for m_ in dAKHA], axis=-3) if as_list else np.asarray(dAKHA, dtype=np.float64)
    d = AKHA.shape[-1]
    M = AKHA[..., None, :, :]                                   # broadcast over K
    P = np.broadcast_to(np.eye(d), AKHA.shape).copy()
    E = np.zeros(dM.shape)
    for bit in bin(int(n))[2:]:
        Pk = P[..., None, :, :]
        E = Pk @ E + E @ Pk
        P = P @ P
        if bit == "1":
            E = M @ E + dM @ P[..., None, :, :]
            P = AKHA @ P
    return (P, [E[..., k, :, :] for k in range(E.shape[-3])]) if as_list else (P, E)


def stack_consts(consts):
    """Per-latent constant dicts (latent_consts / ihgp_consts) -> (AKHA [L,d,d], dAKHA [L,3,d,d])."""
    return (np.stack([c["AKHA"] for c in consts]), np.stack([np.stack([c["dAKHA%d" % k] for k in range(3)]) for c in consts]))


def carry_in_from_block_ends(consts, block_lengths, ends_x, ends_dx, x0, dx0, rank):
    """True carry-in (x [L,d], dx [L,3,d]) of block `rank`, given every block's end state from a zero carry-in.
    consts: list of per-latent dicts, the stacked pair of stack_consts(), or a callable n -> (P [L,d,d], E [L,3,d,d]);
    ends_x [G,L,d], ends_dx [G,L,3,d]."""
    if callable(consts):                                         # n -> (P, E), e.g. MOIHGPSequences.block_transition
        transition = consts
    else:
        AK, dAK = consts if isinstance(consts, tuple) else stack_consts(consts)
        transition = lambda n_: block_transition(AK, dAK, n_)
    x = np.array(x0, dtype=np.float64).copy()
    dx = np.array(dx0, dtype=np.float64).copy()
    cache = {}
    for g in range(rank):
        n = int(block_lengths[g])
        if n not in cache:
            cache[n] = transition(n)
        P, E = cache[n]                                          # [L,d,d], [L,3,d,d]
        xo = x
        x = np.einsum("lij,lj->li", P, xo) + ends_x[g]
        dx = np.einsum("lij,lkj->lki", P, dx) + np.einsum("lkij,lj->lki", E, xo) + ends_dx[g]
    return x, dx


class TimeShardedObjective(object):
    """loss, grad of ONE long sequence whose contiguous time blocks live on different ranks.

    ``evaluate(Y_block, x0, dx0) -> (loss, grad, xT, dxT)`` is the local evaluator (``MOIHGPSequences.objective`` with
    ``want_state=True`` on a GPU box); ``block_lengths[g]`` the number of time steps of rank g's block.

    ``consts`` gives the block transitions of the model's CURRENT hyper-parameters.  Inside an optimiser loop the
    parameters change between calls (``model.update(params)`` then ``obj(Y_block)``), so pass something that is evaluated
    on every call: a callable ``n -> (P [L,d,d], E [L,3,d,d])`` such as ``model.block_transition``, or a zero-argument
    provider returning the per-latent constant dicts (``lambda: [model.latent_consts(l) for l in range(L)]``).  A plain
    list of dicts / a stacked (AKHA, dAKHA) pair is taken as fixed - only right while the parameters do not change."""

    def __init__(self, evaluate, consts, block_lengths, num_param, group=None, device=None, num_latent=None, igp_dim=None):
        self.evaluate, self.block_lengths = evaluate, [int(b) for b in block_lengths]
        self.consts = consts
        self.num_param, self.group, self.device = int(num_param), group, device
        self.num_latent, self.igp_dim = num_latent, igp_dim

    def _current(self):
        """(transition or stacked constants of the current parameters, L, d)"""
        c = self.consts
        if callable(c):
            try:
                c = c()                                  # zero-argument provider of the per-latent constants
            except TypeError:
                if self.num_latent is not None and self.igp_dim is not None:
                    return c, self.num_latent, self.igp_dim
                P, _ = c(1)                              # n -> (P, E): shapes from one call
                return c, P.shape[0], P.shape[-1]
        st = c if isinstance(c, tuple) else stack_consts(c)
        return st, st[0].shape[0], st[0].shape[-1]

    def _gather(self, vec, world):
        import torch
        dist = _dist()
        t = torch.from_numpy(np.ascontiguousarray(vec))
        if self.device is not None:
            t = t.to(self.device)
        out = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(out, t, group=self.group)
        return [o.cpu().numpy() for o in out]

    def __call__(self, Y_block, x0=None, dx0=None):
        import torch
        dist = _dist()
        multi, world, rank = _ranks(self.group)
        consts, L, d = self._current()
        x0 = np.zeros((L, d)) if x0 is None else np.asarray(x0, dtype=np.float64).reshape(L, d)
        dx0 = np.zeros((L, 3, d)) if dx0 is None else np.asarray(dx0, dtype=np.float64).reshape(L, 3, d)
        if not multi:
            loss, grad, xT, dxT = self.evaluate(Y_block, x0, dx0)
            return loss, grad
        # (1) block from a zero carry-in -> its end state; (2) all-gather
        _, _, xT, dxT = self.evaluate(Y_block, np.zeros((L, d)), np.zeros((L, 3, d)))
        flat = np.concatenate([np.asarray(xT).ravel(), np.asarray(dxT).ravel()])
        ends = self._gather(flat, world)
        ends_x = [e[:L * d].reshape(L, d) for e in ends]
        ends_dx = [e[L * d:].reshape(L, 3, d) for e in ends]
        # (3) true carry-in, (4) the block again, (5) all-reduce
        xin, dxin = carry_in_from_block_ends(consts, self.block_lengths, ends_x, ends_dx, x0, dx0, rank)
        loss, grad, _, _ = self.evaluate(Y_block, xin, dxin)
        buf = torch.from_numpy(np.concatenate([[loss], np.asarray(grad, dtype=np.float64)]))
        if self.device is not None:
            buf = buf.to(self.device)
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=self.group)
        buf = buf.cpu().numpy()
        return float(buf[0]), buf[1:].copy()


def time_block_bounds(T, world_size, rank):
    """Contiguous time block [t0, t1) of rank `rank` (same balancing rule as shard_bounds)."""
    return shard_bounds(T, world_size, rank)


def time_block_bounds_aligned(T, world_size, rank, align=256):
    """Like time_block_bounds, but every block except the last is a whole number of `align`-step chunks (the scan's chunk
    length): what the one-pass time-sharded evaluation needs."""
    chunks = int(T) // align
    lo_c, hi_c = shard_bounds(chunks, world_size, rank)
    lo, hi = lo_c * align, hi_c * align
    if rank == world_size - 1:
        hi = int(T)
    return lo, hi


class TimeShardedDeviceObjective(object):
    """One-pass variant on the GPU library, with NO host round trip inside an evaluation: ``objective_begin_async``
    projects the block and leaves its end state from a zero carry-in in device memory, NCCL all-gathers the end states on the
    same stream, ``carry_in_device`` (a tiny kernel: the block transitions T(n_g) by binary powering on the device's power
    tables) forms this rank's true carry-in, ``objective_finish_device`` evaluates from it reusing the projection, and
    [loss, grad] is all-reduced in place.  Everything is queued on torch's current stream; ``__call__`` syncs once, at the
    end, to hand [loss, grad] to the optimiser; ``enqueue`` does not sync at all."""

    def __init__(self, model, block_lengths, group=None, num_sequences=1):
        import torch
        self.model, self.group = model, group
        self.block_lengths = [int(b) for b in block_lengths]
        self.dev = torch.device("cuda", torch.cuda.current_device())
        L, d, N, G = model.num_latent, model.igp_dim, int(num_sequences), len(self.block_lengths)
        f64 = dict(dtype=torch.float64, device=self.dev)
        self.buf = torch.zeros(2 + model.num_param, **f64)
        self.ends = torch.zeros((G, N, L, 4, d), **f64)              # all-gathered block ends
        self.zend = torch.zeros((N, L, 4, d), **f64)                 # this block's end state from a zero carry-in
        self.xin = torch.zeros((N, L, d), **f64)
        self.dxin = torch.zeros((N, L, 3, d), **f64)

    def enqueue(self, Y_block_dev, x0=None, dx0=None):
        """Queue one evaluation on the current stream; the result lands in ``self.buf`` = [loss, pad, grad...].
        x0 / dx0: carried-in state of the WHOLE sequence (torch CUDA tensors or None = zeros)."""
        dist = _dist()
        m = self.model
        multi, world, rank = _ranks(self.group)
        last = rank == world - 1
        m.objective_begin_async(Y_block_dev, None if last else self.zend)
        if multi:
            _all_gather_into(self.ends, self.zend, self.group)
        m.carry_in_device(self.ends, self.block_lengths, rank, self.xin, self.dxin, x0=x0, dx0=dx0)
        m.objective_finish_device(Y_block_dev, self.buf[0:1], self.buf[2:], x0=self.xin, dx0=self.dxin)
        if multi:
            dist.all_reduce(self.buf, op=dist.ReduceOp.SUM, group=self.group)

    def __call__(self, Y_block_dev, x0=None, dx0=None):
        import torch
        to_dev = lambda a, shape: None if a is None else torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(shape))).to(self.dev)
        N, L, d = self.xin.shape
        self.enqueue(Y_block_dev, to_dev(x0, (N, L, d)), to_dev(dx0, (N, L, 3, d)))
        host = self.buf.cpu().numpy()
        return float(host[0]), host[2:].copy()


def forward_carry_in(transition, block_lengths, ends_x, x0, rank):
    """Filter state entering block `rank`: x_in(g+1) = AKHA^n_g x_in(g) + x_end_g, x_in(0) = x0.  ends_x [G,N,L,d] are the
    blocks' end states from a ZERO carry-in, transition(n) -> (AKHA^n [L,d,d], ...), x0 [N,L,d]."""
    x = np.array(x0, dtype=np.float64).copy()
    for g in range(rank):
        P = transition(int(block_lengths[g]))[0]
        x = np.einsum("lij,nlj->nli", P, x) + ends_x[g]
    return x


def backward_carry_in(smoother_power, block_lengths, starts_b, rank):
    """Backward value entering block `rank` from the right (None on the last block): b_end(g) = b_start(g+1),
    b_start(g) = starts_b[g] + G^n_g b_end(g); starts_b [G,N,L,d] are the blocks' first-step backward values computed
    from a ZERO b_end, smoother_power(n) -> G^n [L,d,d].  The mirror image of forward_carry_in (SURVEY 8e)."""
    G_ = len(block_lengths)
    if rank == G_ - 1:
        return None
    b_start = np.array(starts_b[G_ - 1], dtype=np.float64)                # the last block has b_end = 0
    for g in range(G_ - 2, rank, -1):
        b_start = starts_b[g] + np.einsum("lij,nlj->nli", smoother_power(int(block_lengths[g])), b_start)
    return b_start


class TimeShardedFilterSmoother(object):
    """Fused filter + smoother + NLL of ONE long sequence (or N of them) whose contiguous time blocks live on different
    ranks: forward carry exchange, then the mirror-image backward exchange, two all-gathers of O(L d) doubles and one
    all-reduce of the NLL, all queued on the device.  ``model`` provides ``fsn_block_async(phase, ...)`` and
    ``fsn_carry_device(direction, ...)`` (``MOIHGPSequences``); every block but the last holds a multiple of 256 steps
    (``time_block_bounds_aligned``)."""

    def __init__(self, model, block_lengths, smoother_mode=1, group=None, device=None):
        import torch
        self.model, self.group, self.mode = model, group, int(smoother_mode)
        self.block_lengths = [int(b) for b in block_lengths]
        self.dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())

    def _buffers(self, N):
        import torch
        if getattr(self, "_bufN", None) != N:
            L, d, G = self.model.num_latent, self.model.igp_dim, len(self.block_lengths)
            f64 = dict(dtype=torch.float64, device=self.dev)
            self._p1, self._g1 = torch.zeros((N, L, d + 1), **f64), torch.zeros((G, N, L, d + 1), **f64)
            self._p2, self._g2 = torch.zeros((N, L, d), **f64), torch.zeros((G, N, L, d), **f64)
            self._xin, self._uaf, self._bend = torch.zeros((N, L, d), **f64), torch.zeros((N, L), **f64), torch.zeros((N, L, d), **f64)
            self._nll = torch.zeros(N, **f64)
            self._bufN = N
        return self

    def enqueue(self, Y_block, X, Xs, x0=None, nll=None, xT=None):
        """The whole exchange queued on torch's current stream with NO host round trip: phase 1 -> NCCL all-gather ->
        forward carry kernel -> phase 2 -> all-gather -> backward carry kernel -> phase 3 -> all-reduce of the NLL.
        x0: torch CUDA tensor [N,L,d] (state before the first step of the WHOLE sequence) or None.  Returns the device
        tensor that will hold the NLL [N] of the whole sequence."""
        dist = _dist()
        m = self.model
        N = Y_block.shape[0]
        multi, world, rank = _ranks(self.group)
        last = rank == world - 1
        b = self._buffers(N)
        nll_dev = nll if nll is not None else b._nll
        if not multi:
            m.fsn_block_async(1, Y_block, True, self.mode, out=b._p1)
            m.fsn_block_async(2, Y_block, True, self.mode, x0=x0, out=b._p2)
            m.fsn_block_async(3, Y_block, True, self.mode, x0=x0, X=X, Xs=Xs, nll=nll_dev, xT=xT)
            return nll_dev
        m.fsn_block_async(1, Y_block, last, self.mode, out=b._p1)
        _all_gather_into(b._g1, b._p1, self.group)
        m.fsn_carry_device(0, b._g1, self.block_lengths, rank, b._xin, self.mode, x0=x0, u_after=b._uaf)
        u_after = None if last else b._uaf
        m.fsn_block_async(2, Y_block, last, self.mode, x0=b._xin, u_after=u_after, out=b._p2)
        _all_gather_into(b._g2, b._p2, self.group)
        m.fsn_carry_device(1, b._g2, self.block_lengths, rank, b._bend, self.mode)
        m.fsn_block_async(3, Y_block, last, self.mode, x0=b._xin, u_after=u_after, b_end=None if last else b._bend, X=X, Xs=Xs,
                          nll=nll_dev, xT=xT)
        dist.all_reduce(nll_dev, op=dist.ReduceOp.SUM, group=self.group)
        return nll_dev

    def __call__(self, Y_block, X, Xs, x0=None, nll=None, xT=None):
        """``enqueue`` and a synchronise.  Y_block [N,n,p], X / Xs [N,n,L,d] (this rank's block, tensors on the device); x0
        [N,L,d] (NumPy or None) is the state before the first step of the WHOLE sequence; returns its nll [N] (NumPy)."""
        import torch
        N, L, d = Y_block.shape[0], self.model.num_latent, self.model.igp_dim
        if x0 is not None:
            x0 = torch.from_numpy(np.ascontiguousarray(np.asarray(x0, dtype=np.float64).reshape(N, L, d))).to(self.dev)
        # a copy: on a CPU device .cpu() would hand out the buffer the next call overwrites
        return self.enqueue(Y_block, X, Xs, x0=x0, nll=nll, xT=xT).cpu().numpy().copy()


class TimeShardedPosteriorSampler(object):
    """Posterior sample paths of ONE long sequence (or N of them) whose contiguous time blocks live on different ranks
    (DESIGN 4.8, 6): the RTS mean by ``TimeShardedFilterSmoother`` (smoother_mode 1), then the sampler's noise process, whose
    backward exchange is the RTS smoother's with N -> S N: every rank runs its block from a zero carry (sampler phase 1),
    all-gathers the S N L d start values, forms its carry from the right with ``fsn_carry_device(1, ..., smoother_mode=1)``
    and draws its block (phase 2).  The draws equal those of the whole-sequence call with the same seed: the random numbers
    are indexed by the global step.  ``model`` provides the ``TimeShardedFilterSmoother`` interface and ``sample_block_async``
    (``MOIHGPSequences``); every block but the last holds a multiple of 256 steps (``time_block_bounds_aligned``)."""

    def __init__(self, model, block_lengths, group=None, device=None):
        import torch
        self.model, self.group = model, group
        self.block_lengths = [int(b) for b in block_lengths]
        self.dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.mean = TimeShardedFilterSmoother(model, self.block_lengths, 1, group=group, device=self.dev)

    def _buffers(self, N, n, S):
        import torch
        if getattr(self, "_shape", None) != (N, n, S):
            L, d, G = self.model.num_latent, self.model.igp_dim, len(self.block_lengths)
            f64 = dict(dtype=torch.float64, device=self.dev)
            self._X, self._Xs = torch.zeros((N, n, L, d), **f64), torch.zeros((N, n, L, d), **f64)
            self._e1, self._eg, self._eend = (torch.zeros(s, **f64) for s in ((S * N, L, d), (G, S * N, L, d), (S * N, L, d)))
            self._shape = (N, n, S)
        return self

    def enqueue(self, Y_block, num_samples, seed, Xsamp=None, Fsamp=None, Ysamp=None, x0=None, Xs_mean=None):
        """Queue the whole exchange on torch's current stream with NO host round trip: the time-sharded RTS pass into
        ``Xs_mean`` [N,n,L,d] (a workspace when None) -> sampler phase 1 -> all-gather -> backward carry kernel -> sampler
        phase 2 into Xsamp [S,N,n,L,d], Fsamp [S,N,n,L], Ysamp [S,N,n,p] (this rank's block; at least one).  x0 [N,L,d]: the
        state before the first step of the WHOLE sequence or None.  Returns the tensor holding the RTS mean."""
        m = self.model
        N, n, S = int(Y_block.shape[0]), int(Y_block.shape[1]), int(num_samples)
        multi, world, rank = _ranks(self.group)
        last = rank == world - 1
        b = self._buffers(N, n, S)
        Xs = Xs_mean if Xs_mean is not None else b._Xs
        self.mean.enqueue(Y_block, b._X, Xs, x0=x0)
        outs = dict(Xsamp=Xsamp, Fsamp=Fsamp, Ysamp=Ysamp)
        if not multi:
            m.sample_block_async(2, Xs, S, seed, 0, True, **outs)
            return Xs
        t0 = sum(self.block_lengths[:rank])
        m.sample_block_async(1, Xs, S, seed, t0, last, out=b._e1)
        _all_gather_into(b._eg, b._e1, self.group)
        m.fsn_carry_device(1, b._eg, self.block_lengths, rank, b._eend, smoother_mode=1)
        m.sample_block_async(2, Xs, S, seed, t0, last, e_end=None if last else b._eend, **outs)
        return Xs
