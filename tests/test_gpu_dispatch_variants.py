"""GPU tests (-m gpu) of the kernel variants that the default inputs of the other suites never select, each against the CPU
oracle at conftest.TOL and, where the same call on default inputs exists, against that call:
  A. device operands that are 8-byte but not 16-byte aligned (a contiguous view at an odd element offset), between
     sentinel guard zones;
  B. host-buffer calls that span several pipeline slices (double-buffered device buffers, per-slice NaN flags, slices of
     one call on different paths);
  C. the many-chains kernels with fewer sequences per warp (moihgp_cuda_set_chain_seqs_per_warp);
  D. every k_project_rows configuration and k_project_mma, each on shapes that select it.
Every test checks that its variant was reached (profile records, pointer alignment, slice counts, the shape rule of the
projection), so that a later dispatch change fails it instead of leaving it passing without testing anything."""
import numpy as np
import pytest

from conftest import TOL, literal_smoother_err, rel_err

pytestmark = pytest.mark.gpu

SENT = 1234.5      # guard-zone sentinel
GZ = 64            # guard zone (doubles) on either side of a payload


def _model(kernel, p, L, seed, threading=True, table=None):
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_params
    rng = np.random.default_rng(seed)
    params = make_params(rng, p, L, kernel, table)
    m = MOIHGPSequences(0.1, p, L, kernel, threading)
    o = OracleMOIHGP(0.1, p, L, kernel, threading)
    m.update(params)
    o.update(params)
    return m, o, rng


def _data(rng, p, L, N, T):
    from oracle.gen_golden import make_data
    return np.stack([make_data(rng, p, L, T) for _ in range(N)])


def _states_close(a, b, mode, tol, what=None):
    """smoothed (or filtered, mode 1) states a against b: norm-wise in RTS mode; in the literal mode through
    literal_smoother_err (a latent with rho(G) > 1 is compared over the tail where b is finite)"""
    if mode == 1:
        assert rel_err(a, b) < tol, (what, rel_err(a, b))
    else:
        err, steps = literal_smoother_err(a, b)
        assert err < tol and steps >= min(np.asarray(b).shape[-3], 100), (what, err, steps)


def _nll_close(a, b, tol, what=None):
    """same NaN pattern (a sequence with a missing output has a NaN NLL), finite entries within tol"""
    a, b = np.asarray(a), np.asarray(b)
    assert np.array_equal(np.isnan(a), np.isnan(b)), what
    ok = ~np.isnan(b)
    if ok.any():
        assert rel_err(a[ok], b[ok]) < tol, what


class Guarded:
    """Device payloads between sentinel guard zones, either 16-byte aligned or at an 8-byte offset (one double past a
    16-byte boundary: a contiguous view at an odd element offset of a torch allocation)."""

    def __init__(self):
        self.bufs = []

    def new(self, shape, offset, fill=None):
        import torch
        n = int(np.prod(shape))
        lo = GZ + (1 if offset else 0)
        buf = torch.full((lo + n + GZ,), SENT, dtype=torch.float64, device="cuda")
        view = buf[lo:lo + n].view(*shape)
        assert view.data_ptr() % 16 == (8 if offset else 0)
        if fill is not None:
            view.copy_(torch.from_numpy(np.ascontiguousarray(fill, dtype=np.float64)))
        self.bufs.append((buf, lo, n))
        return view

    def check(self):
        import torch
        torch.cuda.synchronize()
        for buf, lo, n in self.bufs:
            h = buf.cpu().numpy()
            assert np.all(h[:lo] == SENT) and np.all(h[lo + n:] == SENT), "store outside the payload"


def _np(t):
    return t.cpu().numpy()


def _profiled(m, fn):
    m.profile(True)
    fn()
    prof = m.profile_read()
    m.profile(False)
    return prof


# ======================================================================================== A. offset device operands
FUSED_OPERANDS = ["Y", "X", "Xs", "Yhat", "x0", "nll", "xT", "all"]


def _fused_device(m, g, Y, x0, mode, off, N, T):
    """the fused pass on guarded device buffers; `off`: names of the operands placed at an 8-byte offset"""
    p, L, d = m.num_output, m.num_latent, m.igp_dim
    t = {"Y": g.new((N, T, p), "Y" in off, Y), "x0": g.new((N, L, d), "x0" in off, x0), "X": g.new((N, T, L, d), "X" in off),
         "Xs": g.new((N, T, L, d), "Xs" in off), "Yhat": g.new((N, T, p), "Yhat" in off), "nll": g.new((N,), "nll" in off),
         "xT": g.new((N, L, d), "xT" in off)}
    prof = _profiled(m, lambda: m.filter_smoother_nll_device(t["Y"], x0=t["x0"], smoother_mode=mode, X=t["X"], Xs=t["Xs"], Yhat=t["Yhat"],
                                                             nll=t["nll"], xT=t["xT"]))
    g.check()
    return {k: _np(t[k]) for k in ("X", "Xs", "Yhat", "nll", "xT")}, prof


@pytest.mark.parametrize("which", FUSED_OPERANDS)
def test_fused_pass_with_an_offset_operand(cuda_lib, which):
    """600 sequences x 8 latents = 150 warps of chains: the automatic choice takes the many-chains kernels on aligned
    buffers.  An offset Y, X or Xs sends the pass to the chunked scan (the many-chains kernels move them in 16-byte pieces);
    an offset Yhat, x0, nll or xT keeps it on the many-chains kernels.  Either way the outputs equal the oracle's and the
    aligned call's (on the same path), and nothing is written outside the payloads."""
    p, L, N, T = 16, 8, 600, 40
    m, o, rng = _model("Matern52", p, L, 61)
    Y = _data(rng, p, L, N, T)
    x0 = 0.2 * rng.standard_normal((N, L, m.igp_dim))
    off = FUSED_OPERANDS[:-1] if which == "all" else [which]
    to_scan = any(k in off for k in ("Y", "X", "Xs"))
    for mode in (1, 0):
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True, nthreads=8)
        r, prof = _fused_device(m, Guarded(), Y, x0, mode, off, N, T)
        assert ("k_scan_final" in prof) == to_scan and ("k_filter_chain" in prof) == (not to_scan), (which, sorted(prof))
        for k in ("X", "Yhat", "xT", "nll"):
            assert rel_err(r[k], ro[k]) < TOL, (which, mode, k)
        _states_close(r["Xs"], ro["Xs"], mode, TOL, (which, mode))
        m.set_path("scan" if to_scan else "auto")              # the same call on aligned buffers, on the same path
        a, aprof = _fused_device(m, Guarded(), Y, x0, mode, [], N, T)
        m.set_path("auto")
        assert ("k_scan_final" in aprof) == to_scan
        for k in ("X", "Yhat", "xT", "nll"):
            assert rel_err(r[k], a[k]) < 1e-13, (which, mode, k)
        _states_close(r["Xs"], a["Xs"], mode, 1e-13, (which, mode))


@pytest.mark.parametrize("which", ["Y", "X", "Xs"])
def test_forced_many_chains_path_refuses_offset_operands(cuda_lib, which):
    """With the path forced to the many-chains kernels an offset Y, X or Xs is refused (nothing is written), and the handle
    serves the next, aligned call correctly."""
    p, L, N, T = 16, 8, 600, 40
    m, o, rng = _model("Matern52", p, L, 62)
    Y = _data(rng, p, L, N, T)
    x0 = 0.2 * rng.standard_normal((N, L, m.igp_dim))
    m.set_path("chain")
    g = Guarded()
    with pytest.raises(RuntimeError, match="many-chains path not available"):
        _fused_device(m, g, Y, x0, 1, [which], N, T)
    g.check()
    r, prof = _fused_device(m, Guarded(), Y, x0, 1, [], N, T)
    assert "k_filter_chain" in prof
    ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=1, nthreads=8)
    for k in ("X", "Xs", "nll", "xT"):
        assert rel_err(r[k], ro[k]) < TOL, k


@pytest.mark.parametrize("kernel,p,L,N,T", [("Matern32", 64, 32, 1, 3000), ("Matern52", 16, 8, 2, 1300), ("Matern32", 12, 5, 2, 700),
                                            ("Matern32", 64, 30, 1, 3000)])
def test_scan_path_with_offset_states(cuda_lib, kernel, p, L, N, T):
    """The chunked scan writing X / Xs / xT at an 8-byte offset: the final-pass kernels then store element by element
    instead of in 16-byte pieces - k_scan_lanes (L a multiple of 8) and the warp-per-chunk k_scan (other L).  Oracle and
    aligned call agree."""
    m, o, rng = _model(kernel, p, L, 63 + p)
    Y = _data(rng, p, L, N, T)
    x0 = 0.3 * rng.standard_normal((N, L, m.igp_dim))
    m.set_path("scan")
    for mode in (1, 0):
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True, nthreads=8)
        r, prof = _fused_device(m, Guarded(), Y, x0, mode, ["X", "Xs", "xT"], N, T)
        assert "k_scan_final" in prof and "k_filter_chain" not in prof
        a, _ = _fused_device(m, Guarded(), Y, x0, mode, [], N, T)
        for k in ("X", "Yhat", "xT", "nll"):
            assert rel_err(r[k], ro[k]) < TOL, (mode, k)
            assert rel_err(r[k], a[k]) < 1e-13, (mode, k)
        _states_close(r["Xs"], ro["Xs"], mode, TOL, mode)
        _states_close(r["Xs"], a["Xs"], mode, 1e-13, mode)


def _with_missing(Y, L, rng):
    """missing outputs: scattered single NaNs (at least L + 2 observed outputs left in a row) and one all-missing row"""
    Y = Y.copy()
    N, T, p = Y.shape
    Y[0, 3, 1] = np.nan
    Y[0, T // 2, :] = np.nan
    Y[N - 1, T - 1, 0] = np.nan
    miss = rng.random((T, p)) < 0.1
    miss[(~miss).sum(axis=1) < L + 2] = False
    Y[N - 1][miss] = np.nan
    return Y


@pytest.mark.parametrize("kernel,p,L,N,T", [("Matern52", 16, 8, 3, 300), ("Matern32", 64, 32, 1, 600), ("Matern32", 40, 12, 2, 257)])
def test_offset_observations_with_even_outputs_and_missing_rows(cuda_lib, kernel, p, L, N, T):
    """An offset Y with an even p >= 8 cannot go through the TMA / tensor-pipe projections: the scalar k_project serves it,
    and k_nan_fix re-projects the rows with missing outputs from the same offset Y."""
    m, o, rng = _model(kernel, p, L, 64 + p)
    Y = _with_missing(_data(rng, p, L, N, T), L, rng)
    x0 = 0.3 * rng.standard_normal((N, L, m.igp_dim))
    ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=1, want_yhat=True, nthreads=8)
    r, prof = _fused_device(m, Guarded(), Y, x0, 1, ["Y"], N, T)
    assert "k_project" in prof and "k_scan_final" in prof
    assert m.nan_status == 1
    m.set_path("scan")
    a, _ = _fused_device(m, Guarded(), Y, x0, 1, [], N, T)
    for k in ("X", "Xs", "Yhat", "xT"):
        assert np.all(np.isfinite(r[k])), k
        assert rel_err(r[k], ro[k]) < TOL, k
        assert rel_err(r[k], a[k]) < 1e-13, k
    _nll_close(r["nll"], ro["nll"], TOL)
    _nll_close(r["nll"], a["nll"], 1e-13)
    assert np.isnan(r["nll"][0])


@pytest.mark.parametrize("kernel,p,L,N,T", [("Matern52", 16, 8, 3, 1300), ("Matern32", 64, 32, 1, 2000), ("Matern32", 8, 4, 5, 512)])
def test_device_objective_with_offset_operands(cuda_lib, kernel, p, L, N, T):
    """objective_device with Y, x0, dx0, loss, grad, xT and dxT at an 8-byte offset: even p and T, but the offset Y sends
    the dU contraction to the scalar k_gradU (and the projection to k_project).  Loss, gradient and final state equal the
    oracle's and the aligned call's (the dU sums run in another order there, hence 1e-12 for the gradient)."""
    import torch
    m, o, rng = _model(kernel, p, L, 65 + p)
    Y = _data(rng, p, L, N, T)
    d, npar = m.igp_dim, m.num_param
    x0 = 0.2 * rng.standard_normal((N, L, d))
    dx0 = 0.1 * rng.standard_normal((N, L, 3, d))
    res = {}
    for off in (True, False):
        g = Guarded()
        t = [g.new((N, T, p), off, Y), g.new((N, L, d), off, x0), g.new((N, L, 3, d), off, dx0), g.new((1,), off),
             g.new((npar,), off), g.new((N, L, d), off), g.new((N, L, 3, d), off)]
        m.objective_device(t[0], t[3], t[4], x0=t[1], dx0=t[2], xT=t[5], dxT=t[6])
        g.check()
        res[off] = [float(_np(t[3])[0]), _np(t[4]), _np(t[5]), _np(t[6])]
    torch.cuda.synchronize()
    lo, go, xo, dxo = o.objective(Y, x0=x0, dx0=dx0)
    lr, gr, xr, dxr = res[True]
    la, ga, xa, dxa = res[False]
    assert abs(lr - lo) <= TOL * abs(lo) and rel_err(gr, go) < TOL
    assert rel_err(xr, xo) < TOL and rel_err(dxr, dxo) < TOL
    assert abs(lr - la) <= 1e-13 * abs(la) and rel_err(gr, ga) < 1e-12
    assert rel_err(xr, xa) < 1e-13 and rel_err(dxr, dxa) < 1e-13


def test_device_sampling_with_offset_outputs(cuda_lib):
    """sample_posterior_device with Y, x0, the RTS mean Xs and the sample outputs X, F, Ysamp at an 8-byte offset: the mean
    pass moves from the many-chains kernels to the chunked scan, the draws are the same (the noise does not depend on the
    path), and the mean equals the oracle's RTS smoother."""
    p, L, N, T, S, seed = 16, 8, 600, 40, 2, 0xABCDEF
    m, o, rng = _model("Matern52", p, L, 66)
    Y = _data(rng, p, L, N, T)
    x0 = 0.2 * rng.standard_normal((N, L, m.igp_dim))
    d = m.igp_dim
    res, profs = {}, {}
    for off in (True, False):
        g = Guarded()
        Yd, x0d = g.new((N, T, p), off, Y), g.new((N, L, d), off, x0)
        Xs, X, F, Ys = g.new((N, T, L, d), off), g.new((S, N, T, L, d), off), g.new((S, N, T, L), off), g.new((S, N, T, p), off)
        profs[off] = _profiled(m, lambda: m.sample_posterior_device(Yd, seed, x0=x0d, Xs=Xs, X=X, F=F, Ysamp=Ys))
        g.check()
        res[off] = [_np(a) for a in (Xs, X, F, Ys)]
    assert "k_scan_final" in profs[True] and "k_filter_chain" not in profs[True]
    assert "k_filter_chain" in profs[False]
    for k, (a, b) in enumerate(zip(res[True], res[False])):
        assert rel_err(a, b) < 1e-13, k
    ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=1, nthreads=8)
    assert rel_err(res[True][0], ro["Xs"]) < TOL
    assert np.array_equal(res[True][2], res[True][1][..., 0])


@pytest.mark.parametrize("kernel,mode", [("Matern52", 1), ("Matern52", 0), ("Matern32", 1), ("Matern32", 0)])
def test_smooth_dev_with_offset_states(cuda_lib, kernel, mode):
    """moihgp_cuda_smooth_dev over caller-supplied filtered states at an 8-byte offset, into Xs at an 8-byte offset: the
    oracle's smoother over the oracle's own filtered states, and the host-buffer call."""
    import torch
    from multioutputihgp_b200.batched import _torch_stream
    p, L, N, T = 8, 4, 3, 333
    m, o, rng = _model(kernel, p, L, 67)
    Y = _data(rng, p, L, N, T)
    ro = o.filter_smoother_nll(Y, smoother_mode=mode)
    d = m.igp_dim
    g = Guarded()
    X, Xs = g.new((N, T, L, d), True, ro["X"]), g.new((N, T, L, d), True)
    m.set_stream(_torch_stream(X.device))
    m._check(m._lib.moihgp_cuda_smooth_dev(m._h, X.data_ptr(), N, T, mode, Xs.data_ptr()))
    g.check()
    torch.cuda.synchronize()
    _states_close(_np(Xs), ro["Xs"], mode, TOL)
    _states_close(_np(Xs), m.smooth(ro["X"], mode), mode, 1e-13)


def test_objective_blocks_with_offset_operands(cuda_lib):
    """The one-pass time-sharded objective on one device (begin / finish per block, as test_objective_begin_finish_blocks_
    equal_the_whole_sequence) with every block's Y, carry-in and [loss, grad] at an 8-byte offset: the blocks add up to the
    whole-sequence evaluation and to the oracle's."""
    import torch
    from multioutputihgp_b200.parallel import carry_in_from_block_ends, stack_consts
    kernel, p, L, T, cut = "Matern52", 8, 4, 3000, 1024
    m, o, rng = _model(kernel, p, L, 68)
    Y = _data(rng, p, L, 1, T)[0]
    lw, gw = m.objective(Y[None])
    d = m.igp_dim
    g = Guarded()
    Yd = [g.new((1, cut, p), True, Y[:cut]), g.new((1, T - cut, p), True, Y[cut:])]
    loss = [g.new((1,), True) for _ in range(2)]
    grad = [g.new((m.num_param,), True) for _ in range(2)]
    ex, edx = m.objective_begin_device(Yd[0])
    m.objective_finish_device(Yd[0], loss[0], grad[0])
    consts = stack_consts([m.latent_consts(l) for l in range(L)])
    xin, dxin = carry_in_from_block_ends(consts, [cut, T - cut], [ex[0], np.zeros((L, d))], [edx[0], np.zeros((L, 3, d))], np.zeros((L, d)),
                                         np.zeros((L, 3, d)), 1)
    m.objective_begin_device(Yd[1], want_end=False)
    m.objective_finish_device(Yd[1], loss[1], grad[1], x0=g.new((1, L, d), True, xin[None]), dx0=g.new((1, L, 3, d), True, dxin[None]))
    g.check()
    torch.cuda.synchronize()
    lt = float(_np(loss[0])[0] + _np(loss[1])[0])
    gt = _np(grad[0]) + _np(grad[1])
    assert abs(lt - lw) <= 1e-10 * abs(lw) and rel_err(gt, gw) < TOL
    lo, go, _, _ = o.objective(Y[None])
    assert abs(lt - lo) <= TOL * abs(lo) and rel_err(gt, go) < TOL


def test_filter_smoother_blocks_with_offset_operands(cuda_lib):
    """The three-phase time-sharded fused pass (as test_time_sharded_filter_smoother_blocks_equal_the_whole_sequence) with
    every block's Y, carries and outputs X, Xs, nll, xT at an 8-byte offset: equal to the whole-sequence pass and the
    oracle's, in both smoother modes."""
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    from multioutputihgp_b200.parallel import backward_carry_in, forward_carry_in
    from oracle.gen_golden import LITERAL_STABLE
    kernel, p, L, N, cuts = "Matern32", 12, 5, 1, (0, 768, 800)
    whole, o, rng = _model(kernel, p, L, 69, table=LITERAL_STABLE)      # rho(G) < 1 in the literal mode: whole sequences compared
    params = whole.params
    T, G = cuts[-1], len(cuts) - 1
    lengths = [cuts[i + 1] - cuts[i] for i in range(G)]
    Y = _data(rng, p, L, N, T)
    whole.set_path("scan")
    d = whole.igp_dim
    x0 = 0.3 * rng.standard_normal((N, L, d))
    models = []
    for _ in range(G):
        mb = MOIHGPSequences(0.1, p, L, kernel, True)
        mb.update(params)
        models.append(mb)
    for mode in (1, 0):
        gd = Guarded()
        Yd = [gd.new((N, lengths[i], p), True, Y[:, cuts[i]:cuts[i + 1]]) for i in range(G)]
        ref = whole.filter_smoother_nll(Y, x0=x0, smoother_mode=mode)
        ph1 = [models[i].fsn_block(1, Yd[i], i == G - 1, mode) for i in range(G)]
        ends, ufirst = [a for a, _ in ph1], [b for _, b in ph1]
        x_in = [gd.new((N, L, d), True, forward_carry_in(models[0].block_transition, lengths, ends, x0, i)) for i in range(G)]
        u_after = [gd.new((N, L), True, ufirst[i + 1]) if i < G - 1 else None for i in range(G)]
        b0 = [models[i].fsn_block(2, Yd[i], i == G - 1, mode, x0=x_in[i], u_after=u_after[i]) for i in range(G)]
        X = [gd.new((N, lengths[i], L, d), True) for i in range(G)]
        Xs = [gd.new((N, lengths[i], L, d), True) for i in range(G)]
        nll = [gd.new((N,), True) for i in range(G)]
        xT = gd.new((N, L, d), True)
        for i in range(G):
            be = backward_carry_in(lambda n_: models[0].smoother_power(n_, mode), lengths, b0, i)
            models[i].fsn_block(3, Yd[i], i == G - 1, mode, x0=x_in[i], u_after=u_after[i], b_end=None if be is None else gd.new((N, L, d), True, be),
                                X=X[i], Xs=Xs[i], nll=nll[i], xT=xT if i == G - 1 else None)
        gd.check()
        torch.cuda.synchronize()
        Xc = np.concatenate([_np(x) for x in X], axis=1)
        Xsc = np.concatenate([_np(x) for x in Xs], axis=1)
        nsum = sum(_np(n_) for n_ in nll)
        assert rel_err(Xc, ref["X"]) < 1e-12 and rel_err(nsum, ref["nll"]) < 1e-12 and rel_err(_np(xT), ref["xT"]) < 1e-12, mode
        _states_close(Xsc, ref["Xs"], mode, 1e-11, mode)
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode)
        assert rel_err(Xc, ro["X"]) < TOL and rel_err(nsum, ro["nll"]) < TOL, mode
        _states_close(Xsc, ro["Xs"], mode, TOL, mode)


# ======================================================================================== B. multi-slice host calls
def _slice_len(N, L):
    """sequences per slice of the pipelined host-buffer pass (fsn_host): a warp of chains per SM, at most sixteen slices,
    a multiple of 32"""
    ns = max(-(-148 * 32 // L), -(-N // 16))
    return min(-(-ns // 32) * 32, N)


@pytest.mark.parametrize("kernel,p,L,N,T,slices,paths", [("Matern52", 16, 8, 1300, 40, [608, 608, 84], ("k_filter_chain", "k_scan_final")),
                                                         ("Matern32", 64, 32, 5000, 8, [320] * 15 + [200], ("k_scan_final",)),
                                                         ("Matern32", 4, 1, 10000, 16, [4736, 4736, 528], ("k_filter_chain", "k_scan_final"))])
def test_host_call_over_several_slices(cuda_lib, kernel, p, L, N, T, slices, paths):
    """Host buffers with N above one pipeline slice: both device buffer sets and the event waits from the third slice on,
    a ragged last slice, full slices on the many-chains kernels and a short last slice on the chunked scan, per-slice NaN
    flags, the values-only extraction, and calls with one and with two buffer sets in a row on one handle."""
    ns = _slice_len(N, L)
    assert [min(ns, N - i) for i in range(0, N, ns)] == slices
    m, o, rng = _model(kernel, p, L, N + T)
    Y = _data(rng, p, L, N, T)
    x0 = 0.2 * rng.standard_normal((N, L, m.igp_dim))
    for mode in (1, 0):
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True, nthreads=8)
        res = {}
        prof = _profiled(m, lambda: res.update(r=m.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True)))
        r = res["r"]
        assert all(k in prof for k in paths), sorted(prof)
        if len(paths) == 1:
            assert "k_filter_chain" not in prof
        for k in ("X", "Yhat", "nll", "xT"):
            assert rel_err(r[k], ro[k]) < TOL, (mode, k)
        _states_close(r["Xs"], ro["Xs"], mode, TOL, mode)
        v = m.filter_smoother_nll_values(Y, x0=x0, smoother_mode=mode, want_yhat=True)
        assert np.array_equal(v["F"], r["X"][..., 0]) and np.array_equal(v["Fs"], r["Xs"][..., 0]), mode
        for k in ("Yhat", "nll", "xT"):
            assert np.array_equal(v[k], r[k]), (mode, k)
    # NLL only, no states
    r1 = m.filter_smoother_nll(Y, x0=x0, smoother_mode=-1, want_states=False)
    assert rel_err(r1["nll"], ro["nll"]) < TOL and rel_err(r1["xT"], ro["xT"]) < TOL
    # a missing output in one sequence of a middle slice and one of the last slice: exactly their NLLs are NaN
    Yn = Y.copy()
    bad = [ns * (len(slices) // 2) + 5, N - 2]
    for n_ in bad:
        Yn[n_, T // 2, 0] = np.nan
    ron = o.filter_smoother_nll(Yn, x0=x0, smoother_mode=1, nthreads=8)
    rn = m.filter_smoother_nll(Yn, x0=x0, smoother_mode=1)
    assert list(np.nonzero(np.isnan(rn["nll"]))[0]) == bad
    _nll_close(rn["nll"], ron["nll"], TOL)
    for k in ("X", "Xs", "xT"):
        assert np.all(np.isfinite(rn[k])) and rel_err(rn[k], ron[k]) < TOL, k
    # one slice (one buffer set), then several slices (two) again, on the same handle
    Nsmall = min(ns, 300)
    rs = m.filter_smoother_nll(Y[:Nsmall], x0=x0[:Nsmall], smoother_mode=1, want_yhat=True)
    ros = o.filter_smoother_nll(Y[:Nsmall], x0=x0[:Nsmall], smoother_mode=1, want_yhat=True, nthreads=8)
    for k in ("X", "Xs", "Yhat", "nll", "xT"):
        assert rel_err(rs[k], ros[k]) < TOL, k
    r2 = m.filter_smoother_nll(Y, x0=x0, smoother_mode=0, want_yhat=True)
    for k in ("X", "Xs", "Yhat", "nll", "xT"):
        assert np.array_equal(r2[k], r[k]), k          # r: the same call (mode 0) before



# ======================================================================================== C. sequences per warp
SPW_16x8, SPW_8x4 = (1, 2, 3, 4, 0), (2, 4, 8, 0)


@pytest.mark.parametrize("kernel,p,L,spws", [("Matern52", 16, 8, SPW_16x8), ("Matern32", 16, 8, SPW_16x8), ("Matern52", 8, 4, SPW_8x4),
                                             ("Matern32", 8, 4, SPW_8x4),
                                             ("Matern52", 12, 6, SPW_16x8),     # padded outputs and latents, served by 16x8
                                             ("Matern32", 6, 3, SPW_8x4),       # ... by 8x4
                                             ("Matern52", 5, 4, SPW_8x4)])      # odd p (8-byte rows of Y), served by 8x4
def test_many_chains_with_fewer_sequences_per_warp(cuda_lib, kernel, p, L, spws):
    """The 16x8 and 8x4 many-chains instantiations also compile k_filter_chain with 2 and 1 (4 and 2) sequences per warp,
    and the smoother then runs with rounds of L steps (RM = 1): every setting of the knob against the oracle and against
    the automatic full warp, with ragged N and T, a carried-in state, missing outputs and both smoother modes."""
    N, T = 11, 83
    m, o, rng = _model(kernel, p, L, 70 + p + L)
    Y = _data(rng, p, L, N, T)
    Y[0, 5, :] = np.nan                         # everything missing
    if p >= L + 3:
        Y[N - 1, T - 2, 0] = np.nan
    x0 = 0.2 * rng.standard_normal((N, L, m.igp_dim))
    m.set_path("chain")
    for mode in (1, 0):
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True)
        base = None
        for spw in reversed(spws):               # 0 (automatic) first
            m.set_chain_seqs_per_warp(spw)
            res = {}
            prof = _profiled(m, lambda: res.update(r=m.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True)))
            r = res["r"]
            assert "k_filter_chain" in prof and "k_smooth_chain" in prof, (spw, sorted(prof))
            for k in ("X", "Yhat", "xT"):
                assert rel_err(r[k], ro[k]) < TOL, (spw, mode, k)
            _nll_close(r["nll"], ro["nll"], TOL, (spw, mode))
            _states_close(r["Xs"], ro["Xs"], mode, TOL, (spw, mode))
            if base is None:
                base = r
            else:
                for k in ("X", "Yhat", "xT"):
                    assert rel_err(r[k], base[k]) < 1e-13, (spw, mode, k)
                _nll_close(r["nll"], base["nll"], 1e-13, (spw, mode))
                _states_close(r["Xs"], base["Xs"], mode, 1e-13, (spw, mode))
    m.set_chain_seqs_per_warp(0)


def test_sequences_per_warp_knob_is_inert_on_full_warp_only_shapes(cuda_lib):
    """32x2 is instantiated with the full warp only: every setting of the knob gives the bitwise-same outputs."""
    p, L, N, T = 32, 2, 19, 70
    m, o, rng = _model("Matern32", p, L, 71)
    Y = _data(rng, p, L, N, T)
    m.set_path("chain")
    m.set_chain_seqs_per_warp(0)
    a = m.filter_smoother_nll(Y, smoother_mode=1, want_yhat=True)
    ro = o.filter_smoother_nll(Y, smoother_mode=1, want_yhat=True)
    assert rel_err(a["X"], ro["X"]) < TOL and rel_err(a["Xs"], ro["Xs"]) < TOL
    for spw in (1, 2, 4, 8):
        m.set_chain_seqs_per_warp(spw)
        b = m.filter_smoother_nll(Y, smoother_mode=1, want_yhat=True)
        for k in ("X", "Xs", "Yhat", "nll", "xT"):
            assert np.array_equal(a[k], b[k]), (spw, k)


# ======================================================================================== D. projection variants
# k_project_rows<NB> configurations in the order of project.cu's try_project_rows -> (warps NW, stages NST, boxes per stage
# NBOX); nb_all = ceil(p / 16)
ROWS_CFGS = {1: lambda nb: (16, 2, min(nb, 2)), 2: lambda nb: (16, 3, 1), 5: lambda nb: (8, 2, min(nb, 2)), 8: lambda nb: (8, 2, 1)}


def _rows_smem(NB, p, nw, nst, nbox):
    """RowsSmem<NB>::bytes (project.cu): 1024 B slack + rings nw * nst * nbox * 2048 B + U (p rounded up to 16) x (8 NB + 4)
    doubles + S^-1/2 (8 NB doubles) + per-warp scratch (2 * 6 * 32 + 2 doubles) + barriers (nw * nst * 8 B)"""
    return 1024 + nw * nst * nbox * 2048 + ((p + 15) & ~15) * (8 * NB + 4) * 8 + 8 * NB * 8 + nw * 386 * 8 + nw * nst * 8


def _projection_variant(NB, p):
    """the kernel launch_project picks for a 16-byte aligned Y with even p >= 8 at panel width NB: the first k_project_rows
    configuration whose shared memory fits into 227 KB, else k_project_mma"""
    for cfg, shape in ROWS_CFGS.items():
        if _rows_smem(NB, p, *shape((p + 15) // 16)) <= 227 * 1024:
            return "rows%d" % cfg
    return "mma"


# one shape per panel width NB (L <= 8, 16, 32, 64): (NB, kernel, L, N, T), N > 1 and T not a multiple of 16 (the unit walk
# wraps into the next sequence inside a CTA's stride); per variant the p of each NB that selects it
PROJ_SHAPES = [(1, "Matern52", 6, 3, 203), (2, "Matern32", 12, 2, 301), (4, "Matern52", 20, 2, 150), (8, "Matern32", 40, 2, 130)]
PROJ_P = {"rows1": (40, 24, 48, 48), "rows2": (600, 400, 200, 120), "rows5": (1000, 700, 400, 200), "rows8": (1600, 1000, 540, 280),
          "mma": (1900, 1100, 600, 320)}


@pytest.mark.parametrize("variant", list(PROJ_P))
def test_projection_variant_matches_oracle(cuda_lib, variant):
    """Each k_project_rows configuration and k_project_mma on one shape per panel width that selects it, through the
    chunked-scan fused pass (both smoother modes, missing outputs) and the objective, against the oracle.  Each shape is
    first checked to select its variant under the rule of launch_project, so that a change of that rule fails here."""
    for (NB, kernel, L, N, T), p in zip(PROJ_SHAPES, PROJ_P[variant]):
        assert 8 * NB >= L > 8 * NB // 2 and p % 2 == 0 and p >= 8
        assert _projection_variant(NB, p) == variant, (NB, p)
        m, o, rng = _model(kernel, p, L, NB)
        Y = _data(rng, p, L, N, T)
        Yn = Y.copy()
        Yn[0, 7, :p - L - 2] = np.nan
        Yn[0, 9, :] = np.nan
        Yn[N - 1, T - 1, 1] = np.nan
        x0 = 0.2 * rng.standard_normal((N, L, m.igp_dim))
        dx0 = 0.1 * rng.standard_normal((N, L, 3, m.igp_dim))
        what = (variant, NB, p)
        m.set_path("scan")
        for mode in (1, 0):
            r = m.filter_smoother_nll(Yn, x0=x0, smoother_mode=mode, want_yhat=True)
            ro = o.filter_smoother_nll(Yn, x0=x0, smoother_mode=mode, want_yhat=True, nthreads=8)
            for k in ("X", "Yhat", "xT"):
                assert rel_err(r[k], ro[k]) < TOL, (what, mode, k)
            _states_close(r["Xs"], ro["Xs"], mode, TOL, (what, mode))
            _nll_close(r["nll"], ro["nll"], TOL, (what, mode))
            assert np.isnan(r["nll"][0]), what
        l, g, xT, dxT = m.objective(Y, x0=x0, dx0=dx0, want_state=True)
        lo, go, xo, dxo = o.objective(Y, x0=x0, dx0=dx0)
        assert abs(l - lo) <= TOL * abs(lo) and rel_err(g, go) < TOL, what
        assert rel_err(xT, xo) < TOL and rel_err(dxT, dxo) < TOL, what
        l, g, xT, dxT = m.objective(Yn, x0=x0, dx0=dx0, want_state=True)
        lo, go, xo, dxo = o.objective(Yn, x0=x0, dx0=dx0)
        assert np.isnan(l) and rel_err(xT, xo) < TOL and rel_err(dxT, dxo) < TOL, what
