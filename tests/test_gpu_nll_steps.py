"""Per-step NLL terms of the filter pass (moihgp_cuda_nll_steps*): nll_steps[n][t] = MOIHGP::negLogLikelihood(x_{t-1}, y_t)
(moihgp.h:614-688), the terms the fused pass sums into nll[n].

The GPU tests (-m gpu) compare every term with the CPU oracle's step + negLogLikelihood loop, on both kernel paths (set_path
"chain" = the many-chains kernels, "scan" = the chunked scan), check the sums against the fused pass, and exercise the
device interface (determinism, CUDA-graph capture, refusals)."""
import numpy as np
import pytest

from conftest import TOL, rel_err

BOTH, SCAN = ("chain", "scan"), ("scan",)

# (kernel, p, L, N, T, paths): what each shape exercises
CASES = [
    ("Matern52", 16, 8, 5, 57, BOTH),     # instantiated 16x8; N not a multiple of 4 sequences per warp; T one step past a round
    ("Matern32", 6, 2, 3, 40, BOTH),      # padded even p (8x2 kernels); 16 sequences per warp
    ("Matern32", 5, 3, 2, 33, BOTH),      # padded odd p and padded L (8x4 kernels)
    ("Matern32", 8, 3, 2, 30, BOTH),      # padded L only
    ("Matern52", 6, 3, 2, 42, BOTH),      # odd L with even T, Matern-5/2 (runs of X of 9 doubles per step)
    ("Matern32", 2, 1, 33, 20, BOTH),     # L = 1 with Matern-3/2; N not a multiple of 32 sequences per warp
    ("Matern32", 4, 2, 3, 1, BOTH),       # T = 1
    ("Matern52", 16, 8, 2, 257, BOTH),    # one step past a scan chunk (256 steps)
    ("Matern32", 40, 20, 2, 30, SCAN),    # p > 32, L > 16
    ("Matern32", 64, 32, 1, 24, SCAN),    # the config-4 shape
    ("Matern32", 256, 64, 1, 6, SCAN),    # the config-5 shape
]
PARAMS = [pytest.param(path, *c[:5], id="%s-%s-p%dL%d-N%dT%d" % ((path,) + c[:5])) for c in CASES for path in c[5]]


def _setup(kernel, p, L, N, T, seed, nan=False, x0=False):
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(seed)
    params = make_params(rng, p, L, kernel)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    d = 2 if kernel == "Matern32" else 3
    if nan and T >= 3:
        Y[0, T // 2, min(1, p - 1)] = np.nan          # one missing output
        Y[-1, T // 3, :] = np.nan                     # a whole missing row
    X0 = 0.2 * rng.standard_normal((N, L, d)) if x0 else None
    return params, Y, X0


def _model(kernel, p, L, params, path):
    from multioutputihgp_b200 import MOIHGPSequences
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    m.update(params)
    m.set_path(path)
    return m


def _oracle_steps(kernel, p, L, params, Y, x0):
    """The reference's loop: negLogLikelihood(x, y_t) on the state before step t, then step(x, y_t)."""
    from oracle.binding import OracleMOIHGP
    o = OracleMOIHGP(0.1, p, L, kernel, True)
    o.update(params)
    N, T, _ = Y.shape
    d = 2 if kernel == "Matern32" else 3
    steps, xT = np.empty((N, T)), np.empty((N, L, d))
    for n in range(N):
        x = np.zeros((L, d)) if x0 is None else x0[n].copy()
        for t in range(T):
            steps[n, t] = o.negLogLikelihood(x, Y[n, t])
            x = o.step(x, Y[n, t])[0]
        xT[n] = x
    return steps, xT


def _assert_terms(got, ref):
    assert got.shape == ref.shape
    assert np.array_equal(np.isnan(got), np.isnan(ref)), (np.argwhere(np.isnan(got)), np.argwhere(np.isnan(ref)))
    fin = ~np.isnan(ref)
    assert np.isfinite(got[fin]).all()
    assert rel_err(got[fin], ref[fin]) < TOL, rel_err(got[fin], ref[fin])


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("path,kernel,p,L,N,T", PARAMS)
def test_nll_steps_match_oracle_loop(cuda_lib, path, kernel, p, L, N, T):
    """Every term equals the oracle's negLogLikelihood(x_{t-1}, y_t) to the parity bar, with a carried-in state and rows with
    missing outputs (NaN terms at exactly the oracle's positions); xT is the oracle's final state."""
    params, Y, x0 = _setup(kernel, p, L, N, T, 100 * p + T, nan=True, x0=True)
    m = _model(kernel, p, L, params, path)
    r = m.nll_steps(Y, x0=x0)
    ref, xT = _oracle_steps(kernel, p, L, params, Y, x0)
    _assert_terms(r["nll_steps"], ref)
    assert rel_err(r["xT"], xT) < TOL
    if T >= 3:
        assert m.nan_status == 1


@pytest.mark.gpu
@pytest.mark.parametrize("path", BOTH)
@pytest.mark.parametrize("kernel,p,L,N,T", [("Matern52", 16, 8, 6, 700), ("Matern32", 5, 3, 3, 300), ("Matern32", 2, 1, 40, 99)])
def test_nll_steps_sum_to_the_fused_pass(cuda_lib, path, kernel, p, L, N, T):
    """Without missing data the terms sum to the fused pass's nll[n]; the returned nll and xT are the fused pass's own."""
    params, Y, x0 = _setup(kernel, p, L, N, T, 7 * T + N, x0=True)
    m = _model(kernel, p, L, params, path)
    r = m.nll_steps(Y, x0=x0)
    f = m.filter_smoother_nll(Y, x0=x0, smoother_mode=-1, want_states=False)
    assert np.isfinite(r["nll_steps"]).all()
    np.testing.assert_allclose(r["nll_steps"].sum(axis=1), f["nll"], rtol=1e-10, atol=0)
    assert rel_err(r["nll"], f["nll"]) < 1e-14
    assert rel_err(r["xT"], f["xT"]) < 1e-14


@pytest.mark.gpu
def test_chain_and_scan_agree_on_a_long_sequence(cuda_lib):
    kernel, p, L, N, T = "Matern52", 16, 8, 4, 16384
    params, Y, _ = _setup(kernel, p, L, N, T, 3)
    a = _model(kernel, p, L, params, "chain").nll_steps(Y)
    b = _model(kernel, p, L, params, "scan").nll_steps(Y)
    assert rel_err(a["nll_steps"], b["nll_steps"]) < TOL
    assert rel_err(a["nll"], b["nll"]) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("path", BOTH)
def test_device_nll_steps_are_deterministic_and_match_the_host_call(cuda_lib, path):
    import torch
    kernel, p, L, N, T = "Matern52", 16, 8, 9, 1000
    params, Y, x0 = _setup(kernel, p, L, N, T, 11, nan=True, x0=True)
    m = _model(kernel, p, L, params, path)
    dev = torch.device("cuda:0")
    Yd, x0d = torch.from_numpy(Y).to(dev), torch.from_numpy(x0).to(dev)
    outs = []
    for _ in range(2):
        steps, nll, xT = torch.empty((N, T), dtype=torch.float64, device=dev), torch.empty(N, dtype=torch.float64, device=dev), \
            torch.empty((N, L, 3), dtype=torch.float64, device=dev)
        m.nll_steps_device(Yd, steps, x0=x0d, nll=nll, xT=xT)
        torch.cuda.synchronize()
        outs.append((steps.cpu().numpy(), nll.cpu().numpy(), xT.cpu().numpy()))
    for a, b in zip(outs[0], outs[1]):
        assert np.array_equal(a, b, equal_nan=True)
    host = m.nll_steps(Y, x0=x0)
    assert np.array_equal(outs[0][0], host["nll_steps"], equal_nan=True)
    assert np.array_equal(outs[0][2], host["xT"])


@pytest.mark.gpu
@pytest.mark.parametrize("path", BOTH)
def test_device_nll_steps_right_after_update_is_capturable_in_a_cuda_graph(cuda_lib, path):
    """nll_steps_device is asynchronous on the caller's stream: right after update(params) it can be captured into a CUDA
    graph; replays on new data equal the host-buffer call."""
    import torch
    from oracle.gen_golden import make_data, make_params
    kernel, p, L, N, T = "Matern32", 8, 4, 16, 300
    rng = np.random.default_rng(5)
    dev = torch.device("cuda:0")
    from multioutputihgp_b200 import MOIHGPSequences
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    m.set_path(path)
    f64 = dict(dtype=torch.float64, device=dev)
    Y = torch.zeros((N, T, p), **f64)
    steps, nll, xT = torch.zeros((N, T), **f64), torch.zeros(N, **f64), torch.zeros((N, L, 2), **f64)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        m.update(make_params(rng, p, L, kernel))
        m.nll_steps_device(Y, steps, nll=nll, xT=xT)               # warm-up on the capture stream: workspaces
        torch.cuda.synchronize()
        m.update(make_params(rng, p, L, kernel))                   # K-setup queued, nothing waits
        with torch.cuda.graph(g, stream=side):
            m.nll_steps_device(Y, steps, nll=nll, xT=xT)
    for rep in range(2):
        Yh = np.stack([make_data(rng, p, L, T) for _ in range(N)])
        Y.copy_(torch.from_numpy(Yh))
        g.replay()
        torch.cuda.synchronize()
        ref = m.nll_steps(Yh)
        for k, t in (("nll_steps", steps), ("nll", nll), ("xT", xT)):
            assert rel_err(t.cpu().numpy(), ref[k]) < TOL, (rep, k)


@pytest.mark.gpu
def test_nll_steps_refuses_bad_requests(cuda_lib):
    import torch
    kernel, p, L, N, T = "Matern32", 4, 2, 2, 10
    params, Y, _ = _setup(kernel, p, L, N, T, 1)
    m = _model(kernel, p, L, params, "auto")
    Yd = torch.from_numpy(Y).cuda()
    with pytest.raises(RuntimeError, match="nll_steps"):
        m.nll_steps_device(Yd, None)
    lib, out = m._lib, np.empty(N * T)
    for n, t in ((0, T), (N, 0)):
        assert lib.moihgp_cuda_nll_steps(m._h, Y.ctypes.data, n, t, None, out.ctypes.data, None, None) != 0
        assert b"positive" in lib.moihgp_cuda_last_error(m._h)
        assert lib.moihgp_cuda_nll_steps_dev(m._h, Yd.data_ptr(), n, t, None, Yd.data_ptr(), None, None) != 0
        assert b"positive" in lib.moihgp_cuda_last_error(m._h)
    assert lib.moihgp_cuda_nll_steps(m._h, Y.ctypes.data, N, T, None, None, None, None) != 0
    assert b"required" in lib.moihgp_cuda_last_error(m._h)
