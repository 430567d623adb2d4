"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against
  * the golden fixtures generated from the reference itself (tests/golden),
  * the CPU oracle on the same seeded inputs at sizes it finishes in seconds,
  * size-independent properties at larger sizes (chunk invariance, carried state, linearity).
Tolerance: 1e-9 norm-wise relative in fp64 (BASELINE.json north_star), written as conftest.TOL."""
import os

import numpy as np
import pytest

from conftest import TOL, golden_cases, literal_smoother_err, load_golden, rel_err

pytestmark = pytest.mark.gpu


def _models(g):
    from multioutputihgp_b200 import MOIHGPSequences
    m = MOIHGPSequences(float(g["dt"]), int(g["p"]), int(g["L"]), str(g["kernel"]), bool(g["threading"]))
    m.update(g["params"])
    return m


def _close(a, b, tol=TOL):
    return abs(a - b) <= tol * abs(b)


def _assert_cov(P, ref, what):
    """a steady-state covariance against the reference's: same non-finite pattern, finite entries within TOL norm-wise"""
    P, ref = np.asarray(P), np.asarray(ref)
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(P), fin), what
    if fin.any():
        assert rel_err(np.where(fin, P, 0.0), np.where(fin, ref, 0.0)) < TOL, what


def _assert_smoothed(r, ro, mode, what=None):
    """smoothed means against the oracle's at TOL in BOTH modes; the literal mode through conftest.literal_smoother_err
    (whole sequence for latents with rho(G) < 1, the finite tail of the reference for the others)"""
    if mode == 1:
        assert rel_err(r["Xs"], ro["Xs"]) < TOL, what
    else:
        err, steps = literal_smoother_err(r["Xs"], ro["Xs"])
        assert err < TOL and steps >= min(r["Xs"].shape[-3], 100), (what, err, steps)


@pytest.mark.parametrize("path", golden_cases(), ids=lambda p: p.split("/")[-1][:-4])
def test_cuda_matches_reference_golden(cuda_lib, path):
    g = load_golden(path)
    m = _models(g)
    p, L, T = int(g["p"]), int(g["L"]), int(g["T"])
    assert rel_err(m.params, g["params_after_update"]) < 1e-12
    # K-setup: steady-state members of every latent (ihgp.h:243-254)
    for l in range(L):
        c = m.latent_consts(l)
        for k, v in c.items():
            ref = g["c%d_%s" % (l, k)]
            if np.max(np.abs(ref)) > 0:
                assert rel_err(np.asarray(v), np.asarray(ref)) < TOL, (l, k)
            else:
                assert np.max(np.abs(v)) == 0, (l, k)
        # IHGP::backwardSmoother's gain and smoothed covariance (ihgp.h:105-107); P is iterate #100 of the reference's
        # un-converged DLyap map (Q2), up to 2.5e162 for the default Matern-3/2 latent - still a well-defined number
        G, P = m.smoother_consts(l, 0)
        assert rel_err(G, g["sm%d_G" % l]) < TOL
        _assert_cov(P, g["sm%d_P" % l], (l, "P"))
    # objective = RegressionObjective loop (moihgp_regression.h:42-50)
    loss, grad, xT, dxT = m.objective(g["Y"], want_state=True)
    assert _close(loss, g["obj_loss"])
    assert rel_err(grad, g["obj_grad"]) < TOL
    assert rel_err(xT[0], g["obj_xT"]) < TOL and rel_err(dxT[0], g["obj_dxT"]) < TOL
    n2 = max(T // 3, 2)
    loss, grad, xT, dxT = m.objective(g["Y"][:n2], g["x0"], g["dx0"], want_state=True)
    assert _close(loss, g["obj2_loss"]) and rel_err(grad, g["obj2_grad"]) < TOL
    assert rel_err(xT[0], g["obj2_xT"]) < TOL and rel_err(dxT[0], g["obj2_dxT"]) < TOL
    # filter + NLL (+ back-projection)
    r = m.filter_smoother_nll(g["Y"], smoother_mode=1, want_yhat=True)
    assert rel_err(r["X"][0], g["flt_X"]) < TOL
    assert rel_err(r["Yhat"][0], g["flt_Yhat"]) < TOL
    assert _close(r["nll"][0], g["flt_nll"])
    assert rel_err(r["xT"][0], g["flt_X"][-1]) < TOL
    # literal smoother (IHGP::backwardSmoother) on the first 40 filtered states, as the fixture holds them (every latent,
    # the unstable ones included: 6.39^40 = 1e32 is still finite)
    n = min(T, 40)
    for path in ("scan", "chain"):
        if path == "chain" and (p, L) not in ((8, 4), (16, 8)):
            continue
        m.set_path(path)
        r0 = m.filter_smoother_nll(g["Y"][:n], smoother_mode=0)
        for l in range(L):
            assert rel_err(r0["Xs"][0][:, l, :], g["sm%d_Xs" % l]) < TOL, (path, l)


@pytest.mark.parametrize("path", golden_cases(), ids=lambda p: p.split("/")[-1][:-4])
def test_legacy_symbols_match_reference_golden(cuda_lib, path, monkeypatch):
    """gp32_* / gp52_* one observation per call (src/wrapper.cpp), incl. missing data and predict-only."""
    g = load_golden(path)
    if str(g["kernel"]) == "Matern52":
        monkeypatch.setenv("MOIHGP_GP52_MATERN52", "1")
    from multioutputihgp_b200 import MOIHGP
    m = MOIHGP(float(g["dt"]), int(g["p"]), int(g["L"]), kernel=str(g["kernel"]), threading=bool(g["threading"]))
    m.update(g["params"])
    assert rel_err(m.params, g["params_after_update"]) < 1e-12
    for i in range(3):
        xn, yh, dxn = m.step(g["one_x"], g["nan%d_y" % i], g["one_dx"])
        assert rel_err(xn, g["nan%d_xn" % i]) < TOL and rel_err(yh, g["nan%d_yh" % i]) < TOL and rel_err(dxn, g["nan%d_dxn" % i]) < TOL
    xn, yh = m.step(g["one_x"])
    assert rel_err(xn, g["pred_xn"]) < TOL and rel_err(yh, g["pred_yh"]) < TOL
    l1, g1 = m.negLogLikelihood(g["one_x"], g["one_y"], g["one_dx"])
    assert _close(l1, g["one_lik1"]) and rel_err(g1, g["one_grad"]) < TOL
    assert _close(m.negLogLikelihood(g["one_x"], g["one_y"]), g["one_lik2"])
    # the reference's own driver loop through the per-observation symbols (online_learning.py:83-89)
    T = min(int(g["T"]), 25)
    x = np.zeros((int(g["L"]), m.igp_dim))
    dx = np.zeros((int(g["L"]), 3, m.igp_dim))
    X = []
    for y in g["Y"][:T]:
        x, yh, dx = m.step(x, y, dx)
        X.append(x)
    assert rel_err(np.array(X), g["flt_X"][:T]) < TOL


CONFIGS = [
    # kernel, threading, p, L, N, T, seed           (shapes after BASELINE configs 1-5, oracle-sized)
    ("Matern32", True, 2, 1, 1, 63, 1),
    ("Matern32", False, 8, 4, 3, 700, 2),
    ("Matern52", True, 16, 8, 5, 1037, 3),
    ("Matern32", True, 64, 32, 1, 2100, 4),
    ("Matern32", True, 40, 12, 2, 300, 5),           # ragged latent group (12 = 8 + 4)
    ("Matern52", False, 3, 3, 4, 256, 6),            # p == L (no residual), exactly one chunk
    ("Matern52", True, 5, 2, 2, 257, 7),             # one step into the second chunk
]


@pytest.mark.parametrize("kernel,threading,p,L,N,T,seed", CONFIGS)
def test_cuda_matches_oracle(cuda_lib, kernel, threading, p, L, N, T, seed):
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(seed)
    params = make_params(rng, p, L, kernel)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    m = MOIHGPSequences(0.1, p, L, kernel, threading)
    o = OracleMOIHGP(0.1, p, L, kernel, threading)
    m.update(params)
    o.update(params)
    assert rel_err(m.U, o.U) < TOL and rel_err(m.params, o.params) < TOL      # polar factor (host Jacobi, or k_polar when p * L >= 2048)
    d = m.igp_dim
    x0 = 0.2 * rng.standard_normal((N, L, d))
    dx0 = 0.1 * rng.standard_normal((N, L, 3, d))
    for mode in (1, 0):
        r = m.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True)
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True)
        assert rel_err(r["X"], ro["X"]) < TOL
        assert rel_err(r["Yhat"], ro["Yhat"]) < TOL
        assert rel_err(r["nll"], ro["nll"]) < TOL
        assert rel_err(r["xT"], ro["xT"]) < TOL
        _assert_smoothed(r, ro, mode, mode)
        for l in range(L):                       # smoothed covariance of every latent, both modes (ihgp.h:105-107)
            _assert_cov(m.smoother_consts(l, mode)[1], o.smoother_consts(l, mode)[1], (mode, l))
    loss, grad, xT, dxT = m.objective(Y, x0=x0, dx0=dx0, want_state=True)
    lo, go, xo, dxo = o.objective(Y, x0=x0, dx0=dx0)
    assert _close(loss, lo)
    assert rel_err(grad, go) < TOL
    assert rel_err(xT, xo) < TOL and rel_err(dxT, dxo) < TOL


@pytest.mark.parametrize("seed", list(range(100, 124)))
def test_random_shapes_match_oracle(cuda_lib, seed):
    """Differential test on seeded random shapes (odd p, p == L, L not a multiple of 8, T across chunk borders, N across
    warp borders, random carried-in state, both kernels, both threading values): every output of the fused pass and of the
    objective against the CPU oracle, on every kernel path that serves the shape."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(seed)
    kernel = ("Matern32", "Matern52")[int(rng.integers(2))]
    threading = bool(rng.integers(2))
    p = int(rng.choice([1, 2, 3, 4, 5, 7, 8, 9, 12, 16, 17, 24, 32, 33, 48]))
    L = int(rng.integers(1, min(p, 20) + 1))
    if seed % 4 == 0:                                   # every fourth case lands on a many-chains shape
        p, L = [(4, 2), (4, 4), (8, 4), (16, 8), (32, 2), (16, 16)][(seed // 4) % 6]
    N = int(rng.choice([1, 2, 3, 5, 9, 33, 150]))
    T = int(rng.choice([1, 2, 31, 32, 33, 255, 256, 257, 300, 511, 513, 700, 1025]))
    if N * T * L > 400000:
        N = max(1, 400000 // (T * L))
    params = make_params(rng, p, L, kernel)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    m = MOIHGPSequences(0.1, p, L, kernel, threading)
    o = OracleMOIHGP(0.1, p, L, kernel, threading)
    m.update(params)
    o.update(params)
    d = m.igp_dim
    x0 = 0.2 * rng.standard_normal((N, L, d))
    dx0 = 0.1 * rng.standard_normal((N, L, 3, d))
    what = (kernel, threading, p, L, N, T)
    paths = ["scan"]
    try:
        m.set_path("chain")
        m.filter_smoother_nll(Y[:1, :1], smoother_mode=-1, want_states=False)
        paths.append("chain")
    except RuntimeError:
        pass
    mode = int(rng.integers(2))
    ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True)
    for path in paths + ["auto"]:
        m.set_path(path)
        r = m.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True)
        for k in ("X", "Yhat", "nll", "xT"):
            assert rel_err(r[k], ro[k]) < TOL, (what, path, k)
        _assert_smoothed(r, ro, mode, (what, path))
    m.set_path("auto")
    loss, grad, xT, dxT = m.objective(Y, x0=x0, dx0=dx0, want_state=True)
    lo, go, xo, dxo = o.objective(Y, x0=x0, dx0=dx0)
    assert _close(loss, lo), what
    assert rel_err(grad, go) < TOL, what
    assert rel_err(xT, xo) < TOL and rel_err(dxT, dxo) < TOL, what


@pytest.mark.parametrize("path,kernel,p,L,N,T", [("chain", "Matern52", 16, 8, 160, 300), ("scan", "Matern32", 12, 5, 2, 1500)])
def test_device_pass_right_after_update_is_capturable_in_a_cuda_graph(cuda_lib, path, kernel, p, L, N, T):
    """The *_dev entry points are asynchronous on the caller's stream: right after update(params) - K-setup still in flight
    - the fused pass neither waits for the device nor touches the host, so it can be captured into a CUDA graph and replayed
    on new data (ADVICE r1: the many-chains path used to synchronise to fetch log S).  Replays equal the oracle."""
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(N + T)
    dev = torch.device("cuda:0")
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    o = OracleMOIHGP(0.1, p, L, kernel, True)
    m.set_path(path)
    d = m.igp_dim
    f64 = dict(dtype=torch.float64, device=dev)
    Y = torch.zeros((N, T, p), **f64)
    X, Xs, nll = torch.zeros((N, T, L, d), **f64), torch.zeros((N, T, L, d), **f64), torch.zeros(N, **f64)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        m.update(make_params(rng, p, L, kernel))
        m.filter_smoother_nll_device(Y, smoother_mode=1, X=X, Xs=Xs, nll=nll)      # warm-up ON the capture stream: workspaces, attributes
        torch.cuda.synchronize()
        params = make_params(rng, p, L, kernel)
        m.update(params)                                                          # new parameters: K-setup is queued, nothing waits
        o.update(params)
        with torch.cuda.graph(g, stream=side):
            m.filter_smoother_nll_device(Y, smoother_mode=1, X=X, Xs=Xs, nll=nll)
    for rep in range(2):
        Yh = np.stack([make_data(rng, p, L, T) for _ in range(N)])
        Y.copy_(torch.from_numpy(Yh))
        g.replay()
        torch.cuda.synchronize()
        ro = o.filter_smoother_nll(Yh, smoother_mode=1)
        assert rel_err(X.cpu().numpy(), ro["X"]) < TOL and rel_err(Xs.cpu().numpy(), ro["Xs"]) < TOL, rep
        assert rel_err(nll.cpu().numpy(), ro["nll"]) < TOL, rep


def test_one_device_model_behind_both_python_interfaces(cuda_lib):
    """MOIHGPSequences.adopt(pywrapper.MOIHGP): the whole-sequence interface on the SAME handle as the per-observation one
    (INTEGRATION.md section 1) - an update through either object is seen by both, and the per-observation step equals the
    first step of the whole-sequence pass."""
    from multioutputihgp_b200 import MOIHGPSequences
    from multioutputihgp_b200.pywrapper import MOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(11)
    p, L, T = 8, 4, 40
    legacy = MOIHGP(0.1, p, L, kernel="Matern32", threading=False)
    seq = MOIHGPSequences.adopt(legacy)
    assert (seq.num_output, seq.num_latent, seq.igp_dim, seq.num_param) == (p, L, 2, legacy.num_param)
    params = make_params(rng, p, L, "Matern32")
    seq.update(params)                                         # through the whole-sequence object ...
    assert np.array_equal(legacy.params, seq.params)           # ... seen by the per-observation one (polar factor taken)
    Y = make_data(rng, p, L, T)
    r = seq.filter_smoother_nll(Y[None], smoother_mode=-1, want_yhat=True)
    x = np.zeros((L, 2))
    for t in range(3):
        x, yhat = legacy.step(x, y=Y[t])[:2]
        assert rel_err(x, r["X"][0, t]) < 1e-12 and rel_err(yhat, r["Yhat"][0, t]) < 1e-12, t
    params2 = make_params(rng, p, L, "Matern32")
    legacy.update(params2)                                     # ... and the other way round
    assert np.array_equal(legacy.params, seq.params)
    del seq                                                    # the adopted handle is not destroyed with the adopter
    assert legacy.params.shape == (legacy.num_param,)


CHAIN_CONFIGS = [
    # kernel, p, L, N, T, seed      shapes instantiated for the many-chains kernels (chain.cu); ragged N and T on purpose
    ("Matern52", 16, 8, 9, 1037, 21),
    ("Matern32", 16, 8, 4, 64, 22),
    ("Matern32", 8, 4, 11, 333, 23),
    ("Matern52", 8, 4, 1, 7, 24),
    ("Matern52", 16, 8, 6, 1, 25),
    ("Matern32", 32, 16, 3, 150, 26),            # further instantiated shapes (full warp only)
    ("Matern52", 32, 8, 5, 97, 27),
    ("Matern52", 32, 4, 9, 65, 28),
    ("Matern32", 16, 16, 2, 200, 29),
    ("Matern52", 16, 4, 10, 130, 30),
    ("Matern32", 16, 2, 17, 60, 31),
    ("Matern52", 8, 8, 5, 120, 32),
    ("Matern32", 8, 2, 33, 50, 33),
    ("Matern52", 4, 2, 17, 90, 36),              # round 2: four-output shapes and (32, 2)
    ("Matern32", 4, 4, 9, 130, 37),
    ("Matern32", 32, 2, 18, 70, 41),
    ("Matern32", 6, 2, 19, 75, 45),              # round 2: p between the instantiated widths (padded variant of k_filter_chain)
    ("Matern52", 6, 4, 9, 130, 46),
    ("Matern52", 10, 4, 11, 99, 47),
    ("Matern32", 12, 8, 6, 140, 48),
    ("Matern52", 14, 2, 33, 40, 49),
    ("Matern32", 20, 16, 3, 170, 50),
    ("Matern52", 30, 4, 10, 61, 51),
    ("Matern32", 26, 8, 5, 88, 52),
    ("Matern52", 3, 2, 21, 66, 53),              # odd p: rows of Y only 8-byte aligned (8-byte copies into the tile)
    ("Matern32", 5, 4, 9, 131, 54),
    ("Matern52", 9, 8, 5, 77, 55),
    ("Matern32", 13, 4, 10, 64, 56),
    ("Matern52", 27, 8, 6, 90, 57),
    ("Matern32", 31, 2, 17, 35, 58),
    ("Matern32", 4, 1, 40, 77, 59),              # one latent (Matern-3/2): rounds of one step, 32 sequences per warp
    ("Matern32", 2, 1, 70, 63, 60),              # the shape of the reference's own examples (p = 2, L = 1)
    ("Matern32", 7, 1, 33, 130, 61),
    ("Matern32", 16, 1, 37, 41, 62),
    ("Matern32", 29, 1, 65, 33, 63),
    ("Matern32", 8, 3, 13, 91, 64),              # L between the instantiated widths: idle lanes, X in the caller's [t][L][d] layout
    ("Matern32", 5, 3, 21, 64, 65),
    ("Matern32", 12, 5, 7, 140, 66),
    ("Matern32", 6, 6, 9, 77, 67),
    ("Matern32", 16, 7, 5, 120, 68),
    ("Matern32", 15, 11, 5, 66, 69),
    ("Matern32", 24, 12, 3, 50, 70),
    ("Matern52", 12, 6, 7, 85, 71),              # ... Matern-5/2: even L only (L * d even)
    ("Matern52", 16, 10, 5, 70, 72),
    ("Matern52", 9, 6, 9, 33, 73),
    ("Matern52", 14, 14, 3, 90, 74),
    ("Matern52", 8, 3, 13, 64, 75),              # ... odd L with Matern-5/2: served when T is even (16-byte aligned runs of X)
    ("Matern52", 12, 5, 7, 140, 76),
    ("Matern52", 16, 7, 5, 90, 77),
    ("Matern52", 15, 9, 5, 66, 78),
]


def test_many_chains_path_refuses_runs_it_cannot_align(cuda_lib):
    """Odd L with Matern-5/2 (L * d odd) and an odd T: the runs of X would not be 16-byte aligned - the many-chains path says so
    (the automatic choice takes the chunked-scan path, which serves the shape)."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(5)
    p, L, N, T = 8, 3, 200, 65
    m = MOIHGPSequences(0.1, p, L, "Matern52", True)
    params = make_params(rng, p, L, "Matern52")
    m.update(params)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    m.set_path("chain")
    with pytest.raises(RuntimeError):
        m.filter_smoother_nll(Y, smoother_mode=1)
    m.set_path("auto")
    r = m.filter_smoother_nll(Y, smoother_mode=1)
    o = OracleMOIHGP(0.1, p, L, "Matern52", True)
    o.update(params)
    ro = o.filter_smoother_nll(Y, smoother_mode=1)
    assert rel_err(r["X"], ro["X"]) < TOL and rel_err(r["Xs"], ro["Xs"]) < TOL and rel_err(r["nll"], ro["nll"]) < TOL


@pytest.mark.parametrize("kernel,p,L,N,T,seed", CHAIN_CONFIGS)
def test_many_chains_path_matches_oracle_and_scan_path(cuda_lib, kernel, p, L, N, T, seed):
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(seed)
    params = make_params(rng, p, L, kernel)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    o = OracleMOIHGP(0.1, p, L, kernel, True)
    m.update(params)
    o.update(params)
    x0 = 0.2 * rng.standard_normal((N, L, m.igp_dim))
    for mode in (1, 0):
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True)
        res = {}
        for path in ("chain", "scan"):
            m.set_path(path)
            res[path] = r = m.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True)
            assert rel_err(r["X"], ro["X"]) < TOL, path
            assert rel_err(r["Yhat"], ro["Yhat"]) < TOL, path
            assert rel_err(r["nll"], ro["nll"]) < TOL, path
            assert rel_err(r["xT"], ro["xT"]) < TOL, path
            _assert_smoothed(r, ro, mode, (path, mode))
        assert rel_err(res["chain"]["X"], res["scan"]["X"]) < 1e-12
    # smoother-only request (no filtered states wanted) and NLL-only request
    m.set_path("chain")
    r = m.filter_smoother_nll(Y, x0=x0, smoother_mode=-1, want_states=False)
    assert rel_err(r["nll"], ro["nll"]) < TOL


def test_many_chains_path_full_T_properties(cuda_lib):
    """BASELINE config 3 at full T = 16384 (fewer sequences): chunk/carry invariance and linearity on the many-chains path."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_params
    rng = np.random.default_rng(31)
    p, L, N, T, cut = 16, 8, 12, 16384, 5003
    m = MOIHGPSequences(0.1, p, L, "Matern52", True)
    m.update(make_params(rng, p, L, "Matern52"))
    m.set_path("chain")
    Y1, Y2 = rng.standard_normal((N, T, p)), rng.standard_normal((N, T, p))
    full = m.filter_smoother_nll(Y1, smoother_mode=1)
    a = m.filter_smoother_nll(Y1[:, :cut], smoother_mode=-1)
    b = m.filter_smoother_nll(Y1[:, cut:], x0=a["xT"], smoother_mode=-1)
    assert rel_err(np.concatenate([a["X"], b["X"]], axis=1), full["X"]) < TOL
    assert rel_err(a["nll"] + b["nll"], full["nll"]) < TOL
    r2 = m.filter_smoother_nll(Y2, smoother_mode=1)
    r3 = m.filter_smoother_nll(0.7 * Y1 - 1.9 * Y2, smoother_mode=1)
    for k in ("X", "Xs"):
        assert rel_err(r3[k], 0.7 * full[k] - 1.9 * r2[k]) < 1e-11
    m.set_path("scan")
    rs = m.filter_smoother_nll(Y1, smoother_mode=1)
    for k in ("X", "Xs", "nll"):
        assert rel_err(rs[k], full[k]) < 1e-11, k


def _smoother_cases():
    import glob
    from conftest import ROOT
    return sorted(glob.glob(os.path.join(ROOT, "tests", "golden_smoother", "*.npz")))


@pytest.mark.parametrize("path", _smoother_cases(), ids=lambda p: p.split("/")[-1][:-4])
def test_literal_smoother_over_whole_sequences_matches_reference(cuda_lib, path):
    """IHGP::backwardSmoother (ihgp.h:103-114) as the reference itself ran it over WHOLE sequences (tests/golden_smoother,
    hyper-parameters with rho(G) < 1): smoothed means of every latent, smoothed covariance P and gain G at 1e-9, on both
    kernel paths."""
    g = load_golden(path)
    p, L = int(g["p"]), int(g["L"])
    from multioutputihgp_b200 import MOIHGPSequences
    m = MOIHGPSequences(float(g["dt"]), p, L, str(g["kernel"]), False)
    m.update(g["params"])
    for l in range(L):
        G, P = m.smoother_consts(l, 0)
        assert rel_err(G, g["sm_G"][l]) < TOL and rel_err(P, g["sm_P"][l]) < TOL, l
    for kpath in ("scan", "chain"):
        if kpath == "chain" and (p, L) not in ((8, 4), (16, 8)):
            continue
        m.set_path(kpath)
        r = m.filter_smoother_nll(g["Y"], smoother_mode=0)
        assert rel_err(r["X"][0], g["flt_X"]) < TOL and _close(r["nll"][0], g["flt_nll"]), kpath
        for l in range(L):
            assert rel_err(r["Xs"][0][:, l], g["sm_Xs"][:, l]) < TOL, (kpath, l)


def _oracle_pass(kernel, threading, p, L, params, Y, mode, x0=None):
    from oracle.binding import OracleMOIHGP
    o = OracleMOIHGP(0.1, p, L, kernel, threading)
    o.update(params)
    return o, o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, nthreads=8)


def test_config3_full_length_matches_oracle(cuda_lib):
    """BASELINE configs[2] at its full length (p = 16, L = 8, Matern-5/2, T = 16384; 8 of the 4096 sequences) on the
    many-chains path that the benchmark times: filtered states, smoothed states in BOTH modes (all four table entries have
    rho(G) < 1 in the literal mode too) and NLL against the oracle at 1e-9; the chunked-scan path on the same input."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(303)
    p, L, N, T = 16, 8, 8, 16384
    params = make_params(rng, p, L, "Matern52")
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    m = MOIHGPSequences(0.1, p, L, "Matern52", True)
    m.update(params)
    for mode in (1, 0):
        o, ro = _oracle_pass("Matern52", True, p, L, params, Y, mode)
        for kpath in ("chain", "scan"):
            m.set_path(kpath)
            r = m.filter_smoother_nll(Y, smoother_mode=mode)
            assert rel_err(r["X"], ro["X"]) < TOL, (kpath, mode)
            assert rel_err(r["Xs"], ro["Xs"]) < TOL, (kpath, mode)
            assert rel_err(r["nll"], ro["nll"]) < TOL, (kpath, mode)
            assert rel_err(r["xT"], ro["xT"]) < TOL, (kpath, mode)
            for l in range(L):
                assert rel_err(r["Xs"][:, :, l], ro["Xs"][:, :, l]) < TOL, (kpath, mode, l)


def test_config4_shape_long_sequence_matches_oracle(cuda_lib):
    """BASELINE configs[3] shape (p = 64, L = 32, Matern-3/2, one sequence) at T = 100 000 = 391 chunks on the chunked-scan
    path: filtered / smoothed states and NLL against the oracle at 1e-9 - RTS mode on the benchmark's table, literal mode on
    the literal-stable table (whole sequence, every latent) - and the objective at T = 20 000."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import LITERAL_STABLE, make_data, make_params
    rng = np.random.default_rng(404)
    p, L, T = 64, 32, 100000
    Y = make_data(rng, p, L, T)[None]
    m = MOIHGPSequences(0.1, p, L, "Matern32", True)
    for mode, table in ((1, None), (0, LITERAL_STABLE), (0, None)):
        params = make_params(rng, p, L, "Matern32", table)
        m.update(params)
        o, ro = _oracle_pass("Matern32", True, p, L, params, Y, mode)
        r = m.filter_smoother_nll(Y, smoother_mode=mode)
        assert rel_err(r["X"], ro["X"]) < TOL and rel_err(r["nll"], ro["nll"]) < TOL and rel_err(r["xT"], ro["xT"]) < TOL, mode
        if table is not None or mode == 1:
            assert rel_err(r["Xs"], ro["Xs"]) < TOL, mode
            for l in range(L):
                assert rel_err(r["Xs"][:, :, l], ro["Xs"][:, :, l]) < TOL, (mode, l)
        else:   # default table, literal mode: latents 0, 4, 8 ... have rho(G) = 6.39 (SURVEY Q3) - finite tail only for those
            _assert_smoothed(r, ro, 0, "default table")
    Yo = Y[:, :20000]
    loss, grad, xT, dxT = m.objective(Yo, want_state=True)
    lo, go, xo, dxo = o.objective(Yo)
    assert _close(loss, lo) and rel_err(grad, go) < TOL and rel_err(xT, xo) < TOL and rel_err(dxT, dxo) < TOL


@pytest.mark.parametrize("threading", [True, False])
def test_objective_at_config5_shape_matches_oracle(cuda_lib, threading):
    """BASELINE configs[4] shape (p = 256, L = 64, Matern-3/2): loss, all 16 641 gradient entries and the final state of
    MOIHGP::negLogLikelihood(x, y, dx, grad) summed over T = 3001 steps (moihgp.h:460-611, moihgp_regression.h:42-50), with a
    carried-in state, against the oracle at 1e-9 - with and without the per-latent loss terms (`threading`, Q5)."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(505)
    p, L, T = 256, 64, 3001
    params = make_params(rng, p, L, "Matern32")
    Y = make_data(rng, p, L, T)[None]
    m = MOIHGPSequences(0.1, p, L, "Matern32", threading)
    o = OracleMOIHGP(0.1, p, L, "Matern32", threading)
    m.update(params)
    o.update(params)
    assert rel_err(m.U, o.U) < TOL
    d = m.igp_dim
    x0 = 0.2 * rng.standard_normal((1, L, d))
    dx0 = 0.1 * rng.standard_normal((1, L, 3, d))
    for a, b in ((None, None), (x0, dx0)):
        loss, grad, xT, dxT = m.objective(Y, x0=a, dx0=b, want_state=True)
        lo, go, xo, dxo = o.objective(Y, x0=a, dx0=b)
        assert _close(loss, lo)
        assert rel_err(grad, go) < TOL
        pL = p * L          # every block of the gradient on its own scale: dU, dS, dsigma, per-latent hyper-parameters
        for sl in (slice(0, pL), slice(pL, pL + L), slice(pL + L, pL + L + 1), slice(pL + L + 1, None)):
            assert rel_err(grad[sl], go[sl]) < TOL, sl
        assert rel_err(xT, xo) < TOL and rel_err(dxT, dxo) < TOL


def test_chunk_and_carry_invariance(cuda_lib):
    """Splitting a sequence in two calls with the carried state equals one call (filter state, NLL, objective)."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(9)
    p, L, T, cut = 16, 8, 5000, 1777
    params = make_params(rng, p, L, "Matern52")
    Y = make_data(rng, p, L, T)[None]
    m = MOIHGPSequences(0.1, p, L, "Matern52", True)
    m.update(params)
    full = m.filter_smoother_nll(Y, smoother_mode=-1)
    a = m.filter_smoother_nll(Y[:, :cut], smoother_mode=-1)
    b = m.filter_smoother_nll(Y[:, cut:], x0=a["xT"], smoother_mode=-1)
    assert rel_err(np.concatenate([a["X"], b["X"]], axis=1), full["X"]) < TOL
    assert _close(a["nll"][0] + b["nll"][0], full["nll"][0])
    lf, gf = m.objective(Y)
    la, ga, xa, dxa = m.objective(Y[:, :cut], want_state=True)
    lb, gb = m.objective(Y[:, cut:], x0=xa, dx0=dxa)
    assert _close(la + lb, lf) and rel_err(ga + gb, gf) < TOL


def test_filter_is_linear_in_the_observations(cuda_lib):
    """x is an LTI-affine function of y with x0 = 0: X(a Y1 + b Y2) = a X(Y1) + b X(Y2); same for the smoother."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_params
    rng = np.random.default_rng(10)
    p, L, N, T = 8, 4, 6, 3000
    m = MOIHGPSequences(0.1, p, L, "Matern32", True)
    m.update(make_params(rng, p, L, "Matern32"))
    Y1, Y2 = rng.standard_normal((N, T, p)), rng.standard_normal((N, T, p))
    r1, r2 = m.filter_smoother_nll(Y1, smoother_mode=1), m.filter_smoother_nll(Y2, smoother_mode=1)
    r3 = m.filter_smoother_nll(0.7 * Y1 - 1.9 * Y2, smoother_mode=1)
    for k in ("X", "Xs"):
        assert rel_err(r3[k], 0.7 * r1[k] - 1.9 * r2[k]) < 1e-11


def test_device_resident_entry_points(cuda_lib):
    """torch CUDA tensors through the *_dev symbols give the same results as host buffers."""
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(12)
    p, L, N, T = 16, 8, 4, 1500
    m = MOIHGPSequences(0.1, p, L, "Matern52", True)
    m.update(make_params(rng, p, L, "Matern52"))
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    host = m.filter_smoother_nll(Y)                  # default smoother mode: the reference's literal recursion
    dev = torch.device("cuda:0")
    Yd = torch.from_numpy(Y).to(dev)
    X = torch.empty((N, T, L, 3), dtype=torch.float64, device=dev)
    Xs = torch.empty_like(X)
    nll = torch.empty(N, dtype=torch.float64, device=dev)
    m.filter_smoother_nll_device(Yd, X=X, Xs=Xs, nll=nll)
    torch.cuda.synchronize()
    assert rel_err(X.cpu().numpy(), host["X"]) == 0.0
    assert rel_err(Xs.cpu().numpy(), host["Xs"]) == 0.0
    assert rel_err(nll.cpu().numpy(), host["nll"]) == 0.0
    loss = torch.zeros(1, dtype=torch.float64, device=dev)
    grad = torch.zeros(m.num_param, dtype=torch.float64, device=dev)
    m.objective_device(Yd, loss, grad)
    torch.cuda.synchronize()
    lh, gh = m.objective(Y)
    assert float(loss.item()) == lh and rel_err(grad.cpu().numpy(), gh) == 0.0


def test_online_learner_runs_like_the_reference_example(cuda_lib):
    """example.py / online_learning.py protocol: 8 outputs, 4 latents, window 2 (BASELINE config 2 shape)."""
    from multioutputihgp_b200 import MOIHGPOnlineLearning
    rng = np.random.default_rng(5)
    gp = MOIHGPOnlineLearning(0.1, 8, 4, gamma=0.9, windowsize=2, threading=False)
    t = np.arange(12) * 0.1
    data = np.stack([np.sin((1 + i % 3) * t) for i in range(8)], axis=1) + 0.05 * rng.standard_normal((12, 8))
    for y in data:
        yhat = gp.step(y)
        assert yhat.shape == (8,) and np.all(np.isfinite(yhat))
    assert np.all(np.isfinite(gp.params)) and gp.covariance.shape == (8, 8)


NAN_CONFIGS = [
    # kernel, p, L, N, T, path
    ("Matern52", 16, 8, 6, 300, "chain"),
    ("Matern52", 16, 8, 6, 300, "scan"),
    ("Matern32", 8, 4, 9, 120, "chain"),
    ("Matern52", 12, 4, 9, 90, "chain"),      # padded variant of the many-chains filter
    ("Matern32", 6, 2, 19, 70, "chain"),
    ("Matern52", 11, 4, 9, 85, "chain"),      # ... with odd p
    ("Matern32", 3, 1, 40, 60, "chain"),      # one latent
    ("Matern32", 10, 3, 11, 75, "chain"),     # padded latents
    ("Matern52", 12, 6, 7, 66, "chain"),
    ("Matern52", 10, 5, 9, 70, "chain"),      # odd L * d, even T
    ("Matern32", 5, 3, 3, 280, "scan"),       # odd p: scalar projection kernel
    ("Matern32", 64, 32, 1, 600, "scan"),     # tensor-pipe projection kernel, large L
]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L,N,T,path", NAN_CONFIGS)
def test_missing_observations_whole_sequence(cuda_lib, kernel, p, L, N, T, path):
    """NaN = missing output (moihgp.h:150-178): least-squares projection on the observed outputs, per observation.
    Filtered / smoothed states and Yhat match the oracle; the NLL of a sequence with missing data is NaN, as the
    reference's is (moihgp.h:651 uses the full y), and untouched sequences keep their NLL."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(1000 + p + T)
    params = make_params(rng, p, L, kernel)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    Y[0, 3, 1] = np.nan                       # a single missing output
    Y[0, 10, :] = np.nan                      # everything missing: Ty = 0 (LDLT of the zero matrix)
    Y[0, 11, : max(0, p - L - 2)] = np.nan    # L + 2 outputs left (with fewer than L observed outputs U0'U0 is singular and the
                                              # reference's LDLT result is rounding noise: no defined answer to compare with)
    Y[0, T - 1, 0] = np.nan                   # last step
    miss = rng.random((T, p)) < 0.15          # scattered, but never fewer than L + 2 observed outputs in a row
    miss[(~miss).sum(axis=1) < L + 2] = False
    miss[:20] = False                         # (N = 1: keep the hand-placed rows of sequence 0 as they are)
    miss[T - 1] = False
    Y[N - 1][miss] = np.nan
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    o = OracleMOIHGP(0.1, p, L, kernel, True)
    m.update(params)
    o.update(params)
    m.set_path(path)
    r = m.filter_smoother_nll(Y, smoother_mode=1, want_yhat=True)
    ro = o.filter_smoother_nll(Y, smoother_mode=1, want_yhat=True)
    for k in ("X", "Xs", "Yhat", "xT"):
        assert np.all(np.isfinite(r[k])), k
        assert rel_err(r[k], ro[k]) < TOL, k
    assert np.array_equal(np.isnan(r["nll"]), np.isnan(ro["nll"]))
    ok = ~np.isnan(ro["nll"])
    assert np.isnan(r["nll"][0]) and (N == 1 or ok.any() or N == 2)
    if ok.any():
        assert rel_err(r["nll"][ok], ro["nll"][ok]) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["online_py_p8L4_w2", "online_py_p4L2_w1"])
def test_online_learner_follows_the_reference_python_driver(cuda_lib, name):
    """BASELINE config 2 protocol (streaming update, online_learning.py:53-105): the golden trajectory was produced by the
    reference's OWN pywrapper.py + online_learning.py on the reference's C ABI (oracle/gen_golden_online.py); here the same
    stream goes through this package's mirror on the GPU.  L-BFGS-B (5 iterations, 3 line-search steps per sample) feeds
    rounding differences back into the parameters, hence the looser tolerance on the trajectory."""
    import os
    from conftest import ROOT
    from multioutputihgp_b200 import MOIHGPOnlineLearning
    z = np.load(os.path.join(ROOT, "tests", "golden_online", name + ".npz"))
    gp = MOIHGPOnlineLearning(float(z["dt"]), int(z["p"]), int(z["L"]), gamma=float(z["gamma"]), windowsize=int(z["window"]), threading=False)
    gp._update(z["params0"])
    worst_y = worst_p = 0.0
    for y, yh_ref, p_ref in zip(z["data"], z["yhat"], z["params"]):
        yh = gp.step(y.copy())
        worst_y = max(worst_y, rel_err(yh, yh_ref))
        worst_p = max(worst_p, rel_err(gp.params, p_ref))
    print(name, "worst rel. err yhat %.2e params %.2e" % (worst_y, worst_p))
    assert worst_y < 1e-9 and worst_p < 1e-9


@pytest.mark.gpu
def test_time_sharded_objective_two_gpus(cuda_lib):
    """SURVEY 8(e): one long sequence split in time over two GPUs (carry all-gather + NCCL all-reduce) equals the
    single-GPU evaluation.  Needs two devices; skipped on a one-GPU box (the gloo twin runs in the CPU suite)."""
    import subprocess
    import sys
    import torch
    from conftest import ROOT
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, TS_T="60000", TS_P="16", TS_L="8")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29541", os.path.join(ROOT, "scripts", "gpu_time_shard.py")], capture_output=True, text=True, env=env, timeout=600)
    print(r.stdout[-2000:], r.stderr[-2000:])
    assert r.returncode == 0 and "time-sharded objective" in r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L,N,cuts", [("Matern32", 8, 4, 1, (0, 512, 1280, 1700)), ("Matern52", 16, 8, 2, (0, 256, 512, 1024)),
                                               ("Matern32", 64, 32, 1, (0, 2048, 4096, 6000))])
def test_time_sharded_filter_smoother_device_side_exchange(cuda_lib, kernel, p, L, N, cuts):
    """The host-round-trip-free protocol of the time-sharded filter + smoother pass on ONE device (one handle per block, as on
    its own GPU): fsn_block_async leaves the phase outputs in device memory, fsn_carry_device (binary powering on the
    device) turns the stacked outputs into every block's x_in / u_after and b_end.  The carries equal the host algebra
    (parallel.forward_carry_in / backward_carry_in); X, Xs, NLL equal the oracle's pass over the whole sequence."""
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    from multioutputihgp_b200.parallel import backward_carry_in, forward_carry_in
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(sum(cuts) + 7)
    params = make_params(rng, p, L, kernel)
    T, G = cuts[-1], len(cuts) - 1
    lengths = [cuts[g + 1] - cuts[g] for g in range(G)]
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    dev = torch.device("cuda:0")
    f64 = dict(dtype=torch.float64, device=dev)
    models = []
    for g in range(G):
        m = MOIHGPSequences(0.1, p, L, kernel, True)
        m.update(params)
        models.append(m)
    d = models[0].igp_dim
    x0 = 0.3 * rng.standard_normal((N, L, d))
    x0d = torch.from_numpy(x0).to(dev)
    Yd = [torch.from_numpy(np.ascontiguousarray(Y[:, cuts[g]:cuts[g + 1]])).to(dev) for g in range(G)]
    ro = OracleMOIHGP(0.1, p, L, kernel, True)
    ro.update(params)
    for mode in (1, 0):
        g1 = torch.zeros((G, N, L, d + 1), **f64)
        g2 = torch.zeros((G, N, L, d), **f64)
        xin = torch.zeros((G, N, L, d), **f64)
        uaf = torch.zeros((G, N, L), **f64)
        bend = torch.zeros((G, N, L, d), **f64)
        for g in range(G):
            models[g].fsn_block_async(1, Yd[g], g == G - 1, mode, out=g1[g])
        for g in range(G):
            models[g].fsn_carry_device(0, g1, lengths, g, xin[g], mode, x0=x0d, u_after=uaf[g])
            models[g].fsn_block_async(2, Yd[g], g == G - 1, mode, x0=xin[g], u_after=None if g == G - 1 else uaf[g], out=g2[g])
        X = [torch.zeros((N, lengths[g], L, d), **f64) for g in range(G)]
        Xs = [torch.zeros_like(X[g]) for g in range(G)]
        nll = torch.zeros((G, N), **f64)
        for g in range(G):
            models[g].fsn_carry_device(1, g2, lengths, g, bend[g], mode)
            models[g].fsn_block_async(3, Yd[g], g == G - 1, mode, x0=xin[g], u_after=None if g == G - 1 else uaf[g],
                                      b_end=None if g == G - 1 else bend[g], X=X[g], Xs=Xs[g], nll=nll[g])
        torch.cuda.synchronize()
        h1, h2 = g1.cpu().numpy(), g2.cpu().numpy()
        for g in range(G):
            xh = forward_carry_in(models[0].block_transition, lengths, list(h1[..., :d]), x0, g)
            assert rel_err(xin[g].cpu().numpy(), xh) < 1e-12, (mode, g)
            if g < G - 1:
                assert np.array_equal(uaf[g].cpu().numpy(), h1[g + 1][..., d]), (mode, g)
                bh = backward_carry_in(lambda n_: models[0].smoother_power(n_, mode), lengths, list(h2), g)
                bd = bend[g].cpu().numpy()                   # literal mode: a latent with rho(G) > 1 overflows on both sides (Q3)
                assert np.array_equal(np.isfinite(bd), np.isfinite(bh)), (mode, g)
                for l in range(L):
                    if np.isfinite(bh[:, l]).all() and np.max(np.abs(bh[:, l])) < 1e100:
                        assert rel_err(bd[:, l], bh[:, l]) < 1e-12, (mode, g, l)
        r = ro.filter_smoother_nll(Y, x0=x0, smoother_mode=mode)
        Xc = np.concatenate([x.cpu().numpy() for x in X], axis=1)
        Xsc = np.concatenate([x.cpu().numpy() for x in Xs], axis=1)
        assert rel_err(Xc, r["X"]) < TOL and rel_err(nll.sum(0).cpu().numpy(), r["nll"]) < TOL, mode
        _assert_smoothed({"Xs": Xsc}, r, mode, ("oracle", mode))


@pytest.mark.gpu
@pytest.mark.parametrize("script,needle,env", [("gpu_time_shard.py", "time-sharded objective", {"TS_T": "60000", "TS_P": "16", "TS_L": "8"}),
                                               ("gpu_time_shard_fsn.py", "block borders agree", {"TS_T": "70001", "TS_P": "16", "TS_L": "8"})])
def test_time_sharded_passes_two_ranks_on_one_gpu(cuda_lib, script, needle, env):
    """The two time-sharded protocols end to end with TWO ranks on whatever GPUs are visible (gloo exchange, ranks share a
    device on a one-GPU box): blocks per rank, device-side carry kernels, all-gathers, all-reduce - against the whole-sequence
    pass.  The NCCL twins (test_time_sharded_*_two_gpus) need two devices."""
    import subprocess
    import sys
    from conftest import ROOT
    e = dict(os.environ, TS_BACKEND="gloo", **env)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29547", os.path.join(ROOT, "scripts", script)], capture_output=True, text=True, env=e, timeout=600)
    print(r.stdout[-2000:], r.stderr[-2000:])
    assert r.returncode == 0 and needle in r.stdout


@pytest.mark.gpu
def test_time_sharded_filter_smoother_two_gpus(cuda_lib):
    """SURVEY 8(e): the fused filter + smoother + NLL pass of one long sequence split in time over two GPUs (forward and
    backward carry all-gathers + NCCL all-reduce of the NLL) equals the single-GPU pass.  Needs two devices."""
    import subprocess
    import sys
    import torch
    from conftest import ROOT
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, TS_T="70001", TS_P="16", TS_L="8")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29543", os.path.join(ROOT, "scripts", "gpu_time_shard_fsn.py")], capture_output=True, text=True, env=env, timeout=600)
    print(r.stdout[-2000:], r.stderr[-2000:])
    assert r.returncode == 0 and "time-sharded filter+smoother+NLL" in r.stdout and "block borders agree" in r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("p,L", [(256, 64), (64, 32), (96, 33), (200, 11)])
def test_update_polar_factor_on_device(cuda_lib, p, L):
    """MOIHGP::update (moihgp.h:431-447): U = polar factor of the raw block; large blocks go through k_polar.  Checked against
    the SVD-based polar factor; update(getParams()) leaves U unchanged (the polar factor of an orthonormal matrix is itself)."""
    from multioutputihgp_b200 import MOIHGPSequences
    rng = np.random.default_rng(p + L)
    m = MOIHGPSequences(0.1, p, L, "Matern32", True)
    raw = rng.standard_normal((p, L)) / np.sqrt(L) + np.eye(p, L)
    params = np.concatenate([raw.ravel(), np.ones(L), [1e-2], np.tile([1.0, 1.0, 0.1], L)])
    m.update(params)
    u, _, vt = np.linalg.svd(raw, full_matrices=False)
    assert rel_err(m.U, u @ vt) < 1e-12
    assert np.max(np.abs(m.U.T @ m.U - np.eye(L))) < 1e-13
    U1 = m.U.copy()
    m.update(m.params)
    assert rel_err(m.U, U1) < 1e-13


@pytest.mark.gpu
def test_bound_data_objective_equals_host_buffer_objective(cuda_lib):
    """moihgp_cuda_bind_data + moihgp_cuda_objective_bound (data resident across the optimiser's evaluations) give the
    same numbers as passing the observations with every call, also after update(params)."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(41)
    p, L, N, T = 16, 8, 3, 900
    m = MOIHGPSequences(0.1, p, L, "Matern52", True)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    m.bind(Y)
    for k in range(2):
        m.update(make_params(rng, p, L, "Matern52"))
        la, ga = m.objective(Y)
        lb, gb = m.objective_bound()
        assert la == lb and np.array_equal(ga, gb)
    m.bind(None)
    with pytest.raises(RuntimeError):
        m.objective_bound()


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["objective", "objective_bound"])
def test_host_objective_refuses_more_than_2_22_missing_rows(cuda_lib, entry):
    """Both host-buffer objective entry points refuse a call with more than 2^22 rows with missing outputs (the rows beyond
    that are not re-projected), whether the observations come with the call or were bound to the device before."""
    from multioutputihgp_b200 import MOIHGPSequences
    p, L, T = 2, 1, (1 << 22) + 64
    m = MOIHGPSequences(0.1, p, L, "Matern32", True)
    Y = np.full((1, T, p), np.nan)
    if entry == "objective_bound":
        m.bind(Y)
    with pytest.raises(RuntimeError, match=r"more than 2\^22 observations with missing \(NaN\) outputs"):
        m.objective(Y) if entry == "objective" else m.objective_bound()
    assert m.nan_status == 2


@pytest.mark.gpu
@pytest.mark.parametrize("path,kernel,p,L,N,T", [("chain", "Matern52", 16, 8, 5, 203), ("chain", "Matern32", 8, 4, 9, 37),
                                                 ("chain", "Matern52", 4, 2, 37, 45), ("chain", "Matern52", 10, 4, 11, 57), ("chain", "Matern32", 22, 8, 5, 43), ("chain", "Matern52", 7, 2, 19, 41), ("chain", "Matern32", 2, 1, 45, 50), ("chain", "Matern32", 9, 5, 9, 47), ("chain", "Matern52", 12, 6, 7, 39), ("chain", "Matern52", 9, 3, 13, 46), ("chain", "Matern32", 32, 2, 19, 70), ("chain", "Matern52", 4, 4, 9, 66),
                                                 ("scan", "Matern52", 16, 8, 3, 515), ("scan", "Matern32", 5, 3, 2, 257)])
def test_outputs_stay_inside_their_buffers(cuda_lib, path, kernel, p, L, N, T):
    """Ragged N / T through the device entry points with every output placed between guard zones: the guards are intact
    afterwards (no out-of-bounds store) and the payload equals the host-buffer result."""
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(3 * N + T)
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    m.update(make_params(rng, p, L, kernel))
    m.set_path(path)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    host = m.filter_smoother_nll(Y, smoother_mode=1, want_yhat=True)
    dev = torch.device("cuda:0")
    d, G, SENT = m.igp_dim, 512, 1234.5

    def guarded(n):
        n_al = (n + 1) & ~1                     # keep the payload 16-byte aligned (the many-chains kernels require it)
        buf = torch.full((G + n_al + G,), SENT, dtype=torch.float64, device=dev)
        return buf, buf[G:G + n]
    bX, X = guarded(N * T * L * d)
    bXs, Xs = guarded(N * T * L * d)
    bYh, Yh = guarded(N * T * p)
    bn, nll = guarded(N)
    bx, xT = guarded(N * L * d)
    Yd = torch.from_numpy(Y).to(dev)
    m.filter_smoother_nll_device(Yd, smoother_mode=1, X=X.view(N, T, L, d), Xs=Xs.view(N, T, L, d), Yhat=Yh.view(N, T, p), nll=nll, xT=xT.view(N, L, d))
    torch.cuda.synchronize()
    for name, buf, n in (("X", bX, N * T * L * d), ("Xs", bXs, N * T * L * d), ("Yhat", bYh, N * T * p), ("nll", bn, N), ("xT", bx, N * L * d)):
        h = buf.cpu().numpy()
        assert np.all(h[:G] == SENT) and np.all(h[G + ((n + 1) & ~1):] == SENT), name
    assert rel_err(X.cpu().numpy().reshape(N, T, L, d), host["X"]) < 1e-13
    assert rel_err(Xs.cpu().numpy().reshape(N, T, L, d), host["Xs"]) < 1e-13
    assert rel_err(Yh.cpu().numpy().reshape(N, T, p), host["Yhat"]) < 1e-13
    assert rel_err(nll.cpu().numpy(), host["nll"]) < 1e-13


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L,T,cut", [("Matern32", 16, 8, 60000, 29952), ("Matern52", 8, 4, 3000, 1024), ("Matern32", 64, 32, 5000, 2560),
                                              ("Matern32", 256, 64, 3001, 1536)])
def test_objective_begin_finish_blocks_equal_the_whole_sequence(cuda_lib, kernel, p, L, T, cut):
    """The one-pass time-sharded protocol on ONE device: block 0 = steps [0, cut), block 1 = [cut, T).  begin returns block
    0's end state from a zero carry-in, finish evaluates each block from its true carry-in; the two [loss, grad] add up to
    the evaluation of the whole sequence."""
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    from multioutputihgp_b200.parallel import carry_in_from_block_ends, stack_consts
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(T + p)
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    m.update(make_params(rng, p, L, kernel))
    Y = make_data(rng, p, L, T)
    lw, gw = m.objective(Y[None])
    dev = torch.device("cuda:0")
    d = m.igp_dim
    Yd = [torch.from_numpy(np.ascontiguousarray(Y[:cut]))[None].to(dev).contiguous(), torch.from_numpy(np.ascontiguousarray(Y[cut:]))[None].to(dev).contiguous()]
    out = [torch.zeros(2 + m.num_param, dtype=torch.float64, device=dev) for _ in range(2)]
    ex, edx = m.objective_begin_device(Yd[0])
    m.objective_finish_device(Yd[0], out[0][0:1], out[0][2:])
    consts = stack_consts([m.latent_consts(l) for l in range(L)])
    xin, dxin = carry_in_from_block_ends(consts, [cut, T - cut], [ex[0], np.zeros((L, d))], [edx[0], np.zeros((L, 3, d))], np.zeros((L, d)), np.zeros((L, 3, d)), 1)
    # the carried state equals the state the whole-block evaluation ends in
    _, _, xT, dxT = m.objective(Y[None, :cut], want_state=True)
    assert rel_err(xin, xT[0]) < 1e-11 and rel_err(dxin, dxT[0]) < 1e-10
    m.objective_begin_device(Yd[1], want_end=False)
    m.objective_finish_device(Yd[1], out[1][0:1], out[1][2:], x0=torch.from_numpy(xin[None]).to(dev), dx0=torch.from_numpy(dxin[None]).to(dev))
    torch.cuda.synchronize()
    h0, h1 = out[0].cpu().numpy(), out[1].cpu().numpy()
    assert abs(h0[0] + h1[0] - lw) <= 1e-10 * abs(lw)
    assert rel_err(h0[2:] + h1[2:], gw) < TOL
    # ... and against the oracle's loop over the whole sequence (not only GPU against GPU)
    from oracle.binding import OracleMOIHGP
    o = OracleMOIHGP(0.1, p, L, kernel, True)
    o.update(m.params)
    lo, go, _, _ = o.objective(Y[None])
    assert _close(h0[0] + h1[0], lo) and rel_err(h0[2:] + h1[2:], go) < TOL


# chunked-scan shapes with several chunks and latent groups: L a multiple of 8 (the thread-per-sub-chunk kernels) and not
# (the warp-per-chunk kernels)
SCAN_LANES_SHAPES = [("Matern32", 64, 32, 1, 5000), ("Matern52", 16, 8, 2, 1300), ("Matern32", 32, 16, 2, 256), ("Matern52", 24, 24, 1, 777)]
OBJ_LANES_SHAPES = [("Matern32", 64, 32, 1, 5000), ("Matern52", 16, 8, 3, 1300), ("Matern32", 32, 16, 2, 256), ("Matern52", 24, 8, 2, 33),
                    ("Matern32", 48, 24, 1, 4097)]
WARP_SHAPES = [("Matern32", 64, 30, 1, 5000), ("Matern52", 16, 5, 2, 1300), ("Matern32", 48, 21, 1, 4097), ("Matern52", 24, 11, 2, 33)]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L,N,T", SCAN_LANES_SHAPES + WARP_SHAPES)
def test_scan_final_kernels_agree(cuda_lib, kernel, p, L, N, T):
    """Both final-pass kernels of the chunked-scan path - thread per sub-chunk (k_scan_lanes, L a multiple of 8) and warp
    per chunk (k_scan, other L) - against the oracle from a carried-in state, in both smoother modes."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    assert (L % 8 == 0) == ((kernel, p, L, N, T) in SCAN_LANES_SHAPES)
    rng = np.random.default_rng(T)
    params = make_params(rng, p, L, kernel)
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    o = OracleMOIHGP(0.1, p, L, kernel, True)
    m.update(params)
    o.update(params)
    m.set_path("scan")
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    x0 = 0.3 * rng.standard_normal((N, L, m.igp_dim))
    for mode in (1, 0):
        r = m.filter_smoother_nll(Y, x0=x0, smoother_mode=mode)
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, nthreads=8)
        for k in ("X", "nll", "xT"):
            assert rel_err(r[k], ro[k]) < TOL, (k, mode)
        _assert_smoothed(r, ro, mode, mode)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L,N,T", OBJ_LANES_SHAPES + WARP_SHAPES)
def test_objective_kernels_agree(cuda_lib, kernel, p, L, N, T):
    """Both implementations of the objective's scan - thread per sub-chunk (k_obj_lanes, L a multiple of 8) and warp per
    chunk (k_obj_scan, other L) - against the oracle: loss, gradient and final state from a carried-in state."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    assert (L % 8 == 0) == ((kernel, p, L, N, T) in OBJ_LANES_SHAPES)
    rng = np.random.default_rng(T + L)
    params = make_params(rng, p, L, kernel)
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    o = OracleMOIHGP(0.1, p, L, kernel, True)
    m.update(params)
    o.update(params)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    x0 = 0.3 * rng.standard_normal((N, L, m.igp_dim))
    dx0 = 0.1 * rng.standard_normal((N, L, 3, m.igp_dim))
    loss, grad, xT, dxT = m.objective(Y, x0=x0, dx0=dx0, want_state=True)
    lo, go, xo, dxo = o.objective(Y, x0=x0, dx0=dx0)
    assert _close(loss, lo)
    assert rel_err(grad, go) < TOL
    assert rel_err(xT, xo) < TOL and rel_err(dxT, dxo) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["Matern32", "Matern52"])
def test_block_transition_matches_the_host_powering(cuda_lib, kernel):
    """moihgp_cuda_block_transition (binary powering on the library's power tables) against parallel.block_transition
    (numpy, from AKHA and dAKHA alone) and against the brute-force sum for a short block."""
    from multioutputihgp_b200 import MOIHGPSequences
    from multioutputihgp_b200.parallel import block_transition, stack_consts
    from oracle.gen_golden import make_params
    rng = np.random.default_rng(5)
    p, L = 6, 3
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    m.update(make_params(rng, p, L, kernel))
    AK, dAK = stack_consts([m.latent_consts(l) for l in range(L)])
    for n in (1, 2, 5, 256, 1000, 123456):
        P, E = m.block_transition(n)
        Pn, En = block_transition(AK, dAK, n)
        assert rel_err(P, Pn) < 1e-12 and rel_err(E, En) < 1e-11, n
    P5, E5 = m.block_transition(5)
    for l in range(L):
        M = AK[l]
        assert rel_err(P5[l], np.linalg.matrix_power(M, 5)) < 1e-13
        for k in range(3):
            brute = sum(np.linalg.matrix_power(M, 4 - i) @ dAK[l, k] @ np.linalg.matrix_power(M, i) for i in range(5))
            assert rel_err(E5[l, k], brute) < 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L,N,cuts", [("Matern32", 8, 4, 1, (0, 512, 1280, 1700)), ("Matern52", 16, 8, 2, (0, 256, 512, 1024)),
                                               ("Matern32", 12, 5, 1, (0, 768, 800)), ("Matern52", 6, 3, 3, (0, 256, 257)),
                                               ("Matern32", 64, 32, 1, (0, 2048, 4096, 6000))])
def test_time_sharded_filter_smoother_blocks_equal_the_whole_sequence(cuda_lib, kernel, p, L, N, cuts):
    """moihgp_cuda_fsn_block_dev: a sequence cut into contiguous blocks (each on its own handle, as on its own GPU), forward
    carry exchange, mirror-image backward exchange (SURVEY 8e) - filtered states, smoothed states and NLL equal the
    whole-sequence pass, in both smoother modes."""
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    from multioutputihgp_b200.parallel import backward_carry_in, forward_carry_in
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(sum(cuts))
    params = make_params(rng, p, L, kernel)
    T, G = cuts[-1], len(cuts) - 1
    lengths = [cuts[g + 1] - cuts[g] for g in range(G)]
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    whole = MOIHGPSequences(0.1, p, L, kernel, True)
    whole.update(params)
    whole.set_path("scan")
    d = whole.igp_dim
    x0 = 0.3 * rng.standard_normal((N, L, d))
    dev = torch.device("cuda:0")
    models = []
    for g in range(G):
        m = MOIHGPSequences(0.1, p, L, kernel, True)
        m.update(params)
        models.append(m)
    Yd = [torch.from_numpy(np.ascontiguousarray(Y[:, cuts[g]:cuts[g + 1]])).to(dev) for g in range(G)]
    to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    for mode in (1, 0):
        ref = whole.filter_smoother_nll(Y, x0=x0, smoother_mode=mode)
        ph1 = [models[g].fsn_block(1, Yd[g], g == G - 1, mode) for g in range(G)]
        ends, ufirst = [a for a, _ in ph1], [b for _, b in ph1]
        x_in = [forward_carry_in(models[0].block_transition, lengths, ends, x0, g) for g in range(G)]
        u_after = [to_dev(ufirst[g + 1]) if g < G - 1 else None for g in range(G)]
        b0 = [models[g].fsn_block(2, Yd[g], g == G - 1, mode, x0=to_dev(x_in[g]), u_after=u_after[g]) for g in range(G)]
        X = [torch.zeros((N, lengths[g], L, d), dtype=torch.float64, device=dev) for g in range(G)]
        Xs = [torch.zeros_like(X[g]) for g in range(G)]
        nll = torch.zeros((G, N), dtype=torch.float64, device=dev)
        xT = torch.zeros((N, L, d), dtype=torch.float64, device=dev)
        for g in range(G):
            be = backward_carry_in(lambda n_: models[0].smoother_power(n_, mode), lengths, b0, g)
            models[g].fsn_block(3, Yd[g], g == G - 1, mode, x0=to_dev(x_in[g]), u_after=u_after[g], b_end=None if be is None else to_dev(be),
                                X=X[g], Xs=Xs[g], nll=nll[g], xT=xT if g == G - 1 else None)
        torch.cuda.synchronize()
        Xc = np.concatenate([x.cpu().numpy() for x in X], axis=1)
        Xsc = np.concatenate([x.cpu().numpy() for x in Xs], axis=1)
        assert rel_err(Xc, ref["X"]) < 1e-12, mode
        assert rel_err(nll.sum(0).cpu().numpy(), ref["nll"]) < 1e-12, mode
        assert rel_err(xT.cpu().numpy(), ref["xT"]) < 1e-12, mode
        assert (rel_err(Xsc, ref["Xs"]) if mode == 1 else literal_smoother_err(Xsc, ref["Xs"])[0]) < 1e-11, mode
        # ... and against the oracle's pass over the whole sequence (not only GPU against GPU)
        ro = OracleMOIHGP(0.1, p, L, kernel, True)
        ro.update(params)
        ro = ro.filter_smoother_nll(Y, x0=x0, smoother_mode=mode)
        assert rel_err(Xc, ro["X"]) < TOL and rel_err(nll.sum(0).cpu().numpy(), ro["nll"]) < TOL, mode
        _assert_smoothed({"Xs": Xsc}, ro, mode, ("oracle", mode))


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,threading,p,L,T", [("Matern32", False, 8, 4, 1), ("Matern32", True, 8, 4, 64), ("Matern52", True, 16, 8, 300),
                                                    ("Matern52", False, 5, 5, 17), ("Matern32", True, 40, 12, 129), ("Matern52", True, 3, 1, 40)])
def test_one_launch_objective_matches_the_general_path_and_the_oracle(cuda_lib, kernel, threading, p, L, T):
    """k_obj_small (one short sequence, one launch: the streaming learner's window) against the general objective path
    (forced with set_path('scan')) and the oracle; with a missing observation it hands over to the general path."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(100 * p + T)
    params = make_params(rng, p, L, kernel)
    Y = make_data(rng, p, L, T)[None]
    m = MOIHGPSequences(0.1, p, L, kernel, threading)
    o = OracleMOIHGP(0.1, p, L, kernel, threading)
    m.update(params)
    o.update(params)
    d = m.igp_dim
    x0 = 0.2 * rng.standard_normal((1, L, d))
    dx0 = 0.1 * rng.standard_normal((1, L, 3, d))
    n0 = m.launch_count
    la, ga, xa, dxa = m.objective(Y, x0=x0, dx0=dx0, want_state=True)
    assert m.launch_count - n0 == 1                     # really the one-launch kernel
    m.set_path("scan")
    lb, gb, xb, dxb = m.objective(Y, x0=x0, dx0=dx0, want_state=True)
    m.set_path("auto")
    lo, go, xo, dxo = o.objective(Y, x0=x0, dx0=dx0)
    for l_, g_, x_, dx_ in ((lb, gb, xb, dxb), (lo, go, xo, dxo)):
        assert _close(la, l_)
        assert rel_err(ga, g_) < TOL
        assert rel_err(xa, x_) < TOL and rel_err(dxa, dx_) < TOL
    # bound (resident) data takes the same kernel
    m.bind(Y)
    lc, gc = m.objective_bound(x0, dx0)
    m.bind(None)
    assert lc == la and np.array_equal(gc, ga)
    if p > L + 2 and T > 2:
        Yn = Y.copy()
        Yn[0, T // 2, 0] = np.nan
        ln, gn = m.objective(Yn, x0=x0, dx0=dx0)[:2]
        assert np.isnan(ln)                              # as the reference's (moihgp.h:501 multiplies the full y)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L,N,cuts", [("Matern32", 16, 8, 1, (0, 512, 1280, 2048, 2300)), ("Matern52", 8, 4, 2, (0, 256, 768, 1000)),
                                               ("Matern32", 256, 64, 1, (0, 1024, 2048, 3001))])
def test_time_sharded_objective_device_side_exchange(cuda_lib, kernel, p, L, N, cuts):
    """The host-round-trip-free protocol of the time-sharded objective on ONE device (one handle per block, as on its own
    GPU): objective_begin_async leaves each block's end state in device memory, carry_in_device (binary powering of the block
    transitions on the device) forms every block's carry-in from the stacked ends, objective_finish_device evaluates from it.
    The carry-ins equal the host algebra (parallel.carry_in_from_block_ends) and the states of the whole-sequence evaluation;
    the blocks' [loss, grad] add up to the whole-sequence evaluation and to the oracle's."""
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    from multioutputihgp_b200.parallel import carry_in_from_block_ends
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(sum(cuts) + p)
    params = make_params(rng, p, L, kernel)
    T, G = cuts[-1], len(cuts) - 1
    lengths = [cuts[g + 1] - cuts[g] for g in range(G)]
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    dev = torch.device("cuda:0")
    models = []
    for g in range(G):
        m = MOIHGPSequences(0.1, p, L, kernel, True)
        m.update(params)
        models.append(m)
    d = models[0].igp_dim
    f64 = dict(dtype=torch.float64, device=dev)
    x0 = 0.2 * rng.standard_normal((N, L, d))
    dx0 = 0.1 * rng.standard_normal((N, L, 3, d))
    x0d, dx0d = torch.from_numpy(x0).to(dev), torch.from_numpy(dx0).to(dev)
    Yd = [torch.from_numpy(np.ascontiguousarray(Y[:, cuts[g]:cuts[g + 1]])).to(dev) for g in range(G)]
    ends = torch.zeros((G, N, L, 4, d), **f64)
    for g in range(G):
        models[g].objective_begin_async(Yd[g], None if g == G - 1 else ends[g])
    out = torch.zeros((G, 2 + models[0].num_param), **f64)
    xin = torch.zeros((G, N, L, d), **f64)
    dxin = torch.zeros((G, N, L, 3, d), **f64)
    for g in range(G):
        models[g].carry_in_device(ends, lengths, g, xin[g], dxin[g], x0=x0d, dx0=dx0d)
        models[g].objective_finish_device(Yd[g], out[g, 0:1], out[g, 2:], x0=xin[g], dx0=dxin[g])
    torch.cuda.synchronize()
    eh = ends.cpu().numpy()
    for g in range(G):
        for n in range(N):
            xh, dxh = carry_in_from_block_ends(models[0].block_transition, lengths, eh[:, n, :, 0], eh[:, n, :, 1:], x0[n], dx0[n], g)
            assert rel_err(xin[g, n].cpu().numpy(), xh) < 1e-12 and rel_err(dxin[g, n].cpu().numpy(), dxh) < 1e-11, (g, n)
    whole = MOIHGPSequences(0.1, p, L, kernel, True)
    whole.update(params)
    for g in range(1, G):                                   # the carried state is the state the sequence has at the cut
        _, _, xT, dxT = whole.objective(Y[:, :cuts[g]], x0=x0, dx0=dx0, want_state=True)
        assert rel_err(xin[g].cpu().numpy(), xT) < 1e-11 and rel_err(dxin[g].cpu().numpy(), dxT) < 1e-10, g
    lw, gw = whole.objective(Y, x0=x0, dx0=dx0)
    tot = out.sum(0).cpu().numpy()
    assert abs(tot[0] - lw) <= 1e-10 * abs(lw) and rel_err(tot[2:], gw) < TOL
    o = OracleMOIHGP(0.1, p, L, kernel, True)
    o.update(params)
    lo, go, _, _ = o.objective(Y, x0=x0, dx0=dx0)
    assert _close(tot[0], lo) and rel_err(tot[2:], go) < TOL


@pytest.mark.gpu
def test_backprojection_with_a_mixing_matrix_larger_than_shared_memory(cuda_lib):
    """Yhat = U sqrt(S) x(0) (moihgp.h:222-225) at p = 512, L = 64: U (256 KB) does not fit into shared memory."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(512)
    p, L, T = 512, 64, 300
    params = make_params(rng, p, L, "Matern32")
    Y = make_data(rng, p, L, T)[None]
    m = MOIHGPSequences(0.1, p, L, "Matern32", True)
    o = OracleMOIHGP(0.1, p, L, "Matern32", True)
    m.update(params)
    o.update(params)
    r = m.filter_smoother_nll(Y, smoother_mode=-1, want_yhat=True)
    ro = o.filter_smoother_nll(Y, smoother_mode=-1, want_yhat=True)
    assert rel_err(r["Yhat"], ro["Yhat"]) < TOL and rel_err(r["X"], ro["X"]) < TOL and rel_err(r["nll"], ro["nll"]) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L,N,T,path", [("Matern52", 16, 8, 70, 300, "chain"), ("Matern32", 8, 4, 3, 1000, "scan"), ("Matern32", 64, 32, 1, 700, "scan")])
def test_function_values_only_output(cuda_lib, kernel, p, L, N, T, path):
    """moihgp_cuda_filter_smoother_nll_values: the same pass, only the function-value component H x = x(0) of the filtered and
    smoothed states comes back ([N,T,L]); equal to component 0 of the full output, several pipeline slices included."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_data, make_params
    rng = np.random.default_rng(N + T)
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    m.update(make_params(rng, p, L, kernel))
    m.set_path(path)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    x0 = 0.2 * rng.standard_normal((N, L, m.igp_dim))
    full = m.filter_smoother_nll(Y, x0=x0, smoother_mode=1, want_yhat=True)
    val = m.filter_smoother_nll_values(Y, x0=x0, smoother_mode=1, want_yhat=True)
    assert np.array_equal(val["F"], full["X"][..., 0]) and np.array_equal(val["Fs"], full["Xs"][..., 0])
    assert np.array_equal(val["nll"], full["nll"]) and np.array_equal(val["xT"], full["xT"]) and np.array_equal(val["Yhat"], full["Yhat"])


@pytest.mark.gpu
@pytest.mark.parametrize("p,L", [(256, 64), (128, 33), (100, 21), (512, 16)])
def test_device_polar_factor_matches_svd_and_falls_back_on_rank_deficiency(cuda_lib, p, L):
    """update() on the device: k_polar_ns (Newton-Schulz, the fast way for a block that is nearly orthonormal, as inside a
    line search) against the SVD polar factor on nearly orthonormal, generic, badly scaled and ill-conditioned blocks; a
    rank-deficient block falls back to k_polar (one-sided Jacobi), whose answer must still be a polar factor."""
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_params
    rng = np.random.default_rng(p + L)
    m = MOIHGPSequences(0.1, p, L, "Matern32", True)
    base = make_params(rng, p, L, "Matern32")
    Q, _ = np.linalg.qr(rng.standard_normal((p, L)))
    sv = np.geomspace(1.0, 1e-5, L)
    blocks = {
        "near-orthonormal": Q + 0.01 * rng.standard_normal((p, L)),
        "generic": rng.standard_normal((p, L)),
        "scaled": 1e4 * rng.standard_normal((p, L)),
        "ill-conditioned": (Q * sv) @ np.linalg.qr(rng.standard_normal((L, L)))[0],
    }
    for name, B in blocks.items():
        params = base.copy()
        params[:p * L] = B.ravel()
        m.update(params)
        U = m.U.copy()
        Wm, _, Vt = np.linalg.svd(B, full_matrices=False)
        tol = 1e-9 if name != "ill-conditioned" else 1e-7           # the polar factor's conditioning is 1 / sigma_min
        assert rel_err(U, Wm @ Vt) < tol, name
        assert np.max(np.abs(U.T @ U - np.eye(L))) < 1e-12, name
    # rank-deficient: no unique polar factor; the iteration gives up and the Jacobi kernel's answer is the result.  Any
    # polar factor B = U H has orthonormal columns, H = U'B symmetric positive semi-definite, and U U'B = B.
    B = rng.standard_normal((p, L))
    B[:, -1] = B[:, 0]
    params = base.copy()
    params[:p * L] = B.ravel()
    m.update(params)
    U = m.U.copy()
    H = U.T @ B
    assert np.max(np.abs(U.T @ U - np.eye(L))) < 1e-12
    assert rel_err(H, H.T) < 1e-12
    assert np.min(np.linalg.eigvalsh(0.5 * (H + H.T))) > -1e-12 * np.max(np.abs(H))
    assert rel_err(U @ H, B) < 1e-9
