"""Models with 64 < L <= 256 latent processes, on every whole-sequence entry point, against the CPU oracle at conftest.TOL.

What is new at these shapes (and which test reaches it):
  - the projection k_project_mma<8, 4> (latent blocks of 64 columns) for even p and a 16-byte aligned Y; the scalar
    k_project for odd p or an offset Y, with 64-step tiles where the 128-step tile does not fit (L >= 186);
  - the many-CTA Newton-Schulz polar factor in update();
  - the missing-output solve with its scratch in global memory in k_nan_fix and k_step (L >= 120) and in k_lik (L >= 118);
  - k_obj_finish sized by L, and k_backproject's 32-step tile (L >= 198);
  - the refusals: create() above 256 latents, the streaming learner above 64."""
import numpy as np
import pytest

from conftest import TOL, literal_smoother_err, rel_err

pytestmark = pytest.mark.gpu


def _model(kernel, p, L, seed, threading=True, scale=1.0):
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_params
    rng = np.random.default_rng(seed)
    params = make_params(rng, p, L, kernel)
    params[:p * L] *= scale
    m = MOIHGPSequences(0.1, p, L, kernel, threading)
    o = OracleMOIHGP(0.1, p, L, kernel, threading)
    m.update(params)
    o.update(params)
    return m, o, rng, params


def _data(rng, p, L, N, T):
    from oracle.gen_golden import make_data
    return np.stack([make_data(rng, p, L, T) for _ in range(N)])


def _states_close(a, b, mode, what):
    """RTS: norm-wise.  Literal smoother: through literal_smoother_err; with a few hundred latents some have rho(G) large
    enough that the reference overflows about a hundred steps from the end, so at least 50 trailing steps are compared."""
    if mode == 1:
        assert rel_err(a, b) < TOL, (what, rel_err(a, b))
    else:
        err, steps = literal_smoother_err(a, b)
        assert err < TOL and steps >= min(np.asarray(b).shape[-3], 50), (what, err, steps)


def _with_nan(Y, L):
    """Rows with some outputs missing (at least L observed: U0'U0 stays regular, as the reference's LDLT needs for a
    well-defined answer) and a row with every output missing (U0'U0 = 0: u = 0)."""
    Y = Y.copy()
    N, T, p = Y.shape
    Y[0, T // 2, [1, p // 2, p - 1]] = np.nan
    Y[-1, T // 3, :] = np.nan
    Y[-1, T // 3 + 1, :max(1, (p - L) // 2)] = np.nan
    return Y


# ------------------------------------------------------------------------------------------------------------ limits
def test_create_accepts_up_to_256_latents_and_refuses_257(cuda_lib, capfd):
    from multioutputihgp_b200 import MOIHGPSequences
    for p, L in ((65, 65), (300, 65), (256, 256), (512, 256)):
        m = MOIHGPSequences(0.1, p, L, "Matern32", True)
        assert m.num_latent == L and m.num_param == p * L + L + 1 + 3 * L
    with pytest.raises(RuntimeError):
        MOIHGPSequences(0.1, 300, 257, "Matern32", True)
    assert "num_latent > 256 is not supported" in capfd.readouterr().err


def test_streaming_learner_refuses_more_than_64_latents(cuda_lib):
    from multioutputihgp_b200 import MOIHGPSequences
    from multioutputihgp_b200.online_learning import MOIHGPOnlineLearning
    m = MOIHGPSequences(0.1, 80, 65, "Matern32", True)
    assert not m.online_begin(4)
    assert "num_latent <= 64" in m._lib.moihgp_cuda_last_error(m._h).decode()
    with pytest.raises(ValueError, match="num_latent <= 64"):
        MOIHGPOnlineLearning(0.1, 80, 65, 0.1, windowsize=4)


CPP_ONLINE_REFUSAL = r"""
#include <cstdio>
#include <stdexcept>
#include <string>
#include <moihgp_b200/moihgp.hpp>
using namespace moihgp_b200;
int main() {
    MOIHGP<Matern32StateSpace> gp(0.1, 80, 65, true);
    try {
        OnlineObjective<Matern32StateSpace> obj(&gp, 0.1, 4);     // what MOIHGPOnlineLearning's constructor builds
    } catch (const std::runtime_error& e) {
        std::printf("refused: %s\n", e.what());
        return std::string(e.what()).find("num_latent <= 64") == std::string::npos;
    }
    std::printf("accepted\n");
    return 1;
}
"""


def test_cpp_streaming_learner_refuses_more_than_64_latents(cuda_lib, tmp_path):
    """The C++ host mirror: the learner's objective throws std::runtime_error with the library's message at L = 65."""
    import os
    import subprocess
    from conftest import ROOT
    src, exe = tmp_path / "online_refusal.cpp", tmp_path / "online_refusal"
    src.write_text(CPP_ONLINE_REFUSAL)
    lib = os.path.join(ROOT, "multioutputihgp_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++11", "-Wall", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe), "-L" + lib,
                           "-lmoihgp", "-Wl,-rpath," + lib, "-Wl,-rpath,/usr/local/cuda/lib64"])
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "refused" in r.stdout and "num_latent <= 64" in r.stdout, (r.stdout, r.stderr)


# ------------------------------------------------------------------------------------------------------------ update
def _assert_device_polar(launches):
    """update() at L > 64 launches 6 kernels around the Newton-Schulz loop, then 3 per step in batches of 6 steps until the
    iteration stops, at most 10 batches (60 steps), plus the K-setup.  On a finite block the start is scaled so that
    max|X'X - I| <= 1, so the loop can only end before its bound through a convergence test: fewer than 10 batches means
    the device produced U, not the host Jacobi the library falls back to."""
    batches, rest = divmod(launches - 1 - 6, 18)
    assert rest == 0 and 1 <= batches < 10, launches


@pytest.mark.parametrize("p,L,scale", [(256, 65, 1.0), (96, 96, 1.0), (200, 128, 30.0), (512, 256, 1.0)])
def test_update_polar_factor_on_device(cuda_lib, p, L, scale):
    """U = the SVD polar factor of the raw block (scale != 1: the iteration starts from a rescaled block), orthonormal;
    update(get_params()) leaves U unchanged; the same input gives the same U bit for bit."""
    from multioutputihgp_b200 import MOIHGPSequences
    rng = np.random.default_rng(p + L)
    m = MOIHGPSequences(0.1, p, L, "Matern32", True)
    raw = scale * (rng.standard_normal((p, L)) / np.sqrt(L) + np.eye(p, L))
    params = np.concatenate([raw.ravel(), np.ones(L), [1e-2], np.tile([1.0, 1.0, 0.1], L)])
    n0 = m.launch_count
    m.update(params)
    _assert_device_polar(m.launch_count - n0)
    u, _, vt = np.linalg.svd(raw, full_matrices=False)
    assert rel_err(m.U, u @ vt) < 1e-12
    assert np.max(np.abs(m.U.T @ m.U - np.eye(L))) < 1e-13
    U1 = m.U.copy()
    n0 = m.launch_count
    m.update(m.params)
    _assert_device_polar(m.launch_count - n0)
    assert rel_err(m.U, U1) < 1e-13
    m.update(params)
    assert np.array_equal(m.U, U1)


# ------------------------------------------------------------------------------------------------------------ fused pass
# (kernel, p, L, N, T): the projection kernel each shape selects
FUSED = [
    ("Matern32", 128, 65, 2, 300),     # k_project_mma<8, 4>, two latent blocks, odd L (scalar U staging)
    ("Matern52", 129, 96, 1, 260),     # odd p: k_project<128>
    ("Matern32", 256, 128, 1, 300),    # k_project_mma<8, 4>, p multiple of the K panel
    ("Matern52", 512, 128, 1, 200),
    ("Matern32", 136, 100, 1, 200),    # p not a multiple of the 16-column K panel
    ("Matern52", 256, 256, 1, 150),    # square U (rho = 0), four latent blocks, k_backproject's 32-step tile
    ("Matern32", 301, 200, 1, 140),    # odd p, L >= 186: k_project<64>; L >= 198: 32-step back-projection
]


@pytest.mark.parametrize("kernel,p,L,N,T", FUSED)
@pytest.mark.parametrize("mode", [0, 1])
def test_fused_pass_matches_oracle(cuda_lib, kernel, p, L, N, T, mode):
    m, o, rng, _ = _model(kernel, p, L, p + L + T)
    Y = _data(rng, p, L, N, T)
    for x0 in (None, 0.2 * rng.standard_normal((N, L, m.igp_dim))):
        r = m.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True)
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True)
        assert rel_err(r["X"], ro["X"]) < TOL
        _states_close(r["Xs"], ro["Xs"], mode, "Xs")
        for k in ("Yhat", "nll", "xT"):
            assert rel_err(r[k], ro[k]) < TOL, (k, rel_err(r[k], ro[k]))
        v = m.filter_smoother_nll_values(Y, x0=x0, smoother_mode=mode, want_yhat=True)
        assert np.array_equal(v["F"], r["X"][..., 0]) and np.array_equal(v["Fs"], r["Xs"][..., 0], equal_nan=True)
        for k in ("Yhat", "nll", "xT"):
            assert np.array_equal(v[k], r[k]), k
    assert m.nan_status == 0


@pytest.mark.parametrize("kernel,p,L", [("Matern32", 128, 96), ("Matern52", 160, 128), ("Matern32", 211, 200)])
def test_missing_outputs_match_oracle(cuda_lib, kernel, p, L):
    """Rows with some and with all outputs NaN: L = 96 solves in shared memory, L >= 128 in global scratch."""
    m, o, rng, _ = _model(kernel, p, L, 7 * L)
    Y = _with_nan(_data(rng, p, L, 2, 120), L)
    r = m.filter_smoother_nll(Y, smoother_mode=1, want_yhat=True)
    ro = o.filter_smoother_nll(Y, smoother_mode=1, want_yhat=True)
    assert m.nan_status == 1
    for k in ("X", "Xs", "Yhat", "xT"):
        assert rel_err(r[k], ro[k]) < TOL, (k, rel_err(r[k], ro[k]))
    assert np.isnan(r["nll"]).all() and np.isnan(ro["nll"]).all()


@pytest.mark.parametrize("L", [117, 118, 119, 128])
def test_per_observation_symbols_with_missing_outputs(cuda_lib, L):
    """gp32_step / gp32_lik (one observation per call) on observations with and without NaNs.  Each kernel moves the LDLT
    scratch to global memory where its own shared memory would pass 227 KB: k_lik from L = 118, k_step from L = 120 (L = 117:
    both in shared memory; 118, 119: k_lik global, k_step shared; 128: both global)."""
    from multioutputihgp_b200 import MOIHGP
    from oracle.binding import OracleMOIHGP
    from oracle.gen_golden import make_params
    p = 150
    rng = np.random.default_rng(3)
    params = make_params(rng, p, L, "Matern32")
    m = MOIHGP(0.1, p, L, kernel="Matern32", threading=True)
    o = OracleMOIHGP(0.1, p, L, "Matern32", True)
    m.update(params)
    o.update(params)
    Y = _data(rng, p, L, 1, 6)[0]
    Y[2, :] = np.nan
    Y[4, :p - L] = np.nan
    x = 0.1 * rng.standard_normal((L, 2))
    dx = 0.1 * rng.standard_normal((L, 3, 2))
    for t in (2, 4):
        got, ref = m.step(x, Y[t], dx), o.step(x, Y[t], dx)
        for a, b in zip(got, ref):
            assert rel_err(a, b) < TOL
    for t in (2, 4, 5):
        (lg, gg), (lr, gr) = m.negLogLikelihood(x, Y[t], dx), o.negLogLikelihood(x, Y[t], dx)
        for a, b in ((np.atleast_1d(lg), np.atleast_1d(lr)), (gg, gr), (np.atleast_1d(m.negLogLikelihood(x, Y[t])),
                                                                        np.atleast_1d(o.negLogLikelihood(x, Y[t])))):
            assert np.array_equal(np.isnan(a), np.isnan(b)), t
            ok = ~np.isnan(b)
            assert not ok.any() or rel_err(a[ok], b[ok]) < TOL, t
    got, ref = m.step(x, Y[5], dx), o.step(x, Y[5], dx)
    for a, b in zip(got, ref):
        assert rel_err(a, b) < TOL


@pytest.mark.parametrize("kernel,p,L", [("Matern32", 128, 65), ("Matern52", 257, 128)])
def test_nll_steps_match_oracle_and_sum_to_the_pass(cuda_lib, kernel, p, L):
    from test_gpu_nll_steps import _oracle_steps
    m, o, rng, params = _model(kernel, p, L, 11 * L)
    Y = _data(rng, p, L, 2, 80)
    x0 = 0.2 * rng.standard_normal((2, L, m.igp_dim))
    r = m.nll_steps(Y, x0=x0)
    ref, xT = _oracle_steps(kernel, p, L, params, Y, x0)
    assert rel_err(r["nll_steps"], ref) < TOL and rel_err(r["xT"], xT) < TOL
    f = m.filter_smoother_nll(Y, x0=x0, smoother_mode=1)
    assert rel_err(r["nll_steps"].sum(axis=1), f["nll"]) < 1e-12


# ------------------------------------------------------------------------------------------------------------ objective
@pytest.mark.parametrize("kernel,p,L,T", [("Matern32", 128, 65, 300), ("Matern52", 256, 128, 260), ("Matern32", 131, 96, 200),
                                          ("Matern52", 256, 256, 120)])
@pytest.mark.parametrize("threading", [True, False])
def test_objective_matches_oracle(cuda_lib, kernel, p, L, T, threading):
    m, o, rng, _ = _model(kernel, p, L, 3 * L + T, threading=threading)
    Y = _data(rng, p, L, 2, T)
    loss, grad = m.objective(Y)
    lo, go, _, _ = o.objective(Y)
    assert abs(loss - lo) <= TOL * abs(lo) and rel_err(grad, go) < TOL
    m.bind(Y)
    lb, gb = m.objective_bound()
    assert lb == loss and np.array_equal(gb, grad)
    m.bind(None)


def test_objective_blocks_add_up_to_the_whole_sequence(cuda_lib):
    """objective_begin_dev / objective_finish_dev over two blocks of one sequence sum to the whole-sequence objective."""
    import torch
    from multioutputihgp_b200.parallel import carry_in_from_block_ends, stack_consts
    kernel, p, L, T, cut = "Matern52", 128, 96, 1024, 512
    m, o, rng, _ = _model(kernel, p, L, 68)
    Y = _data(rng, p, L, 1, T)[0]
    lw, gw = m.objective(Y[None])
    d = m.igp_dim
    f64 = dict(dtype=torch.float64, device="cuda")
    Yd = [torch.from_numpy(Y[None, :cut].copy()).to(**f64), torch.from_numpy(Y[None, cut:].copy()).to(**f64)]
    loss = [torch.zeros(1, **f64) for _ in range(2)]
    grad = [torch.zeros(m.num_param, **f64) for _ in range(2)]
    ex, edx = m.objective_begin_device(Yd[0])
    m.objective_finish_device(Yd[0], loss[0], grad[0])
    consts = stack_consts([m.latent_consts(l) for l in range(L)])
    xin, dxin = carry_in_from_block_ends(consts, [cut, T - cut], [ex[0], np.zeros((L, d))], [edx[0], np.zeros((L, 3, d))], np.zeros((L, d)),
                                         np.zeros((L, 3, d)), 1)
    m.objective_begin_device(Yd[1], want_end=False)
    m.objective_finish_device(Yd[1], loss[1], grad[1], x0=torch.from_numpy(xin[None].copy()).to(**f64),
                              dx0=torch.from_numpy(dxin[None].copy()).to(**f64))
    torch.cuda.synchronize()
    lt = float(loss[0].cpu()[0] + loss[1].cpu()[0])
    gt = grad[0].cpu().numpy() + grad[1].cpu().numpy()
    assert abs(lt - lw) <= 1e-10 * abs(lw) and rel_err(gt, gw) < TOL


# ------------------------------------------------------------------------------------------------------------ sampler
@pytest.mark.parametrize("kernel,p,L", [("Matern32", 128, 96), ("Matern52", 256, 256)])
def test_samples_are_rts_mean_plus_recomputed_noise(cuda_lib, kernel, p, L):
    from test_gpu_sampling import _factors, _outputs, noise
    m, _, rng, _ = _model(kernel, p, L, 5 * L)
    N, T, S, seed = 1, 90, 2, 0xDEADBEEF_0000_0077
    Y = _data(rng, p, L, N, T)
    r = m.sample_posterior(Y, S, seed, want_states=True, want_outputs=True)
    Xs = m.filter_smoother_nll(Y, smoother_mode=1, want_nll=False)["Xs"]
    assert rel_err(r["Xs"], Xs) < TOL
    e = noise(seed, S, N, T, *_factors(m))
    assert rel_err(r["X"], r["Xs"][None] + e) < TOL
    assert np.array_equal(r["F"], r["X"][..., 0])
    assert rel_err(r["Y"], _outputs(m, r["F"])) < 1e-12


# ------------------------------------------------------------------------------------------------------------ device operands
@pytest.mark.parametrize("p,L", [(256, 128), (136, 96), (201, 96), (300, 256)])
@pytest.mark.parametrize("offset", [False, True])
def test_device_pass_with_aligned_and_offset_observations(cuda_lib, p, L, offset):
    """The device pass with a 16-byte aligned Y (tensor-pipe projection for even p) and with Y at an 8-byte offset (the
    scalar projection): the same numbers as the host-buffer call and the oracle, missing outputs included."""
    import torch
    kernel, N, T = "Matern32", 1, 160
    m, o, rng, _ = _model(kernel, p, L, p * L)
    Y = _with_nan(_data(rng, p, L, N, T), L) if L == 96 else _data(rng, p, L, N, T)
    buf = torch.zeros(N * T * p + 2, dtype=torch.float64, device="cuda")
    Yd = buf[int(offset):int(offset) + N * T * p].view(N, T, p)
    assert (Yd.data_ptr() % 16 == 8) == offset
    Yd.copy_(torch.from_numpy(Y))
    f64 = dict(dtype=torch.float64, device="cuda")
    X, Xs, Yhat = (torch.zeros((N, T, L, 2), **f64), torch.zeros((N, T, L, 2), **f64), torch.zeros((N, T, p), **f64))
    nll, xT = torch.zeros(N, **f64), torch.zeros((N, L, 2), **f64)
    m.filter_smoother_nll_device(Yd, smoother_mode=1, X=X, Xs=Xs, Yhat=Yhat, nll=nll, xT=xT)
    torch.cuda.synchronize()
    ro = o.filter_smoother_nll(Y, smoother_mode=1, want_yhat=True)
    for k, t in (("X", X), ("Xs", Xs), ("Yhat", Yhat), ("xT", xT)):
        assert rel_err(t.cpu().numpy(), ro[k]) < TOL, k
    got = nll.cpu().numpy()
    if L == 96:
        assert np.isnan(got).all()
    else:
        assert rel_err(got, ro["nll"]) < TOL


def test_device_pass_right_after_update_is_capturable_in_a_cuda_graph(cuda_lib):
    """L = 128: right after update(params) the device pass can be captured into a CUDA graph; replays on new data equal the
    host-buffer call."""
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_params
    kernel, p, L, N, T = "Matern32", 256, 128, 1, 300
    rng = np.random.default_rng(9)
    f64 = dict(dtype=torch.float64, device="cuda")
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    Y = torch.zeros((N, T, p), **f64)
    X, Xs, nll, xT = (torch.zeros((N, T, L, 2), **f64), torch.zeros((N, T, L, 2), **f64), torch.zeros(N, **f64), torch.zeros((N, L, 2), **f64))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        m.update(make_params(rng, p, L, kernel))
        m.filter_smoother_nll_device(Y, smoother_mode=1, X=X, Xs=Xs, nll=nll, xT=xT)     # warm-up: workspaces
        torch.cuda.synchronize()
        m.update(make_params(rng, p, L, kernel))
        with torch.cuda.graph(g, stream=side):
            m.filter_smoother_nll_device(Y, smoother_mode=1, X=X, Xs=Xs, nll=nll, xT=xT)
    for rep in range(2):
        Yh = _data(rng, p, L, N, T)
        Y.copy_(torch.from_numpy(Yh))
        g.replay()
        torch.cuda.synchronize()
        ref = m.filter_smoother_nll(Yh, smoother_mode=1)
        for k, t in (("X", X), ("Xs", Xs), ("nll", nll), ("xT", xT)):
            assert rel_err(t.cpu().numpy(), ref[k]) < TOL, (rep, k)
