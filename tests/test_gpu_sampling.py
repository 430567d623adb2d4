"""Posterior sample paths (moihgp_cuda_sample_posterior*): steady-state forward-filtering, backward-sampling in RTS form,
x~ = Xs_rts + e with e[T-1] = LF z[T-1], e[t] = G e[t+1] + LC z[t].

The CPU tests check the two pieces the GPU tests rely on: a NumPy Philox4x32-10 against the Random123 known-answer vectors,
and the decomposition x~ = Xs_rts + e against the direct FFBS recursion.  The GPU tests (-m gpu) recompute e in NumPy from
the same counters and the library's own factors, and check the moments of many draws against the steady-state covariances."""
import numpy as np
import pytest

from conftest import TOL, rel_err

_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al., SC'11; Random123) on arrays: ctr = 4 broadcastable uint32 arrays, key = 2 ints."""
    c0, c1, c2, c3 = np.broadcast_arrays(*[np.asarray(c, dtype=np.uint64) & _MASK for c in ctr])
    k0, k1 = np.uint64(key[0]) & _MASK, np.uint64(key[1]) & _MASK
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2     # 32 x 32 -> 64 bits, no overflow
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _MASK
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _MASK, (k1 + np.uint64(0xBB67AE85)) & _MASK
    return c0, c1, c2, c3


def normals(seed, s, n, l, t, d):
    """z[..., :d] of the draws (s, n, l, t) (broadcast): counter (t, n, l, s), key (seed lo, seed hi), Box-Muller in fp64."""
    w = philox4x32_10((t, n, l, s), (seed & 0xFFFFFFFF, seed >> 32))
    u = [(wi.astype(np.float64) + 0.5) * 2.0 ** -32 for wi in w]
    r0 = np.sqrt(-2.0 * np.log(u[0]))
    z = [r0 * np.cos(2 * np.pi * u[1]), r0 * np.sin(2 * np.pi * u[1])]
    if d > 2:
        z.append(np.sqrt(-2.0 * np.log(u[2])) * np.cos(2 * np.pi * u[3]))
    return np.stack(z, axis=-1)


def noise(seed, S, N, T, G, LC, LF):
    """e [S,N,T,L,d] of samples 0..S-1; G, LC, LF [L,d,d]."""
    L, d = G.shape[0], G.shape[1]
    z = normals(seed, np.arange(S)[:, None, None, None], np.arange(N)[None, :, None, None], np.arange(L)[None, None, None, :],
                np.arange(T)[None, None, :, None], d)
    e = np.empty_like(z)
    e[:, :, T - 1] = np.einsum("lij,snlj->snli", LF, z[:, :, T - 1])
    for t in range(T - 2, -1, -1):
        e[:, :, t] = np.einsum("lij,snlj->snli", G, e[:, :, t + 1]) + np.einsum("lij,snlj->snli", LC, z[:, :, t])
    return e


def _psd(rng, d, scale=1.0):
    B = rng.standard_normal((d, d))
    return scale * (B @ B.T + 0.1 * np.eye(d))


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_numpy_philox_matches_random123_known_answers():
    cases = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
             ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
             ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in cases:
        assert tuple(int(w) for w in philox4x32_10(ctr, key)) == want, (ctr, key)


def test_rts_mean_plus_noise_equals_direct_ffbs():
    """x~ = Xs_rts + e is the direct recursion x~[t] = X[t] + G (x~[t+1] - A X[t]) + LC z[t] rearranged (any A, G, X)."""
    rng = np.random.default_rng(7)
    S, N, T, L, d, seed = 3, 2, 37, 3, 3, 0x1234_5678_9ABC
    A = 0.5 * rng.standard_normal((L, d, d))
    G = 0.4 * rng.standard_normal((L, d, d))
    LF = np.linalg.cholesky(np.stack([_psd(rng, d) for _ in range(L)]))
    LC = np.linalg.cholesky(np.stack([_psd(rng, d, 0.1) for _ in range(L)]))
    X = rng.standard_normal((N, T, L, d))
    Xs = X.copy()
    for t in range(T - 2, -1, -1):
        Xs[:, t] = X[:, t] + np.einsum("lij,nlj->nli", G, Xs[:, t + 1] - np.einsum("lij,nlj->nli", A, X[:, t]))
    z = normals(seed, np.arange(S)[:, None, None, None], np.arange(N)[None, :, None, None], np.arange(L)[None, None, None, :],
                np.arange(T)[None, None, :, None], d)
    direct = np.empty((S, N, T, L, d))
    direct[:, :, T - 1] = X[None, :, T - 1] + np.einsum("lij,snlj->snli", LF, z[:, :, T - 1])
    for t in range(T - 2, -1, -1):
        pred = np.einsum("lij,nlj->nli", A, X[:, t])[None]
        direct[:, :, t] = (X[None, :, t] + np.einsum("lij,snlj->snli", G, direct[:, :, t + 1] - pred)
                           + np.einsum("lij,snlj->snli", LC, z[:, :, t]))
    assert rel_err(Xs[None] + noise(seed, S, N, T, G, LC, LF), direct) < 1e-12


def test_normals_depend_only_on_the_draw_index():
    d, seed = 3, 99
    a = normals(seed, np.arange(4)[:, None], 2, 1, np.arange(10)[None, :], d)
    b = normals(seed, 3, 2, 1, 7, d)
    assert np.array_equal(a[3, 7], b)
    assert abs(np.mean(normals(seed, 0, 0, 0, np.arange(20000), d))) < 0.05


# ---------------------------------------------------------------------------------------------------------------- GPU
def _model(kernel, p, L, seed, dt=0.1, igp=None):
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_params
    rng = np.random.default_rng(seed)
    params = make_params(rng, p, L, kernel)
    if igp is not None:
        params[p * L + L + 1:] = igp
    m = MOIHGPSequences(dt, p, L, kernel, True)
    m.update(params)
    return m, params, rng


def _factors(m):
    L = m.num_latent
    G = np.stack([m.smoother_consts(l, 1)[0] for l in range(L)])
    LF, LC = (np.stack(f) for f in zip(*[m.sampler_consts(l) for l in range(L)]))
    return G, LC, LF


def _outputs(m, F):
    p, L = m.num_output, m.num_latent
    Usq = m.U * np.sqrt(m.params[p * L:p * L + L])[None, :]
    return np.einsum("rl,sntl->sntr", Usq, F)


SAMPLE_CASES = [
    # kernel, p, L, N, T, x0, nan
    ("Matern52", 16, 8, 33, 300, True, False),     # many-chains mean, N not a multiple of 32, T = 9 chunks + 12 steps
    ("Matern32", 5, 3, 2, 1000, False, True),      # odd L, rows with missing outputs, T = 31 chunks + 8 steps
    ("Matern32", 4, 1, 3, 1, True, False),         # L = 1, T = 1
    ("Matern52", 3, 3, 2, 257, False, True),       # p == L
    ("Matern32", 8, 4, 40, 129, True, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["scan", "chain"])
@pytest.mark.parametrize("kernel,p,L,N,T,with_x0,with_nan", SAMPLE_CASES)
def test_samples_are_rts_mean_plus_recomputed_noise(cuda_lib, path, kernel, p, L, N, T, with_x0, with_nan):
    """Exact parity: x~ = the library's RTS mean + e recomputed in NumPy (Philox normals, the library's factors), on both
    variants of the sampler (set_path: scan = time-chunked, chain = one pass per chain)."""
    from oracle.gen_golden import make_data
    m, params, rng = _model(kernel, p, L, 10 * N + T)
    d, S, seed = m.igp_dim, 3, 0xDEADBEEF_0000_0011 + T
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    if with_nan:
        Y[0, T // 2, 1] = np.nan
        Y[-1, T // 3, :] = np.nan
    x0 = 0.2 * rng.standard_normal((N, L, d)) if with_x0 else None
    m.set_path(path)
    r = m.sample_posterior(Y, S, seed, x0=x0, want_states=True, want_outputs=True)
    m.set_path("auto")
    assert m.nan_status == (1 if with_nan else 0)
    Xs = m.filter_smoother_nll(Y, x0=x0, smoother_mode=1, want_nll=False)["Xs"]
    assert rel_err(r["Xs"], Xs) < TOL
    e = noise(seed, S, N, T, *_factors(m))
    assert rel_err(r["X"], r["Xs"][None] + e) < TOL
    assert np.array_equal(r["F"], r["X"][..., 0])
    assert rel_err(r["Y"], _outputs(m, r["F"])) < 1e-12


def _dlyap(G, C):
    """P = G P G' + C"""
    d = G.shape[0]
    return np.linalg.solve(np.eye(d * d) - np.kron(G, G), C.ravel()).reshape(d, d)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["Matern32", "Matern52"])
def test_sampler_factors(cuda_lib, kernel):
    """LF LF' = PF and LC LC' = C = PF - G PPc G' (PPc = A PF A' + Q) with A, Q, PF from the oracle and G its RTS gain; both
    lower-triangular.  C is a difference of terms of the size of PF, so its error is measured against PF's scale.
    The Matern-5/2 state space replicated from the reference (Pinf consistent with sqrt(5)/l, F with sqrt(3)/l) has an
    indefinite Q and hence an indefinite C: there the factor is that of C's positive semi-definite part (negative
    eigenvalues set to zero), the nearest covariance to C."""
    from oracle.binding import OracleMOIHGP
    p, L = 6, 4
    m, params, _ = _model(kernel, p, L, 3)
    o = OracleMOIHGP(0.1, p, L, kernel, True)
    o.update(params)

    def psd_part(M):
        w, V = np.linalg.eigh((M + M.T) / 2)
        return (V * np.maximum(w, 0.0)) @ V.T

    for l in range(L):
        c = o.ihgp_consts(l)
        G = o.smoother_consts(l, 1)[0]
        PF = c["PF"]
        C = PF - G @ (c["A"] @ PF @ c["A"].T + c["Q"]) @ G.T
        LF, LC = m.sampler_consts(l)
        scale = np.max(np.abs(PF))
        assert np.array_equal(LF, np.tril(LF)) and np.array_equal(LC, np.tril(LC)), l
        assert rel_err(LF @ LF.T, psd_part(PF)) < 1e-9, l
        if kernel == "Matern32":
            assert np.linalg.eigvalsh(C).min() > 0 and np.linalg.eigvalsh(PF).min() > 0, l
            assert rel_err(LF @ LF.T, PF) < 1e-12, l
            assert np.max(np.abs(LC @ LC.T - C)) < 1e-12 * scale, l
        else:
            assert np.linalg.eigvalsh((C + C.T) / 2).min() < 0, l
            assert np.max(np.abs(LC @ LC.T - psd_part(C))) < 1e-9 * scale, l


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,path", [("Matern32", "chain"), ("Matern52", "scan")])
def test_sample_moments_match_the_steady_state_covariances(cuda_lib, kernel, path):
    """2048 draws, 2 latents, moderate lengthscales: mean of x~ - Xs is 0, the covariance far from the end is P = G P G' +
    LC LC' (= Ps[1] where C is positive semi-definite, i.e. for Matern-3/2), at T-1 it is LF LF' (= PF), and the lag-one
    covariance is G P - each within 6 standard errors sqrt((P_ii P_jj + P_ij^2) / n)."""
    from oracle.gen_golden import make_data
    p, L, T, S = 3, 2, 400, 2048
    m, params, rng = _model(kernel, p, L, 5, igp=np.array([1.0, 0.6, 0.1, 1.5, 1.2, 0.05]))
    Y = make_data(rng, p, L, T)[None]
    m.set_path(path)
    r = m.sample_posterior(Y, S, 2024, want_states=True, want_outputs=False)
    m.set_path("auto")
    e = r["X"][:, 0] - r["Xs"][0][None]                           # [S, T, L, d]
    far = slice(0, T // 2)

    def within(est, ref, Pa, Pb, what):
        se = np.sqrt((np.outer(np.diag(Pa), np.diag(Pb)) + ref ** 2) / S)
        assert np.all(np.abs(est - ref) <= 6 * se), (what, est, ref)

    for l in range(L):
        G, Ps = m.smoother_consts(l, 1)
        LF, LC = m.sampler_consts(l)
        P, PF = _dlyap(G, LC @ LC.T), LF @ LF.T
        if kernel == "Matern32":
            assert rel_err(P, Ps) < 1e-10 and rel_err(PF, m.latent_consts(l)["PF"]) < 1e-12, l
        el = e[:, :, l, :]
        sd = np.sqrt(np.maximum(np.diag(P), np.diag(PF)))[None, :]
        assert np.all(np.abs(el.mean(axis=0)) <= 6 * sd / np.sqrt(S)), l
        cov_far = np.einsum("sti,stj->ij", el[:, far], el[:, far]) / (S * (T // 2))
        within(cov_far, P, P, P, ("far", l))
        within(np.einsum("si,sj->ij", el[:, -1], el[:, -1]) / S, PF, PF, PF, ("end", l))
        lag = np.einsum("sti,stj->ij", el[:, :T // 2], el[:, 1:T // 2 + 1]) / (S * (T // 2))
        within(lag, G @ P, P, P, ("lag1", l))


@pytest.mark.gpu
def test_draws_are_deterministic_and_independent_of_variant_and_sample_count(cuda_lib):
    from oracle.gen_golden import make_data
    p, L, N, T = 8, 4, 3, 700
    m, _, rng = _model("Matern52", p, L, 11)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    out = {}
    for path in ("scan", "chain"):
        m.set_path(path)
        a = m.sample_posterior(Y, 8, 42, want_states=True)
        b = m.sample_posterior(Y, 8, 42, want_states=True)
        c = m.sample_posterior(Y, 3, 42, want_states=True)
        d = m.sample_posterior(Y, 8, 43, want_states=True)
        for k in ("X", "F", "Y"):
            assert np.array_equal(a[k], b[k]), (path, k)
            assert np.array_equal(a[k][:3], c[k]), (path, k)
            assert not np.array_equal(a[k], d[k]), (path, k)
        assert np.array_equal(a["F"], a["X"][..., 0])
        assert rel_err(a["Y"], _outputs(m, a["F"])) < 1e-12
        out[path] = a
    m.set_path("auto")
    for k in ("X", "F", "Y"):
        assert rel_err(out["scan"][k], out["chain"][k]) < 1e-12, k


@pytest.mark.gpu
@pytest.mark.parametrize("path,kernel,p,L,N,T", [("chain", "Matern52", 16, 8, 160, 300), ("scan", "Matern32", 12, 5, 2, 1500)])
def test_device_sampling_right_after_update_is_capturable_in_a_cuda_graph(cuda_lib, path, kernel, p, L, N, T):
    """sample_posterior_device is asynchronous on the caller's stream: right after update(params) it can be captured into a
    CUDA graph; replays on new data equal the host-buffer call."""
    import torch
    from oracle.gen_golden import make_data, make_params
    from multioutputihgp_b200 import MOIHGPSequences
    rng = np.random.default_rng(N + T)
    dev = torch.device("cuda:0")
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    m.set_path(path)
    d, S, seed = m.igp_dim, 2, 77
    f64 = dict(dtype=torch.float64, device=dev)
    Y = torch.zeros((N, T, p), **f64)
    Xs, X, F, Ys = (torch.zeros(s, **f64) for s in ((N, T, L, d), (S, N, T, L, d), (S, N, T, L), (S, N, T, p)))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        m.update(make_params(rng, p, L, kernel))
        m.sample_posterior_device(Y, seed, Xs=Xs, X=X, F=F, Ysamp=Ys)        # warm-up on the capture stream: workspaces
        torch.cuda.synchronize()
        m.update(make_params(rng, p, L, kernel))                           # K-setup queued, nothing waits
        with torch.cuda.graph(g, stream=side):
            m.sample_posterior_device(Y, seed, Xs=Xs, X=X, F=F, Ysamp=Ys)
    for rep in range(2):
        Yh = np.stack([make_data(rng, p, L, T) for _ in range(N)])
        Y.copy_(torch.from_numpy(Yh))
        g.replay()
        torch.cuda.synchronize()
        ref = m.sample_posterior(Yh, S, seed, want_states=True)
        for k, t in (("Xs", Xs), ("X", X), ("F", F), ("Y", Ys)):
            assert rel_err(t.cpu().numpy(), ref[k]) < TOL, (rep, k)


@pytest.mark.gpu
def test_sampling_refuses_bad_requests(cuda_lib):
    import torch
    from oracle.gen_golden import make_data
    p, L, N, T = 4, 2, 1, 10
    m, _, rng = _model("Matern32", p, L, 1)
    Yh = make_data(rng, p, L, T)[None]
    with pytest.raises(RuntimeError, match="S must be positive"):
        m.sample_posterior(Yh, 0, 1)
    Y = torch.from_numpy(Yh).cuda()
    with pytest.raises(RuntimeError, match="no output requested"):
        m.sample_posterior_device(Y, 1)
    F = torch.zeros((1, N, T, L), dtype=torch.float64, device="cuda")
    big = 2 ** 32
    for n_, t_, s_ in ((big, T, 1), (N, big, 1), (N, T, big)):
        for fn in (m._lib.moihgp_cuda_sample_posterior_dev, m._lib.moihgp_cuda_sample_posterior):
            ptrs = (Y.data_ptr(), F.data_ptr()) if fn is m._lib.moihgp_cuda_sample_posterior_dev else (Yh.ctypes.data, np.empty(1).ctypes.data)
            assert fn(m._h, ptrs[0], n_, t_, None, s_, 5, None, None, ptrs[1], None) != 0
            assert "below 2^32" in m._lib.moihgp_cuda_last_error(m._h).decode()
    torch.cuda.synchronize()
