"""Carries of the chunked recursions with slowly forgetting latent processes.

Every long-sequence pass cuts a recursion with constant matrices into pieces - lanes of 8 steps, chunks of 256, groups
(16 384 steps on the chunked scan, 65 536 on the objective), super-blocks (262 144 steps), blocks of a sequence sharded in
time - and joins them with powers of the transition: AKHA^n forward, G^n backward, (AKHA^n, E_k(n)) for the objective's
sensitivities.  With the hyper-parameters of oracle/gen_golden.py every such power is below rounding (AKHA^256 <= 3e-18 at
dt = 0.1), so a wrong power, or another latent's table, changes nothing a test can see.  The tables here mix latents that
carry their state across each of these spans (l/dt up to 1e5) with fast-forgetting ones, and every test first asserts that
regime with memory(): a slow latent keeps 1e-2 <= ||M^n|| <= 1e3 over the span it stands for, a fast one ||AKHA^256|| <= 1e-12.

Two kinds of check:
  * pure carry: with Y = 0 and a non-zero x0 (dx0) every output is a linear map of the library's own matrices applied to
    x0.  It is compared step by step with the same quantity in mpmath (40 digits) at every chunk, group and super-block
    boundary +-1, the last step and 100 random steps, each step on the scale of its map (carry_err).  fp64 binary powering
    stays within 1e-11 of mpmath up to n = 5e5 on these tables, so 1e-9 leaves a margin of about 30.
  * driven parity with the CPU oracle at 1e-9: norm-wise, and within every 256-step window on that window's own scale.
The CPU part (-m "not gpu") checks the mpmath reference against the oracle and the regimes under the oracle's constants.
"""
import mpmath
import numpy as np
import pytest

from conftest import TOL, literal_smoother_err, rel_err

DT = 0.1
CH, GROUP, OBJ_GROUP, SUPER = 256, 32 * 2 * 256, 32 * 8 * 256, 16 * 32 * 2 * 256
DPS = 40

# (magnitude, lengthscale, noise) per latent, cycled over l % 5: slow, fast, slow, fast, slow.  The spans each slow entry
# stands for (which matrix, n) at dt = 0.1, with ||M^n|| under the library's constants (literal DARE iterate).
# At long lengthscales the Matern-3/2 AKHA has a complex pair of eigenvalues whose half period in steps grows like l^1.5.
# Half a period on, ||M^n|| dips to rho^n while any binary powering rounds on the scale cond(V) rho^n: at l/dt = 1e4 (half
# period 217 593 steps) fp64 powering on the CPU is 2e-8 off mpmath at n = 435 200.  That is a property of powering,
# not of a carry, so the group-level entry is l/dt = 4e4 (half period 1.7e6 steps; fp64 powering within 2.3e-10 up to 1e6).
SLOW = {
    "Matern32": [(1, 3, .1), (.5, .5, .1), (1, 4000, .1), (2, .3, .05), (1, 1e4, .1)],
    "Matern52": [(1, 2000, 10), (.5, .5, .1), (1, 5, 1.0), (.5, .3, .05), (1, 200, 10)],
}
SPANS = {
    # AKHA^256 0.63, G_rts^256 0.055 | AKHA^16384 806, AKHA^65536 383 | AKHA^262144 279
    "Matern32": {0: [("M", CH), ("G", CH)], 2: [("M", GROUP), ("M", OBJ_GROUP)], 4: [("M", SUPER)]},
    # AKHA^262144 26 (Jordan-like growth to 3e5 on the way) | AKHA^256 0.02, G_rts^256 1.9, G_rts^16384 2.2 | AKHA^16384 16
    "Matern52": {0: [("M", SUPER)], 2: [("M", CH), ("G", CH), ("G", GROUP)], 4: [("M", GROUP)]},
}
FAST = (1, 3)


# ---------------------------------------------------------------------------------------------- mpmath reference
def _mp(A):
    """float64 array -> object array of mpmath numbers (exact); an object array passes through"""
    if isinstance(A, np.ndarray) and A.dtype == object:
        return A
    return np.vectorize(mpmath.mpf, otypes=[object])(np.asarray(A, dtype=np.float64))


def _f64(A):
    return np.vectorize(float, otypes=[np.float64])(A)


def memory(M, n):
    """||M^n||_2 in mpmath (40 digits)."""
    with mpmath.workdps(DPS):
        return float(max(mpmath.svd_r(mpmath.matrix(np.asarray(M, dtype=np.float64).tolist()) ** n, compute_uv=False)))


class _Powers:
    """M^n v and the pairs (G^n, S(n)), S(n) = sum_{i<n} G^i C M^i, by binary decomposition on tables of 2^k, in mpmath."""

    def __init__(self, M, G=None, C=None, nbits=21):
        with mpmath.workdps(DPS):
            self.M, self.G, self.S = [_mp(M)], [None if G is None else _mp(G)], [None if C is None else _mp(C)]
            for _ in range(1, nbits):
                Mk, Gk, Sk = self.M[-1], self.G[-1], self.S[-1]
                if Gk is not None:
                    self.S.append(Sk + Gk.dot(Sk).dot(Mk))
                    self.G.append(Gk.dot(Gk))
                self.M.append(Mk.dot(Mk))
        self.d = self.M[0].shape[0]
        self._gaps = {}

    def apply(self, n, v):
        with mpmath.workdps(DPS):
            k = 0
            while n:
                if n & 1:
                    v = self.M[k].dot(v)
                n >>= 1
                k += 1
            return v

    def gap(self, n):
        """(G^n, S(n)):  S(a + b) = S(a) + G^a S(b) M^a"""
        if n not in self._gaps:
            with mpmath.workdps(DPS):
                I = _mp(np.eye(self.d))
                Ga, Ma, Sa = I, I, _mp(np.zeros((self.d, self.d)))
                k, m = 0, n
                while m:
                    if m & 1:
                        Sa = Sa + Ga.dot(self.S[k]).dot(Ma)
                        Ga, Ma = Ga.dot(self.G[k]), Ma.dot(self.M[k])
                    m >>= 1
                    k += 1
                self._gaps[n] = (Ga, Sa)
        return self._gaps[n]


class PureCarry:
    """What the fused pass, the per-step NLL and the objective give at Y = 0 from a carried-in state, per latent, in mpmath,
    as the linear maps from that state (so that each step can be judged on the scale of its map, see carry_err).

    Filter: X[t] = AKHA^(t+1) x0.  Literal smoother: Xs[T-1] = X[T-1], Xs[j] = G Xs[j+1] + (I - A) X[j+1].  RTS smoother:
    Xs[j] = X[j] + b[j], b[T-1] = 0, b[j] = G b[j+1] - G K HA' X[j].  Objective: x_T = AKHA^T x0, dx_T,k = AKHA^T dx0_k
    + E_k(T) x0 with E_k(n) = sum_i AKHA^(n-1-i) dAKHA_k AKHA^i (the upper right block of [[AKHA, dAKHA_k], [0, AKHA]]^n)."""

    def __init__(self, consts, G):
        """consts: latent_consts() of every latent; G: {mode: [L] smoother gains}"""
        self.c, self.G = consts, G
        self._cache = {}

    def _pw(self, l, mode):
        c = self.c[l]
        key = (mode, c["AKHA"].tobytes(), None if mode is None else self.G[mode][l].tobytes())
        if key not in self._cache:
            if mode is None:
                self._cache[key] = _Powers(c["AKHA"])
            else:
                G = self.G[mode][l]
                with mpmath.workdps(DPS):
                    C = _mp(np.eye(len(c["K"])) - c["A"]) if mode == 0 else -np.outer(_mp(G).dot(_mp(c["K"])), _mp(c["HA"]))
                self._cache[key] = _Powers(c["AKHA"], G, C)
        return self._cache[key]

    def filter(self, l, steps):
        """{t: AKHA^(t+1)}: X[t] = AKHA^(t+1) x0"""
        pw = self._pw(l, None)
        P, cur, out = _mp(np.eye(len(self.c[l]["K"]))), -1, {}
        for t in sorted(set(steps)):
            P = pw.apply(t - cur, P)
            cur = t
            out[t] = P
        return out

    def smoothed(self, l, T, steps, mode):
        """{t: W_t}: Xs[t] = W_t x0, smoother mode 0 (literal) or 1 (RTS)"""
        steps = sorted(set(steps) | {T - 1})
        X = self.filter(l, set(steps) | {t + 1 for t in steps if t + 1 < T})
        pw = self._pw(l, mode)
        d, out = len(self.c[l]["K"]), {}
        with mpmath.workdps(DPS):
            prev, b = T - 1, (X[T - 1] if mode == 0 else _mp(np.zeros((d, d))))
            for j in reversed(steps):
                if j < prev:
                    Gg, Sg = pw.gap(prev - j)
                    b = Gg.dot(b) + Sg.dot(X[j + 1] if mode == 0 else X[j])
                    prev = j
                out[j] = b if mode == 0 else X[j] + b
        return out

    def objective_end(self, l, T):
        """[3] maps [AKHA^T, E_k(T)] (d x 2d): dx_T,k = map_k [dx0_k; x0], and x_T = AKHA^T x0 = the map's left block x0"""
        c = self.c[l]
        d = len(c["K"])
        return [_Powers(np.block([[c["AKHA"], c["dAKHA%d" % k]], [np.zeros((d, d)), c["AKHA"]]])).apply(T, _mp(np.eye(2 * d)))[:d]
                for k in range(3)]


# ---------------------------------------------------------------------------------------------- regimes and metrics
def assert_regime(kernel, consts, G_rts):
    """every slow latent keeps 1e-2 <= ||M^n|| <= 1e3 over each span it stands for; every fast one ||AKHA^256|| <= 1e-12"""
    for l, c in enumerate(consts):
        r = l % len(SLOW[kernel])
        if r in FAST:
            assert memory(c["AKHA"], CH) <= 1e-12, (kernel, l)
        for which, n in SPANS[kernel].get(r, []):
            mem = memory(c["AKHA"] if which == "M" else G_rts[l], n)
            assert 1e-2 <= mem <= 1e3, (kernel, l, which, n, mem)


def steps_to_compare(T, rng, spans=(CH, GROUP, SUPER)):
    """every chunk, group and super-block boundary +-1, the first and last two steps, 100 random steps"""
    s = {0, 1, T - 2, T - 1} | set(rng.integers(0, T, 100).tolist())
    for span in spans:
        for b in range(span, T, span):
            s |= {b - 1, b, b + 1}
    return sorted(t for t in s if 0 <= t < T)


def per_step_err(got, ref, scale=None):
    """worst relative error of got [K, d] against ref [K, d], every row on its own scale (its norm, or scale [K]); rows whose
    scale is below 1e-200 (a fast latent long after it forgot x0) must be below 1e-190"""
    nr = np.linalg.norm(ref, axis=-1) if scale is None else np.asarray(scale)
    live = nr > 1e-200
    assert np.all(np.linalg.norm(got[~live], axis=-1) <= 1e-190)
    return float(np.max(np.linalg.norm(got - ref, axis=-1)[live] / nr[live])) if live.any() else 0.0


def carry_err(got, maps, v):
    """worst relative error of got [K, d] against maps [K] (mpmath, d x d') applied to the carried-in v [d'], every step on
    the scale of its map, ||W_t||_F ||v||: the size the carried state can have at step t, whichever v the test drew."""
    with mpmath.workdps(DPS):
        vm = _mp(v)
        ref = _f64(np.array([W.dot(vm) for W in maps]))
    Wn = np.array([np.linalg.norm(_f64(W)) for W in maps])
    return per_step_err(got, ref, Wn * np.linalg.norm(v))


def window_err(a, b, latents=None, scale=None):
    """worst relative error of a against b [N, T, L, d] within each 256-step window and latent, on that window's own maximum
    (or on the window's maximum of |scale| [N, T, L, d], if larger)"""
    a, b = np.asarray(a), np.asarray(b)
    N, T, L, d = b.shape
    W = -(-T // CH)
    pad = lambda x: np.concatenate([x, np.zeros((N, W * CH - T, L, d))], axis=1).reshape(N, W, CH, L, d)
    with np.errstate(invalid="ignore"):                 # inf - inf in a literal-smoother latent that diverges (not selected)
        diff = np.max(np.abs(pad(a - b)), axis=(0, 2, 4))
    scale = np.max(np.abs(pad(b if scale is None else np.maximum(np.abs(b), np.abs(scale)))), axis=(0, 2, 4))
    sel = np.zeros((W, L), dtype=bool)
    sel[:, list(range(L)) if latents is None else list(latents)] = True
    live = sel & (scale > 1e-200)
    assert np.all(diff[sel & ~live] <= 1e-190)
    return float(np.max(diff[live] / scale[live]))


def literal_ok(G_lit):
    """latents whose literal smoother gain has rho < 1 (the others diverge in the reference too, SURVEY Q3)"""
    return [l for l, G in enumerate(G_lit) if np.max(np.abs(np.linalg.eigvals(G))) < 1]


def _params(kernel, p, L, seed):
    from oracle.gen_golden import make_params
    rng = np.random.default_rng(seed)
    return make_params(rng, p, L, kernel, SLOW), rng


def _oracle(kernel, p, L, params):
    from oracle.binding import OracleMOIHGP
    o = OracleMOIHGP(DT, p, L, kernel, True)
    o.update(params)
    return o


def _device_model(kernel, p, L, seed):
    """(model, oracle, params, rng, consts, gains {mode: [L]}) after checking the device constants, DARE iteration counts
    and smoother gains against the oracle's and the regime of every latent"""
    from multioutputihgp_b200 import MOIHGPSequences
    params, rng = _params(kernel, p, L, seed)
    m = MOIHGPSequences(DT, p, L, kernel, True)
    m.update(params)
    o = _oracle(kernel, p, L, params)
    consts = [m.latent_consts(l) for l in range(L)]
    for l in range(L):
        assert m.latent_iters(l) == o.ihgp_iters(l), l
        for k, v in o.ihgp_consts(l).items():
            v = np.asarray(v)
            if np.max(np.abs(v)) > 0:
                assert rel_err(np.asarray(consts[l][k]), v) < TOL, (l, k)
            else:
                assert np.max(np.abs(consts[l][k])) == 0, (l, k)
    G = {mode: [m.smoother_consts(l, mode)[0] for l in range(L)] for mode in (0, 1)}
    for mode in (0, 1):
        for l in range(L):
            assert rel_err(G[mode][l], o.smoother_consts(l, mode)[0]) < TOL, (mode, l)
    assert_regime(kernel, consts, G[1])
    return m, o, params, rng, consts, G


def _nll_term(c, x):
    """the carry-dependent part of one step's NLL at y = 0 for one latent: (HA . x)^2 / (2 S)"""
    with mpmath.workdps(DPS):
        v = _mp(c["HA"]).dot(x)
        return v * v / (2 * mpmath.mpf(c["S"]))


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("kernel", ["Matern32", "Matern52"])
def test_tables_reach_their_regimes_under_the_oracle_constants(kernel):
    L = len(SLOW[kernel])
    params, _ = _params(kernel, L, L, 1)
    o = _oracle(kernel, L, L, params)
    assert_regime(kernel, [o.ihgp_consts(l) for l in range(L)], [o.smoother_consts(l, 1)[0] for l in range(L)])
    # the same check fails on the tables every other test uses
    from oracle.gen_golden import TABLE, make_params
    o.update(make_params(np.random.default_rng(1), L, L, kernel, TABLE))
    with pytest.raises(AssertionError):
        assert_regime(kernel, [o.ihgp_consts(l) for l in range(L)], [o.smoother_consts(l, 1)[0] for l in range(L)])


@pytest.mark.parametrize("kernel", ["Matern32", "Matern52"])
def test_mpmath_propagation_equals_the_oracle_at_zero_observations(kernel):
    """PureCarry against the oracle's sequential fp64 loops at Y = 0: filtered and smoothed states of every step in both
    modes, the per-step NLL terms and the objective's final state and sensitivities (T = 700, three chunks)."""
    L, T = len(SLOW[kernel]), 700
    params, rng = _params(kernel, L, L, 2)
    o = _oracle(kernel, L, L, params)
    consts = [o.ihgp_consts(l) for l in range(L)]
    G = {mode: [o.smoother_consts(l, mode)[0] for l in range(L)] for mode in (0, 1)}
    ref = PureCarry(consts, G)
    d = o.d
    x0 = 0.3 * rng.standard_normal((L, d))
    dx0 = 0.1 * rng.standard_normal((L, 3, d))
    Y = np.zeros((1, T, L))
    steps = list(range(T))
    for mode in (0, 1):
        r = o.filter_smoother_nll(Y, x0=x0[None], smoother_mode=mode)
        for l in range(L):
            X = ref.filter(l, steps)                                   # pins the index convention X[t] = AKHA^(t+1) x0
            assert carry_err(r["X"][0, :, l], [X[t] for t in steps], x0[l]) < 1e-12, (mode, l)
            if mode == 1 or l in literal_ok(G[0]):
                Xs = ref.smoothed(l, T, steps, mode)
                assert carry_err(r["Xs"][0, :, l], [Xs[t] for t in steps], x0[l]) < 1e-11, (mode, l)
    # step t's NLL term is evaluated on the state before the step, X[t-1] (x0 at t = 0)
    const = o.negLogLikelihood(np.zeros((L, d)), np.zeros(L))
    for t in (0, 1, 255, 256, 699):
        x_prev = np.stack([x0[l] if t == 0 else _f64(ref.filter(l, [t - 1])[t - 1].dot(_mp(x0[l]))) for l in range(L)])
        got = o.negLogLikelihood(x_prev, np.zeros(L)) - const
        want = float(sum(_nll_term(consts[l], _mp(x_prev[l])) for l in range(L)))
        assert abs(got - want) <= 1e-12 * abs(want) + 1e-14 * abs(const), t
    _, _, xT, dxT = o.objective(Y, x0=x0[None], dx0=dx0[None])
    for l in range(L):
        U = ref.objective_end(l, T)
        assert carry_err(xT[0, l][None], [U[0][:, :d]], x0[l]) < 1e-12, l
        for k in range(3):
            assert carry_err(dxT[0, l, k][None], [U[k]], np.concatenate([dx0[l, k], x0[l]])) < 1e-11, (l, k)


# ---------------------------------------------------------------------------------------------------------------- GPU
LONG = 2 * SUPER + GROUP + 37            # two super-blocks, a group and a ragged last chunk
MID = 3 * GROUP + 5 * CH + 37            # three groups, five chunks and a ragged last chunk
OBJ_T = 2 * OBJ_GROUP + 3 * CH + 37      # two objective groups and a ragged last chunk


def _profiled(m, fn):
    m.profile(True)
    out = fn()
    prof = m.profile_read()
    m.profile(False)
    return out, prof


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,L,T", [("Matern32", 5, LONG), ("Matern52", 8, LONG), ("Matern32", 8, MID), ("Matern52", 5, MID)])
def test_pure_carry_of_the_chunked_scan_and_its_nll_steps(cuda_lib, kernel, L, T):
    """Y = 0, one sequence, carried-in x0: filtered and smoothed states of the chunked-scan pass (final kernel k_scan_lanes
    for L % 8 == 0, k_scan otherwise; both smoother modes) and the per-step NLL terms against PureCarry, every compared step
    on the scale of its map.  Worst error on a B200 (1000 W power limit) over T = 540 709 steps: 4.8e-11 (Matern-3/2),
    3.1e-11 (Matern-5/2); the objective's x_T and dx_T there: 2.6e-11."""
    m, o, params, rng, consts, G = _device_model(kernel, L, L, T + L)
    d = m.igp_dim
    x0 = 0.3 * rng.standard_normal((1, L, d))
    Y = np.zeros((1, T, L))
    steps = steps_to_compare(T, rng)
    ref = PureCarry(consts, G)
    m.set_path("scan")
    worst = {}
    for mode in (1, 0):
        r, prof = _profiled(m, lambda: m.filter_smoother_nll(Y, x0=x0, smoother_mode=mode))
        assert {"k_scan_summaries", "k_response", "k_carry", "k_scan_final"} <= set(prof), sorted(prof)
        for l in range(L):
            if mode == 1:
                X = ref.filter(l, steps)
                worst["X", l] = carry_err(r["X"][0, steps, l], [X[t] for t in steps], x0[0, l])
            if mode == 1 or l in literal_ok(G[0]):
                Xs = ref.smoothed(l, T, steps, mode)
                worst["Xs%d" % mode, l] = carry_err(r["Xs"][0, steps, l], [Xs[t] for t in steps], x0[0, l])
    r, prof = _profiled(m, lambda: m.nll_steps(Y, x0=x0))
    assert "k_nll_steps" in prof and "k_carry" in prof, sorted(prof)
    const = m.nll_steps(Y)["nll_steps"][0, 0]                      # x0 = 0: every step is the constant part alone
    prev = {l: ref.filter(l, [t - 1 for t in steps if t > 0]) for l in range(L)}
    for t in steps:
        want = float(sum(_nll_term(consts[l], _mp(x0[0, l]) if t == 0 else prev[l][t - 1].dot(_mp(x0[0, l]))) for l in range(L)))
        got = r["nll_steps"][0, t] - const
        assert abs(got - want) <= TOL * abs(want) + 1e-14 * abs(const), (t, got, want)
    print("pure carry %s L=%d T=%d: worst per-step error %.2e (%s)" % (kernel, L, T, max(worst.values()), max(worst, key=worst.get)))
    assert max(worst.values()) < TOL, worst


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,L,T", [("Matern32", 8, OBJ_T), ("Matern32", 5, OBJ_T), ("Matern52", 8, LONG), ("Matern52", 5, OBJ_T)])
def test_pure_carry_of_the_objective(cuda_lib, kernel, L, T):
    """Y = 0 with carried-in x0 and dx0: the objective's final state x_T = AKHA^T x0 and sensitivities
    dx_T,k = AKHA^T dx0_k + E_k(T) x0 (k_obj_lanes for L % 8 == 0, k_obj_scan otherwise) against mpmath, every latent and k
    on the scale of its map."""
    m, o, params, rng, consts, G = _device_model(kernel, L, L, T + 2 * L)
    d = m.igp_dim
    x0 = 0.3 * rng.standard_normal((1, L, d))
    dx0 = 0.1 * rng.standard_normal((1, L, 3, d))
    (loss, grad, xT, dxT), prof = _profiled(m, lambda: m.objective(np.zeros((1, T, L)), x0=x0, dx0=dx0, want_state=True))
    assert {"k_obj_scan_summaries", "k_obj_carry", "k_obj_scan_final"} <= set(prof), sorted(prof)
    ref = PureCarry(consts, G)
    worst = 0.0
    for l in range(L):
        U = ref.objective_end(l, T)
        worst = max(worst, carry_err(xT[0, l][None], [U[0][:, :d]], x0[0, l]))
        for k in range(3):
            worst = max(worst, carry_err(dxT[0, l, k][None], [U[k]], np.concatenate([dx0[0, l, k], x0[0, l]])))
    print("pure carry objective %s L=%d T=%d: worst error %.2e" % (kernel, L, T, worst))
    assert worst < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L,N,T", [("Matern32", 8, 8, 2, MID), ("Matern52", 6, 5, 2, MID), ("Matern52", 8, 8, 1, LONG),
                                            ("Matern32", 5, 5, 1, LONG)])
def test_driven_chunked_scan_matches_the_oracle(cuda_lib, kernel, p, L, N, T):
    """make_data inputs, carried-in x0, both final kernels and both smoother modes against the oracle: norm-wise and within
    every 256-step window.  Literal mode: the latents whose gain is stable (the others through literal_smoother_err), each
    window on the scale of the filtered states as well: that smoother forms Xs from (I - A) X, so with A close to I
    (l/dt = 2e4) Xs lies 3-4 orders below X and carries X's rounding in absolute terms, in the reference's recursion too."""
    from oracle.gen_golden import make_data
    m, o, params, rng, consts, G = _device_model(kernel, p, L, T + p)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    x0 = 0.3 * rng.standard_normal((N, L, m.igp_dim))
    m.set_path("scan")
    for mode in (1, 0):
        r, prof = _profiled(m, lambda: m.filter_smoother_nll(Y, x0=x0, smoother_mode=mode))
        assert {"k_carry", "k_scan_final"} <= set(prof) and "k_filter_chain" not in prof, sorted(prof)
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, nthreads=8)
        for k in ("X", "nll", "xT"):
            assert rel_err(r[k], ro[k]) < TOL, (k, mode)
        assert window_err(r["X"], ro["X"]) < TOL, mode
        if mode == 1:
            assert rel_err(r["Xs"], ro["Xs"]) < TOL and window_err(r["Xs"], ro["Xs"]) < TOL
        else:
            err, n = literal_smoother_err(r["Xs"], ro["Xs"])
            assert err < TOL and n >= 100, (err, n)
            assert window_err(r["Xs"], ro["Xs"], literal_ok(G[0]), scale=ro["X"]) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L", [("Matern32", 8, 4), ("Matern52", 16, 8)])
def test_driven_many_chains_path_matches_the_oracle_and_the_scan(cuda_lib, kernel, p, L):
    """The many-chains path (one pass per sequence, no chunk carries) on the same tables: against the oracle and against the
    chunked scan, both modes."""
    from oracle.gen_golden import make_data
    N, T = 4, GROUP + 3 * CH + 5
    m, o, params, rng, consts, G = _device_model(kernel, p, L, 77 + L)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    x0 = 0.3 * rng.standard_normal((N, L, m.igp_dim))
    for mode in (1, 0):
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, nthreads=8)
        out = {}
        for path, kname in (("chain", "k_filter_chain"), ("scan", "k_scan_final")):
            m.set_path(path)
            out[path], prof = _profiled(m, lambda: m.filter_smoother_nll(Y, x0=x0, smoother_mode=mode))
            assert kname in prof, (path, sorted(prof))
            assert rel_err(out[path]["X"], ro["X"]) < TOL and window_err(out[path]["X"], ro["X"]) < TOL, (path, mode)
            assert rel_err(out[path]["nll"], ro["nll"]) < TOL, (path, mode)
            ok, sc = (list(range(L)), None) if mode == 1 else (literal_ok(G[0]), ro["X"])
            assert window_err(out[path]["Xs"], ro["Xs"], ok, sc) < TOL, (path, mode)
        assert window_err(out["chain"]["X"], out["scan"]["X"]) < 1e-11, mode
        assert window_err(out["chain"]["Xs"], out["scan"]["Xs"], ok, sc) < 1e-11, mode


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L,N,T", [("Matern32", 8, 8, 1, OBJ_T), ("Matern32", 6, 5, 2, OBJ_T), ("Matern52", 8, 8, 1, OBJ_T)])
def test_driven_objective_matches_the_oracle(cuda_lib, kernel, p, L, N, T):
    """Loss, every gradient block on its own scale, x_T and dx_T from carried-in x0 / dx0 over two objective groups and a
    ragged chunk (k_obj_lanes for L % 8 == 0, k_obj_scan otherwise)."""
    from oracle.gen_golden import make_data
    m, o, params, rng, consts, G = _device_model(kernel, p, L, T + 3 * p)
    d = m.igp_dim
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    x0 = 0.3 * rng.standard_normal((N, L, d))
    dx0 = 0.1 * rng.standard_normal((N, L, 3, d))
    (loss, grad, xT, dxT), prof = _profiled(m, lambda: m.objective(Y, x0=x0, dx0=dx0, want_state=True))
    assert {"k_obj_carry", "k_obj_scan_final"} <= set(prof), sorted(prof)
    lo, go, xo, dxo = o.objective(Y, x0=x0, dx0=dx0)
    assert abs(loss - lo) <= TOL * abs(lo)
    pL = p * L
    for sl in [slice(0, pL), slice(pL, pL + L), slice(pL + L, pL + L + 1)] + [slice(pL + L + 1 + 3 * l, pL + L + 4 + 3 * l) for l in range(L)]:
        assert rel_err(grad[sl], go[sl]) < TOL, sl
    for l in range(L):
        assert rel_err(xT[:, l], xo[:, l]) < TOL and rel_err(dxT[:, l], dxo[:, l]) < TOL, l


@pytest.mark.gpu
def test_objective_blocks_with_long_cuts_match_the_oracle(cuda_lib):
    """objective_begin_async / carry_in_device / objective_finish_device over blocks of 16 384 and 32 768 steps, across
    which the group-level latent keeps its state: the carry-ins equal the whole-sequence states at the cuts, and the blocks'
    [loss, grad] add up to the oracle's."""
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_data
    kernel, p, L, N = "Matern32", 6, 5, 1
    cuts = (0, GROUP, 3 * GROUP, 3 * GROUP + 4 * CH, 3 * GROUP + 4 * CH + 999)
    T, Gn = cuts[-1], len(cuts) - 1
    lengths = [cuts[g + 1] - cuts[g] for g in range(Gn)]
    whole, o, params, rng, consts, G = _device_model(kernel, p, L, 4242)
    assert max(memory(c["AKHA"], n) for c in consts for n in lengths[:-1]) >= 1e-2
    d = whole.igp_dim
    dev = torch.device("cuda:0")
    f64 = dict(dtype=torch.float64, device=dev)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    x0, dx0 = 0.2 * rng.standard_normal((N, L, d)), 0.1 * rng.standard_normal((N, L, 3, d))
    models = []
    for g in range(Gn):
        mg = MOIHGPSequences(DT, p, L, kernel, True)
        mg.update(params)
        models.append(mg)
    Yd = [torch.from_numpy(np.ascontiguousarray(Y[:, cuts[g]:cuts[g + 1]])).to(dev) for g in range(Gn)]
    ends = torch.zeros((Gn, N, L, 4, d), **f64)
    for g in range(Gn):
        models[g].objective_begin_async(Yd[g], None if g == Gn - 1 else ends[g])
    out = torch.zeros((Gn, 2 + whole.num_param), **f64)
    xin, dxin = torch.zeros((Gn, N, L, d), **f64), torch.zeros((Gn, N, L, 3, d), **f64)
    for g in range(Gn):
        models[g].carry_in_device(ends, lengths, g, xin[g], dxin[g], x0=torch.from_numpy(x0).to(dev), dx0=torch.from_numpy(dx0).to(dev))
        models[g].objective_finish_device(Yd[g], out[g, 0:1], out[g, 2:], x0=xin[g], dx0=dxin[g])
    torch.cuda.synchronize()
    for g in range(1, Gn):
        _, _, xo, dxo = o.objective(Y[:, :cuts[g]], x0=x0, dx0=dx0)
        for l in range(L):
            assert rel_err(xin[g, :, l].cpu().numpy(), xo[:, l]) < TOL and rel_err(dxin[g, :, l].cpu().numpy(), dxo[:, l]) < TOL, (g, l)
    lo, go, _, _ = o.objective(Y, x0=x0, dx0=dx0)
    tot = out.sum(0).cpu().numpy()
    assert abs(tot[0] - lo) <= TOL * abs(lo) and rel_err(tot[2:], go) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,p,L,N", [("Matern52", 6, 5, 2), ("Matern32", 8, 8, 1)])
def test_time_sharded_fused_pass_with_long_blocks_matches_the_oracle(cuda_lib, kernel, p, L, N):
    """fsn_block_async / fsn_carry_device over four blocks of whole chunks, thousands of steps long, that slow latents cross
    forwards (AKHA) and, for Matern-5/2, backwards (the RTS gain): X, Xs, NLL against the oracle's whole-sequence pass."""
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_data
    cuts = (0, 16 * CH, 48 * CH, 64 * CH, 64 * CH + 777)
    T, Gn = cuts[-1], len(cuts) - 1
    lengths = [cuts[g + 1] - cuts[g] for g in range(Gn)]
    whole, o, params, rng, consts, G = _device_model(kernel, p, L, 99 + L)
    for n in lengths[:-1]:
        assert max(memory(c["AKHA"], n) for c in consts) >= 1e-2, n
        if kernel == "Matern52":
            assert max(memory(g_, n) for g_ in G[1]) >= 1e-2, n
    d = whole.igp_dim
    dev = torch.device("cuda:0")
    f64 = dict(dtype=torch.float64, device=dev)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    x0 = 0.3 * rng.standard_normal((N, L, d))
    models = []
    for g in range(Gn):
        mg = MOIHGPSequences(DT, p, L, kernel, True)
        mg.update(params)
        models.append(mg)
    Yd = [torch.from_numpy(np.ascontiguousarray(Y[:, cuts[g]:cuts[g + 1]])).to(dev) for g in range(Gn)]
    x0d = torch.from_numpy(x0).to(dev)
    for mode in (1, 0):
        g1, g2 = torch.zeros((Gn, N, L, d + 1), **f64), torch.zeros((Gn, N, L, d), **f64)
        xin, uaf, bend = torch.zeros((Gn, N, L, d), **f64), torch.zeros((Gn, N, L), **f64), torch.zeros((Gn, N, L, d), **f64)
        for g in range(Gn):
            models[g].fsn_block_async(1, Yd[g], g == Gn - 1, mode, out=g1[g])
        for g in range(Gn):
            models[g].fsn_carry_device(0, g1, lengths, g, xin[g], mode, x0=x0d, u_after=uaf[g])
            models[g].fsn_block_async(2, Yd[g], g == Gn - 1, mode, x0=xin[g], u_after=None if g == Gn - 1 else uaf[g], out=g2[g])
        X = [torch.zeros((N, lengths[g], L, d), **f64) for g in range(Gn)]
        Xs = [torch.zeros_like(X[g]) for g in range(Gn)]
        nll = torch.zeros((Gn, N), **f64)
        for g in range(Gn):
            models[g].fsn_carry_device(1, g2, lengths, g, bend[g], mode)
            models[g].fsn_block_async(3, Yd[g], g == Gn - 1, mode, x0=xin[g], u_after=None if g == Gn - 1 else uaf[g],
                                      b_end=None if g == Gn - 1 else bend[g], X=X[g], Xs=Xs[g], nll=nll[g])
        torch.cuda.synchronize()
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, nthreads=8)
        Xc = np.concatenate([x.cpu().numpy() for x in X], axis=1)
        Xsc = np.concatenate([x.cpu().numpy() for x in Xs], axis=1)
        assert rel_err(Xc, ro["X"]) < TOL and window_err(Xc, ro["X"]) < TOL, mode
        assert rel_err(nll.sum(0).cpu().numpy(), ro["nll"]) < TOL, mode
        assert (window_err(Xsc, ro["Xs"]) if mode == 1 else window_err(Xsc, ro["Xs"], literal_ok(G[0]), ro["X"])) < TOL, mode


@pytest.mark.gpu
def test_time_chunked_sampler_with_a_slow_rts_gain(cuda_lib):
    """The time-chunked sampler (set_path('scan')) where the RTS gain keeps the noise across chunks (G_rts^256 = 1.9): the
    draws equal the RTS mean plus the noise recomputed by the sequential NumPy recursion of test_gpu_sampling, and
    sample_block_async over three blocks equals the whole-sequence draw."""
    import torch
    from test_gpu_sampling import _factors, noise
    from oracle.gen_golden import make_data
    kernel, p, L, N, S, T = "Matern52", 6, 5, 1, 2, 12 * CH + 33
    m, o, params, rng, consts, G = _device_model(kernel, p, L, 555)
    seed = 0x5EED_1234
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    m.set_path("scan")
    r, prof = _profiled(m, lambda: m.sample_posterior(Y, S, seed, want_states=True, want_outputs=False))
    assert "k_sample_carry" in prof and "k_sample_final" in prof, sorted(prof)
    ro = o.filter_smoother_nll(Y, smoother_mode=1)
    assert window_err(r["Xs"], ro["Xs"]) < TOL
    e = noise(seed, S, N, T, *_factors(m))
    for s in range(S):
        assert window_err(r["X"][s] - r["Xs"], e[s]) < TOL, s
    # three blocks of the same draw (each block on its own handle, as on its own GPU)
    from test_gpu_time_sharded_sampling import _sharded
    from multioutputihgp_b200 import MOIHGPSequences
    cuts = (0, 4 * CH, 8 * CH, T)
    models = []
    for _ in range(len(cuts) - 1):
        mg = MOIHGPSequences(DT, p, L, kernel, True)
        mg.update(params)
        mg.set_path("scan")
        models.append(mg)
    Xs = torch.from_numpy(r["Xs"]).cuda()
    got = _sharded(models, Xs, cuts, S, seed)
    torch.cuda.synchronize()
    assert window_err(got["X"].cpu().numpy().reshape(S * N, T, L, -1), r["X"].reshape(S * N, T, L, -1)) < TOL
