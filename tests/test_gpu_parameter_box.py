"""The steady-state setup (k_setup) and every pass built on it, across the box the optimisers search and at sampling
intervals other than dt = 0.1.

The learners and scripts/fit_lbfgs.py search S in [1e-4, 1e4] and sigma, magnitude, lengthscale, noise in [1e-4, 1e2]
(learners.hpp, moihgp_regression.h); every other test uses dt = 0.1 and hyper-parameters near one.  REGIMES below names,
per kernel, the points of that box (and dt in {1e-3, 0.1, 0.37, 1, 10}) where k_setup takes another branch:
  * the scaling-and-squaring expm with 0, 1, 2 and several squarings, on both sides of each threshold 5.3719 * 2^k, for
    dt F and - separately, it has its own norm - for the 2d x 2d block dt [F 0; dF F] behind dA of the lengthscale;
  * a DARE that converges in a few iterations, one capped at 100, one that stops after its first iterate; DLyaps of one
    latent that stop after one iterate and at the cap;
  * gains near 1 (noise 1e-4: PF nearly singular) and near 0, magnitude and noise at both bounds.
The CPU part (-m "not gpu") asserts every regime an entry claims from the oracle's own numbers (squarings from the
1-norms, iteration counts and convergence flags, gain, PF conditioning) and sorts each entry into one of three classes:
  * ill-posed: stiff points where the oracle's A or block exponential is more than 1e-12 off mpmath (50 digits, on its
    own scale), and points where a constant, the filter, the NLL or the objective over PASS_T steps is not finite.  There
    is no defined answer to be bit-compatible with (cf. DESIGN 4.6): no GPU test runs there.
  * unbounded: the constants are well defined, but the steady-state filter (rho(AKHA) >= 1) or the RTS smoother
    (rho(G_rts) >= 1) does not forget, so states or smoothed states grow like rho^t and a long enough pass overflows in
    the reference too.  The GPU tests of the constants, the power tables and the sampler factors run there; the passes
    do not.
  * bounded: every GPU test, including the passes on models whose latents each sit in another regime.
Every GPU comparison is against the oracle at 1e-9, each latent, field and gradient block on its own scale.
"""
from collections import namedtuple

import mpmath
import numpy as np
import pytest

from conftest import TOL, rel_err

THETA = 5.371920351148152          # Higham's theta_13: expm scales dt F down to a 1-norm <= THETA
DPS = 50
CAP = 100                          # dare.h:8

Entry = namedtuple("Entry", "name kernel dt mag ls noise sq dare dlyap gain pf ill unbounded")


def E(name, kernel, dt, mag, ls, noise, sq, dare, dlyap, gain=None, pf=None, ill=None, unbounded=None):
    """sq: squarings of (dt F, the lengthscale block); dare / dlyap: iteration class ('one', 'few' <= 30, 'many' < 100,
    'cap' = stopped at 100 unconverged) of the DARE and of the three hyper-parameters' DLyaps; gain: K[0] near '1' or
    '0'; pf: 'near-singular' (PF's eigenvalue ratio below 1e-4); ill: why the entry is ill-posed; unbounded: which
    recursion does not forget (see the module docstring)."""
    return Entry(name, kernel, dt, mag, ls, noise, sq, dare, dlyap, gain, pf, ill, unbounded)


M32, M52 = "Matern32", "Matern52"
CAPPED = ("cap", "cap", "cap")
REGIMES = [
    # ---- Matern-3/2
    E("m32_suite", M32, 0.1, 1, 1, .1, (0, 0), "few", CAPPED),
    E("m32_A0_below", M32, 1, 1, .833, .1, (0, 2), "few", CAPPED),                  # ||dt F||_1 = 5.16
    E("m32_A0_above", M32, 1, 1, .755, .1, (1, 2), "few", CAPPED),                  # 5.59
    E("m32_A1_below", M32, 1, 1, .539, .1, (1, 4), "few", CAPPED),                  # 10.3
    E("m32_A1_above", M32, 1, 1, .518, .1, (2, 4), "few", CAPPED),                  # 11.2
    E("m32_A2_below", M32, 1, 1, .381, .1, (2, 5), "few", CAPPED),                  # 20.7
    E("m32_A2_above", M32, 1, 1, .366, .1, (3, 5), "few", CAPPED),                  # 22.4
    E("m32_B0_below", M32, 1, 1, 1.42, .1, (0, 0), "few", CAPPED),                  # block 5.16
    E("m32_B0_above", M32, 1, 1, 1.33, .1, (0, 1), "few", CAPPED),                  # block 5.56: only the block squares
    E("m32_B1_below", M32, 1, 1, .95, .1, (0, 1), "few", CAPPED),                   # block 10.3
    E("m32_B1_above", M32, 1, 1, .922, .1, (0, 2), "few", CAPPED),                  # block 11.2
    E("m32_B2_below", M32, 1, 1, .735, .1, (1, 2), "few", CAPPED),                  # block 20.7
    E("m32_B2_above", M32, 1, 1, .714, .1, (1, 3), "few", CAPPED),                  # block 22.4
    E("m32_dt10", M32, 10, 1, 1, .1, (4, 5), "one", ("one", "few", "one")),
    E("m32_dt10_noise_hi", M32, 10, 1, 5, 100, (2, 2), "few", CAPPED),
    E("m32_dt10_gain1", M32, 10, 100, 1, 1e-4, (4, 5), "one", ("one", "few", "one"), gain="1", pf="near-singular"),
    E("m32_dt1e-3", M32, 1e-3, 1, 1, .1, (0, 0), "cap", ("few", "few", "few"),
      unbounded="the DARE stops at the cap on an iterate whose AKHA has spectral radius 1.0039"),
    E("m32_ls_hi", M32, 0.1, 1, 100, .1, (0, 0), "cap", ("one", "one", "one"), gain="0"),
    E("m32_noise_lo", M32, 0.1, 1, 1, 1e-4, (0, 0), "few", CAPPED, gain="1", pf="near-singular"),
    E("m32_noise_hi", M32, 0.1, 1, 1, 100, (0, 0), "many", ("few", "few", "few")),
    E("m32_mag_lo", M32, 0.37, 1e-4, 1, .1, (0, 0), "few", ("many", "many", "many")),
    E("m32_mag_hi", M32, 0.37, 100, 1, .1, (0, 0), "few", CAPPED, gain="1"),
    E("m32_pf_singular", M32, 0.37, 100, .1, 1e-4, (5, 9), "few", CAPPED, gain="1", pf="near-singular"),
    E("m32_mixed_dlyap", M32, 1, 1e-4, 1, 100, (0, 1), "few", ("cap", "cap", "one"), gain="0"),
    E("m32_stiff", M32, 1, 1, .01, .1, (13, 21), "one", ("one", "few", "one"),
      ill="stiff (||dt F||_1 = 3e4): the oracle's A is 2e-9 off exp(dt F), its block 3e-3"),
    E("m32_overflow", M32, 10, 1, 100, .1, (1, 1), "many", CAPPED,
      ill="the capped DLyap iterates grow without bound: the objective's gradient overflows"),
    # ---- Matern-5/2
    E("m52_suite", M52, 0.1, 1, 1, .1, (0, 0), "cap", CAPPED),
    E("m52_A0_below", M52, 1, 1, 1.47, .1, (0, 2), "cap", CAPPED),                  # ||dt F||_1 = 5.17
    E("m52_A0_above", M52, 1, 1, 1.4, .1, (1, 2), "cap", CAPPED),                   # 5.59
    E("m52_A1_below", M52, 1, 1, .983, .1, (1, 3), "few", CAPPED),                  # 10.3
    E("m52_A1_above", M52, 1, 1, .941, .1, (2, 4), "few", CAPPED),                  # 11.2
    E("m52_A2_below", M52, 1, 1, .677, .1, (2, 6), "few", CAPPED),                  # 20.6
    E("m52_A2_above", M52, 1, 1, .649, .1, (3, 6), "few", CAPPED),                  # 22.4
    E("m52_B0_below", M52, 1, 1, 2.3, .1, (0, 0), "cap", CAPPED,                    # block 5.17
      unbounded="the RTS gain has spectral radius 1.085"),
    E("m52_B0_above", M52, 1, 1, 2.22, 1, (0, 1), "few", ("cap", "cap", "many"),    # block 5.57: only the block squares
      unbounded="the RTS gain has spectral radius 6.65: smoothed states overflow within 700 steps"),
    E("m52_B0_below_037", M52, 0.37, 1, 1.5, .1, (0, 0), "cap", CAPPED),            # block 5.14
    E("m52_B0_above_037", M52, 0.37, 1, 1.45, .1, (0, 1), "cap", CAPPED),           # block 5.60: only the block squares
    E("m52_B1_below", M52, 1, 1, 1.69, 1, (0, 1), "few", CAPPED),                   # block 10.4
    E("m52_B1_above", M52, 1, 1, 1.64, .1, (0, 2), "cap", CAPPED),                  # block 11.1
    E("m52_B2_below", M52, 1, 1, 1.28, 1, (1, 2), "few", CAPPED),                   # block 20.8
    E("m52_B2_above", M52, 1, 1, 1.25, 1, (1, 3), "few", CAPPED),                   # block 22.1
    E("m52_dt10", M52, 10, 1, 1, .1, (5, 7), "one", ("cap", "cap", "one")),
    E("m52_dt10_gain1", M52, 10, 100, 1, 1e-4, (5, 7), "few", ("cap", "cap", "one"), gain="1", pf="near-singular"),
    E("m52_dt10_ls2", M52, 10, 100, 2, 1e-4, (3, 4), "few", CAPPED, gain="1", pf="near-singular"),
    E("m52_dt1e-3", M52, 1e-3, 1, 1, .1, (0, 0), "cap", ("few", "few", "few")),
    E("m52_ls_hi", M52, 0.1, 1, 100, 100, (0, 0), "one", ("one", "one", "one"), gain="0"),
    E("m52_dt037", M52, 0.37, 1, 1, .1, (0, 2), "cap", CAPPED),
    E("m52_noise_lo", M52, 0.1, 1, 1, 1e-4, (0, 0), "cap", CAPPED, gain="1", pf="near-singular"),
    E("m52_noise_hi", M52, 0.1, 1, 1, 100, (0, 0), "cap", ("many", "many", "few")),
    E("m52_mag_lo", M52, 0.37, 1e-4, 1, .1, (0, 2), "few", ("cap", "cap", "many")),
    E("m52_mag_hi", M52, 0.37, 100, 1, .1, (0, 2), "cap", CAPPED, gain="1", pf="near-singular"),
    E("m52_pf_singular", M52, 1, 100, 1, 1e-4, (1, 3), "few", CAPPED, gain="1", pf="near-singular"),
    E("m52_mixed_dlyap", M52, 1, 1e-4, 1, 100, (1, 3), "few", ("cap", "cap", "one"), gain="0"),
    E("m52_stiff", M52, 0.1, 1, .01, .1, (17, 26), "few", CAPPED, gain="1",
      ill="stiff (||dt F||_1 = 5e5): the oracle's A is 6e-8 off exp(dt F), its block 3e-2"),
    E("m52_ls_lo", M52, 0.1, 1, 1e-4, .1, (37, 53), "one", ("cap", "cap", "one"),
      ill="stiff (||dt F||_1 = 5e11): the squared Pade approximant overflows, A is not finite"),
    E("m52_ls_hi_037", M52, 0.37, 1, 100, .1, (0, 0), "cap", ("few", "few", "few"), gain="0",
      unbounded="the DARE stops at the cap on an iterate whose AKHA has spectral radius 1.116: states reach 1e32 in 700 steps"),
    E("m52_overflow", M52, 10, 1, 100, .1, (1, 1), "cap", CAPPED,
      ill="the capped DARE and DLyap iterates diverge: the passes overflow"),
]
SETUP = [e for e in REGIMES if e.ill is None]                  # constants, power tables, sampler factors
BOUNDED = [e for e in SETUP if e.unbounded is None]            # and the passes
PASS_T = 700                                                   # the length of the pass tests' sequences
BY_NAME = {e.name: e for e in REGIMES}

# the mixing parameters at the box's bounds: S per latent cycles through S_CYCLE, sigma is one of SIGMAS per model
S_CYCLE = (1e-4, 1.0, 1e4, 0.5)
SIGMAS = (1e-4, 1.0, 1e2)


def _ids(entries):
    return [e.name for e in entries]


# ---------------------------------------------------------------------------------------------- references
def state_space(kernel, ls):
    """(F, dF of the lengthscale) of matern32ss.h / matern52ss.h"""
    lam = np.sqrt(3.0) / ls
    if kernel == M32:
        return np.array([[0, 1], [-lam * lam, -2 * lam]]), np.array([[0, 0], [6.0 / ls ** 3, 2 * lam / ls]])
    F = np.array([[0, 1, 0], [0, 0, 1], [-lam * lam * lam, -3 * lam * lam, -3 * lam]])
    dF = np.zeros((3, 3))
    dF[2] = [15 * np.sqrt(5) / ls ** 4, 30 / ls ** 3, np.sqrt(5) * lam * lam]
    return F, dF


def exponents(e):
    """(dt F, dt [F 0; dF F])"""
    F, dF = state_space(e.kernel, e.ls)
    d = F.shape[0]
    B = np.zeros((2 * d, 2 * d))
    B[:d, :d] = B[d:, d:] = F * e.dt
    B[d:, :d] = dF * e.dt
    return F * e.dt, B


def squarings(M):
    """the number of squarings expm takes for M (setup.cu: expm, oracle/moihgp_oracle.cpp: expm)"""
    l1 = np.abs(M).sum(axis=0).max()
    return 0 if l1 <= THETA else int(np.frexp(l1 / THETA)[1])


def mp_expm(M):
    with mpmath.workdps(DPS):
        return np.array(mpmath.expm(mpmath.matrix(M.tolist())).tolist(), dtype=np.float64)


def own_scale_err(a, b):
    """max |a - b| over max |b|; inf if either holds a non-finite entry"""
    if not (np.all(np.isfinite(a)) and np.all(np.isfinite(b))):
        return np.inf
    return rel_err(a, b)


def iter_class(n, conv):
    if n == CAP and not conv:
        return "cap"
    assert conv and n < CAP, (n, conv)
    return "one" if n == 1 else ("few" if n <= 30 else "many")


def _igp(entries):
    return np.array([[e.mag, e.ls, e.noise] for e in entries], dtype=np.float64).ravel()


def make_params(rng, p, entries, sigma):
    L = len(entries)
    U = (np.eye(p, L) + 0.3 * rng.standard_normal((p, L))).ravel()
    S = np.array([S_CYCLE[l % len(S_CYCLE)] for l in range(L)])
    return np.concatenate([U, S, [sigma], _igp(entries)])


def _oracle(e_or_dt, kernel, p, params):
    from oracle.binding import OracleMOIHGP
    o = OracleMOIHGP(e_or_dt, p, (len(params) - 1) // (p + 4), kernel, True)
    o.update(params)
    return o


def _single(e):
    """the oracle with entry e as its one latent (p = 3)"""
    return _oracle(e.dt, e.kernel, 3, make_params(np.random.default_rng(0), 3, [e], 0.05))


_PROBE = {}


def probe(e):
    """what the oracle gives at entry e: squarings, iteration classes, gain, PF conditioning, expm errors against mpmath,
    spectral radii of AKHA and of the RTS gain, finiteness of the constants and of a PASS_T-step filter, NLL and objective"""
    if e.name in _PROBE:
        return _PROBE[e.name]
    from oracle.gen_golden import make_data
    o = _single(e)
    c = o.ihgp_consts(0)
    it = o.ihgp_iters(0)
    FA, B = exponents(e)
    d = FA.shape[0]
    PF = c["PF"]
    w = np.linalg.eigvalsh((PF + PF.T) / 2) if np.all(np.isfinite(PF)) else np.array([np.nan, 1.0])
    Y = make_data(np.random.default_rng(1), 3, 1, PASS_T, e.dt)[None]
    G = o.smoother_consts(0, 1)[0]
    finite = all(np.all(np.isfinite(v)) for v in c.values()) and bool(np.all(np.isfinite(G)))
    r = o.filter_smoother_nll(Y, smoother_mode=-1)
    finite &= bool(np.isfinite(r["X"]).all() and np.isfinite(r["nll"]).all())
    loss, grad, _, _ = o.objective(Y)
    finite &= bool(np.isfinite(loss) and np.isfinite(grad).all())
    radius = lambda M: np.max(np.abs(np.linalg.eigvals(M))) if np.all(np.isfinite(M)) else np.inf
    out = dict(rho=radius(c["AKHA"]), rho_G=radius(G), sq=(squarings(FA), squarings(B)), dare=iter_class(it[0], it[4]), dlyap=tuple(iter_class(it[1 + k], it[5 + k]) for k in range(3)),
               K0=c["K"][0], pf_ratio=w.min() / w.max(), err_A=own_scale_err(c["A"], mp_expm(FA)),
               err_block=own_scale_err(c["dA1"], mp_expm(B)[d:, :d]), finite=finite, l1=(np.abs(FA).sum(0).max(), np.abs(B).sum(0).max()))
    _PROBE[e.name] = out
    return out


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("e", REGIMES, ids=_ids(REGIMES))
def test_entry_reaches_its_regime_under_the_oracle(e):
    r = probe(e)
    assert r["sq"] == e.sq, r
    assert r["dare"] == e.dare and r["dlyap"] == e.dlyap, r
    if e.gain == "1":
        assert r["K0"] > 0.99, r
    elif e.gain == "0":
        assert abs(r["K0"]) < 1e-3, r
    if e.pf == "near-singular":
        assert 0 < r["pf_ratio"] < 1e-4, r


@pytest.mark.parametrize("e", REGIMES, ids=_ids(REGIMES))
def test_entry_is_sorted_by_the_oracle_against_mpmath(e):
    """ill-posed unless the oracle's A = expm(dt F) and its block exponential are within 1e-12 of mpmath (50 digits), each
    on its own scale, and the constants and a PASS_T-step filter, NLL and objective are finite; unbounded if well-posed
    but rho(AKHA) >= 1 or rho(G_rts) >= 1"""
    r = probe(e)
    ill = not (r["err_A"] <= 1e-12 and r["err_block"] <= 1e-12 and r["finite"])
    assert ill == (e.ill is not None), r
    assert (not ill and max(r["rho"], r["rho_G"]) >= 1) == (e.unbounded is not None), r


@pytest.mark.parametrize("kernel", [M32, M52])
def test_table_covers_every_regime(kernel):
    es = [e for e in REGIMES if e.kernel == kernel]
    assert len({e.dt for e in es} - {0.1}) >= 4
    for which in (0, 1):                                        # dt F, the lengthscale block
        assert {0, 1, 2} <= {e.sq[which] for e in es} and max(e.sq[which] for e in es) >= 4
        for k in range(3):                                      # both sides of THETA 2^k, within 10 %
            t = THETA * 2 ** k
            l1 = [probe(e)["l1"][which] for e in es if e in BOUNDED]
            assert any(t / 1.1 <= v <= t for v in l1) and any(t < v <= 1.1 * t for v in l1), (which, k)
    assert any(e.sq[0] == 0 and e.sq[1] > 0 for e in es if e in BOUNDED)
    assert {"one", "few", "cap"} <= {e.dare for e in BOUNDED if e.kernel == kernel}
    for k in range(3):
        assert {"one", "cap"} <= {e.dlyap[k] for e in BOUNDED if e.kernel == kernel}, k
    assert any("one" in e.dlyap and "cap" in e.dlyap for e in BOUNDED if e.kernel == kernel)
    for field, lo, hi in (("noise", 1e-4, 1e2), ("mag", 1e-4, 1e2)):
        vals = {getattr(e, field) for e in BOUNDED if e.kernel == kernel}
        assert lo in vals and hi in vals, field
    assert 1e2 in {e.ls for e in BOUNDED if e.kernel == kernel}
    assert {"0", "1"} <= {e.gain for e in BOUNDED if e.kernel == kernel}
    assert any(e.pf == "near-singular" for e in BOUNDED if e.kernel == kernel)
    assert any(e.ill and "stiff" in e.ill for e in es) and any(e.ill and "overflow" in e.ill for e in es)
    assert any(e.unbounded for e in es if e in SETUP)


# ---------------------------------------------------------------------------------------------------------------- GPU
def _device(kernel, dt, p, params):
    from multioutputihgp_b200 import MOIHGPSequences
    L = (len(params) - 1) // (p + 4)
    m = MOIHGPSequences(dt, p, L, kernel, True)
    m.update(params)
    return m


def _same(a, b):
    """a against b on b's own scale; an exactly-zero b must be matched exactly, a non-finite pattern too"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    fin = np.isfinite(b)
    assert np.array_equal(np.isfinite(a), fin)
    if not fin.any() or np.max(np.abs(b[fin])) == 0:
        return np.array_equal(a[fin], b[fin])
    return rel_err(a[fin], b[fin]) < TOL


def _power_close(got, want, tol):
    """a block power on its own scale; one below 1e-100 only has to be negligible too.  There M^n is a product of
    near-cancelling factors (||M^n|| << ||M||^n), and its relative digits depend on the order of the products: the
    library's tables and the host's doubling differ by up to 8e-12 there (magnitude 1e-4: AKHA^1000 = 3e-279)."""
    if np.max(np.abs(want)) < 1e-100:
        return np.max(np.abs(got)) < 1e-90
    return rel_err(got, want) < tol


def _binary_power(M, n):
    """M^n by binary powering on the table M^(2^k), the order the library composes its tables in"""
    P, Mk = np.eye(M.shape[0]), M.copy()
    while n:
        if n & 1:
            P = Mk @ P
        Mk = Mk @ Mk
        n >>= 1
    return P


@pytest.mark.gpu
@pytest.mark.parametrize("e", SETUP, ids=_ids(SETUP))
def test_setup_constants_match_the_oracle(cuda_lib, e):
    """every LatentConsts field latent_consts() returns, one field at a time on its own scale; the DARE / DLyap iteration
    counts and convergence flags exactly; both smoother modes' gain and covariance; the power tables against host
    binary powering of the library's own AKHA and G."""
    from multioutputihgp_b200.parallel import block_transition, stack_consts
    params = make_params(np.random.default_rng(0), 3, [e], 0.05)
    o = _oracle(e.dt, e.kernel, 3, params)
    m = _device(e.kernel, e.dt, 3, params)
    assert m.latent_iters(0) == o.ihgp_iters(0)
    c, co = m.latent_consts(0), o.ihgp_consts(0)
    assert set(c) == set(co)
    for k in co:
        assert _same(c[k], co[k]), k
    for mode in (0, 1):
        G, P = m.smoother_consts(0, mode)
        Go, Po = o.smoother_consts(0, mode)
        assert _same(G, Go), mode
        assert _same(P, Po), mode
    AK, dAK = stack_consts([c])
    for n in (1, 2, 3, 256, 1000):
        Pn, En = m.block_transition(n)
        Ph, Eh = block_transition(AK, dAK, n)
        assert _power_close(Pn[0], Ph[0], 1e-12), n
        for k in range(3):
            assert _power_close(En[0, k], Eh[0, k], 1e-11), (n, k)
    for mode in (0, 1):
        G = m.smoother_consts(0, mode)[0]
        for n in (1, 3, 256):
            want = _binary_power(G, n)
            got = m.smoother_power(n, mode)[0]
            if np.all(np.isfinite(want)) and np.max(np.abs(want)) < 1e250:
                assert _power_close(got, want, 1e-12), (mode, n)


def _psd_part(M):
    w, V = np.linalg.eigh((M + M.T) / 2)
    return (V * np.maximum(w, 0.0)) @ V.T


@pytest.mark.gpu
@pytest.mark.parametrize("e", SETUP, ids=_ids(SETUP))
def test_sampler_factors_at_the_entry(cuda_lib, e):
    """LF LF' = PF and LC LC' = C = PF - G PPc G' (PPc = A PF A' + Q, oracle constants, RTS gain), both lower-triangular
    and NaN-free, on PF's scale: to 1e-12 where the matrix is positive definite, else its positive semi-definite part to
    1e-9 (the Matern-5/2 state space replicated from the reference has an indefinite Q, test_gpu_sampling)."""
    params = make_params(np.random.default_rng(0), 3, [e], 0.05)
    o = _oracle(e.dt, e.kernel, 3, params)
    m = _device(e.kernel, e.dt, 3, params)
    c = o.ihgp_consts(0)
    G = o.smoother_consts(0, 1)[0]
    PF = c["PF"]
    C = PF - G @ (c["A"] @ PF @ c["A"].T + c["Q"]) @ G.T
    LF, LC = m.sampler_consts(0)
    scale = np.max(np.abs(PF))
    for Lo, M in ((LF, PF), (LC, C)):
        assert np.all(np.isfinite(Lo)) and np.array_equal(Lo, np.tril(Lo))
        w = np.linalg.eigvalsh((M + M.T) / 2)
        assert np.max(np.abs(Lo @ Lo.T - _psd_part(M))) <= 1e-9 * scale
        if w.min() > 1e-6 * scale:
            assert np.max(np.abs(Lo @ Lo.T - M)) <= 1e-12 * scale


# ---- passes on models whose latents each sit in another regime
def _group(kernel, dt):
    return [e for e in BOUNDED if e.kernel == kernel and e.dt == dt]


PASS_DTS = (0.1, 0.37, 1, 10)


def _mixed(kernel, dt, p, L, sigma, seed):
    """(params, entries): latent l in regime l % (number of bounded entries at (kernel, dt))"""
    grp = _group(kernel, dt)
    assert len(grp) >= 3, (kernel, dt)
    entries = [grp[l % len(grp)] for l in range(L)]
    return make_params(np.random.default_rng(seed), p, entries, sigma), entries


def _per_latent(a, b, axis):
    """worst relative error over latents, each latent (index `axis`) on its own scale.  The reference must be finite (the
    passes run at bounded entries only); a non-finite value in `a` gives NaN, which np.max carries and `< TOL` rejects."""
    a, b = np.asarray(a), np.asarray(b)
    assert np.all(np.isfinite(b)), "reference not finite"
    return float(np.max([rel_err(np.take(a, l, axis=axis), np.take(b, l, axis=axis)) for l in range(b.shape[axis])]))


def _literal_per_latent(a, b, X, latents, big=1e100):
    """the literal smoother [N,T,L,d] of `latents` (those whose gain forgets, rho(G_lit) < 1; the others diverge in the
    reference too, SURVEY Q3) over the trailing steps where the reference stays below `big`, on the scale of that tail's
    smoothed and filtered states: this smoother forms Xs from (I - A) X, so it carries X's rounding in absolute terms
    (test_gpu_long_memory).  A non-finite value of `a` in the compared tail gives NaN."""
    errs = []
    T = b.shape[1]
    for l in latents:
        with np.errstate(invalid="ignore"):
            mx = np.max(np.abs(b[:, :, l]), axis=(0, 2))
        bad = ~(np.isfinite(mx) & (mx < big))
        t0 = int(np.max(np.nonzero(bad)[0])) + 1 if bad.any() else 0
        assert T - t0 >= 50, (l, t0)
        diff = np.max(np.abs(a[:, t0:, l] - b[:, t0:, l]))
        scale = max(np.max(np.abs(b[:, t0:, l])), np.max(np.abs(X[:, t0:, l])))
        errs.append(diff / scale)
    return float(np.max(errs))


def _profiled(m, fn):
    m.profile(True)
    out = fn()
    prof = m.profile_read()
    m.profile(False)
    return out, prof


def _grad_blocks(p, L):
    pL = p * L
    return ([("dU", slice(0, pL)), ("dS", slice(pL, pL + L)), ("dsigma", slice(pL + L, pL + L + 1))]
            + [("latent%d" % l, slice(pL + L + 1 + 3 * l, pL + L + 4 + 3 * l)) for l in range(L)])


def _assert_objective(got, want, p, L):
    loss, grad, xT, dxT = got
    lo, go, xo, dxo = want
    assert abs(loss - lo) <= TOL * abs(lo), (loss, lo)
    for name, sl in _grad_blocks(p, L):
        assert rel_err(grad[sl], go[sl]) < TOL, name
    if xT is not None:
        assert _per_latent(xT, xo, 1) < TOL and _per_latent(dxT, dxo, 1) < TOL


PASS_CASES = [(k, dt, p, L) for k in (M32, M52) for dt in PASS_DTS for p, L in ((16, 8), (12, 5))]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,dt,p,L", PASS_CASES)
def test_passes_on_a_mixed_model_match_the_oracle(cuda_lib, kernel, dt, p, L):
    """The fused pass on every path that serves the shape (many-chains for p = 16, L = 8; the chunked scan, with a ragged
    latent group for L = 5; the automatic choice) in both smoother modes from a carried-in x0, the per-step NLL terms and
    the objective from x0 / dx0: every latent, output, field and gradient block on its own scale."""
    from oracle.gen_golden import make_data
    N, T = 2, PASS_T
    sigma = SIGMAS[(PASS_DTS.index(dt) + L) % len(SIGMAS)]
    params, entries = _mixed(kernel, dt, p, L, sigma, 11 * L + int(10 * dt))
    rng = np.random.default_rng(L)
    m = _device(kernel, dt, p, params)
    o = _oracle(dt, kernel, p, params)
    d = m.igp_dim
    Y = np.stack([make_data(rng, p, L, T, dt) for _ in range(N)])
    x0 = 0.3 * rng.standard_normal((N, L, d))
    dx0 = 0.1 * rng.standard_normal((N, L, 3, d))
    stable = [l for l in range(L) if np.max(np.abs(np.linalg.eigvals(o.smoother_consts(l, 0)[0]))) < 1]
    paths = [("chain", "k_filter_chain"), ("scan", "k_scan_final"), ("auto", None)] if L == 8 else [("scan", "k_scan_final"), ("auto", None)]
    for mode in (1, 0):
        ro = o.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True, nthreads=8)
        for path, kname in paths:
            m.set_path(path)
            r, prof = _profiled(m, lambda: m.filter_smoother_nll(Y, x0=x0, smoother_mode=mode, want_yhat=True))
            where = (path, mode)
            if kname:
                assert kname in prof, (where, sorted(prof))
            assert _per_latent(r["X"], ro["X"], 2) < TOL, where
            assert _per_latent(r["xT"], ro["xT"], 1) < TOL, where
            assert _per_latent(r["Yhat"], ro["Yhat"], 2) < TOL, where           # every output on its own scale
            assert rel_err(r["nll"], ro["nll"]) < TOL, where
            if mode == 1:
                assert _per_latent(r["Xs"], ro["Xs"], 2) < TOL, where
            else:
                assert _literal_per_latent(r["Xs"], ro["Xs"], ro["X"], stable) < TOL, where
    m.set_path("auto")
    r = m.nll_steps(Y, x0=x0)
    assert rel_err(r["nll"], ro["nll"]) < TOL and _per_latent(r["xT"], ro["xT"], 1) < TOL
    for n in range(N):            # step t's term is negLogLikelihood(x[t-1], y[t]) on the oracle's filtered states
        prev = np.concatenate([x0[n][None], ro["X"][n, :-1]])
        want = np.array([o.negLogLikelihood(prev[t], Y[n, t]) for t in range(T)])
        assert rel_err(r["nll_steps"][n], want) < TOL, n
    got = m.objective(Y, x0=x0, dx0=dx0, want_state=True)
    _assert_objective(got, o.objective(Y, x0=x0, dx0=dx0), p, L)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [M32, M52])
def test_one_launch_objective_and_the_online_window_at_dt_1(cuda_lib, kernel):
    """k_obj_small (N = 1, T <= 1024: one launch) through objective() and through the streaming learner's resident window
    (online_objective), on a mixed model at dt = 1, against the oracle block by block."""
    from oracle.gen_golden import make_data
    dt, p, L, T = 1, 12, 5, 300
    params, _ = _mixed(kernel, dt, p, L, 1e-4, 7)
    m = _device(kernel, dt, p, params)
    o = _oracle(dt, kernel, p, params)
    rng = np.random.default_rng(3)
    Y = make_data(rng, p, L, T, dt)[None]
    d = m.igp_dim
    x0, dx0 = 0.2 * rng.standard_normal((1, L, d)), 0.1 * rng.standard_normal((1, L, 3, d))
    n0 = m.launch_count
    got = m.objective(Y, x0=x0, dx0=dx0, want_state=True)
    assert m.launch_count - n0 == 1
    _assert_objective(got, o.objective(Y, x0=x0, dx0=dx0), p, L)
    assert m.online_begin(T)
    m.online_set_proximal()                                     # no proximal term: the window's objective alone
    for t in range(T):
        m.online_push(Y[0, t], ma_given=np.zeros(p))
    x, dx = m.online_state()
    assert not x.any() and not dx.any()                          # nothing has left the window yet
    params2 = params.copy()
    params2[p * L + L + 1:] *= 1.01                              # another point of the same regimes, set by the launch itself
    loss, grad = m.online_objective(params2)
    o.update(params2)
    lo, go, _, _ = o.objective(Y)
    _assert_objective((loss, grad, None, None), (lo, go, None, None), p, L)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [M32, M52])
def test_samples_on_a_mixed_model_with_a_noise_1em4_latent(cuda_lib, kernel):
    """x~ = the library's RTS mean + e recomputed in NumPy from the library's own factors (test_gpu_sampling), on both
    sampler variants, each latent on its own scale; the model holds a latent with noise 1e-4 (gain ~ 1, PF nearly
    singular)."""
    from test_gpu_sampling import _factors, noise
    from oracle.gen_golden import make_data
    dt, p, L, N, T, S = 0.1, 12, 5, 2, 300, 2
    params, entries = _mixed(kernel, dt, p, L, 1.0, 21)
    assert any(e.noise == 1e-4 for e in entries)
    m = _device(kernel, dt, p, params)
    rng = np.random.default_rng(4)
    Y = np.stack([make_data(rng, p, L, T, dt) for _ in range(N)])
    x0 = 0.2 * rng.standard_normal((N, L, m.igp_dim))
    seed = 0x5EED_0BAD_F00D
    Xs = m.filter_smoother_nll(Y, x0=x0, smoother_mode=1)["Xs"]
    e = noise(seed, S, N, T, *_factors(m))
    for path in ("scan", "chain"):
        m.set_path(path)
        r = m.sample_posterior(Y, S, seed, x0=x0, want_states=True, want_outputs=False)
        assert _per_latent(r["Xs"], Xs, 2) < TOL, path
        assert np.all(np.isfinite(r["X"]))
        assert _per_latent(r["X"], r["Xs"][None] + e, 3) < TOL, path
    m.set_path("auto")


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,dt", [(M32, 0.37), (M32, 10), (M52, 1), (M52, 0.37)])
def test_per_observation_symbols_at_other_dt(cuda_lib, kernel, dt, monkeypatch):
    """gp32_* / gp52_* (pywrapper.MOIHGP: gpXX_new carries dt) over a short stream against the oracle's step and
    negLogLikelihood: states and sensitivities per latent, the loss, and every gradient block on its own scale."""
    if kernel == M52:
        monkeypatch.setenv("MOIHGP_GP52_MATERN52", "1")
    from multioutputihgp_b200 import MOIHGP
    from oracle.gen_golden import make_data
    p, L, T = 6, 3, 20
    params, _ = _mixed(kernel, dt, p, L, 1e2, 5)
    m = MOIHGP(dt, p, L, kernel=kernel, threading=True)
    m.update(params)
    o = _oracle(dt, kernel, p, params)
    Y = make_data(np.random.default_rng(6), p, L, T, dt)
    x, dx = np.zeros((L, m.igp_dim)), np.zeros((L, 3, m.igp_dim))
    for t, y in enumerate(Y):
        lg, gg = m.negLogLikelihood(x, y, dx)
        lo, go = o.negLogLikelihood(x, y, dx)
        assert abs(lg - lo) <= TOL * abs(lo), t
        for name, sl in _grad_blocks(p, L):
            assert rel_err(gg[sl], go[sl]) < TOL, (t, name)
        xp, yp = m.step(x)
        xpo, ypo = o.step(x)
        assert _per_latent(xp, xpo, 0) < TOL and rel_err(yp, ypo) < TOL, t
        xn, yh, dxn = m.step(x, y, dx)
        xo, yo, dxo = o.step(x, y, dx)
        assert _per_latent(xn, xo, 0) < TOL and _per_latent(dxn, dxo, 0) < TOL and rel_err(yh, yo) < TOL, t
        x, dx = xo, dxo
