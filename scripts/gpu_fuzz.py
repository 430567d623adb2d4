"""Differential fuzz on the GPU: random shapes through the chunked-scan pass and the general objective against the CPU
oracle (L drawn on both sides of the multiple-of-8 rule, so both the thread-per-sub-chunk and the warp-per-chunk kernels
run), and through the alternative implementations of the same pass - many-chains vs chunked-scan path, one-launch vs
general objective, time-sharded blocks vs the whole sequence.  Prints a summary; exits non-zero on a mismatch."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from multioutputihgp_b200 import MOIHGPSequences
from multioutputihgp_b200.parallel import backward_carry_in, forward_carry_in
from oracle.binding import OracleMOIHGP
from oracle.gen_golden import make_data, make_params

TOL = 1e-9          # fp64 agreement with the oracle, norm-wise relative (tests/conftest.py)
CASES = int(os.environ.get("FUZZ_CASES", 120))
rng = np.random.default_rng(int(os.environ.get("FUZZ_SEED", 2024)))
dev = torch.device("cuda:0")


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(float(np.max(np.abs(b))), 1e-300))


worst = {}


def note(name, e, tol, ctx):
    worst[name] = max(worst.get(name, 0.0), e)
    if not e < tol:
        print("MISMATCH %s: %.3e (tol %.1e) at %s" % (name, e, tol, ctx))
        sys.exit(1)


for case in range(CASES):
    kernel = ("Matern32", "Matern52")[int(rng.integers(2))]
    L = int(rng.choice([1, 2, 3, 4, 5, 8, 8, 12, 16, 16, 24, 32]))
    p = L + int(rng.integers(0, 3 * L + 2))
    N = int(rng.choice([1, 1, 1, 2, 3, 5]))
    T = int(rng.choice([1, 2, 31, 32, 33, 255, 256, 257, 511, 512, 513, 700, 1023, 1025, 1300, 2049]))
    ctx = (kernel, p, L, N, T)
    params = make_params(rng, p, L, kernel)
    Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
    threading = bool(rng.integers(2))
    m = MOIHGPSequences(0.1, p, L, kernel, threading)
    o = OracleMOIHGP(0.1, p, L, kernel, threading)
    m.update(params)
    o.update(params)
    d = m.igp_dim
    x0 = 0.3 * rng.standard_normal((N, L, d))
    dx0 = 0.1 * rng.standard_normal((N, L, 3, d))
    # --- scan path (final pass: k_scan_lanes when L % 8 == 0, else k_scan) against the oracle
    m.set_path("scan")
    a = m.filter_smoother_nll(Y, x0=x0, smoother_mode=1)
    ao = o.filter_smoother_nll(Y, x0=x0, smoother_mode=1, nthreads=8)
    for k in ("X", "Xs", "nll", "xT"):
        note("scan vs oracle " + k, rel(a[k], ao[k]), TOL, ctx)
    # --- many-chains path where instantiated
    try:
        m.set_path("chain")
        c = m.filter_smoother_nll(Y, x0=x0, smoother_mode=1)
        for k in ("X", "Xs", "nll", "xT"):
            note("chain vs scan " + k, rel(c[k], a[k]), 1e-10, ctx)
    except RuntimeError:
        pass
    m.set_path("auto")
    # --- objective: general path (k_obj_lanes when L % 8 == 0, else k_obj_scan) against the oracle, one-launch vs general
    m.set_path("scan")                                   # general path (no one-launch kernel)
    la, ga, xa, dxa = m.objective(Y, x0=x0, dx0=dx0, want_state=True)
    m.set_path("auto")
    lo, go, xo, dxo = o.objective(Y, x0=x0, dx0=dx0)
    note("objective vs oracle loss", abs(la - lo) / abs(lo), TOL, ctx)
    note("objective vs oracle grad", rel(ga, go), TOL, ctx)
    note("objective vs oracle state", max(rel(xa, xo), rel(dxa, dxo)), TOL, ctx)
    if N == 1:
        lc, gc, xc, dxc = m.objective(Y, x0=x0, dx0=dx0, want_state=True)
        note("objective one-launch vs general loss", abs(lc - la) / abs(la), 1e-11, ctx)
        note("objective one-launch vs general grad", rel(gc, ga), 1e-10, ctx)
        note("objective one-launch vs general state", max(rel(xc, xa), rel(dxc, dxa)), 1e-10, ctx)
    # --- time-sharded blocks (separate handles) vs the whole sequence
    if T >= 513:
        cuts = [0, 256 * int(rng.integers(1, (T - 1) // 256 + 1)), T]
        if cuts[1] >= T:
            cuts[1] = 256
        lengths = [cuts[1], T - cuts[1]]
        models = []
        for g in range(2):
            mg = MOIHGPSequences(0.1, p, L, kernel, True)
            mg.update(params)
            models.append(mg)
        Yd = [torch.from_numpy(np.ascontiguousarray(Y[:, cuts[g]:cuts[g + 1]])).to(dev) for g in range(2)]
        to_dev = lambda z: torch.from_numpy(np.ascontiguousarray(z)).to(dev)
        ph1 = [models[g].fsn_block(1, Yd[g], g == 1, 1) for g in range(2)]
        ends, uf = [q[0] for q in ph1], [q[1] for q in ph1]
        x_in = [forward_carry_in(models[0].block_transition, lengths, ends, x0, g) for g in range(2)]
        ua = [to_dev(uf[1]), None]
        b0 = [models[g].fsn_block(2, Yd[g], g == 1, 1, x0=to_dev(x_in[g]), u_after=ua[g]) for g in range(2)]
        Xb = [torch.zeros((N, lengths[g], L, d), dtype=torch.float64, device=dev) for g in range(2)]
        Xsb = [torch.zeros_like(Xb[g]) for g in range(2)]
        nllb = torch.zeros((2, N), dtype=torch.float64, device=dev)
        for g in range(2):
            be = backward_carry_in(lambda n_: models[0].smoother_power(n_, 1), lengths, b0, g)
            models[g].fsn_block(3, Yd[g], g == 1, 1, x0=to_dev(x_in[g]), u_after=ua[g], b_end=None if be is None else to_dev(be), X=Xb[g], Xs=Xsb[g], nll=nllb[g])
        torch.cuda.synchronize()
        note("time-sharded X", rel(np.concatenate([q.cpu().numpy() for q in Xb], 1), a["X"]), 1e-11, ctx)
        note("time-sharded Xs", rel(np.concatenate([q.cpu().numpy() for q in Xsb], 1), a["Xs"]), 1e-10, ctx)
        note("time-sharded nll", rel(nllb.sum(0).cpu().numpy(), a["nll"]), 1e-11, ctx)
# --- host-buffer call in several pipeline slices vs the device-resident call
for (kernel, p, L, N, T) in (("Matern52", 16, 8, 1300, 40), ("Matern32", 8, 4, 2500, 33)):
    params = make_params(rng, p, L, kernel)
    Y = rng.standard_normal((N, T, p))
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    m.update(params)
    d = m.igp_dim
    x0 = 0.3 * rng.standard_normal((N, L, d))
    host = m.filter_smoother_nll(Y, x0=x0, smoother_mode=1, want_yhat=True)
    Xd = torch.zeros((N, T, L, d), dtype=torch.float64, device=dev)
    Xsd = torch.zeros_like(Xd)
    Yh = torch.zeros((N, T, p), dtype=torch.float64, device=dev)
    nd = torch.zeros(N, dtype=torch.float64, device=dev)
    m.filter_smoother_nll_device(torch.from_numpy(Y).to(dev), x0=torch.from_numpy(x0).to(dev), smoother_mode=1, X=Xd, Xs=Xsd, Yhat=Yh, nll=nd)
    torch.cuda.synchronize()
    ctx = (kernel, p, L, N, T)
    note("host slices vs device X", rel(host["X"], Xd.cpu().numpy()), 1e-13, ctx)
    note("host slices vs device Xs", rel(host["Xs"], Xsd.cpu().numpy()), 1e-13, ctx)
    note("host slices vs device Yhat", rel(host["Yhat"], Yh.cpu().numpy()), 1e-13, ctx)
    note("host slices vs device nll", rel(host["nll"], nd.cpu().numpy()), 1e-13, ctx)
print("fuzz: %d cases, worst relative differences:" % CASES)
for k in sorted(worst):
    print("   %-45s %.2e" % (k, worst[k]))
