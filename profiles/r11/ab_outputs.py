"""Bitwise A/B of two builds of libmoihgp.so: profiles/r06/ab_outputs.py plus the time-sharded entry points whose code
moved in round 11 (one carry kernel for the three exchanges, one packing path for the block phases): the host outputs of
fsn_block phases 1 and 2, and the time-sharded sampler (sample_block_async around the backward carry).

    MOIHGP_B200_LIB=<lib> python profiles/r11/ab_outputs.py run OUTDIR      every output of the cases below -> OUTDIR/*.npy
    python profiles/r11/ab_outputs.py compare DIR_A DIR_B                   byte-for-byte comparison (np.array_equal and
                                                                            identical bytes, so NaN == NaN in the same place)
Inputs are seeded (NumPy, or torch's CUDA generator for the large objective), so both libraries see the same data."""
import glob
import os
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def run(out):
    import torch
    from conftest import golden_cases, load_golden
    from multioutputihgp_b200 import MOIHGP, MOIHGPSequences
    from oracle.gen_golden import make_data, make_params
    os.makedirs(out, exist_ok=True)
    dev = torch.device("cuda:0")
    f64 = dict(dtype=torch.float64, device=dev)

    def save(name, a):
        a = a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a, dtype=np.float64)
        np.save(os.path.join(out, name + ".npy"), a)

    def model(kernel, p, L, seed):
        rng = np.random.default_rng(seed)
        params = make_params(rng, p, L, kernel)
        m = MOIHGPSequences(0.1, p, L, kernel, True)
        m.update(params)
        return m, params, rng

    # block transitions and smoother powers (host entry points)
    for kernel, p, L in (("Matern32", 8, 4), ("Matern52", 16, 8)):
        m, _, _ = model(kernel, p, L, 1)
        for n in (0, 1, 5, 256, 10 ** 7):
            P, E = m.block_transition(n)
            save("bt_%s_%d_P" % (kernel, n), P)
            save("bt_%s_%d_E" % (kernel, n), E)
            for mode in (0, 1):
                save("sp_%s_%d_%d" % (kernel, n, mode), m.smoother_power(n, mode))

    # time-sharded filter + smoother: both carry directions (k_fsn_carry) in both smoother modes, one handle per block
    for kernel, p, L, N, cuts in (("Matern52", 16, 8, 2, (0, 256, 512, 1024)), ("Matern32", 64, 32, 1, (0, 2048, 4096, 6000)),
                                  ("Matern32", 8, 4, 3, (0, 256, 2560, 2816, 300000))):
        rng = np.random.default_rng(sum(cuts) + 7)
        params = make_params(rng, p, L, kernel)
        T, G = cuts[-1], len(cuts) - 1
        lengths = [cuts[g + 1] - cuts[g] for g in range(G)]
        Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
        models = []
        for g in range(G):
            m = MOIHGPSequences(0.1, p, L, kernel, True)
            m.update(params)
            models.append(m)
        d = models[0].igp_dim
        x0d = torch.from_numpy(0.3 * rng.standard_normal((N, L, d))).to(dev)
        Yd = [torch.from_numpy(np.ascontiguousarray(Y[:, cuts[g]:cuts[g + 1]])).to(dev) for g in range(G)]
        for mode in (1, 0):
            tag = "fsn_%s_%d_%d" % (kernel, p, mode)
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
            for name, a in (("g1", g1), ("g2", g2), ("xin", xin), ("uaf", uaf), ("bend", bend), ("nll", nll),
                            ("X", torch.cat(X, 1)), ("Xs", torch.cat(Xs, 1))):
                save(tag + "_" + name, a)
            # the same phases 1 and 2 with their outputs copied to host memory (moihgp_cuda_fsn_block_dev)
            for g in range(G):
                xe, uf = models[g].fsn_block(1, Yd[g], g == G - 1, mode)
                b0 = models[g].fsn_block(2, Yd[g], g == G - 1, mode, x0=xin[g], u_after=None if g == G - 1 else uaf[g])
                save("%s_host1x_%d" % (tag, g), xe)
                save("%s_host1u_%d" % (tag, g), uf)
                save("%s_host2_%d" % (tag, g), b0)

    # time-sharded objective: the carry-in from the gathered block ends (k_block_carry)
    for kernel, p, L, N, cuts in (("Matern32", 16, 8, 1, (0, 512, 1280, 2048, 2300)), ("Matern52", 8, 4, 2, (0, 256, 768, 1000)),
                                  ("Matern32", 256, 64, 1, (0, 1024, 2048, 3001)), ("Matern52", 8, 4, 1, (0, 256, 512, 10496, 700000))):
        rng = np.random.default_rng(sum(cuts) + p)
        params = make_params(rng, p, L, kernel)
        T, G = cuts[-1], len(cuts) - 1
        lengths = [cuts[g + 1] - cuts[g] for g in range(G)]
        Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
        models = []
        for g in range(G):
            m = MOIHGPSequences(0.1, p, L, kernel, True)
            m.update(params)
            models.append(m)
        d = models[0].igp_dim
        x0d = torch.from_numpy(0.2 * rng.standard_normal((N, L, d))).to(dev)
        dx0d = torch.from_numpy(0.1 * rng.standard_normal((N, L, 3, d))).to(dev)
        Yd = [torch.from_numpy(np.ascontiguousarray(Y[:, cuts[g]:cuts[g + 1]])).to(dev) for g in range(G)]
        ends = torch.zeros((G, N, L, 4, d), **f64)
        for g in range(G):
            models[g].objective_begin_async(Yd[g], None if g == G - 1 else ends[g])
        res = torch.zeros((G, 2 + models[0].num_param), **f64)
        xin = torch.zeros((G, N, L, d), **f64)
        dxin = torch.zeros((G, N, L, 3, d), **f64)
        for g in range(G):
            models[g].carry_in_device(ends, lengths, g, xin[g], dxin[g], x0=x0d, dx0=dx0d)
            models[g].objective_finish_device(Yd[g], res[g, 0:1], res[g, 2:], x0=xin[g], dx0=dxin[g])
        torch.cuda.synchronize()
        tag = "tso_%s_%d_%d" % (kernel, p, T)
        for name, a in (("ends", ends), ("xin", xin), ("dxin", dxin), ("out", res)):
            save(tag + "_" + name, a)

    # the chunked sampler (k_sample_carry: G^chunk_len by binary powering)
    for kernel, p, L, N, S, T in (("Matern32", 8, 4, 2, 4, 200000), ("Matern52", 16, 8, 2, 4, 200000), ("Matern52", 6, 3, 1, 2, 5000)):
        m, _, rng = model(kernel, p, L, 11)
        Yd = torch.from_numpy(np.stack([make_data(rng, p, L, T) for _ in range(N)])).to(dev)
        d = m.igp_dim
        Xs = torch.zeros((N, T, L, d), **f64)
        F = torch.zeros((S, N, T, L), **f64)
        m.sample_posterior_device(Yd, 1234, Xs=Xs, F=F)
        torch.cuda.synchronize()
        save("sample_%s_%d_Xs" % (kernel, p), Xs)
        save("sample_%s_%d_F" % (kernel, p), F)

    # the time-sharded sampler: phase 1 per block, the backward carry over the gathered starts, phase 2 (one handle per block)
    for kernel, p, L, N, S, cuts in (("Matern32", 8, 4, 2, 3, (0, 256, 2560, 2816, 300000)), ("Matern52", 16, 8, 1, 2, (0, 512, 1024, 1500))):
        rng = np.random.default_rng(sum(cuts) + 13)
        params = make_params(rng, p, L, kernel)
        T, G = cuts[-1], len(cuts) - 1
        lengths = [cuts[g + 1] - cuts[g] for g in range(G)]
        models = []
        for g in range(G):
            m = MOIHGPSequences(0.1, p, L, kernel, True)
            m.update(params)
            models.append(m)
        d = models[0].igp_dim
        Xs = torch.from_numpy(0.5 * rng.standard_normal((N, T, L, d))).to(dev)
        Xb = [Xs[:, cuts[g]:cuts[g + 1]].contiguous() for g in range(G)]
        e1 = torch.zeros((G, S * N, L, d), **f64)
        eend = torch.zeros((G, S * N, L, d), **f64)
        F = [torch.zeros((S, N, lengths[g], L), **f64) for g in range(G)]
        for g in range(G):
            models[g].sample_block_async(1, Xb[g], S, 99, cuts[g], g == G - 1, out=e1[g])
        for g in range(G):
            models[g].fsn_carry_device(1, e1, lengths, g, eend[g], smoother_mode=1)
            models[g].sample_block_async(2, Xb[g], S, 99, cuts[g], g == G - 1, e_end=None if g == G - 1 else eend[g], Fsamp=F[g])
        torch.cuda.synchronize()
        tag = "tss_%s_%d_%d" % (kernel, p, T)
        for name, a in (("e1", e1), ("eend", eend), ("F", torch.cat(F, 2))):
            save(tag + "_" + name, a)

    # legacy per-observation symbols (k_step / k_lik) on the golden rows with missing outputs, and on NaN rows at L = 64
    for path in golden_cases():
        g = load_golden(path)
        os.environ["MOIHGP_GP52_MATERN52"] = "1" if str(g["kernel"]) == "Matern52" else "0"
        m = MOIHGP(float(g["dt"]), int(g["p"]), int(g["L"]), kernel=str(g["kernel"]), threading=bool(g["threading"]))
        m.update(g["params"])
        tag = "legacy_" + os.path.basename(path)[:-4]
        for i in range(3):
            for j, a in enumerate(m.step(g["one_x"], g["nan%d_y" % i], g["one_dx"])):
                save("%s_nan%d_step%d" % (tag, i, j), a)
            l1, g1 = m.negLogLikelihood(g["one_x"], g["nan%d_y" % i], g["one_dx"])
            save("%s_nan%d_lik1" % (tag, i), [l1])
            save("%s_nan%d_grad" % (tag, i), g1)
            save("%s_nan%d_lik2" % (tag, i), [m.negLogLikelihood(g["one_x"], g["nan%d_y" % i])])
        l1, g1 = m.negLogLikelihood(g["one_x"], g["one_y"], g["one_dx"])
        save(tag + "_lik1", [l1])
        save(tag + "_grad", g1)
    os.environ.pop("MOIHGP_GP52_MATERN52", None)
    for kernel, p in (("Matern32", 96), ("Matern32", 64)):
        L = 64
        rng = np.random.default_rng(p)
        m = MOIHGP(0.1, p, L, kernel=kernel, threading=True)
        m.update(make_params(rng, p, L, kernel))
        d = m.igp_dim
        x = rng.standard_normal((L, d))
        dx = rng.standard_normal((L, 3, d))
        y = rng.standard_normal(p)
        for case, miss in (("some", rng.choice(p, 20, replace=False)), ("under", rng.choice(p, p - L // 2, replace=False)), ("all", np.arange(p))):
            yy = y.copy()
            yy[miss] = np.nan
            tag = "legacy_L64_%d_%s" % (p, case)
            for j, a in enumerate(m.step(x, yy, dx)):
                save("%s_step%d" % (tag, j), a)
            l1, g1 = m.negLogLikelihood(x, yy, dx)
            save(tag + "_lik1", [l1])
            save(tag + "_grad", g1)
            save(tag + "_lik2", [m.negLogLikelihood(x, yy)])
        l1, g1 = m.negLogLikelihood(x, y, dx)
        save("legacy_L64_%d_lik1" % p, [l1])
        save("legacy_L64_%d_grad" % p, g1)

    # the objective at the config-5 shape (p = 256, L = 64, T = 10^6; k_obj_finish)
    m, params, rng = model("Matern32", 256, 64, 5)
    gen = torch.Generator(device=dev)
    gen.manual_seed(5)
    Yd = torch.randn((1, 10 ** 6, 256), generator=gen, **f64)
    loss = torch.zeros(1, **f64)
    grad = torch.zeros(m.num_param, **f64)
    m.objective_device(Yd, loss, grad)
    torch.cuda.synchronize()
    save("obj_c5_Ysum", [float(Yd.sum())])
    save("obj_c5_loss", loss)
    save("obj_c5_grad", grad)
    del Yd

    # the fused pass on both paths (many-chains: the host NLL constant; chunked scan: k_nll_reduce), both smoother modes,
    # one sequence with missing outputs
    for kernel, p, L, N, T in (("Matern52", 16, 8, 64, 3000), ("Matern32", 8, 4, 40, 1500)):
        m, _, rng = model(kernel, p, L, 21)
        Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
        Y[3, 100, :p // 2] = np.nan
        Y[3, 700, :] = np.nan
        Yd = torch.from_numpy(Y).to(dev)
        d = m.igp_dim
        x0d = torch.from_numpy(0.3 * rng.standard_normal((N, L, d))).to(dev)
        for path in ("chain", "scan"):
            m.set_path(path)
            for mode in (0, 1):
                X = torch.zeros((N, T, L, d), **f64)
                Xs = torch.zeros_like(X)
                Yhat = torch.zeros((N, T, p), **f64)
                nll = torch.zeros(N, **f64)
                xT = torch.zeros((N, L, d), **f64)
                m.filter_smoother_nll_device(Yd, x0=x0d, smoother_mode=mode, X=X, Xs=Xs, Yhat=Yhat, nll=nll, xT=xT)
                torch.cuda.synchronize()
                tag = "fused_%s_%d_%s_%d" % (kernel, p, path, mode)
                for name, a in (("X", X), ("Xs", Xs), ("Yhat", Yhat), ("nll", nll), ("xT", xT)):
                    save(tag + "_" + name, a)
        m.set_path("auto")
    print("wrote %d arrays to %s" % (len(glob.glob(os.path.join(out, "*.npy"))), out))


def compare(a, b):
    fa = sorted(os.path.basename(f) for f in glob.glob(os.path.join(a, "*.npy")))
    fb = sorted(os.path.basename(f) for f in glob.glob(os.path.join(b, "*.npy")))
    assert fa and fa == fb, "no outputs, or different sets of outputs"
    bad, elems, nan = [], 0, 0
    for f in fa:
        x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
        elems += x.size
        nan += int(np.isnan(x).sum())
        if not (x.shape == y.shape and x.tobytes() == y.tobytes() and np.array_equal(x, y, equal_nan=True)):
            bad.append(f)
    print("%d outputs, %d values (%d NaN), identical: %d, different: %d %s" % (len(fa), elems, nan, len(fa) - len(bad), len(bad), bad))
    return not bad


if __name__ == "__main__":
    if sys.argv[1] == "run":
        run(sys.argv[2])
    else:
        sys.exit(0 if compare(sys.argv[2], sys.argv[3]) else 1)
