"""Checksums of seeded sample_posterior_dev outputs at the config-3 and config-4 shapes, on both variants of the sampler
(set_path 1: time-chunked, 2: one pass): run it against two builds of the library (MOIHGP_B200_LIB selects one) and compare
the two JSON files to show that the draws are bit for bit the same.  The outputs stay on the device: each is reduced to
two 64-bit checksums of its bit patterns (a plain and an index-weighted wrap-around sum).

    MOIHGP_B200_LIB=<lib> python scripts/ab_sample_outputs.py OUT.json
    python scripts/ab_outputs.py --compare A.json B.json"""
import json
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch

from bench import model_params, DT
from multioutputihgp_b200 import MOIHGPSequences, _lib

# name, kernel, p, L, N, T, S (config-3: 4096 sequences of 16384 steps; config-4: one sequence of 10^7 steps)
SHAPES = [("c3", "Matern52", 16, 8, 4096, 16384, 1), ("c4", "Matern32", 64, 32, 1, 10000000, 2)]


def checksum(x):
    v = x.contiguous().view(torch.int64).ravel()
    w = (torch.arange(v.numel(), device=v.device, dtype=torch.int64) % 1000003) * 2 + 1
    return [int(v.sum()), int((v * w).sum())]


def run(out):
    res = {}
    print("library:", _lib.LIB_PATH)
    dev = torch.device("cuda", 0)
    f64 = dict(dtype=torch.float64, device=dev)
    for name, kernel, p, L, N, T, S in SHAPES:
        params, Hmix = model_params(p, L, kernel, 1234)
        m = MOIHGPSequences(DT, p, L, kernel, threading=True)
        m.update(params)
        d = m.igp_dim
        t = torch.arange(T, **f64)[None, :, None] * DT
        k = torch.arange(N, **f64)[:, None, None]
        Fl = torch.sin(t * (1.0 + 3.0 * torch.arange(L, **f64) / max(L - 1, 1))[None, None, :] + 0.1 * k)
        Y = (Fl @ torch.from_numpy(Hmix.T.copy()).to(dev) + 0.05 * torch.cos(7.3 * t + torch.arange(p, **f64) + k)).contiguous()
        del Fl
        for path in (1, 2):
            m.set_path(path)
            Xs, X, F = torch.zeros((N, T, L, d), **f64), torch.zeros((S, N, T, L, d), **f64), torch.zeros((S, N, T, L), **f64)
            m.sample_posterior_device(Y, 777, Xs=Xs, X=X, F=F)
            torch.cuda.synchronize()
            for key, v in (("Xs", Xs), ("X", X), ("F", F)):
                res["%s-path%d:%s" % (name, path, key)] = checksum(v)
            del Xs, X, F
        del Y
        torch.cuda.empty_cache()
    with open(out, "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
    print("%d checksums -> %s" % (len(res), out))


if __name__ == "__main__":
    run(sys.argv[1])
