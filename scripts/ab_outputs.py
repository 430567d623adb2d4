"""Outputs of seeded calls at L <= 64 shapes, one per path and projection variant, as SHA-256 digests of their bytes: run it
in two trees (for instance a change and its parent) and compare the two JSON files to show that the results are bit for bit
the same.

    python scripts/ab_outputs.py OUT.json            (in each tree)
    python scripts/ab_outputs.py --compare A.json B.json"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)

# (kernel, p, L, N, T, path, offset Y): many-chains path, chunked scan with each projection kernel (k_project_rows,
# k_project_mma, k_project for odd p and for an offset Y), missing outputs
SHAPES = [
    ("Matern52", 16, 8, 64, 700, "chain", False),
    ("Matern32", 64, 32, 4, 3000, "scan", False),
    ("Matern32", 256, 64, 1, 4000, "scan", False),
    ("Matern52", 1000, 64, 1, 600, "scan", False),
    ("Matern32", 33, 17, 3, 900, "scan", False),
    ("Matern52", 64, 48, 2, 1000, "scan", True),
]


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(np.asarray(a, dtype=np.float64)).tobytes()).hexdigest()


def run(out):
    import torch
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_data, make_params
    res = {}
    for kernel, p, L, N, T, path, offset in SHAPES:
        rng = np.random.default_rng(p * 1000 + L)
        params = make_params(rng, p, L, kernel)
        m = MOIHGPSequences(0.1, p, L, kernel, True)
        m.update(params)
        m.set_path(path)
        Y = np.stack([make_data(rng, p, L, T) for _ in range(N)])
        Y[0, T // 2, 1] = np.nan
        tag = "%s-p%dL%d-N%dT%d-%s%s" % (kernel, p, L, N, T, path, "-offset" if offset else "")
        res[tag + ":U"] = digest(m.U)
        if offset:
            buf = torch.zeros(Y.size + 1, dtype=torch.float64, device="cuda")
            Yd = buf[1:].view(*Y.shape)
            Yd.copy_(torch.from_numpy(Y))
            d = m.igp_dim
            X, Xs = (torch.zeros((N, T, L, d), dtype=torch.float64, device="cuda") for _ in range(2))
            Yhat = torch.zeros((N, T, p), dtype=torch.float64, device="cuda")
            m.filter_smoother_nll_device(Yd, smoother_mode=1, X=X, Xs=Xs, Yhat=Yhat)
            torch.cuda.synchronize()
            r = {"X": X.cpu().numpy(), "Xs": Xs.cpu().numpy(), "Yhat": Yhat.cpu().numpy()}
        else:
            r = m.filter_smoother_nll(Y, smoother_mode=1, want_yhat=True)
        for k, v in r.items():
            if v is not None:
                res[tag + ":" + k] = digest(v)
        Yc = Y.copy()
        Yc[0, T // 2, 1] = 0.0
        res[tag + ":nll_steps"] = digest(m.nll_steps(Yc)["nll_steps"])
        loss, grad = m.objective(Yc)
        res[tag + ":objective"] = digest(np.concatenate([[loss], grad]))
        res[tag + ":sample"] = digest(m.sample_posterior(Yc, 2, 12345, want_states=True)["X"])
    with open(out, "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
    print("%d digests -> %s" % (len(res), out))


def compare(a, b):
    A, B = json.load(open(a)), json.load(open(b))
    diff = sorted(k for k in set(A) | set(B) if A.get(k) != B.get(k))
    print("%d outputs compared, %d differ%s" % (len(set(A) | set(B)), len(diff), (": " + ", ".join(diff)) if diff else ""))
    return 1 if diff else 0


if __name__ == "__main__":
    if sys.argv[1] == "--compare":
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    run(sys.argv[1])
