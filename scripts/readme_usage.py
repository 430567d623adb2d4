"""The usage snippet of README.md, run as written (on a B200): every call of the snippet on a small model."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from multioutputihgp_b200 import MOIHGPSequences, MOIHGPOnlineLearning

rng = np.random.default_rng(0)
m = MOIHGPSequences(dt=0.1, num_output=16, num_latent=8, kernel="Matern52")
params = m.params
params[16 * 8:16 * 8 + 8] = 1.0 + 0.1 * np.arange(8)
m.update(params)
Y = rng.standard_normal((6, 300, 16))
r = m.filter_smoother_nll(Y)
print("filter_smoother_nll:", {k: np.asarray(v).shape for k, v in r.items() if v is not None})
loss, grad = m.objective(Y)[:2]
print("objective:", loss, grad.shape)
m.bind(Y)
loss_b, grad_b = m.objective_bound()[:2]
assert abs(loss_b - loss) <= 1e-12 * abs(loss) and np.allclose(grad_b, grad, rtol=1e-12, atol=0)
e = m.nll_steps(Y)
assert e["nll_steps"].shape == (6, 300) and np.allclose(e["nll_steps"].sum(axis=1), r["nll"], rtol=1e-10, atol=0)
learner = MOIHGPOnlineLearning(0.1, 8, 4, gamma=0.9, windowsize=1)
for t in range(5):
    yhat = learner.step(rng.standard_normal(8))
print("online step:", yhat.shape)
print("README usage ok")
