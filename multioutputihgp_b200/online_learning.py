"""Online learner with the reference's interface (moihgp/online_learning.py:10-115).

Same constructor, ``step(y)`` protocol, parameter bounds, EMA mean, sliding window and SciPy
L-BFGS-B settings (maxiter=5, maxls=3) as the reference.  The difference is where the work runs:
the window, the state carried in front of it and the model stay RESIDENT on the device
(``moihgp_cuda_online_*``): one objective evaluation is one CUDA-graph launch (parameters in,
polar factor, K-setup, whole-window objective, loss and gradient out) instead of 2 x window ctypes
calls (online_learning.py:83-89); the filter steps use the legacy per-observation symbols.
A window with missing observations takes the reference's per-observation loop.
"""
import numpy as np
try:
    from scipy.optimize.lbfgsb import _minimize_lbfgsb, MemoizeJac
except Exception:  # newer SciPy
    from scipy.optimize._lbfgsb_py import _minimize_lbfgsb
    try:
        from scipy.optimize._optimize import MemoizeJac
    except Exception:
        from scipy.optimize.optimize import MemoizeJac

from .batched import MOIHGPSequences
from .pywrapper import MOIHGP


class MOIHGPOnlineLearning:

    def __init__(self, dt, num_output, num_latent, gamma, x_init=None, windowsize=None, kernel="Matern32", threading=False):
        self.moihgp = MOIHGP(dt, num_output, num_latent, kernel=kernel, threading=threading)
        # whole-window objective on the GPU, on the SAME device model as self.moihgp (one handle: one update serves both)
        self._seq = MOIHGPSequences.adopt(self.moihgp)
        self._held = None                                  # the parameters the device model holds, when known
        self.num_output = num_output
        self.num_latent = num_latent
        self.ihgp_dim = self.moihgp.igp_dim
        self.ihgp_nparam = self.moihgp.num_igp_param
        self.parameter_bounds = [(-np.inf, np.inf)] * (num_output * num_latent) + [(1e-4, np.inf)] * num_latent + \
            [(1e-4, 1e+2)] + [(1e-2, 1e+2), (1e-2, 1e+2), (1e-4, 1e+2)] * num_latent      # online_learning.py:18-28
        self.gamma = gamma
        self.x = np.zeros((num_latent, self.ihgp_dim), dtype=np.float64) if x_init is None else x_init
        self.dx = np.zeros((num_latent, self.ihgp_nparam, self.ihgp_dim), dtype=np.float64)
        self.xinit = np.zeros((num_latent, self.ihgp_dim), dtype=np.float64) if x_init is None else x_init
        self.dxinit = np.zeros((num_latent, self.ihgp_nparam, self.ihgp_dim), dtype=np.float64)
        self.hess_inv = np.eye(len(self.moihgp.params))
        self.buffer = []
        self.windowsize = 1 if windowsize is None else windowsize
        self.ma = None
        self.dma = np.zeros((num_output,), dtype=np.float64)
        self._resident = self._seq.online_begin(self.windowsize)
        if not self._resident and num_latent > 64:
            raise ValueError("MOIHGPOnlineLearning: " + self._seq._lib.moihgp_cuda_last_error(self._seq._h).decode())
        if self._resident:
            self._seq.online_set_proximal(None)           # the proximal term stays here (hess_inv solve, as the reference's)

    @staticmethod
    def _seq_kernel(kernel):
        import os
        # gp52_* binds Matern-3/2 unless MOIHGP_GP52_MATERN52=1 (wrapper.cpp:22, SURVEY Q7): stay consistent
        if kernel == "Matern52" and os.environ.get("MOIHGP_GP52_MATERN52", "0")[:1] != "1":
            return "Matern32"
        return kernel

    def _update(self, params):
        if self._held is not None and np.array_equal(self._held, params):
            return                                         # the model already holds them (left there by the last evaluation)
        self._seq.update(params)
        self._held = np.array(params, dtype=np.float64, copy=True)

    def step(self, y=None):
        if self.ma is None:                                                  # online_learning.py:54-64
            self.ma = y.copy()
            self.ma[np.isnan(self.ma)] = 0.0
        else:
            ma_old = self.ma.copy()
            for i, yi in enumerate(y):
                if np.isnan(yi):
                    self.ma[i] += self.dma[i]
                else:
                    self.ma[i] = 0.5 * yi + 0.5 * ma_old[i]
            self.dma = self.ma - ma_old
        self.buffer.append(y)
        if self._resident:
            # window slide + carried-state step on the device, with this learner's own centre (the exponential mean)
            self._seq.online_push(y, ma_given=self.ma)
            while len(self.buffer) > self.windowsize:
                self.buffer.pop(0)
        else:
            while len(self.buffer) > self.windowsize:                        # online_learning.py:66-68 (Q12)
                self.buffer.pop(0)
                self.xinit, _, self.dxinit = self.moihgp.step(self.xinit, y=self.buffer[0] - self.ma, dx=self.dxinit)
        xnew, yhat, dxnew = self.moihgp.step(self.x, y=y - self.ma, dx=self.dx)
        yhat += self.ma
        self.x = xnew
        self.dx = dxnew
        oldparams = self.moihgp.params.copy()
        window = np.array(self.buffer) - self.ma
        has_nan = bool(np.isnan(window).any())
        if self._resident and has_nan:
            self.xinit, self.dxinit = self._seq.online_state()

        def objective(params, eval_gradient=True):                           # online_learning.py:74-98
            dparams = params - oldparams
            p = np.linalg.solve(self.hess_inv, dparams)
            if self._resident and not has_nan:
                l, g = self._seq.online_objective(params)                    # update(params) + window loop: one graph launch
                self._held = np.array(params, dtype=np.float64, copy=True)
                loss = self.gamma * 0.5 * dparams.dot(p) + l
                return (loss, self.gamma * p + g) if eval_gradient else loss
            self._update(params)
            if has_nan:
                # missing observations: per-observation symbols, exactly the reference's loop
                xt, dxt = self.xinit, self.dxinit
                loss = self.gamma * 0.5 * dparams.dot(p)
                grad = self.gamma * p
                for yt in window:
                    xtnew, _, dxtnew = self.moihgp.step(xt, y=yt, dx=dxt)
                    l, g = self.moihgp.negLogLikelihood(xt, yt, dxt)
                    loss += l
                    grad += g
                    xt, dxt = xtnew, dxtnew
                return (loss, grad) if eval_gradient else loss
            l, g = self._seq.objective(window[None], x0=self.xinit[None], dx0=self.dxinit[None])
            loss = self.gamma * 0.5 * dparams.dot(p) + l
            if eval_gradient:
                return loss, self.gamma * p + g
            return loss

        fun = MemoizeJac(objective)
        jac = fun.derivative
        res = _minimize_lbfgsb(fun, oldparams, bounds=self.parameter_bounds, jac=jac, maxiter=5, maxls=3)
        newparams = res['x']
        self._update(newparams)
        self.hess_inv = res['hess_inv'].todense()
        return yhat

    @property
    def covariance(self):
        return self.moihgp.covariance

    @property
    def params(self):
        return self.moihgp.params
