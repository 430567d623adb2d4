"""TEST INFRASTRUCTURE ONLY: ctypes bindings for the CPU oracle and (where built) the reference.

* ``OracleMOIHGP``  - oracle/_build/liboracle.so, the Eigen-free restatement (moihgp_oracle.cpp).
* ``RefMOIHGP``     - oracle/_ref/libmoihgp_ref*.so, the UNMODIFIED reference sources compiled against
                      the Eigen-API shim (only exists where /root/reference was present at build time).

Only tests/, ``__graft_entry__.smoke()``, bench.py's CPU-baseline legs and scripts/gpu_fuzz.py may import this module.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_dp = ctypes.POINTER(ctypes.c_double)
_vp = ctypes.c_void_p
_sz = ctypes.c_size_t


def _P(a):
    if a is None:
        return ctypes.cast(None, _dp)
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_dp)


def build(force=False):
    """Compile liboracle.so (and oracle/_ref when the reference tree is present)."""
    so = os.path.join(_HERE, "_build", "liboracle.so")
    src = os.path.join(_HERE, "moihgp_oracle.cpp")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "_build/liboracle.so"], stdout=subprocess.DEVNULL)
    if os.path.isdir("/root/reference/moihgp/include") and (force or not os.path.exists(os.path.join(_HERE, "_ref", "libmoihgp_ref_probe_O3.so"))
                                                            or os.path.getmtime(os.path.join(_HERE, "_ref", "libmoihgp_ref_probe_O3.so")) < os.path.getmtime(os.path.join(_HERE, "ref_probe.cpp"))):
        subprocess.check_call(["make", "-C", _HERE, "ref"], stdout=subprocess.DEVNULL)
    return so


_oracle_lib = None


def oracle_lib():
    global _oracle_lib
    if _oracle_lib is None:
        lib = ctypes.CDLL(build())
        lib.oracle_new.restype = _vp
        lib.oracle_new.argtypes = [ctypes.c_int, ctypes.c_double, _sz, _sz, ctypes.c_int]
        lib.oracle_del.argtypes = [_vp]
        lib.oracle_set_intended_hda.argtypes = [_vp, ctypes.c_int]
        lib.oracle_igp_dim.restype = _sz
        lib.oracle_igp_dim.argtypes = [_vp]
        lib.oracle_num_param.restype = _sz
        lib.oracle_num_param.argtypes = [_vp]
        lib.oracle_update.argtypes = [_vp, _dp]
        lib.oracle_get_params.argtypes = [_vp, _dp]
        lib.oracle_get_U.argtypes = [_vp, _dp]
        lib.oracle_step1.argtypes = [_vp] + [_dp] * 6
        lib.oracle_step2.argtypes = [_vp] + [_dp] * 5
        lib.oracle_step3.argtypes = [_vp] + [_dp] * 4
        lib.oracle_step4.argtypes = [_vp] + [_dp] * 3
        lib.oracle_lik1.restype = ctypes.c_double
        lib.oracle_lik1.argtypes = [_vp, _dp, _dp, _dp, _dp, ctypes.c_int]
        lib.oracle_lik2.restype = ctypes.c_double
        lib.oracle_lik2.argtypes = [_vp, _dp, _dp, ctypes.c_int]
        lib.oracle_ihgp_consts.restype = _sz
        lib.oracle_ihgp_consts.argtypes = [_vp, _sz, _dp]
        lib.oracle_ihgp_iters.argtypes = [_vp, _sz, ctypes.POINTER(ctypes.c_int)]
        lib.oracle_smoother_consts.argtypes = [_vp, _sz, ctypes.c_int, _dp, _dp]
        lib.oracle_ihgp_smooth.argtypes = [_vp, _sz, ctypes.c_int, _dp, _sz, _dp]
        lib.oracle_objective.restype = ctypes.c_double
        lib.oracle_objective.argtypes = [_vp, _dp, _sz, _sz, _dp, _dp, _dp, ctypes.c_int]
        lib.oracle_filter_smoother_nll.argtypes = [_vp, _dp, _sz, _sz, _dp, _dp, _dp, _dp, _dp, ctypes.c_int, ctypes.c_int]
        _oracle_lib = lib
    return _oracle_lib


def consts_layout(d):
    """Names/shapes of the flat per-latent constant vector (oracle_ihgp_consts / probeXX_ihgp_consts)."""
    lay = [("A", (d, d)), ("Q", (d, d)), ("K", (d,)), ("S", ()), ("PF", (d, d)), ("HA", (d,)), ("AKHA", (d, d))]
    for k in range(3):
        lay += [("dS%d" % k, ()), ("dA%d" % k, (d, d)), ("dK%d" % k, (d,)), ("dAKHA%d" % k, (d, d)), ("HdA%d" % k, (d,))]
    return lay


def unpack_consts(flat, d):
    out, o = {}, 0
    for name, shp in consts_layout(d):
        n = int(np.prod(shp)) if shp else 1
        out[name] = flat[o:o + n].reshape(shp) if shp else float(flat[o])
        o += n
    return out


class OracleMOIHGP:
    """The CPU restatement, with the reference's MOIHGP method names (moihgp.h:76-757)."""

    def __init__(self, dt, num_output, num_latent, kernel="Matern32", threading=False):
        self.lib = oracle_lib()
        self.kernel = {"Matern32": 32, "Matern52": 52}[kernel]
        self.p, self.L = num_output, num_latent
        self.h = self.lib.oracle_new(self.kernel, dt, num_output, num_latent, int(threading))
        self.d = int(self.lib.oracle_igp_dim(self.h))
        self.num_param = int(self.lib.oracle_num_param(self.h))

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.oracle_del(self.h)
            self.h = None

    def set_intended_hda(self, on):
        self.lib.oracle_set_intended_hda(self.h, int(on))

    def update(self, params):
        params = np.ascontiguousarray(params, dtype=np.float64)
        assert params.size == self.num_param
        self.lib.oracle_update(self.h, _P(params))

    @property
    def params(self):
        out = np.zeros(self.num_param)
        self.lib.oracle_get_params(self.h, _P(out))
        return out

    @property
    def U(self):
        out = np.zeros((self.p, self.L))
        self.lib.oracle_get_U(self.h, _P(out))
        return out

    def step(self, x, y=None, dx=None):
        x = np.ascontiguousarray(x, dtype=np.float64)
        xn = np.zeros_like(x)
        yh = np.zeros(self.p)
        if y is None:
            self.lib.oracle_step4(self.h, _P(x), _P(xn), _P(yh))
            return xn, yh
        y = np.ascontiguousarray(y, dtype=np.float64)
        if dx is None:
            self.lib.oracle_step3(self.h, _P(x), _P(y), _P(xn), _P(yh))
            return xn, yh
        dx = np.ascontiguousarray(dx, dtype=np.float64)
        dxn = np.zeros_like(dx)
        self.lib.oracle_step1(self.h, _P(x), _P(y), _P(dx), _P(xn), _P(yh), _P(dxn))
        return xn, yh, dxn

    def negLogLikelihood(self, x, y, dx=None, literal=False):
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64)
        if dx is None:
            return float(self.lib.oracle_lik2(self.h, _P(x), _P(y), int(literal)))
        dx = np.ascontiguousarray(dx, dtype=np.float64)
        g = np.zeros(self.num_param)
        loss = float(self.lib.oracle_lik1(self.h, _P(x), _P(y), _P(dx), _P(g), int(literal)))
        return loss, g

    def ihgp_consts(self, l):
        flat = np.zeros(256)
        n = int(self.lib.oracle_ihgp_consts(self.h, l, _P(flat)))
        return unpack_consts(flat[:n], self.d)

    def ihgp_iters(self, l):
        out = (ctypes.c_int * 8)()
        self.lib.oracle_ihgp_iters(self.h, l, out)
        return list(out)

    def smoother_consts(self, l, mode):
        G = np.zeros((self.d, self.d))
        P = np.zeros((self.d, self.d))
        self.lib.oracle_smoother_consts(self.h, l, mode, _P(G), _P(P))
        return G, P

    def ihgp_smooth(self, l, mode, X):
        X = np.ascontiguousarray(X, dtype=np.float64)
        Xs = np.zeros_like(X)
        self.lib.oracle_ihgp_smooth(self.h, l, mode, _P(X), X.shape[0], _P(Xs))
        return Xs

    def objective(self, Y, x0=None, dx0=None, literal=False):
        """Sum over sequences of the RegressionObjective loop.  Y: [N,T,p] or [T,p]."""
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        if Y.ndim == 2:
            Y = Y[None]
        N, T, _ = Y.shape
        x = np.zeros((N, self.L, self.d)) if x0 is None else np.array(x0, dtype=np.float64).reshape(N, self.L, self.d).copy()
        dx = np.zeros((N, self.L, 3, self.d)) if dx0 is None else np.array(dx0, dtype=np.float64).reshape(N, self.L, 3, self.d).copy()
        g = np.zeros(self.num_param)
        loss = float(self.lib.oracle_objective(self.h, _P(Y), N, T, _P(x), _P(dx), _P(g), int(literal)))
        return loss, g, x, dx

    def filter_smoother_nll(self, Y, x0=None, smoother_mode=1, want_yhat=False, nthreads=1, want_states=True):
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        if Y.ndim == 2:
            Y = Y[None]
        N, T, _ = Y.shape
        x = np.zeros((N, self.L, self.d)) if x0 is None else np.array(x0, dtype=np.float64).reshape(N, self.L, self.d).copy()
        X = np.zeros((N, T, self.L, self.d)) if want_states else None
        Xs = np.zeros((N, T, self.L, self.d)) if (want_states and smoother_mode >= 0) else None
        Yhat = np.zeros((N, T, self.p)) if want_yhat else None
        nll = np.zeros(N)
        self.lib.oracle_filter_smoother_nll(self.h, _P(Y), N, T, _P(x), _P(X), _P(Xs), _P(Yhat), _P(nll), smoother_mode, nthreads)
        return {"X": X, "Xs": Xs, "Yhat": Yhat, "nll": nll, "xT": x}


def ref_available():
    return os.path.exists(os.path.join(_HERE, "_ref", "libmoihgp_ref_probe.so"))


class RefMOIHGP:
    """The reference itself (shim-compiled): gp32_* from src/wrapper.cpp for Matern32, and the
    probe52_* harness (oracle/ref_probe.cpp) for Matern52, which wrapper.cpp cannot reach (Q7)."""

    def __init__(self, dt, num_output, num_latent, kernel="Matern32", threading=False):
        self.p, self.L = num_output, num_latent
        self.dt = dt
        self.kernel = kernel
        if kernel == "Matern32":
            # -O0 build for the threaded path (moihgp.h:45-72 UB), -O2 build otherwise
            name = "libmoihgp_ref.so" if threading else "libmoihgp_ref_O2.so"
            self.lib = ctypes.CDLL(os.path.join(_HERE, "_ref", name))
            pre = "gp32_"
        else:
            self.lib = ctypes.CDLL(os.path.join(_HERE, "_ref", "libmoihgp_ref_probe.so"))
            pre = "probe52_"
        self.probe = ctypes.CDLL(os.path.join(_HERE, "_ref", "libmoihgp_ref_probe.so"))
        f = lambda n: getattr(self.lib, pre + n)
        f("new").restype = _vp
        f("new").argtypes = [ctypes.c_double, _sz, _sz, ctypes.c_bool]
        self.h = f("new")(dt, num_output, num_latent, threading)
        f("igp_dim").restype = _sz
        f("igp_dim").argtypes = [_vp]
        f("num_param").restype = _sz
        f("num_param").argtypes = [_vp]
        self.d = int(f("igp_dim")(self.h))
        self.num_param = int(f("num_param")(self.h))
        self._step1, self._step2, self._step3, self._step4 = f("step1"), f("step2"), f("step3"), f("step4")
        self._lik1, self._lik2, self._update, self._get = f("lik1"), f("lik2"), f("update"), f("get_params")
        self._step1.argtypes = [_vp] + [_dp] * 6
        self._step2.argtypes = [_vp] + [_dp] * 5
        self._step3.argtypes = [_vp] + [_dp] * 4
        self._step4.argtypes = [_vp] + [_dp] * 3
        self._lik1.restype = ctypes.c_double
        self._lik1.argtypes = [_vp] + [_dp] * 4
        self._lik2.restype = ctypes.c_double
        self._lik2.argtypes = [_vp] + [_dp] * 2
        self._update.argtypes = [_vp, _dp]
        self._get.argtypes = [_vp, _dp]
        for s in (self._step1, self._step2, self._step3, self._step4, self._update, self._get):
            s.restype = None

    def update(self, params):
        params = np.ascontiguousarray(params, dtype=np.float64)
        self._update(self.h, _P(params))

    @property
    def params(self):
        out = np.zeros(self.num_param)
        self._get(self.h, _P(out))
        return out

    def step(self, x, y=None, dx=None):
        x = np.ascontiguousarray(x, dtype=np.float64)
        xn = np.zeros_like(x)
        yh = np.zeros(self.p)
        if y is None:
            self._step4(self.h, _P(x), _P(xn), _P(yh))
            return xn, yh
        y = np.ascontiguousarray(y, dtype=np.float64)
        if dx is None:
            self._step3(self.h, _P(x), _P(y), _P(xn), _P(yh))
            return xn, yh
        dx = np.ascontiguousarray(dx, dtype=np.float64)
        dxn = np.zeros_like(dx)
        self._step1(self.h, _P(x), _P(y), _P(dx), _P(xn), _P(yh), _P(dxn))
        return xn, yh, dxn

    def negLogLikelihood(self, x, y, dx=None):
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64)
        if dx is None:
            return float(self._lik2(self.h, _P(x), _P(y)))
        dx = np.ascontiguousarray(dx, dtype=np.float64)
        g = np.zeros(self.num_param)
        loss = float(self._lik1(self.h, _P(x), _P(y), _P(dx), _P(g)))
        return loss, g

    def objective(self, Y, x0=None, dx0=None):
        """RegressionObjective::operator() loop (moihgp_regression.h:42-50) driven through the
        reference's own per-step entry points, exactly as online_learning.py:83-89 does."""
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        x = np.zeros((self.L, self.d)) if x0 is None else np.array(x0, dtype=np.float64)
        dx = np.zeros((self.L, 3, self.d)) if dx0 is None else np.array(dx0, dtype=np.float64)
        loss, grad = 0.0, np.zeros(self.num_param)
        for y in Y:
            xn, _, dxn = self.step(x, y, dx)
            l, g = self.negLogLikelihood(x, y, dx)
            loss += l
            grad += g
            x, dx = xn, dxn
        return loss, grad, x, dx

    def filter_nll(self, Y, x0=None):
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        x = np.zeros((self.L, self.d)) if x0 is None else np.array(x0, dtype=np.float64)
        X, Yhat, nll = [], [], 0.0
        for y in Y:
            nll += self.negLogLikelihood(x, y)
            x, yh = self.step(x, y)
            X.append(x.copy())
            Yhat.append(yh.copy())
        return np.array(X), np.array(Yhat), nll

    def ihgp_consts(self, igp_params):
        pre = "probe32_" if self.kernel == "Matern32" else "probe52_"
        fn = getattr(self.probe, pre + "ihgp_consts")
        fn.restype = _sz
        fn.argtypes = [ctypes.c_double, _dp, _dp]
        flat = np.zeros(256)
        n = int(fn(self.dt, _P(np.ascontiguousarray(igp_params, dtype=np.float64)), _P(flat)))
        return unpack_consts(flat[:n], self.d)

    def ihgp_smoother(self, igp_params, X):
        pre = "probe32_" if self.kernel == "Matern32" else "probe52_"
        fn = getattr(self.probe, pre + "ihgp_smoother")
        fn.restype = None
        fn.argtypes = [ctypes.c_double, _dp, _dp, _sz, _dp, _dp, _dp]
        X = np.ascontiguousarray(X, dtype=np.float64)
        Xs = np.zeros_like(X)
        P = np.zeros((self.d, self.d))
        G = np.zeros((self.d, self.d))
        fn(self.dt, _P(np.ascontiguousarray(igp_params, dtype=np.float64)), _P(X), X.shape[0], _P(Xs), _P(P), _P(G))
        return Xs, P, G


class RefPass:
    """The reference's own classes running the fused pass (oracle/ref_probe.cpp: run_pass), -O3 build, threading=false.
    One instance per host thread (the reference's objects are not thread-safe).  CPU arm of bench.py only."""

    def __init__(self, dt, num_output, num_latent, kernel, params):
        self.lib = ctypes.CDLL(os.path.join(_HERE, "_ref", "libmoihgp_ref_probe_O3.so"))
        self.pre = "probe32_" if kernel == "Matern32" else "probe52_"
        f = lambda n: getattr(self.lib, self.pre + n)
        f("new").restype = _vp
        f("new").argtypes = [ctypes.c_double, _sz, _sz, ctypes.c_bool]
        f("update").argtypes = [_vp, _dp]
        f("run_pass").restype = ctypes.c_double
        f("run_pass").argtypes = [_vp, ctypes.c_double, _dp, _dp, _sz, _dp, _dp, ctypes.c_int]
        self.dt, self.p, self.L = dt, num_output, num_latent
        self.h = f("new")(dt, num_output, num_latent, False)
        params = np.ascontiguousarray(params, dtype=np.float64)
        f("update")(self.h, _P(params))
        self.igp = np.ascontiguousarray(params[num_output * num_latent + num_latent + 1:])
        self._run = f("run_pass")

    def run(self, Y, X=None, Xs=None, smooth=True):
        """Y [T][p] -> summed NLL (and, if given, the filtered / smoothed states [T][L][d])."""
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        return float(self._run(self.h, self.dt, _P(self.igp), _P(Y), Y.shape[0], _P(X), _P(Xs), int(smooth)))


def ref_pass_available():
    return os.path.exists(os.path.join(_HERE, "_ref", "libmoihgp_ref_probe_O3.so"))
