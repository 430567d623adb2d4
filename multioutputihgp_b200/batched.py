"""Whole-sequence interface to the B200 library (the moihgp_cuda_* entry points).

``MOIHGPSequences`` keeps the reference's model vocabulary (``update(params)``, ``params``,
``negLogLikelihood``) but takes whole sequences ``Y[N][T][p]`` where the reference's callers loop
over observations (RegressionObjective::operator(), moihgp_regression.h:34-52; OnlineObjective,
moihgp_online.h:40-72; MOIHGPRegression::predict, moihgp_regression.h:127-139).

NumPy arrays go through the host entry points (copies inside the call); torch CUDA tensors go
through the ``*_dev`` entry points on torch's current stream and stay resident in HBM.
Every array a caller passes is checked against the sizes include/moihgp_b200.h specifies before its address reaches the
library, which receives bare addresses and cannot check them.
"""
import ctypes

import numpy as np

from . import _lib

SMOOTH_NONE, SMOOTH_REFERENCE_LITERAL, SMOOTH_RTS = -1, 0, 1
_KERNELS = {"Matern32": 32, "Matern52": 52}


def _refuse(where, name, want, got):
    raise ValueError("%s: %s must be %s, got %s" % (where, name, want, got))


def _host(where, **args):
    """Host pointer arguments, args[name] = (array or None, element count): each array as C-contiguous float64 (a copy if it
    is not one already) holding exactly `count` values.  Returns the pointers in argument order; each keeps its array alive."""
    ptrs = []
    for name, (a, count) in args.items():
        if a is not None:
            a = np.ascontiguousarray(a, dtype=np.float64)
            if a.size != count:
                _refuse(where, name, "%d values" % count, a.size)
            a = a.ctypes.data_as(_lib.c_double_p)
        ptrs.append(a)
    return ptrs


def _host_seqs(where, name, A, tail):
    """Host sequences A [N,T,*tail] (or one sequence [T,*tail]) -> (pointer as _host, N, T)."""
    A = np.ascontiguousarray(A, dtype=np.float64)
    if A.ndim == len(tail) + 1:
        A = A[None]
    if A.shape[2:] != tuple(tail) or A.ndim != len(tail) + 2:
        _refuse(where, name, "[N,T,{0}] or [T,{0}]".format(",".join(map(str, tail))), "shape %s" % (A.shape,))
    return A.ctypes.data_as(_lib.c_double_p), A.shape[0], A.shape[1]


def _dev(where, **args):
    """Device pointer arguments, args[name] = (tensor or None, element count): torch tensors, float64, contiguous, exactly
    `count` elements, all on the CUDA device of the first.  Every dtype, layout and size is checked before any device."""
    import torch
    given = [(name, t, count) for name, (t, count) in args.items() if t is not None]
    for name, t, count in given:
        if not isinstance(t, torch.Tensor):
            _refuse(where, name, "a torch CUDA tensor", type(t).__name__)
        if t.dtype != torch.float64:
            _refuse(where, name, "torch.float64", t.dtype)
        if not t.is_contiguous():
            _refuse(where, name, "contiguous", "strides %s" % (t.stride(),))
        if t.numel() != count:
            _refuse(where, name, "%d elements" % count, t.numel())
    for name, t, _ in given:
        if not t.is_cuda:
            _refuse(where, name, "a CUDA tensor", t.device)
        if t.device != given[0][1].device:
            _refuse(where, name, "on %s like %s" % (given[0][1].device, given[0][0]), t.device)
    return [None if t is None else t.data_ptr() for t, _ in args.values()]


def _addr(a):
    """address of an array this module allocated (None passes through)"""
    return None if a is None else a.ctypes.data


def _torch_stream(device):
    """cudaStream_t of torch's current stream on `device`.  torch reports its default stream as handle 0, which the C ABI
    reads as "the handle's own stream": pass CUDA's explicit alias of the legacy default stream (cudaStreamLegacy = 0x1)
    instead, so that the library's kernels are ordered with torch's own work on that stream."""
    import torch
    return torch.cuda.current_stream(device).cuda_stream or 1


class MOIHGPSequences(object):

    def __init__(self, dt, num_output, num_latent, kernel="Matern32", threading=False, device=-1):
        self._lib = _lib.load()
        h = ctypes.c_void_p()
        rc = self._lib.moihgp_cuda_create(ctypes.byref(h), _KERNELS[kernel], dt, num_output, num_latent, int(threading), device)
        if rc != 0 or not h:
            raise RuntimeError("moihgp_cuda_create failed (no B200-class CUDA device? there is no CPU fallback)")
        self._h = h
        self.dt, self.num_output, self.num_latent, self.kernel = dt, num_output, num_latent, kernel
        self.igp_dim = int(self._lib.moihgp_cuda_igp_dim(h))
        self.num_param = int(self._lib.moihgp_cuda_num_param(h))
        self.num_igp_param = int(self._lib.moihgp_cuda_num_igp_param(h))

    @classmethod
    def adopt(cls, model):
        """The whole-sequence interface on the handle of an existing per-observation model (``pywrapper.MOIHGP``): ONE model on
        the device, shared - ``update`` through either object is seen by both.  ``model`` keeps ownership of the handle (and
        is kept alive by the returned object)."""
        import ctypes as _ct
        self = cls.__new__(cls)
        self._lib = _lib.load()
        self._h = _ct.c_void_p(model.handle)
        self._owner = model
        self.dt, self.num_output, self.num_latent, self.kernel = model.dt, model.num_output, model.num_latent, None
        self.igp_dim = int(self._lib.moihgp_cuda_igp_dim(self._h))
        self.num_param = int(self._lib.moihgp_cuda_num_param(self._h))
        self.num_igp_param = int(self._lib.moihgp_cuda_num_igp_param(self._h))
        return self

    def __del__(self):
        if getattr(self, "_h", None) and getattr(self, "_owner", None) is None:
            self._lib.moihgp_cuda_destroy(self._h)
        self._h = None

    def _dims(self, where, Y):
        """(N, T, L, d) of device sequences Y [N,T,p]"""
        if getattr(Y, "ndim", None) != 3:
            _refuse(where, "Y", "a [N,T,p] tensor", "shape %s" % (getattr(Y, "shape", type(Y).__name__),))
        return Y.shape[0], Y.shape[1], self.num_latent, self.igp_dim

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError("libmoihgp: " + self._lib.moihgp_cuda_last_error(self._h).decode())

    # ---- model ------------------------------------------------------------------------------
    def update(self, params):
        self._check(self._lib.moihgp_cuda_update(self._h, *_host("update", params=(params, self.num_param))))

    @property
    def params(self):
        out = np.zeros(self.num_param)
        self._check(self._lib.moihgp_cuda_get_params(self._h, out.ctypes.data_as(_lib.c_double_p)))
        return out

    @property
    def U(self):
        out = np.zeros((self.num_output, self.num_latent))
        self._check(self._lib.moihgp_cuda_get_U(self._h, out.ctypes.data_as(_lib.c_double_p)))
        return out

    def latent_consts(self, l):
        flat = np.zeros(256)
        n = self._lib.moihgp_cuda_latent_consts(self._h, l, flat.ctypes.data_as(_lib.c_double_p), flat.size)
        if n < 0:
            raise RuntimeError("moihgp_cuda_latent_consts failed")
        d, out, o = self.igp_dim, {}, 0
        lay = [("A", (d, d)), ("Q", (d, d)), ("K", (d,)), ("S", ()), ("PF", (d, d)), ("HA", (d,)), ("AKHA", (d, d))]
        for k in range(3):
            lay += [("dS%d" % k, ()), ("dA%d" % k, (d, d)), ("dK%d" % k, (d,)), ("dAKHA%d" % k, (d, d)), ("HdA%d" % k, (d,))]
        for name, shp in lay:
            m = int(np.prod(shp)) if shp else 1
            out[name] = flat[o:o + m].reshape(shp).copy() if shp else float(flat[o])
            o += m
        return out

    def latent_iters(self, l):
        out = (ctypes.c_int * 8)()
        self._check(self._lib.moihgp_cuda_latent_iters(self._h, l, out))
        return list(out)

    def smoother_consts(self, l, mode):
        d = self.igp_dim
        G, P = np.zeros((d, d)), np.zeros((d, d))
        self._check(self._lib.moihgp_cuda_smoother_consts(self._h, l, mode, G.ctypes.data_as(_lib.c_double_p), P.ctypes.data_as(_lib.c_double_p)))
        return G, P

    @property
    def nan_status(self):
        """0 / 1 / 2 (none / handled / overflow) for the last whole-sequence call; waits for the stream.  The *_device methods
        are asynchronous and cannot raise on an overflow of the missing-observation list themselves."""
        out = ctypes.c_int(0)
        self._check(self._lib.moihgp_cuda_nan_status(self._h, ctypes.byref(out)))
        return int(out.value)

    @property
    def launch_count(self):
        return int(self._lib.moihgp_cuda_launch_count(self._h))

    def set_path(self, path):
        """0 auto, 1 chunked scan, 2 many-chains (see moihgp_cuda_set_path)."""
        self._check(self._lib.moihgp_cuda_set_path(self._h, {"auto": 0, "scan": 1, "chain": 2}.get(path, path)))

    def set_chain_seqs_per_warp(self, n):
        """Tuning knob of the many-chains kernels (0 = automatic); see moihgp_cuda_set_chain_seqs_per_warp."""
        self._check(self._lib.moihgp_cuda_set_chain_seqs_per_warp(self._h, int(n)))

    def profile(self, enable):
        self._check(self._lib.moihgp_cuda_profile(self._h, int(enable)))

    def profile_read(self):
        """{kernel name: (total ms, launches)} since profile(True); clears the record."""
        out = {}
        for line in self._lib.moihgp_cuda_profile_read(self._h).decode().splitlines():
            name, ms, cnt = line.split()
            out[name] = (float(ms), int(cnt))
        return out

    def set_stream(self, cuda_stream_ptr):
        self._check(self._lib.moihgp_cuda_set_stream(self._h, cuda_stream_ptr))

    def synchronize(self):
        self._check(self._lib.moihgp_cuda_sync(self._h))

    # ---- fused pass: filter + smoother + NLL ----------------------------------------------------
    def filter_smoother_nll(self, Y, x0=None, smoother_mode=SMOOTH_REFERENCE_LITERAL, want_states=True, want_yhat=False, want_nll=True):
        """Y: [N,T,p] (or [T,p]) NumPy array -> dict of NumPy arrays X, Xs, Yhat, nll, xT.
        smoother_mode defaults to the reference's own recursion (IHGP::backwardSmoother as written, ihgp.h:108-113, SURVEY Q3 -
        unstable for some hyper-parameters, e.g. the default Matern-3/2 latent); SMOOTH_RTS is this library's extension."""
        p, L, d = self.num_output, self.num_latent, self.igp_dim
        Y, N, T = _host_seqs("filter_smoother_nll", "Y", Y, (p,))
        x0, = _host("filter_smoother_nll", x0=(x0, N * L * d))
        X = np.empty((N, T, L, d)) if want_states else None
        Xs = np.empty((N, T, L, d)) if (want_states and smoother_mode >= 0) else None
        Yhat = np.empty((N, T, p)) if want_yhat else None
        nll = np.empty(N) if want_nll else None
        xT = np.empty((N, L, d))
        self._check(self._lib.moihgp_cuda_filter_smoother_nll(self._h, Y, N, T, x0, smoother_mode, _addr(X), _addr(Xs), _addr(Yhat),
                                                              _addr(nll), _addr(xT)))
        return {"X": X, "Xs": Xs, "Yhat": Yhat, "nll": nll, "xT": xT}

    def filter_smoother_nll_values(self, Y, x0=None, smoother_mode=SMOOTH_REFERENCE_LITERAL, want_yhat=False):
        """The same pass returning only the function-value component H x = x(0) of the filtered / smoothed states,
        F and Fs [N,T,L] (d times fewer bytes across PCIe), plus nll, xT and optionally Yhat."""
        p, L, d = self.num_output, self.num_latent, self.igp_dim
        Y, N, T = _host_seqs("filter_smoother_nll_values", "Y", Y, (p,))
        x0, = _host("filter_smoother_nll_values", x0=(x0, N * L * d))
        F = np.empty((N, T, L))
        Fs = np.empty((N, T, L)) if smoother_mode >= 0 else None
        Yhat = np.empty((N, T, p)) if want_yhat else None
        nll, xT = np.empty(N), np.empty((N, L, d))
        self._check(self._lib.moihgp_cuda_filter_smoother_nll_values(self._h, Y, N, T, x0, smoother_mode, _addr(F), _addr(Fs), _addr(Yhat),
                                                                     _addr(nll), _addr(xT)))
        return {"F": F, "Fs": Fs, "Yhat": Yhat, "nll": nll, "xT": xT}

    def filter_smoother_nll_device(self, Y, x0=None, smoother_mode=SMOOTH_REFERENCE_LITERAL, X=None, Xs=None, Yhat=None, nll=None, xT=None):
        """Device-resident variant: all arguments are torch CUDA float64 tensors (outputs pre-allocated by the
        caller, any may be None); runs asynchronously on torch's current stream."""
        N, T, L, d = self._dims("filter_smoother_nll_device", Y)
        p = self.num_output
        ptr = _dev("filter_smoother_nll_device", Y=(Y, N * T * p), x0=(x0, N * L * d), X=(X, N * T * L * d), Xs=(Xs, N * T * L * d),
                   Yhat=(Yhat, N * T * p), nll=(nll, N), xT=(xT, N * L * d))
        self.set_stream(_torch_stream(Y.device))
        self._check(self._lib.moihgp_cuda_filter_smoother_nll_dev(self._h, ptr[0], N, T, ptr[1], smoother_mode, *ptr[2:]))

    # ---- per-step NLL terms (moihgp_cuda_nll_steps*) -----------------------------------------------------------
    def nll_steps(self, Y, x0=None):
        """Y: [N,T,p] (or [T,p]) NumPy array -> dict of NumPy arrays: nll_steps [N,T], the term MOIHGP::negLogLikelihood(x_{t-1},
        y_t) of every step (NaN for a row with a missing output), nll [N] (their sum, as filter_smoother_nll returns it) and xT
        [N,L,d].  Filter only: no smoother, no states."""
        L, d = self.num_latent, self.igp_dim
        Y, N, T = _host_seqs("nll_steps", "Y", Y, (self.num_output,))
        x0, = _host("nll_steps", x0=(x0, N * L * d))
        steps, nll, xT = np.empty((N, T)), np.empty(N), np.empty((N, L, d))
        self._check(self._lib.moihgp_cuda_nll_steps(self._h, Y, N, T, x0, _addr(steps), _addr(nll), _addr(xT)))
        return {"nll_steps": steps, "nll": nll, "xT": xT}

    def nll_steps_device(self, Y, nll_steps, x0=None, nll=None, xT=None):
        """Device-resident variant: torch CUDA float64 tensors, outputs pre-allocated by the caller (nll_steps [N,T] required,
        nll [N] and xT [N,L,d] may be None); runs asynchronously on torch's current stream."""
        N, T, L, d = self._dims("nll_steps_device", Y)
        ptr = _dev("nll_steps_device", Y=(Y, N * T * self.num_output), x0=(x0, N * L * d), nll_steps=(nll_steps, N * T), nll=(nll, N),
                   xT=(xT, N * L * d))
        self.set_stream(_torch_stream(Y.device))
        self._check(self._lib.moihgp_cuda_nll_steps_dev(self._h, ptr[0], N, T, *ptr[1:]))

    # ---- objective: NLL + gradient ----------------------------------------------------------------
    def objective(self, Y, x0=None, dx0=None, want_state=False):
        """sum over sequences and time of negLogLikelihood(x, y, dx, grad) with step v2 advancing the state
        (RegressionObjective::operator(), moihgp_regression.h:42-50).  Returns (loss, grad[, xT, dxT])."""
        L, d = self.num_latent, self.igp_dim
        Y, N, T = _host_seqs("objective", "Y", Y, (self.num_output,))
        x0, dx0 = _host("objective", x0=(x0, N * L * d), dx0=(dx0, N * L * 3 * d))
        loss = np.zeros(1)
        grad = np.zeros(self.num_param)
        xT = np.empty((N, L, d)) if want_state else None
        dxT = np.empty((N, L, 3, d)) if want_state else None
        self._check(self._lib.moihgp_cuda_objective(self._h, Y, N, T, x0, dx0, _addr(loss), _addr(grad), _addr(xT), _addr(dxT)))
        if want_state:
            return float(loss[0]), grad, xT, dxT
        return float(loss[0]), grad

    def objective_begin_device(self, Y, want_end=True):
        """Time-sharded evaluation, step 1 (torch CUDA tensor Y [N,T,p] = this rank's block of time): projection + summaries;
        returns the block's end state from a zero carry-in as (x [N,L,d], dx [N,L,3,d]) NumPy arrays (needs T % 256 == 0)."""
        N, T, L, d = self._dims("objective_begin_device", Y)
        Yp, = _dev("objective_begin_device", Y=(Y, N * T * self.num_output))
        self.set_stream(_torch_stream(Y.device))
        z = np.zeros((N, L, 4, d)) if want_end else None
        self._check(self._lib.moihgp_cuda_objective_begin_dev(self._h, Yp, N, T, _addr(z)))
        return (z[:, :, 0].copy(), z[:, :, 1:].copy()) if want_end else None

    def objective_begin_async(self, Y, zend=None):
        """Like objective_begin_device, without a host round trip: the block's end state from a zero carry-in goes to the
        torch CUDA tensor ``zend`` [N,L,4,d] (None on the last block); asynchronous on torch's current stream."""
        N, T, L, d = self._dims("objective_begin_async", Y)
        ptr = _dev("objective_begin_async", Y=(Y, N * T * self.num_output), zend=(zend, N * L * 4 * d))
        self.set_stream(_torch_stream(Y.device))
        self._check(self._lib.moihgp_cuda_objective_begin_async(self._h, ptr[0], N, T, ptr[1]))

    def carry_in_device(self, ends, block_lengths, rank, xin, dxin, x0=None, dx0=None):
        """This block's true carry-in from the all-gathered block ends ``ends`` [G,N,L,4,d] (torch CUDA tensors throughout):
        z_in(g+1) = T(n_g) z_in(g) + ends_g chained over g < rank; written to xin [N,L,d], dxin [N,L,3,d]."""
        G = len(block_lengths)
        lens = (ctypes.c_longlong * G)(*[int(b) for b in block_lengths])
        N, L, d = xin.shape[0], self.num_latent, self.igp_dim
        ptr = _dev("carry_in_device", ends=(ends, G * N * L * 4 * d), x0=(x0, N * L * d), dx0=(dx0, N * L * 3 * d), xin=(xin, N * L * d),
                   dxin=(dxin, N * L * 3 * d))
        self._check(self._lib.moihgp_cuda_carry_in_dev(self._h, ptr[0], G, lens, int(rank), N, *ptr[1:]))

    def objective_finish_device(self, Y, loss, grad, x0=None, dx0=None):
        """Step 2: loss / grad of the block from its true carry-in (torch CUDA tensors), reusing step 1's projection."""
        N, T, L, d = self._dims("objective_finish_device", Y)
        ptr = _dev("objective_finish_device", Y=(Y, N * T * self.num_output), x0=(x0, N * L * d), dx0=(dx0, N * L * 3 * d), loss=(loss, 1),
                   grad=(grad, self.num_param))
        self._check(self._lib.moihgp_cuda_objective_finish_dev(self._h, ptr[0], N, T, *ptr[1:], None, None))

    def block_transition(self, n):
        """(AKHA^n [L,d,d], E_k(n) [L,3,d,d]): how a block of n steps maps its carry-in (time-sharded evaluation)."""
        L, d = self.num_latent, self.igp_dim
        out = np.zeros((L, 4, d, d))
        self._check(self._lib.moihgp_cuda_block_transition(self._h, int(n), _addr(out)))
        return out[:, 0].copy(), out[:, 1:].copy()

    def smoother_power(self, n, mode=SMOOTH_REFERENCE_LITERAL):
        """G[mode]^n per latent, [L,d,d]: how a backward value crosses a block of n steps (time-sharded smoother)."""
        L, d = self.num_latent, self.igp_dim
        out = np.zeros((L, d, d))
        self._check(self._lib.moihgp_cuda_smoother_power(self._h, int(mode), int(n), _addr(out)))
        return out

    def _fsn_block_args(self, where, phase, Y, x0, u_after, b_end, X, Xs, nll, xT, out=None):
        """(N, T, checked pointers) of the block arguments of fsn_block / fsn_block_async; ``out`` is the phase's output."""
        N, T, L, d = self._dims(where, Y)
        return N, T, _dev(where, Y=(Y, N * T * self.num_output), x0=(x0, N * L * d), u_after=(u_after, N * L), b_end=(b_end, N * L * d),
                          X=(X, N * T * L * d), Xs=(Xs, N * T * L * d), nll=(nll, N), xT=(xT, N * L * d),
                          out=(out, N * L * (d + 1 if phase == 1 else d)))

    def fsn_block(self, phase, Y, seq_end, smoother_mode=SMOOTH_REFERENCE_LITERAL, x0=None, u_after=None, b_end=None, X=None, Xs=None, nll=None, xT=None):
        """One phase (1, 2, 3) of the fused pass on one block of a sequence sharded in time (torch CUDA tensors).
        Phase 1 returns (x_end [N,L,d], u_first [N,L]), phase 2 returns b_start [N,L,d], phase 3 fills X / Xs / nll / xT."""
        N, T, ptr = self._fsn_block_args("fsn_block", phase, Y, x0, u_after, b_end, X, Xs, nll, xT)
        L, d = self.num_latent, self.igp_dim
        host = np.zeros((N, L, d + 1)) if phase == 1 else (np.zeros((N, L, d)) if phase == 2 else None)
        self.set_stream(_torch_stream(Y.device))
        self._check(self._lib.moihgp_cuda_fsn_block_dev(self._h, int(phase), ptr[0], N, T, 1 if seq_end else 0, int(smoother_mode), *ptr[1:-1],
                                                        _addr(host)))
        if phase == 1:
            return host[:, :, :d].copy(), host[:, :, d].copy()
        return host

    def fsn_block_async(self, phase, Y, seq_end, smoother_mode=SMOOTH_REFERENCE_LITERAL, x0=None, u_after=None, b_end=None, X=None, Xs=None,
                        nll=None, xT=None, out=None):
        """fsn_block without a host round trip: the phase's output goes to the torch CUDA tensor ``out`` ([N,L,d+1] after
        phase 1, [N,L,d] after phase 2); asynchronous on torch's current stream."""
        N, T, ptr = self._fsn_block_args("fsn_block_async", phase, Y, x0, u_after, b_end, X, Xs, nll, xT, out)
        self.set_stream(_torch_stream(Y.device))
        self._check(self._lib.moihgp_cuda_fsn_block_async(self._h, int(phase), ptr[0], N, T, 1 if seq_end else 0, int(smoother_mode), *ptr[1:]))

    def fsn_carry_device(self, direction, gathered, block_lengths, rank, out, smoother_mode=SMOOTH_REFERENCE_LITERAL, x0=None, u_after=None):
        """The carry exchanges of the time-sharded pass on the device (torch CUDA tensors): direction 0 turns the all-gathered
        phase-1 outputs [G,N,L,d+1] into this block's x_in (``out`` [N,L,d]) and ``u_after`` [N,L]; direction 1 turns the
        all-gathered phase-2 outputs [G,N,L,d] into this block's b_end (``out`` [N,L,d]; untouched on the last block)."""
        G = len(block_lengths)
        lens = (ctypes.c_longlong * G)(*[int(b) for b in block_lengths])
        N, L, d = out.shape[0], self.num_latent, self.igp_dim
        ptr = _dev("fsn_carry_device", gathered=(gathered, G * N * L * (d + 1 if int(direction) == 0 else d)), x0=(x0, N * L * d),
                   out=(out, N * L * d), u_after=(u_after, N * L))
        self._check(self._lib.moihgp_cuda_fsn_carry_dev(self._h, int(direction), int(smoother_mode), ptr[0], G, lens, int(rank), N, *ptr[1:]))

    def smooth(self, X, smoother_mode=SMOOTH_REFERENCE_LITERAL):
        """IHGP::backwardSmoother (ihgp.h:103-114) of every latent over caller-supplied filtered states X [N,T,L,d] (or
        [T,L,d]); returns Xs of the same shape.  Gains / covariances: ``smoother_consts``."""
        L, d = self.num_latent, self.igp_dim
        Xp, N, T = _host_seqs("smooth", "X", X, (L, d))
        Xs = np.empty((N, T, L, d))
        self._check(self._lib.moihgp_cuda_smooth(self._h, Xp, N, T, int(smoother_mode), _addr(Xs)))
        return Xs[0] if np.ndim(X) == 3 else Xs

    # ---- posterior sample paths (moihgp_cuda_sample_posterior*) ----------------------------------------------------
    def sample_posterior(self, Y, num_samples, seed, x0=None, want_states=False, want_outputs=True):
        """``num_samples`` draws of the latent trajectories from the posterior given Y [N,T,p] (or [T,p]) NumPy array, by
        steady-state forward-filtering, backward-sampling around the RTS-smoothed mean.  Returns a dict of NumPy arrays:
        Xs [N,T,L,d] (the RTS mean), X [S,N,T,L,d] (sampled states, if want_states), F [S,N,T,L] (sampled function values
        x~(0)) and Y [S,N,T,p] (noise-free outputs U sqrt(S) x~(0), if want_outputs).  Draws depend only on (seed, sample,
        sequence, latent, time): see include/moihgp_b200.h for the generator."""
        p, S, L, d = self.num_output, int(num_samples), self.num_latent, self.igp_dim
        Y, N, T = _host_seqs("sample_posterior", "Y", Y, (p,))
        x0, = _host("sample_posterior", x0=(x0, N * L * d))
        Xs = np.empty((N, T, L, d))
        X = np.empty((S, N, T, L, d)) if want_states else None
        F = np.empty((S, N, T, L))
        Ys = np.empty((S, N, T, p)) if want_outputs else None
        self._check(self._lib.moihgp_cuda_sample_posterior(self._h, Y, N, T, x0, S, int(seed) & (2**64 - 1), _addr(Xs), _addr(X), _addr(F),
                                                           _addr(Ys)))
        return {"Xs": Xs, "X": X, "F": F, "Y": Ys}

    def sample_posterior_device(self, Y, seed, x0=None, Xs=None, X=None, F=None, Ysamp=None):
        """Device-resident variant: torch CUDA float64 tensors, outputs pre-allocated by the caller (Xs [N,T,L,d] the RTS mean
        or None, X [S,N,T,L,d], F [S,N,T,L], Ysamp [S,N,T,p], at least one of the last three); the number of samples S is
        their first dimension.  Asynchronous on torch's current stream."""
        N, T, L, d = self._dims("sample_posterior_device", Y)
        p = self.num_output
        outs = [o for o in (X, F, Ysamp) if o is not None]
        S = int(outs[0].shape[0]) if outs else 1
        if any(int(o.shape[0]) != S for o in outs):
            raise ValueError("sample_posterior_device: X, F and Ysamp must hold the same number of samples (their first dimension)")
        ptr = _dev("sample_posterior_device", Y=(Y, N * T * p), x0=(x0, N * L * d), Xs=(Xs, N * T * L * d), X=(X, S * N * T * L * d),
                   F=(F, S * N * T * L), Ysamp=(Ysamp, S * N * T * p))
        self.set_stream(_torch_stream(Y.device))
        self._check(self._lib.moihgp_cuda_sample_posterior_dev(self._h, ptr[0], N, T, ptr[1], S, int(seed) & (2**64 - 1), *ptr[2:]))

    def sample_block_async(self, phase, Xs_mean, num_samples, seed, t0, seq_end, e_end=None, Xsamp=None, Fsamp=None, Ysamp=None, out=None):
        """One phase (1, 2) of the sampler on one block of a sequence sharded in time (torch CUDA tensors, asynchronous on
        torch's current stream).  Xs_mean [N,T,L,d] is the block's RTS mean (fsn_block_async phase 3, smoother_mode 1), t0 the
        global index of its first step.  Phase 1 writes e at the block's first step from a zero e_end to ``out`` [S,N,L,d];
        phase 2 writes X [S,N,T,L,d], F [S,N,T,L] and / or Ysamp [S,N,T,p] from ``e_end`` [S,N,L,d] (None on the block that
        ends the sequence).  Between the phases: fsn_carry_device(1, gathered [G,S*N,L,d], ..., smoother_mode=1)."""
        where = "sample_block_async"
        if getattr(Xs_mean, "ndim", None) != 4:
            _refuse(where, "Xs_mean", "a [N,T,L,d] tensor", "shape %s" % (getattr(Xs_mean, "shape", type(Xs_mean).__name__),))
        N, T = int(Xs_mean.shape[0]), int(Xs_mean.shape[1])
        S, L, d, p = int(num_samples), self.num_latent, self.igp_dim, self.num_output
        ptr = _dev(where, Xs_mean=(Xs_mean, N * T * L * d), e_end=(e_end, S * N * L * d), Xsamp=(Xsamp, S * N * T * L * d),
                   Fsamp=(Fsamp, S * N * T * L), Ysamp=(Ysamp, S * N * T * p), out=(out, S * N * L * d))
        self.set_stream(_torch_stream(Xs_mean.device))
        self._check(self._lib.moihgp_cuda_sample_block_async(self._h, int(phase), ptr[0], N, T, int(t0), 1 if seq_end else 0, S,
                                                             int(seed) & (2**64 - 1), *ptr[1:]))

    def sampler_consts(self, l):
        """(LF, LC) of latent l, [d,d] lower-triangular: LF LF' = PF, LC LC' = PF - G PPc G' (the sampler's noise factors)."""
        d = self.igp_dim
        LF, LC = np.zeros((d, d)), np.zeros((d, d))
        self._check(self._lib.moihgp_cuda_sampler_consts(self._h, l, _addr(LF), _addr(LC)))
        return LF, LC

    # ---- device-resident streaming learner (moihgp_cuda_online_*) -----------------------------------------------
    def online_begin(self, windowsize):
        """Window, moving mean, carried state and proximal term in device memory; False if the shape does not qualify."""
        return self._lib.moihgp_cuda_online_begin(self._h, int(windowsize)) == 0

    def online_push(self, y, ma_given=None, want_ma=False):
        """OnlineObjective::push_back (moihgp_online.h:75-93); ``ma_given``: the caller's own centre instead of the window mean."""
        y, ma_given = _host("online_push", y=(y, self.num_output), ma_given=(ma_given, self.num_output))
        ma = np.empty(self.num_output) if want_ma else None
        self._check(self._lib.moihgp_cuda_online_push(self._h, y, ma_given, _addr(ma)))
        return ma

    def online_set_proximal(self, oldparams=None, B=None):
        """1/2 dparams' B dparams around ``oldparams`` (B None: identity); ``oldparams`` None: no proximal term on the device."""
        n = self.num_param
        self._check(self._lib.moihgp_cuda_online_set_proximal(self._h, *_host("online_set_proximal", oldparams=(oldparams, n), B=(B, n * n))))

    def online_objective(self, params):
        """OnlineObjective::operator() (moihgp_online.h:40-72) at ``params`` on the resident window: one CUDA-graph launch."""
        params, = _host("online_objective", params=(params, self.num_param))
        loss, grad = np.zeros(1), np.zeros(self.num_param)
        self._check(self._lib.moihgp_cuda_online_objective(self._h, params, _addr(loss), _addr(grad)))
        return float(loss[0]), grad

    def online_state(self):
        L, d = self.num_latent, self.igp_dim
        x, dx = np.zeros((L, d)), np.zeros((L, 3, d))
        self._check(self._lib.moihgp_cuda_online_get_state(self._h, _addr(x), _addr(dx)))
        return x, dx

    def bind(self, Y):
        """Copy the observations to the device once; ``objective_bound`` then evaluates on them at the current parameters
        (the L-BFGS loop calls the objective tens of times on the same data).  ``bind(None)`` releases them."""
        if Y is None:
            self._check(self._lib.moihgp_cuda_bind_data(self._h, None, 0, 0))
            self._bound = None
            return
        Y, N, T = _host_seqs("bind", "Y", Y, (self.num_output,))
        self._check(self._lib.moihgp_cuda_bind_data(self._h, Y, N, T))
        self._bound = (N, T)

    def objective_bound(self, x0=None, dx0=None):
        if getattr(self, "_bound", None) is None:
            raise RuntimeError("no data bound: call bind(Y) first")
        N, T = self._bound
        L, d = self.num_latent, self.igp_dim
        x0, dx0 = _host("objective_bound", x0=(x0, N * L * d), dx0=(dx0, N * L * 3 * d))
        loss = np.zeros(1)
        grad = np.zeros(self.num_param)
        self._check(self._lib.moihgp_cuda_objective_bound(self._h, x0, dx0, _addr(loss), _addr(grad), None, None))
        return float(loss[0]), grad

    def objective_device(self, Y, loss, grad, x0=None, dx0=None, xT=None, dxT=None):
        N, T, L, d = self._dims("objective_device", Y)
        ptr = _dev("objective_device", Y=(Y, N * T * self.num_output), x0=(x0, N * L * d), dx0=(dx0, N * L * 3 * d), loss=(loss, 1),
                   grad=(grad, self.num_param), xT=(xT, N * L * d), dxT=(dxT, N * L * 3 * d))
        self.set_stream(_torch_stream(Y.device))
        self._check(self._lib.moihgp_cuda_objective_dev(self._h, ptr[0], N, T, *ptr[1:]))
