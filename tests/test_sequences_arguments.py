"""The argument checks of MOIHGPSequences.  Every array a caller passes reaches the library as a bare address, and the
library reads or writes as many doubles as include/moihgp_b200.h specifies; so a wrong dtype, layout, size or device must
be refused (ValueError naming the argument) before any library call, and a valid call must pass the caller's own
addresses and the right sizes.  The model is built on a recording stand-in for the library: no library is loaded and
nothing reaches a GPU, not even when a check is missing.  The refusals run without a GPU; the valid device calls need
CUDA tensors (-m gpu)."""
import ctypes

import numpy as np
import pytest

from multioutputihgp_b200 import MOIHGPSequences, _lib

P, L, D, T, G = 5, 3, 2, 7, 2              # num_output, num_latent, igp_dim, steps, time blocks
NPAR = P * L + L + 1 + 3 * L
H = 0x5EED                                  # the handle the stand-in model holds
LENS = [256, 100]
BLOCK_ARGS = ("x0", "u_after", "b_end", "X", "Xs", "nll", "xT")


class _Recorder(object):
    """the ctypes library's stand-in: records (entry point without its moihgp_cuda_ prefix, arguments), returns 0"""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def entry(*args):
            self.calls.append((name[len("moihgp_cuda_"):], args))
            return 0
        return entry


class _Buffer(object):
    """expected in place of a buffer the method allocates itself: any non-null address"""

    def __eq__(self, other):
        return isinstance(other, int) and other != 0


BUF = _Buffer()


def _model():
    m = MOIHGPSequences.__new__(MOIHGPSequences)
    m._lib, m._h, m._owner = _Recorder(), ctypes.c_void_p(H), object()
    m.dt, m.num_output, m.num_latent, m.kernel = 0.1, P, L, "Matern32"
    m.igp_dim, m.num_param, m.num_igp_param = D, NPAR, 3
    return m


def _value(a):
    """an argument as the C side sees it: arrays, tensors and pointers as addresses, ctypes arrays as lists"""
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if isinstance(a, ctypes.Array):
        return list(a)
    if isinstance(a, (ctypes.c_void_p, _lib.c_double_p)):
        return ctypes.cast(a, ctypes.c_void_p).value
    return a.data_ptr() if hasattr(a, "data_ptr") else a


def _expect(m, *calls):
    got, m._lib.calls = m._lib.calls, []
    norm = lambda cs: [(name, tuple(_value(a) for a in args)) for name, args in cs]
    assert norm(got) == norm(calls)


# ============================================================================================================ host
def test_host_calls_pass_the_callers_arrays_and_sizes():
    m = _model()
    rng = np.random.default_rng(0)
    N, S = 2, 3
    Y, x0, dx0 = rng.standard_normal((N, T, P)), rng.standard_normal((N, L, D)), rng.standard_normal((N, L, 3, D))
    params = rng.standard_normal(NPAR)
    m.update(params)
    _expect(m, ("update", (H, params)))
    m.update(list(params))                                          # converted: a copy of its own
    _expect(m, ("update", (H, BUF)))
    r = m.filter_smoother_nll(Y, x0=x0, smoother_mode=1, want_yhat=True)
    _expect(m, ("filter_smoother_nll", (H, Y, N, T, x0, 1, r["X"], r["Xs"], r["Yhat"], r["nll"], r["xT"])))
    r = m.filter_smoother_nll(Y[1], smoother_mode=0, want_states=False, want_nll=False)      # one sequence [T,p]
    _expect(m, ("filter_smoother_nll", (H, Y[1], 1, T, None, 0, None, None, None, None, r["xT"])))
    r = m.filter_smoother_nll_values(Y, x0=x0, smoother_mode=-1, want_yhat=True)
    _expect(m, ("filter_smoother_nll_values", (H, Y, N, T, x0, -1, r["F"], None, r["Yhat"], r["nll"], r["xT"])))
    r = m.nll_steps(Y, x0=x0)
    _expect(m, ("nll_steps", (H, Y, N, T, x0, r["nll_steps"], r["nll"], r["xT"])))
    _, grad, xT, dxT = m.objective(Y, x0=x0, dx0=dx0, want_state=True)
    _expect(m, ("objective", (H, Y, N, T, x0, dx0, BUF, grad, xT, dxT)))
    r = m.sample_posterior(Y, S, -1, x0=x0, want_states=True)
    _expect(m, ("sample_posterior", (H, Y, N, T, x0, S, 2**64 - 1, r["Xs"], r["X"], r["F"], r["Y"])))
    assert r["X"].shape == (S, N, T, L, D)
    X = rng.standard_normal((N, T, L, D))
    Xs = m.smooth(X, 1)
    _expect(m, ("smooth", (H, X, N, T, 1, Xs)))
    Xs = m.smooth(X[0], 0)
    _expect(m, ("smooth", (H, X[0], 1, T, 0, Xs)))
    m.bind(Y)
    _, grad = m.objective_bound(x0, dx0)
    m.bind(None)
    _expect(m, ("bind_data", (H, Y, N, T)), ("objective_bound", (H, x0, dx0, BUF, grad, None, None)), ("bind_data", (H, None, 0, 0)))
    assert m.online_begin(4)
    y, ma_given = Y[0, 0], rng.standard_normal(P)
    ma = m.online_push(y, ma_given=ma_given, want_ma=True)
    B = rng.standard_normal((NPAR, NPAR))
    m.online_set_proximal(params, B)
    m.online_set_proximal()
    _, grad = m.online_objective(params)
    x, dx = m.online_state()
    _expect(m, ("online_begin", (H, 4)), ("online_push", (H, y, ma_given, ma)), ("online_set_proximal", (H, params, B)),
            ("online_set_proximal", (H, None, None)), ("online_objective", (H, params, BUF, grad)), ("online_get_state", (H, x, dx)))
    m.block_transition(5)
    Gp = m.smoother_power(5, 1)
    LF, LC = m.sampler_consts(1)
    _expect(m, ("block_transition", (H, 5, BUF)), ("smoother_power", (H, 1, 5, Gp)), ("sampler_consts", (H, 1, LF, LC)))


N1 = 1
HOST_CASES = {      # method -> (call(m, arrays by name), {array argument: shape})
    "update": (lambda m, a: m.update(a["params"]), {"params": (NPAR,)}),
    "filter_smoother_nll": (lambda m, a: m.filter_smoother_nll(a["Y"], x0=a["x0"]), {"Y": (N1, T, P), "x0": (N1, L, D)}),
    "filter_smoother_nll_values": (lambda m, a: m.filter_smoother_nll_values(a["Y"], x0=a["x0"]), {"Y": (N1, T, P), "x0": (N1, L, D)}),
    "nll_steps": (lambda m, a: m.nll_steps(a["Y"], x0=a["x0"]), {"Y": (N1, T, P), "x0": (N1, L, D)}),
    "objective": (lambda m, a: m.objective(a["Y"], x0=a["x0"], dx0=a["dx0"]), {"Y": (N1, T, P), "x0": (N1, L, D), "dx0": (N1, L, 3, D)}),
    "sample_posterior": (lambda m, a: m.sample_posterior(a["Y"], 2, 1, x0=a["x0"]), {"Y": (N1, T, P), "x0": (N1, L, D)}),
    "smooth": (lambda m, a: m.smooth(a["X"]), {"X": (N1, T, L, D)}),
    "bind": (lambda m, a: m.bind(a["Y"]), {"Y": (N1, T, P)}),
    "objective_bound": (lambda m, a: (m.bind(np.zeros((N1, T, P))), m._lib.calls.clear(), m.objective_bound(a["x0"], a["dx0"])),
                        {"x0": (N1, L, D), "dx0": (N1, L, 3, D)}),
    "online_push": (lambda m, a: m.online_push(a["y"], ma_given=a["ma_given"]), {"y": (P,), "ma_given": (P,)}),
    "online_set_proximal": (lambda m, a: m.online_set_proximal(a["oldparams"], a["B"]), {"oldparams": (NPAR,), "B": (NPAR, NPAR)}),
    "online_objective": (lambda m, a: m.online_objective(a["params"]), {"params": (NPAR,)}),
}


@pytest.mark.parametrize("method,arg", [(k, n) for k, (_, shapes) in HOST_CASES.items() for n in shapes])
@pytest.mark.parametrize("bad", ["short", "long", "wrong last dimension"])
def test_host_arrays_of_the_wrong_size_are_refused(method, arg, bad):
    call, shapes = HOST_CASES[method]
    a = {k: np.zeros(s) for k, s in shapes.items()}
    n = int(np.prod(shapes[arg]))
    a[arg] = {"short": np.zeros(n - 1), "long": np.zeros(n + 1), "wrong last dimension": np.zeros(shapes[arg][:-1] + (shapes[arg][-1] + 1,))}[bad]
    m = _model()
    with pytest.raises(ValueError, match=_refusal(method, arg)):
        call(m, a)
    assert m._lib.calls == []
    call(m, {k: np.zeros(s) for k, s in shapes.items()})            # the same call with the right sizes goes through
    assert m._lib.calls


# ========================================================================================================== device
def _device_cases(N, S):
    """method -> (call(m, tensors by name), {tensor argument: shape}, expected library calls (m, tensors, stream))"""
    nld, nl3d, ntld, ntp = (N, L, D), (N, L, 3, D), (N, T, L, D), (N, T, P)
    st = lambda s: ("set_stream", (H, s))

    def block(method, phase, seq_end, **shapes):
        """fsn_block / fsn_block_async on the arguments `shapes` (``out``: fsn_block_async's output)"""
        call = lambda m, a: getattr(m, method)(phase, a["Y"], seq_end, 1, **{k: a[k] for k in shapes if k != "Y"})
        last = lambda a: a.get("out") if method == "fsn_block_async" else (BUF if phase < 3 else None)
        want = lambda m, a, s: [st(s), ({"fsn_block": "fsn_block_dev"}.get(method, method),
                                        (H, phase, a["Y"], N, T, int(seq_end), 1) + tuple(a.get(k) for k in BLOCK_ARGS) + (last(a),))]
        return call, shapes, want

    return {
        "filter_smoother_nll_device": (
            lambda m, a: m.filter_smoother_nll_device(a["Y"], x0=a["x0"], smoother_mode=1, X=a["X"], Xs=a["Xs"], Yhat=a["Yhat"], nll=a["nll"], xT=a["xT"]),
            dict(Y=ntp, x0=nld, X=ntld, Xs=ntld, Yhat=ntp, nll=(N,), xT=nld),
            lambda m, a, s: [st(s), ("filter_smoother_nll_dev", (H, a["Y"], N, T, a["x0"], 1, a["X"], a["Xs"], a["Yhat"], a["nll"], a["xT"]))]),
        "nll_steps_device": (
            lambda m, a: m.nll_steps_device(a["Y"], a["nll_steps"], x0=a["x0"], nll=a["nll"], xT=a["xT"]),
            dict(Y=ntp, x0=nld, nll_steps=(N, T), nll=(N,), xT=nld),
            lambda m, a, s: [st(s), ("nll_steps_dev", (H, a["Y"], N, T, a["x0"], a["nll_steps"], a["nll"], a["xT"]))]),
        "objective_begin_device": (
            lambda m, a: m.objective_begin_device(a["Y"]), dict(Y=ntp),
            lambda m, a, s: [st(s), ("objective_begin_dev", (H, a["Y"], N, T, BUF))]),
        "objective_begin_async": (
            lambda m, a: m.objective_begin_async(a["Y"], a["zend"]), dict(Y=ntp, zend=(N, L, 4, D)),
            lambda m, a, s: [st(s), ("objective_begin_async", (H, a["Y"], N, T, a["zend"]))]),
        "carry_in_device": (
            lambda m, a: m.carry_in_device(a["ends"], LENS, 1, a["xin"], a["dxin"], x0=a["x0"], dx0=a["dx0"]),
            dict(ends=(G, N, L, 4, D), x0=nld, dx0=nl3d, xin=nld, dxin=nl3d),
            lambda m, a, s: [("carry_in_dev", (H, a["ends"], G, LENS, 1, N, a["x0"], a["dx0"], a["xin"], a["dxin"]))]),
        "objective_finish_device": (
            lambda m, a: m.objective_finish_device(a["Y"], a["loss"], a["grad"], x0=a["x0"], dx0=a["dx0"]),
            dict(Y=ntp, x0=nld, dx0=nl3d, loss=(1,), grad=(NPAR,)),
            lambda m, a, s: [("objective_finish_dev", (H, a["Y"], N, T, a["x0"], a["dx0"], a["loss"], a["grad"], None, None))]),
        "fsn_block/1": block("fsn_block", 1, False, Y=ntp, x0=nld),
        "fsn_block/2": block("fsn_block", 2, False, Y=ntp, x0=nld, u_after=(N, L)),
        "fsn_block/3": block("fsn_block", 3, True, Y=ntp, x0=nld, b_end=nld, X=ntld, Xs=ntld, nll=(N,), xT=nld),
        "fsn_block_async/1": block("fsn_block_async", 1, False, Y=ntp, out=(N, L, D + 1)),
        "fsn_block_async/2": block("fsn_block_async", 2, False, Y=ntp, x0=nld, u_after=(N, L), out=nld),
        "fsn_block_async/3": block("fsn_block_async", 3, False, Y=ntp, x0=nld, u_after=(N, L), b_end=nld, X=ntld, Xs=ntld, nll=(N,), xT=nld),
        "fsn_carry_device/0": (
            lambda m, a: m.fsn_carry_device(0, a["gathered"], LENS, 0, a["out"], 1, x0=a["x0"], u_after=a["u_after"]),
            dict(gathered=(G, N, L, D + 1), x0=nld, out=nld, u_after=(N, L)),
            lambda m, a, s: [("fsn_carry_dev", (H, 0, 1, a["gathered"], G, LENS, 0, N, a["x0"], a["out"], a["u_after"]))]),
        "fsn_carry_device/1": (
            lambda m, a: m.fsn_carry_device(1, a["gathered"], LENS, 0, a["out"], 0),
            dict(gathered=(G, N, L, D), out=nld),
            lambda m, a, s: [("fsn_carry_dev", (H, 1, 0, a["gathered"], G, LENS, 0, N, None, a["out"], None))]),
        "sample_posterior_device": (
            lambda m, a: m.sample_posterior_device(a["Y"], -2, x0=a["x0"], Xs=a["Xs"], X=a["X"], F=a["F"], Ysamp=a["Ysamp"]),
            dict(Y=ntp, x0=nld, Xs=ntld, X=(S,) + ntld, F=(S, N, T, L), Ysamp=(S,) + ntp),
            lambda m, a, s: [st(s), ("sample_posterior_dev", (H, a["Y"], N, T, a["x0"], S, 2**64 - 2, a["Xs"], a["X"], a["F"], a["Ysamp"]))]),
        "objective_device": (
            lambda m, a: m.objective_device(a["Y"], a["loss"], a["grad"], x0=a["x0"], dx0=a["dx0"], xT=a["xT"], dxT=a["dxT"]),
            dict(Y=ntp, x0=nld, dx0=nl3d, loss=(1,), grad=(NPAR,), xT=nld, dxT=nl3d),
            lambda m, a, s: [st(s), ("objective_dev", (H, a["Y"], N, T, a["x0"], a["dx0"], a["loss"], a["grad"], a["xT"], a["dxT"]))]),
    }


DEVICE_ARGS = [(k, n) for k, (_, shapes, _) in _device_cases(2, 3).items() for n in shapes]


def _tensors(shapes, device, **given):
    import torch
    a = {k: torch.zeros(s, dtype=torch.float64, device=device) for k, s in shapes.items()}
    a.update(given)
    return a


def _refusal(method, arg, what=""):
    return "^%s: %s must be %s" % (method.split("/")[0], arg, what)


@pytest.mark.parametrize("method,arg", DEVICE_ARGS)
@pytest.mark.parametrize("bad", ["float32", "strided", "short", "long", "numpy"])
def test_device_arguments_of_the_wrong_kind_are_refused(method, arg, bad):
    """Every other argument is a valid host tensor: dtype, layout and size are checked before any device, so no GPU is
    needed.  The one-off sizes use N = S = 1, so that the first dimension the method reads N or S from can stay right."""
    import torch
    call, shapes, _ = _device_cases(1, 1)[method] if bad in ("short", "long") else _device_cases(2, 3)[method]
    shape = shapes[arg]
    n = int(np.prod(shape))
    if bad == "strided" and n == 1:
        pytest.skip("a one-element tensor is contiguous")
    t = {"float32": lambda: torch.zeros(shape, dtype=torch.float32),
         "strided": lambda: torch.zeros(shape + (2,), dtype=torch.float64)[..., 0],
         "short": lambda: torch.zeros((1,) * (len(shape) - 1) + (n - 1,), dtype=torch.float64),
         "long": lambda: torch.zeros((1,) * (len(shape) - 1) + (n + 1,), dtype=torch.float64),
         "numpy": lambda: np.zeros(shape)}[bad]()
    m = _model()
    with pytest.raises(ValueError, match=_refusal(method, arg)):
        call(m, _tensors(shapes, "cpu", **{arg: t}))
    assert m._lib.calls == []


@pytest.mark.parametrize("method", list(_device_cases(2, 3)))
def test_device_calls_on_host_tensors_are_refused(method):
    call, shapes, _ = _device_cases(2, 3)[method]
    m = _model()
    with pytest.raises(ValueError, match=_refusal(method, next(iter(shapes)), "a CUDA tensor, got cpu")):
        call(m, _tensors(shapes, "cpu"))
    assert m._lib.calls == []


def test_device_sequences_are_three_dimensional_with_every_output():
    import torch
    m = _model()
    loss, grad = torch.zeros(1, dtype=torch.float64), torch.zeros(NPAR, dtype=torch.float64)
    for Y in (torch.zeros((T, P), dtype=torch.float64), torch.zeros((1, T, P + 1), dtype=torch.float64), np.zeros((T, P)), None):
        with pytest.raises(ValueError, match=_refusal("objective_device", "Y")):
            m.objective_device(Y, loss, grad)
    assert m._lib.calls == []


def test_sample_outputs_hold_the_same_number_of_samples():
    import torch
    N, S = 2, 3
    m = _model()
    a = _tensors(dict(Y=(N, T, P), X=(S, N, T, L, D), F=(1, S * N, T, L)), "cpu")
    with pytest.raises(ValueError, match="^sample_posterior_device: X, F and Ysamp must hold the same number of samples"):
        m.sample_posterior_device(a["Y"], 1, X=a["X"], F=a["F"])
    assert m._lib.calls == []


@pytest.fixture
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.mark.gpu
@pytest.mark.parametrize("method", list(_device_cases(2, 3)))
@pytest.mark.parametrize("layout", ["shaped", "flattened", "offset"])
def test_valid_device_calls_pass_the_callers_tensors(cuda, method, layout):
    """As shaped, flattened behind the first dimension (where N or S is read; Y keeps its shape) and as contiguous views one
    double past the start of their allocation (8-byte aligned, not 16: the library sends those to other kernels)."""
    from multioutputihgp_b200.batched import _torch_stream
    call, shapes, want = _device_cases(2, 3)[method]
    a = _tensors(shapes, "cuda")
    if layout == "flattened":
        a = {k: t if k == "Y" else t.view(t.shape[0], -1) for k, t in a.items()}
    if layout == "offset":
        a = {k: cuda.zeros(t.numel() + 1, dtype=cuda.float64, device="cuda")[1:].view(t.shape) for k, t in a.items()}
    m = _model()
    call(m, a)
    _expect(m, *want(m, a, _torch_stream(next(iter(a.values())).device)))


@pytest.mark.gpu
@pytest.mark.parametrize("method,arg", DEVICE_ARGS)
def test_a_host_tensor_among_device_tensors_is_refused(cuda, method, arg):
    call, shapes, _ = _device_cases(2, 3)[method]
    a = _tensors(shapes, "cuda")
    a[arg] = a[arg].cpu()
    m = _model()
    with pytest.raises(ValueError, match=_refusal(method, arg, "a CUDA tensor, got cpu")):
        call(m, a)
    assert m._lib.calls == []


@pytest.mark.gpu
@pytest.mark.parametrize("method,arg", [(k, n) for k, n in DEVICE_ARGS if n != next(iter(_device_cases(2, 3)[k][1]))])
def test_a_tensor_on_another_device_is_refused(cuda, method, arg):
    if cuda.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    call, shapes, _ = _device_cases(2, 3)[method]
    a = _tensors(shapes, "cuda:0")
    a[arg] = a[arg].to("cuda:1")
    m = _model()
    with pytest.raises(ValueError, match=_refusal(method, arg, "on cuda:0 like ")):
        call(m, a)
    assert m._lib.calls == []
