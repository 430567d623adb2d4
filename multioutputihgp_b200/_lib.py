"""Loader for multioutputihgp_b200/lib/libmoihgp.so (built by csrc/Makefile for sm_100a).

There is no CPU fallback: if the library is missing this module raises, and creating a model
without a B200-class CUDA device raises (the C side refuses to create a handle)."""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MOIHGP_B200_LIB") or os.path.join(_HERE, "lib", "libmoihgp.so")   # override: A/B experiments only
CSRC = os.path.join(_HERE, "csrc")

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int_p = ctypes.POINTER(ctypes.c_int)

_SOURCES = ["ls_project.cuh", "polar.cu", "chain_kernels.cuh", "chain_inst_16x8.cu", "chain_inst_8x4.cu", "chain_inst_8x2.cu", "chain_inst_8x8.cu", "chain_inst_16x2.cu", "chain_inst_16x4.cu", "chain_inst_16x16.cu", "chain_inst_32x4.cu", "chain_inst_32x8.cu", "chain_inst_32x16.cu", "chain_inst_4x2.cu", "chain_inst_4x4.cu", "chain_inst_32x2.cu", "chain_inst_4x1.cu", "chain_inst_8x1.cu", "chain_inst_16x1.cu", "chain_inst_32x1.cu", "setup.cu", "sample.cu", "project.cu", "scan.cu", "objective.cu", "chain.cu", "step.cu", "capi.cu", "moihgp_device.cuh", "ptx.cuh", "small_mat.cuh", "launch.h", "Makefile"]


def build(force=False, verbose=False):
    """Compile the CUDA library in-tree (nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo)."""
    stale = force or not os.path.exists(LIB_PATH)
    if not stale:
        t = os.path.getmtime(LIB_PATH)
        stale = any(os.path.getmtime(os.path.join(CSRC, s)) > t for s in _SOURCES)
        stale = stale or os.path.getmtime(os.path.join(_HERE, "..", "include", "moihgp_b200.h")) > t
    if stale:
        if not os.path.exists("/usr/local/cuda/bin/nvcc"):
            raise RuntimeError("libmoihgp.so is missing/stale and nvcc is not available to build it")
        out = None if verbose else subprocess.DEVNULL
        subprocess.check_call(["make", "-C", CSRC, "-j8"], stdout=out)
    return LIB_PATH


_lib = None


def load():
    """dlopen libmoihgp.so and declare every symbol of include/moihgp_b200.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, sz, dbl, dp = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_double, c_double_p
    for xx in ("32", "52"):
        g = lambda n: getattr(lib, "gp%s_%s" % (xx, n))
        g("new").restype = vp
        g("new").argtypes = [dbl, sz, sz, ctypes.c_bool]
        g("del").restype = None
        g("del").argtypes = [vp]
        for name, n in (("step1", 6), ("step2", 5), ("step3", 4), ("step4", 3), ("update", 1), ("get_params", 1)):
            g(name).restype = None
            g(name).argtypes = [vp] + [dp] * n
        g("lik1").restype = dbl
        g("lik1").argtypes = [vp] + [dp] * 4
        g("lik2").restype = dbl
        g("lik2").argtypes = [vp] + [dp] * 2
        for name in ("igp_dim", "num_param", "num_igp_param"):
            g(name).restype = sz
            g(name).argtypes = [vp]
    lib.moihgp_cuda_create.restype = ctypes.c_int
    lib.moihgp_cuda_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int, dbl, sz, sz, ctypes.c_int, ctypes.c_int]
    lib.moihgp_cuda_destroy.restype = None
    lib.moihgp_cuda_destroy.argtypes = [vp]
    lib.moihgp_cuda_set_stream.restype = ctypes.c_int
    lib.moihgp_cuda_set_stream.argtypes = [vp, vp]
    lib.moihgp_cuda_sync.restype = ctypes.c_int
    lib.moihgp_cuda_sync.argtypes = [vp]
    lib.moihgp_cuda_last_error.restype = ctypes.c_char_p
    lib.moihgp_cuda_last_error.argtypes = [vp]
    lib.moihgp_cuda_set_path.restype = ctypes.c_int
    lib.moihgp_cuda_set_path.argtypes = [vp, ctypes.c_int]
    lib.moihgp_cuda_set_chain_seqs_per_warp.restype = ctypes.c_int
    lib.moihgp_cuda_set_chain_seqs_per_warp.argtypes = [vp, ctypes.c_int]
    lib.moihgp_cuda_profile.restype = ctypes.c_int
    lib.moihgp_cuda_profile.argtypes = [vp, ctypes.c_int]
    lib.moihgp_cuda_profile_read.restype = ctypes.c_char_p
    lib.moihgp_cuda_profile_read.argtypes = [vp]
    lib.moihgp_cuda_online_begin.restype = ctypes.c_int
    lib.moihgp_cuda_online_begin.argtypes = [vp, sz]
    lib.moihgp_cuda_online_push.restype = ctypes.c_int
    lib.moihgp_cuda_online_push.argtypes = [vp, vp, vp, vp]
    lib.moihgp_cuda_online_set_proximal.restype = ctypes.c_int
    lib.moihgp_cuda_online_set_proximal.argtypes = [vp, vp, vp]
    lib.moihgp_cuda_online_objective.restype = ctypes.c_int
    lib.moihgp_cuda_online_objective.argtypes = [vp, vp, vp, vp]
    lib.moihgp_cuda_online_get_state.restype = ctypes.c_int
    lib.moihgp_cuda_online_get_state.argtypes = [vp, vp, vp]
    lib.moihgp_cuda_nan_status.restype = ctypes.c_int
    lib.moihgp_cuda_nan_status.argtypes = [vp, c_int_p]
    lib.moihgp_cuda_launch_count.restype = ctypes.c_longlong
    lib.moihgp_cuda_launch_count.argtypes = [vp]
    for name in ("igp_dim", "num_param", "num_igp_param"):
        f = getattr(lib, "moihgp_cuda_" + name)
        f.restype = sz
        f.argtypes = [vp]
    lib.moihgp_cuda_update.restype = ctypes.c_int
    lib.moihgp_cuda_update.argtypes = [vp, dp]
    lib.moihgp_cuda_get_params.restype = ctypes.c_int
    lib.moihgp_cuda_get_params.argtypes = [vp, dp]
    lib.moihgp_cuda_get_U.restype = ctypes.c_int
    lib.moihgp_cuda_get_U.argtypes = [vp, dp]
    lib.moihgp_cuda_latent_consts.restype = ctypes.c_longlong
    lib.moihgp_cuda_latent_consts.argtypes = [vp, sz, dp, sz]
    lib.moihgp_cuda_latent_iters.restype = ctypes.c_int
    lib.moihgp_cuda_latent_iters.argtypes = [vp, sz, c_int_p]
    lib.moihgp_cuda_smoother_consts.restype = ctypes.c_int
    lib.moihgp_cuda_smoother_consts.argtypes = [vp, sz, ctypes.c_int, dp, dp]
    fsn = [vp, vp, sz, sz, vp, ctypes.c_int, vp, vp, vp, vp, vp]
    lib.moihgp_cuda_filter_smoother_nll.restype = ctypes.c_int
    lib.moihgp_cuda_filter_smoother_nll.argtypes = fsn
    lib.moihgp_cuda_filter_smoother_nll_values.restype = ctypes.c_int
    lib.moihgp_cuda_filter_smoother_nll_values.argtypes = fsn
    lib.moihgp_cuda_filter_smoother_nll_dev.restype = ctypes.c_int
    lib.moihgp_cuda_filter_smoother_nll_dev.argtypes = fsn
    obj = [vp, vp, sz, sz, vp, vp, vp, vp, vp, vp]
    lib.moihgp_cuda_objective.restype = ctypes.c_int
    lib.moihgp_cuda_objective.argtypes = obj
    lib.moihgp_cuda_objective_dev.restype = ctypes.c_int
    lib.moihgp_cuda_objective_dev.argtypes = obj
    lib.moihgp_cuda_objective_begin_dev.restype = ctypes.c_int
    lib.moihgp_cuda_objective_begin_dev.argtypes = [vp, vp, sz, sz, vp]
    lib.moihgp_cuda_objective_finish_dev.restype = ctypes.c_int
    lib.moihgp_cuda_objective_finish_dev.argtypes = obj
    lib.moihgp_cuda_objective_begin_async.restype = ctypes.c_int
    lib.moihgp_cuda_objective_begin_async.argtypes = [vp, vp, sz, sz, vp]
    lib.moihgp_cuda_carry_in_dev.restype = ctypes.c_int
    lib.moihgp_cuda_carry_in_dev.argtypes = [vp, vp, sz, ctypes.POINTER(ctypes.c_longlong), sz, sz, vp, vp, vp, vp]
    lib.moihgp_cuda_block_transition.restype = ctypes.c_int
    lib.moihgp_cuda_block_transition.argtypes = [vp, sz, vp]
    lib.moihgp_cuda_fsn_block_dev.restype = ctypes.c_int
    lib.moihgp_cuda_fsn_block_dev.argtypes = [vp, ctypes.c_int, vp, sz, sz, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.moihgp_cuda_fsn_block_async.restype = ctypes.c_int
    lib.moihgp_cuda_fsn_block_async.argtypes = [vp, ctypes.c_int, vp, sz, sz, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.moihgp_cuda_fsn_carry_dev.restype = ctypes.c_int
    lib.moihgp_cuda_fsn_carry_dev.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, sz, ctypes.POINTER(ctypes.c_longlong), sz, sz, vp, vp, vp]
    lib.moihgp_cuda_smoother_power.restype = ctypes.c_int
    lib.moihgp_cuda_smoother_power.argtypes = [vp, ctypes.c_int, sz, vp]
    for name in ("moihgp_cuda_smooth", "moihgp_cuda_smooth_dev"):
        getattr(lib, name).restype = ctypes.c_int
        getattr(lib, name).argtypes = [vp, vp, sz, sz, ctypes.c_int, vp]
    for name in ("moihgp_cuda_sample_posterior", "moihgp_cuda_sample_posterior_dev"):
        getattr(lib, name).restype = ctypes.c_int
        getattr(lib, name).argtypes = [vp, vp, sz, sz, vp, sz, ctypes.c_uint64, vp, vp, vp, vp]
    for name in ("moihgp_cuda_nll_steps", "moihgp_cuda_nll_steps_dev"):
        getattr(lib, name).restype = ctypes.c_int
        getattr(lib, name).argtypes = [vp, vp, sz, sz, vp, vp, vp, vp]
    lib.moihgp_cuda_sample_block_async.restype = ctypes.c_int
    lib.moihgp_cuda_sample_block_async.argtypes = [vp, ctypes.c_int, vp, sz, sz, ctypes.c_uint64, ctypes.c_int, sz, ctypes.c_uint64, vp, vp, vp,
                                                   vp, vp]
    lib.moihgp_cuda_sampler_consts.restype = ctypes.c_int
    lib.moihgp_cuda_sampler_consts.argtypes = [vp, sz, vp, vp]
    lib.moihgp_cuda_bind_data.restype = ctypes.c_int
    lib.moihgp_cuda_bind_data.argtypes = [vp, vp, sz, sz]
    lib.moihgp_cuda_objective_bound.restype = ctypes.c_int
    lib.moihgp_cuda_objective_bound.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    _lib = lib
    return lib


# every symbol include/moihgp_b200.h declares (checked by tests/test_abi.py)
LEGACY_NAMES = ["new", "del", "step1", "step2", "step3", "step4", "update", "lik1", "lik2", "get_params", "igp_dim",
                "num_param", "num_igp_param"]
CUDA_NAMES = ["create", "destroy", "set_stream", "sync", "last_error", "launch_count", "profile", "profile_read", "set_path", "set_chain_seqs_per_warp", "igp_dim", "num_param",
              "num_igp_param", "update", "get_params", "get_U", "latent_consts", "latent_iters", "smoother_consts",
              "filter_smoother_nll", "filter_smoother_nll_values", "filter_smoother_nll_dev", "objective", "objective_dev", "bind_data", "objective_bound", "objective_begin_dev", "objective_finish_dev", "block_transition", "fsn_block_dev", "fsn_block_async", "fsn_carry_dev", "smoother_power", "smooth", "smooth_dev", "objective_begin_async", "carry_in_dev", "nan_status", "online_begin", "online_push", "online_set_proximal",
              "online_objective", "online_get_state", "sample_posterior", "sample_posterior_dev", "sampler_consts",
              "sample_block_async",
              "nll_steps", "nll_steps_dev"]
ALL_SYMBOLS = ["gp%s_%s" % (xx, n) for xx in ("32", "52") for n in LEGACY_NAMES] + ["moihgp_cuda_" + n for n in CUDA_NAMES]
