"""The C++ host mirror (include/moihgp_b200/moihgp.hpp): compile check on CPU, behaviour against the oracle on the GPU."""
import os
import subprocess

import pytest

import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
CPP = os.path.join(ROOT, "tests", "cpp")


def test_header_compiles_with_reference_vector_type():
    """RegressionObjective / OnlineObjective instantiate with an Eigen::VectorXd-shaped type: the reference's functor
    signature (moihgp_regression.h:34, moihgp_online.h:40)."""
    subprocess.check_call(["g++", "-std=c++11", "-fsyntax-only", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "oracle", "eigen_shim"),
                           "-I" + os.path.join(ROOT, "include"), os.path.join(CPP, "compile_with_eigen_types.cpp")])


def test_header_is_plain_c_abi_only():
    """The host mirror depends on nothing but the C ABI header (no torch, no CUDA headers, no oracle)."""
    src = open(os.path.join(ROOT, "include", "moihgp_b200", "moihgp.hpp")).read()
    includes = [l.split()[1] for l in src.splitlines() if l.startswith("#include")]
    assert set(includes) <= {"<algorithm>", "<cmath>", "<cstddef>", "<list>", "<stdexcept>", "<string>", "<vector>", '"../moihgp_b200.h"'}, includes
    src = open(os.path.join(ROOT, "include", "moihgp_b200", "learners.hpp")).read()
    assert [l.split()[1] for l in src.splitlines() if l.startswith("#include")] == ['"moihgp.hpp"']


REF = "/root/reference/moihgp"


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "include", "LBFGSpp")), reason="needs the reference tree (its vendored LBFGS++ and examples)")
@pytest.mark.parametrize("example", ["example_regression", "example_online_learning"])
def test_reference_examples_compile_unchanged_against_the_dropin_headers(example):
    """BASELINE configs[0] / configs[1]: cpp_examples/example_regression.cpp and example_online_learning.cpp AS SHIPPED compile
    against include/moihgp_b200/dropin (the reference's own include paths and class names) with the reference's vendored
    LBFGS++ - only the include path order changes."""
    subprocess.check_call(["g++", "-std=c++11", "-fsyntax-only", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "oracle", "eigen_shim"),
                           "-I" + os.path.join(ROOT, "include", "moihgp_b200", "dropin"), "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(REF, "include"), os.path.join(REF, "cpp_examples", example + ".cpp")])


def _parse_log(text):
    out = {}
    for line in text.splitlines():
        parts = line.split()
        if not parts or parts[0] == "DONE":
            continue
        tag = parts[0]
        try:
            vals = [float(v) for v in parts[1:]]
        except ValueError:
            vals = parts[1:]
        out.setdefault(tag, []).append(vals)
    return out


def test_lbfgs_reference_fixture_is_an_optimiser_run_that_iterates():
    """tests/golden_lbfgs: the reference's learners under the reference's own LBFGS++ on the CPU (tests/cpp/lbfgs_dropin.cpp
    built -DUSE_REFERENCE).  Part A takes real L-BFGS-B iterations: the loss goes down over >= 3 accepted iterations."""
    import gzip
    ref = _parse_log(gzip.open(os.path.join(ROOT, "tests", "golden_lbfgs", "lbfgs_reference_cpu.log.gz"), "rt").read())
    niter, nevals = ref["A_niter"][0]
    losses = [v[1] for v in ref["A_eval"]]
    assert niter >= 3 and nevals == len(losses) and ref["A_fx"][0][0] < 0.6 * losses[0]
    assert len(ref["C_yhat"]) == 40 and len(ref["B_yhat"]) == 63


def _replay_script(ref):
    """The optimiser's decisions in the reference's run, as tests/cpp/replay/LBFGSpp/LBFGSB.h reads them: every point at
    which part A's optimiser evaluated the objective and the point it returned; part B's iteration count (its objective does
    not move the model's parameters, SURVEY Q6); for each sample of part C, the parameters the optimiser returned (its last
    evaluation, which leaves the model holding them)."""
    def vec(v):
        return " ".join(repr(float(x)) for x in v)
    lines = ["call %d" % ref["A_niter"][0][0]]
    lines += ["x " + vec(x[1:]) for x in ref["A_x"]]
    lines += ["final " + vec(ref["A_final"][0]), "call %d" % ref["B_niter"][0][0]]
    for prm in ref["C_params"]:
        lines += ["call 0", "x " + vec(prm[1:]), "final " + vec(prm[1:])]
    return "\n".join(lines) + "\n"


@pytest.mark.gpu
def test_reference_learners_under_lbfgspp_follow_the_cpu_reference(cuda_lib, tmp_path):
    """The drop-in learners MOIHGPRegression / MOIHGPOnlineLearning (the reference's names and members, every objective
    evaluation on the GPU) against the reference's learners under the reference's vendored LBFGS++ on the CPU (fixture
    tests/golden_lbfgs).  LBFGS++ is not part of this repository, so no optimiser runs here: tests/cpp/lbfgs_dropin.cpp is
    built against tests/cpp/replay/LBFGSpp, which replays the recorded optimiser's decisions.  What is compared with the
    reference, within 1e-9: the loss and gradient at every one of part A's 149 evaluation points and at its final point, the
    parameters and predict() of part B, and the streamed predictions of part C (the online learner, its model moved to the
    recorded parameters after every sample).  What the replay sets, and is therefore only checked for consistency: iteration
    counts, the points evaluated, the final points, and C's parameters.  OnlineObjective's loss and gradient, with and without
    BFGS corrections, are compared with the oracle by test_cpp_host_api_matches_oracle."""
    import gzip
    import numpy as np
    exe = os.path.join(CPP, "_build", "lbfgs_replay")
    subprocess.check_call(["make", "-C", CPP, "_build/lbfgs_replay"], stdout=subprocess.DEVNULL)
    ref = _parse_log(gzip.open(os.path.join(ROOT, "tests", "golden_lbfgs", "lbfgs_reference_cpu.log.gz"), "rt").read())
    script = tmp_path / "lbfgs_replay.txt"
    script.write_text(_replay_script(ref))
    r = subprocess.run([exe], capture_output=True, text=True, timeout=900, env=dict(os.environ, MOIHGP_LBFGS_REPLAY=str(script)))
    print(r.stdout[-1500:], r.stderr[-2000:])
    assert r.returncode == 0 and r.stdout.strip().endswith("DONE")
    got = _parse_log(r.stdout)
    assert set(got) == set(ref)

    def rel(a, b):
        a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
        assert a.shape == b.shape, (a.shape, b.shape)
        return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))
    worst = {}
    for tag in sorted(ref):
        assert len(got[tag]) == len(ref[tag]), tag
        worst[tag] = max(rel(g, f) for g, f in zip(got[tag], ref[tag]))
    print({k: "%.2e" % v for k, v in worst.items()})
    replayed = ("A_niter", "A_x", "A_final", "B_niter", "C_params")
    assert all(worst[k] == 0.0 for k in replayed), worst                           # the replay followed the recording
    computed = ("A_y", "A_eval", "A_g", "A_fx", "B_params", "B_yhat", "C_yhat")
    assert set(replayed + computed) == set(ref)
    assert all(worst[k] < 1e-9 for k in computed), worst
    # the functor itself, evaluation by evaluation, against the oracle at the same parameters
    from oracle.binding import OracleMOIHGP
    p, L = 6, 3
    Y = np.array([v[1:] for v in got["A_y"]])
    o = OracleMOIHGP(0.1, p, L, "Matern32", True)
    e_loss = e_grad = 0.0
    for ev, x, g in zip(got["A_eval"], got["A_x"], got["A_g"]):
        o.update(np.array(x[1:]))
        lo, go, _, _ = o.objective(Y)
        e_loss = max(e_loss, abs(ev[1] - lo) / abs(lo))
        e_grad = max(e_grad, rel(g[1:], go))
    print("functor vs oracle over %d evaluations: loss %.2e grad %.2e" % (len(got["A_eval"]), e_loss, e_grad))
    assert e_loss < 1e-9 and e_grad < 1e-9


@pytest.mark.gpu
@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "include", "LBFGSpp")), reason="needs the reference tree (its vendored LBFGS++ and examples)")
@pytest.mark.parametrize("example", ["example_regression", "example_online_learning"])
def test_reference_examples_run_unchanged_on_the_gpu(cuda_lib, example):
    """BASELINE configs[0] / configs[1]: the reference's example programs, compiled UNCHANGED against the drop-in headers
    (tests/cpp/Makefile), run on the GPU.  Their sources and LBFGS++ are the reference's, not this repository's."""
    exe = os.path.join(CPP, "_build", example)
    subprocess.check_call(["make", "-C", CPP], stdout=subprocess.DEVNULL)
    assert os.path.exists(exe), "tests/cpp/_build/%s was not built" % example
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    print(r.stdout[-600:], r.stderr[-1000:])
    assert r.returncode == 0
    assert ("Iteration count:" in r.stdout) if example == "example_regression" else (r.stdout.count("Elapsed time per step") == 63)
    # the same program built against the UNMODIFIED reference headers (CPU, tests/cpp/Makefile: ref_example_*), run beside it on
    # the box's host, for the record (wall times, iteration counts).  The counts are NOT asserted equal: the shipped
    # example_regression.cpp:22-26 writes two values into a one-element vector and multiplies a 2 x 2 matrix with it - out of
    # bounds under real Eigen, a 4-element observation under the Eigen-API shim, on which the reference's own loss is NaN (its
    # L-BFGS-B loop then idles through max_iterations = 1000) while the drop-in reads the first num_output entries and gets a
    # finite loss.  With well-formed data the two builds agree iterate by iterate:
    # test_reference_learners_under_lbfgspp_follow_the_cpu_reference.
    ref = os.path.join(CPP, "_build", "ref_" + example)
    if os.path.exists(ref):
        import time
        t0 = time.perf_counter()
        rr = subprocess.run([ref], capture_output=True, text=True, timeout=600)
        t_ref = time.perf_counter() - t0
        t0 = time.perf_counter()
        subprocess.run([exe], capture_output=True, text=True, timeout=600)
        t_gpu = time.perf_counter() - t0
        assert rr.returncode == 0
        print("%s: GPU drop-in %.2f s wall (incl. CUDA start-up), CPU reference build (-O0, Eigen-API shim) %.2f s; reference says: %s"
              % (example, t_gpu, t_ref, rr.stdout.strip().splitlines()[0] if rr.stdout.strip() else ""))


@pytest.mark.gpu
def test_cpp_host_api_matches_oracle(cuda_lib):
    exe = os.path.join(CPP, "_build", "test_host_api")
    subprocess.check_call(["make", "-C", CPP], stdout=subprocess.DEVNULL)      # no-op when the binary built by build() is current
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0 and r.stdout.strip().endswith("OK")
