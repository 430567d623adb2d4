// TEST INFRASTRUCTURE: a stand-in for LBFGS++'s <LBFGSpp/LBFGSB.h> that REPLAYS a recorded run of the real optimiser.
// LBFGS++ (vendored by the reference, not by this repository) is not available to the tests.  tests/golden_lbfgs holds the
// log of the reference's learners under it (tests/cpp/lbfgs_dropin.cpp built -DUSE_REFERENCE); built against this header
// instead, the same program makes the drop-in learners evaluate the GPU objective at exactly the points the reference's
// optimiser chose, so those evaluations can be compared with the log.  It does NOT exercise an optimiser: iteration counts
// and the optimiser's path come from the recording.  The script named by $MOIHGP_LBFGS_REPLAY holds one record per
// minimize() call, in call order:
//   call <return value>
//   x <v0 v1 ...>          (zero or more: the objective is evaluated at each point, in order, as the optimiser did)
//   final <v0 v1 ...>      (optional: the parameters minimize() leaves in x)
// fx is the value of the last evaluation.  The BFGS matrix holds no correction (get_m() == 0); OnlineObjective with
// corrections is checked against the oracle by tests/cpp/test_host_api.cpp.
#ifndef MOIHGP_B200_TEST_REPLAY_LBFGSB_H
#define MOIHGP_B200_TEST_REPLAY_LBFGSB_H

#include <cstdlib>
#include <fstream>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>
#include <Eigen/Core>
#include <moihgp_b200/moihgp.hpp>

namespace LBFGSpp {

template <typename Scalar>
struct LBFGSBParam {
    int m, past, max_iterations, max_submin, max_linesearch;
    Scalar epsilon, epsilon_rel, delta, ftol, wolfe, min_step, max_step;
    LBFGSBParam()
        : m(6), past(1), max_iterations(0), max_submin(10), max_linesearch(20), epsilon(1e-5), epsilon_rel(1e-5), delta(0),
          ftol(1e-4), wolfe(0.9), min_step(1e-20), max_step(1e20) {}
};

template <typename Scalar, bool LBFGSB = false>
class BFGSMat : public moihgp_b200::NoBFGSMat<Eigen::VectorXd> {};

namespace replay {
struct Call {
    int ret;
    std::vector<std::vector<double> > points;
    std::vector<double> final_x;
};

inline std::vector<double> read_values(std::istringstream& in) {
    std::vector<double> v;
    double d;
    while (in >> d) v.push_back(d);
    return v;
}

// the script, read once; next() hands out its records in order to every solver of the process
inline Call next() {
    static std::vector<Call> calls;
    static size_t cursor = 0;
    static bool loaded = false;
    if (!loaded) {
        const char* path = std::getenv("MOIHGP_LBFGS_REPLAY");
        if (!path) throw std::runtime_error("MOIHGP_LBFGS_REPLAY is not set");
        std::ifstream f(path);
        if (!f) throw std::runtime_error(std::string("cannot open ") + path);
        std::string line;
        while (std::getline(f, line)) {
            std::istringstream in(line);
            std::string tag;
            in >> tag;
            if (tag == "call") {
                Call c;
                in >> c.ret;
                calls.push_back(c);
            } else if (tag == "x" && !calls.empty()) {
                calls.back().points.push_back(read_values(in));
            } else if (tag == "final" && !calls.empty()) {
                calls.back().final_x = read_values(in);
            } else if (!tag.empty()) {
                throw std::runtime_error("bad replay line: " + line);
            }
        }
        loaded = true;
    }
    if (cursor >= calls.size()) throw std::runtime_error("replay script exhausted");
    return calls[cursor++];
}

template <typename Vec>
inline void assign(Vec& x, const std::vector<double>& v) {
    if ((size_t)x.size() != v.size()) throw std::runtime_error("replay point has the wrong length");
    for (size_t i = 0; i < v.size(); ++i) x[i] = v[i];
}
}  // namespace replay

template <typename Scalar>
class LBFGSBSolver {
public:
    explicit LBFGSBSolver(const LBFGSBParam<Scalar>&) {}
    const BFGSMat<Scalar, true>& getBFGSMat() const { return m_bfgs; }

    template <typename Foo, typename Vec>
    int minimize(Foo& f, Vec& x, Scalar& fx, const Vec&, const Vec&) {
        const replay::Call c = replay::next();
        Vec g = x;
        for (size_t k = 0; k < c.points.size(); ++k) {
            replay::assign(x, c.points[k]);
            fx = f(x, g);
        }
        if (!c.final_x.empty()) replay::assign(x, c.final_x);
        return c.ret;
    }

private:
    BFGSMat<Scalar, true> m_bfgs;
};

}  // namespace LBFGSpp
#endif  // MOIHGP_B200_TEST_REPLAY_LBFGSB_H
