// moihgp_b200/moihgp.hpp - host-side C++ mirror of the reference's class API for the hot path, over the C ABI of
// libmoihgp.so (include/moihgp_b200.h).  Header-only, no dependency beyond the C ABI.
//
// Same class and method names, argument meaning and (absent) error behaviour as the reference:
//   moihgp::IHGP<StateSpace>                moihgp/include/moihgp/ihgp.h:17-263     (public members :243-254)
//   moihgp::MOIHGP<StateSpace>              moihgp/include/moihgp/moihgp.h:76-757   (public U, S, dA, sigma :741-744)
//   moihgp::RegressionObjective<StateSpace> moihgp/include/moihgp/moihgp_regression.h:17-70
//   moihgp::OnlineObjective<StateSpace>     moihgp/include/moihgp/moihgp_online.h:18-115
// (the learners MOIHGPRegression / MOIHGPOnlineLearning around LBFGS++ are in learners.hpp) living in namespace
// moihgp_b200 so that both header sets can be included side by side.  include/moihgp_b200/dropin/ holds headers with the
// REFERENCE'S OWN include paths (<moihgp/moihgp_regression.h> ...) that alias these classes into namespace moihgp with
// Eigen types: the reference's cpp_examples compile against them unchanged (INTEGRATION.md).
//
// The reference's vector / matrix types are Eigen::VectorXd / Eigen::MatrixXd.  Eigen is not a dependency here: every
// class takes them as template parameters `Vec` (default std::vector<double>: needs size(), resize(n), operator[]) and
// `Mat` (default DenseMatrix below: needs resize(r, c), operator()(i, j)) - which Eigen provides - so
// `MOIHGP<Matern32StateSpace, Eigen::VectorXd, Eigen::MatrixXd>` gives the reference's exact signatures, and the functors
// plug into LBFGSpp::LBFGSBSolver::minimize(f, x, fx, lb, ub) unchanged.
//
// What runs where: the per-observation methods (step, negLogLikelihood) are one small kernel launch each (the legacy
// gpXX_* path); the objective functors hand the WHOLE window / data set to moihgp_cuda_objective - one fused device pass
// instead of the reference's loop of step + negLogLikelihood per observation.
#ifndef MOIHGP_B200_MOIHGP_HPP
#define MOIHGP_B200_MOIHGP_HPP

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <list>
#include <stdexcept>
#include <string>
#include <vector>

#include "../moihgp_b200.h"

namespace moihgp_b200 {

// StateSpace tags (the reference's duck-typed classes matern32ss.h:13-99 / matern52ss.h:13-110 reduce, on this side of
// the boundary, to the choice of kernel; their arithmetic runs in the K-setup kernel)
// Of the duck type (matern32ss.h:67-91) they keep getDim / getNumParam / getParams / update; F, Pinf, dF, dPinf are
// internal to K-setup and not exposed.
template <int KERNEL, int DIM>
struct StateSpaceTag {
    static constexpr int kernel = KERNEL;
    static constexpr int dim = DIM;
    StateSpaceTag() { _p[0] = 1.0; _p[1] = 1.0; _p[2] = 0.1; }          // matern32ss.h:35 / matern52ss.h:33
    size_t getDim() const { return DIM; }
    size_t getNumParam() const { return 3; }
    template <typename Vec> void update(const Vec& params) { for (int i = 0; i < 3; ++i) _p[i] = params[i]; }
    std::vector<double> getParams() const { return std::vector<double>(_p, _p + 3); }
private:
    double _p[3];
};
typedef StateSpaceTag<MOIHGP_MATERN32, 2> Matern32StateSpace;
typedef StateSpaceTag<MOIHGP_MATERN52, 3> Matern52StateSpace;

// Default matrix type (column-major like Eigen's): just enough for the public members U, A, Q, K, ...
struct DenseMatrix {
    DenseMatrix() : _r(0), _c(0) {}
    DenseMatrix(size_t r, size_t c) : _r(r), _c(c), _d(r * c, 0.0) {}
    void resize(size_t r, size_t c) { _r = r; _c = c; _d.assign(r * c, 0.0); }
    size_t rows() const { return _r; }
    size_t cols() const { return _c; }
    double& operator()(size_t i, size_t j) { return _d[i + j * _r]; }
    const double& operator()(size_t i, size_t j) const { return _d[i + j * _r]; }
    double* data() { return _d.empty() ? NULL : &_d[0]; }
    const double* data() const { return _d.empty() ? NULL : &_d[0]; }
private:
    size_t _r, _c;
    std::vector<double> _d;
};

namespace detail {
template <typename Vec> inline Vec make_vec(size_t n) { Vec v; v.resize(n); for (size_t i = 0; i < n; ++i) v[i] = 0.0; return v; }
inline void check(moihgp_handle* h, int rc, const char* where) {
    if (rc != 0) throw std::runtime_error(std::string(where) + ": " + moihgp_cuda_last_error(h));
}
}  // namespace detail

// ------------------------------------------------------------------------------------------------------------------
// IHGP<StateSpace>   (ihgp.h:17-263): ONE latent infinite-horizon GP.  On this side of the boundary it is a device model
// with one output and one latent whose mixing is the identity (U = 1, S = 1): Ty = y, yhat = xnew(0), and
// MOIHGP::negLogLikelihood(x, y) reduces to 1/2 (v^2 / S + log S) exactly (the residual term is identically 0).
template <typename StateSpace, typename Vec = std::vector<double>, typename Mat = DenseMatrix>
class IHGP {
public:
    IHGP(const double& dt, int device = -1) : _h(NULL), _dim(StateSpace::dim), _num_param(3) {        // ihgp.h:22-34
        if (moihgp_cuda_create(&_h, StateSpace::kernel, dt, 1, 1, 0, device) != 0 || !_h)
            throw std::runtime_error("moihgp_cuda_create failed (no B200-class CUDA device? there is no CPU fallback)");
        refresh();
    }
    ~IHGP() { if (_h) moihgp_cuda_destroy(_h); }

    // ihgp.h:37-57.  NaN = missing observation: prediction step xnew = A x, dxnew_k = dA_k x + A dx_k (:39-47)
    void step(const Vec& x, const double& y, const std::vector<Vec>& dx, Vec& xnew, double& yhat, std::vector<Vec>& dxnew) {
        double xb[3], dxb[9], xn[3], dxn[9], yy = y, yh = 0.0;
        pack(x, dx, xb, dxb);
        gp32_step1(_h, xb, std::isnan(y) ? NULL : &yy, dxb, xn, &yh, dxn);
        unpack(xn, dxn, xnew, &dxnew);
        yhat = yh;
    }
    // ihgp.h:60-78
    void step(const Vec& x, const double& y, const std::vector<Vec>& dx, Vec& xnew, std::vector<Vec>& dxnew) {
        double yhat;
        step(x, y, dx, xnew, yhat, dxnew);
    }
    // ihgp.h:81-93
    void step(const Vec& x, const double& y, Vec& xnew, double& yhat) {
        double xb[3], xn[3], yy = y, yh = 0.0;
        for (size_t i = 0; i < _dim; ++i) xb[i] = x[i];
        if (std::isnan(y)) gp32_step4(_h, xb, xn, &yh); else gp32_step3(_h, xb, &yy, xn, &yh);
        xnew.resize(_dim);
        for (size_t i = 0; i < _dim; ++i) xnew[i] = xn[i];
        yhat = yh;
    }
    // ihgp.h:96-100
    void step(const Vec& x, Vec& xnew, double& yhat) {
        double xb[3], xn[3], yh = 0.0;
        for (size_t i = 0; i < _dim; ++i) xb[i] = x[i];
        gp32_step4(_h, xb, xn, &yh);
        xnew.resize(_dim);
        for (size_t i = 0; i < _dim; ++i) xnew[i] = xn[i];
        yhat = yh;
    }

    // ihgp.h:103-114: the reference's recursion as written (SURVEY Q3), on the caller's filtered states X; like the
    // reference it appends to Xprev and then reverses it.  P, G: smoothed covariance and gain.
    void backwardSmoother(const std::vector<Vec>& X, std::vector<Vec>& Xprev, Mat& P, Mat& G) {
        const size_t n = X.size();
        double g[9], pm[9];
        detail::check(_h, moihgp_cuda_smoother_consts(_h, 0, MOIHGP_SMOOTH_REFERENCE_LITERAL, g, pm), "IHGP::backwardSmoother");
        P.resize(_dim, _dim); G.resize(_dim, _dim);
        for (size_t i = 0; i < _dim; ++i) for (size_t j = 0; j < _dim; ++j) { G(i, j) = g[i * _dim + j]; P(i, j) = pm[i * _dim + j]; }
        if (n == 0) return;
        std::vector<double> xin(n * _dim), xout(n * _dim);
        for (size_t t = 0; t < n; ++t) for (size_t i = 0; i < _dim; ++i) xin[t * _dim + i] = X[t][i];
        detail::check(_h, moihgp_cuda_smooth(_h, &xin[0], 1, n, MOIHGP_SMOOTH_REFERENCE_LITERAL, &xout[0]), "IHGP::backwardSmoother");
        for (size_t k = 0; k < n; ++k) {                 // Xprev.push_back(...) from the last step down (:108-112)
            const size_t t = n - 1 - k;
            Vec v; v.resize(_dim);
            for (size_t i = 0; i < _dim; ++i) v[i] = xout[t * _dim + i];
            Xprev.push_back(v);
        }
        std::reverse(Xprev.begin(), Xprev.end());        // :113
    }

    // ihgp.h:117-201 (K-setup kernel)
    void update(const Vec& params) {
        double pb[6] = {1.0, 1.0, 1e-2, params[0], params[1], params[2]};     // U = 1, S = 1, sigma (unused by an IHGP)
        detail::check(_h, moihgp_cuda_update(_h, pb), "IHGP::update");
        refresh();
    }
    // ihgp.h:204-209
    double negLogLikelihood(const Vec& x, const double& y) {
        double xb[3], yy = y;
        for (size_t i = 0; i < _dim; ++i) xb[i] = x[i];
        return gp32_lik2(_h, xb, &yy);
    }
    // ihgp.h:212-222: loss as above, grad[k] = (v dv_k - 1/2 (v^2/S - 1) dS_k) / S
    double negLogLikelihood(const Vec& x, const double& y, const std::vector<Vec>& dx, Vec& grad) {
        double xb[3], dxb[9], g[6], yy = y;
        pack(x, dx, xb, dxb);
        gp32_lik1(_h, xb, &yy, dxb, g);                  // g = [dU, dS, dsigma, per-latent gradient (3)]
        grad.resize(_num_param);
        for (size_t k = 0; k < _num_param; ++k) grad[k] = g[3 + k];
        return gp32_lik2(_h, xb, &yy);
    }
    Vec getParams() {                                    // ihgp.h:225-228
        double pb[6];
        moihgp_cuda_get_params(_h, pb);
        Vec out = detail::make_vec<Vec>(3);
        for (int k = 0; k < 3; ++k) out[k] = pb[3 + k];
        return out;
    }
    size_t getNumParam() { return _num_param; }          // ihgp.h:231
    size_t getDim() { return _dim; }                     // ihgp.h:237

    // ihgp.h:243-254
    Mat A, Q, K, S, PF, HA, AKHA;
    std::vector<Mat> dS, dA, dK, dAKHA, HdA;

    moihgp_handle* handle() { return _h; }

private:
    IHGP(const IHGP&);
    IHGP& operator=(const IHGP&);
    void pack(const Vec& x, const std::vector<Vec>& dx, double* xb, double* dxb) const {
        for (size_t i = 0; i < _dim; ++i) xb[i] = x[i];
        for (size_t k = 0; k < _num_param; ++k) for (size_t i = 0; i < _dim; ++i) dxb[k * _dim + i] = dx[k][i];
    }
    void unpack(const double* xn, const double* dxn, Vec& xnew, std::vector<Vec>* dxnew) const {
        xnew.resize(_dim);
        for (size_t i = 0; i < _dim; ++i) xnew[i] = xn[i];
        if (dxnew) {
            dxnew->resize(_num_param);
            for (size_t k = 0; k < _num_param; ++k) { (*dxnew)[k].resize(_dim); for (size_t i = 0; i < _dim; ++i) (*dxnew)[k][i] = dxn[k * _dim + i]; }
        }
    }
    static void put(Mat& m, size_t r, size_t c, const double*& src) {        // row-major flat -> matrix
        m.resize(r, c);
        for (size_t i = 0; i < r; ++i) for (size_t j = 0; j < c; ++j) m(i, j) = *src++;
    }
    void refresh() {                                     // the public members, from the device's per-latent record
        double flat[256];
        const long long n = moihgp_cuda_latent_consts(_h, 0, flat, 256);
        if (n < 0) throw std::runtime_error("moihgp_cuda_latent_consts failed");
        const double* s = flat;
        const size_t d = _dim;
        put(A, d, d, s); put(Q, d, d, s); put(K, d, 1, s); put(S, 1, 1, s); put(PF, d, d, s); put(HA, 1, d, s); put(AKHA, d, d, s);
        dS.resize(3); dA.resize(3); dK.resize(3); dAKHA.resize(3); HdA.resize(3);
        for (int k = 0; k < 3; ++k) { put(dS[k], 1, 1, s); put(dA[k], d, d, s); put(dK[k], d, 1, s); put(dAKHA[k], d, d, s); put(HdA[k], d, 1, s); }
    }
    moihgp_handle* _h;
    size_t _dim, _num_param;
};

// ------------------------------------------------------------------------------------------------------------------
// MOIHGP<StateSpace>   (moihgp.h:76-757)
template <typename StateSpace, typename Vec = std::vector<double>, typename Mat = DenseMatrix>
class MOIHGP {
public:
    typedef std::vector<Vec> State;                      // x[l]      : IGP state of latent l            (d)
    typedef std::vector<std::vector<Vec> > DState;       // dx[l][k]  : its derivative w.r.t. parameter k (d)

    // moihgp.h:741-744.  U (p x L polar factor), S (L) and sigma mirror the model on the device and are refreshed by the
    // constructor and by update(); writing to them does not change the model (use update(params)).  dA[r * L + c] is the
    // p x L unit matrix E_rc of the reference's dU loop (moihgp.h:94-101, :545) - generated on access: the reference
    // stores all p*L of them (2 GB at p = 256, L = 64).
    struct UnitMatrices {
        UnitMatrices() : p(0), L(0) {}
        size_t size() const { return p * L; }
        Mat operator[](size_t idx) const { Mat m; m.resize(p, L); for (size_t r = 0; r < p; ++r) for (size_t c = 0; c < L; ++c) m(r, c) = 0.0; m(idx / L, idx % L) = 1.0; return m; }
        size_t p, L;
    };
    Mat U;
    Vec S;
    UnitMatrices dA;
    double sigma;

    // moihgp.h:81-136.  U starts as a random near-identity polar factor like the reference's (moihgp.h:103-125) when
    // `random_U` (the default, as the reference), or as the exact identity block otherwise.
    MOIHGP(const double& dt, const size_t& num_output, const size_t& num_latent, const bool& threading, int device = -1,
           bool random_U = true)
        : _h(NULL), _num_output(num_output), _num_latent(num_latent) {
        if (random_U) {
            _h = StateSpace::kernel == MOIHGP_MATERN32 ? gp32_new(dt, num_output, num_latent, threading) : NULL;
        }
        if (!_h) {
            if (moihgp_cuda_create(&_h, StateSpace::kernel, dt, num_output, num_latent, threading ? 1 : 0, device) != 0 || !_h)
                throw std::runtime_error("moihgp_cuda_create failed (no B200-class CUDA device? there is no CPU fallback)");
            if (random_U) {
                // Matern-5/2 with the reference's random start: draw through a throw-away Matern-3/2 handle (same U recipe)
                moihgp_handle* tmp = gp32_new(dt, num_output, num_latent, threading);
                std::vector<double> p(moihgp_cuda_num_param(tmp));
                moihgp_cuda_get_params(tmp, p.data());
                moihgp_cuda_destroy(tmp);
                moihgp_cuda_update(_h, p.data());
            }
        }
        _dim = moihgp_cuda_igp_dim(_h);
        _num_param = moihgp_cuda_num_param(_h);
        _igp_num_param = moihgp_cuda_num_igp_param(_h);
        _xb.resize(2 * _num_latent * _dim);
        _dxb.resize(2 * _num_latent * _igp_num_param * _dim);
        _yb.resize(2 * _num_output);
        _pb.resize(_num_param);
        dA.p = _num_output; dA.L = _num_latent;
        sync_public();
    }
    ~MOIHGP() { if (_h) moihgp_cuda_destroy(_h); }

    // moihgp.h:148-226  step(x, y, dx, xnew, yhat, dxnew)
    void step(const State& x, const Vec& y, const DState& dx, State& xnew, Vec& yhat, DState& dxnew) {
        pack_x(x, &_xb[0]); pack_dx(dx, &_dxb[0]); pack_y(y, &_yb[0]);
        gp32_step1(_h, &_xb[0], &_yb[0], &_dxb[0], &_xb[nx()], &_yb[_num_output], &_dxb[ndx()]);
        unpack_x(&_xb[nx()], xnew); unpack_dx(&_dxb[ndx()], dxnew); unpack_y(&_yb[_num_output], yhat);
    }
    // moihgp.h:229-301  step(x, y, dx, xnew, dxnew)
    void step(const State& x, const Vec& y, const DState& dx, State& xnew, DState& dxnew) {
        pack_x(x, &_xb[0]); pack_dx(dx, &_dxb[0]); pack_y(y, &_yb[0]);
        gp32_step2(_h, &_xb[0], &_yb[0], &_dxb[0], &_xb[nx()], &_dxb[ndx()]);
        unpack_x(&_xb[nx()], xnew); unpack_dx(&_dxb[ndx()], dxnew);
    }
    // moihgp.h:304-378  step(x, y, xnew, yhat)
    void step(const State& x, const Vec& y, State& xnew, Vec& yhat) {
        pack_x(x, &_xb[0]); pack_y(y, &_yb[0]);
        gp32_step3(_h, &_xb[0], &_yb[0], &_xb[nx()], &_yb[_num_output]);
        unpack_x(&_xb[nx()], xnew); unpack_y(&_yb[_num_output], yhat);
    }
    // moihgp.h:381-428  step(x, xnew, yhat)   (prediction only)
    void step(const State& x, State& xnew, Vec& yhat) {
        pack_x(x, &_xb[0]);
        gp32_step4(_h, &_xb[0], &_xb[nx()], &_yb[_num_output]);
        unpack_x(&_xb[nx()], xnew); unpack_y(&_yb[_num_output], yhat);
    }

    // moihgp.h:431-457
    void update(const Vec& params) {
        for (size_t i = 0; i < _num_param; ++i) _pb[i] = params[i];
        detail::check(_h, moihgp_cuda_update(_h, &_pb[0]), "MOIHGP::update");
        sync_public();
    }
    // moihgp.h:460-611
    double negLogLikelihood(const State& x, const Vec& y, const DState& dx, Vec& grad) {
        pack_x(x, &_xb[0]); pack_dx(dx, &_dxb[0]); pack_y(y, &_yb[0]);
        const double loss = gp32_lik1(_h, &_xb[0], &_yb[0], &_dxb[0], &_pb[0]);
        grad.resize(_num_param);
        for (size_t i = 0; i < _num_param; ++i) grad[i] = _pb[i];
        return loss;
    }
    // moihgp.h:614-688
    double negLogLikelihood(const State& x, const Vec& y) {
        pack_x(x, &_xb[0]); pack_y(y, &_yb[0]);
        return gp32_lik2(_h, &_xb[0], &_yb[0]);
    }

    size_t getIGPDim() { return _dim; }                  // moihgp.h:691
    size_t getNumOutput() { return _num_output; }        // moihgp.h:697
    size_t getNumLatent() { return _num_latent; }        // moihgp.h:703
    size_t getNumParam() { return _num_param; }          // moihgp.h:709
    size_t getNumIGPParam() { return _igp_num_param; }   // moihgp.h:715
    Vec getParams() {                                    // moihgp.h:721-738
        moihgp_cuda_get_params(_h, &_pb[0]);
        Vec out = detail::make_vec<Vec>(_num_param);
        for (size_t i = 0; i < _num_param; ++i) out[i] = _pb[i];
        return out;
    }

    // ---- whole-sequence entry points (the device boundary moved up to the callers' loops) ----------------------------
    // sum_t negLogLikelihood(x_t, y_t, dx_t, g) with step(x, y, dx, xnew, dxnew) advancing the state, over the T rows of
    // the packed Y[T][p]; x/dx are the carried-in state and receive the final state.
    double objective(const double* Y, size_t T, State& x, DState& dx, Vec& grad) {
        pack_x(x, &_xb[0]); pack_dx(dx, &_dxb[0]);
        double loss = 0.0;
        detail::check(_h, moihgp_cuda_objective(_h, Y, 1, T, &_xb[0], &_dxb[0], &loss, &_pb[0], &_xb[nx()], &_dxb[ndx()]), "MOIHGP::objective");
        unpack_x(&_xb[nx()], x); unpack_dx(&_dxb[ndx()], dx);
        grad.resize(_num_param);
        for (size_t i = 0; i < _num_param; ++i) grad[i] = _pb[i];
        return loss;
    }
    // loop of step(x, y, xnew, yhat) (MOIHGPRegression::predict, moihgp_regression.h:127-139) over packed Y[T][p];
    // Yhat[T][p]; optionally the filtered / smoothed states X, Xs [T][L][d] and the summed negLogLikelihood(x, y).
    void predict(const double* Y, size_t T, State& x, double* Yhat, double* X = NULL, double* Xs = NULL,
                 int smoother_mode = MOIHGP_SMOOTH_NONE, double* nll = NULL) {
        pack_x(x, &_xb[0]);
        detail::check(_h, moihgp_cuda_filter_smoother_nll(_h, Y, 1, T, &_xb[0], smoother_mode, X, Xs, Yhat, nll, &_xb[nx()]), "MOIHGP::predict");
        unpack_x(&_xb[nx()], x);
    }
    // negLogLikelihood(x, y) of every step of the same filter loop (moihgp.h:614-688) over packed Y[T][p] into nll_steps[T]
    // (NaN for a row with a missing output); x is the carried-in state and receives the final state.
    void nllSteps(const double* Y, size_t T, State& x, double* nll_steps) {
        pack_x(x, &_xb[0]);
        detail::check(_h, moihgp_cuda_nll_steps(_h, Y, 1, T, &_xb[0], nll_steps, NULL, &_xb[nx()]), "MOIHGP::nllSteps");
        unpack_x(&_xb[nx()], x);
    }

    // Keep the data set resident on the device across objective evaluations (the optimiser calls the functor tens of times
    // on the same observations); the caller re-binds after changing them.  Y = NULL releases it.
    void bindData(const double* Y, size_t T) { detail::check(_h, moihgp_cuda_bind_data(_h, Y, Y ? 1 : 0, T), "MOIHGP::bindData"); }
    double objectiveBound(State& x, DState& dx, Vec& grad) {
        pack_x(x, &_xb[0]); pack_dx(dx, &_dxb[0]);
        double loss = 0.0;
        detail::check(_h, moihgp_cuda_objective_bound(_h, &_xb[0], &_dxb[0], &loss, &_pb[0], &_xb[nx()], &_dxb[ndx()]), "MOIHGP::objectiveBound");
        unpack_x(&_xb[nx()], x); unpack_dx(&_dxb[ndx()], dx);
        grad.resize(_num_param);
        for (size_t i = 0; i < _num_param; ++i) grad[i] = _pb[i];
        return loss;
    }

    // One long sequence sharded in TIME over several devices (one MOIHGP object per device / process; SURVEY 8e): the
    // carry algebra a caller needs around moihgp_cuda_objective_begin_dev / _finish_dev and moihgp_cuda_fsn_block_dev.
    //   blockTransition(n, out): out[L][4][d*d] = [AKHA^n, E_0(n), E_1(n), E_2(n)], row-major
    //   smootherPower(mode, n, out): out[L][d*d] = G[mode]^n
    void blockTransition(size_t n, std::vector<double>& out) {
        out.assign(_num_latent * 4 * _dim * _dim, 0.0);
        detail::check(_h, moihgp_cuda_block_transition(_h, n, &out[0]), "MOIHGP::blockTransition");
    }
    void smootherPower(int smoother_mode, size_t n, std::vector<double>& out) {
        out.assign(_num_latent * _dim * _dim, 0.0);
        detail::check(_h, moihgp_cuda_smoother_power(_h, smoother_mode, n, &out[0]), "MOIHGP::smootherPower");
    }

    // Device-resident streaming learner (moihgp_cuda_online_*: window, moving mean, carried state and proximal term in HBM;
    // one CUDA-graph launch per objective evaluation).  Used by OnlineObjective; false / exception-free probes return false
    // when the shape does not qualify (the caller then keeps the window on the host).  A model with more than 64 latents is
    // refused outright: std::runtime_error with the library's message.
    bool onlineBegin(size_t windowsize) {
        const int rc = moihgp_cuda_online_begin(_h, windowsize);
        if (rc != 0 && _num_latent > 64) detail::check(_h, rc, "MOIHGP::onlineBegin");
        return rc == 0;
    }
    void onlinePush(const Vec& y, Vec& ma) {
        pack_y(y, &_yb[0]);
        detail::check(_h, moihgp_cuda_online_push(_h, &_yb[0], NULL, &_yb[_num_output]), "MOIHGP::onlinePush");
        unpack_y(&_yb[_num_output], ma);
    }
    void onlineSetProximal(const Vec& oldparams, const double* B) {
        for (size_t i = 0; i < _num_param; ++i) _pb[i] = oldparams[i];
        detail::check(_h, moihgp_cuda_online_set_proximal(_h, &_pb[0], B), "MOIHGP::onlineSetProximal");
    }
    double onlineObjective(const Vec& params, Vec& grad) {
        std::vector<double> pin(_num_param);
        for (size_t i = 0; i < _num_param; ++i) pin[i] = params[i];
        double loss = 0.0;
        detail::check(_h, moihgp_cuda_online_objective(_h, &pin[0], &loss, &_pb[0]), "MOIHGP::onlineObjective");
        grad.resize(_num_param);
        for (size_t i = 0; i < _num_param; ++i) grad[i] = _pb[i];
        sync_public();                                   // the model now holds params (host mirror only, no device traffic)
        return loss;
    }

    moihgp_handle* handle() { return _h; }

private:
    MOIHGP(const MOIHGP&);
    MOIHGP& operator=(const MOIHGP&);
    void sync_public() {                                 // U, S, sigma as the device model holds them (moihgp.h:446-449)
        moihgp_cuda_get_params(_h, &_pb[0]);             // U block = the polar factor
        U.resize(_num_output, _num_latent);
        for (size_t r = 0; r < _num_output; ++r) for (size_t c = 0; c < _num_latent; ++c) U(r, c) = _pb[r * _num_latent + c];
        S.resize(_num_latent);
        for (size_t l = 0; l < _num_latent; ++l) S[l] = _pb[_num_output * _num_latent + l];
        sigma = _pb[_num_output * _num_latent + _num_latent];
    }
    size_t nx() const { return _num_latent * _dim; }
    size_t ndx() const { return _num_latent * _igp_num_param * _dim; }
    void pack_x(const State& x, double* b) const { for (size_t l = 0; l < _num_latent; ++l) for (size_t i = 0; i < _dim; ++i) b[l * _dim + i] = x[l][i]; }
    void unpack_x(const double* b, State& x) const {
        x.resize(_num_latent);
        for (size_t l = 0; l < _num_latent; ++l) { x[l].resize(_dim); for (size_t i = 0; i < _dim; ++i) x[l][i] = b[l * _dim + i]; }
    }
    void pack_dx(const DState& dx, double* b) const {
        for (size_t l = 0; l < _num_latent; ++l) for (size_t k = 0; k < _igp_num_param; ++k) for (size_t i = 0; i < _dim; ++i)
            b[(l * _igp_num_param + k) * _dim + i] = dx[l][k][i];
    }
    void unpack_dx(const double* b, DState& dx) const {
        dx.resize(_num_latent);
        for (size_t l = 0; l < _num_latent; ++l) {
            dx[l].resize(_igp_num_param);
            for (size_t k = 0; k < _igp_num_param; ++k) { dx[l][k].resize(_dim); for (size_t i = 0; i < _dim; ++i) dx[l][k][i] = b[(l * _igp_num_param + k) * _dim + i]; }
        }
    }
    void pack_y(const Vec& y, double* b) const { for (size_t i = 0; i < _num_output; ++i) b[i] = y[i]; }
    void unpack_y(const double* b, Vec& y) const { y.resize(_num_output); for (size_t i = 0; i < _num_output; ++i) y[i] = b[i]; }

    moihgp_handle* _h;
    size_t _num_output, _num_latent, _dim, _num_param, _igp_num_param;
    std::vector<double> _xb, _dxb, _yb, _pb;
};

// ------------------------------------------------------------------------------------------------------------------
// RegressionObjective<StateSpace>   (moihgp_regression.h:17-70): the L-BFGS-B functor over the data set Y.
// The reference's operator() never calls _gp->update(params) (SURVEY Q6: it optimises a function that is constant in
// params); `update_params = false` keeps that, `true` evaluates the objective AT params like OnlineObjective does.
template <typename StateSpace, typename Vec = std::vector<double>, typename Mat = DenseMatrix>
class RegressionObjective {
public:
    typedef MOIHGP<StateSpace, Vec, Mat> GP;
    RegressionObjective(const size_t& num_data, GP* gp, bool update_params = false) : _gp(gp), _update(update_params), _bound(0) { Y.reserve(num_data); }

    // Copy Y to the device once: every later operator() evaluates on that resident copy until rebind() / unbind().
    // (The optimiser calls the functor tens of times on the same data; call rebind() after changing Y.)
    void rebind() {
        const size_t p = _gp->getNumOutput(), T = Y.size();
        _buf.resize(T * p);
        for (size_t t = 0; t < T; ++t) for (size_t r = 0; r < p; ++r) _buf[t * p + r] = Y[t][r];
        _gp->bindData(T ? &_buf[0] : NULL, T);
        _bound = T;
    }
    void unbind() { _gp->bindData(NULL, 0); _bound = 0; }

    double operator()(const Vec& params, Vec& grad) {
        if (_update) _gp->update(params);
        if (_bound) {
            typename GP::State xb(_gp->getNumLatent(), detail::make_vec<Vec>(_gp->getIGPDim()));
            typename GP::DState dxb(_gp->getNumLatent(), std::vector<Vec>(_gp->getNumIGPParam(), detail::make_vec<Vec>(_gp->getIGPDim())));
            return _gp->objectiveBound(xb, dxb, grad);
        }
        const size_t p = _gp->getNumOutput(), T = Y.size();
        _buf.resize(T * p);
        for (size_t t = 0; t < T; ++t) for (size_t r = 0; r < p; ++r) _buf[t * p + r] = Y[t][r];
        typename GP::State x(_gp->getNumLatent(), detail::make_vec<Vec>(_gp->getIGPDim()));                 // zero start, :38-41
        typename GP::DState dx(_gp->getNumLatent(), std::vector<Vec>(_gp->getNumIGPParam(), detail::make_vec<Vec>(_gp->getIGPDim())));
        if (T == 0) { grad.resize(_gp->getNumParam()); for (size_t i = 0; i < _gp->getNumParam(); ++i) grad[i] = 0.0; return 0.0; }
        return _gp->objective(&_buf[0], T, x, dx, grad);                                                    // :42-50 in one pass
    }

    std::vector<Vec> Y;                                  // moihgp_regression.h:55

private:
    GP* _gp;
    bool _update;
    size_t _bound;
    std::vector<double> _buf;
};

// A stand-in for LBFGSpp::BFGSMat<double, true> with no corrections stored (get_m() == 0): the proximal term of
// OnlineObjective then uses the identity (moihgp_online.h:51-54).  Any type with get_m() and
// apply_Hv(v, a, res) -- e.g. the reference's vendored LBFGSpp::BFGSMat -- can be used instead.
template <typename Vec>
struct NoBFGSMat {
    int get_m() const { return 0; }
    void apply_Hv(const Vec&, const double&, Vec&) const {}
};

// ------------------------------------------------------------------------------------------------------------------
// OnlineObjective<StateSpace>   (moihgp_online.h:18-115): sliding-window objective with the BFGS-proximal term.
// Device-resident (SURVEY 8 f2): the window, its moving mean, the carried state (_x, _dx) and the proximal matrix live on the
// device (moihgp_cuda_online_*); push_back is one small kernel (+ one step kernel when the window slides), operator() is ONE
// CUDA-graph launch.  The public members Y, ma, oldparams, bfgs_mat keep the reference's meaning; Y and ma are host copies.
// When the shape does not qualify for the resident path (window > 1024 steps, very large p * L) the window stays on the host
// and every evaluation hands it to moihgp_cuda_objective, as before.
template <typename StateSpace, typename Vec = std::vector<double>, typename BFGSMat = NoBFGSMat<Vec>, typename Mat = DenseMatrix>
class OnlineObjective {
public:
    typedef MOIHGP<StateSpace, Vec, Mat> GP;
    OnlineObjective(GP* gp, const double& gamma, const size_t& windowsize) : _gp(gp), _gamma(gamma), _windowsize(windowsize), _prox_m(-1) {
        oldparams = _gp->getParams();
        _x = typename GP::State(_gp->getNumLatent(), detail::make_vec<Vec>(_gp->getIGPDim()));
        _dx = typename GP::DState(_gp->getNumLatent(), std::vector<Vec>(_gp->getNumIGPParam(), detail::make_vec<Vec>(_gp->getIGPDim())));
        ma = detail::make_vec<Vec>(_gp->getNumOutput());
        _resident = _gp->onlineBegin(windowsize);
    }

    // Upload the proximal term (oldparams, B) once per streamed sample - MOIHGPOnlineLearning::step calls it right after
    // setting bfgs_mat / oldparams (moihgp_online.h:182-183).  B's column j is bfgs_mat.apply_Hv(e_j, gamma) (:45-48); the
    // identity while the BFGS matrix holds no correction (:50-53).  operator() calls it by itself when oldparams changed.
    void prepare() {
        if (!_resident) return;
        const size_t np = _gp->getNumParam();
        if (bfgs_mat.get_m() > 0) {
            std::vector<double> B(np * np);
            Vec e = detail::make_vec<Vec>(np), col = detail::make_vec<Vec>(np);
            for (size_t j = 0; j < np; ++j) {
                e[j] = 1.0;
                bfgs_mat.apply_Hv(e, _gamma, col);
                e[j] = 0.0;
                for (size_t i = 0; i < np; ++i) B[i * np + j] = col[i];
            }
            _gp->onlineSetProximal(oldparams, &B[0]);
        } else {
            _gp->onlineSetProximal(oldparams, NULL);
        }
        _prox_old.assign(np, 0.0);
        for (size_t i = 0; i < np; ++i) _prox_old[i] = oldparams[i];
        _prox_m = bfgs_mat.get_m();
    }

    // moihgp_online.h:40-72
    double operator()(const Vec& params, Vec& grad) {
        const size_t np = _gp->getNumParam(), p = _gp->getNumOutput();
        if (_resident && !Y.empty()) {
            bool stale = _prox_m != (int)bfgs_mat.get_m() || _prox_old.size() != np;
            for (size_t i = 0; i < np && !stale; ++i) stale = _prox_old[i] != oldparams[i];
            if (stale) prepare();
            return _gp->onlineObjective(params, grad);   // update(params) + window loop + proximal term: one graph launch
        }
        Vec dparams = detail::make_vec<Vec>(np), Bp = detail::make_vec<Vec>(np);
        for (size_t i = 0; i < np; ++i) dparams[i] = params[i] - oldparams[i];
        _gp->update(params);                                                     // :43
        if (bfgs_mat.get_m() > 0) bfgs_mat.apply_Hv(dparams, _gamma, Bp);        // :45-48
        else for (size_t i = 0; i < np; ++i) Bp[i] = dparams[i];                 // :50-53
        double loss = 0.0;
        for (size_t i = 0; i < np; ++i) loss += dparams[i] * Bp[i];
        loss *= 0.5;                                                             // :54
        const size_t W = Y.size();
        _buf.resize(W * p);
        size_t t = 0;
        for (typename std::list<Vec>::const_iterator it = Y.begin(); it != Y.end(); ++it, ++t)
            for (size_t r = 0; r < p; ++r) _buf[t * p + r] = (*it)[r] - ma[r];   // :63
        typename GP::State x = _x;                                               // :57-58
        typename GP::DState dx = _dx;
        Vec g = detail::make_vec<Vec>(np);
        if (W > 0) loss += _gp->objective(&_buf[0], W, x, dx, g);                // :61-70 in one pass
        grad.resize(np);
        for (size_t i = 0; i < np; ++i) grad[i] = Bp[i] + g[i];
        return loss;
    }

    // moihgp_online.h:75-93 (including Q12: the carried state advances with the NEW front element)
    void push_back(const Vec& y) {
        const size_t p = _gp->getNumOutput();
        Y.push_back(y);
        if (_resident) {
            _gp->onlinePush(y, ma);                      // mean, slide and carried-state step on the device
            while (Y.size() > _windowsize) Y.pop_front();
            return;
        }
        for (size_t r = 0; r < p; ++r) ma[r] = 0.0;
        for (typename std::list<Vec>::const_iterator it = Y.begin(); it != Y.end(); ++it) for (size_t r = 0; r < p; ++r) ma[r] += (*it)[r];
        for (size_t r = 0; r < p; ++r) ma[r] /= double(Y.size());
        while (Y.size() > _windowsize) {
            Y.pop_front();
            Vec yc = detail::make_vec<Vec>(p);
            for (size_t r = 0; r < p; ++r) yc[r] = Y.front()[r] - ma[r];
            typename GP::State xnew;
            typename GP::DState dxnew;
            _gp->step(_x, yc, _dx, xnew, dxnew);
            _x = xnew;
            _dx = dxnew;
        }
    }

    bool resident() const { return _resident; }

    Vec oldparams;                                       // moihgp_online.h:96-99
    BFGSMat bfgs_mat;
    std::list<Vec> Y;
    Vec ma;

private:
    GP* _gp;
    double _gamma;
    size_t _windowsize;
    bool _resident;
    int _prox_m;
    std::vector<double> _prox_old;
    typename GP::State _x;
    typename GP::DState _dx;
    std::vector<double> _buf;
};

}  // namespace moihgp_b200
#endif  // MOIHGP_B200_MOIHGP_HPP
