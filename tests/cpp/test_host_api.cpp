// GPU test of the C++ host mirror (include/moihgp_b200/moihgp.hpp) against the CPU oracle (oracle/_build/liboracle.so,
// test infrastructure).  Reads like the reference's own usage (cpp_examples/example_regression.cpp:11-41,
// example_online_learning.cpp): build a MOIHGP, fill the objective's Y, evaluate the functor the optimiser would call.
// Prints "OK" and exits 0 when every comparison is within 1e-9 (norm-wise relative).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>
#include <moihgp_b200/moihgp.hpp>

extern "C" {
void* oracle_new(int kernel, double dt, size_t p, size_t L, int threading);
void oracle_del(void* h);
size_t oracle_num_param(void* h);
void oracle_update(void* h, const double* params);
void oracle_step1(void* h, const double* x, const double* y, const double* dx, double* xn, double* yh, double* dxn);
void oracle_step2(void* h, const double* x, const double* y, const double* dx, double* xn, double* dxn);
double oracle_lik1(void* h, const double* x, const double* y, const double* dx, double* grad, int literal);
double oracle_lik2(void* h, const double* x, const double* y, int literal);
double oracle_objective(void* h, const double* Y, size_t N, size_t T, double* x, double* dx, double* grad, int literal);
size_t oracle_ihgp_consts(void* h, size_t l, double* out);
void oracle_smoother_consts(void* h, size_t l, int mode, double* G, double* P);
void oracle_ihgp_smooth(void* h, size_t l, int mode, const double* X, size_t n, double* Xs);
void oracle_filter_smoother_nll(void* h, const double* Y, size_t N, size_t T, double* x, double* X, double* Xs, double* Yhat, double* nll,
                                int smoother_mode, int nthreads);
}

typedef std::vector<double> Vec;
static int failures = 0;

static double rel_err(const double* a, const double* b, size_t n) {
    double num = 0.0, den = 0.0;
    for (size_t i = 0; i < n; ++i) { num = std::fmax(num, std::fabs(a[i] - b[i])); den = std::fmax(den, std::fabs(b[i])); }
    return num / std::fmax(den, 1e-300);
}
static void expect(const char* what, double err, double tol = 1e-9) {
    std::printf("%-58s rel.err %.3e %s\n", what, err, err <= tol ? "ok" : "FAIL");
    if (!(err <= tol)) ++failures;
}

// A BFGS matrix holding corrections (get_m() > 0), H = I + w w^T with w_i = 0.1 cos(i): apply_Hv(v, a, res) = a H v, the
// call the proximal term of OnlineObjective makes (moihgp_online.h:45-48)
struct DenseBFGSMat {
    int get_m() const { return 2; }
    void apply_Hv(const Vec& v, const double& a, Vec& res) const {
        double wv = 0.0;
        for (size_t i = 0; i < v.size(); ++i) wv += 0.1 * std::cos(double(i)) * v[i];
        res.assign(v.size(), 0.0);
        for (size_t i = 0; i < v.size(); ++i) res[i] = a * (v[i] + 0.1 * std::cos(double(i)) * wv);
    }
};

template <typename SS>
static void run(int kernel, size_t p, size_t L, size_t T, bool threading, unsigned seed) {
    using namespace moihgp_b200;
    std::mt19937 gen(seed);
    std::normal_distribution<> nrm(0.0, 1.0);
    const double dt = 0.1;
    MOIHGP<SS> gp(dt, p, L, threading);
    void* o = oracle_new(kernel, dt, p, L, threading ? 1 : 0);
    const size_t np = gp.getNumParam(), d = gp.getIGPDim();
    if (np != oracle_num_param(o)) { std::printf("num_param mismatch\n"); ++failures; }
    // hyper-parameters: U block near identity (update() takes its polar factor), S, sigma, (magnitude, lengthscale, noise) x L
    Vec params(np);
    for (size_t r = 0; r < p; ++r) for (size_t c = 0; c < L; ++c) params[r * L + c] = (r == c ? 1.0 : 0.0) + 0.3 * nrm(gen);
    for (size_t l = 0; l < L; ++l) params[p * L + l] = 0.5 + 0.25 * l;
    params[p * L + L] = 0.05;
    const double table[4][3] = {{1, 1, .1}, {.5, .5, .1}, {2, .3, .05}, {.5, .3, .5}};
    for (size_t l = 0; l < L; ++l) for (int k = 0; k < 3; ++k) params[p * L + L + 1 + 3 * l + k] = table[l % 4][k];
    gp.update(params);
    oracle_update(o, params.data());

    // data: mixed sinusoids + noise (cpp_examples/example_regression.cpp:18-28)
    std::vector<Vec> Y(T, Vec(p));
    std::vector<double> Yflat(T * p);
    for (size_t t = 0; t < T; ++t) for (size_t r = 0; r < p; ++r) {
        Y[t][r] = std::sin((1.0 + r % 3) * dt * t) + 0.1 * nrm(gen);
        Yflat[t * p + r] = Y[t][r];
    }

    // (1) RegressionObjective::operator() == the oracle's loop of step + negLogLikelihood
    RegressionObjective<SS> f(T, &gp, /*update_params=*/true);
    f.Y = Y;
    Vec grad(np), go(np), x0(L * d, 0.0), dx0(L * 3 * d, 0.0);
    const double loss = f(params, grad);
    const double lo = oracle_objective(o, Yflat.data(), 1, T, x0.data(), dx0.data(), go.data(), 0);
    expect("RegressionObjective loss", std::fabs(loss - lo) / std::fabs(lo));
    expect("RegressionObjective grad", rel_err(grad.data(), go.data(), np));
    // the data set resident on the device (what the optimiser loop uses): identical results
    {
        f.rebind();
        Vec gb(np);
        const double lb = f(params, gb);
        expect("RegressionObjective (bound data) loss", std::fabs(lb - loss) / std::fabs(loss), 0.0);
        expect("RegressionObjective (bound data) grad", rel_err(gb.data(), grad.data(), np), 0.0);
        f.unbind();
    }

    // (2) per-observation methods: a few steps of step(x,y,dx,xnew,yhat,dxnew) + both negLogLikelihood overloads
    typename MOIHGP<SS>::State x(L, Vec(d, 0.0)), xn;
    typename MOIHGP<SS>::DState dx(L, std::vector<Vec>(3, Vec(d, 0.0))), dxn;
    Vec xo(L * d, 0.0), dxo(L * 3 * d, 0.0), xno(L * d), dxno(L * 3 * d), yh, yho(p), g1, g1o(np);
    double e_x = 0, e_y = 0, e_l1 = 0, e_l2 = 0, e_g = 0;
    for (size_t t = 0; t < 5 && t < T; ++t) {
        const double l1 = gp.negLogLikelihood(x, Y[t], dx, g1), l1o = oracle_lik1(o, xo.data(), Yflat.data() + t * p, dxo.data(), g1o.data(), 0);
        const double l2 = gp.negLogLikelihood(x, Y[t]), l2o = oracle_lik2(o, xo.data(), Yflat.data() + t * p, 0);
        gp.step(x, Y[t], dx, xn, yh, dxn);
        oracle_step1(o, xo.data(), Yflat.data() + t * p, dxo.data(), xno.data(), yho.data(), dxno.data());
        Vec flat(L * d);
        for (size_t l = 0; l < L; ++l) for (size_t i = 0; i < d; ++i) flat[l * d + i] = xn[l][i];
        e_x = std::fmax(e_x, rel_err(flat.data(), xno.data(), L * d));
        e_y = std::fmax(e_y, rel_err(yh.data(), yho.data(), p));
        e_l1 = std::fmax(e_l1, std::fabs(l1 - l1o) / std::fabs(l1o));
        e_l2 = std::fmax(e_l2, std::fabs(l2 - l2o) / std::fabs(l2o));
        e_g = std::fmax(e_g, rel_err(g1.data(), g1o.data(), np));
        x = xn; dx = dxn; xo = xno; dxo = dxno;
    }
    expect("MOIHGP::step xnew", e_x);
    expect("MOIHGP::step yhat", e_y);
    expect("MOIHGP::negLogLikelihood(x,y,dx,grad) loss", e_l1);
    expect("MOIHGP::negLogLikelihood(x,y,dx,grad) grad", e_g);
    expect("MOIHGP::negLogLikelihood(x,y)", e_l2);

    // (3) OnlineObjective: window maintenance + objective == the same loop on the oracle, with the identity proximal term (no BFGS
    //     corrections yet) and with a BFGS matrix holding corrections
    {
        const size_t W = 4;
        OnlineObjective<SS> fo(&gp, 0.9, W);
        // oracle twin of the window logic (moihgp_online.h:75-93)
        std::vector<Vec> win;
        Vec ma(p, 0.0), sx(L * d, 0.0), sdx(L * 3 * d, 0.0), tx(L * d), tdx(L * 3 * d);
        for (size_t t = 0; t < 9 && t < T; ++t) {
            fo.push_back(Y[t]);
            win.push_back(Y[t]);
            for (size_t r = 0; r < p; ++r) { ma[r] = 0.0; for (size_t k = 0; k < win.size(); ++k) ma[r] += win[k][r]; ma[r] /= double(win.size()); }
            while (win.size() > W) {
                win.erase(win.begin());
                Vec yc(p);
                for (size_t r = 0; r < p; ++r) yc[r] = win.front()[r] - ma[r];
                oracle_step2(o, sx.data(), yc.data(), sdx.data(), tx.data(), tdx.data());
                sx = tx; sdx = tdx;
            }
        }
        Vec p2 = params;
        for (size_t i = 0; i < np; ++i) p2[i] *= 1.0 + 0.01 * std::sin(double(i));          // a trial point of the line search
        // keep the U block orthonormal-ish is not needed: update() re-takes the polar factor
        Vec g2(np), g2o(np);
        const double l2 = fo(p2, g2);
        oracle_update(o, p2.data());
        std::vector<double> wflat(win.size() * p);
        for (size_t k = 0; k < win.size(); ++k) for (size_t r = 0; r < p; ++r) wflat[k * p + r] = win[k][r] - ma[r];
        Vec cx = sx, cdx = sdx;
        double l2o = oracle_objective(o, wflat.data(), 1, win.size(), cx.data(), cdx.data(), g2o.data(), 0);
        double prox = 0.0;
        // oldparams = getParams() at construction: holds the POLAR FACTOR in its U block, not the raw block (moihgp_online.h:31, Q22)
        for (size_t i = 0; i < np; ++i) { const double dp = p2[i] - fo.oldparams[i]; prox += 0.5 * dp * dp; g2o[i] += dp; }
        l2o += prox;
        expect("OnlineObjective loss (window 4, proximal identity)", std::fabs(l2 - l2o) / std::fabs(l2o));
        expect("OnlineObjective grad", rel_err(g2.data(), g2o.data(), np));
        gp.update(params);
        oracle_update(o, params.data());
        // the same window with BFGS corrections: prepare() builds B column by column from apply_Hv and uploads it
        OnlineObjective<SS, Vec, DenseBFGSMat> fb(&gp, 0.9, W);
        for (size_t t = 0; t < 9 && t < T; ++t) fb.push_back(Y[t]);
        fb.prepare();
        Vec g3(np), g3o(np), dp(np), Bp(np);
        const double l3 = fb(p2, g3);
        oracle_update(o, p2.data());
        cx = sx;
        cdx = sdx;
        double l3o = oracle_objective(o, wflat.data(), 1, win.size(), cx.data(), cdx.data(), g3o.data(), 0);
        for (size_t i = 0; i < np; ++i) dp[i] = p2[i] - fb.oldparams[i];
        fb.bfgs_mat.apply_Hv(dp, 0.9, Bp);
        for (size_t i = 0; i < np; ++i) { l3o += 0.5 * dp[i] * Bp[i]; g3o[i] += Bp[i]; }
        expect("OnlineObjective loss (window 4, BFGS corrections)", std::fabs(l3 - l3o) / std::fabs(l3o));
        expect("OnlineObjective grad (BFGS corrections)", rel_err(g3.data(), g3o.data(), np));
        gp.update(params);
        oracle_update(o, params.data());
    }

    // (4) predict(): loop of step(x, y, xnew, yhat) + smoother, one device pass
    {
        typename MOIHGP<SS>::State xs(L, Vec(d, 0.0));
        std::vector<double> Yh(T * p), X(T * L * d), Xs(T * L * d), Yho(T * p), Xo(T * L * d), Xso(T * L * d), xz(L * d, 0.0);
        double nll = 0.0, nllo = 0.0;
        gp.predict(Yflat.data(), T, xs, Yh.data(), X.data(), Xs.data(), MOIHGP_SMOOTH_RTS, &nll);
        oracle_filter_smoother_nll(o, Yflat.data(), 1, T, xz.data(), Xo.data(), Xso.data(), Yho.data(), &nllo, 1, 1);
        expect("predict Yhat", rel_err(Yh.data(), Yho.data(), T * p));
        expect("predict filtered states", rel_err(X.data(), Xo.data(), T * L * d));
        expect("predict smoothed states (RTS)", rel_err(Xs.data(), Xso.data(), T * L * d));
        expect("predict NLL", std::fabs(nll - nllo) / std::fabs(nllo));
    }
    // (5) blockTransition / smootherPower: the carry algebra of a sequence sharded in time.  The filter is affine in its
    //     initial state, x_T(x0) - x_T(0) = AKHA^T x0, and G^(a+b) = G^a G^b.
    {
        typename MOIHGP<SS>::State xa(L, Vec(d, 0.0)), xb(L, Vec(d, 0.0));
        for (size_t l = 0; l < L; ++l) for (size_t i = 0; i < d; ++i) xa[l][i] = 0.1 * (double)(l + 1) - 0.07 * (double)i;
        typename MOIHGP<SS>::State x0 = xa;
        const size_t Ts = T < 6 ? T : 6;                 // a short block: AKHA^n x0 decays geometrically
        gp.predict(Yflat.data(), Ts, xa, NULL, NULL, NULL, MOIHGP_SMOOTH_NONE, NULL);
        gp.predict(Yflat.data(), Ts, xb, NULL, NULL, NULL, MOIHGP_SMOOTH_NONE, NULL);
        std::vector<double> tr, lhs(L * d), rhs(L * d);
        gp.blockTransition(Ts, tr);
        for (size_t l = 0; l < L; ++l) for (size_t i = 0; i < d; ++i) {
            double a = 0.0;
            for (size_t j = 0; j < d; ++j) a += tr[(l * 4 + 0) * d * d + i * d + j] * x0[l][j];
            rhs[l * d + i] = a;
            lhs[l * d + i] = xa[l][i] - xb[l][i];
        }
        expect("blockTransition: x_n(x0) - x_n(0) = AKHA^n x0", rel_err(lhs.data(), rhs.data(), L * d));
        std::vector<double> g5, g7, g12, prod(L * d * d);
        gp.smootherPower(MOIHGP_SMOOTH_RTS, 5, g5); gp.smootherPower(MOIHGP_SMOOTH_RTS, 7, g7); gp.smootherPower(MOIHGP_SMOOTH_RTS, 12, g12);
        for (size_t l = 0; l < L; ++l) for (size_t i = 0; i < d; ++i) for (size_t j = 0; j < d; ++j) {
            double a = 0.0;
            for (size_t q = 0; q < d; ++q) a += g5[l * d * d + i * d + q] * g7[l * d * d + q * d + j];
            prod[l * d * d + i * d + j] = a;
        }
        expect("smootherPower: G^12 = G^5 G^7", rel_err(prod.data(), g12.data(), L * d * d));
    }
    oracle_del(o);
}

// IHGP<StateSpace> (ihgp.h:17-263): public members, the four step overloads (incl. the NaN prediction branch), both
// negLogLikelihood overloads, backwardSmoother, update / getParams - against the oracle's single-latent model.
template <typename SS>
static void run_ihgp(int kernel, unsigned seed) {
    using namespace moihgp_b200;
    std::mt19937 gen(seed);
    std::normal_distribution<> nrm(0.0, 1.0);
    const double dt = 0.1;
    IHGP<SS> gp(dt);
    void* o = oracle_new(kernel, dt, 1, 1, 0);
    const size_t d = gp.getDim();
    Vec prm(3);
    prm[0] = 0.5; prm[1] = 0.5; prm[2] = 0.1;                                 // rho(G) < 1 in the literal smoother too
    gp.update(prm);
    const double op[6] = {1.0, 1.0, 1e-2, prm[0], prm[1], prm[2]};
    oracle_update(o, op);
    expect("IHGP::getParams", rel_err(gp.getParams().data(), prm.data(), 3));
    // public members (ihgp.h:243-254) against the oracle's flat record: A Q K S PF HA AKHA, then per k: dS dA dK dAKHA HdA
    double flat[256];
    oracle_ihgp_consts(o, 0, flat);
    std::vector<double> mine;
    auto add = [&](const DenseMatrix& m) { for (size_t i = 0; i < m.rows(); ++i) for (size_t j = 0; j < m.cols(); ++j) mine.push_back(m(i, j)); };
    add(gp.A); add(gp.Q); add(gp.K); add(gp.S); add(gp.PF); add(gp.HA); add(gp.AKHA);
    for (int k = 0; k < 3; ++k) { add(gp.dS[k]); add(gp.dA[k]); add(gp.dK[k]); add(gp.dAKHA[k]); add(gp.HdA[k]); }
    expect("IHGP public members A..HdA", rel_err(mine.data(), flat, mine.size()));
    // steps + likelihoods along a short sequence
    Vec x(d, 0.0), xn, xo(d, 0.0), xno(d), dxo(3 * d, 0.0), dxno(3 * d), g, go(6);
    std::vector<Vec> dx(3, Vec(d, 0.0)), dxn;
    std::vector<Vec> X;
    double e_x = 0, e_dx = 0, e_y = 0, e_l = 0, e_g = 0;
    for (int t = 0; t < 60; ++t) {
        const double y = std::sin(0.3 * t) + 0.1 * nrm(gen);
        double yh = 0.0, yho = 0.0;
        const double l1 = gp.negLogLikelihood(x, y, dx, g), l2 = gp.negLogLikelihood(x, y);
        const double l2o = oracle_lik2(o, xo.data(), &y, 0);
        oracle_lik1(o, xo.data(), &y, dxo.data(), go.data(), 0);
        gp.step(x, y, dx, xn, yh, dxn);
        oracle_step1(o, xo.data(), &y, dxo.data(), xno.data(), &yho, dxno.data());
        Vec dflat(3 * d);
        for (int k = 0; k < 3; ++k) for (size_t i = 0; i < d; ++i) dflat[k * d + i] = dxn[k][i];
        e_x = std::fmax(e_x, rel_err(xn.data(), xno.data(), d));
        e_dx = std::fmax(e_dx, rel_err(dflat.data(), dxno.data(), 3 * d));
        e_y = std::fmax(e_y, std::fabs(yh - yho) / std::fmax(std::fabs(yho), 1e-300));
        e_l = std::fmax(e_l, std::fmax(std::fabs(l1 - l2o), std::fabs(l2 - l2o)) / std::fabs(l2o));
        e_g = std::fmax(e_g, rel_err(g.data(), go.data() + 3, 3));
        x = xn; dx = dxn; xo = xno; dxo = dxno;
        X.push_back(x);
    }
    expect("IHGP::step xnew", e_x);
    expect("IHGP::step dxnew", e_dx);
    expect("IHGP::step yhat", e_y);
    expect("IHGP::negLogLikelihood (both overloads) loss", e_l);
    expect("IHGP::negLogLikelihood grad", e_g);
    // NaN observation: prediction step xnew = A x, dxnew_k = dA_k x + A dx_k (ihgp.h:39-47), also through step(x, xnew, yhat)
    {
        double yh = 0.0, yh4 = 0.0;
        Vec x4;
        gp.step(x, std::nan(""), dx, xn, yh, dxn);
        gp.step(x, x4, yh4);
        Vec want(d, 0.0), wd(3 * d, 0.0), got(3 * d);
        for (size_t i = 0; i < d; ++i) for (size_t j = 0; j < d; ++j) want[i] += gp.A(i, j) * x[j];
        for (int k = 0; k < 3; ++k) for (size_t i = 0; i < d; ++i) {
            for (size_t j = 0; j < d; ++j) wd[k * d + i] += gp.dA[k](i, j) * x[j] + gp.A(i, j) * dx[k][j];
            got[k * d + i] = dxn[k][i];
        }
        expect("IHGP::step(NaN) xnew = A x", rel_err(xn.data(), want.data(), d), 1e-14);
        expect("IHGP::step(NaN) dxnew = dA x + A dx", rel_err(got.data(), wd.data(), 3 * d), 1e-13);
        expect("IHGP::step(x, xnew, yhat)", rel_err(x4.data(), want.data(), d) + std::fabs(yh4 - want[0]) + std::fabs(yh - want[0]), 1e-14);
    }
    // backwardSmoother (ihgp.h:103-114) on the filtered states
    {
        std::vector<Vec> Xprev;
        DenseMatrix P, G;
        gp.backwardSmoother(X, Xprev, P, G);
        std::vector<double> xin(X.size() * d), xso(X.size() * d), xs(X.size() * d), Go(d * d), Po(d * d), Gm(d * d), Pm(d * d);
        for (size_t t = 0; t < X.size(); ++t) for (size_t i = 0; i < d; ++i) { xin[t * d + i] = X[t][i]; xs[t * d + i] = Xprev[t][i]; }
        oracle_ihgp_smooth(o, 0, 0, xin.data(), X.size(), xso.data());
        oracle_smoother_consts(o, 0, 0, Go.data(), Po.data());
        for (size_t i = 0; i < d; ++i) for (size_t j = 0; j < d; ++j) { Gm[i * d + j] = G(i, j); Pm[i * d + j] = P(i, j); }
        expect("IHGP::backwardSmoother Xprev", Xprev.size() == X.size() ? rel_err(xs.data(), xso.data(), xs.size()) : 1.0);
        expect("IHGP::backwardSmoother G", rel_err(Gm.data(), Go.data(), d * d));
        expect("IHGP::backwardSmoother P", rel_err(Pm.data(), Po.data(), d * d));
    }
    oracle_del(o);
}

// MOIHGP public members U, S, dA, sigma (moihgp.h:741-744)
static void run_public_members() {
    using namespace moihgp_b200;
    const size_t p = 5, L = 2;
    MOIHGP<Matern32StateSpace> gp(0.1, p, L, false);
    Vec prm = gp.getParams();
    prm[p * L] = 1.7; prm[p * L + 1] = 0.4; prm[p * L + L] = 0.03;
    for (size_t i = 0; i < p * L; ++i) prm[i] += 0.05 * std::sin(1.0 + i);
    gp.update(prm);
    Vec now = gp.getParams();
    double e = 0.0, orth = 0.0;
    for (size_t r = 0; r < p; ++r) for (size_t c = 0; c < L; ++c) e = std::fmax(e, std::fabs(gp.U(r, c) - now[r * L + c]));
    for (size_t a = 0; a < L; ++a) for (size_t b = 0; b < L; ++b) {
        double s = 0.0;
        for (size_t r = 0; r < p; ++r) s += gp.U(r, a) * gp.U(r, b);
        orth = std::fmax(orth, std::fabs(s - (a == b ? 1.0 : 0.0)));
    }
    expect("MOIHGP::U == polar factor held by the model", e, 0.0);
    expect("MOIHGP::U orthonormal columns", orth, 1e-13);
    expect("MOIHGP::S, sigma", std::fabs(gp.S[0] - 1.7) + std::fabs(gp.S[1] - 0.4) + std::fabs(gp.sigma - 0.03), 0.0);
    DenseMatrix E = gp.dA[1 * L + 1];
    double s = 0.0;
    for (size_t r = 0; r < p; ++r) for (size_t c = 0; c < L; ++c) s += E(r, c);
    expect("MOIHGP::dA[idx] = unit matrix E_rc", std::fabs(s - 1.0) + std::fabs(E(1, 1) - 1.0) + (gp.dA.size() == p * L ? 0.0 : 1.0), 0.0);
}

int main() {
    std::printf("-- IHGP<Matern32>, IHGP<Matern52>\n");
    run_ihgp<moihgp_b200::Matern32StateSpace>(32, 5);
    run_ihgp<moihgp_b200::Matern52StateSpace>(52, 6);
    run_public_members();
    std::printf("-- Matern32, p=2, L=1, T=63 (example_regression shape)\n");
    run<moihgp_b200::Matern32StateSpace>(32, 2, 1, 63, false, 1);
    std::printf("-- Matern32, p=8, L=4, T=300, threading\n");
    run<moihgp_b200::Matern32StateSpace>(32, 8, 4, 300, true, 2);
    std::printf("-- Matern52, p=16, L=8, T=700, threading\n");
    run<moihgp_b200::Matern52StateSpace>(52, 16, 8, 700, true, 3);
    if (failures) { std::printf("FAILED: %d comparison(s)\n", failures); return 1; }
    std::printf("OK\n");
    return 0;
}
