// Shared device-side types for the MOIHGP hot path (sm_100a).
//
// Everything per-latent that is time-invariant ("infinite horizon": the steady-state gain, the
// innovation variance, their hyper-parameter derivatives, the smoother gain) lives in one
// LatentConsts record in HBM, produced by the K-setup kernel (setup.cu) once per update(params)
// and read by every other kernel.  Matrices are row-major with a fixed row stride of 3
// (state dimension d = 2 for Matern-3/2, 3 for Matern-5/2); unused entries are zero.
#pragma once
#include <cstddef>
#include <cstdint>
#include <math.h>

namespace moihgp {

constexpr int DMAX = 3;        // largest state dimension (Matern-5/2)
constexpr int NPAR = 3;        // hyper-parameters per latent: magnitude, lengthscale, noise
constexpr int NPOW = 40;       // A^(2^k) tables, k = 0..NPOW-1 (T < 2^40)

// reference: IHGP public members, ihgp.h:243-254 (+ the locals of IHGP::update / backwardSmoother)
struct LatentConsts {
    double A[9];          // expm(dt F)                                  ihgp.h:120
    double Q[9];          // sym(Pinf - A Pinf A')                       ihgp.h:121-122
    double PP[9];         // literal DARE iterate                        ihgp.h:125, dare.h:10-33
    double PF[9];         // PP - K H PP                                 ihgp.h:128
    double AKHA[9];       // A - K H A                                   ihgp.h:130
    double K[3];          // PP H' / S                                   ihgp.h:127
    double HA[3];         // H A                                         ihgp.h:129
    double S;             // H PP H' + R                                 ihgp.h:126
    double hak;           // HA . K                                      moihgp.h:511
    double logS;
    double dS[3];         // ihgp.h:188
    double dA[3][9];      // ihgp.h:143,167
    double dAKHA[3][9];   // ihgp.h:192,197
    double dK[3][3];      // ihgp.h:189
    double HdA[3][3];     // ihgp.h:193,198
    double G[2][9];       // smoother gain: [0] reference_literal (ihgp.h:106), [1] rts_correct
    double Ps[2][9];      // smoothed covariance: [0] literal DLyap iterate (ihgp.h:107), [1] exact
    double GK[3];         // G[1] K   (drive of the rts_correct error recursion)
    double ImA[9];        // I - A    (drive of the literal recursion, ihgp.h:111)
    double Bs[9];         // I - G[1] A   (rts_correct written as Xs[j] = Bs X[j] + G Xs[j+1])
    double params[3];     // magnitude, lengthscale, noise
    double powM[NPOW][9]; // AKHA^(2^k)
    double powG[2][NPOW][9];  // G[mode]^(2^k)
    int iters[4];         // DARE, DLyap x3 iteration counts (1-based)
    int conv[4];          // their converged flags (ignored by the reference; diagnostics here)
    int smooth_iters;     // literal smoother DLyap iterations
    int dim;
    // posterior sampling (sample.cu), lower-triangular factors of positive semi-definite matrices
    double LF[9];         // LF LF' = PF                               (the end of a sequence)
    double LC[9];         // LC LC' = PF - G[1] PPc G[1]'  (PPc = A PF A' + Q: x[t] given x[t+1])
};

// OILMM mixing parameters (moihgp.h:741-744) as the kernels see them
struct MixView {
    const double* U;      // [p][L] row-major, orthonormal columns (polar factor, moihgp.h:431-447)
    const double* S;      // [L]
    double sigma;
    int p, L;
};

// The NLL's constant per time step, 1/2 log(sum_l S_l) + 1/2 m_n log(sigma) with m_n = max(p - L, 0)   moihgp.h:502-503
__host__ __device__ inline double nll_step_const(const double* S, int p, int L, double sigma) {
    const double m_n = fmax((double)(p - L), 0.0);
    double Ssum = 0.0;
    for (int l = 0; l < L; ++l) Ssum += S[l];
    return 0.5 * log(Ssum) + 0.5 * m_n * log(sigma);
}

}  // namespace moihgp
