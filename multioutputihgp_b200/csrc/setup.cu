// K-setup: per-latent steady-state solve, one warp per latent (sm_100a).
//
// Replaces (reference, /root/reference/moihgp/include):
//   moihgp/matern32ss.h:40-64, moihgp/matern52ss.h:38-75   state-space matrices and derivatives
//   moihgp/ihgp.h:117-201                                   IHGP::update
//   utils/dare.h:10-33, :36-58                              DARE / DLyap fixed-point iterations
//   moihgp/ihgp.h:105-107                                   smoother gain / covariance
//
// Parity notes (SURVEY.md section 9).  DARE and DLyap are the reference's LITERAL fixed-point
// iterations (<= 100 iterations, tol 1e-8, signed-max stop test), not doubling or Schur solvers:
// the reference's results are whatever iterate the loop stops on.  This file is compiled with
// -fmad=false so that the stop decisions see the same roundings as the host compiler's.
//
// Work split: one CTA per latent, six warps with one job each (see k_setup below) - the independent pieces (the three
// hyper-parameters' DLyap iterations, both smoothers, the block exponential, the 2^k power tables of AKHA / G used by the
// chunked scans) run concurrently instead of as serialised divergent lanes of one warp.
#include <cuda_runtime.h>
#include <math.h>
#include "moihgp_device.cuh"

namespace moihgp {

namespace {

constexpr double kDareTol = 1e-8;   // dare.h:7
constexpr int kDareMaxIter = 100;   // dare.h:8

// ---- tiny dense helpers, compile-time sizes, row-major --------------------------------------
template <int R, int K, int C>
__device__ __forceinline__ void mm(const double* a, const double* b, double* out) {
    double t[R * C];
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
        for (int j = 0; j < C; ++j) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < K; ++k) s += a[i * K + k] * b[k * C + j];
            t[i * C + j] = s;
        }
#pragma unroll
    for (int i = 0; i < R * C; ++i) out[i] = t[i];
}
template <int R, int C>
__device__ __forceinline__ void tr(const double* a, double* out) {
    double t[R * C];
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
        for (int j = 0; j < C; ++j) t[j * R + i] = a[i * C + j];
#pragma unroll
    for (int i = 0; i < R * C; ++i) out[i] = t[i];
}
template <int N> __device__ __forceinline__ void addv(const double* a, const double* b, double* o) {
#pragma unroll
    for (int i = 0; i < N; ++i) o[i] = a[i] + b[i];
}
template <int N> __device__ __forceinline__ void subv(const double* a, const double* b, double* o) {
#pragma unroll
    for (int i = 0; i < N; ++i) o[i] = a[i] - b[i];
}
template <int N> __device__ __forceinline__ void scl(const double* a, double s, double* o) {
#pragma unroll
    for (int i = 0; i < N; ++i) o[i] = a[i] * s;
}
template <int N> __device__ __forceinline__ void cpy(const double* a, double* o) {
#pragma unroll
    for (int i = 0; i < N; ++i) o[i] = a[i];
}
template <int N> __device__ __forceinline__ void zero(double* o) {
#pragma unroll
    for (int i = 0; i < N; ++i) o[i] = 0.0;
}
template <int N> __device__ __forceinline__ bool all_zero(const double* a) {
    bool z = true;
#pragma unroll
    for (int i = 0; i < N; ++i) z = z && (a[i] == 0.0);
    return z;
}
template <int N> __device__ __forceinline__ void eye(double* o) {
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) o[i * N + j] = (i == j) ? 1.0 : 0.0;
}

// Solve A X = B, A (N x N), B (N x M): Gaussian elimination with partial pivoting.
template <int N, int M>
__device__ void solve_lu(double* A, double* B, double* X) {
    for (int k = 0; k < N; ++k) {
        int piv = k;
        for (int i = k + 1; i < N; ++i) if (fabs(A[i * N + k]) > fabs(A[piv * N + k])) piv = i;
        if (piv != k) {
            for (int j = 0; j < N; ++j) { double t = A[k * N + j]; A[k * N + j] = A[piv * N + j]; A[piv * N + j] = t; }
            for (int j = 0; j < M; ++j) { double t = B[k * M + j]; B[k * M + j] = B[piv * M + j]; B[piv * M + j] = t; }
        }
        for (int i = k + 1; i < N; ++i) {
            const double f = A[i * N + k] / A[k * N + k];
            for (int j = k; j < N; ++j) A[i * N + j] -= f * A[k * N + j];
            for (int j = 0; j < M; ++j) B[i * M + j] -= f * B[k * M + j];
        }
    }
    for (int j = 0; j < M; ++j)
        for (int i = N - 1; i >= 0; --i) {
            double s = B[i * M + j];
            for (int k = i + 1; k < N; ++k) s -= A[i * N + k] * X[k * M + j];
            X[i * M + j] = s / A[i * N + i];
        }
}

// Matrix exponential, Higham (2005) scaling and squaring with the [13/13] Pade approximant -
// the published algorithm behind Eigen's MatrixBase::exp() that the reference calls at
// ihgp.h:120 and ihgp.h:167.
template <int N>
__device__ void expm(const double* Ain, double* out) {
    constexpr int NN = N * N;
    double l1 = 0.0;
    for (int j = 0; j < N; ++j) { double s = 0.0; for (int i = 0; i < N; ++i) s += fabs(Ain[i * N + j]); l1 = fmax(l1, s); }
    int sq = 0;
    if (l1 > 5.371920351148152) { int e = 0; frexp(l1 / 5.371920351148152, &e); sq = e > 0 ? e : 0; }
    double A[NN], A2[NN], A4[NN], A6[NN], U[NN], V[NN], I[NN], T[NN];
    scl<NN>(Ain, ldexp(1.0, -sq), A);
    eye<N>(I);
    mm<N, N, N>(A, A, A2);
    mm<N, N, N>(A2, A2, A4);
    mm<N, N, N>(A4, A2, A6);
    const double b[14] = {64764752532480000., 32382376266240000., 7771770303897600., 1187353796428800.,
                          129060195264000., 10559470521600., 670442572800., 33522128640., 1323241920.,
                          40840800., 960960., 16380., 182., 1.};
    for (int i = 0; i < NN; ++i) T[i] = b[13] * A6[i] + b[11] * A4[i] + b[9] * A2[i];
    mm<N, N, N>(A6, T, U);
    for (int i = 0; i < NN; ++i) U[i] = U[i] + b[7] * A6[i] + b[5] * A4[i] + b[3] * A2[i] + b[1] * I[i];
    mm<N, N, N>(A, U, U);
    for (int i = 0; i < NN; ++i) T[i] = b[12] * A6[i] + b[10] * A4[i] + b[8] * A2[i];
    mm<N, N, N>(A6, T, V);
    for (int i = 0; i < NN; ++i) V[i] = V[i] + b[6] * A6[i] + b[4] * A4[i] + b[2] * A2[i] + b[0] * I[i];
    double den[NN], num[NN];
    subv<NN>(V, U, den);
    addv<NN>(V, U, num);
    solve_lu<N, N>(den, num, out);
    for (int i = 0; i < sq; ++i) mm<N, N, N>(out, out, out);
}

template <int D> __device__ __forceinline__ double max_coeff(const double* a) {
    double m = a[0];
#pragma unroll
    for (int i = 1; i < D * D; ++i) m = a[i] > m ? a[i] : m;
    return m;
}
template <int D> __device__ __forceinline__ void symmetrize(const double* a, double* o) {
    double t[D * D];
    tr<D, D>(a, t);
#pragma unroll
    for (int i = 0; i < D * D; ++i) o[i] = (a[i] + t[i]) / 2.0;
}

// dare.h:10-33 with Bd = H' = e0 and a 1x1 R (the only way ihgp.h:125 calls it).  The chain
// AdT*P*Bd*(R+BdT*P*Bd)^-1*BdT*P*Ad collapses, without changing any rounding (products with
// exact 0/1 entries), to (col0(AdT*P) * inv) (x) row0(P) * Ad.
template <int D>
__device__ bool dare_literal(const double* Ad, const double* Q, double R, double* P, int* iters) {
    constexpr int DD = D * D;
    double AdT[DD];
    tr<D, D>(Ad, AdT);
    cpy<DD>(Q, P);                                                    // dare.h:12
    for (int it = 0; it < kDareMaxIter; ++it) {
        double AtP[DD], T1[DD], T2[DD], W[DD], Pn[DD], Df[DD];
        mm<D, D, D>(AdT, P, AtP);
        mm<D, D, D>(AtP, Ad, T1);
        const double inv = 1.0 / (R + P[0]);
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = 0; j < D; ++j) W[i * D + j] = (AtP[i * D] * inv) * P[j];
        mm<D, D, D>(W, Ad, T2);
#pragma unroll
        for (int i = 0; i < DD; ++i) Pn[i] = (T1[i] - T2[i]) + Q[i];  // dare.h:23
        subv<DD>(Pn, P, Df);
        const double diff = fabs(max_coeff<D>(Df));                   // dare.h:25 (signed max, Q1)
        symmetrize<D>(Pn, P);                                         // dare.h:26
        if (diff < kDareTol) { *iters = it + 1; return true; }        // dare.h:27
    }
    *iters = kDareMaxIter;
    return false;                                                     // dare.h:32
}

// dare.h:36-58: P <- Ad' P Ad - P + Q   (sic, Q2)
template <int D>
__device__ bool dlyap_literal(const double* Ad, const double* Q, double* P, int* iters) {
    constexpr int DD = D * D;
    double AdT[DD];
    tr<D, D>(Ad, AdT);
    cpy<DD>(Q, P);
    for (int it = 0; it < kDareMaxIter; ++it) {
        double T[DD], Pn[DD], Df[DD];
        mm<D, D, D>(AdT, P, T);
        mm<D, D, D>(T, Ad, T);
#pragma unroll
        for (int i = 0; i < DD; ++i) Pn[i] = (T[i] - P[i]) + Q[i];    // dare.h:48
        subv<DD>(Pn, P, Df);
        const double diff = fabs(max_coeff<D>(Df));                   // dare.h:50
        symmetrize<D>(Pn, P);                                         // dare.h:51
        if (diff < kDareTol) { *iters = it + 1; return true; }
    }
    *iters = kDareMaxIter;
    return false;
}

template <int D>
struct StateSpace {
    double F[D * D], Pinf[D * D], dF1[D * D], dPinf0[D * D], dPinf1[D * D], R;
};

// matern32ss.h:40-64
__device__ void state_space(StateSpace<2>& s, double magnitude, double lengthscale, double noise) {
    const double lam = sqrt(3.0) / lengthscale;                       // :44
    const double lam2 = lam * lam;
    const double len3 = 6.0 / (lengthscale * lengthscale * lengthscale);  // :46
    zero<4>(s.F); zero<4>(s.Pinf); zero<4>(s.dF1); zero<4>(s.dPinf0); zero<4>(s.dPinf1);
    s.F[1] = 1.0; s.F[2] = -lam2; s.F[3] = -2.0 * lam;                // matern32ss.h:20,47-48
    s.Pinf[0] = magnitude; s.Pinf[3] = magnitude * lam2;              // :49-50
    s.R = noise;
    s.dF1[2] = len3; s.dF1[3] = 2.0 * lam / lengthscale;              // :54-55
    s.dPinf0[0] = 1.0; s.dPinf0[3] = lam2;                            // :27 (identity) + :58
    s.dPinf1[3] = -magnitude * len3;                                  // :61
}
// matern52ss.h:38-75 (lam = sqrt(3)/l in F, sqrt(5)-consistent Pinf and dF: Q4, replicated)
__device__ void state_space(StateSpace<3>& s, double magnitude, double lengthscale, double noise) {
    const double lam = sqrt(3.0) / lengthscale;                       // :42
    const double lam2 = lam * lam;
    const double len2 = lengthscale * lengthscale, len3 = len2 * lengthscale, len4 = len2 * len2;
    const double kappa = 5.0 / 3.0 * magnitude / len2;                // :47
    const double kappa2 = -2.0 * kappa / lengthscale;                 // :48
    const double sq5 = sqrt(5.0);
    zero<9>(s.F); zero<9>(s.Pinf); zero<9>(s.dF1); zero<9>(s.dPinf0); zero<9>(s.dPinf1);
    s.F[1] = 1.0; s.F[5] = 1.0;                                       // :20-21
    s.F[6] = -lam2 * lam; s.F[7] = -3.0 * lam2; s.F[8] = -3.0 * lam;  // :50-52
    s.Pinf[0] = magnitude; s.Pinf[8] = 25.0 * magnitude / len4;       // :53-54
    s.Pinf[4] = kappa; s.Pinf[6] = -kappa; s.Pinf[2] = -kappa;        // :55-57
    s.R = noise;
    s.dF1[6] = 15.0 * sq5 / len4; s.dF1[7] = 30.0 / len3; s.dF1[8] = sq5 * lam2;   // :61-63
    for (int i = 0; i < 9; ++i) s.dPinf0[i] = s.Pinf[i] / magnitude;  // :66
    s.dPinf1[4] = kappa2; s.dPinf1[6] = -kappa2; s.dPinf1[2] = -kappa2;   // :69-71
    s.dPinf1[8] = -100.0 * magnitude / len2 / len3;                   // :72
}

// scratch shared by the lanes of one warp
template <int D>
struct WarpScratch {
    StateSpace<D> ss;
    double A[D * D], Q[D * D], PP[D * D], PF[D * D], AKHA[D * D], K[D], HA[D], AK[D], AAKH[D * D], S;
    double G[2][D * D];
};

template <int D> __device__ __forceinline__ void store_mat(const double* m, double* dst9) {
    for (int i = 0; i < 9; ++i) dst9[i] = 0.0;
    for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) dst9[i * 3 + j] = m[i * D + j];
}
template <int D> __device__ __forceinline__ void store_vec(const double* v, double* dst3) {
    for (int i = 0; i < 3; ++i) dst3[i] = i < D ? v[i] : 0.0;
}
// Lower-triangular Lo with Lo Lo' = M for a symmetric positive SEMI-definite M (its lower triangle is read).  A pivot at or
// below 1e-13 x the largest diagonal entry leaves its column zero: the matrix is (numerically) rank-deficient there, and the
// square root of a rounding-negative pivot is never taken.  Returns false if a pivot is below -1e-13 x that entry: M is
// indefinite, Lo is not its factor.
template <int D> __device__ bool chol_psd(const double* M, double* Lo) {
    double dmax = 0.0;
    for (int i = 0; i < D; ++i) dmax = fmax(dmax, M[i * D + i]);
    const double tiny = 1e-13 * dmax;
    bool psd = true;
    zero<D * D>(Lo);
    for (int j = 0; j < D; ++j) {
        double s = M[j * D + j];
        for (int k = 0; k < j; ++k) s -= Lo[j * D + k] * Lo[j * D + k];
        if (!(s > tiny)) { psd = psd && s >= -tiny; continue; }
        const double r = sqrt(s);
        Lo[j * D + j] = r;
        for (int i = j + 1; i < D; ++i) {
            double t = M[i * D + j];
            for (int k = 0; k < j; ++k) t -= Lo[i * D + k] * Lo[j * D + k];
            Lo[i * D + j] = t / r;
        }
    }
    return psd;
}

// The nearest positive semi-definite matrix (Frobenius norm) to a symmetric M: its negative eigenvalues set to zero.
// Cyclic Jacobi rotations (Numerical Recipes' convention A <- P' A P).
template <int D> __device__ void psd_part(const double* M, double* out) {
    double A[D * D], V[D * D];
    symmetrize<D>(M, A);
    eye<D>(V);
    for (int sweep = 0; sweep < 20; ++sweep) {
        double off = 0.0, nrm = 0.0;
        for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) { nrm += A[i * D + j] * A[i * D + j]; if (i != j) off += A[i * D + j] * A[i * D + j]; }
        if (off <= 1e-32 * nrm) break;
        for (int p = 0; p < D - 1; ++p)
            for (int q = p + 1; q < D; ++q) {
                if (A[p * D + q] == 0.0) continue;
                const double theta = (A[q * D + q] - A[p * D + p]) / (2.0 * A[p * D + q]);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < D; ++k) {
                    const double kp = A[k * D + p], kq = A[k * D + q];
                    A[k * D + p] = c * kp - s * kq; A[k * D + q] = s * kp + c * kq;
                }
                for (int k = 0; k < D; ++k) {
                    const double pk = A[p * D + k], qk = A[q * D + k];
                    A[p * D + k] = c * pk - s * qk; A[q * D + k] = s * pk + c * qk;
                }
                for (int k = 0; k < D; ++k) {
                    const double kp = V[k * D + p], kq = V[k * D + q];
                    V[k * D + p] = c * kp - s * kq; V[k * D + q] = s * kp + c * kq;
                }
            }
    }
    for (int i = 0; i < D; ++i)
        for (int j = 0; j < D; ++j) {
            double a = 0.0;
            for (int k = 0; k < D; ++k) a += V[i * D + k] * fmax(A[k * D + k], 0.0) * V[j * D + k];
            out[i * D + j] = a;
        }
}

// the sampler's factor of a covariance: Cholesky where M is positive semi-definite, else of M's positive semi-definite part
template <int D> __device__ void sampling_factor(const double* M, double* Lo) {
    if (chol_psd<D>(M, Lo)) return;
    double P[D * D];
    psd_part<D>(M, P);
    chol_psd<D>(P, Lo);
}

template <int D> __device__ void power_table(const double* M, double (*tab)[9]) {
    double P[D * D];
    cpy<D * D>(M, P);
    for (int k = 0; k < NPOW; ++k) {
        store_mat<D>(P, tab[k]);
        mm<D, D, D>(P, P, P);
    }
}

// One CTA per latent, SIX warps, lane 0 of each doing one of the independent jobs (different code paths in different warps
// run concurrently; as lanes of one warp they would be serialised):
//   phase A   warp 0: state space, A = expm(dt F), Q, the literal DARE, gains             (ihgp.h:120-133)
//             warp 1: the 2d x 2d block exponential behind dA of the lengthscale (:163-167) - needs only F, dF, dt
//   phase B   warps 0..2: one hyper-parameter each (QLyap, literal DLyap, dS, dK, dAKHA, HdA)   (:136-200)
//             warp 3: literal smoother constants + G^(2^k) table, warp 4: rts_correct ones + table, warp 5: AKHA^(2^k) table
// Every quantity is computed by the same instruction sequence as before: results are bit-identical, only the schedule changed.
template <int D>
__global__ void __launch_bounds__(192) k_setup(const double* __restrict__ igp_params /*[L][3]*/, double dt, int L,
                                              LatentConsts* __restrict__ out) {
    constexpr int DD = D * D;
    __shared__ WarpScratch<D> w;
    __shared__ double dA_len[DD];                  // dA of the lengthscale, from warp 1's block exponential
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int l = blockIdx.x;
    LatentConsts& o = out[l];
    const double* prm = igp_params + 3 * l;

    if (warp == 1 && lane == 0) {
        StateSpace<D> ss1;                          // the same state space as warp 0 builds (deterministic), privately
        state_space(ss1, prm[0], prm[1], prm[2]);
        if (!all_zero<DD>(ss1.dF1)) {
            constexpr int E = 2 * D;
            double FF[E * E], EX[E * E];
            for (int i = 0; i < E * E; ++i) FF[i] = 0.0;
            for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) {     // ihgp.h:163-166
                FF[i * E + j] = ss1.F[i * D + j] * dt;
                FF[(D + i) * E + D + j] = ss1.F[i * D + j] * dt;
                FF[(D + i) * E + j] = ss1.dF1[i * D + j] * dt;
            }
            expm<E>(FF, EX);                                          // ihgp.h:167
            for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) dA_len[i * D + j] = EX[(D + i) * E + j];
        }
    }
    if (warp == 0 && lane == 0) {
        state_space(w.ss, prm[0], prm[1], prm[2]);
        double tF[DD], t1[DD], t2[DD];
        scl<DD>(w.ss.F, dt, tF);
        expm<D>(tF, w.A);                                             // ihgp.h:120
        double AT[DD];
        tr<D, D>(w.A, AT);
        mm<D, D, D>(w.A, w.ss.Pinf, t1);
        mm<D, D, D>(t1, AT, t2);
        subv<DD>(w.ss.Pinf, t2, t1);                                  // ihgp.h:121
        symmetrize<D>(t1, w.Q);                                       // ihgp.h:122
        int it = 0;
        const bool conv = dare_literal<D>(w.A, w.Q, w.ss.R, w.PP, &it);   // ihgp.h:125
        o.iters[0] = it; o.conv[0] = conv ? 1 : 0;
        w.S = w.PP[0] + w.ss.R;                                       // ihgp.h:126 (H = e0')
        for (int i = 0; i < D; ++i) w.K[i] = w.PP[i * D] / w.S;       // ihgp.h:127
        for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) w.PF[i * D + j] = w.PP[i * D + j] - w.K[i] * w.PP[j];   // ihgp.h:128
        for (int j = 0; j < D; ++j) w.HA[j] = w.A[j];                 // ihgp.h:129
        for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) w.AKHA[i * D + j] = w.A[i * D + j] - w.K[i] * w.HA[j];  // ihgp.h:130
        for (int i = 0; i < D; ++i) { double s = 0.0; for (int k = 0; k < D; ++k) s += w.A[i * D + k] * w.K[k]; w.AK[i] = s; }   // ihgp.h:132
        for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) w.AAKH[i * D + j] = w.A[i * D + j] - (j == 0 ? w.AK[i] : 0.0);   // ihgp.h:133
        store_mat<D>(w.A, o.A); store_mat<D>(w.Q, o.Q); store_mat<D>(w.PP, o.PP); store_mat<D>(w.PF, o.PF);
        store_mat<D>(w.AKHA, o.AKHA); store_vec<D>(w.K, o.K); store_vec<D>(w.HA, o.HA);
        o.S = w.S; o.logS = log(w.S);
        double hak = 0.0;
        for (int j = 0; j < D; ++j) hak += w.HA[j] * w.K[j];
        o.hak = hak;
        double ImA[DD];
        for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) ImA[i * D + j] = (i == j ? 1.0 : 0.0) - w.A[i * D + j];
        store_mat<D>(ImA, o.ImA);
        for (int i = 0; i < 3; ++i) o.params[i] = prm[i];
        o.dim = D;
    }
    __syncthreads();
    if (lane != 0) return;

    if (warp < 3) {
        // ---- one hyper-parameter per warp: ihgp.h:136-200 --------------------------------------
        const int idx = warp;
        double AT[DD], dA[DD], dAT[DD], dQ[DD], QL[DD], t1[DD], t2[DD];
        tr<D, D>(w.A, AT);
        // exact-zero tests of ihgp.h:141,144,152: dF is non-zero only for the lengthscale (idx 1),
        // dPinf for magnitude/lengthscale (idx 0,1), dR only for the noise (idx 2)
        const double* dPinf = idx == 0 ? w.ss.dPinf0 : w.ss.dPinf1;
        const bool dF_zero = (idx != 1) || all_zero<DD>(w.ss.dF1);
        const bool dPinf_zero = (idx == 2) || all_zero<DD>(dPinf);
        const double dR = idx == 2 ? 1.0 : 0.0;
        if (dF_zero) {
            zero<DD>(dA);                                             // :143
            if (dPinf_zero) zero<DD>(dQ);                             // :146
            else { mm<D, D, D>(w.A, dPinf, t1); mm<D, D, D>(t1, AT, t2); subv<DD>(dPinf, t2, dQ); }   // :150
            if (dR == 0.0) cpy<DD>(dQ, QL);                           // :154
            else {
                // :158 is a (d x d)*(1 x 1) product in the reference - undefined behaviour there (Q19).
                // The INTENDED AK dR AK' + dQ (cf. :183) is implemented, as in the oracle.
                for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) QL[i * D + j] = (w.AK[i] * w.AK[j]) * dR + dQ[i * D + j];
            }
        } else {
            cpy<DD>(dA_len, dA);                                      // :163-167, computed by warp 1 in phase A
            tr<D, D>(dA, dAT);                                        // :168
            double a[DD], b[DD], c[DD];
            mm<D, D, D>(dA, w.ss.Pinf, t1); mm<D, D, D>(t1, AT, a);   // dA Pinf A'
            mm<D, D, D>(w.A, w.ss.Pinf, t1); mm<D, D, D>(t1, dAT, c); // A Pinf dA'
            if (dPinf_zero) { for (int i = 0; i < DD; ++i) dQ[i] = -a[i] - c[i]; }                 // :171
            else { mm<D, D, D>(w.A, dPinf, t1); mm<D, D, D>(t1, AT, b); for (int i = 0; i < DD; ++i) dQ[i] = ((dPinf[i] - a[i]) - b[i]) - c[i]; }   // :175
            // :179 / :183
            double q1[DD], q2[DD], q3[DD], q4[DD], dAPP[DD], PPdAT[DD];
            mm<D, D, D>(dA, w.PP, dAPP); mm<D, D, D>(dAPP, AT, q1);   // dA PP A'
            mm<D, D, D>(w.A, w.PP, t1); mm<D, D, D>(t1, dAT, q2);     // A PP dA'
            for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) q3[i * D + j] = dAPP[i * D] * w.AK[j];   // dA PP H' AK'
            mm<D, D, D>(w.PP, dAT, PPdAT);
            for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) q4[i * D + j] = w.AK[i] * PPdAT[j];      // AK H PP dA'
            for (int i = 0; i < DD; ++i) QL[i] = ((q1[i] + q2[i]) - q3[i]) - q4[i];
            if (dR != 0.0) for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) QL[i * D + j] += (w.AK[i] * dR) * w.AK[j];
            for (int i = 0; i < DD; ++i) QL[i] += dQ[i];
        }
        double dPP[DD];
        int it = 0;
        const bool conv = dlyap_literal<D>(w.AAKH, QL, dPP, &it);     // :187
        o.iters[1 + idx] = it; o.conv[1 + idx] = conv ? 1 : 0;
        const double dS = dPP[0] + dR;                                // :188
        double dK[D], dAKHA[DD], HdA[D];
        for (int i = 0; i < D; ++i) dK[i] = (dPP[i * D] - w.PP[i * D] * dS / w.S) / w.S;   // :189
        if (dF_zero) {
            for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) dAKHA[i * D + j] = (-dK[i]) * w.A[j];   // :192
            zero<D>(HdA);                                             // :193
        } else {
            for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) dAKHA[i * D + j] = (dA[i * D + j] - dK[i] * w.A[j]) - w.K[i] * dA[j];   // :197
            for (int j = 0; j < D; ++j) HdA[j] = dA[j];               // :198
        }
        o.dS[idx] = dS;
        store_mat<D>(dA, o.dA[idx]); store_mat<D>(dAKHA, o.dAKHA[idx]);
        store_vec<D>(dK, o.dK[idx]); store_vec<D>(HdA, o.HdA[idx]);
    } else if (warp == 3) {
        // ---- reference_literal smoother constants: ihgp.h:105-107 (Q3) ---------------------------
        double PPs[DD], t1[DD], APF[DD], sym[DD], X[DD], G[DD], C[DD], P[DD];
        mm<D, D, D>(w.A, w.PF, APF);
        mm<D, D, D>(APF, w.A, t1);                                    // A*PF*A  (sic: no transpose)
        addv<DD>(t1, w.Q, PPs);                                       // :105
        // PP.ldlt() reads only the lower triangle of the (non-symmetric) PPs
        for (int j = 0; j < D; ++j) for (int i = j; i < D; ++i) { sym[i * D + j] = PPs[i * D + j]; sym[j * D + i] = PPs[i * D + j]; }
        double rhs[DD];
        cpy<DD>(APF, rhs);
        solve_lu<D, D>(sym, rhs, X);
        tr<D, D>(X, G);                                               // :106
        double GT[DD];
        tr<D, D>(G, GT);
        mm<D, D, D>(G, PPs, t1); mm<D, D, D>(t1, GT, C);
        subv<DD>(w.PF, C, C);
        int it = 0;
        dlyap_literal<D>(G, C, P, &it);                               // :107
        o.smooth_iters = it;
        store_mat<D>(G, o.G[0]); store_mat<D>(P, o.Ps[0]);
        power_table<D>(G, o.powG[0]);               // G^(2^k) for the chunked scans
    } else if (warp == 4) {
        // ---- rts_correct smoother constants (OUR extension, SURVEY section 11 item 5) -------------
        //   PPc = A PF A' + Q,  G = PF A' PPc^-1,  P_s = G P_s G' + PF - G PPc G'  (exact solve)
        double AT[DD], t1[DD], PPc[DD], PFAT[DD], G[DD], C[DD];
        tr<D, D>(w.A, AT);
        mm<D, D, D>(w.A, w.PF, t1); mm<D, D, D>(t1, AT, PPc);
        addv<DD>(PPc, w.Q, PPc);
        mm<D, D, D>(w.PF, AT, PFAT);
        double lhs[DD], rhs[DD], X[DD];
        tr<D, D>(PPc, lhs); tr<D, D>(PFAT, rhs);
        solve_lu<D, D>(lhs, rhs, X);                                  // PPc' G' = (PF A')'
        tr<D, D>(X, G);
        double GT[DD];
        tr<D, D>(G, GT);
        mm<D, D, D>(G, PPc, t1); mm<D, D, D>(t1, GT, C);
        subv<DD>(w.PF, C, C);
        // vec(P) = (I - G (x) G)^-1 vec(C)
        constexpr int N2 = DD;
        double Mx[N2 * N2], rv[N2], pv[N2];
        for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) {
            const int row = i * D + j;
            rv[row] = C[row];
            for (int k = 0; k < D; ++k) for (int m = 0; m < D; ++m)
                Mx[row * N2 + (k * D + m)] = (row == k * D + m ? 1.0 : 0.0) - G[i * D + k] * G[j * D + m];
        }
        solve_lu<N2, 1>(Mx, rv, pv);
        double GK[D];
        for (int i = 0; i < D; ++i) { double s = 0.0; for (int k = 0; k < D; ++k) s += G[i * D + k] * w.K[k]; GK[i] = s; }
        double GA[DD], Bs[DD];
        mm<D, D, D>(G, w.A, GA);
        for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) Bs[i * D + j] = (i == j ? 1.0 : 0.0) - GA[i * D + j];
        store_mat<D>(G, o.G[1]); store_mat<D>(pv, o.Ps[1]); store_vec<D>(GK, o.GK); store_mat<D>(Bs, o.Bs);
        double LF[DD], LC[DD];                      // posterior sampling: x[T-1] ~ N(., PF), x[t] | x[t+1] ~ N(., C)
        sampling_factor<D>(w.PF, LF);
        sampling_factor<D>(C, LC);
        store_mat<D>(LF, o.LF); store_mat<D>(LC, o.LC);
        power_table<D>(G, o.powG[1]);
    } else if (warp == 5) {
        power_table<D>(w.AKHA, o.powM);             // AKHA^(2^k) for the chunked scans
    }
}

}  // namespace

cudaError_t launch_setup(int dim, const double* d_igp_params, double dt, int L, LatentConsts* d_out, cudaStream_t stream) {
    if (dim == 2) k_setup<2><<<L, 192, 0, stream>>>(d_igp_params, dt, L, d_out);
    else k_setup<3><<<L, 192, 0, stream>>>(d_igp_params, dt, L, d_out);
    return cudaGetLastError();
}

}  // namespace moihgp
