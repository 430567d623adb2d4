// d x d (d = 2, 3) matrix helpers shared by the scan and objective kernels and the host entry points.  Matrices in
// LatentConsts are row-major with a fixed row stride of 3 (moihgp_device.cuh); in registers they are packed d x d.
#pragma once
#include "moihgp_device.cuh"

// `#pragma unroll` in __host__ __device__ code: the host compiler does not know the pragma
#ifdef __CUDA_ARCH__
#define HD_UNROLL _Pragma("unroll")
#else
#define HD_UNROLL
#endif

namespace moihgp {

template <int D> __device__ __forceinline__ void load_mat(const double* src9, double* dst) {
#pragma unroll
    for (int i = 0; i < D; ++i)
#pragma unroll
        for (int j = 0; j < D; ++j) dst[i * D + j] = __ldg(src9 + i * 3 + j);
}
template <int D> __device__ __forceinline__ void load_vec(const double* src3, double* dst) {
#pragma unroll
    for (int i = 0; i < D; ++i) dst[i] = __ldg(src3 + i);
}
template <int D> __device__ __forceinline__ void mv(const double* M, const double* x, double* y) {  // y = M x
#pragma unroll
    for (int i = 0; i < D; ++i) {
        double s = M[i * D] * x[0];
#pragma unroll
        for (int j = 1; j < D; ++j) s = fma(M[i * D + j], x[j], s);
        y[i] = s;
    }
}
template <int D> __device__ __forceinline__ void mv_acc(const double* M, const double* x, double* y) {  // y += M x
#pragma unroll
    for (int i = 0; i < D; ++i) {
        double s = y[i];
#pragma unroll
        for (int j = 0; j < D; ++j) s = fma(M[i * D + j], x[j], s);
        y[i] = s;
    }
}

// C = A B (C distinct; A with row stride SA, B and C packed)
template <int D, int SA = D> __host__ __device__ __forceinline__ void mat_mul(const double* A, const double* B, double* C) {
    HD_UNROLL
    for (int i = 0; i < D; ++i)
        HD_UNROLL
        for (int j = 0; j < D; ++j) {
            double s = 0.0;
            HD_UNROLL
            for (int q = 0; q < D; ++q) s += A[i * SA + q] * B[q * D + j];
            C[i * D + j] = s;
        }
}

// P = M^n by binary powering on the table tab[k] = M^(2^k) (row stride 3): the bits of n from the least significant,
// P <- tab[j] P for each set bit j.  All powers of one matrix commute, so the order of the factors is free.
template <int D> __host__ __device__ __forceinline__ void mat_pow(const double (*tab)[9], unsigned long long n, double* P) {
    HD_UNROLL
    for (int i = 0; i < D * D; ++i) P[i] = (i / D == i % D) ? 1.0 : 0.0;
    for (int j = 0; (n >> j) != 0 && j < NPOW; ++j) {
        if (!((n >> j) & 1)) continue;
        double t[D * D];
        mat_mul<D, 3>(tab[j], P, t);
        HD_UNROLL
        for (int i = 0; i < D * D; ++i) P[i] = t[i];
    }
}

// The transition of the objective's state [x; dx_0; dx_1; dx_2] over n steps: x -> P x, dx_k -> P dx_k + E_k x with
// P = M^n, E_k(n) = sum_i M^(n-1-i) dM_k M^i (ihgp.h:71-77 unrolled), M = AKHA, dM_k = dAKHA[k].  The bits of n from the
// least significant: (Pb, Eb) = T(2^j) by doubling, (P, E) = T(bits seen so far); appending a span b after a span a:
// P <- Pb P,  E_k <- Pb E_k + Eb_k P.
template <int D>
__host__ __device__ __forceinline__ void block_transition(const LatentConsts& c, unsigned long long n, double* P, double (*E)[D * D]) {
    double Pb[D * D], Eb[3][D * D], t1[D * D], t2[D * D];
    HD_UNROLL
    for (int i = 0; i < D * D; ++i) P[i] = (i / D == i % D) ? 1.0 : 0.0;
    HD_UNROLL
    for (int k = 0; k < 3; ++k)
        HD_UNROLL
        for (int i = 0; i < D; ++i)
            HD_UNROLL
            for (int j = 0; j < D; ++j) { E[k][i * D + j] = 0.0; Eb[k][i * D + j] = c.dAKHA[k][i * 3 + j]; }
    for (int j = 0; (n >> j) != 0 && j < NPOW; ++j) {
        HD_UNROLL
        for (int i = 0; i < D; ++i)
            HD_UNROLL
            for (int q = 0; q < D; ++q) Pb[i * D + q] = c.powM[j][i * 3 + q];
        if ((n >> j) & 1) {
            HD_UNROLL
            for (int k = 0; k < 3; ++k) {
                mat_mul<D>(Pb, E[k], t1);
                mat_mul<D>(Eb[k], P, t2);
                HD_UNROLL
                for (int i = 0; i < D * D; ++i) E[k][i] = t1[i] + t2[i];
            }
            mat_mul<D>(Pb, P, t1);
            HD_UNROLL
            for (int i = 0; i < D * D; ++i) P[i] = t1[i];
        }
        HD_UNROLL
        for (int k = 0; k < 3; ++k) {                               // E(2b) = E(b) M^b + M^b E(b)
            mat_mul<D>(Eb[k], Pb, t1);
            mat_mul<D>(Pb, Eb[k], t2);
            HD_UNROLL
            for (int i = 0; i < D * D; ++i) Eb[k][i] = t1[i] + t2[i];
        }
    }
}

}  // namespace moihgp
