// One observation per call: the kernels behind the legacy gp32_* / gp52_* entry points (sm_100a).
//
// Replaces (reference, /root/reference/moihgp/include/moihgp):
//   moihgp.h:148-428   the four MOIHGP::step overloads, incl. the missing-data (NaN) least-squares
//                      projection  Ty = S^-1/2 (U0'U0)^-1 U0' y_obs  (:167-178)
//   moihgp.h:460-688   the two MOIHGP::negLogLikelihood overloads
//   ihgp.h:37-100, :204-222   the per-latent step / NLL they call
// These are latency-bound by construction (one tiny launch per observation); the whole-sequence
// kernels (project.cu / scan.cu / objective.cu) are the throughput path.  One CTA does the call.
#include <cuda_runtime.h>
#include <math.h>
#include "moihgp_device.cuh"
#include "launch.h"
#include "ls_project.cuh"

namespace moihgp {

namespace {

constexpr int ST = 128;

// Ty for one observation.  Ty[L] (out) in shared memory, sc[ls_scratch_doubles(L)] in shared memory or, where the kernel's
// shared memory with it would pass 227 KB (k_step: L >= 120, k_lik: L >= 118), in global memory (StepArgs / LikArgs::ls_scratch).
// Full observation: Ty = (S^-1/2 U') y (moihgp.h:181).  With NaNs: the least-squares projection on the observed rows
// (ls_project.cuh), over the CTA.
__device__ void project_one(const double* __restrict__ U, const double* __restrict__ S, const double* __restrict__ y, int p, int L,
                            double* Ty, double* sc, int* s_nmiss) {
    const int tid = threadIdx.x;
    if (tid == 0) *s_nmiss = 0;
    __syncthreads();
    int miss = 0;
    for (int r = tid; r < p; r += ST) miss += isnan(y[r]) ? 1 : 0;
    if (miss) atomicAdd(s_nmiss, miss);
    __syncthreads();
    if (*s_nmiss == 0) {
        for (int l = tid; l < L; l += ST) {
            const double si = 1 / sqrt(S[l]);
            double s = 0.0;
            for (int r = 0; r < p; ++r) s += (si * U[(size_t)r * L + l]) * y[r];
            Ty[l] = s;
        }
        __syncthreads();
        return;
    }
    double* v = sc + 2 * L * L + L;
    ls_solve_coop(p, L, [&](int r) { return y[r]; }, [&](int r, int l) { return U[(size_t)r * L + l]; },
                  sc, sc + L * L, sc + 2 * L * L, v, reinterpret_cast<int*>(sc + 2 * L * L + 2 * L), tid, ST, [] { __syncthreads(); });
    for (int l = tid; l < L; l += ST) Ty[l] = (1 / sqrt(S[l])) * v[l];
    __syncthreads();
}

__global__ void __launch_bounds__(ST) k_step(StepArgs a) {
    extern __shared__ double sm[];
    const int L = a.L, p = a.p, d = a.dim, tid = threadIdx.x;
    double* Ty = sm;                 // [L]
    double* Tyhat = Ty + L;          // [L]
    double* sc = a.ls_scratch ? a.ls_scratch : Tyhat + L;                   // [ls_scratch_doubles(L)]
    int* s_nmiss = (int*)(Tyhat + L + (a.ls_scratch ? 0 : ls_scratch_doubles(L)));
    if (a.y) project_one(a.U, a.S, a.y, p, L, Ty, sc, s_nmiss);
    for (int l = tid; l < L; l += ST) {
        const LatentConsts& c = a.consts[l];
        const double* x = a.x + (size_t)l * d;
        double* xn = a.xnew + (size_t)l * d;
        const bool predict = a.y == nullptr || isnan(Ty[l]);                // ihgp.h:96-100 / :39
        const double yy = predict ? 0.0 : Ty[l];
        const double* M = predict ? c.A : c.AKHA;
        for (int i = 0; i < d; ++i) {
            double s = 0.0;
            for (int j = 0; j < d; ++j) s += M[i * 3 + j] * x[j];
            xn[i] = predict ? s : s + c.K[i] * yy;                          // ihgp.h:41 / :50
        }
        Tyhat[l] = xn[0];                                                   // ihgp.h:42 / :51
        if (a.dx && a.dxnew) {
            for (int k = 0; k < 3; ++k) {
                const double* dM = predict ? c.dA[k] : c.dAKHA[k];
                const double* dxk = a.dx + ((size_t)l * 3 + k) * d;
                double* dxn = a.dxnew + ((size_t)l * 3 + k) * d;
                for (int i = 0; i < d; ++i) {
                    double s1 = 0.0, s2 = 0.0;
                    for (int j = 0; j < d; ++j) { s1 += dM[i * 3 + j] * x[j]; s2 += M[i * 3 + j] * dxk[j]; }
                    dxn[i] = predict ? s1 + s2 : s1 + s2 + c.dK[k][i] * yy; // ihgp.h:45 / :54
                }
            }
        }
    }
    __syncthreads();
    if (a.yhat) {
        for (int r = tid; r < p; r += ST) {                                 // moihgp.h:222-225
            double s = 0.0;
            for (int l = 0; l < L; ++l) s += (a.U[(size_t)r * L + l] * sqrt(a.S[l])) * Tyhat[l];
            a.yhat[r] = s;
        }
    }
}

__global__ void __launch_bounds__(ST) k_lik(LikArgs a) {
    extern __shared__ double sm[];
    const int L = a.L, p = a.p, d = a.dim, tid = threadIdx.x;
    double* Ty = sm;                 // [L]
    double* w = Ty + L;              // [L]   U'y
    double* pv = w + L;              // [L]
    double* li = pv + L;             // [L]   per-latent loss
    double* gi = li + L;             // [3L]  per-latent grads
    double* red = gi + 3 * L;        // [ST]
    double* sc = a.ls_scratch ? a.ls_scratch : red + ST;                    // [ls_scratch_doubles(L)]
    int* s_nmiss = (int*)(red + ST + (a.ls_scratch ? 0 : ls_scratch_doubles(L)));
    project_one(a.U, a.S, a.y, p, L, Ty, sc, s_nmiss);
    for (int l = tid; l < L; l += ST) {
        double s = 0.0;
        for (int r = 0; r < p; ++r) s += a.U[(size_t)r * L + l] * a.y[r];
        w[l] = s;
    }
    __syncthreads();
    double q = 0.0;
    for (int r = tid; r < p; r += ST) {                                     // moihgp.h:501 / :651
        double e = a.y[r];
        for (int l = 0; l < L; ++l) e -= a.U[(size_t)r * L + l] * w[l];
        q += e * e;
    }
    red[tid] = q;
    __syncthreads();
    for (int o = ST / 2; o > 0; o >>= 1) { if (tid < o) red[tid] += red[tid + o]; __syncthreads(); }
    const double yu = sqrt(red[0]);
    for (int l = tid; l < L; l += ST) {
        const LatentConsts& c = a.consts[l];
        const double* x = a.x + (size_t)l * d;
        double hax = 0.0;
        for (int j = 0; j < d; ++j) hax += c.HA[j] * x[j];
        const double v = Ty[l] - hax;                                       // ihgp.h:206 / :214
        li[l] = 0.5 * (v * v / c.S + log(c.S));                             // ihgp.h:207 / :215
        if (a.dx) {
            pv[l] = (a.y[l] - hax) * (1 - c.hak) / c.S;                     // moihgp.h:510-511 (raw y(l), Q8)
            for (int k = 0; k < 3; ++k) {
                const double* dxk = a.dx + ((size_t)l * 3 + k) * d;
                double hd = 0.0;
                for (int j = 0; j < d; ++j) hd += c.HA[j] * dxk[j];
                const double dv = -c.HdA[k][0] * x[0] - hd;                 // ihgp.h:218 (Q20 de facto)
                gi[3 * l + k] = (v * dv - 0.5 * (v * v / c.S - 1) * c.dS[k]) / c.S;   // ihgp.h:219
            }
        }
    }
    __syncthreads();
    const int sizeU = p * L;
    if (a.dx && a.grad) {
        for (int i = tid; i < sizeU; i += ST) {                             // moihgp.h:538-552 in its rank-1 form
            const int r = i / L, c = i - r * L;
            a.grad[i] = a.y[r] * (-w[c] / a.sigma + pv[c] * (1 / sqrt(a.S[c])));
        }
    }
    if (tid == 0) {
        const double m_n = fmax((double)(p - L), 0.0);                      // moihgp.h:502
        double loss = nll_step_const(a.S, p, L, a.sigma) + 0.5 * yu / a.sigma;   // moihgp.h:503
        if (a.dx && a.grad) {
            double gsig = 0.5 * (m_n - yu / a.sigma) / a.sigma;             // moihgp.h:563
            for (int l = 0; l < L; ++l) {
                const double Sl = a.S[l], rs = sqrt(Sl);
                double gS = 0.5 / Sl + pv[l] * (-0.5 * (1 / rs / rs / rs) * w[l]);   // moihgp.h:555-561
                if (a.threading) loss += li[l];                             // moihgp.h:588 vs :601 (Q5)
                const double dn = gi[3 * l + 2];
                gS -= dn * a.sigma / Sl / Sl;                               // moihgp.h:591 / :604
                gsig += dn / Sl;                                            // moihgp.h:592 / :605
                a.grad[sizeU + l] = gS;
                for (int k = 0; k < 3; ++k) a.grad[sizeU + L + 1 + 3 * l + k] = gi[3 * l + k];   // moihgp.h:608-609
            }
            a.grad[sizeU + L] = gsig;
        } else {
            for (int l = 0; l < L; ++l) loss += li[l];                      // moihgp.h:675 / :684 (always)
        }
        *a.loss = loss;
    }
}

// IHGP::backwardSmoother (ihgp.h:108-113) over caller-supplied filtered states X[N][T][L][d] (any X, not necessarily the
// output of this library's filter): one thread per (sequence, latent) chain walks backwards in time.  The generic,
// shape-independent form behind moihgp_cuda_smooth; the fused passes use k_smooth_chain / k_scan_lanes instead.
//   mode 0 (reference, literal): Xs[T-1] = X[T-1],  Xs[j] = X[j+1] + G Xs[j+1] - A X[j+1]
//   mode 1 (RTS):                Xs[T-1] = X[T-1],  Xs[j] = X[j] + G (Xs[j+1] - A X[j])
__global__ void __launch_bounds__(128) k_smooth_seq(const double* __restrict__ X, const LatentConsts* __restrict__ consts, int L, int d,
                                                   long long N, long long T, int mode, double* __restrict__ Xs) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * L) return;
    const long long n = i / L;
    const int l = (int)(i - n * L);
    const LatentConsts& c = consts[l];
    const size_t stride = (size_t)L * d;
    const double* x = X + ((size_t)n * T * L + l) * d;
    double* xs = Xs + ((size_t)n * T * L + l) * d;
    double s[DMAX], nx[DMAX];
    for (int a = 0; a < d; ++a) { s[a] = x[(size_t)(T - 1) * stride + a]; nx[a] = s[a]; xs[(size_t)(T - 1) * stride + a] = s[a]; }
    for (long long j = T - 2; j >= 0; --j) {
        double cur[DMAX], out[DMAX];
        for (int a = 0; a < d; ++a) cur[a] = x[(size_t)j * stride + a];
        const double* drive = mode == 0 ? nx : cur;          // the literal form is driven by X[j+1] (Q3), RTS by X[j]
        const double* B = mode == 0 ? c.ImA : c.Bs;          // I - A  /  I - G A
        for (int a = 0; a < d; ++a) {
            double acc = c.G[mode][a * 3] * s[0];
            for (int b = 1; b < d; ++b) acc = fma(c.G[mode][a * 3 + b], s[b], acc);
            for (int b = 0; b < d; ++b) acc = fma(B[a * 3 + b], drive[b], acc);
            out[a] = acc;
        }
        for (int a = 0; a < d; ++a) { s[a] = out[a]; nx[a] = cur[a]; xs[(size_t)j * stride + a] = out[a]; }
    }
}

size_t step_smem(int L, bool global_scratch) {
    return sizeof(double) * (2 * (size_t)L + (global_scratch ? 0 : ls_scratch_doubles(L))) + sizeof(int);
}
size_t lik_smem(int L, bool global_scratch) {
    return sizeof(double) * (7 * (size_t)L + ST + (global_scratch ? 0 : ls_scratch_doubles(L))) + sizeof(int);
}
constexpr size_t SMEM_MAX = 227 * 1024;     // dynamic shared memory of one CTA

}  // namespace

size_t step_global_doubles(int L) { return step_smem(L, false) <= SMEM_MAX ? 0 : (size_t)ls_scratch_doubles(L); }
size_t lik_global_doubles(int L) { return lik_smem(L, false) <= SMEM_MAX ? 0 : (size_t)ls_scratch_doubles(L); }

cudaError_t launch_step(const StepArgs& a, cudaStream_t st) {
    if ((step_global_doubles(a.L) != 0) != (a.ls_scratch != nullptr)) return cudaErrorInvalidValue;
    const size_t smem = step_smem(a.L, a.ls_scratch != nullptr);
    if (smem > 48 * 1024) cudaFuncSetAttribute(k_step, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    k_step<<<1, ST, smem, st>>>(a);
    return cudaGetLastError();
}

// OnlineObjective::push_back (moihgp_online.h:75-93) on the device-resident window: append y, recompute the moving mean over
// every element held (the one about to be dropped included, as the reference does), drop the oldest element when the window
// is over-full, and leave the NEW front element minus the mean in front_centred (the observation the carried state is then
// advanced with, SURVEY Q12).  win holds the window oldest-first, contiguously.  count[0] = elements held, count[1] = 1 if
// an element was dropped by this push.
__global__ void __launch_bounds__(128) k_online_push(const double* __restrict__ y_new, const double* __restrict__ ma_given, int p, int W,
                                                    double* __restrict__ win, int* __restrict__ count, double* __restrict__ ma,
                                                    double* __restrict__ front_centred) {
    const int tid = threadIdx.x;
    const int n = count[0] + 1;                                  // after the push_back (:77)
    for (int r = tid; r < p; r += 128) {
        win[(size_t)(n - 1) * p + r] = y_new[r];
        if (ma_given) { ma[r] = ma_given[r]; continue; }         // the caller's own centre (online_learning.py:54-64: an EMA)
        double s = 0.0;
        for (int k = 0; k < n; ++k) s += win[(size_t)k * p + r];  // ma += *it, oldest first (:79-82)
        ma[r] = s / double(n);                                   // :83
    }
    __syncthreads();
    const bool drop = n > W;                                     // :84 (at most one element per push: n <= W + 1)
    if (drop) {
        for (int r = tid; r < p; r += 128) {
            for (int k = 0; k + 1 < n; ++k) win[(size_t)k * p + r] = win[(size_t)(k + 1) * p + r];   // pop_front (:88)
            front_centred[r] = win[r] - ma[r];                   // Y.front() - ma (:89), after the pop
        }
    }
    __syncthreads();
    if (tid == 0) { count[0] = drop ? n - 1 : n; count[1] = drop ? 1 : 0; }
}

// Proximal term of OnlineObjective::operator() (moihgp_online.h:42-54) added to the window objective:
//   dparams = params - oldparams,  Bp = B dparams (B = null: the identity, :50-53),  loss += 1/2 dparams' Bp,  grad += Bp;
// also appends the model's polar factor U to the output block so that ONE device-to-host copy refreshes the host mirror.
__global__ void __launch_bounds__(256) k_online_prox(const double* __restrict__ params, const double* __restrict__ oldparams,
                                                    const double* __restrict__ B, int np, int pL, const double* __restrict__ U,
                                                    double* __restrict__ out) {
    __shared__ double red[256];
    const int tid = threadIdx.x;
    double part = 0.0;
    for (int i = tid; oldparams && i < np; i += 256) {           // oldparams = null: no proximal term (the caller adds its own)
        double bp;
        if (B) {
            bp = 0.0;
            for (int j = 0; j < np; ++j) bp += B[(size_t)i * np + j] * (params[j] - oldparams[j]);
        } else bp = params[i] - oldparams[i];
        part += (params[i] - oldparams[i]) * bp;
        out[2 + i] += bp;
    }
    for (int i = tid; i < pL; i += 256) out[2 + np + i] = U[i];
    red[tid] = part;
    __syncthreads();
    if (tid == 0) {
        double s = 0.0;
        for (int i = 0; i < 256; ++i) s += red[i];                // fixed order
        out[0] += 0.5 * s;
    }
}

// F[i] = X[i][0]: the function-value component H x of every state (H = e0', matern32ss.h:22)
__global__ void __launch_bounds__(256) k_extract_values(const double* __restrict__ X, double* __restrict__ F, long long n, int d) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) F[i] = X[i * d];
}
cudaError_t launch_extract_values(const double* X, double* F, long long n, int d, cudaStream_t st) {
    const long long blocks = (n + 255) / 256;
    k_extract_values<<<(unsigned)(blocks < 148 * 16 ? (blocks < 1 ? 1 : blocks) : 148 * 16), 256, 0, st>>>(X, F, n, d);
    return cudaGetLastError();
}

cudaError_t launch_online_push(const double* y_new, const double* ma_given, int p, int W, double* win, int* count, double* ma,
                               double* front_centred, cudaStream_t st) {
    k_online_push<<<1, 128, 0, st>>>(y_new, ma_given, p, W, win, count, ma, front_centred);
    return cudaGetLastError();
}

cudaError_t launch_online_prox(const double* params, const double* oldparams, const double* B, int np, int pL, const double* U, double* out,
                               cudaStream_t st) {
    k_online_prox<<<1, 256, 0, st>>>(params, oldparams, B, np, pL, U, out);
    return cudaGetLastError();
}

cudaError_t launch_smooth_seq(const double* X, const LatentConsts* consts, int L, int d, long long N, long long T, int mode, double* Xs,
                              cudaStream_t st) {
    const long long chains = N * L;
    k_smooth_seq<<<(unsigned)((chains + 127) / 128), 128, 0, st>>>(X, consts, L, d, N, T, mode, Xs);
    return cudaGetLastError();
}

cudaError_t launch_lik(const LikArgs& a, cudaStream_t st) {
    if ((lik_global_doubles(a.L) != 0) != (a.ls_scratch != nullptr)) return cudaErrorInvalidValue;
    const size_t smem = lik_smem(a.L, a.ls_scratch != nullptr);
    if (smem > 48 * 1024) cudaFuncSetAttribute(k_lik, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    k_lik<<<1, ST, smem, st>>>(a);
    return cudaGetLastError();
}

}  // namespace moihgp
