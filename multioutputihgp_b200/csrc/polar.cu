// K-polar: the polar factor U = W V' of the p x L block of the parameter vector, on the device (sm_100a).
//
// Replaces MOIHGP::update's  U = svd.matrixU() * svd.matrixV().transpose()  (moihgp.h:431-447; JacobiSVD / BDCSVD) for
// large p*L, where the host Jacobi costs milliseconds per objective evaluation (SURVEY.md 8 f4).  One-sided Jacobi on
// A V = W diag(s): columns live contiguously in shared memory (Wt[j][r], Vt[j][r]); each sweep is a round-robin
// tournament of Lp - 1 rounds with Lp / 2 disjoint column pairs, one warp per pair per round.  The polar factor is
// unique, so the rotation order only moves the result by rounding (~1e-16).
// k_polar_ns (below) gets the same factor by the Newton-Schulz iteration and runs first; the Jacobi kernel is its fallback.
#include <cuda_runtime.h>
#include <math.h>
#include <algorithm>
#include "launch.h"
#include "ptx.cuh"

namespace moihgp {

namespace {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// one CTA; dynamic shared memory: Wt[Lp][p], Vt[Lp][Lp], norms[Lp]
__global__ void __launch_bounds__(1024) k_polar(const double* __restrict__ A /*[p][L] row-major*/, int p, int L, double* __restrict__ U,
                                               const int* __restrict__ status) {
    if (status && status[0] == 0) return;          // k_polar_ns has already produced U
    extern __shared__ double sm[];
    __shared__ double off_max;
    const int Lp = (L + 1) & ~1;
    double* Wt = sm;
    double* Vt = Wt + (size_t)Lp * p;
    double* nrm = Vt + (size_t)Lp * Lp;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    for (int i = tid; i < Lp * p; i += blockDim.x) {
        const int c = i / p, r = i - c * p;
        Wt[i] = c < L ? A[(size_t)r * L + c] : 0.0;
    }
    for (int i = tid; i < Lp * Lp; i += blockDim.x) Vt[i] = (i / Lp) == (i % Lp) ? 1.0 : 0.0;
    __syncthreads();
    const int n1 = Lp - 1;
    for (int sweep = 0; sweep < 60; ++sweep) {
        if (tid == 0) off_max = 0.0;
        __syncthreads();
        double my_off = 0.0;
        for (int rnd = 0; rnd < n1; ++rnd) {
            for (int pr = warp; pr < Lp / 2; pr += nwarps) {
                int i, j;
                if (pr == 0) { i = n1; j = rnd; }
                else {                                   // (rnd +- pr) mod n1 with 0 <= rnd, pr < n1
                    i = rnd + pr; if (i >= n1) i -= n1;
                    j = rnd - pr; if (j < 0) j += n1;
                }
                if (i > j) { const int t = i; i = j; j = t; }
                double* wi = Wt + (size_t)i * p;
                double* wj = Wt + (size_t)j * p;
                double al = 0.0, be = 0.0, ga = 0.0;
                for (int r = lane; r < p; r += 32) { const double x = wi[r], y = wj[r]; al = fma(x, x, al); be = fma(y, y, be); ga = fma(x, y, ga); }
                al = warp_sum(al); be = warp_sum(be); ga = warp_sum(ga);
                // relative size of the off-diagonal entry, |ga| / sqrt(al be), compared through squares (no sqrt / division on
                // this latency chain): >= 1e-15 keeps the sweeps going, <= 3e-17 is not worth a rotation
                const double g2 = ga * ga, prod = al * be;
                if (g2 > 1e-30 * prod) my_off = 1.0;
                if (g2 > 1e-33 * prod) {
                    // Jacobi angle, |theta| <= pi/4, tan(2 theta) = 2 ga / (be - al), without a division on the chain:
                    // cos(2 theta) = |d| / h, h = hypot(d, 2 ga);  c = sqrt((1 + cos 2theta) / 2);  s = sin(2 theta) / (2 c)
                    const double d = be - al;
                    const double rh = rsqrt(fma(d, d, 4.0 * g2));
                    const double x = fma(0.5 * fabs(d), rh, 0.5);
                    const double ic = rsqrt(x);
                    const double c = x * ic, s = copysign(ga * rh * ic, d * ga);
                    for (int r = lane; r < p; r += 32) { const double x = wi[r], y = wj[r]; wi[r] = c * x - s * y; wj[r] = s * x + c * y; }
                    double* vi = Vt + (size_t)i * Lp;
                    double* vj = Vt + (size_t)j * Lp;
                    for (int r = lane; r < Lp; r += 32) { const double x = vi[r], y = vj[r]; vi[r] = c * x - s * y; vj[r] = s * x + c * y; }
                }
            }
            __syncthreads();
        }
        if (lane == 0 && my_off > 0.0) off_max = 1.0;               // some pair was still above 1e-15 in this sweep
        __syncthreads();
        const double off = off_max;
        __syncthreads();
        if (off == 0.0) break;
    }
    for (int j = warp; j < Lp; j += nwarps) {
        const double* wj = Wt + (size_t)j * p;
        double q = 0.0;
        for (int r = lane; r < p; r += 32) q = fma(wj[r], wj[r], q);
        q = warp_sum(q);
        if (lane == 0) nrm[j] = q > 0.0 ? 1.0 / sqrt(q) : 0.0;       // 1 / singular value (0 for a zero column)
    }
    __syncthreads();
    for (int i = tid; i < L * p; i += blockDim.x) Wt[i] *= nrm[i / p];   // W <- W diag(1/s): orthonormal columns
    __syncthreads();
    for (int i = tid; i < p * L; i += blockDim.x) {
        const int r = i / L, c = i - r * L;
        double s = 0.0;
        for (int k = 0; k < L; ++k) s = fma(Wt[(size_t)k * p + r], Vt[(size_t)k * Lp + c], s);
        U[i] = s;
    }
}

// k_polar_ns: the same polar factor by the Newton-Schulz iteration  X <- X (3/2 I - 1/2 X'X),  X_0 = A (scaled so that it
// converges), which is nothing but two small dense products per step - tens of microseconds on one SM where a Jacobi
// sweep is a latency chain of L - 1 dependent rounds.  Inside an optimiser's line search the raw block is the previous
// polar factor plus a small step, X'X is already close to I and three or four steps reach rounding level (the iteration
// converges quadratically).  The polar factor is unique, so the two kernels agree to ~1e-15; k_polar (Jacobi) stays as the
// fallback: status[0] = 1 asks for it when the iteration did not reach rounding level (rank-deficient / wildly scaled block).
// One CTA of 1024 threads; dynamic shared memory: X[p][PX], C[Lp][PX] (PX = Lp + 2), red[1024].
__global__ void __launch_bounds__(1024) k_polar_ns(const double* __restrict__ A /*[p][L] row-major*/, int p, int L, double* __restrict__ U,
                                                  int* __restrict__ status) {
    extern __shared__ double sm[];
    const int Lp = (L + 1) & ~1, PX = Lp + 2;
    double* X = sm;                         // [p][PX]
    double* C = X + (size_t)p * PX;         // [Lp][PX]
    double* red = C + (size_t)Lp * PX;      // [1024]
    __shared__ double s_scale;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x, nwarps = nthr >> 5;
    for (int i = tid; i < p * PX; i += nthr) {
        const int r = i / PX, c = i - r * PX;
        X[i] = c < L ? A[(size_t)r * L + c] : 0.0;
    }
    __syncthreads();
    // block-wide max of a per-thread value (all threads call it)
    auto block_max = [&](double v) -> double {
        red[tid] = v;
        __syncthreads();
        for (int o = nthr >> 1; o > 0; o >>= 1) {
            if (tid < o) red[tid] = fmax(red[tid], red[tid + o]);
            __syncthreads();
        }
        const double r = red[0];
        __syncthreads();
        return r;
    };
    // G = X'X as 2 x 2 register tiles (tile row = warp index, tile column = lane, strided over the matrix); stores
    // C = 3/2 I - 1/2 G and returns max |G - I| over the live L x L block
    auto gram = [&]() -> double {
        double e = 0.0;
        const int nt = Lp >> 1;                                   // tiles per dimension
        for (int ti = warp; ti < nt; ti += nwarps)
            for (int tj = lane; tj < nt; tj += 32) {
                const int i0 = 2 * ti, j0 = 2 * tj;
                double g00 = 0.0, g01 = 0.0, g10 = 0.0, g11 = 0.0;
                for (int r = 0; r < p; ++r) {
                    const double2 a = *reinterpret_cast<const double2*>(X + (size_t)r * PX + i0);
                    const double2 b = *reinterpret_cast<const double2*>(X + (size_t)r * PX + j0);
                    g00 = fma(a.x, b.x, g00); g01 = fma(a.x, b.y, g01); g10 = fma(a.y, b.x, g10); g11 = fma(a.y, b.y, g11);
                }
                const double g[2][2] = {{g00, g01}, {g10, g11}};
#pragma unroll
                for (int a = 0; a < 2; ++a)
#pragma unroll
                    for (int b = 0; b < 2; ++b) {
                        const int i = i0 + a, j = j0 + b;
                        const double id = i == j ? 1.0 : 0.0;
                        if (i < L && j < L) e = fmax(e, fabs(g[a][b] - id));
                        C[(size_t)i * PX + j] = 1.5 * id - 0.5 * g[a][b];
                    }
            }
        return block_max(e);
    };
    // X <- X C, four rows per warp at a time (L <= 64: lane owns columns lane and lane + 32; the old rows are only read
    // before the warp writes them back)
    auto update = [&]() {
        const int j0 = lane, j1 = lane + 32;
        for (int r0 = 4 * warp; r0 < p; r0 += 4 * nwarps) {
            double acc[4][2];
#pragma unroll
            for (int a = 0; a < 4; ++a) { acc[a][0] = 0.0; acc[a][1] = 0.0; }
            for (int k = 0; k < Lp; ++k) {
                const double c0 = j0 < Lp ? C[(size_t)k * PX + j0] : 0.0, c1 = j1 < Lp ? C[(size_t)k * PX + j1] : 0.0;
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    const double x = r0 + a < p ? X[(size_t)(r0 + a) * PX + k] : 0.0;
                    acc[a][0] = fma(x, c0, acc[a][0]);
                    acc[a][1] = fma(x, c1, acc[a][1]);
                }
            }
            __syncwarp();
#pragma unroll
            for (int a = 0; a < 4; ++a)
                if (r0 + a < p) {
                    if (j0 < Lp) X[(size_t)(r0 + a) * PX + j0] = acc[a][0];
                    if (j1 < Lp) X[(size_t)(r0 + a) * PX + j1] = acc[a][1];
                }
            __syncwarp();
        }
    };
    // ---- starting point: as it is when X'X is already close to I, else scaled below the convergence radius --------------
    double E = gram();
    if (!(E * (double)Lp < 0.9)) {
        // scale by the largest singular value: lambda_max(G) by a dozen power iterations on G = X'X = 3 I - 2 C (one warp;
        // || G v || approaches lambda_max from below, hence the margin; a bad estimate only costs iterations, and past the
        // convergence radius the loop below hands over to the Jacobi kernel)
        if (warp == 0) {
            const double v_init = 1.0 / sqrt((double)L);
            double v0 = lane < L ? v_init : 0.0, v1 = lane + 32 < L ? v_init : 0.0, lam = 0.0;
            for (int it = 0; it < 12; ++it) {
                red[lane] = v0;
                red[lane + 32] = v1;
                __syncwarp();
                double w0 = 0.0, w1 = 0.0;
                for (int k = 0; k < L; ++k) {
                    const double vk = red[k];
                    if (lane < L) w0 = fma((lane == k ? 3.0 : 0.0) - 2.0 * C[(size_t)lane * PX + k], vk, w0);
                    if (lane + 32 < L) w1 = fma((lane + 32 == k ? 3.0 : 0.0) - 2.0 * C[(size_t)(lane + 32) * PX + k], vk, w1);
                }
                lam = sqrt(warp_sum(w0 * w0 + w1 * w1));
                const double inv = lam > 0.0 ? 1.0 / lam : 0.0;
                v0 = w0 * inv;
                v1 = w1 * inv;
                __syncwarp();
            }
            if (lane == 0) s_scale = lam > 0.0 ? 1.0 / sqrt(1.05 * lam) : 0.0;
        }
        __syncthreads();
        const double sc = s_scale;
        for (int i = tid; i < p * PX; i += nthr) X[i] *= sc;
        __syncthreads();
        E = gram();
    }
    bool ok = false;
    double Eprev = 1e300;
    for (int it = 0; it < 60; ++it) {
        if (E < 1e-14) { ok = true; break; }
        if (!(E == E) || E > 2.5) break;                          // NaN / outside the convergence radius: hand over
        update();
        __syncthreads();
        if (E < 3e-8) { ok = true; break; }                      // quadratic convergence: this step ended below rounding level
        if (it >= 3 && E < 1e-12 && E >= 0.5 * Eprev) { ok = true; break; }     // stagnation at the rounding floor of X'X
        Eprev = E;
        E = gram();
    }
    if (tid == 0) status[0] = ok ? 0 : 1;
    __syncthreads();
    if (ok)
        for (int i = tid; i < p * L; i += nthr) {
            const int r = i / L, c = i - r * L;
            U[i] = X[(size_t)r * PX + c];
        }
}

// ---------------------------------------------------------------------------------------------------------------------
// The Newton-Schulz iteration of k_polar_ns for L > 64, over many CTAs: G = X'X and X <- X (3/2 I - 1/2 G) on the FP64
// tensor pipe (DMMA m8n8k4), one warp per 8 x 8 output tile, each tile's sum over k in one fixed order (bitwise
// reproducible); max |G - I| by an integer atomicMax on the bit pattern (exact for non-negative doubles, NaN above every
// number).  The decisions of k_polar_ns (starting scale, stop tests, hand-over) are taken by one thread of k_nsw_ctl on the
// device; the host launches the iterations in batches and reads one flag between them.
struct NsState {
    int active, do_mul, ok, cur, scaled;
    double Eprev, scale;
    unsigned long long Ebits;              // max |G - I| of the last G, as bits
};

// max that keeps a NaN (fmax would drop it)
__device__ __forceinline__ double nan_max(double a, double b) { return a != a ? a : (b != b ? b : fmax(a, b)); }

// grid-stride over the warps of the launch: warp w takes tile (w / ntc, w % ntc) of an [ntr x ntc] grid of 8 x 8 tiles
__device__ __forceinline__ bool next_tile(long long& w, long long nw, int ntr, int ntc, int& t0, int& t1) {
    if (w >= (long long)ntr * ntc) return false;
    t0 = (int)(w / ntc) * 8;
    t1 = (int)(w % ntc) * 8;
    w += nw;
    return true;
}

__global__ void __launch_bounds__(256) k_nsw_start(const double* __restrict__ A, long long n, double* __restrict__ X0, NsState* st) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) X0[i] = A[i];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        st->active = 1; st->do_mul = 0; st->ok = 0; st->cur = 0; st->scaled = 0;
        st->Eprev = 1e300; st->scale = 1.0; st->Ebits = 0ull;
    }
}

// G = X'X of X = Xb[cur], and max |G - I| into st->Ebits.  only_scaled: run only if the start was rescaled.
__global__ void __launch_bounds__(256) k_nsw_gram(const double* __restrict__ X0, const double* __restrict__ X1, int p, int L,
                                                 double* __restrict__ G, NsState* st, int only_scaled) {
    if (!st->active || (only_scaled && !st->scaled)) return;
    const double* X = st->cur ? X1 : X0;
    const int lane = threadIdx.x & 31, g4 = lane >> 2, q4 = lane & 3;
    const int nt = (L + 7) / 8;
    long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    int i0, j0;
    while (next_tile(w, nw, nt, nt, i0, j0)) {
        double c0 = 0.0, c1 = 0.0;
        const bool ia = i0 + g4 < L, jb = j0 + g4 < L;
        for (int r0 = 0; r0 < p; r0 += 4) {
            const int r = r0 + q4;
            const double a = (r < p && ia) ? X[(size_t)r * L + i0 + g4] : 0.0;
            const double b = (r < p && jb) ? X[(size_t)r * L + j0 + g4] : 0.0;
            dmma884(c0, c1, a, b);
        }
        double e = 0.0;
        const int i = i0 + g4;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int j = j0 + 2 * q4 + k;
            const double g = k ? c1 : c0;
            if (i < L && j < L) {
                G[(size_t)i * L + j] = g;
                e = nan_max(e, fabs(g - (i == j ? 1.0 : 0.0)));
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) e = nan_max(e, __shfl_xor_sync(FULL, e, o));
        if (lane == 0) atomicMax(&st->Ebits, (unsigned long long)__double_as_longlong(e));
    }
}

// the starting point of k_polar_ns: X as it is when X'X is close to I, else scaled so that every singular value is <= 1
// (by the Frobenius norm sqrt(trace G) >= sigma_max; the small singular values then take a few more linear steps)
__global__ void k_nsw_scale_ctl(const double* __restrict__ G, int L, NsState* st) {
    const double E = __longlong_as_double((long long)st->Ebits);
    const int Lp = (L + 1) & ~1;
    if (!(E * (double)Lp < 0.9)) {
        double tr = 0.0;
        for (int i = 0; i < L; ++i) tr += G[(size_t)i * L + i];
        st->scale = (tr > 0.0 && tr < 1e300) ? 1.0 / sqrt(tr) : 0.0;
        st->scaled = 1;
        st->Ebits = 0ull;
    }
}

__global__ void __launch_bounds__(256) k_nsw_scale(double* __restrict__ X0, long long n, const NsState* st) {
    if (!st->scaled) return;
    const double sc = st->scale;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) X0[i] *= sc;
}

// one step of k_polar_ns's loop, decided on the last E (the same tests in the same order)
__global__ void k_nsw_ctl(NsState* st, int it) {
    st->do_mul = 0;
    if (!st->active) return;
    const double E = __longlong_as_double((long long)st->Ebits);
    if (E < 1e-14) { st->ok = 1; st->active = 0; return; }
    if (!(E == E) || E > 2.5) { st->active = 0; return; }                  // NaN / outside the convergence radius: hand over
    st->do_mul = 1;
    st->cur ^= 1;
    const bool stop = E < 3e-8 || (it >= 3 && E < 1e-12 && E >= 0.5 * st->Eprev);
    st->Eprev = E;
    st->Ebits = 0ull;
    if (stop) { st->ok = 1; st->active = 0; }
}

// Xb[cur] = Xb[cur ^ 1] (3/2 I - 1/2 G)
__global__ void __launch_bounds__(256) k_nsw_mul(double* __restrict__ X0, double* __restrict__ X1, int p, int L, const double* __restrict__ G,
                                                const NsState* st) {
    if (!st->do_mul) return;
    const double* X = st->cur ? X0 : X1;
    double* Xn = st->cur ? X1 : X0;
    const int lane = threadIdx.x & 31, g4 = lane >> 2, q4 = lane & 3;
    const int nr = (p + 7) / 8, nc = (L + 7) / 8;
    long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    int r0, j0;
    while (next_tile(w, nw, nr, nc, r0, j0)) {
        double c0 = 0.0, c1 = 0.0;
        const int r = r0 + g4, j = j0 + g4;
        for (int k0 = 0; k0 < L; k0 += 4) {
            const int k = k0 + q4;
            const double a = (r < p && k < L) ? X[(size_t)r * L + k] : 0.0;
            const double b = (k < L && j < L) ? (k == j ? 1.5 : 0.0) - 0.5 * G[(size_t)k * L + j] : 0.0;
            dmma884(c0, c1, a, b);
        }
        if (r < p) {
            const int jc = j0 + 2 * q4;
            if (jc < L) Xn[(size_t)r * L + jc] = c0;
            if (jc + 1 < L) Xn[(size_t)r * L + jc + 1] = c1;
        }
    }
}

__global__ void __launch_bounds__(256) k_nsw_finish(const double* __restrict__ X0, const double* __restrict__ X1, long long n,
                                                   const NsState* st, double* __restrict__ U, int* __restrict__ status) {
    if (blockIdx.x == 0 && threadIdx.x == 0) status[0] = st->ok ? 0 : 1;
    if (!st->ok) return;
    const double* X = st->cur ? X1 : X0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) U[i] = X[i];
}

}  // namespace

size_t polar_wide_doubles(int p, int L) { return 2 * (size_t)p * L + (size_t)L * L + (sizeof(NsState) + 7) / 8; }

cudaError_t launch_polar_wide(const double* A, int p, int L, double* U, double* work, int* status, bool* converged, int* launched,
                              cudaStream_t st) {
    constexpr int MAX_IT = 60, BATCH = 6;
    const long long n = (long long)p * L;
    double* X0 = work;
    double* X1 = X0 + n;
    double* G = X1 + n;
    NsState* s = reinterpret_cast<NsState*>(G + (size_t)L * L);
    auto grid_of = [](long long warps) { return (unsigned)std::max<long long>(1, std::min<long long>((warps + 7) / 8, 148LL * 8)); };
    const long long ntl = (L + 7) / 8;
    const unsigned g_gram = grid_of(ntl * ntl), g_mul = grid_of(((p + 7) / 8) * ntl);
    const unsigned g_copy = (unsigned)std::min<long long>((n + 255) / 256, 148LL * 8);
    k_nsw_start<<<g_copy, 256, 0, st>>>(A, n, X0, s);
    k_nsw_gram<<<g_gram, 256, 0, st>>>(X0, X1, p, L, G, s, 0);
    k_nsw_scale_ctl<<<1, 1, 0, st>>>(G, L, s);
    k_nsw_scale<<<g_copy, 256, 0, st>>>(X0, n, s);
    k_nsw_gram<<<g_gram, 256, 0, st>>>(X0, X1, p, L, G, s, 1);
    *launched = 6;
    for (int it0 = 0; it0 < MAX_IT; it0 += BATCH) {
        for (int it = it0; it < it0 + BATCH && it < MAX_IT; ++it) {
            k_nsw_ctl<<<1, 1, 0, st>>>(s, it);
            k_nsw_mul<<<g_mul, 256, 0, st>>>(X0, X1, p, L, G, s);
            k_nsw_gram<<<g_gram, 256, 0, st>>>(X0, X1, p, L, G, s, 0);
            *launched += 3;
        }
        int active = 0;
        cudaError_t e = cudaMemcpyAsync(&active, &s->active, sizeof(int), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return e;
        if (!active) break;
    }
    k_nsw_finish<<<g_copy, 256, 0, st>>>(X0, X1, n, s, U, status);
    int stat = 1;
    cudaError_t e = cudaMemcpyAsync(&stat, status, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return e;
    *converged = stat == 0;
    return cudaGetLastError();
}

size_t polar_smem_bytes(int p, int L) {
    const size_t Lp = (size_t)((L + 1) & ~1);
    return sizeof(double) * (Lp * p + Lp * Lp + Lp);
}

size_t polar_ns_smem_bytes(int p, int L) {
    const size_t Lp = (size_t)((L + 1) & ~1), PX = Lp + 2;
    return sizeof(double) * ((size_t)p * PX + Lp * PX + 1024);
}

// status: one device int (workspace).  Where its shared memory fits, Newton-Schulz runs first and the Jacobi kernel only if
// it asks; elsewhere the Jacobi kernel alone.
cudaError_t launch_polar(const double* A, int p, int L, double* U, int* status, cudaStream_t st) {
    const size_t smem = polar_smem_bytes(p, L);
    if (smem > 200 * 1024) return cudaErrorInvalidValue;
    static std::atomic<int> attr_done[64];          // per device: function attributes belong to the device's context
    if (AttrOnce once(attr_done); once) {
        cudaFuncSetAttribute(k_polar, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(k_polar_ns, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    }
    const size_t ns = polar_ns_smem_bytes(p, L);
    const bool use_ns = ns <= 200 * 1024;
    if (use_ns) k_polar_ns<<<1, 1024, ns, st>>>(A, p, L, U, status);
    const int Lp = (L + 1) & ~1;
    int warps = Lp / 2;
    if (warps > 32) warps = 32;
    if (warps < 1) warps = 1;
    k_polar<<<1, 32 * warps, smem, st>>>(A, p, L, U, use_ns ? status : nullptr);
    return cudaGetLastError();
}

}  // namespace moihgp
