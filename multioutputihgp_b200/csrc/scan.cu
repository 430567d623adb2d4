// K-scan: the steady-state Kalman filter, the backward smoother and the per-step innovation
// log-likelihood as ONE chunked parallel scan over time (sm_100a).
//
// Replaces (reference, /root/reference/moihgp/include/moihgp):
//   ihgp.h:81-93     IHGP::step             x+ = AKHA x + K y        (the LTI-affine recursion)
//   ihgp.h:204-209   IHGP::negLogLikelihood v = y - HA x; 1/2 (v^2/S + log S)   on the PRE-step state
//   ihgp.h:108-113   IHGP::backwardSmoother recursion (reference_literal mode, Q3)
//   moihgp_regression.h:127-139 / :42-50    the per-observation driver loops
// plus the rts_correct smoother mode (our extension, SURVEY.md section 11).
//
// Parallel structure.  The recursion has constant matrices, so a chunk of c steps maps its
// carry-in affinely:  x_end = M^c x_in + f,  and likewise backwards.  One WARP owns one
// (sequence, latent, chunk of CH = 256 steps); lane s owns SUB = 8 consecutive steps:
//   1. every lane runs its 8 steps from zero (lane 0 from the chunk carry-in),
//   2. a Kogge-Stone warp-shuffle scan with the precomputed powers M^(8*2^k) turns the lane
//      end states into true lane start states,
//   3. every lane re-runs its 8 steps from the true start state - this is the literal
//      recurrence of the reference, so per-step values differ from the sequential loop only
//      through the ~1e-16 rounding of the carry,
//   4. the same three steps run backwards for the smoother, fused in the same kernel.
// Across chunks: k_scan<.., FINAL=false> produces per-chunk summaries from zero carries,
// k_response the (constant) linear response of a chunk to its carry-in, k_carry chains them
// (a length T/256 recurrence per (sequence, latent)), and the final pass produces the outputs from
// the true carries: k_scan_lanes (one thread per 32-step sub-chunk, latents in groups of 16 or 8)
// or k_scan<.., FINAL=true> (any shape).  The input series u[n][l][t] is read with unit stride; the
// outputs X/Xs [n][t][l][d] are written as contiguous rows.
// A block of a longer sequence sharded in time over several devices runs the same kernels in three
// phases (run_scan; ScanArgs::phase, seq_end, u_after, b_end): SURVEY.md section 8(e).
#include <cuda_runtime.h>
#include <math.h>
#include "moihgp_device.cuh"
#include "small_mat.cuh"
#include "ptx.cuh"
#include "launch.h"

namespace moihgp {

namespace {

#ifndef MOIHGP_SCAN_LOG2_SUB
#define MOIHGP_SCAN_LOG2_SUB 3
#endif
constexpr int LOG2_SUB = MOIHGP_SCAN_LOG2_SUB;   // powM[LOG2_SUB + k] = M^(SUB * 2^k)
constexpr int SUB = 1 << LOG2_SUB;               // steps per lane
constexpr int CH = 32 * SUB;                     // steps per warp-chunk
constexpr int LOG2_CH = 5 + LOG2_SUB;            // powM[LOG2_CH]     = M^CH
constexpr int LGMAX = 8;          // latents (warps) per CTA
constexpr unsigned FULL = 0xffffffffu;

template <int D>
struct LC {                       // per-warp register copy of the latent's constants
    double M[D * D], K[D], HA[D], G[D * D], drv[D * D];
};

template <int D, int MODE>
__device__ __forceinline__ void load_lc(const LatentConsts* c, LC<D>& o) {
    load_mat<D>(c->AKHA, o.M);
    load_vec<D>(c->K, o.K);
    load_vec<D>(c->HA, o.HA);
    load_mat<D>(c->G[MODE], o.G);
    if (MODE == 0) load_mat<D>(c->ImA, o.drv);
    else load_vec<D>(c->GK, o.drv);
}

// Where a lane's steps live in the CTA's shared-memory output tile:
// tile[t][lw][dd], rows of RS = lg*D doubles, each group of SUB rows padded by 2 doubles so that the
// 32 lanes of a warp (row stride SUB*RS+2) spread over the banks.
__host__ __device__ __forceinline__ int tile_group_stride(int RS) { return SUB * RS + 2; }

// One warp, one (sequence, latent, chunk).  uu[i] = u at global step tf + i (0 beyond T), u_next = u at the first
// step of the next chunk (0 if none), tf = global index of this lane's first step.
//   FINAL = false: x_in / b_in are zero (or a unit vector for k_response); returns f_end (lane 31) and beta (lane 0).
//   FINAL = true : additionally stores X / Xs rows into the shared tiles and returns sum v^2 (per lane); vrow (or null) receives
//                  each step's v^2 at its global step index.
//   INTERIOR     : every step of the chunk is < T - 1 (no end-of-sequence predicates).
//   pw           : the latent's scan powers, [2][5][D*D] doubles: M^(SUB 2^k) then G^(SUB 2^k), k = 0..4.
template <int D, int MODE, bool FINAL, bool INTERIOR>
__device__ __forceinline__ void chunk_pass(const LC<D>& c, const double* __restrict__ pw, const double (&uu)[SUB], double u_next,
                                           long long tf, long long T, const double (&x_in)[D], const double (&b_in)[D],
                                           int lane, double (&f_end)[D], double (&beta)[D], double& vsq,
                                           double* tX, double* tXs, int RS, double (&x_last_out)[D], double* __restrict__ vrow) {
    // ---- forward, local --------------------------------------------------------------------
    double z[D];
#pragma unroll
    for (int q = 0; q < D; ++q) z[q] = lane == 0 ? x_in[q] : 0.0;
#pragma unroll
    for (int i = 0; i < SUB; ++i) {
        double zn[D];
        mv<D>(c.M, z, zn);
#pragma unroll
        for (int q = 0; q < D; ++q) z[q] = fma(c.K[q], uu[i], zn[q]);      // ihgp.h:90
    }
    // ---- forward, inclusive scan over lanes ------------------------------------------------
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const int o = 1 << k;
        double zo[D], P[D * D];
#pragma unroll
        for (int q = 0; q < D; ++q) { const double t = __shfl_up_sync(FULL, z[q], o); zo[q] = lane >= o ? t : 0.0; }
#pragma unroll
        for (int q = 0; q < D * D; ++q) P[q] = pw[k * D * D + q];
        mv_acc<D>(P, zo, z);
    }
#pragma unroll
    for (int q = 0; q < D; ++q) f_end[q] = z[q];
    // ---- forward, final: the literal recurrence from the true start state --------------------
    double x[D];
#pragma unroll
    for (int q = 0; q < D; ++q) {
        const double up = __shfl_up_sync(FULL, z[q], 1);
        x[q] = lane == 0 ? x_in[q] : up;
    }
    double v[SUB], X[SUB][D];
    vsq = 0.0;
#pragma unroll
    for (int i = 0; i < SUB; ++i) {
        double hax = c.HA[0] * x[0];
#pragma unroll
        for (int q = 1; q < D; ++q) hax = fma(c.HA[q], x[q], hax);
        v[i] = uu[i] - hax;                                                  // ihgp.h:206
        double xn[D];
        mv<D>(c.M, x, xn);
#pragma unroll
        for (int q = 0; q < D; ++q) { x[q] = fma(c.K[q], uu[i], xn[q]); X[i][q] = x[q]; }   // ihgp.h:90
        if (FINAL && (INTERIOR || tf + i < T)) {
            vsq = fma(v[i], v[i], vsq);
            if (vrow) vrow[tf + i] = v[i] * v[i];
#pragma unroll
            for (int q = 0; q < D; ++q) tX[i * RS + q] = x[q];
        }
    }
#pragma unroll
    for (int q = 0; q < D; ++q) x_last_out[q] = x[q];
    // ---- what the step after this lane's last one looks like (drive of the backward pass) --------
    double v_next = 0.0, X_next[D];
    if (MODE == 1) {
        double hax = c.HA[0] * x[0];
#pragma unroll
        for (int q = 1; q < D; ++q) hax = fma(c.HA[q], x[q], hax);
        const double mine = u_next - hax;
        const double dn = __shfl_down_sync(FULL, v[0], 1);
        v_next = lane == 31 ? mine : dn;
    } else {
        double xn[D];
        mv<D>(c.M, x, xn);
#pragma unroll
        for (int q = 0; q < D; ++q) {
            const double mine = fma(c.K[q], u_next, xn[q]);
            const double dn = __shfl_down_sync(FULL, X[0][q], 1);
            X_next[q] = lane == 31 ? mine : dn;
        }
    }
    // drive g_i of the backward recursion b[j] = G b[j+1] + g[j]:
    //   rts_correct      : g[j] = G K v[j+1]            (j < T-1), 0 at j = T-1;   Xs[j] = X[j] + b[j]
    //   reference_literal: g[j] = (I - A) X[j+1]        (j < T-1), X[T-1] at j = T-1 (ihgp.h:108,111);  Xs[j] = b[j]
    auto drive = [&](int i, double (&g)[D]) {
        const long long t = tf + i;
        if (MODE == 1) {
            const double vn = (i + 1 < SUB) ? v[(i + 1) % SUB] : v_next;
            const double s = (INTERIOR || t < T - 1) ? vn : 0.0;
#pragma unroll
            for (int q = 0; q < D; ++q) g[q] = c.drv[q] * s;
        } else {
            double xn[D];
#pragma unroll
            for (int q = 0; q < D; ++q) xn[q] = (i + 1 < SUB) ? X[(i + 1) % SUB][q] : X_next[q];
            double im[D];
            mv<D>(c.drv, xn, im);
#pragma unroll
            for (int q = 0; q < D; ++q) g[q] = (INTERIOR || t < T - 1) ? im[q] : (t == T - 1 ? X[i][q] : 0.0);
        }
    };
    // ---- backward, local --------------------------------------------------------------------
    double b[D];
#pragma unroll
    for (int q = 0; q < D; ++q) b[q] = lane == 31 ? b_in[q] : 0.0;
#pragma unroll
    for (int i = SUB - 1; i >= 0; --i) {
        double g[D], bn[D];
        drive(i, g);
        mv<D>(c.G, b, bn);
#pragma unroll
        for (int q = 0; q < D; ++q) b[q] = bn[q] + g[q];
    }
    // ---- backward, inclusive scan (towards lane 0) --------------------------------------------
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const int o = 1 << k;
        double bo[D], P[D * D];
#pragma unroll
        for (int q = 0; q < D; ++q) { const double t = __shfl_down_sync(FULL, b[q], o); bo[q] = lane + o < 32 ? t : 0.0; }
#pragma unroll
        for (int q = 0; q < D * D; ++q) P[q] = pw[(5 + k) * D * D + q];
        mv_acc<D>(P, bo, b);
    }
#pragma unroll
    for (int q = 0; q < D; ++q) beta[q] = b[q];
    if (!FINAL) return;
    // ---- backward, final ----------------------------------------------------------------------
#pragma unroll
    for (int q = 0; q < D; ++q) {
        const double dn = __shfl_down_sync(FULL, b[q], 1);
        b[q] = lane == 31 ? b_in[q] : dn;
    }
#pragma unroll
    for (int i = SUB - 1; i >= 0; --i) {
        double g[D], bn[D];
        drive(i, g);
        mv<D>(c.G, b, bn);
#pragma unroll
        for (int q = 0; q < D; ++q) b[q] = bn[q] + g[q];
        if (INTERIOR || tf + i < T) {
#pragma unroll
            for (int q = 0; q < D; ++q) tXs[i * RS + q] = MODE == 1 ? tX[i * RS + q] + b[q] : b[q];
        }
    }
}

// grid: N * nG * nLG CTAs (latent-group minor), block: 32 * lg threads (lg = latents in the group, <= LGMAX); CTA
// (n, g, latent group) walks the chunks c_base + g * cpc ... (cpc chunks, fewer for the last group) so that the latent
// constants and power tables are loaded once per CTA, not once per chunk.
// Per-chunk carries are laid out [n][l][c][D] (chunk-minor: the carry kernel reads them with unit stride); vsq is [c][n][l].
template <int D, int MODE, bool FINAL>
__global__ void __launch_bounds__(32 * LGMAX, 2) k_scan(const double* __restrict__ u, const LatentConsts* __restrict__ consts,
                                                    int L, long long N, long long T, long long nC, int nLG,
                                                    long long c_base, long long c_cnt, long long cpc,
                                                    const double* __restrict__ xin, const double* __restrict__ bin,
                                                    double* __restrict__ fsum, double* __restrict__ bsum,
                                                    double* __restrict__ X, double* __restrict__ Xs,
                                                    double* __restrict__ vsq_out, double* __restrict__ xT,
                                                    const double* __restrict__ u_after, int seq_end, double* __restrict__ vstep) {
    extern __shared__ double tile[];
    __shared__ double pws[LGMAX][10 * D * D];       // per latent of the CTA: M^(SUB 2^k), then G^(SUB 2^k), k = 0..4
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    const long long nG = (c_cnt + cpc - 1) / cpc;
    const long long bid = blockIdx.x;
    const int lgi = (int)(bid % nLG);
    const long long gi = (bid / nLG) % nG;
    const long long n = bid / ((long long)nLG * nG);
    const int l0 = lgi * LGMAX;
    const int lg = min(LGMAX, L - l0);          // == blockDim.x / 32 for all but a ragged last group
    const int l = l0 + wi;
    const bool active = wi < lg;
    const int RS = lg * D;
    const int GS = tile_group_stride(RS);
    double* tileX = tile;
    double* tileXs = tile + 32 * GS;
    // 16-byte copy-out needs even row widths / offsets and aligned output bases (GS = SUB RS + 2 is then even too)
    const bool vec_out = FINAL && (RS & 1) == 0 && (((size_t)L * D) & 1) == 0 && ((l0 * D) & 1) == 0 &&
                         (reinterpret_cast<size_t>(X) & 15) == 0 && (reinterpret_cast<size_t>(Xs) & 15) == 0;
    for (int i = threadIdx.x; i < lg * 10 * D * D; i += blockDim.x) {
        const int w = i / (10 * D * D), r = i - w * (10 * D * D);
        const int m = r / (D * D), e = r - m * (D * D);
        const LatentConsts* lcw = consts + l0 + w;
        const double* src = m < 5 ? lcw->powM[LOG2_SUB + m] : lcw->powG[MODE][LOG2_SUB + m - 5];
        pws[w][r] = src[(e / D) * 3 + (e % D)];
    }
    __syncthreads();
    const LatentConsts* lc = consts + (active ? l : l0);
    LC<D> cst;
    load_lc<D, MODE>(lc, cst);
    const double* up = u + ((size_t)n * L + (active ? l : l0)) * T;
    double* const vrow = FINAL && vstep ? vstep + ((size_t)n * L + (active ? l : l0)) * T : nullptr;   // laid out like u
    const long long c_lo = c_base + gi * cpc, c_hi = min(c_base + c_cnt, c_lo + cpc);

    for (long long c = c_lo; c < c_hi; ++c) {
        const long long t0 = c * CH;
        if (active) {
            const long long tf = t0 + (long long)lane * SUB;
            double uu[SUB];
            if (tf + SUB <= T && ((reinterpret_cast<size_t>(up + tf) & 15) == 0)) {
#pragma unroll
                for (int i = 0; i < SUB; i += 2) {
                    const double2 t2 = __ldg(reinterpret_cast<const double2*>(up + tf + i));
                    uu[i] = t2.x;
                    uu[i + 1] = t2.y;
                }
            } else {
#pragma unroll
                for (int i = 0; i < SUB; ++i) uu[i] = tf + i < T ? __ldg(up + tf + i) : 0.0;
            }
            // the step after the chunk: the next chunk's first, or (block of a longer sequence) the next block's first
            const double u_next = t0 + CH < T ? __ldg(up + t0 + CH) : (u_after ? __ldg(u_after + (size_t)n * L + l) : 0.0);
            double x_in[D], b_in[D], f_end[D], beta[D], x_last[D], vsq;
            const size_t ci = (((size_t)n * L + l) * nC + c) * D;      // carries are chunk-minor: [n][l][chunk][D]
#pragma unroll
            for (int q = 0; q < D; ++q) {
                x_in[q] = FINAL ? xin[ci + q] : 0.0;
                b_in[q] = FINAL ? bin[ci + q] : 0.0;
            }
            double* tX = tileX + lane * GS + wi * D;
            double* tXs = tileXs + lane * GS + wi * D;
            if (t0 + CH < T || !seq_end) chunk_pass<D, MODE, FINAL, true>(cst, pws[wi], uu, u_next, tf, T, x_in, b_in, lane, f_end, beta, vsq, tX, tXs, RS, x_last, vrow);
            else chunk_pass<D, MODE, FINAL, false>(cst, pws[wi], uu, u_next, tf, T, x_in, b_in, lane, f_end, beta, vsq, tX, tXs, RS, x_last, vrow);
            if (!FINAL) {
                if (lane == 31) {
#pragma unroll
                    for (int q = 0; q < D; ++q) fsum[ci + q] = f_end[q];
                }
                if (lane == 0) {
#pragma unroll
                    for (int q = 0; q < D; ++q) bsum[ci + q] = beta[q];
                }
            } else {
                // deterministic warp reduction of sum v^2
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) vsq += __shfl_xor_sync(FULL, vsq, o);
                if (lane == 0) vsq_out[((size_t)c * N + n) * L + l] = vsq;
                // final filtered state of the sequence: X[T-1]
                if (xT && T - 1 >= tf && T - 1 < tf + SUB) {
                    const int i = (int)(T - 1 - tf);
#pragma unroll
                    for (int q = 0; q < D; ++q) xT[((size_t)n * L + l) * D + q] = tX[i * RS + q];
                }
            }
        }
        if (FINAL) {
            __syncthreads();
            // ---- coalesced copy-out of the staged rows ------------------------------------------------
            const int rows = (int)min((long long)CH, T - t0);
            const size_t grow = (size_t)L * D;                       // global row pitch (doubles)
            const size_t gbase = ((size_t)n * T + t0) * grow + (size_t)l0 * D;
            // element (row, col) of the staged tile, walked without integer divisions: this thread starts at
            // (tid / W, tid % W) and advances by blockDim.x elements per iteration (W = row width in copy units)
            if (vec_out) {
                const int W = RS >> 1;                               // 16-byte units per row
                int row = threadIdx.x / W, col = threadIdx.x - row * W;
                const int drow = blockDim.x / W, dcol = blockDim.x - drow * W;
                while (row < rows) {
                    const int so = (row / SUB) * GS + (row % SUB) * RS + 2 * col;
                    const size_t go = gbase + (size_t)row * grow + 2 * col;
                    if (X) *reinterpret_cast<double2*>(X + go) = *reinterpret_cast<const double2*>(tileX + so);
                    if (Xs) *reinterpret_cast<double2*>(Xs + go) = *reinterpret_cast<const double2*>(tileXs + so);
                    row += drow; col += dcol;
                    if (col >= W) { col -= W; ++row; }
                }
            } else {
                int row = threadIdx.x / RS, col = threadIdx.x - row * RS;
                const int drow = blockDim.x / RS, dcol = blockDim.x - drow * RS;
                while (row < rows) {
                    const int so = (row / SUB) * GS + (row % SUB) * RS + col;
                    const size_t go = gbase + (size_t)row * grow + col;
                    if (X) X[go] = tileX[so];
                    if (Xs) Xs[go] = tileXs[so];
                    row += drow; col += dcol;
                    if (col >= RS) { col -= RS; ++row; }
                }
            }
            __syncthreads();                                        // the tiles are reused by the next chunk
        }
    }
}

// Summaries of the INTERIOR chunks (every chunk but the last of a sequence) from zero carries.  Both summaries are
// linear in the chunk's inputs, so they are dot products with the weights k_scan_weights tabulated (f_end and beta per
// unit input) plus beta's response to u_next.  One warp per (sequence, latent, group of chunks): the lane's 2 D x SUB
// weights stay in registers while it walks its chunks - the pass is a pure stream over u.
constexpr int WS_STRIDE = 2 * DMAX * CH + 4;       // doubles per latent in Wsum (even: 16-byte loads)
template <int D>
__global__ void __launch_bounds__(128) k_scan_summaries_dot(const double* __restrict__ u, const double* __restrict__ Wsum, int L,
                                                           long long N, long long T, long long nC, long long cpw,
                                                           double* __restrict__ fsum, double* __restrict__ bsum) {
    const int lane = threadIdx.x & 31;
    const long long nI = nC - 1;                                    // interior chunks
    const long long nG = (nI + cpw - 1) / cpw;
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (wid >= N * L * nG) return;
    const long long g = wid % nG;
    const int l = (int)((wid / nG) % L);
    const long long n = wid / (nG * L);
    const double* wl = Wsum + (size_t)l * WS_STRIDE;
    double w[2 * D][SUB], wn[D];
    // a dot product does not care which lane owns which step: lane takes steps 64 i + 2 lane + {0, 1}, i = 0..3, so that
    // every warp-wide 16-byte load of u is one contiguous 512-byte run
#pragma unroll
    for (int k = 0; k < 2 * D; ++k)
#pragma unroll
        for (int i = 0; i < SUB; i += 2) {
            const double2 t2 = __ldg(reinterpret_cast<const double2*>(wl + k * CH + 32 * i + 2 * lane));
            w[k][i] = t2.x;
            w[k][i + 1] = t2.y;
        }
#pragma unroll
    for (int q = 0; q < D; ++q) wn[q] = __ldg(wl + 2 * D * CH + q);
    const double* up = u + ((size_t)n * L + l) * T;
    const bool vec = (reinterpret_cast<size_t>(up) & 15) == 0;      // chunk starts are multiples of 256 steps
    const long long c_hi = min(nI, (g + 1) * cpw);
    // software pipeline: the loads of chunk c + 1 are in flight while chunk c is reduced (one chunk per warp in flight
    // leaves 32 KB per SM outstanding - not enough to cover the HBM latency at full bandwidth)
    auto load_chunk = [&](long long c, double (&uu)[SUB], double& u_next) {
        const long long tb = c * CH + 2 * lane;
        if (vec) {
#pragma unroll
            for (int i = 0; i < SUB; i += 2) {
                const double2 t2 = __ldg(reinterpret_cast<const double2*>(up + tb + 32 * i));
                uu[i] = t2.x;
                uu[i + 1] = t2.y;
            }
        } else {
#pragma unroll
            for (int i = 0; i < SUB; i += 2) { uu[i] = __ldg(up + tb + 32 * i); uu[i + 1] = __ldg(up + tb + 32 * i + 1); }
        }
        u_next = __ldg(up + (c + 1) * CH);
    };
    double un[SUB], un_next = 0.0;
    if (g * cpw < c_hi) load_chunk(g * cpw, un, un_next);
    for (long long c = g * cpw; c < c_hi; ++c) {
        double uu[SUB];
#pragma unroll
        for (int i = 0; i < SUB; ++i) uu[i] = un[i];
        const double u_next = un_next;
        if (c + 1 < c_hi) load_chunk(c + 1, un, un_next);
        double acc[2 * D];
#pragma unroll
        for (int k = 0; k < 2 * D; ++k) {
            double a = w[k][0] * uu[0];
#pragma unroll
            for (int i = 1; i < SUB; ++i) a = fma(w[k][i], uu[i], a);
            acc[k] = a;
        }
#pragma unroll
        for (int k = 0; k < 2 * D; ++k)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(FULL, acc[k], o);
        if (lane == 0) {
            const size_t ci = (((size_t)n * L + l) * nC + c) * D;
#pragma unroll
            for (int q = 0; q < D; ++q) { fsum[ci + q] = acc[q]; bsum[ci + q] = fma(wn[q], u_next, acc[D + q]); }
        }
    }
}

// Weights of the summaries of an INTERIOR chunk run from zero carries: with unit input at step i (or at u_next) the chunk
// returns f_end (lane 31) and beta (lane 0).  Layout per latent (stride WS_STRIDE): [2 D][CH] (f_end rows, then beta
// rows), then beta's response to u_next [D].  grid: L * (CH + 1) blocks of one warp.
template <int D, int MODE>
__global__ void __launch_bounds__(32) k_scan_weights(const LatentConsts* __restrict__ consts, double* __restrict__ Wsum) {
    const int lane = threadIdx.x;
    const int i = blockIdx.x % (CH + 1);
    const int l = blockIdx.x / (CH + 1);
    const LatentConsts* lc = consts + l;
    LC<D> cst;
    load_lc<D, MODE>(lc, cst);
    __shared__ double pw[10 * D * D];
    for (int k = lane; k < 10 * D * D; k += 32) {
        const int m = k / (D * D), e = k - m * (D * D);
        const double* src = m < 5 ? lc->powM[LOG2_SUB + m] : lc->powG[MODE][LOG2_SUB + m - 5];
        pw[k] = src[(e / D) * 3 + (e % D)];
    }
    __syncwarp();
    double uu[SUB];
#pragma unroll
    for (int k = 0; k < SUB; ++k) uu[k] = (i < CH && lane * SUB + k == i) ? 1.0 : 0.0;
    double x_in[D], b_in[D], f_end[D], beta[D], x_last[D], vsq;
#pragma unroll
    for (int q = 0; q < D; ++q) { x_in[q] = 0.0; b_in[q] = 0.0; }
    chunk_pass<D, MODE, false, true>(cst, pw, uu, i == CH ? 1.0 : 0.0, (long long)lane * SUB, 1LL << 60, x_in, b_in, lane, f_end, beta, vsq, nullptr, nullptr, 0, x_last, nullptr);
    double* wl = Wsum + (size_t)l * WS_STRIDE;
    if (i < CH) {
        if (lane == 31) {
#pragma unroll
            for (int q = 0; q < D; ++q) wl[q * CH + i] = f_end[q];
        }
        if (lane == 0) {
#pragma unroll
            for (int q = 0; q < D; ++q) wl[(D + q) * CH + i] = beta[q];
        }
    } else if (lane == 0) {
#pragma unroll
        for (int q = 0; q < D; ++q) wl[2 * D * CH + q] = beta[q];
    }
}

// Linear response of a chunk's backward summary to its forward carry-in: column k of Bx is beta(u = 0, x_in = e_k).
// kind 0: interior chunk (CH steps, a next chunk exists); kind 1: last chunk of the sequence (r_last steps).
// grid: L * 2 * D blocks of one warp.  Bx layout [l][kind][D*D] row-major.
template <int D, int MODE>
__global__ void __launch_bounds__(32) k_response(const LatentConsts* __restrict__ consts, long long r_last, double* __restrict__ Bx) {
    const int lane = threadIdx.x;
    const int k = blockIdx.x % D;
    const int kind = (blockIdx.x / D) % 2;
    const int l = blockIdx.x / (2 * D);
    const LatentConsts* lc = consts + l;
    LC<D> cst;
    load_lc<D, MODE>(lc, cst);
    __shared__ double pw[10 * D * D];
    for (int i = lane; i < 10 * D * D; i += 32) {
        const int m = i / (D * D), e = i - m * (D * D);
        const double* src = m < 5 ? lc->powM[LOG2_SUB + m] : lc->powG[MODE][LOG2_SUB + m - 5];
        pw[i] = src[(e / D) * 3 + (e % D)];
    }
    __syncwarp();
    double uu[SUB];
#pragma unroll
    for (int i = 0; i < SUB; ++i) uu[i] = 0.0;
    double x_in[D], b_in[D], f_end[D], beta[D], x_last[D], vsq;
#pragma unroll
    for (int q = 0; q < D; ++q) { x_in[q] = q == k ? 1.0 : 0.0; b_in[q] = 0.0; }
    const long long T = kind == 0 ? (1LL << 60) : r_last;
    chunk_pass<D, MODE, false, false>(cst, pw, uu, 0.0, (long long)lane * SUB, T, x_in, b_in, lane, f_end, beta, vsq, nullptr, nullptr, 0, x_last, nullptr);
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < D; ++q) Bx[((size_t)l * 2 + kind) * D * D + q * D + k] = beta[q];
    }
}

// Chain the chunk summaries.
//   forward : xin[c+1] = M^CH xin[c] + f[c]
//   backward: bin[c-1] = beta0[c] + Bx(kind c) xin[c] + G^CH bin[c]
// Three levels (a single long sequence has tens of thousands of chunks: BASELINE config 4, T = 1e7, 39 063 chunks):
//   group       = 32 CG chunks scanned by one warp (lane = CG consecutive chunks, Kogge-Stone over lanes with the
//                 powers M^(CH CG 2^k));
//   super-block = SB consecutive groups walked in sequence by that warp;
//   k_carry_super chains the super-blocks (one thread per (sequence, latent), power M^(CH CG 32 SB)).
// k_carry<DIR, PHASE>: PHASE 0 runs every super-block from a zero carry and only reports its end value; PHASE 1 runs it
// from the true carry and writes xin / bin.  When there is one super-block PHASE 1 alone is launched.
// Granularity of the carry chain, swept on config 4 (39 063 chunks per latent; profiles/r02/carry_granularity.txt): chunks per
// lane 8 / 4 / 2 / 1 with 8 groups per super-block: k_carry 0.193 / 0.122 / 0.114 / - ms; with 16 groups: - / 0.137 / 0.107 /
// 0.126 ms.  Fewer chunks per lane = shorter sequential walks inside a lane, more warps.
#ifndef MOIHGP_SCAN_LOG2_CG
#define MOIHGP_SCAN_LOG2_CG 1
#endif
#ifndef MOIHGP_SCAN_LOG2_SB
#define MOIHGP_SCAN_LOG2_SB 4
#endif
constexpr int LOG2_CG = MOIHGP_SCAN_LOG2_CG;
constexpr int CG = 1 << LOG2_CG;   // chunks per lane
constexpr int LOG2_SB = MOIHGP_SCAN_LOG2_SB;
constexpr int SB = 1 << LOG2_SB;   // groups per super-block
template <int D, int MODE, int DIR, int PHASE>
__global__ void __launch_bounds__(128) k_carry(const LatentConsts* __restrict__ consts, const double* __restrict__ Bx, int L,
                                              long long N, long long nC, long long nS, const double* __restrict__ x0,
                                              const double* __restrict__ fsum, const double* __restrict__ bsum,
                                              double* __restrict__ xin, double* __restrict__ bin,
                                              const double* __restrict__ sb_in, double* __restrict__ sb_end,
                                              const double* __restrict__ b_end, int seq_end) {
    const int lane = threadIdx.x & 31;
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (wid >= N * L * nS) return;
    const long long sbi = wid % nS;                                  // super-block
    const long long id = wid / nS;                                   // (sequence, latent)
    const int l = (int)(id % L);
    const LatentConsts* lc = consts + l;
    double TC[D * D];                                                // one-chunk transition: M^CH (forward) / G^CH (backward)
    load_mat<D>(DIR == 0 ? lc->powM[LOG2_CH] : lc->powG[MODE][LOG2_CH], TC);
    double Bf[D * D], Bl[D * D];
    if (DIR == 1) {
#pragma unroll
        for (int i = 0; i < D * D; ++i) { Bf[i] = Bx[((size_t)l * 2 + 0) * D * D + i]; Bl[i] = Bx[((size_t)l * 2 + 1) * D * D + i]; }
    }
    __shared__ double pcs[4][5 * D * D];       // per warp: the scan powers T^(CG 2^k), k = 0..4
    {
        double* pc = pcs[threadIdx.x >> 5];
        for (int i = lane; i < 5 * D * D; i += 32) {
            const int m = i / (D * D), e = i - m * (D * D);
            const double* src = DIR == 0 ? lc->powM[LOG2_CH + LOG2_CG + m] : lc->powG[MODE][LOG2_CH + LOG2_CG + m];
            pc[i] = src[(e / D) * 3 + (e % D)];
        }
        __syncwarp();
    }
    const double* pcw = pcs[threadIdx.x >> 5];
    const size_t stride = D;                   // between consecutive chunks of one (sequence, latent): [n][l][chunk][D]
    const size_t base = (size_t)id * nC * D;
    const long long nG = (nC + 32 * CG - 1) / (32 * CG);
    const long long g_lo = sbi * SB, g_hi = min(nG, g_lo + SB);

    double carry[D];
#pragma unroll
    for (int q = 0; q < D; ++q) {
        if (PHASE == 0) carry[q] = 0.0;
        else if (sb_in) carry[q] = sb_in[(size_t)wid * D + q];
        else carry[q] = (DIR == 0 && x0) ? x0[(size_t)id * D + q] : 0.0;
    }
    // drive of chunk c:  forward f[c] (f of the last chunk is never used);  backward d[c] = beta0[c] + B(kind c) xin[c]
    auto load_drive = [&](long long g, double (&dv)[CG][D]) {
        const long long c0 = (g * 32 + lane) * CG;
#pragma unroll
        for (int i = 0; i < CG; ++i) {
            const long long c = c0 + i;
            if (DIR == 0) {
#pragma unroll
                for (int q = 0; q < D; ++q) dv[i][q] = (c < nC - 1) ? fsum[c * stride + base + q] : 0.0;
            } else if (c >= 1 && c < nC) {
                double xi[D], bn[D];
#pragma unroll
                for (int q = 0; q < D; ++q) { xi[q] = xin[c * stride + base + q]; bn[q] = bsum[c * stride + base + q]; }
                mv_acc<D>((c == nC - 1 && seq_end) ? Bl : Bf, xi, bn);
                if (c == nC - 1 && b_end) {              // the value entering the block from the right: + G^CH b_end
                    double be[D];
#pragma unroll
                    for (int q = 0; q < D; ++q) be[q] = b_end[(size_t)id * D + q];
                    mv_acc<D>(TC, be, bn);
                }
#pragma unroll
                for (int q = 0; q < D; ++q) dv[i][q] = bn[q];
            } else {
#pragma unroll
                for (int q = 0; q < D; ++q) dv[i][q] = 0.0;
            }
        }
    };
    const int lane_in = DIR == 0 ? 0 : 31;       // the lane that receives the carry
    for (long long gg = 0; gg < g_hi - g_lo; ++gg) {
        const long long g = DIR == 0 ? g_lo + gg : g_hi - 1 - gg;
        const long long c0 = (g * 32 + lane) * CG;
        double dv[CG][D];
        load_drive(g, dv);
        // local run of this lane's CG chunks (ascending for the forward chain, descending for the backward one)
        double z[D];
#pragma unroll
        for (int q = 0; q < D; ++q) z[q] = lane == lane_in ? carry[q] : 0.0;
#pragma unroll
        for (int ii = 0; ii < CG; ++ii) {
            const int i = DIR == 0 ? ii : CG - 1 - ii;
            double zn[D];
            mv<D>(TC, z, zn);
#pragma unroll
            for (int q = 0; q < D; ++q) z[q] = zn[q] + dv[i][q];
        }
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const int o = 1 << k;
            double zo[D], P[D * D];
#pragma unroll
            for (int q = 0; q < D; ++q) {
                const double t = DIR == 0 ? __shfl_up_sync(FULL, z[q], o) : __shfl_down_sync(FULL, z[q], o);
                zo[q] = (DIR == 0 ? lane >= o : lane + o < 32) ? t : 0.0;
            }
#pragma unroll
            for (int q = 0; q < D * D; ++q) P[q] = pcw[k * D * D + q];
            mv_acc<D>(P, zo, z);
        }
        double x[D];                                 // the value entering this lane's first chunk (forward) / last chunk (backward)
#pragma unroll
        for (int q = 0; q < D; ++q) {
            const double nb = DIR == 0 ? __shfl_up_sync(FULL, z[q], 1) : __shfl_down_sync(FULL, z[q], 1);
            x[q] = lane == lane_in ? carry[q] : nb;
            carry[q] = __shfl_sync(FULL, z[q], DIR == 0 ? 31 : 0);
        }
        if (PHASE == 1) {
#pragma unroll
            for (int ii = 0; ii < CG; ++ii) {
                const int i = DIR == 0 ? ii : CG - 1 - ii;
                const long long c = c0 + i;
                if (c < nC) {
#pragma unroll
                    for (int q = 0; q < D; ++q) {
                        if (DIR == 0) xin[c * stride + base + q] = x[q];
                        else bin[c * stride + base + q] = c == nC - 1 ? (b_end ? b_end[(size_t)id * D + q] : 0.0) : x[q];
                    }
                }
                double xn[D];
                mv<D>(TC, x, xn);
#pragma unroll
                for (int q = 0; q < D; ++q) x[q] = xn[q] + dv[i][q];
            }
        }
    }
    if (PHASE == 0 && lane == 0) {
#pragma unroll
        for (int q = 0; q < D; ++q) sb_end[(size_t)wid * D + q] = carry[q];
    }
}

// What leaves a block on the left: the backward value at its first step, b_out = beta0[0] + B xin[0] + G^CH bin[0]
// (the previous block's b_end).  One thread per (sequence, latent).
template <int D, int MODE>
__global__ void __launch_bounds__(128) k_block_start(const LatentConsts* __restrict__ consts, const double* __restrict__ Bx, int L,
                                                    long long N, long long nC, int seq_end, const double* __restrict__ xin,
                                                    const double* __restrict__ bsum, const double* __restrict__ bin,
                                                    double* __restrict__ b_out) {
    const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= N * L) return;
    const int l = (int)(id % L);
    double TC[D * D], B[D * D], xi[D], bi[D], o[D];
    load_mat<D>(consts[l].powG[MODE][LOG2_CH], TC);
    const int kind = (nC == 1 && seq_end) ? 1 : 0;
#pragma unroll
    for (int i = 0; i < D * D; ++i) B[i] = Bx[((size_t)l * 2 + kind) * D * D + i];
    const size_t ci = (size_t)id * nC * D;
#pragma unroll
    for (int q = 0; q < D; ++q) { xi[q] = xin[ci + q]; bi[q] = bin[ci + q]; o[q] = bsum[ci + q]; }
    mv_acc<D>(B, xi, o);
    mv_acc<D>(TC, bi, o);
#pragma unroll
    for (int q = 0; q < D; ++q) b_out[(size_t)id * D + q] = o[q];
}

// Filtered state after the last step of a block of whole chunks: x_end = M^CH xin[nC-1] + fsum[nC-1].  One thread per
// (sequence, latent).
template <int D>
__global__ void __launch_bounds__(128) k_block_end(const LatentConsts* __restrict__ consts, int L, long long N, long long nC,
                                                  const double* __restrict__ xin, const double* __restrict__ fsum,
                                                  double* __restrict__ x_end) {
    const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= N * L) return;
    double TC[D * D], x[D], o[D];
    load_mat<D>(consts[(int)(id % L)].powM[LOG2_CH], TC);
    const size_t ci = ((size_t)id * nC + (nC - 1)) * D;
#pragma unroll
    for (int q = 0; q < D; ++q) x[q] = xin[ci + q];
    mv<D>(TC, x, o);
#pragma unroll
    for (int q = 0; q < D; ++q) x_end[(size_t)id * D + q] = o[q] + fsum[ci + q];
}

// Chain the super-blocks: one thread per (sequence, latent).  forward: in[S+1] = M^span in[S] + end[S], in[0] = x0;
// backward: in[S-1] = G^span in[S] + end[S], in[nS-1] = 0.  span = CH * CG * 32 * SB steps.
template <int D, int MODE, int DIR>
__global__ void __launch_bounds__(128) k_carry_super(const LatentConsts* __restrict__ consts, int L, long long N, long long nS,
                                                    const double* __restrict__ x0, const double* __restrict__ sb_end,
                                                    double* __restrict__ sb_in) {
    const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= N * L) return;
    const LatentConsts* lc = consts + (int)(id % L);
    double P[D * D], v[D];
    load_mat<D>(DIR == 0 ? lc->powM[LOG2_CH + LOG2_CG + 5 + LOG2_SB] : lc->powG[MODE][LOG2_CH + LOG2_CG + 5 + LOG2_SB], P);
#pragma unroll
    for (int q = 0; q < D; ++q) v[q] = (DIR == 0 && x0) ? x0[(size_t)id * D + q] : 0.0;
#pragma unroll 8                      // the loads of sb_end do not depend on the chain: eight of them in flight
    for (long long k = 0; k < nS; ++k) {
        const long long sb = DIR == 0 ? k : nS - 1 - k;
        const size_t o = ((size_t)id * nS + sb) * D;
        double vn[D];
#pragma unroll
        for (int q = 0; q < D; ++q) sb_in[o + q] = v[q];
        mv<D>(P, v, vn);
#pragma unroll
        for (int q = 0; q < D; ++q) v[q] = vn[q] + sb_end[o + q];
    }
}

// nll[n] = sum_t [ 1/2 log(sum S) + 1/2 m_n log(sigma) + 1/2 rho_t / sigma ]            moihgp.h:653
//        + sum_l sum_t 1/2 ( v^2 / S_l + log S_l )                                       ihgp.h:207, moihgp.h:675,684
// Two stages, fixed order (deterministic): nll_nsplit(N) CTAs per sequence, then one thread per sequence.
// The split count follows the number of sequences: few long sequences (config 4: one sequence, 625 000 + 1 250 000 terms)
// get 1024 CTAs per sequence, many sequences 64 (k_nll_partial 56 -> 9 us at config 4).
__host__ __device__ inline int nll_nsplit(long long N) { return N >= 16 ? 64 : 1024; }
__global__ void __launch_bounds__(256) k_nll_partial(const double* __restrict__ rho_part, const double* __restrict__ vsq,
                                                    const LatentConsts* __restrict__ consts, double sigma, int L, long long N,
                                                    long long tiles, long long nC, int nsplit, double* __restrict__ part) {
    __shared__ double red[256];
    __shared__ double hinvS[64];                                         // 1 / (2 S_l)
    const long long n = blockIdx.x / nsplit;
    const int sp = blockIdx.x % nsplit;
    const int tid = threadIdx.x;
    const bool inv_sm = L <= 64;
    if (inv_sm && tid < L) hinvS[tid] = 0.5 / consts[tid].S;
    __syncthreads();
    double acc = 0.0;
    const long long tb = (tiles + nsplit - 1) / nsplit;
    for (long long i = sp * tb + tid; i < min(tiles, (sp + 1) * tb); i += 256) acc += rho_part[n * tiles + i];
    acc *= 0.5 / sigma;
    const long long cb = (nC + nsplit - 1) / nsplit;
    for (long long i = sp * cb * L + tid; i < min(nC, (sp + 1) * cb) * L; i += 256) {
        const long long c = i / L;
        const int l = (int)(i - c * L);
        const double v = vsq[((size_t)c * N + n) * L + l];
        acc += inv_sm ? v * hinvS[l] : 0.5 * v / consts[l].S;
    }
    red[tid] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o) red[tid] += red[tid + o];
        __syncthreads();
    }
    if (tid == 0) part[n * nsplit + sp] = red[0];
}
// one WARP per sequence: lane i sums the partials i, i + 32, ... in order, then a fixed-order butterfly - deterministic, and
// the nsplit loads are spread over the lanes instead of queued behind one thread (48 -> 6 us at nsplit = 1024)
__global__ void __launch_bounds__(128) k_nll_reduce(const double* __restrict__ part, const LatentConsts* __restrict__ consts,
                                                   const double* __restrict__ S, double sigma, int p, int L, long long N,
                                                   long long T, int nsplit, double* __restrict__ nll) {
    const long long n = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    double acc = 0.0;
    for (int i = lane; i < nsplit; i += 32) acc += part[n * nsplit + i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane != 0) return;
    double logs = 0.0;
    for (int l = 0; l < L; ++l) logs += consts[l].logS;
    nll[n] = acc + (double)T * (nll_step_const(S, p, L, sigma) + 0.5 * logs);   // moihgp.h:652
}

// Per-step terms of the same sum (MOIHGP::negLogLikelihood(x_{t-1}, y_t), moihgp.h:614-688), one thread per (sequence, step):
//   nll_steps[n][t] = 1/2 rho_t / sigma + sum_l 1/2 v_{l,t}^2 / S_l + nll_step_const + 1/2 sum_l log S_l
// rho_t arrives in nll_steps itself (the projection's per-row residual norms) and is replaced in place; vstep[n][l][t] holds v^2
// (the final scan pass).  The latents are summed in order l = 0 .. L-1: deterministic, no atomics.
__global__ void __launch_bounds__(256) k_nll_steps(const double* __restrict__ vstep, const LatentConsts* __restrict__ consts,
                                                  const double* __restrict__ S, double sigma, int p, int L, long long N, long long T,
                                                  double* __restrict__ nll_steps) {
    __shared__ double hinvS[64];                                         // 1 / (2 S_l)
    __shared__ double cst;
    const int tid = threadIdx.x;
    const bool inv_sm = L <= 64;
    if (inv_sm && tid < L) hinvS[tid] = 0.5 / consts[tid].S;
    if (tid == 0) {
        double logs = 0.0;
        for (int l = 0; l < L; ++l) logs += consts[l].logS;
        cst = nll_step_const(S, p, L, sigma) + 0.5 * logs;
    }
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + tid;
    if (i >= N * T) return;
    const long long n = i / T, t = i - n * T;
    const double* vr = vstep + (size_t)n * L * T + t;
    double vs = 0.0;
    for (int l = 0; l < L; ++l) vs += vr[(size_t)l * T] * (inv_sm ? hinvS[l] : 0.5 / consts[l].S);
    nll_steps[i] = 0.5 * nll_steps[i] / sigma + vs + cst;
}

// ---------------------------------------------------------------------------------------------------------------------
// k_scan_lanes: the FINAL pass with one THREAD per (latent, sub-chunk of SL = 32 steps) instead of one warp per
// (latent, chunk).  A CTA owns (sequence, group of LG latents, chunk of CH = 256 steps): thread (s, l) runs sub-chunk s
// of latent l sequentially, exactly as the reference's loop does (ihgp.h:81-93, :108-113), four times:
//   A  forward from zero                          -> sub-chunk summary f_s
//      carries: x_in(s+1) = M^32 x_in(s) + f_s, x_in(0) = the chunk's carry-in (k_carry)
//   B  forward from the true carry: X (registers -> HBM, 16 bytes per lane, LG*D*8 contiguous bytes per step) and a
//      private copy in shared memory for the way back; sum v^2
//   C  backward from zero over the stored X       -> beta_s;  b_in(s-1) = G^32 b_in(s) + beta_s
//   D  backward from the true carry: Xs -> HBM.
// No warp shuffles, no staging tile, ~45 instructions per latent-step and lane (the warp-per-chunk kernel above executes
// ~215): the pass becomes a stream over u (read) and X, Xs (written).  The per-step arithmetic is the literal recurrence;
// as in k_scan only the carries differ from the sequential loop, by rounding.
constexpr int SL = 32;                 // steps per thread
constexpr int NSUBC = CH / SL;         // sub-chunks per chunk
constexpr int LOG2_SL = 5;

template <int D, int MODE, int LG, bool INTERIOR>
__device__ __forceinline__ void lanes_chunk(const LC<D>& c, const double (&PM)[D * D], const double (&PG)[D * D],
                                            const double* __restrict__ up, double u_nx, long long ts, long long T, int s, int li, int tid,
                                            const double* x_chunk, const double* b_chunk, double* tile,
                                            unsigned long long* ubar, unsigned uphase,
                                            double (*exch)[LG][D], double (*vred)[LG], double* __restrict__ Xg,
                                            double* __restrict__ Xsg, size_t gstride, bool vec_x, double* __restrict__ vsq_dst,
                                            double* __restrict__ xT_dst, double* __restrict__ vrow) {
    constexpr int NT = NSUBC * LG;
    const int len = INTERIOR ? SL : (int)max(0LL, min((long long)SL, T - ts));
    // ---- inputs: this thread's 32 steps of u (contiguous) and the step after them --------------------------------
    // A lane-private 256-byte run per thread would cost 32 LSU wavefronts per warp-wide load; instead every thread has
    // the copy engine (cp.async.bulk) drop its run into a slot of the (currently idle) X tile and reads it back with
    // conflict-free 16-byte shared-memory loads (slot pitch 34 doubles).
    constexpr int UP = SL + 2;
    double* slot = tile + tid * UP;
    const bool bulk = (INTERIOR || len == SL) && ((reinterpret_cast<size_t>(up + ts) & 15) == 0);
    fence_async_smem();                               // the tile was last read through the generic proxy (previous chunk)
    if (bulk) {
        mbar_expect_tx(ubar, SL * (unsigned)sizeof(double));
        bulk_g2s(slot, up + ts, SL * (unsigned)sizeof(double), ubar);
    } else mbar_arrive(ubar);
    if (!bulk) {                                      // ragged end of the sequence / odd alignment: fill the slot by hand
        for (int j = 0; j < SL; ++j) slot[j] = (INTERIOR || j < len) ? __ldg(up + ts + j) : 0.0;
    }
    mbar_wait(ubar, uphase);
    double uu[SL];
#pragma unroll
    for (int j = 0; j < SL; j += 2) {
        const double2 t2 = reinterpret_cast<const double2*>(slot)[j >> 1];
        uu[j] = t2.x;
        uu[j + 1] = t2.y;
    }
    // ---- A: forward from zero ---------------------------------------------------------------------------------------
    double z[D];
#pragma unroll
    for (int q = 0; q < D; ++q) z[q] = 0.0;
#pragma unroll
    for (int j = 0; j < SL; ++j) {
        if (INTERIOR || j < len) {
            double zn[D];
            mv<D>(c.M, z, zn);
#pragma unroll
            for (int q = 0; q < D; ++q) z[q] = fma(c.K[q], uu[j], zn[q]);
        }
    }
#pragma unroll
    for (int q = 0; q < D; ++q) exch[s][li][q] = z[q];
    __syncthreads();
    double x[D];
#pragma unroll
    for (int q = 0; q < D; ++q) x[q] = x_chunk[q];
    for (int k = 0; k < s; ++k) {                    // sub-chunks before s are complete (32 steps) whenever s has any step
        double xn[D];
        mv<D>(PM, x, xn);
#pragma unroll
        for (int q = 0; q < D; ++q) x[q] = xn[q] + exch[k][li][q];
    }
    // ---- B: forward from the true carry ---------------------------------------------------------------------------
    double vsq = 0.0;
#pragma unroll
    for (int j = 0; j < SL; ++j) {
        if (INTERIOR || j < len) {
            double hax = c.HA[0] * x[0];
#pragma unroll
            for (int q = 1; q < D; ++q) hax = fma(c.HA[q], x[q], hax);
            const double v = uu[j] - hax;                                   // ihgp.h:206 (pre-step state)
            vsq = fma(v, v, vsq);
            if (vrow) vrow[j] = v * v;
            double xn[D];
            mv<D>(c.M, x, xn);
#pragma unroll
            for (int q = 0; q < D; ++q) x[q] = fma(c.K[q], uu[j], xn[q]);   // ihgp.h:90
            if (D == 2) {
                reinterpret_cast<double2*>(tile)[j * NT + tid] = make_double2(x[0], x[1]);
            } else {
#pragma unroll
                for (int q = 0; q < D; ++q) tile[(q * SL + j) * NT + tid] = x[q];
            }
            if (Xg) {
                double* dst = Xg + (size_t)j * gstride;
                if (D == 2 && vec_x) *reinterpret_cast<double2*>(dst) = make_double2(x[0], x[1]);
                else {
#pragma unroll
                    for (int q = 0; q < D; ++q) dst[q] = x[q];
                }
            }
        }
    }
    if (xT_dst && !INTERIOR && len > 0 && ts + len == T) {
#pragma unroll
        for (int q = 0; q < D; ++q) xT_dst[q] = x[q];
    }
    // fixed-order reduction of sum v^2 over the chunk's sub-chunks
    vred[s][li] = vsq;
    asm volatile("" ::: "memory");                    // X comes back from shared memory, not from 64 live registers
    // ---- the step after this thread's last one (drive of the backward recursion at j = SL - 1) --------------------
    double v_next = 0.0, X_next[D];
    if (MODE == 1) {
        double hax = c.HA[0] * x[0];
#pragma unroll
        for (int q = 1; q < D; ++q) hax = fma(c.HA[q], x[q], hax);
        v_next = u_nx - hax;
    } else {
        double xn[D];
        mv<D>(c.M, x, xn);
#pragma unroll
        for (int q = 0; q < D; ++q) X_next[q] = fma(c.K[q], u_nx, xn[q]);
    }
    auto tile_load = [&](int j, double (&o)[D]) {
        if (D == 2) {
            const double2 t2 = reinterpret_cast<const double2*>(tile)[j * NT + tid];
            o[0] = t2.x;
            o[1] = t2.y;
        } else {
#pragma unroll
            for (int q = 0; q < D; ++q) o[q] = tile[(q * SL + j) * NT + tid];
        }
    };
    // one step of b[j] = G b[j+1] + g[j]  (drives as in chunk_pass above); Xj = X[j], Xn = X[j+1] (literal mode)
    auto back_step = [&](int j, const double (&Xj)[D], const double (&Xn)[D], double (&b)[D]) {
        const long long t = ts + j;
        double g[D];
        if (MODE == 1) {
            double vn;
            if (j + 1 < SL) {
                double hax = c.HA[0] * Xj[0];
#pragma unroll
                for (int q = 1; q < D; ++q) hax = fma(c.HA[q], Xj[q], hax);
                vn = uu[(j + 1) % SL] - hax;
            } else vn = v_next;
            const double sgn = (INTERIOR || t < T - 1) ? vn : 0.0;
#pragma unroll
            for (int q = 0; q < D; ++q) g[q] = c.drv[q] * sgn;
        } else {
            double im[D];
            mv<D>(c.drv, Xn, im);
#pragma unroll
            for (int q = 0; q < D; ++q) g[q] = (INTERIOR || t < T - 1) ? im[q] : Xj[q];
        }
        double bn[D];
        mv<D>(c.G, b, bn);
#pragma unroll
        for (int q = 0; q < D; ++q) b[q] = bn[q] + g[q];
    };
    // ---- C: backward from zero ----------------------------------------------------------------------------------------
    double b[D], Xn[D];
#pragma unroll
    for (int q = 0; q < D; ++q) { b[q] = 0.0; Xn[q] = X_next[q]; }
#pragma unroll
    for (int j = SL - 1; j >= 0; --j) {
        if (INTERIOR || j < len) {
            double Xj[D];
            tile_load(j, Xj);
            back_step(j, Xj, Xn, b);
#pragma unroll
            for (int q = 0; q < D; ++q) Xn[q] = Xj[q];
        }
    }
    __syncthreads();                                  // everyone is done reading the forward summaries
#pragma unroll
    for (int q = 0; q < D; ++q) exch[s][li][q] = b[q];
    __syncthreads();
    if (vsq_dst && s == 0) {
        double a = vred[0][li];
#pragma unroll
        for (int k = 1; k < NSUBC; ++k) a += vred[k][li];
        *vsq_dst = a;
    }
#pragma unroll
    for (int q = 0; q < D; ++q) b[q] = b_chunk[q];
    for (int k = NSUBC - 1; k > s; --k) {
        double bn[D];
        mv<D>(PG, b, bn);
#pragma unroll
        for (int q = 0; q < D; ++q) b[q] = bn[q] + exch[k][li][q];
    }
    // ---- D: backward from the true carry ------------------------------------------------------------------------------
#pragma unroll
    for (int q = 0; q < D; ++q) Xn[q] = X_next[q];
#pragma unroll
    for (int j = SL - 1; j >= 0; --j) {
        if (INTERIOR || j < len) {
            double Xj[D];
            tile_load(j, Xj);
            back_step(j, Xj, Xn, b);
#pragma unroll
            for (int q = 0; q < D; ++q) Xn[q] = Xj[q];
            if (Xsg) {
                double o[D];
#pragma unroll
                for (int q = 0; q < D; ++q) o[q] = MODE == 1 ? Xj[q] + b[q] : b[q];
                double* dst = Xsg + (size_t)j * gstride;
                if (D == 2 && vec_x) *reinterpret_cast<double2*>(dst) = make_double2(o[0], o[1]);
                else {
#pragma unroll
                    for (int q = 0; q < D; ++q) dst[q] = o[q];
                }
            }
        }
    }
    __syncthreads();                                  // exch / vred are reused by the next chunk
}

// grid: N * nG * (L / LG) CTAs (latent-group minor), block: NSUBC * LG threads; CTA (n, g, latent group) walks cpc chunks.
template <int D, int MODE, int LG>
__global__ void __launch_bounds__(NSUBC * LG, (D == 2 ? 384 : 256) / (NSUBC * LG)) k_scan_lanes(const double* __restrict__ u, const LatentConsts* __restrict__ consts,
                                                          int L, long long N, long long T, long long nC, long long cpc,
                                                          const double* __restrict__ xin, const double* __restrict__ bin,
                                                          double* __restrict__ X, double* __restrict__ Xs,
                                                          double* __restrict__ vsq_out, double* __restrict__ xT,
                                                          const double* __restrict__ u_after, int seq_end, double* __restrict__ vstep) {
    extern __shared__ double tile[];                  // the CTA's filtered states: [SL][NT] double2 (D = 2) or [D][SL][NT]
    __shared__ double exch[NSUBC][LG][D];
    __shared__ double vred[NSUBC][LG];
    __shared__ unsigned long long ubar;               // completion of the chunk's u copies (one phase per chunk)
    const int tid = threadIdx.x, s = tid / LG, li = tid % LG;
    if (tid == 0) {
        mbar_init(&ubar, NSUBC * LG);
        mbar_fence_init();
    }
    __syncthreads();
    const int nLG = L / LG;
    const long long nG = (nC + cpc - 1) / cpc;
    const long long bid = blockIdx.x;
    const int lgi = (int)(bid % nLG);
    const long long gi = (bid / nLG) % nG;
    const long long n = bid / ((long long)nLG * nG);
    const int l = lgi * LG + li;
    const LatentConsts* lc = consts + l;
    LC<D> cst;
    load_lc<D, MODE>(lc, cst);
    double PM[D * D], PG[D * D];
    load_mat<D>(lc->powM[LOG2_SL], PM);
    load_mat<D>(lc->powG[MODE][LOG2_SL], PG);
    const double* up = u + ((size_t)n * L + l) * T;
    const size_t gstride = (size_t)L * D;
    const bool vec_x = D == 2 && (reinterpret_cast<size_t>(X) & 15) == 0 && (reinterpret_cast<size_t>(Xs) & 15) == 0;
    const long long c_lo = gi * cpc, c_hi = min(nC, c_lo + cpc);
    for (long long c = c_lo; c < c_hi; ++c) {
        const long long ts = c * CH + (long long)s * SL;
        const size_t ci = (((size_t)n * L + l) * nC + c) * D;
        double x_chunk[D], b_chunk[D];
#pragma unroll
        for (int q = 0; q < D; ++q) { x_chunk[q] = xin[ci + q]; b_chunk[q] = bin[ci + q]; }
        const size_t go = ((size_t)n * T + ts) * gstride + (size_t)l * D;
        double* Xg = X ? X + go : nullptr;
        double* Xsg = Xs ? Xs + go : nullptr;
        double* vdst = vsq_out + ((size_t)c * N + n) * L + l;
        double* xTd = xT ? xT + ((size_t)n * L + l) * D : nullptr;
        double* vrow = vstep ? vstep + ((size_t)n * L + l) * T + ts : nullptr;
        // the step after this thread's last one: in the block, or the next block's first (sequence sharded in time)
        const double u_nx = ts + SL < T ? __ldg(up + ts + SL) : (u_after ? __ldg(u_after + (size_t)n * L + l) : 0.0);
        if (c * CH + CH < T || !seq_end)
            lanes_chunk<D, MODE, LG, true>(cst, PM, PG, up, u_nx, ts, T, s, li, tid, x_chunk, b_chunk, tile, &ubar, (unsigned)((c - c_lo) & 1), exch, vred, Xg, Xsg, gstride, vec_x, vdst, xTd, vrow);
        else
            lanes_chunk<D, MODE, LG, false>(cst, PM, PG, up, u_nx, ts, T, s, li, tid, x_chunk, b_chunk, tile, &ubar, (unsigned)((c - c_lo) & 1), exch, vred, Xg, Xsg, gstride, vec_x, vdst, xTd, vrow);
    }
}

template <int D, int MODE, int LG>
cudaError_t launch_scan_lanes(const ScanArgs& a, long long nC, cudaStream_t st) {
    constexpr int NT = NSUBC * LG;
    const size_t smem = sizeof(double) * D * SL * NT;
    static std::atomic<int> attr_done[64];
    if (AttrOnce once(attr_done); once) {
        cudaError_t e = cudaFuncSetAttribute(k_scan_lanes<D, MODE, LG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const int nLG = a.L / LG;
    const long long target = 148LL * 96;           // swept 6 .. 192 on config 4: flat, 96 best by 1 % (profiles/r02)
    const long long cpc = chunks_per_group(a.N * nLG, nC, target);
    const long long nG = (nC + cpc - 1) / cpc;
    k_scan_lanes<D, MODE, LG><<<(unsigned)(a.N * nG * nLG), NT, smem, st>>>(a.u, a.consts, a.L, a.N, a.T, nC, cpc, a.xin, a.bin, a.X, a.Xs,
                                                                            a.vsq, a.xT, a.u_after, a.seq_end, a.vstep);
    return cudaGetLastError();
}

template <int D, int MODE>
cudaError_t run_scan(const ScanArgs& a, cudaStream_t st) {
    const long long nC = (a.T + CH - 1) / CH;
    const int nLG = (a.L + LGMAX - 1) / LGMAX;
    const int lg = a.L < LGMAX ? a.L : LGMAX;
    const long long r_last = a.T - (nC - 1) * CH;
    const int RS = lg * D;
    const size_t smem = sizeof(double) * 2 * 32 * (size_t)tile_group_stride(RS);
    if (smem > 48 * 1024) {
        cudaFuncSetAttribute(k_scan<D, MODE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    const long long target = 148LL * 16;           // swept 4 .. 128 on config 4: 16 and above are equal, below it the machine is not filled
    // Phases (a.phase): 0 = the whole pass.  A block of a longer sequence sharded in time runs 1 (summaries + forward
    // chain from a.x0 -> x_end), 2 (last-chunk summary with the true u_after, forward chain from the true x0, backward
    // chain from b_end = 0 -> b_out) and 3 (backward chain from the true b_end + the final pass); the carries of the
    // blocks are exchanged between the phases (capi.cu, multioutputihgp_b200/parallel.py).
    const int ph = a.phase;
    const bool sharded = ph != 0;
    if (ph <= 1 && (nC > 1 || sharded)) {
        // summaries: interior chunks as dot products with tabulated weights, the last chunk by the recurrence itself
        k_scan_weights<D, MODE><<<a.L * (CH + 1), 32, 0, st>>>(a.consts, a.Wsum);
        const long long nI = nC - 1;
        if (nI > 0) {
            const long long cpw = chunks_per_group(a.N * a.L, nI, target);
            const long long warps = a.N * a.L * ((nI + cpw - 1) / cpw);
            k_scan_summaries_dot<D><<<(unsigned)((warps + 3) / 4), 128, 0, st>>>(a.u, a.Wsum, a.L, a.N, a.T, nC, cpw, a.fsum, a.bsum);
        }
    }
    if ((ph == 0 && nC > 1) || ph == 1 || ph == 2) {
        k_scan<D, MODE, false><<<(unsigned)(a.N * nLG), 32 * lg, 0, st>>>(a.u, a.consts, a.L, a.N, a.T, nC, nLG, nC - 1, 1, 1, nullptr, nullptr,
                                                                         a.fsum, a.bsum, nullptr, nullptr, nullptr, nullptr, a.u_after, a.seq_end, nullptr);
        mark(a.mk, "k_scan_summaries");
    }
    if ((ph == 0 && nC > 1) || ph == 2) {
        k_response<D, MODE><<<a.L * 2 * D, 32, 0, st>>>(a.consts, r_last, a.Bx);
        mark(a.mk, "k_response");
    }
    {
        const long long nGr = (nC + 32 * CG - 1) / (32 * CG), nS = (nGr + SB - 1) / SB;
        const unsigned gw = (unsigned)((a.N * a.L * nS * 32 + 127) / 128), gt = (unsigned)((a.N * a.L + 127) / 128);
        const double* in = nullptr;
        if (ph <= 2) {
            if (nS > 1) {
                k_carry<D, MODE, 0, 0><<<gw, 128, 0, st>>>(a.consts, a.Bx, a.L, a.N, nC, nS, a.x0, a.fsum, a.bsum, a.xin, a.bin, nullptr, a.sb_end, nullptr, a.seq_end);
                k_carry_super<D, MODE, 0><<<gt, 128, 0, st>>>(a.consts, a.L, a.N, nS, a.x0, a.sb_end, a.sb_in);
                in = a.sb_in;
            }
            k_carry<D, MODE, 0, 1><<<gw, 128, 0, st>>>(a.consts, a.Bx, a.L, a.N, nC, nS, a.x0, a.fsum, a.bsum, a.xin, a.bin, in, nullptr, nullptr, a.seq_end);
        }
        if (ph == 1) {
            if (a.x_end) k_block_end<D><<<gt, 128, 0, st>>>(a.consts, a.L, a.N, nC, a.xin, a.fsum, a.x_end);
            mark(a.mk, "k_carry");
            return cudaGetLastError();
        }
        if (nS > 1) {
            k_carry<D, MODE, 1, 0><<<gw, 128, 0, st>>>(a.consts, a.Bx, a.L, a.N, nC, nS, a.x0, a.fsum, a.bsum, a.xin, a.bin, nullptr, a.sb_end, a.b_end, a.seq_end);
            k_carry_super<D, MODE, 1><<<gt, 128, 0, st>>>(a.consts, a.L, a.N, nS, a.x0, a.sb_end, a.sb_in);
            in = a.sb_in;
        }
        k_carry<D, MODE, 1, 1><<<gw, 128, 0, st>>>(a.consts, a.Bx, a.L, a.N, nC, nS, a.x0, a.fsum, a.bsum, a.xin, a.bin, in, nullptr, a.b_end, a.seq_end);
        if (a.b_out) k_block_start<D, MODE><<<gt, 128, 0, st>>>(a.consts, a.Bx, a.L, a.N, nC, a.seq_end, a.xin, a.bsum, a.bin, a.b_out);
    }
    mark(a.mk, "k_carry");
    if (ph == 2) return cudaGetLastError();
    // final pass: thread-per-sub-chunk kernel when the latents come in whole groups of 16 or 8, else the warp-per-chunk one
    if (a.L % 8 == 0) {
        const cudaError_t e = a.L % 16 == 0 ? launch_scan_lanes<D, MODE, 16>(a, nC, st) : launch_scan_lanes<D, MODE, 8>(a, nC, st);
        mark(a.mk, "k_scan_final");
        return e;
    }
    const long long cpc = chunks_per_group(a.N * nLG, nC, target);
    const long long nG = (nC + cpc - 1) / cpc;
    k_scan<D, MODE, true><<<(unsigned)(a.N * nG * nLG), 32 * lg, smem, st>>>(a.u, a.consts, a.L, a.N, a.T, nC, nLG, 0, nC, cpc, a.xin, a.bin,
                                                                            nullptr, nullptr, a.X, a.Xs, a.vsq, a.xT, a.u_after, a.seq_end, a.vstep);
    mark(a.mk, "k_scan_final");
    return cudaGetLastError();
}

}  // namespace

size_t scan_chunks(long long T) { return (size_t)((T + CH - 1) / CH); }

int scan_launch_count(long long T) {
    const long long nC = (T + CH - 1) / CH, nS = ((nC + 32 * CG - 1) / (32 * CG) + SB - 1) / SB;
    return (nC > 1 ? 5 : 1) + (nS > 1 ? 6 : 2);
}

size_t scan_superblocks(long long T) { const long long nC = (T + CH - 1) / CH; return (size_t)(((nC + 32 * CG - 1) / (32 * CG) + SB - 1) / SB); }

size_t scan_weights_doubles(int L) { return (size_t)L * WS_STRIDE; }

cudaError_t launch_scan(int dim, int mode, const ScanArgs& a, cudaStream_t st) {
    if (dim == 2) return mode == 0 ? run_scan<2, 0>(a, st) : run_scan<2, 1>(a, st);
    return mode == 0 ? run_scan<3, 0>(a, st) : run_scan<3, 1>(a, st);
}

cudaError_t launch_nll_reduce(const double* rho_part, const double* vsq, const LatentConsts* consts, const double* S, double sigma,
                              int p, int L, long long N, long long T, double* part, double* nll, cudaStream_t st) {
    const long long nC = (T + CH - 1) / CH;
    const long long tiles = (long long)project_tiles(T);
    const int nsplit = nll_nsplit(N);
    k_nll_partial<<<(unsigned)(N * nsplit), 256, 0, st>>>(rho_part, vsq, consts, sigma, L, N, tiles, nC, nsplit, part);
    k_nll_reduce<<<(unsigned)((N * 32 + 127) / 128), 128, 0, st>>>(part, consts, S, sigma, p, L, N, T, nsplit, nll);
    return cudaGetLastError();
}

size_t nll_partials(long long N) { return (size_t)N * nll_nsplit(N); }

cudaError_t launch_nll_steps(const double* vstep, const LatentConsts* consts, const double* S, double sigma, int p, int L, long long N,
                             long long T, double* nll_steps, cudaStream_t st) {
    k_nll_steps<<<(unsigned)((N * T + 255) / 256), 256, 0, st>>>(vstep, consts, S, sigma, p, L, N, T, nll_steps);
    return cudaGetLastError();
}

// ---- one long sequence sharded in TIME (moihgp_cuda_fsn_block_*): the two carry exchanges on the device ----------------
// forward  (DIR 0): gathered[g][n][l][D + 1] = [end state of block g from a zero carry-in | first projected observation of g];
//                   x_in(g+1) = AKHA^n_g x_in(g) + x_end_g chained over g < rank from x0 -> out[n][l][D];
//                   u_after[n][l] = first observation of block rank + 1 (untouched on the last block)
// backward (DIR 1): gathered[g][n][l][D] = backward value at block g's first step from a ZERO b_end;
//                   b_start(G-1) = gathered[G-1], b_start(g) = gathered[g] + G^n_g b_start(g+1); out = b_start(rank + 1)
//                   (untouched on the last block, whose b_end is not used)
// Powers by binary powering on the latent's 2^k tables (mat_pow).  One thread per (sequence, latent) - the arithmetic of
// parallel.forward_carry_in / backward_carry_in.
struct FsnBlockLens { long long n[64]; };

template <int D>
__global__ void __launch_bounds__(128) k_fsn_carry(const LatentConsts* __restrict__ consts, int L, long long N, int rank, int G, int dir, int mode,
                                                  FsnBlockLens lens, const double* __restrict__ gathered, const double* __restrict__ x0,
                                                  double* __restrict__ out, double* __restrict__ u_after) {
    const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= N * L) return;
    const LatentConsts& c = consts[id % L];
    const double (*tab)[9] = dir == 0 ? c.powM : c.powG[mode];  // M = AKHA (forward) or G[mode] (backward)
    double P[D * D];
    long long have = -1;
    auto power = [&](long long n) {                       // P = M^n
        if (n == have) return;
        mat_pow<D>(tab, n, P);
        have = n;
    };
    double v[D];
    if (dir == 0) {
        const int W = D + 1;
#pragma unroll
        for (int q = 0; q < D; ++q) v[q] = x0 ? x0[id * D + q] : 0.0;
        for (int g = 0; g < rank; ++g) {
            power(lens.n[g]);
            const double* e = gathered + ((size_t)g * N * L + id) * W;
            double vn[D];
#pragma unroll
            for (int i = 0; i < D; ++i) {
                double a = 0.0;
#pragma unroll
                for (int q = 0; q < D; ++q) a += P[i * D + q] * v[q];
                vn[i] = a + e[i];
            }
#pragma unroll
            for (int i = 0; i < D; ++i) v[i] = vn[i];
        }
#pragma unroll
        for (int q = 0; q < D; ++q) out[id * D + q] = v[q];
        if (u_after && rank + 1 < G) u_after[id] = gathered[((size_t)(rank + 1) * N * L + id) * W + D];
    } else {
        if (rank >= G - 1) return;
        const double* e = gathered + ((size_t)(G - 1) * N * L + id) * D;
#pragma unroll
        for (int q = 0; q < D; ++q) v[q] = e[q];
        for (int g = G - 2; g > rank; --g) {
            power(lens.n[g]);
            e = gathered + ((size_t)g * N * L + id) * D;
            double vn[D];
#pragma unroll
            for (int i = 0; i < D; ++i) {
                double a = 0.0;
#pragma unroll
                for (int q = 0; q < D; ++q) a += P[i * D + q] * v[q];
                vn[i] = e[i] + a;
            }
#pragma unroll
            for (int i = 0; i < D; ++i) v[i] = vn[i];
        }
#pragma unroll
        for (int q = 0; q < D; ++q) out[id * D + q] = v[q];
    }
}

cudaError_t launch_fsn_carry(int dim, int direction, int mode, const LatentConsts* consts, int L, long long N, int rank, int G,
                             const long long* block_lengths, const double* gathered, const double* x0, double* out, double* u_after,
                             cudaStream_t st) {
    if (G < 1 || G > 64 || rank < 0 || rank >= G) return cudaErrorInvalidValue;
    FsnBlockLens lens;
    for (int g = 0; g < 64; ++g) lens.n[g] = g < G ? block_lengths[g] : 0;
    const unsigned grid = (unsigned)((N * L + 127) / 128);
    if (dim == 3) k_fsn_carry<3><<<grid, 128, 0, st>>>(consts, L, N, rank, G, direction, mode, lens, gathered, x0, out, u_after);
    else k_fsn_carry<2><<<grid, 128, 0, st>>>(consts, L, N, rank, G, direction, mode, lens, gathered, x0, out, u_after);
    return cudaGetLastError();
}

}  // namespace moihgp
