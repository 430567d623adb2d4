// K-objective: negative log-likelihood and its hyper-parameter gradient over whole sequences (sm_100a).
//
// Replaces the per-observation loop of RegressionObjective::operator() (moihgp_regression.h:42-50)
// and OnlineObjective::operator() (moihgp_online.h:61-70):
//     for each y_t:  MOIHGP::step v2 (moihgp.h:229-301)  +  MOIHGP::negLogLikelihood(x, y, dx, grad) (moihgp.h:460-611)
// i.e. per latent the sensitivity recursion ihgp.h:60-78
//     x+ = AKHA x + K u,      dx_k+ = dAKHA_k x + AKHA dx_k + dK_k u
// and the per-step loss / gradient ihgp.h:212-222, with the mixing terms of moihgp.h:499-609.
//
// The reference's O(p^3 L^2)-per-step dU loop (moihgp.h:538-552) is the rank-1 update
// y_r * ( -(U'y)_c / sigma + pv_c / sqrt(S_c) ) (SURVEY.md section 0; oracle test_rank1), so summed over
// time it is ONE dense contraction  dU = Y' W  (k_gradU, split over time and reduced in fixed order).
//
// Scan structure: as scan.cu.  The dx_k chains are LTI recurrences with the SAME transition AKHA
// and a drive dAKHA_k x_t + dK_k u_t that depends on the true filtered state, so inside a warp
// the x chain is resolved first and each dx_k chain is then scanned with the same AKHA powers;
// across chunks the coupling is the constant matrix E_k = sum_i AKHA^(CH-1-i) dAKHA_k AKHA^i.
//
// Quirks kept for parity (SURVEY.md section 9): Q5 (per-latent loss terms only when `threading`),
// Q8 (pv uses the RAW y(l)), Q9 (norm not squared; 1/2 log(sum S)), Q20 (dv_k uses HdA_k(0) x(0)).
#include <cuda_runtime.h>
#include <math.h>
#include "moihgp_device.cuh"
#include "small_mat.cuh"
#include "ptx.cuh"
#include "launch.h"

namespace moihgp {

namespace {

constexpr int SUB = 8;
constexpr int CH = 32 * SUB;
constexpr int LOG2_SUB = 3;
constexpr int LOG2_CH = 8;
constexpr unsigned FULL = 0xffffffffu;
constexpr int NPART = 8;          // per-chunk partial sums: loss, g0, g1, g2, pv*w (3 spare)


// Warp-level LTI scan  z+ = M z + r_i  over this lane's SUB steps: returns, per step, the state BEFORE
// the step (pre[i]) and the lane's end state after the inclusive scan (z_end; lane 31 = chunk end).
template <int D>
__device__ __forceinline__ void lti_scan(const double (&M)[D * D], const double* __restrict__ pw /*[5][D*D]: M^(SUB 2^k)*/,
                                         const double (&r)[SUB][D], const double (&z_in)[D], int lane, double (&pre)[SUB][D],
                                         double (&z_end)[D]) {
    double z[D];
#pragma unroll
    for (int q = 0; q < D; ++q) z[q] = lane == 0 ? z_in[q] : 0.0;
#pragma unroll
    for (int i = 0; i < SUB; ++i) {
        double zn[D];
        mv<D>(M, z, zn);
#pragma unroll
        for (int q = 0; q < D; ++q) z[q] = zn[q] + r[i][q];
    }
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
    for (int q = 0; q < D; ++q) z_end[q] = z[q];
    double x[D];
#pragma unroll
    for (int q = 0; q < D; ++q) {
        const double up = __shfl_up_sync(FULL, z[q], 1);
        x[q] = lane == 0 ? z_in[q] : up;
    }
#pragma unroll
    for (int i = 0; i < SUB; ++i) {
#pragma unroll
        for (int q = 0; q < D; ++q) pre[i][q] = x[q];
        double xn[D];
        mv<D>(M, x, xn);
#pragma unroll
        for (int q = 0; q < D; ++q) x[q] = xn[q] + r[i][q];
    }
}

// grid: N * L * nG warps, 4 warps per CTA; warp (n, l, g) walks the chunks g * cpw ... (cpw chunks, fewer for the last
// group): the latent's constants and scan powers are loaded once per warp, not once per chunk.
template <int D, bool FINAL>
__global__ void __launch_bounds__(128, 3) k_obj_scan(const double* __restrict__ u, const double* __restrict__ w,
                                                 const double* __restrict__ yl, const LatentConsts* __restrict__ consts,
                                                 const double* __restrict__ S, double sigma, int L, long long N, long long T,
                                                 long long nC, long long c_base, long long c_cnt, long long cpw,
                                                 const double* __restrict__ zin, double* __restrict__ zsum,
                                                 double* __restrict__ wgt, double* __restrict__ part,
                                                 double* __restrict__ xT, double* __restrict__ dxT) {
    const int lane = threadIdx.x & 31;
    __shared__ double pws[4][5 * D * D];
    const long long nG = (c_cnt + cpw - 1) / cpw;
    const long long wid0 = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
    const bool live = wid0 < N * L * nG;
    const long long wid = live ? wid0 : 0;
    const long long g = wid % nG;
    const int l = (int)((wid / nG) % L);
    const long long n = wid / (nG * L);
    const LatentConsts* lc = consts + l;
    {
        double* pwm = pws[threadIdx.x >> 5];
        for (int i = lane; i < 5 * D * D; i += 32) {
            const int m = i / (D * D), e = i - m * (D * D);
            pwm[i] = lc->powM[LOG2_SUB + m][(e / D) * 3 + (e % D)];
        }
        __syncwarp();
    }
    if (!live) return;
    const double* pw = pws[threadIdx.x >> 5];
    const size_t so = ((size_t)n * L + l) * T;
    double M[D * D], K[D], HA[D];
    load_mat<D>(lc->AKHA, M);
    load_vec<D>(lc->K, K);
    load_vec<D>(lc->HA, HA);
    const long long c_lo = c_base + g * cpw, c_hi = min(c_base + c_cnt, c_lo + cpw);
  for (long long c = c_lo; c < c_hi; ++c) {
    const long long tf = c * CH + (long long)lane * SUB;
    // this lane's 8 consecutive steps: 16-byte loads when the run is whole and aligned (T even or an aligned row start)
    const bool vec = tf + SUB <= T && (((so + tf) & 1) == 0) && ((reinterpret_cast<size_t>(u) & 15) == 0) &&
                     ((reinterpret_cast<size_t>(w) & 15) == 0) && ((reinterpret_cast<size_t>(yl) & 15) == 0) &&
                     (wgt == nullptr || (reinterpret_cast<size_t>(wgt) & 15) == 0);
    auto load8 = [&](const double* src, double (&dst)[SUB]) {
        if (vec) {
#pragma unroll
            for (int i = 0; i < SUB; i += 2) {
                const double2 t2 = __ldg(reinterpret_cast<const double2*>(src + so + tf + i));
                dst[i] = t2.x;
                dst[i + 1] = t2.y;
            }
        } else {
#pragma unroll
            for (int i = 0; i < SUB; ++i) dst[i] = tf + i < T ? __ldg(src + so + tf + i) : 0.0;
        }
    };
    double uu[SUB];
    load8(u, uu);

    const size_t ci = (((size_t)n * L + l) * nC + c) * 4 * D;     // carries are chunk-minor: [n][l][chunk][4*D]
    double zi[4][D];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int q = 0; q < D; ++q) zi[a][q] = FINAL ? zin[ci + a * D + q] : 0.0;

    // ---- x chain ----------------------------------------------------------------------------------
    double r[SUB][D], xpre[SUB][D], zend[D];
#pragma unroll
    for (int i = 0; i < SUB; ++i)
#pragma unroll
        for (int q = 0; q < D; ++q) r[i][q] = K[q] * uu[i];
    lti_scan<D>(M, pw, r, zi[0], lane, xpre, zend);
    if (!FINAL && lane == 31) {
#pragma unroll
        for (int q = 0; q < D; ++q) zsum[ci + q] = zend[q];
    }
    const bool last_lane = FINAL && (T - 1 >= tf && T - 1 < tf + SUB);    // this lane owns step T-1
    const int ilast = (int)(T - 1 - tf);
    if (last_lane && xT) {
        // state after step T-1: one more literal step from the pre-step state
#pragma unroll
        for (int i = 0; i < SUB; ++i)
            if (i == ilast) {
                double xn[D];
                mv<D>(M, xpre[i], xn);
#pragma unroll
                for (int q = 0; q < D; ++q) xT[((size_t)n * L + l) * D + q] = xn[q] + r[i][q];
            }
    }

    double v[SUB];
    double acc_loss = 0.0, acc_g[3] = {0.0, 0.0, 0.0}, acc_pvw = 0.0;
    const double Si = __ldg(&lc->S), logSi = __ldg(&lc->logS), hak = __ldg(&lc->hak);
    if (FINAL) {
        const double Sl = __ldg(S + l);
        const double rsS = 1.0 / sqrt(Sl);
        double ww[SUB], yy[SUB], wg[SUB];
        load8(w, ww);
        load8(yl, yy);
#pragma unroll
        for (int i = 0; i < SUB; ++i) {
            double hax = HA[0] * xpre[i][0];
#pragma unroll
            for (int q = 1; q < D; ++q) hax = fma(HA[q], xpre[i][q], hax);
            v[i] = uu[i] - hax;                                                     // ihgp.h:214
            const double pv = (yy[i] - hax) * (1 - hak) / Si;                       // moihgp.h:510-511 (raw y(l), Q8)
            wg[i] = -ww[i] / sigma + pv * rsS;                                      // moihgp.h:546-550 (rank-1 form)
            if (tf + i < T) {
                acc_loss += 0.5 * (v[i] * v[i] / Si + logSi);                       // ihgp.h:215
                acc_pvw = fma(pv, ww[i], acc_pvw);                                  // moihgp.h:558-560
            }
        }
        if (vec) {
#pragma unroll
            for (int i = 0; i < SUB; i += 2) *reinterpret_cast<double2*>(wgt + so + tf + i) = make_double2(wg[i], wg[i + 1]);
        } else {
#pragma unroll
            for (int i = 0; i < SUB; ++i)
                if (tf + i < T) wgt[so + tf + i] = wg[i];
        }
    }

    // ---- dx_k chains ------------------------------------------------------------------------------
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        double dM[D * D], dK[D], pre[SUB][D];
        load_mat<D>(lc->dAKHA[k], dM);
        load_vec<D>(lc->dK[k], dK);
#pragma unroll
        for (int i = 0; i < SUB; ++i) {
            double t1[D];
            mv<D>(dM, xpre[i], t1);
#pragma unroll
            for (int q = 0; q < D; ++q) r[i][q] = fma(dK[q], uu[i], t1[q]);         // ihgp.h:75
        }
        lti_scan<D>(M, pw, r, zi[1 + k], lane, pre, zend);
        if (!FINAL) {
            if (lane == 31) {
#pragma unroll
                for (int q = 0; q < D; ++q) zsum[ci + (1 + k) * D + q] = zend[q];
            }
        } else {
            const double hda0 = __ldg(&lc->HdA[k][0]), dSk = __ldg(&lc->dS[k]);
#pragma unroll
            for (int i = 0; i < SUB; ++i) {
                if (tf + i < T) {
                    double hd = HA[0] * pre[i][0];
#pragma unroll
                    for (int q = 1; q < D; ++q) hd = fma(HA[q], pre[i][q], hd);
                    const double dv = -hda0 * xpre[i][0] - hd;                      // ihgp.h:218 (Q20 de facto)
                    acc_g[k] += (v[i] * dv - 0.5 * (v[i] * v[i] / Si - 1) * dSk) / Si;   // ihgp.h:219
                }
            }
            if (last_lane && dxT) {
#pragma unroll
                for (int i = 0; i < SUB; ++i)
                    if (i == ilast) {
                        double xn[D];
                        mv<D>(M, pre[i], xn);
#pragma unroll
                        for (int q = 0; q < D; ++q) dxT[(((size_t)n * L + l) * 3 + k) * D + q] = xn[q] + r[i][q];
                    }
            }
        }
    }
    if (FINAL) {
        double s[5] = {acc_loss, acc_g[0], acc_g[1], acc_g[2], acc_pvw};
#pragma unroll
        for (int j = 0; j < 5; ++j)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s[j] += __shfl_xor_sync(FULL, s[j], o);
        if (lane == 0) {
            double* pp = part + (((size_t)c * N + n) * L + l) * NPART;
#pragma unroll
            for (int j = 0; j < 5; ++j) pp[j] = s[j];
        }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// k_obj_lanes: the same two passes with one THREAD per (latent, sub-chunk of SL = 32 steps) running the reference's
// loop (ihgp.h:60-78, :212-222) sequentially - no warp scans.  A CTA owns (sequence, LG latents, chunk of CH steps):
//   A  augmented state from zero over the sub-chunk                 -> summary f_s
//      carries across the sub-chunks: z <- Z^32 z + f_s with the span-32 coupling E_k(32) (built once per CTA)
//   FINAL = false: the chunk summary  Z^32 z_in(7) + f_7  -> zsum     (interior chunks only: all sub-chunks are whole)
//   FINAL = true : B  the literal recurrence from the true carry: per-step loss / gradient terms and the dU weights.
// Every thread's inputs (u in the summaries pass; U'y and raw y(l) in the final pass: 256-byte runs of the latent-major series) are brought into a private
// shared-memory slot by the copy engine (cp.async.bulk) and the dU weights leave the same way: no per-lane HBM
// instructions, no uncoalesced wavefronts.  ~115 FP64 instructions per latent-step (the warp-scan kernel: ~650).
constexpr int SL = 32;                 // steps per thread
constexpr int NSUBC = CH / SL;         // sub-chunks per chunk
constexpr int LOG2_SL = 5;
constexpr int UP3 = 2 * SL + 2;        // slot pitch in doubles of the final pass ([U'y -> dU weight | y(l)] + pad): UP3 / 2 odd => conflict-free
                                       // 16-byte loads.  u = S^-1/2 U'y is formed from U'y in the kernel (the same product k_project
                                       // forms, bit for bit): a third less shared memory per CTA = six instead of four CTAs per SM

template <int D>
struct ObjLC {
    double M[D * D], K[D], HA[D], dM[3][D * D], dK[3][D];
};

// z <- Z^32 z + f   on the augmented state [x; dx_0; dx_1; dx_2];  cp = [P = M^32 | E_0(32) | E_1(32) | E_2(32)]
template <int D>
__device__ __forceinline__ void advance32(const double* __restrict__ cp, const double* __restrict__ f, double (&z)[4][D]) {
    double P[D * D], zn[4][D];
#pragma unroll
    for (int i = 0; i < D * D; ++i) P[i] = cp[i];
    mv<D>(P, z[0], zn[0]);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        double E[D * D];
#pragma unroll
        for (int i = 0; i < D * D; ++i) E[i] = cp[(1 + k) * D * D + i];
        mv<D>(P, z[1 + k], zn[1 + k]);
        mv_acc<D>(E, z[0], zn[1 + k]);
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int q = 0; q < D; ++q) z[a][q] = zn[a][q] + f[a * D + q];
}

// one step of the augmented recurrence (ihgp.h:71-77): dx_k+ = dAKHA_k x + AKHA dx_k + dK_k u uses the PRE-step x
template <int D>
__device__ __forceinline__ void aug_step(const ObjLC<D>& c, double uj, double (&z)[4][D]) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        double t1[D], xn[D];
        mv<D>(c.dM[k], z[0], t1);
        mv<D>(c.M, z[1 + k], xn);
#pragma unroll
        for (int q = 0; q < D; ++q) z[1 + k][q] = xn[q] + fma(c.dK[k][q], uj, t1[q]);
    }
    double xn[D];
    mv<D>(c.M, z[0], xn);
#pragma unroll
    for (int q = 0; q < D; ++q) z[0][q] = xn[q] + c.K[q] * uj;
}

template <int D, int LG, bool FINAL>
__global__ void __launch_bounds__(NSUBC * LG) k_obj_lanes(const double* __restrict__ u, const double* __restrict__ w,
                                                         const double* __restrict__ yl, const LatentConsts* __restrict__ consts,
                                                         const double* __restrict__ S, double sigma, int L, long long N, long long T,
                                                         long long nC, long long c_cnt, long long cpc,
                                                         const double* __restrict__ zin, double* __restrict__ zsum,
                                                         double* zsub, double* __restrict__ wgt, double* __restrict__ part,
                                                         double* __restrict__ xT, double* __restrict__ dxT) {
    constexpr int NT = NSUBC * LG;
    constexpr int PITCH = FINAL ? UP3 : SL + 2;
    extern __shared__ double slots[];                 // [NT][PITCH]
    __shared__ __align__(16) double exch[NSUBC][LG][4 * D];   // sub-chunk summaries, then (FINAL) the partial sums of the sub-chunks
    __shared__ double cpl[LG][4 * D * D];
    __shared__ unsigned long long bar;
    const int tid = threadIdx.x, s = tid / LG, li = tid % LG;
    const int nLG = L / LG;
    const long long nG = (c_cnt + cpc - 1) / cpc;
    const long long bid = blockIdx.x;
    const int lgi = (int)(bid % nLG);
    const long long gi = (bid / nLG) % nG;
    const long long n = bid / ((long long)nLG * nG);
    const int l = lgi * LG + li;
    const LatentConsts* lc = consts + l;
    if (tid == 0) {
        mbar_init(&bar, NT);
        mbar_fence_init();
    }
    ObjLC<D> c;
    load_mat<D>(lc->AKHA, c.M);
    load_vec<D>(lc->K, c.K);
    load_vec<D>(lc->HA, c.HA);
#pragma unroll
    for (int k = 0; k < 3; ++k) { load_mat<D>(lc->dAKHA[k], c.dM[k]); load_vec<D>(lc->dK[k], c.dK[k]); }
    if (s == 0) {
        // span-32 transition of the augmented state: P = M^32 and E_k(32) by doubling, E(2n) = E(n) M^n + M^n E(n)
        double P[D * D];
        load_mat<D>(lc->powM[LOG2_SL], P);
#pragma unroll
        for (int i = 0; i < D * D; ++i) cpl[li][i] = P[i];
        for (int k = 0; k < 3; ++k) {
            double E[D * D];
#pragma unroll
            for (int i = 0; i < D * D; ++i) E[i] = c.dM[k][i];
            for (int lev = 0; lev < LOG2_SL; ++lev) {
                double Mn[D * D], a[D * D];
                load_mat<D>(lc->powM[lev], Mn);
#pragma unroll
                for (int i = 0; i < D; ++i)
#pragma unroll
                    for (int j = 0; j < D; ++j) {
                        double acc = 0.0;
#pragma unroll
                        for (int q = 0; q < D; ++q) acc += E[i * D + q] * Mn[q * D + j] + Mn[i * D + q] * E[q * D + j];
                        a[i * D + j] = acc;
                    }
#pragma unroll
                for (int i = 0; i < D * D; ++i) E[i] = a[i];
            }
#pragma unroll
            for (int i = 0; i < D * D; ++i) cpl[li][(1 + k) * D * D + i] = E[i];
        }
    }
    __syncthreads();
    const double Si = __ldg(&lc->S), logSi = __ldg(&lc->logS), hak = __ldg(&lc->hak);
    const double c1 = (1.0 - hak) / Si;                          // moihgp.h:510-511
    const double rsS = FINAL ? 1.0 / sqrt(__ldg(S + l)) : 0.0;
    const double rsig = 1.0 / sigma;
    double hda0[3], dSk[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { hda0[k] = __ldg(&lc->HdA[k][0]); dSk[k] = __ldg(&lc->dS[k]); }
    const size_t so = ((size_t)n * L + l) * T;
    const bool al = FINAL ? (((reinterpret_cast<size_t>(w) | reinterpret_cast<size_t>(yl) | reinterpret_cast<size_t>(wgt)) & 15) == 0)
                          : ((reinterpret_cast<size_t>(u) & 15) == 0);
    double* slot = slots + (size_t)tid * PITCH;
    const long long c_lo = gi * cpc, c_hi = min(c_cnt, c_lo + cpc);
    for (long long ch = c_lo; ch < c_hi; ++ch) {
        const long long ts = ch * CH + (long long)s * SL;
        const int len = (int)max(0LL, min((long long)SL, T - ts));
        const bool bulk = al && len == SL && (((so + ts) & 1) == 0);
        constexpr unsigned RUN = SL * (unsigned)sizeof(double);
        if (FINAL) bulk_wait_read<0>();               // the previous chunk's weight store has read this slot
        fence_async_smem();
        if (bulk) {
            mbar_expect_tx(&bar, FINAL ? 2 * RUN : RUN);
            bulk_g2s(slot, (FINAL ? w : u) + so + ts, RUN, &bar);
            if (FINAL) bulk_g2s(slot + SL, yl + so + ts, RUN, &bar);
        } else {
            for (int j = 0; j < SL; ++j) {
                slot[j] = j < len ? __ldg((FINAL ? w : u) + so + ts + j) : 0.0;
                if (FINAL) slot[SL + j] = j < len ? __ldg(yl + so + ts + j) : 0.0;
            }
            mbar_arrive(&bar);
        }
        const size_t ci = (((size_t)n * L + l) * nC + ch) * 4 * D;
        double z[4][D];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int q = 0; q < D; ++q) z[a][q] = FINAL ? zin[ci + a * D + q] : 0.0;
        mbar_wait(&bar, (unsigned)((ch - c_lo) & 1));
        // ---- A: from zero (FINAL: the summaries pass has already done it for the interior chunks) ---------------------
        double* zs = zsub ? zsub + ((((size_t)n * nC + ch) * NSUBC + s) * L + l) * 4 * D : nullptr;
        if (FINAL && zs && ch < nC - 1) {
#pragma unroll
            for (int e = 0; e < 4 * D; e += 2)
                *reinterpret_cast<double2*>(&exch[s][li][e]) = *reinterpret_cast<const double2*>(zs + e);
        } else {
            double f[4][D];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int q = 0; q < D; ++q) f[a][q] = 0.0;
            if (len == SL) {                          // whole sub-chunk: straight-line code
#pragma unroll 4
                for (int j = 0; j < SL; j += 2) {
                    const double2 u2 = reinterpret_cast<const double2*>(slot)[j >> 1];
                    aug_step<D>(c, FINAL ? u2.x * rsS : u2.x, f);                 // final pass: the slot holds U'y
                    aug_step<D>(c, FINAL ? u2.y * rsS : u2.y, f);
                }
            } else {
#pragma unroll 1
                for (int j = 0; j < len; ++j) aug_step<D>(c, FINAL ? slot[j] * rsS : slot[j], f);
            }
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int q = 0; q < D; ++q) exch[s][li][a * D + q] = f[a][q];
            if (!FINAL && zs) {
#pragma unroll
                for (int e = 0; e < 4 * D; e += 2)
                    *reinterpret_cast<double2*>(zs + e) = make_double2(f[e / D][e % D], f[(e + 1) / D][(e + 1) % D]);
            }
        }
        __syncthreads();
        for (int k = 0; k < s; ++k) advance32<D>(cpl[li], exch[k][li], z);
        if (!FINAL) {
            if (s == NSUBC - 1) {
                advance32<D>(cpl[li], exch[NSUBC - 1][li], z);
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int q = 0; q < D; ++q) zsum[ci + a * D + q] = z[a][q];
            }
            __syncthreads();
            continue;
        }
        // ---- B: the literal recurrence from the true carry ----------------------------------------------------------
        double sv2 = 0.0, svd[3] = {0.0, 0.0, 0.0}, spw = 0.0;
        // one step: loss / gradient terms on the PRE-step state, the dU weight, then the recurrence
        auto step_b = [&](double wj, double yj) -> double {
            const double uj = wj * rsS;                                              // moihgp.h:181, as k_project forms it
            double hax = c.HA[0] * z[0][0];
#pragma unroll
            for (int q = 1; q < D; ++q) hax = fma(c.HA[q], z[0][q], hax);
            const double v = uj - hax;                                               // ihgp.h:214
            const double pv = (yj - hax) * c1;                                       // moihgp.h:510-511 (raw y(l), Q8)
            sv2 = fma(v, v, sv2);
            spw = fma(pv, wj, spw);                                                  // moihgp.h:558-560
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                double hd = c.HA[0] * z[1 + k][0];
#pragma unroll
                for (int q = 1; q < D; ++q) hd = fma(c.HA[q], z[1 + k][q], hd);
                const double dv = -hda0[k] * z[0][0] - hd;                           // ihgp.h:218 (Q20 de facto)
                svd[k] = fma(v, dv, svd[k]);
            }
            aug_step<D>(c, uj, z);
            return fma(pv, rsS, -wj * rsig);                                         // moihgp.h:546-550 (rank-1 form)
        };
        if (len == SL) {                              // whole sub-chunk: straight-line code
#pragma unroll 2
            for (int j = 0; j < SL; j += 2) {
                const double2 w2 = reinterpret_cast<const double2*>(slot)[j >> 1];
                const double2 y2 = reinterpret_cast<const double2*>(slot + SL)[j >> 1];
                const double g0 = step_b(w2.x, y2.x);
                const double g1 = step_b(w2.y, y2.y);
                reinterpret_cast<double2*>(slot)[j >> 1] = make_double2(g0, g1);
            }
        } else {
#pragma unroll 1
            for (int j = 0; j < len; ++j) slot[j] = step_b(slot[j], slot[SL + j]);
        }
        if (len > 0 && ts + len == T) {                                              // this thread owns step T-1
            if (xT) {
#pragma unroll
                for (int q = 0; q < D; ++q) xT[((size_t)n * L + l) * D + q] = z[0][q];
            }
            if (dxT) {
#pragma unroll
                for (int k = 0; k < 3; ++k)
#pragma unroll
                    for (int q = 0; q < D; ++q) dxT[(((size_t)n * L + l) * 3 + k) * D + q] = z[1 + k][q];
            }
        }
        // the dU weights leave through the copy engine
        if (bulk) {
            fence_async_smem();
            bulk_s2g(wgt + so + ts, slot, RUN);
            bulk_commit();
        } else {
            for (int j = 0; j < len; ++j) wgt[so + ts + j] = slot[j];
        }
        // per-chunk partial sums (ihgp.h:215, :219), fixed order over the sub-chunks
        __syncthreads();                              // everyone is done with the forward summaries in exch
        {
            const double q2 = sv2 / Si;
            exch[s][li][0] = 0.5 * (q2 + (double)len * logSi);
#pragma unroll
            for (int k = 0; k < 3; ++k) exch[s][li][1 + k] = (svd[k] - 0.5 * (q2 - (double)len) * dSk[k]) / Si;
            exch[s][li][4] = spw;
        }
        __syncthreads();
        if (s == 0) {
            double* pp = part + (((size_t)ch * N + n) * L + l) * NPART;
#pragma unroll
            for (int jj = 0; jj < 5; ++jj) {
                double a = exch[0][li][jj];
#pragma unroll
                for (int k = 1; k < NSUBC; ++k) a += exch[k][li][jj];
                pp[jj] = a;
            }
        }
        __syncthreads();
    }
    if (FINAL) bulk_wait_read<0>();
}

template <int D, bool FINAL>
void launch_obj_lanes(const ObjArgs& a, long long nC, long long c_cnt, cudaStream_t st) {
    constexpr int LG = 8, NT = NSUBC * LG;
    const size_t smem = sizeof(double) * NT * (FINAL ? UP3 : SL + 2);
    static std::atomic<int> attr_done[64];
    if (AttrOnce once(attr_done); once)
        cudaFuncSetAttribute(k_obj_lanes<D, LG, FINAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int nLG = a.L / LG;
    const long long cpc = chunks_per_group(a.N * nLG, c_cnt, 148LL * 32);
    const long long nG = (c_cnt + cpc - 1) / cpc;
    k_obj_lanes<D, LG, FINAL><<<(unsigned)(a.N * nG * nLG), NT, smem, st>>>(a.u, a.w, a.yl, a.consts, a.S, a.sigma, a.L, a.N, a.T, nC, c_cnt, cpc,
                                                                            a.zin, a.zsum, a.zsub, a.wgt, a.part, a.xT, a.dxT);
}

// Cross-chunk coupling matrices by doubling: for a span of n steps  E_k(n) = sum_i M^(n-1-i) dM_k M^i,  and
// E(2n) = E(n) M^n + M^n E(n).  Levels stored for spans of 2^j CHUNKS, j = 0..NLEV-1 (j = 0: one chunk), which is what
// the carry scan over chunks needs.  One thread per (latent, k).  Ek layout [level][l][3][D*D].
#ifndef MOIHGP_OBJ_LOG2_CG
#define MOIHGP_OBJ_LOG2_CG 3
#endif
constexpr int LOG2_CG = MOIHGP_OBJ_LOG2_CG;
constexpr int CG = 1 << LOG2_CG;   // chunks per lane in the carry scan
constexpr int NLEV = LOG2_CG + 5 + 1;
static_assert(NLEV <= 16, "the Ek workspace holds 16 levels (capi.cu)");
template <int D>
__global__ void k_obj_coupling(const LatentConsts* __restrict__ consts, int L, double* __restrict__ Ek) {
    const int id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= 3 * L) return;
    const int l = id / 3, k = id % 3;
    const LatentConsts* lc = consts + l;
    double E[D * D], Mn[D * D];
    load_mat<D>(lc->dAKHA[k], E);
    for (int lev = 0; lev < LOG2_CH + NLEV - 1; ++lev) {
        if (lev >= LOG2_CH)
            for (int i = 0; i < D * D; ++i) Ek[(((size_t)(lev - LOG2_CH) * L + l) * 3 + k) * D * D + i] = E[i];
        load_mat<D>(lc->powM[lev], Mn);
        double a[D * D];
        for (int i = 0; i < D; ++i) for (int j = 0; j < D; ++j) {
            double s = 0.0;
            for (int q = 0; q < D; ++q) s += E[i * D + q] * Mn[q * D + j] + Mn[i * D + q] * E[q * D + j];
            a[i * D + j] = s;
        }
        for (int i = 0; i < D * D; ++i) E[i] = a[i];
    }
    for (int i = 0; i < D * D; ++i) Ek[(((size_t)(NLEV - 1) * L + l) * 3 + k) * D * D + i] = E[i];
}

// zin[c+1] = Z^CH zin[c] + zsum[c] on the augmented state z = [x; dx_0; dx_1; dx_2]:
//   x' = M^CH x + f_x,   dx_k' = M^CH dx_k + E_k x + f_k.
// One WARP (= one CTA) per (sequence, latent): groups of 256 chunks (lane = 8 consecutive chunks, Kogge-Stone over lanes
// with the span-(8 * 2^j) transition), groups in sequence.  The chain is latency-bound (a handful of warps on the whole
// GPU), so nothing on it may wait for HBM: a group's 256 summaries (one contiguous run) are staged into shared memory
// with coalesced loads, the carries are written back the same way, and the scan-level matrices sit in shared memory.
template <int D>
__global__ void __launch_bounds__(32) k_obj_carry(const LatentConsts* __restrict__ consts, const double* __restrict__ Ek, int L,
                                                 long long N, long long nC, const double* __restrict__ x0,
                                                 const double* __restrict__ dx0, const double* __restrict__ zsum,
                                                 double* __restrict__ zin) {
    constexpr int ZD = 4 * D;                 // doubles per chunk
    constexpr int BLK = CG * ZD;              // doubles per lane and group
    constexpr int PITCH = BLK + 2;            // PITCH / 2 odd: conflict-free 16-byte accesses across lanes
    extern __shared__ double stage[];         // [32][PITCH]
    __shared__ double lev[5][4 * D * D];      // per scan level: M^(CH 8 2^j), E_k(CH 8 2^j)
    const int lane = threadIdx.x;
    const long long id = blockIdx.x;
    const int l = (int)(id % L);
    double MC[D * D], E[3][D * D];
    load_mat<D>(consts[l].powM[LOG2_CH], MC);
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int i = 0; i < D * D; ++i) E[k][i] = Ek[((size_t)l * 3 + k) * D * D + i];
    for (int i = lane; i < 5 * 4 * D * D; i += 32) {
        const int j = i / (4 * D * D), r = i - j * (4 * D * D);
        const int m = r / (D * D), e = r - m * (D * D);
        lev[j][r] = m == 0 ? consts[l].powM[LOG2_CH + LOG2_CG + j][(e / D) * 3 + (e % D)]
                           : Ek[(((size_t)(LOG2_CG + j) * L + l) * 3 + (m - 1)) * D * D + e];
    }
    const size_t base = (size_t)id * nC * ZD;      // [n][l][chunk][4*D]
    const long long nG = (nC + 32 * CG - 1) / (32 * CG);
    double carry[4][D];
#pragma unroll
    for (int q = 0; q < D; ++q) {
        carry[0][q] = x0 ? x0[(size_t)id * D + q] : 0.0;
#pragma unroll
        for (int k = 0; k < 3; ++k) carry[1 + k][q] = dx0 ? dx0[((size_t)id * 3 + k) * D + q] : 0.0;
    }
    double* mine = stage + lane * PITCH;
    // one chunk: z <- Z^CH z + f   (the summary of the sequence's last chunk is never used)
    auto advance = [&](double (&z)[4][D], const double (&f)[ZD]) {
        double zn[4][D];
        mv<D>(MC, z[0], zn[0]);
#pragma unroll
        for (int k = 0; k < 3; ++k) { mv<D>(MC, z[1 + k], zn[1 + k]); mv_acc<D>(E[k], z[0], zn[1 + k]); }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int q = 0; q < D; ++q) z[a][q] = zn[a][q] + f[a * D + q];
    };
    auto load_f = [&](int i, long long c, double (&f)[ZD]) {
#pragma unroll
        for (int e = 0; e < ZD; e += 2) {
            const double2 t2 = *reinterpret_cast<const double2*>(mine + i * ZD + e);
            f[e] = c < nC - 1 ? t2.x : 0.0;
            f[e + 1] = c < nC - 1 ? t2.y : 0.0;
        }
    };
    for (long long g = 0; g < nG; ++g) {
        const long long cbeg = g * 32 * CG;
        const int pairs = (int)min((long long)32 * CG, nC - cbeg) * ZD / 2;      // 16-byte units of this group
        const double2* src = reinterpret_cast<const double2*>(zsum + base + cbeg * ZD);
        __syncwarp();
        for (int e = lane; e < pairs; e += 32) {
            const int blk = e / (BLK / 2), off = e - blk * (BLK / 2);
            *reinterpret_cast<double2*>(stage + blk * PITCH + 2 * off) = src[e];
        }
        __syncwarp();
        const long long c0 = cbeg + (long long)lane * CG;
        double z[4][D];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int q = 0; q < D; ++q) z[a][q] = lane == 0 ? carry[a][q] : 0.0;
#pragma unroll 2
        for (int i = 0; i < CG; ++i) {
            double f[ZD];
            load_f(i, c0 + i, f);
            advance(z, f);
        }
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            const int o = 1 << j;
            double zo[4][D], P[D * D];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int q = 0; q < D; ++q) zo[a][q] = __shfl_up_sync(FULL, z[a][q], o);
#pragma unroll
            for (int i = 0; i < D * D; ++i) P[i] = lev[j][i];
            if (lane >= o) {
#pragma unroll
                for (int a = 0; a < 4; ++a) mv_acc<D>(P, zo[a], z[a]);
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    double Ej[D * D];
#pragma unroll
                    for (int i = 0; i < D * D; ++i) Ej[i] = lev[j][(1 + k) * D * D + i];
                    mv_acc<D>(Ej, zo[0], z[1 + k]);
                }
            }
        }
        double x[4][D];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int q = 0; q < D; ++q) {
                const double up = __shfl_up_sync(FULL, z[a][q], 1);
                x[a][q] = lane == 0 ? carry[a][q] : up;
                carry[a][q] = __shfl_sync(FULL, z[a][q], 31);
            }
#pragma unroll 2
        for (int i = 0; i < CG; ++i) {
            double f[ZD];
            load_f(i, c0 + i, f);
            double xf[ZD];                                   // the carry INTO chunk c0 + i replaces its summary in the stage
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int q = 0; q < D; ++q) xf[a * D + q] = x[a][q];
#pragma unroll
            for (int e = 0; e < ZD; e += 2) *reinterpret_cast<double2*>(mine + i * ZD + e) = make_double2(xf[e], xf[e + 1]);
            advance(x, f);
        }
        __syncwarp();
        double2* dst = reinterpret_cast<double2*>(zin + base + cbeg * ZD);
        for (int e = lane; e < pairs; e += 32) {
            const int blk = e / (BLK / 2), off = e - blk * (BLK / 2);
            dst[e] = *reinterpret_cast<const double2*>(stage + blk * PITCH + 2 * off);
        }
    }
}

// End state of the block from its carry-in: z_end = Z^CH zin[nC-1] + zsum[nC-1] (exact when the last chunk is full, i.e.
// T is a multiple of CH).  One thread per (sequence, latent).  zend layout [N][L][4][D].
template <int D>
__global__ void __launch_bounds__(128) k_obj_block_end(const LatentConsts* __restrict__ consts, const double* __restrict__ Ek, int L,
                                                      long long N, long long nC, const double* __restrict__ zsum,
                                                      const double* __restrict__ zin, double* __restrict__ zend) {
    const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= N * L) return;
    const int l = (int)(id % L);
    double MC[D * D];
    load_mat<D>(consts[l].powM[LOG2_CH], MC);
    const size_t o = ((size_t)id * nC + (nC - 1)) * 4 * D;
    double x[D], out[D];
#pragma unroll
    for (int q = 0; q < D; ++q) x[q] = zin[o + q];
    mv<D>(MC, x, out);
#pragma unroll
    for (int q = 0; q < D; ++q) zend[(size_t)id * 4 * D + q] = out[q] + zsum[o + q];
    for (int k = 0; k < 3; ++k) {
        double dz[D], E[D * D];
#pragma unroll
        for (int q = 0; q < D; ++q) dz[q] = zin[o + (1 + k) * D + q];
#pragma unroll
        for (int i = 0; i < D * D; ++i) E[i] = Ek[((size_t)l * 3 + k) * D * D + i];
        mv<D>(MC, dz, out);
        mv_acc<D>(E, x, out);
#pragma unroll
        for (int q = 0; q < D; ++q) zend[(size_t)id * 4 * D + (1 + k) * D + q] = out[q] + zsum[o + (1 + k) * D + q];
    }
}

// dU partials: gU_part[split][r][c] = sum over the split's (n, t) range of Y[n][t][r] * wgt[n][c][t].
// CTA tile: 64 x 64 outputs, 16 x 16 threads, 4 x 4 outputs per thread, K panels of 16 steps.
constexpr int GT = 64, GK = 16;
__global__ void __launch_bounds__(256) k_gradU(const double* __restrict__ Y, const double* __restrict__ wgt, int p, int L,
                                              long long N, long long T, long long slabs_per_split, double* __restrict__ gU_part) {
    __shared__ double ys[GK][GT + 1];
    __shared__ double wsm[GK][GT + 1];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int rt = blockIdx.x, ct = blockIdx.y, split = blockIdx.z;
    const int r0 = rt * GT, c0 = ct * GT;
    const long long slabs_per_seq = (T + GK - 1) / GK;
    const long long total = N * slabs_per_seq;
    const long long s_begin = (long long)split * slabs_per_split;
    const long long s_end = min(total, s_begin + slabs_per_split);
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
    for (long long s = s_begin; s < s_end; ++s) {
        const long long n = s / slabs_per_seq;
        const long long t0 = (s - n * slabs_per_seq) * GK;
        __syncthreads();
        for (int i = threadIdx.x; i < GK * GT; i += 256) {
            const int kk = i / GT, rr = i - kk * GT;          // consecutive threads -> consecutive outputs r (contiguous in Y)
            const long long t = t0 + kk;
            ys[kk][rr] = (t < T && r0 + rr < p) ? Y[((size_t)n * T + t) * p + r0 + rr] : 0.0;
        }
        for (int i = threadIdx.x; i < GK * GT; i += 256) {
            const int cc = i / GK, kk = i - cc * GK;          // consecutive threads -> consecutive t (contiguous in wgt)
            const long long t = t0 + kk;
            wsm[kk][cc] = (t < T && c0 + cc < L) ? wgt[((size_t)n * L + c0 + cc) * T + t] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GK; ++kk) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { a[i] = ys[kk][ty + 16 * i]; b[i] = wsm[kk][tx + 16 * i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
        }
    }
    double* out = gU_part + (size_t)split * p * L;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = r0 + ty + 16 * i, c = c0 + tx + 16 * j;
            if (r < p && c < L) out[(size_t)r * L + c] = acc[i][j];
        }
}

// The same contraction on the FP64 tensor pipe (DMMA m8n8k4): CTA tile 64 (outputs r) x 64 (latents c), K panels of 16
// time steps double-buffered by cp.async; 8 warps, warp w owns rows 8w..8w+7 and all 8 column blocks.
// A[m = r][k = t] = Y[t][r] comes from the staged panel ys[t][r] (pitch 68), B[k = t][n = c] = wgt[c][t] from ws[c][t]
// (pitch 20): both fragment loads are bank-conflict free.  Needs p even, T even and 16-byte aligned bases.
constexpr int GYP = GT + 4;       // pitch of ys rows (doubles)
constexpr int GWP = GK + 4;       // pitch of ws rows (doubles)
__global__ void __launch_bounds__(256) k_gradU_mma(const double* __restrict__ Y, const double* __restrict__ wgt, int p, int L,
                                                  long long N, long long T, long long slabs_per_split, double* __restrict__ gU_part) {
    __shared__ __align__(16) double ys[2][GK][GYP];
    __shared__ __align__(16) double ws[2][GT][GWP];
    const int tid = threadIdx.x, lane = tid & 31, wi = tid >> 5;
    const int g4 = lane >> 2, q4 = lane & 3;
    const int r0 = blockIdx.x * GT, c0 = blockIdx.y * GT, split = blockIdx.z;
    const long long slabs_per_seq = (T + GK - 1) / GK;
    const long long total = N * slabs_per_seq;
    const long long s_begin = (long long)split * slabs_per_split;
    const long long s_end = min(total, s_begin + slabs_per_split);
    double acc[8][2];
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) { acc[nb][0] = 0.0; acc[nb][1] = 0.0; }

    auto stage = [&](long long sl, int buf) {
        const long long n = sl / slabs_per_seq;
        const long long t0 = (sl - n * slabs_per_seq) * GK;
#pragma unroll
        for (int i = 0; i < 2; ++i) {                       // Y panel: 16 steps x 32 chunks of 2 outputs
            const int q = tid + 256 * i;
            const int kk = q >> 5, ch = q & 31;
            const long long t = t0 + kk;
            const int col = r0 + 2 * ch;
            const int bytes = (t < T && col < p) ? 16 : 0;
            cp_async16_zfill(&ys[buf][kk][2 * ch], Y + ((size_t)n * T + (t < T ? t : 0)) * p + (col < p ? col : 0), bytes);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {                       // weights panel: 64 latents x 8 chunks of 2 steps
            const int q = tid + 256 * i;
            const int cc = q >> 3, ch = q & 7;
            const long long t = t0 + 2 * ch;
            const int bytes = (c0 + cc < L && t < T) ? 16 : 0;
            cp_async16_zfill(&ws[buf][cc][2 * ch], wgt + ((size_t)n * L + (c0 + cc < L ? c0 + cc : 0)) * T + (t < T ? t : 0), bytes);
        }
        cp_async_commit();
    };

    if (s_begin < s_end) stage(s_begin, 0);
    for (long long sl = s_begin; sl < s_end; ++sl) {
        const int buf = (int)((sl - s_begin) & 1);
        if (sl + 1 < s_end) { stage(sl + 1, buf ^ 1); cp_async_wait<1>(); }
        else cp_async_wait<0>();
        __syncthreads();
#pragma unroll
        for (int kb = 0; kb < GK / 4; ++kb) {
            const double a = ys[buf][4 * kb + q4][8 * wi + g4];
            double b[8];
#pragma unroll
            for (int nb = 0; nb < 8; ++nb) b[nb] = ws[buf][8 * nb + g4][4 * kb + q4];
#pragma unroll
            for (int nb = 0; nb < 8; ++nb) dmma884(acc[nb][0], acc[nb][1], a, b[nb]);
        }
        __syncthreads();
    }
    double* out = gU_part + (size_t)split * p * L;
    const int r = r0 + 8 * wi + g4;
#pragma unroll
    for (int nb = 0; nb < 8; ++nb)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int c = c0 + 8 * nb + 2 * q4 + e;
            if (r < p && c < L) out[(size_t)r * L + c] = acc[nb][e];
        }
}

// Per-latent reduction of the chunk partials (blocks 0..L-1) and of rho (block L): fixed order.
constexpr int RSPLIT = 16;        // CTAs per latent in k_obj_reduce (fixed-order partials, summed in k_obj_finish)
__global__ void __launch_bounds__(256) k_obj_reduce(const double* __restrict__ part, const double* __restrict__ rho, int L,
                                                   long long N, long long tiles, long long nC,
                                                   double* __restrict__ lat_part /*[L+1][RSPLIT][8]*/) {
    __shared__ double red[256][5];
    const int tid = threadIdx.x;
    const int l = blockIdx.x / RSPLIT, sp = blockIdx.x % RSPLIT;
    double s[5] = {0, 0, 0, 0, 0};
    if (l < L) {
        const long long tot = nC * N, per = (tot + RSPLIT - 1) / RSPLIT;
        const long long hi = min(tot, (sp + 1) * per);
        for (long long i = sp * per + tid; i < hi; i += 256) {
            const double* pp = part + ((size_t)i * L + l) * NPART;
#pragma unroll
            for (int j = 0; j < 5; ++j) s[j] += pp[j];
        }
    } else {
        const long long tot = N * tiles, per = (tot + RSPLIT - 1) / RSPLIT;
        const long long hi = min(tot, (sp + 1) * per);
        for (long long i = sp * per + tid; i < hi; i += 256) s[0] += rho[i];
    }
#pragma unroll
    for (int j = 0; j < 5; ++j) red[tid][j] = s[j];
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o) {
#pragma unroll
            for (int j = 0; j < 5; ++j) red[tid][j] += red[tid + o][j];
        }
        __syncthreads();
    }
    if (tid < 5) lat_part[((size_t)l * RSPLIT + sp) * 8 + tid] = red[0][tid];
}

// Assemble loss and gradient [U (p*L row-major) | S (L) | sigma | (mag, len, noise) x L]  (moihgp.h:553-609)
// grid: one CTA of 256 threads per 32 entries of dU (fixed-order sum over the split-K partials);
// thread 0 of CTA 0 assembles the scalar / per-latent entries.
__global__ void __launch_bounds__(256) k_obj_finish(const double* __restrict__ lat_part, const double* __restrict__ gU_part,
                                                   int nsplit, const double* __restrict__ S, double sigma, int p, int L,
                                                   long long N, long long T, int threading, double* __restrict__ loss,
                                                   double* __restrict__ grad) {
    const int tid = threadIdx.x;
    const int sizeU = p * L;
    {
        // a CTA sums 32 entries of dU: thread (j, e) adds the split-K partials j, j + 8, ... of entry e in order (a warp
        // reads 32 consecutive entries: 256 contiguous bytes), then the eight sub-sums are added in fixed order -
        // deterministic, and 8 x more loads in flight than one thread per entry (58 -> 12 us at config 5)
        __shared__ double sub[8][32];
        const int e = tid & 31, j = tid >> 5;
        const int i = blockIdx.x * 32 + e;
        double s = 0.0;
        if (i < sizeU)
            for (int k = j; k < nsplit; k += 8) s += gU_part[(size_t)k * sizeU + i];
        sub[j][e] = s;
        __syncthreads();
        if (j == 0 && i < sizeU) {
            double a = sub[0][e];
#pragma unroll
            for (int q = 1; q < 8; ++q) a += sub[q][e];
            grad[i] = a;
        }
    }
    // CTA 0: the RSPLIT partials of every per-latent sum in fixed order, then the scalar / per-latent entries.
    // Dynamic shared memory: lat_sums[(L + 1) * 8], gs_term[L].
    extern __shared__ double fin_sm[];
    double* lat_sums = fin_sm;
    if (blockIdx.x == 0) {
        for (int i = tid; i < (L + 1) * 5; i += 256) {
            const int l = i / 5, j = i - l * 5;
            double a = 0.0;
            for (int sp = 0; sp < RSPLIT; ++sp) a += lat_part[((size_t)l * RSPLIT + sp) * 8 + j];
            lat_sums[l * 8 + j] = a;
        }
    }
    __syncthreads();
    if (blockIdx.x != 0) return;
    // the per-latent entries in parallel (thread l), the two scalars by thread 0 in latent order - the same operations in the
    // same order as a single thread would do them, without 64 latents' worth of divisions queued behind one lane
    double* gs_term = lat_sums + (size_t)(L + 1) * 8;
    const double steps = (double)N * (double)T;
    for (int l = tid; l < L; l += 256) {
        const double* q = lat_sums + (size_t)l * 8;
        const double Sl = S[l], rs = sqrt(Sl);
        const double g2 = q[3];
        grad[sizeU + l] = steps * 0.5 / Sl - 0.5 * (1.0 / rs / rs / rs) * q[4] - g2 * sigma / Sl / Sl;   // :555-562, :591
        gs_term[l] = g2 / Sl;                                                              // :592
        for (int k = 0; k < 3; ++k) grad[sizeU + L + 1 + 3 * l + k] = q[1 + k];            // :608-609
    }
    __syncthreads();
    if (tid == 0) {
        const double rho_sum = lat_sums[(size_t)L * 8];
        const double m_n = fmax((double)(p - L), 0.0);                                     // moihgp.h:502
        double ls = steps * nll_step_const(S, p, L, sigma) + 0.5 * rho_sum / sigma;        // moihgp.h:503
        double gsig = 0.5 * (steps * m_n - rho_sum / sigma) / sigma;                       // moihgp.h:563
        for (int l = 0; l < L; ++l) {
            if (threading) ls += lat_sums[(size_t)l * 8];                                  // moihgp.h:588 vs :601 (Q5)
            gsig += gs_term[l];
        }
        grad[sizeU + L] = gsig;
        *loss = ls;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// k_obj_small: the WHOLE objective of one short sequence in ONE kernel launch (one CTA): projection, residual norms, the
// sensitivity recursion, the dU contraction and the assembly of loss / gradient - what the streaming learner evaluates
// a handful of times per sample on its window (moihgp_online.h:40-72; BASELINE configs[1]: p = 8, L = 4, window <= 64),
// where the general path is nothing but launch latency (8 launches, ~65 us of device time for ~5 us of arithmetic).
// Four lanes per latent: lane 0 of the group carries x, lanes 1..3 carry dx_k (ihgp.h:71-77); the pre-step x is broadcast
// inside the group each step.  Same quirks as the general path (Q5, Q8, Q9, Q20).  Observations with missing outputs are
// not handled here: the kernel raises out[1] and the caller re-runs the general path.
// out = [loss, nan flag, grad[num_param]]; dynamic shared memory: U[p][L], Y[T][p], u[T][L], w -> dU weights [T][L], lat[L][5].
template <int D>
__global__ void __launch_bounds__(128) k_obj_small(const double* __restrict__ Y, const double* __restrict__ U, const double* __restrict__ S,
                                                  double sigma_host, const LatentConsts* __restrict__ consts, int p, int L, int T, int threading,
                                                  const double* __restrict__ x0, const double* __restrict__ dx0, double* __restrict__ out,
                                                  double* __restrict__ xT, double* __restrict__ dxT,
                                                  const double* __restrict__ centre /*[p] subtracted from every observation, or null*/,
                                                  const double* __restrict__ sigma_dev /*sigma on the device (CUDA-graph replays), or null*/) {
    const double sigma = sigma_dev ? *sigma_dev : sigma_host;
    extern __shared__ double sm[];
    double* sU = sm;
    double* sY = sU + p * L;
    double* su = sY + (size_t)T * p;
    double* sw = su + (size_t)T * L;
    double* lat = sw + (size_t)T * L;            // [L][5]
    __shared__ double red[128];
    __shared__ int bad;
    const int tid = threadIdx.x;
    if (tid == 0) bad = 0;
    for (int i = tid; i < p * L; i += 128) sU[i] = U[i];
    for (int i = tid; i < T * p; i += 128) sY[i] = centre ? Y[i] - centre[i % p] : Y[i];     // moihgp_online.h:63 (y - ma)
    __syncthreads();
    // ---- projection  w = U'y, u = S^-1/2 w   (moihgp.h:481-498 without missing data) --------------------------------
    for (int i = tid; i < T * L; i += 128) {
        const int t = i / L, l = i - t * L;
        double a = 0.0;
        for (int r = 0; r < p; ++r) a = fma(sU[r * L + l], sY[t * p + r], a);
        sw[i] = a;
        su[i] = a * (1.0 / sqrt(S[l]));
    }
    __syncthreads();
    // ---- residual norms  rho_t = || (I - U U') y_t ||_2   (moihgp.h:499-501; norm, not squared: Q9) -------------------
    double rho = 0.0;
    for (int t = tid; t < T; t += 128) {
        double ysq = 0.0, wsq = 0.0;
        for (int r = 0; r < p; ++r) ysq = fma(sY[t * p + r], sY[t * p + r], ysq);
        for (int l = 0; l < L; ++l) wsq = fma(sw[t * L + l], sw[t * L + l], wsq);
        double q = ysq - wsq;
        if (!(ysq == ysq)) bad = 1;              // a missing (NaN) output somewhere in this observation
        if (p == L && ysq == ysq) q = 0.0;       // square orthogonal U: the residual vanishes identically
        else if (!(q >= 1e-4 * ysq)) {           // cancellation: the explicit form
            q = 0.0;
            for (int r = 0; r < p; ++r) {
                double e = sY[t * p + r];
                for (int l = 0; l < L; ++l) e = fma(-sU[r * L + l], sw[t * L + l], e);
                q = fma(e, e, q);
            }
        }
        rho += sqrt(q);
    }
    red[tid] = rho;
    __syncthreads();
    // ---- the recursion: lane (l, c), c = 0: x, c = 1..3: dx_{c-1} ------------------------------------------------------
    {
        const int l = min(tid >> 2, L - 1), c = tid & 3;
        const bool live = (tid >> 2) < L;
        const LatentConsts* lc = consts + l;
        double M[D * D], HA[D], Dm[D * D], Dk[D], z[D];
        load_mat<D>(lc->AKHA, M);
        load_vec<D>(lc->HA, HA);
        if (c == 0) {
#pragma unroll
            for (int i = 0; i < D * D; ++i) Dm[i] = 0.0;
            load_vec<D>(lc->K, Dk);
        } else {
            load_mat<D>(lc->dAKHA[c - 1], Dm);
            load_vec<D>(lc->dK[c - 1], Dk);
        }
#pragma unroll
        for (int q = 0; q < D; ++q)
            z[q] = c == 0 ? (x0 ? x0[l * D + q] : 0.0) : (dx0 ? dx0[(l * 3 + c - 1) * D + q] : 0.0);
        const double Si = lc->S, logSi = lc->logS, c1 = (1.0 - lc->hak) / Si;
        const double rsS = 1.0 / sqrt(S[l]), rsig = 1.0 / sigma;
        const double hda0 = c > 0 ? lc->HdA[c - 1][0] : 0.0, dSk = c > 0 ? lc->dS[c - 1] : 0.0;
        double sv2 = 0.0, acc = 0.0;             // acc: sum pv * w (c = 0) or sum v * dv_k (c > 0)
        for (int j = 0; j < T; ++j) {
            const double uj = su[j * L + l];
            double x[D];
#pragma unroll
            for (int q = 0; q < D; ++q) x[q] = __shfl_sync(FULL, z[q], 0, 4);     // the group's pre-step x
            double hax = HA[0] * x[0];
#pragma unroll
            for (int q = 1; q < D; ++q) hax = fma(HA[q], x[q], hax);
            const double v = uj - hax;                                           // ihgp.h:214
            sv2 = fma(v, v, sv2);
            if (c == 0) {
                const double wj = sw[j * L + l];
                const double pv = (sY[j * p + l] - hax) * c1;                    // moihgp.h:510-511 (raw y(l), Q8)
                acc = fma(pv, wj, acc);                                          // moihgp.h:558-560
                if (live) sw[j * L + l] = fma(pv, rsS, -wj * rsig);              // moihgp.h:546-550 (rank-1 form)
            } else {
                double hd = HA[0] * z[0];
#pragma unroll
                for (int q = 1; q < D; ++q) hd = fma(HA[q], z[q], hd);
                const double dv = -hda0 * x[0] - hd;                             // ihgp.h:218 (Q20 de facto)
                acc = fma(v, dv, acc);
            }
            double t1[D], zn[D];
            mv<D>(Dm, x, t1);
            mv<D>(M, z, zn);
#pragma unroll
            for (int q = 0; q < D; ++q) z[q] = zn[q] + fma(Dk[q], uj, t1[q]);   // ihgp.h:73-77
        }
        if (live) {
            const double q2 = sv2 / Si;
            if (c == 0) {
                lat[l * 5 + 0] = 0.5 * (q2 + (double)T * logSi);                 // ihgp.h:215
                lat[l * 5 + 4] = acc;
                if (xT) {
#pragma unroll
                    for (int q = 0; q < D; ++q) xT[l * D + q] = z[q];
                }
            } else {
                lat[l * 5 + c] = (acc - 0.5 * (q2 - (double)T) * dSk) / Si;      // ihgp.h:219
                if (dxT) {
#pragma unroll
                    for (int q = 0; q < D; ++q) dxT[(l * 3 + c - 1) * D + q] = z[q];
                }
            }
        }
    }
    __syncthreads();
    // ---- dU = Y' W   (moihgp.h:538-552 as the rank-1 sum) ------------------------------------------------------------
    double* grad = out + 2;
    const int sizeU = p * L;
    for (int i = tid; i < sizeU; i += 128) {
        const int r = i / L, cc = i - r * L;
        double a = 0.0;
        for (int t = 0; t < T; ++t) a = fma(sY[t * p + r], sw[t * L + cc], a);
        grad[i] = a;
    }
    // ---- loss and the remaining gradient entries (moihgp.h:553-609), as k_obj_finish ------------------------------------
    if (tid == 0) {
        double rho_sum = 0.0;
        for (int i = 0; i < 128; ++i) rho_sum += red[i];
        const double steps = (double)T;
        const double m_n = fmax((double)(p - L), 0.0);
        double ls = steps * nll_step_const(S, p, L, sigma) + 0.5 * rho_sum / sigma;
        double gsig = 0.5 * (steps * m_n - rho_sum / sigma) / sigma;
        for (int l = 0; l < L; ++l) {
            const double* q = lat + l * 5;
            if (threading) ls += q[0];
            const double Sl = S[l], rs = sqrt(Sl);
            const double g2 = q[3];
            grad[sizeU + l] = steps * 0.5 / Sl - 0.5 * (1.0 / rs / rs / rs) * q[4] - g2 * sigma / Sl / Sl;
            gsig += g2 / Sl;
            for (int k = 0; k < 3; ++k) grad[sizeU + L + 1 + 3 * l + k] = q[1 + k];
        }
        grad[sizeU + L] = gsig;
        out[0] = ls;
        out[1] = bad ? 1.0 : 0.0;
    }
}

template <int D>
cudaError_t run_objective(const ObjArgs& a, cudaStream_t st) {
    const long long nC = (a.T + CH - 1) / CH;
    const long long cpw = chunks_per_group(a.N * a.L, nC, 148LL * 48);
    const long long warps = a.N * a.L * ((nC + cpw - 1) / cpw);
    const unsigned grid = (unsigned)((warps + 3) / 4);
    double* Ek = a.Ek;
    // phase 0: the whole evaluation; phase 1 ("begin"): summaries + the block's end state from a zero carry-in;
    // phase 2 ("finish"): from the true carry-in, reusing the projected series and the summaries of phase 1
    // thread-per-sub-chunk kernels when the latents come in whole groups of 8, else the warp-scan kernel
    const bool lanes = a.L % 8 == 0;
    if (a.phase != 2 && (nC > 1 || a.phase == 1)) {
        if (lanes) {
            // interior chunks (whole) by k_obj_lanes; the last chunk of the sequence (possibly ragged) by the warp-scan kernel
            if (nC > 1) launch_obj_lanes<D, false>(a, nC, nC - 1, st);
            k_obj_scan<D, false><<<(unsigned)((a.N * a.L + 3) / 4), 128, 0, st>>>(a.u, a.w, a.yl, a.consts, a.S, a.sigma, a.L, a.N, a.T, nC, nC - 1, 1, 1,
                                                                                 nullptr, a.zsum, nullptr, nullptr, nullptr, nullptr);
        } else {
            k_obj_scan<D, false><<<grid, 128, 0, st>>>(a.u, a.w, a.yl, a.consts, a.S, a.sigma, a.L, a.N, a.T, nC, 0, nC, cpw, nullptr, a.zsum,
                                                       nullptr, nullptr, nullptr, nullptr);
        }
        mark(a.mk, "k_obj_scan_summaries");
    }
    k_obj_coupling<D><<<(3 * a.L + 63) / 64, 64, 0, st>>>(a.consts, a.L, Ek);
    {
        constexpr size_t carry_smem = sizeof(double) * 32 * (CG * 4 * D + 2);
        static std::atomic<int> attr_done_c[64];
        if (AttrOnce once(attr_done_c); once) {
            if (carry_smem > 48 * 1024) cudaFuncSetAttribute(k_obj_carry<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)carry_smem);
        }
        k_obj_carry<D><<<(unsigned)(a.N * a.L), 32, carry_smem, st>>>(a.consts, Ek, a.L, a.N, nC, a.x0, a.dx0, a.zsum, a.zin);
    }
    mark(a.mk, "k_obj_carry");
    if (a.phase == 1) {
        if (a.zend) k_obj_block_end<D><<<(unsigned)((a.N * a.L + 127) / 128), 128, 0, st>>>(a.consts, Ek, a.L, a.N, nC, a.zsum, a.zin, a.zend);
        return cudaGetLastError();
    }
    if (lanes) launch_obj_lanes<D, true>(a, nC, nC, st);
    else k_obj_scan<D, true><<<grid, 128, 0, st>>>(a.u, a.w, a.yl, a.consts, a.S, a.sigma, a.L, a.N, a.T, nC, 0, nC, cpw, a.zin, nullptr, a.wgt,
                                                   a.part, a.xT, a.dxT);
    mark(a.mk, "k_obj_scan_final");
    const size_t nsplit = obj_gu_splits(a.N, a.T);
    const long long slabs = a.N * ((a.T + GK - 1) / GK);
    const long long per = (slabs + (long long)nsplit - 1) / (long long)nsplit;
    dim3 gg((a.p + GT - 1) / GT, (a.L + GT - 1) / GT, (unsigned)nsplit);
    const bool mma_ok = a.p % 2 == 0 && a.T % 2 == 0 && (reinterpret_cast<size_t>(a.Y) & 15) == 0 && (reinterpret_cast<size_t>(a.wgt) & 15) == 0;
    if (mma_ok) k_gradU_mma<<<gg, 256, 0, st>>>(a.Y, a.wgt, a.p, a.L, a.N, a.T, per, a.gU_part);
    else k_gradU<<<gg, 256, 0, st>>>(a.Y, a.wgt, a.p, a.L, a.N, a.T, per, a.gU_part);
    mark(a.mk, "k_gradU");
    double* lat_sums = a.lat_sums;
    k_obj_reduce<<<(a.L + 1) * RSPLIT, 256, 0, st>>>(a.part, a.rho, a.L, a.N, (long long)project_tiles(a.T), nC, lat_sums);
    k_obj_finish<<<(a.p * a.L + 31) / 32, 256, sizeof(double) * ((size_t)(a.L + 1) * 8 + a.L), st>>>(lat_sums, a.gU_part, (int)nsplit, a.S, a.sigma, a.p, a.L, a.N, a.T, a.threading, a.loss, a.grad);
    mark(a.mk, "k_obj_reduce");
    return cudaGetLastError();
}

}  // namespace

size_t obj_chunks(long long T) { return (size_t)((T + CH - 1) / CH); }

// number of split-K partial buffers of the dU contraction: enough CTAs to fill the GPU, never more than slabs
size_t obj_gu_splits(long long N, long long T) {
    const long long slabs = N * ((T + GK - 1) / GK);
    long long s = 296;   // 2 x 148 SMs
    if (s > slabs) s = slabs;
    if (s < 1) s = 1;
    return (size_t)s;
}

int obj_launch_count(long long T, int L) {
    const bool many = (T + CH - 1) / CH > 1;
    return many ? (L % 8 == 0 ? 8 : 7) : 6;
}

// one short sequence, one launch (k_obj_small): shared memory it needs, 0 if the shape does not qualify
size_t obj_small_smem(int p, int L, long long T) {
    if (L > 32 || T > 1024) return 0;                 // beyond ~1000 steps the sequential loop loses to the chunked scan
    const size_t b = sizeof(double) * ((size_t)p * L + (size_t)T * p + 2 * (size_t)T * L + 5 * (size_t)L);
    return b <= 96 * 1024 ? b : 0;
}

cudaError_t launch_objective_small(int dim, const double* Y, const double* U, const double* S, double sigma, const LatentConsts* consts,
                                   int p, int L, long long T, int threading, const double* x0, const double* dx0, double* out, double* xT,
                                   double* dxT, cudaStream_t st, const double* centre, const double* sigma_dev) {
    const size_t smem = obj_small_smem(p, L, T);
    static std::atomic<int> attr_done[64];
    if (AttrOnce once(attr_done); once) {
        cudaFuncSetAttribute(k_obj_small<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
        cudaFuncSetAttribute(k_obj_small<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    }
    if (dim == 2) k_obj_small<2><<<1, 128, smem, st>>>(Y, U, S, sigma, consts, p, L, (int)T, threading, x0, dx0, out, xT, dxT, centre, sigma_dev);
    else k_obj_small<3><<<1, 128, smem, st>>>(Y, U, S, sigma, consts, p, L, (int)T, threading, x0, dx0, out, xT, dxT, centre, sigma_dev);
    return cudaGetLastError();
}

cudaError_t launch_objective(int dim, const ObjArgs& a, cudaStream_t st) {
    return dim == 2 ? run_objective<2>(a, st) : run_objective<3>(a, st);
}

}  // namespace moihgp
