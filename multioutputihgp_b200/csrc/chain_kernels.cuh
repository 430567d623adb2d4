#pragma once
// Many-chains path: one thread per (sequence, latent) chain, sequential in time (sm_100a).
//
// When there are tens of thousands of independent (sequence, latent) recurrences (BASELINE config 3:
// 4096 x 8), time-parallel scanning only adds redundant flops; here every recurrence is evaluated
// exactly once, as the reference's loop does, and the kernels are HBM streams.
//
// Replaces the same reference code as project.cu + scan.cu:
//   moihgp.h:159-182, :499-501   projection and residual norm            (phase 1 of k_filter_chain)
//   ihgp.h:81-93, :204-209       IHGP::step / IHGP::negLogLikelihood     (phase 2 of k_filter_chain)
//   moihgp.h:614-688             MOIHGP::negLogLikelihood(x, y)          (per-sequence reduction, k_filter_chain)
//   ihgp.h:108-113               IHGP::backwardSmoother recursion        (k_smooth_chain; literal and RTS forms)
//
// k_filter_chain<P, L, D>: one WARP owns NS = 32 / L sequences for all T steps, in rounds of L steps
// (32 rows of Y per round).
//   load   : the [32 rows][P] tile of Y (NS contiguous runs of L*P*8 bytes) is staged by cp.async into a ring
//            of shared-memory stages; the 16-byte chunks of each row are XOR-swizzled with the row index so
//            that both the tensor-core fragment loads and "one row per lane" reads are bank-conflict free.
//   phase 1: W = Ytile[32 x P] * U[P x L] on the FP64 tensor pipe (mma.sync m8n8k4: 4 row blocks x P/4 k blocks);
//            U lives in registers as B fragments.  The residual norm || y - U U' y || comes from
//            ||y||^2 - ||U'y||^2 (U has orthonormal columns: polar factor, moihgp.h:431-447); rows where that
//            difference cancels (below 1e-4 ||y||^2, or NaN) take the explicit (I - U U') y evaluation instead.
//            u = S^-1/2 U' y goes to a small exchange tile.
//   phase 2: lane (s, l) picks latent l of the L steps out of the exchange tile and runs the recurrence
//            x+ = AKHA x + K u, accumulating the innovation likelihood; states go to a staging tile.
//   store  : the staging tile leaves as NS contiguous runs of L*L*D doubles with 16-byte stores.
// k_smooth_chain<L, D, MODE>: the same lane mapping streaming backwards over the stored X.
// Full rounds of full sequence groups run a predicate-free fast path; the ragged last round / last CTA
// take a clamped-and-predicated path.
#include <cuda_runtime.h>
#include <math.h>
#include <cmath>
#include "moihgp_device.cuh"
#include "ptx.cuh"
#include "launch.h"
#include "ls_project.cuh"

namespace moihgp {

namespace {

constexpr unsigned FULL = 0xffffffffu;
// Ring depth of the filter's cp.async tiles.  Measured on B200, config 3 (profiles/r02/ab_smoother_ring_depth.txt):
// 2 / 3 / 4 / 6 stages = 3.62 / 3.75 / 3.84 / 5.17 ms - one tile in flight per warp is enough (seven warps per SM keep
// 28 KB of reads outstanding) and deeper rings only crowd the stores out; evict-first stores (__stcs) for X changed nothing.
#ifndef MOIHGP_FSTAGES
#define MOIHGP_FSTAGES 2
#endif
constexpr int STAGES = MOIHGP_FSTAGES;

template <int P, int L>
struct ProjConsts {          // passed by value: lives in the constant bank
    double U[P][L];
    double rs[L];            // S^-1/2
};

// one latent's state in the staging tile: a single 16-byte access when D = 2
template <int D> __device__ __forceinline__ void store_state(double* p, const double (&v)[D]) {
    if (D == 2) *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]);
    else {
#pragma unroll
        for (int a = 0; a < D; ++a) p[a] = v[a];
    }
}
template <int D> __device__ __forceinline__ void load_state(const double* p, double (&v)[D]) {
    if (D == 2) { const double2 t = *reinterpret_cast<const double2*>(p); v[0] = t.x; v[1] = t.y; }
    else {
#pragma unroll
        for (int a = 0; a < D; ++a) v[a] = p[a];
    }
}

// v[rb] summed over the 4 lanes of a quad; lane q of the quad receives the total of v[q].
__device__ __forceinline__ double quad_transpose_reduce(const double (&v)[4], int lane) {
    const bool b0 = lane & 1, b1 = lane & 2;
    const double k0 = b0 ? v[1] : v[0], s0 = b0 ? v[0] : v[1];
    const double k1 = b0 ? v[3] : v[2], s1 = b0 ? v[2] : v[3];
    const double a0 = k0 + __shfl_xor_sync(FULL, s0, 1);
    const double a1 = k1 + __shfl_xor_sync(FULL, s1, 1);
    const double k = b1 ? a1 : a0, s = b1 ? a0 : a1;
    return k + __shfl_xor_sync(FULL, s, 2);
}

// Pitch (doubles) of one sequence's [L steps][L*D] staging tile such that the 8-byte state stores / loads of a
// half-warp (lanes (s, l) -> s * pitch + l * D + a) fall into 16 distinct 8-byte bank pairs; even, so that the
// 16-byte copy-out stays aligned.
constexpr int staging_pitch(int L, int D) {
    const int run = L * L * D;
    if (D % 2 == 0) return run + 4;            // 16-byte state stores: any pitch that staggers the sequences
    for (int pad = 0; pad < 16; pad += 2) {
        bool ok = true;
        for (int a = 0; a < 16 && ok; ++a)
            for (int b = a + 1; b < 16 && ok; ++b) {
                const int ua = (a / L) * (run + pad) + (a % L) * D, ub = (b / L) * (run + pad) + (b % L) * D;
                if ((ua - ub) % 16 == 0) ok = false;
            }
        if (ok) return run + pad;
    }
    return run + 4;
}

template <int P, int L, int D, int NS_>
struct FilterCfg {
    static constexpr int NS = NS_;                     // sequences per warp (<= 32 / L)
    static constexpr int R = NS * L;                   // rows of Y per round (8, 16 or 32)
    static constexpr int RB = R / 8;                   // 8-row blocks of the tensor-core projection
    static constexpr int ROWB = P * 8;                 // bytes per row of Y
    static constexpr int CH = P / 2;                   // 16-byte chunks per row
    static constexpr int TILE = R * ROWB;              // bytes per stage
    static constexpr int KB = P / 4;                   // k blocks of the tensor-core projection
    static constexpr int LP = L < 8 ? 8 : L;           // latents padded to the n = 8 of m8n8k4
    static constexpr int NB = LP / 8;
    static constexpr int XROW = LP;                    // exchange tile row pitch (doubles): 16-byte fragment stores of two
                                                       // adjacent rows cover one 128-byte line
    static constexpr int XSEQ = L * XROW + L + (L & 1);   // per-sequence pitch (doubles): staggers the sequences of a half-warp; even (16-byte stores)
    static constexpr int LD = L * D;                   // doubles per time step of X
    static constexpr int RUN = L * LD;                 // doubles per sequence-round of X
    static constexpr int OSEQ = staging_pitch(L, D);   // staging tile per-sequence pitch (doubles), 16B-aligned
    static constexpr int PS = RUN / 2;                 // 16-byte pieces per sequence-round of X
    static constexpr int RPP = 32 / CH > 0 ? 32 / CH : 1;   // rows of Y covered by one warp-wide cp.async pass
    static constexpr int PASSES = R / RPP;             // cp.async passes per round
    static constexpr int XCH = NS * XSEQ < 32 ? 32 : NS * XSEQ;   // exchange tile (doubles); also holds 32 partial sums at the end
    static constexpr int OSTD = NS * OSEQ > ls_scratch_doubles(L) ? NS * OSEQ : ls_scratch_doubles(L);   // staging tile; also the NaN-row scratch
    static constexpr int PSD = PS / 32 > 0 ? PS / 32 : 1;
    static constexpr int BYTES = STAGES * TILE + XCH * 8 + OSTD * 8;
    // XOR swizzle of the 16-byte chunk index within a row.  A tensor-core A-fragment load is an 8-byte access of
    // lanes (row g, columns 4 kb + q): a half-warp covers 4 consecutive rows x 2 adjacent chunks, which this
    // swizzle spreads over 8 distinct 16-byte bank groups.
    __host__ __device__ static constexpr int swz(int row) { return CH >= 8 ? 2 * (row & 3) : (CH == 4 ? 2 * ((row >> 1) & 1) : 0); }
};

// grid: ceil(N / NS) CTAs of ONE warp.  NS < 32 / L leaves lanes idle in phase 2 but puts more warps in flight
// (the recurrence is latency-bound: see DESIGN.md).
// PADP: the model has p < P outputs: rows of Y are p doubles apart in global memory and land in the first p columns of the
// P-column tile rows (16-byte copies when p is even, 8-byte copies when it is odd and the rows are only 8-byte aligned); the other columns are zeroed once and U has zero rows
// there (run_chain_ns), so every later stage - tensor-pipe projection, squared norms, explicit residual, missing-data
// projection - sees a P-output model whose extra outputs are identically zero and carry no weight.
// The same variant serves L_real < L latents (L_real * D even, or T even: 16-byte aligned runs of X either way): U has zero columns there, lanes (s, j >= L_real) own no
// chain, and X keeps the CALLER'S layout [t][L_real][D] - a sequence-round is L steps of L_real * D doubles, staged and
// copied out with run-time lengths.
// STEPS: the filter-only variant that also writes every step's NLL term, nll_steps[n][t] (MOIHGP::negLogLikelihood(x_{t-1}, y_t),
// moihgp.h:614-688); X must be null.  The owner lane of each row leaves sqrt(q) in the padding of its sequence's exchange tile,
// lane (s, j) overwrites the u it consumed with v^2, and after phase 2 lane (s, i) sums v^2 / (2 S_l) of its row over the
// L_real latents in a fixed order that starts at latent i mod L_real (a row read from column 0 would put 16 lanes on one bank
// pair): the stores leave as NS contiguous runs of L steps.  1 / (2 S_l), 1 / (2 sigma) and the per-step constant sit in
// 8 (L + 2) extra bytes of dynamic shared memory, not in registers.
template <int P, int L, int D, int NS_, bool PADP, bool STEPS>
__global__ void __launch_bounds__(32, 14) k_filter_chain(const double* __restrict__ Y, const __grid_constant__ ProjConsts<P, L> pc,
                                                    const LatentConsts* __restrict__ consts, double sigma, double nll_const,
                                                    long long N, long long T, const double* __restrict__ x0,
                                                    double* __restrict__ X, double* __restrict__ nll, double* __restrict__ xT,
                                                    int* __restrict__ nan_flag, int p_real, int L_real, double* __restrict__ nll_steps) {
    using C = FilterCfg<P, L, D, NS_>;
    constexpr int NS = C::NS, CH = C::CH, KB = C::KB, NB = C::NB, LD = C::LD, R = C::R, RB = C::RB;
    static_assert(P % 4 == 0 && (CH & (CH - 1)) == 0 && CH <= 32, "P must be 4, 8, 16, 32 or 64");
    static_assert(32 % L == 0 && L <= 32, "L must divide the warp");
    static_assert(R % 8 == 0 && R <= 32 && R % C::RPP == 0, "rows per round must be 8, 16 or 32 and tile the cp.async passes");
    static_assert(C::RPP <= L ? (L % C::RPP == 0) : (C::RPP % L == 0), "row passes must tile the sequences");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned char* ytile = smem_raw;                                           // [STAGES][32 rows][P] swizzled
    double* xch = reinterpret_cast<double*>(smem_raw + STAGES * C::TILE);      // [NS][L][XROW]
    double* ost = xch + C::XCH;                                                // [NS][L][L*D]
    double* kst = ost + C::OSTD;                                               // STEPS: [L] 1 / (2 S_l), the per-step constant, 1 / (2 sigma)
    const int lane = threadIdx.x;
    const int s = lane / L, j = lane % L;                                      // phase 2: (sequence, latent)
    const long long n0 = (long long)blockIdx.x * NS;
    const int nvalid = (int)(N - n0 < NS ? N - n0 : NS);                       // sequences of this warp that exist
    const long long n = n0 + s;
    const int Lr = PADP ? L_real : L;                                          // latents of the model
    const int LDr = PADP ? L_real * D : LD;                                    // doubles per time step of X (the caller's layout)
    const bool active = lane < R && (!PADP || j < Lr);                         // phase 2 lanes that own a chain
    const bool seq_ok = s < nvalid;
    const long long rounds = (T + L - 1) / L;

    // ---- per-lane constants -------------------------------------------------------------------------
    // phase 1: B fragments of U and the S^-1/2 of this lane's two output columns per n block
    const int g4 = lane >> 2, q4 = lane & 3;
    double bf[KB][NB];
#pragma unroll
    for (int kb = 0; kb < KB; ++kb)
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) bf[kb][nb] = (8 * nb + g4 < L) ? pc.U[4 * kb + q4][(8 * nb + g4) % L] : 0.0;
    // A fragment byte offsets within a row block (rows 8 rb + g4): element (g4, 4 kb + q4)
    int offA[KB];
#pragma unroll
    for (int kb = 0; kb < KB; ++kb) offA[kb] = g4 * C::ROWB + (((2 * kb + (q4 >> 1)) ^ C::swz(g4)) << 4) + ((q4 & 1) << 3);
    // the row this lane owns after the quad transpose-reduce: row block q4, row g4 of the block
    const int own_row = 8 * q4 + g4, own_s = own_row / L, own_i = own_row % L;
    // phase 2: the latent's filter constants
    const bool owner = q4 < RB;
    const LatentConsts* lc = consts + (PADP ? min(j, Lr - 1) : j);
    double M[D * D], K[D], HA[D];
#pragma unroll
    for (int a = 0; a < D; ++a) {
        K[a] = __ldg(&lc->K[a]);
        HA[a] = __ldg(&lc->HA[a]);
#pragma unroll
        for (int b = 0; b < D; ++b) M[a * D + b] = __ldg(&lc->AKHA[a * 3 + b]);
    }
    double x[D];
#pragma unroll
    for (int a = 0; a < D; ++a) x[a] = (x0 && active && seq_ok) ? x0[((size_t)n * Lr + j) * D + a] : 0.0;
    const double rs_j = pc.rs[j];                                              // S_j^-1/2  (moihgp.h:181)
    double rho_acc = 0.0, vsq_acc = 0.0;
    bool saw_nan = false;
    if (STEPS) {
        if (lane < L) kst[lane] = lane < Lr ? 0.5 / __ldg(&consts[lane].S) : 0.0;   // read by phase 2 after the first round's __syncwarp
        if (lane == 0) {
            double logs = 0.0;
            for (int l = 0; l < Lr; ++l) logs += __ldg(&consts[l].logS);
            kst[L] = nll_const + 0.5 * logs;                                   // moihgp.h:652, ihgp.h:207
            kst[L + 1] = 0.5 / sigma;
        }
    }

    // ---- cp.async producer: tile of round r into stage r % STAGES ----------------------------------
    // pass k of a round covers rows lr + RPP * k (lr = lane / CH), chunk lc16 = lane % CH of each
    const int lr = lane / CH, lc16 = lane % CH;
    const size_t growb = PADP ? (size_t)p_real * 8 : (size_t)C::ROWB;          // bytes between rows of Y in global memory
    const bool col_ok = !PADP || 2 * lc16 < p_real;                            // this lane's 16-byte chunk holds real outputs
    const bool odd_p = PADP && (p_real & 1);
    // one 16-byte chunk of a row: whole (even p), or its 8-byte halves that hold real outputs (odd p)
    auto copy_chunk = [&](unsigned char* dst, const unsigned char* src) {
        if (!col_ok) return;
        if (!odd_p) cp_async16(dst, src);
        else {
            cp_async8(dst, src);
            if (2 * lc16 + 1 < p_real) cp_async8(dst + 8, src + 8);
        }
    };
    const size_t seq_stride = (size_t)T * growb;                               // bytes between sequences of Y
    const unsigned char* Ybytes = reinterpret_cast<const unsigned char*>(Y) + (size_t)n0 * seq_stride;
    const size_t lane_src = (size_t)(lr / L) * seq_stride + (size_t)(lr % L) * growb + lc16 * 16;
    if (PADP) {                                                                // the pad columns stay zero for the whole kernel
        for (int i = lane; i < STAGES * C::TILE / 16; i += 32) reinterpret_cast<double2*>(ytile)[i] = make_double2(0.0, 0.0);
        __syncwarp();
    }
    auto issue = [&](long long r) {
        if (r < rounds) {
            unsigned char* st = ytile + (size_t)(r % STAGES) * C::TILE;
            const long long t0 = r * L;
            if (nvalid == NS && t0 + L <= T) {
                const unsigned char* src = Ybytes + (size_t)t0 * growb + lane_src;
#pragma unroll
                for (int k = 0; k < C::PASSES; ++k) {
                    const int row = lr + C::RPP * k;
                    copy_chunk(st + row * C::ROWB + ((lc16 ^ C::swz(row)) << 4),
                               src + (size_t)((C::RPP * k) / L) * seq_stride + (size_t)((C::RPP * k) % L) * growb);
                }
            } else {
                // ragged: rows beyond T / sequences beyond N re-read the last valid row / sequence (never used)
                const int rows = (int)(T - t0 < L ? T - t0 : L);
#pragma unroll
                for (int k = 0; k < C::PASSES; ++k) {
                    const int row = lr + C::RPP * k;
                    const int rs_ = min(row / L, nvalid - 1), ri = min(row % L, rows - 1);
                    copy_chunk(st + row * C::ROWB + ((lc16 ^ C::swz(row)) << 4),
                               Ybytes + (size_t)rs_ * seq_stride + (size_t)(t0 + ri) * growb + lc16 * 16);
                }
            }
        }
        cp_async_commit();
    };
#pragma unroll
    for (int r = 0; r < STAGES - 1; ++r) issue(r);

    double* const xw = xch + (g4 / L) * C::XSEQ + (g4 % L) * C::XROW + 2 * q4;   // + row-block offset below
    double* const xc = xch + s * C::XSEQ + j;
    double* const oc = ost + s * C::OSEQ + j * D;
    double* const Xcta = !STEPS && X ? X + (size_t)n0 * T * LDr : nullptr;     // STEPS writes no X: its copy-out is dead code

    for (long long r = 0; r < rounds; ++r) {
        issue(r + STAGES - 1);
        cp_async_wait<STAGES - 1>();
        __syncwarp();
        const long long t0 = r * L;
        const bool fast = nvalid == NS && t0 + L <= T;
        const unsigned char* tile = ytile + (size_t)(r % STAGES) * C::TILE;
        // ---- phase 1: W = Ytile * U on the tensor pipe; residual norm from the two squared norms ------
        {
            double sy[4] = {0.0, 0.0, 0.0, 0.0}, sw[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
            for (int rb = 0; rb < RB; ++rb) {
                const unsigned char* blk = tile + rb * 8 * C::ROWB;
                double a[KB], c[NB][2];
#pragma unroll
                for (int kb = 0; kb < KB; ++kb) a[kb] = *reinterpret_cast<const double*>(blk + offA[kb]);
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) { c[nb][0] = 0.0; c[nb][1] = 0.0; }
#pragma unroll
                for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                    for (int nb = 0; nb < NB; ++nb) dmma884(c[nb][0], c[nb][1], a[kb], bf[kb][nb]);   // U' y   moihgp.h:181
                double ay = a[0] * a[0];
#pragma unroll
                for (int kb = 1; kb < KB; ++kb) ay = fma(a[kb], a[kb], ay);
                double aw = c[0][0] * c[0][0];
                aw = fma(c[0][1], c[0][1], aw);
#pragma unroll
                for (int nb = 1; nb < NB; ++nb) { aw = fma(c[nb][0], c[nb][0], aw); aw = fma(c[nb][1], c[nb][1], aw); }
                sy[rb] = ay;
                sw[rb] = aw;
                // w = U' y of row 8 rb + g4 into the exchange tile
                double* xr = xw + ((8 * rb) / L) * C::XSEQ + ((8 * rb) % L) * C::XROW;
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) *reinterpret_cast<double2*>(xr + 8 * nb) = make_double2(c[nb][0], c[nb][1]);
            }
            const double ysq = quad_transpose_reduce(sy, lane);
            const double wsq = quad_transpose_reduce(sw, lane);
            double q = ysq - wsq;                                                 // || (I - U U') y ||^2
            // P == L: U is square and orthogonal, (I - U U') y vanishes identically and the explicit form would return
            // rounding noise for EVERY row: rho = 0 unless the row holds a NaN
            const bool square = PADP ? p_real == Lr : P == L;                     // of the MODEL, not of the instantiated shape
            if (square && ysq == ysq) q = 0.0;
            const bool bad = owner && !(q >= 1e-4 * ysq) && !(square && ysq == ysq);   // cancellation (or NaN): evaluate explicitly
            if (__any_sync(FULL, bad)) {
                // explicit  || y - U (U' y) ||^2  of row `lane` (moihgp.h:651), w read back from the exchange tile
                __syncwarp();
                const int rl = lane < R ? lane : R - 1;
                const unsigned char* row = tile + rl * C::ROWB;
                const double* Up = &pc.U[0][0];
                asm volatile("" : "+l"(Up));      // opaque: keeps the 128 loop-invariant U loads of this cold path out of registers
                const double* wr = xch + (rl / L) * C::XSEQ + (rl % L) * C::XROW;
                double w[L];
#pragma unroll
                for (int l = 0; l < L; l += 2) {
                    const double2 t = *reinterpret_cast<const double2*>(wr + l);
                    w[l] = t.x;
                    if (l + 1 < L) w[l + 1] = t.y;
                }
                double qe = 0.0;
#pragma unroll
                for (int c = 0; c < CH; ++c) {
                    const double2 y2 = *reinterpret_cast<const double2*>(row + ((c ^ C::swz(rl)) << 4));
                    double e0 = y2.x, e1 = y2.y;
#pragma unroll
                    for (int l = 0; l < L; ++l) { e0 = fma(-Up[(2 * c) * L + l], w[l], e0); e1 = fma(-Up[(2 * c + 1) * L + l], w[l], e1); }
                    qe = fma(e0, e0, qe);
                    qe = fma(e1, e1, qe);
                }
                const double mine = __shfl_sync(FULL, qe, own_row & 31);
                if (bad) q = mine;
            }
            const bool own_ok = owner && (fast || (own_s < nvalid && t0 + own_i < T));
            if (own_ok) {
                saw_nan = saw_nan || (q != q);
                rho_acc += sqrt(q);                                               // norm, not squared (Q9); NaN row => NaN NLL, as the reference
            }
            // the row's residual norm into the padding after its sequence's L exchange rows (nothing else writes there)
            if (STEPS && owner) xch[own_s * C::XSEQ + L * C::XROW + own_i] = sqrt(q);
            // missing observations (NaN): least-squares projection on the observed outputs, moihgp.h:167-178.  Rare: the
            // whole warp solves one such row at a time, scratch in the (idle) staging tile.
            unsigned nanrows = __ballot_sync(FULL, own_ok && (ysq != ysq));
            while (nanrows) {
                const int ol = __ffs(nanrows) - 1;
                nanrows &= nanrows - 1;
                const int row = 8 * (ol & 3) + (ol >> 2);
                const unsigned char* yrow = tile + row * C::ROWB;
                const int sw_ = C::swz(row);
                double* sc = ost;
                ls_solve_coop(P, Lr,
                              [&](int r) { return *reinterpret_cast<const double*>(yrow + (((r >> 1) ^ sw_) << 4) + ((r & 1) << 3)); },
                              [&](int r, int l) { return pc.U[r][l]; },
                              sc, sc + L * L, sc + 2 * L * L, sc + 2 * L * L + L, reinterpret_cast<int*>(sc + 2 * L * L + 2 * L),
                              lane, 32, [] { __syncwarp(); });
                if (lane < L) xch[(row / L) * C::XSEQ + (row % L) * C::XROW + lane] = lane < Lr ? sc[2 * L * L + L + lane] : 0.0;   // z; phase 2 applies S^-1/2
                __syncwarp();
            }
        }
        __syncwarp();
        // ---- phase 2: latent (s, j) over the L steps of the round --------------------------------------
        double uu[L];
        if (active) {
#pragma unroll
            for (int i = 0; i < L; ++i) uu[i] = xc[i * C::XROW] * rs_j;
        }
        if (!active) {
        } else if (fast) {
#pragma unroll
            for (int i = 0; i < L; ++i) {
                const double u = uu[i];
                double hax = HA[0] * x[0];
#pragma unroll
                for (int a = 1; a < D; ++a) hax = fma(HA[a], x[a], hax);
                const double v = u - hax;                                         // ihgp.h:206
                double xn[D];
#pragma unroll
                for (int a = 0; a < D; ++a) {
                    double acc = M[a * D] * x[0];
#pragma unroll
                    for (int b = 1; b < D; ++b) acc = fma(M[a * D + b], x[b], acc);
                    xn[a] = fma(K[a], u, acc);                                    // ihgp.h:90
                }
                vsq_acc = fma(v, v, vsq_acc);
#pragma unroll
                for (int a = 0; a < D; ++a) x[a] = xn[a];
                if (STEPS) xc[i * C::XROW] = v * v * kst[j];                      // ihgp.h:207, into this lane's own u slot (already read)
                else store_state<D>(oc + i * LDr, xn);
            }
        } else {
#pragma unroll
            for (int i = 0; i < L; ++i) {
                const double u = uu[i];
                double hax = HA[0] * x[0];
#pragma unroll
                for (int a = 1; a < D; ++a) hax = fma(HA[a], x[a], hax);
                const double v = u - hax;
                double xn[D];
#pragma unroll
                for (int a = 0; a < D; ++a) {
                    double acc = M[a * D] * x[0];
#pragma unroll
                    for (int b = 1; b < D; ++b) acc = fma(M[a * D + b], x[b], acc);
                    xn[a] = fma(K[a], u, acc);
                }
                if (seq_ok && t0 + i < T) {
                    vsq_acc = fma(v, v, vsq_acc);
#pragma unroll
                    for (int a = 0; a < D; ++a) x[a] = xn[a];
                }
                if (STEPS) xc[i * C::XROW] = v * v * kst[j];
                else store_state<D>(oc + i * LDr, x);
            }
        }
        __syncwarp();
        // ---- per-step NLL terms: lane (s, i) sums row i of sequence s over the latents, in order ------------
        if (STEPS && lane < R) {
            const double* xr = xch + s * C::XSEQ + j * C::XROW;                   // lane (s, j) serves step i = j
            double vs = 0.0;
            if (!PADP) {
#pragma unroll
                for (int k = 0; k < L; ++k) vs += xr[(j + k) & (L - 1)];
            } else {
                int l = j % Lr;
                for (int k = 0; k < Lr; ++k) {
                    vs += xr[l];
                    if (++l == Lr) l = 0;
                }
            }
            const double rho = xch[s * C::XSEQ + L * C::XROW + j];
            if (seq_ok && t0 + j < T) nll_steps[(size_t)n * T + t0 + j] = rho * kst[L + 1] + vs + kst[L];   // moihgp.h:652-653
        }
        // ---- store: NS contiguous runs of L rows ------------------------------------------------------
        if (Xcta && PADP && Lr != L) {
            // padded latents: a sequence-round is L steps of LDr doubles (even), copied out in 16-byte pieces with run-time lengths
            double* Xr = Xcta + (size_t)t0 * LDr;
            const int PSr = L * LDr / 2;
            const long long rows_left = T - t0;
            const int valid16 = (int)(rows_left >= L ? PSr : rows_left * LDr / 2);
            for (int q = lane; q < NS * PSr; q += 32) {
                const int qs = q / PSr, qo = q - qs * PSr;
                if (qs < nvalid && qo < valid16)
                    *reinterpret_cast<double2*>(Xr + (size_t)qs * T * LDr + 2 * qo) = *reinterpret_cast<const double2*>(ost + qs * C::OSEQ + 2 * qo);
            }
        } else if (Xcta) {
            double* Xr = Xcta + (size_t)t0 * LD;
            if (fast) {
                constexpr int NPASS = (NS * C::PS + 31) / 32;
                double2 v[NPASS];
#pragma unroll
                for (int k = 0; k < NPASS; ++k) {
                    int qs, qo;
                    if (C::PS % 32 == 0) { qs = k / C::PSD; qo = lane + 32 * (k % C::PSD); }
                    else { const int q = lane + 32 * k; qs = q / C::PS; qo = q % C::PS; }
                    if ((NS * C::PS) % 32 == 0 || qs < NS) v[k] = *reinterpret_cast<const double2*>(ost + qs * C::OSEQ + 2 * qo);
                }
#pragma unroll
                for (int k = 0; k < NPASS; ++k) {
                    int qs, qo;
                    if (C::PS % 32 == 0) { qs = k / C::PSD; qo = lane + 32 * (k % C::PSD); }
                    else { const int q = lane + 32 * k; qs = q / C::PS; qo = q % C::PS; }
                    if ((NS * C::PS) % 32 == 0 || qs < NS) *reinterpret_cast<double2*>(Xr + (size_t)qs * T * LD + 2 * qo) = v[k];
                }
            } else {
                const long long rows_left = T - t0;
                const int valid16 = (int)(rows_left >= L ? C::PS : rows_left * (LD / 2));
#pragma unroll
                for (int k = 0; k < (NS * C::PS + 31) / 32; ++k) {
                    const int q = lane + 32 * k;
                    const int qs = q / C::PS, qo = q % C::PS;
                    if (qs < nvalid && qo < valid16) {
                        const double2 v = *reinterpret_cast<const double2*>(ost + qs * C::OSEQ + 2 * qo);
                        *reinterpret_cast<double2*>(Xr + (size_t)qs * T * LD + 2 * qo) = v;
                    }
                }
            }
        }
        __syncwarp();
    }
    cp_async_wait<0>();
    // ---- final state and NLL of each sequence ---------------------------------------------------------
    if (xT && active && seq_ok) {
#pragma unroll
        for (int a = 0; a < D; ++a) xT[((size_t)n * Lr + j) * D + a] = x[a];
    }
    if (saw_nan) *nan_flag = 1;
    if (nll) {
        // sum_t 1/2 rho_t / sigma  +  sum_l 1/2 sum_t v^2 / S_l          moihgp.h:653, ihgp.h:207
        xch[lane] = rho_acc;                                                      // owner lane -> sequence own_s
        __syncwarp();
        double part = active ? 0.5 * vsq_acc / __ldg(&lc->S) : 0.0;
#pragma unroll
        for (int o = 1; o < L; o <<= 1) part += __shfl_xor_sync(FULL, part, o);
        if (j == 0 && active && seq_ok) {
            double rho = 0.0;
            for (int q = 0; q < 32; ++q)
                if ((q & 3) < RB && (8 * (q & 3) + (q >> 2)) / L == s) rho += xch[q];
            // + T (1/2 log sum S + 1/2 m_n log sigma + 1/2 sum_l log S_l)   moihgp.h:652-653, ihgp.h:207: the first two terms
            // come from the host (parameters), the innovation variances S_l from K-setup's records - read here so that the
            // host never has to wait for them
            double logs = 0.0;
            for (int l = 0; l < Lr; ++l) logs += __ldg(&consts[l].logS);
            nll[n] = 0.5 * rho / sigma + part + (double)T * (nll_const + 0.5 * logs);
        }
    }
}

#ifndef MOIHGP_SSTAGES
#define MOIHGP_SSTAGES 4
#endif
// Measured on B200, config 3 (profiles/r02/ab_smoother_ring_depth.txt): 3 / 4 / 5 / 6 stages = 4.35 / 4.0 / 4.43 / 4.17 ms -
// four stages (9 one-warp CTAs per SM instead of 7) bring the smoother to the measured copy bandwidth (25.8 GB in 4.0 ms).
constexpr int SSTAGES = MOIHGP_SSTAGES;   // smoother ring: SSTAGES - 2 loads in flight, 1 tile being processed, 1 tile being stored

template <int L, int D, int NS_, int RM_>
struct SmoothCfg {
    static constexpr int NS = NS_;
    static constexpr int RM = RM_;                     // a round covers RM * L steps of each sequence
    static constexpr int RL = RM * L;
    static constexpr int LD = L * D;
    static constexpr int RUN = RL * LD;                // doubles per sequence-round
    static constexpr int OSEQ = RUN + (staging_pitch(L, D) - L * LD);
    static constexpr int BYTES = SSTAGES * NS * OSEQ * 8 + SSTAGES * 8;
};

// Backward sweep over the stored filtered states.  MODE 0: reference_literal (ihgp.h:108-113, Q3)
//   Xs[T-1] = X[T-1];  Xs[j] = (I - A) X[j+1] + G Xs[j+1]
// MODE 1: rts_correct   Xs[j] = X[j] + G (Xs[j+1] - A X[j]) = (I - G A) X[j] + G Xs[j+1].
// grid: ceil(N / NS) CTAs of one warp; rounds of L steps from the end of the sequence.  Each sequence-round of X is one
// contiguous run of L*L*D doubles: it is brought in by ONE TMA bulk copy (mbarrier-tracked), smoothed in place in
// shared memory, and written out by ONE bulk store - no per-lane load/store instructions touch HBM.
// PADL: the model has L_real < L latents (L_real * D even, or T even): lanes (s, j >= L_real) own no chain and the runs keep the caller's
// layout, RL steps of L_real * D doubles.
template <int L, int D, int MODE, int NS_, int RM_, bool PADL>
__global__ void __launch_bounds__(32, 14) k_smooth_chain(const double* __restrict__ X, const LatentConsts* __restrict__ consts,
                                                        long long N, long long T, double* __restrict__ Xs, int L_real) {
    using C = SmoothCfg<L, D, NS_, RM_>;
    constexpr int NS = C::NS, RL = C::RL, RM = C::RM;
    const int Lr = PADL ? L_real : L;
    const int LD = PADL ? L_real * D : C::LD;      // doubles per time step (the caller's layout)
    constexpr int LOOK = SSTAGES - 2;                  // loads in flight ahead of the round being processed
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* tiles = reinterpret_cast<double*>(smem_raw);                                   // [SSTAGES][NS][OSEQ]
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(tiles + SSTAGES * NS * C::OSEQ);
    const int lane = threadIdx.x;
    const int s = lane / L, j = lane % L;
    const bool active = lane < NS * L && (!PADL || j < Lr);
    const long long n0 = (long long)blockIdx.x * NS;
    const int nvalid = (int)(N - n0 < NS ? N - n0 : NS);
    const long long rounds = (T + RL - 1) / RL;
    const LatentConsts* lc = consts + (PADL ? min(j, Lr - 1) : j);
    double G[D * D], B[D * D];                     // B: I - A (literal, applied to X[j+1]) or I - G A (rts, applied to X[j])
#pragma unroll
    for (int a = 0; a < D; ++a)
#pragma unroll
        for (int b = 0; b < D; ++b) {
            G[a * D + b] = __ldg(&lc->G[MODE][a * 3 + b]);
            B[a * D + b] = MODE == 0 ? __ldg(&lc->ImA[a * 3 + b]) : __ldg(&lc->Bs[a * 3 + b]);
        }
    const double* const Xcta = X + (size_t)n0 * T * LD;
    double* const Xscta = Xs + (size_t)n0 * T * LD;
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < SSTAGES; ++i) mbar_init(bars + i, 1);
        mbar_fence_init();
    }
    __syncwarp();

    // round index k counts from the END: it covers steps t0 = (rounds - 1 - k) * L ...; bytes of one sequence's run
    auto run_bytes = [&](long long t0) { return (unsigned)((T - t0 >= RL ? (long long)RL : T - t0) * LD * 8); };
    auto issue = [&](long long k) {               // lane 0 only
        if (k < rounds) {
            const int st = (int)(k % SSTAGES);
            double* tile = tiles + (size_t)st * NS * C::OSEQ;
            const long long t0 = (rounds - 1 - k) * RL;
            const unsigned bytes = run_bytes(t0);
            bulk_wait_read<1>();                   // the store that last read this stage (two rounds ago) is done with it
            mbar_expect_tx(bars + st, bytes * (unsigned)nvalid);
            for (int qs = 0; qs < nvalid; ++qs) bulk_g2s(tile + qs * C::OSEQ, Xcta + ((size_t)qs * T + t0) * LD, bytes, bars + st);
        }
    };
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < LOOK; ++k) issue(k);
    }

    double xs[D], xnext[D];                       // Xs[j+1] and X[j+1]
#pragma unroll
    for (int a = 0; a < D; ++a) { xs[a] = 0.0; xnext[a] = 0.0; }
    for (long long k = 0; k < rounds; ++k) {
        if (lane == 0) issue(k + LOOK);
        const int stg = (int)(k % SSTAGES);
        mbar_wait(bars + stg, (unsigned)((k / SSTAGES) & 1));
        double* stw = tiles + (size_t)stg * NS * C::OSEQ;
        double* st = stw + s * C::OSEQ + j * D;
        const long long t0 = (rounds - 1 - k) * RL;
        const bool fast = nvalid == NS && t0 + RL <= T;
        if (!active) {
        } else if (fast && t0 + RL < T) {
            // interior round: no boundary, no predicates; L steps at a time (registers)
#pragma unroll
            for (int h = RM - 1; h >= 0; --h) {
                double* sth = st + h * L * LD;
                double xin[L][D];
#pragma unroll
                for (int i = 0; i < L; ++i) load_state<D>(sth + i * LD, xin[i]);
#pragma unroll
                for (int i = L - 1; i >= 0; --i) {
                    double xx[D], out[D];
#pragma unroll
                    for (int a = 0; a < D; ++a) xx[a] = xin[i][a];
#pragma unroll
                    for (int a = 0; a < D; ++a) {
                        double acc = G[a * D] * xs[0];
#pragma unroll
                        for (int b = 1; b < D; ++b) acc = fma(G[a * D + b], xs[b], acc);
#pragma unroll
                        for (int b = 0; b < D; ++b) acc = fma(B[a * D + b], MODE == 0 ? xnext[b] : xx[b], acc);
                        out[a] = acc;
                    }
#pragma unroll
                    for (int a = 0; a < D; ++a) { xs[a] = out[a]; xnext[a] = xx[a]; }
                    store_state<D>(sth + i * LD, out);
                }
            }
        } else if (s < nvalid) {
#pragma unroll 1
            for (int i = RL - 1; i >= 0; --i) {
                const long long t = t0 + i;
                if (t < T) {
                    double xx[D], out[D];
                    load_state<D>(st + i * LD, xx);
                    if (t == T - 1) {
#pragma unroll
                        for (int a = 0; a < D; ++a) out[a] = xx[a];                // ihgp.h:108
                    } else {
#pragma unroll
                        for (int a = 0; a < D; ++a) {                              // ihgp.h:111 / RTS
                            double acc = G[a * D] * xs[0];
#pragma unroll
                            for (int b = 1; b < D; ++b) acc = fma(G[a * D + b], xs[b], acc);
#pragma unroll
                            for (int b = 0; b < D; ++b) acc = fma(B[a * D + b], MODE == 0 ? xnext[b] : xx[b], acc);
                            out[a] = acc;
                        }
                    }
#pragma unroll
                    for (int a = 0; a < D; ++a) { xs[a] = out[a]; xnext[a] = xx[a]; }
                    store_state<D>(st + i * LD, out);
                }
            }
        }
        fence_async_smem();                        // this lane's shared-memory writes -> visible to the bulk-copy engine
        __syncwarp();
        if (lane == 0) {
            const unsigned bytes = run_bytes(t0);
            for (int qs = 0; qs < nvalid; ++qs) bulk_s2g(Xscta + ((size_t)qs * T + t0) * LD, stw + qs * C::OSEQ, bytes);
            bulk_commit();
        }
    }
    if (lane == 0) bulk_wait_read<0>();            // shared memory must outlive the last bulk store's reads
}

// STEPS: the filter-only pass with per-step NLL terms (a.nll_steps; a.X and a.Xs null)
template <int P, int L, int D, int NS, bool STEPS>
cudaError_t run_chain_ns(const ChainArgs& a, cudaStream_t st) {
    using FS = FilterCfg<P, L, D, NS>;
    constexpr int FBYTES = FS::BYTES + (STEPS ? 8 * (L + 2) : 0);     // STEPS: the table of k_filter_chain's kst
    constexpr int SNS = (NS >= 2 && NS == 32 / L) ? NS / 2 : NS;     // smoother: half the sequences per warp ...
    constexpr int SRM = (NS >= 2 && NS == 32 / L) ? 2 : 1;           // ... rounds twice as long: 2x longer contiguous runs per bulk copy
    using SS = SmoothCfg<L, D, SNS, SRM>;
    ProjConsts<P, L> pc;
    const int p_real = a.p > 0 ? a.p : P, L_real = a.L > 0 ? a.L : L;       // the model's own sizes (<= the instantiated ones)
    for (int r = 0; r < P; ++r)
        for (int l = 0; l < L; ++l) pc.U[r][l] = (r < p_real && l < L_real) ? a.U_host[(size_t)r * L_real + l] : 0.0;
    for (int l = 0; l < L; ++l) pc.rs[l] = l < L_real ? 1.0 / std::sqrt(a.S_host[l]) : 0.0;
    const bool padded = p_real != P || L_real != L, padL = L_real != L;
    if (padL && (L_real * D) % 2 != 0 && a.T % 2 != 0) return cudaErrorInvalidValue;   // chain_supported() excludes it: runs of X would not be 16-byte aligned
    const unsigned grid = (unsigned)((a.N + NS - 1) / NS);
    static std::atomic<int> attr_done[64];          // per device: function attributes belong to the device's context
    if (AttrOnce once(attr_done); once) {
        cudaFuncSetAttribute(k_filter_chain<P, L, D, NS, false, STEPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, FBYTES);
        cudaFuncSetAttribute(k_filter_chain<P, L, D, NS, true, STEPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, FBYTES);
        if constexpr (!STEPS) {
            cudaFuncSetAttribute(k_smooth_chain<L, D, 0, SNS, SRM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SS::BYTES);
            cudaFuncSetAttribute(k_smooth_chain<L, D, 1, SNS, SRM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SS::BYTES);
            cudaFuncSetAttribute(k_smooth_chain<L, D, 0, SNS, SRM, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SS::BYTES);
            cudaFuncSetAttribute(k_smooth_chain<L, D, 1, SNS, SRM, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SS::BYTES);
        }
    }
    if (!padded) k_filter_chain<P, L, D, NS, false, STEPS><<<grid, 32, FBYTES, st>>>(a.Y, pc, a.consts, a.sigma, a.nll_const, a.N, a.T, a.x0, a.X, a.nll, a.xT, a.nan_flag, P, L, a.nll_steps);
    else k_filter_chain<P, L, D, NS, true, STEPS><<<grid, 32, FBYTES, st>>>(a.Y, pc, a.consts, a.sigma, a.nll_const, a.N, a.T, a.x0, a.X, a.nll, a.xT, a.nan_flag, p_real, L_real, a.nll_steps);
    mark(a.mk, "k_filter_chain");
    if constexpr (STEPS) return cudaGetLastError();
    if (a.Xs) {
        const unsigned sgrid = (unsigned)((a.N + SNS - 1) / SNS);
        if (padL) {
            if (a.mode == 0) k_smooth_chain<L, D, 0, SNS, SRM, true><<<sgrid, 32, SS::BYTES, st>>>(a.X, a.consts, a.N, a.T, a.Xs, L_real);
            else k_smooth_chain<L, D, 1, SNS, SRM, true><<<sgrid, 32, SS::BYTES, st>>>(a.X, a.consts, a.N, a.T, a.Xs, L_real);
        } else {
            if (a.mode == 0) k_smooth_chain<L, D, 0, SNS, SRM, false><<<sgrid, 32, SS::BYTES, st>>>(a.X, a.consts, a.N, a.T, a.Xs, L);
            else k_smooth_chain<L, D, 1, SNS, SRM, false><<<sgrid, 32, SS::BYTES, st>>>(a.X, a.consts, a.N, a.T, a.Xs, L);
        }
        mark(a.mk, "k_smooth_chain");
    }
    return cudaGetLastError();
}

// Sequences per warp.  Measured on B200 (BASELINE config 3, profiles/r01): a full warp (32 / L sequences) is fastest
// even when that leaves < 2 warps per SM sub-partition - the pass is bound by HBM, not by latency - so that is the
// automatic choice; fewer sequences per warp (idle lanes in the recurrence phase, more warps) stay selectable.
// The per-step NLL pass always takes the full warp: its variant is instantiated for that choice only.
template <int P, int L, int D, bool ALLNS>
cudaError_t run_chain(const ChainArgs& a, cudaStream_t st) {
    constexpr int NSMAX = 32 / L, NSMIN = L >= 8 ? 1 : 8 / L;
    if (a.nll_steps) {
        if constexpr (L == 1 && D == 3) return cudaErrorInvalidValue;     // not served (chain.cu: find_shape)
        else return run_chain_ns<P, L, D, NSMAX, true>(a, st);
    }
    if constexpr (!ALLNS) {
        return run_chain_ns<P, L, D, NSMAX, false>(a, st);
    } else {
        const int ns = a.seqs_per_warp <= 0 ? NSMAX : a.seqs_per_warp;
        if (ns >= NSMAX) return run_chain_ns<P, L, D, NSMAX, false>(a, st);
        if (NSMAX / 2 >= NSMIN && ns >= NSMAX / 2) return run_chain_ns<P, L, D, (NSMAX / 2 >= NSMIN ? NSMAX / 2 : NSMAX), false>(a, st);
        return run_chain_ns<P, L, D, (NSMAX / 4 >= NSMIN ? NSMAX / 4 : NSMIN), false>(a, st);
    }
}

}  // namespace

}  // namespace moihgp

// one translation unit per shape (chain_inst_*.cu): keeps the build parallel
#define MOIHGP_CHAIN_INSTANCE(P, L, ALLNS)                                                                      \
    namespace moihgp {                                                                                         \
    cudaError_t launch_chain_##P##x##L(int dim, const ChainArgs& a, cudaStream_t st) {                          \
        return dim == 3 ? run_chain<P, L, 3, ALLNS>(a, st) : run_chain<P, L, 2, ALLNS>(a, st);                  \
    }                                                                                                          \
    }
