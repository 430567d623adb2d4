// K-project: OILMM projection of the observations onto the L orthogonal latents (sm_100a).
//
// Replaces (reference, /root/reference/moihgp/include/moihgp/moihgp.h):
//   :159-182  Ty = diag(S^-1/2) U' y         (and the identical blocks at :240-263, :314-336, :471-498, :625-648)
//   :499-501  || (I - U U') y ||_2           (norm, not squared: Q9)
//   :222-225  yhat = U diag(sqrt S) Tyhat    (back-projection, k_backproject)
//
// Layouts.  Y is the caller's [N][T][p] (time-major, like the reference's vector<VectorXd>).
// The projected series is written LATENT-MAJOR, u[n][l][t], so that the scan kernels read each
// latent's time series with unit stride.  The residual norms are only ever summed over time
// (moihgp.h:503,563 through the callers' loops), so each CTA (a tile of PT = 128 time steps of one
// sequence) writes ONE partial sum rho_part[n][tile], reduced later in fixed order.
//
// k_project_mma<NB>: W[128 x L] = Ytile[128 x p] * U[p x L] on the FP64 tensor pipe (DMMA m8n8k4), K panels of 16
//   columns double-buffered through shared memory by cp.async; 8 warps x 16 rows, accumulators in registers
//   (L <= 8 NB).  The residual norm comes from ||y||^2 - ||U'y||^2 (U has orthonormal columns); rows where that
//   difference cancels (< 1e-4 ||y||^2) or is NaN are re-evaluated explicitly.  Needs p even (16-byte rows).
//   k_project_mma<8, 4> serves 64 < L <= 256 in up to four latent blocks of 64 columns.
// k_project<TP>: the scalar-FMA version for every other shape, TP = 128 time steps per CTA, 64 where that tile does not fit
//   into shared memory (L >= 186).
// k_project_rows<NB, NW, NST>: the same contraction as a PERSISTENT kernel without CTA-wide barriers in its loop.  U is
//   staged into shared memory once per CTA; every warp owns units of 16 consecutive rows of Y and its own ring of NST
//   stages, filled by TMA tensor copies (cp.async.bulk.tensor, 128-byte swizzle, mbarrier completion) NST - 1 items
//   ahead of the tensor-pipe loop.  Used for even p >= 8 and a 16-byte aligned Y whenever U (padded) and the rings of one
//   of the four configurations of try_project_rows fit into shared memory; k_project_mma serves the other such shapes.
// The residual norms are written as one partial sum per 16 rows: rho_part[n][ceil(T / 16)] (project_tiles).
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <algorithm>
#include "moihgp_device.cuh"
#include "launch.h"
#include "ls_project.cuh"
#include "ptx.cuh"

namespace moihgp {

namespace {

constexpr int PT = 128;   // time steps per CTA (k_project, k_project_mma)
constexpr int RU = 16;    // time steps per residual-norm partial sum (= rows of one warp unit of k_project_rows)
constexpr int PC = 16;    // columns of Y per staged panel
constexpr int LB = 8;     // latents accumulated in registers per pass (scalar kernel)
constexpr unsigned FULL = 0xffffffffu;

// fixed-order sum of one value per thread over the CTA; result valid in thread 0
template <int NT>
__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int i = 0; i < NT / 32; ++i) s += red[i];
    return s;
}

// grid: ceil(T / PT) * N CTAs (tile-minor).  Outputs:
//   u[n][l][t]    = S_l^-1/2 * sum_r U[r][l] y[r]          (always)
//   w[n][l][t]    = sum_r U[r][l] y[r]                      (optional, objective path)
//   yl[n][l][t]   = y[l]  (raw output l, for pv: moihgp.h:510, Q8)   (optional, objective path)
//   rho_part[n][tile] = sum over the tile of || y - U U' y ||_2      (optional)
//   rho_row[n][t] = || y_t - U U' y_t ||_2 of every row               (optional; only together with rho_part)
//   nan_info      = {flag, count}: flag set to 1 if any y is NaN; rows with a NaN are appended to nan_rows (global row
//                   index n*T + t, at most nan_cap entries) and re-projected by k_nan_fix (missing-data LS projection)
__device__ __forceinline__ void note_nan_row(int* nan_info, long long* nan_rows, long long nan_cap, long long row) {
    nan_info[0] = 1;
    const int idx = atomicAdd(nan_info + 1, 1);
    if (idx < nan_cap) nan_rows[idx] = row;
    else nan_info[0] = 2;                    // overflow: reported by the host entry points
}

template <int TP>
__global__ void __launch_bounds__(TP) k_project(const double* __restrict__ Y, const double* __restrict__ U,
                                               const double* __restrict__ S, int p, int L, long long T,
                                               double* __restrict__ u, double* __restrict__ w, double* __restrict__ yl,
                                               double* __restrict__ rho_part, double* __restrict__ rho_row, int* __restrict__ nan_info,
                                               long long* __restrict__ nan_rows, long long nan_cap) {
    extern __shared__ double sm[];
    __shared__ double red[TP / 32];
    const long long rho_tiles = (T + RU - 1) / RU;          // rho_part is [N][ceil(T / 16)]: this tile's sum goes to its first slot
    double* ys = sm;                       // [TP][PC + 1]
    double* us = ys + TP * (PC + 1);       // [PC][L]
    double* ws = us + PC * L;              // [TP][L + 1]   projected (unscaled) values of this tile
    const int tid = threadIdx.x;
    const long long tiles = (T + TP - 1) / TP;
    const long long n = blockIdx.x / tiles;
    const long long tile = blockIdx.x - n * tiles;
    const long long t0 = tile * TP;
    const long long t = t0 + tid;
    const bool live = t < T;
    const double* Yn = Y + n * T * p;
    const int rows = (int)min((long long)TP, T - t0);
    bool saw_nan = false;

    // ---- pass 1: w = U' y, LB latents at a time -----------------------------------------------
    for (int l0 = 0; l0 < L; l0 += LB) {
        double acc[LB];
#pragma unroll
        for (int j = 0; j < LB; ++j) acc[j] = 0.0;
        for (int r0 = 0; r0 < p; r0 += PC) {
            const int pc = min(PC, p - r0);
            __syncthreads();
            for (int i = tid; i < rows * pc; i += TP) {
                const int row = i / pc, col = i - row * pc;
                ys[row * (PC + 1) + col] = Yn[(t0 + row) * p + r0 + col];
            }
            for (int i = tid; i < pc * L; i += TP) us[i] = U[(size_t)r0 * L + i];
            __syncthreads();
            if (live) {
                for (int c = 0; c < pc; ++c) {
                    const double y = ys[tid * (PC + 1) + c];
                    if (l0 == 0) saw_nan = saw_nan || isnan(y);
#pragma unroll
                    for (int j = 0; j < LB; ++j)
                        if (l0 + j < L) acc[j] = fma(us[c * L + l0 + j], y, acc[j]);
                }
            }
        }
        if (live) {
#pragma unroll
            for (int j = 0; j < LB; ++j)
                if (l0 + j < L) {
                    const int l = l0 + j;
                    ws[tid * (L + 1) + l] = acc[j];
                    const size_t o = ((size_t)n * L + l) * T + t;
                    u[o] = acc[j] * (1.0 / sqrt(S[l]));
                    if (w) w[o] = acc[j];
                }
        }
    }
    if (saw_nan) note_nan_row(nan_info, nan_rows, nan_cap, n * T + t);

    // ---- pass 2: residual norm and raw y(l) ---------------------------------------------------
    if (rho_part || yl) {
        double q = 0.0;
        for (int r0 = 0; r0 < p; r0 += PC) {
            const int pc = min(PC, p - r0);
            __syncthreads();
            for (int i = tid; i < rows * pc; i += TP) {
                const int row = i / pc, col = i - row * pc;
                ys[row * (PC + 1) + col] = Yn[(t0 + row) * p + r0 + col];
            }
            for (int i = tid; i < pc * L; i += TP) us[i] = U[(size_t)r0 * L + i];
            __syncthreads();
            if (live) {
                for (int c = 0; c < pc; ++c) {
                    const double y = ys[tid * (PC + 1) + c];
                    double e = y;
                    for (int l = 0; l < L; ++l) e = fma(-us[c * L + l], ws[tid * (L + 1) + l], e);
                    q = fma(e, e, q);
                    if (yl && r0 + c < L) yl[((size_t)n * L + (r0 + c)) * T + t] = y;
                }
            }
        }
        if (rho_part) {
            if (rho_row && live) rho_row[n * T + t] = sqrt(q);
            const double s = block_sum<TP>(live ? sqrt(q) : 0.0, red);
            if (tid == 0) rho_part[n * rho_tiles + tile * (TP / RU)] = s;
        }
    }
}

// -------------------------------------------------------------------------------------------------
constexpr int MW = 8;                 // warps per CTA, 16 rows each
constexpr int MT = 32 * MW;           // threads
constexpr int KP = 16;                // columns of Y per K panel (4 k blocks)
constexpr int YROWB = KP * 8;         // bytes per row of a staged Y panel (128)

template <int NB>
struct MmaSmem {
    static constexpr int LP = 8 * NB;
    static constexpr int UPITCH = LP + 4;                   // doubles: the 4 k rows of a B fragment land in distinct bank groups
    static constexpr int YBYTES = PT * YROWB;               // one Y panel
    static constexpr int UBYTES = KP * UPITCH * 8;          // one U panel
    static constexpr int BYTES = 2 * YBYTES + 2 * UBYTES;
};

// grid: ceil(T / PT) * N CTAs (tile-minor), MT threads.  Same outputs as k_project.
// NLB > 1 (L > 64): the latents are taken in blocks of 8 NB columns, one after the other; every block streams the CTA's Y tile
// again (from L2 or HBM: at 2 flop per byte and block the product stays bound by the tensor pipe).  ||U'y||^2 of a row is
// summed over the blocks in block order, so the residual norm is as deterministic as with one block.
template <int NB, int NLB>
__global__ void __launch_bounds__(MT, NB <= 4 ? 3 : 2) k_project_mma(const double* __restrict__ Y, const double* __restrict__ U,
                                                   const double* __restrict__ S, int p, int L, long long T,
                                                   double* __restrict__ u, double* __restrict__ w, double* __restrict__ yl,
                                                   double* __restrict__ rho_part, double* __restrict__ rho_row, int* __restrict__ nan_info,
                                                   long long* __restrict__ nan_rows, long long nan_cap) {
    using SMC = MmaSmem<NB>;
    extern __shared__ __align__(16) unsigned char smraw[];
    __shared__ double red[MW];
    __shared__ double rs_s[8 * NB * NLB];           // S^-1/2 per latent (moihgp.h:181)
    __shared__ int any_bad;
    unsigned char* ysm = smraw;                                                   // [2][PT][KP] swizzled 16-byte chunks
    double* usm = reinterpret_cast<double*>(smraw + 2 * SMC::YBYTES);             // [2][KP][UPITCH]
    const int tid = threadIdx.x, lane = tid & 31, wi = tid >> 5;
    const int g4 = lane >> 2, q4 = lane & 3;
    const long long tiles = (T + PT - 1) / PT;
    const long long rho_tiles = (T + RU - 1) / RU;
    const long long n = blockIdx.x / tiles;
    const long long tile = blockIdx.x - n * tiles;
    const long long t0 = tile * PT;
    const int rows = (int)min((long long)PT, T - t0);
    const double* Yn = Y + ((size_t)n * T + t0) * p;
    const int npanels = (p + KP - 1) / KP;
    if (tid == 0) any_bad = 0;
    for (int i = tid; i < 8 * NB * NLB; i += MT) rs_s[i] = i < L ? 1.0 / sqrt(__ldg(S + i)) : 0.0;
    const bool u_vec = L % 2 == 0 && (reinterpret_cast<size_t>(U) & 15) == 0;
    const int nlb = NLB == 1 ? 1 : (L + 8 * NB - 1) / (8 * NB);

    // stage panel kp of latent block l0: Y rows [0, PT) x columns [kp*KP, kp*KP + KP) and U rows [kp*KP, +KP) x [l0, l0 + LP)
    auto stage = [&](int kp, int buf, int l0) {
        unsigned char* yb = ysm + buf * SMC::YBYTES;
        const int c0 = kp * KP;
#pragma unroll
        for (int i = 0; i < PT * (KP / 2) / MT; ++i) {
            const int q = tid + MT * i;
            const int row = q >> 3, ch = q & 7;                                   // 8 chunks of 2 columns per row
            const int col = c0 + 2 * ch;
            int bytes = row < rows ? max(0, min(2, p - col)) * 8 : 0;
            const double* src = Yn + (size_t)(row < rows ? row : 0) * p + (col < p ? col : 0);
            cp_async16_zfill(yb + row * YROWB + ((ch ^ (2 * (row & 3))) << 4), src, bytes);
        }
        double* ub = usm + buf * (SMC::UBYTES / 8);
        if (u_vec) {
            // U rows are 16-byte aligned (L even): asynchronous 16-byte copies, zero fill beyond p / L
            for (int i = tid; i < KP * (SMC::LP / 2); i += MT) {
                const int k = i / (SMC::LP / 2), l = 2 * (i - k * (SMC::LP / 2));
                const int bytes = (c0 + k < p && l0 + l < L) ? 16 : 0;
                cp_async16_zfill(ub + k * SMC::UPITCH + l, U + (size_t)(c0 + k < p ? c0 + k : 0) * L + (l0 + l < L ? l0 + l : 0), bytes);
            }
        } else {
            for (int i = tid; i < KP * SMC::LP; i += MT) {
                const int k = i / SMC::LP, l = i - k * SMC::LP;
                ub[k * SMC::UPITCH + l] = (c0 + k < p && l0 + l < L) ? __ldg(U + (size_t)(c0 + k) * L + l0 + l) : 0.0;
            }
        }
        cp_async_commit();
    };

    double sy[2] = {0.0, 0.0}, sw[2] = {0.0, 0.0};
    const int row0 = wi * 16 + g4;                                                // this lane's rows: row0, row0 + 8
    const long long tA = t0 + row0, tB = tA + 8;

    for (int lb = 0; lb < nlb; ++lb) {
        const int l0 = 8 * NB * lb;
        double acc[2][NB][2];
#pragma unroll
        for (int rb = 0; rb < 2; ++rb)
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) { acc[rb][nb][0] = 0.0; acc[rb][nb][1] = 0.0; }

        stage(0, 0, l0);
        for (int kp = 0; kp < npanels; ++kp) {
            const int buf = kp & 1;
            if (kp + 1 < npanels) { stage(kp + 1, buf ^ 1, l0); cp_async_wait<1>(); }
            else cp_async_wait<0>();
            __syncthreads();
            const unsigned char* yb = ysm + buf * SMC::YBYTES;
            const double* ub = usm + buf * (SMC::UBYTES / 8);
#pragma unroll
            for (int kb = 0; kb < KP / 4; ++kb) {
                double a[2], b[NB];
#pragma unroll
                for (int rb = 0; rb < 2; ++rb) {
                    const int row = row0 + 8 * rb;
                    a[rb] = *reinterpret_cast<const double*>(yb + row * YROWB + (((2 * kb + (q4 >> 1)) ^ (2 * (row & 3))) << 4) + ((q4 & 1) << 3));
                    if (lb == 0) sy[rb] = fma(a[rb], a[rb], sy[rb]);
                }
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) b[nb] = ub[(4 * kb + q4) * SMC::UPITCH + 8 * nb + g4];
#pragma unroll
                for (int rb = 0; rb < 2; ++rb)
#pragma unroll
                    for (int nb = 0; nb < NB; ++nb) dmma884(acc[rb][nb][0], acc[rb][nb][1], a[rb], b[nb]);   // U' y   moihgp.h:181
                // raw y(l) for l < L (pv uses it: moihgp.h:510, Q8)
                if (yl && lb == 0) {
                    const int col = kp * KP + 4 * kb + q4;
                    if (col < L) {
                        if (tA < T) yl[((size_t)n * L + col) * T + tA] = a[0];
                        if (tB < T) yl[((size_t)n * L + col) * T + tB] = a[1];
                    }
                }
            }
            __syncthreads();
        }

        // ---- outputs of the latent block ---------------------------------------------------------------
#pragma unroll
        for (int nb = 0; nb < NB; ++nb)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int l = l0 + 8 * nb + 2 * q4 + e;
                if (l < L) {
                    const double rs = rs_s[l];
#pragma unroll
                    for (int rb = 0; rb < 2; ++rb) {
                        const long long t = rb == 0 ? tA : tB;
                        const double c = acc[rb][nb][e];
                        sw[rb] = fma(c, c, sw[rb]);
                        if (t < T) {
                            const size_t o = ((size_t)n * L + l) * T + t;
                            u[o] = c * rs;
                            if (w) w[o] = c;
                        }
                    }
                }
            }
    }
    // residual norm of rows tA, tB: quad all-reduce of the two squared norms
    double rho_sum = 0.0;
    bool bad_row[2];
#pragma unroll
    for (int rb = 0; rb < 2; ++rb) {
        double ysq = sy[rb], wsq = sw[rb];
        ysq += __shfl_xor_sync(FULL, ysq, 1); ysq += __shfl_xor_sync(FULL, ysq, 2);
        wsq += __shfl_xor_sync(FULL, wsq, 1); wsq += __shfl_xor_sync(FULL, wsq, 2);
        const double q = ysq - wsq;
        const long long t = rb == 0 ? tA : tB;
        // p == L: U is square and orthogonal, (I - U U') y vanishes identically - the difference is pure cancellation and
        // the explicit form would only return rounding noise (1e-16 ||y||), for every row: rho = 0 unless y holds a NaN
        const bool square_ok = p == L && ysq == ysq;
        bad_row[rb] = t < T && !(q >= 1e-4 * ysq) && !square_ok;
        if (q4 == 0 && t < T && !bad_row[rb] && q >= 1e-4 * ysq) rho_sum += sqrt(q);
        if (rho_row && q4 == 0 && t < T && !bad_row[rb]) rho_row[n * T + t] = q >= 1e-4 * ysq ? sqrt(q) : 0.0;
    }
    if (bad_row[0] || bad_row[1]) any_bad = 1;
    __syncthreads();
    if (any_bad) {
        // explicit || y - U (U' y) ||_2 (moihgp.h:651) for the rows whose norm difference cancelled (or is NaN): one
        // lane of the quad per row, straight from global memory.  Rare.
#pragma unroll
        for (int rb = 0; rb < 2; ++rb) {
            if (bad_row[rb] && q4 == 0) {
                const double* yr = Yn + (size_t)(row0 + 8 * rb) * p;
                double wl[8 * NB * NLB];
                bool isn = false;
                for (int l = 0; l < L; ++l) {
                    double a = 0.0;
                    for (int r = 0; r < p; ++r) a = fma(__ldg(U + (size_t)r * L + l), yr[r], a);
                    wl[l] = a;
                }
                double q = 0.0;
                for (int r = 0; r < p; ++r) {
                    double e = yr[r];
                    isn = isn || isnan(e);
                    for (int l = 0; l < L; ++l) e = fma(-__ldg(U + (size_t)r * L + l), wl[l], e);
                    q = fma(e, e, q);
                }
                if (isn) note_nan_row(nan_info, nan_rows, nan_cap, n * T + t0 + row0 + 8 * rb);
                rho_sum += sqrt(q);
                if (rho_row) rho_row[n * T + t0 + row0 + 8 * rb] = sqrt(q);
            }
        }
    }
    if (rho_part) {
        const double s = block_sum<MT>(rho_sum, red);
        if (tid == 0) rho_part[n * rho_tiles + tile * (PT / RU)] = s;
    }
}

// -------------------------------------------------------------------------------------------------
// k_project_rows: persistent, one ring of TMA stages per WARP, no CTA-wide barrier after the prologue.
//   Y is described by a 2-D tensor map ([N*T rows][p columns] fp64); one item = 16 rows x KP = 16 * NBOX columns arrives as
//   NBOX boxes of 16 x 16 doubles (cp.async.bulk.tensor, SASS UTMALDG) with the 128-byte swizzle: row r of a box is 128 bytes
//   whose 16-byte chunks are XOR-ed with (r & 7), which makes the tensor-pipe fragment loads (8 rows x 4 columns per
//   instruction) hit every bank pair exactly twice - the minimum for 256 bytes.  Columns beyond p and rows beyond N*T are
//   zero-filled by the copy engine.
//   The product is taken TRANSPOSED, C[latent][time] = U'[latent][k] * Y'[k][time]: a lane then owns two consecutive time
//   steps of one latent and the latent-major outputs leave as 16-byte stores.
template <int NB>
struct RowsSmem {
    static constexpr int LP = 8 * NB;
    static constexpr int UPITCH = LP + 4;                   // doubles: the 4 k rows of a fragment land in distinct bank groups
    __host__ __device__ static constexpr int p16(int p) { return (p + 15) & ~15; }
    static constexpr int SCRATCH = 2 * 6 * 32 + 2;          // doubles per warp: [RBATCH][RSLOTS][32] partial sums + unit ids
    __host__ __device__ static constexpr size_t stage_bytes(int nbox) { return (size_t)nbox * 2048; }
    __host__ __device__ static constexpr size_t bytes(int p, int nbox, int nw, int nst) {
        return 1024 /*alignment slack*/ + (size_t)nw * nst * stage_bytes(nbox) + (size_t)p16(p) * UPITCH * 8 + (size_t)LP * 8 +
               (size_t)nw * SCRATCH * 8 + (size_t)nw * nst * 8;
    }
};

__device__ __forceinline__ bool elect_one() {
    unsigned pred;
    asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tma_load_box(void* dst_smem, const CUtensorMap* tm, int col, int row, unsigned long long* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n"
                 ::"r"(smem_u32(dst_smem)), "l"(tm), "r"(col), "r"(row), "r"(smem_u32(bar)) : "memory");
}

// Residual norms: the per-lane partial sums of ||y||^2 and ||U'y||^2 of a unit go to a per-warp scratch; every RBATCH
// units one pass over the scratch (one lane per row) forms rho_t = sqrt(||y_t||^2 - ||U'y_t||^2) and the unit sums - so the
// shuffle / square-root latency chain runs once per RBATCH units and not inside every unit's epilogue.
constexpr int RBATCH = 2;
constexpr int RSLOTS = 6;        // per lane and unit: sy[rb], sw[rb][e]

template <int NB, int NW, int NST>
__global__ void __launch_bounds__(32 * NW, 1) k_project_rows(const __grid_constant__ CUtensorMap tmY, const double* __restrict__ Y,
                                                            const double* __restrict__ U, const double* __restrict__ S, int p, int L,
                                                            long long T, unsigned units_per_seq, unsigned total_units, int nbox,
                                                            double* __restrict__ u, double* __restrict__ w, double* __restrict__ yl,
                                                            double* __restrict__ rho_part, double* __restrict__ rho_row, int* __restrict__ nan_info,
                                                            long long* __restrict__ nan_rows, long long nan_cap) {
    using SMC = RowsSmem<NB>;
    extern __shared__ unsigned char smraw_unaligned[];
    unsigned char* smraw = smraw_unaligned + ((1024u - (smem_u32(smraw_unaligned) & 1023u)) & 1023u);   // swizzle atoms are 1 KB
    const int tid = threadIdx.x, lane = tid & 31;
    const int wi = __shfl_sync(FULL, tid >> 5, 0);           // provably warp-uniform: the TMA issue path stays in uniform registers
    const int g4 = lane >> 2, q4 = lane & 3;
    const int P16 = SMC::p16(p);
    const unsigned stage_bytes = (unsigned)SMC::stage_bytes(nbox);
    unsigned char* ring = smraw + (size_t)wi * NST * stage_bytes;                             // this warp's [NST][nbox][16][128 B]
    double* usm = reinterpret_cast<double*>(smraw + (size_t)NW * NST * stage_bytes);          // [P16][UPITCH], zero beyond p / L
    double* rs_s = usm + (size_t)P16 * SMC::UPITCH;                                           // [LP] S^-1/2 (moihgp.h:181)
    double* scr = rs_s + SMC::LP + (size_t)wi * SMC::SCRATCH;                                 // this warp's [RBATCH][RSLOTS][32] + unit ids
    unsigned* scr_id = reinterpret_cast<unsigned*>(scr + RBATCH * RSLOTS * 32);               // [RBATCH][2]: sequence, unit
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(rs_s + SMC::LP + (size_t)NW * SMC::SCRATCH) + wi * NST;
    for (int i = tid; i < P16 * SMC::LP; i += 32 * NW) {
        const int k = i / SMC::LP, l = i - k * SMC::LP;
        usm[k * SMC::UPITCH + l] = (k < p && l < L) ? __ldg(U + (size_t)k * L + l) : 0.0;
    }
    if (tid < SMC::LP) rs_s[tid] = tid < L ? 1.0 / sqrt(__ldg(S + tid)) : 0.0;
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < NST; ++i) mbar_init(bars + i, 1);
        mbar_fence_init();
    }
    __syncthreads();

    const unsigned gw0 = blockIdx.x * NW + wi, gstride = gridDim.x * NW;
    const int KP = 16 * nbox;
    const int NP = (p + KP - 1) / KP;
    // units advance by gstride: (sequence, unit within it, first row) are carried along without divisions
    const unsigned dq = gstride / units_per_seq, dr = gstride - dq * units_per_seq;
    const int drow = (int)((long long)dq * T + (long long)dr * RU), wrap_row = (int)(T - (long long)units_per_seq * RU);
    // ---- producer side (lane 0): the next (unit, panel) item to fetch ----------------------------------
    unsigned ig = gw0;           // unit of the next item to issue, its row in Y[N*T][p], its panel and its stage
    int irow = (int)((long long)(gw0 / units_per_seq) * T + (long long)(gw0 % units_per_seq) * RU);
    unsigned iunit = gw0 % units_per_seq;
    int ipn = 0, ist = 0;
    auto issue_next = [&]() {
        if (ig < total_units) {
            const int c0 = ipn * KP;
            const int nb_ = min(nbox, (p - c0 + 15) >> 4);                                    // boxes that hold columns < p
            unsigned char* stg = ring + (size_t)ist * stage_bytes;
            if (elect_one()) {
                mbar_expect_tx(bars + ist, 2048u * (unsigned)nb_);
#pragma unroll 4
                for (int j = 0; j < nb_; ++j) tma_load_box(stg + j * 2048, &tmY, c0 + 16 * j, irow, bars + ist);
            }
            if (++ipn == NP) {
                ipn = 0; ig += gstride; iunit += dr; irow += drow;
                if (iunit >= units_per_seq) { iunit -= units_per_seq; irow += wrap_row; }
            }
            if (++ist == NST) ist = 0;
        }
    };
#pragma unroll
    for (int i = 0; i < NST - 1; ++i) issue_next();

    // Fragment rows: block rb of the tensor-pipe product takes the unit's time steps 2 g + rb (g = 0..7), so that a half-warp
    // (g4 = 0..3 or 4..7) reads rows whose swizzle masks (row & 7) are {0,2,4,6} or {1,3,5,7}: with the two chunks a k block
    // spans that is eight distinct 16-byte bank groups per half-warp - no conflict.  In the transposed product a lane then
    // owns time steps 4 q4 .. 4 q4 + 3 of latent 8 nb + g4: acc[rb][nb][e] is time step 4 q4 + 2 e + rb.
    unsigned yoff[2][4];
#pragma unroll
    for (int rb = 0; rb < 2; ++rb)
#pragma unroll
        for (int k3 = 0; k3 < 4; ++k3) {
            const int row = 2 * g4 + rb;
            yoff[rb][k3] = (unsigned)(row * 128 + ((((2 * k3 + (q4 >> 1)) ^ row) & 7) << 4) + ((q4 & 1) << 3));
        }
    const bool vec_ok = (T & 1) == 0;                        // latent-major rows start 16-byte aligned

    // one pass over the scratch: lane = (unit slot k, time step tau) of `nk` recorded units
    auto flush_rho = [&](int nk) {
        __syncwarp();
        const int k = lane >> 4, tau = lane & 15;
        double rho = 0.0;
        unsigned n_k = 0, unit_k = 0;
        if (k < nk) {
            n_k = scr_id[2 * k]; unit_k = scr_id[2 * k + 1];
            const double* sk = scr + (size_t)k * RSLOTS * 32;
            const long long t = (long long)unit_k * RU + tau;
            // ||y||^2: slot rb = tau & 1 of the quad g4 = tau / 2; ||U'y||^2: slot 2 + 2 rb + e of the lanes (g4 = 0..7, q4),
            // tau = 4 q4 + 2 e + rb
            const int rb = tau & 1, e = (tau >> 1) & 1, qq = tau >> 2;
            const double* py = sk + rb * 32 + 4 * (tau >> 1);
            const double ysq = (py[0] + py[1]) + (py[2] + py[3]);
            const double* pw = sk + (2 + 2 * rb + e) * 32 + qq;
            const double wsq = ((pw[0] + pw[4]) + (pw[8] + pw[12])) + ((pw[16] + pw[20]) + (pw[24] + pw[28]));
            const double q = ysq - wsq;
            if (t < T) {
                if (q >= 1e-4 * ysq) rho = sqrt(q);
                else if (p == L && ysq == ysq) rho = 0.0;      // square orthogonal U: (I - U U') y vanishes identically (see k_project_mma)
                else {
                    // explicit || y - U (U' y) ||_2 (moihgp.h:651) for a row whose norm difference cancelled (or is NaN),
                    // straight from global memory.  Rare.
                    const double* yr = Y + ((size_t)n_k * T + t) * p;
                    double wl[8 * NB];
                    bool isn = false;
                    for (int l = 0; l < L; ++l) {
                        double a = 0.0;
                        for (int r = 0; r < p; ++r) a = fma(usm[r * SMC::UPITCH + l], yr[r], a);
                        wl[l] = a;
                    }
                    double qe = 0.0;
                    for (int r = 0; r < p; ++r) {
                        double ev = yr[r];
                        isn = isn || isnan(ev);
                        for (int l = 0; l < L; ++l) ev = fma(-usm[r * SMC::UPITCH + l], wl[l], ev);
                        qe = fma(ev, ev, qe);
                    }
                    if (isn) note_nan_row(nan_info, nan_rows, nan_cap, (long long)n_k * T + t);
                    rho = sqrt(qe);
                }
            }
        }
        if (rho_row && k < nk && (long long)unit_k * RU + tau < T) rho_row[(size_t)n_k * T + (size_t)unit_k * RU + tau] = rho;
        __syncwarp();
#pragma unroll
        for (int o = 8; o >= 1; o >>= 1) rho += __shfl_xor_sync(FULL, rho, o);       // fixed-order sum over the unit's 16 rows
        if (tau == 0 && k < nk) rho_part[(size_t)n_k * units_per_seq + unit_k] = rho;
    };

    int cst = 0;                 // consumer stage and its phase parity
    unsigned cph = 0;
    int nrec = 0;                // units recorded in the scratch
    unsigned n = gw0 / units_per_seq, unit = gw0 % units_per_seq;
    for (unsigned g = gw0; g < total_units; g += gstride, n += dq, unit += dr) {
        if (unit >= units_per_seq) { unit -= units_per_seq; ++n; }
        const long long t0 = (long long)unit * RU;
        double acc[2][NB][2];    // [rb][nb][e]: latent 8 nb + g4, time step t0 + 4 q4 + 2 e + rb
#pragma unroll
        for (int rb = 0; rb < 2; ++rb)
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) { acc[rb][nb][0] = 0.0; acc[rb][nb][1] = 0.0; }
        double sy[2] = {0.0, 0.0};
        for (int pn = 0; pn < NP; ++pn) {
            issue_next();        // refills the stage consumed one item ago (every lane passed the __syncwarp that closed it)
            mbar_wait(bars + cst, cph);
            const unsigned char* ys = ring + (size_t)cst * stage_bytes;
            const int c0 = pn * KP;
            const int nbx = min(nbox, (p - c0 + 15) >> 4);
            const double* ub = usm + (size_t)(c0 + q4) * SMC::UPITCH + g4;
            for (int j = 0; j < nbx; ++j) {
#pragma unroll
                for (int k3 = 0; k3 < 4; ++k3) {
                    double yv[2], uv[NB];
                    yv[0] = *reinterpret_cast<const double*>(ys + j * 2048 + yoff[0][k3]);
                    yv[1] = *reinterpret_cast<const double*>(ys + j * 2048 + yoff[1][k3]);
                    sy[0] = fma(yv[0], yv[0], sy[0]);
                    sy[1] = fma(yv[1], yv[1], sy[1]);
#pragma unroll
                    for (int nb = 0; nb < NB; ++nb) uv[nb] = ub[(size_t)(16 * j + 4 * k3) * SMC::UPITCH + 8 * nb];
#pragma unroll
                    for (int rb = 0; rb < 2; ++rb)
#pragma unroll
                        for (int nb = 0; nb < NB; ++nb) dmma884(acc[rb][nb][0], acc[rb][nb][1], uv[nb], yv[rb]);   // (U' y)'   moihgp.h:181
                    if (yl) {    // raw y(l) for l < L (pv uses it: moihgp.h:510, Q8): this lane holds y[col] of time steps 2 g4 + rb
                        const int col = c0 + 16 * j + 4 * k3 + q4;
                        const long long tA = t0 + 2 * g4;
                        if (col < L) {
                            if (tA < T) yl[((size_t)n * L + col) * T + tA] = yv[0];
                            if (tA + 1 < T) yl[((size_t)n * L + col) * T + tA + 1] = yv[1];
                        }
                    }
                }
            }
            __syncwarp();
            if (++cst == NST) { cst = 0; cph ^= 1u; }
        }

        // ---- outputs of the unit: time steps t0 + 4 q4 .. + 3 of latent 8 nb + g4 as two 16-byte stores ------------
        const bool full = t0 + RU <= T;
        double sw[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
        const size_t o0 = ((size_t)n * L + g4) * T + t0 + 4 * q4;
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) {
            const int l = 8 * nb + g4;
            const double rs = rs_s[l];
            const size_t o = o0 + (size_t)(8 * nb) * T;
            const double c00 = acc[0][nb][0], c10 = acc[1][nb][0], c01 = acc[0][nb][1], c11 = acc[1][nb][1];   // steps +0, +1, +2, +3
            sw[0][0] = fma(c00, c00, sw[0][0]); sw[1][0] = fma(c10, c10, sw[1][0]);
            sw[0][1] = fma(c01, c01, sw[0][1]); sw[1][1] = fma(c11, c11, sw[1][1]);
            if (l < L) {
                if (full && vec_ok) {
                    *reinterpret_cast<double2*>(u + o) = make_double2(c00 * rs, c10 * rs);
                    *reinterpret_cast<double2*>(u + o + 2) = make_double2(c01 * rs, c11 * rs);
                    if (w) { *reinterpret_cast<double2*>(w + o) = make_double2(c00, c10); *reinterpret_cast<double2*>(w + o + 2) = make_double2(c01, c11); }
                } else {
                    const long long t = t0 + 4 * q4;
                    const double cv[4] = {c00, c10, c01, c11};
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (t + i < T) { u[o + i] = cv[i] * rs; if (w) w[o + i] = cv[i]; }
                }
            }
        }
        if (rho_part) {          // partial sums of the unit -> scratch; reduced every RBATCH units
            double* sk = scr + (size_t)nrec * RSLOTS * 32 + lane;
            sk[0] = sy[0]; sk[32] = sy[1]; sk[64] = sw[0][0]; sk[96] = sw[0][1]; sk[128] = sw[1][0]; sk[160] = sw[1][1];
            if (lane == 0) { scr_id[2 * nrec] = n; scr_id[2 * nrec + 1] = unit; }
            if (++nrec == RBATCH) { flush_rho(RBATCH); nrec = 0; }
        }
    }
    if (rho_part && nrec > 0) flush_rho(nrec);
}

// Missing observations (moihgp.h:167-178): every listed row gets  u = S^-1/2 (U0'U0)^-1 U0' y_obs  (and w unscaled).
// grid-stride over the list, one CTA per row, scratch in dynamic shared memory - or, where that does not fit (gsc != null,
// L >= 120), a slice of gsc[gridDim.x][ls_scratch_doubles(L)] in global memory per CTA.
__global__ void __launch_bounds__(128) k_nan_fix(const double* __restrict__ Y, const double* __restrict__ U, const double* __restrict__ S,
                                                int p, int L, long long T, const int* __restrict__ nan_info,
                                                const long long* __restrict__ nan_rows, long long nan_cap,
                                                double* __restrict__ u, double* __restrict__ w, double* __restrict__ gsc) {
    extern __shared__ double sm_sc[];
    double* sc = gsc ? gsc + (size_t)blockIdx.x * ls_scratch_doubles(L) : sm_sc;
    long long count = nan_info[1];
    if (count > nan_cap) count = nan_cap;
    for (long long i = blockIdx.x; i < count; i += gridDim.x) {
        const long long row = nan_rows[i];
        const long long n = row / T, t = row - n * T;
        const double* yr = Y + (size_t)row * p;
        ls_solve_coop(p, L, [&](int r) { return yr[r]; }, [&](int r, int l) { return __ldg(U + (size_t)r * L + l); },
                      sc, sc + L * L, sc + 2 * L * L, sc + 2 * L * L + L, reinterpret_cast<int*>(sc + 2 * L * L + 2 * L),
                      (int)threadIdx.x, (int)blockDim.x, [] { __syncthreads(); });
        for (int l = threadIdx.x; l < L; l += blockDim.x) {
            const double z = sc[2 * L * L + L + l];
            const size_t o = ((size_t)n * L + l) * T + t;
            u[o] = z * (1.0 / sqrt(S[l]));
            if (w) w[o] = z;
        }
        __syncthreads();
    }
}

// Back-projection of the filtered function values: Yhat[n][t][r] = sum_l U[r][l] sqrt(S_l) X[n][t][l][0]
// (ihgp.h:51 yhat = xnew(0); moihgp.h:222-225).  grid: ceil(T / PT) * N CTAs.  U_SMEM: U sqrt(S) staged in shared memory; for
// shapes where it does not fit next to the tile of function values (p L > ~20 000) it is read through the L1/L2 instead.
// TP: time steps per CTA; 32 where the 128-step tile of function values alone would pass 200 KB (L >= 198).
template <bool U_SMEM, int TP>
__global__ void __launch_bounds__(128) k_backproject(const double* __restrict__ X, const double* __restrict__ U,
                                                   const double* __restrict__ S, int p, int L, int d, long long T,
                                                   double* __restrict__ Yhat) {
    extern __shared__ double sm[];
    double* fs = sm;                          // [TP][L + 1]
    double* sq = fs + (size_t)TP * (L + 1);   // [L] sqrt(S)
    double* us = sq + L;                      // [p][L] scaled by sqrt(S)   (U_SMEM only)
    const int tid = threadIdx.x;
    const long long tiles = (T + TP - 1) / TP;
    const long long n = blockIdx.x / tiles;
    const long long t0 = (blockIdx.x - n * tiles) * TP;
    const int rows = (int)min((long long)TP, T - t0);
    for (int i = tid; i < L; i += 128) sq[i] = sqrt(S[i]);
    if (U_SMEM) for (int i = tid; i < p * L; i += 128) us[i] = U[i] * sqrt(S[i % L]);
    const double* Xn = X + ((size_t)n * T + t0) * L * d;
    for (int i = tid; i < rows * L; i += 128) fs[(i / L) * (L + 1) + (i % L)] = Xn[(size_t)i * d];
    __syncthreads();
    double* Yo = Yhat + ((size_t)n * T + t0) * p;
    for (int i = tid; i < rows * p; i += 128) {
        const int row = i / p, r = i - row * p;
        double s = 0.0;
        if (U_SMEM) for (int l = 0; l < L; ++l) s = fma(us[r * L + l], fs[row * (L + 1) + l], s);
        else for (int l = 0; l < L; ++l) s = fma(__ldg(U + (size_t)r * L + l) * sq[l], fs[row * (L + 1) + l], s);
        Yo[i] = s;
    }
}

template <int NB, int NLB>
cudaError_t run_project_mma(const double* Y, const double* U, const double* S, int p, int L, long long N, long long T, double* u,
                            double* w, double* yl, double* rho_part, double* rho_row, int* nan_info, long long* nan_rows, long long nan_cap,
                            cudaStream_t stream) {
    using SMC = MmaSmem<NB>;
    static std::atomic<int> attr_done[64];          // per device: function attributes belong to the device's context
    if (AttrOnce once(attr_done); once) cudaFuncSetAttribute(k_project_mma<NB, NLB>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMC::BYTES);
    const unsigned grid = (unsigned)(((T + PT - 1) / PT) * N);
    k_project_mma<NB, NLB><<<grid, MT, SMC::BYTES, stream>>>(Y, U, S, p, L, T, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap);
    return cudaGetLastError();
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) f = nullptr;
        return reinterpret_cast<EncodeTiledFn>(f);
    }();
    return fn;
}

template <int NB, int NW, int NST>
cudaError_t run_project_rows(const CUtensorMap& tm, const double* Y, const double* U, const double* S, int p, int L, long long N, long long T,
                             int nbox, double* u, double* w, double* yl, double* rho_part, double* rho_row, int* nan_info, long long* nan_rows,
                             long long nan_cap, cudaStream_t stream) {
    using SMC = RowsSmem<NB>;
    const size_t smem = SMC::bytes(p, nbox, NW, NST);
    static std::atomic<int> attr_done[64];
    if (AttrOnce once(attr_done); once) cudaFuncSetAttribute(k_project_rows<NB, NW, NST>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    const long long ups = (T + RU - 1) / RU, total = ups * N;
    const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(4, (size_t)(227 * 1024) / (smem + 1024)));
    const long long grid = std::min<long long>((total + NW - 1) / NW, 148LL * per_sm);
    k_project_rows<NB, NW, NST><<<(unsigned)grid, 32 * NW, smem, stream>>>(tm, Y, U, S, p, L, T, (unsigned)ups, (unsigned)total, nbox, u, w, yl,
                                                                           rho_part, rho_row, nan_info, nan_rows, nan_cap);
    return cudaGetLastError();
}

// the first configuration (warps, stages, boxes per stage), in order of falling ring size, whose rings fit into 227 KB
// beside U: 1 = (16, 2, up to 2), 2 = (16, 3, 1), 5 = (8, 2, up to 2), 8 = (8, 2, 1); false = shape not served by
// k_project_rows
template <int NB>
bool try_project_rows(cudaError_t& e, const double* Y, const double* U, const double* S, int p, int L, long long N, long long T, double* u,
                      double* w, double* yl, double* rho_part, double* rho_row, int* nan_info, long long* nan_rows, long long nan_cap, cudaStream_t stream) {
    using SMC = RowsSmem<NB>;
    const size_t cap = 227 * 1024;
    const long long rows = N * T, ups = (T + RU - 1) / RU;
    if (rows >= (1LL << 31) || ups * N >= (1LL << 31) || !encode_tiled_fn()) return false;
    const int nb_all = (p + 15) / 16;
    const int nb_narrow = nb_all < 2 ? nb_all : 2;
    alignas(64) CUtensorMap tm;
    const cuuint64_t gdim[2] = {(cuuint64_t)p, (cuuint64_t)rows};
    const cuuint64_t gstr[1] = {(cuuint64_t)p * 8};
    const cuuint32_t box[2] = {16, (cuuint32_t)RU}, estr[2] = {1, 1};
    if (encode_tiled_fn()(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(Y), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return false;
#define MOIHGP_TRY_ROWS(NW_, NST_, NBOX_)                                                                                           \
    if (SMC::bytes(p, NBOX_, NW_, NST_) <= cap) {                                                                                   \
        e = run_project_rows<NB, NW_, NST_>(tm, Y, U, S, p, L, N, T, NBOX_, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap, stream); \
        return true;                                                                                                                \
    }
    MOIHGP_TRY_ROWS(16, 2, nb_narrow)   // 1
    MOIHGP_TRY_ROWS(16, 3, 1)           // 2
    MOIHGP_TRY_ROWS(8, 2, nb_narrow)    // 5
    MOIHGP_TRY_ROWS(8, 2, 1)            // 8
#undef MOIHGP_TRY_ROWS
    return false;
}

}  // namespace

size_t project_tiles(long long T) { return (size_t)((T + RU - 1) / RU); }

// k_nan_fix keeps the scratch of the missing-output solve in shared memory up to this size, in ls_global_doubles(L) of global
// memory beyond it (one slice per CTA of a grid of NANFIX_GLOBAL_CTAS)
constexpr size_t NANFIX_SMEM_MAX = 227 * 1024;
constexpr int NANFIX_GLOBAL_CTAS = 148;
size_t ls_global_doubles(int L) {
    return sizeof(double) * (size_t)ls_scratch_doubles(L) <= NANFIX_SMEM_MAX ? 0 : (size_t)NANFIX_GLOBAL_CTAS * ls_scratch_doubles(L);
}

cudaError_t launch_project(const double* Y, const double* U, const double* S, int p, int L, long long N, long long T,
                           double* u, double* w, double* yl, double* rho_part, double* rho_row, int* nan_info, long long* nan_rows, long long nan_cap,
                           double* ls_scratch, cudaStream_t stream) {
    const bool aligned = (reinterpret_cast<size_t>(Y) & 15) == 0;
    const bool mma_ok = p % 2 == 0 && aligned && p >= 8;
    cudaError_t e = cudaSuccess;
    bool done = false;
    if (mma_ok && L <= 64) {
        if (L <= 8) done = try_project_rows<1>(e, Y, U, S, p, L, N, T, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap, stream);
        else if (L <= 16) done = try_project_rows<2>(e, Y, U, S, p, L, N, T, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap, stream);
        else if (L <= 32) done = try_project_rows<4>(e, Y, U, S, p, L, N, T, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap, stream);
        else done = try_project_rows<8>(e, Y, U, S, p, L, N, T, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap, stream);
    }
    // the tile kernels write one partial sum per 128 (k_project<64>: 64) steps into the first of its slots: clear the others
    if (!done && rho_part) cudaMemsetAsync(rho_part, 0, sizeof(double) * (size_t)N * project_tiles(T), stream);
    if (done) {
    } else if (mma_ok && L <= 64) {
        if (L <= 8) e = run_project_mma<1, 1>(Y, U, S, p, L, N, T, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap, stream);
        else if (L <= 16) e = run_project_mma<2, 1>(Y, U, S, p, L, N, T, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap, stream);
        else if (L <= 32) e = run_project_mma<4, 1>(Y, U, S, p, L, N, T, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap, stream);
        else e = run_project_mma<8, 1>(Y, U, S, p, L, N, T, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap, stream);
    } else if (mma_ok && L <= MAX_LATENT) {
        e = run_project_mma<8, MAX_LATENT / 64>(Y, U, S, p, L, N, T, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap, stream);
    } else {
        // odd p or a Y that is not 16-byte aligned: the scalar kernel, with 64-step tiles where the 128-step tile does not fit
        auto smem_of = [&](int tp) { return sizeof(double) * ((size_t)tp * (PC + 1) + (size_t)PC * L + (size_t)tp * (L + 1)); };
        if (smem_of(PT) <= 227 * 1024) {
            const size_t smem = smem_of(PT);
            if (smem > 48 * 1024) cudaFuncSetAttribute(k_project<PT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            const unsigned grid = (unsigned)(((T + PT - 1) / PT) * N);
            k_project<PT><<<grid, PT, smem, stream>>>(Y, U, S, p, L, T, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap);
        } else {
            const size_t smem = smem_of(PT / 2);
            cudaFuncSetAttribute(k_project<PT / 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            const unsigned grid = (unsigned)(((T + PT / 2 - 1) / (PT / 2)) * N);
            k_project<PT / 2><<<grid, PT / 2, smem, stream>>>(Y, U, S, p, L, T, u, w, yl, rho_part, rho_row, nan_info, nan_rows, nan_cap);
        }
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return e;
    // missing-data rows (usually none: the kernel then exits at once)
    if (ls_global_doubles(L) == 0) {
        const size_t sc = sizeof(double) * (size_t)ls_scratch_doubles(L);
        if (sc > 48 * 1024) cudaFuncSetAttribute(k_nan_fix, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc);
        k_nan_fix<<<592, 128, sc, stream>>>(Y, U, S, p, L, T, nan_info, nan_rows, nan_cap, u, w, nullptr);
    } else {
        if (!ls_scratch) return cudaErrorInvalidValue;
        k_nan_fix<<<NANFIX_GLOBAL_CTAS, 128, 0, stream>>>(Y, U, S, p, L, T, nan_info, nan_rows, nan_cap, u, w, ls_scratch);
    }
    return cudaGetLastError();
}

cudaError_t launch_backproject(const double* X, const double* U, const double* S, int p, int L, int d, long long N,
                               long long T, double* Yhat, cudaStream_t stream) {
    const size_t base = sizeof(double) * ((size_t)PT * (L + 1) + L), full = base + sizeof(double) * (size_t)p * L;
    const unsigned grid = (unsigned)(((T + PT - 1) / PT) * N);
    if (full <= 200 * 1024) {
        if (full > 48 * 1024) cudaFuncSetAttribute(k_backproject<true, PT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)full);
        k_backproject<true, PT><<<grid, PT, full, stream>>>(X, U, S, p, L, d, T, Yhat);
    } else if (base <= 200 * 1024) {
        if (base > 48 * 1024) cudaFuncSetAttribute(k_backproject<false, PT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)base);
        k_backproject<false, PT><<<grid, PT, base, stream>>>(X, U, S, p, L, d, T, Yhat);
    } else {
        // L >= 198: 32 time steps per CTA (about 66 KB of function values at L = 256), U read through L1 / L2
        constexpr int TPW = 32;
        const size_t small = sizeof(double) * ((size_t)TPW * (L + 1) + L);
        cudaFuncSetAttribute(k_backproject<false, TPW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small);
        k_backproject<false, TPW><<<(unsigned)(((T + TPW - 1) / TPW) * N), 128, small, stream>>>(X, U, S, p, L, d, T, Yhat);
    }
    return cudaGetLastError();
}

}  // namespace moihgp
