/* moihgp_b200.h - C ABI of libmoihgp.so, the B200-native (sm_100a) drop-in for the hot path of
 * lim271/MultiOutputIHGP: the OILMM-decoupled steady-state Kalman filter, smoother and
 * negative-log-likelihood / gradient evaluation.
 *
 * Two groups of entry points:
 *
 *  (1) LEGACY symbols - exactly the 26 symbols of the reference's moihgp/src/wrapper.cpp
 *      (gp32_* at wrapper.cpp:31-326, gp52_* at :329-624) with the same signatures, argument
 *      layouts and (absent) error convention, so that the reference's moihgp/pywrapper.py
 *      (ctypes bindings at pywrapper.py:28-145) loads this library unchanged.  One observation
 *      per call; each call is one small kernel launch on the GPU.  One extension: gpXX_step1 / gpXX_step2 accept
 *      y == NULL and then take the prediction step with the derivative states (xnew = A x, dxnew_k = dA_k x + A dx_k:
 *      IHGP::step's NaN branch, ihgp.h:39-47), which the reference's wrapper cannot express.
 *
 *  (2) WHOLE-SEQUENCE symbols (moihgp_cuda_*) - the device boundary moved up to where the
 *      reference's callers loop over observations:
 *        RegressionObjective::operator()   moihgp/include/moihgp/moihgp_regression.h:34-52
 *        OnlineObjective::operator()       moihgp/include/moihgp/moihgp_online.h:40-72
 *        MOIHGPRegression::predict         moihgp/include/moihgp/moihgp_regression.h:127-139
 *        IHGP::backwardSmoother            moihgp/include/moihgp/ihgp.h:103-114
 *      These return an int status (0 = ok); moihgp_cuda_last_error() gives the message.
 *
 * All arrays are C-contiguous IEEE fp64.  Layouts (as wrapper.cpp:51-93 / pywrapper.py:146-167):
 *   x, xnew   [L][d]            filter state per latent (d = 2 Matern-3/2, 3 Matern-5/2)
 *   dx, dxnew [L][3][d]         its derivative w.r.t. (magnitude, lengthscale, noise)
 *   y, yhat   [p]               one observation (NaN = missing, moihgp.h:154)
 *   params, grad [p*L + L + 1 + 3L] = [ U row-major | S | sigma | (magnitude, lengthscale, noise) x L ]
 *                               (moihgp.h:436-456, :721-738)
 *   Y, Yhat   [N][T][p]         N independent sequences, time-major like the reference's vector<VectorXd>
 *   X, Xs     [N][T][L][d]      filtered (post-update) / smoothed states
 * There is no CPU fallback: every entry point needs a CUDA device of compute capability 10.0.
 */
#ifndef MOIHGP_B200_H
#define MOIHGP_B200_H

#include <stdbool.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ (1) legacy symbols */
typedef struct moihgp_handle GP32;   /* wrapper.cpp:21 */
typedef struct moihgp_handle GP52;   /* wrapper.cpp:22 (bound to Matern-3/2 there too, SURVEY Q7; see MOIHGP_GP52_MATERN52) */

#define MOIHGP_LEGACY_DECL(XX, GP)                                                                                          \
    GP* gp##XX##_new(double dt, size_t num_output, size_t num_latent, bool threading);        /* wrapper.cpp:31  / :329 */  \
    void gp##XX##_del(GP* gp);                                                                /* wrapper.cpp:37  / :335 */  \
    void gp##XX##_step1(GP* gp, double* x, double* y, double* dx, double* xnew, double* yhat, double* dxnew); /* :43  / :341 */ \
    void gp##XX##_step2(GP* gp, double* x, double* y, double* dx, double* xnew, double* dxnew);               /* :98  / :396 */ \
    void gp##XX##_step3(GP* gp, double* x, double* y, double* xnew, double* yhat);            /* wrapper.cpp:148 / :446 */  \
    void gp##XX##_step4(GP* gp, double* x, double* xnew, double* yhat);                       /* wrapper.cpp:187 / :485 */  \
    void gp##XX##_update(GP* gp, double* params);                                             /* wrapper.cpp:224 / :522 */  \
    double gp##XX##_lik1(GP* gp, double* x, double* y, double* dx, double* grad);             /* wrapper.cpp:232 / :530 */  \
    double gp##XX##_lik2(GP* gp, double* x, double* y);                                       /* wrapper.cpp:273 / :571 */  \
    void gp##XX##_get_params(GP* gp, double* params);                                         /* wrapper.cpp:300 / :598 */  \
    size_t gp##XX##_igp_dim(GP* gp);                                                          /* wrapper.cpp:311 / :609 */  \
    size_t gp##XX##_num_param(GP* gp);                                                        /* wrapper.cpp:317 / :615 */  \
    size_t gp##XX##_num_igp_param(GP* gp);                                                    /* wrapper.cpp:323 / :621 */

MOIHGP_LEGACY_DECL(32, GP32)
MOIHGP_LEGACY_DECL(52, GP52)

/* ------------------------------------------------------------------ (2) whole-sequence symbols */
typedef struct moihgp_handle moihgp_handle;

enum { MOIHGP_MATERN32 = 32, MOIHGP_MATERN52 = 52 };
/* smoother modes: the reference's IHGP::backwardSmoother as written (ihgp.h:103-114, SURVEY Q3),
 * or the Rauch-Tung-Striebel recursion on the same steady-state quantities (our extension). */
enum { MOIHGP_SMOOTH_NONE = -1, MOIHGP_SMOOTH_REFERENCE_LITERAL = 0, MOIHGP_SMOOTH_RTS = 1 };

/* MOIHGP<StateSpace>(dt, num_output, num_latent, threading)  moihgp.h:81-136.
 * U starts as the p x L identity block (the reference draws a random near-identity U, moihgp.h:105-125:
 * use the legacy gpXX_new for that behaviour), S = 1, sigma = 1e-2, latents at (1, 1, 0.1).
 * `threading` only selects the reference's loss semantics (moihgp.h:588 vs :601, forced off for L < 2). */
int moihgp_cuda_create(moihgp_handle** out, int kernel, double dt, size_t num_output, size_t num_latent,
                       int threading, int device);
/* Limits the reference does not have: 1 <= num_latent <= min(num_output, 256); the streaming learner (moihgp_cuda_online_begin)
 * takes num_latent <= 64.  Every entry point runs on the handle's device
 * and restores the caller's current CUDA device before it returns. */
void moihgp_cuda_destroy(moihgp_handle* h);
/* run every kernel of this handle on `cuda_stream` (a cudaStream_t); NULL = the handle's own (non-blocking) stream.
 * To share the legacy default stream pass cudaStreamLegacy ((cudaStream_t)0x1), not 0. */
int moihgp_cuda_set_stream(moihgp_handle* h, void* cuda_stream);
int moihgp_cuda_sync(moihgp_handle* h);
const char* moihgp_cuda_last_error(moihgp_handle* h);
/* per-kernel device timing: while enabled, a CUDA event is recorded on the launching stream after every kernel of
 * the whole-sequence entry points; _read() returns "name total_ms launches" lines accumulated since it was enabled
 * (and clears the record).  Used by bench.py for the roofline figures; off by default. */
int moihgp_cuda_profile(moihgp_handle* h, int enable);
const char* moihgp_cuda_profile_read(moihgp_handle* h);
/* which kernels serve a call; 0 = automatic everywhere.  Results agree to rounding; used by the parity tests to cover
 * every variant.  The setting has three effects:
 *   - the fused pass (moihgp_cuda_filter_smoother_nll*): 0 = the many-chains kernels when there are enough independent
 *     (sequence, latent) chains and the shape is instantiated, else the time-parallel chunked scan; 1 = chunked scan;
 *     2 = many-chains (fails if unavailable);
 *   - the posterior sampler (moihgp_cuda_sample_posterior*): 1 = time-chunked, 2 = one pass per chain, 0 = by the number
 *     of chains.  Its mean pass follows the fused-pass choice, except that 2 takes the chunked scan where the many-chains
 *     kernels are unavailable instead of failing;
 *   - the host-buffer objective (moihgp_cuda_objective, moihgp_cuda_objective_bound): 1 sends a single short sequence
 *     to the general kernels instead of the one-launch kernel; 0 and 2 leave the one-launch kernel in use. */
int moihgp_cuda_set_path(moihgp_handle* h, int path);
/* tuning knob of the many-chains kernels: sequences handled per warp (a power of two <= 32 / num_latent);
 * 0 = automatic (a full warp, 32 / num_latent sequences, whatever the batch size) */
int moihgp_cuda_set_chain_seqs_per_warp(moihgp_handle* h, int n);
/* kernels launched by this handle since creation (bench.py's gpu_launches) */
long long moihgp_cuda_launch_count(moihgp_handle* h);

/* Missing observations (NaN) are found on the device.  The host-buffer entry points report an overflow of the
 * re-projection list (> 2^22 rows with missing outputs in one call) through their status; the asynchronous *_dev entry
 * points cannot (they do not wait for the device) - ask afterwards: *status = 0 none seen, 1 some (handled), 2 overflow (the
 * rows beyond 2^22 keep u = NaN).  Waits for the handle's stream. */
int moihgp_cuda_nan_status(moihgp_handle* h, int* status);

size_t moihgp_cuda_igp_dim(moihgp_handle* h);         /* MOIHGP::getIGPDim      moihgp.h:691 */
size_t moihgp_cuda_num_param(moihgp_handle* h);       /* MOIHGP::getNumParam    moihgp.h:709 */
size_t moihgp_cuda_num_igp_param(moihgp_handle* h);   /* MOIHGP::getNumIGPParam moihgp.h:715 */

/* MOIHGP::update(params)  moihgp.h:431-457 -> IHGP::update  ihgp.h:117-201 (K-setup kernel) */
int moihgp_cuda_update(moihgp_handle* h, const double* params);
/* MOIHGP::getParams()  moihgp.h:721-738 */
int moihgp_cuda_get_params(moihgp_handle* h, double* params);
/* U (p x L row-major), the polar factor held by the model  moihgp.h:741 */
int moihgp_cuda_get_U(moihgp_handle* h, double* U);
/* IHGP public members of latent l after update (ihgp.h:243-254), flat:
 *   A[d*d] Q[d*d] K[d] S PF[d*d] HA[d] AKHA[d*d], then for k = 0..2: dS dA[d*d] dK[d] dAKHA[d*d] HdA[d]
 * (matrices row-major).  Returns the number of doubles written (<= cap) or a negative status. */
long long moihgp_cuda_latent_consts(moihgp_handle* h, size_t l, double* out, size_t cap);
/* iteration counts / converged flags the reference discards (ihgp.h:125,187):
 * out[0] DARE iterations, out[1..3] DLyap iterations, out[4] DARE converged, out[5..7] DLyap converged */
int moihgp_cuda_latent_iters(moihgp_handle* h, size_t l, int* out8);
/* smoother gain G and smoothed covariance P of latent l (IHGP::backwardSmoother outputs, ihgp.h:105-107), d x d row-major */
int moihgp_cuda_smoother_consts(moihgp_handle* h, size_t l, int mode, double* G, double* P);

/* The fused pass on N independent sequences, HOST buffers (copies inside the call):
 *   filter  : X[n][t] = state after observation t   (loop of MOIHGP::step v3, moihgp_regression.h:127-139)
 *   Yhat    : U sqrt(S) X[.][0]                     (moihgp.h:222-225)
 *   nll[n]  : sum_t MOIHGP::negLogLikelihood(x_t, y_t) on the pre-update state (moihgp.h:614-688)
 *   smoother: Xs per `smoother_mode`                (IHGP::backwardSmoother, ihgp.h:103-114)
 * x0 [N][L][d] carried-in state (NULL = zeros); X, Xs, Yhat, nll, xT may each be NULL. */
int moihgp_cuda_filter_smoother_nll(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0,
                                    int smoother_mode, double* X, double* Xs, double* Yhat, double* nll, double* xT);
/* same pass, but only the FUNCTION-VALUE component H x = x(0) of every filtered / smoothed state crosses PCIe:
 * F, Fs [N][T][L] (what predict-style callers consume: yhat = U sqrt(S) x(0), moihgp.h:222-225) - d times fewer bytes out. */
int moihgp_cuda_filter_smoother_nll_values(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0,
                                           int smoother_mode, double* F, double* Fs, double* Yhat, double* nll, double* xT);
/* same, DEVICE buffers already resident in HBM; asynchronous on the handle's stream: no host synchronisation, also right
 * after moihgp_cuda_update, so the call can be captured into a CUDA graph once its workspaces exist (one warm-up call with
 * the same sizes on the same stream; moihgp_cuda_set_stream refuses to move the handle onto a stream that is capturing) */
int moihgp_cuda_filter_smoother_nll_dev(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0,
                                        int smoother_mode, double* X, double* Xs, double* Yhat, double* nll, double* xT);

/* Per-step NLL terms of the filter pass (no smoother, no states written):
 *   nll_steps[n][t] = MOIHGP::negLogLikelihood(x_{t-1}, y_t)  (moihgp.h:614-688), the term the fused pass sums into nll[n]:
 *                     1/2 ||y_t - U U' y_t|| / sigma + sum_l 1/2 v_{l,t}^2 / S_l + the per-step constant + 1/2 sum_l log S_l
 * A row with a missing output (NaN) gives a NaN term, as in the reference, and the least-squares projection carries the
 * filter on (moihgp_cuda_nan_status); the other terms stay finite.  Summed over t the terms give nll[n] up to rounding.
 * nll_steps [N][T] is required; nll [N] and xT [N][L][d] may be NULL; x0 as for the fused pass.  moihgp_cuda_set_path 1 / 2
 * forces the chunked scan / the many-chains kernels as for the fused pass (the many-chains kernels then take a full warp of
 * sequences whatever moihgp_cuda_set_chain_seqs_per_warp says).
 *   _dev : DEVICE buffers, asynchronous on the handle's stream (capturable into a CUDA graph like the fused pass).
 * The host-buffer twin copies in, calls the _dev entry point and copies out. */
int moihgp_cuda_nll_steps_dev(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, double* nll_steps,
                              double* nll, double* xT);
int moihgp_cuda_nll_steps(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, double* nll_steps,
                          double* nll, double* xT);

/* IHGP::backwardSmoother(X, Xprev, P, G) (ihgp.h:103-114) for every latent, over CALLER-SUPPLIED filtered states
 * X[N][T][L][d] (not necessarily produced by this library): Xs[N][T][L][d] per `smoother_mode` (0 = the reference's
 * recursion as written, 1 = RTS).  G and P of each latent come from moihgp_cuda_smoother_consts.  HOST / DEVICE buffers. */
int moihgp_cuda_smooth(moihgp_handle* h, const double* X, size_t N, size_t T, int smoother_mode, double* Xs);
int moihgp_cuda_smooth_dev(moihgp_handle* h, const double* X, size_t N, size_t T, int smoother_mode, double* Xs);

/* Posterior sample paths of the latent processes (steady-state forward-filtering, backward-sampling in RTS form):
 *   x~[T-1] = Xs[T-1] + e[T-1],  e[T-1] = LF z[T-1],   x~[t] = Xs[t] + e[t],  e[t] = G e[t+1] + LC z[t]
 * with Xs the RTS-smoothed mean (MOIHGP_SMOOTH_RTS), G = its gain, LF LF' = PF and LC LC' = PF - G (A PF A' + Q) G'.
 * z[t] is d standard normals from ONE Philox4x32-10 call with counter (t, n, l, s) and key (seed & 0xffffffff, seed >> 32):
 * uniforms u_i = (w_i + 0.5) 2^-32, Box-Muller in fp64 (z_2k = r cos(2 pi u_2k+1), z_2k+1 = r sin(2 pi u_2k+1),
 * r = sqrt(-2 ln u_2k)), the first d of z0..z3.  A draw depends on (seed, s, n, l, t) only; T, N and S must be < 2^32.
 * The noise process is the steady-state one, the approximation the smoother itself makes.
 *   _dev : DEVICE buffers, asynchronous on the handle's stream (capturable into a CUDA graph like the fused pass).  Runs the
 *          fused pass with MOIHGP_SMOOTH_RTS into Xs_mean [N][T][L][d] (NULL = a workspace), then the sampler.
 *   Xsamp [S][N][T][L][d], Fsamp [S][N][T][L] (x~(0)), Ysamp [S][N][T][p] (U sqrt(S) x~(0), noise-free outputs): any may be
 *   NULL, not all three.  Missing observations (NaN) are handled as in the fused pass (moihgp_cuda_nan_status).
 *   moihgp_cuda_set_path also selects the sampler's variant.
 * The host-buffer twin copies in, calls the _dev entry point and copies out. */
int moihgp_cuda_sample_posterior_dev(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, size_t S,
                                     unsigned long long seed, double* Xs_mean, double* Xsamp, double* Fsamp, double* Ysamp);
int moihgp_cuda_sample_posterior(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, size_t S,
                                 unsigned long long seed, double* Xs_mean, double* Xsamp, double* Fsamp, double* Ysamp);
/* the sampler's factors LF, LC of latent l (lower-triangular, d x d row-major; either may be NULL) */
int moihgp_cuda_sampler_consts(moihgp_handle* h, size_t l, double* LF, double* LC);
/* The sampler on one contiguous BLOCK of a longer sequence sharded in time (DESIGN 4.8, 6).  DEVICE buffers, asynchronous on
 * the handle's stream, capturable into a CUDA graph.  The block holds steps t0 .. t0 + T - 1 of the sequence (the Philox
 * counter is the global step, so the draws are those of the whole-sequence call); seq_end = 1 on the block that ends it.
 * Xs_mean [N][T][L][d] is the block's RTS mean: phase 3 of moihgp_cuda_fsn_block_async with smoother_mode = 1.  Two phases:
 *   1  dev_out [S][N][L][d] = e at the block's first step from a zero e_end (from LF z on the block that ends the sequence).
 *      Xs_mean may be NULL.
 *      -> caller: all-gather dev_out of every block into gathered [G][S N][L][d], then this block's
 *         e_end = moihgp_cuda_fsn_carry_dev(h, 1, 1, gathered, G, block_lengths, rank, S * N, NULL, e_end, NULL)
 *         (the backward exchange of the RTS smoother: the layout [S][N][L][d] is [S N][L][d])
 *   2  e_end [S][N][L][d] (NULL on the block that ends the sequence): Xsamp, Fsamp, Ysamp of the block, laid out as in
 *      moihgp_cuda_sample_posterior_dev with T steps; any may be NULL, not all three.
 * t0 + T <= 2^32 and S N < 2^32.  moihgp_cuda_set_path selects the variant as for the whole sequence. */
int moihgp_cuda_sample_block_async(moihgp_handle* h, int phase, const double* Xs_mean, size_t N, size_t T, unsigned long long t0, int seq_end,
                                   size_t S, unsigned long long seed, const double* e_end, double* Xsamp, double* Fsamp, double* Ysamp,
                                   double* dev_out);

/* RegressionObjective::operator() / OnlineObjective::operator() window loop over N sequences
 * (moihgp_regression.h:42-50, moihgp_online.h:61-70): loss = sum_n sum_t negLogLikelihood(x, y, dx, grad)
 * with MOIHGP::step v2 advancing (x, dx); grad[num_param] summed the same way.  x0 [N][L][d] and
 * dx0 [N][L][3][d] are the carried-in state (NULL = zeros); xT / dxT receive the final state (may be NULL).
 * HOST buffers. */
int moihgp_cuda_objective(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, const double* dx0,
                          double* loss, double* grad, double* xT, double* dxT);
/* The optimiser evaluates the objective many times on the SAME observations (LBFGSB.h:137, LineSearchMoreThuente.h:212,
 * :295): bind_data copies Y[N][T][p] to the device once (Y = NULL unbinds), objective_bound evaluates on the bound data
 * at the handle's current parameters.  The caller must re-bind after changing the observations. */
int moihgp_cuda_bind_data(moihgp_handle* h, const double* Y, size_t N, size_t T);
int moihgp_cuda_objective_bound(moihgp_handle* h, const double* x0, const double* dx0, double* loss, double* grad,
                                double* xT, double* dxT);
/* same, DEVICE buffers (loss[1], grad[num_param] on the device); asynchronous on the handle's stream */
int moihgp_cuda_objective_dev(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, const double* dx0,
                              double* loss, double* grad, double* xT, double* dxT);

/* The streaming learner with its data resident on the device (SURVEY 8 f2; OnlineObjective, moihgp_online.h:18-115):
 *   online_begin        window of `windowsize` observations, moving mean, carried state (zeros), proximal term (identity
 *                       around the current parameters) - all in device memory
 *   online_push         OnlineObjective::push_back(y)   moihgp_online.h:75-93: append, recompute the mean, slide the window
 *                       and advance the carried state with the new front element (Q12).  ma_given = NULL: the window mean
 *                       (the reference's C++ learner); else the caller's centre (online_learning.py keeps an exponential
 *                       mean).  ma_out (or NULL) receives the centre in use.
 *   online_set_proximal oldparams and the matrix B of the term 1/2 dparams' B dparams (:42-54); B = NULL: the identity;
 *                       oldparams = NULL: no proximal term on the device (the caller adds its own)
 *   online_objective    OnlineObjective::operator()     moihgp_online.h:40-72 at `params`: update + window loop + proximal
 *                       term; ONE CUDA-graph launch per evaluation (H2D params, polar factor, K-setup, window objective,
 *                       proximal term, D2H [loss, grad]).  The model then holds `params`, as after moihgp_cuda_update.
 *   online_get_state    the state carried in front of the window. */
int moihgp_cuda_online_begin(moihgp_handle* h, size_t windowsize);
int moihgp_cuda_online_push(moihgp_handle* h, const double* y, const double* ma_given, double* ma_out);
int moihgp_cuda_online_set_proximal(moihgp_handle* h, const double* oldparams, const double* B);
int moihgp_cuda_online_objective(moihgp_handle* h, const double* params, double* loss, double* grad);
int moihgp_cuda_online_get_state(moihgp_handle* h, double* x, double* dx);

/* ONE long sequence sharded over several devices in TIME (one process per GPU): every device holds a contiguous block of
 * T steps, DEVICE buffers.  begin projects the block and returns (HOST, zend[N][L][4][d] = [x; dx_0; dx_1; dx_2]) its end
 * state from a ZERO carry-in - needs T % 256 == 0; pass NULL on the last block, whose end state nobody needs.  The caller
 * exchanges the end states, forms this block's true carry-in (z_in(g+1) = T(n_g) z_in(g) + zend_g, see
 * multioutputihgp_b200/parallel.py) and calls finish, which evaluates loss / grad of the block from that carry-in reusing
 * the projection of begin; the blocks' [loss, grad] are then summed (all-reduce). */
int moihgp_cuda_objective_begin_dev(moihgp_handle* h, const double* Y, size_t N, size_t T, double* zend_host);
int moihgp_cuda_objective_finish_dev(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, const double* dx0,
                                     double* loss, double* grad, double* xT, double* dxT);
/* The same exchange WITHOUT host round trips (everything asynchronous on the handle's stream, so that the caller's
 * all-gather - NCCL on the same stream - sits between the two calls):
 *   begin_async : like begin, the end state goes to DEVICE memory zend_dev[N][L][4][d] (NULL on the last block)
 *   carry_in_dev: ends_dev[G][N][L][4][d] = every block's end state (all-gathered); block `rank`'s true carry-in
 *                 z_in(g+1) = T(n_g) z_in(g) + ends_g, chained over g < rank from (x0, dx0) (device, NULL = zeros), is
 *                 written to xin_dev[N][L][d], dxin_dev[N][L][3][d] - pass them to finish_dev.  block_lengths: G host values. */
int moihgp_cuda_objective_begin_async(moihgp_handle* h, const double* Y, size_t N, size_t T, double* zend_dev);
int moihgp_cuda_carry_in_dev(moihgp_handle* h, const double* ends_dev, size_t G, const long long* block_lengths, size_t rank, size_t N,
                             const double* x0_dev, const double* dx0_dev, double* xin_dev, double* dxin_dev);
/* The block transition T(n) of the carry exchange above, per latent: out[L][4][d*d] = [AKHA^n, E_0(n), E_1(n), E_2(n)]
 * (row-major d x d), E_k(n) = sum_i AKHA^(n-1-i) dAKHA_k AKHA^i, so that for a block of n steps
 *   x_out = AKHA^n x_in + x_out(0),   dx_k,out = AKHA^n dx_k,in + E_k(n) x_in + dx_k,out(0)      (ihgp.h:71-77 unrolled).
 * Host arithmetic on the handle's copy of the per-latent constants; no device work. */
int moihgp_cuda_block_transition(moihgp_handle* h, size_t n, double* out);

/* The fused filter + smoother + NLL pass on one contiguous BLOCK of a longer sequence sharded in time (SURVEY 8e: forward
 * carry exchange, then the mirror-image backward exchange for IHGP::backwardSmoother, ihgp.h:108-113).  DEVICE buffers,
 * chunked-scan path; seq_end = 1 on the block that ends the sequence, otherwise T % 256 == 0.  Three phases per block:
 *   1  project the block, chunk summaries, forward chain from x0 (normally NULL = zeros).
 *      host_out[N][L][d + 1] = [state after the block's last step | the block's first projected observation]
 *      -> caller: x_in(g+1) = AKHA^n_g x_in(g) + x_end_g (moihgp_cuda_block_transition), u_after(g) = first observation of g+1
 *   2  x0 = true carry-in, u_after [N][L]: forward chain, backward chain from a zero b_end.
 *      host_out[N][L][d] = backward value at the block's first step
 *      -> caller, from the last block down: b_end(g) = b_start(g+1), b_start(g) = host_out_g + G^n_g b_end(g)
 *         (moihgp_cuda_smoother_power)
 *   3  b_end [N][L][d] (NULL on the last block): backward chain + the final pass: X, Xs [N][T][L][d], nll[N] (the block's
 *      share: sum the blocks), xT (meaningful on the last block).  x0 / u_after as in phase 2.
 * With the literal smoother (mode 0) b is Xs itself, with mode 1 it is Xs - X. */
int moihgp_cuda_fsn_block_dev(moihgp_handle* h, int phase, const double* Y, size_t N, size_t T, int seq_end, int smoother_mode,
                              const double* x0, const double* u_after, const double* b_end, double* X, double* Xs, double* nll,
                              double* xT, double* host_out);
/* The same three phases WITHOUT host round trips (asynchronous on the handle's stream; the caller's all-gathers - NCCL on
 * the same stream - sit between the calls):
 *   fsn_block_async: like fsn_block_dev, the phase's output goes to DEVICE memory dev_out ([N][L][d + 1] after phase 1,
 *                    [N][L][d] after phase 2)
 *   fsn_carry_dev  : direction 0 (after phase 1): gathered_dev[G][N][L][d + 1] -> out_dev[N][L][d] = this block's true x_in
 *                    (chained over the blocks before `rank` from x0_dev, NULL = zeros) and u_after_dev[N][L] = the next
 *                    block's first projected observation (untouched on the last block);
 *                    direction 1 (after phase 2): gathered_dev[G][N][L][d] -> out_dev[N][L][d] = this block's b_end
 *                    (untouched on the last block).  The arithmetic of moihgp_cuda_block_transition /
 *                    moihgp_cuda_smoother_power in a one-thread-per-(sequence, latent) kernel.  block_lengths: G host values. */
int moihgp_cuda_fsn_block_async(moihgp_handle* h, int phase, const double* Y, size_t N, size_t T, int seq_end, int smoother_mode,
                                const double* x0, const double* u_after, const double* b_end, double* X, double* Xs, double* nll,
                                double* xT, double* dev_out);
int moihgp_cuda_fsn_carry_dev(moihgp_handle* h, int direction, int smoother_mode, const double* gathered_dev, size_t G,
                              const long long* block_lengths, size_t rank, size_t N, const double* x0_dev, double* out_dev,
                              double* u_after_dev);
/* G[mode]^n per latent: out[L][d*d] row-major (host arithmetic on the handle's power tables) */
int moihgp_cuda_smoother_power(moihgp_handle* h, int smoother_mode, size_t n, double* out);

#ifdef __cplusplus
}
#endif
#endif /* MOIHGP_B200_H */
