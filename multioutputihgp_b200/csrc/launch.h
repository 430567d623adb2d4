// Host-side launchers of the MOIHGP kernels (internal to libmoihgp.so; the public boundary is
// include/moihgp_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <mutex>
#include <string>
#include <utility>
#include <vector>
#include "moihgp_device.cuh"

namespace moihgp {

// Optional per-kernel timing: one CUDA event recorded on the launching stream after every kernel
// (bench.py's roofline figures come from these, measured live, never under a profiler).
struct Marker {
    cudaStream_t st = nullptr;
    std::vector<std::pair<std::string, cudaEvent_t>> ev;
    void mark(const char* name) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        ev.emplace_back(name, e);
    }
};
inline void mark(Marker* m, const char* name) { if (m) m->mark(name); }

// Chunks per CTA / warp of a chunked pass over `units` independent units: about `target` CTAs / warps, enough to fill
// the machine several times over, with as few chunk prologues as that allows.
inline long long chunks_per_group(long long units, long long chunks, long long target) {
    long long groups = (target + units - 1) / units;
    if (groups < 1) groups = 1;
    if (groups > chunks) groups = chunks;
    return (chunks + groups - 1) / groups;
}

// setup.cu
cudaError_t launch_setup(int dim, const double* d_igp_params, double dt, int L, LatentConsts* d_out, cudaStream_t stream);

// polar.cu  (MOIHGP::update's polar factor on the device, for large p * L)
size_t polar_smem_bytes(int p, int L);
cudaError_t launch_polar(const double* A /*[p][L]*/, int p, int L, double* U, int* status /*device int*/, cudaStream_t st);
// L > 64: the Newton-Schulz iteration over many CTAs (tensor pipe); work: polar_wide_doubles(p, L) doubles.  Waits for the
// stream; *converged = false (U untouched) asks the caller for the host Jacobi
size_t polar_wide_doubles(int p, int L);
cudaError_t launch_polar_wide(const double* A /*[p][L]*/, int p, int L, double* U, double* work, int* status /*device int*/, bool* converged,
                              int* launched, cudaStream_t st);

// Largest number of latent processes a model may have (moihgp_cuda_create)
constexpr int MAX_LATENT = 256;

// project.cu
size_t project_tiles(long long T);     // tiles of 128 time steps per sequence: rho_part is [N][project_tiles(T)]
// doubles of global scratch k_nan_fix needs at this L: one slice of the missing-output solve per CTA of its grid (0: the
// solve runs in shared memory)
size_t ls_global_doubles(int L);
cudaError_t launch_project(const double* Y, const double* U, const double* S, int p, int L, long long N, long long T,
                           double* u, double* w, double* yl, double* rho_part, double* rho_row /*[N][T] or null*/, int* nan_info /*{flag, count}*/, long long* nan_rows,
                           long long nan_cap, double* ls_scratch /*[ls_global_doubles(L)] or null when that is 0*/, cudaStream_t stream);
cudaError_t launch_backproject(const double* X, const double* U, const double* S, int p, int L, int d, long long N,
                               long long T, double* Yhat, cudaStream_t stream);

// Function attributes (dynamic shared memory size) belong to the device's context: they are set once per device, not once
// per process.  `if (AttrOnce once(flags); once) { cudaFuncSetAttribute(...); }` runs the body on the first use on the
// current device; concurrent host threads are serialised and nobody sees the flag before the attributes are set.
struct AttrOnce {
    std::atomic<int>* flag = nullptr;
    bool first = true;
    explicit AttrOnce(std::atomic<int> (&flags)[64]) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev >= 0 && dev < 64) {
            flag = &flags[dev];
            first = flag->load(std::memory_order_acquire) == 0;
        }
        if (first) mutex().lock();
    }
    ~AttrOnce() {
        if (first) {
            if (flag) flag->store(1, std::memory_order_release);
            mutex().unlock();
        }
    }
    explicit operator bool() const { return first; }
    static std::mutex& mutex() { static std::mutex m; return m; }
};

// scan.cu
struct ScanArgs {
    const double* u;              // [N][L][T] projected observations
    const LatentConsts* consts;   // [L]
    int L;
    long long N, T;
    const double* x0;             // [N][L][D] carried-in filter state or null (zeros)
    double *fsum, *bsum, *xin, *bin;   // [N][L][nC][D] chunk summaries / carries (workspace)
    double* Bx;                   // [L][2][D*D] chunk responses (workspace)
    double* Wsum;                 // [L][scan_weights_doubles / L] weights of the interior-chunk summaries (workspace)
    double *sb_end, *sb_in;       // [N][L][scan_superblocks(T)][D] carries of the super-blocks (workspace)
    double *X, *Xs;               // [N][T][L][D] outputs (either may be null)
    double* vsq;                  // [nC][N][L] sum of squared innovations (workspace)
    double* xT;                   // [N][L][D] final filtered state or null
    // ---- one long sequence sharded in TIME over several devices (this call = one contiguous block of it) ----
    int seq_end = 1;              // 1: the block ends the sequence; 0: more steps follow (then T % 256 == 0)
    const double* u_after = nullptr;   // [N][L] projected observation of the first step AFTER the block (seq_end == 0)
    const double* b_end = nullptr;     // [N][L][D] backward value at the first step after the block (null = zeros)
    double* b_out = nullptr;      // [N][L][D] backward value at the block's FIRST step (the previous block's b_end)
    double* x_end = nullptr;      // phase 1: [N][L][D] filtered state after the block's last step, from x0
    int phase = 0;                // 0: whole pass; 1: summaries + forward chain -> x_end; 2: forward chain from the true
                                  // x0, backward chain from b_end = 0 -> b_out; 3: backward chain from b_end + final pass
    double* nll_steps = nullptr;  // [N][T] per-step NLL terms or null (phase 0; scan_pass in capi.cu)
    double* vstep = nullptr;      // [N][L][T] squared innovations of the final pass (workspace of nll_steps) or null
    Marker* mk = nullptr;
};
size_t scan_chunks(long long T);
size_t scan_weights_doubles(int L);
size_t scan_superblocks(long long T);
int scan_launch_count(long long T);
cudaError_t launch_scan(int dim, int mode, const ScanArgs& a, cudaStream_t st);
size_t nll_partials(long long N);
// per-step NLL terms: nll_steps holds the per-row residual norms on entry (launch_project's rho_row) and the terms on return
cudaError_t launch_nll_steps(const double* vstep, const LatentConsts* consts, const double* S, double sigma, int p, int L, long long N,
                             long long T, double* nll_steps, cudaStream_t st);
cudaError_t launch_nll_reduce(const double* rho_part, const double* vsq, const LatentConsts* consts, const double* S, double sigma,
                              int p, int L, long long N, long long T, double* part, double* nll, cudaStream_t st);

// chain.cu  (many-chains path: thread per (sequence, latent), sequential in time)
struct ChainArgs {
    const double* Y;              // [N][T][p], 16-byte aligned
    int p = 0, L = 0;             // outputs / latents of the model (0 = the instantiated P / L); smaller ones run the padded variants
    const double *U_host, *S_host;    // host copies (become constant-bank kernel parameters)
    const LatentConsts* consts;   // device
    double sigma, nll_const;      // nll_const = 1/2 log sum S + 1/2 m_n log sigma (per step; the kernel adds 1/2 sum_l log S_l from the device records)
    long long N, T;
    int mode;                     // smoother mode 0 / 1 (used when Xs != null)
    const double* x0;
    double *X, *Xs, *nll, *xT;    // X must be non-null when Xs is requested
    int* nan_flag;                // set to 1 if a NaN observation was seen
    int seqs_per_warp = 0;        // 0 = automatic
    double* nll_steps = nullptr;  // [N][T] per-step NLL terms (filter-only pass: X and Xs null) or null
    Marker* mk = nullptr;
};
bool chain_supported(int p, int L, int dim, long long T);     // a many-chains instantiation serves the shape (exactly, or padded to the next widths)
bool chain_preferred(int p, int L, int dim, long long T);     // ... and it is the faster path for many sequences (automatic choice)
cudaError_t launch_chain(int p, int L, int dim, const ChainArgs& a, cudaStream_t st);

// objective.cu
struct ObjArgs {
    const double* Y;              // [N][T][p]
    const double *u, *w, *yl, *rho;   // [N][L][T] x3, rho_part [N][project_tiles(T)]   (from k_project)
    double* wgt;                  // [N][L][T] workspace: per-step weights of the dU contraction
    const LatentConsts* consts;
    const double *U, *S;
    double sigma;
    int p, L, threading;
    long long N, T;
    const double *x0, *dx0;       // [N][L][D], [N][L][3][D] carried-in state or null
    double *zsum, *zin;           // [nC][N][L][4*D] chunk summaries / carries
    double* zsub = nullptr;       // [N][nC][8][L][4*D] summaries of the 32-step sub-chunks (k_obj_lanes; workspace, may be null)
    double* part;                 // [nC][N][L][8] per-chunk partial sums
    double* gU_part;              // [nSplit][p][L] split-K partials of dU
    double* Ek;                   // [L][3][D*D] cross-chunk coupling matrices (workspace)
    double* lat_sums;             // [L+1][16][8] per-latent partial sums (workspace)
    double *loss, *grad;          // [1], [num_param] outputs (device)
    double *xT, *dxT;             // final state or null
    int phase = 0;                // 0: whole evaluation, 1: begin (summaries + block end from zero carry), 2: finish
    double* zend = nullptr;       // phase 1: [N][L][4][D] end state of the block from a zero carry-in (device)
    Marker* mk = nullptr;
};
size_t obj_chunks(long long T);
size_t obj_gu_splits(long long N, long long T);
int obj_launch_count(long long T, int L);
cudaError_t launch_objective(int dim, const ObjArgs& a, cudaStream_t st);
// carry-in of time block `rank` from the gathered block ends (device arithmetic of moihgp_cuda_block_transition)
cudaError_t launch_block_carry(int dim, const LatentConsts* consts, int L, long long N, int rank, const long long* block_lengths,
                               const double* ends /*[G][N][L][4][D]*/, const double* x0, const double* dx0, double* xin, double* dxin,
                               cudaStream_t st);
// the two carry exchanges of the time-sharded filter + smoother pass on the device (scan.cu)
cudaError_t launch_fsn_carry(int dim, int direction, int mode, const LatentConsts* consts, int L, long long N, int rank, int G,
                             const long long* block_lengths, const double* gathered, const double* x0, double* out, double* u_after,
                             cudaStream_t st);
size_t obj_small_smem(int p, int L, long long T);
cudaError_t launch_objective_small(int dim, const double* Y, const double* U, const double* S, double sigma, const LatentConsts* consts,
                                   int p, int L, long long T, int threading, const double* x0, const double* dx0, double* out, double* xT,
                                   double* dxT, cudaStream_t st, const double* centre = nullptr, const double* sigma_dev = nullptr);
// streaming learner, device-resident (moihgp_online.h:75-93 window maintenance; :45-54 proximal term)
cudaError_t launch_online_push(const double* y_new, const double* ma_given /*or null*/, int p, int W, double* win /*[W+1][p]*/, int* count,
                               double* ma, double* front_centred, cudaStream_t st);
cudaError_t launch_online_prox(const double* params, const double* oldparams, const double* B /*[np][np] or null*/, int np, int pL,
                               const double* U, double* out /*[loss, flag, grad[np], U[pL]]*/, cudaStream_t st);

// sample.cu  (posterior sample paths: the RTS mean plus the data-independent backward noise process)
struct SampleArgs {
    const LatentConsts* consts;   // [L]
    long long S, N, T, L;
    unsigned long long seed;
    const double* Xs;             // [N][T][L][D] RTS-smoothed mean
    double* Xsamp;                // [S][N][T][L][D] or null
    double* F;                    // [S][N][T][L] function values x~(0) or null (not both null)
    double* carry;                // time-chunked variant: [chunks][S N L][D] workspace (sample_carry_doubles)
    Marker* mk = nullptr;
};
bool sample_chunked(long long T, long long chains, int path);   // path: 0 automatic, 1 time-chunked, 2 one pass
long long sample_chunk_len(long long T, long long chains);
size_t sample_carry_doubles(int dim, long long T, long long chains);
int sample_launch_count(bool chunked);
cudaError_t launch_sample(int dim, const SampleArgs& a, bool chunked, cudaStream_t st);
// one block of a sequence sharded in time: phase 1 leaves e at the block's first step from a zero e_end in e_start
// [S N L][D]; phase 2 writes the paths from e_end (null on the block that ends the sequence).  t0: the block's first step
int sample_block_launch_count(int phase, bool chunked);
cudaError_t launch_sample_block(int dim, int phase, const SampleArgs& a, bool chunked, unsigned long long t0, int seq_end, const double* e_end,
                                double* e_start, cudaStream_t st);

// step.cu  (one observation per call: the legacy gpXX_* entry points)
struct StepArgs {
    const LatentConsts* consts;
    const double *U, *S;
    double sigma;
    int p, L, dim, threading;
    const double *x, *y, *dx;     // device staging: [L][D], [p] (null = predict only), [L][3][D] (may be null)
    double *xnew, *yhat, *dxnew;  // outputs (yhat/dxnew may be null)
    double* ls_scratch = nullptr; // [step_global_doubles(L)] global scratch of the missing-output solve where that is > 0, else null
};
// doubles of global scratch k_step / k_lik need at this L (0: the missing-output solve runs in shared memory)
size_t step_global_doubles(int L);
size_t lik_global_doubles(int L);
cudaError_t launch_step(const StepArgs& a, cudaStream_t st);
struct LikArgs {
    const LatentConsts* consts;
    const double *U, *S;
    double sigma;
    int p, L, dim, threading;
    const double *x, *y, *dx;     // dx null => lik2 (no gradient)
    double* loss;                 // [1]
    double* grad;                 // [num_param] or null
    double* ls_scratch = nullptr; // [lik_global_doubles(L)] where that is > 0, else null
};
cudaError_t launch_lik(const LikArgs& a, cudaStream_t st);
cudaError_t launch_extract_values(const double* X, double* F, long long n, int d, cudaStream_t st);
// IHGP::backwardSmoother over caller-supplied filtered states (generic: one thread per chain)
cudaError_t launch_smooth_seq(const double* X, const LatentConsts* consts, int L, int d, long long N, long long T, int mode, double* Xs,
                              cudaStream_t st);

}  // namespace moihgp
