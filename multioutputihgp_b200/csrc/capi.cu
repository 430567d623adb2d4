// C ABI of libmoihgp.so (declared in include/moihgp_b200.h): the model handle, its device
// workspace, and the host-side glue between the reference-facing entry points and the kernels.
//
// Host-side pieces of the reference that live here:
//   MOIHGP::MOIHGP      moihgp.h:81-136   construction (random near-identity U for the legacy symbols)
//   MOIHGP::update      moihgp.h:431-457  polar factor of the U block (host one-sided Jacobi; the
//                                         per-latent steady-state solve is the K-setup kernel)
//   MOIHGP::getParams   moihgp.h:721-738
//   src/wrapper.cpp:31-624                the 26 legacy symbols (argument marshalling only)
// Everything numerical on the hot path runs on the device; there is no CPU fallback.
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <random>
#include <string>
#include <vector>
#include "../../include/moihgp_b200.h"
#include "launch.h"
#include "small_mat.cuh"

using namespace moihgp;

extern "C" void moihgp_cuda_destroy(moihgp_handle* h);

namespace {

struct Buf {
    void* p = nullptr;
    size_t cap = 0;
};

}  // namespace

struct moihgp_handle {
    int kernel = 32, dim = 2, p = 0, L = 0, threading = 0, device = 0, num_param = 0;
    double dt = 0.0, sigma = 1e-2;
    std::vector<double> U, S, igp;            // host copies: [p*L], [L], [L*3]
    std::vector<LatentConsts> consts;         // host copy of the per-latent constants (refreshed on demand: mirror())
    bool consts_fresh = false;
    double* h_small = nullptr;                // pinned staging of the one-launch objective (k_obj_small)
    size_t h_small_cap = 0;
    double *d_U = nullptr, *d_S = nullptr, *d_igp = nullptr;
    LatentConsts* d_consts = nullptr;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t s_in = nullptr, s_out = nullptr;   // copy streams of the pipelined host-buffer pass (created on first use)
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_c[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    int* h_flags = nullptr;                   // pinned per-slice status words
    double* d_bound = nullptr;                // data set bound by moihgp_cuda_bind_data (resident in HBM across evaluations)
    size_t bound_N = 0, bound_T = 0;
    size_t h_flags_cap = 0;
    std::map<std::string, Buf> ws;            // grow-only device workspace
    double* h_stage = nullptr;                // pinned host staging for the per-observation calls
    double* d_stage = nullptr;
    size_t stage_cap = 0;
    long long launches = 0;
    Marker marker;                            // per-kernel events, only while profiling is on
    bool profiling = false;
    int path = 0;                             // 0 auto, 1 chunked scan, 2 many-chains
    int chain_spw = 0;                        // many-chains kernels: sequences per warp (0 = automatic)
    std::string prof_text;
    std::string err;
    // ---- device-resident streaming learner (moihgp_online.h:18-115): window, moving mean, carried state, proximal term ----
    struct Online {
        size_t W = 0, count = 0;
        double *d_win = nullptr, *d_ma = nullptr, *d_ynew = nullptr, *d_magiven = nullptr, *d_front = nullptr;
        double *d_x = nullptr, *d_dx = nullptr, *d_x2 = nullptr, *d_dx2 = nullptr;     // carried state (and the step's output)
        double *d_params = nullptr, *d_old = nullptr, *d_B = nullptr, *d_out = nullptr;
        double *h_params = nullptr, *h_out = nullptr, *h_y = nullptr;                  // pinned
        int *d_count = nullptr, *d_pst = nullptr;
        bool has_B = false, has_prox = true;
        std::map<long long, int> seen;                    // evaluations per (window length, proximal kind)
        std::map<long long, cudaGraphExec_t> graphs;
    } on;
};

namespace {

// Every entry point runs on the handle's device and leaves the CALLER'S current device as it found it (a single process
// may hold handles on several GPUs next to its own allocations).
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev); else prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                           \
            return -1;                                                                             \
        }                                                                                          \
    } while (0)

int fail(moihgp_handle* h, const std::string& m) {
    h->err = m;
    return -2;
}

template <typename T>
int ws_get(moihgp_handle* h, const char* name, size_t count, T** out) {
    Buf& b = h->ws[name];
    const size_t bytes = std::max<size_t>(count * sizeof(T), 16);
    if (b.cap < bytes) {
        if (b.p) cudaFree(b.p);
        b.p = nullptr;
        b.cap = 0;
        CK(cudaMalloc(&b.p, bytes));
        b.cap = bytes;
    }
    *out = static_cast<T*>(b.p);
    return 0;
}

// Workspace of the projection (k_project), shared by the scan and the objective passes: one handle alternating between
// them reuses the same buffers.  Rows with a missing output are listed for re-projection, at most nan_cap of them.
struct ProjectWs {
    double *u, *rho;
    int* nanf;                    // {status, count} (moihgp_cuda_nan_status)
    long long* nanrows;
    size_t nan_cap;
    double* lsg;                  // global scratch of the missing-output solve (null where it runs in shared memory)
};

int project_ws(moihgp_handle* h, size_t N, size_t T, ProjectWs* w) {
    w->nan_cap = std::min<size_t>(N * T, (size_t)1 << 22);
    if (ws_get(h, "nanrows", w->nan_cap, &w->nanrows) || ws_get(h, "u", N * h->L * T, &w->u) ||
        ws_get(h, "rho", N * project_tiles((long long)T), &w->rho) || ws_get(h, "nanf", 4, &w->nanf))
        return -1;
    w->lsg = nullptr;
    if (ls_global_doubles(h->L) && ws_get(h, "lsg", ls_global_doubles(h->L), &w->lsg)) return -1;
    return 0;
}

// A pass that meets more than 2^22 rows with missing outputs re-projects only the first 2^22 of them, so the host-buffer
// entry points refuse such a call.  status: the status words of the call's passes, already on the host; null reads the
// handle's own (that of the last pass), waiting for the stream.
int refuse_nan_overflow(moihgp_handle* h, const int* status = nullptr, size_t n = 1) {
    int last = 0;
    if (!status) {
        if (moihgp_cuda_nan_status(h, &last)) return -1;
        status = &last;
    }
    for (size_t i = 0; i < n; ++i)
        if (status[i] == 2) return fail(h, "more than 2^22 observations with missing (NaN) outputs in one call: split the batch");
    return 0;
}

// Which kernels serve one fused pass over Y [N][T][p] into X / Xs (moihgp_cuda_set_path): 1 the many-chains kernels,
// 0 the chunked scan.  The many-chains kernels need an instantiated shape and 16-byte aligned Y, X and Xs; the automatic
// choice takes them where they are the faster path and the chains give every SM a warp.  A forced many-chains path that
// cannot serve the pass fails (-2) when `strict`, else it takes the scan - as the automatic choice would, since
// chain_preferred implies chain_supported.
int chain_path(moihgp_handle* h, size_t N, size_t T, const void* Y, const void* X, const void* Xs, bool strict) {
    auto aligned16 = [](const void* q) { return (reinterpret_cast<size_t>(q) & 15) == 0; };
    const bool aligned = aligned16(Y) && aligned16(X) && aligned16(Xs);
    if (h->path == 1) return 0;
    if (h->path == 2) {
        if (aligned && chain_supported(h->p, h->L, h->dim, (long long)T)) return 1;
        return strict ? fail(h, "many-chains path not available for this shape/alignment") : 0;
    }
    const size_t chain_warps = (N * (size_t)h->L + 31) / 32;
    return aligned && chain_preferred(h->p, h->L, h->dim, (long long)T) && chain_warps >= 148;
}

// Polar factor U = W V' of a (p x L, row-major, p >= L) via one-sided Jacobi: a V = W diag(s).
// (MOIHGP::update forms svd.matrixU() * svd.matrixV().transpose(), moihgp.h:439,446.)
void polar_factor(const double* a, int p, int L, double* out) {
    // columns stored contiguously (Wt[j][r], Vt[j][r]): the pair sweeps are unit-stride and vectorise
    std::vector<double> Wt((size_t)L * p), Vt((size_t)L * L, 0.0);
    for (int r = 0; r < p; ++r) for (int c = 0; c < L; ++c) Wt[(size_t)c * p + r] = a[(size_t)r * L + c];
    for (int i = 0; i < L; ++i) Vt[(size_t)i * L + i] = 1.0;
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0.0;
        for (int i = 0; i < L - 1; ++i)
            for (int j = i + 1; j < L; ++j) {
                double* wi = &Wt[(size_t)i * p];
                double* wj = &Wt[(size_t)j * p];
                double al = 0.0, be = 0.0, ga = 0.0;
                for (int r = 0; r < p; ++r) { al += wi[r] * wi[r]; be += wj[r] * wj[r]; ga += wi[r] * wj[r]; }
                if (ga == 0.0) continue;
                off = std::max(off, std::fabs(ga) / std::sqrt(al * be));
                const double zeta = (be - al) / (2.0 * ga);
                const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (std::fabs(zeta) + std::sqrt(1.0 + zeta * zeta));
                const double c = 1.0 / std::sqrt(1.0 + t * t), s = c * t;
                for (int r = 0; r < p; ++r) { const double x = wi[r], y = wj[r]; wi[r] = c * x - s * y; wj[r] = s * x + c * y; }
                double* vi = &Vt[(size_t)i * L];
                double* vj = &Vt[(size_t)j * L];
                for (int r = 0; r < L; ++r) { const double x = vi[r], y = vj[r]; vi[r] = c * x - s * y; vj[r] = s * x + c * y; }
            }
        if (off < 1e-15) break;
    }
    for (int j = 0; j < L; ++j) {
        double* wj = &Wt[(size_t)j * p];
        double q = 0.0;
        for (int r = 0; r < p; ++r) q += wj[r] * wj[r];
        const double s = std::sqrt(q);
        for (int r = 0; r < p; ++r) wj[r] = s > 0.0 ? wj[r] / s : 0.0;
    }
    for (int r = 0; r < p; ++r)
        for (int c = 0; c < L; ++c) {
            double s = 0.0;
            for (int k = 0; k < L; ++k) s += Wt[(size_t)k * p + r] * Vt[(size_t)k * L + c];
            out[(size_t)r * L + c] = s;
        }
}

// device_polar: d_U already holds the polar factor (k_polar); bring it to the host copy instead of uploading it
int push_model(moihgp_handle* h, bool device_polar = false) {
    if (device_polar) CK(cudaMemcpyAsync(h->U.data(), h->d_U, sizeof(double) * h->U.size(), cudaMemcpyDeviceToHost, h->stream));
    else CK(cudaMemcpyAsync(h->d_U, h->U.data(), sizeof(double) * h->U.size(), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_S, h->S.data(), sizeof(double) * h->S.size(), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_igp, h->igp.data(), sizeof(double) * h->igp.size(), cudaMemcpyHostToDevice, h->stream));
    CK(launch_setup(h->dim, h->d_igp, h->dt, h->L, h->d_consts, h->stream));
    h->launches += 1;
    h->consts_fresh = false;          // no host round trip here: update() returns while k_setup runs (mirror() fetches on demand)
    return 0;
}

// host copy of the per-latent constants, fetched when somebody on the host needs them
int mirror(moihgp_handle* h) {
    if (h->consts_fresh) return 0;
    CK(cudaMemcpyAsync(h->consts.data(), h->d_consts, sizeof(LatentConsts) * h->L, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->consts_fresh = true;
    return 0;
}

int create(moihgp_handle** out, int kernel, double dt, size_t p, size_t L, int threading, int device, bool random_U) {
    if (!out) return -2;
    *out = nullptr;
    moihgp_handle* h = new moihgp_handle();
    auto bail = [&](const std::string& m) {
        std::fprintf(stderr, "libmoihgp (B200): %s\n", m.c_str());
        moihgp_cuda_destroy(h);                  // frees whatever was allocated so far (stream, device / pinned buffers)
        return -1;
    };
    h->device = -1;                              // until a valid device is known (destroy() then frees nothing on a device)
    if (kernel != 32 && kernel != 52) return bail("kernel must be 32 (Matern-3/2) or 52 (Matern-5/2)");
    if (p == 0 || L == 0 || L > p) return bail("need 1 <= num_latent <= num_output");
    if (L > (size_t)MAX_LATENT) return bail("num_latent > 256 is not supported (need 1 <= num_latent <= min(num_output, 256))");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return bail("no CUDA device: this library has no CPU fallback");
    if (device < 0) cudaGetDevice(&device);
    if (device >= ndev) return bail("bad device index");
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    if (prop.major != 10) return bail(std::string("device '") + prop.name + "' is not compute capability 10.x (built for sm_100a only)");
    DeviceGuard guard(device);
    h->kernel = kernel; h->dim = kernel == 32 ? 2 : 3; h->p = (int)p; h->L = (int)L; h->dt = dt; h->device = device;
    h->threading = L < 2 ? 0 : (threading ? 1 : 0);                       // moihgp.h:128-135
    h->num_param = (int)(p * L + L + 1 + 3 * L);                          // moihgp.h:93
    h->U.assign(p * L, 0.0);
    if (random_U) {                                                       // moihgp.h:103-125
        std::random_device rd;
        std::mt19937 gen(rd());
        std::normal_distribution<> distr(0.0, 1e-3);
        std::vector<double> raw(p * L, 0.0);
        for (size_t r = 0; r < p; ++r) for (size_t c = 0; c < L; ++c) raw[r * L + c] = (r == c ? 1.0 : 0.0) + distr(gen);
        polar_factor(raw.data(), (int)p, (int)L, h->U.data());
    } else {
        for (size_t i = 0; i < L; ++i) h->U[i * L + i] = 1.0;
    }
    h->S.assign(L, 1.0);                                                  // moihgp.h:126
    h->sigma = 1e-2;                                                      // moihgp.h:127
    h->igp.resize(3 * L);
    for (size_t l = 0; l < L; ++l) { h->igp[3 * l] = 1.0; h->igp[3 * l + 1] = 1.0; h->igp[3 * l + 2] = 0.1; }   // matern32ss.h:35
    h->consts.resize(L);
    if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess) return bail("cudaStreamCreate failed");
    h->stream = h->own_stream;
    bool ok = cudaMalloc(&h->d_U, sizeof(double) * p * L) == cudaSuccess && cudaMalloc(&h->d_S, sizeof(double) * L) == cudaSuccess &&
              cudaMalloc(&h->d_igp, sizeof(double) * 3 * L) == cudaSuccess && cudaMalloc(&h->d_consts, sizeof(LatentConsts) * L) == cudaSuccess;
    if (!ok) return bail("cudaMalloc failed");
    h->stage_cap = (size_t)(2 * (L * 3 + L * 9) + 2 * p + 2 * h->num_param + 16);
    if (cudaMallocHost(&h->h_stage, sizeof(double) * h->stage_cap) != cudaSuccess || cudaMalloc(&h->d_stage, sizeof(double) * h->stage_cap) != cudaSuccess)
        return bail("staging allocation failed");
    if (push_model(h) != 0) return bail(h->err);
    *out = h;
    return 0;
}

// ---- one observation: marshalling for the legacy symbols -------------------------------------------
struct StageLayout {
    size_t x, dx, y, xnew, dxnew, yhat, loss, grad, total_in;
};
StageLayout stage_layout(const moihgp_handle* h) {
    StageLayout s;
    const size_t Ld = (size_t)h->L * h->dim;
    s.x = 0; s.dx = s.x + Ld; s.y = s.dx + 3 * Ld; s.total_in = s.y + h->p;
    s.xnew = s.total_in; s.dxnew = s.xnew + Ld; s.yhat = s.dxnew + 3 * Ld; s.loss = s.yhat + h->p; s.grad = s.loss + 2;
    return s;
}

int step_call(moihgp_handle* h, const double* x, const double* y, const double* dx, double* xnew, double* yhat, double* dxnew) {
    DeviceGuard guard(h->device);
    const StageLayout s = stage_layout(h);
    const size_t Ld = (size_t)h->L * h->dim;
    std::memcpy(h->h_stage + s.x, x, sizeof(double) * Ld);
    if (dx) std::memcpy(h->h_stage + s.dx, dx, sizeof(double) * 3 * Ld);
    if (y) std::memcpy(h->h_stage + s.y, y, sizeof(double) * h->p);
    CK(cudaMemcpyAsync(h->d_stage, h->h_stage, sizeof(double) * s.total_in, cudaMemcpyHostToDevice, h->stream));
    StepArgs a;
    a.consts = h->d_consts; a.U = h->d_U; a.S = h->d_S; a.sigma = h->sigma; a.p = h->p; a.L = h->L; a.dim = h->dim; a.threading = h->threading;
    a.x = h->d_stage + s.x; a.y = y ? h->d_stage + s.y : nullptr; a.dx = dx ? h->d_stage + s.dx : nullptr;
    a.xnew = h->d_stage + s.xnew; a.yhat = yhat ? h->d_stage + s.yhat : nullptr; a.dxnew = (dx && dxnew) ? h->d_stage + s.dxnew : nullptr;
    if (step_global_doubles(h->L) && ws_get(h, "lsg1", step_global_doubles(h->L), &a.ls_scratch)) return -1;
    CK(launch_step(a, h->stream));
    h->launches += 1;
    CK(cudaMemcpyAsync(h->h_stage + s.xnew, h->d_stage + s.xnew, sizeof(double) * (s.loss - s.xnew), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    std::memcpy(xnew, h->h_stage + s.xnew, sizeof(double) * Ld);
    if (dx && dxnew) std::memcpy(dxnew, h->h_stage + s.dxnew, sizeof(double) * 3 * Ld);
    if (yhat) std::memcpy(yhat, h->h_stage + s.yhat, sizeof(double) * h->p);
    return 0;
}

int lik_call(moihgp_handle* h, const double* x, const double* y, const double* dx, double* loss, double* grad) {
    DeviceGuard guard(h->device);
    const StageLayout s = stage_layout(h);
    const size_t Ld = (size_t)h->L * h->dim;
    std::memcpy(h->h_stage + s.x, x, sizeof(double) * Ld);
    if (dx) std::memcpy(h->h_stage + s.dx, dx, sizeof(double) * 3 * Ld);
    std::memcpy(h->h_stage + s.y, y, sizeof(double) * h->p);
    CK(cudaMemcpyAsync(h->d_stage, h->h_stage, sizeof(double) * s.total_in, cudaMemcpyHostToDevice, h->stream));
    LikArgs a;
    a.consts = h->d_consts; a.U = h->d_U; a.S = h->d_S; a.sigma = h->sigma; a.p = h->p; a.L = h->L; a.dim = h->dim; a.threading = h->threading;
    a.x = h->d_stage + s.x; a.y = h->d_stage + s.y; a.dx = dx ? h->d_stage + s.dx : nullptr;
    a.loss = h->d_stage + s.loss; a.grad = (dx && grad) ? h->d_stage + s.grad : nullptr;
    if (lik_global_doubles(h->L) && ws_get(h, "lsg1", lik_global_doubles(h->L), &a.ls_scratch)) return -1;
    CK(launch_lik(a, h->stream));
    h->launches += 1;
    const size_t nout = 2 + ((dx && grad) ? (size_t)h->num_param : 0);
    CK(cudaMemcpyAsync(h->h_stage + s.loss, h->d_stage + s.loss, sizeof(double) * nout, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *loss = h->h_stage[s.loss];
    if (dx && grad) std::memcpy(grad, h->h_stage + s.grad, sizeof(double) * h->num_param);
    return 0;
}

void legacy_fatal(moihgp_handle* h, const char* where) {
    // The reference's C ABI has no error channel (all void / value returns).  A CUDA failure here
    // cannot be reported to the caller, so fail loudly rather than return garbage.
    std::fprintf(stderr, "libmoihgp (B200): %s failed: %s\n", where, h ? h->err.c_str() : "null handle");
    std::abort();
}

moihgp_handle* legacy_new(int kernel, double dt, size_t p, size_t L, bool threading) {
    moihgp_handle* h = nullptr;
    if (create(&h, kernel, dt, p, L, threading ? 1 : 0, -1, /*random_U=*/true) != 0) {
        std::fprintf(stderr, "libmoihgp (B200): gpXX_new failed (no CPU fallback)\n");
        std::abort();
    }
    return h;
}

int kernel_for_gp52() {
    // wrapper.cpp:22 typedefs GP52 to the Matern-3/2 class (SURVEY Q7); the drop-in keeps that
    // behaviour unless MOIHGP_GP52_MATERN52=1 asks for the kernel the name promises.
    const char* e = std::getenv("MOIHGP_GP52_MATERN52");
    return (e && e[0] == '1') ? 52 : 32;
}

}  // namespace

// =============================================================================================
extern "C" {

int moihgp_cuda_create(moihgp_handle** out, int kernel, double dt, size_t p, size_t L, int threading, int device) {
    return create(out, kernel, dt, p, L, threading, device, /*random_U=*/false);
}

void moihgp_cuda_destroy(moihgp_handle* h) {
    if (!h) return;
    if (h->device < 0) { delete h; return; }     // creation failed before a device was chosen: nothing lives on a device
    DeviceGuard guard(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (auto& kv : h->ws) if (kv.second.p) cudaFree(kv.second.p);
    cudaFree(h->d_U); cudaFree(h->d_S); cudaFree(h->d_igp); cudaFree(h->d_consts); cudaFree(h->d_stage);
    if (h->h_stage) cudaFreeHost(h->h_stage);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    if (h->s_in) cudaStreamDestroy(h->s_in);
    if (h->s_out) cudaStreamDestroy(h->s_out);
    if (h->h_flags) cudaFreeHost(h->h_flags);
    if (h->h_small) cudaFreeHost(h->h_small);
    if (h->d_bound) cudaFree(h->d_bound);
    for (auto& kv : h->on.graphs) cudaGraphExecDestroy(kv.second);
    {
        moihgp_handle::Online& o = h->on;
        double* dev[] = {o.d_win, o.d_ma, o.d_ynew, o.d_magiven, o.d_front, o.d_x, o.d_dx, o.d_x2, o.d_dx2, o.d_params, o.d_old, o.d_B, o.d_out};
        for (double* q : dev) if (q) cudaFree(q);
        if (o.d_count) cudaFree(o.d_count);
        if (o.d_pst) cudaFree(o.d_pst);
        if (o.h_params) cudaFreeHost(o.h_params);
        if (o.h_out) cudaFreeHost(o.h_out);
        if (o.h_y) cudaFreeHost(o.h_y);
    }
    for (int i = 0; i < 2; ++i) { if (h->ev_in[i]) cudaEventDestroy(h->ev_in[i]); if (h->ev_c[i]) cudaEventDestroy(h->ev_c[i]); if (h->ev_out[i]) cudaEventDestroy(h->ev_out[i]); }
    delete h;
}

int moihgp_cuda_set_stream(moihgp_handle* h, void* s) {
    if (!h) return -2;
    cudaStream_t ns = s ? static_cast<cudaStream_t>(s) : h->own_stream;
    if (ns != h->stream) {
        // moving the handle waits for the old stream - not possible while the new stream is being captured into a CUDA
        // graph (the wait would invalidate the capture): refuse, the caller moves the handle once BEFORE the capture
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(ns, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive)
            return fail(h, "set_stream: the new stream is capturing - move the handle to it (any call on that stream) before the capture begins");
        cudaStreamSynchronize(h->stream);      // work queued on the old stream finishes before the handle moves
        h->stream = ns;
    }
    return 0;
}

int moihgp_cuda_sync(moihgp_handle* h) {
    if (!h) return -2;
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int moihgp_cuda_set_path(moihgp_handle* h, int path) {
    if (!h || path < 0 || path > 2) return -2;
    h->path = path;
    return 0;
}

int moihgp_cuda_set_chain_seqs_per_warp(moihgp_handle* h, int n) {
    if (!h || n < 0 || n > 32) return -2;
    h->chain_spw = n;
    return 0;
}

int moihgp_cuda_profile(moihgp_handle* h, int enable) {
    if (!h) return -2;
    cudaStreamSynchronize(h->stream);
    for (auto& e : h->marker.ev) cudaEventDestroy(e.second);
    h->marker.ev.clear();
    h->profiling = enable != 0;
    return 0;
}

// "name total_ms launches" per line, accumulated since moihgp_cuda_profile(h, 1); resets the record
const char* moihgp_cuda_profile_read(moihgp_handle* h) {
    if (!h) return "";
    cudaStreamSynchronize(h->stream);
    std::vector<std::string> order;
    std::map<std::string, std::pair<double, long long>> acc;
    auto& ev = h->marker.ev;
    for (size_t i = 1; i < ev.size(); ++i) {
        if (ev[i].first == "begin") continue;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev[i - 1].second, ev[i].second);
        if (!acc.count(ev[i].first)) order.push_back(ev[i].first);
        acc[ev[i].first].first += ms;
        acc[ev[i].first].second += 1;
    }
    h->prof_text.clear();
    char line[256];
    for (auto& n : order) {
        std::snprintf(line, sizeof(line), "%s %.6f %lld\n", n.c_str(), acc[n].first, acc[n].second);
        h->prof_text += line;
    }
    for (auto& e : ev) cudaEventDestroy(e.second);
    ev.clear();
    return h->prof_text.c_str();
}

const char* moihgp_cuda_last_error(moihgp_handle* h) { return h ? h->err.c_str() : "null handle"; }
long long moihgp_cuda_launch_count(moihgp_handle* h) { return h ? h->launches : 0; }
size_t moihgp_cuda_igp_dim(moihgp_handle* h) { return h ? (size_t)h->dim : 0; }
size_t moihgp_cuda_num_param(moihgp_handle* h) { return h ? (size_t)h->num_param : 0; }
size_t moihgp_cuda_num_igp_param(moihgp_handle* h) { return h ? 3 : 0; }

// 0: no missing observation seen by the last whole-sequence call on this handle, 1: some (re-projected, moihgp.h:167-178),
// 2: more than 2^22 rows with missing outputs - the rows beyond that were NOT re-projected (their u is NaN).
int moihgp_cuda_nan_status(moihgp_handle* h, int* status) {
    if (!h || !status) return -2;
    DeviceGuard guard(h->device);
    *status = 0;
    auto it = h->ws.find("nanf");
    if (it == h->ws.end() || !it->second.p) return 0;
    int flag[2] = {0, 0};
    CK(cudaMemcpyAsync(flag, it->second.p, sizeof(flag), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *status = flag[0];
    return 0;
}

int moihgp_cuda_update(moihgp_handle* h, const double* params) {
    if (!h || !params) return -2;
    DeviceGuard guard(h->device);
    const int p = h->p, L = h->L;
    // moihgp.h:436-446: polar factor of the U block - on the device when the block is large (k_polar), else host Jacobi.
    // L > 64: the many-CTA Newton-Schulz iteration, and the host Jacobi where it does not converge.
    bool dev_polar = L <= 64 && (size_t)p * L >= 2048 && polar_smem_bytes(p, L) <= 200 * 1024;
    if (L > 64) {
        double *d_raw, *work;
        int* pst;
        if (ws_get(h, "Uraw", (size_t)p * L, &d_raw) || ws_get(h, "polar_wide", polar_wide_doubles(p, L), &work) ||
            ws_get(h, "polar_status", 4, &pst))
            return -1;
        CK(cudaMemcpyAsync(d_raw, params, sizeof(double) * p * L, cudaMemcpyHostToDevice, h->stream));
        int launched = 0;
        CK(launch_polar_wide(d_raw, p, L, h->d_U, work, pst, &dev_polar, &launched, h->stream));
        h->launches += launched;
        if (!dev_polar) polar_factor(params, p, L, h->U.data());
    } else if (dev_polar) {
        double* d_raw;
        if (ws_get(h, "Uraw", (size_t)p * L, &d_raw)) return -1;
        CK(cudaMemcpyAsync(d_raw, params, sizeof(double) * p * L, cudaMemcpyHostToDevice, h->stream));
        int* pst;
        if (ws_get(h, "polar_status", 4, &pst)) return -1;
        CK(launch_polar(d_raw, p, L, h->d_U, pst, h->stream));
        h->launches += 2;
    } else {
        polar_factor(params, p, L, h->U.data());
    }
    for (int l = 0; l < L; ++l) h->S[l] = params[p * L + l];               // moihgp.h:448
    h->sigma = params[p * L + L];                                          // moihgp.h:449
    for (int i = 0; i < 3 * L; ++i) h->igp[i] = params[p * L + L + 1 + i]; // moihgp.h:450-456
    return push_model(h, dev_polar);
}

int moihgp_cuda_get_params(moihgp_handle* h, double* params) {
    if (!h || !params) return -2;
    const int p = h->p, L = h->L;
    std::copy(h->U.begin(), h->U.end(), params);
    std::copy(h->S.begin(), h->S.end(), params + p * L);
    params[p * L + L] = h->sigma;
    std::copy(h->igp.begin(), h->igp.end(), params + p * L + L + 1);
    return 0;
}

int moihgp_cuda_get_U(moihgp_handle* h, double* U) {
    if (!h || !U) return -2;
    std::copy(h->U.begin(), h->U.end(), U);
    return 0;
}

long long moihgp_cuda_latent_consts(moihgp_handle* h, size_t l, double* out, size_t cap) {
    if (!h || !out || l >= (size_t)h->L) return -2;
    if (mirror(h)) return -1;
    const LatentConsts& c = h->consts[l];
    const int d = h->dim;
    std::vector<double> v;
    auto mat = [&](const double* m) { for (int i = 0; i < d; ++i) for (int j = 0; j < d; ++j) v.push_back(m[i * 3 + j]); };
    auto vec = [&](const double* m) { for (int i = 0; i < d; ++i) v.push_back(m[i]); };
    mat(c.A); mat(c.Q); vec(c.K); v.push_back(c.S); mat(c.PF); vec(c.HA); mat(c.AKHA);
    for (int k = 0; k < 3; ++k) { v.push_back(c.dS[k]); mat(c.dA[k]); vec(c.dK[k]); mat(c.dAKHA[k]); vec(c.HdA[k]); }
    if (v.size() > cap) return -3;
    std::copy(v.begin(), v.end(), out);
    return (long long)v.size();
}

int moihgp_cuda_block_transition(moihgp_handle* h, size_t n, double* out) {
    if (!h || !out) return -2;
    if (mirror(h)) return -1;
    for (int l = 0; l < h->L; ++l) {                                      // out[l] = [P | E_0 | E_1 | E_2]
        double* o = out + (size_t)l * 4 * h->dim * h->dim;
        if (h->dim == 2) block_transition<2>(h->consts[l], n, o, reinterpret_cast<double(*)[4]>(o + 4));
        else block_transition<3>(h->consts[l], n, o, reinterpret_cast<double(*)[9]>(o + 9));
    }
    return 0;
}

int moihgp_cuda_latent_iters(moihgp_handle* h, size_t l, int* out8) {
    if (!h || !out8 || l >= (size_t)h->L) return -2;
    if (mirror(h)) return -1;
    for (int i = 0; i < 4; ++i) { out8[i] = h->consts[l].iters[i]; out8[4 + i] = h->consts[l].conv[i]; }
    return 0;
}

int moihgp_cuda_smoother_consts(moihgp_handle* h, size_t l, int mode, double* G, double* P) {
    if (!h || l >= (size_t)h->L || mode < 0 || mode > 1) return -2;
    if (mirror(h)) return -1;
    const int d = h->dim;
    for (int i = 0; i < d; ++i) for (int j = 0; j < d; ++j) {
        if (G) G[i * d + j] = h->consts[l].G[mode][i * 3 + j];
        if (P) P[i * d + j] = h->consts[l].Ps[mode][i * 3 + j];
    }
    return 0;
}

// The chunked-scan pass (project.cu + scan.cu) over Y [N][T][p] with N = a.N, T = a.T: a.phase 0 is the whole pass, 1 / 2 / 3
// one block of a sequence sharded in time (ScanArgs).  The caller sets a's inputs, outputs, phase and marker; this takes the
// workspace, projects Y (phases 0 and 1), scans, and reduces the NLL into nll (phases 0 and 3, when nll is set) and, when
// a.nll_steps is set (phase 0), into per-step terms.  On return a.u holds the projected observations.
static int scan_pass(moihgp_handle* h, const double* Y, int mode, double* nll, ScanArgs& a) {
    const size_t N = (size_t)a.N, T = (size_t)a.T, L = h->L, D = h->dim, nC = scan_chunks(a.T), nSB = scan_superblocks(a.T);
    ProjectWs pw;
    double *fsum, *bsum, *xin, *bin, *Bx, *vsq, *npart, *Wsum, *sbe, *sbi;
    if (project_ws(h, N, T, &pw) || ws_get(h, "npart", nll_partials(a.N), &npart) || ws_get(h, "fsum", nC * N * L * D, &fsum) ||
        ws_get(h, "bsum", nC * N * L * D, &bsum) || ws_get(h, "xin", nC * N * L * D, &xin) || ws_get(h, "bin", nC * N * L * D, &bin) ||
        ws_get(h, "Bx", L * 2 * 9, &Bx) || ws_get(h, "Wsum", scan_weights_doubles((int)L), &Wsum) || ws_get(h, "sbe", N * L * nSB * D, &sbe) ||
        ws_get(h, "sbi", N * L * nSB * D, &sbi) || ws_get(h, "vsq", nC * N * L, &vsq))
        return -1;
    if (a.nll_steps && ws_get(h, "vstep", N * L * T, &a.vstep)) return -1;
    if (a.phase <= 1) {
        // the projection residuals rho feed only the NLL; a block keeps them from phase 1 for its phase 3
        CK(cudaMemsetAsync(pw.nanf, 0, 2 * sizeof(int), h->stream));
        // per-step terms: the projection leaves each row's residual norm in nll_steps, k_nll_steps completes them in place
        CK(launch_project(Y, h->d_U, h->d_S, h->p, (int)L, a.N, a.T, pw.u, nullptr, nullptr, (nll || a.phase == 1 || a.nll_steps) ? pw.rho : nullptr,
                          a.nll_steps, pw.nanf, pw.nanrows, (long long)pw.nan_cap, pw.lsg, h->stream));
        h->launches += 2;
        mark(a.mk, "k_project");
    }
    a.u = pw.u; a.consts = h->d_consts; a.L = (int)L;
    a.fsum = fsum; a.bsum = bsum; a.xin = xin; a.bin = bin; a.Bx = Bx; a.Wsum = Wsum; a.sb_end = sbe; a.sb_in = sbi; a.vsq = vsq;
    CK(launch_scan((int)D, mode, a, h->stream));
    h->launches += scan_launch_count(a.T);
    if ((a.phase == 0 || a.phase == 3) && nll) {
        CK(launch_nll_reduce(pw.rho, vsq, h->d_consts, h->d_S, h->sigma, h->p, (int)L, a.N, a.T, npart, nll, h->stream));
        h->launches += 2;
        mark(a.mk, "k_nll_reduce");
    }
    if (a.phase == 0 && a.nll_steps) {
        CK(launch_nll_steps(a.vstep, h->d_consts, h->d_S, h->sigma, h->p, (int)L, a.N, a.T, a.nll_steps, h->stream));
        h->launches += 1;
        mark(a.mk, "k_nll_steps");
    }
    return 0;
}

// strict_chain: a forced many-chains path that cannot serve the pass fails (the entry point) or takes the scan (the sampler).
// nll_steps ([N][T] per-step NLL terms) is the filter-only pass of moihgp_cuda_nll_steps_dev: mode -1, X, Xs and Yhat null.
static int fused_pass(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, int mode, double* X, double* Xs,
                      double* Yhat, double* nll, double* xT, bool strict_chain, double* nll_steps = nullptr) {
    if (!h || !Y) return -2;
    if (N == 0 || T == 0) return fail(h, "N and T must be positive");
    if (mode < -1 || mode > 1) return fail(h, "smoother_mode must be -1, 0 or 1");
    if (mode < 0 && Xs) return fail(h, "Xs requested with smoother_mode = none");
    DeviceGuard guard(h->device);
    const int L = h->L, D = h->dim;
    double* Xtmp = nullptr;
    if ((Yhat || Xs) && !X) { if (ws_get(h, "Xtmp", N * T * L * D, &Xtmp)) return -1; X = Xtmp; }
    Marker* mk = h->profiling ? &h->marker : nullptr;
    if (mk) { mk->st = h->stream; mk->mark("begin"); }
    const int use_chain = chain_path(h, N, T, Y, X, Xs, strict_chain);
    if (use_chain < 0) return use_chain;
    if (use_chain) {
        // one thread per (sequence, latent) chain, sequential in time: chain.cu
        int* nanf;
        if (ws_get(h, "nanf", 4, &nanf)) return -1;
        CK(cudaMemsetAsync(nanf, 0, 2 * sizeof(int), h->stream));
        ChainArgs c;                               // no mirror(h): nothing here waits for K-setup (asynchronous, capturable)
        c.Y = Y; c.U_host = h->U.data(); c.S_host = h->S.data(); c.consts = h->d_consts; c.sigma = h->sigma;
        c.nll_const = nll_step_const(h->S.data(), h->p, L, h->sigma);
        c.N = (long long)N; c.T = (long long)T; c.mode = mode < 0 ? 1 : mode; c.x0 = x0; c.X = X; c.Xs = Xs; c.nll = nll; c.xT = xT; c.mk = mk; c.nan_flag = nanf; c.seqs_per_warp = h->chain_spw;
        c.nll_steps = nll_steps;
        CK(launch_chain(h->p, L, D, c, h->stream));
        h->launches += Xs ? 2 : 1;
    } else {
        ScanArgs a{};
        a.mk = mk;
        a.N = (long long)N; a.T = (long long)T; a.x0 = x0; a.X = X; a.Xs = Xs; a.xT = xT; a.nll_steps = nll_steps;
        if (const int rc = scan_pass(h, Y, mode < 0 ? 1 : mode, nll, a)) return rc;
    }
    if (Yhat) { CK(launch_backproject(X, h->d_U, h->d_S, h->p, L, D, (long long)N, (long long)T, Yhat, h->stream)); h->launches += 1; mark(mk, "k_backproject"); }
    return 0;
}

int moihgp_cuda_filter_smoother_nll_dev(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, int mode,
                                        double* X, double* Xs, double* Yhat, double* nll, double* xT) {
    return fused_pass(h, Y, N, T, x0, mode, X, Xs, Yhat, nll, xT, /*strict_chain=*/true);
}

int moihgp_cuda_nll_steps_dev(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, double* nll_steps, double* nll,
                              double* xT) {
    if (!h) return -2;
    if (!nll_steps) return fail(h, "nll_steps: the output nll_steps [N][T] is required");
    if (N == 0 || T == 0) return fail(h, "N and T must be positive");
    return fused_pass(h, Y, N, T, x0, MOIHGP_SMOOTH_NONE, nullptr, nullptr, nullptr, nll, xT, /*strict_chain=*/true, nll_steps);
}

// Host buffers: copy in, the device pass, copy out (the input dominates the traffic: no slice pipeline).
int moihgp_cuda_nll_steps(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, double* nll_steps, double* nll,
                          double* xT) {
    if (!h) return -2;
    if (!nll_steps) return fail(h, "nll_steps: the output nll_steps [N][T] is required");
    if (!Y) return -2;
    if (N == 0 || T == 0) return fail(h, "N and T must be positive");
    DeviceGuard guard(h->device);
    const size_t L = h->L, D = h->dim, p = h->p;
    double *dY, *dx0 = nullptr, *dsteps, *dnll = nullptr, *dxT = nullptr;
    if (ws_get(h, "nsY", N * T * p, &dY) || ws_get(h, "nsSteps", N * T, &dsteps)) return -1;
    if (x0 && ws_get(h, "nsx0", N * L * D, &dx0)) return -1;
    if (nll && ws_get(h, "nsNll", N, &dnll)) return -1;
    if (xT && ws_get(h, "nsxT", N * L * D, &dxT)) return -1;
    CK(cudaMemcpyAsync(dY, Y, sizeof(double) * N * T * p, cudaMemcpyHostToDevice, h->stream));
    if (x0) CK(cudaMemcpyAsync(dx0, x0, sizeof(double) * N * L * D, cudaMemcpyHostToDevice, h->stream));
    const int rc = moihgp_cuda_nll_steps_dev(h, dY, N, T, dx0, dsteps, dnll, dxT);
    if (rc) { cudaStreamSynchronize(h->stream); return rc; }
    CK(cudaMemcpyAsync(nll_steps, dsteps, sizeof(double) * N * T, cudaMemcpyDeviceToHost, h->stream));
    if (nll) CK(cudaMemcpyAsync(nll, dnll, sizeof(double) * N, cudaMemcpyDeviceToHost, h->stream));
    if (xT) CK(cudaMemcpyAsync(xT, dxT, sizeof(double) * N * L * D, cudaMemcpyDeviceToHost, h->stream));
    return refuse_nan_overflow(h);                       // waits for the copies
}

// One contiguous block of a longer sequence sharded in TIME over several devices (chunked-scan path), in three phases
// with the blocks' carries exchanged by the caller in between (include/moihgp_b200.h).
static int fsn_block_impl(moihgp_handle* h, int phase, const double* Y, size_t N, size_t T, int seq_end, int mode,
                          const double* x0, const double* u_after, const double* b_end, double* X, double* Xs, double* nll,
                          double* xT, double* host_out, double* dev_out) {
    if (!h) return -2;
    if (phase < 1 || phase > 3) return fail(h, "phase must be 1, 2 or 3");
    if (N == 0 || T == 0) return fail(h, "N and T must be positive");
    if (mode < 0 || mode > 1) return fail(h, "smoother_mode must be 0 or 1");
    if (!seq_end && T % 256 != 0) return fail(h, "a block that does not end the sequence must hold a multiple of 256 steps");
    if (phase == 1 && !Y) return -2;
    if (phase == 3 && Xs && !X) return fail(h, "Xs needs X");
    DeviceGuard guard(h->device);
    const int L = h->L, D = h->dim;
    // phases 1 and 2 leave their output in dev_out, or in a workspace that host_out is copied from
    double *xe, *out = dev_out;
    if (ws_get(h, "blk_xe", N * L * D, &xe) || (phase < 3 && !out && ws_get(h, "blk_out", N * L * (D + 1), &out))) return -1;
    ScanArgs a{};
    a.N = (long long)N; a.T = (long long)T; a.x0 = x0;
    a.X = phase == 3 ? X : nullptr; a.Xs = phase == 3 ? Xs : nullptr; a.xT = phase == 3 ? xT : nullptr;
    a.phase = phase; a.seq_end = seq_end ? 1 : 0; a.u_after = seq_end ? nullptr : u_after; a.b_end = phase == 3 ? b_end : nullptr;
    a.x_end = phase == 1 ? xe : nullptr; a.b_out = phase == 2 ? out : nullptr;
    if (const int rc = scan_pass(h, Y, mode, nll, a)) return rc;
    if (phase == 1) {
        // [N][L][D + 1]: the block's end state from x0, then its first projected observation (the previous block's u_after)
        CK(cudaMemcpy2DAsync(out, sizeof(double) * (D + 1), xe, sizeof(double) * D, sizeof(double) * D, N * L, cudaMemcpyDeviceToDevice, h->stream));
        CK(cudaMemcpy2DAsync(out + D, sizeof(double) * (D + 1), a.u, sizeof(double) * T, sizeof(double), N * L, cudaMemcpyDeviceToDevice, h->stream));
    }
    if (phase < 3 && host_out) {
        CK(cudaMemcpyAsync(host_out, out, sizeof(double) * N * L * (phase == 1 ? D + 1 : D), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

// The carry kernel of the time-sharded passes takes the block lengths by value (launch_block_carry)
static int check_time_blocks(moihgp_handle* h, size_t G, size_t rank) {
    if (G == 0 || G > (size_t)MAX_TIME_BLOCKS || rank >= G)
        return fail(h, "need 1 <= G <= " + std::to_string(MAX_TIME_BLOCKS) + " time blocks and rank < G");
    return 0;
}

int moihgp_cuda_fsn_block_dev(moihgp_handle* h, int phase, const double* Y, size_t N, size_t T, int seq_end, int mode,
                              const double* x0, const double* u_after, const double* b_end, double* X, double* Xs, double* nll,
                              double* xT, double* host_out) {
    return fsn_block_impl(h, phase, Y, N, T, seq_end, mode, x0, u_after, b_end, X, Xs, nll, xT, host_out, nullptr);
}

int moihgp_cuda_fsn_block_async(moihgp_handle* h, int phase, const double* Y, size_t N, size_t T, int seq_end, int mode,
                                const double* x0, const double* u_after, const double* b_end, double* X, double* Xs, double* nll,
                                double* xT, double* dev_out) {
    return fsn_block_impl(h, phase, Y, N, T, seq_end, mode, x0, u_after, b_end, X, Xs, nll, xT, nullptr, dev_out);
}

int moihgp_cuda_fsn_carry_dev(moihgp_handle* h, int direction, int mode, const double* gathered_dev, size_t G, const long long* block_lengths,
                              size_t rank, size_t N, const double* x0_dev, double* out_dev, double* u_after_dev) {
    if (!h || !gathered_dev || !block_lengths || !out_dev) return -2;
    if (direction < 0 || direction > 1) return fail(h, "direction must be 0 (forward) or 1 (backward)");
    if (mode < 0 || mode > 1) return fail(h, "smoother_mode must be 0 or 1");
    if (const int rc = check_time_blocks(h, G, rank)) return rc;
    DeviceGuard guard(h->device);
    CK(launch_block_carry(h->dim, direction, mode, h->d_consts, h->L, (long long)N, (int)rank, (int)G, block_lengths, gathered_dev, x0_dev,
                          nullptr, out_dev, nullptr, u_after_dev, h->stream));
    h->launches += 1;
    return 0;
}

int moihgp_cuda_smoother_power(moihgp_handle* h, int mode, size_t n, double* out) {
    if (!h || !out || mode < 0 || mode > 1) return -2;
    if (mirror(h)) return -1;
    for (int l = 0; l < h->L; ++l) {
        if (h->dim == 2) mat_pow<2>(h->consts[l].powG[mode], n, out + (size_t)l * 4);
        else mat_pow<3>(h->consts[l].powG[mode], n, out + (size_t)l * 9);
    }
    return 0;
}

// Host buffers.  Independent sequences are processed in slices, software-pipelined over three streams: the H2D copy of
// slice i+1 and the D2H copy of slice i-1 overlap the kernels of slice i (PCIe is full duplex), with two sets of
// device buffers.  (Pinned host memory is needed for the copies to be asynchronous; pageable memory still works.)
// values_only: X / Xs receive the FUNCTION-VALUE component H x = x(0) of every state only, [N][T][L] (what predict-style
// callers consume: yhat = U sqrt(S) x(0), moihgp.h:222-225) - d times fewer bytes across PCIe.
static int fsn_host(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, int mode, double* X,
                    double* Xs, double* Yhat, double* nll, double* xT, bool values_only) {
    if (!h || !Y) return -2;
    if (N == 0 || T == 0) return fail(h, "N and T must be positive");
    if (mode < -1 || mode > 1) return fail(h, "smoother_mode must be -1, 0 or 1");
    if (mode < 0 && Xs) return fail(h, "Xs requested with smoother_mode = none");
    DeviceGuard guard(h->device);
    const size_t L = h->L, D = h->dim, p = h->p;
    // slices: the call is PCIe-bound (D2H of the states), so what matters is how soon the first results can start to
    // flow back: slices as small as one warp of chains per SM allows, at most sixteen; a multiple of 32 sequences
    size_t Ns = std::max<size_t>((148 * 32 + L - 1) / L, (N + 15) / 16);
    Ns = ((Ns + 31) / 32) * 32;
    if (Ns > N) Ns = N;
    const size_t nsl = (N + Ns - 1) / Ns;
    if (!h->s_in) {
        CK(cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            CK(cudaEventCreateWithFlags(&h->ev_in[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&h->ev_c[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&h->ev_out[i], cudaEventDisableTiming));
        }
    }
    const int nbuf = nsl > 1 ? 2 : 1;
    double *dY[2] = {}, *dx0[2] = {}, *dX[2] = {}, *dXs[2] = {}, *dYh[2] = {}, *dnll[2] = {}, *dxT[2] = {}, *dF[2] = {}, *dFs[2] = {};
    static const char* names[2][9] = {{"hY0", "hx00", "hX0", "hXs0", "hYh0", "hnll0", "hxT0", "hF0", "hFs0"},
                                      {"hY1", "hx01", "hX1", "hXs1", "hYh1", "hnll1", "hxT1", "hF1", "hFs1"}};
    for (int b = 0; b < nbuf; ++b) {
        if (ws_get(h, names[b][0], Ns * T * p, &dY[b])) return -1;
        if (x0 && ws_get(h, names[b][1], Ns * L * D, &dx0[b])) return -1;
        if ((X || Yhat || Xs) && ws_get(h, names[b][2], Ns * T * L * D, &dX[b])) return -1;
        if (Xs && ws_get(h, names[b][3], Ns * T * L * D, &dXs[b])) return -1;
        if (Yhat && ws_get(h, names[b][4], Ns * T * p, &dYh[b])) return -1;
        if (nll && ws_get(h, names[b][5], Ns, &dnll[b])) return -1;
        if (xT && ws_get(h, names[b][6], Ns * L * D, &dxT[b])) return -1;
        if (values_only && X && ws_get(h, names[b][7], Ns * T * L, &dF[b])) return -1;
        if (values_only && Xs && ws_get(h, names[b][8], Ns * T * L, &dFs[b])) return -1;
    }
    int* nanf;
    if (ws_get(h, "nanf", 4, &nanf)) return -1;
    if (h->h_flags_cap < nsl) {
        if (h->h_flags) cudaFreeHost(h->h_flags);
        h->h_flags = nullptr;
        h->h_flags_cap = 0;
        CK(cudaMallocHost(&h->h_flags, sizeof(int) * nsl));
        h->h_flags_cap = nsl;
    }
    int* flags = h->h_flags;
    for (size_t i = 0; i < nsl; ++i) flags[i] = 0;
    CK(cudaStreamSynchronize(h->stream));            // earlier work on the compute stream may still use the buffers
    for (size_t i = 0; i < nsl; ++i) {
        const int b = (int)(i & 1) % nbuf;
        const size_t n0 = i * Ns, ns = std::min(Ns, N - n0);
        if (i >= 2) CK(cudaStreamWaitEvent(h->s_in, h->ev_c[b], 0));                   // input buffer b is free again
        CK(cudaMemcpyAsync(dY[b], Y + n0 * T * p, sizeof(double) * ns * T * p, cudaMemcpyHostToDevice, h->s_in));
        if (x0) CK(cudaMemcpyAsync(dx0[b], x0 + n0 * L * D, sizeof(double) * ns * L * D, cudaMemcpyHostToDevice, h->s_in));
        CK(cudaEventRecord(h->ev_in[b], h->s_in));
        CK(cudaStreamWaitEvent(h->stream, h->ev_in[b], 0));
        if (i >= 2) CK(cudaStreamWaitEvent(h->stream, h->ev_out[b], 0));               // output buffers b have been copied out
        const int rc = moihgp_cuda_filter_smoother_nll_dev(h, dY[b], ns, T, x0 ? dx0[b] : nullptr, mode, dX[b], dXs[b], dYh[b], dnll[b], dxT[b]);
        if (rc) {                                    // drain the copies already in flight into the caller's buffers
            cudaStreamSynchronize(h->s_in);
            cudaStreamSynchronize(h->stream);
            cudaStreamSynchronize(h->s_out);
            return rc;
        }
        CK(cudaMemcpyAsync(&flags[i], nanf, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaEventRecord(h->ev_c[b], h->stream));
        CK(cudaStreamWaitEvent(h->s_out, h->ev_c[b], 0));
        if (values_only) {
            // component 0 of every state, compacted on the device (in place is not possible: strides differ), then copied out
            if (X) CK(launch_extract_values(dX[b], dF[b], (long long)(ns * T * L), (int)D, h->stream));
            if (Xs) CK(launch_extract_values(dXs[b], dFs[b], (long long)(ns * T * L), (int)D, h->stream));
            h->launches += (X ? 1 : 0) + (Xs ? 1 : 0);
            CK(cudaEventRecord(h->ev_c[b], h->stream));
            CK(cudaStreamWaitEvent(h->s_out, h->ev_c[b], 0));
            if (X) CK(cudaMemcpyAsync(X + n0 * T * L, dF[b], sizeof(double) * ns * T * L, cudaMemcpyDeviceToHost, h->s_out));
            if (Xs) CK(cudaMemcpyAsync(Xs + n0 * T * L, dFs[b], sizeof(double) * ns * T * L, cudaMemcpyDeviceToHost, h->s_out));
        } else {
            if (X) CK(cudaMemcpyAsync(X + n0 * T * L * D, dX[b], sizeof(double) * ns * T * L * D, cudaMemcpyDeviceToHost, h->s_out));
            if (Xs) CK(cudaMemcpyAsync(Xs + n0 * T * L * D, dXs[b], sizeof(double) * ns * T * L * D, cudaMemcpyDeviceToHost, h->s_out));
        }
        if (Yhat) CK(cudaMemcpyAsync(Yhat + n0 * T * p, dYh[b], sizeof(double) * ns * T * p, cudaMemcpyDeviceToHost, h->s_out));
        if (nll) CK(cudaMemcpyAsync(nll + n0, dnll[b], sizeof(double) * ns, cudaMemcpyDeviceToHost, h->s_out));
        if (xT) CK(cudaMemcpyAsync(xT + n0 * L * D, dxT[b], sizeof(double) * ns * L * D, cudaMemcpyDeviceToHost, h->s_out));
        CK(cudaEventRecord(h->ev_out[b], h->s_out));
    }
    CK(cudaStreamSynchronize(h->s_out));
    CK(cudaStreamSynchronize(h->stream));
    return refuse_nan_overflow(h, flags, nsl);
}

int moihgp_cuda_filter_smoother_nll(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, int mode, double* X,
                                    double* Xs, double* Yhat, double* nll, double* xT) {
    return fsn_host(h, Y, N, T, x0, mode, X, Xs, Yhat, nll, xT, false);
}

int moihgp_cuda_filter_smoother_nll_values(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, int mode, double* F,
                                           double* Fs, double* Yhat, double* nll, double* xT) {
    return fsn_host(h, Y, N, T, x0, mode, F, Fs, Yhat, nll, xT, true);
}

int moihgp_cuda_smooth_dev(moihgp_handle* h, const double* X, size_t N, size_t T, int mode, double* Xs) {
    if (!h || !X || !Xs) return -2;
    if (N == 0 || T == 0) return fail(h, "N and T must be positive");
    if (mode < 0 || mode > 1) return fail(h, "smoother_mode must be 0 or 1");
    DeviceGuard guard(h->device);
    CK(launch_smooth_seq(X, h->d_consts, h->L, h->dim, (long long)N, (long long)T, mode, Xs, h->stream));
    h->launches += 1;
    return 0;
}

int moihgp_cuda_smooth(moihgp_handle* h, const double* X, size_t N, size_t T, int mode, double* Xs) {
    if (!h || !X || !Xs) return -2;
    if (N == 0 || T == 0) return fail(h, "N and T must be positive");
    DeviceGuard guard(h->device);
    const size_t n = N * T * (size_t)h->L * h->dim;
    double *dX, *dXs;
    if (ws_get(h, "smX", n, &dX) || ws_get(h, "smXs", n, &dXs)) return -1;
    CK(cudaMemcpyAsync(dX, X, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    const int rc = moihgp_cuda_smooth_dev(h, dX, N, T, mode, dXs);
    if (rc) return rc;
    CK(cudaMemcpyAsync(Xs, dXs, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

}  // extern "C"

namespace {

const char* sample_refusal(size_t N, size_t T, size_t S, bool any_output) {
    if (N == 0 || T == 0) return "N and T must be positive";
    if (S == 0) return "sample_posterior: the number of samples S must be positive";
    const size_t lim = (size_t)1 << 32;                  // the Philox counter holds t, n and s in 32-bit words
    if (T >= lim || N >= lim || S >= lim) return "sample_posterior: T, N and S must each be below 2^32";
    if (!any_output) return "sample_posterior: no output requested (Xsamp, Fsamp and Ysamp are all NULL)";
    return nullptr;
}

}  // namespace

extern "C" {

int moihgp_cuda_sampler_consts(moihgp_handle* h, size_t l, double* LF, double* LC) {
    if (!h || l >= (size_t)h->L) return -2;
    if (mirror(h)) return -1;
    const int d = h->dim;
    for (int i = 0; i < d; ++i) for (int j = 0; j < d; ++j) {
        if (LF) LF[i * d + j] = h->consts[l].LF[i * 3 + j];
        if (LC) LC[i * d + j] = h->consts[l].LC[i * 3 + j];
    }
    return 0;
}

int moihgp_cuda_sample_posterior_dev(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, size_t S,
                                     unsigned long long seed, double* Xs_mean, double* Xsamp, double* Fsamp, double* Ysamp) {
    if (!h || !Y) return -2;
    if (const char* m = sample_refusal(N, T, S, Xsamp || Fsamp || Ysamp)) return fail(h, m);
    DeviceGuard guard(h->device);
    const int L = h->L, D = h->dim;
    if (!Xs_mean && ws_get(h, "sXs", N * T * L * D, &Xs_mean)) return -1;
    // set_path also selects the sampler's variant (1 time-chunked, 2 one pass); the mean pass then takes the many-chains
    // kernels only where they serve the shape
    const int rc = fused_pass(h, Y, N, T, x0, MOIHGP_SMOOTH_RTS, nullptr, Xs_mean, nullptr, nullptr, nullptr, /*strict_chain=*/false);
    if (rc) return rc;
    const long long chains = (long long)(S * N * L);
    const bool chunked = sample_chunked((long long)T, chains, h->path);
    SampleArgs a;
    a.consts = h->d_consts; a.S = (long long)S; a.N = (long long)N; a.T = (long long)T; a.L = L; a.seed = seed;
    a.Xs = Xs_mean; a.Xsamp = Xsamp; a.F = Fsamp; a.carry = nullptr;
    a.mk = h->profiling ? &h->marker : nullptr;
    if (Ysamp && !Fsamp && ws_get(h, "sF", S * N * T * L, &a.F)) return -1;
    if (chunked && ws_get(h, "scarry", sample_carry_doubles(D, (long long)T, chains), &a.carry)) return -1;
    CK(launch_sample(D, a, chunked, h->stream));
    h->launches += sample_launch_count(chunked);
    if (Ysamp) {                                         // U sqrt(S) x~(0), the latent values as states of dimension 1
        CK(launch_backproject(a.F, h->d_U, h->d_S, h->p, L, 1, (long long)(S * N), (long long)T, Ysamp, h->stream));
        h->launches += 1;
        mark(a.mk, "k_backproject");
    }
    return 0;
}

int moihgp_cuda_sample_block_async(moihgp_handle* h, int phase, const double* Xs_mean, size_t N, size_t T, unsigned long long t0, int seq_end,
                                   size_t S, unsigned long long seed, const double* e_end, double* Xsamp, double* Fsamp, double* Ysamp,
                                   double* dev_out) {
    if (!h) return -2;
    if (phase < 1 || phase > 2) return fail(h, "sample_block: phase must be 1 or 2");
    if (N == 0 || T == 0) return fail(h, "N and T must be positive");
    if (S == 0) return fail(h, "sample_block: the number of samples S must be positive");
    const unsigned long long lim = 1ull << 32;           // the Philox counter holds t0 + t, n and s in 32-bit words
    if (t0 > lim || T > lim - t0) return fail(h, "sample_block: t0 + T must not exceed 2^32");
    if (N >= lim || S >= lim || S * N >= lim) return fail(h, "sample_block: S * N must be below 2^32");
    if (phase == 1 && !dev_out) return fail(h, "sample_block: phase 1 needs dev_out [S][N][L][d]");
    if (phase == 2 && !(Xsamp || Fsamp || Ysamp)) return fail(h, "sample_block: no output requested (Xsamp, Fsamp and Ysamp are all NULL)");
    if (phase == 2 && !Xs_mean) return fail(h, "sample_block: phase 2 needs Xs_mean [N][T][L][d]");
    if (phase == 2 && !seq_end && !e_end) return fail(h, "sample_block: phase 2 of a block that does not end the sequence needs e_end");
    DeviceGuard guard(h->device);
    const int L = h->L, D = h->dim;
    const long long chains = (long long)(S * N * L);
    const bool chunked = sample_chunked((long long)T, chains, h->path);
    SampleArgs a;
    a.consts = h->d_consts; a.S = (long long)S; a.N = (long long)N; a.T = (long long)T; a.L = L; a.seed = seed;
    a.Xs = Xs_mean; a.Xsamp = phase == 2 ? Xsamp : nullptr; a.F = phase == 2 ? Fsamp : nullptr; a.carry = nullptr;
    a.mk = h->profiling ? &h->marker : nullptr;
    if (phase == 2 && Ysamp && !Fsamp && ws_get(h, "sF", S * N * T * L, &a.F)) return -1;
    if (chunked && ws_get(h, "scarry", sample_carry_doubles(D, (long long)T, chains), &a.carry)) return -1;
    CK(launch_sample_block(D, phase, a, chunked, t0, seq_end, e_end, dev_out, h->stream));
    h->launches += sample_block_launch_count(phase, chunked);
    if (phase == 2 && Ysamp) {
        CK(launch_backproject(a.F, h->d_U, h->d_S, h->p, L, 1, (long long)(S * N), (long long)T, Ysamp, h->stream));
        h->launches += 1;
        mark(a.mk, "k_backproject");
    }
    return 0;
}

int moihgp_cuda_sample_posterior(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, size_t S,
                                 unsigned long long seed, double* Xs_mean, double* Xsamp, double* Fsamp, double* Ysamp) {
    if (!h || !Y) return -2;
    if (const char* m = sample_refusal(N, T, S, Xsamp || Fsamp || Ysamp)) return fail(h, m);
    DeviceGuard guard(h->device);
    const size_t L = h->L, D = h->dim, p = h->p;
    double *dY, *dx0 = nullptr, *dXs = nullptr, *dX = nullptr, *dF = nullptr, *dYs = nullptr;
    if (ws_get(h, "spY", N * T * p, &dY)) return -1;
    if (x0 && ws_get(h, "spx0", N * L * D, &dx0)) return -1;
    if (Xs_mean && ws_get(h, "spXs", N * T * L * D, &dXs)) return -1;
    if (Xsamp && ws_get(h, "spX", S * N * T * L * D, &dX)) return -1;
    if (Fsamp && ws_get(h, "spF", S * N * T * L, &dF)) return -1;
    if (Ysamp && ws_get(h, "spYs", S * N * T * p, &dYs)) return -1;
    CK(cudaMemcpyAsync(dY, Y, sizeof(double) * N * T * p, cudaMemcpyHostToDevice, h->stream));
    if (x0) CK(cudaMemcpyAsync(dx0, x0, sizeof(double) * N * L * D, cudaMemcpyHostToDevice, h->stream));
    const int rc = moihgp_cuda_sample_posterior_dev(h, dY, N, T, dx0, S, seed, dXs, dX, dF, dYs);
    if (rc) { cudaStreamSynchronize(h->stream); return rc; }
    if (Xs_mean) CK(cudaMemcpyAsync(Xs_mean, dXs, sizeof(double) * N * T * L * D, cudaMemcpyDeviceToHost, h->stream));
    if (Xsamp) CK(cudaMemcpyAsync(Xsamp, dX, sizeof(double) * S * N * T * L * D, cudaMemcpyDeviceToHost, h->stream));
    if (Fsamp) CK(cudaMemcpyAsync(Fsamp, dF, sizeof(double) * S * N * T * L, cudaMemcpyDeviceToHost, h->stream));
    if (Ysamp) CK(cudaMemcpyAsync(Ysamp, dYs, sizeof(double) * S * N * T * p, cudaMemcpyDeviceToHost, h->stream));
    return refuse_nan_overflow(h);                       // waits for the copies
}

// phase 0: whole evaluation; 1: begin (projection, summaries, block end from a zero carry-in -> zend, device);
// 2: finish (from the true carry-in; reuses the workspace phase 1 filled)
static int objective_phase(moihgp_handle* h, int phase, const double* Y, size_t N, size_t T, const double* x0, const double* dx0,
                           double* loss, double* grad, double* xT, double* dxT, double* zend) {
    if (!h || !Y) return -2;
    if (N == 0 || T == 0) return fail(h, "N and T must be positive");
    DeviceGuard guard(h->device);
    const int L = h->L, D = h->dim, p = h->p;
    const size_t nC = obj_chunks((long long)T), nsplit = obj_gu_splits((long long)N, (long long)T);
    ProjectWs pw;
    double *w, *yl, *zsum, *zin, *zsub, *part, *gU, *Ek, *lat;
    if (project_ws(h, N, T, &pw) || ws_get(h, "w", N * L * T, &w) || ws_get(h, "yl", N * L * T, &yl) ||
        ws_get(h, "zsum", nC * N * L * 4 * D, &zsum) || ws_get(h, "zin", nC * N * L * 4 * D, &zin) || ws_get(h, "zsub", nC * 8 * N * L * 4 * D, &zsub) ||
        ws_get(h, "part", nC * N * L * 8, &part) ||
        ws_get(h, "gU", nsplit * p * L, &gU) || ws_get(h, "Ek", (size_t)L * 27 * 16, &Ek) || ws_get(h, "lat", ((size_t)L + 1) * 8 * 16, &lat))
        return -1;
    Marker* mk = h->profiling ? &h->marker : nullptr;
    if (mk) { mk->st = h->stream; mk->mark("begin"); }
    if (phase != 2) {
        CK(cudaMemsetAsync(pw.nanf, 0, 2 * sizeof(int), h->stream));
        CK(launch_project(Y, h->d_U, h->d_S, p, L, (long long)N, (long long)T, pw.u, w, yl, pw.rho, nullptr, pw.nanf, pw.nanrows, (long long)pw.nan_cap, pw.lsg, h->stream));
        mark(mk, "k_project");
        h->launches += 2;
    }
    ObjArgs a;
    a.mk = mk;
    a.phase = phase;
    a.zend = zend;
    a.Y = Y; a.u = pw.u; a.w = w; a.yl = yl; a.rho = pw.rho; a.wgt = w;   // the weights overwrite w in place (same thread, same index)
    a.consts = h->d_consts; a.U = h->d_U; a.S = h->d_S; a.sigma = h->sigma; a.p = p; a.L = L; a.threading = h->threading;
    a.N = (long long)N; a.T = (long long)T; a.x0 = x0; a.dx0 = dx0; a.zsum = zsum; a.zin = zin; a.zsub = zsub; a.part = part; a.gU_part = gU;
    a.Ek = Ek; a.lat_sums = lat; a.loss = loss; a.grad = grad; a.xT = xT; a.dxT = dxT;
    CK(launch_objective(D, a, h->stream));
    h->launches += obj_launch_count((long long)T, L);
    return 0;
}

int moihgp_cuda_objective_dev(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, const double* dx0,
                              double* loss, double* grad, double* xT, double* dxT) {
    if (!loss || !grad) return -2;
    return objective_phase(h, 0, Y, N, T, x0, dx0, loss, grad, xT, dxT, nullptr);
}

// Time-sharded evaluation (SURVEY 8(e)): this device holds a contiguous block of T time steps of each sequence.
int moihgp_cuda_objective_begin_dev(moihgp_handle* h, const double* Y, size_t N, size_t T, double* zend_host) {
    if (!h) return -2;
    if (zend_host && T % 256 != 0) return fail(h, "objective_begin: the block end state needs a block length that is a multiple of 256 steps");
    double* dz = nullptr;
    const size_t nz = N * (size_t)h->L * 4 * h->dim;
    if (zend_host && ws_get(h, "zend", nz, &dz)) return -1;
    const int rc = objective_phase(h, 1, Y, N, T, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, dz);
    if (rc) return rc;
    if (zend_host) {
        CK(cudaMemcpyAsync(zend_host, dz, sizeof(double) * nz, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

int moihgp_cuda_objective_begin_async(moihgp_handle* h, const double* Y, size_t N, size_t T, double* zend_dev) {
    if (!h) return -2;
    if (zend_dev && T % 256 != 0) return fail(h, "objective_begin: the block end state needs a block length that is a multiple of 256 steps");
    return objective_phase(h, 1, Y, N, T, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, zend_dev);
}

int moihgp_cuda_carry_in_dev(moihgp_handle* h, const double* ends_dev, size_t G, const long long* block_lengths, size_t rank, size_t N,
                             const double* x0_dev, const double* dx0_dev, double* xin_dev, double* dxin_dev) {
    if (!h || !xin_dev || !dxin_dev || (rank > 0 && (!ends_dev || !block_lengths))) return -2;
    if (const int rc = check_time_blocks(h, G, rank)) return rc;
    DeviceGuard guard(h->device);
    CK(launch_block_carry(h->dim, 0, 0, h->d_consts, h->L, (long long)N, (int)rank, (int)G, block_lengths, ends_dev, x0_dev, dx0_dev, xin_dev,
                          dxin_dev, nullptr, h->stream));
    h->launches += 1;
    return 0;
}

int moihgp_cuda_objective_finish_dev(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, const double* dx0,
                                     double* loss, double* grad, double* xT, double* dxT) {
    if (!loss || !grad) return -2;
    return objective_phase(h, 2, Y, N, T, x0, dx0, loss, grad, xT, dxT, nullptr);
}

// One short sequence (the streaming learner's window): everything in ONE launch, inputs and outputs through one pinned
// staging buffer (one H2D, k_obj_small, one D2H).  Y_resident != null: the observations are already on the device.
// Returns 1 if the kernel met a missing (NaN) output - the caller then takes the general path.
static int objective_small(moihgp_handle* h, const double* Y, const double* Y_resident, size_t T, const double* x0, const double* dx0,
                           double* loss, double* grad, double* xT, double* dxT) {
    const size_t L = h->L, D = h->dim, p = h->p, np = h->num_param;
    const size_t nY = Y_resident ? 0 : T * p, nx = L * D, ndx = 3 * L * D;
    const size_t nin = nY + nx + ndx, nout = np + 2 + nx + ndx;
    if (h->h_small_cap < nin + nout) {
        if (h->h_small) cudaFreeHost(h->h_small);
        h->h_small = nullptr;
        h->h_small_cap = 0;
        CK(cudaMallocHost(&h->h_small, sizeof(double) * (nin + nout)));
        h->h_small_cap = nin + nout;
    }
    double* dbuf;
    if (ws_get(h, "small", nin + nout, &dbuf)) return -1;
    double* hb = h->h_small;
    if (nY) std::copy(Y, Y + nY, hb);
    if (x0) std::copy(x0, x0 + nx, hb + nY); else std::fill(hb + nY, hb + nY + nx, 0.0);
    if (dx0) std::copy(dx0, dx0 + ndx, hb + nY + nx); else std::fill(hb + nY + nx, hb + nin, 0.0);
    CK(cudaMemcpyAsync(dbuf, hb, sizeof(double) * nin, cudaMemcpyHostToDevice, h->stream));
    double* dout = dbuf + nin;
    CK(launch_objective_small((int)D, Y_resident ? Y_resident : dbuf, h->d_U, h->d_S, h->sigma, h->d_consts, (int)p, (int)L, (long long)T,
                              h->threading, dbuf + nY, dbuf + nY + nx, dout, dout + np + 2, dout + np + 2 + nx, h->stream));
    h->launches += 1;
    CK(cudaMemcpyAsync(hb + nin, dout, sizeof(double) * nout, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const double* ho = hb + nin;
    if (ho[1] != 0.0) return 1;
    *loss = ho[0];
    std::copy(ho + 2, ho + 2 + np, grad);
    if (xT) std::copy(ho + np + 2, ho + np + 2 + nx, xT);
    if (dxT) std::copy(ho + np + 2 + nx, ho + nout, dxT);
    return 0;
}

// The objective on host buffers, over host Y (copied in) or over Y_resident, observations already on the device.
static int objective_host(moihgp_handle* h, const double* Y, const double* Y_resident, size_t N, size_t T, const double* x0,
                          const double* dx0, double* loss, double* grad, double* xT, double* dxT) {
    DeviceGuard guard(h->device);
    if (N == 1 && h->path != 1 && obj_small_smem(h->p, h->L, (long long)T)) {
        const int rs = objective_small(h, Y, Y_resident, T, x0, dx0, loss, grad, xT, dxT);
        if (rs <= 0) return rs;                  // 1: missing observations -> the general path below
    }
    const size_t L = h->L, D = h->dim, p = h->p, np = h->num_param;
    double *dY = nullptr, *dx = nullptr, *ddx = nullptr, *dout, *dxT_ = nullptr, *ddxT = nullptr;
    if (!Y_resident && ws_get(h, "hY", N * T * p, &dY)) return -1;
    if (ws_get(h, "hout", np + 2, &dout)) return -1;
    if (x0 && ws_get(h, "hx0", N * L * D, &dx)) return -1;
    if (dx0 && ws_get(h, "hdx0", N * L * 3 * D, &ddx)) return -1;
    if (xT && ws_get(h, "hxT", N * L * D, &dxT_)) return -1;
    if (dxT && ws_get(h, "hdxT", N * L * 3 * D, &ddxT)) return -1;
    if (!Y_resident) CK(cudaMemcpyAsync(dY, Y, sizeof(double) * N * T * p, cudaMemcpyHostToDevice, h->stream));
    if (x0) CK(cudaMemcpyAsync(dx, x0, sizeof(double) * N * L * D, cudaMemcpyHostToDevice, h->stream));
    if (dx0) CK(cudaMemcpyAsync(ddx, dx0, sizeof(double) * N * L * 3 * D, cudaMemcpyHostToDevice, h->stream));
    const int rc = moihgp_cuda_objective_dev(h, Y_resident ? Y_resident : dY, N, T, dx, ddx, dout, dout + 2, dxT_, ddxT);
    if (rc) return rc;
    std::vector<double> host(np + 2);
    CK(cudaMemcpyAsync(host.data(), dout, sizeof(double) * (np + 2), cudaMemcpyDeviceToHost, h->stream));
    if (xT) CK(cudaMemcpyAsync(xT, dxT_, sizeof(double) * N * L * D, cudaMemcpyDeviceToHost, h->stream));
    if (dxT) CK(cudaMemcpyAsync(dxT, ddxT, sizeof(double) * N * L * 3 * D, cudaMemcpyDeviceToHost, h->stream));
    if (const int refused = refuse_nan_overflow(h)) return refused;   // waits for the copies
    *loss = host[0];
    std::copy(host.begin() + 2, host.end(), grad);
    return 0;   // with NaN observations the loss is NaN, exactly as the reference's (moihgp.h:501 uses the full y)
}

int moihgp_cuda_objective(moihgp_handle* h, const double* Y, size_t N, size_t T, const double* x0, const double* dx0, double* loss,
                          double* grad, double* xT, double* dxT) {
    if (!h || !Y || !loss || !grad) return -2;
    if (N == 0 || T == 0) return fail(h, "N and T must be positive");
    return objective_host(h, Y, nullptr, N, T, x0, dx0, loss, grad, xT, dxT);
}

// Resident data set: the L-BFGS loop evaluates the objective tens of times on the SAME observations (LBFGSB.h:137,
// LineSearchMoreThuente.h:212,295), so the H2D copy of Y is paid once.
int moihgp_cuda_bind_data(moihgp_handle* h, const double* Y, size_t N, size_t T) {
    if (!h) return -2;
    DeviceGuard guard(h->device);
    CK(cudaStreamSynchronize(h->stream));
    if (h->d_bound) { cudaFree(h->d_bound); h->d_bound = nullptr; }
    h->bound_N = h->bound_T = 0;
    if (!Y || N == 0 || T == 0) return 0;                    // unbind
    CK(cudaMalloc(&h->d_bound, sizeof(double) * N * T * h->p));
    CK(cudaMemcpyAsync(h->d_bound, Y, sizeof(double) * N * T * h->p, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->bound_N = N;
    h->bound_T = T;
    return 0;
}

int moihgp_cuda_objective_bound(moihgp_handle* h, const double* x0, const double* dx0, double* loss, double* grad, double* xT, double* dxT) {
    if (!h || !loss || !grad) return -2;
    if (!h->d_bound) return fail(h, "no data bound: call moihgp_cuda_bind_data first");
    return objective_host(h, nullptr, h->d_bound, h->bound_N, h->bound_T, x0, dx0, loss, grad, xT, dxT);
}

}  // extern "C"

// =============================================================================================
// Device-resident streaming learner (SURVEY 8 f2; moihgp_online.h:40-93, :173-187).  The window of observations, its moving
// mean, the state carried in front of the window and the proximal matrix live in HBM; one objective evaluation is
//   H2D params -> polar factor -> K-setup -> one-launch window objective -> proximal term -> D2H [loss, grad, U]
// queued on the handle's stream and, from the second evaluation of a given window length on, replayed as ONE CUDA graph.
static int online_enqueue(moihgp_handle* h, size_t T, bool has_B) {
    moihgp_handle::Online& o = h->on;
    const int p = h->p, L = h->L, np = h->num_param, pL = p * L;
    CK(cudaMemcpyAsync(o.d_params, o.h_params, sizeof(double) * np, cudaMemcpyHostToDevice, h->stream));
    CK(launch_polar(o.d_params, p, L, h->d_U, o.d_pst, h->stream));                                     // moihgp.h:436-446
    CK(cudaMemcpyAsync(h->d_S, o.d_params + pL, sizeof(double) * L, cudaMemcpyDeviceToDevice, h->stream));   // moihgp.h:448
    CK(launch_setup(h->dim, o.d_params + pL + L + 1, h->dt, L, h->d_consts, h->stream));                // moihgp.h:450-456
    CK(launch_objective_small(h->dim, o.d_win, h->d_U, h->d_S, 0.0, h->d_consts, p, L, (long long)T, h->threading, o.d_x, o.d_dx, o.d_out,
                              nullptr, nullptr, h->stream, o.d_ma, o.d_params + pL + L));               // moihgp_online.h:57-70
    CK(launch_online_prox(o.d_params, o.has_prox ? o.d_old : nullptr, has_B ? o.d_B : nullptr, np, pL, h->d_U, o.d_out, h->stream));   // moihgp_online.h:42-54
    CK(cudaMemcpyAsync(o.h_out, o.d_out, sizeof(double) * (2 + np + pL), cudaMemcpyDeviceToHost, h->stream));
    return 0;
}

extern "C" {

int moihgp_cuda_online_begin(moihgp_handle* h, size_t windowsize) {
    if (!h) return -2;
    if (windowsize < 1) windowsize = 1;                                   // moihgp_online.h:144-151
    // the learner's CUDA graph holds the one-CTA polar factor, whose Newton-Schulz kernel handles at most 64 columns
    if (h->L > 64) return fail(h, "online_begin: the streaming learner supports num_latent <= 64");
    if (!obj_small_smem(h->p, h->L, (long long)windowsize)) return fail(h, "online_begin: window too long / model too large for the one-launch objective");
    if (polar_smem_bytes(h->p, h->L) > 200 * 1024) return fail(h, "online_begin: p * L too large for the one-CTA polar factor");
    DeviceGuard guard(h->device);
    CK(cudaStreamSynchronize(h->stream));
    moihgp_handle::Online& o = h->on;
    for (auto& kv : o.graphs) cudaGraphExecDestroy(kv.second);
    o.graphs.clear();
    o.seen.clear();
    const size_t p = h->p, L = h->L, D = h->dim, np = h->num_param, pL = p * L;
    auto dalloc = [&](double** q, size_t n) { if (*q) cudaFree(*q); *q = nullptr; return cudaMalloc(q, sizeof(double) * std::max<size_t>(n, 2)); };
    CK(dalloc(&o.d_win, (windowsize + 1) * p)); CK(dalloc(&o.d_ma, p)); CK(dalloc(&o.d_ynew, p)); CK(dalloc(&o.d_magiven, p)); CK(dalloc(&o.d_front, p));
    CK(dalloc(&o.d_x, L * D)); CK(dalloc(&o.d_dx, L * 3 * D)); CK(dalloc(&o.d_x2, L * D)); CK(dalloc(&o.d_dx2, L * 3 * D));
    CK(dalloc(&o.d_params, np)); CK(dalloc(&o.d_old, np)); CK(dalloc(&o.d_out, 2 + np + pL));
    if (o.d_B) { cudaFree(o.d_B); o.d_B = nullptr; }
    if (!o.d_count) CK(cudaMalloc(&o.d_count, 4 * sizeof(int)));
    if (!o.d_pst) CK(cudaMalloc(&o.d_pst, 4 * sizeof(int)));
    if (o.h_params) cudaFreeHost(o.h_params);
    if (o.h_out) cudaFreeHost(o.h_out);
    if (o.h_y) cudaFreeHost(o.h_y);
    CK(cudaMallocHost(&o.h_params, sizeof(double) * np));
    CK(cudaMallocHost(&o.h_out, sizeof(double) * (2 + np + pL)));
    CK(cudaMallocHost(&o.h_y, sizeof(double) * 2 * p));
    CK(cudaMemsetAsync(o.d_count, 0, 4 * sizeof(int), h->stream));
    CK(cudaMemsetAsync(o.d_x, 0, sizeof(double) * L * D, h->stream));
    CK(cudaMemsetAsync(o.d_dx, 0, sizeof(double) * L * 3 * D, h->stream));
    CK(cudaMemsetAsync(o.d_ma, 0, sizeof(double) * p, h->stream));
    // the proximal term starts from the current parameters and the identity (moihgp_online.h:31, :50-53)
    std::vector<double> cur(np);
    moihgp_cuda_get_params(h, cur.data());
    CK(cudaMemcpyAsync(o.d_old, cur.data(), sizeof(double) * np, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    o.W = windowsize; o.count = 0; o.has_B = false; o.has_prox = true;
    return 0;
}

// OnlineObjective::push_back(y)  moihgp_online.h:75-93.  ma_given = NULL: the moving mean is the mean of the window (the
// element about to be dropped included, as the reference computes it); otherwise the caller's own centre is used
// (online_learning.py:54-64 keeps an exponential mean).  ma_out (may be NULL) receives the centre in use.
int moihgp_cuda_online_push(moihgp_handle* h, const double* y, const double* ma_given, double* ma_out) {
    if (!h || !y) return -2;
    moihgp_handle::Online& o = h->on;
    if (o.W == 0) return fail(h, "online_push: call moihgp_cuda_online_begin first");
    DeviceGuard guard(h->device);
    const size_t p = h->p, L = h->L, D = h->dim;
    std::memcpy(o.h_y, y, sizeof(double) * p);
    if (ma_given) std::memcpy(o.h_y + p, ma_given, sizeof(double) * p);
    CK(cudaMemcpyAsync(o.d_ynew, o.h_y, sizeof(double) * p, cudaMemcpyHostToDevice, h->stream));
    if (ma_given) CK(cudaMemcpyAsync(o.d_magiven, o.h_y + p, sizeof(double) * p, cudaMemcpyHostToDevice, h->stream));
    CK(launch_online_push(o.d_ynew, ma_given ? o.d_magiven : nullptr, (int)p, (int)o.W, o.d_win, o.d_count, o.d_ma, o.d_front, h->stream));
    h->launches += 1;
    if (o.count + 1 > o.W) {
        // the window slid: the carried state advances with the NEW front element (Q12), step v2 (moihgp_online.h:89)
        StepArgs a;
        a.consts = h->d_consts; a.U = h->d_U; a.S = h->d_S; a.sigma = h->sigma; a.p = h->p; a.L = h->L; a.dim = h->dim; a.threading = h->threading;
        a.x = o.d_x; a.y = o.d_front; a.dx = o.d_dx; a.xnew = o.d_x2; a.yhat = nullptr; a.dxnew = o.d_dx2;
        CK(launch_step(a, h->stream));
        h->launches += 1;
        CK(cudaMemcpyAsync(o.d_x, o.d_x2, sizeof(double) * L * D, cudaMemcpyDeviceToDevice, h->stream));
        CK(cudaMemcpyAsync(o.d_dx, o.d_dx2, sizeof(double) * L * 3 * D, cudaMemcpyDeviceToDevice, h->stream));
    } else {
        o.count += 1;
    }
    if (ma_out) {
        CK(cudaMemcpyAsync(o.h_y, o.d_ma, sizeof(double) * p, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        std::memcpy(ma_out, o.h_y, sizeof(double) * p);
    }
    return 0;
}

// The proximal term 1/2 dparams' B dparams (moihgp_online.h:42-54): oldparams [num_param] and the matrix B [num_param]^2
// row-major, e.g. column j = bfgs_mat.apply_Hv(e_j, gamma) (NULL = the identity, the reference's choice while the BFGS
// matrix holds no correction).  Set once per streamed sample (moihgp_online.h:182-183).
int moihgp_cuda_online_set_proximal(moihgp_handle* h, const double* oldparams, const double* B) {
    if (!h) return -2;
    moihgp_handle::Online& o = h->on;
    if (o.W == 0) return fail(h, "online_set_proximal: call moihgp_cuda_online_begin first");
    DeviceGuard guard(h->device);
    const size_t np = h->num_param;
    if (!oldparams) {                                   // no proximal term on the device: the caller adds its own
        CK(cudaStreamSynchronize(h->stream));
        o.has_prox = false; o.has_B = false;
        return 0;
    }
    o.has_prox = true;
    CK(cudaMemcpyAsync(o.d_old, oldparams, sizeof(double) * np, cudaMemcpyHostToDevice, h->stream));
    if (B) {
        if (!o.d_B) CK(cudaMalloc(&o.d_B, sizeof(double) * np * np));
        CK(cudaMemcpyAsync(o.d_B, B, sizeof(double) * np * np, cudaMemcpyHostToDevice, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));              // the caller's buffers may be reused right away
    o.has_B = B != nullptr;
    return 0;
}

// OnlineObjective::operator()(params, grad)  moihgp_online.h:40-72 on the resident window: update(params) + the window loop
// of step v2 + negLogLikelihood(x, y, dx, grad) from the carried state + the proximal term.  loss[1], grad[num_param] (host).
// The model afterwards holds `params` (polar factor taken), exactly as after moihgp_cuda_update(params).
int moihgp_cuda_online_objective(moihgp_handle* h, const double* params, double* loss, double* grad) {
    if (!h || !params || !loss || !grad) return -2;
    moihgp_handle::Online& o = h->on;
    if (o.W == 0 || o.count == 0) return fail(h, "online_objective: no window (online_begin / online_push first)");
    DeviceGuard guard(h->device);
    const int p = h->p, L = h->L, np = h->num_param, pL = p * L;
    std::memcpy(o.h_params, params, sizeof(double) * np);
    const long long key = (long long)o.count * 4 + (o.has_prox ? 2 : 0) + (o.has_B ? 1 : 0);
    const int seen = o.seen[key]++;
    auto it = o.graphs.find(key);
    if (it == o.graphs.end() && seen >= 1) {
        // second evaluation with this window length: record the sequence once (the first one ran eagerly and set every
        // function attribute / workspace), replay it from now on
        cudaGraph_t g = nullptr;
        cudaGraphExec_t ge = nullptr;
        if (cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            const int rc = online_enqueue(h, o.count, o.has_B);
            const cudaError_t ce = cudaStreamEndCapture(h->stream, &g);
            if (rc == 0 && ce == cudaSuccess && g && cudaGraphInstantiate(&ge, g, 0) == cudaSuccess) it = o.graphs.emplace(key, ge).first;
            if (g) cudaGraphDestroy(g);
        }
        cudaGetLastError();                              // a failed capture falls back to the eager sequence below
    }
    if (it != o.graphs.end()) { CK(cudaGraphLaunch(it->second, h->stream)); h->launches += 5; }
    else { if (online_enqueue(h, o.count, o.has_B)) return -1; h->launches += 5; }
    CK(cudaStreamSynchronize(h->stream));
    if (o.h_out[1] != 0.0) return fail(h, "online_objective: missing (NaN) outputs in the window are not handled on the resident path");
    *loss = o.h_out[0];
    std::memcpy(grad, o.h_out + 2, sizeof(double) * np);
    // host mirror of the model (moihgp_cuda_get_params / get_U): the polar factor came back with the result
    std::copy(o.h_out + 2 + np, o.h_out + 2 + np + pL, h->U.begin());
    for (int l = 0; l < L; ++l) h->S[l] = params[pL + l];
    h->sigma = params[pL + L];
    for (int i = 0; i < 3 * L; ++i) h->igp[i] = params[pL + L + 1 + i];
    h->consts_fresh = false;
    return 0;
}

// the state carried in front of the window (OnlineObjective::_x, _dx): x [L][d], dx [L][3][d]
int moihgp_cuda_online_get_state(moihgp_handle* h, double* x, double* dx) {
    if (!h) return -2;
    moihgp_handle::Online& o = h->on;
    if (o.W == 0) return fail(h, "online_get_state: call moihgp_cuda_online_begin first");
    DeviceGuard guard(h->device);
    const size_t L = h->L, D = h->dim;
    if (x) CK(cudaMemcpyAsync(x, o.d_x, sizeof(double) * L * D, cudaMemcpyDeviceToHost, h->stream));
    if (dx) CK(cudaMemcpyAsync(dx, o.d_dx, sizeof(double) * L * 3 * D, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

}  // extern "C"

extern "C" {

// ---------------------------------------------------------------------------------------------
// legacy symbols (src/wrapper.cpp:31-624).  Same signatures; errors cannot be returned, so they abort.
#define LEGACY_DEF(XX, KERNEL_EXPR)                                                                                        \
    moihgp_handle* gp##XX##_new(double dt, size_t num_output, size_t num_latent, bool threading) {                          \
        return legacy_new(KERNEL_EXPR, dt, num_output, num_latent, threading);                                              \
    }                                                                                                                       \
    void gp##XX##_del(moihgp_handle* gp) { moihgp_cuda_destroy(gp); }                                                       \
    void gp##XX##_step1(moihgp_handle* gp, double* x, double* y, double* dx, double* xnew, double* yhat, double* dxnew) {   \
        if (step_call(gp, x, y, dx, xnew, yhat, dxnew)) legacy_fatal(gp, "gp" #XX "_step1");                                \
    }                                                                                                                       \
    void gp##XX##_step2(moihgp_handle* gp, double* x, double* y, double* dx, double* xnew, double* dxnew) {                 \
        if (step_call(gp, x, y, dx, xnew, nullptr, dxnew)) legacy_fatal(gp, "gp" #XX "_step2");                             \
    }                                                                                                                       \
    void gp##XX##_step3(moihgp_handle* gp, double* x, double* y, double* xnew, double* yhat) {                              \
        if (step_call(gp, x, y, nullptr, xnew, yhat, nullptr)) legacy_fatal(gp, "gp" #XX "_step3");                         \
    }                                                                                                                       \
    void gp##XX##_step4(moihgp_handle* gp, double* x, double* xnew, double* yhat) {                                         \
        if (step_call(gp, x, nullptr, nullptr, xnew, yhat, nullptr)) legacy_fatal(gp, "gp" #XX "_step4");                   \
    }                                                                                                                       \
    void gp##XX##_update(moihgp_handle* gp, double* params) {                                                               \
        if (moihgp_cuda_update(gp, params)) legacy_fatal(gp, "gp" #XX "_update");                                           \
    }                                                                                                                       \
    double gp##XX##_lik1(moihgp_handle* gp, double* x, double* y, double* dx, double* grad) {                               \
        double loss = 0.0;                                                                                                  \
        if (lik_call(gp, x, y, dx, &loss, grad)) legacy_fatal(gp, "gp" #XX "_lik1");                                        \
        return loss;                                                                                                        \
    }                                                                                                                       \
    double gp##XX##_lik2(moihgp_handle* gp, double* x, double* y) {                                                         \
        double loss = 0.0;                                                                                                  \
        if (lik_call(gp, x, y, nullptr, &loss, nullptr)) legacy_fatal(gp, "gp" #XX "_lik2");                                \
        return loss;                                                                                                        \
    }                                                                                                                       \
    void gp##XX##_get_params(moihgp_handle* gp, double* params) { moihgp_cuda_get_params(gp, params); }                     \
    size_t gp##XX##_igp_dim(moihgp_handle* gp) { return (size_t)gp->dim; }                                                  \
    size_t gp##XX##_num_param(moihgp_handle* gp) { return (size_t)gp->num_param; }                                          \
    size_t gp##XX##_num_igp_param(moihgp_handle* gp) { return 3; }

LEGACY_DEF(32, 32)
LEGACY_DEF(52, kernel_for_gp52())

}  // extern "C"
