// Posterior sample paths of the latent processes: steady-state forward-filtering, backward-sampling (sm_100a).
//
// In RTS form a draw is  x~[T-1] = X[T-1] + LF z[T-1],  x~[t] = X[t] + G (x~[t+1] - A X[t]) + LC z[t]  with G = G[1],
// LF LF' = PF and LC LC' = PF - G PPc G' (k_setup).  Subtracting the RTS mean recursion leaves  x~ = Xs_rts + e  with
//   e[T-1] = LF z[T-1],   e[t] = G e[t+1] + LC z[t],
// a process that does not depend on the data: one RTS pass of the fused kernels serves every sample, and these kernels add
// the noise.  Every (sample s, sequence n, latent l) chain is independent.
//
// Random numbers: one Philox4x32-10 call per (s, n, l, t) with counter (t, n, l, s) and key (seed lo, seed hi), uniforms
// (w + 0.5) 2^-32, Box-Muller in fp64; z = the first d normals.  A draw depends on (seed, s, n, l, t) only - not on the
// variant, the launch shape or the number of samples - so the time-parallel variant regenerates its numbers instead of
// storing them.
//
// Variants (launch_sample picks one from the number of chains):
//   one pass     k_sample<D, 0>: a thread per chain walks backwards over the whole sequence.
//   time-chunked k_sample<D, 1> runs every chunk of time backwards from a zero carry and keeps only its start value;
//                k_sample_carry chains the chunk starts from the end of the sequence with G^len (binary powering on the
//                powG[1] tables); k_sample<D, 2> runs every chunk again from its true carry and writes the outputs.
//   k_sample_block: the same kernels on one block of a sequence sharded in time over several devices (DESIGN 4.8).
#include <cuda_runtime.h>
#include <curand_philox4x32_x.h>
#include "launch.h"
#include "small_mat.cuh"

namespace moihgp {

namespace {

constexpr int kThreads = 128;

// z[0..D-1] of the draw (s, n, l, t)
template <int D>
__device__ __forceinline__ void normals(uint2 key, unsigned s, unsigned n, unsigned l, unsigned t, double* z) {
    const uint4 w = curand_Philox4x32_10(make_uint4(t, n, l, s), key);
    constexpr double k2m32 = 2.3283064365386962890625e-10;     // 2^-32
    double sn, cs;
    const double r0 = sqrt(-2.0 * log(((double)w.x + 0.5) * k2m32));
    sincospi(2.0 * (((double)w.y + 0.5) * k2m32), &sn, &cs);
    z[0] = r0 * cs;
    z[1] = r0 * sn;
    if (D > 2) {                                                 // z2 = r1 cos(2 pi u3); z3 is not needed
        const double r1 = sqrt(-2.0 * log(((double)w.z + 0.5) * k2m32));
        z[2] = r1 * cospi(2.0 * (((double)w.w + 0.5) * k2m32));
    }
}

// e <- M e + Lo z   (Lo lower-triangular)
template <int D>
__device__ __forceinline__ void step(const double* M, const double* Lo, const double* z, double* e) {
    double en[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
        double a = 0.0;
#pragma unroll
        for (int k = 0; k <= i; ++k) a = fma(Lo[i * D + k], z[k], a);
#pragma unroll
        for (int k = 0; k < D; ++k) a = fma(M[i * D + k], e[k], a);
        en[i] = a;
    }
#pragma unroll
    for (int i = 0; i < D; ++i) e[i] = en[i];
}

// One block of a sequence sharded in time (moihgp_cuda_sample_block_async): t0 is the global index of its first step (the
// Philox counter is t0 + t), seq_end says whether it ends the sequence, e_end [S N L][D] is e at the first step after it
// (null: zero, the phase-1 start).  The whole sequence is {0, 1, null}.
struct SampleBlock {
    unsigned long long t0 = 0;
    int seq_end = 1;
    const double* e_end = nullptr;
};

// PHASE 0: one pass over the whole sequence, outputs written.  PHASE 1: chunk from a zero carry, start value -> carry.
// PHASE 2: chunk from its true carry (carry[c + 1]), outputs written.  Thread index = chunk * chains + chain,
// chain = (s N + n) L + l, so that the lanes of a warp write neighbouring latents of one state row.
// BLOCK: the call covers one block of the sequence (b); false compiles the whole-sequence kernels, which ignore b.
template <int D, int PHASE, bool BLOCK>
__device__ __forceinline__ void sample_chunk(const SampleArgs& a, long long chunk_len, long long nC, const SampleBlock& b) {
    const long long chains = a.S * a.N * a.L;
    const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= chains * nC) return;
    const long long c = id / chains, chain = id - c * chains;
    const int l = (int)(chain % a.L);
    const long long sn = chain / a.L, s = sn / a.N, n = sn - s * a.N;
    const LatentConsts& k = a.consts[l];
    double G[D * D], LC[D * D], LF[D * D];
#pragma unroll
    for (int i = 0; i < D; ++i)
#pragma unroll
        for (int j = 0; j < D; ++j) {
            G[i * D + j] = k.G[1][i * 3 + j];
            LC[i * D + j] = k.LC[i * 3 + j];
            LF[i * D + j] = k.LF[i * 3 + j];
        }
    const uint2 key = make_uint2((unsigned)(a.seed & 0xffffffffull), (unsigned)(a.seed >> 32));
    const long long t_lo = c * chunk_len, t_hi = min(a.T, t_lo + chunk_len);
    const long long stride = (long long)a.L * D;                 // one time step of a [.][T][L][D] array
    const double* xs = a.Xs + ((size_t)n * a.T * a.L + l) * D;
    double* xo = a.Xsamp ? a.Xsamp + ((size_t)sn * a.T * a.L + l) * D : nullptr;
    double* fo = a.F ? a.F + (size_t)sn * a.T * a.L + l : nullptr;
    double e[D], z[D];
    auto emit = [&](long long t) {
        if (PHASE == 1) return;
        if (xo) {
#pragma unroll
            for (int i = 0; i < D; ++i) xo[t * stride + i] = xs[t * stride + i] + e[i];
            if (fo) fo[t * a.L] = xo[t * stride];
        } else {
            fo[t * a.L] = xs[t * stride] + e[0];
        }
    };
    const unsigned t0 = BLOCK ? (unsigned)b.t0 : 0u;             // t0 + t < 2^32 (moihgp_cuda_sample_block_async)
    long long t = t_hi - 1;
    if (t_hi == a.T && (!BLOCK || b.seq_end)) {                  // the end of the sequence: e = LF z
        normals<D>(key, (unsigned)s, (unsigned)n, (unsigned)l, t0 + (unsigned)t, z);
#pragma unroll
        for (int i = 0; i < D; ++i) e[i] = 0.0;
        step<D>(G, LF, z, e);
        emit(t);
        --t;
    } else if (BLOCK && t_hi == a.T && b.e_end) {                // the block's last step: e_end from the next block
#pragma unroll
        for (int i = 0; i < D; ++i) e[i] = b.e_end[chain * D + i];
    } else if (PHASE == 1 || (BLOCK && t_hi == a.T)) {
#pragma unroll
        for (int i = 0; i < D; ++i) e[i] = 0.0;
    } else {
        const double* cin = a.carry + ((size_t)(c + 1) * chains + chain) * D;
#pragma unroll
        for (int i = 0; i < D; ++i) e[i] = cin[i];
    }
#pragma unroll 2
    for (; t >= t_lo; --t) {
        normals<D>(key, (unsigned)s, (unsigned)n, (unsigned)l, t0 + (unsigned)t, z);
        step<D>(G, LC, z, e);
        emit(t);
    }
    if (PHASE == 1) {
        double* co = a.carry + ((size_t)c * chains + chain) * D;
#pragma unroll
        for (int i = 0; i < D; ++i) co[i] = e[i];
    }
}

template <int D, int PHASE>
__global__ void __launch_bounds__(kThreads) k_sample(const SampleArgs a, long long chunk_len, long long nC) {
    sample_chunk<D, PHASE, false>(a, chunk_len, nC, SampleBlock{});
}

template <int D, int PHASE>
__global__ void __launch_bounds__(kThreads) k_sample_block(const SampleArgs a, long long chunk_len, long long nC, const SampleBlock b) {
    sample_chunk<D, PHASE, true>(a, chunk_len, nC, b);
}

// carry[c][chain] <- e at the start of chunk c:  E(nC-1) = carry(nC-1),  E(c) = carry(c) + G^chunk_len E(c+1).
// One thread per chain; the next chunks' values are loaded ahead of the dependent matrix-vector chain.
template <int D>
__global__ void __launch_bounds__(kThreads) k_sample_carry(const SampleArgs a, long long chunk_len, long long nC) {
    const long long chains = a.S * a.N * a.L;
    const long long chain = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (chain >= chains) return;
    const LatentConsts& k = a.consts[chain % a.L];
    double P[D * D];
    mat_pow<D>(k.powG[1], chunk_len, P);                         // P = G^chunk_len
    double* cv = a.carry + (size_t)chain * D;
    const size_t cs = (size_t)chains * D;                        // one chunk of the carry array
    double e[D];
#pragma unroll
    for (int i = 0; i < D; ++i) e[i] = cv[(size_t)(nC - 1) * cs + i];
    constexpr int U = 8;
    for (long long c0 = nC - 2; c0 >= 0; c0 -= U) {
        double v[U][D];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int i = 0; i < D; ++i) v[u][i] = c0 - u >= 0 ? cv[(size_t)(c0 - u) * cs + i] : 0.0;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (c0 - u < 0) break;
            double en[D];
#pragma unroll
            for (int i = 0; i < D; ++i) {
                double s = v[u][i];
#pragma unroll
                for (int q = 0; q < D; ++q) s = fma(P[i * D + q], e[q], s);
                en[i] = s;
            }
#pragma unroll
            for (int i = 0; i < D; ++i) { e[i] = en[i]; cv[(size_t)(c0 - u) * cs + i] = en[i]; }
        }
    }
}

unsigned blocks(long long threads) { return (unsigned)((threads + kThreads - 1) / kThreads); }

template <int D>
cudaError_t run_sample(const SampleArgs& a, bool chunked, cudaStream_t st) {
    const long long chains = a.S * a.N * a.L;
    if (!chunked) {
        k_sample<D, 0><<<blocks(chains), kThreads, 0, st>>>(a, a.T, 1);
        mark(a.mk, "k_sample");
        return cudaGetLastError();
    }
    const long long cl = sample_chunk_len(a.T, chains), nC = (a.T + cl - 1) / cl;
    k_sample<D, 1><<<blocks(chains * nC), kThreads, 0, st>>>(a, cl, nC);
    mark(a.mk, "k_sample_chunks");
    k_sample_carry<D><<<blocks(chains), kThreads, 0, st>>>(a, cl, nC);
    mark(a.mk, "k_sample_carry");
    k_sample<D, 2><<<blocks(chains * nC), kThreads, 0, st>>>(a, cl, nC);
    mark(a.mk, "k_sample_final");
    return cudaGetLastError();
}

// One block of a sharded sequence.  Phase 1: e at the block's first step from a zero e_end -> e_start [S N L][D] (one pass:
// a walk with no stores; chunked: the chain's chunk-0 value).  Phase 2: the paths, the last chunk starting from b.e_end
// (LF z on the block that ends the sequence).
template <int D>
cudaError_t run_sample_block(int phase, SampleArgs a, bool chunked, SampleBlock b, double* e_start, cudaStream_t st) {
    const long long chains = a.S * a.N * a.L;
    if (phase == 1) b.e_end = nullptr;
    if (!chunked) {
        if (phase == 1) {
            a.carry = e_start;
            k_sample_block<D, 1><<<blocks(chains), kThreads, 0, st>>>(a, a.T, 1, b);
        } else {
            k_sample_block<D, 0><<<blocks(chains), kThreads, 0, st>>>(a, a.T, 1, b);
        }
        mark(a.mk, "k_sample_block");
        return cudaGetLastError();
    }
    const long long cl = sample_chunk_len(a.T, chains), nC = (a.T + cl - 1) / cl;
    k_sample_block<D, 1><<<blocks(chains * nC), kThreads, 0, st>>>(a, cl, nC, b);
    mark(a.mk, "k_sample_block_chunks");
    k_sample_carry<D><<<blocks(chains), kThreads, 0, st>>>(a, cl, nC);
    mark(a.mk, "k_sample_carry");
    if (phase == 1) {
        const cudaError_t e = cudaMemcpyAsync(e_start, a.carry, sizeof(double) * chains * D, cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) return e;
    } else {
        k_sample_block<D, 2><<<blocks(chains * nC), kThreads, 0, st>>>(a, cl, nC, b);
        mark(a.mk, "k_sample_block_final");
    }
    return cudaGetLastError();
}

}  // namespace

// One pass as soon as the chains alone give every SM eight warps: with fewer, the one-pass loop cannot hide its fp64
// latency and the time-chunked variant is faster despite drawing every normal twice (config 3 at S = 1, 7 warps per SM:
// 19.2 ms chunked vs 23.0 ms one pass on a B200, profiles/r03).  Chunks are sized for about 2048 threads per SM (>= 32 steps).
bool sample_chunked(long long T, long long chains, int path) {
    if (path == 1) return true;
    if (path == 2) return false;
    return chains < 148LL * 8 * 32 && T > 32;
}

long long sample_chunk_len(long long T, long long chains) {
    const long long want = (148LL * 2048 + chains - 1) / chains;   // chunks per chain
    const long long cl = (T + want - 1) / want;
    return cl < 32 ? 32 : cl;
}

size_t sample_carry_doubles(int dim, long long T, long long chains) {
    const long long cl = sample_chunk_len(T, chains);
    return (size_t)((T + cl - 1) / cl) * chains * dim;
}

int sample_launch_count(bool chunked) { return chunked ? 3 : 1; }

cudaError_t launch_sample(int dim, const SampleArgs& a, bool chunked, cudaStream_t st) {
    return dim == 3 ? run_sample<3>(a, chunked, st) : run_sample<2>(a, chunked, st);
}

int sample_block_launch_count(int phase, bool chunked) { return chunked ? (phase == 1 ? 2 : 3) : 1; }

cudaError_t launch_sample_block(int dim, int phase, const SampleArgs& a, bool chunked, unsigned long long t0, int seq_end, const double* e_end,
                                double* e_start, cudaStream_t st) {
    SampleBlock b;
    b.t0 = t0; b.seq_end = seq_end ? 1 : 0; b.e_end = e_end;
    return dim == 3 ? run_sample_block<3>(phase, a, chunked, b, e_start, st) : run_sample_block<2>(phase, a, chunked, b, e_start, st);
}

}  // namespace moihgp
