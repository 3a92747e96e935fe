// Shared device/host helpers for the morfem_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include "../../include/morfem_b200.h"

typedef double2 cplx;   // interleaved complex128, layout-compatible with mf_c128

extern thread_local char g_mf_err[512];
extern std::atomic<long long> g_mf_launches;

#define MF_FAIL_ARG(idx, msg)                                                         \
    do { snprintf(g_mf_err, sizeof(g_mf_err), "%s: argument %d: %s", __func__, (idx), (msg)); return -(idx); } while (0)

#define MF_CHECK_LAUNCH()                                                             \
    do {                                                                              \
        g_mf_launches.fetch_add(1, std::memory_order_relaxed);                        \
        cudaError_t e__ = cudaGetLastError();                                         \
        if (e__ != cudaSuccess) {                                                     \
            snprintf(g_mf_err, sizeof(g_mf_err), "%s: launch failed: %s", __func__, cudaGetErrorString(e__)); \
            return (int)e__;                                                          \
        }                                                                             \
    } while (0)

#define MF_CHECK_CUDA(call)                                                           \
    do {                                                                              \
        cudaError_t e__ = (call);                                                     \
        if (e__ != cudaSuccess) {                                                     \
            snprintf(g_mf_err, sizeof(g_mf_err), "%s: %s: %s", __func__, #call, cudaGetErrorString(e__)); \
            return (int)e__;                                                          \
        }                                                                             \
    } while (0)

__host__ __device__ __forceinline__ cplx cmake(double re, double im) { return make_double2(re, im); }
__device__ __forceinline__ cplx cadd(cplx a, cplx b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ cplx csub(cplx a, cplx b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ cplx cmul(cplx a, cplx b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ cplx cconj(cplx a) { return make_double2(a.x, -a.y); }
__device__ __forceinline__ cplx cscale(double s, cplx a) { return make_double2(s * a.x, s * a.y); }
// acc += a*b
__device__ __forceinline__ void cfma(cplx& acc, cplx a, cplx b) {
    acc.x = fma(a.x, b.x, acc.x); acc.x = fma(-a.y, b.y, acc.x);
    acc.y = fma(a.x, b.y, acc.y); acc.y = fma(a.y, b.x, acc.y);
}
// acc -= a*b
__device__ __forceinline__ void cfms(cplx& acc, cplx a, cplx b) {
    acc.x = fma(-a.x, b.x, acc.x); acc.x = fma(a.y, b.y, acc.x);
    acc.y = fma(-a.x, b.y, acc.y); acc.y = fma(-a.y, b.x, acc.y);
}
// |re| + |im|: the magnitude LAPACK's izamax (pivot search in zgetrf) uses; equals |x| for real data (idamax)
__device__ __forceinline__ double cabs1(cplx a) { return fabs(a.x) + fabs(a.y); }
__device__ __forceinline__ double cnorm2(cplx a) { return a.x * a.x + a.y * a.y; }
// 1/a with scaling against overflow (Smith's method)
__device__ __forceinline__ cplx crecip(cplx a) {
    if (fabs(a.x) >= fabs(a.y)) {
        double t = a.y / a.x, d = a.x + a.y * t;
        return make_double2(1.0 / d, -t / d);
    } else {
        double t = a.x / a.y, d = a.x * t + a.y;
        return make_double2(t / d, -1.0 / d);
    }
}

// D(8x8) += A(8x4) * B(4x8), fp64 tensor pipe (SASS DMMA.8x8x4).
// lane = 4*g + t:  a = A[g][t], b = B[t][g], c0 = D[g][2t], c1 = D[g][2t+1].
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// Complex 8x8x4 block product in Gauss's three-multiplication form ("3M", as in ZGEMM3M): three real DMMAs instead of four.
// With a = ar + i ai (A fragment) and b = br + i bi (B fragment), three accumulator planes take
//   k1 += (ar + ai) br,   k2 += ar (bi - br),   k3 += ai (br + bi),   and then   re = k1 - k3,   im = k1 + k2.
// The operand combinations are formed once per fragment and reused by every tile the fragment feeds.  On real data embedded in
// complex128 (ai = bi = 0) k1 is the same DMMA sequence as the real plane of the four-product form, k2 = -k1 and k3 = 0 exactly, so
// re is bit-identical to it and im is exactly zero.  On complex data the error stays normwise of order k eps |A| |B| with a somewhat
// larger constant than the four-product form.
__device__ __forceinline__ void cmma3(double (&k1)[2], double (&k2)[2], double (&k3)[2], double ar, double ai, double as,
                                      double br, double bd, double bs) {
    dmma884(k1[0], k1[1], as, br);
    dmma884(k2[0], k2[1], ar, bd);
    dmma884(k3[0], k3[1], ai, bs);
}

// Ampere-style async copy, 16 bytes, global -> shared (SASS LDGSTS), with zero-fill predicate.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, bool valid) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    int bytes = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" :: "r"(s), "l"(gmem_src), "r"(bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" :: "n"(N)); }

// Device-wide barriers of a co-resident (cooperative) grid.
// (1) shared arrival counter: thread 0 of every CTA adds 1 and polls the counter with a back-off (~2.4 us with 128 CTAs).
__device__ __forceinline__ void mf_grid_barrier_counter(unsigned* counter, unsigned& epoch, unsigned nblocks) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned target = (epoch + 1u) * nblocks;
        atomicAdd(counter, 1u);
        while (*((volatile unsigned*)counter) < target) { __nanosleep(32); }
        __threadfence();
    }
    epoch += 1u;
    __syncthreads();
}
// (2) one flag word per CTA, polled by the first warp of every CTA: no atomics, but every CTA reads every flag, so it
// only pays for small grids (measured: 128 CTAs polling 128 words turn the flag lines into an L2 hot spot and the
// barrier gets twice as slow as the counter; with the <= 32 CTAs of the fused Cholesky kernel it is the faster one).
__device__ __forceinline__ void mf_grid_barrier_flags(unsigned* flags, unsigned& epoch, unsigned nblocks) {
    __syncthreads();
    epoch += 1u;
    if (threadIdx.x < 32) {
        if (threadIdx.x == 0) {
            __threadfence();
            *((volatile unsigned*)(flags + blockIdx.x)) = epoch;
        }
        bool done;
        do {
            done = true;
            for (unsigned i = threadIdx.x; i < nblocks; i += 32) done = done && (*((volatile unsigned*)(flags + i)) >= epoch);
            done = __all_sync(0xffffffffu, done);
            if (!done) __nanosleep(20);
        } while (!done);
        __threadfence();
    }
    __syncthreads();
}

static inline int mf_num_sms() {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    return sms;
}
