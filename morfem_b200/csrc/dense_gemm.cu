// FP64 tensor-pipe (DMMA.8x8x4) complex128 contractions of the basis and projection stages.
//
//   gemm_tn : C (ra x rb) = op(A)^T B, reduction over the long row index n (tall-skinny Gram / Q^T Y).
//             Replaces BLAS gemm behind `(q_t @ a) @ q` (implementation.py:181-183) and forms the Gram
//             matrices of the CholeskyQR2 replacement of np.linalg.svd (implementation.py:226/298/210).
//   gemm_nn : Out (n x rb) = A (n x ra) W (ra x rb): the `S R^-1` and `Q1 (R2^-1 U)` applications.
//
// Complex data stays interleaved: one 16-byte shared-memory load yields the (re, im) pair of a fragment.  Each complex
// 8x8x4 block product is three real DMMAs in Gauss's form (cmma3, common.cuh) instead of four: a warp forms the operand
// combinations of a fragment once (one DADD per A fragment, two per B fragment) and reuses them across its warp tile, and
// the three accumulator planes are combined into (re, im) in the epilogue.  Three planes of a 32 x 32 warp tile would not
// fit the register file next to the fragments, so a warp owns 32 x 16 (96 accumulator registers) and the CTAs have twice
// the warps of the four-product kernels at the same CTA tile.  Operand tiles are staged with cp.async (LDGSTS) in a 3-stage
// ring; shared-memory leading dimensions are padded so every quarter-warp fragment load is conflict-free.
// Roofline: FP64 tensor pipe (37.05 TFLOP/s measured, tools/fp64_peaks.cu) for r >~ 48, HBM below that.
#include "common.cuh"

namespace {

constexpr int KC = 16;        // rows of the reduction index per pipeline stage
constexpr int STAGES = 3;

// ------------------------------------------------------------------------------------------------ gemm_tn
constexpr int TN_TI = 64, TN_TJ = 64, TN_THREADS = 256;      // 2 x 4 warps, each 32 x 16
constexpr int TN_LDA = TN_TI + 2, TN_LDB = TN_TJ + 2;        // == 2 (mod 8) complex -> conflict-free fragments
constexpr int TN_STAGE_ELEMS = KC * (TN_LDA + TN_LDB);

// CONJ: C = A^H B.  With a = ar - i ai the 3M planes are k1 += (ar - ai) br and k3 += ai (br + bi) with re = k1 + k3, so no operand
// is negated in the loop.
template <bool CONJ>
__global__ void __launch_bounds__(TN_THREADS, 2)      // <= 128 registers: two CTAs (16 warps) per SM
gemm_tn_kernel(const cplx* __restrict__ A, long long lda, int ra, const cplx* __restrict__ B, long long ldb, int rb,
               long long n, long long rows_per_split, cplx* __restrict__ part, int herm) {
    extern __shared__ __align__(16) cplx smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wi = warp >> 2, wj = warp & 3;
    const int ntj = (rb + TN_TJ - 1) / TN_TJ;
    const int ti = blockIdx.x / ntj, tj = blockIdx.x - ti * ntj;
    if (herm && ti > tj) return;               // Gram matrix A^H A: the lower tiles are the conjugate transposes of the upper ones
    const int i0 = ti * TN_TI, j0 = tj * TN_TJ;
    const long long n0 = (long long)blockIdx.y * rows_per_split;
    long long n1 = n0 + rows_per_split; if (n1 > n) n1 = n;
    const int nchunks = n1 > n0 ? (int)((n1 - n0 + KC - 1) / KC) : 0;

    auto load_stage = [&](int stage, int chunk) {
        cplx* As = smem + stage * TN_STAGE_ELEMS;
        cplx* Bs = As + KC * TN_LDA;
        const long long row_base = n0 + (long long)chunk * KC;
#pragma unroll
        for (int q = 0; q < (KC * TN_TI) / TN_THREADS; ++q) {
            int idx = tid + q * TN_THREADS;
            int rr = idx / TN_TI, cc = idx - rr * TN_TI;
            long long row = row_base + rr;
            bool ok = row < n1 && (i0 + cc) < ra;
            const cplx* src = A + (ok ? row * lda + i0 + cc : 0);
            cp_async16(As + rr * TN_LDA + cc, src, ok);
        }
#pragma unroll
        for (int q = 0; q < (KC * TN_TJ) / TN_THREADS; ++q) {
            int idx = tid + q * TN_THREADS;
            int rr = idx / TN_TJ, cc = idx - rr * TN_TJ;
            long long row = row_base + rr;
            bool ok = row < n1 && (j0 + cc) < rb;
            const cplx* src = B + (ok ? row * ldb + j0 + cc : 0);
            cp_async16(Bs + rr * TN_LDB + cc, src, ok);
        }
    };

    double k1[4][2][2], k2[4][2][2], k3[4][2][2];            // the three 3M planes of a 4 x 2 grid of 8 x 8 tiles
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) k1[i][j][e] = k2[i][j][e] = k3[i][j][e] = 0.0;

    for (int s = 0; s < STAGES - 1; ++s) { if (s < nchunks) load_stage(s, s); cp_async_commit(); }
    for (int c = 0; c < nchunks; ++c) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        { int nc = c + STAGES - 1; if (nc < nchunks) load_stage(nc % STAGES, nc); cp_async_commit(); }
        const cplx* As = smem + (c % STAGES) * TN_STAGE_ELEMS;
        const cplx* Bs = As + KC * TN_LDA;
#pragma unroll
        for (int kk = 0; kk < KC / 4; ++kk) {
            double br[2], bd[2], bs[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const cplx b = Bs[(kk * 4 + t) * TN_LDB + wj * 16 + j * 8 + g];
                br[j] = b.x; bd[j] = b.y - b.x; bs[j] = b.x + b.y;
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const cplx a = As[(kk * 4 + t) * TN_LDA + wi * 32 + i * 8 + g];
                const double as = CONJ ? a.x - a.y : a.x + a.y;
#pragma unroll
                for (int j = 0; j < 2; ++j) cmma3(k1[i][j], k2[i][j], k3[i][j], a.x, a.y, as, br[j], bd[j], bs[j]);
            }
        }
    }
    cp_async_wait<0>();
    // partial tile -> part[split][ra][rb]; the planes are combined here, so the split-K summation sees (re, im) as before
    cplx* out = part + (long long)blockIdx.y * ra * rb;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            int row = i0 + wi * 32 + i * 8 + g;
            int col = j0 + wj * 16 + j * 8 + 2 * t;
            if (row < ra) {
#pragma unroll
                for (int e = 0; e < 2; ++e)
                    if (col + e < rb)
                        out[(long long)row * rb + col + e] = cmake(CONJ ? k1[i][j][e] + k3[i][j][e] : k1[i][j][e] - k3[i][j][e],
                                                                   k1[i][j][e] + k2[i][j][e]);
            }
        }
}

// C = sum over splits of part[s] in a FIXED order (deterministic: replicated r x r factorisations on several ranks see
// bit-identical input).  One CTA per 32 consecutive elements: lane -> element (coalesced 512-byte rows), warp w sums
// splits w, w+8, ... with independent loads in flight; the eight warp partials are combined in warp order.
constexpr int RED_WARPS = 8;
__global__ void __launch_bounds__(RED_WARPS * 32)
reduce_partials_kernel(const cplx* __restrict__ part, int nsplit, int ra, int rb, cplx* __restrict__ C, long long ldc, int herm) {
    __shared__ cplx red[RED_WARPS][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long total = (long long)ra * rb;
    const long long oidx = (long long)blockIdx.x * 32 + lane;
    long long idx = oidx;
    bool mirror = false;
    if (herm && oidx < total) {                // lower tiles were not computed: read the mirrored element and conjugate
        const int i = (int)(oidx / rb), j = (int)(oidx - (long long)i * rb);
        if (i / TN_TI > j / TN_TJ) { idx = (long long)j * rb + i; mirror = true; }
    }
    cplx acc0 = cmake(0.0, 0.0), acc1 = cmake(0.0, 0.0);
    if (idx < total) {
        int s = warp;
        for (; s + RED_WARPS < nsplit; s += 2 * RED_WARPS) {
            const cplx v0 = part[(long long)s * total + idx], v1 = part[(long long)(s + RED_WARPS) * total + idx];
            acc0 = cadd(acc0, v0); acc1 = cadd(acc1, v1);
        }
        if (s < nsplit) acc0 = cadd(acc0, part[(long long)s * total + idx]);
    }
    red[warp][lane] = cadd(acc0, acc1);
    __syncthreads();
    if (warp == 0 && oidx < total) {
        cplx acc = red[0][lane];
#pragma unroll
        for (int w = 1; w < RED_WARPS; ++w) acc = cadd(acc, red[w][lane]);
        if (mirror) acc.y = -acc.y;
        const int i = (int)(oidx / rb), j = (int)(oidx - (long long)i * rb);
        C[i * ldc + j] = acc;
    }
}

// `symm`: only the upper-triangular tiles do work (Gram matrices), so the row index is split into more, shorter ranges
void tn_plan(int ra, int rb, long long n, int& tiles, int& nsplit, long long& rows_per_split, bool symm = false) {
    tiles = ((ra + TN_TI - 1) / TN_TI) * ((rb + TN_TJ - 1) / TN_TJ);
    const int nt = (ra + TN_TI - 1) / TN_TI;
    const int work_tiles = symm ? nt * (nt + 1) / 2 : tiles;
    const int target = 148 * 2 * 2;   // two waves of two resident CTAs per SM (B200: 148 SMs)
    long long max_split = (n + (long long)KC * 8 - 1) / ((long long)KC * 8);
    if (max_split < 1) max_split = 1;
    long long s = target / work_tiles; if (s < 1) s = 1; if (s > max_split) s = max_split;
    rows_per_split = (n + s - 1) / s;
    rows_per_split = (rows_per_split + KC - 1) / KC * KC;
    if (rows_per_split < KC) rows_per_split = KC;
    nsplit = (int)((n + rows_per_split - 1) / rows_per_split); if (nsplit < 1) nsplit = 1;
}

// ------------------------------------------------------------------------------------------------ gemm_nn
constexpr int NN_TM = 128, NN_TN = 64, NN_THREADS = 512;     // 4 x 4 warps, each 32 x 16
constexpr int NN_LDA = KC + 4;          // == 4 (mod 8): A-fragment (row g, col t) loads conflict-free
constexpr int NN_LDW = NN_TN + 2;
constexpr int NN_STAGE_ELEMS = NN_TM * NN_LDA + KC * NN_LDW;

__global__ void __launch_bounds__(NN_THREADS, 1)      // <= 128 registers: one 16-warp CTA per SM
gemm_nn_kernel(const cplx* __restrict__ A, long long lda, long long n, int ra, const cplx* __restrict__ W, long long ldw, int rb,
               cplx* __restrict__ Out, long long ldo, int w_upper) {
    extern __shared__ __align__(16) cplx smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp >> 2, wn = warp & 3;          // 4 x 4 warps, each 32 x 16
    const int ntn = (rb + NN_TN - 1) / NN_TN;
    const long long tm = blockIdx.x / ntn; const int tn = (int)(blockIdx.x - tm * ntn);
    const long long m0 = tm * NN_TM; const int j0 = tn * NN_TN;
    // upper-triangular W (the R^-1 of a Cholesky-QR pass): rows k >= j0 + NN_TN of this column tile are zero, skip them
    const int kmax = (w_upper && j0 + NN_TN < ra) ? j0 + NN_TN : ra;
    const int nchunks = (kmax + KC - 1) / KC;

    // A rows of this thread: tid / KC + q NN_THREADS / KC, column tid % KC of every chunk (row pointer and bounds fixed once:
    // the 16-warp CTA runs at the 128-register cap)
    constexpr int NN_AQ = (NN_TM * KC) / NN_THREADS, NN_AROWS = NN_THREADS / KC;
    const int a_rr = tid / KC, a_cc = tid - a_rr * KC;
    const cplx* a_src = A + (m0 + a_rr) * lda + a_cc;
    unsigned a_rows_ok = 0;
#pragma unroll
    for (int q = 0; q < NN_AQ; ++q) a_rows_ok |= (m0 + a_rr + q * NN_AROWS < n) ? 1u << q : 0u;

    auto load_stage = [&](int stage, int chunk) {
        cplx* As = smem + stage * NN_STAGE_ELEMS;
        cplx* Ws = As + NN_TM * NN_LDA;
        const int k0 = chunk * KC;
#pragma unroll
        for (int q = 0; q < NN_AQ; ++q) {
            const bool ok = ((a_rows_ok >> q) & 1u) && (k0 + a_cc) < ra;
            const cplx* src = ok ? a_src + q * NN_AROWS * lda + k0 : A;
            cp_async16(As + (a_rr + q * NN_AROWS) * NN_LDA + a_cc, src, ok);
        }
#pragma unroll
        for (int q = 0; q < (KC * NN_TN) / NN_THREADS; ++q) {
            int idx = tid + q * NN_THREADS;
            int rr = idx / NN_TN, cc = idx - rr * NN_TN;
            bool ok = (k0 + rr) < ra && (j0 + cc) < rb;
            const cplx* src = W + (ok ? (long long)(k0 + rr) * ldw + j0 + cc : 0);
            cp_async16(Ws + rr * NN_LDW + cc, src, ok);
        }
    };

    double k1[4][2][2], k2[4][2][2], k3[4][2][2];            // the three 3M planes of a 4 x 2 grid of 8 x 8 tiles
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) k1[i][j][e] = k2[i][j][e] = k3[i][j][e] = 0.0;

    for (int s = 0; s < STAGES - 1; ++s) { if (s < nchunks) load_stage(s, s); cp_async_commit(); }
    for (int c = 0; c < nchunks; ++c) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        { int nc = c + STAGES - 1; if (nc < nchunks) load_stage(nc % STAGES, nc); cp_async_commit(); }
        const cplx* As = smem + (c % STAGES) * NN_STAGE_ELEMS;
        const cplx* Ws = As + NN_TM * NN_LDA;
#pragma unroll
        for (int kk = 0; kk < KC / 4; ++kk) {
            double br[2], bd[2], bs[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const cplx b = Ws[(kk * 4 + t) * NN_LDW + wn * 16 + j * 8 + g];
                br[j] = b.x; bd[j] = b.y - b.x; bs[j] = b.x + b.y;
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const cplx a = As[(wm * 32 + i * 8 + g) * NN_LDA + kk * 4 + t];
                const double as = a.x + a.y;
#pragma unroll
                for (int j = 0; j < 2; ++j) cmma3(k1[i][j], k2[i][j], k3[i][j], a.x, a.y, as, br[j], bd[j], bs[j]);
            }
        }
    }
    cp_async_wait<0>();
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            long long row = m0 + wm * 32 + i * 8 + g;
            int col = j0 + wn * 16 + j * 8 + 2 * t;
            const double re0 = k1[i][j][0] - k3[i][j][0], im0 = k1[i][j][0] + k2[i][j][0];
            const double re1 = k1[i][j][1] - k3[i][j][1], im1 = k1[i][j][1] + k2[i][j][1];
            if (row < n) {
                if (col + 1 < rb) {
                    // two adjacent complex elements: 32 contiguous bytes
                    double4 v = make_double4(re0, im0, re1, im1);
                    cplx* dst = Out + row * ldo + col;
                    if ((reinterpret_cast<uintptr_t>(dst) & 31) == 0) *reinterpret_cast<double4*>(dst) = v;
                    else { dst[0] = cmake(v.x, v.y); dst[1] = cmake(v.z, v.w); }
                } else if (col < rb) {
                    Out[row * ldo + col] = cmake(re0, im0);
                }
            }
        }
}

}  // namespace

extern "C" size_t mf_gemm_tn_ws_bytes(int ra, int rb, int64_t n) {
    if (ra <= 0 || rb <= 0 || n <= 0) return 16;
    int tiles, nsplit, nsplit2 = 0; long long rps;
    tn_plan(ra, rb, n, tiles, nsplit, rps);
    if (ra == rb) tn_plan(ra, rb, n, tiles, nsplit2, rps, true);       // the Gram path uses more splits
    return sizeof(cplx) * (size_t)(nsplit > nsplit2 ? nsplit : nsplit2) * ra * rb;
}

extern "C" int mf_gemm_tn_c128(const mf_c128* A, int64_t lda, int ra, const mf_c128* B, int64_t ldb, int rb, int64_t n,
                               int conj_a, mf_c128* C, int64_t ldc, void* ws, size_t ws_bytes, void* stream) {
    if (!A) MF_FAIL_ARG(1, "A is NULL");
    if (ra <= 0 || lda < ra) MF_FAIL_ARG(3, "need 0 < ra <= lda");
    if (!B) MF_FAIL_ARG(4, "B is NULL");
    if (rb <= 0 || ldb < rb) MF_FAIL_ARG(6, "need 0 < rb <= ldb");
    if (n < 0) MF_FAIL_ARG(7, "n < 0");
    if (!C || ldc < rb) MF_FAIL_ARG(9, "C is NULL or ldc < rb");
    if (!ws || ws_bytes < mf_gemm_tn_ws_bytes(ra, rb, n)) MF_FAIL_ARG(11, "workspace too small (mf_gemm_tn_ws_bytes)");
    cudaStream_t st = (cudaStream_t)stream;
    int tiles, nsplit; long long rps;
    const int herm = (conj_a && (const void*)A == (const void*)B && lda == ldb && ra == rb) ? 1 : 0;
    tn_plan(ra, rb, n > 0 ? n : 1, tiles, nsplit, rps, herm != 0);
    const size_t smem = sizeof(cplx) * STAGES * TN_STAGE_ELEMS;
    auto kern = conj_a ? gemm_tn_kernel<true> : gemm_tn_kernel<false>;
    MF_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(tiles, nsplit);
    kern<<<grid, TN_THREADS, smem, st>>>((const cplx*)A, lda, ra, (const cplx*)B, ldb, rb, n, rps, (cplx*)ws, herm);
    MF_CHECK_LAUNCH();
    long long total = (long long)ra * rb;
    reduce_partials_kernel<<<(unsigned)((total + 31) / 32), RED_WARPS * 32, 0, st>>>((const cplx*)ws, nsplit, ra, rb, (cplx*)C, ldc, herm);
    MF_CHECK_LAUNCH();
    return 0;
}

static int gemm_nn_c128_impl(const mf_c128* A, int64_t lda, int64_t n, int ra, const mf_c128* W, int64_t ldw, int rb,
                            mf_c128* Out, int64_t ldo, void* stream, int w_upper) {
    if (!A) MF_FAIL_ARG(1, "A is NULL");
    if (ra <= 0 || lda < ra) MF_FAIL_ARG(4, "need 0 < ra <= lda");
    if (n < 0) MF_FAIL_ARG(3, "n < 0");
    if (!W || ldw < rb) MF_FAIL_ARG(5, "W is NULL or ldw < rb");
    if (rb <= 0) MF_FAIL_ARG(7, "rb <= 0");
    if (!Out || ldo < rb) MF_FAIL_ARG(8, "Out is NULL or ldo < rb");
    if ((const void*)Out == (const void*)A) MF_FAIL_ARG(8, "Out must not alias A");
    if (n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = sizeof(cplx) * STAGES * NN_STAGE_ELEMS;
    MF_CHECK_CUDA(cudaFuncSetAttribute(gemm_nn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    long long tiles_m = (n + NN_TM - 1) / NN_TM;
    int tiles_n = (rb + NN_TN - 1) / NN_TN;
    long long grid = tiles_m * tiles_n;
    if (grid > 0x7fffffffLL) MF_FAIL_ARG(3, "n too large for one launch");
    gemm_nn_kernel<<<(unsigned)grid, NN_THREADS, smem, st>>>((const cplx*)A, lda, n, ra, (const cplx*)W, ldw, rb, (cplx*)Out, ldo, w_upper);
    MF_CHECK_LAUNCH();
    return 0;
}

extern "C" int mf_gemm_nn_c128(const mf_c128* A, int64_t lda, int64_t n, int ra, const mf_c128* W, int64_t ldw, int rb,
                               mf_c128* Out, int64_t ldo, void* stream) {
    return gemm_nn_c128_impl(A, lda, n, ra, W, ldw, rb, Out, ldo, stream, 0);
}

extern "C" int mf_trmm_nn_c128(const mf_c128* A, int64_t lda, int64_t n, int r, const mf_c128* W, int64_t ldw,
                               mf_c128* Out, int64_t ldo, void* stream) {
    return gemm_nn_c128_impl(A, lda, n, r, W, ldw, r, Out, ldo, stream, 1);
}
