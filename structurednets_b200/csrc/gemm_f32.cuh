// fp32 SIMT GEMM building block shared by the low-rank (fp32 path), Toeplitz-like and LDR layers:
//     C[M x N] = alpha * op(A)[M x K] * op(B)[K x N] + beta * C  (+ bias[N] broadcast over rows)
// Row-major, arbitrary leading dimensions, op in {N, T}.  128x128x16 CTA tile, 8x8 register tile per
// thread (256 threads), operands staged through shared memory as [k][m] / [k][n] so the inner loop
// reads two float4 pairs per 64 FMAs.  Fully predicated at the edges.
//
// This is deliberately a plain CUDA-core kernel: the fp32 parity bar (1e-5 relative) rules out a
// single-pass TF32/BF16 tensor-core product here; the bf16 configuration of the low-rank layer has
// its own tcgen05 path (lr_tc.cu).
#pragma once
#include <stdlib.h>
#include "common.cuh"
#include "gemm_tf32x3.cuh"

namespace snb {

constexpr int GB_M = 128, GB_N = 128, GB_K = 16, G_THREADS = 256;

// ksplit > 1: blockIdx.z owns a K slice and the epilogue is an atomic accumulation C += alpha*acc
// (used for the batch-reduction GEMMs of the backward passes, whose M x N output is tiny).
template <bool TA, bool TB>
__global__ void __launch_bounds__(G_THREADS)
gemm_f32_kernel(int M, int N, int Kfull, int kslice, float alpha, const float* __restrict__ A, long lda, const float* __restrict__ B,
                long ldb, float beta, float* __restrict__ C, long ldc, const float* __restrict__ bias) {
    __shared__ __align__(16) float As[GB_K][GB_M + 4];
    __shared__ __align__(16) float Bs[GB_K][GB_N + 4];
    const int tid = threadIdx.x;
    const int m0 = blockIdx.y * GB_M, n0 = blockIdx.x * GB_N;
    const int tx = tid & 15, ty = tid >> 4;  // 16 x 16 threads, each 8 x 8 outputs (two 4-wide halves)
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    const int kbeg = blockIdx.z * kslice;
    const int K = min(Kfull, kbeg + kslice);
    const bool atomic_out = gridDim.z > 1;
    for (int k0 = kbeg; k0 < K; k0 += GB_K) {
        // A tile -> As[k][m]
#pragma unroll
        for (int it = 0; it < (GB_M * GB_K) / G_THREADS; ++it) {
            int e = tid + it * G_THREADS;
            int m, k;
            if (TA) { m = e % GB_M; k = e / GB_M; }   // A is K x M in memory: consecutive threads along m
            else    { k = e % GB_K; m = e / GB_K; }   // A is M x K in memory: consecutive threads along k
            int gm = m0 + m, gk = k0 + k;
            float v = 0.f;
            if (gm < M && gk < K) v = TA ? __ldg(A + (size_t)gk * lda + gm) : __ldg(A + (size_t)gm * lda + gk);
            As[k][m] = v;
        }
#pragma unroll
        for (int it = 0; it < (GB_N * GB_K) / G_THREADS; ++it) {
            int e = tid + it * G_THREADS;
            int n, k;
            if (TB) { k = e % GB_K; n = e / GB_K; }   // B is N x K in memory
            else    { n = e % GB_N; k = e / GB_N; }   // B is K x N in memory
            int gn = n0 + n, gk = k0 + k;
            float v = 0.f;
            if (gn < N && gk < K) v = TB ? __ldg(B + (size_t)gn * ldb + gk) : __ldg(B + (size_t)gk * ldb + gn);
            Bs[k][n] = v;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < GB_K; ++k) {
            float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            float4 a1 = *reinterpret_cast<const float4*>(&As[k][64 + ty * 4]);
            float4 b0 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
            float4 b1 = *reinterpret_cast<const float4*>(&Bs[k][64 + tx * 4]);
            float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        int gm = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            int gn = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
            if (gn >= N) continue;
            float v = alpha * acc[i][j];
            float* c = C + (size_t)gm * ldc + gn;
            if (atomic_out) {
                atomicAdd(c, v);
                continue;
            }
            if (bias != nullptr) v += __ldg(bias + gn);
            if (beta != 0.f) v += beta * (*c);
            *c = v;
        }
    }
}

// returns 0 / error code like the C ABI functions
// accumulate = true: C += alpha * op(A) op(B) with split-K over the whole chip (C must hold the running sum)
inline int gemm_f32(bool ta, bool tb, int M, int N, int K, float alpha, const float* A, long lda, const float* B, long ldb,
                    float beta, float* C, long ldc, const float* bias, cudaStream_t stream, bool accumulate = false,
                    const int* kdev = nullptr, const int* mdev = nullptr) {
    if (M <= 0 || N <= 0) return 0;
    if (accumulate && K <= 0) return 0;   // adds nothing (a non-accumulating K = 0 still writes bias or zeros below)
    // tensor-core path (3xTF32, csrc/gemm_tf32x3.cuh) whenever TMA can read the operands; SNB200_GEMM=simt forces the CUDA-core kernel
    {
        const char* e = getenv("SNB200_GEMM");
        const bool force_simt = e != nullptr && e[0] == 's';
        if (!force_simt && K > 0 && (beta == 0.f || accumulate) && t3::t3_eligible(A, lda, B, ldb) && (!accumulate || beta == 1.f) &&
            (accumulate || K <= 4096)) {   // a long non-split K would outgrow the four accumulators' error bound
            int ksplit = 1;
            if (accumulate) {
                const int tiles = ceil_div(N, 128) * ceil_div(M, 128);
                const int maxsplit = ceil_div(K, 256);
                int minsplit = ceil_div(K, 2048);          // at most 2048 of K per CTA (4 accumulators x 512): bounds the truncation error
                if (minsplit < 1) minsplit = 1;
                // among the admissible splits the one with the fewest (waves of CTAs) x (K per CTA + the cost of one accumulating epilogue,
                // charged as 128 of K): at one CTA per SM a grid of 3.46 waves costs four (C4-H's weight gradient: 128 tiles x 4 = 512 CTAs)
                long best = -1;
                for (int cand = minsplit; cand <= maxsplit && cand <= minsplit + 24; ++cand) {
                    const long waves = ceil_div(tiles * cand, 148);
                    const long cost = waves * (round_up(ceil_div(K, cand), 32) + 128);
                    if (best < 0 || cost < best) { best = cost; ksplit = cand; }
                }
                if (ksplit < minsplit) ksplit = minsplit;
            }
            // op(A) = A^T (ta) means A is stored [K][M] (MN-major); op(B) = B (!tb) means B is stored [K][N] (MN-major)
            if (!ta && tb) return t3::gemm_tf32x3_launch<false, false>(M, N, K, alpha, A, lda, B, ldb, C, ldc, bias, ksplit, accumulate, stream, kdev, mdev);
            if (!ta && !tb) return t3::gemm_tf32x3_launch<false, true>(M, N, K, alpha, A, lda, B, ldb, C, ldc, bias, ksplit, accumulate, stream, kdev, mdev);
            if (ta && tb) return t3::gemm_tf32x3_launch<true, false>(M, N, K, alpha, A, lda, B, ldb, C, ldc, bias, ksplit, accumulate, stream, kdev, mdev);
            return t3::gemm_tf32x3_launch<true, true>(M, N, K, alpha, A, lda, B, ldb, C, ldc, bias, ksplit, accumulate, stream, kdev, mdev);
        }
    }
    SN_CHECK_ARG(kdev == nullptr && mdev == nullptr, "gemm_f32: device-side extents need the tensor-core path (16-byte aligned operands, "
                 "row pitches multiples of 4, K <= 4096 or an accumulating epilogue)");
    dim3 grid(ceil_div(N, GB_N), ceil_div(M, GB_M), 1);
    int kslice = K > 0 ? K : 1;
    if (accumulate) {
        int tiles = grid.x * grid.y;
        int want = ceil_div(2 * 148, tiles);                   // ~2 waves of CTAs
        int maxsplit = ceil_div(K, 4 * GB_K);                  // keep >= 64 k per slice
        int ks = want < maxsplit ? want : maxsplit;
        if (ks < 2) ks = 2;                                    // atomic epilogue implements the "+="
        kslice = round_up(ceil_div(K, ks), GB_K);
        grid.z = ceil_div(K, kslice);
        if (grid.z < 2) { grid.z = 2; }
    }
    snb::timing_begin("gemm_f32_kernel", stream);
    if (!ta && !tb) gemm_f32_kernel<false, false><<<grid, G_THREADS, 0, stream>>>(M, N, K, kslice, alpha, A, lda, B, ldb, beta, C, ldc, bias);
    else if (!ta && tb) gemm_f32_kernel<false, true><<<grid, G_THREADS, 0, stream>>>(M, N, K, kslice, alpha, A, lda, B, ldb, beta, C, ldc, bias);
    else if (ta && !tb) gemm_f32_kernel<true, false><<<grid, G_THREADS, 0, stream>>>(M, N, K, kslice, alpha, A, lda, B, ldb, beta, C, ldc, bias);
    else gemm_f32_kernel<true, true><<<grid, G_THREADS, 0, stream>>>(M, N, K, kslice, alpha, A, lda, B, ldb, beta, C, ldc, bias);
    snb::timing_end(stream);
    SN_CHECK_LAUNCH("gemm_f32_kernel");
    return 0;
}

}  // namespace snb
