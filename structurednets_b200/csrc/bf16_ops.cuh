// bf16 helpers shared by the bf16 tensor-core paths (lr_tc.cu, dense_bf16.cu, psm.cu): the tiled transpose, the column sum
// of the bias gradient and the split-K choice of the batch-reduction GEMMs.  Anonymous namespace: every translation unit that
// includes this gets its own copy of the kernels (the library is built without relocatable device code).
#pragma once
#include <cuda_bf16.h>
#include "common.cuh"

namespace {

// dst[c][r] = src[r][c]  (bf16, 32x32 tiles through shared memory)
__global__ void transpose_bf16_kernel(const __nv_bfloat16* __restrict__ src, long lds, __nv_bfloat16* __restrict__ dst, long ldd, long rows, int cols) {
    __shared__ __nv_bfloat16 tile[32][33];
    const long r0 = (long)blockIdx.y * 32;
    const int c0 = blockIdx.x * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const long r = r0 + i;
        const int c = c0 + threadIdx.x;
        tile[i][threadIdx.x] = (r < rows && c < cols) ? src[r * lds + c] : __float2bfloat16(0.f);
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int c = c0 + i;
        const long r = r0 + threadIdx.x;
        if (c < cols && r < rows) dst[(size_t)c * ldd + r] = tile[threadIdx.x][i];
    }
}

// out[c] += sum_r M[r][c]: a thread owns a pair of columns (one 4-byte load per row, coalesced along the row), 64-row slabs
__global__ void colsum_bf16_kernel(const __nv_bfloat16* __restrict__ M, long ld, long rows, int cols, float* __restrict__ out) {
    const int c = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
    if (c >= cols) return;
    const long r0 = (long)blockIdx.y * 64;
    const long r1 = r0 + 64 < rows ? r0 + 64 : rows;
    float s0 = 0.f, s1 = 0.f;
    if (c + 1 < cols && (ld & 1) == 0 && ((reinterpret_cast<uintptr_t>(M) & 3) == 0)) {
#pragma unroll 8
        for (long r = r0; r < r1; ++r) {
            const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(M + r * ld + c);
            s0 += __bfloat162float(v.x);
            s1 += __bfloat162float(v.y);
        }
    } else {
        for (long r = r0; r < r1; ++r) {
            s0 += __bfloat162float(M[r * ld + c]);
            if (c + 1 < cols) s1 += __bfloat162float(M[r * ld + c + 1]);
        }
    }
    atomicAdd(out + c, s0);
    if (c + 1 < cols) atomicAdd(out + c + 1, s1);
}

inline int transpose_bf16(const __nv_bfloat16* src, long lds, __nv_bfloat16* dst, long ldd, long rows, int cols, cudaStream_t st) {
    dim3 grid(snb::ceil_div(cols, 32), (unsigned)((rows + 31) / 32)), block(32, 8);
    SN_LAUNCH("transpose_bf16_kernel", st, transpose_bf16_kernel<<<grid, block, 0, st>>>(src, lds, dst, ldd, rows, cols));
    return 0;
}

// grad_bias[c] += sum over the B rows of M[r][c]  (bf16 M, row pitch ld)
inline int colsum_bf16(const __nv_bfloat16* M, long ld, long B, int cols, float* grad_bias, cudaStream_t st) {
    dim3 grid(snb::ceil_div(cols, 256), (unsigned)((B + 63) / 64));
    SN_LAUNCH("colsum_bf16_kernel", st, colsum_bf16_kernel<<<grid, 128, 0, st>>>(M, ld, B, cols, grad_bias));
    return 0;
}

// split-K factor of a batch-reduction GEMM with `tiles` output tiles and K = batch: enough slices to fill the 148 SMs, at least
// 512 of K per slice
inline int split_for(int tiles, long K) {
    int want = snb::ceil_div(148, tiles > 0 ? tiles : 1);
    long maxs = (K + 511) / 512;   // at least 512 of K per slice
    if (want > maxs) want = (int)maxs;
    return want < 1 ? 1 : want;
}

}  // namespace
