// bf16 batch GEMMs of the layers that multiply their weight out into a dense matrix (PSM dense-product path, H-matrix dense-block
// path, LDR, Toeplitz-like), for bfloat16 features.  W itself is still built in fp32 from the fp32 (LDR: fp64) parameters by the
// layer's own kernels and its dense gradient is projected back by them; only the products with the batch change:
//
//   cast     :  W (fp32) -> W bf16 and / or W^T bf16      one pass, 32x32 tiles through shared memory
//   apply    :  y   = x W^T + b      (B x in)(out x in)^T      tcgen05, K-major operands, bias + bf16 store in the epilogue
//   dW       :  dW += gy^T x         (out x B)(B x in)         tcgen05, MN-major operands read in their natural [sample][feature]
//                                                              layout, split-K over the batch, fp32 reductions
//   grad_x   :  gx  = gy W           (B x out)(in x out)^T     tcgen05 on the bf16 W^T, bf16 store
//   db       += colsum(gy)
//
// MN-major operands are fetched in 64-element boxes along M / N; TMA fills the part of a box past M or N with zeros, so any M and N
// work (the low-rank path already reads M = out_dim = 1000 this way; its rank % 64 guard only concerns the rank-wide operands).
// Every operand needs a 16-byte aligned base and a row pitch that is a multiple of 8 elements (make_map_bf16 checks it).
#include "bf16_ops.cuh"
#include "gemm_tc.cuh"

namespace {

using bf16 = __nv_bfloat16;

// Mb[r][c] = M[r][c], Mtb[c][r] = M[r][c] (either may be null); pad columns of both (c >= cols of Mb, r >= rows of Mtb) are zeroed.
// The grid covers max(rows, ldmtb) x max(cols, ldmb).
__global__ void dense_cast_bf16_kernel(const float* __restrict__ M, int rows, int cols, bf16* __restrict__ Mb, long ldmb, bf16* __restrict__ Mtb,
                                       long ldmtb) {
    __shared__ bf16 tile[32][33];
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int r = r0 + i, c = c0 + threadIdx.x;
        const bf16 v = __float2bfloat16((r < rows && c < cols) ? M[(size_t)r * cols + c] : 0.f);
        tile[i][threadIdx.x] = v;
        if (Mb != nullptr && r < rows && c < ldmb) Mb[(size_t)r * ldmb + c] = v;
    }
    if (Mtb == nullptr) return;
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int c = c0 + i, r = r0 + threadIdx.x;
        if (c < cols && r < ldmtb) Mtb[(size_t)c * ldmtb + r] = tile[threadIdx.x][i];
    }
}

}  // namespace

extern "C" {

int sn_dense_cast_bf16(const float* M, int rows, int cols, void* Mb, int64_t ldmb, void* Mtb, int64_t ldmtb, sn_stream_t stream) {
    SN_CHECK_ARG(M && (Mb || Mtb), "dense_cast_bf16: NULL buffer");
    SN_CHECK_ARG(rows >= 0 && cols >= 0 && (!Mb || ldmb >= cols) && (!Mtb || ldmtb >= rows), "dense_cast_bf16: bad shape");
    if (rows == 0 || cols == 0) return 0;
    const long gr = Mtb ? (ldmtb > rows ? ldmtb : rows) : rows;
    const long gc = Mb ? (ldmb > cols ? ldmb : cols) : cols;
    dim3 grid((unsigned)((gc + 31) / 32), (unsigned)((gr + 31) / 32)), block(32, 8);
    cudaStream_t st = snb::as_stream(stream);
    SN_LAUNCH("dense_cast_bf16_kernel", st, dense_cast_bf16_kernel<<<grid, block, 0, st>>>(M, rows, cols, (bf16*)Mb, (long)ldmb, (bf16*)Mtb, (long)ldmtb));
    return 0;
}

int sn_dense_apply_bf16(const void* Wb, int64_t ldwb, int n_out, int n_in, const void* x, int64_t ldx, void* y, int64_t ldy, const float* bias,
                        int64_t B, sn_stream_t stream) {
    if (B <= 0) return 0;
    SN_CHECK_ARG(Wb && x && y, "dense_apply_bf16: NULL buffer");
    using namespace snb::tc;
    return gemm_bf16_tc<128, STORE_BF16>((int)B, n_out, n_in, x, ldx, Wb, ldwb, y, ldy, bias, 1.f, 1, snb::as_stream(stream));
}

int sn_dense_weight_grad_bf16(const void* x, int64_t ldx, const void* gy, int64_t ldgy, float* dW, int64_t lddw, int n_out, int n_in,
                              float* grad_bias, int64_t B, sn_stream_t stream) {
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && gy && dW, "dense_weight_grad_bf16: NULL buffer");
    cudaStream_t st = snb::as_stream(stream);
    if (grad_bias)
        if (int rc = colsum_bf16((const bf16*)gy, ldgy, B, n_out, grad_bias, st)) return rc;
    using namespace snb::tc;
    const int tiles = snb::ceil_div(n_out, 128) * snb::ceil_div(n_in, 128);
    return gemm_bf16_tc<128, ATOMIC_F32, true>(n_out, n_in, (int)B, gy, ldgy, x, ldx, dW, lddw, nullptr, 1.f, split_for(tiles, B), st);
}

int sn_dense_input_grad_bf16(const void* Wtb, int64_t ldwtb, int n_out, int n_in, const void* gy, int64_t ldgy, void* gx, int64_t ldgx, int64_t B,
                             sn_stream_t stream) {
    if (B <= 0) return 0;
    SN_CHECK_ARG(Wtb && gy && gx, "dense_input_grad_bf16: NULL buffer");
    using namespace snb::tc;
    return gemm_bf16_tc<128, STORE_BF16>((int)B, n_in, n_out, gy, ldgy, Wtb, ldwtb, gx, ldgx, nullptr, 1.f, 1, snb::as_stream(stream));
}

}  // extern "C"
