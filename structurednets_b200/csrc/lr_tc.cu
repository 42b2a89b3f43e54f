// Low-rank layer, bf16 tensor-core path (BASELINE config C2):  y = (x R^T) L^T + b  with bf16 operands, fp32
// accumulation in TMEM and fp32 master parameters / gradients.  Replaces LRLayer.forward (reference
// layers/lr_layer.py:38-46) and its autograd backward for bfloat16 features.
//
//   forward :  h  = x R^T            (B x in)(r x in)^T      tcgen05, K-major operands, bf16 out (kept for backward)
//              y  = h L^T + b        (B x r)(out x r)^T      tcgen05, bf16 out
//   backward:  gh = gy L             (B x out)(r x out)^T    tcgen05 on the pre-transposed L
//              dL += gy^T h          (out x B)(r x B)^T      tcgen05 on transposed copies, split-K over the batch, fp32 atomics
//              dR += gh^T x          (r x B)(in x B)^T       same
//              db += colsum(gy)
// The batch-reduction GEMMs run on bf16 transposes made by a tiled transpose kernel (ranks that are not a multiple of 64);
// otherwise the activations are consumed in their natural [sample][feature] layout through MN-major UMMA descriptors.
#include <stdlib.h>
#include "bf16_ops.cuh"
#include "gemm_tc.cuh"

namespace {

using bf16 = __nv_bfloat16;

// fp32 parameters -> bf16 copies: L (out x r), L^T (r x out), R (r x in)
__global__ void lr_cast_params_kernel(const float* __restrict__ left, const float* __restrict__ right, bf16* __restrict__ Lb, bf16* __restrict__ Ltb,
                                      bf16* __restrict__ Rb, int out_dim, int rank, int in_dim, int ldlt) {
    const size_t nl = (size_t)out_dim * rank, nr = (size_t)rank * in_dim;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < nl + nr; e += (size_t)gridDim.x * blockDim.x) {
        if (e < nl) {
            const int o = (int)(e / rank), k = (int)(e - (size_t)o * rank);
            const bf16 v = __float2bfloat16(left[e]);
            Lb[e] = v;
            Ltb[(size_t)k * ldlt + o] = v;
        } else {
            Rb[e - nl] = __float2bfloat16(right[e - nl]);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Fused forward for rank 128:  y = (x R^T) L^T + b  per 128-sample tile in ONE kernel.  h = x R^T accumulates in TMEM (128 columns),
// the epilogue warps turn it into bf16, keep a copy for the backward and write it to shared memory as the K-major A operand of the
// second product, whose 128-column output tiles alternate between two more TMEM accumulators: h never round-trips through HBM and
// the layer is one launch instead of two.
//   warp 0: TMA producer (x + R tiles, then L tiles) | warp 1: TMEM alloc + MMA issuer | warps 2-5: epilogue (thread = sample)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr));
}
constexpr int LF_THREADS = 192;
constexpr int LF_STAGES = 5;
constexpr int LF_TILE = 128 * 128;                    // 128 rows x 64 bf16 = 16 KB (the A tile of the 64-sample variant uses half of it)
constexpr int LF_STAGE = 2 * LF_TILE;                 // A tile | B tile
constexpr int LF_MAX_OUT = 4096;                      // bias staged in shared memory
constexpr size_t LF_SMEM = (size_t)LF_STAGES * LF_STAGE + 2 * LF_TILE + 1024 + 256 + LF_MAX_OUT * 4;

// BM = samples per CTA: 128 (UMMA M = 128, thread = TMEM lane = sample) or 64 (UMMA M = 64: rows 16 q .. 16 q + 15 of the tile live in
// the first 16 lanes of sub-partition q) -- at B = 8192 the 128-sample tiles fill only 64 of the 148 SMs and every CTA is bound by its
// own share of the HBM bandwidth; 64-sample tiles double the CTAs in flight.
template <int BM>
__global__ void __launch_bounds__(LF_THREADS, 1)
lr_tc_fwd_fused_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_r, const __grid_constant__ CUtensorMap map_l,
                       const float* __restrict__ bias, bf16* __restrict__ hidden, bf16* __restrict__ y, long ldy, long B, int in_dim, int out_dim) {
    using namespace snb::tc;
    extern __shared__ uint8_t lf_smem_raw[];
    uint8_t* smem = lf_smem_raw + ((1024u - (smem_u32(lf_smem_raw) & 1023u)) & 1023u);
    uint8_t* htile = smem + LF_STAGES * LF_STAGE;     // 2 k-blocks of [128 rows][64 bf16], SWIZZLE_128B layout written by hand
    uint64_t* full = reinterpret_cast<uint64_t*>(htile + 2 * LF_TILE);
    uint64_t* empty = full + LF_STAGES;
    uint64_t* h_full = empty + LF_STAGES;
    uint64_t* h_ready = h_full + 1;
    uint64_t* y_full = h_ready + 1;      // [2]
    uint64_t* y_empty = y_full + 2;      // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(y_empty + 2);
    float* sbias = reinterpret_cast<float*>(htile + 2 * LF_TILE + 256);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * BM;
    constexpr uint32_t A_BYTES = BM * 128;            // BM rows x 64 bf16
    const int nkb = (in_dim + 63) / 64;
    const int ntile = (out_dim + 127) / 128;
    for (int i = threadIdx.x; i < ntile * 128; i += LF_THREADS) sbias[i] = (bias != nullptr && i < out_dim) ? __ldg(bias + i) : 0.f;

    if (threadIdx.x == 0) {
        for (int s = 0; s < LF_STAGES; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        mbar_init(h_full, 1); mbar_init(h_ready, 128);
        for (int b = 0; b < 2; ++b) { mbar_init(y_full + b, 1); mbar_init(y_empty + b, 128); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (elect_one()) {
            int it = 0;
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int s = it % LF_STAGES, round = it / LF_STAGES;
                if (round > 0) mbar_wait(empty + s, (round - 1) & 1);
                uint8_t* st = smem + s * LF_STAGE;
                mbar_expect_tx(full + s, A_BYTES + LF_TILE);
                tma_load_2d(st, &map_x, kb * 64, m0, full + s);
                tma_load_2d(st + LF_TILE, &map_r, kb * 64, 0, full + s);
            }
            for (int nt = 0; nt < ntile; ++nt) {
                for (int k2 = 0; k2 < 2; ++k2, ++it) {
                    const int s = it % LF_STAGES, round = it / LF_STAGES;
                    if (round > 0) mbar_wait(empty + s, (round - 1) & 1);
                    uint8_t* st = smem + s * LF_STAGE;
                    mbar_expect_tx(full + s, LF_TILE);
                    tma_load_2d(st + LF_TILE, &map_l, k2 * 64, nt * 128, full + s);
                }
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
            constexpr uint32_t idesc = make_idesc_bf16(BM, 128, false);
            int it = 0;
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int s = it % LF_STAGES, round = it / LF_STAGES;
                mbar_wait(full + s, round & 1);
                tc_fence_after();
                uint8_t* st = smem + s * LF_STAGE;
                const uint64_t da = make_kmajor_sw128_desc(st), db = make_kmajor_sw128_desc(st + LF_TILE);
#pragma unroll
                for (int k = 0; k < 4; ++k) umma_bf16(tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
                umma_commit(empty + s);
            }
            umma_commit(h_full);
            mbar_wait(h_ready, 0);
            tc_fence_after();
            for (int nt = 0; nt < ntile; ++nt) {
                const int b = nt & 1;
                if (nt >= 2) mbar_wait(y_empty + b, ((nt >> 1) - 1) & 1);
                tc_fence_after();
                const uint32_t acc = tmem + 128 + b * 128;
                for (int k2 = 0; k2 < 2; ++k2, ++it) {
                    const int s = it % LF_STAGES, round = it / LF_STAGES;
                    mbar_wait(full + s, round & 1);
                    tc_fence_after();
                    const uint64_t da = make_kmajor_sw128_desc(htile + k2 * LF_TILE);
                    const uint64_t db = make_kmajor_sw128_desc(smem + s * LF_STAGE + LF_TILE);
#pragma unroll
                    for (int k = 0; k < 4; ++k) umma_bf16(acc, da + 2 * k, db + 2 * k, idesc, (k2 | k) ? 1u : 0u);
                    umma_commit(empty + s);
                }
                umma_commit(y_full + b);
            }
        }
    } else {
        const int q = warp & 3;
        const bool has_row = BM == 128 || lane < 16;  // M = 64: 16 rows per sub-partition, lanes 16..31 hold nothing
        const int r = BM == 128 ? q * 32 + lane : q * 16 + (lane & 15);   // row of the tile
        const long row = has_row ? (long)m0 + r : B;  // lanes without a row never store
        const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
        mbar_wait(h_full, 0);
        tc_fence_after();
#pragma unroll 1
        for (int c0 = 0; c0 < 128; c0 += 16) {
            uint32_t v[16];
            tmem_ld16(lane_base + c0, v);
            uint32_t pk[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                __nv_bfloat162 h2 = __floats2bfloat162_rn(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
                pk[j] = *reinterpret_cast<uint32_t*>(&h2);
            }
            const uint4 lo4 = make_uint4(pk[0], pk[1], pk[2], pk[3]), hi4 = make_uint4(pk[4], pk[5], pk[6], pk[7]);
            if (row < B) {
                uint4* hp = reinterpret_cast<uint4*>(hidden + (size_t)row * 128 + c0);
                hp[0] = lo4;
                hp[1] = hi4;
            }
            if (has_row) {
                uint8_t* trow = htile + (c0 >> 6) * LF_TILE + r * 128;
                const int ch = (c0 & 63) >> 3;        // 16-byte chunk index of the first 8 columns within the 128-byte row
                *reinterpret_cast<uint4*>(trow + (((ch) ^ (r & 7)) << 4)) = lo4;
                *reinterpret_cast<uint4*>(trow + (((ch + 1) ^ (r & 7)) << 4)) = hi4;
            }
        }
        tc_fence_before();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_arrive(h_ready);
        for (int nt = 0; nt < ntile; ++nt) {
            const int b = nt & 1;
            mbar_wait(y_full + b, (nt >> 1) & 1);
            tc_fence_after();
            const uint32_t acc = lane_base + 128 + b * 128;
#pragma unroll 1
            for (int c0 = 0; c0 < 128; c0 += 32) {
                uint32_t v[32];
                tmem_ld16_nowait(acc + c0, reinterpret_cast<uint32_t(&)[16]>(v[0]));
                tmem_ld16_nowait(acc + c0 + 16, reinterpret_cast<uint32_t(&)[16]>(v[16]));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                const int nbase = nt * 128 + c0;
                if (row < B && nbase < out_dim) {
                    const float* bs = sbias + nbase;
                    bf16* d = y + (size_t)row * ldy + nbase;
                    if (nbase + 32 <= out_dim && ((reinterpret_cast<uintptr_t>(d) & 15) == 0)) {
                        uint32_t pk[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            __nv_bfloat162 h2 = __floats2bfloat162_rn(__uint_as_float(v[2 * j]) + bs[2 * j], __uint_as_float(v[2 * j + 1]) + bs[2 * j + 1]);
                            pk[j] = *reinterpret_cast<uint32_t*>(&h2);
                        }
#pragma unroll
                        for (int j = 0; j < 4; ++j) reinterpret_cast<uint4*>(d)[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (nbase + j < out_dim) d[j] = __float2bfloat16(__uint_as_float(v[j]) + bs[j]);
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(y_empty + b);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
    }
}

// (SideStream / side_stream(): common.cuh)  The bias gradient and dL run next to gh -> dR on a second stream.
using snb::SideStream;
using snb::side_stream;

}  // namespace

extern "C" {

// bf16 copies of the parameters; lt_ld = row pitch (elements) of left_t_bf16 (>= out_dim, multiple of 8)
int sn_lr_tc_cast_params(const float* left, const float* right, void* left_bf16, void* left_t_bf16, int64_t lt_ld, void* right_bf16,
                         int in_dim, int out_dim, int rank, sn_stream_t stream) {
    SN_CHECK_ARG(left && right && left_bf16 && left_t_bf16 && right_bf16, "lr_tc_cast_params: NULL buffer");
    SN_LAUNCH("lr_cast_params_kernel", snb::as_stream(stream), lr_cast_params_kernel<<<296, 256, 0, snb::as_stream(stream)>>>(left, right, (bf16*)left_bf16, (bf16*)left_t_bf16, (bf16*)right_bf16, out_dim, rank,
                                                                 in_dim, (int)lt_ld));
    return 0;
}

// x (B x in) bf16, hidden (B x rank) bf16 [written], y (B x out) bf16 [written]; all row pitches multiples of 8 elements
int sn_lr_tc_forward(const void* x, int64_t ldx, const void* left_bf16, const void* right_bf16, const float* bias, void* hidden, void* y,
                     int64_t ldy, int64_t B, int in_dim, int out_dim, int rank, sn_stream_t stream) {
    SN_CHECK_ARG(left_bf16 && right_bf16, "lr_tc_forward: NULL buffer");
    SN_CHECK_ARG(rank % 8 == 0 && rank >= 8, "lr_tc_forward: the tensor-core path needs rank %% 8 == 0 (got %d)", rank);
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && hidden && y, "lr_tc_forward: NULL buffer");
    cudaStream_t st = snb::as_stream(stream);
    using namespace snb::tc;
    {
        const char* e = getenv("SNB200_LR_FUSED");
        const bool allow = !(e != nullptr && e[0] == '0');
        if (allow && rank == 128 && in_dim % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0 && out_dim <= LF_MAX_OUT - 128) {
            const char* e64 = getenv("SNB200_LR_BM");
            const bool bm64 = e64 != nullptr ? (e64[0] == '6') : ((B + 127) / 128 < 120);    // 128-sample tiles would leave SMs idle
            CUtensorMap mx, mr, ml;
            if (int rc = make_map_bf16(&mx, x, (uint64_t)B, (uint64_t)in_dim, (uint64_t)ldx, bm64 ? 64 : 128)) return rc;
            if (int rc = make_map_bf16(&mr, right_bf16, (uint64_t)rank, (uint64_t)in_dim, (uint64_t)in_dim, 128)) return rc;
            if (int rc = make_map_bf16(&ml, left_bf16, (uint64_t)out_dim, (uint64_t)rank, (uint64_t)rank, 128)) return rc;
            if (bm64) {
                SN_SET_MAX_SMEM((int)LF_SMEM, lr_tc_fwd_fused_kernel<64>);
                SN_LAUNCH("lr_tc_fwd_fused_kernel", st, lr_tc_fwd_fused_kernel<64><<<(unsigned)((B + 63) / 64), LF_THREADS, LF_SMEM, st>>>(mx, mr, ml, bias, (bf16*)hidden, (bf16*)y, (long)ldy, (long)B, in_dim, out_dim));
            } else {
                SN_SET_MAX_SMEM((int)LF_SMEM, lr_tc_fwd_fused_kernel<128>);
                SN_LAUNCH("lr_tc_fwd_fused_kernel", st, lr_tc_fwd_fused_kernel<128><<<(unsigned)((B + 127) / 128), LF_THREADS, LF_SMEM, st>>>(mx, mr, ml, bias, (bf16*)hidden, (bf16*)y, (long)ldy, (long)B, in_dim, out_dim));
            }
            return 0;
        }
    }
    if (int rc = gemm_bf16_tc<64, STORE_BF16>((int)B, rank, in_dim, x, ldx, right_bf16, in_dim, hidden, rank, nullptr, 1.f, 1, st)) return rc;
    return gemm_bf16_tc<128, STORE_BF16>((int)B, out_dim, rank, hidden, rank, left_bf16, rank, y, ldy, bias, 1.f, 1, st);
}

// grad_left (out x rank), grad_right (rank x in), grad_bias (out) are fp32 and accumulated.  Scratch (bf16): ghid (B x rank),
// gyt (out x ldt) and ht (rank x ldt) when grad_left is given, ght (rank x ldt) and xt (in x ldt) when grad_right is, with ldt = B rounded
// up to a multiple of 8; right_t (in x rank) when grad_x (bf16, B x in, written) is asked for.
int sn_lr_tc_backward(const void* x, int64_t ldx, const void* grad_y, int64_t ldgy, const void* left_t_bf16, int64_t lt_ld,
                      const void* right_bf16, const void* hidden, void* ghid, void* gyt, void* ht, void* ght, void* xt, int64_t ldt,
                      void* right_t, float* grad_left, float* grad_right, float* grad_bias, void* grad_x, int64_t ldgx, int64_t B,
                      int in_dim, int out_dim, int rank, sn_stream_t stream) {
    SN_CHECK_ARG(left_t_bf16, "lr_tc_backward: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && grad_y && hidden && ghid, "lr_tc_backward: NULL buffer");
    SN_CHECK_ARG((grad_left == nullptr || (gyt && ht)) && (grad_right == nullptr || (ght && xt)), "lr_tc_backward: NULL transpose scratch");
    SN_CHECK_ARG(ldt >= B && ldt % 8 == 0, "lr_tc_backward: ldt must be B rounded up to a multiple of 8");
    SN_CHECK_ARG(grad_x == nullptr || (right_bf16 && right_t), "lr_tc_backward: grad_x needs right_bf16 and the right_t scratch");
    SN_CHECK_ARG(grad_x == nullptr || ldgx >= in_dim, "lr_tc_backward: grad_x leading dimension too small (ldgx %lld < in_dim %d)",
                 (long long)ldgx, in_dim);
    SN_CHECK_ARG(grad_x == nullptr || ldgx % 8 == 0, "lr_tc_backward: grad_x leading dimension %lld is not a multiple of 8", (long long)ldgx);
    cudaStream_t st = snb::as_stream(stream);
    using namespace snb::tc;
    // side stream: bias gradient and dL (they need grad_y and the hidden activations only); main stream: gh, then dR
    SideStream* sd = nullptr;
    {
        const char* e = getenv("SNB200_LR_SIDE_STREAM");
        if (!(e != nullptr && e[0] == '0')) sd = side_stream();
    }
    cudaStream_t s2 = st;
    if (sd != nullptr) {
        SN_CHECK_CUDA(cudaEventRecord(sd->fork, st));
        SN_CHECK_CUDA(cudaStreamWaitEvent(sd->stream, sd->fork, 0));
        s2 = sd->stream;
    }
    // gh = gy L : A = gy (B x out), B operand = L^T (rank x out), K = out
    if (int rc = gemm_bf16_tc<64, STORE_BF16>((int)B, rank, out_dim, grad_y, ldgy, left_t_bf16, lt_ld, ghid, rank, nullptr, 1.f, 1, st)) return rc;
    if (grad_x) {   // grad_x = gh R : B operand = R^T (in x rank, K-major); no split-K, so every element has one owner
        if (int rc = transpose_bf16((const bf16*)right_bf16, in_dim, (bf16*)right_t, rank, rank, in_dim, st)) return rc;
        if (int rc = gemm_bf16_tc<128, STORE_BF16>((int)B, in_dim, rank, ghid, rank, right_t, rank, grad_x, ldgx, nullptr, 1.f, 1, st)) return rc;
    }
    if (grad_bias) {
        dim3 grid(snb::ceil_div(out_dim, 256), (unsigned)((B + 63) / 64));
        SN_LAUNCH("colsum_bf16_kernel", s2, colsum_bf16_kernel<<<grid, 128, 0, s2>>>((const bf16*)grad_y, ldgy, B, out_dim, grad_bias));
    }
    const bool mn_ok = (rank % 64 == 0);   // MN-major operands are fetched in 64-element blocks along M / N
    {
        cudaStream_t st_main = st;
        cudaStream_t st = s2;      // the dL block below runs on the side stream
        (void)st_main;
    if (grad_left) {   // dL += gy^T h
        const int tiles = snb::ceil_div(out_dim, 128) * snb::ceil_div(rank, 128);
        if (mn_ok) {   // operands read in their natural [sample][feature] layout through MN-major UMMA descriptors
            if (int rc = gemm_bf16_tc<128, ATOMIC_F32, true>(out_dim, rank, (int)B, grad_y, ldgy, hidden, rank, grad_left, rank, nullptr, 1.f, split_for(tiles, B), st)) return rc;
        } else {
            if (int rc = transpose_bf16((const bf16*)grad_y, ldgy, (bf16*)gyt, ldt, B, out_dim, st)) return rc;
            if (int rc = transpose_bf16((const bf16*)hidden, rank, (bf16*)ht, ldt, B, rank, st)) return rc;
            if (int rc = gemm_bf16_tc<128, ATOMIC_F32>(out_dim, rank, (int)B, gyt, ldt, ht, ldt, grad_left, rank, nullptr, 1.f, split_for(tiles, B), st)) return rc;
        }
    }
    }
    if (grad_right) {  // dR += gh^T x
        const int tiles = snb::ceil_div(rank, 128) * snb::ceil_div(in_dim, 128);
        if (mn_ok) {
            if (int rc = gemm_bf16_tc<128, ATOMIC_F32, true>(rank, in_dim, (int)B, ghid, rank, x, ldx, grad_right, in_dim, nullptr, 1.f, split_for(tiles, B), st)) return rc;
        } else {
            if (int rc = transpose_bf16((const bf16*)ghid, rank, (bf16*)ght, ldt, B, rank, st)) return rc;
            if (int rc = transpose_bf16((const bf16*)x, ldx, (bf16*)xt, ldt, B, in_dim, st)) return rc;
            if (int rc = gemm_bf16_tc<128, ATOMIC_F32>(rank, in_dim, (int)B, ght, ldt, xt, ldt, grad_right, in_dim, nullptr, 1.f, split_for(tiles, B), st)) return rc;
        }
    }
    if (sd != nullptr) {
        SN_CHECK_CUDA(cudaEventRecord(sd->join, sd->stream));
        SN_CHECK_CUDA(cudaStreamWaitEvent(st, sd->join, 0));
    }
    return 0;
}

}  // extern "C"
