// SSS layer on the tensor cores: chunked formulation of the stage recursion (reference layers/sss_layer.py:99-131)
// evaluated as 3xTF32 GEMMs on tcgen05 / TMEM / TMA, fp32-accurate (hi/lo operand split, fp32 accumulation in TMEM).
//
// A chunk j is a run of consecutive stages [k0, k1) with <= 32 outputs, <= 160 inputs and <= 16 stages.  Multiplying
// the stages of a chunk out gives dense chunk matrices (tests/sss_tc_emulator.py is the torch statement of this):
//       y_j     = T_j u_j + O_j s_j + O'_j e_{j+1}        s_j: causal state entering the chunk from below
//       s_{j+1} = R_j u_j + Phi_j s_j                      e_{j+1}: anticausal state entering it from above
//       e_j     = R'_j u_j + Phi'_j e_{j+1}
// Forward   1. sss_tc_build_kernel     params -> W_j = [T_j; R_j; R'_j] (64 x 160, hi and lo tf32 parts), SC_j = {Phi, Phi', O, O'}
//           2. sss_tc_local_gemm_kernel [yloc | r | r'] = u_j W_j^T   for every (128-sample tile, chunk): tcgen05.mma kind::tf32,
//                                       x tiles and W tiles by TMA (SWIZZLE_128B), hi/lo split of x by converter warps,
//                                       accumulators double-buffered in TMEM, persistent CTAs
//           3. sss_tc_scan_fwd_kernel  chunk-level state scans (one thread per sample), y = yloc + O s + O' e + bias;
//                                       saves the chunk-boundary states for the backward
// Backward  4. sss_tc_scan_bwd_kernel  adjoint chunk scans: lambda_j = Phi_j^T lambda_{j+1} + O_j^T gy_j, mu likewise; grad_bias
//           5. sss_tc_grad_gemm_kernel dM_j = [gy_j | lambda_{j+1} | mu_j]^T [u_j | s_j | e_{j+1}]  (K = samples, MN-major operands
//                                       straight from the natural [sample][feature] layouts), split over sample ranges
//           6. sss_tc_build_bwd_kernel chain rule through the chunk-matrix construction: dM -> dA .. dG
#include <stdlib.h>
#include <vector>
#include "common.cuh"
#include "umma.cuh"
#include "util.cuh"
#include "gemm_f32.cuh"

namespace {

using namespace snb::umma;
using snb::ceil_div;

constexpr int DS = SN_SSS_TC_DS;           // 16 padded state dimension
constexpr int PO = SN_SSS_TC_PO;           // 32 outputs per chunk
constexpr int KBW = 32;                    // input columns per k-block (128 bytes)
constexpr int KB_MAX = SN_SSS_TC_KB_MAX;   // 5 k-blocks per chunk
constexpr int LMAX = SN_SSS_TC_LMAX;       // 16 stages per chunk
constexpr int SOUT_MAX = 16;               // outputs of one stage
constexpr int WROWS = 128;                 // 64 hi rows + 64 lo rows
constexpr int WCOLS = KBW * KB_MAX;        // 160
constexpr int SCF = 2 * DS * DS + 2 * PO * DS;   // 1536 floats: Phi, Phi', O, O'
constexpr int DMC = KBW * (KB_MAX + 1);    // 192 columns of dM: u (<=160) then s (16), e (16) right after the last u block
constexpr int COLT = WCOLS + DS;           // 176 columns handled by the build kernels (inputs + unit states)
constexpr int BUILD_THREADS = 192;


__device__ __forceinline__ const sn_sss_stage& stage_of(const sn_sss_stage* stages, int n, int dir, int k) {
    return stages[dir * n + (dir == 0 ? k : n - 1 - k)];
}

// The parameters of ALL stages of a chunk are copied into shared memory once, up front (compact row-major, as in the flat parameter
// buffer; 4-byte cp.async, issued coalesced by the whole CTA): the stage recursions of the build kernels then run out of shared
// memory with broadcast LDS and no global latency between stages.  The plan carries the largest per-chunk parameter count.
constexpr int STG_IN_MAX = KBW * KB_MAX;   // 160
struct StageP {
    int ss, ys, su, yu;   // float offsets into the chunk's parameter buffer: d_out x d_in, out_dim x d_in, d_out x in_dim, out_dim x in_dim
};
__device__ __forceinline__ void cp_async4(float* dst, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// every sub-array starts on a 16-byte boundary, so full-width (16-column) rows can be read as float4
__device__ __forceinline__ int pad4(int x) { return (x + 3) & ~3; }
__device__ __forceinline__ void chunk_params_async(float* pbuf, StageP* ptrs, const sn_sss_stage* sdesc, int nst, const float* __restrict__ params, int tid,
                                                   int nthreads) {
    int off = 0;
    for (int i = 0; i < nst; ++i) {
        const sn_sss_stage& st = sdesc[i];
        const int n_ss = st.d_out * st.d_in, n_ys = st.out_dim * st.d_in, n_su = st.d_out * st.in_dim;
        const int n_yu = st.off_yu >= 0 ? st.out_dim * st.in_dim : 0;
        const int o_ss = off, o_ys = o_ss + pad4(n_ss), o_su = o_ys + pad4(n_ys), o_yu = o_su + pad4(n_su);
        if (tid == 0) ptrs[i] = StageP{o_ss, o_ys, o_su, o_yu};
        for (int e = tid; e < n_ss; e += nthreads) cp_async4(pbuf + o_ss + e, params + st.off_ss + e);
        for (int e = tid; e < n_ys; e += nthreads) cp_async4(pbuf + o_ys + e, params + st.off_ys + e);
        for (int e = tid; e < n_su; e += nthreads) cp_async4(pbuf + o_su + e, params + st.off_su + e);
        for (int e = tid; e < n_yu; e += nthreads) cp_async4(pbuf + o_yu + e, params + st.off_yu + e);
        off = o_yu + pad4(n_yu);
    }
}

__device__ __forceinline__ float dot16(const float* __restrict__ row, const float (&v)[DS]) {   // row: 16 floats, 16-byte aligned, shared memory
    // four partial sums (one per float4 lane): a single accumulator is a chain of 16 dependent FFMAs (64 cycles for 16 issue slots),
    // and the build kernels run 1.5 warps per scheduler -- nothing else hides that latency
    const float4* r4 = reinterpret_cast<const float4*>(row);
    const float4 m0 = r4[0], m1 = r4[1], m2 = r4[2], m3 = r4[3];
    float a0 = m0.x * v[0], a1 = m0.y * v[1], a2 = m0.z * v[2], a3 = m0.w * v[3];
    a0 = fmaf(m1.x, v[4], a0); a1 = fmaf(m1.y, v[5], a1); a2 = fmaf(m1.z, v[6], a2); a3 = fmaf(m1.w, v[7], a3);
    a0 = fmaf(m2.x, v[8], a0); a1 = fmaf(m2.y, v[9], a1); a2 = fmaf(m2.z, v[10], a2); a3 = fmaf(m2.w, v[11], a3);
    a0 = fmaf(m3.x, v[12], a0); a1 = fmaf(m3.y, v[13], a1); a2 = fmaf(m3.z, v[14], a2); a3 = fmaf(m3.w, v[15], a3);
    return (a0 + a1) + (a2 + a3);
}
__device__ __forceinline__ void axpy_row16(const float* __restrict__ row, float w, float (&out)[DS]) {   // out[a] += row[a] * w
    const float4* r4 = reinterpret_cast<const float4*>(row);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float4 m = r4[q];
        out[4 * q] = fmaf(m.x, w, out[4 * q]); out[4 * q + 1] = fmaf(m.y, w, out[4 * q + 1]);
        out[4 * q + 2] = fmaf(m.z, w, out[4 * q + 2]); out[4 * q + 3] = fmaf(m.w, w, out[4 * q + 3]);
    }
}

// One stage applied to one column of the chunk's "identity input": v (state entering) -> yv (the stage's outputs, if WITH_Y), v (state leaving).
// Full-width stages (state dimension 16 in and out: all but the boundary stages) take the float4 path.
template <bool WITH_Y>
__device__ __forceinline__ void stage_apply(const sn_sss_stage& st, const float* pbuf, const StageP& sp, float (&v)[DS], float (&yv)[SOUT_MAX], bool mine,
                                            int local) {
    const int d_in = st.d_in, d_out = st.d_out;
    const float* ss = pbuf + sp.ss;
    const float* ys = pbuf + sp.ys;
    const bool wide = d_in == DS;
    if (WITH_Y) {
#pragma unroll
        for (int r = 0; r < SOUT_MAX; ++r) {
            if (r >= st.out_dim) break;
            float acc = 0.f;
            if (wide) {
                acc = dot16(ys + r * DS, v);
            } else {
#pragma unroll
                for (int a = 0; a < DS; ++a)
                    if (a < d_in) acc = fmaf(ys[r * d_in + a], v[a], acc);
            }
            if (mine && st.off_yu >= 0) acc += pbuf[sp.yu + r * st.in_dim + local];
            yv[r] = acc;
        }
    }
    float nv[DS];
    if (wide && d_out == DS) {
#pragma unroll
        for (int b = 0; b < DS; ++b) nv[b] = dot16(ss + b * DS, v);
    } else {
#pragma unroll
        for (int b = 0; b < DS; ++b) nv[b] = 0.f;
#pragma unroll
        for (int b = 0; b < DS; ++b) {
            if (b >= d_out) break;
            float acc = 0.f;
#pragma unroll
            for (int a = 0; a < DS; ++a)
                if (a < d_in) acc = fmaf(ss[b * d_in + a], v[a], acc);
            nv[b] = acc;
        }
    }
    if (mine) {
#pragma unroll
        for (int b = 0; b < DS; ++b)
            if (b < d_out) nv[b] += pbuf[sp.su + b * st.in_dim + local];
    }
#pragma unroll
    for (int b = 0; b < DS; ++b) v[b] = nv[b];
}

__device__ __forceinline__ void store_hi_lo(float* W, int row, int t, float val) {
    const float hi = tf32_hi(val);
    W[row * WCOLS + t] = hi;
    W[(64 + row) * WCOLS + t] = tf32_hi(val - hi);
}

// ------------------------------------------------------------------------------------------
// 1. chunk matrices.  grid (nchunks, 2 directions); thread t < ncols: input column t of the chunk, ncols <= t < ncols+16: unit state
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BUILD_THREADS)
sss_tc_build_kernel(const sn_sss_stage* __restrict__ stages, int n, const sn_sss_tc_chunk* __restrict__ chunks, const float* __restrict__ params,
                    float* __restrict__ Wall, float* __restrict__ SCall) {
    extern __shared__ __align__(16) float build_smem[];
    __shared__ sn_sss_stage sdesc[LMAX];
    __shared__ StageP sptr[LMAX];
    const sn_sss_tc_chunk c = chunks[blockIdx.x];
    const int dir = blockIdx.y, t = threadIdx.x;
    const bool is_in = t < c.ncols;
    const int sidx = t - c.ncols;
    const bool active = is_in || sidx < DS;
    float* W = Wall + (size_t)blockIdx.x * WROWS * WCOLS;
    float* SC = SCall + (size_t)blockIdx.x * SCF;
    float* Phi = SC + dir * DS * DS;
    float* Omat = SC + 2 * DS * DS + dir * PO * DS;
    const int nst = c.k_end - c.k_begin;
    const int col = c.col0 + t;
    if (t < nst) sdesc[t] = stage_of(stages, n, dir, dir == 0 ? c.k_begin + t : c.k_end - 1 - t);
    __syncthreads();
    chunk_params_async(build_smem, sptr, sdesc, nst, params, t, BUILD_THREADS);
    cp_async_commit();
    cp_async_wait_all();
    __syncthreads();
    if (!active) return;
    float v[DS], yv[SOUT_MAX];
#pragma unroll
    for (int a = 0; a < DS; ++a) v[a] = (!is_in && a == sidx && sidx < sdesc[0].d_in) ? 1.f : 0.f;
    bool activated = false;
    for (int i = 0; i < nst; ++i) {
        const sn_sss_stage& st = sdesc[i];
        const int local = col - st.in_off;
        const bool mine = is_in && local >= 0 && local < st.in_dim;
        stage_apply<true>(st, build_smem, sptr[i], v, yv, mine, local);
        const int rbase = st.out_off - c.row0;
        const bool wr = dir == 0 ? (activated || mine) : activated;
#pragma unroll
        for (int r = 0; r < SOUT_MAX; ++r) {
            if (r >= st.out_dim) break;
            if (is_in) {
                if (wr) store_hi_lo(W, rbase + r, t, yv[r]);
            } else {
                Omat[(rbase + r) * DS + sidx] = yv[r];
            }
        }
        if (mine) activated = true;
    }
#pragma unroll
    for (int b = 0; b < DS; ++b) {
        if (is_in) store_hi_lo(W, PO + dir * DS + b, t, v[b]);
        else Phi[b * DS + sidx] = v[b];
    }
}

// ------------------------------------------------------------------------------------------
// 1'. chunk matrices, B4_LPC threads per column.  grid (nchunks, 2 directions, B4_SPLIT column groups).  The serial depth of kernel 1
//     is 16 stages x a 16 x 16 matrix-vector product per thread, and it ran 1.5 warps per scheduler: pure instruction latency.  Here
//     lane o of a group of B4_LPC lanes owns 16 / B4_LPC state components, the group all-gathers the new state with shuffles, and
//     the columns of a (chunk, direction) are spread over B4_SPLIT CTAs: 4-16x the warps, about the same number of instructions.
//     Warps whose columns are all still "not activated" (their stages come later in the sweep) skip the stage.
// ------------------------------------------------------------------------------------------
#ifndef SN_B4_LPC
#define SN_B4_LPC 8
#endif
constexpr int B4_LPC = SN_B4_LPC;                               // lanes per column: 4, 8 or 16
constexpr int B4_NC = DS / B4_LPC;                              // state components (and output rows) per lane
constexpr int B4_SPLIT = 4;
constexpr int B4_COLS = (COLT + B4_SPLIT - 1) / B4_SPLIT;      // 44 columns per CTA
constexpr int B4_LD = 52;                                       // shared-memory row pitch (floats): a multiple of 4 with LD mod 32 = 20, so the
                                                                // float4 row reads of 8 consecutive rows fall into 8 different bank groups
constexpr int B4_THREADS = B4_LPC * ((B4_COLS * B4_LPC + 31) / 32 * 32 / B4_LPC);   // whole warps
constexpr int B4_TCOLS = B4_THREADS / B4_LPC;                   // columns the thread block has lanes for (>= B4_COLS)
static_assert(B4_LPC == 4 || B4_LPC == 8 || B4_LPC == 16, "lanes per column");
static_assert(B4_TCOLS <= B4_LD && B4_COLS <= B4_TCOLS, "column group wider than the shared-memory rows");

// rows of the state matrices are read B4_NC at a time by the lanes of a column group: 4 floats of padding after every B4_NC rows put
// the lanes' 16-byte reads into different banks
__device__ __forceinline__ int ss_off(int b, int d_in) { return b * d_in + (b / B4_NC) * 4; }
__device__ __forceinline__ int ss_floats(int d_out, int d_in) { return pad4(d_out * d_in) + ((d_out + B4_NC - 1) / B4_NC) * 4; }

__device__ __forceinline__ void cp_async16(float* dst, const float* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
// n floats, 16 bytes at a time when source and count allow it (the destination always starts on a 16-byte boundary)
__device__ __forceinline__ void copy_async(float* dst, const float* __restrict__ src, int nfl, int tid, int nthreads) {
    if (((reinterpret_cast<uintptr_t>(src) & 15) == 0) && (nfl & 3) == 0) {
        for (int e = tid; e < (nfl >> 2); e += nthreads) cp_async16(dst + 4 * e, src + 4 * e);
    } else {
        for (int e = tid; e < nfl; e += nthreads) cp_async4(dst + e, src + e);
    }
}
__device__ __forceinline__ void chunk_params_async_q(float* pbuf, StageP* ptrs, const sn_sss_stage* sdesc, int nst, const float* __restrict__ params, int tid,
                                                     int nthreads) {
    int off = 0;
    for (int i = 0; i < nst; ++i) {
        const sn_sss_stage& st = sdesc[i];
        const int n_ys = st.out_dim * st.d_in, n_su = st.d_out * st.in_dim;
        const int n_yu = st.off_yu >= 0 ? st.out_dim * st.in_dim : 0;
        const int o_ss = off, o_ys = o_ss + ss_floats(st.d_out, st.d_in), o_su = o_ys + pad4(n_ys), o_yu = o_su + pad4(n_su);
        if (tid == 0) ptrs[i] = StageP{o_ss, o_ys, o_su, o_yu};
        // state matrix: groups of B4_NC rows are contiguous in the source and in the padded destination
        const int grp = B4_NC * st.d_in;
        if (grp > 0) {
            const int ngrp = st.d_out / B4_NC, rest = (st.d_out - ngrp * B4_NC) * st.d_in;
            if ((grp & 3) == 0 && ((reinterpret_cast<uintptr_t>(params + st.off_ss) & 15) == 0)) {
                const int per = grp >> 2;
                for (int e = tid; e < ngrp * per; e += nthreads) {
                    const int g = e / per, w = e - g * per;
                    cp_async16(pbuf + o_ss + g * (grp + 4) + 4 * w, params + st.off_ss + g * grp + 4 * w);
                }
            } else {
                for (int e = tid; e < ngrp * grp; e += nthreads) {
                    const int g = e / grp;
                    cp_async4(pbuf + o_ss + e + 4 * g, params + st.off_ss + e);
                }
            }
            for (int e = tid; e < rest; e += nthreads) cp_async4(pbuf + o_ss + ngrp * (grp + 4) + e, params + st.off_ss + ngrp * grp + e);
        }
        copy_async(pbuf + o_ys, params + st.off_ys, n_ys, tid, nthreads);
        copy_async(pbuf + o_su, params + st.off_su, n_su, tid, nthreads);
        copy_async(pbuf + o_yu, params + st.off_yu, n_yu, tid, nthreads);
        off = o_yu + pad4(n_yu);
    }
}

// all-gather inside a column group: v[B4_NC k + j] = piece j of lane k of the group
__device__ __forceinline__ void group_allgather(const float (&mine)[B4_NC], float (&v)[DS], int lane) {
    const int gb = lane & ~(B4_LPC - 1);
#pragma unroll
    for (int k = 0; k < B4_LPC; ++k)
#pragma unroll
        for (int j = 0; j < B4_NC; ++j) v[B4_NC * k + j] = __shfl_sync(0xffffffffu, mine[j], gb + k);
}

// One stage for one column: lane o of the group computes the outputs r = o, o + LPC, .. (WITH_Y) and the state components
// B4_NC o .. B4_NC o + B4_NC - 1, which it also keeps in `own` (addressable without a run-time register index).
template <bool WITH_Y>
__device__ __forceinline__ void stage_apply_q(const sn_sss_stage& st, const float* pbuf, const StageP& sp, float (&v)[DS], float (&own)[B4_NC], float (&yv)[B4_NC],
                                              bool mine, int local, int o, int lane) {
    const int d_in = st.d_in, d_out = st.d_out;
    const float* ys = pbuf + sp.ys;
    const bool wide = d_in == DS;
    if (WITH_Y) {
#pragma unroll
        for (int j = 0; j < B4_NC; ++j) {
            const int r = o + B4_LPC * j;
            float acc = 0.f;
            if (r < st.out_dim) {
                if (wide) {
                    acc = dot16(ys + r * DS, v);
                } else {
#pragma unroll
                    for (int a = 0; a < DS; ++a)
                        if (a < d_in) acc = fmaf(ys[r * d_in + a], v[a], acc);
                }
                if (mine && st.off_yu >= 0) acc += pbuf[sp.yu + r * st.in_dim + local];
            }
            yv[j] = acc;
        }
    }
#pragma unroll
    for (int j = 0; j < B4_NC; ++j) {
        const int b = B4_NC * o + j;
        float acc = 0.f;
        if (b < d_out) {
            const float* row = pbuf + sp.ss + ss_off(b, d_in);
            if (wide) {
                acc = dot16(row, v);
            } else {
#pragma unroll
                for (int a = 0; a < DS; ++a)
                    if (a < d_in) acc = fmaf(row[a], v[a], acc);
            }
            if (mine) acc += pbuf[sp.su + b * st.in_dim + local];
        }
        own[j] = acc;
    }
    group_allgather(own, v, lane);
}

__global__ void __launch_bounds__(B4_THREADS)
sss_tc_build4_kernel(const sn_sss_stage* __restrict__ stages, int n, const sn_sss_tc_chunk* __restrict__ chunks, const float* __restrict__ params,
                     float* __restrict__ Wall, float* __restrict__ SCall) {
    extern __shared__ __align__(16) float build_smem[];
    __shared__ sn_sss_stage sdesc[LMAX];
    __shared__ StageP sptr[LMAX];
    const sn_sss_tc_chunk c = chunks[blockIdx.x];
    const int dir = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const int lc = tid / B4_LPC, o = tid % B4_LPC;
    const int t = blockIdx.z * B4_COLS + lc;                 // column of the chunk: inputs first, then the 16 unit states
    const bool active = lc < B4_COLS && t < c.ncols + DS;
    const bool is_in = t < c.ncols;
    const int sidx = t - c.ncols;
    float* W = Wall + (size_t)blockIdx.x * WROWS * WCOLS;
    float* SC = SCall + (size_t)blockIdx.x * SCF;
    float* Phi = SC + dir * DS * DS;
    float* Omat = SC + 2 * DS * DS + dir * PO * DS;
    const int nst = c.k_end - c.k_begin;
    const int col = c.col0 + t;
    if (blockIdx.z * B4_COLS >= c.ncols + DS) return;        // no column of this group exists (uniform over the CTA)
    if (tid < nst) sdesc[tid] = stage_of(stages, n, dir, dir == 0 ? c.k_begin + tid : c.k_end - 1 - tid);
    __syncthreads();
    chunk_params_async_q(build_smem, sptr, sdesc, nst, params, tid, B4_THREADS);
    cp_async_commit();
    cp_async_wait_all();
    __syncthreads();
    float v[DS], own[B4_NC], yv[B4_NC];
#pragma unroll
    for (int a = 0; a < DS; ++a) v[a] = (active && !is_in && a == sidx && sidx < sdesc[0].d_in) ? 1.f : 0.f;
#pragma unroll
    for (int j = 0; j < B4_NC; ++j) own[j] = (active && !is_in && B4_NC * o + j == sidx && sidx < sdesc[0].d_in) ? 1.f : 0.f;
    bool activated = false;
    for (int i = 0; i < nst; ++i) {
        const sn_sss_stage& st = sdesc[i];
        const int local = col - st.in_off;
        const bool mine = active && is_in && local >= 0 && local < st.in_dim;
        const bool live = active && (!is_in || activated || mine);
        if (!__any_sync(0xffffffffu, live)) continue;        // every column of the warp still waits for its stage
        stage_apply_q<true>(st, build_smem, sptr[i], v, own, yv, mine, local, o, lane);
        const int rbase = st.out_off - c.row0;
        const bool wr = dir == 0 ? (activated || mine) : activated;
        if (active) {
#pragma unroll
            for (int j = 0; j < B4_NC; ++j) {
                const int r = o + B4_LPC * j;
                if (r >= st.out_dim) break;
                if (is_in) {
                    if (wr) store_hi_lo(W, rbase + r, t, yv[j]);
                } else {
                    Omat[(rbase + r) * DS + sidx] = yv[j];
                }
            }
        }
        if (mine) activated = true;
    }
    if (active) {
#pragma unroll
        for (int j = 0; j < B4_NC; ++j) {
            const int b = B4_NC * o + j;
            if (is_in) store_hi_lo(W, PO + dir * DS + b, t, own[j]);
            else Phi[b * DS + sidx] = own[j];
        }
    }
}

// ------------------------------------------------------------------------------------------
// 1''. chunk matrices on the warp-level tensor-core path (mma.sync m16n8k8 tf32, 3xTF32).  The SIMT build kernels above are
//     instruction-bound: 8.4 M warp instructions of which 9 % are FFMAs (ncu: IMAD / ISETP / LDS / BRA dominate), whatever the
//     number of lanes per column.  Here a warp owns a tile of 16 columns of the chunk's "identity input" and keeps their states as
//     the D fragment of V (16 columns x 16 states); one stage is  V <- V A_i^T (+ B_i columns),  Y = V C_i^T (+ D_i)  -- four + two
//     MMAs (x3 for the hi/lo split) whose A operand IS the previous D fragment: with the K index permuted (logical k = t <-> state
//     2t, k = t + 4 <-> state 2t + 1 inside each group of 8) the accumulator registers of one product are the operand registers
//     of the next, no shuffle and no shared-memory round trip.  The B operands (A_i, C_i) come from shared
//     memory (raw fp32, split in registers).  ~110 instructions per stage and 16 columns instead of
//     ~300 per 8 columns.  grid (nchunks, 2 directions, BM_SPLIT); tiles 0..9 = input columns, tile 10 = the 16 unit states.
// ------------------------------------------------------------------------------------------
constexpr int BM_TILES = COLT / 16;                                  // 11
constexpr int BM_SPLIT = 2;
constexpr int BM_WARPS = (BM_TILES + BM_SPLIT - 1) / BM_SPLIT;       // 6 warps per CTA
constexpr int BM_THREADS = BM_WARPS * 32;
static_assert(COLT % 16 == 0 && WCOLS % 16 == 0, "input columns and unit states must fall into separate 16-column tiles");

// The chunk's parameters are staged RAW by cp.async.  In the flat parameter buffer (state_dict order: bias, A.0 .. A.n-1, B.*, C.*, D.*,
// E.*, F.*, G.*) the entries of one list for consecutive stages are adjacent, so a (chunk, direction) needs FOUR contiguous ranges
// (three for the anticausal direction): four copy loops of 16-byte cp.async instead of one small loop per stage and array -- the
// per-array loops cost every thread ~2 000 instructions (17 us of a 40 us kernel, measured by ablation).
struct ListRange { int lo, n, sm; };     // first float in the flat buffer (rounded down to a multiple of 4), floats to copy, shared-memory offset
__device__ __forceinline__ ListRange list_range(int off_first, int n_first, int off_last, int n_last, int sm) {
    int lo = off_first < off_last ? off_first : off_last;
    const int e1 = off_first + n_first, e2 = off_last + n_last;
    const int hi = e1 > e2 ? e1 : e2;
    lo &= ~3;
    return ListRange{lo, hi - lo, sm};
}
__device__ __forceinline__ void copy_range_async(float* pbuf, const float* __restrict__ params, const ListRange& r, int tid, int nthreads) {
    // params + lo is 16-byte aligned when the flat buffer is (torch allocations are); otherwise fall back to 4-byte copies
    const float* src = params + r.lo;
    float* dst = pbuf + r.sm;
    const int n4 = ((reinterpret_cast<uintptr_t>(src) & 15) == 0) ? (r.n >> 2) : 0;
    for (int e = tid; e < n4; e += nthreads) cp_async16(dst + 4 * e, src + 4 * e);
    for (int e = 4 * n4 + tid; e < r.n; e += nthreads) cp_async4(dst + e, src + e);
}
// returns the floats of shared memory used; ptrs[i] = offsets of stage i's matrices inside pbuf
__device__ __forceinline__ int chunk_params_ranges(float* pbuf, StageP* ptrs, const sn_sss_stage* sdesc, int nst, const float* __restrict__ params, int tid,
                                                   int nthreads) {
    const sn_sss_stage& f = sdesc[0];
    const sn_sss_stage& l = sdesc[nst - 1];
    const bool has_yu = f.off_yu >= 0;
    ListRange r_ss = list_range(f.off_ss, f.d_out * f.d_in, l.off_ss, l.d_out * l.d_in, 0);
    ListRange r_ys = list_range(f.off_ys, f.out_dim * f.d_in, l.off_ys, l.out_dim * l.d_in, pad4(r_ss.n));
    ListRange r_su = list_range(f.off_su, f.d_out * f.in_dim, l.off_su, l.d_out * l.in_dim, r_ys.sm + pad4(r_ys.n));
    ListRange r_yu = has_yu ? list_range(f.off_yu, f.out_dim * f.in_dim, l.off_yu, l.out_dim * l.in_dim, r_su.sm + pad4(r_su.n)) : ListRange{0, 0, r_su.sm + pad4(r_su.n)};
    copy_range_async(pbuf, params, r_ss, tid, nthreads);
    copy_range_async(pbuf, params, r_ys, tid, nthreads);
    copy_range_async(pbuf, params, r_su, tid, nthreads);
    if (has_yu) copy_range_async(pbuf, params, r_yu, tid, nthreads);
    if (tid < nst) {
        const sn_sss_stage& st = sdesc[tid];
        ptrs[tid] = StageP{r_ss.sm + st.off_ss - r_ss.lo, r_ys.sm + st.off_ys - r_ys.lo, r_su.sm + st.off_su - r_su.lo, has_yu ? r_yu.sm + st.off_yu - r_yu.lo : 0};
    }
    return r_yu.sm + pad4(r_yu.n);
}

// lo part of a 3xTF32 operand of the warp-level tensor-core products (mma.sync): x - rn_tf32(x) is exact in fp32 and is handed over as
// it is -- the tensor core drops the 13 low mantissa bits of its tf32 operands itself; because hi is rounded to NEAREST the remainder has
// either sign, so that truncation does not bias the product (the tcgen05 paths truncate hi and therefore round lo, see lo_of_trunc).
// cvt.rna.tf32.f32 is not an instruction on sm_100a (ptxas emits add / mask / isfinite / select): a split costs 3 instructions this way
// instead of 9, and the splits were three quarters of the instructions of the scan kernels (ncu source view, r2n).
#ifndef SN_MMA_LO_ROUND
#define SN_MMA_LO_ROUND 0
#endif
__device__ __forceinline__ float mma_lo(float remainder) { return SN_MMA_LO_ROUND ? tf32_hi(remainder) : remainder; }

// B fragment (M[row][col], M[row][col + 1]) of a compact row-major [nrows][ncols] matrix, zero outside; split into tf32 hi / lo
__device__ __forceinline__ void frag_b(const float* M, int row, int nrows, int col, int ncols, float2& hi, float2& lo) {
    float2 r = make_float2(0.f, 0.f);
    if (row < nrows) {
        if (ncols == DS && (reinterpret_cast<uintptr_t>(M) & 7) == 0) {
            r = *reinterpret_cast<const float2*>(M + row * DS + col);
        } else {
            if (col < ncols) r.x = M[row * ncols + col];
            if (col + 1 < ncols) r.y = M[row * ncols + col + 1];
        }
    }
    hi.x = tf32_hi(r.x); hi.y = tf32_hi(r.y);
    lo.x = mma_lo(r.x - hi.x); lo.y = mma_lo(r.y - hi.y);
}

__device__ __forceinline__ void mma_1688(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
struct Frag3 { uint32_t hi[4], lo[4]; };
// D fragment (row g: columns 2t, 2t+1; row g+8: columns 2t, 2t+1) -> A fragment of the next product, K permuted as described above
__device__ __forceinline__ void split_frag(const float (&d)[4], Frag3& f) {
    const float v[4] = {d[0], d[2], d[1], d[3]};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float hi = tf32_hi(v[i]);
        f.hi[i] = __float_as_uint(hi);
        f.lo[i] = __float_as_uint(mma_lo(v[i] - hi));
    }
}
// d += A B with B given pre-split (hi pair, lo pair); small terms first
__device__ __forceinline__ void mma3(float (&d)[4], const Frag3& a, const float2 bh, const float2 bl) {
    mma_1688(d, a.lo, __float_as_uint(bh.x), __float_as_uint(bh.y));
    mma_1688(d, a.hi, __float_as_uint(bl.x), __float_as_uint(bl.y));
    mma_1688(d, a.hi, __float_as_uint(bh.x), __float_as_uint(bh.y));
}

// one of the three terms of d += A B (0: lo * hi, 1: hi * lo, 2: hi * hi): the kernels issue the terms of INDEPENDENT accumulators
// round-robin -- the asm statements keep their order, and an HMMA that adds into the accumulator of its predecessor waits ~27 cycles
template <int TERM>
__device__ __forceinline__ void mma_t(float (&d)[4], const Frag3& a, const float2 bh, const float2 bl) {
    if (TERM == 0) mma_1688(d, a.lo, __float_as_uint(bh.x), __float_as_uint(bh.y));
    else if (TERM == 1) mma_1688(d, a.hi, __float_as_uint(bl.x), __float_as_uint(bl.y));
    else mma_1688(d, a.hi, __float_as_uint(bh.x), __float_as_uint(bh.y));
}

// the two columns (fragment rows g and g + 8) a lane looks after
struct ColPair {
    int tcol[2];      // column of the chunk (input tiles) or unit-state index (state tile)
    bool valid[2];
    bool act[2];
};

__global__ void __launch_bounds__(BM_THREADS)
sss_tc_buildm_kernel(const sn_sss_stage* __restrict__ stages, int n, const sn_sss_tc_chunk* __restrict__ chunks, const float* __restrict__ params,
                     float* __restrict__ Wall, float* __restrict__ SCall, float* __restrict__ VG, int lists_contiguous) {
    extern __shared__ __align__(16) float build_smem[];
    __shared__ sn_sss_stage sdesc[LMAX];
    __shared__ StageP smt[LMAX];
    const sn_sss_tc_chunk c = chunks[blockIdx.x];
    const int dir = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int nst = c.k_end - c.k_begin;
    float* W = Wall + (size_t)blockIdx.x * WROWS * WCOLS;
    float* SC = SCall + (size_t)blockIdx.x * SCF;
    float* Phi = SC + dir * DS * DS;
    float* Omat = SC + 2 * DS * DS + dir * PO * DS;
    if (tid < nst) sdesc[tid] = stage_of(stages, n, dir, dir == 0 ? c.k_begin + tid : c.k_end - 1 - tid);
    __syncthreads();
    if (lists_contiguous) chunk_params_ranges(build_smem, smt, sdesc, nst, params, tid, BM_THREADS);
    else chunk_params_async(build_smem, smt, sdesc, nst, params, tid, BM_THREADS);
    cp_async_commit();
    cp_async_wait_all();
    __syncthreads();
#if defined(SN_BUILD_ABL) && SN_BUILD_ABL == 1
    return;                                                 // ablation: parameter staging only
#endif
    const int tile = BM_SPLIT * warp + blockIdx.z;
    if (tile >= BM_TILES) return;
    const bool state_tile = tile == BM_TILES - 1;
    if (!state_tile && 16 * tile >= c.ncols) return;          // no input column in this tile
    ColPair cp;
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
        cp.tcol[rr] = state_tile ? g + 8 * rr : 16 * tile + g + 8 * rr;
        cp.valid[rr] = state_tile || cp.tcol[rr] < c.ncols;
        cp.act[rr] = false;
    }
    float d[2][4];
#pragma unroll
    for (int hp = 0; hp < 2; ++hp)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int sidx = cp.tcol[k >> 1], a = 8 * hp + 2 * t + (k & 1);
            d[hp][k] = (state_tile && a == sidx && sidx < sdesc[0].d_in) ? 1.f : 0.f;
        }
    for (int i = 0; i < nst; ++i) {
        const sn_sss_stage& st = sdesc[i];
        const StageP& m = smt[i];
        int local[2];
        bool mine[2];
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            local[rr] = c.col0 + cp.tcol[rr] - st.in_off;
            mine[rr] = !state_tile && cp.valid[rr] && local[rr] >= 0 && local[rr] < st.in_dim;
        }
        // the state entering the stage, kept for the backward of the construction: VG[chunk][dir][stage][column][component]
        {
            float* vi = VG + (((size_t)(blockIdx.x * 2 + dir) * LMAX + i) * COLT + 16 * tile) * DS;
#pragma unroll
            for (int hp = 0; hp < 2; ++hp) {
                *reinterpret_cast<float2*>(vi + g * DS + 8 * hp + 2 * t) = make_float2(d[hp][0], d[hp][1]);
                *reinterpret_cast<float2*>(vi + (g + 8) * DS + 8 * hp + 2 * t) = make_float2(d[hp][2], d[hp][3]);
            }
        }
        const bool live = state_tile || cp.act[0] || cp.act[1] || mine[0] || mine[1];
        if (!__any_sync(0xffffffffu, live)) continue;          // every column of the tile still waits for its stage
        Frag3 a[2];
        split_frag(d[0], a[0]);
        split_frag(d[1], a[1]);
        const int rbase = st.out_off - c.row0;
        // outputs of the stage from the state ENTERING it, Y = V ys^T (+ yu), and the state leaving it, V <- V ss^T (+ su): up to four
        // independent accumulators (two output n-tiles, two state halves), their products issued round-robin
        const bool y0on = st.out_dim > 0, y1on = st.out_dim > 8;        // warp-uniform
        float2 ybh[2][2], ybl[2][2], sbh[2][2], sbl[2][2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
                if (nt == 0 ? y0on : y1on) frag_b(build_smem + m.ys, 8 * nt + g, st.out_dim, 8 * h + 2 * t, st.d_in, ybh[nt][h], ybl[nt][h]);
#pragma unroll
            for (int hp = 0; hp < 2; ++hp) frag_b(build_smem + m.ss, 8 * hp + g, st.d_out, 8 * h + 2 * t, st.d_in, sbh[hp][h], sbl[hp][h]);
        }
        float y[2][4], sn[2][4];
#pragma unroll
        for (int q = 0; q < 2; ++q)
#pragma unroll
            for (int k = 0; k < 4; ++k) { y[q][k] = 0.f; sn[q][k] = 0.f; }
#define SN_ROUND(TERM, H)                                                                        \
        if (y0on) mma_t<TERM>(y[0], a[H], ybh[0][H], ybl[0][H]);                                 \
        mma_t<TERM>(sn[0], a[H], sbh[0][H], sbl[0][H]);                                          \
        if (y1on) mma_t<TERM>(y[1], a[H], ybh[1][H], ybl[1][H]);                                 \
        mma_t<TERM>(sn[1], a[H], sbh[1][H], sbl[1][H]);
        SN_ROUND(0, 0) SN_ROUND(1, 0) SN_ROUND(2, 0) SN_ROUND(0, 1) SN_ROUND(1, 1) SN_ROUND(2, 1)
#undef SN_ROUND
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
            if (8 * nt >= st.out_dim) break;
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
                if (!cp.valid[rr]) continue;
                const bool wr = dir == 0 ? (cp.act[rr] || mine[rr]) : cp.act[rr];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int r = 8 * nt + 2 * t + e;
                    if (r >= st.out_dim) continue;
                    float val = y[nt][2 * rr + e];
                    if (mine[rr] && st.off_yu >= 0) val += build_smem[m.yu + r * st.in_dim + local[rr]];
                    if (state_tile) Omat[(rbase + r) * DS + cp.tcol[rr]] = val;
                    else if (wr) store_hi_lo(W, rbase + r, cp.tcol[rr], val);
                }
            }
        }
        // the columns whose stage this is enter the state through su
#pragma unroll
        for (int hp = 0; hp < 2; ++hp) {
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
                if (mine[rr]) {
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int b = 8 * hp + 2 * t + e;
                        if (b < st.d_out) sn[hp][2 * rr + e] += build_smem[m.su + b * st.in_dim + local[rr]];
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) d[hp][k] = sn[hp][k];
        }
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) cp.act[rr] = cp.act[rr] || mine[rr];
    }
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
        if (!cp.valid[rr]) continue;
#pragma unroll
        for (int hp = 0; hp < 2; ++hp)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int b = 8 * hp + 2 * t + e;
                const float val = d[hp][2 * rr + e];
                if (state_tile) Phi[b * DS + cp.tcol[rr]] = val;
                else store_hi_lo(W, PO + dir * DS + b, cp.tcol[rr], val);
            }
    }
}

__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
    hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);   // round to nearest tf32 (ties away), finite inputs
    // lo is rounded too: the tensor core truncates its operands, and a truncated remainder biases every product towards zero
    lo = __uint_as_float((__float_as_uint(x - hi) + 0x1000u) & 0xFFFFE000u);
}
// lo part against the TRUNCATED hi part (what the tensor core itself makes of an unsplit fp32 operand)
__device__ __forceinline__ float lo_of_trunc(float x) {
    const float hi = __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
    return __uint_as_float((__float_as_uint(x - hi) + 0x1000u) & 0xFFFFE000u);
}
__device__ __forceinline__ void lo_of_trunc(const float4& v, float4& l) {
    l.x = lo_of_trunc(v.x); l.y = lo_of_trunc(v.y); l.z = lo_of_trunc(v.z); l.w = lo_of_trunc(v.w);
}
__device__ __forceinline__ void split_tf32(const float4& v, float4& h, float4& l) {
    split_tf32(v.x, h.x, l.x);
    split_tf32(v.y, h.y, l.y);
    split_tf32(v.z, h.z, l.z);
    split_tf32(v.w, h.w, l.w);
}

#if defined(SN_CHAIN_PROF) || defined(SN_SCAN_PROF)
#define CHPROF_DECL(n) long long chp_acc[n]; for (int chp_i = 0; chp_i < n; ++chp_i) chp_acc[chp_i] = 0; long long chp_t = 0; (void)chp_t
#define CHPROF_T0() chp_t = clock64()
#define CHPROF_LAP(i) do { const long long chp_n = clock64(); chp_acc[i] += chp_n - chp_t; chp_t = chp_n; } while (0)
#define CHPROF_PRINT(tag, n, steps) do { if (blockIdx.x == 0 || blockIdx.x == 301 || blockIdx.x == 100) for (int chp_i = 0; chp_i < n; ++chp_i) \
    printf("CHPROF %s blk %d phase %d avg %lld cyc/step\n", tag, (int)blockIdx.x, chp_i, chp_acc[chp_i] / (steps)); } while (0)
#else
#define CHPROF_DECL(n)
#define CHPROF_T0()
#define CHPROF_LAP(i)
#define CHPROF_PRINT(tag, n, steps)
#endif

// shared memory (TMA swizzled layout) -> global tensor box; rows past the tensor's extent are clipped
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// ------------------------------------------------------------------------------------------
// 2. local GEMM: [yloc | r | r'](128 samples x 64) = u_j (128 x 32 nkb) * W_j^T, 3xTF32
//    warp 0: TMA producer | warp 1: TMEM alloc + MMA issuer | warps 2-9: lo-part converters | warps 10-13: epilogue
// ------------------------------------------------------------------------------------------
constexpr int G1_CONV = 256;                          // converter threads: two groups of four warps on alternate stages
constexpr int G1_THREADS = 64 + G1_CONV + 128;
// Three rings of 16 KB tiles with their own depths: the x boxes come from HBM and need the most loads in flight, the W boxes are
// L2 hits, the lo tiles only live between a converter group and the MMA.
#ifndef SN_G1_XS
#define SN_G1_XS 4
#define SN_G1_WS 4
#endif
constexpr int G1_XS = SN_G1_XS, G1_WS = SN_G1_WS, G1_LS = 2;
static_assert(G1_XS % G1_LS == 0 && G1_LS == 2, "a converter group (= lo slot) must own its x slots: it never skips a barrier phase");
constexpr int G1_TILE_BYTES = 128 * 128;              // 128 rows x 128 B
constexpr int G1_X_OFF = 0, G1_W_OFF = G1_XS * G1_TILE_BYTES, G1_L_OFF = G1_W_OFF + G1_WS * G1_TILE_BYTES;
constexpr int G1_OUT_OFF = G1_L_OFF + G1_LS * G1_TILE_BYTES;   // output staging: Y [128][32] (SWIZZLE_128B) | R [128][16] | R' [128][16] (SWIZZLE_64B)
constexpr int G1_BAR_OFF = G1_OUT_OFF + 2 * G1_TILE_BYTES;
#ifndef SN_G1_PF
#define SN_G1_PF 0
#endif
constexpr int G1_PF = SN_G1_PF;                      // L2 prefetch distance in work items
#ifndef SN_G1_PFG
#define SN_G1_PFG 1
#endif
constexpr int G1_PFG = SN_G1_PFG;                    // work items per prefetch burst
constexpr int G1_MAX_CHUNKS = 1024;
constexpr size_t G1_SMEM = (size_t)G1_BAR_OFF + 1024 + 256 + G1_MAX_CHUNKS * 8;

__global__ void __launch_bounds__(G1_THREADS, 1)
sss_tc_local_gemm_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_oy,
                         const __grid_constant__ CUtensorMap map_or, const sn_sss_tc_chunk* __restrict__ chunks, int nchunks, long B, int ntiles) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space (LDS/STS)
    uint64_t* x_full = reinterpret_cast<uint64_t*>(smem + G1_BAR_OFF);
    uint64_t* x_empty = x_full + G1_XS;
    uint64_t* w_full = x_empty + G1_XS;
    uint64_t* w_empty = w_full + G1_WS;
    uint64_t* conv = w_empty + G1_WS;
    uint64_t* l_empty = conv + G1_LS;
    uint64_t* acc_full = l_empty + G1_LS;
    uint64_t* acc_empty = acc_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long total = (long)ntiles * nchunks;
    const long per = (total + gridDim.x - 1) / gridDim.x;
    const long w0 = (long)blockIdx.x * per;
    const long w1 = w0 + per < total ? w0 + per : total;
    if (w0 >= w1) return;

    int2* ctab = reinterpret_cast<int2*>(smem + G1_BAR_OFF + 256);   // (col0, nkb) per chunk: no global load on the issue paths
    for (int i = threadIdx.x; i < nchunks; i += G1_THREADS) ctab[i] = make_int2(chunks[i].col0, chunks[i].nkb);
    if (threadIdx.x == 0) {
        for (int s = 0; s < G1_XS; ++s) { mbar_init(x_full + s, 1); mbar_init(x_empty + s, 1); }
        for (int s = 0; s < G1_WS; ++s) { mbar_init(w_full + s, 1); mbar_init(w_empty + s, 1); }
        for (int s = 0; s < G1_LS; ++s) { mbar_init(conv + s, 128); mbar_init(l_empty + s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(acc_full + b, 1); mbar_init(acc_empty + b, 128); }
        mbar_fence_init();
        tma_prefetch_desc(&map_x);
        tma_prefetch_desc(&map_w);
        tma_prefetch_desc(&map_oy);
        tma_prefetch_desc(&map_or);
    }
    if (warp == 1) tmem_alloc<256>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int tile0 = (int)(w0 / nchunks), ch0 = (int)(w0 % nchunks);   // every role walks (tile, chunk) incrementally: no 64-bit divisions in the loops

    if (warp == 0) {
        if (elect_one()) {
            // x boxes are pulled into L2 G1_PF items ahead of the shared-memory pipeline
            int ptile = tile0, pch = ch0;
            auto prefetch_next = [&]() {
                const int2 c = ctab[pch];
                for (int kb = 0; kb < c.y; ++kb) tma_prefetch_l2_2d(&map_x, c.x + kb * KBW, ptile * 128);
                if (++pch == nchunks) { pch = 0; ++ptile; }
            };
            // in groups of G1_PFG items, so that DRAM sees G1_PFG x 640 contiguous bytes of every sample row at a time
            long pw = w0;
            for (; pw < w0 + G1_PF + G1_PFG && pw < w1; ++pw) prefetch_next();
            uint32_t it = 0;
            int tile = tile0, ch = ch0;
            for (long w = w0; w < w1; ++w) {
                if (pw < w1 && pw - w <= G1_PF)
                    for (int g = 0; g < G1_PFG && pw < w1; ++g, ++pw) prefetch_next();
                const int nkb = ctab[ch].y, col0 = ctab[ch].x;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const uint32_t xs = it % G1_XS, xr = it / G1_XS, ws = it % G1_WS, wr = it / G1_WS;
                    if (xr > 0) mbar_wait(x_empty + xs, (xr - 1) & 1);
                    mbar_expect_tx(x_full + xs, G1_TILE_BYTES);
                    tma_load_2d(smem + G1_X_OFF + xs * G1_TILE_BYTES, &map_x, col0 + kb * KBW, tile * 128, x_full + xs);
                    if (wr > 0) mbar_wait(w_empty + ws, (wr - 1) & 1);
                    mbar_expect_tx(w_full + ws, G1_TILE_BYTES);
                    tma_load_2d(smem + G1_W_OFF + ws * G1_TILE_BYTES, &map_w, kb * KBW, ch * WROWS, w_full + ws);
                }
                if (++ch == nchunks) { ch = 0; ++tile; }
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
            constexpr uint32_t idesc1 = idesc_tf32(128, 128, false, false);   // x_hi * [W_hi ; W_lo]
            constexpr uint32_t idesc2 = idesc_tf32(128, 64, false, false);    // x_lo * W_hi
            uint32_t it = 0, ai = 0;
            int ch = ch0;
            for (long w = w0; w < w1; ++w, ++ai) {
                const int nkb = ctab[ch].y;
                const uint32_t b = ai & 1;
                if (ai >= 2) mbar_wait(acc_empty + b, ((ai >> 1) - 1) & 1);
                tc_fence_after();
                const uint32_t acc = tmem_base + b * 128;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const uint32_t xs = it % G1_XS, ws = it % G1_WS, wr = it / G1_WS, ls = it % G1_LS, lr = it / G1_LS;
                    mbar_wait(w_full + ws, wr & 1);
                    mbar_wait(conv + ls, lr & 1);          // the converters waited for the x box
                    tc_fence_after();
                    const uint64_t dxh = desc_kmajor_sw128(smem + G1_X_OFF + xs * G1_TILE_BYTES);
                    const uint64_t dxl = desc_kmajor_sw128(smem + G1_L_OFF + ls * G1_TILE_BYTES);
                    const uint64_t dw = desc_kmajor_sw128(smem + G1_W_OFF + ws * G1_TILE_BYTES);
#pragma unroll
                    for (int k = 0; k < KBW / 8; ++k) {   // one tf32 UMMA = 8 floats = 32 bytes of K (+2 in 16-byte units)
                        mma_tf32(acc, dxh + 2 * k, dw + 2 * k, idesc1, (kb | k) ? 1u : 0u);
                        mma_tf32(acc, dxl + 2 * k, dw + 2 * k, idesc2, 1u);
                    }
                    umma_commit(l_empty + ls);
                    umma_commit(x_empty + xs);
                    umma_commit(w_empty + ws);
                }
                umma_commit(acc_full + b);
                if (++ch == nchunks) ch = 0;
            }
        }
    } else if (warp < 2 + G1_CONV / 32) {
        // converters: the raw tile is the hi operand (the tensor core truncates its operands to tf32; verified: parity is unchanged),
        // only lo = rn(x - trunc(x)) is written, into the lo ring (identical swizzled layout, so plain 16-byte chunks).
        // A stage costs one converter warp a full LDS -> STS -> proxy-fence round trip, so two groups of four warps take alternate
        // stages (group = lo slot; it owns x slots of its own parity and never skips a phase of their barriers).
        const int grp = (warp - 2) >> 2, ct = (threadIdx.x - 64) & 127;
        uint32_t it = 0;
        int ch = ch0;
        for (long w = w0; w < w1; ++w) {
            const int nkb = ctab[ch].y;
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                if ((int)(it & 1) != grp) continue;
                const uint32_t xs = it % G1_XS, xr = it / G1_XS, lr = it / G1_LS;
                mbar_wait(x_full + xs, xr & 1);
                const float4* xh = reinterpret_cast<const float4*>(smem + G1_X_OFF + xs * G1_TILE_BYTES);
                float4* xl = reinterpret_cast<float4*>(smem + G1_L_OFF + grp * G1_TILE_BYTES);
                float4 v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = xh[ct + 128 * i];
                if (lr > 0) mbar_wait(l_empty + grp, (lr - 1) & 1);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    float4 l;
                    lo_of_trunc(v[i], l);
                    xl[ct + 128 * i] = l;
                }
                fence_async_smem();
                mbar_arrive(conv + grp);
            }
            if (++ch == nchunks) ch = 0;
        }
    } else {
        // epilogue: TMEM lane quarter = warp % 4; thread = one sample row.  The rows go through a swizzled staging tile and leave as
        // three TMA tensor stores (Y [chunk][B][32], R and R' [chunk][B][16]: 16 + 8 + 8 KB of contiguous global memory per item).
        // Per-thread 16-byte stores at a 128-byte lane stride filled every 32-byte sector in two halves: the L2 fetched the sectors
        // from DRAM to merge them (+0.24 GB read per launch) and the kernel was a third slower.
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const bool leader = (warp == 2 + G1_CONV / 32) && lane == 0;
        const uint32_t sy = smem_u32(smem + G1_OUT_OFF), sr = sy + G1_TILE_BYTES, sp = sr + G1_TILE_BYTES / 2;
        const uint32_t oy = sy + r * 128, orr = sr + r * 64, opp = sp + r * 64;
        uint32_t ai = 0;
        int tile = tile0, ch = ch0;
        for (long w = w0; w < w1; ++w, ++ai) {
            const uint32_t b = ai & 1;
            mbar_wait(acc_full + b, (ai >> 1) & 1);
            tc_fence_after();
            const uint32_t acc = tmem_base + b * 128 + ((uint32_t)(q * 32) << 16);
            float out[64];
#pragma unroll
            for (int c0 = 0; c0 < 64; c0 += 16) {
                uint32_t m[16], x2[16];
                tmem_ld16_nowait(acc + c0, m);
                tmem_ld16_nowait(acc + 64 + c0, x2);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 16; ++i) out[c0 + i] = __uint_as_float(m[i]) + __uint_as_float(x2[i]);
            }
            tc_fence_before();
            mbar_arrive(acc_empty + b);
            if (ai > 0) {   // the previous item's stores have read the staging tile
                if (leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                named_bar_sync(1, 128);
            }
#pragma unroll
            for (int c = 0; c < 8; ++c)
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(oy + ((c ^ (r & 7)) << 4)), "f"(out[4 * c]), "f"(out[4 * c + 1]), "f"(out[4 * c + 2]), "f"(out[4 * c + 3]) : "memory");
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const uint32_t o = (uint32_t)((c ^ ((r >> 1) & 3)) << 4);
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(orr + o), "f"(out[32 + 4 * c]), "f"(out[33 + 4 * c]), "f"(out[34 + 4 * c]), "f"(out[35 + 4 * c]) : "memory");
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(opp + o), "f"(out[48 + 4 * c]), "f"(out[49 + 4 * c]), "f"(out[50 + 4 * c]), "f"(out[51 + 4 * c]) : "memory");
            }
            fence_async_smem();
            named_bar_sync(1, 128);
            if (leader) {
                tma_store_3d(&map_oy, sy, 0, tile * 128, ch);
                tma_store_3d(&map_or, sr, 0, tile * 128, ch);
                tma_store_3d(&map_or, sp, 0, tile * 128, nchunks + ch);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            if (++ch == nchunks) { ch = 0; ++tile; }
        }
        if (leader) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<256>(tmem_base);
    }
}

// ------------------------------------------------------------------------------------------
// shared-memory matrix-vector helpers of the SIMT scans (thread = sample)
// ------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 128;

// out[b] += sum_a M[b][a] v[a]   (M row-major DS columns in shared memory, read as broadcast float4)
template <int ROWS>
__device__ __forceinline__ void matvec_acc(const float4* __restrict__ M, const float (&v)[DS], float* out) {
#pragma unroll
    for (int b = 0; b < ROWS; ++b) {
        float acc = out[b];
#pragma unroll
        for (int a4 = 0; a4 < DS / 4; ++a4) {
            const float4 m = M[b * (DS / 4) + a4];
            acc = fmaf(m.x, v[4 * a4], acc);
            acc = fmaf(m.y, v[4 * a4 + 1], acc);
            acc = fmaf(m.z, v[4 * a4 + 2], acc);
            acc = fmaf(m.w, v[4 * a4 + 3], acc);
        }
        out[b] = acc;
    }
}
// ------------------------------------------------------------------------------------------
// 2+3 fused (large batches): one CTA walks whole 128-sample tiles chunk by chunk, so the chunk-level scans run in the
//    epilogue while the tensor core works on the next chunk -- no [yloc | r | r'] round trip through HBM.
//    warp 0: TMA producer | warp 1: MMA issuer | warps 2-5: hi/lo converters
//    warps 6-9  : epilogue, thread = sample: TMEM -> registers, causal state recursion, y = yloc + O s + bias, saves s_j and r'_j
//    warps 10-13: finalizer, thread = sample, one tile behind: anticausal recursion over the saved r'_j, y += O' e, saves e_{j+1}
// ------------------------------------------------------------------------------------------
constexpr int F_THREADS = 448;
constexpr int F_MAX_CHUNKS = 512;
constexpr int F_SC_HALF = DS * DS + PO * DS + PO;   // 800 floats: one direction's Phi and O, then the chunk's bias entries
// the fused variant keeps the original 4-stage ring of (x | x_lo | W) tiles
constexpr int G1_STAGES = 4;
constexpr int G1_STAGE_BYTES = 3 * G1_TILE_BYTES;
constexpr size_t F_SMEM = (size_t)G1_STAGES * G1_STAGE_BYTES + 256 + F_MAX_CHUNKS * 16 + 4 * F_SC_HALF * 4 + 1024;


// cooperative copy of one direction's {Phi (64 float4), O (128 float4)} by 128 threads: registers first (latency hidden behind
// the barrier wait that follows), shared memory later
struct ScRegs { float4 a, b; };
// bias_c (may be NULL): the chunk's bias entries, staged behind the matrices by threads 64..71 (nrows: valid entries)
__device__ __forceinline__ ScRegs sc_fetch(const float* __restrict__ SCj, int dir, int t, const float* __restrict__ bias_c = nullptr,
                                           int nrows = 0, int aligned = 0) {
    const float4* g = reinterpret_cast<const float4*>(SCj);
    ScRegs r;
    const int phi0 = dir * (DS * DS / 4), o0 = 2 * (DS * DS / 4) + dir * (PO * DS / 4);
    r.a = __ldg(g + (t < 64 ? phi0 + t : o0 + (t - 64)));
    r.b = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t < 64) {
        r.b = __ldg(g + o0 + 64 + t);
    } else if (t < 72 && bias_c != nullptr) {
        const int c = 4 * (t - 64);
        if (aligned && c + 4 <= nrows) {
            r.b = __ldg(reinterpret_cast<const float4*>(bias_c + c));
        } else {
            if (c < nrows) r.b.x = __ldg(bias_c + c);
            if (c + 1 < nrows) r.b.y = __ldg(bias_c + c + 1);
            if (c + 2 < nrows) r.b.z = __ldg(bias_c + c + 2);
            if (c + 3 < nrows) r.b.w = __ldg(bias_c + c + 3);
        }
    }
    return r;
}
__device__ __forceinline__ void sc_store(float4* buf, const ScRegs& r, int t) {   // buf: [Phi 64][O 128][bias 8] float4
    buf[t] = r.a;                      // t < 64: Phi[t] ; t >= 64: O[t - 64]  (same index: 64 + (t - 64))
    if (t < 64) buf[128 + t] = r.b;    // O[64 + t]
    else if (t < 72) buf[192 + (t - 64)] = r.b;
}

__global__ void __launch_bounds__(F_THREADS, 1)
sss_tc_fwd_fused_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                        const sn_sss_tc_chunk* __restrict__ chunks, int nchunks, long B, int ntiles, const float* __restrict__ SCall,
                        float* __restrict__ states, float* __restrict__ y, long ldy, const float* __restrict__ bias, int aligned) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space (LDS/STS)
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + G1_STAGES * G1_STAGE_BYTES);
    uint64_t* conv = full + G1_STAGES;
    uint64_t* empty = conv + G1_STAGES;
    uint64_t* acc_full = empty + G1_STAGES;
    uint64_t* acc_empty = acc_full + 2;
    uint64_t* tile_done = acc_empty + 2;
    uint64_t* fin_done = tile_done + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(fin_done + 2);
    int4* ctab = reinterpret_cast<int4*>(smem + G1_STAGES * G1_STAGE_BYTES + 256);        // col0, nkb, row0, nrows
    float4* scE = reinterpret_cast<float4*>(ctab + F_MAX_CHUNKS);                          // 2 x 192 float4
    float4* scF = scE + 2 * (F_SC_HALF / 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t0 = (int)((long)blockIdx.x * ntiles / gridDim.x);
    const int t1 = (int)((long)(blockIdx.x + 1) * ntiles / gridDim.x);
    if (t0 >= t1) return;

    for (int i = threadIdx.x; i < nchunks; i += F_THREADS) ctab[i] = make_int4(chunks[i].col0, chunks[i].nkb, chunks[i].row0, chunks[i].nrows);
    if (threadIdx.x == 0) {
        for (int s = 0; s < G1_STAGES; ++s) { mbar_init(full + s, 1); mbar_init(conv + s, 128); mbar_init(empty + s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(acc_full + b, 1); mbar_init(acc_empty + b, 128); mbar_init(tile_done + b, 128); mbar_init(fin_done + b, 128); }
        mbar_fence_init();
        tma_prefetch_desc(&map_x);
        tma_prefetch_desc(&map_w);
    }
    if (warp == 1) tmem_alloc<256>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (elect_one()) {
            uint32_t it = 0;
            for (int tile = t0; tile < t1; ++tile) {
                for (int ch = 0; ch < nchunks; ++ch) {
                    const int4 c = ctab[ch];
                    for (int kb = 0; kb < c.y; ++kb, ++it) {
                        const uint32_t s = it % G1_STAGES, round = it / G1_STAGES;
                        if (round > 0) mbar_wait(empty + s, (round - 1) & 1);
                        uint8_t* st = smem + s * G1_STAGE_BYTES;
                        mbar_expect_tx(full + s, 2 * G1_TILE_BYTES);
                        tma_load_2d(st, &map_x, c.x + kb * KBW, tile * 128, full + s);
                        tma_load_2d(st + 2 * G1_TILE_BYTES, &map_w, kb * KBW, ch * WROWS, full + s);
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
            constexpr uint32_t idesc1 = idesc_tf32(128, 128, false, false);
            constexpr uint32_t idesc2 = idesc_tf32(128, 64, false, false);
            uint32_t it = 0, ai = 0;
            for (int tile = t0; tile < t1; ++tile) {
                for (int ch = 0; ch < nchunks; ++ch, ++ai) {
                    const int nkb = ctab[ch].y;
                    const uint32_t b = ai & 1;
                    if (ai >= 2) mbar_wait(acc_empty + b, ((ai >> 1) - 1) & 1);
                    tc_fence_after();
                    const uint32_t acc = tmem_base + b * 128;
                    for (int kb = 0; kb < nkb; ++kb, ++it) {
                        const uint32_t s = it % G1_STAGES, round = it / G1_STAGES;
                        mbar_wait(conv + s, round & 1);
                        tc_fence_after();
                        uint8_t* st = smem + s * G1_STAGE_BYTES;
                        const uint64_t dxh = desc_kmajor_sw128(st);
                        const uint64_t dxl = desc_kmajor_sw128(st + G1_TILE_BYTES);
                        const uint64_t dw = desc_kmajor_sw128(st + 2 * G1_TILE_BYTES);
#pragma unroll
                        for (int k = 0; k < KBW / 8; ++k) {
                            mma_tf32(acc, dxh + 2 * k, dw + 2 * k, idesc1, (kb | k) ? 1u : 0u);
                            mma_tf32(acc, dxl + 2 * k, dw + 2 * k, idesc2, 1u);
                        }
                        umma_commit(empty + s);
                    }
                    umma_commit(acc_full + b);
                }
            }
        }
    } else if (warp < 6) {
        const int ct = threadIdx.x - 64;
        uint32_t it = 0;
        for (int tile = t0; tile < t1; ++tile) {
            for (int ch = 0; ch < nchunks; ++ch) {
                const int nkb = ctab[ch].y;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const uint32_t s = it % G1_STAGES, round = it / G1_STAGES;
                    mbar_wait(full + s, round & 1);
                    float4* xh = reinterpret_cast<float4*>(smem + s * G1_STAGE_BYTES);
                    float4* xl = xh + G1_TILE_BYTES / 16;
                    float4 v[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = xh[ct + 128 * i];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        float4 h, l;
                        split_tf32(v[i], h, l);
                        xh[ct + 128 * i] = h;
                        xl[ct + 128 * i] = l;
                    }
                    fence_async_smem();
                    mbar_arrive(conv + s);
                }
            }
        }
    } else if (warp < 10) {
        // ---- epilogue + causal scan ----
        const int q = warp & 3;
        const int et = threadIdx.x - 192;
        uint32_t ai = 0, tl = 0;
        for (int tile = t0; tile < t1; ++tile, ++tl) {
            const long row = (long)tile * 128 + q * 32 + lane;
            const bool valid = row < B;
            float s[DS];
#pragma unroll
            for (int a = 0; a < DS; ++a) s[a] = 0.f;
            for (int ch = 0; ch < nchunks; ++ch, ++ai) {
                const int4 c = ctab[ch];
                const ScRegs scr = sc_fetch(SCall + (size_t)ch * SCF, 0, et, bias != nullptr ? bias + c.z : nullptr, c.w, aligned);
                const uint32_t b = ai & 1;
                mbar_wait(acc_full + b, (ai >> 1) & 1);
                tc_fence_after();
                const uint32_t acc = tmem_base + b * 128 + ((uint32_t)(q * 32) << 16);
                float out[64];
#pragma unroll
                for (int c0 = 0; c0 < 64; c0 += 16) {
                    uint32_t m[16], x2[16];
                    tmem_ld16_nowait(acc + c0, m);
                    tmem_ld16_nowait(acc + 64 + c0, x2);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 16; ++i) out[c0 + i] = __uint_as_float(m[i]) + __uint_as_float(x2[i]);
                }
                tc_fence_before();
                mbar_arrive(acc_empty + b);
                float4* sc = scE + (ai & 1) * (F_SC_HALF / 4);
                sc_store(sc, scr, et);
                named_bar_sync(1, 128);
                if (valid) {
                    float4* sdst = reinterpret_cast<float4*>(states + ((size_t)ch * B + row) * 32);
#pragma unroll
                    for (int i = 0; i < 4; ++i) sdst[i] = make_float4(s[4 * i], s[4 * i + 1], s[4 * i + 2], s[4 * i + 3]);
#pragma unroll
                    for (int i = 0; i < 4; ++i) sdst[4 + i] = make_float4(out[48 + 4 * i], out[49 + 4 * i], out[50 + 4 * i], out[51 + 4 * i]);
                    float* yrow = y + row * ldy + c.z;
                    const float4* Om = sc + DS * DS / 4;
#pragma unroll
                    for (int g = 0; g < PO / 4; ++g) {
                        if (4 * g < c.w) {
                            const float4 b4 = sc[192 + g];   // zero when there is no bias
                            float acc4[4] = {out[4 * g] + b4.x, out[4 * g + 1] + b4.y, out[4 * g + 2] + b4.z, out[4 * g + 3] + b4.w};
                            matvec_acc<4>(Om + g * 4 * (DS / 4), s, acc4);
                            if (aligned && 4 * g + 4 <= c.w) {
                                *reinterpret_cast<float4*>(yrow + 4 * g) = make_float4(acc4[0], acc4[1], acc4[2], acc4[3]);
                            } else {
#pragma unroll
                                for (int i = 0; i < 4; ++i)
                                    if (4 * g + i < c.w) yrow[4 * g + i] = acc4[i];
                            }
                        }
                    }
                }
                float ns[DS];
#pragma unroll
                for (int a = 0; a < DS; ++a) ns[a] = out[32 + a];
                matvec_acc<DS>(sc, s, ns);
#pragma unroll
                for (int a = 0; a < DS; ++a) s[a] = ns[a];
            }
            if (tl >= 2) mbar_wait(fin_done + (tl & 1), ((tl >> 1) - 1) & 1);
            __threadfence_block();
            mbar_arrive(tile_done + (tl & 1));
        }
    } else {
        // ---- finalizer: anticausal scan, one tile behind the epilogue ----
        const int ft = threadIdx.x - 320;
        uint32_t fi = 0, tl = 0;
        for (int tile = t0; tile < t1; ++tile, ++tl) {
            mbar_wait(tile_done + (tl & 1), (tl >> 1) & 1);
            const long row = (long)tile * 128 + ft;
            const bool valid = row < B;
            float e[DS];
#pragma unroll
            for (int a = 0; a < DS; ++a) e[a] = 0.f;
            for (int j = nchunks - 1; j >= 0; --j, ++fi) {
                const ScRegs scr = sc_fetch(SCall + (size_t)j * SCF, 1, ft);
                const int4 c = ctab[j];
                float4* sp = reinterpret_cast<float4*>(states + ((size_t)j * B + (valid ? row : 0)) * 32 + DS);
                float ne[DS];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 r4 = valid ? __ldcg(sp + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                    ne[4 * i] = r4.x; ne[4 * i + 1] = r4.y; ne[4 * i + 2] = r4.z; ne[4 * i + 3] = r4.w;
                }
                float* yrow = y + (valid ? row : 0) * ldy + c.z;
                float yv[PO];
#pragma unroll
                for (int g = 0; g < PO / 4; ++g) {
                    if (valid && aligned && 4 * g + 4 <= c.w) {
                        const float4 v = __ldcg(reinterpret_cast<const float4*>(yrow + 4 * g));
                        yv[4 * g] = v.x; yv[4 * g + 1] = v.y; yv[4 * g + 2] = v.z; yv[4 * g + 3] = v.w;
                    } else {
#pragma unroll
                        for (int i = 0; i < 4; ++i) yv[4 * g + i] = (valid && 4 * g + i < c.w) ? __ldcg(yrow + 4 * g + i) : 0.f;
                    }
                }
                float4* sc = scF + (fi & 1) * (F_SC_HALF / 4);
                sc_store(sc, scr, ft);
                named_bar_sync(2, 128);
                if (valid) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) sp[i] = make_float4(e[4 * i], e[4 * i + 1], e[4 * i + 2], e[4 * i + 3]);
                    const float4* Om = sc + DS * DS / 4;
#pragma unroll
                    for (int g = 0; g < PO / 4; ++g) {
                        if (4 * g < c.w) {
                            matvec_acc<4>(Om + g * 4 * (DS / 4), e, yv + 4 * g);
                            if (aligned && 4 * g + 4 <= c.w) {
                                *reinterpret_cast<float4*>(yrow + 4 * g) = make_float4(yv[4 * g], yv[4 * g + 1], yv[4 * g + 2], yv[4 * g + 3]);
                            } else {
#pragma unroll
                                for (int i = 0; i < 4; ++i)
                                    if (4 * g + i < c.w) yrow[4 * g + i] = yv[4 * g + i];
                            }
                        }
                    }
                }
                matvec_acc<DS>(sc, e, ne);
#pragma unroll
                for (int a = 0; a < DS; ++a) e[a] = ne[a];
            }
            mbar_arrive(fin_done + (tl & 1));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<256>(tmem_base);
    }
}

// ------------------------------------------------------------------------------------------
// 3'/4'. chunk scans, four threads per sample.  The scans are serial in the chunk index, so the only parallelism is across
//    samples (65 536 threads would leave the SMs latency-bound); here thread q of a quad owns state components 4q..4q+3 (and
//    output / grad_y columns 8q..8q+7), forms partial matrix-vector products over its own components and the quad combines
//    them with a 2-step shuffle reduce-scatter.  Coefficients are double-buffered in shared memory with 16-byte cp.async.
// ------------------------------------------------------------------------------------------
constexpr int QS_THREADS = 128;   // 32 samples x 4 threads (64 threads = 16 samples per CTA below 16 k samples: more CTAs per SM)

__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
// out (N/4 values: indices q*N/4 ..) = sum over the quad of p[q*N/4 ..]
template <int N>
__device__ __forceinline__ void quad_reduce_scatter(const float (&p)[N], int q, float (&out)[N / 4]) {
    float h[N / 2];
    const bool hi2 = (q & 2) != 0;
#pragma unroll
    for (int i = 0; i < N / 2; ++i) {
        const float send = hi2 ? p[i] : p[N / 2 + i];
        const float keep = hi2 ? p[N / 2 + i] : p[i];
        h[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    const bool hi1 = (q & 1) != 0;
#pragma unroll
    for (int i = 0; i < N / 4; ++i) {
        const float send = hi1 ? h[i] : h[N / 4 + i];
        const float keep = hi1 ? h[N / 4 + i] : h[i];
        out[i] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
    }
}
__device__ __forceinline__ float dot4(const float4& m, const float (&v)[4]) {
    return fmaf(m.w, v[3], fmaf(m.z, v[2], fmaf(m.y, v[1], m.x * v[0])));
}
// p[0..15] += w * row (16 floats at M[0..3])
__device__ __forceinline__ void axpy16(const float4* __restrict__ M, float w, float (&p)[DS]) {
#pragma unroll
    for (int a4 = 0; a4 < DS / 4; ++a4) {
        const float4 m = M[a4];
        p[4 * a4] = fmaf(m.x, w, p[4 * a4]);
        p[4 * a4 + 1] = fmaf(m.y, w, p[4 * a4 + 1]);
        p[4 * a4 + 2] = fmaf(m.z, w, p[4 * a4 + 2]);
        p[4 * a4 + 3] = fmaf(m.w, w, p[4 * a4 + 3]);
    }
}
__device__ __forceinline__ void sc_prefetch(float4* dst, const float* __restrict__ src, int nfloat4) {
    for (int i = threadIdx.x; i < nfloat4; i += blockDim.x) cp_async16(dst + i, reinterpret_cast<const float4*>(src) + i);
}

__global__ void __launch_bounds__(QS_THREADS)
sss_tc_scan_fwd_q_kernel(const sn_sss_tc_chunk* __restrict__ chunks, int nchunks, const float* __restrict__ SCall, const float* __restrict__ rbuf,
                         float* __restrict__ S, float* __restrict__ y, long ldy, const float* __restrict__ bias, long B, int aligned) {
    __shared__ float4 sc[2][SCF / 4];
    const int q = threadIdx.x & 3;
    const long row = (long)blockIdx.x * (blockDim.x / 4) + (threadIdx.x >> 2);
    const bool valid = row < B;
    const long rr = valid ? row : 0;
    // ---- anticausal states, top chunk first: S[j][row][16..31] = e_{j+1} ----
    float e4[4] = {0.f, 0.f, 0.f, 0.f};
    sc_prefetch(sc[0], SCall + (size_t)(nchunks - 1) * SCF + DS * DS, DS * DS / 4);   // Phi'
    cp_async_commit();
    cp_async_wait_all();
    __syncthreads();
    const size_t NB = (size_t)nchunks * B;
    const float* Yb = rbuf;               // [chunk][B][32]
    const float* Rb = rbuf + NB * 32;     // [chunk][B][16]
    const float* Rpb = rbuf + NB * 48;    // [chunk][B][16]
    float4 nr4 = valid ? __ldg(reinterpret_cast<const float4*>(Rpb + ((size_t)(nchunks - 1) * B + rr) * 16) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int jj = 0; jj < nchunks; ++jj) {
        const int j = nchunks - 1 - jj;
        const float4* Pp = sc[jj & 1];
        const float4 r4 = nr4;
        if (j > 0) {
            sc_prefetch(sc[(jj + 1) & 1], SCall + (size_t)(j - 1) * SCF + DS * DS, DS * DS / 4);
            cp_async_commit();
            if (valid) nr4 = __ldg(reinterpret_cast<const float4*>(Rpb + ((size_t)(j - 1) * B + rr) * 16) + q);
        }
        const size_t base = (size_t)j * B + rr;
        if (valid) *(reinterpret_cast<float4*>(S + base * 32 + DS) + q) = make_float4(e4[0], e4[1], e4[2], e4[3]);
        float p[DS];
#pragma unroll
        for (int b = 0; b < DS; ++b) p[b] = dot4(Pp[b * 4 + q], e4);
        float ne[4];
        quad_reduce_scatter<DS>(p, q, ne);
        e4[0] = r4.x + ne[0]; e4[1] = r4.y + ne[1]; e4[2] = r4.z + ne[2]; e4[3] = r4.w + ne[3];
        cp_async_wait_all();
        __syncthreads();
    }
    // ---- causal states bottom up + outputs; the global loads of chunk j + 1 are issued before chunk j is computed ----
    float s4[4] = {0.f, 0.f, 0.f, 0.f};
    sc_prefetch(sc[0], SCall, SCF / 4);
    cp_async_commit();
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 n_yl0 = z4, n_yl1 = z4, n_r4 = z4, n_ev = z4;
    if (valid) {
        const float4* yp4 = reinterpret_cast<const float4*>(Yb + (size_t)rr * 32);
        n_yl0 = __ldg(yp4 + q); n_yl1 = __ldg(yp4 + 4 + q); n_r4 = __ldg(reinterpret_cast<const float4*>(Rb + (size_t)rr * 16) + q);
        n_ev = *(reinterpret_cast<const float4*>(S + (size_t)rr * 32) + 4 + q);
    }
    cp_async_wait_all();
    __syncthreads();
    for (int j = 0; j < nchunks; ++j) {
        const float4* Pm = sc[j & 1];                    // Phi
        const float4* Om = Pm + 2 * DS * DS / 4;         // O
        const float4* Opm = Om + PO * DS / 4;            // O'
        const float4 yl0 = n_yl0, yl1 = n_yl1, r4 = n_r4, ev = n_ev;
        if (j + 1 < nchunks) {
            sc_prefetch(sc[(j + 1) & 1], SCall + (size_t)(j + 1) * SCF, SCF / 4);
            cp_async_commit();
            if (valid) {
                const size_t nb = (size_t)(j + 1) * B + rr;
                const float4* yp4 = reinterpret_cast<const float4*>(Yb + nb * 32);
                n_yl0 = __ldg(yp4 + q); n_yl1 = __ldg(yp4 + 4 + q); n_r4 = __ldg(reinterpret_cast<const float4*>(Rb + nb * 16) + q);
                n_ev = *(reinterpret_cast<const float4*>(S + nb * 32) + 4 + q);
            }
        }
        const sn_sss_tc_chunk c = chunks[j];
        if (valid) *(reinterpret_cast<float4*>(S + ((size_t)j * B + rr) * 32) + q) = make_float4(s4[0], s4[1], s4[2], s4[3]);
        e4[0] = ev.x; e4[1] = ev.y; e4[2] = ev.z; e4[3] = ev.w;
        // outputs in two halves of 16 columns: thread q ends up with columns 16 h + 4 q .. + 3
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float py[DS];
#pragma unroll
            for (int cc = 0; cc < DS; ++cc) py[cc] = dot4(Om[(16 * h + cc) * 4 + q], s4) + dot4(Opm[(16 * h + cc) * 4 + q], e4);
            float y4[4];
            quad_reduce_scatter<DS>(py, q, y4);
            const float4 yl = h ? yl1 : yl0;
            y4[0] += yl.x; y4[1] += yl.y; y4[2] += yl.z; y4[3] += yl.w;
            const int c0 = 16 * h + 4 * q;
            if (valid && c0 < c.nrows) {
                float* yp = y + row * ldy + c.row0 + c0;
                const float* bp = bias != nullptr ? bias + c.row0 + c0 : nullptr;
                if (aligned && c0 + 4 <= c.nrows) {
                    float4 b4 = z4;
                    if (bp != nullptr) b4 = __ldg(reinterpret_cast<const float4*>(bp));
                    *reinterpret_cast<float4*>(yp) = make_float4(y4[0] + b4.x, y4[1] + b4.y, y4[2] + b4.z, y4[3] + b4.w);
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (c0 + i < c.nrows) yp[i] = y4[i] + (bp != nullptr ? __ldg(bp + i) : 0.f);
                }
            }
        }
        float p[DS];
#pragma unroll
        for (int b = 0; b < DS; ++b) p[b] = dot4(Pm[b * 4 + q], s4);
        float ns[4];
        quad_reduce_scatter<DS>(p, q, ns);
        s4[0] = r4.x + ns[0]; s4[1] = r4.y + ns[1]; s4[2] = r4.z + ns[2]; s4[3] = r4.w + ns[3];
        cp_async_wait_all();
        __syncthreads();
    }
}

// Small-batch variant of the forward scans: the two state chains are independent of each other (only the OUTPUTS need both), so
// they run as the two halves of one grid (blockIdx.y = direction, 32 serial iterations of a 16 x 16 product each), and the outputs
// y_j = yloc_j + O_j s_j + O'_j e_{j+1} + b follow in a kernel that is parallel over (sample, chunk).  Half the serial depth of
// sss_tc_scan_fwd_q_kernel and a third of its work inside the chains.
__global__ void __launch_bounds__(QS_THREADS)
sss_tc_scan_states_q_kernel(int nchunks, const float* __restrict__ SCall, const float* __restrict__ rbuf, float* __restrict__ S, long B) {
    __shared__ float4 sc[2][DS * DS / 4];
    const int q = threadIdx.x & 3, dir = blockIdx.y;
    const long row = (long)blockIdx.x * (blockDim.x / 4) + (threadIdx.x >> 2);
    const bool valid = row < B;
    const long rr = valid ? row : 0;
    const size_t NB = (size_t)nchunks * B;
    const float* Rin = rbuf + NB * 32 + (dir ? NB * 16 : 0);     // r (causal) or r' (anticausal) rows, [chunk][B][16]
    const int phi_off = dir * DS * DS;
    auto chunk_at = [&](int jj) { return dir ? nchunks - 1 - jj : jj; };
    float st4[4] = {0.f, 0.f, 0.f, 0.f};
    sc_prefetch(sc[0], SCall + (size_t)chunk_at(0) * SCF + phi_off, DS * DS / 4);
    cp_async_commit();
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 nr4 = valid ? __ldg(reinterpret_cast<const float4*>(Rin + ((size_t)chunk_at(0) * B + rr) * 16) + q) : z4;
    cp_async_wait_all();
    __syncthreads();
    for (int jj = 0; jj < nchunks; ++jj) {
        const int j = chunk_at(jj);
        const float4* Pm = sc[jj & 1];
        const float4 r4 = nr4;
        if (jj + 1 < nchunks) {
            const int jn = chunk_at(jj + 1);
            sc_prefetch(sc[(jj + 1) & 1], SCall + (size_t)jn * SCF + phi_off, DS * DS / 4);
            cp_async_commit();
            if (valid) nr4 = __ldg(reinterpret_cast<const float4*>(Rin + ((size_t)jn * B + rr) * 16) + q);
        }
        if (valid) *(reinterpret_cast<float4*>(S + ((size_t)j * B + rr) * 32 + (dir ? DS : 0)) + q) = make_float4(st4[0], st4[1], st4[2], st4[3]);
        float p[DS];
#pragma unroll
        for (int b = 0; b < DS; ++b) p[b] = dot4(Pm[b * 4 + q], st4);
        float ns[4];
        quad_reduce_scatter<DS>(p, q, ns);
        st4[0] = r4.x + ns[0]; st4[1] = r4.y + ns[1]; st4[2] = r4.z + ns[2]; st4[3] = r4.w + ns[3];
        cp_async_wait_all();
        __syncthreads();
    }
}

// grid (ceil(B / 32), nchunks), 128 threads = 32 samples x 4: the chunk's O and O' in shared memory
__global__ void __launch_bounds__(QS_THREADS)
sss_tc_scan_out_q_kernel(const sn_sss_tc_chunk* __restrict__ chunks, const float* __restrict__ SCall, const float* __restrict__ rbuf,
                         const float* __restrict__ S, float* __restrict__ y, long ldy, const float* __restrict__ bias, long B, int aligned) {
    __shared__ float4 sc[2 * PO * DS / 4];
    const int j = blockIdx.y, q = threadIdx.x & 3;
    const sn_sss_tc_chunk c = chunks[j];
    for (int i = threadIdx.x; i < 2 * PO * DS / 4; i += QS_THREADS) sc[i] = __ldg(reinterpret_cast<const float4*>(SCall + (size_t)j * SCF + 2 * DS * DS) + i);
    __syncthreads();
    const float4* Om = sc;
    const float4* Opm = sc + PO * DS / 4;
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    {
        const long row = (long)blockIdx.x * (QS_THREADS / 4) + (threadIdx.x >> 2);
        if (row >= B) return;   // whole quads leave together
        const size_t base = (size_t)j * B + row;
        const float4* sp = reinterpret_cast<const float4*>(S + base * 32);
        const float4 sv = __ldg(sp + q), ev = __ldg(sp + 4 + q);
        const float4* yp4 = reinterpret_cast<const float4*>(rbuf + base * 32);
        const float4 yl0 = __ldg(yp4 + q), yl1 = __ldg(yp4 + 4 + q);
        const float s4[4] = {sv.x, sv.y, sv.z, sv.w}, e4[4] = {ev.x, ev.y, ev.z, ev.w};
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float py[DS];
#pragma unroll
            for (int cc = 0; cc < DS; ++cc) py[cc] = dot4(Om[(16 * h + cc) * 4 + q], s4) + dot4(Opm[(16 * h + cc) * 4 + q], e4);
            float y4[4];
            quad_reduce_scatter<DS>(py, q, y4);
            const float4 yl = h ? yl1 : yl0;
            y4[0] += yl.x; y4[1] += yl.y; y4[2] += yl.z; y4[3] += yl.w;
            const int c0 = 16 * h + 4 * q;
            if (c0 < c.nrows) {
                float* yo = y + row * ldy + c.row0 + c0;
                const float* bp = bias != nullptr ? bias + c.row0 + c0 : nullptr;
                if (aligned && c0 + 4 <= c.nrows) {
                    float4 b4 = z4;
                    if (bp != nullptr) b4 = __ldg(reinterpret_cast<const float4*>(bp));
                    *reinterpret_cast<float4*>(yo) = make_float4(y4[0] + b4.x, y4[1] + b4.y, y4[2] + b4.z, y4[3] + b4.w);
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (c0 + i < c.nrows) yo[i] = y4[i] + (bp != nullptr ? __ldg(bp + i) : 0.f);
                }
            }
        }
    }
}

// adjoint scans.  L[j][row][0..15] = lambda_{j+1} (adjoint of the causal state leaving chunk j), L[j][row][16..31] = mu_j (adjoint of
// the anticausal state leaving chunk j); grad_bias += column sums of grad_y.
// padded coefficient layout of the adjoint scans: thread q reads rows 4q.. of Phi and 8q.. of O, so every group of 4 (8) rows is
// followed by one float4 of padding -- the four quads' rows then start 16 bytes apart modulo 128 (conflict-free LDS.128)
constexpr int QB_PHI = 4 * 17, QB_O = 4 * 33, QB_TOTAL = QB_PHI + QB_O;
__device__ __forceinline__ void sc_prefetch_padded(float4* dst, const float* __restrict__ src, int nfloat4, int group) {
    for (int i = threadIdx.x; i < nfloat4; i += blockDim.x) cp_async16(dst + (i / group) * (group + 1) + (i % group), reinterpret_cast<const float4*>(src) + i);
}

template <bool MU>
__device__ __forceinline__ void scan_bwd_pass(float4 (*sc)[QB_TOTAL], float* sbias, const sn_sss_tc_chunk* __restrict__ chunks, int nchunks,
                                              const float* __restrict__ SCall, const float* __restrict__ gy, long ldgy, float* __restrict__ L,
                                              float* __restrict__ gbias, long B, int aligned, int q, long row, bool valid) {
    const int lane = threadIdx.x & 31;
    const int phi_off = MU ? DS * DS : 0, o_off = 2 * DS * DS + (MU ? PO * DS : 0);
    auto prefetch = [&](int buf, int j) {
        sc_prefetch_padded(sc[buf], SCall + (size_t)j * SCF + phi_off, DS * DS / 4, 16);
        sc_prefetch_padded(sc[buf] + QB_PHI, SCall + (size_t)j * SCF + o_off, PO * DS / 4, 32);
        cp_async_commit();
    };
    float a4[4] = {0.f, 0.f, 0.f, 0.f};
    prefetch(0, MU ? 0 : nchunks - 1);
    cp_async_wait_all();
    __syncthreads();
    int prev_row0 = 0, prev_nrows = 0;
    for (int jj = 0; jj < nchunks; ++jj) {
        const int j = MU ? jj : nchunks - 1 - jj;
        const float4* Pm = sc[jj & 1] + 17 * q;           // this thread's 4 rows of Phi
        const float4* Om = sc[jj & 1] + QB_PHI + 33 * q;  // this thread's 8 rows of O
        if (jj + 1 < nchunks) prefetch((jj + 1) & 1, MU ? j + 1 : j - 1);
        const sn_sss_tc_chunk c = chunks[j];
        if (MU && gbias != nullptr && jj > 0 && threadIdx.x < 32) {   // flush the previous chunk's column sums
            float* sb = sbias + ((jj - 1) & 1) * 32;
            if ((int)threadIdx.x < prev_nrows) atomicAdd(gbias + prev_row0 + threadIdx.x, sb[threadIdx.x]);
            sb[threadIdx.x] = 0.f;
        }
        float g8[8];
        {
            const float* src = gy + (valid ? row : 0) * ldgy + c.row0 + 8 * q;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int c0 = 8 * q + 4 * h;
                if (valid && aligned && c0 + 4 <= c.nrows) {
                    const float4 v = __ldg(reinterpret_cast<const float4*>(src + 4 * h));
                    g8[4 * h] = v.x; g8[4 * h + 1] = v.y; g8[4 * h + 2] = v.z; g8[4 * h + 3] = v.w;
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i) g8[4 * h + i] = (valid && c0 + i < c.nrows) ? __ldg(src + 4 * h + i) : 0.f;
                }
            }
        }
        if (valid) *(reinterpret_cast<float4*>(L + ((size_t)j * B + row) * 32 + (MU ? DS : 0)) + q) = make_float4(a4[0], a4[1], a4[2], a4[3]);
        float p[DS];
#pragma unroll
        for (int a = 0; a < DS; ++a) p[a] = 0.f;
#pragma unroll
        for (int bi = 0; bi < 4; ++bi) axpy16(Pm + bi * 4, a4[bi], p);        // Phi[4q + bi][:] * adjoint[4q + bi]
#pragma unroll
        for (int ci = 0; ci < 8; ++ci) axpy16(Om + ci * 4, g8[ci], p);        // O[8q + ci][:] * gy[8q + ci]
        quad_reduce_scatter<DS>(p, q, a4);
        if (MU && gbias != nullptr) {
            // column sums over the warp's 8 samples (lanes with the same q): transposed reduce over lane bits 4, 3, 2
            float h4[4], h2[2];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const bool up = (lane & 16) != 0;
                h4[i] = (up ? g8[4 + i] : g8[i]) + __shfl_xor_sync(0xffffffffu, up ? g8[i] : g8[4 + i], 16);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const bool up = (lane & 8) != 0;
                h2[i] = (up ? h4[2 + i] : h4[i]) + __shfl_xor_sync(0xffffffffu, up ? h4[i] : h4[2 + i], 8);
            }
            const bool up = (lane & 4) != 0;
            const float colsum = (up ? h2[1] : h2[0]) + __shfl_xor_sync(0xffffffffu, up ? h2[0] : h2[1], 4);
            const int colid = 8 * q + ((lane & 16) ? 4 : 0) + ((lane & 8) ? 2 : 0) + ((lane & 4) ? 1 : 0);
            atomicAdd(sbias + (jj & 1) * 32 + colid, colsum);
        }
        prev_row0 = c.row0;
        prev_nrows = c.nrows;
        cp_async_wait_all();
        __syncthreads();
    }
    if (MU && gbias != nullptr && threadIdx.x < 32) {
        float* sb = sbias + ((nchunks - 1) & 1) * 32;
        if ((int)threadIdx.x < prev_nrows) atomicAdd(gbias + prev_row0 + threadIdx.x, sb[threadIdx.x]);
    }
}

__global__ void __launch_bounds__(QS_THREADS)
sss_tc_scan_bwd_q_kernel(const sn_sss_tc_chunk* __restrict__ chunks, int nchunks, const float* __restrict__ SCall, const float* __restrict__ gy,
                         long ldgy, float* __restrict__ L, float* __restrict__ gbias, long B, int aligned) {
    __shared__ float4 sc[2][QB_TOTAL];
    __shared__ float sbias[64];
    if (threadIdx.x < 64) sbias[threadIdx.x] = 0.f;
    const int q = threadIdx.x & 3;
    const long row = (long)blockIdx.x * (blockDim.x / 4) + (threadIdx.x >> 2);
    const bool valid = row < B;
    // gridDim.y == 2: one direction per CTA (half the serial depth; small batches); gridDim.y == 1: both, one after the other
    if (gridDim.y == 1 || blockIdx.y == 0) scan_bwd_pass<false>(sc, sbias, chunks, nchunks, SCall, gy, ldgy, L, gbias, B, aligned, q, row, valid);
    if (gridDim.y == 1 || blockIdx.y == 1) scan_bwd_pass<true>(sc, sbias, chunks, nchunks, SCall, gy, ldgy, L, gbias, B, aligned, q, row, valid);
}

// ------------------------------------------------------------------------------------------
// 3m/4m. chunk scans on the warp-level tensor cores (mma.sync m16n8k8 tf32, 3xTF32): the default scans at every batch size.  The
//    four-threads-per-sample scans above are instruction-bound (ncu at 8 192 samples: 219 warp instructions per chunk step and 8
//    samples for 64 useful FFMA issues).  Here a warp owns 16 samples and keeps their state as the D fragment of a 16 x 16 tile; a step is
//        state' = r + state Phi^T      (r is the accumulator's initial value, the previous D fragment is the next A fragment --
//                                       same register chaining as the build kernel, no shuffle, no shared-memory round trip)
//    The chunk's B fragments (packed once per forward, sss_tc_pack_scan_kernel) and the warp's per-sample rows arrive through cp.async
//    rings in shared memory.  Requires the 16-byte aligned layouts (`aligned`); otherwise the SIMT scans or the tcgen05 chain run.
// ------------------------------------------------------------------------------------------
constexpr int QG_S = 8;                     // cp.async ring depth (steps in flight) of the state scans
constexpr int SM_THREADS = 128;             // 4 warps x 16 samples
template <int N>
__device__ __forceinline__ void cp_async_wait_n() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// A fragment with the K index permuted like split_frag's (logical k = t <-> physical column 2t, k = t + 4 <-> 2t + 1 of the group of 8),
// from two consecutive floats of rows g and g + 8
__device__ __forceinline__ void frag_a_from(const float2 row_a, const float2 row_b, Frag3& f) {
    const float v[4] = {row_a.x, row_b.x, row_a.y, row_b.y};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float h = tf32_hi(v[i]);
        f.hi[i] = __float_as_uint(h);
        f.lo[i] = __float_as_uint(mma_lo(v[i] - h));
    }
}

// ---- warp-level tensor-core scans: layouts ----
// The scans are bound by the L1 / shared-memory data pipe (ncu r2v: 84 % of its peak in the adjoint scan): one wavefront per 128-byte
// line a warp instruction touches.  With the m16n8k8 fragments loaded as they are defined (lane (g, t) holds columns 2t, 2t+1 of rows
// g, g+8) every global access is 8 bytes per lane over 8 rows: 8 wavefronts for 256 bytes.  Samples are independent and the order of the
// state components / output rows inside a product is free as long as both operands agree, so the kernels below let lane t own FOUR
// consecutive floats of a row (one 16-byte access: half the wavefronts per byte) and fold the resulting permutations into the packed
// B fragments:
//   state rows (16 floats: S, L, r):  lane t holds physical components 4t .. 4t+3 = logical (n-tile 0: 2t, 2t+1 | n-tile 1: 2t, 2t+1)
//   32-wide rows (grad_y, [s | e], yloc, y): lane t holds 4t .. 4t+3 and 16+4t .. 16+4t+3 = (k-step or n-tile 0 | 1 | 2 | 3) x 2
__device__ __forceinline__ int pstate(int l) { return 4 * ((l & 7) >> 1) + 2 * (l >> 3) + (l & 1); }            // logical state index -> physical
__device__ __forceinline__ int p32(int blk, int t, int e) { return 16 * (blk >> 1) + 4 * t + 2 * (blk & 1) + e; }  // (block of 8, lane t, e) -> physical

// fragment tiles FS[chunk][direction] = 16 B fragments x 32 lanes x (x0, x1), packed once per forward by sss_tc_pack_scan_kernel: a scan
// step reads a B fragment with one conflict-free 8-byte shared-memory load.  Lane (g, t) of fragment (n-tile nt, k-step ks) holds
// B[k = (ks, t)][n = 8 nt + g] and B[k = (ks, t + 4)][n].
//   0..3    state scans     2 nt + ks      B[k][n] = Phi[n][k]
//   4..7    adjoint scans   4 + 2 nt + ks  B[k][n] = Phi[k][n]           (Phi^T lambda)
//   8..15   adjoint scans   8 + 4 nt + ks  B[k][n] = O[k][n], k < 32     (O^T gy)
constexpr int FS_FRAGS = 16;
constexpr int FS_TILE_FLOATS = FS_FRAGS * 32 * 2;     // 1024 floats = 4 KB per (chunk, direction)
__global__ void __launch_bounds__(256)
sss_tc_pack_scan_kernel(const float* __restrict__ SCall, float* __restrict__ FSall) {
    const int ch = blockIdx.x, dir = blockIdx.y;
    const float* Phi = SCall + (size_t)ch * SCF + dir * DS * DS;
    const float* O = SCall + (size_t)ch * SCF + 2 * DS * DS + dir * PO * DS;
    float2* FS = reinterpret_cast<float2*>(FSall + ((size_t)ch * 2 + dir) * FS_TILE_FLOATS);
    for (int i = threadIdx.x; i < FS_FRAGS * 32; i += 256) {
        const int f = i >> 5, lane = i & 31, g = lane >> 2, t = lane & 3;
        float x0, x1;
        if (f < 8) {
            const int nt = (f & 3) >> 1, ks = f & 1;
            const int n = pstate(8 * nt + g), k0 = pstate(8 * ks + 2 * t), k1 = pstate(8 * ks + 2 * t + 1);
            if (f < 4) { x0 = Phi[n * DS + k0]; x1 = Phi[n * DS + k1]; }
            else       { x0 = Phi[k0 * DS + n]; x1 = Phi[k1 * DS + n]; }
        } else {
            const int nt = (f - 8) >> 2, ks = (f - 8) & 3, n = pstate(8 * nt + g);
            x0 = O[p32(ks, t, 0) * DS + n]; x1 = O[p32(ks, t, 1) * DS + n];
        }
        FS[i] = make_float2(x0, x1);
    }
}
// 16-byte cp.async that reads only `bytes` (0..16) from global memory and zero-fills the rest
__device__ __forceinline__ void cp_async16_zfill(float* dst, const float* src, int bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes) : "memory");
}
// packed B fragment -> (hi.x, hi.y, lo.x, lo.y)
__device__ __forceinline__ float4 split_b(const float2 x) {
    const float h0 = tf32_hi(x.x), h1 = tf32_hi(x.y);
    return make_float4(h0, h1, mma_lo(x.x - h0), mma_lo(x.y - h1));
}
// one of the three terms of d += A B (0: lo * hi, 1: hi * lo, 2: hi * hi; small terms first).  The scans issue the terms of several
// INDEPENDENT accumulators round-robin: an HMMA that adds into the accumulator of its predecessor waits ~27 cycles for it.
template <int TERM>
__device__ __forceinline__ void mma_term(float (&d)[4], const Frag3& a, const float4 b) {
    if (TERM == 0) mma_1688(d, a.lo, __float_as_uint(b.x), __float_as_uint(b.y));
    else if (TERM == 1) mma_1688(d, a.hi, __float_as_uint(b.z), __float_as_uint(b.w));
    else mma_1688(d, a.hi, __float_as_uint(b.x), __float_as_uint(b.y));
}
// A fragments of two k-steps from one float4 per row (rows g and g + 8): k-step 0 <- (x, y), k-step 1 <- (z, w)
__device__ __forceinline__ void frag_a2(const float4 ra, const float4 rb, Frag3& f0, Frag3& f1) {
    frag_a_from(make_float2(ra.x, ra.y), make_float2(rb.x, rb.y), f0);
    frag_a_from(make_float2(ra.z, ra.w), make_float2(rb.z, rb.w), f1);
}

// forward state chains: blockIdx.y = direction (0: s_{j+1} = r_j + Phi_j s_j ascending, 1: e_j = r'_j + Phi'_j e_{j+1} descending);
// saves the state ENTERING every chunk: S[j][row][0..15] = s_j, S[j][row][16..31] = e_{j+1}
__global__ void __launch_bounds__(SM_THREADS)
sss_tc_scan_states_m_kernel(int nchunks, const float* __restrict__ FSall, const float* __restrict__ rbuf, float* __restrict__ S, long B) {
    // rings of QG_S steps: the chunk's four B fragments (shared by the CTA) and, per warp, the step's 16 r rows.  The per-sample rows
    // are staged by cp.async and not by loads into a register ring: a warp has six scoreboards, the compiler folds the ring's loads
    // onto them together with everything else of the step, and an unrelated register write then waits for the youngest load of the
    // group (ncu r2zc: a quarter of the adjoint scan's samples on one CS2R) -- the ring never had its nominal depth.
    __shared__ __align__(16) float2 sc[QG_S][4 * 32];
    __shared__ __align__(16) float rows[SM_THREADS / 32][QG_S][16 * 16];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3, dir = blockIdx.y;
    const long row0 = ((long)blockIdx.x * (SM_THREADS / 32) + warp) * 16;
    const long rowa = row0 + g, rowb = row0 + g + 8;
    const bool va = rowa < B, vb = rowb < B;
    const size_t NB = (size_t)nchunks * B;
    const float* Rin = rbuf + NB * 32 + (dir ? NB * 16 : 0);     // r (causal) or r' (anticausal) rows, [chunk][B][16]
    auto chunk_at = [&](int jj) { return dir ? nchunks - 1 - jj : jj; };
    auto issue = [&](int jj) {
        if (jj < nchunks) {
            const int ch = chunk_at(jj);
            if (threadIdx.x < 64) cp_async16(reinterpret_cast<float*>(sc[jj % QG_S]) + 4 * threadIdx.x, FSall + ((size_t)ch * 2 + dir) * FS_TILE_FLOATS + 4 * threadIdx.x);
            // the warp's 16 rows are 1 KB of contiguous global memory: two 512-byte pieces, same layout in shared memory
            float* dst = rows[warp][jj % QG_S];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int fl = 4 * lane + 128 * i;             // float offset inside the 16 x 16 block; row = fl / 16
                const bool ok = row0 + (fl >> 4) < B;
                cp_async16_zfill(dst + fl, ok ? Rin + ((size_t)ch * B + row0) * 16 + fl : Rin, ok ? 16 : 0);
            }
        }
        cp_async_commit();
    };
#pragma unroll
    for (int s0 = 0; s0 < QG_S - 1; ++s0) issue(s0);
    float d[2][4];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int k = 0; k < 4; ++k) d[nt][k] = 0.f;
#pragma unroll 2
    for (int jj = 0; jj < nchunks; ++jj) {
        cp_async_wait_n<QG_S - 2>();
        __syncthreads();
        issue(jj + QG_S - 1);
        const int j = chunk_at(jj);
        const float2* F = sc[jj % QG_S];
        const float* R = rows[warp][jj % QG_S];
        // the state entering chunk j
        if (va) *reinterpret_cast<float4*>(S + ((size_t)j * B + rowa) * 32 + (dir ? DS : 0) + 4 * t) = make_float4(d[0][0], d[0][1], d[1][0], d[1][1]);
        if (vb) *reinterpret_cast<float4*>(S + ((size_t)j * B + rowb) * 32 + (dir ? DS : 0) + 4 * t) = make_float4(d[0][2], d[0][3], d[1][2], d[1][3]);
        const float4 ra = *reinterpret_cast<const float4*>(R + g * 16 + 4 * t), rb = *reinterpret_cast<const float4*>(R + (g + 8) * 16 + 4 * t);
        Frag3 a[2];
        split_frag(d[0], a[0]);
        split_frag(d[1], a[1]);
        {   // four independent chains of three products: (n-tile, k-step); k-step 1 starts from the step's r values
            float4 f[2][2];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) f[nt][ks] = split_b(F[(2 * nt + ks) * 32 + lane]);
            float acc[2][2][4];
            acc[0][1][0] = ra.x; acc[0][1][1] = ra.y; acc[1][1][0] = ra.z; acc[1][1][1] = ra.w;
            acc[0][1][2] = rb.x; acc[0][1][3] = rb.y; acc[1][1][2] = rb.z; acc[1][1][3] = rb.w;
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) acc[nt][0][0] = acc[nt][0][1] = acc[nt][0][2] = acc[nt][0][3] = 0.f;
#define SN_ROUND(TERM)                                                                    \
            mma_term<TERM>(acc[0][0], a[0], f[0][0]); mma_term<TERM>(acc[1][0], a[0], f[1][0]); \
            mma_term<TERM>(acc[0][1], a[1], f[0][1]); mma_term<TERM>(acc[1][1], a[1], f[1][1]);
            SN_ROUND(0) SN_ROUND(1) SN_ROUND(2)
#undef SN_ROUND
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int k = 0; k < 4; ++k) d[nt][k] = acc[nt][0][k] + acc[nt][1][k];
        }
    }
    cp_async_wait_all();
}

// outputs y_j = yloc_j + O_j s_j + O'_j e_{j+1} + b, parallel over (sample, chunk): grid (ceil(B / (64 * QMO_SUB)), nchunks); a warp
// walks QMO_SUB sub-tiles of 16 samples with the chunk's 16 B fragments (K = [s | e] = 32, N = 32 outputs) split once, in registers.
constexpr int QMO_SUB = 2;
constexpr int SCAN_CTAB = 128;               // chunks whose (row0, nrows) the adjoint scan keeps in shared memory (1 KB: four CTAs of
                                             // 53 KB + this + 1 KB reserved still fit the SM's 228 KB)
__global__ void __launch_bounds__(SM_THREADS)
sss_tc_scan_out_m_kernel(const sn_sss_tc_chunk* __restrict__ chunks, const float* __restrict__ SCall, const float* __restrict__ rbuf,
                         const float* __restrict__ S, float* __restrict__ y, long ldy, const float* __restrict__ bias, long B) {
    __shared__ __align__(16) float sc[2 * PO * DS];       // O (32 x 16) then O' (32 x 16)
    const int j = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    // every global load of the CTA is issued before anything waits: the per-sample rows of ALL the warp's sub-tiles, the chunk's O / O'
    // and its descriptor.  [half: columns 4t.. / 16+4t..][row a / b]
    float4 av[QMO_SUB][2][2], yl[QMO_SUB][2][2];
#pragma unroll
    for (int u = 0; u < QMO_SUB; ++u) {
        const long row0 = (((long)blockIdx.x * QMO_SUB + u) * (SM_THREADS / 32) + warp) * 16;
        const long rowa = row0 + g, rowb = row0 + g + 8;
        const bool va = rowa < B, vb = rowb < B;
        const float* sa = S + ((size_t)j * B + rowa) * 32;
        const float* sb = S + ((size_t)j * B + rowb) * 32;
        const float* ya = rbuf + ((size_t)j * B + rowa) * 32;
        const float* yb = rbuf + ((size_t)j * B + rowb) * 32;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            av[u][h][0] = va ? __ldg(reinterpret_cast<const float4*>(sa + 16 * h + 4 * t)) : z;
            av[u][h][1] = vb ? __ldg(reinterpret_cast<const float4*>(sb + 16 * h + 4 * t)) : z;
            yl[u][h][0] = va ? __ldg(reinterpret_cast<const float4*>(ya + 16 * h + 4 * t)) : z;
            yl[u][h][1] = vb ? __ldg(reinterpret_cast<const float4*>(yb + 16 * h + 4 * t)) : z;
        }
    }
    float4 scv[2 * PO * DS / 4 / SM_THREADS];
#pragma unroll
    for (int i = 0; i < 2 * PO * DS / 4 / SM_THREADS; ++i)
        scv[i] = __ldg(reinterpret_cast<const float4*>(SCall + (size_t)j * SCF + 2 * DS * DS) + threadIdx.x + i * SM_THREADS);
    const int c_row0 = __ldg(&chunks[j].row0), c_nrows = __ldg(&chunks[j].nrows);
#pragma unroll
    for (int i = 0; i < 2 * PO * DS / 4 / SM_THREADS; ++i) reinterpret_cast<float4*>(sc)[threadIdx.x + i * SM_THREADS] = scv[i];
    // bias of the lane's 8 output columns: [half][4]
    float bs[2][4];
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int n = 16 * h + 4 * t + e;
            bs[h][e] = (bias != nullptr && n < c_nrows) ? __ldg(bias + c_row0 + n) : 0.f;
        }
    __syncthreads();
    // B fragments: k-steps 0, 1 = s (O), 2, 3 = e (O'); n-tile nt, lane g <-> output row p32(nt, g >> 1, g & 1); k-slot (ks, t, e) <-> state
    // component 4t + 2 (ks & 1) + e of s (ks < 2) or e (ks >= 2)
    float2 bh[4][4], bl[4][4];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            const float2 r = *reinterpret_cast<const float2*>(sc + (ks >> 1) * PO * DS + p32(nt, g >> 1, g & 1) * DS + 4 * t + 2 * (ks & 1));
            bh[ks][nt].x = tf32_hi(r.x); bh[ks][nt].y = tf32_hi(r.y);
            bl[ks][nt].x = mma_lo(r.x - bh[ks][nt].x); bl[ks][nt].y = mma_lo(r.y - bh[ks][nt].y);
        }
    const bool vec_ok = (c_nrows & 3) == 0;
#pragma unroll
    for (int u = 0; u < QMO_SUB; ++u) {
        const long row0 = (((long)blockIdx.x * QMO_SUB + u) * (SM_THREADS / 32) + warp) * 16;
        const long rowa = row0 + g, rowb = row0 + g + 8;
        const bool va = rowa < B, vb = rowb < B;
        Frag3 a[4];
        frag_a2(av[u][0][0], av[u][0][1], a[0], a[1]);
        frag_a2(av[u][1][0], av[u][1][1], a[2], a[3]);
        float acc[4][4];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            acc[2 * h][0] = yl[u][h][0].x + bs[h][0]; acc[2 * h][1] = yl[u][h][0].y + bs[h][1];
            acc[2 * h][2] = yl[u][h][1].x + bs[h][0]; acc[2 * h][3] = yl[u][h][1].y + bs[h][1];
            acc[2 * h + 1][0] = yl[u][h][0].z + bs[h][2]; acc[2 * h + 1][1] = yl[u][h][0].w + bs[h][3];
            acc[2 * h + 1][2] = yl[u][h][1].z + bs[h][2]; acc[2 * h + 1][3] = yl[u][h][1].w + bs[h][3];
        }
#pragma unroll
        for (int ks = 0; ks < 4; ++ks)
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) mma3(acc[nt], a[ks], bh[ks][nt], bl[ks][nt]);      // four independent accumulators per k-step
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int n0 = 16 * h + 4 * t;
            const float4 oa = make_float4(acc[2 * h][0], acc[2 * h][1], acc[2 * h + 1][0], acc[2 * h + 1][1]);
            const float4 ob = make_float4(acc[2 * h][2], acc[2 * h][3], acc[2 * h + 1][2], acc[2 * h + 1][3]);
            if (n0 + 4 <= c_nrows && vec_ok) {
                if (va) *reinterpret_cast<float4*>(y + rowa * ldy + c_row0 + n0) = oa;
                if (vb) *reinterpret_cast<float4*>(y + rowb * ldy + c_row0 + n0) = ob;
            } else {
                const float oav[4] = {oa.x, oa.y, oa.z, oa.w}, obv[4] = {ob.x, ob.y, ob.z, ob.w};
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (n0 + e < c_nrows) {
                        if (va) y[rowa * ldy + c_row0 + n0 + e] = oav[e];
                        if (vb) y[rowb * ldy + c_row0 + n0 + e] = obv[e];
                    }
            }
        }
    }
}

// adjoint chains: blockIdx.y = 0: lambda_j = Phi_j^T lambda_{j+1} + O_j^T gy_j (descending), 1: mu likewise with Phi', O' (ascending).
// L[j][row][0..15] = lambda_{j+1}, L[j][row][16..31] = mu_j: the adjoint of the state LEAVING chunk j, i.e. the value before the step.
constexpr int GROW = 48;                                  // floats per staged grad_y row: 32 + 16 of padding (conflict-free 16-byte reads)
constexpr int SB_FRAG_FLOATS = 12 * 32 * 2;              // fragments 4..15 of a tile
constexpr size_t sb_smem_bytes(int qg) { return (size_t)qg * (SB_FRAG_FLOATS + (SM_THREADS / 32) * 16 * GROW) * sizeof(float); }
// QG_B = ring depth (steps in flight): 6 when the whole batch is one wave of CTAs at two per SM (the ring hides the memory latency), 3
// above that (46 KB per CTA: four CTAs per SM hide it instead; at 65 536 samples the deep ring ran at 12 % occupancy, 47 % issue slots)
template <int QG_B>
__global__ void __launch_bounds__(SM_THREADS)
sss_tc_scan_bwd_m_kernel(const sn_sss_tc_chunk* __restrict__ chunks, int nchunks, const float* __restrict__ FSall, const float* __restrict__ gy,
                         long ldgy, float* __restrict__ L, float* __restrict__ grad_bias, long B) {
    // rings of QG_B steps in dynamic shared memory: fragments 4..15 of the chunk's tile (shared by the CTA), and per warp the chunk's
    // 32 grad_y columns of its 16 samples (see the state scans for why these are not a register ring)
    extern __shared__ __align__(16) float sb_smem[];
    float* frag_ring = sb_smem;                                           // [QG_B][SB_FRAG_FLOATS]
    float* row_ring = sb_smem + (size_t)QG_B * SB_FRAG_FLOATS;            // [warp][QG_B][16][GROW]
    // grad_bias (may be NULL): the column sums of grad_y come from the rows this kernel stages anyway -- direction mu sums the chunks
    // of its own parity.  A warp meets every chunk exactly once, so its sums go to a slot of its own, [warp][chunk / 2][32], with a plain
    // store (shared-memory atomics of four warps on the same 32 words held 10 % of the kernel's samples at 65 536 samples); one
    // global reduction per (chunk, column) and CTA at the end.
    float* bsum = row_ring + (size_t)(SM_THREADS / 32) * QG_B * 16 * GROW;
    const int nhalf = (nchunks + 1) >> 1;
    __shared__ int2 ctab[SCAN_CTAB];       // (row0, nrows) per chunk: the grad_y addresses must not wait on a load of the chunk table
    for (int i = threadIdx.x; i < nchunks && i < SCAN_CTAB; i += SM_THREADS) ctab[i] = make_int2(chunks[i].row0, chunks[i].nrows);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3, mu = blockIdx.x;   // direction fastest: the two CTAs that read the
    // same grad_y rows (once per direction) are launched next to each other, and the second read comes from L2
    const long row0 = ((long)blockIdx.y * (SM_THREADS / 32) + warp) * 16;
    const long rowa = row0 + g, rowb = row0 + g + 8;
    const bool va = rowa < B, vb = rowb < B;
    float* my_rows = row_ring + (size_t)warp * QG_B * 16 * GROW;
    auto chunk_at = [&](int jj) { return mu ? jj : nchunks - 1 - jj; };
    auto issue = [&](int jj) {
        if (jj < nchunks) {
            const int ch = chunk_at(jj);
            const float* src = FSall + ((size_t)ch * 2 + mu) * FS_TILE_FLOATS + 4 * 32 * 2;
            float* dst = frag_ring + (size_t)(jj % QG_B) * SB_FRAG_FLOATS;
            cp_async16(dst + 4 * threadIdx.x, src + 4 * threadIdx.x);
            if (threadIdx.x < 64) cp_async16(dst + 4 * (threadIdx.x + SM_THREADS), src + 4 * (threadIdx.x + SM_THREADS));
            // grad_y: lane -> (row = 4 i + lane / 8, 16-byte piece = lane % 8): every instruction reads four whole 128-byte rows;
            // bytes past the chunk's nrows and rows past B are zero-filled, never read
            const int2 c = ch < SCAN_CTAB ? ctab[ch] : make_int2(__ldg(&chunks[ch].row0), __ldg(&chunks[ch].nrows));
            float* rdst = my_rows + (size_t)(jj % QG_B) * 16 * GROW;
            const int piece = lane & 7;
            int bytes = 4 * (c.y - 4 * piece);
            bytes = bytes < 0 ? 0 : (bytes > 16 ? 16 : bytes);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = 4 * i + (lane >> 3);
                const bool ok = row0 + r < B && bytes > 0;
                cp_async16_zfill(rdst + r * GROW + 4 * piece, ok ? gy + (row0 + r) * ldgy + c.x + 4 * piece : gy, ok ? bytes : 0);
            }
        }
        cp_async_commit();
    };
#pragma unroll
    for (int s0 = 0; s0 < QG_B - 1; ++s0) issue(s0);
    float d[2][4];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int k = 0; k < 4; ++k) d[nt][k] = 0.f;
#pragma unroll 2
    for (int jj = 0; jj < nchunks; ++jj) {
        cp_async_wait_n<QG_B - 2>();
        __syncthreads();
        issue(jj + QG_B - 1);
        const int j = chunk_at(jj);
        const float2* F = reinterpret_cast<const float2*>(frag_ring + (size_t)(jj % QG_B) * SB_FRAG_FLOATS);
        const float* G = my_rows + (size_t)(jj % QG_B) * 16 * GROW;
        if (va) *reinterpret_cast<float4*>(L + ((size_t)j * B + rowa) * 32 + (mu ? DS : 0) + 4 * t) = make_float4(d[0][0], d[0][1], d[1][0], d[1][1]);
        if (vb) *reinterpret_cast<float4*>(L + ((size_t)j * B + rowb) * 32 + (mu ? DS : 0) + 4 * t) = make_float4(d[0][2], d[0][3], d[1][2], d[1][3]);
        if (grad_bias != nullptr && (j & 1) == mu) {      // lane = column of the chunk; rows past B and columns past nrows are staged as zeros
            float cs = 0.f;
#pragma unroll
            for (int r = 0; r < 16; ++r) cs += G[r * GROW + lane];
            bsum[((size_t)(threadIdx.x >> 5) * nhalf + (j >> 1)) * 32 + lane] = cs;
        }
        Frag3 a[2], ag[4];
#pragma unroll
        for (int h = 0; h < 2; ++h)
            frag_a2(*reinterpret_cast<const float4*>(G + g * GROW + 16 * h + 4 * t), *reinterpret_cast<const float4*>(G + (g + 8) * GROW + 16 * h + 4 * t), ag[2 * h], ag[2 * h + 1]);
        split_frag(d[0], a[0]);
        split_frag(d[1], a[1]);
        {   // per n-tile three independent chains of six products: O^T gy over k-steps (0, 1) and (2, 3), Phi^T over the state's two.
            // The O^T gy chains do not depend on the previous step at all, so only the six Phi^T products sit on the recurrence.
            float4 fo[2][4], fp[2][2];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) fo[nt][ks] = split_b(F[(4 + 4 * nt + ks) * 32 + lane]);     // O^T gy
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) fp[nt][ks] = split_b(F[(2 * nt + ks) * 32 + lane]);         // Phi^T adjoint
            }
            float acc[2][3][4];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int c = 0; c < 3; ++c)
#pragma unroll
                    for (int k = 0; k < 4; ++k) acc[nt][c][k] = 0.f;
#define SN_ROUND(TERM, KS)                                                                                                  \
            mma_term<TERM>(acc[0][0], ag[KS], fo[0][KS]);         mma_term<TERM>(acc[1][0], ag[KS], fo[1][KS]);         \
            mma_term<TERM>(acc[0][1], ag[2 + KS], fo[0][2 + KS]); mma_term<TERM>(acc[1][1], ag[2 + KS], fo[1][2 + KS]); \
            mma_term<TERM>(acc[0][2], a[KS], fp[0][KS]);          mma_term<TERM>(acc[1][2], a[KS], fp[1][KS]);
            SN_ROUND(0, 0) SN_ROUND(1, 0) SN_ROUND(2, 0) SN_ROUND(0, 1) SN_ROUND(1, 1) SN_ROUND(2, 1)
#undef SN_ROUND
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int k = 0; k < 4; ++k) d[nt][k] = (acc[nt][0][k] + acc[nt][1][k]) + acc[nt][2][k];
        }
    }
    cp_async_wait_all();
    if (grad_bias != nullptr) {
        __syncthreads();
        for (int i = threadIdx.x; i < nhalf * 32; i += SM_THREADS) {
            const int j = 2 * (i >> 5) + mu, col = i & 31;
            if (j >= nchunks) continue;
            const int2 c = j < SCAN_CTAB ? ctab[j] : make_int2(__ldg(&chunks[j].row0), __ldg(&chunks[j].nrows));
            float sum = 0.f;
#pragma unroll
            for (int w = 0; w < SM_THREADS / 32; ++w) sum += bsum[(size_t)w * nhalf * 32 + i];
            if (col < c.y) atomicAdd(grad_bias + c.x + col, sum);
        }
    }
}

// ------------------------------------------------------------------------------------------
// 3''/4''. chunk scans on the tensor core.  A scan step is state' = in + M state with a 16 x 16 (plus output rows) matrix per
//    chunk -- serial in the chunk index, but for 128 samples at once it is one tiny UMMA: A = the tile's state vectors
//    [128 x (hi 16 | lo 16)] written to shared memory by the epilogue threads (thread = sample), B = the chunk's packed, pre-split
//    coefficient tile (TMA), D in TMEM.  The chain  MMA -> TMEM -> registers -> shared memory -> MMA  costs about a microsecond
//    per step; several CTAs per SM overlap their chains.  Per-sample global traffic (r, yloc, grad_y rows) is prefetched one step
//    ahead, off the chain.
//    Coefficient tiles CW[chunk][kind] (96 rows x 32 floats, K-major, SWIZZLE_128B by TMA), kind 0/1 = forward causal/anticausal:
//       rows n < 48: [Whi(n,:) | Whi(n,:)], rows 48 + n: [Wlo(n,:) | 0], W = [O ; Phi] (48 x 16)   -> D[:, n] + D[:, 48 + n]
//    kind 2/3 = backward lambda/mu, three 32-row sub-tiles: state (Phi^T), grad_y hi part (O^T), grad_y lo part (O^T).
// ------------------------------------------------------------------------------------------
#ifndef SN_CH_PF
#define SN_CH_PF 1
#endif
constexpr int CH_PF = SN_CH_PF;                  // L2 prefetch distance (steps) of the per-sample rows
constexpr int CW_ROWS = 96;
constexpr int CW_TILE_FLOATS = CW_ROWS * 32;    // 3072 floats = 12 KB
constexpr int CW_TILE_BYTES = CW_TILE_FLOATS * 4;

// one thread per (row, k) entry of a tile
__global__ void __launch_bounds__(256)
sss_tc_pack_chain_kernel(const float* __restrict__ SCall, float* __restrict__ CWall) {
    const int ch = blockIdx.x, kind = blockIdx.y;
    const float* SC = SCall + (size_t)ch * SCF;
    float* CW = CWall + ((size_t)ch * 4 + kind) * CW_TILE_FLOATS;
    const int dir = kind & 1;
    const float* Phi = SC + dir * DS * DS;
    const float* O = SC + 2 * DS * DS + dir * PO * DS;
    for (int i = threadIdx.x; i < CW_TILE_FLOATS; i += 256) {
        const int row = i >> 5, k = i & 31;
        float out = 0.f;
        if (kind < 2) {
            const int n = row % 48, lo = row / 48, a = k & 15;
            const float w = n < PO ? O[n * DS + a] : Phi[(n - PO) * DS + a];
            const float hi = tf32_hi(w);
            out = lo ? (k < 16 ? tf32_hi(w - hi) : 0.f) : hi;
        } else {
            const int sub = row >> 5, r = row & 31, a = r & 15, lo = r >> 4;
            float w;
            if (sub == 0) w = Phi[(k & 15) * DS + a];   // Phi^T: row a, k = b
            else w = O[k * DS + a];                      // O^T:  row a, k = c
            const float hi = tf32_hi(w);
            if (sub == 0) out = lo ? (k < 16 ? tf32_hi(w - hi) : 0.f) : hi;
            else if (sub == 1) out = lo ? tf32_hi(w - hi) : hi;
            else out = lo ? 0.f : hi;
        }
        CW[i] = out;
    }
}

// ---- explicit shared-space accessors (32-bit shared addresses: STS / LDS with immediate offsets, no generic-address arithmetic) ----
__device__ __forceinline__ void sts128(uint32_t a, float x, float y, float z, float w) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t lds32_u(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc_s(uint32_t slot) {   // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ float lds32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
// byte offsets of the 16-byte chunks of row r in the layouts TMA writes: [rows][32 floats] SWIZZLE_128B / [rows][16 floats] SWIZZLE_64B
struct RowOffs {
    uint32_t o128[8], o64[4];
    __device__ __forceinline__ explicit RowOffs(int r) {
#pragma unroll
        for (int c = 0; c < 8; ++c) o128[c] = (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4));
#pragma unroll
        for (int c = 0; c < 4; ++c) o64[c] = (uint32_t)(r * 64 + ((c ^ ((r >> 1) & 3)) << 4));
    }
};
__device__ __forceinline__ void store_row128_s(uint32_t tile, const RowOffs& ro, const float (&v)[32]) {
#pragma unroll
    for (int c = 0; c < 8; ++c) sts128(tile + ro.o128[c], v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
}
__device__ __forceinline__ void load_row128_s(uint32_t tile, const RowOffs& ro, float (&v)[32]) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const float4 t = lds128(tile + ro.o128[c]);
        v[4 * c] = t.x; v[4 * c + 1] = t.y; v[4 * c + 2] = t.z; v[4 * c + 3] = t.w;
    }
}
__device__ __forceinline__ void store_row64_s(uint32_t tile, const RowOffs& ro, const float (&v)[16]) {
#pragma unroll
    for (int c = 0; c < 4; ++c) sts128(tile + ro.o64[c], v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
}
__device__ __forceinline__ void load_row64_s(uint32_t tile, const RowOffs& ro, float (&v)[16]) {
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const float4 t = lds128(tile + ro.o64[c]);
        v[4 * c] = t.x; v[4 * c + 1] = t.y; v[4 * c + 2] = t.z; v[4 * c + 3] = t.w;
    }
}
// state operand row [raw 16 | lo 16]: the tensor core truncates the raw half to tf32 itself, lo = rn(x - trunc(x))
__device__ __forceinline__ void store_state_raw_lo(uint32_t tile, const RowOffs& ro, const float (&st)[DS]) {
#pragma unroll
    for (int c = 0; c < 4; ++c) sts128(tile + ro.o128[c], st[4 * c], st[4 * c + 1], st[4 * c + 2], st[4 * c + 3]);
#pragma unroll
    for (int c = 0; c < 4; ++c)
        sts128(tile + ro.o128[4 + c], lo_of_trunc(st[4 * c]), lo_of_trunc(st[4 * c + 1]), lo_of_trunc(st[4 * c + 2]), lo_of_trunc(st[4 * c + 3]));
}
// writer side: 16-byte chunk c of row `row`
__device__ __forceinline__ float4 read_chunk128_s(uint32_t tile, int row, int c) { return lds128(tile + row * 128 + ((c ^ (row & 7)) << 4)); }
__device__ __forceinline__ float4 read_chunk64_s(uint32_t tile, int row, int c) { return lds128(tile + row * 64 + ((c ^ ((row >> 1) & 3)) << 4)); }

__device__ __forceinline__ uint64_t desc_kmajor_sw128_s(uint32_t tile) {
    uint64_t d = 0;
    d |= (uint64_t)((tile & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__device__ __forceinline__ void mbar_init_s(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx_s(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Releasing a buffer to the async proxy (a TMA refill) after reading it with ld.shared: the arrive must not be performed before the
// loads have RETURNED.  An mbarrier.arrive issued right behind the ld.shared instructions was measured to overtake them about once in
// eight forward passes (scripts/stress_states.py: a few rows of the saved states then held the NEXT step's TMA data), so the arrive
// takes one register of every outstanding 16-byte load as a (otherwise unused) operand, or is placed behind the instructions that
// consume the loaded values.
__device__ __forceinline__ void mbar_arrive_after_s(uint32_t bar, float a, float b, float c, float d) {
    asm volatile("{\n.reg .f32 dep;\nadd.f32 dep, %1, %2;\nadd.f32 dep, dep, %3;\nadd.f32 dep, dep, %4;\nmbarrier.arrive.shared::cta.b64 _, [%0];\n}" ::"r"(bar), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void mbar_arrive_s(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_wait_s(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void umma_commit_s(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_2d_s(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst), "l"(map),
                 "r"(bar), "r"(c0), "r"(c1) : "memory");
}


// The chain is paced by what ONE epilogue thread (thread = sample) does between two MMAs, so that thread's instruction stream is
// kept minimal: explicit LDS / STS on precomputed swizzled offsets, the raw fp32 value as the hi operand (the tensor core
// truncates), everything that is not the state recurrence done while the MMA is in flight or by other warps (bias, column sums).
// No global memory access sits on the chain: a fence.proxy.async waits for the issuing thread's outstanding loads AND stores,
// so the epilogue threads only touch shared memory and TMEM.
//   * inputs: TMA, two steps ahead, into a 2-slot ring (coefficient tile + this step's per-sample rows); L2 prefetch further ahead
//   * outputs: each epilogue thread overwrites ITS OWN row of the slot's input areas (same swizzled layout) with the step's
//     outputs; two writer warps copy the rows to global memory with coalesced stores and then release the slot
//   forward slot : W 12 KB | `in` = r / r' rows [128][16] (SWIZZLE_64B) -> entering state | yl = yloc / ytmp rows [128][32]
//                  (SWIZZLE_128B) -> ytmp / y
//   backward slot: W 8 KB (state sub-tile + grad_y sub-tile) | grad_y rows of the NEXT step [128][32]; checkpoints go through
//                  a separate single 8 KB staging tile
constexpr int CH_THREADS = 224;                 // warps 0-3: epilogue (thread = sample), warp 4: TMA + MMA issuer (one lane), warps 5-6: writers
constexpr int CH_WRITERS = 64;
constexpr int CHF_SLOT = CW_TILE_BYTES + 8192 + 16384;    // W | in (8 KB at +12288) | yl (16 KB at +20480)
constexpr int CHB_W_BYTES = 64 * 128;                      // state sub-tile + grad_y sub-tile
constexpr int CHB_SLOT = CHB_W_BYTES + 16384;              // W | grad_y rows (16 KB at +8192)
// shared-memory map, as byte offsets from the 1024-aligned base (everything a compile-time constant off one register)
template <bool BWD>
struct ChainMap {
    static constexpr uint32_t state = 0;          // 16 KB: [128][state raw 16 | state lo 16], K-major SWIZZLE_128B
    static constexpr uint32_t in_hi = 16384;      // 16 KB (backward only): raw grad_y rows = hi operand
    static constexpr uint32_t in_lo = 32768;      // 16 KB (backward only)
    static constexpr uint32_t lstage = 49152;     // 8 KB (backward only): adjoint checkpoints on their way to global memory
    static constexpr uint32_t slot0 = BWD ? 57344 : 16384;
    static constexpr uint32_t slot_bytes = BWD ? CHB_SLOT : CHF_SLOT;
    static constexpr uint32_t bars = slot0 + 2 * slot_bytes;
    static constexpr uint32_t full = bars, out_ready = bars + 16, slot_free = bars + 32, state_ready = bars + 48, acc_full = bars + 56,
                              chain_done = bars + 64, lst_ready = bars + 72, lst_free = bars + 80, tmem_slot = bars + 88;
};
__device__ __forceinline__ uint32_t chain_base(uint8_t* smem_raw) {
    const uint32_t a = smem_u32(smem_raw);
    return a + ((1024u - (a & 1023u)) & 1023u);
}
constexpr size_t CHF_SMEM = 16384 + 2 * CHF_SLOT + 128 + 1024;
constexpr size_t CHB_SMEM = 57344 + 2 * CHB_SLOT + 128 + 1024;

// forward: steps 0..nc-1 = anticausal chain over chunks nc-1..0 (saves e_{j+1}; ytmp = yloc + O' e goes back into rbuf),
//          steps nc..2nc-1 = causal chain over chunks 0..nc-1 (saves s_j; y = ytmp + O s + bias, the bias added by the writers).
// The accumulator is double-buffered in TMEM, so only the 16 state columns are read between two MMAs of the chain.
__global__ void __launch_bounds__(CH_THREADS, 2)
sss_tc_chain_fwd_kernel(const __grid_constant__ CUtensorMap map_cw, const __grid_constant__ CUtensorMap map_in, const __grid_constant__ CUtensorMap map_yl,
                        const sn_sss_tc_chunk* __restrict__ chunks, int nchunks, float* __restrict__ rbuf, float* __restrict__ S, float* __restrict__ y,
                        long ldy, const float* __restrict__ bias, long B, int aligned) {
    extern __shared__ uint8_t smem_raw[];
    using M = ChainMap<false>;
    const uint32_t sb = chain_base(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nsteps = 2 * nchunks;
    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; ++i) { mbar_init_s(sb + M::full + 8 * i, 1); mbar_init_s(sb + M::out_ready + 8 * i, 128); mbar_init_s(sb + M::slot_free + 8 * i, CH_WRITERS); }
        mbar_init_s(sb + M::state_ready, 128); mbar_init_s(sb + M::acc_full, 1); mbar_init_s(sb + M::chain_done, CH_WRITERS);
        mbar_fence_init();
        tma_prefetch_desc(&map_cw);
        tma_prefetch_desc(&map_in);
        tma_prefetch_desc(&map_yl);
    }
    if (warp == 4) tmem_alloc_s<256>(sb + M::tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = lds32_u(sb + M::tmem_slot);
    auto chunk_of = [&](int t) { return t < nchunks ? nchunks - 1 - t : t - nchunks; };

    if (warp == 4) {
        if (elect_one()) {
            auto issue = [&](int t) {
                const int s = t & 1, j = chunk_of(t);
                const bool anti = t < nchunks;
                const uint32_t slot = sb + M::slot0 + s * M::slot_bytes, fullb = sb + M::full + 8 * s;
                const int rowc = (int)((long)j * B + (long)blockIdx.x * 128);
                mbar_expect_tx_s(fullb, CW_TILE_BYTES + 8192 + 16384);
                tma_load_2d_s(slot, &map_cw, 0, (j * 4 + (anti ? 1 : 0)) * CW_ROWS, fullb);
                tma_load_2d_s(slot + CW_TILE_BYTES, &map_in, 0, rowc + (anti ? (int)((long)nchunks * B) : 0), fullb);   // R' rows follow the R rows
                tma_load_2d_s(slot + CW_TILE_BYTES + 8192, &map_yl, 0, rowc, fullb);
            };
            auto prefetch = [&](int t) {   // into L2 only
                const int j = chunk_of(t);
                const int rowc = (int)((long)j * B + (long)blockIdx.x * 128);
                tma_prefetch_l2_2d(&map_in, 0, rowc + (t < nchunks ? (int)((long)nchunks * B) : 0));
                tma_prefetch_l2_2d(&map_yl, 0, rowc);
            };
            for (int t = 0; t < CH_PF && t < nsteps; ++t) prefetch(t);
            // the second chain (steps >= nchunks) re-reads through TMA the ytmp rows the writers stored, so its first load waits
            // for chain_done (the writers' last ytmp stores + their proxy fence)
            for (int t = 0; t < 2 && t < nchunks; ++t) issue(t);
            constexpr uint32_t idesc = idesc_tf32(128, 96, false, false);
            CHPROF_DECL(4);
            for (int t = 0; t < nsteps; ++t) {
                const int s = t & 1;
                if (t + CH_PF < nsteps) prefetch(t + CH_PF);
                CHPROF_T0();
                mbar_wait_s(sb + M::full + 8 * s, (t >> 1) & 1);
                CHPROF_LAP(0);
                mbar_wait_s(sb + M::state_ready, t & 1);
                CHPROF_LAP(1);
                tc_fence_after();
                const uint64_t dst = desc_kmajor_sw128_s(sb + M::state);
                const uint64_t dw = desc_kmajor_sw128_s(sb + M::slot0 + s * M::slot_bytes);
                const uint32_t acc = tmem + (uint32_t)(s * 128);
#pragma unroll
                for (int k = 0; k < 4; ++k) mma_tf32(acc, dst + 2 * k, dw + 2 * k, idesc, k ? 1u : 0u);
                umma_commit_s(sb + M::acc_full);
                CHPROF_LAP(2);
                // refill the OTHER slot (step t - 1's) with step t + 1, once the writers have copied step t - 1's outputs out of it
                const int q = t + 1;
                if (q >= 2 && q < nsteps) {
                    mbar_wait_s(sb + M::slot_free + 8 * (q & 1), ((q - 2) >> 1) & 1);
                    if (q == nchunks) {
                        mbar_wait_s(sb + M::chain_done, 0);
                        asm volatile("fence.proxy.async;" ::: "memory");
                    }
                    issue(q);
                } else if (q < 2 && q < nsteps && q >= nchunks) {   // nchunks == 1: step 1 belongs to the second chain
                    mbar_wait_s(sb + M::chain_done, 0);
                    asm volatile("fence.proxy.async;" ::: "memory");
                    issue(q);
                }
                CHPROF_LAP(3);
            }
            CHPROF_PRINT("fwd mma", 4, nsteps);
        }
    } else if (warp < 4) {
        const int r = threadIdx.x;                         // TMEM lane = tile row
        const RowOffs ro(r);
        const uint32_t tlane = tmem + ((uint32_t)(warp * 32) << 16);
        float st[DS];
#pragma unroll
        for (int a = 0; a < DS; ++a) st[a] = 0.f;
        store_state_raw_lo(sb + M::state, ro, st);
        fence_async_smem();
        mbar_arrive_s(sb + M::state_ready);
        CHPROF_DECL(6);
        for (int t = 0; t < nsteps; ++t) {
            const int s = t & 1;
            const uint32_t slot = sb + M::slot0 + s * M::slot_bytes;
            const uint32_t tacc = tlane + (uint32_t)(s * 128);
            CHPROF_T0();
            mbar_wait_s(sb + M::full + 8 * s, (t >> 1) & 1);
            float in[DS];
            load_row64_s(slot + CW_TILE_BYTES, ro, in);
            store_row64_s(slot + CW_TILE_BYTES, ro, st);     // the state entering this step (checkpoint for the backward)
            CHPROF_LAP(0);
            mbar_wait_s(sb + M::acc_full, t & 1);
            CHPROF_LAP(1);
            tc_fence_after();
            // state part first: it is the chain
            uint32_t m[16], l[16];
            tmem_ld16_nowait(tacc + 32, m);
            tmem_ld16_nowait(tacc + 80, l);
            tmem_ld_wait();
            const bool last_of_chain = (t == nchunks - 1);
#pragma unroll
            for (int a = 0; a < DS; ++a) st[a] = last_of_chain ? 0.f : in[a] + (__uint_as_float(m[a]) + __uint_as_float(l[a]));
            CHPROF_LAP(2);
            store_state_raw_lo(sb + M::state, ro, st);
            tc_fence_before();
            fence_async_smem();
            mbar_arrive_s(sb + M::state_ready);
            CHPROF_LAP(3);
            // outputs, off the chain (this step's accumulator is not rewritten before step t + 2): into this thread's own row of
            // the slot; the writers take them from there
            uint32_t ym[32], ylo[32];
            tmem_ld16_nowait(tacc, reinterpret_cast<uint32_t(&)[16]>(ym[0]));
            tmem_ld16_nowait(tacc + 16, reinterpret_cast<uint32_t(&)[16]>(ym[16]));
            tmem_ld16_nowait(tacc + 48, reinterpret_cast<uint32_t(&)[16]>(ylo[0]));
            tmem_ld16_nowait(tacc + 64, reinterpret_cast<uint32_t(&)[16]>(ylo[16]));
            float yl[PO];
            load_row128_s(slot + CW_TILE_BYTES + 8192, ro, yl);
            tmem_ld_wait();
            tc_fence_before();
            CHPROF_LAP(4);
#pragma unroll
            for (int c = 0; c < PO; ++c) yl[c] += __uint_as_float(ym[c]) + __uint_as_float(ylo[c]);
            store_row128_s(slot + CW_TILE_BYTES + 8192, ro, yl);
            mbar_arrive_s(sb + M::out_ready + 8 * s);
            CHPROF_LAP(5);
        }
        if (threadIdx.x == 0) { CHPROF_PRINT("fwd epi", 6, nsteps); }
    } else {
        // writers: rows of step t -> global memory, coalesced; then the slot may be refilled
        const int wt = threadIdx.x - 160;
        for (int t = 0; t < nsteps; ++t) {
            const bool anti = t < nchunks;
            const int j = chunk_of(t), s = t & 1;
            const uint32_t slot = sb + M::slot0 + s * M::slot_bytes;
            const sn_sss_tc_chunk c = chunks[j];
            // this thread always handles 16-byte column chunk (wt & 7) of the y rows: its slice of the bias
            float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (!anti && bias != nullptr) {
                const int c0 = 4 * (wt & 7);
                if (c0 < c.nrows) b4.x = __ldg(bias + c.row0 + c0);
                if (c0 + 1 < c.nrows) b4.y = __ldg(bias + c.row0 + c0 + 1);
                if (c0 + 2 < c.nrows) b4.z = __ldg(bias + c.row0 + c0 + 2);
                if (c0 + 3 < c.nrows) b4.w = __ldg(bias + c.row0 + c0 + 3);
            }
            mbar_wait_s(sb + M::out_ready + 8 * s, (t >> 1) & 1);
            float4 sv[8], yv[16];
#pragma unroll
            for (int k = 0; k < 8; ++k) { const int i = k * CH_WRITERS + wt; sv[k] = read_chunk64_s(slot + CW_TILE_BYTES, i >> 2, i & 3); }
#pragma unroll
            for (int k = 0; k < 16; ++k) { const int i = k * CH_WRITERS + wt; yv[k] = read_chunk128_s(slot + CW_TILE_BYTES + 8192, i >> 3, i & 7); }
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int i = k * CH_WRITERS + wt;
                const long row = (long)blockIdx.x * 128 + (i >> 2);
                if (row < B) *(reinterpret_cast<float4*>(S + ((size_t)j * B + row) * 32 + (anti ? DS : 0)) + (i & 3)) = sv[k];
            }
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const int i = k * CH_WRITERS + wt;
                const long row = (long)blockIdx.x * 128 + (i >> 3);
                const int c0 = 4 * (i & 7);
                if (row < B) {
                    if (anti) {
                        *(reinterpret_cast<float4*>(rbuf + ((size_t)j * B + row) * 32) + (i & 7)) = yv[k];
                    } else if (c0 < c.nrows) {
                        float* yp = y + row * ldy + c.row0 + c0;
                        const float4 o = make_float4(yv[k].x + b4.x, yv[k].y + b4.y, yv[k].z + b4.z, yv[k].w + b4.w);
                        if (aligned && c0 + 4 <= c.nrows) {
                            *reinterpret_cast<float4*>(yp) = o;
                        } else {
                            yp[0] = o.x;
                            if (c0 + 1 < c.nrows) yp[1] = o.y;
                            if (c0 + 2 < c.nrows) yp[2] = o.z;
                            if (c0 + 3 < c.nrows) yp[3] = o.w;
                        }
                    }
                }
            }
            // release the slot only now: the stores above have consumed every loaded value (see mbar_arrive_after_s)
            mbar_arrive_after_s(sb + M::slot_free + 8 * s, sv[0].x, sv[7].x, yv[0].x, yv[15].x);
            if (t == nchunks - 1) {
                asm volatile("fence.proxy.async;" ::: "memory");   // ytmp stores -> visible to the TMA reads of the second chain
                __threadfence();
                mbar_arrive_s(sb + M::chain_done);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        tmem_dealloc<256>(tmem);
    }
}

// backward: the lambda chain over chunks nc-1..0 and the mu chain over chunks 0..nc-1, one per CTA (blockIdx.y).
// L[j][row][0..15] = lambda_{j+1}, L[j][row][16..31] = mu_j ; grad_bias += column sums of grad_y (second chain, by the writer warps).
// Ring slot of step t: coefficient tile of step t + the grad_y rows of step t + 1.  The chain is paced by the instruction stream of
// the epilogue threads between two MMAs, so a sample row is shared by TWO threads (warps w and w + 4 read the same TMEM lanes):
// each takes half of the grad_y row and half of the state.  While the MMA of step t is in flight a thread fetches its half row of
// step t + 1 and computes the lo part in registers; after the accumulator arrives it only adds, splits its 8 state values and stores
// the operand rows.  Step 0's rows arrive through a prologue load into the (still unused) lo tile.
constexpr int CHB_EPI = 256;                       // warps 0-7: epilogue, warp 8: TMA + MMA issuer (one lane), warps 9-10: writers
constexpr int CHB_THREADS = CHB_EPI + 32 + CH_WRITERS;
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr));
}
__global__ void __launch_bounds__(CHB_THREADS, 2)
sss_tc_chain_bwd_kernel(const __grid_constant__ CUtensorMap map_cw, const __grid_constant__ CUtensorMap map_gy, const sn_sss_tc_chunk* __restrict__ chunks,
                        int nchunks, float* __restrict__ L, float* __restrict__ gbias, long B) {
    extern __shared__ uint8_t smem_raw[];
    using M = ChainMap<true>;
    const uint32_t sb = chain_base(smem_raw);
    const int warp = threadIdx.x >> 5;
    // grid.y = 2: one adjoint chain per CTA (0: lambda over chunks nc-1..0, 1: mu over chunks 0..nc-1); the two are independent
    const int dir = blockIdx.y;
    const int nsteps = nchunks;
    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; ++i) { mbar_init_s(sb + M::full + 8 * i, 1); mbar_init_s(sb + M::slot_free + 8 * i, CHB_EPI + 1 + CH_WRITERS); }
        mbar_init_s(sb + M::state_ready, CHB_EPI); mbar_init_s(sb + M::acc_full, 1); mbar_init_s(sb + M::chain_done, 1);
        mbar_init_s(sb + M::lst_ready, CHB_EPI); mbar_init_s(sb + M::lst_free, CH_WRITERS);
        mbar_fence_init();
        tma_prefetch_desc(&map_cw);
        tma_prefetch_desc(&map_gy);
    }
    if (warp == 8) tmem_alloc_s<32>(sb + M::tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = lds32_u(sb + M::tmem_slot);
    auto chunk_of = [&](int t) { return dir ? t : nchunks - 1 - t; };

    if (warp == 8) {
        if (elect_one()) {
            auto issue = [&](int t) {
                const int s = t & 1, j = chunk_of(t);
                const uint32_t slot = sb + M::slot0 + s * M::slot_bytes, fullb = sb + M::full + 8 * s;
                const bool has_next = t + 1 < nsteps;
                mbar_expect_tx_s(fullb, CHB_W_BYTES + (has_next ? 16384 : 0));
                tma_load_2d_s(slot, &map_cw, 0, (j * 4 + (dir ? 3 : 2)) * CW_ROWS, fullb);
                if (has_next) tma_load_2d_s(slot + CHB_W_BYTES, &map_gy, chunks[chunk_of(t + 1)].row0, blockIdx.x * 128, fullb);
            };
            auto prefetch = [&](int t) { tma_prefetch_l2_2d(&map_gy, chunks[chunk_of(t)].row0, blockIdx.x * 128); };
            for (int t = 1; t < CH_PF && t < nsteps; ++t) prefetch(t);
            mbar_expect_tx_s(sb + M::chain_done, 16384);
            tma_load_2d_s(sb + M::in_lo, &map_gy, chunks[chunk_of(0)].row0, blockIdx.x * 128, sb + M::chain_done);
            for (int t = 0; t < 2 && t < nsteps; ++t) issue(t);
            constexpr uint32_t idesc32 = idesc_tf32(128, 32, false, false);
            constexpr uint32_t idesc16 = idesc_tf32(128, 16, false, false);
            CHPROF_DECL(4);
            for (int t = 0; t < nsteps; ++t) {
                const int s = t & 1;
                if (t + CH_PF < nsteps) prefetch(t + CH_PF);
                CHPROF_T0();
                mbar_wait_s(sb + M::full + 8 * s, (t >> 1) & 1);
                CHPROF_LAP(0);
                mbar_wait_s(sb + M::state_ready, t & 1);
                CHPROF_LAP(1);
                tc_fence_after();
                const uint32_t slot = sb + M::slot0 + s * M::slot_bytes;
                const uint64_t dst = desc_kmajor_sw128_s(sb + M::state), dih = desc_kmajor_sw128_s(sb + M::in_hi), dil = desc_kmajor_sw128_s(sb + M::in_lo);
                const uint64_t dw0 = desc_kmajor_sw128_s(slot), dw1 = desc_kmajor_sw128_s(slot + 4096);
#pragma unroll
                for (int k = 0; k < 4; ++k) mma_tf32(tmem, dst + 2 * k, dw0 + 2 * k, idesc32, k ? 1u : 0u);   // [Phi^T hi | hi ; lo | 0]
#pragma unroll
                for (int k = 0; k < 4; ++k) mma_tf32(tmem, dih + 2 * k, dw1 + 2 * k, idesc32, 1u);            // grad_y hi x [O^T hi ; O^T lo]
#pragma unroll
                for (int k = 0; k < 4; ++k) mma_tf32(tmem, dil + 2 * k, dw1 + 2 * k, idesc16, 1u);            // grad_y lo x  O^T hi
                umma_commit_s(sb + M::acc_full);
                umma_commit_s(sb + M::slot_free + 8 * s);
                CHPROF_LAP(2);
                if (t + 2 < nsteps) {
                    mbar_wait_s(sb + M::slot_free + 8 * s, (t >> 1) & 1);
                    issue(t + 2);
                }
                CHPROF_LAP(3);
            }
            CHPROF_PRINT("bwd mma", 4, nsteps);
        }
    } else if (warp < 8) {
        const int r = threadIdx.x & 127, h = threadIdx.x >> 7;          // tile row, half
        // byte offsets of this thread's 16-byte chunks (runtime half -> computed here, not indexed out of a table)
        uint32_t og[4], osr[2], osl[2], ock[2];
#pragma unroll
        for (int c = 0; c < 4; ++c) og[c] = (uint32_t)(r * 128 + (((4 * h + c) ^ (r & 7)) << 4));
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            osr[c] = (uint32_t)(r * 128 + (((2 * h + c) ^ (r & 7)) << 4));
            osl[c] = (uint32_t)(r * 128 + (((4 + 2 * h + c) ^ (r & 7)) << 4));
            ock[c] = (uint32_t)(r * 64 + (((2 * h + c) ^ ((r >> 1) & 3)) << 4));
        }
        const uint32_t tacc = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        // this thread's 16-byte chunks: grad_y row chunks 4h..4h+3, state raw chunks 2h, 2h+1 and lo chunks 4+2h, 5+2h, checkpoint chunks 2h, 2h+1
        float st[8], g[16], gl[16];
#pragma unroll
        for (int a = 0; a < 8; ++a) st[a] = 0.f;
        auto load_g = [&](uint32_t tile) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float4 v = lds128(tile + og[c]);
                g[4 * c] = v.x; g[4 * c + 1] = v.y; g[4 * c + 2] = v.z; g[4 * c + 3] = v.w;
            }
#pragma unroll
            for (int c = 0; c < 16; ++c) gl[c] = lo_of_trunc(g[c]);
        };
        auto store_operands = [&]() {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                sts128(sb + M::state + osr[c], st[4 * c], st[4 * c + 1], st[4 * c + 2], st[4 * c + 3]);
                sts128(sb + M::state + osl[c], lo_of_trunc(st[4 * c]), lo_of_trunc(st[4 * c + 1]), lo_of_trunc(st[4 * c + 2]),
                       lo_of_trunc(st[4 * c + 3]));
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                sts128(sb + M::in_hi + og[c], g[4 * c], g[4 * c + 1], g[4 * c + 2], g[4 * c + 3]);
                sts128(sb + M::in_lo + og[c], gl[4 * c], gl[4 * c + 1], gl[4 * c + 2], gl[4 * c + 3]);
            }
        };
        mbar_wait_s(sb + M::chain_done, 0);
        load_g(sb + M::in_lo);        // raw grad_y rows of step 0 (each thread only touches its own half row)
        store_operands();
        fence_async_smem();
        mbar_arrive_s(sb + M::state_ready);
        CHPROF_DECL(6);
        for (int t = 0; t < nsteps; ++t) {
            const int s = t & 1;
            const bool has_next = t + 1 < nsteps;
            CHPROF_T0();
            // checkpoint of the adjoint entering this step -> staging tile (the writers emptied it during the previous step)
            if (t > 0) mbar_wait_s(sb + M::lst_free, (t - 1) & 1);
#pragma unroll
            for (int c = 0; c < 2; ++c) sts128(sb + M::lstage + ock[c], st[4 * c], st[4 * c + 1], st[4 * c + 2], st[4 * c + 3]);
            mbar_arrive_s(sb + M::lst_ready);
            CHPROF_LAP(0);
            // next step's grad_y half row and its lo part, while this step's MMA runs
            mbar_wait_s(sb + M::full + 8 * s, (t >> 1) & 1);
            if (has_next) load_g(sb + M::slot0 + s * M::slot_bytes + CHB_W_BYTES);
            mbar_arrive_after_s(sb + M::slot_free + 8 * s, g[0], g[4], g[8], g[12]);   // only once the four 16-byte loads have returned
            CHPROF_LAP(1);
            mbar_wait_s(sb + M::acc_full, t & 1);
            CHPROF_LAP(2);
            tc_fence_after();
            uint32_t m[8], l[8];
            tmem_ld8_nowait(tacc + 8 * h, m);
            tmem_ld8_nowait(tacc + 16 + 8 * h, l);
            tmem_ld_wait();
            tc_fence_before();
#pragma unroll
            for (int a = 0; a < 8; ++a) st[a] = __uint_as_float(m[a]) + __uint_as_float(l[a]);
            CHPROF_LAP(3);
            if (has_next) {
                store_operands();
                CHPROF_LAP(4);
                fence_async_smem();
                mbar_arrive_s(sb + M::state_ready);
                CHPROF_LAP(5);
            }
        }
        if (threadIdx.x == 0) { CHPROF_PRINT("bwd epi", 6, nsteps); }
    } else {
        // writers: adjoint checkpoints -> L; column sums of the second chain's grad_y rows -> grad_bias
        const int wt = threadIdx.x - (CHB_EPI + 32);
        for (int t = 0; t < nsteps; ++t) {
            const int j = chunk_of(t), s = t & 1;
            mbar_wait_s(sb + M::lst_ready, t & 1);
            float4 sv[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) { const int i = k * CH_WRITERS + wt; sv[k] = read_chunk64_s(sb + M::lstage, i >> 2, i & 3); }
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int i = k * CH_WRITERS + wt;
                const long row = (long)blockIdx.x * 128 + (i >> 2);
                if (row < B) *(reinterpret_cast<float4*>(L + ((size_t)j * B + row) * 32 + (dir ? DS : 0)) + (i & 3)) = sv[k];
            }
            mbar_arrive_after_s(sb + M::lst_free, sv[0].x, sv[2].x, sv[5].x, sv[7].x);   // the staging tile is rewritten by generic stores, but keep one rule
            // the slot of step t holds the grad_y rows of step t + 1: thread = (column, half of the rows); rows past B are zero (TMA fill)
            mbar_wait_s(sb + M::full + 8 * s, (t >> 1) & 1);
            // column sums: the mu CTA covers chunks 1..nc-1 (the rows its slots carry), the lambda CTA adds chunk 0 (its last step's rows);
            // a single-chunk layer has no slot rows at all: the host sums that case
            if (gbias != nullptr && t + 1 < nsteps && (dir == 1 || t + 2 == nsteps)) {
                const uint32_t tile = sb + M::slot0 + s * M::slot_bytes + CHB_W_BYTES;
                const int col = wt & 31, r0 = (wt >> 5) * 64;
                float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
                for (int rr = 0; rr < 64; rr += 4) {
                    const int row = r0 + rr;
                    a0 += lds32(tile + row * 128 + (((col >> 2) ^ (row & 7)) << 4) + (col & 3) * 4);
                    a1 += lds32(tile + (row + 1) * 128 + (((col >> 2) ^ ((row + 1) & 7)) << 4) + (col & 3) * 4);
                    a2 += lds32(tile + (row + 2) * 128 + (((col >> 2) ^ ((row + 2) & 7)) << 4) + (col & 3) * 4);
                    a3 += lds32(tile + (row + 3) * 128 + (((col >> 2) ^ ((row + 3) & 7)) << 4) + (col & 3) * 4);
                }
                mbar_arrive_after_s(sb + M::slot_free + 8 * s, a0, a1, a2, a3);          // the sums depend on every load
                const sn_sss_tc_chunk c = chunks[chunk_of(t + 1)];
                if (col < c.nrows) atomicAdd(gbias + c.row0 + col, (a0 + a1) + (a2 + a3));
            } else {
                mbar_arrive_s(sb + M::slot_free + 8 * s);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) {
        tc_fence_after();
        tmem_dealloc<32>(tmem);
    }
}

// ------------------------------------------------------------------------------------------
// 5. gradient GEMM: dM_j (64 x N) += [gy_j | lambda | mu]^T [u_j | s | e] over a range of samples, 3xTF32 (all four hi/lo terms).
//    K = samples; both operands MN-major straight from TMA boxes of [32 samples][32 floats] (SWIZZLE_128B_ATOM_32B, the one
//    layout kind::tf32 accepts for MN-major operands).
//    A (M = 128): blocks gy_hi, L_hi, gy_lo, L_lo;  B (N = 32 (nkb+1)): x blocks then the state block; hi and lo tiles.
// ------------------------------------------------------------------------------------------
constexpr int G2_STAGES = 3;
constexpr int G2_CONV = 128 * G2_STAGES;         // converter threads: one group of four warps per pipeline stage
constexpr int G2_THREADS = 64 + G2_CONV + 128;
constexpr int G2_KS = 32;                        // samples per stage
constexpr int G2_BLK = G2_KS * 128;              // one 32-feature block: 4 KB
constexpr int G2_A_BYTES = 4 * G2_BLK;           // 16 KB
constexpr int G2_BH_BYTES = (KB_MAX + 1) * G2_BLK;   // 24 KB
constexpr int G2_STAGE_BYTES = G2_A_BYTES + 2 * G2_BH_BYTES;   // 64 KB
#ifndef SN_G2_PF
#define SN_G2_PF 2
#endif
#ifndef SN_G2_ABL
#define SN_G2_ABL 0      // measurements only: 1 = no reductions into dM, 2 = items ordered range-fastest
#endif
// item -> (sample range, chunk)
__device__ __forceinline__ void g2_item(int item, int nchunks, int nranges, int& rg, int& ch) {
#if SN_G2_ABL == 2
    ch = item / nranges; rg = item - ch * nranges;
#else
    rg = item / nchunks; ch = item - rg * nchunks; (void)nranges;
#endif
}
constexpr int G2_PF = SN_G2_PF;                   // L2 prefetch distance in 32-sample steps
constexpr int G2_STG_OFF = 256;                   // behind the barriers: two 8 KB staging tiles of the epilogue, then the chunk table
constexpr size_t G2_SMEM = (size_t)G2_STAGES * G2_STAGE_BYTES + 1024 + G2_STG_OFF + 2 * 8192;

__global__ void __launch_bounds__(G2_THREADS, 1)
sss_tc_grad_gemm_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_gy, const __grid_constant__ CUtensorMap map_l,
                        const __grid_constant__ CUtensorMap map_s, const sn_sss_tc_chunk* __restrict__ chunks, int nchunks, int nranges, int per,
                        long B, float* __restrict__ dM) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space (LDS/STS)
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + G2_STAGES * G2_STAGE_BYTES);
    uint64_t* conv = full + G2_STAGES;
    uint64_t* empty = conv + G2_STAGES;
    uint64_t* acc_full = empty + G2_STAGES;
    uint64_t* acc_empty = acc_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    int4* ctab = reinterpret_cast<int4*>(smem + G2_STAGES * G2_STAGE_BYTES + G2_STG_OFF + 2 * 8192);   // (col0, nkb, row0, -) per chunk

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ntk = (int)((B + G2_KS - 1) / G2_KS);
    const int nitems = nranges * nchunks;           // item = (sample range, chunk), chunk fastest: neighbouring CTAs read neighbouring
    if ((int)blockIdx.x >= nitems) return;          // 512-byte pieces of the same x rows at the same time

    for (int i = threadIdx.x; i < nchunks; i += G2_THREADS) ctab[i] = make_int4(chunks[i].col0, chunks[i].nkb, chunks[i].row0, 0);
    if (threadIdx.x == 0) {
        for (int s = 0; s < G2_STAGES; ++s) { mbar_init(full + s, 1); mbar_init(conv + s, 128); mbar_init(empty + s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(acc_full + b, 1); mbar_init(acc_empty + b, 128); }
        mbar_fence_init();
        tma_prefetch_desc(&map_x);
        tma_prefetch_desc(&map_gy);
        tma_prefetch_desc(&map_l);
        tma_prefetch_desc(&map_s);
    }
    if (warp == 1) tmem_alloc<512>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (elect_one()) {
            // L2 prefetch cursor: G2_PF 32-sample steps ahead of the 3-stage shared-memory pipeline, across item boundaries
            int pitem = blockIdx.x, pt = 0, pt1 = 0, pch = 0, ahead = 0;
            auto pcursor_open = [&]() {
                if (pitem >= nitems) return;
                int rg; g2_item(pitem, nchunks, nranges, rg, pch);
                pt = rg * per;
                pt1 = pt + per < ntk ? pt + per : ntk;
            };
            auto prefetch_one = [&]() {
                if (pitem >= nitems) return;
                const int4 c = ctab[pch];
                tma_prefetch_l2_2d(&map_gy, c.z, pt * G2_KS);
                tma_prefetch_l2_3d(&map_l, 0, pt * G2_KS, pch);
                for (int i = 0; i < c.y; ++i) tma_prefetch_l2_2d(&map_x, c.x + i * KBW, pt * G2_KS);
                tma_prefetch_l2_3d(&map_s, 0, pt * G2_KS, pch);
                if (++pt >= pt1) { pitem += gridDim.x; pcursor_open(); }
            };
            pcursor_open();
            for (; ahead < G2_PF; ++ahead) prefetch_one();
            uint32_t it = 0;
            for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
                int rg, ch; g2_item(item, nchunks, nranges, rg, ch);
                const int4 c = ctab[ch];
                const int nkb = c.y, nblk = nkb + 1;
                const int t0 = rg * per, t1 = t0 + per < ntk ? t0 + per : ntk;
                for (int t = t0; t < t1; ++t, ++it) {
                    prefetch_one();
                    const uint32_t s = it % G2_STAGES, round = it / G2_STAGES;
                    if (round > 0) mbar_wait(empty + s, (round - 1) & 1);
                    uint8_t* st = smem + s * G2_STAGE_BYTES;
                    uint8_t* bh = st + G2_A_BYTES;
                    mbar_expect_tx(full + s, (2 + nblk) * G2_BLK);
                    tma_load_2d(st, &map_gy, c.z, t * G2_KS, full + s);
                    tma_load_3d(st + G2_BLK, &map_l, 0, t * G2_KS, ch, full + s);
                    for (int i = 0; i < nkb; ++i) tma_load_2d(bh + i * G2_BLK, &map_x, c.x + i * KBW, t * G2_KS, full + s);
                    tma_load_3d(bh + nkb * G2_BLK, &map_s, 0, t * G2_KS, ch, full + s);
                }
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
            // the tensor core adds into its accumulator with truncation (an error linear in the number of additions): an item is at
            // most 1024 samples (the host keeps `per` <= 32), and every item has a TMEM accumulator of its own (two, alternating, so
            // that the epilogue of one item runs under the main loop of the next)
            uint32_t it = 0, ai = 0;
            for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++ai) {
                int rg, ch; g2_item(item, nchunks, nranges, rg, ch);
                const int nblk = ctab[ch].y + 1;
                const int t0 = rg * per, t1 = t0 + per < ntk ? t0 + per : ntk;
                const uint32_t idesc = idesc_tf32(128, 32 * nblk, true, true);
                const uint32_t b = ai & 1;
                if (ai >= 2) mbar_wait(acc_empty + b, ((ai >> 1) - 1) & 1);
                tc_fence_after();
                const uint32_t acc = tmem_base + b * 256u;
                for (int t = t0; t < t1; ++t, ++it) {
                    const uint32_t s = it % G2_STAGES, round = it / G2_STAGES;
                    mbar_wait(conv + s, round & 1);
                    tc_fence_after();
                    uint8_t* st = smem + s * G2_STAGE_BYTES;
#pragma unroll
                    for (int k = 0; k < G2_KS / 8; ++k) {   // 8 samples = 8 rows of 128 bytes = 1024 bytes per UMMA
                        const uint64_t da = desc_mnmajor_sw128_32b(st + k * 1024, G2_BLK);
                        const uint64_t dbh = desc_mnmajor_sw128_32b(st + G2_A_BYTES + k * 1024, G2_BLK);
                        const uint64_t dbl = desc_mnmajor_sw128_32b(st + G2_A_BYTES + G2_BH_BYTES + k * 1024, G2_BLK);
                        mma_tf32(acc, da, dbh, idesc, (t == t0 && k == 0) ? 0u : 1u);
                        mma_tf32(acc, da, dbl, idesc, 1u);
                    }
                    umma_commit(empty + s);
                }
                umma_commit(acc_full + b);
            }
        }
    } else if (warp < 2 + G2_CONV / 32) {
        // one group of four converter warps per stage (see the local GEMM; a group must own its stages, or it would skip phases
        // of their `full` barriers)
        const int grp = (warp - 2) >> 2, ct = (threadIdx.x - 64) & 127;
        uint32_t it = 0;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
            int rg, ch; g2_item(item, nchunks, nranges, rg, ch);
            const int nblk = ctab[ch].y + 1;
            const int t0 = rg * per, t1 = t0 + per < ntk ? t0 + per : ntk;
            for (int t = t0; t < t1; ++t, ++it) {
                if ((int)(it % G2_STAGES) != grp) continue;
                const uint32_t s = it % G2_STAGES, round = it / G2_STAGES;
                mbar_wait(full + s, round & 1);
                uint8_t* st = smem + s * G2_STAGE_BYTES;
                {   // A: gy, L (8 KB) -> lo at +8 KB
                    float4* h = reinterpret_cast<float4*>(st);
                    float4* l = h + 2 * G2_BLK / 16;
#pragma unroll
                    for (int i = 0; i < 2 * G2_BLK / 16 / 128; ++i) {
                        float4 ll;
                        lo_of_trunc(h[ct + 128 * i], ll);   // hi = the raw tile (the tensor core truncates)
                        l[ct + 128 * i] = ll;
                    }
                }
                {   // B: x blocks + state block -> lo at +24 KB
                    float4* h = reinterpret_cast<float4*>(st + G2_A_BYTES);
                    float4* l = h + G2_BH_BYTES / 16;
                    const int n16 = nblk * G2_BLK / 16;
#pragma unroll 4
                    for (int i = ct; i < n16; i += 128) {
                        float4 ll;
                        lo_of_trunc(h[i], ll);
                        l[i] = ll;
                    }
                }
                fence_async_smem();
                mbar_arrive(conv + s);
            }
        }
    } else {
        // epilogue.  Rows m and m + 64 of the accumulator are the hi and lo parts of the same dM row and sit in the TMEM lanes of
        // different warps (q and q + 2): they are added through a small swizzled staging tile before they leave as red.global.add, which
        // halves the atomic traffic (measured: 200 MB of reductions per step at B = 65 536 cost the kernel 50 us of its 405).
        // Column groups of 32 alternate roles: warps 2, 3 stage and warps 0, 1 reduce on even groups, the other way round on odd ones;
        // two staging tiles, one named barrier per group (a tile is rewritten two groups later, behind the barrier its readers passed).
        const int q = warp & 3;
        const int r64 = (q & 1) * 32 + lane;             // dM row of the chunk
        const uint32_t stg = smem_u32(smem + G2_STAGES * G2_STAGE_BYTES + G2_STG_OFF);
        const uint32_t myrow = (uint32_t)r64 * 128u;
        uint32_t ai = 0, grp = 0;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++ai) {
            int rg, ch; g2_item(item, nchunks, nranges, rg, ch);
            const int nblk = ctab[ch].y + 1;
            const uint32_t b = ai & 1;
            mbar_wait(acc_full + b, (ai >> 1) & 1);
            tc_fence_after();
            float* drow = dM + ((size_t)ch * 64 + r64) * DMC;
            const uint32_t acc = tmem_base + b * 256u + ((uint32_t)(q * 32) << 16);
            for (int c0 = 0; c0 < 32 * nblk; c0 += 32, ++grp) {
                uint32_t v[32];
                tmem_ld16_nowait(acc + c0, *reinterpret_cast<uint32_t(*)[16]>(v));
                tmem_ld16_nowait(acc + c0 + 16, *reinterpret_cast<uint32_t(*)[16]>(v + 16));
                tmem_ld_wait();
                const uint32_t tile = stg + (grp & 1) * 8192u + myrow;
                const bool stager = ((q >> 1) ^ (int)(grp & 1)) != 0;      // even groups: warps 2, 3 (q >> 1 == 1)
                if (stager) {
#pragma unroll
                    for (int c = 0; c < 8; ++c)
                        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(tile + (uint32_t)((c ^ (r64 & 7)) << 4)), "r"(v[4 * c]), "r"(v[4 * c + 1]),
                                     "r"(v[4 * c + 2]), "r"(v[4 * c + 3]) : "memory");
                }
                named_bar_sync(2, 128);
                if (!stager) {
#if SN_G2_ABL == 1
                    if (v[0] != 0x7fc12345u) continue;    // ablation: no reductions into dM
#endif
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        float4 o;
                        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(o.x), "=f"(o.y), "=f"(o.z), "=f"(o.w) : "r"(tile + (uint32_t)((c ^ (r64 & 7)) << 4)) : "memory");
                        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(drow + c0 + 4 * c), "f"(__uint_as_float(v[4 * c]) + o.x),
                                     "f"(__uint_as_float(v[4 * c + 1]) + o.y), "f"(__uint_as_float(v[4 * c + 2]) + o.z), "f"(__uint_as_float(v[4 * c + 3]) + o.w)
                                     : "memory");
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(acc_empty + b);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<512>(tmem_base);
    }
}

// ------------------------------------------------------------------------------------------
// 6. chain rule through the chunk-matrix construction.  grid (nchunks, 2); thread = column as in the build kernel.
//    Phase 1 replays the construction and stores the state entering every stage; phase 2 walks the stages backwards.
// ------------------------------------------------------------------------------------------
// 6a serial part.  Scratch per (chunk, direction), feature-major over the 192 column threads:
//      V[stage][16][192] state entering the stage | LAM[stage][16][192] adjoint of the state leaving it | GY[stage][16][192] its gy rows
// 6b (sss_tc_build_red_kernel) turns them into the parameter gradients that are sums over the chunk's columns.
constexpr int BB_PLANE = DS * BUILD_THREADS;          // floats of one [16][192] plane
constexpr int BB_SCR = 3 * LMAX * BB_PLANE;           // per (chunk, direction)

__global__ void __launch_bounds__(BUILD_THREADS)
sss_tc_build_bwd_kernel(const sn_sss_stage* __restrict__ stages, int n, const sn_sss_tc_chunk* __restrict__ chunks, const float* __restrict__ params,
                        const float* __restrict__ dMall, float* __restrict__ scratch, float* __restrict__ gparams) {
    extern __shared__ __align__(16) float build_smem[];
    __shared__ sn_sss_stage sdesc[LMAX];
    __shared__ StageP sptr[LMAX];
    float* dMs = build_smem;                      // the chunk's dM tile, 64 x 192
    float* pbuf = build_smem + 64 * DMC;
    const sn_sss_tc_chunk c = chunks[blockIdx.x];
    const int dir = blockIdx.y, t = threadIdx.x;
    const bool is_in = t < c.ncols;
    const int sidx = t - c.ncols;
    const bool active = is_in || sidx < DS;
    float* scr = scratch + ((size_t)blockIdx.x * 2 + dir) * BB_SCR;
    float* Vs = scr;
    float* Ls = scr + LMAX * BB_PLANE;
    float* Gs = scr + 2 * LMAX * BB_PLANE;
    const int nst = c.k_end - c.k_begin;
    const int col = c.col0 + t;
    const int cidx = is_in ? t : c.nkb * KBW + dir * DS + sidx;
    if (t < nst) sdesc[t] = stage_of(stages, n, dir, dir == 0 ? c.k_begin + t : c.k_end - 1 - t);
    {
        const float4* src = reinterpret_cast<const float4*>(dMall + (size_t)blockIdx.x * 64 * DMC);
        for (int e = t; e < 64 * DMC / 4; e += BUILD_THREADS)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dMs + 4 * e)), "l"(src + e) : "memory");
    }
    __syncthreads();
    chunk_params_async(pbuf, sptr, sdesc, nst, params, t, BUILD_THREADS);
    cp_async_commit();
    cp_async_wait_all();
    __syncthreads();

    float v[DS], yv[SOUT_MAX];
#pragma unroll
    for (int a = 0; a < DS; ++a) v[a] = (active && !is_in && a == sidx && sidx < sdesc[0].d_in) ? 1.f : 0.f;
    int my_i = -1;
    // phase 1: replay the construction, keeping the state that enters every stage
    for (int i = 0; i < nst; ++i) {
        const sn_sss_stage& st = sdesc[i];
        const int local = col - st.in_off;
        const bool mine = is_in && local >= 0 && local < st.in_dim;
#pragma unroll
        for (int a = 0; a < DS; ++a) Vs[(i * DS + a) * BUILD_THREADS + t] = v[a];
        if (active) stage_apply<false>(st, pbuf, sptr[i], v, yv, mine, local);
        if (mine) my_i = i;
    }
    // adjoint of the state leaving the last stage: dR / dPhi rows of dM
    float lam[DS];
#pragma unroll
    for (int b = 0; b < DS; ++b) lam[b] = active ? dMs[(PO + dir * DS + b) * DMC + cidx] : 0.f;
    // phase 2: stages backwards
    for (int i = nst - 1; i >= 0; --i) {
        const sn_sss_stage& st = sdesc[i];
        const StageP& ps = sptr[i];
        const int local = col - st.in_off;
        const bool mine = (i == my_i);
        const bool before = is_in ? (my_i >= 0 && my_i < i) : true;
        const bool support = active && (is_in ? (dir == 0 ? (before || mine) : before) : true);
        const int rbase = st.out_off - c.row0;
        float g[SOUT_MAX];
#pragma unroll
        for (int r = 0; r < SOUT_MAX; ++r) g[r] = 0.f;
#pragma unroll
        for (int r = 0; r < SOUT_MAX; ++r) {
            if (r >= st.out_dim) break;
            if (support) g[r] = dMs[(rbase + r) * DMC + cidx];
            Gs[(i * DS + r) * BUILD_THREADS + t] = g[r];
        }
#pragma unroll
        for (int b = 0; b < DS; ++b) Ls[(i * DS + b) * BUILD_THREADS + t] = lam[b];
        if (mine) {
#pragma unroll
            for (int b = 0; b < DS; ++b) {
                if (b >= st.d_out) break;
                gparams[st.off_su + b * st.in_dim + local] += lam[b];
            }
            if (st.off_yu >= 0) {
#pragma unroll
                for (int r = 0; r < SOUT_MAX; ++r) {
                    if (r >= st.out_dim) break;
                    gparams[st.off_yu + r * st.in_dim + local] += g[r];
                }
            }
        }
        // lambda entering the stage: ss^T lam + ys^T g
        float nl[DS];
#pragma unroll
        for (int a = 0; a < DS; ++a) nl[a] = 0.f;
        const float* ss = pbuf + ps.ss;
        const float* ys = pbuf + ps.ys;
        if (st.d_in == DS && st.d_out == DS) {
#pragma unroll
            for (int b = 0; b < DS; ++b) axpy_row16(ss + b * DS, lam[b], nl);
        } else {
#pragma unroll
            for (int b = 0; b < DS; ++b) {
                if (b >= st.d_out) break;
#pragma unroll
                for (int a = 0; a < DS; ++a)
                    if (a < st.d_in) nl[a] = fmaf(ss[b * st.d_in + a], lam[b], nl[a]);
            }
        }
#pragma unroll
        for (int r = 0; r < SOUT_MAX; ++r) {
            if (r >= st.out_dim) break;
            if (st.d_in == DS) {
                axpy_row16(ys + r * DS, g[r], nl);
            } else {
#pragma unroll
                for (int a = 0; a < DS; ++a)
                    if (a < st.d_in) nl[a] = fmaf(ys[r * st.d_in + a], g[r], nl[a]);
            }
        }
#pragma unroll
        for (int a = 0; a < DS; ++a) lam[a] = nl[a];
    }
}

// 6b.  grid (nchunks * LMAX, 2): one CTA per (stage, direction): d_ss[b][a] = sum_t lam_t[b] v_t[a], d_ys[r][a] = sum_t g_t[r] v_t[a]
constexpr int BR_THREADS = 256;
constexpr int BR_LD = 196;   // floats per staged row (multiple of 4: float4 reads; 196 mod 32 = 4: the 8 lanes of a phase hit distinct bank groups)
__global__ void __launch_bounds__(BR_THREADS)
sss_tc_build_red_kernel(const sn_sss_stage* __restrict__ stages, int n, const sn_sss_tc_chunk* __restrict__ chunks, const float* __restrict__ scratch,
                        float* __restrict__ gparams) {
    __shared__ __align__(16) float Xs[(DS + SOUT_MAX) * BR_LD];
    __shared__ __align__(16) float Vt[DS * BR_LD];
    const int ch = blockIdx.x / LMAX, i = blockIdx.x % LMAX, dir = blockIdx.y;
    const sn_sss_tc_chunk c = chunks[ch];
    const int nst = c.k_end - c.k_begin;
    if (i >= nst) return;
    const sn_sss_stage st = stage_of(stages, n, dir, dir == 0 ? c.k_begin + i : c.k_end - 1 - i);
    const float* scr = scratch + ((size_t)ch * 2 + dir) * BB_SCR;
    const float* Vg = scr + (size_t)i * BB_PLANE;
    const float* Lg = scr + (size_t)(LMAX + i) * BB_PLANE;
    const float* Gg = scr + (size_t)(2 * LMAX + i) * BB_PLANE;
    const int ncol = c.ncols + DS;                 // active columns
    const int ncol4 = (ncol + 3) & ~3;
    const int nrow = DS + st.out_dim;
    for (int e = threadIdx.x; e < DS * ncol4; e += BR_THREADS) {
        const int a = e / ncol4, tt = e % ncol4;
        Vt[a * BR_LD + tt] = tt < ncol ? Vg[a * BUILD_THREADS + tt] : 0.f;
        Xs[a * BR_LD + tt] = tt < ncol ? Lg[a * BUILD_THREADS + tt] : 0.f;
    }
    for (int e = threadIdx.x; e < st.out_dim * ncol4; e += BR_THREADS) {
        const int r = e / ncol4, tt = e % ncol4;
        Xs[(DS + r) * BR_LD + tt] = tt < ncol ? Gg[r * BUILD_THREADS + tt] : 0.f;
    }
    __syncthreads();
    for (int o = threadIdx.x; o < nrow * DS; o += BR_THREADS) {
        const int rowi = o / DS, a = o % DS;
        if (a >= st.d_in || (rowi < DS && rowi >= st.d_out)) continue;
        const float4* xr = reinterpret_cast<const float4*>(Xs + rowi * BR_LD);
        const float4* vr = reinterpret_cast<const float4*>(Vt + a * BR_LD);
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        for (int q = 0; q < ncol4 / 4; ++q) {
            const float4 xv = xr[q], vv = vr[q];
            a0 = fmaf(xv.x, vv.x, a0); a1 = fmaf(xv.y, vv.y, a1); a2 = fmaf(xv.z, vv.z, a2); a3 = fmaf(xv.w, vv.w, a3);
        }
        const float acc = (a0 + a1) + (a2 + a3);
        if (rowi < DS) gparams[st.off_ss + rowi * st.d_in + a] += acc;
        else gparams[st.off_ys + (rowi - DS) * st.d_in + a] += acc;
    }
}

// ------------------------------------------------------------------------------------------
// 6'. chain rule through the chunk-matrix construction, B4_LPC threads per column, reductions fused.  grid (nchunks, 2, B4_SPLIT).
//     Phase 1 replays the construction keeping the state entering every stage in shared memory (V[stage][16][column]); phase 2 walks
//     the stages backwards (lane o of a column group owns 16 / B4_LPC adjoint components, all-gather by shuffles) and, per stage,
//     reduces d_ss[b][a] = sum_t lam_t[b] v_t[a] and d_ys[r][a] = sum_t g_t[r] v_t[a] over the CTA's columns straight from shared
//     memory (one atomic per parameter and column group) -- the 37 MB V / LAM / GY scratch round trip of kernels 6a + 6b is gone.
// ------------------------------------------------------------------------------------------
constexpr int BB4_V = LMAX * DS * B4_LD;            // floats: V[stage][a][lc]
constexpr int BB4_DM = 64 * B4_LD;                  // the CTA's columns of the chunk's dM tile
constexpr int BB4_X = 2 * (DS + SOUT_MAX) * B4_LD;  // double-buffered [lam (16 rows) ; g (16 rows)][lc]
constexpr int BB4_FIXED = BB4_V + BB4_DM + BB4_X;

__global__ void __launch_bounds__(B4_THREADS)
sss_tc_build_bwd4_kernel(const sn_sss_stage* __restrict__ stages, int n, const sn_sss_tc_chunk* __restrict__ chunks, const float* __restrict__ params,
                         const float* __restrict__ dMall, float* __restrict__ gparams) {
    extern __shared__ __align__(16) float build_smem[];
    __shared__ sn_sss_stage sdesc[LMAX];
    __shared__ StageP sptr[LMAX];
    float* Vs = build_smem;
    float* dMs = Vs + BB4_V;
    float* Xs = dMs + BB4_DM;
    float* pbuf = Xs + BB4_X;
    const sn_sss_tc_chunk c = chunks[blockIdx.x];
    const int dir = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const int lc = tid / B4_LPC, o = tid % B4_LPC;
    const int t = blockIdx.z * B4_COLS + lc;
    const bool active = lc < B4_COLS && t < c.ncols + DS;
    const bool is_in = t < c.ncols;
    const int sidx = t - c.ncols;
    const int nst = c.k_end - c.k_begin;
    const int col = c.col0 + t;
    if (blockIdx.z * B4_COLS >= c.ncols + DS) return;
    if (tid < nst) sdesc[tid] = stage_of(stages, n, dir, dir == 0 ? c.k_begin + tid : c.k_end - 1 - tid);
    {
        // the CTA's columns of dM (64 x 192 per chunk): input column t, or the state column nkb * 32 + dir * 16 + sidx
        const float* src = dMall + (size_t)blockIdx.x * 64 * DMC;
        for (int e = tid; e < 64 * B4_LD; e += B4_THREADS) {
            const int row = e / B4_LD, l = e - row * B4_LD;
            const int tt = blockIdx.z * B4_COLS + l;
            const bool ok = l < B4_COLS && tt < c.ncols + DS;
            const int cidx = tt < c.ncols ? tt : c.nkb * KBW + dir * DS + (tt - c.ncols);
            dMs[e] = ok ? __ldg(src + row * DMC + cidx) : 0.f;
        }
        // columns of V and X that no thread owns stay zero in the reductions
        for (int e = tid; e < BB4_V; e += B4_THREADS)
            if (e % B4_LD >= B4_TCOLS) Vs[e] = 0.f;
        for (int e = tid; e < BB4_X; e += B4_THREADS)
            if (e % B4_LD >= B4_TCOLS) Xs[e] = 0.f;
    }
    __syncthreads();
    chunk_params_async_q(pbuf, sptr, sdesc, nst, params, tid, B4_THREADS);
    cp_async_commit();
    cp_async_wait_all();
    __syncthreads();

    float v[DS], own[B4_NC], yv[B4_NC];
#pragma unroll
    for (int a = 0; a < DS; ++a) v[a] = (active && !is_in && a == sidx && sidx < sdesc[0].d_in) ? 1.f : 0.f;
#pragma unroll
    for (int j = 0; j < B4_NC; ++j) own[j] = (active && !is_in && B4_NC * o + j == sidx && sidx < sdesc[0].d_in) ? 1.f : 0.f;
    int my_i = -1;
    // phase 1: replay the construction, keeping the state that enters every stage
    {
        bool activated = false;
        for (int i = 0; i < nst; ++i) {
            const sn_sss_stage& st = sdesc[i];
            const int local = col - st.in_off;
            const bool mine = active && is_in && local >= 0 && local < st.in_dim;
#pragma unroll
            for (int j = 0; j < B4_NC; ++j) Vs[(i * DS + B4_NC * o + j) * B4_LD + lc] = own[j];
            const bool live = active && (!is_in || activated || mine);
            if (__any_sync(0xffffffffu, live)) stage_apply_q<false>(st, pbuf, sptr[i], v, own, yv, mine, local, o, lane);
            if (mine) { my_i = i; activated = true; }
        }
    }
    // adjoint of the state leaving the last stage: the dR / dPhi rows of dM
    float lam[DS], lown[B4_NC];
#pragma unroll
    for (int b = 0; b < DS; ++b) lam[b] = dMs[(PO + dir * DS + b) * B4_LD + lc];      // zero for inactive columns
#pragma unroll
    for (int j = 0; j < B4_NC; ++j) lown[j] = dMs[(PO + dir * DS + B4_NC * o + j) * B4_LD + lc];
    // phase 2: stages backwards
    for (int i = nst - 1; i >= 0; --i) {
        const sn_sss_stage& st = sdesc[i];
        const StageP& ps = sptr[i];
        const int local = col - st.in_off;
        const bool mine = (i == my_i);
        const bool before = is_in ? (my_i >= 0 && my_i < i) : true;
        const bool support = active && (is_in ? (dir == 0 ? (before || mine) : before) : true);
        const int rbase = st.out_off - c.row0;
        float* Xb = Xs + (i & 1) * (DS + SOUT_MAX) * B4_LD;
        float g[SOUT_MAX], gown[B4_NC];
#pragma unroll
        for (int r = 0; r < SOUT_MAX; ++r) g[r] = (r < st.out_dim && support) ? dMs[(rbase + r) * B4_LD + lc] : 0.f;
#pragma unroll
        for (int j = 0; j < B4_NC; ++j) gown[j] = (o + B4_LPC * j < st.out_dim && support) ? dMs[(rbase + o + B4_LPC * j) * B4_LD + lc] : 0.f;
#pragma unroll
        for (int j = 0; j < B4_NC; ++j) {
            Xb[(B4_NC * o + j) * B4_LD + lc] = lown[j];
            Xb[(DS + o + B4_LPC * j) * B4_LD + lc] = gown[j];
        }
        if (mine) {
#pragma unroll
            for (int j = 0; j < B4_NC; ++j) {
                const int b = B4_NC * o + j;
                if (b < st.d_out) gparams[st.off_su + b * st.in_dim + local] += lown[j];
            }
            if (st.off_yu >= 0) {
#pragma unroll
                for (int j = 0; j < B4_NC; ++j) {
                    const int r = o + B4_LPC * j;
                    if (r < st.out_dim) gparams[st.off_yu + r * st.in_dim + local] += gown[j];
                }
            }
        }
        // lambda entering the stage, components a = B4_NC o .. : ss^T lam + ys^T g
        float nl[B4_NC];
#pragma unroll
        for (int j = 0; j < B4_NC; ++j) nl[j] = 0.f;
        const float* ys = pbuf + ps.ys;
        const bool live = active && (!is_in || my_i >= 0);       // adjoints of columns whose stage lies later in the sweep stay zero
        if (__any_sync(0xffffffffu, live && (!is_in || my_i <= i))) {
            if (st.d_in == DS) {
#pragma unroll
                for (int b = 0; b < DS; ++b) {
                    if (b >= st.d_out) break;
                    const float* m = pbuf + ps.ss + ss_off(b, DS) + B4_NC * o;
#pragma unroll
                    for (int j = 0; j < B4_NC; ++j) nl[j] = fmaf(m[j], lam[b], nl[j]);
                }
#pragma unroll
                for (int r = 0; r < SOUT_MAX; ++r) {
                    if (r >= st.out_dim) break;
                    const float* m = ys + r * DS + B4_NC * o;
#pragma unroll
                    for (int j = 0; j < B4_NC; ++j) nl[j] = fmaf(m[j], g[r], nl[j]);
                }
            } else {
#pragma unroll
                for (int j = 0; j < B4_NC; ++j) {
                    const int a = B4_NC * o + j;
                    if (a >= st.d_in) continue;
                    float acc = 0.f;
#pragma unroll
                    for (int b = 0; b < DS; ++b)
                        if (b < st.d_out) acc = fmaf(pbuf[ps.ss + ss_off(b, st.d_in) + a], lam[b], acc);
#pragma unroll
                    for (int r = 0; r < SOUT_MAX; ++r)
                        if (r < st.out_dim) acc = fmaf(ys[r * st.d_in + a], g[r], acc);
                    nl[j] = acc;
                }
            }
#pragma unroll
            for (int j = 0; j < B4_NC; ++j) lown[j] = nl[j];
            group_allgather(nl, lam, lane);
        }
        __syncthreads();      // Xb complete (the other buffer was last read before the previous iteration's barrier)
        // reductions over the CTA's columns: rows 0..15 = d_ss, rows 16.. = d_ys
        const float* Vi = Vs + (size_t)i * DS * B4_LD;
        const int nout = (DS + st.out_dim) * DS;
        for (int oo = tid; oo < nout; oo += B4_THREADS) {
            const int rowi = oo >> 4, a = oo & 15;
            if (a >= st.d_in || (rowi < DS && rowi >= st.d_out)) continue;
            const float4* xr = reinterpret_cast<const float4*>(Xb + rowi * B4_LD);
            const float4* vr = reinterpret_cast<const float4*>(Vi + a * B4_LD);
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
            for (int k = 0; k < B4_LD / 4; ++k) {
                const float4 xv = xr[k], vv = vr[k];
                a0 = fmaf(xv.x, vv.x, a0); a1 = fmaf(xv.y, vv.y, a1); a2 = fmaf(xv.z, vv.z, a2); a3 = fmaf(xv.w, vv.w, a3);
            }
            const float acc = (a0 + a1) + (a2 + a3);
            if (rowi < DS) atomicAdd(gparams + st.off_ss + rowi * st.d_in + a, acc);
            else atomicAdd(gparams + st.off_ys + (rowi - DS) * st.d_in + a, acc);
        }
    }
}

// Wsum[chunk][r][c] = W_hi + W_lo (the fp32 chunk matrix [T ; R ; R'] back from its split form), for the input-gradient GEMMs
__global__ void sss_tc_wsum_kernel(const float* __restrict__ Wall, float* __restrict__ Wsum) {
    const float* W = Wall + (size_t)blockIdx.x * WROWS * WCOLS;
    float* o = Wsum + (size_t)blockIdx.x * 64 * WCOLS;
    for (int e = threadIdx.x; e < 64 * WCOLS; e += blockDim.x) o[e] = W[e] + W[64 * WCOLS + e];
}

// ------------------------------------------------------------------------------------------
// 6m. chain rule through the chunk-matrix construction on the warp-level tensor cores.  grid (nchunks, 2, BM_SPLIT), warp = tile of
//     16 columns as in the build kernel, which left the state entering every stage in VG (no replay).
//     Phase A walks the stages backwards:  lam <- lam ss + G ys  (lam = adjoint of the state; the D fragment of one product is the A
//     fragment of the next, as in the build kernel) and leaves every stage's lam in shared memory.
//     Phase B is parallel over the stages (warp w takes stages w, w + 6, ..):
//       d_ss^T[a][b] = sum_col V[col][a] lam[col][b] ,  d_ys^T[a][r] = sum_col V[col][a] G[col][r]     over the CTA's 96 columns,
//     V^T as the A operand straight from global memory, lam / G as B fragments from shared memory; the sums leave as one global
//     atomic per parameter and CTA.  G = the chunk's dM rows, staged per tile with the entries outside a column's support zeroed.
//     (A first version accumulated per-stage partial sums of every warp with shared-memory atomics inside the stage loop and was
//     slower than the SIMT kernel: 1 350 instructions per stage, 16 shared atomics per lane.)
// ------------------------------------------------------------------------------------------
constexpr int BWM_DLD = 20;                                   // pitch of a tile's dM block [64 rows][16 columns]
constexpr int BWM_DM = 64 * BWM_DLD;                          // floats per tile
constexpr int BWM_LLD = 20;                                   // pitch of the lam rows [column][16 components]
constexpr int BWM_NCOL = 16 * BM_WARPS;                       // columns per CTA (96)
constexpr int BWM_LALL = LMAX * BWM_NCOL * BWM_LLD;           // lam of every stage
constexpr int BWM_FIXED = BM_WARPS * BWM_DM + BWM_LALL;

// lam <- lam ss + G ys for one tile.  FAST: full-width stage (16 x 16 state matrix) with at most 8 outputs.
template <bool FAST>
__device__ __forceinline__ void bwm_chain_step(float (&d)[2][4], const float* pbuf, const StageP& m, const sn_sss_stage& st, const float* dMw, int rbase,
                                               int g, int t) {
    Frag3 al[2];
    split_frag(d[0], al[0]);
    split_frag(d[1], al[1]);
    const int d_in = FAST ? DS : st.d_in, d_out = FAST ? DS : st.d_out;
    const int ntr = FAST ? 1 : (st.out_dim + 7) >> 3;             // <= 2 (a stage has at most 16 outputs)
    // B fragments of both halves hp of the new adjoint: ss (k <-> b, n = a = 8 hp + g) and ys (k <-> output r, n = a); G as A fragments
    float2 sbh[2][2], sbl[2][2], ybh[2][2], ybl[2][2];
    Frag3 ag[2];
#pragma unroll
    for (int hp = 0; hp < 2; ++hp) {
        const int a = 8 * hp + g;
#pragma unroll
        for (int h = 0; h < 2; ++h) {                         // B[k <-> b][n = a] = ss[b][a]
            const int b0 = 8 * h + 2 * t;
            float x0, x1;
            if (FAST) {
                x0 = pbuf[m.ss + b0 * DS + a];
                x1 = pbuf[m.ss + (b0 + 1) * DS + a];
            } else {
                x0 = (b0 < d_out && a < d_in) ? pbuf[m.ss + b0 * d_in + a] : 0.f;
                x1 = (b0 + 1 < d_out && a < d_in) ? pbuf[m.ss + (b0 + 1) * d_in + a] : 0.f;
            }
            sbh[hp][h].x = tf32_hi(x0); sbh[hp][h].y = tf32_hi(x1); sbl[hp][h].x = mma_lo(x0 - sbh[hp][h].x); sbl[hp][h].y = mma_lo(x1 - sbh[hp][h].y);
        }
#pragma unroll
        for (int hr = 0; hr < 2; ++hr) {
            if (hr >= ntr) break;
            const int r0 = 8 * hr + 2 * t;
            const bool k0 = r0 < st.out_dim, k1 = r0 + 1 < st.out_dim;
            const float x0 = (k0 && a < d_in) ? pbuf[m.ys + r0 * d_in + a] : 0.f;
            const float x1 = (k1 && a < d_in) ? pbuf[m.ys + (r0 + 1) * d_in + a] : 0.f;
            ybh[hp][hr].x = tf32_hi(x0); ybh[hp][hr].y = tf32_hi(x1); ybl[hp][hr].x = mma_lo(x0 - ybh[hp][hr].x); ybl[hp][hr].y = mma_lo(x1 - ybh[hp][hr].y);
        }
    }
#pragma unroll
    for (int hr = 0; hr < 2; ++hr) {                          // G as an A fragment (rows = columns g, g + 8; k <-> outputs r0, r0 + 1)
        if (hr >= ntr) break;
        const int r0 = 8 * hr + 2 * t;
        const bool k0 = r0 < st.out_dim, k1 = r0 + 1 < st.out_dim;
        const float ga0 = k0 ? dMw[(rbase + r0) * BWM_DLD + g] : 0.f, gb0 = k0 ? dMw[(rbase + r0) * BWM_DLD + g + 8] : 0.f;
        const float ga1 = k1 ? dMw[(rbase + r0 + 1) * BWM_DLD + g] : 0.f, gb1 = k1 ? dMw[(rbase + r0 + 1) * BWM_DLD + g + 8] : 0.f;
        frag_a_from(make_float2(ga0, ga1), make_float2(gb0, gb1), ag[hr]);
    }
    // four independent accumulators (lam ss and G ys, for each half of the new adjoint), products issued round-robin
    float rs[2][4], rg[2][4];
#pragma unroll
    for (int hp = 0; hp < 2; ++hp)
#pragma unroll
        for (int k = 0; k < 4; ++k) { rs[hp][k] = 0.f; rg[hp][k] = 0.f; }
    const bool g0on = ntr > 0, g1on = ntr > 1;
#define SN_ROUND(TERM, H)                                                                              \
    mma_t<TERM>(rs[0], al[H], sbh[0][H], sbl[0][H]); mma_t<TERM>(rs[1], al[H], sbh[1][H], sbl[1][H]);  \
    if (H == 0 ? g0on : g1on) { mma_t<TERM>(rg[0], ag[H], ybh[0][H], ybl[0][H]); mma_t<TERM>(rg[1], ag[H], ybh[1][H], ybl[1][H]); }
    SN_ROUND(0, 0) SN_ROUND(1, 0) SN_ROUND(2, 0) SN_ROUND(0, 1) SN_ROUND(1, 1) SN_ROUND(2, 1)
#undef SN_ROUND
#pragma unroll
    for (int hp = 0; hp < 2; ++hp)
#pragma unroll
        for (int k = 0; k < 4; ++k) d[hp][k] = rs[hp][k] + rg[hp][k];
}

__global__ void __launch_bounds__(BM_THREADS)
sss_tc_build_bwdm_kernel(const sn_sss_stage* __restrict__ stages, int n, const sn_sss_tc_chunk* __restrict__ chunks, const float* __restrict__ params,
                         const float* __restrict__ dMall, const float* __restrict__ VG, float* __restrict__ gparams, int lists_contiguous) {
    extern __shared__ __align__(16) float build_smem[];
    __shared__ sn_sss_stage sdesc[LMAX];
    __shared__ StageP smt[LMAX];
    __shared__ int rowst[PO];          // sweep position of the stage that owns each output row of the chunk (-1: padding row)
    float* dMs = build_smem;
    float* Lall = dMs + BM_WARPS * BWM_DM;
    float* pbuf = Lall + BWM_LALL;
    const sn_sss_tc_chunk c = chunks[blockIdx.x];
    const int dir = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int nst = c.k_end - c.k_begin;
    if (tid < nst) sdesc[tid] = stage_of(stages, n, dir, dir == 0 ? c.k_begin + tid : c.k_end - 1 - tid);
    __syncthreads();
    if (tid < PO) {
        int ir = -1;
        for (int i = 0; i < nst; ++i) {
            const int rl = c.row0 + tid - sdesc[i].out_off;
            if (rl >= 0 && rl < sdesc[i].out_dim) ir = i;
        }
        rowst[tid] = ir;
    }
    if (lists_contiguous) chunk_params_ranges(pbuf, smt, sdesc, nst, params, tid, BM_THREADS);
    else chunk_params_async(pbuf, smt, sdesc, nst, params, tid, BM_THREADS);
    cp_async_commit();
    __syncthreads();

    const int tile = BM_SPLIT * warp + blockIdx.z;
    const bool state_tile = tile == BM_TILES - 1;
    const bool has_tile = tile < BM_TILES && (state_tile || 16 * tile < c.ncols);
    float* dMw = dMs + warp * BWM_DM;
    // the warp's 16 columns of the chunk's dM tile; T rows (stage outputs) are kept only where the column has support:
    // causal sweep: rows of the column's own stage and of later stages; anticausal sweep: rows of stages strictly after it in the sweep
    {
        const float* src = dMall + (size_t)blockIdx.x * 64 * DMC;
        const int l = lane & 15;
        const int tcol = state_tile ? l : 16 * tile + l;
        const bool ok = has_tile && (state_tile || tcol < c.ncols);
        const int cidx = state_tile ? c.nkb * KBW + dir * DS + l : tcol;
        int ic = -1;
        if (ok && !state_tile)
            for (int i = 0; i < nst; ++i) {
                const int cl = c.col0 + tcol - sdesc[i].in_off;
                if (cl >= 0 && cl < sdesc[i].in_dim) ic = i;
            }
#pragma unroll 8
        for (int row = lane >> 4; row < 64; row += 2) {
            float v = ok ? __ldg(src + row * DMC + cidx) : 0.f;
            if (ok && !state_tile && row < PO) {
                const int ir = rowst[row];
                const bool keep = ir >= 0 && ic >= 0 && (dir == 0 ? ic <= ir : ic < ir);
                if (!keep) v = 0.f;
            }
            dMw[row * BWM_DLD + l] = v;
        }
    }
    cp_async_wait_all();
    __syncthreads();
    // ---- phase A: the adjoint chain of the warp's tile; lam of every stage goes to Lall[stage][16 warp + column][component] ----
    {
        int tcol[2], my_i[2];
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            tcol[rr] = state_tile ? g + 8 * rr : 16 * tile + g + 8 * rr;
            my_i[rr] = -1;
            if (has_tile && !state_tile && tcol[rr] < c.ncols)
                for (int i = 0; i < nst; ++i) {
                    const int cl = c.col0 + tcol[rr] - sdesc[i].in_off;
                    if (cl >= 0 && cl < sdesc[i].in_dim) my_i[rr] = i;
                }
        }
        // adjoint of the state leaving the last stage: the dR / dPhi rows of dM, as the D fragment (column g / g + 8, components 2t, 2t+1)
        float d[2][4];
#pragma unroll
        for (int hp = 0; hp < 2; ++hp)
#pragma unroll
            for (int k = 0; k < 4; ++k) d[hp][k] = dMw[(PO + dir * DS + 8 * hp + 2 * t + (k & 1)) * BWM_DLD + g + 8 * (k >> 1)];
        for (int i = nst - 1; i >= 0; --i) {
            const sn_sss_stage& st = sdesc[i];
            const StageP& m = smt[i];
            const int rbase = st.out_off - c.row0;
            float* Li = Lall + ((size_t)i * BWM_NCOL + 16 * warp) * BWM_LLD;
#pragma unroll
            for (int hp = 0; hp < 2; ++hp) {
                *reinterpret_cast<float2*>(Li + g * BWM_LLD + 8 * hp + 2 * t) = make_float2(d[hp][0], d[hp][1]);
                *reinterpret_cast<float2*>(Li + (g + 8) * BWM_LLD + 8 * hp + 2 * t) = make_float2(d[hp][2], d[hp][3]);
            }
            if (!has_tile) continue;                       // (warp-uniform) nothing but zeros in this tile
            // parameter gradients that belong to single columns: d su[b][local] = lam[col][b], d yu[r][local] = G[col][r]
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
                if (i != my_i[rr]) continue;
                const int local = c.col0 + tcol[rr] - st.in_off;
#pragma unroll
                for (int hp = 0; hp < 2; ++hp)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int b = 8 * hp + 2 * t + e;
                        if (b < st.d_out) atomicAdd(gparams + st.off_su + b * st.in_dim + local, d[hp][2 * rr + e]);   // RED: no load on the chain
                    }
                if (st.off_yu >= 0)
                    for (int r = t; r < st.out_dim; r += 4) atomicAdd(gparams + st.off_yu + r * st.in_dim + local, dMw[(rbase + r) * BWM_DLD + g + 8 * rr]);
            }
            if (i == 0) break;                              // the adjoint entering the first stage is not needed
            if (st.d_in == DS && st.d_out == DS && st.out_dim <= 8) bwm_chain_step<true>(d, pbuf, m, st, dMw, rbase, g, t);
            else bwm_chain_step<false>(d, pbuf, m, st, dMw, rbase, g, t);
        }
    }
    __syncthreads();
    // ---- phase B: stage-parallel reductions over the CTA's columns ----
    for (int i = warp; i < nst; i += BM_WARPS) {
        const sn_sss_stage& st = sdesc[i];
        const int rbase = st.out_off - c.row0;
        const int ntr = (st.out_dim + 7) >> 3;
        const float* Li = Lall + (size_t)i * BWM_NCOL * BWM_LLD;
        float rss[2][4], rys[2][4];
#pragma unroll
        for (int hn = 0; hn < 2; ++hn)
#pragma unroll
            for (int k = 0; k < 4; ++k) { rss[hn][k] = 0.f; rys[hn][k] = 0.f; }
        // A = V^T: [m = component][k = column], straight from global memory (L2): ALL of the stage's fragments are requested before the
        // first product -- loaded where they were used, each of the twelve (tile, k-step) rounds waited a full L2 round trip (ncu r2v:
        // 47 % of the kernel's samples on the first use of va)
        float va[BM_WARPS][2][4];
        bool tile_on[BM_WARPS];
#pragma unroll
        for (int w2 = 0; w2 < BM_WARPS; ++w2) {
            const int tile2 = BM_SPLIT * w2 + blockIdx.z;
            tile_on[w2] = tile2 < BM_TILES && (tile2 == BM_TILES - 1 || 16 * tile2 < c.ncols);
            const float* vi = VG + (((size_t)(blockIdx.x * 2 + dir) * LMAX + i) * COLT + 16 * (tile_on[w2] ? tile2 : 0)) * DS;
#pragma unroll
            for (int hk = 0; hk < 2; ++hk) {
                va[w2][hk][0] = tile_on[w2] ? __ldg(vi + (8 * hk + t) * DS + g) : 0.f;
                va[w2][hk][1] = tile_on[w2] ? __ldg(vi + (8 * hk + t) * DS + g + 8) : 0.f;
                va[w2][hk][2] = tile_on[w2] ? __ldg(vi + (8 * hk + t + 4) * DS + g) : 0.f;
                va[w2][hk][3] = tile_on[w2] ? __ldg(vi + (8 * hk + t + 4) * DS + g + 8) : 0.f;
            }
        }
#pragma unroll
        for (int w2 = 0; w2 < BM_WARPS; ++w2) {            // the tile of warp w2
            if (!tile_on[w2]) continue;
            const float* dM2 = dMs + w2 * BWM_DM;
            const float* L2 = Li + 16 * w2 * BWM_LLD;
#pragma unroll
            for (int hk = 0; hk < 2; ++hk) {
                Frag3 av;
#pragma unroll
                for (int q4 = 0; q4 < 4; ++q4) {
                    const float h = tf32_hi(va[w2][hk][q4]);
                    av.hi[q4] = __float_as_uint(h);
                    av.lo[q4] = __float_as_uint(mma_lo(va[w2][hk][q4] - h));
                }
                // four independent accumulators (two halves of d_ss, up to two of d_ys), products issued round-robin
                float2 lbh[2], lbl[2], gbh[2], gbl[2];
#pragma unroll
                for (int hn = 0; hn < 2; ++hn) {
                    const float x0 = L2[(8 * hk + t) * BWM_LLD + 8 * hn + g], x1 = L2[(8 * hk + t + 4) * BWM_LLD + 8 * hn + g];
                    lbh[hn].x = tf32_hi(x0); lbh[hn].y = tf32_hi(x1); lbl[hn].x = mma_lo(x0 - lbh[hn].x); lbl[hn].y = mma_lo(x1 - lbh[hn].y);
                }
#pragma unroll
                for (int hn = 0; hn < 2; ++hn) {
                    if (hn >= ntr) break;
                    const int r = 8 * hn + g;
                    const float x0 = r < st.out_dim ? dM2[(rbase + r) * BWM_DLD + 8 * hk + t] : 0.f;
                    const float x1 = r < st.out_dim ? dM2[(rbase + r) * BWM_DLD + 8 * hk + t + 4] : 0.f;
                    gbh[hn].x = tf32_hi(x0); gbh[hn].y = tf32_hi(x1); gbl[hn].x = mma_lo(x0 - gbh[hn].x); gbl[hn].y = mma_lo(x1 - gbh[hn].y);
                }
#define SN_ROUND(TERM)                                                                     \
                mma_t<TERM>(rss[0], av, lbh[0], lbl[0]); mma_t<TERM>(rss[1], av, lbh[1], lbl[1]); \
                if (ntr > 0) mma_t<TERM>(rys[0], av, gbh[0], gbl[0]);                             \
                if (ntr > 1) mma_t<TERM>(rys[1], av, gbh[1], gbl[1]);
                SN_ROUND(0) SN_ROUND(1) SN_ROUND(2)
#undef SN_ROUND
            }
        }
        // D fragments: rows a = g, g + 8; columns 8 hn + 2t, + 1 (b of d_ss, r of d_ys)
#pragma unroll
        for (int hn = 0; hn < 2; ++hn)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int a = g + 8 * (k >> 1), x = 8 * hn + 2 * t + (k & 1);
                if (a < st.d_in) {
                    if (x < st.d_out) atomicAdd(gparams + st.off_ss + x * st.d_in + a, rss[hn][k]);
                    if (x < st.out_dim) atomicAdd(gparams + st.off_ys + x * st.d_in + a, rys[hn][k]);
                }
            }
    }
}

inline float* vg_of(const sn_sss_tc_plan* p, const float* coef) {
    return const_cast<float*>(coef) + (size_t)p->nchunks * (WROWS * WCOLS + SCF + 4 * CW_TILE_FLOATS);
}
// fragment tiles of the warp-level tensor-core scans, behind VG
inline float* fs_of(const sn_sss_tc_plan* p, const float* coef) { return vg_of(p, coef) + (size_t)p->nchunks * 2 * LMAX * COLT * DS; }

int check_tc_plan(const sn_sss_tc_plan* p) {
    SN_CHECK_ARG(p != nullptr, "sss_tc: NULL plan");
    SN_CHECK_ARG(p->nb_states > 0 && p->input_dim > 0 && p->output_dim > 0 && p->nchunks > 0, "sss_tc: non-positive plan dimension");
    SN_CHECK_ARG(p->stages != nullptr && p->chunks != nullptr, "sss_tc: plan tables missing");
    SN_CHECK_ARG(p->input_dim % 4 == 0, "sss_tc: input_dim must be a multiple of 4 (TMA row pitch)");
    SN_CHECK_ARG(p->nchunks <= G1_MAX_CHUNKS, "sss_tc: more than %d chunks", G1_MAX_CHUNKS);
    SN_CHECK_ARG(p->chunk_param_floats > 0 && p->chunk_param_floats <= 40960, "sss_tc: chunk_param_floats must be in 1..40960 (got %d)", p->chunk_param_floats);
    return 0;
}

int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

// whole tiles per CTA only pay once there are enough tiles to fill most of the chip; below that the (tile, chunk) grid of the
// three-kernel path has more parallelism.  SNB200_SSS_TC_FUSED=0/1 forces the choice (tests).
bool use_fused_forward(const sn_sss_tc_plan* p, int64_t B) {
    if (p->nchunks > F_MAX_CHUNKS) return false;
    const char* e = getenv("SNB200_SSS_TC_FUSED");
    if (e != nullptr && (e[0] == '0' || e[0] == '1')) return e[0] == '1';
    (void)B;
    return false;   // the three-kernel path with the four-threads-per-sample scans is faster at every batch size measured so far
}

// small-batch scans on the warp-level tensor cores (default) or the SIMT four-threads-per-sample kernels (SNB200_SSS_SCAN=simt)
bool use_mma_scans() {
    const char* e = getenv("SNB200_SSS_SCAN");
    return !(e != nullptr && e[0] == 's');
}

// Chunk scans.  The warp-level tensor-core scans (sss_tc_scan_*_m) are the default at every batch size since round 2: they move 20 KB
// per sample where the tcgen05 chain kernels move 24 (no ytmp round trip), are not quantised into waves of 128-sample tiles, and run
// at the HBM roof at large batches.  Measured whole steps (r2zg/r2zh, scans vs chain): 16 384 samples 0.364 vs 0.399 ms, 32 768: 0.651
// vs 0.656, 65 536: 1.216 vs 1.228 (before the bias sums moved into the adjoint scan).  The chain kernels remain for layers whose rows
// are not 16-byte aligned (the SIMT scans are slower than the chain above ~10 k samples) and behind SNB200_SSS_TC_CHAIN=1 (tests).
bool use_tc_chain(int64_t B, bool rows_aligned) {
    const char* e = getenv("SNB200_SSS_TC_CHAIN");
    if (e != nullptr && (e[0] == '0' || e[0] == '1')) return e[0] == '1';
    if (use_mma_scans() && rows_aligned) return false;
    return B >= 10240;
}

// build / build-backward: 2 = warp-level tensor-core kernels (default), 1 = SIMT with several lanes per column
// (SNB200_SSS_BUILD=quad), 0 = SIMT with one thread per column (SNB200_SSS_BUILD=col)
int build_mode() {
    const char* e = getenv("SNB200_SSS_BUILD");
    if (e != nullptr && e[0] == 'c') return 0;
    if (e != nullptr && e[0] == 'q') return 1;
    return 2;
}
bool use_quad_build() { return build_mode() >= 1; }

// SIMT scans: split by direction (+ a parallel output kernel) by default; SNB200_SSS_SPLIT_SCANS=0 keeps the single-kernel scans
bool use_split_scans(int64_t B) {
    (void)B;
    const char* e = getenv("SNB200_SSS_SPLIT_SCANS");
    return !(e != nullptr && e[0] == '0');
}

}  // namespace

extern "C" {

size_t sn_sss_tc_coef_floats(const sn_sss_tc_plan* p) {
    if (p == nullptr) return 0;
    // W | SC | chain tiles | VG: the states entering every stage of every chunk's construction (tensor-core build -> its backward) |
    // FS: fragment tiles of the small-batch scans
    return (size_t)p->nchunks * (WROWS * WCOLS + SCF + 4 * CW_TILE_FLOATS) + (size_t)p->nchunks * 2 * LMAX * COLT * DS +
           (size_t)p->nchunks * 2 * FS_TILE_FLOATS;
}
size_t sn_sss_tc_rbuf_floats(const sn_sss_tc_plan* p, int64_t B) {
    if (p == nullptr || B <= 0 || use_fused_forward(p, B)) return 0;
    return (size_t)p->nchunks * B * 64;
}
size_t sn_sss_tc_states_floats(const sn_sss_tc_plan* p, int64_t B) { return p == nullptr || B <= 0 ? 0 : (size_t)p->nchunks * B * 32; }
size_t sn_sss_tc_backward_workspace_floats(const sn_sss_tc_plan* p, int64_t B) {
    if (p == nullptr || B <= 0) return 0;
    // adjoints L | dM | per-stage scratch of the one-thread-per-column build-backward kernels | W_hi + W_lo (input gradient only)
    return (size_t)p->nchunks * B * 32 + (size_t)p->nchunks * 64 * DMC + (size_t)p->nchunks * 2 * BB_SCR + (size_t)p->nchunks * 64 * WCOLS;
}

int sn_sss_tc_build(const sn_sss_tc_plan* p, const float* params, float* coef, sn_stream_t stream) {
    if (int rc = check_tc_plan(p)) return rc;
    SN_CHECK_ARG(params && coef, "sss_tc_build: NULL buffer");
    float* W = coef;
    float* SC = coef + (size_t)p->nchunks * WROWS * WCOLS;
    if (build_mode() == 2) {
        const size_t bsm = ((size_t)p->chunk_param_floats + 32) * sizeof(float);     // four contiguous list ranges, each with <= 3 floats of lead-in
        SN_SET_MAX_SMEM((int)bsm, sss_tc_buildm_kernel);
        SN_LAUNCH("sss_tc_buildm_kernel", snb::as_stream(stream), sss_tc_buildm_kernel<<<dim3(p->nchunks, 2, BM_SPLIT), BM_THREADS, bsm, snb::as_stream(stream)>>>(p->stages, p->nb_states, p->chunks, params, W, SC, vg_of(p, coef), p->reserved[0]));
    } else if (use_quad_build()) {
        const size_t bsm = ((size_t)p->chunk_param_floats + B4_LPC * LMAX * 4) * sizeof(float);    // + the bank padding of the state matrices
        SN_SET_MAX_SMEM((int)bsm, sss_tc_build4_kernel);
        SN_LAUNCH("sss_tc_build4_kernel", snb::as_stream(stream), sss_tc_build4_kernel<<<dim3(p->nchunks, 2, B4_SPLIT), B4_THREADS, bsm, snb::as_stream(stream)>>>(p->stages, p->nb_states, p->chunks, params, W, SC));
    } else {
        const size_t bsm = (size_t)p->chunk_param_floats * sizeof(float);
        SN_SET_MAX_SMEM((int)bsm, sss_tc_build_kernel);
        SN_LAUNCH("sss_tc_build_kernel", snb::as_stream(stream), sss_tc_build_kernel<<<dim3(p->nchunks, 2), BUILD_THREADS, bsm, snb::as_stream(stream)>>>(p->stages, p->nb_states, p->chunks, params, W, SC));
    }
    // the chain tiles (tensor-core chunk scans of large batches) are packed by sn_sss_tc_forward, next to its local GEMM
    return 0;
}

int sn_sss_tc_forward(const sn_sss_tc_plan* p, const float* coef, const float* x, int64_t ldx, float* y, int64_t ldy, const float* bias,
                      float* rbuf, float* states, int64_t B, sn_stream_t stream) {
    if (int rc = check_tc_plan(p)) return rc;
    SN_CHECK_ARG(coef, "sss_tc_forward: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && y && states, "sss_tc_forward: NULL buffer");
    SN_CHECK_ARG(ldx >= p->input_dim && ldy >= p->output_dim, "sss_tc_forward: leading dimension too small");
    cudaStream_t st = snb::as_stream(stream);
    const float* W = coef;
    const float* SC = coef + (size_t)p->nchunks * WROWS * WCOLS;
    CUtensorMap mx, mw;
    if (int rc = make_map_f32(&mx, x, (uint64_t)p->input_dim, (uint64_t)B, (uint64_t)ldx, 128, 0, 0, false, 32, true)) return rc;
    if (int rc = make_map_f32(&mw, W, (uint64_t)WCOLS, (uint64_t)p->nchunks * WROWS, (uint64_t)WCOLS, 128)) return rc;
    const int ntiles = (int)((B + 127) / 128);
    const int aligned = ((reinterpret_cast<uintptr_t>(y) & 15) == 0 && (ldy & 3) == 0 && (bias == nullptr || (reinterpret_cast<uintptr_t>(bias) & 15) == 0) &&
                         p->rows_aligned) ? 1 : 0;
    if (use_fused_forward(p, B)) {
        const int grid = ntiles < sm_count() ? ntiles : sm_count();
        SN_SET_MAX_SMEM((int)F_SMEM, sss_tc_fwd_fused_kernel);
        SN_LAUNCH("sss_tc_fwd_fused_kernel", st, sss_tc_fwd_fused_kernel<<<grid, F_THREADS, F_SMEM, st>>>(mx, mw, p->chunks, p->nchunks, (long)B, ntiles, SC, states, y, (long)ldy, bias, aligned));
        if (use_tc_chain(B, p->rows_aligned != 0)) {     // the backward's chain kernel reads the packed tiles
            float* CWp = const_cast<float*>(SC) + (size_t)p->nchunks * SCF;
            SN_LAUNCH("sss_tc_pack_chain_kernel", st, sss_tc_pack_chain_kernel<<<dim3(p->nchunks, 4), 256, 0, st>>>(SC, CWp));
        } else if (use_mma_scans()) {
            SN_LAUNCH("sss_tc_pack_scan_kernel", st, sss_tc_pack_scan_kernel<<<dim3(p->nchunks, 2), 256, 0, st>>>(SC, fs_of(p, coef)));
        }
        return 0;
    }
    SN_CHECK_ARG(rbuf != nullptr, "sss_tc_forward: rbuf is NULL");
    const long total = (long)ntiles * p->nchunks;
    const int grid = (int)(total < sm_count() ? total : sm_count());
    SN_SET_MAX_SMEM((int)G1_SMEM, sss_tc_local_gemm_kernel);
    CUtensorMap moy, mor;   // output boxes: Y [chunk][B][32], then R [chunk][B][16] and R' [chunk][B][16] back to back (chunk index nchunks + ch)
    {
        const uint64_t NBo = (uint64_t)p->nchunks * B;
        if (int rc = make_map_f32(&moy, rbuf, 32, (uint64_t)B, 32, 128, (uint64_t)p->nchunks, (uint64_t)B * 32)) return rc;
        if (int rc = make_map_f32(&mor, rbuf + NBo * 32, 16, (uint64_t)B, 16, 128, (uint64_t)2 * p->nchunks, (uint64_t)B * 16, false, 16)) return rc;
    }
    // the scans' coefficient tiles (chain tiles of the tcgen05 chain kernels, or fragment tiles of the warp-level scans) are packed on a
    // second stream while the local GEMM runs (they are not needed before the scans)
    const bool pack_fs = !use_tc_chain(B, p->rows_aligned != 0) && use_mma_scans();     // the backward's adjoint scan reads them whatever y's alignment is
    const bool mma_scans = pack_fs && aligned && ((reinterpret_cast<uintptr_t>(y) & 7) == 0) && (ldy & 1) == 0;
    snb::SideStream* sd = (use_tc_chain(B, p->rows_aligned != 0) || pack_fs) ? snb::side_stream() : nullptr;
    if (use_tc_chain(B, p->rows_aligned != 0) || pack_fs) {
        float* CWp = const_cast<float*>(SC) + (size_t)p->nchunks * SCF;
        float* FSp = fs_of(p, coef);
        cudaStream_t s2 = st;
        if (sd != nullptr) {
            SN_CHECK_CUDA(cudaEventRecord(sd->fork, st));
            SN_CHECK_CUDA(cudaStreamWaitEvent(sd->stream, sd->fork, 0));
            s2 = sd->stream;
        }
        if (sd != nullptr) {   // no per-kernel timing events on the side stream: its span would cover the concurrent local GEMM
            if (pack_fs) sss_tc_pack_scan_kernel<<<dim3(p->nchunks, 2), 256, 0, s2>>>(SC, FSp);
            else sss_tc_pack_chain_kernel<<<dim3(p->nchunks, 4), 256, 0, s2>>>(SC, CWp);
            SN_CHECK_LAUNCH("sss_tc_pack_chain_kernel");
            SN_CHECK_CUDA(cudaEventRecord(sd->join, sd->stream));
        } else if (pack_fs) {
            SN_LAUNCH("sss_tc_pack_scan_kernel", s2, sss_tc_pack_scan_kernel<<<dim3(p->nchunks, 2), 256, 0, s2>>>(SC, FSp));
        } else {
            SN_LAUNCH("sss_tc_pack_chain_kernel", s2, sss_tc_pack_chain_kernel<<<dim3(p->nchunks, 4), 256, 0, s2>>>(SC, CWp));
        }
    }
    SN_LAUNCH("sss_tc_local_gemm_kernel", st, sss_tc_local_gemm_kernel<<<grid, G1_THREADS, G1_SMEM, st>>>(mx, mw, moy, mor, p->chunks, p->nchunks, (long)B, ntiles));
    if (sd != nullptr) SN_CHECK_CUDA(cudaStreamWaitEvent(st, sd->join, 0));
    if (use_tc_chain(B, p->rows_aligned != 0)) {
        CUtensorMap mc;
        const float* CW = SC + (size_t)p->nchunks * SCF;
        if (int rc = make_map_f32(&mc, CW, 32, (uint64_t)p->nchunks * 4 * CW_ROWS, 32, CW_ROWS)) return rc;
        CUtensorMap mi, my;
        SN_CHECK_ARG((long)p->nchunks * B < 2147483647L, "sss_tc_forward: nchunks * B exceeds the TMA coordinate range");
        const uint64_t NB = (uint64_t)p->nchunks * B;
        SN_CHECK_ARG(2 * NB < 2147483647ULL, "sss_tc_forward: 2 * nchunks * B exceeds the TMA coordinate range");
        if (int rc = make_map_f32(&mi, rbuf + NB * 32, 16, 2 * NB, 16, 128, 0, 0, false, 16)) return rc;   // R rows, then R' rows
        if (int rc = make_map_f32(&my, rbuf, 32, NB, 32, 128)) return rc;                                     // yloc / ytmp rows
        SN_SET_MAX_SMEM((int)CHF_SMEM, sss_tc_chain_fwd_kernel);
        SN_LAUNCH("sss_tc_chain_fwd_kernel", st, sss_tc_chain_fwd_kernel<<<ntiles, CH_THREADS, CHF_SMEM, st>>>(mc, mi, my, p->chunks, p->nchunks, rbuf, states, y, (long)ldy, bias, (long)B, aligned));
        return 0;
    }
    if (mma_scans) {
        SN_LAUNCH("sss_tc_scan_states_m_kernel", st, sss_tc_scan_states_m_kernel<<<dim3((unsigned)((B + 63) / 64), 2), SM_THREADS, 0, st>>>(p->nchunks, fs_of(p, coef), rbuf, states, (long)B));
        SN_LAUNCH("sss_tc_scan_out_m_kernel", st, sss_tc_scan_out_m_kernel<<<dim3((unsigned)((B + 64 * QMO_SUB - 1) / (64 * QMO_SUB)), p->nchunks), SM_THREADS, 0, st>>>(p->chunks, SC, rbuf, states, y, (long)ldy, bias, (long)B));
        return 0;
    }
    const int qs_threads = B <= 16384 ? 64 : QS_THREADS;
    if (use_split_scans(B)) {
        SN_LAUNCH("sss_tc_scan_states_q_kernel", st, sss_tc_scan_states_q_kernel<<<dim3((unsigned)((B + qs_threads / 4 - 1) / (qs_threads / 4)), 2), qs_threads, 0, st>>>(p->nchunks, SC, rbuf, states, (long)B));
        SN_LAUNCH("sss_tc_scan_out_q_kernel", st, sss_tc_scan_out_q_kernel<<<dim3((unsigned)((B + 31) / 32), p->nchunks), QS_THREADS, 0, st>>>(p->chunks, SC, rbuf, states, y, (long)ldy, bias, (long)B, aligned));
        return 0;
    }
    SN_LAUNCH("sss_tc_scan_fwd_q_kernel", st, sss_tc_scan_fwd_q_kernel<<<(unsigned)((B + qs_threads / 4 - 1) / (qs_threads / 4)), qs_threads, 0, st>>>(p->chunks, p->nchunks, SC, rbuf, states, y,
                                                                                                             (long)ldy, bias, (long)B, aligned));
    return 0;
}

int sn_sss_tc_backward(const sn_sss_tc_plan* p, const float* params, const float* coef, const float* x, int64_t ldx, const float* grad_y,
                       int64_t ldgy, const float* states, float* workspace, float* grad_params, float* grad_bias, float* grad_x, int64_t ldgx,
                       int64_t B, sn_stream_t stream) {
    if (int rc = check_tc_plan(p)) return rc;
    SN_CHECK_ARG(params && coef, "sss_tc_backward: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && grad_y && states && workspace, "sss_tc_backward: NULL buffer");
    SN_CHECK_ARG(grad_params != nullptr || grad_x != nullptr, "sss_tc_backward: grad_params and grad_x are both NULL (nothing to compute)");
    SN_CHECK_ARG(ldx >= p->input_dim && ldgy >= p->output_dim, "sss_tc_backward: leading dimension too small");
    SN_CHECK_ARG((ldgy & 3) == 0 && (reinterpret_cast<uintptr_t>(grad_y) & 15) == 0, "sss_tc_backward: grad_y must be 16-byte aligned with a row pitch multiple of 4");
    SN_CHECK_ARG(grad_x == nullptr || ldgx >= p->input_dim, "sss_tc_backward: grad_x leading dimension too small");
    cudaStream_t st = snb::as_stream(stream);
    const float* SC = coef + (size_t)p->nchunks * WROWS * WCOLS;
    float* L = workspace;
    float* dM = L + (size_t)p->nchunks * B * 32;
    float* scratch = dM + (size_t)p->nchunks * 64 * DMC;
    const int aligned = p->rows_aligned ? 1 : 0;
    snb::SideStream* bias_side = nullptr;
    bool bias_later = false;
    if (use_tc_chain(B, p->rows_aligned != 0)) {
        CUtensorMap mc;
        const float* CW = SC + (size_t)p->nchunks * SCF;
        CUtensorMap mgy;
        if (int rc = make_map_f32(&mgy, grad_y, (uint64_t)p->output_dim, (uint64_t)B, (uint64_t)ldgy, 128)) return rc;
        if (int rc = make_map_f32(&mc, CW, 32, (uint64_t)p->nchunks * 4 * CW_ROWS, 32, 64)) return rc;   // state + grad_y sub-tiles only
        SN_SET_MAX_SMEM((int)CHB_SMEM, sss_tc_chain_bwd_kernel);
        SN_LAUNCH("sss_tc_chain_bwd_kernel", st, sss_tc_chain_bwd_kernel<<<dim3((unsigned)((B + 127) / 128), 2), CHB_THREADS, CHB_SMEM, st>>>(mc, mgy, p->chunks, p->nchunks, L, grad_bias, (long)B));
        if (p->nchunks == 1 && grad_bias != nullptr)
            if (int rc = snb::colsum_accumulate(grad_y, ldgy, B, p->output_dim, grad_bias, st)) return rc;
    } else if (use_mma_scans() && aligned) {
        // the bias gradient rides on the adjoint scan (it stages every grad_y row in shared memory); layers with so many chunks that the
        // per-CTA sums do not fit two CTAs per SM take the separate column-sum kernel beside the build-backward kernel instead
        SN_CHECK_ARG((B + 63) / 64 <= 65535, "sss_tc_backward: batch too large for the adjoint scan's grid (4 193 280 samples)");
        const unsigned nblk64 = (unsigned)((B + 63) / 64);
        // ring depth: 6 while the batch is one wave of CTAs at two per SM, 3 above that (four CTAs per SM); SNB200_SSS_SCAN_RING=2|3|6 forces
        // one (measurements: depth 2 = five CTAs per SM)
        int ring = 2 * nblk64 <= 2u * (unsigned)sm_count() ? 6 : 3;
        {
            const char* e = getenv("SNB200_SSS_SCAN_RING");
            if (e != nullptr && (e[0] == '2' || e[0] == '3' || e[0] == '6')) ring = e[0] - '0';
        }
        const size_t sb_smem = sb_smem_bytes(ring) + (size_t)(SM_THREADS / 32) * ((p->nchunks + 1) / 2) * 32 * sizeof(float);
        const bool bias_fused = grad_bias != nullptr && sb_smem <= (ring == 6 ? 110 : 56) * 1024;
        bias_later = grad_bias != nullptr && !bias_fused;
#define SN_SCAN_BWD(R)                                                                                                                  \
        do {                                                                                                                            \
            SN_SET_MAX_SMEM((int)sb_smem, sss_tc_scan_bwd_m_kernel<R>);                                                                 \
            SN_LAUNCH("sss_tc_scan_bwd_m_kernel", st, sss_tc_scan_bwd_m_kernel<R><<<dim3(2, nblk64), SM_THREADS, sb_smem, st>>>(        \
                p->chunks, p->nchunks, fs_of(p, coef), grad_y, (long)ldgy, L, bias_fused ? grad_bias : nullptr, (long)B));              \
        } while (0)
        if (ring == 6) SN_SCAN_BWD(6);
        else if (ring == 3) SN_SCAN_BWD(3);
        else SN_SCAN_BWD(2);
#undef SN_SCAN_BWD
    } else {
        const int qs_threads = B <= 16384 ? 64 : QS_THREADS;
        const unsigned ydim = use_split_scans(B) ? 2u : 1u;
        SN_LAUNCH("sss_tc_scan_bwd_q_kernel", st, sss_tc_scan_bwd_q_kernel<<<dim3((unsigned)((B + qs_threads / 4 - 1) / (qs_threads / 4)), ydim), qs_threads, 0, st>>>(p->chunks, p->nchunks, SC, grad_y, (long)ldgy,
                                                                                                                             L, grad_bias, (long)B, aligned));
    }
    if (grad_x != nullptr) {
        // grad_u_j = [gy_j | lambda_{j+1} | mu_j] W_j  (W_j = [T_j ; R_j ; R'_j], 64 x 160): two small tensor-core GEMMs per chunk on the
        // adjoints the scans just left in L.  Optional path (the reference training loop never asks for it, training_helpers.py:34).
        float* Wsum = scratch + (size_t)p->nchunks * 2 * BB_SCR;
        SN_LAUNCH("sss_tc_wsum_kernel", st, sss_tc_wsum_kernel<<<p->nchunks, 256, 0, st>>>(coef, Wsum));
        std::vector<sn_sss_tc_chunk> hc(p->nchunks);
        SN_CHECK_CUDA(cudaMemcpyAsync(hc.data(), p->chunks, sizeof(sn_sss_tc_chunk) * p->nchunks, cudaMemcpyDeviceToHost, st));
        SN_CHECK_CUDA(cudaStreamSynchronize(st));      // the chunk table lives on the device; this optional path reads it back
        for (int j = 0; j < p->nchunks; ++j) {
            const float* Wj = Wsum + (size_t)j * 64 * WCOLS;
            float* gxj = grad_x + hc[j].col0;
            const int kout = hc[j].nrows;
            if (int rc = snb::gemm_f32(false, false, (int)B, hc[j].ncols, kout, 1.f, grad_y + hc[j].row0, ldgy, Wj, WCOLS, 0.f, gxj, ldgx, nullptr, st)) return rc;
            if (int rc = snb::gemm_f32(false, false, (int)B, hc[j].ncols, 32, 1.f, L + (size_t)j * B * 32, 32, Wj + (size_t)PO * WCOLS, WCOLS, 1.f, gxj, ldgx, nullptr, st, true)) return rc;
        }
    }
    if (grad_params == nullptr) {   // input gradient only (frozen parameters): no gradient GEMM, no build backward
        if (bias_later)
            if (int rc = snb::colsum_accumulate(grad_y, ldgy, B, p->output_dim, grad_bias, st)) return rc;
        return 0;
    }
    SN_CHECK_CUDA(cudaMemsetAsync(dM, 0, (size_t)p->nchunks * 64 * DMC * sizeof(float), st));
    CUtensorMap mx, mg, ml, ms;
    if (int rc = make_map_f32(&mx, x, (uint64_t)p->input_dim, (uint64_t)B, (uint64_t)ldx, G2_KS, 0, 0, true, 32, true)) return rc;
    if (int rc = make_map_f32(&mg, grad_y, (uint64_t)p->output_dim, (uint64_t)B, (uint64_t)ldgy, G2_KS, 0, 0, true)) return rc;
    if (int rc = make_map_f32(&ml, L, 32, (uint64_t)B, 32, G2_KS, (uint64_t)p->nchunks, (uint64_t)B * 32, true)) return rc;
    if (int rc = make_map_f32(&ms, states, 32, (uint64_t)B, 32, G2_KS, (uint64_t)p->nchunks, (uint64_t)B * 32, true)) return rc;
    const int ntk = (int)((B + G2_KS - 1) / G2_KS);
    // persistent CTAs over items = (sample range of `per` 32-sample steps, chunk).  per <= 32: at most 1024 samples per TMEM accumulator
    // (accuracy, see the kernel); among those the item size that wastes the least in the last round of items, with two steps' worth of
    // per-item cost (accumulator switch, 48 KB of red.add) charged per item.  SNB200_SSS_G2_PER forces it (measurements).
    int per = 0;
    {
        long best = -1;
        for (int cand = 32; cand >= 1; --cand) {
            const int nr = ceil_div(ntk, cand), pe = ceil_div(ntk, nr);
            const long rounds = ((long)nr * p->nchunks + sm_count() - 1) / sm_count();
            const long cost = rounds * (pe + 2);
            if (best < 0 || cost < best) { best = cost; per = pe; }
        }
        const char* e = getenv("SNB200_SSS_G2_PER");
        if (e != nullptr && atoi(e) >= 1 && atoi(e) <= 32) per = atoi(e);
    }
    const int nranges = ceil_div(ntk, per);
    const long nitems = (long)nranges * p->nchunks;
    const int g2grid = (int)(nitems < sm_count() ? nitems : sm_count());
    const size_t g2smem = G2_SMEM + (size_t)p->nchunks * sizeof(int4);
    SN_CHECK_ARG(g2smem <= 227 * 1024, "sss_tc_backward: too many chunks for the gradient GEMM's chunk table");
    SN_SET_MAX_SMEM((int)g2smem, sss_tc_grad_gemm_kernel);
    SN_LAUNCH("sss_tc_grad_gemm_kernel", st, sss_tc_grad_gemm_kernel<<<g2grid, G2_THREADS, g2smem, st>>>(mx, mg, ml, ms, p->chunks, p->nchunks, nranges, per, (long)B, dM));
    // small-batch path: the bias gradient (column sums of grad_y) runs on a second stream beside the build-backward kernel, which is
    // one latency-bound CTA per (chunk, direction, half) and leaves most of every SM idle.  (Beside the adjoint scans it slowed them
    // down by more than its own duration.)
    if (bias_later) {
        bias_side = snb::side_stream();
        cudaStream_t s2 = st;
        if (bias_side != nullptr) {
            SN_CHECK_CUDA(cudaEventRecord(bias_side->fork, st));
            SN_CHECK_CUDA(cudaStreamWaitEvent(bias_side->stream, bias_side->fork, 0));
            s2 = bias_side->stream;
        }
        if (int rc = snb::colsum_accumulate(grad_y, ldgy, B, p->output_dim, grad_bias, s2)) return rc;
        if (bias_side != nullptr) SN_CHECK_CUDA(cudaEventRecord(bias_side->join, bias_side->stream));
    }
    auto join_bias = [&]() -> int {
        if (bias_side != nullptr) SN_CHECK_CUDA(cudaStreamWaitEvent(st, bias_side->join, 0));
        return 0;
    };
    const size_t bsmm = ((size_t)BWM_FIXED + p->chunk_param_floats + 32) * sizeof(float);
    if (build_mode() == 2 && bsmm <= 227 * 1024) {
        // needs the states the tensor-core build kernel of THIS forward left in coef (same build mode on both sides)
        SN_SET_MAX_SMEM((int)bsmm, sss_tc_build_bwdm_kernel);
        SN_LAUNCH("sss_tc_build_bwdm_kernel", st, sss_tc_build_bwdm_kernel<<<dim3(p->nchunks, 2, BM_SPLIT), BM_THREADS, bsmm, st>>>(p->stages, p->nb_states, p->chunks, params, dM, vg_of(p, coef), grad_params, p->reserved[0]));
        return join_bias();
    }
    const size_t bsm4 = ((size_t)BB4_FIXED + p->chunk_param_floats + B4_LPC * LMAX * 4) * sizeof(float);
    if (use_quad_build() && bsm4 <= 227 * 1024) {
        SN_SET_MAX_SMEM((int)bsm4, sss_tc_build_bwd4_kernel);
        SN_LAUNCH("sss_tc_build_bwd4_kernel", st, sss_tc_build_bwd4_kernel<<<dim3(p->nchunks, 2, B4_SPLIT), B4_THREADS, bsm4, st>>>(p->stages, p->nb_states, p->chunks, params, dM, grad_params));
        return join_bias();
    }
    const size_t bsm = ((size_t)64 * DMC + p->chunk_param_floats) * sizeof(float);
    SN_SET_MAX_SMEM((int)bsm, sss_tc_build_bwd_kernel);
    SN_LAUNCH("sss_tc_build_bwd_kernel", st, sss_tc_build_bwd_kernel<<<dim3(p->nchunks, 2), BUILD_THREADS, bsm, st>>>(p->stages, p->nb_states, p->chunks, params, dM, scratch, grad_params));
    SN_LAUNCH("sss_tc_build_red_kernel", st, sss_tc_build_red_kernel<<<dim3(p->nchunks * LMAX, 2), BR_THREADS, 0, st>>>(p->stages, p->nb_states, p->chunks, scratch, grad_params));
    return join_bias();
}

}  // extern "C"
