// Product-of-sparse-matrices layer:  y = S_0 (S_1 ( ... (S_{n-1} x))) + b.
// Replaces PSMLayer.forward / forward_sparse (reference layers/psm_layer.py:36-60) -- with the factor
// order the reference *intends* (W = S_0 S_1 ... S_{n-1}, approximators/psm_approximator.py:96-105); the
// literal loop order of psm_layer.py:52-54 is only correct for <= 2 factors (SURVEY.md finding F2), where
// both coincide -- and the autograd backward (sparse gradients on the COO pattern).
//
// The chain is applied per tile of 4 samples with every intermediate activation kept in shared memory,
// feature-major [feature][4] (one LDS.128 gathers a feature for the whole tile): only x and y touch HBM.
// The static sparsity pattern is pre-arranged (once, host side) in sliced-ELL form, for S and for S^T:
// rows sorted by length, slices of 32 rows, entry j of the slice's rows stored contiguously -- so a warp
// (lane = row) streams its column indices (uint16) and values with fully coalesced loads, 6 bytes per
// non-zero, instead of chasing three dependent scattered loads per non-zero.  The values are gathered
// from the parameter's own COO array into that order once per call (psm_pack_vals_kernel); the backward
// accumulates dS in the same packed order with coalesced reductions and scatters it back once.
#include "common.cuh"
#include "bf16_ops.cuh"
#include "util.cuh"
#include "gemm_f32.cuh"

namespace {

constexpr int PSM_MAX_FACTORS = 8;
constexpr int PSM_THREADS = 512;
constexpr int PSM_WARPS = PSM_THREADS / 32;
constexpr int NS = 4;   // samples per tile

struct Ell {
    int nrows, nslices, total, pad;
    const int* rowmap;            // [nslices * 32] natural row of position p, -1 = none
    const int* slice_off;         // [nslices + 1]
    const unsigned short* col;    // [total]
    const float* val;             // [total] packed values (this call's)
};

struct Factor {
    int rows, cols;
    Ell fwd, tr;
    float* gpacked;   // [fwd.total], backward only
};

struct Chain {
    int nf, in_dim, out_dim, maxdim;
    Factor f[PSM_MAX_FACTORS];
};

__global__ void psm_pack_vals_kernel(const int* __restrict__ src, const float* __restrict__ vals, float* __restrict__ out, int total) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total) {
        const int s = __ldg(src + i);
        out[i] = s >= 0 ? __ldg(vals + s) : 0.f;
    }
}
__global__ void psm_unpack_grad_kernel(const int* __restrict__ src, const float* __restrict__ gpacked, float* __restrict__ gvals, int total) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total) {
        const int s = __ldg(src + i);
        if (s >= 0) gvals[s] += gpacked[i];   // every COO entry appears exactly once
    }
}

// dst[f][s] = src[t0 + s][f]
__device__ __forceinline__ void load_tile(const float* __restrict__ x, long ldx, long t0, long B, int dim, float* dst) {
    for (int f = threadIdx.x; f < dim; f += PSM_THREADS) {
        float4 v;
        v.x = t0 + 0 < B ? __ldg(x + (size_t)(t0 + 0) * ldx + f) : 0.f;
        v.y = t0 + 1 < B ? __ldg(x + (size_t)(t0 + 1) * ldx + f) : 0.f;
        v.z = t0 + 2 < B ? __ldg(x + (size_t)(t0 + 2) * ldx + f) : 0.f;
        v.w = t0 + 3 < B ? __ldg(x + (size_t)(t0 + 3) * ldx + f) : 0.f;
        reinterpret_cast<float4*>(dst)[f] = v;
    }
}

// out[r][:] = sum_j val_j * in[col_j][:]  for every row r of the ELL pattern (a warp per slice of 32 rows, lane = row)
__device__ __forceinline__ void spmm_ell(const Ell& E, const float* in, float* out) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float4* in4 = reinterpret_cast<const float4*>(in);
    for (int sl = warp; sl < E.nslices; sl += PSM_WARPS) {
        const int base = __ldg(E.slice_off + sl);
        const int len = (__ldg(E.slice_off + sl + 1) - base) >> 5;
        const int r = __ldg(E.rowmap + sl * 32 + lane);
        const unsigned short* cp = E.col + base + lane;
        const float* vp = E.val + base + lane;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int j = 0;
        for (; j + 4 <= len; j += 4) {
            const int c0 = __ldg(cp + (j + 0) * 32), c1 = __ldg(cp + (j + 1) * 32), c2 = __ldg(cp + (j + 2) * 32), c3 = __ldg(cp + (j + 3) * 32);
            const float v0 = __ldg(vp + (j + 0) * 32), v1 = __ldg(vp + (j + 1) * 32), v2 = __ldg(vp + (j + 2) * 32), v3 = __ldg(vp + (j + 3) * 32);
            const float4 x0 = in4[c0], x1 = in4[c1], x2 = in4[c2], x3 = in4[c3];
            acc.x = fmaf(v0, x0.x, acc.x); acc.y = fmaf(v0, x0.y, acc.y); acc.z = fmaf(v0, x0.z, acc.z); acc.w = fmaf(v0, x0.w, acc.w);
            acc.x = fmaf(v1, x1.x, acc.x); acc.y = fmaf(v1, x1.y, acc.y); acc.z = fmaf(v1, x1.z, acc.z); acc.w = fmaf(v1, x1.w, acc.w);
            acc.x = fmaf(v2, x2.x, acc.x); acc.y = fmaf(v2, x2.y, acc.y); acc.z = fmaf(v2, x2.z, acc.z); acc.w = fmaf(v2, x2.w, acc.w);
            acc.x = fmaf(v3, x3.x, acc.x); acc.y = fmaf(v3, x3.y, acc.y); acc.z = fmaf(v3, x3.z, acc.z); acc.w = fmaf(v3, x3.w, acc.w);
        }
        for (; j < len; ++j) {
            const int c0 = __ldg(cp + j * 32);
            const float v0 = __ldg(vp + j * 32);
            const float4 x0 = in4[c0];
            acc.x = fmaf(v0, x0.x, acc.x); acc.y = fmaf(v0, x0.y, acc.y); acc.z = fmaf(v0, x0.z, acc.z); acc.w = fmaf(v0, x0.w, acc.w);
        }
        if (r >= 0) reinterpret_cast<float4*>(out)[r] = acc;
    }
}

// gpacked[entry] += sum_s g[row][s] * in[col][s]   (coalesced reductions: the 32 lanes of a warp hit 32 consecutive floats)
__device__ __forceinline__ void dvals_ell(const Ell& E, const float* g, const float* in, float* __restrict__ gpacked) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float4* in4 = reinterpret_cast<const float4*>(in);
    for (int sl = warp; sl < E.nslices; sl += PSM_WARPS) {
        const int base = __ldg(E.slice_off + sl);
        const int len = (__ldg(E.slice_off + sl + 1) - base) >> 5;
        const int r = __ldg(E.rowmap + sl * 32 + lane);
        const float4 gr = r >= 0 ? reinterpret_cast<const float4*>(g)[r] : make_float4(0.f, 0.f, 0.f, 0.f);
        const unsigned short* cp = E.col + base + lane;
        float* gp = gpacked + base + lane;
#pragma unroll 4
        for (int j = 0; j < len; ++j) {
            const float4 xv = in4[__ldg(cp + j * 32)];
            const float d = fmaf(gr.w, xv.w, fmaf(gr.z, xv.z, fmaf(gr.y, xv.y, gr.x * xv.x)));
            asm volatile("red.global.add.f32 [%0], %1;" ::"l"(gp + j * 32), "f"(d) : "memory");
        }
    }
}

// dst[t0 + s][f] = src[f][s]   (each warp writes 32 consecutive floats of a sample row)
__device__ __forceinline__ void store_tile(float* __restrict__ dst, long ld, long t0, long B, int dim, const float* src) {
    for (int f = threadIdx.x; f < dim; f += PSM_THREADS) {
        const float4 v = reinterpret_cast<const float4*>(src)[f];
        if (t0 + 0 < B) dst[(size_t)(t0 + 0) * ld + f] = v.x;
        if (t0 + 1 < B) dst[(size_t)(t0 + 1) * ld + f] = v.y;
        if (t0 + 2 < B) dst[(size_t)(t0 + 2) * ld + f] = v.z;
        if (t0 + 3 < B) dst[(size_t)(t0 + 3) * ld + f] = v.w;
    }
}

// acts (nullable): the input of every factor but the last, [B][cols_k] row-major, factor 0 first -- kept for the backward, which then
// needs no recomputation (two 16 KB rows per sample and factor through HBM against a whole sparse pass over the pattern)
__global__ void __launch_bounds__(PSM_THREADS)
psm_fwd_kernel(Chain ch, const float* __restrict__ x, long ldx, float* __restrict__ y, long ldy, const float* __restrict__ bias, long B,
               float* __restrict__ acts) {
    extern __shared__ __align__(16) float smem[];
    float* a = smem;
    float* b = smem + (size_t)ch.maxdim * NS;
    const long t0 = (long)blockIdx.x * NS;
    load_tile(x, ldx, t0, B, ch.in_dim, a);
    __syncthreads();
    for (int k = ch.nf - 1; k >= 0; --k) {
        spmm_ell(ch.f[k].fwd, a, b);
        __syncthreads();
        if (acts != nullptr && k > 0) {       // b = output of factor k = input of factor k - 1
            size_t off = 0;
            for (int j = 0; j < k - 1; ++j) off += (size_t)B * ch.f[j].cols;
            store_tile(acts + off, ch.f[k - 1].cols, t0, B, ch.f[k - 1].cols, b);
        }
        float* t = a; a = b; b = t;
    }
    for (int s = 0; s < NS; ++s) {
        if (t0 + s >= B) break;
        float* row = y + (size_t)(t0 + s) * ldy;
        for (int o = threadIdx.x; o < ch.out_dim; o += PSM_THREADS) row[o] = a[(size_t)o * NS + s] + (bias ? __ldg(bias + o) : 0.f);
    }
}

// Backward with the activations the forward kept: two buffers.  G holds the gradient entering factor k from the output side, P the
// input of factor k; after dS_k the product S_k^T G overwrites P and becomes the next G.  gx (nullable): after the last factor's dS,
// one more S_{n-1}^T G gives the tile's grad_x = gy S_0 .. S_{n-1}; each CTA writes only its own samples.  GX = (gx != nullptr): the
// instantiation without grad_x is the kernel as it was before grad_x existed.
template <bool GX>
__global__ void __launch_bounds__(PSM_THREADS)
psm_bwd_acts_kernel(Chain ch, const float* __restrict__ x, long ldx, const float* __restrict__ gy, long ldgy, long B, const float* __restrict__ acts,
                    float* __restrict__ gx, long ldgx) {
    extern __shared__ __align__(16) float smem[];
    const size_t vec = (size_t)ch.maxdim * NS;
    float* G = smem;
    float* P = smem + vec;
    const long t0 = (long)blockIdx.x * NS;
    load_tile(gy, ldgy, t0, B, ch.out_dim, G);
    size_t off = 0;
    for (int k = 0; k < ch.nf; ++k) {
        if (k == ch.nf - 1) load_tile(x, ldx, t0, B, ch.in_dim, P);
        else load_tile(acts + off, ch.f[k].cols, t0, B, ch.f[k].cols, P);
        off += (size_t)B * ch.f[k].cols;
        __syncthreads();
        dvals_ell(ch.f[k].fwd, G, P, ch.f[k].gpacked);
        if (k + 1 < ch.nf || GX) {
            __syncthreads();                      // every warp is done reading P
            spmm_ell(ch.f[k].tr, G, P);           // S_k^T G
            __syncthreads();
            float* t = G; G = P; P = t;
        }
    }
    if (GX) store_tile(gx, ldgx, t0, B, ch.in_dim, G);
}

// Three buffers: P / Q recompute the input of factor k from x (ping-pong), G holds the gradient that enters factor k from the
// output side; S_k^T G lands in whichever of P / Q is free and becomes the next G.  gx (nullable): as in psm_bwd_acts_kernel.
// PSMLayer reaches GX = true only with one factor (with more, its forward keeps the activations whenever a factor takes a gradient);
// sn_psm_backward callers that pass no acts reach it with any number of factors.
template <bool GX>
__global__ void __launch_bounds__(PSM_THREADS)
psm_bwd_kernel(Chain ch, const float* __restrict__ x, long ldx, const float* __restrict__ gy, long ldgy, long B, float* __restrict__ gx, long ldgx) {
    extern __shared__ __align__(16) float smem[];
    const size_t vec = (size_t)ch.maxdim * NS;
    float* P = smem;
    float* Q = smem + vec;
    float* G = smem + 2 * vec;
    const long t0 = (long)blockIdx.x * NS;
    load_tile(gy, ldgy, t0, B, ch.out_dim, G);
    for (int k = 0; k < ch.nf; ++k) {
        // input of factor k: x pushed through factors nf-1 .. k+1
        load_tile(x, ldx, t0, B, ch.in_dim, P);
        __syncthreads();
        for (int kk = ch.nf - 1; kk > k; --kk) {
            spmm_ell(ch.f[kk].fwd, P, Q);
            __syncthreads();
            float* t = P; P = Q; Q = t;
        }
        dvals_ell(ch.f[k].fwd, G, P, ch.f[k].gpacked);
        if (k + 1 < ch.nf || GX) {
            spmm_ell(ch.f[k].tr, G, Q);   // S_k^T G (Q is free: the recomputed input sits in P)
            __syncthreads();
            float* t = G; G = Q; Q = t;
        }
    }
    if (GX) store_tile(gx, ldgx, t0, B, ch.in_dim, G);
}

// Raises psm_fwd_kernel's dynamic shared-memory limit.  The forward and the input-gradient-only backward both launch that kernel, and
// SN_SET_MAX_SMEM remembers per call site what it set: a second site could lower the limit below what the first one believes it set.
int fwd_kernel_smem(size_t smem) {
    SN_SET_MAX_SMEM((int)smem, psm_fwd_kernel);
    return 0;
}

// backward: the transposed patterns are needed, and the factor gradient buffers (grad_vals, grad_packed) are all set or all NULL;
// *param_grad (backward only) tells which
int make_chain(const sn_psm_factor* f, int nf, int in_dim, int out_dim, bool backward, Chain* ch, bool* param_grad = nullptr) {
    SN_CHECK_ARG(f != nullptr && nf >= 1 && nf <= PSM_MAX_FACTORS, "psm: need 1..%d factors", PSM_MAX_FACTORS);
    ch->nf = nf; ch->in_dim = in_dim; ch->out_dim = out_dim; ch->maxdim = in_dim > out_dim ? in_dim : out_dim;
    bool any_grad = false;
    for (int k = 0; k < nf; ++k) any_grad |= f[k].grad_vals != nullptr || f[k].grad_packed != nullptr;
    if (param_grad != nullptr) *param_grad = any_grad;
    for (int k = 0; k < nf; ++k) {
        const sn_psm_factor& s = f[k];
        SN_CHECK_ARG(s.rows > 0 && s.cols > 0 && s.rows <= 65535 && s.cols <= 65535, "psm: factor %d is %d x %d (dimensions must be in 1..65535)", k, s.rows, s.cols);
        SN_CHECK_ARG(s.fwd.rowmap && s.fwd.slice_off && s.fwd.nslices * 32 >= s.rows && (s.fwd.total == 0 || (s.fwd.col && s.fwd.src && s.val_fwd)),
                     "psm: factor %d has an incomplete sliced-ELL pattern", k);
        SN_CHECK_ARG(s.nnz == 0 || s.vals, "psm: factor %d has no value array", k);
        Factor& F = ch->f[k];
        F.rows = s.rows; F.cols = s.cols;
        F.fwd = Ell{s.rows, s.fwd.nslices, s.fwd.total, 0, s.fwd.rowmap, s.fwd.slice_off, s.fwd.col, s.val_fwd};
        F.tr = Ell{s.cols, s.tr.nslices, s.tr.total, 0, s.tr.rowmap, s.tr.slice_off, s.tr.col, s.val_tr};
        F.gpacked = s.grad_packed;
        if (backward) {
            SN_CHECK_ARG(s.tr.rowmap && s.tr.slice_off && (s.tr.total == 0 || (s.tr.col && s.tr.src && s.val_tr)), "psm: factor %d has no transposed pattern", k);
            SN_CHECK_ARG(!any_grad || s.fwd.total == 0 || (s.grad_packed && s.grad_vals),
                         "psm_backward: factor %d has no gradient buffer (the factor gradient buffers are all set or all NULL)", k);
        }
        if (s.rows > ch->maxdim) ch->maxdim = s.rows;
        if (s.cols > ch->maxdim) ch->maxdim = s.cols;
        if (k > 0) SN_CHECK_ARG(f[k - 1].cols == s.rows, "psm: factor %d cols (%d) != factor %d rows (%d)", k - 1, f[k - 1].cols, k, s.rows);
    }
    SN_CHECK_ARG(f[0].rows == out_dim && f[nf - 1].cols == in_dim, "psm: chain maps %d -> %d, layer is %d -> %d", f[nf - 1].cols, f[0].rows, in_dim, out_dim);
    return 0;
}

int pack_vals(const sn_psm_ell& e, const float* vals, float* out, cudaStream_t st) {
    if (e.total <= 0) return 0;
    SN_LAUNCH("psm_pack_vals_kernel", st, psm_pack_vals_kernel<<<snb::ceil_div(e.total, 256), 256, 0, st>>>(e.src, vals, out, e.total));
    return 0;
}


// ------------------------------------------------------------------------------------------
// Dense-product path (large batches).  The product of the factors is batch independent, so for B >> dims the step is cheapest as
//   W^T = (S_0 S_1 ... S_{n-1})^T built once per call by sparse-times-dense row combinations (all matrices kept TRANSPOSED,
//   [dim][out_dim], so every row operation is a coalesced stream of out_dim floats),
//   y = x W^T^T + b and G^T = x^T grad_y on the tensor cores (3xTF32, csrc/gemm_tf32x3.cuh),
//   dS_k[m][j] = < L_k^T[m][:], H_k^T[j][:] > on the pattern, with the prefix products L_k = S_0 .. S_{k-1} kept from the forward and the
//   suffix recursion H_{k-1}^T = S_k H_k^T, H_{n-1}^T = G^T.
// This is also what the reference's default forward does (dense GEMMs on the densified factors, layers/psm_layer.py:47-60).
// ------------------------------------------------------------------------------------------
// Out[r][:] = sum over the entries e of row r of the sparse matrix: vals[src[e]] * In[idx[e]][:]   (In == nullptr: identity rows)
__global__ void __launch_bounds__(256)
psm_rowcomb_kernel(const int* __restrict__ ptr, const int* __restrict__ idx, const int* __restrict__ src, const float* __restrict__ vals,
                   const float* __restrict__ In, float* __restrict__ Out, int width) {
    const int r = blockIdx.x;
    const int e0 = ptr[r], e1 = ptr[r + 1];
    float* out = Out + (size_t)r * width;
    if (In == nullptr) {   // the first factor: row r of S_0^T scattered into a zero row
        for (int c = threadIdx.x; c < width; c += blockDim.x) out[c] = 0.f;
        __syncthreads();
        for (int e = e0 + threadIdx.x; e < e1; e += blockDim.x) atomicAdd(out + idx[e], vals[src[e]]);
        return;
    }
    const int w4 = width >> 2;
    for (int c = threadIdx.x; c < w4; c += blockDim.x) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int e = e0; e < e1; ++e) {
            const float v = __ldg(vals + __ldg(src + e));
            const float4 x = __ldg(reinterpret_cast<const float4*>(In + (size_t)__ldg(idx + e) * width) + c);
            acc.x = fmaf(v, x.x, acc.x); acc.y = fmaf(v, x.y, acc.y); acc.z = fmaf(v, x.z, acc.z); acc.w = fmaf(v, x.w, acc.w);
        }
        reinterpret_cast<float4*>(out)[c] = acc;
    }
}
// one warp per non-zero e = (m, j): g[e] += < Lt[m][:], Ht[j][:] >;  Lt == nullptr (first factor, L_0 = I): g[e] += Ht[j][m]
__global__ void __launch_bounds__(256)
psm_masked_dot_kernel(const int* __restrict__ row, const int* __restrict__ col, int nnz, const float* __restrict__ Lt, const float* __restrict__ Ht,
                      float* __restrict__ g, int width) {
    if (Lt == nullptr) {       // first factor (L_0 = I): one THREAD per non-zero
        const int e = blockIdx.x * blockDim.x + threadIdx.x;
        if (e < nnz) g[e] += __ldg(Ht + (size_t)col[e] * width + row[e]);
        return;
    }
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= nnz) return;
    const int m = row[warp], j = col[warp];
    const float4* a = reinterpret_cast<const float4*>(Lt + (size_t)m * width);
    const float4* b = reinterpret_cast<const float4*>(Ht + (size_t)j * width);
    float acc = 0.f;
    for (int c = lane; c < (width >> 2); c += 32) {
        const float4 x = __ldg(a + c), y = __ldg(b + c);
        acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc); acc = fmaf(x.z, y.z, acc); acc = fmaf(x.w, y.w, acc);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) g[warp] += acc;
}

// Backward of factor k >= 1 in one pass over its rows (CSR): CTA = row m of S_k, warp = some of the row's non-zeros (m, j).  Every H_k^T[j]
// row is read ONCE and used twice: for the gradient of the non-zero, g[e] += < L_k^T[m], H_k^T[j] >, and for the next adjoint,
// H_{k-1}^T[m] = sum_j S_k[m][j] H_k^T[j].  (psm_masked_dot_kernel + psm_rowcomb_kernel read it twice: 126 + 40 us per factor at C3.)
// width <= 1024 floats (a lane holds 8 float4 of a row).
constexpr int PBR_WARPS = 8;
constexpr int PBR_NI = 8;
template <bool DOT>        // DOT = false: only the row combination Hn[m] = sum_j S[m][j] Ht[j] (the forward's prefix products)
__global__ void __launch_bounds__(PBR_WARPS * 32)
psm_bwd_row_kernel(const int* __restrict__ ptr, const int* __restrict__ idx, const int* __restrict__ src, const float* __restrict__ vals,
                   const float* __restrict__ Lt, const float* __restrict__ Ht, float* __restrict__ g, float* __restrict__ Hn, int width) {
    __shared__ float4 part[PBR_WARPS][PBR_NI * 32];
    const int r = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e0 = ptr[r], e1 = ptr[r + 1];
    const int w4 = width >> 2;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 lt[PBR_NI], acc[PBR_NI];
#pragma unroll
    for (int i = 0; i < PBR_NI; ++i) {
        const int c = lane + 32 * i;
        lt[i] = (DOT && c < w4) ? __ldg(reinterpret_cast<const float4*>(Lt + (size_t)r * width) + c) : z;
        acc[i] = z;
    }
    // the row of the warp's NEXT non-zero is requested before the current one is used (two rows in flight per warp)
    float4 xn[PBR_NI];
    int se_n = 0;
    float v_n = 0.f;
    auto fetch = [&](int e) {
        if (e < e1) {
            se_n = __ldg(src + e);
            v_n = __ldg(vals + se_n);
            const float4* hrow = reinterpret_cast<const float4*>(Ht + (size_t)__ldg(idx + e) * width);
#pragma unroll
            for (int i = 0; i < PBR_NI; ++i) {
                const int c = lane + 32 * i;
                xn[i] = (c < w4) ? __ldg(hrow + c) : z;
            }
        }
    };
    fetch(e0 + warp);
    for (int e = e0 + warp; e < e1; e += PBR_WARPS) {
        const int se = se_n;
        const float v = v_n;
        float4 x[PBR_NI];
#pragma unroll
        for (int i = 0; i < PBR_NI; ++i) x[i] = xn[i];
        fetch(e + PBR_WARPS);
        float dot = 0.f;
#pragma unroll
        for (int i = 0; i < PBR_NI; ++i) {
            acc[i].x = fmaf(v, x[i].x, acc[i].x); acc[i].y = fmaf(v, x[i].y, acc[i].y); acc[i].z = fmaf(v, x[i].z, acc[i].z); acc[i].w = fmaf(v, x[i].w, acc[i].w);
            if (DOT) { dot = fmaf(lt[i].x, x[i].x, dot); dot = fmaf(lt[i].y, x[i].y, dot); dot = fmaf(lt[i].z, x[i].z, dot); dot = fmaf(lt[i].w, x[i].w, dot); }
        }
        if (DOT) {
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, off);
            if (lane == 0 && g != nullptr) g[se] += dot;
        }
    }
#pragma unroll
    for (int i = 0; i < PBR_NI; ++i) part[warp][lane + 32 * i] = acc[i];
    __syncthreads();
    for (int c = threadIdx.x; c < w4; c += PBR_WARPS * 32) {
        float4 s4 = part[0][c];
#pragma unroll
        for (int w = 1; w < PBR_WARPS; ++w) {
            const float4 p4 = part[w][c];
            s4.x += p4.x; s4.y += p4.y; s4.z += p4.z; s4.w += p4.w;
        }
        reinterpret_cast<float4*>(Hn + (size_t)r * width)[c] = s4;
    }
}

int check_dense_chain(const sn_psm_dense_factor* f, int nf, int in_dim, int out_dim) {
    SN_CHECK_ARG(f != nullptr && nf >= 1 && nf <= PSM_MAX_FACTORS, "psm_dense: need 1..%d factors", PSM_MAX_FACTORS);
    SN_CHECK_ARG(out_dim % 4 == 0, "psm_dense: output_dim must be a multiple of 4");
    SN_CHECK_ARG(f[0].rows == out_dim && f[nf - 1].cols == in_dim, "psm_dense: the factors do not map input_dim -> output_dim");
    for (int k = 0; k + 1 < nf; ++k) SN_CHECK_ARG(f[k].cols == f[k + 1].rows, "psm_dense: factors %d and %d cannot be multiplied", k, k + 1);
    return 0;
}

// prefix: L_1^T | L_2^T | ... | L_n^T = W^T ([cols_{k-1}][out_dim] each); returns W^T (the last block) in *wt
int build_prefix(const sn_psm_dense_factor* f, int nf, float* prefix, int out_dim, const float** wt, cudaStream_t st) {
    float* cur = prefix;
    const float* prev = nullptr;
    for (int k = 0; k < nf; ++k) {
        // L_{k+1}^T = S_k^T L_k^T: the rows of S_k^T are the columns of S_k (csc)
        // (the pipelined row kernel of the backward, without its dot products, is slower here: 45 vs 35 us per factor at C3)
        SN_LAUNCH("psm_rowcomb_kernel", st, psm_rowcomb_kernel<<<f[k].cols, 256, 0, st>>>(f[k].csc_ptr, f[k].csc_idx, f[k].csc_src, f[k].vals, prev, cur, out_dim));
        prev = cur;
        cur += (size_t)f[k].cols * out_dim;
    }
    *wt = prev;
    return 0;
}

// Projection of the dense gradient onto every factor's pattern.  work starts with H_{n-1}^T = G^T = x^T grad_y [in_dim][out_dim];
// the suffix recursion writes H_{n-2}^T [rows_{n-1}][out_dim], ... behind it.
int project_dense_grad(const sn_psm_dense_factor* f, int nf, const float* prefix, float* work, int out_dim, cudaStream_t st) {
    float* Ht = work;
    // prefix offsets: L_k^T for k >= 1 starts after the first k - 1 blocks
    size_t off[PSM_MAX_FACTORS + 1];
    off[0] = 0;
    for (int k = 0; k < nf; ++k) off[k + 1] = off[k] + (size_t)f[k].cols * out_dim;
    for (int k = nf - 1; k >= 0; --k) {
        const float* Lt = k == 0 ? nullptr : prefix + off[k - 1];
        if (k > 0 && out_dim <= 4 * 32 * PBR_NI) {
            // gradient of the factor's non-zeros and the next adjoint H_{k-1}^T = S_k H_k^T [rows_k][out_dim] in one pass over H_k^T
            float* Hn = Ht + (size_t)f[k].cols * out_dim;
            SN_LAUNCH("psm_bwd_row_kernel", st, psm_bwd_row_kernel<true><<<f[k].rows, PBR_WARPS * 32, 0, st>>>(f[k].csr_ptr, f[k].csr_idx, f[k].csr_src, f[k].vals, Lt, Ht,
                                                                                                       f[k].grad_vals, Hn, out_dim));
            Ht = Hn;
            continue;
        }
        if (f[k].nnz > 0 && f[k].grad_vals != nullptr)
            SN_LAUNCH("psm_masked_dot_kernel", st, psm_masked_dot_kernel<<<(unsigned)(((size_t)f[k].nnz * (Lt == nullptr ? 1 : 32) + 255) / 256), 256, 0, st>>>(
                f[k].coo_row, f[k].coo_col, f[k].nnz, Lt, Ht, f[k].grad_vals, out_dim));
        if (k > 0) {
            float* Hn = Ht + (size_t)f[k].cols * out_dim;   // H_{k-1}^T = S_k H_k^T: [rows_k][out_dim]
            SN_LAUNCH("psm_rowcomb_kernel", st, psm_rowcomb_kernel<<<f[k].rows, 256, 0, st>>>(f[k].csr_ptr, f[k].csr_idx, f[k].csr_src, f[k].vals, Ht, Hn, out_dim));
            Ht = Hn;
        }
    }
    return 0;
}

}  // namespace

extern "C" {

size_t sn_psm_acts_floats(const sn_psm_factor* f, int nf, int64_t B) {
    size_t n = 0;
    for (int k = 0; f != nullptr && k + 1 < nf; ++k) n += (size_t)B * f[k].cols;
    return n;
}

int sn_psm_forward(const sn_psm_factor* factors_host, int nf, const float* x, int64_t ldx, float* y, int64_t ldy, const float* bias,
                   float* acts, int64_t B, int in_dim, int out_dim, sn_stream_t stream) {
    Chain ch;
    if (int rc = make_chain(factors_host, nf, in_dim, out_dim, false, &ch)) return rc;
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && y, "psm_forward: NULL buffer");
    cudaStream_t st = snb::as_stream(stream);
    for (int k = 0; k < nf; ++k)
        if (int rc = pack_vals(factors_host[k].fwd, factors_host[k].vals, factors_host[k].val_fwd, st)) return rc;
    const size_t smem = (size_t)2 * ch.maxdim * NS * sizeof(float);
    SN_CHECK_ARG(smem <= 227 * 1024, "psm_forward: factor dimension %d does not fit in shared memory", ch.maxdim);
    if (int rc = fwd_kernel_smem(smem)) return rc;
    SN_LAUNCH("psm_fwd_kernel", st, psm_fwd_kernel<<<(unsigned)((B + NS - 1) / NS), PSM_THREADS, smem, st>>>(ch, x, ldx, y, ldy, bias, B, acts));
    return 0;
}

int sn_psm_backward(const sn_psm_factor* factors_host, int nf, const float* x, int64_t ldx, const float* grad_y, int64_t ldgy,
                    const float* acts, float* grad_bias, float* grad_x, int64_t ldgx, int64_t B, int in_dim, int out_dim, sn_stream_t stream) {
    Chain ch;
    bool param_grad = false;
    if (int rc = make_chain(factors_host, nf, in_dim, out_dim, true, &ch, &param_grad)) return rc;
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && grad_y, "psm_backward: NULL buffer");
    SN_CHECK_ARG(param_grad || grad_x, "psm_backward: the factor gradient buffers and grad_x are both NULL");
    SN_CHECK_ARG(grad_x == nullptr || ldgx >= in_dim, "psm_backward: grad_x leading dimension too small (ldgx %lld < input_dim %d)",
                 (long long)ldgx, in_dim);
    cudaStream_t st = snb::as_stream(stream);
    if (grad_bias)
        if (int rc = snb::colsum_accumulate(grad_y, ldgy, B, out_dim, grad_bias, st)) return rc;
    if (!param_grad) {
        // grad_x only: the forward chain of the transposed factors in reverse order, S_{n-1}^T .. S_0^T applied to grad_y
        Chain ct = ch;
        ct.in_dim = out_dim;
        ct.out_dim = in_dim;
        for (int j = 0; j < nf; ++j) {
            const Factor& F = ch.f[nf - 1 - j];
            ct.f[j] = Factor{F.cols, F.rows, F.tr, F.fwd, nullptr};
            if (int rc = pack_vals(factors_host[nf - 1 - j].tr, factors_host[nf - 1 - j].vals, factors_host[nf - 1 - j].val_tr, st)) return rc;
        }
        const size_t smem = (size_t)2 * ct.maxdim * NS * sizeof(float);
        SN_CHECK_ARG(smem <= 227 * 1024, "psm_backward: factor dimension %d does not fit in shared memory", ct.maxdim);
        if (int rc = fwd_kernel_smem(smem)) return rc;
        SN_LAUNCH("psm_fwd_kernel", st, psm_fwd_kernel<<<(unsigned)((B + NS - 1) / NS), PSM_THREADS, smem, st>>>(ct, grad_y, ldgy, grad_x, ldgx, nullptr, B,
                                                                                                            nullptr));
        return 0;
    }
    for (int k = 0; k < nf; ++k) {
        const sn_psm_factor& f = factors_host[k];
        if (int rc = pack_vals(f.fwd, f.vals, f.val_fwd, st)) return rc;
        if (int rc = pack_vals(f.tr, f.vals, f.val_tr, st)) return rc;
        if (f.fwd.total > 0) SN_CHECK_CUDA(cudaMemsetAsync(f.grad_packed, 0, (size_t)f.fwd.total * sizeof(float), st));
    }
    if (acts != nullptr) {
        const size_t smem = (size_t)2 * ch.maxdim * NS * sizeof(float);
        SN_CHECK_ARG(smem <= 227 * 1024, "psm_backward: factor dimension %d does not fit in shared memory", ch.maxdim);
        const unsigned grid = (unsigned)((B + NS - 1) / NS);
        if (grad_x != nullptr) {
            SN_SET_MAX_SMEM((int)smem, psm_bwd_acts_kernel<true>);
            SN_LAUNCH("psm_bwd_acts_kernel<gx>", st, psm_bwd_acts_kernel<true><<<grid, PSM_THREADS, smem, st>>>(ch, x, ldx, grad_y, ldgy, B, acts, grad_x, ldgx));
        } else {
            SN_SET_MAX_SMEM((int)smem, psm_bwd_acts_kernel<false>);
            SN_LAUNCH("psm_bwd_acts_kernel", st, psm_bwd_acts_kernel<false><<<grid, PSM_THREADS, smem, st>>>(ch, x, ldx, grad_y, ldgy, B, acts, nullptr, 0));
        }
    } else {
        const size_t smem = (size_t)3 * ch.maxdim * NS * sizeof(float);
        SN_CHECK_ARG(smem <= 227 * 1024, "psm_backward: factor dimension %d does not fit in shared memory", ch.maxdim);
        const unsigned grid = (unsigned)((B + NS - 1) / NS);
        if (grad_x != nullptr) {
            SN_SET_MAX_SMEM((int)smem, psm_bwd_kernel<true>);
            SN_LAUNCH("psm_bwd_kernel<gx>", st, psm_bwd_kernel<true><<<grid, PSM_THREADS, smem, st>>>(ch, x, ldx, grad_y, ldgy, B, grad_x, ldgx));
        } else {
            SN_SET_MAX_SMEM((int)smem, psm_bwd_kernel<false>);
            SN_LAUNCH("psm_bwd_kernel", st, psm_bwd_kernel<false><<<grid, PSM_THREADS, smem, st>>>(ch, x, ldx, grad_y, ldgy, B, nullptr, 0));
        }
    }
    for (int k = 0; k < nf; ++k) {
        const sn_psm_factor& f = factors_host[k];
        if (f.fwd.total > 0)
            SN_LAUNCH("psm_unpack_grad_kernel", st, psm_unpack_grad_kernel<<<snb::ceil_div(f.fwd.total, 256), 256, 0, st>>>(f.fwd.src, f.grad_packed, f.grad_vals, f.fwd.total));
    }
    return 0;
}


size_t sn_psm_dense_prefix_floats(const sn_psm_dense_factor* f, int nf, int out_dim) {
    size_t n = 0;
    for (int k = 0; f != nullptr && k < nf; ++k) n += (size_t)f[k].cols * out_dim;
    return n;
}
size_t sn_psm_dense_backward_floats(const sn_psm_dense_factor* f, int nf, int out_dim) {
    size_t n = 0;
    for (int k = 0; f != nullptr && k < nf; ++k) n += (size_t)f[k].cols * out_dim;
    return n;
}
/* prefix: L_1^T | L_2^T | ... | L_n^T = W^T ([cols_{k-1}][out_dim] each), kept by the caller for the backward */
int sn_psm_dense_forward(const sn_psm_dense_factor* f, int nf, const float* x, int64_t ldx, float* y, int64_t ldy, const float* bias,
                         float* prefix, int64_t B, int in_dim, int out_dim, sn_stream_t stream) {
    if (int rc = check_dense_chain(f, nf, in_dim, out_dim)) return rc;
    SN_CHECK_ARG(prefix, "psm_dense_forward: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && y, "psm_dense_forward: NULL buffer");
    cudaStream_t st = snb::as_stream(stream);
    const float* wt = nullptr;
    if (int rc = build_prefix(f, nf, prefix, out_dim, &wt, st)) return rc;
    // y = x W^T^T + b: W^T is stored [in_dim][out_dim]
    return snb::gemm_f32(false, false, (int)B, out_dim, in_dim, 1.f, x, ldx, wt, out_dim, 0.f, y, ldy, bias, st);
}
/* grad_x = grad_y W from the multiplied-out product the forward left in `prefix` (W^T = its last block, [in_dim][out_dim]) */
int sn_psm_dense_input_grad(const sn_psm_dense_factor* f, int nf, const float* prefix, const float* grad_y, int64_t ldgy, float* grad_x,
                            int64_t ldgx, int64_t B, int in_dim, int out_dim, sn_stream_t stream) {
    if (int rc = check_dense_chain(f, nf, in_dim, out_dim)) return rc;
    SN_CHECK_ARG(prefix, "psm_dense_input_grad: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(grad_y && grad_x, "psm_dense_input_grad: NULL buffer");
    size_t off = 0;
    for (int k = 0; k + 1 < nf; ++k) off += (size_t)f[k].cols * out_dim;
    return snb::gemm_f32(false, true, (int)B, in_dim, out_dim, 1.f, grad_y, ldgy, prefix + off, out_dim, 0.f, grad_x, ldgx, nullptr, snb::as_stream(stream));
}
/* work: sn_psm_dense_backward_floats floats; grad_vals of every factor (COO order) and grad_bias are accumulated into */
int sn_psm_dense_backward(const sn_psm_dense_factor* f, int nf, const float* x, int64_t ldx, const float* grad_y, int64_t ldgy,
                          const float* prefix, float* work, float* grad_bias, int64_t B, int in_dim, int out_dim, sn_stream_t stream) {
    if (int rc = check_dense_chain(f, nf, in_dim, out_dim)) return rc;
    SN_CHECK_ARG(prefix && work, "psm_dense_backward: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && grad_y, "psm_dense_backward: NULL buffer");
    cudaStream_t st = snb::as_stream(stream);
    if (grad_bias)
        if (int rc = snb::colsum_accumulate(grad_y, ldgy, B, out_dim, grad_bias, st)) return rc;
    // work: H_{n-1}^T = G^T [in_dim][out_dim], then H_{n-2}^T [rows_{n-1}][out_dim], ...
    float* Ht = work;
    SN_CHECK_CUDA(cudaMemsetAsync(Ht, 0, (size_t)in_dim * out_dim * sizeof(float), st));
    if (int rc = snb::gemm_f32(true, false, in_dim, out_dim, (int)B, 1.f, x, ldx, grad_y, ldgy, 1.f, Ht, out_dim, nullptr, st, true)) return rc;
    return project_dense_grad(f, nf, prefix, Ht, out_dim, st);
}

/* bf16 features: the same prefix products and projection as above, the batch GEMMs on the bf16 tensor cores of csrc/dense_bf16.cu.
   wb: W bf16 [out_dim][ldwb], written; wtb: W^T bf16 [in_dim][ldwtb], written when not null (sn_dense_input_grad_bf16 reads it). */
int sn_psm_dense_forward_bf16(const sn_psm_dense_factor* f, int nf, const void* x, int64_t ldx, void* y, int64_t ldy, const float* bias,
                              float* prefix, void* wb, int64_t ldwb, void* wtb, int64_t ldwtb, int64_t B, int in_dim, int out_dim,
                              sn_stream_t stream) {
    if (int rc = check_dense_chain(f, nf, in_dim, out_dim)) return rc;
    SN_CHECK_ARG(prefix && wb, "psm_dense_forward_bf16: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && y, "psm_dense_forward_bf16: NULL buffer");
    const float* wt = nullptr;
    if (int rc = build_prefix(f, nf, prefix, out_dim, &wt, snb::as_stream(stream))) return rc;
    // the last prefix block is W^T [in_dim][out_dim]: its copy is W^T, its transpose W
    if (int rc = sn_dense_cast_bf16(wt, in_dim, out_dim, wtb, ldwtb, wb, ldwb, stream)) return rc;
    return sn_dense_apply_bf16(wb, ldwb, out_dim, in_dim, x, ldx, y, ldy, bias, B, stream);
}
int sn_psm_dense_backward_bf16(const sn_psm_dense_factor* f, int nf, const void* x, int64_t ldx, const void* grad_y, int64_t ldgy,
                               const float* prefix, float* work, float* grad_bias, int64_t B, int in_dim, int out_dim, sn_stream_t stream) {
    if (int rc = check_dense_chain(f, nf, in_dim, out_dim)) return rc;
    SN_CHECK_ARG(prefix && work, "psm_dense_backward_bf16: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && grad_y, "psm_dense_backward_bf16: NULL buffer");
    cudaStream_t st = snb::as_stream(stream);
    if (grad_bias)
        if (int rc = colsum_bf16((const __nv_bfloat16*)grad_y, ldgy, B, out_dim, grad_bias, st)) return rc;
    float* Ht = work;
    SN_CHECK_CUDA(cudaMemsetAsync(Ht, 0, (size_t)in_dim * out_dim * sizeof(float), st));
    // H_{n-1}^T = x^T grad_y [in_dim][out_dim]: the weight-gradient GEMM with the roles of the features and grad_y swapped
    if (int rc = sn_dense_weight_grad_bf16(grad_y, ldgy, x, ldx, Ht, out_dim, in_dim, out_dim, nullptr, B, stream)) return rc;
    return project_dense_grad(f, nf, prefix, Ht, out_dim, st);
}

}  // extern "C"
