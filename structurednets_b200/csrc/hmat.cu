// Hierarchical-matrix layer:  y = sum_c scatter_rows(c)[ L_c (R_c x[cols_c]) ] + b  over the leaves c.
// Replaces HMatLayer.forward (reference layers/hmat_layer.py:34-49) and its autograd backward.
//
// Every leaf is a low-rank pair (SURVEY.md F3): thousands of tiny two-stage products of very different
// sizes that all read the same sample's x and add into the same sample's y.  A CTA therefore owns a
// tile of NS samples, keeps x[in][NS] and y[out][NS] (feature-major) in shared memory for the whole
// leaf loop -- x and y touch HBM exactly once -- and its warps walk the leaf table round-robin:
//     stage 1  t[kk][s]  = sum_col R_c[kk][col] * x[c0+col][s]      (rank rows split over the lane halves)
//     stage 2  y[r0+r][s] += sum_kk L_c[r][kk] * t[kk][s]           (shared-memory reduction across leaves)
// The backward recomputes t, forms gt = L_c^T gy, and reduces dL_c = gy t^T, dR_c = gt x^T over the
// tile's samples before one atomic add per parameter and tile.
#include "common.cuh"
#include "util.cuh"

namespace {

struct Leaf {  // 8 x int32, mirrors the host table built by HMatLayer
    int r0, rows, c0, cols, k, offL, offR, reserved;
};

constexpr int HM_THREADS = 256;
constexpr int HM_WARPS = HM_THREADS / 32;
constexpr int HM_KCHUNK = 16;  // rank rows processed per pass (per-warp scratch: 2 x 16 x NS floats)

template <int NS>
__device__ __forceinline__ void load_tile(const float* __restrict__ src, long ld, long t0, long B, int feat, float* dst) {
    // dst[f][s] = src[(t0+s)][f]; coalesced along f
    for (int s = 0; s < NS; ++s) {
        const bool ok = t0 + s < B;
        const float* row = src + (size_t)(t0 + s) * ld;
        for (int f = threadIdx.x; f < feat; f += HM_THREADS) dst[f * NS + s] = ok ? __ldg(row + f) : 0.f;
    }
}

template <int NS>
__device__ __forceinline__ void stage1(const Leaf& lf, const float* __restrict__ R, int kc, int kn, const float* xs, float* tb,
                                       int s, int h) {
    constexpr int H = 32 / NS;
    for (int kk = h; kk < kn; kk += H) {
        const float* Rrow = R + (size_t)(kc + kk) * lf.cols;
        const float* xv = xs + (size_t)lf.c0 * NS + s;
        float acc = 0.f;
#pragma unroll 4
        for (int col = 0; col < lf.cols; ++col) acc = fmaf(__ldg(Rrow + col), xv[col * NS], acc);
        tb[kk * NS + s] = acc;
    }
}

// the transposed stage 1 (as in hmat_bwd_kernel): gt[kk][s] = sum_r L_c[r][kc+kk] * gy[r0+r][s]
template <int NS>
__device__ __forceinline__ void stage1_tr(const Leaf& lf, const float* __restrict__ L, int kc, int kn, const float* gs, float* gtb,
                                          int s, int h) {
    constexpr int H = 32 / NS;
    for (int kk = h; kk < kn; kk += H) {
        const float* gv = gs + (size_t)lf.r0 * NS + s;
        float acc = 0.f;
#pragma unroll 4
        for (int r = 0; r < lf.rows; ++r) acc = fmaf(__ldg(L + (size_t)r * lf.k + kc + kk), gv[r * NS], acc);
        gtb[kk * NS + s] = acc;
    }
}

// TR = false: y = forward(x) + bias.  TR = true: every leaf transposed, y = grad_x (B x in_dim) from x = grad_y (B x out_dim):
//     stage 1  t[kk][s]      = sum_r L_c[r][kk] * gy[r0+r][s]
//     stage 2  gx[c0+col][s] += sum_kk R_c[kk][col] * t[kk][s]
// with the forward's shared-memory layout and size (an input tile and an output tile of in_dim + out_dim features in all); bias unused.
template <int NS, bool TR>
__global__ void __launch_bounds__(HM_THREADS)
hmat_fwd_kernel(const Leaf* __restrict__ leaves, int nleaves, const float* __restrict__ params, const float* __restrict__ x,
                long ldx, float* __restrict__ y, long ldy, const float* __restrict__ bias, long B, int in_dim, int out_dim) {
    extern __shared__ __align__(16) float smem[];
    const int nx = TR ? out_dim : in_dim, ny = TR ? in_dim : out_dim;
    float* xs = smem;
    float* ys = xs + (size_t)nx * NS;
    float* tb = ys + (size_t)ny * NS + (threadIdx.x >> 5) * (HM_KCHUNK * NS);
    const long t0 = (long)blockIdx.x * NS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int s = lane % NS, h = lane / NS;
    constexpr int H = 32 / NS;

    load_tile<NS>(x, ldx, t0, B, nx, xs);
    for (int e = threadIdx.x; e < ny * NS; e += HM_THREADS) ys[e] = (!TR && bias) ? __ldg(bias + e / NS) : 0.f;
    __syncthreads();

    for (int c = warp; c < nleaves; c += HM_WARPS) {
        const Leaf lf = leaves[c];
        const float* L = params + lf.offL;
        const float* R = params + lf.offR;
        for (int kc = 0; kc < lf.k; kc += HM_KCHUNK) {
            const int kn = min(HM_KCHUNK, lf.k - kc);
            if (TR) stage1_tr<NS>(lf, L, kc, kn, xs, tb, s, h);
            else stage1<NS>(lf, R, kc, kn, xs, tb, s, h);
            __syncwarp();
            if (TR) {
                for (int col = h; col < lf.cols; col += H) {
                    const float* Rcol = R + (size_t)kc * lf.cols + col;
                    float acc = 0.f;
                    // left to the compiler, this loop costs the NS = 8 / 16 instantiations a 12-byte spill; "#pragma unroll 1" avoids it
                    // but made the C4-H grad_x 0.83 ms (13 %) slower on a B200 (DESIGN.md 4.5)
                    for (int kk = 0; kk < kn; ++kk) acc = fmaf(__ldg(Rcol + (size_t)kk * lf.cols), tb[kk * NS + s], acc);
                    atomicAdd(&ys[(size_t)(lf.c0 + col) * NS + s], acc);
                }
            } else {
                for (int r = h; r < lf.rows; r += H) {
                    const float* Lrow = L + (size_t)r * lf.k + kc;
                    float acc = 0.f;
                    for (int kk = 0; kk < kn; ++kk) acc = fmaf(__ldg(Lrow + kk), tb[kk * NS + s], acc);
                    atomicAdd(&ys[(size_t)(lf.r0 + r) * NS + s], acc);
                }
            }
            __syncwarp();
        }
    }
    __syncthreads();
    for (int sidx = 0; sidx < NS; ++sidx) {
        if (t0 + sidx >= B) break;
        float* row = y + (size_t)(t0 + sidx) * ldy;
        for (int o = threadIdx.x; o < ny; o += HM_THREADS) row[o] = ys[o * NS + sidx];
    }
}

template <int NS>
__global__ void __launch_bounds__(HM_THREADS)
hmat_bwd_kernel(const Leaf* __restrict__ leaves, int nleaves, const float* __restrict__ params, const float* __restrict__ x,
                long ldx, const float* __restrict__ gy, long ldgy, float* __restrict__ gparams, long B, int in_dim,
                int out_dim) {
    extern __shared__ __align__(16) float smem[];
    float* xs = smem;
    float* gs = xs + (size_t)in_dim * NS;
    float* tb = gs + (size_t)out_dim * NS + (threadIdx.x >> 5) * (2 * HM_KCHUNK * NS);
    float* gtb = tb + HM_KCHUNK * NS;
    const long t0 = (long)blockIdx.x * NS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int s = lane % NS, h = lane / NS;
    constexpr int H = 32 / NS;

    load_tile<NS>(x, ldx, t0, B, in_dim, xs);
    load_tile<NS>(gy, ldgy, t0, B, out_dim, gs);
    __syncthreads();

    for (int c = warp; c < nleaves; c += HM_WARPS) {
        const Leaf lf = leaves[c];
        const float* L = params + lf.offL;
        const float* R = params + lf.offR;
        for (int kc = 0; kc < lf.k; kc += HM_KCHUNK) {
            const int kn = min(HM_KCHUNK, lf.k - kc);
            stage1<NS>(lf, R, kc, kn, xs, tb, s, h);
            for (int kk = h; kk < kn; kk += H) {   // gt[kk][s] = sum_r L[r][kc+kk] * gy[r0+r][s]
                const float* gv = gs + (size_t)lf.r0 * NS + s;
                float acc = 0.f;
#pragma unroll 4
                for (int r = 0; r < lf.rows; ++r) acc = fmaf(__ldg(L + (size_t)r * lf.k + kc + kk), gv[r * NS], acc);
                gtb[kk * NS + s] = acc;
            }
            __syncwarp();
            // dL[r][kc+kk] += sum_s gy[r0+r][s] * t[kk][s]
            for (int e = lane; e < lf.rows * kn; e += 32) {
                const int r = e / kn, kk = e - r * kn;
                const float* gv = gs + (size_t)(lf.r0 + r) * NS;
                const float* tv = tb + kk * NS;
                float acc = 0.f;
#pragma unroll
                for (int q = 0; q < NS; ++q) acc = fmaf(gv[q], tv[q], acc);
                atomicAdd(gparams + lf.offL + (size_t)r * lf.k + kc + kk, acc);
            }
            // dR[kc+kk][col] += sum_s gt[kk][s] * x[c0+col][s]
            for (int e = lane; e < kn * lf.cols; e += 32) {
                const int kk = e / lf.cols, col = e - kk * lf.cols;
                const float* gv = gtb + kk * NS;
                const float* xv = xs + (size_t)(lf.c0 + col) * NS;
                float acc = 0.f;
#pragma unroll
                for (int q = 0; q < NS; ++q) acc = fmaf(gv[q], xv[q], acc);
                atomicAdd(gparams + lf.offR + (size_t)(kc + kk) * lf.cols + col, acc);
            }
            __syncwarp();
        }
    }
}

template <int NS>
size_t hm_smem(int in_dim, int out_dim, bool bwd) {
    return ((size_t)(in_dim + out_dim) * NS + (size_t)HM_WARPS * (bwd ? 2 : 1) * HM_KCHUNK * NS) * sizeof(float);
}


// ------------------------------------------------------------------------------------------
// Dense-block path (default): at training batch sizes the leaves are better served as dense blocks on the tensor cores --
//   W = sum over leaves of L_c R_c placed at the leaf's block (the leaves tile the matrix), y = x W^T + b on gemm_tf32x3,
//   dW = gy^T x on gemm_tf32x3, and the block gradients projected back onto the factors: dL_c = dW_c R_c^T, dR_c = L_c^T dW_c.
// 4.1 MFLOP/sample on tcgen05 instead of 0.7 MFLOP/sample on CUDA cores in 2 560 tiny leaf products: 20x faster at B = 8192.
// ------------------------------------------------------------------------------------------
constexpr int HD_THREADS = 256;
constexpr int HD_ROWS = 32;   // rows of a leaf handled by one CTA of the build kernel
constexpr int HP_SLAB = 32;   // ... and of the gradient projection (same work list)

__global__ void __launch_bounds__(HD_THREADS)
hmat_build_dense_kernel(const Leaf* __restrict__ leaves, const int2* __restrict__ slabs, const float* __restrict__ params, float* __restrict__ W, int ldw) {
    // slabs (the work list of the gradient projection: (leaf, first row) per 32 rows): one CTA per slab.  Without it the grid is
    // (leaves, slabs of the tallest leaf) and nearly all of its CTAs exit at once -- 20 480 CTAs for 2 887 slabs at C4-H, 53 us.
    const int2 sl = slabs != nullptr ? slabs[blockIdx.x] : make_int2((int)blockIdx.x, (int)blockIdx.y * HD_ROWS);
    const Leaf lf = leaves[sl.x];
    const int r0 = sl.y;
    if (r0 >= lf.rows) return;
    const int nr = min(HD_ROWS, lf.rows - r0);
    const float* L = params + lf.offL;    // rows x k
    const float* R = params + lf.offR;   // k x cols
    for (int e = threadIdx.x; e < nr * lf.cols; e += HD_THREADS) {
        const int i = r0 + e / lf.cols, j = e % lf.cols;
        float acc = 0.f;
        for (int k = 0; k < lf.k; ++k) acc = fmaf(__ldg(L + i * lf.k + k), __ldg(R + k * lf.cols + j), acc);
        W[(size_t)(lf.r0 + i) * ldw + lf.c0 + j] = acc;
    }
}

// One CTA per 32-row slab of a leaf (work list built by the host: the 6 + 16 largest leaves of the 2048 -> 1000 layer have 250 / 125
// rows, and one CTA per leaf spent 200 us in them at one outstanding load per thread).
// blockIdx.y == 0: dL[i][k] += sum_j dW[i][j] R[k][j]   warp per row i, lanes along j, eight ranks k at a time in registers
// blockIdx.y == 1: dR[k][j] += sum_i L[i][k] dW[i][j]   thread per column j over the slab's rows (eight loads in flight), atomics
//                                                        across the slabs of a leaf
__global__ void __launch_bounds__(HD_THREADS)
hmat_project_grad_kernel(const Leaf* __restrict__ leaves, const int2* __restrict__ slabs, const float* __restrict__ params, const float* __restrict__ dW,
                         int ldw, float* __restrict__ gparams) {
    const int2 sl = slabs[blockIdx.x];
    const Leaf lf = leaves[sl.x];
    const int r0 = sl.y, nr = min(HP_SLAB, lf.rows - r0);
    const float* L = params + lf.offL;
    const float* R = params + lf.offR;
    const float* D = dW + (size_t)(lf.r0 + r0) * ldw + lf.c0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (blockIdx.y == 0) {
        for (int i = warp; i < nr; i += HD_THREADS / 32) {
            for (int k0 = 0; k0 < lf.k; k0 += 8) {
                float acc[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) acc[q] = 0.f;
                for (int j = lane; j < lf.cols; j += 32) {
                    const float w = __ldg(D + (size_t)i * ldw + j);
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        if (k0 + q < lf.k) acc[q] = fmaf(w, __ldg(R + (k0 + q) * lf.cols + j), acc[q]);
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    float a = acc[q];
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
                    if (lane == 0 && k0 + q < lf.k) gparams[lf.offL + (r0 + i) * lf.k + k0 + q] += a;      // one owner per (row, rank)
                }
            }
        }
    } else {
        const bool single = lf.rows <= HP_SLAB;      // one slab: plain accumulation, no atomics needed
        for (int j = threadIdx.x; j < lf.cols; j += HD_THREADS) {
            for (int k0 = 0; k0 < lf.k; k0 += 8) {
                float acc[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) acc[q] = 0.f;
                for (int i0 = 0; i0 < nr; i0 += 8) {
                    float w[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) w[u] = i0 + u < nr ? __ldg(D + (size_t)(i0 + u) * ldw + j) : 0.f;
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (i0 + u >= nr) break;
#pragma unroll
                        for (int q = 0; q < 8; ++q)
                            if (k0 + q < lf.k) acc[q] = fmaf(__ldg(L + (r0 + i0 + u) * lf.k + k0 + q), w[u], acc[q]);
                    }
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    if (k0 + q >= lf.k) break;
                    float* dst = gparams + lf.offR + (k0 + q) * lf.cols + j;
                    if (single) *dst += acc[q];
                    else atomicAdd(dst, acc[q]);
                }
            }
        }
    }
}

// Launches hmat_fwd_kernel<NS, TR> at the largest sample tile NS whose shared memory fits: 0 = launched, -1 = fits at no NS.
template <bool TR>
int hm_launch_fwd(const Leaf* lv, int nleaves, const float* params, const float* x, long ldx, float* y, long ldy, const float* bias, long B,
                  int in_dim, int out_dim, cudaStream_t st) {
#define HM_LAUNCH_FWD(NS)                                                                                                  \
    {                                                                                                                      \
        size_t smem = hm_smem<NS>(in_dim, out_dim, false);                                                                 \
        if (smem <= 227 * 1024) {                                                                                          \
            SN_SET_MAX_SMEM((int)smem, hmat_fwd_kernel<NS, TR>); \
            hmat_fwd_kernel<NS, TR><<<(unsigned)((B + NS - 1) / NS), HM_THREADS, smem, st>>>(lv, nleaves, params, x, ldx, y, ldy, bias, B, in_dim, out_dim); \
            SN_CHECK_LAUNCH(TR ? "hmat_fwd_kernel<TR>" : "hmat_fwd_kernel");                                               \
            return 0;                                                                                                      \
        }                                                                                                                  \
    }
    HM_LAUNCH_FWD(16)
    HM_LAUNCH_FWD(8)
    HM_LAUNCH_FWD(4)
    HM_LAUNCH_FWD(2)
#undef HM_LAUNCH_FWD
    return -1;
}

// Launches hmat_bwd_kernel<NS> as above: 0 = launched, -1 = fits at no NS.
int hm_launch_bwd(const Leaf* lv, int nleaves, const float* params, const float* x, long ldx, const float* grad_y, long ldgy, float* grad_params,
                  long B, int in_dim, int out_dim, cudaStream_t st) {
#define HM_LAUNCH_BWD(NS)                                                                                                  \
    {                                                                                                                      \
        size_t smem = hm_smem<NS>(in_dim, out_dim, true);                                                                  \
        if (smem <= 227 * 1024) {                                                                                          \
            SN_SET_MAX_SMEM((int)smem, hmat_bwd_kernel<NS>); \
            hmat_bwd_kernel<NS><<<(unsigned)((B + NS - 1) / NS), HM_THREADS, smem, st>>>(lv, nleaves, params, x, ldx, grad_y, ldgy, grad_params, B, in_dim, out_dim); \
            SN_CHECK_LAUNCH("hmat_bwd_kernel");                                                                            \
            return 0;                                                                                                      \
        }                                                                                                                  \
    }
    HM_LAUNCH_BWD(16)
    HM_LAUNCH_BWD(8)
    HM_LAUNCH_BWD(4)
    HM_LAUNCH_BWD(2)
#undef HM_LAUNCH_BWD
    return -1;
}

}  // namespace

extern "C" {

// leaves: device table, 8 int32 per leaf {row_start, rows, col_start, cols, rank, off_left, off_right, 0};
// params: flat parameter buffer holding left_lr (rows x k) and right_lr (k x cols) of every leaf at those offsets.
int sn_hmat_forward(const int32_t* leaves, int nleaves, const float* params, const float* x, int64_t ldx, float* y, int64_t ldy,
                    const float* bias, int64_t B, int in_dim, int out_dim, sn_stream_t stream) {
    SN_CHECK_ARG(params && (leaves || nleaves == 0), "hmat_forward: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && y, "hmat_forward: NULL buffer");
    const int rc = hm_launch_fwd<false>(reinterpret_cast<const Leaf*>(leaves), nleaves, params, x, ldx, y, ldy, bias, B, in_dim, out_dim,
                                        snb::as_stream(stream));
    if (rc < 0) {
        snb::set_error("hmat_forward: in_dim + out_dim = %d does not fit in shared memory", in_dim + out_dim);
        return 1;
    }
    return rc;
}

// grad_params (nullable when grad_x is not) += the leaf gradients; grad_x (nullable; row pitch ldgx >= in_dim) = grad_y W, written by
// a second launch: the forward kernel with every leaf transposed, so every layer whose forward runs also gets its grad_x.
int sn_hmat_backward(const int32_t* leaves, int nleaves, const float* params, const float* x, int64_t ldx, const float* grad_y,
                     int64_t ldgy, float* grad_params, float* grad_bias, float* grad_x, int64_t ldgx, int64_t B, int in_dim, int out_dim,
                     sn_stream_t stream) {
    SN_CHECK_ARG(params && (leaves || nleaves == 0), "hmat_backward: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && grad_y, "hmat_backward: NULL buffer");
    SN_CHECK_ARG(grad_params || grad_x, "hmat_backward: grad_params and grad_x are both NULL");
    SN_CHECK_ARG(grad_x == nullptr || ldgx >= in_dim, "hmat_backward: grad_x leading dimension too small (ldgx %lld < in_dim %d)",
                 (long long)ldgx, in_dim);
    cudaStream_t st = snb::as_stream(stream);
    const Leaf* lv = reinterpret_cast<const Leaf*>(leaves);
    if (grad_bias)
        if (int rc = snb::colsum_accumulate(grad_y, ldgy, B, out_dim, grad_bias, st)) return rc;
    if (grad_params) {
        const int rc = hm_launch_bwd(lv, nleaves, params, x, ldx, grad_y, ldgy, grad_params, B, in_dim, out_dim, st);
        if (rc < 0) {
            snb::set_error("hmat_backward: in_dim + out_dim = %d does not fit in shared memory", in_dim + out_dim);
            return 1;
        }
        if (rc) return rc;
    }
    if (grad_x) {
        const int rc = hm_launch_fwd<true>(lv, nleaves, params, grad_y, ldgy, grad_x, ldgx, nullptr, B, in_dim, out_dim, st);
        if (rc < 0) {
            snb::set_error("hmat_backward: in_dim + out_dim = %d does not fit in shared memory", in_dim + out_dim);
            return 1;
        }
        if (rc) return rc;
    }
    return 0;
}

// W[out_dim x in_dim] (row-major, dense) = the H-matrix (zero where no leaf with rank > 0 lives)
int sn_hmat_build_dense(const int32_t* leaves, int nleaves, int max_rows, const int32_t* slabs, int nslabs, const float* params, float* W, int out_dim, int in_dim,
                        sn_stream_t stream) {
    SN_CHECK_ARG(W != nullptr && out_dim > 0 && in_dim > 0, "hmat_build_dense: bad arguments");
    cudaStream_t st = snb::as_stream(stream);
    SN_CHECK_CUDA(cudaMemsetAsync(W, 0, (size_t)out_dim * in_dim * sizeof(float), st));
    if (nleaves <= 0) return 0;
    SN_CHECK_ARG(leaves && params && max_rows > 0, "hmat_build_dense: NULL buffer");
    static_assert(HD_ROWS == HP_SLAB, "the build kernel walks the projection's slab list");
    const bool listed = slabs != nullptr && nslabs > 0;
    dim3 grid(listed ? nslabs : nleaves, listed ? 1 : snb::ceil_div(max_rows, HD_ROWS));
    SN_LAUNCH("hmat_build_dense_kernel", st, hmat_build_dense_kernel<<<grid, HD_THREADS, 0, st>>>(reinterpret_cast<const Leaf*>(leaves),
                                                                                                  listed ? reinterpret_cast<const int2*>(slabs) : nullptr, params, W, in_dim));
    return 0;
}
// grad_params (flat, accumulated) += the dense block gradients dW projected onto the leaf factors.  slabs: device int32 pairs
// (leaf index in `leaves`, first row of the slab inside the leaf), one per 32 rows of every leaf.
int sn_hmat_project_grad(const int32_t* leaves, int nleaves, const int32_t* slabs, int nslabs, const float* params, const float* dW, int out_dim, int in_dim,
                         float* grad_params, sn_stream_t stream) {
    (void)out_dim;
    if (nleaves <= 0 || nslabs <= 0) return 0;
    SN_CHECK_ARG(leaves && slabs && params && dW && grad_params, "hmat_project_grad: NULL buffer");
    cudaStream_t st = snb::as_stream(stream);
    SN_LAUNCH("hmat_project_grad_kernel", st, hmat_project_grad_kernel<<<dim3(nslabs, 2), HD_THREADS, 0, st>>>(reinterpret_cast<const Leaf*>(leaves), reinterpret_cast<const int2*>(slabs), params, dW, in_dim, grad_params));
    return 0;
}

}  // extern "C"
