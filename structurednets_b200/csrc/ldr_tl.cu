// Low-displacement-rank (tridiagonal-plus-corners operators) and Toeplitz-like layers.
//
// LDR replaces LDRLayer.forward = build_weight_matrix_torch + matmul (reference layers/ldr_layer.py:44-61,
// approximators/ldr_approximator.py:29-39) and its autograd backward.  The reference materialises
//     W = sum_i K(A, g_i) K(B^T, h_i)^T ,   K(M, v) = [v, Mv, ..., M^{n-1} v]
// with matrix_power per column (O(r n^4 log n)).  Here the Krylov blocks are built by the recurrence
//     KA_0 = G, KA_{j+1} = A KA_j ;   KB_0 = H, KB_{j+1} = B^T KB_j          (n x r each, float64, banded operator: O(n r) per step)
// by ONE kernel per call (a CTA keeps a few columns in shared memory and walks all the powers), and
//     W = sum_j KA_j KB_j^T = [KA_0 | KA_1 | ...] [KB_0 | KB_1 | ...]^T
// is a single dense contraction over K = r J on the tensor cores (3xTF32, fp32-accurate: the reference accumulates its float64
// terms into a float32 matrix, approximators/ldr_approximator.py:31,37).  J, the number of powers that matter, is found ON THE
// DEVICE from the columns' max-norms (term j is bounded by sum_i |KA_j[:,i]|_inf |KB_j[:,i]|_inf) and handed to the GEMM through
// device memory (gemm_tf32x3's kdev / mdev): no host synchronisation, the whole step can be captured in a CUDA graph.
// Backward: dKA = dW KB, dKB = dW^T KA (two tensor-core GEMMs), then the adjoint recurrences in float64 (one kernel)
//     abar_{J-1} = dK_{J-1}, abar_j = dK_j + M^T abar_{j+1} ;   dM += pattern( abar_{j+1} K_j^T ) ;   dG (dH) = abar_0 .
//
// Toeplitz-like replaces TLLayer.forward (reference layers/tl_layer.py:11-18,51-68):
//     W = 1/2 sum_j Krylov(Z_1, G[:,j]) Krylov(Z_-1, flip(H[j,:]))
// built as one (n x rn)(rn x n) fp32 GEMM from the two explicitly formed f-circulant Krylov stacks.
#include "gemm_f32.cuh"
#include "util.cuh"

namespace {

// slot map entry: 0..n-1 -> lo, n..2n-1 -> di, 2n..3n-1 -> up, 3n -> corner(0,n-1), 3n+1 -> corner(n-1,0)
//   lo[p] = M[p][p-1] (lo[0] unused = 0), di[p] = M[p][p], up[p] = M[p][p+1] (up[n-1] unused = 0)
__global__ void band_gather_kernel(const double* __restrict__ vals, const int* __restrict__ slot, int nnz, double* __restrict__ band) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < nnz) atomicAdd(band + slot[e], vals[e]);
}
__global__ void band_scatter_grad_kernel(const double* __restrict__ gband, const int* __restrict__ slot, int nnz, double* __restrict__ gvals) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < nnz) gvals[e] += gband[slot[e]];
}
// band of M^T from band of M
__global__ void band_transpose_kernel(const double* __restrict__ b, double* __restrict__ t, int n) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) {
        t[p] = p > 0 ? b[2 * n + p - 1] : 0.0;          // lo'[p] = up[p-1]
        t[n + p] = b[n + p];
        t[2 * n + p] = p + 1 < n ? b[p + 1] : 0.0;      // up'[p] = lo[p+1]
    }
    if (p == 0) { t[3 * n] = b[3 * n + 1]; t[3 * n + 1] = b[3 * n]; }
}

constexpr int KR_THREADS = 1024;
__host__ __device__ inline int kr_cols_fwd(int n) { int c = 12800 / n; return c > 8 ? 8 : c; }          // 2 buffers of n x C doubles <= 200 KB
__host__ __device__ inline int kr_cols_bwd(int n) { int c = (25600 / n - 3) / 2; return c > 8 ? 8 : c; }  // 2 buffers + 3 n-vectors of band gradients

// Krylov blocks of one operator (blockIdx.y = 0: M = A, start G; 1: M = B^T, start H) for the CTA's columns [c0, c0 + C):
//   K64[op][j][i][p]  (float64, p contiguous)  and  K32[op][j r + i][p]  (float32, the MN-major GEMM operand), j < J;
//   colnorm[op][j][i] = max_p |K_j[p][i]|.
__global__ void __launch_bounds__(KR_THREADS)
ldr_krylov_kernel(int n, int r, int J, int C, const double* __restrict__ bands, const double* __restrict__ G, const double* __restrict__ H,
                  double* __restrict__ K64, float* __restrict__ K32, long k32_rows, double* __restrict__ colnorm) {
    extern __shared__ __align__(16) double kr_smem[];
    __shared__ double red[8][32];
    const int op = blockIdx.y, c0 = blockIdx.x * C, nc = min(C, r - c0), tid = threadIdx.x;
    const double* band = bands + (size_t)op * (3 * n + 2);
    const double* lo = band, *di = band + n, *up = band + 2 * n;
    const double cn0 = n > 2 ? band[3 * n] : 0.0, cn1 = n > 2 ? band[3 * n + 1] : 0.0;
    const double* src = op == 0 ? G : H;
    double* cur = kr_smem;
    double* nxt = kr_smem + (size_t)C * n;
    for (int e = tid; e < nc * n; e += KR_THREADS) {       // e = p * nc + c: the n x r row-major source is read nc-contiguous
        const int p = e / nc, c = e - p * nc;
        cur[(size_t)c * n + p] = src[(size_t)p * r + c0 + c];
    }
    __syncthreads();
    double* k64 = K64 + (size_t)op * J * r * n;
    float* k32 = K32 + (size_t)op * k32_rows * n;
    for (int j = 0; j < J; ++j) {
        // one pass over the rows for all of the CTA's columns: two barriers per power (norms, buffer swap)
        double mx[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) mx[c] = 0.0;
        for (int p = tid; p < n; p += KR_THREADS) {
            const double dp = di[p], lp = p > 0 ? lo[p] : 0.0, upp = p + 1 < n ? up[p] : 0.0;
            const int pm = p > 0 ? p - 1 : 0, pp = p + 1 < n ? p + 1 : p;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                if (c >= nc) break;
                const double* v = cur + (size_t)c * n;
                const double x = v[p];
                const size_t row = ((size_t)j * r + c0 + c) * n + p;
                k64[row] = x;
                k32[row] = (float)x;
                mx[c] = fmax(mx[c], fabs(x));
                double acc = dp * x + lp * v[pm] + upp * v[pp];
                if (p == 0) acc += cn0 * v[n - 1];
                if (p == n - 1) acc += cn1 * v[0];
                nxt[(size_t)c * n + p] = acc;
            }
        }
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            if (c >= nc) break;
            double m = mx[c];
            for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
            if ((tid & 31) == 0) red[c][tid >> 5] = m;
        }
        __syncthreads();
        if (tid < 32 * nc) {
            const int c = tid >> 5;
            double m = red[c][tid & 31];
            for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
            if ((tid & 31) == 0) colnorm[((size_t)op * J + j) * r + c0 + c] = m;
        }
        __syncthreads();
        double* t = cur; cur = nxt; nxt = t;
    }
}

// status[0] = J_eff (powers that matter), status[1] = K_eff = min(round_up(J_eff r, 32), k32_rows), status[2] = 1 when the series
// ended inside the J computed powers (or J = n: the reference sums exactly n powers), status[3] = J.
__global__ void ldr_terms_kernel(int n, int r, int J, long k32_rows, double rel_tol, const double* __restrict__ colnorm, int* __restrict__ status) {
    __shared__ double bound[1024];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    for (int j = warp; j < J; j += nwarps) {       // one warp per power: coalesced reads of the two norm rows
        double b = 0.0;
        for (int i = lane; i < r; i += 32) b += colnorm[(size_t)j * r + i] * colnorm[((size_t)J + j) * r + i];
        for (int o = 16; o > 0; o >>= 1) b += __shfl_xor_sync(0xffffffffu, b, o);
        if (lane == 0) bound[j] = b;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double mx = 0.0;
        int terms = J, conv = (J >= n) ? 1 : 0;
        for (int j = 0; j < J; ++j) {
            const double b = bound[j];
            if (j > 0 && !(b > rel_tol * mx)) { terms = j; conv = 1; break; }
            mx = fmax(mx, b);
        }
        long k = ((long)terms * r + 31) / 32 * 32;
        if (k > k32_rows) k = k32_rows;
        status[0] = terms; status[1] = (int)k; status[2] = conv; status[3] = J;
    }
}

// Adjoint recurrences for the CTA's columns; gband[op] += band gradient of M (atomics over CTAs), gsrc (gG or gH, n x r) += abar_0.
// Column i takes part in the powers j < J_i = number of its rows below K_eff in the stacked operand (the GEMM rounds K up to 32).
__global__ void __launch_bounds__(KR_THREADS)
ldr_krylov_bwd_kernel(int n, int r, int J, int C, const double* __restrict__ bands, const double* __restrict__ K64, const float* __restrict__ dK32,
                      long k32_rows, const int* __restrict__ status, double* __restrict__ gbands, double* __restrict__ gG, double* __restrict__ gH) {
    extern __shared__ __align__(16) double kr_smem[];
    const int op = blockIdx.y, c0 = blockIdx.x * C, nc = min(C, r - c0), tid = threadIdx.x;
    const double* band = bands + (size_t)op * (3 * n + 2);
    const double* lo = band, *di = band + n, *up = band + 2 * n;
    const double cn0 = n > 2 ? band[3 * n] : 0.0, cn1 = n > 2 ? band[3 * n + 1] : 0.0;
    const int k_eff = status[1];
    double* cur = kr_smem;                       // abar_{j+1}
    double* nxt = kr_smem + (size_t)C * n;
    double* glo = kr_smem + (size_t)2 * C * n, *gdi = glo + n, *gup = gdi + n;
    __shared__ double gcn[2];
    for (int p = tid; p < n; p += KR_THREADS) { glo[p] = 0.0; gdi[p] = 0.0; gup[p] = 0.0; }
    if (tid < 2) gcn[tid] = 0.0;
    const double* k64 = K64 + (size_t)op * J * r * n;
    const float* dk = dK32 + (size_t)op * k32_rows * n;
    int jmax = 0;                                // powers of the CTA's first column (the largest count among its columns)
    if (k_eff > c0) jmax = (k_eff - c0 + r - 1) / r;
    if (jmax > J) jmax = J;
    for (int e = tid; e < C * n; e += KR_THREADS) cur[e] = 0.0;
    __syncthreads();
    for (int j = jmax - 1; j >= 0; --j) {
        double c0acc = 0.0, c1acc = 0.0;
        for (int p = tid; p < n; p += KR_THREADS) {
            const double dp = di[p], lnext = p + 1 < n ? lo[p + 1] : 0.0, uprev = p > 0 ? up[p - 1] : 0.0;
            const int pm = p > 0 ? p - 1 : 0, pp = p + 1 < n ? p + 1 : p;
            double g_lo = 0.0, g_di = 0.0, g_up = 0.0;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                if (c >= nc) break;
                const bool live = (long)j * r + c0 + c < k_eff;           // uniform over the CTA
                const double* a = cur + (size_t)c * n;                   // abar_{j+1} (zero when j is the column's last power)
                const double* kj = k64 + ((size_t)j * r + c0 + c) * n;   // K_j
                const double ap = a[p];
                // band gradient of the step K_{j+1} = M K_j:  dM[p][p'] += abar_{j+1}[p] K_j[p']
                g_di += ap * kj[p];
                if (p > 0) g_lo += ap * kj[pm];
                if (p + 1 < n) g_up += ap * kj[pp];
                if (p == 0) c0acc += ap * kj[n - 1];
                if (p == n - 1) c1acc += ap * kj[0];
                // abar_j = dK_j + M^T abar_{j+1}
                double acc = dp * ap + lnext * a[pp] + uprev * a[pm];
                if (p == n - 1) acc += cn0 * a[0];
                if (p == 0) acc += cn1 * a[n - 1];
                nxt[(size_t)c * n + p] = live ? acc + (double)dk[((size_t)j * r + c0 + c) * n + p] : 0.0;
            }
            glo[p] += g_lo; gdi[p] += g_di; gup[p] += g_up;
        }
        if (n > 2) {
            if (tid == 0) gcn[0] += c0acc;                          // p = 0 belongs to thread 0
            if (tid == (n - 1) % KR_THREADS) gcn[1] += c1acc;       // p = n - 1 belongs to exactly this thread
        }
        __syncthreads();
        double* t = cur; cur = nxt; nxt = t;
    }
    // cur = abar_0 of the CTA's columns
    double* gsrc = op == 0 ? gG : gH;
    if (gsrc != nullptr)
        for (int e = tid; e < nc * n; e += KR_THREADS) {
            const int p = e / nc, c = e - p * nc;
            gsrc[(size_t)p * r + c0 + c] += cur[(size_t)c * n + p];
        }
    double* gb = gbands + (size_t)op * (3 * n + 2);
    for (int p = tid; p < n; p += KR_THREADS) {
        if (p > 0) atomicAdd(gb + p, glo[p]);
        atomicAdd(gb + n + p, gdi[p]);
        if (p + 1 < n) atomicAdd(gb + 2 * n + p, gup[p]);
    }
    __syncthreads();
    if (tid == 0 && n > 2) { atomicAdd(gb + 3 * n, gcn[0]); atomicAdd(gb + 3 * n + 1, gcn[1]); }
}

inline dim3 grid2(int n) { return dim3(snb::ceil_div(n, 128), n); }
inline unsigned grid1(size_t n) { return (unsigned)((n + 255) / 256); }

// ---- Toeplitz-like helpers ----------------------------------------------------------------------
// K1[p][j*n+i] = G[(p-i) mod n][j]                       (Krylov(Z_1, G[:,j]))
__global__ void tl_k1_kernel(const float* __restrict__ G, float* __restrict__ K1, int n, int r) {
    int c = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;   // c = j*n + i
    if (c >= n * r) return;
    int j = c / n, i = c - j * n;
    int m = p - i; if (m < 0) m += n;
    K1[(size_t)p * n * r + c] = G[(size_t)m * r + j];
}
// K2[j*n+i][q] = v_j[(i-q) mod n] * (i < q ? -1 : 1),  v_j[m] = H[j][n-1-m]     (Krylov(Z_-1, flip(H[j,:])))
__global__ void tl_k2_kernel(const float* __restrict__ H, float* __restrict__ K2, int n, int r) {
    int q = blockIdx.y * blockDim.x + threadIdx.x, row = blockIdx.x;  // row = j*n + i  (n*r rows: on grid.x, grid.y stops at 65 535)
    if (q >= n) return;
    int j = row / n, i = row - j * n;
    int m = i - q; if (m < 0) m += n;
    float v = H[(size_t)j * n + (n - 1 - m)];
    K2[(size_t)row * n + q] = i < q ? -v : v;
}
// dG[m][j] += sum_i dK1[(m+i) mod n][j*n+i]
__global__ void tl_dg_kernel(const float* __restrict__ dK1, float* __restrict__ dG, int n, int r) {
    int j = blockIdx.x * blockDim.x + threadIdx.x, m = blockIdx.y;
    if (j >= r) return;
    float s = 0.f;
    for (int i = 0; i < n; ++i) {
        int p = m + i; if (p >= n) p -= n;
        s += dK1[(size_t)p * n * r + (size_t)j * n + i];
    }
    dG[(size_t)m * r + j] += s;
}
// dH[j][n-1-m] += sum_q sign * dK2[j*n + (m+q) mod n][q]
__global__ void tl_dh_kernel(const float* __restrict__ dK2, float* __restrict__ dH, int n, int r) {
    int m = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    if (m >= n) return;
    float s = 0.f;
    for (int q = 0; q < n; ++q) {
        int i = m + q; if (i >= n) i -= n;
        float v = dK2[((size_t)j * n + i) * n + q];
        s += i < q ? -v : v;
    }
    dH[(size_t)j * n + (n - 1 - m)] += s;
}

}  // namespace

extern "C" {

// Workspace layout (bytes, every part 256-byte aligned); J = max_terms powers are computed, K32 rows = round_up(J r, 32):
//   bands [2][3n+2] f64 (A, B^T) | gbands [2][3n+2] f64 | scratch band [3n+2] f64 | colnorm [2][J][r] f64 | K64 [2][J][r][n] f64
//   | K32 [2][rows][n] f32 | dK32 [2][rows][n] f32
namespace {
struct LdrWs {
    size_t bands, gbands, tmpband, colnorm, k64, k32, dk32, total;
    long rows;
};
inline LdrWs ldr_layout(int n, int r, int J) {
    auto al = [](size_t x) { return (x + 255) / 256 * 256; };
    LdrWs w;
    const size_t nb = 3 * (size_t)n + 2;
    w.rows = ((long)J * r + 31) / 32 * 32;
    if (w.rows < 32) w.rows = 32;
    size_t off = 0;
    w.bands = off; off = al(off + 2 * nb * 8);
    w.gbands = off; off = al(off + 2 * nb * 8);
    w.tmpband = off; off = al(off + nb * 8);
    w.colnorm = off; off = al(off + 2 * (size_t)J * r * 8);
    w.k64 = off; off = al(off + 2 * (size_t)J * r * n * 8);
    w.k32 = off; off = al(off + 2 * (size_t)w.rows * n * 4);
    w.dk32 = off; off = al(off + 2 * (size_t)w.rows * n * 4);
    w.total = off;
    return w;
}
}  // namespace

size_t sn_ldr_workspace_bytes(int n, int r, int max_terms) {
    if (n <= 0 || r < 0 || max_terms < 1) return 0;
    return ldr_layout(n, r, max_terms).total;
}

// Builds W (n x n float32, row-major) from the representation (A, B: COO value arrays + slot maps; G, H: n x r float64
// row-major).  `slot` maps each COO entry to lo/di/up/corner (see band_gather_kernel).  max_terms <= min(n, 1024) Krylov powers are
// computed; status (device int[4]) receives {powers used J_eff, K_eff, converged, max_terms}: converged = 0 means the series had
// not decayed below rel_tol within max_terms powers -- the caller re-runs with a larger max_terms (W is then a truncated sum).
// Never synchronises; the workspace keeps what sn_ldr_backward needs.
int sn_ldr_build_weight(int n, int r, const double* A_vals, const int32_t* A_slot, int A_nnz, const double* B_vals,
                        const int32_t* B_slot, int B_nnz, const double* G, const double* H, void* ws, int max_terms,
                        double rel_tol, float* W_out, int* status, sn_stream_t stream) {
    SN_CHECK_ARG(n > 0 && r >= 0 && ws && W_out && status && max_terms >= 1 && max_terms <= 1024, "ldr_build_weight: bad arguments");
    SN_CHECK_ARG(n % 4 == 0, "ldr_build_weight: n must be a multiple of 4 (TMA row pitch of the Krylov operands), got %d", n);
    SN_CHECK_ARG(n <= 4096, "ldr_build_weight: n = %d is too large for the shared-memory Krylov kernels and the unsplit gradient GEMMs (n <= 4096)", n);
    cudaStream_t st = snb::as_stream(stream);
    const int J = max_terms < n ? max_terms : n;
    const LdrWs L = ldr_layout(n, r, max_terms);
    uint8_t* base = static_cast<uint8_t*>(ws);
    const size_t nb = 3 * (size_t)n + 2, n2 = (size_t)n * n;
    double* bands = reinterpret_cast<double*>(base + L.bands);
    double* tmpband = reinterpret_cast<double*>(base + L.tmpband);
    float* K32 = reinterpret_cast<float*>(base + L.k32);
    SN_CHECK_CUDA(cudaMemsetAsync(W_out, 0, n2 * sizeof(float), st));
    if (r == 0) {
        SN_CHECK_CUDA(cudaMemsetAsync(status, 0, 4 * sizeof(int), st));
        return 0;
    }
    SN_CHECK_CUDA(cudaMemsetAsync(bands, 0, nb * sizeof(double), st));
    SN_CHECK_CUDA(cudaMemsetAsync(tmpband, 0, nb * sizeof(double), st));
    if (A_nnz) { band_gather_kernel<<<grid1(A_nnz), 256, 0, st>>>(A_vals, A_slot, A_nnz, bands); SN_CHECK_LAUNCH("band_gather"); }
    if (B_nnz) { band_gather_kernel<<<grid1(B_nnz), 256, 0, st>>>(B_vals, B_slot, B_nnz, tmpband); SN_CHECK_LAUNCH("band_gather"); }
    band_transpose_kernel<<<snb::ceil_div(n, 128), 128, 0, st>>>(tmpband, bands + nb, n); SN_CHECK_LAUNCH("band_transpose");
    // rows of the stacked operands beyond J r (K is rounded up to the GEMM's 32-row boxes) stay zero
    if (L.rows > (long)J * r) {
        for (int op = 0; op < 2; ++op)
            SN_CHECK_CUDA(cudaMemsetAsync(K32 + ((size_t)op * L.rows + (size_t)J * r) * n, 0, (size_t)(L.rows - (long)J * r) * n * sizeof(float), st));
    }
    const int C = kr_cols_fwd(n);
    const size_t smem = (size_t)2 * C * n * sizeof(double);
    SN_SET_MAX_SMEM((int)smem, ldr_krylov_kernel);
    SN_LAUNCH("ldr_krylov_kernel", st, ldr_krylov_kernel<<<dim3(snb::ceil_div(r, C), 2), KR_THREADS, smem, st>>>(
        n, r, J, C, bands, G, H, reinterpret_cast<double*>(base + L.k64), K32, L.rows, reinterpret_cast<double*>(base + L.colnorm)));
    SN_LAUNCH("ldr_terms_kernel", st, ldr_terms_kernel<<<1, 1024, 0, st>>>(n, r, J, L.rows, rel_tol, reinterpret_cast<double*>(base + L.colnorm), status));
    // W[p][q] = sum_k KA[k][p] KB[k][q]: both operands MN-major, K = status[1] on the device, split-K with reductions into the zeroed W
    return snb::gemm_f32(true, false, n, n, (int)L.rows, 1.f, K32, n, K32 + (size_t)L.rows * n, n, 1.f, W_out, n, nullptr, st, true, status + 1, nullptr);
}

// Backward of the weight build.  dW: n x n float32 (d loss / d W).  Accumulates into gA_vals / gB_vals (COO order,
// float64), gG, gH (n x r float64).  `ws`, `max_terms`, `status` as left behind by sn_ldr_build_weight.
int sn_ldr_backward(int n, int r, const float* dW, const int32_t* A_slot, int A_nnz, const int32_t* B_slot, int B_nnz,
                    void* ws, int max_terms, const int* status, double* gA_vals, double* gB_vals, double* gG, double* gH, sn_stream_t stream) {
    SN_CHECK_ARG(n > 0 && dW && ws && status && max_terms >= 1, "ldr_backward: bad arguments");
    if (r == 0) return 0;
    cudaStream_t st = snb::as_stream(stream);
    const int J = max_terms < n ? max_terms : n;
    const LdrWs L = ldr_layout(n, r, max_terms);
    uint8_t* base = static_cast<uint8_t*>(ws);
    const size_t nb = 3 * (size_t)n + 2;
    double* bands = reinterpret_cast<double*>(base + L.bands);
    double* gbands = reinterpret_cast<double*>(base + L.gbands);
    double* tmpband = reinterpret_cast<double*>(base + L.tmpband);
    float* K32 = reinterpret_cast<float*>(base + L.k32);
    float* dK32 = reinterpret_cast<float*>(base + L.dk32);
    const float* KA = K32, *KB = K32 + (size_t)L.rows * n;
    // dKA[k][p] = sum_q KB[k][q] dW[p][q]  (A operand K-major, B operand = dW as [N = p][K = q], K-major); rows k < K_eff only
    if (int rc = snb::gemm_f32(false, true, (int)L.rows, n, n, 1.f, KB, n, dW, n, 0.f, dK32, n, nullptr, st, false, nullptr, status + 1)) return rc;
    // dKB[k][q] = sum_p KA[k][p] dW[p][q]  (B operand = dW as [K = p][N = q], MN-major)
    if (int rc = snb::gemm_f32(false, false, (int)L.rows, n, n, 1.f, KA, n, dW, n, 0.f, dK32 + (size_t)L.rows * n, n, nullptr, st, false, nullptr, status + 1)) return rc;
    SN_CHECK_CUDA(cudaMemsetAsync(gbands, 0, 2 * nb * sizeof(double), st));
    const int C = kr_cols_bwd(n);
    const size_t smem = ((size_t)2 * C * n + 3 * (size_t)n) * sizeof(double);
    SN_SET_MAX_SMEM((int)smem, ldr_krylov_bwd_kernel);
    SN_LAUNCH("ldr_krylov_bwd_kernel", st, ldr_krylov_bwd_kernel<<<dim3(snb::ceil_div(r, C), 2), KR_THREADS, smem, st>>>(
        n, r, J, C, bands, reinterpret_cast<const double*>(base + L.k64), dK32, L.rows, status, gbands, gG, gH));
    if (gA_vals && A_nnz) { band_scatter_grad_kernel<<<grid1(A_nnz), 256, 0, st>>>(gbands, A_slot, A_nnz, gA_vals); SN_CHECK_LAUNCH("band_scatter_grad"); }
    if (gB_vals && B_nnz) {
        // the second operator is B^T: its band gradient transposed is the band gradient of B
        band_transpose_kernel<<<snb::ceil_div(n, 128), 128, 0, st>>>(gbands + nb, tmpband, n); SN_CHECK_LAUNCH("band_transpose");
        band_scatter_grad_kernel<<<grid1(B_nnz), 256, 0, st>>>(tmpband, B_slot, B_nnz, gB_vals); SN_CHECK_LAUNCH("band_scatter_grad");
    }
    return 0;
}

// y[B x n_out] = x[B x n_in] W^T + bias  and  dW[n_out x n_in] += gy^T x ; plain fp32 GEMMs shared by LDR and TL.
int sn_dense_apply(const float* W, int n_out, int n_in, const float* x, int64_t ldx, float* y, int64_t ldy, const float* bias,
                   int64_t B, sn_stream_t stream) {
    SN_CHECK_ARG(W, "dense_apply: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && y, "dense_apply: NULL buffer");
    return snb::gemm_f32(false, true, (int)B, n_out, n_in, 1.f, x, ldx, W, n_in, 0.f, y, ldy, bias, snb::as_stream(stream));
}
int sn_dense_weight_grad(const float* x, int64_t ldx, const float* gy, int64_t ldgy, float* dW, int n_out, int n_in, float* grad_bias,
                         int64_t B, sn_stream_t stream) {
    SN_CHECK_ARG(dW, "dense_weight_grad: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && gy, "dense_weight_grad: NULL buffer");
    cudaStream_t st = snb::as_stream(stream);
    if (grad_bias)
        if (int rc = snb::colsum_accumulate(gy, ldgy, B, n_out, grad_bias, st)) return rc;
    return snb::gemm_f32(true, false, n_out, n_in, (int)B, 1.f, gy, ldgy, x, ldx, 1.f, dW, n_in, nullptr, st, true);
}

// grad_x[B x n_in] = grad_y[B x n_out] W  (the gradient w.r.t. the input features of every layer that materialises W)
int sn_dense_input_grad(const float* W, int n_out, int n_in, const float* gy, int64_t ldgy, float* gx, int64_t ldgx, int64_t B, sn_stream_t stream) {
    SN_CHECK_ARG(W, "dense_input_grad: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(gy && gx, "dense_input_grad: NULL buffer");
    return snb::gemm_f32(false, false, (int)B, n_in, n_out, 1.f, gy, ldgy, W, n_in, 0.f, gx, ldgx, nullptr, snb::as_stream(stream));
}

// Toeplitz-like weight: W (n x n) from G (n x r), H (r x n); K1 (n x rn) and K2 (rn x n) are caller-provided scratch
// that sn_tl_backward reuses.
int sn_tl_build_weight(int n, int r, const float* G, const float* H, float* K1, float* K2, float* W, sn_stream_t stream) {
    SN_CHECK_ARG(n > 0 && r > 0 && G && H && K1 && K2 && W, "tl_build_weight: bad arguments");
    cudaStream_t st = snb::as_stream(stream);
    tl_k1_kernel<<<dim3(snb::ceil_div(n * r, 128), n), 128, 0, st>>>(G, K1, n, r); SN_CHECK_LAUNCH("tl_k1_kernel");
    tl_k2_kernel<<<dim3(n * r, snb::ceil_div(n, 128)), 128, 0, st>>>(H, K2, n, r); SN_CHECK_LAUNCH("tl_k2_kernel");
    return snb::gemm_f32(false, false, n, n, n * r, 0.5f, K1, (long)n * r, K2, n, 0.f, W, n, nullptr, st);
}
// dK1 / dK2: scratch of the same sizes as K1 / K2; gG (n x r), gH (r x n) are accumulated into.
int sn_tl_backward(int n, int r, const float* dW, const float* K1, const float* K2, float* dK1, float* dK2, float* gG, float* gH,
                   sn_stream_t stream) {
    SN_CHECK_ARG(n > 0 && r > 0 && dW && K1 && K2 && dK1 && dK2 && gG && gH, "tl_backward: bad arguments");
    cudaStream_t st = snb::as_stream(stream);
    // dK1 = 0.5 dW K2^T  (n x n)(rn x n)^T ; dK2 = 0.5 K1^T dW  (n x rn)^T (n x n)
    if (int rc = snb::gemm_f32(false, true, n, n * r, n, 0.5f, dW, n, K2, n, 0.f, dK1, (long)n * r, nullptr, st)) return rc;
    if (int rc = snb::gemm_f32(true, false, n * r, n, n, 0.5f, K1, (long)n * r, dW, n, 0.f, dK2, n, nullptr, st)) return rc;
    tl_dg_kernel<<<dim3(snb::ceil_div(r, 32), n), 32, 0, st>>>(dK1, gG, n, r); SN_CHECK_LAUNCH("tl_dg_kernel");
    tl_dh_kernel<<<dim3(snb::ceil_div(n, 128), r), 128, 0, st>>>(dK2, gH, n, r); SN_CHECK_LAUNCH("tl_dh_kernel");
    return 0;
}

}  // extern "C"
