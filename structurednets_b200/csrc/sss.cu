// SSS (sequentially semiseparable / time-varying state-space) layer: forward and backward.
//
// Replaces SSSLayer.forward (reference layers/sss_layer.py:99-131) and the autograd graph torch
// builds from it.  Math per sample (SURVEY.md section 3b):
//   causal     k = 0..n-1 :  y_k  = C_k x_k + D_k u_k ;  x_{k+1} = A_k x_k + B_k u_k
//   anticausal k = n-1..0 :  y_k += G_k z_{k+1}       ;  z_k     = E_k z_{k+1} + F_k u_k
//
// Data layout.  Both sweeps are expressed as the same "stage step"
//       [ s_out ; y ] = P_k [ s_in ; u_k ]            P_k = [ A B ; C D ]  or  [ E F ; G 0 ]
// on a per-direction stage table (sn_sss_stage).  sn_sss_pack() re-lays the flat parameter buffer
// out per stage as  Pt[i][rows_pad]  (input-major: the forward / recompute loops read one float4
// of 4 consecutive output rows per input i)  followed by  P[r][k_pad]  (row-major: the adjoint loop
// reads one float4 of 4 consecutive inputs per output row r).  Rows are ordered state rows first,
// then y rows, zero padded.
//
// Thread mapping (SIMT fp32; the arithmetic intensity of this layer, ~56 flop/B, is above the
// fp32 ridge, so the FMA pipe is the binding roof -- DESIGN.md).  Per-sample vectors live in shared
// memory FEATURE-MAJOR ([feature][sample]), so a lane reads 4 samples of one feature with one
// LDS.128 and 4 rows of one input with one broadcast float4, giving 16 FMAs per 2 loads:
//   lane = (row-group slot, sample quad);  a warp owns NSW = 4*NQ samples of ONE direction and walks
//   all stages; the state is exchanged between lanes through a ping-pong buffer + __syncwarp().
//
// y is produced by two sweeps that meet in the middle: the first visitor of a stage stores
// (bias + part), the second one adds to it after a block barrier (deterministic, no atomics).
#include "common.cuh"

namespace {

using snb::ceil_div;
using snb::round_up;

constexpr int SSS_HDR = 8;   // floats at the head of every packed stage block: the stage descriptor

struct Geom {
    int rgs;    // row-group slots per warp
    int nq;     // sample quads per warp
    int nsw;    // samples per warp = 4*nq
    int nswp;   // padded row stride (floats) of per-warp buffers
};

// row stride such that consecutive rows start 4,12,20 or 28 banks apart (conflict-free float4 access
// for up to 8 consecutive rows)
__host__ __device__ inline int pad_stride(int n) {
    int s = round_up(n, 4);
    while (((s & 31) & 7) != 4) s += 4;
    return s;
}

inline Geom make_geom(int rows_pad) {
    Geom g;
    int nrg = rows_pad / 4;
    g.rgs = nrg < 8 ? nrg : 8;
    if (g.rgs < 1) g.rgs = 1;
    g.nq = 32 / g.rgs;
    g.nsw = 4 * g.nq;
    g.nswp = pad_stride(g.nsw);
    return g;
}

// ------------------------------------------------------------------------------------------
// pack
// ------------------------------------------------------------------------------------------
__global__ void sss_pack_kernel(const sn_sss_stage* __restrict__ stages, int total_stages, int RP, int KP,
                                const float* __restrict__ params, float* __restrict__ packed) {
    int sidx = blockIdx.x;
    if (sidx >= total_stages) return;
    sn_sss_stage st = stages[sidx];
    const int K = st.d_in + st.in_dim;
    const int rows = st.d_out + st.out_dim;
    int* hdr = reinterpret_cast<int*>(packed + st.pack_off);
    if (threadIdx.x < SSS_HDR) {
        const int h[SSS_HDR] = {st.in_off, st.in_dim, st.out_off, st.out_dim, st.d_in, st.d_out, st.k, 0};
        hdr[threadIdx.x] = h[threadIdx.x];
    }
    float* Pt = packed + st.pack_off + SSS_HDR;
    float* P = Pt + (size_t)KP * RP;
    for (int e = threadIdx.x; e < KP * RP; e += blockDim.x) {
        int i = e / RP, r = e - i * RP;
        float v = 0.f;
        if (i < K && r < rows) {
            if (r < st.d_out) {
                v = (i < st.d_in) ? params[st.off_ss + r * st.d_in + i] : params[st.off_su + r * st.in_dim + (i - st.d_in)];
            } else {
                int ry = r - st.d_out;
                if (i < st.d_in) v = params[st.off_ys + ry * st.d_in + i];
                else if (st.off_yu >= 0) v = params[st.off_yu + ry * st.in_dim + (i - st.d_in)];
            }
        }
        Pt[e] = v;
        P[(size_t)r * KP + i] = v;
    }
}

__device__ __forceinline__ void fma16(float (&acc)[4][4], const float4& p, const float4& v) {
    acc[0][0] = fmaf(p.x, v.x, acc[0][0]); acc[0][1] = fmaf(p.x, v.y, acc[0][1]);
    acc[0][2] = fmaf(p.x, v.z, acc[0][2]); acc[0][3] = fmaf(p.x, v.w, acc[0][3]);
    acc[1][0] = fmaf(p.y, v.x, acc[1][0]); acc[1][1] = fmaf(p.y, v.y, acc[1][1]);
    acc[1][2] = fmaf(p.y, v.z, acc[1][2]); acc[1][3] = fmaf(p.y, v.w, acc[1][3]);
    acc[2][0] = fmaf(p.z, v.x, acc[2][0]); acc[2][1] = fmaf(p.z, v.y, acc[2][1]);
    acc[2][2] = fmaf(p.z, v.z, acc[2][2]); acc[2][3] = fmaf(p.z, v.w, acc[2][3]);
    acc[3][0] = fmaf(p.w, v.x, acc[3][0]); acc[3][1] = fmaf(p.w, v.y, acc[3][1]);
    acc[3][2] = fmaf(p.w, v.z, acc[3][2]); acc[3][3] = fmaf(p.w, v.w, acc[3][3]);
}

// acc += sum_{i<CNT} prow[i*PSTRIDE4] (x) xv[i*VSTRIDE]  -- compile-time trip count and strides: fully unrolled,
// immediate-offset loads the scheduler can hoist (the specialised fast path of the common stage shape)
template <int CNT, int PSTRIDE4, int VSTRIDE>
__device__ __forceinline__ void mac_f4(float (&acc)[4][4], const float4* prow, const float* xv) {
#pragma unroll
    for (int i = 0; i < CNT; ++i) fma16(acc, prow[i * PSTRIDE4], *reinterpret_cast<const float4*>(xv + i * VSTRIDE));
}
// same with the operand gathered from 4 sample rows (natural-layout input buffer of the forward)
template <int CNT, int PSTRIDE4>
__device__ __forceinline__ void mac_s4(float (&acc)[4][4], const float4* prow, const float* u0, const float* u1, const float* u2, const float* u3) {
#pragma unroll
    for (int i = 0; i < CNT; ++i) fma16(acc, prow[i * PSTRIDE4], make_float4(u0[i], u1[i], u2[i], u3[i]));
}

// One stage step for the lanes of one warp:  out rows [4*rg, 4*rg+4) for rg in [rg_slot, nrg) step rgs.
//   state rows -> xn (next state), y rows -> yc (chunk output buffer, may be null: rows skipped)
__device__ __forceinline__ void stage_step(const sn_sss_stage& st, const float* __restrict__ packed, int RP,
                                           const float* xs, float* xn, const float* uc, float* yc,
                                           int stride, int ucol, int yrow, int nrg, int rg_slot, int rgs, int q) {
    const float4* Pt4 = reinterpret_cast<const float4*>(packed + st.pack_off + SSS_HDR);
    const int RP4 = RP >> 2;
    for (int rg = rg_slot; rg < nrg; rg += rgs) {
        float acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
        const float4* prow = Pt4 + rg;
        const float* xv = xs + 4 * q;
#pragma unroll 4
        for (int i = 0; i < st.d_in; ++i) {
            float4 p = __ldg(prow + (size_t)i * RP4);
            float4 v = *reinterpret_cast<const float4*>(xv + i * stride);
            fma16(acc, p, v);
        }
        prow += (size_t)st.d_in * RP4;
        const float* uv = uc + (size_t)ucol * stride + 4 * q;
#pragma unroll 4
        for (int i = 0; i < st.in_dim; ++i) {
            float4 p = __ldg(prow + (size_t)i * RP4);
            float4 v = *reinterpret_cast<const float4*>(uv + i * stride);
            fma16(acc, p, v);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int r = 4 * rg + j;
            float4 o = make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
            if (r < st.d_out) {
                *reinterpret_cast<float4*>(xn + r * stride + 4 * q) = o;
            } else if (yc != nullptr && r < st.d_out + st.out_dim) {
                *reinterpret_cast<float4*>(yc + (size_t)(yrow + r - st.d_out) * stride + 4 * q) = o;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// async-copy / mbarrier helpers (sm_90+ PTX; SASS: SYNCS.*, UBLKCP, LDGSTS)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}\n" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// producer-side wait: back off between probes so the spinning lane does not steal issue slots from the math warps
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) __nanosleep(200);
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared through the TMA engine, completion signalled on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src, bool valid) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst_smem)), "l"(src), "r"(valid ? 16 : 0) : "memory");
}
__device__ __forceinline__ void cp_async4(void* dst_smem, const void* src, bool valid) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_u32(dst_smem)), "l"(src), "r"(valid ? 4 : 0) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// ------------------------------------------------------------------------------------------
// forward
//   CTA = PAIRS (causal, anticausal) warp pairs; a warp owns NSW = 4*NQ samples of one direction and walks all
//   stages.  Per chunk of stages (<= 4):
//     - the chunk's packed parameter blocks (descriptor header + Pt) are fetched with cp.async.bulk (TMA) into a
//       double-buffered per-direction shared-memory area, one chunk ahead, completion on an mbarrier; the warps of
//       one direction meet at a named barrier per chunk, after which the leader lane refills the freed buffer;
//     - the input columns of the chunk are prefetched one chunk ahead with 16-byte cp.async into a natural
//       [sample][col] buffer whose row stride is 4*odd floats (the 4 scalar reads of a lane's interleaved samples
//       are bank-conflict free); out-of-range rows / columns are zero-filled by the copy itself;
//     - the state lives in a feature-major ping-pong buffer, exchanged between lanes with __syncwarp();
//     - y rows are collected per chunk and flushed with 32 B row segments; the second visitor of a stage adds to
//       what the first one stored (after a CTA-wide named barrier) -- deterministic, no atomics.
//   Sample <-> position map inside a warp: position p = 4*q + t holds local sample q + NQ*t (table in smem).
// ------------------------------------------------------------------------------------------
struct FwdSmem {
    int slot_floats;   // one stage: header + Pt
    int pbuf_off, bar_off, pos_off, warp_off, per_warp;   // float offsets
    int uw;            // row stride of the u buffers
    int xs, xn, ub0, ub1, yb;   // offsets inside a warp's region
    int total;
};

inline FwdSmem make_fwd_smem(const sn_sss_plan& p, const Geom& g, int pairs) {
    FwdSmem s;
    s.slot_floats = round_up(SSS_HDR + p.k_pad * p.rows_pad, 4);
    s.pbuf_off = 0;
    s.bar_off = s.pbuf_off + 2 * 2 * p.chunk_len_max * s.slot_floats;   // [dir][buf][stage]
    s.pos_off = s.bar_off + 2 * 4;                                       // 4 mbarriers
    s.warp_off = round_up(s.pos_off + g.nsw, 4);
    s.uw = pad_stride(p.chunk_in_max + 3);
    int o = 0;
    s.xs = o;  o += p.d_pad * g.nswp;
    s.xn = o;  o += p.d_pad * g.nswp;
    s.ub0 = o; o += g.nsw * s.uw;
    s.ub1 = o; o += g.nsw * s.uw;
    s.yb = o;  o += p.chunk_out_max * g.nswp;
    s.per_warp = round_up(o, 4);
    s.total = s.warp_off + 2 * pairs * s.per_warp;
    return s;
}

__device__ __forceinline__ int pos_of(int ls, int nq) { return 4 * (ls % nq) + ls / nq; }

// input columns [col0, col0+ncols) of the warp's samples -> ub[ls][uoff + (col - col0)]; returns uoff
__device__ __forceinline__ int issue_u_load(const float* __restrict__ x, long ldx, long s0, long B, int in_dim, int nsw, int uw,
                                            bool aligned, int col0, int ncols, float* ub, int lane) {
    if (aligned) {
        const int col0a = col0 & ~3;
        const int ngran = (col0 - col0a + ncols + 3) >> 2;
        const int gi0 = lane & 3;
        for (int ls = lane >> 2; ls < nsw; ls += 8) {
            const bool rok = s0 + ls < B;
            const float* row = x + (size_t)(s0 + ls) * ldx + col0a;
            float* drow = ub + ls * uw;
            for (int gi = gi0; gi < ngran; gi += 4) {
                const bool ok = rok && (col0a + 4 * gi < in_dim);
                cp_async16(drow + 4 * gi, ok ? (const void*)(row + 4 * gi) : (const void*)x, ok);
            }
        }
        return col0 - col0a;
    }
    for (int ls = 0; ls < nsw; ++ls) {
        const bool rok = s0 + ls < B;
        const float* row = x + (size_t)(s0 + ls) * ldx + col0;
        for (int c = lane; c < ncols; c += 32) cp_async4(ub + ls * uw + c, rok ? (const void*)(row + c) : (const void*)x, rok);
    }
    return 0;
}

// RP4T / NSWPT > 0: compile-time rows_pad/4 and state row stride of the specialised instantiation (the 4096->1000,
// statespace-16 shape: rows_pad 20, 6 sample quads per warp); 0: generic runtime strides.
template <int PAIRS, int RP4T, int NSWPT>
__global__ void __launch_bounds__(PAIRS * 64)
sss_fwd_kernel(sn_sss_plan plan, const float* __restrict__ packed, const float* __restrict__ x, long ldx,
               float* __restrict__ y, long ldy, const float* __restrict__ bias, float* __restrict__ ckpt, long B,
               Geom g, FwdSmem sm, int x_aligned) {
    extern __shared__ __align__(128) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = plan.nb_states, DP = plan.d_pad, RP = plan.rows_pad, CL = plan.chunk_len_max;
    float* pbuf = smem + sm.pbuf_off;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + sm.bar_off);   // full[dir][buf]
    int* pos_tab = reinterpret_cast<int*>(smem + sm.pos_off);
    constexpr bool FAST = RP4T > 0;
    const int nswp = FAST ? NSWPT : g.nswp, uw = sm.uw, nq = g.nq, nsw = g.nsw;

    if (threadIdx.x == 0) {
        for (int i = 0; i < 4; ++i) mbar_init(bars + i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    for (int ls = threadIdx.x; ls < nsw; ls += PAIRS * 64) pos_tab[ls] = pos_of(ls, nq);
    __syncthreads();

    const int pair = warp >> 1, dir = warp & 1;
    const bool leader = (pair == 0) && (lane == 0);
    const long s0 = ((long)blockIdx.x * PAIRS + pair) * nsw;
    float* wbase = smem + sm.warp_off + (size_t)warp * sm.per_warp;
    float* xs = wbase + sm.xs;
    float* xn = wbase + sm.xn;
    float* const ub_a = wbase + sm.ub0;
    float* const ub_b = wbase + sm.ub1;
    float* yb = wbase + sm.yb;
    const sn_sss_chunk* chunks = plan.chunks + (size_t)dir * plan.nchunks;
    const int rg_slot = lane / nq, q = lane - rg_slot * nq;
    const bool active = rg_slot < g.rgs;
    const int RP4 = FAST ? RP4T : (RP >> 2);
    const size_t blk = SSS_HDR + 2 * (size_t)plan.k_pad * RP;
    const uint32_t slot_bytes = (uint32_t)sm.slot_floats * 4u;

    auto issue_params = [&](int ch, const sn_sss_chunk& cc) {
        const int b = ch & 1, len = cc.kk_end - cc.kk_begin;
        uint64_t* fb = bars + dir * 2 + b;
        mbar_arrive_expect_tx(fb, slot_bytes * (uint32_t)len);
        for (int j = 0; j < len; ++j)
            bulk_g2s(pbuf + ((size_t)(dir * 2 + b) * CL + j) * sm.slot_floats, packed + ((size_t)dir * n + cc.kk_begin + j) * blk, slot_bytes, fb);
    };

    sn_sss_chunk c = chunks[0];
    if (leader) issue_params(0, c);
    int uoff_cur = issue_u_load(x, ldx, s0, B, plan.input_dim, nsw, uw, x_aligned != 0, c.col0, c.ncols, ub_a, lane);
    cp_async_commit();
    bool did_mid = false;
    int ubi = 0;

    for (int ch = 0; ch < plan.nchunks; ++ch) {
        if (c.second_visit && !did_mid) {
            named_bar_sync(1, PAIRS * 64);   // the other direction's first-visit stores to y are visible
            did_mid = true;
        }
        sn_sss_chunk cnext = c;
        if (ch + 1 < plan.nchunks) cnext = chunks[ch + 1];
        named_bar_sync(2 + dir, PAIRS * 32);   // every warp of this direction is done with chunk ch-1: its buffer is free
        int uoff_next = 0;
        if (ch + 1 < plan.nchunks) {
            if (leader) issue_params(ch + 1, cnext);
            uoff_next = issue_u_load(x, ldx, s0, B, plan.input_dim, nsw, uw, x_aligned != 0, cnext.col0, cnext.ncols, ubi ? ub_a : ub_b, lane);
        }
        cp_async_commit();
        cp_async_wait<1>();
        __syncwarp();
        mbar_wait(bars + dir * 2 + (ch & 1), (ch >> 1) & 1);
        const float* ub = ubi ? ub_b : ub_a;
        const float* cbuf = pbuf + (size_t)(dir * 2 + (ch & 1)) * CL * sm.slot_floats;
        // flush geometry: lanes = (row, sample-sub); the second visitor prefetches what the first one stored so the
        // read-modify-write at the end of the chunk does not wait on L2
        const int rl = c.nrows >= 32 ? 32 : (c.nrows >= 16 ? 16 : (c.nrows >= 8 ? 8 : (c.nrows >= 4 ? 4 : (c.nrows >= 2 ? 2 : 1))));
        const int spl = 32 / rl;
        const int lrow = lane & (rl - 1), lsub = lane / rl;
        float yold[8];
        const bool prefetched = c.second_visit && c.nrows <= rl && nsw <= 8 * spl;
        if (prefetched) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int ls = lsub + k * spl;
                yold[k] = (lrow < c.nrows && ls < nsw && s0 + ls < B) ? __ldcg(y + (size_t)(s0 + ls) * ldy + c.row0 + lrow) : 0.f;
            }
        }

        if (ckpt != nullptr) {   // checkpoint of the state entering the chunk, in true sample order
            const int d_first = reinterpret_cast<const int*>(cbuf)[4];
            float* cbase = ckpt + ((size_t)(dir * plan.nchunks + ch) * DP) * B + s0;
            for (int ls = lane; ls < nsw; ls += 32) {
                if (s0 + ls < B) {
                    const float* src = xs + pos_tab[ls];
                    float* dst = cbase + ls;
                    for (int f = 0; f < d_first; ++f) dst[(size_t)f * B] = src[f * nswp];
                }
            }
        }
        for (int kk = c.kk_begin; kk < c.kk_end; ++kk) {
            const float* slot = cbuf + (size_t)(kk - c.kk_begin) * sm.slot_floats;
            const int* hdr = reinterpret_cast<const int*>(slot);
            const int in_off = hdr[0], in_dim = hdr[1], out_off = hdr[2], out_dim = hdr[3], d_in = hdr[4], d_out = hdr[5];
            if (active) {
                const int nrg = (d_out + out_dim + 3) >> 2;
                const float4* Pt4 = reinterpret_cast<const float4*>(slot + SSS_HDR);
                const float* u0 = ub + q * uw + uoff_cur + (in_off - c.col0);
                const float* u1 = u0 + nq * uw;
                const float* u2 = u1 + nq * uw;
                const float* u3 = u2 + nq * uw;
                for (int rg = rg_slot; rg < nrg; rg += g.rgs) {
                    float acc[4][4];
#pragma unroll
                    for (int a = 0; a < 4; ++a)
#pragma unroll
                        for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
                    const float4* prow = Pt4 + rg;
                    const float* xv = xs + 4 * q;
                    if (FAST && d_in == 16) {
                        mac_f4<16, RP4T, NSWPT>(acc, prow, xv);
                        prow += 16 * RP4T;
                    } else {
#pragma unroll 4
                        for (int i = 0; i < d_in; ++i) {
                            const float4 p = prow[0];
                            const float4 v = *reinterpret_cast<const float4*>(xv);
                            prow += RP4;
                            xv += nswp;
                            fma16(acc, p, v);
                        }
                    }
                    if (FAST && in_dim == 8) {
                        mac_s4<8, RP4T>(acc, prow, u0, u1, u2, u3);
                    } else if (FAST && in_dim == 9) {
                        mac_s4<9, RP4T>(acc, prow, u0, u1, u2, u3);
                    } else {
#pragma unroll 4
                        for (int i = 0; i < in_dim; ++i) {
                            const float4 p = prow[0];
                            prow += RP4;
                            const float4 v = make_float4(u0[i], u1[i], u2[i], u3[i]);
                            fma16(acc, p, v);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int r = 4 * rg + j;
                        const float4 o = make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
                        if (r < d_out) *reinterpret_cast<float4*>(xn + r * nswp + 4 * q) = o;
                        else if (r < d_out + out_dim) *reinterpret_cast<float4*>(yb + (out_off - c.row0 + r - d_out) * nswp + 4 * q) = o;
                    }
                }
            }
            __syncwarp();
            float* t = xs; xs = xn; xn = t;
        }
        // flush the chunk's outputs: y[s0 + ls][row0 + row]; lanes = (row, sample-sub), 4 independent samples in flight
        if (prefetched) {
            if (lrow < c.nrows) {
                const float* ysrc = yb + lrow * nswp;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int ls = lsub + k * spl;
                    if (ls < nsw && s0 + ls < B) y[(size_t)(s0 + ls) * ldy + c.row0 + lrow] = ysrc[pos_tab[ls]] + yold[k];
                }
            }
        } else {
            for (int row = lrow; row < c.nrows; row += rl) {
                const float bv = (!c.second_visit && bias != nullptr) ? __ldg(bias + c.row0 + row) : 0.f;
                const float* ysrc = yb + row * nswp;
                for (int lsb = lsub; lsb < nsw; lsb += 4 * spl) {
                    float v[4];
                    float* dst[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int ls = lsb + k * spl;
                        const bool ok = ls < nsw && s0 + ls < B;
                        dst[k] = ok ? y + (size_t)(s0 + ls) * ldy + c.row0 + row : nullptr;
                        v[k] = ok ? ysrc[pos_tab[ls]] : 0.f;
                    }
                    if (c.second_visit) {
                        float o[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) o[k] = dst[k] ? __ldcg(dst[k]) : 0.f;
#pragma unroll
                        for (int k = 0; k < 4; ++k) v[k] += o[k];
                    } else {
#pragma unroll
                        for (int k = 0; k < 4; ++k) v[k] += bv;
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (dst[k]) *dst[k] = v[k];
                }
            }
        }
        __syncwarp();
        if (ch + 1 < plan.nchunks) { ubi ^= 1; uoff_cur = uoff_next; }
        c = cnext;
    }
    cp_async_wait<0>();
    if (!did_mid) named_bar_sync(1, PAIRS * 64);
}

// ------------------------------------------------------------------------------------------
// backward: CTA = BWD_CONS warps (each owning NSW samples), one direction per CTA (blockIdx.y); chunks are visited
// in reverse processing order.  Per chunk:
//   loads   : forward checkpoint, input columns and grad_y rows of the chunk, transposed to feature-major
//             [feature][position] with 4-byte cp.async, double buffered (issued one chunk ahead); the chunk's packed
//             parameter blocks (descriptor + Pt + P) arrive as ONE cp.async.bulk (TMA), issued as soon as the previous
//             chunk's adjoint sweep has released the parameter buffer, i.e. it lands during the gradient phase
//   1. recompute the entry states of the chunk's stages                         (warp-own samples)
//   2. adjoint sweep  lam_in = P^T [lam_out ; gy]                               (warp-own samples)
//   2b. (grad_x only) input gradients  grad_u = the in_dim input columns of P^T [lam_out ; gy]  (own samples, all
//      lanes), staged per stage in a per-warp [column][position] buffer and added to grad_x with coalesced
//      red.global.add: each direction adds its share exactly once onto the zeroed grad_x, so the sum of the two
//      addends is bitwise reproducible.  Runs before the parameter buffer is handed back to the bulk copy.
//   3. parameter gradients  dP_k = [lam_out ; gy] [s_in ; u]^T over the tile's samples (warp-own stages,
//      4x4 register tiles over interleaved rows/cols), atomically accumulated into a packed [r][k_pad]
//      gradient workspace that sss_unpack_grad_kernel folds into the flat gradient buffer afterwards.
//      Skipped when only grad_x is requested (gpacked == NULL).
// ------------------------------------------------------------------------------------------
constexpr int BWD_CONS = 2;
constexpr int BWD_THREADS = BWD_CONS * 32;

struct BwdSmem {
    int nsp;     // padded position stride of the CTA-wide feature-major buffers
    int blk;     // floats per packed stage block
    int hs;      // one history entry (d_pad * nsp)
    int gxs;     // position stride of the grad_u staging buffer (0: no grad_x)
    int params, bars, pos, xh, lh, lcar0, lcar1, ck0, ck1, ut0, ut1, gt0, gt1, zero, gx, total;   // float offsets
};

// with_gx: add the per-warp grad_u staging buffer (one stage's input columns; every stage lies in one half chunk, so half_in_max
// bounds its in_dim).  Without it the layout is exactly that of a parameter-gradient-only backward.
inline BwdSmem make_bwd_smem(const sn_sss_plan& p, const Geom& g, bool with_gx) {
    BwdSmem s;
    const int ns = BWD_CONS * g.nsw;
    s.nsp = pad_stride(ns);
    s.blk = SSS_HDR + 2 * p.k_pad * p.rows_pad;
    s.hs = p.d_pad * s.nsp;
    const int hist = p.chunk_len_max > 1 ? p.chunk_len_max - 1 : 1;
    int o = 0;
    s.params = o; o += round_up(p.chunk_len_max * s.blk, 4);
    s.bars = o;   o += 4;
    s.pos = o;    o += round_up(g.nsw, 4);
    s.xh = o;     o += hist * s.hs;
    s.lh = o;     o += hist * s.hs;
    s.lcar0 = o;  o += s.hs;
    s.lcar1 = o;  o += s.hs;
    s.ck0 = o;    o += s.hs;
    s.ck1 = o;    o += s.hs;
    s.ut0 = o;    o += p.chunk_in_max * s.nsp;
    s.ut1 = o;    o += p.chunk_in_max * s.nsp;
    s.gt0 = o;    o += p.chunk_out_max * s.nsp;
    s.gt1 = o;    o += p.chunk_out_max * s.nsp;
    s.zero = o;   o += s.nsp;
    s.gxs = with_gx ? pad_stride(g.nsw) : 0;
    s.gx = o;     o += with_gx ? BWD_CONS * p.half_in_max * s.gxs : 0;
    s.total = o;
    return s;
}

// issue the (transposing) loads of one chunk for the calling warp's samples: dst[feature][w0 + ls] (the backward keeps
// samples in their natural order: position = local sample)
//   checkpoint [feature][B]   : 16-byte cp.async along the samples when aligned, else 4-byte
//   x / grad_y [sample][feat] : 4-byte cp.async, lanes along the (contiguous) feature index, pointer increments per sample
__device__ __forceinline__ void bwd_issue_loads(const sn_sss_plan& plan, const sn_sss_chunk& c, int d_first, int dir, int ch,
                                                const float* __restrict__ x, long ldx, const float* __restrict__ gy, long ldgy,
                                                const float* __restrict__ ckpt, long B, long samp0, int nvalid, int nsw, int nsp,
                                                float* ck, float* ut, float* gt, int lane) {
    const float* cbase = ckpt + ((size_t)(dir * plan.nchunks + ch) * plan.d_pad) * B + samp0;
    if (((B | samp0) & 3) == 0 && (nsw & 3) == 0) {
        const int nq4 = nsw >> 2;
        for (int e = lane; e < d_first * nq4; e += 32) {
            const int f = e / nq4, q4 = e - f * nq4;
            const bool ok = 4 * q4 + 3 < nvalid;
            if (ok || 4 * q4 >= nvalid) {
                cp_async16(ck + f * nsp + 4 * q4, ok ? (const void*)(cbase + (size_t)f * B + 4 * q4) : (const void*)x, ok);
            } else {
                for (int t = 0; t < 4; ++t) cp_async4(ck + f * nsp + 4 * q4 + t, (4 * q4 + t < nvalid) ? (const void*)(cbase + (size_t)f * B + 4 * q4 + t) : (const void*)x, 4 * q4 + t < nvalid);
            }
        }
    } else {
        for (int ls = lane; ls < nsw; ls += 32) {
            const bool ok = ls < nvalid;
            for (int f = 0; f < d_first; ++f) cp_async4(ck + f * nsp + ls, ok ? (const void*)(cbase + (size_t)f * B + ls) : (const void*)x, ok);
        }
    }
    for (int cc = lane; cc < c.ncols; cc += 32) {
        float* dcol = ut + cc * nsp;
        const float* src = x + (size_t)samp0 * ldx + c.col0 + cc;
        for (int ls = 0; ls < nsw; ++ls, src += ldx) cp_async4(dcol + ls, ls < nvalid ? (const void*)src : (const void*)x, ls < nvalid);
    }
    for (int rr = lane; rr < c.nrows; rr += 32) {
        float* dcol = gt + rr * nsp;
        const float* src = gy + (size_t)samp0 * ldgy + c.row0 + rr;
        for (int ls = 0; ls < nsw; ++ls, src += ldgy) cp_async4(dcol + ls, ls < nvalid ? (const void*)src : (const void*)x, ls < nvalid);
    }
}

// RP4T / KP4T / NSPT > 0: compile-time strides of the specialised instantiation (rows_pad 20, k_pad 28, 48 positions
// per tile padded to 52); 0: generic runtime strides.
template <int RP4T, int KP4T, int NSPT>
__global__ void __launch_bounds__(BWD_THREADS)
sss_bwd_kernel(sn_sss_plan plan, const float* __restrict__ packed, const float* __restrict__ x, long ldx,
               const float* __restrict__ gy, long ldgy, const float* __restrict__ ckpt,
               float* __restrict__ gpacked, float* __restrict__ gbias, float* __restrict__ gx, long ldgx, long B, Geom g, BwdSmem sm) {
    extern __shared__ __align__(128) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int dir = blockIdx.y;
    const int n = plan.nb_states, DP = plan.d_pad, RP = plan.rows_pad, KP = plan.k_pad;
    constexpr bool FAST = RP4T > 0;
    const int NS = BWD_CONS * g.nsw, NSP = FAST ? NSPT : sm.nsp, hs = sm.hs;
    const sn_sss_chunk* chunks = plan.chunks + (size_t)dir * plan.nchunks;
    const sn_sss_stage* stages = plan.stages + (size_t)dir * n;
    float* params = smem + sm.params;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + sm.bars);
    const int nq = g.nq, nsw = g.nsw;

    sn_sss_chunk c = chunks[plan.nchunks - 1];
    if (threadIdx.x == 0) {
        mbar_init(full_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        const uint32_t bytes = (uint32_t)((c.kk_end - c.kk_begin) * sm.blk) * 4u;
        mbar_arrive_expect_tx(full_bar, bytes);
        bulk_g2s(params, packed + ((size_t)dir * n + c.kk_begin) * sm.blk, bytes, full_bar);
    }
    for (int e = threadIdx.x; e < NSP; e += BWD_THREADS) smem[sm.zero + e] = 0.f;
    for (int e = threadIdx.x; e < 2 * hs; e += BWD_THREADS) smem[sm.lcar0 + e] = 0.f;   // lcar0 and lcar1 are adjacent
    __syncthreads();

    const long t0 = (long)blockIdx.x * NS;
    const int w0 = warp * nsw;
    const long samp0 = t0 + w0;
    const int nvalid = (int)(B - samp0 < 0 ? 0 : (B - samp0 > nsw ? nsw : B - samp0));
    const int rg_slot = lane / nq, q = lane - rg_slot * nq;
    const int rgs_state = (DP / 4 < g.rgs) ? DP / 4 : g.rgs;
    const int RP4 = FAST ? RP4T : (RP >> 2), KP4 = FAST ? KP4T : (KP >> 2);
    float* xh = smem + sm.xh;
    float* lh = smem + sm.lh;
    float* lcar_cur = smem + sm.lcar0;
    float* lcar_nxt = smem + sm.lcar1;
    const float* zr = smem + sm.zero;
    int buf = 0;

    int d_first = stages[c.kk_begin].d_in;
    bwd_issue_loads(plan, c, d_first, dir, plan.nchunks - 1, x, ldx, gy, ldgy, ckpt, B, samp0, nvalid, nsw, NSP, smem + sm.ck0 + w0,
                    smem + sm.ut0 + w0, smem + sm.gt0 + w0, lane);
    cp_async_commit();

    int it = 0;
    for (int ch = plan.nchunks - 1; ch >= 0; --ch, ++it) {
        const int len = c.kk_end - c.kk_begin;
        float* ck = smem + (buf ? sm.ck1 : sm.ck0);
        float* ut = smem + (buf ? sm.ut1 : sm.ut0);
        float* gt = smem + (buf ? sm.gt1 : sm.gt0);
        sn_sss_chunk cn = c;
        if (ch > 0) {
            cn = chunks[ch - 1];
            const int d_first_n = stages[cn.kk_begin].d_in;
            bwd_issue_loads(plan, cn, d_first_n, dir, ch - 1, x, ldx, gy, ldgy, ckpt, B, samp0, nvalid, nsw, NSP,
                            smem + (buf ? sm.ck0 : sm.ck1) + w0, smem + (buf ? sm.ut0 : sm.ut1) + w0, smem + (buf ? sm.gt0 : sm.gt1) + w0, lane);
        }
        cp_async_commit();
        cp_async_wait<1>();
        __syncwarp();
        mbar_wait(full_bar, it & 1);

        // ---- 1. recompute entry states of stages 1..len-1 (own samples) -------------------------
        for (int j = 0; j + 1 < len; ++j) {
            const float* slot = params + (size_t)j * sm.blk;
            const int* hdr = reinterpret_cast<const int*>(slot);
            const int in_off = hdr[0], in_dim = hdr[1], d_in = hdr[4], d_out = hdr[5];
            const float* xin = (j == 0 ? ck : xh + (size_t)(j - 1) * hs) + w0 + 4 * q;
            float* xout = xh + (size_t)j * hs + w0 + 4 * q;
            const float* uv0 = ut + (size_t)(in_off - c.col0) * NSP + w0 + 4 * q;
            if (rg_slot < rgs_state) {
                const int nrg = (d_out + 3) >> 2;
                for (int rg = rg_slot; rg < nrg; rg += rgs_state) {
                    float acc[4][4];
#pragma unroll
                    for (int a = 0; a < 4; ++a)
#pragma unroll
                        for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
                    const float4* prow = reinterpret_cast<const float4*>(slot + SSS_HDR) + rg;
                    const float* xv = xin;
                    if (FAST && d_in == 16) {
                        mac_f4<16, RP4T, NSPT>(acc, prow, xv);
                        prow += 16 * RP4T;
                    } else {
#pragma unroll 4
                        for (int i = 0; i < d_in; ++i) {
                            const float4 p = prow[0];
                            const float4 v = *reinterpret_cast<const float4*>(xv);
                            prow += RP4; xv += NSP;
                            fma16(acc, p, v);
                        }
                    }
                    const float* uv = uv0;
                    if (FAST && in_dim == 8) {
                        mac_f4<8, RP4T, NSPT>(acc, prow, uv);
                    } else if (FAST && in_dim == 9) {
                        mac_f4<9, RP4T, NSPT>(acc, prow, uv);
                    } else {
#pragma unroll 4
                        for (int i = 0; i < in_dim; ++i) {
                            const float4 p = prow[0];
                            const float4 v = *reinterpret_cast<const float4*>(uv);
                            prow += RP4; uv += NSP;
                            fma16(acc, p, v);
                        }
                    }
#pragma unroll
                    for (int a = 0; a < 4; ++a) {
                        const int r = 4 * rg + a;
                        if (r < d_out) *reinterpret_cast<float4*>(xout + r * NSP) = make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
                    }
                }
            }
            __syncwarp();
        }
        // ---- 2. adjoint sweep (own samples) -----------------------------------------------------
        for (int j = len - 1; j >= 0; --j) {
            const float* slot = params + (size_t)j * sm.blk;
            const int* hdr = reinterpret_cast<const int*>(slot);
            const int out_off = hdr[2], out_dim = hdr[3], d_in = hdr[4], d_out = hdr[5];
            const float4* P4 = reinterpret_cast<const float4*>(slot + SSS_HDR + KP * RP);
            const float* lout = (j == len - 1 ? lcar_cur : lh + (size_t)j * hs) + w0 + 4 * q;
            const float* gyj = gt + (size_t)(out_off - c.row0) * NSP + w0 + 4 * q;
            float* lin = (j == 0 ? lcar_nxt : lh + (size_t)(j - 1) * hs) + w0 + 4 * q;
            if (rg_slot < rgs_state) {
                const int nig = (d_in + 3) >> 2;
                for (int ig = rg_slot; ig < nig; ig += rgs_state) {
                    float acc[4][4];
#pragma unroll
                    for (int a = 0; a < 4; ++a)
#pragma unroll
                        for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
                    const float4* prow = P4 + ig;
                    const float* lv = lout;
                    if (FAST && d_out == 16) {
                        mac_f4<16, KP4T, NSPT>(acc, prow, lv);
                        prow += 16 * KP4T;
                    } else {
#pragma unroll 4
                        for (int r = 0; r < d_out; ++r) {
                            const float4 p = prow[0];
                            const float4 v = *reinterpret_cast<const float4*>(lv);
                            prow += KP4; lv += NSP;
                            fma16(acc, p, v);
                        }
                    }
                    const float* gv = gyj;
                    if (FAST && out_dim == 2) {
                        mac_f4<2, KP4T, NSPT>(acc, prow, gv);
                    } else {
                        for (int r = 0; r < out_dim; ++r) {
                            const float4 p = prow[0];
                            const float4 v = *reinterpret_cast<const float4*>(gv);
                            prow += KP4; gv += NSP;
                            fma16(acc, p, v);
                        }
                    }
#pragma unroll
                    for (int a = 0; a < 4; ++a) {
                        const int i = 4 * ig + a;
                        if (i < d_in) *reinterpret_cast<float4*>(lin + i * NSP) = make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
                    }
                }
            }
            __syncwarp();
        }
        // ---- 2b. input gradients (own samples, all lanes; off the recurrence) ---------------------
        if (gx != nullptr) {
            float* gxb = smem + sm.gx + (size_t)warp * plan.half_in_max * sm.gxs;
            for (int j = 0; j < len; ++j) {
                const float* slot = params + (size_t)j * sm.blk;
                const int* hdr = reinterpret_cast<const int*>(slot);
                const int in_off = hdr[0], in_dim = hdr[1], out_off = hdr[2], out_dim = hdr[3], d_in = hdr[4], d_out = hdr[5];
                const float4* P4 = reinterpret_cast<const float4*>(slot + SSS_HDR + KP * RP);
                const float* lout = (j == len - 1 ? lcar_cur : lh + (size_t)j * hs) + w0;
                const float* gyj = gt + (size_t)(out_off - c.row0) * NSP + w0;
                // aligned 4-column groups covering the input columns [d_in, d_in + in_dim) of P
                const int cg0 = d_in >> 2, ncg = ((d_in + in_dim + 3) >> 2) - cg0;
                for (int t = lane; t < ncg * nq; t += 32) {
                    const int cg = cg0 + t / nq, qq = t % nq;
                    float acc[4][4];
#pragma unroll
                    for (int a = 0; a < 4; ++a)
#pragma unroll
                        for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
                    const float4* prow = P4 + cg;
                    const float* lv = lout + 4 * qq;
#pragma unroll 4
                    for (int r = 0; r < d_out; ++r) {
                        const float4 p = prow[0];
                        const float4 v = *reinterpret_cast<const float4*>(lv);
                        prow += KP4; lv += NSP;
                        fma16(acc, p, v);
                    }
                    const float* gv = gyj + 4 * qq;
                    for (int r = 0; r < out_dim; ++r) {
                        const float4 p = prow[0];
                        const float4 v = *reinterpret_cast<const float4*>(gv);
                        prow += KP4; gv += NSP;
                        fma16(acc, p, v);
                    }
#pragma unroll
                    for (int a = 0; a < 4; ++a) {
                        const int cc = 4 * cg + a - d_in;
                        if (cc >= 0 && cc < in_dim)
                            *reinterpret_cast<float4*>(gxb + cc * sm.gxs + 4 * qq) = make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
                    }
                }
                __syncwarp();
                // lanes along the stage's contiguous columns of consecutive samples
                for (int e = lane; e < nvalid * in_dim; e += 32) {
                    const int ls = e / in_dim, cc = e - ls * in_dim;
                    atomicAdd(gx + (size_t)(samp0 + ls) * ldgx + in_off + cc, gxb[cc * sm.gxs + ls]);
                }
                __syncwarp();
            }
        }
        // stage descriptors needed by the gradient phase are copied out before the parameter buffer is released
        int h_in_off[2], h_in_dim[2], h_out_off[2], h_out_dim[2], h_d_in[2], h_d_out[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int j = warp + u * BWD_CONS;
            if (j < len) {
                const int* hdr = reinterpret_cast<const int*>(params + (size_t)j * sm.blk);
                h_in_off[u] = hdr[0]; h_in_dim[u] = hdr[1]; h_out_off[u] = hdr[2]; h_out_dim[u] = hdr[3]; h_d_in[u] = hdr[4]; h_d_out[u] = hdr[5];
            }
        }
        // The header words above are ld.shared results that nothing has consumed yet: a barrier does not wait for loads in flight,
        // and the bulk copy issued right after it overwrites the very words they read (seen as an intermittent, large gradient error:
        // a stage's block accumulated with the NEXT chunk's dimensions).  Consume them before arriving.
        {
            int chk = 0;
#pragma unroll
            for (int u = 0; u < 2; ++u)
                if (warp + u * BWD_CONS < len) chk ^= h_in_off[u] ^ h_in_dim[u] ^ h_out_off[u] ^ h_out_dim[u] ^ h_d_in[u] ^ h_d_out[u];
            asm volatile("{\n.reg .pred p;\nsetp.eq.s32 p, %0, 0x7fffffff;\n@p trap;\n}" ::"r"(chk) : "memory");
        }
        named_bar_sync(1, BWD_THREADS);      // every warp is done with the parameter buffer and its history columns are complete
        if (threadIdx.x == 0 && ch > 0) {    // refill the parameter buffer for the next chunk; lands during the gradient phase
            const uint32_t bytes = (uint32_t)((cn.kk_end - cn.kk_begin) * sm.blk) * 4u;
            mbar_arrive_expect_tx(full_bar, bytes);
            bulk_g2s(params, packed + ((size_t)dir * n + cn.kk_begin) * sm.blk, bytes, full_bar);
        }
        // ---- 3. parameter gradients (own stages, all positions of the tile) -----------------------
        if (gbias != nullptr && dir == 0) {
            for (int rr = threadIdx.x; rr < c.nrows; rr += BWD_THREADS) {
                float sacc = 0.f;
                const float* gr = gt + (size_t)rr * NSP;
                for (int e = 0; e < NS; ++e) sacc += gr[e];
                atomicAdd(gbias + c.row0 + rr, sacc);
            }
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {            // chunk_len_max <= 2*BWD_CONS is checked on the host
            const int j = warp + u * BWD_CONS;
            if (j >= len || gpacked == nullptr) break;
            const int in_off = h_in_off[u], in_dim = h_in_dim[u], out_off = h_out_off[u], out_dim = h_out_dim[u], d_in = h_d_in[u], d_out = h_d_out[u];
            const int rows = d_out + out_dim, K = d_in + in_dim;
            const int rgn = (rows + 3) >> 2, cgn = (K + 3) >> 2;
            const float* lout = (j == len - 1 ? lcar_cur : lh + (size_t)j * hs);
            const float* gyj = gt + (size_t)(out_off - c.row0) * NSP;
            const float* xin = (j == 0 ? ck : xh + (size_t)(j - 1) * hs);
            const float* uj = ut + (size_t)(in_off - c.col0) * NSP;
            float* gblk = gpacked + ((size_t)dir * n + c.kk_begin + j) * ((size_t)RP * KP);
            for (int t = lane; t < rgn * cgn; t += 32) {
                const int rg = t / cgn, cg = t - rg * cgn;
                const float* gp[4];
                const float* ip[4];
                int rr[4], ii[4];
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    const int r = rg + a * rgn;
                    rr[a] = r;
                    gp[a] = (r < d_out) ? (lout + r * NSP) : (r < rows ? gyj + (r - d_out) * NSP : zr);
                    const int i = cg + a * cgn;
                    ii[a] = i;
                    ip[a] = (i < d_in) ? (xin + i * NSP) : (i < K ? uj + (i - d_in) * NSP : zr);
                }
                float acc[4][4];
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
                auto body = [&](int sq) {
                    float4 gv[4], iv[4];
#pragma unroll
                    for (int a = 0; a < 4; ++a) {
                        gv[a] = *reinterpret_cast<const float4*>(gp[a] + sq);
                        iv[a] = *reinterpret_cast<const float4*>(ip[a] + sq);
                    }
#pragma unroll
                    for (int a = 0; a < 4; ++a)
#pragma unroll
                        for (int b = 0; b < 4; ++b) {
                            acc[a][b] = fmaf(gv[a].x, iv[b].x, acc[a][b]);
                            acc[a][b] = fmaf(gv[a].y, iv[b].y, acc[a][b]);
                            acc[a][b] = fmaf(gv[a].z, iv[b].z, acc[a][b]);
                            acc[a][b] = fmaf(gv[a].w, iv[b].w, acc[a][b]);
                        }
                };
                if (FAST) {
#pragma unroll 4
                    for (int sq = 0; sq < 48; sq += 4) body(sq);
                } else {
#pragma unroll 2
                    for (int sq = 0; sq < NS; sq += 4) body(sq);
                }
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    if (rr[a] >= rows) continue;
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        if (ii[b] >= K) continue;
                        atomicAdd(gblk + (size_t)rr[a] * KP + ii[b], acc[a][b]);
                    }
                }
            }
        }
        named_bar_sync(1, BWD_THREADS);
        { float* tsw = lcar_cur; lcar_cur = lcar_nxt; lcar_nxt = tsw; }
        buf ^= 1;
        c = cn;
    }
    cp_async_wait<0>();
}

// flat gradient += packed gradient (one block per (direction, stage); every parameter entry has exactly one
// packed entry, so no atomics)
__global__ void sss_unpack_grad_kernel(const sn_sss_stage* __restrict__ stages, int total_stages, int RP, int KP,
                                       const float* __restrict__ gpacked, float* __restrict__ gflat) {
    const int sidx = blockIdx.x;
    if (sidx >= total_stages) return;
    const sn_sss_stage st = stages[sidx];
    const int K = st.d_in + st.in_dim, rows = st.d_out + st.out_dim;
    const float* G = gpacked + (size_t)sidx * RP * KP;
    for (int e = threadIdx.x; e < rows * K; e += blockDim.x) {
        const int r = e / K, i = e - r * K;
        int off;
        if (r < st.d_out) {
            off = (i < st.d_in) ? st.off_ss + r * st.d_in + i : st.off_su + r * st.in_dim + (i - st.d_in);
        } else {
            const int ry = r - st.d_out;
            if (i < st.d_in) off = st.off_ys + ry * st.d_in + i;
            else if (st.off_yu >= 0) off = st.off_yu + ry * st.in_dim + (i - st.d_in);
            else continue;
        }
        gflat[off] += G[(size_t)r * KP + i];
    }
}

int check_plan(const sn_sss_plan* p) {
    SN_CHECK_ARG(p != nullptr, "sss: plan is NULL");
    SN_CHECK_ARG(p->nb_states > 0 && p->input_dim > 0 && p->output_dim > 0, "sss: bad plan dims");
    SN_CHECK_ARG(p->rows_pad > 0 && p->rows_pad % 4 == 0 && p->k_pad > 0 && p->k_pad % 4 == 0 && p->d_pad % 4 == 0 && p->d_pad > 0,
                 "sss: rows_pad/k_pad/d_pad must be positive multiples of 4");
    SN_CHECK_ARG(p->stages != nullptr && p->chunks != nullptr && p->nchunks > 0, "sss: plan tables missing");
    return 0;
}

template <int PAIRS, int RP4T, int NSWPT>
static int launch_fwd(const sn_sss_plan* p, const Geom& g, const float* packed, const float* x, int64_t ldx, float* y, int64_t ldy,
                      const float* bias, float* ckpt, int64_t B, int aligned, cudaStream_t st) {
    FwdSmem sm = make_fwd_smem(*p, g, PAIRS);
    size_t smem = (size_t)sm.total * sizeof(float);
    SN_CHECK_ARG(smem <= 227 * 1024, "sss_forward: stage dims need %zu bytes of shared memory (> 227 KB)", smem);
    static size_t configured = 0;
    if (smem > configured) {
        SN_SET_MAX_SMEM((int)smem, sss_fwd_kernel<PAIRS, RP4T, NSWPT>);
        configured = smem;
    }
    long tile = (long)PAIRS * g.nsw;
    unsigned grid = (unsigned)((B + tile - 1) / tile);
    SN_LAUNCH("sss_fwd_kernel", st, sss_fwd_kernel<PAIRS, RP4T, NSWPT><<<grid, PAIRS * 64, smem, st>>>(*p, packed, x, (long)ldx, y, (long)ldy, bias, ckpt, (long)B, g, sm, aligned));
    return 0;
}

}  // namespace

extern "C" {

size_t sn_sss_packed_floats(const sn_sss_plan* p) {
    if (p == nullptr) return 0;
    return (size_t)2 * p->nb_states * (SSS_HDR + 2 * (size_t)p->k_pad * p->rows_pad);
}

size_t sn_sss_ckpt_floats(const sn_sss_plan* p, int64_t B) {
    if (p == nullptr || B <= 0) return 0;
    return (size_t)2 * p->nchunks * p->d_pad * (size_t)B;
}

int sn_sss_pack(const sn_sss_plan* p, const float* params, float* packed, sn_stream_t stream) {
    if (int rc = check_plan(p)) return rc;
    SN_CHECK_ARG(params != nullptr && packed != nullptr, "sss_pack: NULL buffer");
    sss_pack_kernel<<<2 * p->nb_states, 128, 0, snb::as_stream(stream)>>>(p->stages, 2 * p->nb_states, p->rows_pad,
                                                                           p->k_pad, params, packed);
    SN_CHECK_LAUNCH("sss_pack_kernel");
    return 0;
}

int sn_sss_forward(const sn_sss_plan* p, const float* packed, const float* x, int64_t ldx, float* y, int64_t ldy,
                   const float* bias, float* ckpt, int64_t B, sn_stream_t stream) {
    if (int rc = check_plan(p)) return rc;
    SN_CHECK_ARG(packed, "sss_forward: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && y, "sss_forward: NULL buffer");
    SN_CHECK_ARG(ldx >= p->input_dim && ldy >= p->output_dim, "sss_forward: leading dimension too small");
    Geom g = make_geom(p->rows_pad);
    // 16-byte cp.async path needs 16-byte aligned rows whose length is a multiple of 4 floats
    const int aligned = ((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (ldx & 3) == 0 && (p->input_dim & 3) == 0) ? 1 : 0;
    cudaStream_t st = snb::as_stream(stream);
    // big CTAs (6 warp pairs share one parameter stream) once they still fill the chip twice over; small ones otherwise
    const long big_tiles = (B + 6L * g.nsw - 1) / (6L * g.nsw);
    const bool big = big_tiles >= 2 * 148 && (size_t)make_fwd_smem(*p, g, 6).total * sizeof(float) <= 227 * 1024;
    const bool fast = p->rows_pad == 20 && g.nswp == 28;   // specialised instantiation (compile-time strides)
    if (fast) return big ? launch_fwd<6, 5, 28>(p, g, packed, x, ldx, y, ldy, bias, ckpt, B, aligned, st)
                         : launch_fwd<2, 5, 28>(p, g, packed, x, ldx, y, ldy, bias, ckpt, B, aligned, st);
    return big ? launch_fwd<6, 0, 0>(p, g, packed, x, ldx, y, ldy, bias, ckpt, B, aligned, st)
               : launch_fwd<2, 0, 0>(p, g, packed, x, ldx, y, ldy, bias, ckpt, B, aligned, st);
}

size_t sn_sss_backward_workspace_floats(const sn_sss_plan* p) {
    if (p == nullptr) return 0;
    return (size_t)2 * p->nb_states * p->rows_pad * p->k_pad;
}

int sn_sss_backward(const sn_sss_plan* p, const float* packed, const float* x, int64_t ldx, const float* grad_y,
                    int64_t ldgy, const float* ckpt, float* workspace, float* grad_params, float* grad_bias, float* grad_x,
                    int64_t ldgx, int64_t B, sn_stream_t stream) {
    if (int rc = check_plan(p)) return rc;
    SN_CHECK_ARG(packed, "sss_backward: NULL buffer");
    SN_CHECK_ARG(grad_params == nullptr || workspace != nullptr, "sss_backward: NULL workspace");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && grad_y && ckpt, "sss_backward: NULL buffer");
    SN_CHECK_ARG(grad_params != nullptr || grad_x != nullptr, "sss_backward: grad_params and grad_x are both NULL (nothing to compute)");
    SN_CHECK_ARG(ldx >= p->input_dim && ldgy >= p->output_dim, "sss_backward: leading dimension too small");
    SN_CHECK_ARG(grad_x == nullptr || ldgx >= p->input_dim, "sss_backward: grad_x leading dimension too small");
    cudaStream_t st = snb::as_stream(stream);
    Geom g = make_geom(p->rows_pad);
    BwdSmem sm = make_bwd_smem(*p, g, grad_x != nullptr);
    size_t smem = (size_t)sm.total * sizeof(float);
    SN_CHECK_ARG(smem <= 227 * 1024, "sss_backward: stage dims need %zu bytes of shared memory (> 227 KB)", smem);
    SN_CHECK_ARG(p->chunk_len_max <= 2 * BWD_CONS, "sss_backward: chunks of more than %d stages are not supported", 2 * BWD_CONS);
    const bool fast = p->rows_pad == 20 && p->k_pad == 28 && sm.nsp == 52 && g.nsw == 24;
    SN_SET_MAX_SMEM(227 * 1024, sss_bwd_kernel<5, 7, 52>);
    SN_SET_MAX_SMEM(227 * 1024, sss_bwd_kernel<0, 0, 0>);
    if (grad_params != nullptr) SN_CHECK_CUDA(cudaMemsetAsync(workspace, 0, sn_sss_backward_workspace_floats(p) * sizeof(float), st));
    // both directions add their share of grad_x onto zero (two addends per element: the sum does not depend on their order)
    if (grad_x != nullptr) SN_CHECK_CUDA(cudaMemset2DAsync(grad_x, (size_t)ldgx * sizeof(float), 0, (size_t)p->input_dim * sizeof(float), (size_t)B, st));
    float* gpacked = grad_params != nullptr ? workspace : nullptr;
    long tile = (long)BWD_CONS * g.nsw;
    dim3 grid((unsigned)((B + tile - 1) / tile), 2);
    snb::timing_begin("sss_bwd_kernel", st);
    if (fast) sss_bwd_kernel<5, 7, 52><<<grid, BWD_THREADS, smem, st>>>(*p, packed, x, (long)ldx, grad_y, (long)ldgy, ckpt, gpacked, grad_bias, grad_x, (long)ldgx, (long)B, g, sm);
    else sss_bwd_kernel<0, 0, 0><<<grid, BWD_THREADS, smem, st>>>(*p, packed, x, (long)ldx, grad_y, (long)ldgy, ckpt, gpacked, grad_bias, grad_x, (long)ldgx, (long)B, g, sm);
    snb::timing_end(st);
    SN_CHECK_LAUNCH("sss_bwd_kernel");
    if (grad_params == nullptr) return 0;
    sss_unpack_grad_kernel<<<2 * p->nb_states, 128, 0, st>>>(p->stages, 2 * p->nb_states, p->rows_pad, p->k_pad, workspace, grad_params);
    SN_CHECK_LAUNCH("sss_unpack_grad_kernel");
    return 0;
}

}  // extern "C"
