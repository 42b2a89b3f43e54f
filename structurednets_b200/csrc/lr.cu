// Low-rank layer, fp32 path:  y = (x R^T) L^T + b   with L = left_lr (out x r), R = right_lr (r x in).
// Replaces LRLayer.forward (reference layers/lr_layer.py:38-46) and its autograd backward.
// The hidden activations h = x R^T (B x r) are kept for the backward (r floats per sample).
// (The bf16 tensor-core path of BASELINE config C2 lives in lr_tc.cu.)
#include "gemm_f32.cuh"
#include "util.cuh"

extern "C" {

int sn_lr_forward_f32(const float* x, int64_t ldx, const float* left, const float* right, const float* bias, float* hidden,
                      float* y, int64_t ldy, int64_t B, int in_dim, int out_dim, int rank, sn_stream_t stream) {
    SN_CHECK_ARG(left && right, "lr_forward: NULL buffer");
    SN_CHECK_ARG(in_dim > 0 && out_dim > 0 && rank >= 0 && B >= 0, "lr_forward: bad dims");
    if (B == 0) return 0;
    SN_CHECK_ARG(x && hidden && y, "lr_forward: NULL buffer");
    cudaStream_t s = snb::as_stream(stream);
    // h = x R^T : (B x in) (r x in)^T
    if (int rc = snb::gemm_f32(false, true, (int)B, rank, in_dim, 1.f, x, ldx, right, in_dim, 0.f, hidden, rank, nullptr, s)) return rc;
    // y = h L^T + b : (B x r) (out x r)^T
    return snb::gemm_f32(false, true, (int)B, out_dim, rank, 1.f, hidden, rank, left, rank, 0.f, y, ldy, bias, s);
}

int sn_lr_backward_f32(const float* x, int64_t ldx, const float* grad_y, int64_t ldgy, const float* left, const float* right,
                       const float* hidden, float* grad_hidden_ws, float* grad_left, float* grad_right, float* grad_bias,
                       float* grad_x, int64_t ldgx, int64_t B, int in_dim, int out_dim, int rank, sn_stream_t stream) {
    SN_CHECK_ARG(left && right, "lr_backward: NULL buffer");
    if (B <= 0) return 0;
    SN_CHECK_ARG(x && grad_y && hidden && grad_hidden_ws, "lr_backward: NULL buffer");
    cudaStream_t s = snb::as_stream(stream);
    // gh = gy L : (B x out) (out x r)
    if (int rc = snb::gemm_f32(false, false, (int)B, rank, out_dim, 1.f, grad_y, ldgy, left, rank, 0.f, grad_hidden_ws, rank, nullptr, s)) return rc;
    if (grad_left)   // dL += gy^T h : (out x B) (B x r)
        if (int rc = snb::gemm_f32(true, false, out_dim, rank, (int)B, 1.f, grad_y, ldgy, hidden, rank, 1.f, grad_left, rank, nullptr, s, true)) return rc;
    if (grad_right)  // dR += gh^T x : (r x B) (B x in)
        if (int rc = snb::gemm_f32(true, false, rank, in_dim, (int)B, 1.f, grad_hidden_ws, rank, x, ldx, 1.f, grad_right, in_dim, nullptr, s, true)) return rc;
    if (grad_bias)
        if (int rc = snb::colsum_accumulate(grad_y, ldgy, B, out_dim, grad_bias, s)) return rc;
    if (grad_x)      // gx = gh R : (B x r) (r x in)
        if (int rc = snb::gemm_f32(false, false, (int)B, in_dim, rank, 1.f, grad_hidden_ws, rank, right, in_dim, 0.f, grad_x, ldgx, nullptr, s)) return rc;
    return 0;
}

}  // extern "C"
