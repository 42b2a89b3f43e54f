"""Float64 parity of the dense GEMM entries at tile edges -- needs a B200.

The exported entries are called directly through the C ABI and compared with a float64 product of exactly the same inputs
(torch float64 on the device; for bf16, the bf16 operands converted exactly to float64):

    sn_dense_apply        y  = x Wᵀ + b          gemm_f32 (A = x [M][K], B = W [N][K])          -> gemm_tf32x3_kernel<false, false>
    sn_dense_input_grad   gx = gy W              gemm_f32 (A = gy [M][K], B = W [K][N])         -> gemm_tf32x3_kernel<false, true>
    sn_dense_weight_grad  dW += gyᵀ x, db += Σ gy  accumulating split-K (A = gy [K][M], B = x [K][N]) -> gemm_tf32x3_kernel<true, true>
    sn_dense_cast_bf16 / sn_dense_apply_bf16 / sn_dense_weight_grad_bf16 / sn_dense_input_grad_bf16   -> gemm_bf16_tc_kernel

M, N, K are the dimensions of the GEMM each entry runs (for the weight gradient, K is the batch).  The fourth tf32x3 layout,
<true, false> (A stored [K][M], B stored [N][K]), is reachable from no exported entry, so it is not tested here.

Which fp32 kernel runs is chosen on purpose and asserted through the library's per-kernel timing report: gemm_f32 takes the 3xTF32
tensor-core kernel when TMA can read both operands (16-byte aligned bases, row pitches that are multiples of 4 floats) and K <= 4096 or
the call accumulates; an odd pitch, a base offset by one float, SNB200_GEMM=simt or a non-accumulating K > 4096 select the SIMT kernel.
In sn_dense_apply / sn_dense_input_grad the weight's row pitch is n_in, so a tensor-core case needs n_in % 4 == 0 there.

Two metrics per check, both against the float64 reference C64:

(a) elementwise:  |C - C64|_ij <= tol * ((|A||B|)_ij + |bias_j| + |C0_ij|)   (C0: the initial value of an accumulated output)
    A lost or doubled term anywhere fails this even where entries cancel.
(b) the project's metric: max|C - C64| / max|C64| <= 1e-5 for fp32 with random-sign operands (bf16 stores: 2^-8, see below), on
    outputs of at least 16 entries (a single random-sign dot product may cancel to nearly nothing).

Derived bounds, and the tolerances set from one measurement on an NVIDIA B200 at a 1000 W power limit ("measured": the maximum of
metric (a) over every random-sign case of the kernel).  Each tolerance is 4x that maximum, rounded up; where the derived bound of a
case is smaller (SIMT and the column sums at K <= 4), the bound is its tolerance (see tolerance()).

* 3xTF32 (gemm_tf32x3_kernel).  The tensor core truncates a raw fp32 operand a to a_h (10 mantissa bits, |a - a_h| < 2^-10 |a|);
  a_l = rn_tf32(a - a_h), so a = a_h + a_l + e_a with |e_a| <= 2^-11 |a - a_h| < 2^-21 |a|.  The kernel adds a_h b_h + a_h b_l + a_l b_h
  (TF32 products are exact in fp32) and drops a_l b_l, a_h e_b, e_a b_h: < (2^-20 + 2 * 2^-21) |ab| = 2^-19 |ab| per product.  Each add
  into a TMEM accumulator truncates, at most one ulp (2^-23) of the running sum, itself <= the sum of |ab| so far; K is spread over 4
  accumulators (or over split-K slices of <= 2048), so at most 3 * ceil(K / 4) truncating adds reach one accumulator, and the epilogue
  adds the <= 4 accumulators, the bias or the atomics into C0 in fp32 (2^-24 each).  Bound:
      tol_tc(K) = 2^-19 + 3 * ceil(K / 4) * 2^-23 + 8 * 2^-24          (3.7e-4 at K = 4096; 2.7e-6 at K = 1)
  measured 8.2e-7 (apply, 128 x 1000 x 4096); tolerance 3.5e-6.
* SIMT (gemm_f32_kernel): fp32 FMA chains, at most K roundings of 2^-24 of the running sum, plus the bias add or the split-K atomics:
      tol_simt(K) = (K + 2) * 2^-24                                    (2.4e-4 at K = 4100)
  measured 2.5e-7 (input_grad, 127 x 129 x 4096); tolerance 1.1e-6 (K = 1: measured 8.8e-8, bound 1.8e-7).
* bf16 (gemm_bf16_tc_kernel): bf16 products are exact in fp32 and accumulate in fp32 (truncating adds as above, K of them), so the
  accumulator is within K * 2^-23 * (|A||B|) of C64.  The bf16 store then rounds once to nearest: at most half an ulp of an 8-bit
  significand, 2^-8 of the value (2^-9 on average); a store that truncates instead errs by up to 2^-7.  The elementwise check for the
  bf16 outputs is therefore |C - C64| <= 2^-8 |C64| + tol * ((|A||B|) + |bias|), with tol_bf16(K) = (K + 2) * 2^-23 + 2^-16 as bound;
  measured (beyond the 2^-8 |C64| term) 2.4e-8; tolerance 1e-7.  The fp32 weight gradient (ATOMIC_F32, split-K over the batch, fp32
  reductions into C0) has no store rounding: bound tol_bf16(K), measured 1.7e-7, tolerance 7e-7.
* The bias-gradient column sums (fp32 adds of exact bf16 or fp32 values): bound (K + 2) * 2^-24, measured 6.6e-8, tolerance 3e-7.

Nonnegative operands (x, W in [0, 1)) on the 3xTF32 kernel report the signed mean relative error: the tensor core truncates, so
every error has the same sign there and a bias that grows with K is what an accumulation bug would show (DESIGN section 4.1).  The
derived bound is tol_tc(K) (9.4e-5 at K = 1024, 3.7e-4 at K = 4096).  Measured: -5.1e-6 at K = 1024 and -2.1e-5 at K = 4096 (signed
mean), 5.8e-6 and 2.2e-5 elementwise; tolerances 4x those.  The bias grows linearly with the K each of the four accumulators sums, so
at K = 4096 a nonnegative product misses the project's 1e-5 relative bar by a factor of two (2.2e-5 max-abs / max-abs); random-sign
operands cancel it.
"""
import math

import pytest
import torch

from structurednets_b200 import _lib

DEV = "cuda"
TC, SIMT = "gemm_tf32x3_kernel", "gemm_f32_kernel"

TC_TOL = 3.5e-6
SIMT_TOL = 1.1e-6
BF16_TOL = 1e-7
BF16_DW_TOL = 7e-7
COLSUM_TOL = 3e-7
NONNEG_TOL = {1024: (2.1e-5, 2.4e-5), 4096: (8.3e-5, 8.8e-5)}     # K: (signed mean, elementwise)
REL_TOL_F32 = 1e-5


def tol_tc(K):
    return 2.0 ** -19 + 3 * math.ceil(K / 4) * 2.0 ** -23 + 8 * 2.0 ** -24


def tol_simt(K):
    return (K + 2) * 2.0 ** -24


def tol_bf16(K):
    return (K + 2) * 2.0 ** -23 + 2.0 ** -16


def tolerance(tol, bound):
    """The tolerance of one case: the constant set from the measurement, or the derived bound where that is smaller (short K)."""
    return min(tol, bound)


def round4(n):
    return (n + 3) // 4 * 4


def pad8(n):
    return (n + 7) // 8 * 8


# ---------------------------------------------------------------- operands with a chosen layout
def operand(rows, cols, layout, gen, nonneg=False, dtype=torch.float32, ld=None):
    """(rows x cols) view with row pitch `ld` into a fresh buffer of random values; layout 'pad': ld = round_up(cols, 4),
    'odd': an odd pitch, 'offset': ld = round_up(cols, 4) but the base one element past a 16-byte boundary."""
    if ld is None:
        ld = {"pad": round4(cols), "odd": round4(cols) + 1, "offset": round4(cols)}[layout]
    off = 1 if layout == "offset" else 0
    n = off + rows * ld + 1
    buf = torch.rand(n, generator=gen, device=DEV)
    if not nonneg:
        buf = buf * 2 - 1
    buf = buf.to(dtype)
    return torch.as_strided(buf, (rows, cols), (ld, 1), off)


def expected_kernel(a, lda, b, ldb, K, accumulate, force_simt):
    """gemm_f32's dispatch rule (csrc/gemm_f32.cuh)."""
    eligible = a.data_ptr() % 16 == 0 and b.data_ptr() % 16 == 0 and lda % 4 == 0 and ldb % 4 == 0
    return TC if (not force_simt and K > 0 and eligible and (accumulate or K <= 4096)) else SIMT


def ran_kernels(call):
    """Runs call() with the library's per-kernel timing on; returns the names of the kernels it launched."""
    lib = _lib.lib()
    _lib.timing_report()
    lib.sn_timing_enable(1)
    try:
        rc = call()
        _lib.check(rc, "dense GEMM entry")
        names = set(_lib.timing_report())
    finally:
        lib.sn_timing_enable(0)
    return names


def elementwise_ratio(err, scale):
    """max of err / scale where scale > 0; entries with scale == 0 must be exact."""
    pos = scale > 0
    assert not bool((err[~pos] != 0).any())
    return float((err[pos] / scale[pos]).max()) if bool(pos.any()) else 0.0


def rel_max(C, C64):
    return float((C.double() - C64).abs().max() / C64.abs().max().clamp_min(1e-300))


def report(kind, case, value):
    print("\nPARITY %s %s %.3e" % (kind, case, value))


# ---------------------------------------------------------------- fp32 cases
# (M, N, K, layout of the batch operands, kernel the case is meant for, bias, y base offset by one float)
# 'env': SNB200_GEMM=simt with padded pitches.  The weight's pitch in apply / input_grad is n_in (K of apply, N of input_grad).
APPLY = [
    (127, 16, 32, "pad", TC, True, False),
    (128, 1000, 4096, "pad", TC, True, False),
    (129, 17, 4, "pad", TC, False, True),
    (1, 129, 32, "pad", TC, True, True),
    (300, 15, 4096, "pad", TC, True, True),
    (300, 4, 32, "pad", TC, False, False),
    (127, 1, 4, "pad", TC, True, False),
    (129, 1000, 33, "pad", SIMT, True, False),       # W pitch 33
    (1, 16, 1, "pad", SIMT, True, False),            # W pitch 1
    (300, 17, 31, "pad", SIMT, False, True),         # W pitch 31
    (128, 4, 4100, "pad", SIMT, True, False),        # K > 4096 without accumulation
    (1, 1, 4100, "pad", SIMT, False, False),
    (127, 129, 32, "offset", SIMT, True, False),
    (128, 16, 32, "odd", SIMT, True, False),
    (129, 15, 4096, "env", SIMT, True, False),
]
INPUT_GRAD = [
    (127, 16, 1, "pad", TC, False, False),
    (128, 4, 31, "pad", TC, False, True),
    (129, 1000, 33, "pad", TC, False, False),
    (300, 16, 4096, "pad", TC, False, True),
    (1, 4, 32, "pad", TC, False, False),
    (128, 1000, 4, "pad", TC, False, False),
    (129, 16, 4100, "pad", SIMT, False, False),      # K > 4096 without accumulation
    (300, 15, 32, "pad", SIMT, False, False),        # W pitch 15
    (1, 17, 31, "pad", SIMT, False, True),
    (127, 129, 4096, "pad", SIMT, False, False),
    (128, 1, 4, "pad", SIMT, False, False),
    (128, 1000, 33, "env", SIMT, False, False),
    (300, 4, 4, "offset", SIMT, False, False),
    (129, 16, 1, "odd", SIMT, False, False),
]
WEIGHT_GRAD = [
    (1, 1, 1, "pad", TC, True, False),
    (127, 15, 4, "pad", TC, True, False),
    (128, 17, 31, "pad", TC, False, False),
    (129, 129, 32, "pad", TC, True, False),
    (300, 1000, 33, "pad", TC, True, False),
    (128, 16, 4096, "pad", TC, True, False),
    (300, 4, 4096, "pad", TC, False, False),
    (129, 1000, 4096, "env", SIMT, True, False),
    (1, 16, 32, "odd", SIMT, True, False),
    (127, 4, 33, "offset", SIMT, True, False),
    (300, 129, 1, "odd", SIMT, False, False),
    (128, 1, 31, "env", SIMT, True, False),
    (300, 129, 65536, "pad", TC, True, False),       # split-K and the 2048-per-slice limit
    (129, 17, 65536, "odd", SIMT, True, False),
]
ENTRIES = {"apply": APPLY, "input_grad": INPUT_GRAD, "weight_grad": WEIGHT_GRAD}


def case_id(c):
    M, N, K, layout, kern, bias, yoff = c
    return "%dx%dx%d-%s-%s%s%s" % (M, N, K, layout, "tc" if kern == TC else "simt", "-bias" if bias else "", "-yoff" if yoff else "")


def test_fp32_cases_cover_every_edge_and_both_kernels():
    Ms, Ns, Ks = {1, 127, 128, 129, 300}, {1, 4, 15, 16, 17, 129, 1000}, {1, 4, 31, 32, 33, 4096}
    for name, cases in ENTRIES.items():
        assert Ms <= {c[0] for c in cases}, name
        assert Ns <= {c[1] for c in cases}, name
        assert Ks <= {c[2] for c in cases}, name
        assert {TC, SIMT} == {c[4] for c in cases}, name
        assert {True, False} == {c[5] for c in cases} or name == "input_grad", name
    assert 4100 in {c[2] for c in APPLY} and 4100 in {c[2] for c in INPUT_GRAD}
    assert any(c[6] and c[4] == TC for c in APPLY) and any(c[6] and c[4] == TC for c in INPUT_GRAD)


def output_buffer(M, N, yoff):
    """(M x N) fp32 output prefilled with garbage; yoff: base one float past a 16-byte boundary (the tf32x3 epilogue's scalar stores)."""
    ld = round4(N + 1)
    buf = torch.full((M * ld + 1 + 4,), float("nan"), device=DEV)
    return torch.as_strided(buf, (M, N), (ld, 1), 1 if yoff else 0)


@pytest.mark.gpu
@pytest.mark.parametrize("entry,case", [(e, c) for e, cs in ENTRIES.items() for c in cs], ids=lambda v: v if isinstance(v, str) else case_id(v))
def test_fp32_entry_vs_float64(built_lib, monkeypatch, entry, case):
    M, N, K, layout, kern, use_bias, yoff = case
    force_simt = layout == "env"
    if force_simt:
        monkeypatch.setenv("SNB200_GEMM", "simt")
    else:
        monkeypatch.delenv("SNB200_GEMM", raising=False)
    lay = "pad" if force_simt else layout
    gen = torch.Generator(device=DEV)
    gen.manual_seed(M * 1000003 + N * 1009 + K)
    lib, stream = _lib.lib(), _lib.stream_ptr()
    bias = (torch.rand(N, generator=gen, device=DEV) * 2 - 1) if use_bias else None

    if entry == "apply":            # y[M x N] = x[M x K] W[N x K]^T + b
        x, W = operand(M, K, lay, gen), operand(N, K, "pad", gen, ld=K)
        y = output_buffer(M, N, yoff)
        want = expected_kernel(x, x.stride(0), W, K, K, False, force_simt)
        ran = ran_kernels(lambda: lib.sn_dense_apply(_lib.ptr(W), N, K, _lib.ptr(x), x.stride(0), _lib.ptr(y), y.stride(0), _lib.ptr(bias), M, stream))
        C, C64 = y, x.double() @ W.double().T
        scale = x.double().abs() @ W.double().abs().T
        if bias is not None:
            C64 = C64 + bias.double()
            scale = scale + bias.double().abs()
    elif entry == "input_grad":     # gx[M x N] = gy[M x K] W[K x N]
        gy, W = operand(M, K, lay, gen), operand(K, N, "pad", gen, ld=N)
        gx = output_buffer(M, N, yoff)
        want = expected_kernel(gy, gy.stride(0), W, N, K, False, force_simt)
        ran = ran_kernels(lambda: lib.sn_dense_input_grad(_lib.ptr(W), K, N, _lib.ptr(gy), gy.stride(0), _lib.ptr(gx), gx.stride(0), M, stream))
        C, C64 = gx, gy.double() @ W.double()
        scale = gy.double().abs() @ W.double().abs()
    else:                           # dW[M x N] += gy[K x M]^T x[K x N],  db[M] += colsum(gy)
        gy, x = operand(K, M, lay, gen), operand(K, N, lay, gen)
        dW = torch.rand(M, N, generator=gen, device=DEV) * 2 - 1
        dW0 = dW.clone()
        db = (torch.rand(M, generator=gen, device=DEV) * 2 - 1) if use_bias else None
        db0 = db.clone() if db is not None else None
        want = expected_kernel(gy, gy.stride(0), x, x.stride(0), K, True, force_simt)
        ran = ran_kernels(lambda: lib.sn_dense_weight_grad(_lib.ptr(x), x.stride(0), _lib.ptr(gy), gy.stride(0), _lib.ptr(dW), M, N, _lib.ptr(db), K,
                                                           stream))
        C, C64 = dW, dW0.double() + gy.double().T @ x.double()
        C0 = dW0.double()
        scale = gy.double().abs().T @ x.double().abs() + dW0.double().abs()
        if db is not None:
            ref = db0.double() + gy.double().sum(0)
            r = elementwise_ratio((db.double() - ref).abs(), gy.double().abs().sum(0) + db0.double().abs())
            report("colsum", case_id(case), r)
            assert r <= tolerance(COLSUM_TOL, tol_simt(K)), r

    err = (C.double() - C64).abs()
    r = elementwise_ratio(err, scale)
    report("tc" if kern == TC else "simt", entry + "-" + case_id(case), r)
    assert want == kern, "the case does not select the kernel it is meant for"
    assert want in ran and ({TC, SIMT} - {want}).isdisjoint(ran), ran
    tol = tolerance(TC_TOL, tol_tc(K)) if kern == TC else tolerance(SIMT_TOL, tol_simt(K))
    assert r <= tol, "elementwise error %.3e > %.1e" % (r, tol)
    # the project's metric needs enough entries that max|C64| is of the size of a typical product sum: a single dot product of
    # random-sign terms may cancel to nearly nothing.  The weight gradient is measured on what the call added (dW0 and it may cancel).
    if M * N >= 16:
        if entry == "weight_grad":
            assert rel_max(C.double() - C0, C64 - C0) <= REL_TOL_F32
        else:
            assert rel_max(C, C64) <= REL_TOL_F32


@pytest.mark.gpu
def test_fp32_empty_reduction_writes_bias_or_zeros(built_lib, monkeypatch):
    """K = 0: y = bias (apply with n_in = 0), gx = 0 (input_grad with n_out = 0); dW and db are untouched (weight_grad with B = 0)."""
    monkeypatch.delenv("SNB200_GEMM", raising=False)
    lib, stream = _lib.lib(), _lib.stream_ptr()
    M, N = 129, 17
    dummy = torch.zeros(4, device=DEV)
    bias = torch.randn(N, device=DEV)
    y = torch.full((M, N), float("nan"), device=DEV)
    _lib.check(lib.sn_dense_apply(_lib.ptr(dummy), N, 0, _lib.ptr(dummy), 4, _lib.ptr(y), N, _lib.ptr(bias), M, stream), "sn_dense_apply")
    assert torch.equal(y, bias.expand(M, N))
    _lib.check(lib.sn_dense_apply(_lib.ptr(dummy), N, 0, _lib.ptr(dummy), 4, _lib.ptr(y), N, None, M, stream), "sn_dense_apply")
    assert not bool(y.any())
    gx = torch.full((M, N), float("nan"), device=DEV)
    _lib.check(lib.sn_dense_input_grad(_lib.ptr(dummy), 0, N, _lib.ptr(dummy), 4, _lib.ptr(gx), N, M, stream), "sn_dense_input_grad")
    assert not bool(gx.any())
    dW, db = torch.randn(M, N, device=DEV), torch.randn(M, device=DEV)
    dW0, db0 = dW.clone(), db.clone()
    _lib.check(lib.sn_dense_weight_grad(_lib.ptr(dummy), N, _lib.ptr(dummy), M, _lib.ptr(dW), M, N, _lib.ptr(db), 0, stream), "sn_dense_weight_grad")
    torch.cuda.synchronize()
    assert torch.equal(dW, dW0) and torch.equal(db, db0)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1024, 4096])
def test_tf32x3_nonnegative_operands_accumulation_bias(built_lib, monkeypatch, K):
    """x, W in [0, 1) on the tensor cores: the signed mean relative error (the truncation bias) stays within its bound."""
    monkeypatch.delenv("SNB200_GEMM", raising=False)
    gen = torch.Generator(device=DEV)
    gen.manual_seed(K)
    M, N = 300, 1000
    x, W = operand(M, K, "pad", gen, nonneg=True), operand(N, K, "pad", gen, nonneg=True, ld=K)
    y = torch.empty(M, N, device=DEV)
    lib = _lib.lib()
    ran = ran_kernels(lambda: lib.sn_dense_apply(_lib.ptr(W), N, K, _lib.ptr(x), K, _lib.ptr(y), N, None, M, _lib.stream_ptr()))
    assert TC in ran and SIMT not in ran
    C64 = x.double() @ W.double().T
    mean = float(((y.double() - C64) / C64).mean())
    r = elementwise_ratio((y.double() - C64).abs(), C64)
    report("mean", "nonneg-%dx%dx%d" % (M, N, K), mean)
    report("tc", "nonneg-%dx%dx%d" % (M, N, K), r)
    report("rel", "nonneg-%dx%dx%d" % (M, N, K), rel_max(y, C64))
    mean_tol, tol = NONNEG_TOL[K]
    assert abs(mean) <= mean_tol <= tol_tc(K)
    assert r <= tol <= tol_tc(K)


# ---------------------------------------------------------------- bf16 entries
BF16_DIMS = [8, 56, 64, 72, 1000]


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols", [(8, 56), (56, 8), (64, 72), (72, 64), (1000, 1000), (8, 1000), (1000, 72), (1, 8)])
def test_bf16_cast_matches_torch_and_zeroes_the_pad(built_lib, rows, cols):
    gen = torch.Generator(device=DEV)
    gen.manual_seed(rows * 7919 + cols)
    M = torch.randn(rows, cols, generator=gen, device=DEV) * 4
    # round-to-nearest-even ties, both signs, values beyond bf16's largest finite number's rounding point, fp32 subnormals, zeros
    special = torch.tensor([1 + 2 ** -8, 1 + 3 * 2 ** -8, -(1 + 2 ** -8), 2 ** -8 + 2 ** -16, 3.39e38, -3.4e38, 1e-39, -1e-39, 0.0, -0.0,
                            2 ** -126, 65504.0], device=DEV)
    flat = M.view(-1)
    flat[:min(flat.numel(), special.numel())] = special[:flat.numel()]
    ldmb, ldmtb = pad8(cols) + 8, pad8(rows) + 16
    Mb = torch.full((rows, ldmb), 7.0, dtype=torch.bfloat16, device=DEV)
    Mtb = torch.full((cols, ldmtb), 7.0, dtype=torch.bfloat16, device=DEV)
    lib = _lib.lib()
    _lib.check(lib.sn_dense_cast_bf16(_lib.ptr(M), rows, cols, _lib.ptr(Mb), ldmb, _lib.ptr(Mtb), ldmtb, _lib.stream_ptr()), "sn_dense_cast_bf16")
    want = M.cpu().to(torch.bfloat16)
    bits = lambda t: t.contiguous().cpu().view(torch.int16)
    assert torch.equal(bits(Mb[:, :cols]), bits(want))
    assert torch.equal(bits(Mtb[:, :rows]), bits(want.T))
    assert not bool(Mb[:, cols:].float().any()) and not bool(Mtb[:, rows:].float().any())
    # either output alone
    for Mb_, Mtb_ in ((Mb, None), (None, Mtb)):
        for t in (Mb, Mtb):
            t.fill_(7.0)
        _lib.check(lib.sn_dense_cast_bf16(_lib.ptr(M), rows, cols, _lib.ptr(Mb_), ldmb, _lib.ptr(Mtb_), ldmtb, _lib.stream_ptr()), "sn_dense_cast_bf16")
        if Mb_ is not None:
            assert torch.equal(bits(Mb[:, :cols]), bits(want)) and not bool(Mb[:, cols:].float().any())
            assert bool((Mtb.float() == 7.0).all())
        else:
            assert torch.equal(bits(Mtb[:, :rows]), bits(want.T)) and not bool(Mtb[:, rows:].float().any())
            assert bool((Mb.float() == 7.0).all())


def bf16_operand(rows, cols, gen, extra=8):
    """(rows x cols) bf16 view with a row pitch larger than the width (a multiple of 8, as TMA needs)."""
    return operand(rows, cols, "pad", gen, dtype=torch.bfloat16, ld=pad8(cols) + extra)


def check_bf16_store(C, C64, scale, K, kind, case):
    """bf16 output: one rounding to nearest of the fp32 accumulator, plus the accumulation error."""
    err = (C.double() - C64).abs() - 2.0 ** -8 * C64.abs()
    r = elementwise_ratio(err.clamp_min(0), scale)
    report(kind, case, r)
    assert r <= tolerance(BF16_TOL, tol_bf16(K)), "elementwise error %.3e" % r
    assert rel_max(C, C64) <= 2.0 ** -8 + 1e-5


BF16_GEMM = [  # (M = batch, N, K)
    (1, 8, 64), (127, 56, 8), (128, 64, 56), (129, 72, 1000), (300, 1000, 72), (64, 1000, 1000), (65, 8, 8), (513, 72, 64),
]


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K", BF16_GEMM)
@pytest.mark.parametrize("use_bias", [False, True])
def test_bf16_apply_vs_float64(built_lib, M, N, K, use_bias):
    gen = torch.Generator(device=DEV)
    gen.manual_seed(M * 131 + N * 17 + K)
    x, Wb = bf16_operand(M, K, gen), bf16_operand(N, K, gen, extra=16)
    bias = (torch.rand(N, generator=gen, device=DEV) * 2 - 1) if use_bias else None
    ldy = pad8(N) + 8
    ybuf = torch.full((M, ldy), 7.0, dtype=torch.bfloat16, device=DEV)
    y = ybuf[:, :N]
    _lib.check(_lib.lib().sn_dense_apply_bf16(_lib.ptr(Wb), Wb.stride(0), N, K, _lib.ptr(x), x.stride(0), _lib.ptr(y), ldy, _lib.ptr(bias), M,
                                              _lib.stream_ptr()), "sn_dense_apply_bf16")
    C64 = x.double() @ Wb.double().T
    scale = x.double().abs() @ Wb.double().abs().T
    if bias is not None:
        C64, scale = C64 + bias.double(), scale + bias.double().abs()
    check_bf16_store(y, C64, scale, K, "bf16", "apply-%dx%dx%d" % (M, N, K))
    assert bool((ybuf[:, N:].float() == 7.0).all()), "the store wrote past N"


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K", BF16_GEMM)
def test_bf16_input_grad_vs_float64(built_lib, M, N, K):
    """gx[M x N] = gy[M x K] W[K x N], W given as its bf16 transpose Wt [N][ldwt]."""
    gen = torch.Generator(device=DEV)
    gen.manual_seed(M * 7 + N * 131 + K)
    gy, Wt = bf16_operand(M, K, gen), bf16_operand(N, K, gen, extra=24)
    ldgx = pad8(N) + 8
    gxbuf = torch.full((M, ldgx), 7.0, dtype=torch.bfloat16, device=DEV)
    gx = gxbuf[:, :N]
    _lib.check(_lib.lib().sn_dense_input_grad_bf16(_lib.ptr(Wt), Wt.stride(0), K, N, _lib.ptr(gy), gy.stride(0), _lib.ptr(gx), ldgx, M,
                                                   _lib.stream_ptr()), "sn_dense_input_grad_bf16")
    C64 = gy.double() @ Wt.double().T
    check_bf16_store(gx, C64, gy.double().abs() @ Wt.double().abs().T, K, "bf16", "input_grad-%dx%dx%d" % (M, N, K))
    assert bool((gxbuf[:, N:].float() == 7.0).all()), "the store wrote past N"


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 63, 64, 65, 511, 512, 513, 8193])
@pytest.mark.parametrize("n_out,n_in", [(8, 1000), (1000, 56), (72, 64), (64, 72)])
def test_bf16_weight_grad_vs_float64(built_lib, B, n_out, n_in):
    """dW[n_out x n_in] += gy[B x n_out]^T x[B x n_in] (fp32, split-K over the batch), db += colsum(gy)."""
    gen = torch.Generator(device=DEV)
    gen.manual_seed(B * 31 + n_out * 7 + n_in)
    x, gy = bf16_operand(B, n_in, gen), bf16_operand(B, n_out, gen, extra=16)
    lddw = n_in + (4 if n_out in (8, 72) else 1)     # 16-byte aligned rows (vector reductions) or not (scalar atomics)
    dWbuf = torch.rand(n_out, lddw, generator=gen, device=DEV) * 2 - 1
    dW0 = dWbuf.clone()
    db = torch.rand(n_out, generator=gen, device=DEV) * 2 - 1
    db0 = db.clone()
    _lib.check(_lib.lib().sn_dense_weight_grad_bf16(_lib.ptr(x), x.stride(0), _lib.ptr(gy), gy.stride(0), _lib.ptr(dWbuf), lddw, n_out, n_in,
                                                    _lib.ptr(db), B, _lib.stream_ptr()), "sn_dense_weight_grad_bf16")
    C64 = dW0[:, :n_in].double() + gy.double().T @ x.double()
    scale = gy.double().abs().T @ x.double().abs() + dW0[:, :n_in].double().abs()
    r = elementwise_ratio((dWbuf[:, :n_in].double() - C64).abs(), scale)
    report("bf16_dw", "%dx%dx%d" % (n_out, n_in, B), r)
    assert r <= tolerance(BF16_DW_TOL, tol_bf16(B)), "elementwise error %.3e" % r
    C0 = dW0[:, :n_in].double()
    assert rel_max(dWbuf[:, :n_in].double() - C0, C64 - C0) <= REL_TOL_F32
    assert torch.equal(dWbuf[:, n_in:], dW0[:, n_in:]), "the reductions wrote past n_in"
    ref = db0.double() + gy.double().sum(0)
    r = elementwise_ratio((db.double() - ref).abs(), gy.double().abs().sum(0) + db0.double().abs())
    report("colsum", "bf16-%dx%d" % (n_out, B), r)
    assert r <= tolerance(COLSUM_TOL, tol_simt(B))
