#!/usr/bin/env python
"""Benchmark of the structured-layer hot path (BASELINE.json metric: structured-layer fwd+bwd samples/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload sss|lr|lr_bf16|psm|psm_sparse|hmat|ldr] [--impl ours|reference]
                    [--dump-outputs DIR]

A "step" is one forward + backward (parameter gradients only, as training_helpers.py:141-144 produces)
of the layer over one batch of synthetic features that are already resident in HBM; for N > 1 the
batch is sharded over the ranks (data parallel, strong scaling: the global batch is fixed) and the step
ends with one NCCL all-reduce of the flat gradient buffer.  Prints ONE JSON line (rank 0).

The headline workload is BASELINE config C5 (SSS 4096 -> 1000, global batch 65 536).  At N = 1 the same line carries a
`workloads` dict with the other configs (C1 with host features through get_batch, C2 bf16 low rank, C3 PSM on both CUDA
paths, C4-H, C4-L), each with its step time, roofline fractions, dominant kernel and CPU baseline, a `sustained` figure
(>= 2 s of graph replays with the clocks seen) and `gpu_aten_baseline` (the reference's own torch ops on the same B200).

`--impl reference` times the reference's CPU path (oracle port: the same torch CPU ops the reference
layer issues, autograd backward) on the box's host cores on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import numpy as np
import torch

HBM_FALLBACK_GBS = 6650.0      # /opt/skills/guides/B200_PROFILING.md fallback
BF16_FALLBACK_TFLOPS = 1590.0
FP32_FMA_TFLOPS_NOMINAL = 148 * 128 * 2 * 1.965e9 / 1e12   # 74.4: 148 SMs x 128 FMA lanes x 2 flop x max clock
L2_BYTES = 126 * 2 ** 20


def measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=float(p["hbm_gbs"]), bf16_tflops=float(p["bf16_tflops"]),
                    bf16_tflops_sustained=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), source="measured")
    return dict(hbm_gbs=HBM_FALLBACK_GBS, bf16_tflops=BF16_FALLBACK_TFLOPS, bf16_tflops_sustained=1400.0, source="fallback")


# ----------------------------------------------------------------------------------------------
# workloads
# ----------------------------------------------------------------------------------------------
class SSSWorkload:
    """BASELINE config C5 (= C1's layer): SSSLayer 4096 -> 1000, 500 stages, statespace dim 16, fp32,
    global batch 65536 sharded over the ranks."""
    name = "sss"
    dtype = "f32"
    input_dim, output_dim, nb_states, statespace_dim = 4096, 1000, 500, 16
    global_batch = 65536
    cpu_sample_batch = 256
    bytes_per_sample_kernel = 4 * (4096 + 1000)          # one kernel (fwd: read x, write y; bwd: read gy, re-read x)
    bytes_per_sample = 2 * bytes_per_sample_kernel        # SURVEY.md section 8(d): 40 768 B / sample fwd+bwd
    flop_per_sample = 2277504                              # SURVEY.md section 8(d)
    bound = "hbm"
    # algorithmic bytes per sample of the kernels that touch the layer's inputs / outputs (SURVEY.md 8d: x and grad_y read once per
    # pass, y written once; every other byte a kernel moves is scratch): 16 384 + 4 000 + 4 000 + 20 384 = 40 768
    kernel_bytes_per_sample = {"sss_tc_local_gemm_kernel": 4 * 4096, "sss_tc_chain_fwd_kernel": 4 * 1000, "sss_tc_chain_bwd_kernel": 4 * 1000,
                               "sss_tc_grad_gemm_kernel": 4 * (4096 + 1000), "sss_tc_scan_out_q_kernel": 4 * 1000,
                               "sss_tc_scan_bwd_q_kernel": 4 * 1000, "sss_tc_scan_out_m_kernel": 4 * 1000, "sss_tc_scan_bwd_m_kernel": 4 * 1000}
    # dram__bytes_read.sum + dram__bytes_write.sum per launch at local batch 65 536 from the committed `ncu --set full` captures named in
    # traffic_source (cold-cache replays of the same bench command); only quoted for the batch they were captured at
    traffic_source = "profiles/r2_sss_top_kernels.md, profiles/r2_sss_scans_65536.md"
    traffic_batch = 65536
    traffic_bytes = {"sss_tc_local_gemm_kernel": 1.0775e9 + 0.5096e9, "sss_tc_chain_fwd_kernel": 0.7644e9 + 0.7663e9,
                     "sss_tc_chain_bwd_kernel": 0.5358e9 + 0.2520e9, "sss_tc_grad_gemm_kernel": 1.9522e9 + 0.0064e9,
                     "sss_tc_scan_states_m_kernel": 0.2685e9 + 0.2421e9, "sss_tc_scan_out_m_kernel": 0.5370e9 + 0.2382e9,
                     "sss_tc_scan_bwd_m_kernel": 0.3025e9 + 0.2379e9}

    def describe(self):
        return dict(workload="C5: SSS 4096->1000, 500 stages, statespace 16, fp32 fwd+bwd (param grads), global batch 65536",
                    global_batch=self.global_batch, timed_inputs="resident in HBM; 1 GiB feature matrix per step >> 126 MB L2")

    def system(self):
        from structurednets_b200.synth import random_mixed_system
        return random_mixed_system(self.input_dim, self.output_dim, self.nb_states, self.statespace_dim, seed=5000)

    def make_layer(self, device):
        from structurednets_b200.layers.sss_layer import SSSLayer
        np.random.seed(5000)      # the bias is Glorot-initialised from numpy's global RNG: every run builds the same layer
        layer = SSSLayer(self.input_dim, self.output_dim, 0.105, nb_states=self.nb_states, initial_system_approx=self.system())
        assert layer.statespace_dim == self.statespace_dim
        return layer.to(device)

    def make_inputs(self, batch, device, seed):
        g = torch.Generator(device=device).manual_seed(seed)
        x = torch.rand((batch, self.input_dim), device=device, generator=g) * 2 - 1
        gy = (torch.rand((batch, self.output_dim), device=device, generator=g) * 2 - 1) / batch
        labels = torch.randint(0, self.output_dim, (batch,), device=device, generator=g)
        return x, gy, labels

    def ref_step_fn(self, batch, device="cpu"):
        """The reference's own path for this workload (oracle port of sss_layer.py:99-131 + autograd): the same ATen ops on `device`."""
        from oracle import layers_cpu as O
        sysm = self.system()
        f32 = lambda m: torch.tensor(np.asarray(m)).float().to(device).requires_grad_(True)
        cs, acs = sysm.causal_system.stages, sysm.anticausal_system.stages
        lists = [[f32(s.A_matrix) for s in cs], [f32(s.B_matrix) for s in cs], [f32(s.C_matrix) for s in cs],
                 [f32(s.D_matrix) for s in cs], [f32(s.A_matrix) for s in acs], [f32(s.B_matrix) for s in acs],
                 [f32(s.C_matrix) for s in acs]]
        bias = torch.zeros(self.output_dim, device=device, requires_grad=True)
        rng = np.random.default_rng(5000)
        x = torch.tensor(rng.uniform(-1, 1, size=(batch, self.input_dim)).astype(np.float32)).to(device)
        gy = (torch.tensor(rng.uniform(-1, 1, size=(batch, self.output_dim)).astype(np.float32)) / batch).to(device)
        params = [p for l in lists for p in l] + [bias]

        def step():
            for p in params:
                p.grad = None
            y = O.sss_forward(x, *lists, bias, sysm.dims_in, sysm.dims_out)
            y.backward(gy)
        return step


class _DenseInputsMixin:
    def make_inputs(self, batch, device, seed):
        g = torch.Generator(device=device).manual_seed(seed)
        x = torch.rand((batch, self.input_dim), device=device, generator=g) * 2 - 1
        gy = (torch.rand((batch, self.output_dim), device=device, generator=g) * 2 - 1) / batch
        labels = torch.randint(0, self.output_dim, (batch,), device=device, generator=g)
        return x, gy, labels

    def _cpu_xy(self, batch, seed, device="cpu"):
        rng = np.random.default_rng(seed)
        x = torch.tensor(rng.uniform(-1, 1, size=(batch, self.input_dim)).astype(np.float32))
        gy = torch.tensor(rng.uniform(-1, 1, size=(batch, self.output_dim)).astype(np.float32)) / batch
        return x.to(device), gy.to(device)


class LRWorkload(_DenseInputsMixin):
    """BASELINE config C2's shape in fp32: LRLayer 2048 -> 1000, rank 128, batch 8192 (3xTF32 tensor-core GEMMs, csrc/lr.cu)."""
    name, dtype, bound = "lr", "f32", "hbm"
    input_dim, output_dim, rank = 2048, 1000, 128
    global_batch, cpu_sample_batch = 8192, 8192
    bytes_per_sample_kernel = 4 * (2048 + 1000)
    bytes_per_sample = 2 * bytes_per_sample_kernel
    flop_per_sample = 1816576
    kernels = ("gemm_f32_kernel", "gemm_f32_kernel")

    def describe(self):
        return dict(workload="C2 shape in fp32: low-rank 2048->1000 rank 128, fp32 fwd+bwd (3xTF32 on tcgen05), batch 8192",
                    global_batch=self.global_batch, timed_inputs="resident in HBM")

    def make_layer(self, device):
        from structurednets_b200.layers.lr_layer import LRLayer
        np.random.seed(2000)
        layer = LRLayer(self.input_dim, self.output_dim, 0.1906)
        assert layer.left_lr.shape[1] == self.rank
        return layer.to(device)

    def ref_step_fn(self, batch, device="cpu"):
        from oracle import layers_cpu as O
        np.random.seed(2000)
        lim = lambda shape: np.sqrt(6 / sum(shape))
        L = torch.tensor(np.random.uniform(-lim((1000, 128)), lim((1000, 128)), (1000, 128)).astype(np.float32)).to(device).requires_grad_(True)
        R = torch.tensor(np.random.uniform(-lim((128, 2048)), lim((128, 2048)), (128, 2048)).astype(np.float32)).to(device).requires_grad_(True)
        b = torch.zeros(1000, device=device, requires_grad=True)
        x, gy = self._cpu_xy(batch, 2000, device)

        def step():
            for p in (L, R, b):
                p.grad = None
            O.lr_forward(x, L, R, b).backward(gy)
        return step


class LRBf16Workload(LRWorkload):
    """BASELINE config C2: LRLayer 2048 -> 1000, rank 128, bf16 fwd+bwd (tcgen05 / TMEM / TMA), fp32 master parameters."""
    name, dtype, bound = "lr_bf16", "bf16", "hbm"
    tensor_bound = True
    bytes_per_sample_kernel = 2 * (2048 + 1000)
    bytes_per_sample = 2 * bytes_per_sample_kernel        # SURVEY.md section 8(d): 12 192 B / sample
    kernels = ("gemm_bf16_tc_kernel", "gemm_bf16_tc_kernel")

    def describe(self):
        return dict(workload="C2: low-rank 2048->1000 rank 128, bf16 fwd+bwd on tcgen05 (fp32 accumulate, fp32 master params), batch 8192",
                    global_batch=self.global_batch, timed_inputs="resident in HBM")

    def make_inputs(self, batch, device, seed):
        x, gy, labels = super().make_inputs(batch, device, seed)
        return x.bfloat16(), gy.bfloat16(), labels


class PSMWorkload(_DenseInputsMixin):
    """BASELINE config C3: PSMLayer 4096 -> 1000, 3 factors, nb_params_share 0.1 => 409 599 nnz, batch 8192, intended
    factor order (SURVEY.md F2)."""
    name, dtype, bound = "psm", "f32", "hbm"
    input_dim, output_dim = 4096, 1000
    global_batch, cpu_sample_batch = 8192, 512
    bytes_per_sample_kernel = 4 * (4096 + 1000)
    bytes_per_sample = 2 * bytes_per_sample_kernel
    flop_per_sample = 2184528
    kernels = ("psm_fwd_kernel", "psm_bwd_kernel")

    def describe(self):
        return dict(workload="C3: PSM 4096->1000, 3 sparse factors, 409 599 nnz (share 0.1), fp32 fwd+bwd, batch 8192",
                    global_batch=self.global_batch, timed_inputs="resident in HBM")

    def factors(self):
        import scipy.sparse
        shapes = [(1000, 4096), (4096, 4096), (4096, 4096)]
        out = []
        for k, (r, c) in enumerate(shapes):
            m = scipy.sparse.random(r, c, density=136533 / (r * c), random_state=3000 + k, format="csr", dtype=np.float64)
            m.data = np.random.default_rng(3000 + k).uniform(-0.05, 0.05, size=m.data.shape)
            out.append(m)
        return out

    def make_layer(self, device):
        from structurednets_b200.layers.psm_layer import PSMLayer
        np.random.seed(3000)      # Glorot bias, as in SSSWorkload.make_layer
        return PSMLayer(self.input_dim, self.output_dim, sparse_matrices=self.factors()).to(device)

    def ref_step_fn(self, batch, device="cpu"):
        from oracle import layers_cpu as O
        fs = [torch.tensor(f.toarray()).float().to(device).requires_grad_(True) for f in self.factors()]
        b = torch.zeros(1000, device=device, requires_grad=True)
        x, gy = self._cpu_xy(batch, 3000, device)

        def step():   # the reference's default path: dense mm chain (psm_layer.py:51-58), corrected factor order
            for p in fs + [b]:
                p.grad = None
            O.psm_forward(x, fs, b).backward(gy)
        return step


class PSMSparseWorkload(PSMWorkload):
    """C3 on the sparse chain kernel north_star names (intermediates in shared memory, only x and y touch HBM); the layer's default
    for this batch is the dense-product path (PSMWorkload)."""
    name = "psm_sparse"
    env = {"SNB200_PSM_PATH": "sparse"}

    def describe(self):
        d = super().describe()
        d["workload"] += " -- sparse chain kernel forced (SNB200_PSM_PATH=sparse)"
        return d


class HMatWorkload(_DenseInputsMixin):
    """BASELINE config C4-H: HMatLayer 2048 -> 1000, eta 0.5, min block 2 => 2560 leaves of rank min(6, dim-1), batch 8192."""
    name, dtype, bound = "hmat", "f32", "hbm"
    input_dim, output_dim = 2048, 1000
    global_batch, cpu_sample_batch = 8192, 64
    bytes_per_sample_kernel = 4 * (2048 + 1000)
    bytes_per_sample = 2 * bytes_per_sample_kernel
    flop_per_sample = 2130000
    kernels = ("hmat_fwd_kernel", "hmat_bwd_kernel")

    def describe(self):
        return dict(workload="C4-H: H-matrix 2048->1000, eta 0.5, 2560 leaves (rank <= 6), fp32 fwd+bwd, batch 8192",
                    global_batch=self.global_batch, timed_inputs="resident in HBM")

    def hmatrix(self):
        from structurednets_b200.hmatrix import HMatrix, build_hmat_block_cluster_tree
        rng = np.random.default_rng(4000)
        tree = build_hmat_block_cluster_tree((1000, 2048), eta=0.5, min_block_size=2)
        for leaf in tree.get_all_leaf_elements():
            rows, cols = len(leaf.row_range), len(leaf.col_range)
            k = min(6, min(rows, cols) - 1)
            leaf.set_hmatrix_component(torch.tensor(rng.uniform(-1, 1, (rows, k)) / np.sqrt(k)).float(),
                                       torch.tensor(rng.uniform(-1, 1, (k, cols)) / np.sqrt(cols)).float())
        return HMatrix(tree, shape=(1000, 2048))

    def make_layer(self, device):
        from structurednets_b200.layers.hmat_layer import HMatLayer
        np.random.seed(4000)      # Glorot bias, as in SSSWorkload.make_layer
        return HMatLayer(self.input_dim, self.output_dim, 0.2, initial_hmatrix=self.hmatrix()).to(device)

    def ref_step_fn(self, batch, device="cpu"):
        from oracle import layers_cpu as O
        hm = self.hmatrix()
        comps = [(c.row_range.start, c.row_range.stop, c.col_range.start, c.col_range.stop, c.left_lr.detach().clone().to(device).requires_grad_(True),
                  c.right_lr.detach().clone().to(device).requires_grad_(True)) for c in hm.get_all_hmatrix_components() if c.are_low_rank_components_set()]
        b = torch.zeros(1000, device=device, requires_grad=True)
        x, gy = self._cpu_xy(batch, 4000, device)

        def step():
            for c in comps:
                c[4].grad = None; c[5].grad = None
            O.hmat_forward(x, comps, b, 1000).backward(gy)
        return step


class LDRWorkload(_DenseInputsMixin):
    """BASELINE config C4-L: LDRLayer 2048 -> 2048 (square only, SURVEY.md F1), share 0.1 => displacement rank 99, batch 8192."""
    name, dtype, bound = "ldr", "f64 Krylov recurrences + f32 (3xTF32) contractions", "tensor"
    tensor_bound = True
    input_dim, output_dim = 2048, 2048
    global_batch, cpu_sample_batch = 8192, 1024
    cpu_note = ("oracle float64 Krylov recurrence truncated at 48 powers (the dropped tail is below 1e-90 of the sum); the reference's "
                "literal matrix_power construction is O(r n^4 log n) and cannot run at n = 2048")
    bytes_per_sample_kernel = 4 * (2048 + 2048)
    bytes_per_sample = 2 * bytes_per_sample_kernel
    flop_per_sample = 16.8e6           # 2 n^2 apply + 2 n^2 weight gradient per sample; the batch-independent build is extra
    kernels = ("gemm_tf32x3_kernel", "gemm_tf32x3_kernel")

    def describe(self):
        return dict(workload="C4-L: LDR 2048->2048 (reference is square-only), displacement rank 99, batch 8192; the reference's own "
                             "construction is O(r n^4 log n) and cannot run at this size", global_batch=self.global_batch,
                    timed_inputs="resident in HBM")

    def make_layer(self, device):
        from structurednets_b200.layers.ldr_layer import LDRLayer
        np.random.seed(4100)
        layer = LDRLayer(2048, 2048, 0.1)
        assert layer.representation_matrices[2].shape[1] == 99
        return layer.to(device)

    def ref_step_fn(self, batch, device="cpu"):
        from oracle import layers_cpu as O
        np.random.seed(4100)
        from structurednets_b200.layers.ldr_layer import init_representation_matrices_torch
        rep = [m.detach().to(device).requires_grad_(True) for m in init_representation_matrices_torch((2048, 2048), 99)]
        b = torch.zeros(2048, device=device, requires_grad=True)
        x, gy = self._cpu_xy(batch, 4100, device)

        def step():
            for p in rep + [b]:
                p.grad = None
            O.ldr_forward(x, rep, b, (2048, 2048), nb_terms=48).backward(gy)
        return step


class SSSC1Workload(SSSWorkload):
    """BASELINE config C1: the same layer at batch 256 with the features in HOST numpy, through the reference's own call sites
    (training_helpers.get_batch -> model(X) -> CrossEntropyLoss -> backward, training_helpers.py:31-40,139-144)."""
    name = "sss_c1"
    global_batch = 256
    host_features = True

    def describe(self):
        return dict(workload="C1: SSS 4096->1000, 500 stages, statespace 16, fp32 fwd+bwd, batch 256, features in host numpy through get_batch "
                             "(H2D inside the timed region)", global_batch=256, timed_inputs="host numpy, copied per step like training_helpers.get_batch")


WORKLOADS = {"sss": SSSWorkload, "sss_c1": SSSC1Workload, "lr": LRWorkload, "lr_bf16": LRBf16Workload, "psm": PSMWorkload,
             "psm_sparse": PSMSparseWorkload, "hmat": HMatWorkload, "ldr": LDRWorkload}
# the configs of BASELINE.json reported next to the headline at N = 1 (config id -> workload)
SECONDARY = (("C1", "sss_c1"), ("C2", "lr_bf16"), ("C3", "psm"), ("C3_sparse_chain", "psm_sparse"), ("C4-H", "hmat"), ("C4-L", "ldr"))



# ----------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (recipe's clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.rows = []
        self._stop = threading.Event()
        self._thr = None

    def _run_nvml(self):
        """NVML (nvidia_ml_py) sampling every ~5 ms: the timed region of a fast workload is shorter than one nvidia-smi call."""
        import pynvml as N
        N.nvmlInit()
        h = N.nvmlDeviceGetHandleByIndex(self.gpu_index)
        mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
        bits = (("hw_slowdown", N.nvmlClocksThrottleReasonHwSlowdown), ("hw_thermal_slowdown", N.nvmlClocksThrottleReasonHwThermalSlowdown),
                ("sw_thermal_slowdown", N.nvmlClocksThrottleReasonSwThermalSlowdown), ("sw_power_cap", N.nvmlClocksThrottleReasonSwPowerCap))
        while not self._stop.is_set():
            sm = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
            r = N.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            try:
                pw = N.nvmlDeviceGetPowerUsage(h) / 1000.0
            except Exception:
                pw = 0.0
            self.rows.append([str(self.gpu_index), str(sm), str(mx), str(pw)] + ["Active" if (r & b) else "Not Active" for _, b in bits])
            self._stop.wait(0.005)

    def _run(self):
        try:
            self._run_nvml()
            return
        except Exception:
            pass
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thr.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


DUMP_BYTES = 64 * 2 ** 20


def step_outputs(runner, y):
    """What a caller of the timed step receives: the layer output and the parameter gradients (`grad_flat` is the buffer every dense
    float32 parameter's .grad is a view of, in named_parameters() order; the other parameters' gradients are listed by name)."""
    out = {"y": y}
    if runner.has_flat:
        out["grad_flat"] = runner.layer.flat_grad()
    loose = set(map(id, runner.loose))
    for name, p in runner.layer.named_parameters():
        if id(p) in loose and p.grad is not None:
            out["grad." + name] = p.grad
    return out


def dump_outputs(path, arrays):
    """Writes every tensor of `arrays` to path/<name>.npy, float64 as float64 and everything else as float32, DUMP_BYTES in all.
    An array larger than its equal share keeps a sample of its rows (of its entries if one row is too large) drawn from a fixed
    seed, so two runs with the same arguments store the same elements."""
    os.makedirs(path, exist_ok=True)
    share = (DUMP_BYTES - 4096 * len(arrays)) // len(arrays)      # 4 KB per file left for the .npy header
    for name, t in arrays.items():
        t = t.detach()
        t = t.to_dense() if t.is_sparse else t
        t = t if t.dtype == torch.float64 else t.float()
        if t.dim() == 0 or t[0].numel() * t.element_size() > share:
            t = t.reshape(-1)
        keep = share // (t[0].numel() * t.element_size())
        if t.shape[0] > keep:
            idx = np.sort(np.random.default_rng(0).choice(t.shape[0], keep, replace=False))
            t = t.index_select(0, torch.from_numpy(idx).to(t.device))
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def time_reference_steps(wl, steps, warmup, budget_s=25.0, device="cpu", batch=None):
    """The reference's own ops (oracle port) for this workload on `device`: host cores (cpu_baseline, --impl reference) or the same
    B200 (gpu_aten_baseline: what the reference's use_gpu=True runs)."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    B = batch or wl.cpu_sample_batch
    step = wl.ref_step_fn(B, device)
    sync = (lambda: torch.cuda.synchronize()) if str(device) != "cpu" else (lambda: None)
    for _ in range(warmup):
        step()
    sync()
    times = []
    t_start = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        sync()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s and len(times) >= 2:
            break
    med = float(np.median(times))
    if str(device) == "cpu":
        sample = "%d steps of batch %d (median %.1f ms/step) of the same layer on %s" % (len(times), B, med * 1e3, cpu_model())
        if getattr(wl, "cpu_note", None):
            sample += "; " + wl.cpu_note
        return dict(value=B / med, unit="samples/s", cores=cores, kind="port", sample=sample), med, len(times)
    return dict(value=B / med, unit="samples/s", kind="the reference's torch ops (oracle port) on CUDA tensors of the same B200, eager",
                sample="%d steps of batch %d (median %.2f ms/step, host-synchronised)" % (len(times), B, med * 1e3)), med, len(times)


# ----------------------------------------------------------------------------------------------
# the reference arm
# ----------------------------------------------------------------------------------------------
def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base, med, n = time_reference_steps(wl, steps=args.steps, warmup=max(args.warmup, 1), budget_s=float("inf"))
    cfg = wl.describe()
    cfg["sample_batch"] = wl.cpu_sample_batch
    line = dict(metric="structured-layer fwd+bwd samples/sec", value=base["value"], unit="samples/s", n_gpus=args.gpus, steps=n,
                warmup=max(args.warmup, 1), ms_per_step=med * 1e3, higher_is_better=True, scaling="strong", vs_baseline=None,
                dtype=wl.dtype, data="synthetic", config=cfg, impl="reference", cpu_baseline=base,
                e2e=dict(value=base["value"], unit="samples/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
class StepRunner:
    """One workload on one device: the layer, a ring of input sets (rotated so that consecutive timed steps never find their
    inputs in the 126 MB L2), and the step = zero grads, layer(x), y.backward(gy), optional gradient all-reduce."""

    def __init__(self, wl, device, local_batch, seed, grad_sync_factory=None):
        self.wl, self.device, self.local_batch = wl, device, local_batch
        for k, v in getattr(wl, "env", {}).items():
            os.environ[k] = v
        self.layer = wl.make_layer(device)
        x, gy, labels = wl.make_inputs(local_batch, device, seed=seed)
        set_bytes = x.numel() * x.element_size() + gy.numel() * gy.element_size()
        self.n_sets = int(min(8, max(1, -(-2 * L2_BYTES // set_bytes)))) if set_bytes < 2 * L2_BYTES else 1
        self.sets = [(x, gy, labels)]
        for k in range(1, self.n_sets):
            self.sets.append(wl.make_inputs(local_batch, device, seed=seed + 97 * k))
        self.l2_policy = ("inputs larger than L2 (%.0f MB per step)" % (set_bytes / 2 ** 20) if self.n_sets == 1 else
                          "%d input sets of %.0f MB rotated: consecutive steps never re-read a set that is still in the 126 MB L2" % (self.n_sets, set_bytes / 2 ** 20))
        self.has_flat = hasattr(self.layer, "flat_grad")
        if self.has_flat:
            self.layer.flat_grad()
        # parameters whose gradient does not live in the flat buffer (sparse / float64 ones): found once, not per step -- walking the
        # 3 501 parameter views of the SSS layer costs more host time than the kernels of a step leave
        self.loose = [p for p in self.layer.parameters() if not self.has_flat or p.is_sparse or p.dtype != torch.float32]
        self.grad_sync = grad_sync_factory(self.layer) if grad_sync_factory is not None else None
        self.stream = torch.cuda.current_stream()

    def restore_env(self):
        for k in getattr(self.wl, "env", {}):
            os.environ.pop(k, None)

    def zero_grads(self):
        if self.has_flat:
            self.layer.zero_flat_grad()
        for p in self.loose:
            p.grad = None

    def step(self, i=0, rec=None, inputs=None):
        x, gy, _ = inputs if inputs is not None else self.sets[i % self.n_sets]
        self.zero_grads()
        if rec is not None:
            rec[0].record(self.stream)
        y = self.layer(x)
        if rec is not None:
            rec[1].record(self.stream)
        y.backward(gy)
        if rec is not None:
            rec[2].record(self.stream)
        if self.grad_sync is not None:
            self.grad_sync()
        return y


def _ev():
    return torch.cuda.Event(enable_timing=True)


def _last_output(y, last):
    """The step's output if it is the last one, else None (freed before the next step allocates its own, as when it is dropped).
    Detached: a live autograd graph of an earlier step makes a later CUDA-graph capture fail (its backward would wait on
    uncaptured work)."""
    return y.detach() if last else None


def _capture(runner, n):
    """A CUDA graph of steps 0 .. n-1 and the output of its last step (kept alive, so replays refresh it)."""
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for k in range(n):
            y = _last_output(runner.step(k), k == n - 1)
    return graph, y


def measure(runner, steps, warmup, peaks, local_rank, barrier, use_graph=True, sustained_s=0.0, last_step=None):
    """Eager pass (per-kernel CUDA-event pairs recorded by the library around each of its launches) + CUDA-graph pass (the number
    reported), each of exactly `steps` steps.  Returns a dict; all times in ms, device-timed with CUDA events on the launching stream.
    `last_step(y)`, if given, is called with the output of the reported pass's last step while the layer's gradients are still
    that step's."""
    from structurednets_b200 import _lib
    wl, stream = runner.wl, runner.stream
    _lib.lib().sn_timing_enable(1)
    for i in range(max(warmup, 3)):
        runner.step(i)
    barrier()
    _lib.timing_report()                  # discard the warm-up launches (their events stay in the library's pool)
    _lib.reset_launch_count()
    recs = [(_ev(), _ev(), _ev()) for _ in range(steps)]
    t_begin, t_end = _ev(), _ev()
    with ClockSampler(local_rank) as clocks:
        barrier()
        t_begin.record(stream)
        for i in range(steps):
            y = _last_output(runner.step(i, recs[i]), i == steps - 1)
        t_end.record(stream)
        barrier()
    launches = _lib.launch_count()
    _lib.lib().sn_timing_enable(0)
    kernel_ms = _lib.timing_report()      # {kernel: (launches, total ms)} over the eager timed region
    eager_ms = t_begin.elapsed_time(t_end)
    fwd_ms = float(np.mean([r[0].elapsed_time(r[1]) for r in recs]))
    bwd_ms = float(np.mean([r[1].elapsed_time(r[2]) for r in recs]))
    out = dict(eager_ms_per_step=eager_ms / steps, fwd_ms=fwd_ms, bwd_ms=bwd_ms, launches=int(launches), steps=steps,
               kernel_ms=kernel_ms, eager_total_ms=eager_ms)
    elapsed_ms, timed_steps, graph_note, graph = eager_ms, steps, "eager launches", None
    if use_graph:   # multi-GPU: the NCCL all-reduce of the flat gradient is captured with the step
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                runner.step(0)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph, y = _capture(runner, runner.n_sets)
            # steps that are not a multiple of the input sets end with a graph of the first (steps mod n_sets) sets
            reps, rest = divmod(steps, runner.n_sets)
            tail = None
            if rest:
                tail, y = _capture(runner, rest)
            for _ in range(3):
                graph.replay()
                if tail is not None:
                    tail.replay()
            torch.cuda.synchronize()
            g0, g1 = _ev(), _ev()
            with ClockSampler(local_rank) as clocks:
                barrier()
                g0.record()
                for _ in range(reps):
                    graph.replay()
                if tail is not None:
                    tail.replay()
                g1.record()
                barrier()
            elapsed_ms = g0.elapsed_time(g1)
            graph_note = "CUDA graph of %d step(s) (one per input set), replayed %d times" % (runner.n_sets, reps)
            if tail is not None:
                graph_note += ", then a graph of the first %d" % rest
        except Exception as e:   # a layer whose step cannot be captured (host synchronisation inside) keeps the eager number
            torch.cuda.synchronize()
            graph = None
            graph_note = "eager launches (graph capture failed: %s)" % str(e).splitlines()[0][:120]
            if last_step is not None:   # the warm-up step above overwrote the gradients: the eager pass's last step once more
                y = runner.step(steps - 1).detach()
    if last_step is not None:
        last_step(y)
    out.update(elapsed_ms=elapsed_ms, timed_steps=timed_steps, launch_mode=graph_note, clocks=clocks.summary())
    if sustained_s > 0 and graph is not None:
        ms = elapsed_ms / timed_steps * runner.n_sets
        reps = max(1, int(sustained_s * 1e3 / ms) + 1)
        g0, g1 = _ev(), _ev()
        with ClockSampler(local_rank) as sclocks:
            barrier()
            g0.record()
            for _ in range(reps):
                graph.replay()
            g1.record()
            barrier()
        s_ms = g0.elapsed_time(g1)
        out["sustained"] = dict(ms_per_step=s_ms / (reps * runner.n_sets), steps=reps * runner.n_sets, seconds=s_ms / 1e3, clocks=sclocks.summary())
    return out


def roofline_of(wl, m, ms_per_step, local_batch, peaks):
    """Step-level and dominant-kernel roofline figures from a measure() result.  `frac` is the STEP fraction: SURVEY.md 8(d)'s
    algorithmic bytes per sample x samples / device time of the whole step, over the measured HBM copy bandwidth."""
    kernel_ms, eager_total = m["kernel_ms"], max(m["eager_total_ms"], 1e-9)
    per_kernel = {k: dict(launches=c, avg_ms=t / max(c, 1), share=t / eager_total) for k, (c, t) in kernel_ms.items()}
    dom = max(kernel_ms, key=lambda k: kernel_ms[k][1]) if kernel_ms else "n/a"
    dom_ms_per_step = (kernel_ms[dom][1] / m["steps"]) if kernel_ms else max(m["fwd_ms"], m["bwd_ms"])
    step_s = ms_per_step * 1e-3
    step_gbs = wl.bytes_per_sample * local_batch / step_s / 1e9
    tflops = wl.flop_per_sample * local_batch / step_s / 1e12
    kb = getattr(wl, "kernel_bytes_per_sample", {})
    dom_bytes = kb.get(dom)
    rl = dict(bound=wl.bound, achieved=step_gbs, peak=peaks["hbm_gbs"], unit="GB/s", frac=step_gbs / peaks["hbm_gbs"],
              frac_is="whole step: algorithmic bytes (SURVEY 8d, %d B/sample) x samples / step time / measured HBM copy bandwidth" % wl.bytes_per_sample,
              peak_source=peaks["source"], step_hbm_frac=step_gbs / peaks["hbm_gbs"], kernel=dom, kernel_ms_per_step=dom_ms_per_step,
              kernel_share=dom_ms_per_step * m["steps"] / eager_total, traffic=None, fwd_ms=m["fwd_ms"], bwd_ms=m["bwd_ms"], kernels=per_kernel,
              tflops=tflops, fp32_fma_frac_of_nominal=tflops / FP32_FMA_TFLOPS_NOMINAL,
              tolerance="fp32 parity tests: max-abs error / max-abs of the compared tensor < 1e-5, and RMS-relative < 1e-5 at config size "
                        "(tests/test_config_size_gpu.py); LDR 1e-4; bf16 2e-2")
    if dom_bytes is not None:
        g = dom_bytes * local_batch / (dom_ms_per_step * 1e-3) / 1e9
        rl.update(kernel_algorithmic_bytes_per_sample=dom_bytes, kernel_achieved=g, kernel_frac=g / peaks["hbm_gbs"])
    if getattr(wl, "traffic_bytes", None) and dom in wl.traffic_bytes and local_batch == getattr(wl, "traffic_batch", -1):
        rl.update(traffic=wl.traffic_bytes[dom], traffic_source=wl.traffic_source)
    if getattr(wl, "tensor_bound", False):
        rl.update(tensor_peak_tflops=peaks["bf16_tflops"], tensor_frac=tflops / peaks["bf16_tflops"],
                  tensor_frac_is="SURVEY 8d flop/sample x samples / step time / measured cuBLAS bf16 burst peak")
    return rl


def measure_c1(wl, device, local_rank, steps, warmup, peaks, barrier):
    """BASELINE C1 through the reference's call sites: host numpy features -> get_batch (torch.tensor + .to(device)) -> model ->
    CrossEntropyLoss -> backward, batch 256, wall-clock with a device synchronisation on both sides (H2D inside the timed region);
    next to it the same batch resident in HBM (graph replays)."""
    from structurednets_b200 import training_helpers as TH
    runner = StepRunner(wl, device, wl.global_batch, seed=1000)
    rng = np.random.default_rng(1000)
    nb = 16
    X = rng.uniform(-1, 1, size=(nb * 256, wl.input_dim)).astype(np.float32)
    y = rng.integers(0, wl.output_dim, size=(nb * 256,)).astype(np.int64)
    loss_fn = torch.nn.CrossEntropyLoss()

    def host_step(i):
        Xb, yb = TH.get_batch(X, y, batch_size=256, batch_i=i % nb, use_gpu=True)
        loss = loss_fn(runner.layer(Xb), target=yb)
        runner.zero_grads()
        loss.backward()
        return loss

    for i in range(max(warmup, 3)):
        host_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        host_step(i)
    barrier()
    host_s = (time.perf_counter() - t0) / steps
    m = measure(runner, steps, warmup, peaks, local_rank, barrier)
    ms = m["elapsed_ms"] / m["timed_steps"]
    res = dict(config=wl.describe(), value=256 / host_s, unit="samples/s", ms_per_step=host_s * 1e3,
               value_is="host features through get_batch, per-step pageable H2D + CrossEntropy + backward, wall clock (eager launches)",
               h2d_bytes_per_step=256 * wl.input_dim * 4 + 256 * 8,
               resident=dict(value=256 / (ms * 1e-3), ms_per_step=ms, launch_mode=m["launch_mode"], eager_ms_per_step=m["eager_ms_per_step"],
                             note="at 256 samples the step is launch- and latency-bound: it measures the batch-independent kernels, not bandwidth"),
               roofline=roofline_of(wl, m, ms, 256, peaks), gpu_launches=m["launches"], clocks=m["clocks"])
    runner.restore_env()
    return res


def measure_secondary(name, device, local_rank, steps, warmup, peaks, barrier, cpu=True):
    wl = WORKLOADS[name]()
    if getattr(wl, "host_features", False):
        res = measure_c1(wl, device, local_rank, steps, warmup, peaks, barrier)
    else:
        runner = StepRunner(wl, device, wl.global_batch, seed=5000)
        m = measure(runner, steps, warmup, peaks, local_rank, barrier)
        ms = m["elapsed_ms"] / m["timed_steps"]
        cfg = wl.describe()
        cfg.update(l2_policy=runner.l2_policy, launch_mode=m["launch_mode"], eager_ms_per_step=m["eager_ms_per_step"])
        res = dict(config=cfg, dtype=wl.dtype, value=wl.global_batch / (ms * 1e-3), unit="samples/s", ms_per_step=ms,
                   roofline=roofline_of(wl, m, ms, wl.global_batch, peaks), gpu_launches=m["launches"], clocks=m["clocks"])
        runner.restore_env()
        del runner
    if cpu and wl.cpu_sample_batch:
        res["cpu_baseline"] = time_reference_steps(wl, steps=3, warmup=0, budget_s=6.0)[0]
        try:
            res["gpu_aten_baseline"] = time_reference_steps(wl, steps=5, warmup=1, budget_s=4.0, device=device)[0]
        except Exception as e:
            res["gpu_aten_baseline"] = dict(unavailable=str(e).splitlines()[0][:160])
    torch.cuda.empty_cache()
    return res


def dp_check(runner, n_gpus, rank, device):
    """Numerics of the data-parallel step on the real ranks (NCCL): (1) after the all-reduce every rank holds bit-identical flat
    gradients; (2) on a 4 096-sample sub-batch (4 096 / N per rank) the all-reduced gradient equals the gradient ONE GPU computes
    for the union of the ranks' samples, to 1e-5 of its largest entry."""
    import torch.distributed as dist
    g = runner.layer.flat_grad()
    runner.step(0)
    torch.cuda.synchronize()
    gathered = [torch.empty_like(g) for _ in range(n_gpus)]
    dist.all_gather(gathered, g.clone())
    identical = all(bool(torch.equal(t, gathered[0])) for t in gathered)
    m = 4096 // n_gpus
    x, gy, labels = runner.sets[0]
    sub = (x[:m].contiguous(), gy[:m].contiguous(), labels[:m])
    runner.step(0, inputs=sub)
    torch.cuda.synchronize()
    g_dp = g.clone()
    xs = [torch.empty_like(sub[0]) for _ in range(n_gpus)]
    gys = [torch.empty_like(sub[1]) for _ in range(n_gpus)]
    dist.all_gather(xs, sub[0])
    dist.all_gather(gys, sub[1])
    sync, runner.grad_sync = runner.grad_sync, None
    runner.step(0, inputs=(torch.cat(xs), torch.cat(gys), None))     # every rank computes the union's gradient alone
    torch.cuda.synchronize()
    runner.grad_sync = sync
    ref = g.double()
    scale = float(ref.abs().max())
    err = float((g_dp.double() - ref).abs().max()) / max(scale, 1e-300)
    rms = float(((g_dp.double() - ref) ** 2).mean().sqrt() / (ref ** 2).mean().sqrt())
    flags = torch.tensor([1.0 if identical else 0.0, err, rms], device=device, dtype=torch.float64)
    dist.all_reduce(flags, op=dist.ReduceOp.MAX)
    worst = torch.tensor([1.0 if identical else 0.0], device=device, dtype=torch.float64)
    dist.all_reduce(worst, op=dist.ReduceOp.MIN)
    ok = bool(worst.item() == 1.0) and float(flags[1]) < 1e-5
    return ok, dict(all_ranks_identical=bool(worst.item() == 1.0), union_samples=m * n_gpus, union_max_rel_err=float(flags[1]),
                    union_rms_rel_err=float(flags[2]), tolerance=1e-5)


def run_ours(args, wl):
    import torch.distributed as dist
    from structurednets_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    _lib.lib()      # fails loudly when libsnb200.so is missing
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"
    n_gpus = world

    def barrier():
        if n_gpus > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peaks = measured_peaks()
    local_batch = wl.global_batch // n_gpus
    sync_factory = None
    if n_gpus > 1:
        from structurednets_b200.distributed import GradSynchronizer
        sync_factory = GradSynchronizer
    runner = StepRunner(wl, device, local_batch, seed=5000 + rank, grad_sync_factory=sync_factory)
    layer = runner.layer

    dp_ok, dp_detail = None, None
    if n_gpus > 1 and runner.has_flat:
        dp_ok, dp_detail = dp_check(runner, n_gpus, rank, device)

    grad_transport = runner.grad_sync.transport if (n_gpus > 1 and runner.grad_sync is not None and hasattr(runner.grad_sync, "transport")) else None
    last_step = None
    if args.dump_outputs and rank == 0:
        last_step = lambda y: dump_outputs(args.dump_outputs, step_outputs(runner, y))
    m = measure(runner, args.steps, args.warmup, peaks, local_rank, barrier, use_graph=not args.no_graph,
                sustained_s=2.5 if (n_gpus == 1 and not args.quick) else 0.0, last_step=last_step)
    elapsed_ms = m["elapsed_ms"]
    if n_gpus > 1:
        t = torch.tensor([elapsed_ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / m["timed_steps"]
    value = wl.global_batch / (ms_per_step * 1e-3)

    # ---- end to end through the module API with host buffers (pinned H2D + loss + D2H of the loss) ----
    x, gy, labels = runner.sets[0]
    e2e_steps = max(3, min(args.steps, 5))
    x_host = torch.empty((local_batch, wl.input_dim), dtype=x.dtype, pin_memory=True)
    x_host.copy_(x)
    labels_host = labels.cpu().pin_memory()
    loss_fn = torch.nn.CrossEntropyLoss()

    def e2e_step():
        xd = x_host.to(device, non_blocking=True)
        ld = labels_host.to(device, non_blocking=True)
        runner.zero_grads()
        loss = loss_fn(layer(xd).float(), ld)
        loss.backward()
        if runner.grad_sync is not None:
            runner.grad_sync()
        return float(loss.item())     # device -> host read of the step's result

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    if n_gpus > 1:
        t = torch.tensor([e2e_s], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e = dict(value=wl.global_batch / e2e_s, unit="samples/s", h2d_bytes_per_step=int(x_host.numel() * x_host.element_size() + labels_host.numel() * 8),
               d2h_bytes_per_step=4, steps=e2e_steps, ms_per_step=e2e_s * 1e3)

    if rank == 0:
        roofline = roofline_of(wl, m, ms_per_step, local_batch, peaks)
        cfg = wl.describe()
        cfg.update(local_batch=local_batch, parallelism="dp%d" % n_gpus, l2_policy=runner.l2_policy, launch_mode=m["launch_mode"],
                   eager_ms_per_step=m["eager_ms_per_step"])
        line = dict(metric="structured-layer fwd+bwd samples/sec", value=value, unit="samples/s", n_gpus=n_gpus, steps=m["timed_steps"],
                    warmup=max(args.warmup, 3), ms_per_step=ms_per_step, higher_is_better=True, scaling="strong", vs_baseline=None,
                    dtype=wl.dtype, data="synthetic", config=cfg, clocks=m["clocks"], e2e=e2e, gpu_launches=m["launches"], roofline=roofline)
        if "sustained" in m:
            s = m["sustained"]
            s["value"] = wl.global_batch / (s["ms_per_step"] * 1e-3)
            s["step_hbm_frac"] = wl.bytes_per_sample * local_batch / (s["ms_per_step"] * 1e-3) / 1e9 / peaks["hbm_gbs"]
            line["sustained"] = s
        if dp_ok is not None:
            line["dp_check"] = dp_ok
            line["dp_check_detail"] = dp_detail
        if grad_transport is not None:
            # "p2p": the one-shot all-reduce kernel of csrc/p2p.cu over NVLink peer memory; "nccl": torch.distributed.all_reduce
            line["config"]["grad_allreduce"] = grad_transport
        if n_gpus == 1 and not args.no_cpu_baseline and wl.cpu_sample_batch:
            line["cpu_baseline"] = time_reference_steps(wl, steps=20, warmup=1, budget_s=12.0)[0]
            try:
                line["gpu_aten_baseline"] = time_reference_steps(wl, steps=5, warmup=1, budget_s=5.0, device=device)[0]
            except Exception as e:
                line["gpu_aten_baseline"] = dict(unavailable=str(e).splitlines()[0][:160])
        else:
            line["cpu_baseline"] = None
        if n_gpus == 1 and args.workload == "sss" and not args.quick and not args.global_batch:
            del runner, layer, x, gy, labels, x_host
            torch.cuda.empty_cache()
            line["workloads"] = {}
            for cid, name in SECONDARY:
                try:
                    line["workloads"][cid] = measure_secondary(name, device, local_rank, min(args.steps, 20), args.warmup, peaks, barrier,
                                                               cpu=not args.no_cpu_baseline)
                except Exception as e:      # one broken secondary workload must not cost the headline line
                    line["workloads"][cid] = dict(error=str(e).splitlines()[0][:200])
        print(json.dumps(line))
    if n_gpus > 1:
        # a captured graph holds NCCL work; tearing the process group down underneath it can hang -- make sure every rank is
        # done, flush, and leave without running the destructors
        barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="sss", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of CUDA-graph replays")
    ap.add_argument("--quick", action="store_true", help="headline workload only: no sustained run, no secondary workloads (profiling)")
    ap.add_argument("--global-batch", type=int, default=None, help="profiling only: override the workload's global batch")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's output and parameter gradients to DIR/<name>.npy (rank 0's "
                         "shard; 64 MB in all, larger arrays as a fixed sample of their rows); inputs are seeded, so runs compare")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or getattr(WORKLOADS[args.workload], "host_features", False)):
        ap.error("--dump-outputs is for --impl ours on a workload with resident inputs")
    wl = WORKLOADS[args.workload]()
    if args.global_batch:
        wl.global_batch = args.global_batch
    if args.impl == "reference":
        run_reference(args, wl)
    elif getattr(wl, "host_features", False):
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device")
        torch.cuda.set_device(0)
        res = measure_c1(wl, torch.device("cuda", 0), 0, args.steps, args.warmup, measured_peaks(), torch.cuda.synchronize)
        print(json.dumps(res))
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
