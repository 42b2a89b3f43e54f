"""Cost of the input gradient on the PSM sparse chain, the H-matrix leaf kernels and the bf16 low-rank path.

    python scripts/input_grad_bench.py [--steps 50] [--repeats 5] [--out FILE]

Workloads (the layers of bench.py, each forced onto the path under test):
  psm_sparse_b256    C3 (PSM 4096 -> 1000, 3 factors, 409 599 non-zeros) on the sparse chain, B = 256 (the reference's training batch)
  psm_sparse_b8192   the same at B = 8192
  hmat_leaf_b8192    C4-H (H-matrix 2048 -> 1000, 2 560 leaves) on the leaf kernels, B = 8192
  lr_bf16_b8192      C2 (low rank 2048 -> 1000, rank 128) with bf16 features, B = 8192
One step is one forward and backward through the layer's autograd Function, in three arms:
  params        parameter and bias gradients only (the input does not need a gradient: what bench.py times)
  params+x      the same plus grad_x (a layer inside a network)
  x             grad_x only (every parameter frozen)
Each arm is a CUDA graph of one step, replayed `--steps` times between CUDA events; the arms alternate within each of `--repeats`
rounds in one process.  At B = 8192 the features, output gradient and grad_x exceed the 126 MB L2 for every layer but the bf16 one
(33 + 16 + 33 MB); no cache flush is added between replays.  The card's name, power limit and maximum SM clock come from a read-only
nvidia-smi query.  Prints one JSON line (median and spread = max - min over the rounds, ms per step).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

ARMS = {"params": (True, False), "params+x": (True, True), "x": (False, True)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi query failed)"


def workloads():
    import bench
    return {
        "psm_sparse_b256": (bench.PSMWorkload(), 256, {"SNB200_PSM_PATH": "sparse"}, torch.float32),
        "psm_sparse_b8192": (bench.PSMWorkload(), 8192, {"SNB200_PSM_PATH": "sparse"}, torch.float32),
        "hmat_leaf_b8192": (bench.HMatWorkload(), 8192, {"SNB200_HMAT_PATH": "leaf"}, torch.float32),
        "lr_bf16_b8192": (bench.LRWorkload(), 8192, {}, torch.bfloat16),
    }


def capture(layer, x, gy, params, want_x):
    """A CUDA graph of one fwd + bwd step of the arm (params: parameters take gradients; want_x: the input does)."""
    for p in layer.parameters():
        p.requires_grad_(params)
        p.grad = None
    x.requires_grad_(want_x)
    x.grad = None

    def step():
        layer(x).backward(gy)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(s)
    for p in layer.parameters():
        p.grad = None
    x.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for _ in range(5):
        graph.replay()
    return graph


def time_graph(graph, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    dev = torch.device("cuda")
    result = {"card": card(), "steps": a.steps, "repeats": a.repeats, "workloads": {}}
    for name, (wl, B, env, dtype) in workloads().items():
        os.environ.update(env)
        layer = wl.make_layer(dev)
        g = torch.Generator(device=dev).manual_seed(0)
        x = (torch.rand(B, wl.input_dim, device=dev, generator=g) * 2 - 1).to(dtype)
        gy = ((torch.rand(B, wl.output_dim, device=dev, generator=g) * 2 - 1) / B).to(dtype)
        graphs = {arm: capture(layer, x, gy, *flags) for arm, flags in ARMS.items()}
        times = {arm: [] for arm in ARMS}
        for _ in range(a.repeats):
            for arm, graph in graphs.items():
                times[arm].append(time_graph(graph, a.steps))
        row = {"B": B, "path": env or "bf16 features"}
        for arm, v in times.items():
            row[arm] = {"median_ms": round(float(np.median(v)), 4), "spread_ms": round(max(v) - min(v), 4)}
        row["grad_x_cost_ms"] = round(row["params+x"]["median_ms"] - row["params"]["median_ms"], 4)
        result["workloads"][name] = row
        for k in env:
            del os.environ[k]
        del graphs, layer, x, gy
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
