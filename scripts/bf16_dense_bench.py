"""bf16 features against float32 features on the dense-product layers: one fwd+bwd step of the C3 (PSM), C4-H (H-matrix) and C4-L
(LDR) layers exactly as bench.py builds them, plus a Toeplitz-like layer at n = 2048.

    python scripts/bf16_dense_bench.py [--steps 50] [--repeats 3] [--out FILE]

Each arm is one captured CUDA graph of a whole step (gradients rebound inside the capture), timed with CUDA events around `--steps`
replays after a warm-up; the float32 and bf16 arms alternate in the same process, `--repeats` times, and the median and spread
(max - min) of the per-step times are reported.  PSM also runs at B = 256, where float32 features take the sparse chain: bf16
features always take the dense-product path, and this row shows what that costs at a small batch.

The error columns compare the bf16 path with the float32 CUDA path (pinned to the oracle at 1e-5) on the same bf16-rounded
features and output gradients: max |bf16 - fp32| / max |fp32| for y and for every parameter gradient.  The card's name, power limit
and maximum SM clock come from a read-only nvidia-smi query in the same run.  Prints one JSON line.
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

import bench  # noqa: E402  (only its workload definitions: layers, seeds and inputs)


class TLWorkload(bench._DenseInputsMixin):
    input_dim = output_dim = 2048

    def make_layer(self, device):
        from structurednets_b200.layers.tl_layer import TLLayer
        np.random.seed(6100)
        layer = TLLayer(2048, 2048, 0.008)      # displacement rank 8
        assert layer.G.shape[1] == 8
        return layer.to(device)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi query failed)"


def params_of(layer):
    return [(n, p) for n, p in layer.named_parameters() if p.requires_grad]


def step_fn(layer, x, gy):
    params = [p for _, p in params_of(layer)]

    def step():
        for p in params:
            p.grad = None
        y = layer(x)
        y.backward(gy)
        return y
    return step


def capture(step):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    return g


def time_ms(graph, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        graph.replay()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def grads(layer):
    out = {}
    for n, p in params_of(layer):
        g = p.grad
        out[n] = (g.to_dense() if g.is_sparse else g).detach().double().clone()
    return out


def errors(layer, xb, gyb):
    """bf16 path against the float32 CUDA path on the same bf16-rounded inputs."""
    y32 = step_fn(layer, xb.float(), gyb.float())().detach().double()
    g32 = grads(layer)
    y16 = step_fn(layer, xb, gyb)().detach().double()
    g16 = grads(layer)
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
    out = {"y": rel(y16, y32)}
    for n in g32:
        out["grad " + n] = rel(g16[n], g32[n])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    dev = torch.device("cuda")
    cases = [("C3 psm", bench.PSMWorkload(), 8192, 3000), ("C3 psm", bench.PSMWorkload(), 256, 3000), ("C4-H hmat", bench.HMatWorkload(), 8192, 4000),
             ("C4-L ldr", bench.LDRWorkload(), 8192, 4100), ("tl n=2048 r=8", TLWorkload(), 8192, 6100)]
    rows = []
    for name, wl, B, seed in cases:
        layer = wl.make_layer(dev)
        x, gy, _ = wl.make_inputs(B, dev, seed)
        xb, gyb = x.bfloat16(), gy.bfloat16()
        err = errors(layer, xb, gyb)
        graphs = {"fp32": capture(step_fn(layer, x, gy)), "bf16": capture(step_fn(layer, xb, gyb))}
        times = {"fp32": [], "bf16": []}
        for _ in range(args.repeats):
            for arm in ("fp32", "bf16"):
                times[arm].append(time_ms(graphs[arm], args.steps))
        row = dict(layer=name, batch=B)
        for arm in ("fp32", "bf16"):
            row[arm + "_ms_median"] = round(float(np.median(times[arm])), 4)
            row[arm + "_ms_spread"] = round(float(np.max(times[arm]) - np.min(times[arm])), 4)
        row["speedup"] = round(row["fp32_ms_median"] / row["bf16_ms_median"], 3)
        row["max_rel_err"] = {k: float("%.3g" % v) for k, v in err.items()}
        if len(row["max_rel_err"]) > 8:       # many-leaf layers: the largest error over the parameter gradients
            g = max(v for k, v in err.items() if k != "y")
            row["max_rel_err"] = {"y": float("%.3g" % err["y"]), "grad (max over %d parameters)" % (len(err) - 1): float("%.3g" % g)}
        rows.append(row)
        del graphs, layer, x, gy, xb, gyb
        torch.cuda.empty_cache()
    res = dict(card=card(), steps=args.steps, repeats=args.repeats, timing="CUDA events around graph replays of one fwd+bwd step", rows=rows)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
