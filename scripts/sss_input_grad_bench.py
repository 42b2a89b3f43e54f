"""Cost of the input gradient on the SIMT SSS backward (csrc/sss.cu), and the SIMT backward without it against another build.

    python scripts/sss_input_grad_bench.py [--B 8192] [--steps 50] [--repeats 3] [--baseline-lib PATH] [--out FILE]

Two layers at B = 8192: C1 (4096 -> 1000, 500 stages, state dimension 16) forced onto the SIMT kernels, and the same shape with
state dimension 24, which is outside the tensor-core path's limits (its backward needs about 78 KB of shared memory per CTA; the
call checks this against the 227 KB limit).  One backward step is one sn_sss_backward call on the saved checkpoints of one forward:
  params        parameter and bias gradients (what training the layer alone needs)
  params+x      the same plus grad_x (a layer inside a network)
  x             grad_x only (frozen parameters)
Each arm is a CUDA graph of one call, replayed `--steps` times between CUDA events after a warm-up.  The inputs, checkpoints and
output gradient (about 290 MB at C1) exceed the 126 MB L2, so no cache flush is added between replays.

With --baseline-lib, the `params` arm also runs on that library (for example a build of the parent commit): each repeat runs one
child process per library, alternating, and the children report a hash of the parameter gradient so the two builds can be checked
to compute the same bits.  The card's name, power limit and maximum SM clock come from a read-only nvidia-smi query.  Prints one
JSON line (median and spread = max - min over the repeats, ms per step).
"""
import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

SHAPES = {"c1_simt": 16, "d24": 24}   # 4096 -> 1000, 500 stages, state dimension


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi query failed)"


def child(lib_path, B, steps, with_x):
    from structurednets_b200 import _lib
    from structurednets_b200.layers.sss_layer import SSSLayer
    from structurednets_b200.synth import random_mixed_system

    L = ctypes.CDLL(lib_path)
    _lib._declare(L)
    dev = torch.device("cuda")
    out = {}
    for name, d in SHAPES.items():
        np.random.seed(1001)
        layer = SSSLayer(4096, 1000, 0.105, nb_states=500, initial_system_approx=random_mixed_system(4096, 1000, 500, d, seed=1001)).to(dev)
        plan = layer._device_plan(dev)
        ps = ctypes.byref(plan["struct"])
        flat = layer.flat_parameters()
        packed = torch.empty(int(L.sn_sss_packed_floats(ps)), device=dev)
        _lib.check(L.sn_sss_pack(ps, _lib.ptr(flat), _lib.ptr(packed), _lib.stream_ptr()), "sn_sss_pack")
        g = torch.Generator(device=dev).manual_seed(0)
        x = torch.rand(B, 4096, device=dev, generator=g) * 2 - 1
        gy = (torch.rand(B, 1000, device=dev, generator=g) * 2 - 1) / B
        y = torch.empty(B, 1000, device=dev)
        ckpt = torch.empty(int(L.sn_sss_ckpt_floats(ps, B)), device=dev)
        _lib.check(L.sn_sss_forward(ps, _lib.ptr(packed), _lib.ptr(x), 4096, _lib.ptr(y), 1000, _lib.ptr(layer.bias), _lib.ptr(ckpt), B,
                                    _lib.stream_ptr()), "sn_sss_forward")
        ws = torch.empty(int(L.sn_sss_backward_workspace_floats(ps)), device=dev)
        gflat = torch.zeros_like(flat)
        gx = torch.empty(B, 4096, device=dev)

        def call(params, want_x):
            rc = L.sn_sss_backward(ps, _lib.ptr(packed), _lib.ptr(x), 4096, _lib.ptr(gy), 1000, _lib.ptr(ckpt),
                                   _lib.ptr(ws if params else None), _lib.ptr(gflat if params else None),
                                   _lib.ptr(gflat[:1000] if params else None), _lib.ptr(gx if want_x else None), 4096, B, _lib.stream_ptr())
            _lib.check(rc, "sn_sss_backward")

        arms = {"params": (True, False)}
        if with_x:
            arms.update({"params+x": (True, True), "x": (False, True)})
        res = {}
        for arm, (params, want_x) in arms.items():
            gflat.zero_()
            call(params, want_x)                      # the gradients of one step, hashed below
            torch.cuda.synchronize()
            if params:
                res[arm + ":grad_hash"] = hashlib.sha1(gflat.cpu().numpy().tobytes()).hexdigest()[:16]
            if want_x:
                res[arm + ":grad_x_hash"] = hashlib.sha1(gx.cpu().numpy().tobytes()).hexdigest()[:16]
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(3):
                    call(params, want_x)
            torch.cuda.current_stream().wait_stream(s)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                call(params, want_x)
            for _ in range(5):
                graph.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                graph.replay()
            e1.record()
            torch.cuda.synchronize()
            res[arm] = e0.elapsed_time(e1) / steps
            del graph
        out[name] = res
        del layer, x, gy, y, ckpt, ws, gflat, gx, packed
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=8192)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--baseline-lib", default=None)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child-lib", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--child-with-x", type=int, default=1, help=argparse.SUPPRESS)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    if a.child_lib:
        print(json.dumps(child(a.child_lib, a.B, a.steps, bool(a.child_with_x))))
        return
    from structurednets_b200 import _lib
    libs = [("this", _lib.LIB_PATH, 1)] + ([("baseline", os.path.abspath(a.baseline_lib), 0)] if a.baseline_lib else [])
    runs = {tag: [] for tag, _, _ in libs}
    for _ in range(a.repeats):
        for tag, path, with_x in libs:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--B", str(a.B), "--steps", str(a.steps), "--child-lib", path,
                                "--child-with-x", str(with_x)], capture_output=True, text=True)
            if r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
                raise SystemExit("child run on %s failed" % path)
            runs[tag].append(json.loads(r.stdout.strip().splitlines()[-1]))
    result = {"card": card(), "B": a.B, "steps": a.steps, "repeats": a.repeats, "shapes": {}}
    for shape in SHAPES:
        row = {}
        for tag in runs:
            for key in runs[tag][0][shape]:
                vals = [rr[shape][key] for rr in runs[tag]]
                if key.endswith("_hash"):
                    row["%s:%s" % (tag, key)] = vals[0] if len(set(vals)) == 1 else vals
                else:
                    row["%s:%s" % (tag, key)] = {"median_ms": round(float(np.median(vals)), 4), "spread_ms": round(max(vals) - min(vals), 4)}
        this = row["this:params"]["median_ms"]
        row["grad_x_cost_ms"] = round(row["this:params+x"]["median_ms"] - this, 4)
        if "baseline:params" in row:
            row["this_over_baseline_params"] = round(this / row["baseline:params"]["median_ms"], 4)
            row["same_param_grads_as_baseline"] = row["this:params:grad_hash"] == row["baseline:params:grad_hash"]
        row["params_grads_unchanged_by_grad_x"] = row["this:params:grad_hash"] == row["this:params+x:grad_hash"]
        row["grad_x_same_with_and_without_params"] = row["this:params+x:grad_x_hash"] == row["this:x:grad_x_hash"]
        result["shapes"][shape] = row
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
