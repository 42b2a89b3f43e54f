"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): the reference's own C implementation of the SSS forward as a second,
torch-independent checker.

``speed_comparison/run.c`` (reference :123-368) reads ``layer_description.txt`` (written by ``prepare_run.py:10-31,53-82``),
evaluates a dense layer and the SSS layer for one input vector with plain C loops and compares both results with the "checksum"
vectors stored in the file (absolute tolerance 1e-3, run.c:177,357), exiting non-zero on a mismatch.  Here the file is written from
OUR layer's parameters with the checksum output taken from the path under test (the numpy/torch oracle, or the CUDA kernels through
the C ABI), so run.c acts as the judge.  The binary is compiled from the reference's source where it lies (never copied) into
``oracle/_ref/run`` by ``build_ref()`` / ``make -C oracle``; it travels to the GPU box, ``/root/reference`` does not.
"""
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# SNB200_REFERENCE: a checkout of MatthiasKi/structurednets
REF_SRC = (os.path.join(os.environ["SNB200_REFERENCE"], "src/structurednets/speed_comparison/run.c")
           if os.environ.get("SNB200_REFERENCE") else None)
REF_BIN = os.path.join(HERE, "_ref", "run")


def build_ref(force: bool = False):
    """gcc on the reference's run.c (its own header says ``gcc -o run run.c``, run.c:10).  Returns the binary path or None."""
    if os.path.exists(REF_BIN) and not force:
        return REF_BIN
    if REF_SRC is None or not os.path.exists(REF_SRC):
        return None
    os.makedirs(os.path.dirname(REF_BIN), exist_ok=True)
    subprocess.run(["gcc", "-O1", "-o", REF_BIN, REF_SRC, "-lm"], check=True, capture_output=True)
    return REF_BIN


def _mat(f, name, m):
    m = np.asarray(m, dtype=np.float32)
    if m.ndim == 1:
        m = m.reshape(1, -1)
    f.write("%s %d %d\n" % (name, m.shape[0], m.shape[1]))            # prepare_run.py:14-22
    for row in m:
        f.write(",".join("%.9g" % v for v in row) + "\n")


def _vec(f, name, v):
    v = np.asarray(v, dtype=np.float32).reshape(-1)
    f.write("%s %d\n" % (name, len(v)))                               # prepare_run.py:24-31
    f.write(",".join("%.9g" % x for x in v) + "\n")


def write_layer_description(path, A, B, C, D, E, F, G, sss_bias, checksum_inp, sss_checksum_out, W=None, standard_bias=None):
    """File layout of prepare_run.py:53-82.  ``W`` / ``standard_bias`` describe the dense layer run.c also checks; by default the
    zero matrix, so its checksum is the bias."""
    A, B, C, D, E, F, G = [[np.asarray(m, dtype=np.float32) for m in l] for l in (A, B, C, D, E, F, G)]
    n_in = sum(m.shape[1] for m in B)
    n_out = sum(m.shape[0] for m in D)
    checksum_inp = np.asarray(checksum_inp, dtype=np.float32).reshape(1, n_in)
    if W is None:
        W = np.zeros((n_out, n_in), dtype=np.float32)
    if standard_bias is None:
        standard_bias = np.zeros(n_out, dtype=np.float32)
    standard_out = (np.asarray(W, dtype=np.float64) @ checksum_inp.reshape(-1).astype(np.float64) + np.asarray(standard_bias, dtype=np.float64))
    with open(path, "w") as f:
        f.write("input_size %d\noutput_size %d\n" % (n_in, n_out))
        _mat(f, "checksum_inp", checksum_inp)
        _mat(f, "W", W)
        _vec(f, "standard_bias", standard_bias)
        _vec(f, "standard_checksum_out", standard_out)
        f.write("nb_states %d\n" % len(A))
        f.write("max_state_space_dim %d\n" % max(1, max(max(m.shape) for m in A + E)))
        f.write("max_input_dim %d\n" % max(1, max(m.shape[1] for m in B)))
        f.write("max_output_dim %d\n" % max(1, max(m.shape[0] for m in D)))
        for name, mats in (("A", A), ("B", B), ("C", C), ("D", D), ("E", E), ("F", F), ("G", G)):
            for k, m in enumerate(mats):
                _mat(f, "%s_%d" % (name, k), m)
        _vec(f, "sss_bias", sss_bias)
        _mat(f, "sss_checksum_out", np.asarray(sss_checksum_out, dtype=np.float32).reshape(1, n_out))


def run_reference_check(A, B, C, D, E, F, G, sss_bias, checksum_inp, sss_checksum_out):
    """Runs the reference binary on a description of this layer.  Returns (accepted, stdout): accepted is True when run.c's own
    checksum tests pass (exit code 0 and no ERROR line), i.e. when ``sss_checksum_out`` equals run.c's SSS forward within 1e-3."""
    binary = build_ref()
    if binary is None:
        raise FileNotFoundError("oracle/_ref/run is not built and the reference source is not present")
    with tempfile.TemporaryDirectory() as tmp:
        write_layer_description(os.path.join(tmp, "layer_description.txt"), A, B, C, D, E, F, G, sss_bias, checksum_inp, sss_checksum_out)
        r = subprocess.run([binary], cwd=tmp, capture_output=True, text=True, timeout=300)
    return (r.returncode == 0 and "ERROR" not in r.stdout and "sss_time" in r.stdout), r.stdout
