"""SSS (sequentially semiseparable / time-varying state-space) layer on B200.

Drop-in for ``structurednets.layers.sss_layer.SSSLayer`` (reference layers/sss_layer.py:35-137): same
constructor, same ``ParameterList`` names ``A..G`` and shapes (so the same ``state_dict`` keys
``bias, A.0 .. G.{n-1}``), same ``statespace_dim`` budget rule and the same module-level helpers
(``get_nb_parameters``, ``get_max_statespace_dim``, ``standard_dims_in_dims_out_computation``).
``forward`` + autograd backward run in hand-written sm_100a kernels through the C ABI (include/snb200.h): the tensor-core path of
``csrc/sss_tc.cu`` (``sn_sss_tc_build / sn_sss_tc_forward / sn_sss_tc_backward``: chunked 3xTF32 formulation, DESIGN.md section 4.1) for
layers inside its limits (state dimensions <= 16, <= 16 outputs and <= 160 inputs per stage, input and output dimensions multiples of 4),
the SIMT kernels of ``csrc/sss.cu`` (``sn_sss_pack / sn_sss_forward / sn_sss_backward``) for everything else; ``SNB200_SSS_PATH=tc|simt``
forces one.  There is no CPU path.
"""
import ctypes
import os
import pickle

import numpy as np
import torch
import torch.nn as nn

from structurednets_b200 import _lib
from structurednets_b200.layers.flat_params import FlatParamsMixin
from structurednets_b200.layers.layer_helpers import get_random_glorot_uniform_matrix
from structurednets_b200.layers.structured_layer import StructuredLayer

SSS_CHUNK_LEN = 4  # stages between two state checkpoints (forward saves them, backward recomputes inside)


def get_nb_parameters(optim_mat_shape: tuple, statespace_dim: int, nb_states: int) -> int:
    """Upper-bound parameter count, reference layers/sss_layer.py:15-24."""
    dims_in, dims_out = standard_dims_in_dims_out_computation(input_size=optim_mat_shape[1], output_size=optim_mat_shape[0], nb_states=nb_states)
    nb_params = 0
    for state_i, (inp_dim, out_dim) in enumerate(zip(dims_in, dims_out)):
        if state_i > 0 and state_i < len(dims_in) - 1:
            nb_params += 2 * statespace_dim * statespace_dim
        nb_params += 2 * inp_dim * statespace_dim
        nb_params += 2 * statespace_dim * out_dim
        nb_params += inp_dim * out_dim
    return int(nb_params)


def has_less_parameters_than_allowed(optim_mat: np.ndarray, nb_params_share: float, nb_states: int, state_space_dim: int) -> bool:
    return get_nb_parameters(optim_mat_shape=optim_mat.shape, statespace_dim=state_space_dim, nb_states=nb_states) < int(nb_params_share * optim_mat.size)


def get_max_statespace_dim(optim_mat: np.ndarray, nb_params_share: float, nb_states: int) -> int:
    """Largest statespace_dim whose upper-bound count fits the budget, reference layers/sss_layer.py:26-33."""
    state_space_dim = 0
    while has_less_parameters_than_allowed(optim_mat=optim_mat, nb_params_share=nb_params_share, nb_states=nb_states, state_space_dim=state_space_dim + 1):
        state_space_dim += 1
    return state_space_dim


def standard_dims_in_dims_out_computation(input_size: int, output_size: int, nb_states: int):
    """reference layers/sss_layer.py:139-146"""
    dims_in = int(input_size / nb_states) * np.ones((nb_states,), dtype='int32')
    dims_in[:(input_size - np.sum(dims_in))] += 1
    assert np.sum(dims_in) == input_size, "Sum over input dimensions does not match the input size"
    dims_out = int(output_size / nb_states) * np.ones((nb_states,), dtype='int32')
    dims_out[:(output_size - np.sum(dims_out))] += 1
    assert np.sum(dims_out) == output_size, "Sum over output dimensions does not match the output size"
    return dims_in, dims_out


def _identify_system(T_full: np.ndarray, dims_in, dims_out, statespace_dim: int, device=None):
    """The state-space realisation of a dense matrix: tvsclib's Hankel-SVD identification when it is installed (the reference
    constructor, layers/sss_layer.py:66-68; a git-only, unpinned dependency, reference setup.py:33), otherwise this package's own
    implementation of the same method (structurednets_b200/sss_identification.py).  Either result is a valid realisation --
    they agree up to a state-space similarity, which no reference test pins (SURVEY.md section 8c)."""
    try:
        from tvsclib.mixed_system import MixedSystem
        from tvsclib.toeplitz_operator import ToeplitzOperator
        from tvsclib.system_identification_svd import SystemIdentificationSVD
    except ImportError:
        from structurednets_b200.sss_identification import identify_mixed_system
        return identify_mixed_system(T_full, dims_in, dims_out, statespace_dim, device=device)
    T_operator = ToeplitzOperator(T_full, dims_in, dims_out)
    S = SystemIdentificationSVD(toeplitz=T_operator, max_states_local=statespace_dim)
    return MixedSystem(S)


def _param_version(layer):
    """Version counters that every way of updating the parameters bumps: the flat buffer's (FlatSGD / FlatAdam write it through the
    library and bump it by hand) and those of the first and last parameter (the views do not share the buffer's counter; torch
    optimizers update every parameter in place)."""
    flat = layer.__dict__.get("_flat")
    params = layer._flat_param_list()
    return (flat._version if flat is not None else -1, params[0]._version if params else -1, params[-1]._version if params else -1)


def _check_params_unchanged(ctx, layer):
    """The kernels read the layer-wide coefficient / packed-parameter buffers and the CURRENT flat parameters in backward, not copies
    saved per forward.  That is exact as long as the parameters are the ones the forward saw; an optimizer step (or any other in-place
    write) between a forward and its backward would silently give gradients at the wrong point, so it raises like autograd does for
    saved tensors that were modified in place."""
    if _param_version(layer) != ctx.param_version:
        raise RuntimeError("SSSLayer: the parameters were modified in place between this forward and its backward (an optimizer step or "
                           "a parameter write after the forward); run backward before updating the parameters, or run the forward again")


class _SSSFunction(torch.autograd.Function):
    """fwd: sn_sss_forward (saves chunk-entry state checkpoints); bwd: sn_sss_backward accumulating
    straight into the layer's flat gradient buffer (every ``p.grad`` is a view of it) and / or returning
    the gradient w.r.t. the input features.

    ``anchor`` is passed (a leaf that requires grad) when the parameters take gradients; ``save`` when a
    backward can run at all (parameters or ``U`` need a gradient).  Grad mode is always off inside
    Function.forward, so the layer decides both."""

    @staticmethod
    def forward(ctx, U, anchor, layer, save):
        B = U.shape[0]
        plan = layer._device_plan(U.device)
        packed = layer._packed_params(plan)
        y = torch.empty((B, layer.output_dim), dtype=torch.float32, device=U.device)
        ckpt = None
        if save:
            nck = _lib.lib().sn_sss_ckpt_floats(ctypes.byref(plan["struct"]), B)
            ckpt = torch.empty(max(int(nck), 1), dtype=torch.float32, device=U.device)
        bias = layer.bias if layer.use_bias else None
        rc = _lib.lib().sn_sss_forward(ctypes.byref(plan["struct"]), _lib.ptr(packed), _lib.ptr(U), U.stride(0),
                                       _lib.ptr(y), y.stride(0), _lib.ptr(bias), _lib.ptr(ckpt), B, _lib.stream_ptr())
        _lib.check(rc, "sn_sss_forward")
        ctx.layer = layer
        ctx.plan = plan
        ctx.param_grad = anchor is not None
        ctx.param_version = _param_version(layer)
        ctx.save_for_backward(U, ckpt, packed)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        layer, plan = ctx.layer, ctx.plan
        _check_params_unchanged(ctx, layer)
        U, ckpt, packed = ctx.saved_tensors
        grad_x = torch.empty_like(U) if ctx.needs_input_grad[0] else None
        grad_y = grad_y.contiguous()
        if grad_y.dtype != torch.float32:
            grad_y = grad_y.float()
        g = layer._prepare_grad_accumulation() if ctx.param_grad else None
        gbias = g[:layer.output_dim] if (g is not None and layer.use_bias and layer.bias.requires_grad) else None
        ws = layer._backward_workspace(plan) if g is not None else None
        rc = _lib.lib().sn_sss_backward(ctypes.byref(plan["struct"]), _lib.ptr(packed), _lib.ptr(U), U.stride(0),
                                        _lib.ptr(grad_y), grad_y.stride(0), _lib.ptr(ckpt), _lib.ptr(ws), _lib.ptr(g), _lib.ptr(gbias),
                                        _lib.ptr(grad_x), grad_x.stride(0) if grad_x is not None else 0, U.shape[0], _lib.stream_ptr())
        _lib.check(rc, "sn_sss_backward")
        return grad_x, None, None, None


class _SSSTCFunction(torch.autograd.Function):
    """Tensor-core path (csrc/sss_tc.cu): sn_sss_tc_build + sn_sss_tc_forward, sn_sss_tc_backward.  Arguments as _SSSFunction."""

    @staticmethod
    def forward(ctx, U, anchor, layer, save):
        B = U.shape[0]
        L = _lib.lib()
        tc = layer._tc_plan(U.device)
        ps = ctypes.byref(tc["struct"])
        flat = layer.__dict__["_flat"]
        coef = tc["coef"]
        _lib.check(L.sn_sss_tc_build(ps, _lib.ptr(flat), _lib.ptr(coef), _lib.stream_ptr()), "sn_sss_tc_build")
        y = torch.empty((B, layer.output_dim), dtype=torch.float32, device=U.device)
        nr = int(L.sn_sss_tc_rbuf_floats(ps, B))     # 0 when the fused large-batch forward runs
        rbuf = torch.empty(nr, dtype=torch.float32, device=U.device) if nr else None
        states = torch.empty(max(int(L.sn_sss_tc_states_floats(ps, B)), 1), dtype=torch.float32, device=U.device)
        bias = layer.bias if layer.use_bias else None
        rc = L.sn_sss_tc_forward(ps, _lib.ptr(coef), _lib.ptr(U), U.stride(0), _lib.ptr(y), y.stride(0), _lib.ptr(bias),
                                 _lib.ptr(rbuf), _lib.ptr(states), B, _lib.stream_ptr())
        _lib.check(rc, "sn_sss_tc_forward")
        ctx.layer = layer
        ctx.tc = tc
        ctx.param_grad = anchor is not None
        ctx.param_version = _param_version(layer)
        if save:
            ctx.save_for_backward(U, states)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        layer, tc = ctx.layer, ctx.tc
        _check_params_unchanged(ctx, layer)
        U, states = ctx.saved_tensors
        grad_x = torch.empty_like(U) if ctx.needs_input_grad[0] else None
        grad_y = grad_y.contiguous()
        if grad_y.dtype != torch.float32:
            grad_y = grad_y.float()
        L = _lib.lib()
        ps = ctypes.byref(tc["struct"])
        B = U.shape[0]
        g = layer._prepare_grad_accumulation() if ctx.param_grad else None
        gbias = g[:layer.output_dim] if (g is not None and layer.use_bias and layer.bias.requires_grad) else None
        ws = torch.empty(max(int(L.sn_sss_tc_backward_workspace_floats(ps, B)), 1), dtype=torch.float32, device=U.device)
        # tc["coef"] still holds the chunk matrices of the forward (rebuilt at every forward from the flat parameters)
        rc = L.sn_sss_tc_backward(ps, _lib.ptr(layer.__dict__["_flat"]), _lib.ptr(tc["coef"]), _lib.ptr(U), U.stride(0),
                                  _lib.ptr(grad_y), grad_y.stride(0), _lib.ptr(states), _lib.ptr(ws), _lib.ptr(g), _lib.ptr(gbias),
                                  _lib.ptr(grad_x), grad_x.stride(0) if grad_x is not None else 0, B, _lib.stream_ptr())
        _lib.check(rc, "sn_sss_tc_backward")
        return grad_x, None, None, None


class SSSLayer(FlatParamsMixin, StructuredLayer):
    def __init__(self, input_dim: int, output_dim: int, nb_params_share: float, use_bias=True, initial_weight_matrix=None,
                 initial_bias=None, nb_states=None, initial_system_approx=None, use_gpu=False):
        super(SSSLayer, self).__init__(input_dim=input_dim, output_dim=output_dim, nb_params_share=nb_params_share,
                                       use_bias=use_bias, initial_weight_matrix=initial_weight_matrix, initial_bias=initial_bias)

        if nb_states is None:
            nb_states = int(min(input_dim, output_dim) / 2)
        assert nb_states > 0, "Nb states must be positive"

        assert initial_weight_matrix is None or initial_system_approx is None, "Either pass an initial weight matrix or the initial system approximation - not both"
        if initial_system_approx is not None:
            assert len(initial_system_approx.dims_in) == nb_states, "The given system approximation does not match the expected number of states (dims_in)"
            assert len(initial_system_approx.dims_out) == nb_states, "The given system approximation does not match the expected number of states (dims_out)"

        self.input_dim = input_dim
        self.nb_states = nb_states

        self.use_gpu = use_gpu
        self.init_state_matrices(nb_params_share=nb_params_share, initial_weight_matrix=initial_weight_matrix, initial_system_approx=initial_system_approx)
        self._flatten_parameters()

    def init_state_matrices(self, nb_params_share: float, initial_weight_matrix=None, initial_system_approx=None):
        """reference layers/sss_layer.py:54-91"""
        if initial_weight_matrix is None:
            T_full = get_random_glorot_uniform_matrix(shape=(self.output_dim, self.input_dim))
        else:
            T_full = initial_weight_matrix

        self.statespace_dim = get_max_statespace_dim(T_full, nb_params_share=nb_params_share, nb_states=self.nb_states)

        if has_less_parameters_than_allowed(optim_mat=T_full, nb_params_share=nb_params_share, nb_states=self.nb_states, state_space_dim=self.statespace_dim):
            self.dims_in, self.dims_out = standard_dims_in_dims_out_computation(input_size=self.input_dim, output_size=self.output_dim, nb_states=self.nb_states)

            if initial_system_approx is None:
                # use_gpu also moves the Hankel SVDs of the initialisation to the GPU (cuSOLVER, float64)
                svd_device = "cuda" if (getattr(self, "use_gpu", False) and torch.cuda.is_available()) else None
                system_approx = _identify_system(T_full, self.dims_in, self.dims_out, self.statespace_dim, device=svd_device)
            else:
                system_approx = pickle.loads(pickle.dumps(initial_system_approx))

            self.initial_weight_matrix = system_approx.to_matrix()

            A = [stage.A_matrix for stage in system_approx.causal_system.stages]
            B = [stage.B_matrix for stage in system_approx.causal_system.stages]
            C = [stage.C_matrix for stage in system_approx.causal_system.stages]
            D = [stage.D_matrix for stage in system_approx.causal_system.stages]
            E = [stage.A_matrix for stage in system_approx.anticausal_system.stages]
            F = [stage.B_matrix for stage in system_approx.anticausal_system.stages]
            G = [stage.C_matrix for stage in system_approx.anticausal_system.stages]

            mk = lambda mats: nn.ParameterList([nn.Parameter(torch.tensor(np.asarray(m)).float(), requires_grad=True) for m in mats])
            self.A, self.B, self.C, self.D, self.E, self.F, self.G = mk(A), mk(B), mk(C), mk(D), mk(E), mk(F), mk(G)

            self.state_matrices_initialized = True

    def get_input_index_range_according_to_state(self, state_i):
        return range(np.sum(self.dims_in[:state_i]), np.sum(self.dims_in[:state_i + 1]))

    def get_output_index_range_according_to_state(self, state_i):
        return range(np.sum(self.dims_out[:state_i]), np.sum(self.dims_out[:state_i + 1]))

    # ---- device plan --------------------------------------------------------------------------
    def _on_reflatten(self):
        self.__dict__["_dev_plan"] = None
        self.__dict__["_dev_packed"] = None
        self.__dict__["_dev_packed_version"] = None
        self.__dict__["_dev_bwd_ws"] = None
        self.__dict__["_dev_tc_plan"] = None
        self.__dict__["_tc_eligible"] = None

    def _param_offsets(self):
        """{(list name, k): offset in the flat buffer}; flat order = named_parameters() order."""
        offs = {}
        params = self._flat_param_list()
        by_id = {id(p): o for p, o in zip(params, self.__dict__["_flat_offsets"])}
        for name in "ABCDEFG":
            for k, p in enumerate(getattr(self, name)):
                offs[(name, k)] = by_id[id(p)]
        return offs

    def build_host_plan(self, chunk_len: int = SSS_CHUNK_LEN):
        """Stage and chunk tables of include/snb200.h (sn_sss_stage / sn_sss_chunk) as numpy int32."""
        n = self.nb_states
        offs = self._param_offsets()
        in_off = np.concatenate([[0], np.cumsum(self.dims_in)]).astype(np.int64)
        out_off = np.concatenate([[0], np.cumsum(self.dims_out)]).astype(np.int64)
        stages = np.zeros((2, n, 16), dtype=np.int32)
        for k in range(n):
            a, b, c, d = self.A[k], self.B[k], self.C[k], self.D[k]
            e, f, g = self.E[k], self.F[k], self.G[k]
            assert a.shape[1] == c.shape[1] and a.shape[0] == b.shape[0], "inconsistent causal stage shapes"
            assert e.shape[1] == g.shape[1] and e.shape[0] == f.shape[0], "inconsistent anticausal stage shapes"
            stages[0, k, :12] = [in_off[k], self.dims_in[k], out_off[k], self.dims_out[k], a.shape[1], a.shape[0],
                                 offs[("C", k)], offs[("D", k)], offs[("A", k)], offs[("B", k)], 0, k]
            kk = n - 1 - k
            stages[1, kk, :12] = [in_off[k], self.dims_in[k], out_off[k], self.dims_out[k], e.shape[1], e.shape[0],
                                  offs[("G", k)], -1, offs[("E", k)], offs[("F", k)], 0, k]
        for d in range(2):
            for kk in range(n):
                if kk > 0:
                    assert stages[d, kk, 4] == stages[d, kk - 1, 5], "state dimensions of consecutive stages do not chain"
                else:
                    assert stages[d, 0, 4] == 0, "the first stage of a sweep must have an empty incoming state"
        rows = stages[:, :, 3] + stages[:, :, 5]
        ks = stages[:, :, 1] + stages[:, :, 4]
        ru4 = lambda v: int(max(4, (int(v) + 3) // 4 * 4))
        rows_pad, k_pad = ru4(rows.max()), ru4(ks.max())
        d_pad = ru4(max(stages[:, :, 4].max(), stages[:, :, 5].max()))
        blk = 8 + 2 * rows_pad * k_pad   # 8-float descriptor header + Pt + P (csrc/sss.cu)
        for d in range(2):
            for kk in range(n):
                stages[d, kk, 10] = (d * n + kk) * blk
        # chunks: never straddle the first-visit / second-visit switch
        h = n // 2
        first_visit = [h, n - h]
        chunks = [[], []]
        for d in range(2):
            bounds = []
            for lo, hi, second in ((0, first_visit[d], 0), (first_visit[d], n, 1)):
                s = lo
                while s < hi:
                    e_ = min(s + chunk_len, hi)
                    bounds.append((s, e_, second))
                    s = e_
            for (s, e_, second) in bounds:
                st = stages[d, s:e_]
                col0 = int(st[:, 0].min())
                ncols = int(st[:, 1].sum())
                row0 = int(st[:, 2].min())
                nrows = int(st[:, 3].sum())
                mid = s + (e_ - s + 1) // 2
                sa, sb = stages[d, s:mid], stages[d, mid:e_]
                col0_a, ncols_a = int(sa[:, 0].min()), int(sa[:, 1].sum())
                col0_b, ncols_b = (int(sb[:, 0].min()), int(sb[:, 1].sum())) if len(sb) else (col0_a, 0)
                chunks[d].append([s, e_, col0, ncols, row0, nrows, second, mid, col0_a, ncols_a, col0_b, ncols_b, 0, 0, 0, 0])
        assert len(chunks[0]) == len(chunks[1])
        chunks = np.asarray(chunks, dtype=np.int32)
        meta = dict(nb_states=n, input_dim=self.input_dim, output_dim=self.output_dim, rows_pad=rows_pad, k_pad=k_pad,
                    d_pad=d_pad, nchunks=chunks.shape[1], chunk_in_max=int(chunks[:, :, 3].max()),
                    chunk_out_max=int(max(1, chunks[:, :, 5].max())), chunk_len_max=int((chunks[:, :, 1] - chunks[:, :, 0]).max()),
                    nparams=int(self.__dict__["_flat_total"]), half_in_max=int(max(chunks[:, :, 9].max(), chunks[:, :, 11].max())))
        return stages, chunks, meta

    def _device_plan(self, device):
        self._ensure_flat()
        plan = self.__dict__.get("_dev_plan")
        if plan is not None and plan["device"] == device:
            return plan
        stages, chunks, meta = self.build_host_plan()
        st_dev = torch.from_numpy(stages.reshape(-1)).to(device)
        ch_dev = torch.from_numpy(chunks.reshape(-1)).to(device)
        struct = _lib.SnSssPlan()
        for k, v in meta.items():
            setattr(struct, k, v)
        struct.stages = st_dev.data_ptr()
        struct.chunks = ch_dev.data_ptr()
        plan = dict(device=device, struct=struct, stages=st_dev, chunks=ch_dev, meta=meta)
        self.__dict__["_dev_plan"] = plan
        self.__dict__["_dev_packed"] = None
        return plan

    # ---- tensor-core plan (csrc/sss_tc.cu) -------------------------------------------------------
    TC_DS, TC_PO, TC_KB, TC_KB_MAX, TC_LMAX, TC_SOUT_MAX = 16, 32, 32, 5, 16, 16

    def build_tc_host_plan(self):
        """Chunk table of include/snb200.h (sn_sss_tc_chunk) or None when the layer does not fit the tensor-core path."""
        n = self.nb_states
        if self.input_dim % 4 != 0 or self.output_dim % 4 != 0:
            return None
        for k in range(n):
            dims = (self.A[k].shape[0], self.A[k].shape[1], self.E[k].shape[0], self.E[k].shape[1])
            if max(dims) > self.TC_DS or self.dims_out[k] > self.TC_SOUT_MAX or self.dims_in[k] > self.TC_KB * self.TC_KB_MAX:
                return None
        in_off = np.concatenate([[0], np.cumsum(self.dims_in)]).astype(np.int64)
        out_off = np.concatenate([[0], np.cumsum(self.dims_out)]).astype(np.int64)
        chunks = []
        k = 0
        while k < n:
            k0, nin, nout = k, 0, 0
            while (k < n and k - k0 < self.TC_LMAX and nin + int(self.dims_in[k]) <= self.TC_KB * self.TC_KB_MAX
                   and nout + int(self.dims_out[k]) <= self.TC_PO):
                nin += int(self.dims_in[k])
                nout += int(self.dims_out[k])
                k += 1
            chunks.append([k0, k, int(in_off[k0]), nin, int(out_off[k0]), nout, (nin + self.TC_KB - 1) // self.TC_KB, 0])
        chunks = np.asarray(chunks, dtype=np.int32)
        rows_aligned = int(np.all(chunks[:, 4] % 4 == 0))
        # the build kernels keep every parameter of one direction of a chunk in shared memory
        pad4 = lambda v: (int(v) + 3) // 4 * 4     # every sub-array starts on a 16-byte boundary in shared memory
        per_stage = [(sum(pad4(getattr(self, nm)[k].numel()) for nm in "ABCD"), sum(pad4(getattr(self, nm)[k].numel()) for nm in "EFG")) for k in range(n)]
        pmax = max(max(sum(ps[d] for ps in per_stage[k0:k1]) for d in (0, 1)) for k0, k1 in chunks[:, :2])
        if pmax > 40960:
            return None
        return dict(chunks=chunks, rows_aligned=rows_aligned, chunk_param_floats=max(int(pmax), 1))

    def _tc_plan(self, device):
        tc = self.__dict__.get("_dev_tc_plan")
        if tc is not None and tc["device"] == device:
            return tc
        plan = self._device_plan(device)
        host = self.build_tc_host_plan()
        assert host is not None, "SSSLayer: this layer does not fit the tensor-core path"
        ch_dev = torch.from_numpy(host["chunks"].reshape(-1)).to(device)
        struct = _lib.SnSssTcPlan()
        struct.nb_states, struct.input_dim, struct.output_dim = self.nb_states, self.input_dim, self.output_dim
        struct.nchunks = host["chunks"].shape[0]
        struct.rows_aligned = host["rows_aligned"]
        struct.chunk_param_floats = host["chunk_param_floats"]
        offs = self._param_offsets()
        struct.reserved[0] = int(all(offs[(nm, k + 1)] == offs[(nm, k)] + getattr(self, nm)[k].numel() for nm in "ABCDEFG" for k in range(self.nb_states - 1)))
        struct.stages = plan["stages"].data_ptr()
        struct.chunks = ch_dev.data_ptr()
        ncoef = int(_lib.lib().sn_sss_tc_coef_floats(ctypes.byref(struct)))
        coef = torch.zeros(ncoef, dtype=torch.float32, device=device)   # padding entries stay zero for the life of the plan
        tc = dict(device=device, struct=struct, chunks=ch_dev, stages=plan["stages"], coef=coef, host=host)
        self.__dict__["_dev_tc_plan"] = tc
        return tc

    def _use_tc_path(self) -> bool:
        mode = os.environ.get("SNB200_SSS_PATH", self.__dict__.get("kernel_path", "auto"))
        if mode == "simt":
            return False
        ok = self.__dict__.get("_tc_eligible")
        if ok is None:
            ok = self.build_tc_host_plan() is not None
            self.__dict__["_tc_eligible"] = ok
        if mode == "tc" and not ok:
            raise RuntimeError("SSSLayer: SNB200_SSS_PATH=tc but the layer does not fit the tensor-core path")
        return ok

    def _backward_workspace(self, plan):
        ws = self.__dict__.get("_dev_bwd_ws")
        if ws is None or ws.device != plan["device"]:
            n = _lib.lib().sn_sss_backward_workspace_floats(ctypes.byref(plan["struct"]))
            ws = torch.empty(int(n), dtype=torch.float32, device=plan["device"])
            self.__dict__["_dev_bwd_ws"] = ws
        return ws

    def _packed_params(self, plan):
        """Per-stage re-laid-out copy of the parameters, refreshed on every forward (one ~5 us launch): the
        parameters are updated in place by optimizers and nothing cheaper than re-packing detects that reliably
        (``p.data = view`` does not share the flat buffer's version counter)."""
        flat = self.__dict__["_flat"]
        packed = self.__dict__.get("_dev_packed")
        if packed is None or packed.device != flat.device:
            n = _lib.lib().sn_sss_packed_floats(ctypes.byref(plan["struct"]))
            packed = torch.empty(int(n), dtype=torch.float32, device=flat.device)
            self.__dict__["_dev_packed"] = packed
            self.__dict__["_dev_packed_version"] = None
        rc = _lib.lib().sn_sss_pack(ctypes.byref(plan["struct"]), _lib.ptr(flat), _lib.ptr(packed), _lib.stream_ptr())
        _lib.check(rc, "sn_sss_pack")
        return packed

    # ---- forward ------------------------------------------------------------------------------
    def forward(self, U):
        if hasattr(self, "state_matrices_initialized") and self.state_matrices_initialized:
            self._require_cuda(U, "SSSLayer.forward")
            assert U.dim() == 2 and U.shape[1] == self.input_dim, "SSSLayer expects a (batch, input_dim) input"
            self._ensure_flat()
            flat = self.__dict__["_flat"]
            if flat.device != U.device:
                raise RuntimeError("SSSLayer: module parameters are on %s but the input is on %s" % (flat.device, U.device))
            if U.dtype != torch.float32:
                U = U.float()
            if U.stride(1) != 1:
                U = U.contiguous()
            anchor = self.__dict__.get("_dev_anchor")
            if anchor is None or anchor.device != U.device:
                anchor = torch.zeros(1, device=U.device, requires_grad=True)
                self.__dict__["_dev_anchor"] = anchor
            # the first parameter (the bias, or A[0]) decides at once for a trainable layer; a frozen one is walked in full
            param_grad = torch.is_grad_enabled() and any(p.requires_grad for p in self._flat_param_list())
            save = param_grad or (torch.is_grad_enabled() and U.requires_grad)
            fn = _SSSTCFunction if self._use_tc_path() else _SSSFunction
            return fn.apply(U, anchor if param_grad else None, self, save)
        else:
            # the budget admits not even a block-diagonal D: reference returns zeros (sss_layer.py:130-131)
            return torch.zeros((U.shape[0], self.output_dim), device=U.device)

    def get_nb_parameters(self) -> int:
        if hasattr(self, "state_matrices_initialized") and self.state_matrices_initialized:
            return get_nb_parameters(optim_mat_shape=(self.output_dim, self.input_dim), statespace_dim=self.statespace_dim, nb_states=self.nb_states)
        else:
            return 0
