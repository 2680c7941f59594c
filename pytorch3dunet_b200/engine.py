"""Host-side driver of the B200 3D U-Net engine: sequences the C-ABI kernels of libb200unet.so for the
forward pass and records a tape that replays the matching backward kernels.

PyTorch is used here only for device memory (torch.empty on the caching allocator) and the current CUDA
stream; no torch operator runs on the hot path.  Activations live as bf16 NDHWC tensors ("Act").

Reference semantics implemented (file:line relative to the reference checkout):
  SingleConv / create_conv      pytorch3dunet/unet3d/buildingblocks.py:10-135
  Encoder (MaxPool3d(2))        buildingblocks.py:353-384
  Decoder (nearest + concat)    buildingblocks.py:436-493, 598-614   (virtual concat: Engine._conv3_vcat, csrc/upcat_conv.cu)
  Decoder (deconv + sum)        buildingblocks.py:617-664, :493        (Engine.deconv_up_add)
  ResNetBlock                   buildingblocks.py:230-288              (model.run_res_block; 1x1x1 conv = Engine.pointwise)
  ResNetBlockSE / scSE          buildingblocks.py:291-307, se.py:12-114 (Engine.scse)
  final conv + activation       pytorch3dunet/unet3d/model.py:89-98, 141-147
"""
from __future__ import annotations

import os
import time

import torch

from ._lib import B200Error, lib

ACT_NONE, ACT_RELU, ACT_LEAKY, ACT_ELU = 0, 1, 2, 3
IMPL_AUTO, IMPL_DIRECT, IMPL_TCGEN05 = 0, 1, 2
FINAL_NONE, FINAL_SIGMOID, FINAL_SOFTMAX = 0, 1, 2
_ACT_OF = {"r": (ACT_RELU, 0.0), "l": (ACT_LEAKY, 0.01), "e": (ACT_ELU, 1.0)}


# optional per-launch CUDA-event timing of selected entry points (bench.py roofline leg): list of
# (name, flops, start_event, end_event) appended when enabled
DEBUG = None   # dict: when set, backward closures stash clones of their intermediates (tools/debug_block.py)
TIMING = None
VIRTUAL_CAT = os.environ.get("B200UNET_NO_VIRTUAL_CAT", "0") != "1"  # decoder concat without the concatenated tensor
DECONV_PHASES = os.environ.get("B200UNET_DECONV_PHASES", "1") != "0"  # transposed conv by output parity phases (exact 2x joins)
EXPLICIT_GN = os.environ.get("B200UNET_EXPLICIT_GN", "1") != "0"      # deep levels: GroupNorm as its own pass instead of per-sample weights
EXPLICIT_GN_VOX_PER_COUT = 40
# backward: the small reduction kernels that turn a weight gradient into dW / dgamma / dbeta / the GroupNorm-backward coefficients run
# on a second stream, under the data-gradient convolution of the same layer (which does not depend on them)
SIDE_STREAM = os.environ.get("B200UNET_SIDE_STREAM", "1") != "0"
# a skip connection's GroupNorm backward into an encoder output is applied INSIDE the max-pool backward of the same tensor (one pass)
DEFER_GN_BWD = os.environ.get("B200UNET_DEFER_GN_BWD", "1") != "0"
_SIDE_STREAMS = {}


def _side_stream(device):
    key = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    st = _SIDE_STREAMS.get(key)
    if st is None:
        st = _SIDE_STREAMS[key] = torch.cuda.Stream(device=key)
    return st
PMODE_PHASE_BIAS = 0x100  # B200_PMODE_PHASE_BIAS (include/b200unet.h)
HOST_PROF = None  # dict name -> [calls, seconds] when host profiling is on
TIMED = {"b200_conv3_fwd", "b200_conv3_wgrad", "b200_input_dgrad_conv3", "b200_conv3_up_phase_fwd", "b200_conv3_up_dgrad", "b200_conv3_up_dgrad_zs", "b200_conv3_up_wgrad",

         "b200_pointwise_tc_fwd", "b200_pointwise_tc_wgrad", "b200_deconv_phase_fwd", "b200_deconv_phase_dgrad", "b200_deconv_phase_wgrad"}


def default_impl() -> int:
    return {"auto": IMPL_AUTO, "direct": IMPL_DIRECT, "tcgen05": IMPL_TCGEN05}[os.environ.get("B200UNET_CONV_IMPL", "auto")]


def _p(t):
    return None if t is None else t.data_ptr()


class Act:
    """A bf16 NDHWC activation plus what the engine knows about it."""

    __slots__ = ("t", "act", "slope", "partials", "P", "sums", "_grad", "requires_grad", "grad_partials", "deferred", "pool_pending")

    def __init__(self, t, act=ACT_NONE, slope=0.0, partials=None, P=0, requires_grad=True):
        self.deferred = None      # (dxhat, coef, engine): a GroupNorm backward into this tensor not yet applied (see Engine.defer_gn_bwd)
        self.pool_pending = False  # a max-pool consumer whose backward has not run yet
        self.t = t
        self.act = act          # activation that produced this tensor (needed for the backward mask)
        self.slope = slope
        self.partials = partials  # float [N,P,C,2] partial (sum, sumsq) emitted by the producer, or None
        self.P = P
        self.sums = None        # double [N,C,2], finalised lazily
        self.grad = None        # bf16 NDHWC, gradient w.r.t. the producer's PRE-activation output ("dz form")
        self.grad_partials = None  # (partials [N,P,C,2], P, grad tensor): per-channel totals of `grad` emitted by the kernel that wrote it
        self.requires_grad = requires_grad

    @property
    def grad(self):
        if self.deferred is not None:   # some other reader than the max-pool backward came first: apply the deferred term now
            dxhat, coef, eng = self.deferred
            self.deferred = None
            n, d, h, w, c = self.dims
            eng.gn_bwd_apply(dxhat, self, coef, n, c, d * h * w)
        return self._grad

    @grad.setter
    def grad(self, v):
        self._grad = v

    @property
    def dims(self):
        n, d, h, w, c = self.t.shape
        return n, d, h, w, c

    @property
    def voxels(self):
        return self.t.shape[1] * self.t.shape[2] * self.t.shape[3]


class InputF32:
    """The network input kept in fp32 (reference: ToTensor -> float32, transforms.py:816-826), NDHWC view."""

    __slots__ = ("t", "sums_src", "sums", "partials", "P", "requires_grad", "grad", "act", "slope", "grad_partials")

    def __init__(self, t_ndhwc, ncdhw_src, requires_grad=False):
        self.t = t_ndhwc
        self.sums_src = ncdhw_src
        self.sums = None
        self.partials, self.P = None, 0
        self.requires_grad = requires_grad
        self.grad = None        # fp32 NCDHW (the layout of the network input), unscaled: written by the first layer's backward
        self.grad_partials = None
        self.act, self.slope = ACT_NONE, 0.0

    @property
    def dims(self):
        n, d, h, w, c = self.t.shape
        return n, d, h, w, c

    @property
    def voxels(self):
        return self.t.shape[1] * self.t.shape[2] * self.t.shape[3]


_K188 = {}


def _const_188(device):
    """(1, 8, 8) on the device: scales the GroupNorm-backward coefficients of a tensor that appears 8x in a virtual upsample."""
    key = str(device)
    if key not in _K188:
        _K188[key] = torch.tensor([1.0, 8.0, 8.0], device=device)
    return _K188[key]


class VirtualCat:
    """cat(enc, nearest_up2x(low)) along channels that is never written to memory: its only consumer, the decoder's first
    convolution, runs as conv3_enc(enc) + conv3_up(low) (Engine._conv3_vcat)."""

    __slots__ = ("enc", "low")

    def __init__(self, enc, low):
        self.enc, self.low = enc, low

    @property
    def dims(self):
        n, d, h, w, c0 = self.enc.dims
        return n, d, h, w, c0 + self.low.dims[4]

    @property
    def requires_grad(self):
        return self.enc.requires_grad or self.low.requires_grad


class Engine:
    """One forward (+ optional backward) pass.  Not reusable across passes."""

    def __init__(self, device, impl=None, record=True, sink=None, operand_dtype="bf16", loss_scale=1.0, data_only=False):
        # operand_dtype: the 16-bit type of activations and tensor-core operands ("bf16" | "fp16": two builds of the same kernels).
        # loss_scale (fp16): the seed gradient is multiplied by it and every parameter gradient divided by it, so that the backward
        # pass's activation gradients (~1e-7 for a mean-reduced loss over millions of voxels) stay inside fp16's range
        self.L = lib(operand_dtype)
        self.adt = torch.float16 if operand_dtype in ("fp16", "f16", "float16") else torch.bfloat16
        self.loss_scale = float(loss_scale)
        self.sink = sink      # optim.FlatParameters: parameter gradients are written straight into its flat buffer
        # data_only: the backward computes input gradients only (every parameter frozen): no weight-gradient kernel, no parameter
        # gradient, the GroupNorm-backward sums taken from the data gradients instead of from weight-gradient by-products
        self.data_only = data_only
        self.sunk = set()
        self.device = device
        self.impl = default_impl() if impl is None else impl
        self.record = record
        self.tape = []
        self.param_grads = {}
        self.launches = 0
        self.stream = torch.cuda.current_stream(device).cuda_stream
        self._side_keep = None
        self._k188 = _const_188(device)

    # ---------------------------------------------------------------- helpers
    def empty(self, shape, dtype):
        t = torch.empty(shape, dtype=dtype, device=self.device)
        if self._side_keep is not None:
            self._side_keep.append(t)  # allocated while side-stream work is outstanding: must not be recycled before the join
        return t

    def call(self, name, *args, launches=1, flops=0.0, tag=None, layer=""):
        if HOST_PROF is not None:  # tools/host_profile.py: host seconds spent inside each C-ABI entry point
            t0 = time.perf_counter()
            self.L.call(name, *args, self.stream)
            d = HOST_PROF.setdefault(name, [0, 0.0])
            d[0] += 1
            d[1] += time.perf_counter() - t0
            self.launches += launches
            return
        if TIMING is not None and name in TIMED:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.L.call(name, *args, self.stream)
            e1.record()
            TIMING.append((tag or name, flops, e0, e1, layer))
        else:
            self.L.call(name, *args, self.stream)
        self.launches += launches

    # ---- second stream for the weight-gradient tail (see SIDE_STREAM).  Every buffer the side kernels touch comes from the main
    # stream's allocator and is kept alive until side_join (Engine.empty holds a reference while side work is outstanding), so the
    # caching allocator never hands it out while the side stream uses it.
    def side_begin(self):
        if not SIDE_STREAM or DEBUG is not None or HOST_PROF is not None:
            return False
        main = torch.cuda.current_stream(self.device)
        side = _side_stream(self.device)
        ev = torch.cuda.Event()
        ev.record(main)
        side.wait_event(ev)
        self._main_handle, self.stream = self.stream, side.cuda_stream
        if self._side_keep is None:
            self._side_keep = []
        return True

    def side_mark(self, on):
        """event at the current point of an open side section (None when the section is not open)"""
        if not on:
            return None
        ev = torch.cuda.Event()
        ev.record(_side_stream(self.device))
        return ev

    def side_end(self, on):
        if not on:
            return None
        self.stream = self._main_handle
        ev = torch.cuda.Event()
        ev.record(_side_stream(self.device))
        return ev

    def side_join_event(self, ev):
        """main stream waits for a point of the side stream (side work stays outstanding: buffers are kept)"""
        if ev is not None:
            torch.cuda.current_stream(self.device).wait_event(ev)

    def side_join(self, ev):
        if ev is not None:
            torch.cuda.current_stream(self.device).wait_event(ev)
        self._side_keep = None   # (frees are now ordered after the wait on the main stream)

    def grad_like(self, name, like):
        """output buffer for the gradient of parameter `name`: its slot in the flat gradient buffer when there is one"""
        if self.sink is not None and name not in self.sunk:
            v = self.sink.view(name)
            if v is not None and v.shape == like.shape:
                return v
        return torch.empty_like(like)

    def _add_param_grad(self, name, g):
        if self.data_only:
            return
        if self.loss_scale != 1.0:
            g.mul_(1.0 / self.loss_scale)   # (in place: also when g IS the flat-buffer view the kernel wrote into)
        if self.sink is not None:
            v = self.sink.view(name)
            if v is not None:
                if name in self.sunk:
                    v.add_(g.reshape(v.shape))          # a parameter used twice in one pass (not in the reference's models)
                elif g.data_ptr() != v.data_ptr():
                    v.copy_(g.reshape(v.shape))
                self.sunk.add(name)
                self.sink.written(name)
                return
        if name in self.param_grads:
            self.param_grads[name] = self.param_grads[name] + g
        else:
            self.param_grads[name] = g

    def sums_of(self, x):
        """double [N,C,2] per-(sample, channel) (sum, sum of squares) of x."""
        if x.sums is not None:
            return x.sums
        n, d, h, w, c = x.dims
        vox = d * h * w
        if isinstance(x, InputF32):
            P = self.L.query("b200_stats_ncdhw_f32_partials_count", vox)
            partials = self.empty((n, P, c, 2), torch.float32)
            self.call("b200_stats_ncdhw_f32", _p(x.sums_src), n, c, vox, _p(partials))
        elif x.partials is not None:
            partials, P = x.partials, x.P
        else:
            P = self.L.query("b200_stats_partials_count", n, c, vox)
            partials = self.empty((n, P, c, 2), torch.float32)
            self.call("b200_stats_ndhwc_bf16", _p(x.t), n, c, vox, _p(partials))
        sums = self.empty((n, c, 2), torch.float64)
        self.call("b200_partials_finalize", _p(partials), n, P, c, _p(sums))
        x.sums = sums
        x.partials = None
        return sums

    def gn_coeffs_of(self, x, gamma, beta, groups, vox):
        """(sums, mean_rstd, ab) of GroupNorm(x): straight from the producer's per-block partial sums in one launch when they are still
        there, else sums_of + b200_gn_coeffs"""
        n, c = x.dims[0], x.dims[4]
        ab = self.empty((n, c, 2), torch.float32)
        mean_rstd = self.empty((n, groups, 2), torch.float32)
        if x.sums is None and x.partials is not None and not isinstance(x, InputF32):
            sums = self.empty((n, c, 2), torch.float64)
            self.call("b200_gn_stats_coeffs", _p(x.partials), n, x.P, c, _p(gamma), _p(beta), groups, float(vox), _p(sums), _p(mean_rstd),
                      _p(ab))
            x.sums, x.partials = sums, None
        else:
            sums = self.sums_of(x)
            self.call("b200_gn_coeffs", _p(sums), _p(gamma), _p(beta), groups, float(vox), n, c, _p(mean_rstd), _p(ab))
        return sums, mean_rstd, ab

    def accumulate_grad(self, x, g):
        """x.grad += g where g is already in x's dz form."""
        if x.grad is None:
            x.grad = g
        else:
            # accumulated in place; the totals an earlier writer emitted no longer describe it, the kernel emits the new ones
            self.act_bwd_into(x, g, x.dims[4], 0, x.grad, ACT_NONE, 0.0)

    def act_bwd_into(self, target, g, g_cs, g_co, out, act=None, slope=None):
        """target.grad = g[..., g_co:g_co+C] * act'(target) [+ target.grad], written to `out` (may be g or target.grad itself); the kernel
        also emits the per-channel totals of the result, which spares the producer conv's border-tap sums one read of the tensor"""
        n, d, h, w, c = target.dims
        vox = d * h * w
        act = target.act if act is None else act
        slope = target.slope if slope is None else slope
        P = self.L.query("b200_stats_partials_count", n, c, vox)
        parts = self.empty((n, P, c, 2), torch.float32)
        self.call("b200_act_bwd_stats", _p(g), g_cs, g_co, _p(target.t), n, c, vox, act, float(slope), _p(target.grad), _p(out), _p(parts))
        target.grad = out
        target.grad_partials = (parts, P, out)

    def border_tap_sums(self, out, dz, n, d, h, w, cout):
        """T[n][tap][co] = sum of dz over the voxels whose tap is in bounds; the per-channel totals come from the kernel that produced dz
        when it emitted them (b200_gn_bwd_apply_stats), else from one more pass over dz"""
        L = self.L
        T = self.empty((n, 27, cout), torch.float32)
        scratch = self.empty((L.query("b200_border_tap_sums_workspace", n, d, h, w, cout),), torch.float32)
        gp = out.grad_partials
        if gp is not None and gp[2] is dz:
            self.call("b200_border_tap_sums_pre", _p(dz), n, d, h, w, cout, _p(gp[0]), gp[1], _p(T), _p(scratch), launches=4)
        else:
            self.call("b200_border_tap_sums", _p(dz), n, d, h, w, cout, _p(T), _p(scratch), launches=5)
        return T

    def gn_bwd_apply(self, dxhat, x, coef, n, c, vox):
        """x.grad = (A*dxhat + B*x + C) * act'(x) [+ x.grad], written over dxhat; the kernel also emits the per-channel totals of what it
        writes, which spares the producer conv's border-tap-sum pass one read of the tensor"""
        P = self.L.query("b200_stats_partials_count", n, c, vox)
        parts = self.empty((n, P, c, 2), torch.float32)
        self.call("b200_gn_bwd_apply_stats", _p(dxhat), _p(x.t), _p(coef), n, c, vox, x.act, float(x.slope), _p(x.grad), _p(dxhat), _p(parts))
        x.grad = dxhat
        x.grad_partials = (parts, P, dxhat)

    # ---------------------------------------------------------------- input / output layout
    def input_f32(self, x_ncdhw, requires_grad=False):
        n, c, d, h, w = x_ncdhw.shape
        x_ncdhw = x_ncdhw.contiguous()
        if c == 1:
            t = x_ncdhw.view(n, d, h, w, 1)
        else:
            t = self.empty((n, d, h, w, c), torch.float32)
            self.call("b200_ncdhw_f32_to_ndhwc_f32", _p(x_ncdhw), _p(t), n, c, d, h, w)
        return InputF32(t, x_ncdhw, requires_grad)

    def set_input_grad(self, x, g):
        """x.grad = g for the fp32 network input (fp32 NCDHW, unscaled).  Every model reads x in exactly one layer."""
        if x.grad is not None:
            raise B200Error("the fp32 network input is read by more than one layer: its gradient would need accumulating")
        x.grad = g

    def gn_bwd_coef_from_dgrad(self, dxhat, x, gamma, mean_rstd, groups, vox):
        """GroupNorm-backward coefficients (A, B, C) of x from the data gradient dxhat itself (one pass over dxhat and x): what the
        full backward takes from the weight-gradient by-products (b200_gn_bwd_sums_from_wgrad) when no weight gradient is computed"""
        n, c = x.dims[0], x.dims[4]
        P = self.L.query("b200_stats_partials_count", n, c, vox)
        parts = self.empty((n, P, c, 2), torch.float32)
        self.call("b200_stats2_ndhwc_bf16", _p(dxhat), _p(x.t), n, c, vox, _p(parts))
        sums2 = self.empty((n, c, 2), torch.float64)
        self.call("b200_partials_finalize", _p(parts), n, P, c, _p(sums2))
        return self._gn_bwd_coef(sums2, gamma, mean_rstd, groups, vox, n, c)

    def _gn_bwd_coef(self, sums2, gamma, mean_rstd, groups, vox, n, c):
        coef = self.empty((n, c, 3), torch.float32)
        dgamma, dbeta = self.empty((c,), torch.float32), self.empty((c,), torch.float32)   # (not published: parameters are frozen)
        self.call("b200_gn_bwd_coeffs", _p(sums2), _p(gamma), _p(mean_rstd), groups, float(vox), n, c, _p(coef), _p(dgamma), _p(dbeta))
        return coef

    def input_dgrad_conv3(self, x, dz, W, coef, gn, mean_rstd, vox):
        """gradient w.r.t. the fp32 network input x of the first 3x3x3 conv (csrc/input_grad.cu), GroupNorm backward included when the
        layer starts with one; coef: the layer's GroupNorm-backward coefficients when the full backward already has them, else None"""
        n, d, h, w, cin = x.dims
        cout = W.shape[0]
        inv = 1.0 / self.loss_scale
        dx = self.empty((n, cin, d, h, w), torch.float32)
        parts = None
        if gn is not None and coef is None:
            P = self.L.query("b200_input_dgrad_partials_count", n, d, h, w, cin, cout)
            parts = self.empty((n, P, cin, 2), torch.float32)
        self.call("b200_input_dgrad_conv3", _p(dz), _p(W), n, d, h, w, cin, cout, 1.0 if gn is not None else inv, _p(x.sums_src),
                  _p(dx), _p(parts), flops=2.0 * n * vox * 27 * cin * cout, tag="dgrad_input")
        if gn is not None:
            if coef is None:
                sums2 = self.empty((n, cin, 2), torch.float64)
                self.call("b200_partials_finalize", _p(parts), n, parts.shape[1], cin, _p(sums2))
                coef = self._gn_bwd_coef(sums2, gn[0].contiguous(), mean_rstd, gn[2], vox, n, cin)
            self.call("b200_gn_bwd_apply_ncdhw_f32", _p(dx), _p(x.sums_src), _p(coef), n, cin, vox, inv, _p(dx))
        self.set_input_grad(x, dx)

    def input_bf16(self, x_ncdhw, requires_grad):
        n, c, d, h, w = x_ncdhw.shape
        if c % 8 != 0:
            raise NotImplementedError(f"block-level input with C={c}: internal activations need C % 8 == 0")
        x_ncdhw = x_ncdhw.contiguous()
        t = self.empty((n, d, h, w, c), self.adt)
        self.call("b200_ncdhw_f32_to_ndhwc_bf16", _p(x_ncdhw), _p(t), n, c, d, h, w)
        return Act(t, ACT_NONE, 0.0, requires_grad=requires_grad)

    def to_ncdhw_f32(self, t_ndhwc_bf16):
        n, d, h, w, c = t_ndhwc_bf16.shape
        out = self.empty((n, c, d, h, w), torch.float32)
        self.call("b200_ndhwc_bf16_to_ncdhw_f32", _p(t_ndhwc_bf16), _p(out), n, c, d, h, w)
        return out

    def grad_from_ncdhw(self, y, g_ncdhw):
        """seed y.grad from an external NCDHW fp32 gradient w.r.t. the (post-activation) output y."""
        n, d, h, w, c = y.dims
        g = self.empty((n, d, h, w, c), self.adt)
        g_src = g_ncdhw.contiguous()  # keep the (possible) copy alive until the kernel is enqueued
        self.call("b200_ncdhw_f32_to_ndhwc_bf16", _p(g_src), _p(g), n, c, d, h, w)
        gm = self.empty((n, d, h, w, c), self.adt)
        self.call("b200_act_bwd", _p(g), c, 0, _p(y.t), n, c, d * h * w, y.act, y.slope, None, _p(gm))
        self.accumulate_grad(y, gm)

    # ---------------------------------------------------------------- conv
    def conv3(self, x, W, bias, gn, name, act=(ACT_NONE, 0.0), want_stats=False, residual=None, grad_sink=None):
        """[GroupNorm ->] Conv3d(3x3x3, pad 1) [-> + residual] [-> activation].

        x: Act | InputF32; W: fp32 (Cout,Cin,3,3,3); bias: fp32 (Cout,) | None;
        gn: None | (gamma, beta, num_groups, gamma_name, beta_name); name: parameter name prefix of the conv.
        """
        n, d, h, w, cin = x.dims
        cout = W.shape[0]
        assert W.shape == (cout, cin, 3, 3, 3), (tuple(W.shape), cin)
        if cout % 8 != 0:
            raise NotImplementedError(f"conv with C_out={cout}: the engine needs C_out % 8 == 0")
        if isinstance(x, VirtualCat):
            if residual is None and grad_sink is None and self._vcat_conv_ok(x, cout):
                return self._conv3_vcat(x, W, bias, gn, name, act, want_stats)
            x = self._upcat_materialize(x.enc, x.low, want_stats=gn is not None)
        vox = d * h * w
        is_f32 = isinstance(x, InputF32)
        L = self.L
        impl = L.query("b200_conv3_resolve_impl", self.impl, n, d, h, w, cin, cout, int(is_f32))
        if impl < 0:
            raise B200Error(f"tcgen05 conv requested but unsupported for shape N={n} {d}x{h}x{w} Cin={cin} Cout={cout}")
        W = W.contiguous()
        ab = mean_rstd = None
        n_w = 1
        sums = None
        if gn is not None:
            gamma, beta, groups = gn[0].contiguous(), gn[1].contiguous(), gn[2]
            sums, mean_rstd, ab = self.gn_coeffs_of(x, gamma, beta, groups, vox)
            n_w = n
        wf = self.empty((n_w, 27, cout, cin), self.adt)
        n_b = n_w if (gn is not None or bias is not None) else 0
        biascls = self.empty((n_b, 64, cout), torch.float32) if n_b else None
        self.call("b200_fold_weights_bias", _p(W), _p(ab), _p(bias), _p(sums), float(vox), n, cin, cout, _p(wf), _p(biascls))
        y = self.empty((n, d, h, w, cout), self.adt)
        partials, P = None, 0
        if want_stats:
            P = L.query("b200_conv3_partials_count", impl, n, d, h, w, cin, cout)
            partials = self.empty((n, P, cout, 2), torch.float32)
        self.call("b200_conv3_fwd", impl, _p(x.t), int(is_f32), _p(wf), n_w, _p(biascls), n_b,
                  _p(residual.t) if residual is not None else None, act[0], float(act[1]),
                  n, d, h, w, cin, cout, _p(y), 1 if want_stats else 0, None, _p(partials),
                  flops=2.0 * n * vox * 27 * cin * cout, tag=("fprop_tc" if impl == IMPL_TCGEN05 else "fprop_direct"), layer=name)
        out = Act(y, act[0], act[1], partials, P)
        if DEBUG is not None:
            DEBUG.setdefault("fwd", {})[name] = y

        if self.record:
            def backward():
                dz = out.grad
                if dz is None:
                    return
                need_T = (gn is not None or bias is not None) and not self.data_only
                T = wd = wd_ready = None
                want_dx = x.requires_grad and not is_f32
                if need_T or want_dx:
                    # second stream, under the weight-gradient kernel: the tap-flipped 16-bit weights of the data-gradient conv (needs
                    # only W) and the border tap sums T (only the reduction tail reads them)
                    on_side = self.side_begin() if not self.data_only else False
                    if want_dx:
                        wd = self.empty((27, cin, cout), self.adt)
                        self.call("b200_prep_dgrad_weights", _p(W), cin, cout, _p(wd))
                        wd_ready = self.side_mark(on_side)
                    if need_T:
                        T = self.border_tap_sums(out, dz, n, d, h, w, cout)
                    self.side_end(on_side)
                coef = tail = None
                published = True
                if not self.data_only:
                    wimpl = L.query("b200_conv3_wgrad_resolve_impl", self.impl, n, d, h, w, cin, cout, int(is_f32))
                    if wimpl < 0:
                        raise B200Error("tcgen05 wgrad requested but unsupported for this shape")
                    S = L.query("b200_conv3_wgrad_splits", wimpl, n, d, h, w, cin, cout, int(is_f32))
                    G = self.empty((n, S, 27, cin, cout), torch.float32)
                    self.call("b200_conv3_wgrad", wimpl, _p(x.t), int(is_f32), _p(dz), n, d, h, w, cin, cout, _p(G),
                              launches=1 if (wimpl == IMPL_TCGEN05 or S > 1) else 2, flops=2.0 * n * vox * 27 * cin * cout,
                              tag=("wgrad_tc" if wimpl == IMPL_TCGEN05 else "wgrad_direct"), layer=name)
                    dW = torch.empty_like(W) if grad_sink is not None else self.grad_like(name + "conv.weight", W)
                    Gsum = self.empty((n, 1, 27, cin, cout), torch.float32) if gn is not None else None
                    db = torch.empty_like(bias) if bias is not None else None
                    coef = None
                    if gn is not None:
                        sums2 = self.empty((n, cin, 2), torch.float64)
                        coef = self.empty((n, cin, 3), torch.float32)
                        dgamma, dbeta = torch.empty_like(gamma), torch.empty_like(beta)
                    on_side = self.side_begin()
                    self.call("b200_wgrad_finalize", _p(G), n, S, cin, cout, _p(ab), _p(T) if ab is not None else None, _p(dW), _p(Gsum))
                    if bias is not None:
                        self.call("b200_bias_grad_from_T", _p(T), n, cout, _p(db))
                    if gn is not None:
                        self.call("b200_gn_bwd_sums_from_wgrad", _p(Gsum), 1, _p(T), _p(W), n, cin, cout, _p(sums2))
                        self.call("b200_gn_bwd_coeffs", _p(sums2), _p(gamma), _p(mean_rstd), groups, float(vox), n, cin,
                                  _p(coef), _p(dgamma), _p(dbeta))
                    tail = self.side_end(on_side)

                    def publish():  # main stream, after the join: hand the finished parameter gradients over
                        if grad_sink is not None:
                            grad_sink(dW)  # the weight is a derived tensor (e.g. the conv form of a ConvTranspose3d weight)
                        else:
                            self._add_param_grad(name + "conv.weight", dW)
                        if bias is not None:
                            self._add_param_grad(name + "conv.bias", db)
                        if gn is not None:
                            self._add_param_grad(gn[3], dgamma)
                            self._add_param_grad(gn[4], dbeta)
                    published = not x.requires_grad or DEBUG is not None
                    if published:
                        self.side_join(tail)
                        publish()
                    if DEBUG is not None:
                        DEBUG[name] = dict(dz=dz.clone(), T=None if T is None else T.clone(), G=G.clone(), dW=dW.clone(),
                                           ab=None if ab is None else ab.clone(), x=x.t.clone(), y=out.t.clone(),
                                           sums2=None if gn is None else sums2.clone(), coef=None if coef is None else coef.clone(),
                                           mean_rstd=None if mean_rstd is None else mean_rstd.clone())
                if residual is not None and residual.requires_grad:
                    self.act_bwd_into(residual, dz, cout, 0, self.empty(residual.t.shape, self.adt))
                if x.requires_grad and is_f32:
                    if not published:
                        self.side_join(tail)
                        publish()
                    self.input_dgrad_conv3(x, dz, W, coef, gn, mean_rstd, vox)
                elif x.requires_grad:
                    self.side_join_event(wd_ready)
                    dimpl = L.query("b200_conv3_resolve_impl", self.impl, n, d, h, w, cout, cin, 0)
                    if dimpl < 0:
                        raise B200Error("tcgen05 dgrad requested but unsupported for this shape")
                    dxhat = self.empty((n, d, h, w, cin), self.adt)
                    self.call("b200_conv3_fwd", dimpl, _p(dz), 0, _p(wd), 1, None, 0, None, ACT_NONE, 0.0,
                              n, d, h, w, cout, cin, _p(dxhat), 0, None, None, flops=2.0 * n * vox * 27 * cin * cout,
                              tag=("dgrad_tc" if dimpl == IMPL_TCGEN05 else "dgrad_direct"), layer=name)
                    if not published:
                        self.side_join(tail)
                        publish()
                    if gn is not None and coef is None:   # data-only backward
                        coef = self.gn_bwd_coef_from_dgrad(dxhat, x, gamma, mean_rstd, groups, vox)
                    if coef is not None:
                        self.gn_bwd_apply(dxhat, x, coef, n, cin, vox)
                    else:
                        if x.act != ACT_NONE or x.grad is not None:
                            self.act_bwd_into(x, dxhat, cin, 0, dxhat)
                        else:
                            x.grad = dxhat
                    if DEBUG is not None:
                        DEBUG.setdefault(name, {})["dx"] = dxhat.clone()
                out.grad = None
            self.tape.append(backward)
        return out

    # ---------------------------------------------------------------- GroupNorm after the conv ('cg.', 'c.g')
    def groupnorm_act(self, z, gamma, beta, groups, gname, bname, act=(ACT_NONE, 0.0), want_stats=False, residual=None):
        """y = act(GroupNorm(z) [+ residual]); the residual join is ResNetBlock's `out += residual` after a conv3 whose order ends in
        'g' (the block's own default order 'cge', buildingblocks.py:243-288)."""
        n, d, h, w, c = z.dims
        vox = d * h * w
        gamma, beta = gamma.contiguous(), beta.contiguous()
        sums, mean_rstd, ab = self.gn_coeffs_of(z, gamma, beta, groups, vox)
        y = self.empty(z.t.shape, self.adt)
        partials, P = None, 0
        if want_stats:
            P = self.L.query("b200_stats_partials_count", n, c, vox)
            partials = self.empty((n, P, c, 2), torch.float32)
        self.call("b200_gn_apply_act_res", _p(z.t), _p(ab), _p(residual.t) if residual is not None else None, n, c, vox,
                  act[0], float(act[1]), _p(y), _p(partials))
        out = Act(y, act[0], act[1], partials, P)
        if DEBUG is not None and act[0] != ACT_NONE:
            # (tests) the tensor whose sign pattern is the layer's activation pattern: for conv -> act -> GroupNorm orders that is the
            # conv's own (already stashed) output, not this one
            DEBUG.setdefault("fwd", {})[gname[: -len("groupnorm.weight")]] = y
        if self.record:
            def backward():
                du = out.grad
                if du is None:
                    return
                P2 = self.L.query("b200_stats_partials_count", n, c, vox)
                part2 = self.empty((n, P2, c, 2), torch.float32)
                self.call("b200_stats2_ndhwc_bf16", _p(du), _p(z.t), n, c, vox, _p(part2))
                sums2 = self.empty((n, c, 2), torch.float64)
                self.call("b200_partials_finalize", _p(part2), n, P2, c, _p(sums2))
                coef = self.empty((n, c, 3), torch.float32)
                dgamma, dbeta = torch.empty_like(gamma), torch.empty_like(beta)
                self.call("b200_gn_bwd_coeffs", _p(sums2), _p(gamma), _p(mean_rstd), groups, float(vox), n, c,
                          _p(coef), _p(dgamma), _p(dbeta))
                self._add_param_grad(gname, dgamma)
                self._add_param_grad(bname, dbeta)
                if residual is not None and residual.requires_grad:
                    self.act_bwd_into(residual, du, c, 0, self.empty(residual.t.shape, self.adt))
                if z.requires_grad:
                    self.gn_bwd_apply(du, z, coef, n, c, vox)   # in place over du (not read again), channel totals emitted
                out.grad = None
            self.tape.append(backward)
        return out

    # ---------------------------------------------------------------- SingleConv (order string interpreter)
    def single_conv(self, x, sd, prefix, order, num_groups, want_stats=False, residual=None, final_act=None):
        """buildingblocks.py:10-135.  Supported orders: [g]c[r|l|e], c g [r|l|e], c [r|l|e] g.
        `residual`/`final_act`: ResNetBlock fuses `out += residual; act` into its last conv (:285-286)."""
        if any(ch in order for ch in "bdD"):
            raise NotImplementedError(f"layer_order {order!r}: BatchNorm/Dropout layers are not implemented by the b200 engine")
        ic = order.index("c")
        pre, post = order[:ic], order[ic + 1:]
        if pre not in ("", "g"):
            raise NotImplementedError(f"layer_order {order!r} is not supported")
        W = sd[prefix + "conv.weight"]
        bias = sd.get(prefix + "conv.bias")
        cin, cout = W.shape[1], W.shape[0]
        gn_pre = None
        if pre == "g":
            g = 1 if cin < num_groups else num_groups
            if cin % g != 0:
                raise ValueError(f"GroupNorm: num_channels={cin} not divisible by num_groups={g}")
            gn_pre = (sd[prefix + "groupnorm.weight"], sd[prefix + "groupnorm.bias"], g,
                      prefix + "groupnorm.weight", prefix + "groupnorm.bias")
        acts = [ch for ch in post if ch in _ACT_OF]
        if len(acts) > 1 or post.count("g") > 1 or (pre == "g" and "g" in post):
            raise NotImplementedError(f"layer_order {order!r} is not supported")
        act = _ACT_OF[acts[0]] if acts else (ACT_NONE, 0.0)
        if final_act is not None:
            assert not acts
            act = final_act
        if "g" not in post:
            if gn_pre is not None and isinstance(x, Act) and EXPLICIT_GN and x.voxels < EXPLICIT_GN_VOX_PER_COUT * cout:
                # deep levels (few voxels, wide channels): folding the GroupNorm scale into PER-SAMPLE weight copies moves
                # ~12 * N * 27*C_in*C_out bytes (folded copies, their fp32 gradient sums) while normalising the small activation
                # explicitly moves ~8 * N * voxels * C_in: apply the GroupNorm as its own pass and convolve with the shared weights
                xh = self.groupnorm_act(x, gn_pre[0], gn_pre[1], gn_pre[2], gn_pre[3], gn_pre[4])
                return self.conv3(xh, W, bias, None, prefix, act=act, want_stats=want_stats, residual=residual)
            return self.conv3(x, W, bias, gn_pre, prefix, act=act, want_stats=want_stats, residual=residual)
        g = 1 if cout < num_groups else num_groups
        if cout % g != 0:
            raise ValueError(f"GroupNorm: num_channels={cout} not divisible by num_groups={g}")
        act_first = bool(acts) and post.index(acts[0]) < post.index("g")
        z = self.conv3(x, W, bias, None, prefix, act=act if act_first else (ACT_NONE, 0.0), want_stats=True)
        return self.groupnorm_act(z, sd[prefix + "groupnorm.weight"], sd[prefix + "groupnorm.bias"], g,
                                  prefix + "groupnorm.weight", prefix + "groupnorm.bias",
                                  act=(ACT_NONE, 0.0) if act_first else act, want_stats=want_stats, residual=residual)

    # ---------------------------------------------------------------- pooling / upsample+concat
    def maxpool(self, x, want_stats=True, kind="max"):
        """Encoder pooling, buildingblocks.py:353-363: MaxPool3d(2) or (pool_type='avg') AvgPool3d(2), floor mode."""
        n, d, h, w, c = x.dims
        fwd, bwd = ("b200_maxpool_fwd", "b200_maxpool_bwd") if kind == "max" else ("b200_avgpool_fwd", "b200_avgpool_bwd")
        y = self.empty((n, d // 2, h // 2, w // 2, c), self.adt)
        P = self.L.query("b200_maxpool_partials_count", n, d, h, w, c)
        partials = self.empty((n, P, c, 2), torch.float32) if want_stats else None
        self.call(fwd, _p(x.t), n, d, h, w, c, _p(y), _p(partials))
        out = Act(y, ACT_NONE, 0.0, partials, P)
        if DEBUG is not None and kind == "max":
            DEBUG.setdefault("pool", []).append(x.t)
        if self.record:
            if kind == "max" and isinstance(x, Act):
                x.pool_pending = True

            def backward():
                if isinstance(x, Act):
                    x.pool_pending = False
                if out.grad is None or not x.requires_grad:
                    return
                if isinstance(x, Act) and x.deferred is not None and kind == "max":
                    # the skip connection's GroupNorm backward and the pool scatter in ONE pass; the kernel also emits the channel totals
                    dxhat, coef, _ = x.deferred
                    x.deferred = None
                    PP = self.L.query("b200_maxpool_bwd_partials_count", n, d, h, w, c)
                    parts = self.empty((n, PP, c, 2), torch.float32)
                    self.call("b200_maxpool_bwd_gn", _p(out.grad), _p(x.t), n, d, h, w, c, x.act, float(x.slope), _p(dxhat), _p(coef),
                              _p(dxhat), _p(parts))
                    x.grad = dxhat
                    x.grad_partials = (parts, PP, dxhat)
                    out.grad = None
                    return
                g = x.grad if x.grad is not None else self.empty(x.t.shape, self.adt)
                self.call(bwd, _p(out.grad), _p(x.t), n, d, h, w, c, x.act, x.slope, _p(x.grad), _p(g))
                x.grad = g
                x.grad_partials = None  # (possibly accumulated in place: totals emitted by an earlier writer no longer describe it)
                out.grad = None
            self.tape.append(backward)
        return out

    def upcat(self, enc, x, want_stats=True, allow_virtual=False, mode="nearest"):
        """Decoder joining for interpolation upsampling + concat (buildingblocks.py:482-497, :598-614).  mode 'nearest': when the
        encoder feature is exactly 2x the low-res one the concatenated tensor stays virtual (VirtualCat); otherwise, and for
        mode 'trilinear', it is materialised by one HBM-bound kernel."""
        n, D, H, W, c0 = enc.dims
        n2, d, h, w, c1 = x.dims
        assert n == n2
        if mode != "nearest":
            return self._upcat_materialize(enc, x, want_stats, mode=mode)
        if (allow_virtual and VIRTUAL_CAT and self.impl != IMPL_DIRECT and (D, H, W) == (2 * d, 2 * h, 2 * w) and c0 % 16 == 0 and c1 % 16 == 0
                and isinstance(enc, Act) and isinstance(x, Act)):
            return VirtualCat(enc, x)
        return self._upcat_materialize(enc, x, want_stats)

    def _vcat_conv_ok(self, vc, cout):
        n, D, H, W, c0 = vc.enc.dims
        _, d, h, w, c1 = vc.low.dims
        L = self.L
        return (cout % 16 == 0 and L.query("b200_conv3_up_supported", n, d, h, w, c1, cout)
                and L.query("b200_conv3_resolve_impl", self.impl, n, D, H, W, c0, cout, 0) == IMPL_TCGEN05
                and L.query("b200_conv3_wgrad_resolve_impl", self.impl, n, D, H, W, c0, cout, 0) == IMPL_TCGEN05
                and L.query("b200_conv3_up_wgrad_splits", n, d, h, w, cout, c1) > 0)

    def _conv3_vcat(self, vc, W, bias, gn, name, act, want_stats):
        """[GroupNorm ->] Conv3d(3x3x3) [-> act] of cat(enc, up2x(low)) as conv3_enc(enc) + conv3_up(low): the upsampled part is a
        2x2x2 convolution of the low-res tensor per output parity phase (8/27 of its MACs), see csrc/upcat_conv.cu."""
        enc, low = vc.enc, vc.low
        n, D, H, Wd, c0 = enc.dims
        _, d, h, w, c1 = low.dims
        C, cout = c0 + c1, W.shape[0]
        vox, lvox = D * H * Wd, d * h * w
        L = self.L
        W = W.contiguous()
        ab = mean_rstd = sums = None
        gamma = beta = None
        groups = 1
        n_w = 1
        if gn is not None:
            gamma, beta, groups = gn[0].contiguous(), gn[1].contiguous(), gn[2]
            # statistics of the virtual tensor: every low-res voxel appears 8 times
            sums = torch.cat([self.sums_of(enc), self.sums_of(low) * 8.0], dim=1).contiguous()
            n_w = n
            ab = self.empty((n, C, 2), torch.float32)
            mean_rstd = self.empty((n, groups, 2), torch.float32)
        wf_enc = self.empty((n_w, 27, cout, c0), self.adt)
        wp = self.empty((n_w, 64, cout, c1), self.adt)
        n_b = n_w if (gn is not None or bias is not None) else 0
        biascls = self.empty((n_b, 64, cout), torch.float32) if n_b else None
        self.call("b200_gn_fold_upcat", _p(sums), _p(gamma), _p(beta), groups, float(vox), _p(W), _p(bias), n, c0, c1, cout,
                  _p(wf_enc), _p(wp), _p(biascls), _p(mean_rstd), _p(ab), launches=4 if gn is not None else 3)
        R = self.empty((n, D, H, Wd, cout), self.adt)
        self.call("b200_conv3_up_phase_fwd", _p(low.t), _p(wp), n_w, n, d, h, w, c1, cout, _p(R), launches=1,
                  flops=2.0 * n * vox * 8 * c1 * cout, tag="fprop_tc", layer=name)
        y = self.empty((n, D, H, Wd, cout), self.adt)
        partials, P = None, 0
        if want_stats:
            P = L.query("b200_conv3_partials_count", IMPL_TCGEN05, n, D, H, Wd, c0, cout)
            partials = self.empty((n, P, cout, 2), torch.float32)
        self.call("b200_conv3_fwd", IMPL_TCGEN05, _p(enc.t), 0, _p(wf_enc), n_w, _p(biascls), n_b, _p(R), act[0], float(act[1]),
                  n, D, H, Wd, c0, cout, _p(y), (1 if want_stats else 0) | PMODE_PHASE_BIAS, None, _p(partials),
                  flops=2.0 * n * vox * 27 * c0 * cout, tag="fprop_tc", layer=name)
        out = Act(y, act[0], act[1], partials, P)
        if DEBUG is not None:
            DEBUG.setdefault("fwd", {})[name] = y

        if self.record:
            def backward():
                dz = out.grad
                if dz is None:
                    return
                T = wd_enc = wd_up = wd_ready = None
                want_dx = enc.requires_grad or low.requires_grad
                if self.data_only:
                    self._conv3_vcat_data_backward(vc, dz, W, gn, mean_rstd, name)
                    out.grad = None
                    return
                if gn is not None or bias is not None or want_dx:
                    on_side = self.side_begin()   # under the two weight-gradient kernels
                    if want_dx:
                        wd_enc = self.empty((27, c0, cout), self.adt)
                        wd_up = self.empty((64, c1, cout), self.adt)
                        self.call("b200_upcat_prep_dgrad_weights", _p(W), c0, c1, cout, _p(wd_enc), _p(wd_up))
                        wd_ready = self.side_mark(on_side)
                    if gn is not None or bias is not None:
                        T = self.border_tap_sums(out, dz, n, D, H, Wd, cout)
                    self.side_end(on_side)
                S1 = L.query("b200_conv3_wgrad_splits", IMPL_TCGEN05, n, D, H, Wd, c0, cout, 0)
                G_enc = self.empty((n, S1, 27, c0, cout), torch.float32)
                self.call("b200_conv3_wgrad", IMPL_TCGEN05, _p(enc.t), 0, _p(dz), n, D, H, Wd, c0, cout, _p(G_enc),
                          flops=2.0 * n * vox * 27 * c0 * cout, tag="wgrad_tc", layer=name)
                S2 = L.query("b200_conv3_up_wgrad_splits", n, d, h, w, cout, c1)
                Q = self.empty((n, S2, 64, cout, c1), torch.float32)
                self.call("b200_conv3_up_wgrad", _p(dz), _p(low.t), n, d, h, w, cout, c1, _p(Q),
                          flops=2.0 * n * lvox * 64 * c1 * cout, tag="wgrad_tc", layer=name)
                G = self.empty((n, 1, 27, C, cout), torch.float32)
                dW = self.grad_like(name + "conv.weight", W)
                Gsum = self.empty((n, 1, 27, C, cout), torch.float32) if gn is not None else None
                db = torch.empty_like(bias) if bias is not None else None
                coef = None
                if gn is not None:
                    sums2 = self.empty((n, C, 2), torch.float64)
                    coef = self.empty((n, C, 3), torch.float32)
                    dgamma, dbeta = torch.empty_like(gamma), torch.empty_like(beta)
                on_side = self.side_begin()   # the reductions below run under the two data-gradient convolutions
                self.call("b200_upcat_assemble_wgrad", _p(G_enc), S1, _p(Q), S2, n, c0, c1, cout, _p(G))
                self.call("b200_wgrad_finalize", _p(G), n, 1, C, cout, _p(ab), _p(T) if ab is not None else None, _p(dW), _p(Gsum))
                if bias is not None:
                    self.call("b200_bias_grad_from_T", _p(T), n, cout, _p(db))
                if gn is not None:
                    self.call("b200_gn_bwd_sums_from_wgrad", _p(Gsum), 1, _p(T), _p(W), n, C, cout, _p(sums2))
                    self.call("b200_gn_bwd_coeffs", _p(sums2), _p(gamma), _p(mean_rstd), groups, float(vox), n, C,
                              _p(coef), _p(dgamma), _p(dbeta))
                tail = self.side_end(on_side)
                published = False

                def publish():
                    self._add_param_grad(name + "conv.weight", dW)
                    if bias is not None:
                        self._add_param_grad(name + "conv.bias", db)
                    if gn is not None:
                        self._add_param_grad(gn[3], dgamma)
                        self._add_param_grad(gn[4], dbeta)
                self.side_join_event(wd_ready)
                if enc.requires_grad:
                    ge = self._vcat_dgrad_enc(vc, dz, wd_enc, cout, name)
                    if coef is not None:
                        if not published:
                            self.side_join(tail)
                            publish()
                            published = True
                    self._vcat_apply_enc(vc, ge, coef)
                if low.requires_grad:
                    gl = self._vcat_dgrad_low(vc, dz, wd_up, cout, name)
                    if coef is not None:
                        if not published:
                            self.side_join(tail)
                            publish()
                            published = True
                    self._vcat_apply_low(vc, gl, coef)
                if not published:
                    self.side_join(tail)
                    publish()
                out.grad = None
            self.tape.append(backward)
        return out

    def _vcat_dgrad_enc(self, vc, dz, wd_enc, cout, name):
        """data gradient of conv3_enc: the raw (pre-GroupNorm-backward) gradient of the encoder part of the virtual concat"""
        n, D, H, Wd, c0 = vc.enc.dims
        dimpl = self.L.query("b200_conv3_resolve_impl", self.impl, n, D, H, Wd, cout, c0, 0)
        if dimpl < 0:
            raise B200Error("tcgen05 dgrad requested but unsupported for this shape")
        ge = self.empty(vc.enc.t.shape, self.adt)
        self.call("b200_conv3_fwd", dimpl, _p(dz), 0, _p(wd_enc), 1, None, 0, None, ACT_NONE, 0.0,
                  n, D, H, Wd, cout, c0, _p(ge), 0, None, None, flops=2.0 * n * D * H * Wd * 27 * c0 * cout,
                  tag=("dgrad_tc" if dimpl == IMPL_TCGEN05 else "dgrad_direct"), layer=name)
        return ge

    def _vcat_dgrad_low(self, vc, dz, wd_up, cout, name):
        """data gradient of conv3_up: the gradient of the low-res tensor summed over its 8 copies in the virtual upsample"""
        n, d, h, w, c1 = vc.low.dims
        lvox = d * h * w
        L = self.L
        gl = self.empty(vc.low.t.shape, self.adt)
        if self.impl != IMPL_DIRECT and L.query("b200_conv3_up_dgrad_zs_supported", n, d, h, w, cout, c1):
            parts = self.empty((4,) + tuple(vc.low.t.shape), self.adt)   # one partial gradient per in-plane parity of dz
            self.call("b200_conv3_up_dgrad_zs", _p(dz), _p(wd_up), n, d, h, w, cout, c1, _p(parts), _p(gl), launches=2,
                      flops=2.0 * n * lvox * 64 * c1 * cout, tag="dgrad_tc", layer=name)
            del parts
        else:
            self.call("b200_conv3_up_dgrad", _p(dz), _p(wd_up), n, d, h, w, cout, c1, _p(gl),
                      flops=2.0 * n * lvox * 64 * c1 * cout, tag="dgrad_tc", layer=name)
        return gl

    def _vcat_apply_enc(self, vc, ge, coef):
        enc = vc.enc
        n, D, H, Wd, c0 = enc.dims
        if coef is not None:
            if DEFER_GN_BWD and DEBUG is None and enc.pool_pending and enc.deferred is None and enc._grad is None:
                enc.deferred = (ge, coef[:, :c0].contiguous(), self)   # applied by the max-pool backward of enc
            else:
                self.gn_bwd_apply(ge, enc, coef[:, :c0].contiguous(), n, c0, D * H * Wd)
        else:
            if enc.act != ACT_NONE or enc.grad is not None:
                self.act_bwd_into(enc, ge, c0, 0, ge)
            else:
                enc.grad = ge

    def _vcat_apply_low(self, vc, gl, coef):
        low = vc.low
        n, d, h, w, c1 = low.dims
        c0 = vc.enc.dims[4]
        if coef is not None:
            # d b[u] = sum over its 8 copies of (A dxhat + B x + C) = A sum(dxhat) + 8B b + 8C
            self.gn_bwd_apply(gl, low, (coef[:, c0:] * self._k188).contiguous(), n, c1, d * h * w)
        else:
            if low.act != ACT_NONE or low.grad is not None:
                self.act_bwd_into(low, gl, c1, 0, gl)
            else:
                low.grad = gl

    def _conv3_vcat_data_backward(self, vc, dz, W, gn, mean_rstd, name):
        """input-gradient-only backward of the virtual-concat convolution.  With a GroupNorm in front, its backward sums over the
        concatenated tensor come from the two raw data gradients: sum over the full-res voxels of the upsampled part of (dxhat, dxhat*x)
        equals sum over the low-res voxels of (gl, gl*b), since gl already sums each voxel's 8 copies"""
        enc, low = vc.enc, vc.low
        n, D, H, Wd, c0 = enc.dims
        c1 = low.dims[4]
        cout = W.shape[0]
        wd_enc = self.empty((27, c0, cout), self.adt)
        wd_up = self.empty((64, c1, cout), self.adt)
        self.call("b200_upcat_prep_dgrad_weights", _p(W), c0, c1, cout, _p(wd_enc), _p(wd_up))
        ge = self._vcat_dgrad_enc(vc, dz, wd_enc, cout, name) if (enc.requires_grad or gn is not None) else None
        gl = self._vcat_dgrad_low(vc, dz, wd_up, cout, name) if (low.requires_grad or gn is not None) else None
        coef = None
        if gn is not None:
            sums = []
            for g, t in ((ge, enc), (gl, low)):
                tn, td, th, tw, tc = t.dims
                P = self.L.query("b200_stats_partials_count", tn, tc, td * th * tw)
                parts = self.empty((tn, P, tc, 2), torch.float32)
                self.call("b200_stats2_ndhwc_bf16", _p(g), _p(t.t), tn, tc, td * th * tw, _p(parts))
                s2 = self.empty((tn, tc, 2), torch.float64)
                self.call("b200_partials_finalize", _p(parts), tn, P, tc, _p(s2))
                sums.append(s2)
            coef = self._gn_bwd_coef(torch.cat(sums, dim=1).contiguous(), gn[0].contiguous(), mean_rstd, gn[2], D * H * Wd, n, c0 + c1)
        if enc.requires_grad:
            self._vcat_apply_enc(vc, ge, coef)
        if low.requires_grad:
            self._vcat_apply_low(vc, gl, coef)

    def _upcat_materialize(self, enc, x, want_stats=True, mode="nearest"):
        n, D, H, W, c0 = enc.dims
        n2, d, h, w, c1 = x.dims
        fwd, bwd = {"nearest": ("b200_upcat_fwd", "b200_upcat_bwd"),
                    "trilinear": ("b200_upcat_trilinear_fwd", "b200_upcat_trilinear_bwd")}[mode]
        cat = self.empty((n, D, H, W, c0 + c1), self.adt)
        P = self.L.query("b200_upcat_partials_count", n, D, H, W, c0 + c1)
        partials = self.empty((n, P, c0 + c1, 2), torch.float32) if want_stats else None
        self.call(fwd, _p(enc.t), c0, _p(x.t), c1, n, D, H, W, d, h, w, _p(cat), _p(partials))
        out = Act(cat, ACT_NONE, 0.0, partials, P)
        if self.record:
            def backward():
                dcat = out.grad
                if dcat is None:
                    return
                if x.requires_grad:
                    g = self.empty(x.t.shape, self.adt)
                    self.call(bwd, _p(dcat), c0, c1, _p(x.t), n, D, H, W, d, h, w, x.act, x.slope, _p(g))
                    self.accumulate_grad(x, g)
                if enc.requires_grad:
                    # enc.grad = dcat[..., :c0] * act'(enc) + enc.grad (enc.grad, if any, is already in dz form)
                    self.act_bwd_into(enc, dcat, c0 + c1, 0, self.empty(enc.t.shape, self.adt))
                out.grad = None
            self.tape.append(backward)
        return out

    # ---------------------------------------------------------------- 1x1x1 conv with bias (ResNetBlock.conv1, buildingblocks.py:251)
    def pointwise(self, x, W, bias, wname, bname, want_stats=True):
        n, d, h, w, cin = x.dims
        vox = d * h * w
        cout = W.shape[0]
        if cout % 8 != 0:
            raise NotImplementedError(f"1x1x1 conv with C_out={cout}: the engine needs C_out % 8 == 0")
        is_f32 = isinstance(x, InputF32)
        W2 = W.reshape(cout, cin).contiguous()
        y = self.empty((n, d, h, w, cout), self.adt)
        # tensor-core path: the tcgen05 conv / wgrad kernels over the flat voxel list (C_in, C_out multiples of 16, bf16 input)
        tc = (not is_f32) and self.impl != IMPL_DIRECT and bool(self.L.query("b200_pointwise_tc_supported", n, vox, cin, cout))
        if tc:
            wq = self.empty((cout, cin), self.adt)
            self.call("b200_pointwise_prep_weights", _p(W2), cin, cout, 0, _p(wq))
            P = self.L.query("b200_pointwise_tc_partials_count", n, vox)
            partials = self.empty((n, P, cout, 2), torch.float32) if want_stats else None
            self.call("b200_pointwise_tc_fwd", _p(x.t), _p(wq), _p(bias), n, vox, cin, cout, _p(y), _p(partials),
                      flops=2.0 * n * vox * cin * cout, tag="fprop_tc")
        else:
            P = self.L.query("b200_pointwise_partials_count", n, vox, cout)
            partials = self.empty((n, P, cout, 2), torch.float32) if want_stats else None
            self.call("b200_pointwise_fwd", _p(x.t), int(is_f32), _p(W2), 0, _p(bias), n, vox, cin, cout, _p(y), _p(partials))
        out = Act(y, ACT_NONE, 0.0, partials, P)
        if self.record:
            def backward():
                dy = out.grad
                if dy is None:
                    return
                if self.data_only:
                    pass   # frozen parameters: no weight or bias gradient
                elif tc:
                    S = self.L.query("b200_pointwise_tc_wgrad_splits", n, vox, cin, cout)
                    G = self.empty((n * S, cin * cout), torch.float32)
                    self.call("b200_pointwise_tc_wgrad", _p(x.t), _p(dy), n, vox, cin, cout, _p(G),
                              flops=2.0 * n * vox * cin * cout, tag="wgrad_tc")
                    red = self.empty((cin * cout,), torch.float32)
                    self.call("b200_reduce_rows", _p(G), n * S, cin * cout, _p(red))
                    self._add_param_grad(wname, red.view(cin, cout).t().reshape(W.shape))
                    if bias is not None:
                        self._add_param_grad(bname, self.sums_of(Act(dy, requires_grad=False))[:, :, 0].sum(0).float())
                else:
                    Pw = self.L.query("b200_pointwise_wgrad_partials_count", n, vox)
                    K = cout * cin + cout
                    part = self.empty((n * Pw, K), torch.float32)
                    self.call("b200_pointwise_wgrad", _p(x.t), int(is_f32), _p(dy), n, vox, cin, cout, _p(part))
                    red = self.empty((K,), torch.float32)
                    self.call("b200_reduce_rows", _p(part), n * Pw, K, _p(red))
                    self._add_param_grad(wname, red[: cout * cin].reshape(W.shape))
                    if bias is not None:
                        self._add_param_grad(bname, red[cout * cin:].clone())
                if x.requires_grad and is_f32:
                    dx = self.empty((n, cin, d, h, w), torch.float32)
                    self.call("b200_pointwise_dgrad_f32", _p(dy), _p(W2), n, vox, cin, cout, 1.0 / self.loss_scale, _p(dx))
                    self.set_input_grad(x, dx)
                elif x.requires_grad:
                    g = self.empty(x.t.shape, self.adt)
                    if tc:
                        wqt = self.empty((cin, cout), self.adt)
                        self.call("b200_pointwise_prep_weights", _p(W2), cin, cout, 1, _p(wqt))
                        self.call("b200_pointwise_tc_fwd", _p(dy), _p(wqt), None, n, vox, cout, cin, _p(g), None,
                                  flops=2.0 * n * vox * cin * cout, tag="dgrad_tc")
                    else:
                        self.call("b200_pointwise_fwd", _p(dy), 0, _p(W2), 1, None, n, vox, cout, cin, _p(g), None)
                    if x.act != ACT_NONE or x.grad is not None:
                        self.act_bwd_into(x, g, cin, 0, g)
                    else:
                        x.grad = g
                out.grad = None
            self.tape.append(backward)
        return out

    # ---------------------------------------------------------------- ConvTranspose3d(k3,s2,p1) + nearest resize + sum-join
    def deconv(self, x, Wt, wname):
        """ConvTranspose3d(k3, s2, p1, bias=False) (TransposeConvUpsampling, buildingblocks.py:617-664) -> Act on the (2d-1)^3 grid.

        conv_transpose3d(x, Wt, stride 2, pad 1) == conv3d(zero_insert(x), Wc, pad 1) with Wc[co][ci][k] = Wt[ci][co][26-k], so the
        transposed conv, its input gradient and its weight gradient all run on the tcgen05 3x3x3 kernels (conv3)."""
        n, d, h, w, cin = x.dims
        cout = Wt.shape[1]
        assert tuple(Wt.shape) == (cin, cout, 3, 3, 3), (tuple(Wt.shape), cin, cout)
        Wt = Wt.contiguous()
        sd_, sh_, sw_ = 2 * d - 1, 2 * h - 1, 2 * w - 1
        Wc = self.empty((cout, cin, 3, 3, 3), torch.float32)
        self.call("b200_deconv_weight_permute", _p(Wt), cin, cout, 1, _p(Wc))
        xz_t = self.empty((n, sd_, sh_, sw_, cin), self.adt)
        self.call("b200_zero_insert", _p(x.t), n, d, h, w, cin, _p(xz_t))
        xz = Act(xz_t, ACT_NONE, 0.0, requires_grad=x.requires_grad)
        if self.record:
            def backward_zero_insert():
                if xz.grad is None or not x.requires_grad:
                    return
                gx = self.empty(x.t.shape, self.adt)
                self.call("b200_subsample2_bwd", _p(xz.grad), _p(x.t), n, d, h, w, cin, x.act, x.slope, _p(x.grad), _p(gx))
                x.grad = gx
                xz.grad = None
            self.tape.append(backward_zero_insert)

        def sink(dWc):
            dWt = self.grad_like(wname, Wt)
            self.call("b200_deconv_weight_permute", _p(dWc), cin, cout, 0, _p(dWt))
            self._add_param_grad(wname, dWt)
        return self.conv3(xz, Wc, None, None, wname + "#conv.", want_stats=False, grad_sink=sink)

    def deconv_up_add(self, enc, x, Wt, wname, want_stats=True):
        """TransposeConvUpsampling followed by Decoder._joining(concat=False) (buildingblocks.py:493):
        out = enc + interpolate(conv_transpose3d(x), size=enc.shape[2:]) (nearest resize of the (2d-1)^3 grid)."""
        n, D, H, W_, cout = enc.dims
        n2, d, h, w, cin = x.dims
        assert n == n2
        if (DECONV_PHASES and self.impl != IMPL_DIRECT and (D, H, W_) == (2 * d, 2 * h, 2 * w) and d >= 1
                and self.L.query("b200_device_is_sm100") and self.L.query("b200_deconv_phase_supported", n, d, h, w, cin, cout)
                and self.L.query("b200_deconv_phase_wgrad_splits", n, d, h, w, cout, cin) > 0):
            return self._deconv_up_add_phases(enc, x, Wt, wname, want_stats)
        sd_, sh_, sw_ = 2 * d - 1, 2 * h - 1, 2 * w - 1
        T = self.deconv(x, Wt, wname)
        out_t = self.empty((n, D, H, W_, cout), self.adt)
        P = self.L.query("b200_resize_add_partials_count", n, D, H, W_, cout)
        partials = self.empty((n, P, cout, 2), torch.float32) if want_stats else None
        self.call("b200_resize_add_fwd", _p(T.t), _p(enc.t), n, sd_, sh_, sw_, D, H, W_, cout, _p(out_t), _p(partials))
        out = Act(out_t, ACT_NONE, 0.0, partials, P)
        if self.record:
            def backward():
                g = out.grad
                if g is None:
                    return
                dT = self.empty(T.t.shape, self.adt)
                self.call("b200_deconv_gather", _p(g), n, d, h, w, D, H, W_, cout, _p(dT))
                self.accumulate_grad(T, dT)
                if enc.requires_grad:
                    self.act_bwd_into(enc, g, cout, 0, self.empty(enc.t.shape, self.adt))
                out.grad = None
            self.tape.append(backward)
        return out

    def _deconv_up_add_phases(self, enc, x, Wt, wname, want_stats):
        """deconv_up_add for an encoder feature of exactly twice the low-res size, by output parity phases (csrc: b200_deconv_phase_*):
        27 (phase, tap) products on the low-res lattice instead of 27 taps per voxel of the zero-inserted grid (8x fewer MACs), no
        zero-inserted tensor, the (2d-1)^3 -> (2d)^3 nearest resize folded into the join's index map."""
        n, D, H, W_, cout = enc.dims
        _, d, h, w, cin = x.dims
        Wt = Wt.contiguous()
        wq = self.empty((27, cout, cin), self.adt)
        wd = self.empty((27, cin, cout), self.adt)
        self.call("b200_deconv_phase_weights", _p(Wt), cin, cout, _p(wq), _p(wd))
        Pt = self.empty((n, D, H, W_, cout), self.adt)
        self.call("b200_deconv_phase_fwd", _p(x.t), _p(wq), n, d, h, w, cin, cout, _p(Pt),
                  flops=2.0 * n * d * h * w * 27 * cin * cout, tag="fprop_tc", layer=wname)
        out_t = self.empty((n, D, H, W_, cout), self.adt)
        Pn = self.L.query("b200_upcat_partials_count", n, D, H, W_, cout)
        partials = self.empty((n, Pn, cout, 2), torch.float32) if want_stats else None
        self.call("b200_shift_add_fwd", _p(Pt), _p(enc.t), n, D, H, W_, cout, _p(out_t), _p(partials))
        del Pt
        out = Act(out_t, ACT_NONE, 0.0, partials, Pn)
        if self.record:
            def backward():
                g = out.grad
                if g is None:
                    return
                gp = self.empty((n, D, H, W_, cout), self.adt)
                self.call("b200_shift_fold_bwd", _p(g), n, D, H, W_, cout, _p(gp))
                if not self.data_only:
                    S = self.L.query("b200_deconv_phase_wgrad_splits", n, d, h, w, cout, cin)
                    Q = self.empty((n * S, 27, cout, cin), torch.float32)
                    self.call("b200_deconv_phase_wgrad", _p(gp), _p(x.t), n, d, h, w, cout, cin, _p(Q),
                              flops=2.0 * n * d * h * w * 27 * cin * cout, tag="wgrad_tc", layer=wname)
                    dWt = self.grad_like(wname, Wt)
                    self.call("b200_deconv_phase_wgrad_finalize", _p(Q), n * S, cin, cout, _p(dWt))
                    self._add_param_grad(wname, dWt)
                if x.requires_grad:
                    gx = self.empty(x.t.shape, self.adt)
                    self.call("b200_deconv_phase_dgrad", _p(gp), _p(wd), n, d, h, w, cout, cin, _p(gx),
                              flops=2.0 * n * d * h * w * 27 * cin * cout, tag="dgrad_tc", layer=wname)
                    if x.act != ACT_NONE or x.grad is not None:
                        self.act_bwd_into(x, gx, cin, 0, gx)
                    else:
                        x.grad = gx
                if enc.requires_grad:
                    self.act_bwd_into(enc, g, cout, 0, self.empty(enc.t.shape, self.adt))
                out.grad = None
            self.tape.append(backward)
        return out

    # ---------------------------------------------------------------- scSE (ChannelSpatialSELayer3D, se.py:96-114)
    def scse(self, y, sd, prefix):
        """out = max(cSE(y), sSE(y)) with reduction_ratio 1 (ResNetBlockSE, buildingblocks.py:291-307)."""
        n, d, h, w, c = y.dims
        vox = d * h * w
        W1, b1 = sd[prefix + "cSE.fc1.weight"].contiguous(), sd[prefix + "cSE.fc1.bias"].contiguous()
        W2, b2 = sd[prefix + "cSE.fc2.weight"].contiguous(), sd[prefix + "cSE.fc2.bias"].contiguous()
        ws = sd[prefix + "sSE.conv.weight"].reshape(-1).contiguous()
        bs_t = sd[prefix + "sSE.conv.bias"]
        if W1.shape != (c, c) or W2.shape != (c, c):
            raise NotImplementedError("the b200 engine implements scSE with reduction_ratio=1 (what ResNetBlockSE uses)")
        sums = self.sums_of(y)
        smean = self.empty((n, c), torch.float32)
        hh = self.empty((n, c), torch.float32)
        g = self.empty((n, c), torch.float32)
        self.call("b200_se_gates_fwd", _p(sums), float(vox), _p(W1), _p(b1), _p(W2), _p(b2), n, c, _p(smean), _p(hh), _p(g))
        out_t = self.empty(y.t.shape, self.adt)
        q = self.empty((n, vox), torch.float32)
        bs = bs_t.reshape(-1).contiguous()  # 1-element parameter, read on the device (no host sync)
        self.call("b200_scse_apply_fwd", _p(y.t), _p(g), _p(ws), _p(bs), n, vox, c, _p(out_t), _p(q))
        out = Act(out_t, ACT_NONE, 0.0)
        if DEBUG is not None:
            DEBUG.setdefault("se", {})[prefix] = (y.t, g, q)
        if self.record:
            def backward():
                dout = out.grad
                if dout is None:
                    return
                P = self.L.query("b200_scse_partials_count", n, vox, c)
                tmp = self.empty(y.t.shape, self.adt)
                part = self.empty((n, P, c, 2), torch.float32)
                dbs_part = self.empty((n * P, 1), torch.float32)
                self.call("b200_scse_bwd1", _p(dout), _p(y.t), _p(g), _p(q), _p(ws), n, vox, c, _p(tmp), _p(part), _p(dbs_part))
                sums2 = self.empty((n, c, 2), torch.float64)
                self.call("b200_partials_finalize", _p(part), n, P, c, _p(sums2))
                dbs = self.empty((1,), torch.float32)
                if not self.data_only:
                    self.call("b200_reduce_rows", _p(dbs_part), n * P, 1, _p(dbs))
                coef = self.empty((n, c, 3), torch.float32)
                dW1, db1 = torch.empty_like(W1), torch.empty_like(b1)
                dW2, db2 = torch.empty_like(W2), torch.empty_like(b2)
                dws = self.empty((c,), torch.float32)
                scratch = self.empty((n, 2, c), torch.float32)
                self.call("b200_se_gates_bwd", _p(sums2), _p(smean), _p(hh), _p(g), _p(W1), _p(W2), n, c, float(vox),
                          _p(coef), _p(dW1), _p(db1), _p(dW2), _p(db2), _p(dws), _p(scratch))
                self._add_param_grad(prefix + "cSE.fc1.weight", dW1)
                self._add_param_grad(prefix + "cSE.fc1.bias", db1)
                self._add_param_grad(prefix + "cSE.fc2.weight", dW2)
                self._add_param_grad(prefix + "cSE.fc2.bias", db2)
                self._add_param_grad(prefix + "sSE.conv.weight", dws.reshape(sd[prefix + "sSE.conv.weight"].shape))
                self._add_param_grad(prefix + "sSE.conv.bias", dbs)
                if y.requires_grad:
                    gy = self.empty(y.t.shape, self.adt)
                    self.call("b200_gn_bwd_apply", _p(tmp), _p(y.t), _p(coef), n, c, vox, y.act, y.slope, _p(y.grad), _p(gy))
                    y.grad = gy
                out.grad = None
            self.tape.append(backward)
        return out

    # ---------------------------------------------------------------- final 1x1x1 conv + sigmoid/softmax
    def final_conv(self, x, W, bias, final_act, wname, bname):
        n, d, h, w, c = x.dims
        vox = d * h * w
        cout = W.shape[0]
        W2 = W.reshape(cout, c).contiguous()
        logits = self.empty((n, cout, d, h, w), torch.float32)
        probs = self.empty((n, cout, d, h, w), torch.float32) if final_act != FINAL_NONE else None
        self.call("b200_final_conv_fwd", _p(x.t), n, vox, c, _p(W2), _p(bias), cout, final_act, _p(logits), _p(probs))

        def backward(dlogits):
            dlogits = dlogits.contiguous()
            P = self.L.query("b200_final_conv_bwd_partials_count", n, vox, c, cout)
            K = cout * c + cout
            partials = self.empty((n * P, K), torch.float32)
            dz = self.empty(x.t.shape, self.adt)
            self.call("b200_final_conv_bwd", _p(dlogits), _p(x.t), n, vox, c, _p(W2), cout, x.act, x.slope, _p(dz), _p(partials))
            if not self.data_only:   # (the per-block dW / db partials are a by-product of the dz kernel)
                red = self.empty((K,), torch.float32)
                self.call("b200_reduce_rows", _p(partials), n * P, K, _p(red))
                self._add_param_grad(wname, red[: cout * c].reshape(W.shape))
                if bias is not None:
                    self._add_param_grad(bname, red[cout * c:].clone())
            self.accumulate_grad(x, dz)
        return logits, probs, backward

    # ---------------------------------------------------------------- backward driver
    def run_backward(self):
        for fn in reversed(self.tape):
            fn()
        self.tape = []
