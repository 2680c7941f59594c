"""nn.Module surface of the B200 3D U-Net engine -- the drop-in for `pytorch3dunet.unet3d.model`.

Same constructor keywords, same parameter names / shapes (so reference checkpoints load with
`load_state_dict`, reference utils.py:59-60) and the same `forward(x, return_logits=False)` contract as the
reference (model.py:103-149), but every FLOP of forward and backward runs in libb200unet.so (hand-written
sm_100a CUDA) through `engine.Engine`.  The torch modules below (`nn.Conv3d`, `nn.GroupNorm`, ...) are used as
PARAMETER CONTAINERS only -- their own forward() is never called -- which also gives the reference's default
initialisation and RNG consumption order for free.

Reference constructors mirrored: UNet3D model.py:152-190, ResidualUNet3D :193-234, ResidualUNetSE3D :237-278,
get_model :361-363; block wiring buildingblocks.py:138-227 (DoubleConv), :310-384 (Encoder), :387-493 (Decoder),
:496-574 (create_encoders / create_decoders).
"""
from __future__ import annotations

import os
import threading

import torch
from torch import nn

from . import engine as E


class UnsupportedConfig(NotImplementedError):
    """A configuration that is valid for the reference but that the b200 engine does not build.  Raised at CONSTRUCTION time
    (never on the first batch); `install()`'s get_model catches it and constructs the reference's own class instead
    (SURVEY.md section 8(b): graph-level fallback, no Python re-implementation of arithmetic)."""


INTERP_MODES = ("nearest", "trilinear")   # InterpolateUpsampling modes built as kernels (buildingblocks.py:598-614)


def validate_layer_order(order, residual_block=False):
    """The order strings create_conv accepts (buildingblocks.py:44-94) that the engine fuses: [g]c[r|l|e], c g [r|l|e],
    c [r|l|e] g.  BatchNorm ('b') needs cross-replica running statistics and Dropout ('d'/'D') a device RNG stream
    matching torch's: both stay on the reference."""
    assert "c" in order, "Conv layer MUST be present"
    assert order[0] not in "rle", "Non-linearity cannot be the first operation in the layer"
    for ch in order:
        if ch not in "bgrlecdD":
            raise ValueError(f"Unsupported layer type '{ch}'. MUST be one of ['b', 'g', 'r', 'l', 'e', 'c', 'd', 'D']")
    if any(ch in order for ch in "bdD"):
        raise UnsupportedConfig(f"layer_order {order!r}: BatchNorm/Dropout layers are not built in the b200 engine")
    ic = order.index("c")
    pre, post = order[:ic], order[ic + 1:]
    acts = [ch for ch in post if ch in "rle"]
    if pre not in ("", "g") or order.count("c") != 1 or len(acts) > 1 or post.count("g") > 1 or (pre == "g" and "g" in post):
        raise UnsupportedConfig(f"layer_order {order!r} is not built in the b200 engine")


def number_of_features_per_level(init_channel_number, num_levels):
    """reference utils.py:110-112"""
    return [init_channel_number * 2 ** k for k in range(num_levels)]


# ----------------------------------------------------------------------------------------------------
# autograd bridge: one Function per call of a (sub)network; the engine's tape is the backward graph
# ----------------------------------------------------------------------------------------------------
class _EngineFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, program, n_inputs, names, grad_mode, sink, opts, *tensors):
        inputs, params = tensors[:n_inputs], tensors[n_inputs:]
        x0 = inputs[0]
        if not x0.is_cuda:
            raise RuntimeError("the b200 3D U-Net engine runs on CUDA tensors only (there is no CPU fallback)")
        for t in tensors:
            if t.dtype != torch.float32 or t.device != x0.device:
                raise RuntimeError("b200 engine: inputs and parameters must be float32 tensors on one CUDA device")
        # needs_input_grad mirrors tensor.requires_grad whatever the grad mode is, and grad mode is always off inside
        # Function.forward: the caller's mode comes in as an argument.  Under torch.no_grad() (the predictor's path,
        # reference predictor.py:164) nothing is taped, so no closure pins a layer's activations.
        needs_grad = bool(grad_mode) and any(ctx.needs_input_grad[6:])
        # every parameter frozen, an input requiring grad (a frozen network used as a loss, saliency maps, ...): the backward computes the
        # input gradient only -- no weight-gradient kernel, no parameter gradient, the flat gradient buffer is not touched
        data_only = needs_grad and not any(ctx.needs_input_grad[6 + n_inputs:])
        with torch.cuda.device(x0.device):
            eng = E.Engine(x0.device, record=needs_grad, sink=None if data_only else sink, operand_dtype=opts[0],
                           loss_scale=opts[1] if needs_grad else 1.0, data_only=data_only)
            sd = dict(zip(names, params))
            in_req = [needs_grad and bool(g) for g in ctx.needs_input_grad[6:6 + n_inputs]]
            outs, seed, input_grads = program(eng, [t.detach() for t in inputs], sd, in_req)
        ctx.eng, ctx.seed, ctx.input_grads = eng, seed, input_grads
        ctx.names, ctx.n_inputs = names, n_inputs
        ctx.param_meta = [(p.shape, p.dtype) for p in params]
        ctx.set_materialize_grads(False)
        ctx.device = x0.device
        h = _stats_holder()        # this (forward) thread's counters; backward runs on an autograd thread and writes into the same dict
        h["fwd"], h["bwd"], h["tape"] = eng.launches, 0, len(eng.tape)
        ctx.stats = h
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grad_outs):
        eng = ctx.eng
        if eng is None or not eng.record:
            raise RuntimeError("b200 engine: backward called twice or without a recorded forward")
        if torch.is_grad_enabled():
            # autograd runs backward with grad mode on exactly when create_graph=True: the engine's gradients are not themselves
            # differentiable, so a second-order term would silently come out as zero
            raise RuntimeError("b200 engine: double backward (create_graph=True) is not supported")
        with torch.cuda.device(ctx.device):
            eng.stream = torch.cuda.current_stream(ctx.device).cuda_stream
            l0 = eng.launches
            ctx.seed(eng, grad_outs)
            eng.run_backward()
            in_grads = ctx.input_grads(eng)
            ctx.stats["bwd"] = eng.launches - l0
        pg = eng.param_grads
        grads = []
        for (shape, dtype), name in zip(ctx.param_meta, ctx.names):
            g = pg.get(name)   # names written straight into the flat gradient buffer (eng.sunk) are not in pg: autograd gets None
            grads.append(None if g is None else g.reshape(shape))
        if eng.sink is not None:
            eng.sink.restore_grad_views()
        # drop everything the closures keep alive (activations of the last layer, ...) now instead of when the autograd node dies
        ctx.eng = ctx.seed = ctx.input_grads = None
        return (None, None, None, None, None, None) + tuple(in_grads) + tuple(grads)


_STATS = threading.local()


def _stats_holder():
    """launch counters of the most recent call made FROM THIS HOST THREAD (nn.DataParallel runs replicas on Python threads)"""
    h = getattr(_STATS, "h", None)
    if h is None:
        h = _STATS.h = {"fwd": 0, "bwd": 0, "tape": 0}
    return h


def _named_params(module):
    """[(qualified name, tensor)] in named_parameters() order, also for nn.DataParallel replicas: `replicate` empties each
    replica's `_parameters` and re-attaches the broadcast copies as plain attributes listed in `_former_parameters`
    (torch/nn/parallel/replicate.py), so `named_parameters()` of a replica is empty.  The reference wraps the model in
    DataParallel whenever more than one GPU is visible (trainer.py:203-204, predict.py:63-65)."""
    out = []
    replica = False
    for mname, m in module.named_modules():
        former = getattr(m, "_former_parameters", None)
        replica = replica or bool(former)
        items = list(m._parameters.items())
        if former:
            items += [(k, v) for k, v in former.items() if k not in m._parameters or m._parameters[k] is None]
        for k, p in items:
            if p is not None:
                out.append((f"{mname}.{k}" if mname else k, p))
    return out, replica


def _run(module, program, inputs):
    np_, replica = _named_params(module)
    names = tuple(k for k, _ in np_)
    # optim.FlatParameters registers itself on the model it was built from; DataParallel replicas share that attribute but must
    # not share the buffer (their gradients flow back through the broadcast instead)
    sink = None if replica else getattr(module, "_b200_grad_sink", None)
    opts = operand_options(module)
    return _EngineFn.apply(program, len(inputs), names, torch.is_grad_enabled(), sink, opts, *inputs, *(p for _, p in np_))


DEFAULT_OPERAND_DTYPE = os.environ.get("B200UNET_OPERAND_DTYPE", "bf16")
DEFAULT_LOSS_SCALE_FP16 = float(os.environ.get("B200UNET_LOSS_SCALE", "65536"))


def operand_options(module):
    """(operand dtype, loss scale) of a module: `module.operand_dtype` in {"bf16", "fp16"} (attribute, `operand_dtype=` constructor keyword
    of the models, or B200UNET_OPERAND_DTYPE) and, for fp16, `module.loss_scale` (default 65536: a mean-reduced loss over 4 M voxels
    seeds gradients of ~2e-7, below fp16's normal range; parameter gradients are returned UNscaled)."""
    dt = getattr(module, "operand_dtype", None) or DEFAULT_OPERAND_DTYPE
    if dt in ("fp16", "f16", "float16", "half"):
        return ("fp16", float(getattr(module, "loss_scale", None) or DEFAULT_LOSS_SCALE_FP16))
    if dt not in ("bf16", "bfloat16"):
        raise ValueError(f"operand_dtype {dt!r}: expected 'bf16' or 'fp16'")
    return ("bf16", 1.0)


def last_launch_counts():
    """(forward, backward) number of engine kernels launched by the most recent call (of this host thread)."""
    h = _stats_holder()
    return h["fwd"], h["bwd"]


def last_tape_length():
    """number of backward closures the most recent forward recorded (0 under torch.no_grad())"""
    return _stats_holder()["tape"]


# ----------------------------------------------------------------------------------------------------
# engine programs for the blocks
# ----------------------------------------------------------------------------------------------------
def _has_pre_gn(order):
    return "g" in order and order.index("g") < order.index("c")


def run_double_conv(eng, x, sd, prefix, order, groups, out_stats):
    h = eng.single_conv(x, sd, prefix + "SingleConv1.", order, groups, want_stats=_has_pre_gn(order))
    return eng.single_conv(h, sd, prefix + "SingleConv2.", order, groups, want_stats=out_stats)


def run_res_block(eng, x, sd, prefix, order, groups, out_stats):
    """ResNetBlock.forward, reference buildingblocks.py:277-288: conv1 (1x1x1 + bias, or Identity) -> conv2 (order) ->
    conv3 (order without the non-linearity) -> += residual -> non-linearity.  The add + activation are the epilogue of
    conv3's tensor-core kernel."""
    pre_gn = _has_pre_gn(order)
    if (prefix + "conv1.weight") in sd:
        residual = eng.pointwise(x, sd[prefix + "conv1.weight"], sd.get(prefix + "conv1.bias"), prefix + "conv1.weight",
                                 prefix + "conv1.bias", want_stats=pre_gn)
    else:
        if isinstance(x, E.InputF32):
            raise NotImplementedError("ResNetBlock with in_channels == out_channels directly on the fp32 network input")
        residual = x
    n_order = order.replace("r", "").replace("e", "").replace("l", "")
    if "l" in order:
        block_act = (E.ACT_LEAKY, 0.1)   # buildingblocks.py:271: slope 0.1 here (create_conv's LeakyReLU uses 0.01)
    elif "e" in order:
        block_act = (E.ACT_ELU, 1.0)
    else:
        block_act = (E.ACT_RELU, 0.0)
    h = eng.single_conv(residual, sd, prefix + "conv2.", order, groups, want_stats=_has_pre_gn(n_order))
    return eng.single_conv(h, sd, prefix + "conv3.", n_order, groups, want_stats=out_stats, residual=residual, final_act=block_act)


def run_basic(eng, x, sd, prefix, spec, out_stats=False):
    if spec["basic"] == "double":
        return run_double_conv(eng, x, sd, prefix, spec["layer_order"], spec["num_groups"], out_stats)
    if spec["basic"] == "res":
        return run_res_block(eng, x, sd, prefix, spec["layer_order"], spec["num_groups"], out_stats)
    if spec["basic"] == "res_se":
        # ResNetBlockSE.forward (buildingblocks.py:304-307): ResNetBlock then scSE; the SE means reuse the block output's partial sums
        y = run_res_block(eng, x, sd, prefix, spec["layer_order"], spec["num_groups"], True)
        return eng.scse(y, sd, prefix + "se_module.")
    raise NotImplementedError(f"basic module {spec['basic']!r}")


def run_join(eng, enc, x, sd, prefix, spec, want_stats):
    """Decoder.forward up to the basic module, reference buildingblocks.py:482-493"""
    wkey = prefix + "upsampling.upsample.conv_transposed.weight"
    if spec["upsample"] in INTERP_MODES and spec["concat"]:
        # only DoubleConv consumes the joined tensor through a single 3x3x3 conv, which lets it stay virtual
        return eng.upcat(enc, x, want_stats=want_stats, allow_virtual=spec["basic"] == "double", mode=spec["upsample"])
    if spec["upsample"] == "deconv" and not spec["concat"]:
        return eng.deconv_up_add(enc, x, sd[wkey], wkey, want_stats=want_stats)
    if spec["upsample"] == "deconv":
        # explicit upsample='deconv': the transposed conv's (2d-1)^3 output is nearest-resized to the encoder size and concatenated
        return eng.upcat(enc, eng.deconv(x, sd[wkey], wkey), want_stats=want_stats)
    raise UnsupportedConfig(f"decoder upsample={spec['upsample']!r} concat={spec['concat']} is not built in the b200 engine")


def run_unet(eng, x, sd, spec):
    """AbstractUNet._forward_logits, reference model.py:123-149."""
    order = spec["layer_order"]
    pre_gn = _has_pre_gn(order)
    nlev = len(spec["f_maps"])
    feats = []
    for i in range(nlev):
        if i > 0:
            x = eng.maxpool(x, want_stats=pre_gn)
        # with a virtual concat (nearest + concat into a DoubleConv that starts with a GroupNorm) the statistics of the joined tensor
        # are those of its two parts: have their producers emit them instead of re-reading the tensors
        join_stats = pre_gn and spec["upsample"] == "nearest" and spec["concat"] and spec["basic"] == "double"
        x = run_basic(eng, x, sd, f"encoders.{i}.basic_module.", spec, out_stats=join_stats)
        feats.insert(0, x)
    ndec = len(feats) - 1
    for i, enc in enumerate(feats[1:]):
        x = run_join(eng, enc, x, sd, f"decoders.{i}.", spec, pre_gn)
        x = run_basic(eng, x, sd, f"decoders.{i}.basic_module.", spec, out_stats=join_stats and i + 1 < ndec)
    final = E.FINAL_NONE
    if spec["is_segmentation"]:
        final = E.FINAL_SIGMOID if spec["final_sigmoid"] else E.FINAL_SOFTMAX
    return eng.final_conv(x, sd["final_conv.weight"], sd.get("final_conv.bias"), final, "final_conv.weight", "final_conv.bias")


# ----------------------------------------------------------------------------------------------------
# parameter containers with the reference's names
# ----------------------------------------------------------------------------------------------------
def _conv_layers(in_channels, out_channels, order, num_groups, kernel_size=3, padding=1):
    """(name, module) list with the names create_conv uses (buildingblocks.py:44-94); parameter-free layers
    (activations) are kept so that printing the model reads like the reference's."""
    assert "c" in order, "Conv layer MUST be present"
    assert order[0] not in "rle", "Non-linearity cannot be the first operation in the layer"
    out = []
    for i, ch in enumerate(order):
        if ch == "r":
            out.append(("ReLU", nn.ReLU(inplace=True)))
        elif ch == "l":
            out.append(("LeakyReLU", nn.LeakyReLU(inplace=True)))
        elif ch == "e":
            out.append(("ELU", nn.ELU(inplace=True)))
        elif ch == "c":
            out.append(("conv", nn.Conv3d(in_channels, out_channels, kernel_size, padding=padding,
                                          bias=not ("g" in order or "b" in order))))
        elif ch == "g":
            c = in_channels if i < order.index("c") else out_channels
            g = 1 if c < num_groups else num_groups
            assert c % g == 0, f"Expected number of channels in input to be divisible by num_groups. num_channels={c}, num_groups={g}"
            out.append(("groupnorm", nn.GroupNorm(num_groups=g, num_channels=c)))
        else:
            raise NotImplementedError(f"layer type {ch!r} in layer_order={order!r} is not supported by the b200 engine "
                                      "(supported: c, g, r, l, e)")
    return out


class _EngineModule(nn.Module):
    """Block-level modules are callable on NCDHW fp32 tensors with C % 8 == 0 (parity tests, custom nets)."""

    def _program(self):
        raise NotImplementedError

    def forward(self, *inputs):
        prog = self._program()

        def program(eng, ins, sd, in_req):
            acts = [eng.input_bf16(t, r) for t, r in zip(ins, in_req)]
            y = prog(eng, acts, sd)
            out = eng.to_ncdhw_f32(y.t)

            def seed(eng, grads):
                if grads[0] is not None:
                    eng.grad_from_ncdhw(y, grads[0] * eng.loss_scale if eng.loss_scale != 1.0 else grads[0])

            def input_grads(eng):
                res = []
                for a, r in zip(acts, in_req):
                    if r and a.grad is not None:
                        gi = eng.to_ncdhw_f32(a.grad)
                        res.append(gi / eng.loss_scale if eng.loss_scale != 1.0 else gi)
                    elif r:
                        res.append(torch.zeros((a.t.shape[0], a.t.shape[4]) + tuple(a.t.shape[1:4]), device=a.t.device))
                    else:
                        res.append(None)
                return res
            return [out], seed, input_grads
        return _run(self, program, list(inputs))[0]


class SingleConv(_EngineModule):
    def __init__(self, in_channels, out_channels, kernel_size=3, order="gcr", num_groups=8, padding=1, dropout_prob=0.1, is3d=True):
        super().__init__()
        if not is3d or kernel_size != 3 or padding != 1:
            raise UnsupportedConfig("the b200 engine implements 3-D 3x3x3 convolutions with padding 1")
        validate_layer_order(order)
        self.order, self.num_groups = order, num_groups
        for name, m in _conv_layers(in_channels, out_channels, order, num_groups):
            self.add_module(name, m)

    def _program(self):
        return lambda eng, acts, sd: eng.single_conv(acts[0], sd, "", self.order, self.num_groups)


class DoubleConv(_EngineModule):
    def __init__(self, in_channels, out_channels, encoder, kernel_size=3, order="gcr", num_groups=8, padding=1, upscale=2,
                 dropout_prob=0.1, is3d=True):
        super().__init__()
        if encoder:
            mid = out_channels if upscale == 1 else out_channels // 2
            mid = max(mid, in_channels)
        else:
            mid = out_channels
        self.order, self.num_groups = order, num_groups
        self.SingleConv1 = SingleConv(in_channels, mid, kernel_size, order, num_groups, padding, is3d=is3d)
        self.SingleConv2 = SingleConv(mid, out_channels, kernel_size, order, num_groups, padding, is3d=is3d)

    def _program(self):
        return lambda eng, acts, sd: run_double_conv(eng, acts[0], sd, "", self.order, self.num_groups, False)


class _Marker(nn.Module):
    """parameter-free placeholder so the module tree prints like the reference's (pooling / upsampling)."""

    def __init__(self, text):
        super().__init__()
        self.text = text

    def extra_repr(self):
        return self.text


class Encoder(_EngineModule):
    def __init__(self, in_channels, out_channels, apply_pooling=True, basic="double", conv_layer_order="gcr", num_groups=8,
                 upscale=2, pool_type="max"):
        super().__init__()
        assert pool_type in ("max", "avg")   # buildingblocks.py:352
        self.pool_type = pool_type
        self.pooling = _Marker(f"{'Max' if pool_type == 'max' else 'Avg'}Pool3d(kernel_size=2) [b200 kernel]") if apply_pooling else None
        self.spec = dict(basic=basic, layer_order=conv_layer_order, num_groups=num_groups)
        self.basic_module = _make_basic(basic, in_channels, out_channels, True, conv_layer_order, num_groups, upscale)

    def _program(self):
        def prog(eng, acts, sd):
            x = acts[0]
            if self.pooling is not None:
                x = eng.maxpool(x, want_stats=_has_pre_gn(self.spec["layer_order"]), kind=self.pool_type)
            return run_basic(eng, x, sd, "basic_module.", self.spec)
        return prog


class Decoder(_EngineModule):
    def __init__(self, in_channels, out_channels, basic="double", conv_layer_order="gcr", num_groups=8, upsample="nearest",
                 concat=True):
        super().__init__()
        if upsample == "deconv":
            self.upsampling = _DeconvHolder(in_channels, out_channels)
            if not concat:
                in_channels = out_channels  # adapt_channels, reference buildingblocks.py:466-468
        else:
            self.upsampling = _Marker(f"{upsample} to the encoder feature size [fused b200 kernel]")
        self.spec = dict(basic=basic, layer_order=conv_layer_order, num_groups=num_groups, upsample=upsample, concat=concat)
        self.basic_module = _make_basic(basic, in_channels, out_channels, False, conv_layer_order, num_groups, 2)

    def forward(self, encoder_features, x):
        return super().forward(encoder_features, x)

    def _program(self):
        def prog(eng, acts, sd):
            j = run_join(eng, acts[0], acts[1], sd, "", self.spec, _has_pre_gn(self.spec["layer_order"]))
            return run_basic(eng, j, sd, "basic_module.", self.spec)
        return prog


class ResNetBlock(_EngineModule):
    """parameter names of the reference's ResNetBlock (buildingblocks.py:230-275): conv1 (1x1x1 or Identity), conv2, conv3"""

    def __init__(self, in_channels, out_channels, kernel_size=3, order="cge", num_groups=8, is3d=True, **kwargs):
        super().__init__()
        self.conv1 = nn.Conv3d(in_channels, out_channels, 1) if in_channels != out_channels else nn.Identity()
        self.order, self.num_groups = order, num_groups
        self.conv2 = SingleConv(out_channels, out_channels, kernel_size=kernel_size, order=order, num_groups=num_groups, is3d=is3d)
        n_order = order.replace("r", "").replace("e", "").replace("l", "")
        self.conv3 = SingleConv(out_channels, out_channels, kernel_size=kernel_size, order=n_order, num_groups=num_groups, is3d=is3d)
        if "l" in order:
            self.non_linearity = nn.LeakyReLU(negative_slope=0.1, inplace=True)
        elif "e" in order:
            self.non_linearity = nn.ELU(inplace=True)
        else:
            self.non_linearity = nn.ReLU(inplace=True)

    def _program(self):
        return lambda eng, acts, sd: run_res_block(eng, acts[0], sd, "", self.order, self.num_groups, False)


class _ChannelSE(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.fc1 = nn.Linear(c, c, bias=True)
        self.fc2 = nn.Linear(c, c, bias=True)


class _SpatialSE(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv = nn.Conv3d(c, 1, 1)


class _SCSE(nn.Module):
    """parameters of ChannelSpatialSELayer3D(num_channels, reduction_ratio=1) (se.py:96-111), same creation order"""

    def __init__(self, c):
        super().__init__()
        self.cSE = _ChannelSE(c)
        self.sSE = _SpatialSE(c)


class ResNetBlockSE(ResNetBlock):
    def __init__(self, in_channels, out_channels, kernel_size=3, order="cge", num_groups=8, se_module="scse", **kwargs):
        super().__init__(in_channels, out_channels, kernel_size=kernel_size, order=order, num_groups=num_groups)
        if se_module != "scse":
            raise NotImplementedError("only se_module='scse' (the ResNetBlockSE default) is built in the b200 engine")
        self.se_module = _SCSE(out_channels)

    def _program(self):
        def prog(eng, acts, sd):
            y = run_res_block(eng, acts[0], sd, "", self.order, self.num_groups, True)
            return eng.scse(y, sd, "se_module.")
        return prog


class _DeconvHolder(nn.Module):
    """`upsampling.upsample.conv_transposed.weight` (TransposeConvUpsampling.Upsample, buildingblocks.py:633-664)"""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.upsample = nn.Module()
        self.upsample.conv_transposed = nn.ConvTranspose3d(in_channels, out_channels, kernel_size=3, stride=2, padding=1, bias=False)


def _make_basic(basic, cin, cout, encoder, order, groups, upscale):
    if basic == "double":
        return DoubleConv(cin, cout, encoder, order=order, num_groups=groups, upscale=upscale)
    if basic == "res":
        return ResNetBlock(cin, cout, order=order, num_groups=groups)
    if basic == "res_se":
        return ResNetBlockSE(cin, cout, order=order, num_groups=groups)
    raise NotImplementedError(f"basic module {basic!r}")


# ----------------------------------------------------------------------------------------------------
# models
# ----------------------------------------------------------------------------------------------------
class AbstractUNet(nn.Module):
    """Same construction order as the reference (encoders, decoders, final_conv) => same default init under a seed."""

    def __init__(self, in_channels, out_channels, final_sigmoid, basic, f_maps=64, layer_order="gcr", num_groups=8, num_levels=4,
                 is_segmentation=True, conv_kernel_size=3, pool_kernel_size=2, conv_padding=1, conv_upscale=2, upsample="default",
                 dropout_prob=0.1, is3d=True, operand_dtype=None, loss_scale=None):
        super().__init__()
        # b200 extensions (not reference keywords): 16-bit type of activations / tensor-core operands and the fp16 loss scale
        self.operand_dtype, self.loss_scale = operand_dtype, loss_scale
        operand_options(self)  # validate
        if not is3d:
            raise UnsupportedConfig("2-D models are out of scope of the b200 engine (SURVEY.md section 2, row 1)")
        if conv_kernel_size != 3 or pool_kernel_size != 2 or conv_padding != 1:
            raise UnsupportedConfig("the b200 engine implements conv 3x3x3 / padding 1 / pool 2 (what UNet3D & co. always use)")
        validate_layer_order(layer_order)
        if isinstance(f_maps, int):
            f_maps = number_of_features_per_level(f_maps, num_levels=num_levels)
        assert isinstance(f_maps, (list, tuple))
        assert len(f_maps) > 1, "Required at least 2 levels in the U-Net"
        if "g" in layer_order:
            assert num_groups is not None, "num_groups must be specified if GroupNorm is used"
        f_maps = list(f_maps)
        concat = True   # Decoder.__init__, buildingblocks.py:431-468: only 'default' on a residual block switches to the sum join
        if upsample == "default":
            if basic == "double":
                upsample, concat = "nearest", True
            else:
                upsample, concat = "deconv", False
        elif upsample not in INTERP_MODES + ("deconv",):
            # None / 'none' (no upsampling), 'area' (adaptive average pooling), 'linear' / 'bilinear' (not 5-D modes)
            raise UnsupportedConfig(f"upsample={upsample!r} is not built in the b200 engine (built: 'default', 'nearest', 'trilinear', 'deconv')")
        if any(f % 8 for f in f_maps):
            raise UnsupportedConfig(f"f_maps={f_maps}: the engine's activations need channel counts that are multiples of 8")
        self.spec = dict(basic=basic, f_maps=f_maps, layer_order=layer_order, num_groups=num_groups, upsample=upsample,
                         concat=concat, is_segmentation=is_segmentation, final_sigmoid=final_sigmoid,
                         in_channels=in_channels, out_channels=out_channels)
        self.encoders = nn.ModuleList(
            Encoder(in_channels if i == 0 else f_maps[i - 1], f, apply_pooling=i > 0, basic=basic,
                    conv_layer_order=layer_order, num_groups=num_groups, upscale=conv_upscale)
            for i, f in enumerate(f_maps))
        rf = f_maps[::-1]
        decs = []
        for i in range(len(rf) - 1):
            cin = rf[i] + rf[i + 1] if (basic == "double" and upsample != "deconv") else rf[i]
            decs.append(Decoder(cin, rf[i + 1], basic=basic, conv_layer_order=layer_order, num_groups=num_groups,
                                upsample=upsample, concat=concat))
        self.decoders = nn.ModuleList(decs)
        self.final_conv = nn.Conv3d(f_maps[0], out_channels, 1)
        if is_segmentation:
            self.final_activation = nn.Sigmoid() if final_sigmoid else nn.Softmax(dim=1)
        else:
            self.final_activation = None

    def forward(self, x, return_logits=False):
        spec = self.spec
        if x.dim() != 5 or x.shape[1] != spec["in_channels"]:
            raise ValueError(f"expected input (N,{spec['in_channels']},D,H,W), got {tuple(x.shape)}")
        if x.dtype != torch.float32:
            x = x.float()

        def program(eng, ins, sd, in_req):
            xin = eng.input_f32(ins[0], requires_grad=in_req[0])
            logits, probs, final_bwd = run_unet(eng, xin, sd, spec)
            final = spec["is_segmentation"]
            # the closure must not hold the tensor OBJECT that forward returns: that object gets grad_fn = this autograd node,
            # which holds the closure -> a reference cycle that keeps a step's activations alive until Python's cyclic GC runs
            probs_saved = probs.detach() if probs is not None else None

            def seed(eng, grads):
                g_logits = grads[0]
                g_probs = grads[1] if final and len(grads) > 1 else None
                if g_probs is not None:
                    # chain rule through the final activation (tiny, C_out channels); only when the loss uses probabilities
                    if spec["final_sigmoid"]:
                        t = g_probs * probs_saved * (1 - probs_saved)
                    else:
                        t = probs_saved * (g_probs - (g_probs * probs_saved).sum(dim=1, keepdim=True))
                    g_logits = t if g_logits is None else g_logits + t
                if g_logits is not None:
                    final_bwd(g_logits * eng.loss_scale if eng.loss_scale != 1.0 else g_logits)

            def input_grads(eng):
                # fp32 NCDHW, unscaled; zeros when the loss did not depend on the output
                if not in_req[0]:
                    return [None]
                return [xin.grad if xin.grad is not None else torch.zeros_like(ins[0])]
            outs = [logits, probs] if final else [logits]
            return outs, seed, input_grads
        res = _run(self, program, [x])
        logits = res[0]
        out = res[1] if spec["is_segmentation"] else logits
        if return_logits:
            return out, logits
        return out


class UNet3D(AbstractUNet):
    def __init__(self, in_channels, out_channels, final_sigmoid=True, f_maps=64, layer_order="gcr", num_groups=8, num_levels=4,
                 is_segmentation=True, conv_padding=1, conv_upscale=2, upsample="default", dropout_prob=0.1, **kwargs):
        super().__init__(in_channels, out_channels, final_sigmoid, "double", f_maps=f_maps, layer_order=layer_order,
                         num_groups=num_groups, num_levels=num_levels, is_segmentation=is_segmentation,
                         conv_padding=conv_padding, conv_upscale=conv_upscale, upsample=upsample, dropout_prob=dropout_prob,
                         operand_dtype=kwargs.get("operand_dtype"), loss_scale=kwargs.get("loss_scale"))


class ResidualUNet3D(AbstractUNet):
    def __init__(self, in_channels, out_channels, final_sigmoid=True, f_maps=64, layer_order="gcr", num_groups=8, num_levels=5,
                 is_segmentation=True, conv_padding=1, conv_upscale=2, upsample="default", dropout_prob=0.1, **kwargs):
        super().__init__(in_channels, out_channels, final_sigmoid, "res", f_maps=f_maps, layer_order=layer_order,
                         num_groups=num_groups, num_levels=num_levels, is_segmentation=is_segmentation,
                         conv_padding=conv_padding, conv_upscale=conv_upscale, upsample=upsample, dropout_prob=dropout_prob,
                         operand_dtype=kwargs.get("operand_dtype"), loss_scale=kwargs.get("loss_scale"))


class ResidualUNetSE3D(AbstractUNet):
    def __init__(self, in_channels, out_channels, final_sigmoid=True, f_maps=64, layer_order="gcr", num_groups=8, num_levels=5,
                 is_segmentation=True, conv_padding=1, conv_upscale=2, upsample="default", dropout_prob=0.1, **kwargs):
        super().__init__(in_channels, out_channels, final_sigmoid, "res_se", f_maps=f_maps, layer_order=layer_order,
                         num_groups=num_groups, num_levels=num_levels, is_segmentation=is_segmentation,
                         conv_padding=conv_padding, conv_upscale=conv_upscale, upsample=upsample, dropout_prob=dropout_prob,
                         operand_dtype=kwargs.get("operand_dtype"), loss_scale=kwargs.get("loss_scale"))


_MODELS = {"UNet3D": UNet3D, "ResidualUNet3D": ResidualUNet3D, "ResidualUNetSE3D": ResidualUNetSE3D}


def get_model(model_config):
    """reference model.py:361-363: class by name, whole config dict splatted into the constructor."""
    name = model_config["name"]
    if name not in _MODELS:
        raise NotImplementedError(f"model {name!r} is not provided by the b200 engine (3-D models only: {sorted(_MODELS)})")
    return _MODELS[name](**model_config)


def is_model_2d(model):
    return False
