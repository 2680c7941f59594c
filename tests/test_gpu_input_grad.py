"""GPU: the gradient with respect to the network input (fp32 NCDHW, csrc/input_grad.cu) and the input-gradient-only backward of a
frozen model.  Model-level gradients are judged against the oracle evaluated at the engine's activation pattern and pool argmax, as
the parameter gradients are in test_gpu_model.py; the reference's own grad_x (goldens) is printed as information."""
import pytest
import torch
import torch.nn.functional as F

from tests.gpu_util import p, rel_l2, stream
from tests.helpers import load_golden
from tests.test_gpu_model import E2E_GRAD_TOL, EXTRA_MODEL_CASES, MODEL_CASES, _engine_masks, _engine_pool_idx

pytestmark = pytest.mark.gpu

ALL_CASES = {**MODEL_CASES, **EXTRA_MODEL_CASES}
# last_launch_counts() (forward, backward) of one training step (_small_step) before the input gradient existed, read on a B200
PARENT_COUNTS = {
    "UNet3D/auto": (47, 113),
    "UNet3D/direct": (39, 122),
    "ResidualUNet3D/auto": (46, 142),
    "ResidualUNet3D/direct": (48, 153),
}


def _worst_param_grad(model, ograds):
    worst = ("", 0.0)
    for k, prm in model.named_parameters():
        assert prm.grad is not None, k
        g = ograds[k]
        floor = 5e-3 * ograds[k.rsplit("groupnorm", 1)[0] + "conv.weight"].norm().item() if "groupnorm" in k else 0.0
        err = (prm.grad.detach().cpu().double() - g.double()).norm().item()
        r = rel_l2(prm.grad.cpu(), g)
        if err > floor and r > worst[1] and g.norm() > 1e-4:
            worst = (k, r)
    return worst


def _engine_vs_oracle(cfg, loss_name, sd, x, target, monkeypatch, frozen=False):
    """engine forward + backward with x.requires_grad (parameters trainable or frozen) and the oracle at the engine's pattern"""
    import pytorch3dunet_b200 as P
    from pytorch3dunet_b200 import engine as E
    from oracle import unet3d_oracle as O
    model = P.get_model(cfg)
    model.load_state_dict(sd)
    model = model.cuda()
    if frozen:
        model.requires_grad_(False)
    xe = x.cuda().requires_grad_(True)
    monkeypatch.setattr(E, "DEBUG", {})
    out, logits = model(xe, return_logits=True)
    getattr(P.losses, loss_name)(logits, target.cuda()).backward()
    torch.cuda.synchronize()
    masks, pidx = _engine_masks(E), _engine_pool_idx(E)
    monkeypatch.setattr(E, "DEBUG", None)
    osd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    ox = x.clone().requires_grad_(True)
    o_out, o_logits = O.forward(osd, cfg, ox, masks=masks, pool_idx=pidx)
    getattr(O, loss_name)(o_logits, target).backward()
    return model, xe.grad, ox.grad, {k: v.grad for k, v in osd.items()}


@pytest.mark.parametrize("impl", ["direct", "auto"])
@pytest.mark.parametrize("name", sorted(ALL_CASES))
def test_model_input_grad_matches_oracle(name, impl, monkeypatch):
    """grad_x of every model golden (all three families; gcr, cgr, cl, crg, gcl, gce, cge; C_in 1 and 2; odd sizes; nearest, trilinear and
    deconv joins) against the oracle, with the parameter gradients of the same run"""
    monkeypatch.setenv("B200UNET_CONV_IMPL", impl)
    cfg, loss_name = ALL_CASES[name]
    rec, sd, _ = load_golden(name)
    model, gx, ogx, ograds = _engine_vs_oracle(cfg, loss_name, sd, rec["x"], rec["target"], monkeypatch)
    assert gx is not None and gx.dtype == torch.float32 and gx.shape == rec["x"].shape
    worst = _worst_param_grad(model, ograds)
    rep = {"grad_x": rel_l2(gx.cpu(), ogx), "grad_x_vs_golden(info)": rel_l2(gx.cpu(), rec["grad_x"]), "worst_param": worst}
    print(name, impl, rep)
    assert rep["grad_x"] < E2E_GRAD_TOL, rep
    assert worst[1] < E2E_GRAD_TOL, worst


@pytest.mark.parametrize("name", ["unet3d_f16_l3_s16", "resunet3d_f16_l3_s16", "resunetse3d_f16_l2_gce", "unet3d_f16_l3_odd"])
def test_frozen_model_input_grad(name, monkeypatch):
    """every parameter frozen: grad_x agrees with the full backward's, no weight-gradient kernel runs, no parameter gradient is written,
    a flat gradient buffer stays byte-identical.  Not to rounding order: where a GroupNorm is folded into the next conv, the full
    backward takes its backward sums from the fp32 wgrad accumulators, the frozen one from the 16-bit data gradient (measured on a B200:
    0 where every GroupNorm is explicit, ~8e-3 otherwise, while both sit ~1e-2 from the oracle, test_frozen_model_matches_oracle)"""
    import pytorch3dunet_b200 as P
    from pytorch3dunet_b200 import engine as E
    from pytorch3dunet_b200.optim import FlatParameters
    cfg, loss_name = ALL_CASES[name]
    rec, sd, _ = load_golden(name)
    x, t = rec["x"].cuda(), rec["target"].cuda()

    model = P.get_model(cfg)
    model.load_state_dict(sd)
    model = model.cuda()
    xf = x.clone().requires_grad_(True)
    getattr(P.losses, loss_name)(model(xf, return_logits=True)[1], t).backward()
    g_full = xf.grad.clone()

    model.zero_grad(set_to_none=True)
    flat = FlatParameters(model)
    flat.grad.fill_(7.0)
    before = flat.grad.clone()
    model.requires_grad_(False)
    xd = x.clone().requires_grad_(True)
    monkeypatch.setattr(E, "TIMING", [])
    getattr(P.losses, loss_name)(model(xd, return_logits=True)[1], t).backward()
    torch.cuda.synchronize()
    tags = [rec_[0] for rec_ in E.TIMING]
    monkeypatch.setattr(E, "TIMING", None)
    r = rel_l2(xd.grad, g_full)
    print(name, "frozen vs full grad_x rel", f"{r:.2e}", "timed launches", sorted(set(tags)))
    assert r < 2e-2, r
    assert not any(tg.startswith("wgrad") for tg in tags), tags
    assert torch.equal(flat.grad, before)
    for k, prm in model.named_parameters():   # the flat views are re-attached by FlatParameters, never written
        assert prm.grad is None or torch.equal(prm.grad, before[flat.range_of[k][0]:flat.range_of[k][0] + prm.numel()].view_as(prm)), k


def test_frozen_model_matches_oracle(monkeypatch):
    """the data-gradient-only backward against the oracle (GroupNorm-backward sums from the data gradients)"""
    for name in ["unet3d_f16_l3_s16", "resunetse3d_f16_l3_s16", "unet3d_f16_l2_cgr"]:
        cfg, loss_name = ALL_CASES[name]
        rec, sd, _ = load_golden(name)
        model, gx, ogx, _ = _engine_vs_oracle(cfg, loss_name, sd, rec["x"], rec["target"], monkeypatch, frozen=True)
        assert all(prm.grad is None for prm in model.parameters())
        r = rel_l2(gx.cpu(), ogx)
        print(name, "frozen grad_x vs oracle", f"{r:.2e}")
        assert r < E2E_GRAD_TOL, (name, r)


def test_two_models_in_sequence(monkeypatch):
    """a denoising-style U-Net (is_segmentation=False) feeding a segmentation U-Net, trained end to end: the loss reaches the first
    model's parameters"""
    import pytorch3dunet_b200 as P
    from pytorch3dunet_b200 import engine as E
    from oracle import unet3d_oracle as O
    cfg1 = dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2, is_segmentation=False)
    cfg2 = dict(name="ResidualUNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2)
    torch.manual_seed(3)
    m1, m2 = P.get_model(cfg1), P.get_model(cfg2)
    sd1 = {k: v.clone() for k, v in m1.state_dict().items()}
    sd2 = {k: v.clone() for k, v in m2.state_dict().items()}
    m1, m2 = m1.cuda(), m2.cuda()
    x = torch.rand(1, 1, 24, 32, 32)
    t = (torch.rand(1, 1, 24, 32, 32) > 0.5).float()
    monkeypatch.setattr(E, "DEBUG", {})
    h = m1(x.cuda())
    masks1, pidx1 = _engine_masks(E), _engine_pool_idx(E)
    monkeypatch.setattr(E, "DEBUG", {})
    out, logits = m2(h, return_logits=True)
    masks2, pidx2 = _engine_masks(E), _engine_pool_idx(E)
    monkeypatch.setattr(E, "DEBUG", None)
    P.losses.bce_dice_loss(logits, t.cuda()).backward()
    torch.cuda.synchronize()
    osd1 = {k: v.clone().requires_grad_(True) for k, v in sd1.items()}
    osd2 = {k: v.clone().requires_grad_(True) for k, v in sd2.items()}
    oh, _ = O.forward(osd1, cfg1, x, masks=masks1, pool_idx=pidx1)
    _, ol = O.forward(osd2, cfg2, oh, masks=masks2, pool_idx=pidx2)
    O.bce_dice_loss(ol, t).backward()
    w1 = _worst_param_grad(m1, {k: v.grad for k, v in osd1.items()})
    w2 = _worst_param_grad(m2, {k: v.grad for k, v in osd2.items()})
    print("chained: first model", w1, "second model", w2)
    assert w1[1] < E2E_GRAD_TOL and w2[1] < E2E_GRAD_TOL, (w1, w2)


@pytest.mark.parametrize("name", ["unet3d_f16_l3_s16", "resunet3d_f16_l3_s16"])
def test_fp16_operands_input_grad(name, monkeypatch):
    """fp16 build: the input gradient comes back unscaled (1/loss_scale folded into the first layer's epilogue)"""
    cfg, loss_name = ALL_CASES[name]
    rec, sd, _ = load_golden(name)
    _, gx, ogx, _ = _engine_vs_oracle({**cfg, "operand_dtype": "fp16"}, loss_name, sd, rec["x"], rec["target"], monkeypatch)
    r = rel_l2(gx.cpu(), ogx)
    print(name, "fp16 grad_x", f"{r:.2e}")
    assert r < E2E_GRAD_TOL, r


def test_double_backward_is_refused():
    import pytorch3dunet_b200 as P
    torch.manual_seed(0)
    model = P.get_model(dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2)).cuda()
    x = torch.rand(1, 1, 16, 16, 16, device="cuda", requires_grad=True)
    with pytest.raises(RuntimeError, match="double backward"):
        torch.autograd.grad(model(x).sum(), x, create_graph=True)


def test_cfg2_input_grad_vs_fp32_oracle():
    """BASELINE configs[1] (UNet3D f_maps=32, 4 levels, 2x1x128^3, BCEDice): grad_x against the fp32 oracle on the same GPU (TF32 off)
    at the engine's activation pattern, with the gradient bound of test_gpu_parity_configs.py"""
    import pytorch3dunet_b200 as P
    from pytorch3dunet_b200 import engine as E
    from oracle import unet3d_oracle as O
    from tests.test_gpu_parity_configs import GRAD_TOL
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    cfg = dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=32, num_levels=4)
    torch.manual_seed(0)
    model = P.get_model(cfg).cuda()
    x = torch.rand(2, 1, 128, 128, 128, device="cuda")
    t = (torch.rand(2, 1, 128, 128, 128, device="cuda") > 0.5).float()
    xe = x.clone().requires_grad_(True)
    E.DEBUG = {}
    try:
        _, logits = model(xe, return_logits=True)
        P.losses.bce_dice_loss(logits, t).backward()
        torch.cuda.synchronize()
        masks = {k: (v > 0).permute(0, 4, 1, 2, 3) for k, v in E.DEBUG["fwd"].items()}
        pidx = [F.max_pool3d(v.float().permute(0, 4, 1, 2, 3), 2, return_indices=True)[1] for v in E.DEBUG.get("pool", [])]
    finally:
        E.DEBUG = None
    gx = xe.grad.detach().clone()
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in model.state_dict().items()}
    del model, logits
    torch.cuda.empty_cache()
    ox = x.clone().requires_grad_(True)
    _, ol = O.forward(sd, cfg, ox, masks=masks, pool_idx=pidx)
    O.bce_dice_loss(ol, t).backward()
    r = rel_l2(gx, ox.grad)
    print("cfg2 grad_x rel-L2 vs fp32 oracle", f"{r:.3e}")
    assert r < GRAD_TOL, r


# ---------------------------------------------------------------------------------------------------------------- kernel level
def _dgrad_ref(dz, W):
    """fp64 autograd of conv3d: dz [N,D,H,W,Cout] 16-bit, W fp32 (Cout,Cin,3,3,3) rounded like the kernel's operand"""
    from pytorch3dunet_b200 import engine as E  # noqa: F401
    n, d, h, w, cout = dz.shape
    cin = W.shape[1]
    x = torch.zeros((n, cin, d, h, w), dtype=torch.float64, device=dz.device, requires_grad=True)
    y = F.conv3d(x, W.to(dz.dtype).double(), padding=1)
    y.backward(dz.double().permute(0, 4, 1, 2, 3))
    return x.grad


@pytest.mark.parametrize("shape", [(2, 19, 23, 17), (1, 33, 18, 10)])
@pytest.mark.parametrize("cout", [8, 16, 32])
@pytest.mark.parametrize("cin", [1, 2, 3, 4, 5])
def test_input_dgrad_conv3_kernel(cin, cout, shape):
    from pytorch3dunet_b200._lib import lib
    L = lib()
    n, d, h, w = shape
    g = torch.Generator(device="cuda").manual_seed(cin * 100 + cout)
    dz = torch.randn((n, d, h, w, cout), device="cuda", generator=g).bfloat16()
    W = torch.randn((cout, cin, 3, 3, 3), device="cuda", generator=g) * 0.2
    x = torch.randn((n, cin, d, h, w), device="cuda", generator=g)
    ref = _dgrad_ref(dz, W)
    vox = d * h * w
    P = L.query("b200_input_dgrad_partials_count", n, d, h, w, cin, cout)
    runs = []
    for _ in range(2):
        dx = torch.full((n, cin, d, h, w), float("nan"), device="cuda")
        parts = torch.full((n, P, cin, 2), float("nan"), device="cuda")
        L.call("b200_input_dgrad_conv3", p(dz), p(W), n, d, h, w, cin, cout, 0.5, p(x), p(dx), p(parts), stream())
        runs.append((dx, parts))
    torch.cuda.synchronize()
    dx, parts = runs[0]
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1]), "not bit-reproducible"
    assert rel_l2(dx, 0.5 * ref) < 1e-5, rel_l2(dx, 0.5 * ref)
    # GroupNorm-backward sums from the partials, then the in-place apply pass with the coefficients
    sums = parts.double().sum(dim=1)
    exp = torch.stack([dx.double().sum(dim=(2, 3, 4)), (dx.double() * x.double()).sum(dim=(2, 3, 4))], dim=-1)
    assert (sums - exp).abs().max().item() < 1e-4 * exp.abs().max().item() + 1e-6
    coef = torch.randn((n, cin, 3), device="cuda", generator=g)
    out = dx.clone()
    L.call("b200_gn_bwd_apply_ncdhw_f32", p(out), p(x), p(coef), n, cin, vox, 0.25, p(out), stream())
    torch.cuda.synchronize()
    c = coef.view(n, cin, 3, 1, 1, 1)
    exp_out = 0.25 * (c[:, :, 0] * dx + c[:, :, 1] * x + c[:, :, 2])
    assert rel_l2(out, exp_out) < 1e-6
    # without partials (no GroupNorm in front of the layer)
    dx2 = torch.empty_like(dx)
    L.call("b200_input_dgrad_conv3", p(dz), p(W), n, d, h, w, cin, cout, 0.5, None, p(dx2), None, stream())
    torch.cuda.synchronize()
    assert torch.equal(dx2, dx)


@pytest.mark.parametrize("cin,cout", [(1, 16), (2, 32), (3, 64), (1, 8)])
def test_pointwise_dgrad_f32_kernel(cin, cout):
    from pytorch3dunet_b200._lib import lib
    n, d, h, w = 2, 7, 9, 11
    g = torch.Generator(device="cuda").manual_seed(cout)
    dy = torch.randn((n, d, h, w, cout), device="cuda", generator=g).bfloat16()
    W = torch.randn((cout, cin), device="cuda", generator=g)
    dx = torch.empty((n, cin, d, h, w), device="cuda")
    lib().call("b200_pointwise_dgrad_f32", p(dy), p(W), n, d * h * w, cin, cout, 0.5, p(dx), stream())
    torch.cuda.synchronize()
    ref = 0.5 * torch.einsum("ndhwo,oc->ncdhw", dy.double(), W.double())
    assert rel_l2(dx, ref) < 1e-6


# ---------------------------------------------------------------------------------------------------------------- launch lists
def _small_step(name, impl, monkeypatch, x_grad=False):
    import pytorch3dunet_b200 as P
    from pytorch3dunet_b200 import engine as E
    monkeypatch.setenv("B200UNET_CONV_IMPL", impl)
    torch.manual_seed(0)
    m = P.get_model(dict(name=name, in_channels=1, out_channels=1, f_maps=16, num_levels=3)).cuda()
    x = torch.rand(1, 1, 32, 32, 32, device="cuda")
    t = (torch.rand(1, 1, 32, 32, 32, device="cuda") > 0.5).float()
    if x_grad:
        x.requires_grad_(True)
    monkeypatch.setattr(E, "TIMING", [])
    _, logits = m(x, return_logits=True)
    P.losses.bce_dice_loss(logits, t).backward()
    torch.cuda.synchronize()
    tags = [r[0] for r in E.TIMING]
    monkeypatch.setattr(E, "TIMING", None)
    return P.last_launch_counts(), tags


@pytest.mark.parametrize("impl", ["auto", "direct"])
@pytest.mark.parametrize("name", ["UNet3D", "ResidualUNet3D"])
def test_default_launch_list_unchanged(name, impl, monkeypatch):
    """without x.requires_grad no input-gradient kernel runs and the launch counts are the parent commit's"""
    counts, tags = _small_step(name, impl, monkeypatch)
    assert "dgrad_input" not in tags
    assert tuple(counts) == tuple(PARENT_COUNTS[f"{name}/{impl}"]), counts
    counts_x, tags_x = _small_step(name, impl, monkeypatch, x_grad=True)
    print(name, impl, "launches without / with input gradient", counts, counts_x)
    if name == "UNet3D":
        assert tags_x.count("dgrad_input") == 1
