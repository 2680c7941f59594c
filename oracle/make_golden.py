"""Generate tests/golden/*.npz by running the REFERENCE's own classes (build container only).

TEST INFRASTRUCTURE.  Needs /root/reference (read-only checkout of wolny/pytorch-3dunet @ a33e2c7);
that path does not exist on the GPU box, so the fixtures are committed and this script is the
record of how they were made:

    python oracle/make_golden.py

For every case: seeded weights (the reference modules' own default init under torch.manual_seed),
seeded input/target, the reference forward (probabilities + logits), the loss, and the gradient of
the loss w.r.t. every parameter and the input, all fp32 CPU.
"""
import os
import sys
import types

import numpy as np
import torch

REF = "/root/reference"
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def import_reference():
    # unet3d/utils.py:10 imports skimage.color.label2rgb (TensorBoard formatter only); stub it.
    sk, col = types.ModuleType("skimage"), types.ModuleType("skimage.color")
    col.label2rgb = lambda *a, **k: None
    sk.color = col
    sys.modules.setdefault("skimage", sk)
    sys.modules.setdefault("skimage.color", col)
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from pytorch3dunet.unet3d import buildingblocks, losses, model  # noqa
    return model, buildingblocks, losses


def run_model_case(name, cfg, shape, loss_name, seed, model_mod, losses_mod, perturb_affine=True):
    torch.manual_seed(seed)
    m = model_mod.get_model(dict(cfg))
    if perturb_affine:
        # default GN init is weight=1, bias=0; perturb so the affine path is actually exercised
        g = torch.Generator().manual_seed(seed + 1)
        with torch.no_grad():
            for k, p in m.named_parameters():
                if "groupnorm" in k:
                    p.add_(0.2 * torch.randn(p.shape, generator=g))
    m.train()
    x = torch.rand(shape)
    x.requires_grad_(True)
    out, logits = m(x, return_logits=True)
    c_out = cfg["out_channels"]
    target = (torch.rand(shape[0], c_out, *shape[2:]) > 0.5).float()
    loss = getattr(losses_mod, loss_name)()(logits, target)
    loss.backward()
    rec = {"x": x.detach().numpy(), "target": target.numpy(), "out": out.detach().numpy(),
           "logits": logits.detach().numpy(), "loss": np.float32(loss.item()),
           "grad_x": x.grad.numpy()}
    for k, p in m.state_dict().items():
        rec["sd/" + k] = p.detach().numpy()
    for k, p in m.named_parameters():
        rec["grad/" + k] = p.grad.detach().numpy()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **rec)
    print(f"{name}: loss={loss.item():.6f} params={sum(p.numel() for p in m.parameters())}")


def run_block_case(name, module, x_shape, seed, extra_inputs=None):
    """A single building block: forward + backward of sum(y * r) for a fixed random r."""
    g = torch.Generator().manual_seed(seed + 7)
    with torch.no_grad():
        for k, p in module.named_parameters():
            if "groupnorm" in k:
                p.add_(0.2 * torch.randn(p.shape, generator=g))
    x = torch.rand(x_shape, generator=g) * 2 - 0.5
    x.requires_grad_(True)
    ins = [x]
    if extra_inputs is not None:
        e = torch.rand(extra_inputs, generator=g)
        e.requires_grad_(True)
        ins = [e, x]  # Decoder.forward(encoder_features, x)
    y = module(*ins)
    r = torch.randn(y.shape, generator=g)
    (y * r).sum().backward()
    rec = {"x": x.detach().numpy(), "y": y.detach().numpy(), "r": r.numpy(), "grad_x": x.grad.numpy()}
    if extra_inputs is not None:
        rec["enc"] = ins[0].detach().numpy()
        rec["grad_enc"] = ins[0].grad.numpy()
    for k, p in module.state_dict().items():
        rec["sd/" + k] = p.detach().numpy()
    for k, p in module.named_parameters():
        rec["grad/" + k] = p.grad.detach().numpy()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **rec)
    print(f"{name}: y {tuple(y.shape)}")


def run_state_dict_case(name, cfg, seed, model_mod):
    """The default-initialised state_dict of a model built by the reference's get_model under torch.manual_seed(seed): the
    checkpoint a reference user would hand to the engine (names, order, shapes, values)."""
    torch.manual_seed(seed)
    m = model_mod.get_model(dict(cfg))
    rec = {"sd/" + k: p.detach().numpy() for k, p in m.state_dict().items()}
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **rec)
    print(f"{name}: {len(rec)} tensors")


ONLY = None  # set by `--only name1,name2`: regenerate just these fixtures


def _wanted(name):
    return ONLY is None or name in ONLY


def main():
    global ONLY, run_model_case, run_block_case, run_state_dict_case
    if "--only" in sys.argv:
        ONLY = set(sys.argv[sys.argv.index("--only") + 1].split(","))
        _rm, _rb, _rs = run_model_case, run_block_case, run_state_dict_case
        run_model_case = lambda name, *a, **k: _rm(name, *a, **k) if _wanted(name) else None  # noqa: E731
        run_block_case = lambda name, *a, **k: _rb(name, *a, **k) if _wanted(name) else None  # noqa: E731
        run_state_dict_case = lambda name, *a, **k: _rs(name, *a, **k) if _wanted(name) else None  # noqa: E731
    os.makedirs(OUT, exist_ok=True)
    model_mod, bb, losses_mod = import_reference()
    torch.set_num_threads(1)  # reproducible reductions

    # ---- whole models (small f_maps so fixtures stay small) ------------------------------
    run_model_case("unet3d_f16_l3_s16", dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=3),
                   (1, 1, 16, 16, 16), "BCEDiceLoss", 0, model_mod, losses_mod)
    run_model_case("unet3d_f16_l3_dice_b2", dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=3),
                   (2, 1, 16, 16, 16), "DiceLoss", 1, model_mod, losses_mod)
    # odd, non power-of-two sizes as in the reference's tests/test_models.py:20 (33,65,65), scaled down
    run_model_case("unet3d_f16_l3_odd", dict(name="UNet3D", in_channels=2, out_channels=3, f_maps=16, num_levels=3,
                                              final_sigmoid=False),
                   (1, 2, 9, 17, 13), "BCEDiceLoss", 2, model_mod, losses_mod)
    run_model_case("unet3d_f16_l2_cgr", dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2,
                                             layer_order="cgr"),
                   (1, 1, 8, 8, 8), "BCEDiceLoss", 3, model_mod, losses_mod)
    run_model_case("resunet3d_f16_l3_s16", dict(name="ResidualUNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=3),
                   (1, 1, 16, 16, 16), "BCEDiceLoss", 4, model_mod, losses_mod)
    run_model_case("resunetse3d_f16_l3_s16", dict(name="ResidualUNetSE3D", in_channels=1, out_channels=1, f_maps=16, num_levels=3),
                   (1, 1, 16, 16, 16), "BCEDiceLoss", 5, model_mod, losses_mod)

    # more layer orders / activations (oracle pinning only; CPU tests): conv bias + LeakyReLU(0.01), conv-ReLU-GroupNorm,
    # ResNetBlock's own LeakyReLU(0.1) and ELU (buildingblocks.py:271-275), softmax head with several classes
    run_model_case("unet3d_f16_l2_cl", dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2, layer_order="cl"),
                   (1, 1, 8, 8, 8), "BCEDiceLoss", 6, model_mod, losses_mod)
    run_model_case("unet3d_f16_l2_crg", dict(name="UNet3D", in_channels=1, out_channels=2, f_maps=16, num_levels=2, layer_order="crg",
                                             final_sigmoid=False),
                   (2, 1, 8, 8, 8), "BCEDiceLoss", 7, model_mod, losses_mod)
    run_model_case("resunet3d_f16_l2_gcl", dict(name="ResidualUNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2,
                                                layer_order="gcl"),
                   (1, 1, 8, 8, 8), "BCEDiceLoss", 8, model_mod, losses_mod)
    run_model_case("resunetse3d_f16_l2_gce", dict(name="ResidualUNetSE3D", in_channels=2, out_channels=1, f_maps=16, num_levels=2,
                                                  layer_order="gce"),
                   (1, 2, 8, 8, 8), "DiceLoss", 9, model_mod, losses_mod)

    # upsampling modes reachable through the model config (buildingblocks.py:431-468): trilinear interpolation + concat (odd sizes:
    # a non-2x scale), explicit 'deconv' with the concat join for DoubleConv and for ResNetBlock, and the residual block's own
    # default order 'cge' (GroupNorm between conv3 and the residual add)
    run_model_case("unet3d_f16_l2_trilinear", dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2,
                                                   upsample="trilinear"),
                   (1, 1, 9, 12, 10), "BCEDiceLoss", 20, model_mod, losses_mod)
    run_model_case("unet3d_f16_l2_deconv", dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2,
                                                upsample="deconv"),
                   (1, 1, 8, 8, 8), "BCEDiceLoss", 21, model_mod, losses_mod)
    run_model_case("resunet3d_f16_l2_cge", dict(name="ResidualUNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2,
                                                layer_order="cge"),
                   (1, 1, 8, 8, 8), "BCEDiceLoss", 22, model_mod, losses_mod)
    run_model_case("resunet3d_f16_l2_deconvcat", dict(name="ResidualUNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2,
                                                      upsample="deconv"),
                   (1, 1, 8, 8, 8), "BCEDiceLoss", 23, model_mod, losses_mod)

    # ---- building blocks -----------------------------------------------------------------
    torch.manual_seed(10)
    run_block_case("block_singleconv_gcr_16_32", bb.SingleConv(16, 32, order="gcr", num_groups=8), (2, 16, 8, 8, 8), 10)
    torch.manual_seed(11)
    run_block_case("block_singleconv_cr_16_16", bb.SingleConv(16, 16, order="cr", num_groups=8), (1, 16, 6, 7, 8), 11)
    torch.manual_seed(12)
    run_block_case("block_doubleconv_enc_32_64", bb.DoubleConv(32, 64, encoder=True, order="gcr", num_groups=8), (1, 32, 8, 8, 8), 12)
    torch.manual_seed(13)
    run_block_case("block_doubleconv_dec_96_32", bb.DoubleConv(96, 32, encoder=False, order="gcr", num_groups=8), (1, 96, 8, 8, 8), 13)
    torch.manual_seed(14)
    run_block_case("block_encoder_pool_32_64", bb.Encoder(32, 64, basic_module=bb.DoubleConv), (1, 32, 8, 10, 12), 14)
    torch.manual_seed(15)
    run_block_case("block_decoder_cat_64_32", bb.Decoder(96, 32, basic_module=bb.DoubleConv), (1, 64, 4, 4, 4), 15,
                   extra_inputs=(1, 32, 8, 8, 8))
    torch.manual_seed(16)
    run_block_case("block_decoder_cat_odd", bb.Decoder(48, 16, basic_module=bb.DoubleConv), (1, 32, 2, 4, 3), 16,
                   extra_inputs=(1, 16, 5, 9, 7))
    torch.manual_seed(17)
    run_block_case("block_resnet_16_32", bb.ResNetBlock(16, 32, order="gcr", num_groups=8), (1, 16, 8, 8, 8), 17)
    torch.manual_seed(18)
    run_block_case("block_resnetse_32_32", bb.ResNetBlockSE(32, 32, order="gcr", num_groups=8), (1, 32, 8, 8, 8), 18)
    torch.manual_seed(19)
    run_block_case("block_decoder_deconv_32_16", bb.Decoder(32, 16, basic_module=bb.ResNetBlock), (1, 32, 4, 4, 4), 19,
                   extra_inputs=(1, 16, 8, 8, 8))

    # ---- checkpoints (tests/test_boundary.py: a reference checkpoint loads into the engine and back) ----------------
    run_state_dict_case("state_dict_resunetse3d_f16_l2_c2_seed3",
                        dict(name="ResidualUNetSE3D", in_channels=1, out_channels=2, f_maps=16, num_levels=2, final_sigmoid=False),
                        3, model_mod)


if __name__ == "__main__":
    main()
