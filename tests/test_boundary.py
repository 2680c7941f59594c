"""CPU: the drop-in boundary (SURVEY.md section 8(b)) -- install() rebinding the reference package's model factory, checkpoint
compatibility with the reference's state_dict (golden vectors from oracle/make_golden.py), constructor-time validation,
nn.DataParallel replicas, flat parameter storage and gradient buckets."""
import os
import sys
import types

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REF_MODEL = "pytorch3dunet.unet3d.model"


class _RefModel(torch.nn.Module):
    """stand-in for a reference model class: records the keyword arguments it was constructed with"""

    def __init__(self, **kwargs):
        super().__init__()
        self.kwargs = kwargs


@pytest.fixture
def reference_pkg():
    """A stand-in for the reference's `pytorch3dunet.unet3d.model` with the surface install() works on: the model classes,
    get_model (resolves the class by name in this module at call time and passes it the whole config, model.py:361-363) and
    is_model_2d (model.py:366-369)."""
    ref_model = types.ModuleType(REF_MODEL)
    for name in ("UNet3D", "ResidualUNet3D", "ResidualUNetSE3D", "UNet2D", "ResidualUNet2D"):
        setattr(ref_model, name, type(name, (_RefModel,), {"__module__": REF_MODEL}))
    ref_model.get_model = lambda config: getattr(ref_model, config["name"])(**config)
    ref_model.is_model_2d = lambda model: isinstance(model, ref_model.UNet2D)
    had = sys.modules.get(REF_MODEL)
    sys.modules[REF_MODEL] = ref_model
    yield ref_model
    import pytorch3dunet_b200 as P
    P.uninstall()
    if had is None:
        sys.modules.pop(REF_MODEL, None)
    else:
        sys.modules[REF_MODEL] = had


def test_install_rebinds_get_model_and_keeps_2d_and_unsupported_on_the_reference(reference_pkg):
    import pytorch3dunet_b200 as P
    ref_model = reference_pkg
    ref_unet3d, ref_get_model = ref_model.UNet3D, ref_model.get_model
    # a caller that imported the factory BY NAME before install(), as trainer.py:17 / predict.py:15 do
    caller = types.ModuleType("pytorch3dunet.predict")
    caller.get_model = ref_get_model
    had = sys.modules.get("pytorch3dunet.predict")
    sys.modules["pytorch3dunet.predict"] = caller
    try:
        assert P.install() is True
        assert ref_model.get_model is not ref_get_model and caller.get_model is ref_model.get_model
        assert ref_model.UNet3D is P.UNet3D and ref_model.ResidualUNet3D is P.ResidualUNet3D and ref_model.ResidualUNetSE3D is P.ResidualUNetSE3D
        m = ref_model.get_model(dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2))
        assert isinstance(m, P.UNet3D) and not ref_model.is_model_2d(m)
        # 2-D stays on the reference
        m2 = ref_model.get_model(dict(name="UNet2D", in_channels=1, out_channels=1, f_maps=8, num_levels=2))
        assert type(m2).__module__.startswith("pytorch3dunet.") and ref_model.is_model_2d(m2)
        # valid 3-D configurations the engine does not build are constructed from the reference's own class (graph-level fallback)
        for extra in (dict(layer_order="bcr"), dict(layer_order="gcrd"), dict(upsample="area"), dict(f_maps=[12, 24], num_groups=2)):
            cfg = dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2)
            cfg.update(extra)
            mf = ref_model.get_model(cfg)
            assert type(mf) is ref_unet3d, extra
            assert mf.kwargs == cfg, extra   # with the whole config, as the reference's get_model passes it
        assert P.install() is True  # idempotent
        assert P.uninstall() is True
        assert ref_model.get_model is ref_get_model and ref_model.UNet3D is ref_unet3d and caller.get_model is ref_get_model
    finally:
        if had is None:
            sys.modules.pop("pytorch3dunet.predict", None)
        else:
            sys.modules["pytorch3dunet.predict"] = had


def test_engine_state_dict_loads_into_the_reference_and_back():
    """checkpoint compatibility both ways (utils.py:59-60 load_state_dict), against the state_dict the reference's get_model
    builds for this config under torch.manual_seed(3)"""
    import pytorch3dunet_b200 as P
    cfg = dict(name="ResidualUNetSE3D", in_channels=1, out_channels=2, f_maps=16, num_levels=2, final_sigmoid=False)
    z = np.load(os.path.join(GOLDEN, "state_dict_resunetse3d_f16_l2_c2_seed3.npz"))
    ref = {k[3:]: torch.from_numpy(z[k]) for k in z.files}
    torch.manual_seed(3)
    eng = P.get_model(cfg)
    # engine -> reference: the same names in the same order with the same shapes is what the reference's strict load checks
    assert list(ref.keys()) == list(eng.state_dict().keys())
    for k, v in ref.items():
        assert torch.equal(v, eng.state_dict()[k]), k     # same default init under the same seed
    # reference -> engine
    torch.manual_seed(4)
    other = P.get_model(cfg)
    other.load_state_dict(ref)
    for k, v in other.state_dict().items():
        assert torch.equal(v, ref[k]), k


def test_unsupported_configurations_fail_at_construction_not_on_the_first_batch():
    import pytorch3dunet_b200 as P
    base = dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2)
    for extra in (dict(layer_order="bcr"), dict(layer_order="gcrd"), dict(layer_order="gcgr"), dict(upsample="area"), dict(upsample=None),
                  dict(upsample="bilinear"), dict(f_maps=[12, 24], num_groups=2), dict(conv_padding=0)):
        with pytest.raises(P.UnsupportedConfig):
            P.get_model({**base, **extra})
    with pytest.raises(ValueError):
        P.get_model({**base, "layer_order": "gcx"})          # not a layer type of the reference either (buildingblocks.py:90-93)
    with pytest.raises(AssertionError):
        P.get_model({**base, "layer_order": "rcg"})          # buildingblocks.py:42
    # configurations that ARE built, including the residual block's own default order 'cge' and the explicit upsampling modes
    P.get_model({**base, "upsample": "trilinear"})
    P.get_model({**base, "upsample": "deconv"})
    P.get_model({**base, "name": "ResidualUNet3D", "layer_order": "cge"})
    P.get_model({**base, "name": "ResidualUNet3D", "upsample": "deconv"})
    P.model.ResNetBlock(16, 32)                                # default order='cge'
    P.Encoder(16, 32, pool_type="avg")


def _replicate_like_data_parallel(model):
    """what torch.nn.parallel.replicate does to a module tree, minus the device broadcast (torch/nn/parallel/replicate.py): replicas
    lose their `_parameters`; the copies are plain attributes listed in `_former_parameters`"""
    from collections import OrderedDict
    modules = list(model.modules())
    idx = {m: i for i, m in enumerate(modules)}
    reps = []
    for m in modules:
        r = m._replicate_for_data_parallel()
        r._former_parameters = OrderedDict()
        reps.append(r)
    for i, m in enumerate(modules):
        for key, child in m._modules.items():
            setattr(reps[i], key, None if child is None else reps[idx[child]]) if child is not None else reps[i]._modules.__setitem__(key, None)
        for key, p in m._parameters.items():
            if p is None:
                reps[i]._parameters[key] = None
            else:
                c = p.detach().clone().requires_grad_(True) * 1.0   # non-leaf, like a broadcast copy
                setattr(reps[i], key, c)
                reps[i]._former_parameters[key] = c
    return reps[0]


def test_parameters_are_found_on_data_parallel_replicas():
    """trainer.py:203-204 / predict.py:63-65 wrap the model in nn.DataParallel whenever several GPUs are visible; a replica's
    named_parameters() is empty"""
    import pytorch3dunet_b200 as P
    from pytorch3dunet_b200.model import _named_params
    model = P.get_model(dict(name="ResidualUNetSE3D", in_channels=1, out_channels=1, f_maps=16, num_levels=2))
    rep = _replicate_like_data_parallel(model)
    assert list(rep.named_parameters()) == []
    np_rep, is_rep = _named_params(rep)
    np_model, is_rep0 = _named_params(model)
    assert is_rep and not is_rep0
    assert [k for k, _ in np_rep] == [k for k, _ in np_model] == [k for k, _ in model.named_parameters()]
    for (k, a), (_, b) in zip(np_rep, np_model):
        assert a.shape == b.shape and not a.is_leaf


def test_flat_parameters_views_buckets_and_checkpoints():
    import pytorch3dunet_b200 as P
    from pytorch3dunet_b200.optim import BucketedAllReduce, FlatParameters
    cfg = dict(name="ResidualUNet3D", in_channels=1, out_channels=1, f_maps=16, num_levels=3)
    torch.manual_seed(0)
    model = P.get_model(cfg)
    before = {k: v.clone() for k, v in model.state_dict().items()}
    flat = FlatParameters(model)
    assert flat.numel >= sum(p.numel() for p in model.parameters())
    for k, v in model.state_dict().items():
        assert torch.equal(v, before[k])
    for k, p in model.named_parameters():
        o, n = flat.range_of[k]
        assert p.data_ptr() == flat.data[o:].data_ptr() and p.grad.data_ptr() == flat.grad[o:].data_ptr() and o % 4 == 0
    # a checkpoint load writes through the views
    sd = {k: torch.full_like(v, 0.5) for k, v in before.items()}
    model.load_state_dict(sd)
    o, n = flat.range_of["final_conv.weight"]
    assert torch.all(flat.data[o:o + n] == 0.5)
    # zero_grad(set_to_none=True) drops .grad; the views come back
    for p in model.parameters():
        p.grad = None
    flat.restore_grad_views()
    assert all(p.grad is not None for p in model.parameters())
    # buckets: a partition of all parameters, contiguous ranges, in reverse parameter order
    red = BucketedAllReduce(flat, world=1, n_buckets=4, min_bucket_bytes=1024)
    names = [k for b in red.buckets for k in b]
    assert names == list(reversed(flat.names)) and len(red.buckets) == 4
    covered = sorted(red.ranges)
    assert covered[0][0] == 0 and covered[-1][1] == flat.numel
    for (a0, a1), (b0, b1) in zip(covered, covered[1:]):
        assert a1 == b0
