"""Host-side logic that needs no GPU: module trees / state_dict contracts, init parity with the reference (golden
checksums), conv_sequence rules, fuse_conv_bn and re-parametrisation arithmetic, argument validation, and the
"no CPU fallback" rule."""
import pytest
import torch
from torch import nn

import holocron_b200 as hb
from holocron_b200.models.utils import conv_sequence, fuse_conv_bn
from oracle.models import RepVGGOracle

from conftest import load_golden


def test_conv_sequence_rules():
    # reference tests/test_models.py:21-52: ordering [conv, norm, act, drop], bias only when there is no norm layer
    mods = conv_sequence(3, 32, nn.ReLU(inplace=True), nn.BatchNorm2d, hb.nn.DropBlock2d, kernel_size=3)
    assert [type(m).__name__ for m in mods] == ["Conv2d", "BatchNorm2d", "ReLU", "DropBlock2d"]
    assert mods[0].bias is None and mods[3].inplace
    mods = conv_sequence(3, 32, None, None, kernel_size=3)
    assert len(mods) == 1 and mods[0].bias is not None
    mods = conv_sequence(3, 32, nn.ReLU(), nn.BatchNorm2d, kernel_size=3, bias=True)
    assert mods[0].bias is not None
    mods = conv_sequence(3, 32, nn.ReLU(), nn.BatchNorm2d, bn_channels=16, kernel_size=3)
    assert mods[1].num_features == 16
    with pytest.raises(NotImplementedError):
        conv_sequence(3, 32, blurpool=True, kernel_size=3, stride=2)


def test_fuse_conv_bn_matches_reference_golden():
    f = load_golden("models")["fuse"]
    conv = nn.Conv2d(6, 8, 3, padding=1, bias=False)
    bn = nn.BatchNorm2d(8).eval()
    conv.weight.data = f["conv_w"].clone()
    bn.weight.data, bn.bias.data = f["gamma"].clone(), f["beta"].clone()
    bn.running_mean, bn.running_var = f["mean"].clone(), f["var"].clone()
    k, b = fuse_conv_bn(conv, bn)
    assert torch.equal(k, f["k"]) and torch.equal(b, f["b"])
    with pytest.raises(AssertionError):
        fuse_conv_bn(conv, nn.BatchNorm2d(4))
    # reference tests/test_models.py:55-83: fused conv == bn(conv(x)) on CPU
    x = torch.rand(2, 6, 8, 8)
    with torch.no_grad():
        ref = bn(conv(x))
        out = nn.functional.conv2d(x, k, b, padding=1)
    assert torch.allclose(out, ref, atol=1e-6)


def test_repvgg_tree_init_and_reparam_arithmetic():
    c = load_golden("models")["cfg1"]
    torch.manual_seed(0)
    m = hb.models.repvgg_a0(num_classes=1000)
    assert sum(p.numel() for p in m.parameters()) == c["n_params_train"]
    assert abs(float(sum(p.detach().double().sum() for p in m.parameters())) - c["param_sum"]) < 1e-6
    torch.manual_seed(0)
    o = RepVGGOracle("repvgg_a0", num_classes=1000)
    assert list(m.state_dict().keys()) == list(o.state_dict().keys())
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), o.state_dict().values()))
    # re-parametrisation is weight-sized host arithmetic: exact against the reference's folded block
    for tag, cfg in (("s1", (16, 16, 1, True)), ("s2", (16, 32, 2, False))):
        d = load_golden("models")[f"repblock_{tag}"]
        blk = hb.models.RepBlock(*cfg)
        blk.load_state_dict(d["state_after"])
        blk.reparametrize()
        assert isinstance(blk.branches, nn.Conv2d) and blk.branches.kernel_size == (3, 3)
        assert torch.equal(blk.branches.weight, d["rep_w"]) and torch.equal(blk.branches.bias, d["rep_b"])
        with pytest.raises(AssertionError):
            blk.reparametrize()
    with pytest.raises(ValueError):
        hb.models.RepBlock(16, 32, 1, True)
    m.reparametrize()
    assert not any(isinstance(mod, nn.BatchNorm2d) for mod in m.modules())
    assert sum(p.numel() for p in m.parameters()) == c["n_params"]


def test_module_reprs_and_validation():
    assert repr(hb.nn.FocalLoss()) == "FocalLoss(gamma=2.0, reduction='mean')"
    assert repr(hb.nn.DiceLoss()) == "DiceLoss(reduction='mean', gamma=1.0, eps=1e-08)"
    assert repr(hb.nn.PolyLoss()) == "PolyLoss(eps=2.0, reduction='mean')"
    assert repr(hb.nn.HardMish()) == "HardMish()" and repr(hb.nn.NLReLU()) == "NLReLU()"
    assert repr(hb.nn.GlobalAvgPool2d(flatten=True)) == "GlobalAvgPool2d(flatten=True)"
    with pytest.raises(NotImplementedError):
        hb.nn.FocalLoss(reduction="avg")
    w = hb.nn.FocalLoss(weight=0.25).weight
    assert torch.allclose(w, torch.tensor([0.25, 0.75]))
    assert hb.nn.PolyLoss(weight=[1.0, 2.0]).weight.tolist() == [1.0, 2.0]
    assert "weight" in dict(hb.nn.DiceLoss(weight=torch.ones(3)).named_buffers())
    lin = nn.Linear(4, 2)
    for cls in (hb.optim.AdaBelief, hb.optim.LAMB, hb.optim.TAdam):
        with pytest.raises(ValueError):
            cls(lin.parameters(), lr=-1)
        with pytest.raises(ValueError):
            cls(lin.parameters(), eps=-1)
        with pytest.raises(ValueError):
            cls(lin.parameters(), betas=(0.9, 1.0))
    opt = hb.optim.AdaBelief(lin.parameters(), foreach=False, fused=None)  # Adam's switches are accepted and ignored
    assert opt.defaults["amsgrad"] is False
    assert hb.optim.LAMB(lin.parameters()).scale_clip == (0.0, 10.0)


def test_no_cpu_fallback():
    x = torch.randn(2, 8, 4, 4)
    with pytest.raises(hb.HolocronB200Error):
        hb.nn.functional.hard_mish(x)
    with pytest.raises(hb.HolocronB200Error):
        hb.nn.functional.focal_loss(torch.randn(4, 3), torch.zeros(4, dtype=torch.long))
    with pytest.raises(hb.HolocronB200Error):
        hb.ops.boxes.diou_loss(torch.rand(2, 4), torch.rand(2, 4))
    with pytest.raises(hb.HolocronB200Error):
        hb.models.RepBlock(8, 16, 1, False)(x)
    lin = nn.Linear(4, 2)
    lin(torch.randn(3, 4)).sum().backward()
    with pytest.raises(hb.HolocronB200Error):
        hb.optim.AdaBelief(lin.parameters()).step()


def test_zoo_state_dicts_match_oracle_free_checks():
    # parameter counts of the reference (SURVEY §6 / checkpoints metadata)
    assert sum(p.numel() for p in hb.models.rexnet1_0x(num_classes=1000).parameters()) == 4796186
    assert sum(p.numel() for p in hb.models.repvgg_a0(num_classes=10).parameters()) == 24741642
    assert sum(p.numel() for p in hb.models.darknet53(num_classes=10).parameters()) == 40595178
    assert sum(p.numel() for p in hb.models.cspdarknet53(num_classes=10).parameters()) == 26627434
    y = hb.models.yolov4(num_classes=80)
    assert y.head.head1[-1].out_channels == 255 and float(y.head.head3[-1].bias.abs().sum()) == 0.0
    u = hb.models.unet3p(num_classes=21)
    assert u.classifier.in_channels == 320 and len(u.decoder) == 4


def test_remaining_optimizer_constructors_validate_like_the_reference():
    """Host-side argument checks of Adan / AdEMAMix / LARS / RaLars / Lookahead (reference adan.py:58-66, ademamix.py:63-70,
    lars.py:60-79, ralars.py:38-46, wrapper.py:33-37) - no kernel is launched."""
    import pytest
    import torch

    import holocron_b200 as hb
    w = [torch.nn.Parameter(torch.randn(4, 4))]
    with pytest.raises(ValueError):
        hb.optim.LARS(w, lr=1)
    with pytest.raises(ValueError):
        hb.optim.LARS(w, lr=0.1, momentum=-0.1)
    with pytest.raises(ValueError):
        hb.optim.LARS(w, lr=0.1, nesterov=True)
    with pytest.raises(ValueError):
        hb.optim.AdEMAMix(w, betas=(0.9, 0.999, 1.0))
    with pytest.raises(ValueError):
        hb.optim.RaLars(w, betas=(1.0, 0.9))
    with pytest.raises(ValueError):
        hb.optim.Adan(w, eps=-1.0)
    with pytest.raises(ValueError):
        hb.optim.wrapper.Lookahead(torch.optim.SGD(w, lr=0.1), sync_rate=-0.1)
    assert hb.optim.LARS(w, lr=0.1).scale_clip == (0.0, 10.0) and hb.optim.RaLars(w).scale_clip == (0, 10)
    assert hb.optim.Adan(w).defaults["betas"] == (0.98, 0.92, 0.99)
    assert hb.optim.AdEMAMix(w).defaults["alpha"] == 5.0
    la = hb.optim.wrapper.Lookahead(torch.optim.SGD(w, lr=0.1), sync_period=2)
    assert la.defaults == {"sync_rate": 0.5, "sync_period": 2} and la.fast_steps == 0
    assert la.param_groups[0]["params"][0] is not w[0] and torch.equal(la.param_groups[0]["params"][0], w[0].data)
    assert "base_state_dict" in la.state_dict()
    la.add_param_group({"params": [torch.nn.Parameter(torch.randn(2))]})
    assert len(la.param_groups) == 2 and len(la.base_optimizer.param_groups) == 2
    # a fused step on CPU tensors fails loudly: there is no CPU fallback
    w[0].grad = torch.ones_like(w[0])
    with pytest.raises((RuntimeError, TypeError, ValueError)):
        hb.optim.Adan(w).step()


def test_mixup_collate_matches_reference_draw_for_draw():
    """holocron.utils.data.Mixup (reference utils/data/collate.py:16-64): same one-hot encoding, same RNG draws in the same
    order (Beta sample, permutation), same in-place mixing - seeded batches come out identical to what the unmodified
    reference's Mixup returned on them (tests/golden/make_golden.py --cross)."""
    import pytest
    import torch
    import holocron_b200 as hb
    from conftest import load_golden
    with pytest.raises(ValueError):
        hb.utils.data.Mixup(10, alpha=-0.1)
    mix = hb.utils.data.Mixup(num_classes=7, alpha=0.0)
    x, t = torch.rand(4, 3, 8, 8), torch.tensor([1, 0, 6, 3])
    xo, to = mix(x.clone(), t)
    assert torch.equal(xo, x) and to.shape == (4, 7) and to.dtype == x.dtype and torch.equal(to.argmax(1), t)
    assert hb.utils.data.Mixup(1, 0.0)(x.clone(), torch.tensor([1, 0, 1, 1]))[1].shape == (4, 1)
    for case in load_golden("cross_checks")["mixup"]:
        torch.manual_seed(100 + case["seed"])
        xm, tm = hb.utils.data.Mixup(case["num_classes"], case["alpha"])(case["x"].clone(), case["t"].clone())
        assert torch.equal(case["x_out"], xm) and torch.equal(case["t_out"], tm)
