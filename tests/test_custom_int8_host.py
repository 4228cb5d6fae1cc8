"""INT8 surface of the model.py network on the host: float-layer patterns, QAT checkpoints, and the integer
reference oracle/custom_quant_graph.py against a dequantised fake-quant forward."""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F


def test_quant_spec_str_patterns_and_int_layers():
    from unina_yolo_dla_b200 import quant as Q

    names = ["backbone.stem.conv", "backbone.stage1_conv.conv", "head_p2.cls_branch.0.conv", "head_p2.reg_branch.2",
             "head_p3.cls_branch.2", "model.0.conv", "model.1.conv", "model.2.cv1.conv", "model.12.cv1.conv"]
    q = Q.QuantSpec({n: (1.0, 1.0) for n in names}, ("stem", "head_p2"))
    assert [q.covers(n) for n in names] == [False, True, False, False, True, True, True, True, True]
    q = Q.QuantSpec({n: (1.0, 1.0) for n in names})          # default: model.{0,1,2}, as before
    assert [q.covers(n) for n in names] == [True, True, True, True, True, False, False, False, True]
    q = Q.QuantSpec({n: (1.0, 1.0) for n in names}, (1, "head_p3"))   # both kinds in one list
    assert [q.covers(n) for n in names] == [True, True, True, True, False, True, False, True, True]
    assert not Q.QuantSpec({}, ()).covers("backbone.stage1_conv.conv")   # no amax entry: float


def test_custom_qat_checkpoint_round_trip_on_the_host():
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200 import quant as Q

    m = uyd.UninaCustomB200(base_channels=8).init_synthetic(seed=1)
    convs = [n for n, mod in m.named_modules() if isinstance(mod, nn.Conv2d)]
    assert all(getattr(m.get_submodule(n), "_uyd_name") == n for n in convs)
    amax = {n: (1.0 + i, 0.5 + i) for i, n in enumerate(convs) if n != "backbone.stem.conv"}
    sd = dict(m.state_dict())
    assert not any(k.endswith("_amax") for k in sd)
    ckpt = dict(sd, **uyd.UninaCustomB200(base_channels=8).set_quantization(amax).quant_state_dict())
    assert len(ckpt) == len(sd) + 2 * len(amax)

    fresh = uyd.UninaCustomB200(base_channels=8)
    fresh.load_state_dict(ckpt)
    assert fresh.quant is not None and fresh.quant.amax == amax
    assert fresh.quant.float_layers == uyd.UninaCustomB200.FLOAT_LAYERS
    assert fresh.quant_state_dict().keys() == {k for k in ckpt if k.endswith("_amax")}
    assert all(torch.equal(fresh.state_dict()[k], v) for k, v in sd.items())
    covered = [n for n in convs if fresh.quant.covers(n)]
    assert len(covered) == len(convs) - 1 - 6                  # minus the stem and head_p2's six convs

    plain = uyd.UninaCustomB200(base_channels=8)
    plain.load_state_dict(sd)
    assert plain.quant is None and plain.quant_state_dict() == {}
    plain.set_quantization(amax).set_quantization(None)
    assert plain.quant is None
    plain2, amax2 = Q.split_state_dict(ckpt)
    assert plain2.keys() == sd.keys() and amax2 == amax


def _fake_quant(x, amax):
    from oracle import quant as oq

    s = oq.scale_of(amax)
    return torch.from_numpy(np.clip(np.rint(x.numpy().astype(np.float32) * s), -127, 127).astype(np.float32) / s)


def test_custom_quant_graph_matches_a_fake_quant_forward_within_one_step():
    """The integer reference is the fake-quant network: each conv of a dequantised fp32 forward (inputs and weights
    quantised and dequantised, bf16 activations) agrees with it to within one quantisation step of its input."""
    import unina_yolo_dla_b200 as uyd
    from oracle import custom_graph as cg
    from oracle.custom_quant_graph import CustomInt8Graph
    from oracle.quant_graph import bf16

    torch.manual_seed(0)
    src = uyd.UninaCustomB200(num_classes=4, base_channels=8).init_synthetic(seed=3)
    net = cg.CustomNet(4, 8)
    net.load_state_dict(src.state_dict())
    net.eval()
    x = torch.rand(2, 3, 64, 96, generator=torch.Generator().manual_seed(5))
    convs = {n: mod for n, mod in net.named_modules() if isinstance(mod, nn.Conv2d)}

    # max calibration on the float forward
    amax = {}
    hooks = [mod.register_forward_pre_hook(lambda mod, a, n=n: amax.__setitem__(n, (float(a[0].abs().max()),
                                                                                  float(mod.weight.abs().max()))))
             for n, mod in convs.items() if n != "backbone.stem.conv"]
    with torch.no_grad():
        stem = bf16(net.backbone.stem(x))
        net(x)
    for h in hooks:
        h.remove()
    assert len(amax) == len(convs) - 1

    with torch.no_grad():
        want = CustomInt8Graph(net, amax).forward_from(stem)

    # fake-quant forward: every conv after the stem sees dequantised inputs and weights; activations are bf16
    fq = cg.CustomNet(4, 8)
    fq.load_state_dict(net.state_dict())
    fq.eval()
    step = {}
    for n, mod in fq.named_modules():
        if isinstance(mod, nn.Conv2d) and n in amax:
            ax, aw = amax[n]
            mod.weight.data = _fake_quant(mod.weight.data, aw)
            mod.register_forward_pre_hook(lambda mod, a, ax=ax: (_fake_quant(a[0], ax),))
            # one input quantisation step, through |w|: the most an output can move when each input moves by one step
            step[n] = float(ax / 127 * mod.weight.detach().abs().sum((1, 2, 3)).max())
    for mod in fq.modules():
        if isinstance(mod, cg.CBR):
            mod.forward = lambda t, mod=mod: bf16(F.relu(mod.bn(mod.conv(t))))
    with torch.no_grad():
        fq.backbone.stem.forward = lambda t: stem
        got = fq(x)
    for lvl, (a, b) in enumerate(zip(want, got)):
        for br, (wa, ga) in enumerate(zip(a, b)):
            name = f"head_p{lvl + 2}.{('cls', 'reg')[br]}_branch.2"
            assert wa.shape == ga.shape and wa.dtype == torch.float32
            assert float((wa - ga).abs().max()) <= step[name], (name, float((wa - ga).abs().max()), step[name])
