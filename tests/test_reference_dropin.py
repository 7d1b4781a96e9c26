"""Drop-in claim: the reference's graph code (utils/models/q_resnet.py: Q_ResNet50 / Q_ResUnitBn forward with nn.ReLU,
nn.MaxPool2d, `x + identity`, x.view; utils/models/q_mobilenetv2.py) runs on this package's quant modules and reproduces the
reference's numbers, both un-frozen (calibration, equal ranges) and frozen (integer path through IntActivation payloads; C-ABI
launchers replaced by the numpy ABI model on CPU).

The reference's side is stored under tests/golden (tests/golden/make_golden.py, run on the unmodified reference): the order in
which its graph code calls the quant modules, its calibrated ranges, its logits and its un-frozen MobileNetV2 output.  Every graph
checked here has to match all of them: this package's own graph, which restates the reference's, always; and, where a reference
checkout is present (oracle/ref_harness.py), the reference's unmodified graph code with this package's modules swapped in."""
import json

import numpy as np
import pytest
import torch

import hawq_b200 as hb
from hawq_b200.build import build_library
from hawq_b200.synthetic import synthetic_batch, synthetic_float_mobilenetv2, synthetic_float_resnet
from oracle import ref_harness as rh
from tests import abi_model
from tests.util import QUANT_MODULES, load_golden, load_net_golden, quant_call_order

DROPIN = load_golden("ref_dropin.npz")
OURS = tuple(getattr(hb, n) for n in QUANT_MODULES)


def _graphs(monkeypatch, arch, scheme, float_model):
    """(label, stamped quantized graph) for this package's graph and, if the reference is present, the reference's graph code
    built on this package's modules."""
    ctor = {"resnet18": "q_resnet18", "resnet50": "q_resnet50", "mobilenetv2_w1": "q_mobilenetv2_w1"}[arch]
    q = getattr(hb, ctor)(float_model())
    assert hb.stamp_bit_config(q, hb.get_bit_config(arch, scheme)) == len(hb.get_bit_config(arch, scheme))
    graphs = [("hawq_b200", q)]
    if rh.available():
        ns = rh.load()
        ref = ns.q_mobilenetv2 if arch == "mobilenetv2_w1" else ns.q_resnet
        # the reference graph file did `from ..quant_modules import *`: rebind those names to this package's classes
        for name in QUANT_MODULES:
            monkeypatch.setattr(ref, name, getattr(hb, name))
        q = getattr(ref, ctor)(float_model())
        assert type(q).__module__.startswith("utils.models")
        rh.stamp_like_quant_train(q, ns.bit_config_dict["bit_config_%s_%s" % (arch, scheme)])
        graphs.append(("reference graph code", q))
    for _, q in graphs:
        q.eval()
    return graphs


def _assert_calibrated_like_the_reference(label, q, x, arch, scheme, meta):
    """Un-frozen forward of x: the quant modules are called in the reference's order and end up with the reference's ranges."""
    assert quant_call_order(q, x, OURS) == json.loads(str(DROPIN["calls_%s_%s" % (arch, scheme)])), label
    for name, m in q.named_modules():
        if isinstance(m, hb.QuantAct):
            assert float(m.x_min) == meta["acts"][name]["x_min"] and float(m.x_max) == meta["acts"][name]["x_max"], (label, name)


@pytest.mark.parametrize("arch,scheme", [("resnet18", "uniform4"), ("resnet50", "bops_0.5")])
def test_reference_graph_code_on_our_modules(monkeypatch, arch, scheme):
    build_library()
    logits_g, meta = load_net_golden(arch, scheme)
    graphs = _graphs(monkeypatch, arch, scheme, lambda: synthetic_float_resnet(arch, 0))
    abi_model.install_cpu_backend(monkeypatch)
    for label, q in graphs:
        assert isinstance(q.quant_input, hb.QuantAct)
        _assert_calibrated_like_the_reference(label, q, synthetic_batch(*meta["calib"]), arch, scheme, meta)
        hb.freeze_model(q)                                                    # reference-style traversal, our implementation
        with torch.no_grad():
            out = q(synthetic_batch(*meta["input"]))
        assert np.array_equal(out.numpy(), logits_g), label


def test_reference_mobilenetv2_graph_code_on_our_modules_unfrozen(monkeypatch):
    """MobileNetV2 (Q_LinearBottleneck / Q_MobileNetV2: nn.ReLU6, depthwise QuantBnConv2d, `x + identity` without ReLU,
    QuantConv2d classifier) on this package's modules: the calibration forward gives the reference's ranges and a second un-frozen
    forward the same fp32 outputs as the reference's own modules.  (The frozen integer path of this family is not built:
    DESIGN.md row f3.)"""
    arch, scheme = "mobilenetv2_w1", "uniform8"
    _, meta = load_net_golden(arch, scheme)
    want = torch.from_numpy(DROPIN["unfrozen_%s_%s" % (arch, scheme)])
    x, x2 = synthetic_batch(*meta["calib"]), synthetic_batch(*meta["input"])
    if rh.available():                      # the stored output is what the reference's own modules compute
        ref = rh.build_reference_qmobilenetv2(scheme, synthetic_float_mobilenetv2(0), x, freeze=False)
        with torch.no_grad():
            assert torch.equal(ref(x2), want)
    for label, q in _graphs(monkeypatch, arch, scheme, lambda: synthetic_float_mobilenetv2(0)):
        assert isinstance(q.features.stage2.unit1.conv2, hb.QuantBnConv2d)
        _assert_calibrated_like_the_reference(label, q, x, arch, scheme, meta)
        with torch.no_grad():
            got = q(x2)                     # second un-frozen forward (ranges keep moving, like the reference's)
        assert torch.equal(got, want), label
