"""Shared helpers for the parity tests (test infrastructure; may import oracle/)."""
import hashlib
import json
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name), allow_pickle=False)
    return {k: z[k] for k in z.files}


def load_net_golden(arch, scheme):
    g = load_golden("net_%s_%s.npz" % (arch, scheme))
    meta = json.loads(str(g["meta"]))
    return g["logits"], meta


def sha_i32(a):
    return hashlib.sha256(np.ascontiguousarray(np.asarray(a).astype(np.int32)).tobytes()).hexdigest()


QUANT_MODULES = ("QuantAct", "QuantBnConv2d", "QuantConv2d", "QuantLinear", "QuantAveragePool2d")


def quant_call_order(q, x, kinds):
    """Names of the modules of `q` whose type is in `kinds`, in the order q's graph code calls them during one forward of x."""
    order = []
    hooks = [m.register_forward_pre_hook(lambda mod, inp, name=name: order.append(name))
             for name, m in q.named_modules() if type(m) in kinds]
    try:
        with torch.no_grad():
            q(x)
    finally:
        for h in hooks:
            h.remove()
    return order


def golden_act_ranges(meta):
    return {k: (v["x_min"], v["x_max"]) for k, v in meta["acts"].items()}


def build_fakequant(arch, scheme, meta=None):
    """Oracle fake-quant net on the seed-0 synthetic model, act ranges from the golden file (like loading a checkpoint)."""
    from oracle import fakequant as fq
    from hawq_b200.synthetic import synthetic_float_resnet, synthetic_batch
    from hawq_b200.bit_config import get_bit_config
    net = synthetic_float_resnet(arch, 0)
    m = fq.FakeQuantResNet(arch, net, get_bit_config(arch, scheme))
    if meta is not None:
        m.load_act_ranges(golden_act_ranges(meta))
        m.freeze()
    return m
