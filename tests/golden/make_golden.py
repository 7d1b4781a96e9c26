"""Generate the committed golden vectors by running the UNMODIFIED reference (/root/reference) on CPU.

Run once in the build container:  python tests/golden/make_golden.py
Outputs (small, committed):
  kat_requant.npz      known-answer vectors for batch_frexp / fixedpoint_fn case 0 / case 1
  kat_modules.npz      QuantAct(input) / QuantBnConv2d / QuantConv2d / QuantLinear / QuantAveragePool2d on tiny shapes
  net_<arch>_<scheme>.npz   whole-network: act ranges, per-QuantAct checksums of the activation integers,
                            per-layer checksums of weight_integer / bias_integer, logits  (batch 2)
  net_mobilenetv2_w1_<scheme>.npz   the same for MobileNetV2-1.0 (python tests/golden/make_golden.py --mobilenetv2 uniform8|uniform4)
  ref_dropin.npz       the order in which the reference's graph code calls its quant modules, and an un-frozen MobileNetV2 output
                       (python tests/golden/make_golden.py --dropin)
Nothing here runs on the GPU box; tests only read the .npz files.
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_harness as rh  # noqa: E402
from hawq_b200.synthetic import synthetic_float_resnet, synthetic_batch  # noqa: E402

CALIB_BATCH, CALIB_SEED = 4, 0
PARITY_BATCH, PARITY_SEED = 2, 1
NET_CONFIGS = [("resnet18", "uniform8"), ("resnet18", "uniform4"), ("resnet18", "bops_0.5"),
               ("resnet50", "uniform8"), ("resnet50", "uniform4"), ("resnet50", "bops_0.5")]


def sha_i32(a):
    return hashlib.sha256(np.ascontiguousarray(a.astype(np.int32)).tobytes()).hexdigest()


def nhwc(t):
    a = t.numpy()
    return a.transpose(0, 2, 3, 1) if a.ndim == 4 else a


def make_kat_requant(ns):
    qu = ns.quant_utils
    out = {}
    ratios = np.array([0.25, 0.3, 0.5, 1.0, 0.0625, 1.0 / 3.0, 0.7071067811865476, 1e-3, 3.0517578125e-05,
                       0.9999999999, 0.99999999999999989, 2.5, 1.2e-5, 7.450580596923828e-09], dtype=np.float64)
    rng = np.random.RandomState(7)
    ratios = np.concatenate([ratios, np.exp(rng.uniform(np.log(1e-6), np.log(2.0), 50))])
    m, e = qu.batch_frexp(torch.from_numpy(ratios))
    out["frexp_ratio"], out["frexp_m"], out["frexp_e"] = ratios, m.numpy().astype(np.int64), e.numpy().astype(np.int64)

    # case 0: scales chosen as powers of two times small odd numbers so z = acc*a*w is exact in fp32
    cases = []
    rng = np.random.RandomState(11)
    specs = [(8, 'symmetric'), (4, 'asymmetric'), (16, 'symmetric'), (4, 'symmetric'), (8, 'asymmetric')]
    for idx, (bits, mode) in enumerate(specs):
        C = 6
        a_sf = torch.tensor([2.0 ** -6 * 3], dtype=torch.float32)
        w_sf = torch.tensor((2.0 ** -9) * np.array([1, 3, 5, 1, 7, 9], dtype=np.float32))
        if idx == 0:
            z_sf = torch.tensor([float(a_sf) * 2.0 ** -9 * 16], dtype=torch.float32)   # exact power-of-two ratios for channels 0,3 -> ties
        else:
            z_sf = torch.tensor([float(rng.uniform(0.01, 0.5))], dtype=torch.float32)
        acc = rng.randint(-(2 ** 17), 2 ** 17, size=(3, C, 5, 4)).astype(np.int64)
        acc[0, :, 0, :] = np.array([-24, -8, 8, 24])            # ties at ratio 1/16
        acc[0, :, 1, :] = np.array([40, 56, -40, -56])
        acc[1, :, 0, :] = np.array([0, 1, -1, 2 ** 20])
        z = torch.from_numpy(acc).float() * (a_sf.view(1, -1, 1, 1) * w_sf.view(1, -1, 1, 1))
        back = torch.round(z / a_sf.view(1, -1, 1, 1) / w_sf.view(1, -1, 1, 1)).long().numpy()
        assert np.array_equal(back, acc)
        q = qu.fixedpoint_fn.apply(z, bits, mode, z_sf, 0, a_sf, w_sf)
        cases.append(dict(bits=bits, mode=mode))
        out["c0_%d_acc" % idx] = acc
        out["c0_%d_a_sf" % idx] = a_sf.numpy()
        out["c0_%d_w_sf" % idx] = w_sf.numpy()
        out["c0_%d_z_sf" % idx] = z_sf.numpy()
        out["c0_%d_q" % idx] = q.numpy().astype(np.int64)
    out["c0_specs"] = np.array(json.dumps(cases))

    # SURVEY A.7 vectors
    a7 = []
    for ratio, acc in [(0.25, [-6, -2, 2, 6, 10, 1, 3, 5]), (1.0 / 16, list(range(0, 32))), (1.0 / 16, [-v for v in range(0, 32)])]:
        a_sf = torch.tensor([1.0]); w_sf = torch.tensor([ratio], dtype=torch.float32); z_sf = torch.tensor([1.0])
        z = torch.tensor(acc, dtype=torch.float32).view(1, 1, 1, -1) * ratio
        q = qu.fixedpoint_fn.apply(z, 16, 'symmetric', z_sf, 0, a_sf, w_sf)
        a7.append((ratio, acc, q.view(-1).long().tolist()))
    out["a7"] = np.array(json.dumps(a7))

    # case 1
    for idx in range(3):
        C = 5
        a_sf = torch.tensor([2.0 ** -7 * 5], dtype=torch.float32)
        w_sf = torch.tensor((2.0 ** -10) * np.array([1, 3, 5, 7, 11], dtype=np.float32))
        id_sf = torch.tensor([2.0 ** -8 * 3], dtype=torch.float32)
        id_w_sf = torch.ones(1) if idx == 0 else torch.tensor((2.0 ** -8) * np.array([3, 1, 9, 5, 7], dtype=np.float32))
        z_sf = torch.tensor([float(rng.uniform(0.001, 0.02))], dtype=torch.float32)
        acc = rng.randint(-(2 ** 16), 2 ** 16, size=(2, C, 4, 4)).astype(np.int64)
        idn = rng.randint(-(2 ** 15), 2 ** 15, size=(2, C, 4, 4)).astype(np.int64)
        wy = torch.from_numpy(acc).float() * (a_sf.view(1, -1, 1, 1) * w_sf.view(1, -1, 1, 1))
        ident = torch.from_numpy(idn).float() * (id_sf.view(1, -1, 1, 1) * id_w_sf.view(1, -1, 1, 1))
        z = wy + ident
        # the reference recovers wy_int from (z - identity); keep only cases where that is exact
        back = torch.round((z - ident) / a_sf.view(1, -1, 1, 1) / w_sf.view(1, -1, 1, 1)).long().numpy()
        ok = back == acc
        acc = np.where(ok, acc, back)
        q = qu.fixedpoint_fn.apply(z, 16, 'symmetric', z_sf, 1, a_sf, w_sf, ident, id_sf, id_w_sf)
        out["c1_%d_acc" % idx], out["c1_%d_id" % idx] = acc, idn
        out["c1_%d_a_sf" % idx], out["c1_%d_w_sf" % idx] = a_sf.numpy(), w_sf.numpy()
        out["c1_%d_id_sf" % idx], out["c1_%d_id_w_sf" % idx] = id_sf.numpy(), id_w_sf.numpy()
        out["c1_%d_z_sf" % idx] = z_sf.numpy()
        out["c1_%d_q" % idx] = q.numpy().astype(np.int64)
    np.savez_compressed(os.path.join(HERE, "kat_requant.npz"), **out)


def make_kat_modules(ns):
    qm = ns.quant_modules
    out = {}
    g = torch.Generator().manual_seed(3)
    # QuantAct input branch
    for bits, mode in [(8, 'symmetric'), (4, 'asymmetric')]:
        act = qm.QuantAct(activation_bit=bits, quant_mode=mode)
        x = torch.randn(2, 3, 6, 5, generator=g) * 2
        if mode == 'asymmetric':
            x = x.abs()
        with torch.no_grad():
            y, s = act(x)
        out["act_in_%d_x" % bits], out["act_in_%d_scale" % bits] = x.numpy(), s.numpy()
        out["act_in_%d_q" % bits] = torch.round(y / s).long().numpy()
        out["act_in_%d_range" % bits] = np.array([float(act.x_min), float(act.x_max)], dtype=np.float32)
    # QuantBnConv2d (folded BN) 3x3 s2 p1 and 1x1
    for tag, (cin, cout, k, s, p, wb) in {"bnconv_a": (8, 12, 3, 2, 1, 8), "bnconv_b": (16, 8, 1, 1, 0, 4)}.items():
        conv = torch.nn.Conv2d(cin, cout, k, s, p, bias=False)
        bn = torch.nn.BatchNorm2d(cout)
        with torch.no_grad():
            conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) * 0.2)
            bn.running_var.copy_(torch.rand(cout, generator=g) + 0.5)
            bn.running_mean.copy_(torch.randn(cout, generator=g) * 0.1)
            bn.weight.copy_(torch.rand(cout, generator=g) + 0.5)
            bn.bias.copy_(torch.randn(cout, generator=g) * 0.1)
        mod = qm.QuantBnConv2d(weight_bit=wb, bias_bit=32, per_channel=True, fix_BN=True)
        mod.set_param(conv, bn)
        mod.quantize_bias = True
        mod.fix()
        a_sf = torch.tensor([0.0123], dtype=torch.float32)
        hi = 127 if wb == 8 else 15
        lo = -128 if wb == 8 else 0
        xi = torch.randint(lo, hi + 1, (2, cin, 7, 6), generator=g).float()
        with torch.no_grad():
            y, w_sf = mod(xi * a_sf, a_sf)
        acc = torch.round(y / (w_sf.view(1, -1, 1, 1) * a_sf.view(1, -1, 1, 1))).long()
        out[tag + "_conv_w"], out[tag + "_bn"] = conv.weight.detach().numpy(), np.stack(
            [bn.running_mean.numpy(), bn.running_var.numpy(), bn.weight.detach().numpy(), bn.bias.detach().numpy()])
        out[tag + "_cfg"] = np.array([cin, cout, k, s, p, wb])
        out[tag + "_x_int"], out[tag + "_a_sf"] = xi.long().numpy(), a_sf.numpy()
        out[tag + "_w_int"], out[tag + "_b_int"] = mod.weight_integer.long().numpy(), mod.bias_integer.long().numpy()
        out[tag + "_w_sf"], out[tag + "_acc"] = w_sf.numpy(), acc.numpy()
    # QuantConv2d with bias
    conv = torch.nn.Conv2d(8, 8, 3, 1, 1, bias=True)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) * 0.2)
        conv.bias.copy_(torch.randn(8, generator=g) * 0.3)
    mod = qm.QuantConv2d(weight_bit=8, bias_bit=32, per_channel=True)
    mod.set_param(conv)
    a_sf = torch.tensor([0.02], dtype=torch.float32)
    xi = torch.randint(-128, 128, (1, 8, 5, 5), generator=g).float()
    with torch.no_grad():
        y, w_sf = mod(xi * a_sf, a_sf)
    out["conv_w"], out["conv_b"] = conv.weight.detach().numpy(), conv.bias.detach().numpy()
    out["conv_x_int"], out["conv_a_sf"] = xi.long().numpy(), a_sf.numpy()
    out["conv_w_int"], out["conv_b_int"], out["conv_w_sf"] = mod.weight_integer.long().numpy(), mod.bias_integer.long().numpy(), w_sf.numpy()
    out["conv_acc"] = torch.round(y / (w_sf.view(1, -1, 1, 1) * a_sf.view(1, -1, 1, 1))).long().numpy()
    # QuantLinear
    lin = torch.nn.Linear(32, 10)
    with torch.no_grad():
        lin.weight.copy_(torch.randn(10, 32, generator=g) * 0.1)
        lin.bias.copy_(torch.randn(10, generator=g) * 0.2)
    mod = qm.QuantLinear(weight_bit=8, bias_bit=32, per_channel=True)
    mod.set_param(lin)
    a_sf = torch.tensor([0.031], dtype=torch.float32)
    xi = torch.randint(-128, 128, (3, 32), generator=g).float()
    with torch.no_grad():
        y = mod(xi * a_sf, a_sf)
    out["lin_w"], out["lin_b"], out["lin_x_int"], out["lin_a_sf"] = lin.weight.detach().numpy(), lin.bias.detach().numpy(), xi.long().numpy(), a_sf.numpy()
    out["lin_w_int"], out["lin_b_int"], out["lin_w_sf"] = mod.weight_integer.long().numpy(), mod.bias_integer.long().numpy(), mod.fc_scaling_factor.numpy()
    out["lin_y"] = y.numpy()
    # QuantAveragePool2d (incl. negative sums to pin the trunc(x + 0.01) rule)
    pool = qm.QuantAveragePool2d(kernel_size=7, stride=1)
    sf = torch.tensor([0.004], dtype=torch.float32)
    xi = torch.randint(-300, 3000, (2, 6, 7, 7), generator=g).float()
    xi[0, 0] = -1.0            # sum -49 -> exact negative multiple
    xi[0, 1] = 0.0
    xi[0, 1, 0, 0] = -48.0     # sum -48
    xi[0, 2] = 2.0             # sum 98 -> 2
    xi[1, 0] = -2.0
    xi[1, 0, 0, 0] = -3.0      # sum -99
    with torch.no_grad():
        y, s2 = pool(xi * sf, sf)
    out["pool_x_int"], out["pool_sf"] = xi.long().numpy(), sf.numpy()
    out["pool_q"] = torch.round(y / s2).long().numpy()
    np.savez_compressed(os.path.join(HERE, "kat_modules.npz"), **out)


def make_net(ns, arch, scheme):
    qm = ns.quant_modules
    net = synthetic_float_resnet(arch, 0)
    calib = synthetic_batch(CALIB_BATCH, CALIB_SEED)
    q = rh.build_reference_qresnet(arch, scheme, net, calib)
    x = synthetic_batch(PARITY_BATCH, PARITY_SEED)
    logits, acts = rh.run_with_act_hooks(q, x)
    out = {"logits": logits.numpy()}
    meta = {"arch": arch, "scheme": scheme, "calib": [CALIB_BATCH, CALIB_SEED], "input": [PARITY_BATCH, PARITY_SEED],
            "acts": {}, "convs": {}, "torch": torch.__version__}
    for name, mod in q.named_modules():
        if type(mod) is qm.QuantAct:
            a = nhwc(acts[name])
            meta["acts"][name] = dict(x_min=float(mod.x_min), x_max=float(mod.x_max), scale=float(mod.act_scaling_factor),
                                      bits=mod.activation_bit, mode=mod.quant_mode, shape=list(a.shape),
                                      sha=sha_i32(a), sum=int(a.sum()), abssum=int(np.abs(a).sum()),
                                      min=int(a.min()), max=int(a.max()))
        elif type(mod) is qm.QuantBnConv2d:
            w = mod.weight_integer.numpy().transpose(0, 2, 3, 1)      # OHWI
            meta["convs"][name] = dict(w_sha=sha_i32(w), b_sha=sha_i32(mod.bias_integer.numpy()),
                                       w_bits=mod.weight_bit, shape=list(w.shape),
                                       sf_sha=hashlib.sha256(mod.convbn_scaling_factor.numpy().tobytes()).hexdigest())
        elif type(mod) is qm.QuantLinear:
            meta["fc"] = dict(w_sha=sha_i32(mod.weight_integer.numpy()), b_sha=sha_i32(mod.bias_integer.numpy()),
                              sf_sha=hashlib.sha256(mod.fc_scaling_factor.numpy().tobytes()).hexdigest())
    out["meta"] = np.array(json.dumps(meta))
    np.savez_compressed(os.path.join(HERE, "net_%s_%s.npz" % (arch, scheme)), **out)
    print(arch, scheme, "ok", logits[0, :3].tolist())


def make_net_mobilenetv2(ns, scheme):
    """MobileNetV2-1.0 (reference utils/models/q_mobilenetv2.py) on the synthetic skeleton: frozen logits, every QuantAct's
    integers, integer weights / biases of every convolution (depthwise ones included) and of the 1x1 classifier."""
    from hawq_b200.synthetic import synthetic_float_mobilenetv2
    qm = ns.quant_modules
    net = synthetic_float_mobilenetv2(0)
    calib = synthetic_batch(CALIB_BATCH, CALIB_SEED)
    q = rh.build_reference_qmobilenetv2(scheme, net, calib)
    x = synthetic_batch(PARITY_BATCH, PARITY_SEED)
    logits, acts = rh.run_with_act_hooks(q, x)
    out = {"logits": logits.numpy()}
    meta = {"arch": "mobilenetv2_w1", "scheme": scheme, "calib": [CALIB_BATCH, CALIB_SEED], "input": [PARITY_BATCH, PARITY_SEED],
            "acts": {}, "convs": {}, "torch": torch.__version__}
    for name, mod in q.named_modules():
        if type(mod) is qm.QuantAct:
            a = nhwc(acts[name])
            meta["acts"][name] = dict(x_min=float(mod.x_min), x_max=float(mod.x_max), scale=float(mod.act_scaling_factor),
                                      bits=mod.activation_bit, mode=mod.quant_mode, shape=list(a.shape),
                                      sha=sha_i32(a), sum=int(a.sum()), abssum=int(np.abs(a).sum()),
                                      min=int(a.min()), max=int(a.max()))
        elif type(mod) in (qm.QuantBnConv2d, qm.QuantConv2d):
            w = mod.weight_integer.numpy().transpose(0, 2, 3, 1)      # OHWI (I = 1 for depthwise)
            b = mod.bias_integer
            sf = mod.convbn_scaling_factor if type(mod) is qm.QuantBnConv2d else mod.conv_scaling_factor
            meta["convs"][name] = dict(w_sha=sha_i32(w), b_sha=sha_i32(b.numpy()) if b is not None else None,
                                       w_bits=mod.weight_bit, shape=list(w.shape), groups=int(mod.conv.groups) if hasattr(mod, "conv") else 1,
                                       sf_sha=hashlib.sha256(sf.numpy().tobytes()).hexdigest())
    out["meta"] = np.array(json.dumps(meta))
    np.savez_compressed(os.path.join(HERE, "net_mobilenetv2_w1_%s.npz" % scheme), **out)
    print("mobilenetv2_w1", scheme, "ok", logits[0, :3].tolist())


def make_kat_multibranch(ns):
    """The reference's un-frozen QuantAct on a (tensor, [scale per branch], [channels per branch]) input."""
    out = {}
    g = torch.Generator().manual_seed(11)
    for i, (bits, mode) in enumerate([(8, "symmetric"), (4, "asymmetric"), (8, "asymmetric")]):
        act = ns.quant_modules.QuantAct(activation_bit=bits, quant_mode=mode)
        scales = [torch.tensor([0.021]), torch.tensor([0.0173]), torch.tensor([0.05])]
        chans = [3, 5, 2]
        lo = 0 if mode == "asymmetric" else -100
        x = torch.cat([torch.randint(lo, 100, (2, c, 4, 4), generator=g).float() * s for c, s in zip(chans, scales)], dim=1)
        y, sf = act((x.clone(), [s.clone() for s in scales], chans))
        out["mb_%d_x" % i] = x.numpy()
        out["mb_%d_y" % i] = y.numpy()
        out["mb_%d_sf" % i] = sf.view(-1).numpy()
    out["specs"] = np.array(json.dumps([dict(bits=b, mode=m) for b, m in [(8, "symmetric"), (4, "asymmetric"), (8, "asymmetric")]]))
    np.savez_compressed(os.path.join(HERE, "kat_multibranch.npz"), **out)
    print("kat_multibranch ok")


DROPIN_CONFIGS = [("resnet18", "uniform4"), ("resnet50", "bops_0.5"), ("mobilenetv2_w1", "uniform8")]


def make_ref_dropin(ns):
    """What tests/test_reference_dropin.py compares the reference's graph code against: the order in which the reference's
    ResNet / MobileNetV2 graph code calls its quant modules in the un-frozen calibration forward, and the fp32 output of a second
    un-frozen MobileNetV2 forward (the reference's own modules, ranges still moving)."""
    from hawq_b200.synthetic import synthetic_float_mobilenetv2
    from tests.util import QUANT_MODULES, quant_call_order
    kinds = tuple(getattr(ns.quant_modules, n) for n in QUANT_MODULES)
    out = {}
    calib = synthetic_batch(CALIB_BATCH, CALIB_SEED)
    for arch, scheme in DROPIN_CONFIGS:
        if arch == "mobilenetv2_w1":
            q = ns.q_mobilenetv2.q_mobilenetv2_w1(synthetic_float_mobilenetv2(0))
        else:
            q = {"resnet18": ns.q_resnet.q_resnet18, "resnet50": ns.q_resnet.q_resnet50}[arch](synthetic_float_resnet(arch, 0))
        rh.stamp_like_quant_train(q, ns.bit_config_dict["bit_config_%s_%s" % (arch, scheme)])
        q.eval()
        order = quant_call_order(q, calib, kinds)
        out["calls_%s_%s" % (arch, scheme)] = np.array(json.dumps(order))
        if arch == "mobilenetv2_w1":
            with torch.no_grad():
                out["unfrozen_%s_%s" % (arch, scheme)] = q(synthetic_batch(PARITY_BATCH, PARITY_SEED)).numpy()
    np.savez_compressed(os.path.join(HERE, "ref_dropin.npz"), **out)
    print("ref_dropin ok", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    torch.set_num_threads(os.cpu_count())
    ns = rh.load()
    if len(sys.argv) == 2 and sys.argv[1] == "--multibranch":  # QuantAct on concatenated branches (quant_modules.py:275-286)
        make_kat_multibranch(ns)
        sys.exit(0)
    if len(sys.argv) == 2 and sys.argv[1] == "--dropin":      # reference graph code: quant-module call order, un-frozen output
        make_ref_dropin(ns)
        sys.exit(0)
    if len(sys.argv) == 3 and sys.argv[1] == "--mobilenetv2":  # e.g. --mobilenetv2 uniform8
        make_net_mobilenetv2(ns, sys.argv[2])
        sys.exit(0)
    if len(sys.argv) == 4 and sys.argv[1] == "--net":         # one extra network golden, e.g. --net resnet101 uniform8
        make_net(ns, sys.argv[2], sys.argv[3])
        sys.exit(0)
    make_kat_requant(ns)
    make_kat_modules(ns)
    for arch, scheme in NET_CONFIGS:
        make_net(ns, arch, scheme)
