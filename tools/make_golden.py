#!/usr/bin/env python
"""Generate tests/golden/* by RUNNING THE REFERENCE (jakc4103/DFQ, imported unmodified from /root/reference) in the
build container.  Committed next to its outputs so every fixture can be regenerated.

  topology_<model>.json   node types / layer hyper-parameters / edges of the reference's own trace (PyTransformer) of
                          MobileNetV2, ResNet-18, DeepLab-v3+ (MobileNetV2) and MobileNetV2-SSD-lite with ReLU6 -> ReLU
  ref_<model>.npz         results of the reference's merge_batchnorm -> create_relation -> cross_layer_equalization
                          -> bias_correction (-> quantize_targ_layer) on the seeded random model that
                          dfq_b200.workload.build_graph materialises from the topology: relation lists, sweep counts,
                          every S / bias / fake_weight / fake_bias vector, and per-layer weight digests
                          (sha256 + max|w| + fp64 sum) after each stage
  ref_ops.npz             op-level vectors: _layer_equalization on the shapes of Appendix B, UniformQuantize codes,
                          QuantMeasure updates, _quantize_error

  ref_bc_<model>.npz      the reference's dfq.bias_correction ALONE on seed-regenerable inputs (tests/bc_fixture.py):
                          every post-correction bias and fake_bias vector + sha256 of every input tensor
  main_<cls|seg|ssd>.npz  made by tests/main_harness.py --impl reference (the unmodified main scripts end to end)
  ref_equalization_exact.npz, ref_op_patching.npz, ref_distill.npz
                          the reference's outputs on the seeded inputs of the bit-exact equalization pins, the
                          op-patching test and the distilled-data test (pin_fixtures)

usage: python tools/make_golden.py [topology] [mobilenetv2] [resnet18] [deeplab] [ssd] [ops] [bc] [minmax] [table] [pins]
"""
import hashlib
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

import refenv  # noqa: E402

ref = refenv.install()
os.chdir(refenv.REF_ROOT)
from dfq_b200 import workload  # noqa: E402  (pure python/torch; builds the seeded graphs)


def digest(t: torch.Tensor):
    a = np.ascontiguousarray(t.detach().cpu().numpy())
    return hashlib.sha256(a.tobytes()).hexdigest(), float(np.abs(a).max()), float(a.astype(np.float64).sum())


# ---------------------------------------------------------------------------------------------------------
def trace_topology(name):
    TT = refenv.tracer()
    if name == "mobilenetv2":
        from modeling.classification.MobileNetV2 import mobilenet_v2
        model, data = mobilenet_v2(None), torch.ones((4, 3, 224, 224))
    elif name == "resnet18":
        import torchvision.models as models
        model, data = models.resnet18(), torch.ones((4, 3, 224, 224))
    elif name == "deeplab":
        from modeling.segmentation.deeplab import DeepLab
        model, data = DeepLab(sync_bn=False), torch.ones((4, 3, 513, 513))
    elif name == "ssd":
        from modeling.detection.mobilenet_v2_ssd_lite import create_mobilenetv2_ssd_lite
        model, data = create_mobilenetv2_ssd_lite(21, width_mult=1.0), torch.ones((4, 3, 300, 300))
    else:
        raise ValueError(name)
    model.eval()
    tr = TT()
    model, tr = ref.layer_transform.switch_layers(model, tr, data, {0: [(nn.ReLU6, nn.ReLU)]},
                                                  ignore_layer=[ref.quantize.QuantMeasure], quant_op=False)
    graph, bottoms = tr.log.getGraph(), tr.log.getBottoms()
    names, nodes = {}, []
    for i, key in enumerate(graph):
        if key == "Data":
            nm, rec = "Data", dict(type="Data")
        elif isinstance(graph[key], str):
            nm, rec = key, dict(type="Func")
        else:
            nm = "m%d" % i
            rec = workload.describe_module(graph[key])
        names[key] = nm
        b = bottoms[key]
        rec.update(key=nm, bottoms=None if b is None else [names[x] for x in b])
        nodes.append(rec)
    topo = dict(name=name, input=list(data.shape), source="reference trace (PyTransformer), ReLU6 -> ReLU", nodes=nodes)
    with open(os.path.join(GOLD, "topology_%s.json" % name), "w") as f:
        json.dump(topo, f, separators=(",", ":"))
    print(name, len(nodes), "nodes")
    return topo


# ---------------------------------------------------------------------------------------------------------
def run_reference_pipeline(name, seed=0, signed=False, quantize=True, s_range=(1e-8, 1e8), delete_single=False):
    topo = workload.load_topology(os.path.join(GOLD, "topology_%s.json" % name))
    graph, bottoms, _ = workload.build_graph(topo, seed=seed)
    targ = [nn.Conv2d, nn.Linear]
    keys = list(graph.keys())
    pos = {k: i for i, k in enumerate(keys)}
    out = {}
    t0 = time.time()
    ref.layer_transform.merge_batchnorm(None, graph, bottoms, targ)
    rels = ref.relation.create_relation(graph, bottoms, targ, delete_single=delete_single)
    out["relations"] = np.array([[pos[a], pos[b], pos[c]] for a, b, c in (r.get_idxs() for r in rels)], np.int64)
    tl = [k for k in keys if type(graph[k]) in targ]
    out["targets"] = np.array([pos[k] for k in tl], np.int64)

    def stage(tag):
        dg = [digest(graph[k].weight) for k in tl]
        out[tag + "_w_sha"] = np.array([d[0] for d in dg])
        out[tag + "_w_absmax"] = np.array([d[1] for d in dg])
        out[tag + "_w_sum"] = np.array([d[2] for d in dg])
        for k in tl:
            if graph[k].bias is not None:
                out["%s_bias_%d" % (tag, pos[k])] = graph[k].bias.detach().numpy().copy()
        for k in keys:
            if hasattr(graph[k], "fake_bias") and not isinstance(graph[k], str):
                out["%s_fb_%d" % (tag, pos[k])] = graph[k].fake_bias.numpy().copy()
                out["%s_fw_%d" % (tag, pos[k])] = graph[k].fake_weight.numpy().copy()

    stage("fold")
    # count sweeps by wrapping _layer_equalization
    calls = [0]
    orig = ref.dfq._layer_equalization

    def counted(*a, **kw):
        calls[0] += 1
        return orig(*a, **kw)
    ref.dfq._layer_equalization = counted
    ref.dfq.cross_layer_equalization(graph, rels, targ, s_range=list(s_range), converge_thres=2e-7, signed=signed)
    ref.dfq._layer_equalization = orig
    out["n_sweeps"] = np.array(calls[0] // max(1, len(rels)))
    for i, r in enumerate(rels):
        out["S_%d" % i] = r.S.numpy().copy()
    stage("cle")
    ref.dfq.bias_correction(graph, bottoms, targ, signed=signed)
    stage("bc")
    if quantize:
        ref.layer_transform.quantize_targ_layer(graph, 8, 16, targ)
        stage("q")
    out["meta"] = np.array(json.dumps(dict(model=name, seed=seed, signed=signed, s_range=list(s_range),
                                           delete_single=delete_single, torch=torch.__version__,
                                           seconds=round(time.time() - t0, 1))))
    suffix = ("_signed" if signed else "")
    np.savez_compressed(os.path.join(GOLD, "ref_%s%s.npz" % (name, suffix)), **out)
    print(name, "sweeps", int(out["n_sweeps"]), "relations", len(rels), "%.1fs" % (time.time() - t0))


# ---------------------------------------------------------------------------------------------------------
def op_vectors():
    out = {}
    torch.manual_seed(1)
    shapes = {"dense_dw": ((32, 3, 3, 3), (32, 1, 3, 3)), "dw_pw": ((96, 1, 3, 3), (24, 96, 1, 1)),
              "pw_dw": ((144, 24, 1, 1), (144, 1, 3, 3)), "pw_pw": ((320, 96, 1, 1), (128, 320, 1, 1)),
              "pw_fc": ((128, 32, 1, 1), (10, 128)), "dense": ((64, 32, 3, 3), (48, 64, 3, 3)),
              "grouped": ((32, 8, 3, 3), (24, 16, 3, 3))}
    for tag, (s1, s2) in shapes.items():
        for signed in (False, True):
            w1 = torch.randn(*s1) * (10 ** torch.empty(s1[0]).uniform_(-1, 1)).view(-1, *([1] * (len(s1) - 1)))
            w2 = torch.randn(*s2)
            b1, bw, bb = torch.randn(s1[0]), torch.rand(s1[0]) + 0.5, torch.randn(s1[0])
            key = "eq_%s_%d" % (tag, int(signed))
            for n, t in (("w1", w1), ("w2", w2), ("b1", b1), ("bw", bw), ("bb", bb)):
                out["%s_in_%s" % (key, n)] = t.numpy().copy()
            r = ref.dfq._layer_equalization(w1, w2, b1, bw, bb, signed=signed)
            for n, t in (("w1", w1), ("w2", w2), ("b1", b1), ("bw", bw), ("bb", bb), ("S", r[3])):
                out["%s_out_%s" % (key, n)] = t.numpy().copy()
    # fake-quant codes on the reference's CPU path
    for bits in (8, 4, 16):
        for sym in (False, True):
            x = torch.randn(4096) * 3
            y = ref.quantize.quantize(x, bits, float(x.min()), float(x.max()), symmetric=sym)
            out["q_%d_%d_in" % (bits, int(sym))] = x.numpy().copy()
            out["q_%d_%d_out" % (bits, int(sym))] = y.numpy().copy()
    x = torch.randn(2000)
    out["qerr_in"] = x.numpy().copy()
    out["qerr_out"] = ref.dfq._quantize_error(x, 8, None).numpy().copy()
    out["qerr_out_signed"] = ref.dfq._quantize_error(x, 8, None, True).numpy().copy()
    # implicit-range path (bias quantization in Quant*/Q* layers, min_value=None)
    b = torch.randn(257)
    out["qimp_in"] = b.numpy().copy()
    out["qimp_out16"] = ref.quantize.quantize(b, num_bits=16).numpy().copy()
    out["qimp_out8"] = ref.quantize.quantize(b, num_bits=8).numpy().copy()
    # observer
    qm = ref.quantize.QuantMeasure(True)
    qm.eval()
    acts = torch.randn(8, 3, 16, 16)
    y = qm(acts)
    out["obs_in"] = acts.numpy().copy(); out["obs_out"] = y.numpy().copy()
    out["obs_min"] = np.array(float(qm.running_min)); out["obs_max"] = np.array(float(qm.running_max))
    qm2 = ref.quantize.QuantMeasure(False)
    qm2.train()
    y2 = qm2(acts)
    out["ema_out"] = y2.detach().numpy().copy()
    out["ema_min"] = np.array(float(qm2.running_min)); out["ema_max"] = np.array(float(qm2.running_max))
    # relu expectation as bias_correction forms it
    from scipy.stats import norm
    g = torch.rand(300) + 0.2; bta = torch.randn(300)
    e = g * torch.from_numpy(norm(0, 1).pdf(-bta / g)).float() + bta * (1 - torch.from_numpy(norm.cdf(-bta / g)).float())
    e[e < 0] = 0
    out["expect_g"] = g.numpy().copy(); out["expect_b"] = bta.numpy().copy(); out["expect_out"] = e.numpy().copy()
    np.savez_compressed(os.path.join(GOLD, "ref_ops.npz"), **out)
    print("ops", len(out))


if __name__ == "__main__":
    what = sys.argv[1:] or ["topology", "ops", "resnet18", "mobilenetv2"]
    os.makedirs(GOLD, exist_ok=True)
    if "topology" in what:
        for m in ("mobilenetv2", "resnet18", "deeplab", "ssd"):
            try:
                trace_topology(m)
            except Exception as e:  # noqa
                print("topology", m, "FAILED:", repr(e))
    if "ops" in what:
        op_vectors()
    if "resnet18" in what:
        run_reference_pipeline("resnet18", seed=3)
    if "mobilenetv2" in what:
        run_reference_pipeline("mobilenetv2", seed=0)
    if "mobilenetv2_signed" in what:
        run_reference_pipeline("mobilenetv2", seed=0, signed=True, quantize=False)
    if "deeplab" in what:
        run_reference_pipeline("deeplab", seed=5)
    if "ssd" in what:
        run_reference_pipeline("ssd", seed=7, delete_single=True)


# ---------------------------------------------------------------------------------------------------------
def quant_minmax_fixture(name="mobilenetv2", seed=0):
    """set_quant_minmax (layer_transform.py:347-609) needs the tracer's record of functional ops; trace the reference
    model with Quant layers + observers, store the op record with the topology, run the reference calibration on the
    seeded topology-built graph and store every observer's running_min / running_max."""
    TT = refenv.tracer()
    Q = ref.quantize
    if name == "mobilenetv2":
        from modeling.classification.MobileNetV2 import mobilenet_v2
        model, data = mobilenet_v2(None), torch.ones((4, 3, 224, 224))
    elif name == "resnet18":
        import torchvision.models as models
        model, data = models.resnet18(), torch.ones((4, 3, 224, 224))
    model.eval()
    tr = TT()
    md = {0: [(nn.ReLU6, nn.ReLU)], 1: [(nn.Conv2d, Q.QuantNConv2d), (nn.Linear, Q.QuantNLinear)]}
    model, tr = ref.layer_transform.switch_layers(model, tr, data, md, ignore_layer=[Q.QuantMeasure], quant_op=True)
    record = [list(x) for x in model.name_tensor_op]
    topo = workload.load_topology(os.path.join(GOLD, "topology_%s.json" % name))
    graph0 = tr.log.getGraph()
    assert len(graph0) == len(topo["nodes"]), (len(graph0), len(topo["nodes"]))
    topo["tensor_ops"] = record
    with open(os.path.join(GOLD, "topology_%s.json" % name), "w") as f:
        json.dump(topo, f, separators=(",", ":"))
    # reference calibration on the seeded graph built from the topology, with the reference's own Quant classes
    graph, bottoms, _ = workload.build_graph(topo, seed=seed, conv_cls=Q.QuantNConv2d, linear_cls=Q.QuantNLinear)
    targ = [Q.QuantNConv2d, Q.QuantNLinear]
    LT = ref.layer_transform
    ops = []
    for _, op_name in record:
        ops.extend(Q.QuantMeasure(num_bits=8, momentum=0.1) for _ in range(int(op_name.split('_')[-1])))
    LT.module_tensor_op = LT.CustomTensorOP(ops, [tuple(x) for x in record])
    LT.merge_batchnorm(None, graph, bottoms, targ)
    rels = ref.relation.create_relation(graph, bottoms, targ)
    ref.dfq.cross_layer_equalization(graph, rels, targ, converge_thres=2e-7)
    ref.dfq.bias_correction(graph, bottoms, targ)
    LT.set_quant_minmax(graph, bottoms, verbose=False)
    out = {}
    for i, k in enumerate(graph):
        m = graph[k]
        if hasattr(m, "quant") and not isinstance(m, str):
            out["layer_%d" % i] = np.array([float(m.quant.running_min), float(m.quant.running_max)])
    for j, qm in enumerate(ops):
        out["op_%d" % j] = np.array([float(qm.running_min), float(qm.running_max)])
    np.savez_compressed(os.path.join(GOLD, "ref_minmax_%s.npz" % name), **out)
    print("minmax", name, len(out), "observers;", len(record), "functional ops")


if __name__ == "__main__" and "minmax" in sys.argv[1:]:
    quant_minmax_fixture("mobilenetv2", 0)
    quant_minmax_fixture("resnet18", 3)


# ---------------------------------------------------------------------------------------------------------
def bias_correction_fixture(name):
    """dfq.py:173-293 alone: inputs from tests/bc_fixture.py, outputs of the reference."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import bc_fixture
    graph, bottoms = bc_fixture.build(name)
    out = {"digests": bc_fixture.input_digests(graph), "seed": np.array(bc_fixture.SEEDS[name])}
    ref.dfq.bias_correction(graph, bottoms, bc_fixture.TARG)
    n = 0
    for i, k in enumerate(graph):
        m = graph[k]
        if type(m) in bc_fixture.TARG and m.bias is not None:
            out["out_b_%d" % i] = m.bias.detach().numpy().copy(); n += 1
        elif hasattr(m, "fake_bias") and not isinstance(m, str):
            out["out_fb_%d" % i] = m.fake_bias.numpy().copy()
    np.savez_compressed(os.path.join(GOLD, "ref_bc_%s.npz" % name), **out)
    print("bc", name, n, "corrected layers")


if __name__ == "__main__" and "bc" in sys.argv[1:]:
    bias_correction_fixture("resnet18")
    bias_correction_fixture("mobilenetv2")


# ---------------------------------------------------------------------------------------------------------
def ncnn_table_rows():
    """The 53 + 53 scale values of the reference's checked-in table (modeling/ncnn/model_quant_relu_equal.table): rows 1-53
    `<layer>_param_0 s s s ...` (first value = 128/max|W|), rows 54-106 `<layer> s` (activation scale)."""
    rows = [l.split() for l in open(os.path.join(refenv.REF_ROOT, "modeling", "ncnn", "model_quant_relu_equal.table")).read().strip().splitlines()]
    assert len(rows) == 106
    np.savez_compressed(os.path.join(GOLD, "ncnn_table_rows.npz"), weight_scales=np.array([float(r[1]) for r in rows[:53]]),
                        activation_scales=np.array([float(r[1]) for r in rows[53:]]),
                        names=np.array([r[0] for r in rows[53:]]))
    print("ncnn table rows: 53 + 53")


if __name__ == "__main__" and "table" in sys.argv[1:]:
    ncnn_table_rows()


# ---------------------------------------------------------------------------------------------------------
def pin_fixtures():
    """What the reference computes on the inputs that three tests build from seeds (the inputs are regenerated by the
    tests themselves, so only the reference's outputs are stored)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_distill
    import test_op_patching
    import test_oracle_pins as P
    out = {}
    for i, (s1, s2, opt) in enumerate(P.CASES):
        for signed in (False, True):
            ts, kw = P.equalization_case(s1, s2, opt, signed)
            r = ref.dfq._layer_equalization(*ts, signed=signed, **kw)
            key = "c%d_s%d_" % (i, signed)
            for name, t in zip(P.EQ_NAMES, ts + [r[3]]):
                out[key + name] = P.equalization_digest(t.numpy()) if name in ("w1", "w2") else t.numpy().copy()
    np.savez_compressed(os.path.join(GOLD, "ref_equalization_exact.npz"), **out)
    outs, order = test_op_patching.reference_run(ref.layer_transform, ref.quantize.QuantMeasure)
    np.savez_compressed(os.path.join(GOLD, "ref_op_patching.npz"), observer_order=np.array(order), n_outputs=np.array(len(outs)),
                        **{"output_%d" % k: o.numpy() for k, o in enumerate(outs)})
    import run_main
    run_main.prepare_environment(use_dropin=False)
    from ZeroQ.distill_data import getDistilData
    model = test_distill._tiny()
    torch.manual_seed(123)
    batches = getDistilData(model, "imagenet", 2, **test_distill.DISTIL_ARGS)
    samples, means = test_distill.distil_digest(batches)
    np.savez_compressed(os.path.join(GOLD, "ref_distill.npz"), n_batches=np.array(len(batches)), **samples, **means)
    print("pins: %d equalization arrays, %d op-patching outputs, %d distilled batches" % (len(out), len(outs), len(batches)))


if __name__ == "__main__" and "pins" in sys.argv[1:]:
    pin_fixtures()
