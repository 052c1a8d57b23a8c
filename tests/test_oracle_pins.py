"""Pin the numpy oracle: (1) against fixtures produced by running the reference itself (tests/golden/ref_ops.npz,
tests/golden/ref_equalization_exact.npz, tools/make_golden.py), (2) live against the reference's checked-in ncnn
calibration table when the reference tree is present."""
import os
import sys

import numpy as np
import pytest

from oracle import dfq_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
REF = os.environ.get("DFQ_REFERENCE_ROOT", "/root/reference")
have_ref = os.path.isfile(os.path.join(REF, "dfq.py"))


def _nw(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


@pytest.fixture(scope="module")
def ops():
    return np.load(os.path.join(GOLD, "ref_ops.npz"))


TAGS = ["dense_dw", "dw_pw", "pw_dw", "pw_pw", "pw_fc", "dense", "grouped"]


@pytest.mark.parametrize("tag", TAGS)
@pytest.mark.parametrize("signed", [0, 1])
def test_layer_equalization_vs_reference_fixture(ops, tag, signed):
    """The reference's torch.sqrt is only faithful (<= 1 ulp, MKL VML) so S may differ in the last bit: 1e-6 normwise
    here, bit-exact in the live test below where the same sqrt can be injected."""
    key = "eq_%s_%d" % (tag, signed)
    t = {n: ops["%s_in_%s" % (key, n)].copy() for n in ("w1", "w2", "b1", "bw", "bb")}
    S = O.layer_equalization(t["w1"], t["w2"], t["b1"], t["bw"], t["bb"], signed=bool(signed))
    for n in ("w1", "w2", "b1", "bw", "bb"):
        assert _nw(t[n], ops["%s_out_%s" % (key, n)]) < 1e-6, n
    assert _nw(S, ops["%s_out_S" % key]) < 1e-6
    # at most a few channels may sit on a rounding boundary of the sqrt
    assert (S != ops["%s_out_S" % key]).mean() < 0.05


@pytest.mark.parametrize("bits", [8, 4, 16])
@pytest.mark.parametrize("sym", [0, 1])
def test_fake_quant_bit_exact_vs_reference_fixture(ops, bits, sym):
    x = ops["q_%d_%d_in" % (bits, sym)]
    y = O.quantize(x, bits, float(x.min()), float(x.max()), symmetric=bool(sym))
    assert np.array_equal(y, ops["q_%d_%d_out" % (bits, sym)])


def test_quantize_error_bit_exact(ops):
    assert np.array_equal(O.quantize_error(ops["qerr_in"]), ops["qerr_out"])
    assert np.array_equal(O.quantize_error(ops["qerr_in"], 8, True), ops["qerr_out_signed"])


def test_relu_expectation_matches_reference(ops):
    e = O.relu_expectation(ops["expect_g"], ops["expect_b"])
    assert _nw(e, ops["expect_out"]) < 1e-7


def test_observer_matches_reference(ops):
    x = ops["obs_in"]
    mn, mx = O.observer_update(0.0, 0.0, x)
    assert abs(float(mn) - float(ops["obs_min"])) <= 1e-6 * abs(float(ops["obs_min"]))
    assert abs(float(mx) - float(ops["obs_max"])) <= 1e-6 * abs(float(ops["obs_max"]))
    y = O.quantize(x, 8, float(ops["obs_min"]), float(ops["obs_max"]))
    assert np.array_equal(y, ops["obs_out"])
    rmin, rmax, bmin, bmax = O.observer_ema(0.0, 0.0, x, 0.1)
    assert abs(float(rmin) - float(ops["ema_min"])) <= 2e-6 * abs(float(ops["ema_min"]))
    assert abs(float(rmax) - float(ops["ema_max"])) <= 2e-6 * abs(float(ops["ema_max"]))


def test_eager_port_agrees_with_numpy_oracle():
    """oracle/eager_port.py (the timing companion with the reference's execution structure) == the numpy checker."""
    import torch
    from oracle import eager_port as E
    g = torch.Generator().manual_seed(4)
    w1 = torch.randn(24, 12, 3, 3, generator=g) * (10 ** torch.empty(24).uniform_(-1, 1, generator=g)).view(-1, 1, 1, 1)
    w2 = torch.randn(16, 24, 3, 3, generator=g)
    b1, bw, bb = torch.randn(24, generator=g), torch.rand(24, generator=g) + 0.5, torch.randn(24, generator=g)
    n = [t.clone().numpy() for t in (w1, w2, b1, bw, bb)]
    S = O.layer_equalization(*n)
    S2 = E.equalize_pair_(w1, w2, b1, bw, bb)
    assert _nw(S2.numpy(), S) < 1e-6 and _nw(w1.numpy(), n[0]) < 1e-6 and _nw(w2.numpy(), n[1]) < 1e-6
    x = torch.randn(500, generator=g)
    assert np.array_equal(E.fake_quant(x).numpy(), O.quantize(x.numpy(), 8, float(x.min()), float(x.max())))


# ---------------------------------------------------------------------------------------------------------
# bit-exact pins (the reference's torch.sqrt injected into the oracle)
# ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ref():
    if not have_ref:
        pytest.skip("reference tree not present")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import refenv
    return refenv.install()


def _torch_sqrt(x):
    import torch
    return torch.sqrt(torch.from_numpy(np.ascontiguousarray(x))).numpy()


CASES = [((32, 16, 3, 3), (24, 32, 3, 3), {}), ((32, 3, 3, 3), (32, 1, 3, 3), {}), ((48, 1, 3, 3), (16, 48, 1, 1), {}),
         ((96, 16, 1, 1), (96, 1, 3, 3), {}), ((64, 32, 1, 1), (10, 64), {}), ((32, 8, 3, 3), (24, 16, 3, 3), {}),
         ((32, 16, 3, 3), (24, 32, 3, 3), dict(s_range=(0.5, 2.0))), ((32, 16, 3, 3), (24, 32, 3, 3), dict(s_range=(1 / 3.0, 3.0))),
         ((32, 16, 3, 3), (24, 32, 3, 3), dict(eps=1e-3)), ((32, 16, 3, 3), (24, 32, 3, 3), dict(degenerate=True))]
EQ_NAMES = ("w1", "w2", "b1", "bw", "bb", "S")


def equalization_case(s1, s2, opt, signed):
    """Seeded inputs of one _layer_equalization case: ([w1, w2, b1, bw, bb] as torch tensors, keyword options)."""
    import torch
    torch.manual_seed(hash((s1, s2, signed)) % 1000)
    opt = dict(opt)
    degenerate = opt.pop("degenerate", False)
    w1 = torch.randn(*s1) * (10 ** torch.empty(s1[0]).uniform_(-1, 1)).view(-1, *([1] * (len(s1) - 1)))
    w2 = torch.randn(*s2)
    if degenerate:
        w1[1] = 0; w1[3] = 0.5
        w2.view(s2[0], s2[1], -1)[:, 2] = 0
    b1, bw, bb = torch.randn(s1[0]), torch.rand(s1[0]) + 0.5, torch.randn(s1[0])
    return [w1, w2, b1, bw, bb], opt


def equalization_digest(a):
    """sha256 of the float32 bits, every NaN canonical (the pins compare with equal_nan)."""
    import hashlib
    a = np.array(a, dtype=np.float32)
    a[np.isnan(a)] = np.nan
    return hashlib.sha256(a.tobytes()).hexdigest()


@pytest.fixture(scope="module")
def eq_gold():
    return np.load(os.path.join(GOLD, "ref_equalization_exact.npz"))


@pytest.mark.parametrize("s1,s2,opt", CASES)
@pytest.mark.parametrize("signed", [False, True])
def test_live_layer_equalization_bit_exact_with_reference_sqrt(eq_gold, s1, s2, opt, signed):
    """The reference's _layer_equalization outputs (weights as digests, vectors in full) vs the oracle given the same
    torch.sqrt: equal bit for bit."""
    ts, kw = equalization_case(s1, s2, opt, signed)
    n = [t.numpy() for t in ts]
    S = O.layer_equalization(*n, signed=signed, sqrt_fn=_torch_sqrt, **kw)
    key = "c%d_s%d_" % (CASES.index((s1, s2, opt)), signed)
    for name, got in zip(EQ_NAMES, n + [S]):
        if name in ("w1", "w2"):
            assert equalization_digest(got) == str(eq_gold[key + name]), name
        else:
            assert np.array_equal(got, eq_gold[key + name], equal_nan=True), name


def test_live_golden_ncnn_table(ref):
    """The reference's only checked-in numeric output: modeling/ncnn/model_quant_relu_equal.table rows 1-53 =
    128 / max|W| per layer after BN fold + ReLU6->ReLU + SIGNED equalization of the bundled MobileNetV2 checkpoint
    (convert_ncnn.py:109,178-201).  Reproduced here by the ORACLE (fold + sweeps) on the product's own graph walk."""
    import torch
    import torch.nn as nn
    from dfq_b200 import workload
    from dfq_b200.utils.relation import create_relation
    table = os.path.join(REF, "modeling", "ncnn", "model_quant_relu_equal.table")
    ckpt = os.path.join(REF, "modeling", "classification", "mobilenetv2_1.0-f2a8633.pth.tar")
    if not (os.path.isfile(table) and os.path.isfile(ckpt)):
        pytest.skip("table / checkpoint not present")
    rows = [l.split() for l in open(table).read().strip().splitlines()]
    golden = np.array([float(r[1]) for r in rows[:53]])
    topo = workload.load_topology(os.path.join(GOLD, "topology_mobilenetv2.json"))
    graph, bottoms, modules = workload.build_graph(topo, seed=0)
    # load the bundled weights into the topology-built modules, in trace order == state_dict order of the model file
    sd = torch.load(ckpt, map_location="cpu")
    tensors = [v for k, v in sd.items() if "num_batches_tracked" not in k]
    it = iter(tensors)
    with torch.no_grad():
        for m in modules:
            if isinstance(m, (nn.Conv2d, nn.Linear)):
                m.weight.copy_(next(it))
                if m.bias is not None:
                    m.bias.copy_(next(it))
            elif isinstance(m, nn.BatchNorm2d):
                m.weight.copy_(next(it)); m.bias.copy_(next(it)); m.running_mean.copy_(next(it)); m.running_var.copy_(next(it))
    targ = [nn.Conv2d, nn.Linear]
    keys = list(graph.keys())
    tl = [k for k in keys if type(graph[k]) in targ]
    idx = {k: i for i, k in enumerate(tl)}
    layers, bn_of = [], {}
    for k in tl:
        layers.append(O.OLayer(graph[k].weight.detach().numpy().copy(), None if graph[k].bias is None else graph[k].bias.detach().numpy().copy()))
    bns = []
    for k in keys:                     # BN fold (layer_transform.py:231-276) with the oracle
        if isinstance(graph[k], nn.BatchNorm2d) and bottoms[k] and type(graph[bottoms[k][0]]) in targ:
            bn, li = graph[k], idx[bottoms[k][0]]
            w, b, fw, fb = O.bn_fold(layers[li].w, layers[li].b, bn.weight.detach().numpy(), bn.bias.detach().numpy(),
                                     bn.running_mean.numpy(), bn.running_var.numpy(), bn.eps)
            layers[li].w, layers[li].b = w, b
            bn_of[k] = len(bns); bns.append((fw, fb))
    rels = [O.ORelation(idx[a], idx[b], bn_of[c]) for a, b, c in (r.get_idxs() for r in create_relation(graph, bottoms, targ))]
    assert len(rels) == 37
    n, _ = O.cross_layer_equalization(layers, bns, rels, signed=True)
    got = np.array([128.0 / np.abs(l.w).max() for l in layers])
    assert got.shape == golden.shape
    assert np.abs(got / golden - 1).max() < 2e-6, np.abs(got / golden - 1).max()
