"""The op-patching layer (SURVEY a14; layer_transform.py:16-228): replace_op / restore_op, the patched
Tensor.__add__ / add / __iadd__, torch.cat, torch.mean, F.interpolate, F.softmax and CustomTensorOP's cursor protocol.

The rewrite finds the calling frame with sys._getframe(2) where the reference walks inspect.stack(); these tests pin that
the two agree: on a model whose `forward` uses every patched op, the product's patched run (i) calls the functional-op
observers in the recorded order, each exactly once, with exactly the tensors the ops received, (ii) leaves calls from
functions not named `forward`, calls on other lines and Tensor.add (one frame deeper, never matched - as in the
reference) alone, (iii) equals the same forward run under the REFERENCE's own replace_op (its outputs stored in
tests/golden/ref_op_patching.npz by tools/make_golden.py), (iv) restores the original attributes.  CPU: oracle-backed
executor; -m gpu: the real library on CUDA tensors.
"""
import os

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import fakelib


def helper_outside_forward(a, b):
    return a + b, torch.cat([a, b], 1)


class Net(nn.Module):
    def __init__(self):
        super().__init__()
        self.c1 = nn.Conv2d(3, 4, 3, padding=1)
        self.c2 = nn.Conv2d(3, 4, 3, padding=1)

    def forward(self, x):
        a = self.c1(x)
        b = self.c2(x)
        y = a + b
        z = torch.cat([y, a, b], 1)
        u = F.interpolate(z, scale_factor=2, mode='bilinear', align_corners=True)
        v = torch.mean(u, (2, 3))
        p = F.softmax(v, 1)
        t = a.add(b)
        s, c = helper_outside_forward(a, b)
        q = a + b
        y += q
        return p, y, t, s, c


_L0 = Net.forward.__code__.co_firstlineno
RECORD = [("add_1", "add_%d_2" % (_L0 + 3)), ("torch.cat_2", "torch_cat_%d_3" % (_L0 + 4)),
          ("F.interpolate_3", "F_interpolate_%d_1" % (_L0 + 5)), ("torch.mean_4", "torch_mean_%d_1" % (_L0 + 6)),
          ("F.softmax_5", "F_softmax_%d_1" % (_L0 + 7)), ("iadd_6", "iadd_%d_2" % (_L0 + 11))]
N_OBS = 2 + 3 + 1 + 1 + 1 + 2
# the observers hold fp32 buffers and quantize with float(buffer) (quantize.py:119): use fp32-representable bounds
RANGES = [(float(np.float32(-1.5 - 0.1 * i)), float(np.float32(1.7 + 0.2 * i))) for i in range(N_OBS)]


def _run_patched(LT, QuantMeasure, model, x):
    obs = [QuantMeasure(num_bits=8, momentum=0.1) for _ in range(N_OBS)]
    seen = []
    for i, (q, (lo, hi)) in enumerate(zip(obs, RANGES)):
        q.running_min.fill_(lo); q.running_max.fill_(hi)
        q.to(x.device).eval()      # in the scripts the observers are submodules of the model and follow model.eval()
        q.register_forward_pre_hook(lambda m, args, i=i: seen.append((i, args[0].detach().cpu().clone())))
    LT.module_tensor_op = LT.CustomTensorOP(obs, [tuple(r) for r in RECORD])
    originals = (torch.Tensor.__add__, torch.Tensor.add, torch.Tensor.__iadd__, torch.cat, torch.mean, F.interpolate, F.softmax)
    LT.replace_op()
    try:
        assert torch.Tensor.__add__ is not originals[0] and torch.cat is not originals[3] and F.interpolate is not originals[5]
        with torch.no_grad():
            out = model(x)
    finally:
        LT.restore_op()
    now = (torch.Tensor.__add__, torch.Tensor.add, torch.Tensor.__iadd__, torch.cat, torch.mean, F.interpolate, F.softmax)
    assert all(a is b for a, b in zip(now, originals)), "restore_op must put every original attribute back"
    return [o.detach().cpu() for o in out], seen, LT.module_tensor_op


def _expected(model, x, q):
    """The same forward written out by hand: q(i, t) = observer i's fake-quantization."""
    with torch.no_grad():
        a = model.c1(x); b = model.c2(x)
        y = q(0, a) + q(1, b)
        z = torch.cat([q(2, y), q(3, a), q(4, b)], 1)
        u = F.interpolate(q(5, z), scale_factor=2, mode='bilinear', align_corners=True)
        v = torch.mean(q(6, u), (2, 3))
        p = F.softmax(q(7, v), 1)
        t = a.add(b)
        s, c = a + b, torch.cat([a, b], 1)
        qq = a + b                                   # recorded name is the iadd of the NEXT line: no match here
        y = q(8, y) + q(9, qq)                       # quirk Q5: the in-place add runs as an out-of-place __add__
    return [p, y, t, s, c]


def _check(device, monkeypatch, use_fake):
    if use_fake:
        fakelib.install(monkeypatch)
    from dfq_b200.utils import layer_transform as LT
    from dfq_b200.utils.quantize import QuantMeasure, quantize
    torch.manual_seed(0)
    model = Net().eval().to(device)
    x = torch.randn(2, 3, 6, 6).to(device)
    out, seen, cursor = _run_patched(LT, QuantMeasure, model, x)
    assert [i for i, _ in seen] == list(range(N_OBS)), "observers must fire once each, in the recorded order"
    assert cursor.idx_tensor_op == 0 and cursor.idx_name_tensor_op == 0, "both cursors wrap around after one forward"
    want = _expected(model, x, lambda i, t: quantize(t, 8, RANGES[i][0], RANGES[i][1]))
    for k, (g, w) in enumerate(zip(out, want)):
        assert torch.equal(g, w.cpu()), ("output", k, (g - w.cpu()).abs().max())
    # what each observer received is the op's own operand
    with torch.no_grad():
        a = model.c1(x).cpu(); b = model.c2(x).cpu()
    assert torch.equal(seen[0][1], a) and torch.equal(seen[1][1], b) and torch.equal(seen[3][1], a) and torch.equal(seen[4][1], b)
    return model, x, out


def test_patched_ops_quantize_exactly_the_recorded_calls(monkeypatch):
    _check("cpu", monkeypatch, use_fake=True)


@pytest.mark.gpu
def test_patched_ops_quantize_exactly_the_recorded_calls_gpu(monkeypatch):
    _check("cuda", monkeypatch, use_fake=False)


def reference_run(LT, QuantMeasure):
    """The forward of _check() under an implementation's replace_op: (outputs, observer order)."""
    torch.manual_seed(0)
    model = Net().eval()
    x = torch.randn(2, 3, 6, 6)
    out, seen, _ = _run_patched(LT, QuantMeasure, model, x)
    return out, [i for i, _ in seen]


def test_patched_ops_agree_with_the_reference_implementation(monkeypatch):
    """Same Net (same source lines), same record and ranges: the product's sys._getframe lookup and the reference's
    inspect.stack() lookup must quantize the same calls - outputs equal bit for bit (CPU, true division) to what the
    reference's replace_op produced (reference_run)."""
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_op_patching.npz"))
    model, x, ours = _check("cpu", monkeypatch, use_fake=True)
    assert list(gold["observer_order"]) == list(range(N_OBS))
    assert len(ours) == int(gold["n_outputs"])
    for k, g in enumerate(ours):
        w = torch.from_numpy(gold["output_%d" % k])
        assert torch.equal(g, w), ("output", k, (g - w).abs().max())


def test_no_patching_without_a_cursor_and_on_unrecorded_lines(monkeypatch):
    fakelib.install(monkeypatch)
    from dfq_b200.utils import layer_transform as LT
    from dfq_b200.utils.quantize import QuantMeasure
    torch.manual_seed(1)
    model = Net().eval()
    x = torch.randn(1, 3, 5, 5)
    with torch.no_grad():
        plain = model(x)
    # a record whose line numbers match nothing: every op falls through to the raw implementation
    obs = [QuantMeasure(num_bits=8).eval() for _ in range(2)]
    fired = []
    for q in obs:
        q.register_forward_pre_hook(lambda m, a: fired.append(1))
    LT.module_tensor_op = LT.CustomTensorOP(obs, [("add_1", "add_1_2")])
    LT.replace_op()
    try:
        with torch.no_grad():
            out = model(x)
    finally:
        LT.restore_op()
    assert not fired
    for a, b in zip(out, plain):
        assert torch.equal(a, b)
    assert np.isfinite(out[0].numpy()).all()
