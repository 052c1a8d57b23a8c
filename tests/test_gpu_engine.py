"""-m gpu parity tests of the arena engine (libdfq_sm100.so through dfq_b200.engine.Session) against
the numpy oracle on seeded inputs.  Equalization, BN fold factors and fake-quant are compared
bit-exactly; bias correction to 1e-5 normwise (fp32 mat-vec has no defined order in the reference)."""
import numpy as np
import pytest
import torch

from oracle import dfq_oracle as O

pytestmark = pytest.mark.gpu


def _mk(shape, seed, gain=True):
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(*shape, generator=g)
    if gain:
        w = w * (10 ** torch.empty(shape[0]).uniform_(-1, 1, generator=g)).view(-1, *([1] * (len(shape) - 1)))
    return w.contiguous()


def _normwise(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


PAIRS = [
    ((32, 16, 3, 3), (24, 32, 3, 3)),      # dense -> dense, short rows (warp path, kk=9 columns)
    ((32, 3, 3, 3), (32, 1, 3, 3)),        # dense(27, unaligned rows) -> depthwise  (G = 32)
    ((48, 1, 3, 3), (16, 48, 1, 1)),       # depthwise -> pointwise
    ((96, 16, 1, 1), (96, 1, 3, 3)),       # pointwise -> depthwise
    ((64, 32, 1, 1), (10, 64)),            # pointwise -> linear
    ((32, 8, 3, 3), (24, 16, 3, 3)),       # grouped second conv (G = 2)
    ((64, 128, 3, 3), (48, 64, 3, 3)),     # rows of 1152 floats: CTA-per-row path
    ((40, 512, 3, 3), (24, 40, 3, 3)),     # rows of 4608 floats
    ((8, 2500, 1, 1), (12, 8, 1, 1)),      # rows of 2500 floats (cta vec path, partial)
    ((6, 9001), (5, 6)),                   # row longer than the register tile: generic path, odd length
    ((7, 33, 1, 1), (9, 7, 1, 1)),         # scalar path, 33 elements
]


@pytest.mark.parametrize("s1,s2", PAIRS)
@pytest.mark.parametrize("signed", [False, True])
def test_single_relation_matches_oracle(s1, s2, signed):
    from dfq_b200.engine import Session
    w1, w2 = _mk(s1, 1), _mk(s2, 2, gain=False)
    C1 = s1[0]
    g = torch.Generator().manual_seed(3)
    b1 = torch.randn(C1, generator=g); bw = torch.rand(C1, generator=g) + 0.5; bb = torch.randn(C1, generator=g)
    n = [t.clone().numpy() for t in (w1, w2, b1, bw, bb)]
    S_ref = O.layer_equalization(*n, signed=signed)

    sess = Session()
    l1 = sess.add_layer(w1, b1); l2 = sess.add_layer(w2, None)
    obw, obb = sess.bind(bw), sess.bind(bb)
    sess.upload()
    res, s_offs = sess.run_cle([(l1, l2, obw, obb)], signed=signed, max_sweeps=1)
    S = sess.view(s_offs[0], C1).cpu().numpy()
    sess.download()
    assert res.n_sweeps == 1
    for name, got, ref in (("S", S, S_ref), ("w1", w1.numpy(), n[0]), ("w2", w2.numpy(), n[1]), ("b1", b1.numpy(), n[2]),
                           ("bn_w", bw.numpy(), n[3]), ("bn_b", bb.numpy(), n[4])):
        assert np.array_equal(got, ref), "%s differs: normwise %g" % (name, _normwise(got, ref))


def test_degenerate_channels_and_clamp():
    from dfq_b200.engine import Session
    for s_range in ((1e-8, 1e8), (0.5, 2.0), (1 / 3.0, 3.0)):
        w1, w2 = _mk((32, 16, 3, 3), 5), _mk((24, 32, 3, 3), 6, gain=False)
        w1[1] = 0; w1[3] = 0.5
        w2.view(24, 32, -1)[:, 2] = 0
        b1 = torch.randn(32)
        n = [w1.clone().numpy(), w2.clone().numpy(), b1.clone().numpy()]
        S_ref = O.layer_equalization(n[0], n[1], n[2], None, None, s_range=s_range)
        sess = Session()
        l1 = sess.add_layer(w1, b1); l2 = sess.add_layer(w2, None)
        sess.upload()
        res, s_offs = sess.run_cle([(l1, l2, -1, -1)], s_range=s_range, max_sweeps=1)
        S = sess.view(s_offs[0], 32).cpu().numpy()
        sess.download()
        assert np.array_equal(S, S_ref)
        assert np.array_equal(w1.numpy(), n[0], equal_nan=True)
        assert np.array_equal(w2.numpy(), n[1], equal_nan=True)
        assert np.array_equal(b1.numpy(), n[2])


def _chain_case(shapes, seed):
    ws = [_mk(s, seed + i, gain=(i % 2 == 0)) for i, s in enumerate(shapes)]
    g = torch.Generator().manual_seed(seed + 100)
    bs = [torch.randn(s[0], generator=g) for s in shapes]
    bns = [(torch.rand(s[0], generator=g) + 0.5, torch.randn(s[0], generator=g)) for s in shapes[:-1]]
    return ws, bs, bns


CHAINS = [
    [(32, 3, 3, 3), (32, 1, 3, 3), (16, 32, 1, 1), (96, 16, 1, 1), (96, 1, 3, 3), (24, 96, 1, 1)],   # MobileNetV2 chain 1
    [(144, 24, 1, 1), (144, 1, 3, 3), (32, 144, 1, 1)],                                               # inverted residual
    [(64, 32, 3, 3), (64, 64, 3, 3), (48, 64, 3, 3), (10, 48)],                                       # dense chain: re-scanned middles
    [(16, 8, 3, 3), (32, 8, 3, 3), (32, 1, 3, 3), (20, 32, 1, 1)],                                    # grouped (G=2) then depthwise
    [(1040, 32, 1, 1), (96, 1040, 1, 1), (24, 96, 1, 1)],            # 1040-wide middle: scan and re-scan above 1024 columns
]


@pytest.mark.parametrize("shapes", CHAINS)
@pytest.mark.parametrize("signed", [False, True])
def test_chain_to_convergence_matches_oracle(shapes, signed):
    """Several chains at once, run to the reference's exit rule: sweep count, every weight, bias, BN
    vector and accumulated S must equal the oracle bit for bit."""
    from dfq_b200.engine import Session
    ws, bs, bns = _chain_case(shapes, 11)
    # a second, independent chain (isolated pair) shares the sweep loop, as in a real model
    xw = [_mk((48, 24, 3, 3), 77), _mk((40, 48, 3, 3), 78, gain=False)]
    xb = [torch.randn(48), torch.randn(40)]
    xbn = (torch.rand(48) + 0.5, torch.randn(48))

    layers = [O.OLayer(w.clone().numpy(), b.clone().numpy()) for w, b in zip(ws + xw, bs + xb)]
    obns = [(a.clone().numpy(), b.clone().numpy()) for a, b in bns + [xbn]]
    nl = len(ws)
    rels = [O.ORelation(i, i + 1, i) for i in range(nl - 1)] + [O.ORelation(nl, nl + 1, nl - 1)]
    n_ref, diffs_ref = O.cross_layer_equalization(layers, obns, rels, signed=signed)

    sess = Session()
    ids = [sess.add_layer(w, b) for w, b in zip(ws + xw, bs + xb)]
    bn_offs = [(sess.bind(a), sess.bind(b)) for a, b in bns + [xbn]]
    sess.upload()
    rl = [(ids[i], ids[i + 1], bn_offs[i][0], bn_offs[i][1]) for i in range(nl - 1)]
    rl.append((ids[nl], ids[nl + 1], bn_offs[nl - 1][0], bn_offs[nl - 1][1]))
    res, s_offs = sess.run_cle(rl, signed=signed)
    S = [sess.view(o, sess.layer(r[0])["rows"]).cpu().numpy() for o, r in zip(s_offs, rl)]
    sess.download()

    assert res.n_sweeps == n_ref, (res.n_sweeps, n_ref, res.diffs[:5], diffs_ref[:5])
    assert res.converged
    np.testing.assert_allclose(res.diffs[:len(diffs_ref)][:64], diffs_ref[:64], rtol=1e-6, atol=1e-12)
    for i, (w, b) in enumerate(zip(ws + xw, bs + xb)):
        assert np.array_equal(w.numpy(), layers[i].w), "weight %d normwise %g" % (i, _normwise(w.numpy(), layers[i].w))
        assert np.array_equal(b.numpy(), layers[i].b), "bias %d" % i
    for i, (a, b) in enumerate(bns + [xbn]):
        assert np.array_equal(a.numpy(), obns[i][0]) and np.array_equal(b.numpy(), obns[i][1])
    for i, r in enumerate(rels):
        assert np.array_equal(S[i], r.S), "S of relation %d" % i


def test_bn_fold_matches_oracle():
    from dfq_b200.engine import Session
    sess = Session()
    cases = []
    for i, shape in enumerate([(32, 16, 3, 3), (24, 1, 3, 3), (40, 512, 3, 3), (10, 64), (7, 33, 1, 1)]):
        g = torch.Generator().manual_seed(40 + i)
        w = torch.randn(*shape, generator=g); b = torch.randn(shape[0], generator=g) if i % 2 == 0 else None
        gamma = torch.randn(shape[0], generator=g); beta = torch.randn(shape[0], generator=g)
        mean = torch.randn(shape[0], generator=g); var = torch.rand(shape[0], generator=g) + 0.1
        ref = O.bn_fold(w.numpy().copy(), None if b is None else b.numpy().copy(), gamma.numpy(), beta.numpy(), mean.numpy(),
                        var.numpy(), 1e-5)
        li = sess.add_layer(w, b)
        offs = dict(layer=li, bn_eps=1e-5, gamma_off=sess.bind(gamma, False), beta_off=sess.bind(beta, False),
                    mean_off=sess.bind(mean, False), var_off=sess.bind(var, False),
                    fake_w_off=sess.alloc(shape[0]), fake_b_off=sess.alloc(shape[0]))
        cases.append((w, b, li, offs, ref))
    sess.upload()
    sess.run_bn_fold([c[3] for c in cases])
    out = [(sess.view(sess.layer(c[2])["bias_off"], c[0].shape[0]).cpu().numpy(),
            sess.view(c[3]["fake_w_off"], c[0].shape[0]).cpu().numpy(),
            sess.view(c[3]["fake_b_off"], c[0].shape[0]).cpu().numpy()) for c in cases]
    sess.download()
    for (w, b, li, offs, ref), (bias, fw, fb) in zip(cases, out):
        assert np.array_equal(w.numpy(), ref[0])
        assert np.array_equal(bias, ref[1])
        assert np.array_equal(fw, ref[2]) and np.array_equal(fb, ref[3])


@pytest.mark.parametrize("bits,sym", [(8, False), (8, True), (4, False), (16, False), (16, True)])
def test_quantize_tensors_bit_exact(bits, sym):
    from dfq_b200.engine import Session
    sess = Session()
    ts = [torch.randn(64, 32, 3, 3) * 3, torch.randn(1001), torch.randn(10, 1280) * 0.1, torch.full((17,), 0.25), torch.randn(3)]
    refs = [O.quantize(t.numpy(), bits, float(t.min()), float(t.max()), symmetric=sym) for t in ts]
    offs = [sess.bind(t) for t in ts]
    sess.upload()
    sess.run_quantize([(o, t.numel(), bits, sym) for o, t in zip(offs, ts)])
    sess.download()
    for t, r in zip(ts, refs):
        assert np.array_equal(t.numpy(), r.reshape(t.shape))


BC_VARIANTS = ["engine", "stream"]     # k_bc_engine (small, latency-bound models) / k_bc_stream (large phases)


def _force_bc_variant(monkeypatch, variant):
    monkeypatch.setenv("DFQ_BC_STREAM", "1" if variant == "stream" else "0")


@pytest.mark.parametrize("variant", BC_VARIANTS)
def test_bias_correct_chain_matches_oracle(variant, monkeypatch):
    _force_bc_variant(monkeypatch, variant)
    _bias_correct_chain()


def _bias_correct_chain():
    """conv1+BN1+ReLU -> conv2+BN2 -> conv3 (no ReLU between 2 and 3): two corrected layers in series; the second
    one reads the fake_bias the first one just updated."""
    from dfq_b200.engine import Session
    g = torch.Generator().manual_seed(9)
    w2 = torch.randn(48, 32, 3, 3, generator=g) * 0.1; b2 = torch.randn(48, generator=g)
    w3 = torch.randn(20, 48, 1, 1, generator=g) * 0.2
    bn1 = (torch.rand(32, generator=g) + 0.5, torch.randn(32, generator=g) * 0.3)
    bn2 = (torch.rand(48, generator=g) + 0.5, torch.randn(48, generator=g) * 0.3)
    # oracle
    e1 = O.relu_expectation(bn1[0].numpy(), bn1[1].numpy())
    d2 = O.bias_delta(w2.numpy(), e1)
    b2_ref = b2.numpy() + (-d2)
    fb2 = bn2[1].numpy() + (-d2)
    e2 = fb2                                  # no ReLU after BN2
    d3 = O.bias_delta(w3.numpy(), e2)
    b3_ref = np.zeros(20, np.float32) + (-d3)

    sess = Session()
    l2 = sess.add_layer(w2, b2); l3 = sess.add_layer(w3, None)
    o1 = (sess.bind(bn1[0]), sess.bind(bn1[1])); o2 = (sess.bind(bn2[0]), sess.bind(bn2[1]))
    sess.upload()
    items = [dict(layer=l2, signed=False, level=0, next_bn_b_off=o2[1],
                  terms=[dict(bn_w_off=o1[0], bn_b_off=o1[1], n=32, relu=True, op="set")]),
             dict(layer=l3, signed=False, level=1, next_bn_b_off=-1,
                  terms=[dict(bn_w_off=o2[0], bn_b_off=o2[1], n=48, relu=False, op="set")])]
    doffs = sess.run_bias_correct(items)
    d2_gpu = sess.view(doffs[0], 48).cpu().numpy(); d3_gpu = sess.view(doffs[1], 20).cpu().numpy()
    b3_gpu = sess.view(sess.layer(l3)["bias_off"], 20).cpu().numpy()
    sess.download()
    assert _normwise(d2_gpu, d2) < 1e-5 and _normwise(d3_gpu, d3) < 1e-5
    assert _normwise(b2.numpy(), b2_ref) < 1e-5
    assert _normwise(bn2[1].numpy(), fb2) < 1e-5
    assert _normwise(b3_gpu, b3_ref) < 1e-5


def test_convergence_groups_equal_one_call_per_model():
    """A batch of independent models in one launch (n_groups > 1): every group must stop on ITS exit rule, i.e. give
    exactly what a separate cross_layer_equalization call per model gives (here: the oracle, model by model)."""
    from dfq_b200.engine import Session
    models = [[(32, 16, 3, 3), (24, 32, 3, 3)],
              [(144, 24, 1, 1), (144, 1, 3, 3), (32, 144, 1, 1)],
              [(64, 32, 3, 3), (64, 64, 3, 3), (48, 64, 3, 3)],
              [(40, 512, 3, 3), (24, 40, 3, 3)]]
    sess = Session()
    rl, groups, refs, tensors = [], [], [], []
    for m, shapes in enumerate(models):
        ws, bs, bns = _chain_case(shapes, 200 + 10 * m)
        layers = [O.OLayer(w.clone().numpy(), b.clone().numpy()) for w, b in zip(ws, bs)]
        obns = [(a.clone().numpy(), b.clone().numpy()) for a, b in bns]
        rels = [O.ORelation(i, i + 1, i) for i in range(len(shapes) - 1)]
        n_ref, _ = O.cross_layer_equalization(layers, obns, rels)
        ids = [sess.add_layer(w, b) for w, b in zip(ws, bs)]
        offs = [(sess.bind(a), sess.bind(b)) for a, b in bns]
        for i in range(len(shapes) - 1):
            rl.append((ids[i], ids[i + 1], offs[i][0], offs[i][1])); groups.append(m)
        refs.append((n_ref, layers, obns, rels)); tensors.append((ws, bs, bns))
    sess.upload()
    plan = sess.plan_cle(rl, groups=groups)
    res = sess.run_cle_plan(plan)
    sess.download()
    assert list(res.group_sweeps) == [r[0] for r in refs], (list(res.group_sweeps), [r[0] for r in refs])
    assert res.n_sweeps == max(r[0] for r in refs) and res.converged
    for (n_ref, layers, obns, rels), (ws, bs, bns) in zip(refs, tensors):
        for w, b, l in zip(ws, bs, layers):
            assert np.array_equal(w.numpy(), l.w) and np.array_equal(b.numpy(), l.b)
        for (a, b), (oa, ob) in zip(bns, obns):
            assert np.array_equal(a.numpy(), oa) and np.array_equal(b.numpy(), ob)


def test_large_stack_properties():
    """Size-independent properties on a stack too large for the oracle to finish in seconds (BASELINE config 5 shapes):
    every block converges in 2 sweeps; equalization preserves the function of each pair up to rounding
    (W1[c]*W2[:,c] products are invariant: s * 1/s); re-running on the result is a fixed point in one more sweep."""
    from dfq_b200.engine import Session
    from dfq_b200.workload import DeviceStack
    sess = Session()
    st = DeviceStack(sess, 16, 512, 3, seed=5)
    st.generate()
    C, N = 512, st.N
    w1_before = sess.view(sess.layer(st.layers[0])["w_off"], N).clone().view(C, -1)
    w2_before = sess.view(sess.layer(st.layers[1])["w_off"], N).clone().view(C, C, 9)
    sess.run_bn_fold(st.fold_plan)
    f1 = sess.view(sess.layer(st.layers[0])["w_off"], N).clone().view(C, -1)
    f2 = sess.view(sess.layer(st.layers[1])["w_off"], N).clone().view(C, C, 9)
    res = sess.run_cle_plan(st.cle_plan)
    assert res.converged and set(int(x) for x in res.group_sweeps) == {2}, res.group_sweeps
    e1 = sess.view(sess.layer(st.layers[0])["w_off"], N).view(C, -1)
    e2 = sess.view(sess.layer(st.layers[1])["w_off"], N).view(C, C, 9)
    S = sess.view(st.cle_plan["s_offs"][0], C)
    # rows scaled by S, columns by 1/S (up to two roundings per sweep)
    assert torch.allclose(e1, f1 * S.view(-1, 1), rtol=1e-6, atol=0)
    assert torch.allclose(e2, f2 / S.view(1, -1, 1), rtol=1e-6, atol=0)
    # equalized: per-channel ranges of the pair agree
    r1 = e1.max(1)[0] - e1.min(1)[0]
    r2 = e2.amax((0, 2)) - e2.amin((0, 2))
    assert torch.allclose(r1, r2, rtol=1e-5)
    # idempotence: one more run changes (almost) nothing and stops after its first sweep
    before = sess.view(st.w_begin, 2 * N).clone()
    res2 = sess.run_cle_plan(st.cle_plan)
    assert int(res2.group_sweeps.max()) == 1
    assert torch.allclose(sess.view(st.w_begin, 2 * N), before, rtol=1e-6, atol=0)


@pytest.mark.parametrize("variant", ["engine", "stack"])
def test_config5_blocks_match_the_oracle(variant, monkeypatch):
    monkeypatch.setenv("DFQ_CLE_STACK", "1" if variant == "stack" else "0")
    _config5_blocks()


@pytest.mark.parametrize("channels,k", [(64, 3), (128, 1), (96, 3)])
def test_stack_kernel_equals_engine_on_other_block_shapes(channels, k, monkeypatch):
    """k_cle_stack (streaming variant for stacks of two-layer chains) against k_cle_engine on the same bits: several rows per
    tile (576- and 864-float rows), pointwise blocks (128-float rows, 32 rows per tile), 5 blocks = 5 convergence groups -
    weights, biases, BN vectors, S and the per-group sweep counts must be bit-identical."""
    from dfq_b200.engine import Session
    from dfq_b200.workload import DeviceStack
    outs = []
    for variant in ("0", "1"):
        monkeypatch.setenv("DFQ_CLE_STACK", variant)
        sess = Session()
        st = DeviceStack(sess, 5, channels, k, seed=11)
        st.generate()
        sess.run_bn_fold(st.fold_plan)
        res = sess.run_cle_plan(st.cle_plan, cols_ready=st.fold_plan["scanned"])
        outs.append((st.state().clone(), st.scale_state().clone(), res.group_sweeps.copy(), res.n_sweeps, res.converged))
    assert outs[0][3] == outs[1][3] and outs[0][4] and outs[1][4] and np.array_equal(outs[0][2], outs[1][2]), (outs[0][2], outs[1][2])
    assert torch.equal(outs[0][0], outs[1][0]), "weights / biases / BN vectors differ between the two kernels"
    assert torch.equal(outs[0][1], outs[1][1]), "S differs"


@pytest.mark.parametrize("n_blocks", [16, 40])
def test_mid_size_stacks_run_the_streaming_kernels_and_match_the_oracle(n_blocks):
    """Regression for the ring's phase hazard (bc_stream.cuh::bc_take): stacks of 16-96 blocks - large enough for the streaming
    kernels (k_cle_stack, k_bc_stream are chosen by the library, nothing is forced), small enough that every load starts cold -
    crashed with 'Warp Illegal Instruction' or hung before consumers waited for their item's sequence stamp.  Three full steps
    each, first and last block against the oracle."""
    from dfq_b200.engine import Session
    from dfq_b200.workload import DeviceStack
    from oracle import stack_check
    sess = Session()
    st = DeviceStack(sess, n_blocks, 512, 3, seed=1000 + n_blocks)
    st.generate()
    pristine = st.state().clone()
    for _ in range(3):
        st.state().copy_(pristine)
        res = st.run()
        torch.cuda.synchronize()
    assert res.converged and set(int(x) for x in res.group_sweeps) == {2}
    after = st.state()
    for b in (0, n_blocks - 1):
        r = stack_check.compare_block(st.block_arrays(pristine, b), st.block_arrays(after, b))
        assert r["weights_bit_exact"] and r["vectors_bit_exact"] and r["bias_normwise"] < 1e-5 and r["sweeps"] == 2, (b, r)


def _config5_blocks():
    """The headline workload shape itself (BASELINE configs[4]): Conv[512,512,3,3]+BN+ReLU -> Conv[512,512,3,3]+BN blocks
    through the fused step bench.py times (fold with column scan -> equalization -> correction with range hints) vs the
    oracle on the same bits: weights / first bias / BN vectors bit-exact, corrected bias within 1e-5, 2 sweeps."""
    from dfq_b200.engine import Session
    from dfq_b200.workload import DeviceStack
    from oracle import stack_check
    sess = Session()
    st = DeviceStack(sess, 3, 512, 3, seed=77)
    st.generate()
    pristine = st.state().clone()
    res = st.run()
    assert res.converged
    after = st.state()
    for b in (0, 2):
        r = stack_check.compare_block(st.block_arrays(pristine, b), st.block_arrays(after, b))
        assert r["weights_bit_exact"] and r["vectors_bit_exact"], (b, r)
        assert r["bias_normwise"] < 1e-5 and r["sweeps"] == int(res.group_sweeps[b]) == 2, (b, r, res.group_sweeps)


FUSED_CHAINS = CHAINS + [
    [(24, 16, 3, 3), (12, 24, 32, 32)],        # second layer with rows longer than a stage (9216 floats): direct path
    [(33, 7, 3, 3), (21, 33, 3, 3)],           # unaligned tiles (297-float rows at odd offsets): cooperative path
]


@pytest.mark.parametrize("shapes", FUSED_CHAINS)
def test_fused_fold_scan_and_range_hints_equal_the_unfused_calls(shapes):
    """fold -> equalize -> correct with the two shortcuts of the fused plan (the fold pre-scans the column extrema the
    equalization starts from; the correction takes per-tensor ranges from the column extrema the equalization leaves) must
    give bit-identical results to the three plain calls, and the fold's column extrema must be the true ones."""
    from dfq_b200.engine import Session

    def build():
        sess = Session()
        ws, bs, _ = _chain_case(shapes, 23)
        g = torch.Generator().manual_seed(5)
        ids, vecs = [], []
        for w, b in zip(ws, bs):
            ids.append(sess.add_layer(w, b))
            n = w.shape[0]
            v = dict(gamma=sess.bind(torch.rand(n, generator=g) + 0.5, False), beta=sess.bind(torch.randn(n, generator=g) * 0.2, False),
                     mean=sess.bind(torch.randn(n, generator=g) * 0.1, False), var=sess.bind(torch.rand(n, generator=g) + 0.5, False),
                     fake_w=sess.alloc(n), fake_b=sess.alloc(n))
            vecs.append(v)
        folds = [dict(layer=li, bn_eps=1e-5, gamma_off=v["gamma"], beta_off=v["beta"], mean_off=v["mean"], var_off=v["var"],
                      fake_w_off=v["fake_w"], fake_b_off=v["fake_b"]) for li, v in zip(ids, vecs)]
        rels = [(ids[i], ids[i + 1], vecs[i]["fake_w"], vecs[i]["fake_b"]) for i in range(len(ids) - 1)]
        items = [dict(layer=ids[i], signed=False, level=i, next_bn_b_off=vecs[i]["fake_b"],
                      terms=[dict(bn_w_off=vecs[i - 1]["fake_w"], bn_b_off=vecs[i - 1]["fake_b"], n=ws[i - 1].shape[0], relu=True, op="set")])
                 for i in range(1, len(ids))]
        return sess, ws, bs, ids, vecs, folds, rels, items

    # plain
    sa, wa, ba, ida, va, folds, rels, items = build()
    cle_a = sa.plan_cle(rels); bc_a = sa.plan_bias_correct(items); fold_a = sa.plan_bn_fold(folds)
    sa.upload()
    sa.run_bn_fold(fold_a)
    res_a = sa.run_cle_plan(cle_a)
    sa.run_bias_correct_plan(bc_a, 8)
    fb_a = [sa.view(v["fake_b"], w.shape[0]).cpu().numpy() for v, w in zip(va, wa)]
    sa.download()
    # fused
    sb, wb, bb, idb, vb, folds, rels, items = build()
    cle_b = sb.plan_cle(rels); bc_b = sb.plan_bias_correct(items); fold_b = sb.plan_bn_fold(folds, cle_plan=cle_b)
    assert sorted(fold_b["scanned"]) == sorted(idb[1:])
    sb.upload()
    sb.run_bn_fold(fold_b)
    for i in range(1, len(idb)):               # buffer 0 of every `second` layer = true column extrema of the folded weights
        l = cle_b["lt"][idb[i]]; r = cle_b["rt"][int(l["rel_in"])]
        n = int(l["rows"]) * int(l["cols"]) * int(l["kk"])
        w = sb.view(int(l["w_off"]), n).cpu().numpy().reshape(int(r["groups"]), int(r["go"]), int(r["gi"]), -1)
        Cn = int(r["channels"])
        assert np.array_equal(sb.view(int(l["cmin_off"]), Cn).cpu().numpy(), w.min(axis=(1, 3)).reshape(-1))
        assert np.array_equal(sb.view(int(l["cmax_off"]), Cn).cpu().numpy(), w.max(axis=(1, 3)).reshape(-1))
    res_b = sb.run_cle_plan(cle_b, cols_ready=fold_b["scanned"])
    hints = sb.cle_col_hints(cle_b, res_b)
    assert sorted(hints["layer"].tolist()) == sorted(idb[1:])
    for li, mn_off, mx_off, Cn in zip(*(hints[k].tolist() for k in ("layer", "colmin_off", "colmax_off", "n_col"))):
        # what the equalization left = true column extrema of the final weights
        l = cle_b["lt"][li]; r = cle_b["rt"][int(l["rel_in"])]
        n = int(l["rows"]) * int(l["cols"]) * int(l["kk"])
        w = sb.view(int(l["w_off"]), n).cpu().numpy().reshape(int(r["groups"]), int(r["go"]), int(r["gi"]), -1)
        assert np.array_equal(sb.view(mn_off, Cn).cpu().numpy(), w.min(axis=(1, 3)).reshape(-1))
        assert np.array_equal(sb.view(mx_off, Cn).cpu().numpy(), w.max(axis=(1, 3)).reshape(-1))
    sb.run_bias_correct_plan(bc_b, 8, col_hints=hints)
    fb_b = [sb.view(v["fake_b"], w.shape[0]).cpu().numpy() for v, w in zip(vb, wb)]
    sb.download()
    assert res_a.n_sweeps == res_b.n_sweeps
    for x, y in zip(wa + ba, wb + bb):
        assert np.array_equal(x.numpy(), y.numpy())
    for x, y in zip(fb_a, fb_b):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("variant", BC_VARIANTS)
def test_bias_correction_codes_at_rounding_boundaries_are_the_references(variant, monkeypatch):
    _force_bc_variant(monkeypatch, variant)
    _codes_at_rounding_boundaries()


def _codes_at_rounding_boundaries():
    """Weights placed ON and within a few ulps of every rounding boundary of the 8-bit grid must give the reference's codes
    (true IEEE division, clamp, round-half-even - quantize.py:70-74): with E[x] = 1 the row's delta is sum(eps) in fp64, so a
    single wrong code shows as an error of one quantization step."""
    from dfq_b200.engine import Session
    rng = np.random.default_rng(7)
    lo, hi = np.float32(-1.3717), np.float32(2.0461)
    scale = (float(hi) - float(lo)) / 255.0
    vals = []
    for k in range(255):
        b = np.float32(float(lo) + (k + 0.5) * scale)          # t/scale ~ k + 0.5
        for d in range(-4, 5):
            v = b
            for _ in range(abs(d)):
                v = np.nextafter(v, np.float32(np.inf if d > 0 else -np.inf), dtype=np.float32)
            vals.append(v)
    vals = np.array(vals, np.float32)
    cols = 768
    rows = 3 * ((vals.size + cols - 1) // cols)
    w = rng.uniform(float(lo), float(hi), size=(rows, cols)).astype(np.float32)
    w.reshape(-1)[:vals.size] = vals
    w.reshape(-1)[vals.size] = lo; w.reshape(-1)[vals.size + 1] = hi      # pin the tensor's range
    wt = torch.from_numpy(w.reshape(rows, cols, 1, 1).copy())
    ones = torch.ones(cols); zeros_w = torch.ones(cols)
    d_ref = O.bias_delta(w.reshape(rows, cols, 1, 1), np.ones(cols, np.float32))
    sess = Session()
    li = sess.add_layer(wt, None)
    ow, ob = sess.bind(zeros_w), sess.bind(ones)
    sess.upload()
    doffs = sess.run_bias_correct([dict(layer=li, signed=False, level=0, next_bn_b_off=-1,
                                        terms=[dict(bn_w_off=ow, bn_b_off=ob, n=cols, relu=False, op="set")])])
    d_gpu = sess.view(doffs[0], rows).cpu().numpy()
    step = np.float32(scale)
    assert np.abs(d_gpu.astype(np.float64) - d_ref.astype(np.float64)).max() < 1e-3 * step, \
        "a code differs from the reference's (error in quantization steps: %g)" % (np.abs(d_gpu - d_ref).max() / step)


@pytest.mark.parametrize("variant", BC_VARIANTS)
def test_bias_correct_variants_on_mixed_layer_kinds(variant, monkeypatch):
    """Both bias-correction kernels on every tile kind of the row pipe in one call: 3x3 dense rows (several rows per tile),
    depthwise (cols = 1, groups = C: one expectation value per row), pointwise with more than 512 columns (expectation
    read from global memory), the 27-float rows of a first conv (tiles the TMA unit cannot move), rows longer than a
    stage (processed in global memory), a 'cat' of two BNs and an 'add' of two BNs, signed and unsigned, the raw-sum
    (bias absorption) flags, and 2049- / 4096-column layers (more expectation values than k_bc_engine caches in shared
    memory) - against the oracle, 1e-5 normwise."""
    from dfq_b200.engine import Session
    _force_bc_variant(monkeypatch, variant)
    g = torch.Generator().manual_seed(31)
    R = lambda *s: torch.randn(*s, generator=g)
    bnA = (torch.rand(64, generator=g) + 0.4, R(64) * 0.5)       # feeds 64-channel inputs
    bnB = (torch.rand(40, generator=g) + 0.4, R(40) * 0.5)
    bnC = (torch.rand(24, generator=g) + 0.4, R(24) * 0.5)
    bnD = (torch.rand(3, generator=g) + 0.4, R(3) * 0.5)
    bnE = (torch.rand(640, generator=g) + 0.4, R(640) * 0.5)
    bnF = (torch.rand(1200, generator=g) + 0.4, R(1200) * 0.5)
    cases = [  # (weight, signed, terms, flags)
        (R(48, 64, 3, 3) * 0.1, False, [("A", True, "set")], {}),
        (R(64, 1, 3, 3) * 0.3, False, [("A", True, "set")], {}),                          # depthwise
        (R(36, 640, 1, 1) * 0.05, True, [("E", False, "set")], {}),                        # 640 columns: no register cache
        (R(16, 3, 3, 3) * 0.4, False, [("D", False, "set")], {}),                          # 27-float rows
        (R(6, 1200, 2, 2) * 0.02, False, [("F", True, "set")], {}),                        # 4800-float rows: direct
        (R(20, 64, 1, 1) * 0.2, False, [("B", True, "set"), ("C", False, "cat")], {}),     # cat: 40 + 24
        (R(20, 64, 1, 1) * 0.2, True, [("A", True, "set"), ("A", False, "add")], {}),      # add
        (R(12, 32, 3, 3) * 0.1, False, [("A", True, "set")], {}),                          # grouped: 2 groups x 32 columns
        (R(30, 64, 3, 3) * 0.1, False, [("A", False, "set")], dict(raw_sum=True, add=True)),
    ]
    # wider than the 2048-value expectation cache of k_bc_engine: E[x] read from global memory, the level is not local
    bnG = (torch.rand(4096, generator=g) + 0.4, R(4096) * 0.5)
    bnH = (torch.rand(2049, generator=g) + 0.4, R(2049) * 0.5)
    cases += [
        (R(10, 4096) * 0.02, False, [("G", True, "set")], {}),                             # linear, 4096 columns
        (R(8, 2049, 1, 1) * 0.03, True, [("H", False, "set")], {}),                        # 1x1, 2049 columns
    ]
    bns = dict(A=bnA, B=bnB, C=bnC, D=bnD, E=bnE, F=bnF, G=bnG, H=bnH)
    sess = Session()
    off = {k: (sess.bind(v[0], False), sess.bind(v[1], False)) for k, v in bns.items()}
    items, biases, lids = [], [], []
    for w, signed, terms, flags in cases:
        b = R(w.shape[0])
        biases.append(b.clone())
        li = sess.add_layer(w, b)
        lids.append(li)
        items.append(dict(layer=li, signed=signed, level=0, next_bn_b_off=-1,
                          terms=[dict(bn_w_off=off[k][0], bn_b_off=off[k][1], n=bns[k][0].numel(), relu=relu, op=op) for k, relu, op in terms],
                          **flags))
    sess.upload()
    doffs = sess.run_bias_correct(items)
    for (w, signed, terms, flags), b0, li, doff in zip(cases, biases, lids, doffs):
        ex = None
        for k, relu, op in terms:
            v = O.relu_expectation(bns[k][0].numpy(), bns[k][1].numpy()) if relu else bns[k][1].numpy().copy()
            ex = v if ex is None else (np.concatenate([ex, v]) if op == "cat" else ex + v)
        if flags.get("raw_sum"):
            d = O.bias_absorb_wc(w.numpy(), ex, ex.shape[0])
            want = b0.numpy() + d
        else:
            d = O.bias_delta(w.numpy(), ex, signed=signed)
            want = b0.numpy() + (-d)
        got_d = sess.view(doff, w.shape[0]).cpu().numpy()
        got_b = sess.view(sess.layer(li)["bias_off"], w.shape[0]).cpu().numpy()
        assert _normwise(got_d, d) < 1e-5, (tuple(w.shape), signed, terms, _normwise(got_d, d))
        assert _normwise(got_b, want) < 1e-5, (tuple(w.shape), "bias")


def test_bc_fast_quotient_equals_ieee_division():
    """dfq_selftest_bc_arithmetic: the XU-free arithmetic of k_bc_stream (Markstein-corrected reciprocal product instead of
    div.rn, magic-number rint) must give Q(w) - w bit-identical to the IEEE chain of quantize.py:70-74 whenever its
    per-tensor guard says so - over thousands of (min, max) pairs x numerators that sit ON and within 4 ulps of every
    half-integer quotient plus dense random ones; and the guard must refuse scales with an all-ones mantissa."""
    import ctypes as C
    from dfq_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(5)
    n_ok = n_refused = 0
    bad = []
    for trial in range(1500):
        signed = trial % 5 == 4
        bits = 8 if trial % 7 else (4, 16)[trial % 2]
        mag = 10.0 ** rng.uniform(-6, 4) if trial % 101 else 1e-31      # tiny ranges: outside the exponent window -> refused
        lo = np.float32(-mag * rng.uniform(0.1, 1.0)) if trial % 3 else np.float32(mag * rng.uniform(0.0, 0.5))
        hi = np.float32(float(lo) + mag * rng.uniform(0.2, 2.0))
        if trial % 97 == 0:      # force an all-ones mantissa scale: (hi - lo) / 255 == 0x..7fffff
            s = np.uint32((np.float32(mag).view(np.uint32) & np.uint32(0xff800000)) | np.uint32(0x7fffff)).view(np.float32)
            lo = np.float32(0.0); hi = np.float32(float(s) * 255.0)
        qmax = (2 ** (bits - 1) - 1) if signed else (2 ** bits - 1)
        scale = (max(abs(float(hi)), abs(float(lo))) / qmax) if signed else (float(hi) - float(lo)) / qmax
        mn = 0.0 if signed else float(lo)
        ks = np.arange(-(2 ** (bits - 1)) - 1 if signed else -1, qmax + 2, max(1, (qmax + 3) // 300))
        vals = []
        for k in ks:
            b = np.float32(mn + (k + 0.5) * scale)
            v_up = v_dn = b
            vals.append(b)
            for _ in range(4):
                v_up = np.nextafter(v_up, np.float32(np.inf), dtype=np.float32); v_dn = np.nextafter(v_dn, np.float32(-np.inf), dtype=np.float32)
                vals.append(v_up); vals.append(v_dn)
        vals = np.concatenate([np.array(vals, np.float32), rng.uniform(float(lo), float(hi), 4096).astype(np.float32),
                               np.array([lo, hi, 0.0, np.nextafter(lo, np.float32(np.inf), dtype=np.float32)], np.float32)])
        vals = np.clip(vals, lo, hi)
        w = torch.from_numpy(vals).cuda()
        mm = torch.tensor([float(lo), float(hi)], dtype=torch.float32, device="cuda")
        ef = torch.empty_like(w); ed = torch.empty_like(w); ok = torch.zeros(1, dtype=torch.int32, device="cuda")
        P = lambda t: C.c_void_p(t.data_ptr())
        _lib.check(lib.dfq_selftest_bc_arithmetic(P(w), P(ef), P(ed), w.numel(), P(mm), bits, 1 if signed else 0, P(ok), _lib.stream_ptr()),
                   "dfq_selftest_bc_arithmetic")
        ref = O.quantize(vals, bits, float(lo), float(hi), signed) - vals
        assert np.array_equal(ed.cpu().numpy(), ref), "IEEE chain differs from the oracle"
        if int(ok.item()):
            n_ok += 1
            if not torch.equal(ef, ed):
                bad.append((trial, float(lo), float(hi), bits, signed, int((ef != ed).sum())))
        else:
            n_refused += 1
    assert not bad, bad[:5]
    assert n_ok > 1300 and n_refused >= 10, (n_ok, n_refused)      # 15 tiny-range trials + the all-ones mantissas that survive rounding


def test_invalid_descriptors_are_rejected_with_a_message_not_a_crash():
    """Error behaviour at the C boundary: inconsistent tables return DFQ_E_ARG and set dfq_last_error (surfaced as DfqError)
    before anything is launched; the arena is untouched and the session stays usable."""
    from dfq_b200._lib import DfqError
    from dfq_b200.engine import Session
    sess = Session()
    w1 = torch.randn(8, 4, 3, 3); w2 = torch.randn(6, 8, 3, 3)
    l1 = sess.add_layer(w1, None); l2 = sess.add_layer(w2, None)
    sess.upload()
    plan = sess.plan_cle([(l1, l2, -1, -1)])
    before = sess.view(0, sess.arena.numel()).clone()
    bad = dict(plan); bad["rt"] = plan["rt"].copy(); bad["rt"]["channels"] = 7               # != rows(first)
    with pytest.raises(DfqError, match="channels"):
        sess.run_cle_plan(bad)
    bad = dict(plan); bad["lt"] = plan["lt"].copy(); bad["lt"]["w_off"][l2] = sess.arena.numel()   # weight outside the arena
    with pytest.raises(DfqError, match="arena"):
        sess.run_cle_plan(bad)
    bad = dict(plan); bad["step_layers"] = plan["step_layers"].copy(); bad["step_layers"][0] = 99
    with pytest.raises(DfqError, match="layer index"):
        sess.run_cle_plan(bad)
    n = w1.numel() + w2.numel()
    assert torch.equal(sess.view(0, sess.arena.numel())[:n], before[:n]), "weights touched by a rejected call"
    res = sess.run_cle_plan(plan)                                                          # still usable
    assert res.n_sweeps >= 1
