"""-m gpu: min/max reductions on inputs with negative zeros, and the column-extrema paths above the shared-memory capacities.

Every equalization scale and every quantization range comes from a min or max that the kernels combine across threads and
CTAs with float atomics (common.cuh atomic_min_f / atomic_max_f).  -0.0 is an ordinary weight value: the BN fold multiplies
a zero (pruned) weight by gamma / sqrt(var + eps), which is -0.0 whenever gamma < 0.  Two input patterns:

    max is -0.0     every value <= 0, -0.0 scattered among negatives: the maximum is (negative) zero
    min clobber     mostly positive values, whole tile- or CTA-sized runs of -0.0, one strongly negative element per column /
                    sample / tensor: a partial minimum of -0.0 must not replace the true negative minimum

Extrema are compared by value (==): the sign of a zero result is not part of the contract.  Every test asserts that its
input really contains negative zeros.

The second half runs pruned, negative-gamma Conv+BN blocks through the full fused step (fold with column scan ->
equalization -> bias correction with column hints) against the oracle at widths on both sides of the shared-memory caches
of the fold scan (1024 columns), the equalization's scan and re-scan (1024), its reciprocal-scale cache (2044) and the
correction's expectation cache (2048); and per-tensor quantization of tensors whose extremes are +-0.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import dfq_oracle as O

pytestmark = pytest.mark.gpu
f32 = np.float32
NEG = f32(-5.0)          # the strongly negative element of the "min clobber" pattern


def _neg_zeros(x) -> int:
    x = torch.as_tensor(x)
    return int(((x == 0) & torch.signbit(x)).sum())


def _max_is_neg_zero(n, rng):
    """All values <= 0; about one in eight is -0.0 (at least one)."""
    x = -(np.abs(rng.standard_normal(n)) + 0.1).astype(f32)
    x[rng.random(n) < 0.125] = -0.0
    x[rng.integers(n)] = -0.0
    return x


def _min_clobber(n, rng, run=4096):
    """Positive values; every 7th value and, in tensors longer than `run`, every other `run`-sized block is -0.0; one
    element is NEG (outside the blocks)."""
    x = (np.abs(rng.standard_normal(n)) + 0.1).astype(f32)
    x[::7] = -0.0
    for a in range(0, n if n > run else 0, 2 * run):
        x[a:a + run] = -0.0
    if n > 1:
        free = np.flatnonzero(x > 0)
        x[free[rng.integers(free.size)] if free.size else n - 1] = NEG
    return x


PATTERNS = {"max_neg_zero": _max_is_neg_zero, "min_clobber": _min_clobber}
SIZES = [1, 5, 4099, 2 ** 20 + 3, 12_800_003]


def _cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x, f32)).cuda()


# ---------------------------------------------------------------------------------------------------------------------
# (a) stand-alone reductions
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pattern", sorted(PATTERNS))
@pytest.mark.parametrize("n", SIZES)
def test_tensor_minmax_with_negative_zeros(pattern, n):
    """dfq_minmax (tensor_minmax: the range of _quantize_error and the ncnn export): block reduce, then one float atomic per
    CTA.  The unaligned case starts one float past a 16-byte boundary (the scalar path)."""
    from dfq_b200.utils.quantize import tensor_minmax
    rng = np.random.default_rng(n)
    x = PATTERNS[pattern](n, rng)
    assert _neg_zeros(x) > 0
    xd = _cuda(x)
    got = tensor_minmax(xd).cpu().numpy()
    assert got[0] == x.min() and got[1] == x.max(), (pattern, n, got, x.min(), x.max())
    if n > 1:
        base = torch.empty(n + 1, device="cuda")
        base[1:] = xd
        xu = base[1:]
        assert xu.data_ptr() % 16 == 4
        got = tensor_minmax(xu).cpu().numpy()
        assert got[0] == x.min() and got[1] == x.max(), ("unaligned", pattern, n, got)


@pytest.mark.parametrize("pattern", sorted(PATTERNS))
@pytest.mark.parametrize("batch,per", [(1, 5), (4, 300_007), (3, 2 ** 20 + 3), (37, 4099), (256, 33)])
def test_per_sample_minmax_mean_with_negative_zeros(pattern, batch, per):
    """dfq_act_minmax_per_sample: a sample longer than 4096 floats is split over several CTAs whose partial extrema meet in
    float atomics.  Each sample carries the pattern (its own -0.0 runs and negative element)."""
    from dfq_b200.utils.quantize import per_sample_minmax_mean
    rng = np.random.default_rng(batch * 7 + per)
    x = np.stack([PATTERNS[pattern](per, rng) for _ in range(batch)])
    assert _neg_zeros(x) > 0
    want = O.per_sample_minmax_mean(x)
    got = per_sample_minmax_mean(_cuda(x).view(batch, -1)).cpu().numpy()
    assert got[0] == want[0] and got[1] == want[1], (pattern, batch, per, got, want)


@pytest.mark.parametrize("pattern", sorted(PATTERNS))
@pytest.mark.parametrize("batch,per", [(1, 5), (4, 300_007), (37, 4099)])
def test_observer_with_negative_zeros(pattern, batch, per):
    """dfq_observe_quant (observe_and_quant, update_stat branch): per-sample extrema -> batch mean -> running min/max ->
    fake quantization with that range, against the oracle's observer and quantizer (reciprocal mode, CUDA input)."""
    from dfq_b200.utils.quantize import OBS_UPDATE, observe_and_quant
    rng = np.random.default_rng(batch + per)
    x = np.stack([PATTERNS[pattern](per, rng) for _ in range(batch)])
    assert _neg_zeros(x) > 0
    rmin = torch.full((1,), 1e30, device="cuda"); rmax = torch.full((1,), -1e30, device="cuda")
    want_min, want_max = O.observer_update(1e30, -1e30, x)
    y = observe_and_quant(_cuda(x), 8, OBS_UPDATE, rmin, rmax, batch=batch)
    assert float(rmin) == want_min and float(rmax) == want_max, (pattern, batch, per, float(rmin), float(rmax), want_min, want_max)
    y_ref = O.quantize(x, 8, float(want_min), float(want_max), div_mode="recip")
    assert np.array_equal(y.cpu().numpy(), y_ref), (pattern, batch, per)


@pytest.mark.parametrize("pattern", sorted(PATTERNS))
@pytest.mark.parametrize("n", [5, 4099, 2 ** 20 + 3])
@pytest.mark.parametrize("signed", [False, True])
def test_quantize_error_with_negative_zeros(pattern, n, signed):
    """_quantize_error on a CUDA tensor: its range comes from dfq_minmax; Q(w) - w bit-exact against the oracle."""
    from dfq_b200.dfq import _quantize_error
    rng = np.random.default_rng(n + 1)
    x = PATTERNS[pattern](n, rng)
    assert _neg_zeros(x) > 0
    ref = O.quantize(x, 8, float(x.min()), float(x.max()), signed, div_mode="recip") - x
    got = _quantize_error(_cuda(x), 8, None, signed).cpu().numpy()
    assert np.array_equal(got, ref), (pattern, n, signed, int((got != ref).sum()))


def _range_cols_case(pattern, o, j, kk, groups, rng):
    """W[o, j, kk] with the pattern per column: "max_neg_zero" as in the flat case; "min clobber" with whole 32-row tiles
    (the kernel's tile) of -0.0 and one NEG per column of every group in a random row."""
    if pattern == "max_neg_zero":
        return _max_is_neg_zero(o * j * kk, rng).reshape(o, j, kk)
    w = (np.abs(rng.standard_normal((o, j, kk))) + 0.1).astype(f32)
    w[::3] = -0.0
    go = o // groups
    for g in range(groups):
        for t in range(g * go, (g + 1) * go, 64):
            w[t:min(t + 32, (g + 1) * go)] = -0.0
        rows = g * go + rng.integers(0, go, size=j)
        w[rows, np.arange(j), rng.integers(0, kk, size=j)] = NEG
    return w


@pytest.mark.parametrize("pattern", sorted(PATTERNS))
@pytest.mark.parametrize("o,j,kk,groups", [(256, 64, 9, 1), (96, 16, 9, 2), (1000, 1280, 1, 1), (5, 7, 25, 1)])
def test_range_rows_and_cols_with_negative_zeros(pattern, o, j, kk, groups):
    """dfq_range_cols (32-row tiles, one float atomic per tile and column) and dfq_range_rows (warp- or CTA-per-row
    reductions, no atomics) against numpy."""
    from dfq_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(o * j + kk)
    w_np = _range_cols_case(pattern, o, j, kk, groups, rng)
    assert _neg_zeros(w_np) > 0
    w = _cuda(w_np)
    P = lambda t: C.c_void_p(t.data_ptr())
    cmin = torch.empty(groups * j, device="cuda"); cmax = torch.empty(groups * j, device="cuda")
    _lib.check(lib.dfq_range_cols(P(w), o, j, kk, groups, P(cmin), P(cmax), _lib.stream_ptr()), "dfq_range_cols")
    v = w_np.reshape(groups, o // groups, j, kk)
    want_min, want_max = v.min(axis=(1, 3)).reshape(-1), v.max(axis=(1, 3)).reshape(-1)
    assert np.array_equal(cmin.cpu().numpy(), want_min), (pattern, o, j, kk, groups, "column min")
    assert np.array_equal(cmax.cpu().numpy(), want_max), (pattern, o, j, kk, groups, "column max")
    # rows of the layer (warp per row up to 2048 floats) and, where O divides by 4, rows 4x longer (CTA per row above 2048)
    for rows, row_len in [(o, j * kk)] + ([(o // 4, 4 * j * kk)] if o % 4 == 0 else []):
        rmin = torch.empty(rows, device="cuda"); rmax = torch.empty(rows, device="cuda")
        _lib.check(lib.dfq_range_rows(P(w), rows, row_len, P(rmin), P(rmax), _lib.stream_ptr()), "dfq_range_rows")
        r = w_np.reshape(rows, row_len)
        assert np.array_equal(rmin.cpu().numpy(), r.min(1)) and np.array_equal(rmax.cpu().numpy(), r.max(1)), (pattern, rows, row_len)


# ---------------------------------------------------------------------------------------------------------------------
# (b) pruned, negative-gamma Conv+BN blocks through the fused step
# ---------------------------------------------------------------------------------------------------------------------
def _prune_and_flip(st, seed, zero_rows=0):
    """Edit every block's second conv and its BN in the arena (before the fold):
      - negate gamma for about half of the rows (the fold then writes -0.0 for every zero weight of those rows);
      - zero about 25 % of the (o, j) kernels;
      - make 4 columns non-positive after the fold, with -0.0 in them (their maximum is -0.0): a weight takes the sign
        opposite to its row's gamma, and zeros stay only in negative-gamma rows;
      - zero_rows > 0: also zero that many whole negative-gamma rows (a row block of -0.0 after the fold).
    Returns the edited columns."""
    sess, Cn, kk = st.sess, st.C, st.k * st.k
    rng = np.random.default_rng(seed)
    special = rng.choice(Cn, size=4, replace=False)
    for b in range(st.n_blocks):
        l, v = sess.layer(st.layers[2 * b + 1]), st.vec[2 * b + 1]
        wv = sess.view(l["w_off"], st.N).view(Cn, Cn, kk)
        gv = sess.view(v["gamma"], Cn)
        w = wv.cpu().numpy().copy()
        g = gv.cpu().numpy().copy()
        neg = rng.random(Cn) < 0.5
        neg[:2] = True; neg[2:4] = False
        g[neg] = -g[neg]
        w[rng.random((Cn, Cn)) < 0.25] = 0.0
        for j in special:
            col = np.abs(w[:, j, :])
            col[col == 0] = 0.01
            col[neg & (rng.random(Cn) < 0.4)] = 0.0
            col[np.flatnonzero(neg)[0]] = 0.0
            w[:, j, :] = np.where(neg[:, None], col, -col)
        if zero_rows:
            w[np.flatnonzero(neg)[:zero_rows]] = 0.0
        wv.copy_(torch.from_numpy(w).view(Cn, Cn, kk))
        gv.copy_(torch.from_numpy(g))
    return special


def _check_blocks(st, pristine, res, what):
    from oracle import stack_check
    assert res.converged, what
    after = st.state()
    for b in range(st.n_blocks):
        r = stack_check.compare_block(st.block_arrays(pristine, b), st.block_arrays(after, b))
        assert r["weights_bit_exact"] and r["vectors_bit_exact"], (what, b, r)
        assert r["bias_normwise"] < 1e-5 and r["sweeps"] == int(res.group_sweeps[b]), (what, b, r, res.group_sweeps)


# (C, k, DFQ_CLE_STACK, DFQ_BC_STREAM); None = the library's own choice
BLOCK_CASES = [
    (64, 3, None, None),        # shared-memory atomics of the fold scan, several rows per tile
    (512, 3, "0", None),        # k_cle_engine
    (512, 3, "1", None),        # k_cle_stack (at most 512 input columns)
    (1024, 1, None, None),      # at the fold's and the equalization's scan capacity (a thread per column, no atomics)
    (1040, 1, None, None),      # above it: global atomics
    (1040, 3, None, None),
    (2044, 1, None, None),      # the reciprocal-scale cache is just big enough
    (2045, 1, None, None),      # one column more: generic path
    (2560, 1, None, "0"),       # above the correction's expectation cache: k_bc_engine reads E[x] from global memory
    (2560, 1, None, "1"),       # k_bc_stream
]


@pytest.mark.parametrize("pruned", [True, False])
@pytest.mark.parametrize("channels,k,cle_stack,bc_stream", BLOCK_CASES)
def test_fused_step_on_pruned_negative_gamma_blocks(channels, k, cle_stack, bc_stream, pruned, monkeypatch):
    """Two Conv[C,C,k,k]+BN+ReLU -> Conv[C,C,k,k]+BN blocks (two convergence groups) through DeviceStack.run(): fold with
    the column scan, equalization from those column extrema, bias correction with the column hints; weights and BN vectors
    bit-exact, corrected bias within 1e-5, sweep counts equal.  pruned=False runs the same widths on ordinary weights.
    Above 1024 columns the step is repeated with the equalization doing its own initial column scan (no cols_ready)."""
    from dfq_b200.engine import Session
    from dfq_b200.workload import DeviceStack
    if cle_stack is not None:
        monkeypatch.setenv("DFQ_CLE_STACK", cle_stack)
    if bc_stream is not None:
        monkeypatch.setenv("DFQ_BC_STREAM", bc_stream)
    sess = Session()
    st = DeviceStack(sess, 2, channels, k, seed=channels * 10 + k)
    st.generate()
    if pruned:
        special = _prune_and_flip(st, channels + k)
    pristine = st.state().clone()
    if pruned:
        d = st.block_arrays(pristine, 0)[1]
        w2 = O.bn_fold(d["w"], d["bias"], d["gamma"], d["beta"], d["mean"], d["var"], 1e-5)[0]
        assert _neg_zeros(w2) > channels, "the folded weights hold no -0.0"
        for j in special:
            assert w2[:, j].max() == 0 and _neg_zeros(w2[:, j]) > 0 and not (w2[:, j] > 0).any(), j
    res = st.run()
    _check_blocks(st, pristine, res, "fused step")
    if channels > 1024:
        st.state().copy_(pristine)
        sess.run_bn_fold(st.fold_plan)
        res = sess.run_cle_plan(st.cle_plan)
        sess.run_bias_correct_plan(st.bc_plan, 8, col_hints=sess.cle_col_hints(st.cle_plan, res))
        _check_blocks(st, pristine, res, "equalization's own initial scan")


# ---------------------------------------------------------------------------------------------------------------------
# (c) per-tensor quantization with +-0 extremes
# ---------------------------------------------------------------------------------------------------------------------
def _tile_blocks_tensor(rows, cols, rng, neg_at):
    """Positive values with every other 4096-float tile (the quantization kernels' flat tile) set to -0.0 - a pruned
    negative-gamma row block after the fold - and one NEG at flat position `neg_at` outside those tiles."""
    x = (np.abs(rng.standard_normal((rows, cols))) + 0.1).astype(f32).reshape(-1)
    for a in range(0, x.size, 2 * 4096):
        x[a:a + 4096] = -0.0
    x[neg_at] = NEG
    return x.reshape(rows, cols)


@pytest.mark.parametrize("bits,sym", [(4, False), (4, True), (8, False), (8, True), (16, False), (16, True)])
def test_run_quantize_tensors_with_zero_extremes(bits, sym):
    """dfq_quantize_tensors (k_minmax_tasks + k_quant_tasks): several tensors in one call, bit-exact against the oracle."""
    from dfq_b200.engine import Session
    rng = np.random.default_rng(bits * 2 + sym)
    ts = [_tile_blocks_tensor(64, 1024, rng, 4096 * (2 * k + 1) + 17 * k) for k in range(6)]          # 16 tiles each
    ts += [_tile_blocks_tensor(3, 50_000, rng, 149_999)]                                                 # NEG in the last tile
    ts += [_max_is_neg_zero(n, rng) for n in (5, 4099, 65_539)]
    ts += [_min_clobber(n, rng) for n in (4099, 2 ** 20 + 3)]
    for t in ts:
        assert _neg_zeros(t) > 0
    refs = [O.quantize(t, bits, float(t.min()), float(t.max()), symmetric=sym) for t in ts]
    tensors = [torch.from_numpy(t.copy()) for t in ts]
    sess = Session()
    offs = [sess.bind(t) for t in tensors]
    sess.upload()
    sess.run_quantize([(o, t.numel(), bits, sym) for o, t in zip(offs, tensors)])
    sess.download()
    for i, (t, r) in enumerate(zip(tensors, refs)):
        assert np.array_equal(t.numpy(), r.reshape(t.shape)), (i, bits, sym, int((t.numpy() != r.reshape(t.shape)).sum()))


@pytest.mark.parametrize("channels,k", [(64, 3), (1040, 1)])
def test_stack_quantize_plan_on_pruned_blocks(channels, k):
    """DeviceStack(quantize=True): the 8-bit weight / bias fake-quant that ends the step, on the equalized and corrected
    weights of pruned negative-gamma blocks with whole -0.0 rows; every tensor bit-exact against the oracle on what the step
    left before the quantization."""
    from dfq_b200.engine import Session
    from dfq_b200.workload import DeviceStack
    sess = Session()
    st = DeviceStack(sess, 2, channels, k, seed=3, quantize=True)
    st.generate()
    _prune_and_flip(st, 5, zero_rows=max(8, 2 * 4096 // (channels * k * k)))
    sess.run_bn_fold(st.fold_plan)
    res = sess.run_cle_plan(st.cle_plan, cols_ready=st.fold_plan["scanned"])
    sess.run_bias_correct_plan(st.bc_plan, 8, col_hints=sess.cle_col_hints(st.cle_plan, res))
    tasks = st.quant_plan["qt"]
    before = [sess.view(int(t["off"]), int(t["n"])).cpu().numpy() for t in tasks]
    assert sum(_neg_zeros(b) for b in before) > channels
    sess.run_quantize(st.quant_plan)
    for t, b in zip(tasks, before):
        got = sess.view(int(t["off"]), int(t["n"])).cpu().numpy()
        assert np.array_equal(got, O.quantize(b, 8)), (int(t["off"]), int(t["n"]))
