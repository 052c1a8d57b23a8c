"""bench.py's command-line contract on a box without a GPU: the reference arm prints ONE JSON line with the agreed keys;
the GPU arm refuses to produce a number (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*flags, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *flags], capture_output=True, text=True, timeout=timeout,
                          cwd=ROOT)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run("--impl", "reference", "--cpu-layers", "2", "--steps", "3", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "conv_bn_layer_pairs_equalized_and_corrected_per_second"
    assert d["unit"] == "layers/s" and d["higher_is_better"] is True and d["value"] > 0 and d["steps"] >= 3
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["layers_per_step"] == 2 and d["config"]["sweeps"] == 2        # the stack converges in two sweeps
    assert abs(d["ms_per_step"] * 1e-3 * d["value"] - 2) < 1e-6


def test_gpu_arm_without_cuda_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = _run("--steps", "1", "--warmup", "1", "--layers", "8", "--no-e2e", "--no-mbv2", "--no-cpu-baseline", timeout=300)
    assert r.returncode != 0
    assert not [l for l in r.stdout.splitlines() if l.startswith("{") and '"value"' in l]


@pytest.mark.gpu
def test_dump_outputs_repeat_exactly_and_steps_are_honoured(tmp_path):
    """--dump-outputs writes the last timed step's results (float32/float64, <= 64 MB); the same arguments give the same
    inputs, hence the same outputs, in a second process; --steps sets the timed steps."""
    import numpy as np
    flags = ("--layers", "8", "--warmup", "1", "--no-e2e", "--no-mbv2", "--no-cpu-baseline")
    dumps = []
    for k, steps in enumerate((2, 5)):
        out = tmp_path / ("run%d" % k)
        r = _run("--steps", str(steps), "--dump-outputs", str(out), *flags)
        assert r.returncode == 0, r.stderr[-3000:]
        d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        assert d["steps"] == steps and d["parity_check"]["ok"]
        dumps.append({p.stem: np.load(p) for p in out.glob("*.npy")})
    a, b = dumps
    assert set(a) == {"weights", "bias", "bn_fake_weight", "bn_fake_bias", "scales", "sweeps"}
    assert sum(x.nbytes for x in a.values()) <= 64 * 2 ** 20
    assert a["bias"].shape == a["bn_fake_weight"].shape == (8 * 512,) and a["scales"].shape == (4 * 512,)
    assert a["sweeps"].shape == (4,) and (a["sweeps"] > 0).all()
    for name in a:
        assert a[name].dtype in (np.float32, np.float64), name
        assert np.array_equal(a[name], b[name]), name
        assert np.isfinite(a[name]).all(), name
