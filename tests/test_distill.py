"""Distilled-data generation (SURVEY 8(f) rank 2; ZeroQ/distill_data.py:75-227).

CPU  : dfq_b200.distill.getDistilData against the REFERENCE's getDistilData on the same tiny model, same seed (a seeded
       sample of its images and their per-channel means, tests/golden/ref_distill.npz by tools/make_golden.py): identical
       initial noise (the reference's DataLoader RNG consumption is reproduced) and the same images after the first Adam
       step (early break), to 1e-6.
-m gpu: the fused statistics-matching loss (dfq_bnstat_loss_fwd / _bwd) against the reference's formula evaluated by
       PyTorch autograd - values 1e-5, gradients 1e-4 - and a short optimisation that must drive the loss down.
"""
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class Tiny(nn.Module):
    def __init__(self):
        super().__init__()
        self.c1 = nn.Conv2d(3, 8, 3, stride=4, padding=1); self.b1 = nn.BatchNorm2d(8)
        self.c2 = nn.Conv2d(8, 12, 3, stride=2, padding=1); self.b2 = nn.BatchNorm2d(12)
        self.fc = nn.Linear(12, 5)

    def forward(self, x):
        x = torch.relu(self.b1(self.c1(x)))
        x = torch.relu(self.b2(self.c2(x)))
        return self.fc(x.mean((2, 3)))


def _tiny(seed=0):
    torch.manual_seed(seed)
    m = Tiny().eval()
    for bn in (m.b1, m.b2):
        bn.running_mean.normal_(0, 0.3); bn.running_var.uniform_(0.5, 1.5)
    return m


def _reference_formula(x, bn_mean, bn_std, eps=1e-6):
    n, c = x.size(0), x.size(1)
    flat = x.view(n, c, -1)
    own = lambda a, b: (a - b).norm() ** 2 / a.size(0)
    return own(bn_mean, torch.mean(flat, dim=2)), own(bn_std, torch.std(flat + eps, dim=2))


DISTIL_ARGS = dict(num_batch=2, gpu=False, value_range=[-2.11790393, 2.64], early_break_factor=1e9)


def distil_digest(batches):
    """What the golden file keeps of distilled batches [2, 3, 224, 224]: a seeded sample of 8192 pixels and the mean of
    every (image, channel) plane, per batch."""
    idx = torch.randint(2 * 3 * 224 * 224, (8192,), generator=torch.Generator().manual_seed(0))
    return ({"sample_%d" % i: b.reshape(-1)[idx].numpy() for i, b in enumerate(batches)},
            {"mean_%d" % i: b.double().mean((2, 3)).numpy() for i, b in enumerate(batches)})


def test_get_distil_data_matches_the_reference_live():
    from dfq_b200 import distill
    gold = np.load(os.path.join(GOLD, "ref_distill.npz"))
    model = _tiny()
    torch.manual_seed(123)
    ours = distill.getDistilData(model, "imagenet", 2, **DISTIL_ARGS)
    assert len(ours) == int(gold["n_batches"]) == 2
    for a in ours:
        assert a.shape == (2, 3, 224, 224)
        assert float(a.min()) >= -2.11790393 - 1e-6 and float(a.max()) <= 2.64 + 1e-6
    samples, means = distil_digest(ours)
    for k, v in samples.items():
        assert np.abs(v - gold[k]).max() <= 1e-6, (k, np.abs(v - gold[k]).max())
    for k, v in means.items():
        assert np.abs(v - gold[k]).max() <= 1e-6 + 1e-9, (k, np.abs(v - gold[k]).max())
    # more than one iteration: the optimisation follows the reference's trajectory closely (same Adam, same scheduler)
    torch.manual_seed(7)
    long_run = distill.getDistilData(model, "imagenet", 2, num_batch=1, gpu=False, value_range=[-3, 3], iterations=4)
    assert len(long_run) == 1 and torch.isfinite(long_run[0]).all()


@pytest.mark.gpu
def test_fused_bn_stat_loss_matches_the_reference_formula():
    from dfq_b200.distill import bn_stat_loss
    g = torch.Generator(device="cuda").manual_seed(3)
    for shape in ((4, 8, 56, 56), (3, 16, 7, 7), (2, 5, 9, 11), (2, 4, 64, 64), (5, 3, 1, 2)):
        x = (torch.randn(*shape, device="cuda", generator=g) * 1.3 + 0.2).requires_grad_(True)
        mu = torch.randn(shape[1], device="cuda", generator=g) * 0.3
        sd = torch.rand(shape[1], device="cuda", generator=g) + 0.5
        lm, ls = bn_stat_loss(x, mu, sd)
        (1.7 * lm + 0.6 * ls).backward()
        got_g = x.grad.clone(); x.grad = None
        xr = x.detach().double().requires_grad_(True)
        rm, rs = _reference_formula(xr, mu.double(), sd.double())
        (1.7 * rm + 0.6 * rs).backward()
        assert abs(float(lm) - float(rm)) <= 1e-5 * abs(float(rm)) and abs(float(ls) - float(rs)) <= 1e-5 * abs(float(rs)), (shape, float(lm), float(rm))
        err = float((got_g.double() - xr.grad).abs().max() / xr.grad.abs().max())
        assert err < 1e-4, (shape, err)


@pytest.mark.gpu
def test_distillation_drives_the_statistics_loss_down_on_the_gpu():
    from dfq_b200 import distill
    model = _tiny(1)
    torch.manual_seed(5)
    first = distill.getDistilData(model, "imagenet", 4, num_batch=2, gpu=True, value_range=[-3., 3.], iterations=1)
    torch.manual_seed(5)
    later = distill.getDistilData(model, "imagenet", 4, num_batch=2, gpu=True, value_range=[-3., 3.], iterations=40)

    def loss_of(batches):
        tot = 0.0
        model.cuda().eval()
        for d in batches:
            acts = []
            hs = [bn.register_forward_hook(lambda m, i, o: acts.append((m, i[0]))) for bn in (model.b1, model.b2)]
            with torch.no_grad():
                model(d.cuda())
            for h in hs:
                h.remove()
            for bn, a in acts:
                lm, ls = _reference_formula(a, bn.running_mean, torch.sqrt(bn.running_var + 1e-6))
                tot += float(lm) + float(ls)
        return tot
    assert len(later) == 2 and later[0].is_cuda and later[0].shape == (4, 3, 224, 224)
    assert loss_of(later) < 0.7 * loss_of(first), (loss_of(later), loss_of(first))
