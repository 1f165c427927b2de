"""Host-side logic of the SURVEY.md §8f rows (loss / SWA / validation / waveform augmentation), no GPU needed:
the random draws are the reference's draws in the reference's order, and every module refuses CPU tensors loudly
instead of falling back to a CPU implementation."""
import os

import numpy as np
import pytest
import torch


def test_draw_mixup_is_the_reference_draw():
    """helpers/mixup.py:5-12, against the reference function's own draws (tests/golden/reference_checks.pt)."""
    from passt_b200 import loss as PL
    ref = torch.load(os.path.join(os.path.dirname(__file__), "golden", "reference_checks.pt"))["mixup"]
    torch.manual_seed(ref["torch_seed"]); np.random.seed(ref["numpy_seed"])
    perm, lam = PL.draw_mixup(ref["size"], ref["alpha"])
    assert torch.equal(perm, ref["perm"]) and torch.equal(lam, ref["lam"])
    assert lam.dtype == torch.float32 and float(lam.min()) >= 0.5


def test_wave_draws_follow_the_loader_order():
    """audioset/dataset.py:112 (gain: torch.randint), :333 (roll: numpy integers in [-r, r]), :128-134 (wavmix: torch.rand
    < rate, torch.randint partner, numpy beta) -- per clip, in that order."""
    from passt_b200.waveaug import WaveAugment
    aug = WaveAugment(clip_length=320000, gain_augment=7, roll_range=50, wavmix_rate=0.5, wavmix_beta=0.4)
    B = 6
    torch.manual_seed(3); np.random.seed(4)
    d = aug.draw(B)
    torch.manual_seed(3); np.random.seed(4)
    for b in range(B):
        g = torch.randint(14, (1,)).item() - 7
        assert abs(float(d.gain[b]) - 10 ** (g / 20)) < 1e-6
        s = int(np.random.randint(-50, 51))
        assert int(d.shift[b]) == s
        if torch.rand(1).item() < 0.5:
            j = int(torch.randint(B, (1,)).item())
            l = np.random.beta(0.4, 0.4)
            assert int(d.mix_idx[b]) == j and abs(float(d.mix_lam[b]) - max(l, 1 - l)) < 1e-6
        else:
            assert int(d.mix_idx[b]) == -1 and float(d.mix_lam[b]) == 1.0


def test_frow_modules_refuse_cpu_tensors():
    from passt_b200 import loss as PL
    from passt_b200 import evalpath
    from passt_b200.swa import SWAAverager
    from passt_b200.waveaug import WaveAugment
    z = torch.randn(4, 10, requires_grad=True)
    with pytest.raises(RuntimeError, match="CUDA"):
        PL.bce_with_logits(z, torch.rand(4, 10))
    with pytest.raises(RuntimeError, match="CUDA"):
        PL.cross_entropy(z, torch.randint(10, (4,)))
    with pytest.raises(RuntimeError, match="CUDA"):
        evalpath._sigmoid_mean([z.detach(), z.detach()])
    meter = evalpath.MeanAPMeter()
    meter.update(torch.rand(8, 3), (torch.rand(8, 3) > 0.5).float())
    with pytest.raises(RuntimeError, match="CUDA"):
        meter.average_precision()
    net = torch.nn.Linear(4, 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        SWAAverager(net).update()
    aug = WaveAugment(clip_length=1000)
    with pytest.raises(RuntimeError, match="CUDA"):
        aug(torch.randn(2, 1200), None, aug.draw(2))
