"""Pin the CPU oracle against the reference implementation itself: the reference's outputs on these tests' seeded inputs
are stored in tests/golden/reference_checks.pt (written by tests/golden/make_reference_checks.py from the unmodified
reference).  Mel spectrograms are compared bit-exactly through their SHA-256, logits and features bit-exactly;
gradients element-wise on whole small tensors and strided samples, and on every element through random projections."""
import hashlib
import os

import pytest
import torch

from oracle import passt_oracle as O
from util import golden_projections, golden_sample_index

PATH = os.path.join(os.path.dirname(__file__), "golden", "reference_checks.pt")


@pytest.fixture(scope="module")
def G():
    return torch.load(PATH)


@pytest.fixture(scope="module", autouse=True)
def _reference_thread_count(G):
    """The reference ran with G["num_threads"] intra-op threads; the CPU matrix products' summation order (the last bits
    of the logits) depends on that count, so the oracle runs with the same count."""
    saved = torch.get_num_threads()
    torch.set_num_threads(G["num_threads"])
    yield
    torch.set_num_threads(saved)


@pytest.mark.parametrize("training", [False, True])
@pytest.mark.parametrize("L", [48000, 33001])
def test_mel_bit_exact(G, training, L):
    ref = G["mel"][f"{'train' if training else 'eval'}_{L}"]
    cfg = O.MelCfg()
    torch.manual_seed(0)
    wave = 0.1 * torch.randn(2, L)
    torch.manual_seed(3)
    d = O.draw_mel(cfg, training, 2)
    mine = O.mel_frontend(wave, cfg, d, training)
    assert tuple(mine.shape) == ref["shape"] and mine.dtype == torch.float32
    assert torch.equal(mine.flatten()[golden_sample_index(mine.numel(), G["n_samples"])], ref["samples"])
    assert hashlib.sha256(mine.contiguous().numpy().tobytes()).hexdigest() == ref["sha256"]


def test_mel_banks_match_torchaudio():
    import torchaudio
    for fmin, fmax in [(0.0, 15000.0), (7.0, 14321.0), (9.0, 16000.0)]:
        ref, _ = torchaudio.compliance.kaldi.get_mel_banks(128, 1024, 32000, fmin, fmax, 100.0, -500.0, 1.0)
        assert torch.equal(ref, O.kaldi_mel_banks(128, 1024, 32000, fmin, fmax))


@pytest.mark.parametrize("kw,T", [(dict(s_patchout_t=40, s_patchout_f=4), 1000), (dict(u_patchout=400), 1000),
                                  (dict(s_patchout_t=10, s_patchout_f=3, n_classes=50), 500)])
def test_net_train_forward_backward_light(G, kw, T):
    """3-block model (reference lighten_model cut_depth=9): logits, features, draws and gradients."""
    ref = G["net"][",".join(f"{k}={v}" for k, v in sorted(kw.items())) + f",T={T}"]
    cfg12 = O.NetCfg(**kw)
    cfg = O.NetCfg(depth=3, **kw)
    p = {}
    remap = {0: 0, 10: 1, 11: 2}
    for k, v in O.synth_params(cfg12, 2).items():
        if k.startswith("blocks."):
            i = int(k.split(".")[1])
            if i in remap:
                p[k.replace(f"blocks.{i}.", f"blocks.{remap[i]}.", 1)] = v
        else:
            p[k] = v
    p = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    torch.manual_seed(1)
    x = torch.randn(1, 1, 128, T)
    torch.manual_seed(8)
    d = O.draw_patchout(cfg, 12, (T - 16) // 10 + 1, True)
    lg, ft = O.passt_forward(p, x, cfg, d)
    assert torch.equal(ref["logits"], lg) and torch.equal(ref["features"], ft)
    lg.sum().backward()
    assert set(ref["grads"]) == {k for k, v in p.items() if v.grad is not None}
    for k in ref["no_grad"]:
        assert p[k].grad is None, k
    rtol, atol = G["rtol"], G["atol"]
    for k, rec in ref["grads"].items():
        g = p[k].grad
        assert tuple(g.shape) == rec["shape"], k
        if "full" in rec:
            assert torch.allclose(g, rec["full"], rtol=rtol, atol=atol), k
        else:
            got = g.flatten()[golden_sample_index(g.numel(), G["n_samples"])]
            assert torch.allclose(got, rec["samples"], rtol=rtol, atol=atol), k
        # <g - g_ref, r> for unit-variance r is ~ ||g - g_ref||_2, at most the L2 norm of the element-wise envelope
        pj = golden_projections(k, g, G["n_proj"])
        assert (pj - rec["proj"]).abs().max().item() <= 5 * rec["env_l2"], k
