"""Generate tests/golden/reference_checks.pt: the outputs of the UNMODIFIED reference (kkoutini/PaSST, imported through
tests/ref_shim.py; set PASST_REF_ROOT to its checkout) that tests/test_oracle_vs_reference.py and
tests/test_host_frows.py compare the oracle and the host-side draws against.  The inputs are the tests' own seeded
inputs; run it on the CPU:

    PASST_REF_ROOT=<PaSST checkout> python tests/golden/make_reference_checks.py

To keep the file small:
  * a mel spectrogram is stored as the SHA-256 of its float32 bytes (the test is bit-exact) and a strided sample,
  * a parameter gradient of the 3-block network is stored whole up to FULL_LIMIT elements; larger ones as N_SAMPLES
    strided samples (tests/util.py golden_sample_index), N_PROJ random projections (tests/util.py golden_projections)
    and the L2 norm of the test's allclose envelope (atol + rtol * |g|), which bounds the projections of an error
    that passes the element-wise check,
  * logits and features (at most 527 values per case) are stored whole.
The CPU matrix products' summation order, and with it the last bits of the logits, depends on torch's intra-op thread
count, so the reference runs with NUM_THREADS threads and the test runs the oracle with the same count.
"""
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from ref_shim import REF_ROOT, load_reference, quiet  # noqa: E402
from util import golden_projections, golden_sample_index  # noqa: E402
from oracle import passt_oracle as O  # noqa: E402

OUT = os.path.join(HERE, "reference_checks.pt")
FULL_LIMIT = 1024
N_SAMPLES = 512
N_PROJ = 4
NUM_THREADS = 8
RTOL, ATOL = 1e-5, 1e-7                     # tests/test_oracle_vs_reference.py gradient tolerance
MEL_CASES = [(training, L) for L in (48000, 33001) for training in (False, True)]
NET_CASES = [(dict(s_patchout_t=40, s_patchout_f=4), 1000), (dict(u_patchout=400), 1000),
             (dict(s_patchout_t=10, s_patchout_f=3, n_classes=50), 500)]


def mel_key(training, L):
    return f"{'train' if training else 'eval'}_{L}"


def net_key(kw, T):
    return ",".join(f"{k}={v}" for k, v in sorted(kw.items())) + f",T={T}"


def tensor_digest(t: torch.Tensor) -> str:
    return hashlib.sha256(t.detach().float().contiguous().numpy().tobytes()).hexdigest()


def _mel_records():
    _, rpre = load_reference()
    out = {}
    for training, L in MEL_CASES:
        with quiet():
            mel = rpre.AugmentMelSTFT(n_mels=128, sr=32000, win_length=800, hopsize=320, n_fft=1024, freqm=48,
                                      timem=192, htk=False, fmin=0.0, fmax=None, norm=1, fmin_aug_range=10,
                                      fmax_aug_range=2000).train(training)
        torch.manual_seed(0)
        wave = 0.1 * torch.randn(2, L)
        torch.manual_seed(3)
        with quiet():
            ref = mel(wave)
        out[mel_key(training, L)] = dict(shape=tuple(ref.shape), sha256=tensor_digest(ref),
                                         samples=ref.flatten()[golden_sample_index(ref.numel(), N_SAMPLES)].clone())
    return out


def _grad_record(name, g):
    rec = dict(shape=tuple(g.shape), absmax=float(g.abs().max()), l2=float(g.double().norm()),
               env_l2=float((ATOL + RTOL * g.double().abs()).norm()), proj=golden_projections(name, g, N_PROJ))
    if g.numel() <= FULL_LIMIT:
        rec["full"] = g.detach().clone()
    else:
        rec["samples"] = g.detach().flatten()[golden_sample_index(g.numel(), N_SAMPLES)].clone()
    return rec


def _net_records():
    rp, _ = load_reference()
    out = {}
    for kw, T in NET_CASES:
        cfg12 = O.NetCfg(**kw)
        with quiet():
            net = rp.get_model(arch="passt_s_swa_p16_128_ap476", pretrained=False, n_classes=cfg12.n_classes,
                               u_patchout=cfg12.u_patchout, s_patchout_t=cfg12.s_patchout_t,
                               s_patchout_f=cfg12.s_patchout_f)
            net.load_state_dict(O.synth_params(cfg12, 2), strict=True)
            net = rp.lighten_model(net, cut_depth=9)        # keeps blocks 0, 10, 11
        torch.manual_seed(1)
        x = torch.randn(1, 1, 128, T)
        net.train()
        torch.manual_seed(8)
        with quiet():
            logits, feats = net(x)
        logits.sum().backward()
        grads = {k: _grad_record(k, p.grad) for k, p in net.named_parameters() if p.grad is not None}
        no_grad = sorted(k for k, p in net.named_parameters() if p.grad is None)
        out[net_key(kw, T)] = dict(logits=logits.detach().clone(), features=feats.detach().clone(), grads=grads,
                                   no_grad=no_grad)
    return out


def _mixup_record():
    import importlib.util
    spec = importlib.util.spec_from_file_location("_ref_mixup", os.path.join(REF_ROOT, "helpers", "mixup.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    torch.manual_seed(5)
    np.random.seed(6)
    perm, lam = mod.my_mixup(16, 0.3)
    return dict(size=16, alpha=0.3, torch_seed=5, numpy_seed=6, perm=perm.clone(), lam=lam.clone())


def main():
    torch.set_num_threads(NUM_THREADS)
    G = dict(full_limit=FULL_LIMIT, n_samples=N_SAMPLES, n_proj=N_PROJ, rtol=RTOL, atol=ATOL, num_threads=NUM_THREADS,
             mel=_mel_records(), net=_net_records(), mixup=_mixup_record())
    torch.save(G, OUT)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
