"""Generate tests/golden/passt_golden_grads.pt: every parameter gradient of the FULL-DEPTH (12-block) cfg2-shaped
train step, computed by the UNMODIFIED reference (imported from /root/reference through tests/ref_shim.py) on CPU.
Run in the build container only:

    python tests/golden/make_golden_grads.py

Same weights / input / seeds as passt_golden.pt (make_golden.py), so the two fixtures describe one run.  To keep the
file small, tensors with at most FULL_LIMIT elements are stored whole; larger ones are stored as
  * 1536 evenly strided samples (`samples`, taken at flat indices `arange(n)[::n // 1536][:1536]`),
  * their double-precision sum, max-abs and L2 norm,
  * 4 random projections <g, r_j> with r_j = randn(generator seeded by crc32(name) + j) -- a whole-tensor check.
"""
import os
import sys
import zlib

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from ref_shim import load_reference, quiet  # noqa: E402
from oracle import passt_oracle as O  # noqa: E402

FULL_LIMIT = 10_000
N_SAMPLES = 1536
N_PROJ = 4


def sample_index(n: int) -> torch.Tensor:
    return torch.arange(n)[:: max(1, n // N_SAMPLES)][:N_SAMPLES]


def projections(name: str, g: torch.Tensor) -> torch.Tensor:
    out = []
    flat = g.detach().double().flatten()
    for j in range(N_PROJ):
        gen = torch.Generator().manual_seed((zlib.crc32(name.encode()) + j) & 0x7FFFFFFF)
        r = torch.randn(flat.numel(), generator=gen, dtype=torch.float64)
        out.append(float(flat @ r))
    return torch.tensor(out, dtype=torch.float64)


def summarise(name: str, g: torch.Tensor) -> dict:
    n = g.numel()
    rec = dict(shape=tuple(g.shape), sum=float(g.double().sum()), absmax=float(g.abs().max()),
               l2=float(g.double().norm()), proj=projections(name, g))
    if n <= FULL_LIMIT:
        rec["full"] = g.detach().clone()
    else:
        rec["samples"] = g.detach().flatten()[sample_index(n)].clone()
    return rec


def main():
    rp, _ = load_reference()
    base = torch.load(os.path.join(HERE, "passt_golden.pt"))
    net_kw = base["net_kw"]
    cfg = O.NetCfg(**net_kw)
    with quiet():
        net = rp.get_model(arch="passt_s_swa_p16_128_ap476", pretrained=False, n_classes=527, **net_kw)
    net.load_state_dict(O.synth_params(cfg, seed=base["param_seed"]), strict=True)
    torch.manual_seed(base["input_seed"])
    x = torch.randn(*base["x_shape"])
    net.train()
    torch.manual_seed(base["rng_seed"])
    with quiet():
        logits, feats = net(x)
    assert torch.equal(logits.detach(), base["train_logits"])
    torch.manual_seed(base["grad_weight_seed"])
    w = torch.randn_like(logits)
    (logits * w).sum().backward()
    G = dict(net_kw=net_kw, param_seed=base["param_seed"], input_seed=base["input_seed"], rng_seed=base["rng_seed"],
             x_shape=base["x_shape"], grad_weight_seed=base["grad_weight_seed"], full_limit=FULL_LIMIT,
             n_samples=N_SAMPLES, n_proj=N_PROJ, grads={})
    for k, p in net.named_parameters():
        if p.grad is None:
            continue
        G["grads"][k] = summarise(k, p.grad)
    out = os.path.join(HERE, "passt_golden_grads.pt")
    torch.save(G, out)
    print("wrote", out, os.path.getsize(out), "bytes;", len(G["grads"]), "tensors")


if __name__ == "__main__":
    main()
