"""The built library really contains Blackwell-native code: per kernel, the sm_100a SASS mnemonics that prove tcgen05
tensor-core MMAs (UTCHMMA, .2CTA for cta_group::2), TMEM loads/stores (LDTM / STTM), TMA loads / stores / reduce-adds
(UTMALDG / UTMASTG / UTMAREDG) and programmatic dependent launch (ACQBULK / PREEXIT).  Runs `cuobjdump -sass` on the
in-tree .so; no GPU needed."""
import collections
import os
import re
import shutil
import subprocess

import pytest

KEYS = ("UTCHMMA", "UTCBAR", "UTMALDG", "UTMASTG", "UTMAREDG", "LDTM", "STTM", "MUFU.EX2", "ACQBULK", "PREEXIT")


def _cuobjdump():
    """cuobjdump from PATH, else from the toolkit of the nvcc the library is built with."""
    from passt_b200 import build
    nvcc = shutil.which(build._nvcc())
    for c in (shutil.which("cuobjdump"), nvcc and os.path.join(os.path.dirname(nvcc), "cuobjdump")):
        if c and os.path.isfile(c):
            return c
    return None


@pytest.fixture(scope="module")
def sass_ops():
    cuobjdump = _cuobjdump()
    if cuobjdump is None:
        pytest.skip("cuobjdump not found (neither on PATH nor next to nvcc)")
    from passt_b200 import build
    so = build.build()
    out = subprocess.run([cuobjdump, "-sass", str(so)], capture_output=True, text=True, timeout=600).stdout
    ops = collections.defaultdict(collections.Counter)
    cur = None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
        if m and cur:
            for k in KEYS:
                if m.group(1).startswith(k):
                    ops[cur][m.group(1)] += 1
    assert ops, "no sm_100a SASS found in the library"
    return ops


def _kernels(ops, name):
    hits = {k: v for k, v in ops.items() if name in k}
    assert hits, f"kernel {name} not in the library"
    return hits


def _has(counter, prefix):
    return any(op.startswith(prefix) for op in counter)


def test_gemm_family_is_2cta_tcgen05_with_tma(sass_ops):
    for name, c in _kernels(sass_ops, "gemm2_kernel").items():
        assert _has(c, "UTCHMMA.2CTA") and _has(c, "UTMALDG.2D.2CTA") and _has(c, "UTCBAR.2CTA.MULTICAST"), name
        assert _has(c, "LDTM") and (_has(c, "UTMASTG") or _has(c, "UTMAREDG")), name
    # the weight-gradient mode accumulates its split-K partials with TMA reduce-adds
    assert any(_has(c, "UTMAREDG.2D.ADD") for c in _kernels(sass_ops, "gemm2_kernelILi4E").values())


def test_attention_kernels_use_tensor_memory(sass_ops):
    for kern in ("attn_fwd2_kernel", "attn_fwd3_kernel", "attn_fwd_kernel", "attn_bwd_kernel", "attn_bwd2_kernel"):
        for name, c in _kernels(sass_ops, kern).items():
            assert _has(c, "UTCHMMA") and _has(c, "LDTM") and _has(c, "STTM") and _has(c, "UTMALDG.3D"), name
            assert _has(c, "MUFU.EX2"), name
    for name, c in _kernels(sass_ops, "attn_bwd").items():
        if "dq_pack" in name or "dsum" in name or "f32" in name:
            continue
        assert _has(c, "UTMAREDG.3D.ADD"), name          # dQ tiles are summed over key tiles by TMA reduce-add


def test_patch_embed_is_tma_in_tcgen05_tma_out(sass_ops):
    (name, c), = _kernels(sass_ops, "patch_embed_kernel").items()
    assert _has(c, "UTMALDG.3D") and _has(c, "UTMALDG.2D") and _has(c, "UTCHMMA") and _has(c, "LDTM") and _has(c, "UTMASTG.2D")


def test_hot_path_kernels_are_pdl_aware(sass_ops):
    for kern in ("gemm2_kernel", "attn_fwd2_kernel", "attn_bwd_kernel", "ln_fwd_kernel", "ln_bwd_kernel", "mel_kernel",
                 "im2col_kernel", "adamw_multi_kernel", "loss_bce_kernel"):
        for name, c in _kernels(sass_ops, kern).items():
            assert c["ACQBULK"] >= 1 and c["PREEXIT"] >= 1, name      # griddepcontrol.wait / launch_dependents
