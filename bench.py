#!/usr/bin/env python
"""bench.py — BASELINE.json metric: clips/sec (10 s @ 32 kHz) of a passt_s p16_128 TRAIN step (default), plus the other
BASELINE.json configurations behind --config.

Default workload (BASELINE.json configs[1], SURVEY.md §8d cfg2): passt_s, s_patchout_t=40, s_patchout_f=4 (N=474 tokens),
64 clips per GPU, bf16 tensor-core arithmetic with fp32 master weights / residual stream, synthetic AudioSet-shaped
data (0.1*randn waveforms, multi-hot 527-class targets), random-init weights.  One step = waveform -> fused mel
kernel (band augmentation + SpecAugment on) -> patchout-ViT forward -> BCE-with-logits -> hand-written backward
-> (N>1: NCCL gradient all-reduce) -> AdamW step.  Weak scaling: fixed clips per GPU at every N.

  python bench.py --gpus N --steps K --warmup W          # candidate (sm_100a kernels), cfg2
  python bench.py --config cfg1|cfg3|cfg4|cfg5 ...       # the other BASELINE.json configurations
  python bench.py --impl reference ...                   # the reference algorithm on the host CPU cores (oracle port)

At N=1 the line also carries `stock_gpu`: the reference algorithm as stock PyTorch-CUDA (oracle port = the same torch
ops the reference calls) on the same GPU in the same process — torch.compile'd and eager, fp16+GradScaler (the
reference's default: compile=True, precision=16, ex_audioset.py:74,79) and bf16 — and `vs_stock` = value / fastest
stock arm (north_star's ">= 3x").  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# all host threads the oracle can use productively: torch's intra-op pool stops scaling (and thrashes) well before the
# 100+ hardware threads of the GPU box on these matrix sizes, so cap it; the count actually used is reported as `cores`
CPU_THREADS = max(1, min(os.cpu_count() or 1, int(os.environ.get("PASST_CPU_THREADS", "32"))))

MEL_KW = dict(n_mels=128, sr=32000, win_length=800, hopsize=320, n_fft=1024, freqm=48, timem=192, fmin=0.0, fmax=None,
              fmin_aug_range=10, fmax_aug_range=2000)

# BASELINE.json `configs`, SURVEY.md section 8d
CONFIGS = {
    "cfg1": dict(kind="infer", arch="passt_s_swa_p16_128_ap476", depth=12, net_kw={}, batch=2, clip_len=320000,
                 n_classes=527, mel_kw={},
                 metric="clips/sec (10s@32kHz) passt_s_swa_p16_128_ap476 forward (eval)",
                 workload="passt_s_swa_p16_128_ap476 forward, batch=2, 10s@32kHz, eval (N=1190 tokens)"),
    "cfg2": dict(kind="train", arch="passt_s_swa_p16_128_ap476", depth=12, net_kw=dict(s_patchout_t=40, s_patchout_f=4),
                 batch=64, clip_len=320000, n_classes=527, mel_kw={}, loss="bce", mixup=0.0,
                 metric="clips/sec (10s@32kHz) passt_s p16_128 train step",
                 workload="passt_s p16_128 s_patchout_t=40 s_patchout_f=4, batch=64/GPU, 10s@32kHz, train step bf16"),
    "cfg3": dict(kind="train", arch="passt_s_swa_p16_128_ap476", depth=12, net_kw=dict(u_patchout=400), batch=16,
                 clip_len=320000, n_classes=527, mel_kw={}, loss="bce", mixup=0.3,
                 metric="clips/sec (10s@32kHz) passt_s p16_128 u_patchout=400 mixup train step",
                 workload="passt_s p16_128 u_patchout=400 (N=790), batch=16/GPU (128 on 8 GPUs), spectrogram mixup, "
                          "BCE 527 classes, DDP train step bf16"),
    "cfg4": dict(kind="infer", arch="passt_l_kd_p16_128_ap47", depth=7, net_kw={}, batch=256, clip_len=320000,
                 n_classes=527, mel_kw={},
                 metric="clips/sec (10s@32kHz) passt_l p16_128 no-patchout inference",
                 workload="passt_l p16_128 (7 blocks) no-patchout inference, batch=256, N=1190 (dense-attn roofline)"),
    "cfg5": dict(kind="train", arch="passt_s_kd_p16_128_ap486", depth=12, net_kw=dict(s_patchout_t=10, s_patchout_f=3),
                 batch=16, clip_len=160000, n_classes=50, mel_kw=dict(timem=80), loss="ce", mixup=0.3,
                 metric="clips/sec (5s@32kHz) ESC-50 fine-tune train step",
                 workload="ESC-50 fine-tune head (50 classes), 5s clips, s_patchout_t=10 s_patchout_f=3 (N=353), "
                          "batch=16/GPU (32 on 2 GPUs), CE + mixup, train step bf16"),
}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"], bf16_sustained=p["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source="fallback")


def fwd_flops_per_clip(ntok, depth, n_classes):
    return 2 * (ntok - 2) * 256 * 768 + depth * (2 * ntok * 768 * 9216 + 4 * ntok * ntok * 768) + 2 * 768 * n_classes


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], 0.0, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 0.5 * mx] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ======================================================================================================
# the reference algorithm as plain torch ops (oracle port, validated bit-exact against /root/reference on CPU):
# CPU arm (--impl reference, cpu_baseline) and stock PyTorch-CUDA arm (stock_gpu)
# ======================================================================================================
def _oracle_step_fn(cfg, device, batch, dtype=None, compile_net=False, fused_opt=False):
    """One step of `cfg` with the oracle port on `device` (train: mel + fwd + loss + bwd + AdamW; infer: mel + fwd).
    dtype None = fp32; torch.float16 adds GradScaler (the reference's precision=16), torch.bfloat16 plain autocast."""
    from oracle import passt_oracle as O
    mcfg = O.MelCfg(**{k: v for k, v in cfg["mel_kw"].items() if k in ("freqm", "timem")})
    ncfg = O.NetCfg(depth=cfg["depth"], n_classes=cfg["n_classes"], **cfg["net_kw"])
    train = cfg["kind"] == "train"
    params = {k: v.to(device).requires_grad_(train and not k.startswith("head_dist"))
              for k, v in O.synth_params(ncfg, 0).items()}
    torch.manual_seed(0)
    wave = 0.1 * torch.randn(batch, cfg["clip_len"], device=device)
    if cfg.get("loss") == "ce":
        y = torch.randint(cfg["n_classes"], (batch,), device=device)
    else:
        y = (torch.rand(batch, cfg["n_classes"], device=device) < 0.005).float()
    T = 1 + (cfg["clip_len"] - 1) // 320
    tg = (T - 16) // 10 + 1
    is_cuda = torch.device(device).type == "cuda"

    def net_fn(spec, t_keep, f_keep, u_keep, toffset):
        d = O.StepDraws(t_keep=t_keep, f_keep=f_keep, u_keep=u_keep, toffset=toffset)
        return O.passt_forward(params, spec, ncfg, d)[0]

    fn = torch.compile(net_fn) if compile_net else net_fn
    ac = (lambda: torch.autocast("cuda", dtype=dtype)) if (dtype is not None and is_cuda) else contextlib.nullcontext
    mv = (lambda t: None if t is None else t.to(device))
    if not train:
        def step():
            d = O.draw_mel(mcfg, False, batch, device=device)
            with torch.no_grad():
                spec = O.mel_frontend(wave, mcfg, d, False).unsqueeze(1)
                dp = O.draw_patchout(ncfg, 12, tg, False)
                with ac():
                    logits = fn(spec, None, None, None, dp.toffset)
            return logits
        return step
    opt = torch.optim.AdamW([p for p in params.values() if p.requires_grad], lr=2e-5, weight_decay=1e-4,
                            **(dict(fused=True) if (fused_opt and is_cuda) else {}))
    scaler = torch.amp.GradScaler("cuda", enabled=(dtype == torch.float16 and is_cuda))
    alpha = cfg.get("mixup", 0.0)

    def step():
        d = O.draw_mel(mcfg, True, batch, device=device)
        with torch.no_grad():
            spec = O.mel_frontend(wave, mcfg, d, True).unsqueeze(1)
        lam = perm = None
        if alpha:
            from passt_b200.loss import draw_mixup            # host RNG draws only (helpers/mixup.py:5-12 restated)
            perm, lam = draw_mixup(batch, alpha)
            perm, lam = perm.to(device), lam.to(device)
            spec = spec * lam.reshape(batch, 1, 1, 1) + spec[perm] * (1. - lam.reshape(batch, 1, 1, 1))
        dp = O.draw_patchout(ncfg, 12, tg, True)
        with ac():
            logits = fn(spec, mv(dp.t_keep), mv(dp.f_keep), mv(dp.u_keep), dp.toffset)
        logits = logits.float()
        if cfg["loss"] == "ce":
            if alpha:
                loss = (F.cross_entropy(logits, y, reduction="none") * lam +
                        F.cross_entropy(logits, y[perm], reduction="none") * (1. - lam)).mean()
            else:
                loss = F.cross_entropy(logits, y)
        else:
            yy = y * lam.reshape(batch, 1) + y[perm] * (1. - lam.reshape(batch, 1)) if alpha else y
            loss = F.binary_cross_entropy_with_logits(logits, yy, reduction="none").mean()
        opt.zero_grad(set_to_none=True)
        scaler.scale(loss).backward()
        scaler.step(opt)
        scaler.update()
        return loss.detach()
    return step


def cpu_rate(cfg, sample_clips=1, steps=1, warmup=0):
    """clips/s of the oracle port on the host CPU for `cfg` (bounded sample)."""
    torch.set_num_threads(CPU_THREADS)
    step = _oracle_step_fn(cfg, "cpu", sample_clips)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return sample_clips * steps / dt, dt / steps


def run_reference(args, rank, world):
    """Reference arm: the reference algorithm (oracle port, bit-exact with the reference on CPU) on the host cores.
    One step = one full step of the configuration on a bounded 1-clip sample; exactly --steps steps are timed after
    min(--warmup, 5) warm-up steps, so a run's last step (and --dump-outputs) does not depend on the host's speed."""
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    torch.set_num_threads(CPU_THREADS)
    sample = 1
    step = _oracle_step_fn(cfg, "cpu", sample)
    t_start = time.perf_counter()
    warm = min(max(0, args.warmup), 5)
    for _ in range(warm):
        step()
    warm_s = time.perf_counter() - t_start
    done, t0 = 0, time.perf_counter()
    while done < args.steps:
        result = step()
        done += 1
    dt = time.perf_counter() - t0
    rate = sample * done / dt
    what = "train step (mel train + fwd + bwd + AdamW)" if cfg["kind"] == "train" else "forward (mel eval + net eval)"
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": rate,
        "unit": "clips/s", "n_gpus": args.gpus, "steps": done, "warmup": warm,
        "ms_per_step": dt / done * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": cfg["workload"], "name": args.config,
                   "sample": f"{sample} clip per step on the host CPU ({CPU_THREADS} threads)",
                   "requested_steps": args.steps, "warmup_s": warm_s},
        "cpu_baseline": {"value": rate, "unit": "clips/s", "cores": CPU_THREADS, "kind": "port",
                         "sample": f"{done} x {sample}-clip {what}, oracle port, fp32"},
        "e2e": {"value": rate, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.dump_outputs:
        _write_outputs(args.dump_outputs, {"loss" if cfg["kind"] == "train" else "logits": result})
    _emit(line)


STOCK_BUDGET_S = float(os.environ.get("PASST_STOCK_BUDGET_S", "240"))


def stock_gpu_block(cfg, batch, steps=10, warmup=5):
    """The reference algorithm as stock PyTorch-CUDA on this GPU (SURVEY.md section 8d "Reference GPU baseline"):
    protocol of model_speed_test (ex_audioset.py:364-426: warm-up, then timed steps between synchronizes) extended to
    start from waveforms.  Arms: torch.compile'd and eager, fp16+GradScaler (reference default) and bf16."""
    arms = [("compiled_fp16_gradscaler", torch.float16, True), ("compiled_bf16", torch.bfloat16, True),
            ("eager_fp16_gradscaler", torch.float16, False), ("eager_bf16", torch.bfloat16, False)]
    out, t_start = {}, time.perf_counter()
    for name, dtype, comp in arms:
        if time.perf_counter() - t_start > STOCK_BUDGET_S:
            out[name] = {"skipped": f"time budget {STOCK_BUDGET_S:.0f} s used up"}
            continue
        try:
            torch._dynamo.reset()
            step = _oracle_step_fn(cfg, "cuda", batch, dtype=dtype, compile_net=comp, fused_opt=True)
            t_c = time.perf_counter()
            for _ in range(warmup):
                step()
            torch.cuda.synchronize()
            warm_s = time.perf_counter() - t_c
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[name] = {"clips_per_s": batch / ms * 1e3, "ms_per_step": ms, "steps": steps, "warmup": warmup,
                         "warmup_s": warm_s}
        except Exception as e:  # noqa
            out[name] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
        finally:
            del_step = None  # noqa
            torch.cuda.empty_cache()
    ok = {k: v["clips_per_s"] for k, v in out.items() if "clips_per_s" in v}
    best = max(ok, key=ok.get) if ok else None
    return {"arms": out, "best": best, "best_clips_per_s": ok.get(best) if best else None, "batch": batch,
            "what": "oracle port of the reference (same torch ops: rfft STFT, F.conv2d, F.layer_norm, F.linear, softmax, "
                    "F.gelu) under autocast, torch.optim.AdamW(fused); bit-exact with /root/reference on CPU "
                    "(tests/test_oracle_vs_reference.py); /root/reference itself does not exist on the GPU box"}


# ======================================================================================================
# candidate arm
# ======================================================================================================
def run_candidate(args, rank, local_rank, world):
    import torch.distributed as dist
    from passt_b200 import _lib as L
    from passt_b200 import engine
    from passt_b200 import loss as PL
    from passt_b200.passt import get_model
    from passt_b200.preprocess import AugmentMelSTFT
    from passt_b200.ddp import GradAllReducer

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py candidate arm needs a CUDA device (sm_100a); there is no CPU fallback")
    cfg = CONFIGS[args.config]
    train = cfg["kind"] == "train"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    L.load()
    peaks = load_peaks()
    B = args.batch or cfg["batch"]
    CLIP_LEN, NCLS = cfg["clip_len"], cfg["n_classes"]
    torch.manual_seed(rank)
    np.random.seed(rank)
    with contextlib.redirect_stdout(sys.stderr):     # the module prints the reference's "FMAX is None" notice
        mel = AugmentMelSTFT(**{**MEL_KW, **cfg["mel_kw"]}).to(dev).train(train)
    torch.manual_seed(0)   # identical initial weights on every rank
    net = get_model(arch=cfg["arch"], pretrained=False, n_classes=NCLS, **cfg["net_kw"]).to(dev).train(train)
    if args.precision == "fp32":
        net.precision = "fp32"
    use_graph = bool(args.graph)
    opt = reducer = None
    if train:
        opt_params = [p for n, p in net.named_parameters() if not n.startswith("head_dist")]
        if args.optim == "own":
            from passt_b200.optim import FusedAdamW
            opt = FusedAdamW(opt_params, lr=2e-5, weight_decay=1e-4).attach(net)
        else:
            opt = torch.optim.AdamW(opt_params, lr=2e-5, weight_decay=1e-4, fused=True, capturable=use_graph)
        reducer = GradAllReducer(net, reserve_sms=int(os.environ.get("PASST_DDP_RESERVE", "0"))) if world > 1 else None
    torch.manual_seed(1000 + rank)
    # rotating input batches so that consecutive steps never find their input in L2 (>= 4 batches, >= 256 MB in total)
    n_batches = max(4, -(-256 * 2**20 // (B * CLIP_LEN * 4)))
    host_waves = [(0.1 * torch.randn(B, CLIP_LEN)).pin_memory() for _ in range(n_batches)]
    dev_waves = [w.to(dev) for w in host_waves]
    if cfg.get("loss") == "ce":
        y = torch.randint(NCLS, (B,), device=dev)
        loss_fn = PL.cross_entropy
    else:
        y = (torch.rand(B, NCLS, device=dev) < 0.005).float()
        loss_fn = PL.bce_with_logits
    alpha = cfg.get("mixup", 0.0) if train else 0.0

    def eager_step(wave_dev):
        if not train:
            with torch.no_grad():
                logits, _ = net(mel(wave_dev).unsqueeze(1))
            return logits
        with torch.no_grad():
            spec = mel(wave_dev).unsqueeze(1)
        perm = lam = None
        if alpha:
            perm, lam = PL.draw_mixup(B, alpha)                    # after the mel draws, before the net's (reference order)
            perm, lam = perm.to(dev, non_blocking=True), lam.to(dev, non_blocking=True)
            net.fused_mixup(perm, lam)                             # folded into the patch gather
        logits, _ = net(spec)
        loss = loss_fn(logits, y, perm, lam)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        if reducer is not None:
            reducer.all_reduce()
        opt.step()
        return loss

    graphed = None
    if use_graph and train:
        from passt_b200.graphed import GraphedTrainStep
        graphed = GraphedTrainStep(mel, net, opt, loss_fn, dev_waves[0], y, reducer=reducer, warmup=3,
                                   mixup_alpha=alpha or None)
    elif use_graph:
        from passt_b200.graphed import GraphedInference
        graphed = GraphedInference(mel, net, dev_waves[0])

    def run_step(wave_dev, consumed=None):
        # public API: either the eager modules (mel -> net -> loss.backward -> opt.step) or the same step replayed
        # as one CUDA graph (passt_b200.graphed; inputs are copied into its static buffers).
        # consumed: event recorded once the input buffer may be refilled (graph: right after the staging copy)
        if graphed is not None:
            return graphed(wave_dev, None, consumed=consumed) if train else graphed(wave_dev, consumed=consumed)
        out = eager_step(wave_dev)
        if consumed is not None:
            consumed.record(torch.cuda.current_stream())
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    # ---- warm-up
    n_warm = max(3, args.warmup)
    for i in range(n_warm):
        run_step(dev_waves[i % n_batches])
    barrier()
    ntok = net.last_plan.ntok
    if world > 1 and train:
        # replicas must stay bit-identical: same initial weights + averaged gradients => same parameters on every rank
        chk = torch.stack([p.detach().double().sum() for p in net.parameters()]).sum().reshape(1)
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        if float((hi - lo).abs()) != 0.0:
            raise RuntimeError(f"DDP replicas diverged after warm-up: parameter checksum spread {float(hi - lo)}")

    # ---- (1) device-resident inputs
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    L.reset_launch_count()
    last = [None]

    def timed_step(i):
        last[0] = run_step(dev_waves[i % n_batches])

    ms_dev = timed(timed_step, args.steps)
    launches = L.launch_count()
    # taken before anything below runs another step on the same weights
    dumped = _timed_outputs(net, last[0], train) if (args.dump_outputs and rank == 0) else None
    if graphed is not None:
        # kernels are replayed by the graph; count the launches of one eager step and scale
        L.reset_launch_count()
        eager_step(dev_waves[0])
        launches = L.launch_count() * args.steps
        net._wcache.invalidate()
    clocks = sampler.stop() if rank == 0 else None

    # ---- (2) end to end through the public API with HOST buffers: every step's waveform batch is copied from pinned
    #          host memory (on a copy stream, one batch ahead of the compute, like a prefetching loader) and every
    #          step's result (train: the loss; inference: the logits) is read back to the host (asynchronously,
    #          consumed one step later, like a logging hook).
    copy_stream = torch.cuda.Stream(device=dev)
    dev_bufs = [torch.empty(B, CLIP_LEN, device=dev) for _ in range(2)]
    h2d_done = [torch.cuda.Event() for _ in range(2)]
    buf_free = [torch.cuda.Event() for _ in range(2)]
    res_shape = (1,) if train else (B, NCLS)
    res_hosts = [torch.zeros(res_shape).pin_memory() for _ in range(2)]
    res_done = [torch.cuda.Event() for _ in range(2)]
    checks = []

    def upload(i):
        k = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(buf_free[k])
            dev_bufs[k].copy_(host_waves[i % n_batches], non_blocking=True)
            h2d_done[k].record(copy_stream)

    def e2e_run(steps):
        cur = torch.cuda.current_stream()
        for k in range(2):
            buf_free[k].record(cur)
        upload(0)
        for i in range(steps):
            k = i & 1
            if i + 1 < steps:
                upload(i + 1)
            cur.wait_event(h2d_done[k])
            res = run_step(dev_bufs[k], consumed=buf_free[k])
            res_hosts[k].copy_(res.detach().reshape(res_shape), non_blocking=True)
            res_done[k].record(cur)
            if i > 0:
                res_done[k ^ 1].synchronize()
                checks.append(float(res_hosts[k ^ 1].flatten()[0]))
        res_done[(steps - 1) & 1].synchronize()
        checks.append(float(res_hosts[(steps - 1) & 1].flatten()[0]))

    e2e_run(2)

    def timed_once(fn):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    ms_e2e = timed_once(lambda: e2e_run(args.steps))
    if not all(np.isfinite(c) for c in checks):
        raise RuntimeError("non-finite result read back in the end-to-end run")

    # ---- (3) roofline of the dominant kernel family (tcgen05 GEMM): CUDA events around every GEMM launch in a
    #          repeat of the timed steps (kept out of the headline timing so the events do not perturb it)
    engine.GEMM_TRACE = []
    ms_instr = timed(lambda i: eager_step(dev_waves[i % n_batches]), args.steps)
    torch.cuda.synchronize()
    trace, engine.GEMM_TRACE = engine.GEMM_TRACE, None
    gemm_ms = sum(a.elapsed_time(b) for a, b, _ in trace)
    gemm_flops = sum(f for _, _, f in trace)
    n_gemm = max(1, len(trace))
    achieved_tf = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    peak_tf = peaks["bf16_sustained"]

    # ---- (4) the other kernels the contract names (SURVEY.md section 8d), timed alone with CUDA events
    other = None
    if rank == 0 and world == 1:
        other = _other_kernel_rooflines(mel, net, dev_waves[0], B, ntok, peaks)

    total_clips = B * world * args.steps
    value = total_clips / (ms_dev * 1e-3)
    e2e_value = total_clips / (ms_e2e * 1e-3)
    fwd_flops = fwd_flops_per_clip(ntok, cfg["depth"], NCLS) * B
    step_flops = fwd_flops * (3 if train else 1)

    line = None
    if rank == 0:
        line = {
            "metric": cfg["metric"], "value": value, "unit": "clips/s",
            "n_gpus": world, "steps": args.steps, "warmup": n_warm, "ms_per_step": ms_dev / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32 (3xbf16-split tcgen05 GEMMs, fp32 attention)",
            "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": args.config, "tokens": ntok, "global_batch": B * world,
                       "parallelism": f"dp{world}",
                       "optimizer": (None if not train else
                                     "passt_b200.FusedAdamW (one launch, refreshes the bf16 weight copies), fp32 master weights"
                                     if args.optim == "own" else "torch.optim.AdamW(fused), fp32 master weights"),
                       "loss": (None if not train else
                                ("fused BCE-with-logits" if cfg["loss"] == "bce" else "fused cross entropy") +
                                (f" + mixup alpha={alpha} (targets mixed in the loss kernel, spectrograms in the patch gather)"
                                 if alpha else "") + f", {NCLS} classes"),
                       "cuda_graph": bool(use_graph),
                       "l2": f"{n_batches} rotating input batches ({n_batches * B * CLIP_LEN * 4 / 2**20:.0f} MB) and a "
                             "per-step activation working set >> 126 MB L2",
                       "model_flops_per_step": step_flops,
                       "model_tflops": step_flops * world / (ms_dev / args.steps * 1e-3) / 1e12},
            "e2e": {"value": e2e_value, "unit": "clips/s", "h2d_bytes_per_step": B * CLIP_LEN * 4,
                    "d2h_bytes_per_step": 4 if train else B * NCLS * 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"kernel": "gemm2_kernel<MODE> (tcgen05 cta_group::2 GEMM family: fwd, dgrad, wgrad)",
                         "bound": "tensor",
                         "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved_tf / peak_tf if peak_tf else None,
                         # dram__bytes_read+write of the qkv-forward launch (107.4 GFLOP, 190 MB algorithmic) from
                         # profiles/r1_ncu_gemm2_full_v2.txt (ncu --set full): 50.3 MB read + 89.5 MB written
                         "traffic": 139.7e6, "traffic_launch": "qkv forward M=30336 N=2304 K=768 (cfg2)",
                         "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['source']})",
                         "launches_per_step": n_gemm / args.steps, "avg_launch_ms": gemm_ms / n_gemm,
                         "share_of_step": gemm_ms / ms_instr if ms_instr else None,
                         "how": "CUDA events around each GEMM launch in an eager (non-graph) repeat of the timed steps"},
        }
        if other is not None:
            line["other_kernels"] = other
        if world == 1:
            cpu_v, _ = cpu_rate(cfg, sample_clips=1, steps=3 if train else 5, warmup=1)
            line["cpu_baseline"] = {"value": cpu_v, "unit": "clips/s", "cores": CPU_THREADS, "kind": "port",
                                    "sample": ("3 x 1-clip train step after 1 warm-up (mel + fwd + bwd + AdamW)" if train
                                               else "5 x 1-clip forward after 1 warm-up (mel eval + net eval)") +
                                              " of the CPU oracle port, fp32"}
            if args.stock:
                # free the candidate's CUDA memory first (activations of the big configurations)
                graphed = None
                torch.cuda.empty_cache()
                sb = stock_gpu_block(cfg, B, steps=min(args.steps, 20))
                line["stock_gpu"] = sb
                line["vs_stock"] = value / sb["best_clips_per_s"] if sb["best_clips_per_s"] else None
        if dumped is not None:
            _write_outputs(args.dump_outputs, dumped)
        _emit(line)
    return line


DUMP_SAMPLE = 1 << 20      # elements in a sampled output (4 MB as float32)


def _seeded_sample(tensors, n=DUMP_SAMPLE, seed=0):
    """A fixed sample of the concatenated, flattened `tensors`: the same flat indices (sorted, drawn from a CPU
    generator seeded with `seed`) in every run with the same tensor sizes."""
    flat = torch.cat([t.detach().reshape(-1).float() for t in tensors])
    if flat.numel() <= n:
        return flat
    idx = torch.randint(flat.numel(), (n,), generator=torch.Generator().manual_seed(seed)).sort().values
    return flat[idx.to(flat.device)]


def _timed_outputs(net, result, train):
    """Device copies of what the last timed step gave its caller.  Inference: the logits.  Train: the loss, and seeded
    samples of the trained parameters after the optimizer step and of the gradients that step applied (in
    named_parameters order)."""
    if not train:
        return {"logits": result.detach().float().clone()}
    named = [(n, p) for n, p in net.named_parameters() if not n.startswith("head_dist")]
    missing = [n for n, p in named if p.grad is None]
    if missing:
        raise RuntimeError(f"the timed train step left no gradient for {missing}")
    params = [p for _, p in named]
    return {"loss": result.detach().float().clone(),
            "params_sample": _seeded_sample(params),
            "grads_sample": _seeded_sample([p.grad for p in params])}


def _write_outputs(out_dir, arrays):
    """DIR/<name>.npy per array, float32."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def _other_kernel_rooflines(mel, net, wave, B, ntok, peaks):
    """mel_kernel against the HBM roofline (algorithmic 1.792 MB per 10 s clip) and the attention kernels against the
    tensor roofline (4 / 10 N^2 d flops per clip and head), each timed alone: 3 warm-up + 20 launches.  `traffic` =
    dram bytes per launch from the committed ncu --set full captures of the same launches (profiles/)."""
    from passt_b200 import _lib as L

    def avg_ms(fn, n=20):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    out = {}
    was_training = mel.training
    mel.eval()                       # fixed band, no SpecAugment draws: the launch is the mel kernel alone
    with torch.no_grad():
        ms = avg_ms(lambda: mel(wave))
    mel.train(was_training)
    T = 1 + (wave.shape[1] - 1) // 320
    mel_bytes = B * (wave.shape[1] * 4 + 128 * T * 4)
    gbs = mel_bytes / (ms * 1e-3) / 1e9
    out["mel_kernel"] = {"bound": "hbm", "ms": ms, "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": gbs / peaks["hbm_gbs"], "traffic": NCU_TRAFFIC.get("mel_kernel")}
    H, hd = net.num_heads, net.embed_dim // net.num_heads
    C = H * hd
    dev = wave.device
    qkv = torch.randn(B, ntok, 3 * C, device=dev).bfloat16()
    o = torch.empty(B, ntok, C, device=dev, dtype=torch.bfloat16)
    npad = ((ntok + 127) // 128) * 128
    lse = torch.empty(B, H, npad, device=dev)
    scale = hd ** -0.5
    ms_f = avg_ms(lambda: L.call("passt_attn_fwd", L.ptr(qkv), L.ptr(o), L.ptr(lse), B, ntok, H, scale, L.stream_ptr()))
    peak = peaks["bf16_sustained"]
    items = [("attn_fwd_kernel", ms_f, 4.0)]
    if net.training:
        dO = torch.randn(B, ntok, C, device=dev).bfloat16()
        dqkv = torch.empty_like(qkv)
        ws = torch.empty(L.load().passt_attn_bwd_workspace_bytes(B, ntok, H), dtype=torch.uint8, device=dev)
        ms_b = avg_ms(lambda: L.call("passt_attn_bwd", L.ptr(qkv), L.ptr(o), L.ptr(dO), L.ptr(lse), L.ptr(dqkv), None,
                                     L.ptr(ws), B, ntok, H, scale, L.stream_ptr()))
        items.append(("attn_bwd (D pre-pass + kernel + dQ pack)", ms_b, 10.0))
    for name, ms, k in items:
        tf = k * B * H * ntok * ntok * hd / (ms * 1e-3) / 1e12
        out[name] = {"bound": "tensor", "ms": ms, "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
                     "traffic": NCU_TRAFFIC.get(name.split(" ")[0])}
    return out


# dram__bytes_read.sum + dram__bytes_write.sum per launch at the cfg2 shape, from the committed ncu --set full
# summaries under profiles/ (filled in when a capture is committed; None = no capture of the current kernel version)
NCU_TRAFFIC = {
    # profiles/r2_ncu_kernels_v1.txt (64 clips, N = 474): dram read + write bytes of ONE launch
    "mel_kernel": 82.47e6 + 9.84e6,                 # algorithmic 114.7 MB (part of the 32.8 MB output is still in L2)
    "attn_fwd_kernel": 139.85e6 + 25.77e6,          # qkv read once (139.8 MB) + 46.6 MB output (partly L2-resident)
    "attn_bwd": 282.85e6 + 138.63e6 + 93.21e6 + 4.06e6 + 93.21e6 + 17.38e6,   # main kernel + D pre-pass + dQ pack
}


_REAL_STDOUT_FD = None


def _quiet_stdout():
    """Everything except the one JSON line goes to stderr -- including what C libraries write to fd 1 (NCCL prints
    its version banner there, the reference frontend prints its FMAX notice)."""
    global _REAL_STDOUT_FD
    sys.stdout.flush()
    _REAL_STDOUT_FD = os.dup(1)
    os.dup2(2, 1)


def _emit(line):
    sys.stdout.flush()
    if _REAL_STDOUT_FD is not None:
        os.write(_REAL_STDOUT_FD, (json.dumps(line) + "\n").encode())
    else:
        print(json.dumps(line), flush=True)


def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="candidate", choices=["candidate", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS),
                    help="BASELINE.json configuration (default cfg2 = the headline metric's)")
    ap.add_argument("--batch", type=int, default=0, help="clips per GPU (default: the configuration's)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"],
                    help="bf16: tensor-core tier (default); fp32: 3xbf16-split GEMMs + fp32 attention (inference configs)")
    ap.add_argument("--optim", default="own", choices=["own", "torch"],
                    help="own: passt_b200.optim.FusedAdamW (default); torch: torch.optim.AdamW(fused=True)")
    ap.add_argument("--graph", type=int, default=1, help="1: replay the step as one CUDA graph (default); 0: eager")
    ap.add_argument("--stock", type=int, default=1,
                    help="1 (default, N=1 only): also time the stock PyTorch-CUDA arms in this run (stock_gpu, vs_stock)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy (float32; "
                         "train: loss and seeded samples of the updated parameters and their gradients; inference: "
                         "logits), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        from passt_b200.ddp import suggest_nccl_ctas
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # the gradient all-reduce runs next to persistent 1-CTA-per-SM kernels: give it SMs of its own
        # (passt_b200.ddp.GradAllReducer(reserve_sms=...)), as many as the overlap window needs and no more
        cfg = CONFIGS[args.config]
        if cfg["kind"] == "train" and "PASST_DDP_RESERVE" not in os.environ:
            ntok_est = {"cfg2": 474, "cfg3": 790, "cfg5": 353}.get(args.config, 474)
            bwd_s = (2.0 / 3.0) * 3 * fwd_flops_per_clip(ntok_est, cfg["depth"], cfg["n_classes"]) * \
                (args.batch or cfg["batch"]) / 750e12
            n_bytes = 4 * (86.2e6 if cfg["depth"] == 12 else 50.7e6)
            os.environ["PASST_DDP_RESERVE"] = str(suggest_nccl_ctas(int(n_bytes), world, bwd_s))
        if int(os.environ.get("PASST_DDP_RESERVE", "0")) > 0:
            os.environ.setdefault("NCCL_MAX_CTAS", os.environ["PASST_DDP_RESERVE"])
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_candidate(args, rank, local_rank, world)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
