#!/usr/bin/env python
"""bench.py — denoiser-steps/sec of the NaturalSpeech2 hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one `Model.forward` (the per-timestep denoiser call, ns2.py:929-1000) on the per-GPU batch of the
workload BASELINE.json quotes the metric on: configs[1] = Model(dim=512, depth=12, heads=8) unconditional,
seq=1024, batch=32, bf16 tensor-core operands, random-init weights, synthetic latents — followed by the per-sample
MSE against a fixed synthetic target and its batch mean.  With N GPUs every rank runs its own batch of 32 (weak
scaling, independent samples) and the ranks all-reduce the 4-byte scalar loss over NCCL — the only collective the
path has.  The step (every kernel launch of the forward + the loss kernels) is captured once in a CUDA graph.

Printed JSON (one line, rank 0): the base contract keys plus
  roofline      dominant kernel = the FFN causal-conv GEMM (43% of the step's FLOPs): algorithmic FLOPs per launch /
                mean launch time measured with CUDA events inside real steps, against BOTH measured bf16 peaks of
                MEASURED_PEAKS.json (burst and sustained); step-level fractions beside it
  parity        the step's own output checked in the run: the first CPU_SAMPLE_BATCH samples of the SAME inputs go
                through the reference (oracle/_ref, fp32 on the host) and are compared with the GPU prediction
  cpu_baseline  the reference's own CPU path timed on that bounded sample (N=1 only)
  e2e           the same metric with HOST buffers: pinned-host -> device copy of the step's inputs and device ->
                pinned-host copy of the full prediction inside the timed region (double-buffered on side streams)
  secondary     the other quantities BASELINE.json's metric names: RVQ Mcodes/s (configs[3], 1M frames, bit-exact
                sample check, own roofline) and the conditional denoiser (configs[2], B=16) steps/s
`--impl reference` times the reference arm: the UNMODIFIED reference (pip-installed into oracle/_ref, third-party
imports it does not need on this path stubbed) on the host cores, same metric/unit/config; rank 0 only.
`--dump-outputs DIR` writes what the last timed step computed on rank 0 as DIR/<name>.npy (see dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import types
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

CFG = dict(dim=512, depth=12, heads=8)
CFG3 = dict(dim=512, depth=12, heads=8, dim_prompt=512, condition_on_prompt=True)
BATCH, SEQ = 32, 1024
FLOPS_PER_SAMPLE = 316.37e9          # SURVEY Appendix C, analytic forward FLOPs per sample at N=1024
FLOPS_PER_SAMPLE_CFG3 = 331.97e9
FF_INNER = 1365                      # int(512 * 4 * 2 / 3)
CONV_FLOPS_PER_LAUNCH = 2.0 * BATCH * SEQ * FF_INNER * (3 * FF_INNER)   # algorithmic (unpadded) FLOPs
WORKLOAD = "configs[1]: Model(dim=512, depth=12, heads=8) unconditional, bf16 operands, seq=1024, batch=32 per GPU"
CPU_SAMPLE_BATCH = 4   # bounded sample of the 32-sample workload step for the in-run CPU legs
DUMP_ROWS = 8192       # --dump-outputs keeps this many of the 32 x 1024 prediction rows (16 MiB of the 64 MiB)


def build_config(world: int) -> dict:
    """Identical for both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "global_batch": BATCH * world, "seq_len": SEQ, "parallelism": f"dp{world}",
            "l2": "no flush needed: each step streams ~1.3 GB of activations + 0.5 GB of weights, >> 126 MB L2"}


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()), "measured (MEASURED_PEAKS.json)"
    return ({"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0},
            "fallback (B200_PROFILING.md)")


def _ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the newest committed
    `ncu --set full` capture under profiles/ (not measured in this run: ncu cannot wrap a timed run)."""
    for name in ("r02k_dominant_kernel_ncu.json", "r02_dominant_kernel_ncu.json", "r01_dominant_kernel_ncu.json"):
        p = ROOT / "profiles" / name
        if p.exists():
            d = json.loads(p.read_text())
            vals = [(l["dram_read_MB"] + l["dram_write_MB"]) * 1e6 for l in d["launches"]]
            return round(sum(vals) / len(vals)), f"committed ncu capture profiles/{name}"
    return None, "no capture committed"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        # median over the busier half of the samples = the clock under load
        sm_sorted = sorted(sm)
        return {"sm_mhz": statistics.median(sm_sorted[: max(1, len(sm_sorted) // 2 + 1)]) if sm else None,
                "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# the reference (oracle/_ref) on the host
# ------------------------------------------------------------------------------------------------------
def _host_threads() -> int:
    """CPU threads this process may really use: affinity mask, capped by the cgroup CPU quota (oversubscribing a
    quota-limited container with one thread per visible core makes the CPU baseline many times slower)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


def import_reference():
    """The unmodified reference package from oracle/_ref (`pip install --no-deps --target oracle/_ref`, see
    oracle/reference.py).  Third-party modules it imports at module scope but never touches on the denoiser path are
    stubbed (SURVEY Appendix A).  Returns the `naturalspeech2_pytorch.naturalspeech2_pytorch` module or None."""
    from oracle import reference
    ref_dir = reference.REF_DIR
    if not reference.installed():
        return None
    import torch

    def stub(name, **attrs):
        if name in sys.modules:
            return
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m

    class _SoundStream(torch.nn.Module):
        pass

    class _EncodecWrapper(torch.nn.Module):
        pass

    stub("audiolm_pytorch", SoundStream=_SoundStream, EncodecWrapper=_EncodecWrapper)
    stub("audiolm_pytorch.data", SoundDataset=object, get_dataloader=lambda *a, **k: None)
    stub("accelerate", Accelerator=object)
    stub("ema_pytorch", EMA=object)
    stub("pyworld")
    stub("inflect", engine=lambda: None)
    stub("num2words", num2words=lambda *a, **k: "")
    stub("num_to_words", num_to_word=lambda *a, **k: "")
    if str(ref_dir) not in sys.path:
        sys.path.insert(0, str(ref_dir))
    import contextlib
    import warnings
    warnings.filterwarnings("ignore", category=FutureWarning)
    try:
        with contextlib.redirect_stdout(sys.stderr):   # the reference prints at import / first call; stdout = JSON only
            from naturalspeech2_pytorch import naturalspeech2_pytorch as ns2
    except Exception as e:  # missing dependency on this box
        print(f"bench: reference import failed ({type(e).__name__}: {e}); using the oracle port", file=sys.stderr)
        return None
    return ns2


class HostReference:
    """The reference denoiser on the host cores: oracle/_ref when importable (kind 'reference'), else the
    torch port of the oracle (kind 'port').  Same fp32 weights as the GPU model (state_dict keys are identical)."""

    def __init__(self, state_dict=None):
        import torch
        torch.set_num_threads(_host_threads())
        self.ns2 = import_reference()
        if state_dict is None:
            from naturalspeech2_pytorch_b200 import Model
            torch.manual_seed(0)
            state_dict = Model(**CFG).state_dict()
        sd = {k: v.detach().cpu().float() for k, v in state_dict.items()}
        if self.ns2 is not None:
            self.kind = "reference"
            self.model = self.ns2.Model(**CFG).eval()
            self.model.load_state_dict(sd)
            self.desc = "unmodified reference Model.forward from oracle/_ref, torch fp32 CPU"
        else:
            from oracle import denoiser_oracle, denoiser_torch_port
            self.kind = "port"
            self.P, self.cfg, self.port = sd, denoiser_oracle.ModelConfig(**CFG), denoiser_torch_port
            self.desc = "torch fp32 CPU port of the reference path (oracle/denoiser_torch_port.py)"

    def forward(self, x, t, autocast_bf16=False):
        import contextlib
        import torch
        with torch.no_grad(), contextlib.redirect_stdout(sys.stderr):
            if self.kind == "reference":
                if autocast_bf16:
                    with torch.autocast("cpu", dtype=torch.bfloat16):
                        return self.model(x, t).float()
                return self.model(x, t)
            return self.port.model_forward(self.P, self.cfg, x, t)


def cpu_legs(model, x_host, t_host, gpu_out_head):
    """In-run parity + CPU baseline on the first CPU_SAMPLE_BATCH samples of the inputs the GPU just ran."""
    import torch
    ref = HostReference(model.state_dict())
    xs, ts = x_host[:CPU_SAMPLE_BATCH].clone(), t_host[:CPU_SAMPLE_BATCH].clone()
    t0 = time.perf_counter()
    out32 = ref.forward(xs, ts)   # warm-up (thread pool, page faults) — also the parity ground truth
    best = time.perf_counter() - t0
    for _ in range(2 if best < 15.0 else 0):
        t0 = time.perf_counter()
        ref.forward(xs, ts)
        best = min(best, time.perf_counter() - t0)
    got = gpu_out_head.double()
    d = (got - out32.double()).abs()
    parity = {"checked_samples": CPU_SAMPLE_BATCH, "against": ref.desc, "isfinite": bool(torch.isfinite(got).all()),
              "max_abs": float(d.max()), "rms": float(d.pow(2).mean().sqrt()), "out_std": float(out32.std()),
              "allclose_rtol1e-3_atol1e-5_frac": float(torch.isclose(got, out32.double(), rtol=1e-3, atol=1e-5)
                                                       .double().mean())}
    if ref.kind == "reference":   # the reference's own reduced-precision mode on the same inputs, for scale
        o16 = ref.forward(xs, ts, autocast_bf16=True)
        d16 = (o16.double() - out32.double()).abs()
        parity["ref_bf16_max_abs"] = float(d16.max())
        parity["ref_bf16_rms"] = float(d16.pow(2).mean().sqrt())
        parity["ref_bf16_allclose_frac"] = float(torch.isclose(o16.double(), out32.double(), rtol=1e-3, atol=1e-5)
                                                 .double().mean())
    parity["ok"] = bool(parity["isfinite"] and parity["max_abs"] < 1e-1 and parity["rms"] < 2e-2)
    base = {"value": round(CPU_SAMPLE_BATCH / (best * BATCH), 5), "unit": "steps/s", "cores": _host_threads(),
            "kind": ref.kind,
            "sample": f"{ref.desc}: batch {CPU_SAMPLE_BATCH} x seq 1024 of the 32-sample step in {best:.2f} s "
                      f"(same inputs as the GPU step), scaled x{BATCH // CPU_SAMPLE_BATCH}"}
    return parity, base


# ------------------------------------------------------------------------------------------------------
# secondary quantities of the BASELINE metric (rank 0, N=1)
# ------------------------------------------------------------------------------------------------------
def secondary_rvq(dev, peaks):
    """configs[3]: 8 quantizers x codebook 1024 x dim 128, 1M frames.  Mcodes/s + roofline + bit-exact sample."""
    import numpy as np
    import torch
    from naturalspeech2_pytorch_b200 import EncodecRVQ
    from oracle import rvq_oracle
    F, Q, K = 1 << 20, 8, 1024
    cb = torch.randn(Q, K, 128, generator=torch.Generator().manual_seed(1234))
    codec = EncodecRVQ(cb).to(dev)
    x = torch.randn(F, 128, generator=torch.Generator().manual_seed(1235)).to(dev)
    codes, _ = codec.quantize(x)
    torch.cuda.synchronize()
    from naturalspeech2_pytorch_b200 import ops
    prep = codec._prep()
    out = torch.empty(F, Q, device=dev, dtype=torch.int64)
    for _ in range(2):
        ops.rvq_encode(x, codec.codebooks, prep, codes=out)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 5
    e0.record()
    for _ in range(iters):
        ops.rvq_encode(x, codec.codebooks, prep, codes=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    idx = torch.randperm(F, generator=torch.Generator().manual_seed(0))[:4096]
    ref = rvq_oracle.encode(x[idx.to(dev)].cpu().numpy(), cb.numpy())
    rows_diff = int((out[idx.to(dev)].cpu().numpy() != ref).any(axis=1).sum())
    flops = 2.0 * F * Q * K * 128
    burst = float(peaks.get("bf16_tflops", 1590.0))
    return {"metric": "RVQ Mcodes/sec", "value": round(F * Q / (ms * 1e-3) / 1e6, 1), "unit": "Mcodes/s",
            "workload": "configs[3]: 8 quantizers x 1024 codes x dim 128, 1,048,576 frames, exact (bit-exact) indices",
            "ms_per_launch": round(ms, 3), "bit_exact_rows_diff_of_4096": rows_diff,
            "roofline": {"bound": "tensor", "achieved": round(flops / (ms * 1e-3) / 1e12, 1), "peak": burst,
                         "unit": "TFLOP/s", "frac": round(flops / (ms * 1e-3) / 1e12 / burst, 4),
                         "note": "fp16 tcgen05 distance filter + exact re-score; algorithmic 2*F*Q*K*d FLOPs vs "
                                 "burst bf16 peak (kernel timed alone)"}}


def secondary_cfg3(dev, peaks):
    """configs[2]: conditional Model (Perceiver cross-attention), B=16: steps/s recomputing / caching conditioning."""
    import torch
    from naturalspeech2_pytorch_b200 import Model
    torch.manual_seed(0)
    B = 16
    model = Model(**CFG3).to(dev).eval()
    model.packed()
    model.freeze_packed = True
    g = torch.Generator().manual_seed(7)
    x = torch.randn(B, SEQ, 512, generator=g).to(dev)
    t = torch.rand(B, generator=g).to(dev)
    prompt = torch.randn(B, 103, 512, generator=g).to(dev)
    cond = torch.randn(B, 512, SEQ, generator=g).to(dev)

    def timeit(fn, n=10):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    ms_full = timeit(lambda: model(x, t, prompt=prompt, cond=cond, cond_drop_prob=0.))
    cached = model.precompute_conditioning(prompt, cond, SEQ)
    model.use_cuda_graphs = True
    ms_cached = timeit(lambda: model(x, t, cond_drop_prob=0., _conditioning=cached))
    finite = bool(torch.isfinite(model(x, t, cond_drop_prob=0., _conditioning=cached)).all())
    sus = float(peaks.get("bf16_tflops_sustained", 1400.0))
    tf = FLOPS_PER_SAMPLE_CFG3 * B / (ms_cached * 1e-3) / 1e12
    del model
    torch.cuda.empty_cache()
    return {"metric": "denoiser-steps/sec", "unit": "steps/s",
            "workload": "configs[2]: Model(dim=512, depth=12, dim_prompt=512, condition_on_prompt=True), prompt "
                        "(16,103,512), cond (16,512,1024), batch=16",
            "value": round(1e3 / ms_cached, 2), "value_recomputing_conditioning": round(1e3 / ms_full, 2),
            "ms_per_step": round(ms_cached, 4), "isfinite": finite, "step_tflops": round(tf, 1),
            "step_frac_of_sustained_peak": round(tf / sus, 4)}


def secondary_aligner(dev, peaks):
    """SURVEY f4: `maximum_path` (aligner.py:88-122) at configs[4] scale — 32 samples x 100 phonemes x 1024 mel frames.
    GPU time of the two kernels, the reference's own function on the host cores beside it, bit-exact check."""
    import numpy as np
    import torch
    from naturalspeech2_pytorch_b200 import ops
    b, t_x, t_y = 32, 100, 1024
    g = torch.Generator().manual_seed(77)
    value = torch.randn(b, t_y, t_x, generator=g).mul(2).softmax(-1).transpose(1, 2).contiguous()
    x_lens = torch.randint(20, t_x + 1, (b,), generator=g)
    y_lens = torch.randint(4 * t_x, t_y + 1, (b,), generator=g)
    mask = ((torch.arange(t_x)[None, :, None] < x_lens[:, None, None])
            & (torch.arange(t_y)[None, None, :] < y_lens[:, None, None])).float()
    vd, md = value.to(dev), mask.to(dev)
    for _ in range(3):
        idx, path = ops.maximum_path(vd, md)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 20
    e0.record()
    for _ in range(iters):
        idx, path = ops.maximum_path(vd, md)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    out = {"metric": "alignments/sec", "unit": "alignments/s", "value": round(b / (ms * 1e-3), 1),
           "ms_per_call": round(ms, 4),
           "workload": "maximum_path (monotonic alignment search), value/mask (32, 100, 1024) fp32, dense path out",
           "roofline": {"bound": "latency (serial recursion over the 1024 frames, one CTA per sample); HBM for the "
                                 "expansion kernel",
                        "algorithmic_bytes": 3 * b * t_x * t_y * 4,
                        "achieved_GBps": round(3 * b * t_x * t_y * 4 / (ms * 1e-3) / 1e9, 1),
                        "peak_GBps": float(peaks.get("hbm_gbs", 6650.0))}}
    try:
        if import_reference() is None:
            raise RuntimeError("oracle/_ref is not present")
        import time
        from naturalspeech2_pytorch.aligner import maximum_path as ref_mas
        torch.set_num_threads(_host_threads())
        t0 = time.perf_counter()
        ref = ref_mas(value, mask)
        cpu_s = time.perf_counter() - t0
        out["bit_exact_vs_reference"] = bool(torch.equal(ref, path.cpu()))
        out["cpu_reference"] = {"value": round(b / cpu_s, 1), "unit": "alignments/s", "cores": _host_threads(),
                                "kind": "reference", "sample": f"the same 32 alignments, one call, {cpu_s:.3f} s"}
    except Exception as e:
        from oracle import aligner_oracle
        ref = aligner_oracle.maximum_path(value[:4].numpy(), mask[:4].numpy())
        out["bit_exact_vs_oracle_4_samples"] = bool(np.array_equal(ref, path[:4].cpu().numpy()))
        out["cpu_reference"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def secondary_prompt_encoder(dev, peaks):
    """SURVEY f3: SpeechPromptEncoder (ns2.py:289-341, default dims: 8 k=9 convs up to 2048 channels + 6-layer
    transformer) on the configs[2] prompt batch (16, 103, 128-d codec latents).  Once-per-sample work ahead of the
    denoiser loop; the reference module on the host cores is timed beside it on 2 of the 16 prompts."""
    import time
    import torch
    from naturalspeech2_pytorch_b200.encoders import SpeechPromptEncoder
    B, Np, Dc = 16, 103, 128
    torch.manual_seed(0)
    enc = SpeechPromptEncoder(dim_codebook=Dc).to(dev).eval()
    x_host = torch.randn(B, Np, Dc, generator=torch.Generator().manual_seed(5))
    x = x_host.to(dev)
    for _ in range(3):
        y = enc(x)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 10
    e0.record()
    for _ in range(iters):
        y = enc(x)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    dims = [Dc, 256, 2048, 2048, 2048, 2048, 512, 512, 512]
    conv_flops = 2.0 * Np * 9 * sum(a * b for a, b in zip(dims[:-1], dims[1:]))
    D, Di, depth = 512, 1365, 6
    tr_flops = depth * (2.0 * Np * D * 3 * D + 4.0 * Np * Np * D + 2.0 * Np * D * D + 2.0 * Np * D * 2 * Di + 2.0 * Np * Di * D)
    flops = B * (conv_flops + tr_flops)
    burst = float(peaks.get("bf16_tflops", 1590.0))
    out = {"metric": "prompts/sec", "unit": "prompts/s", "value": round(B / (ms * 1e-3), 1), "ms_per_batch": round(ms, 4),
           "workload": "SpeechPromptEncoder(dim_codebook=128) default dims, prompt batch (16, 103, 128), forward only",
           "isfinite": bool(torch.isfinite(y).all()),
           "roofline": {"bound": "tensor", "achieved": round(flops / (ms * 1e-3) / 1e12, 1), "peak": burst,
                        "unit": "TFLOP/s", "frac": round(flops / (ms * 1e-3) / 1e12 / burst, 4),
                        "flops_per_prompt": conv_flops + tr_flops,
                        "note": "103 of the 128 rows of every tile are real positions (one M tile per prompt)"}}
    try:
        ns2 = import_reference()
        if ns2 is None:
            raise RuntimeError("oracle/_ref is not present")
        torch.set_num_threads(_host_threads())
        ref = ns2.SpeechPromptEncoder(dim_codebook=Dc).eval()
        ref.load_state_dict(enc.state_dict())
        with torch.no_grad():
            ref(x_host[:2])
            t0 = time.perf_counter()
            yr = ref(x_host[:2])
            cpu_s = time.perf_counter() - t0
        d = (y[:2].cpu() - yr).abs()
        out["parity_vs_reference_fp32"] = {"max_abs": float(d.max()), "rms": float(d.pow(2).mean().sqrt()),
                                            "out_std": float(yr.std())}
        out["cpu_reference"] = {"value": round(2 / cpu_s, 2), "unit": "prompts/s", "cores": _host_threads(),
                                "kind": "reference", "sample": f"2 of the 16 prompts, one call, {cpu_s:.3f} s"}
    except Exception as e:
        out["cpu_reference"] = {"error": f"{type(e).__name__}: {e}"}
    del enc
    torch.cuda.empty_cache()
    return out


def train_step_dp(dev, world, peaks, steps=4, warmup=2):
    """configs[4]: conditioned diffusion TRAINING step (Model(512, depth 12, dim_prompt 512, condition_on_prompt) inside
    NaturalSpeech2.forward -> loss.backward() -> fused AdamW), 32 samples per GPU, data parallel: gradient all-reduce
    overlapped with the backward (parallel.GradReducer) + the scalar-loss all-reduce.  Runs on EVERY rank."""
    import torch
    import torch.distributed as dist
    from naturalspeech2_pytorch_b200 import Model, NaturalSpeech2
    from naturalspeech2_pytorch_b200.parallel import GradReducer, global_mean_loss
    rank = int(os.environ.get("RANK", "0"))
    torch.manual_seed(0)
    model = Model(**CFG3).to(dev).train()
    ns = NaturalSpeech2(model, target_sample_hz=24000)
    if world > 1:
        model.grad_reducer = GradReducer()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, fused=True)
    g = torch.Generator().manual_seed(100 + rank)
    B = BATCH
    lat = torch.randn(B, SEQ, 512, generator=g).to(dev)
    prompt = torch.randn(B, 103, 512, generator=g).to(dev)
    cond = torch.randn(B, 512, SEQ, generator=g).to(dev)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = ns(lat, prompt_enc=prompt, cond=cond)
        loss.backward()
        opt.step()
        return global_mean_loss(loss.detach(), B)

    for _ in range(warmup):
        step()
    if world > 1:
        dist.barrier(device_ids=[dev.index])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    nbytes = model.grad_reducer.bytes_reduced // max(1, steps + warmup) if world > 1 else 0
    flops = 3 * FLOPS_PER_SAMPLE_CFG3 * B * world
    sus = float(peaks.get("bf16_tflops_sustained", 1400.0))
    res = {"metric": "train-steps/sec", "unit": "steps/s", "value": round(1e3 / ms, 3), "ms_per_step": round(ms, 3),
           "workload": "configs[4]: conditioned diffusion training step (cfg3 model, fwd + hand-written bwd + fused AdamW), "
                       f"32 samples per GPU, global batch {B * world}, gradient all-reduce overlapped with the backward",
           "n_gpus": world, "global_batch": B * world, "samples_per_s": round(B * world * 1e3 / ms, 1),
           "loss": round(float(loss), 5), "grad_allreduce_bytes_per_step": int(nbytes),
           "tflops_3x_forward": round(flops / (ms * 1e-3) / 1e12, 1),
           "frac_of_sustained_peak_per_gpu": round(flops / world / (ms * 1e-3) / 1e12 / sus, 4)}
    del opt, ns, model
    torch.cuda.empty_cache()
    return res


def dump_outputs(out_dir, pred, loss_rows, loss):
    """What one step of the timed path returns to its caller, as float32 `out_dir/<name>.npy`: `pred` = DUMP_ROWS
    (sample, position) rows of the (32, 1024, 512) prediction, drawn with a fixed seed and kept in ascending flat row
    order (DUMP_ROWS, 512); `loss_rows` = the per-sample MSE (32,); `loss` = the batch-mean loss ().  The inputs are
    seeded too, so runs with the same arguments can be compared file by file across builds."""
    import numpy as np
    import torch
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    rows = torch.randperm(pred.shape[0] * pred.shape[1], generator=torch.Generator().manual_seed(0))[:DUMP_ROWS]
    rows = rows.sort().values.to(pred.device)
    for name, t in (("pred", pred.reshape(-1, pred.shape[-1])[rows]), ("loss_rows", loss_rows), ("loss", loss)):
        np.save(out_dir / f"{name}.npy", t.detach().float().cpu().numpy())


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from naturalspeech2_pytorch_b200 import Model, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=300))

    torch.manual_seed(0)
    model = Model(**CFG).to(dev).eval()
    model.packed()
    model.freeze_packed = True
    g = torch.Generator(device="cpu").manual_seed(1 + rank)
    x_host = torch.randn(BATCH, SEQ, CFG["dim"], generator=g).pin_memory()
    t_host = torch.rand(BATCH, generator=g).pin_memory()
    x = x_host.to(dev)
    times = t_host.to(dev)
    target = torch.randn(BATCH, SEQ, CFG["dim"], device=dev)
    loss_rows = torch.empty(BATCH, device=dev)
    mse_scratch = torch.empty(BATCH * 64, device=dev)
    losses = [torch.zeros((), device=dev) for _ in range(2)]   # ping-pong: the all-reduce of step i overlaps step i+1

    def step_eager(slot=0):
        out = model(x, times, out=pred)
        ops.mse_rows(out, target, loss_rows, mse_scratch, mean_out=losses[slot])
        return out

    pred = torch.empty(BATCH, SEQ, CFG["dim"], device=dev)
    for _ in range(2):
        step_eager()
    torch.cuda.synchronize()
    l0 = ops.launch_count()
    step_eager()
    torch.cuda.synchronize()
    launches_per_step = ops.launch_count() - l0

    # the step = forward + per-sample MSE + batch mean, captured once per loss slot
    graphs = None
    if not args.no_cuda_graphs:
        graphs = []
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step_eager()
        torch.cuda.current_stream().wait_stream(side)
        for slot in range(2):
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr, capture_error_mode="thread_local"):
                step_eager(slot)
            graphs.append(gr)

    pending = [None, None]

    def step(i):
        slot = i & 1
        if pending[slot] is not None:
            pending[slot].wait()       # the loss slot is free again (stream-side wait, no host sync)
            pending[slot] = None
        if graphs is not None:
            graphs[slot].replay()
        else:
            step_eager(slot)
        if world > 1:   # the path's only collective: 4-byte scalar loss (SUM; mean = / world), off the critical path
            pending[slot] = dist.all_reduce(losses[slot], async_op=True)

    def drain():
        for s in range(2):
            if pending[s] is not None:
                pending[s].wait()
                pending[s] = None

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for i in range(warm):
        step(i)
    drain()
    barrier()

    # ------------------------------- timed region: K steps, device-resident inputs -------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        step(i)
    drain()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    t_ms = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_total = float(t_ms.item())
    ms_per_step = ms_total / args.steps
    value = world * args.steps / (ms_total / 1e3)
    gpu_head = pred[:CPU_SAMPLE_BATCH].float().cpu()
    loss_value = float(losses[(args.steps - 1) & 1].item()) / world
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pred, loss_rows, losses[(args.steps - 1) & 1] / world)

    # ------------------------------- e2e: host buffers in, host buffers out --------------------------
    model.use_cuda_graphs = not args.no_cuda_graphs   # the public API call replays the model's own captured graph
    out_host = [torch.empty(BATCH, SEQ, CFG["dim"]).pin_memory() for _ in range(2)]
    x_dev = [torch.empty_like(x) for _ in range(2)]
    t_dev = [torch.empty_like(times) for _ in range(2)]
    o_dev = [torch.empty_like(x) for _ in range(2)]
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    main = torch.cuda.current_stream()

    def e2e_loop(n):
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_free = [torch.cuda.Event() for _ in range(2)]
        ev_done = [torch.cuda.Event() for _ in range(2)]
        ev_out = [torch.cuda.Event() for _ in range(2)]
        for i in range(n):
            b = i & 1
            with torch.cuda.stream(s_in):           # H2D of this step's inputs (pinned host memory)
                if i >= 2:
                    s_in.wait_event(ev_free[b])
                x_dev[b].copy_(x_host, non_blocking=True)
                t_dev[b].copy_(t_host, non_blocking=True)
                ev_in[b].record(s_in)
            main.wait_event(ev_in[b])
            if i >= 2:
                main.wait_event(ev_out[b])          # o_dev[b] has been drained to the host
            model(x_dev[b], t_dev[b], out=o_dev[b])  # the public API call
            ev_free[b].record(main)
            ev_done[b].record(main)
            with torch.cuda.stream(s_out):          # D2H of the step's full prediction
                s_out.wait_event(ev_done[b])
                out_host[b].copy_(o_dev[b], non_blocking=True)
                ev_out[b].record(s_out)
        s_out.synchronize()

    e2e_loop(3)
    barrier()
    w0 = time.perf_counter()
    e2e_loop(args.steps)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - w0
    t_e = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = world * args.steps / float(t_e.item())
    h2d = x_host.numel() * 4 + t_host.numel() * 4
    d2h = out_host[0].numel() * 4
    model.use_cuda_graphs = False

    # ------------------------------- configs[4]: data-parallel training step (all ranks) -------------
    secondary = {}
    if not args.no_secondary:
        try:
            secondary["train_cfg5"] = train_step_dp(dev, world, _peaks()[0])
        except Exception as e:  # a secondary number must never take the headline line down
            secondary["train_cfg5"] = {"error": f"{type(e).__name__}: {e}"}
        barrier()

    # ------------------------------- roofline: the FFN conv GEMM inside real steps -------------------
    roof = parity = cpu_base = None
    if rank == 0:
        model._prof = []
        for _ in range(3):
            model(x, times, out=pred)  # rank-local: no collective here (the other ranks have left the step loop)
        torch.cuda.synchronize()
        by_name = {}
        for (name, a, b) in model._prof:
            by_name.setdefault(name, []).append(a.elapsed_time(b))
        model._prof = None
        conv_mean = statistics.mean(by_name["ff_conv"])
        peaks, peak_src = _peaks()
        burst = float(peaks.get("bf16_tflops", 1590.0))
        sus = float(peaks.get("bf16_tflops_sustained", burst))
        achieved = CONV_FLOPS_PER_LAUNCH / (conv_mean * 1e-3) / 1e12
        step_tf = FLOPS_PER_SAMPLE * BATCH / (ms_per_step * 1e-3) / 1e12
        traffic, traffic_src = _ncu_traffic()
        roof = {"bound": "tensor",
                "kernel": "ns2::gemm2_kernel<256,1,NS2_EPI_BF16> (CTA-pair tcgen05 GEMM; FFN causal conv k=3 as 3 "
                          "shifted-row segments)",
                "achieved": round(achieved, 1), "peak": burst, "unit": "TFLOP/s", "frac": round(achieved / burst, 4),
                "frac_burst": round(achieved / burst, 4), "frac_sustained": round(achieved / sus, 4),
                "peak_burst": burst, "peak_sustained": sus, "peak_source": peak_src,
                "flops_per_launch": CONV_FLOPS_PER_LAUNCH, "ms_per_launch": round(conv_mean, 4),
                "traffic": traffic, "traffic_source": traffic_src,
                "step_tflops": round(step_tf, 1), "step_frac_burst": round(step_tf / burst, 4),
                "step_frac_sustained": round(step_tf / sus, 4),
                "per_op_ms_per_step": {k: round(sum(v) / 3, 4) for k, v in sorted(by_name.items())},
                "per_op_note": "eager profiling pass with a CUDA-event pair around every launch: the sum exceeds "
                               "ms_per_step (graph replay) by the event overhead"}
        if world == 1 and not args.no_cpu_baseline:
            parity, cpu_base = cpu_legs(model, x_host, t_host, gpu_head)
        if world == 1 and not args.no_secondary:
            del model
            torch.cuda.empty_cache()
            for name, fn in (("rvq", secondary_rvq), ("cfg3", secondary_cfg3), ("aligner_mas", secondary_aligner),
                             ("prompt_encoder", secondary_prompt_encoder)):
                try:
                    secondary[name] = fn(dev, peaks)
                except Exception as e:  # a secondary number must never take the headline line down
                    secondary[name] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        cfg = build_config(world)
        line = {
            "metric": "denoiser-steps/sec", "value": round(value, 3), "unit": "steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": round(ms_per_step, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": cfg, "sample_steps_per_s": round(value * BATCH, 1), "loss": round(loss_value, 6),
            "clocks": clocks, "gpu_launches": int(launches_per_step * args.steps),
            "e2e": {"value": round(e2e_value, 3), "unit": "steps/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h},
            "roofline": roof, "parity": parity, "cpu_baseline": cpu_base, "secondary": secondary or None,
        }
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------
# reference arm
# ------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own CPU implementation of the path on the host cores (rank 0 only).  Each timed step is a
    bounded sample of the workload step: the largest batch b in {32,16,8,4,2} for which W+K steps fit ~150 s;
    the value is scaled by b/32 (stated in `cpu_baseline.sample`, `extrapolated`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    ref = HostReference()
    g = torch.Generator().manual_seed(1)
    x_all = torch.randn(BATCH, SEQ, CFG["dim"], generator=g)
    t_all = torch.rand(BATCH, generator=g)
    ref.forward(x_all[:2], t_all[:2])            # thread pool / page faults
    t0 = time.perf_counter()
    ref.forward(x_all[:2], t_all[:2])
    t2 = time.perf_counter() - t0
    warm = max(1, min(args.warmup, 3))
    b = 2
    for cand in (32, 16, 8, 4):
        if cand <= args.ref_max_batch and (args.steps + warm) * t2 * cand / 2 <= 150.0:
            b = cand
            break
    xs, ts = x_all[:b], t_all[:b]
    for _ in range(warm):
        ref.forward(xs, ts)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ref.forward(xs, ts)
    dt = (time.perf_counter() - t0) / args.steps
    value = b / (dt * BATCH)
    full_step_s = None
    if b < BATCH <= args.ref_max_batch and t2 * BATCH / 2 <= 60.0:     # one complete 32-sample step as a linearity check
        t0 = time.perf_counter()
        ref.forward(x_all, t_all)
        full_step_s = time.perf_counter() - t0
    sample = (f"{ref.desc}, {_host_threads()} host threads: batch {b} x seq 1024 per timed step ({dt:.2f} s)"
              + ("" if b == BATCH else f", scaled x{BATCH // b} to the 32-sample workload step")
              + (f"; one full 32-sample step measured once: {full_step_s:.2f} s" if full_step_s else ""))
    line = {"impl": "reference", "metric": "denoiser-steps/sec", "value": round(value, 5), "unit": "steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": warm,
            "ms_per_step": round(dt * BATCH / b * 1e3, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": build_config(args.gpus), "extrapolated": b != BATCH, "sample_batch": b,
            "full_step_s": round(full_step_s, 3) if full_step_s else None,
            "cpu_baseline": {"value": round(value, 5), "unit": "steps/s", "cores": _host_threads(),
                             "kind": ref.kind, "sample": sample},
            "e2e": {"value": round(value, 5), "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


_REAL_STDOUT = None


def _emit(line: dict) -> None:
    """The one JSON line of the contract, on the process's original stdout."""
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-cuda-graphs", action="store_true")
    ap.add_argument("--ref-max-batch", type=int, default=BATCH,
                    help="reference arm: cap on the per-step sample batch (tests use 2)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (rank 0) to DIR/<name>.npy, float32, 16 MiB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner at the first
    # collective, the reference prints a GPU notice at import): send file descriptor 1 to stderr for the whole run and
    # keep a private handle on the real stdout for the final line.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)              # C-level writers (NCCL)
    sys.stdout = sys.stderr    # Python-level writers (the reference's import-time print)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
