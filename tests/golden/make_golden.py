#!/usr/bin/env python
"""Generate the golden fixtures in this directory from the REFERENCE implementation.

Runs only in the authoring container: it imports lucidrains/naturalspeech2-pytorch from /root/reference
(read-only) with `sys.modules` stubs for the third-party packages that are not installed (SURVEY Appendix A),
builds small `Model`s, fills their parameters with tests/param_fill.py (deterministic by state_dict key), runs
the reference forward on CPU in fp64 / fp32 / autocast-bf16, and stores inputs + outputs as .npz.  The GPU box
never sees /root/reference; it only reads the committed fixtures.

    python tests/golden/make_golden.py
"""
from __future__ import annotations

import contextlib
import inspect
import sys
import types
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from param_fill import fill_module, seeded, seeded_uniform  # noqa: E402


def import_reference(path="/root/reference"):
    """Stub the seven missing third-party modules, then import the reference package."""
    def stub(name, **attrs):
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

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
    sys.path.insert(0, path)
    import naturalspeech2_pytorch  # noqa: F401
    from naturalspeech2_pytorch import naturalspeech2_pytorch as ns2
    return ns2


CASES = {
    # name: (model kwargs, B, N, prompt_len, cond_len)
    "uncond_small": (dict(dim=128, depth=2, heads=2, wavenet_layers=3, wavenet_stacks=2), 2, 160, None, None),
    "cond_small": (dict(dim=128, depth=2, heads=2, wavenet_layers=3, wavenet_stacks=2, dim_prompt=192,
                        condition_on_prompt=True, resampler_depth=1), 2, 160, 40, 150),
    "cond_samedim": (dict(dim=128, depth=1, heads=4, wavenet_layers=2, wavenet_stacks=2, dim_prompt=128,
                          condition_on_prompt=True, resampler_depth=2, num_latents_m=16), 3, 130, 25, 200),
    "readme_uncond": (dict(dim=128, depth=6), 1, 1024, None, None),
}

# Slices of the BENCHMARKED configurations (BASELINE.json configs[1] / configs[2]: dim 512, heads 8, seq 1024) at
# depth 2, batch 2: the same kernel instantiations, tile schedules and packed layouts as the bench shapes run here,
# chained through 4 wavenet stacks + transformer layers.  Inputs are regenerated from seeds (param_fill.seeded), and
# only a row subsample of the outputs is stored (first/last 8 positions + every 8th) to keep the fixtures ~2 MB.
BIG_CASES = {
    "cfg2_slice": (dict(dim=512, depth=2, heads=8), 2, 1024, None, None),
    "cfg3_slice": (dict(dim=512, depth=2, heads=8, dim_prompt=512, condition_on_prompt=True), 2, 1024, 103, 1024),
}


def subsample_rows(N):
    rows = sorted(set(range(8)) | set(range(N - 8, N)) | set(range(0, N, 8)))
    return np.array(rows, dtype=np.int64)


def to_np(sd):
    return {k: v.detach().cpu().numpy() for k, v in sd.items()}


def run_case(ns2, name, kwargs, B, N, Np, L, big=False):
    torch.manual_seed(0)
    model = ns2.Model(**kwargs).eval()
    fill_module(model, seed=1234)
    x = seeded((B, N, kwargs["dim"]), 11)
    times = seeded_uniform((B,), 12)
    inputs = {"x": x, "times": times}
    fkw = {}
    if kwargs.get("condition_on_prompt"):
        inputs["prompt"] = seeded((B, Np, kwargs["dim_prompt"]), 13)
        inputs["cond"] = seeded((B, kwargs["dim_prompt"], L), 14)
        fkw = dict(prompt=inputs["prompt"], cond=inputs["cond"])
    out = {}
    with torch.no_grad():
        out["out_fp32"] = model(x, times, **fkw)
        m64 = ns2.Model(**kwargs).double().eval()
        m64.load_state_dict({k: v.double() for k, v in model.state_dict().items()})
        out["out_fp64"] = m64(x.double(), times.double(), **{k: v.double() for k, v in fkw.items()})
        with torch.autocast("cpu", dtype=torch.bfloat16):
            out["out_bf16_autocast"] = model(x, times, **fkw).float()
        if kwargs.get("condition_on_prompt"):
            out["out_fp64_null"] = m64(x.double(), times.double(), cond_drop_prob=1.,
                                       **{k: v.double() for k, v in fkw.items()})
            out["out_fp64_cfg3"] = m64.forward_with_cond_scale(
                x.double(), times.double(), cond_scale=3., **{k: v.double() for k, v in fkw.items()})
    e32 = (out["out_fp32"].double() - out["out_fp64"]).abs().max().item()
    e16 = (out["out_bf16_autocast"].double() - out["out_fp64"]).abs().max().item()
    print(f"{name}: params={sum(p.numel() for p in model.parameters())} out_std={out['out_fp64'].std():.3f} "
          f"|fp32-fp64|max={e32:.2e} |bf16autocast-fp64|max={e16:.2e}")
    if big:
        # whole-tensor statistics of the reference's own reduced-precision runs against its fp64 run
        ref64 = out["out_fp64"]
        arrays = {"in_seeded": np.array(1), "in_shape_x": np.array(x.shape), "rows": subsample_rows(N),
                  "out_std": np.array(ref64.std().item())}
        if kwargs.get("condition_on_prompt"):
            arrays["in_shape_prompt"] = np.array(inputs["prompt"].shape)
            arrays["in_shape_cond"] = np.array(inputs["cond"].shape)
        for k in ("out_fp32", "out_bf16_autocast"):
            d = (out[k].double() - ref64).abs()
            arrays[f"stats_{k}"] = np.array([d.max().item(), d.pow(2).mean().sqrt().item(),
                                             torch.isclose(out[k].double(), ref64, rtol=1e-3, atol=1e-5)
                                             .double().mean().item()])
        rows = torch.from_numpy(arrays["rows"])
        for k, v in out.items():
            arrays[k] = v[:, rows].numpy().astype(np.float64 if "fp64" in k else np.float32)
    else:
        arrays = {"in_" + k: v.numpy() for k, v in inputs.items()}
        for k, v in out.items():
            arrays[k] = v.numpy().astype(np.float64 if "fp64" in k else np.float32)
    arrays["config"] = np.array(repr(sorted(kwargs.items())))
    arrays["fill_seed"] = np.array(1234)
    np.savez_compressed(HERE / f"model_{name}.npz", **arrays)
    return model


def diffusion_goldens(ns2):
    """Loss with injected (times, noise) and a 4-step DDIM sample from fixed initial noise (uncond_small)."""
    kwargs, B, N, _, _ = CASES["uncond_small"]
    model = ns2.Model(**kwargs).eval()  # fp32: the wrapper draws float32 times (ns2.py:1621)
    fill_module(model, seed=1234)
    diff = ns2.NaturalSpeech2(model=model, target_sample_hz=24000, timesteps=4)
    latents = seeded((B, N, kwargs["dim"]), 21)
    # replicate ns2.py:1621-1666 with known times/noise by seeding torch's CPU generator and recording the draws
    torch.manual_seed(77)
    times = torch.zeros((B,)).float().uniform_(0, 1.)
    noise = torch.randn_like(latents)
    torch.manual_seed(77)
    with torch.no_grad():
        loss = diff(latents)
    torch.manual_seed(78)
    init = torch.randn((B, 64, kwargs["dim"]))
    torch.manual_seed(78)
    with torch.no_grad():
        sample = diff.sample(length=64, batch_size=B)
    print(f"diffusion: loss={loss.item():.6f} sample_std={sample.std():.3f}")
    extra = {}
    for obj in ("eps", "x0"):  # the other two parameterisations (ns2.py:1637-1663, 1412-1421), same weights/draws
        d2 = ns2.NaturalSpeech2(model=model, target_sample_hz=24000, timesteps=4, objective=obj)
        torch.manual_seed(77)
        with torch.no_grad():
            extra[f"loss_{obj}"] = np.array(d2(latents).item())
        torch.manual_seed(78)
        with torch.no_grad():
            extra[f"ddim_out_{obj}"] = d2.sample(length=64, batch_size=B).numpy()
        print(f"diffusion[{obj}]: loss={float(extra[f'loss_{obj}']):.6f} sample_std={extra[f'ddim_out_{obj}'].std():.3f}")
    np.savez_compressed(HERE / "diffusion_uncond_small.npz", latents=latents.numpy(), times=times.numpy(),
                        noise=noise.numpy(), loss=np.array(loss.item()), ddim_init=init.numpy(),
                        ddim_out=sample.numpy(), timesteps=np.array(4), **extra)


def gradient_goldens(ns2):
    """d(loss)/d(theta) of the reference in fp64 (golden weights, the diffusion golden's latents/times/noise; the
    conditional case adds the model golden's prompt / cond with cond_drop_prob = 0): every parameter gradient's norm
    plus a few whole tensors — what the `-m gpu` backward tests compare with."""
    keep = {
        "uncond_small": ("transformer.to_pred.1.weight", "transformer.layers.0.1.to_q.weight",
                         "transformer.layers.1.5.2.1.weight", "transformer.layers.0.5.0.bias",
                         "transformer.layers.1.4.to_gamma_beta.weight", "wavenet.init_conv.weight",
                         "wavenet.stacks.0.blocks.2.conv.weight", "wavenet.stacks.1.blocks.0.skip_conv.weight",
                         "wavenet.stacks.1.blocks.1.to_time_cond.bias", "to_time_cond.1.weight", "to_time_cond.0.weights",
                         "transformer.to_pred.0.gamma", "wavenet.final_conv.bias"),
        "cond_small": ("transformer.layers.0.3.to_kv.weight", "transformer.layers.1.3.to_q.weight",
                       "transformer.layers.0.2.to_gamma_beta.weight", "perceiver_resampler.latents",
                       "perceiver_resampler.layers.0.0.to_kv.weight", "perceiver_resampler.layers.0.1.0.weight",
                       "perceiver_resampler.proj_context.weight", "perceiver_resampler.norm.gamma",
                       "cond_to_model_dim.weight", "to_prompt_cond.1.weight", "wavenet.init_conv.weight",
                       "transformer.layers.1.1.to_kv.weight", "to_time_cond.1.weight"),
    }
    zd = np.load(HERE / "diffusion_uncond_small.npz")
    for case in ("uncond_small", "cond_small"):
        kwargs, B, N, _, _ = CASES[case]
        model = ns2.Model(**kwargs)
        fill_module(model, seed=1234)
        model = model.double()
        diff = ns2.NaturalSpeech2.__new__(ns2.NaturalSpeech2)   # only the schedule helpers are needed
        latents = torch.from_numpy(zd["latents"]).double()
        times = torch.from_numpy(zd["times"]).double()
        noise = torch.from_numpy(zd["noise"]).double()
        extra = {}
        if kwargs.get("condition_on_prompt"):
            zm = np.load(HERE / f"model_{case}.npz")
            extra = dict(prompt=torch.from_numpy(zm["in_prompt"]).double(), cond=torch.from_numpy(zm["in_cond"]).double(),
                         cond_drop_prob=0.)
        # ns2.py:1621-1666 with the recorded draws (sigmoid schedule, objective v, min-SNR-5 weight)
        gamma = ns2.sigmoid_schedule(times)
        alpha, sigma = ns2.gamma_to_alpha_sigma(gamma[:, None, None], 1.)
        noised = alpha * latents + sigma * noise
        pred = model(noised, times, **extra)
        target = alpha * noise - sigma * latents
        loss = ((pred - target) ** 2).reshape(B, -1).mean(dim=1)
        snr = (alpha * alpha) / (sigma * sigma)
        weight = snr.clamp(max=5) / (snr + 1)
        loss = (loss * weight).mean()
        loss.backward()
        out = {"loss": np.array(loss.item())}
        names, norms = [], []
        for n, p in model.named_parameters():
            names.append(n)
            g = p.grad if p.grad is not None else torch.zeros_like(p)
            norms.append(g.norm().item())
            if n in keep[case]:
                out["grad::" + n] = g.numpy().astype(np.float32)
        out["names"] = np.array(names)
        out["norms"] = np.array(norms)
        print(f"gradients[{case}]: loss={loss.item():.6f} params={len(names)} "
              f"total grad norm={np.sqrt((np.array(norms) ** 2).sum()):.4f}")
        np.savez_compressed(HERE / f"grads_{case}.npz", **out)


def rvq_goldens():
    """Codes from the HF transformers port of Encodec's residual VQ (fp32 formula) on seeded codebooks.
    Inputs are regenerated from seeds by param_fill.rvq_fixture_inputs(); only the outputs are stored."""
    from transformers import EncodecConfig
    from transformers.models.encodec.modeling_encodec import EncodecResidualVectorQuantizer
    from param_fill import rvq_fixture_inputs
    cfg = EncodecConfig()  # 24 kHz, codebook 1024 x 128
    rvq = EncodecResidualVectorQuantizer(cfg).eval()
    cb, variants = rvq_fixture_inputs()
    Q = cb.shape[0]
    assert (cfg.codebook_size, cfg.codebook_dim) == tuple(cb.shape[1:])
    with torch.no_grad():
        for q in range(Q):
            rvq.layers[q].codebook.embed.copy_(cb[q])
    out = {}
    with torch.no_grad():
        for name, fr in variants.items():
            emb = fr.t()[None]  # (1, d, F)
            bandwidth = Q * math_log2(cfg.codebook_size) * cfg.frame_rate / 1000.0
            codes = rvq.encode(emb, bandwidth=bandwidth)  # (Q, 1, F)
            assert codes.shape[0] == Q, codes.shape
            dec = rvq.decode(codes)  # (1, d, F)
            out[f"codes_{name}"] = codes[:, 0].t().contiguous().numpy().astype(np.int64)
            if name == "random":
                out[f"decoded_{name}"] = dec[0].t().contiguous().numpy()
    np.savez_compressed(HERE / "rvq_encodec.npz", **out)
    print("rvq:", {k: v.shape for k, v in out.items()})


ENCODER_CASES = {
    # name: (class name, ctor kwargs, input spec)
    # the reference annotates dims as Tuple[int] (beartype: a 1-tuple), so small stacks have ONE conv; the default
    # 8-conv stack (256, 2048 x4, 512 x3) is covered by spe_full (depth 1 to keep the fp64 run short)
    "spe_small": ("SpeechPromptEncoder", dict(dim_codebook=128, dims=(256,), depth=2, heads=4), (2, 103)),
    "spe_long": ("SpeechPromptEncoder", dict(dim_codebook=128, dims=(256,), depth=2, heads=4), (1, 300)),
    "spe_full": ("SpeechPromptEncoder", dict(dim_codebook=128, depth=1), (1, 103)),
    "phon_small": ("PhonemeEncoder", dict(num_tokens=50, dim=128, dim_hidden=128, depth=2, heads=2), (2, 37)),
    # duration / pitch predictor: input = phoneme encodings (B, T, D) and encoded prompts (B, Np, D)
    "dpp_small": ("DurationPitchPredictor", dict(dim=128, dim_hidden=128, depth=2, heads=2), (2, 37, 50)),
    "dpp_512": ("DurationPitchPredictor", dict(dim=512, depth=1), (1, 100, 103)),
}


def encoder_inputs(name, cls, kwargs, spec):
    if cls == "DurationPitchPredictor":
        B, T, Np = spec
        D = kwargs.get("dim_hidden", 512)
        return seeded((B, T, D), 23), seeded((B, Np, D), 24)
    B, T = spec
    if cls == "PhonemeEncoder":
        ids = torch.randint(0, kwargs["num_tokens"], (B, T), generator=torch.Generator().manual_seed(21))
        ids[1, T - 9:] = -1                                   # padding (ns2.py:279-280)
        return ids
    return seeded((B, T, kwargs["dim_codebook"]), 22)


def encoder_goldens(ns2):
    """SpeechPromptEncoder / PhonemeEncoder of the reference (ns2.py:228-341): fp64, fp32 and autocast-bf16 outputs."""
    out = {}
    for name, (cls, kwargs, spec) in ENCODER_CASES.items():
        torch.manual_seed(0)
        enc = getattr(ns2, cls)(**kwargs).eval()
        fill_module(enc, seed=1234)
        x = encoder_inputs(name, cls, kwargs, spec)
        if cls == "DurationPitchPredictor":
            x, pr = x
            with torch.no_grad():
                y32 = torch.stack(enc(x, pr))
                e64 = getattr(ns2, cls)(**kwargs).double().eval()
                e64.load_state_dict({k: v.double() for k, v in enc.state_dict().items()})
                y64 = torch.stack(e64(x.double(), pr.double()))
                with torch.autocast("cpu", dtype=torch.bfloat16):
                    y16 = torch.stack(enc(x, pr)).float()
            print(f"{name}: out mean={y64.mean():.3f} std={y64.std():.3f} zeros={float((y64 == 0).double().mean()):.2f} "
                  f"|fp32-fp64|max={(y32.double() - y64).abs().max():.2e} "
                  f"|bf16autocast-fp64|max={(y16.double() - y64).abs().max():.2e}")
            out[f"{name}_in"] = x.numpy()
            out[f"{name}_prompts"] = pr.numpy()
            out[f"{name}_fp64"] = y64.numpy()
            out[f"{name}_bf16_autocast"] = y16.numpy()
            out[f"{name}_keys"] = np.array(repr([(k, tuple(v.shape)) for k, v in enc.state_dict().items()]))
            continue
        with torch.no_grad():
            y32 = enc(x)
            e64 = getattr(ns2, cls)(**kwargs).double().eval()
            e64.load_state_dict({k: v.double() for k, v in enc.state_dict().items()})
            y64 = e64(x if x.dtype == torch.int64 else x.double())
            with torch.autocast("cpu", dtype=torch.bfloat16):
                y16 = enc(x).float()
        print(f"{name}: out_std={y64.std():.3f} |fp32-fp64|max={(y32.double() - y64).abs().max():.2e} "
              f"|bf16autocast-fp64|max={(y16.double() - y64).abs().max():.2e}")
        out[f"{name}_in"] = x.numpy()
        out[f"{name}_fp64"] = y64.numpy()
        out[f"{name}_bf16_autocast"] = y16.numpy()
        out[f"{name}_keys"] = np.array(repr([(k, tuple(v.shape)) for k, v in enc.state_dict().items()]))
    # length regulation (ns2.py:87-104, 164-177, 1449-1455) with the reference's own functions
    g = torch.Generator().manual_seed(31)
    ph = torch.randn(3, 21, 64, generator=g)
    dur = torch.rand(3, 21, generator=g) * 5
    dur[1, 12:] = 0
    dur[2] = dur[2] * 0.3
    pitch = torch.rand(3, 21, generator=g) * 900
    pitch[0, :4] = 0
    table = torch.randn(256, 64, generator=g)
    attn = ns2.generate_mask_from_repeats(dur).float()
    fake = types.SimpleNamespace(pitch_emb=lambda ids: table[ids.long()])
    cond = ns2.NaturalSpeech2.expand_encodings(fake, ph.transpose(1, 2), attn.unsqueeze(1), pitch.unsqueeze(1).clone())
    out.update(expand_phon=ph.numpy(), expand_duration=dur.numpy(), expand_pitch=pitch.numpy(), expand_table=table.numpy(),
               expand_cond=cond.numpy())
    print("expand:", tuple(cond.shape))
    np.savez_compressed(HERE / "encoders.npz", **out)


def aligner_cases():
    """Seeded inputs of the monotonic-alignment fixtures: name -> (value (b,t_x,t_y) f32, x_lens, y_lens)."""
    cases = {}
    g = torch.Generator().manual_seed(4321)
    # soft alignments as Aligner.forward produces them (softmax over the text axis), ragged lengths
    v = torch.randn(3, 90, 37, generator=g).mul(3).softmax(dim=-1).transpose(1, 2).contiguous()
    cases["soft_ragged"] = (v, [37, 20, 5], [90, 64, 33])
    # more text positions than frames, signed scores
    cases["tall_signed"] = (torch.randn(2, 130, 50, generator=g), [130, 77], [50, 41])
    # heavy ties: scores quantised to quarters
    cases["ties"] = (torch.randint(0, 4, (2, 70, 45), generator=g).float() / 4, [70, 33], [45, 45])
    cases["wide16"] = (torch.rand(1, 300, 40, generator=g), [300], [40])
    cases["wide32"] = (torch.rand(1, 600, 24, generator=g), [590], [23])
    cases["narrow"] = (torch.rand(2, 9, 130, generator=g), [9, 1], [130, 2])
    return cases


def aligner_masks(v, x_lens, y_lens):
    b, t_x, t_y = v.shape
    xm = (torch.arange(t_x)[None, :] < torch.tensor(x_lens)[:, None]).float()
    ym = (torch.arange(t_y)[None, :] < torch.tensor(y_lens)[:, None]).float()
    return xm[:, :, None] * ym[:, None, :]                      # attn_mask of Aligner.forward, aligner.py:208-211


def aligner_goldens():
    """maximum_path of the reference (aligner.py:88-122) on the seeded cases -> aligner_mas.npz."""
    from naturalspeech2_pytorch.aligner import maximum_path
    out = {}
    for name, (v, xl, yl) in aligner_cases().items():
        mask = aligner_masks(v, xl, yl)
        path = maximum_path(v, mask)
        assert path.dtype == torch.float32 and set(path.unique().tolist()) <= {0.0, 1.0}
        out[f"{name}_value"] = v.numpy()
        out[f"{name}_xlens"] = np.asarray(xl, dtype=np.int64)
        out[f"{name}_ylens"] = np.asarray(yl, dtype=np.int64)
        out[f"{name}_path"] = path.numpy().astype(np.uint8)
    np.savez_compressed(HERE / "aligner_mas.npz", **out)
    print("aligner:", {k: v.shape for k, v in out.items() if k.endswith("_path")})


# Drop-in surface (tests/test_dropin_cpu.py): BASELINE configs[0..2] (README model, cfg2, cfg3), a small conditional
# model and the model the patch test rebinds.  Recorded per configuration: the reference Model's state_dict keys in
# order with their shapes, and the attributes integration.infer_model_kwargs reads; plus the reference call signatures.
DROPIN_CONFIGS = {
    "cfg1_readme": dict(dim=128, depth=6),
    "cfg2": dict(dim=512, depth=12, heads=8),
    "cfg3": dict(dim=512, depth=12, dim_prompt=512, condition_on_prompt=True),
    "small_cond": dict(dim=128, depth=2, heads=2, wavenet_layers=3, wavenet_stacks=2, dim_prompt=192,
                       condition_on_prompt=True, resampler_depth=1, num_latents_m=16, cond_drop_prob=0.25),
    "patch_small": dict(dim=128, depth=1, heads=2, wavenet_layers=2, wavenet_stacks=2),
}
DROPIN_SIGNATURES = ["Model.__init__", "Model.forward", "Model.forward_with_cond_scale", "NaturalSpeech2.forward",
                     "NaturalSpeech2.sample"]


@contextlib.contextmanager
def shapes_only():
    """Skip the (slow) random initialisation of nn.Linear / nn.Conv1d weights: parameters stay torch.empty."""
    names = ("kaiming_uniform_", "uniform_", "normal_", "zeros_", "ones_", "trunc_normal_")
    saved = {n: getattr(torch.nn.init, n) for n in names}
    try:
        for n in names:
            setattr(torch.nn.init, n, lambda t, *a, **k: t)
        yield
    finally:
        for n, f in saved.items():
            setattr(torch.nn.init, n, f)


def signature_spec(fn):
    """(name, kind, repr(default)) of every parameter of `fn`."""
    return [(p.name, p.kind.name, repr(p.default)) for p in inspect.signature(fn).parameters.values()]


def dropin_goldens(ns2):
    out = {}
    for name, kwargs in DROPIN_CONFIGS.items():
        with shapes_only():
            m = ns2.Model(**kwargs)
        attrs = dict(dim=m.dim, depth=len(m.transformer.layers), heads=m.transformer.layers[0][1].heads,
                     wavenet_layers=len(m.wavenet.stacks[0].blocks), wavenet_stacks=len(m.wavenet.stacks),
                     condition_on_prompt=bool(m.condition_on_prompt), cond_drop_prob=float(m.cond_drop_prob))
        if m.condition_on_prompt:
            attrs["resampler_depth"] = len(m.perceiver_resampler.layers)
        out[f"{name}_keys"] = np.array(repr([(k, tuple(v.shape)) for k, v in m.state_dict().items()]))
        out[f"{name}_attrs"] = np.array(repr(attrs))
    for qual in DROPIN_SIGNATURES:
        cls, meth = qual.split(".")
        out[f"sig_{qual}"] = np.array(repr(signature_spec(getattr(getattr(ns2, cls), meth))))
    np.savez_compressed(HERE / "dropin_surface.npz", **out)
    print("dropin:", sorted(out))


def math_log2(v):
    import math
    return math.log2(v)


def main():
    if not sys.argv[1:] or "rvq" in sys.argv[1:]:
        rvq_goldens()  # before the stubs: transformers probes the real `accelerate` module spec
    ns2 = import_reference()
    only = sys.argv[1:]
    for name, (kwargs, B, N, Np, L) in CASES.items():
        if not only or name in only:
            run_case(ns2, name, kwargs, B, N, Np, L)
    for name, (kwargs, B, N, Np, L) in BIG_CASES.items():
        if not only or name in only:
            run_case(ns2, name, kwargs, B, N, Np, L, big=True)
    if not only or "diffusion" in only:
        diffusion_goldens(ns2)
    if not only or "grads" in only:
        gradient_goldens(ns2)
    if not only or "aligner" in only:
        aligner_goldens()
    if not only or "encoders" in only:
        encoder_goldens(ns2)
    if not only or "dropin" in only:
        dropin_goldens(ns2)


if __name__ == "__main__":
    main()
