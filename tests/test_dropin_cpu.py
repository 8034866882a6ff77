"""CPU: drop-in surface against the UNMODIFIED reference, as recorded from it in tests/golden/dropin_surface.npz
(tests/golden/make_golden.py `dropin`).

For BASELINE configs[0..2] (README model, cfg2, cfg3) and two small models: identical `state_dict` keys, order and
shapes, identical `forward` / `forward_with_cond_scale` parameter lists (the reference's parameters must all be
accepted, in the same order), and `integration.infer_model_kwargs` recovers the constructor arguments from a
reference instance.  Modules are built with the nn.init routines patched out (uninitialised storage, shapes only):
cfg3 alone has 448 M parameters.
"""
import ast
import types
from collections import OrderedDict

import numpy as np
import pytest
import torch

from golden.make_golden import DROPIN_CONFIGS, shapes_only, signature_spec
from helpers import GOLDEN

SURFACE = np.load(GOLDEN / "dropin_surface.npz")


def _golden(key):
    return ast.literal_eval(str(SURFACE[key]))


class ReferenceModel(torch.nn.Module):
    """Stand-in for a reference `Model` instance of configuration `name`: the recorded attributes that
    `infer_model_kwargs` reads, and a state_dict with the reference's keys, order and shapes (meta tensors, or
    seeded values with `values=True`)."""

    def __init__(self, name, values=False):
        super().__init__()
        a = _golden(f"{name}_attrs")
        self.dim, self.condition_on_prompt, self.cond_drop_prob = a["dim"], a["condition_on_prompt"], a["cond_drop_prob"]
        self.transformer = types.SimpleNamespace(layers=[[None, types.SimpleNamespace(heads=a["heads"])]] * a["depth"])
        self.wavenet = types.SimpleNamespace(
            stacks=[types.SimpleNamespace(blocks=[None] * a["wavenet_layers"])] * a["wavenet_stacks"])
        if a["condition_on_prompt"]:
            self.perceiver_resampler = types.SimpleNamespace(layers=[None] * a["resampler_depth"])
        g = torch.Generator().manual_seed(0)
        self._sd = OrderedDict((k, torch.randn(s, generator=g) if values else torch.empty(s, device="meta"))
                               for k, s in _golden(f"{name}_keys"))

    def state_dict(self, *args, **kwargs):
        return OrderedDict(self._sd)

    def forward(self, x, times, prompt=None, prompt_mask=None, cond=None, cond_drop_prob=None):
        return x   # the reference computation is not recorded; patch_reference replaces this method


@pytest.mark.parametrize("name", list(DROPIN_CONFIGS))
def test_state_dict_and_ctor_roundtrip(name):
    from naturalspeech2_pytorch_b200 import Model
    from naturalspeech2_pytorch_b200.integration import infer_model_kwargs
    kw = DROPIN_CONFIGS[name]
    ref = ReferenceModel(name)
    with shapes_only():
        ours = Model(**kw)
    sd_ref = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    sd_ours = {k: tuple(v.shape) for k, v in ours.state_dict().items()}
    assert sd_ref == sd_ours, (set(sd_ref) ^ set(sd_ours))
    assert list(ref.state_dict().keys()) == list(ours.state_dict().keys())   # same order, too
    got = infer_model_kwargs(ref)
    del ours
    with shapes_only():
        rebuilt = Model(**got)
    assert {k: tuple(v.shape) for k, v in rebuilt.state_dict().items()} == sd_ref
    for k, v in kw.items():
        assert got[k] == v, (k, got[k], v)


def test_call_signatures_cover_the_reference():
    from naturalspeech2_pytorch_b200 import Model, NaturalSpeech2
    ref_fwd = _golden("sig_Model.forward")
    ours_fwd = signature_spec(Model.forward)
    assert ours_fwd[:len(ref_fwd)] == ref_fwd                      # same names, order, kinds, defaults
    assert all(k == "KEYWORD_ONLY" for _, k, _ in ours_fwd[len(ref_fwd):])   # extras are opt-in
    assert signature_spec(Model.forward_with_cond_scale) == _golden("sig_Model.forward_with_cond_scale")
    ref_init = [p[0] for p in _golden("sig_Model.__init__")]
    assert [p[0] for p in signature_spec(Model.__init__)] == ref_init
    for meth in ("forward", "sample"):
        ref_p = [p[0] for p in _golden(f"sig_NaturalSpeech2.{meth}")]
        ours_p = [p[0] for p in signature_spec(getattr(NaturalSpeech2, meth))]
        assert ours_p[:len(ref_p)] == ref_p or set(ref_p) <= set(ours_p), (meth, ref_p, ours_p)


def test_patch_reference_rebinds_forward():
    """`patch_reference` on a (CPU) reference instance: the bound methods are replaced and the B200 model carries
    the reference's weights; calling it without a GPU must raise (there is no CPU fallback)."""
    from naturalspeech2_pytorch_b200.integration import patch_reference
    ref = ReferenceModel("patch_small", values=True).eval()
    fast = patch_reference(ref, device="cpu")
    for k, v in ref.state_dict().items():
        assert torch.equal(fast.state_dict()[k], v)
    assert ref.forward.__func__ is not ReferenceModel.forward
    with pytest.raises(RuntimeError):
        ref(torch.randn(1, 64, 128), torch.rand(1))
