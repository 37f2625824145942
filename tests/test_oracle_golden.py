"""The oracle restatement vs. outputs of the VERBATIM reference modules (tests/golden/reference_modules.npz,
made by tests/golden/make_golden.py from a checkout of the original project)."""

import os

import pytest
import torch

from oracle import conditioning, processors, weights
from tests.golden import cases
from tests.golden.store import Golden

GOLD = Golden(os.path.join(os.path.dirname(__file__), "golden", "reference_modules.npz"))


def _close(a: torch.Tensor, name: str, atol=2e-6, rtol=1e-5):
    torch.testing.assert_close(*GOLD.pair(name, a), atol=atol, rtol=rtol)


@pytest.mark.parametrize("case", cases.PROCESSOR_CASES, ids=lambda c: c["name"])
def test_processors_match_reference(case):
    w, x, ehs = cases.processor_inputs(case)
    with torch.no_grad():
        if case["kind"] == "split":
            out = processors.split_injection_attention(w, x, ehs, case["delta_scale"])
        else:
            out = processors.ordinal_ip_attention(w, x, ehs, case["mode"])
    # fp32 sums are ordered by the CPU's thread count and vector width: up to 1.7e-5 apart on outputs of magnitude <= 23
    _close(out, "processor_" + case["name"], atol=3e-5)


def test_role_maps_bit_exact():
    names = cases.cross_attention_processor_names()
    assert [weights.role_of(n) for n in names] == list(GOLD["roles"])
    assert [processors.frequency_mode_of(n) for n in names] == list(GOLD["freq_modes"])


def test_purifier_matches_reference():
    w, img, aoe = cases.purifier_inputs()
    with torch.no_grad():
        _close(conditioning.purifier_forward(w, img, aoe), "purifier", atol=1e-5)


def test_aoe_matches_reference():
    w, labels, src = cases.aoe_inputs()
    with torch.no_grad():
        _close(conditioning.aoe_class_table(w), "aoe_table", atol=0, rtol=0)
        _close(conditioning.aoe_forward(w, labels), "aoe_forward")
        _close(conditioning.aoe_negative(w, labels), "aoe_negative")
        _close(conditioning.aoe_delta(w, src, labels), "aoe_delta")
        d = conditioning.aoe_delta(w, labels, labels)
        _close(d, "aoe_delta_same", atol=0, rtol=0)
        assert d.abs().max().item() == 0.0          # invariant I1


# ---- conditioning front end: oracle vs the real transformers CLIP tower / the verbatim reference resamplers --------------
FE = Golden(os.path.join(os.path.dirname(__file__), "golden", "front_end.npz"))


def test_clip_oracle_matches_transformers_tiny():
    from oracle import image_front_end as fe
    d, w, pixels = cases.clip_inputs("tiny")
    hidden, embeds = fe.clip_hidden_states(w, pixels, d["heads"], d["patch"])
    torch.testing.assert_close(hidden, torch.from_numpy(FE["clip_tiny_hidden"]), atol=2e-5, rtol=1e-5)
    torch.testing.assert_close(embeds, torch.from_numpy(FE["clip_tiny_embeds"]), atol=2e-5, rtol=1e-5)


def test_projection_oracles_match_reference():
    from oracle import image_front_end as fe
    hidden = cases.clip_l14_hidden()
    torch.testing.assert_close(*FE.pair("clip_l14_hidden", hidden), atol=5e-5, rtol=1e-5)      # the resampler's input
    got = fe.projection_plus(cases.projection_plus_inputs(), hidden)
    torch.testing.assert_close(*FE.pair("projection_plus", got), atol=5e-5, rtol=1e-5)
    bw, emb = cases.projection_basic_inputs()
    torch.testing.assert_close(*FE.pair("projection_basic", fe.projection_basic(bw, emb, 4, 768)), atol=2e-5, rtol=1e-5)
