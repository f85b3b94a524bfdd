"""Pins the oracle restatement of the reference's own code (oracle/models_ref.py <- the reference's models.py) to what that code
computes: every shipped config's hint encoder, every processor class (plain / v1 / V2 / post_add / concat_hidden / stacked chains /
scale != 1), and a whole tiny UNet with the reference's processors installed.  The reference's outputs were computed by its
models.py, imported unmodified (tests/golden/reference_import.py stands in for the ten `diffusers` names it imports), on weights
seeded through the oracle classes, and are stored in tests/golden/reference_pin.pt (tests/golden/make_reference_pin.py); the
tests rebuild the same weights and inputs and run the restatement on them.  The golden vectors of the training-step front half
(tests/golden/reference_models.pt, tests/golden/make_reference_golden.py) pin the oracle here and the CUDA path under `-m gpu`."""
import sys
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from oracle import models_ref as MR  # noqa: E402
from tests.golden import make_reference_pin as P  # noqa: E402

@pytest.fixture(autouse=True)
def _single_thread():
    """fp32 summation order of the CPU convolutions depends on the thread count / scheduling; the comparisons below are between two
    programs that issue the same torch calls, so one thread makes them reproducible to the last few ulps."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


GOLD = P.load()


def _close(have, want, tol, floor=0.0):
    """Two digests of the same tensor (shape, strided sample, fp64 norm; tests/golden/make_reference_pin.py): the sampled
    elements within tol x the largest sampled magnitude (+ floor), and the norm of the whole tensor within tol (+ floor)."""
    return (have["shape"] == want["shape"] and have["sample"].shape == want["sample"].shape
            and float((have["sample"] - want["sample"]).abs().max()) <= tol * float(want["sample"].abs().max()) + floor
            and abs(have["norm"] - want["norm"]) <= tol * want["norm"] + floor)


@pytest.mark.parametrize("name", P.CONFIGS)
def test_hint_encoder_restatement_equals_the_reference(name):
    """ControlLoRA.__init__ wiring + forward (models.py:618-835) for every shipped configs/*.json: same state-dict keys / shapes,
    same processor classes and flags, and - on the same seeded weights - the control states and parameter gradients the
    reference computed."""
    gold = GOLD["hint_encoder_outputs"][GOLD["hint_encoder"][name]]
    got = P.hint_encoder_case(MR, GOLD["configs"][name])
    assert got["keys"] == gold["keys"]
    assert got["proc_types"] == gold["proc_types"]
    assert got["proc_attrs"] == gold["proc_attrs"]
    assert got["injected"]
    assert len(got["states"]) == len(gold["states"])
    for i, (a, b) in enumerate(zip(got["states"], gold["states"])):
        assert _close(a, b, 1e-4), f"control state {i}"
    assert list(got["grads"]) == list(gold["grads"])
    for n, b in gold["grads"].items():
        a = got["grads"][n]
        if b is None:
            assert a is None, n
        else:
            assert a is not None and _close(a, b, 1e-3, 1e-9), n


@pytest.mark.parametrize("case", list(P.PROC_CASES))
def test_processor_restatement_equals_the_reference(case):
    """One processor call (models.py:118-152 / 222-287 / 357-431) on the same attention module, hidden states, text states and
    control states: output, d hidden, every parameter gradient, d control - restatement vs what the reference code computed."""
    gold = GOLD["processor"][case]
    got = P.processor_case(MR, case)
    close = lambda a, b: _close(a, b, 2e-5, 1e-8)
    assert close(got["out"], gold["out"]), "output"
    assert close(got["d_hidden"], gold["d_hidden"]), "d hidden"
    assert set(got["grads"]) == set(gold["grads"])
    for n, b in gold["grads"].items():
        assert close(got["grads"][n], b), n
    assert len(got["d_control"]) == len(gold["d_control"]) and (len(gold["d_control"]) > 0) == gold["has_control"] == got["has_control"]
    for a, b in zip(got["d_control"], gold["d_control"]):
        assert close(a, b), "d control"


@pytest.mark.parametrize("variant", list(P.UNET_VARIANTS))
def test_unet_with_reference_processors_equals_unet_with_restated_processors(variant):
    """The whole training-step front half on a tiny SD-style UNet (the UNet restatement is the same on both sides): the reference's
    ControlLoRA + processors + the wiring of train_text_to_image_control_lora.py:469-487 against oracle/models_ref.py."""
    gold = GOLD["unet"][variant]
    got = P.unet_case(MR, variant)
    assert _close(got["pred"], gold["pred"], 2e-5) and abs(got["loss"] - gold["loss"]) <= 1e-6 * abs(gold["loss"])
    assert set(got["grads"]) == set(gold["grads"]) and len(gold["grads"]) > 50
    for n, b in gold["grads"].items():
        assert _close(got["grads"][n], b, 1e-4, 1e-9), n


@pytest.mark.parametrize("case", ["v1_stacked", "v2", "post_add", "concat"])
def test_oracle_matches_the_golden_vectors_generated_by_the_reference(case):
    """Runs everywhere (no /root/reference needed): the committed vectors were computed by the reference's own models.py
    (tests/golden/make_reference_golden.py); the restatement must reproduce them from the same seeded weights and inputs."""
    from tests.golden import make_reference_golden as G

    gold = torch.load(G.OUT, weights_only=False)[case]
    got = G.run_front_half(MR, case)
    close = lambda a, b: float((a - b).abs().max()) <= 2e-5 * float(b.abs().max()) + 1e-9
    assert close(got["pred"], gold["pred"]) and close(got["loss"], gold["loss"]) and close(got["state_norms"], gold["state_norms"])
    assert all(close(a, b) for a, b in zip(got["states"], gold["states"]))
    assert got["grads"]["names"] == gold["grads"]["names"] and got["grad_norms"]["names"] == gold["grad_norms"]["names"]
    assert close(got["grads"]["flat"], gold["grads"]["flat"])
    assert float(((got["grad_norms"]["values"] - gold["grad_norms"]["values"]).abs() / gold["grad_norms"]["values"].clamp_min(1e-12)).max()) < 1e-3
