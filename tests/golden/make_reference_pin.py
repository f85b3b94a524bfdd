"""Generates tests/golden/reference_pin.pt: the outputs of the reference's own models.py (imported unmodified through
tests/golden/reference_import.py) for every case of tests/test_reference_pin.py - each shipped config's hint encoder, each
processor class and wiring, and a tiny UNet driven by the reference's processors.

Weights are seeded through the oracle classes (the two share one state-dict layout) and loaded into the reference's classes;
inputs come from seeded generators.  A machine without the reference therefore rebuilds the same weights and inputs, runs the
oracle restatement on them and compares with the stored reference outputs.  Each tensor is stored as a fixed strided sample
(OUTPUT_SAMPLE elements of an output, GRAD_SAMPLE of a gradient) plus the norm of the whole tensor, and all samples share one flat
tensor in the file (load() restores them), which keeps the file small.

    python -m tests.golden.make_reference_pin          (needs the reference checkout, see reference_import.py)
"""
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from oracle import models_ref as MR  # noqa: E402
from oracle import unet_ref as UR  # noqa: E402

OUT = Path(__file__).resolve().parent / "reference_pin.pt"
OUTPUT_SAMPLE, GRAD_SAMPLE = 512, 64
CONFIGS = ["base", "fill50k", "diffusiondb-canny", "mpii-pose", "diffusiondb-canny-v2", "mpii-pose-v2", "post-add", "danbooru-sketch"]
PROC_ATTRS = ("hidden_size", "cross_attention_dim", "rank", "post_add", "concat_hidden", "control_self_add",
              "key_states_skipped", "value_states_skipped", "output_states_skipped")
PROC_CASES = {
    "plain_self": ("LoRACrossAttnProcessor", False, {}, None, 1.0),
    "plain_cross_post_add": ("LoRACrossAttnProcessor", True, dict(post_add=True), None, 0.7),
    "plain_skips": ("LoRACrossAttnProcessor", True, dict(key_states_skipped=True, output_states_skipped=True), None, 1.0),
    "v1_self": ("ControlLoRACrossAttnProcessor", False, {}, None, 1.0),
    "v1_cross_scale": ("ControlLoRACrossAttnProcessor", True, dict(control_rank=8), None, 0.5),
    "v1_post_add": ("ControlLoRACrossAttnProcessor", False, dict(post_add=True), None, 1.0),
    "v1_concat": ("ControlLoRACrossAttnProcessor", True, dict(concat_hidden=True, control_rank=16, control_channels=96), None, 1.0),
    "v1_stacked_pre_post": ("ControlLoRACrossAttnProcessor", True, {}, "plain", 0.5),
    "v1_stacked_control": ("ControlLoRACrossAttnProcessor", False, {}, "control", 0.8),
    "v2_self": ("ControlLoRACrossAttnProcessorV2", False, dict(control_channels=96), None, 1.0),
    "v2_cross_scale": ("ControlLoRACrossAttnProcessorV2", True, dict(control_channels=96, control_rank=8), None, 0.6),
    "v2_stacked": ("ControlLoRACrossAttnProcessorV2", False, dict(control_channels=96), "plain", 1.0),
    "v2_stacked_control": ("ControlLoRACrossAttnProcessorV2", True, dict(control_channels=96), "control", 0.9),
}
UNET_VARIANTS = {"v1": {}, "v2": dict(lora_control_version=2, lora_pre_conv_skipped=True), "post_add": dict(lora_post_add=True),
                 "concat": dict(lora_concat_hidden=True, lora_control_rank=32, lora_pre_conv_skipped=True, lora_control_self_add=False)}


def digest(t: torch.Tensor, k: int = GRAD_SAMPLE) -> dict:
    """{"shape", "sample": every element, or k elements at a fixed stride, "norm": fp64 norm of the whole tensor}."""
    f = t.detach().reshape(-1).float()
    s = f if f.numel() <= k else f[:: f.numel() // k][:k]
    return {"shape": tuple(t.shape), "sample": s.clone(), "norm": float(f.double().norm())}


def _pack(obj, chunks):
    """Replaces every digest's sample by its (offset, length) in the concatenation of `chunks`."""
    if isinstance(obj, dict) and "sample" in obj:
        off = sum(c.numel() for c in chunks)
        chunks.append(obj["sample"])
        return dict(obj, sample=(off, obj["sample"].numel()))
    if isinstance(obj, dict):
        return {k: _pack(v, chunks) for k, v in obj.items()}
    if isinstance(obj, list):
        return [_pack(v, chunks) for v in obj]
    return obj


def _unpack(obj, flat):
    if isinstance(obj, dict) and "sample" in obj:
        off, n = obj["sample"]
        return dict(obj, sample=flat[off:off + n])
    if isinstance(obj, dict):
        return {k: _unpack(v, flat) for k, v in obj.items()}
    if isinstance(obj, list):
        return [_unpack(v, flat) for v in obj]
    return obj


def load() -> dict:
    """The stored reference outputs, samples restored."""
    d = torch.load(OUT, weights_only=False)
    return _unpack(d["tree"], d["flat"])


def _randomize_(m, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith("up.weight"):
                p.copy_(0.05 * torch.randn(p.shape, generator=g))
            elif "norm" in n:
                p.add_(0.1 * torch.randn(p.shape, generator=g))


def _seeded(M, make, seed):
    """make(module) builds a model; returns M's instance carrying the oracle instance's seeded weights.  The global RNG advances
    exactly as it does for the oracle alone, whichever M is."""
    ora = make(MR)
    _randomize_(ora, seed)
    if M is MR:
        return ora
    with torch.random.fork_rng(devices=[]):
        m = make(M)
    m.load_state_dict(ora.state_dict())
    return m


def hint_encoder_case(M, cfg: dict) -> dict:
    """ControlLoRA.__init__ wiring + forward + backward (models.py:618-835) of M's class for one config."""
    torch.manual_seed(0)
    cl = _seeded(M, lambda mod: mod.ControlLoRA(**cfg), 1)
    g = torch.Generator().manual_seed(2)
    guide = torch.rand(1, 3, 64, 64, generator=g) * 2 - 1
    states = cl(guide).control_states
    ws = [torch.randn(s.shape, generator=g) for s in states]
    sum((s * w).sum() for s, w in zip(states, ws)).backward()
    return {"keys": [(k, tuple(v.shape)) for k, v in cl.state_dict().items()],
            "proc_types": [[type(p).__name__ for p in lvl] for lvl in cl.lora_layers],
            "proc_attrs": [[tuple(getattr(p, a) for a in PROC_ATTRS) for p in lvl] for lvl in cl.lora_layers],
            "states": [digest(s, OUTPUT_SAMPLE) for s in states],
            "grads": {n: (None if p.grad is None else digest(p.grad)) for n, p in cl.named_parameters()},
            # the processors of each level received that level's control states (models.py:826-829)
            "injected": all(torch.equal(p.control_states, s) for lvl, s in zip(cl.lora_layers, states) for p in lvl)}


def processor_case(M, case: str) -> dict:
    """One call of M's processor (models.py:118-152 / 222-287 / 357-431) on the oracle's attention module: output, d hidden,
    every parameter gradient, d control."""
    cls, cross, kw, stack, scale = PROC_CASES[case]
    C, XD, H = 64, 48, 4
    xd = XD if cross else None
    torch.manual_seed(3)
    attn = UR.CrossAttention(C, xd, H, C // H)
    proc = _seeded(M, lambda mod: getattr(mod, cls)(C, xd, **kw), 5)
    stacked = []
    if stack == "plain":
        a = _seeded(M, lambda mod: mod.LoRACrossAttnProcessor(C, xd, rank=2, post_add=True), 7)
        b = _seeded(M, lambda mod: mod.LoRACrossAttnProcessor(C, xd, rank=3), 8)
        proc.inject_pre_lora(a)
        proc.inject_post_lora(b)
        stacked = [a, b]
    elif stack == "control":
        a = _seeded(M, lambda mod: getattr(mod, cls)(C, xd, **kw), 9)
        proc.inject_pre_lora(a)
        stacked = [a]
    g = torch.Generator().manual_seed(11)
    hs = torch.randn(2, 36, C, generator=g)
    ehs = torch.randn(2, 9, XD, generator=g) if cross else None
    w = torch.randn(2, 36, C, generator=g)
    h = hs.clone().requires_grad_(True)
    ctrls = []
    for p in [proc] + ([s for s in stacked if hasattr(s, "inject_control_states")] if stack == "control" else []):
        if hasattr(p, "inject_control_states"):
            cc = p.to_control.down.weight.shape[1] - (C if getattr(p, "concat_hidden", False) else 0)
            c = torch.randn(2, cc, 6, 6, generator=torch.Generator().manual_seed(13 + len(ctrls))).requires_grad_(True)
            p.inject_control_states(c)
            ctrls.append(c)
    y = proc(attn, h, ehs, None, scale)
    (y * w).sum().backward()
    grads = {n: digest(p.grad) for n, p in proc.named_parameters() if p.grad is not None}
    for i, s in enumerate(stacked):
        grads.update({f"stack{i}.{n}": digest(p.grad) for n, p in s.named_parameters() if p.grad is not None})
    return {"out": digest(y, OUTPUT_SAMPLE), "d_hidden": digest(h.grad, OUTPUT_SAMPLE), "grads": grads,
            "d_control": [digest(c.grad, OUTPUT_SAMPLE) for c in ctrls],
            "has_control": hasattr(proc, "inject_control_states")}


def unet_case(M, variant: str) -> dict:
    """The training-step front half on the tiny SD-style UNet (the oracle's UNet restatement) with M's ControlLoRA and processors
    wired as in train_text_to_image_control_lora.py:469-487."""
    from tests.check_unet import TINY, TINY_LORA

    kw = dict(TINY_LORA, **UNET_VARIANTS[variant])
    torch.manual_seed(0)
    cl = _seeded(M, lambda mod: mod.ControlLoRA(**kw), 1)
    u = UR.UNet2DConditionModel(**TINY)
    UR.init_synthetic_(u, seed=1)
    u.requires_grad_(False)
    MR.wire_processors(u, cl)
    g = torch.Generator().manual_seed(4)
    guide = torch.rand(2, 3, 128, 128, generator=g) * 2 - 1
    x = torch.randn(2, 4, 16, 16, generator=g)
    ehs = torch.randn(2, 77, TINY["cross_attention_dim"], generator=g)
    tgt = torch.randn(2, 4, 16, 16, generator=g)
    cl(guide)
    pred = u(x, torch.tensor([10, 900]), ehs, cross_attention_kwargs={"scale": 0.8}).sample
    loss = torch.nn.functional.mse_loss(pred, tgt)
    loss.backward()
    return {"pred": digest(pred, OUTPUT_SAMPLE), "loss": float(loss.detach()), "grads": {n: digest(p.grad) for n, p in cl.named_parameters() if p.grad is not None}}


def main():
    from tests.golden import reference_import as RI

    torch.set_num_threads(1)
    R = RI.reference_models()
    configs = {name: RI.reference_config(name) for name in CONFIGS}
    unique = []                                  # several shipped configs are the same ControlLoRA: their outputs are stored once
    for cfg in configs.values():
        if cfg not in unique:
            unique.append(cfg)
    gold = {"configs": configs,
            "hint_encoder": {name: unique.index(cfg) for name, cfg in configs.items()},
            "hint_encoder_outputs": [hint_encoder_case(R, cfg) for cfg in unique],
            "processor": {case: processor_case(R, case) for case in PROC_CASES},
            "unet": {v: unet_case(R, v) for v in UNET_VARIANTS}}
    chunks = []
    tree = _pack(gold, chunks)
    torch.save({"tree": tree, "flat": torch.cat(chunks)}, OUT)
    print("wrote", OUT, OUT.stat().st_size, "bytes")


if __name__ == "__main__":
    main()
