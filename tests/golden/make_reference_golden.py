"""Generates tests/golden/reference_models.pt: golden vectors computed BY THE REFERENCE'S OWN CODE - /root/reference/models.py imported
unmodified (tests/golden/reference_import.py) - for the training-step front half on the tiny SD-style configuration: hint encoder
(ControlLoRA.forward, models.py:810-835) -> processors wired as in train_text_to_image_control_lora.py:469-487 -> UNet -> MSE ->
backward.  The UNet under the processors is the oracle's restatement of diffusers' (diffusers itself cannot run here); ControlLoRA,
ConvBlock2D, SimpleDownEncoderBlock2D and the three processor classes are the reference's.

Weights are seeded through the oracle classes (identical state-dict layout, checked) and loaded into the reference classes, so that
a machine WITHOUT /root/reference (the GPU box) can rebuild the same weights and compare (tests/check_reference_golden.py):
the fp32 oracle at 1e-5, the CUDA path at its bf16 tolerance.

    python -m tests.golden.make_reference_golden          (needs /root/reference; run in the build container)
"""
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from oracle import models_ref as MR  # noqa: E402
from oracle import unet_ref as UR  # noqa: E402

TINY = dict(block_out_channels=(64, 128, 128, 128), layers_per_block=1, cross_attention_dim=64, attention_head_dim=8)
TINY_LORA = dict(lora_block_out_channels=(64, 128, 128, 128),
                 lora_cross_attention_dims=([None, 64] * 3, [None, 64] * 3, [None, 64] * 3, [None, 64]))
CASES = {
    "v1_stacked": (dict(), True, 0.5),                        # + one rank-4 pre-LoRA per layer (mix_lora_and_control_lora.py), scale 0.5
    "v2": (dict(lora_control_version=2, lora_pre_conv_skipped=True), False, 1.0),
    "post_add": (dict(lora_post_add=True), False, 1.0),
    "concat": (dict(lora_concat_hidden=True, lora_control_rank=32, lora_pre_conv_skipped=True, lora_control_self_add=False), False, 1.0),
}
OUT = Path(__file__).resolve().parent / "reference_models.pt"
GRAD_STRIDE = 3          # every third element of each kept gradient is stored: keeps the file under 1 MB


def grad_sample(g: torch.Tensor) -> torch.Tensor:
    """The stored elements of a gradient tensor (flattened, at GRAD_STRIDE)."""
    return g.detach().float().cpu().reshape(-1)[::GRAD_STRIDE]


def seeded_state(case):
    """(ControlLoRA kwargs, ControlLoRA state dict, stacked pre-LoRA state dicts by processor name, inputs) - no reference needed."""
    kw_extra, stacked, scale = CASES[case]
    kw = dict(TINY_LORA)
    kw.update(kw_extra)
    torch.manual_seed(0)
    cl = MR.ControlLoRA(**kw)
    MR.randomize_lora_up_(cl, seed=3, std=0.05)
    g = torch.Generator().manual_seed(2)
    with torch.no_grad():
        for n, p in cl.named_parameters():
            if "norm" in n:
                p.add_(0.1 * torch.randn(p.shape, generator=g))
    unet = UR.UNet2DConditionModel(**TINY)
    UR.init_synthetic_(unet, seed=1)
    with torch.no_grad():
        for p in unet.parameters():                    # the frozen network runs in bf16 in the reference: share exactly representable weights
            p.copy_(p.to(torch.bfloat16).float())
    unet_sd = {k: v.clone() for k, v in unet.state_dict().items()}       # before any processor is installed on it
    pre = {}
    if stacked:
        gp = torch.Generator().manual_seed(11)
        for name, proc in MR.wire_processors(unet, cl).items():
            op = MR.LoRACrossAttnProcessor(proc.hidden_size, proc.cross_attention_dim, rank=4)
            with torch.no_grad():
                for n_, p_ in op.named_parameters():
                    p_.copy_((0.05 if n_.endswith("up.weight") else 0.25) * torch.randn(p_.shape, generator=gp))
            pre[name] = op.state_dict()
    gi = torch.Generator().manual_seed(5)
    r = lambda *s: torch.randn(*s, generator=gi).to(torch.bfloat16).float()
    inputs = dict(x=r(2, 4, 16, 16), t=torch.tensor([17, 801]), ehs=r(2, 77, 64),
                  guide=(torch.rand(2, 3, 128, 128, generator=gi) * 2 - 1).to(torch.bfloat16).float(), target=torch.randn(2, 4, 16, 16, generator=gi))
    return kw, cl.state_dict(), unet_sd, pre, inputs, scale


def run_front_half(M, case):
    """M: the module providing ControlLoRA / LoRACrossAttnProcessor (the reference's models.py, or oracle.models_ref).  Returns the
    golden dictionary of this case."""
    torch.set_num_threads(1)
    kw, cl_sd, unet_sd, pre, inp, scale = seeded_state(case)
    cl = M.ControlLoRA(**kw)
    cl.load_state_dict(cl_sd)
    unet = UR.UNet2DConditionModel(**TINY)
    unet.load_state_dict(unet_sd)
    unet.requires_grad_(False)
    procs = MR.wire_processors(unet, cl)
    stacked = {}
    for name, sd in pre.items():
        p = procs[name]
        op = M.LoRACrossAttnProcessor(p.hidden_size, p.cross_attention_dim, rank=4)
        op.load_state_dict(sd)
        p.inject_pre_lora(op)
        stacked[name] = op
    states = cl(inp["guide"]).control_states
    pred = unet(inp["x"], inp["t"], inp["ehs"], cross_attention_kwargs={"scale": scale}).sample
    loss = torch.nn.functional.mse_loss(pred, inp["target"])
    loss.backward()
    out = {"pred": pred.detach().clone(), "loss": loss.detach().clone(),
           "states": [s.detach()[:, :16, :4, :4].clone() for s in states], "state_norms": torch.stack([s.detach().norm() for s in states])}
    small, norms = {}, {}
    for n, p in cl.named_parameters():
        if p.grad is None:
            continue
        norms[n] = p.grad.double().norm().float()
        if p.numel() <= 1024 and (n.startswith("lora_layers.") or p.dim() <= 1):     # adapter / control matrices, biases, norm parameters
            small[n] = p.grad.detach().clone()
    for name, op in stacked.items():
        for n, p in op.named_parameters():
            if p.grad is not None:
                small[f"pre_lora::{name}::{n}"] = p.grad.detach().clone()
    # one flat tensor + an index per dictionary (a pickle of ~1000 tiny tensors is mostly per-tensor overhead)
    out["grads"] = {"names": list(small), "shapes": [tuple(v.shape) for v in small.values()],
                    "flat": torch.cat([grad_sample(v) for v in small.values()])}
    out["grad_norms"] = {"names": list(norms), "values": torch.stack(list(norms.values()))}
    return out


def unpack_grads(packed) -> dict:
    """name -> the stored sample (grad_sample) of that gradient; "shapes" are the shapes of the whole tensors."""
    out, off = {}, 0
    for n, shp in zip(packed["names"], packed["shapes"]):
        k = 1
        for d in shp:
            k *= d
        k = -(-k // GRAD_STRIDE)
        out[n] = packed["flat"][off:off + k]
        off += k
    return out


def main():
    from tests.golden import reference_import as RI

    R = RI.reference_models()
    gold = {}
    for case in CASES:
        gold[case] = run_front_half(R, case)
        o = run_front_half(MR, case)
        err = float((o["pred"] - gold[case]["pred"]).abs().max() / gold[case]["pred"].abs().max())
        print(f"{case}: {len(gold[case]['grads']['names'])} gradient tensors kept, oracle vs reference pred {err:.2e}")
    torch.save(gold, OUT)
    print("wrote", OUT, OUT.stat().st_size, "bytes")


if __name__ == "__main__":
    main()
