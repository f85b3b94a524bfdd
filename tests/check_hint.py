"""GPU parity of the hint encoder (fwd + all parameter grads) and of one fused Trainer step against the fp32 oracle.
usage: python tests/check_hint.py [hint_v1|hint_v2|train_v1|train_v2]"""
import os
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from tests._device import DEV  # noqa: E402
from tests.check_unet import TINY, TINY_LORA, rel  # noqa: E402


def hint_case(v2: bool, size=64, B=2):
    import torch
    from oracle import models_ref as MR
    import controllora_b200 as cb

    kw = dict(TINY_LORA)
    if v2:
        kw.update(lora_control_version=2, lora_pre_conv_skipped=True)
    torch.manual_seed(0)
    ocl = MR.ControlLoRA(**kw)
    # non-trivial norm parameters
    g = torch.Generator().manual_seed(2)
    with torch.no_grad():
        for n, p in ocl.named_parameters():
            if "norm" in n:
                p.add_(0.1 * torch.randn(p.shape, generator=g))
    mcl = cb.ControlLoRA(**kw)
    mcl.load_state_dict(ocl.state_dict())
    mcl.to(DEV)
    guide = (torch.rand(B, 3, size, size, generator=g) * 2 - 1)
    guide = guide.to(torch.bfloat16).float()
    so = ocl(guide).control_states
    wts = [torch.randn(s.shape, generator=g) for s in so]
    lo = sum((s * w).sum() for s, w in zip(so, wts))
    lo.backward()
    sm = mcl(guide.to(DEV)).control_states
    lm = sum((s.float() * w.to(DEV)).sum() for s, w in zip(sm, wts))
    lm.backward()
    if DEV == "cuda":
        torch.cuda.synchronize()
    worst = 0.0
    for i, (a, b) in enumerate(zip(sm, so)):
        e = rel(a, b)
        worst = max(worst, e)
        print(f"  control_state[{i}] {tuple(b.shape)} rel={e:.3e}")
    rows = []
    zero_b = _zero_grad_biases(ocl)
    oparams = dict(ocl.named_parameters())
    cat_o, cat_m = [], []
    for (n1, p1), (n2, p2) in zip(ocl.named_parameters(), mcl.named_parameters()):
        if n1.startswith("lora_layers"):
            continue
        assert p2.grad is not None, n2
        g2 = p2.grad.detach().float().cpu()
        if n1 in zero_b:
            # exactly-zero true gradient: ours must stay at noise level next to the layer's weight gradient
            wn = float(oparams[n1[:-4] + "weight"].grad.norm())
            assert float(g2.norm()) < 2e-2 * wn, (n1, float(g2.norm()), wn)
            continue
        rows.append((rel(g2, p1.grad), n1, float(p1.grad.norm())))
        cat_o.append(p1.grad.flatten()); cat_m.append(g2.flatten())
    rows.sort(reverse=True)
    for e, n, nrm in rows[:10]:
        print(f"  grad rel={e:.3e} |g|={nrm:.3e} {n}")
    e_all = rel(torch.cat(cat_m), torch.cat(cat_o))
    print(f"  all hint-encoder gradients (concatenated, {len(rows)} tensors) rel={e_all:.3e}; worst tensor rel={rows[0][0]:.3e}")
    ok = worst < 3e-2 and e_all < 5e-2 and rows[0][0] < 8e-2
    print("CASE_OK" if ok else "CASE_FAIL")
    return ok


def _zero_grad_biases(cl):
    """Conv biases whose TRUE gradient is exactly zero: the conv feeds a GroupNorm with one channel per group (the
    32-channel first pyramid level, models.py:690-748), which removes any per-channel constant.  The oracle shows fp32
    noise there (|g| ~ 1e-9 x the weight gradient); Adam turns that noise into +-lr updates in ANY implementation, so
    these tensors carry no parity information and are excluded from the update / gradient metrics."""
    groups = cl.config["norm_num_groups"] if isinstance(cl.config, dict) else cl.config.norm_num_groups
    return {n for n, p in cl.named_parameters()
            if n.endswith("bias") and p.dim() == 1 and p.numel() == groups and ("conv1" in n or "downsamplers" in n or n == "conv_in.bias")}


def train_case(v2: bool, B=2, HW=16):
    """Two fused Trainer steps vs the oracle driven by torch.optim.AdamW + clip_grad_norm_ (the reference's step glue,
    train_text_to_image_control_lora.py:783-796).  Three separate checks, each with its own tolerance:
      (1) gradient parity: the gradient arena after the fused backward vs the oracle's autograd gradients
          (bf16 pipeline vs fp32: <= 5e-2 relative on the concatenated gradient, tiny config);
      (2) optimizer parity: clip_grad_norm_ + torch.optim.AdamW applied to OUR gradients on the host must reproduce the
          fused clip + AdamW kernel's parameter update (fp32 arithmetic on both sides: <= 2e-3 relative);
      (3) end-to-end parameter update vs the oracle trajectory, provably-zero-gradient biases excluded.  Adam's first
          updates are +-lr * sign(g), so every gradient element whose sign differs costs 2 lr: this number measures the
          fraction of near-zero gradient elements, it is capped loosely (<= 0.25) and reported."""
    import torch
    from oracle import models_ref as MR
    from oracle import unet_ref as UR
    import controllora_b200 as cb
    from controllora_b200.trainer import Trainer

    torch.manual_seed(0)
    ounet = UR.UNet2DConditionModel(**TINY)
    UR.init_synthetic_(ounet, seed=1)
    with torch.no_grad():
        for p in ounet.parameters():
            p.copy_(p.to(torch.bfloat16).float())
    ounet.requires_grad_(False)
    munet = cb.UNet2DConditionModel.from_state_dict({k: v.clone() for k, v in ounet.state_dict().items()}, DEV, TINY)
    kw = dict(TINY_LORA)
    if v2:
        kw.update(lora_control_version=2, lora_pre_conv_skipped=True, lora_key_states_skipped=True, lora_value_states_skipped=True)
    ocl = MR.ControlLoRA(**kw)
    MR.randomize_lora_up_(ocl, seed=3, std=0.05)
    mcl = cb.ControlLoRA(**kw)
    mcl.load_state_dict(ocl.state_dict())
    mcl.to(DEV)
    import copy
    hcl = copy.deepcopy(ocl)                      # host twin that receives OUR gradients (check 2)
    MR.wire_processors(ounet, ocl)
    MR.wire_processors(munet, mcl)
    adam = dict(lr=1e-4, betas=(0.9, 0.999), weight_decay=1e-2, eps=1e-8)
    opt = torch.optim.AdamW(ocl.parameters(), **adam)
    hopt = torch.optim.AdamW(hcl.parameters(), **adam)
    tr = Trainer(munet, mcl, lr=1e-4)
    g = torch.Generator().manual_seed(5)
    size = HW * 8
    zero_b = _zero_grad_biases(ocl)
    names = [n for n, _ in ocl.named_parameters()]
    p0 = {n: p.detach().clone() for n, p in ocl.named_parameters()}
    worst_grad = worst_opt = 0.0
    for step in range(2):
        x = torch.randn(B, 4, HW, HW, generator=g).to(torch.bfloat16).float()
        t = torch.randint(0, 1000, (B,), generator=g)
        e = torch.randn(B, 77, TINY["cross_attention_dim"], generator=g).to(torch.bfloat16).float()
        guide = (torch.rand(B, 3, size, size, generator=g) * 2 - 1).to(torch.bfloat16).float()
        tgt = torch.randn(B, 4, HW, HW, generator=g)
        ocl(guide)
        lo = torch.nn.functional.mse_loss(ounet(x, t, e).sample, tgt)
        lo.backward()
        go = {n: p.grad.detach().clone() for n, p in ocl.named_parameters()}
        gn = torch.nn.utils.clip_grad_norm_(ocl.parameters(), 1.0)
        opt.step()
        opt.zero_grad()
        # ours, split at the gradient: fused forward/backward, read the arena, then the fused clip + AdamW tail
        before = {n: p.detach().cpu().clone() for n, p in mcl.named_parameters()}
        lm = tr._forward_backward(x.to(DEV), t.to(DEV).float(), e.to(DEV).to(torch.bfloat16), guide.to(DEV), tgt.to(DEV))
        gm = {n: tr.arena.grad_of(p).detach().cpu().clone() for n, p in mcl.named_parameters()}
        tr._optimizer_tail()
        if DEV == "cuda":
            torch.cuda.synchronize()
        after = {n: p.detach().cpu().clone() for n, p in mcl.named_parameters()}
        # (1) gradient parity
        sel = [n for n in names if n not in zero_b]
        e_grad = rel(torch.cat([gm[n].flatten() for n in sel]), torch.cat([go[n].flatten() for n in sel]))
        worst_grad = max(worst_grad, e_grad)
        # (2) optimizer parity on our own gradients
        with torch.no_grad():
            for (n, p) in hcl.named_parameters():
                p.copy_(before[n])
                p.grad = gm[n].clone()
        torch.nn.utils.clip_grad_norm_(hcl.parameters(), 1.0)
        hopt.step()
        num = sum(float(((after[n] - before[n]) - (p.detach() - before[n])).pow(2).sum()) for n, p in hcl.named_parameters())
        den = sum(float((p.detach() - before[n]).pow(2).sum()) for n, p in hcl.named_parameters())
        e_opt = (num / max(den, 1e-30)) ** 0.5
        worst_opt = max(worst_opt, e_opt)
        print(f"  step {step}: loss oracle={float(lo):.6f} ours={float(lm):.6f}  oracle grad-norm={float(gn):.4f} "
              f"ours={float(tr.gnorm_sq.sqrt()):.4f}  grad rel={e_grad:.3e}  clip+AdamW rel (same grads)={e_opt:.3e}")
    # (3) end-to-end parameter updates
    num = den = 0.0
    worst = (0.0, "")
    for (n, po), (_, pm) in zip(ocl.named_parameters(), mcl.named_parameters()):
        if n in zero_b:
            continue
        do = po.detach() - p0[n]
        dm = pm.detach().cpu() - p0[n]
        num += float((dm - do).pow(2).sum())
        den += float(do.pow(2).sum())
        e = float((dm - do).norm() / (do.norm() + 1e-12))
        if e > worst[0] and float(do.norm()) > 1e-6:
            worst = (e, n)
    tot = (num / den) ** 0.5
    print(f"  gradient rel (worst step) = {worst_grad:.3e}; clip+AdamW on identical gradients rel = {worst_opt:.3e}")
    print(f"  parameter-update rel vs the oracle trajectory (zero-gradient biases {sorted(zero_b)} excluded) = {tot:.3e}; "
          f"worst tensor {worst[1]} rel={worst[0]:.3e}")
    ok = worst_grad < 5e-2 and worst_opt < 2e-3 and tot < 0.25
    print("CASE_OK" if ok else "CASE_FAIL")
    return ok


def train_lora_only_case(B=4, HW=16, prior_w=0.7):
    """The DreamBooth-LoRA step (train_dreambooth_lora.py:880-918): plain LoRACrossAttnProcessor on every attention layer, no
    ControlLoRA, loss = mse(instance half) + prior_loss_weight * mse(class half), clip + AdamW - Trainer(control_lora=None) against
    the oracle driven by torch autograd + torch.optim.AdamW.  Also the attention-processor file round trip (`save_attn_procs`)."""
    import tempfile

    import torch
    from oracle import models_ref as MR
    from oracle import unet_ref as UR
    import controllora_b200 as cb
    from controllora_b200.trainer import Trainer

    torch.manual_seed(0)
    ounet = UR.UNet2DConditionModel(**TINY)
    UR.init_synthetic_(ounet, seed=1)
    with torch.no_grad():
        for p in ounet.parameters():
            p.copy_(p.to(torch.bfloat16).float())
    ounet.requires_grad_(False)
    munet = cb.UNet2DConditionModel.from_state_dict({k: v.clone() for k, v in ounet.state_dict().items()}, DEV, TINY)
    g = torch.Generator().manual_seed(7)
    oprocs, mprocs = {}, {}
    for name in ounet.attn_processors.keys():
        C = dict(ounet._attn_modules())[name].to_q.weight.shape[0]
        xd = None if name.endswith("attn1.processor") else TINY["cross_attention_dim"]
        op = MR.LoRACrossAttnProcessor(C, xd, rank=4)
        with torch.no_grad():
            for n_, p_ in op.named_parameters():
                if n_.endswith("up.weight"):
                    p_.copy_(0.05 * torch.randn(p_.shape, generator=g))
        mp = cb.LoRACrossAttnProcessor(C, xd, rank=4)
        mp.load_state_dict(op.state_dict())
        oprocs[name], mprocs[name] = op, mp.to(DEV)
    ounet.set_attn_processor(oprocs)
    munet.set_attn_processor(mprocs)
    oparams = [p for op in oprocs.values() for p in op.parameters()]
    opt = torch.optim.AdamW(oparams, lr=1e-4, betas=(0.9, 0.999), weight_decay=1e-2, eps=1e-8)
    tr = Trainer(munet, None, lr=1e-4, prior_loss_weight=prior_w)
    assert tr.numel == sum(p.numel() for p in oparams)
    worst_grad, worst_loss = 0.0, 0.0
    for step in range(2):
        x = torch.randn(B, 4, HW, HW, generator=g).to(torch.bfloat16).float()
        t = torch.randint(0, 1000, (B,), generator=g)
        e = torch.randn(B, 77, TINY["cross_attention_dim"], generator=g).to(torch.bfloat16).float()
        tgt = torch.randn(B, 4, HW, HW, generator=g)
        pred = ounet(x, t, e).sample
        h = B // 2
        lo = torch.nn.functional.mse_loss(pred[:h], tgt[:h]) + prior_w * torch.nn.functional.mse_loss(pred[h:], tgt[h:])
        lo.backward()
        go = torch.cat([p.grad.flatten() for p in oparams])
        torch.nn.utils.clip_grad_norm_(oparams, 1.0)
        opt.step()
        opt.zero_grad()
        lm = tr._forward_backward(x.to(DEV), t.to(DEV).float(), e.to(DEV).to(torch.bfloat16), None, tgt.to(DEV))
        gm = tr.flat_g[:tr.numel].detach().cpu().clone()
        tr.step_idx += 1
        tr._optimizer_tail()
        if DEV == "cuda":
            torch.cuda.synchronize()
        worst_grad = max(worst_grad, rel(gm, go))
        worst_loss = max(worst_loss, abs(float(lm) - float(lo)) / abs(float(lo)))
        print(f"  step {step}: loss oracle={float(lo):.6f} ours={float(lm):.6f}  all-adapter gradient rel={rel(gm, go):.3e}")
    po = torch.cat([p.detach().flatten() for p in oparams])
    pm = tr.flat_p[:tr.numel].detach().cpu()
    with tempfile.TemporaryDirectory() as d:
        f = munet.save_attn_procs(d)
        sd = torch.load(f)
        okeys = [f"{k}.{n}" for k, op in oprocs.items() for n, _ in op.named_parameters()]
        keys_ok = list(sd.keys()) == okeys
        m2 = cb.UNet2DConditionModel.from_state_dict({k: v.clone() for k, v in ounet.state_dict().items() if ".processor." not in k}, DEV, TINY)
        m2.load_attn_procs(d)
        rt_ok = all(torch.equal(a.detach().cpu(), b.detach().cpu()) for a, b in zip(m2.attn_procs_state_dict().values(), munet.attn_procs_state_dict().values()))
    e_upd = rel(pm, po)      # parameters after two steps (Adam's +-lr steps on an O(0.05..0.25) scale: dominated by the unchanged part)
    print(f"  gradient rel (worst step) = {worst_grad:.3e}; loss rel = {worst_loss:.2e}; parameters after 2 steps rel = {e_upd:.3e}; "
          f"attn-procs file keys ok={keys_ok}, round trip ok={rt_ok}")
    ok = worst_grad < 5e-2 and worst_loss < 2e-3 and e_upd < 1e-3 and keys_ok and rt_ok
    print("CASE_OK" if ok else "CASE_FAIL")
    return ok


def accumulate_case(B=2, HW=16, micro=3):
    """`--gradient_accumulation_steps 3` (train_text_to_image_control_lora.py:751 `accelerator.accumulate`, 1/N loss scaling, clip + AdamW
    once per window): Trainer.accumulate() x2 + step() against the oracle + torch.optim.AdamW doing the same."""
    import copy

    import torch
    from oracle import models_ref as MR
    from oracle import unet_ref as UR
    import controllora_b200 as cb
    from controllora_b200.trainer import Trainer

    torch.manual_seed(0)
    ounet = UR.UNet2DConditionModel(**TINY)
    UR.init_synthetic_(ounet, seed=1)
    with torch.no_grad():
        for p in ounet.parameters():
            p.copy_(p.to(torch.bfloat16).float())
    ounet.requires_grad_(False)
    munet = cb.UNet2DConditionModel.from_state_dict({k: v.clone() for k, v in ounet.state_dict().items()}, DEV, TINY)
    kw = dict(TINY_LORA, lora_control_version=2, lora_pre_conv_skipped=True)
    ocl = MR.ControlLoRA(**kw)
    MR.randomize_lora_up_(ocl, seed=3, std=0.05)
    mcl = cb.ControlLoRA(**kw)
    mcl.load_state_dict(ocl.state_dict())
    mcl.to(DEV)
    hcl = copy.deepcopy(ocl)                      # host twin that receives OUR accumulated gradient
    MR.wire_processors(ounet, ocl)
    MR.wire_processors(munet, mcl)
    tr = Trainer(munet, mcl, lr=1e-4)
    g = torch.Generator().manual_seed(5)
    zero_b = _zero_grad_biases(ocl)
    for k in range(micro):
        x = torch.randn(B, 4, HW, HW, generator=g).to(torch.bfloat16).float()
        t = torch.randint(0, 1000, (B,), generator=g)
        e = torch.randn(B, 77, TINY["cross_attention_dim"], generator=g).to(torch.bfloat16).float()
        guide = (torch.rand(B, 3, HW * 8, HW * 8, generator=g) * 2 - 1).to(torch.bfloat16).float()
        tgt = torch.randn(B, 4, HW, HW, generator=g)
        ocl(guide)
        (torch.nn.functional.mse_loss(ounet(x, t, e).sample, tgt) / micro).backward()
        args = (x.to(DEV), t.to(DEV).float(), e.to(DEV).to(torch.bfloat16), guide.to(DEV), tgt.to(DEV))
        if k < micro - 1:
            tr.accumulate(*args)
        else:
            tr.step_idx += 1
            tr._forward_backward(*args)
            gm = {n: (tr.arena.grad_of(p) / micro).detach().cpu().clone() for n, p in mcl.named_parameters()}
            tr._optimizer_tail()
    if DEV == "cuda":
        torch.cuda.synchronize()
    names = [n for n, _ in ocl.named_parameters() if n not in zero_b]
    go = {n: p.grad.detach().clone() for n, p in ocl.named_parameters()}
    e_grad = rel(torch.cat([gm[n].flatten() for n in names]), torch.cat([go[n].flatten() for n in names]))
    # clip + AdamW on OUR accumulated mean gradient must be what the fused tail did
    with torch.no_grad():
        for n, p in hcl.named_parameters():
            p.grad = gm[n].clone()
    hopt = torch.optim.AdamW(hcl.parameters(), lr=1e-4, betas=(0.9, 0.999), weight_decay=1e-2, eps=1e-8)
    torch.nn.utils.clip_grad_norm_(hcl.parameters(), 1.0)
    p0 = {n: p.detach().clone() for n, p in ocl.named_parameters()}
    hopt.step()
    num = sum(float(((pm.detach().cpu() - p0[n]) - (ph.detach() - p0[n])).pow(2).sum()) for (n, ph), (_, pm) in zip(hcl.named_parameters(), mcl.named_parameters()))
    den = sum(float((ph.detach() - p0[n]).pow(2).sum()) for n, ph in hcl.named_parameters())
    e_opt = (num / den) ** 0.5
    print(f"  accumulated over {micro} micro-batches: mean-gradient rel vs oracle = {e_grad:.3e}; clip + AdamW on it rel = {e_opt:.3e}; "
          f"arena zeroed = {float(tr.flat_g.abs().sum()) == 0.0}; micro counter reset = {tr._micro == 0}")
    ok = e_grad < 5e-2 and e_opt < 2e-3 and float(tr.flat_g.abs().sum()) == 0.0 and tr._micro == 0
    print("CASE_OK" if ok else "CASE_FAIL")
    return ok


def resume_case(B=2, HW=16):
    """Resume equivalence (train_text_to_image_control_lora.py:713-735 / 805-809): 3 steps in one run == 2 steps, save_checkpoint, a
    NEW Trainer on freshly initialised models, load_checkpoint, 1 more step - bit for bit (parameters, AdamW moments, device step
    counter, and the device Philox counter: step 3 draws the same noise / timesteps in both runs); on the GPU the restored state bit
    for bit and step 3 to the run-to-run tolerance."""
    import tempfile

    import torch
    import controllora_b200 as cb
    from controllora_b200.trainer import Trainer
    from oracle import models_ref as MR

    def make(seed):
        torch.manual_seed(seed)
        munet = cb.UNet2DConditionModel.synthetic(DEV, TINY, seed=1)
        mcl = cb.ControlLoRA(**dict(TINY_LORA, lora_control_version=2, lora_pre_conv_skipped=True)).to(DEV)
        if seed == 0:
            MR.randomize_lora_up_(mcl, seed=3, std=0.05)
        MR.wire_processors(munet, mcl)
        return Trainer(munet, mcl, lr=1e-3, noise_seed=77), mcl

    g = torch.Generator().manual_seed(8)
    batches = [((0.2 * torch.randn(B, 4, HW, HW, generator=g)).to(DEV), torch.randn(B, 77, 64, generator=g).to(torch.bfloat16).to(DEV),
                (torch.rand(B, 3, HW * 8, HW * 8, generator=g) * 2 - 1).to(DEV)) for _ in range(3)]
    a, _ = make(0)
    for b in batches:
        loss_a = a.step_from_latents(*b)
    draw_a = [t.detach().cpu().clone() for t in a.last_noise_draw]
    b1, _ = make(0)
    for b in batches[:2]:
        b1.step_from_latents(*b)
    with tempfile.TemporaryDirectory() as d:
        path = b1.save_checkpoint(d)
        b2, _ = make(5)                                   # different initial weights: everything must come from the checkpoint
        gs = b2.load_checkpoint(path)
    restored = all(torch.equal(getattr(b1, k), getattr(b2, k)) for k in ("flat_p", "flat_m", "flat_v", "step_dev", "rng_counter"))
    loss_c = b1.step_from_latents(*batches[2])            # b1 goes on uninterrupted from the state it saved
    loss_b = b2.step_from_latents(*batches[2])
    if DEV == "cuda":
        torch.cuda.synchronize()
    draw_b = [t.detach().cpu().clone() for t in b2.last_noise_draw]
    # CPU host-logic mode is deterministic: bit for bit, and the run that wrote the checkpoint equals the one that never did.  On the
    # GPU the weight-gradient kernels reduce with fp32 atomics (split-K + RED, csrc/wgrad.cu), so two RUNS differ at the 1e-7 level,
    # and Adam turns that noise into +-lr steps wherever a gradient element is near zero: after two steps at lr 1e-3 the next
    # gradients, and with them the moments, of two uninterrupted runs (a, b1) differ by more than the 2e-3 tolerance of the
    # eager-vs-graph comparison.  So on the GPU the resumed run is compared with b1 going on from the state it saved: the restored
    # state is exact, one step of atomics noise separates the two.  The restored counters and the step-3 noise draw are exact on both.
    if DEV == "cuda":
        close = lambda x, y: float((x - y).norm() / (y.norm() + 1e-30)) < 2e-3
        ref = b1
    else:
        close = torch.equal
        ref = a
    rd = lambda x, y: float((x - y).norm() / (y.norm() + 1e-30))
    print(f"  two uninterrupted runs (a vs b1) after 3 steps: params rel={rd(b1.flat_p, a.flat_p):.2e} exp_avg rel={rd(b1.flat_m, a.flat_m):.2e} "
          f"exp_avg_sq rel={rd(b1.flat_v, a.flat_v):.2e}; resumed vs b1: params rel={rd(b2.flat_p, b1.flat_p):.2e} "
          f"exp_avg rel={rd(b2.flat_m, b1.flat_m):.2e} exp_avg_sq rel={rd(b2.flat_v, b1.flat_v):.2e}")
    same = {"global_step": gs == 2, "restored": restored, "params": close(b2.flat_p, b1.flat_p) and close(b2.flat_p, ref.flat_p),
            "exp_avg": close(b2.flat_m, b1.flat_m) and close(b2.flat_m, ref.flat_m),
            "exp_avg_sq": close(b2.flat_v, b1.flat_v) and close(b2.flat_v, ref.flat_v),
            "step": a.step_idx == b1.step_idx == b2.step_idx == int(b2.step_dev) == 3,
            "rng_counter": int(a.rng_counter) == int(b1.rng_counter) == int(b2.rng_counter) == 3,
            "loss": all(abs(float(x) - float(loss_b)) <= (2e-3 * abs(float(x)) if DEV == "cuda" else 0.0) for x in (loss_a, loss_c)),
            "noise_draw": all(torch.equal(x, y) for x, y in zip(draw_a[1:], draw_b[1:])) and close(draw_a[0], draw_b[0])}
    print("  resume equivalence:", same)
    ok = all(same.values())
    print("CASE_OK" if ok else "CASE_FAIL")
    return ok


def graph_case(v2: bool = True, B=2, HW=16, steps=5):
    """Trainer(cuda_graph=True) (2 eager warm-up steps, capture, replays) against the eager Trainer on the same
    per-step inputs: the same kernels run in the same order, so losses and parameters must agree to fp32 atomics noise."""
    import torch
    from oracle import unet_ref as UR
    import controllora_b200 as cb
    from controllora_b200.configs import wire_processors
    from controllora_b200.trainer import Trainer

    torch.manual_seed(0)
    ounet = UR.UNet2DConditionModel(**TINY)
    UR.init_synthetic_(ounet, seed=1)
    sd = {k: v.detach().clone() for k, v in ounet.state_dict().items()}
    kw = dict(TINY_LORA)
    if v2:
        kw.update(lora_control_version=2, lora_pre_conv_skipped=True, lora_key_states_skipped=True, lora_value_states_skipped=True)
    trainers = []
    for use_graph in (False, True):
        unet = cb.UNet2DConditionModel.from_state_dict({k: v.clone() for k, v in sd.items()}, DEV, TINY)
        torch.manual_seed(7)
        cl = cb.ControlLoRA(**kw)
        g = torch.Generator().manual_seed(3)
        with torch.no_grad():
            for n_, p_ in cl.named_parameters():
                if n_.endswith("up.weight"):
                    p_.copy_(0.05 * torch.randn(p_.shape, generator=g))
        cl.to(DEV)
        wire_processors(unet, cl)
        trainers.append((Trainer(unet, cl, lr=1e-3, cuda_graph=use_graph), cl))
    g = torch.Generator().manual_seed(5)
    size = HW * 8
    ok = True
    for step in range(steps):
        x = torch.randn(B, 4, HW, HW, generator=g).to(DEV)
        t = torch.randint(0, 1000, (B,), generator=g).float().to(DEV)
        e = torch.randn(B, 77, TINY["cross_attention_dim"], generator=g).to(DEV).to(torch.bfloat16)
        guide = (torch.rand(B, 3, size, size, generator=g) * 2 - 1).to(DEV)
        tgt = torch.randn(B, 4, HW, HW, generator=g).to(DEV)
        losses = [float(tr.step(x, t, e, guide, tgt)) for tr, _ in trainers]
        print(f"  step {step}: loss eager={losses[0]:.6f} graph={losses[1]:.6f} captured={trainers[1][0]._graph is not None}")
        ok = ok and abs(losses[0] - losses[1]) <= 2e-3 * abs(losses[0]) + 1e-6
    num = den = 0.0
    for (n, pe), (_, pg) in zip(trainers[0][1].named_parameters(), trainers[1][1].named_parameters()):
        num += float((pe.detach() - pg.detach()).pow(2).sum())
        den += float(pe.detach().pow(2).sum())
    rel = (num / den) ** 0.5
    print(f"  parameter rel diff eager vs graph after {steps} steps = {rel:.3e}; launches/step = {trainers[1][0].launches_per_step}")
    ok = ok and rel < 2e-3 and trainers[1][0]._graph is not None
    print("CASE_OK" if ok else "CASE_FAIL")
    return ok


CASES = {
    "graph_v2": lambda: graph_case(True),
    "hint_v1": lambda: hint_case(False),
    "hint_v2": lambda: hint_case(True),
    "train_v1": lambda: train_case(False),
    "train_v2": lambda: train_case(True),
    "train_lora_only": train_lora_only_case,
    "resume": resume_case,
    "accumulate": accumulate_case,
}


def main():
    names = sys.argv[1:] or list(CASES)
    if len(names) == 1:
        sys.exit(0 if CASES[names[0]]() else 1)
    res = {}
    for v in names:
        try:
            r = subprocess.run([sys.executable, __file__, v], capture_output=True, text=True, timeout=600)
            ok = r.returncode == 0 and "CASE_OK" in r.stdout
            out = r.stdout + r.stderr
        except subprocess.TimeoutExpired as e:
            ok, out = False, f"TIMEOUT {e}"
        res[v] = ok
        print(f"=== {v}: {'PASS' if ok else 'FAIL'}")
        lines = [l for l in out.strip().splitlines() if "Warning" not in l and "Consider using" not in l]
        for line in (lines if ok else lines[-40:]):
            print("    " + line)
        sys.stdout.flush()
    print("SUMMARY", res)


if __name__ == "__main__":
    main()
