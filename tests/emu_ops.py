"""TEST INFRASTRUCTURE ONLY — a torch-on-CPU restatement of what every `controllora_b200.ops` wrapper asks its CUDA kernel to do.

Why it exists: the product has no CPU path (ops raise `CLError` on CPU tensors, DESIGN.md §1), so without a GPU nothing above
the C ABI could be exercised: the tape engine, the LoRA slot packing, the v1 / V2 control algebra, the hint-encoder program, the
trainer's arena wiring.  `install()` swaps the wrappers of `controllora_b200.ops` for the functions below INSIDE A TEST PROCESS,
so that the `-m "not gpu"` suite can run that host logic end to end and compare it with the fp32 oracle.  The functions follow
the contracts written in `include/controllora_b200.h` (bf16 storage between ops, fp32 arithmetic inside, the same operand
layouts: hi/lo `ext` rows, `[N, rp]` tables, strided raw-pointer outputs).

Every replaced wrapper first runs the REAL wrapper on the same (CPU) tensors: the real argument marshalling of ops.py and the real
C launcher's argument validation execute - a GPU-less box gets as far as the first CUDA call, which fails with CL_ERR_CUDA (-2);
CL_ERR_INVALID / CL_ERR_UNSUPPORTED (-1 / -3) mean the kernel would have refused the host program's arguments and fail the test.

It is never imported by the package, by `bench.py`'s GPU arm or by anything that ships; it proves nothing about the kernels
(the `-m gpu` suite does that against the oracle) — only that the host program issues the right sequence of operations.
"""
from __future__ import annotations

import contextlib
import math

import torch
import torch.nn.functional as F

BF16 = torch.bfloat16
_INSTALLED = {}


def _bf(x: torch.Tensor) -> torch.Tensor:
    return x.to(BF16)


def _req_dtype_only(t, dtype, name):
    if t.dtype != dtype:
        from controllora_b200._lib import CLError

        raise CLError(f"{name}: expected {dtype}, got {t.dtype}")


def _sv(t: torch.Tensor, size, stride, extra_off: int = 0) -> torch.Tensor:
    """The strided window a kernel addresses from a raw pointer: elements base + i*stride_i (+ extra_off)."""
    return torch.as_strided(t, size, stride, t.storage_offset() + extra_off)


# ------------------------------------------------------------------------------------------------------------ GEMM
def _conv_weight(b: torch.Tensor, C: int) -> torch.Tensor:
    N = b.shape[0]
    return b.float().view(N, 3, 3, C).permute(0, 3, 1, 2)          # [N, C, ky, kx]


def gemm(a, b, *, out=None, bias=None, row_bias=None, rows_per_group=0, residual=None, ext=None, lora_up=None,
         lora_scale=1.0, t_add=None, t_out=None, out_fp32=False, conv_stride=0, pad_lo=1, block_n=0):
    assert a.dtype == BF16 and b.dtype == BF16
    N, K = b.shape
    # the argument checks of cl_gemm (csrc/gemm.cu): a host program the kernel would reject must fail here too
    assert N % 4 == 0 and K % 8 == 0 and b.stride(0) % 8 == 0 and b.stride(1) == 1, "cl_gemm: N % 4, K % 8, ldb % 8"
    assert (ext is None) == (lora_up is None) and (lora_up is not None or (t_add is None and t_out is None))
    if lora_up is not None:
        assert lora_up.shape[1] in (4, 8) and ext.stride(0) % 8 == 0 and not conv_stride
    if not conv_stride:
        assert a.stride(1) == 1 and a.stride(0) % 8 == 0, "cl_gemm: lda % 8"
    else:
        assert a.is_contiguous() and a.shape[-1] % 32 == 0 and a.shape[1] % conv_stride == 0 and a.shape[2] % conv_stride == 0
    for t_, nm in ((out, "ldd"), (residual, "ldr")):
        if t_ is not None and not t_.is_contiguous():
            assert t_.dim() == 2 and t_.stride(1) == 1 and t_.stride(0) % 4 == 0, f"cl_gemm: {nm} % 4"
    if conv_stride:
        n, H, W, C = a.shape
        assert K == 9 * C
        x = a.float().permute(0, 3, 1, 2)
        w = _conv_weight(b, C)
        if conv_stride == 1:
            y = F.conv2d(x, w, padding=1)
        elif pad_lo == 1:
            y = F.conv2d(x, w, stride=2, padding=1)
        else:
            y = F.conv2d(F.pad(x, (0, 1, 0, 1)), w, stride=2)
        out_shape = (n, H // conv_stride, W // conv_stride, N)
        acc = y.permute(0, 2, 3, 1).reshape(-1, N)
        a2 = None
    else:
        assert a.dim() == 2 and a.shape[1] == K
        a2 = a.float()
        acc = a2 @ b.float().t()
        out_shape = (a.shape[0], N)
    M = acc.shape[0]
    if bias is not None:
        acc = acc + bias.float()[None, :]
    if row_bias is not None:
        grp = torch.arange(M) // rows_per_group
        acc = acc + row_bias.float()[grp][:, :N]
    if lora_up is not None:
        rp = lora_up.shape[1]
        assert ext.shape == (16, K) and lora_up.shape[0] == N and a2 is not None
        e = a2 @ ext.float().t()                                        # [M, 16]: hi rows 0..7, lo rows 8..15
        t = e[:, :rp] + e[:, 8:8 + rp]
        if t_add is not None:
            t = t + t_add
        acc = acc + float(lora_scale) * (t @ lora_up.float().t())
        if t_out is not None:
            t_out.copy_(t)
    if residual is not None:
        acc = acc + residual.reshape(-1, N).float() if residual.is_contiguous() else acc + residual.float()
    res = acc if out_fp32 else _bf(acc)
    if out is None:
        return res.reshape(out_shape).contiguous()
    o2 = out.view(-1, N) if out.is_contiguous() else out
    o2.copy_(res)
    return out


# ------------------------------------------------------------------------------------------------------------ attention
def _heads(x, H):
    B, N, HD = x.shape
    return x.float().reshape(B, N, H, HD // H).permute(0, 2, 1, 3)   # [B, H, N, d]


def attention_fwd(q, k, v, heads, scale, out=None, need_lse=True):
    qh, kh, vh = _heads(q, heads), _heads(k, heads), _heads(v, heads)
    s = (qh @ kh.transpose(-1, -2)) * scale
    lse = torch.logsumexp(s, -1)
    p = torch.exp(s - lse[..., None])
    o = (p @ vh).permute(0, 2, 1, 3).reshape(q.shape)
    if out is None:
        out = torch.empty(q.shape, dtype=BF16)
    out.copy_(_bf(o))
    return out, (lse if need_lse else None)


def attention_bwd(q, k, v, o, d_o, lse, heads, scale, need_dq=True, need_dkv=True, dq=None, dk=None, dv=None):
    qh, kh, vh, oh, doh = (_heads(t, heads) for t in (q, k, v, o, d_o))
    s = (qh @ kh.transpose(-1, -2)) * scale
    p = torch.exp(s - lse[..., None])
    delta = (doh * oh).sum(-1, keepdim=True)
    dp = doh @ vh.transpose(-1, -2)
    ds = p * (dp - delta)

    def back(x, like, dst):
        x = _bf(x.permute(0, 2, 1, 3).reshape(like.shape))
        if dst is None:
            return x.contiguous()
        dst.copy_(x)
        return dst

    if need_dq:
        dq = back((ds @ kh) * scale, q, dq)
    if need_dkv:
        dk = back((ds.transpose(-1, -2) @ qh) * scale, k, dk)
        dv = back(p.transpose(-1, -2) @ doh, v, dv)
    return dq, dk, dv


# ------------------------------------------------------------------------------------------------------------ norms
def _gn(x, gamma, beta, G, eps, silu):
    n, C = x.shape[0], x.shape[-1]
    xg = x.reshape(n, -1, G, C // G)
    mean = xg.mean(dim=(1, 3), keepdim=True)
    var = xg.var(dim=(1, 3), unbiased=False, keepdim=True)
    y = ((xg - mean) * torch.rsqrt(var + eps)).reshape(x.shape) * gamma + beta
    return F.silu(y) if silu else y


def groupnorm_fwd(x, gamma, beta, G, eps, silu, out=None):
    y = _bf(_gn(x.float(), gamma, beta, G, eps, silu))
    stats = torch.tensor([float(eps)])      # opaque to the host code: the backward below only needs eps back
    if out is not None:
        out.copy_(y)
        y = out
    return y, stats


def groupnorm_bwd(x, dy, gamma, beta, stats, G, silu, dx=None, accumulate=False, dgamma=None, dbeta=None):
    eps = float(stats[0])
    xf = x.float().clone().requires_grad_(True)
    g = gamma.detach().clone().requires_grad_(True)
    b = beta.detach().clone().requires_grad_(True)
    with torch.enable_grad():
        y = _gn(xf, g, b, G, eps, silu)
        gx, gg, gb = torch.autograd.grad(y, (xf, g, b), dy.float())
    if dgamma is not None:
        dgamma += gg
    if dbeta is not None:
        dbeta += gb
    if dx is None:
        return _bf(gx)
    dx.copy_(_bf(dx.float() + gx) if accumulate else _bf(gx))
    return dx


def layernorm_fwd(x, gamma, beta, eps=1e-5):
    C = x.shape[-1]
    y = F.layer_norm(x.float(), (C,), gamma, beta, eps)
    return _bf(y), torch.tensor([float(eps)])


def layernorm_bwd(x, dy, gamma, stats, dx=None, accumulate=False):
    C = x.shape[-1]
    xf = x.float().clone().requires_grad_(True)
    with torch.enable_grad():
        y = F.layer_norm(xf, (C,), gamma, None, float(stats[0]))
        (gx,) = torch.autograd.grad(y, xf, dy.float())
    if dx is None:
        return _bf(gx)
    dx.copy_(_bf(dx.float() + gx) if accumulate else _bf(gx))
    return dx


# ------------------------------------------------------------------------------------------------------------ elementwise
def geglu_fwd(p):
    assert p.dtype == BF16 and p.is_contiguous()
    a, g = p.float().chunk(2, -1)
    return _bf(a * F.gelu(g))


def geglu_bwd(p, dout):
    pf = p.float().clone().requires_grad_(True)
    with torch.enable_grad():
        a, g = pf.chunk(2, -1)
        (gp,) = torch.autograd.grad(a * F.gelu(g), pf, dout.float())
    return _bf(gp)


def add(a, b, out=None):
    assert a.dtype == BF16 and b.dtype == BF16 and (out is None or out.dtype == BF16), "cl_add is a bf16 kernel"
    assert a.is_contiguous() and b.is_contiguous() and a.shape == b.shape and a.numel() % 8 == 0
    r = _bf(a.float() + b.float())
    if out is None:
        return r
    out.copy_(r)
    return out


def upsample2x_fwd(x):
    return x.repeat_interleave(2, 1).repeat_interleave(2, 2).contiguous()


def upsample2x_bwd(dy, dx=None, accumulate=False):
    n, H2, W2, C = dy.shape
    g = dy.float().view(n, H2 // 2, 2, W2 // 2, 2, C).sum(dim=(2, 4))
    if dx is None:
        return _bf(g)
    dx.copy_(_bf(dx.float() + g) if accumulate else _bf(g))
    return dx


def zero_insert2x(x, off):
    n, H, W, C = x.shape
    y = torch.zeros(n, 2 * H, 2 * W, C, dtype=BF16)
    y[:, off::2, off::2] = x
    return y


def concat_channels(a, b):
    assert a.dtype == b.dtype == BF16 and a.shape[-1] % 8 == 0 and b.shape[-1] % 8 == 0
    return torch.cat([a, b], -1).contiguous()


def slice_channels(src, c_off, Cd, dst=None, accumulate=False):
    assert src.dtype == BF16 and (dst is None or dst.dtype == BF16)
    s = src[..., c_off:c_off + Cd]
    if dst is None:
        return s.contiguous()
    dst.copy_(_bf(dst.float() + s.float()) if accumulate else s)
    return dst


def nchw_to_nhwc(x):
    return _bf(x.permute(0, 2, 3, 1)).contiguous()


def nhwc_to_nchw_f32(x, out=None, accumulate=False):
    y = x.float().permute(0, 3, 1, 2)
    if out is None:
        return y.contiguous()
    out.copy_(out + y if accumulate else y)
    return out


def f32_to_bf16(x):
    return _bf(x)


# ------------------------------------------------------------------------------------------------------------ UNet edges
def conv_in(x, w, bias, cout):
    wf = w.float().reshape(cout, 3, 3, -1).permute(0, 3, 1, 2)
    y = F.conv2d(_bf(x).float(), wf, bias, padding=1)
    return _bf(y.permute(0, 2, 3, 1)).contiguous()


def conv_out(x, w, bias):
    wf = w.float().permute(0, 3, 1, 2)                                # [4, C, 3, 3]
    return F.conv2d(x.float().permute(0, 3, 1, 2), wf, bias, padding=1).contiguous()


def conv_out_bwd(dy, w, C_):
    wf = w.float().permute(0, 3, 1, 2)
    dx = F.conv_transpose2d(dy.float(), wf, padding=1)
    return _bf(dx.permute(0, 2, 3, 1)).contiguous()


def timestep_embedding(t, dim):
    t = t.to(torch.float32)
    half = dim // 2
    f = torch.exp(-math.log(10000.0) * torch.arange(half, dtype=torch.float32) / half)
    a = t[:, None] * f[None, :]
    return torch.cat([torch.cos(a), torch.sin(a)], -1)


def small_linear(x, w, bias, silu_in=False, silu_out=False):
    xi = F.silu(x) if silu_in else x
    y = xi @ w.float().t()
    if bias is not None:
        y = y + bias
    return F.silu(y) if silu_out else y


def mse_loss(pred, target, gscale=1.0, need_grad=True, out=None):
    assert pred.dtype == target.dtype == torch.float32 and (out is None or out.dtype == torch.float32)
    d = pred - target
    loss = (d * d).mean().reshape(1)
    g = (2.0 * gscale / pred.numel()) * d
    if out is not None:
        out.copy_(g)
        return loss, out
    return loss, (g if need_grad else None)


def add_noise(x0, sqrt_ac, sqrt_1mac, step_counter, seed, v_prediction=False, out=None):
    """cl_add_noise through the numpy Philox restatement of its counter layout (oracle/sampler_ref.device_noise)."""
    from oracle import sampler_ref as SR

    B = x0.shape[0]
    per = x0.numel() // B
    noise, ts = SR.device_noise(int(seed) & (2**64 - 1), int(step_counter), B, per, sqrt_ac.numel())
    noise = torch.from_numpy(noise).view(x0.shape)
    ts = torch.from_numpy(ts)
    a = sqrt_ac[ts].view(B, *([1] * (x0.dim() - 1)))
    b = sqrt_1mac[ts].view(B, *([1] * (x0.dim() - 1)))
    noisy = a * x0 + b * noise
    target = a * noise - b * x0 if v_prediction else noise
    step_counter += 1
    res = (noisy, target, ts.float())
    if out is not None:
        for o, r in zip(out, res):
            o.copy_(r)
        return out
    return res


# ------------------------------------------------------------------------------------------------------------ LoRA side path
def _pack_run(self):
    for d, (src, dst) in zip(self.descs, self._keep):
        v = float(d.mul) * _sv(src, (d.r, d.K), (d.s_j, d.s_k)).float()      # v[j, k]
        if d.kind == 0:
            hi = _bf(v)
            lo = _bf(v - hi.float())
            _sv(dst, (d.r, d.K), (d.ld, 1), d.row_off * d.ld).copy_(hi)
            _sv(dst, (d.r, d.K), (d.ld, 1), (8 + d.row_off) * d.ld).copy_(lo)
        elif d.kind == 1:
            _sv(dst, (d.K, d.r), (d.ld, 1), d.row_off).copy_(v.t())
        else:
            hi = _bf(v).t()
            _sv(dst, (d.K, d.r), (d.ld, 1), d.row_off).copy_(hi)
            _sv(dst, (d.K, d.r), (d.ld, 1), 8 + d.row_off).copy_(hi)


def skinny_atb(a, r, b, out, so_j, so_c, alpha):
    b2 = b.reshape(-1, b.shape[-1]) if b.is_contiguous() else b
    assert b2.shape[0] == a.shape[0] and a.dtype == torch.float32 and b2.dtype == BF16 and out.dtype == torch.float32
    Cc = b2.shape[1]
    assert 1 <= r <= 8 and Cc % 8 == 0 and Cc // 8 <= 512 and b2.stride(1) == 1 and b2.stride(0) % 8 == 0, "cl_skinny_atb: bad descriptor"
    assert max(1, 512 // (Cc // 8)) * r * Cc * 4 <= 200 * 1024, "cl_skinny_atb_batch: shared memory"
    o = _sv(out, (r, b2.shape[1]), (so_j, so_c))
    o += float(alpha) * (a[:, :r].float().t() @ b2.float())


def _skinny_add(self, a, r, b, out, so_j, so_c, alpha):
    """Like the real queue (ops.SkinnyQueue): reductions are only COLLECTED here and run in batches of CL_SKINNY_MAX or at flush()
    - code that reads a gradient before flushing must see it missing here too."""
    self.keep.append((a, r, b, out, so_j, so_c, alpha))
    self.descs.append(None)
    if len(self.keep) >= self._max:
        _skinny_flush(self)


def _skinny_flush(self):
    for args in self.keep:
        skinny_atb(*args)
    self.descs, self.keep = [], []


def rowdot(a, u):
    a2 = a.reshape(-1, a.shape[-1]) if a.is_contiguous() else a
    assert a2.dtype == BF16 and u.dtype == torch.float32 and u.is_contiguous() and u.shape[1] in (4, 8)
    assert a2.shape[1] % 8 == 0 and a2.stride(0) % 8 == 0 and a2.shape[1] * u.shape[1] * 4 <= 48 * 1024, "cl_rowdot: bad args"
    return a2.float() @ u


def rowmat(a, w, sw_i, sw_j, I, J, alpha, out, ldo, out_mode=0, col_off=0, lo_off=0, accumulate=False):
    M = a.shape[0]
    assert 1 <= I <= 8 and 1 <= J <= 8 and a.dtype == torch.float32, "cl_rowmat: bad args"
    Wm = _sv(w, (I, J), (sw_i, sw_j)).float()
    s = float(alpha) * (a[:, :J].float() @ Wm.t())                       # [M, I]
    if out_mode == 0:
        o = _sv(out, (M, I), (ldo, 1))
        o.copy_(o + s if accumulate else s)
    else:
        hi = _bf(s)
        _sv(out, (M, I), (ldo, 1), col_off).copy_(hi)
        _sv(out, (M, I), (ldo, 1), col_off + lo_off).copy_(_bf(s - hi.float()))


def skinny_small(a, I, b, J, out, alpha):
    assert I <= 8 and J <= 8, "cl_skinny_small: bad args"
    assert a.dtype == b.dtype == out.dtype == torch.float32 and a.shape[0] == b.shape[0]
    out.view(-1)[: I * J].view(I, J).add_(float(alpha) * (a[:, :I].float().t() @ b[:, :J].float()))


def small_matmul(a, sa_i, sa_j, b, sb_j, sb_k, out, so_i, so_k, I, J, K, alpha=1.0, accumulate=False):
    assert a.dtype == b.dtype == out.dtype == torch.float32
    r = float(alpha) * (_sv(a, (I, J), (sa_i, sa_j)).float() @ _sv(b, (J, K), (sb_j, sb_k)).float())
    o = _sv(out, (I, K), (so_i, so_k))
    o.copy_(o + r if accumulate else r)


def hilo_combine(src, nb):
    assert src.dtype == torch.float32 and src.is_contiguous() and src.shape[1] == 16 * nb
    M = src.shape[0]
    s = src.view(M, nb, 16)
    return (s[..., :8] + s[..., 8:]).reshape(M, 8 * nb).contiguous()


def rank_update(x, t, tab, alpha, out=None):
    C = x.shape[-1]
    rp = tab.shape[1]
    assert x.dtype == BF16 and x.is_contiguous() and tab.is_contiguous() and tab.shape[0] == C and t.dtype == torch.float32
    assert C % 8 == 0 and rp in (4, 8) and C * rp * 4 <= 48 * 1024 and t.shape[1] >= rp, "cl_rank_update: bad args"
    y = _bf(x.float().reshape(-1, C) + float(alpha) * (t[:, :rp] @ tab.t())).reshape(x.shape)
    if out is None:
        return y
    out.copy_(y)
    return out


def v2_inject_fwd(x, th16, uc, rc, tab, alpha):
    C = x.shape[-1]
    assert C % 8 == 0 and 1 <= rc <= 4 and C * 16 <= 48 * 1024 and tab.shape == (C, 4), "cl_v2_inject_fwd: bad args"
    t = (th16[:, :8] + th16[:, 8:]).clone()
    if uc is not None:
        t[:, :rc] += uc[:, :rc]
    y = _bf(x.float().reshape(-1, C) + float(alpha) * (t[:, :4] @ tab.t())).reshape(x.shape)
    return y, t


def v2_inject_bwd(dy, up_tab, down_tab, alpha, need_dh):
    C = dy.shape[-1]
    assert C % 8 == 0 and C <= 1280 and up_tab.shape == (C, 4) and (not need_dh or down_tab.shape == (C, 4)), "cl_v2_inject_bwd: bad args"
    d2 = dy.float().reshape(-1, C)
    dt = d2 @ up_tab
    dh = _bf(d2 + float(alpha) * (dt @ down_tab.t())).reshape(dy.shape) if need_dh else None
    return dt, dh


def rank4_project_update(x, proj_tab, upd_tab, uc, rc, alpha):
    C = x.shape[-1]
    assert C % 8 == 0 and C <= 1280 and 0 <= rc <= 4 and proj_tab.shape == (C, 4) and upd_tab.shape == (C, 4), "cl_rank4_project_update"
    x2 = x.float().reshape(-1, C)
    t = x2 @ proj_tab
    if uc is not None:
        t[:, :rc] += uc[:, :rc]
    y = _bf(x2 + float(alpha) * (t @ upd_tab.t())).reshape(x.shape)
    return y, t


def cast_matrix(src, I, J, s_i, s_j, alpha=1.0, out=None):
    v = _bf(float(alpha) * _sv(src, (I, J), (s_i, s_j)))
    if out is None:
        return v.contiguous()
    out.copy_(v)
    return out


def axpy_matrix(src, dst, alpha=1.0):
    I = src.shape[0]
    dst += float(alpha) * src.reshape(I, -1)


# ------------------------------------------------------------------------------------------------------------ hint encoder
def _conv_nchw(x, w, ksize, stride, pad_lo):
    if ksize == 1:
        return F.conv2d(x, w, stride=stride)
    if stride == 1:
        return F.conv2d(x, w, padding=1)
    if pad_lo == 1:
        return F.conv2d(x, w, stride=2, padding=1)
    return F.conv2d(F.pad(x, (0, 1, 0, 1)), w, stride=2)


def conv_wgrad(dy, x, dw, ksize, stride=1, pad_lo=1, alpha=1.0):
    xin = x.float().permute(0, 3, 1, 2)
    w = torch.zeros(dw.shape, requires_grad=True)
    with torch.enable_grad():
        y = _conv_nchw(xin, w, ksize, stride, pad_lo)
        (gw,) = torch.autograd.grad(y, w, dy.float().permute(0, 3, 1, 2))
    dw += float(alpha) * gw


def conv_weight_prep(w, wf, wd=None):
    Cout, Cin, k, _ = w.shape
    wf.view(-1)[: Cout * k * k * Cin].view(Cout, k * k, Cin).copy_(_bf(w.detach().permute(0, 2, 3, 1).reshape(Cout, k * k, Cin)))
    if wd is not None:
        wd.view(-1)[: Cout * k * k * Cin].view(Cin, k * k, Cout).copy_(
            _bf(w.detach().flip(2, 3).permute(1, 2, 3, 0).reshape(Cin, k * k, Cout)))


def colsum(x, out, alpha=1.0):
    assert x.dtype == BF16 and out.dtype == torch.float32
    C = x.shape[-1]
    out += float(alpha) * x.float().reshape(-1, C).sum(0)


def conv_in_wgrad(x, dy, dw):
    w = torch.zeros(dw.shape, requires_grad=True)
    with torch.enable_grad():
        y = F.conv2d(_bf(x).float(), w, padding=1)
        (gw,) = torch.autograd.grad(y, w, dy.float().permute(0, 3, 1, 2))
    dw += gw


# ------------------------------------------------------------------------------------------------------------ optimizer
def sumsq(x, out):
    out += (x.double() ** 2).sum().float()


def _adamw(p, g, m, v, lr, beta1, beta2, eps, wd, step, gnorm_sq, max_norm, grad_scale, zero_grad):
    coef = float(grad_scale)
    if gnorm_sq is not None and max_norm > 0:
        total = math.sqrt(float(gnorm_sq)) * grad_scale
        coef *= min(max_norm / (total + 1e-6), 1.0)
    gi = g * coef
    p.mul_(1.0 - lr * wd)
    m.mul_(beta1).add_(gi, alpha=1.0 - beta1)
    v.mul_(beta2).addcmul_(gi, gi, value=1.0 - beta2)
    bc1 = 1.0 - beta1 ** step
    bc2s = math.sqrt(1.0 - beta2 ** step)
    p.sub_((lr / bc1) * (m / (v.sqrt() / bc2s + eps)))
    if zero_grad:
        g.zero_()


def adamw(p, g, m, v, lr, beta1, beta2, eps, wd, step, gnorm_sq=None, max_norm=0.0, grad_scale=1.0, zero_grad=True):
    _adamw(p, g, m, v, lr, beta1, beta2, eps, wd, int(step), gnorm_sq, max_norm, grad_scale, zero_grad)


def step_begin(gnorm_sq, step_dev):
    gnorm_sq.zero_()
    step_dev += 1


def adamw_dev(p, g, m, v, lr, beta1, beta2, eps, wd, step_dev, gnorm_sq=None, max_norm=0.0, grad_scale=1.0, zero_grad=True):
    _adamw(p, g, m, v, lr, beta1, beta2, eps, wd, int(step_dev), gnorm_sq, max_norm, grad_scale, zero_grad)


# ------------------------------------------------------------------------------------------------------------ sampler / VAE / CLIP
def _cfg(eps2, guidance):
    u, c = eps2.reshape(2, -1)
    return u + guidance * (c - u)


def cfg_ddim_step(eps2, latents, guidance, a_t, a_prev):
    eps = _cfg(eps2, guidance).view_as(latents)
    x0 = (latents - math.sqrt(1 - a_t) * eps) / math.sqrt(a_t)
    latents.copy_(math.sqrt(a_prev) * x0 + math.sqrt(1 - a_prev) * eps)


def cfg_dpmpp_step(eps2, latents, x0_prev, guidance, alpha_s, sigma_s, c_x, c_m0, c_m1):
    eps = _cfg(eps2, guidance).view_as(latents)
    x0 = (latents - sigma_s * eps) / alpha_s
    latents.copy_(c_x * latents + c_m0 * x0 + c_m1 * x0_prev)
    x0_prev.copy_(x0)


def sampler_prep(latents, x2, tt, ts_table, step_ctr):
    x2.view(2, -1).copy_(latents.reshape(1, -1).expand(2, -1))
    tt.fill_(float(ts_table[int(step_ctr)]))


def cfg_solver_step_dev(eps2, latents, x0_prev, coef, step_ctr, guidance, kind):
    c = [float(v) for v in coef[int(step_ctr)]]
    eps = _cfg(eps2, guidance).view_as(latents)
    if kind == 0:
        x0 = (latents - c[1] * eps) / c[0]
        latents.copy_(c[2] * x0 + c[3] * eps)
    else:
        x0 = (latents - c[1] * eps) / c[0]
        latents.copy_(c[2] * latents + c[3] * x0 + c[4] * x0_prev)
        x0_prev.copy_(x0)
    step_ctr += 1


def softmax_rows(s, scale):
    return _bf(torch.softmax(scale * s, -1))


def clip_embed(ids, tok, pos):
    B, T = ids.shape
    return _bf(tok[ids].float() + pos[:T].float()[None])


def quick_gelu_(x):
    xf = x.float()
    x.copy_(_bf(xf * torch.sigmoid(1.702 * xf)))
    return x


def causal_attention_small(qkv, B, T, heads, scale):
    C = qkv.shape[1] // 3
    q, k, v = (_heads(t.reshape(B, T, C), heads) for t in qkv.split(C, 1))
    s = (q @ k.transpose(-1, -2)) * scale
    s = s.masked_fill(torch.ones(T, T, dtype=torch.bool).triu(1), float("-inf"))
    o = torch.softmax(s, -1) @ v
    return _bf(o.permute(0, 2, 1, 3).reshape(B * T, C))


def channel_affine_nchw(x, mul, shift):
    return mul * x + shift.view(1, -1, *([1] * (x.dim() - 2)))


# ------------------------------------------------------------------------------------------------------------ install
_NO_SHADOW = {"add_noise"}        # real wrapper insists on a CUDA step counter before it reaches the launcher


def _accepted(call, name):
    """Run the real wrapper; the launcher must get past its argument checks (it then dies at the first CUDA call: status -2)."""
    from controllora_b200._lib import CLError

    try:
        call()
    except CLError as e:
        if "status -2" not in str(e):
            raise AssertionError(f"{name}: the real launcher rejects the arguments the host program passes: {e}") from None


def _shadow(name, real, emu):
    if name in _NO_SHADOW:
        return emu

    def both(*a, **k):
        _accepted(lambda: real(*a, **k), name)
        return emu(*a, **k)

    both.__name__ = name
    return both


_FUNCS = [
    "gemm", "attention_fwd", "attention_bwd", "groupnorm_fwd", "groupnorm_bwd", "layernorm_fwd", "layernorm_bwd", "geglu_fwd",
    "geglu_bwd", "add", "upsample2x_fwd", "upsample2x_bwd", "zero_insert2x", "concat_channels", "slice_channels", "nchw_to_nhwc",
    "nhwc_to_nchw_f32", "f32_to_bf16", "conv_in", "conv_out", "conv_out_bwd", "timestep_embedding", "small_linear", "mse_loss", "add_noise",
    "skinny_atb", "rowdot", "rowmat", "skinny_small", "small_matmul", "hilo_combine", "rank_update", "v2_inject_fwd",
    "v2_inject_bwd", "rank4_project_update", "cast_matrix", "axpy_matrix", "conv_wgrad", "conv_weight_prep", "colsum",
    "conv_in_wgrad", "sumsq", "adamw", "step_begin", "adamw_dev", "cfg_ddim_step", "cfg_dpmpp_step", "sampler_prep",
    "cfg_solver_step_dev", "softmax_rows", "clip_embed", "quick_gelu_", "causal_attention_small", "channel_affine_nchw",
]


def install() -> None:
    """Replace the kernel wrappers of controllora_b200.ops by the CPU restatements above (idempotent; `uninstall()` undoes it)."""
    from controllora_b200 import ops

    if _INSTALLED:
        return
    import os

    # The real wrappers run on CPU tensors and count on the launcher failing at its first CUDA call.  On a machine with a GPU that
    # call would succeed and launch kernels on host pointers, so host-logic mode hides every device from the process; it has to be
    # installed before anything in the process has initialised CUDA.
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    if torch.cuda.device_count() != 0:
        raise RuntimeError("host-logic mode (CLB_EMU=1) must be installed before the process initialises CUDA")
    _INSTALLED["env"] = os.environ.get("CLB_DRYRUN")
    os.environ["CLB_DRYRUN"] = "1"          # the package's require_cuda() guards accept CPU tensors in host-logic mode only
    g = globals()
    ng = torch.no_grad()                    # kernels are invisible to autograd; so are their restatements
    _INSTALLED["_req"], _INSTALLED["_stream"] = ops._req, ops._stream
    ops._req = _req_dtype_only             # the real wrappers run too (argument marshalling + launcher validation), on CPU tensors
    ops._stream = lambda: None
    for name in _FUNCS:
        _INSTALLED[name] = getattr(ops, name)
        setattr(ops, name, ng(_shadow(name, _INSTALLED[name], g[name])))
    _INSTALLED["PackPlan.run"] = ops.PackPlan.run
    _INSTALLED["SkinnyQueue.add"] = ops.SkinnyQueue.add
    _INSTALLED["SkinnyQueue.flush"] = ops.SkinnyQueue.flush
    real_pack_run, real_add, real_flush = ops.PackPlan.run, ops.SkinnyQueue.add, ops.SkinnyQueue.flush

    def pack_run(self):
        _accepted(lambda: real_pack_run(self), "cl_lora_pack_batch")
        _pack_run(self)

    def skinny_add(self, a, r, b, out, so_j, so_c, alpha):
        # the real queue object collects real descriptors; a private real queue is validated and discarded at flush time
        q = self.__dict__.setdefault("_real_q", None)
        if q is None:
            q = self.__dict__["_real_q"] = object.__new__(ops.SkinnyQueue)
            ops.SkinnyQueue.__init__(q)
        b2 = b.view(-1, b.shape[-1]) if b.is_contiguous() else b
        d = q._Desc()
        d.a, d.lda, d.r = a.data_ptr(), a.stride(0), r
        d.b, d.ldb = b2.data_ptr(), b2.stride(0)
        d.out, d.so_j, d.so_c = out.data_ptr(), so_j, so_c
        d.alpha, d.M, d.C = float(alpha), b2.shape[0], b2.shape[1]
        q.descs.append(d)
        if len(q.descs) >= q._max:          # the real queue launches a full batch here
            _accepted(lambda: real_flush(q), "cl_skinny_atb_batch")
            q.descs, q.keep = [], []
        _skinny_add(self, a, r, b, out, so_j, so_c, alpha)

    def skinny_flush(self):
        q = self.__dict__.get("_real_q")
        if q is not None and q.descs:
            _accepted(lambda: real_flush(q), "cl_skinny_atb_batch")
            q.descs, q.keep = [], []
        _skinny_flush(self)

    ops.PackPlan.run = ng(pack_run)
    ops.SkinnyQueue.add = ng(skinny_add)
    ops.SkinnyQueue.flush = ng(skinny_flush)


def uninstall() -> None:
    from controllora_b200 import ops

    if not _INSTALLED:
        return
    import os

    env = _INSTALLED.pop("env")
    if env is None:
        os.environ.pop("CLB_DRYRUN", None)
    else:
        os.environ["CLB_DRYRUN"] = env
    ops._req, ops._stream = _INSTALLED.pop("_req"), _INSTALLED.pop("_stream")
    ops.PackPlan.run = _INSTALLED.pop("PackPlan.run")
    ops.SkinnyQueue.add = _INSTALLED.pop("SkinnyQueue.add")
    ops.SkinnyQueue.flush = _INSTALLED.pop("SkinnyQueue.flush")
    for name in list(_INSTALLED):
        setattr(ops, name, _INSTALLED.pop(name))


@contextlib.contextmanager
def installed():
    install()
    try:
        yield
    finally:
        uninstall()
