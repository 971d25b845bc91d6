"""GPU parity checks: every sm_100a kernel (through the C ABI) against the fp32 PyTorch composite it
replaces, and the drop-in MIDIModel against the CPU oracle restatement run on the same device.
Each check returns {metric_name: value}; thresholds live in THRESH (asserted by test_gpu_*.py and
reported by tools/run_gpu_checks.py).  Seeds are fixed; sizes are chosen so the oracle finishes in
seconds and so that odd / ragged shapes are covered (S=2047, V=3406, rows not /128, L<8, empty)."""
from __future__ import annotations

import math
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "midi-model_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

from midi_b200 import lib, ops  # noqa: E402
from oracle import midi_oracle as O  # noqa: E402

DEV = "cuda"
BF = torch.bfloat16


def rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def randn(*shape, scale=1.0, seed=0, dtype=BF):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(*shape, generator=g, device=DEV, dtype=torch.float32) * scale).to(dtype)


# ------------------------------------------------------------------------------------------ GEMM
def check_gemm_fwd():
    out = {}
    for i, (M, N, K) in enumerate([(256, 256, 128), (1000, 1024, 1024), (2048, 3072, 1024), (384, 8192, 1024),
                                   (4096, 1024, 4096), (130, 136, 72)]):
        a, w = randn(M, K, seed=i), randn(N, K, scale=0.05, seed=100 + i)
        y = ops.linear(a, w)
        ref = (a.float() @ w.float().T)
        out[f"gemm_tn_{M}x{N}x{K}"] = rel(y.float(), ref)
    # residual epilogue: bf16(bf16(acc) + r)
    M, N, K = 1024, 1024, 1024
    a, w, r = randn(M, K, seed=7), randn(N, K, scale=0.05, seed=8), randn(M, N, seed=9)
    y = ops.linear(a, w, residual=r)
    ref = ((a.float() @ w.float().T).to(BF).float() + r.float())
    out["gemm_residual"] = rel(y.float(), ref)
    # N = 3406 (vocab): pitch 3408, trailing columns zero
    a, w = randn(520, 1024, seed=11), randn(3406, 1024, scale=0.05, seed=12)
    y = ops.linear(a, w, pitch=3408)
    out["gemm_vocab"] = rel(y[:, :3406].float(), a.float() @ w.float().T)
    out["gemm_vocab_padcols_absmax"] = float(y[:, 3406:].float().abs().max())
    return out


def check_gemm_swiglu():
    """gate|up GEMM with SwiGLU in the epilogue == plain GEMM + stand-alone SwiGLU kernel, bit for bit."""
    out = {}
    for i, (M, I, K) in enumerate([(300, 1024, 1024), (2048, 4096, 1024), (1000, 128, 256)]):
        x, w = randn(M, K, seed=60 + i), randn(2 * I, K, scale=0.05, seed=70 + i)
        gu, act = ops.linear_swiglu(x, w)
        gu_ref = ops.linear(x, w)
        out[f"gemm_swiglu_gu_mismatch_{M}x{I}"] = float((gu != gu_ref).sum())
        out[f"gemm_swiglu_act_mismatch_{M}x{I}"] = float((act != ops.swiglu(gu_ref)).sum())
    return out


def check_gemm_dgrad():
    out = {}
    for i, (M, N, K) in enumerate([(256, 256, 128), (1000, 3072, 1024), (2048, 1024, 4096), (520, 3406, 1024)]):
        pitch = (N + 7) // 8 * 8
        dy = torch.zeros(M, pitch, device=DEV, dtype=BF)
        dy[:, :N] = randn(M, N, seed=20 + i)
        w = randn(N, K, scale=0.05, seed=30 + i)
        dx = ops.linear_dgrad(dy, w)
        out[f"gemm_dgrad_{M}x{N}x{K}"] = rel(dx.float(), dy[:, :N].float() @ w.float())
    return out


def check_gemm_wgrad():
    out = {}
    for i, (M, N, K) in enumerate([(256, 256, 128), (4096, 1024, 1024), (3000, 3072, 1024), (2048, 3406, 1024),
                                   (16384, 1024, 1024)]):
        pitch = (N + 7) // 8 * 8
        dy = torch.zeros(M, pitch, device=DEV, dtype=BF)
        dy[:, :N] = randn(M, N, seed=40 + i)
        x = randn(M, K, seed=50 + i)
        dw = torch.empty(N, K, device=DEV, dtype=BF)
        ops.linear_wgrad(dy, x, dw, accumulate=False)
        ref = dy[:, :N].float().T @ x.float()
        out[f"gemm_wgrad_{M}x{N}x{K}"] = rel(dw.float(), ref)
        if i == 1:
            ops.linear_wgrad(dy, x, dw, accumulate=True)
            out["gemm_wgrad_accumulate"] = rel(dw.float(), 2 * ref)
    return out


# ------------------------------------------------------------------------------------------ elementwise
def check_elementwise():
    out = {}
    V, H = 3406, 1024
    table = randn(V, H, scale=0.02, seed=1)
    ids = torch.randint(0, V, (300, 8), device=DEV, generator=torch.Generator(device=DEV).manual_seed(2))
    ids[5] = 0
    y = ops.embed_sum(ids, table)
    ref = F.embedding(ids, table).float().sum(-2).to(BF)
    out["embed_sum_maxabs"] = float((y.float() - ref.float()).abs().max())
    # embedding backward (outer: 8 ids per gradient row; pad row zero)
    dout = randn(300, H, seed=3)
    dtab = torch.empty(V, H, device=DEV, dtype=BF)
    ops.embed_bwd(ids.view(-1), dout, dtab, per_row=8, row_stride=1, row_inner=0, row_off=0, pad_id=0, accumulate=False)
    t32 = table.float().clone().requires_grad_(True)
    F.embedding(ids, t32, padding_idx=0).sum(-2).backward(dout.float())
    out["embed_bwd"] = rel(dtab.float(), t32.grad)
    out["embed_bwd_padrow_absmax"] = float(dtab[0].float().abs().max())
    # inner input builder + its embedding backward (7 ids per event, rows e*8 + 1 + j)
    hid = randn(40, H, seed=4)
    ids7 = torch.randint(0, V, (40, 7), device=DEV, generator=torch.Generator(device=DEV).manual_seed(5))
    xin = ops.inner_input(hid, ids7, table)
    ref = torch.cat([hid[:, None], F.embedding(ids7, table)], 1).reshape(-1, H)
    out["inner_input_equal"] = float((xin != ref).sum())
    dx = randn(40 * 8, H, seed=6)
    ops.embed_bwd(ids7.view(-1), dx, dtab, per_row=7, row_stride=8, row_inner=1, row_off=1, pad_id=0, accumulate=False)
    t32 = table.float().clone().requires_grad_(True)
    F.embedding(ids7, t32, padding_idx=0).backward(dx.float().view(40, 8, H)[:, 1:])
    out["inner_embed_bwd"] = rel(dtab.float(), t32.grad)
    # rmsnorm
    for M in (1, 300, 5000):
        x, w = randn(M, H, seed=7), (1 + 0.1 * randn(H, seed=8).float()).to(BF)
        y, rstd = ops.rmsnorm(x, w, 1e-6, want_rstd=True)
        ref = O.rmsnorm(x, w, 1e-6)
        out[f"rmsnorm_fwd_mismatch_{M}"] = float((y != ref).float().mean())
        out[f"rmsnorm_fwd_{M}"] = rel(y.float(), ref.float())
        dy, dres = randn(M, H, seed=9), randn(M, H, seed=10)
        dw = torch.empty(H, device=DEV, dtype=BF)
        dx = ops.rmsnorm_bwd(dy, x, w, rstd, dres, dw, False)
        x32, w32 = x.float().requires_grad_(True), w.float().requires_grad_(True)
        v = x32.pow(2).mean(-1, keepdim=True)
        (w32 * (x32 * torch.rsqrt(v + 1e-6))).backward(dy.float())
        out[f"rmsnorm_bwd_dx_{M}"] = rel(dx.float(), x32.grad + dres.float())
        out[f"rmsnorm_bwd_dw_{M}"] = rel(dw.float(), w32.grad)
    # rope (bf16-rounded inv_freq, as after model.to(bf16)) on packed qkv
    for (S, nh, D) in ((37, 16, 64), (8, 4, 256)):
        Hh = nh * D
        inv = O.default_inv_freq(D).to(BF).to(DEV)
        cos, sin = ops.rope_table(inv, S)
        rc, rs = O.rope_cos_sin(inv, torch.arange(S, device=DEV), BF)
        out[f"rope_table_mismatch_D{D}"] = float((cos != rc[:, :D // 2]).sum() + (sin != rs[:, :D // 2]).sum())
        qkv = randn(3 * S, 3 * Hh, seed=11)
        q0 = qkv.clone()
        ops.rope_qk_(qkv, cos, sin, S, Hh, D)
        q = q0[:, :Hh].view(3, S, nh, D).transpose(1, 2)
        k = q0[:, Hh:2 * Hh].view(3, S, nh, D).transpose(1, 2)
        rq = O.apply_rope(q, rc, rs).transpose(1, 2).reshape(3 * S, Hh)
        rk = O.apply_rope(k, rc, rs).transpose(1, 2).reshape(3 * S, Hh)
        out[f"rope_fwd_mismatch_D{D}"] = float((qkv[:, :Hh] != rq).sum() + (qkv[:, Hh:2 * Hh] != rk).sum()
                                               + (qkv[:, 2 * Hh:] != q0[:, 2 * Hh:]).sum())
        # backward == transpose of the rotation: <R x, y> == <x, R^T y>
        d = randn(3 * S, 3 * Hh, seed=12)
        d_in = d.clone()
        ops.rope_qk_(d_in, cos, sin, S, Hh, D, backward=True)
        c32 = torch.cat([cos, cos], -1).float()
        s32 = torch.cat([sin, sin], -1).float()

        def rot32(t):
            t4 = t.float().view(3, S, nh, D)
            return (t4 * c32[None, :, None] + O.rotate_half(t4) * s32[None, :, None]).reshape(3 * S, Hh)
        lhs = (rot32(q0[:, :Hh]) * d[:, :Hh].float()).sum()
        rhs = (q0[:, :Hh].float() * d_in[:, :Hh].float()).sum()
        out[f"rope_bwd_adjoint_D{D}"] = float((lhs - rhs).abs() / lhs.abs().clamp_min(1e-6))
    # swiglu
    gu = randn(777, 2 * 1024, seed=13)
    act = ops.swiglu(gu)
    ref = F.silu(gu[:, :1024]) * gu[:, 1024:]
    out["swiglu_fwd_mismatch"] = float((act != ref).float().mean())
    dact = randn(777, 1024, seed=14)
    dgu = ops.swiglu_bwd(gu, dact)
    g32 = gu.float().requires_grad_(True)
    (F.silu(g32[:, :1024]) * g32[:, 1024:]).backward(dact.float())
    out["swiglu_bwd"] = rel(dgu.float(), g32.grad)
    return out


# ------------------------------------------------------------------------------------------ attention
def _sdpa_ref(q, k, v, off):
    # q (B,h,Sq,d) fp32; causal with offset
    Sq, Sk = q.shape[-2], k.shape[-2]
    s = q @ k.transpose(-1, -2) / math.sqrt(q.shape[-1])
    m = torch.arange(Sk, device=q.device)[None] > (torch.arange(Sq, device=q.device)[:, None] + off)
    s = s.masked_fill(m, float("-inf"))
    return torch.softmax(s, -1) @ v


def check_attn_flash():
    """Both attention implementations, forward (output and lse) and backward, directly against fp32 autograd."""
    out = {}
    for impl in ("tc", "mma"):
        for (B, S, nh) in ((2, 64, 4), (1, 200, 16), (2, 2047, 16)):
            D, H = 64, nh * 64
            qkv = randn(B * S, 3 * H, seed=S)
            o, lse = ops.attn_causal_fwd(qkv, B, S, nh, D, want_lse=True, impl=impl)
            q32 = qkv.float().view(B, S, 3, nh, D).permute(2, 0, 3, 1, 4).clone().requires_grad_(True)
            ref = _sdpa_ref(q32[0], q32[1], q32[2], 0)
            out[f"flash_fwd_S{S}_{impl}"] = rel(o.float().view(B, S, nh, D).transpose(1, 2), ref)
            sc = (q32[0] @ q32[1].transpose(-1, -2)) / 8.0
            msk = torch.triu(torch.ones(S, S, device=DEV, dtype=torch.bool), 1)
            out[f"flash_lse_S{S}_{impl}"] = rel(lse, torch.logsumexp(sc.masked_fill(msk, float("-inf")), -1))
            do = randn(B * S, H, seed=S + 1)
            dqkv = ops.attn_causal_bwd(qkv, o, do, lse, B, S, nh, D, impl=impl)
            ref.backward(do.float().view(B, S, nh, D).transpose(1, 2))
            g = q32.grad.permute(1, 3, 0, 2, 4).reshape(B * S, 3 * H)
            out[f"flash_bwd_dq_S{S}_{impl}"] = rel(dqkv[:, :H].float(), g[:, :H])
            out[f"flash_bwd_dk_S{S}_{impl}"] = rel(dqkv[:, H:2 * H].float(), g[:, H:2 * H])
            out[f"flash_bwd_dv_S{S}_{impl}"] = rel(dqkv[:, 2 * H:].float(), g[:, 2 * H:])
    return out


def check_attn_tc05():
    """tcgen05 / TMEM / TMA attention forward vs fp32 SDPA and vs the mma.sync kernel (same semantics)."""
    out = {}
    for (B, S, nh) in ((1, 128, 4), (2, 384, 16), (1, 200, 16), (2, 2047, 16), (8, 2048, 16)):
        D, H = 64, nh * 64
        qkv = randn(B * S, 3 * H, seed=S + B)
        o, lse = ops.attn_causal_fwd(qkv, B, S, nh, D, want_lse=True, impl="tc")
        o2, lse2 = ops.attn_causal_fwd(qkv, B, S, nh, D, want_lse=True, impl="mma")
        torch.cuda.synchronize()
        out[f"tc_vs_mma_fwd_B{B}_S{S}"] = rel(o.float(), o2.float())
        out[f"tc_vs_mma_lse_B{B}_S{S}"] = rel(lse, lse2)
        if B * S <= 4096:
            q32 = qkv.float().view(B, S, 3, nh, D).permute(2, 0, 3, 1, 4)
            ref = _sdpa_ref(q32[0], q32[1], q32[2], 0)
            out[f"tc_fwd_S{S}"] = rel(o.float().view(B, S, nh, D).transpose(1, 2), ref)
    # backward: tcgen05 kernel vs the mma.sync kernels and vs fp32 autograd
    for (B, S, nh) in ((1, 128, 4), (2, 384, 16), (1, 200, 16), (2, 2047, 16)):
        D, H = 64, nh * 64
        qkv = randn(B * S, 3 * H, seed=S + B + 7)
        do = randn(B * S, H, seed=S + B + 8)
        o, lse = ops.attn_causal_fwd(qkv, B, S, nh, D, want_lse=True, impl="mma")
        g_tc = ops.attn_causal_bwd(qkv, o, do, lse, B, S, nh, D, impl="tc")
        g_mm = ops.attn_causal_bwd(qkv, o, do, lse, B, S, nh, D, impl="mma")
        torch.cuda.synchronize()
        out[f"tc_vs_mma_bwd_dq_S{S}"] = rel(g_tc[:, :H].float(), g_mm[:, :H].float())
        out[f"tc_vs_mma_bwd_dk_S{S}"] = rel(g_tc[:, H:2 * H].float(), g_mm[:, H:2 * H].float())
        out[f"tc_vs_mma_bwd_dv_S{S}"] = rel(g_tc[:, 2 * H:].float(), g_mm[:, 2 * H:].float())
        q32 = qkv.float().view(B, S, 3, nh, D).permute(2, 0, 3, 1, 4).clone().requires_grad_(True)
        _sdpa_ref(q32[0], q32[1], q32[2], 0).backward(do.float().view(B, S, nh, D).transpose(1, 2))
        g = q32.grad.permute(1, 3, 0, 2, 4).reshape(B * S, 3 * H)
        out[f"tc_bwd_S{S}"] = rel(g_tc.float(), g)
        # with the RoPE backward fused
        inv = O.default_inv_freq(D).to(BF).to(DEV)
        cos, sin = ops.rope_table(inv, S)
        a = ops.attn_causal_bwd(qkv, o, do, lse, B, S, nh, D, rope=(cos, sin), impl="tc")
        bref = ops.attn_causal_bwd(qkv, o, do, lse, B, S, nh, D, rope=(cos, sin), impl="mma")
        out[f"tc_vs_mma_bwd_rope_S{S}"] = rel(a.float(), bref.float())
    # timing at the benchmark shape (B=8, S=2048, 16 heads): CUDA events, 10 launches each
    qkv = randn(8 * 2048, 3 * 1024, seed=1)
    do = randn(8 * 2048, 1024, seed=2)
    o, lse = ops.attn_causal_fwd(qkv, 8, 2048, 16, 64, want_lse=True, impl="mma")
    for impl in ("tc", "mma"):
        for _ in range(3):
            ops.attn_causal_bwd(qkv, o, do, lse, 8, 2048, 16, 64, impl=impl)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            ops.attn_causal_bwd(qkv, o, do, lse, 8, 2048, 16, 64, impl=impl)
        e1.record()
        torch.cuda.synchronize()
        out[f"time_ms_bwd_{impl}"] = e0.elapsed_time(e1) / 10
    for impl in ("tc", "mma"):
        for _ in range(3):
            ops.attn_causal_fwd(qkv, 8, 2048, 16, 64, want_lse=True, impl=impl)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            ops.attn_causal_fwd(qkv, 8, 2048, 16, 64, want_lse=True, impl=impl)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        out[f"time_ms_{impl}"] = ms
        out[f"tflops_{impl}"] = 4 * 8 * 16 * 2048 * 2049 / 2 * 64 / (ms * 1e-3) / 1e12
    return out


def check_attn_tiny():
    out = {}
    nh, D = 4, 256
    H = nh * D
    for (N, L) in ((50, 8), (33, 5), (7, 1)):
        qkv = randn(N * L, 3 * H, seed=L)
        o = ops.attn_tiny_fwd(qkv, N, L, nh, D)
        q32 = qkv.float().view(N, L, 3, nh, D).permute(2, 0, 3, 1, 4).clone().requires_grad_(True)
        ref = _sdpa_ref(q32[0], q32[1], q32[2], 0)
        out[f"tiny_fwd_L{L}"] = rel(o.float().view(N, L, nh, D).transpose(1, 2), ref)
        do = randn(N * L, H, seed=L + 1)
        dqkv = ops.attn_tiny_bwd(qkv, do, N, L, nh, D)
        ref.backward(do.float().view(N, L, nh, D).transpose(1, 2))
        g = q32.grad.permute(1, 3, 0, 2, 4).reshape(N * L, 3 * H)
        out[f"tiny_bwd_L{L}"] = rel(dqkv.float(), g)
    return out


def check_fused_rope():
    """RoPE fused into the QKV GEMM epilogue (bit-identical to GEMM + stand-alone rope kernel: same rounding
    points, same accumulation order) and into the attention backward kernels (one rounding fewer)."""
    out = {}
    for (nseq, S, nh, D) in ((3, 200, 16, 64), (40, 8, 4, 256)):
        H = nh * D
        inv = O.default_inv_freq(D).to(BF).to(DEV)
        cos, sin = ops.rope_table(inv, S)
        x, w = randn(nseq * S, 1024, seed=S), randn(3 * H, 1024, scale=0.05, seed=S + 1)
        fused = ops.linear_rope(x, w, cos, sin, S, D)
        ref = ops.linear(x, w)
        ops.rope_qk_(ref, cos, sin, S, H, D)
        out[f"linear_rope_mismatch_D{D}"] = float((fused != ref).sum())
        # backward: attention bwd with fused inverse rotation vs attention bwd + stand-alone rope backward
        do = randn(nseq * S, H, seed=S + 2)
        if D == 64:
            o, lse = ops.attn_causal_fwd(ref, nseq, S, nh, D, want_lse=True)
            a = ops.attn_causal_bwd(ref, o, do, lse, nseq, S, nh, D, rope=(cos, sin))
            b = ops.attn_causal_bwd(ref, o, do, lse, nseq, S, nh, D)
        else:
            a = ops.attn_tiny_bwd(ref, do, nseq, S, nh, D, rope=(cos, sin))
            b = ops.attn_tiny_bwd(ref, do, nseq, S, nh, D)
        ops.rope_qk_(b, cos, sin, S, H, D, backward=True)
        out[f"attn_bwd_fused_rope_D{D}"] = rel(a.float(), b.float())
        out[f"attn_bwd_fused_rope_v_mismatch_D{D}"] = float((a[:, 2 * H:] != b[:, 2 * H:]).sum())
        if D == 256:   # forward: RoPE fused into the token-level attention kernel (in-place rotation) == rope kernel + attention
            pre = ops.linear(x, w)
            o_f = ops.attn_tiny_fwd(pre, nseq, S, nh, D, rope=(cos, sin))
            o_r = ops.attn_tiny_fwd(ref, nseq, S, nh, D)
            out["tiny_fused_rope_out_mismatch"] = float((o_f != o_r).sum())
            out["tiny_fused_rope_qkv_mismatch"] = float((pre != ref).sum())
    return out


# ------------------------------------------------------------------------------------------ loss / optimizer
def check_loss_optim():
    out = {}
    V, pitch, R = 3406, 3408, 1000
    logits = torch.zeros(R, pitch, device=DEV, dtype=BF)
    logits[:, :V] = randn(R, V, scale=2.0, seed=1)
    tg = torch.randint(0, V, (R,), device=DEV, generator=torch.Generator(device=DEV).manual_seed(2))
    tg[::5] = 0
    lac, lse = ops.ce_fwd(logits, tg, V, 0)
    l32 = logits[:, :V].float().requires_grad_(True)
    ref = F.cross_entropy(l32, tg, ignore_index=0)
    out["ce_loss_abs"] = float((lac[0] - ref).abs())
    out["ce_count_abs"] = float((lac[1] - (tg != 0).sum()).abs())
    ref.backward()
    ops.ce_bwd_(logits, tg, lse, lac, V, 0, 1.0)
    out["ce_bwd"] = rel(logits[:, :V].float(), l32.grad)
    out["ce_bwd_padcols_absmax"] = float(logits[:, V:].float().abs().max())
    # all-ignored rows -> loss 0, zero grads
    tg0 = torch.zeros(R, dtype=torch.long, device=DEV)
    lac0, _ = ops.ce_fwd(logits, tg0, V, 0)
    out["ce_all_ignored_loss"] = float(lac0[0].abs())
    # AdamW + clip vs torch.optim.AdamW (fp32 reference on the bf16-rounded values)
    n = 256 * 1000
    p = randn(n, scale=0.05, seed=3)
    g = randn(n, scale=0.5, seed=4)
    nodecay = torch.zeros(n // 256, dtype=torch.uint8, device=DEV)
    nodecay[500:] = 1
    pr = p.float().clone()
    m = torch.zeros(n, device=DEV)
    v = torch.zeros(n, device=DEV)
    nc = torch.zeros(2, device=DEV)
    ws = torch.empty(lib.query("b200_gradnorm_parts") * 4, dtype=torch.uint8, device=DEV)
    pa = torch.nn.Parameter(pr[: 500 * 256].clone())
    pb = torch.nn.Parameter(pr[500 * 256:].clone())
    opt = torch.optim.AdamW([dict(params=[pa], weight_decay=0.01), dict(params=[pb], weight_decay=0.0)], lr=1e-3,
                            betas=(0.9, 0.99), eps=1e-8)
    pcur = p.clone()
    for step in (1, 2, 3):
        lib.call("b200_grad_clip_coef", g.data_ptr(), n, 1.0, nc.data_ptr(), ws.data_ptr(), ws.numel(), lib.stream())
        lib.call("b200_adamw_step", pcur.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), nodecay.data_ptr(), n, 1e-3,
                 0.9, 0.99, 1e-8, 0.01, step, nc.data_ptr(), lib.stream())
        pa.grad = g.float()[: 500 * 256].clone()
        pb.grad = g.float()[500 * 256:].clone()
        torch.nn.utils.clip_grad_norm_([pa, pb], 1.0)
        opt.step()
        # the kernel rounds the parameter to bf16 each step; mirror that in the reference
        with torch.no_grad():
            pa.copy_(pa.to(BF).float())
            pb.copy_(pb.to(BF).float())
    out["gradnorm_rel"] = float((nc[0] - g.float().norm()).abs() / g.float().norm())
    out["adamw_maxabs"] = float((pcur.float() - torch.cat([pa, pb]).detach()).abs().max())
    return out


# ------------------------------------------------------------------------------------------ decode kernels
def check_decode():
    out = {}
    from midi_b200 import decode as dec
    from midi_b200.engine import StackCfg
    # skinny GEMM
    for B in (1, 3, 8, 16):
        x, w, r = randn(B, 1024, seed=B), randn(3072, 1024, scale=0.05, seed=B + 1), randn(B, 3072, seed=B + 2)
        y = dec._linear(x, w)
        out[f"gemv_B{B}"] = rel(y.float(), x.float() @ w.float().T)
        y = dec._linear(x, w, residual=r)
        out[f"gemv_res_B{B}"] = rel(y.float(), (x.float() @ w.float().T).to(BF).float() + r.float())
    x, w = randn(2, 1024, seed=40), randn(3406, 1024, scale=0.05, seed=41)
    y = dec._lm_head(x, w, 3408)
    out["gemv_vocab"] = rel(y[:, :3406].float(), x.float() @ w.float().T)
    x, w = randn(4, 4096, seed=42), randn(1024, 4096, scale=0.05, seed=43)
    out["gemv_K4096"] = rel(dec._linear(x, w).float(), x.float() @ w.float().T)
    # paged KV append + single-query attention vs dense reference
    for (nh, D, page, T, sq) in ((16, 64, 64, 300, 1), (16, 64, 64, 1500, 1), (4, 256, 8, 6, 1), (16, 64, 64, 70, 5)):
        Bn, H = 2, nh * D
        cfg = StackCfg("net", 1, nh, H, 4 * H, 1e-6)
        kv = dec.PagedKV(cfg, Bn, 2048 if D == 64 else 8, page, DEV)
        past = T - sq
        hist = randn(Bn * past, 3 * H, seed=T) if past > 0 else None
        new = randn(Bn * sq, 3 * H, seed=T + 1)
        if past > 0:
            lib.call("b200_kv_append", hist.data_ptr(), kv.k[0].data_ptr(), kv.v[0].data_ptr(), kv.block_table.data_ptr(),
                     kv.max_pages, kv.page, nh, D, Bn, past, 0, None, 3 * H, lib.stream())
        lib.call("b200_kv_append", new.data_ptr(), kv.k[0].data_ptr(), kv.v[0].data_ptr(), kv.block_table.data_ptr(),
                 kv.max_pages, kv.page, nh, D, Bn, sq, past, None, 3 * H, lib.stream())
        n_split = max(1, (T + 255) // 256) if D == 64 else 1
        ws = torch.empty(lib.query("b200_attn_decode_workspace_bytes", Bn * sq, nh, D, n_split), dtype=torch.uint8, device=DEV)
        o = torch.empty(Bn * sq, H, device=DEV, dtype=BF)
        lib.call("b200_attn_decode", new.data_ptr(), kv.k[0].data_ptr(), kv.v[0].data_ptr(), kv.block_table.data_ptr(),
                 kv.max_pages, kv.page, o.data_ptr(), Bn, sq, nh, D, past, None, T, 3 * H, H, 1.0 / math.sqrt(D), n_split,
                 ws.data_ptr(), ws.numel(), lib.stream())
        allrows = new.view(Bn, sq, 3 * H) if past == 0 else torch.cat([hist.view(Bn, past, 3 * H), new.view(Bn, sq, 3 * H)], 1)
        q = new.view(Bn, sq, 3, nh, D)[:, :, 0].transpose(1, 2).float()
        k = allrows.view(Bn, T, 3, nh, D)[:, :, 1].transpose(1, 2).float()
        v = allrows.view(Bn, T, 3, nh, D)[:, :, 2].transpose(1, 2).float()
        ref = _sdpa_ref(q, k, v, past)
        out[f"decode_attn_D{D}_T{T}_q{sq}"] = rel(o.float().view(Bn, sq, nh, D).transpose(1, 2), ref)
    # sampler: greedy == argmax; top-k support; distribution sanity
    V = 3406
    g = torch.Generator(device=DEV).manual_seed(5)
    probs = torch.softmax(torch.randn(64, V, generator=g, device=DEV) * 3, -1)
    mask = torch.zeros(V, device=DEV)
    mask[9:137] = 1
    probs = (probs * mask)
    u = torch.rand(64, generator=g, device=DEV)
    o1 = torch.empty(64, dtype=torch.long, device=DEV)
    lib.call("b200_sample_topp_topk", probs.data_ptr(), 0, 64, V, V, 0.98, 1, u.data_ptr(), o1.data_ptr(), lib.stream())
    out["sampler_greedy_mismatch"] = float((o1 != probs.argmax(-1)).sum())
    lib.call("b200_sample_topp_topk", probs.data_ptr(), 0, 64, V, V, 0.98, 20, u.data_ptr(), o1.data_ptr(), lib.stream())
    top20 = probs.topk(20, -1).indices
    out["sampler_topk_outside"] = float((~(top20 == o1[:, None]).any(-1)).sum())
    # fused logits sampler (temperature softmax + grammar range + top-p/top-k) incl. the histogram top-k preselection:
    # greedy == argmax inside the allowed range, top-20 draws stay inside the 20 largest, for narrow and 2048-wide ranges
    from midi_b200.tokenizer_tables import TokenizerTables
    tokz = TokenizerTables("v2")
    glut = dec.GrammarLUT(tokz, DEV)
    logits = torch.zeros(64, 3408, device=DEV, dtype=BF)
    logits[:, :V] = (torch.randn(64, V, generator=g, device=DEV) * 2.5).to(BF)
    uu = torch.rand(64, generator=g, device=DEV)
    ev = torch.full((64,), tokz.event_ids["note"], dtype=torch.long, device=DEV)
    for step, pname in ((1, "time1"), (7, "duration"), (5, "pitch")):
        lo, hi = tokz.parameter_ids[pname][0], tokz.parameter_ids[pname][-1] + 1
        outb = torch.zeros(64, 8, dtype=torch.long, device=DEV)
        dec.sample_from_logits(logits, V, 1.0, 0.98, 1, step, ev, glut, uu, outb)
        ref_arg = logits[:, lo:hi].float().argmax(-1) + lo
        pr = torch.softmax(logits[:, :V].float(), -1).to(BF)
        # ties in bf16 probabilities are broken towards the lowest id: compare probabilities, not ids
        got = outb[:, step]
        out[f"logits_sampler_greedy_{pname}"] = float((pr.gather(1, got[:, None]) != pr.gather(1, ref_arg[:, None])).sum()
                                                       + ((got < lo) | (got >= hi)).sum())
        dec.sample_from_logits(logits, V, 1.0, 1.0, 20, step, ev, glut, uu, outb)
        got = outb[:, step]
        kth = pr[:, lo:hi].float().topk(20, -1).values[:, -1]
        out[f"logits_sampler_top20_{pname}"] = float((pr.gather(1, got[:, None])[:, 0].float() < kth).sum()
                                                      + ((got < lo) | (got >= hi)).sum())
    # empirical distribution of one row vs the reference algorithm's renormalised top-p/top-k weights
    row = probs[:1].repeat(4096, 1).contiguous()
    u = torch.rand(4096, generator=g, device=DEV)
    o2 = torch.empty(4096, dtype=torch.long, device=DEV)
    lib.call("b200_sample_topp_topk", row.data_ptr(), 0, 4096, V, V, 0.9, 8, u.data_ptr(), o2.data_ptr(), lib.stream())
    ps, pi = torch.sort(probs[0], descending=True)
    cs = torch.cumsum(ps, 0)
    ps = torch.where(cs - ps > 0.9, torch.zeros_like(ps), ps)
    ps[8:] = 0
    ps = ps / ps.sum()
    want = torch.zeros(V, device=DEV).scatter(0, pi, ps)
    emp = torch.bincount(o2, minlength=V).float() / 4096
    out["sampler_dist_l1"] = float((emp - want).abs().sum())
    return out


# ------------------------------------------------------------------------------------------ model level
def _model(n_layer=4, seed=0):
    import midi_model as mm
    torch.manual_seed(seed)
    cfg = mm.MIDIModelConfig.get_config("v2", True, n_layer=n_layer, n_head=16, n_embd=1024, n_inner=4096)
    return mm, mm.MIDIModel(cfg)


def _sd(model, dtype, device=DEV):
    return {k: v.detach().to(device=device, dtype=dtype) for k, v in model.state_dict().items()}


def check_model_forward():
    """forward + forward_token logits vs the oracle (fp32 and bf16 on the same device): noise-floor protocol
    of SURVEY.md section 8c tier 2."""
    from midi_b200.synth import synth_batch
    out = {}
    mm, model = _model(4)
    ocfg = O.cfg_from_hf(model.config)
    sd32 = _sd(model, torch.float32)
    model = model.to(DEV, dtype=BF).eval()
    sd16 = _sd(model, BF)
    inv_n = model.net.rotary_emb.inv_freq
    inv_t = model.net_token.rotary_emb.inv_freq
    out["inv_freq_is_bf16"] = float(inv_n.dtype == BF)
    batch = synth_batch(model.tokenizer, 2, 130, seed=1234).to(DEV)
    x, y = batch[:, :-1], batch[:, 1:]
    with torch.no_grad():
        h = model.forward(x)
        lg = model.forward_token(h.reshape(-1, 1024), y.reshape(-1, 8)[:, :-1])
        h32 = O.forward(sd32, ocfg, x)
        l32 = O.forward_token(sd32, ocfg, h32.reshape(-1, 1024), y.reshape(-1, 8)[:, :-1])
        h16 = O.forward(sd16, ocfg, x, inv_freq=inv_n)
        l16 = O.forward_token(sd16, ocfg, h16.reshape(-1, 1024), y.reshape(-1, 8)[:, :-1], inv_freq=inv_t)
    out["hidden_new_vs_fp32"] = rel(h.float(), h32)
    out["hidden_oracle16_vs_fp32"] = rel(h16.float(), h32)
    out["hidden_new_vs_oracle16"] = rel(h.float(), h16.float())
    out["logits_new_vs_fp32"] = rel(lg.float(), l32)
    out["logits_oracle16_vs_fp32"] = rel(l16.float(), l32)
    out["logits_new_vs_oracle16"] = rel(lg.float(), l16.float())
    out["argmax_agree_new_fp32"] = float((lg.float().argmax(-1) == l32.argmax(-1)).float().mean())
    out["argmax_agree_oracle16_fp32"] = float((l16.float().argmax(-1) == l32.argmax(-1)).float().mean())
    # teacher-forced greedy ids: wherever the fp32 oracle's top-1 margin exceeds the bf16 noise floor by a wide
    # factor, the argmax must agree exactly (SURVEY.md section 8c, greedy protocol (i))
    top2 = l32.topk(2, -1).values
    margin = top2[..., 0] - top2[..., 1]
    noise = float((l16.float() - l32).abs().max())
    sel = margin > 4 * noise
    out["margin_filtered_fraction"] = float(sel.float().mean())
    out["margin_filtered_argmax_mismatch"] = float((lg.float().argmax(-1)[sel] != l32.argmax(-1)[sel]).sum())
    # teacher-forced inner stack: feed the oracle's bf16 hidden
    with torch.no_grad():
        lg_tf = model.forward_token(h16.reshape(-1, 1024), y.reshape(-1, 8)[:, :-1])
    out["logits_teacher_forced_vs_oracle16"] = rel(lg_tf.float(), l16.float())
    return out


def check_model_layer_teacher_forced():
    """One decoder layer at a time, fed the oracle's own bf16 input (tier 1: <= 1e-3 on GEMM-dominated ops)."""
    from midi_b200.synth import synth_batch
    out = {}
    mm, model = _model(4)
    ocfg = O.cfg_from_hf(model.config)
    model = model.to(DEV, dtype=BF).eval()
    sd16 = _sd(model, BF)
    rt = model._rt()
    B, S = 2, 96
    x_in = randn(B * S, 1024, seed=3)
    # oracle: a 1-layer stack built from layer 0's weights
    one = O.StackCfg("net", 1, 16, 1024, 4096)
    inv = model.net.rotary_emb.inv_freq
    sd1 = {k: v for k, v in sd16.items() if k.startswith("net.layers.0.") or k == "net.norm.weight"}
    with torch.no_grad():
        ref = O.llama_stack(sd1, one, x_in.view(B, S, 1024), inv)
    eng = rt.outer
    keep = eng.layers
    eng.layers = keep[:1]
    y, _ = eng.forward(x_in, B, S, inv, save=False)
    eng.layers = keep
    out["outer_layer_tf"] = rel(y.float().view(B, S, 1024), ref.float())
    one_t = O.StackCfg("net_token", 1, 4, 1024, 1024)
    sd1 = {k: v for k, v in sd16.items() if k.startswith("net_token.layers.0.") or k == "net_token.norm.weight"}
    inv_t = model.net_token.rotary_emb.inv_freq
    x_in = randn(64 * 8, 1024, seed=4)
    with torch.no_grad():
        ref = O.llama_stack(sd1, one_t, x_in.view(64, 8, 1024), inv_t)
    eng = rt.inner
    keep = eng.layers
    eng.layers = keep[:1]
    y, _ = eng.forward(x_in, 64, 8, inv_t, save=False)
    eng.layers = keep
    out["inner_layer_tf"] = rel(y.float().view(64, 8, 1024), ref.float())
    return out


def check_model_train():
    """Fused loss + all gradients vs the oracle under torch autograd (fp32 weights = the bf16 weights upcast)."""
    from midi_b200.synth import synth_batch
    out = {}
    mm, model = _model(4)
    ocfg = O.cfg_from_hf(model.config)
    model = model.to(DEV, dtype=BF).train()
    batch = synth_batch(model.tokenizer, 2, 66, seed=77, pad_tail=3).to(DEV)
    sd = {k: v.detach().float().requires_grad_(True) for k, v in model.state_dict().items()}
    ref = O.train_loss(sd, ocfg, batch)
    ref.backward()
    loss = model.training_loss(batch)
    out["loss_abs"] = float((loss - ref.detach()).abs())
    out["loss_ref"] = float(ref.detach())
    worst, worst_name = 0.0, ""
    tot_n, tot_d = 0.0, 0.0
    for n, p in model.named_parameters():
        gref = sd[n].grad
        e = rel(p.grad.float(), gref)
        tot_n += float((p.grad.float() - gref).double().pow(2).sum())
        tot_d += float(gref.double().pow(2).sum())
        if e > worst:
            worst, worst_name = e, n
    out["grad_global_rel"] = math.sqrt(tot_n / tot_d)
    out["grad_worst_rel"] = worst
    print("worst grad tensor:", worst_name, worst)
    out["grad_pad_row_outer"] = float(model.net.embed_tokens.weight.grad[0].float().abs().max())
    out["grad_pad_row_inner"] = float(model.net_token.embed_tokens.weight.grad[0].float().abs().max())
    # autograd (drop-in) path == fused path
    fused = {n: p.grad.clone() for n, p in model.named_parameters()}
    for p in model.parameters():
        p.grad = None
    x, y = batch[:, :-1].contiguous(), batch[:, 1:].contiguous()
    hits0 = mm.LAZY_CE_HITS
    hidden = model.forward(x)
    hidden = hidden.reshape(-1, hidden.shape[-1])
    yy = y.reshape(-1, y.shape[-1])
    logits = model.forward_token(hidden, yy[:, :-1])
    l2 = F.cross_entropy(logits.view(-1, model.tokenizer.vocab_size), yy.view(-1), reduction="mean",
                         ignore_index=model.tokenizer.pad_id)
    l2.backward()
    out["lazy_ce_hits"] = float(mm.LAZY_CE_HITS - hits0)          # the reference's loss expression hit the fused CE (8 f2)
    out["autograd_loss_abs"] = float((l2.float() - ref.detach()).abs())
    tot_n = tot_d = 0.0
    for n, p in model.named_parameters():
        tot_n += float((p.grad.float() - sd[n].grad).double().pow(2).sum())
        tot_d += float(sd[n].grad.double().pow(2).sum())
    out["autograd_grad_global_rel"] = math.sqrt(tot_n / tot_d)
    # int16 host data path (midi_b200/data.py): device-side widening + x/y split, prefetcher, same loss bit for bit
    from midi_b200 import data as hostdata
    b16 = hostdata.collate(list(batch.cpu().numpy()), pad_id=model.tokenizer.pad_id)
    xs, ys = ops.batch_to_xy(b16.to(DEV))
    out["xy_split_mismatch"] = float((xs.view(2, -1, 8) != batch[:, :-1]).sum() + (ys.view(2, -1, 8) != batch[:, 1:]).sum())
    fed = list(hostdata.Prefetcher([b16, b16, b16], DEV))
    out["prefetch_mismatch"] = float(sum((f.to(torch.long) != batch).sum() for f in fed)) + abs(len(fed) - 3)
    for p in model.parameters():
        p.grad = None
    loss16 = model.training_loss(fed[0])
    out["int16_path_loss_mismatch"] = float((loss16 - loss).abs())
    # (gradients: the backward accumulates dQ / embedding rows with fp32 reductions whose order is not fixed -> rel. error)
    num = sum(float((p.grad.float() - fused[n].float()).double().pow(2).sum()) for n, p in model.named_parameters())
    den = sum(float(fused[n].float().double().pow(2).sum()) for n, p in model.named_parameters())
    out["int16_path_grad_rel"] = math.sqrt(num / den)
    tok = model.tokenizer
    # --sample-seq (train.py:172-175): forward_token on a random subset of event rows, gradients through the fancy index
    for p_ in model.parameters():
        p_.grad = None
    tb = synth_batch(tok, 2, 130, seed=5).to(DEV)
    xx, yy = tb[:, :-1].contiguous(), tb[:, 1:].contiguous()
    import random
    random.seed(0)
    rand_idx = [-1] + random.sample(list(range(yy.shape[1] - 2)), min(127, (yy.shape[1] - 2) // 2))
    hidden = model.forward(xx)[:, rand_idx]
    ys = yy[:, rand_idx].reshape(-1, 8)
    lg = model.forward_token(hidden.reshape(-1, 1024), ys[:, :-1])
    l_s = F.cross_entropy(lg.view(-1, tok.vocab_size), ys.reshape(-1), reduction="mean", ignore_index=tok.pad_id)
    l_s.backward()
    g_new = {n_: p_.grad.float().clone() for n_, p_ in model.named_parameters()}
    sdg = {k_: v_.detach().float().requires_grad_(True) for k_, v_ in model.state_dict().items()}
    h_o = O.forward(sdg, ocfg, xx, inv_freq=model.net.rotary_emb.inv_freq)[:, rand_idx]
    l_o = F.cross_entropy(O.forward_token(sdg, ocfg, h_o.reshape(-1, 1024), ys[:, :-1], inv_freq=model.net_token.rotary_emb.inv_freq).view(-1, tok.vocab_size), ys.reshape(-1),
                          reduction="mean", ignore_index=tok.pad_id)
    l_o.backward()
    out["sample_seq_loss_abs"] = float((l_s.float() - l_o.detach()).abs())
    num = sum(float((g_new[n_] - sdg[n_].grad).double().pow(2).sum()) for n_ in g_new)
    den = sum(float(sdg[n_].grad.double().pow(2).sum()) for n_ in g_new)
    out["sample_seq_grad_global_rel"] = math.sqrt(num / den)
    return out


def check_model_generate():
    """Greedy (top_k=1) generate and the KV-cached forward vs the oracle."""
    from midi_b200.synth import synth_batch
    out = {}
    mm, model = _model(4)
    ocfg = O.cfg_from_hf(model.config)
    model = model.to(DEV, dtype=BF).eval()
    sd16 = _sd(model, BF)
    tok = model.tokenizer
    batch = synth_batch(tok, 2, 40, seed=5).to(DEV)
    from transformers import DynamicCache
    with torch.no_grad():
        full = model.forward(batch)
        c = DynamicCache()
        parts = [model.forward(batch[:, :17], cache=c), model.forward(batch[:, 17:18], cache=c),
                 model.forward(batch[:, 18:23], cache=c)]
        for t in range(23, 40):
            parts.append(model.forward(batch[:, t:t + 1], cache=c))
    out["cached_vs_full_hidden"] = rel(torch.cat(parts, 1).float(), full.float())
    # fused single-token decode step (norm+QKV, RoPE+append+attention, ..., 5 launches/layer) == unfused kernels, bit for bit
    from midi_b200 import decode as dec
    outs = {}
    for fused in (True, False):
        dec.FUSED_DECODE = fused
        with torch.no_grad():
            c = DynamicCache()
            hs = [model.forward(batch[:, :17], cache=c)]
            for t in range(17, 30):
                hs.append(model.forward(batch[:, t:t + 1], cache=c))
        outs[fused] = torch.cat(hs, 1)
    dec.FUSED_DECODE = True
    out["fused_decode_mismatch"] = float((outs[True] != outs[False]).sum())
    # final norm fused into the lm_head GEMV == rmsnorm kernel + GEMV
    rt = model._rt()
    xpre = randn(4, 1024, seed=9)
    a = dec._gemv_fused(xpre, rt.lm_head, rt.V, norm_w=rt.inner.norm, eps=1e-6, ldy=rt.pitch)[:, :rt.V]
    bref = dec._lm_head(ops.rmsnorm(xpre, rt.inner.norm, 1e-6), rt.lm_head, rt.pitch)[:, :rt.V]
    out["fused_lm_head_mismatch"] = float((a != bref).sum())
    # inner cached path vs uncached logits
    with torch.no_grad():
        hid = full[:, -1]
        ids = batch[:, -1, :7]
        lg = model.forward_token(hid, ids)
        c2 = DynamicCache()
        steps = [model.forward_token(hid, None, cache=c2)]
        for i in range(7):
            steps.append(model.forward_token(None, ids[:, i:i + 1], cache=c2))
    out["inner_cached_vs_full_logits"] = rel(torch.cat(steps, 1).float(), lg.float())
    # greedy generate vs oracle generate (bf16 oracle on the same device), teacher-free
    prompt = batch[:, :6].cpu().numpy()
    ids_new = model.generate(prompt=prompt, batch_size=2, max_len=14, top_k=1, generator=torch.Generator(DEV).manual_seed(0))
    ids_ref = O.generate(sd16, ocfg, tok, prompt, batch_size=2, max_len=14, top_k=1,
                         inv_freq_net=model.net.rotary_emb.inv_freq, inv_freq_tok=model.net_token.rotary_emb.inv_freq)
    n = min(ids_new.shape[1], ids_ref.shape[1])
    out["greedy_len_new"], out["greedy_len_ref"] = float(ids_new.shape[1]), float(ids_ref.shape[1])
    out["greedy_token_agree"] = float((ids_new[:, :n] == ids_ref[:, :n]).mean())
    # the CUDA-graph loop and the host-driven loop run the same kernels: identical greedy ids
    os.environ["B200_GENERATE"] = "eager"
    ids_eager = model.generate(prompt=prompt, batch_size=2, max_len=14, top_k=1, generator=torch.Generator(DEV).manual_seed(0))
    os.environ["B200_GENERATE"] = "nograph"
    ids_ng = model.generate(prompt=prompt, batch_size=2, max_len=14, top_k=1, generator=torch.Generator(DEV).manual_seed(0))
    os.environ["B200_GENERATE"] = "graph"
    ids_graph = model.generate(prompt=prompt, batch_size=2, max_len=14, top_k=1, generator=torch.Generator(DEV).manual_seed(0))
    os.environ.pop("B200_GENERATE")               # default again: the persistent kernel (what ids_new was generated with)
    out["greedy_graph_vs_nograph_mismatch"] = float((ids_graph != ids_ng).sum()) if ids_graph.shape == ids_ng.shape else 1e9
    # persistent kernel vs launch-per-phase loop on flat random-init logits: same arithmetic except the attention's
    # summation order, so near-ties may flip -> agreement fraction here, bit-equality on the peaked checkpoints
    out["greedy_persist_vs_graph_agree"] = float((ids_new == ids_graph).mean()) if ids_new.shape == ids_graph.shape else 0.0
    # (graph replay == the same launches issued from the host; the host-driven loop prefills the last prompt event
    #  with the flash kernel instead of the decode kernel, so on these flat random-init logits it may pick other
    #  near-ties -- it is held to bit-equality on the peaked checkpoint instead, see check_model_peaked_greedy)
    out["greedy_eager_vs_graph_agree"] = float((ids_new == ids_eager).mean()) if ids_new.shape == ids_eager.shape else 0.0
    # grammar validity of sampled generation
    ids_s = model.generate(prompt=None, batch_size=4, max_len=24, generator=torch.Generator(DEV).manual_seed(1))
    bad = 0
    for row in ids_s[:, 1:].reshape(-1, 8):          # skip the BOS event of every row
        if row[0] == tok.eos_id or row[0] == tok.pad_id:
            continue
        if tok.tokens2event(row.tolist()) == []:
            bad += 1
    out["sampled_invalid_events"] = float(bad)
    return out


def _song_batch(tok, B, n_events, seed, fixed_step=3):
    """Deterministic grammar-valid 'songs' (SURVEY.md 8c peaked-checkpoint recipe): bos, one patch_change, then
    notes walking up a scale.  Learnable in a few hundred steps => large top-1 margins, no EOS."""
    rng = np.random.default_rng(seed)
    out = np.zeros((B, n_events, 8), dtype=np.int64)
    for b in range(B):
        ch, step, pitch = int(rng.integers(0, 4)), int(rng.integers(1, 6)), int(rng.integers(40, 80))
        if fixed_step:
            step = fixed_step      # continuation is then a deterministic function of the previous event
        rows = [[tok.bos_id] + [0] * 7, tok.event2tokens(["patch_change", 0, 0, 1, ch, int(rng.integers(0, 128))])]
        k = 0
        while len(rows) < n_events:
            rows.append(tok.event2tokens(["note", 1 if k % 4 == 0 else 0, (4 * k) % 16, 1, ch, pitch, 80, 4]))
            pitch = 40 + ((pitch - 40 + step) % 40)
            k += 1
        out[b] = np.asarray(rows)
    return torch.from_numpy(out)


def check_model_peaked_greedy():
    """Train a 4-layer full-width model with the FUSED sm_100a trainer until it has learnt the token grammar,
    then free-running greedy generate must be bit-identical to the oracle's (bf16, same weights), and the loss
    curve must fall (exercises fwd+bwd+clip+AdamW end to end)."""
    out = {}
    mm, model = _model(4, seed=0)
    ocfg = O.cfg_from_hf(model.config)
    model = model.to(DEV, dtype=BF).train()
    tok = model.tokenizer
    losses = []
    for step in range(1, 241):
        batch = _song_batch(tok, 16, 66, seed=step).to(DEV)
        loss = model.training_loss(batch)
        model.fused_optimizer_step(lr=3e-4 * min(1.0, step / 20), step=step, weight_decay=0.01)
        if step % 20 == 0 or step == 1:
            losses.append(float(loss))
    print("peaked training losses:", [round(x, 3) for x in losses])
    out["peaked_loss_first"], out["peaked_loss_last"] = losses[0], losses[-1]
    model.eval()
    sd16 = _sd(model, BF)
    prompt = _song_batch(tok, 4, 9, seed=999).numpy()
    ids_new = model.generate(prompt=prompt, batch_size=4, max_len=40, top_k=1)          # default: persistent kernel
    os.environ["B200_GENERATE"] = "eager"
    ids_eager = model.generate(prompt=prompt, batch_size=4, max_len=40, top_k=1)        # host-driven loop
    os.environ["B200_GENERATE"] = "graph"
    ids_graph = model.generate(prompt=prompt, batch_size=4, max_len=40, top_k=1)        # CUDA-graph loop
    os.environ.pop("B200_GENERATE")
    out["peaked_eager_vs_graph_mismatch"] = float((ids_eager != ids_graph).sum()) if ids_eager.shape == ids_graph.shape else 1e9
    out["peaked_persist_vs_graph_mismatch"] = float((ids_new != ids_graph).sum()) if ids_new.shape == ids_graph.shape else 1e9
    ids_ref = O.generate(sd16, ocfg, tok, prompt, batch_size=4, max_len=40, top_k=1,
                         inv_freq_net=model.net.rotary_emb.inv_freq, inv_freq_tok=model.net_token.rotary_emb.inv_freq)
    out["peaked_len_new"], out["peaked_len_ref"] = float(ids_new.shape[1]), float(ids_ref.shape[1])
    n = min(ids_new.shape[1], ids_ref.shape[1])
    neq = ids_new[:, :n] != ids_ref[:, :n]
    out["peaked_greedy_mismatch"] = float(neq.sum()) + abs(ids_new.shape[1] - ids_ref.shape[1])
    # tie / margin audit (SURVEY.md 8c (iii)): if the runs diverge, the first differing token must be one where
    # the fp32 oracle's margin between the two candidates is within the bf16 noise
    sd32a = {k: v.float() for k, v in sd16.items()}
    ref_t = torch.from_numpy(ids_ref).to(DEV)
    with torch.no_grad():
        h32a = O.forward(sd32a, ocfg, ref_t[:, :-1])
        l32a = O.forward_token(sd32a, ocfg, h32a.reshape(-1, 1024), ref_t[:, 1:].reshape(-1, 8)[:, :-1]).view(4, n - 1, 8, -1)
    if neq.any():
        first_e = int(np.argwhere(neq.any(-1).any(0))[0][0])
        bs, ts = np.nonzero(neq[:, first_e])
        b0, t0 = int(bs[0]), int(ts[0])
        row = l32a[b0, first_e - 1, t0]
        out["peaked_first_divergence_event"] = float(first_e)
        out["peaked_first_divergence_margin"] = float((row[ids_ref[b0, first_e, t0]] - row[ids_new[b0, first_e, t0]]).abs())
        print("first divergence at event", first_e, "row", b0, "token", t0, "ref", ids_ref[b0, first_e], "new", ids_new[b0, first_e])
    top2 = l32a[:, 8:].topk(2, -1).values
    out["peaked_min_top1_margin_fp32"] = float((top2[..., 0] - top2[..., 1])[ref_t[:, 9:] != 0].min())
    # app.py's streaming loop (SURVEY.md 8 f4): same events as generate() when no option is set, and with the
    # disable_* options the oracle's restatement of app.py:27-120 event for event (greedy), no denied id emitted
    P0 = prompt.shape[1]
    evs = list(model.generate_stream(prompt=prompt, batch_size=4, max_len=40, top_k=1))
    ids_stream = np.stack(evs, axis=1)
    out["stream_vs_generate_mismatch"] = (float((ids_stream != ids_new[:, P0:]).sum())
                                          if ids_stream.shape == ids_new[:, P0:].shape else 1e9)
    chans = [int(c) for c in np.unique([tok.tokens2event(r.tolist())[1 + tok.events["note"].index("channel")]
                                        for r in ids_new[:, P0:].reshape(-1, 8) if r[0] == tok.event_ids["note"]])][:2]
    deny = O.deny_ids(tok, True, True, chans)
    evs = list(model.generate_stream(prompt=prompt, batch_size=4, max_len=40, top_k=1, disable_patch_change=True,
                                     disable_control_change=True, disable_channels=chans))
    ids_masked = np.stack(evs, axis=1)
    ref_masked = O.generate(sd16, ocfg, tok, prompt, batch_size=4, max_len=40, top_k=1, deny=deny, max_context=4096,
                            inv_freq_net=model.net.rotary_emb.inv_freq, inv_freq_tok=model.net_token.rotary_emb.inv_freq)[:, P0:]
    out["stream_masked_mismatch"] = (float((ids_masked != ref_masked).sum()) if ids_masked.shape == ref_masked.shape
                                     else 1e9)
    out["stream_denied_ids_emitted"] = float(np.isin(ids_masked, sorted(deny)).sum())
    out["stream_masked_differs_from_plain"] = float((ids_masked[:, :min(ids_masked.shape[1], ids_stream.shape[1])]
                                                     != ids_stream[:, :min(ids_masked.shape[1], ids_stream.shape[1])]).sum())
    print("stream: disabled channels", chans, "masked events", ids_masked.shape[1], "plain events", ids_stream.shape[1])
    # two generations streaming concurrently from two threads on ONE model (gradio serves app.generate from worker threads,
    # app.py:496): each owns its loop state, so both must reproduce their sequential results; a generator resumed from
    # another thread than the one that created it must work too
    import threading
    prompt_b = _song_batch(tok, 4, 9, seed=321).numpy()
    seq_a = np.stack(list(model.generate_stream(prompt=prompt, batch_size=4, max_len=30, top_k=1)), axis=1)
    seq_b = np.stack(list(model.generate_stream(prompt=prompt_b, batch_size=4, max_len=30, top_k=1)), axis=1)
    got, errs = {}, []

    def drive(name, pr):
        try:
            got[name] = np.stack(list(model.generate_stream(prompt=pr, batch_size=4, max_len=30, top_k=1)), axis=1)
        except Exception as e:     # noqa: BLE001
            errs.append(repr(e))
    th = [threading.Thread(target=drive, args=("a", prompt)), threading.Thread(target=drive, args=("b", prompt_b))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    out["stream_concurrent_errors"] = float(len(errs))
    out["stream_concurrent_mismatch"] = (float((got["a"] != seq_a).sum() + (got["b"] != seq_b).sum())
                                         if not errs and got["a"].shape == seq_a.shape and got["b"].shape == seq_b.shape else 1e9)
    gen = model.generate_stream(prompt=prompt, batch_size=4, max_len=30, top_k=1)
    first = next(gen)
    rest = []
    t2 = threading.Thread(target=lambda: rest.extend(list(gen)))
    t2.start()
    t2.join()
    moved = np.stack([first] + rest, axis=1)
    out["stream_resumed_on_other_thread_mismatch"] = float((moved != seq_a).sum()) if moved.shape == seq_a.shape else 1e9
    if errs:
        print("concurrent stream errors:", errs)
    ids_after = model.generate(prompt=prompt, batch_size=4, max_len=40, top_k=1)      # the mask must not leak into generate()
    out["stream_mask_leak_mismatch"] = float((ids_after != ids_new).sum()) if ids_after.shape == ids_new.shape else 1e9
    # the generated continuation is itself grammar-valid
    bad = sum(1 for row in ids_new[:, 1:].reshape(-1, 8) if row[0] not in (tok.eos_id, tok.pad_id) and tok.tokens2event(row.tolist()) == [])
    out["peaked_invalid_events"] = float(bad)
    # teacher-forced logits on a fresh song vs the oracle bf16 / fp32
    batch = _song_batch(tok, 2, 50, seed=5).to(DEV)
    sd32 = {k: v.float() for k, v in sd16.items()}
    with torch.no_grad():
        h = model.forward(batch[:, :-1])
        lg = model.forward_token(h.reshape(-1, 1024), batch[:, 1:].reshape(-1, 8)[:, :-1])
        h32 = O.forward(sd32, ocfg, batch[:, :-1])
        l32 = O.forward_token(sd32, ocfg, h32.reshape(-1, 1024), batch[:, 1:].reshape(-1, 8)[:, :-1])
    tg = batch[:, 1:].reshape(-1, 8)
    live = tg != 0
    out["peaked_argmax_mismatch_vs_fp32"] = float((lg.float().argmax(-1)[live] != l32.argmax(-1)[live]).sum())
    out["peaked_logits_vs_fp32"] = rel(lg.float(), l32)
    return out


def check_model_large():
    """tv2o-large (24 event-level / 6 token-level layers, BASELINE config 5): fused loss + gradients vs the oracle at a
    small shape, and a short KV-cached generate at the maximum context bookkeeping (max_len 4096 pools)."""
    from midi_b200.synth import synth_batch
    import midi_model as mm
    out = {}
    torch.manual_seed(0)
    model = mm.MIDIModel(mm.MIDIModelConfig.from_name("tv2o-large"))
    out["large_params"] = float(sum(p.numel() for p in model.parameters()))
    ocfg = O.cfg_from_hf(model.config)
    model = model.to(DEV, dtype=BF).train()
    batch = synth_batch(model.tokenizer, 1, 130, seed=3).to(DEV)
    sd = {k: v.detach().float().requires_grad_(True) for k, v in model.state_dict().items()}
    ref = O.train_loss(sd, ocfg, batch)
    ref.backward()
    loss = model.training_loss(batch)
    out["large_loss_abs"] = float((loss - ref.detach()).abs())
    tot_n = tot_d = 0.0
    for n, p in model.named_parameters():
        tot_n += float((p.grad.float() - sd[n].grad).double().pow(2).sum())
        tot_d += float(sd[n].grad.double().pow(2).sum())
    out["large_grad_global_rel"] = math.sqrt(tot_n / tot_d)
    del sd
    model.eval()
    ids = model.generate(batch_size=2, max_len=4096 if False else 40, generator=torch.Generator(DEV).manual_seed(0))
    out["large_generate_events"] = float(ids.shape[1])
    return out



# ------------------------------------------------------------------------------------------ round-2 additions
def _ordered_bf16(t):
    """bf16 bit patterns mapped to integers that are monotonic in the value (for ulp distances)."""
    i = t.contiguous().view(torch.int16).int()
    return torch.where(i >= 0, i, -(i & 0x7FFF))


def _exact_metrics(y, ref64, name, out):
    """y (bf16) vs an fp64 reference: fraction of elements that are not the correctly-rounded bf16 value, the largest
    distance in bf16 ulps among elements that are not tiny, and the worst |err| / (1 ulp + 1e-3 rms) -- a dropped k-block
    or a wrong split-K slice moves whole tiles by many ulps; fp32 summation order moves isolated elements by one."""
    want = ref64.to(torch.float32).to(BF)
    neq = (y != want)
    out[f"exact_frac_{name}"] = float(neq.float().mean())
    rms = float(ref64.pow(2).mean().sqrt())
    big = ref64.abs() > 0.05 * rms
    ulp = (_ordered_bf16(y) - _ordered_bf16(want)).abs()
    out[f"exact_maxulp_{name}"] = float(ulp[big].max()) if bool(big.any()) else 0.0
    tol = ref64.abs() * 2.0 ** -7 + 1e-3 * rms
    out[f"exact_err_over_tol_{name}"] = float(((y.double() - ref64).abs() / tol).max())


def check_gemm_exact():
    """Tensor-core GEMM at the benchmark's own shapes (M = 131 072 rows, K = 131 072 split-K, the tail-split path)
    against an fp64 reference of the same bf16 operands, as mismatch fraction / ulp distance instead of a norm."""
    out = {}
    # forward (K-major x K-major): token-level projections and the event-level MLP shape of the bench step
    for (M, N, K) in ((131072, 1024, 1024), (16384, 8192, 1024), (4096, 3406, 1024)):
        a, w = randn(M, K, seed=M % 97), randn(N, K, scale=0.05, seed=N % 89)
        pitch = (N + 7) // 8 * 8
        y = ops.linear(a, w, pitch=pitch if pitch != N else None)
        ref = a.double() @ w.double().T
        _exact_metrics(y[:, :N], ref, f"fwd_{M}x{N}x{K}", out)
        del a, w, y, ref
    # dgrad (B operand MN-major); [16384, 8192] @ [8192, 1024] takes the K-split of the last partial wave (tail split)
    for (M, N, K) in ((16384, 8192, 1024), (131072, 3072, 1024)):
        dy, w = randn(M, N, seed=5), randn(N, K, scale=0.05, seed=6)
        dx = ops.linear_dgrad(dy, w)
        ref = dy.double() @ w.double()
        _exact_metrics(dx, ref, f"dgrad_{M}x{N}x{K}", out)
        del dy, w, dx, ref
    # wgrad (both operands MN-major): K = 131 072 rows with split-K 9 / 3, and the 16 384-row event-level shapes
    for (M, N, K) in ((131072, 1024, 1024), (131072, 3072, 1024), (16384, 1024, 4096), (16384, 3072, 1024)):
        dy, x = randn(M, N, seed=7), randn(M, K, seed=8)
        dw = torch.empty(N, K, device=DEV, dtype=BF)
        ops.linear_wgrad(dy, x, dw, accumulate=False)
        bn, sp = ops._plan(N, K, M, True)
        out[f"wgrad_splits_{M}x{N}x{K}"] = float(sp)
        ref = dy.double().T @ x.double()
        _exact_metrics(dw, ref, f"wgrad_{M}x{N}x{K}", out)
        del dy, x, dw, ref
    return out


def check_decode_paged():
    """b200_attn_decode_fused (RoPE + KV append + single-query attention, the kernel inside the CUDA-graph generate loop)
    against dense fp32 SDPA with the context crossing 64-position page boundaries, a permuted block table, n_split in
    {1, 2, 16} and the position read from the device (graph mode) or passed by value."""
    out = {}
    from midi_b200 import decode as dec
    from midi_b200.engine import StackCfg
    nh, D, page, Bn, cap = 16, 64, 64, 3, 4096
    H = nh * D
    inv = O.default_inv_freq(D).to(BF).to(DEV)
    cos, sin = ops.rope_table(inv, cap)
    cfg = StackCfg("net", 1, nh, H, 4 * H, 1e-6)
    g = torch.Generator(device=DEV).manual_seed(11)
    scale = 1.0 / math.sqrt(D)
    for T in (1, 63, 64, 65, 257, 1500, 4095):
        pos = T - 1
        for n_split in (1, 2, 16):
            if (T + n_split - 1) // n_split > 1024:
                continue
            kv = dec.PagedKV(cfg, Bn, cap, page, DEV)
            kv.block_table.copy_(torch.randperm(Bn * kv.max_pages, generator=g, device=DEV).int().view(Bn, kv.max_pages))
            hist = randn(Bn * pos, 3 * H, seed=T) if pos > 0 else None
            if pos > 0:
                lib.call("b200_kv_append", hist.data_ptr(), kv.k[0].data_ptr(), kv.v[0].data_ptr(), kv.block_table.data_ptr(),
                         kv.max_pages, kv.page, nh, D, Bn, pos, 0, None, 3 * H, lib.stream())
            new = randn(Bn, 3 * H, seed=T + 1)
            o = torch.empty(Bn, H, device=DEV, dtype=BF)
            ws = torch.empty(lib.query("b200_attn_decode_workspace_bytes", Bn, nh, D, n_split), dtype=torch.uint8, device=DEV)
            # n_split 16 = what the loop with 4096-event pools runs (position from the device counter, max_T = pool size);
            # n_split 1 / 2 = the host-driven path (position by value, max_T = T)
            graph_mode = n_split == 16
            pos_dev = torch.tensor([pos], dtype=torch.int32, device=DEV) if graph_mode else None
            lib.call("b200_attn_decode_fused", new.data_ptr(), kv.k[0].data_ptr(), kv.v[0].data_ptr(), kv.block_table.data_ptr(),
                     kv.max_pages, kv.page, cos.data_ptr(), sin.data_ptr(), o.data_ptr(), Bn, nh, D, 0 if graph_mode else pos,
                     lib.ptr(pos_dev), cap if graph_mode else T, 3 * H, H, scale, n_split, ws.data_ptr(), ws.numel(), lib.stream())
            rc, rs = O.rope_cos_sin(inv, torch.tensor([pos], device=DEV), BF)
            q = O.apply_rope(new[:, :H].view(Bn, 1, nh, D).transpose(1, 2), rc, rs)             # (Bn, nh, 1, D) bf16
            k_new = O.apply_rope(new[:, H:2 * H].view(Bn, 1, nh, D).transpose(1, 2), rc, rs)
            v_new = new[:, 2 * H:].view(Bn, 1, nh, D).transpose(1, 2)
            if pos > 0:
                hk = hist.view(Bn, pos, 3, nh, D)[:, :, 1].transpose(1, 2)
                hv = hist.view(Bn, pos, 3, nh, D)[:, :, 2].transpose(1, 2)
                k_all, v_all = torch.cat([hk, k_new], 2), torch.cat([hv, v_new], 2)
            else:
                k_all, v_all = k_new, v_new
            ref = _sdpa_ref(q.float(), k_all.float(), v_all.float(), pos)
            out[f"decode_fused_T{T}_s{n_split}"] = rel(o.float().view(Bn, 1, nh, D).transpose(1, 2), ref)
            # the new key / value landed in the right page slot (bit-exact RoPE'd key)
            bad = 0
            for b in range(Bn):
                pg = int(kv.block_table[b, pos // page])
                bad += int((kv.k[0][pg, :, pos % page] != k_new[b, :, 0]).sum()) + int((kv.v[0][pg, :, pos % page] != v_new[b, :, 0]).sum())
            out[f"decode_fused_append_mismatch_T{T}_s{n_split}"] = float(bad)
    return out


# The reference's own GPU path: the HF LlamaModels inside MIDIModel (they are the parameter containers, so they read the
# same weights) run exactly as /root/reference/midi_model.py:116-150 runs them -- eager bf16, torch SDPA.
def _hf_forward(model, x, cache=None):
    e = model.net.embed_tokens(x).sum(dim=-2)
    return model.net(inputs_embeds=e, past_key_values=cache, use_cache=cache is not None).last_hidden_state


def _hf_forward_token(model, hidden_state=None, x=None, cache=None):
    if hidden_state is not None:
        hidden_state = hidden_state.unsqueeze(1)
    if x is not None:
        x = model.net_token.embed_tokens(x)
        if hidden_state is not None:
            x = torch.cat([hidden_state, x], dim=1)
        hidden_state = x
    h = model.net_token(inputs_embeds=hidden_state, past_key_values=cache, use_cache=cache is not None).last_hidden_state
    return model.lm_head(h)


def check_model_vs_hf():
    """This implementation vs the reference's eager-bf16 GPU path (HF LlamaModel + torch SDPA on the same device, same
    weights), and the oracle vs that same path: where the oracle's attention rounds differently from the GPU SDPA
    backend, `*_oracle16_vs_hf` shows the distance the teacher-forced tolerance has to absorb."""
    from midi_b200.synth import synth_batch
    out = {}
    mm, model = _model(4)
    ocfg = O.cfg_from_hf(model.config)
    model = model.to(DEV, dtype=BF).eval()
    sd16 = _sd(model, BF)
    rt = model._rt()
    batch = synth_batch(model.tokenizer, 2, 130, seed=1234).to(DEV)
    x, y = batch[:, :-1], batch[:, 1:]
    ids = y.reshape(-1, 8)[:, :-1]
    with torch.no_grad():
        h = model.forward(x)
        lg = model.forward_token(h.reshape(-1, 1024), ids)
        h_hf = _hf_forward(model, x)
        lg_hf = _hf_forward_token(model, h_hf.reshape(-1, 1024), ids)
        h16 = O.forward(sd16, ocfg, x, inv_freq=model.net.rotary_emb.inv_freq)
        l16 = O.forward_token(sd16, ocfg, h16.reshape(-1, 1024), ids, inv_freq=model.net_token.rotary_emb.inv_freq)
        lg_tf = model.forward_token(h_hf.reshape(-1, 1024), ids)                 # token-level stack fed HF's hidden
        lg_hf_tf = lg_hf
    out["hidden_new_vs_hf"] = rel(h.float(), h_hf.float())
    out["hidden_oracle16_vs_hf"] = rel(h16.float(), h_hf.float())
    out["logits_new_vs_hf"] = rel(lg.float(), lg_hf.float())
    out["logits_oracle16_vs_hf"] = rel(l16.float(), lg_hf.float())
    out["logits_tf_new_vs_hf"] = rel(lg_tf.float(), lg_hf_tf.float())
    out["argmax_agree_new_hf"] = float((lg.float().argmax(-1) == lg_hf.float().argmax(-1)).float().mean())
    # one decoder layer, teacher-forced with the same bf16 input (SURVEY.md 8c tier 1), event level and token level
    import torch.nn as nn
    for which, eng, hf, inv, (nseq, S) in (("outer", rt.outer, model.net, model.net.rotary_emb.inv_freq, (2, 96)),
                                           ("inner", rt.inner, model.net_token, model.net_token.rotary_emb.inv_freq, (64, 8))):
        x_in = randn(nseq * S, 1024, seed=3 if which == "outer" else 4)
        keep_hf, keep = hf.layers, eng.layers
        hf.layers = nn.ModuleList(list(keep_hf)[:1])
        eng.layers = keep[:1]
        try:
            with torch.no_grad():
                ref = hf(inputs_embeds=x_in.view(nseq, S, 1024), use_cache=False).last_hidden_state
                ours, _ = eng.forward(x_in, nseq, S, inv, save=False)
                one = O.StackCfg(eng.cfg.prefix, 1, eng.cfg.n_head, 1024, eng.cfg.inner)
                sd1 = {k: v for k, v in sd16.items() if k.startswith(f"{eng.cfg.prefix}.layers.0.") or k == f"{eng.cfg.prefix}.norm.weight"}
                orc = O.llama_stack(sd1, one, x_in.view(nseq, S, 1024), inv)
        finally:
            hf.layers, eng.layers = keep_hf, keep
        out[f"{which}_layer_tf_new_vs_hf"] = rel(ours.float().view(nseq, S, 1024), ref.float())
        out[f"{which}_layer_tf_oracle16_vs_hf"] = rel(orc.float(), ref.float())
    # attention alone: torch SDPA bf16 (the reference's backend) vs this kernel vs the oracle's formulation
    B, S, nh, D = 2, 512, 16, 64
    qkv = randn(B * S, 3 * nh * D, seed=21)
    q, k, v = (qkv.view(B, S, 3, nh, D)[:, :, i].transpose(1, 2) for i in range(3))
    o_new, _ = ops.attn_causal_fwd(qkv, B, S, nh, D, want_lse=False)
    o_new = o_new.view(B, S, nh, D).transpose(1, 2)
    o_sdpa = F.scaled_dot_product_attention(q, k, v, is_causal=True)
    o_orc = O.attention(q, k, v, 0)
    o_32 = _sdpa_ref(q.float(), k.float(), v.float(), 0)
    out["attn_new_vs_sdpa16"] = rel(o_new.float(), o_sdpa.float())
    out["attn_oracle16_vs_sdpa16"] = rel(o_orc.float(), o_sdpa.float())
    out["attn_new_vs_fp32"] = rel(o_new.float(), o_32)
    out["attn_sdpa16_vs_fp32"] = rel(o_sdpa.float(), o_32)
    out["attn_oracle16_vs_fp32"] = rel(o_orc.float(), o_32)
    # which SDPA backend does torch pick for the token-level shape, and how far is each from fp32 / from this kernel
    from torch.nn.attention import SDPBackend, sdpa_kernel
    Nn, L, nh2, D2 = 64, 8, 4, 256
    qkv2 = randn(Nn * L, 3 * nh2 * D2, seed=22)
    q2, k2, v2 = (qkv2.view(Nn, L, 3, nh2, D2)[:, :, i].transpose(1, 2) for i in range(3))
    o32 = _sdpa_ref(q2.float(), k2.float(), v2.float(), 0)
    o_tiny = ops.attn_tiny_fwd(qkv2, Nn, L, nh2, D2).view(Nn, L, nh2, D2).transpose(1, 2)
    o_def = F.scaled_dot_product_attention(q2, k2, v2, is_causal=True)
    out["inner_attn_new_vs_fp32"] = rel(o_tiny.float(), o32)
    out["inner_attn_sdpa_default_vs_fp32"] = rel(o_def.float(), o32)
    out["inner_attn_new_vs_sdpa_default"] = rel(o_tiny.float(), o_def.float())
    for name, be in (("flash", SDPBackend.FLASH_ATTENTION), ("efficient", SDPBackend.EFFICIENT_ATTENTION),
                     ("math", SDPBackend.MATH), ("cudnn", SDPBackend.CUDNN_ATTENTION)):
        try:
            with sdpa_kernel(be):
                ob = F.scaled_dot_product_attention(q2, k2, v2, is_causal=True)
            out[f"inner_sdpa_backend_{name}_vs_fp32"] = rel(ob.float(), o32)
            out[f"inner_sdpa_backend_{name}_equals_default"] = float(torch.equal(ob, o_def))
        except Exception:
            out[f"inner_sdpa_backend_{name}_vs_fp32"] = -1.0          # backend not available for this shape
    # train step: loss and gradients vs HF autograd in bf16 (the reference's training arithmetic, train.py:168-185)
    model.train()
    tb = synth_batch(model.tokenizer, 2, 66, seed=77, pad_tail=3).to(DEV)
    loss = model.training_loss(tb)
    mine = {n: p.grad.clone() for n, p in model.named_parameters()}
    for p in model.parameters():
        p.grad = None
    hx = _hf_forward(model, tb[:, :-1].contiguous())
    yy = tb[:, 1:].reshape(-1, 8)
    lgt = _hf_forward_token(model, hx.reshape(-1, 1024), yy[:, :-1])
    l_hf = F.cross_entropy(lgt.view(-1, model.tokenizer.vocab_size), yy.reshape(-1), reduction="mean", ignore_index=model.tokenizer.pad_id)
    l_hf.backward()
    out["hf_loss_abs"] = float((loss.float() - l_hf.float()).abs())
    num = sum(float((mine[n].float() - p.grad.float()).double().pow(2).sum()) for n, p in model.named_parameters())
    den = sum(float(p.grad.float().double().pow(2).sum()) for n, p in model.named_parameters())
    out["hf_grad_global_rel"] = math.sqrt(num / den)
    return out


def _song_batch_long(tok, B, n_events, seed):
    return _song_batch(tok, B, n_events, seed, fixed_step=3)


def check_model_medium_long():
    """BASELINE config 3 on the real tv2o-medium architecture (12 event-level / 3 token-level layers): train it peaked
    with the fused trainer on long songs, then (a) the CUDA-graph generate loop with 4096-event pools (n_split 16) runs
    >= 600 events past >= 8 KV page boundaries and must emit the oracle's greedy ids bit for bit, (b) the KV-cached
    forward equals the full forward at S = 4096, (c) contexts beyond max_position_embeddings work (app.py: prompt + 4096),
    (d) the loss at the benchmark shape (8 x 2048 events) equals the oracle's on the same weights and batch."""
    import midi_model as mm
    from midi_b200 import decode as dec
    from midi_b200.synth import synth_batch
    from transformers import DynamicCache
    out = {}
    torch.manual_seed(0)
    model = mm.MIDIModel(mm.MIDIModelConfig.from_name("tv2o-medium"))
    ocfg = O.cfg_from_hf(model.config)
    model = model.to(DEV, dtype=BF).train()
    tok = model.tokenizer
    losses = []
    n_steps = 0
    # curriculum: short songs first (many distinct songs per step: the pitch / time rule is learnt after a plateau near 0.47,
    # as in the 4-layer check), then long songs so that positions up to 768 have been trained
    for step in range(1, 1501):
        batch = _song_batch_long(tok, 16, 66, seed=step).to(DEV)
        loss = model.training_loss(batch)
        model.fused_optimizer_step(lr=3e-4 * min(1.0, step / 20), step=step, weight_decay=0.01)
        n_steps = step
        if step % 20 == 0 or step == 1:
            losses.append(float(loss))
            if step >= 100 and max(losses[-2:]) < 0.04:
                break
    short_steps = n_steps
    for step in range(n_steps + 1, n_steps + 401):
        batch = _song_batch_long(tok, 4, 769, seed=step).to(DEV)
        loss = model.training_loss(batch)
        model.fused_optimizer_step(lr=1e-4, step=step, weight_decay=0.01)
        n_steps = step
        if step % 20 == 0:
            losses.append(float(loss))
            if step - short_steps >= 100 and max(losses[-2:]) < 0.02:
                break
    print("medium peaked training losses:", [round(v, 3) for v in losses], "steps", short_steps, n_steps)
    out["medium_peaked_loss_last"] = losses[-1]
    out["medium_peaked_steps"] = float(n_steps)
    # optimizer state round trip (checkpoint / resume of the fused AdamW)
    osd = model.optimizer_state_dict()
    st = model.__dict__["_b200_opt"]
    m0 = st["m"].clone()
    st["m"].zero_()
    resumed = model.load_optimizer_state_dict(osd)
    out["opt_state_roundtrip_mismatch"] = float((st["m"] != m0).sum()) + abs(resumed - n_steps)
    model.eval()
    sd16 = _sd(model, BF)
    inv_n, inv_t = model.net.rotary_emb.inv_freq, model.net_token.rotary_emb.inv_freq
    # ---- (a) long greedy generation, graph loop with 4096-event pools vs the oracle
    P, n_new, Bg = 100, 640, 4
    prompt = _song_batch_long(tok, Bg, P, seed=999).numpy()
    key, gg = model._checkout_generator(Bg, 4096, 1.0, 0.98, 1, None)
    out["long_n_split"] = float(max(1, min(32, (4096 + 255) // 256)))
    try:
        ids_pool = gg.run(torch.from_numpy(prompt).to(DEV), use_graph="persist", max_new=n_new).cpu().numpy()
        ids_pool_graph = gg.run(torch.from_numpy(prompt).to(DEV), use_graph=True, max_new=n_new).cpu().numpy()
    finally:
        model._return_generator(key, gg)
    out["long_persist_vs_graph_mismatch"] = float((ids_pool != ids_pool_graph).sum()) if ids_pool.shape == ids_pool_graph.shape else 1e9
    ids_pub = model.generate(prompt=prompt, batch_size=Bg, max_len=P + n_new, top_k=1)          # public API, exact-size pools
    ids_ref = O.generate(sd16, ocfg, tok, prompt, batch_size=Bg, max_len=P + n_new, top_k=1, inv_freq_net=inv_n, inv_freq_tok=inv_t)
    out["long_len_new"], out["long_len_ref"] = float(ids_pool.shape[1]), float(ids_ref.shape[1])
    n = min(ids_pool.shape[1], ids_ref.shape[1])
    neq = ids_pool[:, :n] != ids_ref[:, :n]
    out["long_greedy_mismatch"] = float(neq.sum()) + abs(ids_pool.shape[1] - ids_ref.shape[1])
    out["long_pool_vs_public_mismatch"] = float((ids_pool != ids_pub).sum()) if ids_pool.shape == ids_pub.shape else 1e9
    out["long_page_boundaries_crossed"] = float((P + n_new - 1) // 64 - (P - 1) // 64)
    bad = sum(1 for row in ids_pool[:, 1:].reshape(-1, 8) if row[0] not in (tok.eos_id, tok.pad_id) and tok.tokens2event(row.tolist()) == [])
    out["long_invalid_events"] = float(bad)
    if neq.any():       # tie audit (SURVEY.md 8c iii): the first divergence must sit on an fp32 near-tie
        first_e = int(np.argwhere(neq.any(-1).any(0))[0][0])
        bs, ts = np.nonzero(neq[:, first_e])
        b0, t0 = int(bs[0]), int(ts[0])
        sd32 = {k_: v_.float() for k_, v_ in sd16.items()}
        ref_t = torch.from_numpy(ids_ref[b0:b0 + 1, :first_e + 1]).to(DEV)
        with torch.no_grad():
            h32 = O.forward(sd32, ocfg, ref_t[:, :-1], inv_freq=inv_n)
            l32 = O.forward_token(sd32, ocfg, h32[:, -1], ref_t[:, -1, :7], inv_freq=inv_t)
        row = l32[0, t0]
        out["long_first_divergence_event"] = float(first_e)
        out["long_first_divergence_margin"] = float((row[ids_ref[b0, first_e, t0]] - row[ids_pool[b0, first_e, t0]]).abs())
        print("long: first divergence at event", first_e, "row", b0, "token", t0, ids_ref[b0, first_e], ids_pool[b0, first_e])
        del sd32
    # ---- (b) KV-cached forward == full forward at S = 4096 (prefill 4000 events, then 96 single-event steps)
    song = _song_batch_long(tok, 1, 4100, seed=31).to(DEV)
    with torch.no_grad():
        full = model.forward(song[:, :4096])
        c = DynamicCache()
        parts = [model.forward(song[:, :4000], cache=c)]
        for t in range(4000, 4096):
            parts.append(model.forward(song[:, t:t + 1], cache=c))
        cached = torch.cat(parts, 1)
    out["cached_vs_full_hidden_S4096"] = rel(cached.float(), full.float())
    out["cached_vs_full_hidden_S4096_tail"] = rel(cached[:, 4000:].float(), full[:, 4000:].float())
    # ---- (c) beyond max_position_embeddings: cached forward to 4100 positions, and generate(max_len=4100)
    with torch.no_grad():
        for t in range(4096, 4100):
            parts.append(model.forward(song[:, t:t + 1], cache=c))
        full2 = model.forward(song[:, :4100])
    out["cached_vs_full_hidden_past4096"] = rel(torch.cat(parts[-4:], 1).float(), full2[:, 4096:].float())
    ids_long = model.generate(prompt=song[:, :4090].cpu().numpy(), batch_size=1, max_len=4100, top_k=1)
    out["generate_past4096_len"] = float(ids_long.shape[1])
    del full, full2, cached, parts, c
    # ---- (d) loss at the benchmark shape vs the oracle (bf16 and fp32 weights, same batch), forward only
    model.train()
    bb = synth_batch(tok, 8, 2049, seed=1234).to(DEV)
    with torch.no_grad():
        def oracle_loss(sd):       # train.py:168-185 with the model's own (bf16-rounded) inv_freq buffers
            yb = bb[:, 1:].reshape(-1, 8)
            hid = O.forward(sd, ocfg, bb[:, :-1].contiguous(), inv_freq=inv_n)
            lgo = O.forward_token(sd, ocfg, hid.reshape(-1, 1024), yb[:, :-1], inv_freq=inv_t)
            return float(F.cross_entropy(lgo.view(-1, ocfg.vocab), yb.reshape(-1), reduction="mean", ignore_index=ocfg.pad_id))
        l_new = float(model.training_loss(bb, backward=False))
        l_16 = oracle_loss(sd16)
        torch.cuda.empty_cache()
        sd32 = {k_: v_.float() for k_, v_ in sd16.items()}
        l_32 = oracle_loss(sd32)
        del sd32
        torch.cuda.empty_cache()
    out["bench_shape_loss_new"], out["bench_shape_loss_oracle32"] = l_new, l_32
    out["bench_shape_loss_abs_vs_oracle32"] = abs(l_new - l_32)
    out["bench_shape_loss_abs_oracle16_vs_oracle32"] = abs(l_16 - l_32)
    return out


def check_lora_train():
    """LoRA training (train.py:439-449: r = 64, lora_alpha = 128, all seven projections, frozen base) on the sm_100a engine.
    (a) the rank-r GEMM shapes the adapters add, through the C ABI, incl. the in-place strided residual epilogue;
    (b) loss and adapter gradients vs the oracle's autograd over W + scale * B A (= peft's unmerged forward in exact
    arithmetic); the frozen base gets no gradient and is bit-identical after the fused optimizer step; drop-in autograd path
    == fused path; (c) inference with injected adapters (merged decode weights) == the training-path forward."""
    from midi_b200.synth import synth_batch
    from midi_b200 import lora
    from transformers import DynamicCache
    out = {}
    r = 64
    # ---- (a) adapter GEMM shapes (rows not a multiple of 128, N = r and K = r smaller than a tile)
    for i, rows in enumerate((1000, 4096)):
        x, A, Bm = randn(rows, 1024, seed=200 + i), randn(r, 1024, scale=0.05, seed=210 + i), randn(1024, r, scale=0.05, seed=220 + i)
        t = ops.linear(x, A)                                                        # [rows, r]
        out[f"lora_gemm_down_{rows}"] = rel(t.float(), x.float() @ A.float().T)
        ts = ops.scale(t, 2.0)
        out[f"lora_scale_mismatch_{rows}"] = float((ts != (t.float() * 2.0).to(BF)).sum())
        y = randn(rows, 3072, seed=230 + i)
        y0 = y.clone()
        yv = y[:, 1024:2048]
        ops.gemm(ts, Bm, rows, 1024, r, lda=r, ldb=r, out=yv, ldc=3072, residual=yv)    # in place on the k third
        ref = ((ts.float() @ Bm.float().T).to(BF).float() + y0[:, 1024:2048].float())
        out[f"lora_gemm_up_inplace_{rows}"] = rel(y[:, 1024:2048].float(), ref)
        out[f"lora_gemm_up_untouched_{rows}"] = float((y[:, :1024] != y0[:, :1024]).sum() + (y[:, 2048:] != y0[:, 2048:]).sum())
        dy = randn(rows, 3072, seed=240 + i)
        dyv = dy[:, 2048:]
        dts = ops.gemm(dyv, Bm, rows, r, 1024, lda=3072, ldb=r, b_mn=True)          # dy . B  -> [rows, r]
        out[f"lora_gemm_dts_{rows}"] = rel(dts.float(), dyv.float() @ Bm.float())
        gB = torch.empty(1024, r, device=DEV, dtype=BF)
        ops.gemm(dyv, ts, 1024, r, rows, lda=3072, ldb=r, a_mn=True, b_mn=True, out=gB, ldc=r, allow_split=True)
        out[f"lora_gemm_gB_{rows}"] = rel(gB.float(), dyv.float().T @ ts.float())
        gA = torch.empty(r, 1024, device=DEV, dtype=BF)
        ops.gemm(dts, x, r, 1024, rows, lda=r, ldb=1024, a_mn=True, b_mn=True, out=gA, ldc=1024, allow_split=True)
        refA = dts.float().T @ x.float()
        out[f"lora_gemm_gA_{rows}"] = rel(gA.float(), refA)
        ops.gemm(dts, x, r, 1024, rows, lda=r, ldb=1024, a_mn=True, b_mn=True, out=gA, ldc=1024, accumulate=True, allow_split=True)
        out[f"lora_gemm_gA_accumulate_{rows}"] = rel(gA.float(), 2 * refA)
        dx = randn(rows, 1024, seed=250 + i)
        dx0 = dx.clone()
        ops.gemm(dts, A, rows, 1024, r, lda=r, ldb=1024, b_mn=True, out=dx, ldc=1024, residual=dx)
        out[f"lora_gemm_dx_inplace_{rows}"] = rel(dx.float(), (dts.float() @ A.float()).to(BF).float() + dx0.float())
        print(f"lora: adapter GEMM shapes at {rows} rows done", flush=True)
    torch.cuda.synchronize()
    # ---- (b) a 4-layer model of the real width: train.py:439-449
    mm, model = _model(4)
    model = model.to(DEV, dtype=BF).train()
    model.requires_grad_(False)
    model.add_adapter(lora.LoraAdapterConfig(r=r, lora_alpha=128, target_modules=["q_proj", "o_proj", "k_proj", "v_proj",
                                             "gate_proj", "up_proj", "down_proj"], lora_dropout=0, bias="none", task_type="CAUSAL_LM"))
    g = torch.Generator(device="cpu").manual_seed(5)
    with torch.no_grad():                                     # B = 0 at init would make dA vanish: give it trained-like values
        for n, p in model.named_parameters():
            if ".lora_B." in n:
                p.copy_((torch.randn(p.shape, generator=g) * 0.02).to(DEV, BF))
    ocfg = O.cfg_from_hf(model.config)
    batch = synth_batch(model.tokenizer, 2, 66, seed=77, pad_tail=3).to(DEV)
    leaf = {n: p.detach().float().requires_grad_(True) for n, p in model.named_parameters()}
    sd = O.lora_effective_sd(leaf, 2.0)          # scaling = lora_alpha / r = 128 / 64
    ref = O.train_loss(sd, ocfg, batch)
    ref.backward()
    before = {n: p.detach().clone() for n, p in model.named_parameters()}
    loss = model.training_loss(batch)
    out["lora_loss_abs"] = float((loss - ref.detach()).abs())
    print("lora: fused training step done, loss", float(loss), "oracle", float(ref.detach()), flush=True)
    tot_n = tot_d = worst = 0.0
    base_grads = 0
    for n, p in model.named_parameters():
        if ".lora_" not in n:
            base_grads += int(p.grad is not None)
            continue
        gref = leaf[n].grad
        tot_n += float((p.grad.float() - gref).double().pow(2).sum())
        tot_d += float(gref.double().pow(2).sum())
        worst = max(worst, rel(p.grad.float(), gref))
    out["lora_grad_global_rel"] = math.sqrt(tot_n / tot_d)
    out["lora_grad_worst_rel_info"] = worst
    out["lora_base_grads_present"] = float(base_grads)
    fused = {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}
    model.fused_optimizer_step(lr=1e-3, step=1)
    torch.cuda.synchronize()
    out["lora_frozen_changed"] = float(sum(int(not torch.equal(p, before[n])) for n, p in model.named_parameters() if ".lora_" not in n))
    out["lora_adapters_changed"] = float(sum(int(not torch.equal(p, before[n])) for n, p in model.named_parameters() if ".lora_" in n))
    with torch.no_grad():
        for n, p in model.named_parameters():
            p.copy_(before[n])
    for p in model.parameters():
        p.grad = None
    x, y = batch[:, :-1].contiguous(), batch[:, 1:].contiguous()
    hidden = model.forward(x)
    yy = y.reshape(-1, y.shape[-1])
    logits = model.forward_token(hidden.reshape(-1, hidden.shape[-1]), yy[:, :-1])
    l2 = F.cross_entropy(logits.view(-1, model.tokenizer.vocab_size), yy.view(-1), reduction="mean", ignore_index=model.tokenizer.pad_id)
    l2.backward()
    num = sum(float((p.grad.float() - fused[n].float()).double().pow(2).sum()) for n, p in model.named_parameters() if n in fused)
    den = sum(float(fused[n].float().double().pow(2).sum()) for n in fused)
    out["lora_dropin_vs_fused_grad_rel"] = math.sqrt(num / den)
    print("lora: drop-in step done", flush=True)
    out["lora_dropin_base_grads_present"] = float(sum(int(p.grad is not None) for n, p in model.named_parameters() if ".lora_" not in n))
    # ---- (c) inference with injected adapters: KV-cached forward (merged decode weights) vs the training-path forward
    model.eval()
    with torch.no_grad():
        full = model.forward(x[:, :40])
        c = DynamicCache()
        parts = [model.forward(x[:, :30], cache=c)] + [model.forward(x[:, t:t + 1], cache=c) for t in range(30, 40)]
        out["lora_cached_vs_full_hidden"] = rel(torch.cat(parts, 1).float(), full.float())
        href = O.forward({k: v.detach() for k, v in sd.items()}, ocfg, x[:, :40], inv_freq=model.net.rotary_emb.inv_freq)
        out["lora_hidden_vs_oracle32"] = rel(full.float(), href)
    ids = model.generate(batch_size=2, max_len=8, top_k=1)
    out["lora_generate_len"] = float(ids.shape[1])
    return out


GROUPS = {
    "gemm_fwd": check_gemm_fwd, "gemm_swiglu": check_gemm_swiglu, "gemm_dgrad": check_gemm_dgrad, "gemm_wgrad": check_gemm_wgrad,
    "elementwise": check_elementwise, "fused_rope": check_fused_rope, "attn_flash": check_attn_flash, "attn_tc05": check_attn_tc05, "attn_tiny": check_attn_tiny,
    "loss_optim": check_loss_optim, "decode": check_decode, "model_forward": check_model_forward,
    "model_layer_tf": check_model_layer_teacher_forced, "model_train": check_model_train,
    "model_generate": check_model_generate, "model_peaked_greedy": check_model_peaked_greedy, "model_large": check_model_large,
    "gemm_exact": check_gemm_exact, "decode_paged": check_decode_paged, "model_vs_hf": check_model_vs_hf,
    "model_medium_long": check_model_medium_long, "lora_train": check_lora_train,
}

# metric-name prefix -> upper bound (first matching prefix wins); "min:" entries are lower bounds
THRESH = [
    # LoRA (train.py:439-449): rank-64 GEMM shapes, adapter gradients vs the oracle's autograd, frozen base untouched
    ("lora_scale_mismatch", 0.0), ("lora_gemm_up_untouched", 0.0), ("lora_gemm_", 4e-3), ("lora_loss_abs", 3e-2),
    ("lora_grad_global_rel", 6e-2), ("lora_base_grads_present", 0.0), ("lora_frozen_changed", 0.0), ("min:lora_adapters_changed", 70.0),
    ("lora_dropin_vs_fused_grad_rel", 2e-2), ("lora_dropin_base_grads_present", 0.0), ("lora_cached_vs_full_hidden", 3e-2),
    ("lora_hidden_vs_oracle32", 3e-2), ("min:lora_generate_len", 2.0),
    # round 2: exactness of the GEMM at benchmark shapes (fraction of non-correctly-rounded elements; fp32 summation order
    # alone moves ~1e-3 of them by one ulp, long-K split sums a few 1e-3), fused decode attention across pages, HF GPU path
    # (measured: 5.6e-4 forward K=1024, 1.7e-3..4.3e-3 dgrad K=3072/8192, 3e-3..2.2e-2 wgrad over 16 384 / 131 072 rows)
    ("exact_maxulp_", 1.0), ("exact_err_over_tol_", 1.0), ("exact_frac_wgrad_", 3e-2), ("exact_frac_", 6e-3), ("wgrad_splits_", 64.0),
    ("decode_fused_append_mismatch", 0.0), ("decode_fused_T", 6e-3),
    ("hidden_new_vs_hf", 3e-2), ("logits_new_vs_hf", 4e-2), ("logits_tf_new_vs_hf", 2e-2), ("min:argmax_agree_new_hf", 0.9),
    # event-level layer: <= 1e-3 against the reference's GPU path (SURVEY.md 8c tier 1; measured 9.6e-4, the oracle's own
    # attention formulation sits 2.2e-3 from that path).  Token-level layer: torch routes (N, 4, 8, 256) to another SDPA
    # backend whose internal rounding differs; this implementation equals the oracle to 2e-5 there and both sit 2.06e-3 from
    # HF (`inner_sdpa_backend_*` metrics record each backend's distance to fp32).  Attention alone: two independent
    # bf16-P implementations are ~1e-3 apart, each 2.0e-3 from fp32.
    ("outer_layer_tf_new_vs_hf", 1e-3), ("inner_layer_tf_new_vs_hf", 3e-3), ("attn_new_vs_sdpa16", 1.5e-3),
    ("hf_loss_abs", 5e-2), ("hf_grad_global_rel", 8e-2),
    ("medium_peaked_loss_last", 0.1), ("opt_state_roundtrip_mismatch", 0.0), ("long_greedy_mismatch", 0.0),
    ("long_pool_vs_public_mismatch", 0.0), ("long_persist_vs_graph_mismatch", 0.0), ("peaked_persist_vs_graph_mismatch", 0.0),
    ("min:greedy_persist_vs_graph_agree", 0.6), ("min:long_page_boundaries_crossed", 8.0), ("long_invalid_events", 0.0),
    ("min:long_len_new", 740.0), ("cached_vs_full_hidden_S4096", 3e-2), ("cached_vs_full_hidden_past4096", 3e-2),
    ("min:generate_past4096_len", 4100.0), ("bench_shape_loss_abs_vs_oracle32", 3e-2), ("sample_seq_loss_abs", 5e-2),
    ("sample_seq_grad_global_rel", 6e-2),
    ("gemm_vocab_padcols_absmax", 0.0), ("gemm_swiglu", 0.0), ("gemm_", 4e-3), ("embed_sum_maxabs", 0.0), ("embed_bwd_padrow_absmax", 0.0),
    ("embed_bwd", 4e-3), ("inner_input_equal", 0.0), ("inner_embed_bwd", 4e-3),
    ("rmsnorm_fwd_mismatch", 2e-3), ("rmsnorm_fwd", 2e-3), ("rmsnorm_bwd", 4e-3),
    ("rope_table_mismatch", 8.0), ("rope_fwd_mismatch", 64.0), ("rope_bwd_adjoint", 2e-2),
    ("swiglu_fwd_mismatch", 2e-2), ("swiglu_bwd", 4e-3),
    ("linear_rope_mismatch", 0.0), ("tiny_fused_rope", 0.0), ("attn_bwd_fused_rope_v_mismatch", 0.0), ("attn_bwd_fused_rope", 5e-3),
    ("tc_vs_mma_bwd", 8e-3), ("tc_bwd", 1.2e-2), ("tc_vs_mma", 4e-3), ("tc_fwd", 6e-3),
    ("flash_fwd", 6e-3), ("flash_lse", 1e-4), ("flash_bwd", 1.2e-2), ("tiny_fwd", 6e-3), ("tiny_bwd", 1.2e-2),
    ("ce_loss_abs", 2e-3), ("ce_count_abs", 0.0), ("ce_bwd_padcols_absmax", 0.0), ("ce_bwd", 6e-3),
    ("ce_all_ignored_loss", 0.0), ("gradnorm_rel", 1e-4), ("adamw_maxabs", 2e-3),
    ("gemv_", 4e-3), ("decode_attn", 6e-3), ("sampler_greedy_mismatch", 0.0), ("logits_sampler_", 0.0), ("sampler_topk_outside", 0.0),
    ("sampler_dist_l1", 0.12),
    ("min:inv_freq_is_bf16", 1.0), ("margin_filtered_argmax_mismatch", 0.0),
    ("hidden_new_vs_oracle16", 3e-2), ("logits_new_vs_oracle16", 4e-2), ("logits_teacher_forced_vs_oracle16", 2e-2),
    ("outer_layer_tf", 6e-3), ("inner_layer_tf", 6e-3),
    ("large_loss_abs", 3e-2), ("large_grad_global_rel", 8e-2), ("min:large_params", 457220096.0),
    ("loss_abs", 3e-2), ("grad_global_rel", 6e-2), ("grad_pad_row", 0.0), ("autograd_loss_abs", 5e-2),
    ("autograd_grad_global_rel", 6e-2),
    ("cached_vs_full_hidden", 3e-2), ("inner_cached_vs_full_logits", 3e-2), ("min:greedy_token_agree", 0.6),
    ("min:lazy_ce_hits", 1.0), ("xy_split_mismatch", 0.0), ("prefetch_mismatch", 0.0), ("int16_path_loss_mismatch", 0.0), ("int16_path_grad_rel", 1e-3), ("stream_vs_generate_mismatch", 0.0), ("stream_masked_mismatch", 0.0), ("stream_denied_ids_emitted", 0.0),
    ("stream_mask_leak_mismatch", 0.0), ("stream_concurrent_errors", 0.0), ("stream_concurrent_mismatch", 0.0),
    ("stream_resumed_on_other_thread_mismatch", 0.0), ("peaked_greedy_mismatch", 0.0), ("peaked_eager_vs_graph_mismatch", 0.0), ("peaked_invalid_events", 0.0), ("peaked_loss_last", 1.5),
    ("peaked_argmax_mismatch_vs_fp32", 0.0), ("peaked_logits_vs_fp32", 3e-2),
    ("sampled_invalid_events", 0.0), ("greedy_graph_vs_nograph_mismatch", 0.0), ("fused_decode_mismatch", 0.0), ("fused_lm_head_mismatch", 0.0),
]


def verdict(metrics: dict):
    """Returns list of (name, value, bound, ok).  Noise-floor rules (tier 2) are added for model_forward."""
    res = []
    for k, v in metrics.items():
        bound, ok = None, True
        for pref, b in THRESH:
            if pref.startswith("min:"):
                if k.startswith(pref[4:]):
                    bound, ok = b, v >= b
                    break
            elif k.startswith(pref):
                bound, ok = b, (v <= b) and not math.isnan(v)
                break
        res.append((k, v, bound, ok))
    if "hidden_new_vs_fp32" in metrics:
        for a, b in (("hidden_new_vs_fp32", "hidden_oracle16_vs_fp32"), ("logits_new_vs_fp32", "logits_oracle16_vs_fp32")):
            res.append((a + "<=1.25x_floor", metrics[a], 1.25 * metrics[b], metrics[a] <= 1.25 * metrics[b]))
    return res
