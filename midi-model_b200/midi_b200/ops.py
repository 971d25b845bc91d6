"""Thin Python wrappers over the C ABI: one function per kernel family, tensors in / tensors out.

Only shapes, pointer extraction and workspace management live here; the arithmetic is in
`csrc/*.cu`.  All tensors are CUDA bf16 unless noted.
"""
from __future__ import annotations

import math
from typing import Optional

import torch

from . import lib

BF16 = torch.bfloat16
_ws_cache: dict = {}
GEMM_PROFILE = None   # bench.py sets this to a list: (start_event, end_event, flops) per tensor-core GEMM launch


def _ws(key, nbytes: int, device, zero: bool = False) -> torch.Tensor:
    """Per-(key, device, stream) byte workspace, grown on demand (kernels are stream-ordered).  `zero`: zero-filled when
    (re)allocated, for kernels that keep a self-cleaning accumulator / ticket in it."""
    k = (key, device.index, torch.cuda.current_stream().cuda_stream)
    t = _ws_cache.get(k)
    if t is None or t.numel() < nbytes:
        alloc = torch.zeros if zero else torch.empty
        t = alloc(max(nbytes, 256), dtype=torch.uint8, device=device)
        _ws_cache[k] = t
    return t


def _check(t: torch.Tensor, name: str):
    if not t.is_cuda or t.dtype != BF16 or not t.is_contiguous():
        raise lib.B200Error(f"{name}: expected a contiguous CUDA bfloat16 tensor, got {t.dtype} on {t.device} "
                            f"(contiguous={t.is_contiguous()}); the B200 path has no fallback")


# ------------------------------------------------------------------ embeddings
def embed_sum(ids: torch.Tensor, table: torch.Tensor) -> torch.Tensor:
    ids = ids.contiguous()            # the kernel assumes row pitch T (a [:, p:p+1] slice reshaped to 2-D is NOT)
    M, T = ids.shape
    V, H = table.shape
    out = torch.empty((M, H), dtype=BF16, device=table.device)
    lib.call("b200_embed_sum_fwd", ids.data_ptr(), table.data_ptr(), out.data_ptr(), M, T, H, V, lib.stream())
    return out


def inner_input(hidden: Optional[torch.Tensor], ids: Optional[torch.Tensor], table: torch.Tensor) -> torch.Tensor:
    V, H = table.shape
    if ids is not None:
        ids = ids.contiguous()
    if hidden is not None:
        hidden = hidden.contiguous()
    n_events = hidden.shape[0] if hidden is not None else ids.shape[0]
    n_ids = 0 if ids is None else ids.shape[1]
    Tin = n_ids + (1 if hidden is not None else 0)
    out = torch.empty((n_events * Tin, H), dtype=BF16, device=table.device)
    lib.call("b200_inner_input_fwd", lib.ptr(hidden), lib.ptr(ids), table.data_ptr(), out.data_ptr(), n_events, n_ids, H, V,
             lib.stream())
    return out


def batch_to_xy(batch: torch.Tensor):
    """int16 [B, S+1, T] token batch (train.py:71) -> (x, y) int64 [B*S, T]: x = batch[:, :-1], y = batch[:, 1:]."""
    if not batch.is_cuda or batch.dtype != torch.int16 or not batch.is_contiguous():
        raise lib.B200Error(f"batch_to_xy: expected a contiguous CUDA int16 batch, got {batch.dtype} on {batch.device}")
    B, S1, T = batch.shape
    x = torch.empty((B * (S1 - 1), T), dtype=torch.long, device=batch.device)
    y = torch.empty_like(x)
    lib.call("b200_batch_to_xy_i16", batch.data_ptr(), B, S1, T, x.data_ptr(), y.data_ptr(), lib.stream())
    return x, y


def embed_bwd(ids: torch.Tensor, dout: torch.Tensor, dtable: torch.Tensor, per_row: int, row_stride: int, row_inner: int,
              row_off: int, pad_id: int, accumulate: bool):
    V, H = dtable.shape
    n = ids.numel()
    nbytes = lib.query("b200_embed_bwd_workspace_bytes", n, V, H)
    ws = _ws("embed_bwd", nbytes, dtable.device)
    lib.call("b200_embed_bwd", ids.data_ptr(), n, dout.data_ptr(), dtable.data_ptr(), V, H, per_row, row_stride, row_inner,
             row_off, pad_id, int(accumulate), ws.data_ptr(), ws.numel(), lib.stream())


# ------------------------------------------------------------------ norm / rope / swiglu
def rmsnorm(x: torch.Tensor, w: torch.Tensor, eps: float, want_rstd: bool = False):
    M, H = x.shape
    y = torch.empty_like(x)
    rstd = torch.empty((M,), dtype=torch.float32, device=x.device) if want_rstd else None
    lib.call("b200_rmsnorm_fwd", x.data_ptr(), w.data_ptr(), y.data_ptr(), lib.ptr(rstd), M, H, eps, lib.stream())
    return (y, rstd) if want_rstd else y


def add_rmsnorm(x: torch.Tensor, res: torch.Tensor, w: torch.Tensor, eps: float):
    """h = x + res (residual add, bf16-rounded), y = rmsnorm(h) * w  ->  (h, y, rstd) in one pass over the rows."""
    M, H = x.shape
    h = torch.empty_like(x)
    y = torch.empty_like(x)
    rstd = torch.empty((M,), dtype=torch.float32, device=x.device)
    lib.call("b200_add_rmsnorm_fwd", x.data_ptr(), res.data_ptr(), w.data_ptr(), h.data_ptr(), y.data_ptr(), rstd.data_ptr(),
             M, H, eps, lib.stream())
    return h, y, rstd


def rmsnorm_bwd(dy, x, w, rstd, dres, dw, accumulate_dw: bool) -> torch.Tensor:
    M, H = x.shape
    dx = torch.empty_like(x)
    parts = lib.query("b200_rmsnorm_bwd_parts")
    ws = _ws("rms_bwd", parts * H * 4, x.device, zero=True)
    lib.call("b200_rmsnorm_bwd", dy.data_ptr(), x.data_ptr(), w.data_ptr(), rstd.data_ptr(), lib.ptr(dres), dx.data_ptr(),
             lib.ptr(dw), M, H, int(accumulate_dw), ws.data_ptr(), ws.numel(), lib.stream())
    return dx


def rope_table(inv_freq: torch.Tensor, n_pos: int, pos0: int = 0):
    """cos/sin tables [n_pos, d/2] from the module's `inv_freq` buffer AS STORED (bf16-rounded after
    model.to(bf16)), upcast to fp32 like hf modeling_llama.py:125-133."""
    inv = inv_freq.detach().to(torch.float32).contiguous()
    half = inv.numel()
    cos = torch.empty((n_pos, half), dtype=BF16, device=inv.device)
    sin = torch.empty_like(cos)
    lib.call("b200_rope_table", inv.data_ptr(), half, n_pos, pos0, None, cos.data_ptr(), sin.data_ptr(), lib.stream())
    return cos, sin


def rope_qk_(qkv: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor, S: int, H: int, D: int, backward: bool = False,
             pos0: int = 0, pos0_dev: Optional[torch.Tensor] = None):
    """cos/sin are indexed by absolute position; row r sits at pos0 (+ *pos0_dev) + r % S."""
    rows, ld = qkv.shape
    lib.call("b200_rope_qk", qkv.data_ptr(), cos.data_ptr(), sin.data_ptr(), rows, S, H, D, ld, int(backward), pos0,
             lib.ptr(pos0_dev), lib.stream())


def swiglu(gu: torch.Tensor) -> torch.Tensor:
    rows, two_i = gu.shape
    act = torch.empty((rows, two_i // 2), dtype=BF16, device=gu.device)
    lib.call("b200_swiglu_fwd", gu.data_ptr(), act.data_ptr(), rows, two_i // 2, lib.stream())
    return act


def swiglu_bwd(gu: torch.Tensor, dact: torch.Tensor) -> torch.Tensor:
    rows, two_i = gu.shape
    dgu = torch.empty_like(gu)
    lib.call("b200_swiglu_bwd", gu.data_ptr(), dact.data_ptr(), dgu.data_ptr(), rows, two_i // 2, lib.stream())
    return dgu


def scale(x: torch.Tensor, s: float) -> torch.Tensor:
    """bf16(x * s) as a new tensor (x itself when s == 1): the LoRA scaling lora_alpha / r (peft lora/layer.py: `* scaling`)."""
    if s == 1.0:
        return x
    _check(x, "scale input")
    y = torch.empty_like(x)
    lib.call("b200_scale_bf16", x.data_ptr(), y.data_ptr(), x.numel(), float(s), lib.stream())
    return y


# ------------------------------------------------------------------ GEMM
_plan_cache: dict = {}


def _plan(M: int, N: int, K: int, allow_split: bool):
    """(block_n, splits) from the library's cost model (cached per shape)."""
    key = (M, N, K, allow_split)
    p = _plan_cache.get(key)
    if p is None:
        import ctypes
        bn, sp = ctypes.c_int(0), ctypes.c_int(0)
        lib.load().b200_gemm_plan(M, N, K, int(allow_split), ctypes.byref(bn), ctypes.byref(sp))
        p = (bn.value, sp.value)
        _plan_cache[key] = p
    return p


_tail_cache: dict = {}


def _tail_bytes(M: int, N: int, K: int, block_n: int) -> int:
    key = (M, N, K, block_n)
    v = _tail_cache.get(key)
    if v is None:
        v = int(lib.query("b200_gemm_tail_workspace_bytes", M, N, K, block_n))
        _tail_cache[key] = v
    return v


def gemm(A: torch.Tensor, B: torch.Tensor, M: int, N: int, K: int, *, lda: int, ldb: int, a_mn: bool = False,
         b_mn: bool = False, out: Optional[torch.Tensor] = None, ldc: Optional[int] = None,
         residual: Optional[torch.Tensor] = None, accumulate: bool = False, allow_split: bool = False) -> torch.Tensor:
    """C[M,N] = A . B^T on tcgen05 tensor cores (see csrc/gemm_tcgen05.cu)."""
    if out is None:
        out = torch.empty((M, N), dtype=BF16, device=A.device)
    if ldc is None:
        ldc = out.stride(0)
    block_n, splits = _plan(M, N, K, bool(allow_split and residual is None and ldc == N and N % 8 == 0))
    ws_ptr, ws_bytes = None, 0
    if splits > 1 or accumulate:
        nbytes = lib.query("b200_gemm_workspace_bytes", M, N, max(splits, 1))
        if nbytes == 0:
            nbytes = M * N * 4
        ws = _ws("gemm", nbytes, A.device)
        ws_ptr, ws_bytes = ws.data_ptr(), ws.numel()
    elif residual is None:
        tb = _tail_bytes(M, N, K, block_n)          # optional: lets the library split the last partial wave along K
        if tb:
            ws = _ws("gemm_tail", tb, A.device)
            ws_ptr, ws_bytes = ws.data_ptr(), ws.numel()
    ldr = residual.stride(0) if residual is not None else 0
    prof = GEMM_PROFILE
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    lib.call("b200_gemm_bf16", A.data_ptr(), B.data_ptr(), out.data_ptr(), lib.ptr(residual), M, N, K, lda, ldb, ldc, ldr,
             int(a_mn), int(b_mn), int(accumulate), block_n, splits, ws_ptr, ws_bytes, lib.stream())
    if prof is not None:
        e1.record()
        prof.append((e0, e1, 2.0 * M * N * K, (M, N, K, int(a_mn), int(b_mn), block_n, splits)))
    return out


def linear(x: torch.Tensor, w: torch.Tensor, residual: Optional[torch.Tensor] = None,
           pitch: Optional[int] = None) -> torch.Tensor:
    """y = x @ w.T (+ residual).  x [M,K], w [N,K].  `pitch`: row pitch of the output when N is not a multiple of
    8 (V = 3406 -> 3408): columns N..roundup8(N) are written as zeros (TMA zero-fills weight rows beyond N)."""
    M, K = x.shape
    N = w.shape[0]
    out = None
    if pitch is not None:
        out = torch.empty((M, pitch), dtype=BF16, device=x.device)
    return gemm(x, w, M, N, K, lda=x.stride(0), ldb=w.stride(0), residual=residual, out=out)


def linear_swiglu(x: torch.Tensor, w_gu: torch.Tensor):
    """(gu, act): gu = x @ w_gu.T with w_gu = [gate | up] rows, act = silu(gate) * up formed in the GEMM epilogue."""
    M, K = x.shape
    I = w_gu.shape[0] // 2
    gu = torch.empty((M, 2 * I), dtype=BF16, device=x.device)
    act = torch.empty((M, I), dtype=BF16, device=x.device)
    prof = GEMM_PROFILE
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    lib.call("b200_gemm_bf16_swiglu", x.data_ptr(), w_gu.data_ptr(), gu.data_ptr(), act.data_ptr(), M, I, K, x.stride(0),
             w_gu.stride(0), 2 * I, I, lib.stream())
    if prof is not None:
        e1.record()
        prof.append((e0, e1, 4.0 * M * I * K, (M, 2 * I, K, 0, 0, 256, 1)))
    return gu, act


def linear_dgrad(dy: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """dx[M,K] = dy[M,:N] @ w[N,K]  (B operand = w as stored, 'MN-major'); dy may have a row pitch > N."""
    M = dy.shape[0]
    N, K = w.shape
    return gemm(dy, w, M, K, N, lda=dy.stride(0), ldb=w.stride(0), b_mn=True)


def linear_wgrad(dy: torch.Tensor, x: torch.Tensor, dw: torch.Tensor, accumulate: bool):
    """dw[N,K] (+)= dy[M,:N]^T @ x[M,K]  (both operands as stored, 'MN-major')."""
    M, K = x.shape
    N = dw.shape[0]
    gemm(dy, x, N, K, M, lda=dy.stride(0), ldb=x.stride(0), a_mn=True, b_mn=True, out=dw, ldc=K, accumulate=accumulate,
         allow_split=True)


# ------------------------------------------------------------------ attention
def _strides_packed(S: int, H: int, D: int, col0: int, ld: int):
    # element strides (batch, row, head) for a [B*S, ld] packed activation, starting at column col0
    return [S * ld, ld, D]


# impl: "tc" = tcgen05 / TMEM / TMA kernels (csrc/attn_tc05.cu); "mma" = mma.sync kernels (csrc/attn_flash.cu), the reference
# the tc kernels are tested against
def attn_causal_fwd(qkv: torch.Tensor, B: int, S: int, n_heads: int, D: int, want_lse: bool, impl: str = "tc"):
    """qkv: [B*S, 3H] packed post-RoPE -> out [B*S, H], lse [B, h, S] fp32."""
    H = n_heads * D
    ld = qkv.stride(0)
    out = torch.empty((B * S, H), dtype=BF16, device=qkv.device)
    lse = torch.empty((B, n_heads, S), dtype=torch.float32, device=qkv.device) if want_lse else None
    st = torch.tensor([S * ld, ld, D] * 3 + [S * H, H, D], dtype=torch.int64)
    base = qkv.data_ptr()
    fn = "b200_attn_causal_fwd_tc" if impl == "tc" else "b200_attn_causal_fwd"
    lib.call(fn, base, base + 2 * H, base + 4 * H, out.data_ptr(), lib.ptr(lse), st.data_ptr(), B,
             n_heads, S, S, D, 1.0 / math.sqrt(D), lib.stream())
    return out, lse


def attn_causal_bwd(qkv: torch.Tensor, out: torch.Tensor, dout: torch.Tensor, lse: torch.Tensor, B: int, S: int,
                    n_heads: int, D: int, rope=None, impl: str = "tc") -> torch.Tensor:
    """`rope=(cos, sin)`: also apply the RoPE backward to dq, dk (gradient w.r.t. the pre-rotation projections)."""
    if impl == "tc":
        return _attn_causal_bwd_tc(qkv, out, dout, lse, B, S, n_heads, D, rope)
    H = n_heads * D
    ld = qkv.stride(0)
    dqkv = torch.empty_like(qkv)
    delta = torch.empty((B, n_heads, S), dtype=torch.float32, device=qkv.device)
    pk = [S * ld, ld, D]
    po = [S * H, H, D]
    st = torch.tensor(pk * 3 + po + po + pk * 3, dtype=torch.int64)
    b, d = qkv.data_ptr(), dqkv.data_ptr()
    lib.call("b200_attn_causal_bwd", b, b + 2 * H, b + 4 * H, out.data_ptr(), dout.data_ptr(), lse.data_ptr(),
             delta.data_ptr(), d, d + 2 * H, d + 4 * H, st.data_ptr(), B, n_heads, S, S, D, 1.0 / math.sqrt(D),
             rope[0].data_ptr() if rope else None, rope[1].data_ptr() if rope else None, lib.stream())
    return dqkv


def _attn_causal_bwd_tc(qkv, out, dout, lse, B, S, n_heads, D, rope):
    H = n_heads * D
    ld = qkv.stride(0)
    dqkv = torch.empty_like(qkv)
    pk = [S * ld, ld, D]
    po = [S * H, H, D]
    st = torch.tensor(pk * 3 + po + po + pk * 3, dtype=torch.int64)
    nbytes = lib.query("b200_attn_causal_bwd_tc_workspace_bytes", B, n_heads, S)
    ws = _ws("attn_bwd_tc", nbytes, qkv.device)
    b, d = qkv.data_ptr(), dqkv.data_ptr()
    lib.call("b200_attn_causal_bwd_tc", b, b + 2 * H, b + 4 * H, out.data_ptr(), dout.data_ptr(), lse.data_ptr(), d, d + 2 * H,
             d + 4 * H, st.data_ptr(), B, n_heads, S, S, D, 1.0 / math.sqrt(D), rope[0].data_ptr() if rope else None,
             rope[1].data_ptr() if rope else None, ws.data_ptr(), ws.numel(), lib.stream())
    return dqkv


def attn_tiny_fwd(qkv: torch.Tensor, n_events: int, L: int, n_heads: int, D: int, rope=None) -> torch.Tensor:
    """`rope=(cos, sin)`: qkv holds pre-RoPE projections; q and k are rotated IN PLACE inside the kernel (fused RoPE)."""
    H = n_heads * D
    out = torch.empty((n_events * L, H), dtype=BF16, device=qkv.device)
    lib.call("b200_attn_tiny_fwd", qkv.data_ptr(), out.data_ptr(), n_events, L, n_heads, D, qkv.stride(0), H,
             1.0 / math.sqrt(D), rope[0].data_ptr() if rope else None, rope[1].data_ptr() if rope else None, lib.stream())
    return out


def attn_tiny_bwd(qkv: torch.Tensor, dout: torch.Tensor, n_events: int, L: int, n_heads: int, D: int, rope=None) -> torch.Tensor:
    dqkv = torch.empty_like(qkv)
    lib.call("b200_attn_tiny_bwd", qkv.data_ptr(), dout.data_ptr(), dqkv.data_ptr(), n_events, L, n_heads, D, qkv.stride(0),
             dout.stride(0), 1.0 / math.sqrt(D), rope[0].data_ptr() if rope else None, rope[1].data_ptr() if rope else None,
             lib.stream())
    return dqkv


def linear_rope(x: torch.Tensor, w_qkv: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor, S: int, D: int) -> torch.Tensor:
    """Packed QKV projection with RoPE applied to the q and k thirds inside the GEMM epilogue."""
    M, K = x.shape
    N = w_qkv.shape[0]
    out = torch.empty((M, N), dtype=BF16, device=x.device)
    prof = GEMM_PROFILE
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    lib.call("b200_gemm_bf16_rope", x.data_ptr(), w_qkv.data_ptr(), out.data_ptr(), M, N, K, x.stride(0), w_qkv.stride(0), N,
             cos.data_ptr(), sin.data_ptr(), S, D, 2 * N // 3, lib.stream())
    if prof is not None:
        e1.record()
        prof.append((e0, e1, 2.0 * M * N * K, (M, N, K, 0, 0, 256, 1)))
    return out


# ------------------------------------------------------------------ loss
def ce_fwd(logits: torch.Tensor, targets: torch.Tensor, V: int, ignore_index: int):
    """logits [R, ld] bf16 (ld >= V), targets [R] int64 -> (loss_and_count fp32[2], lse fp32[R])."""
    R, ld = logits.shape[0], logits.stride(0)
    lse = torch.empty((R,), dtype=torch.float32, device=logits.device)
    row_loss = torch.empty((R,), dtype=torch.float32, device=logits.device)
    lac = torch.empty((2,), dtype=torch.float32, device=logits.device)
    lib.call("b200_ce_fwd", logits.data_ptr(), targets.data_ptr(), lse.data_ptr(), row_loss.data_ptr(), lac.data_ptr(), R, V,
             ld, ignore_index, lib.stream())
    return lac, lse


def ce_bwd_(logits: torch.Tensor, targets: torch.Tensor, lse: torch.Tensor, lac: torch.Tensor, V: int, ignore_index: int,
            grad_scale: float = 1.0, grad_scale_dev: Optional[torch.Tensor] = None):
    """In place: logits <- d(loss)/d(logits) * grad_scale [* grad_scale_dev (0-dim CUDA tensor, fp32 or bf16)]."""
    R, ld = logits.shape[0], logits.stride(0)
    is_bf16 = 0
    if grad_scale_dev is not None:
        if grad_scale_dev.dtype not in (torch.float32, BF16) or not grad_scale_dev.is_cuda:
            grad_scale_dev = grad_scale_dev.to(device=logits.device, dtype=torch.float32)
        is_bf16 = int(grad_scale_dev.dtype == BF16)
    lib.call("b200_ce_bwd", logits.data_ptr(), targets.data_ptr(), lse.data_ptr(), lac.data_ptr(), R, V, ld, ignore_index,
             grad_scale, lib.ptr(grad_scale_dev), is_bf16, lib.stream())
