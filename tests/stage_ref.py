"""Float64 restatement of the engine's decoder stages, rounding at the same points as the kernels.

Every product and sum is float64 on the CPU; values are rounded to bf16 (or the residual stream to
fp32) exactly where the CUDA kernels round, so a kernel can be held to about one bf16 ulp per
stage instead of a fraction of the logit scale.  With `rnd=False` every rounding point is skipped
and the functions are the plain Llama equations (tests/test_stage_reference.py pins that form
against `oracle.llama_oracle` and the reference project's numbers in tests/golden/layer_arith.json).

Rounding points, by kernel:
  RMSNorm        bf16(w * (x * rstd)) of the fp32 residual row
                 (gemm_skinny.cuh:245,321 decode, prefill_tc.cuh:157 prompt pass)
  QKV            fp32 accumulation of bf16 operands, RoPE on the fp32 sums, bf16 q / k / v
                 (gemm_skinny.cuh:587-603, prefill_tc.cuh:327-333)
  RoPE table     fp32 inv_freq (default / linear / llama3 rule), fp32 angle, cos / sin rounded to
                 fp32 (engine.cu:1099-1128); the rotation itself is done here in fp64
  attention      fp32 scores and softmax, probabilities bf16 for P.V, output bf16 (attention.cuh:7-8)
  O, down        fp32 sum added to the fp32 residual (gemm_skinny.cuh:620, prefill_tc.cuh:138-143)
  gate / up      bf16(silu(gate) * up) from the fp32 sums (gemm_skinny.cuh:575-576, prefill_tc.cuh:289-291)
  LM head        fp32 logits of the bf16 normed rows; arg-max, lowest index wins ties (common.cuh:98)
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import torch

F64 = torch.float64


def bf16(x: torch.Tensor, rnd: bool = True) -> torch.Tensor:
    return x.to(torch.bfloat16).to(F64) if rnd else x.to(F64)


def f32(x: torch.Tensor, rnd: bool = True) -> torch.Tensor:
    return x.to(torch.float32).to(F64) if rnd else x.to(F64)


def rope_inv_freq(head_dim: int, theta: float, scaling: Optional[Dict] = None) -> torch.Tensor:
    """fp32 inverse frequencies as transformers' modeling_rope_utils.py computes them."""
    exps = torch.arange(0, head_dim, 2, dtype=torch.int64).to(torch.float32) / head_dim
    inv = 1.0 / (torch.tensor(theta, dtype=torch.float32) ** exps)
    kind = (scaling or {}).get("rope_type", (scaling or {}).get("type", "default"))
    if kind in (None, "default"):
        return inv
    factor = float(scaling["factor"])
    if kind == "linear":
        return inv / factor
    assert kind == "llama3", kind
    lo, hi = float(scaling["low_freq_factor"]), float(scaling["high_freq_factor"])
    old = float(scaling["original_max_position_embeddings"])
    wavelen = 2 * math.pi / inv
    scaled = torch.where(wavelen > old / lo, inv / factor, inv)
    smooth = (old / wavelen - lo) / (hi - lo)
    mid = (1 - smooth) * scaled / factor + smooth * scaled
    medium = ~(wavelen < old / hi) & ~(wavelen > old / lo)
    return torch.where(medium, mid, scaled).to(torch.float32)


def rope_cos_sin(positions: torch.Tensor, head_dim: int, theta: float,
                 scaling: Optional[Dict] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """[n, head_dim / 2] fp32-valued cos / sin (as float64) of the fp32 angle pos * inv_freq."""
    inv = rope_inv_freq(head_dim, theta, scaling)
    ang = positions.to(torch.float32)[:, None] * inv[None, :]
    return ang.to(F64).cos().to(torch.float32).to(F64), ang.to(F64).sin().to(torch.float32).to(F64)


def rms_norm(x: torch.Tensor, w: torch.Tensor, eps: float, rnd: bool = True) -> torch.Tensor:
    """x: [s, h] residual rows, w: [h] -> bf16(w * (x * rstd))."""
    x = x.to(F64)
    rstd = torch.rsqrt((x * x).mean(-1, keepdim=True) + eps)
    return bf16(w.to(F64) * (x * rstd), rnd)


def rotate(x: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor) -> torch.Tensor:
    """x: [s, heads, hd]; pairs (d, d + hd/2) rotated by the angle of pair d (rotate_half)."""
    half = x.shape[-1] // 2
    lo, hi = x[..., :half], x[..., half:]
    c, s = cos[:, None, :], sin[:, None, :]
    return torch.cat([lo * c - hi * s, hi * c + lo * s], dim=-1)


def qkv(xn: torch.Tensor, L: Dict[str, torch.Tensor], cos: torch.Tensor, sin: torch.Tensor,
        heads: int, kv_heads: int, hd: int, rnd: bool = True):
    """Normed rows [s, h] -> q [s, heads, hd], k and v [s, kv_heads, hd] (k, q post-RoPE)."""
    s = xn.shape[0]
    q = (xn @ L["wq"].T).view(s, heads, hd)
    k = (xn @ L["wk"].T).view(s, kv_heads, hd)
    v = (xn @ L["wv"].T).view(s, kv_heads, hd)
    return bf16(rotate(q, cos, sin), rnd), bf16(rotate(k, cos, sin), rnd), bf16(v, rnd)


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, q_pos: torch.Tensor,
              rnd: bool = True) -> torch.Tensor:
    """q [s, H, hd] at positions q_pos; k, v [n, KV, hd] for positions 0..n-1 -> [s, H * hd].
    Query at position p sees keys 0..p."""
    s, H, hd = q.shape
    n, KV, _ = k.shape
    g = H // KV
    kk = k.repeat_interleave(g, dim=1).permute(1, 2, 0)        # [H, hd, n]
    vv = v.repeat_interleave(g, dim=1).permute(1, 0, 2)        # [H, n, hd]
    scores = torch.matmul(q.permute(1, 0, 2), kk) / math.sqrt(hd)   # [H, s, n]
    visible = torch.arange(n)[None, :] <= q_pos[:, None]
    scores = scores.masked_fill(~visible[None], float("-inf"))
    probs = bf16(torch.softmax(scores, dim=-1), rnd)
    out = torch.matmul(probs, vv).permute(1, 0, 2).reshape(s, H * hd)
    return bf16(out, rnd)


def mlp_act(xn: torch.Tensor, L: Dict[str, torch.Tensor], rnd: bool = True) -> torch.Tensor:
    g = xn @ L["wg"].T
    u = xn @ L["wu"].T
    return bf16(g * torch.sigmoid(g) * u, rnd)


def residual_add(x: torch.Tensor, a: torch.Tensor, w: torch.Tensor, rnd: bool = True) -> torch.Tensor:
    """x + a . w^T, stored as the fp32 residual stream."""
    return f32(x.to(F64) + a @ w.T, rnd)


def decoder_layer(x: torch.Tensor, L: Dict[str, torch.Tensor], positions: torch.Tensor,
                  k_past: torch.Tensor, v_past: torch.Tensor, cfg: Dict, rnd: bool = True):
    """One decoder layer on residual rows x [s, h] at `positions` (contiguous, following the
    n_past = k_past.shape[0] cached rows).  Returns (x_out, k_rows, v_rows, parts) where parts
    holds the intermediate stage outputs."""
    hd, H, KV = cfg["head_dim"], cfg["heads"], cfg["kv_heads"]
    cos, sin = rope_cos_sin(positions, hd, cfg["rope_theta"], cfg.get("rope_scaling"))
    xn = rms_norm(x, L["ln1"], cfg["rms_eps"], rnd)
    q, k, v = qkv(xn, L, cos, sin, H, KV, hd, rnd)
    k_all = torch.cat([k_past, k], dim=0)
    v_all = torch.cat([v_past, v], dim=0)
    attn = attention(q, k_all, v_all, positions, rnd)
    x1 = residual_add(f32(x, rnd), attn, L["wo"], rnd)
    act = mlp_act(rms_norm(x1, L["ln2"], cfg["rms_eps"], rnd), L, rnd)
    x2 = residual_add(x1, act, L["wd"], rnd)
    return x2, k, v, dict(q=q, attn=attn, x_attn=x1, act=act)


def lm_head(x: torch.Tensor, final_norm: torch.Tensor, W: torch.Tensor, eps: float,
            rnd: bool = True) -> torch.Tensor:
    return rms_norm(x, final_norm, eps, rnd) @ W.T


def argmax_lowest(logits: torch.Tensor) -> torch.Tensor:
    """Arg-max per row; on exact ties the lowest index wins (torch.argmax returns the first)."""
    best = logits.max(dim=-1, keepdim=True).values
    idx = torch.arange(logits.shape[-1]).expand_as(logits)
    return torch.where(logits == best, idx, logits.shape[-1]).min(dim=-1).values


# ---------------------------------------------------------------------------------------------
# comparison in bf16 units
# ---------------------------------------------------------------------------------------------
def bf16_ulp(x: torch.Tensor) -> torch.Tensor:
    """Spacing of bf16 values at |x| (8 significant bits), as float64; normal range only."""
    a = x.to(F64).abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 7)


def ulp_error(got: torch.Tensor, ref: torch.Tensor, floor) -> torch.Tensor:
    """|got - ref| in bf16 ulps of the unrounded reference.  `floor` (absolute, a float or a tensor
    that broadcasts against `ref`) is the smallest unit used: an element that nearly cancels is
    only as exact as the fp32 sums it came from, whose error scales with the row, not with it."""
    ref = ref.to(F64)
    unit = torch.maximum(bf16_ulp(ref), torch.as_tensor(floor, dtype=F64))
    return (got.to(F64) - ref).abs() / unit


def row_floor(ref: torch.Tensor) -> torch.Tensor:
    """One bf16 ulp of the RMS of each row (dims after the first), shaped to broadcast."""
    dims = tuple(range(1, ref.dim()))
    return bf16_ulp(ref.to(F64).pow(2).mean(dim=dims, keepdim=True).sqrt())
