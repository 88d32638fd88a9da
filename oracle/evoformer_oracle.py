"""TEST INFRASTRUCTURE ONLY — CPU restatement of the reference Evoformer trunk forward.

This is the *oracle* for the hot path of lucidrains/alphafold2 (reference files are
cited as ``alphafold2.py:LINE`` = /root/reference/alphafold2_pytorch/alphafold2.py).
It is a functional (no nn.Module) restatement in plain torch on the CPU, dtype-generic
(fp32 = the parity target, fp64 = ground truth for error budgets), driven by a flat
``dict`` of weights that uses the reference's own ``state_dict`` key names.

Pinned: ``tests/test_oracle_golden.py`` checks every function here against fixtures in
tests/golden/ that were produced by the unmodified reference (oracle/make_golden.py),
and ``tests/test_oracle_vs_reference.py`` checks it against outputs the reference computed
on seeded weights and inputs (oracle/make_golden_vs_reference.py).  It must never be
imported by ``alphafold2_b200``.

Two deliberate differences from the literal reference, both validated against it:
  * ``outer_mean(..., literal=False)`` contracts over the MSA axis with an einsum instead of
    materialising the (S, N, N, d) tensor of alphafold2.py:341 (77 GB at config C3);
    ``literal=True`` follows the reference line by line (used as the CPU baseline).
  * attention can be evaluated in chunks of the folded batch axis to bound memory.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
W = Dict[str, Tensor]


def _lin(w: W, key: str, x: Tensor) -> Tensor:
    """nn.Linear: y = x W^T + b (weight is [out, in])."""
    b = w.get(key + ".bias")
    return F.linear(x, w[key + ".weight"].to(x.dtype), None if b is None else b.to(x.dtype))


def _ln(w: W, key: str, x: Tensor, eps: float = 1e-5) -> Tensor:
    """nn.LayerNorm over the last dim, eps 1e-5, affine (alphafold2.py:82,210,269,289,330)."""
    d = x.shape[-1]
    return F.layer_norm(x, (d,), w[key + ".weight"].to(x.dtype), w[key + ".bias"].to(x.dtype), eps)


# --------------------------------------------------------------------------------------
# FeedForward / GEGLU  (alphafold2.py:69-94)
# --------------------------------------------------------------------------------------
def feed_forward(w: W, p: str, x: Tensor) -> Tensor:
    """LN -> Linear(d, 8d) -> a * gelu_erf(g) -> Linear(4d, d).  No residual (caller adds)."""
    h = _lin(w, p + "net.0", _ln(w, p + "norm", x))
    a, g = h.chunk(2, dim=-1)                       # alphafold2.py:71
    h = a * F.gelu(g)                               # exact erf GELU, alphafold2.py:72
    return _lin(w, p + "net.3", h)


# --------------------------------------------------------------------------------------
# Attention  (alphafold2.py:98-190)  — self-attention form used inside the trunk
# --------------------------------------------------------------------------------------
def attention(w: W, p: str, x: Tensor, heads: int, mask: Optional[Tensor] = None,
              attn_bias: Optional[Tensor] = None, tie_dim: Optional[int] = None) -> Tensor:
    """x: [B', n, d]; mask: [B', n] bool or None; attn_bias: [B' or 1, H, n, n] or None.

    Quirk Q1: the mask is the outer product mask[q] * mask[k] filled with -finfo.max
    (alphafold2.py:162-167), so a masked *query* row attends uniformly to all keys.
    """
    Bp, n, _ = x.shape
    q = _lin(w, p + "to_q", x)
    k, v = _lin(w, p + "to_kv", x).chunk(2, dim=-1)             # alphafold2.py:130
    dh = q.shape[-1] // heads
    q, k, v = (t.reshape(Bp, n, heads, dh).permute(0, 2, 1, 3) for t in (q, k, v))
    q = q * dh ** -0.5                                          # alphafold2.py:138
    if tie_dim is not None:                                     # alphafold2.py:142-151
        q = q.reshape(Bp // tie_dim, tie_dim, heads, n, dh).mean(dim=1)
        k = k.reshape(Bp // tie_dim, tie_dim, heads, n, dh)
        dots = torch.einsum("bhid,brhjd->brhij", q, k).reshape(Bp, heads, n, n)
    else:
        dots = torch.einsum("bhid,bhjd->bhij", q, k)
    if attn_bias is not None:
        dots = dots + attn_bias.to(dots.dtype)
    if mask is not None:
        pair = mask[:, None, :, None] & mask[:, None, None, :]
        dots = dots.masked_fill(~pair, -torch.finfo(dots.dtype).max)
    attn = dots.softmax(dim=-1)
    out = torch.einsum("bhij,bhjd->bhid", attn, v)
    out = out.permute(0, 2, 1, 3).reshape(Bp, n, heads * dh)
    out = out * _lin(w, p + "gating", x).sigmoid()              # alphafold2.py:184-185
    return _lin(w, p + "to_out", out)


# --------------------------------------------------------------------------------------
# AxialAttention  (alphafold2.py:192-255)
# --------------------------------------------------------------------------------------
def axial_attention(w: W, p: str, x: Tensor, heads: int, row_attn: bool,
                    edges: Optional[Tensor] = None, mask: Optional[Tensor] = None,
                    global_query_attn: bool = False, chunk: int = 0) -> Tensor:
    """x: [b, h, w, d].  row_attn folds (b h) and attends along w; col folds (b w), attends along h.

    Quirks Q4/Q5: the pair bias is a bias-free Linear(d, H) of the RAW (un-normalised) edges,
    laid out [b, H, i, j] and repeated unchanged for every folded row/column
    (alphafold2.py:245-248) — not transposed for the column variant.
    """
    b, h, wd, d = x.shape
    xn = _ln(w, p + "norm", x)
    if row_attn:
        xf = xn.reshape(b * h, wd, d)
        mf = None if mask is None else mask.reshape(b * h, wd)
        axial = h
    else:
        xf = xn.permute(0, 2, 1, 3).reshape(b * wd, h, d)
        mf = None if mask is None else mask.permute(0, 2, 1).reshape(b * wd, h)
        axial = wd
    bias = None
    if edges is not None and (p + "edges_to_attn_bias.0.weight") in w:
        eb = F.linear(edges, w[p + "edges_to_attn_bias.0.weight"].to(edges.dtype))   # [b,i,j,H]
        bias = eb.permute(0, 3, 1, 2)                                                # [b,H,i,j]
    tie = axial if global_query_attn else None
    Bp = xf.shape[0]
    if chunk and tie is None and Bp > chunk:
        outs = []
        for s in range(0, Bp, chunk):
            e = min(Bp, s + chunk)
            bb = None
            if bias is not None:
                # folded index = b_idx * axial + r  ->  bias of batch b_idx
                idx = torch.arange(s, e, device=bias.device) // axial
                bb = bias[idx]
            outs.append(attention(w, p + "attn.", xf[s:e], heads, None if mf is None else mf[s:e], bb))
        of = torch.cat(outs, dim=0)
    else:
        bb = None if bias is None else bias.repeat_interleave(axial, dim=0)
        of = attention(w, p + "attn.", xf, heads, mf, bb, tie)
    if row_attn:
        return of.reshape(b, h, wd, d)
    return of.reshape(b, wd, h, d).permute(0, 2, 1, 3)


# --------------------------------------------------------------------------------------
# TriangleMultiplicativeModule  (alphafold2.py:257-317)
# --------------------------------------------------------------------------------------
def triangle_multiply(w: W, p: str, x: Tensor, mix: str, mask: Optional[Tensor] = None) -> Tensor:
    """x: [b, N, N, d]; mask: [b, N, N] bool.  Quirk Q6: 'ingoing' is sum_k L[k,j] R[k,i]."""
    assert x.shape[1] == x.shape[2], "feature map must be symmetrical"
    xn = _ln(w, p + "norm", x)
    left = _lin(w, p + "left_proj", xn)
    right = _lin(w, p + "right_proj", xn)
    if mask is not None:
        mk = mask[..., None].to(x.dtype)
        left = left * mk
        right = right * mk
    left = left * _lin(w, p + "left_gate", xn).sigmoid()
    right = right * _lin(w, p + "right_gate", xn).sigmoid()
    out_gate = _lin(w, p + "out_gate", xn).sigmoid()
    if mix == "outgoing":
        out = torch.einsum("bikd,bjkd->bijd", left, right)      # alphafold2.py:285
    elif mix == "ingoing":
        out = torch.einsum("bkjd,bkid->bijd", left, right)      # alphafold2.py:287
    else:
        raise ValueError(mix)
    out = _ln(w, p + "to_out_norm", out) * out_gate
    return _lin(w, p + "to_out", out)


# --------------------------------------------------------------------------------------
# OuterMean  (alphafold2.py:321-351)
# --------------------------------------------------------------------------------------
def outer_mean(w: W, p: str, m: Tensor, mask: Optional[Tensor] = None, eps: float = 1e-5,
               literal: bool = False) -> Tensor:
    """m: [b, S, N, d]; mask: [b, S, N] bool.

    Quirk Q3: the masked branch divides the *mean over S* by (count + eps) again
    (alphafold2.py:347), and count + eps is evaluated in the default dtype (fp32).
    """
    mn = _ln(w, p + "norm", m)
    left = _lin(w, p + "left_proj", mn)
    right = _lin(w, p + "right_proj", mn)
    S = m.shape[1]
    if literal:
        outer = left[:, :, :, None, :] * right[:, :, None, :, :]            # alphafold2.py:341
        if mask is not None:
            pm = mask[:, :, :, None, None] & mask[:, :, None, :, None]
            outer = outer.masked_fill(~pm, 0.)
            outer = outer.mean(dim=1) / (pm.sum(dim=1) + eps)
        else:
            outer = outer.mean(dim=1)
    else:
        if mask is not None:
            mk = mask[..., None].to(m.dtype)
            left, right = left * mk, right * mk
            outer = torch.einsum("bsid,bsjd->bijd", left, right) / S
            mf = mask.to(torch.float32)
            cnt = torch.einsum("bsi,bsj->bij", mf, mf)                       # exact small integers
            denom = (cnt + eps)[..., None]                                   # fp32 like the reference
            outer = outer / denom
        else:
            outer = torch.einsum("bsid,bsjd->bijd", left, right) / S
    return _lin(w, p + "proj_out", outer.to(m.dtype) if not literal else outer)


# --------------------------------------------------------------------------------------
# Blocks  (alphafold2.py:353-467)
# --------------------------------------------------------------------------------------
def pairwise_attention_block(w: W, p: str, x: Tensor, heads: int, mask=None, msa_repr=None,
                             msa_mask=None, literal_outer: bool = False, chunk: int = 0,
                             global_column_attn: bool = False) -> Tensor:
    if msa_repr is not None:
        x = x + outer_mean(w, p + "outer_mean.", msa_repr, msa_mask, literal=literal_outer)
    x = triangle_multiply(w, p + "triangle_multiply_outgoing.", x, "outgoing", mask) + x
    x = triangle_multiply(w, p + "triangle_multiply_ingoing.", x, "ingoing", mask) + x
    x = axial_attention(w, p + "triangle_attention_outgoing.", x, heads, True, x, mask, chunk=chunk) + x
    x = axial_attention(w, p + "triangle_attention_ingoing.", x, heads, False, x, mask,
                        global_query_attn=global_column_attn, chunk=chunk) + x
    return x


def msa_attention_block(w: W, p: str, m: Tensor, heads: int, mask=None, pairwise_repr=None,
                        chunk: int = 0) -> Tensor:
    m = axial_attention(w, p + "row_attn.", m, heads, True, pairwise_repr, mask, chunk=chunk) + m
    m = axial_attention(w, p + "col_attn.", m, heads, False, None, mask, chunk=chunk) + m
    return m


def evoformer_block(w: W, p: str, x: Tensor, m: Tensor, heads: int, mask=None, msa_mask=None,
                    literal_outer: bool = False, chunk: int = 0, global_column_attn: bool = False):
    """Order (alphafold2.py:438-444): MSA attn -> MSA FF -> pair block (updated m) -> pair FF.
    global_column_attn (alphafold2.py:367, 421): the pair block's ingoing triangle attention ties its queries."""
    m = msa_attention_block(w, p + "layer.2.", m, heads, msa_mask, x, chunk)
    m = feed_forward(w, p + "layer.3.", m) + m
    x = pairwise_attention_block(w, p + "layer.0.", x, heads, mask, m, msa_mask, literal_outer, chunk, global_column_attn)
    x = feed_forward(w, p + "layer.1.", x) + x
    return x, m


def evoformer(w: W, p: str, x: Tensor, m: Tensor, heads: int, depth: int, mask=None, msa_mask=None,
              literal_outer: bool = False, chunk: int = 0, global_column_attn: bool = False):
    for l in range(depth):
        x, m = evoformer_block(w, f"{p}layers.{l}.", x, m, heads, mask, msa_mask, literal_outer, chunk, global_column_attn)
    return x, m


# --------------------------------------------------------------------------------------
# Alphafold2.forward, distogram-only path  (alphafold2.py:630-726, 802-823)
# --------------------------------------------------------------------------------------
def alphafold2_distogram(w: W, seq: Tensor, msa: Optional[Tensor], mask: Optional[Tensor],
                         msa_mask: Optional[Tensor], heads: int, depth: int, max_rel_dist: int = 32,
                         dtype=torch.float32, literal_outer: bool = False, chunk: int = 0,
                         return_trunk: bool = False, extra_msa_mask: Optional[Tensor] = None, extra_depth: int = 0):
    """seq [b,n] int64, msa [b,s,n] int64, mask [b,n] bool, msa_mask [b,s,n] bool -> distance logits.
    extra_depth > 0: the extra-MSA stack of alphafold2.py:789-798 runs first, exactly as the reference does (quirk Q11: it
    embeds `msa` again, keeps only the pair output; its blocks use global_column_attn, alphafold2.py:518-527)."""
    if msa is None:                                                         # alphafold2.py:656-658
        msa = seq[:, None, :]
        msa_mask = mask[:, None, :]
    b, n = seq.shape
    emb = w["token_emb.weight"].to(dtype)
    x1 = emb[seq]
    m = emb[msa] + x1[:, None]
    if msa_mask is None:
        msa_mask = torch.ones_like(msa).bool()
    pr = _lin(w, "to_pairwise_repr", x1)
    xl, xr = pr.chunk(2, dim=-1)
    x = xl[:, :, None, :] + xr[:, None, :, :]
    x_mask = (mask[:, :, None] & mask[:, None, :]) if mask is not None else None
    idx = torch.arange(n, device=seq.device)
    rel = (idx[:, None] - idx[None, :]).clamp(-max_rel_dist, max_rel_dist) + max_rel_dist
    x = x + w["pos_emb.weight"].to(dtype)[rel][None]
    if extra_depth > 0:
        extra_m = emb[msa]                                                    # alphafold2.py:790 (sic: msa, not extra_msa)
        x, _ = evoformer(w, "extra_msa_evoformer.", x, extra_m, heads, extra_depth, x_mask, extra_msa_mask, literal_outer, chunk,
                         global_column_attn=True)
    x, m = evoformer(w, "net.", x, m, heads, depth, x_mask, msa_mask, literal_outer, chunk)
    if return_trunk:
        return x, m
    te = (x + x.transpose(1, 2)) * 0.5
    return _lin(w, "to_distogram_logits.1", _ln(w, "to_distogram_logits.0", te))


# --------------------------------------------------------------------------------------
# rotary.py:9-20 (dead code at HEAD, named in north_star)
# --------------------------------------------------------------------------------------
def apply_rotary_pos_emb(x: Tensor, sin: Tensor, cos: Tensor) -> Tensor:
    """x [b, h, n, dh]; sin/cos [b or 1, n, rot].  Interleaved pairs (x0,x1)->(x0 c - x1 s, x1 c + x0 s);
    channels >= rot pass through unchanged."""
    sin, cos = sin[:, None], cos[:, None]
    rot = sin.shape[-1]
    xr, xp = x[..., :rot], x[..., rot:]
    x2 = xr.reshape(*xr.shape[:-1], rot // 2, 2)
    rot_half = torch.stack((-x2[..., 1], x2[..., 0]), dim=-1).reshape(xr.shape)
    return torch.cat((xr * cos + rot_half * sin, xp), dim=-1)


def fixed_positional_embedding(dim: int, n: int):
    """rotary.py:35-45: returns [sin, cos] each [1, n, dim] with every frequency repeated twice."""
    inv_freq = 1.0 / (10000 ** (torch.arange(0, dim, 2).float() / dim))
    freqs = torch.arange(n).float()[:, None] * inv_freq[None, :]
    freqs = freqs.repeat_interleave(2, dim=-1)[None]
    return freqs.sin(), freqs.cos()


# --------------------------------------------------------------------------------------
# helpers shared by tests / bench
# --------------------------------------------------------------------------------------
def randomize_zero_init_(state: W, std: float = 0.02, seed: int = 1234) -> W:
    """Quirk Q8: to_out / FF out are zero-init and all gates are W=0,b=1, so a fresh model
    is an identity on the MSA track.  Replace every all-zero / all-one tensor by N(0,std)
    (+1 for the all-one gate biases) so parity tests exercise every path."""
    g = torch.Generator().manual_seed(seed)
    for k, t in state.items():
        if not torch.is_floating_point(t) or t.numel() == 0:
            continue
        if bool((t == 0).all()):
            t.copy_(torch.randn(t.shape, generator=g) * std)
        elif bool((t == 1).all()) and (".gating." in k or "_gate." in k):
            t.copy_(1.0 + torch.randn(t.shape, generator=g) * std)
    return state


def seeded_tensors(spec: Dict[str, tuple], seed: int) -> W:
    """spec {name: (shape, mean, std)} -> {name: fp32 tensor of N(mean, std)}, drawn in spec order from one seeded
    generator.  Lets a fixture pin weights and inputs by their statistics instead of storing them."""
    g = torch.Generator().manual_seed(seed)
    return {k: torch.randn(tuple(shape), generator=g) * std + mean for k, (shape, mean, std) in spec.items()}


def sample_index(numel: int, k: int, seed: int) -> Tensor:
    """A fixed, seeded choice of min(k, numel) flat indices, for fixtures that keep a sample of a larger output."""
    return torch.randperm(numel, generator=torch.Generator().manual_seed(seed))[:k]


def evoformer_flops_per_block(N: int, S: int, d: int, H: int, dh: int) -> float:
    """Algorithmic matmul FLOPs (2*MAC) of one EvoformerBlock — SURVEY.md §8(d)."""
    I = H * dh
    Tm, Tx = S * N, N * N
    msa_row = 10 * Tm * d * I + 2 * Tx * d * H + 4 * S * N * N * I
    msa_col = 10 * Tm * d * I + 4 * N * S * S * I
    msa_ff = 24 * Tm * d * d
    outer = 4 * Tm * d * d + 2 * N * N * S * d + 2 * Tx * d * d
    tri_mul = 2 * (12 * Tx * d * d + 2 * N ** 3 * d)
    tri_attn = 2 * (10 * Tx * d * I + 2 * Tx * d * H + 4 * N ** 3 * I)
    pair_ff = 24 * Tx * d * d
    return float(msa_row + msa_col + msa_ff + outer + tri_mul + tri_attn + pair_ff)
