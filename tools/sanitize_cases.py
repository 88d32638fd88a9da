"""Small cases for tools/gpu_sanitize.sh: one C1-shape EvoformerBlock (every fused kernel: CTA-pair projection, tcgen05
attention with resident bias, per-channel GEMMs, TMA channel->token), one fused feed-forward at d = 256 and one attention
with n > 256 (streamed bias)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import alphafold2_b200 as A  # noqa: E402
from bench import randomize_zero_init_  # noqa: E402

torch.manual_seed(0)
case = os.environ.get("AF2_SAN_CASE", "all")
if case in ("all", "block"):
    d, H, dh, N, S = 128, 4, 32, 64, 4
    blk = A.EvoformerBlock(dim=d, seq_len=N, heads=H, dim_head=dh, attn_dropout=0., ff_dropout=0.)
    randomize_zero_init_(blk)
    blk = blk.cuda().eval()
    x, m = torch.randn(1, N, N, d, device="cuda"), torch.randn(1, S, N, d, device="cuda")
    mask = torch.ones(1, N, N, dtype=torch.bool, device="cuda")
    mask[:, -5:] = False
    msa_mask = torch.ones(1, S, N, dtype=torch.bool, device="cuda")
    xo, mo = blk.update_(x, m, mask, msa_mask)
    torch.cuda.synchronize()
    assert torch.isfinite(xo).all() and torch.isfinite(mo).all()
    print("block ok")
if case in ("all", "ff"):
    # fused transition kernel (ff_tc_kernel) at d = 256 with a ragged row count: partial last unit, clusters with 1 and 2 units
    ff = A.FeedForward(dim=256)
    randomize_zero_init_(ff)
    ff = ff.cuda().eval()
    x = torch.randn(1, 3, 391, 256, device="cuda")
    y = ff.add_to_(x.reshape(-1, 256).clone())
    torch.cuda.synchronize()
    assert torch.isfinite(y).all()
    print("fused feed-forward ok")
if case in ("all", "attn"):
    d, H, dh, n, rows = 128, 2, 64, 300, 3
    ax = A.AxialAttention(dim=d, heads=H, dim_head=dh, row_attn=True, col_attn=False, accept_edges=True)
    randomize_zero_init_(ax)
    ax = ax.cuda().eval()
    x = torch.randn(1, rows, n, d, device="cuda")
    edges = torch.randn(1, n, n, d, device="cuda")
    out = ax(x, edges=edges)
    torch.cuda.synchronize()
    assert torch.isfinite(out).all()
    print("attention n>256 ok")
if case in ("all", "strict") and os.environ.get("AF2_SAN_STRICT", "1") != "0" and hasattr(A, "set_precision"):
    try:
        d, H, dh, N, S = 64, 2, 32, 24, 3
        blk = A.EvoformerBlock(dim=d, seq_len=N, heads=H, dim_head=dh, attn_dropout=0., ff_dropout=0.)
        randomize_zero_init_(blk)
        blk = A.set_precision(blk.cuda().eval(), "strict")
        x, m = torch.randn(1, N, N, d, device="cuda"), torch.randn(1, S, N, d, device="cuda")
        xo, mo = blk.update_(x, m, None, None)
        torch.cuda.synchronize()
        assert torch.isfinite(xo).all()
        print("strict block ok")
    except NotImplementedError as e:
        print("strict mode not built:", e)
