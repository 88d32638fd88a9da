"""-m gpu: the fused transition kernel (csrc/ff_tc.cuh: LayerNorm -> Linear -> GEGLU -> Linear -> residual in one launch)
against (a) the two-launch path of the same library (fused LN -> Linear -> GEGLU, then the residual GEMM), switched in-process
with af2_set_ff_fused, and (b) the fp64 oracle."""
import pytest
import torch

from gpu_util import check, to64
from oracle import evoformer_oracle as O

pytestmark = pytest.mark.gpu


def _lib():
    from alphafold2_b200 import _lib as L
    return L.load()


@pytest.fixture(autouse=True)
def _restore():
    yield
    _lib().af2_set_ff_fused(1)


def _module(d, seed):
    import alphafold2_b200 as A
    ff = A.FeedForward(dim=d)
    torch.manual_seed(seed)
    st = {k: v.clone() for k, v in ff.state_dict().items()}
    for k, v in st.items():
        if v.dim() >= 2:
            v.copy_(torch.randn_like(v) * (v.shape[-1] ** -0.5))
        elif "norm" in k and k.endswith("weight"):
            v.copy_(1 + 0.1 * torch.randn_like(v))
        else:
            v.copy_(0.1 * torch.randn_like(v))
    ff.load_state_dict(st)
    return ff.cuda().eval(), st


def _run(ff, x, fused):
    """x + FeedForward(x) through the C ABI with the fused kernel on / off; returns (output, kernel launches issued)"""
    lib = _lib()
    lib.af2_set_ff_fused(1 if fused else 0)
    y = x.clone()
    n0 = lib.af2_launch_count()
    ff.add_to_(y)
    torch.cuda.synchronize()
    return y, lib.af2_launch_count() - n0


@pytest.mark.parametrize("shape", [(1, 256, 256, 256), (1, 128, 256, 256), (1, 8, 250, 256), (1, 3, 391, 128),
                                   (2, 3, 391, 256), (2, 8, 250, 128)])
def test_ff_fused_matches_two_launch(shape):
    d = shape[-1]
    ff, _ = _module(d, 11)
    x = torch.randn(*shape, generator=torch.Generator().manual_seed(12)).cuda()
    a, na = _run(ff, x, True)
    b, nb = _run(ff, x, False)
    assert na == 1 and nb == 2, (na, nb)
    assert torch.isfinite(a).all()
    diff = (a - b).abs().max().item()
    delta_rms = (b - x).double().pow(2).mean().sqrt().item()
    print(f"ff fused vs two-launch {tuple(shape)}: max |diff| {diff:.3e} (rms of the block's update {delta_rms:.3e})")
    # both paths round h to bf16 the same way and add (acc + b2) + x in the same order
    assert diff <= 1e-3 * delta_rms, f"fused / two-launch differ by {diff}"


@pytest.mark.parametrize("shape", [(1, 128, 256, 256), (1, 8, 250, 256), (1, 3, 391, 128), (2, 3, 391, 256)])
def test_ff_fused_oracle(shape):
    d = shape[-1]
    ff, st = _module(d, 13)
    x = torch.randn(*shape, generator=torch.Generator().manual_seed(14))
    y, n = _run(ff, x.cuda(), True)
    assert n == 1
    ref = O.feed_forward(to64(st), "", x.double())
    check(f"ff_fused/{'x'.join(map(str, shape))}", (y.cpu().double() - x.double()), ref)


@pytest.mark.parametrize("d", [192])
def test_ff_unsupported_shape_falls_back(d):
    """dims the fused kernel does not take still run (two launches) and stay correct"""
    ff, st = _module(d, 15)
    x = torch.randn(1, 5, 77, d, generator=torch.Generator().manual_seed(16))
    y, n = _run(ff, x.cuda(), True)
    assert n >= 2
    check(f"ff_fallback/d{d}", (y.cpu().double() - x.double()), O.feed_forward(to64(st), "", x.double()))
