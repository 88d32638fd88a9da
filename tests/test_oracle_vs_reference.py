"""-m "not gpu": the oracle against outputs of the unmodified reference, recorded in tests/golden/oracle_vs_reference.pt
by oracle/make_golden_vs_reference.py.  Weights and inputs are rebuilt from seeds and the per-tensor statistics stored
in the fixture; the reference's outputs are kept as a seeded sample of elements plus each output's max |value|.
Seeds / shapes differ from the other committed fixtures of tests/golden/."""
import pytest
import torch

from conftest import load_golden
from oracle import evoformer_oracle as O


def _sample(out, rec):
    flat = out.reshape(-1)
    return flat[O.sample_index(flat.numel(), len(rec["values"]), rec["seed"])]


@pytest.mark.parametrize("N,S,d,H,dh,depth,masked", [(24, 5, 32, 2, 16, 2, True), (17, 3, 64, 4, 16, 1, False)])
def test_evoformer_matches_live_reference_fp64(N, S, d, H, dh, depth, masked):
    case = next(c for c in load_golden("oracle_vs_reference")["evoformer"]
                if c["cfg"] == dict(N=N, S=S, d=d, H=H, dh=dh, depth=depth))
    assert (case["mask"] is not None) == masked
    st64 = {k: v.double() for k, v in O.seeded_tensors(case["spec"], case["weight_seed"]).items()}
    inp = O.seeded_tensors(case["input_spec"], case["input_seed"])
    ox, om = O.evoformer(st64, "", inp["x"].double(), inp["m"].double(), H, depth, case["mask"], case["msa_mask"])
    # fp64 vs fp64; Q3's count+eps is evaluated in fp32 by the reference -> ~1e-7 relative on the pair track
    rx, rm = case["out"]["x"], case["out"]["m"]
    assert (_sample(ox, rx) - rx["values"]).abs().max().item() <= 1e-6 * max(1.0, rx["absmax"])
    assert (_sample(om, rm) - rm["values"]).abs().max().item() <= 1e-6 * max(1.0, rm["absmax"])


def test_alphafold2_distogram_matches_live_reference_fp32():
    fx = load_golden("oracle_vs_reference")["distogram"]
    cfg = fx["cfg"]
    st = O.seeded_tensors(fx["spec"], fx["weight_seed"])
    o = O.alphafold2_distogram(st, fx["seq"], fx["msa"], fx["mask"], fx["msa_mask"], heads=cfg["heads"], depth=cfg["depth"])
    r = fx["out"]
    assert (_sample(o, r) - r["values"]).abs().max().item() <= 2e-4 * max(1.0, r["absmax"])
