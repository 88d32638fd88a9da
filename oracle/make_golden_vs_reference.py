"""TEST INFRASTRUCTURE ONLY — tests/golden/oracle_vs_reference.pt from the UNMODIFIED reference (run in the dev container):
    python -m oracle.make_golden_vs_reference

The reference's Evoformer (fp64) and Alphafold2.forward (fp32) run on weights and inputs that
``evoformer_oracle.seeded_tensors`` rebuilds from a seed and per-tensor (shape, mean, std), so the fixture stores only
those statistics, the masks, the token ids and a seeded sample (``evoformer_oracle.sample_index``) of every output
together with that output's max |value|.  The statistics are those of the reference's own initialisation after the Q8
randomisation, so the weights have the scales the reference gives them.  tests/test_oracle_vs_reference.py reruns the
oracle on the rebuilt inputs and compares it on the sampled elements.
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.ref_loader import load_reference  # noqa: E402
from oracle.evoformer_oracle import randomize_zero_init_, sample_index, seeded_tensors  # noqa: E402
from oracle.make_golden import OUT  # noqa: E402

SAMPLE = 2048
EVOFORMER_CASES = [(24, 5, 32, 2, 16, 2, True), (17, 3, 64, 4, 16, 1, False)]     # N, S, d, H, dh, depth, masked
DISTOGRAM_KEYS = ("token_emb.", "to_pairwise_repr.", "pos_emb.", "net.", "to_distogram_logits.")


def stats_spec(state):
    return {k: (list(v.shape), v.double().mean().item(), v.double().std(unbiased=False).item()) for k, v in state.items()}


def sampled(out, seed):
    flat = out.reshape(-1)
    return {"seed": seed, "values": flat[sample_index(flat.numel(), SAMPLE, seed)].clone(), "absmax": flat.abs().max().item()}


def main():
    ref = load_reference()
    fx = {"sample": SAMPLE, "evoformer": [], "distogram": None}

    for N, S, d, H, dh, depth, masked in EVOFORMER_CASES:
        torch.manual_seed(11 + N)
        evo = ref.Evoformer(depth=depth, dim=d, seq_len=N, heads=H, dim_head=dh, attn_dropout=0., ff_dropout=0.).eval()
        spec = stats_spec(randomize_zero_init_({k: v.clone() for k, v in evo.state_dict().items()}, seed=N))
        mask = msa_mask = None
        if masked:
            m1 = torch.ones(1, N, dtype=torch.bool)
            m1[:, -3:] = False
            mask = m1[:, :, None] & m1[:, None, :]
            msa_mask = torch.rand(1, S, N) > 0.15
            msa_mask[:, :, -3:] = False
            msa_mask[:, 0, :N - 3] = True
        case = {"cfg": dict(N=N, S=S, d=d, H=H, dh=dh, depth=depth), "weight_seed": N, "spec": spec, "input_seed": 11 + N,
                "input_spec": {"x": ([1, N, N, d], 0.0, 1.0), "m": ([1, S, N, d], 0.0, 1.0)}, "mask": mask, "msa_mask": msa_mask}
        evo.load_state_dict(seeded_tensors(spec, case["weight_seed"]))
        evo = evo.double()
        inp = seeded_tensors(case["input_spec"], case["input_seed"])
        with torch.no_grad():
            rx, rm = evo(inp["x"].double(), inp["m"].double(), mask=mask, msa_mask=msa_mask)
        case["out"] = {"x": sampled(rx, 1), "m": sampled(rm, 2)}
        fx["evoformer"].append(case)
        print("evoformer", case["cfg"], "x absmax", case["out"]["x"]["absmax"])

    torch.manual_seed(5)
    cfg = dict(dim=32, depth=1, heads=2, dim_head=16)
    model = ref.Alphafold2(**cfg).eval()
    full = randomize_zero_init_({k: v.clone() for k, v in model.state_dict().items()}, seed=3)
    spec = stats_spec({k: v for k, v in full.items() if k.startswith(DISTOGRAM_KEYS)})
    full.update(seeded_tensors(spec, 3))                     # the keys the distogram never reads keep the reference's values
    model.load_state_dict(full)
    seq = torch.randint(0, 21, (1, 20))
    msa = torch.randint(0, 21, (1, 3, 20))
    mask = torch.ones(1, 20, dtype=torch.bool)
    mask[:, -2:] = False
    msa_mask = torch.ones(1, 3, 20, dtype=torch.bool)
    msa_mask[:, :, -2:] = False
    with torch.no_grad():
        r = model(seq, msa, mask=mask, msa_mask=msa_mask).distance
    fx["distogram"] = {"cfg": cfg, "weight_seed": 3, "spec": spec, "seq": seq, "msa": msa, "mask": mask, "msa_mask": msa_mask,
                       "out": sampled(r, 3)}
    print("distogram absmax", fx["distogram"]["out"]["absmax"])
    torch.save(fx, os.path.join(OUT, "oracle_vs_reference.pt"))
    print("wrote oracle_vs_reference")


if __name__ == "__main__":
    main()
