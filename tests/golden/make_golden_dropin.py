"""Generates tests/golden/dropin_*.pt: outputs of the UNMODIFIED reference's ESM2 in eager fp32, the results
tests/test_gpu_reference_dropin.py compares the library-backed layer loop against.

    python tests/golden/make_golden_dropin.py <reference checkout (facebookresearch/esm)>

Weights and tokens come from oracle/weights.py (re-created by the tests from the seeds; the state-dict checksum is
stored and verified).  Outputs are sampled with a fixed seed to keep the files small: 32 of the unpadded
representation rows of the small case; 24 representation rows, 128 logit rows and 4096 entries of sequence 0's contact
map of the full-size case (esm2_t33_650M shape, T = 1024).
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle.weights import make_state_dict, make_tokens  # noqa: E402

SOURCE = "facebookresearch/esm @ 2b36991 (fair-esm 2.0.1) ESM2, eager fp32, torch %s CPU" % torch.__version__


def checksum(sd):
    """the same sum as make_golden.checksum"""
    return float(sum(v.double().abs().sum() for k, v in sorted(sd.items())))


def sample(n, k, g):
    return torch.randperm(n, generator=g)[:k].sort().values


def reference_model(esm, L, E, H):
    sd = make_state_dict(L, E, H, seed=0)
    model = esm.model.esm2.ESM2(num_layers=L, embed_dim=E, attention_heads=H, alphabet="ESM-1b")
    model.load_state_dict(sd, strict=True)
    return model.eval(), checksum(sd)


@torch.no_grad()
def small(esm):
    L, E, H = 4, 640, 10
    model, ck = reference_model(esm, L, E, H)
    tokens = make_tokens([200, 131], 202, seed=2, n_mask=1)
    rep = model(tokens, repr_layers=[L])["representations"][L][tokens.ne(1)]
    rows = sample(rep.shape[0], 32, torch.Generator().manual_seed(0))
    return {"config": {"num_layers": L, "embed_dim": E, "attention_heads": H, "seed": 0}, "state_dict_checksum": ck,
            "tokens": tokens, "rep_rows": rows.to(torch.int32), "rep_keep_sample": rep[rows].clone(), "reference": SOURCE}


@torch.no_grad()
def full_size(esm):
    L, E, H = 33, 1280, 20
    model, ck = reference_model(esm, L, E, H)
    tokens = make_tokens([1022, 700], 1024, seed=4, n_mask=3)
    out = model(tokens, repr_layers=[L], return_contacts=True)
    keep = tokens.ne(1)
    rep, logits, contacts = out["representations"][L][keep], out["logits"][keep], out["contacts"][0]
    g = torch.Generator().manual_seed(0)
    rows, lrows, cidx = sample(rep.shape[0], 24, g), sample(logits.shape[0], 128, g), sample(contacts.numel(), 4096, g)
    return {"config": {"num_layers": L, "embed_dim": E, "attention_heads": H, "seed": 0}, "state_dict_checksum": ck,
            "tokens": tokens, "rep_rows": rows.to(torch.int32), "rep_keep_sample": rep[rows].clone(),
            "logit_rows": lrows.to(torch.int32), "logits_keep_sample": logits[lrows].clone(),
            "contacts0_index": cidx.to(torch.int32),
            "contacts0_sample": contacts.reshape(-1)[cidx].clone(), "reference": SOURCE}


def main():
    sys.path.insert(0, os.path.abspath(sys.argv[1]))
    import esm  # the reference
    import esm.model.esm2  # noqa: F401
    torch.set_num_threads(os.cpu_count() or 1)
    for name, make in (("dropin_eager_L4_E640_H10", small), ("dropin_eager_650M_T1024", full_size)):
        path = os.path.join(HERE, name + ".pt")
        torch.save(make(esm), path)
        print(name, "->", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
