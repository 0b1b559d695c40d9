"""GPU (-m gpu): the reference's layer seam running on top of libesmb200.so (INTEGRATION.md Option B).

`esm_b200.integration.patch_reference()` substitutes `TransformerLayer.forward` of the module it is given, the seam
SURVEY §8b names (`esm/modules.py:120-142` called from `esm/model/esm2.py:111-116`), exactly like the reference's own
apex FusedLayerNorm substitution (`esm/modules.py:68-81`).  Here it is given oracle/esm2_oracle.py, whose
TransformerLayer has the reference's parameter names and forward signature and whose esm2_forward(layers=...) runs the
layer loop in the reference's (T, B, E) layout; the embedding prologue, LM head and contact head stay on the host side.
Everything is compared with outputs of the unmodified reference stored under tests/golden (make_golden.py,
make_golden_dropin.py): the reference's eager fp32 results are what `esm-extract` users get today.
"""
import os

import pytest
import torch

from oracle import esm2_oracle
from oracle.weights import make_state_dict

pytestmark = pytest.mark.gpu


def rel_fro(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def checksum(sd):
    return float(sum(v.double().abs().sum() for k, v in sorted(sd.items())))


def _fixture(golden_dir, name):
    fx = torch.load(os.path.join(golden_dir, name + ".pt"), weights_only=False)
    cfg = fx["config"]
    sd = make_state_dict(cfg["num_layers"], cfg["embed_dim"], cfg["attention_heads"], seed=cfg["seed"])
    # the weights are re-created from the seed: make sure they are the ones the reference ran with
    assert abs(checksum(sd) - fx["state_dict_checksum"]) <= 1e-6 * fx["state_dict_checksum"]
    return fx, cfg["num_layers"], cfg["attention_heads"], sd


def _forward(sd, L, H, tokens, patched, **kw):
    """esm2_forward with the layer loop through TransformerLayer modules; `patched`: with the library substituted."""
    from esm_b200 import integration
    layers = esm2_oracle.layer_modules(sd, L, H)
    if patched:
        integration.patch_reference(esm2_oracle)
    try:
        with torch.no_grad():
            return esm2_oracle.esm2_forward(sd, L, H, tokens, layers=layers, **kw)
    finally:
        if patched:
            integration.unpatch_reference(esm2_oracle)


@pytest.mark.parametrize("name", ["tiny_L2_E128_H2", "mid_L3_E256_H4", "t6_8M_like_L6_E320_H20",
                                  "t48_15B_like_L2_E256_H2"])
def test_reference_esm2_forward_on_the_library(name, golden_dir):
    from esm_b200 import _lib
    fx, L, H, sd = _fixture(golden_dir, name)
    sd = {k: v.cuda() for k, v in sd.items()}
    n0 = _lib.load().esmb200_launch_count()
    out = _forward(sd, L, H, fx["tokens"].cuda(), True, repr_layers=fx["repr_layers"], need_head_weights=True,
                   return_contacts=True)
    torch.cuda.synchronize()
    launched = _lib.load().esmb200_launch_count() - n0
    assert launched >= 7 * L, "the layers did not go through libesmb200.so"
    for k, ref in fx["representations"].items():
        assert rel_fro(out["representations"][k].cpu(), ref) <= 3e-3, k
    assert rel_fro(out["logits"].cpu(), fx["logits"]) <= 4e-3
    sub = out["attentions"][:, [0, L - 1]][:, :, [0, H - 1]].cpu()
    assert float((sub - fx["attentions_sub"]).abs().max()) <= 1e-2
    assert float((out["contacts"].cpu() - fx["contacts"]).abs().max()) <= 1e-2


def test_patched_reference_equals_reference_eager_on_the_same_gpu(golden_dir):
    """What `esm-extract` users run today (scripts/extract.py:70-72: model.cuda(), eager fp32; stored) against the
    same model with the substituted layer; plus ESMFold's fp16 variant (esmfold.py:59-62)."""
    fx, L, H, sd = _fixture(golden_dir, "dropin_eager_L4_E640_H10")
    tokens = fx["tokens"].cuda()
    keep = tokens.ne(1)
    rows, eager = fx["rep_rows"].long().cuda(), fx["rep_keep_sample"]  # a fixed sample of the unpadded rows
    sd = {k: v.cuda() for k, v in sd.items()}
    fast = _forward(sd, L, H, tokens, True, repr_layers=[L])["representations"][L]
    fast16 = _forward({k: v.half() for k, v in sd.items()}, L, H, tokens, True,
                      repr_layers=range(L + 1))["representations"]
    assert rel_fro(fast[keep][rows].cpu(), eager) <= 3e-3
    assert fast16[L].dtype == torch.float16 and sorted(fast16.keys()) == list(range(L + 1))
    assert rel_fro(fast16[L].float()[keep][rows].cpu(), eager) <= 8e-3  # fp16 weights + fp16 prologue/tail


def test_reference_650M_full_size_eager_vs_library(golden_dir):
    """BASELINE.json configs[1] at full size: the unmodified reference `ESM2` (33 x 1280 x 20 heads) in eager fp32
    (stored: a fixed sample of the last representation, the logits and sequence 0's contacts) against
    the layer loop with its TransformerLayer.forward substituted, T = 1024, two sequences (one padded to 700 residues)."""
    fx, L, H, sd = _fixture(golden_dir, "dropin_eager_650M_T1024")
    sd = {k: v.cuda() for k, v in sd.items()}
    tokens = fx["tokens"].cuda()
    fast = _forward(sd, L, H, tokens, True, repr_layers=[L], return_contacts=True)
    keep = tokens.ne(1)
    rep = fast["representations"][L][keep][fx["rep_rows"].long().cuda()].cpu()
    r = rel_fro(rep, fx["rep_keep_sample"])
    rl = rel_fro(fast["logits"][keep][fx["logit_rows"].long().cuda()].cpu(), fx["logits_keep_sample"])
    c0 = fast["contacts"][0].reshape(-1)[fx["contacts0_index"].long().cuda()].cpu()
    rc = float((c0 - fx["contacts0_sample"]).abs().max())  # sequence 0 has no padding
    print(f"PARITY reference_eager_650M_T1024 repr={r:.3e} logits={rl:.3e} contacts_abs={rc:.3e}", flush=True)
    assert r <= 3e-3 and rl <= 4e-3 and rc <= 1e-2


def test_cpu_tensors_keep_the_reference_path():
    """Like the FusedLayerNorm precedent: on CPU the substituted class runs the original PyTorch code."""
    L, H = 1, 2
    sd = make_state_dict(L, 128, H, seed=0)
    tokens = torch.tensor([[0, 5, 6, 7, 8, 2]])
    want = _forward(sd, L, H, tokens, False, repr_layers=[1])["representations"][1]
    got = _forward(sd, L, H, tokens, True, repr_layers=[1])["representations"][1]
    assert torch.equal(got, want)
