"""GPU (-m gpu, needs >= 2 GPUs; skipped on a 1-GPU box): the multi-rank path of the extraction driver
(/root/reference/scripts/extract.py:63-131 semantics under torchrun; VERDICT r1 partial row f4).  Token-budget batches
are dealt round-robin to the ranks and every rank writes its own files: the union of the files must equal the
single-rank output, bit for bit (the batches — and therefore every kernel launch — are the same, only their owner
changes)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_torchrun_two_ranks_write_the_same_files_as_one_rank(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from oracle.weights import make_state_dict
    L, E, H = 2, 128, 2
    sd = make_state_dict(L, E, H)
    ckpt = tmp_path / "esm2_tiny.pt"
    torch.save({"cfg": {"model": {"encoder_layers": L, "encoder_embed_dim": E, "encoder_attention_heads": H,
                                  "token_dropout": True}},
                "model": {("encoder.sentence_encoder." + k): v for k, v in sd.items()}}, ckpt)
    g = torch.Generator().manual_seed(0)
    aas = "ACDEFGHIKLMNPQRSTVWY"
    seqs = {}
    for i in range(37):
        n = int(torch.randint(5, 120, (1,), generator=g))
        seqs[f"p{i}/x" if i == 3 else f"p{i}"] = "".join(aas[int(j)] for j in torch.randint(0, 20, (n,), generator=g))
    fasta = tmp_path / "in.fasta"
    fasta.write_text("".join(f">{k}\n{v}\n" for k, v in seqs.items()))
    common = [str(ckpt), str(fasta)]
    tail = ["--toks_per_batch", "256", "--include", "mean", "per_tok", "bos", "contacts"]
    env = dict(os.environ, PYTHONPATH=ROOT)
    one, two = tmp_path / "one", tmp_path / "two"
    subprocess.run([sys.executable, "-m", "esm_b200.extract_cli"] + common + [str(one)] + tail, check=True, env=env,
                   cwd=ROOT, timeout=600)
    subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                    "--master-addr", "127.0.0.1", "--master-port", "29517", "-m", "esm_b200.extract_cli"] + common +
                   [str(two)] + tail, check=True, env=env, cwd=ROOT, timeout=600)
    files_one = sorted(str(p.relative_to(one)) for p in one.rglob("*.pt"))
    files_two = sorted(str(p.relative_to(two)) for p in two.rglob("*.pt"))
    assert files_one == files_two and len(files_one) == len(seqs)
    for f in files_one:
        a, b = torch.load(one / f, weights_only=False), torch.load(two / f, weights_only=False)
        assert a["label"] == b["label"]
        for key in ("representations", "mean_representations", "bos_representations"):
            for layer in a[key]:
                assert torch.equal(a[key][layer], b[key][layer]), (f, key)
        assert torch.equal(a["contacts"], b["contacts"]), f
