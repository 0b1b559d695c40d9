"""ORACLE — test infrastructure only, never a product path.

CPU restatement (PyTorch fp32 ATen ops, batch-major, functional over a plain state dict) of the reference algorithm
for the ESM-2 forward path.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / `--impl reference`
legs may import this module; esm_b200/ never does (tests/test_abi.py greps for that).

Parity pinning: the reference's own tests hold no offline golden vectors for ESM-2 numerics (SURVEY §8c), so this
restatement is pinned against OUTPUTS OF THE REFERENCE ITSELF: tests/golden/make_golden.py imports
/root/reference/esm, loads the deterministic weights of oracle/weights.py into esm.model.esm2.ESM2 and stores its
outputs under tests/golden/*.pt; tests/test_oracle_golden.py checks this file against them (fp32 noise, <= 2e-5).

Each function cites the reference lines it follows (paths relative to /root/reference/).
"""
from __future__ import annotations

import math
from typing import Dict, Iterable, Optional

import torch
import torch.nn.functional as F

PAD, MASK, CLS, EOS = 1, 32, 0, 2  # "ESM-1b" alphabet ids, esm/data.py:151-157 (tests/test_alphabet.py:17-23)


def gelu(x: torch.Tensor) -> torch.Tensor:
    """esm/modules.py:17-24 — exact erf GELU."""
    return x * 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0)))


def layer_norm(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    """esm/modules.py:68-81 — ESM1bLayerNorm resolves to torch.nn.LayerNorm (apex absent), eps 1e-5, affine."""
    return F.layer_norm(x, (x.shape[-1],), w, b, eps)


def rope_tables(inv_freq: torch.Tensor, seq_len: int):
    """esm/rotary_embedding.py:47-61 — angle[t, j] = t * inv_freq[j]; the reference concatenates the table with
    itself on the last dim, i.e. element j and j + d/2 share an angle."""
    t = torch.arange(seq_len).type_as(inv_freq)
    freqs = torch.einsum("i,j->ij", t, inv_freq)
    return freqs.cos(), freqs.sin()  # [T, d/2]


def apply_rope(x: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor) -> torch.Tensor:
    """esm/rotary_embedding.py:11-20 — x*cos + rotate_half(x)*sin with rotate_half(x) = cat(-x2, x1).
    x: [B, H, T, d]; written out per half: (x1*cos - x2*sin, x2*cos + x1*sin)."""
    d2 = x.shape[-1] // 2
    x1, x2 = x[..., :d2], x[..., d2:]
    return torch.cat((x1 * cos - x2 * sin, x2 * cos + x1 * sin), dim=-1)


def attention(x: torch.Tensor, sd: Dict[str, torch.Tensor], pre: str, num_heads: int,
              padding_mask: Optional[torch.Tensor], want_probs: bool):
    """esm/multihead_attention.py:256-261 (q/k/v Linear, q *= d^-1/2), :280-284 (head split n = h*d + j),
    :354-355 (RoPE on q and k), :357 (QK^T), :368-374 (-inf on padded keys), :379 (fp32 softmax),
    :387 (PV), :394-395 (merge heads, out_proj).  x: [B, T, E] (already layer-normed). Returns (y, probs[B,H,T,T])."""
    B, T, E = x.shape
    d = E // num_heads
    q = F.linear(x, sd[pre + "q_proj.weight"], sd[pre + "q_proj.bias"]) * (d ** -0.5)
    k = F.linear(x, sd[pre + "k_proj.weight"], sd[pre + "k_proj.bias"])
    v = F.linear(x, sd[pre + "v_proj.weight"], sd[pre + "v_proj.bias"])
    q = q.view(B, T, num_heads, d).transpose(1, 2)
    k = k.view(B, T, num_heads, d).transpose(1, 2)
    v = v.view(B, T, num_heads, d).transpose(1, 2)
    cos, sin = rope_tables(sd[pre + "rot_emb.inv_freq"], T)
    q, k = apply_rope(q, cos, sin), apply_rope(k, cos, sin)
    s = torch.matmul(q, k.transpose(-1, -2))  # [B,H,T,T]
    if padding_mask is not None:
        s = s.masked_fill(padding_mask[:, None, None, :], float("-inf"))
    p = torch.softmax(s.float(), dim=-1)
    o = torch.matmul(p, v).transpose(1, 2).reshape(B, T, E)
    y = F.linear(o, sd[pre + "out_proj.weight"], sd[pre + "out_proj.bias"])
    return y, (p if want_probs else None)


def transformer_layer(x: torch.Tensor, sd: Dict[str, torch.Tensor], pre: str, num_heads: int,
                      padding_mask: Optional[torch.Tensor], want_probs: bool):
    """esm/modules.py:120-142 — x += MHA(LN1(x)); x += fc2(gelu(fc1(LN2(x)))). x: [B, T, E]."""
    h = layer_norm(x, sd[pre + "self_attn_layer_norm.weight"], sd[pre + "self_attn_layer_norm.bias"])
    a, probs = attention(h, sd, pre + "self_attn.", num_heads, padding_mask, want_probs)
    x = x + a
    h = layer_norm(x, sd[pre + "final_layer_norm.weight"], sd[pre + "final_layer_norm.bias"])
    h = gelu(F.linear(h, sd[pre + "fc1.weight"], sd[pre + "fc1.bias"]))
    x = x + F.linear(h, sd[pre + "fc2.weight"], sd[pre + "fc2.bias"])
    return x, probs


class TransformerLayer(torch.nn.Module):
    """esm/modules.py:84-142 as a module: the reference's parameter names, `use_rotary_embeddings` and forward signature
    ((T, B, E) in and out, per-head probabilities (H, B, T, T) when need_head_weights), evaluated by transformer_layer().
    It gives tests the reference's layer seam (what esm_b200.integration.patch_reference substitutes) without the
    reference package."""

    use_rotary_embeddings = True

    def __init__(self, embed_dim: int, attention_heads: int):
        super().__init__()
        E, nn = embed_dim, torch.nn
        self.self_attn = nn.Module()
        for name in ("q_proj", "k_proj", "v_proj", "out_proj"):
            setattr(self.self_attn, name, nn.Linear(E, E))
        self.self_attn.num_heads = attention_heads
        self.self_attn.bias_k = None
        self.self_attn.rot_emb = nn.Module()
        self.self_attn.rot_emb.register_buffer("inv_freq", torch.zeros(E // attention_heads // 2))
        self.self_attn_layer_norm = nn.LayerNorm(E)
        self.fc1 = nn.Linear(E, 4 * E)
        self.fc2 = nn.Linear(4 * E, E)
        self.final_layer_norm = nn.LayerNorm(E)

    def forward(self, x, self_attn_mask=None, self_attn_padding_mask=None, need_head_weights=False):
        assert self_attn_mask is None
        y, p = transformer_layer(x.transpose(0, 1), self.state_dict(), "", self.self_attn.num_heads,
                                 self_attn_padding_mask, need_head_weights)
        return y.transpose(0, 1), (p.transpose(0, 1) if need_head_weights else None)


def layer_modules(sd: Dict[str, torch.Tensor], num_layers: int, num_heads: int):
    """The layers of a state dict as TransformerLayer modules (on the device and in the dtype of `sd`)."""
    E = sd["embed_tokens.weight"].shape[1]
    layers = []
    for i in range(num_layers):
        pre = f"layers.{i}."
        with torch.device("meta"):  # no initialisation: every tensor is assigned from `sd`
            m = TransformerLayer(E, num_heads)
        m.load_state_dict({k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}, strict=True, assign=True)
        layers.append(m)
    return layers


def embed(tokens: torch.Tensor, sd: Dict[str, torch.Tensor], token_dropout: bool = True) -> torch.Tensor:
    """esm/model/esm2.py:82-95 — embedding gather, <mask> rows zeroed and x * 0.88 / (1 - n_mask/n_nonpad) when
    token_dropout (active at inference), pad rows zeroed."""
    pad = tokens.eq(PAD)
    x = sd["embed_tokens.weight"][tokens]
    if token_dropout:
        x = x.masked_fill((tokens == MASK).unsqueeze(-1), 0.0)
        src_len = (~pad).sum(-1)
        ratio = (tokens == MASK).sum(-1).to(x.dtype) / src_len
        x = x * (1 - 0.15 * 0.8) / (1 - ratio)[:, None, None]
    return x * (1 - pad.unsqueeze(-1).type_as(x))


def lm_head(x: torch.Tensor, sd: Dict[str, torch.Tensor]) -> torch.Tensor:
    """esm/modules.py:308-314 — dense -> gelu -> LayerNorm -> tied-embedding projection + bias."""
    h = gelu(F.linear(x, sd["lm_head.dense.weight"], sd["lm_head.dense.bias"]))
    h = layer_norm(h, sd["lm_head.layer_norm.weight"], sd["lm_head.layer_norm.bias"])
    return F.linear(h, sd["embed_tokens.weight"]) + sd["lm_head.bias"]


def contact_head(tokens: torch.Tensor, attentions: torch.Tensor, sd: Dict[str, torch.Tensor]) -> torch.Tensor:
    """esm/modules.py:338-357 with symmetrize :27-29 and apc :32-41. attentions: [B, L, H, T, T]."""
    keep = tokens.ne(EOS).to(attentions)
    attentions = attentions * (keep.unsqueeze(1) * keep.unsqueeze(2))[:, None, None]
    attentions = attentions[..., 1:-1, 1:-1]  # strip <cls> row/col and the last (eos/pad) row/col
    B, L, H, S, _ = attentions.shape
    a = attentions.reshape(B, L * H, S, S)
    a = a + a.transpose(-1, -2)
    a1, a2, a12 = a.sum(-1, keepdim=True), a.sum(-2, keepdim=True), a.sum((-1, -2), keepdim=True)
    a = a - a1 * a2 / a12
    logit = F.linear(a.permute(0, 2, 3, 1), sd["contact_head.regression.weight"], sd["contact_head.regression.bias"])
    return torch.sigmoid(logit.squeeze(3))


@torch.no_grad()
def esm2_forward(sd: Dict[str, torch.Tensor], num_layers: int, num_heads: int, tokens: torch.Tensor,
                 repr_layers: Iterable[int] = (), need_head_weights: bool = False, return_contacts: bool = False,
                 token_dropout: bool = True, layers=None):
    """esm/model/esm2.py:77-144 — same result dict as ESM2.forward.  `layers`: modules with the reference's
    TransformerLayer interface (layer_modules()) that run the layer loop in its (T, B, E) layout, as esm2.py:105-121
    does; by default the functional transformer_layer() runs it."""
    if return_contacts:
        need_head_weights = True
    repr_layers = set(repr_layers)
    pad = tokens.eq(PAD)
    x = embed(tokens, sd, token_dropout)
    hidden = {}
    if 0 in repr_layers:
        hidden[0] = x
    mask = pad if bool(pad.any()) else None
    probs = []
    for i in range(num_layers):
        if layers is None:
            x, p = transformer_layer(x, sd, f"layers.{i}.", num_heads, mask, need_head_weights)
        else:
            y, p = layers[i](x.transpose(0, 1), self_attn_padding_mask=mask, need_head_weights=need_head_weights)
            x, p = y.transpose(0, 1), (p.transpose(0, 1) if need_head_weights else None)
        if (i + 1) in repr_layers:
            hidden[i + 1] = x
        if need_head_weights:
            probs.append(p)
    x = layer_norm(x, sd["emb_layer_norm_after.weight"], sd["emb_layer_norm_after.bias"])
    if num_layers in repr_layers:
        hidden[num_layers] = x  # esm2.py:127-128: the last representation is post-LayerNorm
    out = {"logits": lm_head(x, sd), "representations": hidden}
    if need_head_weights:
        att = torch.stack(probs, 1)  # [B, L, H, T, T]
        if mask is not None:
            am = 1 - mask.type_as(att)
            att = att * (am.unsqueeze(1) * am.unsqueeze(2))[:, None, None]
        out["attentions"] = att
        if return_contacts:
            out["contacts"] = contact_head(tokens, att, sd)
    return out
