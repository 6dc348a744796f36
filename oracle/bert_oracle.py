"""CPU restatement (fp32, plain torch) of the text encoder the reference runs before its backbone:
``BertModel(text, attention_mask=l_mask)[0]`` (reference lib/_utils.py:52-54, 98-100).

TEST INFRASTRUCTURE ONLY -- imported by tests/, __graft_entry__.smoke() and bench.py's CPU legs, never by the product path.

The reference's ``bert/`` package is absent from the reference checkout: it is a copy of HuggingFace Transformers **v3.0.2**
``modeling_bert.py`` (README.md:9-13), i.e. a third-party dependency.  This file restates that published algorithm
(BertEmbeddings -> 12 x [BertSelfAttention, BertSelfOutput, BertIntermediate, BertOutput]), and is pinned in
tests/test_bert_oracle.py against the ``transformers`` BertModel installed here (same architecture and state-dict keys)
on random-init weights.  Details that matter for parity:
  * embeddings = word[ids] + position[0..Nl) + token_type[0]; LayerNorm eps 1e-12
  * attention scores / sqrt(64) + (1 - mask) * -10000 (v3.0.2 extended mask; newer releases use dtype-min, identical after
    the softmax for any sentence with at least one real token)
  * GELU is the exact erf form; dropout is inactive in eval
"""
from __future__ import annotations

import math
from typing import Dict

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


def bert_forward(sd: Dict[str, Tensor], ids: Tensor, mask: Tensor, pre: str = "text_encoder.", heads: int = 12,
                 eps: float = 1e-12) -> Tensor:
    """ids (B,Nl) int64, mask (B,Nl) {0,1} -> last_hidden_state (B,Nl,H) fp32."""
    B, Nl = ids.shape
    e = pre + "embeddings."
    x = sd[e + "word_embeddings.weight"][ids] + sd[e + "position_embeddings.weight"][:Nl][None] + sd[e + "token_type_embeddings.weight"][0]
    H = x.shape[-1]
    x = F.layer_norm(x, (H,), sd[e + "LayerNorm.weight"], sd[e + "LayerNorm.bias"], eps)
    ext = (1.0 - mask.to(x.dtype))[:, None, None, :] * -10000.0
    hd = H // heads
    i = 0
    while f"{pre}encoder.layer.{i}.attention.self.query.weight" in sd:
        p = f"{pre}encoder.layer.{i}."

        def lin(t, name):
            return t @ sd[p + name + ".weight"].t() + sd[p + name + ".bias"]
        q = lin(x, "attention.self.query").view(B, Nl, heads, hd).transpose(1, 2)
        k = lin(x, "attention.self.key").view(B, Nl, heads, hd).transpose(1, 2)
        v = lin(x, "attention.self.value").view(B, Nl, heads, hd).transpose(1, 2)
        s = q @ k.transpose(-1, -2) / math.sqrt(hd) + ext
        ctx = (s.softmax(-1) @ v).transpose(1, 2).reshape(B, Nl, H)
        x = F.layer_norm(lin(ctx, "attention.output.dense") + x, (H,), sd[p + "attention.output.LayerNorm.weight"],
                         sd[p + "attention.output.LayerNorm.bias"], eps)
        h = F.gelu(lin(x, "intermediate.dense"))
        x = F.layer_norm(lin(h, "output.dense") + x, (H,), sd[p + "output.LayerNorm.weight"], sd[p + "output.LayerNorm.bias"], eps)
        i += 1
    return x
