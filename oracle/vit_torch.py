"""ORACLE (test infrastructure): fp32 PyTorch restatement of the CLIP ViT-L/14 image tower, the
aesthetic head and the tag similarity, as the reference runs them
(processing/scorer.py:661-664, :578-582; models/tagger.py:99-101).

open_clip (requirements.txt:8, `open-clip-torch>=2.20.0`) is third-party, not vendored under
/root/reference and not installed in this image, and the reference has no test that pins its
outputs.  The forward pass below follows open_clip's published `VisionTransformer.forward` /
`ResidualAttentionBlock` with `nn.MultiheadAttention` semantics (fused in_proj, 16 heads, scale
1/sqrt(64)).  Pinned against two independent implementations:
  * `tests/test_oracle_vit_hf.py`: HuggingFace `transformers.CLIPVisionModelWithProjection` (the tower
    open_clip's ViT-L-14 checkpoints convert to) loaded with the same tensors, all 24 layers, pooled
    output and per-layer hidden states at rtol 1e-4;
  * `tests/test_oracle_vit.py`: torch.nn.MultiheadAttention modules on a 2-layer slice.
open_clip's own code cannot be run here, so what remains unpinned is only the claim that open_clip's
`ViT-L-14` is this architecture (SURVEY.md §8c).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

HEADS = 16


def encode_image(sd: dict, x: torch.Tensor, layers: int | None = None, return_tokens: bool = False):
    """x [B,3,224,224] -> un-normalised features [B,768] (open_clip encode_image), in the dtype of x and sd
    (float32, or float64 for an error yardstick).  return_tokens=True also returns the residual stream after
    the last block, [B,257,1024]: (features, tokens)."""
    x = F.conv2d(x, sd["conv1.weight"], bias=None, stride=14)            # [B,1024,16,16]
    b, w = x.shape[0], x.shape[1]
    x = x.reshape(b, w, -1).permute(0, 2, 1)                              # [B,256,1024]
    cls = sd["class_embedding"].to(x.dtype).expand(b, 1, w)
    x = torch.cat([cls, x], dim=1) + sd["positional_embedding"]
    x = F.layer_norm(x, (w,), sd["ln_pre.weight"], sd["ln_pre.bias"], 1e-5)
    n_layers = layers if layers is not None else 1 + max(
        int(k.split(".")[2]) for k in sd if k.startswith("transformer.resblocks."))
    hd = w // HEADS
    for l in range(n_layers):
        p = f"transformer.resblocks.{l}."
        y = F.layer_norm(x, (w,), sd[p + "ln_1.weight"], sd[p + "ln_1.bias"], 1e-5)
        qkv = F.linear(y, sd[p + "attn.in_proj_weight"], sd[p + "attn.in_proj_bias"])
        q, k, v = qkv.split(w, dim=-1)
        q = q.reshape(b, -1, HEADS, hd).transpose(1, 2)
        k = k.reshape(b, -1, HEADS, hd).transpose(1, 2)
        v = v.reshape(b, -1, HEADS, hd).transpose(1, 2)
        att = torch.softmax((q @ k.transpose(-1, -2)) * (hd ** -0.5), dim=-1) @ v
        att = att.transpose(1, 2).reshape(b, -1, w)
        x = x + F.linear(att, sd[p + "attn.out_proj.weight"], sd[p + "attn.out_proj.bias"])
        y = F.layer_norm(x, (w,), sd[p + "ln_2.weight"], sd[p + "ln_2.bias"], 1e-5)
        y = F.gelu(F.linear(y, sd[p + "mlp.c_fc.weight"], sd[p + "mlp.c_fc.bias"]))
        x = x + F.linear(y, sd[p + "mlp.c_proj.weight"], sd[p + "mlp.c_proj.bias"])
    pooled = F.layer_norm(x[:, 0], (w,), sd["ln_post.weight"], sd["ln_post.bias"], 1e-5)
    return (pooled @ sd["proj"], x) if return_tokens else pooled @ sd["proj"]


def score_batch(sd: dict, x: torch.Tensor, tag_embeddings: torch.Tensor | None = None, return_tokens: bool = False):
    """scorer.py:661-671: features -> (embedding, aesthetic in [0,10], raw, tag sims); return_tokens=True adds
    "tokens", the residual stream after the last block [B,257,1024]."""
    with torch.no_grad():
        feats, tokens = encode_image(sd, x, return_tokens=True)
        emb = F.normalize(feats, dim=-1)
        h = F.relu(F.linear(feats, sd["aesthetic_head.0.weight"], sd["aesthetic_head.0.bias"]))
        raw = F.linear(h, sd["aesthetic_head.2.weight"], sd["aesthetic_head.2.bias"]).flatten()
        aesthetic = ((raw + 1) * 5).clamp(0.0, 10.0)
        sims = emb @ tag_embeddings.T if tag_embeddings is not None else None
    out = {"features": feats, "embedding": emb, "aesthetic": aesthetic, "aesthetic_raw": raw, "tag_sims": sims}
    if return_tokens:
        out["tokens"] = tokens
    return out
