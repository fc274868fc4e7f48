"""CPU/torch ORACLE (test infrastructure, NOT product code) for the encoder half of the hot path.

Plain-torch restatement of what the reference executes for a query batch:
  `Contriever.forward` (contriever/src/contriever.py:17-55) = HF `BertModel` (post-LN BERT, add_pooling_layer=False,
  contriever.py:13) -> zero padded positions (:46) -> sum / count mean pooling (:49) or CLS (:51); no L2-normalise
  on the hot path (:29,53).  HF BertModel math as of transformers 5.5.0 (SURVEY.md App. C): embeddings
  word+type+position -> LayerNorm(eps) ; per layer Q,K,V Linear -> softmax(QK^T/sqrt(64) + key mask) V -> Linear +
  residual -> LayerNorm -> Linear -> exact-erf GELU -> Linear + residual -> LayerNorm.

PINNED: unlike the ANN half, the reference's own class imports in the build container, so this restatement is
checked against `contriever.src.contriever.Contriever` itself: `tests/golden/make_encoder_golden.py` runs the
reference class on seeded weights / token batches and commits its outputs (`tests/golden/encoder_*.npz`);
`tests/test_encoder_oracle.py` replays them through this file on CPU.
"""
from __future__ import annotations

import math
from typing import Dict

import torch
import torch.nn.functional as F


def seeded_state_dict(config: dict, seed: int) -> Dict[str, torch.Tensor]:
    """Deterministic (CPU generator) fp32 weights with HF BertModel key names; same recipe as
    retrieval_scaling_b200.encoder.random_state_dict (duplicated here so the oracle does not import the product)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    H, I = config["hidden_size"], config["intermediate_size"]

    def n(*shape, std):
        return torch.randn(*shape, generator=g) * std

    sd = {
        "embeddings.word_embeddings.weight": n(config["vocab_size"], H, std=0.5),
        "embeddings.position_embeddings.weight": n(config["max_position_embeddings"], H, std=0.3),
        "embeddings.token_type_embeddings.weight": n(config["type_vocab_size"], H, std=0.3),
        "embeddings.LayerNorm.weight": 1.0 + n(H, std=0.1),
        "embeddings.LayerNorm.bias": n(H, std=0.1),
    }
    for i in range(config["num_hidden_layers"]):
        p = f"encoder.layer.{i}."
        for nm, (o, k_) in {"attention.self.query": (H, H), "attention.self.key": (H, H), "attention.self.value": (H, H),
                            "attention.output.dense": (H, H), "intermediate.dense": (I, H), "output.dense": (H, I)}.items():
            sd[p + nm + ".weight"] = n(o, k_, std=0.04)
            sd[p + nm + ".bias"] = n(o, std=0.02)
        for nm in ("attention.output.LayerNorm", "output.LayerNorm"):
            sd[p + nm + ".weight"] = 1.0 + n(H, std=0.1)
            sd[p + nm + ".bias"] = n(H, std=0.1)
    return sd


def bert_forward(sd: Dict[str, torch.Tensor], config: dict, input_ids, attention_mask, token_type_ids=None,
                 pooling: str = "average", dtype=torch.float32):
    """Returns [B, hidden] in `dtype` (float32 = exact restatement; float16 on CUDA mirrors `.half()`)."""
    dev = input_ids.device
    w = {k: v.to(device=dev, dtype=dtype) for k, v in sd.items()}
    B, S = input_ids.shape
    H, nh, eps = config["hidden_size"], config["num_attention_heads"], config["layer_norm_eps"]
    hd = H // nh
    if token_type_ids is None:
        token_type_ids = torch.zeros_like(input_ids)
    pos = torch.arange(S, device=dev)
    x = w["embeddings.word_embeddings.weight"][input_ids] + w["embeddings.token_type_embeddings.weight"][token_type_ids] \
        + w["embeddings.position_embeddings.weight"][pos][None]
    x = F.layer_norm(x, (H,), w["embeddings.LayerNorm.weight"], w["embeddings.LayerNorm.bias"], eps)
    mask = attention_mask.bool()
    add_mask = torch.zeros(B, 1, 1, S, device=dev, dtype=dtype).masked_fill(~mask[:, None, None, :], torch.finfo(dtype).min)
    for i in range(config["num_hidden_layers"]):
        p = f"encoder.layer.{i}."
        lin = lambda name, t: F.linear(t, w[p + name + ".weight"], w[p + name + ".bias"])  # noqa: E731
        q = lin("attention.self.query", x).view(B, S, nh, hd).transpose(1, 2)
        k = lin("attention.self.key", x).view(B, S, nh, hd).transpose(1, 2)
        v = lin("attention.self.value", x).view(B, S, nh, hd).transpose(1, 2)
        att = torch.softmax((q @ k.transpose(-1, -2)) / math.sqrt(hd) + add_mask, dim=-1)
        ctx = (att @ v).transpose(1, 2).reshape(B, S, H)
        x = F.layer_norm(lin("attention.output.dense", ctx) + x, (H,), w[p + "attention.output.LayerNorm.weight"],
                         w[p + "attention.output.LayerNorm.bias"], eps)
        ff = F.gelu(lin("intermediate.dense", x))           # exact erf GELU (hidden_act="gelu")
        x = F.layer_norm(lin("output.dense", ff) + x, (H,), w[p + "output.LayerNorm.weight"],
                         w[p + "output.LayerNorm.bias"], eps)
    last = x.masked_fill(~mask[..., None], 0.0)              # contriever.py:46
    if pooling == "average":
        return last.sum(dim=1) / attention_mask.sum(dim=1)[..., None].to(dtype)   # contriever.py:49
    return last[:, 0]                                        # contriever.py:51


# ---- float64 references of the single encoder kernels, computed from the fp16 tensors the kernel receives ----------

def gemm_f64(A, W, bias, residual=None, gelu=False):
    """(A W^T + bias, then erf GELU or + residual) in float64, and |A| |W|^T (the scale of the accumulation error).
    The dense part is returned too: the kernel rounds it to fp16 before it adds the residual."""
    A64, W64 = A.double(), W.double()
    dense = A64 @ W64.T + bias.double()
    absprod = A64.abs() @ W64.abs().T
    if gelu:
        out = 0.5 * dense * (1.0 + torch.erf(dense / math.sqrt(2.0)))
    elif residual is not None:
        out = dense + residual.double()
    else:
        out = dense
    return out, dense, absprod


def attention_f64(qkv, cu_seqlens, heads: int = 12, head_dim: int = 64, scale: float = 0.125):
    """softmax(Q K^T scale) V per (sequence, head) over the un-padded qkv [T, 3 * heads * head_dim] (Q | K | V of each
    token).  Returns ctx [T, heads * head_dim] and sum_j p_j |v_j| [T, heads * head_dim], both float64."""
    H = heads * head_dim
    x = qkv.double()
    T = x.shape[0]
    ctx = torch.zeros((T, H), dtype=torch.float64, device=x.device)
    pv_abs = torch.zeros_like(ctx)
    cu = [int(c) for c in cu_seqlens]
    lens = [cu[i + 1] - cu[i] for i in range(len(cu) - 1)]
    # sequences of equal length are batched together
    for S in sorted(set(lens)):
        if S == 0:
            continue
        starts = torch.tensor([cu[i] for i, n in enumerate(lens) if n == S], device=x.device)
        rows = (starts[:, None] + torch.arange(S, device=x.device)[None]).reshape(-1)
        blk = x[rows].view(-1, S, 3, heads, head_dim).permute(2, 0, 3, 1, 4)   # [3, nseq, heads, S, hd]
        q, k, v = blk[0], blk[1], blk[2]
        p = torch.softmax((q @ k.transpose(-1, -2)) * scale, dim=-1)
        ctx[rows] = (p @ v).permute(0, 2, 1, 3).reshape(-1, H)
        pv_abs[rows] = (p @ v.abs()).permute(0, 2, 1, 3).reshape(-1, H)
    return ctx, pv_abs


def layernorm_f64(x, gamma, beta, eps: float):
    """Row LayerNorm (biased variance) in float64.  Returns the output, 1 / sqrt(var + eps) and mean |x| per row."""
    x64 = x.double()
    mean = x64.mean(dim=1, keepdim=True)
    var = ((x64 - mean) ** 2).mean(dim=1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    out = (x64 - mean) * rstd * gamma.double() + beta.double()
    return out, rstd, x64.abs().mean(dim=1, keepdim=True)
