"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Float64 restatement of Transformer scorer inference (summarizer_b200/models/transformer.py in eval mode) as explicit
operations on a packed batch, on whatever device its input is on:

  attention       softmax(q k^T / sqrt(d)) v per video and head, in query blocks, so that a 33 000-frame video needs
                  a few hundred MB of logits at a time rather than the 70 GB of torch's MultiheadAttention weights
  encoder_layer   post-norm nn.TransformerEncoderLayer (relu; dropout is off in eval): in_proj, attention, out_proj
                  + residual, norm1, linear1 + relu, linear2 + residual, norm2
  scores          the encoder layers, the encoder's final norm (the model's shared ``layer_norm``), + the encoder input
                  when ``more_residuals``, then k1, relu, the shared norm again, k2 and sigmoid

Parameters are the module's own (float32) tensors, widened to float64 as they are used.  Pinned by
tests/test_transformer_plan_gpu.py against ``copy.deepcopy(m).double().eval()`` (torch's own TransformerEncoder).
"""
import math

import torch
import torch.nn.functional as F

BLOCK_BYTES = 256 << 20     # logits of one query block, all heads of one video


def attention(qkv, lengths, n_heads, head_dim=128):
    """qkv: packed rows [sum T, >= 3 * n_heads * head_dim], Q | K | V column blocks, head h at h * head_dim inside each
    -> [sum T, n_heads * head_dim], head h at column h * head_dim, in the dtype and on the device of qkv."""
    w = n_heads * head_dim
    out = qkv.new_empty(qkv.shape[0], w)
    r0 = 0
    for T in lengths:
        q, k, v = (qkv[r0:r0 + T, i * w:(i + 1) * w].reshape(T, n_heads, head_dim).transpose(0, 1) for i in range(3))
        kt = k.transpose(1, 2) / math.sqrt(head_dim)
        step = max(1, BLOCK_BYTES // (n_heads * T * qkv.element_size()))
        for b in range(0, T, step):
            p = torch.softmax(q[:, b:b + step] @ kt, dim=-1)
            out[r0 + b:r0 + min(b + step, T)] = (p @ v).transpose(0, 1).reshape(-1, w)
        r0 += T
    return out


def _layer_norm(x, norm):
    return F.layer_norm(x, x.shape[-1:], norm.weight.detach().to(x), norm.bias.detach().to(x), norm.eps)


def _linear(x, lin):
    return x @ lin.weight.detach().to(x).t() + lin.bias.detach().to(x)


def encoder_layer(L, x, lengths, n_heads):
    """One nn.TransformerEncoderLayer L (norm_first=False, relu) in eval mode on packed rows x."""
    at = L.self_attn
    qkv = x @ at.in_proj_weight.detach().to(x).t() + at.in_proj_bias.detach().to(x)
    a = attention(qkv, lengths, n_heads, x.shape[1] // n_heads)
    del qkv
    x = _layer_norm(x + _linear(a, at.out_proj), L.norm1)
    return _layer_norm(x + _linear(torch.relu(_linear(x, L.linear1)), L.linear2), L.norm2)


def scores(m, x, lengths):
    """Scores of a Transformer module m for packed rows x [sum T, 1024] (positional embeddings already added, as
    ``score_packed`` takes them) -> float64 [sum T] on x's device."""
    x = x.to(torch.float64)
    h = x
    for L in m.transformer_encoder.layers:
        h = encoder_layer(L, h, lengths, m.attention_heads)
    e = _layer_norm(h, m.layer_norm)
    if m.more_residuals:
        e = e + x
    y = _layer_norm(torch.relu(_linear(e, m.k1)), m.layer_norm)
    return torch.sigmoid(_linear(y, m.k2)).reshape(-1)
