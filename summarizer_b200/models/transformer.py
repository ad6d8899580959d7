"""Transformer-encoder scorer (models/transformer.py:19-96): the reference's class, constructor arguments, attribute /
state-dict names (``transformer_encoder_layer``, ``transformer_encoder``, the ONE ``layer_norm`` shared by the encoder's
final norm and the regressor head, ``k1``, ``k2``, optional ``pos_embed``) and forward contract (T, B, 1024) -> (T, B, 1),
so reference checkpoints load.

Inference (eval mode, no autograd graph being built) runs on the sm_100a kernels of libsummarizer_b200.so
(smz_transformer_forward: tcgen05 GEMMs and the fused variable-length attention of smz_attn.cu) for the configurations
they cover: 1024-d input, 8 heads of 128, any number of layers, both positional embeddings, ``more_residuals``, any
``epsilon`` / ``weight_init``.  Training forwards, forwards that build an autograd graph and other head counts run the
torch modules exactly as the reference does.  The trainer is the shared supervised loop (transformer.py:113-190 is the
VASNet loop with another module)."""
import ctypes as C

import torch
import torch.nn as nn

from .. import _native as N
from . import Trainer
from ._packed import NativeModule, Workspace, packed_input, score_sequences, workspace_bytes


class TransformerLayerParams(C.Structure):
    """struct smz_transformer_layer (include/summarizer_b200.h)."""
    _fields_ = [(k, C.c_void_p) for k in ("w_qkv", "b_qkv", "w_out", "b_out", "w1", "b1", "w2", "b2",
                                          "norm1_g", "norm1_b", "norm2_g", "norm2_b")]


class TransformerParams(C.Structure):
    """struct smz_transformer_params (include/summarizer_b200.h)."""
    _fields_ = [("layers", C.c_void_p), ("ln_g", C.c_void_p), ("ln_b", C.c_void_p), ("eps", C.c_float),
                ("more_residuals", C.c_int32), ("k1_w", C.c_void_p), ("k1_b", C.c_void_p), ("head_gw", C.c_void_p),
                ("head_c", C.c_void_p)]


def encoder_params(layers):
    """The parameters of nn.TransformerEncoderLayer modules in smz_transformer_layer order, flat (a weight cache's key)."""
    return [t for L in layers for t in (L.self_attn.in_proj_weight, L.self_attn.in_proj_bias, L.self_attn.out_proj.weight,
                                        L.self_attn.out_proj.bias, L.linear1.weight, L.linear1.bias, L.linear2.weight,
                                        L.linear2.bias, L.norm1.weight, L.norm1.bias, L.norm2.weight, L.norm2.bias)]


def f32(t):
    return t.detach().float().contiguous()


def b16(t):
    return t.detach().to(torch.bfloat16).contiguous()


def encoder_copies(layers):
    """Per layer, the smz_transformer_layer tensors: bfloat16 copies of the matrices, float32 vectors."""
    return [(b16(L.self_attn.in_proj_weight), f32(L.self_attn.in_proj_bias), b16(L.self_attn.out_proj.weight),
             f32(L.self_attn.out_proj.bias), b16(L.linear1.weight), f32(L.linear1.bias), b16(L.linear2.weight),
             f32(L.linear2.bias), f32(L.norm1.weight), f32(L.norm1.bias), f32(L.norm2.weight), f32(L.norm2.bias))
            for L in layers]


def layer_table(copies):
    """The host array of smz_transformer_layer structs over encoder_copies(...); keep it alive for the call.  It is
    rebuilt per call (plain tensors in the cache keep the module deep-copyable)."""
    return (TransformerLayerParams * len(copies))(*(TransformerLayerParams(*(t.data_ptr() for t in ts)) for ts in copies))


def sincos_table(max_length, width):
    """The fixed table of transformer.py:34-38: column i (even) sin(pos / 10000^(2i/width)), column i+1
    cos(pos / 10000^(2(i+1)/width)) — evaluated in float64 and rounded once, like the reference's numpy scalars."""
    pos = torch.arange(max_length, dtype=torch.float64).unsqueeze(1)
    i = torch.arange(0, width, 2, dtype=torch.float64).unsqueeze(0)
    table = torch.zeros(max_length, width)
    table[:, 0::2] = torch.sin(pos / torch.pow(torch.tensor(10000.0, dtype=torch.float64), 2 * i / width)).float()
    table[:, 1::2] = torch.cos(pos / torch.pow(torch.tensor(10000.0, dtype=torch.float64), 2 * (i + 1) / width)).float()
    return table


class Transformer(NativeModule):
    def __init__(self, input_size=1024, encoder_layers=6, attention_heads=8, more_residuals=False, max_length=None,
                 pos_embed="simple", epsilon=1e-5, weight_init=None):
        super().__init__()
        self.input_size = input_size
        self.attention_heads = attention_heads
        self.epsilon = epsilon
        self.max_length = max_length
        if self.max_length:
            self.pos_embed_type = pos_embed
            if pos_embed == "simple":
                self.pos_embed = nn.Embedding(self.max_length, input_size)
            elif pos_embed == "attention":
                self.pos_embed = sincos_table(self.max_length, input_size)     # plain tensor, not a buffer (as upstream)
            else:
                self.max_length = None
        self.more_residuals = more_residuals
        self.dropout = nn.Dropout(0.5)
        self.layer_norm = nn.LayerNorm(input_size, epsilon)
        self.transformer_encoder_layer = nn.TransformerEncoderLayer(d_model=input_size, nhead=attention_heads,
                                                                    dim_feedforward=input_size, dropout=0.1, activation="relu")
        self.transformer_encoder = nn.TransformerEncoder(self.transformer_encoder_layer, num_layers=encoder_layers,
                                                         norm=self.layer_norm)
        self.k1 = nn.Linear(input_size, input_size)
        self.k2 = nn.Linear(input_size, 1)
        self.sigmoid = nn.Sigmoid()
        self.relu = nn.ReLU()
        init = {"he": nn.init.kaiming_uniform_, "kaiming": nn.init.kaiming_uniform_,
                "xavier": nn.init.xavier_uniform_}.get(weight_init.lower()) if weight_init else None
        if init is not None:                                  # transformer.py:57-70: feed-forward + head matrices only
            for layer in self.transformer_encoder.layers:
                init(layer.linear1.weight)
                init(layer.linear2.weight)
            init(self.k1.weight)
            init(self.k2.weight)
        self._ws = Workspace()

    def native_covered(self):
        """True when the sm_100a kernels implement this configuration (1024-d input, 8 heads of width 128, at least one
        layer).  Selected on the observable configuration; other configurations run the torch modules."""
        return self.input_size == 1024 and self.attention_heads == 8 and len(self.transformer_encoder.layers) >= 1

    def _weights(self):
        """The parameter structs over the kernels' weight copies (``_build_weights``, cached in ``self._cache``).  Only
        ``transformer_encoder.layers.*`` run: the top-level ``transformer_encoder_layer`` is a template the encoder
        deep-copied and is never read."""
        layers = list(self.transformer_encoder.layers)
        ps = encoder_params(layers)
        ps += [self.layer_norm.weight, self.layer_norm.bias, self.k1.weight, self.k1.bias, self.k2.weight, self.k2.bias]
        sh = self._cache.get(ps, lambda: self._build_weights(layers), config=(bool(self.more_residuals), float(self.epsilon)))
        arr = layer_table(sh["layers"])
        st = TransformerParams(C.addressof(arr), sh["ln_g"].data_ptr(), sh["ln_b"].data_ptr(), float(self.epsilon),
                               int(bool(self.more_residuals)), sh["k1_w"].data_ptr(), sh["k1_b"].data_ptr(),
                               sh["head_gw"].data_ptr(), sh["head_c"].data_ptr())
        return st, arr

    def _build_weights(self, layers):
        """bfloat16 copies of the encoder / k1 matrices, float32 vectors and the folded regressor head."""
        per_layer = encoder_copies(layers)
        ln_g, ln_b = f32(self.layer_norm.weight), f32(self.layer_norm.bias)
        w2, b2 = f32(self.k2.weight).reshape(-1), f32(self.k2.bias)
        head_gw = (ln_g * w2).contiguous()
        head_c = torch.stack([head_gw.sum(), (ln_b * w2).sum() + b2[0]]).contiguous()
        return dict(layers=per_layer, ln_g=ln_g, ln_b=ln_b, k1_w=b16(self.k1.weight), k1_b=f32(self.k1.bias),
                    head_gw=head_gw, head_c=head_c)

    def score_packed(self, x, lengths):
        """Inference over a ragged batch: ``x`` packed [sum T, 1024] (float32 or bfloat16, device, positional embeddings
        already added), ``lengths`` the per-video frame counts.  Returns float32 scores [sum T]; every video attends
        only to its own frames."""
        if not self.native_covered():
            raise N.NativeError("score_packed: the sm_100a kernels cover 1024-d input with 8 attention heads only")
        x, cu, is_bf16 = packed_input(x, lengths, self.input_size)
        st, arr = self._weights()           # arr: the layer table st points at, alive for the call
        cu_p = cu.ctypes.data_as(C.c_void_p)
        ws = self._ws.get(workspace_bytes(N.lib().smz_transformer_workspace_bytes, cu_p, len(lengths), is_bf16), x.device)
        scores = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
        N.check(N.lib().smz_transformer_forward(N.ptr(x), is_bf16, cu_p, len(lengths), C.byref(st),
                                                len(self.transformer_encoder.layers), N.ptr(scores), N.ptr(ws), ws.numel(),
                                                N.current_stream()))
        return scores

    def forward(self, x):
        """x: (seq_len, batch_size, input_size) -> y: (seq_len, batch_size, 1)"""
        seq_len, batch_size, _ = x.shape
        if self.training:
            self._cache.clear()              # an optimizer step may follow: the weight copies must be rebuilt
        if self.max_length is not None:
            assert self.max_length >= seq_len, "input sequence has higher length than max_length"
            if self.pos_embed_type == "simple":
                pe = self.pos_embed(torch.arange(seq_len, device=x.device))
            else:
                pe = self.pos_embed[:seq_len].to(x.device)
            x += pe.unsqueeze(1)                              # in place on the caller's tensor, as upstream (:84,:86)
        builds_graph = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters()))
        if x.is_cuda and not self.training and not builds_graph and self.native_covered():
            return score_sequences(self.score_packed, x)
        encoder_out = self.transformer_encoder(x)
        if self.more_residuals:
            encoder_out = encoder_out + x
        y = self.layer_norm(self.dropout(self.relu(self.k1(encoder_out))))
        return self.sigmoid(self.k2(y))


class TransformerTrainer(Trainer):
    def _init_model(self):
        ep = self.hps.extra_params or {}
        return Transformer(encoder_layers=int(ep.get("encoder_layers", 6)), attention_heads=int(ep.get("attention_heads", 8)),
                           more_residuals=ep.get("more_residuals", False),
                           max_length=int(ep["max_pos"]) if "max_pos" in ep else None,
                           pos_embed=ep.get("pos_embed", "simple"), epsilon=float(ep.get("epsilon", 1e-5)),
                           weight_init=ep.get("weight_init", None))

    def _packed_scorer(self):
        m = self.model
        return m if m.max_length is None and m.native_covered() and self.hps.use_cuda else None

    def train(self, fold):
        return self._train_supervised(fold)


if __name__ == "__main__":
    model = Transformer()
    print("Trainable parameters in model:", sum(p.numel() for p in model.parameters() if p.requires_grad))
    y = model(torch.randn(10, 3, 1024))
    assert y.shape == (10, 3, 1)
