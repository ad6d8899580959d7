"""SumGAN with attention (models/sumgan_att.py:20-420).  The selector's inference (eval mode, no autograd graph being
built) runs on the sm_100a kernels of libsummarizer_b200.so (smz_sumgan_att_selector_forward: tcgen05 GEMMs and the
fused variable-length attention of smz_attn.cu, heads 256 wide at the default 4 heads, 128 wide at 8) for 1024-d input,
4 or 8 heads and at least one layer.  Training forwards, forwards that build an autograd graph and other head counts run
the torch modules exactly as the reference does; the encoder-decoder autoencoder stays a plain ``torch.nn`` transformer
(outside the hot path, SURVEY.md §2.1).  The discriminator is the same ``GAN`` / ``cLSTM`` as SumGAN and therefore runs
on this library's recurrence kernels.
Class names, constructor arguments and attribute / state-dict names follow the reference so checkpoints interchange.
The trainer reuses SumGANTrainer's phase machinery (per-phase Adam, clip over ALL parameters, data-parallel
all-reduce) with the Wasserstein losses and the autoencoder pre-training of sumgan_att.py:171-230; it scores all test
videos in one packed native call."""
import ctypes as C

import torch
import torch.nn as nn

from .. import _native as N
from ._packed import NativeModule, Workspace, packed_input, score_sequences, workspace_bytes
from .sumgan import GAN, SumGANTrainer
from .transformer import encoder_copies, encoder_params, f32, layer_table


class SelectorParams(C.Structure):
    """struct smz_sumgan_att_selector_params (include/summarizer_b200.h)."""
    _fields_ = [("layers", C.c_void_p), ("n_heads", C.c_int32), ("ln_g", C.c_void_p), ("ln_b", C.c_void_p),
                ("eps", C.c_float), ("out_w", C.c_void_p), ("out_b", C.c_void_p)]


class Transformer(NativeModule):
    """Selector: transformer encoder + Linear/Sigmoid per frame (sumgan_att.py:20-46)."""

    def __init__(self, input_size=1024, encoder_layers=4, attention_heads=8, epsilon=1e-5):
        super().__init__()
        self.input_size = input_size
        self.attention_heads = attention_heads
        self.layer_norm = nn.LayerNorm(input_size, epsilon)
        self.transformer_encoder_layer = nn.TransformerEncoderLayer(d_model=input_size, nhead=attention_heads,
                                                                    dim_feedforward=input_size)
        self.transformer_encoder = nn.TransformerEncoder(self.transformer_encoder_layer, num_layers=encoder_layers,
                                                         norm=self.layer_norm)
        self.out = nn.Sequential(nn.Linear(input_size, 1), nn.Sigmoid())
        self._ws = Workspace()

    def native_covered(self):
        """True when the sm_100a kernels implement this configuration (1024-d input, 4 heads of width 256 or 8 of width
        128, at least one layer).  Selected on the observable configuration; other configurations run the torch modules."""
        return self.input_size == 1024 and self.attention_heads in (4, 8) and len(self.transformer_encoder.layers) >= 1

    def _weights(self):
        """The parameter struct over the kernels' weight copies (cached in ``self._cache``)."""
        layers = list(self.transformer_encoder.layers)
        lin = self.out[0]
        ps = encoder_params(layers) + [self.layer_norm.weight, self.layer_norm.bias, lin.weight, lin.bias]
        sh = self._cache.get(ps, lambda: dict(layers=encoder_copies(layers), ln_g=f32(self.layer_norm.weight),
                                              ln_b=f32(self.layer_norm.bias), out_w=f32(lin.weight).reshape(-1),
                                              out_b=f32(lin.bias)),
                             config=(float(self.layer_norm.eps),))
        arr = layer_table(sh["layers"])
        st = SelectorParams(C.addressof(arr), int(self.attention_heads), sh["ln_g"].data_ptr(), sh["ln_b"].data_ptr(),
                            float(self.layer_norm.eps), sh["out_w"].data_ptr(), sh["out_b"].data_ptr())
        return st, arr

    def score_packed(self, x, lengths):
        """Inference over a ragged batch: ``x`` packed [sum T, 1024] (float32 or bfloat16, device), ``lengths`` the
        per-video frame counts.  Returns float32 scores [sum T]; every video attends only to its own frames."""
        if not self.native_covered():
            raise N.NativeError("score_packed: the sm_100a kernels cover 1024-d input with 4 or 8 attention heads only")
        x, cu, is_bf16 = packed_input(x, lengths, self.input_size)
        st, arr = self._weights()           # arr: the layer table st points at, alive for the call
        cu_p = cu.ctypes.data_as(C.c_void_p)
        ws = self._ws.get(workspace_bytes(N.lib().smz_transformer_workspace_bytes, cu_p, len(lengths), is_bf16), x.device)
        scores = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
        N.check(N.lib().smz_sumgan_att_selector_forward(N.ptr(x), is_bf16, cu_p, len(lengths), C.byref(st),
                                                        len(self.transformer_encoder.layers), N.ptr(scores), N.ptr(ws),
                                                        ws.numel(), N.current_stream()))
        return scores

    def forward(self, x):
        """x: (seq_len, batch_size, input_size) -> scores: (seq_len, batch_size, 1)"""
        if self.training:
            self._cache.clear()              # an optimizer step may follow: the weight copies must be rebuilt
        builds_graph = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters()))
        if x.is_cuda and not self.training and not builds_graph and self.native_covered():
            return score_sequences(self.score_packed, x)
        return self.out(self.transformer_encoder(x))


class AutoencoderTransformer(nn.Module):
    """Encoder-decoder transformer reconstructing its (score-weighted) input (sumgan_att.py:48-80)."""

    def __init__(self, input_size=1024, encoder_layers=4, attention_heads=8, epsilon=1e-5):
        super().__init__()
        self.input_size = input_size
        self.transformer_encoder_layer = nn.TransformerEncoderLayer(d_model=input_size, nhead=attention_heads,
                                                                    dim_feedforward=input_size)
        self.transformer_encoder = nn.TransformerEncoder(self.transformer_encoder_layer, num_layers=encoder_layers)
        self.transformer_decoder_layer = nn.TransformerDecoderLayer(d_model=input_size, nhead=attention_heads,
                                                                    dim_feedforward=input_size)
        self.transformer_decoder = nn.TransformerDecoder(self.transformer_decoder_layer, num_layers=encoder_layers)

    def forward(self, x):
        """x: (seq_len, batch_size, input_size) -> x_hat of the same shape (the decoder attends to the encoded x)"""
        return self.transformer_decoder(x, self.transformer_encoder(x))


class Summarizer(nn.Module):
    def __init__(self, input_size=1024, s_encoder_layers=2, s_attention_heads=4, ae_encoder_layers=2, ae_attention_heads=4):
        """Summarizer: Selector (Transformer) + Autoencoder Transformer."""
        super().__init__()
        self.selector = Transformer(input_size=input_size, encoder_layers=s_encoder_layers, attention_heads=s_attention_heads)
        self.ae = AutoencoderTransformer(input_size=input_size, encoder_layers=ae_encoder_layers,
                                         attention_heads=ae_attention_heads)

    def forward(self, x, uniform=False, p=0.3):
        """x: (seq_len, B, input_size) -> (x_hat (seq_len, B, input_size), scores (seq_len, B, 1))"""
        if uniform:
            scores = torch.rand((x.shape[0], x.shape[1], 1)).to(x.device)
        else:
            scores = self.selector(x)
        return self.ae(x * scores), scores


class SumGANAtt(nn.Module):
    def __init__(self, input_size=1024, s_encoder_layers=2, s_attention_heads=4, ae_encoder_layers=2, ae_attention_heads=4,
                 cLSTM_hidden_size=1024, cLSTM_num_layers=2):
        """SumGAN: Summarizer + GAN"""
        super().__init__()
        self.summarizer = Summarizer(input_size=input_size, s_encoder_layers=s_encoder_layers,
                                     s_attention_heads=s_attention_heads, ae_encoder_layers=ae_encoder_layers,
                                     ae_attention_heads=ae_attention_heads)
        self.gan = GAN(input_size=input_size, hidden_size=cLSTM_hidden_size, num_layers=cLSTM_num_layers)

    def forward(self, x):
        """x: (seq_len, B, input_size) -> scores: (seq_len, B, 1)"""
        return self.summarizer.selector(x)


class SumGANAttTrainer(SumGANTrainer):
    def _init_model(self):
        ep = self.hps.extra_params or {}
        self.input_size = int(ep.get("input_size", 1024))
        self.s_encoder_layers = int(ep.get("s_encoder_layers", 2))
        self.s_attention_heads = int(ep.get("s_attention_heads", 4))
        self.ae_encoder_layers = int(ep.get("ae_encoder_layers", 2))
        self.ae_attention_heads = int(ep.get("ae_attention_heads", 4))
        self.cLSTM_hidden_size = int(ep.get("cLSTM_hidden_size", 256))
        self.cLSTM_num_layers = int(ep.get("cLSTM_num_layers", 2))
        self.sup = bool(ep.get("sup", True))
        self.pretrain_ae = int(ep.get("pretrain_ae", 80))
        self.epoch_noise = int(ep.get("epoch_noise", 0.2 * self.hps.epochs))
        model = SumGANAtt(input_size=self.input_size, s_encoder_layers=self.s_encoder_layers,
                          s_attention_heads=self.s_attention_heads, ae_encoder_layers=self.ae_encoder_layers,
                          ae_attention_heads=self.ae_attention_heads, cLSTM_hidden_size=self.cLSTM_hidden_size,
                          cLSTM_num_layers=self.cLSTM_num_layers)
        self.log.debug("Generator params: {}".format(sum([_.numel() for _ in model.summarizer.parameters()])))
        self.log.debug("Discriminator params: {}".format(sum([_.numel() for _ in model.gan.parameters()])))
        return model

    def _packed_scorer(self):
        sel = self.model.summarizer.selector
        return sel if sel.native_covered() and self.hps.use_cuda else None

    # ---- losses (sumgan_att.py:171-193) ----------------------------------------------------------------------
    def loss_ae(self, x, x_hat):
        """minimize E[l2_norm(x - x_hat)]"""
        return torch.norm(x - x_hat, p=2)

    def loss_sparsity(self, scores, sigma=None):
        """upstream leaves the unsupervised sparsity term as a constant 0"""
        return torch.tensor(0)

    def loss_gan_generator(self, probs_fake, probs_uniform):
        """maximize 0.5 * (cLSTM(x_hat) + cLSTM(x_hat_p))"""
        return torch.mean(-0.5 * (probs_fake + probs_uniform))

    def loss_gan_discriminator(self, probs_real, probs_fake, probs_uniform):
        """maximize cLSTM(x) - 0.5 * (cLSTM(x_hat) + cLSTM(x_hat_p))"""
        return torch.mean(-probs_real + 0.5 * (probs_fake + probs_uniform))

    # ---- phases ------------------------------------------------------------------------------------------------
    def _pretrain_epochs(self):
        return self.pretrain_ae

    def pretrain(self, fold):
        """Pretrain autoencoder before learning the GAN (sumgan_att.py:195-230; learning rate x 10)"""
        train_keys, _ = self._get_train_test_keys(fold)
        ae = self.model.summarizer.ae
        opt = torch.optim.Adam(ae.parameters(), lr=self.hps.lr * 10.0, weight_decay=self.hps.weight_decay)
        dp, rank, world = self._dp()
        for epoch in range(self.pretrain_ae):
            losses = []
            for key, n_active in self._groups(train_keys, dp, rank, world):
                loss = None
                if key is not None:
                    x, _ = self._video_tensors(key)
                    loss = self.loss_ae(x, ae(x))
                    losses.append(loss.detach())
                self._update(opt, loss, dp, n_active)
            if epoch % 10 == 0 or epoch == self.pretrain_ae - 1:
                avg = float(torch.stack(losses).mean()) if losses else float("nan")
                self.log.info(f"Pretrain: {epoch+1:3}/{self.pretrain_ae:3}   Lae: {avg:.05f}")

    def _make_optimizers(self):
        s = self.model.summarizer
        self.s_e_optimizer = self._adam(list(s.selector.parameters()) + list(s.ae.transformer_encoder.parameters())
                                        + list(s.ae.transformer_encoder_layer.parameters()))
        self.d_optimizer = self._adam(list(s.ae.transformer_decoder.parameters())
                                      + list(s.ae.transformer_decoder_layer.parameters()))
        self.c_optimizer = self._adam(self.model.gan.c_lstm.parameters())

    def train_step(self, x, y, epoch, dp=None, n_active=1):
        """The three updates of one video (sumgan_att.py:289-351); None on an idle data-parallel replica."""
        m, idle = self.model, x is None
        loss_s_e = loss_d = loss_c = None
        if not idle:                                             # selector + encoder
            x_hat, scores = m.summarizer(x)
            _, h = m.gan(torch.cat([x, x_hat], 1))
            sparsity = self.loss_sparsity_sup(scores, y) if self.sup else self.loss_sparsity(scores)
            loss_s_e = self.loss_recons(h[0:1], h[1:2]) + sparsity
        self._update(self.s_e_optimizer, loss_s_e, dp, n_active)
        if not idle:                                             # decoder
            x_hat, _ = m.summarizer(x)
            x_hat_p, _ = m.summarizer(x, uniform=True)
            probs, h = m.gan(torch.cat([x, x_hat, x_hat_p], 1))
            loss_d = self.loss_recons(h[0:1], h[1:2]) + self.loss_gan_generator(probs[1:2], probs[2:3])
        self._update(self.d_optimizer, loss_d, dp, n_active)
        if not idle:                                             # discriminator
            x_hat, scores = m.summarizer(x)
            x_hat_p, _ = m.summarizer(x, uniform=True)
            x_in = x
            if epoch < self.epoch_noise:
                x_in = torch.randn_like(x) * x
                x_hat = x_hat * torch.randn_like(x_hat)
                x_hat_p = x_hat_p * torch.randn_like(x_hat_p)
            probs, _ = m.gan(torch.cat([x_in, x_hat, x_hat_p], 1))
            probs_real, probs_fake, probs_uniform = probs[0:1], probs[1:2], probs[2:3]
            loss_c = self.loss_gan_discriminator(probs_real, probs_fake, probs_uniform)
        self._update(self.c_optimizer, loss_c, dp, n_active)
        if idle:
            return None
        return dict(Lse=loss_s_e.detach(), Ld=loss_d.detach(), Lc=loss_c.detach(), D_x=probs_real.detach().mean(),
                    D_x_hat=probs_fake.detach().mean(), D_x_hat_p=probs_uniform.detach().mean(), scores=scores.detach())


if __name__ == "__main__":
    model = SumGANAtt()
    print("Trainable parameters in model:", sum(p.numel() for p in model.parameters() if p.requires_grad))
