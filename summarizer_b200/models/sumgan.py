"""SumGAN — "Unsupervised Video Summarization with Adversarial LSTM Networks" — with the reference's classes,
constructor arguments, parameter names and forward contracts (models/sumgan.py:23-258) and its three-phase
adversarial trainer (sumgan.py:261-533), computed by the sm_100a LSTM kernels (csrc/smz_lstm.cu) and the tcgen05
GEMM instead of cuDNN / cuBLAS.

Every ``nn.LSTM`` / ``nn.Linear`` below only OWNS parameters (state-dict keys ``summarizer.s_lstm.lstm.*``,
``summarizer.vae.e_lstm.{lstm,mu,logvar}.*``, ``summarizer.vae.d_lstm.{lstm,recons}.*``, ``gan.c_lstm.{lstm,out.0}.*``
and the initialisation stream are the reference's); none of them is executed.  Hidden sizes the kernels implement:
1024 (uni- or bidirectional) and 2048 (unidirectional) — the shipped defaults.  There is no CPU fallback."""
import random

import numpy as np
import torch
import torch.nn as nn

from .. import _native as N
from ..dense import linear
from ._packed import NativeModule
from .lstm_stack import lstm_decode, lstm_stack


class NoiseSource:
    """Where the trainer's random tensors come from (sumgan.py:134 reparameterisation noise, :177 uniform scores,
    :466-468 discriminator input noise).  Default: torch's generator of the tensor's device.  ``begin(phase)`` is
    called at the start of every phase ("pretrain", "p1" selector/encoder, "p2" decoder, "p3" discriminator) and
    ``role`` names the draw inside it ("eps" / "eps_p": VAE noise of x_hat / x_hat_p, "uniform", "noise_x",
    "noise_x_hat", "noise_x_hat_p"), so that tests can replay the reference's draws one for one."""

    def begin(self, phase):
        pass

    def randn_like(self, t, role):
        return torch.randn_like(t)

    def rand_like(self, t, role):
        return torch.rand_like(t)


noise = NoiseSource()


def _require_cuda(x, what):
    if not x.is_cuda:
        raise N.NativeError(f"summarizer_b200.{what} runs on a CUDA (sm_100a) device only; move the input with .cuda()")


def _head1(x, lin):
    """Linear(in, 1) on rows of x: a dot product per row (elementwise multiply + row sum)."""
    return (x * lin.weight.reshape(1, -1)).sum(-1, keepdim=True) + lin.bias


class sLSTM(NativeModule):
    def __init__(self, input_size=1024, hidden_size=1024, num_layers=2):
        """Selector LSTM"""
        super().__init__()
        self.lstm = nn.LSTM(input_size=input_size, hidden_size=hidden_size, num_layers=num_layers, bidirectional=True)
        self.out = nn.Linear(hidden_size * 2, 1)
        self.sig = nn.Sigmoid()

    def forward(self, x):
        """x: (seq_len, batch_size, input_size) -> scores: (seq_len, batch_size, 1)"""
        _require_cuda(x, "sLSTM")
        y, _, _ = lstm_stack(self._cache, self.lstm, x.transpose(0, 1))          # [B,T,2H], sequences share each launch
        return torch.sigmoid(_head1(y, self.out)).transpose(0, 1)


class eLSTM(NativeModule):
    def __init__(self, input_size=1024, hidden_size=2048, num_layers=2):
        """Encoder LSTM"""
        super().__init__()
        self.lstm = nn.LSTM(input_size=input_size, hidden_size=hidden_size, num_layers=num_layers, bidirectional=False)
        self.mu = nn.Linear(hidden_size, hidden_size)
        self.logvar = nn.Linear(hidden_size, hidden_size)

    def forward(self, x):
        """x: (seq_len, batch_size, input_size) -> (h_mu, h_logvar), c_last: each (num_layers, batch_size, hidden_size)"""
        _require_cuda(x, "eLSTM")
        _, h_last, c_last = lstm_stack(self._cache, self.lstm, x.transpose(0, 1))  # [L,B,H]
        L, B, H = h_last.shape
        flat = h_last.reshape(L * B, H)
        h_mu = linear(flat, self.mu.weight, self.mu.bias).reshape(L, B, H)
        h_logvar = linear(flat, self.logvar.weight, self.logvar.bias).reshape(L, B, H)
        return (h_mu, h_logvar), c_last


class dLSTM(NativeModule):
    def __init__(self, input_size=1024, hidden_size=2048, num_layers=2):
        """Decoder LSTM"""
        super().__init__()
        self.lstm = nn.LSTM(input_size=hidden_size, hidden_size=hidden_size, num_layers=num_layers, bidirectional=False)
        self.recons = nn.Linear(hidden_size, input_size)

    def forward_step(self, x_prev, h_prev, c_prev):
        """Decode one sequence step: x_prev (1, B, H), h_prev/c_prev (num_layers, B, H) -> x_next, (h_next, c_next)."""
        _require_cuda(x_prev, "dLSTM")
        y, h_n, c_n = lstm_stack(self._cache, self.lstm, x_prev.transpose(0, 1), h_prev, c_prev)
        return y.transpose(0, 1), (h_n, c_n)

    def forward(self, seq_len, h_0, c_0):
        """Decode entire sequence: h_0, c_0 (num_layers, B, H) -> x_hat (seq_len, B, input_size), time-reversed."""
        _require_cuda(h_0, "dLSTM")
        top = lstm_decode(self._cache, self.lstm, int(seq_len), h_0, c_0)         # [B,T,H]: the whole loop of :110-112
        B, T, H = top.shape
        x_hat = linear(top.reshape(B * T, H), self.recons.weight, self.recons.bias).reshape(B, T, -1).transpose(0, 1)
        return torch.flip(x_hat, (0,))


class VAE(nn.Module):
    def __init__(self, input_size=1024, hidden_size=2048, num_layers=2):
        """Variational Auto Encoder LSTM"""
        super().__init__()
        self.e_lstm = eLSTM(input_size=input_size, hidden_size=hidden_size, num_layers=num_layers)
        self.d_lstm = dLSTM(input_size=input_size, hidden_size=hidden_size, num_layers=num_layers)

    def reparameterize(self, mu, logvar, roles=None):
        std = torch.exp(0.5 * logvar)
        if roles is None:
            eps = noise.randn_like(std, "eps")
        else:       # sequences batched along dim 1 draw their noise separately, in the reference's order
            eps = torch.cat([noise.randn_like(std[:, b:b + 1], r) for b, r in enumerate(roles)], 1)
        return mu + eps * std

    def forward(self, x, roles=None):
        """x: (seq_len, B, input_size) -> x_hat (seq_len, B, input_size), (h_mu, h_logvar)"""
        (h_mu, h_logvar), c = self.e_lstm(x)
        h = self.reparameterize(h_mu, h_logvar, roles)
        x_hat = self.d_lstm(x.size(0), h, c)
        return x_hat, (h_mu, h_logvar)


class Summarizer(nn.Module):
    def __init__(self, input_size=1024, sLSTM_hidden_size=1024, sLSTM_num_layers=2, edLSTM_hidden_size=2048,
                 edLSTM_num_layers=2):
        """Summarizer: Selector (sLSTM) + VAE (eLSTM/dLSTM)."""
        super().__init__()
        self.s_lstm = sLSTM(input_size=input_size, hidden_size=sLSTM_hidden_size, num_layers=sLSTM_num_layers)
        self.vae = VAE(input_size=input_size, hidden_size=edLSTM_hidden_size, num_layers=edLSTM_num_layers)

    def forward(self, x, uniform=False):
        """-> x_hat (seq_len, B, input_size), (h_mu, h_logvar), scores (seq_len, B, 1)"""
        if uniform:
            seq_len, batch_size, _ = x.size()
            scores = noise.rand_like(x[:, :, :1], "uniform")
        else:
            scores = self.s_lstm(x)
        x_weighted = x * scores
        x_hat, (h_mu, h_logvar) = self.vae(x_weighted)
        return x_hat, (h_mu, h_logvar), scores


class cLSTM(NativeModule):
    def __init__(self, input_size=1024, hidden_size=1024, num_layers=2):
        """Discriminator as a classifier LSTM"""
        super().__init__()
        self.lstm = nn.LSTM(input_size=input_size, hidden_size=hidden_size, num_layers=num_layers, bidirectional=False)
        self.out = nn.Sequential(nn.Linear(hidden_size, 1), nn.Sigmoid())

    def forward(self, x):
        """x: (seq_len, B, input_size) -> probs (B, 1), h_last (B, hidden_size)"""
        _require_cuda(x, "cLSTM")
        y, _, _ = lstm_stack(self._cache, self.lstm, x.transpose(0, 1))          # [B,T,H]
        h_last = y[:, -1]
        probs = torch.sigmoid(_head1(h_last, self.out[0]))
        return probs, h_last


class GAN(nn.Module):
    def __init__(self, input_size=1024, hidden_size=1024, num_layers=2):
        """GAN: discriminator."""
        super().__init__()
        self.c_lstm = cLSTM(input_size=input_size, hidden_size=hidden_size, num_layers=num_layers)

    def forward(self, x):
        probs, h_last = self.c_lstm(x)
        return probs, h_last


class SumGAN(nn.Module):
    def __init__(self, input_size=1024, sLSTM_hidden_size=1024, sLSTM_num_layers=2, edLSTM_hidden_size=2048,
                 edLSTM_num_layers=2, cLSTM_hidden_size=1024, cLSTM_num_layers=2):
        """SumGAN: Summarizer + GAN"""
        super().__init__()
        self.summarizer = Summarizer(input_size=input_size, sLSTM_hidden_size=sLSTM_hidden_size,
                                     sLSTM_num_layers=sLSTM_num_layers, edLSTM_hidden_size=edLSTM_hidden_size,
                                     edLSTM_num_layers=edLSTM_num_layers)
        self.gan = GAN(input_size=input_size, hidden_size=cLSTM_hidden_size, num_layers=cLSTM_num_layers)

    def forward(self, x):
        """x: (seq_len, B, input_size) -> scores: (seq_len, B, 1)"""
        return self.summarizer.s_lstm(x)


from . import Trainer, clip_grad_norm_, make_adam  # noqa: E402


class SumGANTrainer(Trainer):
    """models/sumgan.py:261-533: VAE pre-training, then per video the selector/encoder, decoder and discriminator
    updates with their own Adam optimizers.  ``--data_parallel`` (BASELINE config 4) gives every replica a different
    video per step and all-reduces each phase's gradients over NCCL before the clip + update."""

    def _init_model(self):
        ep = self.hps.extra_params or {}
        self.sigma = float(ep.get("sigma", 0.3))
        self.input_size = int(ep.get("input_size", 1024))
        self.sLSTM_hidden_size = int(ep.get("sLSTM_hidden_size", 1024))
        self.sLSTM_num_layers = int(ep.get("sLSTM_num_layers", 2))
        self.edLSTM_hidden_size = int(ep.get("edLSTM_hidden_size", 2048))
        self.edLSTM_num_layers = int(ep.get("edLSTM_num_layers", 2))
        self.cLSTM_hidden_size = int(ep.get("cLSTM_hidden_size", 1024))
        self.cLSTM_num_layers = int(ep.get("cLSTM_num_layers", 2))
        self.sup = bool(ep.get("sup", False))
        self.pretrain_vae = int(ep.get("pretrain_vae", 20))
        self.epoch_noise = int(ep.get("epoch_noise", 0.2 * self.hps.epochs))
        model = SumGAN(input_size=self.input_size, sLSTM_hidden_size=self.sLSTM_hidden_size,
                       sLSTM_num_layers=self.sLSTM_num_layers, edLSTM_hidden_size=self.edLSTM_hidden_size,
                       edLSTM_num_layers=self.edLSTM_num_layers, cLSTM_hidden_size=self.cLSTM_hidden_size,
                       cLSTM_num_layers=self.cLSTM_num_layers)
        self.log.debug("Generator params: {}".format(sum([_.numel() for _ in model.summarizer.parameters()])))
        self.log.debug("Discriminator params: {}".format(sum([_.numel() for _ in model.gan.parameters()])))
        return model

    # ---- losses (sumgan.py:288-318) ------------------------------------------------------------------
    def loss_vae(self, x, x_hat, mu, logvar):
        """minimize log(p(x|e)) - D_KL(q(e|x) || p(e))"""
        return self.loss_recons(x, x_hat) + self.loss_prior(mu, logvar)

    def loss_recons(self, h_real, h_fake):
        """minimize E[l2_norm(phi(x) - phi(x_hat))]"""
        return torch.norm(h_real - h_fake, p=2)

    def loss_prior(self, mu, logvar):
        """minimize -D_KL(q(e|x) || p(e))"""
        return -0.5 * torch.sum(1 + logvar - mu.pow(2) - logvar.exp())

    def loss_sparsity(self, scores, sigma):
        """minimize l2_norm(E[s_t] - sigma)"""
        return torch.abs(torch.mean(scores) - sigma)

    def loss_sparsity_sup(self, scores, gtscores):
        """minimize BCE(scores, gtscores)"""
        return self.loss_BCE(scores, gtscores)

    def loss_gan_generator(self, probs_fake, probs_uniform):
        """maximize E[log(cLSTM(x_hat))] + E[log(cLSTM(x_hat_p))]"""
        label_real = torch.full_like(probs_fake, 0.9)
        return self.loss_BCE(probs_fake, label_real) + self.loss_BCE(probs_uniform, label_real)

    def loss_gan_discriminator(self, probs_real, probs_fake, probs_uniform):
        """maximize E[log(cLSTM(x))] + E[log(1 - cLSTM(x_hat))] + E[log(1 - cLSTM(x_hat_p))]"""
        label_real = torch.full_like(probs_real, 0.9)
        label_fake = torch.full_like(probs_fake, 0.1)
        return self.loss_BCE(probs_real, label_real) + self.loss_BCE(probs_fake, label_fake) \
            + self.loss_BCE(probs_uniform, label_fake)

    # ---- optimisation ----------------------------------------------------------------------------------
    def _adam(self, params):
        return make_adam(params, self.hps.lr, self.hps.weight_decay)

    def _update(self, optimizer, loss, dp, n_active):
        """zero_grad of THIS optimizer, backward, clip over ALL parameters (stale gradients of the other
        sub-networks enter the norm exactly as in sumgan.py:433-436), step.

        Data-parallel: only the stepping optimizer's gradients are all-reduced; the stale gradients of the other
        sub-networks are local to each replica (every rank saw a different video), so a locally computed clip
        coefficient would differ per rank and the replicas would drift apart.  The squared total norm is therefore
        averaged over the ranks and ONE shared coefficient is applied everywhere."""
        optimizer.zero_grad()
        if loss is not None:
            loss.backward()
        if dp is None:
            clip_grad_norm_(self.model.parameters(), 5.0)
        else:
            self._dp_allreduce_grads(dp, [p for g in optimizer.param_groups for p in g["params"]], n_active)
            grads = [p.grad for p in self.model.parameters() if p.grad is not None]
            if grads:
                sq = torch.stack([g.float().pow(2).sum() for g in grads]).sum()
            else:
                sq = torch.zeros((), device=next(self.model.parameters()).device)
            dp.all_reduce(sq)
            coef = torch.clamp(5.0 / (torch.sqrt(sq / dp.get_world_size()) + 1e-6), max=1.0)
            for g in grads:
                g.mul_(coef.to(g.dtype))
        optimizer.step()

    def _groups(self, train_keys, dp, rank, world):
        """[(key of this replica or None, active replicas)] per optimizer step."""
        if dp is not None:
            train_keys = self._dp_shuffle(dp, train_keys)
        else:
            random.shuffle(train_keys)
        out = []
        for i0 in range(0, len(train_keys), world):
            group = train_keys[i0:i0 + world]
            out.append((group[rank] if rank < len(group) else None, len(group)))
        return out

    def pretrain(self, fold):
        """Pretrain VAE before learning the GAN, as recommended in paper (sumgan.py:320-355)"""
        train_keys, _ = self._get_train_test_keys(fold)
        vae_optimizer = self._adam(self.model.summarizer.vae.parameters())
        dp, rank, world = self._dp()
        for epoch in range(self.pretrain_vae):
            losses = []
            for key, n_active in self._groups(train_keys, dp, rank, world):
                loss_vae = None
                noise.begin("pretrain")
                if key is not None:
                    x, _ = self._video_tensors(key)
                    x_hat, (mu, logvar) = self.model.summarizer.vae(x)
                    loss_vae = self.loss_vae(x, x_hat, mu, logvar)
                    losses.append(loss_vae.detach())
                self._update(vae_optimizer, loss_vae, dp, n_active)
            if epoch % 10 == 0 or epoch == self.pretrain_vae - 1:
                avg = float(torch.stack(losses).mean()) if losses else float("nan")
                self.log.info(f"Pretrain: {epoch+1:3}/{self.pretrain_vae:3}   Lvae: {avg:.05f}")

    def _pretrain_epochs(self):
        return self.pretrain_vae

    def _make_optimizers(self):
        """sumgan.py:366-380: selector + encoder, decoder, discriminator each with their own Adam."""
        m = self.model
        self.s_e_optimizer = self._adam(list(m.summarizer.s_lstm.parameters()) + list(m.summarizer.vae.e_lstm.parameters()))
        self.d_optimizer = self._adam(m.summarizer.vae.d_lstm.parameters())
        self.c_optimizer = self._adam(m.gan.c_lstm.parameters())

    def train_step(self, x, y, epoch, dp=None, n_active=1):
        """The three updates of one video (sumgan.py:415-480).  x (T,1,1024), y (T,1,1) or None on an idle replica.
        Returns the detached scalars the reference logs, or None."""
        m, idle = self.model, x is None
        # Sequences that go through the same network inside one phase share its recurrence launches (the weights are
        # streamed once per step for all of them): the discriminator sees [x | x_hat | x_hat_p] as one batch of 2-3, the
        # VAE decodes the selector-weighted and the uniformly weighted features together.  Same losses and gradients as
        # the reference's separate calls (sumgan.py:419-421, 442-446, 463-471).
        # ---- selector and encoder
        loss_s_e = None
        noise.begin("p1")
        if not idle:
            x_hat, (mu, logvar), scores = m.summarizer(x)
            _, h = m.gan(torch.cat([x, x_hat], 1))
            loss_sparsity = self.loss_sparsity_sup(scores, y) if self.sup else self.loss_sparsity(scores, self.sigma)
            loss_s_e = self.loss_recons(h[0:1], h[1:2]) + self.loss_prior(mu, logvar) + loss_sparsity
        self._update(self.s_e_optimizer, loss_s_e, dp, n_active)

        def both_reconstructions():
            """x_hat from the selector's scores and x_hat_p from uniform random scores (Summarizer.forward twice)."""
            scores = m.summarizer.s_lstm(x)
            uniform = noise.rand_like(scores, "uniform")
            x_pair, _ = m.summarizer.vae(torch.cat([x * scores, x * uniform], 1), roles=("eps", "eps_p"))
            return x_pair[:, 0:1], x_pair[:, 1:2], scores
        # ---- decoder
        loss_d = None
        noise.begin("p2")
        if not idle:
            x_hat, x_hat_p, _ = both_reconstructions()
            probs, h = m.gan(torch.cat([x, x_hat, x_hat_p], 1))
            loss_d = self.loss_recons(h[0:1], h[1:2]) + self.loss_gan_generator(probs[1:2], probs[2:3])
        self._update(self.d_optimizer, loss_d, dp, n_active)
        # ---- discriminator
        loss_c = None
        noise.begin("p3")
        if not idle:
            x_hat, x_hat_p, scores = both_reconstructions()
            x_in = x
            if epoch < self.epoch_noise:
                x_in = noise.randn_like(x, "noise_x") * x
                x_hat = x_hat * noise.randn_like(x_hat, "noise_x_hat")
                x_hat_p = x_hat_p * noise.randn_like(x_hat_p, "noise_x_hat_p")
            probs, _ = m.gan(torch.cat([x_in, x_hat, x_hat_p], 1))
            probs_real, probs_fake, probs_uniform = probs[0:1], probs[1:2], probs[2:3]
            loss_c = self.loss_gan_discriminator(probs_real, probs_fake, probs_uniform)
        self._update(self.c_optimizer, loss_c, dp, n_active)
        if idle:
            return None
        return dict(Lse=loss_s_e.detach(), Ld=loss_d.detach(), Lc=loss_c.detach(), D_x=probs_real.detach().mean(),
                    D_x_hat=probs_fake.detach().mean(), D_x_hat_p=probs_uniform.detach().mean(), scores=scores.detach())

    def train(self, fold):
        self.model.train()
        train_keys, _ = self._get_train_test_keys(fold)
        self.draw_gtscores(fold, train_keys)
        dp, rank, world = self._dp()
        if dp is not None:
            self._dp_sync_model(dp)
        if self._pretrain_epochs() > 0:
            self.pretrain(fold)
        self._make_optimizers()
        self.loss_BCE = nn.BCELoss()
        best_corr, best_avg_f_score, best_max_f_score = -1.0, 0.0, 0.0
        tags = ("Lse", "Ld", "Lc", "D_x", "D_x_hat", "D_x_hat_p")
        for epoch in range(self.hps.epochs):
            logs, dist_scores = [], {}
            for key, n_active in self._groups(train_keys, dp, rank, world):
                x, y = self._video_tensors(key) if key is not None else (None, None)
                out = self.train_step(x, y, epoch, dp, n_active)
                if out is not None:
                    logs.append(torch.stack([out[t].float() for t in tags]))
                    dist_scores[key] = out["scores"]
            avg = torch.stack(logs).mean(0).tolist()                  # one device sync per epoch
            self.log.info(f"Epoch: {f'{epoch+1}/{self.hps.epochs}':6}   Lse: {avg[0]:.05f}  Ld: {avg[1]:.05f}  "
                          f"Lc: {avg[2]:.05f}  D(x): {avg[3]:.05f}  D(x_hat): {avg[4]:.05f}  D(x_hat_p): {avg[5]:.05f}")
            for t, v in zip(tags, avg):
                self.hps.writer.add_scalar(f"{self.dataset_name}/Fold_{fold+1}/Train/{t}", v, epoch)
            if epoch % self.hps.test_every_epochs == 0:
                avg_corr, (avg_f_score, max_f_score) = self.test(fold)
                self.model.train()
                self.hps.writer.add_scalar(f"{self.dataset_name}/Fold_{fold+1}/Test/Correlation", avg_corr, epoch)
                self.hps.writer.add_scalar(f"{self.dataset_name}/Fold_{fold+1}/Test/F-score_avg", avg_f_score, epoch)
                self.hps.writer.add_scalar(f"{self.dataset_name}/Fold_{fold+1}/Test/F-score_max", max_f_score, epoch)
                best_avg_f_score = max(best_avg_f_score, avg_f_score)
                best_max_f_score = max(best_max_f_score, max_f_score)
                if avg_corr > best_corr:
                    best_corr = avg_corr
                    self.best_weights = self.model.state_dict()
        self.draw_scores(fold, {k: v.cpu().numpy() for k, v in dist_scores.items()})
        return best_corr, best_avg_f_score, best_max_f_score


if __name__ == "__main__":
    model = SumGAN().cuda()
    x = torch.randn(10, 3, 1024).cuda()
    x_hat, (mu, logvar), scores = model.summarizer(x)
    print(x.shape, x_hat.shape, scores.shape, mu.shape, logvar.shape)
    assert x.shape[0] == scores.shape[0] and x.shape[1] == scores.shape[1] and scores.shape[2] == 1
    assert x.shape == x_hat.shape
    probs, h = model.gan(x)
    print(probs.shape, h.shape)
    assert model(x).shape == scores.shape
