"""DSN — Deep Summarization Network scorer with the reference's class, constructor, parameter names and
``forward((T, B, 1024)) -> (T, B, 1)`` contract (models/dsn.py:17-47), computed by smz_dsn_forward /
smz_dsn_backward: one tcgen05 GEMM for the input projections of both directions and a persistent
8-CTA-cluster recurrence kernel with W_hh resident in registers.

Parameters live in an ``nn.LSTM`` / ``nn.Sequential`` pair exactly like the reference, so the state-dict keys
(``rnn.weight_ih_l0``, ``rnn.weight_hh_l0``, ``rnn.bias_ih_l0``, ``rnn.bias_hh_l0``, ``*_reverse``,
``out.0.weight``, ``out.0.bias``) and the initialisation stream are the reference's; the torch modules are
never executed.  Only the default configuration the reference trainer builds (LSTM cell, 1 layer, hidden 256,
dsn.py:58) is implemented; there is no CPU fallback."""
import ctypes as C
import functools

import numpy as np
import torch
import torch.nn as nn

from .. import _native as N
from ._packed import NativeModule, Workspace, packed_input, score_sequences, workspace_bytes


class DsnParams(C.Structure):
    """struct smz_dsn_params (include/summarizer_b200.h)."""
    _fields_ = [(k, C.c_void_p) for k in ("w_ih", "bias", "whh_packed", "whh_t_packed", "w_out", "b_out")]


class DSN(NativeModule):
    """Deep Summarization Network"""

    def __init__(self, input_size=1024, hidden_size=256, num_layers=1, cell="lstm"):
        super().__init__()
        assert cell in ["lstm", "gru"], "cell must be either 'lstm' or 'gru'"
        if cell != "lstm" or input_size != 1024 or hidden_size != 256 or num_layers != 1:
            raise NotImplementedError("the sm_100a DSN kernels implement the configuration the reference trainer uses: "
                                      "LSTM cell, 1024-d input, hidden size 256, one layer (dsn.py:58)")
        self.rnn = nn.LSTM(input_size, hidden_size, num_layers=num_layers, bidirectional=True)
        self.out = nn.Sequential(nn.Linear(hidden_size * 2, 1), nn.Sigmoid())
        self._ws = Workspace()

    def _params(self):
        r, o = self.rnn, self.out[0]
        return (r.weight_ih_l0, r.weight_hh_l0, r.bias_ih_l0, r.bias_hh_l0, r.weight_ih_l0_reverse, r.weight_hh_l0_reverse,
                r.bias_ih_l0_reverse, r.bias_hh_l0_reverse, o.weight, o.bias)

    def _weights(self, training=False):
        """The kernels' weight copies (cached in ``self._cache``; a training forward rebuilds them) and the parameter
        struct over them."""
        sh = self._cache.get(self._params(), self._build_weights, fresh=training)
        return sh, DsnParams(*(sh[k].data_ptr() for k in ("w_ih", "bias", "whh", "whh_t", "w_out", "b_out")))

    def _build_weights(self):
        wih_f, whh_f, bih_f, bhh_f, wih_b, whh_b, bih_b, bhh_b, w_out, b_out = self._params()
        dev = wih_f.device
        sh = dict(w_ih=torch.cat([wih_f, wih_b], 0).to(torch.bfloat16).contiguous(),
                  bias=torch.cat([bih_f + bhh_f, bih_b + bhh_b]).float().contiguous(),
                  whh=torch.empty(2 * 8 * 64 * 256, dtype=torch.int32, device=dev),
                  whh_t=torch.empty(2 * 8 * 64 * 256, dtype=torch.int32, device=dev),
                  w_out=w_out.float().reshape(-1).contiguous(), b_out=b_out.float().contiguous())
        N.check(N.lib().smz_dsn_pack_whh(N.ptr(whh_f.float().contiguous()), N.ptr(whh_b.float().contiguous()),
                                         N.ptr(sh["whh"]), N.ptr(sh["whh_t"]), N.current_stream()))
        return sh

    def score_packed(self, x, lengths):
        """Inference over a ragged batch: x packed [sum T, 1024] (float32 / bfloat16) -> probs [sum T]."""
        x, cu, is_bf16 = packed_input(x, lengths, 1024)
        _, st = self._weights()
        ws = self._ws.get(workspace_bytes(N.lib().smz_dsn_workspace_bytes, int(cu[-1]), len(lengths), 0, is_bf16), x.device)
        probs = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
        N.check(N.lib().smz_dsn_forward(N.ptr(x), is_bf16, cu.ctypes.data_as(C.c_void_p), len(lengths), C.byref(st), 0,
                                        N.ptr(probs), N.ptr(ws), ws.numel(), N.current_stream()))
        return probs

    def forward(self, x):
        """Pass the input video through the LSTM.
        Input
          x: (seq_len, batch_size, input_size)
        Output
          probs: (seq_len, batch_size, 1)
        """
        if not x.is_cuda:
            raise N.NativeError("summarizer_b200.DSN runs on a CUDA (sm_100a) device only; move the input with .cuda()")
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            from .dsn_autograd import dsn_apply
            return score_sequences(functools.partial(dsn_apply, self), x)
        return score_sequences(self.score_packed, x)



from . import StepGraphs, Trainer, clip_grad_norm_, make_adam  # noqa: E402


def compute_rewards(seq, actions, far_sim=False, temp_dist_thre=20, workspace=None):
    """Rewards of all episodes of one video on the device (dsn.py:185-236 for each row of ``actions``).
    seq: (T, 1024) float32 cuda; actions: (E, T) 0/1.  Returns float32 (E,) cuda tensor."""
    N.require_device()
    seq = seq.detach().reshape(-1, 1024).float().contiguous()
    act = actions.detach().reshape(actions.shape[0], -1).to(torch.uint8).contiguous()
    E, T = act.shape
    ws = (workspace or Workspace()).get(workspace_bytes(N.lib().smz_dsn_reward_workspace_bytes, T, E), seq.device)
    rewards = torch.empty(E, dtype=torch.float32, device=seq.device)
    N.check(N.lib().smz_dsn_reward(N.ptr(seq), T, N.ptr(act), E, int(temp_dist_thre), int(bool(far_sim)), N.ptr(rewards),
                                   N.ptr(ws), ws.numel(), N.current_stream()))
    return rewards


class _EpisodeLogProb(torch.autograd.Function):
    """mean_t log_prob(actions_e) for every episode (dsn.py:126,135) with the draw itself (dsn.py:125) in the same
    kernel; the gradient w.r.t. ``probs`` is torch's ``Bernoulli.log_prob`` backward."""

    @staticmethod
    def forward(ctx, probs, n_episodes, state, given):
        p = probs.detach().reshape(-1).float().contiguous()
        T = p.numel()
        actions = torch.empty(n_episodes, T, dtype=torch.uint8, device=p.device)
        logp = torch.empty(n_episodes, dtype=torch.float32, device=p.device)
        N.check(N.lib().smz_bernoulli_logprob(N.ptr(p), T, n_episodes, N.ptr(state), N.ptr(given) if given is not None else None,
                                              N.ptr(actions), N.ptr(logp), N.current_stream()))
        ctx.save_for_backward(p, actions)
        ctx.shape = probs.shape
        ctx.mark_non_differentiable(actions)
        return logp, actions

    @staticmethod
    def backward(ctx, dlogp, _dactions):
        p, actions = ctx.saved_tensors
        E, T = actions.shape
        dprobs = torch.empty_like(p)
        N.check(N.lib().smz_bernoulli_logprob_backward(N.ptr(p), N.ptr(actions), N.ptr(dlogp.float().contiguous()), T, E,
                                                       N.ptr(dprobs), N.current_stream()))
        return dprobs.reshape(ctx.shape), None, None, None


def sample_episodes(probs, n_episodes, state, given=None):
    """All episodes of a REINFORCE step in one launch (dsn.py:112,125-126): draws ``actions ~ Bernoulli(probs)`` for
    every episode and returns ``(mean_t log_prob(actions_e) float32 (E,), actions uint8 (E, T))``.  ``state`` is the
    device-resident draw state of ``episode_state`` (advanced on the device: graph replays draw fresh episodes);
    ``given`` = (E, T) 0/1 actions to evaluate instead of drawing."""
    N.require_device()
    if given is not None:
        given = given.detach().reshape(n_episodes, -1).to(torch.uint8).contiguous()
    return _EpisodeLogProb.apply(probs, int(n_episodes), state, given)


def episode_state(device, seed=None):
    """{Philox seed, call number, 0} as three device int64 words; the seed comes from torch's generator unless given,
    so ``torch.manual_seed`` makes the episode draws reproducible."""
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    return torch.tensor([seed, 0, 0], dtype=torch.int64, device=device)


class DSNTrainer(Trainer):
    """models/dsn.py:50-236 — REINFORCE with the diversity-representativeness reward; extra parameters parsed as
    the reference does (dsn.py:52-57; note ``beta = int(0.01) = 0`` unless ``--beta`` >= 1)."""

    def _init_model(self):
        ep = self.hps.extra_params or {}
        self.beta = int(ep.get("beta", 0.01))
        self.num_episodes = int(ep.get("num_episodes", 5))
        self.eps = float(ep.get("eps", 0.5))
        self.far_sim = bool(ep.get("far_sim", False))
        self.temp_dist_thre = int(ep.get("temp_dist_thre", 20))
        self.sup = bool(ep.get("sup", False))
        self._reward_ws = Workspace()
        return DSN()

    def _draw_actions(self, probs):
        """Hook for tests that replay the reference's draws (dsn.py:124-126): return (num_episodes, T) 0/1 actions to
        use for this step, or None (default) to let the sampling kernel draw them."""
        return None

    def compute_reward(self, seq, actions, far_sim=False, temp_dist_thre=20):
        """One episode (reference signature, dsn.py:185): seq (T,1,1024), actions (T,1,1) -> scalar tensor."""
        return compute_rewards(seq.reshape(-1, 1024), actions.reshape(1, -1), far_sim, temp_dist_thre, self._reward_ws)[0]

    def _packed_scorer(self):
        return self.model

    def train(self, fold):
        import random
        self.model.train()
        train_keys, _ = self._get_train_test_keys(fold)
        self.draw_gtscores(fold, train_keys)
        self.log.debug("Parameters: {}".format(sum(p.numel() for p in self.model.parameters())))
        self.optimizer = make_adam(self.model.parameters(), self.hps.lr, self.hps.weight_decay)
        loss_BCE = torch.nn.BCELoss()
        dev = self._device()
        key_index = {key: i for i, key in enumerate(sorted(train_keys))}
        baselines = torch.zeros(len(train_keys), device=dev)                      # device-resident: no sync per step
        episode_rng = episode_state(dev)                                          # Philox seed + call number, on the device
        reward_writers = {key: [] for key in train_keys}
        best_corr, best_avg_f_score, best_max_f_score = -1.0, 0.0, 0.0
        dist_, rank, world = self._dp()
        params = list(self.model.parameters())
        if dist_ is not None:
            self._dp_sync_model(dist_)
        ep = self.hps.extra_params or {}
        use_graphs = (dist_ is None and all(p.is_cuda for p in params)
                      and str(ep.get("cuda_graphs", "yes")).lower() not in ("no", "0", "false"))
        graphs = StepGraphs(self, use_graphs)            # the library's Adam keeps its step counters on the device: replayable

        def forward_backward(key):
            """REINFORCE loss of one video and its backward pass -> (loss, probs, mean reward, baseline delta)."""
            seq, target = self._video_tensors(key)
            probs = self.model(seq)                                           # (T,1,1), autograd through the device BPTT
            loss = self.beta * (probs.mean() - self.eps) ** 2                 # summary-length penalty [Eq.11]
            if self.sup:
                loss = loss + loss_BCE(probs, target)
            # the E episodes of dsn.py:122-126 in one launch: draws + mean log-probabilities (smz_bernoulli_logprob)
            log_probs, actions = sample_episodes(probs, self.num_episodes, episode_rng, self._draw_actions(probs))
            rewards = compute_rewards(seq, actions, self.far_sim, self.temp_dist_thre, self._reward_ws)
            base = baselines[key_index[key]].detach().clone()
            # policy gradient [Eq.10], dsn.py:134-138 for all episodes at once:
            #   loss -= sum_e mean_t(log_prob(actions_e)) * (reward_e - baseline)
            loss = loss - (log_probs * (rewards - base)).sum()
            loss = loss / float(self.num_episodes)
            loss.backward()
            mean_reward = rewards.mean()
            delta = torch.zeros_like(baselines)                               # moving-average baseline update (dsn.py:149)
            delta[key_index[key]] = 0.1 * (mean_reward - base)
            return loss.detach(), probs.detach(), mean_reward, delta

        def full_step(key):                                                   # what a CUDA graph replays
            self.optimizer.zero_grad(set_to_none=True)
            loss, probs, mean_reward, delta = forward_backward(key)
            baselines.add_(delta)
            clip_grad_norm_(self.model.parameters(), 5.0)
            self.optimizer.step()
            return loss, probs, mean_reward

        for epoch in range(self.hps.epochs):
            epoch_losses, dist_scores = [], {}
            if dist_ is not None:
                train_keys = self._dp_shuffle(dist_, train_keys)
            else:
                random.shuffle(train_keys)
            for i0 in range(0, len(train_keys), world):
                group = train_keys[i0:i0 + world]                  # one video per replica and step
                key = group[rank] if rank < len(group) else None
                if use_graphs:
                    loss, probs, mean_reward = graphs.run(key, full_step)
                    reward_writers[key].append(mean_reward)
                    epoch_losses.append(loss)
                    dist_scores[key] = probs
                    continue
                self.optimizer.zero_grad()
                if key is not None:
                    loss, probs, mean_reward, delta = forward_backward(key)
                    reward_writers[key].append(mean_reward)
                    epoch_losses.append(loss)
                    dist_scores[key] = probs
                else:
                    delta = torch.zeros_like(baselines)
                if dist_ is not None:
                    self._dp_allreduce_grads(dist_, params, len(group))
                    dist_.all_reduce(delta)                                       # every replica keeps every video's baseline
                baselines.add_(delta)
                clip_grad_norm_(self.model.parameters(), 5.0)
                self.optimizer.step()
            seen = [k for k in train_keys if len(reward_writers[k]) > epoch]
            epoch_avg_reward = float(torch.stack([reward_writers[key][epoch] for key in seen]).mean())
            epoch_avg_loss = float(torch.stack(epoch_losses).mean())
            self.log.info(f"Epoch: {f'{epoch+1}/{self.hps.epochs}':6}   Reward: {epoch_avg_reward:.05f}  Loss: {epoch_avg_loss:.05f}")
            self.hps.writer.add_scalar(f"{self.dataset_name}/Fold_{fold+1}/Train/Reward", epoch_avg_reward, epoch)
            self.hps.writer.add_scalar(f"{self.dataset_name}/Fold_{fold+1}/Train/Loss", epoch_avg_loss, epoch)
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
