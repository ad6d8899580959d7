"""Scorer models and the split-driven train/test loop with the reference's module layout and class
surface (models/__init__.py:9-187 ``Trainer``; one ``*Trainer`` subclass per model file).

What differs from the reference is where the work runs: ``test()`` scores the fold's test videos on the
device and evaluates them with the batched sm_100a kernels (shot selection + F-score + rank correlation)
over dataset fields that were uploaded ONCE per fold (``VideoBatch`` / ``CorrBatch``), instead of re-reading
HDF5 and looping in Python per video (models/__init__.py:60-119)."""
import contextlib
import gc
import os
import threading
import weakref

import numpy as np
import torch

from .. import synthetic
from ..batch import VideoBatch
from ..rankcorr import CorrBatch
from ..utils.eval import evaluate_scores, evaluate_summary, generate_scores, generate_summary  # noqa: F401 (reference surface)
from ._packed import NativeModule


def h5_file(path, mode):
    """``h5py.File`` when h5py is installed, else this package's own HDF5 reader / writer (utils/hdf5.py): same
    ``keys() / [] / create_group / create_dataset`` subset, same bytes on disk."""
    try:
        import h5py
        return h5py.File(path, mode)
    except ImportError:
        from ..utils import hdf5
        return hdf5.File(path, mode)


def open_dataset(path, log=None):
    """``h5py.File(path, "r")`` as models/__init__.py:15 (through the built-in HDF5 reader when h5py is not installed);
    when the file does not exist, the seeded synthetic dataset of the same shape (SumMe-/TVSum-shaped, SURVEY.md §8d)
    — the real files are not distributable."""
    if os.path.exists(path):
        return h5_file(path, "r")
    for name in ("summe", "tvsum"):
        if name in os.path.basename(path).lower():
            if log is not None:
                log.warning(f"{path}: file not found -> seeded synthetic {name}-shaped dataset")
            return synthetic.make_dataset(name)
    raise FileNotFoundError(f"dataset {path} not found and no synthetic stand-in is defined for it")


def make_adam(params, lr, weight_decay, capturable=False):
    """torch.optim.Adam's update rule (the reference's optimizer everywhere) on the library's kernel
    (summarizer_b200.optim.Adam: one launch per 64 tensors, device-side step counters, graph-replayable) when every
    parameter is a float32 CUDA tensor; host-only models (tests of the host logic, Rand / Logistic on the CPU) keep
    torch's implementation."""
    params = list(params)
    if params and all(p.is_cuda and p.dtype == torch.float32 for p in params):
        from ..optim import Adam
        return Adam(params, lr=lr, weight_decay=weight_decay)
    return torch.optim.Adam(params, lr=lr, weight_decay=weight_decay, capturable=capturable and bool(params) and all(p.is_cuda for p in params))


def clip_grad_norm_(parameters, max_norm):
    """torch.nn.utils.clip_grad_norm_ on the library's kernels for float32 CUDA gradients (else torch's)."""
    params = [p for p in parameters if p.grad is not None]
    if params and all(p.grad.is_cuda and p.grad.dtype == torch.float32 and p.grad.is_contiguous() for p in params):
        from ..optim import clip_grad_norm_ as clip
        return clip(params, max_norm)
    return torch.nn.utils.clip_grad_norm_(params, max_norm)


_CAPTURE_LOCK = threading.Lock()


@contextlib.contextmanager
def no_gc_during_capture():
    """Python's cyclic garbage collector must not run while a stream capture is open: it can run in ANY thread that
    executes Python (the autograd thread runs the custom Functions' backward) and finalise a ``torch.cuda.CUDAGraph`` left
    in a reference cycle by an earlier fold / trainer — ``cudaGraphExecDestroy`` inside a global-mode capture invalidates
    it ("operation failed due to a previous error during capture"; ``torch.cuda.graph`` no longer collects up front).
    The collector is switched off for the duration of the capture (process-wide, a few milliseconds)."""
    was = gc.isenabled()
    gc.disable()
    try:
        yield
    finally:
        if was:
            gc.enable()


class StepGraphs:
    """Per-video optimizer steps replayed as CUDA graphs.

    A batch-1 training step is launch-bound (VASNet: ~35 kernels of 5-20 us behind ~0.4 ms of Python and launch
    overhead).  ``run(key, step)`` executes ``step(key)`` eagerly on the first visit of a video (allocator warm-up,
    optimizer state, function attributes), captures it on the second visit and replays the graph from then on — one
    graph per video because T differs, all sharing one memory pool.  ``step`` must do the WHOLE update (zero_grad with
    ``set_to_none=True`` first, forward, loss, backward, optimizer step, in-place updates of persistent tensors) and
    return a tuple of tensors; replays hand back clones of them.  Same kernels and arithmetic as the eager step."""

    def __init__(self, trainer, enabled, isolated=False):
        # isolated: always capture in thread-local mode (data-parallel steps hold an NCCL collective, and NCCL's watchdog
        # thread polls events — a "potentially unsafe" call for a global-mode capture)
        self.isolated = bool(isolated)
        # a weak reference: trainer -> StepGraphs -> trainer would keep the CUDA graphs alive until a cyclic collection,
        # i.e. destroy them at an arbitrary later time (see no_gc_during_capture)
        self.trainer, self.enabled = (weakref.proxy(trainer) if trainer is not None else None), bool(enabled)
        self.graphs, self.seen = {}, set()
        # ONE graph memory pool per trainer, reused fold after fold: a fresh pool per fold meant a round of cudaMalloc /
        # cudaFree per fold, which serialises on the driver when several ranks of a box train folds side by side
        if self.enabled and getattr(trainer, "_graph_pool", None) is None:
            trainer._graph_pool = torch.cuda.graph_pool_handle()
        self.pool = trainer._graph_pool if self.enabled else None

    def run(self, key, step):
        if not self.enabled or key not in self.seen:
            self.seen.add(key)
            return step(key)
        if key not in self.graphs:
            try:
                # Fold-concurrent training (main._train_jobs_concurrently) runs this on a worker thread under its own
                # stream: capture on THAT stream (torch's default capture stream is one object shared by all threads),
                # in thread-local capture mode (other workers keep launching / allocating meanwhile), one capture at a
                # time.  On the default stream: torch's defaults, as before.
                cur = torch.cuda.current_stream()
                own = cur != torch.cuda.default_stream()
                kw = dict(stream=cur, capture_error_mode="thread_local") if own else (
                    dict(capture_error_mode="thread_local") if self.isolated else {})
                with _CAPTURE_LOCK, no_gc_during_capture():
                    cur.synchronize() if own else torch.cuda.synchronize()
                    g = torch.cuda.CUDAGraph()
                    # the bf16 weight copies must be REBUILT INSIDE the graph: a copy cached by an eager call (e.g. test()
                    # right before) would be baked in by address and never refreshed on replay
                    self.trainer._invalidate_shadows()
                    with torch.cuda.graph(g, pool=self.pool, **kw):
                        static = tuple(step(key))
                self.graphs[key] = (g, static)
            except Exception as e:                                # capture refused: stay eager (same kernels)
                self.trainer.log.warning(f"CUDA graph capture failed ({type(e).__name__}: {e}); continuing without graphs")
                self.enabled = False
                torch.cuda.synchronize()
                self.trainer._invalidate_shadows()
                return step(key)
        g, static = self.graphs[key]
        g.replay()
        self.trainer._invalidate_shadows()       # the modules' cached bf16 weight copies were rebuilt inside graph memory
        return tuple(t.clone() for t in static)


class Trainer:
    """Abstract class handling the training process"""

    def __init__(self, hps, splits_file):
        self.hps = hps
        self.log = hps.logger
        self.splits_file = splits_file
        self.dataset = open_dataset(hps.dataset_of_file[splits_file], self.log)
        self.dataset_name = hps.dataset_name_of_file[splits_file]
        self._fold_eval = {}
        self._dev_cache = {}

    # ---- reference surface ------------------------------------------------------------------------
    def reset(self):
        """Reset between two folds of the cross-validation"""
        new = self._init_model()
        # (the reference empties the CUDA caching allocator here, models/__init__.py:21: a synchronising round of
        # cudaFree that changes no result; the cached blocks are simply reused by the next fold)
        if self.hps.use_cuda:
            new.cuda()
        old = getattr(self, "model", None)
        if old is not None and self._same_layout(old, new):
            # Same architecture as the previous fold: the freshly initialised weights are copied INTO the existing
            # tensors, so every address the previous folds' CUDA graphs captured stays valid and the per-video step
            # graphs (and the optimizer object, whose state _train_supervised zeroes) are reused instead of being
            # re-captured fold after fold (capture was ~60 % of a 20-epoch SumMe / TVSum fold).
            best = getattr(self, "best_weights", None)
            if best is not None:       # it aliases the live parameters (as the reference): detach it before they change
                self.best_weights = {k: v.detach().clone() for k, v in best.items()}
            with torch.no_grad():
                for dst, src in zip(old.state_dict().values(), new.state_dict().values()):
                    dst.copy_(src)
            self._invalidate_shadows()
        else:
            self.model = new
            self._step_graphs, self._opt_key = None, None
        return self

    @staticmethod
    def _same_layout(a, b):
        if type(a) is not type(b):
            return False
        sa, sb = a.state_dict(), b.state_dict()
        return list(sa.keys()) == list(sb.keys()) and all(
            x.shape == y.shape and x.dtype == y.dtype and x.device == y.device for x, y in zip(sa.values(), sb.values()))

    def _get_train_test_keys(self, fold):
        """Train/Test keys from current split file and fold"""
        self.fold = fold
        self.split = self.hps.splits_of_file[self.splits_file][fold]
        return self.split["train_keys"][:], self.split["test_keys"][:]

    def _init_model(self):
        raise Exception("_init_model has not been implemented")

    def train(self, fold):
        raise Exception("train has not been implemented")

    # ---- data staging -----------------------------------------------------------------------------
    def _device(self):
        return torch.device("cuda", torch.cuda.current_device()) if self.hps.use_cuda else torch.device("cpu")

    def _video_tensors(self, key):
        """(features (T,1,1024), min-max normalised gtscore (T,1,1)) on the model's device, staged once
        (the reference re-reads HDF5 and copies host->device every step, vasnet.py:194-205)."""
        if key not in self._dev_cache:
            d = self.dataset[key]
            seq = torch.from_numpy(np.asarray(d["features"][...], dtype=np.float32)).unsqueeze(1)
            target = torch.from_numpy(np.asarray(d["gtscore"][...], dtype=np.float32)).view(-1, 1, 1).clone()
            target -= target.min()
            target /= target.max() - target.min()
            self._dev_cache[key] = (seq.to(self._device()), target.to(self._device()))
        return self._dev_cache[key]

    def _model_input(self, seq):
        """The cached device features, or a private copy when the model writes into its input (VASNet adds the positional
        embedding IN PLACE to the caller's tensor when ``max_pos`` is set, vasnet.py:110,112; the reference re-reads the
        HDF5 features every step, so the write never accumulates there)."""
        return seq.clone() if getattr(self.model, "max_length", None) is not None else seq

    def _eval_batches(self, test_keys):
        """Resident evaluation inputs of a set of test keys (built once per key set)."""
        tag = tuple(test_keys)
        if tag not in self._fold_eval:
            vids, corr = [], []
            for key in test_keys:
                d = self.dataset[key]
                if "change_points" not in d:
                    raise Exception(f"No /change_points in video {key} for summary evaluation, "
                                    "make sure you have up-to-date .h5 dataset files.")
                if "user_scores" not in d:
                    raise Exception(f"No /user_scores in video {key} for score evaluation, "
                                    "make sure you have up-to-date .h5 dataset files.")
                n_frames = int(d["n_frames"][()])
                vids.append(dict(n_frames=n_frames, picks=d["picks"][...], change_points=d["change_points"][...],
                                 n_frame_per_seg=d["n_frame_per_seg"][...], user_summary=d["user_summary"][...]))
                corr.append((n_frames, d["user_scores"][...]))
            self._fold_eval[tag] = (VideoBatch(vids, proportion=self.hps.summary_proportion), CorrBatch(corr))
        return self._fold_eval[tag]

    # ---- evaluation -------------------------------------------------------------------------------
    def _packed_scorer(self):
        """The module whose ``score_packed`` scores all test videos in ONE call (ragged batch), or None to run the
        model's forward once per video."""
        return None

    def _score_keys(self, keys):
        """Model scores of several videos -> list of (T,) float32 device tensors."""
        scorer = self._packed_scorer()
        with torch.no_grad():
            if scorer is not None:
                feats = [self._video_tensors(k)[0][:, 0] for k in keys]
                lengths = [f.shape[0] for f in feats]
                return list(torch.split(scorer.score_packed(torch.cat(feats), lengths), lengths))
            return [self.model(self._model_input(self._video_tensors(k)[0])).reshape(-1).float() for k in keys]

    def test(self, fold):
        """Test model on test_keys -> (avg_corr, (avg_f_score, max_f_score))  (models/__init__.py:40-58)"""
        self.model.eval()
        _, test_keys = self._get_train_test_keys(fold)
        if not self.hps.use_cuda:
            raise RuntimeError("summarizer_b200 evaluates on the device: run with --use-cuda yes on a B200")
        scores = torch.cat(self._score_keys(test_keys))
        batch, corr = self._eval_batches(test_keys)
        avg_corr = self._eval_scores_device(scores, batch, corr)
        avg_f_score, max_f_score = self._eval_summary_device(scores, batch)
        return avg_corr, (avg_f_score, max_f_score)

    def _eval_scores_device(self, scores, batch, corr):
        """models/__init__.py:60-86 — mean over test keys of the mean Spearman correlation per video."""
        frame_scores = batch.upsample(scores)
        batch.check_status()
        per_video = corr.correlate(frame_scores, "spearmanr").cpu().numpy()
        return np.mean(per_video)

    def _eval_summary_device(self, scores, batch):
        """models/__init__.py:88-119 — mean over test keys of (avg F, max F) per video."""
        batch.select(scores, method=self.hps.selection_algorithm).fscore()
        batch.check_status()
        overlap = batch.overlap[: batch.total_users].cpu().numpy()
        avg = batch.avg_f[: batch.n_videos].cpu().numpy()
        mx = batch.max_f[: batch.n_videos].cpu().numpy()
        avg_f, max_f = [], []
        for i in range(batch.n_videos):   # scalar dtypes as utils/eval.py:156-164 returns them under numpy 2
            kind = np.float64 if (overlap[batch.users_slice(i)] == 0).any() else np.float32
            avg_f.append(kind(avg[i])); max_f.append(kind(mx[i]))
        return np.mean(avg_f), np.mean(max_f)

    # per-key host versions kept for API compatibility (models/__init__.py:60-119)
    def _eval_scores(self, machine_summary_activations, test_keys):
        scores = torch.cat([torch.as_tensor(machine_summary_activations[k]).reshape(-1).float() for k in test_keys])
        batch, corr = self._eval_batches(test_keys)
        return self._eval_scores_device(scores.cuda(), batch, corr)

    def _eval_summary(self, machine_summary_activations, test_keys):
        scores = torch.cat([torch.as_tensor(machine_summary_activations[k]).reshape(-1).float() for k in test_keys])
        batch, _ = self._eval_batches(test_keys)
        return self._eval_summary_device(scores.cuda(), batch)

    # ---- data-parallel single-split training (BASELINE config 4 style): one video per rank and optimizer step ----
    def _dp(self):
        """(dist, rank, world) when ``--data_parallel`` is set and a process group exists, else (None, 0, 1).
        This is the ONE place of the path with a real exchange step: the gradient all-reduce (NCCL over NVLink)."""
        ep = self.hps.extra_params or {}
        if not ep.get("data_parallel", False):
            return None, 0, 1
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return None, 0, 1
        return dist, dist.get_rank(), dist.get_world_size()

    def _dp_sync_model(self, dist):
        """Replicas start from rank 0's initial weights (the reference never seeds its initialisation)."""
        for t in list(self.model.parameters()) + list(self.model.buffers()):
            dist.broadcast(t.data, src=0)

    def _dp_shuffle(self, dist, keys):
        import random
        box = [keys]
        if dist.get_rank() == 0:
            random.shuffle(box[0])
        dist.broadcast_object_list(box, src=0)
        return box[0]

    _flat_grads = {}      # (ids of the parameters) -> persistent flat float32 gradient buffer

    @staticmethod
    def _dp_allreduce_grads(dist, params, n_active):
        """Mean of the replicas' gradients: ONE all-reduce per step of a PERSISTENT flat float32 buffer.  Every
        parameter's ``.grad`` is (made) a view into that buffer, so the next backward accumulates straight into it:
        when the caller zeroes gradients in place (``zero_grad(set_to_none=False)``) a step copies nothing at all,
        otherwise one copy per parameter brings the fresh gradient tensor in — no concatenation, no split-back."""
        params = list(params)
        key = tuple(id(p) for p in params)
        flat = Trainer._flat_grads.get(key)
        total = sum(p.numel() for p in params)
        if flat is None or flat.numel() != total or flat.device != params[0].device:
            if len(Trainer._flat_grads) > 8:
                Trainer._flat_grads.clear()
            flat = Trainer._flat_grads[key] = torch.zeros(total, dtype=torch.float32, device=params[0].device)
        o = 0
        for p in params:
            n = p.numel()
            view = flat[o:o + n].view_as(p)
            g = p.grad
            if g is None:
                view.zero_()
            elif g.data_ptr() != view.data_ptr():
                view.copy_(g)
            p.grad = view
            o += n
        dist.all_reduce(flat)
        flat /= float(n_active)

    def _invalidate_shadows(self):
        """Drop the modules' cached bf16 / packed weight copies (they are rebuilt on the next call)."""
        for m in self.model.modules():
            if isinstance(m, NativeModule):
                m._cache.clear()

    # ---- supervised loop shared by the MSE-trained scorers (vasnet.py:171-238, logistic.py:42-112) ---
    def _train_supervised(self, fold, optimizer_params=None):
        import random
        self.model.train()
        train_keys, _ = self._get_train_test_keys(fold)
        self.draw_gtscores(fold, train_keys)
        from ..optim import mse_loss as criterion                 # torch.nn.MSELoss() in one launch with its gradient
        params = [p for p in self.model.parameters() if p.requires_grad] if optimizer_params is None else optimizer_params
        # same update rule as the reference's torch.optim.Adam (L2 term in the gradient), one multi-tensor kernel of the
        # library on the device (make_adam)
        fused = bool(params) and all(p.is_cuda for p in params)
        dist, rank, world = self._dp()
        # from the second visit of a video on, its whole step (forward, loss, backward, Adam) is replayed as ONE CUDA
        # graph (StepGraphs); `--cuda_graphs no` keeps it eager
        ep = self.hps.extra_params or {}
        # Data-parallel mode: the step can be replayed as a graph with the NCCL all-reduce captured INSIDE it
        # (`--dp_cuda_graphs yes`; 2 B200s: 5.3 s -> 1.5 s for a 12-epoch TVSum cross-validation, replicas
        # identical).  OPT-IN: replicas capture at different steps (their own second visit of a video), and whether NCCL's
        # graph-time buffer registration tolerates that on every topology (NVLS on 8 GPUs) has not been established —
        # the default keeps data-parallel steps eager.
        dp_graphable = dist is None or (str(dist.get_backend()).lower() == "nccl"
                                        and str(ep.get("dp_cuda_graphs", "no")).lower() in ("yes", "1", "true"))
        use_graphs = (fused and dp_graphable and getattr(self.model, "max_length", None) is None
                      and str(ep.get("cuda_graphs", "yes")).lower() not in ("no", "0", "false"))
        opt_key = (tuple(id(p) for p in params), float(self.hps.lr), float(self.hps.weight_decay), fused, use_graphs)
        if use_graphs and getattr(self, "_opt_key", None) == opt_key and getattr(self, "_step_graphs", None) is not None:
            # a later fold on the same parameter tensors (see reset()): a fresh optimizer = the old one with its state
            # zeroed in place, and the step graphs captured by the earlier folds replay as they are
            for st in self.optimizer.state.values():
                for t in st.values():
                    if torch.is_tensor(t):
                        t.zero_()
            graphs = self._step_graphs
        else:
            self.optimizer = make_adam(params, self.hps.lr, self.hps.weight_decay, capturable=use_graphs) if params else None
            graphs = StepGraphs(self, use_graphs, isolated=dist is not None)
            self._step_graphs, self._opt_key = (graphs, opt_key) if use_graphs else (None, None)
        best_corr, best_avg_f_score, best_max_f_score = -1.0, 0.0, 0.0
        if dist is not None:
            self._dp_sync_model(dist)

        def forward_backward(key):
            seq, target = self._video_tensors(key)
            scores = self.model(self._model_input(seq))
            loss = criterion(scores, target)
            if self.optimizer is not None:
                loss.backward()
            return loss.detach(), scores.detach()

        def full_step(key):                                      # what a CUDA graph replays
            self.optimizer.zero_grad(set_to_none=True)
            out = forward_backward(key)
            self.optimizer.step()
            return out

        def full_step_dp(job):                                   # data parallel: (video of this replica, replicas with a video)
            key, n_active = job
            self.optimizer.zero_grad(set_to_none=False)          # gradients stay views of the flat all-reduce buffer
            out = forward_backward(key)
            self._dp_allreduce_grads(dist, params, n_active)
            self.optimizer.step()
            return out

        for epoch in range(self.hps.epochs):
            losses, dist_scores = [], {}
            if dist is not None:
                train_keys = self._dp_shuffle(dist, train_keys)
            else:
                random.shuffle(train_keys)
            for i in range(0, len(train_keys), world):
                group = train_keys[i:i + world]                  # one video per replica and optimizer step
                key = group[rank] if rank < len(group) else None
                if use_graphs and dist is None:
                    loss, scores = graphs.run(key, full_step)
                    losses.append(loss)
                    dist_scores[key] = scores
                    continue
                if use_graphs and key is not None:
                    # one graph per (video, group size) on this replica: forward, loss, backward, the NCCL all-reduce of the
                    # flat gradient buffer and Adam.  Replicas capture at different steps (their own second visit of a
                    # video); a capture only records, the replay right behind it executes — every replica still issues
                    # exactly one all-reduce per step, eager or replayed.  A replica without a video (last, partial group)
                    # takes the eager path below.
                    loss, scores = graphs.run((key, len(group)), full_step_dp)
                    losses.append(loss)
                    dist_scores[key] = scores
                    continue
                if self.optimizer is not None:
                    self.optimizer.zero_grad(set_to_none=dist is None)       # data parallel: gradients stay views of the flat buffer
                if key is not None:
                    loss, scores = forward_backward(key)
                    losses.append(loss)
                    dist_scores[key] = scores
                if self.optimizer is not None:
                    if dist is not None:
                        self._dp_allreduce_grads(dist, params, len(group))
                    self.optimizer.step()
            train_avg_loss = float(torch.stack(losses).mean())          # one sync per epoch, not per step
            self.log.info(f"Epoch: {f'{epoch+1}/{self.hps.epochs}':6}   Loss: {train_avg_loss:.05f}")
            self.hps.writer.add_scalar(f"{self.dataset_name}/Fold_{fold+1}/Train/Loss", train_avg_loss, epoch)
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
                    self.best_weights = self.model.state_dict()      # aliases the live parameters, as the reference
        self.draw_scores(fold, {k: v.cpu().numpy() for k, v in dist_scores.items()})
        return best_corr, best_avg_f_score, best_max_f_score

    # ---- logging / persistence (models/__init__.py:121-187) ------------------------------------------
    def draw_gtscores(self, fold, keys, norm=True):
        for key in keys:
            i = int(key.split("_")[1])
            gtscore = np.array(self.dataset[key]["gtscore"][...], dtype=np.float32)
            if norm:
                gtscore -= gtscore.min()
                gtscore /= gtscore.max() - gtscore.min()
            self.hps.writer.add_histogram(f"{self.dataset_name}/Fold_{fold+1}/Train/gtscores", gtscore, i)

    def draw_scores(self, fold, dist_scores):
        for key, scores in dist_scores.items():
            i = int(key.split("_")[1])
            self.hps.writer.add_histogram(f"{self.dataset_name}/Fold_{fold+1}/Train/final_scores", scores, i)

    def predict_dataset(self, pred_path):
        """Predict on all videos of the dataset (models/__init__.py:142-177): ``<pred_path>`` is an HDF5 file with one
        group per dataset file (its basename) holding, per video key, ``scores``, ``user_summary``,
        ``machine_summary`` and ``machine_scores`` — written with h5py when it is installed, else with the built-in
        writer (utils/hdf5.py); summary.py:40-43 reads it back either way."""
        self.model.load_state_dict(self.best_weights)
        self.model.eval()
        keys = list(self.dataset.keys())
        scores = self._score_keys(keys)
        batch, _ = self._eval_batches(keys)
        packed = torch.cat(scores)
        batch.select(packed, method=self.hps.selection_algorithm)
        machine_scores = batch.upsample(packed)
        batch.check_status()
        group = os.path.basename(self.hps.dataset_of_file[self.splits_file])
        with h5_file(pred_path, "w") as f:
            d, fo = f.create_group(group), 0
            for i, key in enumerate(keys):
                n_frames = int(batch.h_desc[i]["n_frames"])
                k = d.create_group(key)
                k.create_dataset("scores", data=scores[i].cpu().numpy())
                k.create_dataset("user_summary", data=np.asarray(self.dataset[key]["user_summary"][...]))
                k.create_dataset("machine_summary", data=batch.summary_of(i).cpu().numpy())
                k.create_dataset("machine_scores", data=machine_scores[fo:fo + n_frames].cpu().numpy())
                fo += n_frames

    def save_best_weights(self, weights_path):
        if self.best_weights is None:
            raise Exception("best_weights property is empty, can't save model's weights")
        torch.save(self.best_weights, weights_path)

    def load_weights(self, weights_path):
        self.model.load_state_dict(torch.load(weights_path))
