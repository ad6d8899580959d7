"""Hyperparameters / run configuration with the reference's attributes and semantics (utils/config.py:21-200).

Kept verbatim in behaviour: defaults (lr 5e-5, weight decay 1e-5, 10 epochs, test every 2, proportion 0.15,
knapsack), the ``-s`` shorthands (minimal / overfit / tvsum / summe / LOL / all), the model registry, the
dataset lookup by name substring, ``logs/<timestamp>_<Trainer>/`` with ``train.log``, weights and prediction
paths, TensorBoard tags.  Documented supersets: comma-separated lists and single custom paths work for
``splits_files`` (the reference iterates such a string character by character, utils/config.py:41,133), paths
are resolved against the package directory when they do not exist relative to the cwd, and handlers are not
duplicated when several HParameters are created in one process."""
import datetime
import inspect
import logging
import os
import shutil

import torch

from . import parse_splits_filename

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _NullWriter:
    """Stand-in when torch.utils.tensorboard is unavailable."""
    def add_scalar(self, *a, **k): pass
    def add_histogram(self, *a, **k): pass
    def add_hparams(self, *a, **k): pass
    def close(self): pass


def _model_registry():
    """utils/config.py:68-77.  transformer and the sumgan_att selector score on the library's kernels (their training
    stays on torch modules); sumgan_att's autoencoder is a plain-torch module (outside the hot path, SURVEY.md §2.1)."""
    from ..models.logistic import LogisticRegressionTrainer
    from ..models.rand import RandomTrainer
    from ..models.vasnet import VASNetTrainer
    reg = {"random": RandomTrainer, "logistic": LogisticRegressionTrainer, "vasnet": VASNetTrainer, None: RandomTrainer}
    try:
        from ..models.dsn import DSNTrainer
        reg["dsn"] = DSNTrainer
    except ImportError:
        pass
    from ..models.sumgan import SumGANTrainer
    from ..models.sumgan_att import SumGANAttTrainer
    from ..models.transformer import TransformerTrainer
    reg["sumgan"] = SumGANTrainer
    reg["sumgan_att"] = SumGANAttTrainer
    reg["transformer"] = TransformerTrainer
    return reg


class HParameters:
    """Hyperparameters configuration class"""

    def __init__(self):
        self.use_cuda = False
        self.cuda_device = 0
        self.weight_decay = 0.00001
        self.lr = 0.00005
        self.epochs = 10
        self.test_every_epochs = 2
        self.datasets = [
            "datasets/summarizer_dataset_summe_google_pool5.h5",
            "datasets/summarizer_dataset_tvsum_google_pool5.h5",
            "datasets/summarizer_dataset_LOL_google_pool5.h5"]
        self.splits_files = "minimal"
        self.model_class = None
        self.extra_params = None
        self.summary_proportion = 0.15
        self.selection_algorithm = "knapsack"
        self.log_level = "info"
        self.log_root = "logs"
        self.tensorboard = True

    def load_from_args(self, args):
        for key in args:
            val = args[key]
            if val is not None:
                if hasattr(self, key) and isinstance(getattr(self, key), list) and isinstance(val, str):
                    val = val.split(",")
                setattr(self, key, val)
        if self.extra_params is None:
            self.extra_params = {}
        registry = _model_registry()
        self.model_class = registry.get(args["model"], None)     # KeyError when "model" is absent, as the reference
        if self.model_class is None:
            raise KeyError(f"{args['model']} model is not unknown")
        self._init()

    def _resolve(self, path):
        return path if os.path.exists(path) else os.path.join(_PKG, path)

    def _init(self):
        log_dir = str(int(datetime.datetime.now().timestamp())) + "_" + self.model_class.__name__
        # several ranks of one run share ONE log directory: rank 0's name is broadcast (each rank building its own from
        # its wall clock only agreed when all of them started within the same second); only rank 0 writes TensorBoard
        rank = 0
        try:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                rank = dist.get_rank()
                box = [log_dir]
                dist.broadcast_object_list(box, src=0)
                log_dir = box[0]
        except ImportError:
            pass
        self.rank = rank
        self.log_path = os.path.join(self.log_root, log_dir)
        os.makedirs(self.log_path, exist_ok=True)
        self.writer = _NullWriter()
        if self.tensorboard and rank == 0:
            try:
                from torch.utils.tensorboard import SummaryWriter
                self.writer = SummaryWriter(self.log_path)
            except Exception:
                pass

        if self.use_cuda == "default":
            self.use_cuda = torch.cuda.is_available()
        elif self.use_cuda in ("yes", True):
            self.use_cuda = True
        else:
            self.use_cuda = False
        if self.use_cuda:
            torch.cuda.set_device(self.cuda_device)
        elif not getattr(self, "allow_cpu", False):
            # Trainer.test() evaluates with the sm_100a kernels: there is no CPU path to fall back to, so say so now
            # rather than at the first test() (tests that only exercise host logic set allow_cpu)
            raise RuntimeError("summarizer_b200 runs on an sm_100 (B200) device: no CUDA device is available or "
                               "--use-cuda no was given, and there is no CPU fallback")

        shorthands = {
            "minimal": ["splits/tvsum_splits_overfit.json"],
            "overfit": ["splits/tvsum_splits_overfit.json", "splits/summe_splits_overfit.json"],
            "tvsum": ["splits/tvsum_splits.json"],
            "summe": ["splits/summe_splits.json"],
            "LOL": ["splits/LOL_splits.json"],
            "all": ["splits/tvsum_splits.json", "splits/tvsum_splits_overfit.json", "splits/summe_splits.json",
                    "splits/summe_splits_overfit.json", "splits/LOL_splits.json"]}
        if isinstance(self.splits_files, str):
            self.splits_files = shorthands.get(self.splits_files, self.splits_files.split(","))
        self.splits_files = [self._resolve(s.strip()) for s in self.splits_files]

        self.dataset_name_of_file, self.dataset_of_file, self.splits_of_file = {}, {}, {}
        for splits_file in self.splits_files:
            dataset_name, splits = parse_splits_filename(splits_file)
            self.dataset_name_of_file[splits_file] = dataset_name
            self.dataset_of_file[splits_file] = self.get_dataset_by_name(dataset_name).pop()
            self.splits_of_file[splits_file] = splits

        self.weights_path, self.pred_path = {}, {}
        for splits_file in self.splits_files:
            base = os.path.basename(splits_file)
            self.weights_path[splits_file] = os.path.join(self.log_path, f"{base}.pth")
            self.pred_path[splits_file] = os.path.join(self.log_path, f"{base}_preds.h5")

        self.logger = logging.getLogger("summarizer")
        for h in list(self.logger.handlers):
            self.logger.removeHandler(h)
        fmt = logging.Formatter("%(asctime)s::%(levelname)s: %(message)s", "%H:%M:%S")
        log_name = "train.log" if self.rank == 0 else f"train.rank{self.rank}.log"
        for h in (logging.StreamHandler(), logging.FileHandler(os.path.join(self.log_path, log_name))):
            h.setFormatter(fmt)
            self.logger.addHandler(h)
        self.logger.setLevel(getattr(logging, str(self.log_level).upper()))

        src = inspect.getfile(self.model_class)
        shutil.copyfile(src, os.path.join(self.log_path, os.path.basename(src)))

    def get_dataset_by_name(self, dataset_name):
        for d in self.datasets:
            if dataset_name in d:
                return [d]
        return None

    def __str__(self):
        names = ["use_cuda", "cuda_device", "log_level", "weight_decay", "lr", "epochs", "summary_proportion",
                 "selection_algorithm", "log_path", "splits_files", "extra_params"]
        return "\n".join(f"[{i}] {n}: {getattr(self, n, None)}" for i, n in enumerate(names))

    def get_full_hps_dict(self):
        return {n: getattr(self, n) for n in ("weight_decay", "lr", "epochs")}
