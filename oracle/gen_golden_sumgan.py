"""TEST INFRASTRUCTURE — golden vectors for the SumGAN path, produced by the UNMODIFIED reference modules
(summarizer/models/sumgan.py imported from $SMZ_REFERENCE_ROOT through oracle/ref_import.py), CPU float32.

    python oracle/gen_golden_sumgan.py        # writes tests/golden/sumgan_golden.npz

Per case (seed, T): the reference SumGAN is built under ``torch.manual_seed(seed)`` (the same constructor order
reproduces the same parameters in summarizer_b200.models.sumgan.SumGAN; a per-tensor checksum is stored) and run
through the deterministic chain of oracle/models_torch.sumgan_chain — selector scores, encoder statistics, the
step-wise decoder, the discriminator — followed by one backward pass of the probe loss.  Parameter gradients are
stored as (sum, abs-sum, first 8 entries) per tensor: 195 M values do not belong in a fixture."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import ref_import  # noqa: E402
from oracle.gen_golden_models import make_input  # noqa: E402
from oracle.models_torch import sumgan_probes  # noqa: E402

CASES = [("sumgan_t9", 11, 9), ("sumgan_t33", 12, 33)]


def grad_digest(t):
    t = t.detach().double().reshape(-1)
    head = np.zeros(8)
    head[:min(8, t.numel())] = t[:8].numpy()
    return np.concatenate([[float(t.sum()), float(t.abs().sum())], head])


def run_reference(model, x, probes):
    """x (T,1,1024).  Same chain as oracle.models_torch.sumgan_chain, through the reference's own modules."""
    T = x.shape[0]
    scores = model(x)                                                  # SumGAN.forward = s_lstm
    (mu, logvar), c = model.summarizer.vae.e_lstm(x * scores)
    x_hat = model.summarizer.vae.d_lstm(T, mu, c)
    prob, h_last = model.gan(x_hat)
    loss = (x_hat[:, 0] * probes["x_hat"]).sum() + (mu[:, 0] * probes["mu"]).sum() + (logvar[:, 0] * probes["logvar"]).sum() \
        + (h_last[0] * probes["h_last"]).sum() + prob.sum() + (scores.reshape(-1) * probes["scores"]).sum()
    return dict(scores=scores.reshape(-1), mu=mu[:, 0], logvar=logvar[:, 0], c=c[:, 0], x_hat=x_hat[:, 0], prob=prob.reshape(-1),
                h_last=h_last[0], loss=loss)


def generate(ns, golden_dir):
    out = {}
    for name, seed, T in CASES:
        torch.manual_seed(seed)
        model = ns.sumgan.SumGAN()
        x = make_input(seed, T, 1)
        probes = sumgan_probes(seed, T)
        r = run_reference(model, x, probes)
        r["loss"].backward()
        for k in ("scores", "mu", "logvar", "c", "x_hat", "prob", "h_last"):
            out[f"{name}/{k}"] = r[k].detach().numpy().astype(np.float32)
        out[f"{name}/loss"] = np.float64(r["loss"].item())
        names = sorted(n for n, _ in model.named_parameters())
        params = dict(model.named_parameters())
        out[f"{name}/param_names"] = np.asarray(names)
        out[f"{name}/checksum"] = np.asarray([float(params[n].detach().double().abs().sum()) for n in names])
        out[f"{name}/grad_digest"] = np.stack([grad_digest(params[n].grad) for n in names])
    np.savez_compressed(os.path.join(golden_dir, "sumgan_golden.npz"), **out)
    print("sumgan_golden.npz:", [c[0] for c in CASES])


if __name__ == "__main__":
    generate(ref_import.load(), os.path.join(os.path.dirname(HERE), "tests", "golden"))
