"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Golden vectors of the scorer models: the UNMODIFIED reference nn.Modules (imported from $SMZ_REFERENCE_ROOT
through oracle/ref_import.py) run on seeded weights and inputs on the CPU in float32.  The tests rebuild
the same weights and inputs from the seeds, so only the outputs (and per-parameter checksums that prove
the rebuilt weights are the reference's) are stored.   python -m oracle.gen_golden
"""
import os

import numpy as np
import torch

VASNET_CASES = [
    # name, seed, T, B, constructor kwargs, sharpen (factor applied to Q/K weights so attention is peaky)
    ("vas_small", 0, 10, 3, {}, 1.0),                       # the reference's own smoke shape (vasnet.py:255)
    ("vas_t64", 1, 64, 1, {}, 6.0),
    ("vas_t300", 2, 300, 1, {}, 6.0),                       # SumMe video_1 length
    ("vas_t707_b2", 3, 707, 2, {}, 4.0),                    # TVSum video_1 length, ragged tiles
    ("vas_local", 4, 200, 1, {"attention_aperture": 12}, 6.0),
    ("vas_noself", 5, 130, 2, {"ignore_self": True, "scale": 0.06}, 6.0),
    ("vas_he_pos", 6, 96, 1, {"weight_init": "he", "max_length": 128, "pos_embed": "attention"}, 1.0),
    ("vas_pos_simple", 7, 50, 2, {"max_length": 64, "pos_embed": "simple"}, 0.5),   # N(0,1) embeddings: keep logits O(1)
]

DSN_CASES = [("dsn_small", 0, 10, 3), ("dsn_t64", 1, 64, 1), ("dsn_t300", 2, 300, 1), ("dsn_t707_b2", 3, 707, 2)]


def make_input(seed, T, B):
    """Non-negative, L2-normalised rows like GoogLeNet pool5 features (SURVEY.md §8d)."""
    g = torch.Generator().manual_seed(10_000 + seed)
    x = torch.randn(T, B, 1024, generator=g).abs()
    return x / x.norm(dim=2, keepdim=True)


def build_vasnet(cls, seed, kwargs, sharpen):
    torch.manual_seed(seed)
    m = cls(**kwargs)
    with torch.no_grad():
        m.Q.weight.mul_(sharpen)
        m.K.weight.mul_(sharpen)
        # non-trivial LayerNorm affine and biases (the reference initialises them to 1 / 0 / 0.1)
        g = torch.Generator().manual_seed(20_000 + seed)
        m.layer_norm.weight.add_(0.2 * torch.randn(1024, generator=g))
        m.layer_norm.bias.add_(0.1 * torch.randn(1024, generator=g))
        m.k1.bias.add_(0.05 * torch.randn(1024, generator=g))
    return m.eval()


def build_dsn(cls, seed):
    torch.manual_seed(seed)
    return cls().eval()


def checksums(model):
    return np.asarray([float(p.detach().double().abs().sum()) for _, p in sorted(model.state_dict().items())])


def generate(ns, golden_dir):
    out = {}
    for name, seed, T, B, kw, sharpen in VASNET_CASES:
        m = build_vasnet(ns.vasnet.VASNet, seed, kw, sharpen)
        x = make_input(seed, T, B)
        with torch.no_grad():
            y = m(x.clone())
        out[f"{name}/y"] = y.numpy().astype(np.float32)
        out[f"{name}/checksum"] = checksums(m)
    for name, seed, T, B in DSN_CASES:
        m = build_dsn(ns.dsn.DSN, seed)
        x = make_input(seed, T, B)
        with torch.no_grad():
            y = m(x)
        out[f"{name}/y"] = y.numpy().astype(np.float32)
        out[f"{name}/checksum"] = checksums(m)
    np.savez_compressed(os.path.join(golden_dir, "models_golden.npz"), **out)
    print("models_golden.npz:", len(VASNET_CASES), "VASNet +", len(DSN_CASES), "DSN cases")
