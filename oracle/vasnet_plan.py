"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Python restatement of the launch plan of ``smz_vasnet_forward`` (``make_plan`` in summarizer_b200/csrc/smz_vasnet.cu):
for inference, how a packed batch is split into row chunks, attention sub-chunks and lanes; for training
(``smz_vasnet_forward(training=1)`` + ``smz_vasnet_backward``), the per-video regions of the work buffer; and the
work-buffer size that follows.  tests/test_vasnet_plan_gpu.py (inference) and tests/test_vasnet_train_plan_gpu.py
(training) pin it against the library's own ``smz_vasnet_launch_count`` / ``smz_vasnet_workspace_bytes`` (host-only
entry points, no device needed) and then use it to assert that every batch a GPU test runs reaches the plan structure
it is meant to cover.
"""
from typing import List, NamedTuple

ROW_CHUNK = 32768           # kRowChunk: rows per chunk of the row-wise GEMMs
LOGIT_BUDGET = 68 << 20     # logit_budget(): logits per attention sub-chunk (unless SMZ_VASNET_LOGIT_MELEMS is set)
FEAT = 1024                 # kFeat
GEMM_BN = 256               # smz::GEMM_BN: columns per GEMM tile, two row-sum slots per tile
LN_SLOTS = 2 * FEAT // GEMM_BN
PROBLEM_BYTES = 64          # sizeof(smz::GemmProblem)
ROW_WARPS = 8               # warps (one row each per pass) of a CTA of the row kernels, smz_rows.cu


def up(x, m):
    return (x + m - 1) // m * m


class Sub(NamedTuple):
    v0: int         # first video
    v1: int         # one past the last video
    rows: int
    ld: int         # row length of the sub-chunk's logits block


class Chunk(NamedTuple):
    v0: int
    v1: int
    rows: int
    subs: List[Sub]
    ragged: bool    # some video writes fewer row-sum slots than the chunk has: the slots are zeroed first


def row_sum_slots(ld):
    return 2 * ((ld + GEMM_BN - 1) // GEMM_BN)


def plan(lengths, budget=LOGIT_BUDGET):
    """Chunks of an inference call: whole videos up to ROW_CHUNK rows (a longer video is a chunk of its own); inside a
    chunk, sub-chunks of whole videos up to ``budget`` logits (a single larger video is admitted alone).  Chunk k runs
    on lane k & 1 when there are two or more chunks."""
    n = len(lengths)
    assert n > 0 and all(T > 0 for T in lengths)
    chunks, v = [], 0
    while v < n:
        v0, rows = v, 0
        while v < n and (rows == 0 or rows + lengths[v] <= ROW_CHUNK):
            rows += lengths[v]
            v += 1
        subs, u = [], v0
        while u < v:
            s0, srows, max_t = u, 0, 0
            while u < v:
                T = lengths[u]
                nm = max(T, max_t)
                if srows > 0 and (srows + T) * up(nm + 7, 64) > budget:
                    break
                max_t, srows, u = nm, srows + T, u + 1
            subs.append(Sub(s0, u, srows, up(max_t + 7, 64)))
        slots = max(row_sum_slots(s.ld) for s in subs)
        ragged = any(row_sum_slots(T) != slots for T in lengths[v0:v])
        chunks.append(Chunk(v0, v, rows, subs, ragged))
    return chunks


def launch_count(chunks, x_bf16, exact=False):
    """Kernel launches of the call: per chunk [cvt] proj k1 head + (fused-exp logits, alpha.V') per sub-chunk on the
    fast path; [cvt] QKV out layernorm k1 head + (logits, softmax, alpha.V) per sub-chunk on the exact path."""
    cvt = 0 if x_bf16 else 1
    return sum(cvt + (5 + 3 * len(c.subs) if exact else 3 + 2 * len(c.subs)) for c in chunks)


def workspace_bytes(lengths, x_bf16, budget=LOGIT_BUDGET):
    """Work-buffer bytes of an inference call: one copy of the chunk buffers per lane, then the problem tables."""
    chunks = plan(lengths, budget)
    R = up(max(c.rows for c in chunks), 8)
    logits = max(s.rows * s.ld for c in chunks for s in c.subs)
    slots = max(row_sum_slots(s.ld) for c in chunks for s in c.subs)
    lane = sum(up(b, 1024) for b in (
        0 if x_bf16 else R * FEAT * 2,      # float16 copy of float32 features
        R * 3 * FEAT * 2,                   # packed projection rows
        R * FEAT * 2, R * FEAT * 4, R * FEAT * 2, R * FEAT * 4,     # o, y, yn, h
        logits * 4, logits * 2,             # fp32 logits, bf16 probabilities
        R * LN_SLOTS * 3 * 4,               # head sums
        R * slots * 12 + 64,                # softmax row-sum slots
        R * LN_SLOTS * 3 * 4))              # LayerNorm sums
    lanes = 2 if len(chunks) > 1 else 1
    return lanes * lane + up(len(lengths) * 2 * PROBLEM_BYTES, 1024)


# ---- training ------------------------------------------------------------------------------------------------------
class TrainChunk(NamedTuple):
    v: int          # the video (a training chunk holds exactly one, with one attention sub-chunk)
    row0: int       # first row in the row-wise buffers (the packed row of the video)
    rows: int
    vt_off: int     # element offset of the video's V^T (and dV^T) region, [1024, up(T, 8)]
    lg_off: int     # element offset of the video's logits (P, alpha, dP, dS) region, [T, ld]
    ld: int         # row length of that logits region: up(T + 7, 64)


def training_plan(lengths):
    """Chunks of a training call: every video is a chunk of its own and owns a region of each buffer."""
    assert len(lengths) > 0 and all(T > 0 for T in lengths)
    out, row0, vt, lg = [], 0, 0, 0
    for v, T in enumerate(lengths):
        ld = up(T + 7, 64)
        out.append(TrainChunk(v, row0, T, vt, lg, ld))
        row0, vt, lg = row0 + T, vt + FEAT * up(T, 8), lg + T * ld
    return out


def training_launch_count(lengths, x_bf16):
    """Kernel launches of smz_vasnet_forward(training=1): per video [cvt] QK Vt out layernorm k1 head + logits, softmax,
    alpha.V (one sub-chunk)."""
    return len(lengths) * ((0 if x_bf16 else 1) + 6 + 3)


def training_workspace_bytes(lengths, x_bf16, split=False):
    """Work-buffer bytes of a training call (forward and backward share it).  split: the float32-accurate mode
    (SMZ_VASNET_SPLIT), whose second half holds the lo planes at the same offsets."""
    plan = training_plan(lengths)
    R = up(sum(lengths), 8)
    VT = sum(FEAT * up(c.rows, 8) for c in plan)
    LG = sum(c.rows * c.ld for c in plan)
    total = sum(up(b, 1024) for b in (
        0 if x_bf16 else R * FEAT * 2,      # bf16 copy of float32 features
        R * 2 * FEAT * 2,                   # Q | K rows
        VT * 2,                             # V^T of every video
        R * FEAT * 2, R * FEAT * 4, R * FEAT * 2, R * FEAT * 4,     # o, y, yn, h
        LG * 4, LG * 2, LG * 2,             # fp32 logits (dP in the backward), probabilities, dropped-out probabilities
        len(lengths) * 2 * PROBLEM_BYTES,   # GEMM problem tables
        len(lengths) * 8,                   # offsets of the attention keep-masks
        R * 4 * 4,                          # mean / rstd of both LayerNorms
        R * FEAT * 2, R * FEAT * 4, R * FEAT * 2, R * FEAT * 4, R * FEAT * 2,   # dh, dyn, dy, dy float32, dO
        R * 2 * FEAT * 2, VT * 2, LG * 2))  # dQ | dK, dV^T, dS
    return 2 * total if split else total


def row_grid_rows(sm_count):
    """Rows one pass of the capped backward row kernels covers (launch_head_bwd / launch_layernorm_bwd: at most
    2 * sm_count CTAs of ROW_WARPS warps, one row per warp); longer videos make every warp loop over rows."""
    return 2 * sm_count * ROW_WARPS
