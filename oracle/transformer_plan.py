"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Python restatement of the inference launch plan of the Transformer scorer: how ``smz_transformer_forward``
(``make_plan`` in summarizer_b200/csrc/smz_transformer.cu) splits a packed batch into row chunks and sizes its work
buffer, and how ``smz_mha_forward`` (``mha_forward`` in summarizer_b200/csrc/smz_attn.cu) numbers its work units and
hands them to the CTAs of its persistent grid.  tests/test_transformer_plan_gpu.py pins it against the library's own
``smz_transformer_workspace_bytes`` / ``smz_mha_workspace_bytes`` (host-only entry points, no device needed) and then
uses it to assert that every batch a GPU test runs reaches the structure it is meant to cover.
"""
from typing import List, NamedTuple

ROW_CHUNK = 32768           # kRowChunk: rows per chunk of whole videos
FEAT = 1024                 # kFeat
GEMM_BN = 256               # smz::GEMM_BN: columns per GEMM tile, two row-statistic slots per tile
HEAD_SLOTS = 2 * FEAT // GEMM_BN
BQ = BKV = 128              # query rows per attention work unit, keys per key tile
TABLE_ENTRY = 16            # sizeof(MhaVideo): row0, T, unit0, qtiles


def up(x, m):
    return (x + m - 1) // m * m


class Chunk(NamedTuple):
    v0: int         # first video
    v1: int         # one past the last video
    row0: int       # first packed row
    rows: int


class Unit(NamedTuple):
    video: int      # index into the call's lengths
    head: int
    qt: int         # 128-row query tile of the video
    nk: int         # 128-key tiles of the video


def chunks(lengths):
    """Whole videos up to ROW_CHUNK rows per chunk; a longer video is a chunk of its own."""
    n = len(lengths)
    assert n > 0 and all(T > 0 for T in lengths)
    out, v, row0 = [], 0, 0
    while v < n:
        v0, rows = v, 0
        while v < n and (rows == 0 or rows + lengths[v] <= ROW_CHUNK):
            rows += lengths[v]
            v += 1
        out.append(Chunk(v0, v, row0, rows))
        row0 += rows
    return out


def table_bytes(n_videos):
    """smz_mha_workspace_bytes: the work-unit table of n_videos videos."""
    return up(TABLE_ENTRY * n_videos, 1024)


def workspace_bytes(lengths):
    """smz_transformer_workspace_bytes: one set of chunk buffers sized for the largest chunk, then the attention table
    of the whole batch (chunk k writes its part at byte v0 * 16)."""
    R = up(max(c.rows for c in chunks(lengths)), 8)
    return sum(up(b, 1024) for b in (
        R * FEAT * 2,                   # xb: bf16 GEMM operand
        R * FEAT * 4,                   # xf: float32 residual stream
        R * 3 * FEAT * 2,               # qkv
        R * FEAT * 2,                   # a: attention output, then the feed-forward hidden layer
        R * FEAT * 4,                   # y: float32 LayerNorm input
        R * HEAD_SLOTS * 3 * 4,         # head row statistics
    )) + table_bytes(len(lengths))


def mha_schedule(lengths, n_heads, sm_count):
    """The work units of one smz_mha_forward call, per CTA in the order the CTA runs them.  Videos are stably sorted
    longest first; video i of that order owns units [unit0, unit0 + qtiles * n_heads), head-major; the grid is
    min(units, sm_count) CTAs and CTA b runs units b, b + grid, b + 2 * grid, ..."""
    order = sorted(range(len(lengths)), key=lambda v: -lengths[v])     # sorted() is stable
    units: List[Unit] = []
    for v in order:
        T = lengths[v]
        qtiles = (T + BQ - 1) // BQ
        nk = (T + BKV - 1) // BKV
        units += [Unit(v, h, qt, nk) for h in range(n_heads) for qt in range(qtiles)]
    grid = min(len(units), sm_count)
    return [units[b::grid] for b in range(grid)]
