"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Python restatement of the launch plan of shot selection (``select_plan`` / ``select_launch`` / ``smz_eval_batch`` in
summarizer_b200/csrc/smz_select.cu, with ``dp_layout``, ``dp16_layout``, ``select_layout``, ``tail_words`` and
``queue_bytes``): which DP kernel runs (``dp_kernel<K>``, the 16-bit ``dp16_kernel<KW, MK>`` in front of it, or
``select_generic_kernel<BITS_IN_SMEM>``), which pooling route feeds it, whether the summary / F-score tail is fused into
the DP kernels, the work-buffer size, and the kernels a call launches with their grids.

A pure function of the batch maxima, the method, the device's shared-memory opt-in and SM count, and (where a grid
depends on it) the per-SM occupancy of the DP kernels.  tests/test_select_plan_gpu.py pins it against
``smz_select_workspace_bytes`` and against the launches recorded by torch.profiler, and uses it to assert that every
batch it runs reaches the structure it is meant to cover.
"""
from typing import List, NamedTuple, Optional, Tuple

DP_THREADS = 256
POOL_THREADS = 256
FSCORE_MAX_USERS = 1024
FSCORE_CHUNK = 2048                   # SMZ_FSCORE_CHUNK
ORDER_BUCKETS = 64
POOL_WORDS = 12288 - 16               # kPoolWords: staged scores + segment lists of the regular pooling route
POOL_REGULAR_MAX_SEGS = 2048
GRID_Y_MAX = 65535                    # videos per slice of the pooling / F-score kernels (grid.y, or grid.x of pool_regular)
DP_K = (2, 5, 9, 18, 27, 36, 54)
DP16_PAIRS = ((1, 1), (3, 2), (3, 3), (5, 2), (5, 5), (9, 2), (9, 9), (14, 2), (14, 14), (18, 2), (18, 18), (27, 2),
              (27, 27))
QUEUE_INTS = 1 + 2 * ORDER_BUCKETS + 2      # kQueueInts: dp16 queue head, bucket counts and fills, dp queue, fallback count
B200_SMS = 148
B200_OPTIN = 232448                   # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200
SMEM_PER_SM = 233472                  # shared memory of one SM (for the occupancy estimate below)


def cdiv(a, b):
    return -(-a // b)


def tail_words(max_n_segs, max_n_frames):
    return (max_n_segs + 1) + cdiv(max_n_frames, 32) + 2 * FSCORE_MAX_USERS


def dp_layout_total(K, max_n_segs, max_weight, front_words):
    """Words of dp_kernel<K>'s dynamic shared memory: [pad][row0][pad][row1] (or the fused tail), (w, p), picked, reduce."""
    row = K * DP_THREADS
    pad = max(cdiv(max_weight, 32) * 32, 32)
    o = max(2 * (pad + row), front_words)
    o = (o + 1) & ~1
    return o + 3 * max_n_segs + 32


def dp16_layout(KW, MK, max_n_segs, front_words):
    """(wp, total) words of dp16_kernel<KW, MK>: [mirror pad][row0][mirror pad][row1] (or the fused tail), then two
    (w, p) lists and the picked flags.  wp bounds the scores the fused pooling may stage in front of the lists."""
    H, P = KW * DP_THREADS, MK * DP_THREADS
    o = max(2 * (P + H), front_words)
    wp = (o + 1) & ~1
    return wp, wp + 5 * max_n_segs


def select_layout_total(max_n_segs, max_capacity, max_n_frames, bits_in_smem):
    ncell = max_capacity + 1
    row = max(ncell, max_n_segs, 32)
    o = 2 * row + 7 * max_n_segs + 1 + cdiv(max_n_frames, 32) + 4
    if bits_in_smem:
        o += max_n_segs * cdiv(ncell, 32)
    return o


def queue_bytes(n_videos):
    return (QUEUE_INTS + 2 * n_videos) * 4 + 256


def shrink_grid(n_videos, g):
    """More videos than resident CTAs: the smallest grid with the same number of rounds."""
    if n_videos <= g:
        return n_videos
    rounds = cdiv(n_videos, g)
    return cdiv(n_videos, rounds)


def dp16_min_blocks(KW):
    return 6 if KW <= 5 else (5 if KW <= 9 else (3 if KW <= 14 else (2 if KW <= 18 else 1)))


def occupancy_estimate(kernel, smem_bytes):
    """Resident CTAs per SM used where no device is at hand: what shared memory allows, capped at 8 (256-thread CTAs
    of up to 64 registers), at least the launch bounds' minimum of the kernel."""
    by_smem = SMEM_PER_SM // (smem_bytes + 1024)
    est = max(1, min(8, by_smem))
    if kernel.startswith("dp16_kernel"):
        est = max(est, min(dp16_min_blocks(int(kernel.split("<")[1].split(",")[0])), by_smem))
    return est


class Launch(NamedTuple):
    name: str                           # kernel with its template arguments, e.g. "dp16_kernel<9,2>"
    grid: Tuple[int, int, int]
    smem: Optional[int] = None          # dynamic shared memory bytes, where the plan fixes it


class Plan(NamedTuple):
    k: int                              # cells per thread of dp_kernel; 0: generic kernel
    bits_in_smem: bool
    smem_bytes: int
    grid: int
    ws_words_per_cta: int
    pad_weight: int
    kw16: int                           # 0: no 16-bit pass
    mk16: int
    smem16_bytes: int
    grid16: int
    ws16_words_per_cta: int
    front_words: int                    # > 0: the summary / F-score tail is fused into the DP kernels
    workspace_bytes: int                # smz_select_workspace_bytes

    def dp16_name(self):
        return f"dp16_kernel<{self.kw16},{self.mk16}>" if self.kw16 else None


def plan(n_videos, max_n_segs, max_capacity, max_n_frames, max_seg_frames, optin=B200_OPTIN, sm_count=B200_SMS,
         occupancy=occupancy_estimate, fused_tail=True, dp16=True):
    """select_plan.  occupancy(kernel_name, dynamic_smem_bytes) -> resident CTAs per SM.  fused_tail / dp16: False
    restates SMZ_NO_FUSED_TAIL / SMZ_NO_DP16."""
    ncell = max_capacity + 1
    need = max(ncell, max_n_segs)
    pad_weight = min(max_seg_frames, max_capacity)
    k = next((K for K in DP_K if K * DP_THREADS >= need), 0)
    front = 0
    smem = 0
    if k:
        fw = tail_words(max_n_segs, max_n_frames) if fused_tail else 0
        smem = dp_layout_total(k, max_n_segs, pad_weight, fw) * 4
        if smem <= optin:
            front = fw
        else:
            smem = dp_layout_total(k, max_n_segs, pad_weight, 0) * 4
        if smem > optin:
            k = 0
    kw16 = mk16 = smem16 = grid16 = ws16 = 0
    bits_in_smem = False
    if k:
        per_sm = occupancy(f"dp_kernel<{k}>", smem)
        ws = cdiv(max_n_segs, 32) * k * DP_THREADS
        kw = (k + 1) // 2
        mk = 2 if (kw >= 2 and pad_weight <= 2 * DP_THREADS) else kw
        s16 = dp16_layout(kw, mk, max_n_segs, front)[1] * 4
        if dp16 and s16 <= optin:
            p16 = occupancy(f"dp16_kernel<{kw},{mk}>", s16)
            if p16 >= 1:
                kw16, mk16, smem16 = kw, mk, s16
                grid16 = shrink_grid(n_videos, sm_count * p16)
                ws16 = cdiv(max_n_segs, 16) * kw * DP_THREADS
    else:
        with_bits = select_layout_total(max_n_segs, max_capacity, max_n_frames, True) * 4
        without = select_layout_total(max_n_segs, max_capacity, max_n_frames, False) * 4
        if with_bits <= optin:
            bits_in_smem, smem = True, with_bits
        elif without <= optin:
            smem = without
        else:
            raise ValueError("select_shots: the generic kernel's rows do not fit shared memory")
        per_sm = occupancy(f"select_generic_kernel<{'true' if bits_in_smem else 'false'}>", smem)
        ws = 0 if bits_in_smem else max_n_segs * cdiv(ncell, 32)
    grid = min(n_videos, sm_count * max(per_sm, 1))
    bits_bytes = max(grid * ws, grid16 * ws16 if kw16 else 0) * 4
    return Plan(k, bits_in_smem, smem, grid, ws, pad_weight, kw16, mk16, smem16, grid16, ws16, front,
                bits_bytes + queue_bytes(n_videos))


def pooling(p: Plan, n_videos, max_n_segs, max_n_frames, method, optin=B200_OPTIN):
    """Pooling route of select_launch when the scores are pooled on the device (not smz_knapsack): 'fused' (inside
    dp16_kernel), 'regular' (pool_regular_kernel), 'smem' (pool_smem_kernel) or 'cursor' (pool_kernel), and the
    number of scores staged per CTA (fused_pool_intervals / max_intervals).  None on the generic path."""
    if p.k == 0:
        return None, 0
    tiles = cdiv(max_n_segs, POOL_THREADS // 8)
    mi = min(max_n_frames + 1, POOL_WORDS)
    if mi + 4 * max_n_segs > POOL_WORDS:
        mi = max(POOL_WORDS - 4 * max_n_segs, 0)
    if tiles > 0 and max_n_segs <= POOL_REGULAR_MAX_SEGS and method == "knapsack" and p.kw16:
        wp = dp16_layout(p.kw16, p.mk16, max_n_segs, p.front_words)[0]
        fmi = min(mi, wp - 4 * max_n_segs)
        if fmi >= 64:
            return "fused", fmi
    if tiles > 0 and max_n_segs <= POOL_REGULAR_MAX_SEGS:
        return "regular", mi
    if tiles > 0 and (max_n_frames + 1) // 2 * 4 <= optin - 1024 and max_n_frames < 65535:
        return "smem", 0
    return "cursor", 0


def fscore_ranges(n_videos, max_n_frames, sm_count):
    """launch_fscore_counts: frame ranges per video (grid.x of fscore_kernel)."""
    chunks = cdiv(max_n_frames, FSCORE_CHUNK)
    per = min(max((n_videos * chunks) // (sm_count * 6 * 4), 1), chunks)
    return cdiv(chunks, per)


def _slices(n_videos):
    return [min(GRID_Y_MAX, n_videos - v0) for v0 in range(0, n_videos, GRID_Y_MAX)]


def launches(p: Plan, api, n_videos, max_n_segs, max_n_frames, method="knapsack", optin=B200_OPTIN,
             sm_count=B200_SMS, user_bits=False) -> List[Launch]:
    """Kernels one library call launches, in stream order.  api: 'select' (smz_select_shots), 'knapsack'
    (smz_knapsack, explicit values), 'evaluate' (smz_eval_batch, annotator rows as floats or, user_bits, as bits) or
    'fscore' (smz_fscore on the mask of an earlier call)."""
    out = []
    if api == "fscore":
        if max_n_frames > 0:
            r = fscore_ranges(n_videos, max_n_frames, sm_count)
            out += [Launch("fscore_kernel", (r, nv, 1)) for nv in _slices(n_videos)]
        return out + [Launch("fscore_final_kernel", (cdiv(n_videos, 128), 1, 1))]
    fused_tail = False
    if p.k == 0:
        out.append(Launch(f"select_generic_kernel<{'true' if p.bits_in_smem else 'false'}>", (p.grid, 1, 1),
                          p.smem_bytes))
    else:
        if api != "knapsack":
            route, mi = pooling(p, n_videos, max_n_segs, max_n_frames, method, optin)
            if route == "regular":
                out += [Launch("pool_regular_kernel", (nv, 1, 1), (mi + 4 * max_n_segs) * 4) for nv in _slices(n_videos)]
            elif route == "smem":
                out.append(Launch("pool_smem_kernel", (n_videos, 1, 1), (max_n_frames + 1) // 2 * 4))
            elif route == "cursor":
                tiles = cdiv(max_n_segs, POOL_THREADS // 8)
                out += [Launch("pool_kernel", (tiles, nv, 1), 0) for nv in _slices(n_videos)]
        og = cdiv(n_videos, 256)
        out += [Launch("order_count_kernel", (og, 1, 1), 0), Launch("order_fill_kernel", (og, 1, 1), 0)]
        if method == "knapsack" and p.kw16:
            out.append(Launch(p.dp16_name(), (p.grid16, 1, 1), p.smem16_bytes))
        out.append(Launch(f"dp_kernel<{p.k}>", (p.grid, 1, 1), p.smem_bytes))
        fused_tail = p.front_words > 0
        if not fused_tail:
            out.append(Launch("summary_kernel", (n_videos, 1, 1), (max_n_segs + 1 + cdiv(max_n_frames, 32)) * 4))
    if api == "evaluate" and not fused_tail:
        if user_bits:
            out.append(Launch("fscore_bits_kernel", (n_videos, 1, 1)))
            out.append(Launch("fscore_final_kernel", (cdiv(n_videos, 128), 1, 1)))
        else:
            out += launches(p, "fscore", n_videos, max_n_segs, max_n_frames, sm_count=sm_count)
    return out


def k_of_capacity(capacity, n_segs=0):
    """dp_kernel's K for a batch whose largest capacity / segment count are given (0: the generic kernel)."""
    need = max(capacity + 1, n_segs)
    return next((K for K in DP_K if K * DP_THREADS >= need), 0)
