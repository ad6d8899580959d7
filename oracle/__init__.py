"""TEST INFRASTRUCTURE ONLY — CPU restatement ("oracle") of the reference hot path.

Nothing under ``oracle/`` is part of the product.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference``
legs may import it, and there only as the checker or the timed CPU baseline.
The product package (``summarizer_b200``) never imports this package and fails
loudly when its CUDA library is missing.

Parity status (see DESIGN.md "Oracle"):
  * eval path (upsample, segment pooling, summary vector, F-score): pinned
    against the reference's own Python, imported unmodified from
    a checkout named by $SMZ_REFERENCE_ROOT (``oracle/ref_import.py``), with
    golden vectors committed under ``tests/golden/``.
  * knapsack selection under ties: **parity unpinned** — the algorithm lives in
    the third-party dependency ``ortools==7.5.7466`` (summarizer/requirements.txt:11,
    ``ortools/algorithms/knapsack_solver.cc``), which the reference does not
    vendor.  The restatement follows the published
    algorithm; optimal profit and feasibility are pinned against brute force.
  * VASNet / DSN scorers: pinned against the reference ``nn.Module``s imported
    unmodified (golden vectors under ``tests/golden/``).
"""
