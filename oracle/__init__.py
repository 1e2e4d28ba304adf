"""ORACLE — test infrastructure, not product code.

CPU restatement of the reference's algorithm for the PCG hot path (``uibk/deep_preconditioning/cg.py``,
``test.py:61-68,100-109``, ``utils.py:15-43``, ``model.py:53-57``). Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may import it,
and only as the checker or the timed CPU baseline — never from ``deeppreconditioning_b200``.

Pinning status
--------------
* ``oracle.pcg`` (the loop, ``cg.py:15-90``): pinned against the iteration counts the reference function itself
  produced on the same operands (``tests/golden/pcg_golden.json``, made by ``tests/golden/make_golden.py``;
  ``tests/test_oracle.py::test_oracle_matches_reference_golden``).
* ``oracle.sparse.sparse_matvec_mul`` (``utils.py:15-43``): pinned by the reference's own known-answer test
  (``tests/test_utils.py:11-41``).
* ``oracle.sparse`` assembly (``test.py:61-68,100-105``): pinned against ``torch.Tensor.to_sparse_csr`` /
  dense arithmetic, which is literally what the reference executes.
* SpTRSV / level sets: the reference has none (SURVEY D1) — pinned against scipy ``spsolve_triangular``.
* ``oracle.pcg`` at the BASELINE sizes: ``tests/golden/pcg_spread.json`` holds the iteration counts of the unmodified
  reference on 316^2 and 128^3 operands under every thread count / storage / form of ``M`` it may be run with
  (``tests/golden/make_spread.py``); the oracle's count is inside that band (``tests/test_gpu_parity.py``).
* ``oracle.metrics`` (``metrics.py:13-77``): pinned against the values the reference module produced, imported
  unmodified (``tests/golden/metrics_golden.json``, ``tests/test_oracle.py::test_metrics_oracle_matches_golden``).
* IC(0) / ICT: ``ilupp`` 1.0.2 is absent — **parity unpinned** for values; for IC(0) the pattern and the defining
  property ``(L L^T)_ij = A_ij`` on the pattern are tested, for ``oracle.icholt`` (a restatement of the published
  ICT(p, tau) scheme, not of ilupp's source) the dropping rules, the complete-factorisation limit and its use as a
  preconditioner.
* CNN values (spconv 2.3.8 absent): **parity unpinned**; structural properties of
  ``tests/test_model.py:31-42`` are tested.
"""
