"""CPU oracle for the filterpy hot path (TEST INFRASTRUCTURE ONLY).

This package restates, in NumPy (and plain C in ``oracle.c``), the algorithms of
the reference's hot path:

* ``filterpy/kalman/kalman_filter.py`` predict / update / batch_filter
* ``filterpy/kalman/UKF.py`` + ``sigma_points.py`` + ``unscented_transform.py``
* ``filterpy/monte_carlo/resampling.py`` systematic / stratified resample

It is the *checker* for the CUDA path, never the product: only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import it.  Nothing under ``filterpy_b200/``
imports it and the product path has no CPU fallback.

Parity pinning: the oracle is pinned against outputs of the unmodified
reference (rlabbe/filterpy 1.4.5 @ 3b51149); the generating script is
``tests/golden/make_golden.py`` and the vectors are committed under
``tests/golden/*.npz``.  ``tests/test_oracle_golden.py`` checks every oracle
function against them.
"""
