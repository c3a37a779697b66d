"""CPU oracle for the numbskull hot path -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import this package.  The product
package ``numbskull_b200`` never does.
"""
from .oracle import OracleGraph, build, lib, exact_marginals, compute_var_map  # noqa: F401
from . import oracle as rng  # noqa: F401,E402  (Philox streams and draw rules: oracle.rng.*)
from . import coloring  # noqa: F401,E402
