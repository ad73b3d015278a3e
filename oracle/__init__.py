"""CPU oracle bindings (TEST INFRASTRUCTURE ONLY).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this package.  The product (deeppowers_b200/) never does.

PARITY UNPINNED: the reference has no implementation of this path (SURVEY.md §0, §8c);
the oracle restates DESIGN.md §2 and is pinned by its own known-answer tests.
"""
from .binding import Oracle, lib, build, build_ref  # noqa: F401
