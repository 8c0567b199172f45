"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the caption-decoder hot path.

Nothing in the product package (``image-caption-emotion-indonesia_b200/``) may import
this package.  Only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` use it, and only as the
checker / the CPU baseline, never as the thing shipped.

Parity pin status: the reference repository has NO tests, golden vectors or
fixtures for this path (SURVEY.md section 8c: "parity unpinned" by the reference's own
tests).  The oracle is instead pinned against outputs of the reference modules
themselves, executed by ``oracle/make_golden.py`` and committed under
``tests/golden/``; ``tests/test_oracle_pin.py`` re-checks the port against those
vectors (and against the live reference when ``SN_REFERENCE_ROOT`` names a checkout
of the original project).
"""
