"""CPU oracle for the genrec hot path (HSTU block, SASRec attention, RQ-VAE residual argmin).

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is imported by the product
package ``genrec_b200``.  The only legitimate importers are ``tests/``,
``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference`` legs
of ``bench.py`` - and there only as the checker / the CPU arm, never as the thing
that is shipped or measured as "ours".

What it is: a plain-PyTorch (CPU, fp32/fp64) restatement of the reference
algorithm, every function citing the ``/root/reference`` file:line it follows,
plus a C restatement of the RQ-VAE distance+argmin (``rq_argmin.c``).

Pinning: the reference (phonism/genrec @ b0272248) ships NO tests and NO golden
vectors for this path (SURVEY.md section 4), so the oracle is pinned against
outputs of the reference modules themselves, imported in the build container
from ``/root/reference`` by ``oracle/make_golden.py``; the resulting fixtures
are committed under ``tests/golden/`` and checked by
``tests/test_oracle_golden.py``.
"""
