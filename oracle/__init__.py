"""CPU oracle for the reverse-SDE enhancement hot path of sp-uhh/sgmse.

TEST INFRASTRUCTURE ONLY.  Nothing under ``sgmse_b200/`` may import this
package: only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` use it, and there only as the checker /
the timed CPU arm, never as the product path.

The oracle is a plain fp32 (optionally fp64) PyTorch-CPU restatement of the
reference algorithm, written functionally against the reference's
``state_dict`` key layout.  Every function cites the reference file:line it
follows.  It is pinned against the live reference (imported from
``/root/reference`` in the build container, see ``oracle/refshim.py``) by

* ``tests/golden/*.npz`` – outputs of the unmodified reference modules, produced
  by ``oracle/make_golden.py`` (committed together with the fixtures): reduced
  configs of all three backbones (forward, score, PC / SB / ODE samplers, the
  enhancement chain, FIR / STFT ops) and ``full_n30.npz``, the reference's own
  full-size N = 30 enhancement of one 4-s clip (BASELINE.json configs[0]), and
* ``tests/test_oracle_vs_reference.py`` – comparison at full size against
  ``tests/golden/reference_live.npz`` (reference outputs and ScoreModel attribute
  skeletons, also from ``oracle/make_golden.py``); only its
  tests that need the reference's ScoreModel class itself run live.

``oracle/ode.py`` additionally restates a third-party algorithm the reference
calls (scipy's RK45); it is pinned to the installed scipy itself.

The reference itself ships no tests or golden vectors (SURVEY.md §4), so these
fixtures are the only pins that exist: parity is pinned to reference outputs
generated here, not to reference-owned test vectors.
"""
