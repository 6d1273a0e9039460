"""CPU oracle for the mseetc.ocp hot path — TEST INFRASTRUCTURE ONLY.

A restatement (numpy / scipy / sympy, FP64) of the NLP that the reference
builds in ``mseetc/ocp.py:80-307`` and hands to CasADi+IPOPT at ``ocp.py:290,359``.
The algorithm that actually solves the NLP in the reference lives in the
un-vendored third-party wheel ``casadi==3.6.3`` (``setup.py:11``; bundles IPOPT 3.14 +
MUMPS), which the reference repository does not contain.  The oracle
therefore restates IPOPT's *published* algorithm (Waechter & Biegler 2006,
"On the implementation of an interior-point filter line-search algorithm for
large-scale nonlinear programming") on the reference's exact variable/row layout.

Parity pins (see ``tests/test_oracle_pins.py``):
  * ``simulations/figure5.py:96``  minimum trip time 272.4726 s (time-optimal mode)
  * ``simulations/figure4.py:22-23`` braking start speeds (ODE restatement)
  * ``simulations/figure3.py:113-115`` static/dynamic loss ratio band
  * ``gpops/00_var_speed_limit_100_GPOPS{I,II}.csv`` energies (discretisation-level)
  * ``unitTests/curvatureResistance/curvatureResistance.py`` properties
No stored vector of an IPOPT optimum exists in the reference, so energy-optimal
parity is pinned only through the items above ("partially pinned").

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import this package.  The product
(``ms-eetc_b200/``) never does.
"""
