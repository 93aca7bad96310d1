"""CPU oracle for the GraphMPE ``navigation_graph`` hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is part of the product:
only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import it, and there only as the checker (or the
thing timed as the CPU baseline) -- never as a fallback for the CUDA path.

What is here
------------
* ``navgraph.py``   float64 numpy restatement of the reference step / reward /
  observation / graph-observation / info / reset path, batched over envs.
  Every function cites the reference file:line it follows.
* ``formation.py``  the formation-family scenarios (SURVEY.md section 8f, N3) restated one env at a time; pinned by
  ``tests/golden/formation_*.npz`` (``make_formation_golden.py``); covers the FA+FR / FA / OA / RA scenario files, walls included.
* ``lexifair.py``   exact solvers for the lexicographic bottleneck ("lexifair")
  assignment of ``marl_fair_assign.py`` (brute force, threshold descent, and a
  HiGHS MILP restatement of the reference's iterative MILP).
* ``philox.py``     numpy Philox4x32-10, the counter RNG the device reset uses.
* ``edges.py``      the policy-side edge list (``process_adj``) restated.
* ``pyg_stub.py``   stand-in for the torch_geometric primitives the reference policy uses, so that the reference's own
  ``GR_Actor`` / ``GR_Critic`` run here as the checker of ``fair_marl_b200.policy`` (``make_policy_golden.py``).
* ``reference_shim.py`` imports the UNMODIFIED reference from the checkout named by
  ``FAIRMARL_REFERENCE_ROOT`` (only where that is set) to pin the restatement and to
  generate ``tests/golden/*.npz`` (``make_golden.py``).

Parity pinning
--------------
The reference ships no tests / golden vectors for this path (SURVEY.md section 4),
and the assignment solve lives in un-vendored pyomo + gurobi.  The restatement
is therefore pinned against *outputs of the reference itself run in the build
container* (``make_golden.py`` -> ``tests/golden``), plus the one fixed
instance in ``marl_fair_assign.py:63-64``.  The lexifair solve itself is
"parity unpinned" w.r.t. Gurobi (not installable); it is pinned against a
HiGHS restatement of the same MILP sequence and brute force.
"""
