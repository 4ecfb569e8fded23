"""oracle/ -- TEST INFRASTRUCTURE, not product code.

CPU restatements of the reference's refinement path used only as checkers by
``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl
reference`` legs of ``bench.py``.  Nothing under ``vision-sr_b200/`` imports this
package; the product path fails loudly when the CUDA extension is missing.

Modules
  vectorised.py   the reference's bfgs() restated over numpy columns, driven by the
                  very same ``scipy.optimize.minimize(method='BFGS')`` call
                  (reference src/visymre/architectures/bfgs.py:42-215).
                  PINNED: checked restart by restart against the unmodified reference
                  (tests/golden/ref_bfgs_*.json, made by oracle/make_golden.py).
  vm.py           a numpy interpreter for the skeleton bytecode, to check the
                  compiler against sympy.lambdify without a GPU.
  ref_harness.py  imports the UNMODIFIED reference from a checkout named by VISYMRE_REFERENCE
                  through inert stubs for packages absent here; used to generate the
                  golden vectors.
  hostsim/        g++ build of the kernels' portable cores (interpreter + BFGS state
                  machine) for logic checks against scipy on the CPU.
"""
