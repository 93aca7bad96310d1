"""GPU tests of the formation kernels' in-kernel lexifair solvers on exactly tied costs.  A package so that the module is
``formation_ties.test_gpu_formation``: tests/conftest.py runs the formation kernels under one mapping only for modules whose
name ends in ``test_gpu_formation``."""
