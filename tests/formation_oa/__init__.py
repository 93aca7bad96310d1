"""GPU tests of the optimal-assignment formation scenario (OA) at 6 and 7 agents.  A package so that the module is
``formation_oa.test_gpu_formation``: tests/conftest.py runs the formation kernels under one mapping only for modules whose
name ends in ``test_gpu_formation``."""
