"""GPU tests of the formation family in the device rollout loop and of its episode statistics.  A package so that the
module is ``formation_loop.test_gpu_formation``: tests/conftest.py runs the formation kernels under one mapping only
for modules whose name ends in ``test_gpu_formation``."""
