"""GPU tests of the CTA-per-graph mapping of the fused graph network (gnn_wide_kernel).  A package so that the module is
``policy_wide.test_gpu_policy``: tests/conftest.py runs modules whose name ends in ``test_gpu_policy`` once, not once per
simulator mapping."""
