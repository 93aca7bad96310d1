"""GPU tests of the centralised-observation and per-agent critics (critic_head_kernel, the multi-node gather of the fused
graph network, and both critics in RolloutCollector).  A package so that the module is ``critic_cent.test_gpu_policy``:
module basenames under tests/ would collide otherwise, and tests/conftest.py runs modules whose name ends in
``test_gpu_policy`` once, not once per simulator mapping."""
