"""GPU tests of the training side of the device rollout buffer (fm_buffer.cu: returns, advantages, mini-batch gather).
A package so that the module is ``train_buffer.test_gpu_policy``: module basenames under tests/ would collide otherwise,
and tests/conftest.py runs modules whose name ends in ``test_gpu_policy`` once, not once per simulator mapping (these
kernels do not depend on it)."""
