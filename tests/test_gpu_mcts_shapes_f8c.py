"""test_gpu_mcts_shapes.py once more on precision "f16f8c" (the two correction products as fp8 MMAs, 1e-3 grade): the
lockstep searches' leaf forwards run on it; the persistent kernel keeps its fp32 arithmetic."""
from suite_loader import clone_suite

globals().update(clone_suite("test_gpu_mcts_shapes", "f16f8c"))
