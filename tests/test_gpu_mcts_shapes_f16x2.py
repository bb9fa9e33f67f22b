"""test_gpu_mcts_shapes.py once more on precision "f16x2" (every operand split into fp16 hi+lo, 1e-5-grade logits): the
lockstep searches' leaf forwards run on it; the persistent kernel keeps its fp32 arithmetic."""
from suite_loader import clone_suite

globals().update(clone_suite("test_gpu_mcts_shapes", "f16x2"))
