"""test_gpu_mcts_twists.py once more on precision "f16x2w16" (the common weight as one fp16 term, 1e-3 grade): the lockstep
search's leaf forwards run on it; the persistent kernel keeps its fp32 arithmetic."""
from suite_loader import clone_suite

globals().update(clone_suite("test_gpu_mcts_twists", "f16x2w16"))
