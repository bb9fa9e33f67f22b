"""test_gpu_wide_puzzle.py once more on precision "f16x2w16": the same fp32 dispatch of wide Puzzle tables."""
from suite_loader import clone_suite

globals().update(clone_suite("test_gpu_wide_puzzle", "f16x2w16"))
