"""test_gpu_wide_puzzle.py once more on precision "f16f8c": the same fp32 dispatch of wide Puzzle tables."""
from suite_loader import clone_suite

globals().update(clone_suite("test_gpu_wide_puzzle", "f16f8c"))
