"""test_gpu_wide_puzzle.py once more on precision "f16x2": wide Puzzle tables must still take the fp32 kernel on a
tensor-core engine, and a 625-row GridWorld the pair kernel."""
from suite_loader import clone_suite

globals().update(clone_suite("test_gpu_wide_puzzle", "f16x2"))
