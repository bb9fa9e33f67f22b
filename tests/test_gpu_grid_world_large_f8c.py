"""test_gpu_grid_world_large.py once more on precision "f16f8c": GridWorld forwards of 33..64 cells on the pair kernel."""
from suite_loader import clone_suite

globals().update(clone_suite("test_gpu_grid_world_large", "f16f8c"))
