"""Mesh loading and the CUDA phong renderer (the counterpart of auto_pose/meshrenderer for MODEL: reconst)."""
