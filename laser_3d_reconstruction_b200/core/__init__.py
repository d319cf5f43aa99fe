"""Core module (reference core/__init__.py:6-7)."""
from .laser_extractor import FastStegerExtractor, SimpleLaserExtractor
from .reconstruction import LaserPlaneFit, Reconstructor, fit_laser_plane

__all__ = ["SimpleLaserExtractor", "FastStegerExtractor", "Reconstructor", "LaserPlaneFit", "fit_laser_plane"]
