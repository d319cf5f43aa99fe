"""laser_3d_reconstruction_b200 -- B200 (sm_100a) implementation of the per-frame dense vision hot
path of alo-i-sia/laser_3d_reconstruction behind the reference's Python API (reference
__init__.py:11-24).  Importing the package does not touch the GPU; the first call that does work
loads libl3d.so and raises if it (or a GPU) is missing -- there is no CPU fallback.
"""
from .camera.single_usb_stereo_camera import SingleUSBStereoCameraManager
from .config import Config
from .core.laser_extractor import FastStegerExtractor, SimpleLaserExtractor
from .core.reconstruction import LaserPlaneFit, Reconstructor, fit_laser_plane
from .improved_reconstruction import ImprovedLaserReconstructor, fix_roi_alignment, visualize_laser_depth
from .improved_steger import HybridLaserExtractor, ImprovedStegerExtractor, StegerLaserExtractor
from .system import LaserReconstructionSystem

__version__ = "0.1.0"
__all__ = ["SingleUSBStereoCameraManager", "SimpleLaserExtractor", "FastStegerExtractor", "ImprovedStegerExtractor",
           "StegerLaserExtractor", "HybridLaserExtractor", "Reconstructor", "ImprovedLaserReconstructor",
           "fix_roi_alignment", "visualize_laser_depth", "Config", "LaserReconstructionSystem", "LaserPlaneFit",
           "fit_laser_plane"]
