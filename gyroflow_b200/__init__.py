"""gyroflow_b200 — B200 (sm_100a) backend for Gyroflow's per-pixel stabilization warp.

Product code = gyroflow_b200/csrc (CUDA kernels + extern "C" ABI, built into libgyroflow_cuda.so).
This package is the thin host-side mirror used by tests and bench.py.
"""
from . import abi
from .abi import KernelParams, BackendMissing, load_library
from .backend import (BufferDescription, Buffers, FrameTransform, ProcessedInfo, CudaWrapper,
                      GyroflowCoreError, list_devices, ComputeParams, DeviceGyro, zoom_dynamic,
                      scan_tables_dev, bind_thread_to_device, stab_config, get_frame_transform_at, host_register, host_unregister,
                      frame_layout, background_for_plane)
from .render_queue import RenderQueue, FrameRenderQueue

__all__ = ["abi", "KernelParams", "BackendMissing", "load_library", "BufferDescription", "Buffers", "FrameTransform",
           "ProcessedInfo", "CudaWrapper", "GyroflowCoreError", "list_devices", "ComputeParams", "DeviceGyro", "zoom_dynamic",
           "scan_tables_dev", "bind_thread_to_device", "stab_config", "get_frame_transform_at", "RenderQueue", "host_register", "host_unregister",
           "FrameRenderQueue", "frame_layout", "background_for_plane"]
