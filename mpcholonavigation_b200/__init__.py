"""B200-native MPPI optimisation loop behind the plugin surface of nav2_sortham_controller.

Only what the hot path needs lives here: ``csrc/`` (hand-written sm_100a CUDA kernels and the C ABI
declared in ``include/mppi_b200.h``) and a thin ctypes binding (``_abi``, ``api``) used by tests and
``bench.py``.  The C++ host side is outside the Python package: ``include/mppi_optimizer.hpp`` (mirror of
``sortham::Optimizer`` over the ABI) and ``shim/`` (the compiled plugin shim: ``sortham::Optimizer``,
``CriticManager`` and the twelve critic plugins with the reference's interfaces).
"""
from . import _abi as abi  # noqa: F401
from .api import (Cycle, Engine, MppiError, Result, circle_footprint, load_product, make_config,  # noqa: F401
                  make_critic, make_robot, optimize_group_device, optimize_sharded)


def MppiOptimizer(**cfg_kw):
    """Engine bound to the CUDA library (raises MppiError if libmppi_b200.so is not built)."""
    return Engine(load_product(), **cfg_kw)
