"""rustsasa_b200 -- B200 (sm_100a) Shrake-Rupley engine behind RustSASA's hot-path interface.

The product is ``libsasa_b200.so`` (hand-written CUDA + a C ABI, include/sasa_b200.h).  This package is
the thin Python host layer used by the tests and the benchmark: a ctypes binding (``_lib``), an
Engine / Batch wrapper (``engine``) and a mirror of the reference's public interface for the path
(``api``: ``calculate_sasa_internal``, ``SASAOptions`` ...).  There is no CPU fallback.
"""
from .api import (Atom, AtomLevel, ChainLevel, ChainResult, GroupPairResult, InterfacePairsResult,  # noqa: F401
                  InterfaceResult, InterfaceSurfaceResult, ProteinLevel, ProteinResult, ResidueLevel, ResidueResult, SASACalcError, SASAOptions, SurfaceResult,
                  TrajectoryInterfaceResult, calculate_sasa_internal, default_engine, surface_points, trajectory_interface)
from .engine import Batch, BatchResult, Engine, PairResult, PairSums, SasaB200Error, group_pair_table  # noqa: F401
from .structure import read_structure  # noqa: F401

__all__ = ["Atom", "AtomLevel", "ResidueLevel", "ChainLevel", "ProteinLevel", "ChainResult", "ResidueResult",
           "ProteinResult", "SASACalcError", "SASAOptions", "SurfaceResult", "InterfaceResult", "InterfaceSurfaceResult",
           "GroupPairResult", "InterfacePairsResult", "TrajectoryInterfaceResult", "calculate_sasa_internal", "default_engine",
           "surface_points", "trajectory_interface", "Engine",
           "Batch", "BatchResult", "PairResult", "PairSums", "SasaB200Error", "group_pair_table", "read_structure"]
