"""gpu_quantum_simulator_b200 -- B200 (sm_100a) state-vector path behind the reference's interface.

The package is a thin ctypes mirror of include/qsim_b200.h (the C ABI of
libqsim_b200.so) plus circuit generators for the BASELINE.json workloads.  All
compute happens in the hand-written CUDA library; there is no CPU or PyTorch
fallback -- importing works anywhere, running needs a CUDA device.
"""
from ._lib import lib, QsbError, Gate, MatrixOp, Options, RunStats, F32, F64, MODE_TILED, MODE_SWEEP, MODE_DENSE  # noqa: F401
from .simulator import (Simulator, parse_qasm_file, parse_qasm_string, gates_from_circuit, plan_dry_run, sample_uniform,  # noqa: F401
                        expectation_dry_run, pauli_masks, pauli_rotation_dry_run, rotation_gradient_dry_run,
                        matrix_dry_run)
from . import circuits  # noqa: F401

__all__ = ["Simulator", "parse_qasm_file", "parse_qasm_string", "gates_from_circuit", "plan_dry_run", "sample_uniform",
           "expectation_dry_run", "pauli_masks", "pauli_rotation_dry_run", "rotation_gradient_dry_run",
           "matrix_dry_run", "circuits", "lib", "QsbError", "Gate", "MatrixOp", "Options", "RunStats", "F32", "F64", "MODE_TILED", "MODE_SWEEP", "MODE_DENSE"]
