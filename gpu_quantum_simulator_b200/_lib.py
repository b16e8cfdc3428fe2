"""ctypes binding of libqsim_b200.so (include/qsim_b200.h).  Fails loudly if the library is missing."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_SUFFIX = os.environ.get("QSB_LIB_SUFFIX", "")
# A/B builds (make SUFFIX=_x EXTRA=...) live in csrc/_build_x/, never next to the product library
LIB_PATH = os.path.join(_HERE, "csrc", "_build" + _SUFFIX, "libqsim_b200.so") if _SUFFIX else os.path.join(_HERE, "libqsim_b200.so")

F32, F64 = 32, 64
MODE_TILED, MODE_SWEEP, MODE_DENSE = 0, 1, 2


class QsbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"qsim_b200 error {code}: {msg}")
        self.code = code


class Gate(C.Structure):
    _fields_ = [("controls", C.c_uint64), ("target", C.c_int32), ("flags", C.c_int32), ("m", C.c_double * 8)]


class MatrixOp(C.Structure):
    _fields_ = [("controls", C.c_uint64), ("k", C.c_int32), ("targets", C.c_int32 * 6), ("flags", C.c_int32),
                ("m", C.POINTER(C.c_double))]


class Channel(C.Structure):
    _fields_ = [("k", C.c_int32), ("targets", C.c_int32 * 4), ("nkraus", C.c_int32), ("flags", C.c_int32),
                ("kraus", C.POINTER(C.c_double))]


class Options(C.Structure):
    _fields_ = [("precision", C.c_int32), ("device", C.c_int32), ("mode", C.c_int32), ("tile_bits", C.c_int32),
                ("low_bits", C.c_int32), ("rank", C.c_int32), ("world_size", C.c_int32), ("use_graph", C.c_int32),
                ("verbose", C.c_int32), ("reserved", C.c_int32 * 7)]


class RunStats(C.Structure):
    _fields_ = [("device_ms", C.c_double), ("plan_ms", C.c_double), ("source_gates", C.c_uint64),
                ("device_ops", C.c_uint64), ("passes", C.c_uint32), ("rounds", C.c_uint32), ("swaps", C.c_uint32),
                ("kernel_launches", C.c_uint32), ("bytes_moved", C.c_uint64), ("bytes_exchanged", C.c_uint64),
                ("exchange_ms", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# every symbol include/qsim_b200.h declares (tests/test_abi.py checks the list against the header)
SYMBOLS = {
    "qsb_options_default": (None, [C.POINTER(Options)]),
    "qsb_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(Options)]),
    "qsb_destroy": (None, [C.c_void_p]),
    "qsb_reset": (C.c_int, [C.c_void_p]),
    "qsb_num_qubits": (C.c_int, [C.c_void_p]),
    "qsb_precision": (C.c_int, [C.c_void_p]),
    "qsb_apply_gates": (C.c_int, [C.c_void_p, C.POINTER(Gate), C.c_size_t]),
    "qsb_plan_create": (C.c_int, [C.c_void_p, C.POINTER(Gate), C.c_size_t, C.POINTER(C.c_void_p)]),
    "qsb_execute": (C.c_int, [C.c_void_p, C.c_void_p]),
    "qsb_plan_destroy": (None, [C.c_void_p]),
    "qsb_plan_stats": (C.c_int, [C.c_void_p, C.POINTER(RunStats)]),
    "qsb_last_run_stats": (C.c_int, [C.c_void_p, C.POINTER(RunStats)]),
    "qsb_plan_dry_run": (C.c_int, [C.c_int, C.POINTER(Options), C.POINTER(Gate), C.c_size_t, C.POINTER(RunStats)]),
    "qsb_download": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "qsb_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "qsb_download_physical": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "qsb_get_layout": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "qsb_download_native": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "qsb_norm_argmax": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_double)]),
    "qsb_probabilities": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "qsb_cdf": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "qsb_sample": (C.c_int, [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p]),
    "qsb_sample_uniform": (C.c_double, [C.c_uint64, C.c_int]),
    "qsb_expectation_pauli": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "qsb_pauli_from_string": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "qsb_expectation_dry_run": (C.c_int, [C.c_int, C.POINTER(Options), C.c_void_p, C.c_void_p, C.c_size_t,
                                          C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "qsb_apply_pauli_rotations": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "qsb_pauli_rotation_dry_run": (C.c_int, [C.c_int, C.POINTER(Options), C.c_void_p, C.c_void_p, C.c_size_t,
                                             C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "qsb_apply_matrices": (C.c_int, [C.c_void_p, C.POINTER(MatrixOp), C.c_size_t]),
    "qsb_matrix_dry_run": (C.c_int, [C.c_int, C.POINTER(Options), C.POINTER(MatrixOp), C.c_size_t, C.POINTER(C.c_uint32),
                                     C.POINTER(C.c_uint32)]),
    "qsb_pauli_rotation_gradient": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_double), C.c_void_p]),
    "qsb_pauli_rotation_gradient_dry_run": (C.c_int, [C.c_int, C.POINTER(Options), C.c_void_p, C.c_void_p, C.c_size_t,
                                                      C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_uint32),
                                                      C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "qsb_marginal_probabilities": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "qsb_collapse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.POINTER(C.c_double)]),
    "qsb_measure_qubits": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.POINTER(C.c_uint64),
                                     C.POINTER(C.c_double)]),
    "qsb_reset_qubits": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.POINTER(C.c_uint64)]),
    "qsb_reduced_density_matrix": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "qsb_inner_product": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "qsb_copy_state": (C.c_int, [C.c_void_p, C.c_void_p]),
    "qsb_inner_product_dry_run": (C.c_int, [C.c_int, C.POINTER(Options), C.c_void_p, C.POINTER(Options), C.c_void_p,
                                            C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "qsb_apply_channels": (C.c_int, [C.c_void_p, C.POINTER(Channel), C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "qsb_channel_dry_run": (C.c_int, [C.c_int, C.POINTER(Options), C.POINTER(Channel), C.c_size_t, C.POINTER(C.c_uint32),
                                      C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "qsb_save_state": (C.c_int, [C.c_void_p, C.c_char_p]),
    "qsb_load_state": (C.c_int, [C.c_void_p, C.c_char_p]),
    "qsb_comm_unique_id": (C.c_int, [C.c_void_p]),
    "qsb_comm_init": (C.c_int, [C.c_void_p, C.c_void_p]),
    "qsb_parse_qasm_file": (C.c_int, [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.POINTER(Gate)), C.POINTER(C.c_size_t)]),
    "qsb_parse_qasm_string": (C.c_int, [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.POINTER(Gate)), C.POINTER(C.c_size_t)]),
    "qsb_gate_from_name": (C.c_int, [C.c_char_p, C.POINTER(C.c_double), C.c_int, C.POINTER(C.c_int), C.c_int,
                                     C.POINTER(Gate), C.POINTER(C.c_int)]),
    "qsb_free": (None, [C.c_void_p]),
    "qsb_last_error": (C.c_char_p, []),
    "qsb_version": (C.c_char_p, []),
    "qsb_ref_compute_state_vector": (C.POINTER(C.c_double), [C.c_char_p, C.POINTER(C.c_int)]),
    "qsb_ref_execute_single_qubit_gate": (None, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "qsb_ref_execute_cnot": (None, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "qsb_ref_compute_state_cumulative_distribution": (C.POINTER(C.c_double), [C.c_void_p, C.c_int]),
    "qsb_ref_measurement": (C.c_longlong, [C.c_void_p, C.c_int]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C gpu_quantum_simulator_b200/csrc`). There is no fallback path.")
    L = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        f = getattr(L, name)
        f.restype = res
        f.argtypes = args
    return L


lib = _load()


def check(rc):
    if rc != 0:
        raise QsbError(rc, lib.qsb_last_error().decode("utf-8", "replace"))
