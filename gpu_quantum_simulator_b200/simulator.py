"""Host-side mirror of the reference interface for the state-vector path.

`Simulator` wraps one qsb_t handle.  The method names follow the functions of
/root/reference/quantum_simulator.c they stand in for:
    compute_state_vector(file)                 :115-254
    execute_single_qubit_gate(U, target)       :81-92   (same U[4] indexing as the reference)
    execute_cnot(control, target)              :94-106
    compute_state_cumulative_distribution()    :256-268
    measurement(shots, seed)                   :270-283
"""
import ctypes as C
import os

import numpy as np

from ._lib import lib, check, Gate, MatrixOp, Channel, Options, RunStats, F32, F64, MODE_TILED, MODE_SWEEP


def _gate_array(gates):
    if isinstance(gates, C.Array):
        return gates, len(gates)
    arr = (Gate * max(len(gates), 1))()
    for i, g in enumerate(gates):
        arr[i] = g
    return arr, len(gates)


def parse_qasm_file(path):
    """-> (num_qubits, ctypes array of Gate)"""
    nq = C.c_int()
    gp = C.POINTER(Gate)()
    n = C.c_size_t()
    check(lib.qsb_parse_qasm_file(str(path).encode(), C.byref(nq), C.byref(gp), C.byref(n)))
    arr = (Gate * max(n.value, 1))()
    C.memmove(arr, gp, C.sizeof(Gate) * n.value)
    lib.qsb_free(gp)
    return nq.value, (Gate * n.value).from_buffer(arr) if n.value else (Gate * 0)()


def parse_qasm_string(text):
    nq = C.c_int()
    gp = C.POINTER(Gate)()
    n = C.c_size_t()
    check(lib.qsb_parse_qasm_string(text.encode(), C.byref(nq), C.byref(gp), C.byref(n)))
    arr = (Gate * max(n.value, 1))()
    C.memmove(arr, gp, C.sizeof(Gate) * n.value)
    lib.qsb_free(gp)
    return nq.value, (Gate * n.value).from_buffer(arr) if n.value else (Gate * 0)()


def gates_from_circuit(circ):
    """circ: iterable of (name, qubits, params) -> ctypes array of Gate (via qsb_gate_from_name)."""
    out = []
    tmp = (Gate * 3)()
    k = C.c_int()
    for name, qubits, params in circ:
        p = (C.c_double * max(len(params), 1))(*params)
        q = (C.c_int * max(len(qubits), 1))(*qubits)
        check(lib.qsb_gate_from_name(name.encode(), p, len(params), q, len(qubits), tmp, C.byref(k)))
        for i in range(k.value):
            g = Gate()
            C.memmove(C.byref(g), C.byref(tmp[i]), C.sizeof(Gate))
            out.append(g)
    arr = (Gate * max(len(out), 1))()
    for i, g in enumerate(out):
        arr[i] = g
    return (Gate * len(out)).from_buffer(arr) if out else (Gate * 0)()


def _options(precision, mode, low_bits, rank, world_size, device, reserved=None, use_graph=False, dense_k=0):
    """reserved: planner tuning knobs (qsb_options_t.reserved): [0] min gates before a qubit exchange,
    [1] 2 = lazy diagonals on, [2] k+1 = trim tail rounds with < k gates (1 = off), [3] fusion-depth cost cap,
    [4] gate rewrites (5 = CX between two h / two rx left alone, 6 = CX -> controlled phase with an h on one side too),
    [5] exchange flavour, [6] 2 = first-come tiles, 3 / 4 = no / conflicts-only lane relocation; the full list is in
    include/qsim_b200.h.  Knobs left at 0 are searched by the library where it plans several candidates."""
    o = Options()
    lib.qsb_options_default(C.byref(o))
    for k, v in enumerate(reserved or ()):
        o.reserved[k] = int(v)
    o.precision = precision
    o.mode = mode
    o.low_bits = low_bits
    o.rank = rank
    o.world_size = world_size
    o.device = device
    o.use_graph = 1 if use_graph else 0
    o.tile_bits = dense_k          # MODE_DENSE: fusion width k (2..5)
    return o


def plan_dry_run(num_qubits, gates, precision=F32, low_bits=0, world_size=1, rank=0, reserved=None, mode=MODE_TILED, dense_k=0):
    """Host-only scheduling statistics (no GPU needed)."""
    arr, n = _gate_array(gates)
    o = _options(precision, mode, low_bits, rank, world_size, -1, reserved, False, dense_k)
    st = RunStats()
    check(lib.qsb_plan_dry_run(num_qubits, C.byref(o), arr, n, C.byref(st)))
    return st.as_dict()


def pauli_masks(paulis, num_qubits):
    """A Pauli string ("X0 Z3 Y5"; "" or "I" = identity) or a list of them -> (x, z) uint64 arrays of logical
    masks.  The format is defined once, in qsb_pauli_from_string."""
    texts = [paulis] if isinstance(paulis, str) else list(paulis)
    x = np.zeros(len(texts), dtype=np.uint64)
    z = np.zeros(len(texts), dtype=np.uint64)
    xm, zm = C.c_uint64(), C.c_uint64()
    for k, t in enumerate(texts):
        check(lib.qsb_pauli_from_string(t.encode(), num_qubits, C.byref(xm), C.byref(zm)))
        x[k], z[k] = xm.value, zm.value
    return x, z


def expectation_dry_run(num_qubits, paulis, precision=F32, world_size=1):
    """Host-only: {"sweeps", "exchanges"} that Simulator.expectation would run for these Pauli strings from the
    identity qubit layout (sweeps = reads of the local shard, exchanges = partner shards fetched)."""
    x, z = pauli_masks(paulis, num_qubits)
    o = _options(precision, MODE_TILED, 0, 0, world_size, -1)
    sw, ex = C.c_uint32(), C.c_uint32()
    check(lib.qsb_expectation_dry_run(num_qubits, C.byref(o), x.ctypes.data, z.ctypes.data, x.size, C.byref(sw), C.byref(ex)))
    return {"sweeps": sw.value, "exchanges": ex.value}


def pauli_rotation_dry_run(num_qubits, paulis, precision=F32, world_size=1, low_bits=0):
    """Host-only: {"sweeps", "exchanges"} that Simulator.apply_pauli_rotations would run for these Pauli strings (all
    angles taken non-zero) from the identity qubit layout (sweeps = reads and writes of the local shard, exchanges =
    partner shards fetched, one per sweep that flips rank qubits)."""
    x, z = pauli_masks(paulis, num_qubits)
    o = _options(precision, MODE_TILED, low_bits, 0, world_size, -1)
    sw, ex = C.c_uint32(), C.c_uint32()
    check(lib.qsb_pauli_rotation_dry_run(num_qubits, C.byref(o), x.ctypes.data, z.ctypes.data, x.size, C.byref(sw), C.byref(ex)))
    return {"sweeps": sw.value, "exchanges": ex.value}


def rotation_gradient_dry_run(num_qubits, paulis, observable, precision=F32, world_size=1, low_bits=0):
    """Host-only: {"apply_sweeps", "adjoint_sweeps", "exchanges"} that Simulator.rotation_gradient would run besides
    its forward pass and energy, from the identity qubit layout with every angle taken non-zero (apply_sweeps build
    H psi, adjoint_sweeps walk the rotations backwards, exchanges = partner shards fetched by both)."""
    x, z = pauli_masks(paulis, num_qubits)
    hx, hz = pauli_masks(observable, num_qubits)
    o = _options(precision, MODE_TILED, low_bits, 0, world_size, -1)
    ap, ad, ex = C.c_uint32(), C.c_uint32(), C.c_uint32()
    check(lib.qsb_pauli_rotation_gradient_dry_run(num_qubits, C.byref(o), x.ctypes.data, z.ctypes.data, x.size, hx.ctypes.data,
                                                  hz.ctypes.data, hx.size, C.byref(ap), C.byref(ad), C.byref(ex)))
    return {"apply_sweeps": ap.value, "adjoint_sweeps": ad.value, "exchanges": ex.value}


def _matrix_ops(ops, num_qubits=None):
    """[(U, qubits) or (U, qubits, controls)] -> (ctypes array of MatrixOp, the numpy buffers its pointers address).
    U is None in a dry run (only shapes are read); otherwise a (2^k, 2^k) complex array."""
    arr = (MatrixOp * max(len(ops), 1))()
    keep = []
    for i, op in enumerate(ops):
        U, qubits = op[0], [int(x) for x in np.atleast_1d(op[1])]
        controls = [int(x) for x in np.atleast_1d(op[2])] if len(op) > 2 else []
        if len(qubits) > 6:
            raise ValueError(f"op {i}: {len(qubits)} targets, at most 6")
        o = arr[i]
        o.k = len(qubits)
        for j, x in enumerate(qubits):
            o.targets[j] = x
        for c in controls:
            if not 0 <= c < 64:
                raise ValueError(f"op {i}: control {c} outside [0, 64)")
            o.controls |= 1 << c
        if U is not None:
            d = 1 << len(qubits)
            m = np.ascontiguousarray(np.asarray(U, dtype=np.complex128))
            if m.shape != (d, d):
                raise ValueError(f"op {i}: matrix of shape {m.shape} for {len(qubits)} targets, expected ({d}, {d})")
            keep.append(m)
            o.m = m.view(np.float64).ctypes.data_as(C.POINTER(C.c_double))
    return arr, keep


def matrix_dry_run(num_qubits, shapes, precision=F32, world_size=1, low_bits=0):
    """Host-only: {"sweeps", "exchanges"} that Simulator.apply_matrices would run for ops of these shapes from the
    identity qubit layout.  shapes: a list of target lists, or of (targets, controls) pairs (sweeps = reads and writes of
    the local shard, exchanges = partner shards fetched, one per sweep with a target on a rank qubit)."""
    ops = []
    for sh in shapes:
        if len(sh) == 2 and not np.isscalar(sh[0]):
            ops.append((None, sh[0], sh[1]))
        else:
            ops.append((None, sh))
    arr, _ = _matrix_ops(ops)
    o = _options(precision, MODE_TILED, low_bits, 0, world_size, -1)
    sw, ex = C.c_uint32(), C.c_uint32()
    check(lib.qsb_matrix_dry_run(num_qubits, C.byref(o), arr, len(ops), C.byref(sw), C.byref(ex)))
    return {"sweeps": sw.value, "exchanges": ex.value}


def overlap_dry_run(num_qubits, perm_a, perm_b, precision_a=F32, precision_b=F32, world_size=1, rank=0, low_bits_a=0,
                    low_bits_b=0):
    """Host-only: {"steps", "exchanges"} that Simulator.overlap would run on `rank` for handles with these qubit layouts
    (perm[q] = physical bit of qubit q, the format of Simulator.layout; bits >= the local bits are rank bits): steps =
    partner shards of the other state combined, exchanges = those that are copied from another rank."""
    pa = np.zeros(64, dtype=np.int8)
    pb = np.zeros(64, dtype=np.int8)
    pa[:num_qubits] = np.asarray(perm_a, dtype=np.int64)[:num_qubits]
    pb[:num_qubits] = np.asarray(perm_b, dtype=np.int64)[:num_qubits]
    oa = _options(precision_a, MODE_TILED, low_bits_a, rank, world_size, -1)
    ob = _options(precision_b, MODE_TILED, low_bits_b, rank, world_size, -1)
    st, ex = C.c_uint32(), C.c_uint32()
    check(lib.qsb_inner_product_dry_run(num_qubits, C.byref(oa), pa.ctypes.data, C.byref(ob), pb.ctypes.data, C.byref(st),
                                        C.byref(ex)))
    return {"steps": st.value, "exchanges": ex.value}


def _channels(channels):
    """[(kraus_list, qubits)] -> (ctypes array of Channel, the numpy buffers its pointers address).  kraus_list is None in
    a dry run (the channel is then taken as state-dependent); otherwise a list of (2^k, 2^k) complex arrays."""
    arr = (Channel * max(len(channels), 1))()
    keep = []
    for i, (kraus, qubits) in enumerate(channels):
        qubits = [int(x) for x in np.atleast_1d(qubits)]
        if len(qubits) > 4:
            raise ValueError(f"channel {i}: {len(qubits)} targets, at most 4")
        c = arr[i]
        c.k = len(qubits)
        for j, x in enumerate(qubits):
            c.targets[j] = x
        if kraus is None:
            c.nkraus = 1                        # shapes only: the count is checked, the operators are not read
            continue
        d = 1 << len(qubits)
        ks = np.ascontiguousarray(np.asarray(kraus, dtype=np.complex128))
        if ks.ndim != 3 or ks.shape[1:] != (d, d):
            raise ValueError(f"channel {i}: Kraus operators of shape {ks.shape} for {len(qubits)} targets, expected (m, {d}, {d})")
        c.nkraus = ks.shape[0]
        keep.append(ks)
        c.kraus = ks.view(np.float64).ctypes.data_as(C.POINTER(C.c_double))
    return arr, keep


def channel_dry_run(num_qubits, channels, precision=F32, world_size=1, low_bits=0):
    """Host-only: {"sweeps", "gram_sweeps", "exchanges"} that Simulator.apply_channels would run for these channels from the
    identity qubit layout, counting every branch as a non-identity operator (an upper bound): sweeps = launches that read
    and write the local shard, gram_sweeps = launches that only read it, exchanges = partner shards fetched.  channels:
    (kraus_list, qubits) tuples as for apply_channels; kraus_list may be None (taken as state-dependent), and a qubit list
    that is not a tuple stands for (None, qubits)."""
    chs = [c if isinstance(c, tuple) else (None, c) for c in channels]
    arr, keep = _channels(chs)
    o = _options(precision, MODE_TILED, low_bits, 0, world_size, -1)
    sw, gs, ex = C.c_uint32(), C.c_uint32(), C.c_uint32()
    check(lib.qsb_channel_dry_run(num_qubits, C.byref(o), arr, len(chs), C.byref(sw), C.byref(gs), C.byref(ex)))
    del keep
    return {"sweeps": sw.value, "gram_sweeps": gs.value, "exchanges": ex.value}


_PAULI = [np.eye(2, dtype=np.complex128), np.array([[0, 1], [1, 0]], dtype=np.complex128),
          np.array([[0, -1j], [1j, 0]], dtype=np.complex128), np.array([[1, 0], [0, -1]], dtype=np.complex128)]


def depolarizing(p, k=1):
    """Kraus operators of the k-qubit depolarizing channel rho -> (1 - p) rho + p I / 2^k (k = 1 or 2): sqrt(1 - p (4^k - 1)
    / 4^k) I and sqrt(p / 4^k) P for every other Pauli product P (bit i of an index = qubit i of the channel's list)."""
    if k not in (1, 2):
        raise ValueError(f"depolarizing: k = {k}, expected 1 or 2")
    d2 = 4 ** k
    ops = []
    for idx in range(d2):
        P = np.ones((1, 1), dtype=np.complex128)
        for j in range(k):                      # qubit j is bit j of the index: kron(P_{k-1}, ..., P_0)
            P = np.kron(_PAULI[(idx >> (2 * j)) & 3], P)
        ops.append(P * np.sqrt(1.0 - p * (d2 - 1) / d2 if idx == 0 else p / d2))
    return ops


def pauli_channel(px, py, pz):
    """Kraus operators of rho -> (1 - px - py - pz) rho + px X rho X + py Y rho Y + pz Z rho Z."""
    return [np.sqrt(1.0 - px - py - pz) * _PAULI[0], np.sqrt(px) * _PAULI[1], np.sqrt(py) * _PAULI[2], np.sqrt(pz) * _PAULI[3]]


def amplitude_damping(gamma):
    """Kraus operators of amplitude damping: [[1, 0], [0, sqrt(1 - gamma)]] and [[0, sqrt(gamma)], [0, 0]]."""
    return [np.array([[1, 0], [0, np.sqrt(1.0 - gamma)]], dtype=np.complex128),
            np.array([[0, np.sqrt(gamma)], [0, 0]], dtype=np.complex128)]


def phase_damping(lam):
    """Kraus operators of phase damping: [[1, 0], [0, sqrt(1 - lam)]] and [[0, 0], [0, sqrt(lam)]]."""
    return [np.array([[1, 0], [0, np.sqrt(1.0 - lam)]], dtype=np.complex128),
            np.array([[0, 0], [0, np.sqrt(lam)]], dtype=np.complex128)]


class Plan:
    def __init__(self, sim, handle):
        self.sim, self.handle = sim, handle

    def stats(self):
        st = RunStats()
        check(lib.qsb_plan_stats(self.handle, C.byref(st)))
        return st.as_dict()

    def close(self):
        if self.handle:
            lib.qsb_plan_destroy(self.handle)
            self.handle = None

    __del__ = close


class Simulator:
    def __init__(self, num_qubits, precision=F32, mode=MODE_TILED, low_bits=0, rank=0, world_size=1, device=-1, reserved=None,
                 use_graph=False, dense_k=0):
        self._h = C.c_void_p()
        o = _options(precision, mode, low_bits, rank, world_size, device, reserved, use_graph, dense_k)
        check(lib.qsb_create(C.byref(self._h), num_qubits, C.byref(o)))
        self.num_qubits, self.precision = num_qubits, precision
        self.rank, self.world_size = rank, world_size

    # ---- lifecycle
    def close(self):
        if getattr(self, "_h", None):
            lib.qsb_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def reset(self):
        check(lib.qsb_reset(self._h))

    # ---- hot path
    def apply(self, gates):
        arr, n = _gate_array(gates)
        check(lib.qsb_apply_gates(self._h, arr, n))
        return self.last_stats()

    def plan(self, gates):
        arr, n = _gate_array(gates)
        p = C.c_void_p()
        check(lib.qsb_plan_create(self._h, arr, n, C.byref(p)))
        return Plan(self, p)

    def execute(self, plan):
        check(lib.qsb_execute(self._h, plan.handle))
        return self.last_stats()

    def last_stats(self):
        st = RunStats()
        check(lib.qsb_last_run_stats(self._h, C.byref(st)))
        return st.as_dict()

    # ---- reference-named operations
    def execute_single_qubit_gate(self, U, target):
        """U: 4 complex numbers indexed as the reference does: v0' = v0*U[0] + v1*U[2] (quantum_simulator.c:88)."""
        U = np.asarray(U, dtype=np.complex128).reshape(4)
        g = Gate()
        g.target = target
        m = [U[0], U[2], U[1], U[3]]
        for k in range(4):
            g.m[2 * k], g.m[2 * k + 1] = m[k].real, m[k].imag
        return self.apply([g])

    def execute_cnot(self, control, target):
        g = Gate()
        g.controls, g.target = 1 << control, target
        g.m[2] = 1.0
        g.m[4] = 1.0
        return self.apply([g])

    def compute_state_vector(self, path):
        nq, gates = parse_qasm_file(path)
        if nq != self.num_qubits:
            raise ValueError(f"circuit declares {nq} qubits, simulator has {self.num_qubits}")
        self.reset()
        self.apply(gates)
        return self.state()

    # ---- readout
    def _own_range(self):
        n = 1 << self.num_qubits
        return 0, n

    def state(self, first=0, count=None):
        """complex128 amplitudes in logical order."""
        if count is None:
            count = (1 << self.num_qubits) - first
        out = np.empty(2 * count, dtype=np.float64)
        check(lib.qsb_download(self._h, out.ctypes.data, first, count))
        return out.view(np.complex128)

    def state_native(self, first=0, count=None, out=None):
        if count is None:
            count = (1 << self.num_qubits) - first
        dt = np.float32 if self.precision == F32 else np.float64
        if out is None:
            out = np.empty(2 * count, dtype=dt)
        check(lib.qsb_download_native(self._h, out.ctypes.data, first, count))
        return out

    def layout(self):
        """-> (perm, nloc): perm[q] = physical index bit of logical qubit q; bits >= nloc are rank bits."""
        perm = np.zeros(64, dtype=np.int8)
        nloc = C.c_int()
        check(lib.qsb_get_layout(self._h, perm.ctypes.data, C.byref(nloc)))
        return perm, nloc.value

    def shard_physical(self):
        """The local shard exactly as stored (physical index order), complex128."""
        _, nloc = self.layout()
        out = np.empty(2 << nloc, dtype=np.float64)
        check(lib.qsb_download_physical(self._h, out.ctypes.data, 0, 1 << nloc))
        return out.view(np.complex128)

    def shard_head(self, count, out=None):
        """The first `count` amplitudes of the local shard in physical order, as float64 (re, im) pairs."""
        if out is None:
            out = np.empty(2 * count, dtype=np.float64)
        check(lib.qsb_download_physical(self._h, out.ctypes.data, 0, count))
        return out

    def set_state(self, amps, first=0):
        a = np.ascontiguousarray(np.asarray(amps, dtype=np.complex128))
        check(lib.qsb_upload(self._h, a.view(np.float64).ctypes.data, first, a.size))

    def norm_argmax(self):
        norm, idx, p = C.c_double(), C.c_uint64(), C.c_double()
        check(lib.qsb_norm_argmax(self._h, C.byref(norm), C.byref(idx), C.byref(p)))
        return norm.value, idx.value, p.value

    def probabilities(self, first=0, count=None):
        if count is None:
            count = (1 << self.num_qubits) - first
        out = np.empty(count, dtype=np.float64)
        check(lib.qsb_probabilities(self._h, out.ctypes.data, first, count))
        return out

    def compute_state_cumulative_distribution(self, first=0, count=None):
        if count is None:
            count = (1 << self.num_qubits) - first
        out = np.empty(count, dtype=np.float64)
        check(lib.qsb_cdf(self._h, out.ctypes.data, first, count))
        return out

    def measurement(self, shots, seed=0):
        out = np.empty(shots, dtype=np.uint64)
        check(lib.qsb_sample(self._h, seed, shots, out.ctypes.data))
        return out

    def expectation(self, paulis):
        """<psi|P|psi> of a Pauli string ("Z0 Z1", "X0 Y2", "" = identity) as a float, or of a list of them as a
        float64 array, computed on the device without copying the state out.  On a sharded state every rank calls
        it with the same strings and receives every value."""
        x, z = pauli_masks(paulis, self.num_qubits)
        out = np.empty(x.size, dtype=np.float64)
        check(lib.qsb_expectation_pauli(self._h, x.ctypes.data, z.ctypes.data, x.size, out.ctypes.data))
        return float(out[0]) if isinstance(paulis, str) else out

    # ---- Pauli rotations
    def apply_pauli_rotations(self, paulis, thetas):
        """Apply exp(-i theta_k P_k / 2) = cos(theta_k / 2) I - i sin(theta_k / 2) P_k for a Pauli string ("X0 Z3") and an
        angle, or for a list of strings and a list of angles, in list order (the first acts first), on the device.  The
        qubit layout is left as it is; theta = 0 leaves the state untouched.  Sharded: collective, same arguments on every
        rank."""
        x, z = pauli_masks(paulis, self.num_qubits)
        t = np.ascontiguousarray(np.asarray(thetas, dtype=np.float64).reshape(-1))
        if t.size != x.size:
            raise ValueError(f"{x.size} Pauli strings but {t.size} angles")
        check(lib.qsb_apply_pauli_rotations(self._h, x.ctypes.data, z.ctypes.data, t.ctypes.data, x.size))

    def evolve(self, paulis, coeffs, time, steps, order=1):
        """exp(-i H time) for H = sum_k coeffs[k] P_k by a Trotter product of `steps` steps, sent as one call.
        order=1: each step is prod_k exp(-i c_k dt P_k) in list order (theta_k = 2 c_k dt, dt = time / steps);
        order=2: the symmetric step, the list forward with dt / 2 and then backward with dt / 2."""
        texts = [paulis] if isinstance(paulis, str) else list(paulis)
        c = np.asarray(coeffs, dtype=np.float64).reshape(-1)
        if c.size != len(texts):
            raise ValueError(f"{len(texts)} Pauli strings but {c.size} coefficients")
        if steps < 1 or order not in (1, 2):
            raise ValueError("steps must be >= 1 and order 1 or 2")
        dt = float(time) / steps
        if order == 1:
            step_p, step_t = texts, 2.0 * c * dt
        else:
            step_p, step_t = texts + texts[::-1], np.concatenate([c * dt, (c * dt)[::-1]])
        self.apply_pauli_rotations(step_p * steps, np.tile(step_t, steps))

    def rotation_gradient(self, paulis, thetas, observable, coeffs):
        """Apply the rotations like apply_pauli_rotations and return (energy, grad): the energy
        E = sum_j coeffs[j] <psi|observable[j]|psi> of the rotated state psi and the float64 array dE/dtheta_k, by the
        adjoint method on the device.  The handle is left holding psi.  Sharded: collective, same arguments on every
        rank, and every rank receives the same values."""
        x, z = pauli_masks(paulis, self.num_qubits)
        t = np.ascontiguousarray(np.asarray(thetas, dtype=np.float64).reshape(-1))
        if t.size != x.size:
            raise ValueError(f"{x.size} Pauli strings but {t.size} angles")
        hx, hz = pauli_masks(observable, self.num_qubits)
        c = np.ascontiguousarray(np.asarray(coeffs, dtype=np.float64).reshape(-1))
        if c.size != hx.size:
            raise ValueError(f"{hx.size} observable terms but {c.size} coefficients")
        energy = C.c_double()
        grad = np.empty(x.size, dtype=np.float64)
        check(lib.qsb_pauli_rotation_gradient(self._h, x.ctypes.data, z.ctypes.data, t.ctypes.data, x.size, hx.ctypes.data,
                                              hz.ctypes.data, c.ctypes.data, c.size, C.byref(energy), grad.ctypes.data))
        return energy.value, grad

    # ---- dense matrices (bit i of a row or column index is the value of qubits[i])
    def apply_matrix(self, U, qubits, controls=()):
        """Apply the (2^k, 2^k) complex matrix U to the target qubits (k = len(qubits), 1..6): for every index whose
        controls are all 1, a'[targets = r] = sum_c U[r, c] a[targets = c], so [3, 0] means the transposed qubit order of
        [0, 3].  No unitarity check and no renormalisation; the arithmetic is in the state's precision.  The qubit
        layout is left as it is.  Sharded: collective, same arguments on every rank."""
        self.apply_matrices([(U, qubits, controls)])

    def apply_matrices(self, ops):
        """A list of (U, qubits) or (U, qubits, controls), applied in list order (the first acts first) as one call, so
        consecutive ops share sweeps over the state."""
        ops = list(ops)
        arr, keep = _matrix_ops(ops)
        check(lib.qsb_apply_matrices(self._h, arr, len(ops)))
        del keep

    # ---- noise channels (bit i of a row or column index of a Kraus operator is the value of qubits[i])
    def apply_channels(self, channels, r=None, seed=0):
        """Quantum trajectories: for each (kraus_list, qubits) in list order, pick branch i with probability
        w_i / T = ||K_i psi||^2 / sum_j ||K_j psi||^2 (the first i whose prefix sum reaches r[c] * T) and apply
        sqrt(T / w_i) K_i, on the device.  r defaults to sample_uniform(seed, c) for channel c.  Returns (branch uint32
        array, prob float64 array).  Sharded: collective, same arguments (r included) on every rank."""
        chs = list(channels)
        if r is None:
            r = [sample_uniform(seed, c) for c in range(len(chs))]
        rr = np.ascontiguousarray(np.asarray(r, dtype=np.float64).reshape(-1))
        if rr.size != len(chs):
            raise ValueError(f"{len(chs)} channels but {rr.size} values of r")
        arr, keep = _channels(chs)
        branch = np.zeros(len(chs), dtype=np.uint32)
        prob = np.zeros(len(chs), dtype=np.float64)
        check(lib.qsb_apply_channels(self._h, arr, len(chs), rr.ctypes.data, branch.ctypes.data, prob.ctypes.data))
        del keep
        return branch, prob

    def apply_channel(self, kraus, qubits, r):
        """One channel: returns (branch, prob) as an int and a float."""
        b, p = self.apply_channels([(kraus, qubits)], [r])
        return int(b[0]), float(p[0])

    # ---- marginals and projective measurement (bit i of a bin index or an outcome is the value of qubits[i])
    @staticmethod
    def _qubits(qubits):
        return np.ascontiguousarray(np.asarray(qubits, dtype=np.int32).reshape(-1))

    def marginal_probabilities(self, qubits):
        """float64 array of 2^k values: entry b is the probability that qubits[i] reads bit i of b for every i, so
        [3, 0] gives the transposed table of [0, 3].  Computed on the device in one read of the state; the state and
        the qubit layout are left as they are, nothing is renormalised.  1 <= k <= min(n, 20)."""
        qs = self._qubits(qubits)
        out = np.empty(1 << min(qs.size, 20), dtype=np.float64)
        check(lib.qsb_marginal_probabilities(self._h, qs.ctypes.data, qs.size, out.ctypes.data))
        return out

    def collapse(self, qubits, outcome):
        """Project onto `outcome` (bit i = value of qubits[i]) and rescale to norm 1; returns its probability p,
        equal bit for bit to marginal_probabilities(qubits)[outcome].  p == 0 is refused and leaves the state as it is."""
        qs = self._qubits(qubits)
        p = C.c_double()
        check(lib.qsb_collapse(self._h, qs.ctypes.data, qs.size, int(outcome), C.byref(p)))
        return p.value

    def measure_qubits(self, qubits, r):
        """Measure these qubits with the uniform number r in [0, 1) (e.g. sample_uniform(seed, k)) and collapse the
        state onto the outcome; returns (outcome, p), bit i of the outcome = value of qubits[i].  The outcome is the
        first bin whose inclusive prefix sum C_b of the marginal table is != 0 and >= r * total."""
        qs = self._qubits(qubits)
        b, p = C.c_uint64(), C.c_double()
        check(lib.qsb_measure_qubits(self._h, qs.ctypes.data, qs.size, float(r), C.byref(b), C.byref(p)))
        return b.value, p.value

    def reset_qubits(self, qubits, r):
        """measure_qubits, then X on every qubit that came out 1, so the qubits end in |0>; returns the outcome
        (bit i = value qubits[i] had)."""
        qs = self._qubits(qubits)
        b = C.c_uint64()
        check(lib.qsb_reset_qubits(self._h, qs.ctypes.data, qs.size, float(r), C.byref(b)))
        return b.value

    # ---- reduced density matrices (bit i of a row or column index is the value of qubits[i])
    def reduced_density_matrix(self, qubits):
        """complex128 array of shape (2^k, 2^k): rho[a, b] = sum of a_j conj(a_j') over the index pairs that agree on every
        other qubit and read a / b on `qubits`, i.e. the partial trace of |psi><psi| over the other qubits.  Computed on
        the device in fp64 on the state as stored (trace = the norm, nothing is renormalised), exactly Hermitian, bit
        for bit the same on repeat; the state and the qubit layout are left as they are.  1 <= k <= min(n, 12)."""
        qs = self._qubits(qubits)
        d = 1 << min(qs.size, 12)              # larger k is refused by the library before it writes
        out = np.empty(2 * d * d, dtype=np.float64)
        check(lib.qsb_reduced_density_matrix(self._h, qs.ctypes.data, qs.size, out.ctypes.data))
        return out.view(np.complex128).reshape(d, d)

    def entanglement_entropy(self, qubits, base=2):
        """von Neumann entropy -sum w log w of rho / Tr rho for rho = reduced_density_matrix(qubits), from the
        eigenvalues w of np.linalg.eigvalsh on the host; eigenvalues <= 0 count as 0."""
        rho = self.reduced_density_matrix(qubits)
        tr = float(np.trace(rho).real)
        if not tr > 0.0:
            raise ValueError(f"the state has norm {tr}: no entropy")
        w = np.linalg.eigvalsh(rho / tr)
        w = w[w > 0.0]
        return float(-np.sum(w * np.log(w)) / np.log(base))

    # ---- overlaps and state copy
    def _inner(self, other):
        out = np.empty(2, dtype=np.float64)
        norms = np.empty(2, dtype=np.float64)
        check(lib.qsb_inner_product(self._h, other._h, out.ctypes.data, norms.ctypes.data))
        return complex(out[0], out[1]), float(norms[0]), float(norms[1])

    def overlap(self, other):
        """<self|other> = sum_j conj(self_j) other_j as a complex, in fp64 on the device over the states as stored (nothing
        is renormalised).  The precisions and qubit layouts may differ; the states and layouts are left as they are.
        Sharded: collective, every rank receives the same bits."""
        return self._inner(other)[0]

    def fidelity(self, other):
        """|<self|other>|^2 / (<self|self> <other|other>) from one device call; ValueError if either norm is 0."""
        ov, na, nb = self._inner(other)
        if na == 0.0 or nb == 0.0:
            raise ValueError(f"a state has norm 0 (norms {na}, {nb}): no fidelity")
        return (ov.real * ov.real + ov.imag * ov.imag) / (na * nb)

    def copy_from(self, other):
        """This handle's amplitudes and qubit layout become other's (a device-to-device copy of the shard; same qubits,
        precision, world, rank and device).  Plans made for the old layout are then refused, as after any layout change."""
        check(lib.qsb_copy_state(self._h, other._h))

    def save_state(self, path):
        """Dump this rank's shard (device dtype, physical order) with its qubit map; one file per rank."""
        check(lib.qsb_save_state(self._h, os.fsencode(path)))

    def load_state(self, path):
        check(lib.qsb_load_state(self._h, os.fsencode(path)))


def sample_uniform(seed, k):
    """The r in [0, 1) that shot k of Simulator.measurement(seed=seed) searches for."""
    return lib.qsb_sample_uniform(seed, k)
