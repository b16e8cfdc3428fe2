/*
 * qsim_b200.h -- C ABI of libqsim_b200.so, the B200 (sm_100a) state-vector path.
 *
 * This is the drop-in boundary for the ONE hot path of
 * RiccardoFiorentini/GPU_quantum_simulator: "apply a gate list to a 2^n complex
 * state vector".  The reference has no FFI layer; its boundary is the set of
 * non-static C functions of quantum_simulator.c (prototypes at :25-30) plus the
 * CLI of main() (:32-79).  Every entry point below names what it replaces.
 *
 * Plain C: pointers, sizes, ints.  No C++/torch types, no exceptions, the
 * library never calls exit().  All calls are blocking and return QSB_OK (0) or
 * a negative qsb_status; qsb_last_error() gives the message (thread-local).
 * A handle is not re-entrant.  There is NO CPU fallback: without a usable
 * CUDA device qsb_create() fails with QSB_ERR_NOGPU.
 *
 * Conventions (all inherited from the reference, SURVEY.md F4/F12):
 *   - little-endian qubits: qubit k <-> bit k of the amplitude index
 *     (quantum_simulator.c:83, :96-99)
 *   - a gate is a (multi-)controlled single-qubit unitary; the matrix is
 *     row-major  out0 = m00*a + m01*b, out1 = m10*a + m11*b  where a/b are the
 *     amplitudes with target bit 0/1 (quantum_simulator_naive.cu:82-86; equal to
 *     quantum_simulator.c:88-89 for every matrix the reference builds)
 *   - "rz(theta)" in circuit text is the PHASE gate diag(1, e^{i theta})
 *     (quantum_simulator.c:205-208)
 */
#ifndef QSIM_B200_H
#define QSIM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum qsb_status {
    QSB_OK = 0,
    QSB_ERR_ARG = -1,     /* bad argument */
    QSB_ERR_CUDA = -2,    /* CUDA runtime error (message has file:line, cf. CHECK, naive.cu:29-47) */
    QSB_ERR_NOMEM = -3,   /* host or device allocation failed ("Malloc error", quantum_simulator.c:170) */
    QSB_ERR_PARSE = -4,   /* circuit text rejected ("Unknown token", :213) */
    QSB_ERR_NOGPU = -5,   /* no CUDA device: the product has no CPU path */
    QSB_ERR_COMM = -6,    /* multi-GPU exchange failed */
    QSB_ERR_IO = -7       /* cannot open circuit file (:129) */
} qsb_status;

enum { QSB_F32 = 32, QSB_F64 = 64 };

/* One gate of the IR: controls-mask + target + 2x2 complex matrix.
 * Replaces the (U[4], target) / (control, target) argument pairs of
 * execute_single_qubit_gate (:81) and execute_cnot (:94), and one row of the
 * four arrays parse_circuit() fills in the CUDA variants (naive.cu:224-402). */
typedef struct qsb_gate {
    uint64_t controls; /* bit k set: qubit k must be 1 for the gate to act   */
    int32_t target;    /* qubit the 2x2 matrix acts on                        */
    int32_t flags;     /* reserved, 0                                         */
    double m[8];       /* m00 m01 m10 m11, each (re, im)                      */
} qsb_gate_t;

/* Execution modes.  SWEEP = one full pass over the state per gate, the
 * reference's own schedule (naive.cu:163-189) kept as a cross-check and as the
 * "unfused" baseline; TILED = the fused tile-pass schedule (the product). */
enum { QSB_MODE_TILED = 0, QSB_MODE_SWEEP = 1,
       /* DENSE = experiment of BASELINE.json configuration 4: gates merged greedily into dense k-qubit unitaries
        * (k = tile_bits, 2..5; the reference's 4x4 accumulator of quantum_simulator_4x4.cu:327-501 generalised), one
        * sweep per block like kernel_gate_4 (:109-146).  Single GPU.  Measured slower than TILED at every k
        * (DESIGN.md section 3.1); kept for the k sweep and the tensor-core check, not as a product path. */
       QSB_MODE_DENSE = 2 };

typedef struct qsb_options {
    int32_t precision;    /* QSB_F32 | QSB_F64 (state dtype on the device)    */
    int32_t device;       /* CUDA ordinal, -1 = current                       */
    int32_t mode;         /* QSB_MODE_*                                       */
    int32_t tile_bits;    /* TILED: reserved, the tile is 2^12 (f32) / 2^11 (f64) amplitudes (build-time, csrc/tiled.h);
                           * DENSE: the fusion width k, 2..5 (0 = 4) */
    int32_t low_bits;     /* contiguous low index bits every tile keeps, 0 = default (4 f32 / 3 f64) */
    int32_t rank;         /* this process' shard, 0..world-1                  */
    int32_t world_size;   /* power of two; state sharded on the top log2(world) qubits */
    int32_t use_graph;    /* 1 = capture the pass launches of a plan into a CUDA graph on its first qsb_execute and
                           * replay it afterwards (single-GPU tiled plans; for plans executed many times on small
                           * registers, where a pass is shorter than its launch).  0 = plain stream launches. */
    int32_t verbose;
    /* planner / exchange tuning knobs, all 0 = default (used by bench.py A/B runs and the tests):
     *   [0] minimum number of local gates a pass must still find before a qubit exchange is scheduled (default 10)
     *   [1] 2 = keep the qubits of phase gates thread-level at any price ("lazy diagonals")
     *   [2] k+1 = trim tail rounds of SM-bound passes that hold fewer than k gates (default k = 2; 1 = off)
     *   [3] fusion-depth cap: stop adding rounds to a pass at this estimated SM cost (unit-form gate units)
     *   [4] 1 = do not defer phase gates that touch a vector bit; 2 = no 2x2 products of consecutive one-qubit gates;
     *       4 = no merged controlled-phase runs (G_DIAGA); 5 = a CX between two h on its target stays a CX (default: h cx h becomes one
     *       controlled phase); 6 = the rewrite also with an h on one side only (fewer passes, more diagonal slots)
     *   [5] exchange flavour: 1 direct fused peer scatter (victims trade places with the rank bits wherever they are),
     *       2 NCCL all-to-all, 3 pipelined copy-engine exchange, 4 round-1 fused scatter (victims moved to the top local
     *       positions first)   (0: chosen by qsb_comm_init -- 1, or 2 if the peer shards cannot be mapped)
     *       With [0] = 0 a sharded plan is built for a few exchange thresholds and the cheapest schedule kept.
     *   [6] 1 = do not sink thread-level phases to later rounds; 2 = first-come tile choice (no hill climbing);
     *       3 = no lane relocation at the end of a pass (an empty round turns the registers instead, as in round 1);
     *       4 = lane relocation only for the qubits in conflict (default: every pass re-picks the qubits that live on
     *       the lane positions).  With [6] = 0 a sharded plan also tries 4 and keeps the cheaper schedule. */
    int32_t reserved[7];
} qsb_options_t;

typedef struct qsb_sim qsb_t;      /* simulator: owns the device state          */
typedef struct qsb_plan qsb_plan_t; /* a fused, scheduled circuit (device-ready) */

/* Counters of the last qsb_execute / qsb_apply_gates on a handle. */
typedef struct qsb_run_stats {
    double device_ms;         /* CUDA-event time, first pass start -> last pass end */
    double plan_ms;           /* host fusion + scheduling time                 */
    uint64_t source_gates;    /* gates handed in                               */
    uint64_t device_ops;      /* ops after canonicalisation / fusion           */
    uint32_t passes;          /* full sweeps over the local state              */
    uint32_t rounds;          /* shared-memory exchange rounds, all passes     */
    uint32_t swaps;           /* global<->local qubit exchanges (multi-GPU)    */
    uint32_t kernel_launches; /* kernels launched in the timed region          */
    uint64_t bytes_moved;     /* algorithmic HBM bytes: sum over passes of 2*N_loc*B */
    uint64_t bytes_exchanged; /* bytes this rank sent over NVLink              */
    double exchange_ms;       /* part of device_ms spent in exchanges          */
} qsb_run_stats_t;

/* ---- lifecycle ---------------------------------------------------------- */
void qsb_options_default(qsb_options_t *opt);
/* Allocates 2^(num_qubits)/world amplitudes on the device and sets |0...0>.
 * Replaces malloc + init at quantum_simulator.c:168-177 and cudaMalloc +
 * init_state_vector at naive.cu:148-158. */
int qsb_create(qsb_t **out, int num_qubits, const qsb_options_t *opt);
void qsb_destroy(qsb_t *s);
int qsb_reset(qsb_t *s); /* back to |0...0> */
int qsb_num_qubits(const qsb_t *s);
int qsb_precision(const qsb_t *s);

/* ---- the hot path --------------------------------------------------------
 * Replaces the per-gate host loop (quantum_simulator.c:145-243,
 * naive.cu:163-189) and the host "preprocessing" of the CUDA variants
 * (preproces.cu:215-269, 4x4.cu:327-501, 4x4_permute.cu:350-434). */
int qsb_apply_gates(qsb_t *s, const qsb_gate_t *gates, size_t n); /* plan + execute + free */
/* A plan is made for the qubit layout the handle has at qsb_plan_create (the identity after qsb_create /
 * qsb_reset; fused passes leave the qubits permuted, qsb_get_layout).  qsb_execute from any other layout is
 * refused with QSB_ERR_ARG instead of computing on the wrong bits: to run a plan again, qsb_reset first (or
 * plan again from the current layout, which is what qsb_apply_gates does). */
int qsb_plan_create(qsb_t *s, const qsb_gate_t *gates, size_t n, qsb_plan_t **out);
int qsb_execute(qsb_t *s, qsb_plan_t *plan);
void qsb_plan_destroy(qsb_plan_t *plan);
int qsb_plan_stats(const qsb_plan_t *plan, qsb_run_stats_t *out); /* static counters, times = 0 */
int qsb_last_run_stats(const qsb_t *s, qsb_run_stats_t *out);
/* Host-only scheduling (no device needed): what qsb_plan_create would build
 * for a (num_qubits, precision, world) machine.  Used by CPU tests. */
int qsb_plan_dry_run(int num_qubits, const qsb_options_t *opt, const qsb_gate_t *gates,
                     size_t n, qsb_run_stats_t *out);

/* ---- readout --------------------------------------------------------------
 * Amplitudes come back in LOGICAL index order as interleaved (re, im) doubles,
 * i.e. the memory layout of the `complex *v` compute_state_vector returns
 * (quantum_simulator.c:125).  first/count address the GLOBAL index space; in a
 * multi-GPU run each rank may only read its own shard. */
int qsb_download(qsb_t *s, double *re_im, uint64_t first, uint64_t count);
int qsb_upload(qsb_t *s, const double *re_im, uint64_t first, uint64_t count);
/* The shard as it lies on the device: amplitudes first..first+count of the LOCAL PHYSICAL index space
 * (fp64 pairs), plus the qubit layout needed to interpret it: perm64[q] = physical index bit of
 * logical qubit q (bits >= *nloc are the rank bits).  This is how a sharded state is gathered:
 * fused passes may leave the qubits permuted, and no rank owns a contiguous logical range. */
int qsb_download_physical(qsb_t *s, double *re_im, uint64_t first, uint64_t count);
int qsb_get_layout(const qsb_t *s, int8_t *perm64, int *nloc);
/* Raw copy in the device dtype (float or double pairs), logical order. */
int qsb_download_native(qsb_t *s, void *dst, uint64_t first, uint64_t count);
/* sum |a|^2 over the local shard, and the local argmax (global index). */
int qsb_norm_argmax(qsb_t *s, double *norm, uint64_t *argmax_idx, double *argmax_p);
/* |a_i|^2 for i in [first, first+count), fp64. */
int qsb_probabilities(qsb_t *s, double *p, uint64_t first, uint64_t count);
/* Inclusive prefix sum of |a|^2 in logical index order -- compute_state_cumulative_distribution
 * (:256-268).  |a|^2 and the prefix sums are computed on the device (block scans chained by serial
 * offsets: monotone, equal to the reference's single fp64 accumulator up to re-association, <= 1e-12).
 * cdf[k] is the GLOBAL prefix sum at index first + k, i.e. it includes every |a_i|^2 with i < first:
 * any range returns, bit for bit, the slice [first, first + count) of the full call (a range with
 * first > 0 costs one extra read of the amplitudes below first).  One GPU only: on a sharded state it
 * returns QSB_ERR_ARG, since the indices below a rank's own live on other ranks; qsb_sample draws
 * shots from a sharded state. */
int qsb_cdf(qsb_t *s, double *cdf, uint64_t first, uint64_t count);
/* `shots` draws from the distribution; same search rule as measurement() (:270-283: first index
 * with cdf != 0 and cdf >= r, clamped to the last index), r from a seeded generator instead of
 * rand().  Device-side and streaming: no 2^n array is built (segment totals + one re-scanned
 * segment per shot), so it works at any n that fits the device.  On one GPU the result equals a
 * search of qsb_cdf with the same r.  On a sharded state every rank must call it with the same
 * seed and shots (collective: per-rank totals are all-gathered, the shots all-reduced); every rank
 * receives all shots, drawn in rank-major physical order and returned as logical indices. */
int qsb_sample(qsb_t *s, uint64_t seed, int shots, uint64_t *out);
/* The r of shot k for a seed (splitmix64 -> 53-bit uniform in [0,1)): lets a caller replay
 * measurement()'s search on a CDF of its own. */
double qsb_sample_uniform(uint64_t seed, int k);

/* ---- observables ------------------------------------------------------------
 * A Pauli string is a pair of masks over LOGICAL qubits: x bit q = X on qubit q, z bit q = Z on qubit q, both
 * = Y (Y = i X Z = [[0, -i], [i, 0]]).  Its action on an amplitude vector, which tests and callers share:
 *     (P a)_j = i^{popc(x & z)} * (-1)^{popc((j ^ x) & z)} * a_{j ^ x}
 * and the value returned is <psi|P|psi> = sum_j conj(a_j) (P a)_j, real, in fp64, on the state as stored (no
 * renormalisation: x = z = 0 gives the norm).
 *
 * Evaluated on the device in tile sweeps: terms whose X parts differ only inside one tile of the state share a
 * single read of it (diagonal terms all share one sweep; n single-qubit X terms take about n / 8), partial sums
 * are reduced in a fixed order (repeated calls return identical bits).  Cost: one read of the local shard per
 * sweep; on a sharded state, one copy of a partner shard per distinct pattern of X on rank qubits. */
/* out[k] = <psi| P_k |psi> for Pauli strings given as logical masks (x: X or Y, z: Z or Y).
 * Blocking.  Does not change the state or the qubit layout.  On a sharded state every rank
 * calls it with the same terms (collective), and every rank receives every value. */
int qsb_expectation_pauli(qsb_t *s, const uint64_t *x, const uint64_t *z, size_t nterms, double *out);
/* "X0 Z3 Y5" -> masks.  Tokens are [IXYZ]<qubit>, separated by whitespace.
 * "" or "I" is the identity.  A repeated qubit or an unknown letter gives QSB_ERR_PARSE.
 * A qubit >= num_qubits gives QSB_ERR_ARG. */
int qsb_pauli_from_string(const char *text, int num_qubits, uint64_t *x, uint64_t *z);
/* Host only, no device: the number of state sweeps and shard exchanges that qsb_expectation_pauli
 * would run for these terms from the identity layout.  The counterpart of qsb_plan_dry_run. */
int qsb_expectation_dry_run(int num_qubits, const qsb_options_t *opt, const uint64_t *x, const uint64_t *z,
                            size_t nterms, uint32_t *sweeps, uint32_t *exchanges);

/* ---- Pauli rotations ---------------------------------------------------------
 * Rotation k is R_k = exp(-i theta_k P_k / 2) = cos(theta_k / 2) I - i sin(theta_k / 2) P_k for the Pauli string P_k given
 * as logical masks in the format of the observables above (x: X or Y, z: Z or Y), applied to the state as
 *     a <- cos(theta_k / 2) a - i sin(theta_k / 2) (P_k a)      with (P_k a)_j from the action formula above,
 * for k = 0, 1, ..., n - 1 in that order: the first listed rotation acts first, like a gate list.  x = z = 0 multiplies
 * the state by exp(-i theta / 2) (kept, not dropped).  cos and sin are computed in fp64 on the host, the arithmetic is
 * done in the state's precision, and nothing is renormalised.  theta = 0 is skipped: it leaves the state bytes as they
 * are.  Note that "rz" in circuit text is the phase gate diag(1, e^{i theta}), while the rotation of "Z0" is
 * diag(e^{-i theta / 2}, e^{i theta / 2}).
 *
 * Applied on the device in tile sweeps: a sweep carries a consecutive run of rotations whose X parts outside one tile of
 * the state agree (diagonal rotations fit any run; n single-qubit X rotations on distinct qubits take about n / 9) and
 * costs one read and one write of the local shard however many rotations it carries.  Rotations are never reordered.
 * The qubit layout, the state buffer (a captured graph's state), the role of the exchange buffer and the peer mappings
 * are left as they are, so a plan made before the call still executes after it.
 * Errors return QSB_ERR_ARG with the state untouched: a null handle, a null array when n > 0, a qubit >= the handle's
 * qubits, a non-finite theta.  n = 0 is a no-op.  A sharded handle without qsb_comm_init gives QSB_ERR_COMM.  On a
 * sharded state the call is collective (same arguments on every rank): a sweep whose rotations flip rank qubits first
 * receives the partner rank's shard into the exchange buffer, so it costs one shard copy, two reads and one write. */
int qsb_apply_pauli_rotations(qsb_t *s, const uint64_t *x, const uint64_t *z, const double *theta, size_t n);
/* Host only, no device: the number of sweeps (launches that read and write the shard) and partner-shard copies that
 * qsb_apply_pauli_rotations would run for these rotations (all angles taken non-zero) from the identity layout. */
int qsb_pauli_rotation_dry_run(int num_qubits, const qsb_options_t *opt, const uint64_t *x, const uint64_t *z,
                               size_t n, uint32_t *sweeps, uint32_t *exchanges);

/* ---- dense matrices -----------------------------------------------------------
 * A matrix op is a complex 2^k x 2^k matrix m on k distinct LOGICAL target qubits, 1 <= k <= QSB_MATRIX_MAX_K, optionally
 * controlled.  For each op in list order (the first listed acts first, like a gate list) and every index j whose control
 * bits are all 1:
 *     a'[j with targets = r] = sum_c m[r][c] * a[j with targets = c]
 * where bit i of a row / column index r, c is the value of targets[i] -- the index convention of the marginals and the
 * reduced density matrices, so {3, 0} means the transposed qubit order of {0, 3}.  For k = 1 and the same entries this
 * is exactly qsb_gate_t's  out0 = m00 a + m01 b.  Entries are fp64 on the host; the arithmetic is done in the state's
 * precision, and each output is a sum in a fixed order (repeated calls return identical bits).  There is no unitarity
 * check and nothing is renormalised: non-unitary matrices (Kraus operators, projectors, Hamiltonian blocks) are applied
 * as they are.
 *
 * Applied on the device in tile sweeps: a sweep carries a consecutive run of ops whose targets fit one tile of the state
 * and costs one read and one write of the local shard however many ops it carries.  Ops are never reordered.  The qubit
 * layout, the state buffer (a captured graph's state), the role of the exchange buffer and the peer mappings are left as
 * they are, so a plan made before the call still executes after it.
 * Errors return QSB_ERR_ARG with the state untouched: a null handle, a null ops array when n > 0, k outside
 * [1, min(n_qubits, QSB_MATRIX_MAX_K)], a target >= n_qubits or repeated, a control >= n_qubits or equal to a target, a
 * null m, a non-finite entry, flags != 0, and options (the handle's, or a dry run's) whose low_bits is outside the range
 * the tile scheduler accepts (f32 3..6, f64 2..5, 0 = the default), which leaves every tile room for any op.  n = 0 is a
 * no-op.  A sharded handle without qsb_comm_init gives QSB_ERR_COMM.
 * Device scratch is allocated once per call and freed before it returns: the launch table plus the matrices in the
 * state's precision (at most 64 KiB per k = 6 op in f64); QSB_ERR_NOMEM leaves the state untouched.
 * On a sharded state the call is collective (the same ops on every rank).  A sweep whose run has a target on a rank
 * qubit first receives the partner rank's shard into the exchange buffer (one shard copy, two reads, one write).  An op
 * with m >= 2 targets on rank qubits is applied as SWAP(r_i, l_i) ... U' ... SWAP(r_i, l_i) for i = 2..m, with l_i local
 * qubits that are neither targets nor controls of the op standing in for r_i in U': 2 (m - 1) more sweeps and shard
 * copies unless they merge with neighbours, and QSB_ERR_ARG if no such local qubit is free. */
#define QSB_MATRIX_MAX_K 6
typedef struct qsb_matrix_op {
    uint64_t controls;                  /* bit q set: logical qubit q must be 1 for the matrix to act (as qsb_gate_t) */
    int32_t k;                          /* number of targets, 1..QSB_MATRIX_MAX_K */
    int32_t targets[QSB_MATRIX_MAX_K];  /* distinct logical qubits; bit i of a row / column index = value of targets[i] */
    int32_t flags;                      /* reserved, 0 */
    const double *m;                    /* 2 * 4^k doubles, row-major (re, im): entry (a, b) at m[2 * (a * 2^k + b)] */
} qsb_matrix_op_t;

int qsb_apply_matrices(qsb_t *s, const qsb_matrix_op_t *ops, size_t n);
/* Host only, no device: the number of sweeps (launches that read and write the shard) and partner-shard copies that
 * qsb_apply_matrices would run for these ops from the identity layout.  m may be NULL here: only shapes are read. */
int qsb_matrix_dry_run(int num_qubits, const qsb_options_t *opt, const qsb_matrix_op_t *ops, size_t n,
                       uint32_t *sweeps, uint32_t *exchanges);

/* ---- Pauli-rotation gradients -----------------------------------------------
 * For the ansatz psi = R_{n-1} ... R_0 phi_0, R_k = exp(-i theta_k P_k / 2) (rotations rx / rz / theta in the format and
 * order of qsb_apply_pauli_rotations, phi_0 the state in the handle at the call) and the observable H = sum_j coef[j] P_j
 * (hx / hz in the format of the observables above, real coefficients):
 *   - the handle is left holding psi, bit for bit what qsb_apply_pauli_rotations(s, rx, rz, theta, nrot) leaves (it is
 *     that call); the qubit layout, the state buffer (a captured graph's state), the role of the exchange buffer and the
 *     peer mappings are left as they are;
 *   - *energy = sum_j coef[j] <psi|P_j|psi>, each value from qsb_expectation_pauli on psi, summed on the host in fp64 in
 *     term order as e = e + coef[j] * v[j] from e = 0 (product rounded, then added), so it equals that sum by a caller;
 *   - grad[k] = dE/dtheta_k = Im <lambda_k| P_k |phi_k>, phi_k = R_k ... R_0 phi_0, lambda_k = R_{k+1}^dag ... R_{n-1}^dag
 *     H psi, by the adjoint method: one sweep set that builds H psi and one backward pass over the rotations.  It is for
 *     the state as stored (nothing is renormalised); theta_k = 0 gets its gradient too.
 * Reductions run in a fixed order without floating-point atomics: repeated calls return identical bits, and on a
 * sharded state (a collective call, same arguments on every rank) every rank receives the same energy and gradients.
 * nrot = 0 gives the energy only.  Device scratch, allocated before the state is touched and freed before the call
 * returns: two shard-sized buffers on one GPU, three on a sharded state (at 30 qubits f32, 16 GiB beside the 8 GiB
 * state), plus the launch tables and (CTAs x 1024) fp64 partials; QSB_ERR_NOMEM with the state untouched if it fails.
 * Errors return QSB_ERR_ARG with the state untouched: a null handle, a null array when its count is > 0, nterms = 0, a
 * null energy or (nrot > 0) grad, a qubit >= the handle's qubits, a non-finite theta or coefficient.  A sharded handle
 * without qsb_comm_init gives QSB_ERR_COMM. */
int qsb_pauli_rotation_gradient(qsb_t *s,
                                const uint64_t *rx, const uint64_t *rz, const double *theta, size_t nrot,
                                const uint64_t *hx, const uint64_t *hz, const double *coef, size_t nterms,
                                double *energy, double *grad);
/* Host only, no device, from the identity layout with every angle taken non-zero: the sweeps that build H psi, the
 * fused adjoint sweeps, and the partner-shard copies of both.  The forward pass and the energy cost what
 * qsb_pauli_rotation_dry_run and qsb_expectation_dry_run report. */
int qsb_pauli_rotation_gradient_dry_run(int num_qubits, const qsb_options_t *opt,
                                        const uint64_t *rx, const uint64_t *rz, size_t nrot,
                                        const uint64_t *hx, const uint64_t *hz, size_t nterms,
                                        uint32_t *apply_sweeps, uint32_t *adjoint_sweeps, uint32_t *exchanges);

/* ---- marginals and projective measurement ----------------------------------
 * The measured qubits are an array qubits[0..k-1] of distinct LOGICAL qubits, 1 <= k <= min(n, 20).  Bit i of a bin
 * index or an outcome is the value of qubits[i], so {3, 0} gives the transposed table of {0, 3}.  All sums are fp64
 * over the state as stored; nothing is renormalised.  More than 20 qubits are measured in groups: measuring disjoint
 * groups one after another gives the same joint distribution (the Born rule chain p(a) p(b | a)).
 * Errors return QSB_ERR_ARG and leave the state untouched: a repeated qubit, a qubit outside [0, n), k outside
 * [1, min(n, 20)], a null pointer (other than the optional prob / outcome noted below), an outcome >= 2^k.  On a
 * sharded state these calls are collective (same arguments on every rank) and need qsb_comm_init (else QSB_ERR_COMM);
 * every rank receives the same values, bit for bit. */
/* out[b] = sum of |a_j|^2 over every j whose bits qubits[i] equal bit i of b; 2^k values.  One read of the local shard.
 * Deterministic: repeated calls return identical bits.  Does not change the state or the qubit layout. */
int qsb_marginal_probabilities(qsb_t *s, const int *qubits, int k, double *out);
/* Project onto outcome `outcome` of these qubits and scale the kept amplitudes by 1/sqrt(p), p = the marginal of that
 * outcome (equal bit for bit to its qsb_marginal_probabilities entry), so the state has norm 1.  *prob = p (prob may
 * be NULL).  p == 0 -> QSB_ERR_ARG and the state is unchanged.  The qubit layout is unchanged.  Cost: a read of the
 * kept amplitudes for p, then one pass that writes the shard and reads only the kept amplitudes. */
int qsb_collapse(qsb_t *s, const int *qubits, int k, uint64_t outcome, double *prob);
/* The marginal table, then the outcome by the rule of measurement() (quantum_simulator.c:279) on that table: the first
 * b with C_b != 0 and C_b >= r * T, where C_b is the inclusive serial fp64 prefix sum of the table in bin order and
 * T = C_{2^k - 1}; then the collapse onto it (*prob = its table entry; prob may be NULL).  r in [0, 1), e.g. from
 * qsb_sample_uniform.  T == 0, or r outside [0, 1) or NaN -> QSB_ERR_ARG, state unchanged.  With r < 1 and T > 0 the
 * rule always picks a bin with p > 0 (C_b >= r * T is reached at the latest by the last bin, and a bin with p = 0
 * repeats the C of the bin before it), so there is no clamp case.  Sharded: the same r on every rank gives every rank
 * the same outcome. */
int qsb_measure_qubits(qsb_t *s, const int *qubits, int k, double r, uint64_t *outcome, double *prob);
/* qsb_measure_qubits, then X (through qsb_apply_gates) on every measured qubit that came out 1: the qubits end in |0>.
 * *outcome = the measured outcome (outcome may be NULL). */
int qsb_reset_qubits(qsb_t *s, const int *qubits, int k, double r, uint64_t *outcome);

/* ---- reduced density matrices ------------------------------------------------
 * rho = Tr_{other qubits} |psi><psi| for qubits[0..k-1], 1 <= k <= min(n, 12), with the qubit conventions and argument
 * rules of the marginals above: distinct LOGICAL qubits, bit i of a and b is the value of qubits[i], so {3, 0} gives the
 * matrix of {0, 3} with its indices re-ordered.  rho has 2 * 4^k doubles: entry (a, b) at rho[2 * (a * 2^k + b)] (re)
 * and [.. + 1] (im):
 *     rho[a][b] = sum over j, j' that agree on every other qubit, with bits(j) = a and bits(j') = b, of a_j * conj(a_j')
 * Everything is fp64 on the state as stored, with no renormalisation: Tr rho = the norm, and the diagonal is the
 * qsb_marginal_probabilities table up to the order of the additions.  Exactly Hermitian: only the entries with a <= b
 * are computed and the others are their mirror, so rho[b][a] == conj(rho[a][b]) bit for bit and every diagonal imaginary
 * part is +0.0.  Deterministic: reductions run in a fixed order, repeated calls return identical bits.  Does not change
 * the state, the qubit layout, the role of the exchange buffer or the peer mappings.
 * Errors return QSB_ERR_ARG and leave the state untouched: a null handle, qubit array or rho, k outside [1, min(n, 12)],
 * a repeated qubit, a qubit outside [0, n).  A sharded handle without qsb_comm_init gives QSB_ERR_COMM.  The device
 * scratch is one allocation per call, freed before it returns (QSB_ERR_NOMEM if it fails): 2^m 4^(k - m) x 16 bytes for
 * the local matrices (m = measured qubits on rank bits), at most 64 MiB of per-block partials, and on a sharded state
 * world times the local matrices for their all-gather (host memory holds the same); at k = 12 on one GPU that is 256 MiB
 * plus the partials, on 8 ranks with no rank qubit measured 2.25 GiB.
 * Cost: one read of the local shard for 2^k_loc <= 64 (k_loc = measured qubits on local bits), about 2^k_loc / 64 reads
 * above, and 4 * 2^n_loc * (2^k_loc + 1) fp64 flops.  On a sharded state the call is collective (same arguments on every
 * rank), each rank receives the shard of a partner rank into its exchange buffer once per non-zero pattern of the
 * measured rank qubits (2^m - 1 shard copies per call), and every rank receives the same bits. */
int qsb_reduced_density_matrix(qsb_t *s, const int *qubits, int k, double *rho);

/* ---- shard dump / reload ----------------------------------------------------
 * The reference keeps the state only in memory (quantum_simulator.c:75 frees it
 * at exit); long sharded runs want a checkpoint.  File = 128-byte header (magic
 * "QSBSHARD", version, qubits, precision, world, rank, local bits, the logical ->
 * physical qubit map) + the shard exactly as it lies in HBM.  One file per rank;
 * loading checks that the handle has the same shape and restores the qubit map. */
int qsb_save_state(qsb_t *s, const char *path);
int qsb_load_state(qsb_t *s, const char *path);

/* ---- multi-GPU (one process per GPU) --------------------------------------
 * nccl_unique_id: the 128 bytes of an ncclUniqueId, identical on every rank
 * (qsb_comm_unique_id makes one on rank 0; the caller broadcasts it, e.g. with
 * torch.distributed).  The reference has no multi-GPU path (SURVEY.md F11). */
int qsb_comm_unique_id(void *id128);
int qsb_comm_init(qsb_t *s, const void *nccl_unique_id128);

/* ---- QASM front end -------------------------------------------------------
 * Accepts the reference grammar bit-for-bit (quantum_simulator.c:133-242:
 * two header statements, `qubit[n] q;` or `qubit q[n];`, operands `q[k]` or
 * `$k`, CRLF, gate set cx x sx z s sdg t tdg rz h) plus a superset
 * (y p rx ry u cz cp crz swap ccx ..., `gate` definitions, ctrl @ / negctrl @ / inv @ / pow(k) @
 * modifiers, gphase, several registers, whole-register operands, `pi` expressions and the
 * usual functions in parameters; barrier / measure / reset / classical statements ignored).
 * The CUDA variants' "<num_q> <num_g>" header (naive.cu:239-240) is accepted
 * too.  *gates is malloc'ed; release with qsb_free(). */
int qsb_parse_qasm_file(const char *path, int *num_qubits, qsb_gate_t **gates, size_t *n);
int qsb_parse_qasm_string(const char *text, int *num_qubits, qsb_gate_t **gates, size_t *n);
/* Fill `g` with a named gate of the table at quantum_simulator.c:184-211 (+superset). */
int qsb_gate_from_name(const char *name, const double *params, int nparams,
                       const int *qubits, int nqubits, qsb_gate_t *out, int *nout);
void qsb_free(void *p);

const char *qsb_last_error(void);
const char *qsb_version(void);

/* ---- reference-compatible shims --------------------------------------------
 * Same names, argument meaning, ownership (callee mallocs, caller frees) and
 * stdout behaviour as the functions at quantum_simulator.c:25-30, so the
 * reference's own main() links against libqsim_b200.so unchanged (see
 * INTEGRATION.md).  `v` is a host `double complex *`; every call runs on the
 * GPU.  Declared with void* / double* here so this header needs no <complex.h>.
 */
double *qsb_ref_compute_state_vector(const char *filename, int *num_q);       /* -> compute_state_vector */
void qsb_ref_execute_single_qubit_gate(double *v, int num_q, const double U[8], int target); /* U as complex U[4] */
void qsb_ref_execute_cnot(double *v, int num_q, int control, int target);
double *qsb_ref_compute_state_cumulative_distribution(const double *v, int num_q);
long long qsb_ref_measurement(const double *cumul, int num_q);

#ifdef __cplusplus
}
#endif
#endif /* QSIM_B200_H */
