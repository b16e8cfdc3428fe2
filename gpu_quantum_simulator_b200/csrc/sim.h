/* sim.h -- host-side objects behind the opaque handles of qsim_b200.h. */
#pragma once
#include <vector>
#include "common.cuh"
#include "dense.h"

struct TiledPlan; /* tiled.h */

struct qsb_sim {
    int n = 0;        /* logical qubits of the circuit                          */
    int g = 0;        /* log2(world): qubits whose physical bit is the rank     */
    int nloc = 0;     /* physical local index bits (>= min tile, may pad n - g) */
    int nphys = 0;    /* nloc + g: width of the physical global index           */
    int prec = QSB_F32;
    int rank = 0, world = 1, device = 0;
    qsb_options_t opt{};
    void *state = nullptr;   /* 2^nloc amplitudes                               */
    void *state2 = nullptr;  /* exchange target buffer (multi-GPU), lazily made */
    size_t state_bytes = 0;
    BitPerm perm{};          /* logical qubit -> physical bit (identity at reset) */
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream[4] = {nullptr, nullptr, nullptr, nullptr};   /* pipelined exchange: peer copies on the copy engines */
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evx0 = nullptr, evx1 = nullptr;
    /* events of the exchanges of one qsb_execute: created on first use, reused by every later execution (no
     * cudaEventCreate / Destroy inside the timed loop), destroyed with the handle */
    std::vector<cudaEvent_t> ev_pool; size_t ev_next = 0;
    void *staging = nullptr; /* device staging for readout (two halves, double-buffered by the downloads) */
    cudaStream_t dl_stream = nullptr;                        /* device -> host copies of the readout pipeline */
    cudaEvent_t dl_filled[2] = {nullptr, nullptr}, dl_copied[2] = {nullptr, nullptr};
    size_t staging_bytes = 0;
    void *d_scratch = nullptr; /* small device scratch (reductions)             */
    qsb_run_stats_t last{};
    void *comm = nullptr;    /* ncclComm_t                                      */
    /* peer shards mapped through CUDA IPC (filled by qsb_comm_init): a fused-exchange pass stores into them */
    bool peers_ok = false;
    void *peer_state[16] = {nullptr};    /* rank r's current state buffer  (own rank: == state)  */
    void *peer_state2[16] = {nullptr};   /* rank r's second buffer         (own rank: == state2) */
};

struct qsb_plan {
    int mode = QSB_MODE_TILED;
    int n = 0, prec = QSB_F32, world = 1;
    std::vector<COp> cops;   /* canonical ops in source order (sweep mode executes these) */
    double gphase[2] = {1.0, 0.0}; /* global scalar factored out of diagonal gates */
    TiledPlan *tiled = nullptr;
    std::vector<DenseBlock> dense;   /* QSB_MODE_DENSE (experiment): one dense k-qubit unitary per sweep */
    qsb_run_stats_t stats{};
    /* qsb_options_t.use_graph: the pass launches of this plan captured once, replayed by every later qsb_execute */
    cudaGraphExec_t graph_exec = nullptr;
    void *graph_state = nullptr;   /* the state buffer the captured launches point at */
};

/* canonicalise source gates -> COps (+ global phase) */
int qsb_canonicalise(const qsb_gate_t *gates, size_t n, int num_qubits, std::vector<COp> &out, double gphase[2]);

/* QSB_ERR_ARG (with a message naming fn) unless qubits[0..k-1] are distinct qubits of the handle and 1 <= k <=
 * min(n, kmax); hint says what to do about a k above kmax */
int check_qubits(const qsb_sim *s, const int *qubits, int k, int kmax, const char *fn, const char *hint);

/* the rule of measurement() (quantum_simulator.c:279) on a table of weights: the first b whose inclusive serial fp64
 * prefix sum C_b is != 0 and >= r * T, T = the sum of the table; QSB_ERR_ARG (with a message naming fn) if T is not > 0 */
int pick_outcome(const std::vector<double> &tab, double r, uint64_t *b_out, const char *fn);

/* element size of one amplitude */
static inline size_t amp_bytes(int prec) { return prec == QSB_F64 ? 16 : 8; }
