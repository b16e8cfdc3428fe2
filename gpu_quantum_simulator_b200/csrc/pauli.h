/* pauli.h -- Pauli-string helpers and sweep planners defined in expect.cu / pauli_rot.cu / matrix.cu and shared with
 * pauli_grad.cu (host only, no CUDA calls). */
#pragma once
#include <vector>
#include "sim.h"

struct PhysTerm { uint64_t xl, zl, xr, zr; int y; };   /* local / rank-bit parts of the physical masks, y = popc(x&z) & 3 */

inline int parity64(uint64_t v) { return __builtin_popcountll(v) & 1; }

/* tile bits T (12 f32 / 11 f64) and the low bits L every tile keeps, for a precision and the handle's options */
int exp_geometry(int prec, const qsb_options_t *opt, int *T, int *L);
/* QSB_ERR_ARG (with a message naming fn) for a low_bits outside the range the tile scheduler accepts (f32 3..6, f64 2..5,
 * 0 = the default) */
int check_low_bits(int prec, const qsb_options_t *opt, const char *fn);
/* QSB_ERR_ARG (with a message naming fn) for a null array when nterms > 0 or a qubit >= n */
int check_terms(int n, const uint64_t *x, const uint64_t *z, size_t nterms, const char *fn);
/* logical masks -> physical local / rank-bit masks under the layout perm */
void to_physical(int n, int nloc, const BitPerm &perm, const uint64_t *x, const uint64_t *z, size_t nterms, std::vector<PhysTerm> &out);
/* compress the bits of m at the positions pb[0..T-1] */
uint32_t tile_coord(uint64_t m, const int8_t *pb, int T);
/* the options and local bits of a dry run: the checks of qsb_create on (num_qubits, opt), without a device */
int pauli_dry_run_shape(int num_qubits, const qsb_options_t *opt_in, qsb_options_t *opt, int *nloc);

/* ---- term grouping of expect.cu: sweeps that each evaluate every term whose local x outside the tile is x_out */
struct ExpSweep {
    uint64_t xr = 0;               /* rank-bit flips: partner rank = rank ^ xr */
    int8_t pb[16];                 /* tile coordinate bit j -> local physical bit */
    uint64_t bmask = 0, x_out = 0; /* tile bits, local flips outside the tile */
    std::vector<uint32_t> terms;
};
/* greedy cover of the distinct physical x masks by sweeps of T tile bits, grouped by xr (xr == 0 first) */
void exp_plan(int nloc, int T, int L, const std::vector<PhysTerm> &terms, std::vector<ExpSweep> &out);
/* partner shards fetched: one per run of sweeps with the same non-zero xr */
uint32_t count_exchanges(const std::vector<ExpSweep> &sw);

/* ---- rotation grouping and launch tables of pauli_rot.cu */
#define ROT_THREADS 256
#define ROT_TB 8                      /* thread bits of the tile coordinate */
#define ROT_KMAX 1024                 /* rotations per launch (one descriptor table) */

enum { ROT_DIAG = 1 };

struct RotOp {                 /* one step of a launch: a pairing rotation or a stretch of diagonal rotations */
    double c, s;               /* pairing: cos(t/2), +-sin(t/2) (the sign of Z on the own rank bits folded in) */
    uint64_t zout;             /* pairing: Z on the local bits outside the tile, unit-address bits */
    uint32_t xin, zin;         /* pairing: X / Z on the tile coordinate */
    uint32_t flags;            /* ROT_DIAG; bits 1-2: slot flip; bits 3-4: Z parity of the slot bits; bits 5-6: w, the
                                  factor -i * i^{popc(x&z)} = i^w */
    uint32_t d0;               /* diagonal stretch: its terms, grouped by pattern, at d0 + poff[p] .. d0 + poff[p + 1] */
    uint16_t poff[17];
    uint16_t pad[3];
};
static_assert(sizeof(RotOp) == 80, "RotOp is 80 bytes");

struct RotDiag {               /* one diagonal rotation of a stretch */
    double theta;              /* the angle, negated if Z on the own rank bits has odd parity */
    uint64_t zout;             /* Z on the local bits outside the tile, unit-address bits */
    uint32_t zt;               /* Z on the thread bits of the tile coordinate */
    uint32_t sp;               /* Z parity of the slot bits */
};

struct RotSweep {
    uint64_t xr = 0;               /* rank-bit flips: partner rank = rank ^ xr */
    int8_t pb[16];                 /* tile coordinate bit j -> local physical bit */
    uint64_t bmask = 0, x_out = 0; /* tile bits, local flips outside the tile */
    std::vector<uint32_t> rots;    /* indices into the rotation list, in list order */
};

/* greedy grouping of the rotation list into sweeps of T tile bits, in order */
void rot_plan(int nloc, int T, int L, const std::vector<PhysTerm> &rots, std::vector<RotSweep> &out);
/* partner shards fetched: one per sweep with xr != 0 */
uint32_t count_exchanges(const std::vector<RotSweep> &sw);
/* slot bits of a sweep: the x_out partner tile and the partner rank's tiles */
void slot_bits(const RotSweep &sw, int *so_out, int *so_rank, int *ns);
/* the launch table of one sweep of T tile bits (su = 1 for f32 units of two amplitudes): pairing rotations and
 * diagonal stretches, in list order.  op_tags / diag_tags, if given, receive one tag per op / per diagonal entry,
 * parallel to ops / diag: the rotation's position in sw.rots and in bit 31 the parity of its Z on the own rank bits
 * (0 for the op of a diagonal stretch). */
void encode_sweep(const RotSweep &sw, const std::vector<PhysTerm> &pt, const std::vector<double> &theta, int T, int su, int rank,
                  std::vector<RotOp> &ops, std::vector<RotDiag> &diag, std::vector<uint32_t> *op_tags = nullptr,
                  std::vector<uint32_t> *diag_tags = nullptr);

/* ---- dense-matrix grouping of matrix.cu */
#define MAT_KMAX 1024                 /* matrix ops per launch (one descriptor table) */

struct MatPhys {               /* one matrix op under the qubit layout, rank targets reduced to at most one */
    uint64_t tl, tr;           /* targets on local physical bits / on rank bits (bit j = rank bit j) */
    uint64_t cl, cr;           /* controls on local physical bits / on rank bits */
    int k;
    int8_t tq[8];              /* target i -> physical bit (>= nloc: rank bit tq - nloc) */
};

struct MatSweep {
    uint64_t xr = 0;               /* rank-bit target of the run: partner rank = rank ^ xr */
    int8_t pb[16];                 /* tile coordinate bit j -> local physical bit */
    uint64_t bmask = 0;            /* tile bits */
    std::vector<uint32_t> ops;     /* indices into the op list, in list order */
};

/* greedy grouping of the op list into sweeps of T tile bits, in order: a run ends at an op whose local targets do not
 * fit the tile any more, at a second rank target that differs from the run's, or at MAT_KMAX ops.  false if an op fits
 * no tile at all (more local targets outside the low bits than T - L) */
bool matrix_plan(int nloc, int T, int L, const std::vector<MatPhys> &ops, std::vector<MatSweep> &out);
