/*
 * matrix.cu -- dense k-qubit matrices a'[j with targets = r] = sum_c m[r][c] a[j with targets = c] on the device, in
 * list order, k = 1..QSB_MATRIX_MAX_K, optionally controlled (DESIGN.md section 3.3).
 *
 * SWEEP.  A sweep fixes the tile bits B of expect.cu (the low `low_bits` physical bits plus chosen higher bits, 12 bits
 * f32 / 11 f64) and carries a consecutive run of ops whose local targets all lie in B (and whose rank target, if any, is
 * the sweep's xr).  Each tile is then closed under every op of the run.  A CTA stages the tile (and, when xr != 0, the
 * same tile of the partner rank as a second slot) in shared memory as re / im planes, applies the run in order and writes
 * its own rank's tile back in place.  A sweep thus reads and writes the local shard once, however many ops it carries.
 *
 * OP STEP.  The op space of a sweep is the ns << T staged amplitudes, m = slot << T | tile coordinate; a target is a
 * tile coordinate bit or the slot bit T.  Rows are split across threads: a work item is one group (the 2^k amplitudes
 * that differ only in the targets) and a block of RB consecutive rows, and the items are numbered row block major so the
 * 32 lanes of a warp share their rows (the matrix loads are warp-uniform) and differ in their group.  Each thread
 * accumulates its ns << T / 256 outputs in registers over the columns in order c = 0, 1, ..., 2^k - 1 (a fixed-order sum),
 * then a barrier, the in-place write, and a second barrier before the next op reads.
 *
 * CONTROLS.  On a tile bit: a condition on the group's coordinate (controls are never targets, so a group agrees on
 * them).  On a local bit outside the tile: a condition on the tile's base, the same for the whole CTA.  On a rank bit:
 * decided on the host per rank -- an op whose control fails on this rank is left out of this rank's table (the sweeps
 * and exchanges stay the same on every rank) -- except on the sweep's own rank target bit, which is the slot bit.
 *
 * SHARDED.  Before every sweep with xr != 0 the partner shard rank ^ xr is received into state2 with one NCCL
 * send / recv pair on the handle's stream, as in pauli_rot.cu.  On a rank whose bit of xr is 1 the slot bit reads the
 * complement of the qubit's value, so that op's matrix is uploaded with that index bit flipped in rows and columns.  An
 * op with m >= 2 rank targets is rewritten on the host as SWAP(r_i, l_i) ... U' ... SWAP(r_i, l_i), i = 2..m, with local
 * stand-ins l_i (see expand()).  A call that fetched a partner shard ends with an all-reduce on the stream, so no peer's
 * later fused exchange writes into state2 while it is still read.  state / state2 are not swapped and the peer mappings
 * are not touched.
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "pauli.h"
#include "pauli_rot.cuh"
#include "sim.h"
#include "tiled.h"

int tiled_comm_sendrecv(qsb_sim *s, const void *dsend, void *drecv, size_t bytes, int peer);
int tiled_comm_allreduce_sum_u64(qsb_sim *s, void *dbuf, size_t count);

#define MAT_UNITS 2048                /* 16-byte units per tile: 2^12 f32 / 2^11 f64 amplitudes, 32 KiB */
#define MAT_UB 11                     /* log2(MAT_UNITS) */

static_assert(12 <= QSB_T_F32 && 11 <= QSB_T_F64, "the matrix tile must fit the smallest shard");

struct MatOp {                 /* one op of a launch */
    uint64_t cout;             /* controls on the local bits outside the tile, unit-address bits */
    uint32_t cmask, cval;      /* controls on the op space (tile coordinate bits, slot bit T): m & cmask == cval */
    uint32_t moff;             /* first complex entry of its matrix in the matrix table */
    int32_t k;
    int8_t tpos[8];            /* target i -> op-space bit */
    int8_t spos[8];            /* the target bits, ascending */
};

struct MatArgs {
    uint4 *A;                  /* own shard, read and written */
    const uint4 *B;            /* partner shard (state2) of a sweep with xr != 0 */
    const MatOp *ops;
    const void *mats;          /* matrices, (re, im) pairs in the state's precision */
    uint64_t uoff[MAT_UB];     /* unit-address offset of tile unit bit i */
    uint64_t n_work;           /* tiles */
    int8_t opos[64];           /* tile index bit i -> unit-address bit */
    int n_opos, K;
};

/* ================================================================================================ device */

template <typename R> struct MatVec;
template <> struct MatVec<float> { static constexpr int T = 12; };
template <> struct MatVec<double> { static constexpr int T = 11; };

/* one op on the staged planes: NS slots of 2^T amplitudes, K targets */
template <typename R, int T, int K, int NS>
__device__ __forceinline__ void mat_step(R *sre, R *sim, const MatOp &op, const R *__restrict__ mat, uint32_t tid)
{
    constexpr int D = 1 << K;
    constexpr int P = (NS << T) / ROT_THREADS;   /* outputs per thread */
    constexpr int RB = D < 8 ? D : 8;            /* rows per work item */
    constexpr int IT = P / RB;                   /* work items per thread */
    constexpr uint32_t NG = (uint32_t)(NS << T) >> K;   /* groups; >= 32, so a warp shares its row block */
    static_assert(NG >= 32, "a warp must share its row block");
    uint32_t toff[K], spos[K];
#pragma unroll
    for (int i = 0; i < K; i++) { toff[i] = 1u << op.tpos[i]; spos[i] = (uint32_t)op.spos[i]; }
    R ar[IT][RB], ai[IT][RB];
    uint32_t mb[IT], r0[IT];
#pragma unroll
    for (int it = 0; it < IT; it++) {
        const uint32_t w = tid + (uint32_t)it * ROT_THREADS;
        uint32_t m = w % NG;
#pragma unroll
        for (int j = 0; j < K; j++) m = ((m >> spos[j]) << (spos[j] + 1)) | (m & ((1u << spos[j]) - 1));
        mb[it] = m;
        r0[it] = (w / NG) * RB;
        const R *row = mat + 2 * (size_t)r0[it] * D;
#pragma unroll
        for (int j = 0; j < RB; j++) { ar[it][j] = (R)0; ai[it][j] = (R)0; }
#pragma unroll 4
        for (int c = 0; c < D; c++) {
            uint32_t mc = m;
#pragma unroll
            for (int i = 0; i < K; i++) mc |= (c >> i) & 1 ? toff[i] : 0u;
            const R xr = sre[mc], xi = sim[mc];
#pragma unroll
            for (int j = 0; j < RB; j++) {
                R mr, mi;
                if (sizeof(R) == 4) {   /* (re, im) in one load; f64 keeps two, a 16-byte load spills the one-slot kernel */
                    const float2 e = __ldg(reinterpret_cast<const float2 *>(row) + j * D + c);
                    mr = (R)e.x; mi = (R)e.y;
                } else { mr = __ldg(row + 2 * (j * D + c)); mi = __ldg(row + 2 * (j * D + c) + 1); }
                ar[it][j] = fma(mr, xr, ar[it][j]); ar[it][j] = fma(-mi, xi, ar[it][j]);
                ai[it][j] = fma(mr, xi, ai[it][j]); ai[it][j] = fma(mi, xr, ai[it][j]);
            }
        }
    }
    __syncthreads();   /* every input of the op is read: write in place */
#pragma unroll
    for (int it = 0; it < IT; it++) {
        if ((mb[it] & op.cmask) != op.cval) continue;   /* a control on the group fails: the amplitudes stay */
#pragma unroll
        for (int j = 0; j < RB; j++) {
            const uint32_t r = r0[it] + j;
            uint32_t mr = mb[it];
#pragma unroll
            for (int i = 0; i < K; i++) if ((r >> i) & 1) mr |= toff[i];
            sre[mr] = ar[it][j];
            sim[mr] = ai[it][j];
        }
    }
}

template <typename R, int NS>
__global__ void __launch_bounds__(ROT_THREADS, 3 - NS) k_matrix(const __grid_constant__ MatArgs a)
{
    constexpr int T = MatVec<R>::T;
    extern __shared__ uint4 s_raw[];
    R *sre = reinterpret_cast<R *>(s_raw), *sim = sre + ((size_t)NS << T);
    const R *mats = reinterpret_cast<const R *>(a.mats);
    const uint32_t tid = threadIdx.x;
    uint64_t toff = 0;
#pragma unroll
    for (int i = 0; i < ROT_TB; i++) if ((tid >> i) & 1) toff |= a.uoff[i];
    for (uint64_t t = blockIdx.x; t < a.n_work; t += gridDim.x) {
        uint64_t base = 0;
        for (int i = 0; i < a.n_opos; i++) base |= ((t >> i) & 1ULL) << a.opos[i];
#pragma unroll
        for (int slot = 0; slot < NS; slot++)
            stage_tile<R, MAT_UB>(sre, sim, slot ? a.B : a.A, base | toff, a.uoff, slot, tid);
        __syncthreads();
        for (int j = 0; j < a.K; j++) {
            const MatOp &op = a.ops[j];
            if ((base & op.cout) != op.cout) continue;   /* the same for the whole CTA */
            const R *m = mats + 2 * (size_t)op.moff;
            switch (op.k) {
            case 1: mat_step<R, T, 1, NS>(sre, sim, op, m, tid); break;
            case 2: mat_step<R, T, 2, NS>(sre, sim, op, m, tid); break;
            case 3: mat_step<R, T, 3, NS>(sre, sim, op, m, tid); break;
            case 4: mat_step<R, T, 4, NS>(sre, sim, op, m, tid); break;
            case 5: mat_step<R, T, 5, NS>(sre, sim, op, m, tid); break;
            default: mat_step<R, T, 6, NS>(sre, sim, op, m, tid); break;
            }
            __syncthreads();
        }
        store_tile<R, MAT_UB>(a.A, sre, sim, base | toff, a.uoff, 0, tid);   /* the partner rank writes its own tile */
        __syncthreads();   /* the next tile overwrites the planes */
    }
}

/* ================================================================================================ host */

/* Greedy grouping of the op list into sweeps, in order (host only, no CUDA).  false, with out incomplete, if an op's local
 * targets outside the low bits alone do not fit the T - L free tile bits (never with a low_bits the callers accept). */
bool matrix_plan(int nloc, int T, int L, const std::vector<MatPhys> &ops, std::vector<MatSweep> &out)
{
    const uint64_t low = (1ULL << L) - 1;
    const int cap = T - L;
    size_t i = 0;
    while (i < ops.size()) {
        MatSweep sw;
        uint64_t H = 0;
        for (; i < ops.size() && sw.ops.size() < MAT_KMAX; i++) {
            const MatPhys &o = ops[i];
            if (o.tr && sw.xr && o.tr != sw.xr) break;
            const uint64_t add = o.tl & ~low & ~H;
            if (__builtin_popcountll(H | add) > cap) break;
            H |= add;
            if (o.tr) sw.xr = o.tr;
            sw.ops.push_back((uint32_t)i);
        }
        if (sw.ops.empty()) return false;   /* the op at i fits no tile: a run must take at least one op */
        for (int b = L; b < nloc && __builtin_popcountll(H) < cap; b++) if (!((H >> b) & 1)) H |= 1ULL << b;
        sw.bmask = low | H;
        int j = 0;
        for (int b = 0; b < nloc; b++) if ((sw.bmask >> b) & 1) sw.pb[j++] = (int8_t)b;
        out.push_back(std::move(sw));
    }
    return true;
}

namespace {

/* SWAP of (a, b) with a = bit 0 of the index: |01> <-> |10> */
const double k_swap[32] = {1, 0, 0, 0, 0, 0, 0, 0,
                           0, 0, 0, 0, 1, 0, 0, 0,
                           0, 0, 1, 0, 0, 0, 0, 0,
                           0, 0, 0, 0, 0, 0, 1, 0};

struct MatLog {                /* one op of the expanded list, logical qubits */
    uint64_t ctrl;
    int k;
    int t[QSB_MATRIX_MAX_K];
    const double *m;           /* NULL in a dry run */
};

int check_ops(int n, const qsb_matrix_op_t *ops, size_t count, bool need_m, const char *fn)
{
    if (count && !ops) { qsb_set_error("%s: null ops array", fn); return QSB_ERR_ARG; }
    const int kmax = std::min(n, QSB_MATRIX_MAX_K);
    const uint64_t all = n >= 64 ? ~0ULL : (1ULL << n) - 1;
    for (size_t i = 0; i < count; i++) {
        const qsb_matrix_op_t &o = ops[i];
        if (o.flags) { qsb_set_error("%s: op %zu has flags %d, expected 0", fn, i, (int)o.flags); return QSB_ERR_ARG; }
        if (o.k < 1 || o.k > kmax) { qsb_set_error("%s: op %zu has %d targets, expected 1..%d", fn, i, (int)o.k, kmax); return QSB_ERR_ARG; }
        uint64_t seen = 0;
        for (int j = 0; j < o.k; j++) {
            const int q = o.targets[j];
            if (q < 0 || q >= n) { qsb_set_error("%s: op %zu has target %d outside [0, %d)", fn, i, q, n); return QSB_ERR_ARG; }
            if ((seen >> q) & 1) { qsb_set_error("%s: op %zu has target %d twice", fn, i, q); return QSB_ERR_ARG; }
            seen |= 1ULL << q;
        }
        if (o.controls & ~all) {
            qsb_set_error("%s: op %zu has a control >= %d (controls = 0x%llx)", fn, i, n, (unsigned long long)o.controls);
            return QSB_ERR_ARG;
        }
        if (o.controls & seen) {
            qsb_set_error("%s: op %zu has qubit %d as both a control and a target", fn, i, __builtin_ctzll(o.controls & seen));
            return QSB_ERR_ARG;
        }
        if (!need_m) continue;
        if (!o.m) { qsb_set_error("%s: op %zu has a null matrix", fn, i); return QSB_ERR_ARG; }
        const size_t cnt = (size_t)2 << (2 * o.k);
        for (size_t e = 0; e < cnt; e++)
            if (!isfinite(o.m[e])) { qsb_set_error("%s: op %zu has a non-finite entry at %zu", fn, i, e); return QSB_ERR_ARG; }
    }
    return QSB_OK;
}

/* The op list with every op of m >= 2 rank targets rewritten as SWAP(r_i, l_i) ... U' ... SWAP(r_i, l_i), i = 2..m:
 * target r_i of U is replaced by l_i, the lowest-placed local qubit that is neither a target nor a control of the op
 * (nor an earlier stand-in), and each SWAP has the single rank target r_i. */
int expand(int n, int nloc, const BitPerm &perm, const qsb_matrix_op_t *ops, size_t count, bool with_m, const char *fn,
           std::vector<MatLog> &out)
{
    int inv[64];
    for (int p = 0; p < 64; p++) inv[p] = -1;
    for (int q = 0; q < n; q++) inv[perm.pos[q]] = q;
    for (size_t i = 0; i < count; i++) {
        const qsb_matrix_op_t &o = ops[i];
        MatLog u;
        u.ctrl = o.controls;
        u.k = o.k;
        u.m = with_m ? o.m : nullptr;
        uint64_t busy = o.controls;
        for (int j = 0; j < o.k; j++) { u.t[j] = o.targets[j]; busy |= 1ULL << o.targets[j]; }
        std::vector<std::pair<int, int>> sw;   /* (rank qubit, stand-in) */
        bool first = true;
        for (int j = 0; j < o.k; j++) {
            if (perm.pos[o.targets[j]] < nloc) continue;
            if (first) { first = false; continue; }   /* the first rank target stays */
            int l = -1;
            for (int p = 0; p < nloc && l < 0; p++) if (inv[p] >= 0 && !((busy >> inv[p]) & 1)) l = inv[p];
            if (l < 0) {
                qsb_set_error("%s: op %zu has several targets on rank qubits and no free local qubit to stand in for "
                              "target %d (every local qubit is a target or a control of the op)", fn, i, o.targets[j]);
                return QSB_ERR_ARG;
            }
            busy |= 1ULL << l;
            sw.push_back({o.targets[j], l});
            u.t[j] = l;
        }
        for (auto &p : sw) out.push_back(MatLog{0, 2, {p.first, p.second}, with_m ? k_swap : nullptr});
        out.push_back(u);
        for (size_t j = sw.size(); j-- > 0;) out.push_back(MatLog{0, 2, {sw[j].first, sw[j].second}, with_m ? k_swap : nullptr});
    }
    return QSB_OK;
}

void to_phys(int nloc, const BitPerm &perm, const std::vector<MatLog> &lg, std::vector<MatPhys> &out)
{
    out.resize(lg.size());
    for (size_t i = 0; i < lg.size(); i++) {
        MatPhys p; memset(&p, 0, sizeof p);
        p.k = lg[i].k;
        for (int j = 0; j < p.k; j++) {
            const int b = perm.pos[lg[i].t[j]];
            p.tq[j] = (int8_t)b;
            if (b < nloc) p.tl |= 1ULL << b; else p.tr |= 1ULL << (b - nloc);
        }
        for (uint64_t c = lg[i].ctrl; c; c &= c - 1) {
            const int b = perm.pos[__builtin_ctzll(c)];
            if (b < nloc) p.cl |= 1ULL << b; else p.cr |= 1ULL << (b - nloc);
        }
        out[i] = p;
    }
}

/* The tile geometry of a precision and options, refusing a low_bits outside the range the tile scheduler accepts (f32
 * 3..6, f64 2..5, 0 = the default): in that range T - L >= QSB_MATRIX_MAX_K, so every op fits one tile. */
int matrix_geometry(int prec, const qsb_options_t *opt, int *T, int *L, const char *fn)
{
    const int rc = check_low_bits(prec, opt, fn);
    if (rc) return rc;
    exp_geometry(prec, opt, T, L);
    if (*T - *L < QSB_MATRIX_MAX_K) { qsb_set_error("%s: internal: %d free tile bits", fn, *T - *L); return QSB_ERR_ARG; }
    return QSB_OK;
}

/* the grouping, or QSB_ERR_ARG if an op fits no tile (matrix_geometry rules that out) */
int plan_or_refuse(int nloc, int T, int L, const std::vector<MatPhys> &ph, std::vector<MatSweep> &sw, const char *fn)
{
    if (matrix_plan(nloc, T, L, ph, sw)) return QSB_OK;
    qsb_set_error("%s: internal: an op needs more than the %d free tile bits", fn, T - L);
    return QSB_ERR_ARG;
}

uint32_t count_exchanges(const std::vector<MatSweep> &sw)
{
    uint32_t n = 0;
    for (auto &s : sw) n += s.xr != 0;
    return n;
}

/* the launch table of one sweep on this rank, and the matrices (fp64 here) its ops read */
void encode(const MatSweep &sw, const std::vector<MatLog> &lg, const std::vector<MatPhys> &ph, int nloc, int T, int su, int rank,
            std::vector<MatOp> &ops, std::vector<double> &mats)
{
    for (uint32_t idx : sw.ops) {
        const MatPhys &p = ph[idx];
        const uint64_t crk = p.cr & ~sw.xr;
        if (((uint64_t)rank & crk) != crk) continue;   /* a control on this rank's bits fails: the identity here */
        const bool own1 = ((uint64_t)rank & sw.xr) != 0;   /* this rank's value of the rank target bit */
        MatOp o; memset(&o, 0, sizeof o);
        o.k = p.k;
        o.cout = (p.cl & ~sw.bmask) >> su;
        o.cmask = o.cval = tile_coord(p.cl & sw.bmask, sw.pb, T);
        if (p.cr & sw.xr) { o.cmask |= 1u << T; if (!own1) o.cval |= 1u << T; }   /* slot s holds the value own ^ s */
        uint32_t flip = 0;
        for (int j = 0; j < p.k; j++) {
            if (p.tq[j] >= nloc) { o.tpos[j] = (int8_t)T; if (own1) flip = 1u << j; continue; }
            for (int b = 0; b < T; b++) if (sw.pb[b] == p.tq[j]) o.tpos[j] = (int8_t)b;
        }
        memcpy(o.spos, o.tpos, sizeof o.spos);
        std::sort(o.spos, o.spos + p.k);
        o.moff = (uint32_t)(mats.size() / 2);
        const int D = 1 << p.k;
        const double *m = lg[idx].m;
        for (int r = 0; r < D; r++)
            for (int c = 0; c < D; c++) {
                const size_t e = 2 * ((size_t)(r ^ flip) * D + (c ^ flip));
                mats.push_back(m[e]);
                mats.push_back(m[e + 1]);
            }
        ops.push_back(o);
    }
}

struct DevMem {   /* scoped device allocation */
    void *p = nullptr;
    ~DevMem() { if (p) cudaFree(p); }
};

template <typename R, int NS>
int launch(qsb_sim *s, const MatArgs &a, int nsm)
{
    const int T = MatVec<R>::T;
    const size_t smem = (size_t)NS * sizeof(R) * 2 << T;
    QSB_CUDA(cudaFuncSetAttribute(k_matrix<R, NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    QSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_matrix<R, NS>, ROT_THREADS, smem));
    const int grid = (int)std::min<uint64_t>(a.n_work, (uint64_t)nsm * std::max(occ, 1));
    k_matrix<R, NS><<<grid, ROT_THREADS, smem, s->stream>>>(a);
    QSB_CUDA(cudaGetLastError());
    return QSB_OK;
}

}  // namespace

/* ------------------------------------------------------------------------------------------- C ABI */

extern "C" int qsb_matrix_dry_run(int num_qubits, const qsb_options_t *opt_in, const qsb_matrix_op_t *ops, size_t n,
                                  uint32_t *sweeps, uint32_t *exchanges)
{
    qsb_options_t opt;
    int nloc;
    int rc = pauli_dry_run_shape(num_qubits, opt_in, &opt, &nloc);
    if (rc) return rc;
    rc = check_ops(num_qubits, ops, n, false, "qsb_matrix_dry_run");
    if (rc) return rc;
    int T, L;
    rc = matrix_geometry(opt.precision, &opt, &T, &L, "qsb_matrix_dry_run");
    if (rc) return rc;
    BitPerm id; for (int q = 0; q < 64; q++) id.pos[q] = (int8_t)q;
    std::vector<MatLog> lg;
    rc = expand(num_qubits, nloc, id, ops, n, false, "qsb_matrix_dry_run", lg);
    if (rc) return rc;
    std::vector<MatPhys> ph;
    to_phys(nloc, id, lg, ph);
    std::vector<MatSweep> sw;
    rc = plan_or_refuse(nloc, T, L, ph, sw, "qsb_matrix_dry_run");
    if (rc) return rc;
    if (sweeps) *sweeps = (uint32_t)sw.size();
    if (exchanges) *exchanges = count_exchanges(sw);
    return QSB_OK;
}

extern "C" int qsb_apply_matrices(qsb_t *s, const qsb_matrix_op_t *ops, size_t n)
{
    static const char *fn = "qsb_apply_matrices";
    if (!s) { qsb_set_error("%s: null handle", fn); return QSB_ERR_ARG; }
    if (n == 0) return QSB_OK;
    int rc = check_ops(s->n, ops, n, true, fn);
    if (rc) return rc;
    int T, L;
    rc = matrix_geometry(s->prec, &s->opt, &T, &L, fn);
    if (rc) return rc;
    if (s->g && !s->comm) { qsb_set_error("%s: sharded state needs qsb_comm_init first", fn); return QSB_ERR_COMM; }
    std::vector<MatLog> lg;
    rc = expand(s->n, s->nloc, s->perm, ops, n, true, fn, lg);
    if (rc) return rc;
    QSB_CUDA(cudaSetDevice(s->device));
    const bool f32 = s->prec == QSB_F32;
    std::vector<MatPhys> ph;
    to_phys(s->nloc, s->perm, lg, ph);
    std::vector<MatSweep> sw;
    rc = plan_or_refuse(s->nloc, T, L, ph, sw, fn);
    if (rc) return rc;

    /* one table for every launch, uploaded once; the matrices in the state's precision */
    const int su = f32 ? 1 : 0;
    std::vector<MatOp> table;
    std::vector<double> md;
    std::vector<size_t> op0;
    for (auto &w : sw) { op0.push_back(table.size()); encode(w, lg, ph, s->nloc, T, su, s->rank, table, md); }
    op0.push_back(table.size());
    std::vector<float> mf;
    if (f32) mf.assign(md.begin(), md.end());
    const void *mhost = f32 ? (const void *)mf.data() : (const void *)md.data();
    const size_t tab_bytes = (table.size() * sizeof(MatOp) + 15) & ~(size_t)15;
    const size_t mat_bytes = (md.size() * (f32 ? sizeof(float) : sizeof(double)) + 15) & ~(size_t)15;
    DevMem mem;
    QSB_CUDA(cudaMalloc(&mem.p, tab_bytes + mat_bytes + 16));
    MatOp *d_ops = (MatOp *)mem.p;
    char *d_mats = (char *)mem.p + tab_bytes;
    if (!table.empty()) QSB_CUDA(cudaMemcpyAsync(d_ops, table.data(), table.size() * sizeof(MatOp), cudaMemcpyHostToDevice, s->stream));
    if (!md.empty()) QSB_CUDA(cudaMemcpyAsync(d_mats, mhost, md.size() * (f32 ? sizeof(float) : sizeof(double)), cudaMemcpyHostToDevice, s->stream));

    int nsm = 0;
    QSB_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, s->device));
    const int nouter = s->nloc - T;
    for (size_t k = 0; k < sw.size(); k++) {
        const MatSweep &w = sw[k];
        if (w.xr) {   /* the partner's shard as it is before this sweep; ordered after the previous sweep's writes */
            rc = tiled_comm_sendrecv(s, s->state, s->state2, s->state_bytes, s->rank ^ (int)w.xr);
            if (rc) { cudaStreamSynchronize(s->stream); return rc; }
        }
        MatArgs a; memset(&a, 0, sizeof a);
        a.A = (uint4 *)s->state;
        a.B = (const uint4 *)(w.xr ? s->state2 : s->state);
        a.ops = d_ops + op0[k];
        a.mats = d_mats;
        a.K = (int)(op0[k + 1] - op0[k]);
        for (int i = 0; i < MAT_UB; i++) a.uoff[i] = (1ULL << w.pb[su + i]) >> su;
        for (int b = 0; b < s->nloc; b++)
            if (!((w.bmask >> b) & 1)) a.opos[a.n_opos++] = (int8_t)(b - su);
        a.n_work = 1ULL << nouter;
        if (a.K == 0) continue;   /* every op of the run is the identity on this rank */
        if (f32) rc = w.xr ? launch<float, 2>(s, a, nsm) : launch<float, 1>(s, a, nsm);
        else rc = w.xr ? launch<double, 2>(s, a, nsm) : launch<double, 1>(s, a, nsm);
        if (rc) { cudaStreamSynchronize(s->stream); return rc; }
    }
    /* a peer's fused exchange scatters into this rank's state2 without waiting: once the partner shards are read, an
     * all-reduce on the stream orders this call before any later use of state2 by a peer */
    if (count_exchanges(sw)) {
        void *flag = (char *)mem.p + tab_bytes + mat_bytes;
        QSB_CUDA(cudaMemsetAsync(flag, 0, 8, s->stream));
        rc = tiled_comm_allreduce_sum_u64(s, flag, 1);
        if (rc) { cudaStreamSynchronize(s->stream); return rc; }
    }
    /* the tables are freed on return: wait for the launches that read them */
    QSB_CUDA(cudaStreamSynchronize(s->stream));
    return QSB_OK;
}
