/*
 * pauli_rot.cu -- Pauli rotations a <- cos(t/2) a - i sin(t/2) (P a) on the device, in list order (DESIGN.md section 3.3).
 *
 * A rotation is a pair of logical masks (x: X or Y, z: Z or Y) and an angle; (P a)_j is the header's formula
 *   (P a)_j = i^{popc(x&z)} (-1)^{popc((j^x)&z)} a_{j^x},
 * so a rotation with x != 0 mixes each pair (j, j^x) and one with x == 0 multiplies a_j by exp(-i t sigma_j / 2),
 * sigma_j = (-1)^{popc(j&z)}.
 *
 * SWEEP.  A sweep fixes the tile bits B of expect.cu (the low `low_bits` physical bits plus chosen higher bits, 12 bits
 * f32 / 11 f64) and a flip pattern x_out of the local bits outside B, and carries a consecutive run of rotations whose
 * local x outside B is 0 or x_out (and whose x on rank bits is 0 or the sweep's xr).  The tiles t and t ^ x_out (and the
 * same two tiles of rank ^ xr) are then closed under every rotation of the run.  A CTA stages them in shared memory as
 * separate re / im planes (up to 4 x 32 KiB), applies the run in order -- one thread per amplitude pair, a barrier after
 * every rotation -- and writes its own rank's tiles back in place.  A stretch of consecutive diagonal rotations is one
 * step: per thread the angles are summed in fp64 by the pattern of their Z on the thread's varying coordinate bits, a
 * Walsh-Hadamard transform gives each amplitude's total angle, then one sincos per amplitude.  A sweep thus reads and
 * writes the local shard once, however many rotations it carries.
 *
 * SIGNS.  sigma of an amplitude = Z on the tile coordinate, Z on the tile's outer bits (one parity per CTA and
 * rotation), Z on the slot (partner tile / partner rank, precomputed per rotation), Z on the own rank bits (folded into
 * the sine or the angle on the host).  -i * i^{popc(x&z)} = i^{(popc(x&z) + 3) & 3} is a swap of re / im and a sign.
 *
 * GROUPING.  rot_plan() (host only, no CUDA: qsb_pauli_rotation_dry_run calls it on a CPU) walks the list in order.  A
 * sweep takes the next rotation and keeps taking rotations while they fit: the first local x outside the tile becomes
 * x_out for free; any other one adds the fewest tile bits that make it 0 or x_out outside the tile, while the tile has
 * room.  Diagonal rotations always fit.  A run ends at a rotation that does not fit, at a second non-zero xr, or at
 * ROT_KMAX rotations (the per-launch descriptor table).  Commuting rotations are never reordered.
 *
 * SHARDED.  Before every sweep with xr != 0 the partner shard rank ^ xr is received into state2 with one NCCL
 * send / recv pair on the handle's stream; the partner rewrites its shard in the same sweep, so the copy is not reused.
 * The kernel is ordered after the send on the stream, so a rank overwrites its shard only once the partner has it.  A
 * call that fetched a partner shard ends with an all-reduce on the stream, so no peer's later fused exchange writes into
 * state2 while it is still read.  state / state2 are not swapped and the peer mappings are not touched.
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

#define ROT_UNITS 2048                /* 16-byte units per tile: 2^12 f32 / 2^11 f64 amplitudes, 32 KiB */
#define ROT_UB 11                     /* log2(ROT_UNITS) */

/* a sweep reads pb[0..T-1], which exist because every shard has nloc >= tiled_min_local_bits() = QSB_T_* local bits */
static_assert(12 <= QSB_T_F32 && 11 <= QSB_T_F64, "the rotation tile must fit the smallest shard");

struct RotArgs {
    uint4 *A;                  /* own shard, read and written */
    const uint4 *B;            /* partner shard (state2) of a sweep with xr != 0 */
    const RotOp *ops;
    const RotDiag *diag;
    uint64_t uoff[ROT_UB];     /* unit-address offset of tile unit bit i */
    uint64_t x_out;            /* partner tile = tile ^ x_out (unit-address bits) */
    uint64_t n_work;           /* tile groups */
    int8_t opos[64];           /* group index bit i -> unit-address bit */
    int n_opos, K;
    int ns;                    /* slots: 1, 2 or 4 tiles */
    int so_out, so_rank;       /* slot bit of the x_out partner tile / of the partner rank (0: none) */
};

/* ================================================================================================ device */

template <typename R> struct RotVec;
template <> struct RotVec<float> { static constexpr int T = 12; };
template <> struct RotVec<double> { static constexpr int T = 11; };

template <typename R>
__global__ void __launch_bounds__(ROT_THREADS) k_pauli_rot(const __grid_constant__ RotArgs a)
{
    constexpr int T = RotVec<R>::T;
    extern __shared__ uint4 s_raw[];
    R *sre = reinterpret_cast<R *>(s_raw), *sim = sre + ((size_t)a.ns << T);
    const uint32_t tid = threadIdx.x;
    uint64_t toff = 0;
#pragma unroll
    for (int i = 0; i < ROT_TB; i++) if ((tid >> i) & 1) toff |= a.uoff[i];
    for (uint64_t t = blockIdx.x; t < a.n_work; t += gridDim.x) {
        uint64_t base = 0;
        for (int i = 0; i < a.n_opos; i++) base |= ((t >> i) & 1ULL) << a.opos[i];
        for (int slot = 0; slot < a.ns; slot++)
            stage_tile<R, ROT_UB>(sre, sim, (slot & a.so_rank) ? a.B : a.A, (base ^ ((slot & a.so_out) ? a.x_out : 0)) | toff, a.uoff, slot, tid);
        __syncthreads();
        for (int j = 0; j < a.K; j++) {
            const RotOp &op = a.ops[j];
            if (op.flags & ROT_DIAG) rot_diag<R, T>(sre, sim, op, a.diag, base, a.ns, tid);
            else rot_pairs<R, T>(sre, sim, op, base, a.ns, tid);
            __syncthreads();
        }
        for (int slot = 0; slot < a.ns; slot++)
            if (!(slot & a.so_rank))   /* the partner rank writes its own tiles */
                store_tile<R, ROT_UB>(a.A, sre, sim, (base ^ ((slot & a.so_out) ? a.x_out : 0)) | toff, a.uoff, slot, tid);
        __syncthreads();   /* the next tile group overwrites the planes */
    }
}

/* ================================================================================================ host */

/* Greedy grouping of the rotation list into sweeps, in order (host only, no CUDA). */
void rot_plan(int nloc, int T, int L, const std::vector<PhysTerm> &rots, std::vector<RotSweep> &out)
{
    const uint64_t low = (1ULL << L) - 1;
    const int cap = T - L;
    size_t i = 0;
    while (i < rots.size()) {
        RotSweep sw;
        uint64_t H = 0, xout = 0;
        for (; i < rots.size() && sw.rots.size() < ROT_KMAX; i++) {
            const PhysTerm &r = rots[i];
            if (r.xr && sw.xr && r.xr != sw.xr) break;
            const uint64_t rem = r.xl & ~low & ~H;
            if (rem && rem != xout) {
                if (!xout) xout = rem;   /* the one flip pattern outside the tile costs no tile bit */
                else {                   /* absorb rem into the tile, or make it equal x_out outside the tile */
                    const uint64_t add = __builtin_popcountll(rem) <= __builtin_popcountll(rem ^ xout) ? rem : rem ^ xout;
                    if (__builtin_popcountll(H | add) > cap) break;
                    H |= add;
                    xout &= ~H;
                }
            }
            if (r.xr) sw.xr = r.xr;
            sw.rots.push_back((uint32_t)i);
        }
        /* fill the tile up to T bits: bits of x_out first (fewer tiles to stage), then the lowest free bits */
        for (uint64_t r = xout; r && __builtin_popcountll(H) < cap; r &= r - 1) H |= r & -r;
        for (int b = L; b < nloc && __builtin_popcountll(H) < cap; b++) if (!((H >> b) & 1)) H |= 1ULL << b;
        xout &= ~H;
        sw.bmask = low | H;
        sw.x_out = xout;
        int j = 0;
        for (int b = 0; b < nloc; b++) if ((sw.bmask >> b) & 1) sw.pb[j++] = (int8_t)b;
        out.push_back(std::move(sw));
    }
}

uint32_t count_exchanges(const std::vector<RotSweep> &sw)
{
    uint32_t n = 0;
    for (auto &s : sw) n += s.xr != 0;
    return n;
}

void slot_bits(const RotSweep &sw, int *so_out, int *so_rank, int *ns)
{
    *so_out = sw.x_out ? 1 : 0;
    *so_rank = sw.xr ? (sw.x_out ? 2 : 1) : 0;
    *ns = 1 << ((sw.x_out ? 1 : 0) + (sw.xr ? 1 : 0));
}

void encode_sweep(const RotSweep &sw, const std::vector<PhysTerm> &pt, const std::vector<double> &theta, int T, int su, int rank,
                  std::vector<RotOp> &ops, std::vector<RotDiag> &diag, std::vector<uint32_t> *op_tags, std::vector<uint32_t> *diag_tags)
{
    const int NI = 1 << (T - ROT_TB);
    int so_out, so_rank, ns;
    slot_bits(sw, &so_out, &so_rank, &ns);
    size_t k = 0;
    while (k < sw.rots.size()) {
        RotOp op; memset(&op, 0, sizeof op);
        const PhysTerm &p = pt[sw.rots[k]];
        if (!p.xl && !p.xr) {   /* a stretch of diagonal rotations, grouped by pattern */
            op.flags = ROT_DIAG;
            op.d0 = (uint32_t)diag.size();
            std::vector<std::vector<RotDiag>> by(NI);
            std::vector<std::vector<uint32_t>> tag_by(NI);
            for (; k < sw.rots.size() && !pt[sw.rots[k]].xl && !pt[sw.rots[k]].xr; k++) {
                const PhysTerm &d = pt[sw.rots[k]];
                const uint32_t zin = tile_coord(d.zl, sw.pb, T);
                RotDiag e;
                e.theta = parity64((uint64_t)rank & d.zr) ? -theta[sw.rots[k]] : theta[sw.rots[k]];
                e.zout = (d.zl & ~sw.bmask) >> su;
                e.zt = zin & ((1u << ROT_TB) - 1);
                e.sp = (uint32_t)(parity64(sw.x_out & d.zl) * so_out + parity64(sw.xr & d.zr) * so_rank);
                by[zin >> ROT_TB].push_back(e);
                tag_by[zin >> ROT_TB].push_back((uint32_t)k | (uint32_t)parity64((uint64_t)rank & d.zr) << 31);
            }
            for (int q = 0; q < NI; q++) {
                op.poff[q + 1] = (uint16_t)(op.poff[q] + by[q].size());
                diag.insert(diag.end(), by[q].begin(), by[q].end());
                if (diag_tags) diag_tags->insert(diag_tags->end(), tag_by[q].begin(), tag_by[q].end());
            }
        } else {
            const double t = theta[sw.rots[k]];
            op.c = cos(0.5 * t);
            op.s = parity64((uint64_t)rank & p.zr) ? -sin(0.5 * t) : sin(0.5 * t);
            op.xin = tile_coord(p.xl, sw.pb, T);
            op.zin = tile_coord(p.zl, sw.pb, T);
            op.zout = (p.zl & ~sw.bmask) >> su;
            const uint32_t flip = ((p.xl & ~sw.bmask) ? so_out : 0) | (p.xr ? so_rank : 0);
            const uint32_t sp = (uint32_t)(parity64(sw.x_out & p.zl) * so_out + parity64(sw.xr & p.zr) * so_rank);
            op.flags = flip << 1 | sp << 3 | (uint32_t)((p.y + 3) & 3) << 5;
            if (op_tags) op_tags->push_back((uint32_t)k | (uint32_t)parity64((uint64_t)rank & p.zr) << 31);
            k++;
        }
        if (op_tags && (op.flags & ROT_DIAG)) op_tags->push_back(0);
        ops.push_back(op);
    }
}

namespace {

struct DevMem {   /* scoped device allocation */
    void *p = nullptr;
    ~DevMem() { if (p) cudaFree(p); }
};

}  // namespace

/* ------------------------------------------------------------------------------------------- C ABI */

extern "C" int qsb_pauli_rotation_dry_run(int num_qubits, const qsb_options_t *opt_in, const uint64_t *x, const uint64_t *z,
                                          size_t n, uint32_t *sweeps, uint32_t *exchanges)
{
    qsb_options_t opt;
    int nloc;
    int rc = pauli_dry_run_shape(num_qubits, opt_in, &opt, &nloc);
    if (rc) return rc;
    rc = check_terms(num_qubits, x, z, n, "qsb_pauli_rotation_dry_run");
    if (rc) return rc;
    BitPerm id; for (int q = 0; q < 64; q++) id.pos[q] = (int8_t)q;
    int T, L;
    exp_geometry(opt.precision, &opt, &T, &L);
    std::vector<PhysTerm> pt;
    to_physical(num_qubits, nloc, id, x, z, n, pt);
    std::vector<RotSweep> sw;
    rot_plan(nloc, T, L, pt, sw);
    if (sweeps) *sweeps = (uint32_t)sw.size();
    if (exchanges) *exchanges = count_exchanges(sw);
    return QSB_OK;
}

extern "C" int qsb_apply_pauli_rotations(qsb_t *s, const uint64_t *x, const uint64_t *z, const double *theta, size_t n)
{
    if (!s) { qsb_set_error("qsb_apply_pauli_rotations: null handle"); return QSB_ERR_ARG; }
    if (n == 0) return QSB_OK;
    if (!theta) { qsb_set_error("qsb_apply_pauli_rotations: null angle array"); return QSB_ERR_ARG; }
    int rc = check_terms(s->n, x, z, n, "qsb_apply_pauli_rotations");
    if (rc) return rc;
    for (size_t i = 0; i < n; i++)
        if (!isfinite(theta[i])) { qsb_set_error("qsb_apply_pauli_rotations: rotation %zu has a non-finite angle", i); return QSB_ERR_ARG; }
    if (s->g && !s->comm) { qsb_set_error("qsb_apply_pauli_rotations: sharded state needs qsb_comm_init first"); return QSB_ERR_COMM; }
    /* theta == 0 is the identity: skipped, so the state keeps its bytes */
    std::vector<uint64_t> ax, az;
    std::vector<double> at;
    for (size_t i = 0; i < n; i++)
        if (theta[i] != 0.0) { ax.push_back(x[i]); az.push_back(z[i]); at.push_back(theta[i]); }
    if (at.empty()) return QSB_OK;
    QSB_CUDA(cudaSetDevice(s->device));
    const bool f32 = s->prec == QSB_F32;
    int T, L;
    exp_geometry(s->prec, &s->opt, &T, &L);
    std::vector<PhysTerm> pt;
    to_physical(s->n, s->nloc, s->perm, ax.data(), az.data(), at.size(), pt);
    std::vector<RotSweep> sw;
    rot_plan(s->nloc, T, L, pt, sw);

    /* one table for every launch, uploaded once */
    std::vector<RotOp> ops;
    std::vector<RotDiag> diag;
    std::vector<size_t> op0;
    for (auto &w : sw) { op0.push_back(ops.size()); encode_sweep(w, pt, at, T, f32 ? 1 : 0, s->rank, ops, diag); }
    op0.push_back(ops.size());
    const size_t ops_bytes = ops.size() * sizeof(RotOp), diag_bytes = diag.size() * sizeof(RotDiag);
    DevMem mem;
    QSB_CUDA(cudaMalloc(&mem.p, ops_bytes + diag_bytes + 16));
    RotOp *d_ops = (RotOp *)mem.p;
    RotDiag *d_diag = (RotDiag *)((char *)mem.p + ops_bytes);
    QSB_CUDA(cudaMemcpyAsync(d_ops, ops.data(), ops_bytes, cudaMemcpyHostToDevice, s->stream));
    if (diag_bytes) QSB_CUDA(cudaMemcpyAsync(d_diag, diag.data(), diag_bytes, cudaMemcpyHostToDevice, s->stream));

    int nsm = 0, occ = 0;
    QSB_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, s->device));
    const int smem_max = 4 * ROT_UNITS * 16;
    if (f32) QSB_CUDA(cudaFuncSetAttribute(k_pauli_rot<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
    else QSB_CUDA(cudaFuncSetAttribute(k_pauli_rot<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
    const int su = f32 ? 1 : 0, nouter = s->nloc - T;
    for (size_t k = 0; k < sw.size(); k++) {
        const RotSweep &w = sw[k];
        if (w.xr) {   /* the partner's shard as it is before this sweep; ordered after the previous sweep's writes */
            rc = tiled_comm_sendrecv(s, s->state, s->state2, s->state_bytes, s->rank ^ (int)w.xr);
            if (rc) { cudaStreamSynchronize(s->stream); return rc; }
        }
        RotArgs a; memset(&a, 0, sizeof a);
        a.A = (uint4 *)s->state;
        a.B = (const uint4 *)(w.xr ? s->state2 : s->state);
        a.ops = d_ops + op0[k];
        a.diag = d_diag;
        a.K = (int)(op0[k + 1] - op0[k]);
        for (int i = 0; i < ROT_UB; i++) a.uoff[i] = (1ULL << w.pb[su + i]) >> su;
        a.x_out = w.x_out >> su;
        slot_bits(w, &a.so_out, &a.so_rank, &a.ns);
        const int skip = w.x_out ? 63 - __builtin_clzll(w.x_out) : -1;   /* the group (t, t ^ x_out) from the t with this bit 0 */
        for (int b = 0; b < s->nloc; b++)
            if (!((w.bmask >> b) & 1) && b != skip) a.opos[a.n_opos++] = (int8_t)(b - su);
        a.n_work = 1ULL << (nouter - (w.x_out ? 1 : 0));
        const size_t smem = (size_t)a.ns * ROT_UNITS * 16;
        if (f32) QSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_pauli_rot<float>, ROT_THREADS, smem));
        else QSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_pauli_rot<double>, ROT_THREADS, smem));
        const int grid = (int)std::min<uint64_t>(a.n_work, (uint64_t)nsm * std::max(occ, 1));
        if (f32) k_pauli_rot<float><<<grid, ROT_THREADS, smem, s->stream>>>(a);
        else k_pauli_rot<double><<<grid, ROT_THREADS, smem, s->stream>>>(a);
        QSB_CUDA(cudaGetLastError());
    }
    /* a peer's fused exchange scatters into this rank's state2 without waiting: once the partner shards are read, an
     * all-reduce on the stream orders this call before any later use of state2 by a peer */
    if (count_exchanges(sw)) {
        void *flag = (char *)mem.p + ops_bytes + diag_bytes;
        QSB_CUDA(cudaMemsetAsync(flag, 0, 8, s->stream));
        rc = tiled_comm_allreduce_sum_u64(s, flag, 1);
        if (rc) { cudaStreamSynchronize(s->stream); return rc; }
    }
    /* the table is freed on return: wait for the launches that read it */
    QSB_CUDA(cudaStreamSynchronize(s->stream));
    return QSB_OK;
}
