/*
 * pauli_grad.cu -- the energy E = sum_j c_j <psi|P_j|psi> of psi = R_{n-1} ... R_0 phi_0, R_k = exp(-i theta_k P_k / 2),
 * and its gradient dE/dtheta_k = Im <lambda_k| P_k |phi_k> by the adjoint method (DESIGN.md section 3.3), with
 *   phi_k = R_k ... R_0 phi_0,   lambda_k = R_{k+1}^dag ... R_{n-1}^dag H psi.
 *
 * FORWARD.  qsb_apply_pauli_rotations leaves psi in the handle and qsb_expectation_pauli gives every <P_j>; the
 * energy is their coefficient sum on the host in term order.  psi is then copied into the scratch phi.
 *
 * LAMBDA = H psi (k_hpsi).  The terms are grouped by exp_plan() of expect.cu: a sweep fixes the tile bits and one
 * flip pattern x_out outside the tile (and one rank pattern xr), so output tile t reads only source tile t ^ x_out of
 * the shard of rank ^ xr.  A CTA stages that source tile, adds up sum_j c_j (P_j psi) for its own tile in registers, one
 * amplitude per thread and tile coordinate (m = i << ROT_TB | tid), and writes lambda; a later sweep first reads the
 * lambda tile and adds to it, so the sum is in sweep order.  The diagonal terms of a sweep are one step: per thread the
 * coefficients are summed in fp64 by the pattern of their Z on the bits of i, a Walsh-Hadamard transform gives each
 * amplitude's d_m = sum_j c_j sigma_j(m), then one multiply.  The sign of Z on the source rank's bits is folded into
 * the coefficient on the host.
 *
 * ADJOINT SWEEP (k_pauli_adj).  The rotation list is walked backwards: rot_plan() of pauli_rot.cu on the reversed list,
 * zero angles kept, with one tile bit fewer than the forward sweep (11 f32 / 10 f64), so that phi and lambda of up to
 * four slots fit a CTA's shared memory (4 slots x 2 vectors x 16 KiB).  The launch table is encode_sweep() of the
 * reversed list with negated angles, so its steps are R_k^dag.  For each step, in order:
 *   pairing rotation: the thread's pairs give sum Im(conj(lambda_j) (P_k phi)_j) over the own rank's amplitudes (a
 *     partner rank's slots are sources only); then R_k^dag is applied to phi and lambda, unless theta_k = 0;
 *   diagonal stretch: its rotations commute with each other and with their P_k, so every overlap is taken from the same
 *     (lambda, phi) before the stretch: w_m = Im(conj(lambda_m) phi_m), a Walsh-Hadamard transform over the bits of i,
 *     and each rotation reads the transform at the pattern of its Z with the signs of its other Z bits; then the
 *     stretch's inverse is applied.
 * Per rotation the thread values go through a fixed xor-tree over the warp into one fp64 accumulator per warp and
 * rotation in shared memory; k_adj_finish adds the per-CTA partials in CTA order.  No floating-point atomics.
 *
 * SHARDED.  A lambda sweep with xr != 0 first receives the partner's psi into state2 (once per distinct xr, exp_plan
 * groups them).  An adjoint sweep with xr != 0 first receives the partner's phi into state2 and its lambda into the
 * extra scratch buffer.  Per-rank gradients are all-gathered and added on the host in rank order.  A call that fetched
 * a partner shard ends with the all-reduce of qsb_apply_pauli_rotations, for the same reason.
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <array>
#include <vector>

#include "pauli.h"
#include "pauli_rot.cuh"
#include "sim.h"
#include "tiled.h"

int tiled_comm_sendrecv(qsb_sim *s, const void *dsend, void *drecv, size_t bytes, int peer);
int tiled_comm_allreduce_sum_u64(qsb_sim *s, void *dbuf, size_t count);
int tiled_comm_allgather(qsb_sim *s, const void *dsrc, void *ddst, size_t bytes);

#define HPS_UB 11                     /* lambda sweep: the tile of expect.cu, 2048 16-byte units */
#define ADJ_UB 10                     /* adjoint sweep: one tile bit fewer, 1024 units = 16 KiB per vector and slot */
#define ADJ_UNITS (1 << ADJ_UB)
#define ADJ_WARPS (ROT_THREADS / 32)
#define ADJ_SKIP (1u << 30)           /* op tag: theta = 0 (every theta of a diagonal stretch), no apply */
#define ADJ_POS 0xffffu               /* op / diagonal tag: position in the sweep */
#define GRAD_GRID_CAP 8               /* CTAs per SM at most (the partial buffer) */

static_assert(12 <= QSB_T_F32 && 11 <= QSB_T_F64, "the lambda tile must fit the smallest shard");
static_assert(ROT_KMAX <= ADJ_POS + 1, "a sweep position fits the tag");

struct HTerm {                 /* one non-diagonal term of a lambda sweep (32 bytes) */
    double c;                  /* coefficient, negated if Z on the source rank's bits has odd parity */
    uint64_t zout;             /* Z on the local bits outside the tile, unit-address bits */
    uint32_t xin, zin;         /* X / Z on the tile coordinate */
    uint32_t w, pad;           /* i^w = i^{popc(x&z)} */
};
static_assert(sizeof(HTerm) == 32, "HTerm is 32 bytes");

struct HArgs {
    const uint4 *src;          /* psi: own shard, or the partner's in state2 */
    uint4 *lam;
    const HTerm *terms;        /* K non-diagonal terms */
    const RotDiag *diag;       /* the diagonal terms (theta = coefficient), grouped by pattern at poff[p] .. poff[p + 1] */
    uint64_t uoff[HPS_UB];     /* unit-address offset of tile unit bit i */
    uint64_t x_out;            /* source tile = tile ^ x_out (unit-address bits) */
    uint64_t n_work;           /* tiles */
    uint32_t poff[17];
    int8_t opos[64];           /* tile index bit i -> unit-address bit */
    int n_opos, K, first;      /* first: write lambda instead of adding to it */
};

struct AdjArgs {
    uint4 *phi, *lam;          /* own phi / lambda, read and written */
    const uint4 *phi2, *lam2;  /* the partner rank's phi / lambda of a sweep with xr != 0 */
    const RotOp *ops;          /* R_k^dag steps */
    const RotDiag *diag;
    const uint32_t *op_tags, *diag_tags;
    double *partial;           /* [gridDim.x][nrot] */
    uint64_t uoff[ADJ_UB];
    uint64_t x_out, n_work;
    int8_t opos[64];
    int n_opos, K, nrot;       /* steps, rotations of the sweep */
    int ns, so_out, so_rank;
};

/* ================================================================================================ device */

template <typename R> struct GradVec;
template <> struct GradVec<float> { static constexpr int T = 12, TA = 11; };
template <> struct GradVec<double> { static constexpr int T = 11, TA = 10; };

template <typename R>
__global__ void __launch_bounds__(ROT_THREADS) k_hpsi(const __grid_constant__ HArgs a)
{
    constexpr int T = GradVec<R>::T, NI = 1 << (T - ROT_TB);
    extern __shared__ uint4 s_raw[];
    R *sre = reinterpret_cast<R *>(s_raw), *sim = sre + (2 << T);   /* slot 0: psi; slot 1: lambda before the sweep */
    const uint32_t tid = threadIdx.x;
    uint64_t toff = 0;
#pragma unroll
    for (int i = 0; i < ROT_TB; i++) if ((tid >> i) & 1) toff |= a.uoff[i];
    for (uint64_t t = blockIdx.x; t < a.n_work; t += gridDim.x) {
        uint64_t base = 0;
        for (int i = 0; i < a.n_opos; i++) base |= ((t >> i) & 1ULL) << a.opos[i];
        const uint64_t sbase = base ^ a.x_out;
        stage_tile<R, HPS_UB>(sre, sim, a.src, sbase | toff, a.uoff, 0, tid);
        if (!a.first) stage_tile<R, HPS_UB>(sre, sim, a.lam, base | toff, a.uoff, 1, tid);
        __syncthreads();
        R ar[NI], ai[NI];
        if (a.poff[NI] != a.poff[0]) {   /* diagonal terms: d_m = sum_p C[p] (-1)^{popc(i & p)} */
            double C[NI];
#pragma unroll
            for (int p = 0; p < NI; p++) {
                double acc = 0.0;
                for (uint32_t k = a.poff[p]; k < a.poff[p + 1]; k++) {
                    const RotDiag e = a.diag[k];
                    acc += ((__popc(tid & e.zt) + __popcll(sbase & e.zout)) & 1) ? -e.theta : e.theta;
                }
                C[p] = acc;
            }
#pragma unroll
            for (int hb = 1; hb < NI; hb <<= 1)
#pragma unroll
                for (int i = 0; i < NI; i++)
                    if (!(i & hb)) { const double u = C[i], v = C[i + hb]; C[i] = u + v; C[i + hb] = u - v; }
#pragma unroll
            for (int i = 0; i < NI; i++) {
                const uint32_t m = ((uint32_t)i << ROT_TB) | tid;
                ar[i] = (R)C[i] * sre[m];
                ai[i] = (R)C[i] * sim[m];
            }
        } else {
#pragma unroll
            for (int i = 0; i < NI; i++) { ar[i] = 0; ai[i] = 0; }
        }
        for (int j = 0; j < a.K; j++) {   /* (P psi)_m = i^w sigma(m ^ x) psi_{m ^ x} */
            const HTerm h = a.terms[j];
            const uint32_t tpar = __popcll(sbase & h.zout) & 1;
            const R c = (R)h.c;
#pragma unroll
            for (int i = 0; i < NI; i++) {
                const uint32_t ms = (((uint32_t)i << ROT_TB) | tid) ^ h.xin;
                R vr = sre[ms], vi = sim[ms];
                mul_iw(vr, vi, h.w);
                const R cs = ((__popc(ms & h.zin) + tpar) & 1) ? -c : c;
                ar[i] += cs * vr;
                ai[i] += cs * vi;
            }
        }
        if (!a.first) {
#pragma unroll
            for (int i = 0; i < NI; i++) {
                const uint32_t m = (1u << T) | ((uint32_t)i << ROT_TB) | tid;
                ar[i] = sre[m] + ar[i];
                ai[i] = sim[m] + ai[i];
            }
        }
        __syncthreads();   /* every thread is done with the source planes */
#pragma unroll
        for (int i = 0; i < NI; i++) {
            const uint32_t m = ((uint32_t)i << ROT_TB) | tid;
            sre[m] = ar[i];
            sim[m] = ai[i];
        }
        __syncthreads();
        store_tile<R, HPS_UB>(a.lam, sre, sim, base | toff, a.uoff, 0, tid);
        __syncthreads();   /* the next tile overwrites the planes */
    }
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

/* sum over the thread's pairs of Im(conj(lambda_j) (P phi)_j) for the own slots' j, without the own rank sign:
 * (P phi)_{m0} = i sigma(m1) i^w phi_{m1}, and Im(conj(l) i u) = Re(conj(l) u) */
template <typename R, int T>
__device__ __forceinline__ double adj_pair_overlap(const R *pre, const R *pim, const R *lre, const R *lim, const RotOp &op,
                                                   uint64_t base, int ns, int so_rank, uint32_t tid)
{
    const uint32_t F = ((op.flags >> 1) & 3u) << T | op.xin;
    const int h = 31 - __clz(F);
    const uint32_t lowm = (1u << h) - 1, cmask = (1u << T) - 1, sp = (op.flags >> 3) & 3u, w = (op.flags >> 5) & 3u;
    const uint32_t tpar = __popcll(base & op.zout) & 1;
    const uint32_t npairs = (uint32_t)ns << (T - 1);
    double acc = 0.0;
    for (uint32_t p = tid; p < npairs; p += ROT_THREADS) {
        const uint32_t m0 = ((p & ~lowm) << 1) | (p & lowm), m1 = m0 ^ F;
        if (!((m0 >> T) & so_rank)) {
            R ur = pre[m1], ui = pim[m1];
            mul_iw(ur, ui, w);
            const double v = (double)(lre[m0] * ur + lim[m0] * ui);
            acc += ((__popc(m1 & cmask & op.zin) + __popc((m1 >> T) & sp) + tpar) & 1) ? -v : v;
        }
        if (!((m1 >> T) & so_rank)) {
            R ur = pre[m0], ui = pim[m0];
            mul_iw(ur, ui, w);
            const double v = (double)(lre[m1] * ur + lim[m1] * ui);
            acc += ((__popc(m0 & cmask & op.zin) + __popc((m0 >> T) & sp) + tpar) & 1) ? -v : v;
        }
    }
    return acc;
}

/* every rotation of a diagonal stretch: sum over the own slots of sigma_k(m) w_m, w_m = Im(conj(lambda_m) phi_m), from
 * the Walsh-Hadamard transform of w over the bits of i; one warp sum per rotation into s_acc */
template <typename R, int T>
__device__ __forceinline__ void adj_diag_overlap(const R *pre, const R *pim, const R *lre, const R *lim, const RotOp &op,
                                                 const RotDiag *diag, const uint32_t *tags, uint64_t base, int nown,
                                                 uint32_t tid, double *s_acc_warp, bool lane0)
{
    constexpr int NI = 1 << (T - ROT_TB);
    double W[2][NI];
#pragma unroll
    for (int slot = 0; slot < 2; slot++) {
#pragma unroll
        for (int i = 0; i < NI; i++) {
            const uint32_t m = ((uint32_t)slot << T) | ((uint32_t)i << ROT_TB) | tid;
            W[slot][i] = slot < nown ? (double)lre[m] * (double)pim[m] - (double)lim[m] * (double)pre[m] : 0.0;
        }
#pragma unroll
        for (int hb = 1; hb < NI; hb <<= 1)
#pragma unroll
            for (int i = 0; i < NI; i++)
                if (!(i & hb)) { const double u = W[slot][i], v = W[slot][i + hb]; W[slot][i] = u + v; W[slot][i + hb] = u - v; }
    }
#pragma unroll
    for (int p = 0; p < NI; p++) {
        for (int k = op.poff[p]; k < op.poff[p + 1]; k++) {
            const RotDiag e = diag[op.d0 + k];
            const uint32_t tag = tags[op.d0 + k];
            double v = (e.sp & 1) ? W[0][p] - W[1][p] : W[0][p] + W[1][p];   /* slot 1 (own) is the x_out partner tile */
            if ((__popc(tid & e.zt) + __popcll(base & e.zout) + (tag >> 31)) & 1) v = -v;
            v = warp_sum(v);
            if (lane0) s_acc_warp[tag & ADJ_POS] += v;
        }
    }
}

template <typename R>
__global__ void __launch_bounds__(ROT_THREADS) k_pauli_adj(const __grid_constant__ AdjArgs a)
{
    constexpr int T = GradVec<R>::TA;
    extern __shared__ uint4 s_raw[];
    const size_t plane = (size_t)a.ns << T;
    R *pre = reinterpret_cast<R *>(s_raw), *pim = pre + plane, *lre = pim + plane, *lim = lre + plane;
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    double *s_acc = reinterpret_cast<double *>(lim + plane);   /* [ADJ_WARPS][nrot] */
    double *s_acc_warp = s_acc + (size_t)warp * a.nrot;
    for (int j = tid; j < ADJ_WARPS * a.nrot; j += ROT_THREADS) s_acc[j] = 0.0;
    const int nown = a.so_out ? 2 : 1;   /* own slots: 0 and, with an x_out partner tile, 1 */
    uint64_t toff = 0;
#pragma unroll
    for (int i = 0; i < ROT_TB; i++) if ((tid >> i) & 1) toff |= a.uoff[i];
    for (uint64_t t = blockIdx.x; t < a.n_work; t += gridDim.x) {
        uint64_t base = 0;
        for (int i = 0; i < a.n_opos; i++) base |= ((t >> i) & 1ULL) << a.opos[i];
        for (int slot = 0; slot < a.ns; slot++) {
            const bool own = !(slot & a.so_rank);
            const uint64_t ub = (base ^ ((slot & a.so_out) ? a.x_out : 0)) | toff;
            stage_tile<R, ADJ_UB>(pre, pim, own ? a.phi : a.phi2, ub, a.uoff, slot, tid);
            stage_tile<R, ADJ_UB>(lre, lim, own ? a.lam : a.lam2, ub, a.uoff, slot, tid);
        }
        __syncthreads();
        for (int j = 0; j < a.K; j++) {
            const RotOp &op = a.ops[j];
            const uint32_t tag = a.op_tags[j];
            if (op.flags & ROT_DIAG) {
                adj_diag_overlap<R, T>(pre, pim, lre, lim, op, a.diag, a.diag_tags, base, nown, tid, s_acc_warp, lane == 0);
                if (!(tag & ADJ_SKIP)) {
                    rot_diag<R, T>(pre, pim, op, a.diag, base, a.ns, tid);
                    rot_diag<R, T>(lre, lim, op, a.diag, base, a.ns, tid);
                }
            } else {
                double v = adj_pair_overlap<R, T>(pre, pim, lre, lim, op, base, a.ns, a.so_rank, tid);
                v = warp_sum(tag >> 31 ? -v : v);
                if (lane == 0) s_acc_warp[tag & ADJ_POS] += v;
                if (!(tag & ADJ_SKIP)) {
                    rot_pairs<R, T>(pre, pim, op, base, a.ns, tid);
                    rot_pairs<R, T>(lre, lim, op, base, a.ns, tid);
                }
            }
            __syncthreads();
        }
        for (int slot = 0; slot < a.ns; slot++) {
            if (slot & a.so_rank) continue;   /* the partner rank writes its own tiles */
            const uint64_t ub = (base ^ ((slot & a.so_out) ? a.x_out : 0)) | toff;
            store_tile<R, ADJ_UB>(a.phi, pre, pim, ub, a.uoff, slot, tid);
            store_tile<R, ADJ_UB>(a.lam, lre, lim, ub, a.uoff, slot, tid);
        }
        __syncthreads();   /* the next tile group overwrites the planes */
    }
    __syncthreads();
    for (int j = tid; j < a.nrot; j += ROT_THREADS) {
        double acc = s_acc[j];
        for (int w = 1; w < ADJ_WARPS; w++) acc += s_acc[(size_t)w * a.nrot + j];
        a.partial[(size_t)blockIdx.x * a.nrot + j] = acc;
    }
}

/* per rotation of a sweep: the CTA partials in CTA order, into the gradient at the rotation's list index */
__global__ void k_adj_finish(const double *partial, int nblk, int nrot, const uint32_t *gidx, double *grad)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nrot) return;
    double acc = 0.0;
    for (int b = 0; b < nblk; b++) acc += partial[(size_t)b * nrot + j];
    grad[gidx[j]] = acc;
}

/* ================================================================================================ host */

namespace {

struct DevMem {   /* scoped device allocation */
    void *p = nullptr;
    ~DevMem() { if (p) cudaFree(p); }
};

/* the lambda table of one sweep: the diagonal terms grouped by pattern into diag (poff relative to d0), the others
 * into terms */
void encode_hsweep(const ExpSweep &sw, const std::vector<PhysTerm> &pt, const double *coef, int T, int su, int rank,
                   std::vector<HTerm> &terms, std::vector<RotDiag> &diag, uint32_t poff[17])
{
    const int NI = 1 << (T - ROT_TB);
    std::vector<std::vector<RotDiag>> by(NI);
    for (uint32_t i : sw.terms) {
        const PhysTerm &p = pt[i];
        const double c = parity64(((uint64_t)rank ^ p.xr) & p.zr) ? -coef[i] : coef[i];
        const uint32_t zin = tile_coord(p.zl, sw.pb, T);
        if (!p.xl && !p.xr) {
            RotDiag e; memset(&e, 0, sizeof e);
            e.theta = c;
            e.zout = (p.zl & ~sw.bmask) >> su;
            e.zt = zin & ((1u << ROT_TB) - 1);
            by[zin >> ROT_TB].push_back(e);
        } else {
            HTerm h; memset(&h, 0, sizeof h);
            h.c = c;
            h.zout = (p.zl & ~sw.bmask) >> su;
            h.xin = tile_coord(p.xl, sw.pb, T);
            h.zin = zin;
            h.w = (uint32_t)p.y;
            terms.push_back(h);
        }
    }
    memset(poff, 0, 17 * sizeof(uint32_t));
    for (int q = 0; q < NI; q++) {
        poff[q + 1] = poff[q] + (uint32_t)by[q].size();
        diag.insert(diag.end(), by[q].begin(), by[q].end());
    }
}

/* the sweeps of the gradient from a layout: lambda = H psi (exp_plan) and the adjoint sweeps (rot_plan on the reversed
 * list, one tile bit fewer); rt holds the reversed list's physical terms */
void grad_plans(int prec, const qsb_options_t *opt, int n, int nloc, const BitPerm &perm, const uint64_t *rx, const uint64_t *rz,
                size_t nrot, const uint64_t *hx, const uint64_t *hz, size_t nterms, std::vector<PhysTerm> &ht,
                std::vector<ExpSweep> &hs, std::vector<PhysTerm> &rt, std::vector<RotSweep> &as)
{
    int T, L;
    exp_geometry(prec, opt, &T, &L);
    to_physical(n, nloc, perm, hx, hz, nterms, ht);
    exp_plan(nloc, T, L, ht, hs);
    std::vector<uint64_t> vx(nrot), vz(nrot);
    for (size_t r = 0; r < nrot; r++) { vx[r] = rx[nrot - 1 - r]; vz[r] = rz[nrot - 1 - r]; }
    to_physical(n, nloc, perm, vx.data(), vz.data(), nrot, rt);
    rot_plan(nloc, T - 1, std::min(L, T - 1), rt, as);
}

int check_gradient_args(int n, const uint64_t *rx, const uint64_t *rz, size_t nrot, const uint64_t *hx, const uint64_t *hz,
                        size_t nterms, const char *fn)
{
    if (nterms == 0) { qsb_set_error("%s: the observable needs at least one term", fn); return QSB_ERR_ARG; }
    int rc = check_terms(n, rx, rz, nrot, fn);
    if (!rc) rc = check_terms(n, hx, hz, nterms, fn);
    return rc;
}

}  // namespace

/* ------------------------------------------------------------------------------------------- C ABI */

extern "C" int qsb_pauli_rotation_gradient_dry_run(int num_qubits, const qsb_options_t *opt_in, const uint64_t *rx, const uint64_t *rz,
                                                   size_t nrot, const uint64_t *hx, const uint64_t *hz, size_t nterms,
                                                   uint32_t *apply_sweeps, uint32_t *adjoint_sweeps, uint32_t *exchanges)
{
    qsb_options_t opt;
    int nloc;
    int rc = pauli_dry_run_shape(num_qubits, opt_in, &opt, &nloc);
    if (!rc) rc = check_gradient_args(num_qubits, rx, rz, nrot, hx, hz, nterms, "qsb_pauli_rotation_gradient_dry_run");
    if (rc) return rc;
    BitPerm id; for (int q = 0; q < 64; q++) id.pos[q] = (int8_t)q;
    std::vector<PhysTerm> ht, rt;
    std::vector<ExpSweep> hs;
    std::vector<RotSweep> as;
    grad_plans(opt.precision, &opt, num_qubits, nloc, id, rx, rz, nrot, hx, hz, nterms, ht, hs, rt, as);
    if (apply_sweeps) *apply_sweeps = (uint32_t)hs.size();
    if (adjoint_sweeps) *adjoint_sweeps = (uint32_t)as.size();
    if (exchanges) *exchanges = count_exchanges(hs) + count_exchanges(as);
    return QSB_OK;
}

extern "C" int qsb_pauli_rotation_gradient(qsb_t *s, const uint64_t *rx, const uint64_t *rz, const double *theta, size_t nrot,
                                           const uint64_t *hx, const uint64_t *hz, const double *coef, size_t nterms,
                                           double *energy, double *grad)
{
    static const char *fn = "qsb_pauli_rotation_gradient";
    if (!s) { qsb_set_error("%s: null handle", fn); return QSB_ERR_ARG; }
    int rc = check_gradient_args(s->n, rx, rz, nrot, hx, hz, nterms, fn);
    if (rc) return rc;
    if (!coef || !energy || (nrot && (!theta || !grad))) { qsb_set_error("%s: null angle, coefficient or output array", fn); return QSB_ERR_ARG; }
    for (size_t i = 0; i < nrot; i++)
        if (!isfinite(theta[i])) { qsb_set_error("%s: rotation %zu has a non-finite angle", fn, i); return QSB_ERR_ARG; }
    for (size_t j = 0; j < nterms; j++)
        if (!isfinite(coef[j])) { qsb_set_error("%s: term %zu has a non-finite coefficient", fn, j); return QSB_ERR_ARG; }
    if (s->g && !s->comm) { qsb_set_error("%s: sharded state needs qsb_comm_init first", fn); return QSB_ERR_COMM; }
    QSB_CUDA(cudaSetDevice(s->device));
    const bool f32 = s->prec == QSB_F32;
    const int su = f32 ? 1 : 0;
    int T, L;
    exp_geometry(s->prec, &s->opt, &T, &L);
    const int TA = T - 1;

    /* plans and tables from the layout, which the forward pass leaves as it is */
    std::vector<PhysTerm> ht, rt;
    std::vector<ExpSweep> hs;
    std::vector<RotSweep> as;
    if (nrot) grad_plans(s->prec, &s->opt, s->n, s->nloc, s->perm, rx, rz, nrot, hx, hz, nterms, ht, hs, rt, as);
    std::vector<HTerm> hterms;
    std::vector<RotDiag> hdiag;
    std::vector<size_t> h0;
    std::vector<std::array<uint32_t, 17>> hpoff(hs.size());
    for (size_t k = 0; k < hs.size(); k++) {
        h0.push_back(hterms.size());
        const size_t d0 = hdiag.size();
        encode_hsweep(hs[k], ht, coef, T, su, s->rank, hterms, hdiag, hpoff[k].data());
        for (auto &p : hpoff[k]) p += (uint32_t)d0;
    }
    h0.push_back(hterms.size());
    std::vector<double> negt(nrot);   /* the reversed list's angles, negated: the steps are R_k^dag */
    for (size_t r = 0; r < nrot; r++) negt[r] = -theta[nrot - 1 - r];
    std::vector<RotOp> ops;
    std::vector<RotDiag> diag;
    std::vector<uint32_t> op_tags, diag_tags, gidx;
    std::vector<size_t> op0, g0;
    for (auto &w : as) {
        op0.push_back(ops.size());
        g0.push_back(gidx.size());
        const size_t first_op = ops.size();
        encode_sweep(w, rt, negt, TA, su, s->rank, ops, diag, &op_tags, &diag_tags);
        for (size_t j = first_op; j < ops.size(); j++) {   /* theta = 0: the overlap but no apply */
            bool zero = true;
            if (ops[j].flags & ROT_DIAG) {
                for (uint32_t d = ops[j].d0; d < ops[j].d0 + ops[j].poff[1 << (TA - ROT_TB)]; d++) zero = zero && diag[d].theta == 0.0;
            } else {
                zero = negt[w.rots[op_tags[j] & ADJ_POS]] == 0.0;
            }
            if (zero) op_tags[j] |= ADJ_SKIP;
        }
        for (uint32_t r : w.rots) gidx.push_back((uint32_t)(nrot - 1 - r));
    }
    op0.push_back(ops.size());
    g0.push_back(gidx.size());

    /* device scratch before the forward pass: phi, lambda (and the partner's lambda), the tables, the partials */
    int nsm = 0;
    QSB_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, s->device));
    const int grid_cap = nsm * GRAD_GRID_CAP;
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t sb = s->state_bytes;
    const size_t vec_bytes = nrot ? sb * (s->g ? 3 : 2) : 0;
    const size_t hterm_bytes = al(hterms.size() * sizeof(HTerm)), hdiag_bytes = al(hdiag.size() * sizeof(RotDiag));
    const size_t ops_bytes = al(ops.size() * sizeof(RotOp)), diag_bytes = al(diag.size() * sizeof(RotDiag));
    const size_t tag_bytes = al((op_tags.size() + diag_tags.size() + gidx.size()) * sizeof(uint32_t));
    const size_t grad_bytes = al(nrot * sizeof(double)), all_bytes = s->g ? al((size_t)s->world * nrot * sizeof(double)) : 0;
    const size_t partial_bytes = nrot ? al((size_t)grid_cap * ROT_KMAX * sizeof(double)) : 0;
    const size_t total = vec_bytes + hterm_bytes + hdiag_bytes + ops_bytes + diag_bytes + tag_bytes + grad_bytes + all_bytes + partial_bytes + 256;
    DevMem mem;
    if (nrot) {
        const cudaError_t e = cudaMalloc(&mem.p, total);
        if (e != cudaSuccess) {
            cudaGetLastError();
            mem.p = nullptr;
            qsb_set_error("%s: cannot allocate %zu bytes of device scratch (%s)", fn, total, cudaGetErrorString(e));
            return e == cudaErrorMemoryAllocation ? QSB_ERR_NOMEM : QSB_ERR_CUDA;
        }
    }

    /* forward and energy through the existing calls */
    rc = qsb_apply_pauli_rotations(s, rx, rz, theta, nrot);
    if (rc) return rc;
    std::vector<double> v(nterms);
    rc = qsb_expectation_pauli(s, hx, hz, nterms, v.data());
    if (rc) return rc;
    double e = 0.0;
    for (size_t j = 0; j < nterms; j++) {
        volatile double prod = coef[j] * v[j];   /* rounded product, then the sum: never contracted to an FMA */
        e = e + prod;
    }
    *energy = e;
    if (!nrot) return QSB_OK;

    char *cur = (char *)mem.p;
    auto take = [&](size_t b) { char *p = cur; cur += b; return p; };
    uint4 *phi = (uint4 *)take(sb), *lam = (uint4 *)take(sb), *lam2 = s->g ? (uint4 *)take(sb) : nullptr;
    HTerm *d_hterms = (HTerm *)take(hterm_bytes);
    RotDiag *d_hdiag = (RotDiag *)take(hdiag_bytes);
    RotOp *d_ops = (RotOp *)take(ops_bytes);
    RotDiag *d_diag = (RotDiag *)take(diag_bytes);
    uint32_t *d_optags = (uint32_t *)take(tag_bytes), *d_diagtags = d_optags + op_tags.size(), *d_gidx = d_diagtags + diag_tags.size();
    double *d_grad = (double *)take(grad_bytes), *d_all = (double *)take(all_bytes), *d_partial = (double *)take(partial_bytes);
    void *flag = take(256);
    cudaStream_t st = s->stream;
    auto up = [&](void *dst, const void *src, size_t b) { return b ? cudaMemcpyAsync(dst, src, b, cudaMemcpyHostToDevice, st) : cudaSuccess; };
    QSB_CUDA(up(d_hterms, hterms.data(), hterms.size() * sizeof(HTerm)));
    QSB_CUDA(up(d_hdiag, hdiag.data(), hdiag.size() * sizeof(RotDiag)));
    QSB_CUDA(up(d_ops, ops.data(), ops.size() * sizeof(RotOp)));
    QSB_CUDA(up(d_diag, diag.data(), diag.size() * sizeof(RotDiag)));
    QSB_CUDA(up(d_optags, op_tags.data(), op_tags.size() * sizeof(uint32_t)));
    QSB_CUDA(up(d_diagtags, diag_tags.data(), diag_tags.size() * sizeof(uint32_t)));
    QSB_CUDA(up(d_gidx, gidx.data(), gidx.size() * sizeof(uint32_t)));
    QSB_CUDA(cudaMemcpyAsync(phi, s->state, sb, cudaMemcpyDeviceToDevice, st));
    uint32_t exchanged = 0;

    /* lambda = H psi */
    const int nouter = s->nloc - T;
    const size_t hsmem = (size_t)4 << T << (f32 ? 2 : 3);   /* 2 slots x re / im planes */
    if (f32) QSB_CUDA(cudaFuncSetAttribute(k_hpsi<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem));
    else QSB_CUDA(cudaFuncSetAttribute(k_hpsi<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem));
    int occ = 0;
    if (f32) QSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_hpsi<float>, ROT_THREADS, hsmem));
    else QSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_hpsi<double>, ROT_THREADS, hsmem));
    uint64_t fetched = 0;
    for (size_t k = 0; k < hs.size(); k++) {
        const ExpSweep &w = hs[k];
        if (w.xr && w.xr != fetched) {   /* the partner's psi, once per distinct xr */
            rc = tiled_comm_sendrecv(s, s->state, s->state2, sb, s->rank ^ (int)w.xr);
            if (rc) { cudaStreamSynchronize(st); return rc; }
            fetched = w.xr;
            exchanged++;
        }
        HArgs a; memset(&a, 0, sizeof a);
        a.src = (const uint4 *)(w.xr ? s->state2 : s->state);
        a.lam = lam;
        a.terms = d_hterms + h0[k];
        a.K = (int)(h0[k + 1] - h0[k]);
        a.diag = d_hdiag;
        memcpy(a.poff, hpoff[k].data(), sizeof a.poff);
        for (int i = 0; i < HPS_UB; i++) a.uoff[i] = (1ULL << w.pb[su + i]) >> su;
        a.x_out = w.x_out >> su;
        for (int b = 0; b < s->nloc; b++)
            if (!((w.bmask >> b) & 1)) a.opos[a.n_opos++] = (int8_t)(b - su);
        a.n_work = 1ULL << nouter;
        a.first = k == 0;
        const int grid = (int)std::min<uint64_t>(a.n_work, (uint64_t)nsm * std::max(occ, 1));
        if (f32) k_hpsi<float><<<grid, ROT_THREADS, hsmem, st>>>(a);
        else k_hpsi<double><<<grid, ROT_THREADS, hsmem, st>>>(a);
        QSB_CUDA(cudaGetLastError());
    }

    /* the adjoint sweeps */
    const size_t adj_smem_max = (size_t)4 * 2 * ADJ_UNITS * 16 + (size_t)ADJ_WARPS * ROT_KMAX * sizeof(double);   /* 192 KiB */
    if (f32) QSB_CUDA(cudaFuncSetAttribute(k_pauli_adj<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)adj_smem_max));
    else QSB_CUDA(cudaFuncSetAttribute(k_pauli_adj<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)adj_smem_max));
    const int anouter = s->nloc - TA;
    for (size_t k = 0; k < as.size(); k++) {
        const RotSweep &w = as[k];
        if (w.xr) {   /* the partner's phi and lambda as they are before this sweep */
            rc = tiled_comm_sendrecv(s, phi, s->state2, sb, s->rank ^ (int)w.xr);
            if (!rc) rc = tiled_comm_sendrecv(s, lam, lam2, sb, s->rank ^ (int)w.xr);
            if (rc) { cudaStreamSynchronize(st); return rc; }
            exchanged++;
        }
        AdjArgs a; memset(&a, 0, sizeof a);
        a.phi = phi; a.lam = lam;
        a.phi2 = (const uint4 *)(w.xr ? s->state2 : phi);
        a.lam2 = w.xr ? lam2 : lam;
        a.ops = d_ops + op0[k];
        a.op_tags = d_optags + op0[k];
        a.diag = d_diag;
        a.diag_tags = d_diagtags;
        a.K = (int)(op0[k + 1] - op0[k]);
        a.nrot = (int)w.rots.size();
        a.partial = d_partial;
        for (int i = 0; i < ADJ_UB; i++) a.uoff[i] = (1ULL << w.pb[su + i]) >> su;
        a.x_out = w.x_out >> su;
        slot_bits(w, &a.so_out, &a.so_rank, &a.ns);
        const int skip = w.x_out ? 63 - __builtin_clzll(w.x_out) : -1;   /* the group (t, t ^ x_out) from the t with this bit 0 */
        for (int b = 0; b < s->nloc; b++)
            if (!((w.bmask >> b) & 1) && b != skip) a.opos[a.n_opos++] = (int8_t)(b - su);
        a.n_work = 1ULL << (anouter - (w.x_out ? 1 : 0));
        const size_t smem = (size_t)a.ns * 2 * ADJ_UNITS * 16 + (size_t)ADJ_WARPS * a.nrot * sizeof(double);
        if (f32) QSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_pauli_adj<float>, ROT_THREADS, smem));
        else QSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_pauli_adj<double>, ROT_THREADS, smem));
        const int grid = (int)std::min<uint64_t>(a.n_work, (uint64_t)std::min(grid_cap, nsm * std::max(occ, 1)));
        if (f32) k_pauli_adj<float><<<grid, ROT_THREADS, smem, st>>>(a);
        else k_pauli_adj<double><<<grid, ROT_THREADS, smem, st>>>(a);
        k_adj_finish<<<(a.nrot + 127) / 128, 128, 0, st>>>(d_partial, grid, a.nrot, d_gidx + g0[k], d_grad);
        QSB_CUDA(cudaGetLastError());
    }

    if (!s->g) {
        QSB_CUDA(cudaMemcpyAsync(grad, d_grad, nrot * sizeof(double), cudaMemcpyDeviceToHost, st));
        QSB_CUDA(cudaStreamSynchronize(st));
        return QSB_OK;
    }
    rc = tiled_comm_allgather(s, d_grad, d_all, nrot * sizeof(double));
    if (rc) { cudaStreamSynchronize(st); return rc; }
    /* a peer's fused exchange scatters into this rank's state2 without waiting: once the partner shards are read, an
     * all-reduce on the stream orders this call before any later use of state2 by a peer */
    if (exchanged) {
        QSB_CUDA(cudaMemsetAsync(flag, 0, 8, st));
        rc = tiled_comm_allreduce_sum_u64(s, flag, 1);
        if (rc) { cudaStreamSynchronize(st); return rc; }
    }
    std::vector<double> all((size_t)s->world * nrot);
    QSB_CUDA(cudaMemcpyAsync(all.data(), d_all, all.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    QSB_CUDA(cudaStreamSynchronize(st));
    for (size_t k = 0; k < nrot; k++) {
        double acc = 0.0;
        for (int r = 0; r < s->world; r++) acc += all[(size_t)r * nrot + k];
        grad[k] = acc;
    }
    return QSB_OK;
}
