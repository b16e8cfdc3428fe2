/*
 * overlap.cu -- <a|b> = sum_j conj(a_j) b_j over the 2^n logical amplitudes of two handles, and the state copy (DESIGN.md
 * section 3.3).  fp64 over the states as stored, nothing is renormalised.
 *
 * LAYOUT MAP.  Logical qubit q sits at A-physical bit PA(q) and at B-physical bit PB(q).  The free qubits F are those
 * local in both handles; a step sweeps them in A's physical space, with every other local bit fixed: padding bits at 0,
 * A-local bits that are rank bits of B at the step's value, B-local bits that are rank bits of A at this rank's value.
 * The tile is T free qubits (12 f32 / 11 f64, the smaller when the precisions differ): those on A's low L_A bits, those on
 * B's low L_B bits, then the lowest other free A bits.  A tile coordinate c (bit i = the i-th tile qubit by A position)
 * reads A at base_A | deposit(c), in runs of at least 2^L_A amplitudes; the same tile of B is staged in shared memory in
 * B-coordinate order (bit k = the k-th tile qubit by B position, so runs of 2^L_B amplitudes) and read through the
 * tile-internal bit map.  Deposits and the bit map are two 64-entry tables each (low / high 6 coordinate bits).  With
 * equal layouts this is a streaming dot product of the two shards.
 *
 * SUMS.  Each element is converted to fp64 and adds ar*br + ai*bi to Re, ar*bi - ai*br to Im and the same expression to
 * <a|a> and <b|b>, every product rounded on its own (no FMA contraction), so a == b gives Im == +0 and Re == <a|a> ==
 * <b|b> bit for bit.  Threads sum their elements in order, a warp butterfly and the warps in order make the CTA partial,
 * k_overlap_finish sums the CTAs in order.  No floating-point atomics: repeated calls return identical bits.
 *
 * SHARDED.  R_A, R_B = the logical qubits on the rank bits, C = R_A & R_B, D_A = R_A \ R_B, D_B = R_B \ R_A (|D_A| =
 * |D_B| = d, each in ascending qubit order, D_A[i] paired with D_B[i]).  u(r) = rank r's values of D_A carried onto D_B.
 * Step t = 0 .. 2^d - 1 combines rank r's A shard with the B shard of src(r, t) = the B rank with r's values on C and
 * u(r) ^ t on D_B; the A slice read is the one whose D_B bits equal u(r) ^ t.  r -> src(r, t) is a bijection, so a step
 * is one grouped send / receive on B's communicator into B's state2; src == r needs no copy.  A call that used state2
 * ends with an all-reduce on B's communicator (a peer's fused exchange scatters into state2 without waiting).  The
 * per-rank sums are all-gathered on A's communicator and added on the host in rank order: every rank gets the same bits.
 * Neither handle's state buffer, layout, state2 role or peer mappings change.
 */
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "pauli.h"
#include "sim.h"
#include "tiled.h"

int tiled_comm_sendrecv_peers(qsb_sim *s, const void *dsend, int send_peer, void *drecv, int recv_peer, size_t bytes);
int tiled_comm_allgather(qsb_sim *s, const void *dsrc, void *ddst, size_t bytes);
int tiled_comm_allreduce_sum_u64(qsb_sim *s, void *dbuf, size_t count);

#define OV_THREADS 256
#define OV_TMAX 12                     /* tile bits: 12 f32 / 11 f64 */
#define OV_TILE_BYTES 32768            /* the staged B tile: 2^12 float2 / 2^11 double2 */

static_assert(OV_TMAX <= QSB_T_F32 && OV_TMAX - 1 <= QSB_T_F64, "the overlap tile must fit the smallest shard");

struct OvArgs {
    const void *A, *B;         /* A shard; B shard (own, or the partner's in B's state2) */
    double *partial;           /* [gridDim.x][4]: Re, Im, <a|a>, <b|b> */
    uint64_t baseA, baseB;     /* the fixed bits of the step, element offsets */
    uint64_t n_work;           /* tiles */
    int t, n_out;              /* tile bits, outer bits */
    int pairA, pairB;          /* f32: coordinate bit 0 is physical bit 0, so one 16-byte unit holds amplitudes 2i, 2i + 1 */
    int8_t tposA[OV_TMAX];     /* tile coordinate bit i -> A physical bit (ascending) */
    int8_t tposB[OV_TMAX];     /* B coordinate bit k -> B physical bit (ascending) */
    int8_t bco[OV_TMAX];       /* tile coordinate bit i -> its B coordinate bit */
    int8_t outA[64], outB[64]; /* tile index bit i -> A / B physical bit */
};

/* ================================================================================================ device */

__device__ __forceinline__ double2 ov_load(const float *s, uint64_t p)   /* f32 unit { re0 re1 im0 im1 } */
{
    const float *u = s + ((p >> 1) << 2) + (p & 1);
    return make_double2((double)__ldg(u), (double)__ldg(u + 2));   /* the unit's other amplitude is read from L1 */
}
__device__ __forceinline__ double2 ov_load(const double *s, uint64_t p) { return __ldcs(reinterpret_cast<const double2 *>(s) + p); }

/* both amplitudes of the f32 unit holding even element p */
__device__ __forceinline__ void ov_load2(const float *s, uint64_t p, double2 &x0, double2 &x1)
{
    const float4 v = __ldcs(reinterpret_cast<const float4 *>(s) + (p >> 1));
    x0 = make_double2((double)v.x, (double)v.z);
    x1 = make_double2((double)v.y, (double)v.w);
}

template <typename R> struct OvPair;
template <> struct OvPair<float> { typedef float2 T; };
template <> struct OvPair<double> { typedef double2 T; };

/* ar*br + ai*bi, both products rounded, added in this order */
__device__ __forceinline__ double ov_dot(double ar, double ai, double br, double bi)
{
    return __dadd_rn(__dmul_rn(ar, br), __dmul_rn(ai, bi));
}

/* one element pair into the four sums (the same expression for Re and both norms) */
__device__ __forceinline__ void ov_add(double2 x, double yr, double yi, double &re, double &im, double &na, double &nb)
{
    re = __dadd_rn(re, ov_dot(x.x, x.y, yr, yi));
    im = __dadd_rn(im, __dsub_rn(__dmul_rn(x.x, yi), __dmul_rn(x.y, yr)));
    na = __dadd_rn(na, ov_dot(x.x, x.y, x.x, x.y));
    nb = __dadd_rn(nb, ov_dot(yr, yi, yr, yi));
}

template <typename RA, typename RB>
__global__ void __launch_bounds__(OV_THREADS) k_overlap(const __grid_constant__ OvArgs a)
{
    typedef typename OvPair<RB>::T PB;
    __shared__ PB s_b[OV_TILE_BYTES / sizeof(PB)];
    __shared__ uint64_t s_da[2][64], s_db[2][64];   /* deposits of the low / high 6 coordinate bits into A / B */
    __shared__ uint32_t s_map[2][64];               /* tile coordinate -> B coordinate, low / high 6 bits */
    __shared__ double s_w[OV_THREADS / 32][4];
    const uint32_t tid = threadIdx.x;
    const RA *A = reinterpret_cast<const RA *>(a.A);
    const RB *B = reinterpret_cast<const RB *>(a.B);
    if (tid < 128) {
        const int h = tid >> 6, v = tid & 63;
        uint64_t da = 0, db = 0;
        uint32_t m = 0;
        for (int j = 0; j < 6; j++) {
            const int i = 6 * h + j;
            if (i >= a.t || !((v >> j) & 1)) continue;
            da |= 1ULL << a.tposA[i];
            db |= 1ULL << a.tposB[i];
            m |= 1u << a.bco[i];
        }
        s_da[h][v] = da; s_db[h][v] = db; s_map[h][v] = m;
    }
    __syncthreads();
    const uint32_t size = 1u << a.t;
    double re = 0.0, im = 0.0, na = 0.0, nb = 0.0;
    for (uint64_t tile = blockIdx.x; tile < a.n_work; tile += gridDim.x) {
        uint64_t bA = a.baseA, bB = a.baseB;
        for (int i = 0; i < a.n_out; i++)
            if ((tile >> i) & 1) { bA |= 1ULL << a.outA[i]; bB |= 1ULL << a.outB[i]; }
        if (sizeof(RB) == 4 && a.pairB) {
#pragma unroll 4
            for (uint32_t k = 2 * tid; k < size; k += 2 * OV_THREADS) {
                double2 v0, v1;
                ov_load2(reinterpret_cast<const float *>(B), bB | s_db[0][k & 63] | s_db[1][k >> 6], v0, v1);
                s_b[k].x = (RB)v0.x; s_b[k].y = (RB)v0.y;   /* exact: v holds B's own precision */
                s_b[k + 1].x = (RB)v1.x; s_b[k + 1].y = (RB)v1.y;
            }
        } else {
#pragma unroll 4
            for (uint32_t k = tid; k < size; k += OV_THREADS) {
                const double2 v = ov_load(B, bB | s_db[0][k & 63] | s_db[1][k >> 6]);
                s_b[k].x = (RB)v.x; s_b[k].y = (RB)v.y;
            }
        }
        __syncthreads();
        if (sizeof(RA) == 4 && a.pairA) {
#pragma unroll 4
            for (uint32_t c = 2 * tid; c < size; c += 2 * OV_THREADS) {
                double2 x0, x1;
                ov_load2(reinterpret_cast<const float *>(A), bA | s_da[0][c & 63] | s_da[1][c >> 6], x0, x1);
                const PB y0 = s_b[s_map[0][c & 63] | s_map[1][c >> 6]], y1 = s_b[s_map[0][(c + 1) & 63] | s_map[1][c >> 6]];
                ov_add(x0, (double)y0.x, (double)y0.y, re, im, na, nb);
                ov_add(x1, (double)y1.x, (double)y1.y, re, im, na, nb);
            }
        } else {
#pragma unroll 4
            for (uint32_t c = tid; c < size; c += OV_THREADS) {
                const double2 x = ov_load(A, bA | s_da[0][c & 63] | s_da[1][c >> 6]);
                const PB yb = s_b[s_map[0][c & 63] | s_map[1][c >> 6]];
                ov_add(x, (double)yb.x, (double)yb.y, re, im, na, nb);
            }
        }
        __syncthreads();   /* the next tile overwrites s_b */
    }
    double v[4] = {re, im, na, nb};
#pragma unroll
    for (int k = 0; k < 4; k++)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] = __dadd_rn(v[k], __shfl_xor_sync(0xffffffffu, v[k], o));
    if ((tid & 31) == 0) for (int k = 0; k < 4; k++) s_w[tid >> 5][k] = v[k];
    __syncthreads();
    if (tid < 4) {
        double acc = s_w[0][tid];
        for (int w = 1; w < OV_THREADS / 32; w++) acc = __dadd_rn(acc, s_w[w][tid]);
        a.partial[(size_t)blockIdx.x * 4 + tid] = acc;
    }
}

/* the CTA partials in CTA order, added to the sums of the earlier steps (step 0 starts them) */
__global__ void k_overlap_finish(const double *partial, int nblk, int first, double *res)
{
    const int k = threadIdx.x;
    if (k >= 4) return;
    double acc = partial[k];
    for (int b = 1; b < nblk; b++) acc = __dadd_rn(acc, partial[(size_t)b * 4 + k]);
    res[k] = first ? acc : __dadd_rn(res[k], acc);
}

/* ================================================================================================ host */

namespace {

struct OvSide { int n, g, nloc, prec, T, L; BitPerm perm; };

int rank_bit(const OvSide &h, int q) { return h.perm.pos[q] - h.nloc; }   /* < 0: local */

/* The rank-qubit sets and the tile of a pair of layouts (the same on every rank). */
struct OvPlan {
    std::vector<int> C, DA, DB;        /* logical qubits: rank in both; rank in A only; rank in B only (ascending) */
    std::vector<int> tile, outer;      /* free qubits (local in both): tile, by A position; the others, by A position */
    int T = 0;
};

int ov_plan(const OvSide &A, const OvSide &B, OvPlan &p, const char *fn)
{
    std::vector<int> free;
    for (int q = 0; q < A.n; q++) {
        const bool ra = rank_bit(A, q) >= 0, rb = rank_bit(B, q) >= 0;
        if (ra && rb) p.C.push_back(q);
        else if (ra) p.DA.push_back(q);
        else if (rb) p.DB.push_back(q);
        else free.push_back(q);
    }
    std::sort(free.begin(), free.end(), [&](int x, int y) { return A.perm.pos[x] < A.perm.pos[y]; });
    p.T = std::min(A.T, B.T);
    const int t = std::min<int>(p.T, (int)free.size());
    std::vector<char> in(A.n, 0);
    int cnt = 0;
    for (int q : free) if (A.perm.pos[q] < A.L) { in[q] = 1; cnt++; }
    for (int q : free) if (!in[q] && B.perm.pos[q] < B.L) { in[q] = 1; cnt++; }
    if (cnt > t) { qsb_set_error("%s: internal: the low bits of both layouts need %d tile bits, %d available", fn, cnt, t); return QSB_ERR_ARG; }
    for (int q : free) if (!in[q] && cnt < t) { in[q] = 1; cnt++; }
    for (int q : free) (in[q] ? p.tile : p.outer).push_back(q);
    return QSB_OK;
}

/* step t of rank r: the B rank whose shard is combined, and the rank that receives r's B shard */
void ov_peers(const OvSide &A, const OvSide &B, const OvPlan &p, int r, uint32_t t, int *src, int *dst)
{
    int s = 0, d = 0;
    for (int q : p.C) {
        s |= ((r >> rank_bit(A, q)) & 1) << rank_bit(B, q);
        d |= ((r >> rank_bit(B, q)) & 1) << rank_bit(A, q);
    }
    for (size_t i = 0; i < p.DA.size(); i++) {
        const int u = (r >> rank_bit(A, p.DA[i])) & 1, ti = (t >> i) & 1;
        s |= (u ^ ti) << rank_bit(B, p.DB[i]);
        d |= (((r >> rank_bit(B, p.DB[i])) & 1) ^ ti) << rank_bit(A, p.DA[i]);
    }
    *src = s; *dst = d;
}

/* the launch arguments of step t on rank r (A / B pointers and partials left to the caller) */
void ov_args(const OvSide &A, const OvSide &B, const OvPlan &p, int r, uint32_t t, OvArgs &a)
{
    memset(&a, 0, sizeof a);
    for (size_t i = 0; i < p.DA.size(); i++) {
        const uint64_t u = (r >> rank_bit(A, p.DA[i])) & 1;
        a.baseA |= (u ^ ((t >> i) & 1)) << A.perm.pos[p.DB[i]];   /* the A slice whose D_B bits equal u(r) ^ t */
        a.baseB |= u << B.perm.pos[p.DA[i]];                     /* r's values of D_A, local in B */
    }
    a.t = (int)p.tile.size();
    std::vector<int> byb(p.tile);
    std::sort(byb.begin(), byb.end(), [&](int x, int y) { return B.perm.pos[x] < B.perm.pos[y]; });
    for (int i = 0; i < a.t; i++) {
        a.tposA[i] = A.perm.pos[p.tile[i]];
        a.tposB[i] = B.perm.pos[byb[i]];
        a.bco[i] = (int8_t)(std::find(byb.begin(), byb.end(), p.tile[i]) - byb.begin());
    }
    a.n_out = (int)p.outer.size();
    for (int i = 0; i < a.n_out; i++) { a.outA[i] = A.perm.pos[p.outer[i]]; a.outB[i] = B.perm.pos[p.outer[i]]; }
    a.n_work = 1ULL << a.n_out;
    a.pairA = A.prec == QSB_F32 && a.t > 0 && a.tposA[0] == 0;
    a.pairB = B.prec == QSB_F32 && a.t > 0 && a.tposB[0] == 0;
}

int ov_side(int n, const qsb_options_t *opt, int nloc, const BitPerm &perm, OvSide &h, const char *fn)
{
    h.n = n; h.prec = opt->precision; h.nloc = nloc; h.perm = perm;
    h.g = 0; while ((1 << h.g) < opt->world_size) h.g++;
    const int rc = check_low_bits(h.prec, opt, fn);
    if (rc) return rc;
    exp_geometry(h.prec, opt, &h.T, &h.L);
    return QSB_OK;
}

/* steps and partner-shard copies on rank r; any = some rank copies a shard in some step */
void ov_count(const OvSide &A, const OvSide &B, const OvPlan &p, int r, int world, uint32_t *steps, uint32_t *copies, bool *any)
{
    const uint32_t ns = 1u << p.DA.size();
    uint32_t c = 0;
    bool x = false;
    for (uint32_t t = 0; t < ns; t++)
        for (int q = 0; q < world; q++) {
            int src, dst;
            ov_peers(A, B, p, q, t, &src, &dst);
            if (src != q) { x = true; if (q == r) c++; }
        }
    *steps = ns;
    *copies = c;
    if (any) *any = x;
}

struct DevMem {   /* scoped device allocation */
    void *p = nullptr;
    ~DevMem() { if (p) cudaFree(p); }
};

struct Events {   /* scoped events that order the two handles' streams */
    cudaEvent_t a = nullptr, b = nullptr;
    ~Events() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
};

/* `waiter` waits for the work enqueued so far on `s` */
int ov_order(cudaStream_t waiter, cudaStream_t s, cudaEvent_t e)
{
    if (waiter == s) return QSB_OK;
    QSB_CUDA(cudaEventRecord(e, s));
    QSB_CUDA(cudaStreamWaitEvent(waiter, e, 0));
    return QSB_OK;
}

template <typename RA, typename RB>
int ov_launch(cudaStream_t st, const OvArgs &a, int grid, double *res, bool first)
{
    k_overlap<RA, RB><<<grid, OV_THREADS, 0, st>>>(a);
    k_overlap_finish<<<1, 32, 0, st>>>(a.partial, grid, first ? 1 : 0, res);
    QSB_CUDA(cudaGetLastError());
    return QSB_OK;
}

template <typename RA, typename RB>
int ov_grid(int device, uint64_t n_work, int *grid)
{
    int nsm = 0, occ = 0;
    QSB_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device));
    QSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_overlap<RA, RB>, OV_THREADS, 0));
    *grid = (int)std::min<uint64_t>(n_work, (uint64_t)nsm * std::max(occ, 1));
    return QSB_OK;
}

int ov_grid_for(int pa, int pb, int device, uint64_t n_work, int *grid)
{
    if (pa == QSB_F32) return pb == QSB_F32 ? ov_grid<float, float>(device, n_work, grid) : ov_grid<float, double>(device, n_work, grid);
    return pb == QSB_F32 ? ov_grid<double, float>(device, n_work, grid) : ov_grid<double, double>(device, n_work, grid);
}

int ov_launch_for(int pa, int pb, cudaStream_t st, const OvArgs &a, int grid, double *res, bool first)
{
    if (pa == QSB_F32) return pb == QSB_F32 ? ov_launch<float, float>(st, a, grid, res, first) : ov_launch<float, double>(st, a, grid, res, first);
    return pb == QSB_F32 ? ov_launch<double, float>(st, a, grid, res, first) : ov_launch<double, double>(st, a, grid, res, first);
}

}  // namespace

/* ------------------------------------------------------------------------------------------- C ABI */

extern "C" int qsb_inner_product_dry_run(int num_qubits, const qsb_options_t *opt_a, const int8_t *perm_a,
                                         const qsb_options_t *opt_b, const int8_t *perm_b, uint32_t *steps, uint32_t *exchanges)
{
    static const char *fn = "qsb_inner_product_dry_run";
    if (!perm_a || !perm_b) { qsb_set_error("%s: null layout", fn); return QSB_ERR_ARG; }
    qsb_options_t oa, ob;
    int nla, nlb;
    int rc = pauli_dry_run_shape(num_qubits, opt_a, &oa, &nla);
    if (rc) return rc;
    rc = pauli_dry_run_shape(num_qubits, opt_b, &ob, &nlb);
    if (rc) return rc;
    if (oa.world_size != ob.world_size || oa.rank != ob.rank) {
        qsb_set_error("%s: the handles differ in world (%d, %d) or rank (%d, %d)", fn, oa.world_size, ob.world_size, oa.rank, ob.rank);
        return QSB_ERR_ARG;
    }
    if (oa.rank < 0 || oa.rank >= oa.world_size) { qsb_set_error("%s: rank %d outside world of %d", fn, oa.rank, oa.world_size); return QSB_ERR_ARG; }
    OvSide A, B;
    const int8_t *pp[2] = {perm_a, perm_b};
    const int nl[2] = {nla, nlb};
    BitPerm perm[2];
    for (int h = 0; h < 2; h++) {
        memset(perm[h].pos, -1, sizeof perm[h].pos);
        const int nphys = nl[h] + __builtin_ctz((unsigned)oa.world_size);
        uint64_t seen = 0;
        for (int q = 0; q < num_qubits; q++) {
            const int b = pp[h][q];
            if (b < 0 || b >= nphys || ((seen >> b) & 1)) {
                qsb_set_error("%s: layout %c is not a permutation of the %d physical bits (qubit %d -> %d)", fn, "ab"[h], nphys, q, b);
                return QSB_ERR_ARG;
            }
            seen |= 1ULL << b;
            perm[h].pos[q] = (int8_t)b;
        }
    }
    if ((rc = ov_side(num_qubits, &oa, nla, perm[0], A, fn)) || (rc = ov_side(num_qubits, &ob, nlb, perm[1], B, fn))) return rc;
    OvPlan p;
    if ((rc = ov_plan(A, B, p, fn))) return rc;
    uint32_t ns, nc;
    ov_count(A, B, p, oa.rank, oa.world_size, &ns, &nc, nullptr);
    if (steps) *steps = ns;
    if (exchanges) *exchanges = nc;
    return QSB_OK;
}

extern "C" int qsb_inner_product(qsb_t *a, qsb_t *b, double out[2], double norms[2])
{
    static const char *fn = "qsb_inner_product";
    if (!a || !b || !out) { qsb_set_error("%s: null handle or output", fn); return QSB_ERR_ARG; }
    if (a->n != b->n || a->world != b->world || a->rank != b->rank || a->device != b->device) {
        qsb_set_error("%s: the handles differ: %d / %d qubits, world %d / %d, rank %d / %d, device %d / %d", fn, a->n, b->n,
                      a->world, b->world, a->rank, b->rank, a->device, b->device);
        return QSB_ERR_ARG;
    }
    OvSide A, B;
    int rc;
    if ((rc = ov_side(a->n, &a->opt, a->nloc, a->perm, A, fn)) || (rc = ov_side(b->n, &b->opt, b->nloc, b->perm, B, fn))) return rc;
    if (a->g && (!a->comm || !b->comm)) { qsb_set_error("%s: sharded states need qsb_comm_init first on both handles", fn); return QSB_ERR_COMM; }
    OvPlan p;
    if ((rc = ov_plan(A, B, p, fn))) return rc;
    uint32_t ns, ncopies;
    bool any_copy = false;
    ov_count(A, B, p, a->rank, a->world, &ns, &ncopies, &any_copy);
    QSB_CUDA(cudaSetDevice(a->device));

    OvArgs a0;
    ov_args(A, B, p, a->rank, 0, a0);
    int grid = 0;
    if ((rc = ov_grid_for(a->prec, b->prec, a->device, a0.n_work, &grid))) return rc;
    /* one allocation: CTA partials, this rank's sums, the all-gather of every rank's sums, the all-reduce flag */
    const size_t part_bytes = (size_t)grid * 4 * sizeof(double), res_bytes = 4 * sizeof(double);
    const size_t all_bytes = (size_t)a->world * res_bytes;
    DevMem mem;
    QSB_CUDA(cudaMalloc(&mem.p, part_bytes + res_bytes + all_bytes + 16));
    double *d_part = (double *)mem.p, *d_res = d_part + 4 * (size_t)grid, *d_all = d_res + 4;
    void *d_flag = d_all + 4 * (size_t)a->world;
    Events ev;
    QSB_CUDA(cudaEventCreateWithFlags(&ev.a, cudaEventDisableTiming));
    QSB_CUDA(cudaEventCreateWithFlags(&ev.b, cudaEventDisableTiming));

    auto fail = [&](int code) { cudaStreamSynchronize(a->stream); cudaStreamSynchronize(b->stream); return code; };
    /* A's launches read B's shard as B's earlier work leaves it */
    if ((rc = ov_order(a->stream, b->stream, ev.b))) return fail(rc);
    for (uint32_t t = 0; t < ns; t++) {
        int src, dst;
        ov_peers(A, B, p, a->rank, t, &src, &dst);
        OvArgs args;
        ov_args(A, B, p, a->rank, t, args);
        args.A = a->state;
        args.B = src == a->rank ? b->state : b->state2;
        args.partial = d_part;
        if (src != a->rank) {   /* state2 is overwritten once the previous step has read it */
            if ((rc = ov_order(b->stream, a->stream, ev.a))) return fail(rc);
            if ((rc = tiled_comm_sendrecv_peers(b, b->state, dst, b->state2, src, b->state_bytes))) return fail(rc);
            if ((rc = ov_order(a->stream, b->stream, ev.b))) return fail(rc);
        }
        if ((rc = ov_launch_for(a->prec, b->prec, a->stream, args, grid, d_res, t == 0))) return fail(rc);
    }
    if (any_copy) {   /* every rank: no peer's later exchange into B's state2 before the partner shards are read */
        if ((rc = ov_order(b->stream, a->stream, ev.a))) return fail(rc);
        QSB_CUDA(cudaMemsetAsync(d_flag, 0, 8, b->stream));
        if ((rc = tiled_comm_allreduce_sum_u64(b, d_flag, 1))) return fail(rc);
    }
    std::vector<double> all(4 * (size_t)a->world);
    if (a->g) {
        if ((rc = tiled_comm_allgather(a, d_res, d_all, res_bytes))) return fail(rc);
    } else {
        d_all = d_res;
    }
    QSB_CUDA(cudaMemcpyAsync(all.data(), d_all, all_bytes, cudaMemcpyDeviceToHost, a->stream));
    QSB_CUDA(cudaStreamSynchronize(a->stream));
    QSB_CUDA(cudaStreamSynchronize(b->stream));
    double sum[4];
    for (int k = 0; k < 4; k++) {
        sum[k] = all[k];
        for (int r = 1; r < a->world; r++) sum[k] += all[4 * r + k];
    }
    out[0] = sum[0]; out[1] = sum[1];
    if (norms) { norms[0] = sum[2]; norms[1] = sum[3]; }
    return QSB_OK;
}

extern "C" int qsb_copy_state(qsb_t *dst, const qsb_t *src)
{
    static const char *fn = "qsb_copy_state";
    if (!dst || !src) { qsb_set_error("%s: null handle", fn); return QSB_ERR_ARG; }
    if (dst == src) return QSB_OK;
    if (dst->n != src->n || dst->world != src->world || dst->rank != src->rank || dst->device != src->device || dst->prec != src->prec) {
        qsb_set_error("%s: the handles differ: %d / %d qubits, world %d / %d, rank %d / %d, device %d / %d, precision f%d / f%d",
                      fn, dst->n, src->n, dst->world, src->world, dst->rank, src->rank, dst->device, src->device, dst->prec, src->prec);
        return QSB_ERR_ARG;
    }
    QSB_CUDA(cudaSetDevice(dst->device));
    Events ev;
    QSB_CUDA(cudaEventCreateWithFlags(&ev.a, cudaEventDisableTiming));
    int rc = ov_order(dst->stream, src->stream, ev.a);
    if (rc) return rc;
    QSB_CUDA(cudaMemcpyAsync(dst->state, src->state, dst->state_bytes, cudaMemcpyDeviceToDevice, dst->stream));
    QSB_CUDA(cudaStreamSynchronize(dst->stream));
    dst->perm = src->perm;
    return QSB_OK;
}
