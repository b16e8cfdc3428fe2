/*
 * rdm.cu -- reduced density matrices of chosen qubits on the device (DESIGN.md section 3.3).
 *
 * rho[a][b] = sum over j, j' that agree on every unmeasured qubit, with bits(j) = a and bits(j') = b, of a_j conj(a_j'),
 * bit i of a and b = the value of qubits[i].  fp64 over the state as stored, nothing is renormalised.
 *
 * MATRIX VIEW.  The local shard is a matrix A: row = the measured local physical bits (ascending, the pext order of
 * measure.cu), column = the unmeasured local bits (ascending; padding bits of small registers included, their amplitudes
 * are zero).  The local contribution is A A^H, a Hermitian rank update of 2^k_loc rows by 2^(nloc - k_loc) columns.
 *
 * LOADS.  A segment is the low S physical bits (f32: pack bit + 5 unit bits, f64: 5 unit bits): 32 units, 512 contiguous
 * bytes, one warp load.  Measured bits inside the segment are the minor bits of a row, unmeasured ones the minor bits of
 * a column, so a row block of BM >= 2^(measured segment bits) rows by a chunk of KC columns is a set of whole segments:
 * every loaded byte is used, whatever qubits are measured.  A chunk (BM x KC = 4096 amplitudes f32 / 2048 f64) of each
 * operand goes through registers (the next chunk is loaded while the current one is computed) into shared memory,
 * converted to fp64 on the way.
 *
 * COMPUTE.  256 threads, micro-tiles of TM x TM complex fp64 accumulators (TM = min(BM, 4)); when the BM x BM block has
 * fewer micro-tiles than threads, KS = 256 / (BM / TM)^2 threads share one and split the chunk's columns, and their sums
 * are folded by a fixed tree (warp xor butterfly, then warps in order).  One CTA handles one block pair (I <= J of the
 * upper triangle, or every pair in the two-source form) and one of nsplit column ranges; per-CTA partials are summed in
 * split order by k_rdm_finish (nsplit = 1 writes the block straight into the result).  No floating-point atomics: repeated
 * calls return identical bits.  Blocks below the diagonal are not computed; the host mirrors the upper triangle, so the
 * result is Hermitian bit for bit and its diagonal imaginary parts are +0.0.
 *
 * SHARDED.  Measured qubits on rank bits (m of them, pattern D(d) for d = 1..2^m - 1) need cross-rank blocks: the shard
 * of rank r ^ D(d) comes into state2 (tiled_comm_sendrecv, as expect.cu does) and the two-source form computes the full
 * block A_r A_{r^D}^H.  Every rank's 2^m blocks are all-gathered and every rank places and sums them on the host in rank
 * order, so every rank ends with the same bits.  state / state2 are not swapped and the peer mappings are not touched.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "sim.h"
#include "tiled.h"

int tiled_comm_allgather(qsb_sim *s, const void *dsrc, void *ddst, size_t bytes);
int tiled_comm_sendrecv(qsb_sim *s, const void *dsend, void *drecv, size_t bytes, int peer);

#define RDM_THREADS 256
#define RDM_KMAX 12                  /* rho of 12 qubits: 4096 x 4096 complex, 256 MiB */
#define RDM_BMAX 64                  /* rows of a block; >= 2^6, the most measured bits a segment can hold */
#define RDM_UPT 8                    /* 16-byte units per thread and operand chunk */
#define RDM_CH(f32) ((f32) ? 4096 : 2048)   /* amplitudes per operand chunk: RDM_UPT * 256 units */
#define RDM_PARTIAL_BYTES ((size_t)64 << 20)   /* bound of the per-CTA partials of one launch */
/* a segment (the low 6 / 5 physical bits) exists in every shard: nloc >= tiled_min_local_bits() */
static_assert(6 <= QSB_T_F32 && 5 <= QSB_T_F64, "the rdm segment must fit the smallest shard");

struct RdmArgs {
    const uint4 *A, *B;       /* row operand (own shard), column operand (own shard, or the partner shard in state2) */
    double2 *out;             /* nsplit == 1: the R x R result; else partials [gridDim.x][BM][BM] */
    int nb, nsplit, full;     /* blocks per dimension, column splits, 1 = every block pair (two-source form) */
    int cps, KC;              /* chunks per split, columns per chunk */
    int m_low;                /* measured bits among the segment bits */
    uint32_t mlow;            /* those bits (physical bits 0..S-1) */
    int n_m, n_u;             /* measured / unmeasured local bits */
    int8_t mpos[RDM_KMAX];    /* physical bit of row bit i */
    int8_t upos[64];          /* physical bit of column bit i */
};

/* ================================================================================================ device */

__device__ __forceinline__ uint64_t rdm_deposit(uint64_t v, const int8_t *pos, int n)
{
    uint64_t r = 0;
    for (int i = 0; v && i < n; i++, v >>= 1) r |= (v & 1ULL) << pos[i];
    return r;
}

template <int BM, bool F32>
__global__ void __launch_bounds__(RDM_THREADS) k_rdm(const __grid_constant__ RdmArgs a)
{
    constexpr int TM = BM < 4 ? BM : 4;             /* micro-tile TM x TM */
    constexpr int GW = BM / TM, G = GW * GW;        /* micro-tiles per block row / per block */
    constexpr int KS = RDM_THREADS / G;             /* threads per micro-tile (column split inside the CTA) */
    constexpr int SU = F32 ? 1 : 0, S = 5 + SU, APU = 1 + SU;
    constexpr int LD = RDM_CH(F32) / BM + 1;        /* shared row stride (double2), padded against bank conflicts */
    extern __shared__ double2 sm[];                 /* A [BM][LD], then B [BM][LD] */
    __shared__ uint64_t s_rowA[RDM_BMAX], s_rowB[RDM_BMAX], s_col[64];
    const int tid = threadIdx.x, lane = tid & 31;

    const int p = blockIdx.x / a.nsplit, sp = blockIdx.x % a.nsplit;
    int I, J;
    if (a.full) { I = p / a.nb; J = p % a.nb; }
    else { int q = p; I = 0; while (q >= a.nb - I) { q -= a.nb - I; I++; } J = I + q; }
    const bool same = !a.full && I == J;
    double2 *As = sm, *Bs = same ? sm : sm + BM * LD;
    const uint4 *Bsrc = a.full ? a.B : a.A;

    /* unit-address offsets of the row segments of blocks I and J and of the column segments of a chunk */
    const int m_low = a.m_low, lg_ncs = __ffs(a.KC) - 1 - (S - m_low);
    const int nrs = BM >> m_low, ncs = 1 << lg_ncs;
    for (int i = tid; i < nrs; i += RDM_THREADS) {
        s_rowA[i] = rdm_deposit((uint64_t)(I * BM + (i << m_low)), a.mpos, a.n_m) >> SU;
        s_rowB[i] = rdm_deposit((uint64_t)(J * BM + (i << m_low)), a.mpos, a.n_m) >> SU;
    }
    for (int i = tid; i < ncs; i += RDM_THREADS) s_col[i] = rdm_deposit((uint64_t)i << (S - m_low), a.upos, a.n_u) >> SU;
    /* row / column minor bits of this thread's amplitudes (its unit sits at segment offset `lane`) */
    int rl[APU], cl[APU];
#pragma unroll
    for (int l = 0; l < APU; l++) {
        const uint32_t ph = ((uint32_t)lane << SU) | l;
        int r = 0, c = 0, nr = 0, nc = 0;
        for (int b = 0; b < S; b++) {
            if ((a.mlow >> b) & 1) r |= ((ph >> b) & 1) << nr++;
            else c |= ((ph >> b) & 1) << nc++;
        }
        rl[l] = r; cl[l] = c;
    }
    __syncthreads();

    const int nunits = BM * a.KC / APU;
    uint4 ra[RDM_UPT], rb[RDM_UPT];
    auto load = [&](int chunk) {
        const uint64_t cbase = rdm_deposit((uint64_t)chunk * a.KC, a.upos, a.n_u) >> SU;
#pragma unroll
        for (int i = 0; i < RDM_UPT; i++) {
            const int u = tid + i * RDM_THREADS;
            if (u < nunits) {
                const int seg = u >> 5, rh = seg >> lg_ncs, ch = seg & (ncs - 1);
                const uint64_t off = cbase | s_col[ch] | (uint64_t)lane;
                ra[i] = __ldcs(a.A + (s_rowA[rh] | off));
                if (!same) rb[i] = __ldcs(Bsrc + (s_rowB[rh] | off));
            }
        }
    };
    auto stage = [&](const uint4 (&r)[RDM_UPT], double2 *dst) {
#pragma unroll
        for (int i = 0; i < RDM_UPT; i++) {
            const int u = tid + i * RDM_THREADS;
            if (u < nunits) {
                const int seg = u >> 5, rh = seg >> lg_ncs, ch = seg & (ncs - 1);
                const int row0 = rh << m_low, col0 = ch << (S - m_low);
                if (F32) {
                    const float4 x = *reinterpret_cast<const float4 *>(&r[i]);   /* re0 re1 im0 im1 */
                    dst[(row0 | rl[0]) * LD + (col0 | cl[0])] = make_double2(x.x, x.z);
                    dst[(row0 | rl[APU - 1]) * LD + (col0 | cl[APU - 1])] = make_double2(x.y, x.w);
                } else {
                    dst[(row0 | rl[0]) * LD + (col0 | cl[0])] = *reinterpret_cast<const double2 *>(&r[i]);
                }
            }
        }
    };

    const int ks = tid % KS, g = tid / KS, gx = g % GW, gy = g / GW;
    double accr[TM][TM], acci[TM][TM];
#pragma unroll
    for (int i = 0; i < TM; i++)
#pragma unroll
        for (int j = 0; j < TM; j++) { accr[i][j] = 0.0; acci[i][j] = 0.0; }

    const int c0 = sp * a.cps;
    load(c0);
    for (int c = 0; c < a.cps; c++) {
        __syncthreads();   /* the previous chunk has been read */
        stage(ra, As);
        if (!same) stage(rb, Bs);
        __syncthreads();
        if (c + 1 < a.cps) load(c0 + c + 1);
        for (int k = ks; k < a.KC; k += KS) {
            double2 av[TM], bv[TM];
#pragma unroll
            for (int i = 0; i < TM; i++) av[i] = As[(gy + GW * i) * LD + k];
            if (G == 1 && same) {
#pragma unroll
                for (int j = 0; j < TM; j++) bv[j] = av[j];
            } else {
#pragma unroll
                for (int j = 0; j < TM; j++) bv[j] = Bs[(gx + GW * j) * LD + k];
            }
#pragma unroll
            for (int i = 0; i < TM; i++)
#pragma unroll
                for (int j = 0; j < TM; j++) {   /* a conj(b) */
                    accr[i][j] = fma(av[i].x, bv[j].x, accr[i][j]);
                    accr[i][j] = fma(av[i].y, bv[j].y, accr[i][j]);
                    acci[i][j] = fma(av[i].y, bv[j].x, acci[i][j]);
                    acci[i][j] = fma(-av[i].x, bv[j].y, acci[i][j]);
                }
        }
    }

    /* fold the KS column splits of a micro-tile: xor butterfly over the lanes, then the warps in order */
    if (KS > 1) {
#pragma unroll
        for (int o = 1; o < (KS < 32 ? KS : 32); o <<= 1)
#pragma unroll
            for (int i = 0; i < TM; i++)
#pragma unroll
                for (int j = 0; j < TM; j++) {
                    accr[i][j] += __shfl_xor_sync(0xffffffffu, accr[i][j], o);
                    acci[i][j] += __shfl_xor_sync(0xffffffffu, acci[i][j], o);
                }
    }
    const bool direct = a.nsplit == 1;
    const size_t ld = direct ? (size_t)a.nb * BM : BM;
    double2 *dst = direct ? a.out + (size_t)I * BM * ld + (size_t)J * BM : a.out + (size_t)blockIdx.x * BM * BM;
    if (KS <= 32) {
        if (ks == 0) {
#pragma unroll
            for (int i = 0; i < TM; i++)
#pragma unroll
                for (int j = 0; j < TM; j++) dst[(gy + GW * i) * ld + gx + GW * j] = make_double2(accr[i][j], acci[i][j]);
        }
    } else {
        constexpr int WPG = KS / 32;   /* warps per micro-tile */
        __syncthreads();                /* sm is free: every thread is past its last chunk */
        double2 *red = sm;              /* [warp][TM * TM] */
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < TM; i++)
#pragma unroll
                for (int j = 0; j < TM; j++) red[(tid >> 5) * TM * TM + i * TM + j] = make_double2(accr[i][j], acci[i][j]);
        }
        __syncthreads();
        if (tid < G * TM * TM) {
            const int gg = tid / (TM * TM), e = tid % (TM * TM), i = e / TM, j = e % TM;
            double2 v = red[(gg * WPG) * TM * TM + e];
            for (int w = 1; w < WPG; w++) { const double2 x = red[(gg * WPG + w) * TM * TM + e]; v.x += x.x; v.y += x.y; }
            dst[((gg / GW) + GW * i) * ld + (gg % GW) + GW * j] = v;
        }
    }
}

/* result block entries = the nsplit partials of the block pair, summed in split order */
__global__ void k_rdm_finish(const double2 *partial, int nsplit, int BM, int nb, int full, size_t nent, double2 *out)
{
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nent) return;
    const size_t bb = (size_t)BM * BM, p = t / bb, e = t % bb;
    int I, J;
    if (full) { I = (int)(p / nb); J = (int)(p % nb); }
    else { int q = (int)p; I = 0; while (q >= nb - I) { q -= nb - I; I++; } J = I + q; }
    double2 acc = make_double2(0.0, 0.0);
    for (int sp = 0; sp < nsplit; sp++) {
        const double2 x = partial[(p * nsplit + sp) * bb + e];
        acc.x += x.x; acc.y += x.y;
    }
    out[((size_t)I * BM + e / BM) * ((size_t)nb * BM) + (size_t)J * BM + e % BM] = acc;
}

/* ================================================================================================ host */

namespace {

struct RdmGeom {
    bool f32 = true;
    int k = 0, k_loc = 0, BM = 1, nb = 1, KC = 1, nchunks = 1;
    std::vector<int> lq, rq;   /* indices i into qubits[] on local / rank bits, local ones in physical order */
    std::vector<int> rbit;     /* rank bit of qubits[rq[j]] */
    RdmArgs args;              /* the launch-independent fields */
};

void rdm_geometry(const qsb_sim *s, const int *qubits, int k, RdmGeom &G)
{
    G.f32 = s->prec == QSB_F32;
    G.k = k;
    uint64_t mloc = 0;
    for (int i = 0; i < k; i++) {
        const int p = s->perm.pos[qubits[i]];
        if (p < s->nloc) mloc |= 1ULL << p;
        else { G.rq.push_back(i); G.rbit.push_back(p - s->nloc); }
    }
    RdmArgs &a = G.args;
    memset(&a, 0, sizeof a);
    for (int b = 0; b < s->nloc; b++) {
        if ((mloc >> b) & 1) {
            a.mpos[a.n_m++] = (int8_t)b;
            for (int i = 0; i < k; i++) if (s->perm.pos[qubits[i]] == b) G.lq.push_back(i);   /* row bit n_m - 1 */
        } else {
            a.upos[a.n_u++] = (int8_t)b;
        }
    }
    G.k_loc = a.n_m;
    const int S = G.f32 ? 6 : 5;
    a.mlow = (uint32_t)(mloc & ((1u << S) - 1));
    a.m_low = __builtin_popcount(a.mlow);
    const int R = 1 << G.k_loc;
    G.BM = std::min(R, RDM_BMAX);   /* >= 2^m_low: a row block holds whole segments */
    G.nb = R / G.BM;
    const uint64_t C = 1ULL << a.n_u;
    G.KC = (int)std::min<uint64_t>(RDM_CH(G.f32) / G.BM, C);   /* >= 2^(S - m_low): whole segments */
    G.nchunks = (int)(C / G.KC);
    a.KC = G.KC;
    a.nb = G.nb;
}

size_t smem_bytes(const RdmGeom &G, bool two) { return (two ? 2 : 1) * (size_t)G.BM * (RDM_CH(G.f32) / G.BM + 1) * sizeof(double2); }

template <int BM, bool F32>
int launch_bm(qsb_sim *s, const RdmArgs &a, unsigned grid, size_t smem)
{
    QSB_CUDA(cudaFuncSetAttribute(k_rdm<BM, F32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_rdm<BM, F32><<<grid, RDM_THREADS, smem, s->stream>>>(a);
    return QSB_OK;
}

template <bool F32>
int launch_f(qsb_sim *s, int BM, const RdmArgs &a, unsigned grid, size_t smem)
{
    switch (BM) {
    case 1: return launch_bm<1, F32>(s, a, grid, smem);
    case 2: return launch_bm<2, F32>(s, a, grid, smem);
    case 4: return launch_bm<4, F32>(s, a, grid, smem);
    case 8: return launch_bm<8, F32>(s, a, grid, smem);
    case 16: return launch_bm<16, F32>(s, a, grid, smem);
    case 32: return launch_bm<32, F32>(s, a, grid, smem);
    default: return launch_bm<64, F32>(s, a, grid, smem);
    }
}

/* column splits: enough CTAs for several waves, partials within RDM_PARTIAL_BYTES */
int choose_nsplit(const RdmGeom &G, int npairs, int nsm)
{
    const size_t blk = (size_t)G.BM * G.BM * sizeof(double2);
    int ns = 1;
    while (2 * ns <= G.nchunks && (size_t)npairs * ns < (size_t)nsm * 8 && (size_t)npairs * 2 * ns * blk <= RDM_PARTIAL_BYTES) ns *= 2;
    return ns;
}

/* bytes of the per-CTA partials of one launch (0 when a CTA writes its block straight into the result) */
size_t partial_bytes(const RdmGeom &G, int npairs, int nsm)
{
    const int ns = choose_nsplit(G, npairs, nsm);
    return ns > 1 ? (size_t)npairs * ns * G.BM * G.BM * sizeof(double2) : 0;
}

/* rho_loc = A A^H (full = 0: upper block triangle of the own shard) or A B^H (full = 1: B = the partner shard in
 * state2, every block) into d_out (R x R, local row order) */
int launch_rdm(qsb_sim *s, const RdmGeom &G, bool full, int nsm, double2 *d_out, double2 *d_partial)
{
    RdmArgs a = G.args;
    a.A = (const uint4 *)s->state;
    a.B = (const uint4 *)(full ? s->state2 : s->state);
    a.full = full ? 1 : 0;
    const int npairs = full ? G.nb * G.nb : G.nb * (G.nb + 1) / 2;
    a.nsplit = choose_nsplit(G, npairs, nsm);
    a.cps = G.nchunks / a.nsplit;
    a.out = a.nsplit == 1 ? d_out : d_partial;
    const unsigned grid = (unsigned)(npairs * a.nsplit);
    const size_t smem = smem_bytes(G, full || G.nb > 1);
    int rc = G.f32 ? launch_f<true>(s, G.BM, a, grid, smem) : launch_f<false>(s, G.BM, a, grid, smem);
    if (rc) return rc;
    if (a.nsplit > 1) {
        const size_t nent = (size_t)npairs * G.BM * G.BM;
        k_rdm_finish<<<(unsigned)((nent + 255) / 256), 256, 0, s->stream>>>(d_partial, a.nsplit, G.BM, G.nb, a.full, nent, d_out);
    }
    QSB_CUDA(cudaGetLastError());
    return QSB_OK;
}

struct DevMem {   /* scoped device allocation */
    void *p = nullptr;
    ~DevMem() { if (p) cudaFree(p); }
};

/* every rank's 2^m local matrices h[r][d] (R x R, local order; d = 0 holds the upper triangle) placed in qubits[] order
 * and summed in rank order; then the upper triangle mirrored */
void assemble(const qsb_sim *s, const RdmGeom &G, const std::vector<double> &h, double *rho)
{
    const size_t R = (size_t)1 << G.k_loc, K = (size_t)1 << G.k, nd = (size_t)1 << G.rq.size();
    std::vector<uint32_t> idx(R, 0);   /* local row index -> bits of the local qubits in qubits[] order */
    for (int j = 0; j < G.k_loc; j++)
        for (size_t o = 0; o < ((size_t)1 << j); o++) idx[o | ((size_t)1 << j)] = idx[o] | (1u << G.lq[j]);
    auto rank_bits = [&](int r) {
        uint32_t v = 0;
        for (size_t i = 0; i < G.rq.size(); i++) v |= (uint32_t)((r >> G.rbit[i]) & 1) << G.rq[i];
        return v;
    };
    std::fill(rho, rho + 2 * K * K, 0.0);
    for (int r = 0; r < s->world; r++) {
        for (size_t d = 0; d < nd; d++) {
            int D = 0;
            for (size_t i = 0; i < G.rq.size(); i++) if ((d >> i) & 1) D |= 1 << G.rbit[i];
            const uint32_t rbr = rank_bits(r), rbc = rank_bits(r ^ D);
            const double *L = h.data() + ((size_t)r * nd + d) * R * R * 2;
            for (size_t x = 0; x < R; x++) {
                const size_t A = idx[x] | rbr;
                for (size_t y = 0; y < R; y++) {
                    const size_t B = idx[y] | rbc;
                    if (A > B) continue;
                    double *o = rho + 2 * (A * K + B);
                    if (d == 0 && x > y) { const double *v = L + 2 * (y * R + x); o[0] += v[0]; o[1] += -v[1]; }
                    else { const double *v = L + 2 * (x * R + y); o[0] += v[0]; o[1] += v[1]; }
                }
            }
        }
    }
    for (size_t A = 0; A < K; A++) {
        rho[2 * (A * K + A) + 1] = 0.0;
        for (size_t B = 0; B < A; B++) {
            rho[2 * (A * K + B)] = rho[2 * (B * K + A)];
            rho[2 * (A * K + B) + 1] = -rho[2 * (B * K + A) + 1];
        }
    }
}

}  // namespace

/* ------------------------------------------------------------------------------------------- C ABI */

extern "C" int qsb_reduced_density_matrix(qsb_t *s, const int *qubits, int k, double *rho)
{
    const char *fn = "qsb_reduced_density_matrix";
    if (!s) { qsb_set_error("%s: null handle", fn); return QSB_ERR_ARG; }
    int rc = check_qubits(s, qubits, k, RDM_KMAX, fn, "a larger rho needs more than 256 MiB");
    if (rc) return rc;
    if (!rho) { qsb_set_error("%s: null output", fn); return QSB_ERR_ARG; }
    if (s->g && !s->comm) { qsb_set_error("%s: sharded state needs qsb_comm_init first", fn); return QSB_ERR_COMM; }
    QSB_CUDA(cudaSetDevice(s->device));
    RdmGeom G;
    rdm_geometry(s, qubits, k, G);
    int nsm = 0;
    QSB_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, s->device));

    const size_t R = (size_t)1 << G.k_loc, nd = (size_t)1 << G.rq.size();
    const size_t mat = R * R * sizeof(double2), mats = nd * mat;
    const size_t all = s->g ? (size_t)s->world * mats : 0;
    const size_t part = std::max(partial_bytes(G, G.nb * (G.nb + 1) / 2, nsm), nd > 1 ? partial_bytes(G, G.nb * G.nb, nsm) : 0);
    DevMem mem;
    QSB_CUDA(cudaMalloc(&mem.p, mats + all + part));
    double2 *d_mat = (double2 *)mem.p;
    double2 *d_all = (double2 *)((char *)mem.p + mats);
    double2 *d_part = (double2 *)((char *)mem.p + mats + all);

    rc = launch_rdm(s, G, false, nsm, d_mat, d_part);
    for (size_t d = 1; !rc && d < nd; d++) {
        int D = 0;
        for (size_t i = 0; i < G.rq.size(); i++) if ((d >> i) & 1) D |= 1 << G.rbit[i];
        rc = tiled_comm_sendrecv(s, s->state, s->state2, s->state_bytes, s->rank ^ D);
        if (!rc) rc = launch_rdm(s, G, true, nsm, d_mat + d * R * R, d_part);
    }
    /* every rank's matrices (the all-gather also orders this call before any later use of state2 by a peer) */
    if (!rc && s->g) rc = tiled_comm_allgather(s, d_mat, d_all, mats);
    if (rc) { cudaStreamSynchronize(s->stream); return rc; }
    std::vector<double> h(2 * (s->g ? (size_t)s->world : 1) * nd * R * R);
    QSB_CUDA(cudaMemcpyAsync(h.data(), s->g ? d_all : d_mat, h.size() * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    QSB_CUDA(cudaStreamSynchronize(s->stream));
    assemble(s, G, h, rho);
    return QSB_OK;
}
