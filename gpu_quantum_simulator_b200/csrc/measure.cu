/*
 * measure.cu -- marginal probabilities of chosen qubits and projective measurement on the device (DESIGN.md section 3.3).
 *
 * The qubits come as qubits[0..k-1]; bit i of a bin index or outcome is the value of qubits[i].  Everything is fp64 over
 * the state as stored, nothing is renormalised.
 *
 * MARGINAL.  k_marginal reads the shard in physical order, whatever the measured qubits: a CTA of 128 threads takes
 * tiles whose low physical bits are the f32 pack bit (f32) and seven unit-address bits (so a warp reads 512 contiguous
 * bytes), plus up to four unmeasured higher bits as the per-thread units.  The rest of the local bits are outer bits:
 * the measured ones are constant within a CTA (they select the part of the table the CTA feeds), the unmeasured ones
 * are split between the CTAs of that pattern (2^g_bits of them) and the tiles each CTA walks.  So a thread's units all
 * fall into one bin per pack lane: a thread keeps one fp64 sum per lane, serially over its units and tiles; the CTA
 * folds the 256 (f32) / 128 (f64) thread sums over the unmeasured in-tile bits by a fixed tree in shared memory and
 * writes one partial per in-tile bin to scratch; k_marginal_finish sums each bin over its CTAs in CTA order.  No
 * floating-point atomics anywhere, so repeated calls return identical bits.  Padding bits of small registers (zero
 * amplitudes) are never measured; they are read and add zeros.
 *
 * The per-CTA partials live in the staging buffer behind the 2^20-bin table (the calls block, as the downloads do):
 * CTAs x in-tile bins = 2^(m_o + g_bits + m_in) <= 2^max(13 + 8, 22) doubles, at most 32 MiB of the 56 MiB left.
 *
 * COLLAPSE.  One streaming pass: units whose measured bits differ from the outcome are written as zero without being
 * read; kept units are read, scaled by 1/sqrt(p) in fp64 and written (f32 with the pack bit measured: the other lane
 * is zeroed).  The probability p of the outcome comes from the same kernel as the marginal, launched for the CTAs of
 * the outcome's pattern only and with the threads of other in-tile bins idle, so it equals the matching table entry
 * bit for bit and costs a read of the kept amplitudes only.  The state buffer, state2, the peer mappings and a captured
 * graph's buffer stay as they are.
 *
 * SHARDED.  Measured qubits on rank bits select which bins a rank's table feeds.  The per-rank tables over the local
 * measured qubits are all-gathered and every rank sums them on the host in rank order, so every rank holds the same
 * table and draws the same outcome from the same r.  A rank whose rank bits disagree with the outcome zeroes its shard.
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "sim.h"
#include "tiled.h"

int tiled_comm_allgather(qsb_sim *s, const void *dsrc, void *ddst, size_t bytes);

#define MRG_THREADS 128
#define MRG_TB 7                     /* thread bits = unit-address bits 0..6 */
#define MRG_NU 16                    /* units (16 bytes) per thread and tile, at most */
#define MRG_UB 4                     /* log2(MRG_NU) */
#define MRG_KMAX 20                  /* qubits per call */
#define MRG_HINT "measure more than 20 qubits in groups"
#define MRG_TABLE_BYTES ((size_t)8 << 20)   /* 2^20 fp64 bins at the start of the staging buffer */
#define MRG_CTA_TARGET_LOG2 13       /* ~8192 CTAs: many waves of 148 SMs, a small tail */
/* the in-tile bits (pack + thread bits) exist in every shard: nloc >= tiled_min_local_bits() */
static_assert(MRG_TB + 1 <= QSB_T_F32 && MRG_TB <= QSB_T_F64, "the marginal tile must fit the smallest shard");

struct MargArgs {
    const uint4 *A;
    double *partial;              /* [gridDim.x][1 << m_in] */
    uint64_t uoff[MRG_UB];        /* unit-address offset of unit bit b (unmeasured bits) */
    uint64_t P_base;              /* outer measured pattern of CTA 0 */
    int nu;                       /* units per thread and tile */
    int m_o, u_o, g_bits, m_in;   /* outer measured / unmeasured bits, log2(CTAs per pattern), in-tile measured bits */
    uint32_t tmask, tval;         /* threads whose measured thread bits differ from tval read nothing */
    uint32_t fold, mcoord;        /* unmeasured / measured in-tile coordinate bits */
    int8_t mpos[MRG_KMAX];        /* unit-address bit of outer measured bit i */
    int8_t wpos[64];              /* unit-address bit of outer unmeasured bit i */
};

struct MargMap { int8_t pos[MRG_KMAX]; int n; };   /* bit j of an output index -> bit pos[j] of the pext-order index */

/* ================================================================================================ device */

__device__ __forceinline__ uint64_t deposit(uint64_t v, const int8_t *pos, int n)
{
    uint64_t r = 0;
    for (int i = 0; i < n; i++) r |= ((v >> i) & 1ULL) << pos[i];
    return r;
}

template <bool F32>
__global__ void __launch_bounds__(MRG_THREADS) k_marginal(const __grid_constant__ MargArgs a)
{
    constexpr int C = F32 ? 2 * MRG_THREADS : MRG_THREADS;   /* in-tile coordinates: (thread, pack lane) */
    __shared__ double s_part[C];
    const uint32_t tid = threadIdx.x;
    const uint64_t g = blockIdx.x & ((1u << a.g_bits) - 1);
    const uint64_t base_m = deposit(a.P_base + (blockIdx.x >> a.g_bits), a.mpos, a.m_o) | tid;
    const uint64_t ntiles = 1ULL << (a.u_o - a.g_bits);
    double acc0 = 0.0, acc1 = 0.0;
    if ((tid & a.tmask) == a.tval) {
        for (uint64_t i = 0; i < ntiles; i++) {
            const uint64_t base = base_m | deposit((i << a.g_bits) | g, a.wpos, a.u_o);
            uint4 av[MRG_NU];
#pragma unroll
            for (int u = 0; u < MRG_NU; u++) {
                if (u < a.nu) {
                    uint64_t uo = 0;
#pragma unroll
                    for (int b = 0; b < MRG_UB; b++) if ((u >> b) & 1) uo |= a.uoff[b];
                    av[u] = __ldcs(a.A + (base | uo));
                }
            }
#pragma unroll
            for (int u = 0; u < MRG_NU; u++) {
                if (u < a.nu) {
                    if (F32) {
                        const float4 x = *reinterpret_cast<const float4 *>(&av[u]);   /* re0 re1 im0 im1 */
                        const double r0 = x.x, r1 = x.y, i0 = x.z, i1 = x.w;
                        acc0 += r0 * r0 + i0 * i0;
                        acc1 += r1 * r1 + i1 * i1;
                    } else {
                        const double2 x = *reinterpret_cast<const double2 *>(&av[u]);
                        acc0 += x.x * x.x + x.y * x.y;
                    }
                }
            }
        }
    }
    if (F32) { s_part[2 * tid] = acc0; s_part[2 * tid + 1] = acc1; }
    else s_part[tid] = acc0;
    for (uint32_t f = a.fold; f; f &= f - 1) {   /* fixed tree: unmeasured coordinate bits, lowest first */
        const uint32_t bit = f & (0u - f);
        __syncthreads();
        for (uint32_t c = tid; c < C; c += MRG_THREADS) if (!(c & bit)) s_part[c] += s_part[c | bit];
    }
    __syncthreads();
    const uint32_t bins = 1u << a.m_in;
    for (uint32_t j = tid; j < bins; j += MRG_THREADS) {
        uint32_t c = 0, m = a.mcoord;
        for (int i = 0; m; m &= m - 1, i++) if ((j >> i) & 1) c |= m & (0u - m);
        a.partial[(size_t)blockIdx.x * bins + j] = s_part[c];
    }
}

/* out[o] = sum over the CTAs of the bin's pattern, in CTA order.  The bin is L = L_base | deposit(o, map): outer
 * measured pattern L >> m_in (relative to the P_base of the launch), in-tile bin L & (2^m_in - 1). */
__global__ void k_marginal_finish(const double *partial, int g_bits, int m_in, uint32_t nout, uint64_t L_base, uint64_t P_base,
                                  const __grid_constant__ MargMap map, double *out)
{
    const uint32_t o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= nout) return;
    const uint64_t L = L_base | deposit(o, map.pos, map.n);
    const size_t G = (size_t)1 << g_bits, bins = (size_t)1 << m_in;
    const size_t first = ((L >> m_in) - P_base) * G * bins + (L & (bins - 1));
    double acc = 0.0;
    for (size_t g = 0; g < G; g++) acc += partial[first + g * bins];
    out[o] = acc;
}

/* Units whose measured bits (umask) differ from uval become zero without being read; kept units are scaled.  lane >= 0
 * (f32, pack bit measured): only that lane of a kept unit is kept. */
template <bool F32>
__global__ void __launch_bounds__(256) k_collapse(uint4 *A, uint64_t nunits, uint64_t umask, uint64_t uval, int lane, double scale)
{
    constexpr int U = 4;   /* units per thread and step, loads issued together */
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x * U;
    for (uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x * U + threadIdx.x; i0 < nunits; i0 += step) {
        uint4 v[U];
        bool keep[U];
#pragma unroll
        for (int j = 0; j < U; j++) {
            const uint64_t i = i0 + (uint64_t)j * blockDim.x;
            keep[j] = i < nunits && (i & umask) == uval;
            v[j] = keep[j] ? __ldcs(A + i) : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
        for (int j = 0; j < U; j++) {
            const uint64_t i = i0 + (uint64_t)j * blockDim.x;
            if (i >= nunits) break;
            if (keep[j]) {
                if (F32) {
                    float4 x = *reinterpret_cast<const float4 *>(&v[j]);
                    x.x = (float)((double)x.x * scale); x.y = (float)((double)x.y * scale);
                    x.z = (float)((double)x.z * scale); x.w = (float)((double)x.w * scale);
                    if (lane == 0) { x.y = 0.f; x.w = 0.f; }
                    else if (lane == 1) { x.x = 0.f; x.z = 0.f; }
                    v[j] = *reinterpret_cast<const uint4 *>(&x);
                } else {
                    double2 x = *reinterpret_cast<const double2 *>(&v[j]);
                    x.x *= scale; x.y *= scale;
                    v[j] = *reinterpret_cast<const uint4 *>(&x);
                }
            }
            __stcs(A + i, v[j]);
        }
    }
}

/* ================================================================================================ host */

/* the argument rules shared by the calls that take a list of qubits (measure.cu, rdm.cu) */
int check_qubits(const qsb_sim *s, const int *qubits, int k, int kmax, const char *fn, const char *hint)
{
    if (!qubits) { qsb_set_error("%s: null qubit array", fn); return QSB_ERR_ARG; }
    kmax = std::min(s->n, kmax);
    if (k < 1 || k > kmax) {
        qsb_set_error("%s: %d qubits, expected 1..%d (%s)", fn, k, kmax, hint);
        return QSB_ERR_ARG;
    }
    uint64_t seen = 0;
    for (int i = 0; i < k; i++) {
        const int q = qubits[i];
        if (q < 0 || q >= s->n) { qsb_set_error("%s: qubit %d outside [0, %d)", fn, q, s->n); return QSB_ERR_ARG; }
        if ((seen >> q) & 1) { qsb_set_error("%s: qubit %d appears twice", fn, q); return QSB_ERR_ARG; }
        seen |= 1ULL << q;
    }
    return QSB_OK;
}

namespace {

struct Geom {
    bool f32 = true;
    int k = 0, k_loc = 0, m_in = 0, m_o = 0, u_o = 0, g_bits = 0, nu_bits = 0;
    uint64_t mloc = 0;                 /* measured local physical bits */
    uint32_t mcoord = 0, fold = 0;     /* in-tile coordinate bits (physical bits 0..7 f32 / 0..6 f64) */
    uint64_t uoff[MRG_UB] = {0, 0, 0, 0};
    int8_t mpos[MRG_KMAX] = {0}, wpos[64] = {0};
    std::vector<int> lq, rq;           /* indices i into qubits[] on local / rank bits, in qubits[] order */
    std::vector<int> lphys, rbit;      /* their physical bit / rank bit */
};

void geometry(const qsb_sim *s, const int *qubits, int k, Geom &G)
{
    G.f32 = s->prec == QSB_F32;
    G.k = k;
    const int su = G.f32 ? 1 : 0, cb = MRG_TB + su;
    for (int i = 0; i < k; i++) {
        const int p = s->perm.pos[qubits[i]];
        if (p < s->nloc) { G.lq.push_back(i); G.lphys.push_back(p); G.mloc |= 1ULL << p; }
        else { G.rq.push_back(i); G.rbit.push_back(p - s->nloc); }
    }
    G.k_loc = (int)G.lq.size();
    const uint32_t cmask = (1u << cb) - 1;
    G.mcoord = (uint32_t)G.mloc & cmask;
    G.fold = cmask & ~G.mcoord;
    G.m_in = __builtin_popcount(G.mcoord);
    for (int b = cb; b < s->nloc; b++) {
        if ((G.mloc >> b) & 1) G.mpos[G.m_o++] = (int8_t)(b - su);
        else if (G.nu_bits < MRG_UB) G.uoff[G.nu_bits++] = 1ULL << (b - su);
        else G.wpos[G.u_o++] = (int8_t)(b - su);
    }
    /* partials: 2^(m_o + g_bits + m_in) <= 2^max(13 + m_in, 22) doubles */
    G.g_bits = std::max(0, std::min({MRG_CTA_TARGET_LOG2 - G.m_o, G.u_o, 22 - G.k_loc}));
}

/* the local pext-order index (measured local physical bits, ascending) of the local qubit j */
int lbit(const Geom &G, int j) { return __builtin_popcountll(G.mloc & ((1ULL << G.lphys[j]) - 1)); }

struct DevMem {   /* scoped device allocation */
    void *p = nullptr;
    ~DevMem() { if (p) cudaFree(p); }
};

double *partial_buf(qsb_sim *s) { return (double *)((char *)s->staging + MRG_TABLE_BYTES); }

/* Launches the reduction.  restricted: only the bin of pext-order index Lstar, into d_out[0]; otherwise the whole local
 * table in local-qubit order (bit j = the j-th local qubit of qubits[]) into d_out. */
int launch_marginal(qsb_sim *s, const Geom &G, bool restricted, uint64_t Lstar, double *d_out)
{
    static_assert(((size_t)1 << 22) * sizeof(double) <= ((size_t)64 << 20) - MRG_TABLE_BYTES, "partials fit the staging buffer");
    if (s->staging_bytes < ((size_t)64 << 20)) { qsb_set_error("staging buffer too small for the marginal partials"); return QSB_ERR_NOMEM; }
    MargArgs a; memset(&a, 0, sizeof a);
    a.A = (const uint4 *)s->state;
    a.partial = partial_buf(s);
    memcpy(a.uoff, G.uoff, sizeof a.uoff);
    a.nu = 1 << G.nu_bits;
    a.m_o = G.m_o; a.u_o = G.u_o; a.g_bits = G.g_bits; a.m_in = G.m_in;
    a.fold = G.fold; a.mcoord = G.mcoord;
    memcpy(a.mpos, G.mpos, sizeof a.mpos);
    memcpy(a.wpos, G.wpos, sizeof a.wpos);
    const int su = G.f32 ? 1 : 0;
    uint64_t grid;
    MargMap map; memset(&map, 0, sizeof map);
    uint32_t nout;
    uint64_t L_base = 0;
    if (restricted) {
        a.P_base = Lstar >> G.m_in;
        uint32_t cval = 0, m = G.mcoord;   /* the in-tile bin as coordinate bits */
        for (int i = 0; m; m &= m - 1, i++) if ((Lstar >> i) & 1) cval |= m & (0u - m);
        a.tmask = G.mcoord >> su;
        a.tval = cval >> su;
        grid = 1ULL << G.g_bits;
        nout = 1; L_base = Lstar;
    } else {
        grid = 1ULL << (G.m_o + G.g_bits);
        map.n = G.k_loc;
        for (int j = 0; j < G.k_loc; j++) map.pos[j] = (int8_t)lbit(G, j);
        nout = 1u << G.k_loc;
    }
    if (G.f32) k_marginal<true><<<(unsigned)grid, MRG_THREADS, 0, s->stream>>>(a);
    else k_marginal<false><<<(unsigned)grid, MRG_THREADS, 0, s->stream>>>(a);
    k_marginal_finish<<<(nout + 255) / 256, 256, 0, s->stream>>>(a.partial, G.g_bits, G.m_in, nout, L_base, a.P_base, map, d_out);
    QSB_CUDA(cudaGetLastError());
    return QSB_OK;
}

/* does rank r hold the amplitudes whose measured rank qubits carry the values of `outcome`? */
bool rank_matches(const Geom &G, int r, uint64_t outcome)
{
    for (size_t i = 0; i < G.rq.size(); i++)
        if (((outcome >> G.rq[i]) & 1) != (uint64_t)((r >> G.rbit[i]) & 1)) return false;
    return true;
}

/* The full table in bin order (bit i = qubits[i]) on the host of every rank. */
int marginal_table(qsb_sim *s, const Geom &G, double *out)
{
    double *d_tab = (double *)s->staging;
    int rc = launch_marginal(s, G, false, 0, d_tab);
    if (rc) { cudaStreamSynchronize(s->stream); return rc; }
    const size_t nloc_bins = (size_t)1 << G.k_loc;
    if (!s->g) {   /* every qubit is local and in qubits[] order: the table is the answer */
        QSB_CUDA(cudaMemcpyAsync(out, d_tab, nloc_bins * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
        QSB_CUDA(cudaStreamSynchronize(s->stream));
        return QSB_OK;
    }
    /* every rank's table: into the partials area, free again once k_marginal_finish has run (same stream); only
     * many ranks with k_loc near 20 need more than its 56 MiB */
    const size_t all_bytes = (size_t)s->world * nloc_bins * sizeof(double);
    DevMem big;
    void *d_all = partial_buf(s);
    if (all_bytes > s->staging_bytes - MRG_TABLE_BYTES) {
        QSB_CUDA(cudaMalloc(&big.p, all_bytes));
        d_all = big.p;
    }
    rc = tiled_comm_allgather(s, d_tab, d_all, nloc_bins * sizeof(double));
    if (rc) { cudaStreamSynchronize(s->stream); return rc; }
    std::vector<double> h((size_t)s->world * nloc_bins);
    QSB_CUDA(cudaMemcpyAsync(h.data(), d_all, all_bytes, cudaMemcpyDeviceToHost, s->stream));
    QSB_CUDA(cudaStreamSynchronize(s->stream));
    /* local-table index o -> bin bits of the local qubits */
    std::vector<uint32_t> idx(nloc_bins, 0);
    for (int j = 0; j < G.k_loc; j++)
        for (size_t o = 0; o < ((size_t)1 << j); o++) idx[o | ((size_t)1 << j)] = idx[o] | (1u << G.lq[j]);
    std::fill(out, out + ((size_t)1 << G.k), 0.0);
    for (int r = 0; r < s->world; r++) {   /* rank order: every rank adds the same numbers in the same order */
        uint32_t rb = 0;
        for (size_t i = 0; i < G.rq.size(); i++) rb |= (uint32_t)((r >> G.rbit[i]) & 1) << G.rq[i];
        const double *t = h.data() + (size_t)r * nloc_bins;
        for (size_t o = 0; o < nloc_bins; o++) out[idx[o] | rb] += t[o];
    }
    return QSB_OK;
}

/* the outcome's measured local bits as physical bits / as the pext-order index */
uint64_t local_phys(const Geom &G, uint64_t outcome)
{
    uint64_t v = 0;
    for (int j = 0; j < G.k_loc; j++) if ((outcome >> G.lq[j]) & 1) v |= 1ULL << G.lphys[j];
    return v;
}
uint64_t local_pext(const Geom &G, uint64_t outcome)
{
    uint64_t v = 0;
    for (int j = 0; j < G.k_loc; j++) if ((outcome >> G.lq[j]) & 1) v |= 1ULL << lbit(G, j);
    return v;
}

/* p of one outcome, equal bit for bit to its entry of marginal_table() */
int outcome_probability(qsb_sim *s, const Geom &G, uint64_t outcome, double *p)
{
    double *d_p = (double *)s->staging;
    const bool mine = rank_matches(G, s->rank, outcome);
    if (mine) {
        int rc = launch_marginal(s, G, true, local_pext(G, outcome), d_p);
        if (rc) { cudaStreamSynchronize(s->stream); return rc; }
    }
    if (!s->g) {
        QSB_CUDA(cudaMemcpyAsync(p, d_p, sizeof(double), cudaMemcpyDeviceToHost, s->stream));
        QSB_CUDA(cudaStreamSynchronize(s->stream));
        return QSB_OK;
    }
    if (!mine) QSB_CUDA(cudaMemsetAsync(d_p, 0, sizeof(double), s->stream));
    double *d_all = d_p + 1;
    int rc = tiled_comm_allgather(s, d_p, d_all, sizeof(double));
    if (rc) { cudaStreamSynchronize(s->stream); return rc; }
    std::vector<double> h(s->world);
    QSB_CUDA(cudaMemcpyAsync(h.data(), d_all, s->world * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    QSB_CUDA(cudaStreamSynchronize(s->stream));
    double acc = 0.0;   /* the additions of marginal_table() for this bin */
    for (int r = 0; r < s->world; r++) if (rank_matches(G, r, outcome)) acc += h[r];
    *p = acc;
    return QSB_OK;
}

int collapse_pass(qsb_sim *s, const Geom &G, uint64_t outcome, double p)
{
    if (!rank_matches(G, s->rank, outcome)) {
        QSB_CUDA(cudaMemsetAsync(s->state, 0, s->state_bytes, s->stream));
    } else {
        const int su = G.f32 ? 1 : 0;
        const uint64_t pv = local_phys(G, outcome);
        const uint64_t nunits = 1ULL << (s->nloc - su);
        const int lane = (G.f32 && (G.mloc & 1)) ? (int)(pv & 1) : -1;
        const unsigned grid = (unsigned)std::min<uint64_t>((nunits + 1023) / 1024, 148ULL * 32);
        const double scale = 1.0 / sqrt(p);
        if (G.f32) k_collapse<true><<<grid, 256, 0, s->stream>>>((uint4 *)s->state, nunits, G.mloc >> 1, pv >> 1, lane, scale);
        else k_collapse<false><<<grid, 256, 0, s->stream>>>((uint4 *)s->state, nunits, G.mloc, pv, -1, scale);
    }
    QSB_CUDA(cudaGetLastError());
    QSB_CUDA(cudaStreamSynchronize(s->stream));
    return QSB_OK;
}

}  // namespace

/* declared in sim.h */
int pick_outcome(const std::vector<double> &tab, double r, uint64_t *b_out, const char *fn)
{
    double T = 0.0;
    for (double v : tab) T += v;
    if (!(T > 0.0)) { qsb_set_error("%s: the measured qubits have total probability %g", fn, T); return QSB_ERR_ARG; }
    const double target = r * T;
    double c = 0.0;
    for (size_t b = 0; b < tab.size(); b++) {
        c += tab[b];
        if (c != 0.0 && c >= target) { *b_out = b; return QSB_OK; }
    }
    *b_out = tab.size() - 1;   /* not reached: C_last = T >= r * T and T != 0 */
    return QSB_OK;
}

namespace {

int measure_common(qsb_sim *s, const int *qubits, int k, double r, uint64_t *outcome, double *prob, const char *fn)
{
    if (!s) { qsb_set_error("%s: null handle", fn); return QSB_ERR_ARG; }
    int rc = check_qubits(s, qubits, k, MRG_KMAX, fn, MRG_HINT);
    if (rc) return rc;
    if (!outcome) { qsb_set_error("%s: null outcome", fn); return QSB_ERR_ARG; }
    if (!(r >= 0.0 && r < 1.0)) { qsb_set_error("%s: r = %g outside [0, 1)", fn, r); return QSB_ERR_ARG; }
    if (s->g && !s->comm) { qsb_set_error("%s: sharded state needs qsb_comm_init first", fn); return QSB_ERR_COMM; }
    QSB_CUDA(cudaSetDevice(s->device));
    Geom G;
    geometry(s, qubits, k, G);
    std::vector<double> tab((size_t)1 << k);
    rc = marginal_table(s, G, tab.data());
    if (rc) return rc;
    uint64_t b = 0;
    rc = pick_outcome(tab, r, &b, fn);
    if (rc) return rc;
    rc = collapse_pass(s, G, b, tab[b]);
    if (rc) return rc;
    *outcome = b;
    if (prob) *prob = tab[b];
    return QSB_OK;
}

}  // namespace

/* ------------------------------------------------------------------------------------------- C ABI */

extern "C" int qsb_marginal_probabilities(qsb_t *s, const int *qubits, int k, double *out)
{
    if (!s) { qsb_set_error("qsb_marginal_probabilities: null handle"); return QSB_ERR_ARG; }
    int rc = check_qubits(s, qubits, k, MRG_KMAX, "qsb_marginal_probabilities", MRG_HINT);
    if (rc) return rc;
    if (!out) { qsb_set_error("qsb_marginal_probabilities: null output"); return QSB_ERR_ARG; }
    if (s->g && !s->comm) { qsb_set_error("qsb_marginal_probabilities: sharded state needs qsb_comm_init first"); return QSB_ERR_COMM; }
    QSB_CUDA(cudaSetDevice(s->device));
    Geom G;
    geometry(s, qubits, k, G);
    return marginal_table(s, G, out);
}

extern "C" int qsb_collapse(qsb_t *s, const int *qubits, int k, uint64_t outcome, double *prob)
{
    if (!s) { qsb_set_error("qsb_collapse: null handle"); return QSB_ERR_ARG; }
    int rc = check_qubits(s, qubits, k, MRG_KMAX, "qsb_collapse", MRG_HINT);
    if (rc) return rc;
    if (outcome >> k) { qsb_set_error("qsb_collapse: outcome %llu >= 2^%d", (unsigned long long)outcome, k); return QSB_ERR_ARG; }
    if (s->g && !s->comm) { qsb_set_error("qsb_collapse: sharded state needs qsb_comm_init first"); return QSB_ERR_COMM; }
    QSB_CUDA(cudaSetDevice(s->device));
    Geom G;
    geometry(s, qubits, k, G);
    double p = 0.0;
    rc = outcome_probability(s, G, outcome, &p);
    if (rc) return rc;
    if (!(p > 0.0)) { qsb_set_error("qsb_collapse: outcome %llu has probability %g", (unsigned long long)outcome, p); return QSB_ERR_ARG; }
    rc = collapse_pass(s, G, outcome, p);
    if (rc) return rc;
    if (prob) *prob = p;
    return QSB_OK;
}

extern "C" int qsb_measure_qubits(qsb_t *s, const int *qubits, int k, double r, uint64_t *outcome, double *prob)
{
    return measure_common(s, qubits, k, r, outcome, prob, "qsb_measure_qubits");
}

extern "C" int qsb_reset_qubits(qsb_t *s, const int *qubits, int k, double r, uint64_t *outcome)
{
    uint64_t b = 0;
    int rc = measure_common(s, qubits, k, r, &b, nullptr, "qsb_reset_qubits");
    if (rc) return rc;
    std::vector<qsb_gate_t> xs;
    for (int i = 0; i < k; i++) {
        if (!((b >> i) & 1)) continue;
        qsb_gate_t g; memset(&g, 0, sizeof g);
        g.target = qubits[i];
        g.m[2] = 1.0; g.m[4] = 1.0;   /* X: m01 = m10 = 1 */
        xs.push_back(g);
    }
    if (!xs.empty()) rc = qsb_apply_gates(s, xs.data(), xs.size());
    if (rc) return rc;
    if (outcome) *outcome = b;
    return QSB_OK;
}
