/*
 * expect.cu -- Pauli-string expectation values <psi| P |psi> on the device (DESIGN.md section 3.3).
 *
 * A term is a pair of logical masks (x: X or Y, z: Z or Y).  For the state as stored
 *   <psi|P|psi> = sum_j conj(a_j) i^{popc(x&z)} (-1)^{popc((j^x)&z)} a_{j^x},
 * a sum over every index, so no index gather is needed: only the pairing j <-> j^x.
 *
 * SWEEP.  A sweep fixes a tile bit set B (the low `low_bits` physical bits, so loads stay coalesced and the f32
 * pack bit is inside, plus chosen higher bits up to 12 (f32) / 11 (f64) bits, the tile of tiled.h) and a flip
 * pattern x_out of the local bits outside B.  It evaluates every term whose physical local x equals x_out outside
 * B, whatever its x inside B.  A CTA holds its own tile in registers and stages the partner tile t ^ x_out into
 * shared memory (the tile itself when x_out == 0); then it runs through the batch of terms.  P is Hermitian, so
 * the contribution of the partner tile is the complex conjugate of the tile's own: each pair of tiles is visited
 * once (the tile whose highest x_out bit is clear) and counted twice.  A sweep thus reads the local shard once.
 *
 * SIGNS.  Z bits on the thread bits of the tile coordinate give one sign per thread and term, Z bits on the
 * per-thread unit bits one bit of a 16-bit word per term, Z bits outside B one sign per tile and term, Z bits on
 * rank bits one sign per rank (applied on the host).  i^{popc(x&z)} is a real part or an imaginary part and a sign.
 *
 * GROUPING.  exp_plan() (host only, no CUDA: qsb_expectation_dry_run calls it on a CPU) covers the distinct
 * physical x masks greedily: a sweep starts from the smallest uncovered mask and keeps adding the mask that needs
 * the fewest new tile bits while the tile has room.  Diagonal terms all share one sweep; n weight-1 X terms take
 * ceil((n - low_bits) / (tile - low_bits)); X on every qubit takes one.  A sweep with more than EXP_KMAX terms
 * runs as several launches, each of which rereads the state.
 *
 * REDUCTION.  Deterministic, no floating-point atomics: per thread a short f32 run (8 amplitudes, f32 states) or
 * an fp64 sum, a fixed xor-tree over the warp, one fp64 accumulator per warp and term in shared memory (tiles in
 * a fixed order per CTA), per-CTA partials summed by a second kernel in CTA order.
 *
 * SHARDED.  Terms that flip rank bits (x_rank != 0) need the partner rank's shard: one NCCL send/recv pair per
 * distinct x_rank into state2 (scratch between executions); state / state2 are not swapped and the peer mappings
 * are not touched.  Per-rank values are all-gathered and summed on the host in rank order with the rank signs.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <vector>

#include "pauli.h"
#include "sim.h"
#include "tiled.h"

int tiled_comm_allgather(qsb_sim *s, const void *dsrc, void *ddst, size_t bytes);
int tiled_comm_sendrecv(qsb_sim *s, const void *dsend, void *drecv, size_t bytes, int peer);

#define EXP_THREADS 128
#define EXP_TB 7                    /* thread bits of the tile coordinate */
#define EXP_NU 16                   /* 16-byte units per thread and tile (2 amplitudes f32, 1 amplitude f64) */
#define EXP_UB 4                    /* log2(EXP_NU) */
#define EXP_T_F32 (1 + EXP_TB + EXP_UB)   /* 12: pack lane + thread + unit bits */
#define EXP_T_F64 (EXP_TB + EXP_UB)       /* 11 */
/* a sweep reads pb[0..T-1], which exist because every shard has nloc >= tiled_min_local_bits() = QSB_T_* local bits */
static_assert(EXP_T_F32 <= QSB_T_F32 && EXP_T_F64 <= QSB_T_F64, "the expectation tile must fit the smallest shard");
#define EXP_TILE_UNITS (EXP_THREADS * EXP_NU)
#define EXP_KMAX 512                /* terms per launch: 32 KiB tile + 4 x 512 fp64 accumulators = 48 KiB */
#define EXP_CTAS_PER_SM(f32) ((f32) ? 4 : 3)   /* f64: the tile in registers and fp64 addresses need more than 128 registers */
#define EXP_RUN 4                   /* f32: units (8 amplitudes) summed in f32 before the fp64 accumulator */

enum { EXP_ODD = 1, EXP_SWAP = 2, EXP_LANE_NEG = 4, EXP_NEG = 8 };

struct ExpTerm {           /* one term of a launch, in the sweep's tile coordinates (32 bytes) */
    uint32_t xh_t, xh_u;   /* partner unit = own unit ^ (xh_t | xh_u << EXP_TB) */
    uint32_t zt;           /* Z on the thread bits */
    uint32_t uword;        /* bit u: parity(u & Z on the unit bits) ^ parity(x_in & z_in) */
    uint32_t flags;        /* EXP_ODD: imaginary part (popc(x&z) odd); EXP_SWAP: f32 x on the pack lane;
                              EXP_LANE_NEG: f32 z on the pack lane; EXP_NEG: the value changes sign */
    uint32_t out;          /* position of the value in the caller's array */
    uint64_t zout;         /* Z outside the tile, unit-address bits */
};
static_assert(sizeof(ExpTerm) == 32, "ExpTerm is 32 bytes");

struct ExpArgs {
    const uint4 *A, *B;           /* own shard; partner shard (== A unless the sweep flips rank bits) */
    const ExpTerm *terms;
    double *partial;              /* [gridDim.x][K] */
    uint64_t toff[EXP_TB];        /* unit offset of thread bit i */
    uint64_t uoff[EXP_UB];        /* unit offset of unit bit b */
    uint64_t x_out;               /* partner tile = own tile ^ x_out (unit-address bits) */
    uint64_t n_work;              /* tiles visited */
    int8_t opos[64];              /* tile index bit i -> unit-address bit */
    int n_opos, K, same;          /* same: the partner tile is the tile itself (staged from the registers) */
};

/* ================================================================================================ device */

__device__ __forceinline__ uint32_t exp_sign(uint32_t w, int u) { return (w << (31 - u)) & 0x80000000u; }

template <bool ODD, bool SWAP>
__device__ __forceinline__ double exp_term_f32(const uint4 (&av)[EXP_NU], const uint4 *s_tile, uint32_t sbase, uint32_t w, float ls)
{
    double acc = 0.0;
#pragma unroll
    for (int r = 0; r < EXP_NU; r += EXP_RUN) {
        float run = 0.f;
#pragma unroll
        for (int u = r; u < r + EXP_RUN; u++) {
            const float4 b = *reinterpret_cast<const float4 *>(&s_tile[sbase ^ ((uint32_t)u << EXP_TB)]);
            const float4 x = *reinterpret_cast<const float4 *>(&av[u]);   /* re0 re1 im0 im1 */
            const float b0r = SWAP ? b.y : b.x, b1r = SWAP ? b.x : b.y, b0i = SWAP ? b.w : b.z, b1i = SWAP ? b.z : b.w;
            float p0, p1;
            if (ODD) { p0 = fmaf(x.x, b0i, -x.z * b0r); p1 = fmaf(x.y, b1i, -x.w * b1r); }
            else { p0 = fmaf(x.x, b0r, x.z * b0i); p1 = fmaf(x.y, b1r, x.w * b1i); }
            const float q = fmaf(ls, p1, p0);
            run += __uint_as_float(__float_as_uint(q) ^ exp_sign(w, u));
        }
        acc += (double)run;
    }
    return acc;
}

template <bool ODD>
__device__ __forceinline__ double exp_term_f64(const uint4 (&av)[EXP_NU], const uint4 *s_tile, uint32_t sbase, uint32_t w)
{
    double acc = 0.0;
#pragma unroll
    for (int u = 0; u < EXP_NU; u++) {
        const double2 b = *reinterpret_cast<const double2 *>(&s_tile[sbase ^ ((uint32_t)u << EXP_TB)]);
        const double2 x = *reinterpret_cast<const double2 *>(&av[u]);
        const double p = ODD ? fma(x.x, b.y, -x.y * b.x) : fma(x.x, b.x, x.y * b.y);
        acc += __hiloint2double(__double2hiint(p) ^ (int)exp_sign(w, u), __double2loint(p));
    }
    return acc;
}

template <bool F32>
__global__ void __launch_bounds__(EXP_THREADS, EXP_CTAS_PER_SM(F32)) k_expect(const __grid_constant__ ExpArgs a)
{
    extern __shared__ uint4 s_tile[];                                 /* EXP_TILE_UNITS, then [4 warps][K] fp64 */
    double *s_acc = reinterpret_cast<double *>(s_tile + EXP_TILE_UNITS);
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int j = tid; j < 4 * a.K; j += EXP_THREADS) s_acc[j] = 0.0;
    uint64_t toff = 0;
#pragma unroll
    for (int i = 0; i < EXP_TB; i++) if ((tid >> i) & 1) toff |= a.toff[i];
    uint4 av[EXP_NU];
    for (uint64_t t = blockIdx.x; t < a.n_work; t += gridDim.x) {
        uint64_t outer = 0;
        for (int i = 0; i < a.n_opos; i++) outer |= ((t >> i) & 1ULL) << a.opos[i];
        const uint64_t base = outer | toff;
        if (!a.same) {   /* partner tile straight into shared memory (no registers: the own tile holds 64 of them) */
            const uint64_t pbase = base ^ a.x_out;
#pragma unroll
            for (int u = 0; u < EXP_NU; u++) {
                uint64_t uo = 0;
#pragma unroll
                for (int b = 0; b < EXP_UB; b++) if ((u >> b) & 1) uo |= a.uoff[b];
                const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&s_tile[tid | ((uint32_t)u << EXP_TB)]);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(__cvta_generic_to_global(a.B + (pbase | uo))) : "memory");
            }
            asm volatile("cp.async.commit_group;\n" ::: "memory");
        }
#pragma unroll
        for (int u = 0; u < EXP_NU; u++) {
            uint64_t uo = 0;
#pragma unroll
            for (int b = 0; b < EXP_UB; b++) if ((u >> b) & 1) uo |= a.uoff[b];
            av[u] = __ldcs(a.A + (base | uo));
        }
        if (a.same) {
#pragma unroll
            for (int u = 0; u < EXP_NU; u++) s_tile[tid | ((uint32_t)u << EXP_TB)] = av[u];
        } else {
            asm volatile("cp.async.wait_all;\n" ::: "memory");
        }
        __syncthreads();
        const uint64_t pouter = outer ^ a.x_out;
        for (int j = 0; j < a.K; j++) {
            const ExpTerm T = a.terms[j];
            const uint32_t flip = ((__popc(tid & T.zt) ^ __popcll(pouter & T.zout)) & 1) ? 0xffffu : 0u;
            const uint32_t w = T.uword ^ flip;
            const uint32_t sbase = (tid ^ T.xh_t) | (T.xh_u << EXP_TB);
            double v;
            if (F32) {
                const float ls = (T.flags & EXP_LANE_NEG) ? -1.f : 1.f;
                switch (T.flags & (EXP_ODD | EXP_SWAP)) {
                case 0: v = exp_term_f32<false, false>(av, s_tile, sbase, w, ls); break;
                case EXP_ODD: v = exp_term_f32<true, false>(av, s_tile, sbase, w, ls); break;
                case EXP_SWAP: v = exp_term_f32<false, true>(av, s_tile, sbase, w, ls); break;
                default: v = exp_term_f32<true, true>(av, s_tile, sbase, w, ls); break;
                }
            } else {
                v = (T.flags & EXP_ODD) ? exp_term_f64<true>(av, s_tile, sbase, w) : exp_term_f64<false>(av, s_tile, sbase, w);
            }
#pragma unroll
            for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) s_acc[warp * a.K + j] += v;
        }
        __syncthreads();   /* the next tile overwrites s_tile */
    }
    __syncthreads();
    for (int j = tid; j < a.K; j += EXP_THREADS)
        a.partial[(size_t)blockIdx.x * a.K + j] = ((s_acc[j] + s_acc[a.K + j]) + s_acc[2 * a.K + j]) + s_acc[3 * a.K + j];
}

/* per term: the CTA partials in CTA order, times the pairing weight and the sign of i^{popc(x&z)} */
__global__ void k_expect_finish(const double *partial, int nblk, int K, const ExpTerm *terms, double weight, double *res)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= K) return;
    double acc = 0.0;
    for (int b = 0; b < nblk; b++) acc += partial[(size_t)b * K + j];
    acc *= weight;
    res[terms[j].out] = (terms[j].flags & EXP_NEG) ? 0.0 - acc : acc;   /* not -acc: a zero value stays +0.0 */
}

/* ================================================================================================ host */

int exp_geometry(int prec, const qsb_options_t *opt, int *T, int *L)
{
    *T = prec == QSB_F64 ? EXP_T_F64 : EXP_T_F32;
    int l = opt && opt->low_bits > 0 ? opt->low_bits : (prec == QSB_F64 ? 3 : 4);
    if (prec == QSB_F32 && l < 1) l = 1;   /* the pack lane is tile bit 0 */
    *L = std::min(l, *T);
    return QSB_OK;
}

int check_terms(int n, const uint64_t *x, const uint64_t *z, size_t nterms, const char *fn)
{
    if (nterms && (!x || !z)) { qsb_set_error("%s: null term array", fn); return QSB_ERR_ARG; }
    const uint64_t bad = n >= 64 ? 0 : ~((1ULL << n) - 1);
    for (size_t i = 0; i < nterms; i++)
        if ((x[i] | z[i]) & bad) {
            qsb_set_error("%s: term %zu has a qubit >= %d (x = 0x%llx, z = 0x%llx)", fn, i, n, (unsigned long long)x[i], (unsigned long long)z[i]);
            return QSB_ERR_ARG;
        }
    return QSB_OK;
}

void to_physical(int n, int nloc, const BitPerm &perm, const uint64_t *x, const uint64_t *z, size_t nterms, std::vector<PhysTerm> &out)
{
    out.resize(nterms);
    for (size_t i = 0; i < nterms; i++) {
        uint64_t px = 0, pz = 0;
        for (int q = 0; q < n; q++) {
            if ((x[i] >> q) & 1) px |= 1ULL << perm.pos[q];
            if ((z[i] >> q) & 1) pz |= 1ULL << perm.pos[q];
        }
        const uint64_t loc = (1ULL << nloc) - 1;
        out[i] = PhysTerm{px & loc, pz & loc, px >> nloc, pz >> nloc, __builtin_popcountll(x[i] & z[i]) & 3};
    }
}

uint32_t tile_coord(uint64_t m, const int8_t *pb, int T)
{
    uint32_t r = 0;
    for (int j = 0; j < T; j++) r |= (uint32_t)((m >> pb[j]) & 1) << j;
    return r;
}

static int ilog2i(int v) { int r = 0; while ((1 << r) < v) r++; return r; }

int pauli_dry_run_shape(int num_qubits, const qsb_options_t *opt_in, qsb_options_t *opt, int *nloc)
{
    if (num_qubits < 1 || num_qubits > 40) { qsb_set_error("num_qubits %d out of range 1..40", num_qubits); return QSB_ERR_ARG; }
    if (opt_in) *opt = *opt_in; else qsb_options_default(opt);
    if (opt->precision == 0) opt->precision = QSB_F32;
    if (opt->precision != QSB_F32 && opt->precision != QSB_F64) { qsb_set_error("precision must be 32 or 64"); return QSB_ERR_ARG; }
    if (opt->world_size <= 0) opt->world_size = 1;
    if (opt->world_size & (opt->world_size - 1)) { qsb_set_error("world_size must be a power of two"); return QSB_ERR_ARG; }
    const int g = ilog2i(opt->world_size), min_loc = tiled_min_local_bits(opt->precision, opt);
    if (g > 0 && num_qubits - g < min_loc + g) { qsb_set_error("%d qubits are too few to shard over %d ranks", num_qubits, opt->world_size); return QSB_ERR_ARG; }
    *nloc = std::max(num_qubits - g, min_loc);
    return QSB_OK;
}

/* Greedy cover of the distinct physical x masks by sweeps (host only, no CUDA).  Sweeps come grouped by xr,
 * xr == 0 first, so that each partner shard is fetched once. */
void exp_plan(int nloc, int T, int L, const std::vector<PhysTerm> &terms, std::vector<ExpSweep> &out)
{
    const uint64_t low = (1ULL << L) - 1, loc = nloc >= 64 ? ~0ULL : (1ULL << nloc) - 1;
    const int cap = T - L;
    std::map<uint64_t, std::map<uint64_t, std::vector<uint32_t>>> classes;   /* xr -> xl -> term indices */
    for (uint32_t i = 0; i < terms.size(); i++) classes[terms[i].xr][terms[i].xl].push_back(i);
    for (auto &cl : classes) {
        std::vector<uint64_t> masks;
        std::vector<const std::vector<uint32_t> *> lists;
        for (auto &m : cl.second) { masks.push_back(m.first); lists.push_back(&m.second); }
        std::vector<char> done(masks.size(), 0);
        size_t left = masks.size(), first = 0;
        while (left) {
            while (done[first]) first++;
            ExpSweep sw;
            sw.xr = cl.first;
            const uint64_t hi = masks[first] & ~low;
            uint64_t H = 0;
            for (uint64_t r = hi; r && __builtin_popcountll(H) < cap; r &= r - 1) H |= r & -r;
            uint64_t xout = hi & ~H;
            std::vector<size_t> members{first};
            done[first] = 1; left--;
            for (;;) {   /* take every mask that fits as is, then the one that needs the fewest new tile bits */
                size_t best = SIZE_MAX; int bestc = cap - __builtin_popcountll(H) + 1;
                for (size_t i = first; i < masks.size(); i++) {
                    if (done[i]) continue;
                    const int c = __builtin_popcountll((masks[i] & ~low & ~H) ^ xout);
                    if (c == 0) { done[i] = 1; left--; members.push_back(i); }
                    else if (c < bestc) { bestc = c; best = i; }
                }
                if (best == SIZE_MAX) break;
                H |= (masks[best] & ~low & ~H) ^ xout;
                xout &= ~H;
                done[best] = 1; left--; members.push_back(best);
            }
            /* fill the tile up to T bits: bits of x_out first (they become in-tile flips), then the lowest free bits */
            for (uint64_t r = xout; r && __builtin_popcountll(H) < cap; r &= r - 1) H |= r & -r;
            for (int b = L; b < nloc && __builtin_popcountll(H) < cap; b++) if (!((H >> b) & 1)) H |= 1ULL << b;
            xout &= ~H;
            sw.bmask = (low | H) & loc;
            sw.x_out = xout;
            int j = 0;
            for (int b = 0; b < nloc; b++) if ((sw.bmask >> b) & 1) sw.pb[j++] = (int8_t)b;
            std::sort(members.begin(), members.end());
            for (size_t i : members) sw.terms.insert(sw.terms.end(), lists[i]->begin(), lists[i]->end());
            out.push_back(std::move(sw));
        }
    }
}

uint32_t count_exchanges(const std::vector<ExpSweep> &sw)
{
    uint32_t n = 0; uint64_t last = 0;
    for (auto &s : sw) if (s.xr && s.xr != last) { n++; last = s.xr; }
    return n;
}

namespace {

uint32_t count_launches(const std::vector<ExpSweep> &sw)
{
    uint32_t n = 0;
    for (auto &s : sw) n += (uint32_t)((s.terms.size() + EXP_KMAX - 1) / EXP_KMAX);
    return n;
}

ExpTerm encode_term(const PhysTerm &p, const ExpSweep &sw, bool f32, uint32_t out_index)
{
    const int T = f32 ? EXP_T_F32 : EXP_T_F64, s = f32 ? 1 : 0;   /* s: unit-address shift (f32 units hold two amplitudes) */
    const uint32_t xin = tile_coord(p.xl, sw.pb, T), zin = tile_coord(p.zl, sw.pb, T);
    ExpTerm e; memset(&e, 0, sizeof e);
    e.xh_t = (xin >> s) & ((1u << EXP_TB) - 1);
    e.xh_u = (xin >> (s + EXP_TB)) & (EXP_NU - 1);
    e.zt = (zin >> s) & ((1u << EXP_TB) - 1);
    const uint32_t zu = (zin >> (s + EXP_TB)) & (EXP_NU - 1);
    const int c0 = __builtin_popcount(xin & zin) & 1;
    for (int u = 0; u < EXP_NU; u++) e.uword |= (uint32_t)((__builtin_popcount(u & zu) & 1) ^ c0) << u;
    e.flags = (p.y & 1 ? EXP_ODD : 0) | (p.y == 1 || p.y == 2 ? EXP_NEG : 0);
    if (f32) e.flags |= (xin & 1 ? EXP_SWAP : 0) | (zin & 1 ? EXP_LANE_NEG : 0);
    e.out = out_index;
    e.zout = (p.zl & ~sw.bmask) >> s;
    return e;
}

struct DevMem {   /* scoped device allocation */
    void *p = nullptr;
    ~DevMem() { if (p) cudaFree(p); }
};

}  // namespace

/* ------------------------------------------------------------------------------------------- C ABI */

extern "C" int qsb_pauli_from_string(const char *text, int num_qubits, uint64_t *x, uint64_t *z)
{
    if (!text || !x || !z) { qsb_set_error("qsb_pauli_from_string: null argument"); return QSB_ERR_ARG; }
    if (num_qubits < 1 || num_qubits > 64) { qsb_set_error("qsb_pauli_from_string: num_qubits %d out of range 1..64", num_qubits); return QSB_ERR_ARG; }
    uint64_t mx = 0, mz = 0, seen = 0;
    const char *p = text;
    for (;;) {
        while (*p == ' ' || *p == '\t' || *p == '\n' || *p == '\r') p++;
        if (!*p) break;
        const char c = *p++;
        if (c != 'I' && c != 'X' && c != 'Y' && c != 'Z') { qsb_set_error("Pauli string \"%s\": unknown letter '%c'", text, c); return QSB_ERR_PARSE; }
        if (*p < '0' || *p > '9') {
            if (c == 'I' && (*p == 0 || *p == ' ' || *p == '\t' || *p == '\n' || *p == '\r')) continue;   /* bare I: identity */
            qsb_set_error("Pauli string \"%s\": '%c' needs a qubit index", text, c); return QSB_ERR_PARSE;
        }
        long q = 0;
        while (*p >= '0' && *p <= '9') { if (q < 1000000) q = q * 10 + (*p - '0'); p++; }
        if (*p && *p != ' ' && *p != '\t' && *p != '\n' && *p != '\r') { qsb_set_error("Pauli string \"%s\": unexpected '%c' after qubit %ld", text, *p, q); return QSB_ERR_PARSE; }
        if (q >= num_qubits) { qsb_set_error("Pauli string \"%s\": qubit %ld >= %d", text, q, num_qubits); return QSB_ERR_ARG; }
        if ((seen >> q) & 1) { qsb_set_error("Pauli string \"%s\": qubit %ld appears twice", text, q); return QSB_ERR_PARSE; }
        seen |= 1ULL << q;
        if (c == 'X' || c == 'Y') mx |= 1ULL << q;
        if (c == 'Z' || c == 'Y') mz |= 1ULL << q;
    }
    *x = mx; *z = mz;
    return QSB_OK;
}

extern "C" int qsb_expectation_dry_run(int num_qubits, const qsb_options_t *opt_in, const uint64_t *x, const uint64_t *z,
                                       size_t nterms, uint32_t *sweeps, uint32_t *exchanges)
{
    qsb_options_t opt;
    int nloc;
    int rc = pauli_dry_run_shape(num_qubits, opt_in, &opt, &nloc);
    if (rc) return rc;
    rc = check_terms(num_qubits, x, z, nterms, "qsb_expectation_dry_run");
    if (rc) return rc;
    BitPerm id; for (int q = 0; q < 64; q++) id.pos[q] = (int8_t)q;
    int T, L;
    exp_geometry(opt.precision, &opt, &T, &L);
    std::vector<PhysTerm> pt;
    to_physical(num_qubits, nloc, id, x, z, nterms, pt);
    std::vector<ExpSweep> sw;
    exp_plan(nloc, T, L, pt, sw);
    if (sweeps) *sweeps = count_launches(sw);
    if (exchanges) *exchanges = count_exchanges(sw);
    return QSB_OK;
}

extern "C" int qsb_expectation_pauli(qsb_t *s, const uint64_t *x, const uint64_t *z, size_t nterms, double *out)
{
    if (!s) { qsb_set_error("qsb_expectation_pauli: null handle"); return QSB_ERR_ARG; }
    if (nterms == 0) return QSB_OK;
    if (!out) { qsb_set_error("qsb_expectation_pauli: null output"); return QSB_ERR_ARG; }
    int rc = check_terms(s->n, x, z, nterms, "qsb_expectation_pauli");
    if (rc) return rc;
    if (s->g && !s->comm) { qsb_set_error("qsb_expectation_pauli: sharded state needs qsb_comm_init first"); return QSB_ERR_COMM; }
    QSB_CUDA(cudaSetDevice(s->device));
    const bool f32 = s->prec == QSB_F32;
    int T, L;
    exp_geometry(s->prec, &s->opt, &T, &L);
    std::vector<PhysTerm> pt;
    to_physical(s->n, s->nloc, s->perm, x, z, nterms, pt);
    std::vector<ExpSweep> sw;
    exp_plan(s->nloc, T, L, pt, sw);

    /* one table for every launch, uploaded once */
    std::vector<ExpTerm> table;
    table.reserve(nterms);
    for (auto &w : sw) for (uint32_t i : w.terms) table.push_back(encode_term(pt[i], w, f32, i));

    int nsm = 0, occ = 0;
    QSB_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, s->device));
    const size_t smem_max = EXP_TILE_UNITS * 16 + 4 * EXP_KMAX * sizeof(double);
    if (f32) QSB_CUDA(cudaFuncSetAttribute(k_expect<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    else QSB_CUDA(cudaFuncSetAttribute(k_expect<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    const int grid_cap = nsm * 8;
    const size_t table_bytes = nterms * sizeof(ExpTerm), res_bytes = nterms * sizeof(double);
    const size_t all_bytes = s->g ? (size_t)s->world * res_bytes : 0, partial_bytes = (size_t)grid_cap * EXP_KMAX * sizeof(double);
    DevMem mem;
    QSB_CUDA(cudaMalloc(&mem.p, table_bytes + res_bytes + all_bytes + partial_bytes));
    ExpTerm *d_terms = (ExpTerm *)mem.p;
    double *d_res = (double *)((char *)mem.p + table_bytes);
    double *d_all = (double *)((char *)d_res + res_bytes);
    double *d_partial = (double *)((char *)d_all + all_bytes);
    QSB_CUDA(cudaMemcpyAsync(d_terms, table.data(), table_bytes, cudaMemcpyHostToDevice, s->stream));

    const int s_unit = f32 ? 1 : 0;
    const int nouter = s->nloc - T;
    uint64_t fetched = 0;   /* xr of the partner shard currently in state2 */
    size_t t0 = 0;
    for (auto &w : sw) {
        if (w.xr && w.xr != fetched) {
            rc = tiled_comm_sendrecv(s, s->state, s->state2, s->state_bytes, s->rank ^ (int)w.xr);
            if (rc) { cudaStreamSynchronize(s->stream); return rc; }
            fetched = w.xr;
        }
        ExpArgs a; memset(&a, 0, sizeof a);
        a.A = (const uint4 *)s->state;
        a.B = (const uint4 *)(w.xr ? s->state2 : s->state);
        const int first_t = f32 ? 1 : 0;
        for (int i = 0; i < EXP_TB; i++) a.toff[i] = (1ULL << w.pb[first_t + i]) >> s_unit;
        for (int b = 0; b < EXP_UB; b++) a.uoff[b] = (1ULL << w.pb[first_t + EXP_TB + b]) >> s_unit;
        a.x_out = w.x_out >> s_unit;
        const bool paired = !w.xr && w.x_out;   /* pair (t, t ^ x_out) visited once from the tile whose top x_out bit is 0 */
        const int skip = paired ? 63 - __builtin_clzll(w.x_out) : -1;
        for (int b = 0; b < s->nloc; b++)
            if (!((w.bmask >> b) & 1) && b != skip) a.opos[a.n_opos++] = (int8_t)(b - s_unit);
        a.n_work = 1ULL << (nouter - (paired ? 1 : 0));
        a.same = !w.xr && !w.x_out;
        for (size_t k0 = 0; k0 < w.terms.size(); k0 += EXP_KMAX) {
            const int K = (int)std::min<size_t>(EXP_KMAX, w.terms.size() - k0);
            const size_t smem = EXP_TILE_UNITS * 16 + 4 * (size_t)K * sizeof(double);
            if (f32) QSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_expect<true>, EXP_THREADS, smem));
            else QSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_expect<false>, EXP_THREADS, smem));
            const int grid = (int)std::min<uint64_t>(a.n_work, (uint64_t)std::min(grid_cap, nsm * std::max(occ, 1)));
            a.terms = d_terms + t0;
            a.partial = d_partial;
            a.K = K;
            if (f32) k_expect<true><<<grid, EXP_THREADS, smem, s->stream>>>(a);
            else k_expect<false><<<grid, EXP_THREADS, smem, s->stream>>>(a);
            k_expect_finish<<<(K + 127) / 128, 128, 0, s->stream>>>(d_partial, grid, K, d_terms + t0, paired ? 2.0 : 1.0, d_res);
            QSB_CUDA(cudaGetLastError());
            t0 += K;
        }
    }
    if (!s->g) {
        QSB_CUDA(cudaMemcpyAsync(out, d_res, res_bytes, cudaMemcpyDeviceToHost, s->stream));
        QSB_CUDA(cudaStreamSynchronize(s->stream));
        return QSB_OK;
    }
    /* every rank's values (the all-gather also orders this call before any later use of state2 by a peer) */
    rc = tiled_comm_allgather(s, d_res, d_all, res_bytes);
    if (rc) { cudaStreamSynchronize(s->stream); return rc; }
    std::vector<double> all((size_t)s->world * nterms);
    QSB_CUDA(cudaMemcpyAsync(all.data(), d_all, all_bytes, cudaMemcpyDeviceToHost, s->stream));
    QSB_CUDA(cudaStreamSynchronize(s->stream));
    for (size_t i = 0; i < nterms; i++) {
        double acc = 0.0;
        for (int r = 0; r < s->world; r++) {
            const double v = all[(size_t)r * nterms + i];
            acc += parity64(((uint64_t)r ^ pt[i].xr) & pt[i].zr) ? -v : v;
        }
        out[i] = acc;
    }
    return QSB_OK;
}
