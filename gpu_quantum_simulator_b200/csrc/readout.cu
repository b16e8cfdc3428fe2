/*
 * readout.cu -- what follows the apply path: cumulative distribution and measurement sampling on the
 * device, and raw shard dump / reload (SURVEY.md 8f-1, 8f-4).
 *
 * Reference functions replaced (all in /root/reference/):
 *   compute_state_cumulative_distribution   quantum_simulator.c:256-268 -> qsb_cdf      (2^n doubles out)
 *   measurement                             quantum_simulator.c:270-283 -> qsb_sample   (streaming, no 2^n array)
 * The reference builds the whole CDF on the host with one serial fp64 accumulator and then searches it
 * linearly per shot.  Here |a|^2, the prefix sums and the per-shot search all run on the GPU:
 *
 *   qsb_cdf     chunk of |a|^2 in logical order -> per-block totals -> serial offsets (one thread, <= 1024
 *               values) -> per-block scan.  Every value is  offset_b + (excl_t + run_i)  and every level's
 *               total is produced by exactly the arithmetic of its last element, so the result is monotone
 *               like the serial sum; it differs from the reference's single accumulator only by fp64
 *               re-association (<= 1e-12 in the parity tests).
 *   qsb_sample  never materialises the CDF: one sweep leaves the totals of 2^seg-amplitude segments, one
 *               small scan makes them cumulative, and each shot is one CTA that bisects the segment table
 *               and re-scans a single segment with the same arithmetic.  Rule of measurement(): the first
 *               index with cdf != 0 and cdf >= r, clamped to the last index (:277-281).  Works for any n
 *               that fits the device and for sharded states (per-rank totals all-gathered, exclusive scan
 *               over ranks on every rank, one all-reduce collects the shots).
 *
 * Sampling order: logical index order on one GPU (identical to bisecting qsb_cdf); on a sharded state the
 * physical order (rank-major, then the local address), which is the same distribution -- the drawn index
 * is mapped back to the logical index before it is returned.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "sim.h"
#include "tiled.h"

int tiled_comm_allgather(qsb_sim *s, const void *dsrc, void *ddst, size_t bytes);
int tiled_comm_allreduce_sum_u64(qsb_sim *s, void *dbuf, size_t count);

struct OrderArg { int8_t pos[64]; int n; };   /* order-index bit q -> local physical address bit pos[q] */

__device__ __forceinline__ uint64_t order_to_phys(uint64_t k, const OrderArg &P, int lo, int hi)
{
    uint64_t r = 0;
    for (int q = lo; q < hi; q++) r |= ((k >> q) & 1ULL) << P.pos[q];
    return r;
}

template <typename R>
__device__ __forceinline__ double prob_at(const R *st, uint64_t i)
{
    double r = (double)st[Lay<R>::re(i)], m = (double)st[Lay<R>::im(i)];
    return r * r + m * m;
}

/* ---------------------------------------------------------------------------------------------------
 * The one summation scheme every kernel below shares.  A CTA of 256 threads owns `len` consecutive
 * values; thread t owns the run [t*run, (t+1)*run).  run_total = serial sum of the run from zero;
 * excl[t] = serial sum of the run totals of the threads before t (thread 0 does it);
 * total = excl[255] + run_total[255].  Element i of thread t has the inclusive value excl[t] + (serial
 * sum of its run up to i), so the last element of the CTA equals `total` bit for bit.
 * ------------------------------------------------------------------------------------------------- */
#define RB 256

__device__ __forceinline__ double cta_exclusive(double run_total, double *s_excl, double *cta_total)
{
    __shared__ double s_tot[RB];
    s_tot[threadIdx.x] = run_total;
    __syncthreads();
    if (threadIdx.x == 0) {
        double acc = 0.0;
        for (int t = 0; t < RB; t++) { s_excl[t] = acc; acc += s_tot[t]; }
        s_excl[RB] = acc;
    }
    __syncthreads();
    *cta_total = s_excl[RB];
    return s_excl[threadIdx.x];
}

/* totals of the segments [seg << seg_log2, +2^seg_log2) of the order-index space */
template <typename R>
__global__ void __launch_bounds__(RB) k_segment_totals(const R *st, double *seg_total, uint64_t nseg, int seg_log2, OrderArg P)
{
    __shared__ double s_excl[RB + 1];
    const uint64_t S = 1ULL << seg_log2;
    const uint64_t run = S >= RB ? S / RB : 1;
    for (uint64_t seg = blockIdx.x; seg < nseg; seg += gridDim.x) {
        const uint64_t base_phys = order_to_phys(seg << seg_log2, P, seg_log2, P.n);
        double acc = 0.0;
        const uint64_t j0 = threadIdx.x * run;
        if (j0 < S)
            for (uint64_t j = j0; j < j0 + run; j++) acc += prob_at(st, base_phys | order_to_phys(j, P, 0, seg_log2));
        double total;
        (void)cta_exclusive(acc, s_excl, &total);
        if (threadIdx.x == 0) seg_total[seg] = total;
        __syncthreads();
    }
}

/* seg_total[] -> inclusive cumulative values in place: 1024 threads, each a contiguous run of segments;
 * thread 0 chains the run totals.  incl[j] = run_ex[t] + (prev[j] + total[j]) with prev[j] = serial sum of
 * the run before j; prev[] and run_ex[] are kept so that k_draw can rebuild any value with the very same
 * additions.  *grand = the last value. */
__global__ void __launch_bounds__(1024) k_segment_scan(double *seg, double *prev, double *run_ex, uint64_t nseg, double *grand)
{
    __shared__ double s_tot[1024];
    __shared__ double s_excl[1025];
    const uint64_t run = (nseg + 1023) / 1024;
    const uint64_t j0 = threadIdx.x * run, j1 = j0 + run < nseg ? j0 + run : nseg;
    double acc = 0.0;
    for (uint64_t j = j0; j < j1; j++) acc += seg[j];
    s_tot[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0;
        for (int t = 0; t < 1024; t++) { s_excl[t] = a; a += s_tot[t]; }
        s_excl[1024] = a;
        *grand = a;
    }
    __syncthreads();
    const double ex = s_excl[threadIdx.x];
    run_ex[threadIdx.x] = ex;
    acc = 0.0;
    for (uint64_t j = j0; j < j1; j++) { prev[j] = acc; acc += seg[j]; seg[j] = ex + acc; }
}

__device__ __forceinline__ bool reaches(double c, double r) { return c != 0.0 && c >= r; }   /* quantum_simulator.c:279 */

/* One CTA per shot.  rank_base = cumulative total of the ranks before this one; shots whose owner is another
 * rank are left untouched (the host zeroed them).  out[k] = rank-global physical/order index. */
template <typename R>
__global__ void __launch_bounds__(RB) k_draw(const R *st, const double *seg_incl, const double *seg_prev, const double *run_ex,
                                              uint64_t nseg, int seg_log2, OrderArg P,
                                              const double *rnd, const int *owner, int my_rank, double rank_base,
                                              uint64_t rank_index_base, unsigned long long *out)
{
    __shared__ double s_excl[RB + 1];
    __shared__ unsigned long long s_first;
    __shared__ uint64_t s_seg;
    const int k = blockIdx.x;
    if (owner[k] != my_rank) return;
    const double r = rnd[k];
    const uint64_t S = 1ULL << seg_log2;
    if (threadIdx.x == 0) {
        /* first segment whose cumulative value reaches r (monotone table -> bisection) */
        uint64_t lo = 0, hi = nseg - 1;
        while (lo < hi) { uint64_t mid = (lo + hi) >> 1; if (reaches(rank_base + seg_incl[mid], r)) hi = mid; else lo = mid + 1; }
        s_seg = lo;
        s_first = ~0ULL;
    }
    __syncthreads();
    const uint64_t seg = s_seg;
    /* value of element i of this segment = rank_base + (ex_run + (prev + (ex + run_i))): the additions of the table */
    const double ex_run = run_ex[seg / ((nseg + 1023) / 1024)], seg_prev_v = seg_prev[seg];
    const uint64_t base_phys = order_to_phys(seg << seg_log2, P, seg_log2, P.n);
    const uint64_t run = S >= RB ? S / RB : 1;
    const uint64_t j0 = threadIdx.x * run;
    double acc = 0.0;
    if (j0 < S)
        for (uint64_t j = j0; j < j0 + run; j++) acc += prob_at(st, base_phys | order_to_phys(j, P, 0, seg_log2));
    double total;
    const double ex = cta_exclusive(acc, s_excl, &total);
    /* the run that contains the crossing: its end reaches r, its start does not */
    if (j0 < S && reaches(rank_base + (ex_run + (seg_prev_v + (ex + acc))), r) && !(threadIdx.x && reaches(rank_base + (ex_run + (seg_prev_v + ex)), r))) {
        acc = 0.0;
        for (uint64_t j = j0; j < j0 + run; j++) {
            acc += prob_at(st, base_phys | order_to_phys(j, P, 0, seg_log2));
            if (reaches(rank_base + (ex_run + (seg_prev_v + (ex + acc))), r)) { atomicMin(&s_first, (unsigned long long)j); break; }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint64_t j = s_first == ~0ULL ? S - 1 : (uint64_t)s_first;   /* r beyond the total: last index (:278) */
        out[k] = rank_index_base + ((seg << seg_log2) | j);
    }
}

/* ---- CDF to the host: chunk kernels ---------------------------------------------------------------------- */
#define CB 4096   /* values per CTA */

__global__ void __launch_bounds__(RB) k_chunk_totals(const double *p, uint64_t count, double *blk_total)
{
    __shared__ double s_excl[RB + 1];
    const uint64_t b0 = (uint64_t)blockIdx.x * CB;
    const uint64_t j0 = b0 + threadIdx.x * (CB / RB);
    double acc = 0.0;
    for (uint64_t j = j0; j < j0 + CB / RB && j < count; j++) acc += p[j];
    double total;
    (void)cta_exclusive(acc, s_excl, &total);
    if (threadIdx.x == 0) blk_total[blockIdx.x] = total;
}

/* blk_total[] -> exclusive offsets in place, chained serially from *carry; *carry advances by the chunk's total */
__global__ void k_chunk_offsets(double *blk, int nblk, double *carry)
{
    if (threadIdx.x || blockIdx.x) return;
    double acc = *carry;
    for (int b = 0; b < nblk; b++) { double t = blk[b]; blk[b] = acc; acc += t; }
    *carry = acc;
}

__global__ void __launch_bounds__(RB) k_chunk_scan(double *p, uint64_t count, const double *blk_off)
{
    __shared__ double s_excl[RB + 1];
    const uint64_t b0 = (uint64_t)blockIdx.x * CB;
    const uint64_t j0 = b0 + threadIdx.x * (CB / RB);
    double v[CB / RB];
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < CB / RB; i++) { v[i] = j0 + i < count ? p[j0 + i] : 0.0; acc += v[i]; }
    double total;
    const double ex = cta_exclusive(acc, s_excl, &total);
    const double off = blk_off[blockIdx.x];
    acc = 0.0;
#pragma unroll
    for (int i = 0; i < CB / RB; i++) { acc += v[i]; if (j0 + i < count) p[j0 + i] = off + (ex + acc); }
}

template <typename R>
__global__ void k_probs_order(const R *st, double *out, uint64_t first, uint64_t count, OrderArg P)
{
    uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    out[k] = prob_at(st, order_to_phys(first + k, P, 0, P.n));
}

/* ================================================================================================ host */

/* order index -> local address: the logical order when the state is on one GPU, the physical order otherwise */
static OrderArg order_arg(const qsb_sim *s, int *bits)
{
    OrderArg P; memset(&P, 0, sizeof P);
    if (s->g == 0) { P.n = s->n; for (int q = 0; q < s->n; q++) P.pos[q] = s->perm.pos[q]; }
    else { P.n = s->nloc; for (int q = 0; q < s->nloc; q++) P.pos[q] = (int8_t)q; }
    *bits = P.n;
    return P;
}

/* Chunks sit at fixed multiples of `chunk` in the logical index space, so every value is produced by the same
 * additions whatever (first, count) asks for: cdf(first, count) is cdf(0, 2^n)[first, first + count) bit for bit.
 * Chunks wholly below `first` only advance the carry (|a|^2, block totals, offsets; no scan, no copy). */
extern "C" int qsb_cdf(qsb_t *s, double *cdf, uint64_t first, uint64_t count)
{
    if (!s || (!cdf && count)) { qsb_set_error("qsb_cdf: null argument"); return QSB_ERR_ARG; }
    const uint64_t total = 1ULL << s->n;
    if (first > total || count > total - first) { qsb_set_error("range [%llu, +%llu) exceeds 2^%d amplitudes", (unsigned long long)first, (unsigned long long)count, s->n); return QSB_ERR_ARG; }
    if (s->g) {
        qsb_set_error("qsb_cdf: the state is sharded over %d ranks and the prefix sum below this rank's indices lives on the others; "
                      "draw shots with qsb_sample, which works on sharded states", s->world);
        return QSB_ERR_ARG;
    }
    if (count == 0) return QSB_OK;
    QSB_CUDA(cudaSetDevice(s->device));
    int bits = 0;
    const OrderArg P = order_arg(s, &bits);   /* one GPU: order = logical index */
    const uint64_t chunk = std::min<uint64_t>(s->staging_bytes / 8, (uint64_t)CB * 1024);   /* <= 1024 CTA totals per chunk */
    double *d_p = (double *)s->staging;
    double *d_blk = (double *)((char *)s->d_scratch + 131072);        /* 1024 doubles */
    double *d_carry = (double *)((char *)s->d_scratch + 131072 + 8192);
    QSB_CUDA(cudaMemsetAsync(d_carry, 0, sizeof(double), s->stream));
    const uint64_t end = first + count;
    for (uint64_t c0 = 0; c0 < end; c0 += chunk) {
        const uint64_t c = std::min(chunk, end - c0);
        const unsigned nblk = (unsigned)((c + CB - 1) / CB);
        if (s->prec == QSB_F32) k_probs_order<float><<<(unsigned)((c + 255) / 256), 256, 0, s->stream>>>((const float *)s->state, d_p, c0, c, P);
        else k_probs_order<double><<<(unsigned)((c + 255) / 256), 256, 0, s->stream>>>((const double *)s->state, d_p, c0, c, P);
        k_chunk_totals<<<nblk, RB, 0, s->stream>>>(d_p, c, d_blk);
        k_chunk_offsets<<<1, 32, 0, s->stream>>>(d_blk, (int)nblk, d_carry);
        QSB_CUDA(cudaGetLastError());
        if (c0 + c <= first) continue;
        k_chunk_scan<<<nblk, RB, 0, s->stream>>>(d_p, c, d_blk);
        QSB_CUDA(cudaGetLastError());
        const uint64_t skip = first > c0 ? first - c0 : 0;
        QSB_CUDA(cudaMemcpyAsync(cdf + (c0 + skip - first), d_p + skip, (c - skip) * 8, cudaMemcpyDeviceToHost, s->stream));
        QSB_CUDA(cudaStreamSynchronize(s->stream));
    }
    return QSB_OK;
}

static inline uint64_t splitmix64(uint64_t *x)
{
    uint64_t z = (*x += 0x9E3779B97F4A7C15ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

extern "C" double qsb_sample_uniform(uint64_t seed, int k)
{
    uint64_t st = seed, z = 0;
    for (int i = 0; i <= k; i++) z = splitmix64(&st);
    return (double)(z >> 11) * (1.0 / 9007199254740992.0);
}

struct DevBuf {   /* scoped device allocation */
    void *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
};

extern "C" int qsb_sample(qsb_t *s, uint64_t seed, int shots, uint64_t *out)
{
    if (!s || shots < 0 || (shots && !out)) { qsb_set_error("qsb_sample: bad argument"); return QSB_ERR_ARG; }
    if (shots == 0) return QSB_OK;
    if (s->g && !s->comm) { qsb_set_error("qsb_sample: sharded state needs qsb_comm_init first"); return QSB_ERR_COMM; }
    QSB_CUDA(cudaSetDevice(s->device));
    int bits = 0;
    const OrderArg P = order_arg(s, &bits);
    const int seg_log2 = std::min(bits, std::max(12, bits - 20));
    const uint64_t nseg = 1ULL << (bits - seg_log2);
    if (nseg * 16 + 8192 > s->staging_bytes) { qsb_set_error("qsb_sample: segment table does not fit the staging buffer"); return QSB_ERR_NOMEM; }
    double *d_seg = (double *)s->staging, *d_prev = d_seg + nseg, *d_runex = d_prev + nseg;
    double *d_grand = (double *)((char *)s->d_scratch + 131072 + 8192 + 64);
    double *d_all = d_grand + 8;                                      /* world doubles */
    const unsigned grid = (unsigned)std::min<uint64_t>(nseg, 148ULL * 8);
    if (s->prec == QSB_F32) k_segment_totals<float><<<grid, RB, 0, s->stream>>>((const float *)s->state, d_seg, nseg, seg_log2, P);
    else k_segment_totals<double><<<grid, RB, 0, s->stream>>>((const double *)s->state, d_seg, nseg, seg_log2, P);
    k_segment_scan<<<1, 1024, 0, s->stream>>>(d_seg, d_prev, d_runex, nseg, d_grand);
    QSB_CUDA(cudaGetLastError());

    /* totals of every rank, in rank order, identical on every rank */
    std::vector<double> rank_total(s->world, 0.0);
    if (s->g) {
        int rc = tiled_comm_allgather(s, d_grand, d_all, sizeof(double));
        if (rc) return rc;
        QSB_CUDA(cudaMemcpyAsync(rank_total.data(), d_all, sizeof(double) * s->world, cudaMemcpyDeviceToHost, s->stream));
    } else {
        QSB_CUDA(cudaMemcpyAsync(rank_total.data(), d_grand, sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    }
    QSB_CUDA(cudaStreamSynchronize(s->stream));
    std::vector<double> rank_base(s->world + 1, 0.0);
    for (int r = 0; r < s->world; r++) rank_base[r + 1] = rank_base[r] + rank_total[r];

    /* the draws (same stream of numbers on every rank) and the rank each one falls on */
    std::vector<double> rnd(shots);
    std::vector<int> owner(shots);
    uint64_t st = seed;
    for (int k = 0; k < shots; k++) {
        const double r = (double)(splitmix64(&st) >> 11) * (1.0 / 9007199254740992.0);
        rnd[k] = r;
        int o = s->world - 1;
        for (int q = 0; q < s->world; q++) if (rank_base[q + 1] != 0.0 && rank_base[q + 1] >= r) { o = q; break; }
        owner[k] = o;
    }
    DevBuf d_rnd, d_owner, d_out;
    QSB_CUDA(cudaMalloc(&d_rnd.p, sizeof(double) * shots));
    QSB_CUDA(cudaMalloc(&d_owner.p, sizeof(int) * shots));
    QSB_CUDA(cudaMalloc(&d_out.p, sizeof(uint64_t) * shots));
    QSB_CUDA(cudaMemcpyAsync(d_rnd.p, rnd.data(), sizeof(double) * shots, cudaMemcpyHostToDevice, s->stream));
    QSB_CUDA(cudaMemcpyAsync(d_owner.p, owner.data(), sizeof(int) * shots, cudaMemcpyHostToDevice, s->stream));
    QSB_CUDA(cudaMemsetAsync(d_out.p, 0, sizeof(uint64_t) * shots, s->stream));
    const uint64_t index_base = (uint64_t)s->rank << s->nloc;
    for (int k0 = 0; k0 < shots; k0 += 65535) {
        const int c = std::min(65535, shots - k0);
        if (s->prec == QSB_F32)
            k_draw<float><<<c, RB, 0, s->stream>>>((const float *)s->state, d_seg, d_prev, d_runex, nseg, seg_log2, P, (const double *)d_rnd.p + k0, (const int *)d_owner.p + k0,
                                                   s->rank, rank_base[s->rank], index_base, (unsigned long long *)d_out.p + k0);
        else
            k_draw<double><<<c, RB, 0, s->stream>>>((const double *)s->state, d_seg, d_prev, d_runex, nseg, seg_log2, P, (const double *)d_rnd.p + k0, (const int *)d_owner.p + k0,
                                                    s->rank, rank_base[s->rank], index_base, (unsigned long long *)d_out.p + k0);
    }
    QSB_CUDA(cudaGetLastError());
    if (s->g) {
        int rc = tiled_comm_allreduce_sum_u64(s, d_out.p, (size_t)shots);
        if (rc) return rc;
    }
    QSB_CUDA(cudaMemcpyAsync(out, d_out.p, sizeof(uint64_t) * shots, cudaMemcpyDeviceToHost, s->stream));
    QSB_CUDA(cudaStreamSynchronize(s->stream));
    if (s->g) {   /* physical global index -> logical index */
        for (int k = 0; k < shots; k++) {
            uint64_t L = 0;
            for (int q = 0; q < s->n; q++) L |= ((out[k] >> s->perm.pos[q]) & 1ULL) << q;
            out[k] = L;
        }
    }
    return QSB_OK;
}

/* ---- shard dump / reload (SURVEY.md 8f-4) ------------------------------------------------------------------
 * File = 128-byte header + the shard exactly as it lies in HBM (device dtype, physical order, layout of
 * common.cuh).  The header carries the logical -> physical qubit map, so a reloaded shard continues with
 * any circuit.  One file per rank. */
struct ShardHeader {
    char magic[8];        /* "QSBSHARD" */
    uint32_t version, num_qubits, precision, world, rank, nloc;
    int8_t perm[64];
    uint8_t pad[32];
};
static_assert(sizeof(ShardHeader) == 128, "shard header is 128 bytes");

extern "C" int qsb_save_state(qsb_t *s, const char *path)
{
    if (!s || !path) { qsb_set_error("qsb_save_state: null argument"); return QSB_ERR_ARG; }
    QSB_CUDA(cudaSetDevice(s->device));
    FILE *f = fopen(path, "wb");
    if (!f) { qsb_set_error("ERROR: cannot open state file %s", path); return QSB_ERR_IO; }
    ShardHeader h; memset(&h, 0, sizeof h);
    memcpy(h.magic, "QSBSHARD", 8);
    h.version = 1; h.num_qubits = (uint32_t)s->n; h.precision = (uint32_t)s->prec; h.world = (uint32_t)s->world;
    h.rank = (uint32_t)s->rank; h.nloc = (uint32_t)s->nloc;
    memcpy(h.perm, s->perm.pos, 64);
    bool ok = fwrite(&h, sizeof h, 1, f) == 1;
    const size_t chunk = (size_t)32 << 20;
    void *host = nullptr;
    if (cudaMallocHost(&host, chunk) != cudaSuccess) { (void)cudaGetLastError(); fclose(f); qsb_set_error("Malloc error: pinned staging"); return QSB_ERR_NOMEM; }
    for (size_t off = 0; ok && off < s->state_bytes; off += chunk) {
        const size_t c = std::min(chunk, s->state_bytes - off);
        if (cudaMemcpyAsync(host, (const char *)s->state + off, c, cudaMemcpyDeviceToHost, s->stream) != cudaSuccess ||
            cudaStreamSynchronize(s->stream) != cudaSuccess) { ok = false; qsb_set_error("%s while reading the shard", cudaGetErrorString(cudaGetLastError())); cudaFreeHost(host); fclose(f); return QSB_ERR_CUDA; }
        ok = fwrite(host, 1, c, f) == c;
    }
    cudaFreeHost(host);
    if (fclose(f) != 0) ok = false;
    if (!ok) { qsb_set_error("ERROR: short write to state file %s", path); return QSB_ERR_IO; }
    return QSB_OK;
}

extern "C" int qsb_load_state(qsb_t *s, const char *path)
{
    if (!s || !path) { qsb_set_error("qsb_load_state: null argument"); return QSB_ERR_ARG; }
    QSB_CUDA(cudaSetDevice(s->device));
    FILE *f = fopen(path, "rb");
    if (!f) { qsb_set_error("ERROR: cannot open state file %s", path); return QSB_ERR_IO; }
    ShardHeader h;
    if (fread(&h, sizeof h, 1, f) != 1 || memcmp(h.magic, "QSBSHARD", 8) != 0 || h.version != 1) {
        fclose(f); qsb_set_error("%s is not a shard file", path); return QSB_ERR_PARSE;
    }
    if ((int)h.num_qubits != s->n || (int)h.precision != s->prec || (int)h.world != s->world || (int)h.rank != s->rank || (int)h.nloc != s->nloc) {
        fclose(f);
        qsb_set_error("shard file is for %u qubits f%u rank %u/%u, the handle is %d qubits f%d rank %d/%d",
                      h.num_qubits, h.precision, h.rank, h.world, s->n, s->prec, s->rank, s->world);
        return QSB_ERR_ARG;
    }
    /* the qubit map must be a permutation of the physical bits */
    uint64_t seen = 0;
    for (int q = 0; q < s->n; q++) {
        const int p = h.perm[q];
        if (p < 0 || p >= s->nphys || ((seen >> p) & 1)) { fclose(f); qsb_set_error("shard file has a corrupt qubit map"); return QSB_ERR_PARSE; }
        seen |= 1ULL << p;
    }
    const size_t chunk = (size_t)32 << 20;
    void *host = nullptr;
    if (cudaMallocHost(&host, chunk) != cudaSuccess) { (void)cudaGetLastError(); fclose(f); qsb_set_error("Malloc error: pinned staging"); return QSB_ERR_NOMEM; }
    for (size_t off = 0; off < s->state_bytes; off += chunk) {
        const size_t c = std::min(chunk, s->state_bytes - off);
        if (fread(host, 1, c, f) != c) { cudaFreeHost(host); fclose(f); qsb_set_error("shard file %s is truncated", path); return QSB_ERR_IO; }
        if (cudaMemcpyAsync((char *)s->state + off, host, c, cudaMemcpyHostToDevice, s->stream) != cudaSuccess ||
            cudaStreamSynchronize(s->stream) != cudaSuccess) { qsb_set_error("%s while writing the shard", cudaGetErrorString(cudaGetLastError())); cudaFreeHost(host); fclose(f); return QSB_ERR_CUDA; }
    }
    cudaFreeHost(host);
    fclose(f);
    memcpy(s->perm.pos, h.perm, 64);
    return QSB_OK;
}
