/*
 * tiled_exec.cu -- execution of a TiledPlan: one kernel launch per pass on the
 * handle's stream.  Pass descriptors travel as kernel parameters, so the timed
 * region contains nothing but the pass kernels and, when the state is sharded
 * over several GPUs, the global<->local qubit exchanges.
 *
 * Exchange (the reference has no multi-GPU path, SURVEY.md F11): the state is
 * sharded on the top g = log2(P) physical index bits, one process per GPU.  An
 * exchange swaps those rank bits with the top g LOCAL bits: the local buffer is
 * P contiguous chunks, chunk j goes to rank j and the chunk received from rank
 * j lands at position j of the second buffer -- an all-to-all of contiguous
 * chunks over NVLink, issued as one NCCL group of send/recv pairs.  NCCL is
 * loaded at run time (dlopen) so the library has no link-time dependency on it.
 */
#include <dlfcn.h>
#include <stdio.h>
#include <algorithm>
#include <utility>
#include <string.h>

#include "sim.h"
#include "tiled.h"

int tiled_launch_pass(qsb_sim *s, const TiledPlan *p, size_t k, const void *src, void *dst, const PeerTab *peers, uint64_t tile0, uint64_t ntile);

int tiled_plan_build(int n, int prec, int g, int nloc, int rank, const qsb_options_t *opt, const BitPerm &start,
                     const std::vector<COp> &cops, const double gphase[2], bool /*with_device*/,
                     TiledPlan **out, qsb_run_stats_t *stats)
{
    TiledPlan *p = nullptr;
    int rc = tiled_plan_search(n, prec, g, nloc, rank, opt, start, cops, gphase, &p);   /* tiled_plan.cpp: plans the candidates, keeps the cheapest */
    if (rc) return rc;
    uint64_t n_ops = 0, n_rounds = 0, sweeps = 0, swaps = 0;
    for (auto &hp : p->passes) {
        if (hp.is_swap) { swaps++; continue; }
        if (hp.fused_swap) swaps++;
        sweeps++; n_ops += hp.ops.size(); n_rounds += hp.rounds.size();
    }
    const uint64_t local_bytes = ((uint64_t)1 << nloc) * amp_bytes(prec);
    stats->device_ops = n_ops;
    stats->passes = (uint32_t)sweeps;
    stats->rounds = (uint32_t)n_rounds;
    stats->kernel_launches = (uint32_t)sweeps;
    stats->bytes_moved = sweeps * 2ULL * local_bytes;
    stats->swaps = (uint32_t)swaps;
    stats->bytes_exchanged = swaps * (local_bytes - (local_bytes >> g));
    *out = p;
    return QSB_OK;
}

void tiled_plan_free(TiledPlan *p) { delete p; }
void tiled_plan_end_perm(const TiledPlan *p, BitPerm *out) { *out = p->end_perm; }
bool tiled_plan_starts_at(const TiledPlan *p, const BitPerm &perm)
{
    for (int q = 0; q < p->n; q++) if (p->start_perm.pos[q] != perm.pos[q]) return false;
    return true;
}
double tiled_last_exchange_ms(const TiledPlan *p) { return p ? p->last_exchange_ms : 0.0; }

/* ------------------------------------------------------------------ NCCL (dlopen) */
typedef struct { char internal[128]; } qsb_nccl_id_t;
typedef void *qsb_nccl_comm_t;
struct NcclApi {
    void *lib = nullptr;
    int (*GetUniqueId)(qsb_nccl_id_t *) = nullptr;
    int (*CommInitRank)(qsb_nccl_comm_t *, int, qsb_nccl_id_t, int) = nullptr;
    int (*CommDestroy)(qsb_nccl_comm_t) = nullptr;
    int (*Send)(const void *, size_t, int, int, qsb_nccl_comm_t, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, qsb_nccl_comm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, qsb_nccl_comm_t, cudaStream_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, qsb_nccl_comm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;

static int nccl_load()
{
    if (g_nccl.lib) return QSB_OK;
    const char *names[] = {"libnccl.so.2", "libnccl.so", nullptr};
    void *h = nullptr;
    for (int i = 0; names[i] && !h; i++) h = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
    if (!h) { qsb_set_error("cannot load NCCL (libnccl.so.2): %s", dlerror()); return QSB_ERR_COMM; }
#define SYM(field, name) *(void **)(&g_nccl.field) = dlsym(h, name); if (!g_nccl.field) { qsb_set_error("NCCL symbol %s missing", name); return QSB_ERR_COMM; }
    SYM(GetUniqueId, "ncclGetUniqueId") SYM(CommInitRank, "ncclCommInitRank") SYM(CommDestroy, "ncclCommDestroy")
    SYM(Send, "ncclSend") SYM(Recv, "ncclRecv") SYM(GroupStart, "ncclGroupStart") SYM(GroupEnd, "ncclGroupEnd")
    SYM(GetErrorString, "ncclGetErrorString") SYM(AllGather, "ncclAllGather") SYM(AllReduce, "ncclAllReduce")
#undef SYM
    g_nccl.lib = h;
    return QSB_OK;
}
#define QSB_NCCL(call) do { int r_ = (call); if (r_ != 0) { qsb_set_error("NCCL: %s in %s at line %d", g_nccl.GetErrorString(r_), __FILE__, __LINE__); return QSB_ERR_COMM; } } while (0)

extern "C" int qsb_comm_unique_id(void *id128)
{
    if (!id128) { qsb_set_error("qsb_comm_unique_id: null argument"); return QSB_ERR_ARG; }
    int rc = nccl_load();
    if (rc) return rc;
    qsb_nccl_id_t id;
    QSB_NCCL(g_nccl.GetUniqueId(&id));
    memcpy(id128, &id, 128);
    return QSB_OK;
}

extern "C" int qsb_comm_init(qsb_t *s, const void *id128)
{
    if (!s || !id128) { qsb_set_error("qsb_comm_init: null argument"); return QSB_ERR_ARG; }
    if (s->world == 1) return QSB_OK;
    int rc = nccl_load();
    if (rc) return rc;
    QSB_CUDA(cudaSetDevice(s->device));
    qsb_nccl_id_t id; memcpy(&id, id128, 128);
    qsb_nccl_comm_t c = nullptr;
    QSB_NCCL(g_nccl.CommInitRank(&c, s->world, id, s->rank));
    s->comm = c;
    if (!s->state2) {
        cudaError_t e = cudaMalloc(&s->state2, s->state_bytes);
        if (e != cudaSuccess) { qsb_set_error("Malloc error: exchange buffer of %zu bytes (%s)", s->state_bytes, cudaGetErrorString(e)); (void)cudaGetLastError(); return QSB_ERR_NOMEM; }
    }
    /* Map every peer's two shard buffers (CUDA IPC over NVLink peer access): the fused-exchange passes store
     * straight into them.  If the mapping is not possible the planner keeps the NCCL all-to-all. */
    s->peers_ok = false;
    if (s->world <= QSB_MAX_PEERS && !(s->opt.reserved[5] == 2)) {
        struct Handles { cudaIpcMemHandle_t a, b; };
        Handles mine; memset(&mine, 0, sizeof mine);
        bool ok = cudaIpcGetMemHandle(&mine.a, s->state) == cudaSuccess && cudaIpcGetMemHandle(&mine.b, s->state2) == cudaSuccess;
        (void)cudaGetLastError();
        char *dbuf = (char *)s->d_scratch;                       /* 1 MiB scratch: [mine | all] */
        std::vector<Handles> all(s->world);
        QSB_CUDA(cudaMemcpyAsync(dbuf, &mine, sizeof mine, cudaMemcpyHostToDevice, s->stream));
        QSB_NCCL(g_nccl.AllGather(dbuf, dbuf + 4096, sizeof mine, 1 /* ncclUint8 */, c, s->stream));
        QSB_CUDA(cudaMemcpyAsync(all.data(), dbuf + 4096, sizeof(Handles) * s->world, cudaMemcpyDeviceToHost, s->stream));
        QSB_CUDA(cudaStreamSynchronize(s->stream));
        for (int r = 0; r < s->world && ok; r++) {
            if (r == s->rank) { s->peer_state[r] = s->state; s->peer_state2[r] = s->state2; continue; }
            if (cudaIpcOpenMemHandle(&s->peer_state[r], all[r].a, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
                cudaIpcOpenMemHandle(&s->peer_state2[r], all[r].b, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) ok = false;
        }
        (void)cudaGetLastError();
        /* every rank must take the same decision: the plans have to agree on where the exchanges are */
        int *flag = (int *)(dbuf + 65536);
        const int mine_ok = ok ? 1 : 0; int all_ok = 0;
        QSB_CUDA(cudaMemcpyAsync(flag, &mine_ok, sizeof(int), cudaMemcpyHostToDevice, s->stream));
        QSB_NCCL(g_nccl.AllReduce(flag, flag + 1, 1, 2 /* ncclInt32 */, 3 /* ncclMin */, c, s->stream));
        QSB_CUDA(cudaMemcpyAsync(&all_ok, flag + 1, sizeof(int), cudaMemcpyDeviceToHost, s->stream));
        QSB_CUDA(cudaStreamSynchronize(s->stream));
        s->peers_ok = all_ok == 1;
        if (!s->peers_ok) {   /* some rank could not map its peers: drop the mappings made here */
            for (int r = 0; r < s->world; r++) if (r != s->rank) {
                if (s->peer_state[r]) cudaIpcCloseMemHandle(s->peer_state[r]);
                if (s->peer_state2[r]) cudaIpcCloseMemHandle(s->peer_state2[r]);
                s->peer_state[r] = s->peer_state2[r] = nullptr;
            }
            (void)cudaGetLastError();
        }
    }
    /* exchange flavour of the plans made from now on: 1 = fused peer scatter (direct: the victims trade places with the
     * rank bits wherever they are), 4 = the round-1 fused flavour (victims moved to the top local positions first),
     * 3 = pipelined copy-engine exchange, 2 = plain NCCL all-to-all (also the fallback when the peer shards cannot be
     * mapped).  Measured on 34 q (DESIGN.md section 6): round 1 preferred the pipelined exchange with one peer
     * (2 GPUs: 1585 vs 1640 ms); the direct fused exchange needs no extra pass and wins there too (round 2, same box:
     * 1275 ms vs 1355 pipelined vs 1347 round-1 fused), so it is the default at every world size. */
    if (s->peers_ok && s->opt.reserved[5] == 0) s->opt.reserved[5] = 1;
    if (!s->peers_ok) s->opt.reserved[5] = 2;
    return QSB_OK;
}

/* small collectives for the readout (readout.cu): buffers are device pointers, the calls are ordered on s->stream */
int tiled_comm_allgather(qsb_sim *s, const void *dsrc, void *ddst, size_t bytes)
{
    if (!s->comm) { qsb_set_error("sharded readout needs qsb_comm_init first"); return QSB_ERR_COMM; }
    QSB_NCCL(g_nccl.AllGather(dsrc, ddst, bytes, 1 /* ncclUint8 */, (qsb_nccl_comm_t)s->comm, s->stream));
    return QSB_OK;
}
int tiled_comm_allreduce_sum_u64(qsb_sim *s, void *dbuf, size_t count)
{
    if (!s->comm) { qsb_set_error("sharded readout needs qsb_comm_init first"); return QSB_ERR_COMM; }
    QSB_NCCL(g_nccl.AllReduce(dbuf, dbuf, count, 5 /* ncclUint64 */, 0 /* ncclSum */, (qsb_nccl_comm_t)s->comm, s->stream));
    return QSB_OK;
}

/* one send / receive pair with `peer` (expectation values: the partner shard of terms that flip rank bits) */
int tiled_comm_sendrecv(qsb_sim *s, const void *dsend, void *drecv, size_t bytes, int peer)
{
    if (!s->comm) { qsb_set_error("sharded readout needs qsb_comm_init first"); return QSB_ERR_COMM; }
    QSB_NCCL(g_nccl.GroupStart());
    QSB_NCCL(g_nccl.Send(dsend, bytes, 1 /* ncclUint8 */, peer, (qsb_nccl_comm_t)s->comm, s->stream));
    QSB_NCCL(g_nccl.Recv(drecv, bytes, 1, peer, (qsb_nccl_comm_t)s->comm, s->stream));
    QSB_NCCL(g_nccl.GroupEnd());
    return QSB_OK;
}

void tiled_comm_destroy(qsb_sim *s)
{
    if (s->peers_ok) {
        for (int r = 0; r < s->world; r++) if (r != s->rank) {
            /* peer_state / peer_state2 may have traded places: close both mappings whatever their current role */
            if (s->peer_state[r]) cudaIpcCloseMemHandle(s->peer_state[r]);
            if (s->peer_state2[r]) cudaIpcCloseMemHandle(s->peer_state2[r]);
        }
        s->peers_ok = false;
    }
    if (s->comm && g_nccl.CommDestroy) { g_nccl.CommDestroy((qsb_nccl_comm_t)s->comm); s->comm = nullptr; }
}

/* next event of the handle's pool (timing enabled: some bracket the exchange for exchange_ms) */
static int pool_event(qsb_sim *s, cudaEvent_t *out)
{
    if (s->ev_next == s->ev_pool.size()) { cudaEvent_t e; QSB_CUDA(cudaEventCreate(&e)); s->ev_pool.push_back(e); }
    *out = s->ev_pool[s->ev_next++];
    return QSB_OK;
}

static int exchange(qsb_sim *s)
{
    if (!s->comm) { qsb_set_error("plan needs a qubit exchange but qsb_comm_init was not called"); return QSB_ERR_COMM; }
    const int P = s->world;
    const size_t chunk = s->state_bytes / P;
    char *src = (char *)s->state, *dst = (char *)s->state2;
    QSB_NCCL(g_nccl.GroupStart());
    for (int j = 0; j < P; j++) {
        if (j == s->rank) continue;
        QSB_NCCL(g_nccl.Send(src + (size_t)j * chunk, chunk, 1 /* ncclUint8 */, j, (qsb_nccl_comm_t)s->comm, s->stream));
        QSB_NCCL(g_nccl.Recv(dst + (size_t)j * chunk, chunk, 1, j, (qsb_nccl_comm_t)s->comm, s->stream));
    }
    QSB_NCCL(g_nccl.GroupEnd());
    QSB_CUDA(cudaMemcpyAsync(dst + (size_t)s->rank * chunk, src + (size_t)s->rank * chunk, chunk, cudaMemcpyDeviceToDevice, s->stream));
    void *t = s->state; s->state = s->state2; s->state2 = t;
    if (s->peers_ok) for (int r = 0; r < s->world; r++) std::swap(s->peer_state[r], s->peer_state2[r]);
    return QSB_OK;
}

/* Pipelined exchange (reserved[5] = 3): the in-tile permutation pass that precedes an exchange runs in
 * slices of tiles; as soon as a slice is through, its part of every chunk goes to the peers' second
 * buffers with cudaMemcpyAsync on a second stream (copy engines over NVLink) while the SMs compute the
 * next slice.  A slice fixes the top S outer index bits; tile bits lying above the lowest of them split
 * its address range into 2^m contiguous pieces per chunk. */
static int pipelined_exchange(qsb_sim *s, TiledPlan *p, size_t k_pass, bool have_pass, std::vector<cudaEvent_t> &ev)
{
    const int NCS = 4;   /* several copy streams so that the transfers spread over the copy engines */
    for (int i = 0; i < NCS; i++) if (!s->copy_stream[i]) QSB_CUDA(cudaStreamCreateWithFlags(&s->copy_stream[i], cudaStreamNonBlocking));
    int next_cs = 0;
    const int P = s->world, g = s->g, nloc = s->nloc;
    const size_t AMP = amp_bytes(s->prec), chunk = s->state_bytes / P;
    std::vector<int> slice_pos;                     /* positions of the slicing bits, highest first */
    uint64_t n_tiles = 1;
    if (have_pass) {
        const HostPass &hp = p->passes[k_pass];
        n_tiles = hp.hdr.n_tiles;
        std::vector<int> outer;                     /* outer positions, ascending = tile-id bit order */
        for (uint32_t r = 0; r < hp.hdr.n_runs; r++) for (int b = 0; b < hp.hdr.run_len[r]; b++) outer.push_back(hp.hdr.run_start[r] + b);
        int S = std::min<int>(3, (int)outer.size());
        if (!outer.empty() && outer.back() >= nloc - g) S = 0;   /* chunk-select bits outside the tile: no slicing */
        while (S > 0) {
            const int lo = outer[outer.size() - S];
            int m = 0;
            for (int q = lo + 1; q < nloc - g; q++) if (std::find(outer.begin(), outer.end(), q) == outer.end()) m++;
            if (m <= 4) break;
            S--;
        }
        for (int i = 0; i < S; i++) slice_pos.push_back(outer[outer.size() - 1 - i]);
    }
    const int S = (int)slice_pos.size(), K = 1 << S;
    const int lo = S ? slice_pos.back() : nloc - g;  /* everything below `lo` is contiguous inside a piece */
    std::vector<int> mid;                            /* tile bits between lo and the chunk-select bits */
    for (int q = lo + 1; q < nloc - g; q++) if (std::find(slice_pos.begin(), slice_pos.end(), q) == slice_pos.end()) mid.push_back(q);
    const size_t piece = ((size_t)1 << lo) * AMP;
    cudaEvent_t x0, x1;
    { int rc = pool_event(s, &x0); if (rc) return rc; rc = pool_event(s, &x1); if (rc) return rc; }
    for (int sl = 0; sl < K; sl++) {
        if (have_pass) {
            int rc = tiled_launch_pass(s, p, k_pass, s->state, s->state, nullptr, (uint64_t)sl * (n_tiles / K), n_tiles / K);
            if (rc) return rc;
        }
        cudaEvent_t e; { int rc = pool_event(s, &e); if (rc) return rc; }
        QSB_CUDA(cudaEventRecord(e, s->stream));
        for (int i = 0; i < NCS; i++) QSB_CUDA(cudaStreamWaitEvent(s->copy_stream[i], e, 0));
        if (sl == K - 1) QSB_CUDA(cudaEventRecord(x0, s->stream));   /* what follows is exposed transfer time */
        /* slice sl = the slicing bits take the value sl (highest slicing bit = highest bit of sl) */
        uint64_t base = 0;
        for (int i = 0; i < S; i++) if ((sl >> (S - 1 - i)) & 1) base |= 1ULL << slice_pos[i];
        for (uint64_t mm = 0; mm < (1ULL << mid.size()); mm++) {
            uint64_t off = base;
            for (size_t b = 0; b < mid.size(); b++) if ((mm >> b) & 1) off |= 1ULL << mid[b];
            for (int jj = 0; jj < P; jj++) {
                const int j = (s->rank + jj) % P;    /* start with the local chunk, then round-robin over the peers */
                const char *src = (const char *)s->state + (size_t)j * chunk + off * AMP;
                char *dst = (char *)s->peer_state2[j] + (size_t)s->rank * chunk + off * AMP;
                QSB_CUDA(cudaMemcpyAsync(dst, src, piece, cudaMemcpyDeviceToDevice, s->copy_stream[next_cs]));
                next_cs = (next_cs + 1) % NCS;
            }
        }
    }
    for (int i = 0; i < NCS; i++) {
        cudaEvent_t done; { int rc = pool_event(s, &done); if (rc) return rc; }
        QSB_CUDA(cudaEventRecord(done, s->copy_stream[i]));
        QSB_CUDA(cudaStreamWaitEvent(s->stream, done, 0));
    }
    int *flag = (int *)((char *)s->d_scratch + 65536);
    QSB_NCCL(g_nccl.AllReduce(flag, flag + 1, 1, 2 /* ncclInt32 */, 3 /* ncclMin */, (qsb_nccl_comm_t)s->comm, s->stream));
    QSB_CUDA(cudaEventRecord(x1, s->stream));
    ev.push_back(x0); ev.push_back(x1);
    std::swap(s->state, s->state2);
    for (int r = 0; r < P; r++) std::swap(s->peer_state[r], s->peer_state2[r]);
    return QSB_OK;
}

int tiled_execute(qsb_sim *s, TiledPlan *p)
{
    std::vector<cudaEvent_t> ev;      /* (start, end) pairs that bracket the exchanges; all from the handle's pool */
    s->ev_next = 0;
    const bool pipelined = s->peers_ok && s->opt.reserved[5] == 3;
    for (size_t k = 0; k < p->passes.size(); k++) {
        if (pipelined && !p->passes[k].is_swap && k + 1 < p->passes.size() && p->passes[k + 1].is_swap) {
            int rc = pipelined_exchange(s, p, k, true, ev);
            if (rc) return rc;
            k++;                                    /* the marker is consumed */
            continue;
        }
        if (pipelined && p->passes[k].is_swap) {
            int rc = pipelined_exchange(s, p, k, false, ev);
            if (rc) return rc;
            continue;
        }
        if (p->passes[k].is_swap) {
            cudaEvent_t a, b;
            { int rc = pool_event(s, &a); if (rc) return rc; rc = pool_event(s, &b); if (rc) return rc; }
            QSB_CUDA(cudaEventRecord(a, s->stream));
            int rc = exchange(s);
            if (rc) return rc;
            QSB_CUDA(cudaEventRecord(b, s->stream));
            ev.push_back(a); ev.push_back(b);
            continue;
        }
        if (p->passes[k].fused_swap) {
            /* the pass scatters into every rank's SECOND buffer; once all ranks are through (an all-reduce on the
             * stream is the barrier) the buffers trade places everywhere */
            if (!s->peers_ok) { qsb_set_error("plan has fused exchanges but the peer shards are not mapped"); return QSB_ERR_COMM; }
            cudaEvent_t a, b;
            { int rc = pool_event(s, &a); if (rc) return rc; rc = pool_event(s, &b); if (rc) return rc; }
            PeerTab pt; memset(&pt, 0, sizeof pt);
            for (int r = 0; r < s->world; r++) pt.p[r] = (char *)s->peer_state2[r];
            pt.shard_bytes = s->state_bytes; pt.world = (uint32_t)s->world;
            int rc = tiled_launch_pass(s, p, k, s->state, s->state2, &pt, 0, 0);
            if (rc) return rc;
            QSB_CUDA(cudaEventRecord(a, s->stream));
            int *flag = (int *)((char *)s->d_scratch + 65536);
            QSB_NCCL(g_nccl.AllReduce(flag, flag + 1, 1, 2 /* ncclInt32 */, 3 /* ncclMin */, (qsb_nccl_comm_t)s->comm, s->stream));
            QSB_CUDA(cudaEventRecord(b, s->stream));
            ev.push_back(a); ev.push_back(b);
            std::swap(s->state, s->state2);
            for (int r = 0; r < s->world; r++) std::swap(s->peer_state[r], s->peer_state2[r]);
            continue;
        }
        int rc = tiled_launch_pass(s, p, k, s->state, s->state, nullptr, 0, 0);
        if (rc) return rc;
    }
    s->perm = p->end_perm;
    p->last_exchange_ms = 0.0;
    if (!ev.empty()) {
        QSB_CUDA(cudaStreamSynchronize(s->stream));
        for (size_t i = 0; i < ev.size(); i += 2) {
            float ms = 0; cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
            p->last_exchange_ms += ms;
        }
    }
    return QSB_OK;
}
