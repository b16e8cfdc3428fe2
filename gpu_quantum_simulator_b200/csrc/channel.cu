/*
 * channel.cu -- noise channels by quantum trajectories: Kraus channels applied in list order, one branch per channel drawn
 * from a caller-given r (DESIGN.md section 3.3, noise channels).
 *
 * HOST RESOLUTION.  The walk over the list keeps a pending run: operators chosen but not yet applied.
 *   - A fixed-weight channel (every K_i^dag K_i = q_i I) is resolved at once from r and q_i; K_i / sqrt(q_i) joins the
 *     pending run unless it is an identity branch.
 *   - A state-dependent channel starts a group; consecutive channels of either kind join it while the union U of their
 *     targets has at most 4 qubits.  The group needs rho_U, the Gram matrix (reduced density matrix) of the state after
 *     the pending run on U.  Given rho_U, the host resolves every channel of the group exactly in fp64, in order: each K_i
 *     embedded into U, w_i = Re Tr(K_i rho K_i^dag) in a fixed order, the branch by pick_outcome (measure.cu),
 *     rho <- (T / w_i) K_i rho K_i^dag.  The chosen sqrt(T / w_i) K_i, on the channel's own targets, join the pending
 *     run.  The weights of later channels of a group thus come from rho_U carried on the host, not from a new read.
 *   - At the end of the list the pending run is applied.
 *
 * DEVICE.  A pending run is one qsb_apply_matrices call (matrix.cu: consecutive ops share a sweep whenever their targets
 * fit one tile) and rho_U one qsb_reduced_density_matrix call (rdm.cu: one read of the shard for u <= 4).  Both are
 * deterministic, keep the layout, the state buffer and the peer mappings, and on a sharded state are collective with the
 * same bits on every rank (partner-shard receive and SWAP expansion for rank targets, per-rank blocks all-gathered and
 * summed in rank order for rho), so every rank resolves the same branches.  A fused sweep that applies the run and
 * accumulates rho_U from its staged tiles was measured slower than this at 30 qubits f32 (DESIGN.md section 3.3, noise
 * channels) and is not kept.
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <deque>
#include <vector>

#include "pauli.h"
#include "sim.h"

#define CH_UMAX 4                          /* qubits of a group's Gram matrix */

/* ================================================================================================ host */

namespace {

struct Chan {                   /* one checked channel */
    int k, t[QSB_CHANNEL_MAX_K], nk;
    const double *kraus;        /* NULL in a dry run without operators */
    bool fixed;                 /* every K_i^dag K_i = q_i I */
    std::vector<double> q;      /* fixed: q_i */
};

inline size_t op_doubles(int k) { return (size_t)2 << (2 * k); }

/* max abs entry of sum_i K_i^dag K_i - I; fixed-weight classification and q_i on the way */
void gram_of_set(const Chan &c, double *dev_tp, bool *fixed, std::vector<double> &q)
{
    const int D = 1 << c.k;
    std::vector<double> S(2 * D * D, 0.0), M(2 * D * D);
    *fixed = true;
    q.assign(c.nk, 0.0);
    for (int i = 0; i < c.nk; i++) {
        const double *K = c.kraus + i * op_doubles(c.k);
        for (int a = 0; a < D; a++)
            for (int b = 0; b < D; b++) {   /* (K^dag K)[a][b] = sum_r conj(K[r][a]) K[r][b] */
                double re = 0.0, im = 0.0;
                for (int r = 0; r < D; r++) {
                    const double xr = K[2 * (r * D + a)], xi = K[2 * (r * D + a) + 1];
                    const double yr = K[2 * (r * D + b)], yi = K[2 * (r * D + b) + 1];
                    re += xr * yr + xi * yi;
                    im += xr * yi - xi * yr;
                }
                M[2 * (a * D + b)] = re; M[2 * (a * D + b) + 1] = im;
                S[2 * (a * D + b)] += re; S[2 * (a * D + b) + 1] += im;
            }
        double tr = 0.0;
        for (int a = 0; a < D; a++) tr += M[2 * (a * D + a)];
        q[i] = tr / D;
        for (int a = 0; a < D && *fixed; a++)
            for (int b = 0; b < D; b++) {
                const double dr = M[2 * (a * D + b)] - (a == b ? q[i] : 0.0), di = M[2 * (a * D + b) + 1];
                if (std::max(fabs(dr), fabs(di)) > 1e-12) { *fixed = false; break; }
            }
    }
    double dev = 0.0;
    for (int a = 0; a < D; a++)
        for (int b = 0; b < D; b++)
            dev = std::max(dev, std::max(fabs(S[2 * (a * D + b)] - (a == b ? 1.0 : 0.0)), fabs(S[2 * (a * D + b) + 1])));
    *dev_tp = dev;
}

/* the argument checks of qsb_apply_channels / qsb_channel_dry_run (need_kraus: a null kraus is refused) */
int check_channels(int n, const qsb_channel_t *ch, size_t count, bool need_kraus, const char *fn, std::vector<Chan> &out)
{
    if (count && !ch) { qsb_set_error("%s: null channel array", fn); return QSB_ERR_ARG; }
    const int kmax = std::min(n, QSB_CHANNEL_MAX_K);
    out.resize(count);
    for (size_t c = 0; c < count; c++) {
        const qsb_channel_t &h = ch[c];
        Chan &o = out[c];
        if (h.flags) { qsb_set_error("%s: channel %zu has flags %d, expected 0", fn, c, (int)h.flags); return QSB_ERR_ARG; }
        if (h.k < 1 || h.k > kmax) { qsb_set_error("%s: channel %zu has %d targets, expected 1..%d", fn, c, (int)h.k, kmax); return QSB_ERR_ARG; }
        uint64_t seen = 0;
        for (int j = 0; j < h.k; j++) {
            const int t = h.targets[j];
            if (t < 0 || t >= n) { qsb_set_error("%s: channel %zu has target %d outside [0, %d)", fn, c, t, n); return QSB_ERR_ARG; }
            if ((seen >> t) & 1) { qsb_set_error("%s: channel %zu has target %d twice", fn, c, t); return QSB_ERR_ARG; }
            seen |= 1ULL << t;
            o.t[j] = t;
        }
        const int nmax = 1 << (2 * h.k);
        if (h.nkraus < 1 || h.nkraus > nmax) {
            qsb_set_error("%s: channel %zu has %d Kraus operators, expected 1..%d", fn, c, (int)h.nkraus, nmax);
            return QSB_ERR_ARG;
        }
        o.k = h.k;
        o.nk = h.nkraus;
        o.kraus = h.kraus;
        o.fixed = false;
        if (!h.kraus) {
            if (need_kraus) { qsb_set_error("%s: channel %zu has a null kraus array", fn, c); return QSB_ERR_ARG; }
            continue;
        }
        const size_t cnt = (size_t)h.nkraus * op_doubles(h.k);
        for (size_t e = 0; e < cnt; e++)
            if (!isfinite(h.kraus[e])) { qsb_set_error("%s: channel %zu has a non-finite entry at %zu", fn, c, e); return QSB_ERR_ARG; }
        double dev;
        gram_of_set(o, &dev, &o.fixed, o.q);
        if (!(dev <= 1e-10)) {
            qsb_set_error("%s: channel %zu is not trace-preserving (max |sum K^dag K - I| = %g > 1e-10)", fn, c, dev);
            return QSB_ERR_ARG;
        }
    }
    return QSB_OK;
}

/* a positive real multiple of the identity: applying it (rescaled to keep the norm) changes nothing */
bool is_identity(const double *K, int k)
{
    const int D = 1 << k;
    const double d0 = K[0];
    if (!(d0 > 0.0)) return false;
    for (int a = 0; a < D; a++)
        for (int b = 0; b < D; b++) {
            const double re = K[2 * (a * D + b)], im = K[2 * (a * D + b) + 1];
            if (im != 0.0 || re != (a == b ? d0 : 0.0)) return false;
        }
    return true;
}

/* what the walk does with a step: count it (dry run) or run it */
struct Exec {
    virtual ~Exec() {}
    /* apply the run; u > 0: then rho (2 * 4^u doubles) = the Gram matrix of U */
    virtual int step(const std::vector<qsb_matrix_op_t> &run, const int *U, int u, double *rho) = 0;
};

struct DryExec : Exec {
    int n = 0, nloc = 0;
    qsb_options_t opt{};
    uint32_t sweeps = 0, gram_sweeps = 0, exchanges = 0;
    int step(const std::vector<qsb_matrix_op_t> &run, const int *U, int u, double *) override
    {
        if (!run.empty()) {
            uint32_t sw = 0, ex = 0;
            const int rc = qsb_matrix_dry_run(n, &opt, run.data(), run.size(), &sw, &ex);
            if (rc) return rc;
            sweeps += sw;
            exchanges += ex;
        }
        if (u) {   /* the reduced density matrix: one read, plus one partner shard and read per pattern of rank qubits */
            int m = 0;
            for (int i = 0; i < u; i++) m += U[i] >= nloc;
            gram_sweeps += 1u << m;
            exchanges += (1u << m) - 1;
        }
        return QSB_OK;
    }
};

struct DevExec : Exec {
    qsb_sim *s = nullptr;
    int step(const std::vector<qsb_matrix_op_t> &run, const int *U, int u, double *rho) override
    {
        if (!run.empty()) {
            const int rc = qsb_apply_matrices(s, run.data(), run.size());
            if (rc) return rc;
        }
        return u ? qsb_reduced_density_matrix(s, U, u, rho) : QSB_OK;
    }
};

/* E = K embedded into U (bit i of an index = value of U[i]): E[a][b] = K[a|t][b|t] where a and b agree off the targets */
void embed(const double *K, const int *t, int k, const int *U, int u, std::vector<double> &E)
{
    const int D = 1 << u, d = 1 << k;
    int pos[QSB_CHANNEL_MAX_K];
    uint32_t tmask = 0;
    for (int j = 0; j < k; j++) {
        for (int i = 0; i < u; i++) if (U[i] == t[j]) pos[j] = i;
        tmask |= 1u << pos[j];
    }
    auto ext = [&](int a) { int v = 0; for (int j = 0; j < k; j++) v |= ((a >> pos[j]) & 1) << j; return v; };
    E.assign(2 * D * D, 0.0);
    for (int a = 0; a < D; a++)
        for (int b = 0; b < D; b++) {
            if ((a & ~tmask) != (b & ~tmask)) continue;
            const int e = ext(a) * d + ext(b);
            E[2 * (a * D + b)] = K[2 * e];
            E[2 * (a * D + b) + 1] = K[2 * e + 1];
        }
}

/* X = E rho E^dag (D x D complex) */
void sandwich(const std::vector<double> &E, const std::vector<double> &rho, int D, std::vector<double> &X)
{
    std::vector<double> Y(2 * D * D);
    for (int a = 0; a < D; a++)
        for (int b = 0; b < D; b++) {   /* Y = E rho */
            double re = 0.0, im = 0.0;
            for (int c = 0; c < D; c++) {
                const double er = E[2 * (a * D + c)], ei = E[2 * (a * D + c) + 1];
                const double rr = rho[2 * (c * D + b)], ri = rho[2 * (c * D + b) + 1];
                re += er * rr - ei * ri;
                im += er * ri + ei * rr;
            }
            Y[2 * (a * D + b)] = re; Y[2 * (a * D + b) + 1] = im;
        }
    X.assign(2 * D * D, 0.0);
    for (int a = 0; a < D; a++)
        for (int b = 0; b < D; b++) {   /* X = Y E^dag: X[a][b] = sum_c Y[a][c] conj(E[b][c]) */
            double re = 0.0, im = 0.0;
            for (int c = 0; c < D; c++) {
                const double yr = Y[2 * (a * D + c)], yi = Y[2 * (a * D + c) + 1];
                const double er = E[2 * (b * D + c)], ei = E[2 * (b * D + c) + 1];
                re += yr * er + yi * ei;
                im += yi * er - yr * ei;
            }
            X[2 * (a * D + b)] = re; X[2 * (a * D + b) + 1] = im;
        }
}

/* The walk over the channel list (module comment).  dry: no operator is read, every branch is a non-identity op. */
int walk(const std::vector<Chan> &cs, const double *r, bool dry, Exec &ex, uint32_t *branch, double *prob, const char *fn)
{
    std::vector<qsb_matrix_op_t> run;
    std::deque<std::vector<double>> store;   /* the matrices of the pending run (stable addresses) */
    auto push = [&](const Chan &c, const double *K, double scale) {
        qsb_matrix_op_t o; memset(&o, 0, sizeof o);
        o.k = c.k;
        for (int j = 0; j < c.k; j++) o.targets[j] = c.t[j];
        if (K) {
            store.emplace_back(K, K + op_doubles(c.k));
            for (double &v : store.back()) v *= scale;
            o.m = store.back().data();
        }
        run.push_back(o);
    };
    size_t c = 0;
    while (c < cs.size()) {
        if (cs[c].fixed) {   /* resolved from q_i alone */
            const Chan &h = cs[c];
            if (!dry) {
                uint64_t b = 0;
                int rc = pick_outcome(h.q, r[c], &b, fn);
                if (rc) return rc;
                branch[c] = (uint32_t)b;
                if (prob) prob[c] = h.q[b];
                const double *K = h.kraus + b * op_doubles(h.k);
                if (!is_identity(K, h.k)) push(h, K, 1.0 / sqrt(h.q[b]));
            } else {
                push(h, nullptr, 1.0);
            }
            c++;
            continue;
        }
        /* a group: channels c..e-1, U = the union of their targets in order of appearance */
        int U[CH_UMAX], u = 0;
        size_t e = c;
        for (; e < cs.size(); e++) {
            int nu = u, V[CH_UMAX + QSB_CHANNEL_MAX_K];
            for (int i = 0; i < u; i++) V[i] = U[i];
            for (int j = 0; j < cs[e].k; j++) {
                bool in = false;
                for (int i = 0; i < nu; i++) in |= V[i] == cs[e].t[j];
                if (!in) V[nu++] = cs[e].t[j];
            }
            if (nu > CH_UMAX) break;
            for (int i = 0; i < nu; i++) U[i] = V[i];
            u = nu;
        }
        const int D = 1 << u;
        std::vector<double> rho(2 * D * D), E, X;
        int rc = ex.step(run, U, u, rho.data());
        if (rc) return rc;
        run.clear();
        store.clear();
        for (; c < e; c++) {
            const Chan &h = cs[c];
            if (dry) { push(h, nullptr, 1.0); continue; }
            std::vector<double> w(h.nk);
            std::vector<std::vector<double>> Xs(h.nk);
            for (int i = 0; i < h.nk; i++) {
                embed(h.kraus + i * op_doubles(h.k), h.t, h.k, U, u, E);
                sandwich(E, rho, D, Xs[i]);
                double tr = 0.0;
                for (int a = 0; a < D; a++) tr += Xs[i][2 * (a * D + a)];
                w[i] = std::max(tr, 0.0);
            }
            const std::vector<double> &tab = h.fixed ? h.q : w;
            double T = 0.0;
            for (double v : tab) T += v;
            if (!(T > 0.0)) { qsb_set_error("%s: channel %zu: the state has norm %g", fn, c, T); return QSB_ERR_ARG; }
            uint64_t b = 0;
            rc = pick_outcome(tab, r[c], &b, fn);
            if (rc) return rc;
            branch[c] = (uint32_t)b;
            const double p = h.fixed ? h.q[b] : w[b] / T, scale = h.fixed ? 1.0 / h.q[b] : T / w[b];
            if (prob) prob[c] = p;
            const double *K = h.kraus + b * op_doubles(h.k);
            if (is_identity(K, h.k)) continue;
            push(h, K, sqrt(scale));
            for (size_t x = 0; x < rho.size(); x++) rho[x] = scale * Xs[b][x];
        }
    }
    if (!run.empty()) return ex.step(run, nullptr, 0, nullptr);
    return QSB_OK;
}

int check_r(const double *r, size_t n, const char *fn)
{
    for (size_t c = 0; c < n; c++)
        if (!(r[c] >= 0.0 && r[c] < 1.0)) { qsb_set_error("%s: r[%zu] = %g outside [0, 1)", fn, c, r[c]); return QSB_ERR_ARG; }
    return QSB_OK;
}

}  // namespace

/* ------------------------------------------------------------------------------------------- C ABI */

extern "C" int qsb_channel_dry_run(int num_qubits, const qsb_options_t *opt_in, const qsb_channel_t *ch, size_t n,
                                   uint32_t *sweeps, uint32_t *gram_sweeps, uint32_t *exchanges)
{
    static const char *fn = "qsb_channel_dry_run";
    DryExec dx;
    int rc = pauli_dry_run_shape(num_qubits, opt_in, &dx.opt, &dx.nloc);
    if (rc) return rc;
    std::vector<Chan> cs;
    rc = check_channels(num_qubits, ch, n, false, fn, cs);
    if (rc) return rc;
    rc = check_low_bits(dx.opt.precision, &dx.opt, fn);
    if (rc) return rc;
    dx.n = num_qubits;
    rc = walk(cs, nullptr, true, dx, nullptr, nullptr, fn);
    if (rc) return rc;
    if (sweeps) *sweeps = dx.sweeps;
    if (gram_sweeps) *gram_sweeps = dx.gram_sweeps;
    if (exchanges) *exchanges = dx.exchanges;
    return QSB_OK;
}

extern "C" int qsb_apply_channels(qsb_t *s, const qsb_channel_t *ch, size_t n, const double *r, uint32_t *branch, double *prob)
{
    static const char *fn = "qsb_apply_channels";
    if (!s) { qsb_set_error("%s: null handle", fn); return QSB_ERR_ARG; }
    if (n == 0) return QSB_OK;
    if (!r || !branch) { qsb_set_error("%s: null %s", fn, !r ? "r" : "branch"); return QSB_ERR_ARG; }
    std::vector<Chan> cs;
    int rc = check_channels(s->n, ch, n, true, fn, cs);
    if (rc) return rc;
    rc = check_r(r, n, fn);
    if (rc) return rc;
    rc = check_low_bits(s->prec, &s->opt, fn);
    if (rc) return rc;
    if (s->g && !s->comm) { qsb_set_error("%s: sharded state needs qsb_comm_init first", fn); return QSB_ERR_COMM; }
    DevExec dx;
    dx.s = s;
    return walk(cs, r, false, dx, branch, prob, fn);
}
