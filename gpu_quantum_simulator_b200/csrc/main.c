/*
 * main.c -- `qsim`, the C host driver.  Drop-in for the reference CLIs:
 *   C program   : <exe> <circuit_file> <number_of_measurement>   (quantum_simulator.c:39-43)
 *   CUDA programs: <exe> <circuit_file>                           (quantum_simulator_naive.cu:135-139)
 * stdout line 1 is the elapsed seconds "%lf\n" exactly as the reference prints
 * it (quantum_simulator.c:248).  Everything else is opt-in and follows the
 * formats the reference left commented out:
 *   --dump-amplitudes   "%llu : %f + %f i" per non-zero amplitude, then
 *                       "MOST LIKELY MEASUREMENT: %llu (%f)"   (naive.cu:207-216)
 *   <number_of_measurement> > 0 with --shots: "MEASUREMENT: <bits> (%ld)" (quantum_simulator.c:68-73)
 *   --save-state FILE / --load-state FILE   raw shard + qubit map after / before the circuit (checkpoint;
 *                       the reference keeps the state only in memory, quantum_simulator.c:75)
 *   --matrix "0 3" FILE   (repeatable) the dense 2^k x 2^k matrix in FILE (2 * 4^k whitespace-separated numbers: re im,
 *                       row-major; row / column index bit i = value of the i-th qubit listed) applied on the device after
 *                       the circuit and --load-state; all --matrix flags go in flag order as one call, before --pauli-rot,
 *                       --gradient and --save-state, so every later line reads the transformed state.  The files and
 *                       qubit lists are checked before the circuit runs
 *   --pauli-rot "X0 Z3" 0.25   (repeatable) the rotation exp(-i 0.25 P / 2) applied on the device after the circuit (after
 *                       --load-state, before --save-state), in flag order, so the lines below read the rotated state
 *   --gradient "Z0 Z1" 0.5   (repeatable) a term 0.5 P of an observable H; with any, the --pauli-rot list is applied
 *                       through the gradient call, which prints "ENERGY e" (<psi|H|psi>) and "GRADIENT g0 g1 ..." (dE/dtheta
 *                       of each --pauli-rot angle in flag order, %.17g) after the --profile line
 *   --expect "Z0 Z1"    (repeatable) <psi|P|psi> of a Pauli string after the circuit, computed on the device:
 *                       one "EXPECTATION <text>: %.17g" line per flag, in flag order, after the --profile line
 *   --marginal "0 3 5"  (repeatable) marginal probabilities of these qubits after the circuit, computed on the device:
 *                       one "MARGINAL <qubits>: p_0 ... p_{2^k-1}" line (%.17g, bin b: bit i = value of the i-th
 *                       qubit listed) per flag, in flag order, after the EXPECTATION lines
 *   --rdm "0 3"         (repeatable) reduced density matrix of these qubits after the circuit, computed on the device:
 *                       one "RDM <qubits>: re_00 im_00 re_01 im_01 ..." line (%.17g, row-major, row / column index: bit i
 *                       = value of the i-th qubit listed) per flag, in flag order, after the MARGINAL lines
 *   --plan-only [--gpus N]   host-side fusion only (no GPU needed): one JSON line with the passes, rounds, ops and
 *                       qubit exchanges the circuit would run as on N ranks, instead of running it
 * Errors go to stdout followed by exit(1), like the reference (:56,:129,:213-219).
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/time.h>
#include <time.h>

#include "qsim_b200.h"

static double now_s(void)
{
    struct timeval tv;
    gettimeofday(&tv, NULL);
    return tv.tv_sec + tv.tv_usec * 1e-6;
}

static void putb(unsigned long long n, int len) /* MSB first, quantum_simulator.c:285-293 */
{
    for (int k = len - 1; k >= 0; k--) putchar('0' + (int)((n >> k) & 1ULL));
}

static void usage(const char *exe)
{
    printf("QUANTUM CIRCUIT SIMULATOR\n");
    printf("Usage: %s <circuit_file_name> <number_of_measurement>\n", exe);
}

static void format_help(void)
{
    printf("Input format: \n\n");
    printf("OPENQASM 3.0;\n");
    printf("include \"stdgates.inc\";\n");
    printf("qubit[<num_qubit>] q; or qubit q[<num_qubit>]; \\\\single quantum register \n");
    printf("<quantum_circuit>\n\n");
    printf("Supported operations: cx, x, sx, z, s, sdg, t, tdg, rz, h\n");
    printf("(extensions: y p rx ry u cz cy ch cp swap ccx, gate definitions, ctrl/negctrl/inv/pow modifiers, gphase, pi expressions)\n");
}

/* "0 3 5": whitespace-separated qubits -> qs[0..*k-1]; 0 when the text is not such a list */
static int parse_qubits(const char *text, int qs[64], int *k)
{
    const char *p = text;
    *k = 0;
    for (;;) {
        while (*p == ' ' || *p == '\t') p++;
        if (!*p) return 1;
        char *end;
        long v = strtol(p, &end, 10);
        if (end == p || (*end && *end != ' ' && *end != '\t') || v < 0 || v > 1000000 || *k == 64) return 0;
        qs[(*k)++] = (int)v;
        p = end;
    }
}

int main(int argc, char **argv)
{
    const char *file = NULL, *dump_bin = NULL, *save_state = NULL, *load_state = NULL;
    long num_m = 0;
    int precision = 32, dump = 0, shots = 0, prec_out = 0, profile = 0, sweep = 0, have_m = 0, plan_only = 0, gpus = 1;
    unsigned long long seed = 0; int have_seed = 0;
    const char **expect = (const char **)calloc((size_t)argc, sizeof(char *)); int n_expect = 0;
    const char **marginal = (const char **)calloc((size_t)argc, sizeof(char *)); int n_marginal = 0;
    const char **rdm = (const char **)calloc((size_t)argc, sizeof(char *)); int n_rdm = 0;
    const char **rot = (const char **)calloc((size_t)argc, sizeof(char *)); int n_rot = 0;
    double *rot_theta = (double *)calloc((size_t)argc, sizeof(double));
    const char **gterm = (const char **)calloc((size_t)argc, sizeof(char *)); int n_gterm = 0;
    double *gcoef = (double *)calloc((size_t)argc, sizeof(double));
    double energy = 0.0, *grad = (double *)calloc((size_t)argc, sizeof(double));
    const char **mat_q = (const char **)calloc((size_t)argc, sizeof(char *)), **mat_f = (const char **)calloc((size_t)argc, sizeof(char *));
    int n_mat = 0;
    for (int i = 1; i < argc; i++) {
        if (!strcmp(argv[i], "--precision") && i + 1 < argc) precision = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--dump-amplitudes")) dump = 1;
        else if (!strcmp(argv[i], "--precision-out") && i + 1 < argc) prec_out = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--dump-bin") && i + 1 < argc) dump_bin = argv[++i];
        else if (!strcmp(argv[i], "--save-state") && i + 1 < argc) save_state = argv[++i];
        else if (!strcmp(argv[i], "--load-state") && i + 1 < argc) load_state = argv[++i];
        else if (!strcmp(argv[i], "--shots")) shots = 1;
        else if (!strcmp(argv[i], "--seed") && i + 1 < argc) { seed = strtoull(argv[++i], NULL, 10); have_seed = 1; }
        else if (!strcmp(argv[i], "--profile")) profile = 1;
        else if (!strcmp(argv[i], "--plan-only")) plan_only = 1;
        else if (!strcmp(argv[i], "--gpus") && i + 1 < argc) gpus = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--sweep")) sweep = 1;
        else if (!strcmp(argv[i], "--expect") && i + 1 < argc) expect[n_expect++] = argv[++i];
        else if (!strcmp(argv[i], "--marginal") && i + 1 < argc) marginal[n_marginal++] = argv[++i];
        else if (!strcmp(argv[i], "--rdm") && i + 1 < argc) rdm[n_rdm++] = argv[++i];
        else if (!strcmp(argv[i], "--matrix") && i + 2 < argc) { mat_q[n_mat] = argv[++i]; mat_f[n_mat++] = argv[++i]; }
        else if (!strcmp(argv[i], "--pauli-rot") && i + 2 < argc) {
            char *end;
            rot[n_rot] = argv[++i];
            rot_theta[n_rot] = strtod(argv[++i], &end);
            if (end == argv[i] || *end) { printf("--pauli-rot \"%s\" %s: expected an angle\n", rot[n_rot], argv[i]); return 1; }
            n_rot++;
        }
        else if (!strcmp(argv[i], "--gradient") && i + 2 < argc) {
            char *end;
            gterm[n_gterm] = argv[++i];
            gcoef[n_gterm] = strtod(argv[++i], &end);
            if (end == argv[i] || *end) { printf("--gradient \"%s\" %s: expected a coefficient\n", gterm[n_gterm], argv[i]); return 1; }
            n_gterm++;
        }
        else if (!file) file = argv[i];
        else if (!have_m) { num_m = atol(argv[i]); have_m = 1; }
    }
    if (!file) { usage(argv[0]); return 1; }
    if (!have_seed) seed = (unsigned long long)time(NULL);   /* srand(time(NULL)), :46 */
    /* --matrix files are read and checked before the circuit runs, so a bad file costs nothing */
    qsb_matrix_op_t *mops = (qsb_matrix_op_t *)calloc((size_t)n_mat + 1, sizeof(qsb_matrix_op_t));
    if (!mops) { printf("Malloc error\n"); return 1; }
    for (int m = 0; m < n_mat; m++) {
        int qs[64], k = 0;
        if (!parse_qubits(mat_q[m], qs, &k) || k < 1 || k > QSB_MATRIX_MAX_K) {
            printf("--matrix \"%s\": expected a whitespace-separated list of 1..%d qubits\n", mat_q[m], QSB_MATRIX_MAX_K); return 1;
        }
        const size_t want = (size_t)2 << (2 * k);
        double *e = (double *)malloc(sizeof(double) * want);
        FILE *f = fopen(mat_f[m], "r");
        if (!e) { printf("Malloc error\n"); return 1; }
        if (!f) { printf("--matrix \"%s\" %s: cannot open the file\n", mat_q[m], mat_f[m]); return 1; }
        size_t got = 0;
        double v;
        while (got <= want && fscanf(f, "%lf", &v) == 1) { if (got < want) e[got] = v; got++; }
        int ch;
        while ((ch = fgetc(f)) == ' ' || ch == '\t' || ch == '\n' || ch == '\r') {}
        const int clean = ch == EOF;   /* nothing but numbers and white space */
        fclose(f);
        if (got != want || !clean) {
            printf("--matrix \"%s\" %s: expected %zu numbers (re im of a %d x %d matrix, row-major)%s\n", mat_q[m], mat_f[m],
                   want, 1 << k, 1 << k, got > want ? ", found more" : !clean ? ", found text that is not a number" : "");
            return 1;
        }
        mops[m].k = k;
        for (int i = 0; i < k; i++) mops[m].targets[i] = qs[i];
        mops[m].m = e;
    }

    int nq = 0; qsb_gate_t *gates = NULL; size_t n = 0;
    int rc = qsb_parse_qasm_file(file, &nq, &gates, &n);
    if (rc == QSB_ERR_IO) { printf("ERROR: cannot open circuit file\n"); return 1; }
    if (rc) {
        printf("%s\n", qsb_last_error());
        if (rc == QSB_ERR_PARSE) format_help();
        printf("ERROR while parsing quantum circuit\n");
        return 1;
    }

    double t0 = now_s();
    qsb_options_t o; qsb_options_default(&o);
    o.precision = precision == 64 ? QSB_F64 : QSB_F32;
    if (sweep) o.mode = QSB_MODE_SWEEP;
    if (plan_only) {
        qsb_run_stats_t st;
        o.world_size = gpus;
        if (qsb_plan_dry_run(nq, &o, gates, n, &st)) { printf("%s\n", qsb_last_error()); return 1; }
        printf("{\"qubits\": %d, \"gates\": %llu, \"ranks\": %d, \"precision\": %d, \"passes\": %u, \"rounds\": %u, \"device_ops\": %llu, "
               "\"exchanges\": %u, \"bytes_moved_per_rank\": %llu, \"bytes_exchanged_per_rank\": %llu, \"plan_ms\": %.3f, \"lib\": \"%s\"}\n",
               nq, (unsigned long long)st.source_gates, gpus, precision == 64 ? 64 : 32, st.passes, st.rounds, (unsigned long long)st.device_ops,
               st.swaps, (unsigned long long)st.bytes_moved, (unsigned long long)st.bytes_exchanged, st.plan_ms, qsb_version());
        qsb_free(gates);
        return 0;
    }
    /* the qubits and entries of every --matrix against the circuit's register, before the circuit runs */
    if (n_mat && qsb_matrix_dry_run(nq, &o, mops, (size_t)n_mat, NULL, NULL)) { printf("%s\n", qsb_last_error()); return 1; }
    qsb_t *s = NULL;
    rc = qsb_create(&s, nq, &o);
    if (!rc && load_state) rc = qsb_load_state(s, load_state);
    if (!rc) rc = qsb_apply_gates(s, gates, n);
    if (!rc && n_mat) rc = qsb_apply_matrices(s, mops, (size_t)n_mat);   /* one call: consecutive ops share sweeps */
    if (!rc && (n_rot || n_gterm)) {   /* one call for all rotations: consecutive ones share sweeps over the state */
        uint64_t *rx = (uint64_t *)malloc(sizeof(uint64_t) * 2 * (n_rot + n_gterm) + 16);
        if (!rx) { printf("Malloc error\n"); return 1; }
        uint64_t *hx = rx + 2 * n_rot;
        for (int k = 0; k < n_rot && !rc; k++) rc = qsb_pauli_from_string(rot[k], nq, &rx[k], &rx[n_rot + k]);
        for (int k = 0; k < n_gterm && !rc; k++) rc = qsb_pauli_from_string(gterm[k], nq, &hx[k], &hx[n_gterm + k]);
        if (!rc && n_gterm)
            rc = qsb_pauli_rotation_gradient(s, rx, rx + n_rot, rot_theta, (size_t)n_rot, hx, hx + n_gterm, gcoef, (size_t)n_gterm, &energy, grad);
        else if (!rc) rc = qsb_apply_pauli_rotations(s, rx, rx + n_rot, rot_theta, (size_t)n_rot);
        free(rx);
    }
    if (!rc && save_state) rc = qsb_save_state(s, save_state);
    if (rc) { printf("%s\n", qsb_last_error()); return 1; }
    printf("%lf\n", now_s() - t0);

    if (profile) {
        qsb_run_stats_t st; qsb_last_run_stats(s, &st);
        printf("{\"qubits\": %d, \"gates\": %llu, \"passes\": %u, \"rounds\": %u, \"device_ms\": %.6f, \"plan_ms\": %.3f, "
               "\"bytes_moved\": %llu, \"gbps\": %.1f, \"gates_per_sec\": %.1f}\n",
               nq, (unsigned long long)st.source_gates, st.passes, st.rounds, st.device_ms, st.plan_ms,
               (unsigned long long)st.bytes_moved, st.device_ms > 0 ? st.bytes_moved / st.device_ms * 1e-6 : 0.0,
               st.device_ms > 0 ? st.source_gates / st.device_ms * 1e3 : 0.0);
    }
    if (n_gterm) {
        printf("ENERGY %.17g\n", energy);
        printf("GRADIENT");
        for (int k = 0; k < n_rot; k++) printf(" %.17g", grad[k]);
        printf("\n");
    }
    if (n_expect) {   /* one call for all terms: they share the sweeps over the state */
        uint64_t *ex = (uint64_t *)malloc(sizeof(uint64_t) * 2 * n_expect);
        double *ev = (double *)malloc(sizeof(double) * n_expect);
        if (!ex || !ev) { printf("Malloc error\n"); return 1; }
        for (int k = 0; k < n_expect && !rc; k++) rc = qsb_pauli_from_string(expect[k], nq, &ex[k], &ex[n_expect + k]);
        if (!rc) rc = qsb_expectation_pauli(s, ex, ex + n_expect, (size_t)n_expect, ev);
        if (rc) { printf("%s\n", qsb_last_error()); return 1; }
        for (int k = 0; k < n_expect; k++) printf("EXPECTATION %s: %.17g\n", expect[k], ev[k]);
        free(ex); free(ev);
    }
    for (int m = 0; m < n_marginal; m++) {
        int qs[64], k = 0;
        if (!parse_qubits(marginal[m], qs, &k)) {
            printf("--marginal \"%s\": expected a whitespace-separated list of qubits\n", marginal[m]); return 1;
        }
        double *mp = (double *)malloc(sizeof(double) * ((size_t)1 << (k < 20 ? k : 20)));
        if (!mp) { printf("Malloc error\n"); return 1; }
        if (qsb_marginal_probabilities(s, qs, k, mp)) { printf("%s\n", qsb_last_error()); return 1; }
        printf("MARGINAL");
        for (int i = 0; i < k; i++) printf(" %d", qs[i]);
        printf(":");
        for (size_t b = 0; b < ((size_t)1 << k); b++) printf(" %.17g", mp[b]);
        printf("\n");
        free(mp);
    }
    for (int m = 0; m < n_rdm; m++) {
        int qs[64], k = 0;
        if (!parse_qubits(rdm[m], qs, &k)) {
            printf("--rdm \"%s\": expected a whitespace-separated list of qubits\n", rdm[m]); return 1;
        }
        const size_t d = (size_t)1 << (k < 12 ? k : 12);   /* a larger k is refused before anything is written */
        double *rho = (double *)malloc(sizeof(double) * 2 * d * d);
        if (!rho) { printf("Malloc error\n"); return 1; }
        if (qsb_reduced_density_matrix(s, qs, k, rho)) { printf("%s\n", qsb_last_error()); return 1; }
        printf("RDM");
        for (int i = 0; i < k; i++) printf(" %d", qs[i]);
        printf(":");
        for (size_t e = 0; e < 2 * d * d; e++) printf(" %.17g", rho[e]);
        printf("\n");
        free(rho);
    }
    const unsigned long long N = 1ULL << nq;
    if (dump || dump_bin) {
        const unsigned long long chunk = 1ULL << 20;
        double *buf = (double *)malloc(sizeof(double) * 2 * (N < chunk ? N : chunk));
        FILE *fb = dump_bin ? fopen(dump_bin, "wb") : NULL;
        if (!buf || (dump_bin && !fb)) { printf("Malloc error\n"); return 1; }
        for (unsigned long long f = 0; f < N; f += chunk) {
            unsigned long long c = N - f < chunk ? N - f : chunk;
            if (qsb_download(s, buf, f, c)) { printf("%s\n", qsb_last_error()); return 1; }
            if (fb) fwrite(buf, sizeof(double), 2 * c, fb);
            if (dump) for (unsigned long long k = 0; k < c; k++) {
                double re = buf[2 * k], im = buf[2 * k + 1];
                if (re * re + im * im > 0.0) {
                    if (prec_out > 0) printf("%llu : %.*g + %.*g i\n", f + k, prec_out, re, prec_out, im);
                    else printf("%llu : %f + %f i\n", f + k, re, im);
                }
            }
        }
        if (fb) fclose(fb);
        free(buf);
        if (dump) {
            double norm, p; uint64_t idx;
            if (qsb_norm_argmax(s, &norm, &idx, &p)) { printf("%s\n", qsb_last_error()); return 1; }
            printf("MOST LIKELY MEASUREMENT: %llu (%f)\n", (unsigned long long)idx, p);
        }
    }
    if (shots && num_m > 0) {
        uint64_t *out = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)num_m);
        if (!out) { printf("Malloc error\n"); return 1; }
        if (qsb_sample(s, seed, (int)num_m, out)) { printf("%s\n", qsb_last_error()); return 1; }
        for (long i = 0; i < num_m; i++) {
            printf("MEASUREMENT: "); putb(out[i], nq); printf(" (%ld)\n", (long)out[i]);
        }
        free(out);
    }
    qsb_destroy(s);
    qsb_free(gates);
    free(expect);
    free(marginal);
    free(rdm);
    free(rot);
    free(rot_theta);
    free(gterm);
    free(gcoef);
    free(grad);
    for (int m = 0; m < n_mat; m++) free((void *)mops[m].m);
    free(mops);
    free(mat_q);
    free(mat_f);
    return 0;
}
