/* pauli.h -- Pauli-string helpers defined in expect.cu and shared by pauli_rot.cu (host only, no CUDA calls). */
#pragma once
#include <vector>
#include "sim.h"

struct PhysTerm { uint64_t xl, zl, xr, zr; int y; };   /* local / rank-bit parts of the physical masks, y = popc(x&z) & 3 */

inline int parity64(uint64_t v) { return __builtin_popcountll(v) & 1; }

/* tile bits T (12 f32 / 11 f64) and the low bits L every tile keeps, for a precision and the handle's options */
int exp_geometry(int prec, const qsb_options_t *opt, int *T, int *L);
/* QSB_ERR_ARG (with a message naming fn) for a null array when nterms > 0 or a qubit >= n */
int check_terms(int n, const uint64_t *x, const uint64_t *z, size_t nterms, const char *fn);
/* logical masks -> physical local / rank-bit masks under the layout perm */
void to_physical(int n, int nloc, const BitPerm &perm, const uint64_t *x, const uint64_t *z, size_t nterms, std::vector<PhysTerm> &out);
/* compress the bits of m at the positions pb[0..T-1] */
uint32_t tile_coord(uint64_t m, const int8_t *pb, int T);
/* the options and local bits of a dry run: the checks of qsb_create on (num_qubits, opt), without a device */
int pauli_dry_run_shape(int num_qubits, const qsb_options_t *opt_in, qsb_options_t *opt, int *nloc);
