"""Readout and expectation kernels at the edges where their work is split: CDF chunks and ranges that do not start at
0, download pipeline halves, probability and upload chunks, 256-index export runs, sampler launches, expectation
batches of more than one launch, every tile bit class of the Pauli sign bookkeeping, and the low_bits range.  Every
value is compared with a plain host reference: numpy in fp64, np.longdouble for prefix sums, or the exact answer
bit for bit where one is known."""
import itertools

import numpy as np
import pytest

import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import circuits
from test_gpu_expectation import TOL, expect_np, random_terms
from test_gpu_readout import cdf_ranges, check_shots, oracle_measure

pytestmark = pytest.mark.gpu

F32, F64 = q.F32, q.F64
PRECS = pytest.mark.parametrize("prec", [F32, F64], ids=["f32", "f64"])
CDF_CHUNK = 1 << 22          # qsb_cdf: values per chunk (4096-value blocks, <= 1024 of them)
EXP_KMAX = 512               # qsb_expectation_pauli: terms per launch


def permuted(n, prec, low_bits=0):
    """A handle on which fused circuits have left the qubit layout permuted, so logical and physical order differ."""
    s = q.Simulator(n, precision=prec, low_bits=low_bits, device=0)
    for seed in range(1, 30):
        s.apply(q.gates_from_circuit(circuits.random_layered(n, depth=2, seed=seed)))
        if not np.array_equal(s.layout()[0][:n], np.arange(n)):
            return s
    s.close()
    raise AssertionError(f"no circuit left a permuted layout (n={n}, prec={prec}, low_bits={low_bits})")


def random_state(n, seed):
    rng = np.random.default_rng(seed)
    a = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    return a / np.linalg.norm(a)


def as_stored(a, prec):
    """The amplitudes a handle of this precision holds after set_state(a), as complex128."""
    return a if prec == F64 else a.astype(np.complex64).astype(np.complex128)


def logical_from_physical(s, n):
    """s.shard_physical() gathered into logical order through s.layout()."""
    perm, _ = s.layout()
    idx = np.arange(1 << n, dtype=np.uint64)
    phys = np.zeros_like(idx)
    for k in range(n):
        phys |= ((idx >> np.uint64(k)) & np.uint64(1)) << np.uint64(int(perm[k]))
    return s.shard_physical()[phys]


def uniforms(seed, count):
    """The r of shots 0..count-1 of measurement(seed=seed): splitmix64, top 53 bits, vectorised."""
    x = np.uint64(seed) + np.arange(1, count + 1, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    z = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    z ^= z >> np.uint64(31)
    return (z >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def bits_of(v):
    return np.asarray(v, dtype=np.float64).view(np.uint64)


# ---------------------------------------------------------------------------------------------------------- CDF

@PRECS
def test_cdf_across_chunks(prec):
    """24 qubits = four 4 Mi-value chunks, so the carry chains from chunk to chunk; zero stretches (one across the
    first chunk boundary, one a whole chunk) make flat blocks and a flat carry."""
    n = 24
    N = 1 << n
    a = random_state(n, seed=24)
    zeros = [(0, 1000), (CDF_CHUNK - 5000, CDF_CHUNK + 7000), (2 * CDF_CHUNK, 3 * CDF_CHUNK), (3 * CDF_CHUNK + 123, 3 * CDF_CHUNK + 3 * 4096), (N - 777, N)]
    for z0, z1 in zeros:
        a[z0:z1] = 0.0
    with permuted(n, prec) as s:
        s.set_state(a)
        st = s.state()
        cdf = s.compute_state_cumulative_distribution()
        norm = s.norm_argmax()[0]
        p = st.real.astype(np.longdouble) ** 2 + st.imag.astype(np.longdouble) ** 2
        want = np.cumsum(p)
        assert float(np.max(np.abs(cdf - want))) <= 1e-12
        assert np.all(np.diff(cdf) >= 0.0)
        assert abs(cdf[-1] - norm) <= 1e-12
        for z0, z1 in zeros[1:]:                              # adding zeros leaves every level's value unchanged
            assert np.all(cdf[z0:z1] == cdf[z0 - 1]), (z0, z1)
        assert np.all(cdf[:1000] == 0.0)
        firsts = [CDF_CHUNK + d for d in (-4097, -1, 0, 1)] + [3 * CDF_CHUNK + 5]
        for first, count in cdf_ranges(n, firsts) + [(CDF_CHUNK - 1, CDF_CHUNK + 2)]:
            part = s.compute_state_cumulative_distribution(first, count)
            assert np.array_equal(part, cdf[first:first + count]), (first, count)


# ------------------------------------------------------------------------------------- downloads, upload

def transfer_ranges(N):
    """(first, count) at and around 256-index export runs, the download pipeline half (2^21 fp64 / 2^22 f32 items),
    the upload chunk (2^22) and the probabilities chunk (2^23)."""
    big = [c + d for c in (1 << 21, 1 << 22, 1 << 23) for d in (-1, 0, 1)]
    pairs = [(f, c) for f in (0, 1, 255, 256, 257) for c in (1, 255, 256, 257)]
    pairs += [(f, c) for f in (0, 1, 257) for c in big]
    pairs += [(f, c) for f in big for c in (1, 257, (1 << 21) + 1)]
    return [(f, c) for f, c in pairs if f + c <= N]


@PRECS
def test_downloads_probabilities_and_upload_across_chunks(prec):
    n = 24
    N = 1 << n
    a = random_state(n, seed=5)
    ref = as_stored(a, prec)
    native = (a.astype(np.complex64) if prec == F32 else a).view(np.float32 if prec == F32 else np.float64)
    p_ref = ref.real ** 2 + ref.imag ** 2
    with permuted(n, prec) as s:
        s.set_state(a)
        assert np.array_equal(s.state(), ref)
        for first, count in transfer_ranges(N):
            assert np.array_equal(s.state(first, count), ref[first:first + count]), (first, count)
            assert np.array_equal(s.state_native(first, count), native[2 * first:2 * (first + count)]), (first, count)
            p = s.probabilities(first, count)
            w = p_ref[first:first + count]
            assert np.all(np.abs(p - w) <= 1e-15 * w), (first, count)
        assert np.array_equal(logical_from_physical(s, n), ref)

    b = random_state(n, seed=6)
    cur = as_stored(b, prec).copy()
    with permuted(n, prec) as s:
        s.set_state(b)
        for first, count in transfer_ranges(N):
            s.set_state(a[first:first + count], first)
            cur[first:first + count] = ref[first:first + count]
            lo, hi = max(first - 1, 0), min(first + count + 1, N)        # the neighbours keep their values
            assert np.array_equal(s.state(lo, hi - lo), cur[lo:hi]), (first, count)
        assert np.array_equal(s.state(), cur)
        assert np.array_equal(logical_from_physical(s, n), cur)


# ------------------------------------------------------------------------------------------------- sampler

@PRECS
def test_sampler_over_several_launches(prec):
    """150 000 shots are three k_draw launches of at most 65 535 CTAs; every shot is checked, and the first 1000
    equal a 1000-shot call with the same seed."""
    n, shots_n, seed = 10, 150_000, 31
    rs = uniforms(seed, shots_n)
    for k in (0, 1, 999, 65534, 65535, 65536, 131069, 131070, 131071, shots_n - 1):
        assert rs[k] == q.sample_uniform(seed, k)
    with permuted(n, prec) as s:
        cdf = s.compute_state_cumulative_distribution()
        shots = s.measurement(shots_n, seed=seed)
        head = s.measurement(1000, seed=seed)
    check_shots(shots, cdf, n, seed, rs=rs)
    assert np.array_equal(shots[:1000], head)


@PRECS
def test_sampler_clamps_draws_beyond_a_subnormalised_total(prec):
    """Norm 0.5 and the last 100 amplitudes zero: about half of the draws exceed the total, and the reference's
    rule then returns the last index although its probability is 0."""
    n, shots_n, seed = 14, 4000, 8
    N = 1 << n
    a = random_state(n, seed=14)
    a[-100:] = 0.0
    a *= np.sqrt(0.5) / np.linalg.norm(a)
    rs = uniforms(seed, shots_n)
    with permuted(n, prec) as s:
        s.set_state(a)
        cdf = s.compute_state_cumulative_distribution()
        shots = s.measurement(shots_n, seed=seed)
    beyond = rs > cdf[-1]
    assert 1500 < int(beyond.sum()) < 2500
    for k in np.flatnonzero(beyond):
        assert oracle_measure(cdf, n, float(rs[k])) == N - 1
        assert int(shots[k]) == N - 1, (k, rs[k], cdf[-1])
    check_shots(shots[~beyond], cdf, n, seed, rs=rs[~beyond])
    assert int(shots[~beyond].max()) < N - 100


# ------------------------------------------------------------------------------------- expectation values

def diag_strings(n, qubits=None, weights=(2, 3)):
    qubits = range(n) if qubits is None else qubits
    return [" ".join(f"Z{k}" for k in c) for w in weights for c in itertools.combinations(qubits, w)]


def low_weight_strings(n, max_weight):
    """Every Pauli string of weight <= max_weight."""
    out = [""]
    for w in range(1, max_weight + 1):
        for qs in itertools.combinations(range(n), w):
            for letters in itertools.product("XYZ", repeat=w):
                out.append(" ".join(f"{p}{k}" for p, k in zip(letters, qs)))
    return out


def near_all_x_strings(n, max_changes):
    """Every string that differs from X on every qubit in at most max_changes positions (each I, Y or Z): their X
    masks have more high bits than a tile holds, so these take the paired path of tiles t and t ^ x_out."""
    out = []
    for w in range(max_changes + 1):
        for qs in itertools.combinations(range(n), w):
            for letters in itertools.product("IYZ", repeat=w):
                sub = dict(zip(qs, letters))
                out.append(" ".join(f"{sub.get(k, 'X')}{k}" for k in range(n) if sub.get(k, "X") != "I"))
    return out


def check_alone_and_shuffled(s, batch, got, prec, seed):
    """Each value equals the term evaluated alone and the same term in a shuffled batch (to TOL: launches of other
    sizes run other CTA counts, so the partial sums are grouped differently)."""
    tol = TOL[prec]
    alone = np.array([s.expectation(t) for t in batch])
    assert np.max(np.abs(alone - got)) <= tol
    order = np.random.default_rng(seed).permutation(len(batch))
    shuffled = s.expectation([batch[i] for i in order])
    assert np.max(np.abs(shuffled - got[order])) <= tol


@PRECS
def test_expectation_batches_of_several_launches(prec):
    """One sweep holding 512, 513, 1024 and 1300 diagonal terms; groups of 688 and 792 terms that share one X mask
    each, in tile (X3 X9) and across tiles (X on qubits 0..12, more high bits than a tile holds: the paired path).
    The dry run counts launches, so it shows that every batch but the first takes two or more.  How a sweep splits
    into launches depends on the term count alone, so 16 qubits do, and keep the numpy reference of every term cheap."""
    n = 16
    diag = diag_strings(n, weights=(2, 3, 4))[:1300]                  # 120 pairs, 560 triples, then quadruples
    others = [k for k in range(n) if k not in (3, 9)]
    in_tile = [f"{p3}3 {p9}9 {z}".strip() for p3 in "XY" for p9 in "XY"
               for z in ([""] + diag_strings(n, others, (1, 2, 3)))[:172]]
    paired = [(" ".join(f"{'Y' if k in ys else 'X'}{k}" for k in range(13)) + " " + z).strip()
              for r in range(8) for ys in itertools.combinations(range(0, 13, 2), r)
              for z in [""] + diag_strings(n, range(13, 16), (1, 2, 3))][:792]
    assert len(diag) == 1300 and len(in_tile) == 688 and len(paired) == 792
    everything = diag + in_tile + paired
    cases = [(diag[:K], -(-K // EXP_KMAX)) for K in (512, 513, 1024, 1300)]
    cases += [(in_tile, 2), (paired, 2), (everything, 6)]            # diagonal and X3 X9 terms: one sweep, 4 launches
    with permuted(n, prec) as s:
        s.set_state(random_state(n, seed=20))
        want = dict(zip(everything, expect_np(s.state(), everything, n)))
        for batch, launches in cases:
            assert q.expectation_dry_run(n, batch, prec)["sweeps"] == launches
            got = s.expectation(batch)
            err = np.abs(got - np.array([want[t] for t in batch]))
            assert np.max(err) <= TOL[prec], (len(batch), float(np.max(err)), batch[int(np.argmax(err))])
        check_alone_and_shuffled(s, everything, got, prec, seed=3)


LOW_BITS = {F32: (0, 3, 6), F64: (0, 2, 5)}
EXHAUSTIVE = [(prec, n, low) for prec in (F32, F64) for n in ((12 if prec == F32 else 11), 13, 14, 16) for low in LOW_BITS[prec]]


@pytest.mark.parametrize("prec,n,low_bits", EXHAUSTIVE, ids=[f"f{p}-n{n}-low{lb}" for p, n, lb in EXHAUSTIVE])
def test_expectation_of_every_low_weight_string(prec, n, low_bits):
    """Every string of weight <= 2 and every string within two positions of X on all qubits; at the size where the
    tile is the whole shard also every string of weight 3.  13 and 14 qubits leave one or two bits outside the tile
    (nothing at low_bits 0 means the default)."""
    terms = low_weight_strings(n, 3 if n == (12 if prec == F32 else 11) else 2) + near_all_x_strings(n, 2)
    with permuted(n, prec, low_bits) as s:
        s.set_state(random_state(n, seed=1000 + n))
        got = s.expectation(terms)
        want = expect_np(s.state(), terms, n)
    err = np.abs(got - want)
    assert np.max(err) <= TOL[prec], (float(np.max(err)), terms[int(np.argmax(err))])


def tile_classes(prec, n):
    """Physical bits of the diagonal sweep's tile by role: f32 pack lane, thread bits, unit bits, then the bits
    outside the tile."""
    if prec == F32:
        return [range(0, 1), range(1, 8), range(8, 12), range(12, n)]
    return [range(0, 7), range(7, 11), range(11, n)]


@PRECS
def test_expectation_on_basis_states_is_exact(prec):
    """<j|Z..Z|j> = (-1)^popc(j & z) and <j|P|j> = +0.0 for any P with an X part, bit for bit."""
    n = 14
    N = 1 << n
    diagonal = [" ".join(f"Z{k}" for k in c) for w in range(3) for c in itertools.combinations(range(n), w)]
    diagonal.append(" ".join(f"Z{k}" for k in range(n)))
    flipping = [t for t in low_weight_strings(n, 2) if "X" in t or "Y" in t] + near_all_x_strings(n, 1)
    flipping += [" ".join(f"Y{k}" for k in range(n))]
    _, zmask = q.pauli_masks(diagonal, n)
    rng = np.random.default_rng(7)
    with permuted(n, prec) as s:
        perm = s.layout()[0]
        js = [0, N - 1]
        while len(js) < 6:                                            # random indices with a bit in every class
            j = int(rng.integers(1, N - 1))
            phys = {int(perm[k]) for k in range(n) if (j >> k) & 1}
            if all(phys.intersection(c) for c in tile_classes(prec, n)):
                js.append(j)
        for j in js:
            v = np.zeros(N, dtype=np.complex128)
            v[j] = 1.0
            s.set_state(v)
            want = np.array([-1.0 if bin(j & int(z)).count("1") % 2 else 1.0 for z in zmask])
            assert np.array_equal(bits_of(s.expectation(diagonal)), bits_of(want)), j
            assert np.array_equal(bits_of(s.expectation(flipping)), np.zeros(len(flipping), dtype=np.uint64)), j


@PRECS
def test_expectation_repeats_and_zero_state(prec):
    """Repeats of a string in a batch of <= 512 terms share its launch and return identical bits; an all-zero state
    gives +0.0 for every term."""
    n = 16
    distinct = random_terms(n, 120, seed=16)
    rng = np.random.default_rng(4)
    batch = [distinct[i] for i in rng.permutation(np.repeat(np.arange(len(distinct)), 4))]
    assert len(batch) <= EXP_KMAX
    with permuted(n, prec) as s:
        s.set_state(random_state(n, seed=16))
        got = s.expectation(batch)
        assert np.max(np.abs(got - expect_np(s.state(), batch, n))) <= TOL[prec]
        for t in distinct:
            at = [i for i, b in enumerate(batch) if b == t]
            assert len(set(bits_of(got[at]).tolist())) == 1, t
        s.set_state(np.zeros(1 << n))
        terms = low_weight_strings(n, 2) + distinct
        assert np.array_equal(bits_of(s.expectation(terms)), np.zeros(len(terms), dtype=np.uint64))
