"""The tree step (metrify + UPGMA, ``snacc_upgma``) on matrices with ties: scipy's linkage matrix bit for bit.

An NCD is a ratio of integer compressed sizes, so real matrices have many equal entries: genomes of similar length,
duplicated genomes, near-identical ones.  With ties, the order in which merges are made decides the tree, not only
the order of its rows.  scipy's average linkage runs ``nn_chain``: a nearest-neighbour chain walked from the first
active cluster, merged clusters kept in the higher slot, the merges sorted stably by height and relabelled by a
union-find (``label``).  ``scipy_nn_chain`` below restates that; it is the specification the device kernel follows,
and the CPU tests pin it to scipy itself so that a change of scipy's tie rules shows up here first.
``global_min_linkage`` restates the textbook rule (merge the globally closest pair), which builds the same tree when
there are no ties; it is a witness that the tie families below really do separate the two rules.

The GPU tests (-m gpu) compare the device with scipy exactly: every column of Z with ``np.array_equal`` and the
Newick string of the reference.
"""
import json
import os

import numpy as np
import pytest

from oracle import snacc_oracle, tree_oracle


# ---- the two rules, restated --------------------------------------------------------------------------------------

def scipy_nn_chain(D):
    """scipy.cluster.hierarchy.linkage(squareform(D), "average"): nn_chain, the stable sort by height, label()"""
    D = np.array(D, dtype=np.float64)
    n = D.shape[0]
    size = [1] * n
    chain = []
    raw = []
    for _ in range(n - 1):
        if not chain:
            chain.append(next(i for i in range(n) if size[i]))
        while True:
            x = chain[-1]
            if len(chain) > 1:
                y = chain[-2]
                cur = D[x, y]
            else:
                cur = np.inf
            for i in range(n):
                if size[i] and i != x and D[x, i] < cur:          # strict: ties keep the earlier candidate
                    cur, y = D[x, i], i
            if len(chain) > 1 and y == chain[-2]:
                break
            chain.append(y)
        del chain[-2:]
        x, y = min(x, y), max(x, y)
        nx, ny = size[x], size[y]
        raw.append((x, y, cur, nx + ny))
        size[x], size[y] = 0, nx + ny                             # the merged cluster lives in the higher slot
        for i in range(n):
            if size[i] and i != y:
                D[i, y] = D[y, i] = (nx * D[i, x] + ny * D[i, y]) / (nx + ny)
    Z = np.array(raw, dtype=np.float64)
    Z = Z[np.argsort(Z[:, 2], kind="mergesort")]
    parent = list(range(2 * n - 1))
    count = [1] * (2 * n - 1)

    def find(a):
        while parent[a] != a:
            a = parent[a]
        return a

    for k in range(n - 1):
        a, b = find(int(Z[k, 0])), find(int(Z[k, 1]))
        Z[k, 0], Z[k, 1] = min(a, b), max(a, b)
        parent[a] = parent[b] = n + k
        count[n + k] = count[a] + count[b]
        Z[k, 3] = count[n + k]
    return Z


def global_min_linkage(D):
    """merge the globally closest pair (ties: smallest row, then smallest column), the merged cluster keeps the lower
    slot; not scipy's rule once there are ties"""
    D = np.array(D, dtype=np.float64)
    n = D.shape[0]
    active = np.ones(n, dtype=bool)
    size = np.ones(n, dtype=np.int64)
    label = list(range(n))
    Z = np.zeros((n - 1, 4))
    for t in range(n - 1):
        best = (np.inf, -1, -1)
        for a in range(n):
            if not active[a]:
                continue
            for b in range(a + 1, n):
                if active[b] and D[a, b] < best[0]:
                    best = (D[a, b], a, b)
        h, a, b = best
        Z[t] = (min(label[a], label[b]), max(label[a], label[b]), h, size[a] + size[b])
        for k in range(n):
            if active[k] and k != a and k != b:
                D[k, a] = D[a, k] = (size[a] * D[k, a] + size[b] * D[k, b]) / (size[a] + size[b])
        size[a] += size[b]
        label[a] = n + t
        active[b] = False
    return Z


def names(n):
    return [f"genome_{i}.fasta" for i in range(n)]


def has_newick(Z):
    """scipy's to_tree, and so the reference's Newick writer, refuses negative heights (linkage accepts them)"""
    return bool((Z[:, 2] >= 0).all())


def same_tree(Z, Zref):
    """exact equality of the whole linkage matrix and of the reference's Newick string"""
    n = Z.shape[0] + 1
    return np.array_equal(Z, Zref) and (not has_newick(Zref) or
                                        tree_oracle.newick(Z, names(n)) == tree_oracle.newick(Zref, names(n)))


# ---- tie families: each returns the matrix before metrify (the reference clusters metrify(D)) ----------------------

def _tree_extra(n, rng, scale):
    """a tree-like integer extra for S: the genomes are joined pairwise in random order at integer heights that grow
    by 0 .. scale per join; the extra of a pair is the height at which the two met (small, so that many pairs tie)"""
    X = np.zeros((n, n), dtype=np.int64)
    groups = [[i] for i in range(n)]
    h = 0
    while len(groups) > 1:
        i, j = sorted(rng.choice(len(groups), 2, replace=False))
        h += int(rng.integers(0, scale + 1))
        X[np.ix_(groups[i], groups[j])] = h
        X[np.ix_(groups[j], groups[i])] = h
        groups[i] = groups[i] + groups[j]
        del groups[j]
    return X


def ncd_sizes(n, seed):
    """C in [1000, 1012), S = max(C_i, C_j) + a tree-like extra, S(i, j) and S(j, i) apart by at most one"""
    rng = np.random.default_rng(seed)
    C = rng.integers(1000, 1012, n)
    S = np.maximum(C[:, None], C[None, :]) + _tree_extra(n, rng, 3) + rng.integers(0, 2, (n, n))
    np.fill_diagonal(S, C + 2)
    return C, S


def ncd_vectorised(C, S, bias=snacc_oracle.GETSIZEOF_BIAS):
    """snacc_oracle.ncd_from_sizes as whole-array numpy (the same correctly rounded divisions), for large n"""
    C = np.asarray(C, dtype=np.int64) + bias
    S = np.asarray(S, dtype=np.int64) + bias
    lo = np.minimum(C[:, None], C[None, :]).astype(np.float64)
    hi = np.maximum(C[:, None], C[None, :]).astype(np.float64)
    return np.minimum((S - lo) / hi, (S.T - lo) / hi)


def ncd_family(n, seed):
    """(a) NCD from integer sizes in a narrow range"""
    return snacc_oracle.ncd_from_sizes(*ncd_sizes(n, seed))


def duplicated_family(n, seed):
    """(b) genomes duplicated once and twice: rows and columns copied in C and S before the NCD"""
    rng = np.random.default_rng(seed)
    m = max(2, n - 3)
    C = rng.integers(5000, 5400, m)
    S = np.maximum(C[:, None], C[None, :]) + rng.integers(50, 400, (m, m))
    np.fill_diagonal(S, C + 3)
    src = list(range(m)) + [int(rng.integers(0, m))] * 2 + [int(rng.integers(0, m))]
    src = np.array(src[:n])
    rng.shuffle(src)
    return snacc_oracle.ncd_from_sizes(C[src], S[np.ix_(src, src)])     # a copy and its twin: S(x, x)


def quantised_family(n, seed):
    """(c) values quantised to 0.1"""
    return np.round(np.random.default_rng(seed).random((n, n)), 1)


def constant_family(n, seed):
    """(d) every off-diagonal entry equal"""
    D = np.full((n, n), 0.7 + 0.01 * (seed % 7))
    np.fill_diagonal(D, 0.0)
    return D


def zeros_family(n, seed):
    """(e) exact-zero off-diagonal distances (identical genomes) among a few small values"""
    return np.random.default_rng(seed).integers(0, 3, (n, n)) * 0.25


def negative_family(n, seed):
    """(f) negative entries, which scipy accepts"""
    return np.round(np.random.default_rng(seed).random((n, n)) - 0.3, 1)


FAMILIES = {"ncd": ncd_family, "duplicated": duplicated_family, "quantised": quantised_family,
            "constant": constant_family, "zeros": zeros_family, "negative": negative_family}


# ---- CPU: the specification against scipy -------------------------------------------------------------------------

@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_nn_chain_restatement_equals_scipy_bit_for_bit(family):
    for n in range(2, 14):
        for seed in range(12):
            D = tree_oracle.metrify(FAMILIES[family](n, seed))
            assert np.array_equal(scipy_nn_chain(D), tree_oracle.hierarchical(D)), (family, n, seed)


@pytest.mark.parametrize("n", [40, 100])
def test_nn_chain_restatement_equals_scipy_on_larger_ncd_matrices(n):
    for seed in range(3):
        D = tree_oracle.metrify(ncd_family(n, seed))
        assert np.array_equal(scipy_nn_chain(D), tree_oracle.hierarchical(D)), (n, seed)


@pytest.mark.parametrize("family", ["ncd", "quantised"])
def test_global_minimum_rule_differs_from_scipy_on_ties(family):
    """the tie families are strong enough to tell the two rules apart: in ids or in the Newick string"""
    differ = 0
    for n in range(3, 14):
        for seed in range(12):
            D = tree_oracle.metrify(FAMILIES[family](n, seed))
            differ += not same_tree(global_min_linkage(D), tree_oracle.hierarchical(D))
    assert differ > 0


def test_global_minimum_rule_agrees_with_scipy_without_ties():
    """the witness itself is right where the rules must agree: points in general position"""
    rng = np.random.default_rng(5)
    for n in (2, 5, 17):
        pts = rng.random((n, 4))
        D = np.sqrt(((pts[:, None] - pts[None, :]) ** 2).sum(-1))
        Z, Zref = global_min_linkage(D), tree_oracle.hierarchical(D)
        assert np.array_equal(Z[:, [0, 1, 3]], Zref[:, [0, 1, 3]])
        assert np.allclose(Z[:, 2], Zref[:, 2], rtol=1e-12, atol=0)


def test_families_have_ties_at_the_minimum():
    """each family really has equal distances: some row's two smallest off-diagonal entries are equal"""
    for family, make in FAMILIES.items():
        D = tree_oracle.metrify(make(12, 0)) + np.diag(np.full(12, np.inf))
        two = np.sort(D, axis=1)[:, :2]
        assert (two[:, 0] == two[:, 1]).any(), family


def test_vectorised_ncd_equals_the_oracle():
    C, S = ncd_sizes(60, 3)
    assert np.array_equal(ncd_vectorised(C, S), snacc_oracle.ncd_from_sizes(C, S))


# ---- GPU: the device tree against scipy, exactly ------------------------------------------------------------------

def _assert_device_equals_scipy(engine, D):
    """both entry points (metrify on the device, and UPGMA of the host-metrified matrix) give scipy's Z bit for bit
    and the reference's Newick string"""
    from snacc_b200 import distmatrix_to_tree as d2t
    D_sym = tree_oracle.metrify(D)
    Zref = tree_oracle.hierarchical(D_sym)
    Z = d2t.linkage_from_distances(D, engine=engine)
    bad = np.flatnonzero((Z != Zref).any(axis=1))
    assert bad.size == 0, (D.shape[0], bad[:5].tolist(), Z[bad[:3]].tolist(), Zref[bad[:3]].tolist())
    assert np.array_equal(d2t.hierarchical(D_sym, engine=engine), Zref)
    n = D.shape[0]
    if has_newick(Zref):
        assert d2t.newick_from_linkage(Z, names(n)) == tree_oracle.newick(Zref, names(n))


@pytest.mark.gpu
@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_device_tree_equals_scipy_on_tie_families(engine, family):
    for n in (2, 3, 4, 5, 8, 13, 40, 100, 300):
        for seed in range(4 if n < 100 else 2):
            _assert_device_equals_scipy(engine, FAMILIES[family](n, seed))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 3, 1023, 1024, 1025, 2049])
def test_device_tree_equals_scipy_where_the_thread_loops_wrap(engine, n):
    """n around the 1024 threads and 32 warps of the one CTA"""
    C, S = ncd_sizes(n, n)
    _assert_device_equals_scipy(engine, ncd_vectorised(C, S))
    _assert_device_equals_scipy(engine, quantised_family(n, n))


@pytest.mark.gpu
def test_device_tree_equals_scipy_on_a_tie_heavy_matrix_of_c3_size(engine):
    """10 000 genomes, as in the c3 configuration"""
    C, S = ncd_sizes(10_000, 7)
    _assert_device_equals_scipy(engine, ncd_vectorised(C, S))


def _mutants(genomes, rng):
    """exact duplicates and 1 to 3 point mutants of some of the genomes, mixed in among them"""
    out = list(genomes)
    for i in rng.choice(len(genomes), 6, replace=False):
        out.append(genomes[i].copy())
    for i in rng.choice(len(genomes), 8, replace=False):
        g = genomes[i].copy()
        for p in rng.choice(g.size, int(rng.integers(1, 4)), replace=False):
            g[p] = np.frombuffer(b"ACGT", np.uint8)[(b"ACGT".index(bytes([g[p]])) + 1) % 4]
        out.append(g)
    perm = rng.permutation(len(out))
    return [out[k] for k in perm]


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["lz4", "gzip"])
def test_device_tree_equals_scipy_on_the_engine_ncd_of_near_identical_genomes(engine, algo):
    """the real pipeline: c3-shaped genomes (about 10.7 kbp) with duplicates and point mutants, NCD on the device"""
    from snacc_b200 import synth
    rng = np.random.default_rng(11)
    genomes = _mutants(synth.phylogeny(24, 10_700, seed=31, sub_rate=0.002), rng)
    n = len(genomes)
    engine.upload_sequences(genomes)
    C = engine.single_sizes(algo)
    S = engine.tile_sizes(algo, 0, n, 0, n)
    D = engine.ncd(C, S)
    assert np.array_equal(D, snacc_oracle.ncd_from_sizes(C, S))
    D_sym = tree_oracle.metrify(D)
    upper = D_sym[np.triu_indices(n, 1)]
    assert np.unique(upper).size < upper.size                          # ties, as duplicated genomes give
    _assert_device_equals_scipy(engine, D)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["lz4", "lz4_rc", "gzip", "gzip_rc", "zlib", "zlib_rc"])
def test_device_tree_equals_scipy_on_golden_sizes_with_duplicates(engine, golden_dir, case):
    """the reference's sizes of the 9 golden files, two of them duplicated (a copy against its twin: S(x, x))"""
    ref = json.load(open(os.path.join(golden_dir, "reference_sizes.json")))
    bias = ref["bias"]
    C = np.array(ref["cases"][case]["C"]) - bias
    S = np.array(ref["cases"][case]["S"]) - bias
    n = C.size
    for dup in ([2, 3], [4, 4], [0, 8]):
        src = np.array(list(range(n)) + dup)
        D = snacc_oracle.ncd_from_sizes(C[src], S[np.ix_(src, src)], bias)
        _assert_device_equals_scipy(engine, D)


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["nan", "inf", "neg_inf", "nonfinite_after_metrify"])
def test_upgma_rejects_nonfinite_input(engine, what):
    """scipy's linkage refuses non-finite distances with ValueError; so does the device path, before clustering"""
    from snacc_b200 import distmatrix_to_tree as d2t
    D = tree_oracle.metrify(quantised_family(6, 1))
    if what == "nonfinite_after_metrify":
        D[1, 4], D[4, 1] = np.inf, -np.inf                                # metrify: 0.5 (inf - inf) = nan
    else:
        D[1, 4] = D[4, 1] = {"nan": np.nan, "inf": np.inf, "neg_inf": -np.inf}[what]
    with pytest.raises(ValueError):
        tree_oracle.hierarchical(tree_oracle.metrify(D))
    with pytest.raises(ValueError, match="finite"):
        d2t.linkage_from_distances(D, engine=engine)
    if what != "nonfinite_after_metrify":
        with pytest.raises(ValueError, match="finite"):
            d2t.hierarchical(D, engine=engine)
    _assert_device_equals_scipy(engine, quantised_family(6, 1))       # the context still works


@pytest.mark.gpu
def test_upgma_rejects_what_squareform_rejects(engine):
    """with metrify off the matrix must be symmetric with a zero diagonal, as squareform checks; with metrify on the
    diagonal is zeroed first, so even a NaN there is accepted, as in the reference"""
    from snacc_b200 import distmatrix_to_tree as d2t
    D = tree_oracle.metrify(quantised_family(7, 2))
    asym = D.copy()
    asym[2, 5] += 0.1
    diag = D.copy()
    diag[3, 3] = 0.5
    nan_diag = D.copy()
    nan_diag[3, 3] = np.nan
    for bad, word in ((asym, "symmetric"), (diag, "diagonal"), (nan_diag, "diagonal")):
        with pytest.raises(ValueError):
            tree_oracle.hierarchical(bad)
        with pytest.raises(ValueError, match=word):
            d2t.hierarchical(bad, engine=engine)
    assert np.array_equal(d2t.linkage_from_distances(nan_diag, engine=engine),
                          tree_oracle.hierarchical(tree_oracle.metrify(nan_diag)))
    assert np.array_equal(d2t.linkage_from_distances(asym, engine=engine),
                          tree_oracle.hierarchical(tree_oracle.metrify(asym)))


@pytest.mark.gpu
def test_upgma_rejects_fewer_than_two_genomes(engine):
    from snacc_b200 import distmatrix_to_tree as d2t
    for D in (np.zeros((1, 1)), np.zeros((0, 0)), np.zeros((2, 3)), np.zeros(4)):
        with pytest.raises(ValueError):
            d2t.linkage_from_distances(D, engine=engine)
