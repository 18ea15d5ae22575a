"""GPU parity of K1 (likelihood + substitution mapping) against the CPU oracle, through
the C ABI.  Tolerance: 1e-9 relative on mapping vectors (north_star), fp64."""
import numpy as np
import pytest
import helpers as H
import oracle_binding as O
from comap_b200 import synthetic as syn

pytestmark = pytest.mark.gpu
RTOL = 1e-9


@pytest.fixture(scope="module")
def ctx():
    from comap_b200 import api
    c = api.Context()
    yield c
    c.close()


def _setup(ctx, c):
    ctx.set_tree(c["parent"], c["brlen"])
    ctx.set_model(c["Q"], c["pi"], c["rates"], c["probs"])
    ctx.set_alignment(c["codes"], c["code_mask"])


def _check(r, q, atol=1e-14):
    assert np.allclose(r["n"], q["n"], rtol=RTOL, atol=atol)
    assert np.allclose(r["norm"], q["norm"], rtol=RTOL)
    assert np.allclose(r["loglik"], q["loglik"], rtol=1e-12)
    assert np.allclose(r["post_rate"], q["post_rate"], rtol=RTOL)
    assert np.array_equal(r["rate_class"], q["rate_class"])


@pytest.mark.parametrize("T,S,seed,amb", [(3, 1, 1, 0.0), (5, 40, 1, 0.0), (12, 300, 2, 0.1), (40, 777, 3, 0.02),
                                          (200, 513, 4, 0.0)])
def test_map_dna_vs_oracle(ctx, T, S, seed, amb):
    c = H.random_dna_case(T, S, seed, ambiguity=amb)
    _setup(ctx, c)
    r = ctx.map()
    q = O.map_sites(c["parent"], c["brlen"], c["Q"], c["pi"], c["rates"], c["probs"], c["codes"], c["code_mask"])
    _check(r, q)


@pytest.mark.parametrize("C", [1, 2, 3, 6, 7, 8])
def test_map_dna_class_counts(ctx, C):
    """Every rate-class count the tensor-core kernels are instantiated for (1..8), with gaps."""
    c = H.random_dna_case(17, 260, 10 + C, C=C, ambiguity=0.05)
    _setup(ctx, c)
    r = ctx.map()
    q = O.map_sites(c["parent"], c["brlen"], c["Q"], c["pi"], c["rates"], c["probs"], c["codes"], c["code_mask"])
    _check(r, q)


def test_map_dna_deep_tree(ctx):
    """500 taxa (the bench tree shape): message stack several levels deep, cherries, long walks."""
    c = H.random_dna_case(500, 300, 20251018, mean_brlen=0.02)
    _setup(ctx, c)
    r = ctx.map()
    q = O.map_sites(c["parent"], c["brlen"], c["Q"], c["pi"], c["rates"], c["probs"], c["codes"], c["code_mask"])
    _check(r, q)


def test_map_invariant_five_classes(ctx):
    """GTR + Invariant(Gamma4): C = 5 with a rate-0 class -> two class blocks (4 + 1)."""
    parent, brlen = syn.random_tree(30, 7, 0.1)
    Q, pi = syn.gtr(1.6, 0.55, 0.35, 0.30, 0.28, [0.25, 0.2, 0.3, 0.25])
    rates, probs = syn.invariant(*syn.gamma_rates(0.737, 4), p=0.3666)
    codes = H.simulate_np(parent, brlen, Q, pi, rates, np.random.default_rng(5), 400)
    mask = syn.identity_code_mask(4)
    ctx.set_tree(parent, brlen); ctx.set_model(Q, pi, rates, probs); ctx.set_alignment(codes, mask)
    r = ctx.map()
    q = O.map_sites(parent, brlen, Q, pi, rates, probs, codes, mask)
    _check(r, q)


def test_map_multifurcations(ctx):
    """Polytomies are binarised internally with virtual zero-length edges."""
    parent = np.array([6, 6, 6, 6, 7, 7, 9, 9, 9, -1], np.int32)  # leaf 8 attaches to the root too
    brlen = np.array([0.1, 0.2, 0.05, 0.3, 0.15, 0.02, 0.2, 0.1, 0.4, 0.0])
    Q, pi = syn.hky85(2.0, [0.3, 0.2, 0.2, 0.3])
    rates, probs = syn.gamma_rates(0.6, 4)
    rng = np.random.default_rng(0)
    codes = rng.integers(0, 4, (7, 100)).astype(np.uint8)
    mask = syn.identity_code_mask(4)
    ctx.set_tree(parent, brlen); ctx.set_model(Q, pi, rates, probs); ctx.set_alignment(codes, mask)
    r = ctx.map()
    q = O.map_sites(parent, brlen, Q, pi, rates, probs, codes, mask)
    _check(r, q)


def test_map_myoglobin_golden(ctx):
    """Protein path (A = 20) against the oracle AND the reference's golden vectors."""
    m = H.myoglobin_inputs()
    _setup(ctx, m)
    r = ctx.map()
    q = O.map_sites(m["parent"], m["brlen"], m["Q"], m["pi"], m["rates"], m["probs"], m["codes"], m["code_mask"])
    _check(r, q, atol=1e-16)
    gold = m["golden"]["vec_unif"].T
    rel = np.abs(r["n"] - gold) / np.abs(gold)
    assert np.median(rel) < 5e-6 and rel.max() < 1e-4
    assert np.all(np.abs(r["loglik"] - m["golden"]["infos_logl"]) <= 6e-6 * np.abs(m["golden"]["infos_logl"]))


@pytest.mark.parametrize("method,key", [("naive", "vec_naive"), ("naive", "vec_naive_grantham"), ("laplace", "vec_laplace"),
                                        ("uniformization", "vec_unif_grantham"), ("decomposition", "vec_decomp_grantham")])
def test_map_count_methods_and_weights_vs_reference_goldens(ctx, method, key):
    """nijt=Naive and the Grantham-weighted counts on the device against the oracle (1e-9) and against
    the reference's own golden vectors (examples/Proteins/Benchmark/CoMap/Myo_*.vec, printed precision)."""
    import os
    m = H.myoglobin_inputs()
    W = None
    if key.endswith("grantham"):
        path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "comap_b200", "data", "grantham.dat")
        W = np.array([[float(x) for x in ln.split()] for ln in open(path) if ln.strip() and not ln.startswith("#")])
    ctx.set_tree(m["parent"], m["brlen"])
    ctx.set_model(m["Q"], m["pi"], m["rates"], m["probs"], count_method=method, weights=W)
    ctx.set_alignment(m["codes"], m["code_mask"])
    r = ctx.map()
    q = O.map_sites(m["parent"], m["brlen"], m["Q"], m["pi"], m["rates"], m["probs"], m["codes"], m["code_mask"],
                    method=method, weights=W)
    assert np.allclose(r["n"], q["n"], rtol=RTOL, atol=1e-15)
    gold = m["golden"][key].T
    big = gold > 1e-9
    rel = np.abs(r["n"] - gold)[big] / gold[big]
    # Laplace: the unconverged series amplifies the 2012 library's last digits on the longest branches (absolute bar)
    assert np.median(rel) < 5e-6 and (rel.max() < 3e-4 or (method == "laplace" and np.abs(r["n"] - gold).max() < 2e-5))
    if method == "laplace":  # Laplace(trunc=10) is the default order; weights are refused as Bio++ has none for it
        ctx.set_model(m["Q"], m["pi"], m["rates"], m["probs"], count_method=("laplace", 10))
        ctx.set_alignment(m["codes"], m["code_mask"])
        assert np.array_equal(ctx.map()["n"], r["n"])
        with pytest.raises(RuntimeError, match="Laplace"):
            ctx.set_model(m["Q"], m["pi"], m["rates"], m["probs"], count_method="laplace", weights=np.ones((20, 20)))


def test_errors_are_reported(ctx):
    from comap_b200 import api
    c2 = api.Context()
    with pytest.raises(RuntimeError, match="cmb_set_alignment"):
        c2.lib.cmb_map  # symbol exists
        c2._chk(c2.lib.cmb_map(c2.h, None, None, None, None, None))
    with pytest.raises(RuntimeError, match="post-order"):
        c2.set_tree(np.array([1, 0, -1], np.int32), np.array([0.1, 0.1, 0.0]))
    c2.close()


def _variant_mismatch(r, q):
    """Entries of two mappings that differ beyond 1e-9: for the variants that pick a most probable state or pair,
    device and oracle tables differ in the last bits (different eigen-solvers), so an arg-max between two states
    of (numerically) equal probability may fall the other way."""
    bad = ~np.isclose(r, q, rtol=RTOL, atol=1e-14)
    return int(bad.sum()), bad


@pytest.mark.parametrize("average,joint", [(True, False), (False, True), (False, False)])
def test_map_variants_vs_oracle(ctx, average, joint):
    """nijt.average = no / nijt.joint = no (CoETools.cpp:393-407): ...Marginal, ...NoAveraging and
    ...NoAveragingMarginal on the device (k1_variants.cu) against the oracle's restatement, nucleotides with
    unknown characters and polytomies, and the Myoglobin proteins; likelihood columns are those of the normal path."""
    cases = [H.random_dna_case(14, 333, 7, ambiguity=0.05), H.random_dna_case(60, 130, 8, C=3), H.myoglobin_inputs()]
    try:
        for c in cases:
            _setup(ctx, c)
            ctx.set_map_mode(average, joint)
            r = ctx.map()
            O.set_map_mode(average, joint)
            q = O.map_sites(c["parent"], c["brlen"], c["Q"], c["pi"], c["rates"], c["probs"], c["codes"], c["code_mask"])
            nbad, bad = _variant_mismatch(r["n"], q["n"])
            if average:
                assert nbad == 0
            else:
                assert nbad <= 2e-4 * r["n"].size, nbad
            ok = ~bad.any(axis=1)
            assert np.allclose(r["norm"][ok], q["norm"][ok], rtol=RTOL)
            assert np.allclose(r["loglik"], q["loglik"], rtol=1e-12) and np.array_equal(r["rate_class"], q["rate_class"])
            # the variant really is another mapping, and switching back restores the tensor-core one
            O.set_map_mode()
            base = O.map_sites(c["parent"], c["brlen"], c["Q"], c["pi"], c["rates"], c["probs"], c["codes"], c["code_mask"])
            assert np.abs(q["n"] - base["n"]).max() > 1e-3
            ctx.set_map_mode()
            assert np.allclose(ctx.map()["n"], base["n"], rtol=RTOL, atol=1e-14)
    finally:
        O.set_map_mode()
        ctx.set_map_mode()


def test_label_counts_without_averaging_are_labels(ctx):
    """nijt=Label with nijt.average=no (what statistic=MI needs, CoETools.cpp:577-589): every entry of the mapping
    is the label of ONE substitution type, 0..A(A-1), on the device as in the oracle."""
    c = H.random_dna_case(20, 400, 11, mean_brlen=0.1)
    try:
        for joint in (True, False):
            ctx.set_tree(c["parent"], c["brlen"])
            ctx.set_model(c["Q"], c["pi"], c["rates"], c["probs"], count_method="label")
            ctx.set_alignment(c["codes"], c["code_mask"])
            ctx.set_map_mode(False, joint)
            r = ctx.map()
            O.set_map_mode(False, joint)
            q = O.map_sites(c["parent"], c["brlen"], c["Q"], c["pi"], c["rates"], c["probs"], c["codes"], c["code_mask"], method="label")
            lab = np.rint(r["n"])
            assert np.abs(r["n"] - lab).max() < 1e-9 and lab.min() == 0 and 1 <= lab.max() <= 12 and (lab > 0).mean() > 0.01
            assert (np.rint(q["n"]) != lab).sum() <= 2e-4 * lab.size
    finally:
        O.set_map_mode()
        ctx.set_map_mode()


def test_prob_one_jump_count_on_the_device(ctx):
    """nijt=ProbOneJump (OneJumpSubstitutionCount): device vs oracle, nucleotides and proteins."""
    for c in (H.random_dna_case(30, 280, 41, ambiguity=0.03), H.myoglobin_inputs()):
        ctx.set_tree(c["parent"], c["brlen"])
        ctx.set_model(c["Q"], c["pi"], c["rates"], c["probs"], count_method="one_jump")
        ctx.set_alignment(c["codes"], c["code_mask"])
        r = ctx.map()
        q = O.map_sites(c["parent"], c["brlen"], c["Q"], c["pi"], c["rates"], c["probs"], c["codes"], c["code_mask"], method="one_jump")
        assert np.allclose(r["n"], q["n"], rtol=RTOL, atol=1e-14)
        assert r["n"].min() >= -1e-12 and r["n"].max() <= 1 + 1e-12     # every entry is a probability


def test_marginal_ancestral_states_vs_oracle(ctx):
    """asr.method = marginal (CoMap.cpp:168-198): state of largest marginal posterior at every node, device vs oracle;
    the leaves of resolved columns come back as observed."""
    for c in (H.random_dna_case(25, 300, 31, ambiguity=0.04), H.myoglobin_inputs()):
        _setup(ctx, c)
        ctx.map()
        a = ctx.ancestral_states()
        q = O.ancestral_states(c["parent"], c["brlen"], c["Q"], c["pi"], c["rates"], c["probs"], c["codes"], c["code_mask"])
        assert a.shape == q.shape == (len(c["parent"]), c["codes"].shape[1])
        assert (a != q).mean() < 2e-4
        has_child = np.zeros(len(c["parent"]), bool); has_child[c["parent"][c["parent"] >= 0]] = True
        leaves = a[~has_child]
        A = len(c["pi"])
        res = c["codes"] < A
        assert np.array_equal(leaves[res], c["codes"][res])
        assert a.max() < A and len(np.unique(a[has_child])) > 1
