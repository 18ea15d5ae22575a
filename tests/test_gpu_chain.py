"""The whole north_star chain against the oracle running ALONE (VERDICT r1, weak #1).

Every other p-value test hands the oracle the device's own vectors and sorted null.  Here the
only thing both sides share is the input: the observed alignment and the simulated alignments
(exported by cmb_simulate for the global site indices the device null uses).  The oracle then
maps, builds its own null distribution from its own vectors and scores the pairs against it
(CoETools.cpp:638-724, AnalysisTools.cpp:564-658); the device does the same with its RNG.

Compared: Stat 1e-9, Nmin / PRmin 1e-9, RCmin and Nsim exact, bin occupancy exact, and the
p-values: the NUMBER of rows whose p-value differs is reported, and every such row must be
explained by null samples within 1e-9 (relative) of the row's statistic -- K1 on the FP64
tensor cores sums in a different order than the oracle, so statistics differ in the last bits
and `#{sim < stat}` (CoETools.cpp:715) can move only where a null value ties with the statistic
at that precision.  The counts are printed and collected in chain_parity.json under pytest's temporary
directory (quoted in DESIGN.md s5).
"""
import json
import os

import numpy as np
import pytest
import helpers as H
import oracle_binding as O

pytestmark = pytest.mark.gpu
TIE = 1e-9


@pytest.fixture(scope="module")
def ctx():
    from comap_b200 import api
    c = api.Context()
    yield c
    c.close()


@pytest.fixture(scope="module")
def report(tmp_path_factory):
    return os.path.join(str(tmp_path_factory.mktemp("chain")), "chain_parity.json")


def _record(path, name, rec):
    try:
        cur = json.load(open(path))
    except Exception:
        cur = {}
    cur[name] = rec
    json.dump(cur, open(path, "w"), indent=1, sort_keys=True)


def _chain(ctx, report, c, stat, seed, rep_cpu, rep_ram, K, name):
    S = c["codes"].shape[1]
    ctx.set_tree(c["parent"], c["brlen"])
    ctx.set_model(c["Q"], c["pi"], c["rates"], c["probs"])
    ctx.set_alignment(c["codes"], c["code_mask"])
    ctx.map()
    # ---- device: its own RNG, its own vectors, its own null
    ctx.null_intra(stat, seed, rep_cpu, rep_ram, K=K, nmax=-1.0)
    g = ctx.null_get()
    gp, k = ctx.pairs(stat, use_null=True)
    # ---- the same simulated alignments, exported
    s1 = np.stack([ctx.simulate(seed, (2 * i) * rep_ram, rep_ram)[0] for i in range(rep_cpu)])
    s2 = np.stack([ctx.simulate(seed, (2 * i + 1) * rep_ram, rep_ram)[0] for i in range(rep_cpu)])
    # ---- oracle alone
    q = O.map_sites(c["parent"], c["brlen"], c["Q"], c["pi"], c["rates"], c["probs"], c["codes"], c["code_mask"])
    if stat == "corrected_correlation":
        O.mean_vector(q["n"])
    nmax = float(q["norm"].max())
    on = O.null_intra(c["parent"], c["brlen"], c["Q"], c["pi"], c["rates"], c["probs"], stat, s1, s2, K, nmax)
    op = O.pairs(stat, q["n"], q["norm"], q["post_rate"], q["rate_class"],
                 null=(K, nmax, on["bin_offsets"], on["sorted"]))
    # ---- compare
    assert k == len(op["i"]) == S * (S - 1) // 2
    assert np.array_equal(gp["i"], op["i"]) and np.array_equal(gp["j"], op["j"])
    nan = np.isnan(op["stat"])
    assert np.array_equal(np.isnan(gp["stat"]), nan)
    assert np.allclose(gp["stat"][~nan], op["stat"][~nan], rtol=1e-9, atol=1e-12)
    assert np.allclose(gp["nmin"], op["nmin"], rtol=1e-9) and np.allclose(gp["prmin"], op["prmin"], rtol=1e-9)
    assert np.array_equal(gp["rcmin"], op["rcmin"])
    assert abs(g["nmax"] - nmax) <= 1e-9 * nmax
    assert np.array_equal(g["bin_offsets"], on["bin_offsets"]), "null bin occupancy differs"
    assert np.array_equal(gp["nsim"], op["nsim"]), "Nsim differs"
    fin = ~np.isnan(on["sorted"])
    assert np.array_equal(np.isnan(g["sorted"]), ~fin)
    assert np.allclose(g["sorted"][fin], on["sorted"][fin], rtol=1e-9, atol=1e-12)
    pv_nan = np.isnan(op["pvalue"])
    assert np.array_equal(np.isnan(gp["pvalue"]), pv_nan)
    diff = np.flatnonzero(~pv_nan & (gp["pvalue"] != op["pvalue"]))
    exact_stat = int(np.sum(gp["stat"][~nan] == op["stat"][~nan]))
    # every differing row: the two counts bracket only null values tied with the statistic at 1e-9
    worst = 0
    w = (nmax / K)
    for r in diff:
        cat = O.domain_index(0, nmax, K, float(op["nmin"][r]))
        lo, hi = on["bin_offsets"][cat], on["bin_offsets"][cat + 1]
        sim = on["sorted"][lo:hi]
        st = float(op["stat"][r])
        tol = TIE * max(abs(st), 1e-3)
        c_lo = int(np.searchsorted(sim, st - tol, side="left"))
        c_hi = int(np.searchsorted(sim, st + tol, side="right"))
        nsim = hi - lo
        cnt_dev = nsim + 1 - gp["pvalue"][r] * (nsim + 1)
        cnt_orc = nsim + 1 - op["pvalue"][r] * (nsim + 1)
        assert c_lo - 0.5 <= cnt_dev <= c_hi + 0.5 and c_lo - 0.5 <= cnt_orc <= c_hi + 0.5, \
            "row %d: p-value differs without a tie (stat %r, counts %r / %r, tie window %d..%d)" % (r, st, cnt_dev, cnt_orc, c_lo, c_hi)
        worst = max(worst, int(round(abs(cnt_dev - cnt_orc))))
    rec = dict(statistic=stat, sites=int(S), pairs=int(k), null_samples=int(rep_cpu * rep_ram), bins=int(K),
               pvalue_rows_compared=int((~pv_nan).sum()), pvalue_mismatches=int(len(diff)),
               largest_count_shift=int(worst), stat_bit_identical_rows=exact_stat, stat_rows=int((~nan).sum()),
               every_mismatch_is_a_tie_within=TIE, nsim_exact=True, bin_occupancy_exact=True)
    _record(report, name, rec)
    print("chain parity %s: %s" % (name, json.dumps(rec)))
    return rec


@pytest.mark.parametrize("stat", ["correlation", "compensation", "cosubstitution"])
def test_chain_dna_oracle_alone(ctx, report, stat):
    c = H.random_dna_case(24, 150, 11, mean_brlen=0.08, C=4)
    rec = _chain(ctx, report, c, stat, seed=99, rep_cpu=4, rep_ram=500, K=6, name="dna_24x150_" + stat)
    # a mismatch needs null values within 1e-9 of the statistic (asserted row by row in _chain): pairs of
    # near-constant sites, whose statistics tie in exact arithmetic (r = 1) and are ordered by rounding alone
    assert rec["pvalue_mismatches"] <= 0.25 * rec["pvalue_rows_compared"]
    if stat == "cosubstitution":
        assert rec["pvalue_mismatches"] == 0  # integer statistic: no last-bit differences


def test_chain_myoglobin_oracle_alone(ctx, report):
    """Protein path (A = 20): the reference's Myoglobin benchmark inputs, pairwise correlation + null."""
    m = H.myoglobin_inputs()
    rec = _chain(ctx, report, m, "correlation", seed=7, rep_cpu=3, rep_ram=300, K=5, name="myoglobin_129_correlation")
    assert rec["pvalue_mismatches"] <= 0.25 * rec["pvalue_rows_compared"]


def test_null_with_100_bins_vs_oracle(ctx):
    """statistic.null.nb_rate_classes >= 64 (ADVICE r1: the offsets kernel only filled 64 bins)."""
    c = H.random_dna_case(16, 120, 5, mean_brlen=0.08, C=4)
    ctx.set_tree(c["parent"], c["brlen"]); ctx.set_model(c["Q"], c["pi"], c["rates"], c["probs"])
    ctx.set_alignment(c["codes"], c["code_mask"])
    r = ctx.map()
    rep_cpu, rep_ram, K = 3, 400, 100
    s1 = np.stack([ctx.simulate(3, (2 * i) * rep_ram, rep_ram)[0] for i in range(rep_cpu)])
    s2 = np.stack([ctx.simulate(3, (2 * i + 1) * rep_ram, rep_ram)[0] for i in range(rep_cpu)])
    nmax = float(r["norm"].max())
    ctx.null_intra_from_alignments("correlation", s1, s2, K=K, nmax=nmax)
    o = O.null_intra(c["parent"], c["brlen"], c["Q"], c["pi"], c["rates"], c["probs"], "correlation", s1, s2, K, nmax)
    g = ctx.null_get()
    assert g["K"] == K and len(g["bin_offsets"]) == K + 1
    assert np.array_equal(g["bin_offsets"], o["bin_offsets"])
    gp, k = ctx.pairs("correlation", use_null=True)
    op = O.pairs("correlation", r["n"], r["norm"], r["post_rate"], r["rate_class"],
                 null=(K, nmax, g["bin_offsets"], g["sorted"]))
    assert np.array_equal(gp["nsim"], op["nsim"])
    a, b = gp["pvalue"], op["pvalue"]
    assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)])


def test_saturated_site_is_refused(ctx):
    """A site whose likelihood underflows to 0 must not yield NaN vectors silently (CoETools.cpp:233-262):
    cmb_map fails, naming the number of such sites, instead of returning NaN vectors."""
    from comap_b200 import synthetic as syn
    T = 1400                                      # saturated branches: L ~ 4^-1400 underflows fp64
    parent, brlen = syn.random_tree(T, 3, 2.0)
    brlen = np.maximum(brlen, 50.0)
    Q, pi = syn.hky85(2.5, [0.3, 0.2, 0.2, 0.3])
    rates, probs = syn.gamma_rates(0.5, 4)
    ctx.set_tree(parent, brlen); ctx.set_model(Q, pi, rates, probs)
    codes = np.random.default_rng(0).integers(0, 4, size=(T, 64)).astype(np.uint8)
    ctx.set_alignment(codes, syn.identity_code_mask(4))
    with pytest.raises(RuntimeError, match="likelihood is 0"):
        ctx.map()
    with pytest.raises(RuntimeError):             # and nothing downstream runs on it
        ctx.pairs("correlation", use_null=False)
