"""Pattern compression of the nucleotide null: a column pattern that occurs at least MIN_RUN times among the two
simulated alignments of a batch is mapped once (CMB_NULL_DEDUP_MIN_RUN=2: every repeated one).  Raw null rows, bin
offsets and the sorted null equal the uncompressed run (CMB_NULL_DEDUP=0) bit for bit, the mapping walks exactly the
columns the rule gives, and a short hash (runs of equal hashes that mix different columns) changes nothing but how
many columns are walked."""
import numpy as np
import pytest
import helpers as H

pytestmark = pytest.mark.gpu

# 262 145 sites per alignment: three replicates fill a batch of 2^20 sites, so four replicates run as two batches
REP_CPU, REP_RAM, SEED, K, NMAX = 4, 262145, 23, 4, 1.0
MIN_RUN = 16  # capi_stats.cu kMinMergedRun


@pytest.fixture(scope="module")
def ctx():
    from comap_b200 import api
    c = api.Context()
    yield c
    c.close()


def _setup(ctx, T, seed):
    # short branches on few taxa: a few hundred column patterns, most of them varied, repeat over and over
    c = H.random_dna_case(T, 100, seed, mean_brlen=0.05, C=4)
    ctx.set_tree(c["parent"], c["brlen"])
    ctx.set_model(c["Q"], c["pi"], c["rates"], c["probs"])
    ctx.set_alignment(c["codes"], c["code_mask"])
    ctx.map()


def _run(ctx, monkeypatch, env, fn):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ctx.profile_reset()
    raw = fn()
    out = (raw, ctx.null_get(), ctx.profile_get("sites_simulated")[0], ctx.profile_get("sites_mapped_null")[0])
    for k in env:
        monkeypatch.delenv(k)
    return out


def _assert_same(a, b):
    assert np.array_equal(a[0], b[0], equal_nan=True)
    assert np.array_equal(a[1]["bin_offsets"], b[1]["bin_offsets"])
    assert np.array_equal(a[1]["sorted"], b[1]["sorted"], equal_nan=True)
    assert a[2] == b[2] == 2 * REP_CPU * REP_RAM


def _alignments(ctx):
    s1 = np.stack([ctx.simulate(SEED, (2 * i) * REP_RAM, REP_RAM)[0] for i in range(REP_CPU)])
    s2 = np.stack([ctx.simulate(SEED, (2 * i + 1) * REP_RAM, REP_RAM)[0] for i in range(REP_CPU)])
    return s1, s2


def _walked_per_batch(s1, s2, min_run):
    """Columns mapped per batch of replicates (both alignments together), summed over the batches: one per
    pattern that occurs at least min_run times in the batch, every column of the rarer ones."""
    rpb = (1 << 20) // REP_RAM
    total = 0
    for r0 in range(0, REP_CPU, rpb):
        cols = np.concatenate([s[r] for r in range(r0, min(REP_CPU, r0 + rpb)) for s in (s1, s2)], axis=1)
        rows = np.ascontiguousarray(cols.T).view(np.dtype((np.void, cols.shape[0])))
        counts = np.unique(rows, return_counts=True)[1]
        total += int(np.where(counts >= min_run, 1, counts).sum())
    return total


@pytest.mark.parametrize("T", [10, 37])
def test_repeated_columns_mapped_once(ctx, monkeypatch, T):
    """T = 10 (one packed word) and 37 (three, the last one partial); device simulation, discrete and continuous
    rates, and the same alignments from the host, over two batches per call."""
    _setup(ctx, T, 40 + T)
    try:
        for cont in (False, True):
            if cont:
                ctx.set_continuous_rates("gamma", 0.7)
            s1, s2 = _alignments(ctx)
            distinct = _walked_per_batch(s1, s2, 2)
            assert distinct < 0.5 * 2 * REP_CPU * REP_RAM                      # duplicates dominate
            dev = lambda: ctx.null_intra("correlation", SEED, REP_CPU, REP_RAM, K=K, nmax=NMAX, want_raw=True)
            host = lambda: ctx.null_intra_from_alignments("correlation", s1, s2, K=K, nmax=NMAX)
            ref = _run(ctx, monkeypatch, {"CMB_NULL_DEDUP": "0"}, dev)
            assert ref[3] == ref[2]                                             # uncompressed: every column walked
            for env, want in (({}, _walked_per_batch(s1, s2, MIN_RUN)), ({"CMB_NULL_DEDUP_MIN_RUN": "2"}, distinct)):
                for fn in (dev, host):
                    got = _run(ctx, monkeypatch, env, fn)
                    _assert_same(ref, got)
                    assert got[3] == want
    finally:
        ctx.set_continuous_rates("off")


def test_hash_collisions_cost_merges_not_results(ctx, monkeypatch):
    """CMB_NULL_DEDUP_HASH_BITS=3: eight runs of equal hashes, each holding many different columns.  A column joins
    its run's head only when their tips are equal, so the results stay bit-identical and the walked count rises above
    the distinct count.  The simulator's keys and k2_column_keys' keys of the same columns are the same: the host
    path walks exactly as many columns."""
    _setup(ctx, 12, 7)
    s1, s2 = _alignments(ctx)
    distinct = _walked_per_batch(s1, s2, 2)
    dev = lambda: ctx.null_intra("correlation", SEED, REP_CPU, REP_RAM, K=K, nmax=NMAX, want_raw=True)
    host = lambda: ctx.null_intra_from_alignments("correlation", s1, s2, K=K, nmax=NMAX)
    ref = _run(ctx, monkeypatch, {"CMB_NULL_DEDUP": "0"}, dev)
    walked = []
    for fn in (dev, host):
        got = _run(ctx, monkeypatch, {"CMB_NULL_DEDUP_HASH_BITS": "3", "CMB_NULL_DEDUP_MIN_RUN": "2"}, fn)
        _assert_same(ref, got)
        assert distinct < got[3] < got[2]
        walked.append(got[3])
    assert walked[0] == walked[1]
