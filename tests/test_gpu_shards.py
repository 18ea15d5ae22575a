"""Mica and the two-data-set null spread over GPUs: the permutation test by pair shard (cmb_mica_permutations_shard),
the parametric bootstrap and the inter-gene null by outer-replicate range (cmb_mica_null_parametric_range /
_sharded, cmb_null_inter_range), and `comap_b200.gpus=N` on the command line.  Every result must be the one-call
result bit for bit: the shuffles and the simulators are keyed by global pair / site indices."""
import os
import subprocess
import sys
import threading
import numpy as np
import pytest
import helpers as H
from test_host import BIN, write_fixture, dry_run, decode

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(ctx, c):
    ctx.set_tree(c["parent"], c["brlen"])
    ctx.set_model(c["Q"], c["pi"], c["rates"], c["probs"])
    ctx.set_alignment(c["codes"], c["code_mask"])


def _dna_case():
    """tests/test_gpu_mica.py's A = 4 case: ambiguity codes, a column constant once unknowns are ignored, one all-unknown."""
    c = H.random_dna_case(26, 60, 11, mean_brlen=0.2, ambiguity=0.05)
    c["codes"][:, 7] = 2; c["codes"][3, 7] = 4
    c["codes"][:, 19] = 4
    return c


@pytest.fixture(scope="module")
def bacteria(tmp_path_factory):
    """examples/RNA/BacteriaSSU as options_perm.mica reads it: 760 sites x 40 taxa, the alignment's sequence order."""
    from comap_b200 import build as b
    b.build_host()
    tmp = str(tmp_path_factory.mktemp("ssu"))
    write_fixture(tmp, "bacteria_ssu")
    _, o = dry_run(BIN, tmp, "param=options_perm.mica")
    c = decode(o)
    row = {name: k for k, name in enumerate(o["leaves"])}
    c["codes"] = np.ascontiguousarray(c["codes"][[row[name] for name in o["sequences"]]])
    c["parent"] = c["parent"].astype(np.int32)
    return c


CASES = {"dna": (_dna_case, 300), "protein": (H.myoglobin_inputs, 60), "bacteria_ssu": (None, 1000)}


def _case(name, bacteria):
    make, max_perm = CASES[name]
    return (bacteria if make is None else make()), max_perm


def _union(ctxs, seed, max_perm, n_shards, n_pairs):
    """Every shard on its own context, rows scattered back to their pair index idx = shard + k * n_shards."""
    pv, nb = np.full(n_pairs, np.nan), np.full(n_pairs, -1, np.int32)
    for r in range(n_shards):
        p, n = ctxs[r].mica_permutations(seed, max_perm, shard_index=r, shard_count=n_shards)
        assert len(p) == len(range(r, n_pairs, n_shards))
        pv[r::n_shards] = p; nb[r::n_shards] = n
    return pv, nb


@pytest.mark.parametrize("name", ["dna", "protein", "bacteria_ssu"])
def test_permutation_shards_equal_the_whole_table(name, bacteria):
    from comap_b200 import api
    c, max_perm = _case(name, bacteria)
    ctxs = [api.Context(device=0) for _ in range(8)]
    for ctx in ctxs:
        _load(ctx, c)
    S = c["codes"].shape[1]
    n_pairs = S * (S - 1) // 2
    pv, nb = ctxs[0].mica_permutations(4242, max_perm)
    assert nb.max() > 0
    for n_shards in (1, 2, 3, 8):
        upv, unb = _union(ctxs, 4242, max_perm, n_shards, n_pairs)
        assert np.array_equal(upv, pv) and np.array_equal(unb, nb), n_shards
    for ctx in ctxs:
        ctx.close()


FILTER_OFF = r"""
import sys, numpy as np
sys.path.insert(0, %(root)r); sys.path.insert(0, %(tests)r)
from comap_b200 import api
d = np.load(%(case)r)
ctxs = [api.Context(device=0) for _ in range(3)]
S = d["codes"].shape[1]; n = S * (S - 1) // 2
pv, nb = np.full(n, np.nan), np.full(n, -1, np.int32)
for r, ctx in enumerate(ctxs):
    ctx.set_tree(d["parent"], d["brlen"]); ctx.set_model(d["Q"], d["pi"], d["rates"], d["probs"])
    ctx.set_alignment(d["codes"], d["code_mask"])
    p, k = ctx.mica_permutations(4242, int(d["max_perm"]), shard_index=r, shard_count=3)
    pv[r::3] = p; nb[r::3] = k
np.savez(%(out)r, pv=pv, nb=nb)
"""


@pytest.mark.parametrize("name", ["dna", "bacteria_ssu"])
def test_permutation_shards_without_the_interval_filter(name, bacteria, tmp_path):
    """CMB_K5_FILTER=0 (read once per process) sends every shuffle through the reference's formula: the union of three
    shards must still be the filtered one-call table, so the filter's tie path does not depend on the shard."""
    from comap_b200 import api
    c, max_perm = _case(name, bacteria)
    ctx = api.Context(device=0)
    _load(ctx, c)
    pv, nb = ctx.mica_permutations(4242, max_perm)
    ctx.close()
    case, out = str(tmp_path / "case.npz"), str(tmp_path / "out.npz")
    np.savez(case, max_perm=max_perm, **{k: c[k] for k in ("parent", "brlen", "Q", "pi", "rates", "probs", "codes", "code_mask")})
    script = FILTER_OFF % dict(root=ROOT, tests=os.path.join(ROOT, "tests"), case=case, out=out)
    p = subprocess.run([sys.executable, "-c", script], env=dict(os.environ, CMB_K5_FILTER="0"), capture_output=True, text=True,
                       timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    r = np.load(out)
    assert np.array_equal(r["pv"], pv) and np.array_equal(r["nb"], nb)


def test_empty_and_bad_permutation_shards():
    from comap_b200 import api
    c = H.random_dna_case(12, 3, 5, mean_brlen=0.3)        # 3 sites: 3 pairs
    ctx = api.Context(device=0)
    _load(ctx, c)
    pv, nb = ctx.mica_permutations(9, 100)
    for r in range(5):
        p, n = ctx.mica_permutations(9, 100, shard_index=r, shard_count=5)
        if r < 3:
            assert len(p) == 1 and p[0] == pv[r] and n[0] == nb[r]
        else:
            assert len(p) == 0 and len(n) == 0
    for si, sc in ((5, 5), (7, 5), (0, 0), (0, -2), (-1, 3)):
        with pytest.raises(RuntimeError, match="bad shard"):
            ctx.mica_permutations(9, 100, shard_index=si, shard_count=sc)
    ctx.close()


def test_parametric_null_ranges_concatenate():
    from comap_b200 import api
    c = H.random_dna_case(20, 70, 9, mean_brlen=0.12)
    ctx = api.Context(device=0)
    _load(ctx, c)
    ctx.map()
    rep_cpu, rep_ram, K = 7, 150, 4
    whole = ctx.mica_null_parametric(17, rep_cpu, rep_ram, K=K)
    g1 = ctx.null_get()
    p1 = ctx.mica_pairs("nmin", use_null=True)
    parts = [ctx.mica_null_parametric(17, rep_cpu, rep_ram, K=K, rep_begin=a, rep_end=b) for a, b in ((0, 2), (2, 3), (3, 7))]
    assert [len(p) for p in parts] == [2 * rep_ram, rep_ram, 4 * rep_ram]
    assert np.array_equal(np.concatenate(parts), whole)
    with pytest.raises(RuntimeError, match="bad replicate range"):
        ctx.mica_null_parametric(17, rep_cpu, rep_ram, rep_begin=3, rep_end=8)
    # without a communicator the sharded entry point is the whole null: same bins, same sorted samples, same p-values
    ctx.mica_null_parametric_sharded(17, rep_cpu, rep_ram, K=K)
    g2 = ctx.null_get()
    assert g1["K"] == g2["K"] and g1["nmax"] == g2["nmax"]
    assert np.array_equal(g1["bin_offsets"], g2["bin_offsets"]) and np.array_equal(g1["sorted"], g2["sorted"])
    p2 = ctx.mica_pairs("nmin", use_null=True)
    assert np.array_equal(p1["pvalue"], p2["pvalue"], equal_nan=True) and np.array_equal(p1["nsim"], p2["nsim"])
    ctx.close()


@pytest.mark.parametrize("stat,weighted", [("correlation", False), ("corrected_correlation", False), ("correlation", True)])
def test_inter_null_ranges_concatenate(stat, weighted):
    from comap_b200 import api
    c1 = H.random_dna_case(18, 80, 3, mean_brlen=0.1)
    c2 = dict(c1, codes=H.random_dna_case(18, 50, 4, mean_brlen=0.1)["codes"])
    a, b = api.Context(device=0), api.Context(device=0)
    _load(a, c1); _load(b, c2)
    a.map(); b.map()
    rep_cpu, rep_ram = 7, 120
    whole = a.null_inter(b, stat, 23, rep_cpu, rep_ram, weighted_classes=weighted)
    parts = [a.null_inter(b, stat, 23, rep_cpu, rep_ram, weighted_classes=weighted, rep_begin=x, rep_end=y)
             for x, y in ((0, 2), (2, 3), (3, 7))]
    assert np.array_equal(np.concatenate(parts), whole, equal_nan=True)
    a.close(); b.close()


def _two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")


def test_two_gpu_parametric_null_equals_one_gpu():
    """Two contexts joined by cmb_comm_init_all, rep_cpu = 5: shards of 3 and 2 replicates, so the all-gather carries
    NaN padding.  The union's bins, sorted samples and the table's p-values equal the one-context null."""
    _two_gpus()
    from comap_b200 import api
    c = H.random_dna_case(20, 90, 9, mean_brlen=0.12)
    rep_cpu, rep_ram, K = 5, 130, 4

    def setup(dev):
        ctx = api.Context(device=dev)
        _load(ctx, c)
        ctx.map(want_vectors=False)
        return ctx

    one = setup(0)
    whole = one.mica_null_parametric(31, rep_cpu, rep_ram, K=K)
    g1, p1 = one.null_get(), one.mica_pairs("nmin", use_null=True)
    ctxs = [setup(0), setup(1)]
    api.comm_init_all(ctxs)
    raws, err = [None, None], []

    def work(r):
        try:
            raws[r] = ctxs[r].mica_null_parametric_sharded(31, rep_cpu, rep_ram, K=K, want_raw=True)
        except Exception as e:  # noqa: BLE001
            err.append(e)

    th = [threading.Thread(target=work, args=(r,)) for r in range(2)]
    [t.start() for t in th]; [t.join() for t in th]
    assert not err, err
    assert [len(x) for x in raws] == [3 * rep_ram, 2 * rep_ram] and np.array_equal(np.concatenate(raws), whole)
    for ctx in ctxs:
        g2, p2 = ctx.null_get(), ctx.mica_pairs("nmin", use_null=True)
        assert np.array_equal(g1["bin_offsets"], g2["bin_offsets"]) and np.array_equal(g1["sorted"], g2["sorted"])
        assert np.array_equal(p1["pvalue"], p2["pvalue"], equal_nan=True) and np.array_equal(p1["nsim"], p2["nsim"])
    for ctx in ctxs + [one]:
        ctx.close()


def _run(cwd, *args, prog=BIN):
    p = subprocess.run([prog] + list(args), cwd=cwd, capture_output=True, text=True)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]


def _same(tmp, a, b):
    assert open(os.path.join(tmp, a), "rb").read() == open(os.path.join(tmp, b), "rb").read(), a


def test_two_gpu_command_lines_write_the_same_files(tmp_path):
    _two_gpus()
    from comap_b200 import build as b
    b.build_host()
    mica = os.path.join(os.path.dirname(BIN), "mica_b200")
    tmp = str(tmp_path)
    write_fixture(tmp, "bacteria_ssu")
    for n in (1, 2):
        _run(tmp, "param=options_perm.mica", "--seed=21", "output.file=perm%d.txt" % n, "comap_b200.gpus=%d" % n, prog=mica)
        _run(tmp, "param=options_pbs.mica", "--seed=21", "output.file=pbs%d.txt" % n, "null.output.file=pbs_null%d.txt" % n,
             "null.nb_rep_CPU=5", "comap_b200.gpus=%d" % n, prog=mica)
    _same(tmp, "perm1.txt", "perm2.txt")
    _same(tmp, "pbs1.txt", "pbs2.txt")
    _same(tmp, "pbs_null1.txt", "pbs_null2.txt")
    write_fixture(tmp, "myoglobin")
    common = ["param=comap.bpp", "input.sequence.file=Myoglobin.aln.sel.mase", "input.tree.file=Myo.dnd", "nijt=Uniformization",
              "--seed=11", "analysis=pairwise", "input.sequence.file2=Myoglobin.aln.sel.mase", "statistic.min_rate_class2=2",
              "statistic.min=0.2", "statistic.null=yes", "statistic.null.nb_rep_CPU=5", "statistic.null.nb_rep_RAM=150"]
    for stat in ("Correlation", "CorrectedCorrelation"):
        for n in (1, 2):
            _run(tmp, *common, "statistic=" + stat, "statistic.output.file=inter%d.txt" % n,
                 "statistic.null.output.file=inter_null%d.txt" % n, "output.infos2=infos2_%d.txt" % n, "comap_b200.gpus=%d" % n)
        _same(tmp, "inter1.txt", "inter2.txt")
        _same(tmp, "inter_null1.txt", "inter_null2.txt")
        _same(tmp, "infos2_1.txt", "infos2_2.txt")
