"""Every launch shape of the mapping pass (K1) against the CPU oracle.

The K1 launchers pick a template instance at run time from the batch size, the rate-class count C, the down
pass' message-stack depth, the shared memory that fits and whether the batch was simulated on the device
(STATES).  Each test here records, with torch.profiler, which instances its calls launched, asserts that they
are the ones it is about, and compares the result with the oracle (1e-9, rate_class exact) or bit for bit with
another shape.  The last test checks that the file as a whole ran every instance the launchers can select on
this device, except those listed in NOT_RUN with the reason they are not reached."""
import contextlib
import json
import os
import re
import subprocess
import sys
import tempfile
import textwrap

import numpy as np
import pytest
import oracle_binding as O
from comap_b200 import synthetic as syn

pytestmark = pytest.mark.gpu
RTOL = 1e-9
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ------------------------------------------------------------------------------------------ kernel recorder
_K1 = re.compile(r"\b(k1_\w+?)(<[^()]*>)?\(")
SEEN = set()          # every K1 instance this module launched (subprocesses included)


def instance_of(kernel_name):
    """'void cmb::(anonymous namespace)::k1_up_mma<2, 4, 128, 2, false>(...)' -> 'k1_up_mma<2,4,128,2,false>'."""
    m = _K1.search(kernel_name)
    return None if m is None else m.group(1) + (m.group(2) or "").replace(" ", "")


def parse_instance(inst):
    """'k1_up_mma<2,4,128,2,false>' -> ('k1_up_mma', (2, 4, 128, 2, False))."""
    name, _, args = inst.partition("<")
    conv = {"true": True, "false": False}
    return name, tuple(conv[a] if a in conv else int(a) for a in args.rstrip(">").split(",") if a)


class Launches(list):
    """(instance, shared memory bytes) of every K1 kernel launched inside `recorded()`; `others`: the rest."""

    def __init__(self, *a):
        super().__init__(*a)
        self.others = []

    def __repr__(self):
        return "Launches(%s, others=%s)" % (list.__repr__(self), self.others)

    def instances(self, prefix=""):
        return {i for i, _ in self if i.startswith(prefix)}

    def args(self, kernel):
        return {parse_instance(i)[1] for i, _ in self if parse_instance(i)[0] == kernel}

    def smem(self, kernel):
        return {s for i, s in self if parse_instance(i)[0] == kernel}


@contextlib.contextmanager
def recorded(ctx=None):
    """Runs the body under torch.profiler (CUDA activity) and fills the yielded Launches from its trace.

    On a B200 a library kernel was twice missing from the trace, both times the first kernel of its window, so
    each window opens with a small torch kernel and a device synchronisation before the library runs.  With `ctx`, the number of
    libcomap_b200 kernels in the trace must equal the launches the library counted (cmb_launch_count): a
    dropped launch fails the test instead of passing an assertion that some instance did not run."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    out = Launches()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        torch.ones(1, device="cuda").add_(1)
        torch.cuda.synchronize()
        n0 = ctx.launch_count() if ctx is not None else 0
        yield out
        torch.cuda.synchronize()
        n1 = ctx.launch_count() if ctx is not None else 0
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    for e in events:
        if e.get("cat") == "kernel":
            inst = instance_of(e.get("name", ""))
            if inst:
                out.append((inst, int(e.get("args", {}).get("shared memory", -1))))
            else:
                out.others.append(e.get("name", ""))
    SEEN.update(out.instances())
    if ctx is not None:
        lib = len(out) + sum("cmb::" in n for n in out.others)
        assert lib == n1 - n0, "the trace holds %d library kernels, the library launched %d: %r" % (lib, n1 - n0, out)


# ------------------------------------------------------------------------------------------ library rules
def pad_sites(n):
    """capi.cu pad_sites: 256-site blocks, an odd number of them."""
    blocks = (n + 255) // 256
    return (blocks + (blocks % 2 == 0)) * 256


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def narrow_max():
    """Largest site count k1_mma.cu narrow_batch() maps in 32-site CTAs: n_pad / 128 < #SMs."""
    s = 256 * (sm_count() * 128 // 256)
    while pad_sites(s) // 128 >= sm_count():
        s -= 256
    return pad_sites(s)


def down_stack_depth(parent):
    """schedule.cpp build_tree: binarised tree, post-order with the larger child first, depth of the stack of
    messages that wait for their sibling (a restatement of lines 81-113)."""
    n = len(parent)
    kids = [[] for _ in range(n)]
    for v in range(n - 1):
        kids[parent[v]].append(v)
    left, right, par = [-1] * n, [-1] * n, [-1] * n
    for v in range(n):
        k = kids[v]
        if not k:
            continue
        cur = v
        for i in range(len(k) - 2):                      # k-ary node -> chain of binary nodes
            u = len(left)
            left.append(-1); right.append(-1); par.append(-1)
            left[cur], right[cur], par[k[i]], par[u] = k[i], u, cur, cur
            cur = u
        left[cur], right[cur], par[k[-2]], par[k[-1]] = k[-2], k[-1], cur, cur
    leaves = [0] * len(left)
    st = [(n - 1, 0)]
    while st:
        v, ph = st.pop()
        if left[v] < 0:
            leaves[v] = 1
        elif ph == 0:
            st += [(v, 1), (left[v], 0), (right[v], 0)]
        else:
            leaves[v] = leaves[left[v]] + leaves[right[v]]

    def larger_first(v):
        a, b = left[v], right[v]
        return (b, a) if leaves[b] > leaves[a] else (a, b)
    order, st = [], [(n - 1, 0)]
    while st:
        v, ph = st.pop()
        if left[v] < 0:
            continue
        if ph == 0:
            a, b = larger_first(v)
            st += [(v, 1), (b, 0), (a, 0)]
        else:
            order.append(v)
    sp = depth = 0
    for v in order:
        a, _ = larger_first(v)
        if left[a] >= 0:
            sp -= 1
        if v != n - 1 and larger_first(par[v])[0] == v:
            sp += 1
            depth = max(depth, sp)
    return depth


def balanced_tree(k, total_length=12.0):
    """Rooted balanced binary tree of 2^k leaves (down stack depth k - 1), ids in post-order.  The branches
    are short (total_length in all) so that no site likelihood underflows on thousands of taxa."""
    parent = []

    def build(level):
        if level == 0:
            parent.append(-1)
            return len(parent) - 1
        a, b = build(level - 1), build(level - 1)
        parent.append(-1)
        parent[a] = parent[b] = len(parent) - 1
        return len(parent) - 1
    build(k)
    p = np.array(parent, np.int32)
    return p, np.full(len(p), total_length / (len(p) - 1))


def caterpillar_tree(T, brlen=0.08):
    """Every inner node has a leaf child: no node of the up pass has two stored partials."""
    parent = [2, 2, -1]                  # post-order: leaf, leaf, inner, then (leaf, inner) pairs
    for _ in range(T - 2):
        parent += [-1, -1]
        parent[-3] = parent[-2] = len(parent) - 1
    p = np.array(parent, np.int32)
    return p, np.full(len(p), brlen)


# ------------------------------------------------------------------------------------------ comparisons
def _check_rows(r, q, idx=slice(None)):
    assert np.all(np.isfinite(q["loglik"]))
    assert np.allclose(r["n"][idx], q["n"], rtol=RTOL, atol=1e-14)
    assert np.allclose(r["norm"][idx], q["norm"], rtol=RTOL)
    assert np.allclose(r["loglik"][idx], q["loglik"], rtol=1e-12)
    assert np.allclose(r["post_rate"][idx], q["post_rate"], rtol=RTOL)
    assert np.array_equal(r["rate_class"][idx], q["rate_class"])


def _same(a, b):
    for k in ("n", "norm", "loglik", "post_rate", "rate_class"):
        assert np.array_equal(a[k], b[k]), k


def map_vs_oracle(ctx, m, codes, mask, n_sample=None, seed=0):
    """Maps `codes` on the device, compares all sites (or a seeded sample) with the oracle."""
    ctx.set_alignment(codes, mask)
    with recorded(ctx) as rec:
        r = ctx.map()
    S = codes.shape[1]
    idx = np.arange(S) if n_sample is None else np.sort(np.random.default_rng(seed).choice(S, n_sample, replace=False))
    q = O.map_sites(m["parent"], m["brlen"], m["Q"], m["pi"], m["rates"], m["probs"],
                    np.ascontiguousarray(codes[:, idx]), mask)
    _check_rows(r, q, idx)
    return r, rec


NULL_K, NULL_NMAX = 10, 40.0


def null_vs_oracle(ctx, m, seed, rep_cpu, rep_ram, reps, n=48):
    """Device-simulated null; replicates `reps` re-scored by the oracle on the alignments the device simulator
    exports for the same global site indices: statistic and Nmin 1e-9, bin of every row exact."""
    with recorded() as rec:
        raw = ctx.null_intra("correlation", seed, rep_cpu, rep_ram, K=NULL_K, nmax=NULL_NMAX, want_raw=True)
    g = ctx.null_get()
    bins = np.array([O.domain_index(0.0, NULL_NMAX, NULL_K, x) for x in raw[:, 3]])
    assert np.array_equal(np.concatenate([[0], np.cumsum(np.bincount(bins[bins >= 0], minlength=NULL_K))]),
                          g["bin_offsets"])
    for rep in reps:
        a = ctx.simulate(seed, (2 * rep) * rep_ram, n)[0]
        b = ctx.simulate(seed, (2 * rep + 1) * rep_ram, n)[0]
        o = O.null_intra(m["parent"], m["brlen"], m["Q"], m["pi"], m["rates"], m["probs"], "correlation",
                         a[None], b[None], NULL_K, NULL_NMAX)
        mine = raw[rep * rep_ram:rep * rep_ram + n]
        fin = ~np.isnan(o["raw"][:, 0])
        assert np.array_equal(fin, ~np.isnan(mine[:, 0]))
        assert np.allclose(mine[fin, 0], o["raw"][fin, 0], rtol=RTOL, atol=1e-12)
        assert np.allclose(mine[:, 3], o["raw"][:, 3], rtol=RTOL)
        assert np.array_equal(mine[:, 1], o["raw"][:, 1])
        mb = bins[rep * rep_ram:rep * rep_ram + n]
        ob = np.array([O.domain_index(0.0, NULL_NMAX, NULL_K, x) for x in o["raw"][:, 3]])
        assert np.array_equal(mb, ob)
    return raw, rec


def set_model(ctx, m):
    ctx.set_tree(m["parent"], m["brlen"])
    ctx.set_model(m["Q"], m["pi"], m["rates"], m["probs"])


def dna_model(parent, brlen, C):
    Q, pi = syn.hky85(2.5, [0.3, 0.2, 0.2, 0.3])
    rates, probs = syn.gamma_rates(0.5, C)
    return dict(parent=parent, brlen=brlen, Q=Q, pi=pi, rates=rates, probs=probs)


def protein_model(parent, brlen, C):
    Q, pi = syn.jtt92()
    if C == 5:
        rates, probs = syn.invariant(*syn.gamma_rates(0.8, 4), p=0.2)
    elif C == 1:
        rates, probs = np.ones(1), np.ones(1)
    else:
        rates, probs = syn.gamma_rates(0.8, C)
    return dict(parent=parent, brlen=brlen, Q=Q, pi=pi, rates=rates, probs=probs)


def with_ambiguity(codes, frac, seed, unknown=4):
    rng = np.random.default_rng(seed)
    return np.where(rng.random(codes.shape) < frac, unknown, codes).astype(np.uint8)


@pytest.fixture(scope="module")
def ctx():
    from comap_b200 import api
    c = api.Context()
    yield c
    c.close()


DNA_MASK = syn.identity_code_mask(4)
PROT_MASK = syn.identity_code_mask(20)


# ------------------------------------------------------------------------------------------ A = 4
def test_recorder_lists_the_library_kernels(ctx):
    """CUPTI through torch.profiler sees the kernels libcomap_b200.so launches on its own runtime and stream."""
    m = dna_model(*syn.random_tree(12, 4, 0.1), 4)
    set_model(ctx, m)
    codes = O.simulate(m["parent"], m["brlen"], m["Q"], m["pi"], m["rates"], m["probs"], 1, 0, 40)[0]
    _, rec = map_vs_oracle(ctx, m, codes, DNA_MASK)
    assert rec.instances("k1_down_mma<") == {"k1_down_mma<2,4,32,2,false>"}, rec
    assert rec.instances("k1_up_mma<") == {"k1_up_mma<2,4,32,2,false>"}, rec
    assert "k1_finish" in rec.instances()


def test_observed_alignment_on_both_sides_of_the_narrow_threshold(ctx):
    """The largest narrow batch and the smallest wide one (18 688 / 18 689 sites on 148 SMs), HKY85 + Gamma4,
    2 % unknown characters; then the first 5000 sites alone (narrow) against the wide result, bit for bit:
    every site is computed by the same lane arithmetic whatever the CTA size, with no atomics."""
    nmax = narrow_max()
    assert pad_sites(nmax) // 128 < sm_count() <= pad_sites(nmax + 1) // 128
    m = dna_model(*syn.random_tree(20, 1618, 0.08), 4)
    set_model(ctx, m)
    sim = ctx.simulate(21, 0, nmax + 1)[0]
    codes = with_ambiguity(sim, 0.02, 5)
    r_n, rec_n = map_vs_oracle(ctx, m, np.ascontiguousarray(codes[:, :nmax]), DNA_MASK)
    assert rec_n.args("k1_down_mma") == {(2, 4, 32, 2, False)} and rec_n.args("k1_up_mma") == {(2, 4, 32, 2, False)}
    r_w, rec_w = map_vs_oracle(ctx, m, codes, DNA_MASK)
    assert rec_w.args("k1_down_mma") == {(2, 4, 128, 2, False)} and rec_w.args("k1_up_mma") == {(2, 4, 128, 2, False)}
    ctx.set_alignment(np.ascontiguousarray(codes[:, :5000]), DNA_MASK)
    with recorded() as rec:
        r5 = ctx.map()
    assert {a[2] for a in rec.args("k1_up_mma") | rec.args("k1_down_mma")} == {32}
    _same(r5, {k: v[:5000] for k, v in r_w.items()})
    _same(r5, {k: v[:5000] for k, v in r_n.items()})


# trees of the class-count sweep: down stack depth 2, 5 and 10, and one without inner-inner nodes in the up pass
def _sweep_trees():
    return {"shallow": syn.random_tree(20, 77, 0.08), "deep500": syn.random_tree(500, 20251018, 0.02),
            "balanced2048": balanced_tree(11), "caterpillar": caterpillar_tree(24)}


DEPTHS = {"shallow": 2, "deep500": 5, "balanced2048": 10, "caterpillar": 1}


@pytest.mark.parametrize("C", [1, 2, 3, 4, 5, 6, 7, 8])
def test_dna_class_counts_in_every_shape(ctx, C):
    """C = 1..8: narrow and wide observed mappings, narrow and wide device nulls, on trees whose down stack is
    2, 5 and 10 levels deep -- the wide MINB = 2, wide MINB = 1 and narrow MINB = 1 down passes and both wide
    up passes -- each against the oracle (all sites of small trees, a sample on the large ones)."""
    trees = _sweep_trees()
    S = narrow_max() + 1
    seen = Launches()
    for name, (parent, brlen) in trees.items():
        assert down_stack_depth(parent) == DEPTHS[name], name
        m = dna_model(parent, brlen, C)
        set_model(ctx, m)
        big = len(parent) > 100
        codes = with_ambiguity(ctx.simulate(100 + C, 0, S)[0], 0.02, C)
        _, rec = map_vs_oracle(ctx, m, codes, DNA_MASK, n_sample=48 if big else None, seed=C)
        assert {a[2:] for a in rec.args("k1_up_mma")} <= {(128, 2, False), (128, 1, False)}, rec
        assert {a[4] for a in rec.args("k1_down_mma")} == {False} and len(rec.args("k1_down_mma")) == 1, rec
        seen += rec
        _, rec = null_vs_oracle(ctx, m, 7 + C, 4, 2500, reps=(0, 3))
        assert {a[4] for a in rec.args("k1_up_mma") | rec.args("k1_down_mma")} == {True}, rec
        assert all(a[2] != 32 for a in rec.args("k1_up_mma")), rec
        seen += rec
        if name == "shallow":
            _, rec = map_vs_oracle(ctx, m, np.ascontiguousarray(codes[:, :300]), DNA_MASK)
            assert rec.args("k1_up_mma") == {(2, C, 32, 2, False)}, rec
            seen += rec
            _, rec = null_vs_oracle(ctx, m, 3, 2, 300, reps=(1,))
            assert rec.args("k1_up_mma") == {(2, C, 32, 2, True)}, rec
            seen += rec
    down = seen.args("k1_down_mma")
    # what the shared-memory arithmetic of try_down_mma gives for these depths (NOT_RUN lists the rest)
    want_down = {(128, 2)} | ({(128, 1)} if C >= 3 else set()) | ({(32, 1)} if C >= 6 else set())
    for states in (False, True):
        assert {a[2:4] for a in down if a[4] == states} >= want_down, (states, down)
    up = seen.args("k1_up_mma")
    assert (2, C, 128, 2, False) in up and ((2, C, 128, 1, False) in up) == (C >= 7), up
    assert (2, C, 64, 3, True) in up and ((2, C, 128, 1, True) in up) == (C == 8), up


def test_wide_null_with_and_without_pattern_compression(ctx, monkeypatch):
    """C = 4 and 8, wide device nulls (STATES = true; the 64-site up pass at C = 4, the 128-site one at C = 8):
    raw rows equal with CMB_NULL_DEDUP=0, and equal again when the same alignments come from the host
    (null_intra_from_alignments: STATES = false, wide)."""
    rep_cpu, rep_ram = 4, 2500
    for C in (4, 8):
        m = dna_model(*syn.random_tree(40, 9, 0.06), C)
        set_model(ctx, m)
        raw, rec = null_vs_oracle(ctx, m, 11, rep_cpu, rep_ram, reps=(1, 2))
        assert {a[4] for a in rec.args("k1_up_mma")} == {True}
        assert rec.args("k1_up_mma") == ({(2, 4, 64, 3, True)} if C == 4 else {(2, 8, 128, 1, True)}), rec
        monkeypatch.setenv("CMB_NULL_DEDUP", "0")
        raw0 = ctx.null_intra("correlation", 11, rep_cpu, rep_ram, K=NULL_K, nmax=NULL_NMAX, want_raw=True)
        monkeypatch.delenv("CMB_NULL_DEDUP")
        assert np.array_equal(raw0, raw, equal_nan=True)
        s1 = np.stack([ctx.simulate(11, (2 * i) * rep_ram, rep_ram)[0] for i in range(rep_cpu)])
        s2 = np.stack([ctx.simulate(11, (2 * i + 1) * rep_ram, rep_ram)[0] for i in range(rep_cpu)])
        with recorded() as rec:
            rawh = ctx.null_intra_from_alignments("correlation", s1, s2, K=NULL_K, nmax=NULL_NMAX)
        assert {a[2] for a in rec.args("k1_down_mma")} == {128} and {a[4] for a in rec.args("k1_up_mma")} == {False}, rec
        assert np.array_equal(rawh, raw, equal_nan=True)


# ------------------------------------------------------------------------------------------ A = 20
@pytest.mark.parametrize("C", [1, 2, 3, 5, 6, 7, 8])
def test_protein_class_counts(ctx, C):
    """JTT92 with C = 1, 2, 3, Invariant + Gamma4 (5), 6, 7, 8 on an 80-taxon tree: one CTA per class and
    64-site chunk, k1_sum_classes over the [C][B][S_pad] partials; 63, 64, 65 and 300 sites, then a device
    null, against the oracle."""
    m = protein_model(*syn.random_tree(80, 30 + C, 0.1), C)
    set_model(ctx, m)
    seen = Launches()
    for S in (63, 64, 65, 300):
        codes = O.simulate(m["parent"], m["brlen"], m["Q"], m["pi"], m["rates"], m["probs"], 40 + C, 0, S)[0]
        _, rec = map_vs_oracle(ctx, m, codes, PROT_MASK)
        seen += rec
    _, rec = null_vs_oracle(ctx, m, 5, 2, 64, reps=(0, 1))
    seen += rec
    assert seen.args("k1_down_mma20") == {(2, False), (2, True)}, seen
    assert seen.args("k1_up_mma20") == {(2, False), (2, True)}, seen
    assert "k1_sum_classes" in seen.instances()


@pytest.mark.parametrize("k,depth,C", [(11, 10, 2), (13, 12, 1), (14, 13, 1)])
def test_protein_down_stack_depth_switch(ctx, k, depth, C):
    """Balanced trees of 2^k taxa: down stack depth 10 runs k1_down_mma20 at one CTA per SM, 12 (the deepest the
    tensor-core path takes, capi.cu) still the tensor-core kernels, 13 the thread-per-site ones; 16 sites."""
    parent, brlen = balanced_tree(k)
    assert down_stack_depth(parent) == depth
    m = protein_model(parent, brlen, C)
    set_model(ctx, m)
    codes = ctx.simulate(3, 0, 16)[0]
    _, rec = map_vs_oracle(ctx, m, codes, PROT_MASK)
    if depth <= 12:
        assert rec.args("k1_down_mma20") == {(1 if depth >= 10 else 2, False)}, rec
        assert rec.args("k1_up_mma20") == {(2, False)} and not rec.instances("k1_down<"), rec
    else:
        assert rec.instances("k1_down<") == {"k1_down<20,1,0>"} and not rec.instances("k1_down_mma20"), rec
        assert rec.instances("k1_up<") == {"k1_up<20,1,192,1,0,0>"}, rec


@pytest.mark.parametrize("C", [4, 5, 8])
def test_protein_scalar_kernels(ctx, monkeypatch, C):
    """CMB_K1_PROTEIN=scalar (read when the model is set): k1_down<20,1,0> and k1_up<20,1,192,1>, which holds at
    most four classes -- C = 5 (Invariant + Gamma4) and 8 run it once per class block, the second block adding
    to the first's output.  CMB_DOWN_GLOBAL_TIPS=1 (read per launch) gives the same bits."""
    monkeypatch.setenv("CMB_K1_PROTEIN", "scalar")
    m = protein_model(*syn.random_tree(60, 50 + C, 0.1), C)
    set_model(ctx, m)
    codes = O.simulate(m["parent"], m["brlen"], m["Q"], m["pi"], m["rates"], m["probs"], 60 + C, 0, 200)[0]
    r, rec = map_vs_oracle(ctx, m, codes, PROT_MASK)
    assert rec.instances("k1_down") == {"k1_down<20,1,0>"} and rec.instances("k1_up") == {"k1_up<20,1,192,1,0,0>"}, rec
    assert sum(i.startswith("k1_up<") for i, _ in rec) == (1 if C <= 4 else 2), rec
    _, rec = null_vs_oracle(ctx, m, 9, 2, 100, reps=(1,))
    assert rec.instances("k1_down") == {"k1_down<20,1,0>"} and rec.instances("k1_up") == {"k1_up<20,1,192,1,0,0>"}, rec
    monkeypatch.setenv("CMB_DOWN_GLOBAL_TIPS", "1")
    ctx.set_alignment(codes, PROT_MASK)
    _same(ctx.map(), r)
    monkeypatch.delenv("CMB_K1_PROTEIN")
    monkeypatch.delenv("CMB_DOWN_GLOBAL_TIPS")
    set_model(ctx, m)                     # the tensor-core kernels again
    _, rec = map_vs_oracle(ctx, m, codes, PROT_MASK)
    assert rec.args("k1_down_mma20") == {(2, False)} and rec.args("k1_up_mma20") == {(2, False)}, rec
    assert not rec.instances("k1_up<") and not rec.instances("k1_down<"), rec


# ------------------------------------------------------------------------------------------ switches read once
SWITCH_SCRIPT = textwrap.dedent("""
    import json, sys
    import numpy as np
    sys.path[:0] = [{root!r}, {tests!r}]
    import test_gpu_k1_shapes as K
    from comap_b200 import api, synthetic as syn
    out = sys.argv[1]
    ctx = api.Context()
    m = K.dna_model(*syn.random_tree(20, 1618, 0.08), 4)
    K.set_model(ctx, m)
    codes = K.with_ambiguity(ctx.simulate(21, 0, K.narrow_max() + 1)[0], 0.02, 5)
    res, launches = {{}}, {{}}
    for case, cols in (("wide", codes), ("narrow", codes[:, :5000])):
        ctx.set_alignment(np.ascontiguousarray(cols), K.DNA_MASK)
        with K.recorded() as rec:
            r = ctx.map()
        launches[case] = rec
        res.update({{case + "_" + k: v for k, v in r.items()}})
    with K.recorded() as rec:
        res["null"] = ctx.null_intra("correlation", 11, 4, 2500, K=10, nmax=40.0, want_raw=True)
    launches["null"] = rec
    ctx.close()
    np.savez(out + ".npz", **res)
    json.dump({{k: list(v) for k, v in launches.items()}}, open(out + ".json", "w"))
""")

SWITCHES = {"default": {}, "narrow1": {"CMB_K1_NARROW": "1"}, "narrow0": {"CMB_K1_NARROW": "0"},
            "up_sg128": {"CMB_UP_SG": "128"}, "up_stages2": {"CMB_UP_STAGES": "2"}, "ring40": {"CMB_UP_RING_KB": "40"}}


def test_switches_read_once_per_process_leave_results_unchanged(tmp_path):
    """CMB_K1_NARROW, CMB_UP_SG, CMB_UP_STAGES and CMB_UP_RING_KB are read into statics on first use, so each
    setting runs in a fresh process: the same wide and narrow mappings and wide device null, bit for bit, while
    the recorder shows the instance or ring size each switch changes."""
    script = tmp_path / "run.py"
    script.write_text(SWITCH_SCRIPT.format(root=ROOT, tests=os.path.join(ROOT, "tests")))
    res, logs = {}, {}
    for name, extra in SWITCHES.items():
        env = {k: v for k, v in os.environ.items() if not k.startswith("CMB_")}
        env.update(extra)
        p = subprocess.run([sys.executable, str(script), str(tmp_path / name)], env=env, cwd=str(tmp_path),
                           capture_output=True, text=True, timeout=300)
        assert p.returncode == 0, p.stderr[-3000:]
        res[name] = dict(np.load(tmp_path / (name + ".npz")))
        logs[name] = {k: Launches(tuple(x) for x in v) for k, v in json.load(open(tmp_path / (name + ".json"))).items()}
        SEEN.update(*[v.instances() for v in logs[name].values()])
    for name in SWITCHES:
        for k, v in res["default"].items():
            assert np.array_equal(res[name][k], v, equal_nan=True), (name, k)
    d = logs["default"]
    assert d["wide"].args("k1_up_mma") == {(2, 4, 128, 2, False)} and d["narrow"].args("k1_up_mma") == {(2, 4, 32, 2, False)}
    assert d["null"].args("k1_up_mma") == {(2, 4, 64, 3, True)} and d["null"].args("k1_down_mma") == {(2, 4, 128, 2, True)}
    for case in ("wide", "null"):
        assert {a[2] for a in logs["narrow1"][case].args("k1_up_mma") | logs["narrow1"][case].args("k1_down_mma")} == {32}
    assert logs["narrow0"]["narrow"].args("k1_up_mma") == {(2, 4, 128, 2, False)}
    assert logs["narrow0"]["narrow"].args("k1_down_mma") == {(2, 4, 128, 2, False)}
    assert logs["up_sg128"]["null"].args("k1_up_mma") == {(2, 4, 128, 2, True)}
    for name, case in (("up_stages2", "narrow"), ("up_stages2", "null"), ("ring40", "null")):
        assert logs[name][case].args("k1_up_mma") == d[case].args("k1_up_mma")
        assert max(logs[name][case].smem("k1_up_mma")) < min(d[case].smem("k1_up_mma")), (name, case)


# ------------------------------------------------------------------------------------------ coverage
def all_instances():
    """Every K1 instance the launchers can select (k1_mma.cu, k1_mma20.cu, k1_map.cu)."""
    out = set()
    for C in range(1, 9):
        for st in ("false", "true"):
            for sg, minb in ((32, 2), (128, 2), (128, 1), (32, 1)):
                out.add("k1_down_mma<2,%d,%d,%d,%s>" % (C, sg, minb, st))
            for sg, minb in ((32, 2), (128, 2), (128, 1)) + (((64, 3),) if st == "true" else ()):
                out.add("k1_up_mma<2,%d,%d,%d,%s>" % (C, sg, minb, st))
    for minb in (1, 2):
        for st in ("false", "true"):
            out |= {"k1_down_mma20<%d,%s>" % (minb, st), "k1_up_mma20<%d,%s>" % (minb, st)}
    return out | {"k1_sum_classes", "k1_down<20,1,0>", "k1_up<20,1,192,1,0,0>"}


# Instances this file does not reach, and why.  Depth d of the down stack needs a tree of >= 2^(d+1) taxa.
# Shared memory per CTA on a B200: 227 KB opt-in, less 2 KB, per MINB CTAs.
def _not_run():
    out = {}
    for st in ("false", "true"):
        for C in (1, 2):
            out["k1_down_mma<2,%d,128,1,%s>" % (C, st)] = (
                "wide MINB=2 holds the whole down stack up to depth %s; needs >= 2^14 taxa" % ("20 (kMaxStack)" if C == 1 else "12"))
        for C in (1, 2, 3, 4, 5):
            out["k1_down_mma<2,%d,32,1,%s>" % (C, st)] = (
                "wide MINB=1 holds the stack up to depth %s at C = %d" % ({1: "20", 2: "20", 3: "17", 4: "12", 5: "10"}[C], C)
                + ("; deeper needs a tree of 2^%d taxa, not run here to keep the file short" % {4: 14, 5: 12}[C]
                   if C >= 4 else "; deeper is refused (kMaxStack = 20) or needs more than 180 GB of partials"))
        for C in range(1, 7):
            out["k1_up_mma<2,%d,128,1,%s>" % (C, st)] = (
                "the largest up stage at C <= 6 (two stored 128-site chunks, 55 KB) fits two stages at MINB=2")
    for C in range(1, 9):
        if C != 4:
            out["k1_up_mma<2,%d,128,2,true>" % C] = ("device-simulated batches take the 64-site up pass unless "
                                                     "CMB_UP_SG=128; the switch test runs that at C = 4")
    out["k1_up_mma<2,8,128,2,true>"] = ("C = 8 and a tree with two stored children: neither 64/3 nor 128/2 "
                                        "fits; without such nodes the 64-site pass fits")
    out["k1_up_mma<2,7,128,1,true>"] = ("C = 7: the 64-site, 3-CTA up pass always fits (36 KB stages); only "
                                        "CMB_UP_SG=128 reaches this one")
    for st in ("false", "true"):
        out["k1_up_mma20<1,%s>" % st] = ("the protein up stage (44 KB: one class, two stored 64-site chunks) "
                                         "always fits two stages at MINB=2")
    out["k1_down_mma20<1,true>"] = "a device null on a tree of >= 2048 taxa (depth >= 10): not run here"
    return out


NOT_RUN = _not_run()


def test_every_selectable_instance_ran(request):
    """The union of what this file launched covers every instance in all_instances() not listed in NOT_RUN."""
    mine = [i for i in request.session.items if i.module is request.module and i is not request.node]
    defined = [n for n in dir(request.module) if n.startswith("test_") and n != request.node.name]
    if {i.originalname for i in mine} != set(defined):
        pytest.skip("runs only with the whole file")
    assert set(NOT_RUN) <= all_instances()
    missing = all_instances() - set(NOT_RUN) - SEEN
    assert not missing, sorted(missing)
