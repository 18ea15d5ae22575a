"""Every launch shape of Mica's kernels (K5) against the CPU oracle.

The permutation launcher picks its CTA width and dynamic shared memory from the number of sequences T, and the kernel
draws one or two shuffle indices per generator word depending on T. Each permutation test here records, with
torch.profiler, the instance, CTA width and shared memory of the launch, asserts them against a Python restatement of
launch_mica_permutations, and compares Perm.p.value / Perm.nb of every pair with the oracle's replay of the same
shuffle stream. The table kernels (k5_entropy, k5_pairs, k5_average, k5_rows, k5_listed) are compared at the edges of
their grids and above 65535 sequences, where the packed 16-bit joint table of pair_stats no longer holds a cell. The
last test checks that the file ran every instance the launchers can select, except those listed in NOT_RUN with the
reason they are not reached."""
import json
import math
import os
import re
import subprocess
import sys
import tempfile
import textwrap
import time

import numpy as np
import pytest
import oracle_binding as O
from comap_b200 import synthetic as syn

pytestmark = pytest.mark.gpu
RTOL = 1e-9
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ------------------------------------------------------------------------------------------ kernel recorder
_K5 = re.compile(r"\b(k5_\w+?)(<[^()]*>)?\(")
SEEN = set()          # every K5 instance this module launched, permutation kernels as 'instance@CTA width'


def instance_of(kernel_name):
    """'void cmb::(anonymous namespace)::k5_permutations<4, 5>(int, ...)' -> 'k5_permutations<4,5>'."""
    m = _K5.search(kernel_name)
    return None if m is None else m.group(1) + (m.group(2) or "").replace(" ", "")


class Launches(list):
    """(instance, CTA width, dynamic + static shared memory) of every K5 kernel launched inside one `recorded()` window;
    `others`: the names of the other kernels, `memsets`: the number of device memsets."""

    def __init__(self, *a):
        super().__init__(*a)
        self.others = []
        self.memsets = 0

    def __repr__(self):
        return "Launches(%s, others=%s, memsets=%d)" % (list.__repr__(self), self.others, self.memsets)

    def instances(self, prefix=""):
        return {i for i, _, _ in self if i.startswith(prefix)}

    def shapes(self, prefix):
        """{(instance, CTA width, shared memory)} of the kernels whose name starts with prefix."""
        return {x for x in self if x[0].startswith(prefix)}

    def keys(self):
        return {i + "@%d" % w if i.startswith("k5_permutations") else i for i, w, _ in self}


def _window(fn, ctx, lead):
    """fn() under torch.profiler (CUDA activity), after `lead` seconds of small torch kernels and a marker kernel
    (x *= 2): (its value, Launches, launches the library counted meanwhile)."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    out = Launches()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        x = torch.ones(1, device="cuda")
        t0 = time.perf_counter()
        while True:
            x.add_(1)
            torch.cuda.synchronize()
            if time.perf_counter() - t0 >= lead:
                break
        x.mul_(2)
        torch.cuda.synchronize()
        n0 = ctx.launch_count() if ctx is not None else 0
        value = fn()
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
                a = e.get("args", {})
                out.append((inst, int(a.get("block", [-1])[0]), int(a.get("shared memory", -1))))
            else:
                out.others.append(e.get("name", ""))
        elif e.get("cat") == "gpu_memset":
            out.memsets += 1
    return value, out, n1 - n0


def recorded(fn, ctx=None, setup=None, leads=(0.01, 0.05, 0.25, 1.0, 4.0)):
    """Runs fn() under torch.profiler and returns (its value, the Launches of its trace).

    A window's trace can miss the kernels of its first moments: test_gpu_k1_shapes saw a library kernel missing when
    it was the first of its window, and on a B200, after other modules had profiled in the same process, whole
    windows of these short calls came back empty, the torch kernels included, or held only their last kernel.  So
    each window opens with small torch kernels for a lead time, then a marker kernel, both followed by a device
    synchronisation.  A trace without the marker did not capture the window: fn (a deterministic library call) runs
    again in a new window with a longer lead, after setup() outside the window (to drop what the library cached from
    the lost run).
    With `ctx`, the library kernels and memsets in the captured trace must add up to the launches the library counted
    (cmb_launch_count counts the permutation test's work-counter reset, a memset, with its kernel): a dropped launch
    fails the test instead of passing an assertion that some instance did not run."""
    for lead in leads:
        if setup is not None:
            setup()
        value, out, counted = _window(fn, ctx, lead)
        if any("MulFunctor" in n for n in out.others):
            break
        print("profiler window not captured after a %g s lead (no marker kernel in the trace): running it again" % lead)
    SEEN.update(out.keys())
    if ctx is not None:
        lib = len(out) + sum("cmb::" in n for n in out.others) + out.memsets
        assert lib == counted, "the trace holds %d library launches, the library counted %d: %r" % (lib, counted, out)
    return value, out


# ------------------------------------------------------------------------------------------ library rules
SMEM_CAP = 200 * 1024


def perm_shape(T):
    """launch_mica_permutations: (CTA width, dynamic shared memory), None when refused.  256 masks | c / T and
    (c / T) ln(c / T) for c = 0..T | each warp's two columns | two private columns per lane, four characters a word;
    the width halves while the CTA needs more than 64 KB."""
    T4 = (T + 3) // 4
    q = ((T + 1) * 16 + 15) & ~15

    def size(nt):
        return 1024 + q + (nt // 32) * 8 * T4 + 8 * T4 * nt
    nt = 128
    while nt > 32 and size(nt) > 64 * 1024:
        nt //= 2
    return None if size(nt) > SMEM_CAP else (nt, size(nt))


def perm_instance(A):
    """One permutation instance per alphabet, at the register budget of 5 CTAs per SM."""
    return "k5_permutations<%d,5>" % A


def pair_index(i, j, S):
    return i * S - i * (i + 1) // 2 + (j - i - 1)


def pair_of(idx, S):
    """Inverse of pair_index in exact integer arithmetic."""
    b = 2 * S - 1
    i = (b - math.isqrt(b * b - 8 * idx)) // 2
    while i > 0 and pair_index(i, i + 1, S) > idx:
        i -= 1
    while i < S - 2 and pair_index(i + 1, i + 2, S) <= idx:
        i += 1
    return i, i + 1 + idx - pair_index(i, i + 1, S)


def test_restated_launch_rules():
    """The regimes the tests below are built on: CTA width, shared memory and the draw rule switch at these T."""
    widths = {T: perm_shape(T)[0] for T in (2, 228, 229, 256, 257, 434, 435, 2484)}
    assert widths == {2: 128, 228: 128, 229: 64, 256: 64, 257: 64, 434: 64, 435: 32, 2484: 32}
    assert perm_shape(434)[1] == 65536 and perm_shape(2484)[1] == 204728 and perm_shape(2485) is None
    S = 65535
    for idx in (0, 1, S - 2, S - 1, 12345678, S * (S - 1) // 2 - 1):
        i, j = pair_of(idx, S)
        assert 0 <= i < j < S and pair_index(i, j, S) == idx


# ------------------------------------------------------------------------------------------ inputs
# code masks: the states, the fully unknown character (code A), then ambiguity codes
DNA_MASK = np.array([1, 2, 4, 8, 15, 0b0101, 0b1010, 0b1110], np.uint32)          # A C G T | N | R Y B
AA = syn.AA_ORDER
PROT_MASK = np.array([1 << k for k in range(20)] + [(1 << 20) - 1, (1 << AA.index("D")) | (1 << AA.index("N")),
                                                     (1 << AA.index("E")) | (1 << AA.index("Q"))], np.uint32)  # | X | B Z
MASKS = {4: DNA_MASK, 20: PROT_MASK}
AMBIGUOUS = {4: [5, 6, 7], 20: [20, 21, 22]}
COPY, NOISY, CONST, UNKNOWN = 1, 2, 3, 4          # column roles (column 0 is random)


def star_tree(T):
    """Leaves 0..T-1 under root T, as the front-end builds without use_model: its binarised chain has down stack depth 1."""
    parent = np.full(T + 1, T, np.int32)
    parent[T] = -1
    return parent, np.full(T + 1, 0.1)


def model(A):
    Q, pi = syn.hky85(2.5, [0.3, 0.2, 0.2, 0.3]) if A == 4 else syn.jtt92()
    return Q, pi, np.ones(1), np.ones(1)


def load(ctx, codes, A):
    """Star tree, one-class model of alphabet A (nothing is mapped: the model only sets A), the alignment."""
    ctx.set_tree(*star_tree(codes.shape[0]))
    ctx.set_model(*model(A))
    ctx.set_alignment(codes, MASKS[A])


def columns(T, S, A, seed, ambiguity=0):
    """[T][S] codes: column 0 random, 1 its copy (runs the whole budget), 2 a noisy copy, 3 constant once its unknown
    characters are ignored, 4 all unknown, the rest independent, every other one dominated by one state.
    ambiguity = k: k ambiguity codes in column 5 (one: the generic evaluation for the pairs of that column only)."""
    rng = np.random.default_rng(seed)
    codes = rng.integers(0, A, size=(T, S)).astype(np.uint8)
    for s in range(5, S, 2):
        codes[:, s] = np.where(rng.random(T) < 0.6, rng.integers(A), codes[:, s])
    codes[:, COPY] = codes[:, 0]
    codes[:, NOISY] = np.where(rng.random(T) < 0.15, rng.integers(0, A, T), codes[:, 0])
    codes[:, CONST] = rng.integers(A)
    codes[rng.random(T) < 0.2, CONST] = A
    codes[0, CONST] = A
    codes[:, UNKNOWN] = A
    if ambiguity:
        rows = rng.choice(T, min(T, ambiguity), replace=False)
        codes[rows, 5] = rng.choice(AMBIGUOUS[A], len(rows))
    return codes


def check_table(ctx, codes, A):
    """cmb_mica_pairs' MI / Hjoint of every pair against orc_site_pair, 1e-9; returns the MI column."""
    mask = MASKS[A]
    p = ctx.mica_pairs("hmin")
    S = codes.shape[1]
    ii, jj = np.triu_indices(S, 1)
    assert np.array_equal(p["i"], ii) and np.array_equal(p["j"], jj)
    for t in range(len(ii)):
        mi, hj = O.site_pair(codes[:, ii[t]], codes[:, jj[t]], A, mask)
        assert abs(p["mi"][t] - mi) <= RTOL * max(1.0, abs(mi)), (ii[t], jj[t], p["mi"][t], mi)
        assert abs(p["hjoint"][t] - hj) <= RTOL * max(1.0, abs(hj)), (ii[t], jj[t], p["hjoint"][t], hj)
    return p


def perm_vs_oracle(ctx, codes, A, seed, max_perm, const_cols=(CONST, UNKNOWN)):
    """One permutation test: the launch shape against perm_shape, every pair against orc_mica_permutations.  A pair may
    stop elsewhere than on the host only when one of its shuffled MIs came within rounding of its MI (a tie that the
    device and host logarithms may settle differently).  Below 16 sequences a shuffled table is often a relabelling of
    the observed one, so such ties are the rule there rather than the exception.  The pairs of const_cols get p = 1
    after 0 shuffles."""
    T, S = codes.shape
    load(ctx, codes, A)
    mi = check_table(ctx, codes, A)["mi"]
    (pv, nb), rec = recorded(lambda: ctx.mica_permutations(seed, max_perm), ctx)
    nt, smem = perm_shape(T)
    assert rec.shapes("k5_permutations") == {(perm_instance(A), nt, smem)}, rec
    opv, onb, closest = O.mica_permutations(codes, A, MASKS[A], seed, max_perm)
    n = S * (S - 1) // 2
    assert len(pv) == n and nb.min() >= 0 and nb.max() <= max_perm and pv.min() > 0 and pv.max() <= 1
    diff = (nb != onb) | (pv != opv)
    assert np.all(closest[diff] <= 1e-12 * np.maximum(1.0, np.abs(mi[diff]))), \
        "pairs %s differ without a rounding tie" % np.flatnonzero(diff & (closest > 1e-12 * np.maximum(1.0, np.abs(mi))))
    assert diff.sum() <= max(1, (0.25 if T < 16 else 0.02) * n), "pairs that differ: %d of %d" % (diff.sum(), n)
    ii, jj = np.triu_indices(S, 1)
    const = np.isin(ii, const_cols) | np.isin(jj, const_cols)
    assert np.all(nb[const] == 0) and np.all(pv[const] == 1.0)
    stopped = (nb < max_perm) & (nb > 0)
    assert np.all(pv[stopped] == 6.0 / (nb[stopped] + 1.0))
    return pv, nb, opv, onb


@pytest.fixture(scope="module")
def ctx():
    from comap_b200 import api
    c = api.Context()
    yield c
    c.close()


# ------------------------------------------------------------------------------------------ permutation test, A = 4
# word edges of the four-character private copies (2, 3, 5, 8, 9), both sides of each CTA-width switch (228 | 229,
# 434 | 435), both sides of the draw rule (256: two draws per word, 257: one) and the largest T that fits (2484)
PERM_T4 = [2, 3, 5, 8, 9, 228, 229, 256, 257, 434, 435, 2484]
LONG = {8, 228, 257, 2484}                        # cases run with the reference's budget of 1000 shuffles


@pytest.mark.parametrize("ambiguity", [0, 1])
@pytest.mark.parametrize("T", PERM_T4)
def test_dna_permutations_in_every_regime(ctx, T, ambiguity):
    """A = 4, 10 sites: the filtered state-index evaluation, and with one ambiguous character the generic one for the
    pairs of its column.  A column against its copy runs the whole budget once T is large enough that no shuffle can
    match it by chance."""
    max_perm = 1000 if T in LONG else 200
    codes = columns(T, 10, 4, 1000 + T, ambiguity)
    pv, nb, _, onb = perm_vs_oracle(ctx, codes, 4, 31 + T, max_perm)
    if T >= 100:
        assert nb[pair_index(0, COPY, 10)] == max_perm and onb[pair_index(0, COPY, 10)] == max_perm
    print("T = %d: %d pairs, %d shuffles" % (T, len(nb), nb.sum()))


# ------------------------------------------------------------------------------------------ permutation test, A = 20
@pytest.mark.parametrize("ambiguity", [0, 6])
@pytest.mark.parametrize("T", [100, 229, 300, 600])
def test_protein_permutations(ctx, T, ambiguity):
    """A = 20 (JTT92): CTA widths 128 (100), 64 with two draws per word (229) and with one (300), 32 (600); with B, Z
    and X in one column, its pairs take the generic evaluation."""
    codes = columns(T, 10, 20, 2000 + T, ambiguity)
    perm_vs_oracle(ctx, codes, 20, 77 + T, 300)


# ------------------------------------------------------------------------------------------ refusal
def test_permutations_refused_above_the_largest_shape(ctx):
    """T = 2485 needs 205 008 B in a one-warp CTA: refused before any launch; the context then still works."""
    assert perm_shape(2485) is None
    codes = columns(2485, 6, 4, 5)
    load(ctx, codes, 4)
    def refused():
        with pytest.raises(RuntimeError, match="shared memory"):
            ctx.mica_permutations(1, 100)
    _, rec = recorded(refused, ctx)
    assert not rec.instances("k5_permutations") and rec.memsets == 0, rec
    h, avg = ctx.mica_sites()
    oh, oavg = O.mica_sites(codes, 4, DNA_MASK)
    assert np.allclose(h, oh, rtol=RTOL, atol=1e-13) and np.allclose(avg, oavg, rtol=RTOL, atol=1e-13)
    perm_vs_oracle(ctx, columns(30, 6, 4, 6), 4, 2, 100)


# ------------------------------------------------------------------------------------------ budget edges
def test_budget_at_the_warp_trip_edges(ctx):
    """max_perm in {1, 5, 31, 32, 33, 63, 64, 65}: a warp scores 32 shuffles a trip (the first trip 31 and the observed
    table), so these end a budget on either side of a trip.  For each budget >= 5 the alignment holds pairs whose
    fifth hit is exactly the last allowed shuffle, away from any rounding tie: Perm.nb == max_perm with
    p = 6 / (max_perm + 1), on both sides."""
    T, S, seed = 40, 60, 99
    rng = np.random.default_rng(7)
    base = rng.integers(0, 4, size=T)
    codes = np.empty((T, S), np.uint8)
    for s in range(S):                    # noisy copies of one column: pairs stop anywhere from 5 to 1000 shuffles
        codes[:, s] = np.where(rng.random(T) < rng.uniform(0.3, 1.0), rng.integers(0, 4, T), base)
    _, onb_free, closest = O.mica_permutations(codes, 4, DNA_MASK, seed, 1000)
    for max_perm in (1, 5, 31, 32, 33, 63, 64, 65):
        pv, nb, opv, onb = perm_vs_oracle(ctx, codes, 4, seed, max_perm, const_cols=())
        if max_perm == 1:
            assert np.all(nb == 1)
            continue
        edge = np.flatnonzero((onb_free == max_perm) & (closest > 1e-11))           # MI <= ln 4
        assert len(edge), "no pair stops at exactly %d shuffles: change the alignment's seed" % max_perm
        assert np.all(nb[edge] == max_perm) and np.all(onb[edge] == max_perm)
        assert np.all(pv[edge] == 6.0 / (max_perm + 1)) and np.all(opv[edge] == 6.0 / (max_perm + 1))


# ------------------------------------------------------------------------------------------ pair-index decode
def test_pair_decode_at_the_largest_table(ctx):
    """S = 65 535 (the largest table k5_pairs accepts): shards of 2^20 hold ~2 000 pairs spread over the whole
    triangle; every row against orc_mica_permutation_test called with the pair index decoded on the host.  T = 32:
    with a handful of sequences nearly every pair meets a rounding tie, which would let a wrongly decoded pair pass."""
    S, T, seed, max_perm, shard_count = 65535, 32, 4321, 40, 1 << 20
    n_pairs = S * (S - 1) // 2
    codes = np.random.default_rng(3).integers(0, 4, size=(T, S)).astype(np.uint8)
    load(ctx, codes, 4)
    last = (n_pairs - 1) % shard_count
    for shard in sorted({0, 1, 777777, shard_count - 1, last}):
        (pv, nb), rec = recorded(lambda: ctx.mica_permutations(seed, max_perm, shard_index=shard, shard_count=shard_count),
                                 ctx)
        assert rec.shapes("k5_permutations") == {("k5_permutations<4,5>",) + perm_shape(T)}, rec
        idx = np.arange(shard, n_pairs, shard_count)
        assert len(pv) == len(idx) > 2000
        differ = 0
        for k, p in enumerate(idx):
            i, j = pair_of(int(p), S)
            mi, opv, onb, closest = O.mica_permutation_test(codes[:, i], codes[:, j], 4, DNA_MASK, seed, int(p), max_perm)
            if (pv[k], nb[k]) != (opv, onb):
                assert closest <= 1e-12 * max(1.0, abs(mi)), (shard, k, int(p), i, j, pv[k], nb[k], opv, onb)
                differ += 1
        assert differ <= 0.05 * len(idx), differ
        if shard == last:
            assert pair_of(int(idx[-1]), S) == (S - 2, S - 1)


# ------------------------------------------------------------------------------------------ table kernels
@pytest.mark.parametrize("A", [4, 20])
@pytest.mark.parametrize("S", [2, 3, 128, 129, 130, 257])
def test_table_kernels_at_their_grid_edges(ctx, A, S):
    """k5_entropy, k5_pairs, k5_average, k5_rows at S on both sides of a 128-thread CTA (k5_pairs' and k5_rows' rows
    hold S - 1 - i pairs), with ambiguity codes in a few columns; k5_listed at n on both sides of one CTA."""
    T = 37
    codes = columns(T, S, A, 3000 + S, ambiguity=3) if S > 5 else \
        np.random.default_rng(S).integers(0, A + 1, size=(T, S)).astype(np.uint8)
    mask = MASKS[A]
    load(ctx, codes, A)
    (h, avg), rec = recorded(ctx.mica_sites, ctx, setup=lambda: ctx.set_alignment(codes, mask))
    assert rec.instances() == {"k5_entropy<%d>" % A, "k5_pairs<%d>" % A, "k5_average"}, rec
    oh, oavg = O.mica_sites(codes, A, mask)
    assert np.allclose(h, oh, rtol=RTOL, atol=1e-13) and np.allclose(avg, oavg, rtol=RTOL, atol=1e-13)
    p, rec = recorded(lambda: check_table(ctx, codes, A), ctx)
    assert rec.instances() == {"k5_rows"}, rec
    ii, jj = np.triu_indices(S, 1)
    assert np.array_equal(p["hmin"], np.minimum(h[ii], h[jj]))
    rng = np.random.default_rng(S + A)
    for n in (1, 127, 128, 129):
        a, b = rng.integers(0, S, n), rng.integers(0, S, n)
        (mi, hj), rec = recorded(lambda: ctx.mica_pair_list(a, b), ctx)
        assert rec.instances() == {"k5_listed<%d>" % A}, rec
        for k in range(n):
            emi, ehj = O.site_pair(codes[:, a[k]], codes[:, b[k]], A, mask)
            assert abs(mi[k] - emi) <= RTOL * max(1.0, abs(emi)) and abs(hj[k] - ehj) <= RTOL * max(1.0, abs(ehj))


def test_parametric_null_rows(ctx):
    """The parametric bootstrap's pairs (k5_listed over the simulated tip matrix, k5_min2 for Nmin) against the oracle."""
    parent, brlen = syn.random_tree(20, 9, 0.12)
    Q, pi = syn.hky85(2.5, [0.3, 0.2, 0.2, 0.3])
    rates, probs = syn.gamma_rates(0.5, 4)
    ctx.set_tree(parent, brlen)
    ctx.set_model(Q, pi, rates, probs)
    ctx.set_alignment(ctx.simulate(5, 0, 70)[0], syn.identity_code_mask(4))
    ctx.map()
    rep_cpu, rep_ram = 2, 150
    raw, rec = recorded(lambda: ctx.mica_null_parametric(17, rep_cpu, rep_ram, K=4))
    assert {"k5_listed<4>", "k5_min2"} <= rec.instances(), rec
    for rep in range(rep_cpu):
        s1 = ctx.simulate(17, (2 * rep) * rep_ram, rep_ram)[0]
        s2 = ctx.simulate(17, (2 * rep + 1) * rep_ram, rep_ram)[0]
        m1 = O.map_sites(parent, brlen, Q, pi, rates, probs, s1, syn.identity_code_mask(4))
        m2 = O.map_sites(parent, brlen, Q, pi, rates, probs, s2, syn.identity_code_mask(4))
        rows = raw[rep * rep_ram:(rep + 1) * rep_ram]
        assert np.allclose(rows[:, 2], np.minimum(m1["norm"], m2["norm"]), rtol=RTOL, atol=1e-12)
        for j in range(rep_ram):
            mi, hj = O.site_pair(s1[:, j], s2[:, j], 4, syn.identity_code_mask(4))
            assert abs(rows[j, 0] - mi) <= 1e-9 and abs(rows[j, 1] - hj) <= 1e-9


# ------------------------------------------------------------------------------------------ 65 536 sequences
def many_sequences(T, S=40, seed=11):
    """A = 4 columns whose joint cells reach the 16-bit edge: columns 0 and 1 are state 0 but in the same four
    sequences (cell (0, 0) = T - 4, 65 536 at T = 65 540); columns 2 and 3 are state 3 but in three sequences between
    them (cell (3, 3) = T - 3, the last field of the word); columns 4-9 hold one state in 99 % of the sequences;
    column 10 a few unknown characters (the generic path); the rest are random."""
    rng = np.random.default_rng(seed)
    codes = rng.integers(0, 4, size=(T, S)).astype(np.uint8)
    codes[:, 0] = 0; codes[:, 1] = 0
    codes[[1, 2, 3, 4], 0] = [1, 2, 3, 1]
    codes[[1, 2, 3, 4], 1] = [2, 3, 1, 3]
    codes[:, 2] = 3; codes[:, 3] = 3
    codes[[5, 6], 2] = [0, 1]
    codes[[5, 7], 3] = [2, 0]
    for s in range(4, 10):
        codes[:, s] = np.where(rng.random(T) < 0.99, s % 4, codes[:, s])
    codes[rng.choice(T, 10, replace=False), 10] = 4
    return codes


@pytest.mark.parametrize("T", [65535, 65540])
def test_joint_table_beyond_65535_sequences(ctx, T):
    """The table, the average MI and listed pairs of a star tree of T sequences against the oracle at 1e-9.  At
    T = 65 540 cell (0, 0) of the pair (0, 1) holds 65 536 and cell (3, 3) of (2, 3) 65 537; T = 65 535 is the
    largest alignment whose cells all fit 16 bits."""
    codes = many_sequences(T)
    load(ctx, codes, 4)
    check_table(ctx, codes, 4)
    h, avg = ctx.mica_sites()
    oh, oavg = O.mica_sites(codes, 4, DNA_MASK)
    assert np.allclose(h, oh, rtol=RTOL, atol=1e-13)
    assert np.allclose(avg, oavg, rtol=RTOL, atol=1e-13), np.abs(avg - oavg).max()
    a = np.array([0, 1, 2, 3, 0, 3, 4, 10, 5]); b = np.array([1, 0, 3, 2, 3, 0, 5, 11, 5])
    mi, hj = ctx.mica_pair_list(a, b)
    for k in range(len(a)):
        emi, ehj = O.site_pair(codes[:, a[k]], codes[:, b[k]], 4, DNA_MASK)
        assert abs(mi[k] - emi) <= RTOL * max(1.0, abs(emi)) and abs(hj[k] - ehj) <= RTOL * max(1.0, abs(ehj)), (k, mi[k], emi)


# ------------------------------------------------------------------------------------------ switches read once
SWITCH_SCRIPT = textwrap.dedent("""
    import json, sys
    import numpy as np
    sys.path[:0] = [{root!r}, {tests!r}]
    import test_gpu_k5_shapes as K
    from comap_b200 import api
    out = sys.argv[1]
    ctx = api.Context()
    res, launches = {{}}, {{}}
    for T in K.SWITCH_T:
        K.load(ctx, K.columns(T, 12, 4, 500 + T, ambiguity=1), 4)
        (res["pv%d" % T], res["nb%d" % T]), rec = K.recorded(lambda: ctx.mica_permutations(91, 1000), ctx)
        launches[T] = list(rec)
    ctx.close()
    np.savez(out + ".npz", **res)
    json.dump(launches, open(out + ".json", "w"))
""")
SWITCH_T = (100, 300, 600)
SWITCHES = {"default": {}, "filter0": {"CMB_K5_FILTER": "0"}}


def test_switches_read_once_per_process_leave_results_unchanged(tmp_path):
    """CMB_K5_FILTER=0 (every shuffle through the reference's formula) is read into a static on first use, so each
    setting runs in a fresh process at T = 100, 300 and 600 (CTA widths 128, 64, 32): the same table bit for bit, from
    the same instance."""
    script = tmp_path / "run.py"
    script.write_text(SWITCH_SCRIPT.format(root=ROOT, tests=os.path.join(ROOT, "tests")))
    res = {}
    for name, extra in SWITCHES.items():
        env = {k: v for k, v in os.environ.items() if not k.startswith("CMB_")}
        env.update(extra)
        p = subprocess.run([sys.executable, str(script), str(tmp_path / name)], env=env, cwd=str(tmp_path),
                           capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-3000:]
        res[name] = dict(np.load(tmp_path / (name + ".npz")))
        logs = json.load(open(tmp_path / (name + ".json")))
        for T in SWITCH_T:
            rec = Launches(tuple(x) for x in logs[str(T)])
            assert rec.shapes("k5_permutations") == {(perm_instance(4),) + perm_shape(T)}, (name, T, rec)
            SEEN.update(rec.keys())
    for name in SWITCHES:
        for k, v in res["default"].items():
            assert np.array_equal(res[name][k], v), (name, k)
    assert all(res["default"]["nb%d" % T].max() == 1000 for T in SWITCH_T)


# ------------------------------------------------------------------------------------------ coverage
def all_instances():
    """Every K5 instance the launchers can select (k5_mica.cu), each permutation instance at every CTA width its T
    range allows (T <= 2484: 128, 64 and 32 for both)."""
    out = {"k5_%s<%d>" % (k, A) for k in ("entropy", "pairs", "listed") for A in (4, 20)}
    out |= {"k5_average", "k5_rows", "k5_min2"}
    for inst in ("k5_permutations<4,5>", "k5_permutations<20,5>"):
        out |= {"%s@%d" % (inst, w) for w in (128, 64, 32)}
    return out


NOT_RUN = {}          # instance -> why this file does not reach it; every instance is reached


def test_every_selectable_instance_ran(request):
    """The union of what this file launched covers every instance in all_instances() not listed in NOT_RUN."""
    mine = [i for i in request.session.items if i.module is request.module and i is not request.node]
    defined = [n for n in dir(request.module) if n.startswith("test_") and n != request.node.name]
    if {i.originalname for i in mine} != set(defined):
        pytest.skip("runs only with the whole file")
    assert set(NOT_RUN) <= all_instances()
    missing = all_instances() - set(NOT_RUN) - SEEN
    assert not missing, sorted(missing)
