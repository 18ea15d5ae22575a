"""ctypes binding of oracle/liboracle.so -- the CPU parity oracle (test infrastructure).

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this.
"""
import ctypes as C
import os
import subprocess
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SO = os.path.join(ROOT, "oracle", "liboracle.so")

STAT = {"correlation": 0, "covariance": 1, "cosinus": 2, "cosubstitution": 3, "compensation": 4,
        "corrected_correlation": 5, "mi": 6, "mi_label": 7}
DIST = {"correlation": 0, "compensation": 1, "euclidian": 2}
LINK = {"complete": 0, "single": 1, "average": 2}
COUNT = {"uniformization": 0, "decomposition": 1, "naive": 2, "laplace": 3, "label": 4, "one_jump": 5}


def count_id(method):
    """'uniformization' | 'decomposition' | 'naive' | 'laplace' | ('laplace', trunc) -> count_method word."""
    if isinstance(method, tuple):
        return COUNT[method[0]] | (int(method[1]) << 8)
    return COUNT[method]

_lib = None


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(ROOT, "oracle", "comap_oracle.c")
        if (not os.path.exists(_SO)) or os.path.getmtime(_SO) < os.path.getmtime(src):
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
        _lib = C.CDLL(_SO)
        _lib.orc_last_error.restype = C.c_char_p
        _lib.orc_stat.restype = C.c_double
        _lib.orc_stat_group.restype = C.c_double
    return _lib


def _p(a, t):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


def _d(a):
    return _p(a, C.c_double)


def _chk(rc):
    if rc != 0:
        raise RuntimeError("oracle: " + lib().orc_last_error().decode())


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def pmatrix(Q, pi, t):
    A = len(pi)
    P = np.empty((A, A))
    _chk(lib().orc_pmatrix(A, _d(_f64(Q)), _d(_f64(pi)), C.c_double(t), _d(P)))
    return P


def counts(Q, pi, t, method="uniformization", weights=None):
    A = len(pi)
    N = np.empty((A, A))
    w = None if weights is None else _f64(weights)
    _chk(lib().orc_counts(count_id(method), A, _d(_f64(Q)), _d(_f64(pi)), _d(w), C.c_double(t), _d(N)))
    return N


def _tree_args(parent, brlen):
    parent = np.ascontiguousarray(parent, dtype=np.int32)
    brlen = _f64(brlen)
    return (len(parent), _p(parent, C.c_int32), _d(brlen)), (parent, brlen)


def _model_args(Q, pi, rates, probs):
    Q, pi, rates, probs = _f64(Q), _f64(pi), _f64(rates), _f64(probs)
    return (len(pi), _d(Q), _d(pi), len(rates), _d(rates), _d(probs)), (Q, pi, rates, probs)


def map_sites(parent, brlen, Q, pi, rates, probs, codes, code_mask, method="uniformization",
              weights=None, want_vectors=True):
    ta, keep1 = _tree_args(parent, brlen)
    ma, keep2 = _model_args(Q, pi, rates, probs)
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    T, S = codes.shape
    code_mask = np.ascontiguousarray(code_mask, dtype=np.uint32)
    B = len(parent) - 1
    n = np.empty((S, B)) if want_vectors else None
    norm = np.empty(S) if want_vectors else None
    pr = np.empty(S); rc = np.empty(S, dtype=np.int32); ll = np.empty(S)
    w = None if weights is None else _f64(weights)
    _chk(lib().orc_map(*ta, *ma, count_id(method), _d(w), C.c_int64(S), _p(codes, C.c_uint8),
                       len(code_mask), _p(code_mask, C.c_uint32), _d(n), _d(norm), _d(pr),
                       _p(rc, C.c_int32), _d(ll)))
    return dict(n=n, norm=norm, post_rate=pr, rate_class=rc, loglik=ll)


def ancestral_states(parent, brlen, Q, pi, rates, probs, codes, code_mask):
    """asr.method = marginal (CoMap.cpp:168-198): [n_nodes][S] marginal reconstruction."""
    ta, keep1 = _tree_args(parent, brlen)
    ma, keep2 = _model_args(Q, pi, rates, probs)
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    T, S = codes.shape
    code_mask = np.ascontiguousarray(code_mask, dtype=np.uint32)
    out = np.empty((len(parent), S), dtype=np.uint8)
    _chk(lib().orc_ancestral_states(*ta, *ma, C.c_int64(S), _p(codes, C.c_uint8), len(code_mask), _p(code_mask, C.c_uint32),
                                    _p(out, C.c_uint8)))
    return out


def site_entropy(col, A, code_mask):
    col = np.ascontiguousarray(col, dtype=np.uint8); m = np.ascontiguousarray(code_mask, dtype=np.uint32)
    lib().orc_site_entropy.restype = C.c_double
    return lib().orc_site_entropy(len(col), _p(col, C.c_uint8), A, len(m), _p(m, C.c_uint32))


def site_pair(c1, c2, A, code_mask):
    """(MI, Hjoint) of two alignment columns: SiteTools::mutualInformation / jointEntropy(.., true) (Mica.cpp)."""
    c1 = np.ascontiguousarray(c1, dtype=np.uint8); c2 = np.ascontiguousarray(c2, dtype=np.uint8)
    m = np.ascontiguousarray(code_mask, dtype=np.uint32)
    mi = C.c_double(); hj = C.c_double()
    lib().orc_site_pair(len(c1), _p(c1, C.c_uint8), _p(c2, C.c_uint8), A, len(m), _p(m, C.c_uint32), C.byref(mi), C.byref(hj))
    return mi.value, hj.value


def mica_sites(codes, A, code_mask):
    """Entropy and average MI of every site (Mica.cpp:341-361); codes [T][S]."""
    codes = np.ascontiguousarray(codes, dtype=np.uint8); m = np.ascontiguousarray(code_mask, dtype=np.uint32)
    T, S = codes.shape
    h = np.empty(S); a = np.empty(S)
    lib().orc_mica_sites(C.c_int64(S), T, _p(codes, C.c_uint8), A, len(m), _p(m, C.c_uint32), _d(h), _d(a))
    return h, a


def mica_permutations(codes, A, code_mask, seed, max_perm):
    """miTest of every pair (Mica.cpp:92-118) with the device's shuffle stream: p-value, number of shuffles, and the
    smallest |shuffled MI - MI| met on the way; codes [T][S]."""
    codes = np.ascontiguousarray(codes, dtype=np.uint8); m = np.ascontiguousarray(code_mask, dtype=np.uint32)
    T, S = codes.shape
    n = S * (S - 1) // 2
    pv = np.empty(n); nb = np.empty(n, np.int32); cl = np.empty(n)
    lib().orc_mica_permutations(C.c_int64(S), T, _p(codes, C.c_uint8), A, len(m), _p(m, C.c_uint32), C.c_uint64(seed),
                                int(max_perm), _d(pv), _p(nb, C.c_int32), _d(cl))
    return pv, nb, cl


def mica_permutation_test(c1, c2, A, code_mask, seed, pair, max_perm):
    """miTest of one pair of columns with the shuffle stream of pair index `pair` (idx = i S - i (i + 1) / 2 + j - i - 1
    in mica's order): (MI, p-value, number of shuffles, smallest |shuffled MI - MI|)."""
    c1 = np.ascontiguousarray(c1, dtype=np.uint8); c2 = np.ascontiguousarray(c2, dtype=np.uint8)
    m = np.ascontiguousarray(code_mask, dtype=np.uint32)
    mi, pv, nb, cl = C.c_double(), C.c_double(), C.c_int(), C.c_double()
    lib().orc_mica_permutation_test(len(c1), _p(c1, C.c_uint8), _p(c2, C.c_uint8), A, len(m), _p(m, C.c_uint32), C.c_uint64(seed),
                                    C.c_uint64(pair), int(max_perm), C.byref(mi), C.byref(pv), C.byref(nb), C.byref(cl))
    return mi.value, pv.value, nb.value, cl.value


def set_mi_threshold(t):
    lib().orc_set_mi_threshold(C.c_double(t))


def set_mi_label(n_states):
    """statistic=MI with nijt=Label (CoETools.cpp:577-589): one category per substitution label."""
    lib().orc_set_mi_label(int(n_states))


def set_map_mode(average=True, joint=True):
    """nijt.average / nijt.joint (CoETools.cpp:393-407) for every later mapping; reset with set_map_mode()."""
    lib().orc_set_map_mode(int(bool(average)), int(bool(joint)))


def mean_vector(n):
    """Mean vector of a mapping as CoMap builds it (CoMap.cpp:350-359); also installs it for the
    corrected correlation."""
    n = _f64(n); S, B = n.shape
    mv = np.empty(B)
    lib().orc_mean_vector(C.c_int64(S), B, _d(n), _d(mv))
    lib().orc_set_mean_vector(B, _d(mv))
    return mv


def mean_vectors(n1, n2):
    """Installs the two data sets' mean vectors (setMeanVectors, CoMap.cpp:295-309)."""
    mv2 = mean_vector(n2).copy()
    mv1 = mean_vector(n1).copy()
    lib().orc_set_mean_vectors(len(mv1), _d(mv1), _d(mv2))
    return mv1, mv2


def pairs_inter(stat_name, m1, m2, min_rate_class1=0, min_rate_class2=0, min_rate1=0.0, min_rate2=0.0,
                max_rate_class_diff=-1, max_rate_diff=-1.0, min_stat=0.0, independent=False, nmin_by_row=True):
    """m1, m2: dicts with n, norm, post_rate, rate_class of the two data sets."""
    n1, n2 = _f64(m1["n"]), _f64(m2["n"])
    S1, B = n1.shape; S2 = n2.shape[0]
    cap = S1 * S2
    oi = np.empty(cap, np.int32); oj = np.empty(cap, np.int32); st = np.empty(cap)
    rcm = np.empty(cap, np.int32); prm = np.empty(cap); nm = np.empty(cap); nr = C.c_int64(0)
    rc1 = np.ascontiguousarray(m1["rate_class"], dtype=np.int32); rc2 = np.ascontiguousarray(m2["rate_class"], dtype=np.int32)
    _chk(lib().orc_pairs_inter(STAT[stat_name], C.c_int64(S1), C.c_int64(S2), B, _d(n1), _d(n2), _d(_f64(m1["norm"])),
                               _d(_f64(m2["norm"])), _d(_f64(m1["post_rate"])), _d(_f64(m2["post_rate"])),
                               _p(rc1, C.c_int32), _p(rc2, C.c_int32), min_rate_class1, min_rate_class2,
                               C.c_double(min_rate1), C.c_double(min_rate2), max_rate_class_diff,
                               C.c_double(max_rate_diff), C.c_double(min_stat), int(independent), int(nmin_by_row),
                               C.c_int64(cap), _p(oi, C.c_int32), _p(oj, C.c_int32), _d(st), _p(rcm, C.c_int32),
                               _d(prm), _d(nm), C.byref(nr)))
    k = nr.value
    return dict(i=oi[:k], j=oj[:k], stat=st[:k], rcmin=rcm[:k], prmin=prm[:k], nmin=nm[:k])


def stat(name, v1, v2):
    v1, v2 = _f64(v1), _f64(v2)
    return lib().orc_stat(STAT[name], len(v1), _d(v1), _d(v2))


def stat_group(name, n, members):
    n = _f64(n); m = np.ascontiguousarray(members, dtype=np.int32)
    return lib().orc_stat_group(STAT[name], n.shape[1], _d(n), len(m), _p(m, C.c_int32))


def domain_index(lo, hi, K, x):
    return lib().orc_domain_index(C.c_double(lo), C.c_double(hi), K, C.c_double(x))


def pairs(stat_name, n, norm, post_rate, rate_class, min_rate_class=0, min_rate=0.0,
          max_rate_class_diff=-1, max_rate_diff=-1.0, min_stat=0.0, null=None):
    """null = (K, nmax, bin_offsets, sorted) or None."""
    n = _f64(n); S, B = n.shape
    norm, post_rate = _f64(norm), _f64(post_rate)
    rate_class = np.ascontiguousarray(rate_class, dtype=np.int32)
    cap = S * (S - 1) // 2
    oi = np.empty(cap, np.int32); oj = np.empty(cap, np.int32); st = np.empty(cap)
    rcm = np.empty(cap, np.int32); prm = np.empty(cap); nm = np.empty(cap)
    pv = np.full(cap, np.nan); ns = np.zeros(cap, np.int64); nr = C.c_int64(0)
    if null is None:
        K, nmax, offs, srt = 0, 0.0, None, None
    else:
        K, nmax, offs, srt = null
        offs = np.ascontiguousarray(offs, dtype=np.int64); srt = _f64(srt)
    _chk(lib().orc_pairs(STAT[stat_name], C.c_int64(S), B, _d(n), _d(norm), _d(post_rate),
                         _p(rate_class, C.c_int32), min_rate_class, C.c_double(min_rate),
                         max_rate_class_diff, C.c_double(max_rate_diff), C.c_double(min_stat),
                         K, C.c_double(nmax), _p(offs, C.c_int64), _d(srt), C.c_int64(cap),
                         _p(oi, C.c_int32), _p(oj, C.c_int32), _d(st), _p(rcm, C.c_int32), _d(prm),
                         _d(nm), _d(pv), _p(ns, C.c_int64), C.byref(nr)))
    k = nr.value
    return dict(i=oi[:k], j=oj[:k], stat=st[:k], rcmin=rcm[:k], prmin=prm[:k], nmin=nm[:k],
                pvalue=pv[:k], nsim=ns[:k])


def simulate(parent, brlen, Q, pi, rates, probs, seed, first_site, n, weighted_classes=False):
    ta, keep1 = _tree_args(parent, brlen)
    ma, keep2 = _model_args(Q, pi, rates, probs)
    from comap_b200.synthetic import n_leaves_of
    T = n_leaves_of(np.asarray(parent))
    states = np.empty((T, n), dtype=np.uint8); cls = np.empty(n, dtype=np.int32)
    _chk(lib().orc_simulate(*ta, *ma, C.c_uint64(seed), C.c_int64(first_site), C.c_int64(n),
                            int(weighted_classes), _p(states, C.c_uint8), _p(cls, C.c_int32)))
    return states, cls


def simulate_continuous(parent, brlen, Q, pi, kind, alpha, p_inv, seed, first_site, n):
    """simulations.continuous = yes: (states [T][n], rate per site)."""
    ta, keep1 = _tree_args(parent, brlen)
    Q, pi = _f64(Q), _f64(pi)
    from comap_b200.synthetic import n_leaves_of
    T = n_leaves_of(np.asarray(parent))
    states = np.empty((T, n), dtype=np.uint8); rates = np.empty(n)
    k = {"constant": 1, "gamma": 2, "invariant": 3}[kind]
    _chk(lib().orc_simulate_continuous(*ta, len(pi), _d(Q), _d(pi), k, C.c_double(alpha), C.c_double(p_inv),
                                       C.c_uint64(seed), C.c_int64(first_site), C.c_int64(n), _p(states, C.c_uint8), _d(rates)))
    return states, rates


def null_intra(parent, brlen, Q, pi, rates, probs, stat_name, sim1, sim2, K, nmax,
               method="uniformization", weights=None):
    ta, keep1 = _tree_args(parent, brlen)
    ma, keep2 = _model_args(Q, pi, rates, probs)
    sim1 = np.ascontiguousarray(sim1, dtype=np.uint8); sim2 = np.ascontiguousarray(sim2, dtype=np.uint8)
    rep_cpu, T, rep_ram = sim1.shape
    tot = rep_cpu * rep_ram
    raw = np.empty((tot, 4)); offs = np.zeros(K + 1, dtype=np.int64); srt = np.empty(tot)
    w = None if weights is None else _f64(weights)
    _chk(lib().orc_null_intra(*ta, *ma, count_id(method), _d(w), STAT[stat_name], rep_cpu, rep_ram,
                              _p(sim1, C.c_uint8), _p(sim2, C.c_uint8), K, C.c_double(nmax),
                              _d(raw), _p(offs, C.c_int64), _d(srt)))
    return dict(raw=raw, bin_offsets=offs, sorted=srt[:offs[-1]])


def distance_matrix(dist_name, n):
    n = _f64(n); S, B = n.shape
    mat = np.empty((S, S))
    _chk(lib().orc_distance_matrix(DIST[dist_name], C.c_int64(S), B, _d(n), _d(mat)))
    return mat


def hclust(linkage, mat):
    mat = np.array(mat, dtype=np.float64, order="C"); S = mat.shape[0]
    left = np.empty(S - 1, np.int32); right = np.empty(S - 1, np.int32); height = np.empty(S - 1)
    _chk(lib().orc_hclust(LINK[linkage], C.c_int64(S), _d(mat), _p(left, C.c_int32),
                          _p(right, C.c_int32), _d(height)))
    return left, right, height


def groups(dist_name, n, norm, left, right, height, max_size):
    n = _f64(n); S, B = n.shape; norm = _f64(norm)
    left = np.ascontiguousarray(left, np.int32); right = np.ascontiguousarray(right, np.int32)
    height = _f64(height)
    members = np.empty(max(1, (S - 1) * max_size), np.int32); offs = np.zeros(S + 1, np.int64)
    gh = np.empty(S); gs = np.empty(S); gn = np.empty(S); ng = C.c_int64(0)
    _chk(lib().orc_groups(DIST[dist_name], C.c_int64(S), B, _d(n), _d(norm), _p(left, C.c_int32),
                          _p(right, C.c_int32), _d(height), max_size, _p(members, C.c_int32),
                          _p(offs, C.c_int64), _d(gh), _d(gs), _d(gn), C.byref(ng)))
    k = ng.value
    return dict(members=[members[offs[g]:offs[g + 1]].copy() for g in range(k)], height=gh[:k],
                stat=gs[:k], nmin=gn[:k])


def group_stat_min(name, vectors):
    """AbstractMinimumStatistic::getValueForGroup (Statistics.h:118-131): minimum over i > j of
    getValueForPair(v[i], v[j]); NaN never replaces the running minimum."""
    mini = np.inf
    for i in range(1, len(vectors)):
        for j in range(i):
            val = stat(name, vectors[i], vectors[j])
            if val < mini:
                mini = val
    return mini


def candidates_reference(stat_name, n_obs, norm_obs, groups, omega, min_sim, max_trials, batches, analysable=None):
    """Pure-Python restatement (small cases only) of CandidateGroupSet (CoETools.h:139-300,
    CoETools.cpp:901-1038) + computePValuesForCandidateGroups (CoETools.cpp:1042-1087).
    `batches` yields (vectors [R][B], norms [R]) of successive simulated batches."""
    G = len(groups)
    an = [True] * G if analysable is None else [bool(x) for x in analysable]
    gstat = (lambda vs: stat_group(stat_name, np.stack(vs), np.arange(len(vs)))) if stat_name == "compensation" else \
            (lambda vs: group_stat_min(stat_name, vs))
    observed = [gstat([n_obs[s] for s in g]) if an[k] else np.nan for k, g in enumerate(groups)]
    lo = [[norm_obs[s] - omega for s in g] for g in groups]
    hi = [[norm_obs[s] + omega for s in g] for g in groups]
    n1 = [0] * G; n2 = [0] * G
    st = dict(g=0, s=0, completed=0, trials=0)
    n_an = sum(an)

    def next_site():
        if n2[st["g"]] < min_sim:
            st["s"] += 1
            if st["s"] >= len(groups[st["g"]]):
                st["g"] = (st["g"] + 1) % G
                st["s"] = 0
        start = st["g"]
        if n2[st["g"]] >= min_sim or not an[st["g"]]:
            while n2[st["g"]] >= min_sim or not an[st["g"]]:
                st["g"] = (st["g"] + 1) % G
                assert st["g"] != start
            st["s"] = 0

    test, n_sim = True, 0
    for vec, norms in batches:
        if not test:
            break
        n_sim += len(norms)
        pending = [[[] for _ in g] for g in groups]
        test_free = True
        i = 0
        while test and i < len(norms):
            first, test_norm = True, False
            while test and not test_norm:
                next_site()
                if first:
                    start, first = (st["g"], st["s"]), False
                elif (st["g"], st["s"]) == start:
                    break
                g, s = st["g"], st["s"]
                test_norm = lo[g][s] <= norms[i] <= hi[g][s]
                if test_norm:
                    pending[g][s].append(vec[i])
                    if all(len(q) > 0 for q in pending[g]):
                        vs = [q.pop(0) for q in pending[g]]
                        n2[g] += 1
                        if gstat(vs) >= observed[g]:
                            n1[g] += 1
                        if n2[g] == min_sim:
                            st["completed"] += 1
                        test_free = False
                    if st["completed"] == n_an:
                        test = False
            i += 1
        if test_free:
            st["trials"] += 1
        test = test and st["trials"] < max_trials
    pv = [(n1[k] + 1.0) / (n2[k] + 1.0) if an[k] else np.nan for k in range(G)]
    return dict(stat=np.array(observed), pvalue=np.array(pv), n1=np.array(n1), n2=np.array(n2), n_simulated=n_sim)
