"""ctypes binding of libcomap_b200.so -- the C ABI of include/comap_b200.h.

Thin, explicit and numpy-only; the CUDA library is the product, this file only marshals
arrays.  Loading fails loudly when the library has not been built (no CPU fallback).
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcomap_b200.so")

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

# every symbol include/comap_b200.h declares (checked by tests/test_abi.py)
SYMBOLS = [
    "cmb_last_error", "cmb_version", "cmb_host_alloc", "cmb_host_free", "cmb_ctx_create",
    "cmb_ctx_destroy", "cmb_sync", "cmb_set_tree", "cmb_set_model", "cmb_set_alignment", "cmb_map",
    "cmb_simulate", "cmb_null_intra", "cmb_null_intra_from_alignments", "cmb_null_samples_dev",
    "cmb_null_load_dev", "cmb_null_get", "cmb_pairs", "cmb_pairs_resident", "cmb_pairs_fetch", "cmb_distance_matrix", "cmb_cluster",
    "cmb_groups", "cmb_cluster_null", "cmb_profile_enable", "cmb_profile_reset", "cmb_profile_get",
    "cmb_launch_count", "cmb_pairs_inter", "cmb_null_inter", "cmb_load_vectors", "cmb_candidates", "cmb_set_async", "cmb_set_mi_threshold", "cmb_set_map_mode", "cmb_ancestral_states",
    "cmb_mica_sites", "cmb_mica_pairs", "cmb_mica_pair_list", "cmb_mica_permutations", "cmb_mica_null_parametric", "cmb_null_load",
    "cmb_comm_unique_id", "cmb_comm_init", "cmb_comm_init_all", "cmb_comm_set", "cmb_comm_destroy", "cmb_comm_rank",
    "cmb_comm_group_start", "cmb_comm_group_end", "cmb_null_intra_sharded", "cmb_set_continuous_rates",
    "cmb_mica_permutations_shard", "cmb_mica_null_parametric_range", "cmb_mica_null_parametric_sharded", "cmb_null_inter_range",
]


class Filters(C.Structure):
    _fields_ = [("min_rate_class", C.c_int32), ("max_rate_class_diff", C.c_int32),
                ("min_rate", C.c_double), ("max_rate_diff", C.c_double), ("min_stat", C.c_double)]


_lib = None


def load():
    """Loads the CUDA library; raises if it is missing (build with python -m comap_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libcomap_b200.so is not built (python -m comap_b200.build); "
                               "comap_b200 has no CPU fallback")
        _lib = C.CDLL(LIB_PATH)
        _lib.cmb_last_error.restype = C.c_char_p
        _lib.cmb_launch_count.restype = C.c_int64
    return _lib


def _p(a, t):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


def _d(a):
    return _p(a, C.c_double)


def _i32(a):
    return _p(a, C.c_int32)


def _i64(a):
    return _p(a, C.c_int64)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def comm_unique_id():
    """128-byte NCCL id (rank 0 creates it, the launcher hands it to every rank)."""
    buf = (C.c_char * 128)()
    lib = load()
    if lib.cmb_comm_unique_id(buf) != 0:
        raise RuntimeError("comap_b200: " + lib.cmb_last_error().decode())
    return bytes(buf)


def comm_init_all(contexts):
    """One process, several contexts on distinct devices: joins them in one communicator."""
    lib = load()
    arr = (C.c_void_p * len(contexts))(*[c.h for c in contexts])
    if lib.cmb_comm_init_all(arr, len(contexts)) != 0:
        raise RuntimeError("comap_b200: " + lib.cmb_last_error().decode())


class Context:
    """One GPU, one stream.  Mirrors the reference's flow: set tree / model / alignment, map,
    null distribution, pairs or clustering (CoMap.cpp:96-737)."""

    def __init__(self, device=-1, stream=None):
        self.lib = load()
        h = C.c_void_p()
        self._chk(self.lib.cmb_ctx_create(int(device), C.c_void_p(stream), C.byref(h)))
        self.h = h
        self.S = self.B = self.T = 0

    def _chk(self, rc):
        if rc != 0:
            raise RuntimeError("comap_b200: " + self.lib.cmb_last_error().decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.cmb_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        self._chk(self.lib.cmb_sync(self.h))

    # ------------------------------------------------------------------ setup
    def set_tree(self, parent, brlen):
        parent = np.ascontiguousarray(parent, dtype=np.int32)
        brlen = _f64(brlen)
        self._chk(self.lib.cmb_set_tree(self.h, len(parent), _i32(parent), _d(brlen)))
        has_child = np.zeros(len(parent), bool)
        has_child[parent[parent >= 0]] = True
        self.T = int((~has_child).sum())
        self.B = len(parent) - 1

    def set_model(self, Q, pi, rates, probs, count_method="uniformization", weights=None):
        Q, pi, rates, probs = _f64(Q), _f64(pi), _f64(rates), _f64(probs)
        w = None if weights is None else _f64(weights)
        self.A, self.C = len(pi), len(rates)
        self._chk(self.lib.cmb_set_model(self.h, len(pi), _d(Q), _d(pi), len(rates), _d(rates), _d(probs),
                                         count_id(count_method), _d(w)))

    def set_alignment(self, codes, code_mask):
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        code_mask = np.ascontiguousarray(code_mask, dtype=np.uint32)
        T, S = codes.shape
        if T != self.T:
            raise ValueError("alignment has %d rows, tree has %d leaves" % (T, self.T))
        self._chk(self.lib.cmb_set_alignment(self.h, C.c_int64(S), _p(codes, C.c_uint8), len(code_mask),
                                             _p(code_mask, C.c_uint32)))
        self.S = S

    # ------------------------------------------------------------------ mapping
    def map(self, want_vectors=True):
        S, B = self.S, self.B
        n = np.empty((S, B)) if want_vectors else None
        norm = np.empty(S); pr = np.empty(S); rc = np.empty(S, np.int32); ll = np.empty(S)
        self._chk(self.lib.cmb_map(self.h, _d(n), _d(norm), _d(pr), _i32(rc), _d(ll)))
        return dict(n=n, norm=norm, post_rate=pr, rate_class=rc, loglik=ll)

    def map_async(self):
        """cmb_map without host outputs: enqueued on a side stream; the next call that needs the mapping
        (pairs, the null's binning, ...) completes it."""
        self._chk(self.lib.cmb_map(self.h, None, None, None, None, None))

    # ------------------------------------------------------------------ simulation / null
    def simulate(self, seed, first_site, n, weighted_classes=False):
        states = np.empty((self.T, n), np.uint8); cls = np.empty(n, np.int32)
        self._chk(self.lib.cmb_simulate(self.h, C.c_uint64(seed), C.c_int64(first_site), C.c_int64(n),
                                        int(weighted_classes), _p(states, C.c_uint8), _i32(cls)))
        return states, cls

    def null_intra(self, stat, seed, rep_cpu, rep_ram, K=10, nmax=-1.0, rep_begin=0, rep_end=None,
                   weighted_classes=False, want_raw=False):
        rep_end = rep_cpu if rep_end is None else rep_end
        raw = np.empty(((rep_end - rep_begin) * rep_ram, 4)) if want_raw else None
        self._chk(self.lib.cmb_null_intra(self.h, STAT[stat], C.c_uint64(seed), rep_cpu, rep_ram, rep_begin,
                                          rep_end, int(weighted_classes), K, C.c_double(nmax), _d(raw)))
        return raw

    def null_intra_from_alignments(self, stat, sim1, sim2, K=10, nmax=-1.0, want_raw=True):
        sim1 = np.ascontiguousarray(sim1, np.uint8); sim2 = np.ascontiguousarray(sim2, np.uint8)
        rep_cpu, T, rep_ram = sim1.shape
        raw = np.empty((rep_cpu * rep_ram, 4)) if want_raw else None
        self._chk(self.lib.cmb_null_intra_from_alignments(self.h, STAT[stat], rep_cpu, rep_ram,
                                                          _p(sim1, C.c_uint8), _p(sim2, C.c_uint8), K,
                                                          C.c_double(nmax), _d(raw)))
        return raw

    def set_map_mode(self, average=True, joint=True):
        """nijt.average / nijt.joint (CoETools.cpp:393-407): which mapping function fills the vectors from now on."""
        self._chk(self.lib.cmb_set_map_mode(self.h, int(bool(average)), int(bool(joint))))

    def ancestral_states(self):
        """asr.method = marginal (CoMap.cpp:168-198): [n_nodes][S] state of largest marginal posterior probability."""
        out = np.empty((self.B + 1, self.S), dtype=np.uint8)
        self._chk(self.lib.cmb_ancestral_states(self.h, out.ctypes.data_as(C.POINTER(C.c_uint8))))
        return out

    # ------------------------------------------------------------------ Mica (CoMap/Mica.cpp)
    def mica_sites(self):
        """Entropy of every site and its average MI with all the others (Mica.cpp:341-361)."""
        h = np.empty(self.S); a = np.empty(self.S)
        self._chk(self.lib.cmb_mica_sites(self.h, _d(h), _d(a)))
        return h, a

    def mica_pairs(self, key="nmin", use_null=False):
        """All pairs in mica's order: MI, Hjoint, Hmin, Nmin and the bootstrap p-value / Nsim (Mica.cpp:646-689)."""
        n = self.S * (self.S - 1) // 2
        r = dict(i=np.empty(n, np.int32), j=np.empty(n, np.int32), mi=np.empty(n), hjoint=np.empty(n), hmin=np.empty(n),
                 nmin=np.empty(n), pvalue=np.full(n, np.nan), nsim=np.zeros(n, np.int32))
        k = C.c_int64(0)
        self._chk(self.lib.cmb_mica_pairs(self.h, {"nmin": 1, "hmin": 2}[key], int(bool(use_null)), C.c_int64(n),
                                          r["i"].ctypes.data_as(C.POINTER(C.c_int32)), r["j"].ctypes.data_as(C.POINTER(C.c_int32)),
                                          _d(r["mi"]), _d(r["hjoint"]), _d(r["hmin"]), _d(r["nmin"]), _d(r["pvalue"]),
                                          r["nsim"].ctypes.data_as(C.POINTER(C.c_int32)), C.byref(k)))
        assert k.value == n
        return r

    def mica_pair_list(self, site1, site2):
        a = np.ascontiguousarray(site1, dtype=np.int32); b = np.ascontiguousarray(site2, dtype=np.int32)
        mi = np.empty(len(a)); hj = np.empty(len(a))
        self._chk(self.lib.cmb_mica_pair_list(self.h, C.c_int64(len(a)), a.ctypes.data_as(C.POINTER(C.c_int32)),
                                              b.ctypes.data_as(C.POINTER(C.c_int32)), _d(mi), _d(hj)))
        return mi, hj

    def mica_permutations(self, seed, max_permutations=1000, shard_index=0, shard_count=1):
        """null.method = permutations (miTest, Mica.cpp:92-118): Perm.p.value and Perm.nb of every pair, mica's order.
        shard_count > 1: only the pairs idx = shard_index + k * shard_count, row k holding pair idx."""
        n = self.S * (self.S - 1) // 2
        n = max(0, (n - 1 - shard_index) // shard_count + 1) if 0 <= shard_index < shard_count else 0
        pv = np.empty(n); nb = np.empty(n, np.int32)
        k = C.c_int64(0)
        self._chk(self.lib.cmb_mica_permutations_shard(self.h, C.c_uint64(seed), int(max_permutations), int(shard_index),
                                                       int(shard_count), C.c_int64(n), _d(pv), _i32(nb), C.byref(k)))
        assert k.value == n
        return pv, nb

    def mica_null_parametric(self, seed, rep_cpu, rep_ram, K=10, nmax=-1.0, weighted_classes=False, rep_begin=0, rep_end=None):
        """null.method = parametric-bootstrap (Mica.cpp:470-545); returns the [n][3] rows MI, Hjoint, Nmin of the outer
        replicates [rep_begin, rep_end) (default: all of them)."""
        rep_end = rep_cpu if rep_end is None else rep_end
        raw = np.empty((max(0, rep_end - rep_begin) * rep_ram, 3))
        self._chk(self.lib.cmb_mica_null_parametric_range(self.h, C.c_uint64(seed), int(rep_cpu), int(rep_ram), int(rep_begin),
                                                          int(rep_end), int(bool(weighted_classes)), int(K), C.c_double(nmax),
                                                          _d(raw)))
        return raw

    def mica_null_parametric_sharded(self, seed, rep_cpu, rep_ram, K=10, nmax=-1.0, weighted_classes=False, want_raw=False):
        """This rank's share of the parametric-bootstrap replicates, all-gather of the (MI, Nmin) samples and binning of
        the union (cmb_mica_null_parametric_sharded).  want_raw: the rows of this rank's replicates."""
        raw = None
        if want_raw:
            rank, n = self.comm_rank()
            q, m = divmod(rep_cpu, n)
            raw = np.empty(((q + (1 if rank < m else 0)) * rep_ram, 3))
        self._chk(self.lib.cmb_mica_null_parametric_sharded(self.h, C.c_uint64(seed), int(rep_cpu), int(rep_ram),
                                                            int(bool(weighted_classes)), int(K), C.c_double(nmax), _d(raw)))
        return raw

    def null_load(self, stat, key, K, kmax):
        """A null distribution from host arrays: statistics and the key they are binned by."""
        s = np.ascontiguousarray(stat, dtype=np.float64); k = np.ascontiguousarray(key, dtype=np.float64)
        self._chk(self.lib.cmb_null_load(self.h, _d(s), _d(k), C.c_int64(len(s)), int(K), C.c_double(kmax)))

    def set_mi_threshold(self, threshold):
        """Threshold of statistic 'mi' (MI(threshold=0.99) upstream)."""
        self._chk(self.lib.cmb_set_mi_threshold(self.h, C.c_double(threshold)))

    # ------------------------------------------------------------------ multi-GPU
    def comm_init(self, n_ranks, rank, unique_id):
        """Joins the NCCL communicator named by the 128-byte id of comm_unique_id() (one process per GPU)."""
        buf = (C.c_char * 128).from_buffer_copy(bytes(unique_id))
        self._chk(self.lib.cmb_comm_init(self.h, int(n_ranks), int(rank), buf))

    def comm_destroy(self):
        self._chk(self.lib.cmb_comm_destroy(self.h))

    def comm_rank(self):
        r = C.c_int32(); n = C.c_int32()
        self._chk(self.lib.cmb_comm_rank(self.h, C.byref(r), C.byref(n)))
        return r.value, n.value

    def null_intra_sharded(self, stat, seed, rep_cpu, rep_ram, K=10, nmax=-1.0, weighted_classes=False, want_raw=False):
        """This rank's share of the null replicates, ncclAllGather of the samples on the context's stream,
        binning + sort of the union (cmb_null_intra_sharded).  want_raw: the rows of this rank's replicates."""
        raw = None
        if want_raw:
            rank, n = self.comm_rank()
            q, m = divmod(rep_cpu, n)
            raw = np.empty(((q + (1 if rank < m else 0)) * rep_ram, 4))
        self._chk(self.lib.cmb_null_intra_sharded(self.h, STAT[stat], C.c_uint64(seed), rep_cpu, rep_ram,
                                                  int(weighted_classes), K, C.c_double(nmax), _d(raw)))
        return raw

    def set_continuous_rates(self, kind, alpha=1.0, p_invariant=0.0):
        """simulations.continuous: kind 'off' | 'constant' | 'gamma' | 'invariant' (+ gamma)."""
        k = {"off": 0, "constant": 1, "gamma": 2, "invariant": 3}[kind]
        self._chk(self.lib.cmb_set_continuous_rates(self.h, k, C.c_double(alpha), C.c_double(p_invariant)))

    def set_async(self, on=True):
        """null_intra(K=0) returns without waiting for the device (order consumers with sync())."""
        self._chk(self.lib.cmb_set_async(self.h, int(on)))

    def null_samples_dev(self):
        s = C.c_void_p(); m = C.c_void_p(); n = C.c_int64()
        self._chk(self.lib.cmb_null_samples_dev(self.h, C.byref(s), C.byref(m), C.byref(n)))
        return s.value, m.value, n.value

    def null_load_dev(self, stat_ptr, nmin_ptr, n, K, nmax=-1.0):
        self._chk(self.lib.cmb_null_load_dev(self.h, C.c_void_p(stat_ptr), C.c_void_p(nmin_ptr), C.c_int64(n), K,
                                             C.c_double(nmax)))

    def null_get(self):
        K = C.c_int32(); nmax = C.c_double()
        self._chk(self.lib.cmb_null_get(self.h, C.byref(K), C.byref(nmax), None, None, C.c_int64(0)))
        offs = np.zeros(K.value + 1, np.int64)
        self._chk(self.lib.cmb_null_get(self.h, C.byref(K), C.byref(nmax), _i64(offs), None, C.c_int64(0)))
        srt = np.empty(max(1, offs[-1]))
        self._chk(self.lib.cmb_null_get(self.h, C.byref(K), C.byref(nmax), _i64(offs), _d(srt), C.c_int64(len(srt))))
        return dict(K=K.value, nmax=nmax.value, bin_offsets=offs, sorted=srt[:offs[-1]])

    # ------------------------------------------------------------------ pairs
    def pairs(self, stat, use_null=True, filters=None, shard_index=0, shard_count=1, columns=None, capacity=None):
        """columns: subset of {'i','j','stat','rcmin','prmin','nmin','pvalue','nsim'} (default: all)."""
        S = self.S
        cap = S * (S - 1) // 2 if capacity is None else capacity
        cols = set(columns) if columns else {"i", "j", "stat", "rcmin", "prmin", "nmin", "pvalue", "nsim"}
        if not use_null:
            cols -= {"pvalue", "nsim"}
        f = Filters(0, -1, 0.0, -1.0, 0.0)
        if filters:
            for k, v in filters.items():
                setattr(f, k, v)
        mk = lambda name, dt: np.empty(cap, dt) if name in cols else None
        oi, oj = mk("i", np.int32), mk("j", np.int32)
        st, rcm, prm, nm = mk("stat", np.float64), mk("rcmin", np.int32), mk("prmin", np.float64), mk("nmin", np.float64)
        pv, ns = mk("pvalue", np.float64), mk("nsim", np.int32)
        nr = C.c_int64()
        self._chk(self.lib.cmb_pairs(self.h, STAT[stat], C.byref(f), int(use_null), shard_index, shard_count,
                                     C.c_int64(cap), _i32(oi), _i32(oj), _d(st), _i32(rcm), _d(prm), _d(nm), _d(pv),
                                     _i32(ns), C.byref(nr)))
        k = nr.value
        out = dict(i=oi, j=oj, stat=st, rcmin=rcm, prmin=prm, nmin=nm, pvalue=pv, nsim=ns)
        return {name: (a[:k] if a is not None else None) for name, a in out.items()}, k

    def load_vectors(self, n):
        """Replaces the mapping of the mapped alignment with vectors read from a file
        (input.vectors.file, CoETools.cpp:374-385); returns their norms."""
        n = _f64(n)
        assert n.shape == (self.S, self.B)
        norm = np.empty(self.S)
        self._chk(self.lib.cmb_load_vectors(self.h, _d(n), _d(norm)))
        return norm

    # ------------------------------------------------------------------ candidate groups
    def candidates(self, stat, groups, omega=0.25, min_sim=1000, max_trials=10, rep_ram=1000, seed=0,
                   weighted_classes=False, analysable=None):
        """groups: list of lists of site indices (of the mapped alignment).  Returns the observed
        group statistics, p-values (n1+1)/(n2+1), n1, n2 and the number of simulated sites
        (CoMap.cpp:592-711; CoETools.cpp:901-1087)."""
        off = np.zeros(len(groups) + 1, np.int64)
        off[1:] = np.cumsum([len(g) for g in groups])
        sites = np.ascontiguousarray(np.concatenate([np.asarray(g, np.int32) for g in groups]) if len(groups) else
                                     np.zeros(0, np.int32), dtype=np.int32)
        an = None if analysable is None else np.ascontiguousarray(analysable, dtype=np.uint8)
        G = len(groups)
        st, pv = np.empty(G), np.empty(G)
        n1, n2 = np.empty(G, np.int64), np.empty(G, np.int64)
        ns = C.c_int64()
        self._chk(self.lib.cmb_candidates(self.h, STAT[stat], G, _i64(off), _i32(sites), _p(an, C.c_uint8),
                                          C.c_double(omega), C.c_int64(min_sim), int(max_trials), int(rep_ram),
                                          C.c_uint64(seed), int(weighted_classes), _d(st), _d(pv), _i64(n1), _i64(n2),
                                          C.byref(ns)))
        return dict(stat=st, pvalue=pv, n1=n1, n2=n2, n_simulated=ns.value)

    # ------------------------------------------------------------------ two data sets
    def pairs_inter(self, other, stat, filters=None, min_rate_class2=0, min_rate2=0.0, independent=False,
                    nmin_by_row=True):
        """Statistic of every site of this data set with every site of `other` (CoETools.cpp:732-840);
        independent: site i with site i only.  nmin_by_row reproduces upstream's Nmin (norms2[i])."""
        cap = self.S if independent else self.S * other.S
        f = Filters(0, -1, 0.0, -1.0, 0.0)
        if filters:
            for k, v in filters.items():
                setattr(f, k, v)
        oi, oj = np.empty(cap, np.int32), np.empty(cap, np.int32)
        st, rcm, prm, nm = np.empty(cap), np.empty(cap, np.int32), np.empty(cap), np.empty(cap)
        nr = C.c_int64()
        self._chk(self.lib.cmb_pairs_inter(self.h, other.h, STAT[stat], C.byref(f), int(min_rate_class2),
                                           C.c_double(min_rate2), int(independent), int(nmin_by_row), C.c_int64(cap),
                                           _i32(oi), _i32(oj), _d(st), _i32(rcm), _d(prm), _d(nm), C.byref(nr)))
        k = nr.value
        return dict(i=oi[:k], j=oj[:k], stat=st[:k], rcmin=rcm[:k], prmin=prm[:k], nmin=nm[:k]), k

    def null_inter(self, other, stat, seed, rep_cpu, rep_ram, weighted_classes=False, rep_begin=0, rep_end=None):
        """rep_cpu x rep_ram paired null statistics of the two data sets' simulators
        (AnalysisTools.cpp:662-735); rows Stat, RCmin, PRmin, Nmin of the outer replicates [rep_begin, rep_end)."""
        rep_end = rep_cpu if rep_end is None else rep_end
        raw = np.empty((max(0, rep_end - rep_begin) * rep_ram, 4))
        self._chk(self.lib.cmb_null_inter_range(self.h, other.h, STAT[stat], C.c_uint64(seed), rep_cpu, rep_ram,
                                                rep_begin, rep_end, int(weighted_classes), _d(raw)))
        return raw

    COLS = ("i", "j", "stat", "rcmin", "prmin", "nmin", "pvalue", "nsim")
    COL_DTYPE = (np.int32, np.int32, np.float64, np.int32, np.float64, np.float64, np.float64, np.int32)

    def pairs_resident(self, stat, use_null=True, filters=None, shard_index=0, shard_count=1, columns=0xFF):
        f = Filters(0, -1, 0.0, -1.0, 0.0)
        if filters:
            for k, v in filters.items():
                setattr(f, k, v)
        nr = C.c_int64()
        self._chk(self.lib.cmb_pairs_resident(self.h, STAT[stat], C.byref(f), int(use_null), shard_index,
                                              shard_count, C.c_uint32(columns), C.byref(nr)))
        return nr.value

    def pairs_fetch(self, column, host_array):
        """Asynchronous copy of one resident column into host_array (pinned for speed); sync() after."""
        self._chk(self.lib.cmb_pairs_fetch(self.h, column, C.c_void_p(host_array.ctypes.data),
                                           C.c_int64(host_array.size)))

    # ------------------------------------------------------------------ clustering
    def distance_matrix(self, dist, want=True):
        mat = np.empty((self.S, self.S)) if want else None
        self._chk(self.lib.cmb_distance_matrix(self.h, DIST[dist], _d(mat)))
        return mat

    def cluster(self, linkage):
        S = self.S
        left = np.empty(S - 1, np.int32); right = np.empty(S - 1, np.int32); height = np.empty(S - 1)
        self._chk(self.lib.cmb_cluster(self.h, LINK[linkage], _i32(left), _i32(right), _d(height)))
        return left, right, height

    def groups(self, dist, max_size, as_lists=True):
        """as_lists=False returns the flat member array and its offsets instead of one array per group."""
        S = self.S
        members = np.empty(max(1, (S - 1) * max_size), np.int32); offs = np.zeros(S + 1, np.int64)
        gh = np.empty(S); gs = np.empty(S); gn = np.empty(S); ng = C.c_int64()
        self._chk(self.lib.cmb_groups(self.h, DIST[dist], max_size, _i32(members), _i64(offs), _d(gh), _d(gs),
                                      _d(gn), C.byref(ng)))
        k = ng.value
        if not as_lists:
            return dict(members_flat=members[:offs[k]], offsets=offs[:k + 1], height=gh[:k], stat=gs[:k], nmin=gn[:k])
        return dict(members=[members[offs[g]:offs[g + 1]].copy() for g in range(k)], height=gh[:k], stat=gs[:k],
                    nmin=gn[:k])

    def cluster_null(self, dist, linkage, seed, rep_begin, rep_end, max_size, weighted_classes=False, as_lists=True):
        S = self.S
        nrep = rep_end - rep_begin
        cap_rows = nrep * (S - 1); cap_mem = cap_rows * max_size
        rep = np.empty(cap_rows, np.int32); size = np.empty(cap_rows, np.int32)
        dmax = np.empty(cap_rows); st = np.empty(cap_rows); nm = np.empty(cap_rows)
        members = np.empty(max(1, cap_mem), np.int32); offs = np.zeros(cap_rows + 1, np.int64); nr = C.c_int64()
        self._chk(self.lib.cmb_cluster_null(self.h, DIST[dist], LINK[linkage], C.c_uint64(seed), rep_begin, rep_end,
                                            int(weighted_classes), max_size, C.c_int64(cap_rows), C.c_int64(cap_mem),
                                            _i32(rep), _i32(size), _d(dmax), _d(st), _d(nm), _i32(members), _i64(offs),
                                            C.byref(nr)))
        k = nr.value
        if not as_lists:
            return dict(rep=rep[:k], size=size[:k], dmax=dmax[:k], stat=st[:k], nmin=nm[:k], members_flat=members[:offs[k]],
                        offsets=offs[:k + 1])
        return dict(rep=rep[:k], size=size[:k], dmax=dmax[:k], stat=st[:k], nmin=nm[:k],
                    members=[members[offs[g]:offs[g + 1]].copy() for g in range(k)])

    # ------------------------------------------------------------------ measurement
    def profile_enable(self, on=True):
        self.lib.cmb_profile_enable(self.h, int(on))

    def profile_reset(self):
        self._chk(self.lib.cmb_profile_reset(self.h))

    def profile_get(self, name):
        ms = C.c_double(); n = C.c_int64()
        self._chk(self.lib.cmb_profile_get(self.h, name.encode(), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def launch_count(self):
        return int(self.lib.cmb_launch_count(self.h))
