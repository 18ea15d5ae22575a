"""Test-side helpers: mini readers for the reference's input formats and an independent
numpy restatement of likelihood + mapping (second opinion for the C oracle)."""
import io
import os
import re
import numpy as np
from comap_b200 import synthetic as syn

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    """The arrays of tests/golden/<name>.npz.  The reference's .vec tables are stored as their text (tab-separated,
    6 significant digits, one row per branch), which keeps the file small; they come back as float64 [branch][site]."""
    with np.load(os.path.join(GOLDEN, name + ".npz")) as z:
        return {k: np.loadtxt(io.StringIO(text(z[k])), delimiter="\t", ndmin=2) if k.startswith("vec_") and z[k].dtype == np.uint8
                else z[k] for k in z.files}


def text(arr):
    return bytes(arr).decode()


def read_mase(txt):
    names, seqs, cur = [], [], None
    for ln in txt.split("\n"):
        if ln.startswith(";;"):
            continue
        if ln.startswith(";"):
            cur = "name"; continue
        if cur == "name":
            names.append(ln.strip()); seqs.append(""); cur = "seq"; continue
        if cur == "seq":
            seqs[-1] += ln.strip()
    return names, seqs


def read_phylip_sequential_extended(txt):
    lines = txt.split("\n")
    n, L = [int(x) for x in lines[0].split()]
    names, seqs = [], []
    k = 1
    while len(names) < n:
        ln = lines[k]; k += 1
        if not ln.strip():
            continue
        parts = ln.split(None, 1)
        names.append(parts[0]); s = parts[1].replace(" ", "") if len(parts) > 1 else ""
        while len(s) < L:
            s += lines[k].replace(" ", "").strip(); k += 1
        seqs.append(s)
    return names, seqs


def parse_newick(s):
    """Returns (parent, brlen, leaf_names) with post-order ids (leaf_names in leaf id order)."""
    s = s.strip().rstrip(";").strip()
    pos = 0
    parent, brlen, names, kids = [], [], [], []

    def rec():
        nonlocal pos
        ch = []
        if s[pos] == "(":
            pos += 1
            while True:
                ch.append(rec())
                if s[pos] == ",":
                    pos += 1; continue
                if s[pos] == ")":
                    pos += 1; break
        m = re.match(r"[^:,()]*", s[pos:]); name = m.group(0); pos += len(name)
        ln = 0.0
        if pos < len(s) and s[pos] == ":":
            pos += 1
            m = re.match(r"[-+0-9.eE]+", s[pos:]); ln = float(m.group(0)); pos += len(m.group(0))
        nid = len(parent)
        parent.append(-1); brlen.append(ln); names.append(name.strip()); kids.append(ch)
        for c in ch:
            parent[c] = nid
        return nid

    rec()
    leaf_names = [names[i] for i in range(len(parent)) if not kids[i]]
    return np.array(parent, np.int32), np.array(brlen), leaf_names


PROT_AMBIG = {"B": "DN", "Z": "EQ", "J": "IL", "X": syn.AA_ORDER, "?": syn.AA_ORDER, "-": syn.AA_ORDER}
NUC_AMBIG = {"R": "AG", "Y": "CT", "S": "CG", "W": "AT", "K": "GT", "M": "AC", "B": "CGT", "D": "AGT",
             "H": "ACT", "V": "ACG", "N": "ACGT", "X": "ACGT", "?": "ACGT", "-": "ACGT", "O": "ACGT", "0": "ACGT"}


def encode_alignment(names, seqs, leaf_names, states, ambig, cols):
    """codes [T][S] (rows in leaf order) + code_mask; one code per distinct character."""
    row = {n: i for i, n in enumerate(names)}
    chars = sorted(set("".join(seqs[row[l]][c] for l in leaf_names for c in cols)))
    code_of = {}
    mask = []
    for k, st in enumerate(states):
        code_of[st] = k; mask.append(1 << k)
    for ch in chars:
        u = ch.upper()
        if u == "U":
            u = "T"
        if u in code_of:
            code_of[ch] = code_of[u]; continue
        m = 0
        for c in ambig[u]:
            m |= 1 << states.index(c)
        code_of[ch] = len(mask); mask.append(m)
    codes = np.array([[code_of[seqs[row[l]][c]] for c in cols] for l in leaf_names], dtype=np.uint8)
    return codes, np.array(mask, dtype=np.uint32)


def is_constant(col, states):
    st = set(c for c in col if c in states)
    return len(st) <= 1


def myoglobin_inputs():
    """The Benchmark/CoMap run: Myoglobin, nogap + remove_const, JTT92 + Gamma(4, 0.985435)."""
    g = golden("myoglobin")
    names, seqs = read_mase(text(g["mase"]))
    parent, brlen, leaf_names = parse_newick(text(g["dnd"]))
    L = len(seqs[0])
    nogap = [j for j in range(L) if all(s[j] != "-" for s in seqs)]
    cols = [j for j in nogap if not is_constant([s[j] for s in seqs], syn.AA_ORDER)]
    codes, mask = encode_alignment(names, seqs, leaf_names, list(syn.AA_ORDER), PROT_AMBIG, cols)
    Q, pi = syn.jtt92()
    rates, probs = syn.gamma_rates(0.985435, 4)
    return dict(parent=parent, brlen=brlen, Q=Q, pi=pi, rates=rates, probs=probs, codes=codes,
                code_mask=mask, coords=np.array(cols) + 1, golden=g)


def random_dna_case(T, S, seed, mean_brlen=0.05, alpha=0.5, C=4, ambiguity=0.0):
    parent, brlen = syn.random_tree(T, seed, mean_brlen)
    Q, pi = syn.hky85(2.5, [0.3, 0.2, 0.2, 0.3])
    rates, probs = syn.gamma_rates(alpha, C)
    rng = np.random.default_rng(seed + 1)
    codes = simulate_np(parent, brlen, Q, pi, rates, rng, S)
    mask = syn.identity_code_mask(4)
    if ambiguity > 0:
        codes = np.where(rng.random(codes.shape) < ambiguity, 4, codes).astype(np.uint8)
    return dict(parent=parent, brlen=brlen, Q=Q, pi=pi, rates=rates, probs=probs, codes=codes,
                code_mask=mask)


def expm_rev(Q, pi, t):
    s = np.sqrt(pi)
    M = Q * s[:, None] / s[None, :]
    w, V = np.linalg.eigh((M + M.T) / 2)
    return (V * np.exp(w * t)) @ V.T * s[None, :] / s[:, None]


def simulate_np(parent, brlen, Q, pi, rates, rng, S):
    """numpy forward simulation (test data only; not the Philox stream)."""
    n = len(parent)
    cls = rng.integers(0, len(rates), size=S)
    st = np.zeros((n, S), dtype=np.int64)
    st[n - 1] = rng.choice(len(pi), size=S, p=pi / pi.sum())
    has_child = np.zeros(n, bool); has_child[parent[parent >= 0]] = True
    for v in range(n - 2, -1, -1):
        Ps = np.stack([expm_rev(Q, pi, max(brlen[v], 1e-6) * r) for r in rates])
        cum = np.cumsum(Ps[cls, st[parent[v]]], axis=1)
        u = rng.random(S)
        st[v] = np.minimum((u[:, None] >= cum).sum(1), len(pi) - 1)
    return st[~has_child].astype(np.uint8)


def unif_counts_np(Q, pi, T, weights=None):
    from math import lgamma, log, exp
    A = len(pi)
    if T == 0:
        return np.zeros((A, A))
    mu = np.max(-np.diag(Q)); R = np.eye(A) + Q / mu
    Bm = Q.copy(); np.fill_diagonal(Bm, 0)
    if weights is not None:
        Bm = Bm * weights
    lam = mu * T; nmax = int(np.ceil(4 + 6 * np.sqrt(lam) + lam))
    s = Bm.copy(); Rp = np.eye(A); cnt = np.zeros((A, A))
    for l in range(nmax + 1):
        if l > 0:
            Rp = Rp @ R; s = s @ R + Rp @ Bm
        cnt += s * exp((l + 1) * log(lam) - lam - log(mu) - lgamma(l + 2))
    with np.errstate(all="ignore"):
        c = cnt / expm_rev(Q, pi, T)
    c[~np.isfinite(c)] = 0
    if weights is None:
        c[c < 0] = 0
    return c


def map_np(parent, brlen, Q, pi, rates, probs, codes, code_mask, weights=None):
    """Independent numpy restatement (einsum, LAPACK eigh) of SURVEY.md s3.3."""
    n = len(parent); A = len(pi); C = len(rates); root = n - 1
    T, S = codes.shape
    kids = [[] for _ in range(n)]
    for v in range(n - 1):
        kids[parent[v]].append(v)
    leaf_row = {}
    for v in range(n):
        if not kids[v]:
            leaf_row[v] = len(leaf_row)
    tip = ((code_mask[codes][:, :, None] >> np.arange(A)[None, None, :]) & 1).astype(np.float64)
    P, W = {}, {}
    for v in range(n - 1):
        d = max(brlen[v], 1e-6)
        P[v] = np.stack([expm_rev(Q, pi, d * r) for r in rates])
        W[v] = np.stack([unif_counts_np(Q, pi, d * r, weights) for r in rates]) * P[v]
    D = {}
    for v in range(n):
        if not kids[v]:
            D[v] = np.broadcast_to(tip[leaf_row[v]], (C, S, A)).copy()
        else:
            x = np.ones((C, S, A))
            for c in kids[v]:
                x *= np.einsum("cxy,csy->csx", P[c], D[c])
            D[v] = x
    Lc = (D[root] * pi).sum(2)
    Ls = (Lc * probs[:, None]).sum(0)
    Up = {}
    out = np.zeros((S, n - 1))
    for v in range(n - 2, -1, -1):
        f = parent[v]
        u = np.ones((C, S, A))
        for w in kids[f]:
            if w != v:
                u *= np.einsum("cxy,csy->csx", P[w], D[w])
        if f == root:
            u *= pi
        else:
            u *= np.einsum("cyx,csy->csx", P[f], Up[f])
        Up[v] = u
        out[:, v] = np.einsum("c,csx,cxy,csy->s", probs, u, W[v], D[v]) / Ls
    return dict(n=out, norm=np.sqrt((out ** 2).sum(1)), loglik=np.log(Ls),
                post_rate=(rates[:, None] * probs[:, None] * Lc).sum(0) / Ls, rate_class=Lc.argmax(0))
