"""Regenerates tests/golden/*.npz from a checkout of the reference (CoMap's source tree).

    python tests/golden/make_golden.py <path to the CoMap source tree>

The reference ships exactly one set of numerical outputs for the hot path
(examples/Proteins/Benchmark/CoMap/Myo_*.vec + Myo.infos, SURVEY.md s4/s8c).  They and the
inputs that produced them (Myoglobin alignment + tree) are packed into one .npz so the
tests need nothing outside this repository.  The .vec tables are stored as tab-separated
text with the reference's 6 significant digits (tests/helpers.py golden() parses them back),
which keeps the file under 1 MB.  The RNA example's inputs are packed too (no expected
outputs exist for it).
"""
import numpy as np, os, sys
HERE = os.path.dirname(os.path.abspath(__file__))

def load_vec(p):
    ls = open(p).read().strip().split("\n")
    hdr = ls[0].split("\t")
    rows = [l.split("\t") for l in ls[1:]]
    M = np.array([[float(x) for x in r[1:]] for r in rows])
    return np.array([int(h[4:]) for h in hdr[2:]]), M[:, 0], M[:, 1:]

def pack_bacteria():
    """examples/RNA/BacteriaSSU: alignment, tree, comap's option file and mica's four option files, as shipped."""
    r = REF + "/examples/RNA/BacteriaSSU/"
    rd = lambda fn: np.frombuffer(open(r + fn, "rb").read(), dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, "bacteria_ssu.npz"), phy=rd("Bacteria_SSU.40.phy"), dnd=rd("Bacteria_SSU.ML.dnd"),
                        options=rd("options.comap"), mica_pbs=rd("options_pbs.mica"), mica_npbs=rd("options_npbs.mica"),
                        mica_perm=rd("options_perm.mica"), mica_zscore=rd("options_zscore.mica"))


def main():
    bm = REF + "/examples/Proteins/Benchmark/CoMap/"
    out = {}
    for k in ("unif", "decomp", "naive", "laplace", "unif_grantham", "decomp_grantham", "naive_grantham"):
        coords, mean, M = load_vec(bm + "Myo_%s.vec" % k)
        txt = "".join("\t".join("%.6g" % v for v in row) + "\n" for row in M)   # [branch][site], 6 significant digits
        out["vec_" + k] = np.frombuffer(txt.encode(), dtype=np.uint8)
    out["vec_coords"] = coords
    out["vec_brlen"] = mean
    inf = [l.split("\t") for l in open(bm + "Myo.infos").read().strip().split("\n")[1:]]
    out["infos_coord"] = np.array([int(r[0][1:-1]) for r in inf])
    out["infos_complete"] = np.array([int(r[1]) for r in inf])
    out["infos_const"] = np.array([int(r[2]) for r in inf])
    out["infos_rc"] = np.array([int(r[3]) for r in inf])
    out["infos_pr"] = np.array([float(r[4]) for r in inf])
    out["infos_logl"] = np.array([float(r[5]) for r in inf])
    d = REF + "/examples/Data/Proteins/Myoglobin/"
    out["mase"] = np.frombuffer(open(d + "Myoglobin.aln.sel.mase", "rb").read(), dtype=np.uint8)
    out["dnd"] = np.frombuffer(open(d + "Myo.dnd", "rb").read(), dtype=np.uint8)
    out["options"] = np.frombuffer(open(bm + "comap.bpp", "rb").read(), dtype=np.uint8)
    # BASELINE configs[0] and its siblings: the option files of examples/simple/* (same alignment and tree)
    for ex in ("ProteinPairCorrelation", "ProteinPairCompensation", "ProteinGroupCorrelation", "ProteinGroupCompensation",
               "ProteinMappingOnly"):
        out["simple_" + ex] = np.frombuffer(open(REF + "/examples/simple/" + ex + "/comap.bpp", "rb").read(), dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, "myoglobin.npz"), **out)
    pack_bacteria()
    s = REF + "/examples/Data/Proteins/SRK/"
    np.savez_compressed(os.path.join(HERE, "srk.npz"),
        mase=np.frombuffer(open(s + "SRK.mase", "rb").read(), dtype=np.uint8),
        dnd=np.frombuffer(open(s + "SRK.dnd", "rb").read(), dtype=np.uint8))

if __name__ == "__main__":
    REF = sys.argv[1]
    main()
