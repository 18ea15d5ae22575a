"""Static SASS opcode counts of the hot kernels (cuobjdump -sass of the built objects): the proof that the
tensor-core (DMMA) and TMA (UBLKCP) paths are what the kernels are made of, and how much local memory
(LDL / STL: spills and the message stack) they touch.   python tools/sass_counts.py > profiles/r2_sass_opcodes.txt"""
import collections, os, re, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = os.path.join(ROOT, "comap_b200", "build")
WANT = [("k1_mma.cu.o", r"k1_up_mmaILi2ELi4ELi128ELi2ELb1E"), ("k1_mma.cu.o", r"k1_down_mmaILi2ELi4ELi128ELi2E"),
        ("k1_mma.cu.o", r"k1_up_mmaILi2ELi4ELi32ELi2ELb0E"), ("k1_mma20.cu.o", r"k1_up_mma20ILi2ELb1E"),
        ("k1_mma20.cu.o", r"k1_down_mma20ILi2ELb1E"), ("k2_pairs.cu.o", r"k2_tilesILi0E"),
        ("k2_pairs.cu.o", r"k2_pairedILi0E"), ("k3_simulate.cu.o", r"k3_simulate"), ("k4_rnn.cu.o", r"k4r_rounds"),
        ("k4_cluster.cu.o", r"k4_clusterILi1E"), ("k5_mica.cu.o", r"k5_permutationsILi4ELi5E"), ("k5_mica.cu.o", r"k5_pairsILi4E"),
        ("k5_mica.cu.o", r"k5_pairsILi20E")]
KEYS = ["DMMA", "DFMA", "DMUL", "DADD", "UBLKCP", "SYNCS", "LDS", "STS", "LDL", "STL", "LDG", "STG", "SHFL", "REDUX", "ATOMG", "BAR", "VOTE"]
print("# cuobjdump -sass opcode counts (static) of the sm_100a objects; DMMA = FP64 tensor-core MMA, UBLKCP = cp.async.bulk (TMA),")
print("# SYNCS = mbarrier ops, LDL/STL = local memory (message stack + spills)")
print("%-44s %6s " % ("kernel", "instr") + " ".join("%6s" % k for k in KEYS))
for obj, pat in WANT:
    txt = subprocess.run(["cuobjdump", "-sass", os.path.join(OBJ, obj)], capture_output=True, text=True).stdout
    cur, counts = None, collections.defaultdict(collections.Counter)
    for ln in txt.splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            cur = m.group(1); continue
        m = re.match(r"\s+/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", ln)
        if m and cur:
            counts[cur][m.group(1)] += 1
    for fn, c in counts.items():
        if re.search(pat, fn):
            name = subprocess.run(["c++filt", fn], capture_output=True, text=True).stdout.strip()
            name = name.replace("(anonymous namespace)::", "").replace("cmb::", "").replace("void ", "")
            name = re.sub(r"\(.*", "", name)[:44]
            print("%-44s %6d " % (name, sum(c.values())) + " ".join("%6d" % c.get(k, 0) for k in KEYS))
            break
