"""Strong scaling of mica's permutation test over GPUs (comap_b200.gpus=N on the mica command line).

    python tools/mica_scaling.py [--sites 3000] [--steps 5] [--max-gpus 8]

One process, one context per device, each holding the same alignment: the columns of examples/RNA/BacteriaSSU
(tests/golden/bacteria_ssu.npz, 760 sites x 40 taxa) resampled with replacement to --sites columns with a fixed seed.
The duplicated columns give pairs that run all 1000 shuffles, as coevolving stems do; the other pairs keep the
fixture's spread.  For N = 1, 2, 4, 8 (up to the devices present) GPU r tests the pairs r, r + N, r + 2N, ... on
its own host thread (cmb_mica_permutations_shard; N = 1 is the one-call cmb_mica_permutations), after a warm-up
call per context.  A call is timed from the first launch to the last device synchronise.

Prints one JSON line per N: the card's name and power limit (nvidia-smi's query form, read in the same run), ms per
call, pairs/s, each GPU's kernel time (the context's profile of k5_permutations, from a separate profiled call) and an
order-independent checksum of the (pair, p-value, shuffle count) rows, which must be the same at every N.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    except OSError:
        return "unknown", "unknown"
    first = q.stdout.strip().split("\n")[0].split(",") if q.returncode == 0 and q.stdout.strip() else ["unknown", "unknown"]
    return first[0].strip(), first[1].strip()


def alignment(sites, seed):
    """The fixture as options_perm.mica reads it (the binary's own parser, via its --dry-run dump), columns resampled."""
    from comap_b200 import build as b
    from test_host import BIN, write_fixture, dry_run, decode
    b.build_host()
    with tempfile.TemporaryDirectory() as tmp:
        write_fixture(tmp, "bacteria_ssu")
        p, o = dry_run(BIN, tmp, "param=options_perm.mica")
        if p.returncode != 0:
            raise RuntimeError(p.stdout[-2000:])
    c = decode(o)
    row = {name: k for k, name in enumerate(o["leaves"])}
    codes = c["codes"][[row[name] for name in o["sequences"]]]
    cols = np.random.default_rng(seed).integers(0, codes.shape[1], size=sites)
    c["codes"] = np.ascontiguousarray(codes[:, cols])
    c["parent"] = c["parent"].astype(np.int32)
    return c


def checksum(pv, nb):
    """Sum over rows of a 64-bit mix of (pair index, p-value bits, shuffle count): independent of the rows' order."""
    idx = np.arange(len(pv), dtype=np.uint64)
    h = idx * np.uint64(0x9E3779B97F4A7C15) ^ pv.view(np.uint64) ^ (nb.astype(np.uint64) << np.uint64(40))
    h ^= h >> np.uint64(29)
    h *= np.uint64(0xBF58476D1CE4E5B9)
    h ^= h >> np.uint64(32)
    return "%016x" % int(h.sum(dtype=np.uint64))


def run(ctxs, seed, max_perm, n_pairs):
    """The whole permutation test over len(ctxs) GPUs; rows scattered back to pair order."""
    n = len(ctxs)
    if n == 1:
        return ctxs[0].mica_permutations(seed, max_perm)
    pv, nb, err = np.empty(n_pairs), np.empty(n_pairs, np.int32), []

    def work(r):
        try:
            p, k = ctxs[r].mica_permutations(seed, max_perm, shard_index=r, shard_count=n)
            pv[r::n] = p; nb[r::n] = k
        except Exception as e:  # noqa: BLE001
            err.append(e)

    th = [threading.Thread(target=work, args=(r,)) for r in range(n)]
    [t.start() for t in th]; [t.join() for t in th]
    if err:
        raise err[0]
    return pv, nb


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=3000)
    ap.add_argument("--seed", type=int, default=2026, help="column resampling")
    ap.add_argument("--perm-seed", type=int, default=21)
    ap.add_argument("--max-perm", type=int, default=1000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--max-gpus", type=int, default=8)
    args = ap.parse_args()
    import torch
    from comap_b200 import api
    n_dev = torch.cuda.device_count()
    if n_dev < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    name, power = card()
    c = alignment(args.sites, args.seed)
    S = c["codes"].shape[1]
    n_pairs = S * (S - 1) // 2
    ctxs = []
    for d in range(min(n_dev, args.max_gpus)):
        ctx = api.Context(device=d)
        ctx.set_tree(c["parent"], c["brlen"]); ctx.set_model(c["Q"], c["pi"], c["rates"], c["probs"])
        ctx.set_alignment(c["codes"], c["code_mask"])
        ctxs.append(ctx)
    for n in (1, 2, 4, 8):
        if n > len(ctxs):
            break
        use = ctxs[:n]
        run(use, args.perm_seed, args.max_perm, n_pairs)                      # warm-up: module load, shared-memory set-up
        times = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            pv, nb = run(use, args.perm_seed, args.max_perm, n_pairs)
            for ctx in use:
                ctx.sync()
            times.append((time.perf_counter() - t0) * 1e3)
        for ctx in use:
            ctx.profile_reset(); ctx.profile_enable(True)
        run(use, args.perm_seed, args.max_perm, n_pairs)
        kernel_ms = [ctx.profile_get("mica_perm")[0] for ctx in use]
        for ctx in use:
            ctx.profile_enable(False)
        ms = float(np.median(times))
        print(json.dumps(dict(tool="mica_scaling", gpu=name, power_limit=power, n_gpus=n, sites=S, taxa=int(c["codes"].shape[0]),
                              pairs=n_pairs, max_permutations=args.max_perm, mi_evaluations=int(nb.sum()) + n_pairs,
                              steps=args.steps, ms_per_call=ms, ms_min=float(min(times)), ms_max=float(max(times)),
                              pairs_per_s=n_pairs / (ms * 1e-3), kernel_ms_per_gpu=kernel_ms,
                              checksum=checksum(pv, nb))), flush=True)
    for ctx in ctxs:
        ctx.close()


if __name__ == "__main__":
    main()
