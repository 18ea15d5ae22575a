#!/usr/bin/env python
"""bench.py -- CoMap hot path on B200: site-pairs scored per second, mapping + null included.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[3], SURVEY.md s8d "config 4"): synthetic 5,000-site x
500-taxon nucleotide alignment, HKY85(kappa=2.5, pi=.3/.2/.2/.3) + Gamma(4, alpha=0.5),
random-join tree with Exp(0.02) branches (numpy seed 20251018); one step =
  map the alignment -> parametric-bootstrap null (1000 x 1000 paired simulated sites:
  2,000,000 sites simulated + mapped, 1,000,000 null statistics, binned by Nmin and sorted)
  -> all 12,497,500 site pairs scored (correlation) with p-values.
pairs per step = S(S-1)/2 + rep_cpu*rep_ram (BASELINE.md B5).

`value`  : device-resident throughput (inputs in HBM, results left in HBM), CUDA events.
`e2e`    : same step through the C ABI with host buffers: alignment H2D from pinned memory,
           per-site columns and all 8 pair-table columns D2H into pinned memory.
`roofline`: the dominant kernel family (K1 mapping pass: down + finish + up launches over
           one batch of sites), algorithmic bytes per site from SURVEY.md s8(d).
`cpu_baseline` / --impl reference: the CPU oracle port of the reference's algorithm
           (the upstream binary needs Bio++ and cannot be built here) on a bounded sample,
           extrapolated linearly to the full step and labelled as such.  The reference is
           single-threaded; like its users we run one process per host core (shards of the
           null replicates and pair rows), all at once, and add their throughputs.
Multi-GPU: strong scaling of the same job -- null replicates and pair rows are sharded,
null samples are all-gathered with NCCL, every rank bins/sorts the union.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from comap_b200 import synthetic as syn  # noqa: E402

CFG = dict(sites=5000, taxa=500, kappa=2.5, pi=[0.3, 0.2, 0.2, 0.3], alpha=0.5, classes=4,
           mean_brlen=0.02, tree_seed=20251018, aln_seed=1, null_seed=2, rep_cpu=1000, rep_ram=1000,
           null_bins=10, statistic="correlation")


def workload(cfg):
    parent, brlen = syn.random_tree(cfg["taxa"], cfg["tree_seed"], cfg["mean_brlen"])
    Q, pi = syn.hky85(cfg["kappa"], cfg["pi"])
    rates, probs = syn.gamma_rates(cfg["alpha"], cfg["classes"])
    return dict(parent=parent, brlen=brlen, Q=Q, pi=pi, rates=rates, probs=probs,
                code_mask=syn.identity_code_mask(4))


def algorithmic_bytes_per_site(T, C, A, B):
    """SURVEY.md s8(d), K1: tips + inner down-partials written once and read once + output."""
    return T + 2 * (T - 3) * C * A * 8 + 8 * B + 28


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.p = index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for ln in self.p.stdout:
            self.rows.append(ln.strip().split(", "))

    def stop(self):
        if not self.p:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.p.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for k, nm in enumerate(names):
                    if r[4 + k].strip().lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle port on a bounded sample
# ------------------------------------------------------------------------------------------
def cpu_sample(cfg, w, aln_codes=None, sample_sites=None, sample_ram=None, seed=0):
    """Times the oracle (1 thread) on a bounded sample of the step WITH THE STEP'S OWN COMPOSITION.

    The step scores S(S-1)/2 observed pairs and rep_cpu x rep_ram null pairs (two simulated + mapped sites each).  The
    default sample keeps that ratio -- 807 observed sites (325 221 pairs) and 26 outer replicates of 1000 null pairs,
    1/38 of configs[3] -- so `value` = pairs of the sample / seconds of the sample is the metric itself, measured, and
    nothing is extrapolated; the p-value scan runs against a null of the full step's size (its cost per pair is the
    reference's linear scan of a bin, CoETools.cpp:712-716).  Components timed: (a) simulate + map + paired statistic
    of the null pairs, replicate by replicate as AnalysisTools.cpp:589-656 does, (b) mapping of the observed sites,
    (c) all their pairs with p-values.  The linear per-unit model of round 1 is still reported (`extrapolated_value`).
    """
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding as O
    S, R, RC, K = cfg["sites"], cfg["rep_ram"], cfg["rep_cpu"], cfg["null_bins"]
    if sample_sites is None:
        sample_sites = min(S, 807)
    if sample_ram is None:   # null pairs in the proportion of the step
        sample_ram = max(1, int(round(RC * R * (sample_sites * (sample_sites - 1) / 2) / (S * (S - 1) / 2))))
    reps = (sample_ram + 999) // 1000          # outer replicates of at most 1000 pairs, as the real job's
    chunk = (sample_ram + reps - 1) // reps
    sample_ram = reps * chunk
    t0 = time.perf_counter()
    s1 = np.stack([O.simulate(w["parent"], w["brlen"], w["Q"], w["pi"], w["rates"], w["probs"], cfg["null_seed"] + seed,
                              (2 * i) * chunk, chunk)[0] for i in range(reps)])
    s2 = np.stack([O.simulate(w["parent"], w["brlen"], w["Q"], w["pi"], w["rates"], w["probs"], cfg["null_seed"] + seed,
                              (2 * i + 1) * chunk, chunk)[0] for i in range(reps)])
    t_sim = time.perf_counter() - t0
    t0 = time.perf_counter()
    nl = O.null_intra(w["parent"], w["brlen"], w["Q"], w["pi"], w["rates"], w["probs"], cfg["statistic"],
                      s1, s2, K, 10.0)
    t_null = time.perf_counter() - t0
    if aln_codes is None:
        aln_codes, _ = O.simulate(w["parent"], w["brlen"], w["Q"], w["pi"], w["rates"], w["probs"], cfg["aln_seed"], 0, sample_sites)
    t0 = time.perf_counter()
    m = O.map_sites(w["parent"], w["brlen"], w["Q"], w["pi"], w["rates"], w["probs"], aln_codes[:, :sample_sites], w["code_mask"])
    t_map = time.perf_counter() - t0
    # null of the full step's size for the p-value scan: resample the small null
    rng = np.random.default_rng(seed)
    raw = nl["raw"]
    ok = ~np.isnan(raw[:, 0])
    nmax = float(m["norm"].max())
    big = rng.choice(np.flatnonzero(ok), size=RC * R, replace=True)
    cat = np.minimum((raw[big, 3] / (nmax / K)).astype(np.int64), K)
    order = np.lexsort((raw[big, 0], cat))
    keep = cat[order] < K
    srt = raw[big, 0][order][keep]
    offs = np.searchsorted(cat[order][keep], np.arange(K + 1))
    t0 = time.perf_counter()
    pr = O.pairs(cfg["statistic"], m["n"], m["norm"], m["post_rate"], m["rate_class"], null=(K, nmax, offs, srt))
    t_pairs = time.perf_counter() - t0
    n_pairs_s = len(pr["i"])
    sub = min(sample_sites, 200)      # statistic alone on a subset: splits the pair cost into base + p-value scan
    t0 = time.perf_counter()
    O.pairs(cfg["statistic"], m["n"][:sub], m["norm"][:sub], m["post_rate"][:sub], m["rate_class"][:sub])
    per_pair_base = (time.perf_counter() - t0) / max(1, sub * (sub - 1) // 2)
    per_null_site = (t_sim + t_null) / (2 * sample_ram)   # simulate + map (+ paired stat) per simulated site
    per_obs_site = t_map / sample_sites
    per_obs_pair = t_pairs / max(1, n_pairs_s)
    full = per_null_site * 2 * RC * R + per_obs_site * S + per_obs_pair * (S * (S - 1) // 2)
    total_pairs = S * (S - 1) // 2 + RC * R
    sample_pairs = n_pairs_s + sample_ram
    sample_time = t_sim + t_null + t_map + t_pairs
    mean_nsim = float(np.mean(pr["nsim"])) if n_pairs_s else 1.0
    fit = dict(per_null_site=per_null_site, per_obs_site=per_obs_site, per_pair_base=per_pair_base,
               per_pair_scan_per_sample=max(0.0, per_obs_pair - per_pair_base) / max(1.0, mean_nsim))
    value = sample_pairs / sample_time
    return dict(value=value, full_step_seconds=total_pairs / value, sample_seconds=sample_time, fit=fit,
                sample_pairs=sample_pairs, sample_pairs_per_s=value, extrapolated_value=total_pairs / full,
                sample_fraction=sample_pairs / total_pairs,
                sample=("oracle port, 1 thread, 1/%.0f of the step with the step's composition: simulate+map+pair %d null site "
                        "pairs in %d replicates (%.2fs), map %d observed sites (%.2fs), score their %d pairs with p-value "
                        "scan against a %d-sample null (%.2fs); value = sample pairs / sample seconds, measured"
                        % (total_pairs / sample_pairs, sample_ram, reps, t_sim + t_null, sample_sites, t_map, n_pairs_s,
                           RC * R, t_pairs)))


def cpu_validation(cfg, w, fit, sites=400, rep_cpu=10, rep_ram=1000, seed=777):
    """One COMPLETE reduced-size job on the CPU oracle, nothing extrapolated: map `sites` observed sites, simulate +
    map + score rep_cpu x rep_ram null pairs, bin + sort, score all pairs with p-values -- timed, and compared with
    what the linear model fitted on the bounded sample (`fit` = cpu_sample's per-unit costs) predicts for it."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding as O
    K = cfg["null_bins"]
    t0 = time.perf_counter()
    aln, _ = O.simulate(w["parent"], w["brlen"], w["Q"], w["pi"], w["rates"], w["probs"], cfg["aln_seed"], 0, sites)
    m = O.map_sites(w["parent"], w["brlen"], w["Q"], w["pi"], w["rates"], w["probs"], aln, w["code_mask"])
    s1 = np.stack([O.simulate(w["parent"], w["brlen"], w["Q"], w["pi"], w["rates"], w["probs"], seed, (2 * i) * rep_ram, rep_ram)[0]
                   for i in range(rep_cpu)])
    s2 = np.stack([O.simulate(w["parent"], w["brlen"], w["Q"], w["pi"], w["rates"], w["probs"], seed, (2 * i + 1) * rep_ram, rep_ram)[0]
                   for i in range(rep_cpu)])
    nmax = float(m["norm"].max())
    nl = O.null_intra(w["parent"], w["brlen"], w["Q"], w["pi"], w["rates"], w["probs"], cfg["statistic"], s1, s2, K, nmax)
    pr = O.pairs(cfg["statistic"], m["n"], m["norm"], m["post_rate"], m["rate_class"],
                 null=(K, nmax, nl["bin_offsets"], nl["sorted"]))
    measured = time.perf_counter() - t0
    n_pairs = len(pr["i"])
    # the reference counts #{sim < stat} by scanning the sorted bin (CoETools.cpp:712-716): the scan term scales
    # with the samples per bin
    scan = fit["per_pair_scan_per_sample"] * float(np.mean(pr["nsim"])) if n_pairs else 0.0
    predicted = (fit["per_null_site"] * 2 * rep_cpu * rep_ram + fit["per_obs_site"] * (sites + 0) +
                 (fit["per_pair_base"] + scan) * n_pairs)
    return dict(job="%d observed sites, %dx%d null, %d pairs with p-values, complete (not extrapolated)"
                    % (sites, rep_cpu, rep_ram, n_pairs), measured_seconds=measured, predicted_seconds=predicted,
                measured_over_predicted=measured / predicted, pairs_per_s=(n_pairs + rep_cpu * rep_ram) / measured)


def _cpu_worker(job):
    cfg, w, aln_codes, seed = job
    return cpu_sample(cfg, w, aln_codes=aln_codes, seed=seed)


def cpu_sample_all_cores(cfg, w, aln_codes=None, seed=0, n_proc=None):
    """The only parallelism the reference admits is independent processes (shards of the outer null
    replicates and of the pair rows): one oracle sample per host core, all running at the same time;
    the job's throughput is the sum of the per-process throughputs measured under that load."""
    import multiprocessing as mp
    n_proc = n_proc or os.cpu_count() or 1
    if n_proc == 1:
        r = cpu_sample(cfg, w, aln_codes=aln_codes, seed=seed)
        return dict(r, cores=1)
    ctx = mp.get_context("spawn")  # the parent may hold a CUDA context
    with ctx.Pool(n_proc) as pool:
        rs = pool.map(_cpu_worker, [(cfg, w, aln_codes, seed * 1000 + i) for i in range(n_proc)])
    value = float(sum(r["value"] for r in rs))
    total_pairs = cfg["sites"] * (cfg["sites"] - 1) // 2 + cfg["rep_cpu"] * cfg["rep_ram"]
    return dict(value=value, full_step_seconds=total_pairs / value, cores=n_proc,
                sample_seconds=float(max(r["sample_seconds"] for r in rs)),
                sample_pairs=int(sum(r["sample_pairs"] for r in rs)),
                sample_pairs_per_s=float(sum(r["sample_pairs_per_s"] for r in rs)),
                extrapolated_value=float(sum(r["extrapolated_value"] for r in rs)),
                sample_fraction=float(sum(r["sample_fraction"] for r in rs)),
                sample="%d concurrent processes, each: %s" % (n_proc, rs[0]["sample"]))


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = workload(cfg)
    for i in range(args.warmup):
        cpu_sample(cfg, w, sample_sites=16, sample_ram=16, seed=100 + i)
    # one step = one bounded sample per host core, all at once: ms_per_step is its measured wall time and
    # value = the pairs the cores scored / that time -- the metric on 16/38 of the workload, nothing extrapolated
    vals, secs, last = [], [], None
    for i in range(args.steps):
        t0 = time.perf_counter()
        last = cpu_sample_all_cores(cfg, w, seed=i)
        secs.append(time.perf_counter() - t0)
        vals.append(last["value"])
    v = float(np.mean(vals))
    line = dict(impl="reference", metric="site_pairs_scored_per_s_incl_mapping_and_null", value=v, unit="pairs/s",
                n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=float(np.mean(secs) * 1e3),
                higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f64", data="synthetic",
                config=config_dict(cfg, args.gpus),
                cpu_baseline=dict(value=v, unit="pairs/s", cores=last["cores"], kind="port", sample=last["sample"],
                                  host_cores=os.cpu_count(), sample_pairs_per_step=last["sample_pairs"],
                                  sample_fraction_of_workload=last["sample_fraction"],
                                  full_step_seconds_implied=last["full_step_seconds"],
                                  extrapolated_value=last["extrapolated_value"],
                                  note="upstream CoMap needs Bio++ >= 3.0 (not installable offline); this is the "
                                       "CPU oracle restatement; each step scores a bounded sample with the workload's "
                                       "composition, value = sample pairs / measured seconds; extrapolated_value = the "
                                       "per-unit linear model of round 1 for comparison"),
                e2e=dict(value=v, unit="pairs/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def config_dict(cfg, n_gpus):
    return dict(workload="configs[3]: synthetic %d-site x %d-taxon nucleotide alignment, HKY85+Gamma4, all-pairs "
                         "%s + %dx%d null" % (cfg["sites"], cfg["taxa"], cfg["statistic"], cfg["rep_cpu"], cfg["rep_ram"]),
                sites=cfg["sites"], taxa=cfg["taxa"], branches=2 * cfg["taxa"] - 3, rate_classes=cfg["classes"],
                rep_cpu=cfg["rep_cpu"], rep_ram=cfg["rep_ram"], null_bins=cfg["null_bins"],
                pairs_per_step=cfg["sites"] * (cfg["sites"] - 1) // 2 + cfg["rep_cpu"] * cfg["rep_ram"],
                parallelism="null replicates + pair rows sharded over %d GPU(s); NCCL all-gather of null samples" % n_gpus,
                l2="per-step working set (down-partials of each null batch, GBs) exceeds the 126 MB L2; no explicit flush")


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
METRIC = "site_pairs_scored_per_s_incl_mapping_and_null"


def load_peaks():
    """HBM peak: MEASURED_PEAKS.json (driver-written) else the profiling recipe's fallback; FP64 peaks:
    PEAKS_FP64.json (tools/dmmabench + tools/fp64bench on this pool's B200s, committed)."""
    out = dict(hbm_gbs=6650.0, hbm_source="fallback 6650 GB/s (B200_PROFILING.md)", fp64_dmma_tflops=37.0,
               fp64_dfma_tflops=34.0, fp64_source="PEAKS_FP64.json missing: nominal")
    try:
        m = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        out["hbm_gbs"] = float(m["hbm_gbs"]); out["hbm_source"] = "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        pass
    try:
        f = json.load(open(os.path.join(ROOT, "PEAKS_FP64.json")))
        out["fp64_dmma_tflops"] = float(f["fp64_dmma_tflops"]); out["fp64_dfma_tflops"] = float(f["fp64_dfma_tflops"])
        out["fp64_source"] = "PEAKS_FP64.json (%s)" % f.get("how", "")
    except Exception:
        pass
    return out


def profile_dram_bytes(pattern):
    """dram__bytes_read.sum + dram__bytes_write.sum and the grid size of the newest committed `ncu --set full`
    summary whose file name matches `pattern` (profiles/r*_<kernel>.txt, written by tools/ncu_summary.py)."""
    import glob
    import re
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", pattern))):
        best = path
    if not best:
        return None
    txt = open(best).read()
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    tot = 0.0
    for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
        m = re.search(r"^%s\s+(\S+)\s+([0-9.eE+-]+)" % re.escape(key), txt, re.M)
        if not m:
            return None
        tot += float(m.group(2)) * unit.get(m.group(1), 1.0)
    g = re.search(r"^launch__grid_size\s+([0-9.]+)", txt, re.M)
    d = re.search(r"^gpu__time_duration.sum\s+(\S+)\s+([0-9.eE+-]+)", txt, re.M)
    sg = re.search(r"k1_(?:up|down)_mma<\d+, \d+, (\d+),", txt)      # sites per CTA: third template argument
    return dict(file=os.path.relpath(best, ROOT), dram_bytes=tot, grid=float(g.group(1)) if g else None,
                sites_per_cta=int(sg.group(1)) if sg else 128,
                ms=float(d.group(2)) * {"ms": 1.0, "us": 1e-3, "s": 1e3, "ns": 1e-6}.get(d.group(1), 1.0) if d else None)


def table_checksum(cols, n):
    """Order-independent 64-bit checksum of the (i, j, Stat, PValue, Nsim) rows: every row is hashed from the bit
    patterns of its fields and the hashes are summed modulo 2^64, so shards can be added across ranks."""
    M = np.uint64
    with np.errstate(over="ignore"):
        h = cols[0][:n].astype(np.uint64) * M(0x9E3779B97F4A7C15)
        h ^= cols[1][:n].astype(np.uint64) * M(0xC2B2AE3D27D4EB4F)
        h ^= cols[2][:n].view(np.uint64) * M(0x165667B19E3779F9)
        h ^= cols[6][:n].view(np.uint64) * M(0x27D4EB2F165667C5)
        h ^= cols[7][:n].astype(np.uint64) * M(0x85EBCA77C2B2AE63)
        h ^= h >> M(29); h *= M(0xBF58476D1CE4E5B9); h ^= h >> M(32)
        return int(h.sum(dtype=np.uint64))


DUMP_PAIR_ROWS = 1 << 19        # 9 float64 columns of 4 MB each + the 8 MB null: 44 MB of the 64 MB allowed
DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(out_dir, arrays):
    """--dump-outputs: every array as out_dir/<name>.npy in float64 (the integer columns are exact in it)."""
    arrays = {name: np.asarray(a, dtype=np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("bench.py: %d bytes of outputs exceed the %d-byte dump limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args, cfg):
    import torch
    import torch.distributed as dist
    from comap_b200 import api, parallel as par

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("bench.py: --dump-outputs needs one process (each rank holds only its shard of the pair table)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; comap_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.Stream()
    w = workload(cfg)
    S, T, R, RC, K = cfg["sites"], cfg["taxa"], cfg["rep_ram"], cfg["rep_cpu"], cfg["null_bins"]
    A = len(w["pi"])
    B = 2 * T - 3
    stat = cfg["statistic"]
    r0, r1 = par.replicate_bounds(RC, world)[rank]

    with torch.cuda.stream(stream):
        ctx = api.Context(device=local, stream=stream.cuda_stream)
        ctx.set_tree(w["parent"], w["brlen"])
        ctx.set_model(w["Q"], w["pi"], w["rates"], w["probs"])
        if world > 1:
            # the library drives NCCL itself (cmb_comm_init + cmb_null_intra_sharded); torch.distributed only
            # carries the 128-byte id to the other ranks and the timing / checksum reductions
            uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                uid = torch.frombuffer(bytearray(api.comm_unique_id()), dtype=torch.uint8).cuda()
            dist.broadcast(uid, 0)
            ctx.comm_init(world, rank, uid.cpu().numpy().tobytes())
        codes, _ = ctx.simulate(cfg["aln_seed"], 0, S)     # the synthetic alignment (project's own simulator)
        pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True).numpy()
        codes_pin = pin((T, S), torch.uint8); codes_pin[:] = codes
        ctx.set_alignment(codes_pin, w["code_mask"])
        n_own = par.owned_pairs(S, rank, world)
        cols_pin = [pin((max(1, n_own),), {np.int32: torch.int32, np.float64: torch.float64, np.int64: torch.int64}[dt])
                    for dt in api.Context.COL_DTYPE]

        def null_dist():
            ctx.null_intra_sharded(stat, cfg["null_seed"], RC, R, K=K, nmax=-1.0)

        def step_resident(overlap=True):
            if overlap:
                ctx.map_async()          # enqueued on a side stream: the null replicates overlap it
            else:
                ctx.map(want_vectors=False)
            null_dist()
            return ctx.pairs_resident(stat, use_null=True, shard_index=rank, shard_count=world)

        def step_e2e():
            # the six null-independent columns are scored first and copied out while the null
            # distribution is simulated; PValue / Nsim follow once the null exists
            ctx.set_alignment(codes_pin, w["code_mask"])
            ctx.map(want_vectors=False)
            ctx.pairs_resident(stat, use_null=False, shard_index=rank, shard_count=world, columns=0x3F)
            for k in range(6):
                ctx.pairs_fetch(k, cols_pin[k])
            null_dist()
            n = ctx.pairs_resident(stat, use_null=True, shard_index=rank, shard_count=world, columns=0xC0)
            for k in (6, 7):
                ctx.pairs_fetch(k, cols_pin[k])
            ctx.sync()
            return n

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        def timed(fn, steps):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                fn()
            e1.record(stream)
            barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            return float(ms.item())

        for _ in range(max(3, args.warmup)):
            n_rows = step_resident()
        step_e2e()
        if args.dump_outputs:
            dump_rows = np.sort(np.random.default_rng(0).choice(n_rows, min(n_rows, DUMP_PAIR_ROWS), replace=False))

        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        l0 = ctx.launch_count()
        ms = timed(step_resident, args.steps)              # the timed region: no per-kernel events inside
        launches = ctx.launch_count() - l0
        if args.dump_outputs:
            # what the last timed step left on the device: the pair table (sampled rows, in the reference's order)
            # and the binned null distribution; written once the measurements are over
            for k in range(len(api.Context.COLS)):
                ctx.pairs_fetch(k, cols_pin[k])
            ctx.sync()
            g = ctx.null_get()
            dumped = {"pairs_" + c: cols_pin[k][dump_rows] for k, c in enumerate(api.Context.COLS)}
            dumped.update(pairs_row=dump_rows, null_sorted=g["sorted"], null_bin_offsets=g["bin_offsets"],
                          null_nmax=np.array([g["nmax"]]))
        ms_e2e = timed(step_e2e, args.steps)
        clocks = sampler.stop() if rank == 0 else None
        # per-kernel device time: the same steps again with CUDA events around every kernel family
        # (cmb_profile_*; the events cost host time, so this pass is NOT the one `value` is taken from)
        ctx.profile_reset(); ctx.profile_enable(True)
        for _ in range(args.steps):
            step_resident(overlap=False)   # one stream: every family's events bracket its own kernels only
        names = ("map_down", "map_up", "simulate", "null_pairs", "sort", "pairs")
        prof = {k: ctx.profile_get(k) for k in names}
        prof["compress"] = ctx.profile_get("compress")
        null_simulated = ctx.profile_get("sites_simulated")[0]    # simulated sites of this rank's replicates ...
        null_mapped = ctx.profile_get("sites_mapped_null")[0]     # ... and the distinct columns the mapping walked
        ctx.profile_enable(False)

        # ---- correctness carried with the number (outside the timed region): checksum of this rank's rows,
        #      summed over ranks; at N > 1 rank 0 also runs the whole job on its own GPU and must get the same
        own = table_checksum(cols_pin, n_rows)
        tot = torch.tensor([own - (1 << 64) if own >= (1 << 63) else own], dtype=torch.int64, device="cuda")
        nr = torch.tensor([n_rows], dtype=torch.int64, device="cuda")
        lt = torch.tensor([launches], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(tot); dist.all_reduce(nr); dist.all_reduce(lt)
        check = dict(rows=int(nr.item()), checksum="%016x" % (int(tot.item()) & ((1 << 64) - 1)),
                     columns="i j Stat PValue Nsim", how="sum mod 2^64 of per-row hashes over all ranks")
        if world > 1 and rank == 0:
            one = api.Context(device=local, stream=stream.cuda_stream)
            one.set_tree(w["parent"], w["brlen"]); one.set_model(w["Q"], w["pi"], w["rates"], w["probs"])
            one.set_alignment(codes_pin, w["code_mask"]); one.map(want_vectors=False)
            one.null_intra(stat, cfg["null_seed"], RC, R, K=K, nmax=-1.0)
            full, kk = one.pairs(stat, use_null=True)
            ref = table_checksum([full[c] for c in api.Context.COLS], kk)
            check["single_gpu_checksum"] = "%016x" % ref
            check["equal_to_single_gpu"] = bool(ref == (int(tot.item()) & ((1 << 64) - 1)) and kk == int(nr.item()))
            one.close()

        pairs_per_step = S * (S - 1) // 2 + RC * R
        if rank == 0:
            peaks = load_peaks()
            C = cfg["classes"]
            # constant simulated columns are mapped once per state and batch (pattern compression, as Bio++ maps
            # distinct site patterns): the roofline counts the columns the kernels actually walked
            sites_mapped = args.steps * S + (null_mapped if null_mapped > 0 else args.steps * 2 * (r1 - r0) * R)
            passes = max(1, prof["map_up"][1])
            hbm = peaks["hbm_gbs"]

            def hbm_entry(kernel, bytes_per_site, ms_total, prof_glob, note):
                ach = sites_mapped * bytes_per_site / (ms_total * 1e-3) / 1e9 if ms_total > 0 else 0.0
                e = dict(kernel=kernel, bound="hbm", achieved=ach, peak=hbm, unit="GB/s", frac=ach / hbm,
                         algorithmic_bytes_per_site=bytes_per_site, avg_launch_ms=ms_total / passes,
                         sites_per_launch=sites_mapped / passes, note=note, traffic=None)
                pd = profile_dram_bytes(prof_glob)
                if pd and pd["grid"]:
                    per_site = pd["dram_bytes"] / (pd["grid"] * pd["sites_per_cta"])   # captured without pattern compression
                    e["traffic"] = per_site * sites_mapped / passes
                    e["traffic_source"] = "%s: dram__bytes_read.sum + dram__bytes_write.sum, scaled by sites" % pd["file"]
                    e["measured_dram_frac"] = per_site * sites_mapped / (ms_total * 1e-3) / 1e9 / hbm
                return e

            # SURVEY.md s8(d) K1 bytes per site, split by pass: down = tips + inner partials written once,
            # up = inner partials read once + output rows + tips (28 B of per-site scalars belong to k1_finish)
            part = (T - 3) * C * A * 8
            up = hbm_entry("k1_up_mma" if A == 4 else "k1_up", part + 8 * B + T, prof["map_up"][0], "r2*_k1_up_mma.txt",
                           "mapping up pass + contraction; cherry partials are recomputed, so DRAM traffic is below the algorithmic bytes")
            down = hbm_entry("k1_down_mma (+ k1_finish)" if A == 4 else "k1_down", part + T + 28, prof["map_down"][0],
                             "r2*_k1_down_mma.txt", "mapping down pass; cherry partials are never stored")
            flops = 2.0 * B * (n_rows * args.steps)
            tiles_ms = prof["pairs"][0]
            tiles = dict(kernel="k2_tiles<correlation>", bound="fp64", achieved=flops / (tiles_ms * 1e-3) / 1e12 if tiles_ms > 0 else 0.0,
                         peak=peaks["fp64_dfma_tflops"], unit="TFLOP/s", algorithmic_flops_per_pair=2 * B,
                         peak_source=peaks["fp64_source"], avg_launch_ms=tiles_ms / max(1, prof["pairs"][1]),
                         note="unfused DMUL + DADD in the reference's summation order (bit-exact p-values given vectors): "
                              "at most half the FMA peak")
            tiles["frac"] = tiles["achieved"] / tiles["peak"]
            paired_bytes = 2.0 * B * 8 * ((r1 - r0) * R * args.steps)
            paired = dict(kernel="k2_paired<correlation>", bound="hbm", achieved=paired_bytes / (prof["null_pairs"][0] * 1e-3) / 1e9
                          if prof["null_pairs"][0] > 0 else 0.0, peak=hbm, unit="GB/s", algorithmic_bytes_per_pair=2 * B * 8)
            paired["frac"] = paired["achieved"] / hbm
            kernel_ms = {k: v[0] / args.steps for k, v in prof.items()}
            line = dict(metric=METRIC, value=pairs_per_step * args.steps / (ms * 1e-3), unit="pairs/s", n_gpus=world,
                        steps=args.steps, warmup=max(3, args.warmup), ms_per_step=ms / args.steps, higher_is_better=True,
                        scaling="strong", vs_baseline=None, dtype="f64", data="synthetic", config=config_dict(cfg, world),
                        clocks=clocks,
                        e2e=dict(value=pairs_per_step * args.steps / (ms_e2e * 1e-3), unit="pairs/s",
                                 ms_per_step=ms_e2e / args.steps, h2d_bytes_per_step=int(T * S + 4 * 256),
                                 d2h_bytes_per_step=int(sum(c.itemsize for c in cols_pin) * n_rows + S * 8 * 4)),
                        gpu_launches=int(lt.item()),
                        roofline=dict(up, peak_source=peaks["hbm_source"],
                                      why="dominant kernel: %.0f %% of the step's device time" %
                                          (100.0 * kernel_ms["map_up"] / max(1e-9, sum(kernel_ms.values())))),
                        rooflines=[down, up, paired, tiles],
                        kernel_ms_per_step=kernel_ms, kernel_ms_sum=sum(kernel_ms.values()),
                        null_sites=dict(simulated_per_step=null_simulated / args.steps, mapped_per_step=null_mapped / args.steps,
                                        note="columns whose tips all carry one state are mapped once per state and batch"),
                        host_gap_frac=(ms / args.steps - sum(kernel_ms.values())) / (ms / args.steps),
                        host_gap_note="kernel times come from a serialised pass; the timed step overlaps the observed "
                                      "alignment's mapping (~0.5 ms) with the null, so a small negative gap is possible",
                        table_check=check)
            if world == 1 and not args.no_cpu_baseline:
                cb = cpu_sample_all_cores(cfg, w, aln_codes=codes)
                one = cpu_sample(cfg, w, aln_codes=codes, sample_sites=400, seed=12345) # the other cores idle
                line["cpu_baseline"] = dict(value=cb["value"], unit="pairs/s", cores=cb["cores"], kind="port", sample=cb["sample"],
                                            host_cores=os.cpu_count(), sample_seconds=cb["sample_seconds"],
                                            sample_fraction_of_workload=cb["sample_fraction"],
                                            extrapolated_value=cb["extrapolated_value"],
                                            one_thread_value=one["value"],
                                            one_thread_extrapolated_value=one["extrapolated_value"],
                                            validation=cpu_validation(cfg, w, one["fit"]))
            print(json.dumps(line), flush=True)
        ctx.close()
    if args.dump_outputs:
        write_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------
# other workloads (N = 1): BASELINE.json configs[1] (proteins, pairwise + null) and configs[4] (clustering)
# ------------------------------------------------------------------------------------------
PROTEINS = dict(sites=129, taxa=100, alpha=0.985435, classes=4, mean_brlen=0.05, tree_seed=7, aln_seed=1, null_seed=2,
                rep_cpu=100, rep_ram=1000, null_bins=10, statistic="correlation")
CLUSTERING = dict(sites=20000, taxa=200, alpha=1.0, classes=4, mean_brlen=0.05, tree_seed=2, aln_seed=1, null_seed=7,
                  null_reps=4, max_group=10)


def _timed_gpu(torch, stream, fn, steps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def run_proteins(args):
    """configs[1]-shaped: Myoglobin-sized protein alignment (100 taxa, 129 sites) under JTT92 + Gamma(4),
    all-pairs correlation with the default 100 x 1000 simulated null (CoETools.cpp:853-854).  The protein
    mapping kernels (A = 20) are FP64-bound (SURVEY.md s8d): roofline against the measured DMMA peak."""
    import torch
    from comap_b200 import api
    cfg = dict(PROTEINS)
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    S, T, R, RC, K = cfg["sites"], cfg["taxa"], cfg["rep_ram"], cfg["rep_cpu"], cfg["null_bins"]
    B, C, A = 2 * T - 3, cfg["classes"], 20
    parent, brlen = syn.random_tree(T, cfg["tree_seed"], cfg["mean_brlen"])
    Q, pi = syn.jtt92()
    rates, probs = syn.gamma_rates(cfg["alpha"], C)
    with torch.cuda.stream(stream):
        ctx = api.Context(device=0, stream=stream.cuda_stream)
        ctx.set_tree(parent, brlen); ctx.set_model(Q, pi, rates, probs)
        codes, _ = ctx.simulate(cfg["aln_seed"], 0, S)
        mask = syn.identity_code_mask(A)

        def step():
            ctx.set_alignment(codes, mask)
            ctx.map(want_vectors=False)
            ctx.null_intra(cfg["statistic"], cfg["null_seed"], RC, R, K=K, nmax=-1.0)
            return ctx.pairs(cfg["statistic"], use_null=True)[1]

        for _ in range(max(3, args.warmup)):
            n_rows = step()
        sampler = ClockSampler(0); sampler.start()
        l0 = ctx.launch_count()
        ms = _timed_gpu(torch, stream, step, args.steps)
        launches = ctx.launch_count() - l0
        clocks = sampler.stop()
        ctx.profile_reset(); ctx.profile_enable(True)
        for _ in range(args.steps):
            step()
        prof = {k: ctx.profile_get(k) for k in ("map_down", "map_up", "simulate", "null_pairs", "sort", "pairs")}
        ctx.profile_enable(False)
        peaks = load_peaks()
        sites_mapped = args.steps * (S + 2 * RC * R)
        k1_ms = prof["map_down"][0] + prof["map_up"][0]
        flops_site = 6.0 * B * C * A * A                     # SURVEY.md s8(d): down 2, up 2, contraction 2 x B C A^2
        ach = sites_mapped * flops_site / (k1_ms * 1e-3) / 1e12
        pairs_per_step = S * (S - 1) // 2 + RC * R
        kernel_ms = {k: v[0] / args.steps for k, v in prof.items()}
        line = dict(metric=METRIC, value=pairs_per_step * args.steps / (ms * 1e-3), unit="pairs/s", n_gpus=1, steps=args.steps,
                    warmup=max(3, args.warmup), ms_per_step=ms / args.steps, higher_is_better=True, scaling="strong",
                    vs_baseline=None, dtype="f64", data="synthetic",
                    config=dict(workload="configs[1]-shaped: synthetic %d-site x %d-taxon protein alignment, JTT92+Gamma4, all-pairs "
                                         "correlation + %dx%d null" % (S, T, RC, R), sites=S, taxa=T, branches=B, rate_classes=C,
                                rep_cpu=RC, rep_ram=R, null_bins=K, pairs_per_step=pairs_per_step,
                                l2="null batch working set (GBs of partials) exceeds the 126 MB L2; no explicit flush"),
                    clocks=clocks, gpu_launches=launches,
                    e2e=dict(value=pairs_per_step * args.steps / (ms * 1e-3), unit="pairs/s", ms_per_step=ms / args.steps,
                             h2d_bytes_per_step=int(T * S), d2h_bytes_per_step=int(n_rows * 44),
                             note="this workload's step already runs through the host-buffer C ABI"),
                    roofline=dict(kernel="K1 protein mapping (down + up, A = 20)", bound="fp64", achieved=ach,
                                  peak=peaks["fp64_dmma_tflops"], unit="TFLOP/s", frac=ach / peaks["fp64_dmma_tflops"],
                                  algorithmic_flops_per_site=flops_site, peak_source=peaks["fp64_source"], traffic=None),
                    kernel_ms_per_step=kernel_ms, kernel_ms_sum=sum(kernel_ms.values()))
        print(json.dumps(line), flush=True)
        ctx.close()


def run_clustering(args):
    """configs[4]: synthetic 20,000-site x 200-taxon protein alignment (JTT92 + Gamma4), clustering analysis:
    map -> correlation distance matrix -> complete-linkage dendrogram -> groups <= 10, plus a short clustering
    null.  pairs per step = (1 + nrep) S (S - 1) / 2 (SURVEY.md s8d)."""
    import torch
    from comap_b200 import api
    cfg = dict(CLUSTERING)
    if args.sites:
        cfg["sites"] = args.sites
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    S, T, C, A = cfg["sites"], cfg["taxa"], cfg["classes"], 20
    B = 2 * T - 3
    nrep = cfg["null_reps"]
    parent, brlen = syn.random_tree(T, cfg["tree_seed"], cfg["mean_brlen"])
    Q, pi = syn.jtt92()
    rates, probs = syn.gamma_rates(cfg["alpha"], C)
    with torch.cuda.stream(stream):
        ctx = api.Context(device=0, stream=stream.cuda_stream)
        ctx.set_tree(parent, brlen); ctx.set_model(Q, pi, rates, probs)
        codes, _ = ctx.simulate(cfg["aln_seed"], 0, S)
        mask = syn.identity_code_mask(A)
        out = {}

        def step():
            ctx.set_alignment(codes, mask)
            ctx.map(want_vectors=False)
            ctx.distance_matrix("correlation", want=False)
            out["dendro"] = ctx.cluster("complete")
            out["groups"] = ctx.groups("correlation", cfg["max_group"], as_lists=False)
            out["null"] = ctx.cluster_null("correlation", "complete", cfg["null_seed"], 0, nrep, cfg["max_group"], as_lists=False)

        for _ in range(max(1, min(2, args.warmup))):
            step()
        sampler = ClockSampler(0); sampler.start()
        l0 = ctx.launch_count()
        ms = _timed_gpu(torch, stream, step, args.steps)
        launches = ctx.launch_count() - l0
        clocks = sampler.stop()
        ctx.profile_reset(); ctx.profile_enable(True)
        step()
        prof = {k: ctx.profile_get(k) for k in ("map_down", "map_up", "simulate", "distance", "cluster")}
        ctx.profile_enable(False)
        peaks = load_peaks()
        pairs_per_step = (1 + nrep) * S * (S - 1) // 2
        n_dendro = 1 + nrep
        cl_ms = prof["cluster"][0] / n_dendro
        ach = 8.0 * S * S / (cl_ms * 1e-3) / 1e9        # SURVEY.md s8(d) K4b: O(S^2) bytes = one pass over the matrix
        line = dict(metric=METRIC, value=pairs_per_step * args.steps / (ms * 1e-3), unit="pairs/s", n_gpus=1, steps=args.steps,
                    warmup=max(1, min(2, args.warmup)), ms_per_step=ms / args.steps, higher_is_better=True, scaling="strong",
                    vs_baseline=None, dtype="f64", data="synthetic",
                    config=dict(workload="configs[4]: synthetic %d-site x %d-taxon protein alignment, JTT92+Gamma4, clustering "
                                         "(cor distance, complete linkage, groups <= %d) + %d null replicates"
                                         % (S, T, cfg["max_group"], nrep), sites=S, taxa=T, branches=B, rate_classes=C,
                                null_reps=nrep, pairs_per_step=pairs_per_step,
                                l2="a 3.2 GB distance matrix per dendrogram: far beyond L2; no explicit flush"),
                    clocks=clocks, gpu_launches=launches,
                    e2e=dict(value=pairs_per_step * args.steps / (ms * 1e-3), unit="pairs/s", ms_per_step=ms / args.steps,
                             h2d_bytes_per_step=int(T * S), d2h_bytes_per_step=int(n_dendro * (S - 1) * 16),
                             note="this workload's step already runs through the host-buffer C ABI"),
                    roofline=dict(kernel="k4 agglomeration (one dendrogram)", bound="hbm", achieved=ach, peak=peaks["hbm_gbs"],
                                  unit="GB/s", frac=ach / peaks["hbm_gbs"], algorithmic_bytes_per_dendrogram=8.0 * S * S,
                                  ms_per_dendrogram=cl_ms, peak_source=peaks["hbm_source"], traffic=None),
                    kernel_ms_per_step={k: v[0] for k, v in prof.items()},
                    groups=len(out["groups"]["height"]), null_rows=len(out["null"]["rep"]))
        print(json.dumps(line), flush=True)
        ctx.close()


MICA = dict(sites=760, taxa=40, mean_brlen=0.12, tree_seed=11, aln_seed=1, perm_seed=3, max_perm=1000)


def profile_metric(pattern, key):
    """One metric of the newest committed ncu summary whose file name matches `pattern` (tools/ncu_summary.py format)."""
    import glob
    import re
    paths = sorted(glob.glob(os.path.join(ROOT, "profiles", pattern)))
    if not paths:
        return None, None
    m = re.search(r"^%s\s+(\S*)\s+([0-9.eE+,-]+)\s*$" % re.escape(key), open(paths[-1]).read(), re.M)
    return (float(m.group(2).replace(",", "")) if m else None), os.path.relpath(paths[-1], ROOT)


def run_mica(args):
    """mica with null.method = permutations (examples/RNA/BacteriaSSU/options_perm.mica: 760 complete variable sites x
    40 taxa, at most 1000 shuffles per pair): one step = alignment H2D -> entropies, dense MI / joint entropy, average
    MI -> the other columns of the table -> the permutation test of all 288,420 pairs -> table D2H.  The dominant kernel
    (k5_permutations) moves almost no memory -- private column copies in shared memory, 12 bytes out per pair -- and is
    bound by instruction issue; its roofline is warp instructions per second against 4 per SM per clock."""
    import torch
    from comap_b200 import api
    cfg = dict(MICA)
    if args.sites:
        cfg["sites"] = args.sites
    if args.taxa:
        cfg["taxa"] = args.taxa
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    S, T, A = cfg["sites"], cfg["taxa"], 4
    parent, brlen = syn.random_tree(T, cfg["tree_seed"], cfg["mean_brlen"])
    Q, pi = syn.hky85(CFG["kappa"], CFG["pi"])
    rates, probs = syn.gamma_rates(CFG["alpha"], CFG["classes"])
    with torch.cuda.stream(stream):
        ctx = api.Context(device=0, stream=stream.cuda_stream)
        ctx.set_tree(parent, brlen); ctx.set_model(Q, pi, rates, probs)
        codes, _ = ctx.simulate(cfg["aln_seed"], 0, S)
        mask = syn.identity_code_mask(A)
        out = {}

        def step():
            ctx.set_alignment(codes, mask)
            out["sites"] = ctx.mica_sites()
            out["pairs"] = ctx.mica_pairs("hmin")
            out["perm"] = ctx.mica_permutations(cfg["perm_seed"], cfg["max_perm"])

        W = max(3, args.warmup)
        for _ in range(W):
            step()
        sampler = ClockSampler(0); sampler.start()
        l0 = ctx.launch_count()
        ms = _timed_gpu(torch, stream, step, args.steps)
        launches = ctx.launch_count() - l0
        clocks = sampler.stop()
        ctx.profile_reset(); ctx.profile_enable(True)
        for _ in range(args.steps):
            step()
        prof = {k: ctx.profile_get(k) for k in ("mica_pairs", "mica_perm")}
        ctx.profile_enable(False)
        pv, nb = out["perm"]
        n_pairs = S * (S - 1) // 2
        evaluations = int(nb.sum()) + n_pairs                       # shuffled MIs + the observed one of every pair
        perm_ms = prof["mica_perm"][0] / args.steps
        inst, src = profile_metric("r2*_k5_permutations.txt", "smsp__inst_executed.sum")
        inst_pairs, _ = profile_metric("r2*_k5_permutations.txt", "launch__grid_size")
        sm_mhz = clocks.get("sm_mhz") or 1900.0
        peak = 148 * 4 * sm_mhz * 1e6 / 1e9                          # warp instructions per ns-second: 4 schedulers per SM
        roof = dict(kernel="k5_permutations<4>", bound="issue", unit="Gwarp-inst/s", peak=peak,
                    peak_source="148 SMs x 4 warp schedulers x %.0f MHz (median SM clock during the timed region)" % sm_mhz,
                    ms_per_launch=perm_ms, evaluations_per_launch=evaluations, traffic=None,
                    algorithmic_bytes_per_launch=n_pairs * (2 * T + 12))
        if inst:
            roof.update(achieved=inst / (perm_ms * 1e-3) / 1e9, frac=inst / (perm_ms * 1e-3) / 1e9 / peak,
                        warp_instructions_per_launch=inst, profile=src)
            dr = profile_dram_bytes("r2*_k5_permutations.txt")
            if dr:
                roof["traffic"] = dr["dram_bytes"]
        else:
            roof.update(achieved=None, frac=None, note="no committed ncu summary of k5_permutations yet")
        line = dict(metric="mica_site_pairs_per_s_incl_permutation_test", value=n_pairs * args.steps / (ms * 1e-3), unit="pairs/s",
                    n_gpus=1, steps=args.steps, warmup=W, ms_per_step=ms / args.steps, higher_is_better=True, scaling="strong",
                    vs_baseline=None, dtype="f64", data="synthetic",
                    config=dict(workload="examples/RNA/BacteriaSSU/options_perm.mica-shaped: synthetic %d-site x %d-taxon nucleotide "
                                         "alignment, MI of all pairs + permutation test (at most %d shuffles per pair)"
                                         % (S, T, cfg["max_perm"]), sites=S, taxa=T, max_permutations=cfg["max_perm"],
                                pairs_per_step=n_pairs, mi_evaluations_per_step=evaluations, mean_shuffles_per_pair=float(nb.mean()),
                                l2="the alignment (30 KB) lives in L1 / shared memory; outputs are written once: no flush needed"),
                    clocks=clocks, gpu_launches=launches,
                    e2e=dict(value=n_pairs * args.steps / (ms * 1e-3), unit="pairs/s", ms_per_step=ms / args.steps,
                             h2d_bytes_per_step=int(T * S), d2h_bytes_per_step=int(n_pairs * (8 + 4 * 8 + 12) + 16 * S),
                             note="this workload's step already runs through the host-buffer C ABI"),
                    roofline=roof, kernel_ms_per_step={k: v[0] / args.steps for k, v in prof.items()})
        if not args.no_cpu_baseline:     # the oracle's miTest on the first pairs of the same table, one thread
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_binding as O
            sub = 90                                                 # 4005 pairs of the first 90 sites
            t0 = time.perf_counter()
            opv, onb, _ = O.mica_permutations(codes[:, :sub], A, mask, cfg["perm_seed"], cfg["max_perm"])
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = dict(value=len(opv) / dt, unit="pairs/s", cores=1, kind="port",
                                        sample="the permutation test of the %d pairs among the first %d sites (%.1f s, %d MI "
                                               "evaluations), CPU oracle restatement; MI of the pairs included, table output not"
                                               % (len(opv), sub, dt, int(onb.sum()) + len(opv)))
        print(json.dumps(line), flush=True)
        ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="nucleotides", choices=["nucleotides", "proteins", "clustering", "mica"],
                    help="nucleotides = BASELINE.json configs[3] (the metric's configuration, default); proteins = "
                         "configs[1]-shaped; clustering = configs[4]; mica = the permutation test of "
                         "examples/RNA/BacteriaSSU/options_perm.mica (all three N = 1, ours only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64): a fixed "
                         "seeded sample of the pair table's rows (pairs_<column>, pairs_row = their row numbers) and the "
                         "binned null (null_sorted, null_bin_offsets, null_nmax); default workload, one process")
    for k in ("sites", "taxa", "rep_cpu", "rep_ram"):
        ap.add_argument("--" + k.replace("_", "-"), type=int, default=None)
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "nucleotides"):
        ap.error("--dump-outputs is implemented for the default workload (--impl ours --workload nucleotides)")
    cfg = dict(CFG)
    for k in ("sites", "taxa", "rep_cpu", "rep_ram"):
        if getattr(args, k) is not None:
            cfg[k] = getattr(args, k)
    if args.impl == "reference":
        run_reference(args, cfg)
    elif args.workload == "proteins":
        run_proteins(args)
    elif args.workload == "clustering":
        run_clustering(args)
    elif args.workload == "mica":
        run_mica(args)
    else:
        run_ours(args, cfg)


if __name__ == "__main__":
    main()
