#!/usr/bin/env python
"""bench.py -- GCUPS of the adaptive-banded sequence-to-POA-graph DP hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--groups G] [--dump-outputs DIR]

Workload (BASELINE.json configs[2], the one the metric is quoted on): synthetic read groups,
50 reads x 10 kbp, 5 % ONT-like error, global alignment, convex gaps (-O 4,24 -E 2,1).
One STEP = one complete progressive MSA of every group of the batch (1000 groups at N=1;
weak scaling: every rank gets its own 1000 groups) = 49 alignments per group.

Printed JSON (rank 0):
  value     whole-job GCUPS of the DP + backtrace kernels with every flattened alignment job
            (graph + read) already resident in HBM: all jobs of the step are captured, uploaded
            once, and re-launched back to back with CUDA-event timing (abpoa_gpu_replay).
  e2e       the same metric through the public C ABI (abpoa_gpu_msa_batch) from HOST buffers:
            graph flattening, H2D, kernels, D2H of graph-CIGARs, host graph fusion, consensus --
            wall clock between barriers, max over ranks.
  roofline  dominant kernel (poa_align_kernel): algorithmic bytes = cells x S x (P + R x d) with
            the measured in-degree d, divided by the replay's kernel time, against the measured
            HBM copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline  the UNMODIFIED reference (oracle/_ref/libabpoa_ref.so, AVX2) on the host cores,
            one process per physical core, on a bounded sample of the same groups.
--impl reference prints the reference arm's line (CPU only; rank 0 alone runs).
--dump-outputs DIR  (rank 0) writes what the last timed step returned to its caller as DIR/<name>.npy: per group the DP
            cells, aligned reads and consensus length, and for a fixed sample of groups the consensus bases and their
            coverage (see dump_outputs).  The inputs are seeded, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

# one hardware work queue per stream of the batch engine (must be set before CUDA initialises)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
os.environ.setdefault("CUDA_MODULE_LOADING", "EAGER")

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "GCUPS (DP cells/s), global/convex 10 kbp"
REF_LIB = ROOT / "oracle" / "_ref" / "libabpoa_ref.so"      # the unmodified reference (oracle/Makefile builds it where its sources are)


def physical_cores() -> int:
    try:
        out = subprocess.run(["lscpu", "-p=core,socket"], capture_output=True, text=True).stdout
        cores = {ln for ln in out.splitlines() if ln and not ln.startswith("#")}
        if cores:
            return len(cores)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


# ------------------------------------------------------------------------------------------------
# reference arm (CPU): oracle/_ref/libabpoa_ref.so, one process per core, whole groups per process
# ------------------------------------------------------------------------------------------------
def rank_cpu_share(rank: int, world: int) -> list[int]:
    """CPUs for one rank when several ranks share the host: the allowed physical cores, sorted by
    (package, core), are cut into `world` contiguous slices and a rank takes ALL hardware threads
    of its slice (ranks 0..world/2-1 land on socket 0, the rest on socket 1 on a two-socket box)."""
    allowed = sorted(os.sched_getaffinity(0))
    by_core: dict[tuple[int, int], list[int]] = {}
    for c in allowed:
        try:
            pkg = int(Path(f"/sys/devices/system/cpu/cpu{c}/topology/physical_package_id").read_text())
            core = int(Path(f"/sys/devices/system/cpu/cpu{c}/topology/core_id").read_text())
        except Exception:
            pkg, core = 0, c
        by_core.setdefault((pkg, core), []).append(c)
    cores = sorted(by_core)
    n = len(cores)
    lo, hi = n * rank // world, n * (rank + 1) // world
    if hi <= lo:
        return allowed
    return sorted(c for k in cores[lo:hi] for c in by_core[k])


ALL_CPUS = sorted(os.sched_getaffinity(0))        # before any rank pinning: the reference arm may use every core of the box


def socket_cpus() -> dict[int, list[int]]:
    """One hardware thread per physical core, grouped by socket."""
    out: dict[int, dict[int, int]] = {}
    for c in ALL_CPUS:
        try:
            pkg = int(Path(f"/sys/devices/system/cpu/cpu{c}/topology/physical_package_id").read_text())
            core = int(Path(f"/sys/devices/system/cpu/cpu{c}/topology/core_id").read_text())
        except Exception:
            pkg, core = 0, c
        out.setdefault(pkg, {}).setdefault(core, c)
    return {p: sorted(v.values()) for p, v in out.items()}


def _ref_worker(args):
    wname, seeds, n_reads, length, cpu = args
    import resource
    if cpu is not None:
        try:
            os.sched_setaffinity(0, {cpu})
        except OSError:
            pass
    from abpoa_b200 import capi, synth
    from abpoa_b200.aligner import PoaSession
    w = synth.WORKLOADS[wname]
    lib = capi.load_library(REF_LIB)
    cells = 0
    reads_done = 0
    groups = [synth.make_group(seed, n_reads, length, w.err, w.cfg.m) for seed in seeds]     # outside the timed window
    cons = []
    with PoaSession(w.cfg, lib) as s:
        ru0 = resource.getrusage(resource.RUSAGE_SELF)
        t0 = time.perf_counter()
        for reads in groups:
            for a in s.run_reads(reads):
                cells += a.cells
            reads_done += len(reads)
            s.generate()
            cons.append(bytes(s.consensus()[0]) if s.consensus() else b"")
        dt = time.perf_counter() - t0
        ru1 = resource.getrusage(resource.RUSAGE_SELF)
    return cells, reads_done, dt, ru1.ru_utime - ru0.ru_utime, ru1.ru_stime - ru0.ru_stime, list(zip(seeds, cons))


def reference_pass(wname: str, n_groups: int, cpus: list[int], n_reads: int, length: int, base_seed: int):
    """Time the reference on `n_groups` groups spread over one process per CPU of `cpus` (each pinned).
    Returns a dict: cells, reads, wall_s, user_s, sys_s, cons {seed: consensus bytes}."""
    cores = len(cpus)
    seeds = [base_seed + g for g in range(n_groups)]
    shards = [(seeds[i::cores], cpus[i]) for i in range(cores)]
    shards = [s for s in shards if s[0]]
    ctx = mp.get_context("fork")
    with ctx.Pool(len(shards)) as pool:
        res = pool.map(_ref_worker, [(wname, s, n_reads, length, c) for s, c in shards])
    # all workers start together; the job ends when the slowest one does (process start-up,
    # read generation and imports are outside each worker's clock)
    cons = {}
    for r in res:
        cons.update(dict(r[5]))
    return {"cells": sum(r[0] for r in res), "reads": sum(r[1] for r in res), "wall_s": max(r[2] for r in res),
            "user_s": sum(r[3] for r in res), "sys_s": sum(r[4] for r in res), "procs": len(shards), "cons": cons}


def cpu_baseline_block(wname: str, w, ref_groups: int, base_seed: int) -> tuple[dict, dict]:
    """The unmodified reference on every physical core of the box (both sockets) and on the cores of ONE
    socket (what north_star calls the single-socket baseline); user+sys next to wall (SURVEY 8d: the
    reference's quadratic, sparsely touched slab makes it page-fault bound at 10 kbp)."""
    socks = socket_cpus()
    all_cores = sorted(c for v in socks.values() for c in v)
    one = socks[sorted(socks)[0]]
    a = reference_pass(wname, ref_groups or len(all_cores), all_cores, w.n_reads, w.length, base_seed)
    blk = {"value": a["cells"] / a["wall_s"] / 1e9, "unit": "GCUPS", "cores": a["procs"], "kind": "reference", "reads_per_s": a["reads"] / a["wall_s"],
           "wall_s": a["wall_s"], "user_s": a["user_s"], "sys_s": a["sys_s"],
           "sample": f"{len(a['cons'])} groups of the same workload ({a['reads']} reads, {a['cells'] / 1e9:.1f} G cells), one pinned process per physical core "
                     f"({a['procs']} cores, {len(socks)} sockets), {a['wall_s']:.1f} s wall; CPU time {a['user_s']:.0f} s user + {a['sys_s']:.0f} s sys"}
    if len(socks) > 1:
        b = reference_pass(wname, len(one), one, w.n_reads, w.length, base_seed)
        blk["single_socket"] = {"value": b["cells"] / b["wall_s"] / 1e9, "cores": b["procs"], "reads_per_s": b["reads"] / b["wall_s"],
                                "wall_s": b["wall_s"], "user_s": b["user_s"], "sys_s": b["sys_s"]}
    return blk, a


DUMP_SAMPLE_GROUPS = 256            # groups whose consensus and coverage are written by --dump-outputs (seeded choice)


def dump_outputs(out_dir: str, results) -> None:
    """The results of one step (BatchEngine.run_packed with keep_results=True), as .npy files under `out_dir`:
    group_dp_cells, group_n_aligned, group_cons_len (float64, one per group), sample_groups (the sampled group
    indices), sample_cons_offsets (float64, start of each sampled consensus in the concatenation, plus the end),
    sample_cons_bases and sample_cons_cov (float32, the first consensus of each sampled group, concatenated)."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    n = len(results)
    k = min(n, DUMP_SAMPLE_GROUPS)
    sample = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False)) if n else np.zeros(0, dtype=np.int64)
    first = lambda arrs: arrs[0] if arrs else np.zeros(0)
    bases = [first(results[g].cons) for g in sample]
    cov = [first(results[g].cov) for g in sample]
    arrays = {
        "group_dp_cells": np.array([r.dp_cells for r in results], dtype=np.float64),
        "group_n_aligned": np.array([r.n_aligned for r in results], dtype=np.float64),
        "group_cons_len": np.array([sum(len(c) for c in r.cons) for r in results], dtype=np.float64),
        "sample_groups": sample.astype(np.float64),
        "sample_cons_offsets": np.concatenate([[0], np.cumsum([len(b) for b in bases])]).astype(np.float64),
        "sample_cons_bases": np.concatenate(bases).astype(np.float32) if bases else np.zeros(0, dtype=np.float32),
        "sample_cons_cov": np.concatenate(cov).astype(np.float32) if cov else np.zeros(0, dtype=np.float32),
    }
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"--dump-outputs would write {total} bytes"
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self) -> dict:
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 3 + k and r[3 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="convex_10k")
    ap.add_argument("--groups", type=int, default=0, help="groups per GPU (default: the config's 1000)")
    ap.add_argument("--ref-groups", type=int, default=0, help="groups in one reference sample (default: one per core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if not REF_LIB.exists():
        if args.impl == "reference":
            ap.error(f"{REF_LIB} is not built")
        args.no_cpu_baseline = True          # the CPU baseline needs the reference library; the GPU measurement does not
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    from abpoa_b200 import synth
    w = synth.WORKLOADS[args.workload]
    n_groups = args.groups or w.n_groups
    cores = physical_cores()
    cfgdesc = {"workload": f"{args.workload}: {n_groups} groups/GPU x {w.n_reads} reads x {w.length} bp, err {w.err}, "
                           f"{'global' if w.cfg.align_mode == 0 else 'local'}, O={w.cfg.gap_open1},{w.cfg.gap_open2} E={w.cfg.gap_ext1},{w.cfg.gap_ext2}",
               "groups_per_gpu": n_groups, "reads_per_group": w.n_reads, "read_len": w.length,
               "l2_policy": "inputs larger than L2 (job blobs + DP planes of one step >> 126 MB)"}

    # ---------------------------------------------------------------- reference arm
    if args.impl == "reference":
        if rank != 0:
            return
        socks = socket_cpus()
        all_cores = sorted(c for v in socks.values() for c in v)
        cores = len(all_cores)
        ref_groups = args.ref_groups or cores
        # bounded sample: one group per core per step keeps the whole run within minutes
        per_step = []
        for s in range(args.warmup + args.steps):
            if s < args.warmup and s > 0:
                continue                      # the CPU needs no repeated warm-up; one untimed pass suffices
            r = reference_pass(args.workload, ref_groups, all_cores, w.n_reads, w.length, 1000 + 7919 * s)
            if s >= args.warmup:
                per_step.append(r)
        cells = sum(p["cells"] for p in per_step)
        reads = sum(p["reads"] for p in per_step)
        wall = sum(p["wall_s"] for p in per_step)
        user_s, sys_s = sum(p["user_s"] for p in per_step), sum(p["sys_s"] for p in per_step)
        val = cells / wall / 1e9
        sample = (f"{ref_groups} groups ({ref_groups * w.n_reads} reads) per step, one pinned process per physical core ({cores} cores, {len(socks)} sockets); "
                  f"cells counted from ab->abm->dp_beg/dp_end; CPU time {user_s:.0f} s user + {sys_s:.0f} s sys over {wall:.1f} s wall")
        single = None
        if len(socks) > 1:            # north_star's "single-socket" figure: the same sample shape on the cores of socket 0 only
            one = socks[sorted(socks)[0]]
            b = reference_pass(args.workload, len(one), one, w.n_reads, w.length, 1000)
            single = {"value": b["cells"] / b["wall_s"] / 1e9, "cores": b["procs"], "reads_per_s": b["reads"] / b["wall_s"], "wall_s": b["wall_s"], "user_s": b["user_s"], "sys_s": b["sys_s"]}
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": val, "unit": "GCUPS", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": wall / max(len(per_step), 1) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int16/int32 (AVX2)", "data": "synthetic", "config": cfgdesc, "reads_per_s": reads / wall,
            "cpu_baseline": {"value": val, "unit": "GCUPS", "cores": cores, "kind": "reference", "sample": sample, "user_s": user_s, "sys_s": sys_s, "wall_s": wall, "single_socket": single},
            "e2e": {"value": val, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    # ---------------------------------------------------------------- B200 arm
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # the version banner goes to stdout, which carries exactly one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from abpoa_b200 import capi
    from abpoa_b200.aligner import make_para
    from abpoa_b200.batch import BatchEngine, PackedGroups

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    groups = w.groups(n_groups, base_seed=1000 + 100000 * rank)       # independent groups per rank: no data-path collective
    packed = PackedGroups(groups)
    lib = capi.product()
    abpt = make_para(lib, w.cfg)
    # host threads: one per physical core at N=1 (32 measured best: more streams than hardware queues hurts);
    # with several ranks on one host every rank gets its own slice of cores and uses all their hardware threads
    if world > 1:
        share = rank_cpu_share(local_rank, world)
        os.sched_setaffinity(0, share)                 # the engine pins its workers inside the process's CPU set
        workers = int(os.environ.get("ABPOA_GPU_WORKERS", "0")) or max(4, min(32, len(share)))
    else:
        workers = int(os.environ.get("ABPOA_GPU_WORKERS", "0")) or max(4, min(32, (os.cpu_count() or 8) // 2))
    gpl = int(os.environ.get("ABPOA_GPU_GROUPS_PER_LAUNCH", "0"))      # 0: the engine spreads the groups over workers x pipe depth
    eng = BatchEngine(device=local_rank, n_workers=workers, groups_per_launch=gpl)

    for _ in range(args.warmup):
        eng.run_packed(abpt, packed, keep_results=False)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    eng.reset_stats()
    barrier()
    t0 = time.perf_counter()
    cells = 0
    cons_bases = 0
    last = None
    for step in range(args.steps):
        if args.dump_outputs and step == args.steps - 1:
            # the last step also hands its consensus arrays back to the caller, to be written after the timed region
            last = eng.run_packed(abpt, packed, keep_results=True)
            res = [(r.dp_cells, r.n_aligned, sum(len(c) for c in r.cons)) for r in last]
        else:
            res = eng.run_packed(abpt, packed, keep_results=False)
        cells += sum(r[0] for r in res)
        cons_bases += sum(r[2] for r in res)
    barrier()
    elapsed = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    st = eng.stats()
    if last is not None and rank == 0:
        dump_outputs(args.dump_outputs, last)
        last = None
    t = torch.tensor([elapsed, st["chain_device_ms"]], dtype=torch.float64, device="cuda")
    c = torch.tensor([float(cells), float(packed.total_reads * args.steps), float(st["launches"]), float(st["h2d_bytes"]), float(st["d2h_bytes"]),
                      float(st["chain_cells"]), float(st["chain_groups"]), float(st["chain_fallback_groups"]), st["chain_dp_ms"], st["chain_fuse_ms"],
                      st["chain_wait_ms"], float(st["chain_dp_launches"])],
                     dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
    elapsed, chain_ms = [float(x) for x in t.tolist()]
    tot_cells, tot_reads, launches, h2d, d2h, chain_cells, chain_groups, chain_fallback, chain_dp_ms, chain_fuse_ms, chain_wait_ms, chain_alns = [float(x) for x in c.tolist()]
    e2e_gcups = tot_cells / elapsed / 1e9
    used_chain = chain_groups > 0 and chain_ms > 0

    # device-resident measurement of the DP + backtrace kernel ALONE: capture one step's alignment jobs through the launch
    # engine, upload once, replay back to back with CUDA-event timing (per-launch numbers for the roofline)
    eng.run_packed(abpt, packed, keep_results=False, capture=True)
    barrier()
    rp = eng.replay(abpt, warmup=1, repeats=args.steps)
    eng.clear_capture()
    kt = torch.tensor([rp["kernel_ms"]], dtype=torch.float64, device="cuda")
    kc = torch.tensor([float(rp["cells"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(kt, op=dist.ReduceOp.MAX)
        dist.all_reduce(kc, op=dist.ReduceOp.SUM)
    kernel_s = float(kt.item()) / 1e3
    kernel_only_gcups = float(kc.item()) / kernel_s / 1e9
    # `value`: whole-job throughput with the inputs resident in HBM when the timed region starts.  With the chain engine that
    # is the complete progressive MSA on the device (every alignment AND every graph fusion, chain dependencies included),
    # CUDA events from "reads uploaded" to "last group fused", max over ranks.  Workloads outside the chain's scope (local
    # mode) keep the replay of all captured alignment jobs.
    value = chain_cells / (chain_ms / 1e3) / 1e9 if used_chain else kernel_only_gcups

    # N > 1: exercise the scatter -> compute -> gather path itself (abpoa_b200.parallel.distributed_msa: packed reads scattered
    # from rank 0 and packed consensus gathered back as uint8 tensors over NCCL) on a small set, outside the timed region
    dist_check = None
    if world > 1:
        from abpoa_b200.parallel import distributed_msa
        small = w.groups(8 * world, base_seed=900000)
        small = [[r[: min(len(r), 1500)] for r in g[: min(len(g), 10)]] for g in small]
        run_here = lambda c_, gs: [list(r.cons) + list(r.cov) for r in eng.run(c_, gs)]
        got = distributed_msa(small if rank == 0 else None, w.cfg, runner=run_here)
        if rank == 0:
            import numpy as np
            local = run_here(w.cfg, small)
            same = sum(1 for a, b in zip(got, local) if len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b)))
            dist_check = {"groups": len(small), "identical_to_single_rank": same, "backend": dist.get_backend(), "ranks": world}

    # parity sample: consensus of the first groups of rank 0 against the reference's (computed in the cpu_baseline leg)
    sample_cons = None
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        k = min(n_groups, args.ref_groups or len([c_ for v in socket_cpus().values() for c_ in v]))
        sub = PackedGroups(groups[:k])
        sample_cons = [bytes(r.cons[0]) if r.cons else b"" for r in eng.run_packed(abpt, sub, keep_results=True)]

    if rank != 0:
        eng.close()
        if world > 1:
            dist.destroy_process_group()
        return

    # roofline of the dominant kernel (the DP + backtrace kernel): algorithmic bytes per cell = S * (P + R * d), SURVEY 8d
    gap = {0: (1, 1), 1: (3, 2), 2: (5, 3)}[2 if (w.cfg.gap_open1 and w.cfg.gap_open2) else (1 if w.cfg.gap_open1 else 0)]
    P, R = gap
    d = rp["preds"] / max(rp["rows"], 1)
    bytes16 = rp["cells16"] * 2 * (P + R * d)
    bytes32 = (rp["cells"] - rp["cells16"]) * 4 * (P + R * d)
    achieved = (bytes16 + bytes32) / (rp["kernel_ms"] / 1e3) / 1e9
    peaks_file = ROOT / "MEASURED_PEAKS.json"
    if peaks_file.exists():
        peak = json.loads(peaks_file.read_text())["hbm_gbs"]
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    # DRAM bytes of one launch of the dominant kernel from the committed `ncu --set full` capture (profiles/)
    traffic, traffic_note, dram_frac = None, None, None
    gapname = {1: "linear", 3: "affine", 5: "convex"}[P]
    for cand in (ROOT / "profiles" / f"r02_ncu_traffic_{gapname}.json", ROOT / "profiles" / "r01_ncu_traffic.json"):
        if cand.exists():
            t_ = json.loads(cand.read_text())
            if cand.name.startswith("r01") and P != 5:
                continue
            traffic = t_["dram_bytes_read"] + t_["dram_bytes_write"]
            dram_frac = traffic / (t_["duration_ms"] / 1e3) / 1e9 / peak
            traffic_note = (f"ncu capture of one launch of {t_.get('kernel', 'the kernel').split('(')[0]} ({t_['jobs']} jobs, {t_['duration_ms']:.1f} ms): "
                            f"{t_['dram_bytes_write'] / 1e9:.1f} GB written + {t_['dram_bytes_read'] / 1e9:.1f} GB read; see {t_['source']}")
            break
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note,
                "dram_frac_measured": dram_frac,
                "kernel": "poa_align_kernel_p16 / poa_chain_align_kernel_p16 (same job function)", "bytes_per_cell": (bytes16 + bytes32) / max(rp["cells"], 1), "mean_in_degree": d,
                "peak_source": peak_src, "launches_per_pass": rp["launches"], "replay_mismatches": rp["mismatches"],
                "int16_cell_fraction": rp["cells16"] / max(rp["cells"], 1), "kernel_alone_gcups": kernel_only_gcups,
                "timing": "CUDA events around back-to-back replay launches of all captured alignment jobs of one step (kernel alone on the device)"}

    cpu = None
    parity = None
    if not args.no_cpu_baseline and world == 1:        # N=1 only (the contract); workers are pinned over ALL cores of the box
        cpu, ref_run = cpu_baseline_block(args.workload, w, args.ref_groups, 1000)
        if sample_cons is not None:                    # rank 0's groups g = seed 1000 + g: the very groups the reference just ran
            same = sum(1 for g, cb in enumerate(sample_cons) if ref_run["cons"].get(1000 + g) == cb)
            parity = {"groups_compared": len(sample_cons), "consensus_identical": same,
                      "what": "consensus of the first groups of the timed workload, product (this run) vs the unmodified reference (cpu_baseline leg)"}

    chain = None
    if used_chain:
        chain = {"device_ms_per_step": chain_ms / args.steps, "groups_on_device": int(chain_groups / args.steps), "groups_handed_back": int(chain_fallback / args.steps),
                 "backtrace_share_of_dp_kernel_cycles": st["bt_clk"] / max(st["fwd_clk"] + st["bt_clk"], 1)}
        if st["chain_free_running"]:
            # free-running schedule: two persistent kernels, every group advances at its own pace.  Per-group averages of where a
            # group's chain spends its time: inside its alignments, waiting for a fuse worker (queueing + the fuse), inside the fuse.
            ng = max(chain_groups, 1.0)
            chain.update({"schedule": "free-running (2 persistent kernels per wave)",
                          "per_group_ms_in_alignments": chain_dp_ms / ng, "per_group_ms_waiting_for_fuse": chain_wait_ms / ng,
                          "per_group_ms_in_fuse": chain_fuse_ms / ng, "mean_alignment_ms": chain_dp_ms / max(chain_alns, 1.0),
                          "dp_share_of_chain_time": chain_dp_ms / max(chain_dp_ms + chain_wait_ms, 1e-9)})
        else:
            chain.update({"schedule": "lock-step rounds (2 kernels per round and cohort)",
                          "dp_kernel_ms_sum_over_streams": chain_dp_ms / args.steps, "fuse_kernel_ms_sum_over_streams": chain_fuse_ms / args.steps,
                          "dp_share_of_kernel_time": chain_dp_ms / max(chain_dp_ms + chain_fuse_ms, 1e-9)})
    print(json.dumps({
        "metric": METRIC, "value": value, "unit": "GCUPS", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int16 (packed int16x2 DPX arithmetic; int32 kernel only as overflow fallback)", "data": "synthetic", "config": cfgdesc,
        "clocks": clocks, "reads_per_s": tot_reads / elapsed,
        "value_definition": ("device-resident progressive MSA (chain engine): every alignment and every graph fusion of the step on the GPU, reads resident in HBM, CUDA events"
                             if used_chain else "replay of all captured alignment jobs from HBM, CUDA events"),
        "e2e": {"value": e2e_gcups, "unit": "GCUPS", "h2d_bytes_per_step": h2d / args.steps / world, "d2h_bytes_per_step": d2h / args.steps / world,
                "reads_per_s": tot_reads / elapsed, "per_gpu": e2e_gcups / world, "host_threads_per_gpu": workers,
                "engine": (("device-resident chain, free-running (one persistent alignment kernel + one persistent fuse kernel per wave" if st["chain_free_running"]
                            else "device-resident chain, round schedule (align + fuse kernels per round") + "; host only for upload / final consensus)") if used_chain
                          else "launch engine: pipelined launches, one per half-chunk round, host graph fusion"},
        "gpu_launches": int(launches),
        "roofline": roofline, "cpu_baseline": cpu, "parity_sample": parity, "chain": chain, "distributed_check": dist_check,
        "kernel_only": {"ms_per_pass": rp["kernel_ms"], "ms_min": rp["kernel_ms_min"], "jobs": rp["n_jobs"], "cells": rp["cells"], "hbm_resident_input_bytes": rp["input_bytes"],
                        "gcups": kernel_only_gcups},
    }))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
