#!/usr/bin/env python
"""bench.py — aligned long-read Gbp/s through lead -> cluster -> consensus (BASELINE.json metric).

    python bench.py --gpus 1 --steps K --warmup W                  # this repo's CUDA path
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # one rank per GPU
    python bench.py --impl reference --gpus N --steps K --warmup W  # CPU arm (oracle port, host cores)
    python bench.py ... --dump-outputs DIR                          # also the last timed step's outputs, DIR/<name>.npy

A "step" is one pass of the hot path over the whole synthetic workload (--config: BASELINE config 2 by default:
30x ONT whole genome, 24 GRCh38-length contigs, ~6M reads at --scale 1; 1 = one 1 Mb contig, 3 = 60x HiFi --mosaic,
5 = INS-heavy region).  With N ranks the contigs are LPT-sharded over the ranks (strong scaling: the genome is fixed),
every rank runs the three stages on its contigs and the per-rank candidate buffers (records, ALT arena, read names) are
concatenated with one NCCL all-gather issued by the library (snfb_allgather_candidates).  `value` is timed with the inputs resident in HBM (CUDA events on the
library's stream, max over ranks); `e2e` goes through the same C-ABI call with HOST buffers:
pinned host arenas -> H2D -> kernels -> D2H of the candidate SoA and ALT bytes, every step.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def passing_mask(blk, cfg):
    """(mask, query_alignment_length) of the records that pass the A2 filters (leadprov.py:494-503)"""
    rec = blk.rec
    first = blk.cigar[rec["cigar_off"]]
    last = blk.cigar[rec["cigar_off"] + rec["n_cigar"] - 1]
    lead = np.where((first & 15) == 4, first >> 4, 0).astype(np.int64)
    trail = np.where(((last & 15) == 4) & (rec["n_cigar"] > 1), last >> 4, 0).astype(np.int64)
    alen = rec["l_seq"].astype(np.int64) - lead - trail
    t = blk.task[rec["task"]]
    ok = (rec["mapq"] >= cfg.mapq) & ((rec["flag"] & 256) == 0) & (alen >= cfg.min_alignment_length) & (rec["pos"] >= t["start"]) & (rec["pos"] < t["end"])
    return ok, alen


def aligned_bp_passing(blk, cfg):
    """sum of query_alignment_length over the records that pass the A2 filters (leadprov.py:494-503)"""
    if len(blk.rec) == 0:
        return 0
    ok, alen = passing_mask(blk, cfg)
    return int(alen[ok].sum())


def algorithmic_bytes_stage_a(blk, cfg):
    """Algorithmic bytes of one launch of the streaming kernel k_chunk_sum (DESIGN.md section 3): the CIGAR16 words of every passing
    record (2 bytes each, the record's span rounded up to 16 bytes) read once, plus per chunk of 16 groups an 8-byte descriptor read and
    an 8-byte (read advance, reference advance) pair written."""
    if len(blk.rec) == 0:
        return 0, 0
    ok, _ = passing_mask(blk, cfg)
    g = (blk.rec16["n_cigar"].astype(np.int64)[ok] + 7) // 8
    chunks = int(((g + 15) // 16).sum())
    rd = int(16 * g.sum()) + 8 * chunks
    return rd + 8 * chunks, rd


class ClockSampler(threading.Thread):
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.05)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(name="k_chunk_sum_dram.json"):
    """DRAM bytes per launch of a kernel (group) from the committed ncu capture, if any."""
    p = os.path.join(ROOT, "profiles", name)
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return None


def bind_near_gpu(index):
    """Run on the CPUs of the GPU's NUMA node while the block is generated, packed and pinned: first-touch then places the host
    arenas next to the GPU's PCIe root, so the e2e host->device copy does not cross the socket interconnect.  Best effort."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(index)
        dev = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{dev}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            log(f"[bench] GPU {index} ({dev}): no NUMA node reported")
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        old = os.sched_getaffinity(0)
        new = cpus & old
        if not new or new == old:
            log(f"[bench] GPU {index} ({dev}) is on NUMA node {node}; affinity unchanged ({len(old)} CPUs)")
            return None
        os.sched_setaffinity(0, new)
        log(f"[bench] GPU {index} ({dev}) is on NUMA node {node}: building the block on its {len(new)} of {len(old)} CPUs")
        return old
    except Exception as e:          # no sysfs entry, old torch, container without the node files
        log(f"[bench] NUMA binding skipped: {e}")
        return None


# ------------------------------------------------------------------------------------------------ workloads (BASELINE.json configs)
def workload_spec(args):
    """contig lengths, reference CLI arguments and a description for --config"""
    from sniffles_b200 import synth
    c, sc = args.config, args.scale
    if c == 1:
        return dict(lens=[int(1_000_000 * sc)], cli=[], coverage=20.0, desc=f"BASELINE config 1: one 1 Mb contig x scale {sc}, ~200 ONT reads of ~100 kb @20x, germline")
    if c == 2:
        return dict(lens=[max(200000, int(x * sc)) for x in synth.GRCH38], cli=[], coverage=30.0, desc=f"BASELINE config 2: synthetic 30x ONT WGS, 24 GRCh38-length contigs x scale {sc}, germline")
    if c == 3:
        return dict(lens=[max(200000, int(x * sc)) for x in synth.GRCH38], cli=["--mosaic"], coverage=60.0, desc=f"BASELINE config 3: synthetic 60x PacBio HiFi WGS, 24 GRCh38-length contigs x scale {sc}, --mosaic low-VAF")
    if c == 5:
        return dict(lens=[int(5_000_000 * sc)], cli=[], coverage=20.0, desc=f"BASELINE config 5: INS-heavy stress, one 5 Mb region x scale {sc}, ~5000 sites x 20 reads, insertions 50-5000 bp")
    raise SystemExit(f"--config {c}: no synthetic shape (config 4, population combine, is not part of this path)")


def workload(args, mask, threads):
    from sniffles_b200 import synth
    t0 = time.time()
    blk = synth.config_block(args.config, args.scale, threads=threads, contig_mask=mask)
    dt = time.time() - t0
    log(f"[bench] generated config {args.config} scale {args.scale}: {len(blk.rec)} records, {blk.cigar.nbytes / 1e9:.2f} GB CIGAR, {blk.seq.nbytes / 1e9:.2f} GB seq in {dt:.1f}s")
    return blk, dt


def cpu_sample(blk, cfg, ccfg, threads, target_bp=6e9):
    """Bounded sample for the CPU arm: the smallest tasks of the block first, up to ~target_bp aligned bases; one host thread per contig
    (the reference's own grain of parallelism, sniffles:313-358)."""
    import oracle.oracle as orc
    rec = blk.rec
    tasks, counts = np.unique(rec["task"], return_counts=True)
    chosen, bp = [], 0
    for t in tasks[np.argsort(counts)]:
        chosen.append(int(t))
        bp += int(rec["l_seq"][rec["task"] == t].sum())
        if bp >= target_bp:
            break
    keep = np.isin(rec["task"], chosen)
    sub = type(blk)(rec=np.ascontiguousarray(rec[keep]), cigar=blk.cigar, var=blk.var, seq=blk.seq, task=blk.task, contig=blk.contig, tr=blk.tr, contig_names=blk.contig_names)
    abp = aligned_bp_passing(sub, cfg)
    nthr = max(1, min(threads, len(chosen)))
    t0 = time.perf_counter()
    res = orc.run(sub, ccfg, 3, nthr)
    dt = time.perf_counter() - t0
    cpu_sample.last_result = res
    cpu_sample.whole_block = len(chosen) == len(tasks)
    return dict(value=abp / dt / 1e9, unit="Gbp/s", cores=nthr, kind="port",
                sample=f"oracle/snf_oracle.c (C port of the pure-Python reference) on tasks {sorted(chosen)} = {abp / 1e9:.3f} Gbp aligned, {len(res.cand)} candidates, {dt:.2f}s"), abp, dt


def python_reference_baseline():
    """The committed measurement of the reference's own Python code (oracle/pyref/timing.py, BASELINE.md §3), labelled as measured
    elsewhere: the benchmark reads nothing outside this repository.  Never a silent quote."""
    p = os.path.join(ROOT, "tests", "expected", "python_reference_timing.json")
    if os.path.exists(p):
        with open(p) as f:
            m = json.load(f)
        return {"absent_on_this_box": True, "measured_elsewhere": m}
    return {"absent_on_this_box": True}


HASH_FIELDS = ["task", "svtype", "pos", "end", "svlen", "support", "qual", "precise", "fwd", "rev", "support_long", "support_sa", "cov_upstream", "cov_start", "cov_center", "cov_end",
               "cov_downstream", "hap_counts", "sa_count", "sa_total", "bnd_mate_contig", "bnd_mate_pos", "bnd_is_first", "bnd_is_reverse", "n_strands", "support_inline", "lead_n", "long_n",
               "alt_len", "hp_top", "hp_support", "hp_other", "ps_top", "ps_top_null", "ps_support", "ps_other", "stdev_pos", "stdev_len"]


def callset_hash(cand, alt, rnames, rn_off):
    """sha256 of the call set in emission order (task id, then the producing rank's own order): every candidate field that does not
    depend on where a rank's arenas start, the ALT bytes and the read-name hashes of every candidate.  Identical for every sharding."""
    import hashlib
    order = np.argsort(cand["task"], kind="stable")
    c = cand[order]
    h = hashlib.sha256()
    for f in HASH_FIELDS:
        h.update(np.ascontiguousarray(c[f]).tobytes())
    alt = np.asarray(alt)
    ao, al = cand["alt_off"], cand["alt_len"]
    lo, hi = rn_off[:-1], rn_off[1:]
    for i in order:
        if ao[i] >= 0:
            h.update(alt[int(ao[i]):int(ao[i]) + int(al[i])].tobytes())
        h.update(rnames[int(lo[i]):int(hi[i])].tobytes())
    return h.hexdigest()


def committed_hashes():
    p = os.path.join(ROOT, "tests", "expected", "callset_hashes.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return {}


DUMP_BYTES = 60_000_000         # --dump-outputs: array bytes in all, under 64 MB with the .npy headers
DUMP_SEED = 1729


def _float_columns(a, name):
    """{file name: column} of a plain or structured array, rows first: float32 where that is exact (integers of up to 16 bits,
    float32), float64 otherwise; a 64-bit integer column (hashes, arena offsets) becomes two exact columns `<name>_hi`, `<name>_lo`.
    Every value written is finite: a floating-point column (where NaN stands for an undefined result, e.g. the stdev of one value)
    has its non-finite values written as 0 and a column `<name>_nonfinite` saying which they were: 0 finite, 1 NaN, 2 +inf, 3 -inf."""
    if a.dtype.names:
        out = {}
        for f in a.dtype.names:
            if not f.startswith("_"):
                out.update(_float_columns(a[f], f"{name}.{f}"))
        return out
    if a.dtype.kind in "iu" and a.dtype.itemsize == 8:
        u = a.astype("<u8")
        return {f"{name}_hi": (u >> np.uint64(32)).astype(np.float64), f"{name}_lo": (u & np.uint64(0xFFFFFFFF)).astype(np.float64)}
    out = a.astype(np.float32 if a.dtype.itemsize <= 2 or a.dtype == np.float32 else np.float64)
    if a.dtype.kind != "f":
        return {name: out}
    kind = np.select([np.isnan(out), out == np.inf, out == -np.inf], [1, 2, 3], 0).astype(np.float32)
    return {name: np.where(kind == 0, out, 0).astype(out.dtype), f"{name}_nonfinite": kind}


def dump_outputs(dirname, tables, prefix=""):
    """--dump-outputs: every array of `tables` ({name: array, rows first}) as DIR/<prefix><name>[.<field>].npy.  A table larger than its
    share of DUMP_BYTES (the smaller tables are kept whole first) keeps a seeded sample of its rows, the same rows for the same row
    count, whose indices go to <name>.rows.npy.  The dump lets two builds be compared output for output on identical inputs."""
    os.makedirs(dirname, exist_ok=True)
    tables = {k: np.asarray(a) for k, a in tables.items() if a is not None}
    row_bytes = {k: sum(c.itemsize * max(1, c[:1].size) for c in _float_columns(a[:1], k).values()) for k, a in tables.items()}
    left, order = DUMP_BYTES, sorted(tables, key=lambda k: len(tables[k]) * row_bytes[k])
    for i, k in enumerate(order):
        a, share = tables[k], left // (len(order) - i)
        if len(a) * row_bytes[k] > share:
            m = share // (row_bytes[k] + 8)
            rows = np.sort(np.random.default_rng(DUMP_SEED).choice(len(a), m, replace=False))
            log(f"[bench] --dump-outputs: {k} sampled, {m} of {len(a)} rows")
            np.save(os.path.join(dirname, f"{prefix}{k}.rows.npy"), rows.astype(np.float64))
            a = a[rows]
            left -= 8 * m
        for name, col in _float_columns(a, k).items():
            np.save(os.path.join(dirname, f"{prefix}{name}.npy"), col)
            left -= col.nbytes


def result_tables(res):
    """the arrays a caller of Context.run / oracle.run receives"""
    return {"leads": res.leads, "cand": res.cand, "cand_leads": res.cand_leads, "rnames": res.rnames, "rn_off": res.rn_off,
            "task_cov_mean": res.task_cov_mean, "alt": res.alt}


PARITY_FIELDS = ["task", "svtype", "pos", "end", "svlen", "support", "qual", "precise", "fwd", "rev", "cov_upstream", "cov_start", "cov_center", "cov_end",
                 "cov_downstream", "sa_count", "bnd_mate_contig", "bnd_mate_pos", "lead_n", "alt_off", "alt_len", "stdev_pos", "stdev_len"]


def same_candidates(dev, ora):
    """bit-for-bit comparison of the device run with the oracle pass the cpu_baseline leg just timed on the same block (checker only)"""
    if len(dev.cand) != len(ora.cand) or len(dev.alt) != len(ora.alt):
        return False
    for f in PARITY_FIELDS:
        a, b = dev.cand[f], ora.cand[f]
        if not (((a == b) | ((a != a) & (b != b))).all()):
            return False
    return bool((np.asarray(dev.alt) == np.asarray(ora.alt)).all())


def sample_mask(args, spec):
    """contigs of the CPU arm's bounded sample (smallest first, up to --cpu-sample-gbp of sequenced bases)"""
    lens = spec["lens"]
    mask, bp = [False] * len(lens), 0.0
    for c in sorted(range(len(lens)), key=lambda k: lens[k]):
        mask[c] = True
        bp += spec["coverage"] * lens[c]
        if bp >= args.cpu_sample_gbp * 1e9:
            break
    return mask


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from sniffles_b200 import abi, config as sconfig
    spec = workload_spec(args)
    cfg = sconfig.default_config(*spec["cli"])
    ccfg = abi.Config.from_sniffles(cfg)
    ncores = os.cpu_count() or 1
    # generate only the contigs the bounded sample will use
    blk, _ = workload(args, sample_mask(args, spec) if len(spec["lens"]) > 1 else None, ncores)
    per_step = []
    info = None
    for i in range(args.warmup + args.steps):
        info, abp, dt = cpu_sample(blk, cfg, ccfg, ncores, target_bp=args.cpu_sample_gbp * 1e9)
        if i >= args.warmup:
            per_step.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, result_tables(cpu_sample.last_result))
    ms = 1e3 * sum(per_step) / len(per_step)
    val = abp / (ms / 1e3) / 1e9
    info["value"] = val
    print(json.dumps({"impl": "reference", "metric": "aligned long-read Gbp/s through lead->cluster->consensus", "value": val, "unit": "Gbp/s",
                      "n_gpus": args.gpus, "steps": len(per_step), "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                      "vs_baseline": None, "dtype": "int32", "data": "synthetic",
                      "config": {"workload": f"{spec['desc']}; CPU arm on a bounded sample ({info['sample']})"},
                      "cpu_baseline": info, "cpu_baseline_python": python_reference_baseline(),
                      "e2e": {"value": val, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def consensus_algorithmic_bytes(res):
    """SURVEY 8d stage C: per INS candidate with a consensus, sum over its seq-bearing leads of ceil(len / 2) packed bases read + len(best) ALT bytes written"""
    c = res.cand
    ins = (c["svtype"] == 0) & (c["alt_off"] >= 0)
    if not ins.any():
        return 0
    has = (res.cand_leads["flags"] & (1 << 10)) != 0
    nb = np.where(has, (res.cand_leads["seq_len"].astype(np.int64) + 1) // 2, 0)
    cs = np.concatenate([[0], np.cumsum(nb)])
    lo, n = c["lead_off"][ins].astype(np.int64), c["lead_n"][ins].astype(np.int64)
    return int((cs[lo + n] - cs[lo]).sum() + c["alt_len"][ins].astype(np.int64).sum())


def run_b200(args):
    import torch
    from sniffles_b200 import abi, binding, config as sconfig, dist as sdist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()          # rank 0 has finished build() before anybody loads the libraries
    spec = workload_spec(args)
    cfg = sconfig.default_config(*spec["cli"])
    ccfg = abi.Config.from_sniffles(cfg)
    lens = spec["lens"]
    owner = sdist.lpt_assign(lens, world)
    mask = [o == rank for o in owner] if world > 1 else None
    ncores = os.cpu_count() or 1
    old_affinity = bind_near_gpu(local)
    prep = {}
    blk, prep["generate_s"] = workload(args, mask, max(1, min(len(os.sched_getaffinity(0)), ncores // world if world > 1 else ncores)))
    abp_local = aligned_bp_passing(blk, cfg)
    L = binding.lib()
    t0 = time.time()
    blk.pack16()            # BAM CIGAR words -> CIGAR16, once per block (part of packing the block, like dropping the base qualities)
    prep["pack_cigar16_s"] = time.time() - t0
    log(f"[bench] packed CIGAR16: {blk.cigar.nbytes / 1e9:.2f} GB -> {blk.cigar16.nbytes / 1e9:.2f} GB in {prep['pack_cigar16_s']:.1f}s")
    pinned = []
    if not args.no_pin:
        t0 = time.time()
        for a in (blk.rec16, blk.cigar16, blk.var, blk.seq):
            if a.nbytes and L.snfb_pin_host(C.c_void_p(a.ctypes.data), a.nbytes) == 0:
                pinned.append(a)
        prep["pin_s"] = time.time() - t0
        log(f"[bench] pinned {sum(a.nbytes for a in pinned) / 1e9:.2f} GB of host arenas in {prep['pin_s']:.1f}s")
    if old_affinity:            # every thread (the OpenMP pool was created under the narrow mask) gets all CPUs back
        for tid in os.listdir("/proc/self/task"):
            try:
                os.sched_setaffinity(int(tid), old_affinity)
            except OSError:
                pass
    ctx = binding.Context(local)
    ctx.set_config(ccfg)
    os.environ.setdefault("NCCL_DEBUG", "WARN")          # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line
    if world > 1:           # the library's own NCCL communicator: the id travels through the launcher's process group
        box = [binding.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        ctx.comm_init(box[0], rank, world)
    ctx.load(blk)

    def step():
        res = ctx.run(want_leads=False, want_cands=True, want_seqs=True, copy=False)
        if world > 1:       # ONE all-gather of the per-rank candidate buffers before VCF emission (SURVEY 8e), result left in device memory
            ctx.allgather_candidates(device_only=True)
        return res

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    for _ in range(args.warmup):
        res = step()
    barrier()
    launches0, reruns0 = ctx.launch_count(), ctx.rerun_count()
    sampler = ClockSampler(local)
    sampler.start()
    dev_ms, kern = 0.0, {}
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = step()
        for name, ms, by in ctx.timings():
            if name == "h2d_records":
                continue
            if name == "total":
                dev_ms += ms
            else:
                kern.setdefault(name, [0.0, by])[0] += ms
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    launches = ctx.launch_count() - launches0
    reruns = ctx.rerun_count() - reruns0
    if args.dump_outputs:           # before the runs below reuse the library's output buffers that `res` views
        dump_outputs(args.dump_outputs, result_tables(res), f"rank{rank}." if world > 1 else "")
    # max over ranks
    tt = torch.tensor([dev_ms, wall * 1e3, float(abp_local)], device="cuda", dtype=torch.float64)
    if dist is not None:
        mx = tt.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = tt.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_ms_max, wall_ms_max, abp_total = float(mx[0]), float(mx[1]), float(sm[2])
    else:
        dev_ms_max, wall_ms_max, abp_total = dev_ms, wall * 1e3, float(abp_local)
    ms_per_step = wall_ms_max / args.steps
    value = abp_total / (ms_per_step / 1e3) / 1e9

    # ---- end to end through the C ABI with host buffers (H2D + kernels + D2H every step) ----
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    full_bytes = blk.rec16.nbytes + blk.cigar16.nbytes + blk.var.nbytes + blk.seq.nbytes
    ctx.load(blk, seq_on_demand=not args.e2e_full_seq)          # untimed: sizes the seq-on-demand buffers
    step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ctx.load(blk, seq_on_demand=not args.e2e_full_seq)      # host arenas; the 4-bit seq arena is fetched on demand (slices only)
        res = step()
    slice_bytes = sum(by for name, ms, by in ctx.timings() if name == "h2d_seq_slices")
    h2d = blk.rec16.nbytes + blk.cigar16.nbytes + blk.var.nbytes + (blk.seq.nbytes if args.e2e_full_seq else slice_bytes)
    barrier()
    e2e_wall = (time.perf_counter() - t0) / e2e_steps
    d2h = res.cand.nbytes + res.cand_leads.nbytes + res.rnames.nbytes + res.alt.nbytes
    # the same call fed the BAM's own 32-bit CIGAR words: the library converts them to CIGAR16 on the host inside snfb_load_records
    t0 = time.perf_counter()
    ctx.load(blk, seq_on_demand=not args.e2e_full_seq, cigar16=False)
    step()
    barrier()
    e2e_bam32 = time.perf_counter() - t0
    et = torch.tensor([e2e_wall, e2e_bam32], device="cuda", dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(et, op=dist.ReduceOp.MAX)
    e2e_val = abp_total / float(et[0]) / 1e9

    # ---- parity: the gathered call set of this run against the committed hash of the N = 1 run (itself checked against the oracle) ----
    ctx.load(blk)
    full = ctx.run(want_leads=True, want_cands=True, want_seqs=True, copy=False)       # also the run the full-size parity check compares with the oracle
    if world > 1:
        g = ctx.allgather_candidates(device_only=False)
        n_all = g.n_cand
        digest = callset_hash(g.cand, g.alt, g.rnames, g.rn_off) if rank == 0 else None
    else:
        n_all = len(full.cand)
        digest = callset_hash(full.cand, full.alt, full.rnames, full.rn_off)
    key = f"config{args.config}_scale{args.scale}"
    committed = committed_hashes().get(key)

    # ---- rooflines: the streaming stage-A kernel, and the consensus kernels (dominant on config 5) ----
    peak, peak_src = measured_peak()
    alg, alg_read = algorithmic_bytes_stage_a(blk, cfg)
    k_ms = kern.get("k_scan", [0.0, 0])[0] / args.steps
    achieved = alg / (k_ms / 1e3) / 1e9 if k_ms > 0 else 0.0
    traffic = ncu_traffic("k_chunk_sum_dram.json") if (args.config == 2 and args.scale == 1.0 and world == 1) else None      # the capture is of this workload at full size
    roof_a = {"bound": "hbm", "kernel": "extract::k_chunk_sum", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
              "peak_source": peak_src, "algorithmic_bytes_per_launch": alg, "kernel_ms": k_ms, "traffic": traffic.get("dram_bytes_per_launch") if traffic else None}
    c_ms = sum(kern.get(k, [0.0, 0])[0] for k in ("consensus", "consensus_align", "consensus_vote")) / args.steps
    c_alg = consensus_algorithmic_bytes(full)
    c_ach = c_alg / (c_ms / 1e3) / 1e9 if c_ms > 0 else 0.0
    roof_c = {"bound": "hbm", "kernel": "consensus::k_prep + k_align + k_vote", "achieved": c_ach, "peak": peak, "unit": "GB/s", "frac": c_ach / peak if peak else None, "peak_source": peak_src,
              "algorithmic_bytes_per_launch": c_alg, "kernel_ms": c_ms, "traffic": (ncu_traffic("consensus_dram.json") or {}).get("dram_bytes_per_launch") if traffic else None}
    # `roofline` = the kernel (group) that moves the most algorithmic bytes of the step: the CIGAR stream on the genome-sized configs, the
    # consensus group on the INS-heavy config 5.  By TIME the latency-bound kernels can be longer (round 2, config 2: consensus k_align 1.37 ms and
    # the cluster kernel 1.07 ms against 0.87 ms for the stream); `rooflines` lists both groups and `stage_ms` every stage.
    roof = dict(roof_c if c_alg > alg else roof_a)
    roof["choice"] = "kernel group with the most algorithmic bytes per step; both groups are in `rooflines`"
    if rank == 0:
        out = {"metric": "aligned long-read Gbp/s through lead->cluster->consensus", "value": value, "unit": "Gbp/s", "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_per_step, "device_ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": "int32", "data": "synthetic",
               "config": {"workload": f"{spec['desc']}, {abp_total / 1e9:.3f} Gbp aligned",
                          "records_rank0": int(len(blk.rec)), "candidates_total": int(n_all), "parallelism": f"contig LPT over {world} GPU(s), one NCCL all-gather (library call) of candidate records + ALT arena + read names",
                          "l2": f"inputs {full_bytes / 1e9:.2f} GB per rank vs 126 MB L2" + ("" if full_bytes > 4e8 else "; the whole input fits in L2 (stated, not flushed: the reference-sized workload is this small)"),
                          "cigar": f"CIGAR16 ({blk.cigar16.nbytes / 1e9:.3f} GB; the BAM words are {blk.cigar.nbytes / 1e9:.3f} GB)"},
               "clocks": clocks, "gpu_launches": int(launches), "reruns_in_timed_region": int(reruns),
               "e2e": {"value": e2e_val, "unit": "Gbp/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, "ms_per_step": float(et[0]) * 1e3,
                       "pinned": bool(pinned), "seq": "full arena" if args.e2e_full_seq else "on demand (slices requested by the device, gathered on the host)",
                       "bam32_in_ms": float(et[1]) * 1e3, "bam32_in_note": "one step fed BAM CIGAR words: snfb_load_records converts them to CIGAR16 on the host first"},
               "host_prep": {k: round(v, 3) for k, v in prep.items()},
               "roofline": roof, "rooflines": [roof_a, roof_c], "stage_ms": {k: v[0] / args.steps for k, v in kern.items()},
               "callset_sha256": digest}
        if committed:
            out["parity_vs_n1"] = {"identical": digest == committed["sha256"], "n1_candidates": committed.get("n_cand"), "this_run_candidates": int(n_all),
                                   "source": "tests/expected/callset_hashes.json (written by the 1-GPU run whose call set equals the oracle's)"}
        elif world > 1:
            out["parity_vs_n1"] = {"identical": None, "note": f"no committed N=1 hash for {key}"}
        if world == 1 and not args.no_cpu:
            info, _, _ = cpu_sample(blk, cfg, ccfg, ncores, target_bp=args.cpu_sample_gbp * 1e9)
            out["cpu_baseline"] = info
            if cpu_sample.whole_block:        # the oracle saw the whole block: compare it with the device run, candidate by candidate
                same = same_candidates(full, cpu_sample.last_result)
                out["parity_full_size"] = {"candidates": int(len(full.cand)), "alt_bytes": int(len(full.alt)), "identical_to_oracle": same}
                if same and args.write_hash:
                    hs = committed_hashes()
                    hs[key] = {"sha256": digest, "n_cand": int(len(full.cand)), "alt_bytes": int(len(full.alt))}
                    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
                    with open(os.path.join(ROOT, "gpurun_out", "callset_hashes.json"), "w") as f:
                        json.dump(hs, f, indent=1, sort_keys=True)
            out["cpu_baseline_python"] = python_reference_baseline()
        print(json.dumps(out))
    for a in pinned:
        L.snfb_unpin_host(C.c_void_p(a.ctypes.data))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------- config 4: population combine
def combine_workload(n_samples, scale, seed=1004):
    """Candidate-level synthetic population (BASELINE config 4): `n_samples` samples that share planted sites on 24 GRCh38-length contigs (one per
    120 kb), each sample carrying 80 % of them with jittered position / length, per-sample support and, for INS, its own noisy copy of the inserted
    sequence.  Served to CombineTask.plan through reader objects with the SNF reader's interface, so the chunks are formed by the product code."""
    import types
    from sniffles_b200 import synth
    rng = np.random.default_rng(seed)
    lens = [max(200000, int(x * scale)) for x in synth.GRCH38]
    bs, step = 100000, 500
    blocks = [dict() for _ in range(n_samples)]                      # per sample: (contig, block) -> block dict
    code = np.frombuffer(b"ACGT", np.uint8)
    for ci, clen in enumerate(lens):
        name = f"ctg{ci + 1}"
        nsite = max(1, clen // 120000)
        pos = np.sort(rng.integers(1000, clen - 1000, nsite))
        kind = rng.choice(5, nsite, p=[0.45, 0.45, 0.04, 0.03, 0.03])   # INS DEL DUP INV BND
        size = np.exp(rng.uniform(np.log(50), np.log(2000), nsite)).astype(np.int64)
        for si in range(nsite):
            t = ("INS", "DEL", "DUP", "INV", "BND")[kind[si]]
            base = code[rng.integers(0, 4, size[si])] if t == "INS" else None
            carriers = np.nonzero(rng.random(n_samples) < 0.8)[0]
            for sm in carriers:
                p_ = int(pos[si] + rng.integers(-6, 7)); ln = int(size[si] + rng.integers(-3, 4))
                if t == "INS":
                    sq = base.copy(); k = max(1, len(sq) // 50); sq[rng.integers(0, len(sq), k)] = code[rng.integers(0, 4, k)]
                    alt = sq.tobytes().decode()
                else:
                    alt = f"<{t}>"
                c = types.SimpleNamespace(svtype=t, pos=p_, svlen=-ln if t == "DEL" else (0 if t == "BND" else ln), support=int(rng.integers(3, 30)), alt=alt, bnd_info=None)
                if t == "BND":
                    c.bnd_info = types.SimpleNamespace(mate_contig=f"ctg{(ci + 3) % len(lens) + 1}", mate_ref_start=int(1000 + (pos[si] * 7) % 100000 + rng.integers(-5, 6)))
                b = (p_ // bs) * bs
                blk = blocks[sm].get((name, b))
                if blk is None:
                    blk = blocks[sm][(name, b)] = {"INS": [], "DEL": [], "DUP": [], "INV": [], "BND": [], "_COVERAGE": {b + i * step: 30 for i in range(bs // step)}}
                blk[t].append(c)

    class Reader:
        def __init__(self, d):
            self.d = d

        def read_blocks(self, contig, block_index):
            b = self.d.get((contig, block_index))
            return None if b is None else [b]

        def close(self):
            pass
    return lens, [Reader(d) for d in blocks]


def run_combine(args):
    """--config 4: the multi-sample grouping through snfb_combine_groups (host buffers in and out, so the timed call IS the end-to-end call)"""
    import torch
    from sniffles_b200 import binding, combine, config as sconfig
    sys.path.insert(0, ROOT)
    n_samples = 50
    t0 = time.time()
    lens, readers = combine_workload(n_samples, args.scale)
    cfg = sconfig.default_config(*(["--combine-pctseq", os.environ["SNFB_COMBINE_PCTSEQ"]] if "SNFB_COMBINE_PCTSEQ" in os.environ else []))
    cfg.mode = "combine"
    cfg.snf_input_info = [{"internal_id": k, "sample_id": f"S{k}", "filename": None} for k in range(n_samples)]
    cfg.sample_ids_vcf = [(k, f"S{k}") for k in range(n_samples)]
    rd = {k: r for k, r in enumerate(readers)}
    plan, tasks = combine.Plan(), []
    for ti, clen in enumerate(lens):
        task = combine.CombineTask(ti, f"ctg{ti + 1}", 0, clen - 1, cfg)
        task.plan(rd, plan, task_index=ti)
        tasks.append(task)
    arrays = combine.plan_arrays(plan, cfg)
    n = len(plan.cands)
    log(f"[bench] config 4: {n_samples} samples, {n} candidates, {len(plan.chains)} chains, {len(plan.chunks)} chunks, ALT arena {len(arrays['alt']) / 1e6:.1f} MB, built in {time.time() - t0:.1f}s")
    ctx = binding.Context(0)
    call = lambda: ctx.combine_groups(plan, cfg, arrays=arrays)
    for _ in range(max(args.warmup, 1)):
        out = call()
    sampler = ClockSampler(0); sampler.start()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    kern_ms = 0.0
    for _ in range(args.steps):
        out = call()
        kern_ms += max([ms for nm, ms, _ in ctx.timings() if nm == "combine_groups"] or [0.0])
    torch.cuda.synchronize()
    wall = time.perf_counter() - t1
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("cand_group", "emit_chunk", "emit_ord", "cov_non"), out)))
    ms_per_step = wall / args.steps * 1e3
    n_groups = int((out[1][:n] >= 0).sum())
    h2d = sum(int(arrays[k].nbytes) for k in ("chains", "chunks", "pos", "svlen", "sample", "mate_contig", "mate_pos", "block_start", "cov", "alt", "alt_off", "alt_len"))
    d2h = 12 * n + 4 * n * n_samples
    res = {"metric": "multi-sample combine: candidates grouped per second (BASELINE config 4; the Gbp/s metric does not apply to SNF inputs)", "value": n / (wall / args.steps), "unit": "candidates/s",
           "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64 / int32", "data": "synthetic",
           "config": {"workload": f"BASELINE config 4: {n_samples} samples x ~{n // n_samples} candidates on 24 GRCh38-length contigs x scale {args.scale}, --combine-pctseq {cfg.combine_pctseq} (edit distance on)",
                      "candidates": n, "groups": n_groups, "chains": len(plan.chains), "chunks": len(plan.chunks), "l2": "host-buffer call: inputs cross PCIe every step"},
           "clocks": clocks, "gpu_launches": int(args.steps), "kernel_ms_per_step": kern_ms / args.steps,
           "e2e": {"value": n / (wall / args.steps), "unit": "candidates/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "note": "snfb_combine_groups takes and returns host buffers: the timed call is the end-to-end call"},
           "roofline": {"bound": "latency", "kernel": "combine::k_combine", "note": "one warp per (contig, svtype) chain, sequential along the chain by construction (groups carry over): the longest chain is the step", "achieved": None, "peak": None, "unit": None, "frac": None, "traffic": None}}
    if not args.no_cpu:
        # CPU arm: the grouping restatement (oracle/combine.py, pinned against the reference's CombineTask) on a bounded sample: the chains of the smallest contigs
        from oracle import combine as ocombine
        order = sorted(range(len(lens)), key=lambda i: lens[i])
        sub, tot = combine.Plan(), 0
        for ti in order:
            tasks[ti].plan(rd, sub, task_index=ti)
            tot = len(sub.cands)
            if tot >= 8000:
                break
        sa = combine.plan_arrays(sub, cfg)
        t2 = time.perf_counter()
        ref = ocombine.combine_groups(sa, cfg)
        dt = time.perf_counter() - t2
        dev = ctx.combine_groups(sub, cfg, arrays=sa)
        m = len(sub.cands)
        res["cpu_baseline"] = {"value": m / dt, "unit": "candidates/s", "cores": 1, "kind": "port", "sample": f"{m} candidates (the smallest contigs), oracle/combine.py (pure Python + numpy edit distance; the reference itself calls edlib, C code that is absent here) in {dt:.1f}s",
                               "identical_to_device": bool(np.array_equal(ref[0][:m], dev[0][:m]) and np.array_equal(ref[1][:m], dev[1][:m]))}
    print(json.dumps(res))
    ctx.close()


_INGEST_ZB, _INGEST_BLOCKS = b"", []


def _ingest_inflate_slice(arg):
    """CPU arm of --config 6: one worker inflates every nthr-th BGZF block of the file (zlib, raw DEFLATE) and returns the bytes produced"""
    import zlib
    k, n = arg
    zb, tot = _INGEST_ZB, 0
    for off, ln in _INGEST_BLOCKS[k::n]:
        tot += len(zlib.decompress(zb[off:off + ln], -15))
    return tot


def run_ingest(args):
    """--config 6 (SURVEY 8 (f)3, not a BASELINE config): compressed BAM bytes -> the packed record block, on the device (snfb_load_bam).
    Workload: a coordinate-sorted BAM written from the config-2 generator (noisy base qualities, so the DEFLATE streams look like a real
    file's), its blocks tiled `--ingest-tiles` times as independent tasks.  value = inflated BAM bytes per second of the ingest kernels
    (CUDA events); e2e = the whole snfb_load_bam call from pinned host memory, plus the full path (ingest + lead -> cluster -> consensus)."""
    import tempfile
    import torch
    from sniffles_b200 import abi, bamio, binding, synth, config as sconfig
    t0 = time.time()
    lens = [int(1_500_000 * args.scale)] * 4
    blk = synth.generate(606, lens, 30.0, len_mean=15000.0, len_sd=6000.0, sv_spacing=8000.0, phased_frac=0.3, tr_frac=0.2)
    tmp = tempfile.mkdtemp(prefix="snfb_ingest_")
    path = os.path.join(tmp, "bench.bam")
    bamio.write_bam(path, blk, level=int(os.environ.get("SNFB_BAM_LEVEL", "6")), qual_seed=7)
    f = bamio.BamFile(path)
    regions = [(n, 0, f.get_reference_length(n)) for n in blk.contig_names]
    bgzf1, spans1 = f.device_input(regions)
    # CPU arm first, in forked workers, BEFORE this process touches CUDA or pins memory (forking a process that holds a CUDA context and
    # gigabytes of page-locked memory took the box down twice)
    cpu_arm = None
    if not args.no_cpu:
        import multiprocessing as mp
        zb = bgzf1.tobytes()
        blocks = []
        o = 0
        while o < len(zb):
            xlen = zb[o + 10] | (zb[o + 11] << 8); bs = (zb[o + 16] | (zb[o + 17] << 8)) + 1
            blocks.append((o + 12 + xlen, bs - 12 - xlen - 8)); o += bs
        nthr = min(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1), 64)
        global _INGEST_ZB, _INGEST_BLOCKS
        _INGEST_ZB, _INGEST_BLOCKS = zb, blocks
        with mp.get_context("fork").Pool(nthr) as pool:
            one = sum(pool.map(_ingest_inflate_slice, [(k, nthr) for k in range(nthr)]))          # warm the workers; the file's inflated size
            reps = max(1, min(64, int(16e9 // max(1, one))))
            t2 = time.perf_counter()
            tot = sum(pool.map(_ingest_inflate_slice, [(k % nthr, nthr) for k in range(nthr * reps)], chunksize=1))
            dt = time.perf_counter() - t2
        _INGEST_ZB, _INGEST_BLOCKS = b"", []
        cpu_arm = {"value": tot / dt / 1e9, "unit": "GB/s", "cores": nthr, "kind": "port",
                   "sample": f"zlib inflate (the C library htslib calls behind bam.fetch), {nthr} forked worker processes, {len(blocks) * reps} BGZF blocks = {tot / 1e9:.2f} GB inflated in {dt:.1f}s; "
                             "inflate only: htslib's record decode and pysam's accessors come on top in the reference"}
        log(f"[bench] config 6 CPU arm: {cpu_arm['value']:.2f} GB/s on {nthr} processes")
    tiles = max(1, args.ingest_tiles)
    bgzf = np.tile(bgzf1, tiles)
    spans = np.tile(spans1, tiles)
    nt1 = len(regions)
    for k in range(tiles):
        sl = slice(k * len(spans1), (k + 1) * len(spans1))
        spans["cbeg"][sl] += k * len(bgzf1); spans["cend"][sl] += k * len(bgzf1); spans["task"][sl] += k * nt1
    tables = bamio.pack_records(f.contigs, [], [(t % nt1, 0, regions[t % nt1][2], t) for t in range(nt1 * tiles)])
    binding.lib().snfb_pin_host(bgzf.ctypes.data, bgzf.nbytes)
    log(f"[bench] config 6: BAM of {len(blk.rec)} records written in {time.time() - t0:.1f}s, x{tiles} tiles = {bgzf.nbytes / 1e9:.3f} GB of BGZF, {len(spans)} spans, {nt1 * tiles} tasks")
    cfg = sconfig.default_config()
    ctx = binding.Context(0)
    ctx.set_config(abi.Config.from_sniffles(cfg))
    for _ in range(max(args.warmup, 1)):
        z = ctx.load_bam(bgzf, spans, tables)
    raw_bytes, n_rec = z["raw_bytes"], z["n_rec"]
    assert n_rec == tiles * len(blk.rec), (n_rec, len(blk.rec))
    sampler = ClockSampler(0); sampler.start()
    stage, wall = {}, 0.0
    for _ in range(args.steps):
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        ctx.load_bam(bgzf, spans, tables)
        wall += time.perf_counter() - t1
        for nm, ms, _b in ctx.timings():
            stage[nm] = stage.get(nm, 0.0) + ms / args.steps
    clocks = sampler.stop()
    if args.dump_outputs:           # the record block the last load built in device memory
        dump_outputs(args.dump_outputs, dict(zip(("rec", "cigar16", "var", "seq"), ctx.ingest_fetch())))
    kern_ms = sum(stage.get(k, 0.0) for k in ("inflate", "walk_records", "parse_records", "record_sizes", "pack_records"))
    e2e_ms = wall / args.steps * 1e3
    # the whole path fed compressed bytes: ingest + stages A-C, candidates back on the host
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    ctx.load_bam(bgzf, spans, tables)
    res_run = ctx.run(want_leads=False)
    path_ms = (time.perf_counter() - t1) * 1e3
    peak, peak_src = measured_peak()
    inf_bytes = bgzf.nbytes + raw_bytes
    res = {"metric": "BAM ingest on the device: inflated BAM bytes per second, BGZF bytes -> packed record block (SURVEY 8 (f)3; not a BASELINE config)", "value": raw_bytes / (kern_ms * 1e-3) / 1e9, "unit": "GB/s",
           "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": kern_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
           "config": {"workload": f"coordinate-sorted BAM from the config-2 generator (4 contigs x {lens[0]} bp, 30x ONT, noisy qualities, zlib level {os.environ.get('SNFB_BAM_LEVEL', '6')}) x {tiles} tiles",
                      "records": n_rec, "bgzf_bytes": int(bgzf.nbytes), "inflated_bytes": int(raw_bytes), "bgzf_blocks": z["n_blocks"], "spans": len(spans), "l2": f"inputs {bgzf.nbytes / 1e9:.2f} GB + {raw_bytes / 1e9:.2f} GB inflated vs 126 MB L2"},
           "clocks": clocks, "gpu_launches": int(ctx.launch_count()), "stage_ms": stage,
           "e2e": {"value": raw_bytes / (e2e_ms * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(bgzf.nbytes), "d2h_bytes_per_step": 256, "pinned": True,
                   "bam_to_candidates_ms": path_ms, "candidates": int(len(res_run.cand))},
           "roofline": {"bound": "hbm", "kernel": "ingest::k_inflate", "achieved": inf_bytes / (stage.get("inflate", 1e9) * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": inf_bytes / (stage.get("inflate", 1e9) * 1e-3) / 1e9 / peak, "peak_source": peak_src, "algorithmic_bytes_per_launch": int(inf_bytes), "kernel_ms": stage.get("inflate"), "traffic": None,
                        "note": "compressed bytes read + inflated bytes written; a Huffman decode is a serial bit-dependent chain per block, so the bound in practice is instruction latency x resident warps, not HBM"}}
    if cpu_arm is not None:
        res["cpu_baseline"] = cpu_arm
    print(json.dumps(res))
    ctx.close()
    f.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=int(os.environ.get("SNFB_BENCH_CONFIG", "2")), help="BASELINE.json config index: 1, 2 (default: 30x ONT WGS), 3 (60x HiFi --mosaic), 4 (50-sample combine; its own metric), 5 (INS-heavy); 6 = device BAM ingest (SURVEY 8 (f)3, not a BASELINE config)")
    ap.add_argument("--scale", type=float, default=float(os.environ.get("SNFB_BENCH_SCALE", "1.0")), help="contig length multiplier (1.0 = the named size)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--cpu-sample-gbp", type=float, default=1000.0, help="sequenced Gbp of the CPU arm's sample (smallest contigs first); the default takes every contig: one host thread per contig, the reference's own grain")
    ap.add_argument("--ingest-tiles", type=int, default=8, help="--config 6: how many times the BAM's blocks are tiled (independent tasks)")
    ap.add_argument("--no-pin", action="store_true")
    ap.add_argument("--e2e-full-seq", action="store_true", help="e2e: copy the whole seq arena every step instead of the on-demand slices")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--write-hash", action="store_true", help="1 GPU: when the call set equals the oracle's, write its hash to gpurun_out/callset_hashes.json (to be committed under tests/expected/)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the arrays the timed path returned in its last step as DIR/<name>.npy "
                    "(float32 / float64, at most 64 MB: larger outputs are sampled with a fixed seed), to compare two builds on identical inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "b200":
        log("[bench] note: timing rules ask for >= 3 warm-up steps")
    import __graft_entry__ as g
    if int(os.environ.get("RANK", "0")) == 0:
        g.build()
    elif args.impl == "b200":
        time.sleep(2.0)         # let rank 0 check/refresh the in-tree libraries first
    if args.config == 6:
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "config 6 (device BAM ingest) is not a BASELINE config; its CPU arm is the cpu_baseline of `bench.py --config 6`"}))
        else:
            run_ingest(args)
    elif args.config == 4:
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "config 4 has no Gbp/s metric; its CPU arm is the cpu_baseline of `bench.py --config 4`"}))
        else:
            run_combine(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
