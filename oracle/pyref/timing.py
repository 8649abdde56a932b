"""Times the UNMODIFIED reference (build_leadtab + call_candidates + finalize_candidates, parallel.py:90-201) on seeded
synthetic blocks, htslib decode excluded (the reads are materialised before the clock starts) — the committed measurement
bench.py reports as `cpu_baseline_python` (BASELINE.md §3).  TEST / BASELINE INFRASTRUCTURE: runs only where the reference
tree exists (harness.REFERENCE_SRC).

    python oracle/pyref/timing.py --write          # refresh tests/expected/python_reference_timing.json (build container)
"""
import json
import logging
import multiprocessing as mp
import os
import platform
import sys
import time

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(_HERE))
sys.path[:0] = [ROOT, _HERE]
OUT = os.path.join(ROOT, "tests", "expected", "python_reference_timing.json")


def available():
    import harness
    return os.path.isdir(harness.REFERENCE_SRC)


def _time_task(args):
    """one reference task on pre-built reads; returns (seconds, aligned bp passing the filters, candidates)"""
    kw, t, cli = args
    logging.disable(logging.CRITICAL)
    import harness
    from sniffles_b200 import synth
    kw = dict(kw)
    blk = synth.generate(kw.pop("seed"), kw.pop("contig_len"), kw.pop("coverage"), **kw)
    harness.import_reference()
    from sniffles import leadprov, parallel
    from sniffles.region import Region
    config = harness.make_config(*cli)
    if not hasattr(config, "mode"):
        config.mode = "call_sample"
    task = blk.task[t]
    contig = blk.contig_names[int(task["contig"])]
    bam = harness.DuckBam(blk, t)
    reads = [harness.DuckRead(blk, int(i)) for i in bam.idx]            # "decode": excluded on both sides
    for r in reads:
        r.query_sequence
    bam.fetch = lambda contig, start, end, until_eof=False: (r for r in reads if r.reference_start < end and r.reference_end > start)
    tr = None
    if int(task["tr_n"]) > 0:
        o, n = int(task["tr_off"]), int(task["tr_n"])
        tr = [(int(blk.tr[2 * (o + k)]), int(blk.tr[2 * (o + k) + 1])) for k in range(n)]
    tk = parallel.CallTask(id=int(task["task_id"]), sv_id=0, contig=contig, start=int(task["start"]), end=int(task["end"]), config=config, tandem_repeats=tr)
    config.task_read_id_offset_mult = 10 ** 9
    abp = sum(r.query_alignment_length for r in reads if not (r.mapping_quality < config.mapq or r.is_secondary or r.query_alignment_length < config.min_alignment_length))
    t0 = time.perf_counter()
    tk.lead_provider = leadprov.LeadProvider(config, tk.id * config.task_read_id_offset_mult, contig)
    tk.lead_provider.build_leadtab([Region(contig, tk.start, tk.end)], bam)
    qc = not (config.snf is not None or config.no_qc)
    cands = tk.call_candidates(qc, config)
    final = tk.finalize_candidates(cands, not qc, config)
    dt = time.perf_counter() - t0
    return dt, int(abp), len(final)


SHAPES = {
    # BASELINE config 1 exactly (one 1 Mb contig, ~200 ONT reads of ~100 kb): --threads 1
    "config1": (dict(seed=1001, contig_len=[1_000_000], coverage=20.0, len_model=0, len_mean=100000.0, len_sd=10000.0, len_min=1000, len_max=200000,
                     tech="ont", sv_spacing=25000.0), []),
    # BASELINE config 2's shape on eight small contigs: one process per contig over the host cores (the reference's own grain)
    "config2_small": (dict(seed=1002, contig_len=[400_000] * 8, coverage=30.0, len_model=1, len_mean=15000.0, len_sd=600.0, len_min=1000, len_max=200000,
                           tech="ont"), []),
}


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return platform.processor() or "unknown"


def measure(nproc=None):
    nproc = nproc or os.cpu_count() or 1
    out = dict(python=platform.python_version(), numpy=np.__version__, cpu=cpu_model(), nproc=nproc, decode="excluded (reads materialised before the clock starts)",
               functions="LeadProvider.build_leadtab + Task.call_candidates + Task.finalize_candidates (parallel.py:90-201), unmodified reference")
    kw, cli = SHAPES["config1"]
    dt, abp, nc = _time_task((kw, 0, cli))
    out["config1_threads1"] = dict(seconds=dt, aligned_bp=abp, gbp_per_s=abp / dt / 1e9, calls=nc, processes=1)
    kw, cli = SHAPES["config2_small"]
    n = len(kw["contig_len"])
    with mp.get_context("spawn").Pool(min(nproc, n)) as pool:
        t0 = time.perf_counter()
        rs = pool.map(_time_task, [(kw, t, cli) for t in range(n)])
        wall = time.perf_counter() - t0
    abp = sum(r[1] for r in rs)
    out["config2_small_pool"] = dict(wall_seconds=wall, sum_task_seconds=sum(r[0] for r in rs), aligned_bp=abp, gbp_per_s_wall=abp / wall / 1e9,
                                     gbp_per_s_per_core=abp / sum(r[0] for r in rs) / 1e9, processes=min(nproc, n), calls=sum(r[2] for r in rs),
                                     note="wall includes block generation and read materialisation in every worker; per-core figure uses the timed region only")
    return out


if __name__ == "__main__":
    if not available():
        raise SystemExit("reference tree not found")
    res = measure()
    print(json.dumps(res, indent=1))
    if "--write" in sys.argv:
        res["where"] = "build container (no GPU)"
        with open(OUT, "w") as f:
            json.dump(res, f, indent=1)
