#!/usr/bin/env python3
"""Throughput of the BAM ingest path on one GPU: N config-2 reads -> BAM (zlib level L, binned qualities) in pinned host
memory -> pssgpu_feed_bam, against the same reads as SAM text through pssgpu_feed.  Prints one JSON line."""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import torch
    from pss_testlib import Synth, reads_cfg_config2
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=4_000_000)
    ap.add_argument("--level", type=int, default=6)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--genome-mb", type=int, default=200)
    ap.add_argument("--group", type=int, default=0, help="also feed the BAM to a group of this many GPUs (pssgpu_group_feed_bam)")
    ap.add_argument("--chunk-mb", type=int, default=0, help="feed the BAM in pieces of this size (0: one call)")
    ap.add_argument("--batch-mbs", default="", help="comma list: also time the one-GPU BAM path with these $PSSGPU_BAM_BATCH_MB values")
    a = ap.parse_args()
    Synth.set_threads(os.cpu_count() or 1)
    g = Synth.genome(35, [a.genome_mb * 600_000, a.genome_mb * 400_000], n_frac=0.01, lower_frac=0.03)
    cfg = reads_cfg_config2(seed=10)
    cap = Synth.sam_bound(cfg, 0, a.reads)
    host = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
    nb = Synth.sam_into(cfg, g, 0, a.reads, host.data_ptr(), cap)
    bcap = Synth.lib().synth_bam_bound(nb, 3)
    hbam = torch.empty(bcap, dtype=torch.uint8, pin_memory=True)
    t0 = time.perf_counter()
    nbam = Synth.bam_into(host.data_ptr(), nb, list(zip(g.names, g.lens)) + [("chrUn_synthetic_decoy", 1000)], hbam.data_ptr(), bcap,
                          level=a.level, qual_mode=1)
    t_conv = time.perf_counter() - t0
    pkg = importlib.import_module("pss-bam_b200")
    ctx = pkg.Context(0)
    ctx.upload_genome(list(zip(g.names, g.seqs)))

    def run(fn):
        best = None
        for _ in range(a.reps):
            ctx.pss_begin(pkg.PssOptions())
            ctx.timing_reset(True)
            t0 = time.perf_counter()
            fn()
            f, r = ctx.pss_finish()
            dt = time.perf_counter() - t0
            tm = ctx.timing()
            if best is None or dt < best[0]:
                best = (dt, tm, f, r)
        return best
    sam_t, sam_tm, sf, sr = run(lambda: ctx.feed_ptr(host.data_ptr(), nb, last=True))
    bam_t, bam_tm, bf, br = run(lambda: ctx.feed_bam_ptr(hbam.data_ptr(), nbam, last=True))
    info = ctx.bam_info()
    out = {"reads": a.reads, "sam_bytes": int(nb), "bam_bytes": int(nbam), "zlib_level": a.level, "bam_conversion_s": t_conv,
           "tables_equal": bool(np.array_equal(sf, bf) and np.array_equal(sr, br)),
           "sam_text": {"s": sam_t, "reads_per_s": a.reads / sam_t, "gb_per_s": nb / sam_t / 1e9, "kernel_ms": sam_tm["kernel_ms"]},
           "bam": {"s": bam_t, "reads_per_s": a.reads / bam_t, "compressed_gb_per_s": nbam / bam_t / 1e9,
                   "kernel_ms_inflate_render_tally": bam_tm["kernel_ms"], "launches": bam_tm["launches"], "info": info}}
    ctx.close()
    for mb in [int(x) for x in a.batch_mbs.split(",") if x]:
        os.environ["PSSGPU_BAM_BATCH_MB"] = str(mb)            # read when a context first ingests BAM
        ctx = pkg.Context(0)
        ctx.upload_genome(list(zip(g.names, g.seqs)))
        t, tm, f2, r2 = run(lambda: ctx.feed_bam_ptr(hbam.data_ptr(), nbam, last=True))
        out.setdefault("batch_mb", {})[str(mb)] = {"s": t, "reads_per_s": a.reads / t, "kernel_ms": tm["kernel_ms"], "batches": ctx.bam_info()["batches"],
                                                   "tables_equal": bool(np.array_equal(sf, f2) and np.array_equal(sr, r2))}
        ctx.close()
        del os.environ["PSSGPU_BAM_BATCH_MB"]
    if a.group > 1:
        grp = pkg.Group(list(range(a.group)))
        grp.upload_genome(list(zip(g.names, g.seqs)))
        step = (a.chunk_mb << 20) or nbam

        def feed_group():
            for off in range(0, nbam, step):
                grp.feed_bam_ptr(hbam.data_ptr() + off, min(step, nbam - off), last=False)
            grp.feed_bam_ptr(hbam.data_ptr(), 0, last=True)
        best = None
        for _ in range(a.reps):
            grp.pss_begin(pkg.PssOptions())
            t0 = time.perf_counter()
            feed_group()
            f, r = grp.pss_finish()
            dt = time.perf_counter() - t0
            if best is None or dt < best:
                best = dt
        out["bam_group"] = {"gpus": a.group, "s": best, "reads_per_s": a.reads / best, "compressed_gb_per_s": nbam / best / 1e9,
                            "speedup_vs_one_gpu": bam_t / best, "tables_equal": bool(np.array_equal(sf, f) and np.array_equal(sr, r)),
                            "chunk_mb": a.chunk_mb, "info": grp.bam_info(), "reduce": grp.reduce_backend}
        grp.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
