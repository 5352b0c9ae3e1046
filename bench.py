#!/usr/bin/env python3
"""bench.py -- pss-bam PSS tally throughput on B200 (contract: one JSON line on stdout from rank 0).

Workload (BASELINE.json configs[1]): synthetic 3.1 Gb human-scale genome (24 contigs, ~1 % N runs, soft-masked
stretches) + 200 M variable-length (30-150 bp) reads with indel / soft-clip CIGARs, filtered flags, paired records,
QUAL '*', unknown contigs and MD/NM tags, read-sharded over 8 GPUs: every GPU holds a full packed genome replica and
tallies its 25 M-read shard (weak scaling: the per-GPU shard is fixed, N GPUs process N x 25 M reads).

A step = one pass of the hot path over the rank's shard:
    pssgpu_pss_begin -> pssgpu_feed_device (SAM text resident in HBM) -> pssgpu_pss_finish_device
    [-> NCCL all-reduce of the 2x17x16 u64 count tables when N > 1] -> tables to the host.
`value` = reads of all ranks / max-over-ranks device time (CUDA events on the library's stream).
`e2e`   = same metric through the C ABI with HOST (pinned) SAM text: pssgpu_feed copies it to the device inside the
          timed region, tables come back to the host.
`roofline` = algorithmic bytes of the tally kernel / its CUDA-event duration, against the measured HBM copy peak.
`cpu_baseline` = the unmodified reference binary (oracle/_ref/pss-bam, stock -O0 flags) on a bounded sample.

    python bench.py                      # 1 GPU
    torchrun --nproc-per-node 8 bench.py --gpus 8
    python bench.py --impl reference     # the reference's CPU path on this box's host cores
    python bench.py --dump-outputs DIR   # also write the last timed step's tables to DIR/*.npy (compare two builds)
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HUMAN_CONTIGS = [  # hs37-like lengths, 3.096 Gb in total, every contig < 536 870 911 (fasta-genome-io.h:9)
    ("chr1", 249250621), ("chr2", 243199373), ("chr3", 198022430), ("chr4", 191154276), ("chr5", 180915260),
    ("chr6", 171115067), ("chr7", 159138663), ("chr8", 146364022), ("chr9", 141213431), ("chr10", 135534747),
    ("chr11", 135006516), ("chr12", 133851895), ("chr13", 115169878), ("chr14", 107349540), ("chr15", 102531392),
    ("chr16", 90354753), ("chr17", 81195210), ("chr18", 78077248), ("chr19", 59128983), ("chr20", 63025520),
    ("chr21", 48129895), ("chr22", 51304566), ("chrX", 155270560), ("chrY", 59373566),
]
GENOME_SEED = 31
READS_SEED = 2002
METRIC = "aligned reads/s (PSS tally)"
UNIT = "reads/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads-per-gpu", type=int, default=25_000_000, help="200 M reads / 8 GPUs")
    ap.add_argument("--genome-scale", type=float, default=1.0, help="shrink the 3.1 Gb genome (developer runs only)")
    ap.add_argument("--cpu-sample-reads", type=int, default=1_500_000)
    ap.add_argument("--cpu-genome-mb", type=int, default=100)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the oracle check of the benchmarked shard's tables")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --reads-per-gpu on every GPU (the default; 8 GPUs = the 200 M reads of configs[1]); "
                         "strong: the 8 x --reads-per-gpu reads of configs[1] split over the GPUs in use")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned to DIR/pss_fwd.npy, pss_rev.npy, pss_stats.npy (float64)")
    return ap.parse_args()


def dump_outputs(d, tables, stats, R):
    """The last timed step's result as float64 arrays (exact: every count is far below 2**53).  pss_fwd / pss_rev are
    the (R+2) x 16 count tables pssgpu_pss_finish_device wrote (all-reduced when N > 1); pss_stats holds rank 0's
    outcome counters lines, counted, no_contig, filtered, parse_fail, undefined.  The inputs are seeded, so two builds
    run with the same arguments can be compared array for array."""
    os.makedirs(d, exist_ok=True)
    t = tables.numpy().astype(np.float64).reshape(2, R + 2, 16)
    np.save(os.path.join(d, "pss_fwd.npy"), t[0])
    np.save(os.path.join(d, "pss_rev.npy"), t[1])
    keys = ("lines", "counted", "no_contig", "filtered", "parse_fail", "undefined")
    np.save(os.path.join(d, "pss_stats.npy"), np.array([stats[k] for k in keys], dtype=np.float64))


def contig_plan(scale):
    return [(n, max(1000, int(l * scale))) for n, l in HUMAN_CONTIGS]


def reads_per_rank(a, world):
    return a.reads_per_gpu if a.scaling == "weak" else (8 * a.reads_per_gpu) // max(1, world)


def workload_name(a, world=1):
    if a.scaling == "weak":
        s = "configs[1] shard: 3.1 Gb synthetic genome replica + %d of the 200 M variable-length (30-150 bp) reads " \
            "(200 M / 8 GPUs, read-sharded)" % a.reads_per_gpu
    else:
        s = "configs[1] whole: 3.1 Gb synthetic genome replica per GPU + all %d variable-length (30-150 bp) reads split " \
            "over %d GPU(s), %d each" % (8 * a.reads_per_gpu, world, reads_per_rank(a, world))
    if a.genome_scale != 1.0:
        s += " [genome scaled x%g]" % a.genome_scale
    return s


def reference_workload_name(a, cores, per):
    """What --impl reference really runs (BASELINE.md "Scale": a bounded prefix, extrapolated linearly)."""
    return ("EXTRAPOLATED, reduced config: the unmodified reference program on configs[1]-distributed reads (same generator, "
            "same seed, same reject mix, 30-150 bp), %d reads per process x %d single-threaded processes, against a %d Mb "
            "4-contig genome instead of the 3.1 Gb one (its FASTA loader needs ~150 s per process for 3.1 Gb; load time is "
            "measured with an empty SAM and subtracted); reads/s is per-read streaming cost (pss-bam.c:764-783), linear in reads; "
            "a one-off run on the full 3.1 Gb genome with >= 10 M reads is in profiles/r2_reference_fullscale.json"
            % (per, cores, a.cpu_genome_mb))


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if not self.p:
            return None
        time.sleep(0.15)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            return None
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- reference arm
def ref_paths():
    d = os.path.join(ROOT, "oracle", "_ref")
    return d, os.path.join(d, "pss-bam"), os.path.join(d, "samtools")


def _port_worker(args):
    """One process of the oracle-port baseline: tally one shard with oracle/liboracle.so (checker code, timed here only
    because the contract asks for a CPU baseline when the reference binary is not available)."""
    fasta_path, sam_path = args
    from pss_testlib import Oracle, PssParams
    ora = Oracle(fasta_path=fasta_path)
    with open(sam_path, "rb") as f:
        sam = f.read()
    t0 = time.perf_counter()
    ora.pss(sam, PssParams())
    dt = time.perf_counter() - t0
    ora.close()
    return dt


class ReferenceSample:
    """The unmodified reference binary on a bounded sample: `n_proc` single-threaded processes in parallel (the
    reference has no threads), each on its own shard of config-2 reads against a `genome_mb` Mb genome.  Files are
    written once; every run() times one pass; the FASTA load time (same concurrency, empty SAM) is measured once
    and subtracted, because the B200 arm also starts its clock with the genome resident."""

    def __init__(self, n_proc, reads_per_proc, genome_mb, seed):
        from pss_testlib import Synth, reads_cfg_config2
        d, exe, shim = ref_paths()
        # "reference": the unmodified binary (make -C oracle ref); "port": the oracle restatement, used only
        # when that binary did not travel to this box
        self.kind = "reference" if (os.path.exists(exe) and os.path.exists(shim)) else "port"
        self.exe, self.n_proc, self.reads = exe, n_proc, n_proc * reads_per_proc
        nc = 4
        g = Synth.genome(GENOME_SEED + 1, [genome_mb * 1_000_000 // nc] * nc, n_frac=0.01, lower_frac=0.03)
        self.work = tempfile.mkdtemp(prefix="pssbench_ref_")
        with open(os.path.join(self.work, "genome.fa"), "wb") as f:
            f.write(g.fasta_bytes())
        cfg = reads_cfg_config2(seed=seed)
        for p in range(n_proc):
            with open(os.path.join(self.work, f"shard{p}.sam"), "wb") as f:
                f.write(Synth.sam(cfg, g, p * reads_per_proc, (p + 1) * reads_per_proc))
        open(os.path.join(self.work, "empty.sam"), "wb").close()
        self.env = dict(os.environ)
        self.env["PATH"] = d + os.pathsep + self.env.get("PATH", "")
        self.load = min(self._run(["empty.sam"] * n_proc) for _ in range(2)) if self.kind == "reference" else 0.0

    def _run(self, sams):
        if self.kind == "port":                                  # tally time only, measured inside each process
            import multiprocessing as mp
            with mp.get_context("spawn").Pool(self.n_proc) as pool:
                return max(pool.map(_port_worker, [(os.path.join(self.work, "genome.fa"), os.path.join(self.work, s)) for s in sams]))
        t0 = time.perf_counter()
        ps = [subprocess.Popen([self.exe, "-F", "genome.fa", "-B", s, "-o", f"out{i}"], cwd=self.work, env=self.env,
                               stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL) for i, s in enumerate(sams)]
        for p in ps:
            if p.wait() != 0:
                raise RuntimeError("reference pss-bam failed")
        return time.perf_counter() - t0

    def run(self):
        """-> (reads per second, tally seconds) of one pass over all shards."""
        total = self._run([f"shard{p}.sam" for p in range(self.n_proc)])
        tally = max(total - self.load, 1e-9)
        return self.reads / tally, tally

    def close(self):
        shutil.rmtree(self.work, ignore_errors=True)


def main_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from pss_testlib import Synth
    cores = os.cpu_count() or 1
    Synth.set_threads(cores)                                  # torchrun exports OMP_NUM_THREADS=1
    # bounded: about 1 s of tally per step on every core, so that any --steps/--warmup ends within minutes
    per = max(20_000, min(a.cpu_sample_reads // 4, 400_000))
    line = {"impl": "reference", "metric": METRIC, "unit": UNIT, "higher_is_better": True, "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "scaling": a.scaling, "vs_baseline": None, "dtype": "u64",
            "data": "synthetic", "config": {"workload": reference_workload_name(a, cores, per), "extrapolated": True,
                                            "b200_arm_workload": workload_name(a, a.gpus), "reads_per_process": per,
                                            "processes": cores, "genome_mb": a.cpu_genome_mb},
            "gpu_launches": 0}
    ref = None
    try:
        ref = ReferenceSample(cores, per, a.cpu_genome_mb, READS_SEED)
        for _ in range(a.warmup):
            ref.run()
        t0 = time.perf_counter()
        runs = [ref.run() for _ in range(a.steps)]
        value = statistics.mean(v for v, _ in runs)
        what = ("unmodified reference oracle/_ref/pss-bam (stock Makefile flags -gdwarf-2 -g, no -O)" if ref.kind == "reference"
                else "oracle port oracle/liboracle.so (-O2; oracle/_ref was not found on this box)")
        sample = (f"{what}, {cores} single-threaded processes in parallel, {per} config-2 reads each on a "
                  f"{a.cpu_genome_mb} Mb 4-contig genome; FASTA load time ({ref.load:.2f} s at the same concurrency, "
                  f"empty SAM) subtracted from every step")
        line.update({"value": value, "ms_per_step": 1e3 * statistics.mean(t for _, t in runs),
                     "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": ref.kind, "sample": sample},
                     "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     "wall_s": time.perf_counter() - t0})
    except Exception as ex:
        line.update({"unavailable": f"{type(ex).__name__}: {ex}"})
    finally:
        if ref:
            ref.close()
    print(json.dumps(line), flush=True)


def config0_case(pkg, device, torch, with_reference):
    """BASELINE.json configs[0], the case the reference runs as is: 10 Mb genome (4 x 2.5 Mb), 1 M unpaired 50-bp reads
    with 5' C->T / 3' G->A damage.  Whole-program view on both sides: genome made resident + tally + tables, against the
    unmodified reference binary on one core (it has no threads) -- with its FASTA load also given separately."""
    from pss_testlib import Synth, reads_cfg_config1
    g = Synth.genome(GENOME_SEED + 2, [2_500_000] * 4, n_frac=0.01, lower_frac=0.03)
    n = 1_000_000
    cfg = reads_cfg_config1(seed=READS_SEED + 1)
    cap = Synth.sam_bound(cfg, 0, n)
    host = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
    nb = Synth.sam_into(cfg, g, 0, n, host.data_ptr(), cap)
    out = {"reads": n, "sam_bytes": int(nb), "genome_bases": 10_000_000}
    c2 = pkg.Context(device)
    try:
        best = {}
        for _ in range(3):
            t0 = time.perf_counter()
            c2.upload_genome(list(zip(g.names, g.seqs)))
            t1 = time.perf_counter()
            c2.pss_begin(pkg.PssOptions())
            c2.timing_reset(True)
            c2.feed_ptr(host.data_ptr(), nb, last=True)
            fwd, rev = c2.pss_finish()
            t2 = time.perf_counter()
            cur = {"gpu_genome_upload_ms": (t1 - t0) * 1e3, "gpu_tally_from_host_ms": (t2 - t1) * 1e3,
                   "gpu_kernel_ms": c2.timing()["kernel_ms"]}
            if not best or cur["gpu_tally_from_host_ms"] < best["gpu_tally_from_host_ms"]:
                best = cur
        out.update(best)
        out["gpu_reads_per_s_from_host"] = n / (best["gpu_tally_from_host_ms"] * 1e-3)
        out["counted"] = c2.stats()["counted"]
    finally:
        c2.close()
    d, exe, shim = ref_paths()
    if with_reference and os.path.exists(exe) and os.path.exists(shim):
        work = tempfile.mkdtemp(prefix="pssbench_cfg0_")
        try:
            with open(os.path.join(work, "genome.fa"), "wb") as f:
                f.write(g.fasta_bytes())
            with open(os.path.join(work, "reads.sam"), "wb") as f:
                f.write(bytes(host[:nb].numpy()))
            open(os.path.join(work, "empty.sam"), "wb").close()
            env = dict(os.environ)
            env["PATH"] = d + os.pathsep + env.get("PATH", "")
            def run(sam):
                t0 = time.perf_counter()
                subprocess.run([exe, "-F", "genome.fa", "-B", sam, "-o", "out"], cwd=work, env=env, check=True,
                               stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                return time.perf_counter() - t0
            load = run("empty.sam")
            total = run("reads.sam")
            out.update({"reference_1core_total_s": total, "reference_1core_fasta_load_s": load,
                        "reference_reads_per_s": n / max(total - load, 1e-9)})
        finally:
            shutil.rmtree(work, ignore_errors=True)
    return out


# ----------------------------------------------------------------------------------------------- B200 arm
def main_b200(a):
    import torch
    import torch.distributed as dist
    from pss_testlib import Synth, reads_cfg_config2

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line: anything libraries print there (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world != a.gpus:
        if world == 1 and a.gpus > 1:
            raise SystemExit("launch with: python -m torch.distributed.run --nproc-per-node %d bench.py --gpus %d" % (a.gpus, a.gpus))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    try:                                                     # host threads and pinned buffers next to this rank's GPU
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
    except Exception:
        pass
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cores = os.cpu_count() or 1
    try:
        mine = len(os.sched_getaffinity(0))
    except Exception:
        mine = cores
    Synth.set_threads(max(1, min(mine, cores // max(1, world))))   # torchrun exports OMP_NUM_THREADS=1

    pkg = importlib.import_module("pss-bam_b200")
    ctx = pkg.Context(local)
    stream = torch.cuda.ExternalStream(ctx.cuda_stream, device=torch.device("cuda", local))

    # ---- synthetic inputs (seeded; every rank builds the same genome and its own read shard)
    plan = contig_plan(a.genome_scale)
    t0 = time.perf_counter()
    g = Synth.genome(GENOME_SEED, [l for _, l in plan], names=[n for n, _ in plan], n_frac=0.01, lower_frac=0.03)
    ctx.upload_genome(list(zip(g.names, g.seqs)))
    ginfo = ctx.genome_info()
    t_genome = time.perf_counter() - t0
    bam_refs = list(zip(g.names, g.lens)) + [("chrUn_synthetic_decoy", 1000)]      # the @SQ dictionary of the BAM variant
    cfg = reads_cfg_config2(seed=READS_SEED)
    n_reads = reads_per_rank(a, world)
    lo, hi = rank * n_reads, (rank + 1) * n_reads
    # the shard is generated in pieces of at most 25 M reads through one pinned buffer; the host keeps the whole shard
    # (for the host-fed e2e run and the oracle check) while it is at most 25 M reads, else only the device does
    piece = min(n_reads, 25_000_000)
    cap = Synth.sam_bound(cfg, 0, piece)
    host = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
    host_has_all = n_reads <= piece
    dev = torch.empty(int(n_reads * 252) + (1 << 20), dtype=torch.uint8, device="cuda")
    n_bytes = 0
    for p0 in range(lo, hi, piece):
        nb = Synth.sam_into(cfg, g, p0, min(hi, p0 + piece), host.data_ptr(), cap)
        assert n_bytes + nb + 64 <= dev.numel(), "device text buffer too small"
        dev[n_bytes:n_bytes + nb].copy_(host[:nb])
        n_bytes += nb
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t0
    verify = not a.no_verify
    if not verify:
        del g.seqs[:]

    R = 15
    opts = pkg.PssOptions()
    tables = torch.zeros(2 * (R + 2) * 16, dtype=torch.int64, device="cuda")
    tables_host = torch.zeros(2 * (R + 2) * 16, dtype=torch.int64).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        ctx.pss_begin(opts)
        ctx.feed_device(dev.data_ptr(), n_bytes)
        ctx.pss_finish_device(tables.data_ptr())          # waits for the tally
        if world > 1:
            dist.all_reduce(tables)                        # NCCL sum of the count tables over NVLink
        tables_host.copy_(tables)
        torch.cuda.synchronize()

    def step_e2e():
        ctx.pss_begin(opts)
        ctx.feed_ptr(host.data_ptr(), n_bytes, last=True)  # H2D staging + tally launches, pipelined per 64 MiB
        ctx.pss_finish_device(tables.data_ptr())
        if world > 1:
            dist.all_reduce(tables)
        tables_host.copy_(tables)
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        w0 = time.perf_counter()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        wall = time.perf_counter() - w0
        ms = max(e0.elapsed_time(e1), 0.0)
        # the steps also run host-side calls and (N>1) NCCL on torch's stream: take the larger of device and wall time
        t = torch.tensor([max(ms, wall * 1e3)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(a.warmup):
        step_resident()
    ctx.timing_reset(True)
    sampler = ClockSampler(local) if rank == 0 else None
    ms_total = timed(step_resident, a.steps)
    clocks = sampler.stop() if sampler else None
    tm = ctx.timing()
    stats = ctx.stats()
    ctx.timing_reset(False)
    check_tables = tables_host.clone()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, check_tables, stats, R)

    # ---- end to end through the C ABI with HOST buffers, copies inside the timed region.  Two inputs: the SAM text
    #      `samtools view` would have piped (pssgpu_feed) and the BAM file itself (pssgpu_feed_bam: BGZF inflate + BAM
    #      decoding on the device) -- the reference's real input is the BAM (pss-bam.c:148-162).
    e2e = None
    e2e_variants = {}
    if not a.no_e2e and host_has_all:
        e2e_steps = max(1, min(a.steps, 5))
        step_e2e()
        ctx.timing_reset(False)
        ms_e2e = timed(step_e2e, e2e_steps)
        assert torch.equal(tables_host, check_tables), "host-fed and device-resident tallies differ"
        tm2 = ctx.timing()
        e2e_variants["sam_text"] = {
            "value": world * n_reads * e2e_steps / (ms_e2e * 1e-3), "unit": UNIT, "input": "SAM text in pinned host memory (pssgpu_feed)",
            "h2d_bytes_per_step": int(n_bytes), "d2h_bytes_per_step": int(tables_host.numel() * 8),
            "ms_per_step": ms_e2e / e2e_steps, "host_gb_per_s": n_bytes * world * e2e_steps / (ms_e2e * 1e-3) / 1e9,
            "launches_per_step": int(tm2["launches"] // e2e_steps) if tm2["launches"] else None}
        try:
            refs = bam_refs
            bcap = Synth.lib().synth_bam_bound(n_bytes, len(refs))
            hbam = torch.empty(bcap, dtype=torch.uint8, pin_memory=True)
            tb = time.perf_counter()
            n_bam = Synth.bam_into(host.data_ptr(), n_bytes, refs, hbam.data_ptr(), bcap, level=6, qual_mode=1)
            t_bam = time.perf_counter() - tb

            def step_e2e_bam():
                ctx.pss_begin(opts)
                ctx.feed_bam_ptr(hbam.data_ptr(), n_bam, last=True)     # H2D of the compressed file + inflate + decode + tally
                ctx.pss_finish_device(tables.data_ptr())
                if world > 1:
                    dist.all_reduce(tables)
                tables_host.copy_(tables)
                torch.cuda.synchronize()
            step_e2e_bam()
            ctx.timing_reset(False)
            ms_bam = timed(step_e2e_bam, e2e_steps)
            assert torch.equal(tables_host, check_tables), "BAM-fed and device-resident tallies differ"
            tm3 = ctx.timing()
            e2e_variants["bam"] = {
                "value": world * n_reads * e2e_steps / (ms_bam * 1e-3), "unit": UNIT,
                "input": "the same alignments as a BAM file (BGZF, zlib level 6, binned qualities) in pinned host memory (pssgpu_feed_bam)",
                "h2d_bytes_per_step": int(n_bam), "d2h_bytes_per_step": int(tables_host.numel() * 8),
                "ms_per_step": ms_bam / e2e_steps, "host_gb_per_s": n_bam * world * e2e_steps / (ms_bam * 1e-3) / 1e9,
                "launches_per_step": int(tm3["launches"] // e2e_steps) if tm3["launches"] else None,
                "bam_bytes_per_read": n_bam / n_reads, "bam_conversion_s": t_bam, "info": ctx.bam_info()}
            del hbam
        except Exception as ex:                                     # the text path stays the end-to-end number
            e2e_variants["bam"] = {"error": f"{type(ex).__name__}: {ex}"}
        best = max((v for v in e2e_variants.values() if "value" in v), key=lambda v: v["value"])
        e2e = dict(best)
        e2e["variants"] = e2e_variants

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        PEAK = (float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)")
    else:
        PEAK = (6650.0, "fallback (B200_PROFILING.md)")

    # ---- the sibling hot paths on the same resident data (configs[2], configs[3]); reported, not the headline
    other = None
    try:
        fko = pkg.FragkonOptions(klen=8)
        ctx.fragkon_begin(fko)
        ctx.feed_device(dev.data_ptr(), n_bytes)
        ctx.sync()                                            # warm-up
        ctx.fragkon_begin(fko)
        ctx.timing_reset(True)
        ctx.feed_device(dev.data_ptr(), n_bytes)
        ctx.sync()
        fk_ms = ctx.timing()["kernel_ms"]
        fk_stats = ctx.stats()
        ctx.both_begin(opts, fko)                             # pss-bam + fragkon from one scan (configs[4] workflow)
        ctx.feed_device(dev.data_ptr(), n_bytes)
        ctx.sync()
        ctx.both_begin(opts, fko)
        ctx.timing_reset(True)
        ctx.feed_device(dev.data_ptr(), n_bytes)
        ctx.sync()
        both_ms = ctx.timing()["kernel_ms"]
        spec = {}
        counts = torch.zeros(1 << 24, dtype=torch.int64, device="cuda")
        for k in (8, 12):
            ctx.kmer_spectrum_device(k, counts.data_ptr())   # warm-up
            ctx.timing_reset(True)
            ctx.kmer_spectrum_device(k, counts.data_ptr())
            spec[k] = ctx.timing()["kernel_ms"]
        ctx.timing_reset(False)
        # configs[3] over N GPUs: every rank counts its slice of the packed genome, then one NCCL all-reduce of the 4^k
        # u64 counters (128 MiB at k = 12 -- the only bandwidth-relevant collective of the project)
        sharded = None
        if world > 1:
            sharded = {}
            for k in (8, 12):
                nb = 1 << (2 * k)
                best = None
                for _ in range(3):
                    barrier()
                    ctx.timing_reset(True)
                    ctx.kmer_spectrum_device(k, counts.data_ptr(), rank, world)      # synchronous: returns when the shard is counted
                    k_ms = ctx.timing()["kernel_ms"]
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    barrier()
                    e0.record()
                    dist.all_reduce(counts[:nb])
                    e1.record()
                    torch.cuda.synchronize()
                    t = torch.tensor([k_ms, e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    cur = [float(x) for x in t.tolist()]
                    if best is None or sum(cur) < sum(best):
                        best = cur
                sharded[f"k{k}"] = {"count_ms_max_rank": best[0], "allreduce_ms": best[1], "allreduce_bytes": nb * 8,
                                    "allreduce_busbw_gb_per_s": 2 * (world - 1) / world * nb * 8 / (best[1] * 1e-3) / 1e9,
                                    "gbase_per_s": ginfo["n_bases"] / ((best[0] + best[1]) * 1e-3) / 1e9,
                                    "total_kmers": int(counts[:nb].sum().item())}
            ctx.timing_reset(False)
        # configs[4]: both programs over one scan with -q 30 -l 30 -L 150 (pss-bam.c:96-103,409; fragkon.c:52-58,139)
        o4 = pkg.PssOptions(min_len=30, max_len=150, min_mq=30)
        f4 = pkg.FragkonOptions(klen=8, min_len=30, max_len=150, min_mq=30)
        ctx.both_begin(o4, f4)
        ctx.feed_device(dev.data_ptr(), n_bytes)
        ctx.sync()
        ctx.both_begin(o4, f4)
        ctx.timing_reset(True)
        ctx.feed_device(dev.data_ptr(), n_bytes)
        ctx.sync()
        c4_ms = ctx.timing()["kernel_ms"]
        c4_counted, c4_counted_fk = ctx.stats()["counted"], ctx.fragkon_stats()["counted"]
        ctx.timing_reset(False)

        def roof(alg_bytes, ms, bound="hbm"):
            ach = alg_bytes / (ms * 1e-3) / 1e9
            return {"bound": bound, "achieved": ach, "peak": PEAK[0], "unit": "GB/s", "frac": ach / PEAK[0], "traffic": None,
                    "kernel_ms": ms, "algorithmic_bytes_per_launch": int(alg_bytes)}

        fk_counted = fk_stats["counted"]
        other = {"fragkon_k8": {"reads_per_s_per_gpu": n_reads / (fk_ms * 1e-3), "sam_gb_per_s_per_gpu": n_bytes / (fk_ms * 1e-3) / 1e9,
                                "kernel_ms": fk_ms, "kernel": "tally_kernel<fragkon>",
                                # SURVEY 8(d): record bytes + accepted x 2 x ceil(2K / 8)
                                "roofline": roof(n_bytes + fk_counted * 2 * 2, fk_ms)},
                 "pss_and_fragkon_fused": {"reads_per_s_per_gpu": n_reads / (both_ms * 1e-3), "kernel_ms": both_ms,
                                           "kernel": "tally_kernel<both>",
                                           "vs_two_passes": (tm["kernel_ms"] / max(1, int(tm["launches"])) + fk_ms) / both_ms,
                                           "roofline": roof(n_bytes + stats["counted"] * 9 + fk_counted * 4, both_ms)},
                 "config4_q30_l30_L150_fused": {"workload": "configs[4] per-GPU share: pss-bam + fragkon (K = 8) from one scan of this "
                                                            "rank's reads with -q 30 -l 30 -L 150",
                                                "reads_per_s_per_gpu": n_reads / (c4_ms * 1e-3), "kernel_ms": c4_ms,
                                                "counted_pss": c4_counted, "counted_fragkon": c4_counted_fk,
                                                "roofline": roof(n_bytes + c4_counted * 9 + c4_counted_fk * 4, c4_ms)},
                 "genome_kmer_count": {f"k{k}": {"kernel_ms": ms, "gbase_per_s_per_gpu": ginfo["n_bases"] / (ms * 1e-3) / 1e9,
                                                 "kernels": "spectrum_smem_kernel<8>, widen_kernel" if k <= 9
                                                 else "radix_count / radix_scan / radix_scatter / radix_hist, widen_kernel",
                                                 # DESIGN 3.2: packed genome in (0.5 B per base) + 4^k x 8 B table out
                                                 "roofline": roof(ginfo["hbm_bytes"] + (1 << (2 * k)) * 8, ms),
                                                 "bound": "shared-memory atomics / instruction issue (not HBM)" if k <= 9
                                                 else "radix partition: instruction issue of the in-tile sort (not HBM)"}
                                       for k, ms in spec.items()}}
        if sharded:
            other["genome_kmer_count_sharded_allreduce"] = sharded
        del counts
        if rank == 0 and world == 1:
            other["config0_10Mb_1M_50bp"] = config0_case(pkg, local, torch, not a.no_cpu_baseline)
    except Exception as ex:                                   # never let the side measurements break the contract line
        other = {"error": f"{type(ex).__name__}: {ex}"}

    # ---- parity gate on what was benchmarked: this rank's exact shard through the oracle on the host cores; with
    #      N > 1 the sum of the ranks' oracle tables against the all-reduced device tables
    verify_result = "skipped (--no-verify)"
    verify_s = None
    if verify and not host_has_all:
        verify_result = "skipped (shard larger than the host keeps; run with the default --scaling weak)"
    elif verify:
        from pss_testlib import Oracle, PssParams, oracle_parallel
        tv = time.perf_counter()
        ora = Oracle(contigs=list(zip(g.names, g.seqs)))
        threads = max(1, min(mine, cores // max(1, world)))
        of, orv, ost = oracle_parallel(ora, host[:n_bytes].numpy(), "pss", PssParams(), threads)
        ora.close()
        del g.seqs[:]
        want = torch.from_numpy(np.concatenate([of.reshape(-1), orv.reshape(-1)]).astype(np.int64)).cuda()
        ost_t = torch.tensor([ost[k] for k in ("lines", "counted", "no_contig", "filtered", "parse_fail", "undefined")],
                             dtype=torch.int64, device="cuda")
        gst_t = torch.tensor([stats[k] for k in ("lines", "counted", "no_contig", "filtered", "parse_fail", "undefined")],
                             dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(want)
            dist.all_reduce(ost_t)
            dist.all_reduce(gst_t)
        same = bool(torch.equal(want.cpu(), check_tables)) and bool(torch.equal(ost_t, gst_t))
        verify_s = time.perf_counter() - tv
        verify_result = "oracle-equal" if same else "MISMATCH"
        assert same, "benchmarked tables differ from the oracle"

    # ---- gather totals
    tot = torch.tensor([float(n_bytes), float(stats["counted"]), float(stats["lines"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tot)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    total_bytes, total_counted, total_lines = (float(x) for x in tot.tolist())
    # with N > 1 the all-reduced tables hold every rank's reads; the tables are reset at every step (pssgpu_pss_begin),
    # so one step's worth: row 1 of the 5' table holds at most one increment per counted read
    fwd = check_tables[: (R + 2) * 16].view(R + 2, 16)
    assert 0 < int(fwd[1].sum()) <= int(total_counted)
    assert int(total_lines) == world * n_reads

    value = world * n_reads * a.steps / (ms_total * 1e-3)
    launches = int(tm["launches"])
    kern_ms = tm["kernel_ms"] / max(1, launches)
    alg_bytes = n_bytes + stats["counted"] * 9          # SURVEY 8(d): record bytes + accepted x ceil(2*(R+2)*2 bit / 8)
    peak, peak_src = PEAK
    achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "tally_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            if tj.get("sam_bytes") == int(n_bytes):
                traffic = tj.get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "verify": verify_result,
        "config": {"workload": workload_name(a, world), "reads_per_gpu": n_reads, "sam_bytes_per_gpu": int(n_bytes),
                   "bytes_per_read": n_bytes / n_reads, "genome_bases": ginfo["n_bases"], "genome_hbm_bytes": ginfo["hbm_bytes"],
                   "region_len": R, "l2": "input (%.1f GB/GPU) larger than L2, no flush needed" % (n_bytes / 1e9),
                   "seeds": {"genome": GENOME_SEED, "reads": READS_SEED},
                   "accepted_fraction": total_counted / max(1.0, total_lines),
                   "setup_s": {"genome_synth_upload_pack": t_genome, "total": t_setup, "oracle_verify": verify_s},
                   "verify": "after the timed loop every rank's exact shard is tallied by the CPU oracle (oracle/liboracle.so, all "
                             "host cores) and the (all-reduced) tables and outcome counters must be equal"},
        "sam_gb_per_s": total_bytes * a.steps / (ms_total * 1e-3) / 1e9,
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": "tally_kernel<pss>", "kernel_ms": kern_ms,
                     "algorithmic_bytes_per_launch": int(alg_bytes), "peak_source": peak_src},
        "clocks": clocks,
        "e2e": e2e,
        "other_paths": other,
    }
    if not a.no_cpu_baseline:
        try:
            ref = ReferenceSample(1, a.cpu_sample_reads, a.cpu_genome_mb, READS_SEED)
            v, tally = ref.run()
            load = ref.load
            ref.close()
            line["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": 1, "kind": ref.kind,
                "sample": ((f"unmodified reference oracle/_ref/pss-bam (stock flags -gdwarf-2 -g, no -O; single-threaded), "
                            if ref.kind == "reference" else "oracle port oracle/liboracle.so (-O2; oracle/_ref not found), ") +
                           f"{a.cpu_sample_reads} config-2 reads on a {a.cpu_genome_mb} Mb 4-contig genome, "
                           f"{tally:.1f} s tally after subtracting {load:.1f} s FASTA load"),
                "host_cores_available": cores}
        except Exception as ex:
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 1, "kind": "reference",
                                    "sample": f"unavailable: {type(ex).__name__}: {ex}"}
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse_args()
    if args.impl == "reference":
        main_reference(args)
    else:
        main_b200(args)
