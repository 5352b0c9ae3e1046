"""Parity at the scale BASELINE.json names: the 3.1 Gb / 24-contig synthetic genome of bench.py (base offsets beyond
2^31, contigs of up to 249 Mb) with slices of the 200 M-read set, against the oracle (on all host cores); the
size-independent properties the bench relies on (shard invariance, host-fed == device-resident); configs[3] -- the
k = 8 and k = 12 spectra of the whole genome, 32- and 64-bit bins -- and configs[4] -- pss-bam + fragkon from one scan
with -q 30 -l 30 -L 150."""
import importlib
import os
import sys

import numpy as np
import pytest

from pss_testlib import (FkParams, Oracle, PssParams, RefBin, Synth, oracle_parallel, oracle_spectrum_parallel,
                         reads_cfg_config2, tmpdir)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("pss-bam_b200")
CORES = os.cpu_count() or 1


@pytest.fixture(scope="module")
def full():
    """(genome, oracle, context with the genome resident) -- built once for the module."""
    import bench
    Synth.set_threads(CORES)
    plan = bench.contig_plan(1.0)
    g = Synth.genome(bench.GENOME_SEED, [l for _, l in plan], names=[n for n, _ in plan], n_frac=0.01, lower_frac=0.03)
    assert sum(g.lens) > 3_000_000_000
    ctx = pkg.Context(0)
    ctx.upload_genome(list(zip(g.names, g.seqs)))
    ora = Oracle(contigs=list(zip(g.names, g.seqs)))
    yield g, ora, ctx
    ctx.close()
    ora.close()


def test_full_size_genome_slice_of_reads(full):
    import bench
    import torch
    g, ora, ctx = full
    cfg = reads_cfg_config2(seed=bench.READS_SEED)
    lo, n = 5 * 25_000_000, 1_500_000                       # a slice of rank 5's shard of the 200 M reads
    sam = Synth.sam(cfg, g, lo, lo + n)

    f, r, st = oracle_parallel(ora, sam, "pss", PssParams(), CORES)
    fp, tp, fst = oracle_parallel(ora, sam, "fragkon", FkParams(klen=8), CORES)

    gf, gr = ctx.pss(sam)
    assert ctx.stats() == st and st["counted"] > 1_000_000
    assert np.array_equal(gf, f) and np.array_equal(gr, r)
    gfp, gtp = ctx.fragkon(sam, pkg.FragkonOptions(klen=8))
    assert ctx.stats() == fst
    assert np.array_equal(gfp, fp) and np.array_equal(gtp, tp)

    # device-resident input gives the same tables as host-fed input
    dev = torch.frombuffer(bytearray(sam), dtype=torch.uint8).cuda()
    ctx.pss_begin(pkg.PssOptions())
    ctx.feed_device(dev.data_ptr(), len(sam))
    df, dr = ctx.pss_finish()
    assert np.array_equal(df, f) and np.array_equal(dr, r)

    # shard invariance: two halves cut at a newline sum to the whole
    d = importlib.import_module("pss-bam_b200.dist")
    parts = []
    for rank in range(2):
        a, b = d.shard_sam_bytes(sam, rank, 2)
        parts.append(ctx.pss(sam[a:b]))
    assert np.array_equal(parts[0][0] + parts[1][0], f) and np.array_equal(parts[0][1] + parts[1][1], r)


def test_config4_filters_fused_pass(full):
    """BASELINE.json configs[4]: pss-bam + fragkon over the same stream with -q 30 -l 30 -L 150 (pss-bam.c:96-103,409,
    676-678; fragkon.c:52-58,139), both tallies from ONE scan (pssgpu_both_begin), on the full-size genome, against two
    separate oracle runs.  Read lengths 20..170 so that both length bounds reject something."""
    import bench
    g, ora, ctx = full
    cfg = reads_cfg_config2(seed=bench.READS_SEED + 4, min_len=20, max_len=170)
    sam = Synth.sam(cfg, g, 3_000_000, 3_000_000 + 1_500_000)
    pp = PssParams(min_len=30, max_len=150, min_mq=30)
    fkp = FkParams(klen=8, min_len=30, max_len=150, min_mq=30)
    f, r, st = oracle_parallel(ora, sam, "pss", pp, CORES)
    fp, tp, fst = oracle_parallel(ora, sam, "fragkon", fkp, CORES)
    assert 200_000 < st["counted"] < 900_000                 # the filters bite (about half the MAPQs are < 30)

    ctx.both_begin(pkg.PssOptions(min_len=30, max_len=150, min_mq=30), pkg.FragkonOptions(klen=8, min_len=30, max_len=150, min_mq=30))
    ctx.feed(sam, last=True)
    gf, gr = ctx.pss_finish()
    gfp, gtp = ctx.fragkon_finish()
    assert ctx.stats() == st and ctx.fragkon_stats() == fst
    assert np.array_equal(gf, f) and np.array_equal(gr, r)
    assert np.array_equal(gfp, fp) and np.array_equal(gtp, tp)
    # and each program on its own with the same options
    gf2, gr2 = ctx.pss(sam, pkg.PssOptions(min_len=30, max_len=150, min_mq=30))
    assert np.array_equal(gf2, f) and np.array_equal(gr2, r) and ctx.stats() == st
    a2, b2 = ctx.fragkon(sam, pkg.FragkonOptions(klen=8, min_len=30, max_len=150, min_mq=30))
    assert np.array_equal(a2, fp) and np.array_equal(b2, tp) and ctx.stats() == fst


@pytest.mark.parametrize("k", [8, 12])
def test_full_size_spectrum_vs_oracle(full, k):
    """BASELINE.json configs[3] at full size (genome-kmer-count.c:56-58,68-79): k = 8 (shared-memory bins) and k = 12
    (radix partition through a 6 GB scratch buffer) of the 3.1 Gb genome against the oracle, contig by contig on all
    host cores; shards add up; and the 64-bit-bin instantiations (PSSGPU_SPECTRUM_WIDE forces them) give the same."""
    g, ora, ctx = full
    want = oracle_spectrum_parallel(ora, k, CORES)
    got = ctx.kmer_spectrum(k)
    assert int(want.sum()) > 0.95 * sum(g.lens)
    assert np.array_equal(got, want)
    assert np.array_equal(sum(ctx.kmer_spectrum(k, s, 3) for s in range(3)), want)
    os.environ["PSSGPU_SPECTRUM_WIDE"] = "1"
    try:
        assert np.array_equal(ctx.kmer_spectrum(k), want)
    finally:
        del os.environ["PSSGPU_SPECTRUM_WIDE"]


def _spectrum_genome(mb):
    """A genome as large as the reference's trie walk counts in seconds."""
    Synth.set_threads(CORES)
    return Synth.genome(77, [mb * 600_000, mb * 400_000 - 7], n_frac=0.01, lower_frac=0.03)


@pytest.mark.parametrize("k,mb", [(8, 48), (12, 8)])
def test_spectrum_vs_reference_binary(k, mb):
    """The same two paths against the UNMODIFIED reference program (oracle/_ref/genome-kmer-count-O2, stdout parsed);
    32- and 64-bit bins."""
    if not RefBin.available():
        pytest.skip(RefBin.MISSING)
    g = _spectrum_genome(mb)
    d = tmpdir()
    fa = os.path.join(d, "g.fa")
    with open(fa, "wb") as f:
        f.write(g.fasta_bytes())
    out = RefBin.genome_kmer_count(fa, k, binary="genome-kmer-count-O2")
    lines = out.split(b"\n")
    assert lines[0] == b"Parsed input genome. Found 2 sequences."
    want = np.array([int(ln.split(b"\t")[1]) for ln in lines[1:] if ln], dtype=np.uint64)
    assert want.size == 1 << (2 * k)
    ctx = pkg.Context(0)
    ctx.upload_genome(list(zip(g.names, g.seqs)))
    assert np.array_equal(ctx.kmer_spectrum(k), want)
    os.environ["PSSGPU_SPECTRUM_WIDE"] = "1"
    try:
        assert np.array_equal(ctx.kmer_spectrum(k), want)
    finally:
        del os.environ["PSSGPU_SPECTRUM_WIDE"]
    ctx.close()


@pytest.mark.parametrize("k,mb", [(8, 48), (12, 8)])
def test_spectrum_wide_bins_vs_oracle(k, mb):
    """The genomes of test_spectrum_vs_reference_binary against the oracle, which needs no reference binary: k in 32-
    and 64-bit bins, and k = 5, 9, 13 (the atomics paths) in 64-bit bins."""
    g = _spectrum_genome(mb)
    ctx = pkg.Context(0)
    ctx.upload_genome(list(zip(g.names, g.seqs)))
    ora = Oracle(contigs=list(zip(g.names, g.seqs)))
    want = oracle_spectrum_parallel(ora, k, CORES)
    assert np.array_equal(ctx.kmer_spectrum(k), want)
    os.environ["PSSGPU_SPECTRUM_WIDE"] = "1"
    try:
        assert np.array_equal(ctx.kmer_spectrum(k), want)
        for kk in (5, 9, 13):
            assert np.array_equal(ctx.kmer_spectrum(kk), oracle_spectrum_parallel(ora, kk, CORES)), kk
    finally:
        del os.environ["PSSGPU_SPECTRUM_WIDE"]
    ctx.close()
    ora.close()
