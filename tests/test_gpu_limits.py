"""GPU parity at the limits of the tally kernel, where the bulk tests never go.

A. The 16-bit partial sums.  Every lane of the tally keeps two 16-bit cell counts per register (tally_set16 /
   tally_rows) and flushes them into the CTA table every kFlushEvery = 1900 warp-loads; 1900 x 32 = 60 800 < 65 536 is
   what keeps a half-word from carrying into its neighbour.  Runs of hundreds of thousands of identical records, walked
   by one CTA, push every cell of every read row past 32 768 between two flushes, with -r 14, 15, 16, 17 and 30 (every
   instantiation of the transposed and the ballot rows) and through the fused pass.
B. Every -r from 0 to 32, the -r that pick a different instantiation (15, 16, 17, 30, 31) and large -r up to the largest
   accepted (2045), over text that holds records longer than a tile and longer than fgets' buffer: the one-thread
   long_record path in every mode and with every kind of table.
C. fragkon at every K (1 ... 14) on that text; the spectrum at k = 14 and the hot-bin genome at k = 11 ... 14.
D. One CTA over more than 4 GiB of text: the 64-bit range and tile arithmetic.

The reference is always the CPU oracle.  Where the text is many copies of a few lines or blocks, the expected tables and
counters are the oracle's result for each line or block times its number of copies, summed in u64: the tallies are sums
over lines, so this is exact, and the oracle's cost does not grow with the text.

Memory: fragkon at K = 14 and the spectrum at k = 14 have 4^14 bins.  The device then holds a 4 GiB fragkon table (two
2 GiB halves), and the host holds two 2 GiB arrays for the device's result and two for the oracle's (one of each for the
spectrum).  Item D keeps about 4.6 GB of text on the device.

Out of scope:
- the u32 per-CTA tables and outcome counters: they overflow only past 2^32 records in one CTA, hundreds of GB of text;
- the L2-atomics fallback of the spectrum: it runs only when its 6 GB allocation fails, which cannot be forced without
  starving everything else on the GPU;
- the BAM ingest: tests/test_gpu_bam.py covers it.
"""
import importlib
import random

import numpy as np
import pytest

from pss_testlib import FkParams, Oracle, PssParams, Synth, reads_cfg_config2
from test_gpu_edge import _line_offsets, _opts
from test_record_logic import _mutate

pytestmark = pytest.mark.gpu
pkg = importlib.import_module("pss-bam_b200")

TILE = 256               # records per tile (kThreads): one warp-load for each of the 8 warps of a CTA
FLUSH_EVERY = 1900       # warp-loads between flushes of the 16-bit partial sums (kFlushEvery)
FGETS = 200000           # fgets' stretch (MAX_LINE_LEN)
COUNTED = 0              # outcome code of a counted line


def _fk_opts(fk):
    return pkg.FragkonOptions(fk.klen, fk.min_len, fk.max_len, fk.min_mq, fk.merged_only)


def _tally(ctx, feed, p=None, fk=None):
    """One pss (p), fragkon (fk) or fused (both) tally of what feed() feeds: (pss tables, fragkon tables, stats,
    fragkon stats of the fused pass); None where the mode has no such result."""
    if p is not None and fk is not None:
        ctx.both_begin(_opts(p), _fk_opts(fk))
    elif p is not None:
        ctx.pss_begin(_opts(p))
    else:
        ctx.fragkon_begin(_fk_opts(fk))
    feed()
    pt = ctx.pss_finish() if p is not None else None
    ft = ctx.fragkon_finish() if fk is not None else None
    fst = ctx.fragkon_stats() if p is not None and fk is not None else None
    return pt, ft, ctx.stats(), fst


def _scaled(ora, pieces, p=None, fk=None):
    """The oracle's result for text made of `pieces` = [(bytes, copies)], each piece whole lines: every table and
    counter of each piece times its copies, summed in u64.  Same tuple as _tally."""
    pt = ft = st = fst = None
    for text, n in pieces:
        n64 = np.uint64(n)
        if p is not None:
            f, r, s = ora.pss(text, p)
            pt = (f * n64, r * n64) if pt is None else (pt[0] + f * n64, pt[1] + r * n64)
            st = {k: v * n for k, v in s.items()} if st is None else {k: st[k] + v * n for k, v in s.items()}
        if fk is not None:
            a, b, s = ora.fragkon(text, fk)
            ft = (a * n64, b * n64) if ft is None else (ft[0] + a * n64, ft[1] + b * n64)
            if p is None:
                st = {k: v * n for k, v in s.items()} if st is None else {k: st[k] + v * n for k, v in s.items()}
            else:
                fst = {k: v * n for k, v in s.items()} if fst is None else {k: fst[k] + v * n for k, v in s.items()}
    return pt, ft, st, fst


def _assert_same(got, want):
    gpt, gft, gst, gfst = got
    pt, ft, st, fst = want
    assert gst == st
    assert gfst == fst
    if pt is not None:
        assert np.array_equal(gpt[0], pt[0]) and np.array_equal(gpt[1], pt[1])
    if ft is not None:
        assert np.array_equal(gft[0], ft[0]) and np.array_equal(gft[1], ft[1])


def _each_range_setting(monkeypatch, nbytes):
    """One range over the whole text (a single CTA walks it), then the default ranges."""
    monkeypatch.setenv("PSSGPU_RANGE_KB", str(nbytes // 1024 + 1))
    yield "one range"
    monkeypatch.delenv("PSSGPU_RANGE_KB")
    yield "default ranges"


# --------------------------------------------------------------------------- A. 16-bit partial sums at saturation
HP_BLOCK = 400
HP_SPACER = b"ACGTTGCA" * 4
RUN_TILES = 2100
LONG_RUN_TILES = 6200


def _hp_genome():
    """Contig "hp": spacer, then A..., C..., G..., T... blocks of HP_BLOCK bases, each followed by a spacer; and an
    ordinary random contig.  Returns (contigs, 1-based POS of a 32M read well inside block i)."""
    seq = HP_SPACER + b"".join(bytes([b]) * HP_BLOCK + HP_SPACER for b in b"ACGT")
    contigs = [("hp", np.frombuffer(seq, dtype=np.uint8).copy()), ("chr1", Synth.genome(81, [20000]).seqs[0])]
    pos = [len(HP_SPACER) + i * (HP_BLOCK + len(HP_SPACER)) + 100 + 1 for i in range(4)]
    return contigs, pos


def _hp_runs(pos):
    """[(line, copies)]: every (block i, read base j) variant forward in a run of RUN_TILES tiles, four of them also
    reverse (flag 16), and one forward variant in a run of LONG_RUN_TILES tiles."""
    def line(i, j, flag):
        base = b"ACGT"[j:j + 1]
        return b"hp%d%d_%d\t%d\thp\t%d\t60\t32M\t*\t0\t0\t%s\t%s\n" % (i, j, flag, flag, pos[i], base * 32, b"I" * 32)
    runs = [(line(i, j, 0), RUN_TILES * TILE) for i in range(4) for j in range(4)]
    runs += [(line(i, (i + 1) % 4, 16), RUN_TILES * TILE) for i in range(4)]
    runs.insert(4, (line(2, 1, 0), LONG_RUN_TILES * TILE))
    return runs


@pytest.fixture(scope="module")
def saturating():
    import torch
    contigs, pos = _hp_genome()
    ora = Oracle(contigs=contigs)
    ctx = pkg.Context(0)
    ctx.upload_genome(contigs)
    runs = _hp_runs(pos)
    dev = torch.cat([torch.frombuffer(bytearray(ln), dtype=torch.uint8).cuda().repeat(n) for ln, n in runs])
    yield ora, ctx, runs, dev
    del dev
    ctx.close()


@pytest.mark.parametrize("R,K", [(14, None), (15, None), (16, None), (17, None), (30, None), (15, 3), (16, 9), (30, 12)])
def test_partial_sums_at_saturation(saturating, monkeypatch, R, K):
    """Runs of identical records drive every 16-bit partial sum of the read rows past 32 768 between two flushes.

    With one range, one CTA walks the text; each of its 8 warps takes 32 consecutive records of every 256-record tile,
    one warp-load.  A run of RUN_TILES = 2100 tiles (537 600 records) holds at least 2098 whole tiles of its variant: at
    least 2048 consecutive warp-loads per warp, with a slack of 52 tiles for the tiles shared with the neighbouring runs.
    Flushes 1900 warp-loads apart leave at most two flushes inside 2048 warp-loads, so one stretch of at least 1024
    consecutive flush-free warp-loads of a single variant (max(f, 2048 - f), or the 1900 between two flushes).  Each of
    them adds 32 to the same cell in the same lane: >= 32 768 there, bit 15 of the half-word set.  The 16 (block, read
    base) variants put every cell of every read row of both tables through this, forward and reverse reads too.
    The run of LONG_RUN_TILES = 6200 tiles holds 6198 >= 4096 + 2048 whole tiles: with any flush interval I from 2048
    to 4096, either the first flush comes after >= 2048 warp-loads or the next one comes a whole I later, still inside
    the run; 2048 x 32 = 65 536 does not fit a half-word.
    """
    ora, ctx, runs, dev = saturating
    lens = [n for _, n in runs]
    assert min(lens) >= RUN_TILES * TILE and RUN_TILES - 2 >= 2048 and 1024 * 32 == 1 << 15
    assert max(lens) >= LONG_RUN_TILES * TILE and LONG_RUN_TILES - 2 >= 4096 + 2048
    assert FLUSH_EVERY >= 1024 and FLUSH_EVERY * 32 < 1 << 16
    p = PssParams(region_len=R)
    fk = FkParams(klen=K) if K else None
    want = _scaled(ora, runs, p, fk)
    fwd, rev = want[0]
    # not vacuous: every cell of every read row holds at least one whole run
    assert fwd[2:].min() >= RUN_TILES * TILE and rev[2:].min() >= RUN_TILES * TILE
    assert want[2]["counted"] == sum(lens)
    for _ in _each_range_setting(monkeypatch, dev.numel()):
        got = _tally(ctx, lambda: ctx.feed_device(dev.data_ptr(), dev.numel()), p, fk)
        _assert_same(got, want)


# --------------------------------------------------------------------------- B. every -r, long records
R_ALL = list(range(33)) + [45, 63, 64, 150, 512, 1000, 2044, 2045]
SHARED_MAX_R = 64        # -r up to this use the shared text of 30..150-base reads


def _long_record_text(g, ora, seed, min_len, max_len, n, R_sel):
    """Config-2 reads with some mutated lines, and three lines that only long_record handles:
    - a good record made longer than a tile (about 64 KiB) by an 80 KB tag, one fgets stretch;
    - a 400 KB run of 'q' and then a good record: its third fgets stretch is that record;
    - an unparseable line longer than a tile.
    Returns (text, offsets of the two good long stretches).  The good record is one the oracle counts at -r R_sel."""
    rng = random.Random(seed)
    good = Synth.sam(reads_cfg_config2(seed=seed, min_len=min_len, max_len=max_len), g, 0, n).split(b"\n")[:-1]
    _, _, _, status = ora.pss(b"\n".join(good) + b"\n", PssParams(region_len=R_sel), want_status=True)
    base = good[int(np.flatnonzero(status == COUNTED)[0])]
    lines = [_mutate(rng, ln) if rng.random() < 0.1 else ln for ln in good]
    long_good = base + b"\tXX:Z:" + b"t" * 80000
    overlong = b"q" * (2 * FGETS) + base
    lines[n // 4:n // 4] = [long_good]
    lines[n // 2:n // 2] = [overlong]
    lines[3 * n // 4:3 * n // 4] = [b"u" * 70000]
    text = b"\n".join(lines) + b"\n"
    at = np.array([text.index(long_good + b"\n"), text.index(overlong + b"\n") + 2 * FGETS], dtype=np.uint64)
    return text, at


@pytest.fixture(scope="module")
def long_world():
    g = Synth.genome(91, [300000, 120000, 5000], n_frac=0.01, lower_frac=0.05)
    ora = Oracle(fasta=g.fasta_bytes())
    ctx = pkg.Context(0)
    ctx.upload_genome(ora.contigs())
    cache = {}

    def text(R):
        """The item-B text for -r R: the shared one for R <= SHARED_MAX_R, else reads of R to R + 200 bases."""
        key = 0 if R <= SHARED_MAX_R else R
        if key not in cache:
            cache[key] = (_long_record_text(g, ora, 101, 30, 150, 6000, SHARED_MAX_R) if key == 0
                          else _long_record_text(g, ora, 100 + R, R, R + 200, 1500, R))
        return cache[key]

    yield g, ora, ctx, text
    ctx.close()


def _check_logged(ctx, ora, text, at, p=None, fk=None):
    """Tables, counters and the per-line outcome log against the oracle's; the long records must be counted."""
    if p is not None:
        a, b, st, status = ora.pss(text, p, want_status=True)
    else:
        a, b, st, status = ora.fragkon(text, fk, want_status=True)
    ctx.debug_status(True)
    ga, gb = ctx.pss(text, _opts(p)) if p is not None else ctx.fragkon(text, _fk_opts(fk))
    gst = ctx.stats()
    off, code = ctx.debug_fetch()
    ctx.debug_status(False)
    offs = _line_offsets(text)
    assert np.array_equal(off, offs)
    bad = np.flatnonzero(code != status)
    assert bad.size == 0, (bad[:5], code[bad[:5]], status[bad[:5]])
    assert gst == st
    assert np.array_equal(ga, a) and np.array_equal(gb, b)
    idx = np.searchsorted(offs, at)
    assert np.array_equal(offs[idx], at)
    return a, b, code[idx]


@pytest.mark.parametrize("R", R_ALL)
def test_every_region_length(long_world, R):
    """Each -r over text with records longer than a tile and than fgets' buffer.  -r 14 is the largest whose rows
    all fit one transposed set, 15 the <., 9, 17> instantiation, 16 the only -r with ballot row 17, 17 the first of
    <., 16, 0>, 30 the last of it; from 31 on pss_record_wide and global atomics."""
    g, ora, ctx, text = long_world
    sam, at = text(R)
    f, r, codes = _check_logged(ctx, ora, sam, at, p=PssParams(region_len=R))
    assert f[-1].any() and r[-1].any()               # the last row of both tables is reached
    assert (codes == COUNTED).all()                  # the long records went through long_record and were counted


@pytest.mark.parametrize("R,K", [(0, 1), (14, 5), (15, 8), (16, 6), (17, 7), (30, 10), (31, 4), (2045, 12), (15, 13), (15, 14)])
def test_fused_pass_with_long_records(long_world, R, K):
    """The fused pass (long_record<kModeBoth>) against separate oracle runs of both programs, outcome counters of
    both included."""
    g, ora, ctx, text = long_world
    sam, at = text(R)
    p, fk = PssParams(region_len=R), FkParams(klen=K)
    f, r, st, status = ora.pss(sam, p, want_status=True)
    assert (status[np.searchsorted(_line_offsets(sam), at)] == COUNTED).all()
    want = _scaled(ora, [(sam, 1)], p, fk)
    got = _tally(ctx, lambda: ctx.feed(sam, last=True), p, fk)
    _assert_same(got, want)
    assert f[-1].any() and r[-1].any() and want[1][0].any() and want[1][1].any()


# --------------------------------------------------------------------------- C. fragkon at every K, spectrum edges
@pytest.mark.parametrize("K", range(1, 15))
def test_fragkon_every_k(long_world, K):
    g, ora, ctx, text = long_world
    sam, at = text(15)
    fp, tp, codes = _check_logged(ctx, ora, sam, at, fk=FkParams(klen=K))
    assert fp.any() and tp.any()
    assert (codes == COUNTED).all()                  # the long records went through long_record and were counted


def test_spectrum_k14_parity_genome():
    g = Synth.genome(11, [400000, 250000, 1000, 90], n_frac=0.01, lower_frac=0.05)
    ora = Oracle(fasta=g.fasta_bytes())
    ctx = pkg.Context(0)
    ctx.upload_genome(ora.contigs())
    want = ora.kmer_spectrum(14)
    assert np.array_equal(ctx.kmer_spectrum(14), want)
    parts = ctx.kmer_spectrum(14, 0, 3)
    for s in (1, 2):
        parts += ctx.kmer_spectrum(14, s, 3)
    assert np.array_equal(parts, want)
    ctx.close()


@pytest.fixture(scope="module")
def hot_genome():
    """The low-complexity genome of test_gpu_edge.test_spectrum_hot_bins."""
    g = Synth.genome(71, [9_000_000, 6_000_000, 1_000_003], n_frac=0.01, lower_frac=0.02)
    for s, (at, n, motif) in zip(g.seqs, [(1_000_000, 5_000_000, b"A"), (500_000, 4_000_000, b"CA"), (1000, 700_000, b"CAG")]):
        s[at:at + n] = np.frombuffer((motif * (n // len(motif) + 1))[:n], dtype=np.uint8)
    g.seqs[0][3_000_000:3_000_040] = np.frombuffer(b"N" * 40, dtype=np.uint8)
    ora = Oracle(contigs=list(zip(g.names, g.seqs)))
    ctx = pkg.Context(0)
    ctx.upload_genome(list(zip(g.names, g.seqs)))
    yield ora, ctx
    ctx.close()


@pytest.mark.parametrize("k", [11, 12, 13, 14])
def test_spectrum_hot_bins_large_k(hot_genome, monkeypatch, k):
    """k = 11, 12: the radix instantiations; 13, 14: global atomics; each in 32-bit and in 64-bit bins."""
    ora, ctx = hot_genome
    want = ora.kmer_spectrum(k)
    assert int(want.max()) > 3_000_000
    assert np.array_equal(ctx.kmer_spectrum(k), want)
    monkeypatch.setenv("PSSGPU_SPECTRUM_WIDE", "1")
    assert np.array_equal(ctx.kmer_spectrum(k), want)


# --------------------------------------------------------------------------- D. one CTA over more than 4 GiB
def test_one_cta_over_4gib(long_world, monkeypatch):
    """A 32 MiB block of whole lines, repeated on the device past 4.5 GB and fed at once.  With one range a single CTA
    walks all of it: range, tile and copy offsets beyond 2^32 bytes inside one CTA."""
    import torch
    g, ora, ctx, _ = long_world
    rng = random.Random(7)
    good = Synth.sam(reads_cfg_config2(seed=111), g, 0, 135000).split(b"\n")[:-1]
    lines = [_mutate(rng, ln) if rng.random() < 0.05 else ln for ln in good]
    lines.insert(1000, good[5] + b"\tXX:Z:" + b"t" * 90000)
    block = b"\n".join(lines) + b"\n"
    assert 30 << 20 <= len(block) <= 40 << 20
    reps = -(-4_500_000_000 // len(block))
    dev = torch.frombuffer(bytearray(block), dtype=torch.uint8).cuda().repeat(reps)
    assert dev.numel() > 4_500_000_000 > 1 << 32
    for p, fk in ((PssParams(), None), (PssParams(region_len=30), FkParams(klen=8))):
        want = _scaled(ora, [(block, reps)], p, fk)
        assert want[2]["counted"] > 0 and want[2]["parse_fail"] > 0
        for _ in _each_range_setting(monkeypatch, dev.numel()):
            _assert_same(_tally(ctx, lambda: ctx.feed_device(dev.data_ptr(), dev.numel()), p, fk), want)
    del dev
