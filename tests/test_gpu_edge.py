"""GPU parity on the paths the bulk tests do not reach: records longer than a tile's look-ahead, lines longer than
fgets' buffer, tiles with more newlines than one pass holds, the global contig table (> 64 contigs), long contig
names, exotic -U/-D bytes (exception list), device-resident input, error codes."""
import importlib
import random

import numpy as np
import pytest

from pss_testlib import FkParams, Oracle, PssParams, Synth, reads_cfg_config1, reads_cfg_config2
from test_record_logic import _mutate

pytestmark = pytest.mark.gpu
pkg = importlib.import_module("pss-bam_b200")


def _opts(p):
    return pkg.PssOptions(p.region_len, p.min_len, p.max_len, p.min_mq, p.up_ctx, p.down_ctx, p.merged_only)


def _line_offsets(sam):
    """fgets view of the stream: a line ends after '\\n' or after 200000 bytes."""
    offs, i, n = [], 0, len(sam)
    while i < n:
        offs.append(i)
        j = sam.find(b"\n", i, i + 200000)
        i = (j + 1) if j >= 0 else min(n, i + 200000)
    return np.array(offs, dtype=np.uint64)


def _check(ctx, ora, sam, p=PssParams(), fk=None):
    f, r, st, status = ora.pss(sam, p, want_status=True)
    ctx.debug_status(True)
    gf, gr = ctx.pss(sam, _opts(p))
    gst = ctx.stats()
    off, code = ctx.debug_fetch()
    ctx.debug_status(False)
    assert np.array_equal(off, _line_offsets(sam))
    bad = np.flatnonzero(code != status)
    assert bad.size == 0, (bad[:5], code[bad[:5]], status[bad[:5]])
    assert gst == st
    assert np.array_equal(gf, f) and np.array_equal(gr, r)
    if fk is not None:
        fp, tp, fst = ora.fragkon(sam, fk)
        gfp, gtp = ctx.fragkon(sam, pkg.FragkonOptions(fk.klen, fk.min_len, fk.max_len, fk.min_mq, fk.merged_only))
        assert ctx.stats() == fst
        assert np.array_equal(gfp, fp) and np.array_equal(gtp, tp)


@pytest.fixture(scope="module")
def small():
    g = Synth.genome(61, [80000, 50000, 3000], names=["chr1", "chr2", "chrM"], n_frac=0.01, lower_frac=0.05)
    g.seqs[1][500:520] = np.frombuffer(b"RYKMSWBDHVNrykmswbdh", dtype=np.uint8)
    g.seqs[1][600:604] = np.frombuffer(b"*-.X", dtype=np.uint8)
    ora = Oracle(fasta=g.fasta_bytes())
    ctx = pkg.Context(0)
    ctx.upload_genome(ora.contigs())
    yield g, ora, ctx
    ctx.close()


def test_long_records_and_overlong_lines(small):
    g, ora, ctx = small
    good = Synth.sam(reads_cfg_config1(seed=5), g, 0, 400).split(b"\n")[:-1]
    lines = []
    for i, ln in enumerate(good):
        lines.append(ln)
        if i % 40 == 7:
            lines.append(ln + b"\tXX:Z:" + b"t" * (2500 + 97 * i))          # good record, longer than the look-ahead
        if i % 97 == 11:
            lines.append(b"x" * 199999)                                     # exactly fgets' buffer with its newline
            lines.append(b"y" * 200000)                                     # splits into two lines
            lines.append(b"z" * 199990 + b" " + ln + b"\t" + b"t" * 250000)  # tail chunk of a 450 KB line parses
    _check(ctx, ora, b"\n".join(lines) + b"\n", fk=FkParams(klen=6))
    _check(ctx, ora, b"\n".join(lines))                                     # no final newline


def test_more_newlines_than_one_pass(small):
    g, ora, ctx = small
    good = Synth.sam(reads_cfg_config2(seed=6, min_len=20, max_len=60), g, 0, 3000).split(b"\n")[:-1]
    rng = random.Random(3)
    lines = []
    for ln in good:
        lines.append(ln)
        lines.extend([b""] * rng.choice([0, 0, 3, 40]))                     # bursts of empty lines
        if rng.random() < 0.05:
            lines.extend([b"a\tb"] * 700)                                   # > 1024 short lines per 32 KiB tile
    _check(ctx, ora, b"\n".join(lines) + b"\n", fk=FkParams(klen=5))
    _check(ctx, ora, b"\n" * 100000 + good[0] + b"\n")


def test_malformed_lines(small):
    g, ora, ctx = small
    for seed in (21, 22):
        rng = random.Random(seed)
        good = Synth.sam(reads_cfg_config2(seed=seed, min_len=20, max_len=70), g, 0, 4000).split(b"\n")[:-1]
        lines = [_mutate(rng, ln) if rng.random() < 0.7 else ln for ln in good]
        _check(ctx, ora, b"\n".join(lines) + b"\n", fk=FkParams(klen=7))


def test_control_bytes_that_look_like_newlines(small):
    """The scan takes "<= 0x20 with bit 1 set" as a newline candidate and verifies it against the byte: VT, 0x02,
    0x0e ... must send their tile to the exact listing, never split a line."""
    g, ora, ctx = small
    good = Synth.sam(reads_cfg_config2(seed=31, min_len=30, max_len=150), g, 0, 6000).split(b"\n")[:-1]
    rng = random.Random(17)
    odd = [0x02, 0x03, 0x06, 0x07, 0x0b, 0x0e, 0x0f, 0x12, 0x16, 0x1a, 0x1e, 0x1f, 0x0c, 0x0d, 0x01, 0x08, 0x20]
    lines = []
    for i, ln in enumerate(good):
        if 1500 <= i < 4500 and rng.random() < 0.04:          # the first and last tiles stay clean (fast path)
            b = bytearray(ln)
            for _ in range(rng.choice([1, 1, 2])):
                b[rng.randrange(len(b))] = rng.choice(odd)
            ln = bytes(b)
        lines.append(ln)
    _check(ctx, ora, b"\n".join(lines) + b"\n", fk=FkParams(klen=6))
    _check(ctx, ora, b"\r\n".join(lines[:2000]) + b"\r\n")        # CRLF text


def test_high_bytes_next_to_separators(small):
    """SWAR classification next to bytes >= 0x80 (UTF-8 names, binary junk): no carry may leak into a neighbouring
    space, tab or newline."""
    g, ora, ctx = small
    good = Synth.sam(reads_cfg_config2(seed=51, min_len=30, max_len=150), g, 0, 6000).split(b"\n")[:-1]
    rng = random.Random(23)
    lines = []
    for i, ln in enumerate(good):
        if 1000 <= i < 5000 and rng.random() < 0.03:
            f = ln.split(b"\t")
            k = rng.randrange(6)
            if k == 0: f[0] = b"r\xc3\xa9ad" + f[0]                         # UTF-8 in QNAME
            elif k == 1: f[-1] = f[-1] + b"\tCO:Z:caf\xff comment \xa1 x"     # 0xff / 0xa1 right before a space
            elif k == 2: f[0] = f[0] + b"\xa1"                                # high byte right before a tab
            elif k == 3: f[-1] = f[-1] + b"\xfe"                              # ... right before the newline
            elif k == 4: f[9] = f[9][:5] + b"\x80" + f[9][6:]                 # 0x80: no carry, still not ASCII
            elif k == 5: ln = b"\xff " + ln; f = None                         # 0xff then the space that sscanf skips
            if f is not None: ln = b"\t".join(f)
        lines.append(ln)
    _check(ctx, ora, b"\n".join(lines) + b"\n", fk=FkParams(klen=6))


def test_tiny_ranges(small, monkeypatch):
    """Ranges of 1 KiB and 3 KiB (a developer switch of the library): a handful of records per range, so every kind of
    range boundary occurs -- inside a record, right after a newline, inside a line longer than the range or a tile."""
    g, ora, ctx = small
    rng = random.Random(5)
    good = Synth.sam(reads_cfg_config2(seed=41, min_len=30, max_len=150), g, 0, 5000).split(b"\n")[:-1]
    lines = []
    for i, ln in enumerate(good):
        lines.append(_mutate(rng, ln) if rng.random() < 0.1 else ln)
        if i % 500 == 250:
            lines.append(ln + b"\tXX:Z:" + b"t" * (3000 + 40 * i))           # longer than a range
        if i == 2500:
            lines.append(b"q" * 70000)                                      # longer than a tile
            lines.extend([b""] * 300)
    sam = b"\n".join(lines) + b"\n"
    for kb in ("1", "3"):
        monkeypatch.setenv("PSSGPU_RANGE_KB", kb)
        _check(ctx, ora, sam, fk=FkParams(klen=6))
        _check(ctx, ora, sam[:-1])                                          # no final newline
    monkeypatch.delenv("PSSGPU_RANGE_KB")


def test_exotic_context_bytes(small):
    g, ora, ctx = small
    sam = Synth.sam(reads_cfg_config1(seed=9, read_len=40), g, 0, 200).split(b"\n")[:-1]
    # reads placed right next to the IUPAC / exotic bytes of chr2 so that their context base is one of them
    seq = g.seqs[1].tobytes().upper()
    extra = []
    for pos0 in range(470, 640):
        rd = seq[pos0:pos0 + 30].replace(b"*", b"A").replace(b"-", b"A").replace(b".", b"A")
        for flag in (0, 16):
            extra.append(b"\t".join([b"e%d" % pos0, str(flag).encode(), b"chr2", str(pos0 + 1).encode(), b"30", b"30M", b"*",
                                     b"0", b"0", rd, b"I" * 30]))
    data = b"\n".join(sam + extra) + b"\n"
    for p in (PssParams(), PssParams(up_ctx=b"ACGTN", down_ctx=b"ACGTRYKM"), PssParams(up_ctx=b"*-.X", down_ctx=b"ACGT*"),
              PssParams(up_ctx=b"ACGT-", down_ctx=b"."), PssParams(up_ctx=b"acgt", down_ctx=b"ACGT")):
        _check(ctx, ora, data, p)


def test_many_contigs_and_long_names():
    names = [f"scaffold_{i:05d}_with_a_rather_long_name" for i in range(150)] + ["x", "chrUn_" + "y" * 200]
    lens = [900 + 7 * i for i in range(150)] + [5000, 4000]
    g = Synth.genome(71, lens, names=names, n_frac=0.01)
    ora = Oracle(fasta=g.fasta_bytes())
    ctx = pkg.Context(0)
    ctx.upload_genome(ora.contigs()[::-1])                      # any order
    sam = Synth.sam(reads_cfg_config2(seed=72, min_len=20, max_len=60), g, 0, 20000)
    _check(ctx, ora, sam, fk=FkParams(klen=8))
    for k in (2, 9):
        assert np.array_equal(ctx.kmer_spectrum(k), ora.kmer_spectrum(k))
    ctx.close()
    # <= 64 contigs but names longer than 16 bytes: shared-memory table with multi-word names
    g2 = Synth.genome(73, [3000] * 20, names=[f"contig_number_{i}_of_the_assembly" for i in range(20)])
    ora2 = Oracle(fasta=g2.fasta_bytes())
    ctx2 = pkg.Context(0)
    ctx2.upload_genome(ora2.contigs())
    _check(ctx2, ora2, Synth.sam(reads_cfg_config2(seed=74, min_len=20, max_len=60), g2, 0, 10000))
    ctx2.close()


def test_device_resident_input_and_reuse(small):
    import torch
    g, ora, ctx = small
    sam = Synth.sam(reads_cfg_config2(seed=11, min_len=20, max_len=90), g, 0, 30000)
    f, r, st = ora.pss(sam, PssParams())
    dev = torch.frombuffer(bytearray(sam), dtype=torch.uint8).cuda()
    tab = torch.zeros(2 * 17 * 16, dtype=torch.int64, device="cuda")
    for _ in range(2):                                           # begin/feed/finish twice on one context
        ctx.pss_begin(pkg.PssOptions())
        ctx.feed_device(dev.data_ptr(), len(sam))
        ctx.pss_finish_device(tab.data_ptr())
        got = tab.cpu().numpy().astype(np.uint64).reshape(2, 17, 16)
        assert np.array_equal(got[0], f) and np.array_equal(got[1], r)
    gf, gr = ctx.pss_finish()                                    # finish may be repeated
    assert np.array_equal(gf, f)
    ctx.feed(sam, last=True)                                     # and the tally stays open
    gf, gr = ctx.pss_finish()
    assert np.array_equal(gf, 2 * f) and np.array_equal(gr, 2 * r)
    # genome uploaded from device memory
    ctx2 = pkg.Context(0)
    keep = [torch.frombuffer(bytearray(s), dtype=torch.uint8).cuda() for _, s in ora.contigs()]
    ctx2.upload_genome_device([(cid, t.data_ptr(), t.numel()) for (cid, _), t in zip(ora.contigs(), keep)])
    gf2, gr2 = ctx2.pss(sam)
    assert np.array_equal(gf2, f) and np.array_equal(gr2, r)
    ctx2.close()


def test_packed_genome_save_and_load(small, tmp_path):
    g, ora, ctx = small
    sam = Synth.sam(reads_cfg_config2(seed=12), g, 0, 5000)
    f, r, st = ora.pss(sam, PssParams())
    path = str(tmp_path / "genome.pssgpu")
    ctx.save_genome(path)
    ctx2 = pkg.Context(0)
    ctx2.load_genome(path)
    assert ctx2.genome_info() == ctx.genome_info()
    gf, gr = ctx2.pss(sam)
    assert ctx2.stats() == st and np.array_equal(gf, f) and np.array_equal(gr, r)
    for k in (4, 8, 11):
        assert np.array_equal(ctx2.kmer_spectrum(k), ora.kmer_spectrum(k))
    p = PssParams(up_ctx=b"*-.X", down_ctx=b"ACGT*")                        # needs the exception list of the cache
    f2, r2, _ = ora.pss(sam, p)
    gf2, gr2 = ctx2.pss(sam, _opts(p))
    assert np.array_equal(gf2, f2) and np.array_equal(gr2, r2)
    # not a cache / truncated cache: refused, no genome resident afterwards
    bad = str(tmp_path / "bad.pssgpu")
    with open(path, "rb") as src, open(bad, "wb") as dst:
        dst.write(src.read()[:-8])
    for pth in (bad, __file__, str(tmp_path / "missing")):
        with pytest.raises(pkg.PssGpuError) as e:
            ctx2.load_genome(pth)
        assert e.value.code == -1
    with pytest.raises(pkg.PssGpuError) as e:
        ctx2.pss_begin(pkg.PssOptions())
    assert e.value.code == -4
    ctx2.close()


def test_error_codes(small):
    g, ora, ctx = small
    with pytest.raises(pkg.PssGpuError) as e:
        ctx.pss_begin(pkg.PssOptions(region_len=2046))        # a counted read has at most 2047 bases
    assert e.value.code == -5
    with pytest.raises(pkg.PssGpuError):
        ctx.fragkon_begin(pkg.FragkonOptions(klen=15))
    with pytest.raises(pkg.PssGpuError):
        ctx.kmer_spectrum(0)
    fresh = pkg.Context(0)
    with pytest.raises(pkg.PssGpuError) as e:
        fresh.pss_begin(pkg.PssOptions())
    assert e.value.code == -4                                    # no genome resident
    with pytest.raises(pkg.PssGpuError):
        fresh.upload_genome([("a", b"ACGT"), ("a", b"GGGG")])    # duplicate ids
    with pytest.raises(pkg.PssGpuError):
        fresh.upload_genome([("a", b"AC\x00GT")])                # NUL byte
    fresh.close()
    ctx.pss_begin(pkg.PssOptions())
    ctx.feed(b"r1\t0\tchr1\t100\t30\t3")                         # unterminated line pending
    with pytest.raises(pkg.PssGpuError):
        ctx.pss_finish()
    ctx.feed(b"", last=True)
    ctx.pss_finish()


def test_fused_pss_and_fragkon_pass(small):
    """One scan of the text feeding both programs' tables == the two separate runs (== the oracle)."""
    g, ora, ctx = small
    rng = random.Random(5)
    good = Synth.sam(reads_cfg_config2(seed=31, min_len=20, max_len=90), g, 0, 20000).split(b"\n")[:-1]
    lines = [_mutate(rng, ln) if rng.random() < 0.2 else ln for ln in good]
    lines.insert(100, good[0] + b"\tXX:Z:" + b"t" * 5000)                   # a record longer than the look-ahead
    sam = b"\n".join(lines) + b"\n"
    for p, fk in ((PssParams(), FkParams(klen=8)),
                  (PssParams(region_len=20, min_len=30, max_len=80, min_mq=20, merged_only=1), FkParams(klen=5, min_len=25, min_mq=7)),
                  (PssParams(region_len=5), FkParams(klen=3)),
                  (PssParams(region_len=40), FkParams(klen=10))):
        f, r, st = ora.pss(sam, p)
        fp, tp, fst = ora.fragkon(sam, fk)
        ctx.both_begin(_opts(p), pkg.FragkonOptions(fk.klen, fk.min_len, fk.max_len, fk.min_mq, fk.merged_only))
        for i in range(0, len(sam), 300007):
            ctx.feed(sam[i:i + 300007], last=(i + 300007 >= len(sam)))
        gf, gr = ctx.pss_finish()
        gfp, gtp = ctx.fragkon_finish()
        assert ctx.stats() == st and ctx.fragkon_stats() == fst
        assert np.array_equal(gf, f) and np.array_equal(gr, r)
        assert np.array_equal(gfp, fp) and np.array_equal(gtp, tp)


def test_line_longer_than_the_staging_buffer(small):
    """pssgpu_feed stages 68 MiB at a time; a longer "line" is cut at a multiple of fgets' 200000 bytes
    (pss-bam.c:761-764) so that the stretches the kernel tallies are the ones line2saml would have been handed --
    among them one that happens to be a good record."""
    g, ora, ctx = small
    good = Synth.sam(reads_cfg_config1(seed=9), g, 0, 50).split(b"\n")[:-1]
    n_pad = 360 * 200000                                                      # 72 MB, a multiple of the fgets stretch
    monster = b"q" * n_pad + good[3] + b"\tXX:Z:" + b"t" * 1000               # ... so this tail parses as a record
    sam = b"\n".join(good[:10]) + b"\n" + monster + b"\n" + b"\n".join(good[10:]) + b"\n"
    f, r, st = ora.pss(sam, PssParams())
    assert st["lines"] == 50 + 360 + 1 and st["counted"] >= 45
    for chunk in (len(sam), 50_000_001):
        ctx.pss_begin(pkg.PssOptions())
        for off in range(0, len(sam), chunk):
            ctx.feed(sam[off:off + chunk], last=(off + chunk >= len(sam)))
        gf, gr = ctx.pss_finish()
        assert ctx.stats() == st
        assert np.array_equal(gf, f) and np.array_equal(gr, r)


def test_spectrum_hot_bins():
    """Low-complexity genome: poly-A, (CA)n and (CAG)n stretches put 10^6 .. 10^7 k-mers into single bins -- far beyond
    the 16-bit shared-memory counters of the k = 7..9 kernel, whose on-the-fly drain must stay exact -- next to N runs
    and contig ends; 64-bit global bins (PSSGPU_SPECTRUM_WIDE) give the same."""
    import os
    g = Synth.genome(71, [9_000_000, 6_000_000, 1_000_003], n_frac=0.01, lower_frac=0.02)
    for s, (at, n, motif) in zip(g.seqs, [(1_000_000, 5_000_000, b"A"), (500_000, 4_000_000, b"CA"), (1000, 700_000, b"CAG")]):
        s[at:at + n] = np.frombuffer((motif * (n // len(motif) + 1))[:n], dtype=np.uint8)
    g.seqs[0][3_000_000:3_000_040] = np.frombuffer(b"N" * 40, dtype=np.uint8)          # an N run inside the poly-A stretch
    ora = Oracle(contigs=list(zip(g.names, g.seqs)))
    ctx = pkg.Context(0)
    ctx.upload_genome(list(zip(g.names, g.seqs)))
    for k in (6, 7, 8, 9, 10):
        want = ora.kmer_spectrum(k)
        assert int(want.max()) > 3_000_000
        assert np.array_equal(ctx.kmer_spectrum(k), want), k
        assert np.array_equal(sum(ctx.kmer_spectrum(k, s, 5) for s in range(5)), want), k
        os.environ["PSSGPU_SPECTRUM_WIDE"] = "1"
        try:
            assert np.array_equal(ctx.kmer_spectrum(k), want), k
        finally:
            del os.environ["PSSGPU_SPECTRUM_WIDE"]
    ctx.close()
