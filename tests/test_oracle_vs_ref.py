"""Oracle vs the UNMODIFIED reference binaries (oracle/_ref, built by `make -C oracle ref REF=<reference sources>`).
Runs where those binaries exist; elsewhere the committed golden fixtures (test_oracle_golden.py) pin the oracle.
Fresh seeded inputs, including malformed lines, byte-compared."""
import os
import random

import numpy as np
import pytest

from pss_testlib import FkParams, Oracle, PssParams, RefBin, Synth, reads_cfg_config1, reads_cfg_config2, tmpdir
from test_record_logic import _mutate

pytestmark = pytest.mark.skipif(not RefBin.available(), reason=RefBin.MISSING)


@pytest.fixture(scope="module")
def world():
    g = Synth.genome(41, [50000, 30000, 900], names=["chr1", "chr2", "chrM"], n_frac=0.02, lower_frac=0.05)
    g.seqs[1][700:710] = np.frombuffer(b"RYKMSWBDHV", dtype=np.uint8)
    d = tmpdir()
    fa = g.fasta_bytes()
    open(os.path.join(d, "genome.fa"), "wb").write(fa)
    ora = Oracle(fasta=fa)
    yield g, ora, d
    ora.close()


def _strip_headers(sam):
    return b"".join(ln + b"\n" for ln in sam.split(b"\n")[:-1] if not ln.startswith(b"@"))


def _pss_vs_ref(ora, d, sam, p=PssParams(), name="reads.sam"):
    open(os.path.join(d, name), "wb").write(sam)
    counts, rates = RefBin.pss_bam("genome.fa", name, "ref", extra=p.cli_args(), cwd=d)
    fwd, rev, st = ora.pss(_strip_headers(sam), p)
    cwd = os.getcwd()
    os.chdir(d)
    try:
        ora.write_pss("genome.fa", name, "ref", fwd, rev, p.region_len)
        assert open("ref.pss.counts.txt", "rb").read() == counts
        assert open("ref.pss.rates.txt", "rb").read() == rates
    finally:
        os.chdir(cwd)
    return st


@pytest.mark.parametrize("p", [PssParams(), PssParams(region_len=7, min_len=35, max_len=100, min_mq=13),
                               PssParams(up_ctx=b"CTN", down_ctx=b"AGR"), PssParams(merged_only=1), PssParams(region_len=25)],
                         ids=repr)
def test_pss_random_reads(world, p):
    g, ora, d = world
    st = _pss_vs_ref(ora, d, Synth.sam(reads_cfg_config2(seed=5, min_len=20, max_len=150), g, 0, 6000), p)
    assert st["counted"] > 500


def test_pss_config1(world):
    g, ora, d = world
    _pss_vs_ref(ora, d, Synth.sam(reads_cfg_config1(seed=6), g, 0, 5000))


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_pss_malformed_lines_against_the_real_sscanf(world, seed):
    """Mutated records through the reference binary itself.  Mutations that overflow its fixed buffers (tokens
    > 2047 bytes, TLEN large enough to blow its stack, NUL bytes fgets cannot see past) are left out: the oracle
    reports those as 'undefined'."""
    g, ora, d = world
    rng = random.Random(seed)
    good = Synth.sam(reads_cfg_config2(seed=seed, min_len=20, max_len=70), g, 0, 2500).split(b"\n")[:-1]
    lines = []
    for ln in good:
        if rng.random() < 0.6:
            m = _mutate(rng, ln)
            if len(m) > 1500 or b"\x00" in m or b"2000000000" in m or b"0x7fffffff" in m or b"-2147483648" in m or m.startswith(b"@"):
                m = ln
            lines.append(m)
        else:
            lines.append(ln)
    st = _pss_vs_ref(ora, d, b"\n".join(lines) + b"\n")
    assert st["undefined"] < 30 and st["parse_fail"] > 50      # undefined here: paired TLEN just above 1e6 (the reference survives those)


@pytest.mark.parametrize("K", [1, 2, 3, 4, 5, 6, 7, 8])
def test_fragkon_random_reads(world, K):
    g, ora, d = world
    sam = Synth.sam(reads_cfg_config2(seed=20 + K, min_len=10, max_len=120), g, 0, 4000)
    open(os.path.join(d, "fk.sam"), "wb").write(sam)
    p = FkParams(klen=K, min_mq=10 if K % 3 == 0 else 0, merged_only=K % 2)
    want = RefBin.fragkon("genome.fa", "fk.sam", extra=p.cli_args(), cwd=d)
    fp, tp, st = ora.fragkon(sam, p)
    import ctypes as C
    lib = ora.lib()
    libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p
    libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    libc.fclose.argtypes = [C.c_void_p]
    lib.ora_fragkon_write.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_int, C.c_void_p, C.c_void_p]
    fn = os.path.join(d, "fk_out.txt").encode()
    f = libc.fopen(fn, b"w")
    lib.ora_fragkon_write(f, b"genome.fa", b"fk.sam", K, fp.ctypes.data, tp.ctypes.data)
    libc.fclose(f)
    assert open(fn, "rb").read() == want


def test_fragkon_k_above_8_with_stdbuf(world):
    g, ora, d = world
    sam = Synth.sam(reads_cfg_config2(seed=77, min_len=20, max_len=100), g, 0, 3000)
    open(os.path.join(d, "fk9.sam"), "wb").write(sam)
    out = RefBin.fragkon("genome.fa", "fk9.sam", extra=["-k", "9"], cwd=d)     # crashes in destroy_KSP after printing
    assert out.count(b"\n") == 4 ** 9 + 4
    fp, tp, _ = ora.fragkon(sam, FkParams(klen=9))
    rows = out.split(b"\n")[4:-1]
    got5 = np.array([int(r.split(b"\t")[1]) for r in rows], dtype=np.uint64)
    got3 = np.array([int(r.split(b"\t")[2]) for r in rows], dtype=np.uint64)
    assert np.array_equal(got5, fp) and np.array_equal(got3, tp)


@pytest.mark.parametrize("k", [1, 4, 8, 10])
def test_genome_kmer_count(world, k):
    g, ora, d = world
    out = RefBin.genome_kmer_count("genome.fa", k, cwd=d)
    rows = out.split(b"\n")
    assert rows[0] == f"Parsed input genome. Found {ora.n_contigs} sequences.".encode()
    got = np.array([int(r.split(b"\t")[1]) for r in rows[1:-1]], dtype=np.uint64)
    assert np.array_equal(got, ora.kmer_spectrum(k))
