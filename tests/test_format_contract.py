"""Format contract with the consumers of the two pss-bam tables (SURVEY 4.2 / 8f-4).

The reference's `pss-bam-plot.py:37-71` (`get_counts`, `get_rates`) and `pss-bam-gnuplot-template.gp:45-80` are what
reads `<prefix>.pss.counts.txt` / `<prefix>.pss.rates.txt`.  Their parsing is restated here call for call (same pandas
calls, same arguments -- matplotlib and gnuplot are not in the image, and the plotting itself is out of scope) and run
over files written by THIS repo's table writers (host/pss_tables.c, no GPU needed) for -r 5 / 15 / 30, and over the
reference's own golden files:

  * a line starting "### Reverse" separates the blocks; every other header line starts with '#'
  * counts: R+2 rows per block, 1 label + 16 count columns (AA AC .. TT), white-space separated, trailing tab
  * rates:  R rows per block, 1 label + 12 rate columns (AC AG AT CA CG CT GA GC GT TA TC TG)
  * the reverse block runs R-1 .. 0, then the context rows "1", "2"  (plot: index = arange(R-1, -3, -1))
  * gnuplot: two data blocks (`index 0` / `index 1`) = two blank lines between them, columns $1..$17
"""
import ctypes as C
import json
import os
import re
import subprocess

import numpy as np
import pandas as pd
import pytest

from pss_testlib import parse_counts_file, tmpdir

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "pss-bam_b200", "host")
GOLD = os.path.join(ROOT, "tests", "golden", "v1")
MAN = json.load(open(os.path.join(GOLD, "manifest.json")))
SO = os.path.join(ROOT, "tests", "host_emul", "libpsshostapi_fmt.so")

# pss-bam-plot.py:16-20
nt_pairs = ["AA", "AC", "AG", "AT", "CA", "CC", "CG", "CT", "GA", "GC", "GG", "GT", "TA", "TC", "TG", "TT"]
sub_pairs = [p for p in nt_pairs if p not in ["AA", "CC", "GG", "TT"]]


def _skip_to_reverse(fn):
    """pss-bam-plot.py:38-44 / :59-65"""
    with open(fn, "r") as f:
        n_skip = 0
        line = f.readline()
        while line and not line.startswith("### Reverse"):
            n_skip += 1
            line = f.readline()
        assert line, "no line starting with '### Reverse'"
        return n_skip + 1


def get_counts(counts_fn, region_len):
    """pss-bam-plot.py:37-55"""
    n_skip = _skip_to_reverse(counts_fn)
    fp_df = pd.read_table(counts_fn, sep=r"\s+", comment="#", names=nt_pairs, nrows=region_len + 2)
    tp_df = pd.read_table(counts_fn, sep=r"\s+", skiprows=n_skip, names=nt_pairs, nrows=region_len + 2)
    tp_df.index = np.arange(region_len - 1, -3, -1)
    for df in [fp_df, tp_df]:
        df["A"] = df["AA"] + df["AC"] + df["AG"] + df["AT"]
        df["C"] = df["CA"] + df["CC"] + df["CG"] + df["CT"]
        df["G"] = df["GA"] + df["GC"] + df["GG"] + df["GT"]
        df["T"] = df["TA"] + df["TC"] + df["TG"] + df["TT"]
    return fp_df, tp_df


def get_rates(rates_fn, region_len):
    """pss-bam-plot.py:58-71"""
    n_skip = _skip_to_reverse(rates_fn)
    fp_df = pd.read_table(rates_fn, sep=r"\s+", comment="#", names=sub_pairs, nrows=region_len, dtype=float)
    tp_df = pd.read_table(rates_fn, sep=r"\s+", skiprows=n_skip, names=sub_pairs, nrows=region_len, dtype=float)
    tp_df.index = np.arange(region_len - 1, -1, -1)
    return fp_df, tp_df


def gnuplot_blocks(fn):
    """gnuplot's data-file rules as the template relies on them: '#' starts a comment line, a run of two or more
    blank lines starts a new `index`, columns are white-space separated."""
    blocks, cur, blanks = [], [], 0
    for ln in open(fn).read().split("\n"):
        if ln.startswith("#"):
            continue
        if ln.strip() == "":
            blanks += 1
            continue
        if blanks >= 2 and cur:
            blocks.append(cur)
            cur = []
        blanks = 0
        cur.append(ln.split())
    if cur:
        blocks.append(cur)
    return blocks


@pytest.fixture(scope="module")
def lib():
    srcs = [os.path.join(HOST, f) for f in ("pss_tables.c",)]
    subprocess.run(["gcc", "-O2", "-g", "-std=gnu11", "-Wall", "-fPIC", "-shared", "-o", SO, *srcs], check=True)
    h = C.CDLL(SO)
    h.pss_sub_rates.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    h.pss_write_counts.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_int]
    h.pss_write_rates.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_int]
    return h


def _check_files(counts_fn, rates_fn, R, fwd, rev, fr, rr):
    # ---- pss-bam-plot.py
    fp, tp = get_counts(counts_fn, R)
    assert fp.shape == (R + 2, 20) and tp.shape == (R + 2, 20)          # 16 pairs + A C G T
    assert list(fp.index) == list(range(-2, R))                         # label column became the index
    assert np.array_equal(fp[nt_pairs].to_numpy(dtype=np.uint64), fwd)
    # reverse block: rows R-1 .. 0 (table rows R+1 .. 2), then "1" (row 1) and "2" (row 0); the plot indexes it R-1 .. -2
    want_tp = np.concatenate([rev[2:][::-1], rev[1:2], rev[0:1]])
    assert np.array_equal(tp[nt_pairs].to_numpy(dtype=np.uint64), want_tp)
    assert list(tp.index) == list(range(R - 1, -3, -1))
    assert np.array_equal(fp["C"].to_numpy(dtype=np.uint64), fwd[:, 4:8].sum(axis=1))
    fpr, tpr = get_rates(rates_fn, R)
    assert fpr.shape == (R, 12) and tpr.shape == (R, 12)
    assert list(fpr.index) == list(range(R)) and list(tpr.index) == list(range(R - 1, -1, -1))
    # "%.5e" text: equal to the doubles after the same rounding
    assert np.array_equal(fpr.to_numpy(), np.array([[float("%.5e" % x) for x in row] for row in fr]))
    assert np.array_equal(tpr.to_numpy(), np.array([[float("%.5e" % x) for x in row] for row in rr[::-1]]))
    # ---- gnuplot template: two blocks, 17 columns ($1 = position, $2..$17 = AA..TT), ($1+2) = table row in block 0
    cb = gnuplot_blocks(counts_fn)
    assert len(cb) == 2 and all(len(b) == R + 2 for b in cb) and all(len(r) == 17 for b in cb for r in b)
    assert [int(r[0]) + 2 for r in cb[0]] == list(range(R + 2))
    assert [int(r[0]) for r in cb[1]] == list(range(R - 1, -1, -1)) + [1, 2]
    rb = gnuplot_blocks(rates_fn)
    assert len(rb) == 2 and all(len(b) == R for b in rb) and all(len(r) == 13 for b in rb for r in b)
    # ---- raw layout the two parsers lean on
    text = open(counts_fn).read()
    assert len(re.findall(r"(?m)^### Reverse", text)) == 1
    body = [ln for ln in text.split("\n") if ln and not ln.startswith("#")]
    assert all(ln.endswith("\t") for ln in body)                         # "%lu\t" per cell (pss-bam.c:559-563)
    assert "\n\n\n" in text                                              # pss-bam.c:566


@pytest.mark.parametrize("R", [5, 15, 30])
def test_consumers_parse_our_tables(lib, R):
    rng = np.random.default_rng(R)
    fwd = rng.integers(0, 5_000_000_000, size=(R + 2, 16), dtype=np.uint64)   # beyond 32 bits on purpose
    rev = rng.integers(0, 3_000_000, size=(R + 2, 16), dtype=np.uint64)
    for t in (fwd, rev):                       # context rows only ever hold diagonal cells (pss-bam.c:169-189)
        for c in range(16):
            if c not in (0, 5, 10, 15):
                t[0, c] = t[1, c] = 0
    rev[5, 1] = rev[5, 5] = rev[5, 9] = rev[5, 13] = 0       # a reference base never seen: the row's rates stay 0
    fr = np.zeros((R, 12))
    rr = np.zeros((R, 12))
    lib.pss_sub_rates(fwd.ctypes.data, R, fr.ctypes.data)
    lib.pss_sub_rates(rev.ctypes.data, R, rr.ctypes.data)
    assert not rr[3].any()
    d = tmpdir()
    prefix = os.path.join(d, "out").encode()
    assert lib.pss_write_counts(b"genome.fa", b"reads.bam", prefix, fwd.ctypes.data, rev.ctypes.data, R) == 0
    assert lib.pss_write_rates(b"genome.fa", b"reads.bam", prefix, fr.ctypes.data, rr.ctypes.data, R) == 0
    _check_files(prefix.decode() + ".pss.counts.txt", prefix.decode() + ".pss.rates.txt", R, fwd, rev, fr, rr)


@pytest.mark.parametrize("case", MAN["pss"], ids=lambda c: c["sam"] + "".join(c["args"]))
def test_consumers_parse_reference_goldens(lib, case):
    """The same parsers over the files the unmodified reference wrote (tests/golden/v1): pins the restated parsing to
    the reference's real output, for every -r in the golden set."""
    R = 15
    if "-r" in case["args"]:
        R = int(case["args"][case["args"].index("-r") + 1])
    if R < 1:
        pytest.skip("-r 0: pandas has nothing to parse (the plot script needs at least one interior row)")
    counts_fn, rates_fn = os.path.join(GOLD, case["counts"]), os.path.join(GOLD, case["rates"])
    fwd, rev = parse_counts_file(open(counts_fn, "rb").read(), R)
    fr = np.zeros((R, 12))
    rr = np.zeros((R, 12))
    lib.pss_sub_rates(fwd.ctypes.data, R, fr.ctypes.data)
    lib.pss_sub_rates(rev.ctypes.data, R, rr.ctypes.data)
    _check_files(counts_fn, rates_fn, R, fwd, rev, fr, rr)
