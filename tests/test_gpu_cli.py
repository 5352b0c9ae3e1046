"""The three host programs (pss-bam_b200/bin, C host + libpssgpu.so) against the reference's golden outputs:
same command lines, byte-identical files / stdout."""
import json
import os
import subprocess
import time

import pytest

from pss_testlib import REF_DIR, tmpdir

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "v1")
MAN = json.load(open(os.path.join(GOLD, "manifest.json")))
BIN = os.path.join(ROOT, "pss-bam_b200", "bin")
SHIM = os.path.join(ROOT, "oracle", "samtools_shim.sh")


@pytest.fixture(scope="module")
def env():
    import importlib
    importlib.import_module("pss-bam_b200").build_library()
    subprocess.run(["make", "-C", os.path.join(ROOT, "pss-bam_b200", "host")], check=True, capture_output=True)
    d = tmpdir()
    shim = os.path.join(d, "samtools")            # `samtools view` stand-in (samtools is not in the image)
    with open(SHIM) as f, open(shim, "w") as o:
        o.write(f.read())
    os.chmod(shim, 0o755)
    e = dict(os.environ)
    e["PATH"] = d + os.pathsep + e.get("PATH", "")
    for fn in [MAN["fasta"], *MAN["sams"].values()]:
        os.symlink(os.path.join(GOLD, fn), os.path.join(d, fn))
    return d, e


def _gold(name):
    return open(os.path.join(GOLD, name), "rb").read()


@pytest.mark.parametrize("case", MAN["pss"], ids=lambda c: c["sam"] + "".join(c["args"]))
def test_pss_bam_cli(env, case):
    d, e = env
    r = subprocess.run([os.path.join(BIN, "pss-bam"), "-F", "genome.fa", "-B", case["sam"] + ".sam", "-o", "out", *case["args"]],
                       cwd=d, env=e, capture_output=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert open(os.path.join(d, "out.pss.counts.txt"), "rb").read() == _gold(case["counts"])
    assert open(os.path.join(d, "out.pss.rates.txt"), "rb").read() == _gold(case["rates"])


@pytest.mark.parametrize("case", MAN["fragkon"], ids=lambda c: c["sam"] + "".join(c["args"]))
def test_fragkon_cli(env, case):
    d, e = env
    r = subprocess.run([os.path.join(BIN, "fragkon"), "-F", "genome.fa", "-B", case["sam"] + ".sam", *case["args"]],
                       cwd=d, env=e, capture_output=True)
    assert r.returncode == 0, r.stderr[-2000:]
    out = r.stdout
    if case["sparse"]:
        lines = out.split(b"\n")
        out = b"\n".join(lines[:4] + [ln for ln in lines[4:] if ln and not ln.endswith(b"\t0\t0")]) + b"\n"
    assert out == _gold(case["out"])


@pytest.mark.parametrize("case", MAN["gkc"], ids=lambda c: f"k{c['k']}")
def test_genome_kmer_count_cli(env, case):
    d, e = env
    r = subprocess.run([os.path.join(BIN, "genome-kmer-count"), "-f", "genome.fa", "-k", str(case["k"])],
                       cwd=d, env=e, capture_output=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout == _gold(case["out"])


def test_cli_with_packed_genome_cache(env):
    """$PSSGPU_GENOME_CACHE: the first run writes <dir>/genome.fa.<hash of realpath>.pssgpu, the second one loads it
    instead of parsing the FASTA -- same bytes.  A damaged cache, a cache whose FASTA changed since (size / mtime tag)
    and a cache of another FASTA of the same basename are all refused and the FASTA is parsed again."""
    import glob
    import shutil
    d0, e = env
    case = MAN["pss"][0]
    # copies, not the links to tests/golden: the test changes the FASTA's mtime
    d = os.path.join(d0, "cached")
    os.makedirs(d, exist_ok=True)
    for fn in (MAN["fasta"], case["sam"] + ".sam"):
        shutil.copy(os.path.join(d0, fn), d)
    cdir = os.path.join(d, "cache")
    shutil.rmtree(cdir, ignore_errors=True)
    os.makedirs(cdir)
    e2 = dict(e, PSSGPU_GENOME_CACHE=cdir)
    cmd = [os.path.join(BIN, "pss-bam"), "-F", "genome.fa", "-B", case["sam"] + ".sam", "-o", "out", *case["args"]]

    def caches():
        return sorted(glob.glob(os.path.join(cdir, "genome.fa.*.pssgpu")))

    def check_outputs(where=d):
        assert open(os.path.join(where, "out.pss.counts.txt"), "rb").read() == _gold(case["counts"])
        assert open(os.path.join(where, "out.pss.rates.txt"), "rb").read() == _gold(case["rates"])

    for rnd in range(2):
        r = subprocess.run(cmd, cwd=d, env=e2, capture_output=True)
        assert r.returncode == 0, r.stderr[-2000:]
        assert len(caches()) == 1 and b"ignoring genome cache" not in r.stderr
        check_outputs()
    cache = caches()[0]
    gk = MAN["gkc"][0]
    r = subprocess.run([os.path.join(BIN, "genome-kmer-count"), "-f", "genome.fa", "-k", str(gk["k"])], cwd=d, env=e2, capture_output=True)
    assert r.returncode == 0 and r.stdout == _gold(gk["out"])
    # the FASTA is touched (newer mtime): the tag no longer matches, the cache is refused and rewritten
    os.utime(os.path.join(d, "genome.fa"), ns=(time.time_ns(), time.time_ns() + 5_000_000_000))
    r = subprocess.run(cmd, cwd=d, env=e2, capture_output=True)
    assert r.returncode == 0 and b"ignoring genome cache" in r.stderr and b"different source" in r.stderr
    check_outputs()
    r = subprocess.run(cmd, cwd=d, env=e2, capture_output=True)
    assert r.returncode == 0 and b"ignoring genome cache" not in r.stderr
    # a damaged cache is refused (with a warning) and the FASTA is parsed again
    with open(cache, "r+b") as f:
        f.truncate(1000)
    r = subprocess.run(cmd, cwd=d, env=e2, capture_output=True)
    assert r.returncode == 0 and b"ignoring genome cache" in r.stderr
    check_outputs()
    # a table entry out of range (contig 0's base offset) is caught by the range checks, not by a kernel fault
    r = subprocess.run(cmd, cwd=d, env=e2, capture_output=True)
    assert r.returncode == 0 and b"ignoring genome cache" not in r.stderr
    with open(cache, "r+b") as f:
        f.seek(8 + 6 * 8 + 4 * 4 + 4 * 8)         # CacheHeader: magic, six u64, four u32, the tag -> first DevContig
        f.write((1 << 50).to_bytes(8, "little"))
    r = subprocess.run(cmd, cwd=d, env=e2, capture_output=True)
    assert r.returncode == 0 and b"damaged" in r.stderr
    check_outputs()
    # another FASTA with the same basename in another directory gets its own cache file (the path hash keys the name)
    d2 = os.path.join(d, "other")
    os.makedirs(d2, exist_ok=True)
    with open(os.path.join(d2, "genome.fa"), "wb") as f:
        f.write(b">zz\n" + b"ACGT" * 100 + b"\n")
    shutil.copy(os.path.join(d, case["sam"] + ".sam"), d2)
    r = subprocess.run(cmd, cwd=d2, env=e2, capture_output=True)
    assert r.returncode == 0 and len(caches()) == 2
    r = subprocess.run(cmd, cwd=d, env=e2, capture_output=True)
    assert r.returncode == 0 and b"ignoring genome cache" not in r.stderr
    check_outputs()


@pytest.mark.parametrize("prog", ["pss-bam", "fragkon"])
def test_cli_reads_real_bam_files(env, prog):
    """-B with a real BAM (BGZF) file: decoded on the GPU, no samtools on PATH at all -- byte-identical outputs to the
    golden files the reference wrote from the same alignments as SAM text; -R through the native filter."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from pss_testlib import Synth
    d, e = env
    e2 = dict(e, PATH="/usr/bin:/bin")                     # no samtools shim
    refs = []
    name = None
    for ln in open(os.path.join(GOLD, MAN["fasta"]), "rb").read().split(b"\n"):
        if ln.startswith(b">"):
            name = ln[1:].split()[0].decode()
            refs.append([name, 0])
        elif name:
            refs[-1][1] += len(ln.strip())
    refs.append(["chrUn_synthetic_decoy", 1000])
    cases = MAN["pss"][:4] if prog == "pss-bam" else MAN["fragkon"][:4]
    done = 0
    for case in cases:
        sam = open(os.path.join(GOLD, case["sam"] + ".sam"), "rb").read()
        try:
            bam = Synth.bam(sam, refs, block_payload=3000)
        except RuntimeError:
            continue                                        # the edge corpus holds lines no BAM can represent
        done += 1
        # same file NAME as in the golden run (the headers of the outputs embed it), BAM content
        bam_fn = os.path.join(d, "bamdir_" + prog, case["sam"] + ".sam")
        os.makedirs(os.path.dirname(bam_fn), exist_ok=True)
        with open(bam_fn, "wb") as f:
            f.write(bam)
        wd = os.path.dirname(bam_fn)
        if not os.path.exists(os.path.join(wd, "genome.fa")):
            os.symlink(os.path.join(GOLD, MAN["fasta"]), os.path.join(wd, "genome.fa"))
        if prog == "pss-bam":
            r = subprocess.run([os.path.join(BIN, "pss-bam"), "-F", "genome.fa", "-B", case["sam"] + ".sam", "-o", "out", *case["args"]],
                               cwd=wd, env=e2, capture_output=True)
            assert r.returncode == 0, r.stderr[-2000:]
            assert open(os.path.join(wd, "out.pss.counts.txt"), "rb").read() == _gold(case["counts"])
            assert open(os.path.join(wd, "out.pss.rates.txt"), "rb").read() == _gold(case["rates"])
        else:
            r = subprocess.run([os.path.join(BIN, "fragkon"), "-F", "genome.fa", "-B", case["sam"] + ".sam", *case["args"]],
                               cwd=wd, env=e2, capture_output=True)
            assert r.returncode == 0, r.stderr[-2000:]
            assert not case["sparse"] and r.stdout == _gold(case["out"]), case
    assert done >= 2


def test_cli_bam_file_in_pieces_and_by_parallel_reads(env):
    """The BAM reader of the host programs: 1 MiB pieces (BGZF blocks cut by every piece boundary) read with three
    concurrent pread()s, and plain fread()s, against the samtools-shim text path on the same alignments."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from pss_testlib import Synth, reads_cfg_config2
    d, e = env
    g = Synth.genome(61, [500_000, 250_000], n_frac=0.01, lower_frac=0.03)
    sam = Synth.sam(reads_cfg_config2(seed=62), g, 0, 60_000)
    bam = Synth.bam(sam, list(zip(g.names, g.lens)) + [("chrUn_synthetic_decoy", 1000)], level=6, qual_mode=1)
    assert len(bam) > (3 << 20)
    outs = []
    for k, (content, extra) in enumerate(((sam, {}), (bam, {"PSS_BAM_CHUNK_MB": "1", "PSS_READ_THREADS": "3"}),
                                          (bam, {"PSS_BAM_CHUNK_MB": "1", "PSS_READ_THREADS": "0"}), (bam, {}))):
        wd = os.path.join(d, f"pieces_{k}")
        os.makedirs(wd)
        with open(os.path.join(wd, "genome.fa"), "wb") as f:
            f.write(g.fasta_bytes())
        with open(os.path.join(wd, "reads.bam"), "wb") as f:
            f.write(content)
        r = subprocess.run([os.path.join(BIN, "pss-bam"), "-F", "genome.fa", "-B", "reads.bam", "-o", "out"], cwd=wd, env=dict(e, **extra),
                           capture_output=True)
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append((open(os.path.join(wd, "out.pss.counts.txt"), "rb").read(), open(os.path.join(wd, "out.pss.rates.txt"), "rb").read()))
    assert outs[0][0].count(b"\n") > 30 and all(o == outs[0] for o in outs[1:])
