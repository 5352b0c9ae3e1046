#!/usr/bin/env python3
"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference programs.

Needs oracle/_ref (built by `make -C oracle ref REF=<dir>` from the reference's sources, which this repository
does not carry).  Inputs come from the seeded generators in tests/synth plus a hand-written edge-case corpus (the cases
SURVEY.md section 8c lists); outputs are whatever the reference binaries print.  Everything written here is
committed, so the CPU test-suite can pin the oracle on machines without the reference.

    python tests/golden/make_golden.py
"""
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from pss_testlib import RefBin, Synth, reads_cfg_config1, reads_cfg_config2  # noqa: E402


def edge_corpus(g):
    """Hand-written records around every filter boundary (SURVEY 8c).  chrA = g.seqs[0] (3000 bp)."""
    s0 = g.seqs[0].tobytes().upper()
    L = len(s0)

    def rec(name, flag, rname, pos, mapq, cigar, tlen, seq, qual=None, mrnm=b"*", mpos=0, tags=b""):
        qual = (b"I" * len(seq)) if qual is None else qual
        f = [name, str(flag).encode(), rname, str(pos).encode(), str(mapq).encode(), cigar, mrnm, str(mpos).encode(),
             str(tlen).encode(), seq, qual]
        ln = b"\t".join(f)
        return ln + (b"\t" + tags if tags else b"")

    def rc(b):
        return b[::-1].translate(bytes.maketrans(b"ACGT", b"TGCA"))

    out = []
    rd = lambda pos, n: s0[pos - 1:pos - 1 + n]                                        # noqa: E731
    n = 30
    out.append(rec(b"ok_fwd", 0, b"chrA", 100, 30, b"30M", 0, rd(100, n)))
    out.append(rec(b"ok_rev", 16, b"chrA", 200, 30, b"30M", 0, rd(200, n)))
    out.append(rec(b"qual_star", 0, b"chrA", 100, 30, b"30M", 0, rd(100, n), qual=b"*"))
    out.append(rec(b"space_sep", 0, b"chrA", 300, 30, b"30M", 0, rd(300, n)).replace(b"\t", b" "))
    out.append(rec(b"crlf", 0, b"chrA", 310, 30, b"30M", 0, rd(310, n)) + b"\r")
    out.append(rec(b"dup", 1024, b"chrA", 320, 30, b"30M", 0, rd(320, n)))
    out.append(rec(b"cig_eq", 0, b"chrA", 330, 30, b"30=", 0, rd(330, n)))
    out.append(rec(b"cig_split", 0, b"chrA", 340, 30, b"15M15M", 0, rd(340, n)))
    out.append(rec(b"cig_zero", 0, b"chrA", 350, 30, b"030M", 0, rd(350, n)))
    out.append(rec(b"cig_clip", 0, b"chrA", 360, 30, b"5S25M", 0, rd(360, n)))
    out.append(rec(b"unknown", 0, b"chrZ", 100, 30, b"30M", 0, rd(100, n)))
    out.append(rec(b"pos2", 0, b"chrA", 2, 30, b"30M", 0, rd(2, n)))
    out.append(rec(b"pos3", 0, b"chrA", 3, 30, b"30M", 0, rd(3, n)))
    out.append(rec(b"end_ok", 0, b"chrA", L - 2 - n + 1, 30, b"30M", 0, rd(L - 2 - n + 1, n)))   # e+2 == len-1
    out.append(rec(b"end_bad", 0, b"chrA", L - 1 - n + 1, 30, b"30M", 0, rd(L - 1 - n + 1, n)))
    out.append(rec(b"n14", 0, b"chrA", 400, 30, b"14M", 0, rd(400, 14)))
    out.append(rec(b"n15", 0, b"chrA", 410, 30, b"15M", 0, rd(410, 15)))
    out.append(rec(b"hexflag", b"0x10".decode(), b"chrA", 420, 30, b"30M", 0, rd(420, n)))
    out.append(rec(b"negpos", 0, b"chrA", -5, 30, b"30M", 0, rd(100, n)))
    out.append(rec(b"r1_ok", 99, b"chrA", 500, 30, b"30M", 30, rd(500, n), mrnm=b"=", mpos=500))
    out.append(rec(b"r1_tlen", 99, b"chrA", 510, 30, b"30M", 180, rd(510, n), mrnm=b"=", mpos=660))
    out.append(rec(b"r2_ok", 147, b"chrA", 520, 30, b"30M", -30, rd(520, n), mrnm=b"=", mpos=520))
    out.append(rec(b"r2_fwd", 163, b"chrA", 530, 30, b"30M", 30, rd(530, n), mrnm=b"=", mpos=530))
    out.append(rec(b"r1_rev", 83, b"chrA", 540, 30, b"30M", -30, rd(540, n), mrnm=b"=", mpos=540))
    out.append(rec(b"pair_notproper", 65, b"chrA", 550, 30, b"30M", 30, rd(550, n), mrnm=b"=", mpos=550))
    out.append(rec(b"pair_munmap", 73, b"chrA", 560, 30, b"30M", 30, rd(560, n), mrnm=b"=", mpos=560))
    out.append(rec(b"lower", 0, b"chrA", 600, 30, b"30M", 0, rd(600, n).lower()))
    out.append(rec(b"read_n", 0, b"chrA", 610, 30, b"30M", 0, rd(610, 3) + b"N" + rd(614, n - 4)))
    out.append(rec(b"mq5", 0, b"chrA", 620, 5, b"30M", 0, rd(620, n)))
    out.append(rec(b"mq9", 0, b"chrA", 630, 9, b"30M", 0, rd(630, n)))
    out.append(rec(b"tags", 0, b"chrA", 640, 30, b"30M", 0, rd(640, n), tags=b"NM:i:0\tMD:Z:30\tRG:Z:lib1"))
    out.append(rec(b"tags2", 16, b"chrA", 650, 30, b"30M", 0, rd(650, n), tags=b"NM:i:0\tRG:Z:lib2"))
    out.append(rec(b"long", 0, b"chrA", 700, 60, b"150M", 0, rd(700, 150)))
    out.append(rec(b"unmapped", 4, b"chrA", 710, 0, b"30M", 0, rd(710, n)))
    out.append(rec(b"secondary", 256, b"chrA", 720, 30, b"30M", 0, rd(720, n)))
    out.append(rec(b"qcfail", 512, b"chrA", 730, 30, b"30M", 0, rd(730, n)))
    out.append(rec(b"supp", 2048, b"chrA", 740, 30, b"30M", 0, rd(740, n)))
    out.append(b"@HD\tVN:1.6\tSO:coordinate")
    out.append(b"")
    out.append(rec(b"few_fields", 0, b"chrA", 750, 30, b"30M", 0, rd(750, n)).rsplit(b"\t", 3)[0])
    out.append(rec(b"flag_garbage", b"0x".decode(), b"chrA", 760, 30, b"30M", 0, rd(760, n)))
    out.append(rec(b"near_start_rev", 16, b"chrA", 4, 30, b"30M", 0, rd(4, n)))
    out.append(rec(b"pos0", 0, b"chrA", 0, 30, b"30M", 0, rd(1, n)))
    out.append(rec(b"pos1_rev", 16, b"chrA", 1, 30, b"30M", 0, rd(1, n)))
    out.append(rec(b"chrB_n", 0, b"chrB", 40, 30, b"30M", 0, g.seqs[1].tobytes().upper()[39:69].replace(b"N", b"A")))
    return b"\n".join(out) + b"\n"


def main():
    assert RefBin.available(), "build the reference first: make -C oracle ref"
    import numpy as np
    g = Synth.genome(20261018, [3000, 2000, 500], names=["chrA", "chrB", "chrC_short"], n_frac=0.03, lower_frac=0.1)
    # soft-masked + IUPAC codes in chrB so that -U/-D lists with non-ACGT letters have something to match
    b = g.seqs[1]
    b[100:104] = np.frombuffer(b"RYKM", dtype=np.uint8)
    fasta = g.fasta_bytes()
    sams = {
        "c1": Synth.sam(reads_cfg_config1(seed=101, read_len=50), g, 0, 300),
        "c2": Synth.sam(reads_cfg_config2(seed=102, min_len=30, max_len=150), g, 0, 800),
        "edge": edge_corpus(g),
    }
    pss_cases = [
        ("c1", []), ("c2", []), ("edge", []),
        ("c2", ["-r", "5", "-l", "40", "-L", "120", "-q", "20"]),
        ("c2", ["-U", "CT", "-D", "AGN"]),
        ("c2", ["-m"]),
        ("c2", ["-r", "30"]),
        ("edge", ["-q", "9"]), ("edge", ["-q", "10"]), ("edge", ["-m"]), ("edge", ["-r", "5"]), ("edge", ["-U", "A"]),
        ("edge", ["-R", "lib1"]),
    ]
    fk_cases = [("c1", ["-k", "3"]), ("c2", ["-k", "2"]), ("c2", ["-k", "3"]), ("c2", ["-k", "4", "-q", "20"]),
                ("c2", ["-k", "5", "-m"]), ("edge", ["-k", "3"]), ("edge", ["-k", "4"]), ("edge", ["-k", "1"]),
                ("c2", ["-k", "9", "-l", "60"])]
    gkc_cases = [1, 2, 3, 5]

    for name in os.listdir(HERE):
        p = os.path.join(HERE, name)
        if os.path.isdir(p):
            shutil.rmtree(p)
    work = os.path.join(HERE, "_work")
    os.makedirs(work)
    with open(os.path.join(work, "genome.fa"), "wb") as f:
        f.write(fasta)
    manifest = {"fasta": "genome.fa", "sams": {}, "pss": [], "fragkon": [], "gkc": []}
    for k, v in sams.items():
        with open(os.path.join(work, k + ".sam"), "wb") as f:
            f.write(v)
        manifest["sams"][k] = k + ".sam"

    for i, (sam, args) in enumerate(pss_cases):
        counts, rates = RefBin.pss_bam("genome.fa", sam + ".sam", "out", extra=args, cwd=work)
        cn, rn = f"pss_{i:02d}.counts.txt", f"pss_{i:02d}.rates.txt"
        open(os.path.join(work, cn), "wb").write(counts)
        open(os.path.join(work, rn), "wb").write(rates)
        manifest["pss"].append({"sam": sam, "args": args, "counts": cn, "rates": rn})
    for i, (sam, args) in enumerate(fk_cases):
        out = RefBin.fragkon("genome.fa", sam + ".sam", extra=args, cwd=work)
        fn = f"fragkon_{i:02d}.txt"
        k = int(args[args.index("-k") + 1])
        assert out.count(b"\n") == 4 ** k + 4, (args, out.count(b"\n"))
        if k > 6:   # keep the fixture small: non-zero rows only
            lines = out.split(b"\n")
            out = b"\n".join(lines[:4] + [ln for ln in lines[4:] if ln and not ln.endswith(b"\t0\t0")]) + b"\n"
        open(os.path.join(work, fn), "wb").write(out)
        manifest["fragkon"].append({"sam": sam, "args": args, "out": fn, "sparse": k > 6})
    for k in gkc_cases:
        out = RefBin.genome_kmer_count("genome.fa", k, cwd=work)
        fn = f"gkc_k{k}.txt"
        open(os.path.join(work, fn), "wb").write(out)
        manifest["gkc"].append({"k": k, "out": fn})

    for fn in ("out.pss.counts.txt", "out.pss.rates.txt"):
        os.remove(os.path.join(work, fn))
    os.rename(work, os.path.join(HERE, "v1"))
    with open(os.path.join(HERE, "v1", "manifest.json"), "w") as f:
        json.dump(manifest, f, indent=1)
    print("wrote", os.path.join(HERE, "v1"))


if __name__ == "__main__":
    main()
