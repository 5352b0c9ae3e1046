"""Shared test/bench helpers (NOT product code).

* ``Synth``  -- ctypes binding of tests/synth/libpsssynth.so (seeded FASTA/SAM generators)
* ``Oracle`` -- ctypes binding of oracle/liboracle.so (CPU restatement of the reference,
  see oracle/oracle_pss.h for who may use it)
* ``RefBin`` -- runner for the unmodified reference binaries in oracle/_ref (only when
  they exist; they are built from the reference's sources by ``make -C oracle ref REF=<dir>``)
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from dataclasses import dataclass, field

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SYNTH_SO = os.path.join(ROOT, "tests", "synth", "libpsssynth.so")
ORACLE_SO = os.path.join(ROOT, "oracle", "liboracle.so")
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def _run(cmd, **kw):
    r = subprocess.run(cmd, capture_output=True, text=True, **kw)
    if r.returncode != 0:
        raise RuntimeError(f"{' '.join(cmd)} failed:\n{r.stdout}\n{r.stderr}")
    return r


def _locked_build(target, newest, force, make_cmd):
    """Build `target` unless it is up to date: one process at a time (torchrun ranks, pytest-xdist workers), into a
    temporary file that is renamed into place -- nobody ever dlopens a half-written library."""
    import fcntl

    def fresh():
        return os.path.exists(target) and os.path.getsize(target) > 0 and os.path.getmtime(target) >= newest

    if not force and fresh():
        return target
    with open(target + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if force or not fresh():
                tmp = target + f".tmp{os.getpid()}"
                _run(make_cmd(tmp))
                os.replace(tmp, target)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return target


def build_synth(force=False):
    src = os.path.join(ROOT, "tests", "synth", "pss_synth.c")
    return _locked_build(SYNTH_SO, os.path.getmtime(src), force,
                         lambda out: ["gcc", "-O2", "-g", "-fopenmp", "-fPIC", "-shared", "-o", out, src, "-lm", "-lz"])


def build_oracle(force=False):
    src = os.path.join(ROOT, "oracle", "oracle_pss.c")
    hdr = os.path.join(ROOT, "oracle", "oracle_pss.h")
    newest = max(os.path.getmtime(src), os.path.getmtime(hdr))
    if force or not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < newest:
        _run(["make", "-C", os.path.join(ROOT, "oracle"), "-B", "liboracle.so"])
    return ORACLE_SO


# --------------------------------------------------------------------------- synth
class _ReadsCfg(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64),
        ("min_len", C.c_uint32), ("max_len", C.c_uint32),
        ("p_reverse", C.c_double), ("p_indel", C.c_double), ("p_softclip", C.c_double),
        ("p_badflag", C.c_double), ("p_paired", C.c_double), ("p_qualstar", C.c_double),
        ("p_unknown_contig", C.c_double), ("p_edge", C.c_double), ("p_read_n", C.c_double),
        ("damage5", C.c_double), ("damage3", C.c_double), ("err", C.c_double),
        ("max_mapq", C.c_uint32), ("with_tags", C.c_uint32), ("sorted_total", C.c_uint64),
    ]


def reads_cfg_config1(seed=1, read_len=50):
    """SURVEY 8(d) config 1: fixed-length unpaired reads, all '<n>M', damage + 0.2% errors."""
    return _ReadsCfg(seed=seed, min_len=read_len, max_len=read_len, p_reverse=0.5,
                     p_indel=0, p_softclip=0, p_badflag=0, p_paired=0, p_qualstar=0,
                     p_unknown_contig=0, p_edge=0, p_read_n=0,
                     damage5=0.3, damage3=0.3, err=0.002, max_mapq=60, with_tags=1)


def reads_cfg_config2(seed=2, min_len=30, max_len=150):
    """SURVEY 8(d) config 2: variable length, reject-path mix, paired mix."""
    return _ReadsCfg(seed=seed, min_len=min_len, max_len=max_len, p_reverse=0.5,
                     p_indel=0.10, p_softclip=0.10, p_badflag=0.05, p_paired=0.05,
                     p_qualstar=0.01, p_unknown_contig=0.005, p_edge=0.002, p_read_n=0.02,
                     damage5=0.3, damage3=0.3, err=0.002, max_mapq=60, with_tags=1)


@dataclass
class SynthGenome:
    names: list
    seqs: list            # list of np.uint8 arrays (ASCII, may contain lower case / N)
    seed: int = 0
    _keep: list = field(default_factory=list)

    @property
    def lens(self):
        return [len(s) for s in self.seqs]

    def fasta_bytes(self, width=60) -> bytes:
        lib = Synth.lib()
        out = []
        for name, seq in zip(self.names, self.seqs):
            cap = len(seq) + len(seq) // width + len(name) + 8
            buf = np.empty(cap, dtype=np.uint8)
            n = lib.synth_fasta_record(name.encode(), seq.ctypes.data_as(C.c_char_p),
                                       C.c_uint64(len(seq)), C.c_uint32(width),
                                       buf.ctypes.data_as(C.c_char_p))
            out.append(buf[:n].tobytes())
        return b"".join(out)


class Synth:
    _lib = None

    @classmethod
    def lib(cls):
        if cls._lib is None:
            build_synth()
            lib = C.CDLL(SYNTH_SO)
            lib.synth_contig.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64, C.c_double, C.c_double, C.c_char_p]
            lib.synth_contig.restype = None
            lib.synth_sam_bound.argtypes = [C.POINTER(_ReadsCfg), C.c_uint64, C.c_uint64]
            lib.synth_sam_bound.restype = C.c_size_t
            lib.synth_sam.argtypes = [C.POINTER(_ReadsCfg), C.POINTER(C.c_char_p), C.POINTER(C.c_uint64),
                                      C.POINTER(C.c_char_p), C.c_uint32, C.c_uint64, C.c_uint64,
                                      C.c_void_p, C.c_size_t]
            lib.synth_sam.restype = C.c_size_t
            lib.synth_fasta_record.argtypes = [C.c_char_p, C.c_char_p, C.c_uint64, C.c_uint32, C.c_char_p]
            lib.synth_fasta_record.restype = C.c_size_t
            lib.synth_set_threads.argtypes = [C.c_int]
            lib.synth_set_threads.restype = None
            lib.synth_bam_bound.argtypes = [C.c_size_t, C.c_uint32]
            lib.synth_bam_bound.restype = C.c_size_t
            lib.synth_sam_to_bam.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_char_p), C.POINTER(C.c_uint64), C.c_uint32,
                                             C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_void_p, C.c_size_t]
            lib.synth_sam_to_bam.restype = C.c_size_t
            cls._lib = lib
        return cls._lib

    @classmethod
    def set_threads(cls, n: int):
        cls.lib().synth_set_threads(int(n))

    @classmethod
    def genome(cls, seed, contig_lens, names=None, n_frac=0.0, lower_frac=0.0) -> SynthGenome:
        lib = cls.lib()
        names = names or [f"chr{i + 1}" for i in range(len(contig_lens))]
        seqs = []
        for i, L in enumerate(contig_lens):
            a = np.empty(L, dtype=np.uint8)
            lib.synth_contig(seed, i, L, n_frac, lower_frac, a.ctypes.data_as(C.c_char_p))
            seqs.append(a)
        return SynthGenome(names=list(names), seqs=seqs, seed=seed)

    @classmethod
    def sam_into(cls, cfg: _ReadsCfg, g: SynthGenome, begin: int, end: int, out_ptr: int, out_cap: int) -> int:
        """Generate reads [begin,end) as SAM text into a caller buffer; returns bytes."""
        lib = cls.lib()
        nc = len(g.seqs)
        seqp = (C.c_char_p * nc)(*[C.cast(s.ctypes.data, C.c_char_p) for s in g.seqs])
        lens = (C.c_uint64 * nc)(*g.lens)
        namep = (C.c_char_p * nc)(*[n.encode() for n in g.names])
        n = lib.synth_sam(C.byref(cfg), seqp, lens, namep, nc, begin, end, C.c_void_p(out_ptr), out_cap)
        if n == 0 and end > begin:
            raise RuntimeError("synth_sam: output buffer too small")
        return n

    @classmethod
    def bam_into(cls, sam_ptr: int, sam_len: int, refs, out_ptr: int, out_cap: int, level=6, rg_mode=0, qual_mode=0,
                 block_payload=0) -> int:
        """SAM text (whole lines, as synth_sam writes them) at sam_ptr -> BAM file bytes at out_ptr.  refs: list of
        (name, length) -- the @SQ dictionary; every RNAME of the text must be in it.  Returns the BAM size."""
        lib = cls.lib()
        n = len(refs)
        names = (C.c_char_p * n)(*[r[0].encode() if isinstance(r[0], str) else r[0] for r in refs])
        lens = (C.c_uint64 * n)(*[int(r[1]) for r in refs])
        got = lib.synth_sam_to_bam(C.c_void_p(sam_ptr), sam_len, names, lens, n, level, rg_mode, qual_mode, block_payload,
                                   C.c_void_p(out_ptr), out_cap)
        if got == 0:
            raise RuntimeError("synth_sam_to_bam: a line the writer cannot represent, or the output buffer is too small")
        return got

    @classmethod
    def bam(cls, sam: bytes, refs, **kw) -> bytes:
        a = np.frombuffer(sam, dtype=np.uint8)
        cap = cls.lib().synth_bam_bound(len(sam), len(refs))
        if kw.get("block_payload"):
            cap += (2 * len(sam) // kw["block_payload"] + 16) * 40         # 26 bytes of framing per block
        out = np.empty(cap, dtype=np.uint8)
        n = cls.bam_into(a.ctypes.data, a.size, refs, out.ctypes.data, cap, **kw)
        return out[:n].tobytes()

    @classmethod
    def sam_bound(cls, cfg, begin, end) -> int:
        return cls.lib().synth_sam_bound(C.byref(cfg), begin, end)

    @classmethod
    def sam(cls, cfg: _ReadsCfg, g: SynthGenome, begin: int, end: int) -> bytes:
        cap = cls.sam_bound(cfg, begin, end)
        buf = np.empty(cap, dtype=np.uint8)
        n = cls.sam_into(cfg, g, begin, end, buf.ctypes.data, cap)
        return buf[:n].tobytes()


# --------------------------------------------------------------------------- oracle
class _OraContig(C.Structure):
    _fields_ = [("id", C.c_char_p), ("seq", C.c_void_p), ("len", C.c_size_t)]


class _OraGenome(C.Structure):
    _fields_ = [("ctg", C.POINTER(_OraContig)), ("n", C.c_size_t)]


class _OraPssParams(C.Structure):
    _fields_ = [("region_len", C.c_int), ("min_len", C.c_ulong), ("max_len", C.c_ulong),
                ("min_mq", C.c_int), ("up_ctx", C.c_char_p), ("down_ctx", C.c_char_p),
                ("merged_only", C.c_uint)]


class _OraFkParams(C.Structure):
    _fields_ = [("klen", C.c_int), ("min_len", C.c_ulong), ("max_len", C.c_ulong),
                ("min_mq", C.c_int), ("merged_only", C.c_int)]


class _OraStats(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("lines", "counted", "no_contig", "filtered", "parse_fail", "undefined")]

    def asdict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


@dataclass
class PssParams:
    region_len: int = 15
    min_len: int = 0
    max_len: int = 250000000
    min_mq: int = 0
    up_ctx: bytes = b"ACGT"
    down_ctx: bytes = b"ACGT"
    merged_only: int = 0

    def cli_args(self):
        a = ["-r", str(self.region_len), "-l", str(self.min_len), "-L", str(self.max_len),
             "-q", str(self.min_mq), "-U", self.up_ctx.decode(), "-D", self.down_ctx.decode()]
        if self.merged_only:
            a.append("-m")
        return a


@dataclass
class FkParams:
    klen: int = 8
    min_len: int = 0
    max_len: int = 250000000
    min_mq: int = 0
    merged_only: int = 0

    def cli_args(self):
        a = ["-k", str(self.klen), "-l", str(self.min_len), "-L", str(self.max_len), "-q", str(self.min_mq)]
        if self.merged_only:
            a.append("-m")
        return a


class Oracle:
    """CPU oracle (checker only)."""
    _lib = None

    @classmethod
    def lib(cls):
        if cls._lib is None:
            build_oracle()
            lib = C.CDLL(ORACLE_SO)
            lib.ora_genome_parse.argtypes = [C.c_char_p, C.c_size_t]
            lib.ora_genome_parse.restype = C.POINTER(_OraGenome)
            lib.ora_genome_load.argtypes = [C.c_char_p]
            lib.ora_genome_load.restype = C.POINTER(_OraGenome)
            lib.ora_genome_free.argtypes = [C.POINTER(_OraGenome)]
            lib.ora_genome_from_contigs.argtypes = [C.POINTER(C.c_char_p), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_size_t]
            lib.ora_genome_from_contigs.restype = C.POINTER(_OraGenome)
            lib.ora_pss_tally.argtypes = [C.POINTER(_OraGenome), C.c_void_p, C.c_size_t, C.POINTER(_OraPssParams),
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(_OraStats)]
            lib.ora_pss_tally.restype = C.c_uint64
            lib.ora_pss_rates.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
            lib.ora_pss_write_counts.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_int]
            lib.ora_pss_write_rates.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_int]
            lib.ora_fragkon_tally.argtypes = [C.POINTER(_OraGenome), C.c_void_p, C.c_size_t, C.POINTER(_OraFkParams),
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(_OraStats)]
            lib.ora_fragkon_tally.restype = C.c_uint64
            lib.ora_kmer_spectrum.argtypes = [C.POINTER(_OraGenome), C.c_int, C.c_void_p]
            lib.ora_kmer_spectrum.restype = None
            cls._lib = lib
        return cls._lib

    def __init__(self, fasta: bytes | None = None, fasta_path: str | None = None, contigs=None):
        """fasta: FASTA text; fasta_path: file; contigs: list of (name, np.uint8 array) -- no FASTA round trip."""
        lib = self.lib()
        if contigs is not None:
            n = len(contigs)
            ids = (C.c_char_p * n)(*[c[0].encode() for c in contigs])
            seqs = (C.c_void_p * n)(*[c[1].ctypes.data for c in contigs])
            lens = (C.c_size_t * n)(*[len(c[1]) for c in contigs])
            self.g = lib.ora_genome_from_contigs(ids, seqs, lens, n)
        elif fasta is not None:
            self.g = lib.ora_genome_parse(fasta, len(fasta))
        else:
            self.g = lib.ora_genome_load(fasta_path.encode())
            if not self.g:
                raise FileNotFoundError(fasta_path)

    def close(self):
        if self.g:
            self.lib().ora_genome_free(self.g)
            self.g = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def n_contigs(self):
        return int(self.g.contents.n)

    def contigs(self):
        out = []
        for i in range(self.n_contigs):
            c = self.g.contents.ctg[i]
            out.append((c.id.decode("latin1"), C.string_at(c.seq, c.len)))
        return out

    def pss(self, sam, p: PssParams = PssParams(), want_status=False):
        """Returns (fwd[(R+2),16] u64, rev, stats dict[, status int8 per line])."""
        lib = self.lib()
        R = p.region_len
        fwd = np.zeros(((R + 2), 16), dtype=np.uint64)
        rev = np.zeros(((R + 2), 16), dtype=np.uint64)
        st = _OraStats()
        cp = _OraPssParams(R, p.min_len, p.max_len, p.min_mq, p.up_ctx, p.down_ctx, p.merged_only)
        sam_ptr, sam_len, keep = _as_ptr(sam)
        status = None
        cap = 0
        if want_status:
            cap = _count_lines(sam) + 8
            status = np.full(cap, 99, dtype=np.int8)
        n = lib.ora_pss_tally(self.g, sam_ptr, sam_len, C.byref(cp), fwd.ctypes.data, rev.ctypes.data,
                              status.ctypes.data if want_status else None, cap, C.byref(st))
        del keep
        if want_status:
            return fwd, rev, st.asdict(), status[:n]
        return fwd, rev, st.asdict()

    def rates(self, counts: np.ndarray, R: int):
        out = np.zeros((R, 12), dtype=np.float64)
        c = np.ascontiguousarray(counts, dtype=np.uint64)
        self.lib().ora_pss_rates(c.ctypes.data, R, out.ctypes.data)
        return out

    def write_pss(self, fasta_fn, bam_fn, prefix, fwd, rev, R):
        lib = self.lib()
        fwd = np.ascontiguousarray(fwd, dtype=np.uint64)
        rev = np.ascontiguousarray(rev, dtype=np.uint64)
        fr, rr = self.rates(fwd, R), self.rates(rev, R)
        assert lib.ora_pss_write_counts(fasta_fn.encode(), bam_fn.encode(), prefix.encode(),
                                        fwd.ctypes.data, rev.ctypes.data, R) == 0
        assert lib.ora_pss_write_rates(fasta_fn.encode(), bam_fn.encode(), prefix.encode(),
                                       fr.ctypes.data, rr.ctypes.data, R) == 0

    def fragkon(self, sam, p: FkParams = FkParams(), want_status=False):
        lib = self.lib()
        nb = 1 << (2 * p.klen)
        fp = np.zeros(nb, dtype=np.uint64)
        tp = np.zeros(nb, dtype=np.uint64)
        st = _OraStats()
        cp = _OraFkParams(p.klen, p.min_len, p.max_len, p.min_mq, p.merged_only)
        sam_ptr, sam_len, keep = _as_ptr(sam)
        status = None
        cap = 0
        if want_status:
            cap = _count_lines(sam) + 8
            status = np.full(cap, 99, dtype=np.int8)
        n = lib.ora_fragkon_tally(self.g, sam_ptr, sam_len, C.byref(cp), fp.ctypes.data, tp.ctypes.data,
                                  status.ctypes.data if want_status else None, cap, C.byref(st))
        del keep
        if want_status:
            return fp, tp, st.asdict(), status[:n]
        return fp, tp, st.asdict()

    def kmer_spectrum(self, k: int):
        counts = np.zeros(1 << (2 * k), dtype=np.uint64)
        self.lib().ora_kmer_spectrum(self.g, k, counts.ctypes.data)
        return counts


def _newline_cuts(a: np.ndarray, parts: int):
    """Cut points of a SAM byte array into `parts` pieces that end after a newline."""
    n = a.size
    cuts = [0]
    for i in range(1, parts):
        pos = max(cuts[-1], n * i // parts)
        while pos < n:
            nl = np.flatnonzero(a[pos:min(n, pos + (1 << 20))] == 10)
            if nl.size:
                pos += int(nl[0]) + 1
                break
            pos = min(n, pos + (1 << 20))
        cuts.append(min(pos, n))
    cuts.append(n)
    return cuts


def oracle_parallel(ora: "Oracle", sam, what: str, params, threads: int):
    """The oracle over `sam` on `threads` host threads (ctypes releases the GIL; the oracle's tally is re-entrant and
    the genome is shared, read only): the text is cut after newlines, every piece tallied on its own, tables and
    outcome counters summed -- integer sums, so the result equals one sequential pass.  what: "pss" | "fragkon".
    Returns (table_a, table_b, stats)."""
    from concurrent.futures import ThreadPoolExecutor
    a = sam if isinstance(sam, np.ndarray) else np.frombuffer(sam, dtype=np.uint8)
    threads = max(1, int(threads))
    cuts = _newline_cuts(a, threads * 4)
    fn = ora.pss if what == "pss" else ora.fragkon
    with ThreadPoolExecutor(threads) as ex:
        res = list(ex.map(lambda i: fn(a[cuts[i]:cuts[i + 1]], params), range(len(cuts) - 1)))
    ta = sum(r[0] for r in res)
    tb = sum(r[1] for r in res)
    st = {k: sum(r[2][k] for r in res) for k in res[0][2]}
    return ta, tb, st


def oracle_spectrum_parallel(ora: "Oracle", k: int, threads: int):
    """ora_kmer_spectrum contig by contig on `threads` host threads (k-mers never span contigs,
    genome-kmer-count.c:56-58), summed."""
    from concurrent.futures import ThreadPoolExecutor
    lib = ora.lib()
    n = ora.n_contigs
    order = sorted(range(n), key=lambda i: -int(ora.g.contents.ctg[i].len))        # longest first

    def one(i):
        sub = _OraGenome(C.cast(C.byref(ora.g.contents.ctg[i]), C.POINTER(_OraContig)), 1)
        counts = np.zeros(1 << (2 * k), dtype=np.uint64)
        lib.ora_kmer_spectrum(C.byref(sub), k, counts.ctypes.data)
        return counts

    total = np.zeros(1 << (2 * k), dtype=np.uint64)
    with ThreadPoolExecutor(max(1, int(threads))) as ex:
        for c in ex.map(one, order):
            total += c
    return total


def _as_ptr(buf):
    """bytes / bytearray / np.uint8 array -> (void*, len, keepalive)."""
    if isinstance(buf, np.ndarray):
        a = np.ascontiguousarray(buf, dtype=np.uint8)
        return C.c_void_p(a.ctypes.data), a.size, a
    a = np.frombuffer(buf, dtype=np.uint8)
    return C.c_void_p(a.ctypes.data), a.size, a


def _count_lines(buf) -> int:
    a = buf if isinstance(buf, np.ndarray) else np.frombuffer(buf, dtype=np.uint8)
    n = int(np.count_nonzero(a == 10))
    # fgets also splits lines longer than 200000 bytes
    return n + 1 + a.size // 200000


# --------------------------------------------------------------------------- reference binaries
class RefBin:
    """The unmodified reference programs (oracle/_ref), run with the samtools shim on PATH."""
    MISSING = "reference programs not built: make -C oracle ref REF=<directory of the unmodified pss-bam sources>"

    @staticmethod
    def available() -> bool:
        return all(os.path.exists(os.path.join(REF_DIR, b))
                   for b in ("pss-bam", "fragkon", "genome-kmer-count", "samtools"))

    @staticmethod
    def env():
        e = dict(os.environ)
        e["PATH"] = REF_DIR + os.pathsep + e.get("PATH", "")
        return e

    @classmethod
    def pss_bam(cls, fasta_path, sam_path, prefix, extra=(), binary="pss-bam", cwd=None):
        cmd = [os.path.join(REF_DIR, binary), "-F", fasta_path, "-B", sam_path, "-o", prefix, *extra]
        r = subprocess.run(cmd, capture_output=True, env=cls.env(), cwd=cwd)
        if r.returncode != 0:
            raise RuntimeError(f"reference pss-bam failed ({r.returncode}): {r.stderr[-2000:]}")
        with open((os.path.join(cwd, prefix) if cwd else prefix) + ".pss.counts.txt", "rb") as f:
            counts = f.read()
        with open((os.path.join(cwd, prefix) if cwd else prefix) + ".pss.rates.txt", "rb") as f:
            rates = f.read()
        return counts, rates

    @classmethod
    def fragkon(cls, fasta_path, sam_path, extra=(), binary="fragkon", cwd=None) -> bytes:
        # stdbuf -oL: for k>8 the reference crashes in destroy_KSP (kmer.c:220-231) after
        # printing; line buffering keeps the complete table (SURVEY 8a).
        cmd = ["stdbuf", "-oL", os.path.join(REF_DIR, binary), "-F", fasta_path, "-B", sam_path, *extra]
        r = subprocess.run(cmd, capture_output=True, env=cls.env(), cwd=cwd)
        return r.stdout

    @classmethod
    def genome_kmer_count(cls, fasta_path, k, binary="genome-kmer-count", cwd=None) -> bytes:
        cmd = [os.path.join(REF_DIR, binary), "-f", fasta_path, "-k", str(k)]
        r = subprocess.run(cmd, capture_output=True, env=cls.env(), cwd=cwd)
        if r.returncode != 0:
            raise RuntimeError(f"reference genome-kmer-count failed: {r.stderr[-2000:]}")
        return r.stdout


def parse_counts_file(text: bytes, R: int):
    """Parse <prefix>.pss.counts.txt back into (fwd, rev) arrays laid out like the tally tables."""
    rows = [ln for ln in text.decode().split("\n") if ln and not ln.startswith("#")]
    assert len(rows) == 2 * (R + 2), len(rows)
    fwd = np.zeros((R + 2, 16), dtype=np.uint64)
    rev = np.zeros((R + 2, 16), dtype=np.uint64)
    for i in range(R + 2):
        f = rows[i].split("\t")
        assert int(f[0]) == i - 2
        fwd[i] = [int(x) for x in f[1:17]]
    for j in range(R):                      # rows R-1 .. 0
        f = rows[R + 2 + j].split("\t")
        pos = int(f[0])
        assert pos == R - 1 - j
        rev[pos + 2] = [int(x) for x in f[1:17]]
    f1 = rows[2 * R + 2].split("\t")        # labelled "1" -> rev row 1
    f2 = rows[2 * R + 3].split("\t")        # labelled "2" -> rev row 0
    rev[1] = [int(x) for x in f1[1:17]]
    rev[0] = [int(x) for x in f2[1:17]]
    return fwd, rev


def tmpdir():
    return tempfile.mkdtemp(prefix="psstest_")


# --------------------------------------------------------------------------- host build of the device record logic
EMUL_SO = os.path.join(ROOT, "tests", "host_emul", "libpssemul.so")


def build_emul(force=False):
    src = os.path.join(ROOT, "tests", "host_emul", "pss_emul.cpp")
    hdr = os.path.join(ROOT, "pss-bam_b200", "csrc", "pss_record.h")
    newest = max(os.path.getmtime(src), os.path.getmtime(hdr))
    return _locked_build(EMUL_SO, newest, force,
                         lambda out: ["g++", "-O2", "-g", "-std=c++17", "-Wno-unknown-pragmas", "-fPIC", "-shared", "-o", out, src])


class Emul:
    """pss_record.h compiled for the host (a TEST of the device logic, never a product path)."""
    _lib = None

    @classmethod
    def lib(cls):
        if cls._lib is None:
            build_emul()
            lib = C.CDLL(EMUL_SO)
            lib.emul_genome_new.argtypes = [C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.POINTER(C.c_uint64), C.c_uint32]
            lib.emul_genome_new.restype = C.c_void_p
            lib.emul_genome_free.argtypes = [C.c_void_p]
            lib.emul_scan11.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64),
                                        C.POINTER(C.c_uint32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
            lib.emul_tally.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_uint64, C.c_uint64,
                                       C.c_int, C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                       C.POINTER(C.c_uint64)]
            lib.emul_tally.restype = C.c_uint64
            lib.emul_spectrum.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
            cls._lib = lib
        return cls._lib

    def __init__(self, contigs):
        """contigs: list of (id str/bytes, seq bytes) -- e.g. Oracle.contigs()."""
        lib = self.lib()
        n = len(contigs)
        self._ids = [c[0].encode("latin1") if isinstance(c[0], str) else c[0] for c in contigs]
        self._seqs = [bytes(c[1]) for c in contigs]
        ids = (C.c_char_p * n)(*self._ids)
        seqs = (C.c_char_p * n)(*self._seqs)
        lens = (C.c_uint64 * n)(*[len(s) for s in self._seqs])
        self.g = lib.emul_genome_new(ids, seqs, lens, n)

    def close(self):
        if self.g:
            self.lib().emul_genome_free(self.g)
            self.g = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _tally(self, sam, mode, R, min_len, max_len, min_mq, up, down, merged_only, K, force_slow):
        lib = self.lib()
        fwd = np.zeros((R + 2, 16), dtype=np.uint64)
        rev = np.zeros((R + 2, 16), dtype=np.uint64)
        nb = 1 << (2 * K) if K else 1
        fp = np.zeros(nb, dtype=np.uint64)
        tp = np.zeros(nb, dtype=np.uint64)
        ptr, n, keep = _as_ptr(sam)
        cap = _count_lines(sam) + 8
        status = np.full(cap, 99, dtype=np.int8)
        fast = C.c_uint64(0)
        nl = lib.emul_tally(self.g, ptr, n, mode, R, min_len, max_len, min_mq, up, down, merged_only, K, force_slow,
                            fwd.ctypes.data, rev.ctypes.data, fp.ctypes.data, tp.ctypes.data,
                            status.ctypes.data, cap, C.byref(fast))
        del keep
        return fwd, rev, fp, tp, status[:nl], int(fast.value)

    def pss(self, sam, p: PssParams = PssParams(), force_slow=0):
        fwd, rev, _, _, st, fast = self._tally(sam, 0, p.region_len, p.min_len, p.max_len, p.min_mq,
                                               p.up_ctx, p.down_ctx, p.merged_only, 0, force_slow)
        return fwd, rev, st, fast

    def fragkon(self, sam, p: FkParams = FkParams(), force_slow=0):
        _, _, fp, tp, st, fast = self._tally(sam, 1, 0, p.min_len, p.max_len, p.min_mq, b"ACGT", b"ACGT",
                                             p.merged_only, p.klen, force_slow)
        return fp, tp, st, fast

    def kmer_spectrum(self, k):
        counts = np.zeros(1 << (2 * k), dtype=np.uint64)
        self.lib().emul_spectrum(self.g, k, counts.ctypes.data)
        return counts


# --------------------------------------------------------------------------- BAM: independent reader + host build of the device logic
def bgzf_blocks(bam: bytes):
    """[(offset, total, payload offset, payload length, isize)] of every BGZF block (SAM spec 4.1)."""
    out, at = [], 0
    while at < len(bam):
        assert bam[at:at + 4] == b"\x1f\x8b\x08\x04", at
        xlen = int.from_bytes(bam[at + 10:at + 12], "little")
        sub, bsize = at + 12, None
        while sub < at + 12 + xlen:
            slen = int.from_bytes(bam[sub + 2:sub + 4], "little")
            if bam[sub:sub + 2] == b"BC":
                bsize = int.from_bytes(bam[sub + 4:sub + 6], "little")
            sub += 4 + slen
        total = bsize + 1
        isize = int.from_bytes(bam[at + total - 4:at + total], "little")
        out.append((at, total, at + 12 + xlen, total - 12 - xlen - 8, isize))
        at += total
    return out


def bgzf_inflate(bam: bytes) -> bytes:
    """The inflated stream, by zlib, CRCs checked."""
    import zlib
    parts = []
    for at, total, po, pl, isize in bgzf_blocks(bam):
        d = zlib.decompress(bam[po:po + pl], -15)
        assert len(d) == isize and zlib.crc32(d) == int.from_bytes(bam[at + total - 8:at + total - 4], "little")
        parts.append(d)
    return b"".join(parts)


def bam_to_sam(bam: bytes, read_group=None) -> bytes:
    """What `samtools view [-r RG]` prints for this BAM: an independent reader (zlib + struct), all eleven fields and the
    optional fields with their types.  Python loops: small inputs only."""
    import struct
    u = bgzf_inflate(bam)
    assert u[:4] == b"BAM\x01"
    l_text, = struct.unpack_from("<i", u, 4)
    n_ref, = struct.unpack_from("<i", u, 8 + l_text)
    p = 12 + l_text
    names = []
    for _ in range(n_ref):
        l_name, = struct.unpack_from("<i", u, p)
        names.append(u[p + 4:p + 4 + l_name - 1])
        p += 8 + l_name
    out = []
    seqtab = b"=ACMGRSVTWYHKDBN"
    while p < len(u):
        bs, ref, pos, lrn, mapq, _bin, ncig, flag, lseq, nref, npos, tlen = struct.unpack_from("<iiiBBHHHiiii", u, p)
        q = p + 36
        qname = u[q:q + lrn - 1]; q += lrn
        cig = b"".join(b"%d%c" % (v >> 4, b"MIDNSHP=XB??????"[v & 15]) for v in struct.unpack_from("<%dI" % ncig, u, q)) or b"*"
        q += 4 * ncig
        sb = u[q:q + (lseq + 1) // 2]; q += (lseq + 1) // 2
        seq = bytes(seqtab[(sb[i >> 1] >> 4) if not i & 1 else (sb[i >> 1] & 15)] for i in range(lseq)) or b"*"
        qb = u[q:q + lseq]; q += lseq
        qual = b"*" if (lseq == 0 or qb[0] == 0xff) else bytes(c + 33 for c in qb)
        tags, rg, end = [], None, p + 4 + bs
        while q < end:
            tag, ty = u[q:q + 2], u[q + 2:q + 3]; q += 3
            if ty in b"ZH":
                z = u.index(b"\0", q); val = u[q:z]; q = z + 1
                tags.append(tag + b":" + ty + b":" + val)
                if tag == b"RG" and ty == b"Z" and rg is None:
                    rg = val
            elif ty == b"A":
                tags.append(tag + b":A:" + u[q:q + 1]); q += 1
            elif ty == b"f":
                tags.append(tag + b":f:" + (b"%g" % struct.unpack_from("<f", u, q)[0])); q += 4
            elif ty == b"B":
                st = u[q:q + 1]; n, = struct.unpack_from("<I", u, q + 1)
                fmt = {b"c": "b", b"C": "B", b"s": "h", b"S": "H", b"i": "i", b"I": "I", b"f": "f"}[st]
                vals = struct.unpack_from("<%d%s" % (n, fmt), u, q + 5)
                tags.append(tag + b":B:" + st + b"".join(b",%d" % v for v in vals))
                q += 5 + n * struct.calcsize(fmt)
            else:
                fmt = {b"c": "b", b"C": "B", b"s": "h", b"S": "H", b"i": "i", b"I": "I"}[ty]
                tags.append(tag + b":i:%d" % struct.unpack_from("<" + fmt, u, q)[0]); q += struct.calcsize(fmt)
        p = end
        if read_group is not None and rg != (read_group.encode() if isinstance(read_group, str) else read_group):
            continue
        rname = names[ref] if ref >= 0 else b"*"
        rnext = b"*" if nref < 0 else (b"=" if nref == ref else names[nref])
        out.append(b"\t".join([qname, b"%d" % flag, rname, b"%d" % (pos + 1), b"%d" % mapq, cig, rnext, b"%d" % (npos + 1),
                                b"%d" % tlen, seq, qual] + tags) + b"\n")
    return b"".join(out)


BAM_EMUL_SO = os.path.join(ROOT, "tests", "host_emul", "libpssbamemul.so")


# other shapes of the inflate tables: a second-level area too small for real blocks (the canonical-walk fallback runs)
# and a 9-bit first level (more second-level look-ups)
BAM_EMUL_VARIANTS = {"": [], "walk": ["-DPSS_INF_LIT_SUB=8"], "lit9": ["-DPSS_INF_LIT_BITS=9"]}


def build_bam_emul(force=False, variant=""):
    src = os.path.join(ROOT, "tests", "host_emul", "pss_bam_emul.cpp")
    hdrs = [os.path.join(ROOT, "pss-bam_b200", "csrc", h) for h in ("pss_inflate.h", "pss_bamrec.h", "pss_record.h", "pss_crc32.h")]
    newest = max(os.path.getmtime(f) for f in [src] + hdrs)
    target = BAM_EMUL_SO if not variant else BAM_EMUL_SO.replace(".so", f"_{variant}.so")
    return _locked_build(target, newest, force,
                         lambda out: ["g++", "-O2", "-g", "-std=c++17", "-Wno-unknown-pragmas", "-fPIC", "-shared",
                                      *BAM_EMUL_VARIANTS[variant], "-o", out, src])


class BamEmul:
    """pss_inflate.h / pss_bamrec.h compiled for the host (a TEST of the device logic, never a product path)."""
    _lib = None

    @classmethod
    def variant_lib(cls, variant):
        """emul_inflate of a differently shaped build of the inflate tables (BAM_EMUL_VARIANTS)."""
        lib = C.CDLL(build_bam_emul(variant=variant))
        lib.emul_inflate.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
        return lib

    @classmethod
    def lib(cls):
        if cls._lib is None:
            build_bam_emul()
            lib = C.CDLL(BAM_EMUL_SO)
            lib.emul_inflate.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
            lib.emul_bam_render.argtypes = [C.c_void_p, C.c_uint64, C.c_char_p, C.c_void_p, C.c_uint64,
                                            C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
            lib.emul_bam_render.restype = C.c_long
            lib.emul_bam_guess_stats.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint64)]
            lib.emul_crc32.argtypes = [C.c_void_p, C.c_uint32]
            lib.emul_crc32.restype = C.c_uint32
            cls._lib = lib
        return cls._lib

    @classmethod
    def crc32(cls, data: np.ndarray, offset: int, n: int) -> int:
        """CRC-32 of data[offset : offset + n] by the lane code of the inflate kernel (pss_crc32.h)."""
        assert data.dtype == np.uint8 and offset + n <= data.size
        return int(cls.lib().emul_crc32(data.ctypes.data + offset, n))

    @classmethod
    def inflate(cls, bam: bytes) -> bytes:
        """Every BGZF payload through the device inflate logic."""
        lib = cls.lib()
        parts = []
        for at, total, po, pl, isize in bgzf_blocks(bam):
            src = np.frombuffer(bam, dtype=np.uint8, count=pl + 8 if po + pl + 8 <= len(bam) else pl, offset=po)
            src = np.concatenate([src[:pl], np.zeros(8, dtype=np.uint8)])
            out = np.zeros(isize + 16, dtype=np.uint8)
            rc = lib.emul_inflate(src.ctypes.data, pl, out.ctypes.data, isize)
            if rc != 0:
                raise ValueError(f"inflate error {rc} in the block at {at}")
            parts.append(out[:isize].tobytes())
        return b"".join(parts)

    @classmethod
    def render(cls, inflated: bytes, read_group=None):
        lib = cls.lib()
        u = np.frombuffer(inflated + b"\0" * 16, dtype=np.uint8)
        cap = 4 * len(inflated) + 4096
        text = np.zeros(cap, dtype=np.uint8)
        nr, nd = C.c_uint64(), C.c_uint64()
        n = lib.emul_bam_render(u.ctypes.data, len(inflated), None if read_group is None else read_group.encode(), text.ctypes.data,
                                cap, C.byref(nr), C.byref(nd))
        if n < 0:
            raise ValueError(f"render error {n}")
        return text[:n].tobytes(), int(nr.value), int(nd.value)

    @classmethod
    def guess_stats(cls, inflated: bytes, block=65280):
        lib = cls.lib()
        u = np.frombuffer(inflated + b"\0" * 16, dtype=np.uint8)
        out = (C.c_uint64 * 3)()
        assert lib.emul_bam_guess_stats(u.ctypes.data, len(inflated), block, out) == 0
        return [int(x) for x in out]
