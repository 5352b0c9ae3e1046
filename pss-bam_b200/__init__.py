"""pss-bam_b200 -- B200 (sm_100a) hot path of pss-bam / fragkon / genome-kmer-count.

The product is ``lib/libpssgpu.so`` (C ABI in ``include/pssgpu.h``, kernels in
``csrc/``).  This module is a thin ctypes binding of that ABI for tests, the
benchmark and Python callers; it holds no compute of its own and there is no
CPU fallback: if the library or a B200 is missing, calls raise.

The directory name contains a hyphen (it mirrors the reference's name), so
import it with ``importlib.import_module("pss-bam_b200")``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "lib", "libpssgpu.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--expt-extended-lambda", "-shared", "-Xcompiler", "-fPIC"]


class PssGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"pssgpu error {code}: {msg}")
        self.code = code


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/pssgpu.cu for sm_100a into lib/libpssgpu.so (nvcc cross-compiles without a GPU).

    Safe under torchrun: one process builds (file lock), into a temporary file that is renamed into place, so no other
    rank ever dlopens a half-written library."""
    import fcntl
    srcs = [os.path.join(CSRC, f) for f in ("pssgpu.cu", "pssgpu_bam.cu", "pssgpu_group.cu", "pssgpu_internal.h", "pss_kernels.cuh", "pss_record.h",
                                            "pss_inflate.h", "pss_bamrec.h", "pss_crc32.h")]
    srcs.append(os.path.join(ROOT, "include", "pssgpu.h"))
    newest = max(os.path.getmtime(s) for s in srcs)

    def fresh():
        return os.path.exists(LIB_PATH) and os.path.getsize(LIB_PATH) > 0 and os.path.getmtime(LIB_PATH) >= newest

    if not force and fresh():
        return LIB_PATH
    os.makedirs(os.path.dirname(LIB_PATH), exist_ok=True)
    with open(os.path.join(os.path.dirname(LIB_PATH), ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and fresh():                         # another process built it while we waited
                return LIB_PATH
            nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
            tmp = LIB_PATH + f".tmp{os.getpid()}"
            cmd = [nvcc, *NVCC_FLAGS, "--threads", "3", "-o", tmp, os.path.join(CSRC, "pssgpu.cu"), os.path.join(CSRC, "pssgpu_bam.cu"),
                   os.path.join(CSRC, "pssgpu_group.cu"), "-ldl"]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
            os.replace(tmp, LIB_PATH)
            if verbose:
                print(r.stderr)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH


# ---- ctypes mirror of include/pssgpu.h ------------------------------------------------------
class _Contig(C.Structure):
    _fields_ = [("id", C.c_char_p), ("seq", C.c_void_p), ("len", C.c_uint64)]


class _GenomeTag(C.Structure):
    _fields_ = [("source_size", C.c_uint64), ("source_mtime_ns", C.c_int64), ("source_path_hash", C.c_uint64),
                ("user", C.c_uint64)]


class _PssParams(C.Structure):
    _fields_ = [("region_len", C.c_int), ("min_len", C.c_ulong), ("max_len", C.c_ulong), ("min_mq", C.c_int),
                ("up_ctx", C.c_char_p), ("down_ctx", C.c_char_p), ("merged_only", C.c_uint)]


class _FkParams(C.Structure):
    _fields_ = [("klen", C.c_int), ("min_len", C.c_ulong), ("max_len", C.c_ulong), ("min_mq", C.c_int),
                ("merged_only", C.c_int)]


class _Stats(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("lines", "counted", "no_contig", "filtered", "parse_fail", "undefined")]


class _BamStats(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("records", "dropped_by_read_group", "references", "batches", "blocks_rewalked")]


class _Timing(C.Structure):
    _fields_ = [("launches", C.c_uint64), ("kernel_ms", C.c_double), ("bytes_scanned", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64)]


#: every symbol include/pssgpu.h declares (tests check the built library exports all of them)
ABI_SYMBOLS = (
    "pssgpu_abi_version", "pssgpu_device_count", "pssgpu_init", "pssgpu_destroy", "pssgpu_last_error",
    "pssgpu_cuda_stream", "pssgpu_host_alloc", "pssgpu_host_free",
    "pssgpu_genome_upload", "pssgpu_genome_upload_device", "pssgpu_genome_save", "pssgpu_genome_load", "pssgpu_genome_save_tagged", "pssgpu_genome_load_tagged",
    "pssgpu_genome_info",
    "pssgpu_pss_default_params", "pssgpu_pss_begin", "pssgpu_feed", "pssgpu_feed_device", "pssgpu_sync",
    "pssgpu_feed_bam", "pssgpu_bam_read_group", "pssgpu_bam_info", "pssgpu_feed_async", "pssgpu_feed_wait",
    "pssgpu_group_init", "pssgpu_group_destroy", "pssgpu_group_size", "pssgpu_group_ctx", "pssgpu_group_last_error",
    "pssgpu_group_reduce_backend", "pssgpu_group_last_reduce_ms", "pssgpu_group_genome_upload", "pssgpu_group_genome_load_tagged",
    "pssgpu_group_pss_begin", "pssgpu_group_fragkon_begin", "pssgpu_group_both_begin", "pssgpu_group_feed", "pssgpu_group_sync",
    "pssgpu_group_feed_bam", "pssgpu_group_bam_read_group", "pssgpu_group_bam_info",
    "pssgpu_group_pss_finish", "pssgpu_group_fragkon_finish", "pssgpu_group_get_stats", "pssgpu_group_kmer_spectrum",
    "pssgpu_pss_finish", "pssgpu_pss_finish_device", "pssgpu_get_stats", "pssgpu_both_begin", "pssgpu_get_fragkon_stats",
    "pssgpu_fragkon_default_params", "pssgpu_fragkon_begin", "pssgpu_fragkon_finish", "pssgpu_fragkon_finish_device",
    "pssgpu_kmer_spectrum", "pssgpu_kmer_spectrum_shard", "pssgpu_kmer_spectrum_shard_device",
    "pssgpu_timing_reset", "pssgpu_timing_get", "pssgpu_debug_status", "pssgpu_debug_fetch",
)

_lib = None


def load_library():
    """dlopen lib/libpssgpu.so (building it first if the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    lib = C.CDLL(build_library())
    P = C.c_void_p
    lib.pssgpu_abi_version.restype = C.c_int
    lib.pssgpu_device_count.restype = C.c_int
    lib.pssgpu_init.argtypes = [C.c_int, C.POINTER(P)]
    lib.pssgpu_destroy.argtypes = [P]
    lib.pssgpu_destroy.restype = None
    lib.pssgpu_last_error.argtypes = [P]
    lib.pssgpu_last_error.restype = C.c_char_p
    lib.pssgpu_cuda_stream.argtypes = [P]
    lib.pssgpu_cuda_stream.restype = P
    lib.pssgpu_host_alloc.argtypes = [C.c_size_t]
    lib.pssgpu_host_alloc.restype = P
    lib.pssgpu_host_free.argtypes = [P]
    lib.pssgpu_host_free.restype = None
    lib.pssgpu_genome_upload.argtypes = [P, C.POINTER(_Contig), C.c_uint64]
    lib.pssgpu_genome_upload_device.argtypes = [P, C.POINTER(_Contig), C.c_uint64]
    lib.pssgpu_genome_info.argtypes = [P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.pssgpu_genome_save.argtypes = [P, C.c_char_p]
    lib.pssgpu_genome_load.argtypes = [P, C.c_char_p]
    lib.pssgpu_genome_save_tagged.argtypes = [P, C.c_char_p, C.POINTER(_GenomeTag)]
    lib.pssgpu_genome_load_tagged.argtypes = [P, C.c_char_p, C.POINTER(_GenomeTag)]
    lib.pssgpu_pss_default_params.argtypes = [C.POINTER(_PssParams)]
    lib.pssgpu_pss_default_params.restype = None
    lib.pssgpu_pss_begin.argtypes = [P, C.POINTER(_PssParams)]
    lib.pssgpu_feed.argtypes = [P, P, C.c_size_t, C.c_int]
    lib.pssgpu_feed_device.argtypes = [P, P, C.c_size_t]
    lib.pssgpu_sync.argtypes = [P]
    lib.pssgpu_feed_async.argtypes = [P, P, C.c_size_t, C.c_int]
    lib.pssgpu_feed_wait.argtypes = [P]
    lib.pssgpu_group_init.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(P)]
    lib.pssgpu_group_destroy.argtypes = [P]
    lib.pssgpu_group_destroy.restype = None
    lib.pssgpu_group_size.argtypes = [P]
    lib.pssgpu_group_ctx.argtypes = [P, C.c_int]
    lib.pssgpu_group_ctx.restype = P
    lib.pssgpu_group_last_error.argtypes = [P]
    lib.pssgpu_group_last_error.restype = C.c_char_p
    lib.pssgpu_group_reduce_backend.argtypes = [P]
    lib.pssgpu_group_reduce_backend.restype = C.c_char_p
    lib.pssgpu_group_last_reduce_ms.argtypes = [P]
    lib.pssgpu_group_last_reduce_ms.restype = C.c_double
    lib.pssgpu_group_genome_upload.argtypes = [P, C.POINTER(_Contig), C.c_uint64]
    lib.pssgpu_group_genome_load_tagged.argtypes = [P, C.c_char_p, C.POINTER(_GenomeTag)]
    lib.pssgpu_group_pss_begin.argtypes = [P, C.POINTER(_PssParams)]
    lib.pssgpu_group_fragkon_begin.argtypes = [P, C.POINTER(_FkParams)]
    lib.pssgpu_group_both_begin.argtypes = [P, C.POINTER(_PssParams), C.POINTER(_FkParams)]
    lib.pssgpu_group_feed.argtypes = [P, P, C.c_size_t, C.c_int]
    lib.pssgpu_group_feed_bam.argtypes = [P, P, C.c_size_t, C.c_int]
    lib.pssgpu_group_bam_read_group.argtypes = [P, C.c_char_p]
    lib.pssgpu_group_bam_info.argtypes = [P, P, P]
    lib.pssgpu_group_sync.argtypes = [P]
    lib.pssgpu_group_pss_finish.argtypes = [P, P, P]
    lib.pssgpu_group_fragkon_finish.argtypes = [P, P, P]
    lib.pssgpu_group_get_stats.argtypes = [P, C.POINTER(_Stats), C.c_int]
    lib.pssgpu_group_kmer_spectrum.argtypes = [P, C.c_int, P]
    lib.pssgpu_feed_bam.argtypes = [P, P, C.c_size_t, C.c_int]
    lib.pssgpu_bam_read_group.argtypes = [P, C.c_char_p]
    lib.pssgpu_bam_info.argtypes = [P, C.POINTER(_BamStats)]
    lib.pssgpu_pss_finish.argtypes = [P, P, P]
    lib.pssgpu_pss_finish_device.argtypes = [P, P]
    lib.pssgpu_get_stats.argtypes = [P, C.POINTER(_Stats)]
    lib.pssgpu_get_fragkon_stats.argtypes = [P, C.POINTER(_Stats)]
    lib.pssgpu_both_begin.argtypes = [P, C.POINTER(_PssParams), C.POINTER(_FkParams)]
    lib.pssgpu_fragkon_default_params.argtypes = [C.POINTER(_FkParams)]
    lib.pssgpu_fragkon_default_params.restype = None
    lib.pssgpu_fragkon_begin.argtypes = [P, C.POINTER(_FkParams)]
    lib.pssgpu_fragkon_finish.argtypes = [P, P, P]
    lib.pssgpu_fragkon_finish_device.argtypes = [P, P]
    lib.pssgpu_kmer_spectrum.argtypes = [P, C.c_int, P]
    lib.pssgpu_kmer_spectrum_shard.argtypes = [P, C.c_int, C.c_int, C.c_int, P]
    lib.pssgpu_kmer_spectrum_shard_device.argtypes = [P, C.c_int, C.c_int, C.c_int, P]
    lib.pssgpu_timing_reset.argtypes = [P, C.c_int]
    lib.pssgpu_timing_get.argtypes = [P, C.POINTER(_Timing)]
    lib.pssgpu_debug_status.argtypes = [P, C.c_int]
    lib.pssgpu_debug_fetch.argtypes = [P, P, P, C.c_uint64, C.POINTER(C.c_uint64)]
    _lib = lib
    return lib


@dataclass
class PssOptions:
    """pss-bam.c:12-18 (same defaults)."""
    region_len: int = 15
    min_len: int = 0
    max_len: int = 250000000
    min_mq: int = 0
    up_ctx: bytes = b"ACGT"
    down_ctx: bytes = b"ACGT"
    merged_only: int = 0


@dataclass
class FragkonOptions:
    """fragkon.c:14-18 (same defaults)."""
    klen: int = 8
    min_len: int = 0
    max_len: int = 250000000
    min_mq: int = 0
    merged_only: int = 0


def _host_view(buf):
    """bytes / bytearray / memoryview / np.uint8 array -> (address, nbytes, keepalive)."""
    if isinstance(buf, np.ndarray):
        a = np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
    else:
        a = np.frombuffer(buf, dtype=np.uint8)
    return a.ctypes.data, a.size, a


def _contig_array(contigs, device=False):
    """(id, seq) pairs with seq in host memory, or with device=True (id, device_ptr, len) triples ->
    (_Contig array, count, keepalive)."""
    contigs = list(contigs)
    arr = (_Contig * max(1, len(contigs)))()
    keep = []
    for i, c in enumerate(contigs):
        if device:
            (cid, addr, n), ka = c, None
        else:
            cid, seq = c
            addr, n, ka = _host_view(seq)
        cid = cid.encode("latin1") if isinstance(cid, str) else bytes(cid)
        keep.append((cid, ka))
        arr[i] = _Contig(cid, addr, n)
    return arr, len(contigs), keep


def _pss_params(o: PssOptions):
    return _PssParams(o.region_len, o.min_len, o.max_len, o.min_mq, bytes(o.up_ctx), bytes(o.down_ctx), o.merged_only)


def _fk_params(o: FragkonOptions):
    return _FkParams(o.klen, o.min_len, o.max_len, o.min_mq, o.merged_only)


def _table_pair(shape):
    """The two tables a *_finish call fills: pss forward / reverse, or fragkon's two histograms."""
    return np.zeros(shape, dtype=np.uint64), np.zeros(shape, dtype=np.uint64)


class Context:
    """One GPU.  Mirrors the call order of the reference mains: load genome, tally a SAM stream, read tables."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.pssgpu_init(device, C.byref(h))
        if rc != 0:
            raise PssGpuError(rc, self.lib.pssgpu_last_error(None).decode())
        self.h = h
        self.device = device
        self._mode = None
        self._R = None
        self._K = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.pssgpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise PssGpuError(rc, self.lib.pssgpu_last_error(self.h).decode())

    @property
    def cuda_stream(self) -> int:
        return int(self.lib.pssgpu_cuda_stream(self.h) or 0)

    # ---- genome (init_genome's result, fasta-genome-io.c:221-238)
    def upload_genome(self, contigs):
        """contigs: iterable of (id, seq) with seq bytes / np.uint8 (host) -- any order."""
        arr, n, keep = _contig_array(contigs)
        self._ck(self.lib.pssgpu_genome_upload(self.h, arr, n))

    def upload_genome_device(self, contigs):
        """contigs: iterable of (id, device_ptr, len)."""
        arr, n, keep = _contig_array(contigs, device=True)
        self._ck(self.lib.pssgpu_genome_upload_device(self.h, arr, n))

    def save_genome(self, path, tag=None):
        """Write the resident packed genome to `path` (pssgpu_genome_save[_tagged]); tag = (size, mtime_ns, path_hash, user)."""
        if tag is None:
            self._ck(self.lib.pssgpu_genome_save(self.h, os.fsencode(path)))
        else:
            t = _GenomeTag(*tag)
            self._ck(self.lib.pssgpu_genome_save_tagged(self.h, os.fsencode(path), C.byref(t)))

    def load_genome(self, path, tag=None):
        """Make the packed genome of `path` resident (pssgpu_genome_load[_tagged]) instead of upload_genome()."""
        if tag is None:
            self._ck(self.lib.pssgpu_genome_load(self.h, os.fsencode(path)))
        else:
            t = _GenomeTag(*tag)
            self._ck(self.lib.pssgpu_genome_load_tagged(self.h, os.fsencode(path), C.byref(t)))

    def genome_info(self):
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._ck(self.lib.pssgpu_genome_info(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return {"n_contigs": a.value, "n_bases": b.value, "hbm_bytes": c.value}

    # ---- tallies
    def pss_begin(self, o: PssOptions = PssOptions()):
        self._ck(self.lib.pssgpu_pss_begin(self.h, C.byref(_pss_params(o))))
        self._mode, self._R = "pss", o.region_len

    def fragkon_begin(self, o: FragkonOptions = FragkonOptions()):
        self._ck(self.lib.pssgpu_fragkon_begin(self.h, C.byref(_fk_params(o))))
        self._mode, self._K = "fragkon", o.klen

    def both_begin(self, o: PssOptions = PssOptions(), f: FragkonOptions = FragkonOptions()):
        """pss-bam and fragkon tallies from one scan of the text."""
        self._ck(self.lib.pssgpu_both_begin(self.h, C.byref(_pss_params(o)), C.byref(_fk_params(f))))
        self._mode, self._R, self._K = "both", o.region_len, f.klen

    def fragkon_stats(self):
        s = _Stats()
        self._ck(self.lib.pssgpu_get_fragkon_stats(self.h, C.byref(s)))
        return {k: int(getattr(s, k)) for k, _ in _Stats._fields_}

    def feed(self, sam, last: bool = False):
        addr, n, keep = _host_view(sam)
        self._ck(self.lib.pssgpu_feed(self.h, addr, n, 1 if last else 0))
        del keep

    def feed_ptr(self, host_ptr: int, nbytes: int, last: bool = False):
        self._ck(self.lib.pssgpu_feed(self.h, host_ptr, nbytes, 1 if last else 0))

    def feed_bam(self, bam, last: bool = False):
        """Bytes of a BAM file (BGZF), any chunking (pssgpu_feed_bam)."""
        addr, n, keep = _host_view(bam)
        self._ck(self.lib.pssgpu_feed_bam(self.h, addr, n, 1 if last else 0))
        del keep

    def feed_bam_ptr(self, host_ptr: int, nbytes: int, last: bool = False):
        self._ck(self.lib.pssgpu_feed_bam(self.h, host_ptr, nbytes, 1 if last else 0))

    def bam_read_group(self, rg):
        """samtools view -r RG, natively; None switches the filter off."""
        self._ck(self.lib.pssgpu_bam_read_group(self.h, None if rg is None else (rg.encode() if isinstance(rg, str) else bytes(rg))))

    def bam_info(self):
        s = _BamStats()
        self._ck(self.lib.pssgpu_bam_info(self.h, C.byref(s)))
        return {k: int(getattr(s, k)) for k, _ in _BamStats._fields_}

    def feed_device(self, dev_ptr: int, nbytes: int):
        self._ck(self.lib.pssgpu_feed_device(self.h, dev_ptr, nbytes))

    def sync(self):
        self._ck(self.lib.pssgpu_sync(self.h))

    def pss_finish(self):
        fwd, rev = _table_pair((self._R + 2, 16))
        self._ck(self.lib.pssgpu_pss_finish(self.h, fwd.ctypes.data, rev.ctypes.data))
        return fwd, rev

    def pss_finish_device(self, dev_ptr: int):
        self._ck(self.lib.pssgpu_pss_finish_device(self.h, dev_ptr))

    def fragkon_finish(self):
        fp, tp = _table_pair(1 << (2 * self._K))
        self._ck(self.lib.pssgpu_fragkon_finish(self.h, fp.ctypes.data, tp.ctypes.data))
        return fp, tp

    def fragkon_finish_device(self, dev_ptr: int):
        self._ck(self.lib.pssgpu_fragkon_finish_device(self.h, dev_ptr))

    def stats(self):
        s = _Stats()
        self._ck(self.lib.pssgpu_get_stats(self.h, C.byref(s)))
        return {k: int(getattr(s, k)) for k, _ in _Stats._fields_}

    # ---- one-call conveniences (what the three mains do between genome load and table printing)
    def pss(self, sam, o: PssOptions = PssOptions()):
        self.pss_begin(o)
        self.feed(sam, last=True)
        return self.pss_finish()

    def fragkon(self, sam, o: FragkonOptions = FragkonOptions()):
        self.fragkon_begin(o)
        self.feed(sam, last=True)
        return self.fragkon_finish()

    def kmer_spectrum(self, k: int, shard: int = 0, n_shards: int = 1):
        counts = np.zeros(1 << (2 * k), dtype=np.uint64)
        self._ck(self.lib.pssgpu_kmer_spectrum_shard(self.h, k, shard, n_shards, counts.ctypes.data))
        return counts

    def kmer_spectrum_device(self, k: int, dev_ptr: int, shard: int = 0, n_shards: int = 1):
        self._ck(self.lib.pssgpu_kmer_spectrum_shard_device(self.h, k, shard, n_shards, dev_ptr))

    # ---- measurement / debugging hooks
    def timing_reset(self, enable=True):
        self._ck(self.lib.pssgpu_timing_reset(self.h, 1 if enable else 0))

    def timing(self):
        t = _Timing()
        self._ck(self.lib.pssgpu_timing_get(self.h, C.byref(t)))
        return {k: getattr(t, k) for k, _ in _Timing._fields_}

    def debug_status(self, enable=True):
        self._ck(self.lib.pssgpu_debug_status(self.h, 1 if enable else 0))

    def debug_fetch(self, cap=1 << 23):
        off = np.zeros(cap, dtype=np.uint64)
        code = np.zeros(cap, dtype=np.int8)
        n = C.c_uint64()
        self._ck(self.lib.pssgpu_debug_fetch(self.h, off.ctypes.data, code.ctypes.data, cap, C.byref(n)))
        k = int(n.value)
        order = np.argsort(off[:k], kind="stable")
        return off[:k][order], code[:k][order]


class Group:
    """Several GPUs of one box in one process (pssgpu_group_*): reads dealt line-wise to the members, genome replicated,
    tables summed with NCCL (or peer copies) when they are read."""

    def __init__(self, devices=None):
        self.lib = load_library()
        h = C.c_void_p()
        if devices is None:
            rc = self.lib.pssgpu_group_init(None, 0, C.byref(h))
        else:
            arr = (C.c_int * len(devices))(*devices)
            rc = self.lib.pssgpu_group_init(arr, len(devices), C.byref(h))
        if rc != 0:
            raise PssGpuError(rc, self.lib.pssgpu_last_error(None).decode())
        self.h = h
        self._R = self._K = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.pssgpu_group_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise PssGpuError(rc, self.lib.pssgpu_group_last_error(self.h).decode())

    @property
    def size(self):
        return int(self.lib.pssgpu_group_size(self.h))

    @property
    def reduce_backend(self):
        return self.lib.pssgpu_group_reduce_backend(self.h).decode()

    @property
    def last_reduce_ms(self):
        return float(self.lib.pssgpu_group_last_reduce_ms(self.h))

    def upload_genome(self, contigs):
        arr, n, keep = _contig_array(contigs)
        self._ck(self.lib.pssgpu_group_genome_upload(self.h, arr, n))

    def pss_begin(self, o: PssOptions = PssOptions()):
        self._ck(self.lib.pssgpu_group_pss_begin(self.h, C.byref(_pss_params(o))))
        self._R = o.region_len

    def fragkon_begin(self, o: FragkonOptions = FragkonOptions()):
        self._ck(self.lib.pssgpu_group_fragkon_begin(self.h, C.byref(_fk_params(o))))
        self._K = o.klen

    def feed(self, sam, last=False):
        addr, n, keep = _host_view(sam)
        self._ck(self.lib.pssgpu_group_feed(self.h, addr, n, 1 if last else 0))
        del keep

    def feed_bam(self, bam, last=False):
        """Bytes of a BAM file: the inflate is dealt to the members, member 0 frames, renders and tallies (pssgpu_group_feed_bam)."""
        addr, n, keep = _host_view(bam)
        self._ck(self.lib.pssgpu_group_feed_bam(self.h, addr, n, 1 if last else 0))
        del keep

    def feed_bam_ptr(self, host_ptr: int, nbytes: int, last: bool = False):
        self._ck(self.lib.pssgpu_group_feed_bam(self.h, host_ptr, nbytes, 1 if last else 0))

    def bam_read_group(self, rg):
        self._ck(self.lib.pssgpu_group_bam_read_group(self.h, None if rg is None else (rg.encode() if isinstance(rg, str) else bytes(rg))))

    def bam_info(self):
        s = _BamStats()
        per = (C.c_uint64 * self.size)()
        self._ck(self.lib.pssgpu_group_bam_info(self.h, C.byref(s), per))
        d = {k: int(getattr(s, k)) for k, _ in _BamStats._fields_}
        d["batches_per_member"] = [int(x) for x in per]
        return d

    def sync(self):
        self._ck(self.lib.pssgpu_group_sync(self.h))

    def pss_finish(self):
        fwd, rev = _table_pair((self._R + 2, 16))
        self._ck(self.lib.pssgpu_group_pss_finish(self.h, fwd.ctypes.data, rev.ctypes.data))
        return fwd, rev

    def fragkon_finish(self):
        fp, tp = _table_pair(1 << (2 * self._K))
        self._ck(self.lib.pssgpu_group_fragkon_finish(self.h, fp.ctypes.data, tp.ctypes.data))
        return fp, tp

    def stats(self, fragkon=False):
        s = _Stats()
        self._ck(self.lib.pssgpu_group_get_stats(self.h, C.byref(s), 1 if fragkon else 0))
        return {k: int(getattr(s, k)) for k, _ in _Stats._fields_}

    def kmer_spectrum(self, k: int):
        counts = np.zeros(1 << (2 * k), dtype=np.uint64)
        self._ck(self.lib.pssgpu_group_kmer_spectrum(self.h, k, counts.ctypes.data))
        return counts
