"""ctypes binding of libmicrocket_b200.so — one Python method per C entry point.

Host-side mirror of the reference's program interfaces (SURVEY.md §8b):
  Sam2Pairs  <-> sam2pairs <in.sam> <flash|unc> <prefix> [T] [ratio] [Q] [sam]   (sam2pairs.cpp:25-54)
  Krmdup     <-> krmdup -i <fq> -o <prefix> [-k -K -s -S]                         (krmdup.cpp:229-276)
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libmicrocket_b200.so")

PAIR_DTYPE = np.dtype([("pos1", "<u4"), ("pos2", "<u4"), ("chr1", "<u2"), ("chr2", "<u2"),
                       ("strands", "u1"), ("cls", "u1"), ("lane", "<u2")])


class MkError(RuntimeError):
    pass


class S2PCfg(C.Structure):
    _fields_ = [("mode", C.c_int), ("min_mapped_ratio", C.c_float), ("min_mapq", C.c_int), ("write_sam", C.c_int),
                ("emu_threads", C.c_int), ("device", C.c_int), ("emit_text", C.c_int), ("emit_packed", C.c_int),
                ("window_bytes", C.c_size_t), ("lane", C.c_uint16), ("sharded", C.c_int),
                ("rmdup", C.c_int), ("rmdup_capacity", C.c_uint64), ("hskip1", C.c_int), ("klen1", C.c_int), ("hskip2", C.c_int), ("klen2", C.c_int)]


class S2PStats(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("lowMap", "manyHits", "unpaired", "selfCircle", "trans", "cis10K", "cis1K", "cis0")] + \
               [(n, C.c_uint64) for n in ("selfCircle_true", "groups", "lines", "cigar_errors", "pairs")]

    def log_text(self):
        """The 8 lines of <prefix>.<mode>2pairs.log (sam2pairs.cpp:211-218)."""
        return ("lowMap\t%d\nmanyHits\t%d\nunpaired\t%d\nselfCircle\t%d\ntrans\t%d\ncis10K\t%d\ncis1K\t%d\ncis0\t%d\n" %
                (self.lowMap, self.manyHits, self.unpaired, self.selfCircle, self.trans, self.cis10K, self.cis1K, self.cis0)).encode()


class S2PDevIO(C.Structure):
    _fields_ = [("d_pairs_text", C.c_void_p), ("pairs_text_cap", C.c_size_t), ("d_pairs", C.c_void_p), ("pairs_cap", C.c_size_t),
                ("d_sam_text", C.c_void_p), ("sam_text_cap", C.c_size_t), ("d_line_off", C.c_void_p), ("line_off_cap", C.c_size_t),
                ("line_off_base", C.c_uint64), ("pairs_text_len", C.c_size_t), ("n_pairs", C.c_size_t), ("sam_text_len", C.c_size_t), ("consumed", C.c_size_t)]


class SynthOpts(C.Structure):
    _fields_ = [("dup_per_1024", C.c_int), ("dup_universe", C.c_uint64), ("chimeric_per_1024", C.c_int),
                ("noise_per_1024", C.c_int), ("selfcircle_per_1024", C.c_int)]


def synth_opts(dup_per_1024=0, dup_universe=0, chimeric_per_1024=-1, noise_per_1024=-1, selfcircle_per_1024=-1):
    return SynthOpts(dup_per_1024, dup_universe, chimeric_per_1024, noise_per_1024, selfcircle_per_1024)


class NormStats(C.Structure):
    _fields_ = [("kr_outer_max", C.c_uint32), ("kr_matvecs", C.c_uint32), ("kr_failed", C.c_uint32), ("kr_residual_max", C.c_double)]


NORM_TYPES = {"VC": 1, "VC_SQRT": 2, "KR": 4}
NORM_SCOPES = {"GW": 1, "INTER": 2}


class BgzfMember(C.Structure):
    _fields_ = [("in_off", C.c_uint64), ("out_off", C.c_uint64), ("in_len", C.c_uint32), ("isize", C.c_uint32)]


class DedupCfg(C.Structure):
    _fields_ = [("hskip1", C.c_int), ("klen1", C.c_int), ("hskip2", C.c_int), ("klen2", C.c_int), ("device", C.c_int),
                ("window_bytes", C.c_size_t), ("async_pull", C.c_int)]


class DedupStats(C.Structure):
    _fields_ = [("uniq", C.c_uint32), ("dup", C.c_uint32), ("discard", C.c_uint32), ("pairs", C.c_uint64)]

    def log_text(self):
        """The 4 lines appended to <prefix>.log (krmdup.cpp:386-389)."""
        return ("Total\t%d\nUniq\t%d\nDup\t%d\nDiscard\t%d\n" %
                (self.uniq + self.dup + self.discard, self.uniq, self.dup, self.discard)).encode()


def build(force=False, verbose=False):
    """Compile libmicrocket_b200.so for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h", ".hpp", ".cpp", "Makefile"))]
    srcs.append(os.path.join(os.path.dirname(HERE), "include", "microcket_b200.h"))
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(s) <= os.path.getmtime(LIB_PATH) for s in srcs):
        return LIB_PATH
    r = subprocess.run(["make", "-j8", "-C", CSRC, "all"], capture_output=True, text=True)
    if verbose or r.returncode:
        print(r.stdout[-4000:], r.stderr[-4000:])
    if r.returncode:
        raise MkError("building libmicrocket_b200.so failed")
    return LIB_PATH


class Lib:
    """Loaded libmicrocket_b200.so with typed prototypes."""

    def __init__(self, path=LIB_PATH):
        if not os.path.exists(path):
            raise MkError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
        L = self.L = C.CDLL(path)
        vp, sz, i, u64 = C.c_void_p, C.c_size_t, C.c_int, C.c_uint64
        P = C.POINTER
        L.mk_last_error.restype = C.c_char_p
        L.mk_version.restype = i
        L.mk_device_count.restype = i
        L.mk_destroy.argtypes = [vp]
        L.mk_copy_device.argtypes = [vp, vp, sz]
        L.mk_s2p_default_cfg.argtypes = [P(S2PCfg)]
        L.mk_s2p_create.argtypes = [P(S2PCfg), P(C.c_char_p), i, P(vp)]
        L.mk_s2p_push.argtypes = [vp, C.c_char_p, sz, i]
        L.mk_s2p_pull.argtypes = [vp, vp, sz, P(sz), vp, sz, P(sz)]
        L.mk_s2p_pull_packed.argtypes = [vp, vp, sz, P(sz)]
        L.mk_s2p_finish.argtypes = [vp, P(S2PStats)]
        L.mk_s2p_finish_sharded.argtypes = [vp, u64, u64, P(S2PStats)]
        L.mk_s2p_rmdup_stats.argtypes = [vp, P(DedupStats)]
        L.mk_s2p_reset.argtypes = [vp]
        L.mk_s2p_chrom_count.argtypes = [vp]
        L.mk_s2p_chrom_name.argtypes = [vp, i, C.c_char_p, sz]
        L.mk_s2p_run_device.argtypes = [vp, vp, sz, i, P(S2PDevIO), vp]
        L.mk_launch_count.argtypes = [vp]
        L.mk_s2p_attach_xchg.argtypes = [vp, vp, C.c_uint32]
        L.mk_launch_count.restype = u64
        L.mk_synth_host.argtypes = [u64, i, i, u64, u64, vp, sz, P(sz)]
        L.mk_synth_device.argtypes = [i, u64, i, i, u64, u64, vp, sz, P(sz), vp]
        L.mk_synth_host_ex.argtypes = [u64, i, i, P(SynthOpts), u64, u64, vp, sz, P(sz)]
        L.mk_synth_device_ex.argtypes = [i, u64, i, i, P(SynthOpts), u64, u64, vp, sz, P(sz), vp]
        for name, args in (("mk_dedup_default_cfg", [P(DedupCfg)]), ("mk_dedup_create", [P(DedupCfg), P(vp)]),
                           ("mk_dedup_push", [vp, C.c_char_p, sz, i]), ("mk_dedup_pull", [vp, vp, sz, P(sz), vp, sz, P(sz)]),
                           ("mk_dedup_finish", [vp, P(DedupStats)]), ("mk_dedup_reset", [vp]),
                           ("mk_dedup_keys_device", [i, vp, sz, vp, P(u64), vp]),
                           ("mk_pairs_ws_create", [i, sz, P(vp)]), ("mk_pairs_ws_destroy", [vp]),
                           ("mk_pairs_dedup_device", [vp, vp, sz, P(sz), vp]),
                           ("mk_pairs_bin_device", [vp, vp, sz, P(C.c_uint32), i, P(C.c_uint16), i, C.c_uint32, vp, vp, vp, sz, P(sz), vp]),
                           ("mk_pairs_dedup_bin_host", [vp, vp, sz, i, P(C.c_uint32), i, P(C.c_uint16), i, C.c_uint32, vp, vp, vp, sz, P(sz), P(sz)]),
                           ("mk_s2p_enable_timing", [vp, i]), ("mk_s2p_kernel_times", [vp, P(C.c_double), P(u64)]),
                           ("mk_pairs_dedup_bin_device", [vp, vp, sz, P(C.c_uint32), i, P(C.c_uint16), i, C.c_uint32, C.c_uint16, vp, vp, vp, sz, P(sz), P(sz), vp]),
                           ("mk_pairs_dedup_bin_indexed_device", [vp, vp, sz, P(C.c_uint32), i, P(C.c_uint16), i, C.c_uint32, C.c_uint16, vp, vp, vp, sz, vp, vp, P(sz), P(sz), vp]),
                           ("mk_pairs_dropped", [vp]),
                           ("mk_pairs_sort_text_device", [vp, vp, sz, vp, vp, vp, P(C.c_uint16), i, C.c_uint32, vp, sz, P(sz), P(sz), vp]),
                           ("mk_pairs_filter_text_device", [vp, sz, vp, vp, vp, vp, sz, P(sz), vp]),
                           ("mk_pairs_chrom_ranks", [P(C.c_char_p), i, P(C.c_uint16)]),
                           ("mk_pairs_parse_text_device", [vp, vp, sz, P(C.c_char_p), i, vp, sz, P(sz), P(sz), vp]),
                           ("mk_hist_cells", [P(C.c_uint32), i, C.c_uint32, P(u64), P(u64)]),
                           ("mk_hist_create", [i, P(C.c_uint32), i, P(C.c_uint32), i, P(vp), P(vp)]),
                           ("mk_hist_destroy", [vp]), ("mk_hist_reset", [vp, vp]),
                           ("mk_hist_add_device", [vp, vp, sz, P(C.c_uint16), i, vp]),
                           ("mk_hist_matrix", [vp, i, P(vp), P(u64), P(u64)]),
                           ("mk_hist_coo_device", [vp, i, vp, vp, vp, sz, P(sz), P(u64), vp]),
                           ("mk_hist_dropped", [vp]), ("mk_hist_launch_count", [vp]),
                           ("mk_xchg_create", [i, i, i, sz, P(vp)]), ("mk_xchg_destroy", [vp]), ("mk_xchg_handle", [vp, vp]),
                           ("mk_xchg_connect", [vp, vp]), ("mk_xchg_connect_local", [P(vp), i]),
                           ("mk_xchg_scatter_device", [vp, vp, sz, C.c_uint32, vp]), ("mk_xchg_finish_device", [vp, P(vp), P(sz), vp]),
                           ("mk_xchg_launch_count", [vp]), ("mk_xchg_begin", [vp]), ("mk_xchg_end_device", [vp, vp]),
                           ("mk_xchg_scatter_part_device", [vp, vp, vp, C.c_uint32, vp]),
                           ("mk_pairs_partition_device", [vp, vp, sz, i, C.c_uint32, vp, P(u64), vp]),
                           ("mk_pairs_launch_count", [vp]),
                           ("mk_norm_create", [i, P(C.c_uint32), i, C.c_uint32, sz, P(vp)]), ("mk_norm_destroy", [vp]),
                           ("mk_norm_device", [vp, vp, vp, vp, sz, i, vp, vp, vp, P(C.c_uint8), P(NormStats), vp]),
                           ("mk_norm_genome_device", [vp, vp, vp, vp, sz, i, i, vp, vp, P(C.c_uint8), P(NormStats), vp]),
                           ("mk_norm_launch_count", [vp]), ("mk_norm_enable_timing", [vp, i]),
                           ("mk_norm_kernel_times", [vp, P(C.c_double), P(u64)]),
                           ("mk_bgzf_scan", [vp, sz, P(BgzfMember), sz, P(sz), P(sz), P(u64)]), ("mk_bgzf_create", [i, sz, P(vp)]),
                           ("mk_bgzf_destroy", [vp]), ("mk_bgzf_inflate_device", [vp, vp, P(BgzfMember), sz, vp, sz, vp]),
                           ("mk_bgzf_text_stats", [vp, P(u64), P(C.c_int64)]), ("mk_bgzf_launch_count", [vp]),
                           ("mk_bgzf_deflate_bound", [sz]), ("mk_bgzf_enc_create", [i, sz, P(vp)]), ("mk_bgzf_enc_destroy", [vp]),
                           ("mk_bgzf_deflate_device", [vp, vp, sz, i, vp, sz, P(sz), P(BgzfMember), sz, P(sz), vp]),
                           ("mk_bgzf_enc_launch_count", [vp])):
            if hasattr(L, name):
                getattr(L, name).argtypes = args
        if hasattr(L, "mk_pairs_owner"):
            L.mk_pairs_owner.argtypes = [C.c_uint32] * 5
            L.mk_pairs_owner.restype = C.c_uint32
        if hasattr(L, "mk_pairs_launch_count"):
            L.mk_pairs_launch_count.restype = u64
        if hasattr(L, "mk_pairs_dropped"):
            L.mk_pairs_dropped.restype = u64
        for name in ("mk_hist_dropped", "mk_hist_launch_count", "mk_xchg_launch_count", "mk_norm_launch_count", "mk_bgzf_launch_count",
                     "mk_bgzf_enc_launch_count"):
            if hasattr(L, name):
                getattr(L, name).restype = u64
        if hasattr(L, "mk_bgzf_deflate_bound"):
            L.mk_bgzf_deflate_bound.restype = sz

    def check(self, rc):
        if rc != 0:
            raise MkError(f"microcket_b200 error {rc}: {self.L.mk_last_error().decode(errors='replace')}")

    def device_count(self):
        return self.L.mk_device_count()

    def check_cuda_copy(self, dst, src, nbytes):
        """device-to-device copy between raw pointers (library-owned buffers have no torch tensor)"""
        self.check(self.L.mk_copy_device(dst, src, nbytes))

    def require_gpu(self):
        if self.device_count() < 1:
            raise MkError("no CUDA device visible: microcket_b200 has no CPU fallback")


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = Lib()
    return _lib


class S2PConfig:
    def __init__(self, mode="unc", ratio=0.5, min_mapq=10, write_sam=False, threads=8, device=0, emit_text=True,
                 emit_packed=False, window_bytes=0, lane=0, sharded=False, rmdup=False, rmdup_capacity=0, key=(5, 16, 5, 16)):
        self.c = S2PCfg()
        lib().L.mk_s2p_default_cfg(C.byref(self.c))
        self.c.mode = {"flash": 0, "unc": 1}[mode]
        self.c.min_mapped_ratio = ratio
        self.c.min_mapq = min_mapq
        self.c.write_sam = int(write_sam)
        self.c.emu_threads = threads
        self.c.device = device
        self.c.emit_text = int(emit_text)
        self.c.emit_packed = int(emit_packed)
        self.c.window_bytes = window_bytes
        self.c.lane = lane
        self.c.sharded = int(sharded)
        # SAM-space krmdup (src/preprocess/krmdup.cpp taken on the SAM): key = (hskip1, klen1, hskip2, klen2)
        self.c.rmdup = int(rmdup)
        self.c.rmdup_capacity = rmdup_capacity
        self.c.hskip1, self.c.klen1, self.c.hskip2, self.c.klen2 = key


class Sam2Pairs:
    """One sam2pairs run (one reference process).  Host streaming: push()/pull()/finish()."""

    def __init__(self, cfg: S2PConfig, chrom_names=None):
        self.lib = lib()
        self.lib.require_gpu()
        self.cfg = cfg
        names = [n.encode() for n in (chrom_names or [])]
        arr = (C.c_char_p * max(len(names), 1))(*names)
        self.h = C.c_void_p()
        self.lib.check(self.lib.L.mk_s2p_create(C.byref(cfg.c), arr, len(names), C.byref(self.h)))
        self._buf = C.create_string_buffer(8 << 20)
        self._buf2 = C.create_string_buffer(8 << 20)

    def close(self):
        if self.h:
            self.lib.L.mk_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def push(self, data: bytes, is_last=False):
        self.lib.check(self.lib.L.mk_s2p_push(self.h, data, len(data), int(is_last)))

    def pull(self):
        """→ (pairs_text, sam_text) produced so far."""
        out, out2 = [], []
        n, n2 = C.c_size_t(), C.c_size_t()
        while True:
            self.lib.check(self.lib.L.mk_s2p_pull(self.h, C.addressof(self._buf), len(self._buf), C.byref(n),
                                                  C.addressof(self._buf2), len(self._buf2), C.byref(n2)))
            if n.value == 0 and n2.value == 0:
                break
            out.append(self._buf.raw[:n.value])
            out2.append(self._buf2.raw[:n2.value])
        return b"".join(out), b"".join(out2)

    def pull_packed(self):
        chunks = []
        cap = 1 << 18
        arr = np.empty(cap, dtype=PAIR_DTYPE)
        n = C.c_size_t()
        while True:
            self.lib.check(self.lib.L.mk_s2p_pull_packed(self.h, arr.ctypes.data, cap, C.byref(n)))
            if n.value == 0:
                break
            chunks.append(arr[:n.value].copy())
        return np.concatenate(chunks) if chunks else np.empty(0, dtype=PAIR_DTYPE)

    def finish(self, group_base=None, total_groups=None) -> S2PStats:
        st = S2PStats()
        if group_base is None:
            self.lib.check(self.lib.L.mk_s2p_finish(self.h, C.byref(st)))
        else:
            self.lib.check(self.lib.L.mk_s2p_finish_sharded(self.h, group_base, total_groups, C.byref(st)))
        return st

    def reset(self):
        self.lib.check(self.lib.L.mk_s2p_reset(self.h))

    def chrom_names(self):
        n = self.lib.L.mk_s2p_chrom_count(self.h)
        buf = C.create_string_buffer(64)
        out = []
        for i in range(n):
            self.lib.check(self.lib.L.mk_s2p_chrom_name(self.h, i, buf, 64))
            out.append(buf.value.decode())
        return out

    def run(self, sam: bytes, chunk=None):
        """Whole input through push/pull.  → (pairs_text, sam_text, stats)"""
        if chunk is None:
            self.push(sam, True)
        else:
            for o in range(0, len(sam), chunk):
                self.push(sam[o:o + chunk], False)
            self.push(b"", True)
        p, s = self.pull()
        return p, s, self.finish()

    def run_device(self, d_ptr, n, is_last, d_text=0, text_cap=0, d_pairs=0, pairs_cap=0, d_sam=0, sam_cap=0, stream=0,
                   d_line_off=0, line_off_cap=0, line_off_base=0):
        io = S2PDevIO(d_text, text_cap, d_pairs, pairs_cap, d_sam, sam_cap, d_line_off, line_off_cap, line_off_base, 0, 0, 0, 0)
        self.lib.check(self.lib.L.mk_s2p_run_device(self.h, d_ptr, n, int(is_last), C.byref(io), stream))
        return io

    def launches(self):
        return self.lib.L.mk_launch_count(self.h)

    def rmdup_stats(self) -> "DedupStats":
        """krmdup's log of the SAM-space duplicate removal (cfg.rmdup); call after finish()"""
        st = DedupStats()
        self.lib.check(self.lib.L.mk_s2p_rmdup_stats(self.h, C.byref(st)))
        return st

    def attach_xchg(self, xchg, res):
        """every window's packed pairs leave for their owners on a side stream while the next window is parsed"""
        self.lib.check(self.lib.L.mk_s2p_attach_xchg(self.h, xchg.h if xchg is not None else None, res))

    def enable_timing(self, on=True):
        self.lib.check(self.lib.L.mk_s2p_enable_timing(self.h, int(on)))

    def kernel_times(self):
        """→ {name: (total_ms, launches)} measured with CUDA events on the launching stream."""
        ms = (C.c_double * 8)()
        cnt = (C.c_uint64 * 8)()
        self.lib.check(self.lib.L.mk_s2p_kernel_times(self.h, ms, cnt))
        return {n: (ms[k], cnt[k]) for k, n in enumerate(("k_scan_chunks", "k_parse", "k_group", "k_emit", "k_copy_sam", "k_chunk_index", "k_rmdup"))}

    def push_ptr(self, ptr, n, is_last=False):
        """push() from a raw host pointer (e.g. a pinned torch tensor): no Python-side copy."""
        self.lib.check(self.lib.L.mk_s2p_push(self.h, C.cast(ptr, C.c_char_p), n, int(is_last)))

    def pull_into(self, text_ptr, text_cap, pairs_ptr=0, pairs_cap=0):
        """pull pair text (+ packed pairs) straight into caller memory → (text_bytes, n_pairs)"""
        n, n2, npk = C.c_size_t(), C.c_size_t(), C.c_size_t()
        self.lib.check(self.lib.L.mk_s2p_pull(self.h, text_ptr, text_cap, C.byref(n), None, 0, C.byref(n2)))
        if pairs_ptr:
            self.lib.check(self.lib.L.mk_s2p_pull_packed(self.h, pairs_ptr, pairs_cap, C.byref(npk)))
        return n.value, npk.value


class Krmdup:
    """One krmdup process (persistent key sets): push()/pull()/finish()."""

    def __init__(self, hskip1=5, klen1=16, hskip2=5, klen2=16, device=0, window_bytes=0, async_pull=False):
        self.lib = lib()
        self.lib.require_gpu()
        c = DedupCfg()
        self.lib.L.mk_dedup_default_cfg(C.byref(c))
        c.hskip1, c.klen1, c.hskip2, c.klen2, c.device, c.window_bytes = hskip1, klen1, hskip2, klen2, device, window_bytes
        c.async_pull = int(async_pull)
        self.h = C.c_void_p()
        self.lib.check(self.lib.L.mk_dedup_create(C.byref(c), C.byref(self.h)))
        self._b1 = C.create_string_buffer(8 << 20)
        self._b2 = C.create_string_buffer(8 << 20)

    def close(self):
        if self.h:
            self.lib.L.mk_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def push(self, data: bytes, is_last=False):
        self.lib.check(self.lib.L.mk_dedup_push(self.h, data, len(data), int(is_last)))

    def pull(self):
        o1, o2 = [], []
        n1, n2 = C.c_size_t(), C.c_size_t()
        while True:
            self.lib.check(self.lib.L.mk_dedup_pull(self.h, C.addressof(self._b1), len(self._b1), C.byref(n1),
                                                    C.addressof(self._b2), len(self._b2), C.byref(n2)))
            if n1.value == 0 and n2.value == 0:
                break
            o1.append(self._b1.raw[:n1.value])
            o2.append(self._b2.raw[:n2.value])
        return b"".join(o1), b"".join(o2)

    def reset(self):
        self.lib.check(self.lib.L.mk_dedup_reset(self.h))

    def finish(self) -> DedupStats:
        st = DedupStats()
        self.lib.check(self.lib.L.mk_dedup_finish(self.h, C.byref(st)))
        return st

    def run(self, fq: bytes, chunk=None):
        if chunk is None:
            self.push(fq, True)
        else:
            for o in range(0, len(fq), chunk):
                self.push(fq[o:o + chunk], False)
            self.push(b"", True)
        r1, r2 = self.pull()
        return r1, r2, self.finish()


class PairsWorkspace:
    """Device workspace for coordinate dedup + binning of packed pairs (device pointers in, device pointers out)."""

    def __init__(self, max_pairs, device=0):
        self.lib = lib()
        self.lib.require_gpu()
        self.h = C.c_void_p()
        self.lib.check(self.lib.L.mk_pairs_ws_create(device, max_pairs, C.byref(self.h)))

    def close(self):
        if self.h:
            self.lib.L.mk_pairs_ws_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def dedup(self, d_pairs, n, stream=0):
        kept = C.c_size_t()
        self.lib.check(self.lib.L.mk_pairs_dedup_device(self.h, d_pairs, n, C.byref(kept), stream))
        return kept.value

    def bin(self, d_pairs, n, chrom_len, res, d_bin1, d_bin2, d_cnt, cap, chrom_id_map=None, stream=0):
        cl = (C.c_uint32 * len(chrom_len))(*chrom_len)
        if chrom_id_map is not None:
            mp = (C.c_uint16 * len(chrom_id_map))(*chrom_id_map)
            nm = len(chrom_id_map)
        else:
            mp, nm = None, 0
        nnz = C.c_size_t()
        self.lib.check(self.lib.L.mk_pairs_bin_device(self.h, d_pairs, n, cl, len(chrom_len), mp, nm, res,
                                                      d_bin1, d_bin2, d_cnt, cap, C.byref(nnz), stream))
        return nnz.value

    def launches(self):
        return self.lib.L.mk_pairs_launch_count(self.h)

    def dedup_bin(self, d_pairs, n, chrom_len, res, d_bin1, d_bin2, d_cnt, cap, chrom_id_map=None, max_lane=0, stream=0,
                  d_keep=0, d_kept_idx=0):
        """One-sort duplicate removal + binning → (n_kept, nnz); d_keep / d_kept_idx: which input pairs survive"""
        cl = (C.c_uint32 * len(chrom_len))(*chrom_len)
        if chrom_id_map is not None:
            mp = (C.c_uint16 * len(chrom_id_map))(*chrom_id_map); nm = len(chrom_id_map)
        else:
            mp, nm = None, 0
        kept, nnz = C.c_size_t(), C.c_size_t()
        self.lib.check(self.lib.L.mk_pairs_dedup_bin_indexed_device(self.h, d_pairs, n, cl, len(chrom_len), mp, nm, res, max_lane,
                                                                    d_bin1, d_bin2, d_cnt, cap, d_keep, d_kept_idx,
                                                                    C.byref(kept), C.byref(nnz), stream))
        return kept.value, nnz.value

    def dropped(self):
        return self.lib.L.mk_pairs_dropped(self.h)

    def parse_text(self, d_text, n_bytes, chrom_names, d_out, cap, stream=0):
        """.pairs text on the device → packed pairs, one per line → (lines, lines that are not pairs of known chromosomes)"""
        arr = (C.c_char_p * len(chrom_names))(*[n.encode() for n in chrom_names])
        nl, ns = C.c_size_t(), C.c_size_t()
        self.lib.check(self.lib.L.mk_pairs_parse_text_device(self.h, d_text, n_bytes, arr, len(chrom_names), d_out, cap, C.byref(nl), C.byref(ns), stream))
        return nl.value, ns.value

    def sort_text(self, d_pairs, n, d_keep, d_text, d_line_off, chrom_rank, max_pos, d_out, out_cap, stream=0):
        """Lines of the kept pairs in `sort -k2,2d -k4,4d -k3,3n -k5,5n` order → (bytes, lines)"""
        rk = (C.c_uint16 * len(chrom_rank))(*chrom_rank)
        ol, nl = C.c_size_t(), C.c_size_t()
        self.lib.check(self.lib.L.mk_pairs_sort_text_device(self.h, d_pairs, n, d_keep, d_text, d_line_off, rk, len(chrom_rank), max_pos,
                                                            d_out, out_cap, C.byref(ol), C.byref(nl), stream))
        return ol.value, nl.value

    def filter_text(self, n, d_keep, d_text, d_line_off, d_out, out_cap, stream=0):
        ol = C.c_size_t()
        self.lib.check(self.lib.L.mk_pairs_filter_text_device(self.h, n, d_keep, d_text, d_line_off, d_out, out_cap, C.byref(ol), stream))
        return ol.value

    def partition(self, d_pairs, n, world, res, d_out, stream=0):
        counts = (C.c_uint64 * world)()
        self.lib.check(self.lib.L.mk_pairs_partition_device(self.h, d_pairs, n, world, res, d_out, counts, stream))
        return list(counts)

    def dedup_bin_host(self, pairs_ptr, n, chrom_len, res, b1_ptr, b2_ptr, c_ptr, cap, do_dedup=True, chrom_id_map=None):
        cl = (C.c_uint32 * len(chrom_len))(*chrom_len)
        if chrom_id_map is not None:
            mp = (C.c_uint16 * len(chrom_id_map))(*chrom_id_map); nm = len(chrom_id_map)
        else:
            mp, nm = None, 0
        kept, nnz = C.c_size_t(), C.c_size_t()
        self.lib.check(self.lib.L.mk_pairs_dedup_bin_host(self.h, pairs_ptr, n, int(do_dedup), cl, len(chrom_len), mp, nm, res,
                                                          b1_ptr, b2_ptr, c_ptr, cap, C.byref(kept), C.byref(nnz)))
        return kept.value, nnz.value


class Hist:
    """Dense multi-resolution contact histogram (csrc/hist.cu): add() packed pairs, then coo() per resolution."""

    def __init__(self, chrom_len, resolutions, device=0, cells_ptrs=None):
        self.lib = lib()
        self.lib.require_gpu()
        self.res = list(resolutions)
        self.chrom_len = list(chrom_len)
        cl = (C.c_uint32 * len(chrom_len))(*chrom_len)
        rs = (C.c_uint32 * len(self.res))(*self.res)
        ptrs = None
        if cells_ptrs is not None:
            ptrs = (C.c_void_p * len(self.res))(*cells_ptrs)
        self.h = C.c_void_p()
        self.lib.check(self.lib.L.mk_hist_create(device, cl, len(chrom_len), rs, len(self.res), ptrs, C.byref(self.h)))

    @staticmethod
    def cells(chrom_len, res):
        """→ (bins, cells of the upper triangle) at one resolution"""
        cl = (C.c_uint32 * len(chrom_len))(*chrom_len)
        nb, nc = C.c_uint64(), C.c_uint64()
        L = lib()
        L.check(L.L.mk_hist_cells(cl, len(chrom_len), res, C.byref(nb), C.byref(nc)))
        return nb.value, nc.value

    def close(self):
        if self.h:
            self.lib.L.mk_hist_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def add(self, d_pairs, n, chrom_id_map=None, stream=0):
        if chrom_id_map is not None:
            mp = (C.c_uint16 * len(chrom_id_map))(*chrom_id_map); nm = len(chrom_id_map)
        else:
            mp, nm = None, 0
        self.lib.check(self.lib.L.mk_hist_add_device(self.h, d_pairs, n, mp, nm, stream))

    def reset(self, stream=0):
        self.lib.check(self.lib.L.mk_hist_reset(self.h, stream))

    def matrix(self, k):
        """→ (device pointer, cells, bins) of resolution k's upper-triangle matrix"""
        p, nc, nb = C.c_void_p(), C.c_uint64(), C.c_uint64()
        self.lib.check(self.lib.L.mk_hist_matrix(self.h, k, C.byref(p), C.byref(nc), C.byref(nb)))
        return p.value, nc.value, nb.value

    def coo(self, k, d_bin1, d_bin2, d_cnt, cap, stream=0):
        """→ (nnz, sum of counts)"""
        nnz, tot = C.c_size_t(), C.c_uint64()
        self.lib.check(self.lib.L.mk_hist_coo_device(self.h, k, d_bin1, d_bin2, d_cnt, cap, C.byref(nnz), C.byref(tot), stream))
        return nnz.value, tot.value

    def dropped(self):
        return self.lib.L.mk_hist_dropped(self.h)

    def launches(self):
        return self.lib.L.mk_hist_launch_count(self.h)


class Norm:
    """Balancing of one resolution's contact matrices (csrc/norm.cu): VC, VC_SQRT and KR vectors per chromosome from the COO."""

    def __init__(self, chrom_len, res, max_nnz, device=0):
        self.lib = lib()
        self.lib.require_gpu()
        self.chrom_len, self.res = list(chrom_len), res
        self.n_bins = sum(l // res + 1 for l in self.chrom_len)
        cl = (C.c_uint32 * len(chrom_len))(*chrom_len)
        self.h = C.c_void_p()
        self.lib.check(self.lib.L.mk_norm_create(device, cl, len(chrom_len), res, max_nnz, C.byref(self.h)))

    def run(self, d_bin1, d_bin2, d_cnt, nnz, types=("VC", "VC_SQRT", "KR"), d_vc=0, d_vc_sqrt=0, d_kr=0, stream=0):
        """device COO in, n_bins doubles per requested type written to the device pointers -> (chrom_status list, NormStats)"""
        mask = 0
        for t in types:
            mask |= NORM_TYPES[t]
        status = (C.c_uint8 * len(self.chrom_len))()
        st = NormStats()
        self.lib.check(self.lib.L.mk_norm_device(self.h, d_bin1, d_bin2, d_cnt, nnz, mask, d_vc or None, d_vc_sqrt or None, d_kr or None,
                                                 status, C.byref(st), stream))
        return list(status), st

    def run_genome(self, d_bin1, d_bin2, d_cnt, nnz, scope="GW", types=("VC", "KR"), d_vc=0, d_kr=0, stream=0):
        """the genome-wide vectors: scope "GW" (every entry) or "INTER" (inter-chromosomal entries), types from ("VC", "KR");
        n_bins doubles per requested type written to the device pointers -> (status, NormStats); status 0 ok, 1 empty matrix,
        2 KR failed.  A scope or type outside these goes to the library as is, which refuses it."""
        mask = 0
        for t in types:
            mask |= NORM_TYPES[t] if isinstance(t, str) else t
        status = C.c_uint8()
        st = NormStats()
        sc = NORM_SCOPES[scope] if isinstance(scope, str) else scope
        self.lib.check(self.lib.L.mk_norm_genome_device(self.h, d_bin1, d_bin2, d_cnt, nnz, sc, mask, d_vc or None, d_kr or None,
                                                        C.byref(status), C.byref(st), stream))
        return status.value, st

    def launches(self):
        return self.lib.L.mk_norm_launch_count(self.h)

    def enable_timing(self, on=True):
        self.lib.check(self.lib.L.mk_norm_enable_timing(self.h, int(on)))

    def kernel_times(self):
        """-> {name: (ms, count)}: CUDA events around the kernels, host clock around the KR loop"""
        ms = (C.c_double * 8)()
        cnt = (C.c_uint64 * 8)()
        self.lib.check(self.lib.L.mk_norm_kernel_times(self.h, ms, cnt))
        names = ("build", "kr_product", "kr_vector", "kr_wall", "product", "vector")
        return {n: (ms[k], cnt[k]) for k, n in enumerate(names)}

    def close(self):
        if self.h:
            self.lib.L.mk_norm_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bgzf_scan(data, cap=None):
    """BGZF member walk over host bytes (mk_bgzf_scan) -> (members: BgzfMember array, bytes the whole members take, output bytes)"""
    cap = len(data) // 20 + 1 if cap is None else cap
    arr = (BgzfMember * max(cap, 1))()
    n, nb, no = C.c_size_t(), C.c_size_t(), C.c_uint64()
    L = lib()
    L.check(L.L.mk_bgzf_scan(data, len(data), arr, cap, C.byref(n), C.byref(nb), C.byref(no)))
    return (BgzfMember * n.value).from_buffer_copy(arr) if n.value else (BgzfMember * 0)(), nb.value, no.value


class Bgzf:
    """Inflate of BGZF members in HBM (csrc/bgzf.cu): one reusable object for calls of up to max_members members."""

    def __init__(self, max_members, device=0):
        self.lib = lib()
        self.lib.require_gpu()
        self.h = C.c_void_p()
        self.lib.check(self.lib.L.mk_bgzf_create(device, max_members, C.byref(self.h)))

    def inflate(self, d_in, members, d_out, out_cap, stream=0):
        """members (BgzfMember array or list, e.g. from bgzf_scan) of the compressed bytes at device pointer d_in -> d_out"""
        if not isinstance(members, C.Array):
            members = (BgzfMember * len(members))(*members)
        self.lib.check(self.lib.L.mk_bgzf_inflate_device(self.h, d_in, members, len(members), d_out, out_cap, stream))

    def text_stats(self):
        """-> (newline bytes the last call wrote, offset of the last one from d_out or -1)"""
        nl, last = C.c_uint64(), C.c_int64()
        self.lib.check(self.lib.L.mk_bgzf_text_stats(self.h, C.byref(nl), C.byref(last)))
        return nl.value, last.value

    def launches(self):
        return self.lib.L.mk_bgzf_launch_count(self.h)

    def close(self):
        if self.h:
            self.lib.L.mk_bgzf_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bgzf_decompress(data, device=0):
    """bytes of whole BGZF members -> their inflated bytes, through the GPU (torch tensors in and out)"""
    import torch
    mem, nb, n_out = bgzf_scan(data)
    if nb != len(data):
        raise MkError(f"BGZF input: {len(data) - nb} bytes after the last whole member (a truncated member)")
    d_in = torch.frombuffer(bytearray(data) or bytearray(1), dtype=torch.uint8).to(f"cuda:{device}")
    d_out = torch.empty(max(n_out, 1), dtype=torch.uint8, device=f"cuda:{device}")
    bz = Bgzf(max(len(mem), 1), device)
    try:
        bz.inflate(d_in.data_ptr(), mem, d_out.data_ptr(), n_out)
    finally:
        bz.close()
    return d_out[:n_out].cpu().numpy().tobytes()


BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")   # bgzip's end-of-file member


def bgzf_deflate_bound(n):
    """worst-case bytes of the members mk_bgzf_deflate_device writes for n input bytes (no EOF member)"""
    return lib().L.mk_bgzf_deflate_bound(n)


class BgzfDeflate:
    """BGZF members written in HBM (csrc/bgzf_deflate.cu): one reusable object for calls of up to max_bytes input bytes."""

    def __init__(self, max_bytes, device=0):
        self.lib = lib()
        self.lib.require_gpu()
        self.h = C.c_void_p()
        self.lib.check(self.lib.L.mk_bgzf_enc_create(device, max_bytes, C.byref(self.h)))

    def deflate(self, d_in, n, d_out, out_cap, level=-1, stream=0):
        """n bytes at device pointer d_in -> members back to back at d_out; -> (bytes written, BgzfMember table of the output)"""
        nm = -(-n // 65280)
        arr = (BgzfMember * max(nm, 1))()
        out_len, got = C.c_size_t(), C.c_size_t()
        self.lib.check(self.lib.L.mk_bgzf_deflate_device(self.h, d_in, n, level, d_out, out_cap, C.byref(out_len), arr, nm,
                                                         C.byref(got), stream))
        return out_len.value, (BgzfMember * got.value).from_buffer_copy(arr) if got.value else (BgzfMember * 0)()

    def launches(self):
        return self.lib.L.mk_bgzf_enc_launch_count(self.h)

    def close(self):
        if self.h:
            self.lib.L.mk_bgzf_enc_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bgzf_compress(data, level=-1, eof=True, device=0):
    """bytes -> BGZF bytes compressed on the GPU (bgzip's member cut), with bgzip's EOF member unless eof=False"""
    import torch
    d_in = torch.frombuffer(bytearray(data) or bytearray(1), dtype=torch.uint8).to(f"cuda:{device}")
    cap = bgzf_deflate_bound(len(data))
    d_out = torch.empty(max(cap, 1), dtype=torch.uint8, device=f"cuda:{device}")
    bd = BgzfDeflate(max(len(data), 1), device)
    try:
        n, _ = bd.deflate(d_in.data_ptr(), len(data), d_out.data_ptr(), cap, level)
    finally:
        bd.close()
    return d_out[:n].cpu().numpy().tobytes() + (BGZF_EOF if eof else b"")


class Xchg:
    """One rank of the NVLink peer-memory exchange of packed pairs (csrc/xchg.cu)."""

    def __init__(self, world, rank, cap_pairs, device=0):
        self.lib = lib()
        self.lib.require_gpu()
        self.world, self.rank = world, rank
        self.h = C.c_void_p()
        self.lib.check(self.lib.L.mk_xchg_create(device, world, rank, cap_pairs, C.byref(self.h)))

    def handle(self) -> bytes:
        buf = C.create_string_buffer(128)
        self.lib.check(self.lib.L.mk_xchg_handle(self.h, buf))
        return buf.raw

    def connect(self, all_handles: bytes):
        assert len(all_handles) == 128 * self.world
        self.lib.check(self.lib.L.mk_xchg_connect(self.h, all_handles))

    @staticmethod
    def connect_local(xs):
        arr = (C.c_void_p * len(xs))(*[x.h for x in xs])
        L = lib()
        L.check(L.L.mk_xchg_connect_local(arr, len(xs)))

    def scatter(self, d_pairs, n, res, stream=0):
        self.lib.check(self.lib.L.mk_xchg_scatter_device(self.h, d_pairs, n, res, stream))

    def finish(self, stream=0):
        """→ (device pointer of the pairs this rank owns, their number)"""
        p, n = C.c_void_p(), C.c_size_t()
        self.lib.check(self.lib.L.mk_xchg_finish_device(self.h, C.byref(p), C.byref(n), stream))
        return p.value or 0, n.value

    def launches(self):
        return self.lib.L.mk_xchg_launch_count(self.h)

    def close(self):
        if self.h:
            self.lib.L.mk_xchg_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def chrom_ranks(names):
    """rank of every chromosome name under `sort -d` (C locale), as mk_pairs_sort_text_device wants them"""
    arr = (C.c_char_p * max(len(names), 1))(*[n.encode() for n in names])
    out = (C.c_uint16 * max(len(names), 1))()
    L = lib()
    L.check(L.L.mk_pairs_chrom_ranks(arr, len(names), out))
    return list(out)[:len(names)]


def synth_host(seed, mode, genome, first, count, opts=None) -> bytes:
    """Synthetic SAM ('flash'/'unc') or interleaved FASTQ ('fastq') for groups/pairs [first, first+count) — host side."""
    m = {"flash": 0, "unc": 1, "fastq": 2}[mode]
    g = {"hg38": 0, "mm10": 1}[genome]
    L = lib()
    n = C.c_size_t()
    o = C.byref(opts) if opts is not None else None
    L.check(L.L.mk_synth_host_ex(seed, m, g, o, first, count, None, 0, C.byref(n)))
    buf = C.create_string_buffer(n.value + 16)
    L.check(L.L.mk_synth_host_ex(seed, m, g, o, first, count, C.addressof(buf), n.value, C.byref(n)))
    return buf.raw[:n.value]


def synth_device(torch, seed, mode, genome, first, count, device=0, opts=None):
    """The same bytes generated on the GPU → (uint8 cuda tensor, n_bytes); the tensor has 64 spare bytes behind the text."""
    m = {"flash": 0, "unc": 1, "fastq": 2}[mode]
    g = {"hg38": 0, "mm10": 1}[genome]
    L = lib()
    n = C.c_size_t()
    o = C.byref(opts) if opts is not None else None
    L.check(L.L.mk_synth_device_ex(device, seed, m, g, o, first, count, None, 0, C.byref(n), None))
    buf = torch.empty(n.value + 64, dtype=torch.uint8, device=f"cuda:{device}")
    L.check(L.L.mk_synth_device_ex(device, seed, m, g, o, first, count, buf.data_ptr(), n.value, C.byref(n), None))
    return buf, n.value
