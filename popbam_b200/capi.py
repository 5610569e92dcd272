"""ctypes binding of include/popbam_b200.h.  No fallback: if the library is missing, importing the symbols works but
`lib()` raises, and every call goes through `lib()`."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent
MAXS = 64

AN = dict(NUCDIV=0x001, SFS=0x002, LD_ZNS=0x004, LD_OMEGA=0x008, LD_WALL=0x010, DIVERGE_IND=0x020,
          DIVERGE_POP=0x040, HAPLO_K=0x080, HAPLO_EHHS=0x100, HAPLO_DXY=0x200, SNP=0x400, TREE=0x800,
          THETA_W=0x1000, FULI=0x2000, LD_DPRIME=0x4000, FST=0x8000, ABBA=0x10000, GARUD=0x20000, SPECTRUM=0x40000,
          NUCDIV_MISSING=0x80000)
FLAG = dict(ILLUMINA=0x02, SUBSTITUTE=0x10, HETEROZYGOTE=0x20, OUTGROUP=0x40, EMIT_CB=0x10000)

EXPORTS = ["pb_create", "pb_destroy", "pb_last_error", "pb_version", "pb_set_contig", "pb_region_begin", "pb_push_batch", "pb_push_batch_async",
           "pb_push_record", "pb_region_reserve", "pb_region_end", "pb_region_launch", "pb_region_wait", "pb_region_relaunch", "pb_stream",
           "pb_kernel_launches", "pb_region_path", "pb_region_reruns", "pb_stage_times", "pb_window_grid", "pb_build_errmod_tables", "pb_errmod_tables_cached", "pb_errmod_tables_cached_ex", "pb_host_alloc", "pb_host_free", "pb_format_window",
           "pb_region_get_extras", "pb_format_window_ext", "pb_region_get_fst", "pb_set_snn_perms", "pb_format_window_fst",
           "pb_region_get_abba", "pb_set_abba", "pb_format_window_abba", "pb_region_get_garud", "pb_format_window_garud",
           "pb_region_get_spectrum", "pb_set_spectra", "pb_format_spectrum_dadi", "pb_region_get_nucdiv_missing",
           "pb_format_window_nucdiv_missing"]


def _p(t):
    return C.POINTER(t)


class Params(C.Structure):
    _fields_ = [("n_samples", C.c_int32), ("n_pops", C.c_int32),
                ("pop_mask", C.c_uint64 * MAXS), ("pop_nsmpl", C.c_uint8 * MAXS),
                ("min_depth", C.c_int32), ("max_depth", C.c_int32), ("min_rmsQ", C.c_int32),
                ("min_snpQ", C.c_int32), ("min_mapQ", C.c_int32), ("min_baseQ", C.c_int32),
                ("flags", C.c_uint32), ("outidx", C.c_int32), ("min_freq", C.c_int32),
                ("device", C.c_int32)]


class Tables(C.Structure):
    _fields_ = [("fk", _p(C.c_double)), ("beta", _p(C.c_double)), ("lhet", _p(C.c_double))]


class Batch(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("n_cigar", C.c_int64), ("n_bases", C.c_int64),
                ("pos", _p(C.c_int32)), ("meta", _p(C.c_uint32)),
                ("cig_off", _p(C.c_uint32)), ("cigar", _p(C.c_uint32)),
                ("base_off", _p(C.c_uint32)), ("seq4", _p(C.c_uint8)),
                ("qual", _p(C.c_uint8))]


class Result(C.Structure):
    _fields_ = [("n_windows", C.c_int32), ("n_pops", C.c_int32), ("n_samples", C.c_int32),
                ("analyses", C.c_uint32),
                ("win_beg", _p(C.c_int32)), ("win_end", _p(C.c_int32)), ("num_sites", _p(C.c_int32)),
                ("segsites", _p(C.c_int32)), ("seg_off", _p(C.c_int64)), ("seg_pos", _p(C.c_uint32)),
                ("seg_idx", _p(C.c_uint32)), ("seg_type", _p(C.c_uint64)), ("seg_ref", _p(C.c_uint8)),
                ("seg_cb", _p(C.c_uint64)),
                ("piw", _p(C.c_double)), ("pib", _p(C.c_double)), ("min_dxy", _p(C.c_uint16)),
                ("sfs_num_snps", _p(C.c_int32)), ("td", _p(C.c_double)), ("fwh", _p(C.c_double)),
                ("ld_num_snps", _p(C.c_int32)), ("zns", _p(C.c_double)), ("omegamax", _p(C.c_double)),
                ("wall_num_snps", _p(C.c_int32)), ("wallb", _p(C.c_double)), ("wallq", _p(C.c_double)),
                ("ind_div", _p(C.c_uint16)), ("pop_div", _p(C.c_uint16)), ("div_num_snps", _p(C.c_int32)),
                ("nhaps", _p(C.c_int32)), ("hdiv", _p(C.c_double)), ("ehhs", _p(C.c_double)),
                ("span_beg", C.c_int32), ("span_end", C.c_int32),
                ("cb", _p(C.c_uint64)), ("site_type", _p(C.c_uint64)), ("site_flag", _p(C.c_uint8)),
                ("reads_pushed", C.c_int64), ("reads_used", C.c_int64), ("aligned_bases", C.c_int64),
                ("tree_diff", _p(C.c_uint16))]


class Extras(C.Structure):
    """pb_region_extras: the PB_AN_THETA_W / FULI / LD_DPRIME arrays, [NW*P] each."""
    _fields_ = [("pop_segsites", _p(C.c_int32)), ("theta_w", _p(C.c_double)), ("fuli_d", _p(C.c_double)),
                ("fuli_ds", _p(C.c_double)), ("fuli_eta_e", _p(C.c_int32)), ("fuli_eta_s", _p(C.c_int32)),
                ("ld_kept", _p(C.c_int32)), ("ld_dprime", _p(C.c_double)), ("ld_complete", _p(C.c_int64))]


EXT_BITS = AN["THETA_W"] | AN["FULI"] | AN["LD_DPRIME"]


class Fst(C.Structure):
    """pb_region_fst: the PB_AN_FST arrays, [NW*P*P] each, indexed like pib (snn_p / snn_ge only with permutations)."""
    _fields_ = [("hud_num", _p(C.c_int64)), ("hud_den", _p(C.c_int64)), ("wc_num", _p(C.c_int64)), ("wc_den", _p(C.c_int64)),
                ("fst_hudson", _p(C.c_double)), ("fst_wc", _p(C.c_double)), ("snn", _p(C.c_double)), ("snn_p", _p(C.c_double)),
                ("snn_ge", _p(C.c_int64))]


class Abba(C.Structure):
    """pb_region_abba: the PB_AN_ABBA arrays, [NW*NT] each, index w*NT + t, and the triples the region ran with."""
    _fields_ = [("n_triples", C.c_int32), ("outgroup_pop", C.c_int32), ("triples", _p(C.c_int32)), ("sites", _p(C.c_int32)),
                ("abba", _p(C.c_int64)), ("baba", _p(C.c_int64)), ("fd_den", _p(C.c_int64)), ("fdm_den", _p(C.c_int64)),
                ("d", _p(C.c_double)), ("fd", _p(C.c_double)), ("fdm", _p(C.c_double))]


class Garud(C.Structure):
    """pb_region_garud: the PB_AN_GARUD arrays, [NW*P] each, index w*P + p."""
    _fields_ = [("n_hap", _p(C.c_int32)), ("c1", _p(C.c_int32)), ("c2", _p(C.c_int32)), ("c3", _p(C.c_int32)), ("hh", _p(C.c_int32)),
                ("h1", _p(C.c_double)), ("h12", _p(C.c_double)), ("h123", _p(C.c_double)), ("h2h1", _p(C.c_double))]


class Spectrum(C.Structure):
    """pb_region_spectrum: the PB_AN_SPECTRUM arrays; counts [NW*n_bins], index w*n_bins + set_off[s] + bin."""
    _fields_ = [("n_sets", C.c_int32), ("n_bins", C.c_int32), ("sets", _p(C.c_int32)), ("set_off", _p(C.c_int32)),
                ("counts", _p(C.c_int32))]


class NucdivMissing(C.Structure):
    """pb_region_nucdiv_missing: the PB_AN_NUCDIV_MISSING arrays; pi_* [NW*P] (w*P + p), dxy_* [NW*P*P] (w*P*P + i*P + (j-(i+1)))."""
    _fields_ = [("pi_sites", _p(C.c_int32)), ("pi_diffs", _p(C.c_int64)), ("pi_comps", _p(C.c_int64)), ("pi_missing", _p(C.c_int64)),
                ("pi", _p(C.c_double)), ("dxy_sites", _p(C.c_int32)), ("dxy_diffs", _p(C.c_int64)), ("dxy_comps", _p(C.c_int64)),
                ("dxy_missing", _p(C.c_int64)), ("dxy", _p(C.c_double))]


class PrintOpts(C.Structure):
    _fields_ = [("chrom", C.c_char_p), ("pop_names", _p(C.c_char_p)), ("sample_names", _p(C.c_char_p)),
                ("min_sites", C.c_int32), ("min_snps", C.c_int32), ("jc", C.c_int32), ("snp_output", C.c_int32),
                ("ref_name", C.c_char_p)]


def lib_path():
    return PKG / "_build" / "libpopbam_b200.so"


def build(verbose=False):
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-C", str(PKG / "csrc")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("building libpopbam_b200.so failed:\n" + r.stdout)
    if verbose:
        print(r.stdout)
    return lib_path()


_lib = None


def lib():
    """Load libpopbam_b200.so; raises if it has not been built (there is no other implementation)."""
    global _lib
    if _lib is None:
        so = lib_path()
        if not so.exists():
            raise RuntimeError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(popbam_b200 has no CPU fallback)" % so)
        L = C.CDLL(str(so))
        L.pb_create.restype = C.c_void_p
        L.pb_create.argtypes = [_p(Params), _p(Tables), _p(C.c_int)]
        L.pb_destroy.argtypes = [C.c_void_p]
        L.pb_last_error.restype = C.c_char_p
        L.pb_last_error.argtypes = [C.c_void_p]
        L.pb_version.restype = C.c_char_p
        L.pb_set_contig.argtypes = [C.c_void_p, C.c_int32, C.c_char_p, C.c_int64]
        L.pb_region_begin.argtypes = [C.c_void_p, C.c_uint32, C.c_int32, _p(C.c_int32), _p(C.c_int32)]
        L.pb_push_batch.argtypes = [C.c_void_p, _p(Batch)]
        L.pb_push_batch_async.argtypes = [C.c_void_p, _p(Batch)]
        L.pb_push_record.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]
        L.pb_region_end.argtypes = [C.c_void_p, _p(Result)]
        L.pb_region_launch.argtypes = [C.c_void_p]
        L.pb_region_wait.argtypes = [C.c_void_p, _p(Result)]
        L.pb_region_relaunch.argtypes = [C.c_void_p]
        L.pb_stream.restype = C.c_void_p
        L.pb_stream.argtypes = [C.c_void_p]
        L.pb_kernel_launches.restype = C.c_int64
        L.pb_kernel_launches.argtypes = [C.c_void_p]
        L.pb_stage_times.argtypes = [C.c_void_p, _p(C.c_double)]
        L.pb_region_path.argtypes = [C.c_void_p]
        L.pb_region_reruns.argtypes = [C.c_void_p]
        L.pb_window_grid.restype = C.c_int64
        L.pb_window_grid.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int64, _p(C.c_int32), _p(C.c_int32)]
        L.pb_build_errmod_tables.argtypes = [_p(C.c_double)] * 3
        L.pb_errmod_tables_cached_ex.argtypes = [_p(C.c_double)] * 3 + [C.c_char_p, _p(C.c_int)]
        L.pb_host_alloc.restype = C.c_void_p
        L.pb_host_alloc.argtypes = [C.c_size_t]
        L.pb_host_free.argtypes = [C.c_void_p]
        L.pb_format_window.restype = C.c_int64
        L.pb_format_window.argtypes = [C.c_void_p, _p(Result), C.c_int32, C.c_uint32, _p(PrintOpts), C.c_char_p, C.c_int64]
        L.pb_region_get_extras.argtypes = [C.c_void_p, _p(Extras)]
        L.pb_format_window_ext.restype = C.c_int64
        L.pb_format_window_ext.argtypes = [C.c_void_p, _p(Result), _p(Extras), C.c_int32, C.c_uint32, _p(PrintOpts), C.c_char_p, C.c_int64]
        L.pb_region_get_fst.argtypes = [C.c_void_p, _p(Fst)]
        L.pb_set_snn_perms.argtypes = [C.c_void_p, C.c_int64, C.c_uint64]
        L.pb_format_window_fst.restype = C.c_int64
        L.pb_format_window_fst.argtypes = [C.c_void_p, _p(Result), _p(Extras), _p(Fst), C.c_int32, C.c_uint32, _p(PrintOpts), C.c_char_p,
                                           C.c_int64]
        L.pb_region_get_abba.argtypes = [C.c_void_p, _p(Abba)]
        L.pb_set_abba.argtypes = [C.c_void_p, C.c_int32, C.c_int32, _p(C.c_int32)]
        L.pb_format_window_abba.restype = C.c_int64
        L.pb_format_window_abba.argtypes = [C.c_void_p, _p(Result), _p(Abba), C.c_int32, _p(PrintOpts), C.c_char_p, C.c_int64]
        L.pb_region_get_garud.argtypes = [C.c_void_p, _p(Garud)]
        L.pb_format_window_garud.restype = C.c_int64
        L.pb_format_window_garud.argtypes = [C.c_void_p, _p(Result), _p(Garud), C.c_int32, C.c_uint32, _p(PrintOpts), C.c_char_p, C.c_int64]
        L.pb_region_get_spectrum.argtypes = [C.c_void_p, _p(Spectrum)]
        L.pb_set_spectra.argtypes = [C.c_void_p, C.c_int32, _p(C.c_int32)]
        L.pb_format_spectrum_dadi.restype = C.c_int64
        L.pb_format_spectrum_dadi.argtypes = [C.c_void_p, _p(C.c_int32), _p(C.c_int64), _p(PrintOpts), C.c_char_p, C.c_char_p, C.c_int64]
        L.pb_region_get_nucdiv_missing.argtypes = [C.c_void_p, _p(NucdivMissing)]
        L.pb_format_window_nucdiv_missing.restype = C.c_int64
        L.pb_format_window_nucdiv_missing.argtypes = [C.c_void_p, _p(Result), _p(NucdivMissing), C.c_int32, C.c_int32, _p(PrintOpts),
                                                      C.c_char_p, C.c_int64]
        _lib = L
    return _lib


class PopbamError(RuntimeError):
    pass


class Context:
    """One pb_ctx (one GPU, one host thread)."""

    def __init__(self, params, tables=None):
        L = lib()
        st = C.c_int(0)
        tp = None
        if tables is not None:
            self._tables = Tables(*[a.ctypes.data_as(_p(C.c_double)) for a in tables])
            tp = C.byref(self._tables)
        self.h = L.pb_create(C.byref(params), tp, C.byref(st))
        if not self.h:
            raise PopbamError("pb_create failed (%d): %s" % (st.value, L.pb_last_error(None).decode()))
        self.L, self.params = L, params
        self.res = Result()
        self.ext = Extras()
        self.fst = Fst()
        self.abba = Abba()
        self.garud = Garud()
        self.spectrum = Spectrum()
        self.nucdiv_missing = NucdivMissing()

    def _chk(self, rc):
        if rc != 0:
            raise PopbamError("popbam_b200 error %d: %s" % (rc, self.L.pb_last_error(self.h).decode()))

    def close(self):
        if getattr(self, "h", None):
            self.L.pb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_contig(self, tid, ref_bytes):
        self._chk(self.L.pb_set_contig(self.h, tid, ref_bytes, len(ref_bytes)))

    def region_begin(self, analyses, win_beg, win_end):
        wb = np.ascontiguousarray(win_beg, dtype=np.int32)
        we = np.ascontiguousarray(win_end, dtype=np.int32)
        self._chk(self.L.pb_region_begin(self.h, analyses, len(wb), wb.ctypes.data_as(_p(C.c_int32)), we.ctypes.data_as(_p(C.c_int32))))

    def push_batch(self, batch):
        self._chk(self.L.pb_push_batch(self.h, C.byref(batch)))

    def push_batch_async(self, batch):
        """The arrays of `batch` must stay untouched until region_end / wait has returned."""
        self._chk(self.L.pb_push_batch_async(self.h, C.byref(batch)))

    def region_end(self):
        self._chk(self.L.pb_region_end(self.h, C.byref(self.res)))
        self._chk(self.L.pb_region_get_extras(self.h, C.byref(self.ext)))
        self._chk(self.L.pb_region_get_fst(self.h, C.byref(self.fst)))
        self._chk(self.L.pb_region_get_abba(self.h, C.byref(self.abba)))
        self._chk(self.L.pb_region_get_garud(self.h, C.byref(self.garud)))
        self._chk(self.L.pb_region_get_spectrum(self.h, C.byref(self.spectrum)))
        self._chk(self.L.pb_region_get_nucdiv_missing(self.h, C.byref(self.nucdiv_missing)))
        return self.res

    def launch(self):
        self._chk(self.L.pb_region_launch(self.h))

    def relaunch(self):
        self._chk(self.L.pb_region_relaunch(self.h))

    def wait(self):
        self._chk(self.L.pb_region_wait(self.h, C.byref(self.res)))
        self._chk(self.L.pb_region_get_extras(self.h, C.byref(self.ext)))
        self._chk(self.L.pb_region_get_fst(self.h, C.byref(self.fst)))
        self._chk(self.L.pb_region_get_abba(self.h, C.byref(self.abba)))
        self._chk(self.L.pb_region_get_garud(self.h, C.byref(self.garud)))
        self._chk(self.L.pb_region_get_spectrum(self.h, C.byref(self.spectrum)))
        self._chk(self.L.pb_region_get_nucdiv_missing(self.h, C.byref(self.nucdiv_missing)))
        return self.res

    def set_snn_perms(self, n_perms, seed=0):
        """Snn permutations per (window, population pair) for the regions that follow (PB_AN_FST); 0 = none."""
        self._chk(self.L.pb_set_snn_perms(self.h, n_perms, seed))

    def set_abba(self, outgroup_pop, triples):
        """Triples [(P1, P2, P3), ...] against population outgroup_pop for the PB_AN_ABBA regions that follow; [] clears them."""
        flat = np.ascontiguousarray([k for t in triples for k in t], dtype=np.int32)
        self._chk(self.L.pb_set_abba(self.h, outgroup_pop, len(flat) // 3, flat.ctypes.data_as(_p(C.c_int32)) if len(flat) else None))

    def set_spectra(self, sets):
        """Spectrum sets [(P1,), (P1, P2), (P1, P2, P3), ...] for the PB_AN_SPECTRUM regions that follow; [] clears them."""
        flat = np.ascontiguousarray([k for t in sets for k in (list(t) + [-1, -1])[:3]], dtype=np.int32)
        self._chk(self.L.pb_set_spectra(self.h, len(flat) // 3, flat.ctypes.data_as(_p(C.c_int32)) if len(flat) else None))

    def stage_times(self):
        ms = (C.c_double * 4)()
        self._chk(self.L.pb_stage_times(self.h, ms))
        return list(ms)

    def kernel_launches(self):
        return self.L.pb_kernel_launches(self.h)

    def path(self):
        """1: the last region took the counting pileup (k_pile_reads), 0: the single-kernel pileup."""
        return self.L.pb_region_path(self.h)

    def reruns(self):
        return self.L.pb_region_reruns(self.h)

    def text(self, analysis, opts, windows=None):
        out = []
        buf = C.create_string_buffer(1 << 20)

        def fmt(w, buf):
            if analysis & AN["ABBA"]:
                return self.L.pb_format_window_abba(self.h, C.byref(self.res), C.byref(self.abba), w, C.byref(opts), buf, len(buf))
            if analysis & AN["GARUD"]:
                return self.L.pb_format_window_garud(self.h, C.byref(self.res), C.byref(self.garud), w, analysis, C.byref(opts), buf, len(buf))
            if analysis & AN["FST"]:
                return self.L.pb_format_window_fst(self.h, C.byref(self.res), C.byref(self.ext), C.byref(self.fst), w, analysis, C.byref(opts),
                                                   buf, len(buf))
            return self.L.pb_format_window_ext(self.h, C.byref(self.res), C.byref(self.ext), w, analysis, C.byref(opts), buf, len(buf))
        for w in (range(self.res.n_windows) if windows is None else windows):
            k = fmt(w, buf)
            if k < 0:
                raise PopbamError("pb_format_window failed: %d" % k)
            if k >= len(buf):
                buf = C.create_string_buffer(int(k) + 16)
                k = fmt(w, buf)
            out.append(buf.raw[:k].decode())
        return "".join(out)

    def missing_text(self, pairs, opts, windows=None):
        """Lines of `nucdiv --missing`'s PREFIX_pi.txt (pairs = 0) or PREFIX_dxy.txt (pairs = 1), without the header line."""
        out = []
        buf = C.create_string_buffer(1 << 16)
        for w in (range(self.res.n_windows) if windows is None else windows):
            k = self.L.pb_format_window_nucdiv_missing(self.h, C.byref(self.res), C.byref(self.nucdiv_missing), w, pairs, C.byref(opts), buf, len(buf))
            if k < 0:
                raise PopbamError("pb_format_window_nucdiv_missing failed: %d" % k)
            if k >= len(buf):
                buf = C.create_string_buffer(int(k) + 16)
                k = self.L.pb_format_window_nucdiv_missing(self.h, C.byref(self.res), C.byref(self.nucdiv_missing), w, pairs, C.byref(opts), buf,
                                                           len(buf))
            out.append(buf.raw[:k].decode())
        return "".join(out)
