"""ctypes binding of libdbslmm_b200.so (the C ABI in include/dbslmm_b200.h).

The product path has no CPU fallback: if the shared library is missing or no B200 is
visible, constructing an Engine raises.
"""
import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DBSLMM_B200_LIB") or os.path.join(_PKG, "libdbslmm_b200.so")      # override: kernel-variant builds (tools/build_variants.sh)

SOLVER_CHOLESKY = 0
SOLVER_PCG = 1
FLAG_KEEP_INT_GRAM = 1
FLAG_FULL_SIGMA = 2
FLAG_PLAN_CACHED = 4
FLAG_PANEL_SUBSET = 8
LD_WIND_COORD = 0
LD_WIND_SNPS = 1
LD_MAX_ANNOT = 4096
ERR_SINK = -5
# dbslmm_b200_ld_sink: (user, a0, a1, off[a1 - a0 + 1], b, r) -> 0 to go on
LD_SINK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int32),
                      C.POINTER(C.c_double))

EXPORTS = [
    "dbslmm_b200_abi_version", "dbslmm_b200_device_count", "dbslmm_b200_create", "dbslmm_b200_destroy",
    "dbslmm_b200_last_error", "dbslmm_b200_load_bed", "dbslmm_b200_snp_stats", "dbslmm_b200_plan_shards",
    "dbslmm_b200_fit", "dbslmm_b200_fit_multi", "dbslmm_b200_host_alloc", "dbslmm_b200_host_free", "dbslmm_b200_score", "dbslmm_b200_score_prefetch", "dbslmm_b200_score_stream", "dbslmm_b200_ldscore", "dbslmm_b200_ldscore_annot", "dbslmm_b200_ld_windows", "dbslmm_b200_ld_pairs", "dbslmm_b200_get_row_codes", "dbslmm_b200_get_block_sigma",
    "dbslmm_b200_get_block_factor", "dbslmm_b200_get_block_gram", "dbslmm_b200_get_block_iters",
]


class Timing(C.Structure):
    _fields_ = [("h2d_ms", C.c_float), ("decode_ms", C.c_float), ("gram_ms", C.c_float),
                ("solve_ms", C.c_float), ("d2h_ms", C.c_float), ("total_ms", C.c_float),
                ("n_launches", C.c_int32), ("n_chol_launches", C.c_int32),
                ("gram_ops", C.c_double), ("solve_flops", C.c_double), ("decode_bytes", C.c_double),
                ("chol_ms", C.c_double), ("class_ms", C.c_float * 4), ("streamed", C.c_int32), ("n_blocks_missing", C.c_int32)]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_}
        d["class_ms"] = list(self.class_ms)
        return d


class FitArgs(C.Structure):
    _fields_ = [("n_blocks", C.c_int32), ("s_off", C.c_void_p), ("s_pos", C.c_void_p), ("s_z", C.c_void_p),
                ("l_off", C.c_void_p), ("l_pos", C.c_void_p), ("l_z", C.c_void_p),
                ("n_folds", C.c_int32), ("sigma_s", C.c_void_p), ("n_obs", C.c_int64), ("tau", C.c_double),
                ("solver", C.c_int32), ("flags", C.c_int32),
                ("beta_s_out", C.c_void_p), ("beta_l_out", C.c_void_p), ("block_status_out", C.c_void_p),
                ("timing", C.POINTER(Timing)),
                ("test_bed", C.c_void_p), ("test_n_snp", C.c_int64), ("test_n_total", C.c_int32),
                ("test_indicator", C.c_void_p), ("s_tpos", C.c_void_p), ("l_tpos", C.c_void_p),
                ("variance_out", C.c_void_p),
                ("bed", C.c_void_p), ("bed_n_snp", C.c_int64), ("bed_n_ref", C.c_int32),
                ("quadform_out", C.c_void_p)]


_lib = None


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -m dbslmm_b200.build` "
                               "(the B200 path has no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        lib.dbslmm_b200_last_error.restype = C.c_char_p
        lib.dbslmm_b200_last_error.argtypes = [C.c_void_p]
        lib.dbslmm_b200_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        lib.dbslmm_b200_destroy.argtypes = [C.c_void_p]
        lib.dbslmm_b200_destroy.restype = None
        lib.dbslmm_b200_load_bed.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32]
        lib.dbslmm_b200_snp_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        lib.dbslmm_b200_plan_shards.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                                C.c_void_p, C.c_void_p]
        lib.dbslmm_b200_fit.argtypes = [C.c_void_p, C.POINTER(FitArgs)]
        lib.dbslmm_b200_fit_multi.argtypes = [C.POINTER(C.c_void_p), C.c_int32, C.POINTER(FitArgs)]
        lib.dbslmm_b200_host_alloc.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]
        lib.dbslmm_b200_host_free.argtypes = [C.c_void_p, C.c_void_p]
        lib.dbslmm_b200_host_free.restype = None
        lib.dbslmm_b200_score.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64,
                                          C.c_void_p, C.c_int32, C.c_void_p, C.POINTER(C.c_float)]
        lib.dbslmm_b200_score_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64,
                                                 C.c_void_p, C.c_int32, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.POINTER(C.c_int32), C.POINTER(C.c_float)]
        lib.dbslmm_b200_ldscore.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                            C.c_int32, C.c_int32, C.c_void_p, C.c_double, C.c_double, C.c_int64, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
        lib.dbslmm_b200_ldscore_annot.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                                  C.c_int32, C.c_int32, C.c_void_p, C.c_double, C.c_double, C.c_int64,
                                                  C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                  C.POINTER(C.c_float)]
        lib.dbslmm_b200_ld_pairs.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                             C.c_int32, C.c_void_p, C.c_int32, C.c_double, C.c_double, C.c_int64, LD_SINK,
                                             C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                             C.POINTER(C.c_float)]
        lib.dbslmm_b200_ld_windows.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_void_p]
        lib.dbslmm_b200_score_prefetch.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32]
        lib.dbslmm_b200_get_row_codes.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32]
        lib.dbslmm_b200_get_block_sigma.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        lib.dbslmm_b200_get_block_factor.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        lib.dbslmm_b200_get_block_gram.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.dbslmm_b200_get_block_iters.argtypes = [C.c_void_p, C.c_int32]
        _lib = lib
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data


def ld_windows(coord, max_dist, m=None):
    """The window rule of Engine.ldscore over the kept SNPs of one chromosome (host code, no GPU): (lo, hi) int32 arrays,
    W(k) = lo[k]..hi[k] inclusive.  coord=None: a window of max_dist SNPs over m SNPs."""
    if coord is not None:
        coord = np.ascontiguousarray(coord, np.float64)
        m = coord.size
    lo = np.zeros(max(int(m), 1), np.int32)
    hi = np.zeros(max(int(m), 1), np.int32)
    if load().dbslmm_b200_ld_windows(_ptr(coord), int(m), float(max_dist), lo.ctypes.data, hi.ctypes.data) != 0:
        raise ValueError("ld_windows: bad arguments")
    return lo[:m], hi[:m]


class EngineError(RuntimeError):
    pass


class Engine:
    """One handle = one GPU."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.dbslmm_b200_create(int(device), C.byref(h))
        if rc != 0:
            raise EngineError(f"dbslmm_b200_create(device={device}) failed with {rc}: no usable sm_100 GPU "
                              "(there is no CPU fallback)")
        self.h = h
        self.n_snp = 0
        self.n_ref = 0
        self._keep = []
        self._outbuf = {}

    def close(self):
        if getattr(self, "h", None):
            self.lib.dbslmm_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc < 0:
            raise EngineError(f"{what} failed ({rc}): {self.lib.dbslmm_b200_last_error(self.h).decode()}")
        return rc

    def load_bed(self, bed, n_ref):
        """bed: uint8[n_snp, ceil(n_ref/4)] -- payload after the 3 magic bytes (numpy or pinned torch-backed)."""
        bed = np.ascontiguousarray(bed, dtype=np.uint8)
        pitch = (n_ref + 3) // 4
        n_snp = bed.size // pitch
        self._check(self.lib.dbslmm_b200_load_bed(self.h, bed.ctypes.data, n_snp, n_ref), "load_bed")
        self._bed_keep = bed          # the upload is asynchronous: the buffer must outlive this call (see the C header)
        self.n_snp, self.n_ref = n_snp, n_ref

    def snp_stats(self):
        maf = np.zeros(self.n_snp, np.float64)
        nn = np.zeros(self.n_snp, np.int32)
        self._check(self.lib.dbslmm_b200_snp_stats(self.h, maf.ctypes.data, nn.ctypes.data), "snp_stats")
        return maf, nn

    def plan_shards(self, m_s, m_l, n_ref, n_ranks):
        m_s = np.ascontiguousarray(m_s, np.int32)
        m_l = None if m_l is None else np.ascontiguousarray(m_l, np.int32)
        owner = np.zeros(m_s.size, np.int32)
        cost = np.zeros(n_ranks, np.float64)
        rc = self.lib.dbslmm_b200_plan_shards(m_s.size, m_s.ctypes.data, _ptr(m_l), n_ref, n_ranks,
                                              owner.ctypes.data, cost.ctypes.data)
        if rc != 0:
            raise EngineError(f"plan_shards failed ({rc})")
        return owner, cost

    def fit(self, s_off, s_pos, s_z, l_off=None, l_pos=None, l_z=None, *, sigma_s, n_obs, tau=0.8,
            solver=SOLVER_CHOLESKY, flags=0, test=None, bed=None, n_ref=None, reuse_outputs=False):
        """Returns dict(beta_s[n_folds, S], beta_l[n_folds, L], status[n_blocks], n_bad, timing[, variance]).
        test = dict(bed=uint8[n_snp_t, pitch_t], n_total=int, indicator=int[n_total], s_tpos=int[S], l_tpos=int[L])
        switches the fork's asymptotic-variance side channel on: variance[n_folds, n_blocks, n_test].
        bed = uint8[n_snp, ceil(n_ref/4)] (with n_ref): the reference panel travels with the call, as in the reference's
        DBSLMMFIT::est(bed_str, ...); its upload overlaps the fit, and it stays resident afterwards."""
        s_off = np.ascontiguousarray(s_off, np.int32)
        s_pos = np.ascontiguousarray(s_pos, np.int32)
        s_z = np.ascontiguousarray(s_z, np.float64)
        nb = s_off.size - 1
        sig = np.atleast_1d(np.asarray(sigma_s, np.float64)).copy()
        nf = sig.size
        def out(name, shape):
            if not reuse_outputs:
                return np.zeros(shape, np.float64)
            buf = self._outbuf.get(name)
            if buf is None or buf.shape != shape:
                buf = self._outbuf[name] = np.zeros(shape, np.float64)
            return buf
        beta_s = out("beta_s", (nf, s_pos.size))
        if l_off is not None:
            l_off = np.ascontiguousarray(l_off, np.int32)
            l_pos = np.ascontiguousarray(l_pos, np.int32)
            l_z = np.ascontiguousarray(l_z, np.float64)
            beta_l = out("beta_l", (nf, max(l_pos.size, 1)))
            nl = l_pos.size
        else:
            beta_l = None
            nl = 0
        status = np.zeros(max(nb, 1), np.int32)
        tm = Timing()
        a = FitArgs(nb, s_off.ctypes.data, _ptr(s_pos), _ptr(s_z), _ptr(l_off), _ptr(l_pos), _ptr(l_z),
                    nf, sig.ctypes.data, int(n_obs), float(tau), int(solver), int(flags),
                    beta_s.ctypes.data, _ptr(beta_l), status.ctypes.data, C.pointer(tm))
        var = None
        if test is not None:
            tbed = np.ascontiguousarray(test["bed"], np.uint8)
            ind = np.ascontiguousarray(test["indicator"], np.int32)
            stp = np.ascontiguousarray(test["s_tpos"], np.int32)
            ltp = None if l_off is None else np.ascontiguousarray(test["l_tpos"], np.int32)
            n_total = int(test["n_total"])
            var = np.zeros((nf, max(nb, 1), max(int((ind != 0).sum()), 1)), np.float64)
            a.test_bed, a.test_n_snp, a.test_n_total = tbed.ctypes.data, tbed.size // ((n_total + 3) // 4), n_total
            a.test_indicator, a.s_tpos, a.l_tpos, a.variance_out = ind.ctypes.data, _ptr(stp), _ptr(ltp), var.ctypes.data
            self._keep = [tbed, ind, stp, ltp]
        if bed is not None:
            bed = np.ascontiguousarray(bed, dtype=np.uint8)
            pitch = (int(n_ref) + 3) // 4
            a.bed, a.bed_n_snp, a.bed_n_ref = bed.ctypes.data, bed.size // pitch, int(n_ref)
            self.n_snp, self.n_ref = bed.size // pitch, int(n_ref)
        rc = self._check(self.lib.dbslmm_b200_fit(self.h, C.byref(a)), "fit")
        out = {"beta_s": beta_s, "beta_l": None if beta_l is None else beta_l[:, :nl], "status": status[:nb],
               "n_bad": rc, "timing": tm.as_dict()}
        if var is not None:
            out["variance"] = var
        return out

    def quadform(self, off, pos, z, tau=1.0):
        """z_b' Sigma_b z_b per block (Sigma_b = tau X'X/n + (1-tau) I of the block's SNPs): the `deno` of the reference's
        external-validation tool `valid` (scr/validate.cpp:255-258, tau = 1).  Returns float64[n_blocks]."""
        off = np.ascontiguousarray(off, np.int32)
        pos = np.ascontiguousarray(pos, np.int32)
        z = np.ascontiguousarray(z, np.float64)
        nb = off.size - 1
        out = np.zeros(max(nb, 1), np.float64)
        a = FitArgs()
        a.n_blocks, a.s_off, a.s_pos, a.s_z = nb, off.ctypes.data, _ptr(pos), _ptr(z)
        a.tau, a.solver, a.quadform_out = float(tau), SOLVER_CHOLESKY, out.ctypes.data
        self._check(self.lib.dbslmm_b200_fit(self.h, C.byref(a)), "fit(quadform)")
        return out[:nb]

    def score_prefetch(self, bed_val, n_val):
        """Announce the validation panel of the next score(None, ...) call: uploaded in the shadow of the next fit."""
        bed_val = np.ascontiguousarray(bed_val, np.uint8)
        pitch = (n_val + 3) // 4
        self._val_keep = bed_val                       # must outlive the next score call (see the C header)
        self._check(self.lib.dbslmm_b200_score_prefetch(self.h, bed_val.ctypes.data, bed_val.size // pitch, int(n_val)), "score_prefetch")
        self._val_n = int(n_val)

    def score(self, bed_val, n_val, pos, beta, flip=None):
        """PRS over a validation panel: returns (scores[n_folds, n_val], kernel_ms).  bed_val = None: the panel announced
        by score_prefetch / left resident by the previous call."""
        if bed_val is None:
            n_val = self._val_n
            bptr, n_snp_val = None, 0
        else:
            bed_val = np.ascontiguousarray(bed_val, np.uint8)
            pitch = (n_val + 3) // 4
            bptr, n_snp_val = bed_val.ctypes.data, bed_val.size // pitch
            self._val_n = int(n_val)
        pos = np.ascontiguousarray(pos, np.int32)
        beta = np.ascontiguousarray(np.atleast_2d(beta), np.float64)
        fl = None if flip is None else np.ascontiguousarray(flip, np.uint8)
        out = np.zeros((beta.shape[0], n_val), np.float64)
        ms = C.c_float(0)
        self._check(self.lib.dbslmm_b200_score(self.h, bptr, n_snp_val, n_val, pos.ctypes.data, _ptr(fl),
                                               pos.size, beta.ctypes.data, beta.shape[0], out.ctypes.data, C.byref(ms)), "score")
        return out, ms.value

    def score_stream(self, bed_val, n_val, pos, beta, flip=None, chunk_bytes=0):
        """PRS over a target panel of any size, streamed through the GPU chunk by chunk (dbslmm_b200_score_stream).
        bed_val: uint8 payload after the magic bytes ([n_snp, ceil(n_val/4)] or flat), e.g. a numpy.memmap of the .bed
        opened with offset=3: only the rows named by pos are read.  Returns (scores[n_folds, n_val], cnt[n_val], cnt2[n_val])
        with PLINK's CNT / CNT2; the summed kernel time of the call is left in self.last_kernel_ms and the number of scored
        rows without a called genotype in self.last_empty_rows."""
        n_val = int(n_val)
        pitch = (n_val + 3) // 4
        if not (isinstance(bed_val, np.ndarray) and bed_val.dtype == np.uint8 and bed_val.flags.c_contiguous):
            bed_val = np.ascontiguousarray(bed_val, np.uint8)          # a contiguous memmap is used in place, never copied
        pos = np.ascontiguousarray(pos, np.int32)
        beta = np.ascontiguousarray(np.atleast_2d(beta), np.float64)
        if beta.shape[1] != pos.size or (flip is not None and np.size(flip) != pos.size):
            raise ValueError("score_stream: beta must be [n_folds, pos.size] and flip [pos.size]")
        fl = None if flip is None else np.ascontiguousarray(flip, np.uint8)
        out = np.zeros((beta.shape[0], n_val), np.float64)
        empty = C.c_int32(0)
        cnt = np.zeros(n_val, np.int32)
        cnt2 = np.zeros(n_val, np.int32)
        ms = C.c_float(0)
        self._check(self.lib.dbslmm_b200_score_stream(self.h, bed_val.ctypes.data, bed_val.size // pitch, n_val, pos.ctypes.data,
                                                      _ptr(fl), pos.size, beta.ctypes.data, beta.shape[0], int(chunk_bytes),
                                                      out.ctypes.data, cnt.ctypes.data, cnt2.ctypes.data, C.byref(empty),
                                                      C.byref(ms)),
                    "score_stream")
        self.last_kernel_ms = ms.value
        self.last_empty_rows = empty.value
        return out, cnt, cnt2

    def ldscore(self, bed, n_ref, rows, chr_off, coord=None, *, max_dist, maf_min=0.0, segment_rows=0, stats_only=False,
                annot=None):
        """LD Scores of .bed rows `rows` (dbslmm_b200_ldscore, `ldsc.py --l2`): chromosome c is rows[chr_off[c]:chr_off[c+1]],
        in coordinate order.  coord (float64[rows.size], cM or bp) gives a window of |c_k - c_j| <= max_dist; coord=None a
        window of max_dist kept SNPs.  bed: uint8 payload after the magic bytes ([n_snp, ceil(n_ref/4)] or flat), e.g. a
        numpy.memmap of the .bed opened with offset=3: only the listed rows are read.  Returns (l2, kept, maf, guard):
        l2 float64[rows.size] (NaN where not kept), kept bool, maf float64, guard bool[n_chr] (the window of a chromosome's
        last kept SNP reaches its first).  stats_only=True stops after the statistics pass (l2 is then None).  The summed
        kernel time is left in self.last_kernel_ms.
        annot (float64 [rows.size, C], `ldsc.py --l2 --annot`): partitioned LD Scores (dbslmm_b200_ldscore_annot), l2 is then
        [rows.size, C], column c the window sum of r2adj(j, k) a_kc."""
        n_ref = int(n_ref)
        pitch = (n_ref + 3) // 4
        if not (isinstance(bed, np.ndarray) and bed.dtype == np.uint8 and bed.flags.c_contiguous):
            bed = np.ascontiguousarray(bed, np.uint8)                  # a contiguous memmap is used in place, never copied
        rows = np.ascontiguousarray(rows, np.int32)
        chr_off = np.ascontiguousarray(chr_off, np.int32)
        if coord is not None:
            coord = np.ascontiguousarray(coord, np.float64)
            if coord.size != rows.size:
                raise ValueError("ldscore: coord must have one entry per row")
        n_chr = chr_off.size - 1
        if n_chr < 0:
            raise ValueError("ldscore: chr_off needs n_chr + 1 entries")
        if annot is not None:
            annot = np.ascontiguousarray(annot, np.float64)
            if annot.ndim != 2 or annot.shape[0] != rows.size:
                raise ValueError("ldscore: annot must be [rows.size, n_annot]")
        l2 = np.zeros(rows.size if annot is None else annot.shape, np.float64)
        kept = np.zeros(rows.size, np.uint8)
        maf = np.zeros(rows.size, np.float64)
        guard = np.zeros(max(n_chr, 1), np.int32)
        ms = C.c_float(0)
        common = (self.h, bed.ctypes.data, bed.size // pitch, n_ref, rows.ctypes.data, rows.size, chr_off.ctypes.data, n_chr,
                  LD_WIND_SNPS if coord is None else LD_WIND_COORD, _ptr(coord), float(max_dist), float(maf_min), int(segment_rows))
        outs = (kept.ctypes.data, maf.ctypes.data, None if stats_only else l2.ctypes.data, guard.ctypes.data, C.byref(ms))
        if annot is None:
            self._check(self.lib.dbslmm_b200_ldscore(*common, *outs), "ldscore")
        else:
            self._check(self.lib.dbslmm_b200_ldscore_annot(*common, annot.ctypes.data, annot.shape[1], *outs), "ldscore_annot")
        self.last_kernel_ms = ms.value
        return None if stats_only else l2, kept.astype(bool), maf, guard[:n_chr].astype(bool)

    def ld_pairs(self, bed, n_ref, rows, chr_off, coord, *, max_snps=10, max_dist=1000000.0, r2_min=0.2, segment_rows=0):
        """SNP pairs within a window and their r (dbslmm_b200_ld_pairs, `plink --r2`): chromosome c is
        rows[chr_off[c]:chr_off[c+1]], coord (float64[rows.size]) its base-pair positions.  A pair (a, b), a < b positions in
        rows, is kept when b - a <= max_snps - 1, coord[b] - coord[a] <= max_dist and r^2 >= r2_min.  Returns (a, b, r):
        int64, int32 and float64 arrays in ascending (a, b) order.  self.last_usable (bool[rows.size]: rows that can form a
        pair), self.last_n_miss_pairs (pairs with a SNP with missing calls) and self.last_kernel_ms are left behind."""
        n_ref = int(n_ref)
        pitch = (n_ref + 3) // 4
        if not (isinstance(bed, np.ndarray) and bed.dtype == np.uint8 and bed.flags.c_contiguous):
            bed = np.ascontiguousarray(bed, np.uint8)
        rows = np.ascontiguousarray(rows, np.int32)
        chr_off = np.ascontiguousarray(chr_off, np.int32)
        coord = np.ascontiguousarray(coord, np.float64)
        if coord.size != rows.size:
            raise ValueError("ld_pairs: coord must have one entry per row")
        if chr_off.size < 1:
            raise ValueError("ld_pairs: chr_off needs n_chr + 1 entries")
        parts_a, parts_b, parts_r = [], [], []
        err = []

        def take(user, a0, a1, off, b, r):
            try:
                o = np.ctypeslib.as_array(off, (a1 - a0 + 1,)).copy()
                n = int(o[-1])
                parts_a.append(np.repeat(np.arange(a0, a1, dtype=np.int64), np.diff(o)))
                parts_b.append(np.ctypeslib.as_array(b, (n,)).copy() if n else np.zeros(0, np.int32))
                parts_r.append(np.ctypeslib.as_array(r, (n,)).copy() if n else np.zeros(0, np.float64))
                return 0
            except BaseException as e:        # an exception must not cross the C frames
                err.append(e)
                return 1

        sink = LD_SINK(take)
        usable = np.zeros(rows.size, np.uint8)
        n_pairs, n_miss, ms = C.c_int64(0), C.c_int64(0), C.c_float(0)
        rc = self.lib.dbslmm_b200_ld_pairs(self.h, bed.ctypes.data, bed.size // pitch, n_ref, rows.ctypes.data, rows.size,
                                           chr_off.ctypes.data, chr_off.size - 1, coord.ctypes.data, int(max_snps),
                                           float(max_dist), float(r2_min), int(segment_rows), sink, None, usable.ctypes.data,
                                           C.byref(n_pairs), C.byref(n_miss), C.byref(ms))
        if err:
            raise err[0]
        self._check(rc, "ld_pairs")
        self.last_usable = usable.astype(bool)
        self.last_n_miss_pairs = n_miss.value
        self.last_kernel_ms = ms.value
        cat = lambda p, t: np.concatenate(p) if p else np.zeros(0, t)
        a, b, r = cat(parts_a, np.int64), cat(parts_b, np.int32), cat(parts_r, np.float64)
        assert a.size == n_pairs.value
        return a, b, r

    # ---- inspection hooks (parity tests)
    def row_codes(self, block, j, n, plane=0):
        """int8 codes of SNP j of `block` in the last fit: plane 0 = allele counts, plane 1 = call mask."""
        out = np.zeros(n, np.int8)
        self._check(self.lib.dbslmm_b200_get_row_codes(self.h, int(block), int(j), int(plane), out.ctypes.data, n), "get_row_codes")
        return out

    def block_sigma(self, block, m):
        out = np.zeros((m, m), np.float64)
        self._check(self.lib.dbslmm_b200_get_block_sigma(self.h, int(block), out.ctypes.data), "get_block_sigma")
        return out

    def block_factor(self, block, m):
        """(L, y) of `block` from the last fold of the last Cholesky fit: L = m x m lower-triangular factor of
        K = Sigma + c diag(1_small, 0_large) (small SNPs first), y = L^-1 z."""
        L = np.zeros((m, m), np.float64)
        y = np.zeros(m, np.float64)
        self._check(self.lib.dbslmm_b200_get_block_factor(self.h, int(block), L.ctypes.data, y.ctypes.data), "get_block_factor")
        return L, y

    def block_gram(self, block, m):
        q = np.zeros((m, m), np.int32)
        a = np.zeros((m, m), np.int32)
        n = np.zeros((m, m), np.int32)
        self._check(self.lib.dbslmm_b200_get_block_gram(self.h, int(block), q.ctypes.data, a.ctypes.data,
                                                        n.ctypes.data), "get_block_gram")
        return q, a, n

    def block_iters(self, block):
        return self._check(self.lib.dbslmm_b200_get_block_iters(self.h, int(block)), "get_block_iters")


def fit_multi(engines, s_off, s_pos, s_z, l_off=None, l_pos=None, l_z=None, *, sigma_s, n_obs, bed, n_ref, tau=0.8,
              solver=SOLVER_CHOLESKY):
    """dbslmm_b200_fit_multi: one fit fanned out over several handles (normally one per GPU); the panel must come with the
    call.  Returns dict(beta_s[n_folds, S], beta_l[n_folds, L], status[n_blocks], n_bad, timing)."""
    lib = load()
    s_off = np.ascontiguousarray(s_off, np.int32); s_pos = np.ascontiguousarray(s_pos, np.int32)
    s_z = np.ascontiguousarray(s_z, np.float64)
    nb = s_off.size - 1
    sig = np.atleast_1d(np.asarray(sigma_s, np.float64)).copy()
    nf = sig.size
    beta_s = np.zeros((nf, s_pos.size), np.float64)
    if l_off is not None:
        l_off = np.ascontiguousarray(l_off, np.int32); l_pos = np.ascontiguousarray(l_pos, np.int32)
        l_z = np.ascontiguousarray(l_z, np.float64)
        beta_l = np.zeros((nf, max(l_pos.size, 1)), np.float64)
        nl = l_pos.size
    else:
        beta_l, nl = None, 0
    status = np.zeros(max(nb, 1), np.int32)
    tm = Timing()
    bed = np.ascontiguousarray(bed, np.uint8)
    pitch = (int(n_ref) + 3) // 4
    a = FitArgs(nb, s_off.ctypes.data, _ptr(s_pos), _ptr(s_z), _ptr(l_off), _ptr(l_pos), _ptr(l_z),
                nf, sig.ctypes.data, int(n_obs), float(tau), int(solver), 0,
                beta_s.ctypes.data, _ptr(beta_l), status.ctypes.data, C.pointer(tm))
    a.bed, a.bed_n_snp, a.bed_n_ref = bed.ctypes.data, bed.size // pitch, int(n_ref)
    hs = (C.c_void_p * len(engines))(*[e.h for e in engines])
    rc = lib.dbslmm_b200_fit_multi(hs, len(engines), C.byref(a))
    if rc < 0:
        raise EngineError(f"fit_multi failed ({rc}): {lib.dbslmm_b200_last_error(engines[0].h).decode()}")
    return {"beta_s": beta_s, "beta_l": None if beta_l is None else beta_l[:, :nl], "status": status[:nb], "n_bad": rc,
            "timing": tm.as_dict()}
