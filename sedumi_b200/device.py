"""Device-resident hot path: Python binding of libsedumi_b200's `*_dev` entry points.

This is the library's public API for callers that keep the iteration state in HBM (the
benchmark's `value` leg, and any host that wants to chain the kernels without crossing the
MEX boundary between them).  torch is used only for device memory and streams -- every
arithmetic step is one of our CUDA kernels, reached through the C-ABI in
include/sedumi_b200.h.  There is no CPU fallback: importing works without a GPU (so the
symbol table can be checked), but any compute call raises when no device is present.

One `HotPath` object = one problem (iteration-invariant structure uploaded once) and runs
the reference's per-iteration recipe (sedumi.m:442-466 + the solves of wrapPcg.m:56-59):

    invcholfac -> getada1 -> [getada2] -> getada3 -> blkchol -> nsolve x (fwblkslv, ./d, bwblkslv)
    -> npsdscale x psdscale
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libsedumi_b200.so")
_lib = None

I64 = C.c_int64
VP = C.c_void_p


class SB200Error(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load libsedumi_b200.so (raises ImportError when it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise ImportError(f"{_LIB_PATH} missing: run __graft_entry__.build() (nvcc, sm_100a) first")
        L = C.CDLL(_LIB_PATH)
        L.sb200_last_error.restype = C.c_char_p
        L.sb200_kernel_launches.restype = I64
        L.sb200_stream.restype = VP
        L.sb200_chol_plan_nnzL.restype = I64
        L.sb200_chol_plan_rect_size.restype = I64
        L.sb200_ada_plan_nnz.restype = I64
        L.sb200_psd_plan_lenud.restype = I64
        L.sb200_chol_plan_lb_dev.restype = VP
        L.sb200_wrappcg_full_work.restype = I64
        _lib = L
    return _lib


def check(rc: int, who: str = "sb200") -> None:
    if rc != 0:
        raise SB200Error(f"{who}: {lib().sb200_last_error().decode(errors='replace')}")


def _i64(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a).ravel(), dtype=np.int64)


def _p(a):
    """ctypes pointer of a numpy array or torch tensor (device or host)."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(VP)
    return VP(a.data_ptr())


EXPORTS = [
    "sb200_init", "sb200_shutdown", "sb200_last_error", "sb200_device_count", "sb200_sync", "sb200_stream",
    "sb200_kernel_launches", "sb200_xfer_bytes", "sb200_dev_alloc", "sb200_dev_free", "sb200_h2d", "sb200_d2h",
    "sb200_chol_plan_create", "sb200_chol_plan_destroy", "sb200_chol_plan_nnzL", "sb200_chol_plan_rect_size",
    "sb200_blkchol_dev", "sb200_chol_rect_to_csc_dev", "sb200_chol_csc_to_rect_dev", "sb200_blkchol",
    "sb200_fwblkslv_dev", "sb200_bwblkslv_dev", "sb200_ldl_solve_dev", "sb200_chol_shard_create", "sb200_chol_shard_info",
    "sb200_blkchol_shard_local_dev", "sb200_blkchol_shard_top_dev", "sb200_fw_shard_local_dev", "sb200_solve_shard_top_dev",
    "sb200_bw_shard_finish_dev", "sb200_fwblkslv", "sb200_bwblkslv", "sb200_fwblkslv_sparse",
    "sb200_psd_plan_get", "sb200_psd_plan_lenud", "sb200_psd_plan_sumn", "sb200_invcholfac_dev", "sb200_psdscale_dev",
    "sb200_invcholfac", "sb200_psdscale", "sb200_invcholfac_h", "sb200_psdscale_h", "sb200_psdframeit_h", "sb200_psdinvjmul_h", "sb200_urotorder_h", "sb200_givensrot_h", "sb200_psdframeit_dev", "sb200_psdinvjmul_dev", "sb200_psdframeit",
    "sb200_psdinvjmul", "sb200_urotorder", "sb200_givensrot", "sb200_urotorder_dev", "sb200_givensrot_dev", "sb200_dpr1fact", "sb200_dpr1solve", "sb200_prof_begin", "sb200_prof_end", "sb200_graph_begin", "sb200_graph_end", "sb200_graph_launch",
    "sb200_graph_destroy",
    "sb200_ada_plan_get", "sb200_ada_plan_get_h", "sb200_ada_plan_nnz", "sb200_ada_plan_retain", "sb200_ada_plan_release", "sb200_ada_fused_profile", "sb200_ada_set_At_values", "sb200_getada1_dev", "sb200_getada2_dev",
    "sb200_getada3_dev", "sb200_getada1", "sb200_getada2", "sb200_getada3", "sb200_getdatm_dev", "sb200_ada_plan_datq",
    "sb200_ddot_dense_dev", "sb200_qblkmul_dev", "sb200_quadadd_dev", "sb200_ddot_dense", "sb200_ddot_sparse",
    "sb200_qblkmul", "sb200_quadadd", "sb200_adendotd",
    "sb200_comm_unique_id", "sb200_comm_init_rank", "sb200_comm_size", "sb200_comm_rank", "sb200_comm_nccl_version",
    "sb200_comm_stats", "sb200_allreduce_sum_dev", "sb200_allreduce_sum2_dev", "sb200_comm_destroy",
    "sb200_blkchol_sharded_dev", "sb200_ldl_solve_sharded_dev",
    "sb200_wrappcg_dev", "sb200_wrappcg_full_dev", "sb200_wrappcg_full_work", "sb200_ldl_solve2_dev", "sb200_ada_plan_csr", "sb200_psd_plan_blocks",
    "sb200_dpr1_plan_create", "sb200_dpr1_plan_destroy", "sb200_dpr1fact_dev", "sb200_dpr1solve_dev", "sb200_dpr1_plan_download",
    "sb200_gather_dev", "sb200_scale_by_d_dev", "sb200_chol_plan_lb_dev",
]


def comm_init(rank: int, world: int, device: int, bcast) -> None:
    """Join the library's own NCCL communicator (include/sedumi_b200.h "multi-GPU"): rank 0 draws the unique id,
    `bcast(bytearray(128)) -> bytes` moves it to every rank over whatever channel the host has (bench.py: a
    torch.distributed broadcast), then all ranks call sb200_comm_init_rank.  Collective."""
    L = lib()
    check(L.sb200_init(C.c_int(device)), "init")
    buf = (C.c_char * 128)()
    if rank == 0:
        check(L.sb200_comm_unique_id(buf), "comm_unique_id")
    raw = bcast(bytes(buf.raw))
    buf2 = (C.c_char * 128).from_buffer_copy(raw)
    check(L.sb200_comm_init_rank(C.c_int(world), C.c_int(rank), buf2), "comm_init_rank")


def comm_stats():
    calls, nbytes = I64(0), I64(0)
    lib().sb200_comm_stats(C.byref(calls), C.byref(nbytes))
    return int(calls.value), int(nbytes.value)


class _CholPars(C.Structure):
    _fields_ = [("abstol", C.c_double), ("canceltol", C.c_double), ("maxu", C.c_double)]


class CgPars(C.Structure):
    """cgpars of wrapPcg / loopPcg; the defaults are checkpars.m:171-191."""
    _fields_ = [("restol", C.c_double), ("stagtol", C.c_double), ("maxiter", C.c_int), ("refine", C.c_int), ("qprec", C.c_int)]
    DEFAULTS = dict(restol=5e-3, stagtol=5e-14, maxiter=49, refine=1, qprec=1)


class _PcgCones(C.Structure):
    _fields_ = [("nq", I64), ("qdim", I64), ("qbs", VP), ("det", VP), ("q1", VP), ("q2", VP), ("auxdet", VP), ("auxtr", VP),
                ("nden", I64), ("den_cols", VP), ("denA", VP), ("ndenq", I64)]


class _PcgStatus(C.Structure):
    _fields_ = [("k", I64), ("stop", C.c_int), ("trials", C.c_int), ("normr", C.c_double)]


class HotPath:
    """Device-resident state + the per-iteration call sequence for one problem."""

    def __init__(self, S, device: int = 0, chol_pars=None):
        import torch
        self.torch = torch
        L = lib()
        check(L.sb200_init(C.c_int(device)), "init")
        self.dev = torch.device("cuda", device)
        self.S = S
        K = S.K
        m = self.m = S.m
        At = S.At
        self.nq = len(K["q"])
        s = np.asarray(K["s"], dtype=np.int64)
        self.s = s
        self.lenud = int((s ** 2).sum())
        self.lpN = int(K["l"])
        pars = dict(abstol=1e-20, canceltol=1e-12, maxu=5e5)
        pars.update(chol_pars or {})
        self.pars = _CholPars(pars["abstol"], pars["canceltol"], pars["maxu"])
        # ---- plans
        Ajc, Air = _i64(At.indptr), _i64(At.indices)
        Ajc1 = _i64(S.Ablkjc[:, 2])
        qstart = _i64(np.asarray(K["qblkstart"]) - 1)
        bs = _i64(np.asarray(K["sblkstart"])[:len(s)] - 1) if len(s) else _i64([])
        adajc, adair = _i64(S.ADA.indptr), _i64(S.ADA.indices)
        self.ada = VP()
        check(L.sb200_ada_plan_get(C.byref(self.ada), I64(At.shape[0]), I64(m), _p(Ajc), _p(Air), _p(Ajc1),
                                   I64(self.lpN), I64(self.nq), _p(qstart), I64(len(s)), _p(bs), _p(_i64(s)),
                                   _p(adajc), _p(adair)), "ada_plan")
        L.sb200_ada_plan_retain(self.ada)          # the cache may not evict a plan this object (and its graphs) uses
        check(L.sb200_ada_set_At_values(self.ada, _p(np.ascontiguousarray(At.data, dtype=np.float64))), "At values")
        self.psd = VP()
        check(L.sb200_psd_plan_get(C.byref(self.psd), I64(len(s)), _p(_i64(s))), "psd_plan")
        Lst = S.L
        LL = Lst["L"]
        self.chol = VP()
        check(L.sb200_chol_plan_create(C.byref(self.chol), I64(m), I64(len(Lst["xsuper"].ravel()) - 1),
                                       _p(_i64(Lst["xsuper"].ravel() - 1)), _p(_i64(LL.indptr)), _p(_i64(LL.indices)),
                                       _p(_i64(Lst["perm"].ravel() - 1)), _p(adajc), _p(adair)), "chol_plan")
        self.nnzADA = int(S.ADA.nnz)
        self.rect = int(L.sb200_chol_plan_rect_size(self.chol))
        f64 = dict(dtype=torch.float64, device=self.dev)
        z = lambda n: torch.zeros(max(int(n), 1), **f64)
        self.d_l, self.d_det = z(self.lpN), z(self.nq)
        # Lorentz part of the scaling and of the iterate (getDAtm, qblkmul/ddot/quadadd streams)
        q = np.asarray(K["q"], dtype=np.int64)
        self.qdim = int((q - 1).sum()) if self.nq else 0
        self.d_q1, self.d_q2 = z(self.nq), z(self.qdim)
        self.d_auxdet, self.d_auxtr = z(self.nq), z(self.nq)
        if self.nq:
            bsq = np.r_[0, np.cumsum(q - 1)].astype(np.int64)
            self.qbs = torch.from_numpy(bsq).to(self.dev)
            self.q_mu, self.q_x, self.q_y, self.q_dd = z(self.nq), z(self.qdim), z(self.qdim), z(self.nq)
            self.r_hi, self.r_lo, self.r_y = z(m), z(m), z(m)
            jc, ir, pr, nnz = C.c_void_p(), C.c_void_p(), C.c_void_p(), I64(0)
            check(L.sb200_ada_plan_datq(self.ada, C.byref(jc), C.byref(ir), C.byref(pr), C.byref(nnz)), "datq")
            self.datq = (jc, ir, pr, int(nnz.value))
        self.d_u, self.udsqr = z(self.lenud), z(self.lenud)
        self.d_perm = torch.zeros(max(int(s.sum()), 1), dtype=torch.int32, device=self.dev)
        self.has_perm = False
        # ADA values and absd share one allocation: the sharded path reduces both at the Schur-assembly boundary
        self._ada_absd = z(self.nnzADA + m + 8)
        self.ADA, self.absd = self._ada_absd[:max(self.nnzADA, 1)], self._ada_absd[self.nnzADA:self.nnzADA + max(m, 1)]
        self.Lrect, self.dvec, self.sval = z(self.rect), z(m), z(m)
        self.flag = torch.zeros(max(m, 1), dtype=torch.int32, device=self.dev)
        self.psd_x, self.psd_y = z(self.lenud), z(self.lenud)
        self.rhs = self.y = self.w = None
        self.shard = None
        # scaling update (updtransfo.m:99-108): frames of the PSD iterate, re-ordered factor, rotation list
        sumn = int(s.sum())
        self.sumn = sumn
        self.s64 = _i64(s)
        self.frms, self.lab = z(self.lenud), z(sumn)
        self.psd_z, self.psd_f = z(self.lenud), z(self.lenud)
        self.u_new, self.urot_work = z(self.lenud), z(self.lenud + sumn)
        self.g = z(int((s * (s - 1)).sum()))
        self.perm_new = torch.zeros(max(sumn, 1), dtype=torch.int32, device=self.dev)
        self.gjc = torch.zeros(max(sumn, 1), dtype=torch.int32, device=self.dev)
        self.maxu_urot = 1.1                        # updtransfo.m:100
        # ---- dense columns (getdense.m): product-form factor on top of the sparse one (deninfac.m:57-79)
        self.nden = len(S.dense.cols) if getattr(S, "dense", None) is not None else 0
        self.dpr1 = None
        if self.nden:
            from .host import symbolic
            assert len(S.dense.q) == 0, "dense Lorentz blocks are not wired into the device chain"
            self.symLden = symbolic.symbcholden(S.L, S.dense)
            dz = self.symLden["dz"]
            self.dpr1 = VP()
            check(L.sb200_dpr1_plan_create(C.byref(self.dpr1), I64(m), I64(self.nden), _p(_i64(dz.indptr)), _p(_i64(dz.indices)),
                                           _p(_i64(self.symLden["perm"].ravel() - 1)), _p(_i64(self.symLden["first"].ravel() - 1))), "dpr1_plan")
            Ad = np.asfortranarray(np.asarray(S.dense.A.todense(), dtype=np.float64))          # m x nden, deninfac.m:59 (LP columns)
            self.Ad = torch.from_numpy(np.ascontiguousarray(Ad.T)).to(self.dev)                 # rows = columns of Ad (column-major m x nden)
            self.LAD = torch.zeros_like(self.Ad)
            self.den_idx = torch.from_numpy((S.dense.cols[:S.dense.l].astype(np.int64) - 1).astype(np.int32)).to(self.dev)
            self.smult = z(self.nden)
            self.dvec_den = z(m)
            self.maxuden = 5e2                       # checkpars.m:158-166

    def __del__(self):
        try:
            if getattr(self, "ada", None) and _lib is not None:
                _lib.sb200_ada_plan_release(self.ada)
                self.ada = None
        except Exception:
            pass

    # ------------------------------------------------------------------ data movement
    def set_scaling(self, d: dict, non_blocking=False) -> int:
        """Host -> device copy of the NT scaling; returns bytes moved."""
        t = self.torch
        nbytes = 0
        for name, dst in (("l", self.d_l), ("det", self.d_det), ("u", self.d_u), ("q1", self.d_q1), ("q2", self.d_q2),
                          ("auxdet", self.d_auxdet), ("auxtr", self.d_auxtr)):
            if name not in d:
                continue
            a = np.ascontiguousarray(np.asarray(d[name], dtype=np.float64).ravel())
            if a.size:
                dst[:a.size].copy_(t.from_numpy(a), non_blocking=non_blocking)
                nbytes += a.nbytes
        p = np.asarray(d.get("perm", np.zeros(0))).ravel()
        self.has_perm = p.size > 0
        if self.has_perm:
            p0 = (p.astype(np.int64) - 1).astype(np.int32)
            self.d_perm[:p0.size].copy_(t.from_numpy(p0), non_blocking=non_blocking)
            nbytes += p0.nbytes
        return nbytes

    def set_rhs(self, r: np.ndarray) -> int:
        t = self.torch
        r = np.ascontiguousarray(np.asarray(r, dtype=np.float64).reshape(self.m, -1, order="F").T)   # rows = rhs
        self.nrhs = r.shape[0]
        self.rhs = t.from_numpy(r).to(self.dev)
        self.y = t.empty_like(self.rhs)
        self.w = t.empty_like(self.rhs)
        return r.nbytes

    # ------------------------------------------------------------------ kernels
    def invcholfac(self):
        check(lib().sb200_invcholfac_dev(self.psd, _p(self.d_u), _p(self.d_perm) if self.has_perm else None,
                                         _p(self.udsqr)), "invcholfac")

    def getada(self):
        L = lib()
        if self.nq:        # getDAtm.m:40-43 on the device; its pattern lives in the plan
            check(L.sb200_getdatm_dev(self.ada, _p(self.d_q1), _p(self.d_q2)), "getdatm")
        check(L.sb200_getada1_dev(self.ada, _p(self.d_l), _p(self.d_det), None, _p(self.ADA)), "getada1")
        if self.nq:
            jc, ir, pr, _ = self.datq
            check(L.sb200_getada2_dev(self.ada, jc, ir, pr, None, _p(self.ADA), _p(self.ADA)), "getada2")
        check(L.sb200_getada3_dev(self.ada, _p(self.udsqr), None, I64(0), _p(self.ADA), _p(self.absd), C.c_int(1)), "getada3")

    def blkchol(self):
        check(lib().sb200_blkchol_dev(self.chol, _p(self.ADA), _p(self.absd), self.pars, _p(self.Lrect), _p(self.dvec),
                                      _p(self.flag), _p(self.sval)), "blkchol")

    def solve(self):
        """y = L' \\ ((L \\ r(perm)) ./ d), all right-hand sides (wrapPcg.m:56-59); with dense columns the product-form
        factor sits in the middle: fwblkslv -> fwdpr1 -> ./d -> bwdpr1 -> bwblkslv."""
        L = lib()
        if self.dpr1 is None:
            check(L.sb200_ldl_solve_dev(self.chol, _p(self.Lrect), _p(self.dvec), _p(self.flag), _p(self.rhs),
                                        _p(self.w), _p(self.y), I64(self.nrhs)), "ldl_solve")
            return
        check(L.sb200_fwblkslv_dev(self.chol, _p(self.Lrect), _p(self.rhs), _p(self.w), I64(self.nrhs)), "fwblkslv")
        check(L.sb200_dpr1solve_dev(self.dpr1, C.c_int(0), _p(self.w), I64(self.nrhs)), "fwdpr1")
        check(L.sb200_scale_by_d_dev(I64(self.m), I64(self.nrhs), _p(self.dvec_den), _p(self.flag), VP(L.sb200_chol_plan_lb_dev(self.chol)),
                                     _p(self.w)), "./d")
        check(L.sb200_dpr1solve_dev(self.dpr1, C.c_int(1), _p(self.w), I64(self.nrhs)), "bwdpr1")
        check(L.sb200_bwblkslv_dev(self.chol, _p(self.Lrect), _p(self.w), _p(self.y), I64(self.nrhs)), "bwblkslv")

    def deninfac(self):
        """deninfac.m:57-79 on the device: LAD = L \\ Ad(perm,:), smult = d.l(dense.cols), product-form factor, updated d."""
        if self.dpr1 is None:
            return
        L = lib()
        check(L.sb200_fwblkslv_dev(self.chol, _p(self.Lrect), _p(self.Ad), _p(self.LAD), I64(self.nden)), "sparfwslv")
        check(L.sb200_gather_dev(I64(self.nden), _p(self.den_idx), _p(self.d_l), _p(self.smult)), "smult")
        check(L.sb200_dpr1fact_dev(self.dpr1, _p(self.LAD), _p(self.smult), C.c_double(self.maxuden), _p(self.dvec), _p(self.dvec_den)), "dpr1fact")

    # ------------------------------------------------------------------ subtree-sharded factor / solve (SURVEY 8e)
    def shard_factor_setup(self, world: int, rank: int):
        """Deal the elimination-tree subtrees below a replicated top to `world` ranks (this object is rank `rank`)."""
        L = lib()
        check(L.sb200_chol_shard_create(self.chol, I64(world), I64(rank)), "chol_shard_create")
        t0, off, ln, col0, cm = I64(0), I64(0), I64(0), I64(0), C.c_void_p()
        check(L.sb200_chol_shard_info(self.chol, C.byref(t0), C.byref(off), C.byref(ln), C.byref(col0), C.byref(cm)), "chol_shard_info")
        self.shard = dict(world=world, rank=rank, t0=int(t0.value), top_off=int(off.value), top_len=int(ln.value), col0=int(col0.value))
        return self.shard

    def blkchol_shard_local(self):
        check(lib().sb200_blkchol_shard_local_dev(self.chol, _p(self.ADA), _p(self.absd), self.pars, _p(self.Lrect), _p(self.dvec),
                                                  _p(self.flag), _p(self.sval)), "blkchol_shard_local")

    def blkchol_shard_top(self):
        check(lib().sb200_blkchol_shard_top_dev(self.chol, self.pars, _p(self.Lrect), _p(self.dvec), _p(self.flag), _p(self.sval)),
              "blkchol_shard_top")

    def top_panels(self):
        sh = self.shard
        return self.Lrect[sh["top_off"]:sh["top_off"] + sh["top_len"]]

    def blkchol_sharded(self):
        """Own subtrees, ONE all-reduce of the top panels, top (replicated) -- collectives inside the library."""
        check(lib().sb200_blkchol_sharded_dev(self.chol, _p(self.ADA), _p(self.absd), self.pars, _p(self.Lrect), _p(self.dvec),
                                              _p(self.flag), _p(self.sval)), "blkchol_sharded")

    def solve_shard_local(self):
        check(lib().sb200_fw_shard_local_dev(self.chol, _p(self.Lrect), _p(self.rhs), _p(self.w), I64(self.nrhs)), "fw_shard_local")

    def solve_shard_top(self):
        check(lib().sb200_solve_shard_top_dev(self.chol, _p(self.Lrect), _p(self.dvec), _p(self.flag), _p(self.w), I64(self.nrhs)),
              "solve_shard_top")

    def solve_shard_finish(self):
        check(lib().sb200_bw_shard_finish_dev(self.chol, _p(self.w), _p(self.y), I64(self.nrhs)), "bw_shard_finish")

    def solve_sharded(self):
        """Forward over the own subtrees, all-reduce of the top segment, top + backward, all-reduce of the solution."""
        check(lib().sb200_ldl_solve_sharded_dev(self.chol, _p(self.Lrect), _p(self.dvec), _p(self.flag), _p(self.rhs),
                                                _p(self.w), _p(self.y), I64(self.nrhs)), "ldl_solve_sharded")

    def psdscale(self, transp: int):
        check(lib().sb200_psdscale_dev(self.psd, _p(self.d_u), _p(self.d_perm) if self.has_perm else None,
                                       _p(self.psd_x), C.c_int(transp), _p(self.psd_y)), "psdscale")

    def set_frames(self, lab: np.ndarray, frms: np.ndarray) -> int:
        """Spectral factor of the PSD iterate (vfrm.lab PSD part, vfrm.s), host -> device."""
        t = self.torch
        lab = np.ascontiguousarray(np.asarray(lab, dtype=np.float64).ravel()[-self.sumn:]) if self.sumn else np.zeros(0)
        frms = np.ascontiguousarray(np.asarray(frms, dtype=np.float64).ravel())
        if lab.size:
            self.lab[:lab.size].copy_(t.from_numpy(lab))
            self.frms[:frms.size].copy_(t.from_numpy(frms))
        return lab.nbytes + frms.nbytes

    def psdinvjmul(self):
        """z = psdinvjmul(lab, frms, psd_y): solves X Z + Z X = 2 Y per block (psdinvjmul.c:101-157)."""
        check(lib().sb200_psdinvjmul_dev(self.psd, _p(self.lab), _p(self.frms), _p(self.psd_y), _p(self.psd_z)), "psdinvjmul")

    def psdframeit(self):
        check(lib().sb200_psdframeit_dev(self.psd, _p(self.lab), _p(self.frms), _p(self.psd_f)), "psdframeit")

    def urotorder(self):
        check(lib().sb200_urotorder_dev(I64(len(self.s)), _p(self.s64), _p(self.d_u), C.c_double(self.maxu_urot),
                                        _p(self.u_new), _p(self.perm_new), _p(self.gjc), _p(self.g), _p(self.urot_work)),
              "urotorder")

    def givensrot(self):
        check(lib().sb200_givensrot_dev(I64(len(self.s)), _p(self.s64), _p(self.gjc), _p(self.g), _p(self.psd_f),
                                        _p(self.psd_z)), "givensrot")

    def lorentz_streams(self):
        """The Lorentz-cone vector work of one iteration (SURVEY 8d recipe for sum(K.s)==0):
        6 x qblkmul, 3 x ddot (dense), 1 x quadadd on device-resident vectors."""
        if not self.nq:
            return
        L = lib()
        for _ in range(6):
            check(L.sb200_qblkmul_dev(I64(self.nq), _p(self.qbs), I64(self.qdim), _p(self.q_mu), _p(self.q_x), _p(self.q_y)), "qblkmul")
        for _ in range(3):
            check(L.sb200_ddot_dense_dev(I64(self.nq), _p(self.qbs), _p(self.d_q2), _p(self.q_x), I64(self.qdim), I64(1), _p(self.q_dd)), "ddot")
        check(L.sb200_quadadd_dev(I64(self.m), _p(self.r_hi), _p(self.r_lo), _p(self.r_y), _p(self.r_hi), _p(self.r_lo)), "quadadd")

    def update_scaling_tail(self):
        """psdinvjmul -> 2 x psdframeit -> urotorder -> givensrot (SURVEY 8d recipe; updtransfo.m:99-108)."""
        if not self.lenud:
            return
        self.psdinvjmul()
        self.psdframeit()
        self.psdframeit()
        self.urotorder()
        self.givensrot()

    def allreduce_ada(self):
        """The collective at the Schur-assembly boundary (SURVEY 8e): sum the per-rank partial ADA values and absd
        (one contiguous buffer, one NCCL call) on the library stream right behind getada3."""
        check(lib().sb200_allreduce_sum_dev(_p(self._ada_absd), I64(self.nnzADA + self.m)), "allreduce(ADA,absd)")

    def iteration(self, nsolve=4, npsdscale=12, sharded=False):
        self.invcholfac()
        self.getada()
        if sharded:
            self.allreduce_ada()
        if sharded and getattr(self, "shard", None):
            self.blkchol_sharded()
            for _ in range(nsolve):
                self.solve_sharded()
        else:
            self.blkchol()
            self.deninfac()
            for _ in range(nsolve):
                self.solve()
        if self.lenud:
            for i in range(npsdscale):
                self.psdscale(i & 1)
            self.update_scaling_tail()
        else:
            self.lorentz_streams()

    def capture(self, nsolve=4, npsdscale=12, sharded=False):
        """Record one iteration -- kernels AND, when sharded, the library's NCCL collectives -- into a CUDA graph;
        returns a callable that replays it."""
        L = lib()
        self.iteration(nsolve, npsdscale, sharded)          # warm: lazy allocations / attribute changes happen here
        self.sync()
        l0 = L.sb200_kernel_launches()
        check(L.sb200_graph_begin(), "graph_begin")
        try:
            self.iteration(nsolve, npsdscale, sharded)
        finally:
            g = VP()
            rc = L.sb200_graph_end(C.byref(g))
        check(rc, "graph_end")
        self.launches_per_iteration = int(L.sb200_kernel_launches() - l0)
        self._graph = g
        return lambda: check(L.sb200_graph_launch(g), "graph_launch")

    def wrappcg(self, rv: np.ndarray, rb: np.ndarray | None = None):
        """The direct step of wrapPcg.m:42-97 on the device (factor and scaling already resident: call after blkchol).
        rv: N = K.l + sum(K.s.^2) right-hand side in x-space, rb: m or None.  Returns dict(y, dx, r, ssqrNew, ssqrdx,
        alpha, normr) as host arrays / floats (one D2H at the end)."""
        t = self.torch
        N = self.lpN + self.lenud
        rv = np.ascontiguousarray(np.asarray(rv, dtype=np.float64).ravel())
        assert rv.size == N, (rv.size, N)
        with t.cuda.stream(self.stream()):
            if getattr(self, "_pcg", None) is None:
                f64 = dict(dtype=t.float64, device=self.dev)
                self._pcg = dict(work=t.zeros(3 * N + 2 * self.m + 600, **f64), y=t.zeros(self.m, **f64), dx=t.zeros(N, **f64),
                                 r=t.zeros(self.m, **f64), scal=t.zeros(4, **f64), rv=t.zeros(N, **f64), rb=t.zeros(self.m, **f64))
            P = self._pcg
            P["rv"].copy_(t.from_numpy(rv))
            if rb is not None:
                P["rb"].copy_(t.from_numpy(np.ascontiguousarray(np.asarray(rb, dtype=np.float64).ravel())))
            check(lib().sb200_wrappcg_dev(self.ada, self.psd, self.chol, _p(self.d_l), _p(self.d_u),
                                          _p(self.d_perm) if self.has_perm else None, _p(self.Lrect), _p(self.dvec), _p(self.flag),
                                          _p(P["rv"]), _p(P["rb"]) if rb is not None else None, _p(P["y"]), _p(P["dx"]), _p(P["r"]),
                                          _p(P["scal"]), _p(P["work"])), "wrappcg")
            self.sync()
            sc = P["scal"].cpu().numpy()
            return dict(y=P["y"].cpu().numpy(), dx=P["dx"].cpu().numpy(), r=P["r"].cpu().numpy(), ssqrNew=float(sc[0]),
                        ssqrdx=float(sc[1]), alpha=float(sc[2]), normr=float(sc[3]))

    def pcg(self, rv: np.ndarray, rb: np.ndarray | None = None, y0: float = 1.0, cgpars: dict | None = None):
        """The search direction of wrapPcg.m:43-130 on the device: the direct step, then loopPcg refinement while
        |r|_inf >= y0 * cgpars["restol"].  Valid after blkchol (and deninfac with dense columns) for LP, Lorentz and PSD
        cones; the scaling is the one set_scaling uploaded last (with d.auxdet, d.auxtr when there are Lorentz cones).
        rv: N = K.l + sum(K.q) + sum(K.s.^2) in x-space, rb: m or None; cgpars: any of restol, stagtol, maxiter, refine,
        qprec (defaults: checkpars.m).  Returns dict(y, dx, r, k, stop, trials, normr) as host arrays / numbers.
        Raises SB200Error while the library stream is being captured: the loop reads its status back on the host."""
        t = self.torch
        L = lib()
        N = self.lpN + self.nq + self.qdim + self.lenud
        cg = dict(CgPars.DEFAULTS, **(cgpars or {}))
        pars = CgPars(cg["restol"], cg["stagtol"], int(cg["maxiter"]), int(cg["refine"]), int(cg["qprec"]))
        P = getattr(self, "_pcgf", None)
        st = _PcgStatus()
        with t.cuda.stream(self.stream()):
            if t.cuda.is_current_stream_capturing():
                # nothing may be enqueued into the capture: let the entry refuse before any upload
                cones = _PcgCones(self.nq, self.qdim, None, None, None, None, None, None, self.nden, None, None, 0)
                check(L.sb200_wrappcg_full_dev(self.ada, self.psd, self.chol, self.dpr1, C.byref(cones), C.byref(pars),
                                               *([None] * 8), C.c_double(y0), None, None, None, C.byref(st), None), "wrappcg_full")
            rv = np.ascontiguousarray(np.asarray(rv, dtype=np.float64).ravel())
            assert rv.size == N, (rv.size, N)
            if P is None:
                f64 = dict(dtype=t.float64, device=self.dev)
                nw = int(L.sb200_wrappcg_full_work(I64(N), I64(self.m), I64(self.nq), I64(self.qdim)))
                P = self._pcgf = dict(work=t.zeros(nw, **f64), y=t.zeros(self.m, **f64), dx=t.zeros(N, **f64),
                                      r=t.zeros(self.m, **f64), rv=t.zeros(N, **f64), rb=t.zeros(self.m, **f64))
            P["rv"].copy_(t.from_numpy(rv))
            if rb is not None:
                P["rb"].copy_(t.from_numpy(np.ascontiguousarray(np.asarray(rb, dtype=np.float64).ravel())))
            nq = self.nq
            cones = _PcgCones(nq, self.qdim, _p(self.qbs) if nq else None, _p(self.d_det), _p(self.d_q1), _p(self.d_q2),
                              _p(self.d_auxdet), _p(self.d_auxtr), self.nden, _p(self.den_idx) if self.nden else None,
                              _p(self.Ad) if self.nden else None, 0)
            check(L.sb200_wrappcg_full_dev(self.ada, self.psd, self.chol, self.dpr1, C.byref(cones), C.byref(pars), _p(self.d_l),
                                           _p(self.d_u), _p(self.d_perm) if self.has_perm else None, _p(self.Lrect),
                                           _p(self.dvec_den if self.nden else self.dvec), _p(self.flag), _p(P["rv"]),
                                           _p(P["rb"]) if rb is not None else None, C.c_double(y0), _p(P["y"]), _p(P["dx"]),
                                           _p(P["r"]), C.byref(st), _p(P["work"])), "wrappcg_full")
            self.sync()
            return dict(y=P["y"].cpu().numpy(), dx=P["dx"].cpu().numpy(), r=P["r"].cpu().numpy(), k=int(st.k), stop=int(st.stop),
                        trials=int(st.trials), normr=float(st.normr))

    def profile(self, nsolve=4, npsdscale=12, sharded=False, reps=3):
        """Per-kernel device time of one iteration, averaged over `reps`: {kernel name: (launches, ms)}.  An event is
        recorded after every launch; sb200_prof_begin parks a ~3 ms spin kernel on the stream first, so the host has
        enqueued the iteration before the GPU starts on it and the intervals contain no host launch gaps."""
        L = lib()
        self.iteration(nsolve, npsdscale, sharded)
        self.sync()
        out = {}
        for _ in range(reps):
            check(L.sb200_prof_begin(), "prof_begin")
            self.iteration(nsolve, npsdscale, sharded)
            buf = C.create_string_buffer(1 << 16)
            check(L.sb200_prof_end(buf, I64(len(buf))), "prof_end")
            for ln in buf.value.decode().splitlines():
                nm, cnt, tot = ln.split()
                c0, t0 = out.get(nm, (0, 0.0))
                out[nm] = (c0 + int(cnt), t0 + float(tot))
        return {k: (v[0] // reps, v[1] / reps) for k, v in out.items()}

    def sync(self):
        check(lib().sb200_sync(), "sync")

    def stream(self):
        return self.torch.cuda.ExternalStream(lib().sb200_stream(), device=self.dev)
