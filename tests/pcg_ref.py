"""Restatement of the search direction of the reference -- TEST INFRASTRUCTURE for the wrapPcg / loopPcg tests.

wrapPcg.m:43-130, loopPcg.m:53-170, PopK.m:39-55, asmDxq.m:41-69 and Amul.m:40-56 (with LP dense columns) follow the
M source statement by statement in numpy.  They have no C source; the C pieces they call are the reference's own MEX
targets compiled into oracle/_ref (fwblkslv, bwblkslv, fwdpr1, bwdpr1, vecsym, ddot, qblkmul, quadadd, blkchol,
dpr1fact), driven through oracle/refpath.py, and psdscale.m comes from oracle/restate.py.
"""
import os
import sys

import numpy as np

from helpers import ROOT

sys.path.insert(0, os.path.join(ROOT, "oracle"))

import refpath  # noqa: E402
import restate  # noqa: E402
from sedumi_b200.host import setup as hsetup  # noqa: E402


# --------------------------------------------------------------------------- search direction (wrapPcg / loopPcg helpers)
# These drive the reference's compiled ddot / qblkmul (a MexDir passed as `mex`) for the Lorentz arithmetic; x is a
# full-length vector in the internal layout [K.l | Lorentz trace entries | norm-bound parts | PSD].
def asmDxq(mex, d, x, K, ddotx=None, want_t=False):
    """asmDxq.m:41-69: y = P(d)^{1/2} x on the Lorentz part (trace rows, then norm-bound rows).  With want_t the
    two-output form: (y without the t d terms, t)."""
    q = np.asarray(K["q"]).ravel()
    if q.size == 0:
        return (np.zeros(0), np.zeros(0)) if want_t else np.zeros(0)
    x = np.asarray(x, dtype=float).ravel()
    if x.size >= int(K["lq"]):
        i1, i2 = int(K["mainblks"][0]), int(K["mainblks"][1])
    else:
        i1, i2 = 1, q.size + 1
    bs = np.asarray(K["qblkstart"], dtype=float).reshape(1, -1)
    x1 = x[i1 - 1:i2 - 1]
    if ddotx is None:
        ddotx = d["q1"] * x1 + np.asarray(mex.ddot(d["q2"], x.reshape(-1, 1), bs)).ravel()
    t = (np.asarray(ddotx, dtype=float).ravel() + x1 * d["auxdet"]) / d["auxtr"]
    sdet = np.sqrt(d["det"])
    y = np.r_[t * d["auxdet"] - sdet * x1, np.asarray(mex.qblkmul(sdet, x.reshape(-1, 1), bs)).ravel()]
    if want_t:
        return y, t
    return y + np.r_[t * d["q1"], np.asarray(mex.qblkmul(t, np.asarray(d["q2"], dtype=float).reshape(-1, 1), bs)).ravel()]


def PopK(mex, d, x, K):
    """PopK.m:39-55 (lpq = 0): (y, ddotx, Dx, xTy) with y = P(d) x, ddotx = d[k]' x[k] per Lorentz cone,
    Dx = psdscale(d, x, K) and xTy = x' P(d) x."""
    x = np.asarray(x, dtype=float).ravel()
    i1, i2 = int(K["mainblks"][0]), int(K["mainblks"][1])
    nq = len(np.asarray(K["q"]).ravel())
    y = np.asarray(d["l"], dtype=float).ravel() * x[:i1 - 1]
    ddotx = np.zeros(0)
    if nq:
        bs = np.asarray(K["qblkstart"], dtype=float).reshape(1, -1)
        x1 = x[i1 - 1:i2 - 1]
        y = np.r_[y, -d["det"] * x1, np.asarray(mex.qblkmul(d["det"], x.reshape(-1, 1), bs)).ravel()]
        ddotx = d["q1"] * x1 + np.asarray(mex.ddot(d["q2"], x.reshape(-1, 1), bs)).ravel()
    ud = {"u": d.get("u", np.zeros(0)), "perm": d.get("perm", np.zeros(0))}
    Dx = restate.psdscale(ud, x, K)
    y = np.r_[y, restate.psdscale(ud, Dx, K, 1)]
    lq = int(K["lq"])
    xTy = float(x[:lq] @ y[:lq] + np.sum(ddotx ** 2) + np.sum(Dx ** 2))
    return y, ddotx, Dx, xTy


def Amul(At, dense, x, transp=0):
    """Amul.m:40-56: y = (x' At)' (+ dense.A x(dense.cols)) resp. y = At x with y(dense.cols) = dense.A' x."""
    x = np.asarray(x, dtype=float).ravel()
    cols = np.asarray(dense.cols if dense is not None else np.zeros(0)).ravel().astype(np.int64) - 1
    if transp == 0:
        y = np.asarray(x @ At).ravel()
        if cols.size:
            y = y + np.asarray(dense.A @ x[cols]).ravel()
    else:
        y = np.asarray(At @ x).ravel()
        if cols.size:
            y[cols] = np.asarray(dense.A.T @ x).ravel()
    return y


CG_PARS = {"qprec": 1, "restol": 5e-3, "stagtol": 5e-14, "maxiter": 49, "refine": 1}    # checkpars.m:171-191


def factor_with_dense(R: "refpath.RefHotPath", ADA, absd, d, maxuden=5e2):
    """blkchol, then deninfac.m:57-93: with LP dense columns the product-form factor Lden from the reference's
    dpr1fact (through DenseColumnRef) and its updated d; the skipped pivots repaired last.  Returns (L, Lden) with
    L["d"] the d wrapPcg divides by; Lden is None without dense columns."""
    S = R.S
    L = dict(S.L)
    LL, Ld, skip, add = R.mex.blkchol(hsetup.L_for_mex(L), ADA, R.pars, absd, nlhs=4)
    L.update(L=LL, d=Ld.ravel().copy(), skip=skip, add=add)
    Lden = None
    if len(S.dense.cols):
        DC = refpath.DenseColumnRef(S, L)
        LAD, Ld0, sym, smult = DC.inputs(d, L["d"].copy())
        Lden, Ld = R.mex.dpr1fact(LAD, Ld0, sym, smult, maxuden, nlhs=2)
        Lden.update(dz=sym["dz"], first=sym["first"], perm=sym["perm"])        # deninfac.m:73-75
        L["d"] = np.asarray(Ld, dtype=float).ravel().copy()
    sk = skip.indices
    if sk.size:
        dtol = np.maximum(R.pars["canceltol"] * np.asarray(absd).ravel()[L["perm"].ravel().astype(int)[sk] - 1], R.pars["abstol"])
        fix = L["d"][sk] <= dtol
        L["d"][sk[fix]] = 1.0
    return L, Lden


def wrappcg(R: "refpath.RefHotPath", L: dict, d: dict, rv, rb=None, y0=1.0, cgpars=None, Lden=None):
    """wrapPcg.m:43-130 with loopPcg.m:53-170 (PopK.m, asmDxq.m, Amul.m restated above) on the
    reference's own fwblkslv / bwblkslv / fwdpr1 / bwdpr1 / vecsym / ddot / qblkmul / quadadd.  LP, Lorentz and real PSD
    cones, LP dense columns (Lden from factor_with_dense).  Returns dict(y, dx, r, k, stop, trials, normr, hist,
    restol): stop is the STOP of the last loopPcg call (0: none ran), trials the refinement trials, hist the normr
    after the direct step, after every CG step and after every loopPcg call, in that order."""
    S, mex = R.S, R.mex
    K = S.K
    At = S.At
    dense = S.dense if len(S.dense.cols) else None
    cg = dict(CG_PARS, **(cgpars or {}))
    l = int(K["l"])
    m = S.m
    rv = np.asarray(rv, dtype=float).ravel()
    rb = None if rb is None else np.asarray(rb, dtype=float).ravel()
    sl = np.sqrt(np.asarray(d["l"], dtype=float).ravel())
    ud = {"u": d.get("u", np.zeros(0)), "perm": d.get("perm", np.zeros(0))}
    Lm = hsetup.L_for_mex({k: L[k] for k in ("perm", "L", "xsuper", "tmpsiz")})
    Ld = np.asarray(L["d"], dtype=float).ravel()
    DAtq = R.DAtq(d) if len(K["q"]) else None

    def D(x, transp, ddotx=None):                # [sqrt(d.l).*x(1:K.l); asmDxq(d,x,K[,ddotx]); psdscale(d,x,K[,1])]
        return np.r_[sl * x[:l], asmDxq(mex, d, x, K, ddotx), restate.psdscale(ud, x, K, transp)]

    def fw(r):                                   # fwdpr1(Lden, sparfwslv(L, r))
        z = np.asarray(mex.fwblkslv(Lm, r.reshape(-1, 1)))
        return np.asarray(mex.fwdpr1(Lden, z) if Lden is not None else z).ravel()

    def bw(z):                                   # sparbwslv(L, bwdpr1(Lden, z))
        z = z.reshape(-1, 1)
        if Lden is not None:
            z = np.asarray(mex.bwdpr1(Lden, z))
        return np.asarray(mex.bwblkslv(Lm, z)).ravel()

    def vecsym_At(p):                            # vecsym(Amul(At, dense, p, 1), K)
        return np.asarray(mex.vecsym(Amul(At, dense, p, 1).reshape(-1, 1), R.Km)).ravel()

    def resid(x):
        r = Amul(At, dense, x)
        return r + rb if rb is not None else r

    hist = []
    restol = y0 * cg["restol"]                                           # wrapPcg.m:46
    dx = D(rv, 1)
    r = resid(dx)
    p = fw(r)                                                            # wrapPcg.m:56-59
    y = p / Ld
    ssqrNew = float(p @ y)
    p = bw(y)
    x = vecsym_At(p)                                                     # wrapPcg.m:65-67
    dx = D(x, 0)
    ssqrdx = float(dx @ dx)
    out = lambda **kw: dict(dict(stop=0, trials=0, hist=hist, restol=restol), **kw)
    if ssqrdx <= 0.0:                                                    # wrapPcg.m:68-73
        return out(y=np.zeros(m), k=0, dx=rv.copy(), r=r, normr=float(np.abs(r).max()))
    k = 1
    alpha = ssqrNew / ssqrdx
    y = alpha * p
    dx = rv - alpha * dx
    r = resid(D(dx, 1))                                                  # wrapPcg.m:85-90
    normr = float(np.abs(r).max())
    hist.append(normr)
    if normr < restol:
        return out(y=y, k=k, dx=dx, r=r, normr=normr)
    trial, stop = 0, 0

    def loop_pcg(b, p, ssqrNew):                                         # loopPcg.m:56-170
        k, STOP, r, finew = 0, 0, b.copy(), 0.0
        yv = None                                                        # [] (all-0); a tuple (hi, lo) when qprec
        normrmin = float(np.abs(r).max())
        ymin = None
        alpha = Ap = DApq = DAps = None
        while STOP == 0:
            Lr = fw(r)
            tmp = Lr / Ld
            if p is None:
                ssqrNew = float(Lr @ tmp)
                p = bw(tmp)
            else:
                ssqrOld = ssqrNew
                ssqrNew = float(Lr @ tmp)
                p = (ssqrNew / ssqrOld) * p
                p = p + bw(tmp)
            Ap = vecsym_At(p)
            DDAp, DApq, DAps, ssqrDAp = PopK(mex, d, Ap, K)
            if ssqrDAp > 0.0:
                k += 1
                alpha = ssqrNew / ssqrDAp
                if yv is not None:
                    if isinstance(yv, tuple):
                        hi, lo = mex.quadadd(yv[0].reshape(-1, 1), yv[1].reshape(-1, 1), (alpha * p).reshape(-1, 1), nlhs=2)
                        yv = (np.asarray(hi).ravel(), np.asarray(lo).ravel())
                    else:
                        yv = yv + alpha * p
                elif cg["qprec"] > 0:
                    yv = (alpha * p, np.zeros(p.size))
                else:
                    yv = alpha * p
                tmp = Amul(At, dense, DDAp)                      # loopPcg.m:113-115
                if DAtq is not None:
                    tmp = tmp + np.asarray(DAtq.T @ DApq).ravel()
                r = r - alpha * tmp
                fiprev = finew
                finew = float((b + r) @ yv[0] + (b + r) @ yv[1]) if isinstance(yv, tuple) else float((b + r) @ yv)
                nr = float(np.abs(r).max())
                hist.append(nr)
                if nr < normrmin:
                    ymin, normrmin = yv, nr
                if nr < restol:
                    STOP = 1
                elif finew - fiprev < cg["stagtol"] * fiprev:
                    STOP = 2
                elif k >= cg["maxiter"]:
                    STOP = 2
            else:
                STOP = 1
        if STOP == 2:
            yv = ymin
        if yv is None:
            return None, k, None, STOP
        if k == 1:                                                       # loopPcg.m:153-154
            DAy = alpha * np.r_[sl * Ap[:l], asmDxq(mex, d, Ap, K, DApq), DAps]
        else:
            yh = yv[0] if isinstance(yv, tuple) else yv
            DAy = D(vecsym_At(yh), 0)
            if isinstance(yv, tuple):
                DAy = DAy + D(vecsym_At(yv[1]), 0)
        return (yv[0] if isinstance(yv, tuple) else yv), k, DAy, STOP

    while True:                                                          # wrapPcg.m:100-130
        dy, dk, x, stop = loop_pcg(r, p, ssqrNew)
        if dy is None:
            return out(y=y, k=k, dx=dx, r=r, normr=normr, stop=stop, trials=trial)
        k += dk
        y = y + dy
        dx = dx - x
        r = resid(D(dx, 1))
        normr = float(np.abs(r).max())
        hist.append(normr)
        if normr < restol or trial >= cg["refine"]:
            return out(y=y, k=k, dx=dx, r=r, normr=normr, stop=stop, trials=trial)
        p = None
        trial += 1
