"""Problems, scalings and right-hand sides shared by the wrapPcg / loopPcg tests (CPU oracle and device)."""
import os
import sys

import numpy as np

from helpers import ROOT
from sedumi_b200.host import cones, problems, setup

sys.path.insert(0, os.path.join(ROOT, "oracle"))


def lorentz_consistent(d, K):
    """problems.scaling with d.q1 set so that det(d) = (q1^2 - |q2|^2)/2 = d.det, SeDuMi's convention (sdinit.m:75-76,
    updtransfo.m:82-83) under which asmDxq is the square root of PopK's P(d)."""
    e = dict(d)
    q = np.asarray(K["q"], dtype=np.int64)
    if q.size:
        bs = np.r_[0, np.cumsum(q - 1)]
        e["q1"] = np.array([np.sqrt(2 * d["det"][k] + d["q2"][bs[k]:bs[k + 1]] @ d["q2"][bs[k]:bs[k + 1]]) for k in range(q.size)])
        e["auxdet"] = np.sqrt(2 * e["det"])
        e["auxtr"] = np.sqrt(2) * (e["q1"] + e["auxdet"])
    return e


def scaling(K, seed):
    return lorentz_consistent(problems.scaling(K, "S1", seed=seed), K)


def perturb(d, K, eps, seed):
    """A scaling near d: every part multiplied / shifted by O(eps), kept in the interior of the cone
    (Lorentz: q1 = sqrt(det + |q2|^2); PSD: upper factor with positive diagonal, mirrored as urotorder stores it)."""
    rng = np.random.default_rng(seed)
    e = dict(d)
    e["l"] = d["l"] * np.exp(eps * rng.standard_normal(d["l"].size))
    q = np.asarray(K["q"], dtype=np.int64)
    if q.size:
        e["det"] = d["det"] * np.exp(eps * rng.standard_normal(q.size))
        e["q2"] = d["q2"] + eps * rng.standard_normal(d["q2"].size)
        bs = np.r_[0, np.cumsum(q - 1)]
        e["q1"] = np.array([np.sqrt(2 * e["det"][k] + e["q2"][bs[k]:bs[k + 1]] @ e["q2"][bs[k]:bs[k + 1]]) for k in range(q.size)])
        e["auxdet"] = np.sqrt(2 * e["det"])
        e["auxtr"] = np.sqrt(2) * (e["q1"] + e["auxdet"])
    us, off = [], 0
    for n in np.asarray(K["s"], dtype=np.int64):
        n = int(n)
        U = np.triu(d["u"][off:off + n * n].reshape(n, n, order="F"))
        U = U * (1 + eps * rng.standard_normal((n, n)))
        U = np.triu(U)
        us.append((U + np.triu(U, 1).T).ravel(order="F"))
        off += n * n
    e["u"] = np.concatenate(us) if us else np.zeros(0)
    return e


def build(raw, perm=None, denf=10.0):
    At, b, c, K = cones.pretransfo(*raw)[:4]
    return setup.build_setup(At, b, c, K, denf=denf, perm=perm)


def mixed(seed=7):
    """LP + Lorentz (q = 4, 3, 5) + PSD."""
    return build(problems.synth_small_mixed(seed=seed, m=30, l=6, q=(4, 3, 5), s=(7, 5), density=0.3))


def dense_lp(seed=4, ndense=3):
    """LP block with dense columns, PSD blocks (the dpr1 tests' problem)."""
    raw = problems.synth_blockdiag_sdp(nblk=4, n=10, m=48, nlink=6, density=0.08, dense_lp=ndense, seed=seed)
    S = build(raw, perm=np.arange(raw[0].shape[1]), denf=0.3)
    assert len(S.dense.cols) == ndense and S.dense.l == ndense and len(S.dense.q) == 0
    return S


def reference(S, d_fact, d, rv, rb=None, **kw):
    """The restated wrapPcg with the factor of scaling d_fact and the products of scaling d."""
    import pcg_ref
    import refpath
    R = refpath.RefHotPath(S)
    udsqr, ADA, absd = R.assemble(d_fact)
    L, Lden = pcg_ref.factor_with_dense(R, ADA, absd, d_fact)
    return pcg_ref.wrappcg(R, L, d, rv, rb, Lden=Lden, **kw)


def rhs(S, seed, use_rb=True):
    rng = np.random.default_rng(seed)
    return rng.standard_normal(S.At.shape[0]), (rng.standard_normal(S.m) if use_rb else None)
