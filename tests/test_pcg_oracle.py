"""The restated wrapPcg / loopPcg / PopK / asmDxq / Amul (tests/pcg_ref.py) against
independent dense linear algebra: asmDxq is P(d)^{1/2}, PopK is P(d), and the search direction solves
A P(d) A' y = A P(d)^{1/2} rv + rb to the residual tolerance.  Needs the compiled reference (oracle/_ref)."""
import os

import numpy as np
import pytest
import scipy.linalg as sla

import pcg_cases as pc
from helpers import ROOT

pytestmark = pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "qblkmul.so")),
                                reason="oracle/_ref not built")


def _explicit(S, d):
    """Dense D (= [sqrt(d.l); P_k(d)^{1/2} per Lorentz cone; psdscale(d, ., K)]), the PSD vecsym projector and A'
    with the dense columns put back, all as N x N / N x m arrays."""
    import restate
    K = S.K
    N = S.At.shape[0]
    l, q, s = int(K["l"]), np.asarray(K["q"], dtype=np.int64), np.asarray(K["s"], dtype=np.int64)
    D = np.zeros((N, N))
    D[:l, :l] = np.diag(np.sqrt(d["l"]))
    nq, o2 = q.size, l + q.size
    for k in range(nq):
        rows = [l + k] + list(range(o2, o2 + q[k] - 1))
        dk = np.r_[d["q1"][k], d["q2"][o2 - l - nq:o2 - l - nq + q[k] - 1]]
        P = np.outer(dk, dk) + d["det"][k] * np.diag(np.r_[-1.0, np.ones(q[k] - 1)])     # PopK.m:45 + DAt.q'DAt.q
        w, V = np.linalg.eigh(P)
        assert w.min() > 0
        D[np.ix_(rows, rows)] = (V * np.sqrt(w)) @ V.T
        o2 += q[k] - 1
    o = o2
    ud = {"u": d["u"], "perm": d["perm"]}
    nps = int((s ** 2).sum())
    for i in range(nps):
        e = np.zeros(nps); e[i] = 1.0
        D[o:, o + i] = restate.psdscale(ud, e, K)
    V = np.eye(N)
    for n in s:
        n = int(n)
        for i in range(n):
            for j in range(n):
                a, b = o + i + j * n, o + j + i * n
                V[a, a] = V[a, b] = 0.5 if a != b else 1.0
        o += n * n
    At = S.At.toarray()
    if len(S.dense.cols):
        At[S.dense.cols.astype(int) - 1, :] = S.dense.A.T.toarray()
    return D, V, At


@pytest.mark.parametrize("given", [False, True])
def test_asmdxq_is_square_root_of_P(given):
    import pcg_ref
    import refpath
    S = pc.mixed()
    d = pc.scaling(S.K, 3)
    mex = refpath.ref_dir()
    D, _, _ = _explicit(S, d)
    x = np.random.default_rng(5).standard_normal(S.At.shape[0])
    l, nq = int(S.K["l"]), len(S.K["q"])
    lq = int(S.K["lq"])
    ddotx = None
    if given:
        _, ddotx, _, _ = pcg_ref.PopK(mex, d, x, S.K)
    y = pcg_ref.asmDxq(mex, d, x, S.K, ddotx)
    assert np.linalg.norm(y - D[l:lq, l:lq] @ x[l:lq]) <= 1e-13 * np.linalg.norm(y)
    assert nq == 3


def test_popk_is_P():
    import pcg_ref
    import refpath
    S = pc.mixed()
    d = pc.scaling(S.K, 3)
    mex = refpath.ref_dir()
    D, _, _ = _explicit(S, d)
    x = np.random.default_rng(6).standard_normal(S.At.shape[0])
    y, ddotx, Dx, xTy = pcg_ref.PopK(mex, d, x, S.K)
    l, nq, lq = int(S.K["l"]), len(S.K["q"]), int(S.K["lq"])
    # the Lorentz rank-one part d d'x travels separately (ddotx, through DAt.q in loopPcg.m:113)
    ddfull = y.copy()
    q = np.asarray(S.K["q"], dtype=np.int64); o2 = l + nq
    for k in range(nq):
        ddfull[l + k] += ddotx[k] * d["q1"][k]
        ddfull[o2:o2 + q[k] - 1] += ddotx[k] * d["q2"][o2 - l - nq:o2 - l - nq + q[k] - 1]
        o2 += q[k] - 1
    P = D.T @ D
    assert np.linalg.norm(ddfull - P @ x) <= 1e-12 * np.linalg.norm(P @ x)
    assert abs(xTy - np.linalg.norm(D @ x) ** 2) <= 1e-12 * xTy


CASES = {"mixed": pc.mixed, "dense_lp": pc.dense_lp}


@pytest.mark.parametrize("case", sorted(CASES))
def test_exact_factor_takes_one_step(case):
    S = CASES[case]()
    d = pc.scaling(S.K, 3)
    rv, rb = pc.rhs(S, 1)
    ref = pc.reference(S, d, d, rv, rb)
    assert ref["k"] == 1 and ref["stop"] == 0 and ref["trials"] == 0
    assert ref["normr"] < ref["restol"]


@pytest.mark.parametrize("qprec", [0, 1])
@pytest.mark.parametrize("case", sorted(CASES))
def test_other_factor_refines_to_dense_solution(case, qprec):
    S = CASES[case]()
    d0 = pc.scaling(S.K, 3)
    d1 = pc.perturb(d0, S.K, 0.3, 9)
    rv, rb = pc.rhs(S, 1)
    ref = pc.reference(S, d0, d1, rv, rb, cgpars={"qprec": qprec})
    assert ref["k"] > 1 and ref["stop"] == 1
    D, V, At = _explicit(S, d1)
    M = At.T @ D.T @ D @ V @ At
    f = At.T @ D.T @ rv + rb
    res = f - M @ ref["y"]
    assert np.abs(res).max() < ref["restol"]
    assert np.linalg.norm(res - ref["r"]) <= 1e-8 * np.linalg.norm(f)
    ysol = sla.solve(M, f, assume_a="sym")
    assert np.linalg.norm(ref["y"] - ysol) <= 1e-2 * np.linalg.norm(ysol)
    assert np.linalg.norm(ref["dx"] - (rv - D @ V @ At @ ref["y"])) <= 1e-8 * np.linalg.norm(rv)
