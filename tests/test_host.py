"""CPU tests of the host-side logic (cone re-layout, setup structures, symbolic factorisation)."""
import numpy as np
import pytest
import scipy.sparse as sp

import golden_io
from sedumi_b200.host import cones, problems, setup, symbolic


def test_pretransfo_layout_control07():
    At, b, c, K = problems.internal_problem("control07")
    assert K["l"] == 1 and list(K["s"]) == [70, 35] and At.shape == (1 + 4900 + 1225, 666)
    assert At.nnz == 107940                                 # folded to the lower triangle (SURVEY 8: 107 940)
    assert list(K["blkstart"]) == [2, 2, 4902, 6127]
    # PSD coefficients live in the lower triangle only (pretransfo.m:434-454)
    rows = At.indices[At.indices >= 1] - 1
    r70 = rows[rows < 4900]
    assert np.all(r70 % 70 >= r70 // 70)


def test_pretransfo_diag_block_to_lp_arch0():
    At, b, c, K = problems.internal_problem("arch0")
    assert K["l"] == 175 and list(K["s"]) == [161]          # 174-block is diagonal -> LP (pretransfo.m:231-241)


def test_pretransfo_preserves_inner_products():
    """<A_i, X> is invariant under the fold: sum over folded lower coefficients against a symmetric X."""
    raw = problems.synth_small_mixed(seed=3, m=10, l=2, q=(3,), s=(4,), density=0.6)
    At0, b0, c0, K0 = raw
    At, b, c, K, QR = cones.pretransfo(*raw)
    rng = np.random.default_rng(0)
    Xs = rng.standard_normal((4, 4)); Xs = Xs + Xs.T
    x0 = np.r_[rng.standard_normal(2 + 3), Xs.ravel(order="F")]
    x = QR @ x0
    # after the fold, the PSD part pairs folded coefficients with the lower triangle of X twice-counted
    xi = x.copy()
    n = 4
    P = xi[-n * n:].reshape(n, n, order="F")
    xi[-n * n:] = ((P + P.T) / 2 * 1.0).ravel(order="F")
    lhs = np.asarray(sp.csc_matrix(At0).T @ x0).ravel()
    Xl = np.tril(Xs).ravel(order="F")
    xx = np.r_[0.0, x[1:-n * n], Xl]                       # x0 slot, LP+Lorentz, lower triangle of X
    assert np.allclose(At.T @ xx, lhs, rtol=1e-12, atol=1e-12)


def test_free_and_rotated_cones_reach_internal_form():
    raw = problems.synth_small_mixed(seed=9, m=12, l=3, q=(3,), s=(5,), f=2, r=(4,))
    At, b, c, K = cones.pretransfo(*raw)[:4]
    assert list(K["q"]) == [3, 3, 4]                        # [free-cone (f+1), K.q, K.r]
    assert K["l"] == 1 + 3 and At.shape[0] == K["N"]


@pytest.mark.parametrize("name", ["arch0", "control07", "nb", "trto3"])
def test_setup_matches_reference_mex(name):
    """Ablkjc, sperm and dz against the reference's partitA and incorder on the same problem (stored outputs)."""
    At, b, c, K = problems.internal_problem(name)
    S = setup.build_setup(At, b, c, K)
    g = golden_io.load(f"host_setup_{name}")
    assert np.array_equal(g["Ablkjc"], S.Ablkjc)
    assert np.array_equal(g["sperm"].ravel(), S.Aord["sperm"].ravel())
    dz = g["dz"]
    assert np.array_equal(dz.indptr, S.Aord["dz"].indptr) and np.array_equal(dz.indices, S.Aord["dz"].indices)
    assert S.ADA.nnz == S.m * S.m and len(S.L["xsuper"]) == 2      # every shipped fixture: dense ADA, 1 supernode


@pytest.mark.parametrize("m,density", [(50, 0.08), (300, 0.01)])
def test_symbolic_factor_is_valid_and_supernodal(m, density):
    from helpers import random_sparse_spd
    X = random_sparse_spd(m, density, 1)
    L = symbolic.symbolic_factor(X)
    p = L["perm"].ravel().astype(int) - 1
    assert sorted(p) == list(range(m))
    pat = L["L"].toarray() != 0
    Xp = X.toarray()[np.ix_(p, p)]
    Lnum = np.linalg.cholesky(Xp)
    assert np.all(pat[np.abs(Lnum) > 1e-14])                # the pattern covers the numeric factor
    xs = L["xsuper"].ravel().astype(int) - 1
    ip, ind = L["L"].indptr, L["L"].indices
    for a, e in zip(xs[:-1], xs[1:]):                       # nested columns inside each supernode
        for j in range(a, e - 1):
            assert np.array_equal(ind[ip[j] + 1:ip[j + 1]], ind[ip[j + 1]:ip[j + 2]])


def test_symbolic_matches_reference_fill():
    """Fill against the reference's ordmmdmex + symfctmex, tmpsiz against its choltmpsiz (stored outputs)."""
    from helpers import random_sparse_spd
    X = random_sparse_spd(300, 0.01, 2)
    L = symbolic.symbolic_factor(X)
    g = golden_io.load("host_symbolic_fill300")
    assert abs(L["L"].nnz - int(g["nnzL"])) <= 0.15 * int(g["nnzL"])      # both minimum-degree orderings
    assert L["tmpsiz"] == float(g["tmpsiz"])


def test_scaling_generators_are_interior():
    At, b, c, K = cones.pretransfo(*problems.synth_small_mixed())[:4]
    d = problems.scaling(K, "S1", seed=1)
    assert np.all(d["l"] > 0) and np.all(d["det"] > 0)
    off = 0
    for n in K["s"].astype(int):
        U = np.triu(d["u"][off:off + n * n].reshape(n, n, order="F"))
        assert np.all(np.diag(U) > 0)
        off += n * n


def test_symbcholden_restatement_matches_reference_symbolic_chain():
    """host.symbolic.symbcholden (symbfwblk + incorder + finsymbden restated for LP dense columns) against the reference's
    own symbolic MEX files (symbcholden.m:45-62; stored outputs of oracle/refpath.py's DenseColumnRef)."""
    for seed, nd in ((4, 3), (8, 4)):
        raw = problems.synth_blockdiag_sdp(nblk=4, n=10, m=48, nlink=6, density=0.08, dense_lp=nd, seed=seed)
        At, b, c, K = cones.pretransfo(*raw)[:4]
        S = setup.build_setup(At, b, c, K, denf=0.3, perm=np.arange(At.shape[1]))
        assert len(S.dense.cols) == nd
        ref_sym = golden_io.load(f"host_symbcholden_seed{seed}")
        mine = symbolic.symbcholden(S.L, S.dense)
        for k in ("LAD", "dz"):
            a, r = sp.csc_matrix(mine[k]), ref_sym[k]
            a.sort_indices()
            assert np.array_equal(a.indptr, r.indptr) and np.array_equal(a.indices, r.indices), k
        assert np.array_equal(mine["perm"].ravel(), np.asarray(ref_sym["perm"]).ravel())
        assert np.array_equal(mine["first"].ravel(), np.asarray(ref_sym["first"]).ravel())
