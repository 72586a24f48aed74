"""wrapPcg with loopPcg refinement on the device (HotPath.pcg -> sb200_wrappcg_full_dev) against the restated
wrapPcg.m / loopPcg.m driving the reference's own MEX files (tests/pcg_ref.py::wrappcg).  Gates: y, dx 1e-8 relative,
r on the scale of the data, and the CG step count, STOP code and refinement trials equal."""
import numpy as np
import pytest

import pcg_cases as pc
from sedumi_b200.host import cones, problems, setup

pytestmark = pytest.mark.gpu


def _device(S, d_fact, d, rv, rb, **kw):
    import torch
    from sedumi_b200 import device
    hp = device.HotPath(S)
    with torch.cuda.stream(hp.stream()):
        hp.set_scaling(d_fact)
        hp.invcholfac(); hp.getada(); hp.blkchol(); hp.deninfac()
        hp.set_scaling(d)
        hp.sync()
    return hp, hp.pcg(rv, rb, **kw)


def _check(S, d_fact, d, rv, rb=None, margin=True, **kw):
    ref = pc.reference(S, d_fact, d, rv, rb, y0=kw.get("y0", 1.0), cgpars=kw.get("cgpars"))
    if margin:      # equal step counts are only well posed when no normr sits on the tolerance
        h = np.asarray(ref["hist"])
        assert np.all(np.abs(h / ref["restol"] - 1.0) >= 0.01), (h, ref["restol"])
    hp, got = _device(S, d_fact, d, rv, rb, **kw)
    for k in ("y", "dx"):
        assert np.linalg.norm(got[k] - ref[k]) <= 1e-8 * np.linalg.norm(ref[k]), (k, np.linalg.norm(got[k] - ref[k]), np.linalg.norm(ref[k]))
    scale = np.linalg.norm(rv) + (np.linalg.norm(rb) if rb is not None else 0.0)
    assert np.linalg.norm(got["r"] - ref["r"]) <= 1e-8 * scale
    assert abs(got["normr"] - ref["normr"]) <= 1e-8 * scale
    assert (got["k"], got["stop"], got["trials"]) == (ref["k"], ref["stop"], ref["trials"])
    return got, ref


def test_direct_step_with_lorentz_terms():
    S = pc.mixed()
    d = pc.scaling(S.K, 3)
    rv, rb = pc.rhs(S, 1)
    got, ref = _check(S, d, d, rv, rb, margin=False)
    assert got["k"] == 1 and got["normr"] < 1e-8 * np.linalg.norm(rv)


@pytest.mark.parametrize("qprec", [0, 1])
def test_forced_refinement(qprec):
    S = pc.mixed()
    d0 = pc.scaling(S.K, 3)
    d1 = pc.perturb(d0, S.K, 0.3, 9)
    rv, rb = pc.rhs(S, 1)
    got, ref = _check(S, d0, d1, rv, rb, cgpars={"qprec": qprec})
    assert got["k"] > 3 and got["stop"] == 1


def test_maxiter_stop2_ymin_and_no_refinement():
    S = pc.mixed()
    d0 = pc.scaling(S.K, 3)
    d1 = pc.perturb(d0, S.K, 0.3, 9)
    rv, rb = pc.rhs(S, 1)
    got, ref = _check(S, d0, d1, rv, rb, cgpars={"maxiter": 2, "refine": 0})
    assert got["stop"] == 2 and got["trials"] == 0


def test_skipped_pivots_need_refinement():
    """A duplicated constraint: blkchol skips a pivot and deninfac.m:88-93 repairs it; the result, step count and
    STOP code follow the reference (rb keeps the duplicated rows consistent)."""
    At, b, c, K = cones.pretransfo(*problems.synth_small_mixed(seed=7, m=30, l=6, q=(4, 3, 5), s=(7, 5), density=0.3))[:4]
    import scipy.sparse as sp
    At = sp.csc_matrix(sp.hstack([At, At[:, [3]]]))
    b = np.r_[np.asarray(b).ravel(), np.asarray(b).ravel()[3]]
    S = setup.build_setup(At, b, c, K)
    d = pc.scaling(K, 3)
    rv = np.random.default_rng(1).standard_normal(S.At.shape[0])
    rb = np.random.default_rng(2).standard_normal(S.m)
    rb[-1] = rb[3]
    import pcg_ref
    import refpath
    R = refpath.RefHotPath(S)
    _, ADA, absd = R.assemble(d)
    L, _ = pcg_ref.factor_with_dense(R, ADA, absd, d)
    assert L["skip"].nnz > 0
    _check(S, d, d, rv, rb)


def test_dense_lp_columns():
    S = pc.dense_lp()
    d0 = pc.scaling(S.K, 3)
    rv, rb = pc.rhs(S, 1)
    _check(S, d0, d0, rv, rb, margin=False)
    d1 = pc.perturb(d0, S.K, 0.3, 9)
    got, _ = _check(S, d0, d1, rv, rb)
    assert got["k"] > 3


def test_nb_fixture_forced_refinement():
    S = pc.build(problems.load_fixture("nb"))
    assert int(np.asarray(S.K["s"]).sum()) == 0 and len(S.K["q"]) == 793
    d0 = pc.scaling(S.K, 3)
    d1 = pc.perturb(d0, S.K, 0.3, 9)
    rv, rb = pc.rhs(S, 2)
    got, _ = _check(S, d0, d1, rv, rb)
    assert got["k"] > 1


def test_blockdiag64_forced_refinement():
    raw = problems.synth_blockdiag_sdp()
    S = pc.build(raw, perm=np.arange(raw[0].shape[1]))
    d0 = pc.scaling(S.K, problems.SEED0 + 2)
    d1 = pc.perturb(d0, S.K, 0.1, 9)
    rv, rb = pc.rhs(S, 2)
    got, _ = _check(S, d0, d1, rv, rb)
    assert got["k"] > 1


def test_refuses_dense_lorentz_blocks():
    from sedumi_b200 import device
    raw = problems.synth_small_mixed(seed=3, m=30, l=2, q=(6, 5), s=(), density=0.9)
    S = pc.build(raw, denf=0.2)
    assert len(S.dense.q) > 0
    with pytest.raises(AssertionError, match="dense Lorentz"):
        device.HotPath(S)


def test_refuses_while_capturing():
    import ctypes as C
    import torch
    from sedumi_b200 import device
    S = pc.mixed()
    d = pc.scaling(S.K, 3)
    rv, rb = pc.rhs(S, 1)
    hp, _ = _device(S, d, d, rv, rb)
    L = device.lib()
    device.check(L.sb200_graph_begin(), "graph_begin")
    try:
        with pytest.raises(device.SB200Error, match="being captured"):
            hp.pcg(rv, rb)
    finally:
        g = C.c_void_p()
        device.check(L.sb200_graph_end(C.byref(g)), "graph_end")
        L.sb200_graph_destroy(g)
    with torch.cuda.stream(hp.stream()):
        assert not torch.cuda.is_current_stream_capturing()
    assert hp.pcg(rv, rb)["k"] == 1           # the library stream works normally afterwards
