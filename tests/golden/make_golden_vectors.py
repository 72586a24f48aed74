"""Generate golden input/output vectors for the hot path from the reference itself.

Runs the UNMODIFIED reference MEX targets (oracle/_ref, built from /root/reference by
oracle/Makefile) on small seeded inputs and stores inputs + outputs as .npz.  The reference holds
no per-kernel vectors of its own (SURVEY.md section 8c), so these files -- produced by the
reference's code on this container -- are the known-answer tests that travel to the GPU box.

    python tests/golden/make_golden_vectors.py
"""
import os
import sys

import numpy as np
import scipy.sparse as sp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import refpath  # noqa: E402
from helpers import CHOL_PARS, dense_L, full_pattern, random_sparse_spd, random_spd  # noqa: E402
from sedumi_b200.host import cones, problems, setup, symbolic  # noqa: E402

OUT = os.path.join(HERE, "vectors")
ref = refpath.ref_dir()


def csc(a):
    a = sp.csc_matrix(a)
    return dict(data=a.data, indices=a.indices.astype(np.int64), indptr=a.indptr.astype(np.int64), shape=np.array(a.shape))


def save(name, **kw):
    flat = {}
    for k, v in kw.items():
        if isinstance(v, dict):
            for kk, vv in v.items():
                flat[f"{k}__{kk}"] = vv
        else:
            flat[k] = np.asarray(v)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **flat)


# ---- blkchol / solves: dense with skips and adds, and a sparse multi-supernode case
def chol_case(name, L, X, pars, absd, nrhs=2, seed=0):
    LL, d, skip, add = ref.blkchol(L, X, pars, absd, nlhs=4)
    Lf = dict(L, L=LL)
    b = np.random.default_rng(seed).standard_normal((X.shape[0], nrhs))
    save(name, X=csc(X), Lpat=csc(L["L"]), perm=L["perm"], xsuper=L["xsuper"], tmpsiz=L["tmpsiz"],
         pars=np.array([pars["abstol"], pars["canceltol"], pars["maxu"]]), absd=absd,
         LL=LL.data, d=d, skip_idx=skip.indices, skip_val=skip.data, add_idx=add.indices, add_val=add.data,
         b=b, fw=ref.fwblkslv(Lf, b), bw=ref.bwblkslv(Lf, b))


m = 48
X = random_spd(m, seed=1, cond=1e4)
chol_case("chol_dense48", dense_L(m), full_pattern(X), CHOL_PARS, np.diag(X).copy())
rng = np.random.default_rng(2)
B = rng.standard_normal((40, 30))
chol_case("chol_rankdef40", dense_L(40), full_pattern(B @ B.T), dict(CHOL_PARS, canceltol=1e-9),
          np.einsum("ij,ij->i", np.abs(B), np.abs(B)))
s = 10.0 ** rng.uniform(-5, 5, 60)
Xs = random_spd(60, seed=63, cond=1e2) * np.outer(s, s)
chol_case("chol_diagadd60", dense_L(60), full_pattern(Xs), dict(CHOL_PARS, maxu=5e2), np.diag(Xs).copy())
Xsp = random_sparse_spd(120, 0.03, 5)
chol_case("chol_sparse120", symbolic.symbolic_factor(Xsp), Xsp, CHOL_PARS, np.asarray(Xsp.diagonal()).copy())

# ---- the ADA chain + psd ops on a small mixed-cone problem
At, b, c, K = cones.pretransfo(*problems.synth_small_mixed())[:4]
S = setup.build_setup(At, b, c, K)
d = problems.scaling(K, "S1", seed=3)
R = refpath.RefHotPath(S)
udsqr, ADA, absd = R.assemble(d)
save("ada_small_mixed", At=csc(S.At), Ablkjc=S.Ablkjc, lqperm=S.Aord["lqperm"], qperm=S.Aord["qperm"], sperm=S.Aord["sperm"],
     dz=csc(S.Aord["dz"]), ADApat=csc(S.ADA), K_l=K["l"], K_q=K["q"], K_s=K["s"],
     d_l=d["l"], d_det=d["det"], d_q1=d["q1"], d_q2=d["q2"], d_u=d["u"], d_perm=d["perm"],
     udsqr=udsqr, ADA=ADA.data, absd=absd)

# ---- host-side structures: what the reference's own MEX files make of the same inputs (tests/test_host.py)
dbg = refpath.ref_dir(debug=True)
for name in ("arch0", "control07", "nb", "trto3"):
    At, b, c, K = problems.internal_problem(name)
    S = setup.build_setup(At, b, c, K)
    sperm, dz = dbg.incorder(S.At, S.Ablkjc[:, 2], K["mainblks"][2], nlhs=2)
    save(f"host_setup_{name}", Ablkjc=dbg.partitA(S.At, K["mainblks"].reshape(1, -1)), sperm=sperm, dz=csc(dz))
Xf = random_sparse_spd(300, 0.01, 2)
Lf = symbolic.symbolic_factor(Xf)
save("host_symbolic_fill300", nnzL=ref.symfctmex(Xf, ref.ordmmdmex(Xf))["L"].nnz, tmpsiz=dbg.choltmpsiz(Lf).ravel()[0])
for seed, nd in ((4, 3), (8, 4)):
    raw = problems.synth_blockdiag_sdp(nblk=4, n=10, m=48, nlink=6, density=0.08, dense_lp=nd, seed=seed)
    At, b, c, K = cones.pretransfo(*raw)[:4]
    S = setup.build_setup(At, b, c, K, denf=0.3, perm=np.arange(At.shape[1]))
    sym = refpath.DenseColumnRef(S, dict(S.L)).sym
    save(f"host_symbcholden_seed{seed}", LAD=csc(sym["LAD"]), dz=csc(sym["dz"]), perm=sym["perm"], first=sym["first"])
print("golden vectors written to", OUT, sorted(os.listdir(OUT)))
