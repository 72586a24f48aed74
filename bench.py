#!/usr/bin/env python
"""bench.py -- IPM iterations/s over SeDuMi's normal-equations hot path on B200.

Contract: `python bench.py --gpus N --steps K --warmup W [--impl reference]` prints ONE JSON line.
A "step" is one pass of the per-iteration recipe (SURVEY 8d; sedumi.m:442-466, wrapPcg.m:56-59,
updtransfo.m:99-108) over the frozen state of the workload:

    invcholfac -> getada1 -> getada2 -> getada3 -> blkchol -> 4 x (fwblkslv, ./d, bwblkslv) -> 12 x psdscale
    -> psdinvjmul -> 2 x psdframeit -> urotorder -> givensrot

Headline workload at every N: BASELINE.json configs[3], the synthetic block-diagonal SDP with 64 PSD blocks of
order 200 and m=5000 constraints (arrow-shaped ADA: 64 elimination-tree subtrees + a 72-column border).
  N = 1  : the whole problem on one GPU.
  N > 1  : STRONG scaling of the same problem -- PSD blocks and elimination-tree subtrees sharded over the ranks
           (owner computes), collectives issued by libsedumi_b200 itself over NCCL on the library stream and
           captured into the iteration's CUDA graph: all-reduce(ADA,absd), all-reduce(top fronts), two small
           all-reduces per solve.
`value` = device-resident iterations/s (inputs in HBM, CUDA events on the library stream, max over ranks);
`e2e`   = the same recipe with HOST buffers: at N=1 through the reference-facing MEX plugins (every call copies
          in and out), at N>1 through the device API with pinned host buffers copied in/out every step;
`parity` = the SURVEY 8d gates evaluated in this run, before the timed region, against one reference iteration on
          the same inputs (oracle/gates.py); that reference iteration is also the `cpu_baseline` sample;
`secondary` = control07 / nb / arch0 / maxcut4000 (the other BASELINE configs) on one GPU, each with its own gates.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NSOLVE, NPSD = 4, 12
METRIC = "IPM iterations/sec (ADA'+Cholesky+solve) over the hot-path recipe"
HEADLINE = "blockdiag64"
DESCR = {
    "blockdiag64": ("synthetic block-diagonal SDP (BASELINE.json configs[3]): 64 PSD blocks of order 200, m=5000, 4928 local "
                    "constraints (sprandsym density 0.02) + 72 linking constraints (diagonal on every block); arrow ADA, 65 supernodes",
                    "synthetic problem (seeded generator, SURVEY 8d config 4), synthetic S1 scaling / rhs / frames"),
    "control07": ("control07 (BASELINE.json configs[1]): K.s=[70,35], m=666, dense ADA, 1 supernode",
                  "reference example control07.mat (converted fixture), synthetic S1 scaling / rhs / frames"),
    "arch0": ("arch0 (BASELINE.json configs[0]): K.l=175, K.s=[161], m=174", "reference example arch0.mat (converted fixture), synthetic S1 scaling / rhs / frames"),
    "nb": ("nb (BASELINE.json configs[2]): 793 Lorentz cones, m=123, no PSD block",
           "reference example nb.mat (converted fixture), synthetic S1 scaling / rhs / Lorentz vectors"),
    "maxcut4000": ("synthetic MaxCut SDP (BASELINE.json configs[4]): one PSD block n=4000, m=4000, A_j = e_j e_j'",
                   "synthetic problem (seeded generator, SURVEY 8d config 5), synthetic S1 scaling / rhs / frames"),
    "maxcut1000": ("synthetic MaxCut SDP n=1000, m=1000", "synthetic"),
    "blockdiag_small": ("synthetic block-diagonal SDP 8 x 60, m=400", "synthetic"),
    "dense1000": ("synthetic dense-coefficient SDP (SURVEY 8d config 5'): one PSD block n=1000, m=4000, A_j rank 8 dense",
                  "synthetic problem (seeded generator), synthetic S1 scaling / rhs / frames"),
    "densecol": ("block-diagonal SDP 64x200 with 8 dense LP columns (SURVEY 8d config 4'')", "synthetic"),
}


def load_workload(name):
    """-> namespace(S, d, rhs, psd_x, frames=(lab, frms), lor=(mu, x, rhi, rlo, ry), name)."""
    from sedumi_b200.host import cones, problems, setup
    if name in ("control07", "arch0", "nb"):
        raw = problems.load_fixture(name)
    elif name == "blockdiag64":
        raw = problems.synth_blockdiag_sdp()
    elif name == "maxcut4000":
        raw = problems.synth_maxcut()
    elif name == "maxcut1000":
        raw = problems.synth_maxcut(n=1000, p=0.02)
    elif name == "blockdiag_small":
        raw = problems.synth_blockdiag_sdp(nblk=8, n=60, m=400, nlink=16, density=0.03)
    elif name == "dense1000":
        raw = problems.synth_dense_sdp()
    elif name == "densecol":
        raw = problems.synth_blockdiag_sdp(dense_lp=8)
    else:
        raise SystemExit(f"unknown workload {name}")
    At, b, c, K = cones.pretransfo(*raw)[:4]
    perm = np.arange(At.shape[1]) if name.startswith("blockdiag") or name == "densecol" else None
    S = setup.build_setup(At, b, c, K, perm=perm)
    d = problems.scaling(K, "S1", seed=problems.SEED0 + 2)
    rng = np.random.default_rng(problems.SEED0)
    rhs = rng.standard_normal((S.m, 1))
    psd_x = rng.standard_normal(int((np.asarray(K["s"]) ** 2).sum()))
    frames = problems.synth_frames(K["s"])         # (lab, frms): product-form spectral factor of the PSD iterate
    nq, qd = len(K["q"]), int((np.asarray(K["q"]) - 1).sum()) if len(K["q"]) else 0
    lor = (rng.standard_normal(nq), rng.standard_normal(qd), rng.standard_normal(S.m), 1e-17 * rng.standard_normal(S.m),
           rng.standard_normal(S.m))                # mu, x(norm-bound part), residual hi/lo/increment for the Lorentz streams
    return types.SimpleNamespace(S=S, d=d, rhs=rhs, psd_x=psd_x, frames=frames, lor=lor, name=name)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            t = [x.strip() for x in line.split(",")]
            if len(t) < 9:
                continue
            try:
                sm.append(float(t[1])); mx.append(float(t[2]))
            except ValueError:
                continue
            for nm, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), t[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        return {}


# ----------------------------------------------------------------------------- algorithmic work (SURVEY 8d)
def getada3_work(S):
    """SURVEY 8d: F = sum_k sum_{j in J_k} [2 n_k nnz_full(A_jk) + n_k^2 c_jk] + sum_k nnz_fold(V_k) (m_k + 1);
    B = 8 lenud + 12 nnz(At_psd) + 8 nnz(ADA) + 8 m."""
    K = S.K
    s = np.asarray(K["s"], dtype=np.int64)
    if not s.size:
        return 0.0, 0.0
    m, At = S.m, S.At
    start = int(K["mainblks"][2]) - 1
    bs = start + np.r_[0, np.cumsum(s ** 2)]
    F = 0.0
    nnz_fold = np.zeros(s.size)
    mk = np.zeros(s.size)
    for j in range(m):
        rows = At.indices[int(S.Ablkjc[j, 2]):At.indptr[j + 1]]
        if not rows.size:
            continue
        kk = np.searchsorted(bs, rows, side="right") - 1
        for k in np.unique(kk):
            sel = rows[kk == k] - bs[k]
            n = int(s[k])
            p, q = sel % n, sel // n
            nfull = 2 * sel.size - int((p == q).sum())
            c = np.unique(np.r_[p, q]).size
            F += 2.0 * n * nfull + float(n) * n * c
            nnz_fold[k] += sel.size
            mk[k] += 1
    F += float((nnz_fold * (mk + 1)).sum())
    nnz_psd = int((At.indptr[1:] - S.Ablkjc[:, 2]).sum())
    B = 8.0 * float((s ** 2).sum()) + 12.0 * nnz_psd + 8.0 * S.ADA.nnz + 8.0 * m
    return F, B


_WORK_CACHE = {}


def kernel_work(S, name, key):
    """Algorithmic flops / bytes of the named kernel over ONE iteration (SURVEY 8d figures, DESIGN.md section 4)."""
    K = S.K
    s = np.asarray(K["s"], dtype=np.int64)
    m = S.m
    nnzL = S.L["L"].nnz
    n3 = float((s ** 3).sum())
    if key not in _WORK_CACHE:
        _WORK_CACHE[key] = getada3_work(S)
    F3, B3 = _WORK_CACHE[key]
    if name in ("ada3_fused_kernel", "ada3_fused_small_kernel", "ada3_strip_kernel"):
        return dict(bound="tensor", work=F3, unit="TFLOP/s", bytes=B3, what="getada3 (SURVEY 8d F and B)")
    if name == "gemm_nt_kernel":
        # invcholfac (n^3/3 MACs), psdscale (two triangular products, n^3 flops each), psdinvjmul (two full 2n^3
        # + two lower n^3 products), 2 x psdframeit (lower, n^3), compact-WY accumulation of Q for very large blocks;
        # plus getada3's W products when they run on this engine (unfused path)
        fl = n3 / 3 * 2 + NPSD * 2 * n3 + 6 * n3 + 2 * n3
        if s.size and s.max() > 2300:
            fl += 3 * 4.0 / 3.0 * n3
        return dict(bound="tensor", work=fl, unit="TFLOP/s", what="PSD block products (invcholfac, psdscale, frames)")
    if name in ("trail_kernel", "diag_kernel", "trsm_kernel", "factor_small_kernel", "dense_ldl_kernel", "update_kernel",
                "dense_ldl_cluster_kernel", "dense_trail_dmma_kernel"):
        cj = np.diff(S.L["L"].indptr) - 1
        return dict(bound="tensor", work=float((cj * (cj + 1)).sum()), unit="TFLOP/s", what="blkchol F = sum c_j (c_j + 1)")
    if name in ("psdscale_small_kernel", "psdscale_small_dmma_kernel"):
        return dict(bound="tensor", work=NPSD * 4.0 * n3, unit="TFLOP/s", what="psdscale congruences")
    if name == "ada3_dots_kernel":
        return dict(bound="hbm", work=B3, unit="GB/s", what="getada3 B (SURVEY 8d)")
    if name in ("fwsolve_kernel", "bwsolve_kernel", "dense_solve_kernel<fw>", "dense_solve_kernel<bw>", "snode_solve_kernel"):
        return dict(bound="hbm", work=NSOLVE * (8.0 * nnzL + 24.0 * m), unit="GB/s", what="solves B = 8 nnz(L) + 24 m per rhs")
    return dict(bound="hbm", work=8.0 * (S.ADA.nnz + nnzL), unit="GB/s", what="8 (nnz(ADA) + nnz(L))")


def f64_gemm_peak(torch, dev):
    """Measured FP64 GEMM rate (TFLOP/s) on this GPU: torch.matmul f64 4096^3, best of 5."""
    n = 4096
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record(); e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


# ----------------------------------------------------------------------------- reference arm / cpu baseline
def _ref_iteration(R, W, d, S):
    """One pass of the recipe through the reference; returns (seconds inside mexFunctions + numpy pieces, split)."""
    m0 = R.mex.mex_seconds()
    t_np = 0.0
    t1 = time.perf_counter()
    mm = R.mex.mex_seconds()
    udsqr, ADA, absd = R.assemble(d)
    if not len(S.K["s"]):                        # getada.m restated in numpy: count it (minus the MEX time inside it)
        t_np += (time.perf_counter() - t1) - (R.mex.mex_seconds() - mm)
    t_asm = R.mex.mex_seconds() - m0 + t_np
    L = R.factor(ADA, absd)
    for _ in range(NSOLVE):
        R.solve(L, W.rhs)
    t_fs = R.mex.mex_seconds() - m0 + t_np - t_asm
    if len(S.K["s"]):
        t1 = time.perf_counter()
        ps = None
        for i in range(NPSD):
            ps = R.psdscale(d, W.psd_x_local, i & 1)
        t_np += time.perf_counter() - t1
        R.scaling_tail(d, W.frames_local[0], W.frames_local[1], np.asarray(ps).ravel())
    else:
        R.lorentz_streams(d, *W.lor)
    tot = R.mex.mex_seconds() - m0 + t_np
    return tot, dict(assemble=t_asm, factor_solve=t_fs, psd_tail=tot - t_asm - t_fs)


def run_reference(W, steps, warmup, sample_blocks=0):
    """The reference's own CPU implementation of the recipe (oracle/_ref: unmodified reference C, gcc -O2, one thread
    like the reference) + numpy for the M-only psdscale.  sample_blocks > 0: a step runs the recipe on a shard holding
    that many of the PSD blocks (all constraints, the full factor and solves); the per-block part of the time
    (getada3, invcholfac, psdscale, frames, rotations -- all plain sums over blocks, SURVEY 8e) is scaled by
    nblk / sample_blocks, the rest (getada1/2, blkchol, solves) is taken as measured."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import refpath
    S, d = W.S, W.d
    nblk = len(S.K["s"])
    scale = 1.0
    W.psd_x_local, W.frames_local = W.psd_x, W.frames
    if sample_blocks and nblk > sample_blocks:
        from sedumi_b200.host import problems, shard as hshard
        owned = list(range(0, nblk, nblk // sample_blocks))[:sample_blocks]
        s_all = np.asarray(S.K["s"], dtype=np.int64)
        xo = np.r_[0, np.cumsum(s_all ** 2)]
        S, d = hshard.shard_compact(W.S, W.d, owned, 0)
        W.psd_x_local = np.concatenate([W.psd_x[xo[k]:xo[k + 1]] for k in owned])
        W.frames_local = problems.synth_frames(S.K["s"])
        scale = nblk / float(len(owned))
    R = refpath.RefHotPath(S)
    for _ in range(warmup):
        _ref_iteration(R, W, d, S)
    w0 = time.perf_counter()
    tot = 0.0
    for _ in range(steps):
        t, sp = _ref_iteration(R, W, d, S)
        # block-additive part scaled to the whole cone: getada3 dominates `assemble`; getada1/2 are a negligible,
        # unscaled part of it for PSD problems, so scaling all of `assemble` would overstate the reference's time --
        # only the measured getada3 + invcholfac + psd tail share is scaled
        tot += (sp["assemble"] + sp["psd_tail"]) * scale + sp["factor_solve"]
    return dict(seconds=tot, wall=time.perf_counter() - w0, steps=steps, scale=scale,
                sample=(f"recipe on {int(round(nblk / scale))} of {nblk} PSD blocks per step, per-block time scaled x{scale:g}"
                        if scale != 1.0 else "full iterations of the recipe on the same inputs"))


# ----------------------------------------------------------------------------- device-resident run
DUMP_CAP = 1 << 19          # entries per dumped array (4 MiB in float64): a dump stays well below 64 MiB


def dump_outputs(hp, S, dump_dir):
    """Write what a caller of the iteration receives (oracle/gates.py device_outputs, plus the Lorentz vectors) as
    dump_dir/<name>.npy in float64.  An array longer than DUMP_CAP is written as the entries at a fixed, seeded,
    sorted sample of its indices, so two builds given the same arguments can be compared file by file."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gates
    outs = gates.device_outputs(hp, S, int(S.L["L"].nnz))
    if hp.nq:
        outs.update(qblkmul=hp.q_y.cpu().numpy()[:hp.qdim], ddot=hp.q_dd.cpu().numpy()[:hp.nq],
                    quadadd_hi=hp.r_hi.cpu().numpy()[:hp.m], quadadd_lo=hp.r_lo.cpu().numpy()[:hp.m])
    os.makedirs(dump_dir, exist_ok=True)
    for name, a in outs.items():
        a = np.asarray(a, dtype=np.float64).ravel()
        if a.size > DUMP_CAP:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_CAP, replace=False))]
        np.save(os.path.join(dump_dir, name + ".npy"), a)


def device_run(W, args, rank, world, local_rank, sharded, dist, steps, warmup, want_parity=True, flush_mb=256, dump_dir=None):
    import torch
    from sedumi_b200 import device as sbdev
    S, d = W.S, W.d
    S_local = d_local = None
    psd_x, frames = W.psd_x, W.frames
    colmask = None
    par = "1 GPU"
    if sharded:
        from sedumi_b200.host import problems as _pb, shard as hshard
        owned = hshard.partition_blocks(S.K["s"], world)[rank]
        s_all = np.asarray(S.K["s"], dtype=np.int64)
        xo = np.r_[0, np.cumsum(s_all ** 2)]
        S_local, d_local = hshard.shard_compact(S, d, owned, rank)      # owner computes: this rank's PSD blocks only
        psd_x = np.concatenate([psd_x[xo[k]:xo[k + 1]] for k in owned]) if owned else np.zeros(0)
        frames = _pb.synth_frames(S_local.K["s"], seed=_pb.SEED0 + 7 + rank)
    Sl = S_local if sharded else S
    dl = d_local if sharded else d
    hp = sbdev.HotPath(Sl, device=local_rank)
    info = None
    if sharded:
        if len(np.asarray(Sl.L["xsuper"]).ravel()) - 1 > 2:
            info = hp.shard_factor_setup(world, rank)           # elimination-tree subtrees per rank, replicated top
            par = (f"strong scaling: PSD blocks and etree subtrees sharded over {world} ranks (owner computes); collectives per iteration, "
                   f"issued by libsedumi_b200 over NCCL inside the CUDA graph: all-reduce(ADA+absd, {hp.nnzADA + hp.m} doubles), "
                   f"all-reduce(top fronts, {info['top_len']} doubles), 2 per solve (top segment {hp.m - info['col0']}, solution {hp.m} doubles)")
        else:
            par = (f"strong scaling: PSD blocks sharded over {world} ranks (owner computes), 1 all-reduce(ADA+absd)/iteration, "
                   "factor+solves replicated")
    lib = sbdev.lib()
    stream = hp.stream()
    dev = hp.dev
    out = types.SimpleNamespace(hp=hp, parallelism=par)
    with torch.cuda.stream(stream):
        hp.set_scaling(dl)
        hp.set_rhs(W.rhs)
        hp.psd_x[:psd_x.size].copy_(torch.from_numpy(psd_x))
        hp.set_frames(*frames)
        if hp.nq:
            for dst, src in zip((hp.q_mu, hp.q_x, hp.r_hi, hp.r_lo, hp.r_y), W.lor):
                dst[:src.size].copy_(torch.from_numpy(src))
        flush = torch.empty(flush_mb << 20, dtype=torch.uint8, device=dev)
        stream.synchronize()

        def barrier():
            stream.synchronize()
            if world > 1 and dist is not None:
                dist.barrier()
            stream.synchronize()

        for _ in range(warmup):
            hp.iteration(NSOLVE, NPSD, sharded)
        # ---- parity gates (untimed): the state the device holds after one iteration vs one reference iteration
        out.parity = None
        if want_parity and rank == 0:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import gates
            if sharded and info is not None:
                import ctypes as C
                t0, off, ln, col0, cm = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_void_p()
                sbdev.check(lib.sb200_chol_shard_info(hp.chol, C.byref(t0), C.byref(off), C.byref(ln), C.byref(col0), C.byref(cm)), "shard_info")
                colmask = np.zeros(hp.m, dtype=np.int32)
                sbdev.check(lib.sb200_d2h(colmask.ctypes.data_as(C.c_void_p), cm, C.c_int64(4 * hp.m)), "d2h colmask")
                colmask[int(col0.value):] = 1
            out.parity = gates.run_gates(hp, S, d, W.rhs, psd_x, frames, NSOLVE, NPSD, S_local=S_local, d_local=d_local, colmask=colmask)
        # the iteration is latency-bound at small sizes: replay it as one CUDA graph (collectives included when sharded)
        run_iter = hp.capture(NSOLVE, NPSD, sharded) if not args.no_graph else (lambda: hp.iteration(NSOLVE, NPSD, sharded))
        for _ in range(2):
            run_iter()
        barrier()
        sampler = ClockSampler(local_rank) if rank == 0 else None
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        l0 = lib.sb200_kernel_launches()
        c0 = sbdev.comm_stats()
        barrier()
        t_wall0 = time.perf_counter()
        for k in range(steps):
            flush.fill_(k & 255)                      # evict L2 between timed iterations (untimed)
            ev[k][0].record(stream)
            run_iter()
            ev[k][1].record(stream)
        barrier()
        out.wall = time.perf_counter() - t_wall0
        if dump_dir and rank == 0:
            dump_outputs(hp, S, dump_dir)
        launches = lib.sb200_kernel_launches() - l0
        if not args.no_graph:
            launches = hp.launches_per_iteration * steps      # kernels inside the replayed graphs
        out.launches = int(launches)
        ms = sum(a.elapsed_time(b) for a, b in ev)
        # also a back-to-back (no flush) figure for context
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            run_iter()
        e1.record(stream)
        stream.synchronize()
        out.ms_warm = e0.elapsed_time(e1) / steps
        out.clocks = sampler.stop() if sampler else None
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1 and dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out.ms_max = float(t.item())
        c1 = sbdev.comm_stats()
        per = max(steps * (1 if args.no_graph else 0), 1)
        out.comm = {"nccl_version": int(lib.sb200_comm_nccl_version()), "world": int(lib.sb200_comm_size()),
                    "collectives_per_iteration": ((c1[0] - c0[0]) / per if args.no_graph else None)}

        # ---- per-kernel timing pass (CUDA events after every launch on the library stream); every rank takes part
        # because the sharded iteration contains collectives
        nprof = 1
        cs0 = sbdev.comm_stats()
        hp.iteration(NSOLVE, NPSD, sharded)
        cs1 = sbdev.comm_stats()
        out.comm["collectives_per_iteration"] = cs1[0] - cs0[0]
        out.comm["allreduce_bytes_per_iteration"] = cs1[1] - cs0[1]
        barrier()
        prof = hp.profile(NSOLVE, NPSD, sharded)
        barrier()
        out.roof = None
        if rank == 0 and prof:
            tot_ms = sum(v[1] for v in prof.values())
            kern = {k: v for k, v in prof.items() if k != "nccl_allreduce"}
            nm, (cnt, tms) = max(kern.items(), key=lambda kv: kv[1][1])
            w = kernel_work(Sl, nm, (W.name, world if sharded else 1))
            per_iter_ms = tms / nprof
            peaks = measured_peaks()
            if w["bound"] == "hbm":
                achieved = w["work"] / (per_iter_ms * 1e-3) / 1e9
                peak = peaks.get("hbm_gbs", 6650.0)
                src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
            else:
                achieved = w["work"] / (per_iter_ms * 1e-3) / 1e12
                with torch.cuda.stream(torch.cuda.default_stream()):
                    peak = f64_gemm_peak(torch, dev)
                src = ("FP64 (bound=tensor means the FP64 DMMA/FMA pipes): measured in-run, torch.matmul f64 4096^3 best of 5 "
                       "-- MEASURED_PEAKS.json has no FP64 entry")
            traffic = None
            try:        # DRAM bytes per iteration of that kernel from the committed ncu --set full capture
                traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic_r02.json"))).get(W.name, {}).get(nm)
            except (OSError, ValueError):
                pass
            out.roof = {"kernel": nm, "bound": w["bound"], "achieved": achieved, "peak": peak, "unit": w["unit"],
                        "frac": achieved / peak, "traffic": traffic, "peak_source": src, "work_model": w["what"],
                        "algorithmic_bytes": w.get("bytes"),
                        "launches_per_step": cnt / nprof, "ms_per_step_in_kernel": per_iter_ms,
                        "share_of_step": tms / tot_ms,
                        "kernel_ms_per_step": {k: round(v[1] / nprof, 5) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])}}
    return out


def e2e_device_api(W, hp, sharded, steps, world, dist, local_psd_x):
    """The recipe through the device API with HOST buffers: every step copies this rank's scaling (d.u, d.l, d.perm),
    the right-hand side and the PSD iterate from pinned host memory, replays the iteration graph and reads the search
    direction and the scaled PSD iterate back to pinned host memory.  Inputs are perturbed every step."""
    import torch
    stream = hp.stream()
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).pin_memory()
    hu = pin(hp.d_u.cpu().numpy()[:max(hp.lenud, 1)])
    hl = pin(hp.d_l.cpu().numpy())
    hr = pin(hp.rhs.cpu().numpy())
    hx = pin(local_psd_x if local_psd_x.size else np.zeros(1))
    hy = torch.empty_like(hp.y, device="cpu").pin_memory()
    hpsd = torch.empty(max(hp.lenud, 1), dtype=torch.float64).pin_memory()
    run = hp.capture(NSOLVE, NPSD, sharded)
    h2d = hu.numel() * 8 + hl.numel() * 8 + hr.numel() * 8 + hx.numel() * 8
    d2h = hy.numel() * 8 + hpsd.numel() * 8
    with torch.cuda.stream(stream):
        def step(k):
            hr[0, k % hr.shape[1]] += 1e-3            # the inputs change every step, as in a real run
            hu[0] *= 1.0 + 1e-12
            hp.d_u[:hu.numel()].copy_(hu, non_blocking=True)
            hp.d_l[:hl.numel()].copy_(hl, non_blocking=True)
            hp.rhs.copy_(hr, non_blocking=True)
            hp.psd_x[:hx.numel()].copy_(hx, non_blocking=True)
            run()
            hy.copy_(hp.y, non_blocking=True)
            hpsd.copy_(hp.psd_y[:hpsd.numel()], non_blocking=True)
            stream.synchronize()
        step(0)
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        for k in range(steps):
            step(k + 1)
        e1.record(stream)
        stream.synchronize()
        wall = time.perf_counter() - t0
    sec = max(e0.elapsed_time(e1) * 1e-3, 0.0)
    if world > 1:
        tt = torch.tensor([sec], dtype=torch.float64, device=hp.dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        sec = float(tt.item())
    return {"value": steps / sec, "unit": "iterations/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "steps": steps, "seconds": sec,
            "timed": "device API (sedumi_b200.device.HotPath) with pinned HOST buffers: per step H2D of this rank's d.u, d.l, rhs, PSD iterate; "
                     "the iteration graph; D2H of y and of the scaled PSD iterate; CUDA events, max over ranks; bytes are per rank "
                     f"(wall {wall / steps * 1e3:.2f} ms/step)"}


def run_e2e_mex(W, steps):
    """The recipe through the reference-facing MEX plugins: host numpy in, host numpy out; d.l, d.u, rhs and the PSD
    iterate change every step (so the content-addressed device mirrors only hit where a real run would: ADA and L
    travelling between consecutive plugin calls, At and the structure arrays)."""
    import ctypes as C
    import scipy.sparse as sp
    from sedumi_b200 import device as sbdev
    from sedumi_b200.host import setup as hsetup
    from sedumi_b200.mx import MexDir
    S, d = W.S, {k: (np.array(v, copy=True) if isinstance(v, np.ndarray) else v) for k, v in W.d.items()}
    gpu = MexDir(os.path.join(ROOT, "sedumi_b200", "mex"))
    Km = S.Kmex()
    ADA0 = sp.csc_matrix((np.zeros(S.ADA.nnz), S.ADA.indices, S.ADA.indptr), shape=S.ADA.shape)
    Lm = hsetup.L_for_mex(S.L)
    pars = {"canceltol": 1e-12, "maxu": 5e5, "abstol": 1e-20}
    nq = len(S.K["q"])
    DAt = {"q": sp.csc_matrix((nq, S.m))}
    lenud = int((np.asarray(S.K["s"]) ** 2).sum())
    qbs = S.K["qblkstart"].reshape(1, -1)
    rhs = W.rhs.copy()
    xfull = np.r_[np.zeros(1), W.psd_x]
    lab, frms = W.frames
    LOR = W.lor

    def step(k):
        # a new iterate every step
        rhs[k % S.m, 0] += 1e-3
        if d["l"].size:
            d["l"][k % d["l"].size] *= 1.0 + 1e-9
        if lenud:
            d["u"][0] *= 1.0 + 1e-12
            xfull[1 + k % lenud] += 1e-6
        dstruct = {"l": d["l"], "det": d["det"]}
        if nq:                                       # getDAtm.m:40-43 through the ddot plugin
            d["q2"][k % d["q2"].size] *= 1.0 + 1e-9
            tr = hsetup.extractA(S.At, S.Ablkjc, 1, 2, int(S.K["mainblks"][0]), int(S.K["mainblks"][1]))
            DAt["q"] = sp.csc_matrix(sp.diags(d["q1"]) @ tr + gpu.ddot(d["q2"], S.At, qbs, S.Ablkjc))
        ud = gpu.invcholfac(d["u"], Km, d["perm"])
        A1 = gpu.getada1(ADA0, S.At, S.Ablkjc[:, 2], S.Aord["lqperm"], dstruct, qbs)
        A2 = gpu.getada2(A1, DAt, S.Aord, Km)
        A3, absd = gpu.getada3(A2, S.At, S.Ablkjc[:, 2], S.Aord, ud, Km, nlhs=2)
        LL, Ld, sk, ad = gpu.blkchol(Lm, A3, pars, absd, nlhs=4)
        Lf = dict(Lm, L=LL)
        y = None
        for _ in range(NSOLVE):
            p = gpu.fwblkslv(Lf, rhs)
            y = gpu.bwblkslv(Lf, p / Ld)
        ps = None
        for i in range(NPSD if lenud else 0):
            xfull[1 + (k * NPSD + i) % lenud] += 1e-6       # every psdscale call of a real run scales a different vector
            ps = gpu.psdscale({"u": d["u"], "perm": d["perm"]}, xfull, Km, float(i & 1))
        if not lenud and nq:
            for _ in range(6):
                gpu.qblkmul(LOR[0], LOR[1], qbs)
            for _ in range(3):
                gpu.ddot(d["q2"], LOR[1], qbs)
            gpu.quadadd(LOR[2], LOR[3], LOR[4], nlhs=2)
        if lenud:
            gpu.psdinvjmul(lab, frms, ps, Km)
            f = gpu.psdframeit(lab, frms, Km)
            f = gpu.psdframeit(lab, frms, Km)
            u2, p2, gjc, g = gpu.urotorder(d["u"], Km, 1.1, nlhs=4)
            gpu.givensrot(gjc, g, f, Km)
        return y

    step(0)
    L = sbdev.lib()
    h0, d0 = C.c_int64(0), C.c_int64(0)
    L.sb200_xfer_bytes(C.byref(h0), C.byref(d0))
    t0 = gpu.mex_seconds()
    w0 = time.perf_counter()
    for k in range(steps):
        step(k + 1)
    t = gpu.mex_seconds() - t0
    wall = time.perf_counter() - w0
    h1, d1 = C.c_int64(0), C.c_int64(0)
    L.sb200_xfer_bytes(C.byref(h1), C.byref(d1))
    return {"value": steps / t, "seconds": t, "unit": "iterations/s",
            "h2d_bytes_per_step": int((h1.value - h0.value) / steps), "d2h_bytes_per_step": int((d1.value - d0.value) / steps),
            "bytes": "counted by the library around every cudaMemcpyAsync (sb200_xfer_bytes)",
            "timed": "time inside the plugins' mexFunction (host numpy buffers in/out, all H2D/D2H and hashing inside), d.l, d.u, rhs, x "
                     f"perturbed every step; Python marshalling of mxArrays excluded; wall incl. marshalling {wall / steps * 1e3:.2f} ms/step",
            "steps": steps}


def secondary_entry(name, args, local_rank):
    """One of the other BASELINE configs on one GPU: device-resident it/s + its own parity gates."""
    t0 = time.perf_counter()
    W = load_workload(name)
    big = name.startswith("maxcut4") or name.startswith("dense")
    steps = 5 if big else 40
    out = device_run(W, args, 0, 1, local_rank, False, None, steps, 3, want_parity=not (big and args.quick_secondary))
    e = {"workload": DESCR[name][0], "value": steps / (out.ms_max * 1e-3), "unit": "iterations/s", "ms_per_step": out.ms_max / steps,
         "steps": steps, "gpu_launches_per_step": out.launches // steps,
         "top_kernel": None if not out.roof else {k: out.roof[k] for k in ("kernel", "bound", "achieved", "peak", "unit", "frac", "share_of_step")},
         "kernel_ms_per_step": None if not out.roof else dict(list(out.roof["kernel_ms_per_step"].items())[:6])}
    if out.parity is not None:
        p = out.parity
        e["parity"] = {"ok": p["ok"], "err": {k: float(f"{v:.3g}") for k, v in p["err"].items()}, "skip_equal": p.get("skip_equal"),
                       "add_equal": p.get("add_equal"), "urotorder_bit_exact": p.get("urotorder_bit_exact")}
        e["cpu_baseline"] = {"value": 1.0 / p["ref_seconds"], "unit": "iterations/s", "cores": 1, "kind": "reference",
                             "sample": "the one reference iteration of the parity gate"}
    else:
        e["parity"] = "not run in the bench (see tests/test_fullsize_gpu.py)"
    if not big and not args.no_e2e:
        e2 = run_e2e_mex(W, 10)
        e["e2e"] = {k: e2[k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "steps")}
    e["seconds_spent"] = round(time.perf_counter() - t0, 1)
    del out
    return e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=HEADLINE)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--secondary", default="control07,nb,arch0,maxcut4000,densecol")
    ap.add_argument("--full-secondary", dest="quick_secondary", action="store_false",
                    help="also run the oracle gates of the large secondary workloads (maxcut4000: about a minute of CPU)")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels one by one instead of replaying a CUDA graph")
    ap.add_argument("--replicas", action="store_true", help="N>1: N independent replicas (weak scaling) instead of sharding")
    ap.add_argument("--ref-blocks", type=int, default=4, help="reference arm: PSD blocks in the per-step sample (0 = all)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64, at most 64 MiB)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    name = args.workload
    descr, data = DESCR.get(name, (name, "synthetic"))
    config = {"workload": descr,
              "recipe": f"invcholfac,getada1,getada2,getada3,blkchol,{NSOLVE}x(fwblkslv,./d,bwblkslv),{NPSD}xpsdscale,"
                        "psdinvjmul,2xpsdframeit,urotorder,givensrot (SURVEY 8d)",
              "scaling_state": "S1 mid-run NT scaling (SURVEY 8d), seed 20260926",
              "l2": "L2 flushed (256 MiB write) between timed iterations",
              "launch": "one CUDA graph per iteration (kernels + NCCL collectives)" if not args.no_graph else "stream launches"}

    if args.impl == "reference":
        if rank != 0:
            return
        W = load_workload(name)
        r = run_reference(W, args.steps, args.warmup, sample_blocks=args.ref_blocks)
        v = r["steps"] / r["seconds"]
        config["parallelism"] = "reference C is single-threaded: 1 host core regardless of --gpus"
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "iterations/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / r["steps"],
                "higher_is_better": True, "scaling": "weak" if args.replicas else "strong", "vs_baseline": None,
                "dtype": "f64", "data": data, "config": config, "reference_scope": "1 core (the reference C is single-threaded; "
                "the same single-core figure at every --gpus)",
                "cpu_baseline": {"value": v, "unit": "iterations/s", "cores": 1, "kind": "reference",
                                 "sample": f"{r['steps']} steps: {r['sample']}; time inside the reference mexFunctions (oracle/_ref, gcc -O2) "
                                           f"+ numpy psdscale; harness marshalling excluded (wall {r['wall']:.1f}s)"},
                "e2e": {"value": v, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    from sedumi_b200 import device as sbdev
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    W = load_workload(name)
    nblk = len(W.S.K["s"])
    sharded = world > 1 and not args.replicas and nblk >= world
    if world > 1 and not sharded and not args.replicas:
        args.replicas = True                     # a problem with fewer PSD blocks than ranks does not shard: replicas only
    if sharded:
        def bcast(raw):
            t = torch.tensor(list(raw), dtype=torch.uint8, device=torch.device("cuda", local_rank))
            dist.broadcast(t, 0)
            return bytes(t.cpu().tolist())
        sbdev.comm_init(rank, world, local_rank, bcast)
    out = device_run(W, args, rank, world, local_rank, sharded, dist if world > 1 else None, args.steps, args.warmup,
                     want_parity=not args.no_parity, dump_dir=args.dump_outputs)
    config["parallelism"] = out.parallelism if sharded else (f"replicas x{world} (no data-path collective)" if world > 1 else "1 GPU")
    value = (1 if sharded else world) * args.steps / (out.ms_max * 1e-3)
    line = {"metric": METRIC, "value": value, "unit": "iterations/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": out.ms_max / args.steps, "higher_is_better": True,
            "scaling": "strong" if (sharded or world == 1) else "weak", "vs_baseline": None,
            "dtype": "f64", "data": data, "config": config,
            "gpu_launches": out.launches, "ms_per_step_no_flush": out.ms_warm, "wall_s": out.wall}
    if sharded:
        line["comm"] = out.comm
    # ---- e2e
    e2e = None
    if not args.no_e2e:
        if world > 1:
            dist.barrier()
        nsteps_e2e = max(20, min(40, args.steps))
        if world == 1:
            e2e = run_e2e_mex(W, nsteps_e2e if W.S.m < 2000 else 20)
            e2e["route"] = "MEX plugins (reference-facing boundary), host buffers"
        else:
            local_x = out.hp.psd_x.cpu().numpy()[:out.hp.lenud]
            e2e = e2e_device_api(W, out.hp, sharded, nsteps_e2e, world, dist, local_x)
            e2e["route"] = "device API with pinned host buffers (the MEX boundary is single-process / single-GPU)"
            if not sharded:
                e2e["value"] *= world
    if rank == 0:
        line["clocks"] = out.clocks
        line["roofline"] = out.roof
        if e2e is not None:
            line["e2e"] = e2e
        if out.parity is not None:
            p = out.parity
            line["parity"] = {"ok": p["ok"], "err": {k: float(f"{v:.3g}") for k, v in p["err"].items()}, "tol": p["tol"],
                              "skip_equal": p.get("skip_equal"), "add_equal": p.get("add_equal"), "nskip": p.get("nskip"), "nadd": p.get("nadd"),
                              "urotorder_bit_exact": p.get("urotorder_bit_exact"), "factor_scope": p.get("factor_scope", "all columns"),
                              "oracle": "oracle/_ref (unmodified reference C) on the same inputs, one iteration, before the timed region; "
                                        "psdscale against the numpy restatement of psdscale.m (M-only in the reference: parity unpinned beyond that)"}
            if not args.no_cpu_baseline:
                line["cpu_baseline"] = {"value": 1.0 / p["ref_seconds"], "unit": "iterations/s", "cores": 1, "kind": "reference",
                                        "sample": "1 full iteration of the same recipe on the same inputs (the one the parity gates compare against): "
                                                  f"reference mexFunctions (oracle/_ref, gcc -O2, single-threaded like the reference) + numpy psdscale, "
                                                  f"{p['ref_seconds']:.1f}s; harness marshalling excluded"}
        if not args.no_secondary and world == 1 and name == HEADLINE:
            sec = []
            for nm in [s for s in args.secondary.split(",") if s]:
                try:
                    sec.append(secondary_entry(nm, args, local_rank))
                except Exception as ex:          # a secondary workload must not take the headline line down with it
                    sec.append({"workload": nm, "error": f"{type(ex).__name__}: {ex}"})
            line["secondary"] = sec
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        # The communicators (torch's and the library's) are torn down by process exit: destroying an NCCL communicator
        # whose collectives live in instantiated CUDA graphs blocked for minutes on the B200 box (round-2 N=2 run).
        os._exit(0)


if __name__ == "__main__":
    main()
