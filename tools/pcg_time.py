"""Device time of the search direction (HotPath.pcg -> sb200_wrappcg_full_dev): the direct step alone (exact factor)
and the cost of one CG step (factor of a perturbed scaling, so that loopPcg runs), with CUDA events, on the 64x200
block-diagonal SDP (BASELINE.json configs[3]) and on nb.  Prints one JSON object; the card's name and power limit are
read in the same run.  Usage: python tools/pcg_time.py [--reps R] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import pcg_cases as pc  # noqa: E402
from sedumi_b200 import device  # noqa: E402
from sedumi_b200.host import problems  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(hp, rv, rb, reps, **kw):
    import torch
    L = device.lib()
    hp.pcg(rv, rb, **kw)                      # warm-up: allocations, plan views
    ms, out = [], None
    l0 = L.sb200_kernel_launches()
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(hp.stream()):
            e0.record()
            out = hp.pcg(rv, rb, **kw)
            e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    launches = (L.sb200_kernel_launches() - l0) / reps
    return float(np.median(ms)), out, launches


def run(name, S, d0, eps, reps):
    import torch
    d1 = pc.perturb(d0, S.K, eps, 9)
    rv, rb = pc.rhs(S, 2)
    hp = device.HotPath(S)
    with torch.cuda.stream(hp.stream()):
        hp.set_scaling(d0)
        hp.invcholfac(); hp.getada(); hp.blkchol(); hp.deninfac()
        hp.sync()
    t_direct, o_direct, l_direct = timed(hp, rv, rb, reps)
    hp.set_scaling(d1)
    t_ref, o_ref, l_ref = timed(hp, rv, rb, reps)
    steps = o_ref["k"] - 1
    return dict(problem=name, m=S.m, N=int(S.At.shape[0]), direct_step_ms=t_direct, direct_k=o_direct["k"],
                direct_launches=l_direct, refined_ms=t_ref, refined_k=o_ref["k"], refined_trials=o_ref["trials"],
                refined_stop=o_ref["stop"], ms_per_cg_step=(t_ref - t_direct) / max(steps, 1),
                launches_per_cg_step=(l_ref - l_direct) / max(steps, 1),
                note="per CG step = (refined call - direct call) / (k - 1); includes the per-step status read-back "
                     "and the final D A'y product of each loopPcg call")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    raw = problems.synth_blockdiag_sdp()
    S64 = pc.build(raw, perm=np.arange(raw[0].shape[1]))
    Snb = pc.build(problems.load_fixture("nb"))
    res = dict(card=card(), reps=a.reps, timing="CUDA events around HotPath.pcg on the library stream, median of reps",
               results=[run("blockdiag64 (64 x 200, m=5000)", S64, pc.scaling(S64.K, problems.SEED0 + 2), 0.1, a.reps),
                        run("nb (793 Lorentz cones, m=123)", Snb, pc.scaling(Snb.K, 3), 0.3, a.reps)])
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
