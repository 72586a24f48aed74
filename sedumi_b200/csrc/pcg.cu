// pcg.cu -- wrapPcg on the device (SURVEY 8f row 1): the scaling operations, the products with the constraint matrix,
// the factor solves, the residuals and the PCG refinement loop of one search-direction computation.
//
// Reference semantics (wrapPcg.m:43-130, loopPcg.m:53-170, PopK.m:39-55, asmDxq.m:41-69, Amul.m:40-56, vecsym.c,
// psdscale.m).  The direct step:
//     dx  = D' rv            D' = [sqrt(d.l) .* ; asmDxq(d, .) ; psdscale(d, ., K, 1)]
//     r   = A dx + rb        (Amul: (x' At)' + dense.A x(dense.cols))
//     p   = L \ r ; y = p ./ L.d ; ssqrNew = p' y ; p = L' \ y        (with dense columns: fwdpr1 / bwdpr1 around ./d)
//     x   = vecsym(At p) ;  dx2 = D x ;  ssqrdx = |dx2|^2 ;  alpha = ssqrNew / ssqrdx
//     y   = alpha p ;  dx = rv - alpha dx2
//     r   = A D' dx + rb ;  normr = |r|_inf
// sb200_wrappcg_dev stops there (LP + PSD, no dense columns; scalars stay on the device and nothing synchronises).
// sb200_wrappcg_full_dev runs the same direct step with the Lorentz terms and LP dense columns, then loopPcg: each CG
// step ends in a few bytes of status read back through a pinned buffer, and the host side of the entry takes the
// decisions of loopPcg.m:126-136 and wrapPcg.m:100-130 on them.
//
// Layout of x (length N): [K.l | nq Lorentz trace entries | norm-bound parts (qdim) | PSD blocks (lenud)].
#include <algorithm>
#include <cmath>
#include "sb_internal.h"

extern "C" int sb200_ada_plan_csr(sb200_ada_plan *plan, const long long **Ajc, const int **Air, const double **Apr,
                                  const long long **rowptr, const int **rowcol, const int **rowsrc, sb_idx *N, sb_idx *m,
                                  sb_idx *lpN, sb_idx *nq);
extern "C" int sb200_psd_plan_blocks(sb200_psd_plan *plan, const int **n_dev, const long long **off_dev, int *nblk, int *maxn);
extern "C" int sb200_ldl_solve2_dev(sb200_chol_plan *plan, const double *Lrect_dev, const double *d_dev, const int *flag_dev,
                                    const double *b_dev, double *w_dev, double *y_dev, sb_idx nrhs, double *ssqr_dev);

namespace sb {

// y(j) = sum_r At(r,j) x(r) + sum_c Ad(j,c) x(cols(c)) (+ add(j)): one warp per column of At (Amul.m:46,52).
// Ad is dense.A, column-major m x nden; the At rows of dense columns are zero (setup), so the two sums do not overlap.
__global__ void __launch_bounds__(256)
pcg_at_dot_kernel(int m, const long long *Ajc, const int *Air, const double *Apr, const double *x, const double *add, double *y,
                  int nden, const double *Ad, const int *dcols) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (j >= m) return;
  double acc = 0.0;
  for (long long p = Ajc[j] + lane; p < Ajc[j + 1]; p += 32) acc += Apr[p] * x[Air[p]];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    if (nden) { double s = 0.0; for (int c = 0; c < nden; c++) s += Ad[(long long)c * m + j] * x[dcols[c]]; acc += s; }
    y[j] = acc + (add ? add[j] : 0.0);
  }
}
// y(r) = sum_j At(r,j) p(j): row-wise gather through the CSR copy of the pattern (deterministic, no atomics)
__global__ void pcg_at_mul_kernel(long long N, const long long *rowptr, const int *rowcol, const int *rowsrc, const double *Apr,
                                  const double *p, double *y) {
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < N; r += (long long)gridDim.x * blockDim.x) {
    double acc = 0.0;
    for (long long t = rowptr[r]; t < rowptr[r + 1]; t++) acc += Apr[rowsrc[t]] * p[rowcol[t]];
    y[r] = acc;
  }
}
// Amul.m:54: y(dense.cols(c)) = dense.A(:,c)' p, one warp per dense column
__global__ void pcg_dense_t_kernel(int m, int nden, const double *Ad, const int *dcols, const double *p, double *y) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (c >= nden) return;
  double acc = 0.0;
  for (int i = lane; i < m; i += 32) acc += Ad[(long long)c * m + i] * p[i];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  if (lane == 0) y[dcols[c]] = acc;
}
// vecsym.c:60-76 on every PSD block: Y = (X + X')/2, in place (each unordered pair is owned by its lower entry)
__global__ void pcg_vecsym_kernel(int nblk, const int *bn, const long long *boff, double *x) {
  const int k = blockIdx.y, n = bn[k];
  double *X = x + boff[k];
  const long long tot = (long long)n * n;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < tot; idx += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(idx % n), j = (int)(idx / n);
    if (i > j) { const double v = (X[idx] + X[j + (long long)i * n]) / 2; X[idx] = v; X[j + (long long)i * n] = v; }
  }
}
__global__ void pcg_lp_scale_kernel(int n, const double *dl, const double *x, double *y) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) y[i] = sqrt(dl[i]) * x[i];
}
// asmDxq.m:53-67, per Lorentz cone k (x1 = trace entry):  ddotx = given ? ddotx : q1 x1 + dd ;
// t = (ddotx + x1 auxdet) / auxtr ;  y_tr = t auxdet - sqrt(det) x1 (+ t q1) ;  sdet, t kept for the norm-bound rows
__global__ void pcg_asmdxq_tr_kernel(int nq, const double *x1, const double *ddotx_given, const double *dd, const double *det,
                                     const double *q1, const double *auxdet, const double *auxtr, double *ytr, double *sdet, double *tv) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < nq; k += gridDim.x * blockDim.x) {
    const double ddx = ddotx_given ? ddotx_given[k] : q1[k] * x1[k] + dd[k];
    const double t = (ddx + x1[k] * auxdet[k]) / auxtr[k], s = sqrt(det[k]);
    ytr[k] = (t * auxdet[k] - s * x1[k]) + t * q1[k];
    sdet[k] = s; tv[k] = t;
  }
}
__global__ void pcg_add_kernel(long long n, double *y, const double *x) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) y[i] += x[i];
}
// PopK.m:45-46, LP and trace rows:  y = [d.l .* x(1:K.l) ; -d.det .* x1] ;  ddotx = q1 .* x1 + dd
__global__ void pcg_popk_lt_kernel(int l, int nq, const double *dl, const double *det, const double *q1, const double *x,
                                   const double *dd, double *y, double *ddotx) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < l + nq; i += gridDim.x * blockDim.x) {
    if (i < l) y[i] = dl[i] * x[i];
    else { const int k = i - l; y[i] = -det[k] * x[i]; ddotx[k] = q1[k] * x[i] + dd[k]; }
  }
}
// deterministic reductions: per-block partials in a fixed partition, then one block sums them in order
template <int OP>   // 0: sum of squares, 1: max |.|, 2: sum x.*z
__global__ void __launch_bounds__(256) pcg_reduce1_kernel(long long n, const double *x, double *part, const double *z = nullptr) {
  __shared__ double sh[8];
  const long long per = (n + gridDim.x - 1) / gridDim.x, lo = blockIdx.x * per, hi = min(n, lo + per);
  double a = 0.0;
  for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    const double v = x[i];
    a = OP == 0 ? a + v * v : OP == 1 ? fmax(a, fabs(v)) : a + v * z[i];
  }
  for (int o = 16; o > 0; o >>= 1) { const double b = __shfl_down_sync(0xffffffffu, a, o); a = OP == 1 ? fmax(a, b) : a + b; }
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) { double t = sh[0]; for (int w = 1; w < 8; w++) t = OP == 1 ? fmax(t, sh[w]) : t + sh[w]; part[blockIdx.x] = t; }
}
template <int OP>
__global__ void pcg_reduce2_kernel(int np, const double *part, double *out, const double *num, double *ratio) {
  if (threadIdx.x == 0) {
    double t = part[0];
    for (int i = 1; i < np; i++) t = OP == 1 ? fmax(t, part[i]) : t + part[i];
    *out = t;
    if (ratio) *ratio = t > 0.0 ? *num / t : 0.0;          // alpha = ssqrNew / ssqrdx (0 when dx vanishes, wrapPcg.m:68-73)
  }
}
// y = alpha p ;  dx = rv - alpha dx2
__global__ void pcg_step_kernel(long long N, int m, const double *alpha, const double *p, double *y, const double *rv, const double *dx2, double *dx) {
  const double a = *alpha;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N + m; i += (long long)gridDim.x * blockDim.x) {
    if (i < m) y[i] = a * p[i];
    else { const long long t = i - m; dx[t] = rv[t] - a * dx2[t]; }
  }
}

// ---- loopPcg (loopPcg.m:66-141) device pieces.  Scalar slots of one CG step, in device memory:
enum { S_SSQRNEW = 0, S_SSQROLD, S_SSQRDAP, S_ALPHA, S_FINEW, S_NORMR, S_SSQRDX, S_NSLOT };

// loopPcg.m:74-85: p = q (first step of a trial) or p = (ssqrNew/ssqrOld) p + q
__global__ void pcg_pupdate_kernel(int m, int first, const double *sc, const double *q, double *p) {
  const double beta = first ? 0.0 : sc[S_SSQRNEW] / sc[S_SSQROLD];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) p[i] = first ? q[i] : beta * p[i] + q[i];
}
// xTy (PopK.m:53-55) from three partial sets; alpha = ssqrNew / ssqrDAp, written only when ssqrDAp > 0 (loopPcg.m:93-98)
__global__ void pcg_popk_reduce2_kernel(int np, const double *part, double *sc) {
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0, c = 0.0;
    for (int i = 0; i < np; i++) a += part[i];
    for (int i = 0; i < np; i++) b += part[np + i];
    for (int i = 0; i < np; i++) c += part[2 * np + i];
    const double s = (a + b) + c;
    sc[S_SSQRDAP] = s;
    if (s > 0.0) sc[S_ALPHA] = sc[S_SSQRNEW] / s;
  }
}
// ap = alpha p (the increment quadadd adds), or y += alpha p directly when qprec = 0
__global__ void pcg_axpy_kernel(int m, const double *sc, const double *p, double *ap, const double *yin, double *yout) {
  const double a = sc[S_SSQRDAP] > 0.0 ? sc[S_ALPHA] : 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
    if (ap) ap[i] = a * p[i];
    else yout[i] = yin[i] + a * p[i];
  }
}
// loopPcg.m:113-115: tmp = Amul(At, dense, DDAp) + DAt.q' ddotx ;  r = r - alpha tmp.  One warp per constraint.
__global__ void __launch_bounds__(256)
pcg_resid_kernel(int m, const long long *Ajc, const int *Air, const double *Apr, const double *x, int nden, const double *Ad,
                 const int *dcols, const long long *Qjc, const int *Qir, const double *Qpr, const double *ddotx, const double *sc, double *r) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (j >= m) return;
  double acc = 0.0, accq = 0.0;
  for (long long p = Ajc[j] + lane; p < Ajc[j + 1]; p += 32) acc += Apr[p] * x[Air[p]];
  if (Qjc) for (long long p = Qjc[j] + lane; p < Qjc[j + 1]; p += 32) accq += Qpr[p] * ddotx[Qir[p]];
  for (int o = 16; o > 0; o >>= 1) { acc += __shfl_down_sync(0xffffffffu, acc, o); accq += __shfl_down_sync(0xffffffffu, accq, o); }
  if (lane == 0) {
    if (nden) { double s = 0.0; for (int c = 0; c < nden; c++) s += Ad[(long long)c * m + j] * x[dcols[c]]; acc += s; }
    const double a = sc[S_SSQRDAP] > 0.0 ? sc[S_ALPHA] : 0.0;
    r[j] = r[j] - a * (acc + accq);
  }
}
// loopPcg.m:119-125 partials: (b+r)'y.hi, (b+r)'y.lo and |r|_inf over a fixed partition
__global__ void __launch_bounds__(256) pcg_cgstat1_kernel(int m, const double *b, const double *r, const double *yhi, const double *ylo, double *part) {
  __shared__ double sh[3][8];
  const int per = (m + gridDim.x - 1) / gridDim.x, lo = blockIdx.x * per, hi = min(m, lo + per);
  double s1 = 0.0, s2 = 0.0, mx = 0.0;
  for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    const double br = b[i] + r[i];
    s1 += br * yhi[i];
    if (ylo) s2 += br * ylo[i];
    mx = fmax(mx, fabs(r[i]));
  }
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_down_sync(0xffffffffu, s1, o); s2 += __shfl_down_sync(0xffffffffu, s2, o);
    mx = fmax(mx, __shfl_down_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s1; sh[1][threadIdx.x >> 5] = s2; sh[2][threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = sh[0][0], c = sh[1][0], e = sh[2][0];
    for (int w = 1; w < 8; w++) { a += sh[0][w]; c += sh[1][w]; e = fmax(e, sh[2][w]); }
    part[blockIdx.x] = a; part[gridDim.x + blockIdx.x] = c; part[2 * gridDim.x + blockIdx.x] = e;
  }
}
__global__ void pcg_cgstat2_kernel(int np, const double *part, double *sc) {
  if (threadIdx.x == 0) {
    double a = part[0], c = part[np], e = part[2 * np];
    for (int i = 1; i < np; i++) { a += part[i]; c += part[np + i]; e = fmax(e, part[2 * np + i]); }
    sc[S_FINEW] = a + c;
    sc[S_NORMR] = e;
  }
}
__global__ void pcg_scale_kernel(long long n, const double *sc, double *x) {
  const double a = sc[S_ALPHA];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) x[i] *= a;
}
// wrapPcg.m:112-114: y = y + dy ; dx = dx - x
__global__ void pcg_accum_kernel(int m, long long N, double *y, const double *dy, double *dx, const double *x) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < m + N; i += (long long)gridDim.x * blockDim.x) {
    if (i < m) y[i] = y[i] + dy[i];
    else dx[i - m] = dx[i - m] - x[i - m];
  }
}

static unsigned pgrid(long long n) { return (unsigned)std::max<long long>(1, std::min<long long>((n + 255) / 256, 2048)); }
static const int NP = 256;     // partials of every reduction: a fixed partition, independent of the device

// Everything one search-direction computation needs; the direct step and the CG step are methods on it.
struct Pcg {
  cudaStream_t st;
  // At (column and row views), cone layout
  const long long *Ajc, *rowptr; const int *Air, *rowcol, *rowsrc; const double *Apr;
  sb_idx N, m, lpN, nq, qdim, lenud;
  sb200_psd_plan *pp; sb200_chol_plan *cp; sb200_dpr1_plan *dpr1;
  const double *dl, *u; const int *perm;
  const double *Lrect, *Ld; const int *flag;
  const sb200_pcg_cones *cq;             // NULL: no Lorentz cones, no dense columns
  const long long *Qjc = nullptr; const int *Qir = nullptr; const double *Qpr = nullptr;   // DAt.q (nq x m CSC)
  const double *rb;
  // scratch
  double *part, *qdd, *qt, *qsdet, *qtmp, *lrcopy;

  int nden() const { return cq ? (int)cq->nden : 0; }
  const double *Ad() const { return cq ? cq->denA_dev : nullptr; }
  const int *dcols() const { return cq ? cq->den_cols_dev : nullptr; }

  // y = Amul(At, dense, x) (+ add)
  int amul(const double *x, const double *add, double *y) {
    pcg_at_dot_kernel<<<(unsigned)((m + 7) / 8), 256, 0, st>>>((int)m, Ajc, Air, Apr, x, add, y, nden(), Ad(), dcols());
    SB_LAUNCH_CHECK_N("pcg_at_dot_kernel");
    return 0;
  }
  // y = vecsym(Amul(At, dense, p, 1), K)
  int amul_t(const double *p, double *y) {
    pcg_at_mul_kernel<<<pgrid(N), 256, 0, st>>>(N, rowptr, rowcol, rowsrc, Apr, p, y);
    SB_LAUNCH_CHECK_N("pcg_at_mul_kernel");
    if (nden()) {
      pcg_dense_t_kernel<<<(unsigned)((nden() + 7) / 8), 256, 0, st>>>((int)m, nden(), Ad(), dcols(), p, y);
      SB_LAUNCH_CHECK_N("pcg_dense_t_kernel");
    }
    if (lenud) {
      const int *bn; const long long *boff; int nblk, maxn;
      SB_TRY(sb200_psd_plan_blocks(pp, &bn, &boff, &nblk, &maxn));
      dim3 g((unsigned)std::min<long long>(((long long)maxn * maxn + 255) / 256, 1024), (unsigned)nblk);
      pcg_vecsym_kernel<<<g, 256, 0, st>>>(nblk, bn, boff, y + lpN + nq + qdim);
      SB_LAUNCH_CHECK_N("pcg_vecsym_kernel");
    }
    return 0;
  }
  // asmDxq(d, x, K [, ddotx]) into y (trace rows and norm-bound rows, x and y full-length)
  int asmdxq(const double *x, const double *ddotx_given, double *y) {
    const double *x1 = x + lpN, *x2 = x + lpN + nq;
    if (!ddotx_given) SB_TRY(sb200_ddot_dense_dev(nq, cq->qbs_dev, cq->q2_dev, x2, qdim, 1, qdd));
    pcg_asmdxq_tr_kernel<<<pgrid(nq), 256, 0, st>>>((int)nq, x1, ddotx_given, qdd, cq->det_dev, cq->q1_dev, cq->auxdet_dev,
                                                     cq->auxtr_dev, y + lpN, qsdet, qt);
    SB_LAUNCH_CHECK_N("pcg_asmdxq_tr_kernel");
    SB_TRY(sb200_qblkmul_dev(nq, cq->qbs_dev, qdim, qsdet, x2, y + lpN + nq));     // qblkmul(sdet, x)
    SB_TRY(sb200_qblkmul_dev(nq, cq->qbs_dev, qdim, qt, cq->q2_dev, qtmp));         // + qblkmul(t, d.q2)
    pcg_add_kernel<<<pgrid(qdim), 256, 0, st>>>(qdim, y + lpN + nq, qtmp);
    SB_LAUNCH_CHECK_N("pcg_add_kernel");
    return 0;
  }
  // y = D x (transp 0) resp. D' x (transp 1); ddotx_given: asmDxq's 4th argument
  int scaleD(const double *x, double *y, int transp, const double *ddotx_given = nullptr) {
    if (lpN) { pcg_lp_scale_kernel<<<pgrid(lpN), 256, 0, st>>>((int)lpN, dl, x, y); SB_LAUNCH_CHECK_N("pcg_lp_scale_kernel"); }
    if (nq) SB_TRY(asmdxq(x, ddotx_given, y));
    if (lenud) SB_TRY(sb200_psdscale_dev(pp, u, perm, x + lpN + nq + qdim, transp, y + lpN + nq + qdim));
    return 0;
  }
  // w = (L \ r) ./ d, q = L' \ w, *ssqr = (L \ r)' w   (wrapPcg.m:56-59, loopPcg.m:72-76; Lden between when dense)
  int precond(const double *r, double *w, double *q, double *ssqr) {
    if (!dpr1) return sb200_ldl_solve2_dev(cp, Lrect, Ld, flag, r, w, q, 1, ssqr);
    SB_TRY(sb200_fwblkslv_dev(cp, Lrect, r, w, 1));
    SB_TRY(sb200_dpr1solve_dev(dpr1, 0, w, 1));
    SB_CUDA(cudaMemcpyAsync(lrcopy, w, sizeof(double) * m, cudaMemcpyDeviceToDevice, st));
    SB_TRY(sb200_scale_by_d_dev(m, 1, Ld, flag, sb200_chol_plan_lb_dev(cp), w));
    pcg_reduce1_kernel<2><<<NP, 256, 0, st>>>(m, lrcopy, part, w);
    SB_LAUNCH_CHECK_N("pcg_reduce_kernel");
    pcg_reduce2_kernel<2><<<1, 32, 0, st>>>(NP, part, ssqr, nullptr, nullptr);
    SB_LAUNCH_CHECK_N("pcg_reduce_kernel");
    SB_TRY(sb200_dpr1solve_dev(dpr1, 1, w, 1));
    return sb200_bwblkslv_dev(cp, Lrect, w, q, 1);
  }
  // r = A D' dx + rb ; *normr = |r|_inf
  int residual(const double *dx, double *t, double *r, double *normr) {
    SB_TRY(scaleD(dx, t, 1));
    SB_TRY(amul(t, rb, r));
    pcg_reduce1_kernel<1><<<NP, 256, 0, st>>>(m, r, part + NP);
    SB_LAUNCH_CHECK_N("pcg_reduce_kernel");
    pcg_reduce2_kernel<1><<<1, 32, 0, st>>>(NP, part + NP, normr, nullptr, nullptr);
    SB_LAUNCH_CHECK_N("pcg_reduce_kernel");
    return 0;
  }
  // wrapPcg.m:46-90.  t1..t3: N doubles each; pv, wv: m.  scal[0..3] = ssqrNew, ssqrdx, alpha, normr.
  int direct_step(const double *rv, double *y, double *dx, double *r, double *scal, double *t1, double *t2, double *t3, double *pv, double *wv) {
    SB_TRY(scaleD(rv, t1, 1));                                   // dx = D' rv ; r = A dx + rb
    SB_TRY(amul(t1, rb, r));
    SB_TRY(precond(r, wv, pv, scal + 0));                        // p = L' \ ((L \ r) ./ d), ssqrNew
    SB_TRY(amul_t(pv, t1));                                      // x = vecsym(At p) ; dx2 = D x ; ssqrdx ; alpha
    SB_TRY(scaleD(t1, t2, 0));
    pcg_reduce1_kernel<0><<<NP, 256, 0, st>>>(N, t2, part);
    SB_LAUNCH_CHECK_N("pcg_reduce_kernel");
    pcg_reduce2_kernel<0><<<1, 32, 0, st>>>(NP, part, scal + 1, scal + 0, scal + 2);
    SB_LAUNCH_CHECK_N("pcg_reduce_kernel");
    pcg_step_kernel<<<pgrid(N + m), 256, 0, st>>>(N, (int)m, scal + 2, pv, y, rv, t2, dx);   // y = alpha p ; dx = rv - alpha dx2
    SB_LAUNCH_CHECK_N("pcg_step_kernel");
    return residual(dx, t3, r, scal + 3);                        // r = A D' dx + rb ; normr
  }
};

// pinned status words read back by the host side of the CG loop (allocated once, kept for the process)
static double *pinned_status() {
  static double *h = nullptr;
  if (!h && cudaHostAlloc((void **)&h, 16 * sizeof(double), cudaHostAllocDefault) != cudaSuccess) h = nullptr;
  return h;
}
static int read_status(const double *sc_dev, int n, double *out) {
  double *h = pinned_status();
  SB_CHECK(h, "wrappcg_full_dev: pinned status buffer could not be allocated");
  SB_CUDA(cudaMemcpyAsync(h, sc_dev, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx().stream));
  SB_CUDA(cudaStreamSynchronize(ctx().stream));
  for (int i = 0; i < n; i++) out[i] = h[i];
  return 0;
}

}  // namespace sb
using namespace sb;

extern "C" {

// work_dev: 3 N + 2 m + 600 doubles of scratch.  scal_dev[0..3] = ssqrNew, ssqrdx, alpha, normr.
int sb200_wrappcg_dev(sb200_ada_plan *ap, sb200_psd_plan *pp, sb200_chol_plan *cp, const double *dl_dev, const double *u_dev,
                      const int *perm_dev, const double *Lrect_dev, const double *Ld_dev, const int *flag_dev, const double *rv_dev,
                      const double *rb_dev, double *y_dev, double *dx_dev, double *r_dev, double *scal_dev, double *work_dev) {
  SB_TRY(ensure_init());
  Pcg P{};
  SB_TRY(sb200_ada_plan_csr(ap, &P.Ajc, &P.Air, &P.Apr, &P.rowptr, &P.rowcol, &P.rowsrc, &P.N, &P.m, &P.lpN, &P.nq));
  SB_CHECK(P.nq == 0, "wrappcg_dev: Lorentz cones are not handled on the device (asmDxq.m)");
  P.lenud = sb200_psd_plan_lenud(pp);
  SB_CHECK(P.lpN + P.lenud == P.N, "wrappcg_dev: cone layout does not match At (%lld + %lld != %lld)", (long long)P.lpN,
           (long long)P.lenud, (long long)P.N);
  P.st = ctx().stream; P.qdim = 0; P.pp = pp; P.cp = cp; P.dpr1 = nullptr; P.cq = nullptr;
  P.dl = dl_dev; P.u = u_dev; P.perm = perm_dev; P.Lrect = Lrect_dev; P.Ld = Ld_dev; P.flag = flag_dev; P.rb = rb_dev;
  const sb_idx N = P.N, m = P.m;
  double *t1 = work_dev, *t2 = t1 + N, *t3 = t2 + N, *pv = t3 + N, *wv = pv + m;
  P.part = wv + m;
  return P.direct_step(rv_dev, y_dev, dx_dev, r_dev, scal_dev, t1, t2, t3, pv, wv);
}

sb_idx sb200_wrappcg_full_work(sb_idx N, sb_idx m, sb_idx nq, sb_idx qdim) {
  return 8 * N + 13 * m + 4 * nq + qdim + 4 * NP + 64;
}

int sb200_wrappcg_full_dev(sb200_ada_plan *ap, sb200_psd_plan *pp, sb200_chol_plan *cp, sb200_dpr1_plan *dpr1,
                           const sb200_pcg_cones *cq, const sb200_cgpars *cg, const double *dl_dev, const double *u_dev,
                           const int *perm_dev, const double *Lrect_dev, const double *Ld_dev, const int *flag_dev,
                           const double *rv_dev, const double *rb_dev, double y0, double *y_dev, double *dx_dev, double *r_dev,
                           sb200_pcg_status *status, double *work_dev) {
  SB_TRY(ensure_init());
  cudaStream_t st = ctx().stream;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  SB_CUDA(cudaStreamIsCapturing(st, &cs));
  SB_CHECK(cs == cudaStreamCaptureStatusNone && !ctx().capturing,
           "wrappcg_full_dev: the library stream is being captured; the PCG loop reads its status back on the host and "
           "cannot run inside a CUDA graph");
  SB_CHECK(cq && cg && status, "wrappcg_full_dev: cones, cgpars and status must be given");
  SB_CHECK(cq->ndenq == 0, "wrappcg_full_dev: dense Lorentz blocks (dense.q) are not handled on the device");
  SB_CHECK((cq->nden == 0) == (dpr1 == nullptr), "wrappcg_full_dev: LP dense columns need the dpr1 plan, and only they");
  Pcg P{};
  SB_TRY(sb200_ada_plan_csr(ap, &P.Ajc, &P.Air, &P.Apr, &P.rowptr, &P.rowcol, &P.rowsrc, &P.N, &P.m, &P.lpN, &P.nq));
  SB_CHECK(P.nq == cq->nq, "wrappcg_full_dev: %lld Lorentz cones in At, %lld given", (long long)P.nq, (long long)cq->nq);
  P.qdim = P.nq ? cq->qdim : 0;
  P.lenud = sb200_psd_plan_lenud(pp);
  SB_CHECK(P.lpN + P.nq + P.qdim + P.lenud == P.N, "wrappcg_full_dev: cone layout does not match At (%lld + %lld + %lld + %lld != %lld)",
           (long long)P.lpN, (long long)P.nq, (long long)P.qdim, (long long)P.lenud, (long long)P.N);
  P.st = st; P.pp = pp; P.cp = cp; P.dpr1 = dpr1; P.cq = cq;
  P.dl = dl_dev; P.u = u_dev; P.perm = perm_dev; P.Lrect = Lrect_dev; P.Ld = Ld_dev; P.flag = flag_dev; P.rb = rb_dev;
  const sb_idx N = P.N, m = P.m, nq = P.nq;
  // scratch
  double *w = work_dev;
  auto take = [&](sb_idx n) { double *p = w; w += std::max<sb_idx>(n, 1); return p; };
  double *t1 = take(N), *t2 = take(N), *t3 = take(N), *Ap = take(N), *DDAp = take(N), *Dx = take(N), *xN = take(N), *DAy = take(N);
  double *pv = take(m), *wv = take(m), *qv = take(m), *bv = take(m), *rl = take(m), *apv = take(m);
  double *yh[2] = {take(m), take(m)}, *yl[2] = {take(m), take(m)}, *ymh = take(m), *yml = take(m);
  P.lrcopy = take(m);
  P.qdd = take(nq); P.qt = take(nq); P.qsdet = take(nq);
  double *ddotx = take(nq);
  P.qtmp = take(P.qdim);
  P.part = take(4 * NP);
  double *scal = take(8), *sc = take(S_NSLOT + 2);
  if (nq) {            // DAt.q of the given scaling (getDAtm.m:40-43), the plan's own CSC
    SB_TRY(sb200_getdatm_dev(ap, cq->q1_dev, cq->q2_dev));
    const long long *jc; const int *ir; const double *pr; sb_idx nnz;
    SB_TRY(sb200_ada_plan_datq(ap, &jc, &ir, &pr, &nnz));
    if (nnz) { P.Qjc = jc; P.Qir = ir; P.Qpr = pr; }
  }
  const int qprec = cg->qprec > 0;
  const double restol = y0 * cg->restol;                         // wrapPcg.m:46
  *status = sb200_pcg_status{0, 0, 0, 0.0};

  // ---- direct step: one read-back (ssqrdx, normr)
  SB_TRY(P.direct_step(rv_dev, y_dev, dx_dev, r_dev, scal, t1, t2, t3, pv, wv));
  double hs[4];
  SB_TRY(read_status(scal, 4, hs));
  status->normr = hs[3];
  if (hs[1] <= 0.0) {                                          // wrapPcg.m:68-73: y = 0, k = 0, dx = rv
    SB_CUDA(cudaMemsetAsync(y_dev, 0, sizeof(double) * m, st));
    SB_CUDA(cudaMemcpyAsync(dx_dev, rv_dev, sizeof(double) * N, cudaMemcpyDeviceToDevice, st));
    SB_CUDA(cudaStreamSynchronize(st));
    return 0;
  }
  status->k = 1;
  if (hs[3] < restol) return 0;                                  // wrapPcg.m:91-93
  // ssqrNew of the direct step seeds the first loopPcg call (its p is pv)
  SB_CUDA(cudaMemcpyAsync(sc + S_SSQRNEW, scal + 0, sizeof(double), cudaMemcpyDeviceToDevice, st));
  int trial = 0;
  bool p_empty = false;
  for (;;) {
    // ---- loopPcg.m:56-141
    SB_CUDA(cudaMemcpyAsync(bv, r_dev, sizeof(double) * m, cudaMemcpyDeviceToDevice, st));
    SB_CUDA(cudaMemcpyAsync(rl, r_dev, sizeof(double) * m, cudaMemcpyDeviceToDevice, st));
    SB_CUDA(cudaMemsetAsync(yh[0], 0, sizeof(double) * m, st));
    SB_CUDA(cudaMemsetAsync(yl[0], 0, sizeof(double) * m, st));
    int cur = 0, stop = 0;
    sb_idx k = 0;
    bool y_empty = true, ymin_empty = true;
    double finew = 0.0, normrmin = hs[3];                        // norm(b, inf): b is the current wrapPcg residual
    while (stop == 0) {
      // preconditioner and conjugate direction
      if (!p_empty) SB_CUDA(cudaMemcpyAsync(sc + S_SSQROLD, sc + S_SSQRNEW, sizeof(double), cudaMemcpyDeviceToDevice, st));
      SB_TRY(P.precond(rl, wv, qv, sc + S_SSQRNEW));
      pcg_pupdate_kernel<<<pgrid(m), 256, 0, st>>>((int)m, p_empty ? 1 : 0, sc, qv, pv);
      SB_LAUNCH_CHECK_N("pcg_pupdate_kernel");
      p_empty = false;
      // Ap = vecsym(Amul(At, dense, p, 1)) ; PopK: DDAp, ddotx, Dx, ssqrDAp ; alpha
      SB_TRY(P.amul_t(pv, Ap));
      if (nq) SB_TRY(sb200_ddot_dense_dev(nq, cq->qbs_dev, cq->q2_dev, Ap + P.lpN + nq, P.qdim, 1, P.qdd));
      if (P.lpN + nq) {
        pcg_popk_lt_kernel<<<pgrid(P.lpN + nq), 256, 0, st>>>((int)P.lpN, (int)nq, dl_dev, nq ? cq->det_dev : nullptr,
                                                               nq ? cq->q1_dev : nullptr, Ap, P.qdd, DDAp, ddotx);
        SB_LAUNCH_CHECK_N("pcg_popk_lt_kernel");
      }
      if (nq) SB_TRY(sb200_qblkmul_dev(nq, cq->qbs_dev, P.qdim, cq->det_dev, Ap + P.lpN + nq, DDAp + P.lpN + nq));
      const sb_idx o = P.lpN + nq + P.qdim, lq = o;
      if (P.lenud) {
        SB_TRY(sb200_psdscale_dev(pp, u_dev, perm_dev, Ap + o, 0, Dx + o));
        SB_TRY(sb200_psdscale_dev(pp, u_dev, perm_dev, Dx + o, 1, DDAp + o));
      }
      pcg_reduce1_kernel<2><<<NP, 256, 0, st>>>(lq, Ap, P.part, DDAp);
      SB_LAUNCH_CHECK_N("pcg_reduce_kernel");
      pcg_reduce1_kernel<0><<<NP, 256, 0, st>>>(nq, ddotx, P.part + NP);
      SB_LAUNCH_CHECK_N("pcg_reduce_kernel");
      pcg_reduce1_kernel<0><<<NP, 256, 0, st>>>(P.lenud, Dx + o, P.part + 2 * NP);
      SB_LAUNCH_CHECK_N("pcg_reduce_kernel");
      pcg_popk_reduce2_kernel<<<1, 32, 0, st>>>(NP, P.part, sc);
      SB_LAUNCH_CHECK_N("pcg_popk_reduce2_kernel");
      // y := y + alpha p into the other buffer pair (kept only when ssqrDAp > 0)
      const int nxt = 1 - cur;
      if (qprec) {
        pcg_axpy_kernel<<<pgrid(m), 256, 0, st>>>((int)m, sc, pv, apv, nullptr, nullptr);
        SB_LAUNCH_CHECK_N("pcg_axpy_kernel");
        SB_TRY(sb200_quadadd_dev(m, yh[cur], yl[cur], apv, yh[nxt], yl[nxt]));
      } else {
        pcg_axpy_kernel<<<pgrid(m), 256, 0, st>>>((int)m, sc, pv, nullptr, yh[cur], yh[nxt]);
        SB_LAUNCH_CHECK_N("pcg_axpy_kernel");
      }
      // r := r - alpha (Amul(At, dense, DDAp) + DAt.q' ddotx) ; finew, normr
      pcg_resid_kernel<<<(unsigned)((m + 7) / 8), 256, 0, st>>>((int)m, P.Ajc, P.Air, P.Apr, DDAp, P.nden(), P.Ad(), P.dcols(),
                                                                 P.Qjc, P.Qir, P.Qpr, ddotx, sc, rl);
      SB_LAUNCH_CHECK_N("pcg_resid_kernel");
      pcg_cgstat1_kernel<<<NP, 256, 0, st>>>((int)m, bv, rl, yh[nxt], qprec ? yl[nxt] : nullptr, P.part);
      SB_LAUNCH_CHECK_N("pcg_cgstat_kernel");
      pcg_cgstat2_kernel<<<1, 32, 0, st>>>(NP, P.part, sc);
      SB_LAUNCH_CHECK_N("pcg_cgstat_kernel");
      double h[S_NSLOT];
      SB_TRY(read_status(sc, S_NSLOT, h));
      if (h[S_SSQRDAP] > 0.0) {
        k++;
        cur = nxt; y_empty = false;
        const double fiprev = finew, normr = h[S_NORMR];
        finew = h[S_FINEW];
        if (normr < normrmin) {
          SB_CUDA(cudaMemcpyAsync(ymh, yh[cur], sizeof(double) * m, cudaMemcpyDeviceToDevice, st));
          if (qprec) SB_CUDA(cudaMemcpyAsync(yml, yl[cur], sizeof(double) * m, cudaMemcpyDeviceToDevice, st));
          ymin_empty = false;
          normrmin = normr;
        }
        if (normr < restol) stop = 1;
        else if (finew - fiprev < cg->stagtol * fiprev) stop = 2;
        else if (k >= cg->maxiter) stop = 2;
      } else {
        stop = 1;                                                // loopPcg.m:137-140: DAp == 0, cannot go on
      }
    }
    status->stop = stop;
    // ---- loopPcg.m:145-170: the result y and DAy = D A' y
    const double *ryh = yh[cur], *ryl = yl[cur];
    bool empty = y_empty;
    if (stop == 2) { ryh = ymh; ryl = yml; empty = ymin_empty; }
    if (empty) return 0;                                         // wrapPcg.m:103-104: y, dx as they are
    if (k == 1) {
      // alpha [sqrt(d.l) Ap(1:K.l) ; asmDxq(d, Ap, K, DApq) ; DAps]: Ap, Dx hold the last PopK call, alpha its last step
      if (P.lpN) { pcg_lp_scale_kernel<<<pgrid(P.lpN), 256, 0, st>>>((int)P.lpN, dl_dev, Ap, DAy); SB_LAUNCH_CHECK_N("pcg_lp_scale_kernel"); }
      if (nq) SB_TRY(P.asmdxq(Ap, ddotx, DAy));
      if (P.lenud) SB_CUDA(cudaMemcpyAsync(DAy + P.lpN + nq + P.qdim, Dx + P.lpN + nq + P.qdim, sizeof(double) * P.lenud, cudaMemcpyDeviceToDevice, st));
      pcg_scale_kernel<<<pgrid(N), 256, 0, st>>>(N, sc, DAy);
      SB_LAUNCH_CHECK_N("pcg_scale_kernel");
    } else {
      SB_TRY(P.amul_t(ryh, t1));
      SB_TRY(P.scaleD(t1, DAy, 0));
      if (qprec) {
        SB_TRY(P.amul_t(ryl, t1));
        SB_TRY(P.scaleD(t1, t2, 0));
        pcg_add_kernel<<<pgrid(N), 256, 0, st>>>(N, DAy, t2);
        SB_LAUNCH_CHECK_N("pcg_add_kernel");
      }
    }
    // ---- wrapPcg.m:112-128
    status->k += k;
    pcg_accum_kernel<<<pgrid(m + N), 256, 0, st>>>((int)m, N, y_dev, ryh, dx_dev, DAy);
    SB_LAUNCH_CHECK_N("pcg_accum_kernel");
    SB_TRY(P.residual(dx_dev, xN, r_dev, scal + 3));
    SB_TRY(read_status(scal, 4, hs));
    status->normr = hs[3];
    if (hs[3] < restol || trial >= cg->refine) return 0;
    p_empty = true;                                              // refine: restart with p = []
    trial++;
    status->trials = trial;
  }
}

}  // extern "C"
