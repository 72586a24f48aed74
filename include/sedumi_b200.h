/* sedumi_b200.h -- C-ABI of libsedumi_b200.so: the B200 (sm_100a) implementation of
 * SeDuMi's per-iteration normal-equations hot path.
 *
 * Boundary contract.  The reference's FFI for this path is the MEX plugin interface:
 * one `mexFunction(nlhs, plhs, nrhs, prhs)` per target (install_sedumi.m:70-110).  The
 * MEX stubs in sedumi_b200/mex/<target>.cpp keep those names and mxArray signatures and
 * do nothing but unpack mxArrays into the plain pointers below.  Every entry point cites
 * the reference mexFunction it stands behind.
 *
 * Conventions
 *   - all matrices column-major IEEE double; sparse matrices CSC with 0-based int64 jc/ir
 *     (bit-compatible with MATLAB's mwIndex on 64-bit platforms);
 *   - index vectors that MATLAB passes as 1-based doubles (perm, xsuper, blkstart...) are
 *     converted by the stub to 0-based int64 before they get here;
 *   - functions return 0 on success, nonzero on failure (sb200_last_error() has the text);
 *     nothing in this library calls exit()/abort() on CUDA failure;
 *   - `*_dev` variants take DEVICE pointers (inputs already resident in HBM) and enqueue
 *     on the library stream without synchronising; host variants copy in, run, copy out;
 *   - plans hold iteration-invariant structure on the device (symbolic factor, patterns).
 *     Host entry points look plans up in a content-addressed cache, so every call stays a
 *     pure function of its arguments (SURVEY.md section 8b "Threading / re-entrancy").
 */
#ifndef SEDUMI_B200_H
#define SEDUMI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int64_t sb_idx;

/* ------------------------------------------------------------------ context */
int         sb200_init(int device);              /* idempotent; selects device, creates stream */
void        sb200_shutdown(void);
const char *sb200_last_error(void);
int         sb200_device_count(void);
int         sb200_sync(void);                     /* cudaStreamSynchronize(library stream) */
void       *sb200_stream(void);                   /* cudaStream_t of the library */
int64_t     sb200_kernel_launches(void);          /* kernels launched by this library so far */
int         sb200_xfer_bytes(int64_t *h2d, int64_t *d2h);   /* bytes this library copied host->device / device->host so far */
/* per-kernel timing with CUDA events on the library stream: begin, run, end -> text report
 * "kernel_name launches total_ms" per line */
int         sb200_prof_begin(void);
int         sb200_prof_end(char *buf, int64_t buflen);
/* CUDA-graph capture of a sequence of *_dev calls on the library stream, and its replay */
int         sb200_graph_begin(void);
int         sb200_graph_end(void **graph_exec);
int         sb200_graph_launch(void *graph_exec);
int         sb200_graph_destroy(void *graph_exec);
int         sb200_dev_alloc(void **p, int64_t bytes);
int         sb200_dev_free(void *p);
int         sb200_h2d(void *dst, const void *src, int64_t bytes);
int         sb200_d2h(void *dst, const void *src, int64_t bytes);

/* ------------------------------------------------------------------ multi-GPU (SURVEY 8e)
 * One process per GPU.  Rank 0 calls sb200_comm_unique_id and hands the 128 bytes to every rank (any host channel);
 * all ranks call sb200_comm_init_rank after sb200_init(device).  The all-reduce is in place, on the library stream,
 * and may be captured into a CUDA graph with the kernels around it.  NCCL (libnccl.so.2) is loaded on first use. */
int sb200_comm_unique_id(void *id128);
int sb200_comm_init_rank(int nranks, int rank, const void *id128);
int sb200_comm_size(void);
int sb200_comm_rank(void);
int sb200_comm_nccl_version(void);
int sb200_comm_stats(int64_t *calls, int64_t *bytes);
int sb200_allreduce_sum_dev(double *buf_dev, int64_t count);
int sb200_allreduce_sum2_dev(double *a_dev, int64_t na, double *b_dev, int64_t nb);
int sb200_comm_destroy(void);

/* ------------------------------------------------------------------ supernodal LDL'
 * blkchol.c:239-440 (mexFunction), blkchol2.c:96-167 (cholonBlk), :346-420 (precorrect),
 * :464-563 (blkLDL); fwblkslv.c:77-134,193-320; bwblkslv.c:73-125,182-298.             */
typedef struct sb200_chol_plan sb200_chol_plan;

/* Symbolic structure: L.L pattern (Ljc/Lir expanded per column, ascending, diagonal
 * first, nested inside supernodes), L.xsuper, L.perm (all 0-based) and the CSC pattern
 * of the matrix X=ADA to be factored (full symmetric pattern). */
int sb200_chol_plan_create(sb200_chol_plan **plan, sb_idx m, sb_idx nsuper,
                           const sb_idx *xsuper, const sb_idx *Ljc, const sb_idx *Lir,
                           const sb_idx *perm, const sb_idx *Xjc, const sb_idx *Xir);
void sb200_chol_plan_destroy(sb200_chol_plan *plan);
sb_idx sb200_chol_plan_nnzL(const sb200_chol_plan *plan);
sb_idx sb200_chol_plan_rect_size(const sb200_chol_plan *plan);   /* doubles in internal layout */

typedef struct {
  double abstol;     /* pars.chol.abstol    (blkchol.c:292-306)  */
  double canceltol;  /* pars.chol.canceltol                        */
  double maxu;       /* pars.chol.maxu                             */
} sb200_chol_pars;

/* Numeric factorisation, device-resident.  Xpr_dev: values of X in its CSC pattern.
 * absd_dev may be NULL (then lb uses diag(X), blkchol.c:374-379).
 * Outputs (device): Lrect_dev  internal rectangular supernode panels (plan_rect_size),
 *                   d_dev[m], flag_dev[m] (0 none,1 skipped,2 diag-add), sval_dev[m]
 *                   (skip: pivot value when skipped; add: amount added). */
int sb200_blkchol_dev(sb200_chol_plan *plan, const double *Xpr_dev, const double *absd_dev,
                      sb200_chol_pars pars, double *Lrect_dev, double *d_dev,
                      int *flag_dev, double *sval_dev);
/* internal panels -> L.L values in the CSC pattern given at plan creation (unit diagonal,
 * skipped columns = e_i, blkchol.c:409-414) */
int sb200_chol_rect_to_csc_dev(sb200_chol_plan *plan, const double *Lrect_dev,
                               const int *flag_dev, double *Lpr_dev);
int sb200_chol_csc_to_rect_dev(sb200_chol_plan *plan, const double *Lpr_dev, double *Lrect_dev);

/* Host-pointer entry = what mex/blkchol.cpp calls.  skip/add index outputs are 0-based,
 * ascending; arrays must have room for m entries. */
int sb200_blkchol(sb_idx m, sb_idx nsuper, const sb_idx *xsuper, const sb_idx *Ljc,
                  const sb_idx *Lir, const sb_idx *perm, const sb_idx *Xjc, const sb_idx *Xir,
                  const double *Xpr, const double *absd, sb200_chol_pars pars,
                  double *Lpr_out, double *d_out, sb_idx *skip_idx, double *skip_val,
                  sb_idx *nskip, sb_idx *add_idx, double *add_val, sb_idx *nadd);

/* y = L \ b(perm,:)  and  y(perm,:) = L' \ b   (dense right-hand sides, m x nrhs).
 * *_dev: Lrect_dev in internal layout; b_dev/y_dev column-major m x nrhs.  */
/* ---- subtree sharding of the factor over ranks (multi-supernode factors; SURVEY 8e).  Supernodes >= t0 form a
 * replicated top, the forest below is dealt to the ranks.  Call order on every rank (all on the library stream):
 *   sb200_blkchol_shard_local_dev ; all-reduce(sum) rect[top_rect_off, +top_rect_len) ; sb200_blkchol_shard_top_dev
 *   sb200_fw_shard_local_dev ; all-reduce(sum) y[top_col0 .. m) per rhs ; sb200_solve_shard_top_dev (in place: ./d and the
 *   backward pass, foreign columns zeroed) ; all-reduce(sum) y ; sb200_bw_shard_finish_dev (back to the original order).
 * d/flag/sval are complete for a rank's own columns and the top; colmask_dev marks the columns a rank answers for. */
int sb200_chol_shard_create(sb200_chol_plan *plan, sb_idx world, sb_idx rank);
int sb200_chol_shard_info(const sb200_chol_plan *plan, sb_idx *t0, sb_idx *top_rect_off, sb_idx *top_rect_len,
                          sb_idx *top_col0, const int **colmask_dev);
int sb200_blkchol_shard_local_dev(sb200_chol_plan *plan, const double *Xpr_dev, const double *absd_dev,
                                  sb200_chol_pars pars, double *Lrect_dev, double *d_dev, int *flag_dev, double *sval_dev);
int sb200_blkchol_shard_top_dev(sb200_chol_plan *plan, sb200_chol_pars pars, double *Lrect_dev, double *d_dev,
                                int *flag_dev, double *sval_dev);
int sb200_fw_shard_local_dev(sb200_chol_plan *plan, const double *Lrect_dev, const double *b_dev, double *y_dev, sb_idx nrhs);
int sb200_solve_shard_top_dev(sb200_chol_plan *plan, const double *Lrect_dev, const double *d_dev, const int *flag_dev,
                              double *y_dev, sb_idx nrhs);
int sb200_bw_shard_finish_dev(sb200_chol_plan *plan, const double *z_dev, double *y_dev, sb_idx nrhs);
/* The same sequences with the collectives issued by the library (sb200_comm_*, below): call on every rank. */
int sb200_blkchol_sharded_dev(sb200_chol_plan *plan, const double *Xpr_dev, const double *absd_dev, sb200_chol_pars pars,
                              double *Lrect_dev, double *d_dev, int *flag_dev, double *sval_dev);
int sb200_ldl_solve_sharded_dev(sb200_chol_plan *plan, const double *Lrect_dev, const double *d_dev, const int *flag_dev,
                                const double *b_dev, double *w_dev, double *y_dev, sb_idx nrhs);
int sb200_fwblkslv_dev(sb200_chol_plan *plan, const double *Lrect_dev, const double *b_dev,
                       double *y_dev, sb_idx nrhs);
int sb200_bwblkslv_dev(sb200_chol_plan *plan, const double *Lrect_dev, const double *b_dev,
                       double *y_dev, sb_idx nrhs);
/* y = L' \ ((L \ b(perm)) ./ d): wrapPcg.m:56-59 for a problem without dense columns; skipped
 * pivots get d=1 like deninfac.m:88-93 when flag_dev is given.  w_dev: m*nrhs scratch. */
int sb200_ldl_solve_dev(sb200_chol_plan *plan, const double *Lrect_dev, const double *d_dev,
                        const int *flag_dev, const double *b_dev, double *w_dev, double *y_dev, sb_idx nrhs);
int sb200_ldl_solve2_dev(sb200_chol_plan *plan, const double *Lrect_dev, const double *d_dev, const int *flag_dev,
                         const double *b_dev, double *w_dev, double *y_dev, sb_idx nrhs, double *ssqr_dev);
int sb200_fwblkslv(sb_idx m, sb_idx nsuper, const sb_idx *xsuper, const sb_idx *Ljc,
                   const sb_idx *Lir, const double *Lpr, const sb_idx *perm,
                   const double *b, double *y, sb_idx nrhs);
int sb200_bwblkslv(sb_idx m, sb_idx nsuper, const sb_idx *xsuper, const sb_idx *Ljc,
                   const sb_idx *Lir, const double *Lpr, const sb_idx *perm,
                   const double *b, double *y, sb_idx nrhs);
/* Sparse right-hand side (fwblkslv.c:150-183): b CSC m x nrhs, y has the pattern
 * (yjc, yir) produced by symbfwblk; only ypr is written.  (bwblkslv's sparse branch,
 * bwblkslv.c:141-172, is never reached from SeDuMi: sparbwslv.m:48 passes full b.) */
int sb200_fwblkslv_sparse(sb_idx m, sb_idx nsuper, const sb_idx *xsuper, const sb_idx *Ljc,
                          const sb_idx *Lir, const double *Lpr, const sb_idx *perm,
                          sb_idx nrhs, const sb_idx *bjc, const sb_idx *bir, const double *bpr,
                          const sb_idx *yjc, const sb_idx *yir, double *ypr);

/* ------------------------------------------------------------------ PSD block algebra
 * invcholfac.c:59-168 (y = invcholfac(u,K[,perm])) and psdscale.m:45-119
 * (y = psdscale(ud,x,K[,transp]); the reference has no MEX for it -- a MEX of that name
 * shadows the .m).  A psd plan depends only on the list of real PSD block orders K.s.   */
typedef struct sb200_psd_plan sb200_psd_plan;
int    sb200_psd_plan_get(sb200_psd_plan **plan, sb_idx nblk, const sb_idx *n);   /* cached */
sb_idx sb200_psd_plan_lenud(const sb200_psd_plan *plan);
sb_idx sb200_psd_plan_sumn(const sb200_psd_plan *plan);
/* perm_dev: int32, 0-based inside each block, concatenated (sum n_k), or NULL */
int sb200_invcholfac_dev(sb200_psd_plan *plan, const double *u_dev, const int *perm_dev, double *y_dev);
int sb200_psdscale_dev(sb200_psd_plan *plan, const double *u_dev, const int *perm_dev,
                       const double *x_dev, int transp, double *y_dev);
/* psdframeit.c:65-99  X_k = Qb' diag(lab_k) Qb ; psdinvjmul.c:101-157  X Z + Z X = 2 Y.
 * frms: per block n x n, column c = Householder vector c (rows c..n-1), last column = beta. */
int sb200_psdframeit_dev(sb200_psd_plan *plan, const double *lab_dev, const double *frms_dev, double *x_dev);
int sb200_psdinvjmul_dev(sb200_psd_plan *plan, const double *xlab_dev, const double *frms_dev,
                         const double *y_dev, double *z_dev);
int sb200_psdframeit(sb_idx nblk, const sb_idx *n, const double *lab, const double *frms, double *x);
int sb200_psdinvjmul(sb_idx nblk, const sb_idx *n, const double *xlab, const double *frms,
                     const double *y, double *z);
/* urotorder.c:312-490 / givensrot.c:93-168.  perm_out 0-based inside each block; gjc_out n_k entries
 * per block (0-based rotation offsets, last = count); g in the worst-case layout n_k(n_k-1) doubles
 * per block for urotorder, packed back to back for givensrot (as the MEX interface carries it). */
/* Device-pointer variants for hosts that keep the scaling state on the GPU.  perm/gjc are int32;
 * g uses the worst-case layout: rotations of block k start at sum_{j<k} n_j(n_j-1) doubles.
 * work_dev: lenud + sum(n) doubles of scratch. */
int sb200_urotorder_dev(sb_idx nblk, const sb_idx *n, const double *u_dev, double maxu, double *u_out_dev,
                        int *perm_dev, int *gjc_dev, double *g_dev, double *work_dev);
int sb200_givensrot_dev(sb_idx nblk, const sb_idx *n, const int *gjc_dev, const double *g_dev,
                        const double *x_dev, double *y_dev);
/* Mixed real / Hermitian blocks (urotorder.c:420-455, givensrot.c:154-163): u = [vec Re; vec Im] for the blocks
 * [nreal, nblk), rotations (Re x, Im x, y).  urotorder_h: g_out in the worst-case layout, block k at
 * sum_{j<k} (real: n_j(n_j-1), Hermitian: 3 n_j(n_j-1)/2) doubles; givensrot_h: g packed as the reference packs it. */
int sb200_urotorder_h(sb_idx nblk, sb_idx nreal, const sb_idx *n, const double *u, double maxu, double *u_out,
                      sb_idx *perm_out, sb_idx *gjc_out, double *g_out);
int sb200_givensrot_h(sb_idx nblk, sb_idx nreal, const sb_idx *n, const sb_idx *gjc, const double *g, sb_idx glen,
                      const double *x, double *y);
int sb200_urotorder(sb_idx nblk, const sb_idx *n, const double *u, double maxu, double *u_out,
                    sb_idx *perm_out, sb_idx *gjc_out, double *g_out);
int sb200_givensrot(sb_idx nblk, const sb_idx *n, const sb_idx *gjc, const double *g, sb_idx glen,
                    const double *x, double *y);
/* host entries: u, x, y are the lenud-long PSD parts; perm 0-based inside each block or NULL */
int sb200_invcholfac(sb_idx nblk, const sb_idx *n, const double *u, const sb_idx *perm, double *y);
/* Mixed real / Hermitian blocks (K.s with K.rsdpN = nreal leading real blocks).  Layout of the reference:
 * a real block is n^2 doubles, a Hermitian block [vec Re; vec Im] = 2 n^2 doubles (invcholfac.c:122-160,
 * psdscale.m:68-118).  The complex algebra runs on the real embedding [[Re,-Im],[Im,Re]] of order 2n. */
int sb200_invcholfac_h(sb_idx nblk, sb_idx nreal, const sb_idx *n, const double *u, const sb_idx *perm, double *y);
int sb200_psdscale_h(sb_idx nblk, sb_idx nreal, const sb_idx *n, const double *u, const sb_idx *perm,
                     const double *x, int transp, double *y);
/* frms of a Hermitian block: [Re c | Im c | beta] = 2 n^2 + n doubles, the last column of c is the complex
 * sign vector (psdframeit.c:80-97, reflect.c:218-262); lab/xlab: sum(n) doubles. */
int sb200_psdframeit_h(sb_idx nblk, sb_idx nreal, const sb_idx *n, const double *lab, const double *frms, double *x);
int sb200_psdinvjmul_h(sb_idx nblk, sb_idx nreal, const sb_idx *n, const double *xlab, const double *frms,
                       const double *y, double *z);
int sb200_psdscale(sb_idx nblk, const sb_idx *n, const double *u, const sb_idx *perm,
                   const double *x, int transp, double *y);

/* ------------------------------------------------------------------ Schur complement ADA'
 * getada1.c:161-261, getada2.c:126-214, getada3.c:370-569.  The plan holds the patterns of
 * At and ADA, the PSD block layout and the per-(constraint, block) work lists.
 *   Ajc1[j]   absolute offset into At.ir of the first PSD nonzero of column j (Ablkjc(:,3));
 *             it is also the end of the LP/Lorentz part of that column
 *   lpN=K.l, nq=|K.q|, qstart[0..nq] = 0-based first norm-bound row of each Lorentz cone (+end)
 *   blkstart[k], blkn[k] = 0-based first row and order of real PSD block k                    */
typedef struct sb200_ada_plan sb200_ada_plan;
int sb200_ada_plan_get(sb200_ada_plan **plan, sb_idx N, sb_idx m, const sb_idx *Ajc, const sb_idx *Air,
                       const sb_idx *Ajc1, sb_idx lpN, sb_idx nq, const sb_idx *qstart, sb_idx nblk,
                       const sb_idx *blkstart, const sb_idx *blkn, const sb_idx *adajc, const sb_idx *adair);
/* With Hermitian PSD blocks (K.rsdpN = nreal < nblk): blocks [nreal, nblk) occupy 2 n^2 rows of At, [Re (lower
 * triangle); Im (strictly lower)] (pretransfo.m:456-480); udsqr holds [vec Re D; vec Im D] for them (spscale.c:332-435). */
int sb200_ada_plan_get_h(sb200_ada_plan **plan, sb_idx N, sb_idx m, const sb_idx *Ajc, const sb_idx *Air,
                         const sb_idx *Ajc1, sb_idx lpN, sb_idx nq, const sb_idx *qstart, sb_idx nblk, sb_idx nreal,
                         const sb_idx *blkstart, const sb_idx *blkn, const sb_idx *adajc, const sb_idx *adair);
sb_idx sb200_ada_plan_nnz(const sb200_ada_plan *plan);
/* sb200_ada_plan_get hands out plans of a bounded cache; a caller that keeps the pointer beyond one call (device-resident
 * chains, captured CUDA graphs) retains it, which exempts it from eviction until the matching release. */
/* Diagnostics (no reference counterpart): the 128-bit content key under which plans and device mirrors of inputs are
 * cached; a pure host function of the bytes (independent of SB200_HASH_THREADS). */
int sb200_content_hash(const void *data, int64_t bytes, uint64_t out[2]);
int sb200_ada_plan_retain(sb200_ada_plan *plan);
/* Diagnostics (no reference counterpart): cycles per phase of the fused getada3 kernel, see ada.cu. enable=1 arms and
 * zeroes the counters, enable=0 copies out[0..7]. */
int sb200_ada_fused_profile(sb200_ada_plan *plan, int enable, unsigned long long *out);
int sb200_ada_plan_release(sb200_ada_plan *plan);
int sb200_ada_set_At_values(sb200_ada_plan *plan, const double *Atpr);
/* device-resident variants: invperm_dev = inverse of the ordering (int32) or NULL = natural */
int sb200_getada1_dev(sb200_ada_plan *plan, const double *dl_dev, const double *ddet_dev,
                      const int *invperm_dev, double *ada_out_dev);
/* getDAtm.m:40-43 on the device: DAt.q = diag(d.q1) A(trace rows,:) + ddot(d.q2, A) into the plan's own
 * CSC (nq x m, pattern fixed by At); sb200_ada_plan_datq returns its device arrays for getada2_dev. */
int sb200_getdatm_dev(sb200_ada_plan *plan, const double *q1_dev, const double *q2_dev);
int sb200_ada_plan_datq(sb200_ada_plan *plan, const long long **jc_dev, const int **ir_dev,
                        const double **pr_dev, sb_idx *nnz);
int sb200_getada2_dev(sb200_ada_plan *plan, const long long *Qjc_dev, const int *Qir_dev,
                      const double *Qpr_dev, const int *invperm_dev, const double *ada_in_dev,
                      double *ada_out_dev);
int sb200_getada3_dev(sb200_ada_plan *plan, const double *udsqr_dev, const int *invperm_dev,
                      sb_idx first, double *ada_dev, double *absd_dev, int symmetrise);
/* host entries; perm = 0-based Aord.lqperm / qperm / sperm (NULL = natural order) */
int sb200_getada1(sb200_ada_plan *plan, const double *Atpr, const sb_idx *perm, const double *dl,
                  const double *ddet, double *ada_out);
int sb200_getada2(sb200_ada_plan *plan, sb_idx nq, const sb_idx *Qjc, const sb_idx *Qir, const double *Qpr,
                  const sb_idx *perm, const double *ada_in, double *ada_out);
int sb200_getada3(sb200_ada_plan *plan, const double *Atpr, const double *udsqr, sb_idx lenud,
                  const sb_idx *perm, sb_idx first, const double *ada_in, double *ada_out, double *absd_out);

/* ------------------------------------------------------------------ search direction (SURVEY 8f row 1)
 * The direct step of wrapPcg.m:42-97 on device-resident data, LP + PSD cones without dense columns:
 *   dx = D'rv ; r = A dx + rb ; p = L'\((L\r)./d) ; x = vecsym(At p) ; alpha = (p'(p./d)) / |D x|^2 ;
 *   y = alpha p ; dx = rv - alpha D x ; r = A D'dx + rb ; normr = |r|_inf      (Amul.m:42-56, vecsym.c, psdscale.m).
 * rv_dev: N = K.l + sum(K.s.^2) doubles; rb_dev: m doubles or NULL; outputs y (m), dx (N), r (m);
 * scal_dev[0..3] = ssqrNew, ssqrdx, alpha, normr (device); work_dev: 3 N + 2 m + 600 doubles.  Nothing synchronises. */
int sb200_wrappcg_dev(sb200_ada_plan *ada, sb200_psd_plan *psd, sb200_chol_plan *chol, const double *dl_dev,
                      const double *u_dev, const int *perm_dev, const double *Lrect_dev, const double *Ld_dev,
                      const int *flag_dev, const double *rv_dev, const double *rb_dev, double *y_dev, double *dx_dev,
                      double *r_dev, double *scal_dev, double *work_dev);
/* The whole of wrapPcg.m:43-130 with loopPcg.m:53-170 (PopK.m:39-55, asmDxq.m:41-69, Amul.m:40-56 with LP dense
 * columns): the direct step above, then PCG refinement while |r|_inf >= y0 * cgpars.restol.  Cones LP, Lorentz and
 * real PSD; x layout [K.l | nq trace entries | norm-bound parts (qdim) | PSD], so N = K.l + sum(K.q) + sum(K.s.^2).
 *   dpr1: the product-form factor of the LP dense columns (after sb200_dpr1fact_dev), NULL without dense columns;
 *         Ld_dev is then the d that dpr1fact returned (deninfac.m), otherwise L.d.
 *   cones->q1/q2 also refresh the plan's DAt.q (sb200_getdatm_dev), used by the residual update of every CG step.
 *   Outputs y (m), dx (N), r (m) and *status: k = CG steps counted as wrapPcg counts them (0 when |D A' p| = 0, with
 *   y = 0 and dx = rv), stop = STOP of the last loopPcg call (0: none ran), trials = refinement trials, normr = |r|_inf.
 * The host side of the loop reads a few bytes back after the direct step and after every CG step (one synchronisation
 * when the direct step already meets the tolerance), so the entry refuses to run while the library stream is being
 * captured.  Dense Lorentz blocks are refused.  work_dev: sb200_wrappcg_full_work(N, m, nq, qdim) doubles. */
typedef struct sb200_dpr1_plan sb200_dpr1_plan;     /* dense columns, see below */
typedef struct {
  double restol, stagtol;      /* cgpars.restol, cgpars.stagtol (checkpars.m:171-191: 5e-3, 5e-14) */
  int maxiter, refine, qprec;  /* cgpars.maxiter, .refine, .qprec (49, 1, 1) */
} sb200_cgpars;
typedef struct {
  sb_idx nq, qdim;             /* Lorentz cones, sum(K.q - 1) */
  const long long *qbs_dev;    /* nq + 1 norm-bound block starts relative to the first norm-bound entry */
  const double *det_dev, *q1_dev, *q2_dev, *auxdet_dev, *auxtr_dev;    /* d.det, d.q1, d.q2, d.auxdet, d.auxtr */
  sb_idx nden;                 /* LP dense columns (dense.l) */
  const int *den_cols_dev;     /* their 0-based positions in x (dense.cols - 1) */
  const double *denA_dev;      /* dense.A, column-major m x nden */
  sb_idx ndenq;                /* dense Lorentz blocks (dense.q): must be 0 */
} sb200_pcg_cones;
typedef struct { sb_idx k; int stop; int trials; double normr; } sb200_pcg_status;
sb_idx sb200_wrappcg_full_work(sb_idx N, sb_idx m, sb_idx nq, sb_idx qdim);
int sb200_wrappcg_full_dev(sb200_ada_plan *ada, sb200_psd_plan *psd, sb200_chol_plan *chol, sb200_dpr1_plan *dpr1,
                           const sb200_pcg_cones *cones, const sb200_cgpars *cgpars, const double *dl_dev,
                           const double *u_dev, const int *perm_dev, const double *Lrect_dev, const double *Ld_dev,
                           const int *flag_dev, const double *rv_dev, const double *rb_dev, double y0, double *y_dev,
                           double *dx_dev, double *r_dev, sb200_pcg_status *status, double *work_dev);
int sb200_ada_plan_csr(sb200_ada_plan *plan, const long long **Ajc, const int **Air, const double **Apr,
                       const long long **rowptr, const int **rowcol, const int **rowsrc, sb_idx *N, sb_idx *m,
                       sb_idx *lpN, sb_idx *nq);
int sb200_psd_plan_blocks(sb200_psd_plan *plan, const int **n_dev, const long long **off_dev, int *nblk, int *maxn);

/* ------------------------------------------------------------------ PSD algebra of the scaling update (SURVEY 8f row 2)
 * vecsym.c:139-175, sqrtinv.c:86-148, qrK.c:239-297.  x/y/q/r are the lenud-long PSD parts; blocks [nreal, nblk) Hermitian. */
int sb200_vecsym(sb_idx nblk, sb_idx nreal, const sb_idx *n, const double *x, double *y);
int sb200_sqrtinv(sb_idx nblk, sb_idx nreal, const sb_idx *n, const double *q, const double *v, double *y);
int sb200_qrK(sb_idx nblk, const sb_idx *n, const double *x, double *q, double *r);      /* real blocks */
/* M-only in the reference (the plugins shadow the .m files); real blocks.  psdmul: mode 0 = psdjmul.m:38-74, mode 1 =
 * triumtriu.m:38-73; psdfactor.m:37-82 (*ispos = 0: not positive definite); psdinvscale.m:37-83. */
int sb200_psdmul(int mode, sb_idx nblk, const sb_idx *n, const double *x, const double *y, double *z);
int sb200_psdfactor(sb_idx nblk, const sb_idx *n, const double *x, double *ux, int *ispos);
/* [lab,q] = psdeig(x,K) (psdeig.m:40-96; minpsdeig.m:43-68 takes the minimum of lab): eigenvalues of (X_k + X_k')/2 per real
 * PSD block in ascending order, q (NULL: not wanted) the eigenvectors.  The reference defers to the host's eig(); this is a
 * cyclic Jacobi method on the device (vectors agree up to sign / rotation inside eigenspaces). */
int sb200_psdeig(sb_idx nblk, const sb_idx *n, const double *x, double *lab, double *q);
int sb200_psdinvscale(sb_idx nblk, const sb_idx *n, const double *u, const double *x, double *y);

/* ------------------------------------------------------------------ Lorentz streams
 * ddot.c:165-308, qblkmul.c:57-116, quadadd.c:89-130.
 * Dense ddot / qblkmul: bs[0..nblk] are block starts relative to the first norm-bound row. */
int sb200_ddot_dense_dev(sb_idx nblk, const long long *bs_dev, const double *d_dev, const double *X_dev,
                         sb_idx ldx, sb_idx ncol, double *y_dev);
int sb200_qblkmul_dev(sb_idx nblk, const long long *bs_dev, sb_idx qdim, const double *mu_dev,
                      const double *d_dev, double *y_dev);
int sb200_quadadd_dev(sb_idx n, const double *xhi, const double *xlo, const double *y, double *zhi, double *zlo);
int sb200_ddot_dense(sb_idx nblk, const sb_idx *bs, const double *d, const double *X, sb_idx ldx,
                     sb_idx ncol, double *y);
int sb200_ddot_sparse(sb_idx nblk, const sb_idx *bs_abs, const double *d, sb_idx m, const sb_idx *xlo,
                      const sb_idx *xhi, const sb_idx *xir, const double *xpr, sb_idx *yjc, sb_idx *yir,
                      double *ypr, sb_idx *nnz_out);
int sb200_qblkmul(sb_idx nblk, const sb_idx *bs, const double *mu, const double *d, double *y);
/* adendotd.c:134-245: Ad(:,k) on the pattern of Ablk for the nq dense Lorentz blocks */
int sb200_adendotd(sb_idx m, sb_idx nq, sb_idx nden, const sb_idx *adjc, const sb_idx *adir, const sb_idx *sjc,
                   const sb_idx *sir, const double *spr, const sb_idx *ajc, const sb_idx *air, const double *apr,
                   const double *d1q, const sb_idx *colbeg, const double *d2c, double *adpr);
int sb200_quadadd(sb_idx n, const double *xhi, const double *xlo, const double *y, double *zhi, double *zlo);

/* ------------------------------------------------------------------ dense columns (product form)
 * dpr1fact.c:630-848, fwdpr1.c:99-202, bwdpr1.c:171-275.  Index arrays 0-based; betajc_out 0-based
 * (the stub adds 1 like the reference), pivperm 0-based ("C-form" in the reference too).          */
int sb200_dpr1fact(sb_idx m, sb_idx n, const sb_idx *xjc, const sb_idx *xir, const double *xpr, const double *d_in,
                   const sb_idx *dzjc, const sb_idx *dzir, const sb_idx *colperm, const sb_idx *firstpiv,
                   const double *smult, double maxu, double *p_out, double *beta_out, sb_idx *betajc_out,
                   sb_idx *pivperm_out, double *dopiv_out, double *d_out, sb_idx *nbeta, sb_idx *npivperm);
int sb200_dpr1solve(int backward, sb_idx m, sb_idx nrhs, sb_idx nden, const sb_idx *dzjc, const sb_idx *dzir,
                    const double *p, const sb_idx *pivperm, sb_idx permnnz, const double *beta,
                    const sb_idx *betajc, const double *dopiv, double *y);

/* device-resident product form: plan from Lsymb (dz, perm, first; 0-based), factor from the dense block L\Ad (m x n,
 * column-major, rows in the factor's permuted order) and L.d, then in-place solves on m x nrhs device data */
int  sb200_dpr1_plan_create(sb200_dpr1_plan **plan, sb_idx m, sb_idx n, const sb_idx *dzjc, const sb_idx *dzir,
                            const sb_idx *colperm, const sb_idx *firstpiv);
void sb200_dpr1_plan_destroy(sb200_dpr1_plan *plan);
int  sb200_dpr1fact_dev(sb200_dpr1_plan *plan, const double *LAD_dev, const double *smult_dev, double maxu,
                        const double *d_in_dev, double *d_out_dev);
int  sb200_dpr1solve_dev(sb200_dpr1_plan *plan, int backward, double *y_dev, sb_idx nrhs);
int  sb200_gather_dev(sb_idx n, const int *idx_dev, const double *src_dev, double *dst_dev);
int  sb200_scale_by_d_dev(sb_idx m, sb_idx nrhs, const double *d_dev, const int *flag_dev, const double *lb_dev, double *y_dev);
const double *sb200_chol_plan_lb_dev(const sb200_chol_plan *plan);   /* lb_k = max(abstol, canceltol*absd(perm_k)) of the last factorisation */
int  sb200_dpr1_plan_download(sb200_dpr1_plan *plan, double *p, double *beta, int *betajc, int *pivperm, int *ordered);

#ifdef __cplusplus
}
#endif
#endif /* SEDUMI_B200_H */
