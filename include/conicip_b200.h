/*
 * conicip_b200.h -- C ABI of the B200-native KKT engine for ConicIP.jl.
 *
 * This is the drop-in boundary.  Julia (`ccall`), Python (`ctypes`) or C bind
 * exactly these symbols.  Every entry point cites the reference interface it
 * replaces (paths relative to the ConicIP.jl v0.2.0 tree).
 *
 * Conventions
 *   - All matrices passed in are column-major FP64 (Julia `Matrix{Float64}`).
 *   - Every `double*` vector/matrix argument may be a HOST or a DEVICE pointer
 *     (resolved with cudaPointerGetAttributes); host buffers are staged through
 *     pinned memory on the handle's stream.  Outputs are complete when the call
 *     returns (the call synchronises the handle's stream iff an output is in
 *     host memory).
 *   - Inputs are never written (src/ConicIP.jl:901,916 alias r0 into every RHS).
 *   - Return value: 0 = ok; >0 = numerical failure (1-based index of the first
 *     non-positive Cholesky pivot); <0 = CUDA / NCCL / argument error, message
 *     available from cip_last_error().
 *   - Calls on one handle must not overlap (the reference protocol is strictly
 *     sequential, src/ConicIP.jl:667-934).
 *   - There is no CPU fallback anywhere behind this ABI.
 */
#ifndef CONICIP_B200_H
#define CONICIP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cip_engine* cip_handle;

/* cone_type codes == the reference's cone strings (src/ConicIP.jl:519-522) */
#define CIP_CONE_R 0 /* "R" nonnegative orthant */
#define CIP_CONE_Q 1 /* "Q" second-order cone   */
#define CIP_CONE_S 2 /* "S" PSD cone, svec of order k => dim k(k+1)/2 */

/* scaling-block kinds == the Julia block types a `Block` may hold
 * (src/blockmatrices.jl:13-15; docs/src/guides/kkt_solvers.md:22-27) */
#define CIP_BLK_DIAG     0 /* Diagonal{Float64}: fa[] = .diag                           */
#define CIP_BLK_WOODBURY 1 /* SymWoodbury: fa[] = .A.diag, fb[] = .B (vector), fD = .D   */
#define CIP_BLK_VECCONG  2 /* VecCongurance: fR = .R (k*k column-major per S cone)       */

/* which operator cip_apply applies (src/ConicIP.jl:687,689,735,893-894,910-911) */
#define CIP_OP_F      0 /* F*x     */
#define CIP_OP_FT     1 /* F'*x    */
#define CIP_OP_FINVT  2 /* inv(F)'*x  (the reference's F^-T argument) */
#define CIP_OP_FINV   3 /* inv(F)*x   (src/kktsolvers.jl:48)          */

typedef struct cip_options {
  int    struct_size;   /* = sizeof(cip_options), for ABI evolution                       */
  int    device;        /* CUDA ordinal; -1 = current device                              */
  double reg_delta;     /* static regularisation H + delta*I before Cholesky (default 0)  */
  double reg_eps_G;     /* regularisation of the Schur complement S (default 0)           */
  int    q_kind;        /* 0 dense n*n (ldq), 1 diagonal (Q points to n doubles), 2 zero  */
  int    verbose;
  int    dist_chol;     /* sharded handles: 0 replicated Cholesky, 1 block-cyclic distributed, -1 auto */
  double aug_rho;       /* equality block: factor H + rho*G'G (and add rho*G'rw to the rhs) so that H may be
                           singular on range(G') as kktsolver_qr allows (src/kktsolvers.jl:35); same solution.
                           < 0: auto (1.0 when p > 0), 0: off */
  int    ngpus;         /* single-process multi-GPU (SURVEY 8b "Threading", 8e): > 1 slices the rows of A on cone
                           boundaries over the devices device .. device+ngpus-1 (0 .. ngpus-1 when device < 0), one
                           stream and one NCCL communicator per device (ncclCommInitAll), all driven from the
                           calling thread's single call -- the reference calls its kktsolver once from one process
                           (src/ConicIP.jl:667), so this is what `kktsolver = kktsolver_b200(ngpus = 8)` uses.
                           Every entry point below then takes and returns GLOBAL vectors; 0 / 1 = one device */
  int    fold_scaling;  /* K = R^m only (every block of F diagonal): apply W^-2 to the operand fragments inside the
                           SYRK instead of materialising Atil = F^-T A (src/kktsolvers.jl:33) -- halves the resident
                           bytes (no second copy of A), costs ~1.5 % of the SYRK.  0: auto (fold when the second copy
                           would not fit in free device memory), 1: always, 2: never */
  int    row_structure; /* single-device handles: 1 = classify the rows of A at LEVEL 1 and exploit them when forming
                           H (the reference keeps A sparse through this product, src/kktsolvers.jl:289-290).  R rows
                           with one non-zero go straight onto the diagonal of H; the other rows ("rest": every Q / S
                           row and the R rows with >= 2 non-zeros) are kept in a compact copy of A that spans only
                           the columns they touch, and the constant Q + rho*G'G is formed once.  0 = off (default).
                           The environment variable CIP_ROW_STRUCTURE=1 turns it on for single-device handles.
                           2 = the same row split, and the columns of H split too: K ("coupled") holds the columns
                           a rest row touches, the columns where Q has an off-diagonal non-zero in the row or the
                           column, and (resolved aug_rho > 0 and p > 0) the columns where G has a non-zero; D holds
                           the others, where H has nothing but its diagonal.  H_KK is factored densely, D as
                           sqrt(H_jj), the Schur complement gets G_D diag(1/H_jj) G_D' + Z_K Z_K'.  No n_pad x n_pad
                           buffer remains after cip_create, so problems whose coupled columns are few can be solved
                           at any n that fits the vectors, G and the rest rows of A (dense Q input still passes
                           through one transient n_pad x n_pad staging copy; give Q as CSC, diagonal or NULL to
                           avoid it).  cip_get_H scatters into n x n (zeros outside K x K and the diagonal); a
                           failing pivot is still reported as 1 + its global column.  CIP_ROW_STRUCTURE=2 selects it.
                           Sharded handles (ngpus > 1, cip_comm_init) reject 1 and 2. */
} cip_options;

typedef struct cip_stats_t {
  int    n, m, p, n_pad, m_pad, p_pad;
  long long factors, solves;            /* LEVEL-2 / LEVEL-3 call counts                  */
  double ms_scale, ms_syrk, ms_allreduce, ms_chol, ms_schur, ms_solve; /* last call, CUDA events */
  double syrk_flops;                    /* algorithmic m*n^2 of the last SYRK (local rows) */
  double chol_flops;                    /* n^3/3                                           */
  size_t device_bytes;                  /* bytes held by this handle (all devices of a multi-GPU handle) */
  long long kernel_launches;            /* kernels launched by this library so far         */
} cip_stats_t;

const char* cip_last_error(void);
int cip_version(void);

/* ---------------------------------------------------------------- LEVEL 1
 * replaces `solve3x3gen = kktsolver(Q,A,G,cone_dims)`  (src/ConicIP.jl:667;
 * kktsolver_qr src/kktsolvers.jl:18-28; kktsolver_2x2 :281-285).
 * Uploads Q (n*n), A (m*n: THIS RANK'S rows when sharded) and G (p*n) once and
 * re-lays them out for the kernels.  cone_type/cone_dim describe the rows of A
 * (sum(cone_dim) == m). */
int cip_create(cip_handle* out, int n, int m, int p,
               const double* Q, int ldq,
               const double* A, int lda,
               const double* G, int ldg,
               int ncones, const int* cone_type, const int* cone_dim,
               const cip_options* opts);
/* LEVEL 1 from sparse inputs (SURVEY 8f rank 2): Julia's `SparseMatrixCSC{Float64,Int64}` fields
 * (.colptr, .rowval, .nzval; index_base = 1) are passed as they are -- `A`, `G` and `Q` reach conicIP
 * sparse from the MOI wrapper (src/MOI_wrapper.jl:152-275) and from the README example -- and are
 * expanded into the device layout by a scatter kernel, with no dense copy on the host.
 * Q == NULL means Q = 0; G == NULL or G->nrows == 0 means no equality block. */
typedef struct cip_csc {
  int nrows, ncols;
  const int64_t* colptr;   /* ncols + 1 */
  const int64_t* rowval;   /* nnz */
  const double*  nzval;    /* nnz */
  int index_base;          /* 1 for Julia, 0 for C / SciPy */
} cip_csc;
int cip_create_csc(cip_handle* out, int n, const cip_csc* Q, const cip_csc* A, const cip_csc* G,
                   int ncones, const int* cone_type, const int* cone_dim, const cip_options* opts);
int cip_destroy(cip_handle h);

/* Row-sharded multi-GPU across PROCESSES (SURVEY 8e; no counterpart in the reference; the
 * single-process form is cip_options.ngpus): one
 * process per GPU, each created with its own row slab of A.  The 128-byte NCCL
 * unique id is produced on rank 0 and distributed by the host (torch.distributed,
 * MPI, Julia Distributed ...).  After this call cip_factor all-reduces the
 * partial Gram matrices and cip_solve all-reduces A'*(W^-2 v). */
/* How a handle with opts.ngpus = N slices the rows of A (pure host logic, no device needed): contiguous
 * cone-aligned slabs of near-equal size; R cones may be cut anywhere (W is diagonal there), Q / S cones never.
 * row_lo / row_hi [ngpus] out: shard r owns the global rows [row_lo[r], row_hi[r]).  Returns 0 or -1. */
int cip_shard_plan(int ncones, const int* cone_type, const int* cone_dim, int ngpus, int* row_lo, int* row_hi);
int cip_nccl_unique_id(unsigned char id_out[128]);
int cip_comm_init(cip_handle h, int nranks, int rank, const unsigned char id[128]);

/* ---------------------------------------------------------------- LEVEL 2
 * replaces `solve3x3 = solve3x3gen(F, F^-T)`  (src/ConicIP.jl:682;
 * src/kktsolvers.jl:30-35 and :287-295,:320-322): builds
 * H = Q + (F^-T A)'(F^-T A), factors it (Cholesky) and eliminates G.
 * F arrives flattened: kind[ncones]; fa[m] / fb[m] concatenated over cones;
 * fD[ncones]; fR = concatenated k*k column-major R of every VECCONG block
 * (NULL if none).  The initial call passes DIAG blocks of ones for every cone,
 * including Q/S slots (src/ConicIP.jl:704). */
int cip_factor(cip_handle h, const int* kind,
               const double* fa, const double* fb, const double* fD, const double* fR);

/* Device-resident variant: compute the Nesterov-Todd scaling of (v,s) on the
 * GPU (`nt_scaling`, src/ConicIP.jl:589-605,:732-735), keep it as the current
 * F, write lambda = F*v, then do exactly what cip_factor does. */
int cip_factor_from_point(cip_handle h, const double* v, const double* s, double* lambda_out);

/* ---------------------------------------------------------------- LEVEL 3
 * replaces `(a,b,c) = solve3x3(x,y,z)`  (src/ConicIP.jl:688;
 * src/kktsolvers.jl:324-332 with :297-302): solves
 *   Q a + G' b - A' c = ry ;  G a = rw ;  A a + F'F c = rv
 * for the current factorisation.  Outputs are freshly written (never alias
 * inputs).  dw may be NULL when p == 0. */
int cip_solve(cip_handle h, const double* ry, const double* rw, const double* rv,
              double* dy, double* dw, double* dv);

/* Several right-hand sides through the current factorisation (BASELINE north_star: "forward/back triangular solves
 * for the predictor and corrector right-hand sides together"; the reference solves them one `solve3x3` call at a
 * time, src/ConicIP.jl:688,:879,:907,:919 through src/kktsolvers.jl:297-302,:324-332).  Column k of every argument
 * lies at ptr + k*ld (ldy >= n, ldw >= p, ldv >= m); column k of the result equals cip_solve on column k.  The
 * two products with A are shared by pairs of columns (A is streamed once per pair), the rest runs per column.
 * In conicIP itself the corrector's right-hand side depends on the predictor's solution (src/ConicIP.jl:879-907),
 * so the stock loop cannot batch them; callers with independent right-hand sides can. */
int cip_solve_multi(cip_handle h, int nrhs, const double* ry, int ldy, const double* rw, int ldw,
                    const double* rv, int ldv, double* dy, double* dw, double* dv);

/* ---------------------------------------------------------------- cone kernels
 * The reference has no callback for these (closures over private functions,
 * src/ConicIP.jl:571-665); they are exported so the host driver can keep all
 * m-vectors on the device. */
/* nt_scaling (src/ConicIP.jl:589-605; nestod_soc :165-194; nestod_sdc :196-210) */
int cip_nt_scaling(cip_handle h, const double* v, const double* s, double* lambda_out);
/* read back the current F in the flattened format of cip_factor */
int cip_get_scaling(cip_handle h, int* kind, double* fa, double* fb, double* fD, double* fR);
/* set the current F without factoring (flattened format of cip_factor) */
int cip_set_scaling(cip_handle h, const int* kind,
                    const double* fa, const double* fb, const double* fD, const double* fR);
/* Block mat-vec (src/blockmatrices.jl:107-118,176-177; VecCongurance*x src/ConicIP.jl:69) */
int cip_apply(cip_handle h, int op, const double* x, double* y);
/* maxstep (src/ConicIP.jl:571-587; maxstep_rp :212-240, maxstep_soc :242-270,
 * maxstep_sdc :272-303).  d == NULL selects the `nothing` (shift into cone) variant.
 * d_scale divides d first (the reference calls maxstep(z.v, dz.v/(1-DTB)), :927). */
int cip_maxstep(cip_handle h, const double* x, const double* d, double d_scale, double* alpha_out);
/* cone_prod! / cone_div!  (src/ConicIP.jl:622-665, :305-360):
 * prod: o = x o y ;  div: o = y^-1 o x  (argument order of the reference). */
int cip_cone_prod(cip_handle h, const double* x, const double* y, double* o);
int cip_cone_div(cip_handle h, const double* x, const double* y, double* o);

/* ---------------------------------------------------------------- resident operators
 * Residual mat-vecs on the matrices uploaded at LEVEL 1 (src/ConicIP.jl:747-750,
 * :810,:839-841,:912-914).  trans=0: y = M x ; trans=1: y = M' x.  For a sharded
 * handle A is this rank's slab (A'x results are all-reduced across ranks). */
int cip_mul_A(cip_handle h, int trans, const double* x, double* y);
int cip_mul_G(cip_handle h, int trans, const double* x, double* y);
int cip_mul_Q(cip_handle h, const double* x, double* y);

/* ---------------------------------------------------------------- device-resident IP loop
 * SURVEY 8f rank 1 (no counterpart in the reference, whose loop runs in Julia): the whole of
 * `conicIP` (src/ConicIP.jl:468-939: initial point :704-713, NT scaling, predictor :879-887,
 * corrector :893-901, refinement :909-921, step :927-932, stopping / infeasibility tests
 * :763-873) on device-resident vectors behind one call.  c (n), b (m: this rank's rows when
 * sharded), d (p) in; y (n), w (p), v (m) out; host or device pointers. */
#define CIP_STATUS_NONE       0
#define CIP_STATUS_OPTIMAL    1
#define CIP_STATUS_INFEASIBLE 2
#define CIP_STATUS_UNBOUNDED  3
#define CIP_STATUS_ABANDONED  4
#define CIP_STATUS_ERROR      5
typedef struct cip_ipm_options {
  int    struct_size;
  int    maxIters;              /* 100  (src/ConicIP.jl:504) */
  int    maxRefinementSteps;    /* 3    (:503) */
  int    verbose;
  double optTol;                /* 1e-6 (:500) */
  double DTB;                   /* 0.01 (:501) */
  double infeasTol;             /* < 0: = optTol (:506) */
  double refinementThreshold;   /* < 0: = optTol/1e7 (:509) */
} cip_ipm_options;
typedef struct cip_ipm_result {
  int    status, Iter, factors, solves;
  double Mu, prFeas, duFeas, muFeas, pobj, dobj, seconds;
} cip_ipm_result;
int cip_ipm_solve(cip_handle h, const double* c, const double* b, const double* d,
                  const cip_ipm_options* opts, double* y, double* w, double* v, cip_ipm_result* result);

/* ---------------------------------------------------------------- introspection */
int cip_stats(cip_handle h, cip_stats_t* out);
/* How a handle with cip_options.row_structure = 1 split the rows of A (all zero when the option is off). */
typedef struct cip_structure_t {
  int struct_size;      /* = sizeof(cip_structure_t), set by the caller                                */
  int enabled;          /* 1: the structured path runs                                                  */
  int singleton_rows;   /* R rows with exactly one non-zero: added to the diagonal of H                 */
  int empty_rows;       /* R rows without a non-zero                                                    */
  int rest_rows;        /* Q / S rows plus R rows with >= 2 non-zeros: the rows of the SYRK             */
  int rest_cols;        /* |J|: the columns the rest rows touch                                         */
  int compressed;       /* 1: the SYRK runs on the columns J only (round_up(|J|,128) <= n_pad/2; always
                           with row_structure = 2)                                                      */
  int base_has_gtg;     /* 1: the constant part Q + rho*G'G was formed once at creation                 */
} cip_structure_t;
int cip_structure_info(cip_handle h, cip_structure_t* out);
/* How a handle with cip_options.row_structure = 2 split the columns of H (all zero otherwise).  The three
 * cols_from_* counts are of overlapping sets: a column can be coupled for more than one reason. */
typedef struct cip_split_t {
  int struct_size;      /* = sizeof(cip_split_t), set by the caller                                      */
  int enabled;          /* 1: H is factored as a diagonal part plus its coupled block                      */
  int coupled_cols;     /* |K|: columns of the dense block H_KK                                            */
  int diagonal_cols;    /* |D| = n - |K|: columns where H holds only its diagonal                          */
  int cols_from_rest;   /* columns touched by a rest row of A (|J| of cip_structure_t)                     */
  int cols_from_Q;      /* columns with an off-diagonal non-zero of Q in their row or column               */
  int cols_from_G;      /* columns where G has a non-zero, when aug_rho > 0 and p > 0 (else 0)             */
} cip_split_t;
int cip_split_info(cip_handle h, cip_split_t* out);
/* copy the current reduced matrix H (after cip_factor: its Cholesky factor L in the
 * lower triangle) into a column-major n*n buffer -- test/debug hook */
int cip_get_H(cip_handle h, double* out, int ldo);
/* form H = Q + (F^-T A)'(F^-T A) only (no factorisation) -- test/bench hook */
int cip_form_H(cip_handle h);
int cip_factor_H(cip_handle h);
/* x = inv(H) rhs with the current Cholesky factor: the two triangular sweeps of LEVEL 3 alone
 * (src/kktsolvers.jl:299 without the pivot algebra around it) -- test/bench hook; n-vectors */
int cip_solve_H(cip_handle h, const double* rhs, double* x);
int cip_sync(cip_handle h);
/* The handle launches everything on one CUDA stream (its own by default).  cip_set_stream
 * makes it use the caller's stream instead (e.g. PyTorch's current stream; the value 0 is the
 * legacy default stream), so device-pointer arguments produced on that stream need no
 * extra synchronisation. */
void* cip_stream(cip_handle h);
int cip_set_stream(cip_handle h, void* stream);
/* FP64 pipe ceilings measured on this device: DMMA.8x8x4 and DFMA register-only loops */
int cip_measure_fp64_peaks(int device, double* dmma_tflops, double* dfma_tflops);

/* ---------------------------------------------------------------- preprocessor (SURVEY §8f rank 4)
 * Replaces imcols(A, b, eps) -- src/preprocessor.jl:10-28, called twice by preprocess_conicIP (:58-59) on
 * (G, d) and on ([Q A' G[IP,:]'], c): a maximal set of linearly independent rows of the p x n matrix A
 * (rows whose pivot |R_kk| / ||A||_F exceeds eps in a row-pivoted QR of A') and the consistency of
 * A x = b on the dropped rows (norm(A (A[R,:] \ b[R]) - b, Inf) / ||A||_F < eps).
 *   A     column-major, leading dimension lda >= p; host or device pointer.  b likewise, length p.
 *   keep  [p] out: 1 for the rows of the independent set, 0 for redundant ones;  *nkeep = their number
 *   *consistent  out: 1 / 0.   (The reference returns an empty set when inconsistent; the caller decides.)
 * No handle: it runs before cip_create on the device given (-1 = current).  Returns 0, or <0 on error. */
int cip_imcols(int device, const double* A, int lda, int p, int n, const double* b, double eps, int* keep,
               int* nkeep, int* consistent);

#ifdef __cplusplus
}
#endif
#endif /* CONICIP_B200_H */
