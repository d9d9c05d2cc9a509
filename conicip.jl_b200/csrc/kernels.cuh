// Host-callable launchers for the bandwidth-bound kernels (layout, mat-vec, cone, Cholesky
// panel, triangular sweeps).  All take an explicit stream and return 0 / -1.
#pragma once
#include "common.cuh"
#include "gemm_nt.cuh"

namespace cip {

// ---------------------------------------------------------------- layout (layout.cu)
// dst[q4(r,k)] = (r<R && k<K) ? src[r + k*lds] : 0   for r < Rpad, k < Kpad   (Q, G: rows stay rows)
int pack_rows_q4(double* dst, int ld, const double* src, int lds, int R, int K, int Rpad, int Kpad,
                 cudaStream_t s);
// dst[q4(r0+r,k)] = k<K ? src[k + r*lds] : 0   for r < nc, k < Kpad   (A: columns of A become rows;
// src is a chunk of nc columns of the column-major A, so uploads can be chunked)
int pack_trans_q4(double* dst, int ld, int r0, const double* src, int lds, int K, int Kpad, int nc,
                  cudaStream_t s);
int unpack_rows_q4(double* dst, int ldd, const double* src, int ld, int R, int K, cudaStream_t s);
int add_diag_q4(double* X, int ld, int from, int to, double val, int set, cudaStream_t s);
int set_diag_vec_q4(double* X, int ld, int n, const double* v, cudaStream_t s);
// device CSC arrays (colptr[ncols+1], rowval/nzval[nnz], index base 0 or 1) scattered into a zeroed Q4 matrix
// Entries whose row index falls outside [0, nrows) are skipped and flagged: *bad = 1 + column (first one wins).
int scatter_csc_q4(double* dst, int ld, int ncols, const long long* colptr, const long long* rowval,
                   const double* nzval, int base, int transpose, int nrows, long long nnz, int* bad,
                   cudaStream_t s);
// dst[q4(j, k0 + i)] = scale * src[q4(i, j)]  for i < R, j < K   (G -> the augmentation rows of Atil)
int transpose_scale_q4(double* dst, int ldd, int k0, const double* src, int lds, int R, int K, double scale,
                       cudaStream_t s);
int fill_zero(double* p, size_t n, cudaStream_t s);

// ---------------------------------------------------------------- mat-vec on Q4 (matvec.cu)
// out[r] (+)= sum_k X[r,k] v[k]   (thread per row; deterministic two-pass over k splits)
// v must be readable and finite up to round_up(K,4).
// `add` (optional, R doubles) is added in the second pass: out = add + X v
int q4_mv_rows(double* out, const double* X, int ld, int R, int K, const double* v, double* partial,
               int partial_capacity, cudaStream_t s, const double* add = nullptr);
// out[k] = sum_r X[r,k] u[r]      (warp per k-quad)
int q4_mv_k(double* out, const double* X, int ld, int R, int K, const double* u, cudaStream_t s);
// two vectors per pass over X (cip_solve_multi): X is read once; per vector the result equals the one-vector call
int q4_mv_rows2(double* outa, double* outb, const double* X, int ld, int R, int K, const double* va, const double* vb,
                double* partial, int partial_capacity, cudaStream_t s, const double* adda = nullptr,
                const double* addb = nullptr);
int q4_mv_k2(double* outa, double* outb, const double* X, int ld, int R, int K, const double* ua, const double* ub,
             cudaStream_t s);

// ---------------------------------------------------------------- cone kernels (cones.cu)
struct ConeDesc {
  int m, ncones;
  const int* type;      // [ncones] CIP_CONE_*
  const int* off;       // [ncones+1]
  const int* row_cone;  // [m] cone index per row
  const int* qlist;     // [nq] indices of Q cones
  int nq;
  const int* slist;     // [ns] indices of S cones
  int ns;
  int max_q_dim;
  int nr_rows;        // rows that belong to R cones
  int max_s_ord;
  const int* sord;      // [ns] matrix order k of every S cone (slist order)
  const int* roff;      // [ns] offset (in doubles) of its k*k block inside Scaling::R / Ri
  double* sws;          // global workspace of the S-cone kernels for orders above 64 (nullptr if none)
  long long sws_stride; // doubles per CTA
};
struct Scaling {   // flattened block-diagonal operator: per cone  diag(a) + D * b b'   (kind 1) or diag(a) (kind 0)
  int* kind;       // [ncones]
  double* a;       // [m]
  double* b;       // [m]
  double* D;       // [ncones]
  double* R;       // VecCongurance blocks (kind 2): concatenated k*k column-major R ...
  double* Ri;      // ... and inv(R); shared between F and its inverse
};

int cone_nt_scaling(const ConeDesc& c, const double* v, const double* s, Scaling F, Scaling Fi, double* lambda,
                    int* info, cudaStream_t st);
int cone_invert_scaling(const ConeDesc& c, Scaling F, Scaling Fi, cudaStream_t st);
// y = op(F) x with op in CIP_OP_{F,FT,FINVT,FINV}; Fi is the precomputed inverse of the diag/Woodbury part
int cone_apply(const ConeDesc& c, const Scaling& F, const Scaling& Fi, int op, const double* x, double* y,
               cudaStream_t st);
// y = inv(F) inv(F)' x, or y = minus - inv(F) inv(F)' x  (src/kktsolvers.jl:326,328); tmp: m doubles, S cones only
int cone_apply_invsq(const ConeDesc& c, const Scaling& F, const Scaling& Fi, const double* x, double* y,
                     const double* minus, double* tmp, cudaStream_t st);
int cone_prod(const ConeDesc& c, const double* x, const double* y, double* o, cudaStream_t st);
int cone_div(const ConeDesc& c, const double* x, const double* y, double* o, cudaStream_t st);
// result (device scalar) = min over cones; d == nullptr -> `nothing` variant
int cone_maxstep(const ConeDesc& c, const double* x, const double* d, double d_scale, double* partial,
                 int npartial, double* result, cudaStream_t st);
// Atil = F^-T A on the Q4 transposed panel (rows = columns of A, k = rows of A)
int cone_scale_panel(const ConeDesc& c, Scaling Fi, const double* At4, double* Atil4, int ld, int m_pad,
                     int ncols, cudaStream_t st);
// The same for R rows only (the diagonal pass), which also leaves e_j = round(log2 ||Atil[:, j]||) in colexp[ld]
// (the fast SYRK's column equilibration).  colss: scale_panel_norms_chunks(m_pad) * ld doubles of scratch; ld % 256 == 0.
int scale_panel_norms_chunks(int m_pad);
int cone_scale_panel_norms(Scaling Fi, const double* At4, double* Atil4, int ld, int m_pad, double* colss,
                           int* colexp, cudaStream_t st);

// ---------------------------------------------------------------- S (PSD) cones (sdp.cu)
int sdp_max_order();
long long sdp_workspace_doubles(int k);          // per CTA, 0 when the order fits shared memory
int sdp_panel_chunks(int max_order, int ncols);  // grid.y of the S rows of the scaled panel
int sdp_apply(const ConeDesc& c, const Scaling& F, int use_inv, int transpose, const double* x, double* y,
              cudaStream_t st);
int sdp_nt_scaling(const ConeDesc& c, Scaling F, Scaling Fi, const double* v, const double* s, double* lambda,
                   int* info, cudaStream_t st);
int sdp_invert(const ConeDesc& c, Scaling F, cudaStream_t st);
// y = minus - y on the rows of the S cones that carry a VecCongurance block
int sdp_rows_rsub(const ConeDesc& c, const Scaling& F, const double* minus, double* y, cudaStream_t st);
int sdp_prod_div(const ConeDesc& c, const double* x, const double* y, double* o, int divide, cudaStream_t st);
int sdp_maxstep(const ConeDesc& c, const double* x, const double* d, double d_scale, unsigned long long* key,
                cudaStream_t st);
int sdp_scale_panel(const ConeDesc& c, const Scaling& Fi, const double* At4, double* Atil4, int ld, int ncols,
                    cudaStream_t st);

// ---------------------------------------------------------------- Cholesky (chol.cu)
struct CholPlan {
  double* H;        // Q4, ld = n_pad
  int ld;           // n_pad (multiple of 128)
  int npanels;
  double* Winv;     // [npanels][32][128][4]
  GemmOperand mapH;     // over H
  GemmOperand mapWinv;  // over Winv viewed as Q4 with ld = 128, kq_total = 32*npanels
  int* info;        // device int
  // look-ahead: panel factorisation / TRSM / next-column update run on a high-priority stream
  // while the bulk trailing update of the previous panel runs on the caller's stream
  cudaStream_t sc = nullptr;
  cudaEvent_t evT[2] = {}, evR[2] = {}, evS = nullptr;
  // inner look-ahead: the update of the NEXT 128-column panel stays on the chain (sc), the update of the other
  // columns of the outer panel runs beside it on sd
  cudaStream_t sd = nullptr;
  cudaEvent_t evD[2] = {}, evP = nullptr;
  // outer look-ahead: rank-128 updates of the next outer panel's block column, one per finished inner panel (se);
  // distributed variant: broadcasts of the inner panels (sb)
  cudaStream_t se = nullptr, sb = nullptr;
  cudaEvent_t evE = nullptr;
  // panel head on the chain (chol_head_kernel), the rest of the column (sd) and the other columns (sf) beside it
  cudaStream_t sf = nullptr;
  cudaEvent_t evC = nullptr, evH = nullptr, evUc[2] = {}, evUo[2] = {};
  // chol_factor's launch sequence as a CUDA graph (captured on first use)
  cudaGraphExec_t graph_exec = nullptr;
  bool capturing = false, graph_failed = false;
  long long graph_kernels = 0;
  int nranks_hint = 1;      // ranks sharing the factorisation (set by the engine once a communicator exists)
  // persistent triangular sweeps: work units (device), partial sums of split block rows, error flag
  void *units_fwd = nullptr, *units_bwd = nullptr;
  int nunits = 0, maxseg = 1;
  double* sweep_part = nullptr;
  int* sweep_err = nullptr;
};
int chol_make_plan(CholPlan* p, double* H, int n_pad, double* Winv, int* info);
void chol_free_plan(CholPlan* p);
int chol_factor(const CholPlan& p, cudaStream_t s);
// Block-cyclic distributed variant (SURVEY 8f rank 3): every rank holds the full matrix buffer, outer
// panel J is factored by rank J % nranks and broadcast (NCCL), each rank applies it only to the outer
// panels it owns.  On return every rank holds the complete factor L and all inv(L_jj) blocks.
struct CholDist {
  int nranks = 1, rank = 0;
  void* comm = nullptr;   // ncclComm_t
};
int chol_factor_dist(const CholPlan& p, cudaStream_t s, const CholDist& d);
// y receives the solution of L y = b (b is read only; b and y must not alias; both of length n_pad)
int chol_fwd(const CholPlan& p, double* b, double* y, cudaStream_t s);
// x receives the solution of L' x = y
int chol_bwd(const CholPlan& p, double* y, double* x, cudaStream_t s);

// small vector helpers (vecops.cu)
int vec_axpby(double* out, double a, const double* x, double b, const double* y, size_t n, cudaStream_t s);
int vec_copy(double* out, const double* x, size_t n, cudaStream_t s);

// FP64 pipe microbenchmarks (peaks.cu)
int measure_fp64_peaks(double* dmma_tflops, double* dfma_tflops);

}  // namespace cip
