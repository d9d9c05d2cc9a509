// Private definition of the engine handle, shared by engine.cu (C ABI) and ipm.cu (native
// interior-point driver).
#pragma once
#include <vector>

#include "../../include/conicip_b200.h"
#include "kernels.cuh"

constexpr int NV = 8;   // n-length work vectors
constexpr int MV = 10;  // m-length work vectors
constexpr int PV = 6;   // p-length work vectors

namespace cip {
struct Multi;

// cip_options.row_structure (structure.cu).  The rows of A split into singletons (R rows with one non-zero, sorted
// by (column, row) behind a column pointer), empty R rows, and the rest (every Q / S row and the R rows with >= 2
// non-zeros, ascending), which keep a compact Q4 copy At4r (ld = nJ_pad, k = rest rows) over the column support J.
struct RowStructure {
  bool on = false;
  int nsing = 0, nempty = 0, nr = 0, nr_pad = 0, nJ = 0, nJ_pad = 0;
  bool compressed = false, base_has_gtg = false, fold = false;
  double *At4r = nullptr, *Atil4r = nullptr, *Hr4 = nullptr;   // Hr4: nJ_pad^2 Gram scratch (compressed only)
  double* Base4 = nullptr;          // Q + rho G'G (owned when base_has_gtg, else an alias of Qq4)
  GemmOperand map{};                // over Atil4r, or over At4r when folded
  int *rest_row = nullptr, *J = nullptr, *Jinv = nullptr;      // [nr], [nJ], [n] (-1: column outside J)
  int* row_code = nullptr;          // [m]: >= 0 rest index, -1 - s singleton s, INT_MIN empty
  int *sing_ptr = nullptr, *sing_row = nullptr, *sing_col = nullptr;   // [n+1], [nsing], [nsing]
  double* sing_val = nullptr;       // [nsing]
  // cone descriptor of the rest rows: whole Q / S cones and the rest rows of each R cone, in global order
  ConeDesc cd{};
  int *d_type = nullptr, *d_off = nullptr, *d_rowcone = nullptr, *d_qlist = nullptr, *d_slist = nullptr;
  int* cone_map = nullptr;          // [cones of cd] -> global cone
  Scaling Fi{};                     // Fi gathered into rest order (R / Ri shared with the handle's)
  // work vectors of the mat-vecs, two sets (cip_solve_multi pairs): x[rest], y[J], products
  double *xr[2] = {}, *yJ[2] = {}, *outr[2] = {}, *outJ[2] = {};

  // row_structure = 2: the columns of H split into K (coupled: touched by a rest row, by an off-diagonal entry of Q,
  // or -- when rho > 0 -- by G) and D (all others, where H holds only its diagonal h_j).  H_KK is dense and factored
  // with a Cholesky plan over nK_pad; D is factored as sqrt(h_j).  No n_pad^2 buffer exists.
  struct Split {
    bool on = false;
    int nK = 0, nK_pad = 0, from_rest = 0, from_Q = 0, from_G = 0;
    bool g_in_D = false;            // some column of G lies in D: S gets G diag(kscale^2) G' and the solves G u
    bool factored = false;          // HK4 holds L_KK (cip_get_H shows L), else H_KK
    std::vector<int> K;             // host copy: failing K pivot -> global column
    std::vector<char> q_couple;     // per column: Q couples it (LEVEL 1, until K is built)
    struct QEntry { int i, j; double v; };
    std::vector<QEntry> qtrip;      // CSC Q: summed diagonal entries and those between coupled columns (LEVEL 1)
    int *dK = nullptr, *Kpos = nullptr, *JK = nullptr;   // [nK], [n] (-1: column in D), [nJ]: K position of J[a]
    double *QK4 = nullptr, *BaseK4 = nullptr, *HK4 = nullptr, *WinvK = nullptr;   // nK_pad^2, nK_pad * TILE
    double *qD = nullptr, *hD = nullptr, *kscale = nullptr;   // [n_pad]: diagonal of Q, h on D, h^-1/2 on D
    double *GK4 = nullptr, *ZK4 = nullptr;   // p_pad x nK_pad
    CholPlan chol{};
    GemmOperand mapZK{}, mapG{};
    int* fail = nullptr;            // smallest global D column with h_j <= 0 (INT_MAX-ish when none)
    double* kv[2][3] = {};          // per column set b: rhs_K, t_K, products on K (nK_pad + 4 each)
  } sp;
};

// Fast SYRK (fast_syrk.cu): H = Q + Atil'Atil as a blocked SYRK whose off-diagonal blocks take one Strassen-Winograd
// level on power-of-two equilibrated columns, two where the blocks are wide.  Dense single-device R-only handles at
// large n (CIP_FAST_SYRK = 0 / 1 forces it off / on where the handle allows it).  Atil4 then holds 4 K2 rows of
// contraction: the rows of A (zero-padded to 2 K2), then the operand sums of the products; K2 / 2 more for the
// level-2 sums when some depth takes two levels.
struct FastSyrk {
  bool on = false;
  int depth = 0;               // levels of halving of [0, n_pad)
  int leaf = 0;                // n_pad >> depth: width of the diagonal blocks left to the plain SYRK
  int K2 = 0;                  // half the contraction (rows of A, padded), a multiple of 32 (of 64 when two != 0)
  unsigned two = 0;            // bit d: depth d takes a second Winograd level
  int nchunk = 0;              // k chunks of the column sums of squares
  int* colexp = nullptr;       // [n_pad] e_j = round(log2 ||Atil[:, j]||)
  double* colss = nullptr;     // [nchunk * n_pad]
  double* M = nullptr;         // the seven product tiles of every pair of one depth (7 n_pad^2 / 16)
  double* M2 = nullptr;        // the level-2 sub-product tiles of one level-1 product, every pair (two != 0)
  int4* table = nullptr;       // GemmArgs::group entries: the leaves, the products of depth 0, 1, ..., the level-2 ones
};
}  // namespace cip

struct cip_engine {
  // single-process multi-GPU: a handle created with opts.ngpus > 1 is only a front for `multi` (one shard
  // engine per device, each driven by its own host thread); a shard engine points back through `parent`
  cip::Multi* multi = nullptr;
  cip::Multi* parent = nullptr;
  int shard_index = 0;
  bool always_sync = false;   // shard engines: every call returns with its stream idle (outputs may live on another device)
  int n = 0, m = 0, p = 0, n_pad = 0, m_pad = 0, p_pad = 0, ncones = 0;
  int device = 0;
  cudaStream_t stream = nullptr, own_stream = nullptr;
  cip_options opt{};
  // matrices (Q4 layout)
  double *At4 = nullptr, *Atil4 = nullptr, *Qq4 = nullptr, *H4 = nullptr, *Winv = nullptr;
  double *G4 = nullptr, *Z4 = nullptr, *S4 = nullptr, *Sbase4 = nullptr, *WinvS = nullptr;
  cip::GemmOperand mapAtil{}, mapZ{};
  cip::CholPlan cholH{}, cholS{};
  int* info = nullptr;  // [2] device
  // cones
  std::vector<int> h_type, h_off;
  int *d_type = nullptr, *d_off = nullptr, *d_rowcone = nullptr, *d_qlist = nullptr, *d_slist = nullptr;
  int *d_sord = nullptr, *d_roff = nullptr;
  double* d_sws = nullptr;     // S-cone workspace (orders above 64)
  std::vector<int> h_slist, h_sord, h_roff;
  size_t r_total = 0;
  cip::ConeDesc cd{};
  cip::Scaling F{}, Fi{};
  bool have_scaling = false, have_factor = false;
  double* gemm_ws = nullptr;   // split-K workspace of gemm_nt (GEMM_WS_DOUBLES)
  bool fold = false;           // R-only handle without Atil4: the SYRK reads At4 and scales in registers (opts.fold_scaling)
  cip::GemmOperand mapAt{};
  int aug_rows = 0;        // rows of Atil4 beyond m_pad holding sqrt(aug_rho) * G
  double aug_rho = 0.0;
  cip::RowStructure rs;    // opts.row_structure: At4 / Atil4 are not allocated
  cip::FastSyrk fast;      // the Winograd SYRK of form_H (sized at cip_create, dropped when a communicator is attached)
  std::vector<void*> owned;   // further device buffers freed by cip_destroy
  // work vectors
  double* nv[NV] = {};
  double* mv[MV] = {};
  double* pv[PV] = {};
  // second set of the work vectors cip_solve uses (nv[0..5], mv[0..5], pv[0..4]): column b of a pair in
  // cip_solve_multi; allocated on the first call
  double* nv2[6] = {};
  double* mv2[6] = {};
  double* pv2[5] = {};
  double* partial = nullptr;
  int partial_cap = 0;
  double* scalar = nullptr;  // device scratch scalars [8]
  // NCCL
  void* comm = nullptr;
  int nranks = 1, rank = 0;
  // overlapped Gram reduction (row-sharded handles): tile-major partial Gram matrix, all-reduced range by range
  // on `cs` while the SYRK of the later ranges still runs (alternating between the handle's stream and `s2`)
  double* Hp = nullptr;
  cudaStream_t cs = nullptr, s2 = nullptr;
  cudaEvent_t evc[16] = {};
  // stats
  cip_stats_t st{};
  cudaEvent_t ev[8] = {};
  size_t bytes = 0;
  bool need_sync = false;
};


namespace cip {
// sum-all-reduce `count` doubles in place across the row shards (no-op for a single GPU)
int engine_allreduce(cip_engine* h, double* buf, size_t count);
// cip_create / cip_create_csc for one device (engine.cu)
int engine_create_single(cip_handle* out, int n, int m, int p, const double* Q, int ldq, const double* A, int lda,
                         const double* G, int ldg, const cip_csc* Qs, const cip_csc* As, const cip_csc* Gs,
                         int ncones, const int* cone_type, const int* cone_dim, const cip_options* opts);
const char* last_error_string();
// fold the scaling into the SYRK? (opts.fold_scaling / CIP_FOLD_SCALING, else free memory against the mn-double
// second copy); `can`: every row of the SYRK is an R row
int engine_decide_fold(cip_engine* h, bool can, size_t mn, bool* fold);
// buffers / streams of the overlapped Gram reduction, once the communicator exists (engine.cu)
int engine_setup_comm(cip_engine* h);

// ---- fast SYRK (fast_syrk.cu)
// LEVEL 1, before Atil4 is allocated: take the fast path?  `can`: dense, unfolded, every row an R row, no
// augmentation rows.  Sets h->fast (n_pad, free memory, CIP_FAST_SYRK, CIP_FAST_SYRK_LEAF, CIP_FAST_SYRK_LEVELS).
int fast_syrk_plan(cip_engine* h, bool can);
size_t fast_syrk_atil_doubles(const cip_engine* h);     // the size of Atil4 when h->fast.on
// LEVEL 1, after Atil4: exponents, scratch, product tiles, the launch table
int fast_syrk_setup(cip_engine* h);
// a communicator was attached: back to the plain Atil4 and the classical SYRK
int fast_syrk_drop(cip_engine* h);
// LEVEL 2, after cone_scale_panel_norms: H4 = cin + Atil'Atil (lower triangle)
int fast_syrk_form(cip_engine* h, const double* cin);

// ---- row structure (structure.cu)
// LEVEL 1, dense input: classify the rows of the packed At4, build the compact arrays, free At4
int structure_build_dense(cip_engine* h);
// LEVEL 1, CSC input: classify from the CSC arrays and scatter only the rest rows (no dense At4)
int structure_build_csc(cip_engine* h, const cip_csc* A);
// LEVEL 1, after G4: Base4 = Q + rho G'G (or an alias of Qq4), the tensor map of the SYRK operand
int structure_finish(cip_engine* h);
// LEVEL 2: H4 = Base4 + Atil_r'Atil_r (scattered at J x J) + the singleton diagonal; records ev[1], ev[2]
int structure_form_H(cip_engine* h);
// out[n] = add + A' x  (x: m-vector readable up to m); b selects the work vector set
int structure_AT(cip_engine* h, double* out, const double* x, const double* add, int b);
int structure_AT2(cip_engine* h, double* outa, double* outb, const double* xa, const double* xb, const double* adda,
                  const double* addb);
// out[m] = A y  (y: n-vector)
int structure_A(cip_engine* h, double* out, const double* y, int b);
int structure_A2(cip_engine* h, double* outa, double* outb, const double* ya, const double* yb);
// row_structure = 2 (structure.cu).  LEVEL 1, dense Q in h->Qq4 or CSC / diagonal / no Q: the Q diagonal and which
// columns Q couples (the dense staging copy stays until split_build)
int split_classify_csc_Q(cip_engine* h, const cip_csc* Q);
int split_diag_Q(cip_engine* h, const double* q);
// LEVEL 1, after G4 and the row split: K, QK4, BaseK4, GK4, the K Cholesky plan; frees the dense Q staging copy
int split_build(cip_engine* h);
// LEVEL 2: Cholesky of H_KK, the pivots of D (kscale, the smallest failing D column); the Schur block is factor_H's
int split_factor(cip_engine* h);
int split_add_delta(cip_engine* h, double delta);
// LEVEL 3 on one column set: nv[2] = rhs in, nv[5] = dy out; pv[0] = rw, pv[4] = dw out (schur: p > 0)
int split_solve(cip_engine* h, double** nv, double** pv, int b, bool schur);
int split_mul_Q(cip_engine* h, double* y, const double* x);
int split_get_H(cip_engine* h, double* tmp);   // n x n, column-major

// ---- single-process multi-GPU front (multi.cu): same contracts as the C ABI entry points, global vectors
int multi_create(cip_handle* out, int n, int m, int p, const double* Q, int ldq, const double* A, int lda,
                 const double* G, int ldg, const cip_csc* Qs, const cip_csc* As, const cip_csc* Gs, int ncones,
                 const int* cone_type, const int* cone_dim, const cip_options* opts);
int multi_destroy(cip_engine* h);
int multi_factor(cip_engine* h, const int* kind, const double* fa, const double* fb, const double* fD,
                 const double* fR, int factor);      // factor = 0: cip_set_scaling
int multi_get_scaling(cip_engine* h, int* kind, double* fa, double* fb, double* fD, double* fR);
int multi_nt_scaling(cip_engine* h, const double* v, const double* s, double* lambda_out, int factor);
int multi_solve(cip_engine* h, const double* ry, const double* rw, const double* rv, double* dy, double* dw,
                double* dv);
int multi_solve_multi(cip_engine* h, int nrhs, const double* ry, int ldy, const double* rw, int ldw, const double* rv,
                      int ldv, double* dy, double* dw, double* dv);
int multi_apply(cip_engine* h, int op, const double* x, double* y);
int multi_maxstep(cip_engine* h, const double* x, const double* d, double d_scale, double* alpha_out);
int multi_prod_div(cip_engine* h, const double* x, const double* y, double* o, int divide);
int multi_mul_A(cip_engine* h, int trans, const double* x, double* y);
int multi_mul_GQ(cip_engine* h, int which, int trans, const double* x, double* y);   // which: 0 = G, 1 = Q
int multi_ipm_solve(cip_engine* h, const double* c, const double* b, const double* d, const cip_ipm_options* opts,
                    double* y, double* w, double* v, cip_ipm_result* result);
int multi_stats(cip_engine* h, cip_stats_t* out);
int multi_simple(cip_engine* h, int what, double* out, int ldo);   // 0 form_H, 1 factor_H, 2 sync, 3 get_H
void multi_barrier(cip::Multi* m);   // rendezvous of the shard threads inside one dispatched call
}  // namespace cip
