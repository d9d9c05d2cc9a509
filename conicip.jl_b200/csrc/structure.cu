// Row structure of A (cip_options.row_structure).
//
// H = Q + (F^-T A)'(F^-T A) is a sum over the rows of A.  W is diagonal on the R cones, so an R row with a single
// non-zero a_ij adds (Fi.a[i] a_ij)^2 to H_jj and nothing else; the dense SYRK spends m_pad * n_pad^2 flops on
// rows like that.  Here the rows are classified once at LEVEL 1:
//   singletons  R rows with exactly one non-zero: stored sorted by (column, row) behind a column pointer, so every
//               per-column sum runs in a fixed order (bit-reproducible)
//   empty       R rows without a non-zero: contribute nothing
//   rest        every Q / S row (W is not diagonal there) and the R rows with >= 2 non-zeros, in ascending order,
//               kept as a compact Q4 matrix At4r (k = rest rows) over the columns J they touch
// and the constant Q + rho G'G is formed once.  LEVEL 2 then runs the SYRK on the rest only (on J x J when J is
// at most half the columns), scatters it onto the constant part and adds the singletons to the diagonal.
// J can be empty while the rest has rows (a Q or S cone whose rows of A are all zero): those rows add nothing to
// H, A y or A'x, so the operand map, the SYRK, the scatter and the rest mat-vecs are skipped.
// A non-zero is a stored value != 0.0, for dense and CSC input alike.
// row_structure = 2 splits the columns of H on top of this (second half of the file).
#include <climits>
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "engine.h"

namespace cip {
namespace {

constexpr int EMPTY_ROW = INT_MIN;

template <typename T>
int salloc(cip_engine* h, T** p, size_t count) {
  *p = nullptr;
  if (count == 0) count = 1;
  CIP_CUDA(cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T)));
  CIP_CUDA(cudaMemsetAsync(*p, 0, count * sizeof(T), h->stream));
  h->bytes += count * sizeof(T);
  h->owned.push_back(*p);
  return 0;
}
template <typename T>
int supload(cip_engine* h, T** p, const std::vector<T>& v) {
  CIP_TRY(salloc(h, p, v.size()));
  if (!v.empty()) CIP_CUDA(cudaMemcpyAsync(*p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream));
  return 0;
}

// ---------------------------------------------------------------- LEVEL 1 kernels
// one warp per k-quad of At4 (four rows of A): count the non-zeros of each row, first non-zero column and value
__global__ void __launch_bounds__(256)
classify_rows_kernel(const double* __restrict__ At4, int ld, int n, int m, int* __restrict__ cnt,
                     int* __restrict__ col, double* __restrict__ val) {
  const int lane = threadIdx.x & 31;
  const int q = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (q * 4 >= m) return;
  int c[4] = {0, 0, 0, 0}, f[4] = {INT_MAX, INT_MAX, INT_MAX, INT_MAX};
  for (int j = lane; j < n; j += 32) {
    const double2* p = reinterpret_cast<const double2*>(At4 + ((size_t)q * ld + j) * 4);
    const double2 v0 = __ldg(p), v1 = __ldg(p + 1);
    const double v[4] = {v0.x, v0.y, v1.x, v1.y};
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if (v[r] != 0.0) { ++c[r]; f[r] = min(f[r], j); }
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int cs = __reduce_add_sync(0xffffffffu, (unsigned)c[r]);
    const int fm = __reduce_min_sync(0xffffffffu, f[r]);
    const int i = q * 4 + r;
    if (lane == 0 && i < m) {
      cnt[i] = min(cs, 2);
      col[i] = cs > 0 ? fm : -1;
      val[i] = cs > 0 ? At4[q4_index(fm, i, ld)] : 0.0;
    }
  }
}

// touched[j] = 1 when one of the rest rows has a non-zero in column j
__global__ void col_support_kernel(const double* __restrict__ At4, int ld, int n, const int* __restrict__ rest_row,
                                   int nr, int* __restrict__ touched) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  int t = 0;
  for (int kk = 0; kk < nr && !t; ++kk) t = At4[q4_index(j, rest_row[kk], ld)] != 0.0;
  touched[j] = t;
}

// At4r[jj, kk] = At4[J[jj], rest_row[kk]]
__global__ void gather_rest_kernel(double* __restrict__ At4r, int ldr, const double* __restrict__ At4, int ld,
                                   const int* __restrict__ J, int nJ, const int* __restrict__ rest_row, int nr) {
  const int jj = blockIdx.x * blockDim.x + threadIdx.x;
  if (jj >= nJ) return;
  const int j = J[jj];
  for (int kk = blockIdx.y; kk < nr; kk += gridDim.y)
    At4r[q4_index(jj, kk, ldr)] = At4[q4_index(j, rest_row[kk], ld)];
}

// ---------------------------------------------------------------- LEVEL 2 kernels
// the inverse scaling in rest-row order: a, b per row; kind, D per cone (R / Ri are shared)
__global__ void gather_scaling_kernel(Scaling Fi, Scaling Fr, const int* __restrict__ rest_row, int nr,
                                      const int* __restrict__ cone_map, int ncr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nr) {
    const int g = rest_row[i];
    Fr.a[i] = Fi.a[g];
    Fr.b[i] = Fi.b[g];
  }
  if (i < ncr) {
    const int c = cone_map[i];
    Fr.kind[i] = Fi.kind[c];
    Fr.D[i] = Fi.D[c];
  }
}

// H4[J[a], J[b]] += Hr4[a, b] over the lower triangle of the compact Gram matrix.  Inside a diagonal tile of H4 both
// halves are kept (as the SYRK writes them), so the mirror element is added there too.  Every element of H4 has
// one writer.
__global__ void scatter_gram_kernel(double* __restrict__ H4, int ld, const double* __restrict__ Hr4, int ldr,
                                    const int* __restrict__ J, int nJ) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  for (int b = blockIdx.y; b < nJ; b += gridDim.y) {
    if (a >= nJ || a < b) continue;
    const double v = Hr4[q4_index(a, b, ldr)];
    const int ga = J[a], gb = J[b];
    H4[q4_index(ga, gb, ld)] += v;
    if (a != b && ga / TILE == gb / TILE) H4[q4_index(gb, ga, ld)] += v;
  }
}

// H_jj += sum over the singletons of column j of (Fi.a[i] a_ij)^2, rows in ascending order.  With a position map
// (row_structure = 2) column j is row pos[j] of H4, or goes to hD[j] when pos[j] < 0.
__global__ void singleton_diag_kernel(double* __restrict__ H4, int ld, int n, const int* __restrict__ ptr,
                                      const int* __restrict__ row, const double* __restrict__ val,
                                      const double* __restrict__ ia, const int* __restrict__ pos,
                                      double* __restrict__ hD) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int e0 = ptr[j], e1 = ptr[j + 1];
  if (e0 == e1) return;
  double acc = 0;
  for (int e = e0; e < e1; ++e) {
    const double t = ia[row[e]] * val[e];
    acc += t * t;
  }
  const int k = pos ? pos[j] : j;
  if (k >= 0) H4[q4_index(k, k, ld)] += acc;
  else hD[j] += acc;
}

// ---------------------------------------------------------------- mat-vec kernels
__global__ void gather_vec_kernel(double* __restrict__ out, const double* __restrict__ x, const int* __restrict__ idx,
                                  int count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) out[i] = x[idx[i]];
}

// out[j] = add[j] + (At4r' x_rest)[Jinv[j]] + sum over the singletons of column j of a_ij x_i
__global__ void finish_at_kernel(double* __restrict__ out, const double* __restrict__ add,
                                 const double* __restrict__ outJ, const int* __restrict__ Jinv,
                                 const int* __restrict__ ptr, const int* __restrict__ row,
                                 const double* __restrict__ val, const double* __restrict__ x, int n) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int jj = outJ ? Jinv[j] : -1;
  double r = jj >= 0 ? outJ[jj] : 0.0;
  for (int e = ptr[j]; e < ptr[j + 1]; ++e) r += val[e] * x[row[e]];
  out[j] = add ? add[j] + r : r;
}

// out[i] = (At4r y_J)[rest index] on rest rows (0 without outr: J is empty), a_ij y_j on singletons, 0 on empty rows
__global__ void finish_a_kernel(double* __restrict__ out, const double* __restrict__ outr,
                                const int* __restrict__ code, const int* __restrict__ scol,
                                const double* __restrict__ sval, const double* __restrict__ y, int m) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const int c = code[i];
  out[i] = c >= 0 ? (outr ? outr[c] : 0.0) : (c == EMPTY_ROW ? 0.0 : sval[-1 - c] * y[scol[-1 - c]]);
}

inline unsigned nb(long long n, int per) { return (unsigned)std::max<long long>(1, (n + per - 1) / per); }

// ---------------------------------------------------------------- host side of LEVEL 1
// per row of A: number of non-zeros (capped at 2), first non-zero column and its value
struct RowClass {
  std::vector<int> cnt, col;
  std::vector<double> val;
};

// Everything that follows the classification: the row split, cone descriptor, singleton arrays and column support.
// `touched`: columns hit by a non-zero of a rest row (computed by the caller, which needs rest_row first).
struct Plan {
  std::vector<int> rest_row, row_code, sing_ptr, sing_row, sing_col;
  std::vector<double> sing_val;
  std::vector<int> ctype, coff, cmap, rowcone, qlist, slist;
  int nr_rows = 0, nsing = 0, nempty = 0;
};

int make_plan(cip_engine* h, const RowClass& rc, Plan* P) {
  const int m = h->m, n = h->n;
  std::vector<char> is_r(m, 0);
  for (int c = 0; c < h->ncones; ++c)
    if (h->h_type[c] == CIP_CONE_R)
      for (int i = h->h_off[c]; i < h->h_off[c + 1]; ++i) is_r[i] = 1;
  P->row_code.assign(m, EMPTY_ROW);
  std::vector<int> sing;                            // global rows of the singletons
  for (int i = 0; i < m; ++i) {
    if (!is_r[i] || rc.cnt[i] >= 2) {
      P->row_code[i] = (int)P->rest_row.size();
      P->rest_row.push_back(i);
    } else if (rc.cnt[i] == 1) {
      sing.push_back(i);
    } else {
      P->nempty++;
    }
  }
  std::stable_sort(sing.begin(), sing.end(), [&](int a, int b) { return rc.col[a] < rc.col[b]; });  // rows ascending
  P->nsing = (int)sing.size();
  P->sing_ptr.assign(n + 1, 0);
  for (int s = 0; s < P->nsing; ++s) {
    const int i = sing[s];
    P->sing_row.push_back(i);
    P->sing_col.push_back(rc.col[i]);
    P->sing_val.push_back(rc.val[i]);
    P->sing_ptr[rc.col[i] + 1]++;
    P->row_code[i] = -1 - s;
  }
  for (int j = 0; j < n; ++j) P->sing_ptr[j + 1] += P->sing_ptr[j];
  // cones of the rest: whole Q / S cones, and the rest rows of each R cone (contiguous in rest order)
  P->coff.push_back(0);
  for (int c = 0; c < h->ncones; ++c) {
    int k = 0;
    for (int i = h->h_off[c]; i < h->h_off[c + 1]; ++i) k += P->row_code[i] >= 0;
    if (k == 0) continue;
    const int ci = (int)P->ctype.size();
    if (h->h_type[c] == CIP_CONE_Q) P->qlist.push_back(ci);
    else if (h->h_type[c] == CIP_CONE_S) P->slist.push_back(ci);
    else P->nr_rows += k;
    P->ctype.push_back(h->h_type[c]);
    P->cmap.push_back(c);
    P->coff.push_back(P->coff.back() + k);
    for (int r = 0; r < k; ++r) P->rowcone.push_back(ci);
  }
  return 0;
}

// uploads the plan; J from `touched`; decides compression and folding; allocates At4r / Atil4r / Hr4 / work vectors
int upload_plan(cip_engine* h, const Plan& P, const std::vector<int>& touched) {
  RowStructure& rs = h->rs;
  const int n = h->n;
  rs.nr = (int)P.rest_row.size();
  rs.nr_pad = round_up(rs.nr, 32);
  rs.nsing = P.nsing;
  rs.nempty = P.nempty;
  std::vector<int> J;
  for (int j = 0; j < n; ++j)
    if (touched[j]) J.push_back(j);
  // (row_structure = 2 always compresses: H has no n_pad-wide buffer to take the Gram matrix of all columns)
  rs.compressed = rs.nr > 0 && (rs.sp.on || round_up((int)J.size(), TILE) <= h->n_pad / 2);
  if (!rs.compressed) {
    J.resize(n);
    for (int j = 0; j < n; ++j) J[j] = j;
  }
  if (rs.nr == 0) J.clear();
  rs.nJ = (int)J.size();
  rs.nJ_pad = rs.compressed ? round_up(rs.nJ, TILE) : (rs.nr > 0 ? h->n_pad : 0);
  std::vector<int> Jinv(n, -1);
  for (int a = 0; a < rs.nJ; ++a) Jinv[J[a]] = a;
  CIP_TRY(supload(h, &rs.rest_row, P.rest_row));
  CIP_TRY(supload(h, &rs.J, J));
  CIP_TRY(supload(h, &rs.Jinv, Jinv));
  CIP_TRY(supload(h, &rs.row_code, P.row_code));
  CIP_TRY(supload(h, &rs.sing_ptr, P.sing_ptr));
  CIP_TRY(supload(h, &rs.sing_row, P.sing_row));
  CIP_TRY(supload(h, &rs.sing_col, P.sing_col));
  CIP_TRY(supload(h, &rs.sing_val, P.sing_val));
  // cone descriptor of the rest rows; the S cones are all there, in the same order, so their orders, R offsets and
  // workspace are the handle's
  const int ncr = (int)P.ctype.size();
  CIP_TRY(supload(h, &rs.d_type, P.ctype));
  CIP_TRY(supload(h, &rs.d_off, P.coff));
  CIP_TRY(supload(h, &rs.d_rowcone, P.rowcone));
  CIP_TRY(supload(h, &rs.d_qlist, P.qlist));
  CIP_TRY(supload(h, &rs.d_slist, P.slist));
  CIP_TRY(supload(h, &rs.cone_map, P.cmap));
  ConeDesc& c = rs.cd;
  c = h->cd;
  c.m = rs.nr; c.ncones = ncr; c.type = rs.d_type; c.off = rs.d_off; c.row_cone = rs.d_rowcone;
  c.qlist = rs.d_qlist; c.nq = (int)P.qlist.size(); c.slist = rs.d_slist; c.ns = (int)P.slist.size();
  c.nr_rows = P.nr_rows;
  CIP_TRY(salloc(h, &rs.Fi.kind, ncr));
  CIP_TRY(salloc(h, &rs.Fi.a, rs.nr_pad + 4));
  CIP_TRY(salloc(h, &rs.Fi.b, rs.nr_pad + 4));
  CIP_TRY(salloc(h, &rs.Fi.D, ncr));
  rs.Fi.R = h->Fi.R;
  rs.Fi.Ri = h->Fi.Ri;
  for (int b = 0; b < 2; ++b) {
    CIP_TRY(salloc(h, &rs.xr[b], rs.nr_pad + 4));
    CIP_TRY(salloc(h, &rs.outr[b], rs.nr_pad + 4));
    CIP_TRY(salloc(h, &rs.yJ[b], rs.nJ_pad + 4));
    CIP_TRY(salloc(h, &rs.outJ[b], rs.nJ_pad + 4));
  }
  // the scaling folds into the SYRK on the rule of the dense path, applied to the rest (the aug rows are not there)
  const size_t mnr = (size_t)rs.nr_pad * rs.nJ_pad;
  CIP_TRY(engine_decide_fold(h, P.qlist.empty() && P.slist.empty() && rs.nr > 0, mnr, &rs.fold));
  if (rs.nr > 0 && !rs.fold) CIP_TRY(salloc(h, &rs.Atil4r, mnr));
  if (rs.compressed) CIP_TRY(salloc(h, &rs.Hr4, (size_t)rs.nJ_pad * rs.nJ_pad));
  return 0;
}

}  // namespace

int structure_build_dense(cip_engine* h) {
  RowStructure& rs = h->rs;
  cudaStream_t s = h->stream;
  const int m = h->m, n = h->n;
  RowClass rc;
  rc.cnt.resize(m); rc.col.resize(m); rc.val.resize(m);
  int *dcnt = nullptr, *dcol = nullptr;
  double* dval = nullptr;
  CIP_CUDA(cudaMalloc(&dcnt, sizeof(int) * m));
  CIP_CUDA(cudaMalloc(&dcol, sizeof(int) * m));
  CIP_CUDA(cudaMalloc(&dval, sizeof(double) * m));
  classify_rows_kernel<<<nb((m + 3) / 4, 8), 256, 0, s>>>(h->At4, h->n_pad, n, m, dcnt, dcol, dval);
  const cudaError_t le = cudaGetLastError();
  g_launches++;
  cudaMemcpyAsync(rc.cnt.data(), dcnt, sizeof(int) * m, cudaMemcpyDeviceToHost, s);
  cudaMemcpyAsync(rc.col.data(), dcol, sizeof(int) * m, cudaMemcpyDeviceToHost, s);
  cudaMemcpyAsync(rc.val.data(), dval, sizeof(double) * m, cudaMemcpyDeviceToHost, s);
  const cudaError_t se = cudaStreamSynchronize(s);
  cudaFree(dcnt); cudaFree(dcol); cudaFree(dval);
  CIP_CUDA(le);
  CIP_CUDA(se);
  Plan P;
  CIP_TRY(make_plan(h, rc, &P));
  const int nr = (int)P.rest_row.size();
  std::vector<int> touched(n, 0);
  if (nr > 0) {
    int *drest = nullptr, *dtouch = nullptr;
    CIP_CUDA(cudaMalloc(&drest, sizeof(int) * nr));
    CIP_CUDA(cudaMalloc(&dtouch, sizeof(int) * n));
    cudaMemcpyAsync(drest, P.rest_row.data(), sizeof(int) * nr, cudaMemcpyHostToDevice, s);
    col_support_kernel<<<nb(n, 128), 128, 0, s>>>(h->At4, h->n_pad, n, drest, nr, dtouch);
    const cudaError_t e1 = cudaGetLastError();
    g_launches++;
    cudaMemcpyAsync(touched.data(), dtouch, sizeof(int) * n, cudaMemcpyDeviceToHost, s);
    const cudaError_t e2 = cudaStreamSynchronize(s);
    cudaFree(drest); cudaFree(dtouch);
    CIP_CUDA(e1);
    CIP_CUDA(e2);
  }
  CIP_TRY(upload_plan(h, P, touched));
  const size_t mn = (size_t)h->m_pad * h->n_pad;
  if (rs.nr == m && !rs.compressed) {
    // every row is in the rest and J is every column: At4 already is At4r
    rs.At4r = h->At4;
    h->owned.push_back(h->At4);
    h->At4 = nullptr;
    return 0;
  }
  if (rs.nr > 0) {
    CIP_TRY(salloc(h, &rs.At4r, (size_t)rs.nr_pad * rs.nJ_pad));
    dim3 grid(nb(rs.nJ, 128), (unsigned)std::min(rs.nr, 65535));
    gather_rest_kernel<<<grid, 128, 0, s>>>(rs.At4r, rs.nJ_pad, h->At4, h->n_pad, rs.J, rs.nJ, rs.rest_row, rs.nr);
    CIP_CHECK_LAUNCH();
  }
  CIP_CUDA(cudaStreamSynchronize(s));
  cudaFree(h->At4);
  h->At4 = nullptr;
  h->bytes -= mn * sizeof(double);
  return 0;
}

namespace {
// (row, column, value) of the non-zeros of a CSC matrix (host or device arrays), columns ascending, rows ascending
// inside a column, duplicates summed in storage order (as the scatter of the dense path adds them)
struct E { int i, j; double v; };
int read_csc(const cip_csc* A, int m, std::vector<E>* out) {
  std::vector<E>& ent = *out;
  const long long ncols = A->ncols;
  const int base = A->index_base;
  std::vector<long long> cp(ncols + 1);
  CIP_CUDA(cudaMemcpy(cp.data(), A->colptr, (ncols + 1) * 8, cudaMemcpyDefault));
  const long long nnz = cp[ncols] - cp[0];
  std::vector<long long> rv(std::max(nnz, 0LL));
  std::vector<double> nz(std::max(nnz, 0LL));
  if (nnz > 0) {
    CIP_CUDA(cudaMemcpy(rv.data(), A->rowval, nnz * 8, cudaMemcpyDefault));
    CIP_CUDA(cudaMemcpy(nz.data(), A->nzval, nnz * 8, cudaMemcpyDefault));
  }
  std::vector<std::pair<int, double>> colv;
  for (long long j = 0; j < ncols; ++j) {
    const long long e0 = cp[j] - base, e1 = cp[j + 1] - base;
    if (e0 < 0 || e1 < e0 || e1 > nnz) {
      set_error("malformed CSC input: column %lld holds a row index outside [0, %d) or an inverted column pointer", j, m);
      return -1;
    }
    colv.clear();
    for (long long e = e0; e < e1; ++e) {
      const long long i = rv[e] - base;
      if (i < 0 || i >= m) {
        set_error("malformed CSC input: column %lld holds a row index outside [0, %d) or an inverted column pointer", j, m);
        return -1;
      }
      colv.emplace_back((int)i, nz[e]);
    }
    std::stable_sort(colv.begin(), colv.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
    for (size_t t = 0; t < colv.size();) {
      double v = colv[t].second;
      size_t u = t + 1;
      for (; u < colv.size() && colv[u].first == colv[t].first; ++u) v += colv[u].second;
      if (v != 0.0) ent.push_back({colv[t].first, (int)j, v});
      t = u;
    }
  }
  return 0;
}
}  // namespace

int structure_build_csc(cip_engine* h, const cip_csc* A) {
  RowStructure& rs = h->rs;
  const int m = h->m, n = h->n;
  std::vector<E> ent;
  CIP_TRY(read_csc(A, m, &ent));
  RowClass rc;
  rc.cnt.assign(m, 0); rc.col.assign(m, -1); rc.val.assign(m, 0.0);
  for (const E& e : ent) {       // columns ascending: the first entry of a row is its first non-zero column
    if (rc.cnt[e.i] == 0) { rc.col[e.i] = e.j; rc.val[e.i] = e.v; }
    rc.cnt[e.i] = std::min(rc.cnt[e.i] + 1, 2);
  }
  Plan P;
  CIP_TRY(make_plan(h, rc, &P));
  std::vector<int> touched(n, 0);
  for (const E& e : ent)
    if (P.row_code[e.i] >= 0) touched[e.j] = 1;
  CIP_TRY(upload_plan(h, P, touched));
  if (rs.nr == 0) return 0;
  // the rest as a CSC matrix over (rest rows) x J, scattered into At4r
  std::vector<int> Jinv(n, -1);
  {
    int a = 0;
    for (int j = 0; j < n; ++j)
      if (!rs.compressed || touched[j]) Jinv[j] = a++;
  }
  std::vector<long long> rcp(rs.nJ + 1, 0), rrv;
  std::vector<double> rnz;
  for (const E& e : ent)
    if (P.row_code[e.i] >= 0) rcp[Jinv[e.j] + 1]++;
  for (int a = 0; a < rs.nJ; ++a) rcp[a + 1] += rcp[a];
  rrv.resize(rcp[rs.nJ]);
  rnz.resize(rcp[rs.nJ]);
  {
    std::vector<long long> pos(rcp.begin(), rcp.end() - 1);
    for (const E& e : ent) {
      if (P.row_code[e.i] < 0) continue;
      const long long at = pos[Jinv[e.j]]++;
      rrv[at] = P.row_code[e.i];
      rnz[at] = e.v;
    }
  }
  CIP_TRY(salloc(h, &rs.At4r, (size_t)rs.nr_pad * rs.nJ_pad));
  const long long rn = (long long)rrv.size();
  if (rn == 0) return 0;
  cudaStream_t s = h->stream;
  long long *dcp = nullptr, *drv = nullptr;
  double* dnz = nullptr;
  int* dbad = nullptr;
  CIP_CUDA(cudaMalloc(&dcp, rcp.size() * 8));
  CIP_CUDA(cudaMalloc(&drv, rn * 8));
  CIP_CUDA(cudaMalloc(&dnz, rn * 8));
  CIP_CUDA(cudaMalloc(&dbad, sizeof(int)));
  cudaMemcpyAsync(dcp, rcp.data(), rcp.size() * 8, cudaMemcpyHostToDevice, s);
  cudaMemcpyAsync(drv, rrv.data(), rn * 8, cudaMemcpyHostToDevice, s);
  cudaMemcpyAsync(dnz, rnz.data(), rn * 8, cudaMemcpyHostToDevice, s);
  cudaMemsetAsync(dbad, 0, sizeof(int), s);
  const int r = scatter_csc_q4(rs.At4r, rs.nJ_pad, rs.nJ, dcp, drv, dnz, 0, 1, rs.nr, rn, dbad, s);
  const cudaError_t se = cudaStreamSynchronize(s);
  cudaFree(dcp); cudaFree(drv); cudaFree(dnz); cudaFree(dbad);
  CIP_TRY(r);
  CIP_CUDA(se);
  return 0;
}

int structure_finish(cip_engine* h) {
  RowStructure& rs = h->rs;
  cudaStream_t s = h->stream;
  rs.base_has_gtg = h->p > 0 && h->aug_rows > 0;
  if (rs.sp.on) {
    CIP_TRY(split_build(h));
  } else if (rs.base_has_gtg) {
    // Base4 = Q + (sqrt(rho) G)'(sqrt(rho) G): the aug rows leave the per-factor SYRK
    const size_t nn = (size_t)h->n_pad * h->n_pad;
    double* Gt4 = nullptr;
    CIP_CUDA(cudaMalloc(&Gt4, (size_t)h->aug_rows * h->n_pad * sizeof(double)));
    CIP_CUDA(cudaMemsetAsync(Gt4, 0, (size_t)h->aug_rows * h->n_pad * sizeof(double), s));
    CIP_TRY(salloc(h, &rs.Base4, nn));
    int rc = transpose_scale_q4(Gt4, h->n_pad, 0, h->G4, h->p_pad, h->p, h->n, sqrt(h->aug_rho), s);
    GemmOperand g{};
    if (rc == 0) rc = make_q4_tensor_map(&g.map, Gt4, h->n_pad, h->aug_rows / 4);
    if (rc == 0) {
      GemmArgs a{};
      a.lower = 1; a.ntm = a.ntn = h->n_pad / TILE; a.sym = 1; a.nk = h->aug_rows / 32;
      a.Cin = h->Qq4; a.Cout = rs.Base4; a.ldc = h->n_pad; a.alpha = 1.0;
      a.ws = h->gemm_ws; a.ws_doubles = GEMM_WS_DOUBLES;
      rc = launch_gemm_nt(g, g, a, s);
    }
    const cudaError_t se = cudaStreamSynchronize(s);
    cudaFree(Gt4);
    CIP_TRY(rc);
    CIP_CUDA(se);
  } else {
    rs.Base4 = h->Qq4;
  }
  if (rs.nJ > 0) {
    if (rs.fold) CIP_TRY(make_q4_tensor_map(&rs.map.map, rs.At4r, rs.nJ_pad, rs.nr_pad / 4));
    else CIP_TRY(make_q4_tensor_map(&rs.map.map, rs.Atil4r, rs.nJ_pad, rs.nr_pad / 4));
  }
  return 0;
}

int structure_form_H(cip_engine* h) {
  RowStructure& rs = h->rs;
  cudaStream_t s = h->stream;
  const int ncr = rs.cd.ncones;
  if (rs.nJ > 0) {
    gather_scaling_kernel<<<nb(std::max(rs.nr, ncr), 256), 256, 0, s>>>(h->Fi, rs.Fi, rs.rest_row, rs.nr,
                                                                       rs.cone_map, ncr);
    CIP_CHECK_LAUNCH();
    if (!rs.fold) CIP_TRY(cone_scale_panel(rs.cd, rs.Fi, rs.At4r, rs.Atil4r, rs.nJ_pad, rs.nr_pad, rs.nJ, s));
  }
  CIP_CUDA(cudaEventRecord(h->ev[1], s));
  // row_structure = 2 forms H_KK (J mapped to K positions) and h on D; the SYRK writes H directly when its columns
  // are all of H's (J == K, or J every column)
  RowStructure::Split& sp = rs.sp;
  double* H = sp.on ? sp.HK4 : h->H4;
  const int ldH = sp.on ? sp.nK_pad : h->n_pad;
  const double* base = sp.on ? sp.BaseK4 : rs.Base4;
  const int* Jmap = sp.on ? sp.JK : rs.J;
  const bool direct = sp.on ? rs.nJ == sp.nK : !rs.compressed;
  if (rs.nJ > 0) {
    GemmArgs a{};
    a.lower = 1; a.ntm = a.ntn = rs.nJ_pad / TILE; a.sym = 1; a.nk = rs.nr_pad / 32;
    a.Cin = direct ? base : nullptr;
    a.Cout = direct ? H : rs.Hr4;
    a.ldc = rs.nJ_pad; a.alpha = 1.0;
    a.ws = h->gemm_ws; a.ws_doubles = GEMM_WS_DOUBLES;
    if (rs.fold) a.kscale = rs.Fi.a;
    CIP_TRY(launch_gemm_nt(rs.map, rs.map, a, s));
  }
  if ((rs.nJ == 0 || !direct) && ldH > 0) CIP_TRY(vec_copy(H, base, (size_t)ldH * ldH, s));
  if (rs.nJ > 0 && !direct) {
    dim3 grid(nb(rs.nJ, 128), (unsigned)std::min(rs.nJ, 65535));
    scatter_gram_kernel<<<grid, 128, 0, s>>>(H, ldH, rs.Hr4, rs.nJ_pad, Jmap, rs.nJ);
    CIP_CHECK_LAUNCH();
  }
  if (sp.on) {
    CIP_TRY(vec_copy(sp.hD, sp.qD, h->n, s));
    sp.factored = false;
  }
  if (rs.nsing > 0) {
    singleton_diag_kernel<<<nb(h->n, 128), 128, 0, s>>>(H, ldH, h->n, rs.sing_ptr, rs.sing_row, rs.sing_val,
                                                        h->Fi.a, sp.on ? sp.Kpos : nullptr, sp.hD);
    CIP_CHECK_LAUNCH();
  }
  CIP_CUDA(cudaEventRecord(h->ev[2], s));
  h->st.syrk_flops = (double)rs.nr * (double)rs.nJ * (double)rs.nJ;
  return 0;
}

int structure_AT(cip_engine* h, double* out, const double* x, const double* add, int b) {
  RowStructure& rs = h->rs;
  cudaStream_t s = h->stream;
  if (rs.nJ > 0) {
    gather_vec_kernel<<<nb(rs.nr, 256), 256, 0, s>>>(rs.xr[b], x, rs.rest_row, rs.nr);
    CIP_CHECK_LAUNCH();
    CIP_TRY(q4_mv_rows(rs.outJ[b], rs.At4r, rs.nJ_pad, rs.nJ, rs.nr, rs.xr[b], h->partial, h->partial_cap, s));
  }
  finish_at_kernel<<<nb(h->n, 256), 256, 0, s>>>(out, add, rs.nJ > 0 ? rs.outJ[b] : nullptr, rs.Jinv, rs.sing_ptr,
                                                 rs.sing_row, rs.sing_val, x, h->n);
  CIP_CHECK_LAUNCH();
  return 0;
}

int structure_AT2(cip_engine* h, double* outa, double* outb, const double* xa, const double* xb, const double* adda,
                  const double* addb) {
  RowStructure& rs = h->rs;
  cudaStream_t s = h->stream;
  const double* xs[2] = {xa, xb};
  if (rs.nJ > 0) {
    for (int b = 0; b < 2; ++b) {
      gather_vec_kernel<<<nb(rs.nr, 256), 256, 0, s>>>(rs.xr[b], xs[b], rs.rest_row, rs.nr);
      CIP_CHECK_LAUNCH();
    }
    CIP_TRY(q4_mv_rows2(rs.outJ[0], rs.outJ[1], rs.At4r, rs.nJ_pad, rs.nJ, rs.nr, rs.xr[0], rs.xr[1], h->partial,
                        h->partial_cap, s));
  }
  double* outs[2] = {outa, outb};
  const double* adds[2] = {adda, addb};
  for (int b = 0; b < 2; ++b) {
    finish_at_kernel<<<nb(h->n, 256), 256, 0, s>>>(outs[b], adds[b], rs.nJ > 0 ? rs.outJ[b] : nullptr, rs.Jinv,
                                                   rs.sing_ptr, rs.sing_row, rs.sing_val, xs[b], h->n);
    CIP_CHECK_LAUNCH();
  }
  return 0;
}

namespace {
// y restricted to J (y itself when J is every column)
int gather_J(cip_engine* h, const double* y, int b, const double** out) {
  RowStructure& rs = h->rs;
  *out = y;
  if (!rs.compressed) return 0;
  gather_vec_kernel<<<nb(rs.nJ, 256), 256, 0, h->stream>>>(rs.yJ[b], y, rs.J, rs.nJ);
  CIP_CHECK_LAUNCH();
  *out = rs.yJ[b];
  return 0;
}
}  // namespace

int structure_A(cip_engine* h, double* out, const double* y, int b) {
  RowStructure& rs = h->rs;
  cudaStream_t s = h->stream;
  const double* outr = rs.nJ > 0 ? rs.outr[b] : nullptr;
  if (outr) {
    const double* yj;
    CIP_TRY(gather_J(h, y, b, &yj));
    CIP_TRY(q4_mv_k(rs.outr[b], rs.At4r, rs.nJ_pad, rs.nJ, rs.nr, yj, s));
  }
  finish_a_kernel<<<nb(h->m, 256), 256, 0, s>>>(out, outr, rs.row_code, rs.sing_col, rs.sing_val, y, h->m);
  CIP_CHECK_LAUNCH();
  return 0;
}

int structure_A2(cip_engine* h, double* outa, double* outb, const double* ya, const double* yb) {
  RowStructure& rs = h->rs;
  cudaStream_t s = h->stream;
  const bool rest = rs.nJ > 0;
  if (rest) {
    const double *ja, *jb;
    CIP_TRY(gather_J(h, ya, 0, &ja));
    CIP_TRY(gather_J(h, yb, 1, &jb));
    CIP_TRY(q4_mv_k2(rs.outr[0], rs.outr[1], rs.At4r, rs.nJ_pad, rs.nJ, rs.nr, ja, jb, s));
  }
  finish_a_kernel<<<nb(h->m, 256), 256, 0, s>>>(outa, rest ? rs.outr[0] : nullptr, rs.row_code, rs.sing_col, rs.sing_val, ya, h->m);
  CIP_CHECK_LAUNCH();
  finish_a_kernel<<<nb(h->m, 256), 256, 0, s>>>(outb, rest ? rs.outr[1] : nullptr, rs.row_code, rs.sing_col, rs.sing_val, yb, h->m);
  CIP_CHECK_LAUNCH();
  return 0;
}


// ================================================================ row_structure = 2: H split into D and K
// With the rows classified as above, column j of H = Q + (F^-T A)'(F^-T A) + rho G'G + delta I holds more than its
// diagonal only when a rest row touches it (j in J), when Q has an off-diagonal non-zero in row or column j, or when
// rho > 0 and G has a non-zero in column j.  Those columns are K (ascending); the others are D, where H_jj = h_j =
// Q_jj + the singleton sum + delta.  The Cholesky factor in natural column order is then sqrt(h_j) on D and the
// factor of the dense H_KK on K, with no permutation.  The Schur complement on G becomes
//   S = Sbase + G_D diag(1/h) G_D' + Z_K Z_K',   Z_K = G_K L_KK^-T,
// and a solve with H is u = rhs / h on D plus the two sweeps on K.  No n_pad^2 buffer survives cip_create; dense Q
// input is packed into a transient n_pad^2 staging copy, classified and gathered from it, then freed.
namespace {

// flagK[k] = 1 (and flagR[r] = 1) for every non-zero X[r, k], r < R, k < Kc; with flagR, diagonal entries are skipped
__global__ void mark_nz_kernel(const double* __restrict__ X, int ld, int R, int Kc, int* flagR, int* flagK) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  for (int k = blockIdx.y; k < Kc; k += gridDim.y) {
    if (flagR && r == k) continue;
    if (X[q4_index(r, k, ld)] != 0.0) {
      flagK[k] = 1;
      if (flagR) flagR[r] = 1;
    }
  }
}

__global__ void get_diag_kernel(double* __restrict__ d, const double* __restrict__ X, int ld, int n) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) d[j] = X[q4_index(j, j, ld)];
}

// Y[a, b] = X[rmap[a], cmap[b]] for a < R, b < Kc   (Q_KK from the staging Q; G_K from G4 with rmap = nullptr)
__global__ void gather_q4_kernel(double* __restrict__ Y, int ldy, const double* __restrict__ X, int ldx,
                                 const int* __restrict__ rmap, int R, const int* __restrict__ cmap, int Kc) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= R) return;
  const int ga = rmap ? rmap[a] : a;
  for (int b = blockIdx.y; b < Kc; b += gridDim.y) Y[q4_index(a, b, ldy)] = X[q4_index(ga, cmap[b], ldx)];
}

__global__ void shift_kernel(double* __restrict__ x, int n, double v) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) x[j] += v;
}

// the pivots of D: kscale_j = h_j^-1/2 on D, 0 on K and the padding; *fail = min over the D columns with
// h_j <= 0 or NaN
__global__ void split_pivots_kernel(double* __restrict__ kscale, const double* __restrict__ hD,
                                    const int* __restrict__ Kpos, int n, int n_pad, int* fail) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_pad) return;
  double ks = 0.0;
  if (j < n && Kpos[j] < 0) {
    const double hj = hD[j];
    if (hj > 0.0) ks = 1.0 / sqrt(hj);
    else atomicMin(fail, j);
  }
  kscale[j] = ks;
}

// rhsK[Kpos[j]] = rhs[j] on K; u = rhs / h on D, 0 on K
__global__ void split_rhs_kernel(double* __restrict__ rK, double* __restrict__ u, const double* __restrict__ rhs,
                                 const int* __restrict__ Kpos, const double* __restrict__ hD, int n) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int k = Kpos[j];
  if (k >= 0) {
    rK[k] = rhs[j];
    u[j] = 0.0;
  } else {
    u[j] = rhs[j] / hD[j];
  }
}

// dy = dyK on K; u - g / h on D (u without g)
__global__ void split_join_kernel(double* __restrict__ dy, const double* __restrict__ dyK,
                                  const double* __restrict__ u, const double* __restrict__ g,
                                  const int* __restrict__ Kpos, const double* __restrict__ hD, int n) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int k = Kpos[j];
  dy[j] = k >= 0 ? dyK[k] : (g ? u[j] - g[j] / hD[j] : u[j]);
}

// y = yK on K, d .* x on D
__global__ void diag_join_kernel(double* __restrict__ y, const double* __restrict__ yK, const double* __restrict__ d,
                                 const double* __restrict__ x, const int* __restrict__ Kpos, int n) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int k = Kpos[j];
  y[j] = k >= 0 ? yK[k] : d[j] * x[j];
}

// out (n x n, column-major) = H_KK (or L_KK) at K x K, h_j (or sqrt(h_j)) on the diagonal of D, 0 elsewhere
__global__ void split_unpack_kernel(double* __restrict__ out, int n, const double* __restrict__ HK4, int ldk,
                                    const int* __restrict__ Kpos, const double* __restrict__ hD, int factored) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int a = Kpos[r];
  for (int c = blockIdx.y; c < n; c += gridDim.y) {
    const int b = Kpos[c];
    double v = 0.0;
    if (a >= 0 && b >= 0) v = HK4[q4_index(a, b, ldk)];
    else if (r == c) v = factored ? sqrt(hD[r]) : hD[r];
    out[r + (size_t)c * n] = v;
  }
}

int count(const std::vector<char>& f) {
  int c = 0;
  for (char x : f) c += x != 0;
  return c;
}

// flags of a Q4 matrix on the device (see mark_nz_kernel) copied to the host
int mark_nz(cip_engine* h, const double* X, int ld, int R, int Kc, bool sym, std::vector<char>* out) {
  cudaStream_t s = h->stream;
  int* d = nullptr;
  CIP_CUDA(cudaMalloc(&d, sizeof(int) * std::max(Kc, 1)));
  CIP_CUDA(cudaMemsetAsync(d, 0, sizeof(int) * std::max(Kc, 1), s));
  dim3 grid(nb(R, 128), (unsigned)std::min(std::max(Kc, 1), 65535));
  mark_nz_kernel<<<grid, 128, 0, s>>>(X, ld, R, Kc, sym ? d : nullptr, d);
  const cudaError_t le = cudaGetLastError();
  g_launches++;
  std::vector<int> f(Kc);
  cudaMemcpyAsync(f.data(), d, sizeof(int) * Kc, cudaMemcpyDeviceToHost, s);
  const cudaError_t se = cudaStreamSynchronize(s);
  cudaFree(d);
  CIP_CUDA(le);
  CIP_CUDA(se);
  out->assign(f.begin(), f.end());
  return 0;
}

}  // namespace

int split_classify_csc_Q(cip_engine* h, const cip_csc* Q) {
  RowStructure::Split& sp = h->rs.sp;
  const int n = h->n;
  std::vector<E> ent;
  CIP_TRY(read_csc(Q, n, &ent));
  sp.q_couple.assign(n, 0);
  std::vector<double> qd(n, 0.0);
  for (const E& e : ent) {
    if (e.i == e.j) {
      qd[e.j] = e.v;
    } else {
      sp.q_couple[e.i] = 1;
      sp.q_couple[e.j] = 1;
    }
  }
  CIP_TRY(salloc(h, &sp.qD, (size_t)h->n_pad + 4));
  CIP_CUDA(cudaMemcpyAsync(sp.qD, qd.data(), sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
  CIP_CUDA(cudaStreamSynchronize(h->stream));
  // Q_KK is scattered from these once K is known (K also holds columns Q does not couple: their diagonal is needed)
  sp.qtrip.clear();
  for (const E& e : ent)
    if (e.i == e.j || (sp.q_couple[e.i] && sp.q_couple[e.j])) sp.qtrip.push_back({e.i, e.j, e.v});
  return 0;
}

int split_diag_Q(cip_engine* h, const double* q) {
  RowStructure::Split& sp = h->rs.sp;
  sp.q_couple.assign(h->n, 0);
  CIP_TRY(salloc(h, &sp.qD, (size_t)h->n_pad + 4));
  if (q) {
    CIP_CUDA(cudaMemcpyAsync(sp.qD, q, sizeof(double) * h->n, cudaMemcpyDefault, h->stream));
    CIP_CUDA(cudaStreamSynchronize(h->stream));
  }
  return 0;
}

int split_build(cip_engine* h) {
  RowStructure& rs = h->rs;
  RowStructure::Split& sp = rs.sp;
  cudaStream_t s = h->stream;
  const int n = h->n, p = h->p;
  // ---- K
  std::vector<char> inK(n, 0);
  std::vector<int> J(rs.nJ);
  if (rs.nJ > 0) CIP_CUDA(cudaMemcpy(J.data(), rs.J, sizeof(int) * rs.nJ, cudaMemcpyDeviceToHost));
  for (int j : J) inK[j] = 1;
  sp.from_rest = rs.nJ;
  if (h->Qq4) {       // dense Q: classified from the staging copy
    CIP_TRY(mark_nz(h, h->Qq4, h->n_pad, n, n, true, &sp.q_couple));
    CIP_TRY(salloc(h, &sp.qD, (size_t)h->n_pad + 4));
    get_diag_kernel<<<nb(n, 256), 256, 0, s>>>(sp.qD, h->Qq4, h->n_pad, n);
    CIP_CHECK_LAUNCH();
  }
  if (sp.q_couple.empty()) sp.q_couple.assign(n, 0);
  if (!sp.qD) CIP_TRY(salloc(h, &sp.qD, (size_t)h->n_pad + 4));      // no Q
  sp.from_Q = count(sp.q_couple);
  for (int j = 0; j < n; ++j) inK[j] |= sp.q_couple[j];
  std::vector<char> gcol(n, 0);
  if (p > 0) CIP_TRY(mark_nz(h, h->G4, h->p_pad, p, n, false, &gcol));
  if (h->aug_rows > 0) {
    sp.from_G = count(gcol);
    for (int j = 0; j < n; ++j) inK[j] |= gcol[j];
  }
  sp.K.clear();
  std::vector<int> Kpos(n, -1);
  sp.g_in_D = false;
  for (int j = 0; j < n; ++j) {
    if (inK[j]) {
      Kpos[j] = (int)sp.K.size();
      sp.K.push_back(j);
    } else if (gcol[j]) {
      sp.g_in_D = true;
    }
  }
  sp.nK = (int)sp.K.size();
  sp.nK_pad = round_up(sp.nK, TILE);
  std::vector<int> JK(rs.nJ);
  for (int a = 0; a < rs.nJ; ++a) JK[a] = Kpos[J[a]];
  CIP_TRY(supload(h, &sp.dK, sp.K));
  CIP_TRY(supload(h, &sp.Kpos, Kpos));
  CIP_TRY(supload(h, &sp.JK, JK));
  CIP_TRY(salloc(h, &sp.hD, (size_t)h->n_pad + 4));
  CIP_TRY(salloc(h, &sp.kscale, (size_t)h->n_pad + 4));
  CIP_TRY(salloc(h, &sp.fail, 1));
  if (p > 0) CIP_TRY(make_q4_tensor_map(&sp.mapG.map, h->G4, h->p_pad, h->n_pad / 4));
  const int nK = sp.nK, nKp = sp.nK_pad;
  if (nK > 0) {
    // ---- Q_KK (both triangles, identity on the padding)
    const size_t kk = (size_t)nKp * nKp;
    CIP_TRY(salloc(h, &sp.QK4, kk));
    if (h->Qq4) {
      dim3 grid(nb(nK, 128), (unsigned)std::min(nK, 65535));
      gather_q4_kernel<<<grid, 128, 0, s>>>(sp.QK4, nKp, h->Qq4, h->n_pad, sp.dK, nK, sp.dK, nK);
      CIP_CHECK_LAUNCH();
    } else if (!sp.qtrip.empty()) {
      // CSC Q: the summed entries of K x K as a CSC matrix over K positions
      std::vector<long long> cp(nK + 1, 0), rv;
      std::vector<double> nz;
      for (const auto& e : sp.qtrip)
        if (Kpos[e.i] >= 0 && Kpos[e.j] >= 0) cp[Kpos[e.j] + 1]++;
      for (int a = 0; a < nK; ++a) cp[a + 1] += cp[a];
      rv.resize(cp[nK]);
      nz.resize(cp[nK]);
      std::vector<long long> pos(cp.begin(), cp.end() - 1);
      for (const auto& e : sp.qtrip) {
        if (Kpos[e.i] < 0 || Kpos[e.j] < 0) continue;
        const long long at = pos[Kpos[e.j]]++;
        rv[at] = Kpos[e.i];
        nz[at] = e.v;
      }
      const long long nnz = (long long)rv.size();
      if (nnz > 0) {
        long long *dcp = nullptr, *drv = nullptr;
        double* dnz = nullptr;
        int* dbad = nullptr;
        CIP_CUDA(cudaMalloc(&dcp, cp.size() * 8));
        CIP_CUDA(cudaMalloc(&drv, nnz * 8));
        CIP_CUDA(cudaMalloc(&dnz, nnz * 8));
        CIP_CUDA(cudaMalloc(&dbad, sizeof(int)));
        cudaMemcpyAsync(dcp, cp.data(), cp.size() * 8, cudaMemcpyHostToDevice, s);
        cudaMemcpyAsync(drv, rv.data(), nnz * 8, cudaMemcpyHostToDevice, s);
        cudaMemcpyAsync(dnz, nz.data(), nnz * 8, cudaMemcpyHostToDevice, s);
        cudaMemsetAsync(dbad, 0, sizeof(int), s);
        const int r = scatter_csc_q4(sp.QK4, nKp, nK, dcp, drv, dnz, 0, 0, nK, nnz, dbad, s);
        const cudaError_t se = cudaStreamSynchronize(s);
        cudaFree(dcp); cudaFree(drv); cudaFree(dnz); cudaFree(dbad);
        CIP_TRY(r);
        CIP_CUDA(se);
      }
    } else {
      // diagonal or no Q: Q_KK is the diagonal of Q on K
      double* t = nullptr;
      CIP_CUDA(cudaMalloc(&t, sizeof(double) * nK));
      gather_vec_kernel<<<nb(nK, 256), 256, 0, s>>>(t, sp.qD, sp.dK, nK);
      const cudaError_t le = cudaGetLastError();
      g_launches++;
      const int r = le == cudaSuccess ? set_diag_vec_q4(sp.QK4, nKp, nK, t, s) : 0;
      const cudaError_t se = cudaStreamSynchronize(s);
      cudaFree(t);
      CIP_CUDA(le);
      CIP_TRY(r);
      CIP_CUDA(se);
    }
    CIP_TRY(add_diag_q4(sp.QK4, nKp, nK, nKp, 1.0, 1, s));
    // ---- G_K and BaseK4 = Q_KK + rho G_K'G_K
    if (p > 0) {
      CIP_TRY(salloc(h, &sp.GK4, (size_t)h->p_pad * nKp));
      dim3 grid(nb(p, 128), (unsigned)std::min(nK, 65535));
      gather_q4_kernel<<<grid, 128, 0, s>>>(sp.GK4, h->p_pad, h->G4, h->p_pad, nullptr, p, sp.dK, nK);
      CIP_CHECK_LAUNCH();
      CIP_TRY(salloc(h, &sp.ZK4, (size_t)h->p_pad * nKp));
      CIP_TRY(make_q4_tensor_map(&sp.mapZK.map, sp.ZK4, h->p_pad, nKp / 4));
    }
    if (rs.base_has_gtg) {
      double* Gt4 = nullptr;
      CIP_CUDA(cudaMalloc(&Gt4, (size_t)h->aug_rows * nKp * sizeof(double)));
      CIP_CUDA(cudaMemsetAsync(Gt4, 0, (size_t)h->aug_rows * nKp * sizeof(double), s));
      CIP_TRY(salloc(h, &sp.BaseK4, kk));
      int rc = transpose_scale_q4(Gt4, nKp, 0, sp.GK4, h->p_pad, p, nK, sqrt(h->aug_rho), s);
      GemmOperand g{};
      if (rc == 0) rc = make_q4_tensor_map(&g.map, Gt4, nKp, h->aug_rows / 4);
      if (rc == 0) {
        GemmArgs a{};
        a.lower = 1; a.ntm = a.ntn = nKp / TILE; a.sym = 1; a.nk = h->aug_rows / 32;
        a.Cin = sp.QK4; a.Cout = sp.BaseK4; a.ldc = nKp; a.alpha = 1.0;
        a.ws = h->gemm_ws; a.ws_doubles = GEMM_WS_DOUBLES;
        rc = launch_gemm_nt(g, g, a, s);
      }
      const cudaError_t se = cudaStreamSynchronize(s);
      cudaFree(Gt4);
      CIP_TRY(rc);
      CIP_CUDA(se);
    } else {
      sp.BaseK4 = sp.QK4;
    }
    // ---- H_KK and its Cholesky plan
    CIP_TRY(salloc(h, &sp.HK4, kk));
    CIP_TRY(salloc(h, &sp.WinvK, (size_t)nKp * TILE));
    CIP_TRY(chol_make_plan(&sp.chol, sp.HK4, nKp, sp.WinvK, h->info));
    for (int b = 0; b < 2; ++b)
      for (auto& v : sp.kv[b]) CIP_TRY(salloc(h, &v, (size_t)nKp + 4));
  }
  sp.qtrip.clear();
  sp.qtrip.shrink_to_fit();
  // the Gram scratch is not needed when the SYRK writes H_KK directly (J == K)
  if (rs.Hr4 && rs.nJ == nK) {
    CIP_CUDA(cudaStreamSynchronize(s));
    cudaFree(rs.Hr4);
    h->owned.erase(std::find(h->owned.begin(), h->owned.end(), (void*)rs.Hr4));
    h->bytes -= std::max<size_t>((size_t)rs.nJ_pad * rs.nJ_pad, 1) * sizeof(double);
    rs.Hr4 = nullptr;
  }
  if (h->Qq4) {       // the dense staging copy of Q
    CIP_CUDA(cudaStreamSynchronize(s));
    cudaFree(h->Qq4);
    h->Qq4 = nullptr;
    h->bytes -= (size_t)h->n_pad * h->n_pad * sizeof(double);
  }
  return 0;
}

int split_add_delta(cip_engine* h, double delta) {
  RowStructure::Split& sp = h->rs.sp;
  if (sp.nK > 0) CIP_TRY(add_diag_q4(sp.HK4, sp.nK_pad, 0, sp.nK, delta, 0, h->stream));
  shift_kernel<<<nb(h->n, 256), 256, 0, h->stream>>>(sp.hD, h->n, delta);
  CIP_CHECK_LAUNCH();
  return 0;
}

int split_factor(cip_engine* h) {
  RowStructure::Split& sp = h->rs.sp;
  cudaStream_t s = h->stream;
  CIP_CUDA(cudaMemsetAsync(sp.fail, 0x7f, sizeof(int), s));     // 0x7f7f7f7f: no failing D column
  if (sp.nK > 0) CIP_TRY(chol_factor(sp.chol, s));
  split_pivots_kernel<<<nb(h->n_pad, 256), 256, 0, s>>>(sp.kscale, sp.hD, sp.Kpos, h->n, h->n_pad, sp.fail);
  CIP_CHECK_LAUNCH();
  sp.factored = true;
  return 0;
}

int split_solve(cip_engine* h, double** nv, double** pv, int b, bool schur) {
  RowStructure::Split& sp = h->rs.sp;
  cudaStream_t s = h->stream;
  const int n = h->n, p = h->p, nK = sp.nK;
  double *rK = sp.kv[b][0], *tK = sp.kv[b][1], *wK = sp.kv[b][2];
  double* u = nv[3];
  split_rhs_kernel<<<nb(n, 256), 256, 0, s>>>(rK, u, nv[2], sp.Kpos, sp.hD, n);
  CIP_CHECK_LAUNCH();
  if (nK > 0) CIP_TRY(chol_fwd(sp.chol, rK, tK, s));
  const double* g = nullptr;
  if (schur) {
    // r = G u + Z_K t_K - rw;  dw = S^-1 r;  t_K -= Z_K' dw;  g = G' dw
    if (nK > 0) CIP_TRY(q4_mv_rows(pv[1], sp.ZK4, h->p_pad, p, nK, tK, h->partial, h->partial_cap, s));
    else CIP_TRY(fill_zero(pv[1], p, s));
    if (sp.g_in_D) {
      CIP_TRY(q4_mv_rows(pv[3], h->G4, h->p_pad, p, n, u, h->partial, h->partial_cap, s));
      CIP_TRY(vec_axpby(pv[1], 1.0, pv[1], 1.0, pv[3], p, s));
    }
    CIP_TRY(vec_axpby(pv[2], 1.0, pv[1], -1.0, pv[0], p, s));
    CIP_TRY(chol_fwd(h->cholS, pv[2], pv[3], s));
    CIP_TRY(chol_bwd(h->cholS, pv[3], pv[4], s));
    if (nK > 0) {
      CIP_TRY(q4_mv_k(wK, sp.ZK4, h->p_pad, p, nK, pv[4], s));
      CIP_TRY(vec_axpby(tK, 1.0, tK, -1.0, wK, nK, s));
    }
    if (sp.g_in_D) {
      CIP_TRY(q4_mv_k(nv[4], h->G4, h->p_pad, p, n, pv[4], s));
      g = nv[4];
    }
  }
  if (nK > 0) CIP_TRY(chol_bwd(sp.chol, tK, rK, s));
  split_join_kernel<<<nb(n, 256), 256, 0, s>>>(nv[5], rK, u, g, sp.Kpos, sp.hD, n);
  CIP_CHECK_LAUNCH();
  return 0;
}

int split_mul_Q(cip_engine* h, double* y, const double* x) {
  RowStructure::Split& sp = h->rs.sp;
  cudaStream_t s = h->stream;
  const int nK = sp.nK;
  if (nK > 0) {
    gather_vec_kernel<<<nb(nK, 256), 256, 0, s>>>(sp.kv[0][0], x, sp.dK, nK);
    CIP_CHECK_LAUNCH();
    CIP_TRY(q4_mv_rows(sp.kv[0][1], sp.QK4, sp.nK_pad, nK, nK, sp.kv[0][0], h->partial, h->partial_cap, s));
  }
  diag_join_kernel<<<nb(h->n, 256), 256, 0, s>>>(y, sp.kv[0][1], sp.qD, x, sp.Kpos, h->n);
  CIP_CHECK_LAUNCH();
  return 0;
}

int split_get_H(cip_engine* h, double* out) {
  RowStructure::Split& sp = h->rs.sp;
  dim3 grid(nb(h->n, 128), (unsigned)std::min(h->n, 65535));
  split_unpack_kernel<<<grid, 128, 0, h->stream>>>(out, h->n, sp.HK4, sp.nK_pad, sp.Kpos, sp.hD, sp.factored);
  CIP_CHECK_LAUNCH();
  return 0;
}

}  // namespace cip
