// cip_options.eliminate_y: the m-space form of the KKT system.
//
// With D = Q + delta I diagonal and positive, cip_solve's system
//     Q a + G'b - A'c = ry ;  G a = rw ;  A a + F'F c = rv
// is reduced by eliminating a = D^-1 (ry - G'b + A'c):
//     M c - E b = r1,  E'c - P b = r2,      M = F'F + C,  C = A D^-1 A',  E = A D^-1 G',  P = G D^-1 G',
//     r1 = rv - A D^-1 ry,  r2 = rw - G D^-1 ry.
// M = L L', Z = E' L^-T (p x m), S = P - Z Z' (= G H^-1 G'), t = L^-1 r1:
//     b = S^-1 (Z t - r2),  c = L^-T (t + Z'b),  a = D^-1 (ry - G'b + A'c).
// C, E' and P are constant (formed once at cip_create on the DMMA tiles, gemm_nt with kscale = D^-1/2 on the
// contraction); each factorisation adds the block-diagonal F'F to C (ey_assemble_kernel), factors the m x m M and the
// p x p S.  A is kept once, as A4 (rows = rows of A, k = columns): A x is q4_mv_rows, A'x is q4_mv_k.
#include <climits>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "engine.h"

namespace cip {
namespace {

#define EY_SQRT1_2 0.70710678118654752440

int ey_alloc(cip_engine* h, double** p, size_t count) {
  *p = nullptr;
  if (count == 0) count = 1;
  CIP_CUDA(cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(double)));
  h->owned.push_back(*p);
  CIP_CUDA(cudaMemsetAsync(*p, 0, count * sizeof(double), h->stream));
  h->bytes += count * sizeof(double);
  return 0;
}

bool ey_kernel_readable(const void* p, int device) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeManaged || (at.type == cudaMemoryTypeDevice && at.device == device);
}

// ---------------------------------------------------------------- kernels
// diag[c0 + j] = Q[c0 + j, c0 + j] for the nc columns of a chunk (column j of the chunk at src + j * lds); *bad =
// the smallest column with an off-diagonal non-zero (atomicMin, INT_MAX when none)
__global__ void ey_dense_q_kernel(const double* __restrict__ src, int lds, int n, int c0, double* __restrict__ diag,
                                  int* bad) {
  const int j = c0 + blockIdx.x;
  const double* col = src + (size_t)blockIdx.x * lds;
  bool off = false;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double v = col[i];
    if (i == j) diag[j] = v;
    else off |= (v != 0.0);
  }
  if (__syncthreads_or(off) && threadIdx.x == 0) atomicMin(bad, j);
}

// out = d .* (x - y + z), y and z optional (null: 0)
__global__ void ey_dscale_kernel(double* __restrict__ out, const double* __restrict__ d, const double* __restrict__ x,
                                 const double* __restrict__ y, const double* __restrict__ z, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    double v = x[i];
    if (y) v -= y[i];
    if (z) v += z[i];
    out[i] = d[i] * v;
  }
}

// b'b of every Q cone with a Woodbury block (one CTA per Q cone; fixed reduction order)
__global__ void __launch_bounds__(256) ey_qbb_kernel(const int* __restrict__ qlist, const int* __restrict__ off,
                                                     const int* __restrict__ kind, const double* __restrict__ b,
                                                     double* __restrict__ bb) {
  __shared__ double red[256];
  const int c = qlist[blockIdx.x];
  double s = 0.0;
  if (kind[c] == CIP_BLK_WOODBURY)
    for (int r = off[c] + threadIdx.x; r < off[c + 1]; r += 256) s = fma(b[r], b[r], s);
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) bb[c] = red[0];
}

// W = R R' of every S cone with a VecCongurance block (one CTA per S cone; R column-major k x k)
__global__ void __launch_bounds__(256) ey_w_kernel(const int* __restrict__ slist, const int* __restrict__ sord,
                                                   const int* __restrict__ roff, const int* __restrict__ kind,
                                                   const double* __restrict__ R, double* __restrict__ W) {
  const int si = blockIdx.x;
  if (kind[slist[si]] != CIP_BLK_VECCONG) return;
  const int k = sord[si];
  const double* Rs = R + roff[si];
  double* Ws = W + roff[si];
  for (int e = threadIdx.x; e < k * k; e += 256) {
    const int i = e % k, j = e / k;
    double s = 0.0;
    for (int l = 0; l < k; ++l) s = fma(Rs[i + (size_t)l * k], Rs[j + (size_t)l * k], s);
    Ws[e] = s;
  }
}

// svec index (row-major upper triangle of a k x k matrix, sdp.cu) -> (i, j), i <= j
__device__ __forceinline__ void svec_pair(int a, int k, int& i, int& j) {
  i = 0;
  while (a >= k - i) { a -= k - i; ++i; }
  j = i + a;
}

struct AssembleArgs {
  const double* C;
  double* M;
  int ld, m;
  const int *row_cone, *type, *off, *sidx, *sord, *roff;
  const int* kind;
  const double *a, *b, *D, *bb, *W;
};

// M = C + F'F on the lower tiles of the Q4 buffer (ld = mM), identity on the padding.  F'F per cone:
//   DIAG (R rows, and every cone at F = I):  diag(a^2)
//   Woodbury, F = diag(a) + D b b':           diag(a^2) + D (a.*b) b' + D b (a.*b)' + D^2 (b'b) b b'
//   VecCongurance, F x = vecm(R' mat(x) R):   F'F x = vecm(W mat(x) W), W = R R'; in the svec basis the entry
//       of (i,j), (p,q) is k_ij k_pq (W_ip W_jq + W_iq W_jp), k = 1 off the diagonal and 1/sqrt(2) on it
__global__ void __launch_bounds__(256) ey_assemble_kernel(const AssembleArgs g) {
  const size_t total = (size_t)g.ld * g.ld;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const int t = (int)(e & 3);
    const size_t rq = e >> 2;
    const int r = (int)(rq % g.ld), k = (int)(rq / g.ld) * 4 + t;
    if (r / TILE < k / TILE) continue;                      // upper tiles: not part of the factorisation
    double v = g.C[e];
    if (r >= g.m || k >= g.m) {
      g.M[e] = (r == k) ? 1.0 : v;
      continue;
    }
    const int c = g.row_cone[r];
    if (c == g.row_cone[k]) {
      const int kd = g.kind[c];
      if (kd == CIP_BLK_DIAG) {
        if (r == k) v += g.a[r] * g.a[r];
      } else if (kd == CIP_BLK_WOODBURY) {
        const double D = g.D[c], br = g.b[r], bk = g.b[k];
        double f = D * (g.a[r] * br * bk + br * g.a[k] * bk) + D * D * g.bb[c] * br * bk;
        if (r == k) f += g.a[r] * g.a[r];
        v += f;
      } else {
        const int si = g.sidx[c], ko = g.sord[si];
        const double* W = g.W + g.roff[si];
        int i, j, p, q;
        svec_pair(r - g.off[c], ko, i, j);
        svec_pair(k - g.off[c], ko, p, q);
        const double w = W[i + p * ko] * W[j + q * ko] + W[i + q * ko] * W[j + p * ko];
        const double ka = (i == j) ? EY_SQRT1_2 : 1.0, kb = (p == q) ? EY_SQRT1_2 : 1.0;
        v += (ka * kb) * w;
      }
    }
    g.M[e] = v;
  }
}

int grid_for(size_t n, int threads = 256) {
  const size_t b = (n + threads - 1) / threads;
  const size_t cap = (size_t)sm_count() * 16;
  return (int)std::max<size_t>(1, std::min(b, cap));
}

int dscale(double* out, const double* d, const double* x, const double* y, const double* z, int n, cudaStream_t s) {
  if (n <= 0) return 0;
  ey_dscale_kernel<<<grid_for(n), 256, 0, s>>>(out, d, x, y, z, n);
  CIP_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------- LEVEL 1 helpers
// the diagonal of Q into h->ey.hq (host); false (with the message set) when Q has an off-diagonal non-zero
int classify_q(cip_engine* h, const double* Q, int ldq, const cip_csc* Qs, bool* diagonal) {
  const int n = h->n;
  std::vector<double>& q = h->ey.hq;
  q.assign(n, 0.0);
  *diagonal = true;
  if (Qs) {
    if (Qs->ncols == 0) return 0;
    std::vector<long long> cp(Qs->ncols + 1);
    CIP_CUDA(cudaMemcpy(cp.data(), Qs->colptr, cp.size() * 8, cudaMemcpyDefault));
    const long long nnz = cp[Qs->ncols] - cp[0];
    std::vector<long long> rv(std::max(nnz, 1LL));
    std::vector<double> nz(std::max(nnz, 1LL));
    if (nnz > 0) {
      CIP_CUDA(cudaMemcpy(rv.data(), Qs->rowval, nnz * 8, cudaMemcpyDefault));
      CIP_CUDA(cudaMemcpy(nz.data(), Qs->nzval, nnz * 8, cudaMemcpyDefault));
    }
    for (int j = 0; j < Qs->ncols; ++j)
      for (long long e = cp[j] - cp[0]; e < cp[j + 1] - cp[0]; ++e) {
        const long long i = rv[e] - Qs->index_base;
        if (i == j) q[j] += nz[e];
        else if (nz[e] != 0.0) {
          set_error("eliminate_y: Q has an off-diagonal non-zero at (%lld, %d); the m-space form needs a diagonal Q",
                    i, j);
          *diagonal = false;
          return 0;
        }
      }
    return 0;
  }
  if (h->opt.q_kind == 2) return 0;
  if (!Q) { set_error("Q is null"); return -1; }
  if (h->opt.q_kind == 1) {
    CIP_CUDA(cudaMemcpy(q.data(), Q, (size_t)n * 8, cudaMemcpyDefault));
    return 0;
  }
  // dense: one pass over the columns (through a staging buffer when the kernel cannot read Q where it is)
  cudaStream_t s = h->stream;
  double* dq = nullptr;
  int* dbad = nullptr;
  CIP_CUDA(cudaMalloc(&dq, (size_t)n * 8));
  CIP_CUDA(cudaMalloc(&dbad, sizeof(int)));
  const int big = INT_MAX;
  CIP_CUDA(cudaMemcpyAsync(dbad, &big, sizeof(int), cudaMemcpyHostToDevice, s));
  int rc = 0;
  if (ey_kernel_readable(Q, h->device)) {
    ey_dense_q_kernel<<<n, 256, 0, s>>>(Q, ldq, n, 0, dq, dbad);
    g_launches++;
    if (cudaGetLastError() != cudaSuccess) rc = -1;
  } else {
    const int chunk = std::max(1, std::min(n, (int)((256u << 20) / ((size_t)n * 8))));
    double* stg = nullptr;
    if (cudaMalloc(&stg, (size_t)n * chunk * 8) != cudaSuccess) rc = -1;
    for (int c0 = 0; c0 < n && rc == 0; c0 += chunk) {
      const int nc = std::min(chunk, n - c0);
      if (cudaMemcpy2DAsync(stg, (size_t)n * 8, Q + (size_t)c0 * ldq, (size_t)ldq * 8, (size_t)n * 8, nc,
                            cudaMemcpyDefault, s) != cudaSuccess) rc = -1;
      ey_dense_q_kernel<<<nc, 256, 0, s>>>(stg, n, n, c0, dq, dbad);
      g_launches++;
      if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) rc = -1;
    }
    if (stg) cudaFree(stg);
  }
  int bad = big;
  if (rc == 0) {
    cudaMemcpyAsync(q.data(), dq, (size_t)n * 8, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(&bad, dbad, sizeof(int), cudaMemcpyDeviceToHost, s);
    if (cudaStreamSynchronize(s) != cudaSuccess) rc = -1;
  }
  cudaFree(dq);
  cudaFree(dbad);
  if (rc != 0) { set_error("eliminate_y: classifying the dense Q failed (%s)", cudaGetErrorString(cudaGetLastError())); return -1; }
  if (bad != big) {
    set_error("eliminate_y: Q has an off-diagonal non-zero in column %d; the m-space form needs a diagonal Q", bad);
    *diagonal = false;
  }
  return 0;
}

}  // namespace

int ey_decide(cip_engine* h, bool shard, const double* Q, int ldq, const cip_csc* Qs) {
  EliminateY& ey = h->ey;
  const int mode = h->opt.eliminate_y;
  if (mode != 0 && mode != 1 && mode != 2) {
    set_error("cip_create: eliminate_y must be 0, 1 or 2 (got %d)", mode);
    return -1;
  }
  if (mode == 2) return 0;
  // structural conditions
  const char* why = nullptr;
  if (shard) why = "it is supported on single-device handles only (ngpus > 1)";
  else if (h->rs.on) why = "it cannot be combined with row_structure";
  else if (h->m == 0) why = "A has no rows";
  if (why) {
    if (mode == 1) { set_error("eliminate_y = 1: %s", why); return -1; }
    return 0;
  }
  if (mode == 0) {
    // auto: only when the n-space form, after its own fold decision, would not fit in free device memory
    // (the sizes create_body allocates for it, with engine_decide_fold's margin of 1 GB)
    size_t free_b = 0, total_b = 0;
    CIP_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const size_t n_pad = h->n_pad, nn = n_pad * n_pad;
    const size_t k_rows = (size_t)h->m_pad + (h->qs > 0 ? h->aug_rows : 0);
    size_t need = k_rows * n_pad + 2 * nn + n_pad * TILE + (size_t)GEMM_WS_DOUBLES;   // At4, Qq4, H4, Winv, ws
    if (!h->fold) need += (size_t)(h->m_pad + h->aug_rows) * n_pad;                   // Atil4
    if (h->p > 0) need += 2 * (size_t)h->p_pad * n_pad;                               // G4, Z4
    need = need * sizeof(double) + (size_t(1) << 30);
    if (free_b >= need) return 0;
  }
  bool diagonal = true;
  CIP_TRY(classify_q(h, Q, ldq, Qs, &diagonal));
  if (!diagonal) {
    if (mode == 1) return -1;              // (classify_q set the message)
    return 0;
  }
  const double delta = h->opt.reg_delta;
  for (int j = 0; j < h->n; ++j)
    if (!(ey.hq[j] + delta > 0.0)) {
      if (mode == 1) {
        set_error("eliminate_y = 1: Q_jj + reg_delta = %g at column %d; the m-space form needs Q + reg_delta I > 0",
                  ey.hq[j] + delta, j);
        return -1;
      }
      return 0;
    }
  ey.on = true;
  ey.automatic = (mode == 0);
  return 0;
}

int ey_create(cip_engine* h, const double* A, int lda, const cip_csc* As, const double* G, int ldg,
              const cip_csc* Gs) {
  (void)G; (void)ldg; (void)Gs;            // G4 is uploaded by create_body
  EliminateY& ey = h->ey;
  cudaStream_t s = h->stream;
  const int n = h->n, m = h->m, p = h->p, n_pad = h->n_pad;
  ey.mM = round_up(m, TILE);
  const int mM = ey.mM;
  // D, D^-1, D^-1/2 (zero on the padding: padded columns contribute nothing) and Q's diagonal
  {
    std::vector<double> dinv(n_pad, 0.0), ks(n_pad, 0.0);
    for (int j = 0; j < n; ++j) {
      const double d = ey.hq[j] + h->opt.reg_delta;
      dinv[j] = 1.0 / d;
      ks[j] = 1.0 / sqrt(d);
    }
    CIP_TRY(ey_alloc(h, &ey.dinv, n_pad + 4));
    CIP_TRY(ey_alloc(h, &ey.kscale, n_pad + 4));
    CIP_TRY(ey_alloc(h, &ey.qdiag, n_pad + 4));
    CIP_CUDA(cudaMemcpyAsync(ey.dinv, dinv.data(), (size_t)n_pad * 8, cudaMemcpyHostToDevice, s));
    CIP_CUDA(cudaMemcpyAsync(ey.kscale, ks.data(), (size_t)n_pad * 8, cudaMemcpyHostToDevice, s));
    CIP_CUDA(cudaMemcpyAsync(ey.qdiag, ey.hq.data(), (size_t)n * 8, cudaMemcpyHostToDevice, s));
    CIP_CUDA(cudaStreamSynchronize(s));
    std::vector<double>().swap(ey.hq);
  }
  // A4: rows = rows of A, k = columns
  CIP_TRY(ey_alloc(h, &ey.A4, (size_t)mM * n_pad));
  if (As) {
    CIP_TRY(engine_upload_csc(h, ey.A4, mM, As, 0));
  } else if (ey_kernel_readable(A, h->device)) {
    CIP_TRY(pack_rows_q4(ey.A4, mM, A, lda, m, n, mM, n_pad, s));
  } else {
    // column chunks (a multiple of 4) through a staging buffer
    const int chunk = std::max(4, std::min(round_up(n, 4), (int)((512u << 20) / ((size_t)m * 8)) / 4 * 4));
    double* stg = nullptr;
    CIP_CUDA(cudaMalloc(&stg, (size_t)m * chunk * 8));
    for (int c0 = 0; c0 < n; c0 += chunk) {
      const int nc = std::min(chunk, n - c0);
      CIP_CUDA(cudaMemcpy2DAsync(stg, (size_t)m * 8, A + (size_t)c0 * lda, (size_t)lda * 8, (size_t)m * 8, nc,
                                 cudaMemcpyDefault, s));
      CIP_TRY(pack_rows_q4(ey.A4 + (size_t)(c0 / 4) * mM * 4, mM, stg, m, m, nc, mM, round_up(nc, 4), s));
      CIP_CUDA(cudaStreamSynchronize(s));
    }
    cudaFree(stg);
  }
  CIP_TRY(make_q4_tensor_map(&ey.mapA.map, ey.A4, mM, n_pad / 4));
  // C = A D^-1 A' (lower tiles; a few tiles over a long contraction: the split-K tail fills the SMs)
  CIP_TRY(ey_alloc(h, &ey.C4, (size_t)mM * mM));
  CIP_TRY(ey_alloc(h, &ey.M4, (size_t)mM * mM));
  CIP_TRY(ey_alloc(h, &ey.Winv, (size_t)mM * TILE));
  {
    GemmArgs a{};
    a.lower = 1; a.ntm = a.ntn = mM / TILE; a.sym = 1; a.nk = n_pad / 32;
    a.Cin = nullptr; a.Cout = ey.C4; a.ldc = mM; a.alpha = 1.0;
    a.ws = h->gemm_ws; a.ws_doubles = GEMM_WS_DOUBLES;
    a.kscale = ey.kscale;
    CIP_TRY(launch_gemm_nt(ey.mapA, ey.mapA, a, s));
  }
  CIP_TRY(chol_make_plan(&ey.chol, ey.M4, mM, ey.Winv, h->info));
  if (p > 0) {
    // E' = G D^-1 A' (p_pad x mM, rows = rows of G, k = rows of A) and P = G D^-1 G' on top of Sbase4 (which holds
    // the identity on the padding and reg_eps_G I)
    GemmOperand mapG{};
    CIP_TRY(make_q4_tensor_map(&mapG.map, h->G4, h->p_pad, n_pad / 4));
    CIP_TRY(ey_alloc(h, &ey.Et4, (size_t)h->p_pad * mM));
    CIP_TRY(ey_alloc(h, &ey.Z4, (size_t)h->p_pad * mM));
    GemmArgs e{};
    e.lower = 0; e.ntm = h->p_pad / TILE; e.ntn = mM / TILE; e.sym = 0; e.nk = n_pad / 32;
    e.Cin = nullptr; e.Cout = ey.Et4; e.ldc = h->p_pad; e.alpha = 1.0;
    e.ws = h->gemm_ws; e.ws_doubles = GEMM_WS_DOUBLES;
    e.kscale = ey.kscale;
    CIP_TRY(launch_gemm_nt(mapG, ey.mapA, e, s));
    GemmArgs q{};
    q.lower = 1; q.ntm = q.ntn = h->p_pad / TILE; q.sym = 1; q.nk = n_pad / 32;
    q.Cin = h->Sbase4; q.Cout = h->Sbase4; q.ldc = h->p_pad; q.alpha = 1.0;
    q.ws = h->gemm_ws; q.ws_doubles = GEMM_WS_DOUBLES;
    q.kscale = ey.kscale;
    CIP_TRY(launch_gemm_nt(mapG, mapG, q, s));
    CIP_TRY(make_q4_tensor_map(&ey.mapZ.map, ey.Z4, h->p_pad, mM / 4));
  }
  // per-factorisation scratch: b'b per cone, W = R R' per S cone, the S-cone index of every cone
  CIP_TRY(ey_alloc(h, &ey.qbb, h->ncones + 1));
  CIP_TRY(ey_alloc(h, &ey.W, h->r_total + 1));
  {
    std::vector<int> sidx(h->ncones + 1, -1);
    for (size_t si = 0; si < h->h_slist.size(); ++si) sidx[h->h_slist[si]] = (int)si;
    double* d = nullptr;
    CIP_TRY(ey_alloc(h, &d, (sidx.size() + 1) / 2));
    ey.sidx = reinterpret_cast<int*>(d);
    CIP_CUDA(cudaMemcpyAsync(ey.sidx, sidx.data(), sidx.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    CIP_CUDA(cudaStreamSynchronize(s));
  }
  for (auto& v : ey.v) CIP_TRY(ey_alloc(h, &v, mM + 4));
  CIP_CUDA(cudaStreamSynchronize(s));
  return 0;
}

int ey_form_M(cip_engine* h) {
  EliminateY& ey = h->ey;
  cudaStream_t s = h->stream;
  CIP_CUDA(cudaEventRecord(h->ev[1], s));
  if (h->cd.nq > 0) {
    ey_qbb_kernel<<<h->cd.nq, 256, 0, s>>>(h->cd.qlist, h->cd.off, h->F.kind, h->F.b, ey.qbb);
    CIP_CHECK_LAUNCH();
  }
  if (h->cd.ns > 0) {
    ey_w_kernel<<<h->cd.ns, 256, 0, s>>>(h->cd.slist, h->cd.sord, h->cd.roff, h->F.kind, h->F.R, ey.W);
    CIP_CHECK_LAUNCH();
  }
  AssembleArgs g{};
  g.C = ey.C4; g.M = ey.M4; g.ld = ey.mM; g.m = h->m;
  g.row_cone = h->cd.row_cone; g.type = h->cd.type; g.off = h->cd.off; g.sidx = ey.sidx;
  g.sord = h->cd.sord; g.roff = h->cd.roff; g.kind = h->F.kind;
  g.a = h->F.a; g.b = h->F.b; g.D = h->F.D; g.bb = ey.qbb; g.W = ey.W;
  ey_assemble_kernel<<<grid_for((size_t)ey.mM * ey.mM), 256, 0, s>>>(g);
  CIP_CHECK_LAUNCH();
  CIP_CUDA(cudaEventRecord(h->ev[2], s));
  return 0;
}

int ey_solve(cip_engine* h, const double* ry, const double* rw, const double* rv, double* dy, double* dw, double* dv) {
  EliminateY& ey = h->ey;
  cudaStream_t s = h->stream;
  const int n = h->n, m = h->m, p = h->p;
  double *u = h->nv[1], *atc = h->nv[2], *gtb = h->nv[3];
  double *r1 = ey.v[0], *t = ey.v[1], *c = ey.v[2], *tmp = ey.v[3];
  // u = D^-1 ry;  r1 = rv - A u;  r2 = rw - G u
  CIP_TRY(dscale(u, ey.dinv, ry, nullptr, nullptr, n, s));
  CIP_TRY(q4_mv_rows(tmp, ey.A4, ey.mM, m, n, u, h->partial, h->partial_cap, s));
  CIP_TRY(vec_axpby(r1, 1.0, rv, -1.0, tmp, m, s));
  // t = L^-1 r1
  CIP_TRY(chol_fwd(ey.chol, r1, t, s));
  if (p > 0) {
    double **pv = h->pv;
    CIP_TRY(q4_mv_rows(pv[1], h->G4, h->p_pad, p, n, u, h->partial, h->partial_cap, s));
    CIP_TRY(vec_axpby(pv[2], 1.0, rw, -1.0, pv[1], p, s));                     // r2
    CIP_TRY(q4_mv_rows(pv[3], ey.Z4, h->p_pad, p, m, t, h->partial, h->partial_cap, s));   // Z t
    CIP_TRY(vec_axpby(pv[1], 1.0, pv[3], -1.0, pv[2], p, s));                  // Z t - r2
    CIP_TRY(chol_fwd(h->cholS, pv[1], pv[3], s));
    CIP_TRY(chol_bwd(h->cholS, pv[3], dw, s));                                  // b
    CIP_TRY(q4_mv_k(tmp, ey.Z4, h->p_pad, p, m, dw, s));                       // Z'b
    CIP_TRY(vec_axpby(t, 1.0, t, 1.0, tmp, m, s));
  }
  // c = L^-T (t + Z'b)
  CIP_TRY(chol_bwd(ey.chol, t, c, s));
  // a = D^-1 (ry - G'b + A'c)
  CIP_TRY(q4_mv_k(atc, ey.A4, ey.mM, m, n, c, s));
  if (p > 0) CIP_TRY(q4_mv_k(gtb, h->G4, h->p_pad, p, n, dw, s));
  CIP_TRY(dscale(dy, ey.dinv, ry, p > 0 ? gtb : nullptr, atc, n, s));
  CIP_TRY(vec_copy(dv, c, m, s));
  return 0;
}

int ey_solve_H(cip_engine* h, const double* rhs, double* x) {
  EliminateY& ey = h->ey;
  cudaStream_t s = h->stream;
  const int n = h->n, m = h->m;
  double *u = h->nv[1], *atz = h->nv[3];
  double *w = ey.v[0], *t = ey.v[1], *z = ey.v[2];
  // H^-1 rhs = D^-1 rhs - D^-1 A' M^-1 A D^-1 rhs
  CIP_TRY(dscale(u, ey.dinv, rhs, nullptr, nullptr, n, s));
  CIP_TRY(q4_mv_rows(w, ey.A4, ey.mM, m, n, u, h->partial, h->partial_cap, s));
  CIP_TRY(chol_fwd(ey.chol, w, t, s));
  CIP_TRY(chol_bwd(ey.chol, t, z, s));
  CIP_TRY(q4_mv_k(atz, ey.A4, ey.mM, m, n, z, s));
  CIP_TRY(dscale(x, ey.dinv, rhs, atz, nullptr, n, s));
  return 0;
}

int ey_mul_Q(cip_engine* h, double* y, const double* x) {
  return dscale(y, h->ey.qdiag, x, nullptr, nullptr, h->n, h->stream);
}

int ey_get_M(cip_engine* h, double* tmp) {
  return unpack_rows_q4(tmp, h->m, h->ey.M4, h->ey.mM, h->m, h->m, h->stream);
}

}  // namespace cip
