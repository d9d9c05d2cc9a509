// Fast SYRK for the dense single-device path: H = Q + X'X (X = Atil, m x n, all rows R cones) as a blocked SYRK
// whose off-diagonal blocks take one Strassen-Winograd level.
//
// The column range [0, n_pad) is halved `depth` times.  At depth d there are 2^d pairs (a, b) of adjacent column
// ranges of width w = n_pad / 2^(d+1); the off-diagonal block H[b, a] = X_b'X_a is a w x w product with contraction
// m, done as 7 products of half size (h = w / 2, contraction K2 = m / 2) instead of 8.  The 2^depth diagonal leaves
// are the plain lower-triangular SYRK.  About 7/8 of the flops of the off-diagonal blocks remain: at n = 16384,
// depth 3, the whole SYRK does 0.89 m n^2 multiply-adds instead of m n^2 (counting tiles on the diagonal).
//
// Operand sums add columns i and i + h of X (output-index direction), which lets the error of H_ij grow with the
// norms of other columns.  So the columns are equilibrated by exact powers of two first: with e_j = round(log2
// ||x_j||) the sums are formed from x_j 2^-e_j, whose norms lie within a factor of 2 of each other, and the products
// are unscaled by 2^(e_i + e_j) when they are combined.  The error on H_ij is then bounded by c u sqrt(H_ii H_jj),
// the form a Cholesky factorisation is invariant to (Ballard, Benson, Druinsky, Lipshitz, Schwartz, SIMAX 2016).
// Products of raw blocks of X are unscaled by the same powers of two on their output (exact, barring underflow).
//
// Memory: the sums S1..S4 (of X_b) and T1..T4 (of X_a) live in Atil4 itself, in 2 K2 extra rows of contraction
// after the (zero-padded) rows of A, so that one tensor map addresses raw blocks and sums alike and all the products
// of a depth are one grouped launch of the unchanged DMMA tile kernel (GemmArgs::group).  The products go tile-major
// into M and one kernel combines them into H4 with Winograd's signs, adding Q once.
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "engine.h"

namespace cip {

namespace {

constexpr int FAST_SYRK_LEAF = 2048;     // width of the diagonal leaves (scripts/fast_syrk_timing.py)
constexpr int FAST_SYRK_N0 = 12288;      // smallest n_pad that takes the fast path by default (same script)

// S = sums of the four blocks of X_b, T = of X_a, every row scaled by 2^-e first.  Thread (kq, x): pair p = x / h,
// row i = x % h of each half-block; writes S1..S4 at kq_pool + kq, rows ra + {0, h, 2h, 3h} + i, and T1..T4 at
// kq_pool + KQ2 + kq, the same rows.
__global__ void __launch_bounds__(256)
winograd_sums_kernel(double* __restrict__ X, int ld, int KQ2, int h, const int* __restrict__ colexp) {
  const int kq = blockIdx.x;
  const int x = blockIdx.y * blockDim.x + threadIdx.x;
  if (x >= ld / 4) return;
  const int p = x / h, i = x - p * h;
  const int ra = 4 * p * h + i, rb = ra + 2 * h;         // row i of the first half of a / of b
  auto at = [&](int kqq, int r) { return reinterpret_cast<double2*>(X + ((size_t)kqq * ld + r) * 4); };
  auto ld4 = [&](int kqq, int r, double f, double2& lo, double2& hi) {
    const double2* q = at(kqq, r);
    lo = q[0]; hi = q[1];
    lo.x *= f; lo.y *= f; hi.x *= f; hi.y *= f;
  };
  const double fa1 = ldexp(1.0, -colexp[ra]), fa2 = ldexp(1.0, -colexp[ra + h]);
  const double fb1 = ldexp(1.0, -colexp[rb]), fb2 = ldexp(1.0, -colexp[rb + h]);
  double2 a11l, a11h, a12l, a12h, a21l, a21h, a22l, a22h, b11l, b11h, b12l, b12h, b21l, b21h, b22l, b22h;
  ld4(kq, rb, fb1, a11l, a11h);
  ld4(kq + KQ2, rb, fb1, a12l, a12h);
  ld4(kq, rb + h, fb2, a21l, a21h);
  ld4(kq + KQ2, rb + h, fb2, a22l, a22h);
  ld4(kq, ra, fa1, b11l, b11h);
  ld4(kq + KQ2, ra, fa1, b12l, b12h);
  ld4(kq, ra + h, fa2, b21l, b21h);
  ld4(kq + KQ2, ra + h, fa2, b22l, b22h);
  auto add = [](double2 u, double2 v) { return make_double2(u.x + v.x, u.y + v.y); };
  auto sub = [](double2 u, double2 v) { return make_double2(u.x - v.x, u.y - v.y); };
  // S1 = A21 + A22, S2 = S1 - A11, S3 = A11 - A21, S4 = A12 - S2
  const double2 s1l = add(a21l, a22l), s1h = add(a21h, a22h);
  const double2 s2l = sub(s1l, a11l), s2h = sub(s1h, a11h);
  const double2 s3l = sub(a11l, a21l), s3h = sub(a11h, a21h);
  const double2 s4l = sub(a12l, s2l), s4h = sub(a12h, s2h);
  // T1 = B21 - B11, T2 = B22 - T1, T3 = B22 - B21, T4 = T2 - B12   (B = X_a: Winograd's right factor is B')
  const double2 t1l = sub(b21l, b11l), t1h = sub(b21h, b11h);
  const double2 t2l = sub(b22l, t1l), t2h = sub(b22h, t1h);
  const double2 t3l = sub(b22l, b21l), t3h = sub(b22h, b21h);
  const double2 t4l = sub(t2l, b12l), t4h = sub(t2h, b12h);
  const int ks = 2 * KQ2 + kq, kt = 3 * KQ2 + kq;
  auto st4 = [&](int kqq, int r, double2 lo, double2 hi) { double2* q = at(kqq, r); q[0] = lo; q[1] = hi; };
  st4(ks, ra, s1l, s1h);
  st4(ks, ra + h, s2l, s2h);
  st4(ks, ra + 2 * h, s3l, s3h);
  st4(ks, ra + 3 * h, s4l, s4h);
  st4(kt, ra, t1l, t1h);
  st4(kt, ra + h, t2l, t2h);
  st4(kt, ra + 2 * h, t3l, t3h);
  st4(kt, ra + 3 * h, t4l, t4h);
}

// H[b, a] (Q4, ld) = Q[b, a] + the Winograd combination of the seven product tiles of pair blockIdx.y, tile
// blockIdx.x of the h x h half-block grid (column-major, nt tiles a side).  Products of raw blocks carry the
// scaling of their raw side(s), removed here; everything is unscaled by 2^(e_i + e_j) at the end (all exact).
__global__ void __launch_bounds__(256)
winograd_combine_kernel(const double* __restrict__ M, const double* __restrict__ Cin, double* __restrict__ H, int ld,
                        int h, const int* __restrict__ colexp) {
  const int nt = h / TILE, G = nt * nt;
  const int L = blockIdx.x, p = blockIdx.y;
  const int ti = L % nt, tj = L / nt;
  const int ra = 4 * p * h, rb = ra + 2 * h;
  const size_t slab = (size_t)TILE * TILE;
  const double* Mp = M + ((size_t)p * 7 * G + L) * slab;     // product q: Mp + q * G * slab
  for (int e = threadIdx.x * 2; e < TILE * TILE; e += 512) {
    const int quad = e / (TILE * 4), lr = (e % (TILE * 4)) >> 2, c = e & 3;
    const int i = ti * TILE + lr, j = tj * TILE + quad * 4 + c;
    double2 P[7];
#pragma unroll
    for (int q = 0; q < 7; ++q) P[q] = *reinterpret_cast<const double2*>(Mp + (size_t)q * G * slab + e);
    const int eb1 = colexp[rb + i], eb2 = colexp[rb + h + i];
    const int ea1[2] = {colexp[ra + j], colexp[ra + j + 1]};
    const int ea2[2] = {colexp[ra + h + j], colexp[ra + h + j + 1]};
    double o[4][2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const double p1 = k ? P[0].y : P[0].x, p2 = k ? P[1].y : P[1].x, p3 = k ? P[2].y : P[2].x;
      const double p4 = k ? P[3].y : P[3].x, p5 = k ? P[4].y : P[4].x, p6 = k ? P[5].y : P[5].x;
      const double p7 = k ? P[6].y : P[6].x;
      const double u2 = ldexp(p1, -(eb1 + ea1[k])) + p6;    // P1 is raw x raw, P3 raw on a, P4 raw on b
      const double u3 = u2 + p7, u4 = u2 + p5;
      o[0][k] = p1 + p2;                                      // C11 = P1 + P2 is raw already
      o[1][k] = ldexp(u4 + ldexp(p3, -ea2[k]), eb1 + ea2[k]);   // C12
      o[2][k] = ldexp(u3 - ldexp(p4, -eb2), eb2 + ea1[k]);      // C21
      o[3][k] = ldexp(u3 + p5, eb2 + ea2[k]);                   // C22
    }
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const size_t idx = q4_index(rb + (b >> 1) * h + i, ra + (b & 1) * h + j, ld);
      double2 v = make_double2(o[b][0], o[b][1]);
      if (Cin) {
        const double2 q = *reinterpret_cast<const double2*>(Cin + idx);
        v.x += q.x;
        v.y += q.y;
      }
      *reinterpret_cast<double2*>(H + idx) = v;
    }
  }
}

int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return (e && *e) ? atoi(e) : dflt;
}

template <typename T>
int falloc(cip_engine* h, T** p, size_t count) {
  *p = nullptr;
  if (count == 0) count = 1;
  CIP_CUDA(cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T)));
  CIP_CUDA(cudaMemsetAsync(*p, 0, count * sizeof(T), h->stream));
  h->bytes += count * sizeof(T);
  h->owned.push_back(*p);
  return 0;
}

size_t m_doubles(int n_pad) { return (size_t)7 * n_pad / 4 * n_pad / 4; }   // the seven products of depth 0

}  // namespace

int fast_syrk_plan(cip_engine* h, bool can) {
  FastSyrk& f = h->fast;
  f = FastSyrk{};
  const int mode = env_int("CIP_FAST_SYRK", 2);             // 0: never, 1: whenever the handle allows it, else automatic
  if (!can || mode == 0 || h->m_pad == 0) return 0;
  int leaf = std::max(256, env_int("CIP_FAST_SYRK_LEAF", FAST_SYRK_LEAF));
  if (mode == 1) leaf = std::min(leaf, h->n_pad / 2);
  // halve while the off-diagonal block of the level splits into 128-aligned halves and the halves stay >= leaf
  int W = h->n_pad, depth = 0;
  while (W % 512 == 0 && W / 2 >= leaf) { W /= 2; ++depth; }
  if (depth == 0 || (mode != 1 && h->n_pad < FAST_SYRK_N0)) return 0;
  const int K2 = round_up(h->m_pad, 64) / 2;
  const size_t nn = (size_t)h->n_pad * h->n_pad;
  const size_t atil = (size_t)4 * K2 * h->n_pad;             // 2 K2 rows of X, 2 K2 rows of sums
  const size_t colss = (size_t)scale_panel_norms_chunks(h->m_pad) * h->n_pad;
  if (mode != 1) {
    // what is still to be allocated besides: Q, H, the Cholesky workspaces (~ 3 n_pad^2), the split-K workspace, 1 GB
    size_t free_b = 0, total_b = 0;
    CIP_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const size_t need = (atil + m_doubles(h->n_pad) + colss + 3 * nn + (size_t)GEMM_WS_DOUBLES) * 8 + (size_t(1) << 30);
    if (free_b < need) return 0;
  }
  f.on = true;
  f.depth = depth;
  f.leaf = W;
  f.K2 = K2;
  f.nchunk = scale_panel_norms_chunks(h->m_pad);
  return 0;
}

size_t fast_syrk_atil_doubles(const cip_engine* h) { return (size_t)4 * h->fast.K2 * h->n_pad; }

int fast_syrk_setup(cip_engine* h) {
  FastSyrk& f = h->fast;
  if (!f.on) return 0;
  CIP_TRY(falloc(h, &f.colexp, h->n_pad));
  CIP_TRY(falloc(h, &f.colss, (size_t)f.nchunk * h->n_pad));
  CIP_TRY(falloc(h, &f.M, m_doubles(h->n_pad)));
  // GemmArgs::group entries: the 2^depth leaves, then the seven products of every pair of depth 0, 1, ...
  const int KQ2 = f.K2 / 4, PQ0 = 2 * KQ2;
  std::vector<int4> t;
  for (int l = 0; l < (1 << f.depth); ++l) {
    const int r0 = l * f.leaf;
    t.push_back(make_int4(r0, 0, r0, 0));
    t.push_back(make_int4(r0, r0, 0, 0));
  }
  for (int d = 0; d < f.depth; ++d) {
    const int w = h->n_pad >> (d + 1), hh = w / 2;
    for (int p = 0; p < (1 << d); ++p) {
      const int ra = 2 * p * w, rb = ra + w;
      const int4 ops[7] = {
          make_int4(rb, 0, ra, 0),                              // P1 = A11 B11'
          make_int4(rb, KQ2, ra, KQ2),                          // P2 = A12 B12'
          make_int4(ra + 3 * hh, PQ0, ra + hh, KQ2),            // P3 = S4 B22'
          make_int4(rb + hh, KQ2, ra + 3 * hh, PQ0 + KQ2),      // P4 = A22 T4'
          make_int4(ra, PQ0, ra, PQ0 + KQ2),                    // P5 = S1 T1'
          make_int4(ra + hh, PQ0, ra + hh, PQ0 + KQ2),          // P6 = S2 T2'
          make_int4(ra + 2 * hh, PQ0, ra + 2 * hh, PQ0 + KQ2)}; // P7 = S3 T3'
      for (const int4& o : ops) {
        t.push_back(o);
        t.push_back(make_int4(0, 0, 0, 0));
      }
    }
  }
  CIP_TRY(falloc(h, &f.table, t.size()));
  CIP_CUDA(cudaMemcpyAsync(f.table, t.data(), t.size() * sizeof(int4), cudaMemcpyHostToDevice, h->stream));
  CIP_CUDA(cudaStreamSynchronize(h->stream));                // t goes out of scope
  return 0;
}

int fast_syrk_drop(cip_engine* h) {
  FastSyrk& f = h->fast;
  if (!f.on) return 0;
  // a row-sharded handle forms H through the all-reduce paths: Atil4 goes back to its plain size
  CIP_CUDA(cudaStreamSynchronize(h->stream));
  for (void* p : {(void*)f.colexp, (void*)f.colss, (void*)f.M, (void*)f.table}) {
    h->owned.erase(std::find(h->owned.begin(), h->owned.end(), p));
    CIP_CUDA(cudaFree(p));
  }
  CIP_CUDA(cudaFree(h->Atil4));
  h->bytes -= fast_syrk_atil_doubles(h) * 8;
  const size_t mn = (size_t)h->m_pad * h->n_pad;
  CIP_CUDA(cudaMalloc(reinterpret_cast<void**>(&h->Atil4), mn * 8));
  CIP_CUDA(cudaMemsetAsync(h->Atil4, 0, mn * 8, h->stream));
  h->bytes += mn * 8;
  CIP_TRY(make_q4_tensor_map(&h->mapAtil.map, h->Atil4, h->n_pad, h->m_pad / 4));
  f = FastSyrk{};
  return 0;
}

int fast_syrk_form(cip_engine* h, const double* cin) {
  const FastSyrk& f = h->fast;
  cudaStream_t s = h->stream;
  const int KQ2 = f.K2 / 4, L = 1 << f.depth;
  for (int d = 0; d < f.depth; ++d) {
    const int pairs = 1 << d, hh = h->n_pad >> (d + 2), nt = hh / TILE;
    winograd_sums_kernel<<<dim3(KQ2, (h->n_pad / 4 + 255) / 256), 256, 0, s>>>(h->Atil4, h->n_pad, KQ2, hh, f.colexp);
    CIP_CHECK_LAUNCH();
    GemmArgs g{};
    g.lower = 0; g.ntm = g.ntn = nt; g.sym = 0;
    g.nk = f.K2 / 32;
    g.Ctm = f.M; g.ldc = h->n_pad; g.alpha = 1.0;
    g.ws = h->gemm_ws; g.ws_doubles = GEMM_WS_DOUBLES;
    g.group = f.table + 2 * (L + 7 * (pairs - 1));
    g.group_tiles = nt * nt;
    g.tile_count = 7 * pairs * nt * nt;
    CIP_TRY(launch_gemm_nt(h->mapAtil, h->mapAtil, g, s));
    winograd_combine_kernel<<<dim3(nt * nt, pairs), 256, 0, s>>>(f.M, cin, h->H4, h->n_pad, hh, f.colexp);
    CIP_CHECK_LAUNCH();
  }
  const int T = f.leaf / TILE;
  GemmArgs a{};
  a.lower = 1; a.ntm = a.ntn = T; a.sym = 1;
  a.nk = h->m_pad / 32;
  a.Cin = cin; a.Cout = h->H4; a.ldc = h->n_pad; a.alpha = 1.0;
  a.ws = h->gemm_ws; a.ws_doubles = GEMM_WS_DOUBLES;
  a.group = f.table;
  a.group_tiles = T * (T + 1) / 2;
  a.tile_count = L * a.group_tiles;
  CIP_TRY(launch_gemm_nt(h->mapAtil, h->mapAtil, a, s));
  return 0;
}

}  // namespace cip
