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
//
// Second level.  Where the half-blocks are wide (h / 2 >= FAST_SYRK_L2_MIN), each of the seven products of a depth
// is itself done as 7 products of size h/2 x h/2 with contraction K2/2, one level-1 product q at a time: its
// operand sums (8 blocks of (h/2) x (K2/2) per pair, n_pad rows across the pairs) go to K2/2 more rows of
// contraction at the end of Atil4, one grouped launch computes the 7 x pairs sub-products into M2, and
// winograd_combine2_kernel adds them into slot q of M.  Level-2 sums are formed from equilibrated rows (the level-1
// sums are; raw blocks are scaled as they are loaded), and every product of a two-level depth reaches M fully
// scaled, so the level-1 combination unscales each output block once, by 2^(e_i + e_j), at the end.
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "engine.h"

namespace cip {

namespace {

constexpr int FAST_SYRK_LEAF = 2048;     // width of the diagonal leaves (scripts/fast_syrk_timing.py)
constexpr int FAST_SYRK_N0 = 12288;      // smallest n_pad that takes the fast path by default (same script)
constexpr int FAST_SYRK_L2_MIN = 1024;   // narrowest level-2 product a depth takes a second level for: 7.5-9.8 % off
                                         // the depth at 1024-2048, 3-4 % at 512-768 (profiles/r06_fast_syrk_two_level.md)

// One Winograd level of operand sums over the pairs of a depth.  Operand a (Winograd's left factor) has rows
// base + a_row + [0, 2h) and quads a_kq + [0, 2 kqh); operand b (the NT form of the right factor) likewise; base =
// p * pstride for pair p.  Writes S1..S4 (of a) at rows base + s_row + {0, h, 2h, 3h} + i, quads s_kq + kq, and
// T1..T4 (of b) at rows base + t_row + ..., quads t_kq + kq.  A side whose rows are raw columns of Atil is scaled
// by 2^-e_j as it is loaded; sums are equilibrated already.
struct SumsArgs {
  int h, kqh, pstride, count;    // count = pairs * h threads per quad
  int a_row, a_kq, b_row, b_kq, s_row, s_kq, t_row, t_kq;
  int scale_a, scale_b;
};

__device__ __forceinline__ void winograd_sums(double* __restrict__ X, int ld, const SumsArgs& s,
                                              const int* __restrict__ colexp) {
  const int kq = blockIdx.x;
  const int x = blockIdx.y * blockDim.x + threadIdx.x;
  if (x >= s.count) return;
  const int h = s.h, KQ2 = s.kqh;
  const int p = x / h, i = x - p * h, base = p * s.pstride;
  const int xa = base + s.a_row + i, xb = base + s.b_row + i;   // row i of the first half of operand a / b
  const int ka = s.a_kq + kq, kb = s.b_kq + kq;
  auto at = [&](int kqq, int r) { return reinterpret_cast<double2*>(X + ((size_t)kqq * ld + r) * 4); };
  auto ld4 = [&](int kqq, int r, double f, double2& lo, double2& hi) {
    const double2* q = at(kqq, r);
    lo = q[0]; hi = q[1];
    lo.x *= f; lo.y *= f; hi.x *= f; hi.y *= f;
  };
  auto fac = [&](int on, int r) { return on ? ldexp(1.0, -colexp[r]) : 1.0; };
  const double fa1 = fac(s.scale_a, xa), fa2 = fac(s.scale_a, xa + h);
  const double fb1 = fac(s.scale_b, xb), fb2 = fac(s.scale_b, xb + h);
  double2 a11l, a11h, a12l, a12h, a21l, a21h, a22l, a22h, b11l, b11h, b12l, b12h, b21l, b21h, b22l, b22h;
  ld4(ka, xa, fa1, a11l, a11h);
  ld4(ka + KQ2, xa, fa1, a12l, a12h);
  ld4(ka, xa + h, fa2, a21l, a21h);
  ld4(ka + KQ2, xa + h, fa2, a22l, a22h);
  ld4(kb, xb, fb1, b11l, b11h);
  ld4(kb + KQ2, xb, fb1, b12l, b12h);
  ld4(kb, xb + h, fb2, b21l, b21h);
  ld4(kb + KQ2, xb + h, fb2, b22l, b22h);
  auto add = [](double2 u, double2 v) { return make_double2(u.x + v.x, u.y + v.y); };
  auto sub = [](double2 u, double2 v) { return make_double2(u.x - v.x, u.y - v.y); };
  // S1 = A21 + A22, S2 = S1 - A11, S3 = A11 - A21, S4 = A12 - S2
  const double2 s1l = add(a21l, a22l), s1h = add(a21h, a22h);
  const double2 s2l = sub(s1l, a11l), s2h = sub(s1h, a11h);
  const double2 s3l = sub(a11l, a21l), s3h = sub(a11h, a21h);
  const double2 s4l = sub(a12l, s2l), s4h = sub(a12h, s2h);
  // T1 = B21 - B11, T2 = B22 - T1, T3 = B22 - B21, T4 = T2 - B12   (B: Winograd's right factor is B')
  const double2 t1l = sub(b21l, b11l), t1h = sub(b21h, b11h);
  const double2 t2l = sub(b22l, t1l), t2h = sub(b22h, t1h);
  const double2 t3l = sub(b22l, b21l), t3h = sub(b22h, b21h);
  const double2 t4l = sub(t2l, b12l), t4h = sub(t2h, b12h);
  const int ks = s.s_kq + kq, kt = s.t_kq + kq, rs = base + s.s_row + i, rt = base + s.t_row + i;
  auto st4 = [&](int kqq, int r, double2 lo, double2 hi) { double2* q = at(kqq, r); q[0] = lo; q[1] = hi; };
  st4(ks, rs, s1l, s1h);
  st4(ks, rs + h, s2l, s2h);
  st4(ks, rs + 2 * h, s3l, s3h);
  st4(ks, rs + 3 * h, s4l, s4h);
  st4(kt, rt, t1l, t1h);
  st4(kt, rt + h, t2l, t2h);
  st4(kt, rt + 2 * h, t3l, t3h);
  st4(kt, rt + 3 * h, t4l, t4h);
}

// the level-1 sums of a depth and the level-2 sums of one level-1 product (two names for the profiler)
__global__ void __launch_bounds__(256)
winograd_sums_kernel(double* __restrict__ X, int ld, const SumsArgs s, const int* __restrict__ colexp) {
  winograd_sums(X, ld, s, colexp);
}
__global__ void __launch_bounds__(256)
winograd_sums2_kernel(double* __restrict__ X, int ld, const SumsArgs s, const int* __restrict__ colexp) {
  winograd_sums(X, ld, s, colexp);
}

// Level-1 product q of pair blockIdx.y (slot q of M, nt = 2 nt2 tiles a side) = the Winograd combination of its
// seven sub-product tiles in M2 (tile blockIdx.x of the h2 x h2 grid, nt2 tiles a side, column-major).  Its rows
// are rows p * pstride + x_row + [0, 2 h2) of Atil4, its columns p * pstride + y_row + [0, 2 h2); a raw side
// (raw_x / raw_y) left its sub-products P1, P2 and P4 (x) or P1, P2 and P3 (y) unscaled, which is removed here, so
// that the product reaches M fully scaled.
__global__ void __launch_bounds__(256)
winograd_combine2_kernel(const double* __restrict__ M2, double* __restrict__ M, int h2, int q, int pstride,
                         int x_row, int y_row, int raw_x, int raw_y, const int* __restrict__ colexp) {
  const int nt2 = h2 / TILE, G2 = nt2 * nt2, nt = 2 * nt2, G = nt * nt;
  const int L2 = blockIdx.x, p = blockIdx.y;
  const int ti = L2 % nt2, tj = L2 / nt2;
  const int xr = p * pstride + x_row, yr = p * pstride + y_row;
  const size_t slab = (size_t)TILE * TILE;
  const double* Mp = M2 + ((size_t)p * 7 * G2 + L2) * slab;    // sub-product r: Mp + r * G2 * slab
  double* Mq = M + (size_t)(p * 7 + q) * G * slab;
  for (int e = threadIdx.x * 2; e < TILE * TILE; e += 512) {
    const int quad = e / (TILE * 4), lr = (e % (TILE * 4)) >> 2, c = e & 3;
    const int i = ti * TILE + lr, j = tj * TILE + quad * 4 + c;
    double2 P[7];
#pragma unroll
    for (int r = 0; r < 7; ++r) P[r] = *reinterpret_cast<const double2*>(Mp + (size_t)r * G2 * slab + e);
    const int ex1 = raw_x ? colexp[xr + i] : 0, ex2 = raw_x ? colexp[xr + h2 + i] : 0;
    const int ey1[2] = {raw_y ? colexp[yr + j] : 0, raw_y ? colexp[yr + j + 1] : 0};
    const int ey2[2] = {raw_y ? colexp[yr + h2 + j] : 0, raw_y ? colexp[yr + h2 + j + 1] : 0};
    double o[4][2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const double p1 = k ? P[0].y : P[0].x, p2 = k ? P[1].y : P[1].x, p3 = k ? P[2].y : P[2].x;
      const double p4 = k ? P[3].y : P[3].x, p5 = k ? P[4].y : P[4].x, p6 = k ? P[5].y : P[5].x;
      const double p7 = k ? P[6].y : P[6].x;
      const double s1 = ldexp(p1, -(ex1 + ey1[k])), s2 = ldexp(p2, -(ex1 + ey1[k]));
      const double u2 = s1 + p6;
      const double u3 = u2 + p7, u4 = u2 + p5;
      o[0][k] = s1 + s2;
      o[1][k] = u4 + ldexp(p3, -ey2[k]);
      o[2][k] = u3 - ldexp(p4, -ex2);
      o[3][k] = u3 + p5;
    }
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int L = (ti + (b >> 1) * nt2) + (tj + (b & 1) * nt2) * nt;
      *reinterpret_cast<double2*>(Mq + (size_t)L * slab + e) = make_double2(o[b][0], o[b][1]);
    }
  }
}

// H[b, a] (Q4, ld) = Q[b, a] + the Winograd combination of the seven product tiles of pair blockIdx.y, tile
// blockIdx.x of the h x h half-block grid (column-major, nt tiles a side).  Products of raw blocks carry the
// scaling of their raw side(s), removed here, unless `scaled` (a two-level depth: every product is fully scaled);
// everything is unscaled by 2^(e_i + e_j) at the end (all exact).
__global__ void __launch_bounds__(256)
winograd_combine_kernel(const double* __restrict__ M, const double* __restrict__ Cin, double* __restrict__ H, int ld,
                        int h, int scaled, const int* __restrict__ colexp) {
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
      // one level: P1 is raw x raw, P3 raw on a, P4 raw on b
      const double u2 = (scaled ? p1 : ldexp(p1, -(eb1 + ea1[k]))) + p6;
      const double u3 = u2 + p7, u4 = u2 + p5;
      o[0][k] = scaled ? ldexp(p1 + p2, eb1 + ea1[k]) : p1 + p2;                  // C11
      o[1][k] = ldexp(u4 + (scaled ? p3 : ldexp(p3, -ea2[k])), eb1 + ea2[k]);    // C12
      o[2][k] = ldexp(u3 - (scaled ? p4 : ldexp(p4, -eb2)), eb2 + ea1[k]);       // C21
      o[3][k] = ldexp(u3 + p5, eb2 + ea2[k]);                                    // C22
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

// the sub-products of the first two-level depth (the widest): 7 per pair, h2 x h2 each
size_t m2_doubles(int n_pad, unsigned two) {
  if (!two) return 0;
  int d = 0;
  while (!(two >> d & 1u)) ++d;
  const size_t h2 = (size_t)n_pad >> (d + 3);
  return (size_t)7 * ((size_t)1 << d) * h2 * h2;
}

// rows of contraction of Atil4: A (zero-padded to 2 K2), the level-1 sums (2 K2), the level-2 sums (K2 / 2)
size_t atil_rows(const FastSyrk& f) { return (size_t)4 * f.K2 + (f.two ? f.K2 / 2 : 0); }

// The group origins {x_row0, x_kq0, y_row0, y_kq0} of Winograd's seven products of X Y' for an operand pair whose
// first rows / quads are (xr, xk) and (yr, yk), with half-width hh and half-contraction kqh (quads), and sums
// S1..S4 at rows sr + {0, hh, 2hh, 3hh}, quads sk, T1..T4 at rows tr + ..., quads tk (see winograd_sums).
void winograd_ops(int4 ops[7], int xr, int xk, int yr, int yk, int hh, int kqh, int sr, int sk, int tr, int tk) {
  ops[0] = make_int4(xr, xk, yr, yk);                             // P1 = A11 B11'
  ops[1] = make_int4(xr, xk + kqh, yr, yk + kqh);                 // P2 = A12 B12'
  ops[2] = make_int4(sr + 3 * hh, sk, yr + hh, yk + kqh);         // P3 = S4 B22'
  ops[3] = make_int4(xr + hh, xk + kqh, tr + 3 * hh, tk);         // P4 = A22 T4'
  ops[4] = make_int4(sr, sk, tr, tk);                             // P5 = S1 T1'
  ops[5] = make_int4(sr + hh, sk, tr + hh, tk);                   // P6 = S2 T2'
  ops[6] = make_int4(sr + 2 * hh, sk, tr + 2 * hh, tk);           // P7 = S3 T3'
}

// the level-1 products of pair p at depth d (half-width hh)
void level1_ops(int4 ops[7], int p, int hh, int KQ2) {
  const int ra = 4 * p * hh, rb = ra + 2 * hh;
  winograd_ops(ops, rb, 0, ra, 0, hh, KQ2, ra, 2 * KQ2, ra, 3 * KQ2);
}

// the level-2 sub-products of level-1 product `o` of pair p (half-width hh): sums at rows ra + [0, 4 hh), quads 4 KQ2
void level2_ops(int4 ops[7], int4 o, int p, int hh, int KQ2) {
  const int ra = 4 * p * hh;
  winograd_ops(ops, o.x, o.y, o.z, o.w, hh / 2, KQ2 / 2, ra, 4 * KQ2, ra + 2 * hh, 4 * KQ2);
}

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
  // second level on depth d: its products (h2 = n_pad / 2^(d+3) wide) split into whole tiles and are wide enough
  // to pay for their sums.  CIP_FAST_SYRK_LEVELS = 1: never, 2: wherever the tiles allow it (tests)
  const int levels = env_int("CIP_FAST_SYRK_LEVELS", 0);
  unsigned two = 0;
  for (int d = 0; d < depth && levels != 1; ++d) {
    const int h2 = h->n_pad >> (d + 3);
    if (h2 % TILE == 0 && (h2 >= FAST_SYRK_L2_MIN || levels == 2)) two |= 1u << d;
  }
  const size_t nn = (size_t)h->n_pad * h->n_pad;
  const size_t colss = (size_t)scale_panel_norms_chunks(h->m_pad) * h->n_pad;
  for (;; two = 0) {
    f.two = two;
    f.K2 = round_up(h->m_pad, two ? 128 : 64) / 2;            // level-2 halves of the contraction are whole k tiles
    if (mode == 1) break;
    // what is still to be allocated besides: Q, H, the Cholesky workspaces (~ 3 n_pad^2), the split-K workspace, 1 GB
    size_t free_b = 0, total_b = 0;
    CIP_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const size_t need = (atil_rows(f) * h->n_pad + m_doubles(h->n_pad) + m2_doubles(h->n_pad, two) + colss + 3 * nn +
                         (size_t)GEMM_WS_DOUBLES) * 8 + (size_t(1) << 30);
    if (free_b >= need) break;
    if (!two) { f = FastSyrk{}; return 0; }                     // one level does not fit either: classical SYRK
  }
  f.on = true;
  f.depth = depth;
  f.leaf = W;
  f.nchunk = scale_panel_norms_chunks(h->m_pad);
  return 0;
}

size_t fast_syrk_atil_doubles(const cip_engine* h) { return atil_rows(h->fast) * h->n_pad; }

int fast_syrk_setup(cip_engine* h) {
  FastSyrk& f = h->fast;
  if (!f.on) return 0;
  CIP_TRY(falloc(h, &f.colexp, h->n_pad));
  CIP_TRY(falloc(h, &f.colss, (size_t)f.nchunk * h->n_pad));
  CIP_TRY(falloc(h, &f.M, m_doubles(h->n_pad)));
  if (f.two) CIP_TRY(falloc(h, &f.M2, m2_doubles(h->n_pad, f.two)));
  // GemmArgs::group entries: the 2^depth leaves, then the seven products of every pair of depth 0, 1, ..., then for
  // every two-level depth and each level-1 product q the seven sub-products of every pair
  const int KQ2 = f.K2 / 4;
  std::vector<int4> t;
  for (int l = 0; l < (1 << f.depth); ++l) {
    const int r0 = l * f.leaf;
    t.push_back(make_int4(r0, 0, r0, 0));
    t.push_back(make_int4(r0, r0, 0, 0));
  }
  int4 ops[7], sub[7];
  for (int d = 0; d < f.depth; ++d) {
    const int hh = h->n_pad >> (d + 2);
    for (int p = 0; p < (1 << d); ++p) {
      level1_ops(ops, p, hh, KQ2);
      for (const int4& o : ops) {
        t.push_back(o);
        t.push_back(make_int4(0, 0, 0, 0));
      }
    }
  }
  for (int d = 0; d < f.depth; ++d) {
    if (!(f.two >> d & 1u)) continue;
    const int hh = h->n_pad >> (d + 2);
    for (int q = 0; q < 7; ++q)
      for (int p = 0; p < (1 << d); ++p) {
        level1_ops(ops, p, hh, KQ2);
        level2_ops(sub, ops[q], p, hh, KQ2);
        for (const int4& o : sub) {
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
  for (void* p : {(void*)f.colexp, (void*)f.colss, (void*)f.M, (void*)f.M2, (void*)f.table}) {
    if (!p) continue;
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
  int sub_entry = L + 7 * (L - 1);                          // first level-2 group entry
  for (int d = 0; d < f.depth; ++d) {
    const int pairs = 1 << d, hh = h->n_pad >> (d + 2), nt = hh / TILE;
    const bool two = f.two >> d & 1u;
    SumsArgs sa{hh, KQ2, 4 * hh, pairs * hh, 2 * hh, 0, 0, 0, 0, 2 * KQ2, 0, 3 * KQ2, 1, 1};
    winograd_sums_kernel<<<dim3(KQ2, (sa.count + 255) / 256), 256, 0, s>>>(h->Atil4, h->n_pad, sa, f.colexp);
    CIP_CHECK_LAUNCH();
    GemmArgs g{};
    g.lower = 0; g.ntm = g.ntn = nt; g.sym = 0;
    g.nk = f.K2 / 32;
    g.Ctm = f.M; g.ldc = h->n_pad; g.alpha = 1.0;
    g.ws = h->gemm_ws; g.ws_doubles = GEMM_WS_DOUBLES;
    g.group = f.table + 2 * (L + 7 * (pairs - 1));
    g.group_tiles = nt * nt;
    g.tile_count = 7 * pairs * nt * nt;
    if (!two) {
      CIP_TRY(launch_gemm_nt(h->mapAtil, h->mapAtil, g, s));
    } else {
      // one level-1 product at a time through the level-2 sums region and M2
      const int h2 = hh / 2, nt2 = h2 / TILE;
      int4 ops[7];
      level1_ops(ops, 0, hh, KQ2);
      for (int q = 0; q < 7; ++q) {
        const int4 o = ops[q];
        const int raw_x = o.y < 2 * KQ2, raw_y = o.w < 2 * KQ2;   // operands in the rows of A, not sums
        SumsArgs s2{h2, KQ2 / 2, 4 * hh, pairs * h2, o.x, o.y, o.z, o.w, 0, 4 * KQ2, 2 * hh, 4 * KQ2, raw_x, raw_y};
        winograd_sums2_kernel<<<dim3(KQ2 / 2, (s2.count + 255) / 256), 256, 0, s>>>(h->Atil4, h->n_pad, s2, f.colexp);
        CIP_CHECK_LAUNCH();
        GemmArgs g2 = g;
        g2.ntm = g2.ntn = nt2;
        g2.nk = f.K2 / 64;
        g2.Ctm = f.M2;
        g2.group = f.table + 2 * sub_entry;
        g2.group_tiles = nt2 * nt2;
        g2.tile_count = 7 * pairs * nt2 * nt2;
        sub_entry += 7 * pairs;
        CIP_TRY(launch_gemm_nt(h->mapAtil, h->mapAtil, g2, s));
        winograd_combine2_kernel<<<dim3(nt2 * nt2, pairs), 256, 0, s>>>(f.M2, f.M, h2, q, 4 * hh, o.x, o.z, raw_x,
                                                                        raw_y, f.colexp);
        CIP_CHECK_LAUNCH();
      }
    }
    winograd_combine_kernel<<<dim3(nt * nt, pairs), 256, 0, s>>>(f.M, cin, h->H4, h->n_pad, hh, two, f.colexp);
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
