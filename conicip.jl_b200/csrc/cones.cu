// Cone kernels K5-K8: Nesterov-Todd scaling, block apply, max step, Jordan product / division,
// and the scaled panel Atil = F^-T A.  R rows are elementwise (vectorised grid-stride); each
// Q cone is handled by one warp (or one 256-thread group for very large cones) with warp
// reductions.  Replaces src/ConicIP.jl:165-194 (nestod_soc), :212-270 (maxstep_rp/soc),
// :305-345 (drp/xrp/dsoc/xsoc), :571-665 (closures) and src/blockmatrices.jl:107-131 (Block*x).
#include <math_constants.h>

#include "kernels.cuh"
#include "../../include/conicip_b200.h"

namespace cip {

namespace {

// ---- group reductions: G == 32 -> one warp per cone; G == 256 -> one CTA per cone
template <int G>
__device__ __forceinline__ double group_sum(double v, double* sm) {
  v = warp_sum(v);
  if (G == 32) return v;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sm[w] = v;
  __syncthreads();
  double t = 0;
#pragma unroll
  for (int i = 0; i < G / 32; ++i) t += sm[i];
  return t;
}

// order-preserving map double -> uint64 for atomicMin
__device__ __forceinline__ unsigned long long dkey(double x) {
  unsigned long long u = (unsigned long long)__double_as_longlong(x);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

// generic inverse of a flattened scaling (used by cip_factor / cip_set_scaling)
__global__ void inv_diag_kernel(ConeDesc c, Scaling F, Scaling Fi) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < c.m; i += gridDim.x * blockDim.x) {
    const int kd = F.kind[c.row_cone[i]];
    if (kd == CIP_BLK_VECCONG) {          // handled by the S-cone kernels; keep the flat part inert
      F.a[i] = 0.0; F.b[i] = 0.0; Fi.a[i] = 0.0; Fi.b[i] = 0.0;
      continue;
    }
    const double ia = 1.0 / F.a[i];
    Fi.a[i] = ia;
    Fi.b[i] = (kd == CIP_BLK_WOODBURY) ? ia * F.b[i] : 0.0;
  }
}
__global__ void inv_wood_kernel(ConeDesc c, Scaling F, Scaling Fi) {
  // one warp per cone (any type); only kind-1 blocks do work
  const int ci = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (ci >= c.ncones) return;
  if (lane == 0) Fi.kind[ci] = F.kind[ci];
  if (F.kind[ci] != CIP_BLK_WOODBURY) {
    if (lane == 0) Fi.D[ci] = 0.0;
    return;
  }
  const int off = c.off[ci], dim = c.off[ci + 1] - off;
  double bib = 0;
  for (int i = lane; i < dim; i += 32) bib += F.b[off + i] * (F.b[off + i] / F.a[off + i]);
  bib = warp_sum(bib);
  if (lane == 0) Fi.D[ci] = 1.0 / (-1.0 / F.D[ci] - bib);
}

// ================================================================= max step helpers
__device__ __forceinline__ double rp_candidate(double x, const double* d, size_t i, double d_scale) {
  if (d) {
    const double di = d[i] / d_scale;
    return di > 0 ? x / di : CUDART_INF;                           // maxstep_rp, :212-225
  }
  return x > 0 ? 0.0 : -1.0 + x;                                   // :227-240
}
// ================================================================= scaled panel  Atil = F^-T A
__global__ void __launch_bounds__(256)
scale_panel_diag_kernel(const double* __restrict__ At4, double* __restrict__ Atil4, int ld,
                        const double* __restrict__ ia) {
  const int kq = blockIdx.x;
  const double2 s0 = *reinterpret_cast<const double2*>(ia + 4 * kq);
  const double2 s1 = *reinterpret_cast<const double2*>(ia + 4 * kq + 2);
  const size_t base = (size_t)kq * ld * 4;
  for (int j = blockIdx.y * blockDim.x + threadIdx.x; j < ld; j += gridDim.y * blockDim.x) {
    const double2* in = reinterpret_cast<const double2*>(At4 + base + (size_t)j * 4);
    double2 v0 = __ldg(in), v1 = __ldg(in + 1);
    v0.x *= s0.x; v0.y *= s0.y; v1.x *= s1.x; v1.y *= s1.y;
    double2* out = reinterpret_cast<double2*>(Atil4 + base + (size_t)j * 4);
    out[0] = v0;
    out[1] = v1;
  }
}
// The same pass for the fast SYRK (R rows only), which also needs the column norms of Atil: block (k chunk, 256
// columns), a thread walks SCALE_KQ_CHUNK quads of one column and leaves its sum of squares in
// colss[chunk * ld + j], which col_exponent_kernel reduces in a fixed order (deterministic).
constexpr int SCALE_KQ_CHUNK = 256;
__global__ void __launch_bounds__(256)
scale_panel_diag_norms_kernel(const double* __restrict__ At4, double* __restrict__ Atil4, int ld, int kq_total,
                              const double* __restrict__ ia, double* __restrict__ colss) {
  const int j = blockIdx.y * blockDim.x + threadIdx.x;
  const int kq0 = blockIdx.x * SCALE_KQ_CHUNK;
  const int kq1 = min(kq0 + SCALE_KQ_CHUNK, kq_total);
  double ss = 0.0;
#pragma unroll 4
  for (int kq = kq0; kq < kq1; ++kq) {
    const double2 s0 = *reinterpret_cast<const double2*>(ia + 4 * kq);
    const double2 s1 = *reinterpret_cast<const double2*>(ia + 4 * kq + 2);
    const size_t at = ((size_t)kq * ld + j) * 4;
    const double2* in = reinterpret_cast<const double2*>(At4 + at);
    double2 v0 = __ldg(in), v1 = __ldg(in + 1);
    v0.x *= s0.x; v0.y *= s0.y; v1.x *= s1.x; v1.y *= s1.y;
    double2* out = reinterpret_cast<double2*>(Atil4 + at);
    out[0] = v0;
    out[1] = v1;
    ss += v0.x * v0.x + v0.y * v0.y + v1.x * v1.x + v1.y * v1.y;
  }
  colss[(size_t)blockIdx.x * ld + j] = ss;
}
// e_j = round(log2 ||Atil[:, j]||), clamped to +-500 so that 2^-(e_i + e_j) stays a normal number (0 for a zero column)
__global__ void __launch_bounds__(256)
col_exponent_kernel(const double* __restrict__ colss, int nchunk, int ld, int* __restrict__ colexp) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= ld) return;
  double ss = 0.0;
  for (int c = 0; c < nchunk; ++c) ss += colss[(size_t)c * ld + j];
  int e = 0;
  if (ss > 0.0 && isfinite(ss)) e = max(-500, min(500, (int)lrint(0.5 * log2(ss))));
  colexp[j] = e;
}
__global__ void __launch_bounds__(128)
scale_panel_wood_kernel(ConeDesc c, Scaling Fi, const double* __restrict__ At4, double* __restrict__ Atil4,
                        int ld, int ncols) {
  // block (column chunk, cone): thread per column j of A; adds D * b (b' A[:, j]) over the cone's rows
  const int ci = c.qlist[blockIdx.x];
  if (Fi.kind[ci] != CIP_BLK_WOODBURY) return;
  const int j = blockIdx.y * blockDim.x + threadIdx.x;
  if (j >= ncols) return;
  const int off = c.off[ci], end = c.off[ci + 1];
  double dot = 0;
  for (int k = off; k < end; ++k) dot += Fi.b[k] * At4[q4_index(j, k, ld)];
  dot *= Fi.D[ci];
  for (int k = off; k < end; ++k) Atil4[q4_index(j, k, ld)] += Fi.b[k] * dot;
}

// block (cone, 128 columns), thread per column j: the Woodbury dot of scale_panel_wood_kernel, in the same order,
// stored once per k tile of the cone instead of being added to every row
__global__ void __launch_bounds__(128)
qfold_t_kernel(ConeDesc c, Scaling Fi, const double* __restrict__ At4, int ld, int ncols,
               const uint8_t* __restrict__ qslot, int qs, double* __restrict__ T4) {
  const int ci = c.qlist[blockIdx.x];
  const int j = blockIdx.y * blockDim.x + threadIdx.x;
  if (j >= ncols) return;
  const int off = c.off[ci], end = c.off[ci + 1];
  double dot = 0;
  if (Fi.kind[ci] == CIP_BLK_WOODBURY) {
    for (int k = off; k < end; ++k) dot += Fi.b[k] * At4[q4_index(j, k, ld)];
    dot *= Fi.D[ci];
  }
  for (int kt = off / 32; kt * 32 < end; ++kt) {
    const int r = kt * 32 > off ? kt * 32 : off;
    T4[q4_index(j, kt * qs + qslot[r], ld)] = dot;
  }
}

inline int nblocks(int n, int per) {
  int b = (n + per - 1) / per;
  const int cap = sm_count() * 16;
  return b < 1 ? 1 : (b > cap ? cap : b);
}

// ================================================================= fused R + Q kernels
// One launch covers every R row and every Q cone of a call (the S cones, if any, take one more launch in sdp.cu):
// blocks [0, nbR) walk the rows that are not in Q cones (grid-stride, 16-byte vectorised when every row is an R
// row), blocks [nbR, nbR + nbQ) take the Q cones, one cone per group of G threads.  G = 8 for small cones (up to 64
// rows: four cones per warp, three shuffle steps per reduction, no idle lanes at dimension 33), 32 up to 1024
// rows, 256 (one CTA per cone) above.
template <int G>
__device__ __forceinline__ double gsum(double v, double* sm) {
  if (G == 8) {
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
  }
  return group_sum<G>(v, sm);
}
// cone of this group; inactive groups (beyond the last cone) keep running with dim = 0 so that the warp-wide
// shuffles stay convergent
template <int G>
__device__ __forceinline__ bool q_group(const ConeDesc& c, int bq, int& ci, int& off, int& dim, int& lid) {
  const int per_block = blockDim.x / G;
  const int qi = bq * per_block + threadIdx.x / G;
  lid = threadIdx.x % G;
  ci = 0; off = 0; dim = 0;
  if (qi >= c.nq) return false;
  ci = c.qlist[qi];
  off = c.off[ci];
  dim = c.off[ci + 1] - off;
  return true;
}
struct RQGrid { int nbR, nbQ, G; };
inline RQGrid rq_grid(const ConeDesc& c) {
  RQGrid g;
  g.G = c.max_q_dim > 1024 ? 256 : (c.max_q_dim > 64 ? 32 : 8);
  g.nbQ = c.nq > 0 ? (c.nq + (256 / g.G) - 1) / (256 / g.G) : 0;
  const bool all_r = (c.nq + c.ns == 0);
  g.nbR = all_r ? nblocks(c.m / 2 + 1, 256) : ((c.nr_rows + c.ns > 0) ? nblocks(c.m, 256) : 0);
  return g;
}
#define RQ_LAUNCH(kernel, c, st, ...)                                                         \
  do {                                                                                        \
    const RQGrid g_ = rq_grid(c);                                                             \
    if (g_.nbR + g_.nbQ > 0) {                                                                \
      if (g_.G == 256) kernel<256><<<g_.nbR + g_.nbQ, 256, 0, st>>>(g_.nbR, __VA_ARGS__);     \
      else if (g_.G == 32) kernel<32><<<g_.nbR + g_.nbQ, 256, 0, st>>>(g_.nbR, __VA_ARGS__);  \
      else kernel<8><<<g_.nbR + g_.nbQ, 256, 0, st>>>(g_.nbR, __VA_ARGS__);                   \
      CIP_CHECK_LAUNCH();                                                                     \
    }                                                                                         \
  } while (0)

// ---- NT scaling (nt_scaling closure, src/ConicIP.jl:589-605; nestod_soc :165-194)
template <int G>
__global__ void __launch_bounds__(256)
nt_rq_kernel(int nbR, ConeDesc c, const double* __restrict__ v, const double* __restrict__ s, Scaling F, Scaling Fi,
             double* __restrict__ lambda) {
  __shared__ double sm[8];
  if ((int)blockIdx.x < nbR) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = nbR * blockDim.x;
    for (int i = tid; i < c.ncones; i += nth) {               // block kinds of the R cones (Q cones: below)
      if (c.type[i] == CIP_CONE_R) { F.kind[i] = CIP_BLK_DIAG; Fi.kind[i] = CIP_BLK_DIAG; F.D[i] = 0.0; Fi.D[i] = 0.0; }
    }
    if (c.nq + c.ns == 0) {                                   // every row is an R row: two rows per step, no lookups
      const int m2 = c.m >> 1;
      for (int i = tid; i < m2; i += nth) {
        const double2 vv = reinterpret_cast<const double2*>(v)[i], ss = reinterpret_cast<const double2*>(s)[i];
        const double2 f = make_double2(sqrt(ss.x / vv.x), sqrt(ss.y / vv.y));
        reinterpret_cast<double2*>(F.a)[i] = f;
        reinterpret_cast<double2*>(F.b)[i] = make_double2(0.0, 0.0);
        reinterpret_cast<double2*>(Fi.a)[i] = make_double2(1.0 / f.x, 1.0 / f.y);
        reinterpret_cast<double2*>(Fi.b)[i] = make_double2(0.0, 0.0);
        reinterpret_cast<double2*>(lambda)[i] = make_double2(f.x * vv.x, f.y * vv.y);
      }
      if ((c.m & 1) && tid == 0) {
        const int i = c.m - 1;
        const double f = sqrt(s[i] / v[i]);
        F.a[i] = f; F.b[i] = 0.0; Fi.a[i] = 1.0 / f; Fi.b[i] = 0.0; lambda[i] = f * v[i];
      }
      return;
    }
    for (int i = tid; i < c.m; i += nth) {
      const int ty = c.type[c.row_cone[i]];
      if (ty == CIP_CONE_S) { F.a[i] = 0.0; F.b[i] = 0.0; Fi.a[i] = 0.0; Fi.b[i] = 0.0; }
      if (ty != CIP_CONE_R) continue;
      const double f = sqrt(s[i] / v[i]);                     // Diagonal(sqrt.(yI./xI)), src/ConicIP.jl:598
      F.a[i] = f; F.b[i] = 0.0; Fi.a[i] = 1.0 / f; Fi.b[i] = 0.0;
      lambda[i] = f * v[i];
    }
    return;
  }
  int ci, off, dim, lid;
  const bool on = q_group<G>(c, blockIdx.x - nbR, ci, off, dim, lid);
  if (G == 256 && !on) return;
  const double* z = v + off;     // nestod_soc(z = v_I, s = s_I), src/ConicIP.jl:599
  const double* sv = s + off;
  double zz = 0, ss = 0;
  for (int i = lid; i < dim; i += G) { zz += z[i] * z[i]; ss += sv[i] * sv[i]; }
  zz = gsum<G>(zz, sm);
  ss = gsum<G>(ss, sm);
  const double z0 = on ? z[0] : 1.0, s0 = on ? sv[0] : 1.0;
  const double qfz = on ? 2 * z0 * z0 - zz : 1.0;             // QF, src/ConicIP.jl:160
  const double qfs = on ? 2 * s0 * s0 - ss : 1.0;
  const double beta = sqrt(sqrt(qfs / qfz));                  // (QF(s)/QF(z))^(1/4)
  // normalisation by multiplication with the reciprocals (one division per cone instead of four per
  // element; differs from the reference's elementwise z/sqrt(QF(z)) in the last bit only)
  const double irz = 1.0 / sqrt(qfz), irs = 1.0 / sqrt(qfs);
  double zs = 0;
  for (int i = lid; i < dim; i += G) zs += (z[i] * irz) * (sv[i] * irs);
  zs = gsum<G>(zs, sm);
  const double gamma = sqrt((1 + zs) / 2);
  const double inv2g = 1.0 / (2.0 * gamma);
  // w = (s + Jz)/(2 gamma); w1 += 1; w *= sqrt(2 beta)/sqrt(2 w1)
  const double w1 = inv2g * (s0 * irs + z0 * irz) + 1.0;
  const double scal = sqrt(2 * beta) / sqrt(2 * w1);
  double wv = 0, bib = 0;
  for (int i = lid; i < dim; i += G) {
    const double zi = z[i] * irz, si = sv[i] * irs;
    const double w = (i == 0) ? w1 * scal : (inv2g * (si - zi)) * scal;
    const double a = (i == 0) ? -beta : beta;
    F.a[off + i] = a;
    F.b[off + i] = w;
    const double ia = 1.0 / a;                   // Woodbury inverse: W = inv(A), X = W*B
    Fi.a[off + i] = ia;
    Fi.b[off + i] = ia * w;
    wv += w * z[i];
    bib += w * (ia * w);
  }
  wv = gsum<G>(wv, sm);
  bib = gsum<G>(bib, sm);
  for (int i = lid; i < dim; i += G) {                             // lambda = F*v, w recomputed (no re-read)
    const double w = (i == 0) ? w1 * scal : (inv2g * (sv[i] * irs - z[i] * irz)) * scal;
    lambda[off + i] = ((i == 0) ? -beta : beta) * z[i] + w * wv;
  }
  if (on && lid == 0) {
    F.kind[ci] = CIP_BLK_WOODBURY; Fi.kind[ci] = CIP_BLK_WOODBURY;
    F.D[ci] = 1.0;
    Fi.D[ci] = 1.0 / (-1.0 - bib);               // Z = inv(-inv(D) - B'X), D = 1
  }
}

// ---- block apply  y = M x  or, twice == 1,  y = M (M x)  (M = diag(a) + D b b' per cone, symmetric), and with
//      `minus`: y = minus - (that).  Block*x of src/blockmatrices.jl:107-131; the pair is the F^-T F^-T v of
//      src/kktsolvers.jl:326,328 in one pass.
template <int G>
__global__ void __launch_bounds__(256)
apply_rq_kernel(int nbR, ConeDesc c, Scaling S, const double* __restrict__ x, double* __restrict__ y, int twice,
                const double* __restrict__ minus) {
  __shared__ double sm[8];
  if ((int)blockIdx.x < nbR) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = nbR * blockDim.x;
    if (c.nq + c.ns == 0) {
      const int m2 = c.m >> 1;
      for (int i = tid; i < m2; i += nth) {
        const double2 a = reinterpret_cast<const double2*>(S.a)[i], xx = reinterpret_cast<const double2*>(x)[i];
        double2 r = make_double2(a.x * xx.x, a.y * xx.y);
        if (twice) { r.x *= a.x; r.y *= a.y; }
        if (minus) { const double2 z = reinterpret_cast<const double2*>(minus)[i]; r.x = z.x - r.x; r.y = z.y - r.y; }
        reinterpret_cast<double2*>(y)[i] = r;
      }
      if ((c.m & 1) && tid == 0) {
        const int i = c.m - 1;
        double r = S.a[i] * x[i];
        if (twice) r *= S.a[i];
        y[i] = minus ? minus[i] - r : r;
      }
      return;
    }
    for (int i = tid; i < c.m; i += nth) {
      if (c.type[c.row_cone[i]] == CIP_CONE_Q) continue;      // (S rows: a = 0; sdp_apply writes them afterwards)
      double r = S.a[i] * x[i];
      if (twice) r *= S.a[i];
      y[i] = minus ? minus[i] - r : r;
    }
    return;
  }
  int ci, off, dim, lid;
  const bool on = q_group<G>(c, blockIdx.x - nbR, ci, off, dim, lid);
  if (G == 256 && !on) return;
  const bool wood = on && S.kind[ci] == CIP_BLK_WOODBURY;
  const double D = wood ? S.D[ci] : 0.0;
  double bx = 0;
  for (int i = lid; i < dim; i += G) bx += S.b[off + i] * x[off + i];
  bx = gsum<G>(bx, sm) * D;
  if (!twice) {
    for (int i = lid; i < dim; i += G) {
      const double r = S.a[off + i] * x[off + i] + S.b[off + i] * bx;     // A*x + B*(D*(B'x))
      y[off + i] = minus ? minus[off + i] - r : r;
    }
    return;
  }
  double bt = 0;                                                           // b' t with t = M x
  for (int i = lid; i < dim; i += G) bt += S.b[off + i] * (S.a[off + i] * x[off + i] + S.b[off + i] * bx);
  bt = gsum<G>(bt, sm) * D;
  for (int i = lid; i < dim; i += G) {
    const double tt = S.a[off + i] * x[off + i] + S.b[off + i] * bx;
    const double r = S.a[off + i] * tt + S.b[off + i] * bt;
    y[off + i] = minus ? minus[off + i] - r : r;
  }
}

// ---- Jordan product / division (cone_prod!, cone_div!: src/ConicIP.jl:622-665, :305-345)
template <int G>
__global__ void __launch_bounds__(256)
prod_rq_kernel(int nbR, ConeDesc c, const double* __restrict__ x, const double* __restrict__ y, double* __restrict__ o,
               int divide) {
  __shared__ double sm[8];
  if ((int)blockIdx.x < nbR) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = nbR * blockDim.x;
    if (c.nq + c.ns == 0) {
      const int m2 = c.m >> 1;
      for (int i = tid; i < m2; i += nth) {
        const double2 a = reinterpret_cast<const double2*>(x)[i], b = reinterpret_cast<const double2*>(y)[i];
        reinterpret_cast<double2*>(o)[i] = divide ? make_double2(a.x / b.x, a.y / b.y) : make_double2(a.x * b.x, a.y * b.y);
      }
      if ((c.m & 1) && tid == 0) o[c.m - 1] = divide ? x[c.m - 1] / y[c.m - 1] : x[c.m - 1] * y[c.m - 1];
      return;
    }
    for (int i = tid; i < c.m; i += nth) {
      if (c.type[c.row_cone[i]] != CIP_CONE_R) continue;
      o[i] = divide ? x[i] / y[i] : x[i] * y[i];             // drp! / xrp!, src/ConicIP.jl:305-315
    }
    return;
  }
  int ci, off, dim, lid;
  const bool on = q_group<G>(c, blockIdx.x - nbR, ci, off, dim, lid);
  if (G == 256 && !on) return;
  const double* xp = x + off;
  const double* yp = y + off;
  if (!divide) {                                                // xsoc!, :340-345
    double d = 0;
    for (int i = lid; i < dim; i += G) d += xp[i] * yp[i];
    d = gsum<G>(d, sm);
    const double x0 = on ? xp[0] : 0.0, y0 = on ? yp[0] : 0.0;
    for (int i = lid; i < dim; i += G) o[off + i] = (i == 0) ? d : x0 * yp[i] + y0 * xp[i];
    return;
  }
  // o = arrow(y)^-1 x   (dsoc!(y = x_arg, x = y_arg, o), src/ConicIP.jl:317-338)
  double ybyb = 0, ybxb = 0;
  for (int i = lid; i < dim; i += G) {
    if (i > 0) { ybyb += yp[i] * yp[i]; ybxb += yp[i] * xp[i]; }
  }
  ybyb = gsum<G>(ybyb, sm);
  ybxb = gsum<G>(ybxb, sm);
  const double y1 = on ? yp[0] : 1.0, x1 = on ? xp[0] : 0.0;
  const double alpha = y1 * y1 - ybyb;
  const double b1 = (-x1 / alpha) + ybxb / (y1 * alpha);
  const double b2 = 1.0 / y1;
  for (int i = lid; i < dim; i += G) o[off + i] = (i == 0) ? (y1 * x1 - ybxb) / alpha : yp[i] * b1 + xp[i] * b2;
}

// ---- max step (maxstep closure src/ConicIP.jl:571-587; maxstep_rp :212-240, maxstep_soc :242-270).  *key is preset
//      to all ones ("nothing seen" = +Inf) by a memset; every CTA issues at most one atomicMin on the
//      order-preserving integer image of its minimum (exact and order independent).
template <int G>
__global__ void __launch_bounds__(256)
maxstep_rq_kernel(int nbR, ConeDesc c, const double* __restrict__ x, const double* __restrict__ d, double d_scale,
                  unsigned long long* key) {
  __shared__ double sm[8];
  __shared__ double smin[8];
  double best = CUDART_INF;
  if ((int)blockIdx.x < nbR) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = nbR * blockDim.x;
    if (c.nq + c.ns == 0) {
      const int m2 = c.m >> 1;
      for (int i = tid; i < m2; i += nth) {
        const double2 xx = reinterpret_cast<const double2*>(x)[i];
        if (d) {
          const double2 dd = reinterpret_cast<const double2*>(d)[i];
          const double d0 = dd.x / d_scale, d1 = dd.y / d_scale;
          if (d0 > 0) best = fmin(best, xx.x / d0);
          if (d1 > 0) best = fmin(best, xx.y / d1);
        } else {
          best = fmin(best, fmin(xx.x > 0 ? 0.0 : -1.0 + xx.x, xx.y > 0 ? 0.0 : -1.0 + xx.y));
        }
      }
      if ((c.m & 1) && tid == 0) best = fmin(best, rp_candidate(x[c.m - 1], d, c.m - 1, d_scale));
    } else {
      for (int i = tid; i < c.m; i += nth) {
        if (c.type[c.row_cone[i]] != CIP_CONE_R) continue;
        best = fmin(best, rp_candidate(x[i], d, i, d_scale));
      }
    }
    best = warp_min(best);
  } else {
    const int per_block = blockDim.x / G, lid = threadIdx.x % G;
    const double ids = d ? -1.0 / d_scale : 0.0;                    // d <- -d / d_scale
    const int qi = (blockIdx.x - nbR) * per_block + threadIdx.x / G;
    const bool on = qi < c.nq;
    if (G == 256 && !on) return;
    const int ci = on ? c.qlist[qi] : 0, off = on ? c.off[ci] : 0, dim = on ? c.off[ci + 1] - off : 0;
    const double* xp = x + off;
    double res;
    if (!d) {                                                      // maxstep_soc(x, nothing), :264-270
      double nn = 0;
      for (int i = lid; i < dim; i += G) if (i > 0) nn += xp[i] * xp[i];
      nn = gsum<G>(nn, sm);
      const double al = sqrt(nn) - (on ? xp[0] : 1.0);
      res = al < 0 ? 0.0 : -1.0 - al;
    } else if (G == 8) {                                           // maxstep_soc(x, d), :242-262; cone <= 64 rows:
      const double* dp = d + off;                                  // one pass over memory, x and d stay in registers
      double xr[8], dr[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int i = lid + 8 * e;
        xr[e] = i < dim ? xp[i] : 0.0;
        dr[e] = i < dim ? dp[i] * ids : 0.0;
      }
      double xx = 0, xdr = 0;
#pragma unroll
      for (int e = 0; e < 8; ++e) xx += xr[e] * xr[e];
      xx = gsum<G>(xx, sm);
      const double x0 = __shfl_sync(0xffffffffu, xr[0], threadIdx.x & 24);      // element 0 lives in lane 0 of the group
      const double d0 = __shfl_sync(0xffffffffu, dr[0], threadIdx.x & 24);
      const double gam = on ? 2 * x0 * x0 - xx : 1.0;
      const double irg = 1.0 / sqrt(gam);
#pragma unroll
      for (int e = 0; e < 8; ++e) xdr += (xr[e] * irg) * dr[e];
      const double xd = gsum<G>(xdr, sm);
      const double xb0 = x0 * irg;
      const double beta = 2 * xb0 * d0 - xd;
      const double rho1 = beta * irg;
      const double mu = (beta + d0) / (xb0 + 1);
      double r2 = 0;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const double r = dr[e] - mu * (xr[e] * irg);
        if (lid + 8 * e > 0 && lid + 8 * e < dim) r2 += r * r;
      }
      r2 = gsum<G>(r2, sm);
      const double al = sqrt(r2) * irg - rho1;
      res = al < 0 ? CUDART_INF : 1.0 / al;
    } else {                                                       // maxstep_soc(x, d), :242-262
      const double* dp = d + off;
      double xx = 0, xdr = 0;
      for (int i = lid; i < dim; i += G) { xx += xp[i] * xp[i]; }
      xx = gsum<G>(xx, sm);
      const double x0 = on ? xp[0] : 1.0;
      const double gam = on ? 2 * x0 * x0 - xx : 1.0;
      const double irg = 1.0 / sqrt(gam);
      const double d0 = on ? dp[0] * ids : 0.0;
      for (int i = lid; i < dim; i += G) xdr += (xp[i] * irg) * (dp[i] * ids);
      const double xd = gsum<G>(xdr, sm);
      const double xb0 = x0 * irg;
      const double beta = 2 * xb0 * d0 - xd;
      const double rho1 = beta * irg;
      const double mu = (beta + d0) / (xb0 + 1);
      double r2 = 0;
      for (int i = lid; i < dim; i += G) {
        if (i > 0) {
          const double r = dp[i] * ids - mu * (xp[i] * irg);
          r2 += r * r;
        }
      }
      r2 = gsum<G>(r2, sm);
      const double al = sqrt(r2) * irg - rho1;
      res = al < 0 ? CUDART_INF : 1.0 / al;
    }
    best = on ? res : CUDART_INF;
    if (G == 8) best = warp_min(best);                             // four cones per warp
  }
  // CTA minimum through shared memory, one atomic per CTA
  if ((threadIdx.x & 31) == 0) smin[threadIdx.x >> 5] = best;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) best = fmin(best, smin[w]);
    // thousands of CTAs end here: look first (a plain L2 read) and only send the atomic when this CTA would lower
    // the minimum -- after the first few CTAs almost none does, so the same-address atomics no longer queue up
    if (best < CUDART_INF) {
      const unsigned long long mine = dkey(best);
      unsigned long long seen;
      asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(seen) : "l"(key) : "memory");
      if (mine < seen) atomicMin(key, mine);
    }
  }
}

}  // namespace

int cone_nt_scaling(const ConeDesc& c, const double* v, const double* s, Scaling F, Scaling Fi, double* lambda,
                    int* info, cudaStream_t st) {
  if (c.m == 0) return 0;
  RQ_LAUNCH(nt_rq_kernel, c, st, c, v, s, F, Fi, lambda);
  CIP_TRY(sdp_nt_scaling(c, F, Fi, v, s, lambda, info, st));
  return 0;
}

int cone_invert_scaling(const ConeDesc& c, Scaling F, Scaling Fi, cudaStream_t st) {
  if (c.m == 0) return 0;
  inv_diag_kernel<<<nblocks(c.m, 256), 256, 0, st>>>(c, F, Fi);
  CIP_CHECK_LAUNCH();
  inv_wood_kernel<<<(c.ncones + 7) / 8, 256, 0, st>>>(c, F, Fi);
  CIP_CHECK_LAUNCH();
  CIP_TRY(sdp_invert(c, F, st));
  return 0;
}

int cone_apply(const ConeDesc& c, const Scaling& F, const Scaling& Fi, int op, const double* x, double* y,
               cudaStream_t st) {
  if (c.m == 0) return 0;
  const bool inv = (op == CIP_OP_FINVT || op == CIP_OP_FINV);
  const Scaling& S = inv ? Fi : F;           // R / Q blocks are symmetric: F' = F
  RQ_LAUNCH(apply_rq_kernel, c, st, c, S, x, y, 0, (const double*)nullptr);
  // VecCongurance blocks: F -> R, F' -> R', inv(F) -> inv(R), inv(F)' -> inv(R)'
  CIP_TRY(sdp_apply(c, F, inv ? 1 : 0, (op == CIP_OP_FT || op == CIP_OP_FINVT) ? 1 : 0, x, y, st));
  return 0;
}

// y = inv(F) inv(F)' x  (= inv(F'F) x), optionally y = minus - that: the two block applies of src/kktsolvers.jl:326
// and :328 (and the subtraction of :328) in one launch for the R / Q cones; `tmp` (m doubles) is only used when
// there are S cones.
int cone_apply_invsq(const ConeDesc& c, const Scaling& F, const Scaling& Fi, const double* x, double* y,
                     const double* minus, double* tmp, cudaStream_t st) {
  if (c.m == 0) return 0;
  RQ_LAUNCH(apply_rq_kernel, c, st, c, Fi, x, y, 1, minus);
  if (c.ns > 0) {
    // VecCongurance blocks are not symmetric: inv(R)' first, then inv(R), on the S rows only
    CIP_TRY(sdp_apply(c, F, 1, 1, x, tmp, st));
    CIP_TRY(sdp_apply(c, F, 1, 0, tmp, y, st));
    if (minus) CIP_TRY(sdp_rows_rsub(c, F, minus, y, st));
  }
  return 0;
}

int cone_prod(const ConeDesc& c, const double* x, const double* y, double* o, cudaStream_t st) {
  if (c.m == 0) return 0;
  RQ_LAUNCH(prod_rq_kernel, c, st, c, x, y, o, 0);
  CIP_TRY(sdp_prod_div(c, x, y, o, 0, st));
  return 0;
}

int cone_div(const ConeDesc& c, const double* x, const double* y, double* o, cudaStream_t st) {
  if (c.m == 0) return 0;
  RQ_LAUNCH(prod_rq_kernel, c, st, c, x, y, o, 1);
  CIP_TRY(sdp_prod_div(c, x, y, o, 1, st));
  return 0;
}

int cone_maxstep(const ConeDesc& c, const double* x, const double* d, double d_scale, double* partial,
                 int npartial, double* result, cudaStream_t st) {
  (void)partial; (void)npartial;
  unsigned long long* key = reinterpret_cast<unsigned long long*>(result);
  CIP_CUDA(cudaMemsetAsync(key, 0xFF, sizeof(unsigned long long), st));      // "nothing seen": decoded as +Inf
  if (c.m == 0) return 0;
  RQ_LAUNCH(maxstep_rq_kernel, c, st, c, x, d, d_scale, key);
  CIP_TRY(sdp_maxstep(c, x, d, d_scale, key, st));
  return 0;
}

int cone_scale_panel(const ConeDesc& c, Scaling Fi, const double* At4, double* Atil4, int ld, int m_pad,
                     int ncols, cudaStream_t st) {
  if (m_pad == 0) return 0;
  dim3 grid(m_pad / 4, (ld + 255) / 256 > 8 ? 8 : (ld + 255) / 256);
  scale_panel_diag_kernel<<<grid, 256, 0, st>>>(At4, Atil4, ld, Fi.a);
  CIP_CHECK_LAUNCH();
  if (c.nq > 0) {
    dim3 g2(c.nq, (ncols + 127) / 128);
    scale_panel_wood_kernel<<<g2, 128, 0, st>>>(c, Fi, At4, Atil4, ld, ncols);
    CIP_CHECK_LAUNCH();
  }
  CIP_TRY(sdp_scale_panel(c, Fi, At4, Atil4, ld, ncols, st));
  return 0;
}

int cone_qfold_t(const ConeDesc& c, Scaling Fi, const double* At4, int ld, int ncols, const uint8_t* qslot, int qs,
                 double* T4, cudaStream_t st) {
  if (c.nq == 0 || ncols == 0) return 0;
  qfold_t_kernel<<<dim3(c.nq, (ncols + 127) / 128), 128, 0, st>>>(c, Fi, At4, ld, ncols, qslot, qs, T4);
  CIP_CHECK_LAUNCH();
  return 0;
}

int scale_panel_norms_chunks(int m_pad) { return (m_pad / 4 + SCALE_KQ_CHUNK - 1) / SCALE_KQ_CHUNK; }

int cone_scale_panel_norms(Scaling Fi, const double* At4, double* Atil4, int ld, int m_pad, double* colss,
                           int* colexp, cudaStream_t st) {
  const int nchunk = scale_panel_norms_chunks(m_pad);
  if (nchunk > 0) {
    dim3 grid(nchunk, ld / 256 > 0 ? ld / 256 : 1);
    if (ld % 256 != 0) {
      set_error("cone_scale_panel_norms: ld = %d is not a multiple of 256", ld);
      return -1;
    }
    scale_panel_diag_norms_kernel<<<grid, 256, 0, st>>>(At4, Atil4, ld, m_pad / 4, Fi.a, colss);
    CIP_CHECK_LAUNCH();
  }
  col_exponent_kernel<<<(ld + 255) / 256, 256, 0, st>>>(colss, nchunk, ld, colexp);
  CIP_CHECK_LAUNCH();
  return 0;
}

}  // namespace cip
