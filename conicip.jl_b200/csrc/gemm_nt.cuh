// gemm_nt: the one FP64 tensor-core tile kernel behind K1 (scaled SYRK), K2 (Cholesky
// panel TRSM + trailing update) and the Schur-complement block.
//
//     C[i, j] = Cin[i, j] + alpha * sum_k X[i, k] * Y[j, k]       ("NT": both operands K-major)
//
// X, Y, Cin, Cout are all in the Q4 quad-interleaved layout (common.cuh).
// Replaces the reference's BLAS calls at src/kktsolvers.jl:33-34 (`Atil'Atil` -> dsyrk),
// :290 (`A'*(F^-T'*(F^-T*A))`) and the LAPACK factorisation at :35 / :295.
#pragma once
#include "common.cuh"

namespace cip {

struct GemmOperand {
  CUtensorMap map;  // 2-D: dim0 = ld*4 doubles (quad-interleaved rows), dim1 = K/4 quads
};

struct GemmArgs {
  // tile grid
  int lower;     // 1: only tiles ti >= tj of an nt x nt grid (SYRK / trailing update); 0: ntm x ntn
  int ntm, ntn;  // tile counts (lower: ntm == ntn)
  int sym;       // 1: X and Y are the same operand with the same origin (diagonal tiles load once)
  // operand origins
  int x_row0, y_row0;  // first row of tile (0, .) in X / Y
  int x_kq0, y_kq0;    // first k-quad in X / Y
  int nk;              // number of KT-wide k tiles
  // C
  const double* Cin;   // may be nullptr (treated as 0)
  double* Cout;
  int ldc;             // Q4 ld of C
  int c_row0, c_col0;  // C origin
  double alpha;
  // split-K tail.  The tile grid runs in waves of 148 CTAs; the tiles of the last, partial wave (all of
  // them when the grid is smaller than one wave: tall-skinny products with a handful of C tiles and a
  // very long contraction) are cut into `ksplit` contraction ranges so that the tail fills the SMs.
  // Each tail CTA writes its partial tile to ws[((tile - tail0) * ksplit + split) * 128*128 ...] and a
  // second kernel adds the partials in split order (deterministic) onto Cin.  Only used when `ws` is set.
  double* ws;          // workspace, may be nullptr (never split)
  long long ws_doubles;
  int tail0;           // filled in by launch_gemm_nt: first split tile (CTAs below it contract all of K)
  int ksplit, kchunk;  //   number of splits of a tail tile, k tiles per split
  // Tile-major output in ranges (row-sharded SYRK: the partial Gram matrix is all-reduced range by range while
  // later ranges are still being computed).  The launch covers the linear tile indices [tile_begin, tile_begin +
  // tile_count) (tile_count = 0: all); with `Ctm` set, tile t is written to Ctm + t * 128*128 in tile-local Q4
  // (ld = 128) instead of Cout; `reverse` walks the triangular grid backwards (big row bands first), so that
  // the last range, whose all-reduce cannot hide behind compute, is the small tip of the triangle.
  int tile_begin, tile_count, reverse;
  double* Ctm;
  // Y tile is lower triangular (Y[j, k] = 0 for k > j, tile-aligned, nk = 4: the inverse of a diagonal block in
  // the Cholesky TRSM): a consumer warp skips the k tiles that only meet zeros of its 32 columns
  int y_lower_tri;
  int band;            // tile rows per band of the lower-triangular rasterisation (set by launch_gemm_nt)
  // Row scaling folded into the contraction (SYRK of an R-cone problem without a materialised Atil = F^-T A):
  // C += sum_k X[i,k] * kscale[k]^2 * Y[j,k].  The 32 factors of a k tile travel with it through the pipeline (one
  // 256-byte bulk copy per stage) and are applied to the Y fragments in registers.  nullptr: no scaling.
  const double* kscale;
  // Grouped launch (the fast SYRK, fast_syrk.cu): the grid holds several products of the same tile grid and nk, each
  // `group_tiles` consecutive linear tiles.  Linear tile t belongs to product e = t / group_tiles, whose origins come
  // from device memory: group[2e] = {x_row0, x_kq0, y_row0, y_kq0}, group[2e + 1] = {c_row0, c_col0, -, -} (the
  // fields above are ignored).  tile_count must then be set.  nullptr: one product.
  const int4* group;
  int group_tiles;
  // Q-cone scaling folded into the contraction (launch_gemm_nt_qfold): both operands are formed row by row as
  //     Atil[k, j] = qalpha[k] * X[j, k] + qg[k] * T[j, kt * qs + qslot[k]]        (kt = k / 32)
  // before the DMMAs, so C += Atil' Atil keeps the Gram form.  T (Q4, same ld as X) holds, for every 32-row k tile,
  // `qs` contraction rows: one per Q cone that meets the tile (the cone's b' D A row, cone_qfold_t), zero otherwise.
  // qalpha / qg / qslot cover every k row of the contraction (R rows: qg = 0).
  const double* qalpha;
  const double* qg;
  const uint8_t* qslot;
  int qs;
};
constexpr long long GEMM_WS_DOUBLES = 2048ll * 128 * 128;   // 2048 partial tiles (268 MB)

// Creates a tensor map over a Q4 matrix (ld rows, kq_total quads); box_kq: quads of contraction per TMA box
// (0: the gemm_nt k tile, 8 quads).
int make_q4_tensor_map(CUtensorMap* out, const double* base, int ld, long long kq_total, int box_kq = 0);

// Launch on `stream`.
int launch_gemm_nt(const GemmOperand& X, const GemmOperand& Y, const GemmArgs& a, cudaStream_t stream);

// The symmetric SYRK C = Cin + Atil' Atil with the Q-cone scaling folded in (GemmArgs::qalpha ..): X is the only
// operand (a.sym = 1, a.lower = 1), T its slot rows, mapped with box_kq = a.qs / 4.  a.qs must be a value of
// gemm_qfold_slots: 4 (three pipeline stages), 8, 12 or 16 (two).
int launch_gemm_nt_qfold(const GemmOperand& X, const GemmOperand& T, const GemmArgs& a, cudaStream_t stream);
// the slot count a k tile meeting `need` distinct Q cones is given: `need` rounded up to a whole quad (0: above 16)
int gemm_qfold_slots(int need);

// Cout (Q4, ldc) <- the tile-major tiles [tile_begin, tile_begin + tile_count) of Ctm (same grid description as the launch)
int unpack_tile_major(const GemmArgs& a, cudaStream_t stream);

int gemm_nt_smem_bytes();

}  // namespace cip
