// FP64 tensor-core (DMMA.8x8x4) NT tile kernel, TMA + mbarrier pipeline, sm_100a.
// See gemm_nt.cuh for the contract.
//
// CTA = 9 warps: warp 8 is the TMA producer (one elected lane), warps 0..7 are DMMA
// consumers, each owning a 64 x 32 sub-tile of the 128 x 128 CTA tile (64 FP64
// accumulators per thread).  A stage is KT = 32 contraction steps: four TMA boxes
// (X rows 0-63, X rows 64-127, Y rows 0-63, Y rows 64-127), each {256 doubles, 8 quads}
// = 16 KB, landing in shared memory already in DMMA fragment order, so every operand
// fragment is one conflict-free 256-byte LDS.64.
#include "gemm_nt.cuh"

namespace cip {

namespace {
constexpr int BM = 128, BN = 128;
constexpr int KT = 32;
constexpr int KQ = KT / 4;
// Q-fold consumers unroll the 8 quads of a k tile by 2.  The T operands push the 168-register budget (9 warps, one
// CTA per SM) into spills in every unroll (ptxas -v at 2: 56-64 B stack, 84 B spill stores); measured on one B200 at the
// C3 shape (profiles/r07_fold_qcones.md), 2 is the fastest: SYRK +28 % over the materialised one, against +32 % at 1
// and +36 % fully unrolled (8).
constexpr int QUNROLL = 2;


constexpr int STAGES = 3;
constexpr int HALF = 64;
constexpr int BOX_DOUBLES = HALF * 4 * KQ;       // 2048 doubles
constexpr int BOX_BYTES = BOX_DOUBLES * 8;       // 16 KB
constexpr int STAGE_DOUBLES = 4 * BOX_DOUBLES;   // 64 KB
constexpr int CONSUMER_WARPS = 8;
constexpr int BAND_DEFAULT = 12;      // tile rows per band of the lower-triangular rasterisation (GemmArgs::band; CIP_GEMM_BAND)
constexpr int NUM_THREADS = (CONSUMER_WARPS + 1) * 32;
constexpr int SMEM_BYTES = STAGES * STAGE_DOUBLES * 8 + 128 + STAGES * KT * 8;   // tiles | barriers | k scales per stage
// Q-fold variant (QS slot rows of T per k tile, GemmArgs::qs: 4, 8, 12 or 16): the T slabs of X and Y sit between the
// tiles and the barriers; after the row factors (qalpha, in the k-scale slots) come qg and the slot bytes.  Three
// stages fit 4 slots only (3 x 72 KB); 8 to 16 slots run two.
__host__ __device__ constexpr int qf_stages(int qs) { return qs > 4 ? 2 : STAGES; }
__host__ __device__ constexpr int qf_tq_doubles(int qs) { return 4 * HALF * qs; }     // per stage: 2 operands x 2 halves
__host__ __device__ constexpr int qf_smem_bytes(int qs) {
  return qf_stages(qs) * (STAGE_DOUBLES + qf_tq_doubles(qs)) * 8 + 128 + qf_stages(qs) * KT * (8 + 8 + 1);
}
static_assert(qf_smem_bytes(4) <= 227 * 1024 && qf_smem_bytes(16) <= 227 * 1024, "Q-fold stage does not fit");

__device__ __forceinline__ void tile_of(const GemmArgs& a, int t, int& ti, int& tj) {
  if (a.lower) {
    if (a.reverse) t = a.ntm * (a.ntm + 1) / 2 - 1 - t;
    // Band rasterisation of the lower-triangular tile grid: bands of BAND tile rows, column-major
    // inside a band, so the ~148 concurrently resident CTAs cover ~BAND rows x ~148/BAND columns and
    // share their X / Y panels in L2 (instead of one long row of tiles with 148 distinct Y panels).
    const int BAND = a.band > 0 ? a.band : BAND_DEFAULT;
    int b = (int)((sqrtf(8.f * (float)t + 1.f) - 1.f) * 0.5f) / BAND;
    auto before = [BAND](int bb) { const long long R = (long long)bb * BAND; return R * (R + 1) / 2; };
    while (before(b + 1) <= t) ++b;
    while (before(b) > t) --b;
    const int r0 = b * BAND;
    const int h = (a.ntm - r0 < BAND) ? a.ntm - r0 : BAND;
    int local = t - (int)before(b);
    const int full = (r0 + 1) * h;
    if (local < full) {
      tj = local / h;
      ti = r0 + local % h;
    } else {
      local -= full;
      int u = 0, cnt = h - 1;
      while (local >= cnt) { local -= cnt; ++u; --cnt; }
      tj = r0 + 1 + u;
      ti = tj + local;
    }
  } else {
    ti = t % a.ntm;
    tj = t / a.ntm;
  }
}

// 1-D bulk copy global -> shared onto a stage's barrier (16-byte aligned, a multiple of 16 bytes)
__device__ __forceinline__ void bulk_load(const void* smem_dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// where linear tile `tile` of a launch sits: its tile coordinates and the origins of its product (GemmArgs::group)
struct TilePos {
  int ti, tj, x_row0, x_kq0, y_row0, y_kq0, c_row0, c_col0;
};
__device__ __forceinline__ TilePos locate(const GemmArgs& a, int tile) {
  TilePos p{0, 0, a.x_row0, a.x_kq0, a.y_row0, a.y_kq0, a.c_row0, a.c_col0};
  if (a.group) {
    const int e = tile / a.group_tiles;
    tile -= e * a.group_tiles;
    const int4 o = a.group[2 * e], c = a.group[2 * e + 1];
    p.x_row0 = o.x; p.x_kq0 = o.y; p.y_row0 = o.z; p.y_kq0 = o.w;
    p.c_row0 = c.x; p.c_col0 = c.y;
  }
  tile_of(a, tile, p.ti, p.tj);
  return p;
}

// QS = 0: X and Y through tmX / tmY (SCALED: the R-cone row factors of GemmArgs::kscale).  QS > 0: the Q-fold SYRK
// (launch_gemm_nt_qfold): X and Y both come through tmX, tmY maps the slot rows T, and both operands are formed as
// qalpha * A + qg * T before the DMMAs.
template <bool SCALED, int QS = 0>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_nt_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmY,
               const GemmArgs a) {
  constexpr int NST = QS > 0 ? qf_stages(QS) : STAGES;
  constexpr int TQ = QS > 0 ? qf_tq_doubles(QS) : 0;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  double* tiles = reinterpret_cast<double*>(smem_raw);
  double* tqs = tiles + (size_t)NST * STAGE_DOUBLES;                                                // [NST][TQ]
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)NST * (STAGE_DOUBLES + TQ) * 8);
  uint64_t* empty = full + NST;
  double* kscales = reinterpret_cast<double*>(smem_raw + (size_t)NST * (STAGE_DOUBLES + TQ) * 8 + 128);   // [NST][KT]
  double* qgs = kscales + NST * KT;                                                                 // [NST][KT]
  const uint8_t* qsl = reinterpret_cast<const uint8_t*>(qgs + NST * KT);                            // [NST][KT]

  // CTAs below tail0 own a whole tile; above it, ksplit consecutive CTAs share one (k tiles [kt0, kt1))
  const bool split = (int)blockIdx.x >= a.tail0 && a.ksplit > 1;
  const int tile = a.tile_begin + (split ? a.tail0 + ((int)blockIdx.x - a.tail0) / a.ksplit : (int)blockIdx.x);
  const int sp = split ? ((int)blockIdx.x - a.tail0) % a.ksplit : 0;
  const TilePos P = locate(a, tile);
  const int ti = P.ti, tj = P.tj;
  const int kt0 = split ? sp * a.kchunk : 0;
  const int kt1 = split ? ((kt0 + a.kchunk < a.nk) ? kt0 + a.kchunk : a.nk) : a.nk;
  const bool same = a.sym && (ti == tj);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < NST; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], CONSUMER_WARPS);
    }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp == CONSUMER_WARPS) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0 && kt1 > kt0) {
      tma_prefetch_desc(&tmX);
      tma_prefetch_desc(&tmY);
      const int xr = (P.x_row0 + ti * BM) * 4;
      const int yr = (P.y_row0 + tj * BN) * 4;
      const CUtensorMap* mY = QS > 0 ? &tmX : &tmY;        // (Q fold: one operand; tmY maps T)
      uint32_t bytes = (same ? 2u * BOX_BYTES : 4u * BOX_BYTES) + (SCALED ? (uint32_t)(KT * 8) : 0u);
      if (QS > 0) bytes += (same ? 2u : 4u) * (uint32_t)(HALF * QS * 8) + (uint32_t)(KT * (8 + 8 + 1));
      for (int kt = kt0; kt < kt1; ++kt) {
        const int s = (kt - kt0) % NST;
        const uint32_t ph = (uint32_t)((kt - kt0) / NST) & 1u;
        mbar_wait(&empty[s], ph ^ 1u);
        double* st = tiles + (size_t)s * STAGE_DOUBLES;
        mbar_arrive_expect_tx(&full[s], bytes);
        tma_load_2d(st, &tmX, &full[s], xr, P.x_kq0 + kt * KQ);
        tma_load_2d(st + BOX_DOUBLES, &tmX, &full[s], xr + HALF * 4, P.x_kq0 + kt * KQ);
        if (!same) {
          tma_load_2d(st + 2 * BOX_DOUBLES, mY, &full[s], yr, P.y_kq0 + kt * KQ);
          tma_load_2d(st + 3 * BOX_DOUBLES, mY, &full[s], yr + HALF * 4, P.y_kq0 + kt * KQ);
        }
        if (QS > 0) {
          // the S x 128 slot rows of T for the X (and Y) rows of this k tile, then qalpha / qg / slot of its 32 rows
          const int ktg = P.y_kq0 / KQ + kt;
          double* tq = tqs + (size_t)s * TQ;
          tma_load_2d(tq, &tmY, &full[s], xr, ktg * (QS / 4));
          tma_load_2d(tq + HALF * QS, &tmY, &full[s], xr + HALF * 4, ktg * (QS / 4));
          if (!same) {
            tma_load_2d(tq + 2 * HALF * QS, &tmY, &full[s], yr, ktg * (QS / 4));
            tma_load_2d(tq + 3 * HALF * QS, &tmY, &full[s], yr + HALF * 4, ktg * (QS / 4));
          }
          const size_t k0 = (size_t)ktg * KT;
          bulk_load(kscales + s * KT, a.qalpha + k0, KT * 8, &full[s]);
          bulk_load(qgs + s * KT, a.qg + k0, KT * 8, &full[s]);
          bulk_load(qsl + s * KT, a.qslot + k0, KT, &full[s]);
        }
        if (SCALED)      // the 32 row factors of this k tile (1-D bulk copy onto the same barrier)
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                           smem_u32(kscales + s * KT)),
                       "l"(a.kscale + (size_t)(P.y_kq0 + kt * KQ) * 4), "r"((uint32_t)(KT * 8)), "r"(smem_u32(&full[s]))
                       : "memory");
      }
    }
    return;
  }

  // -------------------------------------------------------------- DMMA consumers
  const int g = lane >> 2, t = lane & 3;
  const int warp_m = warp & 1, warp_n = warp >> 1;
  double acc[8][4][2];
#pragma unroll
  for (int mi = 0; mi < 8; ++mi)
#pragma unroll
    for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;

  const int x_off = warp_m * BOX_DOUBLES + g * 4 + t;
  const int y_off = (same ? 0 : 2 * BOX_DOUBLES) + (warp_n >> 1) * BOX_DOUBLES + ((warp_n & 1) * 32 + g) * 4 + t;

  // (Q fold) this thread's T rows: X rows g + 8 mi of its half, Y rows g + 8 ni of its 32 columns
  const int tx_off = warp_m * HALF * QS + g * 4;
  const int ty_off = (same ? 0 : 2 * HALF * QS) + (warp_n >> 1) * HALF * QS + ((warp_n & 1) * 32 + g) * 4;

  for (int kt = kt0; kt < kt1; ++kt) {
    const int s = (kt - kt0) % NST;
    const uint32_t ph = (uint32_t)((kt - kt0) / NST) & 1u;
    mbar_wait(&full[s], ph);
    const double* st = tiles + (size_t)s * STAGE_DOUBLES;
    const double* xs = st + x_off;
    const double* ys = st + y_off;
    if (!(a.y_lower_tri && kt - kt0 > warp_n))
#pragma unroll (QS > 0 ? QUNROLL : KQ)
    for (int q = 0; q < KQ; ++q) {
      double av[8], bv[4];
#pragma unroll
      for (int mi = 0; mi < 8; ++mi) av[mi] = xs[(q * HALF + mi * 8) * 4];
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) bv[ni] = ys[(q * HALF + ni * 8) * 4];
      if (QS > 0) {                                   // fragment element (k = 4q + t, row r): alpha_k a + g_k T[r, slot(k)]
        const int kk = s * KT + q * 4 + t;
        const double al = kscales[kk], gk = qgs[kk];
        const int sl = qsl[kk];
        const double* tq = tqs + (size_t)s * TQ + (sl >> 2) * (HALF * 4) + (sl & 3);
#pragma unroll
        for (int mi = 0; mi < 8; ++mi) av[mi] = __fma_rn(gk, tq[tx_off + mi * 32], al * av[mi]);
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) bv[ni] = __fma_rn(gk, tq[ty_off + ni * 32], al * bv[ni]);
      }
      if (SCALED) {                                   // B fragment element (k = 4q + t, n = g): scale by w_k^2
        const double w = kscales[s * KT + q * 4 + t];
        const double w2 = w * w;
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) bv[ni] *= w2;
      }
#pragma unroll
      for (int mi = 0; mi < 8; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) dmma884(acc[mi][ni][0], acc[mi][ni][1], av[mi], bv[ni]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[s]);
  }

  // -------------------------------------------------------------- epilogue
  const double alpha = a.alpha;
  if (split) {
    // partial tile -> workspace, tile-local Q4 (ld = 128); splitk_reduce_kernel finishes the job
    double* wt = a.ws + (size_t)((int)blockIdx.x - a.tail0) * (size_t)(BM * BN);
    const int lr = warp_m * 64 + g, lc = warp_n * 32 + 2 * t;
#pragma unroll
    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
      for (int mi = 0; mi < 8; ++mi)
        *reinterpret_cast<double2*>(wt + q4_index(lr + mi * 8, lc + ni * 8, BM)) =
            make_double2(alpha * acc[mi][ni][0], alpha * acc[mi][ni][1]);
    return;
  }
  const int row_base = P.c_row0 + ti * BM + warp_m * 64 + g;
  const int col_base = P.c_col0 + tj * BN + warp_n * 32 + 2 * t;
  double* tm = a.Ctm ? a.Ctm + (size_t)tile * (size_t)(BM * BN) : nullptr;
  // Cin and Cout are the same buffer for the Cholesky updates, so the compiler has to keep every load behind the
  // previous store: a load -> add -> store loop is a chain of 32 global-memory latencies (17 us, as long as the
  // whole K = 128 contraction).  Issue the loads of a column group together, then add and store.
#pragma unroll
  for (int ni = 0; ni < 4; ++ni) {
    const int col = col_base + ni * 8;
#pragma unroll
    for (int mh = 0; mh < 8; mh += 4) {
      double2 cin[4];
#pragma unroll
      for (int mi = 0; mi < 4; ++mi) {
        cin[mi] = make_double2(0.0, 0.0);
        if (a.Cin) cin[mi] = *reinterpret_cast<const double2*>(a.Cin + q4_index(row_base + (mh + mi) * 8, col, a.ldc));
      }
#pragma unroll
      for (int mi = 0; mi < 4; ++mi) {
        double2 v = cin[mi];
        v.x += alpha * acc[mh + mi][ni][0];
        v.y += alpha * acc[mh + mi][ni][1];
        if (tm) *reinterpret_cast<double2*>(tm + q4_index(warp_m * 64 + g + (mh + mi) * 8, warp_n * 32 + 2 * t + ni * 8, BM)) = v;
        else *reinterpret_cast<double2*>(a.Cout + q4_index(row_base + (mh + mi) * 8, col, a.ldc)) = v;
      }
    }
  }
}

// C tile = Cin tile + sum over splits (in split order) of the partial tiles in the workspace
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const GemmArgs a) {
  const int tile = a.tile_begin + a.tail0 + blockIdx.x;
  const TilePos P = locate(a, tile);
  double* tm = a.Ctm ? a.Ctm + (size_t)tile * (size_t)(BM * BN) : nullptr;
  const size_t slab = (size_t)(BM * BN);
  const double* wt = a.ws + (size_t)blockIdx.x * a.ksplit * slab;
  for (int e = threadIdx.x * 2; e < BM * BN; e += 512) {
    double2 v = make_double2(0.0, 0.0);
    for (int sp = 0; sp < a.ksplit; ++sp) {
      const double2 w = *reinterpret_cast<const double2*>(wt + sp * slab + e);
      v.x += w.x;
      v.y += w.y;
    }
    const int quad = e / (BM * 4), lr = (e % (BM * 4)) >> 2, c = e & 3;
    const size_t idx = q4_index(P.c_row0 + P.ti * BM + lr, P.c_col0 + P.tj * BN + quad * 4 + c, a.ldc);
    if (a.Cin) {
      const double2 ci = *reinterpret_cast<const double2*>(a.Cin + idx);
      v.x += ci.x;
      v.y += ci.y;
    }
    if (tm) *reinterpret_cast<double2*>(tm + e) = v;             // the workspace tiles are tile-local Q4 already
    else *reinterpret_cast<double2*>(a.Cout + idx) = v;
  }
}

// Cout tile <- tile-major tile (both Q4: 512-double runs move as they are)
__global__ void __launch_bounds__(256) unpack_tiles_kernel(const GemmArgs a) {
  const int tile = a.tile_begin + blockIdx.x;
  const TilePos P = locate(a, tile);
  const double* tm = a.Ctm + (size_t)tile * (size_t)(BM * BN);
  for (int e = threadIdx.x * 2; e < BM * BN; e += 512) {
    const int quad = e / (BM * 4), lr = (e % (BM * 4)) >> 2, c = e & 3;
    const size_t idx = q4_index(P.c_row0 + P.ti * BM + lr, P.c_col0 + P.tj * BN + quad * 4 + c, a.ldc);
    *reinterpret_cast<double2*>(a.Cout + idx) = *reinterpret_cast<const double2*>(tm + e);
  }
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);
PFN_encodeTiled g_encode = nullptr;
std::atomic<unsigned long long> g_attr_set{0}, g_attr_set_scaled{0}, g_attr_set_q[4] = {};
}  // namespace

int gemm_nt_smem_bytes() { return SMEM_BYTES; }

int gemm_qfold_slots(int need) { return need <= 4 ? 4 : (need <= 16 ? (need + 3) / 4 * 4 : 0); }

int make_q4_tensor_map(CUtensorMap* out, const double* base, int ld, long long kq_total, int box_kq) {
  if (box_kq <= 0) box_kq = KQ;
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CIP_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (qres != cudaDriverEntryPointSuccess || !fn) {
      set_error("cuTensorMapEncodeTiled not available from the driver");
      return -1;
    }
    g_encode = reinterpret_cast<PFN_encodeTiled>(fn);
  }
  if (kq_total < box_kq) kq_total = box_kq;  // caller guarantees the allocation covers it
  cuuint64_t gdim[2] = {(cuuint64_t)ld * 4ull, (cuuint64_t)kq_total};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 32ull};
  cuuint32_t box[2] = {(cuuint32_t)(HALF * 4), (cuuint32_t)box_kq};
  cuuint32_t estride[2] = {1, 1};
  CUresult r = g_encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), gdim, gstride, box,
                        estride, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed: CUresult %d (ld=%d kq=%lld base=%p)", (int)r, ld, kq_total,
              (const void*)base);
    return -1;
  }
  return 0;
}

// (A/B knob for the DRAM-traffic experiments of profiles/: the same value must reach every kernel that maps tile
//  indices -- the GEMM, the split-K reduction and the tile-major unpack)
static int gemm_band() {
  static const int v = [] { const char* e = getenv("CIP_GEMM_BAND"); const int x = e ? atoi(e) : 0; return (x >= 1 && x <= 64) ? x : BAND_DEFAULT; }();
  return v;
}

int unpack_tile_major(const GemmArgs& a_in, cudaStream_t stream) {
  GemmArgs a = a_in;
  a.band = gemm_band();
  const long long all_tiles = a.lower ? (long long)a.ntm * (a.ntm + 1) / 2 : (long long)a.ntm * a.ntn;
  const long long tiles = a.tile_count > 0 ? a.tile_count : all_tiles - a.tile_begin;
  if (tiles <= 0) return 0;
  unpack_tiles_kernel<<<(unsigned)tiles, 256, 0, stream>>>(a);
  CIP_CHECK_LAUNCH();
  return 0;
}

// grid of a launch: the split-K tail (b.ksplit, b.kchunk, b.tail0) and the CTA count; false: nothing to do
static bool plan_launch(const GemmArgs& a, GemmArgs& b, long long& tiles, long long& ctas) {
  const int nsm = sm_count();      // one CTA per SM (192 KB of shared memory each): a wave is nsm tiles
  const long long all_tiles = a.lower ? (long long)a.ntm * (a.ntm + 1) / 2 : (long long)a.ntm * a.ntn;
  tiles = a.tile_count > 0 ? a.tile_count : all_tiles - a.tile_begin;
  if (tiles <= 0 || (a.nk <= 0 && !a.Ctm)) return false;      // (nk = 0 with tile-major output: the tiles are Cin, or zero)
  b = a;
  b.band = gemm_band();
  b.ksplit = 1;
  b.kchunk = a.nk;
  b.tail0 = (int)tiles;
  const long long tail = tiles % nsm;
  if (a.ws && tail > 0 && a.nk >= 8) {
    // cost of the tail in units of one full tile: ceil(tail * ks / nsm) / ks  (+ the reduction pass: a split
    // costs about a quarter of one k tile); pick the cheapest ks that fits the workspace
    const long long cap = a.ws_doubles / (long long)(BM * BN);
    int best = 1;
    double best_cost = 1.0;
    for (int ks = 2; ks <= nsm && ks <= a.nk / 4 && tail * ks <= cap; ++ks) {
      const double cost = (double)((tail * ks + nsm - 1) / nsm) / ks + 0.25 * ks / a.nk;
      if (cost < best_cost - 1e-9) { best_cost = cost; best = ks; }
    }
    if (best > 1) {
      b.kchunk = (a.nk + best - 1) / best;
      b.ksplit = (a.nk + b.kchunk - 1) / b.kchunk;                // no empty split
      b.tail0 = (int)(tiles - tail);
    }
  }
  ctas = b.tail0 + (tiles - b.tail0) * b.ksplit;
  return true;
}

static int finish_launch(const GemmArgs& b, long long tiles, cudaStream_t stream) {
  CIP_CHECK_LAUNCH();
  if (b.ksplit > 1) {
    splitk_reduce_kernel<<<(unsigned)(tiles - b.tail0), 256, 0, stream>>>(b);
    CIP_CHECK_LAUNCH();
  }
  return 0;
}

int launch_gemm_nt(const GemmOperand& X, const GemmOperand& Y, const GemmArgs& a, cudaStream_t stream) {
  CIP_TRY(ensure_dyn_smem((const void*)gemm_nt_kernel<false>, SMEM_BYTES, &g_attr_set));
  if (a.kscale) CIP_TRY(ensure_dyn_smem((const void*)gemm_nt_kernel<true>, SMEM_BYTES, &g_attr_set_scaled));
  GemmArgs b;
  long long tiles = 0, ctas = 0;
  if (!plan_launch(a, b, tiles, ctas)) return 0;
  if (a.kscale) gemm_nt_kernel<true><<<(unsigned)ctas, NUM_THREADS, SMEM_BYTES, stream>>>(X.map, Y.map, b);
  else gemm_nt_kernel<false><<<(unsigned)ctas, NUM_THREADS, SMEM_BYTES, stream>>>(X.map, Y.map, b);
  return finish_launch(b, tiles, stream);
}

// one Q-fold instance: QS slots per k tile
template <int QS>
static int launch_qfold_instance(const GemmOperand& X, const GemmOperand& T, const GemmArgs& a, cudaStream_t stream) {
  CIP_TRY(ensure_dyn_smem((const void*)gemm_nt_kernel<false, QS>, qf_smem_bytes(QS), &g_attr_set_q[QS / 4 - 1]));
  GemmArgs b;
  long long tiles = 0, ctas = 0;
  if (!plan_launch(a, b, tiles, ctas)) return 0;
  gemm_nt_kernel<false, QS><<<(unsigned)ctas, NUM_THREADS, qf_smem_bytes(QS), stream>>>(X.map, T.map, b);
  return finish_launch(b, tiles, stream);
}

int launch_gemm_nt_qfold(const GemmOperand& X, const GemmOperand& T, const GemmArgs& a, cudaStream_t stream) {
  if (!a.sym || !a.lower || a.kscale || a.group || !a.qalpha || !a.qg || !a.qslot || gemm_qfold_slots(a.qs) != a.qs) {
    set_error("launch_gemm_nt_qfold: needs a symmetric lower SYRK with qalpha / qg / qslot and qs = 4, 8, 12 or 16 "
              "(qs = %d)", a.qs);
    return -1;
  }
  switch (a.qs) {
    case 4: return launch_qfold_instance<4>(X, T, a, stream);
    case 8: return launch_qfold_instance<8>(X, T, a, stream);
    case 12: return launch_qfold_instance<12>(X, T, a, stream);
    default: return launch_qfold_instance<16>(X, T, a, stream);
  }
}

}  // namespace cip
