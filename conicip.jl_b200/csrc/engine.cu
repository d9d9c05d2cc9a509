// The KKT engine handle and the C ABI of include/conicip_b200.h.
//
// LEVEL 1 (cip_create)  : upload Q, A, G once, re-laid out in the Q4 layout (A transposed, so the
//                         contraction index of every tensor-core product is the interleaved one).
// LEVEL 2 (cip_factor)  : Atil = F^-T A (cone kernel) -> H = Q + Atil'Atil (DMMA SYRK, TMA fed)
//                         -> [NCCL all-reduce of the partial Gram matrices] -> blocked Cholesky
//                         -> Schur complement on G (same DMMA tiles).
// LEVEL 3 (cip_solve)   : the pivot algebra of src/kktsolvers.jl:324-332 on the resident data.
#include <climits>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <math.h>

#include <algorithm>
#include <vector>

#include "engine.h"
#include "nccl_dl.h"

namespace cip {

static thread_local char g_err[1024] = "";
std::atomic<long long> g_launches{0};

int sm_count() {
  static std::atomic<int> cache[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  int v = cache[dev].load(std::memory_order_relaxed);
  if (v == 0) {
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    cache[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}

int ensure_dyn_smem(const void* func, int bytes, std::atomic<unsigned long long>* done) {
  int dev = 0;
  CIP_CUDA(cudaGetDevice(&dev));
  const unsigned long long bit = 1ull << (dev & 63);
  if (done->load(std::memory_order_acquire) & bit) return 0;
  CIP_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  done->fetch_or(bit, std::memory_order_release);
  return 0;
}

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

}  // namespace cip

using namespace cip;

namespace {

template <typename T>
int dev_alloc(cip_engine* h, T** p, size_t count, bool zero = true) {
  *p = nullptr;
  if (count == 0) count = 1;
  CIP_CUDA(cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T)));
  if (zero) CIP_CUDA(cudaMemsetAsync(*p, 0, count * sizeof(T), h->stream));
  h->bytes += count * sizeof(T);
  return 0;
}

bool is_device_ptr(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}
// memory a kernel running on `device` may dereference: managed memory, or device memory of that very device
// (a shard of a multi-GPU handle is handed pointers that live on another GPU: those go through a copy)
bool kernel_readable(const void* p, int device) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeManaged || (at.type == cudaMemoryTypeDevice && at.device == device);
}

// stage an input vector (host or device) into an internal zero-padded device buffer
int stage_in(cip_engine* h, double* dst, const double* src, size_t n) {
  if (n == 0) return 0;
  if (!src) {
    set_error("null input vector");
    return -1;
  }
  CIP_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyDefault, h->stream));
  return 0;
}
int stage_out(cip_engine* h, double* dst, const double* src, size_t n) {
  if (n == 0 || !dst) return 0;
  CIP_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyDefault, h->stream));
  if (!is_device_ptr(dst)) h->need_sync = true;
  return 0;
}
// Vector arguments that already live in this device's memory (16-byte aligned) are used where they are: the
// kernels below index strictly inside [0, n), so no zero-padded private copy is needed.  Host memory, memory of
// another GPU and odd alignments go through the internal staging buffer as before.  `padded`: the consumer reads
// whole quads (the k-major mat-vec), so a direct pointer is only allowed when n is a multiple of 4.
bool direct_ok(const cip_engine* h, const void* p, size_t n, bool padded = false) {
  if (!p || (reinterpret_cast<uintptr_t>(p) & 15) != 0) return false;
  if (padded && (n & 3) != 0) return false;
  return kernel_readable(p, h->device);
}
int vec_in(cip_engine* h, double* stage, const double* src, size_t n, const double** use, bool padded = false) {
  if (n == 0) { *use = stage; return 0; }
  if (direct_ok(h, src, n, padded)) { *use = src; return 0; }
  *use = stage;
  return stage_in(h, stage, src, n);
}
// where a result should be produced: the caller's buffer itself, or the staging buffer (copied out afterwards)
double* vec_out(cip_engine* h, double* stage, double* dst, size_t n) {
  return (n > 0 && direct_ok(h, dst, n)) ? dst : stage;
}
int vec_out_done(cip_engine* h, double* dst, const double* produced, size_t n) {
  if (n == 0 || !dst || produced == dst) return 0;
  return stage_out(h, dst, produced, n);
}

// give-up flag of the persistent sweeps with H's factor (none when row_structure = 2 left K empty)
int* h_sweep_err(const cip_engine* h) {
  return h->rs.sp.on ? (h->rs.sp.nK > 0 ? h->rs.sp.chol.sweep_err : nullptr) : h->cholH.sweep_err;
}

int finish(cip_engine* h) {
  if (h->need_sync || h->always_sync) {
    CIP_CUDA(cudaStreamSynchronize(h->stream));
    h->need_sync = false;
  }
  return 0;
}

int check(cip_handle h) {
  if (!h) {
    set_error("null handle");
    return -1;
  }
  CIP_CUDA(cudaSetDevice(h->device));
  return 0;
}

int allreduce(cip_engine* h, double* buf, size_t count) {
  if (!h->comm || count == 0) return 0;
  const NcclApi* api = nccl_api();
  if (!api) return -1;
  int r = api->AllReduce(buf, buf, count, kNcclFloat64, kNcclSum, h->comm, h->stream);
  if (r != 0) {
    set_error("ncclAllReduce failed: %s", api->GetErrorString(r));
    return -1;
  }
  return 0;
}

int set_scaling_from_user(cip_engine* h, const int* kind, const double* fa, const double* fb, const double* fD,
                          const double* fR) {
  if (!kind || !fa) {
    set_error("cip_factor/cip_set_scaling: kind and fa are required");
    return -1;
  }
  std::vector<int> hk(h->ncones);
  if (is_device_ptr(kind)) {
    CIP_CUDA(cudaMemcpy(hk.data(), kind, sizeof(int) * h->ncones, cudaMemcpyDeviceToHost));
  } else {
    memcpy(hk.data(), kind, sizeof(int) * h->ncones);
  }
  bool any_w = false, any_v = false;
  for (int i = 0; i < h->ncones; ++i) {
    if (hk[i] == CIP_BLK_VECCONG) {
      if (h->h_type[i] != CIP_CONE_S) {
        set_error("VecCongurance block on cone %d, which is not an S cone", i);
        return -1;
      }
      any_v = true;
    } else if (hk[i] != CIP_BLK_DIAG && hk[i] != CIP_BLK_WOODBURY) {
      set_error("unknown scaling block kind %d for cone %d", hk[i], i);
      return -1;
    }
    if (hk[i] == CIP_BLK_WOODBURY && h->h_type[i] != CIP_CONE_Q) {
      // nestod_soc is the only producer of SymWoodbury blocks (src/ConicIP.jl:192,599); the panel scaling
      // only walks the Q cones, so a Woodbury block elsewhere would make H inconsistent with cip_apply
      set_error("SymWoodbury block on cone %d, which is not a Q cone", i);
      return -1;
    }
    any_w |= (hk[i] == CIP_BLK_WOODBURY);
  }
  CIP_CUDA(cudaMemcpyAsync(h->F.kind, hk.data(), sizeof(int) * h->ncones, cudaMemcpyHostToDevice, h->stream));
  CIP_CUDA(cudaStreamSynchronize(h->stream));  // hk goes out of scope
  CIP_TRY(stage_in(h, h->F.a, fa, h->m));
  if (any_w) {
    if (!fb || !fD) {
      set_error("SymWoodbury blocks need fb and fD");
      return -1;
    }
    CIP_TRY(stage_in(h, h->F.b, fb, h->m));
    CIP_TRY(stage_in(h, h->F.D, fD, h->ncones));
  } else {
    CIP_TRY(fill_zero(h->F.b, h->m, h->stream));
    CIP_TRY(fill_zero(h->F.D, h->ncones, h->stream));
  }
  if (any_v) {
    if (!fR) {
      set_error("VecCongurance blocks need fR");
      return -1;
    }
    size_t src = 0;                       // fR is concatenated over the VECCONG blocks in cone order
    for (size_t si = 0; si < h->h_slist.size(); ++si) {
      if (hk[h->h_slist[si]] != CIP_BLK_VECCONG) continue;
      const size_t kk = (size_t)h->h_sord[si] * h->h_sord[si];
      CIP_CUDA(cudaMemcpyAsync(h->F.R + h->h_roff[si], fR + src, kk * sizeof(double), cudaMemcpyDefault, h->stream));
      src += kk;
    }
  }
  CIP_TRY(cone_invert_scaling(h->cd, h->F, h->Fi, h->stream));
  h->have_scaling = true;
  return 0;
}

// Row-sharded form of H: the partial Gram matrix is produced tile-major in a few ranges of the (reversed) tile
// order; each range is all-reduced (NCCL, stream cs) and unpacked into H4 while the next ranges are still being
// computed, so only the last, small range (the tip of the triangle) is exposed.  Ranges alternate between two
// streams: consecutive SYRK launches do not serialise on each other's last wave.
int form_H_sharded(cip_engine* h, const double* cin, int k_rows) {
  const NcclApi* api = nccl_api();
  if (!api) return -1;
  cudaStream_t s = h->stream;
  const int T = h->n_pad / TILE;
  const long long ntiles = (long long)T * (T + 1) / 2;
  const int nsm = sm_count();
  // range ends as fractions of the tiles, rounded to whole waves; small problems: one range
  const double frac[6] = {0.40, 0.70, 0.85, 0.93, 0.97, 1.0};
  long long ends[6];
  int nr = 0;
  long long prev = 0;
  for (int i = 0; i < 6; ++i) {
    long long e = (i == 5) ? ntiles : (long long)(frac[i] * ntiles) / nsm * nsm;
    if (e <= prev) continue;
    if (ntiles < 4LL * nsm) e = ntiles;
    ends[nr++] = e;
    prev = e;
    if (e == ntiles) break;
  }
  CIP_CUDA(cudaEventRecord(h->evc[15], s));                 // Atil ready
  CIP_CUDA(cudaStreamWaitEvent(h->s2, h->evc[15], 0));
  long long t0 = 0;
  for (int i = 0; i < nr; ++i) {
    cudaStream_t st = (i & 1) ? h->s2 : s;
    GemmArgs a{};
    a.lower = 1; a.ntm = a.ntn = T; a.sym = 1; a.reverse = 1;
    a.nk = k_rows / 32;
    a.Cin = cin; a.Cout = h->H4; a.Ctm = h->Hp; a.ldc = h->n_pad; a.alpha = 1.0;
    a.tile_begin = (int)t0; a.tile_count = (int)(ends[i] - t0);
    if (h->fold) a.kscale = h->Fi.a;
    if (i == nr - 1) { a.ws = h->gemm_ws; a.ws_doubles = GEMM_WS_DOUBLES; }     // split-K only for the very last wave
    const GemmOperand& op = h->fold ? h->mapAt : h->mapAtil;
    CIP_TRY(launch_gemm_nt(op, op, a, st));
    CIP_CUDA(cudaEventRecord(h->evc[i], st));
    CIP_CUDA(cudaStreamWaitEvent(h->cs, h->evc[i], 0));
    double* seg = h->Hp + (size_t)t0 * TILE * TILE;
    const int r = api->AllReduce(seg, seg, (size_t)a.tile_count * TILE * TILE, kNcclFloat64, kNcclSum, h->comm, h->cs);
    if (r != 0) {
      set_error("ncclAllReduce failed: %s", api->GetErrorString(r));
      return -1;
    }
    CIP_TRY(unpack_tile_major(a, h->cs));
    t0 = ends[i];
  }
  if (nr > 1) {
    CIP_CUDA(cudaEventRecord(h->evc[14], h->s2));
    CIP_CUDA(cudaStreamWaitEvent(s, h->evc[14], 0));
  }
  CIP_CUDA(cudaEventRecord(h->ev[2], s));                   // every SYRK range done; what follows is the exposed wait
  CIP_CUDA(cudaEventRecord(h->evc[13], h->cs));
  CIP_CUDA(cudaStreamWaitEvent(s, h->evc[13], 0));
  return 0;
}

int form_H(cip_engine* h) {
  if (!h->have_scaling) {
    set_error("no scaling set (call cip_factor / cip_set_scaling / cip_nt_scaling first)");
    return -1;
  }
  cudaStream_t s = h->stream;
  CIP_CUDA(cudaEventRecord(h->ev[0], s));
  if (h->rs.on) {
    CIP_TRY(structure_form_H(h));
    if (h->opt.reg_delta != 0.0) {
      if (h->rs.sp.on) CIP_TRY(split_add_delta(h, h->opt.reg_delta));
      else CIP_TRY(add_diag_q4(h->H4, h->n_pad, 0, h->n, h->opt.reg_delta, 0, s));
    }
    CIP_CUDA(cudaEventRecord(h->ev[3], s));
    return 0;
  }
  const bool fast = h->fast.on && !h->comm;
  if (fast) CIP_TRY(cone_scale_panel_norms(h->Fi, h->At4, h->Atil4, h->n_pad, h->m_pad, h->fast.colss, h->fast.colexp, s));
  else if (h->m_pad > 0 && !h->fold) CIP_TRY(cone_scale_panel(h->cd, h->Fi, h->At4, h->Atil4, h->n_pad, h->m_pad, h->n, s));
  CIP_CUDA(cudaEventRecord(h->ev[1], s));
  const double* cin = (h->rank == 0) ? h->Qq4 : nullptr;
  // rows of Atil beyond m_pad hold sqrt(rho)*G (constant): H' = Q + Atil'Atil + rho G'G, added on rank 0 only
  const int k_rows = h->m_pad + ((h->rank == 0) ? h->aug_rows : 0);
  if (h->comm && h->Hp) {
    CIP_TRY(form_H_sharded(h, cin, k_rows));
    if (h->opt.reg_delta != 0.0) CIP_TRY(add_diag_q4(h->H4, h->n_pad, 0, h->n, h->opt.reg_delta, 0, s));
    CIP_CUDA(cudaEventRecord(h->ev[3], s));
    h->st.syrk_flops = (double)h->m * (double)h->n * (double)h->n;
    return 0;
  }
  if (fast) {
    CIP_TRY(fast_syrk_form(h, cin));       // sums, products, combination and the diagonal leaves: all inside ev[1..2]
  } else if (k_rows > 0) {
    GemmArgs a{};
    a.lower = 1; a.ntm = a.ntn = h->n_pad / TILE; a.sym = 1;
    a.x_row0 = a.y_row0 = 0; a.x_kq0 = a.y_kq0 = 0; a.nk = k_rows / 32;
    a.Cin = cin; a.Cout = h->H4; a.ldc = h->n_pad; a.c_row0 = a.c_col0 = 0; a.alpha = 1.0;
    a.ws = h->gemm_ws; a.ws_doubles = GEMM_WS_DOUBLES;        // tall-skinny A (n << m): split the contraction
    if (h->fold) a.kscale = h->Fi.a;                          // W^-2 applied to the fragments: no Atil4
    const GemmOperand& op = h->fold ? h->mapAt : h->mapAtil;
    // Experiment knob (profiles/r02_syrk_traffic.md): CIP_SYRK_KCHUNK = rows of A per launch, every launch
    // accumulating into H.  Off by default: at C4 it did not lower the DRAM traffic of the operand panels (994 GB in
    // four launches against 812 GB in one) and costs 0.1 % of the SYRK time.
    static const int kchunk_rows = [] { const char* e = getenv("CIP_SYRK_KCHUNK"); const int v = e ? atoi(e) : 0; return v > 0 ? (v + 31) / 32 * 32 : 0; }();
    const int total_kt = k_rows / 32;
    const int chunk_kt = (kchunk_rows > 0 && h->n_pad >= 4096) ? kchunk_rows / 32 : total_kt;
    if (total_kt > chunk_kt + chunk_kt / 2) {
      for (int kt0 = 0; kt0 < total_kt;) {
        int kn = chunk_kt;
        if (total_kt - (kt0 + kn) < chunk_kt / 2) kn = total_kt - kt0;       // fold a short remainder into the last chunk
        GemmArgs c = a;
        c.x_kq0 = c.y_kq0 = kt0 * 8;
        c.nk = kn;
        if (kt0 > 0) c.Cin = h->H4;
        CIP_TRY(launch_gemm_nt(op, op, c, s));
        kt0 += kn;
      }
    } else {
      CIP_TRY(launch_gemm_nt(op, op, a, s));
    }
  } else {
    if (cin) CIP_TRY(vec_copy(h->H4, cin, (size_t)h->n_pad * h->n_pad, s));
    else CIP_TRY(fill_zero(h->H4, (size_t)h->n_pad * h->n_pad, s));
  }
  CIP_CUDA(cudaEventRecord(h->ev[2], s));
  if (h->comm) CIP_TRY(allreduce(h, h->H4, (size_t)h->n_pad * h->n_pad));
  if (h->opt.reg_delta != 0.0) CIP_TRY(add_diag_q4(h->H4, h->n_pad, 0, h->n, h->opt.reg_delta, 0, s));
  CIP_CUDA(cudaEventRecord(h->ev[3], s));
  h->st.syrk_flops = (double)h->m * (double)h->n * (double)h->n;
  return 0;
}

int factor_H(cip_engine* h) {
  cudaStream_t s = h->stream;
  // row_structure = 2: H_KK is factored on its own plan and D by split_factor; the Schur block below runs on Z_K
  const RowStructure::Split& sp = h->rs.sp;
  if (sp.on) {
    CIP_TRY(split_factor(h));
  } else {
    // block-cyclic distributed factorisation when A is row-sharded (every rank holds the reduced H);
    // opts.dist_chol: 0 = replicated, 1 = distributed, -1/unset = distributed iff >= 2 outer panels per rank
    bool dist = false;
    if (h->comm && h->nranks > 1) {
      const int outer_panels = (h->cholH.npanels + 3) / 4;   // 512-column units
      int mode = h->opt.dist_chol;
      if (const char* env = getenv("CIP_DIST_CHOL")) mode = atoi(env);
      dist = (mode == 1) || (mode != 0 && outer_panels >= 2 * h->nranks);
    }
    if (dist) {
      CholDist d;
      d.nranks = h->nranks; d.rank = h->rank; d.comm = h->comm;
      CIP_TRY(chol_factor_dist(h->cholH, s, d));
    } else {
      CIP_TRY(chol_factor(h->cholH, s));
    }
  }
  CIP_CUDA(cudaEventRecord(h->ev[4], s));
  if (h->p > 0) {
    // Z = G L^-T by a right-looking blocked substitution on the DMMA tiles, S = Z Z', S = Ls Ls'.
    // Two-level like the Cholesky: inside an outer panel of four 128-column panels every panel is solved against
    // inv(L_jj) and applied to the rest of the outer panel only; everything right of the outer panel gets ONE update
    // with K = 512, which amortises the C-tile read-modify-write that holds K = 128 tiles at a third of the pipe.
    // (row_structure = 2: Z_K = G_K L_KK^-T over the K columns)
    const CholPlan& L = sp.on ? sp.chol : h->cholH;
    double* Z = sp.on ? sp.ZK4 : h->Z4;
    const GemmOperand& mapZ = sp.on ? sp.mapZK : h->mapZ;
    const int np = (sp.on ? sp.nK_pad : h->n_pad) / TILE, ptiles = h->p_pad / TILE;
    if (np > 0) CIP_TRY(vec_copy(Z, sp.on ? sp.GK4 : h->G4, (size_t)h->p_pad * np * TILE, s));
    auto z_trsm = [&](int jb) -> int {                       // Z[:, jb] <- Z[:, jb] inv(L_jj)'
      GemmArgs t{};
      t.lower = 0; t.ntm = ptiles; t.ntn = 1; t.sym = 0;
      t.x_row0 = 0; t.y_row0 = 0; t.x_kq0 = jb * TILE / 4; t.y_kq0 = 32 * jb; t.nk = TILE / 32;
      t.Cin = nullptr; t.Cout = Z; t.ldc = h->p_pad; t.c_row0 = 0; t.c_col0 = jb * TILE; t.alpha = 1.0;
      return launch_gemm_nt(mapZ, L.mapWinv, t, s);
    };
    auto z_update = [&](int k0, int kn, int c0, int cn) -> int {   // Z[:, c0..c0+cn) -= Z[:, k0..k0+kn) L[c0..c0+cn, k0..k0+kn)'   (panel units)
      GemmArgs u{};
      u.lower = 0; u.ntm = ptiles; u.ntn = cn; u.sym = 0;
      u.x_row0 = 0; u.y_row0 = c0 * TILE; u.x_kq0 = k0 * TILE / 4; u.y_kq0 = k0 * TILE / 4; u.nk = kn * TILE / 32;
      u.Cin = Z; u.Cout = Z; u.ldc = h->p_pad; u.c_row0 = 0; u.c_col0 = c0 * TILE; u.alpha = -1.0;
      return launch_gemm_nt(mapZ, L.mapH, u, s);
    };
    // (few right-hand-side tiles, p <= 384: every launch is latency-bound and the extra level only lengthens the chain --
    //  config 3, p = 256: 1.73 ms single-level against 2.07 ms two-level; config 5, p = 1000: 22.0 ms against 35.6 ms)
    const int ZOUTER = (ptiles >= 4) ? 4 : 1;
    for (int J0 = 0; J0 < np; J0 += ZOUTER) {
      const int J1 = std::min(J0 + ZOUTER, np);
      for (int jb = J0; jb < J1; ++jb) {
        CIP_TRY(z_trsm(jb));
        if (jb + 1 < J1) CIP_TRY(z_update(jb, 1, jb + 1, J1 - jb - 1));
      }
      if (J1 < np) CIP_TRY(z_update(J0, J1 - J0, J1, np - J1));
    }
    GemmArgs a{};
    a.lower = 1; a.ntm = a.ntn = ptiles; a.sym = 1;
    a.x_row0 = a.y_row0 = 0; a.x_kq0 = a.y_kq0 = 0;
    a.Cin = h->Sbase4; a.Cout = h->S4; a.ldc = h->p_pad; a.c_row0 = a.c_col0 = 0; a.alpha = 1.0;
    a.ws = h->gemm_ws; a.ws_doubles = GEMM_WS_DOUBLES;
    if (sp.on && sp.g_in_D) {
      // + G_D diag(1/h) G_D': the folded-scaling SYRK over all of G with kscale = h^-1/2 on D and 0 on K
      GemmArgs g = a;
      g.nk = h->n_pad / 32;
      g.kscale = sp.kscale;
      CIP_TRY(launch_gemm_nt(sp.mapG, sp.mapG, g, s));
      a.Cin = h->S4;
    }
    a.nk = np * TILE / 32;
    if (np > 0) CIP_TRY(launch_gemm_nt(mapZ, mapZ, a, s));
    else if (a.Cin != h->S4) CIP_TRY(vec_copy(h->S4, h->Sbase4, (size_t)h->p_pad * h->p_pad, s));
    CIP_TRY(chol_factor(h->cholS, s));
  }
  CIP_CUDA(cudaEventRecord(h->ev[5], s));
  int hinfo[2] = {0, 0}, dfail = INT_MAX;
  CIP_CUDA(cudaMemcpyAsync(hinfo, h->info, sizeof(hinfo), cudaMemcpyDeviceToHost, s));
  if (sp.on) CIP_CUDA(cudaMemcpyAsync(&dfail, sp.fail, sizeof(int), cudaMemcpyDeviceToHost, s));
  CIP_CUDA(cudaStreamSynchronize(s));
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]); h->st.ms_scale = ms;
  cudaEventElapsedTime(&ms, h->ev[1], h->ev[2]); h->st.ms_syrk = ms;
  cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]); h->st.ms_allreduce = ms;
  cudaEventElapsedTime(&ms, h->ev[3], h->ev[4]); h->st.ms_chol = ms;
  cudaEventElapsedTime(&ms, h->ev[4], h->ev[5]); h->st.ms_schur = ms;
  cudaGetLastError();
  const double nf = sp.on ? sp.nK : h->n;
  h->st.chol_flops = nf * nf * nf / 3.0;
  h->st.factors++;
  h->have_factor = true;
  if (sp.on) {
    // the first failing pivot in natural column order: the smallest failing D column or the K column where the
    // factorisation of H_KK stopped (1-based, as the dense path reports it)
    int col = std::min(dfail, h->n);
    if (hinfo[0] != 0) col = std::min(col, sp.K[hinfo[0] - 1]);
    hinfo[0] = col < h->n ? col + 1 : 0;
  }
  if (hinfo[0] != 0) {
    set_error("Cholesky of H failed: non-positive pivot at column %d", hinfo[0]);
    return hinfo[0];
  }
  if (hinfo[1] != 0) {
    set_error("Cholesky of the Schur complement failed: non-positive pivot at row %d", hinfo[1]);
    return h->n + hinfo[1];
  }
  return 0;
}

}  // namespace

namespace cip {
int engine_allreduce(cip_engine* h, double* buf, size_t count) { return allreduce(h, buf, count); }
int engine_setup_comm(cip_engine* h) {
  if (!h->comm || h->Hp) return 0;
  CIP_TRY(fast_syrk_drop(h));
  h->cholH.nranks_hint = h->nranks;        // the replicated fallback must schedule like the distributed one
  if (const char* env = getenv("CIP_OVERLAP_REDUCE")) if (atoi(env) == 0) return 0;   // A/B switch: plain all-reduce of H4
  CIP_CUDA(cudaSetDevice(h->device));
  const int T = h->n_pad / TILE;
  if (h->m_pad + h->aug_rows == 0) {
    // (a shard without rows still takes part: its tiles are Q or zero) -- the operand map must exist
    CIP_TRY(make_q4_tensor_map(&h->mapAtil.map, h->Atil4, h->n_pad, 8));
  }
  CIP_TRY(dev_alloc(h, &h->Hp, (size_t)T * (T + 1) / 2 * TILE * TILE, false));
  int lo = 0, hi = 0;
  CIP_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
  CIP_CUDA(cudaStreamCreateWithPriority(&h->cs, cudaStreamNonBlocking, hi));
  CIP_CUDA(cudaStreamCreateWithFlags(&h->s2, cudaStreamNonBlocking));
  for (auto& e : h->evc) CIP_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  return 0;
}
const char* last_error_string() { return g_err; }
int engine_decide_fold(cip_engine* h, bool can, size_t mn, bool* fold) {
  // fold the scaling into the SYRK (no Atil4) for pure R-cone rows: on request, or when the second copy of A would
  // not fit next to what is still to be allocated (Q, H, workspaces: ~ 3 n_pad^2 + 2.2 GB)
  int mode = can ? h->opt.fold_scaling : 2;
  if (const char* env = getenv("CIP_FOLD_SCALING")) { if (can) mode = atoi(env); }
  if (mode == 0) {
    size_t free_b = 0, total_b = 0;
    CIP_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const size_t nn = (size_t)h->n_pad * h->n_pad;
    const size_t need = mn * 8 + 3 * nn * 8 + (size_t)GEMM_WS_DOUBLES * 8 + (size_t(1) << 30);
    mode = (free_b < need) ? 1 : 2;
  }
  *fold = (mode == 1);
  return 0;
}
}  // namespace cip

// =================================================================== C ABI
extern "C" {

const char* cip_last_error(void) { return cip::g_err; }
int cip_version(void) { return 100; }

}  // extern "C"

namespace {

// upload a CSC matrix (host or device arrays) and scatter it into a zero-initialised Q4 buffer
int upload_csc(cip_engine* h, double* dst, int ld, const cip_csc* M, int transpose) {
  const long long ncols = M->ncols;
  if (ncols == 0) return 0;
  std::vector<long long> cp(2);
  CIP_CUDA(cudaMemcpy(&cp[0], M->colptr, 8, cudaMemcpyDefault));
  CIP_CUDA(cudaMemcpy(&cp[1], M->colptr + ncols, 8, cudaMemcpyDefault));
  const long long nnz = cp[1] - cp[0];
  if (nnz <= 0) return 0;
  long long *dcp = nullptr, *drv = nullptr;
  double* dnz = nullptr;
  CIP_CUDA(cudaMalloc(&dcp, (ncols + 1) * 8));
  CIP_CUDA(cudaMalloc(&drv, nnz * 8));
  CIP_CUDA(cudaMalloc(&dnz, nnz * 8));
  CIP_CUDA(cudaMemcpyAsync(dcp, M->colptr, (ncols + 1) * 8, cudaMemcpyDefault, h->stream));
  CIP_CUDA(cudaMemcpyAsync(drv, M->rowval, nnz * 8, cudaMemcpyDefault, h->stream));
  CIP_CUDA(cudaMemcpyAsync(dnz, M->nzval, nnz * 8, cudaMemcpyDefault, h->stream));
  int* dbad = nullptr;
  CIP_CUDA(cudaMalloc(&dbad, sizeof(int)));
  CIP_CUDA(cudaMemsetAsync(dbad, 0, sizeof(int), h->stream));
  int rc = scatter_csc_q4(dst, ld, (int)ncols, dcp, drv, dnz, M->index_base, transpose, M->nrows, nnz, dbad, h->stream);
  int bad = 0;
  cudaMemcpyAsync(&bad, dbad, sizeof(int), cudaMemcpyDeviceToHost, h->stream);
  cudaStreamSynchronize(h->stream);
  cudaFree(dcp); cudaFree(drv); cudaFree(dnz); cudaFree(dbad);
  if (rc == 0 && bad != 0) {
    set_error("malformed CSC input: column %d holds a row index outside [0, %d) or an inverted column pointer",
              bad - 1, M->nrows);
    return -1;
  }
  return rc;
}

int create_body(cip_engine* h, int n, int m, int p, const double* Q, int ldq, const double* A, int lda,
                const double* G, int ldg, const cip_csc* Qs, const cip_csc* As, const cip_csc* Gs, int ncones,
                const int* cone_type, const int* cone_dim, const cip_options* opts, bool shard);

// allocates the handle, builds it, and releases everything again if any step fails
int create_impl(cip_handle* out, int n, int m, int p, const double* Q, int ldq, const double* A, int lda,
                const double* G, int ldg, const cip_csc* Qs, const cip_csc* As, const cip_csc* Gs, int ncones,
                const int* cone_type, const int* cone_dim, const cip_options* opts, bool shard = false) {
  if (out) *out = nullptr;
  if (!out || n <= 0 || m < 0 || p < 0 || ncones < 0 || (ncones > 0 && (!cone_type || !cone_dim))) {
    set_error("cip_create: bad dimensions n=%d m=%d p=%d ncones=%d", n, m, p, ncones);
    return -1;
  }
  cip_engine* h = new cip_engine();
  const int rc = create_body(h, n, m, p, Q, ldq, A, lda, G, ldg, Qs, As, Gs, ncones, cone_type, cone_dim, opts, shard);
  if (rc != 0) {
    cip_destroy(h);            // every member is null-checked there
    return rc;
  }
  *out = h;
  return 0;
}

int create_body(cip_engine* h, int n, int m, int p, const double* Q, int ldq, const double* A, int lda,
                const double* G, int ldg, const cip_csc* Qs, const cip_csc* As, const cip_csc* Gs, int ncones,
                const int* cone_type, const int* cone_dim, const cip_options* opts, bool shard) {
  h->opt.dist_chol = -1;
  h->opt.aug_rho = -1.0;
  if (opts) memcpy(&h->opt, opts, std::min<size_t>(sizeof(cip_options), (size_t)opts->struct_size));
  else h->opt.device = -1;
  {
    // (0 when the caller's struct does not reach the field: h->opt starts zeroed)
    int rs = h->opt.row_structure;
    if (const char* env = getenv("CIP_ROW_STRUCTURE")) { if (!shard) rs = atoi(env); }
    if (rs != 0 && rs != 1 && rs != 2) {
      set_error("cip_create: row_structure must be 0, 1 or 2 (got %d)", rs);
      return -1;
    }
    h->rs.on = (rs == 1 || rs == 2) && m > 0;     // no rows: nothing to classify
    h->rs.sp.on = (rs == 2) && m > 0;
  }
  if (h->opt.device < 0) CIP_CUDA(cudaGetDevice(&h->device));
  else h->device = h->opt.device;
  CIP_CUDA(cudaSetDevice(h->device));
  {
    cudaDeviceProp prop;
    CIP_CUDA(cudaGetDeviceProperties(&prop, h->device));
    if (prop.major != 10) {
      set_error("conicip_b200 requires an sm_100a device (found sm_%d%d); there is no fallback path", prop.major,
                prop.minor);
      return -3;
    }
  }
  CIP_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  h->own_stream = h->stream;
  for (auto& e : h->ev) {
    CIP_CUDA(cudaEventCreate(&e));
    CIP_CUDA(cudaEventRecord(e, h->stream));
  }
  h->n = n; h->m = m; h->p = p; h->ncones = ncones;
  h->n_pad = round_up(n, TILE);
  h->m_pad = round_up(m, 32);
  h->p_pad = p > 0 ? round_up(p, TILE) : 0;

  // ---- cones
  h->h_type.assign(cone_type, cone_type + ncones);
  h->h_off.assign(ncones + 1, 0);
  std::vector<int> rowcone(m), qlist, slist;
  int maxq = 0, maxs = 0;
  for (int i = 0; i < ncones; ++i) {
    if (cone_dim[i] <= 0) {
      set_error("cone %d has non-positive dimension", i);
      return -1;
    }
    h->h_off[i + 1] = h->h_off[i] + cone_dim[i];
    if (h->h_off[i + 1] > m) break;
    for (int r = h->h_off[i]; r < h->h_off[i + 1]; ++r) rowcone[r] = i;
    if (cone_type[i] == CIP_CONE_Q) { qlist.push_back(i); maxq = std::max(maxq, cone_dim[i]); }
    else if (cone_type[i] == CIP_CONE_S) {
      const int k = (int)((sqrt(1.0 + 8.0 * cone_dim[i]) - 1.0) / 2.0 + 0.5);
      if (k * (k + 1) / 2 != cone_dim[i]) {
        set_error("S cone %d: dimension %d is not k(k+1)/2", i, cone_dim[i]);
        return -1;
      }
      if (k > sdp_max_order()) {
        set_error("S cone %d: order %d exceeds the supported maximum %d", i, k, sdp_max_order());
        return -2;
      }
      slist.push_back(i);
      h->h_sord.push_back(k);
      h->h_roff.push_back((int)h->r_total);
      h->r_total += (size_t)k * k;
      maxs = std::max(maxs, k);
    }
    else if (cone_type[i] != CIP_CONE_R) {
      set_error("unknown cone type %d", cone_type[i]);
      return -1;
    }
  }
  if (h->h_off[ncones] != m) {
    set_error("cone dimensions sum to %d but A has %d rows", h->h_off[ncones], m);
    return -1;
  }
  CIP_TRY(dev_alloc(h, &h->d_type, ncones));
  CIP_TRY(dev_alloc(h, &h->d_off, ncones + 1));
  CIP_TRY(dev_alloc(h, &h->d_rowcone, m));
  CIP_TRY(dev_alloc(h, &h->d_qlist, qlist.size()));
  CIP_TRY(dev_alloc(h, &h->d_slist, slist.size()));
  CIP_TRY(dev_alloc(h, &h->d_sord, slist.size()));
  CIP_TRY(dev_alloc(h, &h->d_roff, slist.size()));
  h->h_slist = slist;
  if (ncones) CIP_CUDA(cudaMemcpy(h->d_type, h->h_type.data(), sizeof(int) * ncones, cudaMemcpyHostToDevice));
  CIP_CUDA(cudaMemcpy(h->d_off, h->h_off.data(), sizeof(int) * (ncones + 1), cudaMemcpyHostToDevice));
  if (m) CIP_CUDA(cudaMemcpy(h->d_rowcone, rowcone.data(), sizeof(int) * m, cudaMemcpyHostToDevice));
  if (!qlist.empty())
    CIP_CUDA(cudaMemcpy(h->d_qlist, qlist.data(), sizeof(int) * qlist.size(), cudaMemcpyHostToDevice));
  if (!slist.empty()) {
    CIP_CUDA(cudaMemcpy(h->d_slist, slist.data(), sizeof(int) * slist.size(), cudaMemcpyHostToDevice));
    CIP_CUDA(cudaMemcpy(h->d_sord, h->h_sord.data(), sizeof(int) * slist.size(), cudaMemcpyHostToDevice));
    CIP_CUDA(cudaMemcpy(h->d_roff, h->h_roff.data(), sizeof(int) * slist.size(), cudaMemcpyHostToDevice));
  }
  h->cd.m = m; h->cd.ncones = ncones; h->cd.type = h->d_type; h->cd.off = h->d_off;
  h->cd.row_cone = h->d_rowcone; h->cd.qlist = h->d_qlist; h->cd.nq = (int)qlist.size();
  h->cd.slist = h->d_slist; h->cd.ns = (int)slist.size(); h->cd.max_q_dim = maxq; h->cd.max_s_ord = maxs;
  h->cd.sord = h->d_sord; h->cd.roff = h->d_roff;
  h->cd.sws = nullptr; h->cd.sws_stride = sdp_workspace_doubles(maxs);
  if (h->cd.sws_stride > 0) {
    // one slice per CTA of the widest S-cone launch (the scaled panel: ns x chunks)
    const long long ctas = (long long)slist.size() * std::max(1, sdp_panel_chunks(maxs, n));
    CIP_TRY(dev_alloc(h, &h->d_sws, (size_t)(ctas * h->cd.sws_stride)));
    h->cd.sws = h->d_sws;
  }
  h->cd.nr_rows = 0;
  for (int i = 0; i < ncones; ++i)
    if (cone_type[i] == CIP_CONE_R) h->cd.nr_rows += h->h_off[i + 1] - h->h_off[i];
  for (Scaling* S : {&h->F, &h->Fi}) {
    CIP_TRY(dev_alloc(h, &S->kind, ncones));
    CIP_TRY(dev_alloc(h, &S->a, h->m_pad + 4));
    CIP_TRY(dev_alloc(h, &S->b, h->m_pad + 4));
    CIP_TRY(dev_alloc(h, &S->D, ncones));
  }
  CIP_TRY(dev_alloc(h, &h->F.R, h->r_total));
  CIP_TRY(dev_alloc(h, &h->F.Ri, h->r_total));
  h->Fi.R = h->F.R;
  h->Fi.Ri = h->F.Ri;

  // ---- matrices
  const size_t nn = (size_t)h->n_pad * h->n_pad;
  const size_t mn = (size_t)h->m_pad * h->n_pad;
  if (!(h->rs.on && As)) CIP_TRY(dev_alloc(h, &h->At4, mn));     // CSC input with row structure: never dense
  // augmentation rows (H + rho G'G keeps the Cholesky valid when H is singular on range(G'), as kktsolver_qr allows)
  {
    double rho = h->opt.aug_rho;
    if (rho < 0) rho = (p > 0) ? 1.0 : 0.0;
    h->aug_rho = (p > 0) ? rho : 0.0;
    h->aug_rows = (h->aug_rho > 0) ? round_up(p, 32) : 0;
  }
  // (h->opt.fold_scaling is 0 when the caller's struct does not reach the field: h->opt starts zeroed)
  if (!h->rs.on) CIP_TRY(engine_decide_fold(h, slist.empty() && qlist.empty() && h->aug_rows == 0 && m > 0, mn, &h->fold));
  if (!h->rs.on && !h->fold) CIP_TRY(fast_syrk_plan(h, slist.empty() && qlist.empty() && h->aug_rows == 0 && m > 0));
  if (h->fast.on) CIP_TRY(dev_alloc(h, &h->Atil4, fast_syrk_atil_doubles(h)));
  else if (!h->fold && !h->rs.on) CIP_TRY(dev_alloc(h, &h->Atil4, (size_t)(h->m_pad + h->aug_rows) * h->n_pad));
  // row_structure = 2 keeps no n_pad^2 buffer: dense Q is staged in Qq4 until split_build has gathered Q_KK
  const bool split = h->rs.sp.on;
  if (!split || (!Qs && h->opt.q_kind == 0)) CIP_TRY(dev_alloc(h, &h->Qq4, nn));
  if (!split) CIP_TRY(dev_alloc(h, &h->H4, nn));
  CIP_TRY(dev_alloc(h, &h->gemm_ws, (size_t)GEMM_WS_DOUBLES));
  if (!split) CIP_TRY(dev_alloc(h, &h->Winv, (size_t)h->n_pad * TILE));
  CIP_TRY(dev_alloc(h, &h->info, 4));
  cudaStream_t s = h->stream;

  // Q
  if (Qs && split) {
    CIP_TRY(split_classify_csc_Q(h, Qs));
  } else if (Qs) {
    CIP_TRY(upload_csc(h, h->Qq4, h->n_pad, Qs, 0));
  } else if (h->opt.q_kind == 0) {
    if (!Q) { set_error("Q is null"); return -1; }
    if (kernel_readable(Q, h->device)) {
      CIP_TRY(pack_rows_q4(h->Qq4, h->n_pad, Q, ldq, n, n, h->n_pad, h->n_pad, s));
    } else {
      // chunk columns through a staging buffer
      const int chunk = std::max(4, std::min(n, (int)((256u << 20) / ((size_t)n * 8)) / 4 * 4));
      double* stg = nullptr;
      CIP_CUDA(cudaMalloc(&stg, (size_t)n * chunk * 8));
      for (int c0 = 0; c0 < n; c0 += chunk) {
        const int nc = std::min(chunk, n - c0);
        CIP_CUDA(cudaMemcpy2DAsync(stg, (size_t)n * 8, Q + (size_t)c0 * ldq, (size_t)ldq * 8, (size_t)n * 8, nc,
                                   cudaMemcpyDefault, s));
        // columns c0.. -> k range; write quads (c0/4 ..)
        CIP_TRY(pack_rows_q4(h->Qq4 + (size_t)(c0 / 4) * h->n_pad * 4, h->n_pad, stg, n, n, nc, h->n_pad,
                             round_up(nc, 4), s));
        CIP_CUDA(cudaStreamSynchronize(s));
      }
      cudaFree(stg);
    }
  } else if (h->opt.q_kind == 1) {
    if (!Q) { set_error("Q (diagonal) is null"); return -1; }
    if (split) {
      CIP_TRY(split_diag_Q(h, Q));
    } else {
      double* dq = nullptr;
      CIP_CUDA(cudaMalloc(&dq, sizeof(double) * n));
      CIP_CUDA(cudaMemcpyAsync(dq, Q, sizeof(double) * n, cudaMemcpyDefault, s));
      CIP_TRY(set_diag_vec_q4(h->Qq4, h->n_pad, n, dq, s));
      CIP_CUDA(cudaStreamSynchronize(s));
      cudaFree(dq);
    }
  }
  if (h->Qq4) CIP_TRY(add_diag_q4(h->Qq4, h->n_pad, n, h->n_pad, 1.0, 1, s));  // identity on the padding

  // A (transposed into Q4: rows = columns of A)
  if (m > 0) {
    if (!A && !As) { set_error("A is null"); return -1; }
    if (As && h->rs.on) {
      CIP_TRY(structure_build_csc(h, As));
    } else if (As) {
      CIP_TRY(upload_csc(h, h->At4, h->n_pad, As, 1));
    } else if (kernel_readable(A, h->device)) {
      CIP_TRY(pack_trans_q4(h->At4, h->n_pad, 0, A, lda, m, h->m_pad, n, s));
    } else {
      const int chunk = std::max(1, std::min(n, (int)((512u << 20) / ((size_t)m * 8))));
      double* stg = nullptr;
      CIP_CUDA(cudaMalloc(&stg, (size_t)m * chunk * 8));
      for (int c0 = 0; c0 < n; c0 += chunk) {
        const int nc = std::min(chunk, n - c0);
        CIP_CUDA(cudaMemcpy2DAsync(stg, (size_t)m * 8, A + (size_t)c0 * lda, (size_t)lda * 8, (size_t)m * 8, nc,
                                   cudaMemcpyDefault, s));
        CIP_TRY(pack_trans_q4(h->At4, h->n_pad, c0, stg, m, m, h->m_pad, nc, s));
        CIP_CUDA(cudaStreamSynchronize(s));
      }
      cudaFree(stg);
    }
    if (h->rs.on && !As) CIP_TRY(structure_build_dense(h));
  }
  if (h->rs.on) {
    // (structure_finish makes the operand map of the rest rows)
  } else if (h->fold) {
    CIP_TRY(make_q4_tensor_map(&h->mapAt.map, h->At4, h->n_pad, h->m_pad / 4));
  } else if (h->fast.on) {
    CIP_TRY(make_q4_tensor_map(&h->mapAtil.map, h->Atil4, h->n_pad, (long long)(fast_syrk_atil_doubles(h) / h->n_pad / 4)));
    CIP_TRY(fast_syrk_setup(h));
  } else if (h->m_pad + h->aug_rows > 0) {
    CIP_TRY(make_q4_tensor_map(&h->mapAtil.map, h->Atil4, h->n_pad, (h->m_pad + h->aug_rows) / 4));
  }
  if (!split) CIP_TRY(chol_make_plan(&h->cholH, h->H4, h->n_pad, h->Winv, h->info));

  // G
  if (p > 0) {
    if (!G && !Gs) { set_error("G is null"); return -1; }
    const size_t pn = (size_t)h->p_pad * h->n_pad;
    CIP_TRY(dev_alloc(h, &h->G4, pn));
    if (!split) CIP_TRY(dev_alloc(h, &h->Z4, pn));
    CIP_TRY(dev_alloc(h, &h->S4, (size_t)h->p_pad * h->p_pad));
    CIP_TRY(dev_alloc(h, &h->Sbase4, (size_t)h->p_pad * h->p_pad));
    CIP_TRY(dev_alloc(h, &h->WinvS, (size_t)h->p_pad * TILE));
    if (Gs) {
      CIP_TRY(upload_csc(h, h->G4, h->p_pad, Gs, 0));
    } else {
      double* stg = nullptr;
      const double* gsrc = G;
      int gld = ldg;
      if (!kernel_readable(G, h->device)) {
        CIP_CUDA(cudaMalloc(&stg, (size_t)p * n * 8));
        CIP_CUDA(cudaMemcpy2DAsync(stg, (size_t)p * 8, G, (size_t)ldg * 8, (size_t)p * 8, n, cudaMemcpyDefault, s));
        gsrc = stg;
        gld = p;
      }
      CIP_TRY(pack_rows_q4(h->G4, h->p_pad, gsrc, gld, p, n, h->p_pad, h->n_pad, s));
      CIP_CUDA(cudaStreamSynchronize(s));
      if (stg) cudaFree(stg);
    }
    if (h->aug_rows > 0 && !h->rs.on)
      CIP_TRY(transpose_scale_q4(h->Atil4, h->n_pad, h->m_pad, h->G4, h->p_pad, p, n, sqrt(h->aug_rho), s));
    CIP_TRY(add_diag_q4(h->Sbase4, h->p_pad, p, h->p_pad, 1.0, 1, s));
    if (h->opt.reg_eps_G != 0.0) CIP_TRY(add_diag_q4(h->Sbase4, h->p_pad, 0, p, h->opt.reg_eps_G, 1, s));
    if (!split) CIP_TRY(make_q4_tensor_map(&h->mapZ.map, h->Z4, h->p_pad, h->n_pad / 4));
    CIP_TRY(chol_make_plan(&h->cholS, h->S4, h->p_pad, h->WinvS, h->info + 1));
  }
  if (h->rs.on) CIP_TRY(structure_finish(h));

  // ---- work vectors
  for (auto& v : h->nv) CIP_TRY(dev_alloc(h, &v, h->n_pad + 4));
  for (auto& v : h->mv) CIP_TRY(dev_alloc(h, &v, h->m_pad + 4));
  for (auto& v : h->pv) CIP_TRY(dev_alloc(h, &v, h->p_pad + 4));
  h->partial_cap = 4 * sm_count() * 8 * 128 + 64 * std::max(n, std::max(p, 1));
  CIP_TRY(dev_alloc(h, &h->partial, h->partial_cap));
  CIP_TRY(dev_alloc(h, &h->scalar, 8));
  CIP_CUDA(cudaStreamSynchronize(s));
  h->st.n = n; h->st.m = m; h->st.p = p; h->st.n_pad = h->n_pad; h->st.m_pad = h->m_pad; h->st.p_pad = h->p_pad;
  return 0;
}

}  // namespace

namespace cip {
int engine_create_single(cip_handle* out, int n, int m, int p, const double* Q, int ldq, const double* A, int lda,
                         const double* G, int ldg, const cip_csc* Qs, const cip_csc* As, const cip_csc* Gs,
                         int ncones, const int* cone_type, const int* cone_dim, const cip_options* opts) {
  return create_impl(out, n, m, p, Q, ldq, A, lda, G, ldg, Qs, As, Gs, ncones, cone_type, cone_dim, opts,
                     /*shard=*/true);
}
}  // namespace cip

namespace {
// opts.ngpus > 1 (and the field is inside the caller's struct): single-process multi-GPU handle
bool wants_multi(const cip_options* opts) {
  return opts && (size_t)opts->struct_size >= offsetof(cip_options, ngpus) + sizeof(int) && opts->ngpus > 1;
}
// a sharded handle with opts.row_structure = 1: refused before any device work
bool reject_sharded_structure(const cip_options* opts) {
  if (opts && (size_t)opts->struct_size >= offsetof(cip_options, row_structure) + sizeof(int) &&
      opts->row_structure != 0) {
    set_error("row_structure is supported on single-device handles only (ngpus = %d)", opts->ngpus);
    return true;
  }
  return false;
}
}  // namespace

extern "C" {

int cip_create(cip_handle* out, int n, int m, int p, const double* Q, int ldq, const double* A, int lda,
               const double* G, int ldg, int ncones, const int* cone_type, const int* cone_dim,
               const cip_options* opts) {
  if (wants_multi(opts)) {
    if (!out || n <= 0 || m < 0 || p < 0 || ncones < 0 || (ncones > 0 && (!cone_type || !cone_dim))) {
      set_error("cip_create: bad dimensions n=%d m=%d p=%d ncones=%d", n, m, p, ncones);
      return -1;
    }
    if (reject_sharded_structure(opts)) return -1;
    return multi_create(out, n, m, p, Q, ldq, A, lda, G, ldg, nullptr, nullptr, nullptr, ncones, cone_type,
                        cone_dim, opts);
  }
  return create_impl(out, n, m, p, Q, ldq, A, lda, G, ldg, nullptr, nullptr, nullptr, ncones, cone_type, cone_dim,
                     opts);
}

int cip_create_csc(cip_handle* out, int n, const cip_csc* Q, const cip_csc* A, const cip_csc* G, int ncones,
                   const int* cone_type, const int* cone_dim, const cip_options* opts) {
  if (!A || A->ncols != n || (Q && (Q->nrows != n || Q->ncols != n)) || (G && G->nrows > 0 && G->ncols != n)) {
    set_error("cip_create_csc: inconsistent matrix shapes");
    return -1;
  }
  cip_options o{};
  o.dist_chol = -1;
  o.aug_rho = -1.0;
  if (opts) memcpy(&o, opts, std::min<size_t>(sizeof(o), (size_t)opts->struct_size));
  else o.device = -1;
  o.struct_size = sizeof(o);
  o.q_kind = 2;                         // Q comes from the CSC arrays (or is zero when Q == NULL)
  const int p = G ? G->nrows : 0;
  if (wants_multi(&o)) {
    if (!out || n <= 0 || ncones < 0 || (ncones > 0 && (!cone_type || !cone_dim))) {
      set_error("cip_create_csc: bad arguments");
      return -1;
    }
    if (reject_sharded_structure(&o)) return -1;
    return multi_create(out, n, A->nrows, p, nullptr, 0, nullptr, 0, nullptr, 0, Q, A, (p > 0) ? G : nullptr, ncones,
                        cone_type, cone_dim, &o);
  }
  return create_impl(out, n, A->nrows, p, nullptr, 0, nullptr, 0, nullptr, 0, Q, A, (p > 0) ? G : nullptr, ncones,
                     cone_type, cone_dim, &o);
}

int cip_destroy(cip_handle h) {
  if (!h) return 0;
  if (h->multi) return multi_destroy(h);
  cudaSetDevice(h->device);
  if (h->own_stream) cudaStreamSynchronize(h->stream);
  if (h->comm) {
    const NcclApi* api = nccl_api();
    if (api) api->CommDestroy(h->comm);
  }
  void* ptrs[] = {h->At4, h->Atil4, h->Qq4, h->H4, h->Winv, h->G4, h->Z4, h->S4, h->Sbase4, h->WinvS, h->info,
                  h->d_type, h->d_off, h->d_rowcone, h->d_qlist, h->d_slist, h->F.kind, h->F.a, h->F.b, h->F.D,
                  h->Fi.kind, h->Fi.a, h->Fi.b, h->Fi.D, h->partial, h->scalar, h->F.R, h->F.Ri, h->d_sord, h->d_roff, h->gemm_ws};
  for (void* p : ptrs) if (p) cudaFree(p);
  for (void* p : h->owned) cudaFree(p);
  for (auto v : h->nv) if (v) cudaFree(v);
  for (auto v : h->mv) if (v) cudaFree(v);
  for (auto v : h->pv) if (v) cudaFree(v);
  for (auto v : h->nv2) if (v) cudaFree(v);
  for (auto v : h->mv2) if (v) cudaFree(v);
  for (auto v : h->pv2) if (v) cudaFree(v);
  chol_free_plan(&h->cholH);
  chol_free_plan(&h->cholS);
  chol_free_plan(&h->rs.sp.chol);
  if (h->Hp) cudaFree(h->Hp);
  if (h->d_sws) cudaFree(h->d_sws);
  if (h->cs) cudaStreamDestroy(h->cs);
  if (h->s2) cudaStreamDestroy(h->s2);
  for (auto e : h->evc) if (e) cudaEventDestroy(e);
  for (auto e : h->ev) if (e) cudaEventDestroy(e);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  cudaGetLastError();
  delete h;
  return 0;
}

int cip_nccl_unique_id(unsigned char id_out[128]) {
  const NcclApi* api = nccl_api();
  if (!api) return -1;
  NcclId id;
  int r = api->GetUniqueId(&id);
  if (r != 0) {
    set_error("ncclGetUniqueId failed: %s", api->GetErrorString(r));
    return -1;
  }
  memcpy(id_out, id.internal, 128);
  return 0;
}

int cip_comm_init(cip_handle h, int nranks, int rank, const unsigned char id[128]) {
  CIP_TRY(check(h));
  if (h->multi) { set_error("cip_comm_init: a single-process multi-GPU handle (opts.ngpus) owns its communicators"); return -1; }
  if (nranks <= 1) return 0;
  if (h->rs.on) { set_error("cip_comm_init: row_structure is supported on single-device handles only"); return -1; }
  const NcclApi* api = nccl_api();
  if (!api) return -1;
  NcclId nid;
  memcpy(nid.internal, id, 128);
  int r = api->CommInitRank(&h->comm, nranks, nid, rank);
  if (r != 0) {
    set_error("ncclCommInitRank failed: %s", api->GetErrorString(r));
    h->comm = nullptr;
    return -1;
  }
  h->nranks = nranks;
  h->rank = rank;
  return engine_setup_comm(h);
}

int cip_set_scaling(cip_handle h, const int* kind, const double* fa, const double* fb, const double* fD,
                    const double* fR) {
  CIP_TRY(check(h));
  if (h->multi) return multi_factor(h, kind, fa, fb, fD, fR, 0);
  return set_scaling_from_user(h, kind, fa, fb, fD, fR);
}

int cip_form_H(cip_handle h) {
  CIP_TRY(check(h));
  if (h->multi) return multi_simple(h, 0, nullptr, 0);
  CIP_TRY(form_H(h));
  return 0;
}

int cip_factor_H(cip_handle h) {
  CIP_TRY(check(h));
  if (h->multi) return multi_simple(h, 1, nullptr, 0);
  CIP_CUDA(cudaEventRecord(h->ev[3], h->stream));
  return factor_H(h);
}

int cip_factor(cip_handle h, const int* kind, const double* fa, const double* fb, const double* fD,
               const double* fR) {
  CIP_TRY(check(h));
  if (h->multi) return multi_factor(h, kind, fa, fb, fD, fR, 1);
  CIP_TRY(set_scaling_from_user(h, kind, fa, fb, fD, fR));
  CIP_TRY(form_H(h));
  return factor_H(h);
}

int cip_nt_scaling(cip_handle h, const double* v, const double* s, double* lambda_out) {
  CIP_TRY(check(h));
  if (h->multi) return multi_nt_scaling(h, v, s, lambda_out, 0);
  const double *vp, *sp;
  CIP_TRY(vec_in(h, h->mv[7], v, h->m, &vp));
  CIP_TRY(vec_in(h, h->mv[8], s, h->m, &sp));
  double* lp = vec_out(h, h->mv[9], lambda_out, h->m);
  if (h->cd.ns > 0) CIP_CUDA(cudaMemsetAsync(h->info + 2, 0, sizeof(int), h->stream));
  CIP_TRY(cone_nt_scaling(h->cd, vp, sp, h->F, h->Fi, lp, h->info + 2, h->stream));
  h->have_scaling = true;
  CIP_TRY(vec_out_done(h, lambda_out, lp, h->m));
  if (h->cd.ns > 0) {
    // an S-cone iterate that is not positive definite has no NT scaling (PosDefException in the reference,
    // src/ConicIP.jl:201-202): report it as a numerical failure (> 0) instead of handing out garbage
    int bad = 0;
    CIP_CUDA(cudaMemcpyAsync(&bad, h->info + 2, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CIP_CUDA(cudaStreamSynchronize(h->stream));
    h->need_sync = false;
    if (bad != 0) {
      h->have_scaling = false;
      set_error("nt_scaling: the iterate of S cone %d is not positive definite (PosDefException in the reference)",
                bad - 1);
      return bad;
    }
  }
  return finish(h);
}

int cip_factor_from_point(cip_handle h, const double* v, const double* s, double* lambda_out) {
  if (h && h->multi) return multi_nt_scaling(h, v, s, lambda_out, 1);
  CIP_TRY(cip_nt_scaling(h, v, s, lambda_out));      // > 0 (S-cone iterate not PD) is returned as it is
  CIP_TRY(form_H(h));
  return factor_H(h);
}

int cip_get_scaling(cip_handle h, int* kind, double* fa, double* fb, double* fD, double* fR) {
  CIP_TRY(check(h));
  if (h->multi) return multi_get_scaling(h, kind, fa, fb, fD, fR);
  if (!h->have_scaling) { set_error("no scaling set"); return -1; }
  if (kind) {
    CIP_CUDA(cudaMemcpyAsync(kind, h->F.kind, sizeof(int) * h->ncones, cudaMemcpyDefault, h->stream));
    h->need_sync = true;
  }
  CIP_TRY(stage_out(h, fa, h->F.a, h->m));
  CIP_TRY(stage_out(h, fb, h->F.b, h->m));
  CIP_TRY(stage_out(h, fD, h->F.D, h->ncones));
  CIP_TRY(stage_out(h, fR, h->F.R, h->r_total));     // all S cones, slist order (k*k each)
  return finish(h);
}

int cip_apply(cip_handle h, int op, const double* x, double* y) {
  CIP_TRY(check(h));
  if (h->multi) return multi_apply(h, op, x, y);
  if (!h->have_scaling) { set_error("no scaling set"); return -1; }
  if (op < CIP_OP_F || op > CIP_OP_FINV) { set_error("cip_apply: bad op %d", op); return -1; }
  const double* xp;
  CIP_TRY(vec_in(h, h->mv[7], x, h->m, &xp));
  double* yp = (y != x) ? vec_out(h, h->mv[8], y, h->m) : h->mv[8];
  CIP_TRY(cone_apply(h->cd, h->F, h->Fi, op, xp, yp, h->stream));
  CIP_TRY(vec_out_done(h, y, yp, h->m));
  return finish(h);
}

int cip_maxstep(cip_handle h, const double* x, const double* d, double d_scale, double* alpha_out) {
  CIP_TRY(check(h));
  if (h->multi) return multi_maxstep(h, x, d, d_scale, alpha_out);
  const double *xp, *dp = nullptr;
  CIP_TRY(vec_in(h, h->mv[7], x, h->m, &xp));
  if (d) CIP_TRY(vec_in(h, h->mv[8], d, h->m, &dp));
  CIP_TRY(cone_maxstep(h->cd, xp, dp, d_scale, nullptr, 0, h->scalar, h->stream));
  unsigned long long key = 0;
  CIP_CUDA(cudaMemcpyAsync(&key, h->scalar, 8, cudaMemcpyDeviceToHost, h->stream));
  CIP_CUDA(cudaStreamSynchronize(h->stream));
  const unsigned long long u = (key >> 63) ? (key & 0x7fffffffffffffffull) : ~key;
  double r;
  memcpy(&r, &u, 8);
  if (key == ~0ull) r = INFINITY;               // the preset value: no cone bounded the step
  *alpha_out = r;
  return 0;
}

int cip_cone_prod(cip_handle h, const double* x, const double* y, double* o) {
  CIP_TRY(check(h));
  if (h->multi) return multi_prod_div(h, x, y, o, 0);
  const double *xp, *yp;
  CIP_TRY(vec_in(h, h->mv[7], x, h->m, &xp));
  CIP_TRY(vec_in(h, h->mv[8], y, h->m, &yp));
  double* op_ = (o != x && o != y) ? vec_out(h, h->mv[9], o, h->m) : h->mv[9];
  CIP_TRY(cone_prod(h->cd, xp, yp, op_, h->stream));
  CIP_TRY(vec_out_done(h, o, op_, h->m));
  return finish(h);
}

int cip_cone_div(cip_handle h, const double* x, const double* y, double* o) {
  CIP_TRY(check(h));
  if (h->multi) return multi_prod_div(h, x, y, o, 1);
  const double *xp, *yp;
  CIP_TRY(vec_in(h, h->mv[7], x, h->m, &xp));
  CIP_TRY(vec_in(h, h->mv[8], y, h->m, &yp));
  double* op_ = (o != x && o != y) ? vec_out(h, h->mv[9], o, h->m) : h->mv[9];
  CIP_TRY(cone_div(h->cd, xp, yp, op_, h->stream));
  CIP_TRY(vec_out_done(h, o, op_, h->m));
  return finish(h);
}

int cip_solve(cip_handle h, const double* ry, const double* rw, const double* rv, double* dy, double* dw,
              double* dv) {
  CIP_TRY(check(h));
  if (h->multi) return multi_solve(h, ry, rw, rv, dy, dw, dv);
  if (!h->have_factor) { set_error("cip_solve before cip_factor"); return -1; }
  cudaStream_t s = h->stream;
  CIP_CUDA(cudaEventRecord(h->ev[6], s));
  const double *ryp, *rvp;
  CIP_TRY(vec_in(h, h->nv[0], ry, h->n, &ryp));
  if (h->p) CIP_TRY(stage_in(h, h->pv[0], rw, h->p));
  CIP_TRY(vec_in(h, h->mv[0], rv, h->m, &rvp));
  double* dvp = (dv != rv) ? vec_out(h, h->mv[5], dv, h->m) : h->mv[5];
  // t1 = F^-T (F^-T v)                                   (src/kktsolvers.jl:326)
  // (= inv(F'F) v; for the non-symmetric VecCongurance blocks this is inv(F) inv(F)' v, which is
  //  what the 3x3 system requires -- the reference's pivot is only right for symmetric F, SURVEY 3b)
  CIP_TRY(cone_apply_invsq(h->cd, h->F, h->Fi, rvp, h->mv[2], nullptr, h->mv[1], s));
  // rhs = y + A' t1                                      (:327); single GPU: y is added in the mat-vec's second pass
  if (h->rs.on) {
    CIP_TRY(structure_AT(h, h->nv[2], h->mv[2], ryp, 0));
  } else if (h->m && !h->comm) {
    CIP_TRY(q4_mv_rows(h->nv[2], h->At4, h->n_pad, h->n, h->m, h->mv[2], h->partial, h->partial_cap, s, ryp));
  } else {
    if (h->m) CIP_TRY(q4_mv_rows(h->nv[1], h->At4, h->n_pad, h->n, h->m, h->mv[2], h->partial, h->partial_cap, s));
    else CIP_TRY(fill_zero(h->nv[1], h->n, s));
    CIP_TRY(allreduce(h, h->nv[1], h->n));
    CIP_TRY(vec_axpby(h->nv[2], 1.0, ryp, 1.0, h->nv[1], h->n, s));
  }
  if (h->aug_rows > 0) {        // rhs += rho G' rw  (same (dy, dw) as the unaugmented system)
    CIP_TRY(q4_mv_k(h->nv[4], h->G4, h->p_pad, h->p, h->n, h->pv[0], s));
    CIP_TRY(vec_axpby(h->nv[2], 1.0, h->nv[2], h->aug_rho, h->nv[4], h->n, s));
  }
  // 2x2 solve with H = L L' and the Schur complement on G (:299)
  if (h->rs.sp.on) {
    CIP_TRY(split_solve(h, h->nv, h->pv, 0, h->p > 0));
  } else {
    CIP_TRY(chol_fwd(h->cholH, h->nv[2], h->nv[3], s));
    if (h->p) {
      CIP_TRY(q4_mv_rows(h->pv[1], h->Z4, h->p_pad, h->p, h->n, h->nv[3], h->partial, h->partial_cap, s));
      CIP_TRY(vec_axpby(h->pv[2], 1.0, h->pv[1], -1.0, h->pv[0], h->p, s));
      CIP_TRY(chol_fwd(h->cholS, h->pv[2], h->pv[3], s));
      CIP_TRY(chol_bwd(h->cholS, h->pv[3], h->pv[4], s));
      CIP_TRY(q4_mv_k(h->nv[4], h->Z4, h->p_pad, h->p, h->n, h->pv[4], s));
      CIP_TRY(vec_axpby(h->nv[3], 1.0, h->nv[3], -1.0, h->nv[4], h->n, s));
    }
    CIP_TRY(chol_bwd(h->cholH, h->nv[3], h->nv[5], s));
  }
  // dv = t1 - F^-T F^-T (A dy)                           (:328)
  if (h->m) {
    if (h->rs.on) CIP_TRY(structure_A(h, h->mv[3], h->nv[5], 0));
    else CIP_TRY(q4_mv_k(h->mv[3], h->At4, h->n_pad, h->n, h->m, h->nv[5], s));
    CIP_TRY(cone_apply_invsq(h->cd, h->F, h->Fi, h->mv[3], dvp, h->mv[2], h->mv[1], s));   // t1 - (F'F)^-1 (A dy)
  }
  CIP_CUDA(cudaEventRecord(h->ev[7], s));
  CIP_TRY(stage_out(h, dy, h->nv[5], h->n));
  if (h->p) CIP_TRY(stage_out(h, dw, h->pv[4], h->p));
  CIP_TRY(vec_out_done(h, dv, dvp, h->m));
  h->st.solves++;
  if (h->need_sync || h->always_sync) {
    // the call synchronises anyway: also read the give-up flag of the persistent sweeps (a hand-off that never
    // arrived -- a bug, not a numerical condition -- must not pass for a solution)
    int bad[2] = {0, 0};
    if (h_sweep_err(h)) CIP_CUDA(cudaMemcpyAsync(&bad[0], h_sweep_err(h), sizeof(int), cudaMemcpyDeviceToHost, s));
    if (h->p) CIP_CUDA(cudaMemcpyAsync(&bad[1], h->cholS.sweep_err, sizeof(int), cudaMemcpyDeviceToHost, s));
    CIP_TRY(finish(h));
    if (bad[0] || bad[1]) {
      set_error("cip_solve: a triangular sweep gave up waiting for a solution block (internal error)");
      return -4;
    }
    return 0;
  }
  return finish(h);
}

// Several right-hand sides through one factorisation.  The pivot algebra of cip_solve runs column by column (the
// sweeps and the cone kernels are per column), but the two products with A -- 2 x 8mn bytes, nine tenths of a
// solve at config 4 -- are shared by PAIRS of columns: A is streamed once per pair.  Column k of every argument
// lies at ptr + k * ld.  Replaces `Z\[dy;dw]` / `pivot` applied to several right-hand sides
// (src/kktsolvers.jl:297-302, :324-332; north_star "the predictor and corrector right-hand sides together").
int cip_solve_multi(cip_handle h, int nrhs, const double* ry, int ldy, const double* rw, int ldw, const double* rv,
                    int ldv, double* dy, double* dw, double* dv) {
  CIP_TRY(check(h));
  if (nrhs < 0 || (nrhs > 1 && (ldy < h->n || ldv < h->m || (h->p > 0 && ldw < h->p)))) {
    set_error("cip_solve_multi: bad nrhs / leading dimensions (nrhs=%d ldy=%d ldw=%d ldv=%d)", nrhs, ldy, ldw, ldv);
    return -1;
  }
  auto col = [](const double* p, int k, int ld) { return p ? p + (size_t)k * ld : nullptr; };
  auto colw = [](double* p, int k, int ld) { return p ? p + (size_t)k * ld : nullptr; };
  if (h->multi) return multi_solve_multi(h, nrhs, ry, ldy, rw, ldw, rv, ldv, dy, dw, dv);
  if (!h->have_factor) { set_error("cip_solve_multi before cip_factor"); return -1; }
  int k = 0;
  for (; k + 1 < nrhs; k += 2) {
    if (!h->nv2[0]) {
      for (auto& v : h->nv2) CIP_TRY(dev_alloc(h, &v, h->n_pad + 4));
      for (auto& v : h->mv2) CIP_TRY(dev_alloc(h, &v, h->m_pad + 4));
      for (auto& v : h->pv2) CIP_TRY(dev_alloc(h, &v, h->p_pad + 4));
    }
    cudaStream_t s = h->stream;
    double** NVs[2] = {h->nv, h->nv2};
    double** MVs[2] = {h->mv, h->mv2};
    double** PVs[2] = {h->pv, h->pv2};
    const double *ryp[2], *rvp[2];
    double* dvp[2];
    CIP_CUDA(cudaEventRecord(h->ev[6], s));
    for (int b = 0; b < 2; ++b) {
      double **nv = NVs[b], **mv = MVs[b], **pv = PVs[b];
      CIP_TRY(vec_in(h, nv[0], col(ry, k + b, ldy), h->n, &ryp[b]));
      if (h->p) CIP_TRY(stage_in(h, pv[0], col(rw, k + b, ldw), h->p));
      CIP_TRY(vec_in(h, mv[0], col(rv, k + b, ldv), h->m, &rvp[b]));
      double* out = colw(dv, k + b, ldv);
      dvp[b] = (out != rvp[b]) ? vec_out(h, mv[5], out, h->m) : mv[5];
      CIP_TRY(cone_apply_invsq(h->cd, h->F, h->Fi, rvp[b], mv[2], nullptr, mv[1], s));          // t1 (:326)
    }
    // rhs = y + A' t1 (:327) for both columns in one pass over A
    if (h->rs.on) {
      CIP_TRY(structure_AT2(h, h->nv[2], h->nv2[2], h->mv[2], h->mv2[2], ryp[0], ryp[1]));
    } else if (h->m && !h->comm) {
      CIP_TRY(q4_mv_rows2(h->nv[2], h->nv2[2], h->At4, h->n_pad, h->n, h->m, h->mv[2], h->mv2[2], h->partial,
                          h->partial_cap, s, ryp[0], ryp[1]));
    } else {
      if (h->m) {
        CIP_TRY(q4_mv_rows2(h->nv[1], h->nv2[1], h->At4, h->n_pad, h->n, h->m, h->mv[2], h->mv2[2], h->partial,
                            h->partial_cap, s));
      } else {
        CIP_TRY(fill_zero(h->nv[1], h->n, s));
        CIP_TRY(fill_zero(h->nv2[1], h->n, s));
      }
      for (int b = 0; b < 2; ++b) {
        CIP_TRY(allreduce(h, NVs[b][1], h->n));
        CIP_TRY(vec_axpby(NVs[b][2], 1.0, ryp[b], 1.0, NVs[b][1], h->n, s));
      }
    }
    for (int b = 0; b < 2; ++b) {
      double **nv = NVs[b], **pv = PVs[b];
      if (h->aug_rows > 0) {
        CIP_TRY(q4_mv_k(nv[4], h->G4, h->p_pad, h->p, h->n, pv[0], s));
        CIP_TRY(vec_axpby(nv[2], 1.0, nv[2], h->aug_rho, nv[4], h->n, s));
      }
      if (h->rs.sp.on) {
        CIP_TRY(split_solve(h, nv, pv, b, h->p > 0));
        continue;
      }
      CIP_TRY(chol_fwd(h->cholH, nv[2], nv[3], s));
      if (h->p) {
        CIP_TRY(q4_mv_rows(pv[1], h->Z4, h->p_pad, h->p, h->n, nv[3], h->partial, h->partial_cap, s));
        CIP_TRY(vec_axpby(pv[2], 1.0, pv[1], -1.0, pv[0], h->p, s));
        CIP_TRY(chol_fwd(h->cholS, pv[2], pv[3], s));
        CIP_TRY(chol_bwd(h->cholS, pv[3], pv[4], s));
        CIP_TRY(q4_mv_k(nv[4], h->Z4, h->p_pad, h->p, h->n, pv[4], s));
        CIP_TRY(vec_axpby(nv[3], 1.0, nv[3], -1.0, nv[4], h->n, s));
      }
      CIP_TRY(chol_bwd(h->cholH, nv[3], nv[5], s));
    }
    // dv = t1 - F^-T F^-T (A dy) (:328): A dy for both columns in one pass over A
    if (h->m) {
      if (h->rs.on) CIP_TRY(structure_A2(h, h->mv[3], h->mv2[3], h->nv[5], h->nv2[5]));
      else CIP_TRY(q4_mv_k2(h->mv[3], h->mv2[3], h->At4, h->n_pad, h->n, h->m, h->nv[5], h->nv2[5], s));
      for (int b = 0; b < 2; ++b)
        CIP_TRY(cone_apply_invsq(h->cd, h->F, h->Fi, MVs[b][3], dvp[b], MVs[b][2], MVs[b][1], s));
    }
    CIP_CUDA(cudaEventRecord(h->ev[7], s));
    for (int b = 0; b < 2; ++b) {
      CIP_TRY(stage_out(h, colw(dy, k + b, ldy), NVs[b][5], h->n));
      if (h->p) CIP_TRY(stage_out(h, colw(dw, k + b, ldw), PVs[b][4], h->p));
      CIP_TRY(vec_out_done(h, colw(dv, k + b, ldv), dvp[b], h->m));
    }
    h->st.solves += 2;
    int bad[2] = {0, 0};
    if (h->need_sync || h->always_sync) {
      if (h_sweep_err(h)) CIP_CUDA(cudaMemcpyAsync(&bad[0], h_sweep_err(h), sizeof(int), cudaMemcpyDeviceToHost, s));
      if (h->p) CIP_CUDA(cudaMemcpyAsync(&bad[1], h->cholS.sweep_err, sizeof(int), cudaMemcpyDeviceToHost, s));
    }
    CIP_TRY(finish(h));
    if (bad[0] || bad[1]) {
      set_error("cip_solve_multi: a triangular sweep gave up waiting for a solution block (internal error)");
      return -4;
    }
  }
  if (k < nrhs)
    return cip_solve(h, col(ry, k, ldy), col(rw, k, ldw), col(rv, k, ldv), colw(dy, k, ldy), colw(dw, k, ldw),
                     colw(dv, k, ldv));
  return 0;
}

int cip_solve_H(cip_handle h, const double* rhs, double* x) {
  CIP_TRY(check(h));
  if (h->multi) { set_error("cip_solve_H: test hook, single-device handles only"); return -1; }
  if (!h->have_factor) { set_error("cip_solve_H before cip_factor"); return -1; }
  cudaStream_t s = h->stream;
  CIP_TRY(stage_in(h, h->nv[2], rhs, h->n));
  CIP_CUDA(cudaEventRecord(h->ev[6], s));
  if (h->rs.sp.on) {
    CIP_TRY(split_solve(h, h->nv, h->pv, 0, false));
  } else {
    CIP_TRY(chol_fwd(h->cholH, h->nv[2], h->nv[3], s));
    CIP_TRY(chol_bwd(h->cholH, h->nv[3], h->nv[5], s));
  }
  CIP_CUDA(cudaEventRecord(h->ev[7], s));
  CIP_TRY(stage_out(h, x, h->nv[5], h->n));
  h->st.solves++;
  return finish(h);
}

int cip_mul_A(cip_handle h, int trans, const double* x, double* y) {
  CIP_TRY(check(h));
  if (h->multi) return multi_mul_A(h, trans, x, y);
  cudaStream_t s = h->stream;
  if (!trans) {
    const double* xp;
    CIP_TRY(vec_in(h, h->nv[6], x, h->n, &xp));
    double* yp = vec_out(h, h->mv[6], y, h->m);
    if (h->rs.on) CIP_TRY(structure_A(h, yp, xp, 0));
    else CIP_TRY(q4_mv_k(yp, h->At4, h->n_pad, h->n, h->m, xp, s));
    CIP_TRY(vec_out_done(h, y, yp, h->m));
  } else {
    const double* xp;
    CIP_TRY(vec_in(h, h->mv[6], x, h->m, &xp, /*padded=*/true));
    double* yp = vec_out(h, h->nv[6], y, h->n);
    if (h->rs.on) CIP_TRY(structure_AT(h, yp, xp, nullptr, 0));
    else if (h->m) CIP_TRY(q4_mv_rows(yp, h->At4, h->n_pad, h->n, h->m, xp, h->partial, h->partial_cap, s));
    else CIP_TRY(fill_zero(yp, h->n, s));
    CIP_TRY(allreduce(h, yp, h->n));
    CIP_TRY(vec_out_done(h, y, yp, h->n));
  }
  return finish(h);
}

int cip_mul_G(cip_handle h, int trans, const double* x, double* y) {
  CIP_TRY(check(h));
  if (h->multi) return multi_mul_GQ(h, 0, trans, x, y);
  cudaStream_t s = h->stream;
  if (h->p == 0) {
    if (trans) {
      CIP_TRY(fill_zero(h->nv[6], h->n, s));
      CIP_TRY(stage_out(h, y, h->nv[6], h->n));
    }
    return finish(h);
  }
  if (!trans) {
    CIP_TRY(stage_in(h, h->nv[6], x, h->n));
    CIP_TRY(q4_mv_rows(h->pv[5], h->G4, h->p_pad, h->p, h->n, h->nv[6], h->partial, h->partial_cap, s));
    CIP_TRY(stage_out(h, y, h->pv[5], h->p));
  } else {
    CIP_TRY(stage_in(h, h->pv[5], x, h->p));
    CIP_TRY(q4_mv_k(h->nv[6], h->G4, h->p_pad, h->p, h->n, h->pv[5], s));
    CIP_TRY(stage_out(h, y, h->nv[6], h->n));
  }
  return finish(h);
}

int cip_mul_Q(cip_handle h, const double* x, double* y) {
  CIP_TRY(check(h));
  if (h->multi) return multi_mul_GQ(h, 1, 0, x, y);
  cudaStream_t s = h->stream;
  const double* xp;
  CIP_TRY(vec_in(h, h->nv[6], x, h->n, &xp, /*padded=*/true));
  double* yp = (y != x) ? vec_out(h, h->nv[7], y, h->n) : h->nv[7];
  if (h->rs.sp.on) CIP_TRY(split_mul_Q(h, yp, xp));
  else CIP_TRY(q4_mv_rows(yp, h->Qq4, h->n_pad, h->n, h->n, xp, h->partial, h->partial_cap, s));
  CIP_TRY(vec_out_done(h, y, yp, h->n));
  return finish(h);
}

int cip_stats(cip_handle h, cip_stats_t* out) {
  CIP_TRY(check(h));
  if (h->multi) return multi_stats(h, out);
  float ms = 0;
  if (h->st.solves > 0 && cudaEventSynchronize(h->ev[7]) == cudaSuccess &&
      cudaEventElapsedTime(&ms, h->ev[6], h->ev[7]) == cudaSuccess) h->st.ms_solve = ms;
  else cudaGetLastError();
  h->st.device_bytes = h->bytes;
  h->st.kernel_launches = cip::g_launches;
  *out = h->st;
  return 0;
}

int cip_structure_info(cip_handle h, cip_structure_t* out) {
  CIP_TRY(check(h));
  if (!out || out->struct_size < (int)sizeof(int)) {
    set_error("cip_structure_info: out->struct_size must be set");
    return -1;
  }
  cip_structure_t r{};
  r.struct_size = out->struct_size;
  const RowStructure& rs = h->rs;      // (a multi-GPU front never has it on)
  if (rs.on) {
    r.enabled = 1;
    r.singleton_rows = rs.nsing;
    r.empty_rows = rs.nempty;
    r.rest_rows = rs.nr;
    r.rest_cols = rs.nJ;
    r.compressed = rs.compressed || rs.sp.on;
    r.base_has_gtg = rs.base_has_gtg;
  }
  memcpy(out, &r, std::min<size_t>(sizeof(r), (size_t)out->struct_size));
  return 0;
}

int cip_split_info(cip_handle h, cip_split_t* out) {
  CIP_TRY(check(h));
  if (!out || out->struct_size < (int)sizeof(int)) {
    set_error("cip_split_info: out->struct_size must be set");
    return -1;
  }
  cip_split_t r{};
  r.struct_size = out->struct_size;
  const RowStructure::Split& sp = h->rs.sp;      // (a multi-GPU front never has it on)
  if (sp.on) {
    r.enabled = 1;
    r.coupled_cols = sp.nK;
    r.diagonal_cols = h->n - sp.nK;
    r.cols_from_rest = sp.from_rest;
    r.cols_from_Q = sp.from_Q;
    r.cols_from_G = sp.from_G;
  }
  memcpy(out, &r, std::min<size_t>(sizeof(r), (size_t)out->struct_size));
  return 0;
}

int cip_get_H(cip_handle h, double* out, int ldo) {
  CIP_TRY(check(h));
  if (h->multi) return multi_simple(h, 3, out, ldo);
  double* tmp = nullptr;
  CIP_CUDA(cudaMalloc(&tmp, (size_t)h->n * h->n * 8));
  const int rc = h->rs.sp.on ? split_get_H(h, tmp) : unpack_rows_q4(tmp, h->n, h->H4, h->n_pad, h->n, h->n, h->stream);
  if (rc != 0) cudaFree(tmp);
  CIP_TRY(rc);
  CIP_CUDA(cudaMemcpy2DAsync(out, (size_t)ldo * 8, tmp, (size_t)h->n * 8, (size_t)h->n * 8, h->n, cudaMemcpyDefault,
                             h->stream));
  CIP_CUDA(cudaStreamSynchronize(h->stream));
  cudaFree(tmp);
  return 0;
}

int cip_sync(cip_handle h) {
  CIP_TRY(check(h));
  if (h->multi) return multi_simple(h, 2, nullptr, 0);
  CIP_CUDA(cudaStreamSynchronize(h->stream));
  return 0;
}

void* cip_stream(cip_handle h) { return (h && !h->multi) ? (void*)h->stream : nullptr; }

int cip_set_stream(cip_handle h, void* stream) {
  CIP_TRY(check(h));
  if (h->multi) {
    set_error("cip_set_stream: a single-process multi-GPU handle runs one stream per device; calls return with all of them idle");
    return -1;
  }
  CIP_CUDA(cudaStreamSynchronize(h->stream));
  h->stream = reinterpret_cast<cudaStream_t>(stream);
  return 0;
}

int cip_measure_fp64_peaks(int device, double* dmma_tflops, double* dfma_tflops) {
  if (device >= 0) CIP_CUDA(cudaSetDevice(device));
  return measure_fp64_peaks(dmma_tflops, dfma_tflops);
}

}  // extern "C"
