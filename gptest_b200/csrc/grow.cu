// grow.cu - exact GP regression on a GROWING training set: the factor is kept on the device and extended.
//
// GP_parameter_fit.py:61-63 replays an experiment: for every prefix X[:i], Y[:i] (five more points each time) it
// calls gpm.set_XY and predicts on a 100x100 grid (:52), i.e. a full refit per step.  With the hyper-parameters
// fixed, the Cholesky factor of the longer prefix contains the factor of the shorter one, so here appending m
// points to n costs O((n+m)^2 m) instead of (n+m)^3/3, from the same kernels as the full fit:
//
//   rows r0.. of K          se_build (rectangular part left of r0, symmetric block from r0)     HBM bound
//   X <- X L11^-T           non-factor sweep of the new tile rows over the finished columns     DMMA
//   S  = K22 - X X^T        one trailing update with K = r0 (long k loop)                       DMMA
//   S  = L22 L22^T          blocked Cholesky of the trailing block                              DMMA
//   z2 = L22^-1 (y2 - X z1) row_dot + forward substitution steps from tile r0/128               HBM bound
//
// r0 = the start of the 128-tile that holds the first new point (earlier tile columns are final).  The result
// equals a fit from scratch on the enlarged set up to rounding (tests/test_gpu_grow.py).
// Prediction sweeps blocks of test rows against the current factor (no refactorisation).
#include <vector>

#include "../../include/gpb200.h"
#include "gpb_context.cuh"

namespace gpb {

constexpr int64_t PRED_ROWS = 2048;     // test points swept per pass
constexpr int SPLIT_Q = 2;              // split-k chunk of the thin trailing update, in tiles (k = 256 per partial)
constexpr int64_t THIN_MAX = 8;         // appends of up to this many points inside the last tile use the substitution path
                                        // (N = 16384: 1 point 3.0 ms, 5 points 3.9 ms, 16 points 6.1 ms vs 5.4 ms for the tile sweep)

struct GrowState {
  int64_t cap = 0, cap_pad = 0, n = 0;
  int d = 0, kind = 0;
  double mean = 0.0;
  DevBuf X, yc, XsT, sq, A, Dinv, diag, info, par, r, z, tmp, out, part;
  TileMaps mapA, mapD;
  int last_info = 0;
};

void grow_release(gpb_handle* h) {
  delete h->grow;
  h->grow = nullptr;
}

namespace {

// S (128 x 128 at `dst`, pitch ld) -= sum_b P[b] (partials of a split-k product, fixed order: deterministic)
__global__ void __launch_bounds__(256) sub_partials_kernel(double* __restrict__ dst, int64_t ld,
                                                           const double* __restrict__ P, int nb) {
  const int e = blockIdx.x * 256 + threadIdx.x;          // 64 CTAs x 256 threads = one tile
  double s = 0.0;
  for (int b = 0; b < nb; ++b) s += P[static_cast<int64_t>(b) * TILE * TILE + e];
  dst[static_cast<int64_t>(e >> 7) * ld + (e & 127)] -= s;
}

__global__ void sub_vec_kernel(double* r, const double* y, const double* t, int64_t n) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) r[i] = y[i] - t[i];
}

// a view of the stored factor: rows/columns [0, n_pad) of the buffer, `rows_total` rows visible to the sweep
FactorMat view(GrowState* g, int64_t n_pad, int64_t rows_total) {
  FactorMat m;
  m.A = g->A.as<double>(); m.ld = g->cap_pad; m.n_pad = n_pad; m.rows_total = rows_total;
  m.batch = 1; m.batch_stride = 0;
  m.Dinv = g->Dinv.as<double>(); m.dinv_bs = 0;
  m.diag = g->diag.as<double>(); m.diag_bs = 0;
  m.info = g->info.as<int>();
  m.mapA = g->mapA; m.mapD = g->mapD;
  return m;
}

}  // namespace
}  // namespace gpb

using namespace gpb;

extern "C" {

int gpb_gpr_grow_begin(gpb_handle* h, const double* khyp, int32_t d, double mean, int64_t capacity) {
  GPB_ENTRY_BEGIN
  GPB_REQUIRE(khyp && d > 0 && capacity > 0, "grow_begin: khyp, d > 0 and capacity > 0 are required");
  grow_release(h);
  GrowState* g = new GrowState;
  h->grow = g;
  g->cap = capacity; g->cap_pad = round_up(capacity, TILE); g->d = d; g->mean = mean; g->n = 0; g->kind = h->cov_kind;
  const int64_t cp = g->cap_pad, rows_alloc = cp + PRED_ROWS;
  g->X.ensure(static_cast<size_t>(capacity) * d * 8);
  g->yc.ensure(static_cast<size_t>(cp) * 8);
  g->XsT.ensure((static_cast<size_t>(d) * cp + 64) * 8);      // + 64: the thin path reads a 64-point window from n
  g->sq.ensure(static_cast<size_t>(cp + 64) * 8);
  GPB_CUDA(cudaMemsetAsync(g->XsT.p, 0, (static_cast<size_t>(d) * cp + 64) * 8, h->s0));
  GPB_CUDA(cudaMemsetAsync(g->sq.p, 0, static_cast<size_t>(cp + 64) * 8, h->s0));
  g->A.ensure(static_cast<size_t>(rows_alloc) * cp * 8);
  g->Dinv.ensure(static_cast<size_t>(cp) * TILE * 8);
  g->diag.ensure(static_cast<size_t>(cp) * 8);
  g->info.ensure(64);
  g->r.ensure(static_cast<size_t>(cp) * 8);
  g->z.ensure(static_cast<size_t>(cp) * 8);
  g->tmp.ensure(static_cast<size_t>(cp) * 8);
  g->out.ensure(static_cast<size_t>(2 * PRED_ROWS + 8) * 8);
  g->part.ensure(static_cast<size_t>(cp / TILE / SPLIT_Q + 2) * TILE * TILE * 8);     // split-k partial tiles
  GPB_CUDA(cudaMemsetAsync(g->yc.p, 0, static_cast<size_t>(cp) * 8, h->s0));
  GPB_CUDA(cudaMemsetAsync(g->z.p, 0, static_cast<size_t>(cp) * 8, h->s0));
  GPB_CUDA(cudaMemsetAsync(g->info.p, 0, 64, h->s0));
  upload_params(h, g->par, khyp, d);
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  make_tile_maps(&g->mapA, g->A.as<double>(), cp, rows_alloc, 1, cp, rows_alloc * cp);
  make_tile_maps(&g->mapD, g->Dinv.as<double>(), TILE, cp, 1, TILE, cp * TILE);
  GPB_API_END
}

int64_t gpb_gpr_grow_size(gpb_handle* h) { return (h && h->grow) ? h->grow->n : -1; }

int gpb_gpr_grow_append(gpb_handle* h, const double* X_new, const double* y_new, int64_t m, double* nlml,
                        int32_t* info) {
  GPB_ENTRY_BEGIN
  GrowState* g = h->grow;
  GPB_REQUIRE(g != nullptr, "grow_append: call gpb_gpr_grow_begin first");
  GPB_REQUIRE(X_new && y_new && m > 0 && nlml, "grow_append: null argument");
  GPB_REQUIRE(g->n + m <= g->cap, "grow_append: capacity exceeded");
  GPB_REQUIRE(g->last_info == 0, "grow_append: the stored factor is invalid (an earlier append hit a non-positive pivot)");
  const int d = g->d;
  const int64_t cp = g->cap_pad, n0 = g->n, n1 = n0 + m;
  const int64_t r0 = (n0 / TILE) * TILE, np1 = round_up(n1, TILE);
  const int t0 = static_cast<int>(r0 / TILE), nt1 = static_cast<int>(np1 / TILE);
  double* A = g->A.as<double>();
  const double* ell = g->par.as<double>();
  const double* hyp2 = ell + d;
  cudaStream_t st = h->s0;

  GPB_CUDA(cudaEventRecord(h->tev[0], st));
  {
    double* host = h->pinned(static_cast<size_t>(m) * 8);
    for (int64_t i = 0; i < m; ++i) host[i] = y_new[i] - g->mean;          // y - m (GPr.py:64-65)
    GPB_CUDA(cudaMemcpyAsync(g->yc.as<double>() + n0, host, static_cast<size_t>(m) * 8, cudaMemcpyHostToDevice, st));
    GPB_CUDA(cudaMemcpyAsync(g->X.as<double>() + n0 * d, X_new, static_cast<size_t>(m) * d * 8, cudaMemcpyHostToDevice, st));
  }
  const PointSet all{g->XsT.as<double>(), cp, g->sq.as<double>(), n1, np1};
  scale_points(h, all, g->X.as<double>(), d, ell);
  // rows [r0, np1) of K: left of r0 the plain cross-covariance, from r0 the symmetric block (noise, identity padding)
  const PointSet done{all.XsT, cp, all.sq, r0, r0};                          // points of the finished columns
  const PointSet rows{all.XsT + r0, cp, all.sq + r0, n1 - r0, np1 - r0};
  // Thin append: the new points stay inside the partly filled last tile.  The rows already there keep their solved
  // part left of r0; only the m new rows are solved, as m right-hand sides of the forward substitution (one pass
  // over L11, HBM bound) instead of a sweep of a whole 128-row tile (a chain of ~2 t0 small DMMA launches).
  const bool thin = r0 > 0 && n0 > r0 && np1 == r0 + TILE && m <= THIN_MAX;
  if (thin) {
    double* scratch = A + cp * cp;                        // the prediction rows double as scratch
    const PointSet added{all.XsT + n0, cp, all.sq + n0, m, round_up(m, 64)};
    build_cov(h, added, done, d, 2, g->kind, 0, hyp2, scratch, cp);
    launch_trsv_l_multi(A, cp, g->Dinv.as<double>(), r0, scratch, A + n0 * cp, cp, static_cast<int>(m), st);
    h->launches += t0;
  } else if (r0 > 0) {
    build_cov(h, rows, done, d, 2, g->kind, 0, hyp2, A + r0 * cp, cp);
  }
  build_cov(h, rows, rows, d, 1, g->kind, 0, hyp2, A + r0 * cp + r0, cp);
  GPB_CUDA(cudaEventRecord(h->tev[1], st));

  if (r0 > 0) {
    if (!thin) {
      FactorMat v = view(g, r0, np1);                     // new tile rows against the finished columns
      SweepPlan plan;
      plan.factor = false; plan.extra_tile0 = t0; plan.extra_tiles = nt1 - t0;
      chol_sweep(h, v, plan);
    }
    if (thin && t0 >= 8) {
      // one 128 x 128 tile with k = r0: as a single tile it would run on one SM (2 ms at N = 16384); cut k into
      // chunks, one partial tile per chunk from the same kernel (the chunk index rides in the batch coordinate of
      // the tensor map), then subtract the partials in a fixed order
      const int chunks = t0 / SPLIT_Q, rem = t0 - chunks * SPLIT_Q;
      double* P = g->part.as<double>();
      const double* Xrows = A + r0 * cp;
      CUtensorMap mx;
      make_tensor_map(&mx, Xrows, SPLIT_Q * TILE, TILE, chunks, cp, SPLIT_Q * TILE, 64);
      GemmArgs ga{};
      ga.C = P; ga.ldc = TILE; ga.c_batch_stride = TILE * TILE; ga.rows_total = TILE;
      ga.j0 = 0; ga.j1 = 2; ga.R = 2; ga.tri = 0; ga.i0 = 0;
      ga.ka0 = 0; ga.kb0 = 0; ga.nk = SPLIT_Q * TILE / GEMM_KB; ga.a_row0 = 0; ga.b_row0 = 0; ga.epi = 0;
      launch_dmma_gemm(mx, mx, ga, chunks, st, 64);
      if (rem > 0) {
        CUtensorMap mr;
        make_tensor_map(&mr, Xrows + static_cast<int64_t>(chunks) * SPLIT_Q * TILE, rem * TILE, TILE, 1, cp, TILE * cp, 64);
        ga.C = P + static_cast<int64_t>(chunks) * TILE * TILE; ga.nk = rem * TILE / GEMM_KB;
        launch_dmma_gemm(mr, mr, ga, 1, st, 64);
      }
      sub_partials_kernel<<<64, 256, 0, st>>>(A + r0 * cp + r0, cp, P, chunks + (rem > 0 ? 1 : 0));
      GPB_CUDA(cudaGetLastError());
      h->launches += 3;
    } else {
      FactorMat w = view(g, np1, np1);                    // trailing block -= X X^T, k over all finished columns
      chol_trailing_update(h, w, t0, nt1, 0, t0);
    }
  }
  {
    FactorMat f;                                          // the trailing block as a matrix of its own
    f.A = A + r0 * cp + r0; f.ld = cp; f.n_pad = np1 - r0; f.rows_total = np1 - r0; f.batch = 1; f.batch_stride = 0;
    f.Dinv = g->Dinv.as<double>() + r0 * TILE; f.dinv_bs = 0;
    f.diag = g->diag.as<double>() + r0; f.diag_bs = 0;
    f.info = g->info.as<int>();
    make_tile_maps(&f.mapA, f.A, cp - r0, np1 - r0, 1, cp, (np1 - r0) * cp);
    make_tile_maps(&f.mapD, f.Dinv, TILE, np1 - r0, 1, TILE, (np1 - r0) * TILE);
    chol_sweep(h, f, true);
  }
  GPB_CUDA(cudaEventRecord(h->tev[2], st));

  // z = L^-1 (y - m): entries below r0 are final; the rest restart from y2 - L21 z1
  double* r = g->r.as<double>();
  double* z = g->z.as<double>();
  if (np1 > n1) GPB_CUDA(cudaMemsetAsync(g->yc.as<double>() + n1, 0, static_cast<size_t>(np1 - n1) * 8, st));
  if (r0 > 0) {
    launch_row_dot(A + r0 * cp, cp, 0, z, 0, np1 - r0, r0, 0, g->tmp.as<double>(), 0, 1, st);
    sub_vec_kernel<<<static_cast<unsigned>((np1 - r0 + 255) / 256), 256, 0, st>>>(r + r0, g->yc.as<double>() + r0,
                                                                                g->tmp.as<double>(), np1 - r0);
    GPB_CUDA(cudaGetLastError());
    h->launches += 2;
  } else {
    GPB_CUDA(cudaMemcpyAsync(r, g->yc.p, static_cast<size_t>(np1) * 8, cudaMemcpyDeviceToDevice, st));
  }
  launch_trsv_l(A, cp, 0, g->Dinv.as<double>(), 0, np1, r, 0, z, 0, 1, st, t0);
  h->launches += nt1 - t0;
  launch_nlml_finish(z, 0, g->diag.as<double>(), 0, np1, n1, g->out.as<double>(), 1, st);
  ++h->launches;
  GPB_CUDA(cudaEventRecord(h->tev[3], st));
  int fail = read_info(h, g->info.as<int>(), g->out.as<double>(), nlml);
  if (fail > 0) fail += static_cast<int>(r0);            // the trailing factorisation counts from r0
  g->last_info = fail;
  if (info) *info = fail;
  if (fail == 0) g->n = n1;
  for (int i = 0; i < 8; ++i) h->timings[i] = 0.f;
  for (int i = 0; i < 3; ++i) GPB_CUDA(cudaEventElapsedTime(&h->timings[i], h->tev[i], h->tev[i + 1]));
  GPB_CUDA(cudaEventElapsedTime(&h->timings[4], h->tev[0], h->tev[3]));
  GPB_API_END
}

int gpb_gpr_grow_predict(gpb_handle* h, const double* Z, int64_t mz, double* fz, double* cov) {
  GPB_ENTRY_BEGIN
  GrowState* g = h->grow;
  GPB_REQUIRE(g != nullptr && g->n > 0, "grow_predict: nothing has been appended yet");
  GPB_REQUIRE(g->last_info == 0, "grow_predict: the stored factor is invalid");
  GPB_REQUIRE(Z && fz && cov && mz > 0, "grow_predict: null argument");
  const int d = g->d;
  const int64_t cp = g->cap_pad, n = g->n, np = round_up(n, TILE);
  const double* ell = g->par.as<double>();
  const double* hyp2 = ell + d;
  double* A = g->A.as<double>();
  cudaStream_t st = h->s0;
  h->Zd.ensure(static_cast<size_t>(PRED_ROWS) * d * 8);
  h->ZsT.ensure(static_cast<size_t>(d) * PRED_ROWS * 8);
  h->zsq.ensure(static_cast<size_t>(PRED_ROWS) * 8);
  double* outv = g->out.as<double>() + 8;
  const PointSet train{g->XsT.as<double>(), cp, g->sq.as<double>(), n, np};
  GPB_CUDA(cudaEventRecord(h->tev[0], st));
  for (int64_t z0 = 0; z0 < mz; z0 += PRED_ROWS) {
    const int64_t mc = mz - z0 < PRED_ROWS ? mz - z0 : PRED_ROWS, mp64 = round_up(mc, 64);
    GPB_CUDA(cudaMemcpyAsync(h->Zd.p, Z + z0 * d, static_cast<size_t>(mc) * d * 8, cudaMemcpyHostToDevice, st));
    const PointSet z{h->ZsT.as<double>(), mp64, h->zsq.as<double>(), mc, mp64};
    scale_points(h, z, h->Zd.as<double>(), d, ell);
    build_cov(h, z, train, d, 2, g->kind, 0, hyp2, A + cp * cp, cp);       // Kzx rows (GPr.py:46,49) under the factor
    FactorMat v = view(g, np, cp + mp64);
    SweepPlan plan;
    plan.factor = false; plan.extra_tile0 = static_cast<int>(cp / TILE); plan.extra_tiles = static_cast<int>((mp64 + TILE - 1) / TILE);
    chol_sweep(h, v, plan);                               // V = Kzx L^-T
    launch_predict_finish(A + cp * cp, cp, g->z.as<double>(), np, mc, hyp2, outv, outv + mc, st);
    ++h->launches;
    GPB_CUDA(cudaMemcpyAsync(fz + z0, outv, static_cast<size_t>(mc) * 8, cudaMemcpyDeviceToHost, st));
    GPB_CUDA(cudaMemcpyAsync(cov + z0, outv + mc, static_cast<size_t>(mc) * 8, cudaMemcpyDeviceToHost, st));
  }
  GPB_CUDA(cudaEventRecord(h->tev[1], st));
  GPB_CUDA(cudaStreamSynchronize(st));
  for (int i = 0; i < 8; ++i) h->timings[i] = 0.f;
  GPB_CUDA(cudaEventElapsedTime(&h->timings[4], h->tev[0], h->tev[1]));
  GPB_API_END
}

}  // extern "C"
