// batched.cu - B independent evaluations of the regression likelihood on the same (X, y).
//
// This is the shape of GP_parameter_fit.py:32-33: optimize() + optimize_restarts(10) evaluate
// the marginal likelihood of one data set for many hyper-parameter vectors, one after the other.
// Here a chunk of problems is resident at once; every kernel of the sweep carries the problem
// index in blockIdx.y, so the panel kernels (one CTA per problem) fill the machine too.
#include "../../include/gpb200.h"
#include "gpb_context.cuh"

using namespace gpb;

namespace gpb {
int gpr_nlml_grad_chunk(gpb_handle* h, const double* khyp, int64_t B, double mean, double* nlml,
                        double* grad, int32_t* info);   // grad.cu
}


extern "C" int gpb_gpr_nlml_batched(gpb_handle* h, const double* khyp, int64_t B, double mean, double* nlml,
                                    double* grad, int32_t* info) {
  GPB_API_BEGIN
  GPB_REQUIRE(h->n > 0 && h->has_y, "no training data: call gpb_set_train first");
  GPB_REQUIRE(khyp && nlml && B > 0, "null argument");
  if (grad) return gpr_nlml_grad_chunk(h, khyp, B, mean, nlml, grad, info);

  const int64_t np = h->n_pad;
  const int d = h->d;
  // problems resident at once: bounded by memory (A + Dinv per problem) and by option
  // (round 1: 296 = two waves of the 46 us diagonal-tile kernel; with the 26 us kernel fewer, longer chunks win:
  // 296 / 512 / 1024 problems 116.0 / 115.3 / 111.0 ms incl. 4-tile blocks, profiles/r02_ab_sweep.txt)
  const size_t per_problem = static_cast<size_t>(np) * np * 8 + static_cast<size_t>(np) * TILE * 8 +
                             static_cast<size_t>(d + 2) * np * 8;
  const int64_t chunk = plan_chunk(h, B, 1024, static_cast<size_t>(np) * np * 8, per_problem, h->A.bytes + h->Dinv.bytes);

  h->scal.ensure(static_cast<size_t>(chunk) * 8 < 64 ? 64 : static_cast<size_t>(chunk) * 8);
  GPB_CUDA(cudaEventRecord(h->tev[0], h->s0));
  for (int64_t b0 = 0; b0 < B; b0 += chunk) {
    const int bc = static_cast<int>(B - b0 < chunk ? B - b0 : chunk);
    const KernelParams pr = upload_params(h, h->params, khyp + b0 * (d + 2), d, bc);
    FactorMat m = factor_workspace(h, bc, np, np, np, np, true);     // no appended row: see launch_trsv_l below
    const PointSet x = train_points(h, bc);
    scale_points(h, x, h->X.as<double>(), d, pr.ell, bc);
    build_cov(h, x, x, d, 1, h->cov_kind, 0, pr.hyp2, m.A, np, m.batch_stride, bc);
    // right-hand sides: r = y - mean per problem (scratch), z = L^-1 r
    const bool fuse = h->fuse_rhs && tile_potrf_fuses_rhs();
    h->aux0.ensure(static_cast<size_t>(chunk) * np * 8 * (fuse ? 9 : 2));
    double* rv = h->aux0.as<double>();
    double* zv = rv + static_cast<size_t>(chunk) * np * (fuse ? 8 : 1);
    ++h->launches;
    if (fuse) {
      // z = L^-1 r rides on the factorisation: tile k of it is solved by the diagonal-tile kernel, and the panel TRSM
      // takes its columns out of the rows below while it still holds them (8 partial vectors per problem, DESIGN 4.6)
      GPB_CUDA(cudaMemsetAsync(rv, 0, static_cast<size_t>(bc) * np * 8 * 8, h->s0));
      launch_set_y_rows(rv, 8 * np, 0, h->y.as<double>(), h->n, np, mean, bc, h->s0);      // partial 0 <- y - mean
      m.rhs_r = rv; m.rhs_bs = 8 * np; m.rhs_gs = np; m.rhs_z = zv; m.rhs_zbs = np;
      chol_sweep(h, m, true);
    } else {
      launch_set_y_rows(rv, np, 0, h->y.as<double>(), h->n, np, mean, bc, h->s0);
      chol_sweep(h, m, true);
      launch_trsv_l(m.A, m.ld, m.batch_stride, m.Dinv, m.dinv_bs, np, rv, np, zv, np, bc, h->s0);
      h->launches += static_cast<int>(np / TILE);
    }
    launch_nlml_finish(zv, np, m.diag, m.diag_bs, np, h->n, h->scal.as<double>(), bc, h->s0);
    ++h->launches;
    double* hres = h->pinned(static_cast<size_t>(bc) * 8 + static_cast<size_t>(bc) * 4);
    int* hinfo = reinterpret_cast<int*>(hres + bc);
    GPB_CUDA(cudaMemcpyAsync(hres, h->scal.p, static_cast<size_t>(bc) * 8, cudaMemcpyDeviceToHost, h->s0));
    GPB_CUDA(cudaMemcpyAsync(hinfo, m.info, static_cast<size_t>(bc) * 4, cudaMemcpyDeviceToHost, h->s0));
    GPB_CUDA(cudaStreamSynchronize(h->s0));
    for (int b = 0; b < bc; ++b) {
      nlml[b0 + b] = hres[b];
      if (info) info[b0 + b] = hinfo[b];
    }
  }
  GPB_CUDA(cudaEventRecord(h->tev[1], h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  for (float& t : h->timings) t = 0.f;
  GPB_CUDA(cudaEventElapsedTime(&h->timings[4], h->tev[0], h->tev[1]));
  GPB_API_END
}
