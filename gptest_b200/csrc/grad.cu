// grad.cu - value and hyper-parameter gradient of the regression likelihood.
//
//   d nlml / d theta_k = 0.5 * tr((K^-1 - alpha alpha^T) dK/dtheta_k),  theta = log hyper-parameters
//
// The reference never forms gradients (Nelder-Mead, GP_regression_demo.py:44); this is what the
// L-BFGS multi-start of GP_parameter_fit.py:32-33 obtains from GPy (dpotrf + dpotri + kernel
// gradients).  Device plan, all on the DMMA tile kernel:
//   1. factor K with the y row appended              (N^3/3 flop)   -> L, z = L^-1 y, nlml
//   2. sweep an identity block through L             (N^3/3 flop)   -> U = L^-T (upper triangular);
//      tile row q of the identity stays zero left of tile column q and is skipped until then
//   3. K^-1 = U U^T on the lower tiles, k range starting at the tile row (N^3/3 flop)
//   4. alpha = U z (row dot products), then ONE fused pass over the lower triangle that
//      recomputes exp(-r^2/2) and the per-dimension distances from the scaled points and
//      accumulates the D+2 traces - dK/dtheta is never materialised.
// Reductions are fixed-order (per-CTA partials, then one CTA): results are run-to-run identical.
// The same trace pass serves the gradient of the preference Laplace evidence (laplace.cu,
// gpb_pref_evidence_grad): there the dense matrix is A = (K + W^-1)^-1, the rank-one term becomes the
// rank-two alpha b^T + b alpha^T, distances are clipped at 0 (GPy RBF) and there is no noise column.
#include <type_traits>

#include "../../include/gpb200.h"
#include "gpb_context.cuh"
#include "gpb_exp.cuh"

namespace gpb {

namespace {

constexpr int GT = 64;       // tile edge of the trace kernel
constexpr int GDC = 8;       // dimensions per staged chunk

__global__ void set_identity_kernel(double* U, int64_t ld, int64_t n, int64_t batch_stride) {
  double* u = U + blockIdx.y * batch_stride;
  const int64_t total = n * ld;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / ld, c = i - r * ld;
    u[i] = (r == c) ? 1.0 : 0.0;
  }
}

// out[i] = sum_{c >= c_lo(i)} M[i][c] * x[c]; one CTA per row, fixed-order tree
__global__ void __launch_bounds__(256) row_dot_kernel(const double* __restrict__ M, int64_t ld, int64_t m_bs,
                                                      const double* __restrict__ x, int64_t x_bs, int64_t ncols,
                                                      int upper, double* __restrict__ out, int64_t out_bs) {
  __shared__ double sh[256];
  const int64_t i = blockIdx.x;
  const int b = blockIdx.y;
  const double* row = M + b * m_bs + i * ld;
  const double* xv = x + b * x_bs;
  const int64_t c0 = upper ? (i & ~int64_t(1)) : 0;
  double s = 0.0;
  for (int64_t c = c0 + 2 * threadIdx.x; c < ncols; c += 512) {
    const double2 v = *reinterpret_cast<const double2*>(row + c);
    const double2 xx = *reinterpret_cast<const double2*>(xv + c);
    s = fma(v.x, xx.x, s);
    s = fma(v.y, xx.y, s);
  }
  sh[threadIdx.x] = s;
  __syncthreads();
#pragma unroll
  for (int k = 128; k > 0; k >>= 1) {
    if (threadIdx.x < k) sh[threadIdx.x] += sh[threadIdx.x + k];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[b * out_bs + i] = sh[0];
}

struct TraceArgs {
  const double* Kinv; int64_t ld, k_bs;     // lower 64-tiles valid (diagonal tiles full)
  const double* alpha; int64_t a_bs;
  const double* XsT; int64_t x_ld, xs_bs;
  const double* sq; int64_t sq_bs;
  const double* hyp2;                       // per batch [sf2, sn2]
  int64_t n;                                // valid points
  int d;
  double* partial;                          // [batch][ntiles][d+2]
  int64_t ntiles;
  int kind;                                 // radial function (gpb_exp.cuh)
};
// The preference Laplace evidence: Kinv holds A and beta is b.  A type of its own rather than one more member of
// TraceArgs: a larger parameter block alone changes the register allocation of the regression kernels.
struct LaplaceTraceArgs : TraceArgs {
  const double* beta;
};

// TraceArgs:        Q = K^-1 - alpha alpha^T, partials [d length-scales, sf, sn] (regression).
// LaplaceTraceArgs: Q = A - (alpha b^T + b alpha^T), r^2 clipped at 0 as in the assembly (clip = 1), partials
//                   [d length-scales, sf] - the jitter of the Laplace paths is not a hyper-parameter.
template <int KIND, class ARGS = TraceArgs>
__global__ void __launch_bounds__(256) grad_trace_kernel(const ARGS p) {
  constexpr bool LAPLACE = std::is_same_v<ARGS, LaplaceTraceArgs>;
  __shared__ double xr[GDC][GT];
  __shared__ double xc[GDC][GT];
  __shared__ double red[256];
  __shared__ double etab[64];
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int b = blockIdx.y;
  exp_table_to_smem(etab);                       // visible after the barriers of the staging loop
  int64_t ti = static_cast<int64_t>((sqrt(8.0 * blockIdx.x + 1.0) - 1.0) * 0.5);
  while ((ti + 1) * (ti + 2) / 2 <= blockIdx.x) ++ti;
  while (ti * (ti + 1) / 2 > blockIdx.x) --ti;
  const int64_t tj = blockIdx.x - ti * (ti + 1) / 2;
  const int64_t i0 = ti * GT, j0 = tj * GT;
  const double* XsT = p.XsT + b * p.xs_bs;
  const double wgt = (ti == tj) ? 1.0 : 2.0;
  const double sf2 = p.hyp2[2 * b], sn2 = p.hyp2[2 * b + 1];

  // pass 1: expanded-form distance exactly as the assembly kernel computes it
  double dot[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int c = 0; c < 4; ++c) dot[a][c] = 0.0;
  for (int d0 = 0; d0 < p.d; d0 += GDC) {
    const int dc = min(GDC, p.d - d0);
    __syncthreads();
    for (int e = t; e < dc * GT; e += 256) {
      const int k = e / GT, i = e % GT;
      xr[k][i] = XsT[(d0 + k) * p.x_ld + i0 + i];
      xc[k][i] = XsT[(d0 + k) * p.x_ld + j0 + i];
    }
    __syncthreads();
    for (int k = 0; k < dc; ++k)
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) dot[a][c] = fma(xr[k][ty + 16 * a], xc[k][tx + 16 * c], dot[a][c]);
  }
  const double* sq = p.sq + b * p.sq_bs;
  const double* al = p.alpha + b * p.a_bs;
  const double* Kinv = p.Kinv + b * p.k_bs;
  double q[4][4];            // weight * (Kinv - alpha alpha^T) * Kse
  double acc_sf = 0.0, acc_sn = 0.0;
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int64_t r = i0 + ty + 16 * a;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int64_t cc = j0 + tx + 16 * c;
      double v = 0.0;
      if (r < p.n && cc < p.n) {
        double r2 = (sq[r] + sq[cc]) - 2.0 * dot[a][c];
        if constexpr (LAPLACE) r2 = fmax(r2, 0.0);
        double kr, gr;
        radial_and_dl<KIND>(-0.5 * r2, etab, kr, gr);         // same exp as the assembly kernel
        if constexpr (LAPLACE) {
          const double Q = wgt * sf2 * (Kinv[r * p.ld + cc] - fma(al[r], p.beta[cc], p.beta[r] * al[cc]));
          v = Q * gr;
          acc_sf += Q * kr;
        } else {
          const double Q = wgt * sf2 * (Kinv[r * p.ld + cc] - al[r] * al[cc]);
          v = Q * gr;                                         // length-scale derivative weight (SE: gr == kr)
          acc_sf += Q * kr;
          if (r == cc) acc_sn += Kinv[r * p.ld + cc] - al[r] * al[cc];
        }
      }
      q[a][c] = v;
    }
  }
  double* out = p.partial + (static_cast<int64_t>(b) * p.ntiles + blockIdx.x) * (LAPLACE ? p.d + 1 : p.d + 2);

  // pass 2: per-dimension squared differences, one staged chunk at a time
  for (int d0 = 0; d0 < p.d; d0 += GDC) {
    const int dc = min(GDC, p.d - d0);
    __syncthreads();
    for (int e = t; e < dc * GT; e += 256) {
      const int k = e / GT, i = e % GT;
      xr[k][i] = XsT[(d0 + k) * p.x_ld + i0 + i];
      xc[k][i] = XsT[(d0 + k) * p.x_ld + j0 + i];
    }
    __syncthreads();
    for (int k = 0; k < dc; ++k) {
      double s = 0.0;
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const double df = xr[k][ty + 16 * a] - xc[k][tx + 16 * c];
          s = fma(q[a][c], df * df, s);
        }
      red[t] = s;
      __syncthreads();
      for (int w = 128; w > 0; w >>= 1) {
        if (t < w) red[t] += red[t + w];
        __syncthreads();
      }
      if (t == 0) out[d0 + k] = red[0];          // sum Q * Kse * (xs_r - xs_c)^2
      __syncthreads();
    }
  }
  red[t] = acc_sf;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) red[t] += red[t + w];
    __syncthreads();
  }
  if (t == 0) out[p.d] = 2.0 * red[0];            // dK/dlog sf = 2 Kse
  if constexpr (LAPLACE) return;
  __syncthreads();
  red[t] = acc_sn;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) red[t] += red[t + w];
    __syncthreads();
  }
  if (t == 0) out[p.d + 1] = 2.0 * sn2 * red[0];  // dK/dlog sn = 2 sn2 I
}

// grad[b][k] = 0.5 * sum_tiles partial[b][tile][k]   (fixed order)
__global__ void __launch_bounds__(256) grad_reduce_kernel(const double* __restrict__ partial, int64_t ntiles,
                                                          int np, double* __restrict__ grad) {
  __shared__ double red[256];
  const int b = blockIdx.y, k = blockIdx.x;
  const double* src = partial + static_cast<int64_t>(b) * ntiles * np + k;
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < ntiles; i += 256) s += src[i * np];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) grad[b * np + k] = 0.5 * red[0];
}

}  // namespace

void launch_laplace_grad_trace(const double* A, int64_t ld, const double* alpha, const double* beta, const double* XsT,
                               int64_t x_ld, const double* sq, const double* hyp2, int64_t n, int d, double* partial,
                               double* out, cudaStream_t st) {
  const int64_t t64 = ld / GT;
  LaplaceTraceArgs t{};
  t.Kinv = A; t.ld = ld;
  t.alpha = alpha; t.beta = beta;
  t.XsT = XsT; t.x_ld = x_ld; t.sq = sq;
  t.hyp2 = hyp2; t.n = n; t.d = d;
  t.partial = partial; t.ntiles = t64 * (t64 + 1) / 2;
  grad_trace_kernel<0, LaplaceTraceArgs><<<static_cast<unsigned>(t.ntiles), 256, 0, st>>>(t);
  GPB_CUDA(cudaGetLastError());
  grad_reduce_kernel<<<d + 1, 256, 0, st>>>(partial, t.ntiles, d + 1, out);
  GPB_CUDA(cudaGetLastError());
}

// K^-1 into the lower tiles of the symmetric part (overwriting L), given the factor in `m`.
// Layout per batch entry: rows [0,np) L | rows [np, np+128) first appended tile row |
// rows [np+128, 2np+128) identity block -> U.  `m.rows_total` must cover all of them.
void chol_inverse_lower(gpb_handle* h, FactorMat& m) {
  const int64_t np = m.n_pad;
  const int nt = static_cast<int>(np / TILE);
  double* U = m.A + (np + TILE) * m.ld;
  {
    dim3 grid(148 * 8, m.batch);
    set_identity_kernel<<<grid, 256, 0, h->s0>>>(U, m.ld, np, m.batch_stride);
    GPB_CUDA(cudaGetLastError());
    ++h->launches;
  }
  SweepPlan plan;
  plan.factor = false;
  plan.extra_tile0 = nt + 1;
  plan.extra_tiles = nt;
  plan.grow = true;
  chol_sweep(h, m, plan);
  GemmArgs a{};
  a.C = m.A; a.ldc = m.ld; a.c_batch_stride = m.batch_stride; a.rows_total = static_cast<int>(np);
  a.j0 = 0; a.j1 = nt; a.R = nt; a.tri = 1; a.i_off = 0;
  a.a_row0 = a.b_row0 = static_cast<int>(np + TILE);
  a.k_from_row = 1; a.k_end = static_cast<int>(np); a.epi = 0;
  dense_gemm(h, m.mapA, m.mapA, a, m.batch);
  ++h->launches;
}

void launch_row_dot(const double* M, int64_t ld, int64_t m_bs, const double* x, int64_t x_bs, int64_t nrows,
                    int64_t ncols, int upper, double* out, int64_t out_bs, int batch, cudaStream_t st) {
  dim3 grid(static_cast<unsigned>(nrows), batch);
  row_dot_kernel<<<grid, 256, 0, st>>>(M, ld, m_bs, x, x_bs, ncols, upper, out, out_bs);
  GPB_CUDA(cudaGetLastError());
}

int gpr_nlml_grad_chunk(gpb_handle* h, const double* khyp, int64_t B, double mean, double* nlml, double* grad,
                        int32_t* info) {
  const int64_t np = h->n_pad;
  const int d = h->d;
  const int P = d + 2;
  const int nt = static_cast<int>(np / TILE);
  const int64_t rows_alloc = 2 * np + TILE;
  const int64_t t64 = np / GT;
  const int64_t ntiles = t64 * (t64 + 1) / 2;
  const size_t per_problem = static_cast<size_t>(rows_alloc) * np * 8 + static_cast<size_t>(np) * TILE * 8 +
                             static_cast<size_t>(d + 4) * np * 8 + static_cast<size_t>(ntiles) * P * 8;
  const int64_t chunk = plan_chunk(h, B, 64, static_cast<size_t>(rows_alloc) * np * 8, per_problem,
                                   h->A.bytes + h->Dinv.bytes + h->aux0.bytes);

  GPB_CUDA(cudaEventRecord(h->tev[0], h->s0));
  for (int64_t b0 = 0; b0 < B; b0 += chunk) {
    const int bc = static_cast<int>(B - b0 < chunk ? B - b0 : chunk);
    const KernelParams pr = upload_params(h, h->params, khyp + b0 * P, d, bc);
    // one tensor map over all rows of the buffer serves both sweeps and the U U^T product
    FactorMat m = factor_workspace(h, bc, np, rows_alloc, np + 1, rows_alloc, true);
    const PointSet x = train_points(h, bc);
    h->scal.ensure(static_cast<size_t>(chunk) * (P + 1) * 8 + 64);
    h->aux0.ensure(static_cast<size_t>(chunk) * np * 8);                       // alpha
    h->aux1.ensure(static_cast<size_t>(chunk) * ntiles * P * 8);               // trace partials
    scale_points(h, x, h->X.as<double>(), d, pr.ell, bc);
    build_cov(h, x, x, d, 1, h->cov_kind, 0, pr.hyp2, m.A, np, m.batch_stride, bc);
    launch_set_y_rows(m.A, m.batch_stride, np * np, h->y.as<double>(), h->n, np, mean, bc, h->s0);
    ++h->launches;
    if (b0 == 0) GPB_CUDA(cudaEventRecord(h->tev[1], h->s0));
    chol_sweep(h, m, true);
    double* res = h->scal.as<double>();
    launch_nlml_finish(m.A + np * np, m.batch_stride, m.diag, m.diag_bs, np, h->n, res, bc, h->s0);
    ++h->launches;
    if (b0 == 0) GPB_CUDA(cudaEventRecord(h->tev[2], h->s0));

    m.rows_total = rows_alloc;
    chol_inverse_lower(h, m);
    // alpha = L^-T z = U z
    launch_row_dot(m.A + (np + TILE) * np, np, m.batch_stride, m.A + np * np, m.batch_stride, np, np, 1,
                   h->aux0.as<double>(), np, bc, h->s0);
    TraceArgs t{};
    t.Kinv = m.A; t.ld = np; t.k_bs = m.batch_stride;
    t.alpha = h->aux0.as<double>(); t.a_bs = np;
    t.XsT = h->XsT.as<double>(); t.x_ld = np; t.xs_bs = static_cast<int64_t>(d) * np;
    t.sq = h->sq.as<double>(); t.sq_bs = np;
    t.hyp2 = pr.hyp2; t.n = h->n; t.d = d;
    t.partial = h->aux1.as<double>(); t.ntiles = ntiles;
    {
      dim3 grid(static_cast<unsigned>(ntiles), bc);
      t.kind = h->cov_kind;
      if (t.kind == 1) grad_trace_kernel<1><<<grid, 256, 0, h->s0>>>(t);
      else if (t.kind == 2) grad_trace_kernel<2><<<grid, 256, 0, h->s0>>>(t);
      else grad_trace_kernel<0><<<grid, 256, 0, h->s0>>>(t);
      GPB_CUDA(cudaGetLastError());
      dim3 g2(P, bc);
      grad_reduce_kernel<<<g2, 256, 0, h->s0>>>(h->aux1.as<double>(), ntiles, P, res + bc);
      GPB_CUDA(cudaGetLastError());
    }
    h->launches += 3;
    if (b0 == 0) GPB_CUDA(cudaEventRecord(h->tev[3], h->s0));

    double* hres = h->pinned(static_cast<size_t>(bc) * (P + 1) * 8 + static_cast<size_t>(bc) * 4);
    int* hinfo = reinterpret_cast<int*>(hres + static_cast<size_t>(bc) * (P + 1));
    GPB_CUDA(cudaMemcpyAsync(hres, res, static_cast<size_t>(bc) * (P + 1) * 8, cudaMemcpyDeviceToHost, h->s0));
    GPB_CUDA(cudaMemcpyAsync(hinfo, m.info, static_cast<size_t>(bc) * 4, cudaMemcpyDeviceToHost, h->s0));
    GPB_CUDA(cudaStreamSynchronize(h->s0));
    for (int b = 0; b < bc; ++b) {
      nlml[b0 + b] = hres[b];
      for (int k = 0; k < P; ++k) grad[(b0 + b) * P + k] = hres[bc + b * P + k];
      if (info) info[b0 + b] = hinfo[b];
    }
    if (b0 == 0) {
      for (float& x : h->timings) x = 0.f;
      GPB_CUDA(cudaEventElapsedTime(&h->timings[0], h->tev[0], h->tev[1]));
      GPB_CUDA(cudaEventElapsedTime(&h->timings[1], h->tev[1], h->tev[2]));
      GPB_CUDA(cudaEventElapsedTime(&h->timings[3], h->tev[2], h->tev[3]));
    }
  }
  GPB_CUDA(cudaEventRecord(h->tev[4], h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  GPB_CUDA(cudaEventElapsedTime(&h->timings[4], h->tev[0], h->tev[4]));
  return 0;
}

}  // namespace gpb
