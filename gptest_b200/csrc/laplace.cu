// laplace.cu - Laplace / Newton mode finding on the device.
//
//  * preference GP (PreferenceGaussianProcess.calc_laplace, GPpref.py:112-157, PrefProbit
//    GPpref.py:46-94) including the reference's quirks (see gpb200.h);
//  * binary classification (GPc.py intent; Rasmussen & Williams Alg. 3.1 / 3.2).
//
// Per Newton iteration the reference inverts a dense n x n matrix on the host
// (np.linalg.inv, GPpref.py:143) and builds W with a Python loop over the pairs
// (GPpref.py:82-87).  Here one iteration is: a fused per-pair kernel (z, Phi, N, gradient and
// Hessian weights), a per-item kernel that assembles G = K^-1 + W and the right-hand side from a
// CSR view of the comparison graph (deterministic, same per-cell summation order as the
// reference's loop), the blocked DMMA Cholesky of G with the right-hand side riding along as an
// appended row, a blocked backward substitution, and one reduction kernel for the objective and
// max|f_new - f|.  The host only reads back 16 bytes per iteration to decide on convergence.
#include <algorithm>
#include <cmath>
#include <vector>

#include "../../include/gpb200.h"
#include <chrono>
#include <cstdlib>

#include "gpb_context.cuh"

using namespace gpb;

namespace {

constexpr double LOG_2PI = 1.8378770664093453;
constexpr double INV_SQRT_2PI = 0.3989422804014327;
constexpr double SQRT_2_OVER_PI = 0.7978845608028654;
constexpr double INV_SQRT_2 = 0.7071067811865476;

// ---------------------------------------------------------------------------------------
// generic helpers
// ---------------------------------------------------------------------------------------
template <int NT>
__device__ __forceinline__ double cta_sum(double v, double* sh) {
  sh[threadIdx.x] = v;
  __syncthreads();
#pragma unroll
  for (int w = NT / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  const double r = sh[0];
  __syncthreads();
  return r;
}
template <int NT>
__device__ __forceinline__ double cta_max(double v, double* sh) {
  sh[threadIdx.x] = v;
  __syncthreads();
#pragma unroll
  for (int w = NT / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w) sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + w]);
    __syncthreads();
  }
  const double r = sh[0];
  __syncthreads();
  return r;
}

__global__ void __launch_bounds__(512) sum_log_kernel(const double* __restrict__ v, int64_t n, double* __restrict__ out) {
  __shared__ double sh[512];
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += 512) s += log(v[i]);
  const double r = cta_sum<512>(s, sh);
  if (threadIdx.x == 0) out[0] = r;
}

// full symmetric copy of a matrix whose lower 64-tiles (and full diagonal tiles) are valid
__global__ void __launch_bounds__(256) mirror_lower_kernel(const double* __restrict__ src, int64_t ld_s,
                                                           double* __restrict__ dst, int64_t ld_d, int64_t nt64) {
  __shared__ double tt[64][65];
  const int64_t ti = blockIdx.x / nt64, tj = blockIdx.x % nt64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  if (ti >= tj) {
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int64_t r = ti * 64 + ty + 16 * a, cc = tj * 64 + tx + 16 * c;
        dst[r * ld_d + cc] = src[r * ld_s + cc];
      }
  } else {
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c)
        tt[ty + 16 * a][tx + 16 * c] = src[(tj * 64 + ty + 16 * a) * ld_s + ti * 64 + tx + 16 * c];
    __syncthreads();
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c)
        dst[(ti * 64 + ty + 16 * a) * ld_d + tj * 64 + tx + 16 * c] = tt[tx + 16 * c][ty + 16 * a];
  }
}

// lower triangle (row by row) of dst <- rs[r] * src * rs[c] + (r == c ? dadd : 0); rs == nullptr: plain copy
__global__ void __launch_bounds__(256) scale_copy_lower_kernel(const double* __restrict__ src, int64_t ld_s,
                                                               double* __restrict__ dst, int64_t ld_d,
                                                               const double* __restrict__ rs, double dadd) {
  const int64_t r = blockIdx.x;
  const double sr = rs ? rs[r] : 1.0;
  for (int64_t c = threadIdx.x; c <= r; c += 256) {
    double v = src[r * ld_s + c];
    if (rs) v = sr * v * rs[c];
    if (c == r) v += dadd;
    dst[r * ld_d + c] = v;
  }
}

// One step of the blocked backward substitution  L^T x = r  with the inverted diagonal tiles:
//   x_k = W_k^T r_k ;  r_c -= sum_{rows of tile k} L[row][c] x_k[row]   for every column c left of tile k.
__global__ void __launch_bounds__(256) trsv_lt_step_kernel(const double* __restrict__ L, int64_t ld,
                                                           const double* __restrict__ Dinv, int k,
                                                           double* __restrict__ r, double* __restrict__ x) {
  // written for memory-level parallelism: every load below is independent of the running sums
  __shared__ double rk[TILE];
  __shared__ double xk[TILE];
  __shared__ double part[256];
  const int t = threadIdx.x;
  pdl_trigger();
  pdl_wait();                                    // r comes from the previous step
  if (t < TILE) rk[t] = r[k * TILE + t];
  __syncthreads();
  {
    // x_k = W_k^T r_k on all 256 threads: column c, row half h (rows above the diagonal of W hold zeros)
    const int c = t & 127, h = t >> 7;
    const double* W = Dinv + static_cast<int64_t>(k) * TILE * TILE + c;
    double acc[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) acc[u] = 0.0;
#pragma unroll
    for (int i = 0; i < 64; i += 8) {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int row = 64 * h + i + u;
        acc[u] = fma(W[row * TILE], rk[row], acc[u]);
      }
    }
    part[t] = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
  }
  __syncthreads();
  if (t < TILE) {
    const double s = part[t] + part[t + 128];
    xk[t] = s;
    if (blockIdx.x == 0) x[k * TILE + t] = s;
  }
  __syncthreads();
  // r_c -= L[tile k rows][c] . x_k for 64 columns per CTA, the 128 rows cut into 4 quarters
  const int cl = t & 63, q = t >> 6;
  const int64_t c = static_cast<int64_t>(blockIdx.x) * 64 + cl;
  const bool on = c < static_cast<int64_t>(k) * TILE;
  double s = 0.0;
  if (on) {
    const double* Lk = L + (static_cast<int64_t>(k) * TILE + 32 * q) * ld + c;
    double a[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
#pragma unroll
      for (int u = 0; u < 4; ++u) a[u] = fma(Lk[(i + u) * ld], xk[32 * q + i + u], a[u]);
    }
    s = (a[0] + a[1]) + (a[2] + a[3]);
  }
  part[t] = s;
  __syncthreads();
  if (q == 0 && on) r[c] -= (part[cl] + part[cl + 64]) + (part[cl + 128] + part[cl + 192]);
}

void trsv_lt(gpb_handle* h, const FactorMat& m, double* r, double* x) {
  const int nt = static_cast<int>(m.n_pad / TILE);
  for (int k = nt - 1; k >= 0; --k) {
    const int blocks = k == 0 ? 1 : 2 * k;
    launch_chain(trsv_lt_step_kernel, dim3(blocks), dim3(256), 0, h->s0, g_pdl != 0, m.A, m.ld, m.Dinv, k, r, x);
    ++h->launches;
  }
}

// The Laplace work space in h->A, pitch np: rows [0, np) the factor | the appended tile row | S1 (np rows) |
// S2 (np rows).  S1 is where chol_inverse_lower (grad.cu) keeps U.
struct LapMat : FactorMat {
  double* row;       // appended tile row (right-hand side riding on the factorisation)
  double* S1;
  double* S2;
  int t1, t2;        // tile-row index of S1 and S2
};
LapMat laplace_mat(gpb_handle* h, int64_t rows_total) {
  const int64_t np = h->n_pad;
  const int64_t rows_alloc = 3 * np + TILE;
  LapMat m;
  static_cast<FactorMat&>(m) = factor_workspace(h, 1, np, rows_alloc, rows_total, rows_alloc, false);
  m.t1 = static_cast<int>(np / TILE) + 1;
  m.t2 = 2 * m.t1 - 1;
  m.row = m.A + np * m.ld;
  m.S1 = m.A + m.t1 * TILE * m.ld;
  m.S2 = m.A + m.t2 * TILE * m.ld;
  return m;
}

// rows [t0 * 128, t0 * 128 + rows) <- themselves times L^-T; the factor in rows [0, np) stays
void sweep_rows(gpb_handle* h, FactorMat& m, int t0, int64_t rows) {
  SweepPlan plan;
  plan.factor = false;
  plan.extra_tile0 = t0;
  plan.extra_tiles = static_cast<int>((rows + TILE - 1) / TILE);
  m.rows_total = t0 * TILE + rows;
  chol_sweep(h, m, plan);
}

// The np-vectors of the Laplace paths in h->aux0, in this order in memory.  Preference: f | f_new | t (K^-1 f_new in
// the loop, alpha = K^-1 f_hat in the predict) | spare.  Classification: f | f_new | b | sW | t | a | y | g.
struct LapVecs {
  double *f, *f_new, *t;
  double *b, *sW, *a, *y, *g;        // classification only
};
constexpr int PREF_VECS = 4, GPC_VECS = 8;
LapVecs lap_vecs(gpb_handle* h, LaplaceState::Kind kind) {
  double* f = h->aux0.as<double>();
  const int64_t np = h->n_pad;
  if (kind == LaplaceState::PREF) return LapVecs{f, f + np, f + 2 * np, nullptr, nullptr, nullptr, nullptr, nullptr};
  return LapVecs{f, f + np, f + 4 * np, f + 2 * np, f + 3 * np, f + 5 * np, f + 6 * np, f + 7 * np};
}

// The Laplace paths keep the squared exponential whatever cov_kind the handle holds, with r^2 clipped at 0 as GPy's RBF
// does (GPpref.py:122): K (+ jitter on the diagonal) of the training points, lower tiles into dst (mode 1) or full
// (mode 0), and rows k(z_i, X) of test points (mode 2).
constexpr int LAP_KIND = 0, LAP_CLIP = 1;

// The kernel parameters of a Laplace fit on the device: [ell..., variance, jitter]
KernelParams lap_params(gpb_handle* h, const double* khyp, double jitter) {
  return upload_params(h, h->params, khyp, h->d, 1, jitter);
}

// K + eps I for eps = 1e-6, 1e-5, ... until it factors (GPpref.py:123-134).  `build(pr)` writes the lower tiles of
// K + eps I into rows [0, np) of m; on return they hold its factor.  Returns eps.
template <class F>
double factor_with_jitter(gpb_handle* h, FactorMat& m, const double* khyp, int32_t* info, F&& build) {
  double eps = 1e-6;
  for (;;) {
    build(lap_params(h, khyp, eps));
    GPB_CUDA(cudaMemsetAsync(m.info, 0, 4, h->s0));
    m.rows_total = m.n_pad;
    chol_sweep(h, m, true);
    if (read_info(h, m.info) == 0) return eps;
    eps *= 10.0;
    if (!(eps < 1e8)) { if (info) *info = 1; throw Error{"K + eps*I is not positive definite for any jitter"}; }
  }
}

// Rows k(z_i, X) of the mc test points Z (host, mc x d) into dst (pitch ld, n_pad columns) against the training points
// as the fit scaled them.  zd (mc x d), zsT (d x round_up(mc, 64)) and zsq take the points, scaled.
void test_cov_rows(gpb_handle* h, const double* Z, int64_t mc, const KernelParams& pr, double* zd, double* zsT,
                   double* zsq, double* dst, int64_t ld) {
  const int64_t mp64 = round_up(mc, 64);
  GPB_CUDA(cudaMemcpyAsync(zd, Z, static_cast<size_t>(mc) * h->d * 8, cudaMemcpyHostToDevice, h->s0));
  const PointSet z{zsT, mp64, zsq, mc, mp64};
  scale_points(h, z, zd, h->d, pr.ell);
  build_cov(h, z, train_points(h), h->d, 2, LAP_KIND, LAP_CLIP, pr.hyp2, dst, ld);
}

// ---------------------------------------------------------------------------------------
// preference likelihood (PrefProbit, GPpref.py:46-94)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ double pref_hazard(double z) {
  // N(z)/Phi(z) as the reference forms it (GPpref.py:71-72,76); where Phi underflows (z < -37,
  // the reference produces 0/0 = nan) the erfcx form keeps the iteration finite.
  const double phi = normcdf(z);
  if (phi > 1e-300) return exp(-0.5 * z * z) * INV_SQRT_2PI / phi;
  return SQRT_2_OVER_PI / erfcx(-z * INV_SQRT_2);
}

// per pair: d_k = y isqrt2sig N/Phi (GPpref.py:76), w_k = i2var (z N/Phi + (N/Phi)^2) = -inner (GPpref.py:80)
__global__ void pref_pair_kernel(const int64_t* __restrict__ uvi, const double* __restrict__ y, int64_t P,
                                 const double* __restrict__ f, double isqrt2sig, double i2var,
                                 double* __restrict__ dk, double* __restrict__ wk) {
  const int64_t k = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (k >= P) return;
  const int64_t u = uvi[2 * k], v = uvi[2 * k + 1];
  const double z = y[k] * (isqrt2sig * (f[v] - f[u]));       // GPpref.py:56-58
  const double r = pref_hazard(z);
  dk[k] = y[k] * isqrt2sig * r;
  wk[k] = i2var * (z * r + r * r);
}

// per item i: gradient g_i, row i of G = K^-1 + W (lower part), b_i = (W f)_i + g_i.
// Every cell of W is accumulated in pair order like the reference's loop (GPpref.py:82-87) and only
// then added to K^-1 (GPpref.py:142).
__global__ void pref_row_kernel(int64_t n, const PrefGraphDev gr, const double* __restrict__ dk,
                                const double* __restrict__ wk, const double* __restrict__ f, int grad_mode,
                                double* __restrict__ G, int64_t ld, double* __restrict__ b,
                                double* __restrict__ g_out, double* __restrict__ Wdense) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  double g = 0.0;
  if (grad_mode == 0) {
    if (gr.ku[i] >= 0) g = 0.0 - dk[gr.ku[i]];     // column-0 pass: g[u] = 0 + (-d)
    if (gr.kv[i] >= 0) g = g + dk[gr.kv[i]];       // column-1 pass adds to whatever pass 0 left
  }
  const int64_t e0 = gr.row_ptr[i], e1 = gr.row_ptr[i + 1];
  // One thread walks the ~2P/n incident pairs of its item.  Done entry by entry this is a chain of four dependent
  // global loads per entry (index, pair, value, cell: 3 us each, 49 us per Newton iteration at C4 size on 32 SMs);
  // the loads of eight entries are issued together instead, and only the sums stay sequential (same order).
  constexpr int CH = 8;
  double wf = 0.0;
  int32_t cur_j = -1;
  double wij = 0.0, f_cur = 0.0, g_cur = 0.0;
  auto close_group = [&]() {
    if (cur_j < 0) return;
    wf = fma(wij, f_cur, wf);
    if (G && cur_j < i) G[i * ld + cur_j] = g_cur + wij;
    if (Wdense) Wdense[i * n + cur_j] = wij;
  };
  for (int64_t base = e0; base < e1; base += CH) {
    int32_t oj[CH], pk[CH];
    double wv[CH], fv[CH], gv[CH];
#pragma unroll
    for (int q = 0; q < CH; ++q) {
      const bool on = base + q < e1;
      oj[q] = on ? gr.other[base + q] : -1;
      pk[q] = on ? gr.pair_by_other[base + q] : 0;
    }
#pragma unroll
    for (int q = 0; q < CH; ++q) {
      const bool on = oj[q] >= 0;
      wv[q] = on ? wk[pk[q]] : 0.0;
      fv[q] = on ? f[oj[q]] : 0.0;
      gv[q] = (on && G && oj[q] < i) ? G[i * ld + oj[q]] : 0.0;
    }
#pragma unroll
    for (int q = 0; q < CH; ++q) {
      if (oj[q] >= 0) {
        if (oj[q] != cur_j) {
          close_group();
          cur_j = oj[q]; wij = 0.0; f_cur = fv[q]; g_cur = gv[q];
        }
        wij -= wv[q];                                // W[xi, yi] -= -ddpy_df (GPpref.py:86-87)
      }
    }
  }
  close_group();
  double wii = 0.0;
  for (int64_t base = e0; base < e1; base += CH) {
    double wv[CH];
#pragma unroll
    for (int q = 0; q < CH; ++q) wv[q] = base + q < e1 ? wk[gr.pair_sorted[base + q]] : 0.0;
#pragma unroll
    for (int q = 0; q < CH; ++q)
      if (base + q < e1) wii += wv[q];               // W[xi, xi] -= ddpy_df (GPpref.py:84-85)
  }
  if (grad_mode == 1) {
    for (int64_t q = e0; q < e1; ++q) g += gr.is_u[q] ? -dk[gr.pair_by_other[q]] : dk[gr.pair_by_other[q]];
  }
  wf = fma(wii, f[i], wf);
  if (G) G[i * ld + i] += wii;
  if (Wdense) Wdense[i * n + i] = wii;
  if (b) b[i] = wf + g;
  if (g_out) g_out[i] = g;
}

// ---------------------------------------------------------------------------------------
// The Newton loops run on the device (GPpref.py:140-155 tests convergence on the host and prints once per
// iteration).  One iteration is captured into the body of a CUDA-graph WHILE node; the last kernel of the
// iteration (the finish kernel, thread 0) appends (f_error, objective) to a device trace, counts the iteration,
// looks at the factorisation's info word and decides whether the loop goes on: cudaGraphSetConditional.  The
// host launches the graph once and reads counter, status and trace once when it is done - nothing between
// iterations crosses PCIe and the stream never drains.
// ---------------------------------------------------------------------------------------
struct LoopCtl {
  int it;          // iterations completed
  int status;      // 0 running / stopped, 2: the factorisation inside an iteration failed (pivot holds info)
  int pivot;
  int max_iter;
  double delta_f;
};
__device__ __forceinline__ void loop_step(LoopCtl* ctl, double* trace, const int* info, cudaGraphConditionalHandle hc,
                                          double f_error, double objective) {
  const int it = ctl->it;
  trace[2 * it] = f_error;
  trace[2 * it + 1] = objective;
  ctl->it = it + 1;
  const int piv = *info;
  if (piv != 0) { ctl->status = 2; ctl->pivot = piv; }
  // GPpref.py:140: while f_error > delta_f (a NaN error ends the loop, as it does on the host)
  const bool go = piv == 0 && (f_error > ctl->delta_f) && (it + 1 < ctl->max_iter);
  cudaGraphSetConditional(hc, go ? 1u : 0u);
}

// lml = sum log Phi(z(f_new)) - 0.5 f_new' iK f_new - 0.5 logdetK - n/2 log(2 pi)   (GPpref.py:90-94)
// f_error = max |f_new - f| (GPpref.py:151-152); then f <- f_new (GPpref.py:155)
// Two stages: the P log-Phi terms are ~100 FP64 operations each - on ONE SM (round 1) that was 26 us of its FP64
// pipe per Newton iteration; now PREF_PARTS CTAs reduce their slices into partials, and the one-CTA finish kernel
// adds the partials in a fixed order (deterministic) and takes the loop decision.
constexpr int PREF_PARTS = 64;
__global__ void __launch_bounds__(256) pref_terms_kernel(const int64_t* __restrict__ uvi, const double* __restrict__ y,
                                                         int64_t P, int64_t n, double isqrt2sig,
                                                         const double* __restrict__ f_new, const double* __restrict__ f,
                                                         const double* __restrict__ t, double* __restrict__ part) {
  __shared__ double sh[256];
  const int64_t stride = static_cast<int64_t>(gridDim.x) * 256;
  double s = 0.0;
  for (int64_t k = blockIdx.x * 256 + threadIdx.x; k < P; k += stride) {
    const double z = y[k] * (isqrt2sig * (f_new[uvi[2 * k + 1]] - f_new[uvi[2 * k]]));
    s += log(normcdf(z));
  }
  const double slog = cta_sum<256>(s, sh);
  double q = 0.0, mx = 0.0;
  for (int64_t i = blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
    q = fma(f_new[i], t[i], q);
    mx = fmax(mx, fabs(f_new[i] - f[i]));
  }
  const double qs = cta_sum<256>(q, sh);
  const double m = cta_max<256>(mx, sh);
  if (threadIdx.x == 0) {
    part[blockIdx.x] = slog;
    part[PREF_PARTS + blockIdx.x] = qs;
    part[2 * PREF_PARTS + blockIdx.x] = m;
  }
}
__global__ void __launch_bounds__(256) pref_finish_kernel(int64_t n, const double* __restrict__ f_new, double* __restrict__ f,
                                                          const double* __restrict__ part, const double* __restrict__ logdet,
                                                          double* __restrict__ out2, LoopCtl* ctl = nullptr,
                                                          double* trace = nullptr, const int* info = nullptr,
                                                          cudaGraphConditionalHandle hc = 0) {
  for (int64_t i = threadIdx.x; i < n; i += 256) f[i] = f_new[i];
  if (threadIdx.x == 0) {
    double slog = 0.0, qs = 0.0, m = 0.0;
    for (int b = 0; b < PREF_PARTS; ++b) {
      slog += part[b];
      qs += part[PREF_PARTS + b];
      m = fmax(m, part[2 * PREF_PARTS + b]);
    }
    const double lml = slog - 0.5 * qs - 0.5 * logdet[0] - 0.5 * static_cast<double>(n) * LOG_2PI;
    out2[0] = m;
    out2[1] = lml;
    if (ctl) loop_step(ctl, trace, info, hc, m, lml);
  }
}

struct PrefGraphHost {
  std::vector<int64_t> row_ptr, ku, kv;
  std::vector<int32_t> other, pair_by_other, is_u, pair_sorted;
};

PrefGraphHost build_pref_graph(const int64_t* uvi, int64_t P, int64_t n) {
  PrefGraphHost g;
  g.row_ptr.assign(n + 1, 0);
  g.ku.assign(n, -1);
  g.kv.assign(n, -1);
  for (int64_t k = 0; k < P; ++k) {
    const int64_t u = uvi[2 * k], v = uvi[2 * k + 1];
    if (u < 0 || u >= n || v < 0 || v >= n) throw Error{"uvi index out of range"};
    g.ku[u] = k;                       // later pairs overwrite earlier ones
    g.kv[v] = k;
    if (u != v) { ++g.row_ptr[u + 1]; ++g.row_ptr[v + 1]; }     // u == v contributes exactly zero to W
  }
  for (int64_t i = 0; i < n; ++i) g.row_ptr[i + 1] += g.row_ptr[i];
  const int64_t nnz = g.row_ptr[n];
  g.other.resize(nnz); g.pair_by_other.resize(nnz); g.is_u.resize(nnz); g.pair_sorted.resize(nnz);
  std::vector<int64_t> fill(g.row_ptr.begin(), g.row_ptr.end() - 1);
  struct Ent { int32_t other, pair, is_u; };
  std::vector<Ent> ent(nnz);
  for (int64_t k = 0; k < P; ++k) {
    const int64_t u = uvi[2 * k], v = uvi[2 * k + 1];
    if (u == v) continue;
    ent[fill[u]++] = Ent{static_cast<int32_t>(v), static_cast<int32_t>(k), 1};
    ent[fill[v]++] = Ent{static_cast<int32_t>(u), static_cast<int32_t>(k), 0};
  }
  for (int64_t i = 0; i < n; ++i) {
    const int64_t e0 = g.row_ptr[i], e1 = g.row_ptr[i + 1];
    for (int64_t e = e0; e < e1; ++e) g.pair_sorted[e] = ent[e].pair;      // filled in ascending pair order
    std::stable_sort(ent.begin() + e0, ent.begin() + e1, [](const Ent& a, const Ent& b) { return a.other < b.other; });
    for (int64_t e = e0; e < e1; ++e) {
      g.other[e] = ent[e].other;
      g.pair_by_other[e] = ent[e].pair;
      g.is_u[e] = ent[e].is_u;
    }
  }
  return g;
}

PrefDev upload_pref(gpb_handle* h, const PrefGraphHost& g, const int64_t* uvi, const double* y, int64_t P, int64_t n) {
  const int64_t nnz = g.row_ptr[n];
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  const size_t o_rp = take((n + 1) * 8), o_ku = take(n * 8), o_kv = take(n * 8), o_uvi = take(P * 16),
               o_y = take(P * 8), o_dk = take(P * 8), o_wk = take(P * 8), o_ot = take(nnz * 4 + 4),
               o_pb = take(nnz * 4 + 4), o_iu = take(nnz * 4 + 4), o_ps = take(nnz * 4 + 4);
  h->aux1.ensure(off);
  char* base = h->aux1.as<char>();
  auto up = [&](size_t o, const void* src, size_t bytes) {
    if (bytes) GPB_CUDA(cudaMemcpyAsync(base + o, src, bytes, cudaMemcpyHostToDevice, h->s0));
  };
  up(o_rp, g.row_ptr.data(), (n + 1) * 8); up(o_ku, g.ku.data(), n * 8); up(o_kv, g.kv.data(), n * 8);
  up(o_uvi, uvi, P * 16); up(o_y, y, P * 8);
  up(o_ot, g.other.data(), nnz * 4); up(o_pb, g.pair_by_other.data(), nnz * 4);
  up(o_iu, g.is_u.data(), nnz * 4); up(o_ps, g.pair_sorted.data(), nnz * 4);
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  PrefDev d;
  d.gr.row_ptr = reinterpret_cast<const int64_t*>(base + o_rp);
  d.gr.ku = reinterpret_cast<const int64_t*>(base + o_ku);
  d.gr.kv = reinterpret_cast<const int64_t*>(base + o_kv);
  d.gr.other = reinterpret_cast<const int32_t*>(base + o_ot);
  d.gr.pair_by_other = reinterpret_cast<const int32_t*>(base + o_pb);
  d.gr.is_u = reinterpret_cast<const int32_t*>(base + o_iu);
  d.gr.pair_sorted = reinterpret_cast<const int32_t*>(base + o_ps);
  d.uvi = reinterpret_cast<const int64_t*>(base + o_uvi);
  d.y = reinterpret_cast<const double*>(base + o_y);
  d.dk = reinterpret_cast<double*>(base + o_dk);
  d.wk = reinterpret_cast<double*>(base + o_wk);
  return d;
}

// ---------------------------------------------------------------------------------------
// classification likelihood (GPc.py:4-21; R&W eq. 3.15 / 3.16)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void gpc_terms(int link, double y, double f, double& lp, double& g, double& W) {
  if (link == 0) {                                  // probit: log Phi(y f)  (GPc.py:5-6)
    const double x = y * f;
    const double ex = erfcx(-x * INV_SQRT_2);       // Phi(x) = 0.5 erfcx(-x/sqrt2) exp(-x^2/2)
    const double r = SQRT_2_OVER_PI / ex;           // N(f)/Phi(yf), finite for every x
    lp = (x < 0.0) ? log(0.5 * ex) - 0.5 * x * x : log(normcdf(x));
    g = y * r;
    W = r * r + x * r;
  } else {                                          // logistic (GPc.py:13-14)
    const double x = y * f;
    lp = (x > 0.0) ? -log1p(exp(-x)) : x - log1p(exp(x));
    const double pi = 1.0 / (1.0 + exp(-f));
    g = 0.5 * (y + 1.0) - pi;
    W = pi * (1.0 - pi);
  }
}

// b = W f + g ; sW = sqrt(W) ; pads get W = 0
__global__ void gpc_terms_kernel(int link, const double* __restrict__ y, const double* __restrict__ f, int64_t n,
                                 int64_t n_pad, double* __restrict__ sW, double* __restrict__ b, double* __restrict__ g_out) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n_pad) return;
  if (i >= n) { sW[i] = 0.0; b[i] = 0.0; if (g_out) g_out[i] = 0.0; return; }
  double lp, g, W;
  gpc_terms(link, y[i], f[i], lp, g, W);
  sW[i] = sqrt(W);
  b[i] = fma(W, f[i], g);
  if (g_out) g_out[i] = g;
}
__global__ void vec_mul_kernel(double* __restrict__ dst, const double* __restrict__ a, const double* __restrict__ b, int64_t n) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) dst[i] = a[i] * b[i];
}
// a = b - sW * t
__global__ void gpc_a_kernel(double* __restrict__ a, const double* __restrict__ b, const double* __restrict__ sW,
                             const double* __restrict__ t, int64_t n) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) a[i] = b[i] - sW[i] * t[i];
}
// out2 = (max|f_new - f|, -0.5 a'f_new + sum log p(y|f_new)); f <- f_new
__global__ void __launch_bounds__(1024) gpc_finish_kernel(int link, const double* __restrict__ y, int64_t n,
                                                          const double* __restrict__ a, const double* __restrict__ f_new,
                                                          double* __restrict__ f, double* __restrict__ out2, LoopCtl* ctl,
                                                          double* trace, const int* info, cudaGraphConditionalHandle hc) {
  __shared__ double sh[1024];
  double q = 0.0, mx = 0.0, sl = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += 1024) {
    double lp, g, W;
    gpc_terms(link, y[i], f_new[i], lp, g, W);
    sl += lp;
    q = fma(a[i], f_new[i], q);
    mx = fmax(mx, fabs(f_new[i] - f[i]));
    f[i] = f_new[i];
  }
  const double qs = cta_sum<1024>(q, sh);
  const double ls = cta_sum<1024>(sl, sh);
  const double m = cta_max<1024>(mx, sh);
  if (threadIdx.x == 0) {
    out2[0] = m;
    out2[1] = -0.5 * qs + ls;
    if (ctl) loop_step(ctl, trace, info, hc, m, -0.5 * qs + ls);
  }
}
// rows[i][j] *= s[j]
__global__ void scale_cols_kernel(double* __restrict__ rows, int64_t ld, int64_t ncols, const double* __restrict__ s) {
  double* r = rows + blockIdx.x * ld;
  for (int64_t j = threadIdx.x; j < ncols; j += blockDim.x) r[j] *= s[j];
}
// r . t over ncols columns in a CTA of 256 threads, in a fixed order
__device__ __forceinline__ double row_dot256(const double* r, const double* t, int64_t ncols, double* sh) {
  double s = 0.0;
  for (int64_t j = threadIdx.x; j < ncols; j += 256) s = fma(r[j], t[j], s);
  return cta_sum<256>(s, sh);
}

// var_i = sf2 - |row_i|^2 ; prob_i from (mu_i, var_i)
__global__ void __launch_bounds__(256) gpc_predict_finish_kernel(const double* __restrict__ rows, int64_t ld, int64_t ncols,
                                                                 double sf2, int link, const double* __restrict__ mu,
                                                                 double* __restrict__ var, double* __restrict__ prob) {
  __shared__ double sh[256];
  const double* r = rows + blockIdx.x * ld;
  const double ss = row_dot256(r, r, ncols, sh);
  if (threadIdx.x == 0) {
    const double v = sf2 - ss;
    var[blockIdx.x] = v;
    const double m = mu[blockIdx.x];
    prob[blockIdx.x] = (link == 0) ? normcdf(m / sqrt(1.0 + v))                                   // R&W eq. 3.82
                                   : 1.0 / (1.0 + exp(-m / sqrt(1.0 + 0.39269908169872414 * v)));   // MacKay, pi/8
  }
}

// rows <- rows_b - rows (difference of two covariance row blocks); one CTA per row
__global__ void rows_sub_kernel(double* __restrict__ rows, const double* __restrict__ rows_b, int64_t ld, int64_t ncols) {
  double* r = rows + blockIdx.x * ld;
  const double* q = rows_b + blockIdx.x * ld;
  for (int64_t j = threadIdx.x; j < ncols; j += blockDim.x) r[j] = q[j] - r[j];
}
// k** of the quantity predicted: sf2 for one item, k(a,a) + k(b,b) - 2 k(a,b) for a difference (scaled points, pitch ld_t)
__global__ void pref_kss_kernel(const double* __restrict__ zaT, const double* __restrict__ zbT, int64_t ld_t, int d, int64_t m,
                                double sf2, double* __restrict__ kss) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= m) return;
  if (!zbT) { kss[i] = sf2; return; }
  double r2 = 0.0;
  for (int k = 0; k < d; ++k) {
    const double t = zaT[k * ld_t + i] - zbT[k * ld_t + i];
    r2 = fma(t, t, r2);
  }
  kss[i] = 2.0 * sf2 - 2.0 * sf2 * exp(-0.5 * r2);
}
// q1_i = R_i . T_i (two row blocks with the same pitch)
__global__ void __launch_bounds__(256) rows_dot2_kernel(const double* __restrict__ R, const double* __restrict__ T, int64_t ld,
                                                        int64_t ncols, double* __restrict__ out) {
  __shared__ double sh[256];
  const double ss = row_dot256(R + blockIdx.x * ld, T + blockIdx.x * ld, ncols, sh);
  if (threadIdx.x == 0) out[blockIdx.x] = ss;
}
// var_i = kss_i - q1_i + |V_i|^2 ; prob_i = Phi(mean_i / sqrt(2 sigma^2 + var_i)) for differences
__global__ void __launch_bounds__(256) pref_predict_finish_kernel(const double* __restrict__ V, int64_t ld, int64_t ncols,
                                                                  const double* __restrict__ kss, const double* __restrict__ q1,
                                                                  const double* __restrict__ mean, double two_sigma2,
                                                                  double* __restrict__ var, double* __restrict__ prob) {
  __shared__ double sh[256];
  const double* r = V + blockIdx.x * ld;
  const double ss = row_dot256(r, r, ncols, sh);
  if (threadIdx.x == 0) {
    const double v = kss[blockIdx.x] - q1[blockIdx.x] + ss;
    var[blockIdx.x] = v;
    if (prob) prob[blockIdx.x] = normcdf(mean[blockIdx.x] / sqrt(two_sigma2 + fmax(v, 0.0)));
  }
}

// chol(K^-1 + W(f_hat)) into the work space (the loop leaves the factor of the PREVIOUS iterate there)
void pref_factor_at_mode(gpb_handle* h, LaplaceState& ps) {
  if (ps.factored) return;
  const int64_t n = ps.n, np = h->n_pad;
  FactorMat g = laplace_mat(h, np);
  const double* iK = h->aux2.as<double>();
  double* f = lap_vecs(h, LaplaceState::PREF).f;
  const double isq = 1.0 / (ps.sigma * std::sqrt(2.0)), i2v = isq * isq;
  pref_pair_kernel<<<static_cast<unsigned>((ps.P + 255) / 256), 256, 0, h->s0>>>(ps.pd.uvi, ps.pd.y, ps.P, f, isq, i2v,
                                                                               ps.pd.dk, ps.pd.wk);
  scale_copy_lower_kernel<<<static_cast<unsigned>(np), 256, 0, h->s0>>>(iK, np, g.A, g.ld, nullptr, 0.0);
  pref_row_kernel<<<static_cast<unsigned>((n + 63) / 64), 64, 0, h->s0>>>(n, ps.pd.gr, ps.pd.dk, ps.pd.wk, f, 1, g.A,
                                                                            g.ld, nullptr, nullptr, nullptr);
  GPB_CUDA(cudaGetLastError());
  GPB_CUDA(cudaMemsetAsync(g.info, 0, 4, h->s0));
  chol_sweep(h, g, true);
  double* sc = h->scal.as<double>();
  sum_log_kernel<<<1, 512, 0, h->s0>>>(g.diag, np, sc + 8);
  GPB_CUDA(cudaGetLastError());
  h->launches += 4;
  double sum_log_g;
  if (read_info(h, g.info, sc + 8, &sum_log_g)) throw Error{"K^-1 + W is not positive definite at the mode"};
  ps.sum_log_g = sum_log_g;
  ps.factored = true;
}

// ---- gradient of the evidence w.r.t. the hyper-parameters (gpb_pref_evidence_grad; DESIGN.md section 4.3) ---------
// r = N(z)/Phi(z), w = r (z + r), r2 = r ((z + r)(z + 2r) - 1) = -dw/dz.  Below z = -3 the closed forms cancel
// (r2 loses 3e-11 relative at z = -5, 2e-5 at z = -30): with x = -z and the continued fraction of the Mills ratio
// c_k = k / (x + c_{k+1}):  r = x + c_1,  z + r = c_1,  r2 = r c_1^2 c_2 (c_3 - c_2).  64 terms: 3e-12 relative at z = -3.
constexpr double PREF_CF_BELOW = -3.0;
constexpr int PREF_CF_DEPTH = 64;
__device__ __forceinline__ void probit_terms(double z, double& r, double& w, double& r2) {
  if (z < PREF_CF_BELOW) {
    const double x = -z;
    double c = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
    for (int k = PREF_CF_DEPTH; k > 0; --k) {
      c = k / (x + c);
      if (k == 3) c3 = c;
      if (k == 2) c2 = c;
      if (k == 1) c1 = c;
    }
    r = x + c1;
    w = r * c1;
    r2 = r * c1 * c1 * c2 * (c3 - c2);
    return;
  }
  r = pref_hazard(z);
  const double q = z + r;
  w = r * q;
  r2 = r * (q * (z + 2.0 * r) - 1.0);
}

// Per pair: c_k = s^2 (Gi_uu + Gi_vv - 2 Gi_uv) from the lower triangle of G^-1 (pitch ld), and the per-pair
// coefficients of  s2 = sum_k (r2_k c_k / 2) a_k  and  h = sum_k (w_k z_k - r_k) a_k  (a_k = y_k s (e_v - e_u)) into
// cs / ch, already multiplied by y_k s.  The two sigma sums  sum r z  and  sum (r2 z - 2 w) c  go to PREF_PARTS
// fixed-order partials per CTA (grid = PREF_PARTS).
__global__ void __launch_bounds__(256) pref_grad_pair_kernel(const int64_t* __restrict__ uvi, const double* __restrict__ y,
                                                             int64_t P, const double* __restrict__ f, double s,
                                                             const double* __restrict__ Gi, int64_t ld,
                                                             double* __restrict__ cs, double* __restrict__ ch,
                                                             double* __restrict__ part) {
  __shared__ double sh[256];
  const int64_t stride = static_cast<int64_t>(gridDim.x) * 256;
  double srz = 0.0, src = 0.0;
  for (int64_t k = blockIdx.x * 256 + threadIdx.x; k < P; k += stride) {
    const int64_t u = uvi[2 * k], v = uvi[2 * k + 1];
    const double ys = y[k] * s;
    const double z = y[k] * (s * (f[v] - f[u]));                  // as pref_pair_kernel forms it
    double r, w, r2;
    probit_terms(z, r, w, r2);
    const int64_t hi = u > v ? u : v, lo = u > v ? v : u;
    const double c = s * s * ((Gi[u * ld + u] + Gi[v * ld + v]) - 2.0 * Gi[hi * ld + lo]);
    cs[k] = ys * (0.5 * r2 * c);
    ch[k] = ys * (w * z - r);
    srz = fma(r, z, srz);
    src = fma(fma(r2, z, -2.0 * w), c, src);
  }
  const double a = cta_sum<256>(srz, sh);
  const double b = cta_sum<256>(src, sh);
  if (threadIdx.x == 0) {
    part[blockIdx.x] = a;
    part[PREF_PARTS + blockIdx.x] = b;
  }
}

// per item i: s2_i = sum_k cs_k (e_v - e_u)_i and h_i likewise, over the incident pairs in ascending pair order
__global__ void pref_grad_item_kernel(int64_t n, const PrefGraphDev gr, const int64_t* __restrict__ uvi,
                                      const double* __restrict__ cs, const double* __restrict__ ch,
                                      double* __restrict__ s2, double* __restrict__ hv) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  double a = 0.0, b = 0.0;
  for (int64_t e = gr.row_ptr[i]; e < gr.row_ptr[i + 1]; ++e) {
    const int64_t k = gr.pair_sorted[e];
    if (uvi[2 * k + 1] == i) { a += cs[k]; b += ch[k]; }
    else { a -= cs[k]; b -= ch[k]; }
  }
  s2[i] = a;
  hv[i] = b;
}

// b = alpha / 2 + u (the rank-two term of the trace pass);  out[0] = d evidence / d log sigma
//   = -sum r z - 1/2 sum (r2 z - 2 w) c + v'h   (partials of pref_grad_pair_kernel, added in a fixed order)
__global__ void __launch_bounds__(512) pref_grad_finish_kernel(int64_t np, const double* __restrict__ alpha,
                                                               const double* __restrict__ u, const double* __restrict__ v,
                                                               const double* __restrict__ hv, const double* __restrict__ part,
                                                               double* __restrict__ beta, double* __restrict__ out) {
  __shared__ double sh[512];
  double q = 0.0;
  for (int64_t i = threadIdx.x; i < np; i += 512) {
    beta[i] = fma(0.5, alpha[i], u[i]);
    q = fma(v[i], hv[i], q);
  }
  const double vh = cta_sum<512>(q, sh);
  if (threadIdx.x == 0) {
    double srz = 0.0, src = 0.0;
    for (int b = 0; b < PREF_PARTS; ++b) {
      srz += part[b];
      src += part[PREF_PARTS + b];
    }
    out[0] = (vh - srz) - 0.5 * src;
  }
}

// ---- gradient of the classification evidence w.r.t. the hyper-parameters (gpb_gpc_evidence_grad; DESIGN.md 4.3) ---
// One CTA per row i of V = K W^1/2 L_B^-T (fixed-order row reduction): Sigma_ii = K_ii - |V_i|^2, the diagonal of
// (K^-1 + W)^-1, and s2_i = +1/2 Sigma_ii d^3 log p(y_i|f_i) / df_i^3 (R&W Alg. 5.1 line 7 prints the opposite sign,
// which is wrong).  Probit: y r''(y f), tail-safe through probit_terms; logit: -pi (1 - pi)(1 - 2 pi) with the pi of
// gpc_terms, so that s2 differentiates the W the fit used.  Rows of the padding get 0.
__global__ void __launch_bounds__(256) gpc_grad_item_kernel(int link, const double* __restrict__ y,
                                                            const double* __restrict__ f, int64_t n,
                                                            const double* __restrict__ K, int64_t ldk,
                                                            const double* __restrict__ V, int64_t ld, int64_t ncols,
                                                            double* __restrict__ s2) {
  __shared__ double sh[256];
  const int64_t i = blockIdx.x;
  if (i >= n) {
    if (threadIdx.x == 0) s2[i] = 0.0;
    return;
  }
  const double* r = V + i * ld;
  const double ss = row_dot256(r, r, ncols, sh);
  if (threadIdx.x == 0) {
    double d3;
    if (link == 0) {
      double rr, w, r2;
      probit_terms(y[i] * f[i], rr, w, r2);
      d3 = y[i] * r2;
    } else {
      const double pi = 1.0 / (1.0 + exp(-f[i]));
      d3 = -(pi * (1.0 - pi)) * (1.0 - 2.0 * pi);
    }
    s2[i] = 0.5 * (K[i * ldk + i] - ss) * d3;
  }
}

// M[i][j] *= s[i] s[j], one CTA per row: R = W^1/2 B^-1 W^1/2 from the mirrored B^-1 (the product s[i] s[j] is
// formed first, so a symmetric M stays symmetric to the bit)
__global__ void scale_rows_cols_kernel(double* __restrict__ M, int64_t ld, int64_t ncols, const double* __restrict__ s) {
  double* r = M + blockIdx.x * ld;
  const double si = s[blockIdx.x];
  for (int64_t j = threadIdx.x; j < ncols; j += blockDim.x) r[j] *= si * s[j];
}

// b = a/2 + t,  t = s2 - R K s2  (rq = R K s2): the rank-two term of the trace pass
__global__ void gpc_grad_finish_kernel(const double* __restrict__ a, const double* __restrict__ s2,
                                       const double* __restrict__ rq, int64_t n, double* __restrict__ beta) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) beta[i] = fma(0.5, a[i], s2[i] - rq[i]);
}

// chol(I + sW K sW) at the stored mode into rows [0, np) of the work space: the end of gpb_gpc_laplace, and again
// after gpb_gpc_evidence_grad has overwritten it (same kernels, same bits).  sW (in aux0) and K + eps I (in aux2).
void gpc_factor_at_mode(gpb_handle* h) {
  if (h->lap.factored) return;
  const int64_t np = h->n_pad;
  FactorMat g = laplace_mat(h, np);
  g.rows_total = np;
  const double* K = h->aux2.as<double>();
  const double* sW = lap_vecs(h, LaplaceState::GPC).sW;
  scale_copy_lower_kernel<<<static_cast<unsigned>(np), 256, 0, h->s0>>>(K, np, g.A, g.ld, sW, 1.0);
  GPB_CUDA(cudaGetLastError());
  GPB_CUDA(cudaMemsetAsync(g.info, 0, 4, h->s0));
  chol_sweep(h, g, true);
  ++h->launches;
  h->lap.factored = true;
}

// The state of the last fit, if it is of this kind and current.
LaplaceState& lap_state(gpb_handle* h, LaplaceState::Kind kind) {
  LaplaceState& s = h->lap;
  // the entry macro has already counted this call: the state is current iff nothing else ran in between
  GPB_REQUIRE(s.kind == kind && s.n == h->n && h->state_epoch + 1 == h->ws_epoch,
              kind == LaplaceState::PREF
                  ? "no preference Laplace state on this handle: call gpb_pref_laplace first (any other call that uses "
                    "the work space invalidates it)"
                  : "no Laplace state on this handle: call gpb_gpc_laplace first (any other call that uses the work space "
                    "invalidates it)");
  return s;
}

// evidence = sum log Phi - f'K^-1 f/2 - sum log diag L_K - sum log diag chol(K^-1 + W)        (R&W eq. 3.32), from
// lml_ref = sum log Phi - f'K^-1 f/2 - (1/2) sum log diag L_K - n/2 log 2pi   (GPpref.py:90-94,131)
double pref_evidence_value(const LaplaceState& ps) {
  return ps.lml_ref - 0.5 * ps.half_logdet_k + 0.5 * static_cast<double>(ps.n) * LOG_2PI - ps.sum_log_g;
}

// Runs `iteration(handle)` - which enqueues ONE Newton iteration on h->s0 (side streams joined by events, as
// chol_sweep does) and ends with a finish kernel calling loop_step - as the body of a WHILE node until the device
// says stop.  ctl / trace: device; the iteration count, status and trace are read back here.
struct LoopResult {
  int it, status, pivot;         // iterations run; status 2: a factorisation failed, pivot holds its info
  int64_t launches_per_iteration;
  double last_error, last_objective;   // the last trace entry (0 when no iteration ran)
};
template <class F>
LoopResult run_device_loop_once(gpb_handle* h, LoopCtl* ctl_dev, double* trace_dev, double* trace_host, double delta_f,
                                int max_iter, F& iteration) {
  LoopCtl init{0, 0, 0, max_iter, delta_f};
  LoopCtl* hc_host = reinterpret_cast<LoopCtl*>(h->pinned(sizeof(LoopCtl) + 64));
  *hc_host = init;
  GPB_CUDA(cudaMemcpyAsync(ctl_dev, hc_host, sizeof(LoopCtl), cudaMemcpyHostToDevice, h->s0));
  h->prepare_capture();
  // The legacy default stream (what a caller gets from torch.cuda.current_stream() unless it made one) cannot be
  // captured: the loop then runs on a stream of the handle's own, ordered after the caller's stream by an event and
  // synchronised before this function returns.
  struct StreamSwap {
    gpb_handle* h;
    cudaStream_t user;
    bool on;
    ~StreamSwap() { if (on) h->s0 = user; }
  } swap{h, h->s0, h->s0 == nullptr || h->s0 == cudaStreamLegacy || h->s0 == cudaStreamPerThread};
  if (swap.on) {
    if (!h->s_loop) GPB_CUDA(cudaStreamCreateWithFlags(&h->s_loop, cudaStreamNonBlocking));
    cudaEvent_t e = h->next_event();
    GPB_CUDA(cudaEventRecord(e, swap.user));
    GPB_CUDA(cudaStreamWaitEvent(h->s_loop, e, 0));
    h->s0 = h->s_loop;
  }
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  LoopResult res{0, 0, 0, 0};
  const int64_t l0 = h->launches;
  try {
    GPB_CUDA(cudaGraphCreate(&graph, 0));
    cudaGraphConditionalHandle cond;
    GPB_CUDA(cudaGraphConditionalHandleCreate(&cond, graph, 1, cudaGraphCondAssignDefault));
    cudaGraphNodeParams np{};
    np.type = cudaGraphNodeTypeConditional;
    np.conditional.handle = cond;
    np.conditional.type = cudaGraphCondTypeWhile;
    np.conditional.size = 1;
    cudaGraphNode_t node;
    GPB_CUDA(cudaGraphAddNode(&node, graph, nullptr, 0, &np));
    cudaGraph_t body = np.conditional.phGraph_out[0];
    const auto t_cap0 = std::chrono::steady_clock::now();
    GPB_CUDA(cudaStreamBeginCaptureToGraph(h->s0, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
    h->capturing = true;
    g_capturing = 1;
    try {
      iteration(cond);
    } catch (...) {
      h->capturing = false;
      g_capturing = 0;
      cudaGraph_t dummy = nullptr;
      cudaStreamEndCapture(h->s0, &dummy);
      throw;
    }
    h->capturing = false;
    g_capturing = 0;
    GPB_CUDA(cudaStreamEndCapture(h->s0, nullptr));
    res.launches_per_iteration = h->launches - l0;
    h->launches = l0;
    const auto t_cap1 = std::chrono::steady_clock::now();
    // per-node priorities (the look-ahead panel stream is a high-priority stream) only count with this flag
    GPB_CUDA(cudaGraphInstantiate(&exec, graph, cudaGraphInstantiateFlagUseNodePriority));
    const auto t_cap2 = std::chrono::steady_clock::now();
    GPB_CUDA(cudaGraphLaunch(exec, h->s0));
    if (getenv("GPB_DEBUG_LOOP"))
      fprintf(stderr, "[gpb] device loop: %lld launches per iteration, capture %.3f ms, instantiate %.3f ms, pdl %d\n",
              static_cast<long long>(res.launches_per_iteration), std::chrono::duration<double, std::milli>(t_cap1 - t_cap0).count(),
              std::chrono::duration<double, std::milli>(t_cap2 - t_cap1).count(), g_pdl);
    GPB_CUDA(cudaMemcpyAsync(hc_host, ctl_dev, sizeof(LoopCtl), cudaMemcpyDeviceToHost, h->s0));
    GPB_CUDA(cudaStreamSynchronize(h->s0));
    res.it = hc_host->it; res.status = hc_host->status; res.pivot = hc_host->pivot;
    if (res.it > 0 && trace_host) {
      GPB_CUDA(cudaMemcpyAsync(trace_host, trace_dev, static_cast<size_t>(res.it) * 16, cudaMemcpyDeviceToHost, h->s0));
      GPB_CUDA(cudaStreamSynchronize(h->s0));
    }
    h->launches += res.launches_per_iteration * res.it;
  } catch (...) {
    h->launches = l0;
    if (exec) cudaGraphExecDestroy(exec);
    if (graph) cudaGraphDestroy(graph);
    throw;
  }
  cudaGraphExecDestroy(exec);
  cudaGraphDestroy(graph);
  return res;
}
// The Newton loop of a fit: `iteration(ctl, trace_dev, cond)` enqueues one iteration whose finish kernel calls
// loop_step(ctl, trace_dev, ..., cond).  The (f_error, objective) trace goes to `trace` (2 x max_iter, may be null).
template <class F>
LoopResult run_device_loop(gpb_handle* h, double delta_f, int max_iter, double* trace, F&& iteration) {
  h->trace.ensure(static_cast<size_t>(max_iter) * 16);
  double* trace_dev = h->trace.as<double>();
  LoopCtl* ctl = reinterpret_cast<LoopCtl*>(h->scal.as<double>() + 16);
  std::vector<double> trace_local;
  if (!trace) trace_local.resize(static_cast<size_t>(max_iter) * 2);
  double* trace_host = trace ? trace : trace_local.data();
  auto body = [&](cudaGraphConditionalHandle cond) { iteration(ctl, trace_dev, cond); };
  LoopResult r;
  try {
    r = run_device_loop_once(h, ctl, trace_dev, trace_host, delta_f, max_iter, body);
  } catch (const Error&) {
    // Programmatic dependent launches are the one construct of an iteration a graph body may refuse (no kernel has
    // run yet: capture or instantiation failed).  Same graph, plain dependencies.
    if (getenv("GPB_DEBUG_LOOP")) fprintf(stderr, "[gpb] device loop: first attempt failed (%s), retrying without PDL\n", h->err.c_str());
    if (g_pdl == 0) throw;
    cudaGetLastError();
    const int saved = g_pdl;
    g_pdl = 0;
    try {
      r = run_device_loop_once(h, ctl, trace_dev, trace_host, delta_f, max_iter, body);
      g_pdl = saved;
    } catch (...) {
      g_pdl = saved;
      throw;
    }
  }
  if (r.it > 0) {
    r.last_error = trace_host[2 * (r.it - 1)];
    r.last_objective = trace_host[2 * (r.it - 1) + 1];
  }
  return r;
}

}  // namespace

extern "C" {

int gpb_pref_derivatives(gpb_handle* h, const int64_t* uvi, const double* y, int64_t P, int64_t n, const double* f,
                         double sigma, int32_t grad_mode, double* W_out, double* g_out) {
  GPB_API_BEGIN
  GPB_REQUIRE(uvi && y && f && P > 0 && n > 0 && W_out && g_out, "null argument");
  PrefGraphHost g = build_pref_graph(uvi, P, n);
  PrefDev pd = upload_pref(h, g, uvi, y, P, n);
  h->aux0.ensure(static_cast<size_t>(n) * 16);
  h->aux2.ensure(static_cast<size_t>(n) * n * 8);
  double* fd = h->aux0.as<double>();
  double* gd = fd + n;
  GPB_CUDA(cudaMemcpyAsync(fd, f, n * 8, cudaMemcpyHostToDevice, h->s0));
  GPB_CUDA(cudaMemsetAsync(h->aux2.p, 0, static_cast<size_t>(n) * n * 8, h->s0));
  const double isq = 1.0 / (sigma * std::sqrt(2.0)), i2v = isq * isq;      // GPpref.py:53-54
  pref_pair_kernel<<<static_cast<unsigned>((P + 255) / 256), 256, 0, h->s0>>>(pd.uvi, pd.y, P, fd, isq, i2v, pd.dk, pd.wk);
  pref_row_kernel<<<static_cast<unsigned>((n + 63) / 64), 64, 0, h->s0>>>(n, pd.gr, pd.dk, pd.wk, fd, grad_mode,
                                                                            nullptr, 0, nullptr, gd, h->aux2.as<double>());
  GPB_CUDA(cudaGetLastError());
  h->launches += 2;
  GPB_CUDA(cudaMemcpyAsync(W_out, h->aux2.p, static_cast<size_t>(n) * n * 8, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaMemcpyAsync(g_out, gd, n * 8, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  GPB_API_END
}

int gpb_pref_log_marginal(gpb_handle* h, const int64_t* uvi, const double* y, int64_t P, int64_t n, const double* f,
                          const double* iK, double logdetK, double sigma, double* out) {
  GPB_API_BEGIN
  GPB_REQUIRE(uvi && y && f && iK && out && P > 0 && n > 0, "null argument");
  for (int64_t k = 0; k < 2 * P; ++k) GPB_REQUIRE(uvi[k] >= 0 && uvi[k] < n, "uvi index out of range");
  const int64_t ne = round_up(n, 2);                       // even pitch for the 16-byte loads of row_dot
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  const size_t o_uvi = take(P * 16), o_y = take(P * 8), o_f = take(ne * 8), o_f2 = take(ne * 8), o_t = take(ne * 8),
               o_sc = take(64 + 3 * PREF_PARTS * 8);
  h->aux1.ensure(off);
  h->aux2.ensure(static_cast<size_t>(n) * ne * 8);
  char* base = h->aux1.as<char>();
  double* fd = reinterpret_cast<double*>(base + o_f);
  double* f2 = reinterpret_cast<double*>(base + o_f2);
  double* td = reinterpret_cast<double*>(base + o_t);
  double* sc = reinterpret_cast<double*>(base + o_sc);
  GPB_CUDA(cudaMemsetAsync(base, 0, off, h->s0));
  GPB_CUDA(cudaMemsetAsync(h->aux2.p, 0, static_cast<size_t>(n) * ne * 8, h->s0));
  GPB_CUDA(cudaMemcpyAsync(base + o_uvi, uvi, P * 16, cudaMemcpyHostToDevice, h->s0));
  GPB_CUDA(cudaMemcpyAsync(base + o_y, y, P * 8, cudaMemcpyHostToDevice, h->s0));
  GPB_CUDA(cudaMemcpyAsync(fd, f, n * 8, cudaMemcpyHostToDevice, h->s0));
  GPB_CUDA(cudaMemcpyAsync(f2, f, n * 8, cudaMemcpyHostToDevice, h->s0));
  GPB_CUDA(cudaMemcpy2DAsync(h->aux2.p, ne * 8, iK, n * 8, n * 8, n, cudaMemcpyHostToDevice, h->s0));
  GPB_CUDA(cudaMemcpyAsync(sc, &logdetK, 8, cudaMemcpyHostToDevice, h->s0));
  launch_row_dot(h->aux2.as<double>(), ne, 0, fd, 0, n, ne, 0, td, 0, 1, h->s0);            // t = iK f
  const double isq = 1.0 / (sigma * std::sqrt(2.0));
  pref_terms_kernel<<<PREF_PARTS, 256, 0, h->s0>>>(reinterpret_cast<const int64_t*>(base + o_uvi),
                                                   reinterpret_cast<const double*>(base + o_y), P, n, isq, fd, f2, td, sc + 8);
  pref_finish_kernel<<<1, 256, 0, h->s0>>>(n, fd, f2, sc + 8, sc, sc + 2);
  GPB_CUDA(cudaGetLastError());
  h->launches += 2;
  double* host = h->pinned(64);
  GPB_CUDA(cudaMemcpyAsync(host, sc + 2, 16, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  *out = host[1];
  GPB_API_END
}

int gpb_pref_laplace(gpb_handle* h, const int64_t* uvi, const double* y, int64_t P, const double* khyp, double sigma,
                     double delta_f, int32_t max_iter, int32_t grad_mode, int32_t use_f0, double* f_inout, double* lml,
                     int32_t* iters, double* trace, double* jitter, int32_t* info) {
  GPB_API_BEGIN
  h->lap = LaplaceState{};                               // filled only when the fit succeeds
  GPB_REQUIRE(h->n > 0, "no training inputs: call gpb_set_train first");
  GPB_REQUIRE(uvi && y && khyp && f_inout && lml && iters && P > 0 && max_iter > 0, "null argument");
  const int64_t n = h->n, np = h->n_pad;
  if (info) *info = 0;
  PrefGraphHost graph = build_pref_graph(uvi, P, n);
  PrefDev pd = upload_pref(h, graph, uvi, y, P, n);
  tic(h, 0);

  // ---- K + eps I, its factor, log-determinant and explicit inverse (GPpref.py:121-135) ----
  LapMat m = laplace_mat(h, np);
  const double eps = factor_with_jitter(h, m, khyp, info, [&](const KernelParams& pr) {
    const PointSet x = train_points(h);
    scale_points(h, x, h->X.as<double>(), h->d, pr.ell);
    build_cov(h, x, x, h->d, 1, LAP_KIND, LAP_CLIP, pr.hyp2, m.A, m.ld);
  });
  if (jitter) *jitter = eps;
  h->scal.ensure(2048);
  double* sc = h->scal.as<double>();    // [0] logdetK (= sum log diag L, GPpref.py:131)  [2..3] per-iteration out  [16..] loop
  sum_log_kernel<<<1, 512, 0, h->s0>>>(m.diag, np, sc);
  ++h->launches;
  m.rows_total = 2 * np + TILE;
  chol_inverse_lower(h, m);                                                // iK (GPpref.py:129)
  h->aux2.ensure(static_cast<size_t>(np) * np * 8);
  double* iK = h->aux2.as<double>();
  {
    const int64_t nt64 = np / 64;
    mirror_lower_kernel<<<static_cast<unsigned>(nt64 * nt64), 256, 0, h->s0>>>(m.A, m.ld, iK, np, nt64);
    GPB_CUDA(cudaGetLastError());
    ++h->launches;
  }
  tic(h, 1);

  // ---- Newton iterations (GPpref.py:138-155) ----
  h->aux0.ensure(static_cast<size_t>(np) * 8 * PREF_VECS);
  const LapVecs v = lap_vecs(h, LaplaceState::PREF);
  GPB_CUDA(cudaMemsetAsync(v.f, 0, static_cast<size_t>(np) * 8 * PREF_VECS, h->s0));
  if (use_f0) GPB_CUDA(cudaMemcpyAsync(v.f, f_inout, n * 8, cudaMemcpyHostToDevice, h->s0));
  const double isq = 1.0 / (sigma * std::sqrt(2.0)), i2v = isq * isq;      // GPpref.py:53-54
  m.rows_total = np + 1;
  double* part = sc + 32;                            // 3 x PREF_PARTS partial sums of the finish stage
  const LoopResult lr = run_device_loop(h, delta_f, max_iter, trace, [&](LoopCtl* ctl, double* trace_dev,
                                                                          cudaGraphConditionalHandle cond) {
    pref_pair_kernel<<<static_cast<unsigned>((P + 255) / 256), 256, 0, h->s0>>>(pd.uvi, pd.y, P, v.f, isq, i2v, pd.dk, pd.wk);
    scale_copy_lower_kernel<<<static_cast<unsigned>(np), 256, 0, h->s0>>>(iK, np, m.A, m.ld, nullptr, 0.0);
    GPB_CUDA(cudaMemsetAsync(m.row, 0, np * 8, h->s0));
    pref_row_kernel<<<static_cast<unsigned>((n + 63) / 64), 64, 0, h->s0>>>(n, pd.gr, pd.dk, pd.wk, v.f, grad_mode, m.A,
                                                                              m.ld, m.row, nullptr, nullptr);
    GPB_CUDA(cudaGetLastError());
    h->launches += 3;
    GPB_CUDA(cudaMemsetAsync(m.info, 0, 4, h->s0));
    chol_sweep(h, m, true);                                  // G = L L^T, appended row <- L^-1 (W f + grad)
    trsv_lt(h, m, m.row, v.f_new);                           // f_new = G^-1 (W f + grad)   (GPpref.py:143)
    launch_row_dot(iK, np, 0, v.f_new, 0, np, np, 0, v.t, 0, 1, h->s0);
    pref_terms_kernel<<<PREF_PARTS, 256, 0, h->s0>>>(pd.uvi, pd.y, P, n, isq, v.f_new, v.f, v.t, part);
    pref_finish_kernel<<<1, 256, 0, h->s0>>>(n, v.f_new, v.f, part, sc, sc + 2, ctl, trace_dev, m.info, cond);
    GPB_CUDA(cudaGetLastError());
    h->launches += 3;
  });
  if (lr.status == 2) { if (info) *info = lr.pivot; throw Error{"K^-1 + W is not positive definite"}; }
  tic(h, 2);
  double* host = h->pinned(64);
  GPB_CUDA(cudaMemcpyAsync(f_inout, v.f, n * 8, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaMemcpyAsync(host, sc, 8, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  *lml = lr.last_objective;
  *iters = lr.it;
  collect_timings(h, 2);
  LaplaceState& s = h->lap;
  s.n = n; s.khyp.assign(khyp, khyp + h->d + 1); s.eps = eps;
  s.P = P; s.sigma = sigma; s.lml_ref = lr.last_objective; s.half_logdet_k = host[0]; s.grad_mode = grad_mode; s.pd = pd;
  s.kind = LaplaceState::PREF;
  h->state_epoch = h->ws_epoch;
  GPB_API_END
}

int gpb_gpc_laplace(gpb_handle* h, const double* y, const double* khyp, int32_t link, double delta_f, int32_t max_iter,
                    int32_t use_f0, double* f_inout, double* lml, int32_t* iters, double* trace, double* jitter,
                    int32_t* info) {
  GPB_API_BEGIN
  h->lap = LaplaceState{};                               // filled only when the fit succeeds
  GPB_REQUIRE(h->n > 0, "no training inputs: call gpb_set_train first");
  GPB_REQUIRE(y && khyp && f_inout && lml && iters && max_iter > 0, "null argument");
  const int64_t n = h->n, np = h->n_pad;
  if (info) *info = 0;
  tic(h, 0);
  LapMat m = laplace_mat(h, np);
  h->aux2.ensure(static_cast<size_t>(np) * np * 8);
  double* K = h->aux2.as<double>();                      // full symmetric K + eps I
  const double eps = factor_with_jitter(h, m, khyp, info, [&](const KernelParams& pr) {
    const PointSet x = train_points(h);
    scale_points(h, x, h->X.as<double>(), h->d, pr.ell);
    build_cov(h, x, x, h->d, 0, LAP_KIND, LAP_CLIP, pr.hyp2, K, np);
    scale_copy_lower_kernel<<<static_cast<unsigned>(np), 256, 0, h->s0>>>(K, np, m.A, m.ld, nullptr, 0.0);
    ++h->launches;
  });
  if (jitter) *jitter = eps;
  h->aux0.ensure(static_cast<size_t>(np) * 8 * GPC_VECS);
  const LapVecs v = lap_vecs(h, LaplaceState::GPC);
  GPB_CUDA(cudaMemsetAsync(v.f, 0, static_cast<size_t>(np) * 8 * GPC_VECS, h->s0));
  GPB_CUDA(cudaMemcpyAsync(v.y, y, n * 8, cudaMemcpyHostToDevice, h->s0));
  if (use_f0) GPB_CUDA(cudaMemcpyAsync(v.f, f_inout, n * 8, cudaMemcpyHostToDevice, h->s0));
  h->scal.ensure(2048);
  double* sc = h->scal.as<double>();                     // [0] sum log diag L_B  [2..3] per-iteration out  [16..] loop
  m.rows_total = np + 1;
  const unsigned vb = static_cast<unsigned>((np + 255) / 256);
  const LoopResult lr = run_device_loop(h, delta_f, max_iter, trace, [&](LoopCtl* ctl, double* trace_dev,
                                                                          cudaGraphConditionalHandle cond) {
    gpc_terms_kernel<<<vb, 256, 0, h->s0>>>(link, v.y, v.f, n, np, v.sW, v.b, nullptr);               // Alg 3.1 lines 4, 6
    scale_copy_lower_kernel<<<static_cast<unsigned>(np), 256, 0, h->s0>>>(K, np, m.A, m.ld, v.sW, 1.0);  // B = I + sW K sW
    launch_row_dot(K, np, 0, v.b, 0, np, np, 0, v.t, 0, 1, h->s0);                                  // K b
    vec_mul_kernel<<<vb, 256, 0, h->s0>>>(m.row, v.sW, v.t, np);                                     // sW K b
    GPB_CUDA(cudaGetLastError());
    GPB_CUDA(cudaMemsetAsync(m.info, 0, 4, h->s0));
    chol_sweep(h, m, true);                                                                         // L = chol(B), row <- L^-1 (sW K b)
    trsv_lt(h, m, m.row, v.t);                                                                      // L^T \ ( L \ (sW K b) )
    gpc_a_kernel<<<vb, 256, 0, h->s0>>>(v.a, v.b, v.sW, v.t, np);                                   // line 7
    launch_row_dot(K, np, 0, v.a, 0, np, np, 0, v.f_new, 0, 1, h->s0);                              // line 8: f = K a
    gpc_finish_kernel<<<1, 1024, 0, h->s0>>>(link, v.y, n, v.a, v.f_new, v.f, sc + 2, ctl, trace_dev, m.info, cond);
    GPB_CUDA(cudaGetLastError());
    h->launches += 7;
  });
  if (lr.status == 2) { if (info) *info = lr.pivot; throw Error{"I + sW K sW is not positive definite"}; }
  double* host = h->pinned(64);
  // approximate log marginal likelihood at the returned f (Alg 3.1 line 10): W, L re-evaluated at f
  gpc_terms_kernel<<<vb, 256, 0, h->s0>>>(link, v.y, v.f, n, np, v.sW, v.b, v.g);
  gpc_factor_at_mode(h);
  sum_log_kernel<<<1, 512, 0, h->s0>>>(m.diag, np, sc);
  GPB_CUDA(cudaGetLastError());
  h->launches += 2;
  tic(h, 1);
  GPB_CUDA(cudaMemcpyAsync(host, sc, 8, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaMemcpyAsync(f_inout, v.f, n * 8, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  *lml = lr.last_objective - host[0];
  *iters = lr.it;
  collect_timings(h, 1, false);
  // state for gpb_gpc_predict: L and Dinv (in h->A / h->Dinv), sW, grad, kernel parameters; for
  // gpb_gpc_evidence_grad also K (aux2), a, y, the returned lml and jitter
  LaplaceState& s = h->lap;                              // factored: set by gpc_factor_at_mode
  s.n = n; s.khyp.assign(khyp, khyp + h->d + 1); s.eps = eps;
  s.link = link; s.lml = *lml; s.converged = lr.it > 0 && lr.last_error <= delta_f;
  s.kind = LaplaceState::GPC;
  h->state_epoch = h->ws_epoch;
  GPB_API_END
}

int gpb_gpc_predict(gpb_handle* h, const double* Z, int64_t mz, double* mu, double* var, double* prob) {
  GPB_API_BEGIN
  const LaplaceState& s = lap_state(h, LaplaceState::GPC);
  GPB_REQUIRE(Z && mu && var && prob && mz > 0, "null argument");
  gpc_factor_at_mode(h);                       // after gpb_gpc_evidence_grad: B is factored again (same bits)
  const int64_t np = h->n_pad;
  LapMat m = laplace_mat(h, np);               // same buffers: L of B is still in rows [0, np)
  const LapVecs v = lap_vecs(h, LaplaceState::GPC);
  const KernelParams pr = lap_params(h, s.khyp.data(), 0.0);
  const double sf2 = s.khyp[h->d];
  const int64_t cap = np;                      // test rows: S1 (np rows)
  h->outv.ensure(static_cast<size_t>(cap) * 8 * 3);
  double* o = h->outv.as<double>();
  for (int64_t z0 = 0; z0 < mz; z0 += cap) {
    const int64_t mc = mz - z0 < cap ? mz - z0 : cap;
    const int64_t mp64 = round_up(mc, 64);
    h->Zd.ensure(static_cast<size_t>(mc) * h->d * 8);
    h->ZsT.ensure(static_cast<size_t>(h->d) * mp64 * 8);
    h->zsq.ensure(static_cast<size_t>(mp64) * 8);
    test_cov_rows(h, Z + z0 * h->d, mc, pr, h->Zd.as<double>(), h->ZsT.as<double>(), h->zsq.as<double>(), m.S1,
                  m.ld);                                                            // k*^T rows
    launch_row_dot(m.S1, m.ld, 0, v.g, 0, mc, np, 0, o, 0, 1, h->s0);               // Alg 3.2 line 4: k*^T grad
    scale_cols_kernel<<<static_cast<unsigned>(mc), 256, 0, h->s0>>>(m.S1, m.ld, np, v.sW);
    GPB_CUDA(cudaGetLastError());
    h->launches += 2;
    sweep_rows(h, m, m.t1, mc);                                                     // rows <- (L^-1 sW k*)^T  (line 5)
    gpc_predict_finish_kernel<<<static_cast<unsigned>(mc), 256, 0, h->s0>>>(m.S1, m.ld, np, sf2, s.link, o, o + cap, o + 2 * cap);
    GPB_CUDA(cudaGetLastError());
    ++h->launches;
    GPB_CUDA(cudaMemcpyAsync(mu + z0, o, mc * 8, cudaMemcpyDeviceToHost, h->s0));
    GPB_CUDA(cudaMemcpyAsync(var + z0, o + cap, mc * 8, cudaMemcpyDeviceToHost, h->s0));
    GPB_CUDA(cudaMemcpyAsync(prob + z0, o + 2 * cap, mc * 8, cudaMemcpyDeviceToHost, h->s0));
    GPB_CUDA(cudaStreamSynchronize(h->s0));
  }
  h->state_epoch = h->ws_epoch;                // the state is still current: predict again without refitting
  GPB_API_END
}

// Work space (laplace_mat): rows [0, np) L_B -> B^-1 | tile row | S1 [np+128, 2np+128) | S2 [2np+128, 3np+128).
//   S2 <- K diag(sW), swept through L_B:     V = K W^1/2 L_B^-T                     (n^3)
//   S1 <- I, swept (grow) and U U^T:         B^-1 in the lower tiles of [0, np)     (n^3/3 + n^3/3, chol_inverse_lower)
// then Sigma_ii and s2 from V (gpc_grad_item_kernel), B^-1 mirrored into S2 over V and scaled: R = W^1/2 B^-1 W^1/2,
// q = K s2, b = a/2 + s2 - R q, and the trace pass of grad.cu over (R, a, b).  The sweep reads L_B before
// chol_inverse_lower overwrites it.
int gpb_gpc_evidence_grad(gpb_handle* h, double* lml, double* grad) {
  GPB_API_BEGIN
  GPB_REQUIRE(lml && grad, "null argument");
  const LaplaceState& s = lap_state(h, LaplaceState::GPC);
  if (!s.converged) {
    h->state_epoch = h->ws_epoch;              // nothing was touched: the state stays usable
    throw Error{"the evidence gradient needs a converged mode: the last gpb_gpc_laplace stopped at max_iter with "
                "max|f_new - f| > delta_f (the formula is exact only at a stationary point)"};
  }
  const int64_t n = h->n, np = h->n_pad;
  const int d = h->d;
  const KernelParams pr = lap_params(h, s.khyp.data(), s.eps);
  tic(h, 0);
  gpc_factor_at_mode(h);
  tic(h, 1);
  LapMat m = laplace_mat(h, np);
  const double* K = h->aux2.as<double>();
  const LapVecs v = lap_vecs(h, LaplaceState::GPC);
  const int64_t t64 = np / 64, ntiles = t64 * (t64 + 1) / 2;
  h->outv.ensure(static_cast<size_t>(4 * np + d + 1 + ntiles * (d + 1)) * 8);
  double* s2 = h->outv.as<double>();
  double *q = s2 + np, *rq = s2 + 2 * np, *beta = s2 + 3 * np;
  double* res = s2 + 4 * np;                                      // d + 1 traces
  double* partial = res + d + 1;

  GPB_CUDA(cudaMemcpyAsync(m.S2, K, static_cast<size_t>(np) * np * 8, cudaMemcpyDeviceToDevice, h->s0));
  scale_cols_kernel<<<static_cast<unsigned>(np), 256, 0, h->s0>>>(m.S2, m.ld, np, v.sW);   // K diag(sW)
  GPB_CUDA(cudaGetLastError());
  sweep_rows(h, m, m.t2, np);                                     // S2 = V = K W^1/2 L_B^-T
  chol_inverse_lower(h, m);                                       // B^-1 over L_B (S1 = U_B as scratch)
  h->lap.factored = false;                                        // a later predict / gradient factors B again
  tic(h, 2);
  gpc_grad_item_kernel<<<static_cast<unsigned>(np), 256, 0, h->s0>>>(s.link, v.y, v.f, n, K, np, m.S2, m.ld, np, s2);
  mirror_lower_kernel<<<static_cast<unsigned>(t64 * t64), 256, 0, h->s0>>>(m.A, m.ld, m.S2, m.ld, t64);   // B^-1, full
  scale_rows_cols_kernel<<<static_cast<unsigned>(np), 256, 0, h->s0>>>(m.S2, m.ld, np, v.sW);           // R
  GPB_CUDA(cudaGetLastError());
  launch_row_dot(K, np, 0, s2, 0, np, np, 0, q, 0, 1, h->s0);                   // q = K s2
  launch_row_dot(m.S2, m.ld, 0, q, 0, np, np, 0, rq, 0, 1, h->s0);              // R q
  gpc_grad_finish_kernel<<<static_cast<unsigned>((np + 255) / 256), 256, 0, h->s0>>>(v.a, s2, rq, np, beta);
  GPB_CUDA(cudaGetLastError());
  launch_laplace_grad_trace(m.S2, m.ld, v.a, beta, h->XsT.as<double>(), np, h->sq.as<double>(), pr.hyp2, n, d, partial, res,
                            h->s0);
  h->launches += 9;
  tic(h, 3);
  double* host = h->pinned((d + 1) * 8);
  GPB_CUDA(cudaMemcpyAsync(host, res, (d + 1) * 8, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  collect_timings(h, 3);
  *lml = s.lml;
  for (int k = 0; k <= d; ++k) grad[k] = -host[k];               // d lml / d theta_j = -1/2 tr(M dK/dtheta_j)
  h->state_epoch = h->ws_epoch;
  GPB_API_END
}

int gpb_pref_evidence(gpb_handle* h, double* evidence) {
  GPB_API_BEGIN
  GPB_REQUIRE(evidence, "null argument");
  LaplaceState& s = lap_state(h, LaplaceState::PREF);
  pref_factor_at_mode(h, s);
  *evidence = pref_evidence_value(s);
  h->state_epoch = h->ws_epoch;
  GPB_API_END
}

// Work space (laplace_mat): rows [0, np) L_G -> G^-1 | tile row | S1 [np+128, 2np+128) | S2 [2np+128, 3np+128).
//   S2 <- K^-1, swept through L_G:           V = K^-1 L_G^-T                      (n^3)
//   S1 <- I, swept (grow) and U U^T:         G^-1 in the lower tiles of [0, np)   (n^3/3 + n^3/3, chol_inverse_lower)
//   S1 <- K^-1, S1 -= V V^T (DMMA, lower):   A = K^-1 - K^-1 G^-1 K^-1            (n^3)
// then the per-pair / per-item kernels, v = G^-1 s2 (G^-1 mirrored into S2), u = K^-1 v, and the trace pass of grad.cu.
int gpb_pref_evidence_grad(gpb_handle* h, double* evidence, double* grad) {
  GPB_API_BEGIN
  GPB_REQUIRE(evidence && grad, "null argument");
  LaplaceState& s = lap_state(h, LaplaceState::PREF);
  if (s.grad_mode != 1) {
    h->state_epoch = h->ws_epoch;              // nothing was touched: the state stays usable
    throw Error{"the evidence gradient needs the mode of the accumulated-gradient Newton iteration: call "
                "gpb_pref_laplace with grad_mode = 1 (grad_mode = 0 does not stop at a stationary point)"};
  }
  tic(h, 0);
  pref_factor_at_mode(h, s);
  const double ev = pref_evidence_value(s);
  tic(h, 1);
  const int64_t n = s.n, np = h->n_pad, P = s.P;
  const int d = h->d, nt = static_cast<int>(np / TILE);
  LapMat m = laplace_mat(h, np);
  const double* iK = h->aux2.as<double>();
  const double* f = lap_vecs(h, LaplaceState::PREF).f;
  const int64_t t64 = np / 64, ntiles = t64 * (t64 + 1) / 2;
  h->outv.ensure(static_cast<size_t>(6 * np + 2 * PREF_PARTS + ntiles * (d + 1) + d + 2) * 8);
  double* alpha = h->outv.as<double>();
  double *s2 = alpha + np, *hv = alpha + 2 * np, *v = alpha + 3 * np, *u = alpha + 4 * np, *beta = alpha + 5 * np;
  double* part = alpha + 6 * np;
  double* res = part + 2 * PREF_PARTS;                            // [d + 1 traces, d log sigma]
  double* partial = res + d + 2;
  GPB_CUDA(cudaMemsetAsync(alpha, 0, static_cast<size_t>(6 * np) * 8, h->s0));

  GPB_CUDA(cudaMemcpyAsync(m.S2, iK, static_cast<size_t>(np) * np * 8, cudaMemcpyDeviceToDevice, h->s0));
  sweep_rows(h, m, m.t2, np);                                     // S2 = V = K^-1 L_G^-T
  chol_inverse_lower(h, m);                                       // G^-1 over L_G (S1 = U_G as scratch)
  s.factored = false;                                             // a later evidence / predict factors G again
  GPB_CUDA(cudaMemcpyAsync(m.S1, iK, static_cast<size_t>(np) * np * 8, cudaMemcpyDeviceToDevice, h->s0));
  {
    GemmArgs a{};                                                 // S1 -= V V^T on the lower tiles: A
    a.C = m.S1; a.ldc = m.ld; a.c_batch_stride = 0; a.rows_total = static_cast<int>(np);
    a.j0 = 0; a.j1 = nt; a.R = nt; a.tri = 1; a.i_off = 0;
    a.ka0 = 0; a.kb0 = 0; a.nk = static_cast<int>(np / GEMM_KB);
    a.a_row0 = a.b_row0 = m.t2 * TILE; a.epi = 1;
    dense_gemm(h, m.mapA, m.mapA, a);
  }
  tic(h, 2);
  launch_row_dot(iK, np, 0, f, 0, np, np, 0, alpha, 0, 1, h->s0);              // alpha = K^-1 f
  const double sq = 1.0 / (s.sigma * std::sqrt(2.0));
  pref_grad_pair_kernel<<<PREF_PARTS, 256, 0, h->s0>>>(s.pd.uvi, s.pd.y, P, f, sq, m.A, m.ld, s.pd.dk, s.pd.wk, part);
  pref_grad_item_kernel<<<static_cast<unsigned>((n + 127) / 128), 128, 0, h->s0>>>(n, s.pd.gr, s.pd.uvi, s.pd.dk,
                                                                                  s.pd.wk, s2, hv);
  mirror_lower_kernel<<<static_cast<unsigned>(t64 * t64), 256, 0, h->s0>>>(m.A, m.ld, m.S2, m.ld, t64);     // G^-1, full
  GPB_CUDA(cudaGetLastError());
  launch_row_dot(m.S2, m.ld, 0, s2, 0, np, np, 0, v, 0, 1, h->s0);              // v = G^-1 s2
  launch_row_dot(iK, np, 0, v, 0, np, np, 0, u, 0, 1, h->s0);                   // u = K^-1 v
  pref_grad_finish_kernel<<<1, 512, 0, h->s0>>>(np, alpha, u, v, hv, part, beta, res + d + 1);
  GPB_CUDA(cudaGetLastError());
  const KernelParams pr = lap_params(h, s.khyp.data(), s.eps);
  launch_laplace_grad_trace(m.S1, m.ld, alpha, beta, h->XsT.as<double>(), np, h->sq.as<double>(), pr.hyp2, n, d, partial, res,
                            h->s0);
  h->launches += 10;
  tic(h, 3);
  double* host = h->pinned((d + 2) * 8);
  GPB_CUDA(cudaMemcpyAsync(host, res, (d + 2) * 8, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  collect_timings(h, 3);
  *evidence = ev;
  for (int k = 0; k <= d; ++k) grad[k] = -host[k];               // d log Z / d theta_j = -1/2 tr(M dK/dtheta_j)
  grad[d + 1] = host[d + 1];
  h->state_epoch = h->ws_epoch;
  GPB_API_END
}

int gpb_pref_predict(gpb_handle* h, const double* Z, const double* Zb, int64_t mz, double* mean, double* var, double* prob) {
  GPB_API_BEGIN
  GPB_REQUIRE(Z && mean && var && mz > 0 && (prob || !Zb), "null argument");
  LaplaceState& s = lap_state(h, LaplaceState::PREF);
  pref_factor_at_mode(h, s);
  const int64_t np = h->n_pad;
  const int d = h->d;
  LapMat m = laplace_mat(h, np);
  const double* iK = h->aux2.as<double>();
  const LapVecs lv = lap_vecs(h, LaplaceState::PREF);
  double* alpha = lv.t;                                           // K^-1 f_hat
  launch_row_dot(iK, np, 0, lv.f, 0, np, np, 0, alpha, 0, 1, h->s0);
  ++h->launches;
  const KernelParams pr = lap_params(h, s.khyp.data(), s.eps);
  const double sf2 = s.khyp[d];
  // S1: R = k* rows (np rows available);  S2: T = R K^-1, then V = T L_G^-T
  TileMaps map_ik;
  make_tile_maps(&map_ik, iK, np, np, 1, np, np * np);
  const int64_t cap = np;
  h->outv.ensure(static_cast<size_t>(cap) * 8 * 5);
  double* o = h->outv.as<double>();                               // mean | var | prob | kss | q1
  h->Zd.ensure(static_cast<size_t>(cap) * d * 8 * 2);
  h->ZsT.ensure(static_cast<size_t>(d) * cap * 8 * 2);
  h->zsq.ensure(static_cast<size_t>(cap) * 8 * 2);
  double* zd = h->Zd.as<double>();
  double* zsT = h->ZsT.as<double>();
  double* zsq = h->zsq.as<double>();
  for (int64_t z0 = 0; z0 < mz; z0 += cap) {
    const int64_t mc = mz - z0 < cap ? mz - z0 : cap;
    const int64_t mp64 = round_up(mc, 64);
    test_cov_rows(h, Z + z0 * d, mc, pr, zd, zsT, zsq, m.S1, m.ld);
    if (Zb) {
      test_cov_rows(h, Zb + z0 * d, mc, pr, zd + cap * d, zsT + d * cap, zsq + cap, m.S2, m.ld);
      rows_sub_kernel<<<static_cast<unsigned>(mc), 256, 0, h->s0>>>(m.S1, m.S2, m.ld, np);      // rows of f(b) - f(a)
      ++h->launches;
    }
    pref_kss_kernel<<<static_cast<unsigned>((mc + 255) / 256), 256, 0, h->s0>>>(zsT, Zb ? zsT + d * cap : nullptr, mp64, d, mc,
                                                                                sf2, o + 3 * cap);
    launch_row_dot(m.S1, m.ld, 0, alpha, 0, mc, np, 0, o, 0, 1, h->s0);                      // mean = R K^-1 f
    {
      GemmArgs a{};                                               // T = R * iK^T (iK symmetric), 64-tiles
      a.C = m.S2; a.ldc = m.ld; a.c_batch_stride = 0; a.rows_total = static_cast<int>(mp64);
      a.j0 = 0; a.j1 = static_cast<int>(np / 64); a.R = static_cast<int>(mp64 / 64); a.tri = 0; a.i0 = 0;
      a.ka0 = 0; a.kb0 = 0; a.nk = static_cast<int>(np / GEMM_KB);
      a.a_row0 = m.t1 * TILE; a.b_row0 = 0; a.epi = 0;
      launch_dmma_gemm(m.mapA.m64, map_ik.m64, a, 1, h->s0, 64);
    }
    rows_dot2_kernel<<<static_cast<unsigned>(mc), 256, 0, h->s0>>>(m.S1, m.S2, m.ld, np, o + 4 * cap);   // q1 = R K^-1 R'
    GPB_CUDA(cudaGetLastError());
    h->launches += 4;
    sweep_rows(h, m, m.t2, mc);                                   // V = T L_G^-T
    pref_predict_finish_kernel<<<static_cast<unsigned>(mc), 256, 0, h->s0>>>(m.S2, m.ld, np, o + 3 * cap, o + 4 * cap, o,
                                                                            2.0 * s.sigma * s.sigma, o + cap,
                                                                            Zb ? o + 2 * cap : nullptr);
    GPB_CUDA(cudaGetLastError());
    ++h->launches;
    GPB_CUDA(cudaMemcpyAsync(mean + z0, o, mc * 8, cudaMemcpyDeviceToHost, h->s0));
    GPB_CUDA(cudaMemcpyAsync(var + z0, o + cap, mc * 8, cudaMemcpyDeviceToHost, h->s0));
    if (Zb) GPB_CUDA(cudaMemcpyAsync(prob + z0, o + 2 * cap, mc * 8, cudaMemcpyDeviceToHost, h->s0));
    GPB_CUDA(cudaStreamSynchronize(h->s0));
  }
  h->state_epoch = h->ws_epoch;
  GPB_API_END
}

}  // extern "C"
