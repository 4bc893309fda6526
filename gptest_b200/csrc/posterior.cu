// posterior.cu - joint posterior covariance and posterior samples of GP regression (DESIGN.md section 4.8).
//
// The reference keeps only the diagonal of Kzx K^-1 Kxz (GPr.py:50).  Here the whole matrix
//   Sigma* = K(Z,Z) - V V^T,   V = Kzx L^-T,   L L^T = K
// is formed on the device, and joint draws f_s = fz + L* e_s with L* L*^T = Sigma* (+ jitter I):
//   1. K is factored with the Kzx rows riding along (gpb_gpr_predict's code, api.cu): V and fz   n^3/3 + n^2 m
//   2. lower tiles of Kzz (the assembly kernel, identity padded), then Sigma* = Kzz - V V^T in
//      one symmetric long-K launch of the DMMA kernel over the lower tiles                       n m^2
//   3. sampling: a copy of Sigma* + eps I is factored by the blocked Cholesky (the pristine
//      Sigma* stays, so a jitter retry costs one m^2 copy and m^3/3, not a new product)          m^3/3
//   4. E (Philox4x32-10 + Box-Muller, a pure function of (seed, sample, point)), D = E L*^T by
//      the DMMA kernel with the zero upper triangle of L* in place, samples = fz + D               2 S m^2
// The padding of V to whole 128-row tiles comes from the tensor map: rows past the last test row lie outside it and
// TMA fills them with zeros, so the padded part of Sigma* is the identity of the Kzz padding.
#include <cmath>

#include "../../include/gpb200.h"
#include "gpb_context.cuh"

namespace gpb {

namespace {

// Philox4x32-10 (Salmon et al., SC'11; the constants of Random123)
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
    const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}

// E[s][i], s < rows, i < ld (ld even): standard normals for s < nsamp and i < m, zeros elsewhere.  Pair p = i / 2 of
// sample s takes one Philox block, counter (p lo, p hi, s lo, s hi), key (seed lo, seed hi), and Box-Muller:
//   u1 = ((x0 | x1 << 32) >> 11) + 1) 2^-53 in (0, 1],  u2 = ((x2 | x3 << 32) >> 11) 2^-53,
//   e[2p] = sqrt(-2 ln u1) cos(2 pi u2),  e[2p + 1] = sqrt(-2 ln u1) sin(2 pi u2)
// (philox_normals in tests/_posterior_oracle restates it).  Nothing depends on the padding or the grid.
__global__ void __launch_bounds__(256) normal_philox_kernel(double* __restrict__ E, int64_t ld, int64_t m,
                                                            int64_t nsamp, int64_t rows, uint64_t seed) {
  const int64_t pairs = ld / 2, total = rows * pairs;
  const uint2 key = make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
  for (int64_t q = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; q < total;
       q += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t s = q / pairs, p = q - s * pairs, i = 2 * p;
    double2 e = make_double2(0.0, 0.0);
    if (s < nsamp && i < m) {
      const uint4 x = philox4x32_10(make_uint4(static_cast<uint32_t>(p), static_cast<uint32_t>(p >> 32),
                                               static_cast<uint32_t>(s), static_cast<uint32_t>(s >> 32)), key);
      const uint64_t a = (static_cast<uint64_t>(x.y) << 32) | x.x;
      const uint64_t b = (static_cast<uint64_t>(x.w) << 32) | x.z;
      const double u1 = static_cast<double>((a >> 11) + 1) * 0x1p-53;
      const double u2 = static_cast<double>(b >> 11) * 0x1p-53;
      const double r = sqrt(-2.0 * log(u1));
      const double t = (2.0 * 3.141592653589793) * u2;     // (2 pi) u2 rounded once, as numpy's 2 * np.pi * u2
      double sn, cs;
      sincos(t, &sn, &cs);
      e.x = r * cs;
      if (i + 1 < m) e.y = r * sn;
    }
    *reinterpret_cast<double2*>(E + s * ld + i) = e;
  }
}

// out[i][j] (pitch ldo), i, j < m, from the lower triangle of S (pitch lds): exactly symmetric.  32 x 32 tiles through
// shared memory, so that the mirrored half is read by rows too.
__global__ void __launch_bounds__(256) mirror_lower_kernel(const double* __restrict__ S, int64_t lds, int64_t m,
                                                           double* __restrict__ out, int64_t ldo) {
  __shared__ double t[32][33];
  const int64_t bi = blockIdx.y, bj = blockIdx.x;
  const bool upper = bi < bj;
  const int64_t si = upper ? bj : bi, sj = upper ? bi : bj;       // source tile (on or below the diagonal)
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int64_t i = si * 32 + r, j = sj * 32 + threadIdx.x;
    t[r][threadIdx.x] = (i < m && j < m) ? S[i * lds + j] : 0.0;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int64_t i = bi * 32 + r, j = bj * 32 + threadIdx.x;
    if (i >= m || j >= m) continue;
    const int c = threadIdx.x;
    double v;
    if (bi == bj) v = (r >= c) ? t[r][c] : t[c][r];
    else v = upper ? t[c][r] : t[r][c];
    out[i * ldo + j] = v;
  }
}

// F = lower triangle of S (strict upper zero, every tile), plus eps on the first m diagonal entries (not the padding)
__global__ void __launch_bounds__(256) jitter_copy_kernel(const double* __restrict__ S, double* __restrict__ F,
                                                          int64_t ld, int64_t m, double eps) {
  const int64_t total = ld * ld;
  for (int64_t q = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; q < total;
       q += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t i = q / ld, j = q - i * ld;
    double v = 0.0;
    if (i > j) v = S[q];
    else if (i == j) v = (i < m) ? S[q] + eps : S[q];
    F[q] = v;
  }
}

// the factorisation leaves the strict upper part of its diagonal tiles undefined: zero it (one CTA per tile)
__global__ void __launch_bounds__(256) zero_upper_diag_tiles_kernel(double* __restrict__ F, int64_t ld) {
  const int64_t k0 = static_cast<int64_t>(blockIdx.x) * TILE;
  for (int q = threadIdx.x; q < TILE * TILE; q += 256) {
    const int r = q / TILE, c = q % TILE;
    if (c > r) F[(k0 + r) * ld + k0 + c] = 0.0;
  }
}

// samples[s][i] = fz[i] + D[s][i] for s < nsamp, i < m (packed rows of m)
__global__ void __launch_bounds__(256) sample_finish_kernel(const double* __restrict__ D, int64_t ld,
                                                            const double* __restrict__ fz, int64_t m, int64_t nsamp,
                                                            double* __restrict__ out) {
  const int64_t total = nsamp * m;
  for (int64_t q = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; q < total;
       q += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t s = q / m, i = q - s * m;
    out[q] = fz[i] + D[s * ld + i];
  }
}

unsigned grid_for(int64_t work) {
  const int64_t g = (work + 255) / 256;
  return static_cast<unsigned>(g < 148 * 16 ? (g < 1 ? 1 : g) : 148 * 16);
}

struct JointPosterior {
  GprPredictRows r;
  int64_t mp;              // round_up(mz, 128): pitch and extent of Sigma* (h->aux1)
  double* sigma;
  const double* fz;        // device, mz (h->outv)
};

// Stages [0] - [2] of both entry points: fz (= gpb_gpr_predict's, same code) and Sigma* on the lower 128-tiles of
// h->aux1 (pitch mp; the strict upper halves of the diagonal tiles are not part of the result).
JointPosterior joint_posterior(gpb_handle* h, const double* khyp, double mean, const double* Z, int64_t mz, int32_t flags) {
  JointPosterior jp;
  jp.r = gpr_predict_assemble(h, khyp, mean, Z, mz);
  FactorMat& m = jp.r.m;
  const int64_t np = m.n_pad, mp = round_up(mz, TILE);
  jp.mp = mp;
  h->aux1.ensure(static_cast<size_t>(mp) * mp * 8);
  jp.sigma = h->aux1.as<double>();
  // test points again, with the pitch of Sigma* (the same scaling, so the same bits as in the Kzx rows)
  h->ZsT.ensure(static_cast<size_t>(h->d) * mp * 8);
  h->zsq.ensure(static_cast<size_t>(mp) * 8);
  const PointSet z{h->ZsT.as<double>(), mp, h->zsq.as<double>(), mz, mp};
  scale_points(h, z, h->Zd.as<double>(), h->d, jp.r.ell);
  // [sf2, 0]: Kzz of the latent f; [sf2, sn2] (flags bit0) for noisy observations
  const double* hyp_zz = jp.r.hyp2;
  if (!(flags & 1)) {
    h->scal.ensure(64);
    double* hz = h->scal.as<double>();
    GPB_CUDA(cudaMemcpyAsync(hz, jp.r.hyp2, 8, cudaMemcpyDeviceToDevice, h->s0));
    GPB_CUDA(cudaMemsetAsync(hz + 1, 0, 8, h->s0));
    hyp_zz = hz;
  }
  // the distance of a point to itself is exactly 0 (se_prep and the tile kernel share the dot-product chain), so
  // the diagonal is exactly sf2 (+ sn2), the sf2 predict_finish_kernel subtracts from
  build_cov(h, z, z, h->d, 1, h->cov_kind, 0, hyp_zz, jp.sigma, mp);
  tic(h, 1);
  chol_sweep(h, m, true);
  double* outv = h->outv.as<double>();
  launch_predict_finish(jp.r.v, m.ld, jp.r.z, np, mz, jp.r.hyp2, outv, outv + mz, h->s0);
  ++h->launches;
  jp.fz = outv;
  tic(h, 2);
  {
    // Sigma* = Kzz - V V^T on the lower tiles: the symmetric long-K product of chol_inverse_lower (grad.cu) over the
    // whole k range, both operands the V rows of the work space
    const int mt = static_cast<int>(mp / TILE);
    GemmArgs a{};
    a.C = jp.sigma; a.ldc = mp; a.c_batch_stride = 0; a.rows_total = static_cast<int>(mp);
    a.j0 = 0; a.j1 = mt; a.R = mt; a.tri = 1; a.i_off = 0;
    a.a_row0 = a.b_row0 = static_cast<int>(np + 1);
    a.ka0 = a.kb0 = 0; a.nk = static_cast<int>(np / GEMM_KB); a.k_from_row = 0; a.epi = 1;
    dense_gemm(h, m.mapA, m.mapA, a);
    ++h->launches;
  }
  return jp;
}

}  // namespace

}  // namespace gpb

using namespace gpb;

extern "C" {

int gpb_gpr_predict_full(gpb_handle* h, const double* khyp, double mean, const double* Z, int64_t mz,
                         double* fz, double* cov, int32_t cov_is_dev, int32_t flags, int32_t* info) {
  GPB_API_BEGIN
  GPB_REQUIRE(h->n > 0 && h->has_y, "no training data with targets: call gpb_set_train first");
  GPB_REQUIRE(khyp && Z && fz && cov && mz > 0, "null argument");
  JointPosterior jp = joint_posterior(h, khyp, mean, Z, mz, flags);
  tic(h, 3);
  double* dst = cov;
  if (!cov_is_dev) {
    h->aux2.ensure(static_cast<size_t>(mz) * mz * 8);
    dst = h->aux2.as<double>();
  }
  const unsigned tb = static_cast<unsigned>((mz + 31) / 32);
  mirror_lower_kernel<<<dim3(tb, tb), dim3(32, 8), 0, h->s0>>>(jp.sigma, jp.mp, mz, dst, mz);
  GPB_CUDA(cudaGetLastError());
  ++h->launches;
  if (!cov_is_dev) GPB_CUDA(cudaMemcpyAsync(cov, dst, static_cast<size_t>(mz) * mz * 8, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaMemcpyAsync(fz, jp.fz, mz * 8, cudaMemcpyDeviceToHost, h->s0));
  tic(h, 4);
  const int k_info = read_info(h, jp.r.m.info);
  if (info) *info = k_info;
  collect_timings(h, 4);
  h->timings[3] = 0.f;                     // the mirror and the copy-out count in the total only
  GPB_API_END
}

int gpb_gpr_sample(gpb_handle* h, const double* khyp, double mean, const double* Z, int64_t mz, int64_t nsamp,
                   uint64_t seed, int32_t flags, double* samples, double* jitter, int32_t* info) {
  GPB_API_BEGIN
  GPB_REQUIRE(h->n > 0 && h->has_y, "no training data with targets: call gpb_set_train first");
  GPB_REQUIRE(khyp && Z && samples && mz > 0 && nsamp > 0, "null argument");
  if (info) *info = 0;
  if (jitter) *jitter = 0.0;
  JointPosterior jp = joint_posterior(h, khyp, mean, Z, mz, flags);
  tic(h, 3);
  const int k_info = read_info(h, jp.r.m.info);
  if (k_info > 0) {
    if (info) *info = k_info;
    tic(h, 4);
    GPB_CUDA(cudaStreamSynchronize(h->s0));
    collect_timings(h, 4);
    return 0;
  }
  const int64_t mp = jp.mp, sp = round_up(nsamp, TILE);
  // the factor of Sigma* + eps I: its own buffer (h->aux2), the inverted diagonal tiles and pivots of K's are done with
  h->aux2.ensure(static_cast<size_t>(mp) * mp * 8);
  FactorMat f = factor_workspace(h, 1, mp, mp, mp, mp, true, h->aux2.as<double>());
  // jitter policy: 0, then 1e-12 sf2, 1e-11 sf2, ... up to sf2
  static constexpr double kScale[14] = {0.0, 1e-12, 1e-11, 1e-10, 1e-9, 1e-8, 1e-7, 1e-6, 1e-5, 1e-4, 1e-3, 1e-2, 1e-1, 1.0};
  const double sf2 = khyp[h->d];
  double eps = 0.0;
  for (int k = 0;; ++k) {
    if (k == 14) throw Error{"the posterior covariance is not positive definite with a jitter of sf2"};
    eps = kScale[k] * sf2;
    if (k > 0) GPB_CUDA(cudaMemsetAsync(f.info, 0, 4, h->s0));
    jitter_copy_kernel<<<grid_for(mp * mp), 256, 0, h->s0>>>(jp.sigma, f.A, mp, mz, eps);
    GPB_CUDA(cudaGetLastError());
    ++h->launches;
    chol_sweep(h, f, true);
    if (read_info(h, f.info) == 0) break;
  }
  zero_upper_diag_tiles_kernel<<<static_cast<unsigned>(mp / TILE), 256, 0, h->s0>>>(f.A, mp);
  GPB_CUDA(cudaGetLastError());
  // E (sp x mp, zero padded) and D = E L*^T in h->aux0; the samples are packed over E once D is done
  h->aux0.ensure(static_cast<size_t>(2 * sp) * mp * 8);
  double* E = h->aux0.as<double>();
  double* D = E + sp * mp;
  normal_philox_kernel<<<grid_for(sp * mp / 2), 256, 0, h->s0>>>(E, mp, mz, nsamp, sp, seed);
  GPB_CUDA(cudaGetLastError());
  h->launches += 3;
  {
    TileMaps me;
    make_tile_maps(&me, E, mp, sp, 1, mp, sp * mp);
    GemmArgs a{};
    a.C = D; a.ldc = mp; a.c_batch_stride = 0; a.rows_total = static_cast<int>(sp);
    a.j0 = 0; a.j1 = static_cast<int>(mp / TILE); a.R = static_cast<int>(sp / TILE); a.tri = 0; a.i0 = 0;
    a.ka0 = a.kb0 = 0; a.nk = static_cast<int>(mp / GEMM_KB); a.a_row0 = a.b_row0 = 0; a.epi = 0;
    dense_gemm(h, me, f.mapA, a);
  }
  sample_finish_kernel<<<grid_for(nsamp * mz), 256, 0, h->s0>>>(D, mp, jp.fz, mz, nsamp, E);
  GPB_CUDA(cudaGetLastError());
  ++h->launches;
  GPB_CUDA(cudaMemcpyAsync(samples, E, static_cast<size_t>(nsamp) * mz * 8, cudaMemcpyDeviceToHost, h->s0));
  tic(h, 4);
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  if (jitter) *jitter = eps;
  collect_timings(h, 4);
  GPB_API_END
}

}  // extern "C"
