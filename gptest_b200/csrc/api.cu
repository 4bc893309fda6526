// api.cu - the extern "C" boundary (include/gpb200.h): lifecycle, training data, covariance
// assembly, regression likelihood / prediction, dense factorisation hooks.
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "../../include/gpb200.h"
#include "gpb_context.cuh"

using namespace gpb;

static std::string g_create_error;

cudaEvent_t gpb_handle::next_event() {
  if (ev_pool.empty()) {
    ev_pool.resize(256);
    for (auto& e : ev_pool) GPB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  cudaEvent_t e = ev_pool[ev_next];
  ev_next = (ev_next + 1) % ev_pool.size();
  return e;
}

void gpb_handle::prepare_capture() {
  if (ev_pool.empty()) { next_event(); ev_next = 0; }
  while (static_cast<int>(su.size()) < dag_streams) {
    cudaStream_t st;
    GPB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    su.push_back(st);
  }
}

double* gpb_handle::pinned(size_t bytes) {
  if (bytes > h_pinned_bytes) {
    if (h_pinned) cudaFreeHost(h_pinned);
    h_pinned = nullptr;
    size_t want = bytes < 4096 ? 4096 : bytes;
    GPB_CUDA(cudaMallocHost(reinterpret_cast<void**>(&h_pinned), want));
    h_pinned_bytes = want;
  }
  return h_pinned;
}

double* gpb_handle::pinned_params(size_t bytes) {
  if (bytes > h_pinned_par_bytes) {
    if (h_pinned_par) cudaFreeHost(h_pinned_par);
    h_pinned_par = nullptr;
    size_t want = bytes < 4096 ? 4096 : bytes;
    GPB_CUDA(cudaMallocHost(reinterpret_cast<void**>(&h_pinned_par), want));
    h_pinned_par_bytes = want;
  }
  return h_pinned_par;
}

namespace {

// upload [ell_1..ell_d] and [sf2, sn2] for `batch` problems; returns device pointers
struct Params {
  const double* ell;   // batch x d
  const double* hyp2;  // batch x 2
};
Params upload_params(gpb_handle* h, const double* khyp, int64_t batch, int d, bool has_sn2) {
  const int stride = d + (has_sn2 ? 2 : 1);
  const size_t cnt = static_cast<size_t>(batch) * (d + 2);
  // a pinned buffer of its own: the result staging of the same call (pinned()) never overwrites it, and every entry
  // point synchronises before it returns, so the copy below needs no synchronisation of its own (round 1 blocked here)
  double* host = h->pinned_params(cnt * 8);
  for (int64_t b = 0; b < batch; ++b) {
    for (int k = 0; k < d; ++k) host[b * d + k] = khyp[b * stride + k];
    host[batch * d + 2 * b] = khyp[b * stride + d];
    host[batch * d + 2 * b + 1] = has_sn2 ? khyp[b * stride + d + 1] : 0.0;
  }
  h->params.ensure(cnt * 8);
  GPB_CUDA(cudaMemcpyAsync(h->params.p, host, cnt * 8, cudaMemcpyHostToDevice, h->s0));
  return Params{h->params.as<double>(), h->params.as<double>() + batch * d};
}

// scaled training points for `batch` problems
void prep_train(gpb_handle* h, const Params& pr, int batch) {
  const int64_t np = h->n_pad;
  h->XsT.ensure(static_cast<size_t>(batch) * h->d * np * 8);
  h->sq.ensure(static_cast<size_t>(batch) * np * 8);
  launch_se_prep(h->X.as<double>(), h->n, h->d, pr.ell, h->XsT.as<double>(), np, h->sq.as<double>(), batch,
                 h->d, static_cast<int64_t>(h->d) * np, np, h->s0);
  ++h->launches;
}

// K (lower tiles, identity padded) into the symmetric part of m
void build_k_into(gpb_handle* h, FactorMat& m, const Params& pr, int mode, int clip) {
  SeArgs a{};
  a.kind = h->cov_kind;
  a.rT = a.cT = h->XsT.as<double>();
  a.r_ld = a.c_ld = h->n_pad;
  a.r_sq = a.c_sq = h->sq.as<double>();
  a.n_rows_valid = a.n_cols_valid = h->n;
  a.xs_batch_stride = static_cast<int64_t>(h->d) * h->n_pad;
  a.sq_batch_stride = h->n_pad;
  a.d = h->d;
  a.out = m.A; a.ld = m.ld; a.out_batch_stride = m.batch_stride;
  a.rows_pad = a.cols_pad = h->n_pad;
  a.hyp_dev = pr.hyp2;
  a.mode = mode;
  a.clip = clip;
  launch_se_build(a, m.batch, h->s0);
  ++h->launches;
}

// work space for factoring `batch` matrices of h->n_pad with `extra_rows` appended rows each
FactorMat alloc_factor(gpb_handle* h, int batch, int64_t extra_rows_alloc, int64_t extra_rows) {
  FactorMat m;
  const int64_t np = h->n_pad;
  m.ld = np;
  m.n_pad = np;
  m.rows_total = np + extra_rows;
  m.batch = batch;
  m.batch_stride = (np + extra_rows_alloc) * np;
  h->A.ensure(static_cast<size_t>(batch) * m.batch_stride * 8);
  m.A = h->A.as<double>();
  m.dinv_bs = np * TILE;
  h->Dinv.ensure(static_cast<size_t>(batch) * m.dinv_bs * 8);
  m.Dinv = h->Dinv.as<double>();
  m.diag_bs = np;
  h->diag.ensure(static_cast<size_t>(batch) * np * 8);
  m.diag = h->diag.as<double>();
  h->info.ensure(static_cast<size_t>(batch) * 4);
  m.info = h->info.as<int>();
  GPB_CUDA(cudaMemsetAsync(m.info, 0, static_cast<size_t>(batch) * 4, h->s0));
  finalize_factor_mat(m);
  return m;
}

void require_train(gpb_handle* h, bool need_y) {
  GPB_REQUIRE(h->n > 0, "no training data: call gpb_set_train first");
  if (need_y) GPB_REQUIRE(h->has_y, "training targets were not given to gpb_set_train");
}

void set_train_common(gpb_handle* h, const double* X, int64_t n, int32_t d, const double* y, cudaMemcpyKind kind) {
  GPB_REQUIRE(X != nullptr && n > 0 && d > 0, "X must be n x d with n, d > 0");
  h->n = n;
  h->d = d;
  h->n_pad = round_up(n, TILE);
  h->X.ensure(static_cast<size_t>(n) * d * 8);
  GPB_CUDA(cudaMemcpyAsync(h->X.p, X, static_cast<size_t>(n) * d * 8, kind, h->s0));
  h->has_y = (y != nullptr);
  h->y.ensure(static_cast<size_t>(h->n_pad) * 8);
  GPB_CUDA(cudaMemsetAsync(h->y.p, 0, static_cast<size_t>(h->n_pad) * 8, h->s0));
  if (y) GPB_CUDA(cudaMemcpyAsync(h->y.p, y, static_cast<size_t>(n) * 8, kind, h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));     // caller may free / change X, y after return
}

// scaled test points into ZsT / zsq (pitch = m_pad)
void prep_test(gpb_handle* h, const Params& pr, const double* Z, int64_t m, int64_t m_pad) {
  h->Zd.ensure(static_cast<size_t>(m) * h->d * 8);
  GPB_CUDA(cudaMemcpyAsync(h->Zd.p, Z, static_cast<size_t>(m) * h->d * 8, cudaMemcpyHostToDevice, h->s0));
  h->ZsT.ensure(static_cast<size_t>(h->d) * m_pad * 8);
  h->zsq.ensure(static_cast<size_t>(m_pad) * 8);
  launch_se_prep(h->Zd.as<double>(), m, h->d, pr.ell, h->ZsT.as<double>(), m_pad, h->zsq.as<double>(), 1, 0, 0, 0, h->s0);
  ++h->launches;
}

}  // namespace

namespace gpb {

GprPredictRows gpr_predict_assemble(gpb_handle* h, const double* khyp, double mean, const double* Z, int64_t mz) {
  Params pr = upload_params(h, khyp, 1, h->d, true);
  const int64_t np = h->n_pad, mp64 = round_up(mz, 64);
  GprPredictRows r;
  FactorMat& m = r.m;
  m = alloc_factor(h, 1, 1 + mp64, 1 + mz);
  h->outv.ensure(static_cast<size_t>(2 * mz) * 8);
  tic(h, 0);
  prep_train(h, pr, 1);
  prep_test(h, pr, Z, mz, mp64);
  build_k_into(h, m, pr, 1, 0);
  r.z = m.A + np * m.ld;
  r.v = m.A + (np + 1) * m.ld;
  r.ell = pr.ell;
  r.hyp2 = pr.hyp2;
  launch_copy_sub_mean(r.z, h->y.as<double>(), h->n, mean, h->s0);
  ++h->launches;
  if (np > h->n) GPB_CUDA(cudaMemsetAsync(r.z + h->n, 0, (np - h->n) * 8, h->s0));
  {
    // Kzx rows (GPr.py:46,49) appended below the y row
    SeArgs a{};
    a.kind = h->cov_kind;
    a.rT = h->ZsT.as<double>(); a.r_ld = mp64; a.r_sq = h->zsq.as<double>(); a.n_rows_valid = mz;
    a.cT = h->XsT.as<double>(); a.c_ld = np; a.c_sq = h->sq.as<double>(); a.n_cols_valid = h->n;
    a.d = h->d; a.out = r.v; a.ld = m.ld; a.rows_pad = mp64; a.cols_pad = np;
    a.hyp_dev = pr.hyp2; a.mode = 2; a.clip = 0;
    launch_se_build(a, 1, h->s0);
    ++h->launches;
  }
  return r;
}

}  // namespace gpb

extern "C" {

int gpb_version(void) { return 100; }

int gpb_create(int device, gpb_handle** out) {
  if (!out) return -1;
  *out = nullptr;
  gpb_handle* h = nullptr;
  try {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
      throw Error{std::string("no CUDA device available (libgpb200 has no CPU fallback): ") + cudaGetErrorString(e)};
    GPB_REQUIRE(device >= 0 && device < count, "device index out of range");
    GPB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    GPB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
      throw Error{"libgpb200 is built for sm_100a (B200) only; device is sm_" + std::to_string(prop.major) +
                  std::to_string(prop.minor)};
    h = new gpb_handle();
    h->device = device;
    int lo = 0, hi = 0;
    GPB_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    GPB_CUDA(cudaStreamCreateWithPriority(&h->s0, cudaStreamNonBlocking, lo));
    h->own_s0 = true;
    GPB_CUDA(cudaStreamCreateWithPriority(&h->s1, cudaStreamNonBlocking, hi));
    for (auto& e2 : h->tev) GPB_CUDA(cudaEventCreate(&e2));
    dmma_gemm_init();
    tile_potrf_init();
  } catch (const gpb::Error& e) {
    g_create_error = e.msg;
    gpb_destroy(h);               // releases whatever streams / events were created before the failure
    return -2;
  } catch (const std::exception& e) {
    g_create_error = e.what();
    gpb_destroy(h);
    return -3;
  }
  *out = h;
  return 0;
}

int gpb_set_stream(gpb_handle* h, void* stream) {
  GPB_API_BEGIN
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  if (h->own_s0) cudaStreamDestroy(h->s0);
  h->own_s0 = false;
  h->s0 = static_cast<cudaStream_t>(stream);
  GPB_API_END
}

void* gpb_get_stream(gpb_handle* h) { return h ? static_cast<void*>(h->s0) : nullptr; }

int gpb_destroy(gpb_handle* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  if (h->own_s0 && h->s0) cudaStreamDestroy(h->s0);
  if (h->s1) cudaStreamDestroy(h->s1);
  if (h->s_loop) cudaStreamDestroy(h->s_loop);
  for (auto s : h->su) cudaStreamDestroy(s);
  for (auto e : h->ev_pool) cudaEventDestroy(e);
  for (auto e : h->tev) if (e) cudaEventDestroy(e);
  if (h->h_pinned) cudaFreeHost(h->h_pinned);
  if (h->h_pinned_par) cudaFreeHost(h->h_pinned_par);
  gpb::grow_release(h);
  delete h;
  return 0;
}

const char* gpb_last_error(gpb_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int gpb_set_option(gpb_handle* h, const char* name, int64_t value) {
  if (!h || !name) return -1;
  if (!strcmp(name, "lookahead")) h->lookahead = value != 0;
  else if (!strcmp(name, "nb_tiles")) h->nb_tiles = static_cast<int>(value < 0 ? 0 : (value > 8 ? 8 : value));
  else if (!strcmp(name, "batch_chunk")) h->batch_chunk = value;
  else if (!strcmp(name, "batch_plain_width")) h->batch_plain_width = static_cast<int>(value < 1 ? 1 : (value > 8 ? 8 : value));
  else if (!strcmp(name, "small_tile_threshold")) h->small_tile_threshold = value;
  else if (!strcmp(name, "thin_tile_max")) h->thin_tile_max = value;
  else if (!strcmp(name, "trsm_tile_threshold")) h->trsm_tile_threshold = value;
  else if (!strcmp(name, "batch_small_k")) h->batch_small_k = static_cast<int>(value);
  else if (!strcmp(name, "tri_skip")) h->tri_skip = value != 0;
  else if (!strcmp(name, "fuse_rhs")) h->fuse_rhs = value != 0;
  else if (!strcmp(name, "fuse_min_tiles")) h->fuse_min_tiles = static_cast<int>(value);
  else if (!strcmp(name, "split_tiles")) h->split_tiles = value != 0;
  else if (!strcmp(name, "persistent_waves")) dmma_gemm_set_persistent(static_cast<int>(value));
  else if (!strcmp(name, "stagger")) dmma_gemm_set_stagger(static_cast<int>(value));
  else if (!strcmp(name, "pdl")) dmma_gemm_set_pdl(static_cast<int>(value));
  else if (!strcmp(name, "fine_warps")) dmma_gemm_set_fine_warps(static_cast<int>(value));
  else if (!strcmp(name, "trsm_balance")) dmma_gemm_set_trsm_balance(static_cast<int>(value));
  else if (!strcmp(name, "trsm_persist")) dmma_gemm_set_trsm_persist(static_cast<int>(value));
  else if (!strcmp(name, "potrf_variant")) tile_potrf_set_variant(static_cast<int>(value));
  else if (!strcmp(name, "potrf_refine")) tile_potrf_set_refine(static_cast<int>(value));
  else if (!strcmp(name, "dag_streams")) h->dag_streams = static_cast<int>(value < 0 ? 0 : (value > 16 ? 16 : value));
  else if (!strcmp(name, "dag_min_tiles")) h->dag_min_tiles = static_cast<int>(value);
  else if (!strcmp(name, "dag_big_tiles")) h->dag_big_tiles = static_cast<int>(value);
  else if (!strcmp(name, "chain_on_panel_stream")) h->chain_on_panel_stream = static_cast<int>(value);
  else if (!strcmp(name, "pdl_max_tiles")) h->pdl_max_tiles = static_cast<int>(value);
  else if (!strcmp(name, "pdl_tail")) h->pdl_tail = value != 0;
  else if (!strcmp(name, "dag_min_width")) h->dag_min_width = static_cast<int>(value < 1 ? 1 : value);
  else if (!strcmp(name, "nb_switch4")) h->nb_switch4 = static_cast<int>(value);
  else if (!strcmp(name, "nb_switch2")) h->nb_switch2 = static_cast<int>(value);
  else if (!strcmp(name, "nb_switch8")) h->nb_switch8 = static_cast<int>(value);
  else if (!strcmp(name, "la_max_batch")) h->la_max_batch = static_cast<int>(value);
  else if (!strcmp(name, "cov_kind")) {
    if (value < 0 || value > 2) return -4;
    h->cov_kind = static_cast<int>(value);
  }
  else { h->err = std::string("unknown option ") + name; return -1; }
  return 0;
}

int gpb_get_timings(gpb_handle* h, float* ms, int n) {
  if (!h || !ms) return -1;
  for (int i = 0; i < n && i < 8; ++i) ms[i] = h->timings[i];
  return 0;
}

int64_t gpb_launch_count(gpb_handle* h) { return h ? h->launches : -1; }

int gpb_set_train(gpb_handle* h, const double* X, int64_t n, int32_t d, const double* y) {
  GPB_API_BEGIN
  set_train_common(h, X, n, d, y, cudaMemcpyHostToDevice);
  GPB_API_END
}

int gpb_set_train_dev(gpb_handle* h, const double* X, int64_t n, int32_t d, const double* y) {
  GPB_API_BEGIN
  set_train_common(h, X, n, d, y, cudaMemcpyDeviceToDevice);
  GPB_API_END
}

int gpb_se_ard_kxx(gpb_handle* h, const double* khyp, double* K_out, int32_t out_is_dev, int32_t flags) {
  GPB_API_BEGIN
  require_train(h, false);
  GPB_REQUIRE(khyp && K_out, "null argument");
  Params pr = upload_params(h, khyp, 1, h->d, true);
  tic(h, 0);
  prep_train(h, pr, 1);
  const int64_t n = h->n, np64 = round_up(n, 64);
  // full symmetric matrix, written straight into the caller's n x n layout when n % 64 == 0
  double* dst;
  int64_t ld;
  const bool direct = out_is_dev && (n % 64 == 0);
  if (direct) { dst = K_out; ld = n; }
  else { h->A.ensure(static_cast<size_t>(np64) * np64 * 8); dst = h->A.as<double>(); ld = np64; }
  SeArgs a{};
  a.kind = h->cov_kind;
  a.rT = a.cT = h->XsT.as<double>(); a.r_ld = a.c_ld = h->n_pad;
  a.r_sq = a.c_sq = h->sq.as<double>();
  a.n_rows_valid = a.n_cols_valid = n; a.d = h->d;
  a.out = dst; a.ld = ld; a.rows_pad = a.cols_pad = np64;
  a.hyp_dev = pr.hyp2; a.mode = 0; a.clip = flags & 1;
  launch_se_build(a, 1, h->s0);
  ++h->launches;
  tic(h, 1);
  if (!direct) {
    GPB_CUDA(cudaMemcpy2DAsync(K_out, n * 8, dst, ld * 8, n * 8, n,
                               out_is_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->s0));
  }
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  collect_timings(h, 1);
  GPB_API_END
}

static int kxz_common(gpb_handle* h, const double* khyp, const double* Z, int64_t m, double* Kxz_out,
                      int32_t out_is_dev, int mode) {
  GPB_API_BEGIN
  require_train(h, false);
  GPB_REQUIRE(khyp && Z && Kxz_out && m > 0, "null argument");
  Params pr = upload_params(h, khyp, 1, h->d, true);
  prep_train(h, pr, 1);
  const int64_t n = h->n, np64 = round_up(n, 64), mp64 = round_up(m, 64);
  prep_test(h, pr, Z, m, mp64);
  h->A.ensure(static_cast<size_t>(np64) * mp64 * 8);
  SeArgs a{};
  a.kind = h->cov_kind;
  a.rT = h->XsT.as<double>(); a.r_ld = h->n_pad; a.r_sq = h->sq.as<double>(); a.n_rows_valid = n;
  a.cT = h->ZsT.as<double>(); a.c_ld = mp64; a.c_sq = h->zsq.as<double>(); a.n_cols_valid = m;
  a.d = h->d; a.out = h->A.as<double>(); a.ld = mp64; a.rows_pad = np64; a.cols_pad = mp64;
  a.hyp_dev = pr.hyp2; a.mode = mode; a.clip = 0;
  launch_se_build(a, 1, h->s0);
  ++h->launches;
  GPB_CUDA(cudaMemcpy2DAsync(Kxz_out, m * 8, h->A.p, mp64 * 8, m * 8, n,
                             out_is_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  GPB_API_END
}

int gpb_se_ard_kxz(gpb_handle* h, const double* khyp, const double* Z, int64_t m, double* Kxz_out, int32_t out_is_dev) {
  return kxz_common(h, khyp, Z, m, Kxz_out, out_is_dev, 2);
}

int gpb_sqdist(gpb_handle* h, const double* B, int64_t m, double* out) {
  if (!h) return -1;
  std::vector<double> khyp(static_cast<size_t>(h->d) + 2, 1.0);    // unit length scales: raw distances
  return kxz_common(h, khyp.data(), B, m, out, 0, 3);
}

int gpb_gpr_nlml(gpb_handle* h, const double* khyp, double mean, double* nlml, double* grad, int32_t* info) {
  GPB_API_BEGIN
  require_train(h, true);
  GPB_REQUIRE(khyp && nlml, "null argument");
  if (grad) return gpb_gpr_nlml_batched(h, khyp, 1, mean, nlml, grad, info);
  Params pr = upload_params(h, khyp, 1, h->d, true);
  const int64_t np = h->n_pad;
  // The solve L z = y - m rides on the factorisation.  Round 1 appended y as a row under K: one row of data, but a
  // whole 128-row tile in every panel TRSM and every update (0.8 % of the work at N = 16384).  Now (fuse_rhs) the
  // diagonal-tile kernel solves tile k of it and the panel TRSM takes its columns out of the rows below (DESIGN 4.6).
  // ... from fuse_min_tiles tile columns on: the z_k step and the epilogue of the panel TRSM lengthen the chain of panel
  // kernels by ~2.5 us per tile column, an appended row does not (its tiles run beside the others), so below N ~ 9000,
  // where the chain is a visible part of the run time, the row wins (N = 2048: 0.703 vs 0.753 ms, 4096: 1.79 vs 1.83,
  // 8192: 7.56 vs 7.57, 16384: 47.2 vs 46.6)
  const bool fuse = h->fuse_rhs != 0 && tile_potrf_fuses_rhs() && np / TILE >= h->fuse_min_tiles;
  FactorMat m = fuse ? alloc_factor(h, 1, 0, 0) : alloc_factor(h, 1, 1, 1);
  h->scal.ensure(64);
  double* zrow = m.A + np * m.ld;
  tic(h, 0);
  prep_train(h, pr, 1);
  build_k_into(h, m, pr, 1, 0);
  if (fuse) {
    h->aux0.ensure(static_cast<size_t>(np) * 8 * 9);
    double* rv = h->aux0.as<double>();                                             // 8 partial right-hand sides, then z
    zrow = rv + 8 * np;
    GPB_CUDA(cudaMemsetAsync(rv, 0, static_cast<size_t>(np) * 8 * 8, h->s0));
    launch_copy_sub_mean(rv, h->y.as<double>(), h->n, mean, h->s0);               // partial 0 <- y - m  (GPr.py:64-65)
    ++h->launches;
    m.rhs_r = rv; m.rhs_bs = 8 * np; m.rhs_gs = np; m.rhs_z = zrow; m.rhs_zbs = np;
  } else {
    launch_copy_sub_mean(zrow, h->y.as<double>(), h->n, mean, h->s0);
    ++h->launches;
    if (np > h->n) GPB_CUDA(cudaMemsetAsync(zrow + h->n, 0, (np - h->n) * 8, h->s0));
  }
  tic(h, 1);
  chol_sweep(h, m, true);
  tic(h, 2);
  launch_nlml_finish(zrow, 0, m.diag, 0, np, h->n, h->scal.as<double>(), 1, h->s0);
  ++h->launches;
  tic(h, 3);
  double* host = h->pinned(64);
  GPB_CUDA(cudaMemcpyAsync(host, h->scal.p, 8, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaMemcpyAsync(host + 1, m.info, 4, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  *nlml = host[0];
  if (info) *info = *reinterpret_cast<int*>(host + 1);
  collect_timings(h, 3);
  GPB_API_END
}

int gpb_gpr_predict(gpb_handle* h, const double* khyp, double mean, const double* Z, int64_t mz,
                    double* fz, double* cov, int32_t* info) {
  GPB_API_BEGIN
  require_train(h, true);
  GPB_REQUIRE(khyp && Z && fz && cov && mz > 0, "null argument");
  GprPredictRows r = gpr_predict_assemble(h, khyp, mean, Z, mz);
  FactorMat& m = r.m;
  tic(h, 1);
  chol_sweep(h, m, true);
  tic(h, 2);
  double* outv = h->outv.as<double>();
  launch_predict_finish(r.v, m.ld, r.z, m.n_pad, mz, r.hyp2, outv, outv + mz, h->s0);
  ++h->launches;
  tic(h, 3);
  double* host = h->pinned(64);
  GPB_CUDA(cudaMemcpyAsync(fz, outv, mz * 8, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaMemcpyAsync(cov, outv + mz, mz * 8, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaMemcpyAsync(host, m.info, 4, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  if (info) *info = *reinterpret_cast<int*>(host);
  collect_timings(h, 3);
  GPB_API_END
}

int gpb_potrf_lower_dev(gpb_handle* h, double* A_dev, int64_t n, int64_t lda, int32_t* info) {
  GPB_API_BEGIN
  GPB_REQUIRE(A_dev && n > 0 && n % TILE == 0 && lda >= n, "potrf_lower_dev: n must be a positive multiple of 128, lda >= n");
  FactorMat m;
  m.A = A_dev; m.ld = lda; m.n_pad = n; m.rows_total = n; m.batch = 1; m.batch_stride = n * lda;
  m.dinv_bs = n * TILE;
  h->Dinv.ensure(static_cast<size_t>(m.dinv_bs) * 8);
  m.Dinv = h->Dinv.as<double>();
  h->diag.ensure(static_cast<size_t>(n) * 8);
  m.diag = h->diag.as<double>(); m.diag_bs = n;
  h->info.ensure(4);
  m.info = h->info.as<int>();
  GPB_CUDA(cudaMemsetAsync(m.info, 0, 4, h->s0));
  finalize_factor_mat(m);
  // the tensor map addresses columns [0, lda): restrict to the matrix itself
  make_tile_maps(&m.mapA, m.A, n, n, 1, lda, n * lda);
  tic(h, 0);
  tic(h, 1);
  chol_sweep(h, m, true);
  tic(h, 2);
  double* host = h->pinned(64);
  GPB_CUDA(cudaMemcpyAsync(host, m.info, 4, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  if (info) *info = *reinterpret_cast<int*>(host);
  collect_timings(h, 2);
  GPB_API_END
}

int gpb_potrf_lower(gpb_handle* h, double* A, int64_t n, int32_t* info) {
  GPB_API_BEGIN
  GPB_REQUIRE(A && n > 0, "potrf_lower: null argument");
  const int64_t np = round_up(n, TILE);
  h->aux0.ensure(static_cast<size_t>(np) * np * 8);
  double* d = h->aux0.as<double>();
  GPB_CUDA(cudaMemsetAsync(d, 0, static_cast<size_t>(np) * np * 8, h->s0));
  GPB_CUDA(cudaMemcpy2DAsync(d, np * 8, A, n * 8, n * 8, n, cudaMemcpyHostToDevice, h->s0));
  if (np > n) {   // identity padding: unit diagonal
    std::vector<double> ones(np - n, 1.0);
    GPB_CUDA(cudaMemcpy2DAsync(d + n * np + n, (np + 1) * 8, ones.data(), 8, 8, np - n, cudaMemcpyHostToDevice, h->s0));
    GPB_CUDA(cudaStreamSynchronize(h->s0));
  }
  int rc = gpb_potrf_lower_dev(h, d, np, np, info);
  if (rc) return rc;
  GPB_CUDA(cudaMemcpy2DAsync(A, n * 8, d, np * 8, n * 8, n, cudaMemcpyDeviceToHost, h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  for (int64_t i = 0; i < n; ++i)
    for (int64_t j = i + 1; j < n; ++j) A[i * n + j] = 0.0;   // numpy returns a clean lower factor
  GPB_API_END
}

int gpb_dgemm_nt_dev(gpb_handle* h, double* C, int64_t ldc, const double* A, int64_t lda, const double* B,
                     int64_t ldb, int64_t M, int64_t N, int64_t K, double alpha, double beta) {
  GPB_API_BEGIN
  GPB_REQUIRE(C && A && B, "null argument");
  GPB_REQUIRE(M % TILE == 0 && N % TILE == 0 && K % TILE == 0 && M > 0 && N > 0 && K > 0, "M, N, K must be positive multiples of 128");
  int epi;
  if (alpha == 1.0 && beta == 0.0) epi = 0;
  else if (alpha == -1.0 && beta == 1.0) epi = 1;
  else if (alpha == 0.0 && beta == 0.0) epi = 2;      // measurement only: k loop without the epilogue stores
  else throw Error{"dgemm_nt_dev supports (alpha,beta) = (1,0) or (-1,1)"};
  TileMaps ma, mb;
  make_tile_maps(&ma, A, K, M, 1, lda, M * lda);
  make_tile_maps(&mb, B, K, N, 1, ldb, N * ldb);
  GemmArgs a{};
  a.C = C; a.ldc = ldc; a.c_batch_stride = 0; a.rows_total = static_cast<int>(M);
  a.j0 = 0; a.j1 = static_cast<int>(N / TILE); a.R = static_cast<int>(M / TILE); a.tri = 0; a.i0 = 0;
  a.ka0 = 0; a.kb0 = 0; a.nk = static_cast<int>(K / GEMM_KB); a.b_row0 = 0; a.epi = epi;
  if (h->split_tiles) launch_dmma_gemm(ma.m128, mb.m64, a, 1, h->s0, 12864);
  else launch_dmma_gemm(ma.m128, mb.m128, a, 1, h->s0, 128);
  ++h->launches;
  GPB_API_END
}

int gpb_microbench(gpb_handle* h, int32_t kind, double* tflops) {
  GPB_API_BEGIN
  GPB_REQUIRE(tflops, "null argument");
  h->scal.ensure(64);
  launch_microbench(kind, h->scal.as<double>(), h->s0);   // warm-up
  GPB_CUDA(cudaEventRecord(h->tev[0], h->s0));
  double flops = 0;
  for (int i = 0; i < 3; ++i) flops += launch_microbench(kind, h->scal.as<double>(), h->s0);
  GPB_CUDA(cudaEventRecord(h->tev[1], h->s0));
  GPB_CUDA(cudaStreamSynchronize(h->s0));
  float ms = 0;
  GPB_CUDA(cudaEventElapsedTime(&ms, h->tev[0], h->tev[1]));
  *tflops = flops / (ms * 1e-3) / 1e12;
  h->launches += 4;
  GPB_API_END
}

}  // extern "C"
