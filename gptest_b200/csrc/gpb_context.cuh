// gpb_context.cuh - the handle behind the C ABI: device buffers, streams, tensor maps.
#pragma once
#include <vector>

#include "gpb_kernels.cuh"

namespace gpb {

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  void ensure(size_t want) {
    if (want <= bytes) return;
    release();
    GPB_CUDA(cudaMalloc(&p, want));
    bytes = want;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
  template <class T>
  T* as() const { return static_cast<T*>(p); }
  ~DevBuf() { release(); }
};

// A matrix being factored / swept: n_pad x n_pad symmetric part (lower triangle used) followed by
// extra rows (right-hand sides stored as rows, solved "for free" by the sweep).
struct FactorMat {
  double* A = nullptr;
  int64_t ld = 0;            // elements, = columns of the tensor map
  int64_t n_pad = 0;         // multiple of 128
  int64_t rows_total = 0;    // n_pad + number of extra rows
  int batch = 1;
  int64_t batch_stride = 0;  // elements
  double* Dinv = nullptr;    // per batch nt*128 x 128
  int64_t dinv_bs = 0;
  double* diag = nullptr;    // per batch n_pad
  int64_t diag_bs = 0;
  int* info = nullptr;       // per batch
  // optional right-hand side solved along with the factorisation without an appended row (GemmArgs::gemv_*):
  // rhs_r = 8 partial vectors per batch entry (partial g at + g * rhs_gs; the caller puts the right-hand side into
  // partial 0 and zeros into the others; all are overwritten), z <- L^-1 r
  double* rhs_r = nullptr;
  double* rhs_z = nullptr;
  int64_t rhs_bs = 0, rhs_gs = 0, rhs_zbs = 0;
  TileMaps mapA, mapD;
};

struct GrowState;    // grow.cu: factor of a growing training set

// The comparison graph of a preference fit on the device (CSR over the items, laplace.cu)
struct PrefGraphDev {
  const int64_t* row_ptr;      // n + 1
  const int32_t* other;        // per row: the other item of each incident pair, sorted by (other, pair)
  const int32_t* pair_by_other;
  const int32_t* is_u;         // 1: the row item is u (column 0) of that pair
  const int32_t* pair_sorted;  // per row: incident pairs in ascending pair order (diagonal cell)
  const int64_t* ku;           // last pair with u == i, or -1 (GPpref.py:77 last write wins)
  const int64_t* kv;           // last pair with v == i, or -1 (GPpref.py:78)
};

// device copy of the graph + pairs, carved out of one buffer (aux1)
struct PrefDev {
  PrefGraphDev gr;
  const int64_t* uvi;
  const double* y;
  double *dk, *wk;
};

// What the last Laplace fit of either kind left in the work space for its readers (predict, evidence, gradient).
// One per handle: a fit of one kind replaces the state of the other.
struct LaplaceState {
  enum Kind { NONE, PREF, GPC };
  Kind kind = NONE;
  int64_t n = 0;
  std::vector<double> khyp;    // [ell_1..ell_d, sf2]
  double eps = 0.0;            // jitter of the fit's K
  bool factored = false;       // the factor at the mode is in rows [0, n_pad) of the work space
  // classification: link, the lml gpb_gpc_laplace returned, and whether its loop ended on delta_f (not max_iter)
  int link = 0;
  double lml = 0.0;
  bool converged = false;
  // preference
  int64_t P = 0;
  double sigma = 1.0, lml_ref = 0.0, half_logdet_k = 0.0;
  double sum_log_g = 0.0;      // sum log diag chol(K^-1 + W) when factored
  int grad_mode = 0;
  PrefDev pd{};
};

}  // namespace gpb

struct gpb_handle {
  int device = 0;
  cudaStream_t s0 = nullptr;     // the handle's stream (all results are ordered on it)
  bool own_s0 = false;
  cudaStream_t s1 = nullptr;     // high-priority side stream for the look-ahead panel
  cudaStream_t s_loop = nullptr; // origin stream of the Laplace graph loops when s0 is the (uncapturable) legacy default stream
  std::vector<cudaStream_t> su;  // update streams of the chunked schedule (created on first use)
  std::string err;
  int64_t launches = 0;

  // options
  int lookahead = 1;
  int nb_tiles = 0;              // 0 = choose from the remaining matrix size (see chol.cu)
  int nb_switch8 = 96;           // > 0: blocks of 8 tiles (K = 1024) while at least this many tile columns remain
                                 // (N = 16384: 48.15 vs 48.5 ms with the chunked schedule, profiles/r01_dag_ab.json)
  int nb_switch4 = 64, nb_switch2 = 24;   // (round 2: 2-tile blocks down to 24 remaining columns - the faster panel chain hides behind K = 256 updates longer)
    // remaining tile columns from which the block is 4 / 2 tiles wide
  int64_t batch_chunk = 0;       // 0 = auto
  int batch_plain_width = 4;     // outer block width (tiles) of the plain-order sweep of a batch of small matrices
  int dag_streams = 4;           // > 0: while the block is 4 tiles wide, the trailing update is issued as column chunks
                                 // on this many streams, ordered by events only (see chol.cu); 0 = one launch per step
  int pdl_tail = 0;              // switch programmatic dependent launch on for the last pdl_max_tiles tile columns of a big sweep
  int pdl_max_tiles = 40;        // look-ahead sweeps of larger matrices launch without programmatic serialisation
  int chain_on_panel_stream = 1; // the update of the next panel's columns runs on the panel stream (chol.cu)
  int dag_min_width = 4;         // narrowest block (tiles) that still uses the chunked schedule
  int dag_big_tiles = 1;         // chunk updates keep the 128-row tiles although each launch is small
  int dag_min_tiles = 72;        // matrices with fewer tile columns keep the one-launch schedule
  int cov_kind = 0;              // covariance of the regression paths: 0 squared exponential (GPr.py:90-110), 1 Matern 3/2,
                                 // 2 Matern 5/2 (SURVEY 8f rank 4; the Laplace paths stay squared exponential)
  int la_max_batch = 1 << 30;    // batches up to this size use the look-ahead schedule and adaptive widths
                                 // (measured: N=16384 B=4 47.5 vs 50.2 ms/fit, N=4096 B=8 1.08 vs 1.20; 1024x2048 neutral)
  int split_tiles = 1;           // big launches: 1 = 128x64 CTAs, two per SM (finer grain: the look-ahead panel
                                 // kernels get SMs sooner, N=16384: 49.7 vs 52.4 ms); 0 = 128x128, one per SM
  int fuse_min_tiles = 72;       // single fits: the solve rides on the factorisation from this many tile columns on (api.cu)
  int fuse_rhs = 1;              // batched fits: forward substitution fused into the panel TRSM (no second pass over L)
  int tri_skip = 1;              // skip the zero half of the inverted diagonal tile in the panel TRSM and the warp tiles above
                                 // the diagonal in the symmetric updates (same results, fewer DMMAs)
  int64_t thin_tile_max = 74;    // panel TRSM / single-column update launches with at most this many 128-tiles use 32-row CTA-tiles
  int64_t trsm_tile_threshold = 1LL << 40;   // the panel TRSM's switch from 64 x 128 (two CTAs of 8 warps per SM) to 128 x 128 CTA-tiles (one):
                                             // never by default - 1024 x N=2048 sweep 109.3 -> 107.2 ms, single fits unchanged (tools/sweep_trsm_tiles.py)
  int batch_small_k = 512;              // batched updates with k up to this use 64 x 64 CTA-tiles regardless of the tile count
  int64_t small_tile_threshold = 2400;  // launches with fewer 128-tiles than this use 64-tiles (tuned: r01_tune_potrf.json)

  // training data (GPr.py:25-26 keeps trainInput / trainTarget on the object)
  int64_t n = 0, n_pad = 0;
  int d = 0;
  bool has_y = false;
  gpb::DevBuf X, y;

  // per-call work space
  gpb::DevBuf params;            // ell[d] | sf2, sn2   (per batch entry)
  gpb::DevBuf XsT, sq, ZsT, zsq, Zd;
  gpb::DevBuf A, Dinv, diag, info, scal, outv;
  gpb::DevBuf aux0, aux1, aux2;  // stage-specific (gradient / Laplace) scratch
  gpb::DevBuf trace;             // Laplace loops: (f_error, objective) per iteration, written on the device
  bool capturing = false;        // a Newton iteration is being captured into a graph: no allocation, no host sync
  double* h_pinned = nullptr;    // pinned staging for small H2D/D2H
  size_t h_pinned_bytes = 0;
  double* h_pinned_par = nullptr; // second pinned buffer: hyper-parameter uploads (never aliases the result staging above)
  size_t h_pinned_par_bytes = 0;

  std::vector<cudaEvent_t> ev_pool;   // ordering events for the look-ahead
  size_t ev_next = 0;
  cudaEvent_t tev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  float timings[8] = {0, 0, 0, 0, 0, 0, 0, 0};

  // The Laplace entry points leave their factor / mode in the shared work space for the predict calls; any other
  // call that uses the work space bumps ws_epoch, which invalidates that state (checked, never silent).
  gpb::LaplaceState lap;
  uint64_t ws_epoch = 0, state_epoch = ~0ull;

  gpb::GrowState* grow = nullptr;     // gpb_gpr_grow_* state (own buffers: other calls do not disturb it)

  cudaEvent_t next_event();
  void prepare_capture();        // creates everything a sweep may create lazily (event pool, update streams)
  double* pinned(size_t bytes);
  double* pinned_params(size_t bytes);
};

namespace gpb {

void make_tensor_map(CUtensorMap* map, const double* base, int64_t cols, int64_t rows, int64_t batch,
                     int64_t row_pitch_elems, int64_t batch_pitch_elems, int box_rows = TILE);
void make_tile_maps(TileMaps* maps, const double* base, int64_t cols, int64_t rows, int64_t batch,
                    int64_t row_pitch_elems, int64_t batch_pitch_elems);

// Blocked right-looking Cholesky sweep (see chol.cu).  factor == true: factor the symmetric part
// and carry the extra rows along; factor == false: the symmetric part already holds L (and Dinv
// its inverted diagonal tiles) and only the extra rows are swept (X <- X L^-T).
void chol_sweep(gpb_handle* h, FactorMat& m, bool factor);
struct SweepPlan {
  bool factor = true;      // factor the symmetric part (appended rows ride along)
  int extra_tile0 = -1;    // non-factor mode: first tile row swept (default: first row after the matrix)
  int extra_tiles = 0;     // non-factor mode: number of tile rows swept (default: all appended rows)
  bool grow = false;       // the swept block starts as the identity: tile row q is zero left of column q
};
void chol_sweep(gpb_handle* h, FactorMat& m, const SweepPlan& plan);

// K^-1 on the lower tiles of the symmetric part from its factor (grad.cu); needs the buffer layout
// rows [0,np) L | [np, np+128) appended tile row | [np+128, 2np+128) scratch for U = L^-T
void chol_inverse_lower(gpb_handle* h, FactorMat& m);

// out[j] = 1/2 tr((A - alpha b^T - b alpha^T) dK/dtheta_j), theta = [log l_1..log l_d, log sf] of the clipped squared
// exponential over the scaled points XsT / sq (grad.cu; one problem, A lower 64-tiles valid with full diagonal tiles,
// pitch ld = n_pad; hyp2[0] = sf2; partial: (ld/64)(ld/64 + 1)/2 x (d + 1) doubles).  Two launches.
void launch_laplace_grad_trace(const double* A, int64_t ld, const double* alpha, const double* beta, const double* XsT,
                               int64_t x_ld, const double* sq, const double* hyp2, int64_t n, int d, double* partial,
                               double* out, cudaStream_t st);

// A[i,j] -= sum_{k in tile columns [ka,kb)} A[i,k] A[j,k]^T for tile columns j in [c0,c1), rows i >= j (chol.cu)
void chol_trailing_update(gpb_handle* h, FactorMat& m, int c0, int c1, int ka, int kb);

void grow_release(gpb_handle* h);

// The work space of gpb_gpr_predict (api.cu), shared with the joint posterior (posterior.cu) so that both factor K and
// sweep the test rows with the same code: uploads khyp, marks tic(h, 0) and assembles K (lower tiles, identity
// padded) | y - mean | Kzx rows (mz of them, zero padded to 64) into h->A; the test points are scaled into ZsT / zsq
// with pitch round_up(mz, 64).  After chol_sweep(h, m, true): z = L^-1 (y - mean) and the rows at v are V = Kzx L^-T.
struct GprPredictRows {
  FactorMat m;
  double* z;
  double* v;
  const double* ell;     // device [ell_1..ell_d]
  const double* hyp2;    // device [sf2, sn2]
};
GprPredictRows gpr_predict_assemble(gpb_handle* h, const double* khyp, double mean, const double* Z, int64_t mz);

// fills m.mapA / m.mapD from the pointers and extents
void finalize_factor_mat(FactorMat& m);

// Stage timings of an entry point (gpb_get_timings): tic(h, i) marks the end of stage i - 1; collect_timings fills
// slots [0, last) with the stages and slot 4 with the total (only the total when per_stage is false), zeros elsewhere.
inline void tic(gpb_handle* h, int i) { GPB_CUDA(cudaEventRecord(h->tev[i], h->s0)); }
inline void collect_timings(gpb_handle* h, int last, bool per_stage = true) {
  for (int i = 0; i < 8; ++i) h->timings[i] = 0.f;
  if (per_stage)
    for (int i = 0; i < last; ++i) GPB_CUDA(cudaEventElapsedTime(&h->timings[i], h->tev[i], h->tev[i + 1]));
  GPB_CUDA(cudaEventElapsedTime(&h->timings[4], h->tev[0], h->tev[last]));
}

}  // namespace gpb

// Body of an extern "C" entry point that uses the work space: errors become the return code and h->err, and the
// call bumps ws_epoch (which invalidates the Laplace state unless the entry point re-arms it).
#define GPB_API_BEGIN                                       \
  if (!h) return -1;                                        \
  try {                                                     \
    GPB_CUDA(cudaSetDevice(h->device));                     \
    ++h->ws_epoch;
#define GPB_API_END                                         \
  }                                                         \
  catch (const gpb::Error& e) {                             \
    h->err = e.msg;                                         \
    return -2;                                              \
  }                                                         \
  catch (const std::exception& e) {                         \
    h->err = e.what();                                      \
    return -3;                                              \
  }                                                         \
  return 0;
