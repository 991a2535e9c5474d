// C ABI of libgpdla.so (see include/gpdla.h).  Host-side runtime: context, device workspaces,
// batching of quasars, kernel dispatch.  No CPU compute path exists in this library.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <map>
#include <mutex>
#include <numeric>
#include <random>
#include <string>
#include <vector>

#include "../../include/gpdla.h"
#include "gpdla_kernels.cuh"
#include "gpdla_i8_kernels.cuh"
#include "gpdla_preload.cuh"
#include "gpdla_objective.cuh"
#include "gpdla_training.cuh"
#include "gpdla_statistics.cuh"
#include "gpdla_reconstruct.cuh"
#include "gpdla_rest_table.h"

using namespace gpdla;
static_assert(RT_DEG == RT_DEG_DEV, "host builder and device lookup must agree on the table's polynomial degree");

// ---------------------------------------------------------------------------- Lyman series data
// Physical data of the hydrogen Lyman series, members 1..31 (the same atomic data the reference
// tabulates at voigt.c:31-134): wavelength (cm), oscillator strength, transition rate (1/s).
namespace {
struct LymanLine { double wavelength_cm, f, Gamma; };
const LymanLine kLyman[MAX_LINES] = {
    {1.2156701e-05, 0.416400, 6.265e+08},  {1.0257223e-05, 0.079120, 1.897e+08},
    {9.725368e-06, 0.029000, 8.127e+07},   {9.497431e-06, 0.013940, 4.204e+07},
    {9.378035e-06, 0.007799, 2.450e+07},   {9.307483e-06, 0.004814, 1.236e+07},
    {9.262257e-06, 0.003183, 8.255e+06},   {9.231504e-06, 0.002216, 5.785e+06},
    {9.209631e-06, 0.001605, 4.210e+06},   {9.193514e-06, 0.00120, 3.160e+06},
    {9.181294e-06, 0.000921, 2.432e+06},   {9.171806e-06, 0.0007226, 1.911e+06},
    {9.16429e-06, 0.000577, 1.529e+06},    {9.15824e-06, 0.000469, 1.243e+06},
    {9.15329e-06, 0.000386, 1.024e+06},    {9.14919e-06, 0.000321, 8.533e+05},
    {9.14576e-06, 0.000270, 7.186e+05},    {9.14286e-06, 0.000230, 6.109e+05},
    {9.14039e-06, 0.000197, 5.237e+05},    {9.13826e-06, 0.000170, 4.523e+05},
    {9.13641e-06, 0.000148, 3.933e+05},    {9.13480e-06, 0.000129, 3.443e+05},
    {9.13339e-06, 0.000114, 3.030e+05},    {9.13215e-06, 0.000101, 2.679e+05},
    {9.13104e-06, 0.000089, 2.382e+05},    {9.13006e-06, 0.000080, 2.127e+05},
    {9.12918e-06, 0.000071, 1.907e+05},    {9.12839e-06, 0.000064, 1.716e+05},
    {9.12768e-06, 0.000058, 1.550e+05},    {9.12703e-06, 0.000053, 1.405e+05},
    {9.12645e-06, 0.000048, 1.277e+05}};
const double kC = 2.99792458e+10;               // speed of light, cm/s           voigt.c:22
const double kE = 4.803204672997660e-10;        // elementary charge, statC       voigt.c:27
const double kMe = 9.10938356e-28;              // electron mass, g               voigt.c:25
const double kSigma = 9.08537121627923800e+05;  // Gaussian width b/sqrt2, cm/s   voigt.c:41
// BOSS instrument profile, R = 2000, 1e-4 dex pixels, +-3 pixels             voigt.c:242-251
const double kInstrument[7] = {2.17460992138080811e-03, 4.11623059580451742e-02, 2.40309364651846963e-01,
                               4.32707438937454059e-01, 2.40309364651846963e-01, 4.11623059580451742e-02,
                               2.17460992138080811e-03};

void fill_line_constants(LineConstants* lc) {
  for (int i = 0; i < MAX_LINES; ++i) {
    lc->tw[i] = kLyman[i].wavelength_cm;
    // voigt.c:141-143: M_PI * e * e * oscillator_strength * transition_wavelength / (m_e * c)
    lc->lc[i] = M_PI * kE * kE * kLyman[i].f * kLyman[i].wavelength_cm / (kMe * kC);
    // voigt.c:186: Gamma * transition_wavelength / (4 * M_PI)
    lc->gam[i] = kLyman[i].Gamma * kLyman[i].wavelength_cm / (4 * M_PI);
    lc->y[i] = lc->gam[i] / sqrt(2.0) / kSigma;
    lc->y2[i] = lc->y[i] * lc->y[i];
    lc->kcore[i] = lc->lc[i] / (sqrt(2.0 * M_PI) * kSigma);
    lc->kwing[i] = lc->kcore[i] * lc->y[i] / sqrt(M_PI);
  }
  for (int i = 0; i < 7; ++i) lc->ip[i] = kInstrument[i];
  lc->c = kC;
  lc->inv_s2s = 1.0 / (sqrt(2.0) * kSigma);
}

// Lyman-series forest data of the multi-DLA mean-flux suppression: the one table both inference (c_forest) and the
// mean-flux training set (TrainingArgs::forest) read
void fill_forest_constants(ForestConstants* fc, int num_forest_lines) {
  fc->num_forest_lines = num_forest_lines;                // set_parameters_multi.m:76
  fc->prev_beta = 3.65;                                   // ...meanflux.m:37
  const double prev_tau_0 = 0.0023;                       // ...meanflux.m:36
  const double lya_wavelength = 1215.6701, lya_oscillator_strength = 0.416400;
  for (int l = 0; l < MAX_LINES; ++l) fc->wavelength[l] = kLyman[l].wavelength_cm * 1e8;   // set_parameters_multi.m:77-109
  for (int l = 0; l < MAX_LINES; ++l) {
    // tau_0 * lambda_l * f_l / (lambda_1 * f_1) without the tau_0                         ...meanflux.m:255-256
    fc->tau_ratio[l] = fc->wavelength[l] * kLyman[l].f / (fc->wavelength[0] * kLyman[0].f);
    // prev_tau_0 * f_l / f_lya * lambda_l / lya_wavelength                               ...meanflux.m:271-273
    fc->kim_tau[l] = prev_tau_0 * kLyman[l].f / lya_oscillator_strength * fc->wavelength[l] / lya_wavelength;
  }
}

thread_local std::string g_err;   // errors of the context-free entry points

#define CUDA_TRY(expr, errstr)                                                              \
  do {                                                                                      \
    cudaError_t e__ = (expr);                                                               \
    if (e__ != cudaSuccess) {                                                               \
      char buf__[512];                                                                      \
      snprintf(buf__, sizeof buf__, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
      (errstr) = buf__;                                                                     \
      return GPDLA_ERR_CUDA;                                                                \
    }                                                                                       \
  } while (0)

// Every entry point runs on its context's device and leaves the caller's current device as it found it.
struct DeviceGuard {
  int prev = -1;
  cudaError_t status = cudaSuccess;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) status = cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};

// Per-device library state (constant memory, function attributes, occupancy), shared by all contexts of the process
// and guarded by one mutex per device: contexts on several GPUs may be driven from several host threads.
constexpr int MAX_DEVICES = 64;
struct DeviceState {
  std::mutex mu;
  bool constants = false;                    // c_lines, c_forest, c_wing3, stage-index tables uploaded
  std::map<const void*, size_t> smem;        // kernel -> configured dynamic shared memory
  std::map<const void*, int> clusters;       // persistent kernel -> resident clusters
};
DeviceState g_dev[MAX_DEVICES];

// accumulator column -> augmented-triangle index of the epilogue staging area, for rank K
template <int K>
static void fill_stage_index(short* tab) {
  using G = GramShape<K>;
  for (int c = 0; c < G::NCOL; ++c) tab[c] = -1;
  for (int p = 0; p < K; ++p) {
    for (int q = p; q < K; ++q) tab[G::pair_index(p, q)] = (short)aug_index<K>(p, q);
    tab[G::WT * 8 + p] = (short)aug_index<K>(p, K);
  }
}
// INT8 path: accumulator column (CTA rank, n) -> augmented-triangle index (the same for every digit count)
template <int K>
static void fill_i8_stage_index(short* tab) {
  using Sh = i8::Shape<K, 6>;
  using G = GramShape<K>;
  for (int i = 0; i < i8::CLUSTER * 128; ++i) tab[i] = -1;
  for (int p = 0; p < K; ++p) {
    for (int q = p; q < K; ++q) {
      const int c = G::pair_index(p, q);
      tab[(c / Sh::WCOLS) * 128 + c % Sh::WCOLS] = (short)aug_index<K>(p, q);
    }
    tab[i8::WCTAS * 128 + p] = (short)aug_index<K>(p, K);
  }
}

// Compile-time proof that the column blocks of the INT8 path tile the Gram exactly: every pair column and every projection
// column of GramShape<K> is the image of exactly one (block, n), and the blocks beyond the producing cluster's three come in
// whole cluster passes of the contract-only kernel.
template <int K>
constexpr bool i8_blocks_tile_the_gram() {
  using Sh = i8::Shape<K, 6>;
  using G = GramShape<K>;
  int hits[G::NCOL] = {};
  for (int slot = 0; slot < Sh::NSLOT; ++slot)
    for (int n = 0; n < Sh::NMAX; ++n) {
      const int c = Sh::gram_column(slot, n);
      if (c >= G::NCOL) return false;
      if (c >= 0) hits[c]++;
    }
  for (int c = 0; c < G::NCOL; ++c) {
    const bool wanted = c < G::NPAIR || (c >= G::WT * 8 && c < G::WT * 8 + K);
    if (hits[c] != (wanted ? 1 : 0)) return false;
  }
  return (Sh::WBLOCKS - i8::WCTAS) % i8::CLUSTER == 0 && Sh::CPASSES * i8::CLUSTER + i8::WCTAS == Sh::WBLOCKS;
}
static_assert(i8_blocks_tile_the_gram<20>() && i8_blocks_tile_the_gram<40>(), "INT8 column blocks must tile the Gram columns");
static_assert(!i8::Shape<20, 6>::EXT && i8::Shape<40, 6>::EXT && i8::Shape<40, 6>::WBLOCKS == 11 && i8::Shape<40, 6>::CPASSES == 2, "column-block plan");

constexpr int I8_K = 20;   // rank whose INT8 tensor-core Gram fits one cluster's TMEM (shared-memory Cholesky epilogue)
constexpr int I8_K_EXT = 40;   // rank whose Gram columns take contract-only passes as well (i8::Shape::EXT)
// (rank, digits) combinations of the INT8 path compiled into the library
#define GPDLA_FOR_I8(k, digits, CALL)                                                    \
  if ((k) == I8_K && (digits) == 5) { constexpr int K = I8_K, L = 5; (void)K; (void)L; CALL; }        \
  else if ((k) == I8_K) { constexpr int K = I8_K, L = 6; (void)K; (void)L; CALL; }                   \
  else if ((k) == I8_K_EXT) { constexpr int K = I8_K_EXT, L = 6; (void)K; (void)L; CALL; }
constexpr int ORDER_GROUP = 0;   // 0: samples fully sorted by redshift (measured best: 63.5 ms per 296 quasars against 69.9 with
                                 // scattered groups of 4 and 64.7 with scattered groups of 32, DESIGN.md 4.4)

// Constant memory of the current device, once per device.
int upload_device_constants(std::string& err) {
  int dev = -1;
  CUDA_TRY(cudaGetDevice(&dev), err);
  if (dev < 0 || dev >= MAX_DEVICES) { err = "device index out of range"; return GPDLA_ERR_CUDA; }
  std::lock_guard<std::mutex> lock(g_dev[dev].mu);
  if (g_dev[dev].constants) return GPDLA_OK;
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, dev), err);
  if (prop.major != 10) {
    err = "libgpdla.so is built for sm_100a (B200) only; device is sm_" + std::to_string(prop.major) +
          std::to_string(prop.minor);
    return GPDLA_ERR_CUDA;
  }
  LineConstants lc;
  fill_line_constants(&lc);
  CUDA_TRY(cudaMemcpyToSymbol(c_lines, &lc, sizeof lc), err);
  {  // Lyman-series forest data of the multi-DLA mean-flux suppression
    ForestConstants fc;
    fill_forest_constants(&fc, MAX_LINES);
    CUDA_TRY(cudaMemcpyToSymbol(c_forest, &fc, sizeof fc), err);
  }
  {  // three-line wing tables in velocity units (see tau_sum_3_wing)
    const double wa[GPDLA_VOIGT_DEG_A + 1] = GPDLA_VOIGT_WING_A;
    const double wb[GPDLA_VOIGT_DEG_B + 1] = GPDLA_VOIGT_WING_B;
    const double two_s2 = 2.0 * kSigma * kSigma;   // u = two_s2 * q
    Wing3 w3;
    for (int j = 0; j < 3; ++j) {
      double sc = two_s2 * lc.kwing[j];
      for (int i = 0; i <= GPDLA_VOIGT_DEG_A; ++i) { w3.a[j][i] = sc * wa[i]; sc *= two_s2; }
      w3.yy[j] = two_s2 * lc.kwing[j] * lc.y2[j] * two_s2 * wb[0];
    }
    w3.b1 = wb[1] / wb[0] * two_s2;
    w3.v2min = GPDLA_VOIGT_X0 * GPDLA_VOIGT_X0 * two_s2;
    CUDA_TRY(cudaMemcpyToSymbol(c_wing3, &w3, sizeof w3), err);
  }
  {  // 2^(j/256) for exp_nonpos, correctly rounded from long double
    double t[256];
    for (int j = 0; j < 256; ++j) t[j] = (double)exp2l((long double)j / 256.0L);
    CUDA_TRY(cudaMemcpyToSymbol(g_exp2_tab, t, sizeof t), err);
  }
  {  // stage-index tables of every compiled rank (one table per rank: contexts of different k share a device)
    static short t10[GramShape<10>::NCOL], t20[GramShape<20>::NCOL], t40[GramShape<40>::NCOL], ti8[i8::CLUSTER * 128];
    fill_stage_index<10>(t10); fill_stage_index<20>(t20); fill_stage_index<40>(t40); fill_i8_stage_index<I8_K>(ti8);
    CUDA_TRY(cudaMemcpyToSymbol(c_stage_index_10, t10, sizeof t10), err);
    CUDA_TRY(cudaMemcpyToSymbol(c_stage_index_20, t20, sizeof t20), err);
    CUDA_TRY(cudaMemcpyToSymbol(c_stage_index_40, t40, sizeof t40), err);
    CUDA_TRY(cudaMemcpyToSymbol(i8::c_i8_stage, ti8, sizeof ti8), err);
  }
  g_dev[dev].constants = true;
  return GPDLA_OK;
}

// dynamic shared memory opt-in of a kernel on the current context's device, once per (device, kernel, size)
template <class Kern>
static int configure_smem(int dev, Kern kern, size_t smem, std::string& err) {
  std::lock_guard<std::mutex> lock(g_dev[dev].mu);
  size_t& have = g_dev[dev].smem[(const void*)kern];
  if (have < smem) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), err);
    have = smem;
  }
  return GPDLA_OK;
}

// rank dispatch: the ranks compiled into the library
#define GPDLA_FOR_RANK(k, CALL)            \
  switch (k) {                             \
    case 10: { constexpr int K = 10, NSPLIT = 1; (void)NSPLIT; CALL; } break; \
    case 20: { constexpr int K = 20, NSPLIT = 1; (void)NSPLIT; CALL; } break; \
    case 40: { constexpr int K = 40, NSPLIT = 4; (void)NSPLIT; CALL; } break; \
    default: break;                        \
  }
static bool rank_supported(int k) { return k == 10 || k == 20 || k == 40; }
static size_t gram_doubles_per_chunk_all_splits(int k) {
  size_t r = 0;
  GPDLA_FOR_RANK(k, (r = (size_t)SplitShape<K, NSPLIT>::CHUNK_DOUBLES * NSPLIT));
  return r;
}
static int rank_splits(int k) { int r = 1; GPDLA_FOR_RANK(k, r = NSPLIT); return r; }
static int rank_ncol(int k) { int r = 0; GPDLA_FOR_RANK(k, r = GramShape<K>::NCOL); return r; }

template <class T>
int dev_upload(T** dst, const T* src, size_t n, std::string& err) {
  if (*dst) { cudaFree(*dst); *dst = nullptr; }
  CUDA_TRY(cudaMalloc(dst, std::max<size_t>(n, 1) * sizeof(T)), err);
  CUDA_TRY(cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice), err);
  return GPDLA_OK;
}
}  // namespace

struct gpdla_ctx {
  int device = 0;
  std::string err;
  uint64_t launches = 0;
  gpdla_params params;
  // null model
  double *d_rest = nullptr, *d_mu = nullptr, *d_M = nullptr, *d_log_omega = nullptr;
  int n_rest = 0, k = 0;
  double c_0 = 0, tau_0 = 0, beta = 0;
  // DLA samples; d_order = sample indices in ascending redshift offset (the order the kernels walk them in)
  double *d_offset = nullptr, *d_log_nhi = nullptr, *d_nhi = nullptr;
  int32_t* d_order = nullptr;
  int64_t S = 0;
  // rest-frame table of tau / N (gpdla_rest_table.h), rebuilt when num_lines / pixel_spacing change
  double* d_rt = nullptr;
  int rt_ncell = 0, rt_num_lines = 0;
  double rt_pixel_spacing = 0, rt_h = 0;
  // prior catalogue
  double* d_prior_z = nullptr;
  uint8_t* d_prior_dla = nullptr;
  int64_t n_prior = -1;
  // per-batch workspace
  int ws_batch = 0, ws_npix = 0, ws_k = 0;
  int64_t ws_S = 0;
  double *d_gram = nullptr, *d_qld = nullptr;   // column-split ranks: global accumulator staging
  QuasarMeta* d_meta = nullptr;
  double *d_lam = nullptr, *d_lamh = nullptr, *d_pix = nullptr, *d_Mq = nullptr, *d_P = nullptr, *d_sll = nullptr,
         *d_scratch = nullptr;
  int64_t* d_scratch_i = nullptr;
  // INT8 tensor-core Gram path (k = 20): digit operands and scales
  int i8_batch = 0, i8_npix = 0, i8_k = 0;
  int64_t i8_S = 0;
  uint8_t* d_adig = nullptr;          // k = 40: stored W'' digit tiles (i8::Shape::EXT)
  double *d_pix2 = nullptr, *d_pix8 = nullptr, *d_colscale = nullptr, *d_colinv = nullptr;
  uint8_t* d_bop = nullptr;
  int* d_status = nullptr;
  int32_t* d_f64flag = nullptr;       // [batch] flags + {count, list}: quasars the INT8 path leaves to the FP64 kernels
  unsigned long long* d_phase = nullptr;   // GPDLA_I8_PHASES diagnostics
  // staging for the host entry point
  size_t st_bytes = 0;
  void* d_stage = nullptr;
  cudaStream_t stream = nullptr, copy_stream = nullptr;   // the host entries' own (non-default) streams
  cudaStream_t side_stream = nullptr;                     // FP64 kernels running beside the INT8 kernel (f64_share)
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaEvent_t ev_batch[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
  // multi-DLA path
  double* d_lls_nhi = nullptr;
  int64_t lls_S = 0;
  double Z_lls = 0, Z_dla = 0;
  double* d_uniforms = nullptr;       // [3 x S] rand stream of rng('default')
  int mws_batch = 0, mws_npix = 0;
  int64_t mws_S = 0;
  double *d_acache = nullptr, *d_msll = nullptr, *d_mlls = nullptr, *d_cum = nullptr, *d_mscal = nullptr;
  int32_t *d_partners = nullptr, *d_active = nullptr;
  // optional per-kernel timing of the dominant kernel (bench.py's roofline)
  bool profiling = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
};

// Gram arithmetic of this context: digits of the INT8 path (k = 20), 0 = FP64 DMMA kernels
static int i8_digits(const gpdla_ctx* c) {
  int d = c->params.gram_digits;
  if (d == 0) d = 6;
  if (c->k == I8_K_EXT && (d == 5 || d == 6)) return 6;   // k = 40: six digits only
  return (c->k == I8_K && (d == 5 || d == 6)) ? d : 0;
}
// rows of the global accumulator staging per quasar: the S samples + the null-model slot, in whole 128-sample tiles
static int64_t gram_rows(const gpdla_ctx* c) { return ((int64_t)c->S + 1 + i8::TM - 1) / i8::TM * i8::TM; }
static bool use_i8(const gpdla_ctx* c) { return i8_digits(c) > 0; }

static void free_workspace(gpdla_ctx* c) {
  cudaFree(c->d_meta); cudaFree(c->d_lam); cudaFree(c->d_lamh); cudaFree(c->d_pix); cudaFree(c->d_Mq); cudaFree(c->d_P);
  cudaFree(c->d_sll); cudaFree(c->d_scratch); cudaFree(c->d_scratch_i); cudaFree(c->d_gram); cudaFree(c->d_qld);
  c->d_gram = c->d_qld = nullptr;
  c->d_meta = nullptr; c->d_lam = c->d_lamh = c->d_pix = c->d_Mq = c->d_P = c->d_sll = c->d_scratch = nullptr;
  c->d_scratch_i = nullptr;
  c->ws_batch = c->ws_npix = c->ws_k = 0; c->ws_S = 0;
}

static int ensure_workspace(gpdla_ctx* c, int batch, int npix) {
  if (c->ws_batch >= batch && c->ws_npix == npix && c->ws_k == c->k && c->ws_S == c->S) return GPDLA_OK;
  free_workspace(c);
  const size_t B = batch;
  CUDA_TRY(cudaMalloc(&c->d_meta, B * sizeof(QuasarMeta)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_lam, B * (npix + 8) * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_lamh, B * (npix + 8) * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_pix, B * npix * 4 * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_Mq, B * npix * c->k * sizeof(double)), c->err);
  // FP64 Gram operand: the FP64 path's, and the INT8 path's fallback for quasars with zero-noise-variance pixels
  CUDA_TRY(cudaMalloc(&c->d_P, B * (npix / KC) * gram_doubles_per_chunk_all_splits(c->k) * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_sll, B * c->S * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_scratch, B * 16 * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_scratch_i, B * sizeof(int64_t)), c->err);
  if (rank_splits(c->k) > 1) {
    const size_t rows = (size_t)gram_rows(c);
    CUDA_TRY(cudaMalloc(&c->d_gram, B * rows * rank_ncol(c->k) * sizeof(double)), c->err);
    CUDA_TRY(cudaMalloc(&c->d_qld, B * rows * 2 * sizeof(double)), c->err);
  }
  c->ws_batch = batch; c->ws_npix = npix; c->ws_k = c->k; c->ws_S = c->S;
  return GPDLA_OK;
}

// The rest-frame table of tau / N for the context's line count and pixel spacing (built on the host in long double,
// ~10 ms for three lines; gpdla_params.rest_table = -1 disables it: direct evaluation everywhere).
static int ensure_rest_table(gpdla_ctx* c) {
  if (c->params.rest_table < 0) return GPDLA_OK;
  if (c->d_rt && c->rt_num_lines == c->params.num_lines && c->rt_pixel_spacing == c->params.pixel_spacing) return GPDLA_OK;
  LineConstants lc;
  fill_line_constants(&lc);
  const RestTableHost t = build_rest_table(c->params.num_lines, c->params.pixel_spacing, RT_NEAR_PIXELS, lc.tw, lc.lc,
                                           lc.gam, kSigma, kC);
  // device layout: the coefficients of a cell side by side (RestTable)
  std::vector<double> cells((size_t)RT_PLANES * t.ncell * 2, 0.0);   // [plane][cell] pairs
  for (int p = 0; p <= RT_DEG_DEV; ++p)
    for (int ci = 0; ci < t.ncell; ++ci) cells[((size_t)(p / 2) * t.ncell + ci) * 2 + (p & 1)] = t.coef[(size_t)p * t.ncell + ci];
  int rc = dev_upload(&c->d_rt, cells.data(), cells.size(), c->err);
  if (rc) return rc;
  c->rt_ncell = t.ncell; c->rt_h = t.h; c->rt_num_lines = c->params.num_lines; c->rt_pixel_spacing = c->params.pixel_spacing;
  return GPDLA_OK;
}
static RestTable rest_table_args(const gpdla_ctx* c) {
  RestTable rt;
  const bool on = c->params.rest_table >= 0 && c->d_rt != nullptr;
  rt.coef = on ? c->d_rt : nullptr;
  rt.ncell = c->rt_ncell;
  rt.inv_h = 1.0 / (c->params.pixel_spacing * log(10.0));
  rt.lam_lo = RT_LAMBDA_LO;
  return rt;
}

// The FP64 DMMA kernels.  With la.only_list (the INT8 path's fallback) a few grid.y slots stride over the listed quasars.
constexpr int FALLBACK_SLOTS = 8;
template <int K, int NL, int MODE, int NSPLIT>
static int launch_loglik(gpdla_ctx* c, LoglikArgs la, int nq, cudaStream_t st, bool timed = true) {
  using WCfg = WsConfig<K, NSPLIT>;
  auto kern = dla_loglik_ws_kernel<K, NL, MODE, NSPLIT>;
  if (la.only_list) {
    if constexpr (K == I8_K || K == I8_K_EXT) kern = dla_loglik_ws_list_kernel<K, NL, MODE, NSPLIT>;
    else { c->err = "FP64 fallback list: rank without an INT8 path"; return GPDLA_ERR_UNSUPPORTED; }
  }
  const size_t smem = WCfg::smem_bytes(la.num_lines);
  const int TS = WCfg::TS;
  int rc = configure_smem(c->device, kern, smem, c->err);
  if (rc) return rc;
  const unsigned tiles = (unsigned)((la.S + (la.log_likelihoods_no_dla ? 1 : 0) + TS - 1) / TS);
  dim3 grid(tiles, la.only_list ? (unsigned)std::min(nq, FALLBACK_SLOTS) : (unsigned)nq, NSPLIT);
  la.gram = c->d_gram; la.qld = c->d_qld; la.gram_rows = gram_rows(c);
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (c->profiling && timed) {
    CUDA_TRY(cudaEventCreate(&e0), c->err);
    CUDA_TRY(cudaEventCreate(&e1), c->err);
    CUDA_TRY(cudaEventRecord(e0, st), c->err);
  }
  kern<<<grid, WS_THREADS, smem, st>>>(la);
  c->launches++;
  CUDA_TRY(cudaGetLastError(), c->err);
  if (NSPLIT > 1 && !la.only_list) {   // a list is the INT8 path's fallback: its Cholesky launch covers the batch
    CholArgs ca;
    ca.meta = la.meta; ca.gram = c->d_gram; ca.qld = c->d_qld; ca.gram_rows = la.gram_rows; ca.S = la.S;
    ca.sample_log_likelihoods = la.sample_log_likelihoods; ca.sll_stride = la.sll_stride;
    ca.log_likelihoods_no_dla = la.log_likelihoods_no_dla; ca.active = la.active; ca.order = la.order;
    ca.q_offset = la.q_offset;
    rc = configure_smem(c->device, cholesky_kernel<K>, cholesky_smem_bytes<K>(), c->err);
    if (rc) return rc;
    cholesky_kernel<K><<<dim3(tiles * TS / CHOL_SAMPLES, (unsigned)nq), CHOL_THREADS,
                         cholesky_smem_bytes<K>(), st>>>(ca);
    c->launches++;
    CUDA_TRY(cudaGetLastError(), c->err);
  }
  if (c->profiling && timed) {
    CUDA_TRY(cudaEventRecord(e1, st), c->err);
    c->prof_events.emplace_back(e0, e1);
  }
  return GPDLA_OK;
}

static int ensure_i8_workspace(gpdla_ctx* c, int batch, int npix) {
  if (c->i8_batch >= batch && c->i8_npix == npix && c->i8_k == c->k && c->i8_S == c->S) return GPDLA_OK;
  cudaFree(c->d_pix2); cudaFree(c->d_pix8); cudaFree(c->d_colscale); cudaFree(c->d_colinv); cudaFree(c->d_bop); cudaFree(c->d_f64flag);
  cudaFree(c->d_adig);
  c->d_pix2 = c->d_pix8 = c->d_colscale = c->d_colinv = nullptr; c->d_bop = c->d_adig = nullptr; c->d_f64flag = nullptr; c->i8_batch = 0;
  const size_t B = batch;
  size_t ncoltab = 0, chunk_bytes = 0, a_tile = 0;   // the 6-digit layout is the larger one
  GPDLA_FOR_I8(c->k, 6, (ncoltab = i8::Shape<K, L>::NCOLTAB, chunk_bytes = i8::Shape<K, L>::CHUNK_BYTES,
                         a_tile = i8::Shape<K, L>::EXT ? i8::Shape<K, L>::A_TILE : 0));
  CUDA_TRY(cudaMalloc(&c->d_pix2, B * npix * 2 * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_pix8, B * npix * 8 * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_colscale, B * ncoltab * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_colinv, B * ncoltab * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_bop, B * (npix / KC) * chunk_bytes), c->err);
  if (a_tile)   // W'' digit tiles of the whole batch for the contract-only passes
    CUDA_TRY(cudaMalloc(&c->d_adig, B * (size_t)(gram_rows(c) / i8::TM) * (npix / KC) * a_tile), c->err);
  CUDA_TRY(cudaMalloc(&c->d_f64flag, (2 * B + 2) * sizeof(int32_t)), c->err);
  if (!c->d_status) {
    CUDA_TRY(cudaMalloc(&c->d_status, sizeof(int)), c->err);
    CUDA_TRY(cudaMemset(c->d_status, 0, sizeof(int)), c->err);
  }
  c->i8_batch = batch; c->i8_npix = npix; c->i8_k = c->k; c->i8_S = c->S;
  return GPDLA_OK;
}

static i8::I8Args i8_args(gpdla_ctx* c) {
  i8::I8Args xa;
  xa.pix2 = c->d_pix2; xa.pix8 = c->d_pix8; xa.adig = c->d_adig; xa.bop = c->d_bop; xa.colscale = c->d_colscale; xa.colinv = c->d_colinv; xa.status = c->d_status;
  xa.f64flag = c->d_f64flag; xa.f64list = c->d_f64flag + c->i8_batch;
  xa.phase = nullptr;
  if (GPDLA_I8P_PHASES && getenv("GPDLA_I8_PHASES")) {   // diagnostics only: mean barrier waits per tile, printed before the next launch
    if (!c->d_phase) { cudaMalloc(&c->d_phase, 24 * sizeof(unsigned long long)); cudaMemset(c->d_phase, 0, 24 * sizeof(unsigned long long)); }
    unsigned long long h[24];
    cudaMemcpy(h, c->d_phase, sizeof h, cudaMemcpyDeviceToHost);
    if (h[7]) fprintf(stderr, "[i8 persistent waits, mean cycles per tile] producer: stage empty (per warp) %llu | mma: A full %llu, B full %llu, TMEM drained %llu | loader %llu | sender %llu | epilogue (per warp): acc final %llu, triangle free %llu, triangle full %llu, scalars %llu | stage B waits for A (per warp) %llu, A for B %llu | tile (MMA issuer) %llu\n",
                      h[9] / h[7] / 8, h[10] / h[7], h[11] / h[7], h[21] / h[7], h[12] / h[7], h[13] / h[7], h[14] / h[7] / 4, h[18] / h[7] / 4, h[19] / h[7] / 4, h[20] / h[7] / 4, h[22] / h[7] / 8, h[23] / h[7] / 8, h[6] / h[7]);
    cudaMemset(c->d_phase, 0, sizeof h);
    xa.phase = c->d_phase;
  }
  return xa;
}

// K0c + K0d: scales and digit planes of the B operand for a prepared batch
template <int K, int L>
static int build_i8_operands_L(gpdla_ctx* c, int nq, int npix, cudaStream_t st) {
  i8::I8Args xa = i8_args(c);
  i8::i8_scales_kernel<K, L><<<nq, NTHREADS, 0, st>>>(c->d_meta, c->d_pix, c->d_Mq, c->d_lam, c->d_lamh, xa, npix);
  c->launches++;
  CUDA_TRY(cudaGetLastError(), c->err);
  i8::i8_build_operand_kernel<K, L><<<dim3(npix / KC, nq), NTHREADS, 0, st>>>(c->d_meta, c->d_Mq, xa, npix);
  c->launches++;
  CUDA_TRY(cudaGetLastError(), c->err);
  return GPDLA_OK;
}
// Gram operand P of the FP64 kernels for a prepared batch (`only_list`: restricted to the listed quasars)
static int build_f64_operand(gpdla_ctx* c, int q0, int nq, int npix, const int32_t* only_list, cudaStream_t st) {
  const unsigned ny = only_list ? (unsigned)std::min(nq, FALLBACK_SLOTS) : (unsigned)nq;
  GPDLA_FOR_RANK(c->k, (build_gram_operand_kernel<K, NSPLIT><<<dim3(npix / KC, ny, NSPLIT), NTHREADS, 0, st>>>(
                            c->d_Mq, c->d_meta, c->d_P, npix, only_list, q0)));
  c->launches++;
  CUDA_TRY(cudaGetLastError(), c->err);
  return GPDLA_OK;
}

static int build_i8_operands(gpdla_ctx* c, int nq, int npix, cudaStream_t st) {
  int rc = ensure_i8_workspace(c, c->ws_batch, npix);
  if (rc) return rc;
  CUDA_TRY(cudaMemsetAsync(c->d_f64flag, 0, (2 * (size_t)c->i8_batch + 2) * sizeof(int32_t), st), c->err);
  rc = GPDLA_ERR_UNSUPPORTED;
  GPDLA_FOR_I8(c->k, i8_digits(c), (rc = build_i8_operands_L<K, L>(c, nq, npix, st)));
  if (rc) return rc;
  // FP64 operand of the quasars the scales kernel has just flagged (normally none: a handful of idle CTAs)
  return build_f64_operand(c, 0, nq, npix, c->d_f64flag + c->i8_batch, st);
}

// resident 4-CTA clusters of the persistent kernel on this device (0 = query failed)
template <class Kern>
static int max_resident_clusters(Kern kern, size_t smem, int threads) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(i8::CLUSTER * 148, 1, 1); cfg.blockDim = dim3(threads, 1, 1); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = i8::CLUSTER; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

template <int K, int L, int NL, int MODE>
static int launch_loglik_i8(gpdla_ctx* c, LoglikArgs la, int nq, cudaStream_t st) {
  using Sh = i8::Shape<K, L>;
  la.gram = c->d_gram; la.qld = c->d_qld; la.gram_rows = gram_rows(c);
  const int dev = c->device;
  const unsigned clusters = (unsigned)((la.S + (la.log_likelihoods_no_dla ? 1 : 0) + i8::TM - 1) / i8::TM);
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (c->profiling) {
    CUDA_TRY(cudaEventCreate(&e0), c->err);
    CUDA_TRY(cudaEventCreate(&e1), c->err);
    CUDA_TRY(cudaEventRecord(e0, st), c->err);
  }
  auto kern = i8::dla_loglik_i8p_kernel<K, L, NL, MODE>;
  const size_t smem = i8::PShape<K, L>::smem_bytes(la.num_lines);
  int rc = configure_smem(dev, kern, smem, c->err);
  if (rc) return rc;
  int resident;
  {
    std::lock_guard<std::mutex> lock(g_dev[dev].mu);
    int& n = g_dev[dev].clusters[(const void*)kern];
    if (n == 0) {
      // setmaxnreg.inc can only draw on registers the CTA owned at launch (bench_micro/setmaxnreg_pool.cu): a build whose
      // launch allocation is smaller than the warpgroups' budgets would block forever -- refuse it instead
      cudaFuncAttributes fa;
      if (cudaFuncGetAttributes(&fa, kern) == cudaSuccess && fa.numRegs * i8::P_THREADS < i8::REG_BUDGET_TOTAL) {
        c->err = "dla_loglik_i8p_kernel: launch register allocation below the setmaxnreg budgets (rebuild with matching REG_*)";
        return GPDLA_ERR_CUDA;
      }
      n = max_resident_clusters(kern, smem, i8::P_THREADS);
      const char* e = getenv("GPDLA_I8_CLUSTERS");   // tuning aid: grid size only, same arithmetic
      if (e) n = atoi(e);
      if (n <= 0) n = 32;
    }
    resident = n;
  }
  const long long tiles = (long long)nq * clusters;
  const unsigned ncl = (unsigned)std::min<long long>(resident, tiles);
  kern<<<dim3(ncl * i8::CLUSTER, 1, 1), i8::P_THREADS, smem, st>>>(la, i8_args(c), nq, (int)clusters);
  c->launches++;
  CUDA_TRY(cudaGetLastError(), c->err);
  if constexpr (Sh::EXT) {
    // the column blocks beyond the producing cluster's three: contract-only passes over the stored W'' digit tiles
    auto ckern = i8::gram_contract_i8_kernel<K, L>;
    const size_t csmem = i8::CShape<K, L>::SMEM;
    rc = configure_smem(dev, ckern, csmem, c->err);
    if (rc) return rc;
    int cres;
    {
      std::lock_guard<std::mutex> lock(g_dev[dev].mu);
      int& n = g_dev[dev].clusters[(const void*)ckern];
      if (n == 0) n = max_resident_clusters(ckern, csmem, i8::C_THREADS);
      if (n <= 0) n = 32;
      cres = n;
    }
    const unsigned ccl = (unsigned)std::min<long long>(cres, tiles * Sh::CPASSES);
    ckern<<<dim3(ccl * i8::CLUSTER, 1, 1), i8::C_THREADS, csmem, st>>>(la, i8_args(c), nq, (int)clusters);
    c->launches++;
    CUDA_TRY(cudaGetLastError(), c->err);
  }
  if (c->profiling) {
    CUDA_TRY(cudaEventRecord(e1, st), c->err);
    c->prof_events.emplace_back(e0, e1);
  }
  return GPDLA_OK;
}

static int ensure_multi_workspace(gpdla_ctx* c, int batch, int npix) {
  if (c->mws_batch >= batch && c->mws_npix == npix && c->mws_S == c->S) return GPDLA_OK;
  cudaFree(c->d_acache); cudaFree(c->d_msll); cudaFree(c->d_mlls); cudaFree(c->d_cum); cudaFree(c->d_mscal);
  cudaFree(c->d_partners); cudaFree(c->d_active);
  c->d_acache = c->d_msll = c->d_mlls = c->d_cum = c->d_mscal = nullptr; c->d_partners = c->d_active = nullptr;
  c->mws_batch = 0;
  const size_t B = batch, S = (size_t)c->S;
  CUDA_TRY(cudaMalloc(&c->d_acache, B * S * npix * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_msll, B * 4 * S * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_mlls, B * S * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_cum, B * S * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_mscal, B * 8 * sizeof(double)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_partners, B * 3 * S * sizeof(int32_t)), c->err);
  CUDA_TRY(cudaMalloc(&c->d_active, B * sizeof(int32_t)), c->err);
  c->mws_batch = batch; c->mws_npix = npix; c->mws_S = c->S;
  return GPDLA_OK;
}

// FP64 DMMA kernels for the context's rank and line count
template <int MODE>
static int launch_mode(gpdla_ctx* c, const LoglikArgs& la, int nq, cudaStream_t st, bool timed = true) {
  int rc = GPDLA_ERR_UNSUPPORTED;
  if (c->params.num_lines == 3) { GPDLA_FOR_RANK(c->k, (rc = launch_loglik<K, 3, MODE, NSPLIT>(c, la, nq, st, timed))); }
  else { GPDLA_FOR_RANK(c->k, (rc = launch_loglik<K, 0, MODE, NSPLIT>(c, la, nq, st, timed))); }
  return rc;
}

// INT8 path with its FP64 fallback: the persistent kernel skips the quasars whose scales flagged a used pixel with
// zero noise variance (the fixed-point bound of U'' does not exist there, i8_scales_kernel); the FP64 kernels then
// process exactly those -- FALLBACK_SLOTS idle CTA columns when there are none, no host round trip.
template <int MODE>
static int launch_mode_i8(gpdla_ctx* c, const LoglikArgs& la, int nq, cudaStream_t st) {
  int rc = GPDLA_ERR_UNSUPPORTED;
  if (c->params.num_lines == 3) { GPDLA_FOR_I8(c->k, i8_digits(c), (rc = launch_loglik_i8<K, L, 3, MODE>(c, la, nq, st))); }
  else { GPDLA_FOR_I8(c->k, i8_digits(c), (rc = launch_loglik_i8<K, L, 0, MODE>(c, la, nq, st))); }
  if (rc) return rc;
  LoglikArgs lf = la;
  lf.only_list = c->d_f64flag + c->i8_batch;
  rc = launch_mode<MODE>(c, lf, nq, st, false);
  if (rc || c->k != I8_K_EXT) return rc;
  // k = 40: every path above left its accumulators in the global staging rows; one Cholesky launch for the batch
  CholArgs ca;
  ca.meta = la.meta; ca.gram = c->d_gram; ca.qld = c->d_qld; ca.gram_rows = gram_rows(c); ca.S = la.S;
  ca.sample_log_likelihoods = la.sample_log_likelihoods; ca.sll_stride = la.sll_stride;
  ca.log_likelihoods_no_dla = la.log_likelihoods_no_dla; ca.active = la.active; ca.order = la.order;
  ca.q_offset = la.q_offset;
  rc = configure_smem(c->device, cholesky_kernel<I8_K_EXT>, cholesky_smem_bytes<I8_K_EXT>(), c->err);
  if (rc) return rc;
  const int64_t rows = la.S + (la.log_likelihoods_no_dla ? 1 : 0);
  cholesky_kernel<I8_K_EXT><<<dim3((unsigned)((rows + CHOL_SAMPLES - 1) / CHOL_SAMPLES), (unsigned)nq), CHOL_THREADS,
                              cholesky_smem_bytes<I8_K_EXT>(), st>>>(ca);
  c->launches++;
  CUDA_TRY(cudaGetLastError(), c->err);
  return GPDLA_OK;
}

// both stages of the training objective: persistent CTAs with private partial gradients, then their sum
template <int K>
static int launch_objective(ObjectiveArgs a, cudaStream_t st) {
  const size_t smem = objective_smem_bytes<K>(a.P);
  int dev = 0, sms = 0, per_sm = 0;
  CUDA_TRY(cudaGetDevice(&dev), g_err);
  CUDA_TRY(cudaFuncSetAttribute(objective_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), g_err);
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev), g_err);
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, objective_kernel<K>, OBJ_THREADS, smem), g_err);
  const int64_t nx = (int64_t)a.P * (K + 1) + 3;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(a.N, (int64_t)sms * std::max(per_sm, 1)));
  CUDA_TRY(cudaMallocAsync(&a.partial, (size_t)grid * (nx + 1) * sizeof(double), st), g_err);
  objective_kernel<K><<<grid, OBJ_THREADS, smem, st>>>(a);
  CUDA_TRY(cudaGetLastError(), g_err);
  objective_reduce_kernel<<<(unsigned)((nx + 1 + 255) / 256), 256, 0, st>>>(a.partial, grid, nx, a.g, a.f);
  CUDA_TRY(cudaGetLastError(), g_err);
  CUDA_TRY(cudaFreeAsync(a.partial, st), g_err);
  return GPDLA_OK;
}

template <int MODE>
static int launch_mode_any(gpdla_ctx* c, const LoglikArgs& la, int nq, cudaStream_t st) {
  return use_i8(c) ? launch_mode_i8<MODE>(c, la, nq, st) : launch_mode<MODE>(c, la, nq, st);
}

// K0 arguments for quasars [q0, q0 + nq) of a padded catalogue
static PrepArgs prep_args(const gpdla_ctx* c, int64_t q0, int64_t L_max, const double* wavelengths, const double* flux,
                          const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                          const double* z_qsos, int npix, int meanflux) {
  PrepArgs pa;
  pa.wavelengths = wavelengths + q0 * L_max; pa.flux = flux + q0 * L_max;
  pa.noise_variance = noise_variance + q0 * L_max; pa.pixel_mask = pixel_mask + q0 * L_max;
  pa.lengths = lengths + q0; pa.z_qsos = z_qsos + q0; pa.L_max = L_max;
  pa.rest_wavelengths = c->d_rest; pa.mu = c->d_mu; pa.M = c->d_M; pa.log_omega = c->d_log_omega;
  pa.n_rest = c->n_rest; pa.k = c->k; pa.c_0 = c->c_0; pa.tau_0 = c->tau_0; pa.beta = c->beta;
  pa.prior_z_qsos = c->d_prior_z; pa.prior_dla_ind = c->d_prior_dla; pa.n_prior = c->n_prior;
  pa.min_lambda = c->params.min_lambda; pa.max_lambda = c->params.max_lambda;
  pa.lya_wavelength = c->params.lya_wavelength; pa.lyman_limit = c->params.lyman_limit;
  pa.prior_z_qso_increase = c->params.prior_z_qso_increase; pa.min_z_cut = c->params.min_z_cut;
  pa.max_z_cut = c->params.max_z_cut; pa.pixel_spacing = c->params.pixel_spacing;
  pa.meta = c->d_meta; pa.lam_pad = c->d_lam; pa.lamh = c->d_lamh; pa.pix = c->d_pix; pa.Mq = c->d_Mq; pa.NPIX = npix;
  pa.inv_h = 1.0 / (c->params.pixel_spacing * log(10.0));
  pa.meanflux = meanflux;
  return pa;
}

// the batch-invariant part of the fused kernels' arguments
static LoglikArgs loglik_args(const gpdla_ctx* c, int npix) {
  LoglikArgs la;
  memset(&la, 0, sizeof la);
  la.meta = c->d_meta; la.lam_pad = c->d_lam; la.lamh = c->d_lamh; la.rt = rest_table_args(c); la.order = c->d_order;
  la.pix = c->d_pix; la.P = c->d_P;
  la.offset_samples = c->d_offset; la.nhi_samples = c->d_nhi; la.S = c->S;
  la.num_lines = c->params.num_lines; la.NPIX = npix;
  return la;
}

// How many of a batch's nq quasars go to the FP64 DMMA kernels while the INT8 kernel works on the others: the 4-CTA
// clusters of the persistent INT8 kernel occupy 132 of the 148 SMs (cluster placement within the GPCs), and the FP64
// kernel -- no clusters, one CTA per SM -- runs on the 16 that are left, on a second stream.  The share balances the two
// (measured per-SM rates 23.7 against 36.8 quasars/s); small batches stay whole, so that their results do not depend on
// which path a quasar happened to land on.
constexpr int SPLIT_MIN_QUASARS = 148;
static int f64_share(const gpdla_ctx* c, int nq) {
  if (!use_i8(c) || nq < SPLIT_MIN_QUASARS) return 0;
  double share = 0.072;
  if (const char* e = getenv("GPDLA_F64_SHARE")) share = atof(e);   // tuning aid
  return std::max(0, std::min(nq / 2, (int)lround(share * nq)));
}

// K0 + operand builders for one batch; the last `nq_f64` quasars get the FP64 operand (see f64_share)
static int prepare_batch(gpdla_ctx* c, const PrepArgs& pa, int nq, int nq_f64, int npix, cudaStream_t st) {
  prepare_quasars_kernel<<<nq, NTHREADS, 0, st>>>(pa);
  c->launches++;
  CUDA_TRY(cudaGetLastError(), c->err);
  if (!use_i8(c)) return build_f64_operand(c, 0, nq, npix, nullptr, st);
  int rc = build_i8_operands(c, nq - nq_f64, npix, st);
  if (rc == GPDLA_OK && nq_f64 > 0) rc = build_f64_operand(c, nq - nq_f64, nq_f64, npix, nullptr, st);
  return rc;
}

// The fused kernels of one batch in MODE: the INT8 kernel on quasars [0, nq - nq_f64) on `st` and, concurrently on
// the context's side stream, the FP64 kernels on the last nq_f64 quasars; `st` continues when both are done.
template <int MODE>
static int launch_split(gpdla_ctx* c, const LoglikArgs& la, int nq, int nq_f64, cudaStream_t st) {
  if (nq_f64 <= 0) return launch_mode_any<MODE>(c, la, nq, st);
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  const bool timed = c->profiling;
  if (timed) {   // one interval around the concurrent pair
    CUDA_TRY(cudaEventCreate(&e0), c->err);
    CUDA_TRY(cudaEventCreate(&e1), c->err);
    CUDA_TRY(cudaEventRecord(e0, st), c->err);
    c->profiling = false;
  }
  CUDA_TRY(cudaEventRecord(c->ev_fork, st), c->err);
  int rc = launch_mode_i8<MODE>(c, la, nq - nq_f64, st);      // enqueued first: its clusters get their SMs first
  if (rc == GPDLA_OK) {
    CUDA_TRY(cudaStreamWaitEvent(c->side_stream, c->ev_fork, 0), c->err);
    LoglikArgs lf = la;
    lf.q_offset = nq - nq_f64;
    rc = launch_mode<MODE>(c, lf, nq_f64, c->side_stream, false);
    CUDA_TRY(cudaEventRecord(c->ev_join, c->side_stream), c->err);
    CUDA_TRY(cudaStreamWaitEvent(st, c->ev_join, 0), c->err);
  }
  if (timed) {
    c->profiling = true;
    CUDA_TRY(cudaEventRecord(e1, st), c->err);
    c->prof_events.emplace_back(e0, e1);
  }
  return rc;
}

__global__ void fill_i32_kernel(int32_t* p, int32_t v, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

extern "C" {

void gpdla_default_parameters(gpdla_params* p) {
  const double c = 299792458.0;
  p->min_lambda = 911.75; p->max_lambda = 1215.75;
  p->lya_wavelength = 1215.6701; p->lyman_limit = 911.7633;
  p->prior_z_qso_increase = (30000.0 * 1000.0) / c;
  p->min_z_cut = (3000.0 * 1000.0) / c; p->max_z_cut = (3000.0 * 1000.0) / c;
  p->pixel_spacing = 1e-4;
  p->num_lines = 3;
  p->batch_quasars = 0;
  p->gram_digits = 0; p->rest_table = 0;
}

int gpdla_rest_table(int32_t num_lines, double pixel_spacing, double* coef, int32_t* ncell, int32_t* degree, double* h,
                     double* lambda_lo) {
  if (num_lines < 1 || num_lines > GPDLA_MAX_LINES || !(pixel_spacing > 0)) return GPDLA_ERR_INVALID;
  LineConstants lc;
  fill_line_constants(&lc);
  if (degree) *degree = RT_DEG;
  if (lambda_lo) *lambda_lo = RT_LAMBDA_LO;
  if (!coef) {
    const double hh = pixel_spacing * log(10.0);
    if (h) *h = hh;
    if (ncell) *ncell = (int32_t)ceil((log(RT_LAMBDA_HI) - log(RT_LAMBDA_LO)) / hh) + 1;
    return GPDLA_OK;
  }
  const RestTableHost t = build_rest_table(num_lines, pixel_spacing, RT_NEAR_PIXELS, lc.tw, lc.lc, lc.gam, kSigma, kC);
  memcpy(coef, t.coef.data(), t.coef.size() * sizeof(double));
  if (ncell) *ncell = t.ncell;
  if (h) *h = t.h;
  return GPDLA_OK;
}

int gpdla_host_alloc(void** ptr, uint64_t bytes) {
  if (!ptr) return GPDLA_ERR_INVALID;
  *ptr = nullptr;
  CUDA_TRY(cudaHostAlloc(ptr, bytes > 0 ? bytes : 1, cudaHostAllocDefault), g_err);
  return GPDLA_OK;
}
void gpdla_host_free(void* ptr) { if (ptr) cudaFreeHost(ptr); }

void gpdla_line_constants(double* tw, double* lcs, double* gam, double* ip) {
  LineConstants lc;
  fill_line_constants(&lc);
  if (tw) memcpy(tw, lc.tw, sizeof lc.tw);
  if (lcs) memcpy(lcs, lc.lc, sizeof lc.lc);
  if (gam) memcpy(gam, lc.gam, sizeof lc.gam);
  if (ip) memcpy(ip, lc.ip, sizeof lc.ip);
}

int gpdla_create(gpdla_ctx** out, int device) {
  if (!out) return GPDLA_ERR_INVALID;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev || device >= MAX_DEVICES) {
    g_err = "no CUDA device " + std::to_string(device) + " (libgpdla.so has no CPU fallback)";
    return GPDLA_ERR_CUDA;
  }
  DeviceGuard guard(device);
  if (guard.status != cudaSuccess) { g_err = cudaGetErrorString(guard.status); return GPDLA_ERR_CUDA; }
  int rc = upload_device_constants(g_err);
  if (rc != GPDLA_OK) return rc;
  gpdla_ctx* ctx = new gpdla_ctx;
  ctx->device = device;
  gpdla_default_parameters(&ctx->params);
  cudaError_t e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->side_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming);
  for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
    e = cudaEventCreateWithFlags(&ctx->ev_batch[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming);
  }
  if (e != cudaSuccess) { g_err = cudaGetErrorString(e); gpdla_destroy(ctx); return GPDLA_ERR_CUDA; }
  *out = ctx;
  return GPDLA_OK;
}

void gpdla_destroy(gpdla_ctx* c) {
  if (!c) return;
  DeviceGuard guard(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
  if (c->side_stream) cudaStreamSynchronize(c->side_stream);
  free_workspace(c);
  cudaFree(c->d_rest); cudaFree(c->d_mu); cudaFree(c->d_M); cudaFree(c->d_log_omega);
  cudaFree(c->d_offset); cudaFree(c->d_log_nhi); cudaFree(c->d_nhi); cudaFree(c->d_order); cudaFree(c->d_rt);
  cudaFree(c->d_prior_z); cudaFree(c->d_prior_dla); cudaFree(c->d_stage);
  cudaFree(c->d_pix2); cudaFree(c->d_pix8); cudaFree(c->d_colscale); cudaFree(c->d_colinv); cudaFree(c->d_bop); cudaFree(c->d_adig); cudaFree(c->d_status);
  cudaFree(c->d_f64flag); cudaFree(c->d_phase);
  cudaFree(c->d_lls_nhi); cudaFree(c->d_uniforms); cudaFree(c->d_acache); cudaFree(c->d_msll); cudaFree(c->d_mlls);
  cudaFree(c->d_cum); cudaFree(c->d_mscal); cudaFree(c->d_partners); cudaFree(c->d_active);
  for (auto& ev : c->prof_events) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
  for (int i = 0; i < 2; ++i) {
    if (c->ev_batch[i]) cudaEventDestroy(c->ev_batch[i]);
    if (c->ev_copied[i]) cudaEventDestroy(c->ev_copied[i]);
  }
  if (c->stream) cudaStreamDestroy(c->stream);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->side_stream) cudaStreamDestroy(c->side_stream);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  delete c;
}

const char* gpdla_last_error(const gpdla_ctx* c) { return c ? c->err.c_str() : g_err.c_str(); }
uint64_t gpdla_launch_count(const gpdla_ctx* c) { return c ? c->launches : 0; }

int gpdla_set_profiling(gpdla_ctx* c, int enable) {
  if (!c) return GPDLA_ERR_INVALID;
  c->profiling = enable != 0;
  return GPDLA_OK;
}

int gpdla_profile_read(gpdla_ctx* c, double* loglik_ms, int64_t* loglik_launches) {
  if (!c) return GPDLA_ERR_INVALID;
  double total = 0;
  int64_t n = 0;
  for (auto& ev : c->prof_events) {
    CUDA_TRY(cudaEventSynchronize(ev.second), c->err);
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, ev.first, ev.second), c->err);
    total += ms; ++n;
    cudaEventDestroy(ev.first); cudaEventDestroy(ev.second);
  }
  c->prof_events.clear();
  if (loglik_ms) *loglik_ms = total;
  if (loglik_launches) *loglik_launches = n;
  return GPDLA_OK;
}

int gpdla_set_parameters(gpdla_ctx* c, const gpdla_params* p) {
  if (!c || !p) return GPDLA_ERR_INVALID;
  if (p->num_lines < 1 || p->num_lines > GPDLA_MAX_LINES || !(p->max_lambda > p->min_lambda) ||
      !(p->pixel_spacing > 0) || p->batch_quasars < 0 || !(p->rest_table == 0 || p->rest_table == -1) ||
      !(p->gram_digits == 0 || p->gram_digits == -1 || p->gram_digits == 5 || p->gram_digits == 6)) {
    c->err = "gpdla_set_parameters: invalid parameters";
    return GPDLA_ERR_INVALID;
  }
  c->params = *p;
  return GPDLA_OK;
}

int gpdla_set_model(gpdla_ctx* c, const double* rest, int32_t n_rest, const double* mu, const double* M, int32_t k,
                    const double* log_omega, double log_c_0, double log_tau_0, double log_beta) {
  if (!c || !rest || !mu || !M || !log_omega || n_rest < 2 || k < 1) return GPDLA_ERR_INVALID;
  if (!rank_supported(k)) {
    c->err = "gpdla_set_model: rank k=" + std::to_string(k) + " not compiled in (available: 10, 20, 40)";
    return GPDLA_ERR_UNSUPPORTED;
  }
  DeviceGuard guard(c->device);
  int rc;
  if ((rc = dev_upload(&c->d_rest, rest, n_rest, c->err))) return rc;
  if ((rc = dev_upload(&c->d_mu, mu, n_rest, c->err))) return rc;
  if ((rc = dev_upload(&c->d_M, M, (size_t)n_rest * k, c->err))) return rc;
  if ((rc = dev_upload(&c->d_log_omega, log_omega, n_rest, c->err))) return rc;
  c->n_rest = n_rest; c->k = k;
  c->c_0 = exp(log_c_0); c->tau_0 = exp(log_tau_0); c->beta = exp(log_beta);   // process_qsos.m:84-86
  return GPDLA_OK;
}

int gpdla_set_samples(gpdla_ctx* c, const double* offset, const double* log_nhi, const double* nhi, int64_t S) {
  if (!c || !offset || !log_nhi || !nhi || S < 1 || S > 2147483647LL) return GPDLA_ERR_INVALID;
  DeviceGuard guard(c->device);
  int rc;
  if ((rc = dev_upload(&c->d_offset, offset, S, c->err))) return rc;
  if ((rc = dev_upload(&c->d_log_nhi, log_nhi, S, c->err))) return rc;
  if ((rc = dev_upload(&c->d_nhi, nhi, S, c->err))) return rc;
  // Order in which the kernels walk the samples (results are stored under the caller's sample index): ascending
  // redshift offset, so that the four samples a producer warp interleaves are neighbours in redshift and share one
  // cell of the rest-frame table per pixel, and the warps of a CTA find each other's table lines in L1.  (Groups of
  // neighbours dealt out in a scattered order -- GPDLA_ORDER_GROUP=n, a tuning aid -- measured slower: the warps of a
  // cluster then reach the line cores, i.e. the direct evaluation, in different chunks and wait for each other.)
  std::vector<int32_t> sorted((size_t)S), order((size_t)S);
  std::iota(sorted.begin(), sorted.end(), 0);
  std::stable_sort(sorted.begin(), sorted.end(), [&](int32_t a, int32_t b) { return offset[a] < offset[b]; });
  {
    int64_t group = ORDER_GROUP;
    if (const char* e = getenv("GPDLA_ORDER_GROUP")) group = atoll(e);   // tuning aid (0 = fully sorted)
    const int64_t G = group > 0 ? S / group : 0;                         // full groups; a partial last group stays last
    int64_t A = (int64_t)(0.6180339887 * (double)G);
    auto gcd = [](int64_t a, int64_t b) { while (b) { const int64_t t = a % b; a = b; b = t; } return a; };
    while (G > 1 && gcd(A, G) != 1) ++A;
    if (group < 0) std::iota(sorted.begin(), sorted.end(), 0);           // diagnosis: the caller's order
    for (int64_t pos = 0; pos < S; ++pos) {
      const int64_t pg = group > 0 ? pos / group : 0;
      order[(size_t)pos] = (G > 1 && pg < G) ? sorted[(size_t)(((pg * A) % G) * group + pos % group)] : sorted[(size_t)pos];
    }
  }
  if ((rc = dev_upload(&c->d_order, order.data(), (size_t)S, c->err))) return rc;
  if (c->S != S) {   // sub-DLA samples and the resampling stream are per sample count: they must be set again
    cudaFree(c->d_lls_nhi); cudaFree(c->d_uniforms);
    c->d_lls_nhi = c->d_uniforms = nullptr; c->lls_S = 0;
  }
  c->S = S;
  return GPDLA_OK;
}

int gpdla_set_prior(gpdla_ctx* c, const double* z_qsos, const uint8_t* dla_ind, int64_t n) {
  if (!c || n < 0 || (n > 0 && (!z_qsos || !dla_ind))) return GPDLA_ERR_INVALID;
  DeviceGuard guard(c->device);
  int rc;
  if ((rc = dev_upload(&c->d_prior_z, z_qsos, n, c->err))) return rc;
  if ((rc = dev_upload(&c->d_prior_dla, dla_ind, n, c->err))) return rc;
  c->n_prior = n;
  return GPDLA_OK;
}

// One batch (<= workspace batch) of quasars [q0, q0 + nq) of the device-resident catalogue through K0 .. K4.
// `sll` / `llno`: where this batch's [nq x S] sample log-likelihoods and [nq] null-model log-likelihoods go.
static int process_batch(gpdla_ctx* c, int64_t q0, int nq, int64_t L_max, const double* wavelengths, const double* flux,
                         const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                         const double* z_qsos, const gpdla_results* out, double* sll, double* llno, int npix,
                         cudaStream_t st) {
  const int batch = c->ws_batch;
  const int nq_f64 = f64_share(c, nq);
  int rc = prepare_batch(c, prep_args(c, q0, L_max, wavelengths, flux, noise_variance, pixel_mask, lengths, z_qsos, npix, 0),
                         nq, nq_f64, npix, st);
  if (rc) return rc;
  LoglikArgs la = loglik_args(c, npix);
  la.sample_log_likelihoods = sll; la.log_likelihoods_no_dla = llno; la.sll_stride = c->S;
  if ((rc = launch_split<0>(c, la, nq, nq_f64, st))) return rc;

  EvidenceArgs ea;
  ea.meta = c->d_meta; ea.sample_log_likelihoods = sll; ea.log_likelihoods_no_dla = llno;
  ea.offset_samples = c->d_offset; ea.log_nhi_samples = c->d_log_nhi; ea.S = c->S;
  double* scr = c->d_scratch + batch;   // 15 more scratch columns of `batch` doubles
  auto pick = [&](double* p, int col) { return p ? p + q0 : scr + (size_t)col * batch; };
  ea.min_z_dlas = pick(out->min_z_dlas, 0); ea.max_z_dlas = pick(out->max_z_dlas, 1);
  ea.log_priors_no_dla = pick(out->log_priors_no_dla, 2); ea.log_priors_dla = pick(out->log_priors_dla, 3);
  ea.log_likelihoods_dla = pick(out->log_likelihoods_dla, 4);
  ea.log_posteriors_no_dla = pick(out->log_posteriors_no_dla, 5);
  ea.log_posteriors_dla = pick(out->log_posteriors_dla, 6);
  ea.model_posteriors = out->model_posteriors ? out->model_posteriors + 2 * q0 : scr + (size_t)7 * batch;   // 2 cols
  ea.p_no_dlas = pick(out->p_no_dlas, 9); ea.p_dlas = pick(out->p_dlas, 10);
  ea.map_z_dlas = pick(out->map_z_dlas, 11); ea.map_log_nhis = pick(out->map_log_nhis, 12);
  ea.map_inds = out->map_inds ? out->map_inds + q0 : c->d_scratch_i;
  evidence_kernel<<<nq, NTHREADS, 0, st>>>(ea);
  c->launches++;
  CUDA_TRY(cudaGetLastError(), c->err);
  return GPDLA_OK;
}

static int check_ready(gpdla_ctx* c, const char* who) {
  if (!c->d_M || !c->d_offset || c->n_prior < 0) {
    c->err = std::string(who) + ": set_model, set_samples and set_prior must be called first";
    return GPDLA_ERR_STATE;
  }
  return GPDLA_OK;
}
static int default_batch(const gpdla_ctx* c) {
  return c->params.batch_quasars > 0 ? c->params.batch_quasars : (rank_splits(c->k) > 1 ? 37 : 296);
}

int gpdla_process_qsos_device(gpdla_ctx* c, int64_t Q, int64_t L_max, const double* wavelengths, const double* flux,
                              const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                              const double* z_qsos, const gpdla_results* out, void* stream) {
  if (!c) return GPDLA_ERR_INVALID;
  if (Q < 0 || L_max < 1 || !out || (Q > 0 && (!wavelengths || !flux || !noise_variance || !pixel_mask || !lengths || !z_qsos))) {
    c->err = "gpdla_process_qsos_device: invalid arguments";
    return GPDLA_ERR_INVALID;
  }
  int rc = check_ready(c, "gpdla_process_qsos_device");
  if (rc) return rc;
  if (Q == 0) return GPDLA_OK;
  DeviceGuard guard(c->device);
  if ((rc = ensure_rest_table(c))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int npix = (int)((L_max + KC - 1) / KC) * KC;
  if ((rc = ensure_workspace(c, (int)std::min<int64_t>(default_batch(c), Q), npix))) return rc;
  const int batch = c->ws_batch;
  for (int64_t q0 = 0; q0 < Q; q0 += batch) {
    const int nq = (int)std::min<int64_t>(batch, Q - q0);
    double* sll = out->sample_log_likelihoods_dla ? out->sample_log_likelihoods_dla + q0 * c->S : c->d_sll;
    double* llno = out->log_likelihoods_no_dla ? out->log_likelihoods_no_dla + q0 : c->d_scratch;
    if ((rc = process_batch(c, q0, nq, L_max, wavelengths, flux, noise_variance, pixel_mask, lengths, z_qsos, out, sll, llno,
                            npix, st)))
      return rc;
  }
  return GPDLA_OK;
}

// Host buffers in, host buffers out (the drop-in call).  Everything runs on the context's own non-blocking streams:
// inputs go up once, then batch t + 1 is computed while the [nq x S] sample log-likelihoods of batch t -- the one
// large output, 80 KB per quasar -- travel back on the copy stream from a double-buffered device block.
int gpdla_process_qsos(gpdla_ctx* c, int64_t Q, int64_t L_max, const double* wavelengths, const double* flux,
                       const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                       const double* z_qsos, const gpdla_results* out) {
  if (!c) return GPDLA_ERR_INVALID;
  if (Q < 0 || L_max < 1 || !out || (Q > 0 && (!wavelengths || !flux || !noise_variance || !pixel_mask || !lengths || !z_qsos))) {
    c->err = "gpdla_process_qsos: invalid arguments";
    return GPDLA_ERR_INVALID;
  }
  int rc = check_ready(c, "gpdla_process_qsos");
  if (rc) return rc;
  if (Q == 0) return GPDLA_OK;
  DeviceGuard guard(c->device);
  if ((rc = ensure_rest_table(c))) return rc;
  const int npix = (int)((L_max + KC - 1) / KC) * KC;
  if ((rc = ensure_workspace(c, (int)std::min<int64_t>(default_batch(c), Q), npix))) return rc;
  const int batch = c->ws_batch;
  const size_t QL = (size_t)Q * L_max, S = (size_t)c->S;
  const bool want_sll = out->sample_log_likelihoods_dla != nullptr;
  // one device staging block: 3 double planes + z + 14 result columns + map_inds + lengths + mask (+ 2 x [batch x S])
  const size_t n_res = 14;
  size_t bytes = 3 * QL * 8 + (size_t)Q * 8 + (n_res + 1) * Q * 8 + (size_t)Q * 8 + (size_t)Q * 4 + QL + 10 * 16 +
                 (want_sll ? 2 * (size_t)batch * S * 8 : 0);
  if (c->st_bytes < bytes) {
    cudaFree(c->d_stage); c->d_stage = nullptr; c->st_bytes = 0;
    CUDA_TRY(cudaMalloc(&c->d_stage, bytes), c->err);
    c->st_bytes = bytes;
  }
  char* p = (char*)c->d_stage;
  auto take = [&](size_t n) { char* r = p; p += (n + 15) / 16 * 16; return r; };
  double* d_w = (double*)take(QL * 8); double* d_f = (double*)take(QL * 8); double* d_v = (double*)take(QL * 8);
  double* d_z = (double*)take(Q * 8);
  double* d_res = (double*)take((n_res + 1) * Q * 8);
  int64_t* d_map = (int64_t*)take(Q * 8);
  double* d_sllbuf[2] = {nullptr, nullptr};
  if (want_sll) { d_sllbuf[0] = (double*)take((size_t)batch * S * 8); d_sllbuf[1] = (double*)take((size_t)batch * S * 8); }
  int32_t* d_len = (int32_t*)take(Q * 4);
  uint8_t* d_m = (uint8_t*)take(QL);
  cudaStream_t st = c->stream, cs = c->copy_stream;
  CUDA_TRY(cudaMemcpyAsync(d_w, wavelengths, QL * 8, cudaMemcpyHostToDevice, st), c->err);
  CUDA_TRY(cudaMemcpyAsync(d_f, flux, QL * 8, cudaMemcpyHostToDevice, st), c->err);
  CUDA_TRY(cudaMemcpyAsync(d_v, noise_variance, QL * 8, cudaMemcpyHostToDevice, st), c->err);
  CUDA_TRY(cudaMemcpyAsync(d_m, pixel_mask, QL, cudaMemcpyHostToDevice, st), c->err);
  CUDA_TRY(cudaMemcpyAsync(d_len, lengths, Q * 4, cudaMemcpyHostToDevice, st), c->err);
  CUDA_TRY(cudaMemcpyAsync(d_z, z_qsos, Q * 8, cudaMemcpyHostToDevice, st), c->err);
  gpdla_results dr;
  dr.min_z_dlas = d_res + 0 * Q; dr.max_z_dlas = d_res + 1 * Q;
  dr.log_priors_no_dla = d_res + 2 * Q; dr.log_priors_dla = d_res + 3 * Q;
  dr.log_likelihoods_no_dla = d_res + 4 * Q; dr.log_likelihoods_dla = d_res + 5 * Q;
  dr.log_posteriors_no_dla = d_res + 6 * Q; dr.log_posteriors_dla = d_res + 7 * Q;
  dr.p_no_dlas = d_res + 8 * Q; dr.p_dlas = d_res + 9 * Q;
  dr.map_z_dlas = d_res + 10 * Q; dr.map_log_nhis = d_res + 11 * Q;
  dr.model_posteriors = d_res + 12 * Q;   // 2 columns
  dr.map_inds = d_map;
  dr.sample_log_likelihoods_dla = nullptr;
  // batch t is enqueued BEFORE the copy of batch t - 1 is issued: with a pageable destination cudaMemcpyAsync holds
  // the host thread until the copy is done, and the GPU must already have its next batch by then
  auto copy_back = [&](int tt) -> int {
    const int64_t q0 = (int64_t)tt * batch;
    const int nq = (int)std::min<int64_t>(batch, Q - q0);
    const int b = tt & 1;
    CUDA_TRY(cudaStreamWaitEvent(cs, c->ev_batch[b], 0), c->err);
    CUDA_TRY(cudaMemcpyAsync(out->sample_log_likelihoods_dla + (size_t)q0 * S, d_sllbuf[b], (size_t)nq * S * 8,
                             cudaMemcpyDeviceToHost, cs), c->err);
    CUDA_TRY(cudaEventRecord(c->ev_copied[b], cs), c->err);
    return GPDLA_OK;
  };
  int t = 0;
  for (int64_t q0 = 0; q0 < Q; q0 += batch, ++t) {
    const int nq = (int)std::min<int64_t>(batch, Q - q0);
    const int b = t & 1;
    double* sll = want_sll ? d_sllbuf[b] : c->d_sll;
    if (want_sll && t >= 2) CUDA_TRY(cudaStreamWaitEvent(st, c->ev_copied[b], 0), c->err);   // buffer b is on the host
    if ((rc = process_batch(c, q0, nq, L_max, d_w, d_f, d_v, d_m, d_len, d_z, &dr, sll, dr.log_likelihoods_no_dla + q0, npix,
                            st)))
      return rc;
    if (want_sll) {
      CUDA_TRY(cudaEventRecord(c->ev_batch[b], st), c->err);
      if (t >= 1 && (rc = copy_back(t - 1))) return rc;
    }
  }
  if (want_sll && (rc = copy_back(t - 1))) return rc;
  double* hptr[12] = {out->min_z_dlas, out->max_z_dlas, out->log_priors_no_dla, out->log_priors_dla,
                      out->log_likelihoods_no_dla, out->log_likelihoods_dla, out->log_posteriors_no_dla,
                      out->log_posteriors_dla, out->p_no_dlas, out->p_dlas, out->map_z_dlas, out->map_log_nhis};
  for (size_t i = 0; i < 12; ++i)
    if (hptr[i]) CUDA_TRY(cudaMemcpyAsync(hptr[i], d_res + i * Q, Q * 8, cudaMemcpyDeviceToHost, st), c->err);
  if (out->model_posteriors)
    CUDA_TRY(cudaMemcpyAsync(out->model_posteriors, d_res + 12 * Q, 2 * Q * 8, cudaMemcpyDeviceToHost, st), c->err);
  if (out->map_inds) CUDA_TRY(cudaMemcpyAsync(out->map_inds, d_map, Q * 8, cudaMemcpyDeviceToHost, st), c->err);
  CUDA_TRY(cudaStreamSynchronize(st), c->err);
  CUDA_TRY(cudaStreamSynchronize(cs), c->err);
  return GPDLA_OK;
}

// ---------------------------------------------------------------------------- multi-DLA path
void gpdla_matlab_default_rand(double* out, int64_t n) {
  // rng('default') = Mersenne twister, seed 5489; rand = 53-bit doubles (genrand_res53)
  std::mt19937 gen(5489u);
  for (int64_t i = 0; i < n; ++i) {
    const uint32_t a = gen() >> 5, b = gen() >> 6;
    out[i] = (a * 67108864.0 + b) / 9007199254740992.0;
  }
}

int gpdla_set_lls_samples(gpdla_ctx* c, const double* lls_nhi, int64_t S, double Z_lls, double Z_dla) {
  if (!c || !lls_nhi || S < 1 || !(Z_lls > 0) || !(Z_dla > 0)) return GPDLA_ERR_INVALID;
  if (c->S != S) { c->err = "gpdla_set_lls_samples: call gpdla_set_samples first (same sample count)"; return GPDLA_ERR_STATE; }
  DeviceGuard guard(c->device);
  int rc;
  if ((rc = dev_upload(&c->d_lls_nhi, lls_nhi, S, c->err))) return rc;
  std::vector<double> u(3 * (size_t)S);
  gpdla_matlab_default_rand(u.data(), (int64_t)u.size());
  if ((rc = dev_upload(&c->d_uniforms, u.data(), u.size(), c->err))) return rc;
  c->Z_lls = Z_lls; c->Z_dla = Z_dla; c->lls_S = S;
  return GPDLA_OK;
}

int gpdla_process_qsos_multi_device(gpdla_ctx* c, int64_t Q, int64_t L_max, const double* wavelengths,
                                    const double* flux, const double* noise_variance, const uint8_t* pixel_mask,
                                    const int32_t* lengths, const double* z_qsos, int32_t max_dlas,
                                    const int32_t* base_in, const gpdla_multi_results* out, void* stream) {
  if (!c) return GPDLA_ERR_INVALID;
  if (Q < 0 || L_max < 1 || !out || max_dlas < 1 || max_dlas > 4 ||
      (Q > 0 && (!wavelengths || !flux || !noise_variance || !pixel_mask || !lengths || !z_qsos))) {
    c->err = "gpdla_process_qsos_multi_device: invalid arguments (1 <= max_dlas <= 4)";
    return GPDLA_ERR_INVALID;
  }
  const void* required[] = {out->min_z_dlas, out->max_z_dlas, out->log_priors_no_dla, out->log_priors_lls,
                            out->log_priors_dla, out->log_likelihoods_no_dla, out->log_likelihoods_lls,
                            out->log_likelihoods_dla, out->log_posteriors_no_dla, out->log_posteriors_lls,
                            out->log_posteriors_dla, out->model_posteriors, out->p_no_dlas, out->p_lls, out->p_dlas,
                            out->MAP_z_dlas, out->MAP_log_nhis, out->MAP_inds};
  for (const void* r : required)
    if (Q > 0 && !r) { c->err = "gpdla_process_qsos_multi_device: only the three large outputs may be NULL"; return GPDLA_ERR_INVALID; }
  if (!c->d_M || !c->d_offset || c->n_prior < 0 || !c->d_lls_nhi || c->lls_S != c->S) {
    c->err = "gpdla_process_qsos_multi: set_model, set_samples, set_prior and set_lls_samples must be called first";
    return GPDLA_ERR_STATE;
  }
  if (Q == 0) return GPDLA_OK;
  DeviceGuard guard(c->device);
  int rc = ensure_rest_table(c);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int npix = (int)((L_max + KC - 1) / KC) * KC;
  int batch = c->params.batch_quasars > 0 ? c->params.batch_quasars : (rank_splits(c->k) > 1 ? 37 : 148);
  batch = (int)std::min<int64_t>(batch, Q);
  rc = ensure_workspace(c, batch, npix);
  if (rc) return rc;
  rc = ensure_multi_workspace(c, batch, npix);
  if (rc) return rc;
  batch = std::min(c->ws_batch, c->mws_batch);
  const int64_t S = c->S;
  const int MD = max_dlas;
  const double min_z_sep = (3000.0 * 1000.0) / 299792458.0;   // kms_to_z(3000), ...meanflux.m:33

  for (int64_t q0 = 0; q0 < Q; q0 += batch) {
    const int nq = (int)std::min<int64_t>(batch, Q - q0);
    const int nq_f64 = f64_share(c, nq);
    if ((rc = prepare_batch(c, prep_args(c, q0, L_max, wavelengths, flux, noise_variance, pixel_mask, lengths, z_qsos, npix, 1),
                            nq, nq_f64, npix, st)))
      return rc;
    fill_i32_kernel<<<(nq + 255) / 256, 256, 0, st>>>(c->d_active, 1, nq);
    c->launches++;
    CUDA_TRY(cudaMemsetAsync(c->d_partners, 0, (size_t)nq * 3 * c->S * sizeof(int32_t), st), c->err);   // :313 zeros
    CUDA_TRY(cudaGetLastError(), c->err);

    // where this batch's sample log-likelihoods live: caller's [Q x MD x S] array or the workspace
    double* sll = out->sample_log_likelihoods_dla ? out->sample_log_likelihoods_dla + q0 * MD * S : c->d_msll;
    const int64_t sll_stride = (int64_t)MD * S;
    double* slls = out->sample_log_likelihoods_lls ? out->sample_log_likelihoods_lls + q0 * S : c->d_mlls;
    int32_t* partners = c->d_partners;

    LoglikArgs la = loglik_args(c, npix);
    la.acache = c->d_acache; la.partners = partners; la.active = c->d_active;

    MultiLevelArgs ma;
    ma.meta = c->d_meta; ma.S = S; ma.max_dlas = MD; ma.partners = partners;
    ma.partners_in = base_in ? base_in + q0 * 3 * S : nullptr;
    ma.active = c->d_active; ma.offset_samples = c->d_offset; ma.log_nhi_samples = c->d_log_nhi;
    ma.uniforms = c->d_uniforms; ma.min_z_separation = min_z_sep; ma.cum_scratch = c->d_cum;
    ma.map_z = out->MAP_z_dlas + q0 * MD * MD; ma.map_log_nhi = out->MAP_log_nhis + q0 * MD * MD;
    ma.map_inds = out->MAP_inds + q0 * MD * MD;

    // level 1 (+ null model), absorption rows cached                         ...meanflux.m:342-361
    la.nhi_samples = c->d_nhi; la.sample_log_likelihoods = sll; la.sll_stride = sll_stride;
    la.log_likelihoods_no_dla = out->log_likelihoods_no_dla + q0; la.num_partners = 0;
    if ((rc = launch_split<1>(c, la, nq, nq_f64, st))) return rc;
    // sub-DLA model                                                           ...meanflux.m:365-380
    la.nhi_samples = c->d_lls_nhi; la.sample_log_likelihoods = slls; la.sll_stride = S;
    la.log_likelihoods_no_dla = nullptr;
    if ((rc = launch_split<0>(c, la, nq, nq_f64, st))) return rc;
    ma.level = 0; ma.sll = slls; ma.sll_stride = S; ma.log_likelihoods = out->log_likelihoods_lls + q0;
    multi_level_kernel<<<nq, NTHREADS, 0, st>>>(ma);
    c->launches++;
    for (int level = 1; level <= MD; ++level) {
      if (level >= 2) {
        la.nhi_samples = c->d_nhi; la.sample_log_likelihoods = sll + (int64_t)(level - 1) * S;
        la.sll_stride = sll_stride; la.log_likelihoods_no_dla = nullptr; la.num_partners = level - 1;
        if ((rc = launch_split<2>(c, la, nq, nq_f64, st))) return rc;
      }
      ma.level = level; ma.sll = sll + (int64_t)(level - 1) * S; ma.sll_stride = sll_stride;
      ma.log_likelihoods = out->log_likelihoods_dla + q0 * MD;
      multi_level_kernel<<<nq, NTHREADS, 0, st>>>(ma);
      c->launches++;
      CUDA_TRY(cudaGetLastError(), c->err);
    }
    if (out->base_sample_inds && MD > 1) {   // [Q x (MD-1) x S] <- workspace [nq x 3 x S]
      CUDA_TRY(cudaMemcpy2DAsync(out->base_sample_inds + q0 * (MD - 1) * S, (size_t)(MD - 1) * S * sizeof(int32_t),
                                 partners, (size_t)3 * S * sizeof(int32_t), (size_t)(MD - 1) * S * sizeof(int32_t), nq,
                                 cudaMemcpyDeviceToDevice, st), c->err);
    }
    MultiPosteriorArgs mp;
    mp.meta = c->d_meta; mp.Q = nq; mp.max_dlas = MD; mp.Z_lls = c->Z_lls; mp.Z_dla = c->Z_dla;
    mp.log_likelihoods_no_dla = out->log_likelihoods_no_dla + q0; mp.log_likelihoods_lls = out->log_likelihoods_lls + q0;
    mp.log_likelihoods_dla = out->log_likelihoods_dla + q0 * MD;
    mp.min_z_dlas = out->min_z_dlas + q0; mp.max_z_dlas = out->max_z_dlas + q0;
    mp.log_priors_no_dla = out->log_priors_no_dla + q0; mp.log_priors_lls = out->log_priors_lls + q0;
    mp.log_priors_dla = out->log_priors_dla + q0 * MD;
    mp.log_posteriors_no_dla = out->log_posteriors_no_dla + q0; mp.log_posteriors_lls = out->log_posteriors_lls + q0;
    mp.log_posteriors_dla = out->log_posteriors_dla + q0 * MD;
    mp.model_posteriors = out->model_posteriors + q0 * (MD + 2);
    mp.p_no_dlas = out->p_no_dlas + q0; mp.p_lls = out->p_lls + q0; mp.p_dlas = out->p_dlas + q0;
    multi_posterior_kernel<<<(nq + 127) / 128, 128, 0, st>>>(mp);
    c->launches++;
    CUDA_TRY(cudaGetLastError(), c->err);
  }
  return GPDLA_OK;
}

int gpdla_process_qsos_multi(gpdla_ctx* c, int64_t Q, int64_t L_max, const double* wavelengths, const double* flux,
                             const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                             const double* z_qsos, int32_t max_dlas, const int32_t* base_in,
                             const gpdla_multi_results* out) {
  if (!c) return GPDLA_ERR_INVALID;
  if (Q < 0 || L_max < 1 || !out || max_dlas < 1 || max_dlas > 4) {
    c->err = "gpdla_process_qsos_multi: invalid arguments (1 <= max_dlas <= 4)";
    return GPDLA_ERR_INVALID;
  }
  if (Q == 0) return GPDLA_OK;
  if (!wavelengths || !flux || !noise_variance || !pixel_mask || !lengths || !z_qsos) {
    c->err = "gpdla_process_qsos_multi: NULL input array";
    return GPDLA_ERR_INVALID;
  }
  DeviceGuard guard(c->device);
  const size_t QL = (size_t)Q * L_max, S = (size_t)c->S, MD = max_dlas;
  // device staging: inputs, then every output (small ones always, large ones when requested)
  struct Item { void** dev; const void* host_in; void* host_out; size_t bytes; };
  double *d_w, *d_f, *d_v, *d_z; uint8_t* d_m; int32_t *d_len, *d_bin = nullptr;
  gpdla_multi_results dr;
  memset(&dr, 0, sizeof dr);
  std::vector<Item> items = {
      {(void**)&d_w, wavelengths, nullptr, QL * 8}, {(void**)&d_f, flux, nullptr, QL * 8},
      {(void**)&d_v, noise_variance, nullptr, QL * 8}, {(void**)&d_z, z_qsos, nullptr, (size_t)Q * 8},
      {(void**)&d_len, lengths, nullptr, (size_t)Q * 4}, {(void**)&d_m, pixel_mask, nullptr, QL},
      {(void**)&dr.min_z_dlas, nullptr, out->min_z_dlas, (size_t)Q * 8},
      {(void**)&dr.max_z_dlas, nullptr, out->max_z_dlas, (size_t)Q * 8},
      {(void**)&dr.log_priors_no_dla, nullptr, out->log_priors_no_dla, (size_t)Q * 8},
      {(void**)&dr.log_priors_lls, nullptr, out->log_priors_lls, (size_t)Q * 8},
      {(void**)&dr.log_priors_dla, nullptr, out->log_priors_dla, (size_t)Q * MD * 8},
      {(void**)&dr.log_likelihoods_no_dla, nullptr, out->log_likelihoods_no_dla, (size_t)Q * 8},
      {(void**)&dr.log_likelihoods_lls, nullptr, out->log_likelihoods_lls, (size_t)Q * 8},
      {(void**)&dr.log_likelihoods_dla, nullptr, out->log_likelihoods_dla, (size_t)Q * MD * 8},
      {(void**)&dr.log_posteriors_no_dla, nullptr, out->log_posteriors_no_dla, (size_t)Q * 8},
      {(void**)&dr.log_posteriors_lls, nullptr, out->log_posteriors_lls, (size_t)Q * 8},
      {(void**)&dr.log_posteriors_dla, nullptr, out->log_posteriors_dla, (size_t)Q * MD * 8},
      {(void**)&dr.model_posteriors, nullptr, out->model_posteriors, (size_t)Q * (MD + 2) * 8},
      {(void**)&dr.p_no_dlas, nullptr, out->p_no_dlas, (size_t)Q * 8},
      {(void**)&dr.p_lls, nullptr, out->p_lls, (size_t)Q * 8},
      {(void**)&dr.p_dlas, nullptr, out->p_dlas, (size_t)Q * 8},
      {(void**)&dr.MAP_z_dlas, nullptr, out->MAP_z_dlas, (size_t)Q * MD * MD * 8},
      {(void**)&dr.MAP_log_nhis, nullptr, out->MAP_log_nhis, (size_t)Q * MD * MD * 8},
      {(void**)&dr.MAP_inds, nullptr, out->MAP_inds, (size_t)Q * MD * MD * 8}};
  if (out->sample_log_likelihoods_dla)
    items.push_back({(void**)&dr.sample_log_likelihoods_dla, nullptr, out->sample_log_likelihoods_dla, (size_t)Q * MD * S * 8});
  if (out->sample_log_likelihoods_lls)
    items.push_back({(void**)&dr.sample_log_likelihoods_lls, nullptr, out->sample_log_likelihoods_lls, (size_t)Q * S * 8});
  if (out->base_sample_inds && MD > 1)
    items.push_back({(void**)&dr.base_sample_inds, nullptr, out->base_sample_inds, (size_t)Q * (MD - 1) * S * 4});
  std::vector<int32_t> bin3;
  if (base_in && MD > 1) {   // caller's [Q x (MD-1) x S] -> internal [Q x 3 x S]
    bin3.assign((size_t)Q * 3 * S, 0);
    for (size_t q = 0; q < (size_t)Q; ++q)
      memcpy(&bin3[q * 3 * S], base_in + q * (MD - 1) * S, (MD - 1) * S * sizeof(int32_t));
    items.push_back({(void**)&d_bin, bin3.data(), nullptr, bin3.size() * 4});
  }
  size_t bytes = 256;
  for (auto& it : items) bytes += (it.bytes + 255) / 256 * 256;
  if (c->st_bytes < bytes) {
    cudaFree(c->d_stage); c->d_stage = nullptr; c->st_bytes = 0;
    CUDA_TRY(cudaMalloc(&c->d_stage, bytes), c->err);
    c->st_bytes = bytes;
  }
  char* p = (char*)c->d_stage;
  cudaStream_t st = c->stream;
  for (auto& it : items) {
    *it.dev = p; p += (it.bytes + 255) / 256 * 256;
    if (it.host_in) CUDA_TRY(cudaMemcpyAsync(*it.dev, it.host_in, it.bytes, cudaMemcpyHostToDevice, st), c->err);
  }
  int rc = gpdla_process_qsos_multi_device(c, Q, L_max, d_w, d_f, d_v, d_m, d_len, d_z, max_dlas, d_bin, &dr, st);
  if (rc) return rc;
  for (auto& it : items)
    if (it.host_out) CUDA_TRY(cudaMemcpyAsync(it.host_out, *it.dev, it.bytes, cudaMemcpyDeviceToHost, st), c->err);
  CUDA_TRY(cudaStreamSynchronize(st), c->err);
  return GPDLA_OK;
}

int gpdla_voigt_batch_device(const double* lambdas, int64_t num_points, const double* z, const double* N, int64_t S,
                             int32_t num_lines, double* profile, void* stream) {
  if (!lambdas || !z || !N || !profile || num_points < 7 || S < 1 || S > 2147483647LL || (num_points - 6 + NTHREADS - 1) / NTHREADS > 65535 || num_lines < 1 ||
      num_lines > GPDLA_MAX_LINES) {
    g_err = "gpdla_voigt: invalid arguments (need 7 <= num_points <= 16.7M, 1 <= num_lines <= 31, S >= 1)";
    return GPDLA_ERR_INVALID;
  }
  int rc = upload_device_constants(g_err);
  if (rc) return rc;
  const int64_t n_out = num_points - 6;
  dim3 grid((unsigned)S, (unsigned)((n_out + NTHREADS - 1) / NTHREADS));
  voigt_batch_kernel<<<grid, NTHREADS, 0, (cudaStream_t)stream>>>(lambdas, num_points, z, N, num_lines, profile);
  CUDA_TRY(cudaGetLastError(), g_err);
  return GPDLA_OK;
}

int gpdla_voigt(const double* lambdas, int64_t num_points, double z, double N, int32_t num_lines, double* profile) {
  if (!lambdas || !profile || num_points < 7 || num_lines < 1 || num_lines > GPDLA_MAX_LINES || !(z > -1.0) ||
      !isfinite(z) || !isfinite(N)) {
    g_err = "gpdla_voigt: invalid arguments (need num_points >= 7, 1 <= num_lines <= 31, finite z > -1)";
    return GPDLA_ERR_INVALID;
  }
  double* d = nullptr;
  const size_t n_out = num_points - 6;
  CUDA_TRY(cudaMalloc(&d, (num_points + n_out + 2) * sizeof(double)), g_err);
  double zn[2] = {z, N};
  cudaError_t e1 = cudaMemcpy(d, lambdas, num_points * sizeof(double), cudaMemcpyHostToDevice);
  cudaError_t e2 = cudaMemcpy(d + num_points, zn, sizeof zn, cudaMemcpyHostToDevice);
  int rc = GPDLA_ERR_CUDA;
  if (e1 == cudaSuccess && e2 == cudaSuccess) {
    rc = gpdla_voigt_batch_device(d, num_points, d + num_points, d + num_points + 1, 1, num_lines, d + num_points + 2, 0);
    if (rc == GPDLA_OK) {
      cudaError_t e3 = cudaMemcpy(profile, d + num_points + 2, n_out * sizeof(double), cudaMemcpyDeviceToHost);
      if (e3 != cudaSuccess) { g_err = cudaGetErrorString(e3); rc = GPDLA_ERR_CUDA; }
    }
  } else {
    g_err = cudaGetErrorString(e1 != cudaSuccess ? e1 : e2);
  }
  cudaFree(d);
  return rc;
}

void gpdla_default_preload_parameters(gpdla_preload_params* p) {
  p->loading_min_lambda = 910.0; p->loading_max_lambda = 1217.0;                 // set_parameters.m:21-22
  p->normalization_min_lambda = 1310.0; p->normalization_max_lambda = 1325.0;    // :29-30
  p->min_lambda = 911.75; p->max_lambda = 1215.75;                               // :33-34
  p->min_num_pixels = 200; p->reserved = 0;                                      // :26
}

int gpdla_preload_qsos_device(int64_t Q, int64_t L_in, const double* flux, const double* loglam, const double* ivar,
                              const int32_t* and_mask, const int32_t* lengths_in, const double* z_qsos,
                              const uint8_t* filter_flags_in, const gpdla_preload_params* p, int64_t L_out,
                              double* wavelengths, double* out_flux, double* noise_variance, uint8_t* pixel_mask,
                              int32_t* lengths, double* normalizers, uint8_t* filter_flags, void* stream) {
  if (Q < 0 || L_in < 1 || L_out < 1 || !p ||
      (Q > 0 && (!flux || !loglam || !ivar || !and_mask || !lengths_in || !z_qsos || !wavelengths || !out_flux ||
                 !noise_variance || !pixel_mask || !lengths || !normalizers || !filter_flags))) {
    g_err = "gpdla_preload_qsos_device: invalid arguments";
    return GPDLA_ERR_INVALID;
  }
  if (Q == 0) return GPDLA_OK;
  PreloadArgs a;
  a.flux = flux; a.loglam = loglam; a.ivar = ivar; a.and_mask = and_mask; a.lengths_in = lengths_in; a.z_qsos = z_qsos;
  a.filter_flags_in = filter_flags_in; a.L_in = L_in; a.L_out = L_out;
  a.loading_min_lambda = p->loading_min_lambda; a.loading_max_lambda = p->loading_max_lambda;
  a.normalization_min_lambda = p->normalization_min_lambda; a.normalization_max_lambda = p->normalization_max_lambda;
  a.min_lambda = p->min_lambda; a.max_lambda = p->max_lambda; a.min_num_pixels = p->min_num_pixels;
  a.wavelengths = wavelengths; a.out_flux = out_flux; a.noise_variance = noise_variance; a.pixel_mask = pixel_mask;
  a.lengths = lengths; a.normalizers = normalizers; a.filter_flags = filter_flags;
  preload_qsos_kernel<<<(unsigned)Q, PRE_THREADS, 0, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError(), g_err);
  return GPDLA_OK;
}

int gpdla_preload_qsos(int64_t Q, int64_t L_in, const double* flux, const double* loglam, const double* ivar,
                       const int32_t* and_mask, const int32_t* lengths_in, const double* z_qsos,
                       const uint8_t* filter_flags_in, const gpdla_preload_params* p, int64_t L_out,
                       double* wavelengths, double* out_flux, double* noise_variance, uint8_t* pixel_mask,
                       int32_t* lengths, double* normalizers, uint8_t* filter_flags) {
  if (Q < 0 || L_in < 1 || L_out < 1 || !p) { g_err = "gpdla_preload_qsos: invalid arguments"; return GPDLA_ERR_INVALID; }
  if (Q == 0) return GPDLA_OK;
  const size_t QI = (size_t)Q * L_in, QO = (size_t)Q * L_out;
  const size_t bytes = 3 * QI * 8 + QI * 4 + (size_t)Q * (4 + 8 + 1) + 3 * QO * 8 + QO + (size_t)Q * (4 + 8 + 1) + 256;
  char* base = nullptr;
  CUDA_TRY(cudaMalloc(&base, bytes), g_err);
  char* ptr = base;
  auto take = [&](size_t n) { char* r = ptr; ptr += (n + 15) / 16 * 16; return r; };
  double* d_f = (double*)take(QI * 8); double* d_l = (double*)take(QI * 8); double* d_i = (double*)take(QI * 8);
  double* d_z = (double*)take((size_t)Q * 8);
  double* d_ow = (double*)take(QO * 8); double* d_of = (double*)take(QO * 8); double* d_ov = (double*)take(QO * 8);
  double* d_norm = (double*)take((size_t)Q * 8);
  int32_t* d_am = (int32_t*)take(QI * 4); int32_t* d_len = (int32_t*)take((size_t)Q * 4);
  int32_t* d_olen = (int32_t*)take((size_t)Q * 4);
  uint8_t* d_om = (uint8_t*)take(QO); uint8_t* d_fin = (uint8_t*)take((size_t)Q); uint8_t* d_fout = (uint8_t*)take((size_t)Q);
  int rc = GPDLA_ERR_CUDA;
  cudaError_t e = cudaSuccess;
  auto up = [&](void* d, const void* h, size_t n) { if (e == cudaSuccess) e = cudaMemcpy(d, h, n, cudaMemcpyHostToDevice); };
  auto down = [&](void* h, const void* d, size_t n) { if (e == cudaSuccess) e = cudaMemcpy(h, d, n, cudaMemcpyDeviceToHost); };
  up(d_f, flux, QI * 8); up(d_l, loglam, QI * 8); up(d_i, ivar, QI * 8); up(d_am, and_mask, QI * 4);
  up(d_len, lengths_in, (size_t)Q * 4); up(d_z, z_qsos, (size_t)Q * 8);
  if (filter_flags_in) up(d_fin, filter_flags_in, (size_t)Q);
  if (e == cudaSuccess) {
    rc = gpdla_preload_qsos_device(Q, L_in, d_f, d_l, d_i, d_am, d_len, d_z, filter_flags_in ? d_fin : nullptr, p, L_out,
                                   d_ow, d_of, d_ov, d_om, d_olen, d_norm, d_fout, 0);
    if (rc == GPDLA_OK) {
      down(wavelengths, d_ow, QO * 8); down(out_flux, d_of, QO * 8); down(noise_variance, d_ov, QO * 8);
      down(pixel_mask, d_om, QO); down(lengths, d_olen, (size_t)Q * 4); down(normalizers, d_norm, (size_t)Q * 8);
      down(filter_flags, d_fout, (size_t)Q);
      if (e == cudaSuccess) {
        for (int64_t q = 0; q < Q; ++q)
          if (lengths[q] < 0) { g_err = "gpdla_preload_qsos: L_out too small (quasar " + std::to_string(q) + " needs " + std::to_string(-lengths[q]) + " pixels)"; rc = GPDLA_ERR_INVALID; break; }
      }
    }
  }
  if (e != cudaSuccess) { g_err = cudaGetErrorString(e); rc = GPDLA_ERR_CUDA; }
  cudaFree(base);
  return rc;
}

int gpdla_objective_lyseries_device(int64_t num_quasars, int32_t num_pixels, int32_t k, const double* centered_rest_fluxes,
                                    const double* lya_1pzs, const double* rest_noise_variances, int32_t num_forest_lines,
                                    const double* all_transition_wavelengths, const double* all_oscillator_strengths,
                                    const double* x, double* f, double* g, void* stream) {
  if (num_quasars < 0 || num_pixels < 1 || !x || !f || !g || num_forest_lines < 0 || num_forest_lines > GPDLA_MAX_LINES ||
      (num_forest_lines > 0 && (!all_transition_wavelengths || !all_oscillator_strengths)) ||
      (num_quasars > 0 && (!centered_rest_fluxes || !lya_1pzs || !rest_noise_variances))) {
    g_err = "gpdla_objective_device: invalid arguments";
    return GPDLA_ERR_INVALID;
  }
  if (!rank_supported(k)) {
    g_err = "gpdla_objective_device: rank k=" + std::to_string(k) + " not compiled in (available: 10, 20, 40)";
    return GPDLA_ERR_UNSUPPORTED;
  }
  cudaStream_t st = (cudaStream_t)stream;
  ObjectiveArgs a;
  memset(&a, 0, sizeof a);
  a.y = centered_rest_fluxes; a.lya_1pz = lya_1pzs; a.nv = rest_noise_variances; a.x = x; a.f = f; a.g = g;
  a.N = num_quasars; a.P = num_pixels; a.num_forest_lines = num_forest_lines;
  for (int l = 0; l < num_forest_lines; ++l) { a.tw[l] = all_transition_wavelengths[l]; a.osc[l] = all_oscillator_strengths[l]; }
  int rc = GPDLA_OK;
  GPDLA_FOR_RANK(k, (rc = launch_objective<K>(a, st)));
  if (rc) return rc;
  objective_prior_kernel<<<1, 1, 0, st>>>(x, g, (int64_t)num_pixels * (k + 1));
  CUDA_TRY(cudaGetLastError(), g_err);
  return GPDLA_OK;
}

int gpdla_objective_device(int64_t num_quasars, int32_t num_pixels, int32_t k, const double* centered_rest_fluxes,
                           const double* lya_1pzs, const double* rest_noise_variances, const double* x, double* f,
                           double* g, void* stream) {
  return gpdla_objective_lyseries_device(num_quasars, num_pixels, k, centered_rest_fluxes, lya_1pzs, rest_noise_variances, 0,
                                         nullptr, nullptr, x, f, g, stream);
}

int gpdla_objective_lyseries(int64_t num_quasars, int32_t num_pixels, int32_t k, const double* centered_rest_fluxes,
                             const double* lya_1pzs, const double* rest_noise_variances, int32_t num_forest_lines,
                             const double* all_transition_wavelengths, const double* all_oscillator_strengths, const double* x,
                             double* f, double* g) {
  if (num_quasars < 0 || num_pixels < 1 || k < 1 || !x || !f || !g) { g_err = "gpdla_objective: invalid arguments"; return GPDLA_ERR_INVALID; }
  const size_t NP = (size_t)num_quasars * num_pixels, nx = (size_t)num_pixels * (k + 1) + 3;
  double* base = nullptr;
  CUDA_TRY(cudaMalloc(&base, (3 * NP + 2 * nx + 2) * sizeof(double)), g_err);
  double *d_y = base, *d_z = base + NP, *d_v = base + 2 * NP, *d_x = base + 3 * NP, *d_g = d_x + nx, *d_f = d_g + nx;
  cudaError_t e = cudaSuccess;
  auto up = [&](void* d, const void* h, size_t n) { if (e == cudaSuccess && n) e = cudaMemcpy(d, h, n, cudaMemcpyHostToDevice); };
  up(d_y, centered_rest_fluxes, NP * 8); up(d_z, lya_1pzs, NP * 8); up(d_v, rest_noise_variances, NP * 8); up(d_x, x, nx * 8);
  int rc = GPDLA_ERR_CUDA;
  if (e == cudaSuccess) {
    rc = gpdla_objective_lyseries_device(num_quasars, num_pixels, k, d_y, d_z, d_v, num_forest_lines, all_transition_wavelengths,
                                         all_oscillator_strengths, d_x, d_f, d_g, 0);
    if (rc == GPDLA_OK) {
      e = cudaMemcpy(f, d_f, 8, cudaMemcpyDeviceToHost);
      if (e == cudaSuccess) e = cudaMemcpy(g, d_g, nx * 8, cudaMemcpyDeviceToHost);
    }
  }
  if (e != cudaSuccess) { g_err = cudaGetErrorString(e); rc = GPDLA_ERR_CUDA; }
  cudaFree(base);
  return rc;
}

int gpdla_objective(int64_t num_quasars, int32_t num_pixels, int32_t k, const double* centered_rest_fluxes,
                    const double* lya_1pzs, const double* rest_noise_variances, const double* x, double* f, double* g) {
  return gpdla_objective_lyseries(num_quasars, num_pixels, k, centered_rest_fluxes, lya_1pzs, rest_noise_variances, 0, nullptr,
                                  nullptr, x, f, g);
}

// ---- training set + pairwise covariance (learn_qso_model.m:36-95) ----

// rows of X per split of the covariance: a function of N alone, so that the summation order (and the bits) do not depend
// on the device; up to 8 splits give 210 x 8 CTAs for the 1217-pixel grid
static int64_t cov_rows_per_split(int64_t N) {
  const int64_t nsplit = std::min<int64_t>(8, std::max<int64_t>(1, (N + 2047) / 2048));
  return std::max<int64_t>(COV_CHUNK, ((N + nsplit - 1) / nsplit + COV_CHUNK - 1) / COV_CHUNK * COV_CHUNK);
}

// one column statistic of an [N x P] matrix: fixed row blocks, then their sum in block order
static int column_stat(double* X, int64_t N, int P, int mode, const double* centre, double* out, int32_t* count,
                       cudaStream_t st) {
  const int nblocks = (int)((N + COL_ROWS - 1) / COL_ROWS);
  double* psum = nullptr;
  int32_t* pcnt = nullptr;
  if (nblocks > 0) {
    CUDA_TRY(cudaMallocAsync(&psum, (size_t)nblocks * P * (sizeof(double) + sizeof(int32_t)), st), g_err);
    pcnt = reinterpret_cast<int32_t*>(psum + (size_t)nblocks * P);
    column_partial_kernel<<<dim3((P + COL_THREADS - 1) / COL_THREADS, nblocks), COL_THREADS, 0, st>>>(X, N, P, mode, centre,
                                                                                                     psum, pcnt);
  }
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) {
    column_finish_kernel<<<(P + 127) / 128, 128, 0, st>>>(psum, pcnt, nblocks, P, mode, out, count);
    e = cudaGetLastError();
  }
  if (psum) {                                     // freed on the error path too
    const cudaError_t ef = cudaFreeAsync(psum, st);
    if (e == cudaSuccess) e = ef;
  }
  if (e != cudaSuccess) { g_err = std::string("column_stat: ") + cudaGetErrorString(e); return GPDLA_ERR_CUDA; }
  return GPDLA_OK;
}

// The plain (learn_qso_model.m) and the Lyman-series (learn_qso_model_meanflux.m) training set share their checks,
// buffers and reductions; num_forest_lines < 0 selects the plain kernel, 0..31 the mean-flux one.
static int training_set_device_impl(const char* fn, int64_t N, int64_t L_max, const double* wavelengths,
                                    const double* flux, const double* noise_variance, const uint8_t* pixel_mask,
                                    const int32_t* lengths, const double* z_qsos, const double* rest_wavelengths,
                                    int32_t num_pixels, double lya_wavelength, double max_noise_variance,
                                    int32_t num_forest_lines, double* lya_1pzs, double* centered_rest_fluxes,
                                    double* rest_noise_variances, double* lya_absorption, double* mu, double* std_dev,
                                    int32_t* num_observed, void* stream) {
  if (N < 0 || N > INT32_MAX || L_max < 1 || num_pixels < 1 || !rest_wavelengths || !mu || !std_dev || !num_observed ||
      !(lya_wavelength > 0.0) || num_forest_lines > MAX_LINES ||
      (N > 0 && (!wavelengths || !flux || !noise_variance || !pixel_mask || !lengths || !z_qsos || !lya_1pzs ||
                 !centered_rest_fluxes || !rest_noise_variances))) {
    g_err = std::string(fn) + ": invalid arguments";
    return GPDLA_ERR_INVALID;
  }
  const bool lyseries = num_forest_lines >= 0;
  const size_t smem = training_set_smem_bytes(L_max, lyseries);
  int dev = 0, optin = 0;
  CUDA_TRY(cudaGetDevice(&dev), g_err);
  CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev), g_err);
  if (smem > (size_t)optin) {
    g_err = std::string(fn) + ": L_max = " + std::to_string(L_max) + " does not fit in shared memory (at most " +
            std::to_string(optin / (smem / L_max)) + " pixels)";
    return GPDLA_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (N > 0) {
    TrainingArgs a;
    a.wavelengths = wavelengths; a.flux = flux; a.noise_variance = noise_variance; a.pixel_mask = pixel_mask;
    a.lengths = lengths; a.z_qsos = z_qsos; a.rest = rest_wavelengths; a.N = N; a.L_max = L_max; a.P = num_pixels;
    a.lya_wavelength = lya_wavelength; a.max_noise_variance = max_noise_variance;
    a.lya_1pzs = lya_1pzs; a.rest_fluxes = centered_rest_fluxes; a.rest_noise_variances = rest_noise_variances;
    fill_forest_constants(&a.forest, lyseries ? num_forest_lines : 0);
    for (int l = 0; l < MAX_LINES; ++l) a.lya_over_wavelength[l] = lya_wavelength / a.forest.wavelength[l];
    a.lya_absorption = lya_absorption;
    if (lyseries) {
      CUDA_TRY(cudaFuncSetAttribute(training_set_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), g_err);
      training_set_kernel<true><<<(unsigned)N, TS_THREADS, smem, st>>>(a);
    } else {
      CUDA_TRY(cudaFuncSetAttribute(training_set_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), g_err);
      training_set_kernel<false><<<(unsigned)N, TS_THREADS, smem, st>>>(a);
    }
    CUDA_TRY(cudaGetLastError(), g_err);
  }
  int rc;
  // mu = nanmean(rest_fluxes), centred in place (:71-75); std_dev = nanstd of the centred fluxes (:82-95), whose own
  // nanmean is kept in std_dev until the last pass overwrites it
  if ((rc = column_stat(centered_rest_fluxes, N, num_pixels, COL_MEAN, nullptr, mu, num_observed, st))) return rc;
  if ((rc = column_stat(centered_rest_fluxes, N, num_pixels, COL_CENTRE, mu, std_dev, nullptr, st))) return rc;
  if ((rc = column_stat(centered_rest_fluxes, N, num_pixels, COL_SQDEV, std_dev, std_dev, nullptr, st))) return rc;
  return GPDLA_OK;
}

static int training_set_host_impl(const char* fn, int64_t N, int64_t L_max, const double* wavelengths,
                                  const double* flux, const double* noise_variance, const uint8_t* pixel_mask,
                                  const int32_t* lengths, const double* z_qsos, const double* rest_wavelengths,
                                  int32_t num_pixels, double lya_wavelength, double max_noise_variance,
                                  int32_t num_forest_lines, double* lya_1pzs, double* centered_rest_fluxes,
                                  double* rest_noise_variances, double* lya_absorption, double* mu, double* std_dev,
                                  int32_t* num_observed) {
  if (N < 0 || N > INT32_MAX || L_max < 1 || num_pixels < 1 || !rest_wavelengths || !mu || !std_dev || !num_observed ||
      num_forest_lines > MAX_LINES ||
      (N > 0 && (!wavelengths || !flux || !noise_variance || !pixel_mask || !lengths || !z_qsos || !lya_1pzs ||
                 !centered_rest_fluxes || !rest_noise_variances))) {
    g_err = std::string(fn) + ": invalid arguments";
    return GPDLA_ERR_INVALID;
  }
  for (int64_t i = 0; i < N; ++i)
    if (lengths[i] < 0 || lengths[i] > L_max) {
      g_err = std::string(fn) + ": lengths[" + std::to_string(i) + "] = " + std::to_string(lengths[i]) +
              " is outside [0, L_max = " + std::to_string(L_max) + "]";
      return GPDLA_ERR_INVALID;
    }
  for (int32_t p = 1; p < num_pixels; ++p)
    if (!(rest_wavelengths[p] > rest_wavelengths[p - 1])) {
      g_err = std::string(fn) + ": rest_wavelengths must be strictly increasing (entry " + std::to_string(p) + ")";
      return GPDLA_ERR_INVALID;
    }
  const size_t NL = (size_t)N * L_max, NP = (size_t)N * num_pixels, P = (size_t)num_pixels;
  const size_t NA = lya_absorption ? NP : 0;
  const size_t bytes = 3 * NL * 8 + NL + N * (4 + 8) + P * 8 + (3 * NP + NA) * 8 + 2 * P * 8 + P * 4 + 256;
  char* base = nullptr;
  CUDA_TRY(cudaMalloc(&base, bytes), g_err);
  char* ptr = base;
  auto take = [&](size_t n) { char* r = ptr; ptr += (n + 15) / 16 * 16; return r; };
  double* d_w = (double*)take(NL * 8); double* d_f = (double*)take(NL * 8); double* d_v = (double*)take(NL * 8);
  double* d_z = (double*)take((size_t)N * 8); double* d_rest = (double*)take(P * 8);
  double* d_lya = (double*)take(NP * 8); double* d_y = (double*)take(NP * 8); double* d_nv = (double*)take(NP * 8);
  double* d_abs = lya_absorption ? (double*)take(NA * 8) : nullptr;
  double* d_mu = (double*)take(P * 8); double* d_sd = (double*)take(P * 8);
  int32_t* d_len = (int32_t*)take((size_t)N * 4); int32_t* d_cnt = (int32_t*)take(P * 4);
  uint8_t* d_m = (uint8_t*)take(NL);
  cudaError_t e = cudaSuccess;
  auto up = [&](void* d, const void* h, size_t n) { if (e == cudaSuccess && n) e = cudaMemcpy(d, h, n, cudaMemcpyHostToDevice); };
  auto down = [&](void* h, const void* d, size_t n) { if (e == cudaSuccess && n) e = cudaMemcpy(h, d, n, cudaMemcpyDeviceToHost); };
  up(d_w, wavelengths, NL * 8); up(d_f, flux, NL * 8); up(d_v, noise_variance, NL * 8); up(d_m, pixel_mask, NL);
  up(d_len, lengths, (size_t)N * 4); up(d_z, z_qsos, (size_t)N * 8); up(d_rest, rest_wavelengths, P * 8);
  int rc = GPDLA_ERR_CUDA;
  if (e == cudaSuccess) {
    rc = training_set_device_impl(fn, N, L_max, d_w, d_f, d_v, d_m, d_len, d_z, d_rest, num_pixels, lya_wavelength,
                                  max_noise_variance, num_forest_lines, d_lya, d_y, d_nv, d_abs, d_mu, d_sd, d_cnt,
                                  nullptr);
    if (rc == GPDLA_OK) {
      down(lya_1pzs, d_lya, NP * 8); down(centered_rest_fluxes, d_y, NP * 8); down(rest_noise_variances, d_nv, NP * 8);
      if (d_abs) down(lya_absorption, d_abs, NA * 8);
      down(mu, d_mu, P * 8); down(std_dev, d_sd, P * 8); down(num_observed, d_cnt, P * 4);
      if (e == cudaSuccess) {
        for (int32_t p = 0; p < num_pixels; ++p)
          if (num_observed[p] < 2) {
            char buf[256];
            snprintf(buf, sizeof buf, "%s: rest pixel %d (%.2f A) is observed in %d spectra, fewer than 2",
                     fn, p, rest_wavelengths[p], num_observed[p]);
            g_err = buf;
            rc = GPDLA_ERR_INVALID;
            break;
          }
      }
    }
  }
  if (e != cudaSuccess) { g_err = cudaGetErrorString(e); rc = GPDLA_ERR_CUDA; }
  cudaFree(base);
  return rc;
}

int gpdla_training_set_device(int64_t N, int64_t L_max, const double* wavelengths, const double* flux,
                              const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                              const double* z_qsos, const double* rest_wavelengths, int32_t num_pixels,
                              double lya_wavelength, double max_noise_variance, double* lya_1pzs,
                              double* centered_rest_fluxes, double* rest_noise_variances, double* mu, double* std_dev,
                              int32_t* num_observed, void* stream) {
  return training_set_device_impl("gpdla_training_set_device", N, L_max, wavelengths, flux, noise_variance, pixel_mask,
                                  lengths, z_qsos, rest_wavelengths, num_pixels, lya_wavelength, max_noise_variance, -1,
                                  lya_1pzs, centered_rest_fluxes, rest_noise_variances, nullptr, mu, std_dev,
                                  num_observed, stream);
}

int gpdla_training_set(int64_t N, int64_t L_max, const double* wavelengths, const double* flux,
                       const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                       const double* z_qsos, const double* rest_wavelengths, int32_t num_pixels, double lya_wavelength,
                       double max_noise_variance, double* lya_1pzs, double* centered_rest_fluxes,
                       double* rest_noise_variances, double* mu, double* std_dev, int32_t* num_observed) {
  return training_set_host_impl("gpdla_training_set", N, L_max, wavelengths, flux, noise_variance, pixel_mask, lengths,
                                z_qsos, rest_wavelengths, num_pixels, lya_wavelength, max_noise_variance, -1, lya_1pzs,
                                centered_rest_fluxes, rest_noise_variances, nullptr, mu, std_dev, num_observed);
}

int gpdla_training_set_lyseries_device(int64_t N, int64_t L_max, const double* wavelengths, const double* flux,
                                       const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                                       const double* z_qsos, const double* rest_wavelengths, int32_t num_pixels,
                                       double lya_wavelength, double max_noise_variance, int32_t num_forest_lines,
                                       double* lya_1pzs, double* centered_rest_fluxes, double* rest_noise_variances,
                                       double* lya_absorption, double* mu, double* std_dev, int32_t* num_observed,
                                       void* stream) {
  if (num_forest_lines < 0 || num_forest_lines > MAX_LINES) {
    g_err = "gpdla_training_set_lyseries_device: num_forest_lines = " + std::to_string(num_forest_lines) +
            " is outside [0, 31]";
    return GPDLA_ERR_INVALID;
  }
  return training_set_device_impl("gpdla_training_set_lyseries_device", N, L_max, wavelengths, flux, noise_variance,
                                  pixel_mask, lengths, z_qsos, rest_wavelengths, num_pixels, lya_wavelength,
                                  max_noise_variance, num_forest_lines, lya_1pzs, centered_rest_fluxes,
                                  rest_noise_variances, lya_absorption, mu, std_dev, num_observed, stream);
}

int gpdla_training_set_lyseries(int64_t N, int64_t L_max, const double* wavelengths, const double* flux,
                                const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                                const double* z_qsos, const double* rest_wavelengths, int32_t num_pixels,
                                double lya_wavelength, double max_noise_variance, int32_t num_forest_lines,
                                double* lya_1pzs, double* centered_rest_fluxes, double* rest_noise_variances,
                                double* lya_absorption, double* mu, double* std_dev, int32_t* num_observed) {
  if (num_forest_lines < 0 || num_forest_lines > MAX_LINES) {
    g_err = "gpdla_training_set_lyseries: num_forest_lines = " + std::to_string(num_forest_lines) +
            " is outside [0, 31]";
    return GPDLA_ERR_INVALID;
  }
  return training_set_host_impl("gpdla_training_set_lyseries", N, L_max, wavelengths, flux, noise_variance, pixel_mask,
                                lengths, z_qsos, rest_wavelengths, num_pixels, lya_wavelength, max_noise_variance,
                                num_forest_lines, lya_1pzs, centered_rest_fluxes, rest_noise_variances, lya_absorption,
                                mu, std_dev, num_observed);
}

int gpdla_row_nanmedian_fill_device(int64_t N, int32_t P, const double* X, double* out, void* stream) {
  if (N < 0 || N > INT32_MAX || P < 1 || P > MED_MAX_P || !out || (N > 0 && !X)) {
    g_err = "gpdla_row_nanmedian_fill_device: invalid arguments (N >= 0, 1 <= P <= " + std::to_string(MED_MAX_P) + ")";
    return GPDLA_ERR_INVALID;
  }
  if (N == 0) return GPDLA_OK;
  const int S = median_sort_size(P);
  const size_t smem = (size_t)S * sizeof(uint64_t);
  CUDA_TRY(cudaFuncSetAttribute(row_nanmedian_fill_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), g_err);
  row_nanmedian_fill_kernel<<<(unsigned)N, MED_THREADS, smem, (cudaStream_t)stream>>>(X, P, S, out);
  CUDA_TRY(cudaGetLastError(), g_err);
  return GPDLA_OK;
}

int gpdla_row_nanmedian_fill(int64_t N, int32_t P, const double* X, double* out) {
  if (N < 0 || N > INT32_MAX || P < 1 || P > MED_MAX_P || !out || (N > 0 && !X)) {
    g_err = "gpdla_row_nanmedian_fill: invalid arguments (N >= 0, 1 <= P <= " + std::to_string(MED_MAX_P) + ")";
    return GPDLA_ERR_INVALID;
  }
  const size_t NP = (size_t)N * P;
  if (NP == 0) return GPDLA_OK;
  double* d_x = nullptr;
  CUDA_TRY(cudaMalloc(&d_x, NP * 8), g_err);
  cudaError_t e = cudaMemcpy(d_x, X, NP * 8, cudaMemcpyHostToDevice);
  int rc = GPDLA_ERR_CUDA;
  if (e == cudaSuccess) {
    rc = gpdla_row_nanmedian_fill_device(N, P, d_x, d_x, nullptr);          // in place
    if (rc == GPDLA_OK) e = cudaMemcpy(out, d_x, NP * 8, cudaMemcpyDeviceToHost);
  }
  if (e != cudaSuccess) { g_err = cudaGetErrorString(e); rc = GPDLA_ERR_CUDA; }
  cudaFree(d_x);
  return rc;
}

int gpdla_pairwise_covariance_device(int64_t N, int32_t P, const double* X, double* cov, int32_t* counts, void* stream) {
  if (N < 0 || N > INT32_MAX || P < 1 || !cov || !counts || (N > 0 && !X)) {
    g_err = "gpdla_pairwise_covariance_device: invalid arguments";
    return GPDLA_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int tiles_1d = (P + COV_TILE - 1) / COV_TILE;
  const int ntile = tiles_1d * (tiles_1d + 1) / 2;
  const int64_t rps = cov_rows_per_split(N);
  const int nsplit = (int)std::max<int64_t>(1, (N + rps - 1) / rps);
  const size_t tile_elems = (size_t)nsplit * ntile * COV_TILE * COV_TILE;
  double* mean = nullptr;
  CUDA_TRY(cudaMallocAsync(&mean, (size_t)P * (8 + 4) + tile_elems * (8 + 4) + 64, st), g_err);   // mean, counts, partials
  int32_t* mcount = reinterpret_cast<int32_t*>(mean + P);
  double* psum = mean + ((size_t)P + (P + 1) / 2 + 1) / 2 * 2;   // 16-byte aligned: the tile kernel stores double2
  int32_t* pcnt = reinterpret_cast<int32_t*>(psum + tile_elems);
  int rc = column_stat(const_cast<double*>(X), N, P, COL_MEAN, nullptr, mean, mcount, st);   // COL_MEAN only reads X
  cudaError_t e = cudaSuccess;
  if (rc == GPDLA_OK) {
    CovArgs a;
    a.X = X; a.mean = mean; a.N = N; a.P = P; a.ntile = ntile; a.rows_per_split = rps; a.psum = psum; a.pcnt = pcnt;
    pairwise_cov_tile_kernel<<<dim3(ntile, nsplit), COV_THREADS, 0, st>>>(a);
    e = cudaGetLastError();
    if (e == cudaSuccess) {
      const int64_t PP = (int64_t)P * P;
      pairwise_cov_finish_kernel<<<(unsigned)((PP + 255) / 256), 256, 0, st>>>(psum, pcnt, nsplit, ntile, P, cov, counts);
      e = cudaGetLastError();
    }
  }
  const cudaError_t ef = cudaFreeAsync(mean, st);  // freed on the error paths too
  if (rc != GPDLA_OK) return rc;
  if (e == cudaSuccess) e = ef;
  if (e != cudaSuccess) {
    g_err = std::string("gpdla_pairwise_covariance_device: ") + cudaGetErrorString(e);
    return GPDLA_ERR_CUDA;
  }
  return GPDLA_OK;
}

int gpdla_pairwise_covariance(int64_t N, int32_t P, const double* X, double* cov, int32_t* counts) {
  if (N < 0 || N > INT32_MAX || P < 1 || !cov || !counts || (N > 0 && !X)) {
    g_err = "gpdla_pairwise_covariance: invalid arguments";
    return GPDLA_ERR_INVALID;
  }
  const size_t NP = (size_t)N * P, PP = (size_t)P * P;
  char* base = nullptr;
  CUDA_TRY(cudaMalloc(&base, NP * 8 + PP * 12 + 64), g_err);
  double* d_x = (double*)base;
  double* d_c = d_x + NP;
  int32_t* d_n = (int32_t*)(d_c + PP);
  cudaError_t e = cudaSuccess;
  if (NP) e = cudaMemcpy(d_x, X, NP * 8, cudaMemcpyHostToDevice);
  int rc = GPDLA_ERR_CUDA;
  if (e == cudaSuccess) {
    rc = gpdla_pairwise_covariance_device(N, P, d_x, d_c, d_n, nullptr);
    if (rc == GPDLA_OK) {
      e = cudaMemcpy(cov, d_c, PP * 8, cudaMemcpyDeviceToHost);
      if (e == cudaSuccess) e = cudaMemcpy(counts, d_n, PP * 4, cudaMemcpyDeviceToHost);
    }
  }
  if (e != cudaSuccess) { g_err = cudaGetErrorString(e); rc = GPDLA_ERR_CUDA; }
  cudaFree(base);
  return rc;
}

// ---- population statistics of the single-DLA catalogue (CDDF_analysis/calc_cddf.py) ----

// the checks both statistics entries make before any CUDA call
static int stats_check(const char* fn, int64_t Q, int64_t S, const double* ll, const double* p_dlas,
                       const double* min_z_dlas, const double* max_z_dlas, const double* offset_samples,
                       const double* log_nhi_samples, const double* nhi_samples, int32_t n_z, const double* z_edges,
                       int32_t n_nhi, const double* log_nhi_edges, double dla_log_nhi_min, double omega_m,
                       const double* sums) {
  auto fail = [&](const std::string& why) { g_err = std::string(fn) + ": " + why; return GPDLA_ERR_INVALID; };
  if (Q < 0 || Q > INT32_MAX || S < 1 || S > INT32_MAX) return fail("Q must lie in [0, 2^31) and S in [1, 2^31)");
  if (n_z < 1 || n_z > STAT_MAX_Z)
    return fail("n_z = " + std::to_string(n_z) + " is outside [1, " + std::to_string(STAT_MAX_Z) + "]");
  if (n_nhi < 1 || n_nhi > STAT_MAX_NHI)
    return fail("n_nhi = " + std::to_string(n_nhi) + " is outside [1, " + std::to_string(STAT_MAX_NHI) + "]");
  if (!z_edges || !log_nhi_edges || !sums || !offset_samples || !log_nhi_samples || !nhi_samples ||
      (Q > 0 && (!ll || !p_dlas || !min_z_dlas || !max_z_dlas)))
    return fail("a required array is NULL");
  for (int pass = 0; pass < 2; ++pass) {
    const double* e = pass ? log_nhi_edges : z_edges;
    const int n = (pass ? n_nhi : n_z) + 1;
    const char* name = pass ? "log_nhi_edges" : "z_edges";
    for (int i = 0; i < n; ++i) {
      if (!std::isfinite(e[i])) return fail(std::string(name) + "[" + std::to_string(i) + "] is not finite");
      if (i > 0 && !(e[i] > e[i - 1])) return fail(std::string(name) + " must be strictly increasing (entry " + std::to_string(i) + ")");
    }
  }
  if (!std::isfinite(dla_log_nhi_min)) return fail("dla_log_nhi_min is not finite");
  if (!(omega_m > 0.0 && omega_m <= 1.0)) return fail("omega_m must lie in (0, 1]");
  return GPDLA_OK;
}

// log-N class boundaries: the union of the bin edges and the DLA threshold, ascending and distinct
static std::vector<double> stats_bounds(const double* log_nhi_edges, int32_t n_nhi, double dla_log_nhi_min) {
  std::vector<double> bound(log_nhi_edges, log_nhi_edges + n_nhi + 1);
  bound.push_back(dla_log_nhi_min);
  std::sort(bound.begin(), bound.end());
  bound.erase(std::unique(bound.begin(), bound.end()), bound.end());
  return bound;
}

// the 1-based class whose lower boundary is v (v is one of the boundaries)
static int stats_class_of(const std::vector<double>& bound, double v) {
  return (int)(std::lower_bound(bound.begin(), bound.end(), v) - bound.begin()) + 1;
}

// Per-quasar rows of cell values -> sums.  launch(q0, nq, rows) enqueues the rows of quasars [q0, q0 + nq).  The rows
// are reduced over fixed COL_ROWS-row blocks; a chunk of quasars is a whole number of blocks, so the chunking (at most
// 256 MB of rows at a time) does not change the summation order.  The blocks are then added in order into `sums`.
extern "C++" {
template <class Launch>
static cudaError_t stats_rows_to_sums(int64_t Q, int64_t W, double* sums, cudaStream_t st, Launch launch) {
  const int64_t nblocks = (Q + COL_ROWS - 1) / COL_ROWS;
  const int64_t chunk = std::min(nblocks * COL_ROWS,
                                 std::max<int64_t>(COL_ROWS, ((256ll << 20) / (W * 8)) / COL_ROWS * COL_ROWS));
  char* base = nullptr;
  cudaError_t e = cudaMallocAsync(&base, (size_t)chunk * W * 8 + (size_t)nblocks * W * (8 + 4), st);
  if (e != cudaSuccess) return e;
  double* rows = (double*)base;
  double* psum = rows + (size_t)chunk * W;
  int32_t* pcnt = (int32_t*)(psum + (size_t)nblocks * W);
  for (int64_t q0 = 0; q0 < Q && e == cudaSuccess; q0 += chunk) {
    const int64_t nq = std::min(chunk, Q - q0);
    launch(q0, nq, rows);
    const int64_t b0 = q0 / COL_ROWS;
    column_partial_kernel<<<dim3((unsigned)((W + COL_THREADS - 1) / COL_THREADS), (unsigned)((nq + COL_ROWS - 1) / COL_ROWS)),
                            COL_THREADS, 0, st>>>(rows, nq, (int)W, COL_MEAN, nullptr, psum + b0 * W, pcnt + b0 * W);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) {
    stats_finish_kernel<<<(unsigned)((W + 127) / 128), 128, 0, st>>>(psum, (int)nblocks, W, sums);
    e = cudaGetLastError();
  }
  const cudaError_t ef = cudaFreeAsync(base, st);   // freed on the error path too
  return e == cudaSuccess ? ef : e;
}
}  // extern "C++"

int gpdla_dla_statistics_device(int64_t Q, int64_t S, const double* sample_log_likelihoods_dla, const double* p_dlas,
                                const double* min_z_dlas, const double* max_z_dlas, const uint8_t* select,
                                const double* offset_samples, const double* log_nhi_samples, const double* nhi_samples,
                                int32_t n_z, const double* z_edges, int32_t n_nhi, const double* log_nhi_edges,
                                double dla_log_nhi_min, double omega_m, double* sums, void* stream) {
  const char* fn = "gpdla_dla_statistics_device";
  int rc = stats_check(fn, Q, S, sample_log_likelihoods_dla, p_dlas, min_z_dlas, max_z_dlas, offset_samples,
                       log_nhi_samples, nhi_samples, n_z, z_edges, n_nhi, log_nhi_edges, dla_log_nhi_min, omega_m, sums);
  if (rc) return rc;
  if (Q == 0) return GPDLA_OK;
  cudaStream_t st = (cudaStream_t)stream;
  // log-N classes: the intervals between the union of the bin edges and the DLA threshold
  const std::vector<double> bound = stats_bounds(log_nhi_edges, n_nhi, dla_log_nhi_min);
  const int m = (int)bound.size();
  StatsClassArgs ca;
  ca.offset = offset_samples; ca.log_nhi = log_nhi_samples; ca.S = S; ca.nbound = m;
  for (int k = 0; k < m; ++k) ca.bound[k] = bound[k];
  StatsArgs a;
  a.ll = sample_log_likelihoods_dla; a.p_dlas = p_dlas; a.min_z_dlas = min_z_dlas; a.max_z_dlas = max_z_dlas;
  a.select = select; a.S = S; a.n_z = n_z; a.n_nhi = n_nhi; a.nbound = m; a.W = stats_width(n_z, n_nhi);
  for (int e = 0; e <= n_z; ++e) a.z_edges[e] = z_edges[e];
  for (int c = 0; c < n_nhi; ++c) {
    a.nhi_class0[c] = (int16_t)stats_class_of(bound, log_nhi_edges[c]);
    a.nhi_class1[c] = (int16_t)stats_class_of(bound, log_nhi_edges[c + 1]);
  }
  a.dla_class0 = stats_class_of(bound, dla_log_nhi_min);
  a.omega_m = omega_m; a.omega_l = 1.0 - omega_m; a.x_coef = 2.0 / (3.0 * omega_m);
  const int64_t W = a.W;
  int dev = 0, optin = 0;
  CUDA_TRY(cudaGetDevice(&dev), g_err);
  CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev), g_err);
  const bool staged = stats_smem_bytes(true, S, n_z, m) + STAT_THREADS / 32 * 8 + 64 <= (size_t)optin;
  const size_t smem = stats_smem_bytes(staged, S, n_z, m);
  const size_t bytes = (size_t)S * (4 + 8 + 4 + 4 + 8 + 8) + (size_t)(m + 2) * 4 + 8 * 64;
  char* base = nullptr;
  CUDA_TRY(cudaMallocAsync(&base, bytes, st), g_err);
  char* ptr = base;
  auto take = [&](size_t n) { char* r = ptr; ptr += (n + 15) / 16 * 16; return r; };
  double* sorted_offset = (double*)take(S * 8); double* sorted_nhi = (double*)take(S * 8);
  uint64_t* key = (uint64_t*)take(S * 8);
  int32_t* cls = (int32_t*)take(S * 4); int32_t* perm = (int32_t*)take(S * 4); int32_t* rank = (int32_t*)take(S * 4);
  int32_t* class_start = (int32_t*)take((m + 2) * 4);
  ca.cls = cls; ca.key = key;
  a.sorted_offset = sorted_offset; a.sorted_nhi = sorted_nhi; a.perm = perm; a.rank = rank; a.class_start = class_start;
  const unsigned sblocks = (unsigned)((S + STAT_THREADS - 1) / STAT_THREADS);
  stats_class_kernel<<<sblocks, STAT_THREADS, 0, st>>>(ca);
  stats_rank_kernel<<<sblocks, STAT_THREADS, 0, st>>>(cls, key, S, perm);
  stats_gather_kernel<<<sblocks, STAT_THREADS, 0, st>>>(perm, cls, offset_samples, nhi_samples, S, m, sorted_offset,
                                                        sorted_nhi, rank, class_start);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess)
    e = staged ? cudaFuncSetAttribute(dla_stats_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
               : cudaFuncSetAttribute(dla_stats_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess)
    e = stats_rows_to_sums(Q, W, sums, st, [&](int64_t q0, int64_t nq, double* rows) {
      a.q0 = q0; a.rows = rows;
      if (staged) dla_stats_kernel<true><<<(unsigned)nq, STAT_THREADS, smem, st>>>(a);
      else dla_stats_kernel<false><<<(unsigned)nq, STAT_THREADS, smem, st>>>(a);
    });
  const cudaError_t ef = cudaFreeAsync(base, st);   // freed on the error path too
  if (e == cudaSuccess) e = ef;
  if (e != cudaSuccess) { g_err = std::string(fn) + ": " + cudaGetErrorString(e); return GPDLA_ERR_CUDA; }
  return GPDLA_OK;
}

int gpdla_dla_statistics(int64_t Q, int64_t S, const double* sample_log_likelihoods_dla, const double* p_dlas,
                         const double* min_z_dlas, const double* max_z_dlas, const uint8_t* select,
                         const double* offset_samples, const double* log_nhi_samples, const double* nhi_samples,
                         int32_t n_z, const double* z_edges, int32_t n_nhi, const double* log_nhi_edges,
                         double dla_log_nhi_min, double omega_m, double* sums) {
  const char* fn = "gpdla_dla_statistics";
  int rc = stats_check(fn, Q, S, sample_log_likelihoods_dla, p_dlas, min_z_dlas, max_z_dlas, offset_samples,
                       log_nhi_samples, nhi_samples, n_z, z_edges, n_nhi, log_nhi_edges, dla_log_nhi_min, omega_m, sums);
  if (rc) return rc;
  const size_t QS = (size_t)Q * S, W = (size_t)stats_width(n_z, n_nhi), Sb = (size_t)S * 8;
  const size_t bytes = QS * 8 + (size_t)Q * (3 * 8 + 1) + 3 * Sb + W * 8 + 6 * 64;
  char* base = nullptr;
  CUDA_TRY(cudaMalloc(&base, bytes), g_err);
  char* ptr = base;
  auto take = [&](size_t n) { char* r = ptr; ptr += (n + 15) / 16 * 16; return r; };
  double* d_ll = (double*)take(QS * 8); double* d_p = (double*)take((size_t)Q * 8);
  double* d_zlo = (double*)take((size_t)Q * 8); double* d_zhi = (double*)take((size_t)Q * 8);
  double* d_off = (double*)take(Sb); double* d_lnhi = (double*)take(Sb); double* d_nhi = (double*)take(Sb);
  double* d_sums = (double*)take(W * 8);
  uint8_t* d_sel = select ? (uint8_t*)take((size_t)Q) : nullptr;
  cudaError_t e = cudaSuccess;
  auto up = [&](void* d, const void* h, size_t n) { if (e == cudaSuccess && n) e = cudaMemcpy(d, h, n, cudaMemcpyHostToDevice); };
  up(d_ll, sample_log_likelihoods_dla, QS * 8); up(d_p, p_dlas, (size_t)Q * 8); up(d_zlo, min_z_dlas, (size_t)Q * 8);
  up(d_zhi, max_z_dlas, (size_t)Q * 8); up(d_off, offset_samples, Sb); up(d_lnhi, log_nhi_samples, Sb);
  up(d_nhi, nhi_samples, Sb); up(d_sums, sums, W * 8);
  if (d_sel) up(d_sel, select, (size_t)Q);
  rc = GPDLA_ERR_CUDA;
  if (e == cudaSuccess) {
    rc = gpdla_dla_statistics_device(Q, S, d_ll, d_p, d_zlo, d_zhi, d_sel, d_off, d_lnhi, d_nhi, n_z, z_edges, n_nhi,
                                     log_nhi_edges, dla_log_nhi_min, omega_m, d_sums, nullptr);
    if (rc == GPDLA_OK) e = cudaMemcpy(sums, d_sums, W * 8, cudaMemcpyDeviceToHost);
  }
  if (e != cudaSuccess) { g_err = std::string(fn) + ": " + cudaGetErrorString(e); rc = GPDLA_ERR_CUDA; }
  cudaFree(base);
  return rc;
}

// ---- population statistics of the multi-DLA catalogue (Ho et al. 2021) ----

// the checks both multi-DLA statistics entries make before any CUDA call: stats_check, then the level count
static int mstats_check(const char* fn, int64_t Q, int64_t S, int32_t max_dlas, const double* ll,
                        const int32_t* base_sample_inds, const double* model_posteriors, const double* min_z_dlas,
                        const double* max_z_dlas, const double* offset_samples, const double* log_nhi_samples,
                        const double* nhi_samples, int32_t n_z, const double* z_edges, int32_t n_nhi,
                        const double* log_nhi_edges, double dla_log_nhi_min, double omega_m, const double* sums) {
  int rc = stats_check(fn, Q, S, ll, model_posteriors, min_z_dlas, max_z_dlas, offset_samples, log_nhi_samples,
                       nhi_samples, n_z, z_edges, n_nhi, log_nhi_edges, dla_log_nhi_min, omega_m, sums);
  if (rc) return rc;
  auto fail = [&](const std::string& why) { g_err = std::string(fn) + ": " + why; return GPDLA_ERR_INVALID; };
  if (max_dlas < 1 || max_dlas > MSTAT_MAX_DLAS)
    return fail("max_dlas = " + std::to_string(max_dlas) + " is outside [1, " + std::to_string(MSTAT_MAX_DLAS) + "]");
  if (Q > 0 && max_dlas > 1 && !base_sample_inds) return fail("base_sample_inds may be NULL only when max_dlas == 1");
  return GPDLA_OK;
}

int gpdla_multi_dla_statistics_device(int64_t Q, int64_t S, int32_t max_dlas, const double* sample_log_likelihoods_dla,
                                      const int32_t* base_sample_inds, const double* model_posteriors,
                                      const double* min_z_dlas, const double* max_z_dlas, const uint8_t* select,
                                      const double* offset_samples, const double* log_nhi_samples,
                                      const double* nhi_samples, int32_t n_z, const double* z_edges, int32_t n_nhi,
                                      const double* log_nhi_edges, double dla_log_nhi_min, double omega_m,
                                      double* sums, void* stream) {
  const char* fn = "gpdla_multi_dla_statistics_device";
  int rc = mstats_check(fn, Q, S, max_dlas, sample_log_likelihoods_dla, base_sample_inds, model_posteriors,
                        min_z_dlas, max_z_dlas, offset_samples, log_nhi_samples, nhi_samples, n_z, z_edges, n_nhi,
                        log_nhi_edges, dla_log_nhi_min, omega_m, sums);
  if (rc) return rc;
  if (Q == 0) return GPDLA_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const std::vector<double> bound = stats_bounds(log_nhi_edges, n_nhi, dla_log_nhi_min);
  const int m = (int)bound.size();
  StatsClassArgs ca;
  ca.offset = offset_samples; ca.log_nhi = log_nhi_samples; ca.S = S; ca.nbound = m;
  for (int k = 0; k < m; ++k) ca.bound[k] = bound[k];
  MultiStatsArgs a;
  a.ll = sample_log_likelihoods_dla; a.partners = max_dlas > 1 ? base_sample_inds : nullptr;
  a.model_posteriors = model_posteriors; a.min_z_dlas = min_z_dlas; a.max_z_dlas = max_z_dlas; a.select = select;
  a.S = S; a.J = max_dlas; a.offset = offset_samples; a.nhi = nhi_samples;
  a.n_z = n_z; a.n_nhi = n_nhi; a.W = stats_width(n_z, n_nhi);
  for (int e = 0; e <= n_z; ++e) a.z_edges[e] = z_edges[e];
  for (int k = 0; k <= m; ++k) a.class_bin[k] = -1;              // class 0: below every boundary, or NaN
  for (int c = 0; c < n_nhi; ++c)
    for (int k = stats_class_of(bound, log_nhi_edges[c]); k < stats_class_of(bound, log_nhi_edges[c + 1]); ++k)
      a.class_bin[k] = (int16_t)c;
  a.dla_class0 = stats_class_of(bound, dla_log_nhi_min);
  a.omega_m = omega_m; a.omega_l = 1.0 - omega_m; a.x_coef = 2.0 / (3.0 * omega_m);
  int dev = 0, optin = 0;
  CUDA_TRY(cudaGetDevice(&dev), g_err);
  CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev), g_err);
  // one accumulator per warp: as many warps (up to 8) as fit; 64 x 128 bins leave one
  const int nw = (int)std::max<int64_t>(1, std::min<int64_t>(STAT_THREADS / 32, (int64_t)(optin - 64) /
                                                             (int64_t)mstats_smem_bytes(1, n_z, n_nhi)));
  const size_t smem = mstats_smem_bytes(nw, n_z, n_nhi);
  char* base = nullptr;
  CUDA_TRY(cudaMallocAsync(&base, (size_t)S * (8 + 4) + 32, st), g_err);
  ca.key = (uint64_t*)base;
  ca.cls = (int32_t*)(base + (size_t)S * 8);
  a.cls = ca.cls;
  stats_class_kernel<<<(unsigned)((S + STAT_THREADS - 1) / STAT_THREADS), STAT_THREADS, 0, st>>>(ca);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaFuncSetAttribute(multi_dla_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess)
    e = stats_rows_to_sums(Q, a.W, sums, st, [&](int64_t q0, int64_t nq, double* rows) {
      a.q0 = q0; a.rows = rows;
      multi_dla_stats_kernel<<<(unsigned)nq, nw * 32, smem, st>>>(a);
    });
  const cudaError_t ef = cudaFreeAsync(base, st);   // freed on the error path too
  if (e == cudaSuccess) e = ef;
  if (e != cudaSuccess) { g_err = std::string(fn) + ": " + cudaGetErrorString(e); return GPDLA_ERR_CUDA; }
  return GPDLA_OK;
}

int gpdla_multi_dla_statistics(int64_t Q, int64_t S, int32_t max_dlas, const double* sample_log_likelihoods_dla,
                               const int32_t* base_sample_inds, const double* model_posteriors,
                               const double* min_z_dlas, const double* max_z_dlas, const uint8_t* select,
                               const double* offset_samples, const double* log_nhi_samples, const double* nhi_samples,
                               int32_t n_z, const double* z_edges, int32_t n_nhi, const double* log_nhi_edges,
                               double dla_log_nhi_min, double omega_m, double* sums) {
  const char* fn = "gpdla_multi_dla_statistics";
  int rc = mstats_check(fn, Q, S, max_dlas, sample_log_likelihoods_dla, base_sample_inds, model_posteriors,
                        min_z_dlas, max_z_dlas, offset_samples, log_nhi_samples, nhi_samples, n_z, z_edges, n_nhi,
                        log_nhi_edges, dla_log_nhi_min, omega_m, sums);
  if (rc) return rc;
  const size_t J = (size_t)max_dlas, P = max_dlas > 1 ? (size_t)Q * (J - 1) * S : 0;
  for (size_t n = 0; n < P; ++n)
    if (base_sample_inds[n] < 0 || base_sample_inds[n] >= S) {
      g_err = std::string(fn) + ": base_sample_inds[" + std::to_string(n / ((J - 1) * S)) + "][" +
              std::to_string(n / S % (J - 1)) + "][" + std::to_string(n % S) + "] = " +
              std::to_string(base_sample_inds[n]) + " is outside [0, S)";
      return GPDLA_ERR_INVALID;
    }
  const size_t QJS = (size_t)Q * J * S, W = (size_t)stats_width(n_z, n_nhi), Sb = (size_t)S * 8;
  const size_t bytes = QJS * 8 + P * 4 + (size_t)Q * ((J + 2) * 8 + 2 * 8 + 1) + 3 * Sb + W * 8 + 8 * 64;
  char* base = nullptr;
  CUDA_TRY(cudaMalloc(&base, bytes), g_err);
  char* ptr = base;
  auto take = [&](size_t n) { char* r = ptr; ptr += (n + 15) / 16 * 16; return r; };
  double* d_ll = (double*)take(QJS * 8); int32_t* d_part = P ? (int32_t*)take(P * 4) : nullptr;
  double* d_mp = (double*)take((size_t)Q * (J + 2) * 8);
  double* d_zlo = (double*)take((size_t)Q * 8); double* d_zhi = (double*)take((size_t)Q * 8);
  double* d_off = (double*)take(Sb); double* d_lnhi = (double*)take(Sb); double* d_nhi = (double*)take(Sb);
  double* d_sums = (double*)take(W * 8);
  uint8_t* d_sel = select ? (uint8_t*)take((size_t)Q) : nullptr;
  cudaError_t e = cudaSuccess;
  auto up = [&](void* d, const void* h, size_t n) { if (e == cudaSuccess && n) e = cudaMemcpy(d, h, n, cudaMemcpyHostToDevice); };
  up(d_ll, sample_log_likelihoods_dla, QJS * 8); up(d_part, base_sample_inds, P * 4);
  up(d_mp, model_posteriors, (size_t)Q * (J + 2) * 8); up(d_zlo, min_z_dlas, (size_t)Q * 8);
  up(d_zhi, max_z_dlas, (size_t)Q * 8); up(d_off, offset_samples, Sb); up(d_lnhi, log_nhi_samples, Sb);
  up(d_nhi, nhi_samples, Sb); up(d_sums, sums, W * 8);
  if (d_sel) up(d_sel, select, (size_t)Q);
  rc = GPDLA_ERR_CUDA;
  if (e == cudaSuccess) {
    rc = gpdla_multi_dla_statistics_device(Q, S, max_dlas, d_ll, d_part, d_mp, d_zlo, d_zhi, d_sel, d_off, d_lnhi, d_nhi,
                                           n_z, z_edges, n_nhi, log_nhi_edges, dla_log_nhi_min, omega_m, d_sums,
                                           nullptr);
    if (rc == GPDLA_OK) e = cudaMemcpy(sums, d_sums, W * 8, cudaMemcpyDeviceToHost);
  }
  if (e != cudaSuccess) { g_err = std::string(fn) + ": " + cudaGetErrorString(e); rc = GPDLA_ERR_CUDA; }
  cudaFree(base);
  return rc;
}

// ---- the fitted model of each quasar under chosen absorbers (CDDF_analysis/qso_loader.py:1654-1774) ----

// the checks both reconstruction entries make before any CUDA call
static int recon_check(gpdla_ctx* c, const char* fn, int64_t Q, int64_t L_max, const double* wavelengths,
                       const double* flux, const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                       const double* z_qsos, int32_t meanflux, int32_t num_absorbers, const double* absorber_z,
                       const double* absorber_nhi, const gpdla_reconstruction* out) {
  if (Q < 0 || Q > 2147483647LL || L_max < 1 || !out || num_absorbers < 0 || num_absorbers > RC_MAX_ABSORBERS ||
      !(meanflux == 0 || meanflux == 1) ||
      (Q > 0 && (!wavelengths || !flux || !noise_variance || !pixel_mask || !lengths || !z_qsos)) ||
      (Q > 0 && num_absorbers > 0 && (!absorber_z || !absorber_nhi))) {
    c->err = std::string(fn) + ": invalid arguments (0 <= num_absorbers <= 4, meanflux 0 or 1, non-NULL inputs)";
    return GPDLA_ERR_INVALID;
  }
  if (!c->d_M) {
    c->err = std::string(fn) + ": set_model must be called first";
    return GPDLA_ERR_STATE;
  }
  if (!rank_supported(c->k)) {
    c->err = std::string(fn) + ": rank k=" + std::to_string(c->k) + " not compiled in (available: 10, 20, 40)";
    return GPDLA_ERR_UNSUPPORTED;
  }
  return GPDLA_OK;
}

// one CTA per quasar; the row of L_max pixels' absorption is staged in shared memory, which bounds L_max
extern "C++" {
template <int K>
static int launch_reconstruct(gpdla_ctx* c, const ReconArgs& ra, int64_t Q, cudaStream_t st) {
  const size_t smem = reconstruct_smem_doubles<K>(ra.L_max) * sizeof(double);
  int optin = 0;
  cudaFuncAttributes fa;
  CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device), c->err);
  CUDA_TRY(cudaFuncGetAttributes(&fa, reconstruct_kernel<K>), c->err);
  if (smem + fa.sharedSizeBytes > (size_t)optin) {
    c->err = "gpdla_reconstruct: L_max=" + std::to_string(ra.L_max) + " does not fit one CTA's shared memory";
    return GPDLA_ERR_UNSUPPORTED;
  }
  int rc = configure_smem(c->device, reconstruct_kernel<K>, smem, c->err);
  if (rc) return rc;
  reconstruct_kernel<K><<<(unsigned)Q, NTHREADS, smem, st>>>(ra);
  return GPDLA_OK;
}
}  // extern "C++"

int gpdla_reconstruct_device(gpdla_ctx* c, int64_t Q, int64_t L_max, const double* wavelengths, const double* flux,
                             const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                             const double* z_qsos, int32_t meanflux, int32_t num_absorbers, const double* absorber_z,
                             const double* absorber_nhi, const gpdla_reconstruction* out, void* stream) {
  if (!c) return GPDLA_ERR_INVALID;
  int rc = recon_check(c, "gpdla_reconstruct_device", Q, L_max, wavelengths, flux, noise_variance, pixel_mask, lengths,
                       z_qsos, meanflux, num_absorbers, absorber_z, absorber_nhi, out);
  if (rc || Q == 0) return rc;
  DeviceGuard guard(c->device);
  ReconArgs ra;
  memset(&ra, 0, sizeof ra);
  ra.wavelengths = wavelengths; ra.flux = flux; ra.noise_variance = noise_variance; ra.pixel_mask = pixel_mask;
  ra.lengths = lengths; ra.z_qsos = z_qsos; ra.L_max = L_max;
  ra.rest_wavelengths = c->d_rest; ra.mu = c->d_mu; ra.M = c->d_M; ra.log_omega = c->d_log_omega; ra.n_rest = c->n_rest;
  ra.c_0 = c->c_0; ra.tau_0 = c->tau_0; ra.beta = c->beta;
  ra.min_lambda = c->params.min_lambda; ra.max_lambda = c->params.max_lambda;
  ra.lya_wavelength = c->params.lya_wavelength; ra.pixel_spacing = c->params.pixel_spacing;
  ra.num_lines = c->params.num_lines; ra.meanflux = meanflux;
  ra.num_absorbers = num_absorbers; ra.absorber_z = absorber_z; ra.absorber_nhi = absorber_nhi;
  ra.absorption = out->absorption; ra.prior_mean = out->prior_mean; ra.prior_sd = out->prior_sd;
  ra.fit_mean = out->fit_mean; ra.continuum = out->continuum; ra.continuum_sd = out->continuum_sd;
  ra.latent = out->latent; ra.chi2 = out->chi2; ra.log_likelihood = out->log_likelihood; ra.num_pixels = out->num_pixels;
  switch (c->k) {
    case 10: rc = launch_reconstruct<10>(c, ra, Q, (cudaStream_t)stream); break;
    case 20: rc = launch_reconstruct<20>(c, ra, Q, (cudaStream_t)stream); break;
    case 40: rc = launch_reconstruct<40>(c, ra, Q, (cudaStream_t)stream); break;
    default: c->err = "gpdla_reconstruct: rank not compiled in"; rc = GPDLA_ERR_UNSUPPORTED;
  }
  if (rc) return rc;
  c->launches++;
  CUDA_TRY(cudaGetLastError(), c->err);
  return GPDLA_OK;
}

int gpdla_reconstruct(gpdla_ctx* c, int64_t Q, int64_t L_max, const double* wavelengths, const double* flux,
                      const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                      const double* z_qsos, int32_t meanflux, int32_t num_absorbers, const double* absorber_z,
                      const double* absorber_nhi, const gpdla_reconstruction* out) {
  if (!c) return GPDLA_ERR_INVALID;
  int rc = recon_check(c, "gpdla_reconstruct", Q, L_max, wavelengths, flux, noise_variance, pixel_mask, lengths, z_qsos,
                       meanflux, num_absorbers, absorber_z, absorber_nhi, out);
  if (rc || Q == 0) return rc;
  const size_t QA = (size_t)Q * num_absorbers;
  for (size_t i = 0; i < QA; ++i) {
    const double z = absorber_z[i], N = absorber_nhi[i];
    if (std::isnan(z)) continue;
    if (!(std::isfinite(z) && z > -1.0 && std::isfinite(N) && N >= 0.0)) {
      c->err = "gpdla_reconstruct: absorber " + std::to_string(i) + " needs z > -1 and a finite N >= 0 (NaN z = none)";
      return GPDLA_ERR_INVALID;
    }
  }
  DeviceGuard guard(c->device);
  const size_t QL = (size_t)Q * L_max;
  struct Item { void** dev; const void* host_in; void* host_out; size_t bytes; };
  double *d_w, *d_f, *d_v, *d_z, *d_az = nullptr, *d_an = nullptr;
  uint8_t* d_m;
  int32_t* d_len;
  gpdla_reconstruction dr;
  memset(&dr, 0, sizeof dr);
  std::vector<Item> items = {
      {(void**)&d_w, wavelengths, nullptr, QL * 8}, {(void**)&d_f, flux, nullptr, QL * 8},
      {(void**)&d_v, noise_variance, nullptr, QL * 8}, {(void**)&d_z, z_qsos, nullptr, (size_t)Q * 8},
      {(void**)&d_len, lengths, nullptr, (size_t)Q * 4}, {(void**)&d_m, pixel_mask, nullptr, QL}};
  if (QA) {
    items.push_back({(void**)&d_az, absorber_z, nullptr, QA * 8});
    items.push_back({(void**)&d_an, absorber_nhi, nullptr, QA * 8});
  }
  auto want = [&](void** dev, void* host, size_t bytes) { if (host) items.push_back({dev, nullptr, host, bytes}); };
  want((void**)&dr.absorption, out->absorption, QL * 8);
  want((void**)&dr.prior_mean, out->prior_mean, QL * 8);
  want((void**)&dr.prior_sd, out->prior_sd, QL * 8);
  want((void**)&dr.fit_mean, out->fit_mean, QL * 8);
  want((void**)&dr.continuum, out->continuum, QL * 8);
  want((void**)&dr.continuum_sd, out->continuum_sd, QL * 8);
  want((void**)&dr.latent, out->latent, (size_t)Q * c->k * 8);
  want((void**)&dr.chi2, out->chi2, (size_t)Q * 8);
  want((void**)&dr.log_likelihood, out->log_likelihood, (size_t)Q * 8);
  want((void**)&dr.num_pixels, out->num_pixels, (size_t)Q * 4);
  size_t bytes = 256;
  for (auto& it : items) bytes += (it.bytes + 255) / 256 * 256;
  if (c->st_bytes < bytes) {
    cudaFree(c->d_stage); c->d_stage = nullptr; c->st_bytes = 0;
    CUDA_TRY(cudaMalloc(&c->d_stage, bytes), c->err);
    c->st_bytes = bytes;
  }
  char* p = (char*)c->d_stage;
  cudaStream_t st = c->stream;
  for (auto& it : items) {
    *it.dev = p; p += (it.bytes + 255) / 256 * 256;
    if (it.host_in) CUDA_TRY(cudaMemcpyAsync(*it.dev, it.host_in, it.bytes, cudaMemcpyHostToDevice, st), c->err);
  }
  rc = gpdla_reconstruct_device(c, Q, L_max, d_w, d_f, d_v, d_m, d_len, d_z, meanflux, num_absorbers, d_az, d_an, &dr, st);
  if (rc) return rc;
  for (auto& it : items)
    if (it.host_out) CUDA_TRY(cudaMemcpyAsync(it.host_out, *it.dev, it.bytes, cudaMemcpyDeviceToHost, st), c->err);
  CUDA_TRY(cudaStreamSynchronize(st), c->err);
  return GPDLA_OK;
}

}  // extern "C"
