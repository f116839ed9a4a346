// Filter bank (include/uahn_filter.h): the EKF states of n sequences on the device, IMU propagation and the IEKF
// measurement update as sm_100a kernels around one batched forward per iteration (DESIGN §11).  The per-element fp64 math
// is ekf_math.h's, the transcription the host consumer (imu_propagate.cpp, ekf_update.cpp) compiles too; this file is
// built with -fmad=false so that every device product and sum rounds like the host's -ffp-contract=off build.
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "../../include/uahn_filter.h"
#include "common.cuh"
#include "ekf_math.h"
#include "kernels.h"

using namespace uahn;
using namespace uahn_ekf;

namespace {

constexpr int PROP_COV_THREADS = 224;                  // the covariance warps of the propagation kernel (7)
// + one warp whose lane 0 runs predict_and_compute.  8 warps = 2 per SM sub-partition leave a thread up to 255
// registers; with 9 the cap is 168 and predict_and_compute spills.
constexpr int PROP_THREADS = PROP_COV_THREADS + 32;
constexpr int UPD_THREADS = 128;
constexpr int BEGIN_THREADS = 128;
constexpr int STATE_DOUBLES = (int)(sizeof(uahn_ekf_state) / sizeof(double));
static_assert(sizeof(uahn_ekf_state) % sizeof(double) == 0, "uahn_ekf_state is a block of doubles");

// the covariance warps only (named barrier 1): the predictor lane is inside predict_and_compute meanwhile
__device__ __forceinline__ void cov_warps_sync() { asm volatile("bar.sync 1, %0;" ::"r"(PROP_COV_THREADS) : "memory"); }

// uahn_imu_propagate for one slot per CTA.  csr = {offsets[n + 1], codes[n]}: slot i's selected readings are
// sel[offsets[i] .. offsets[i+1]), codes[i] != 0 (t1 <= t0) reports that code and leaves the state alone.  The state,
// P included, stays in shared memory for all intervals of the frame.  Interval t: the covariance warps form FP = F_t P,
// then P <- FP F_t^T + Fw_t Q Fw_t^T, while lane 0 of the last warp already runs predict_and_compute for interval t+1
// into the other F / Fw buffer (the mean chain never reads P).  The sums skip F's structurally zero blocks.
__global__ void __launch_bounds__(PROP_THREADS, 1)
filter_propagate_kernel(uahn_ekf_state* states, const uahn_imu_sample* sel, const int* csr, Cfg cfg, int n, int* status) {
  __shared__ uahn_ekf_state s;
  __shared__ double F[2][D * D], Fw[2][D * 15], FP[D * D];
  pdl_wait();
  const int slot = blockIdx.x, tid = threadIdx.x;
  const int code = csr[n + 1 + slot];
  if (code) {
    if (tid == 0) status[slot] = code;
    return;
  }
  const int lo = csr[slot], intervals = csr[slot + 1] - lo - 1;
  if (intervals < 1) return;                                   // fewer than two readings: nothing to integrate
  sel += lo;
  double* sd = reinterpret_cast<double*>(&s);
  double* gd = reinterpret_cast<double*>(states + slot);
  for (int e = tid; e < STATE_DOUBLES; e += PROP_THREADS) sd[e] = gd[e];
  for (int e = tid; e < 2 * D * D; e += PROP_THREADS) (&F[0][0])[e] = 0.0;
  for (int e = tid; e < 2 * D * 15; e += PROP_THREADS) (&Fw[0][0])[e] = 0.0;
  __syncthreads();
  const bool predictor = tid == PROP_COV_THREADS;
  if (predictor) predict_and_compute(cfg, &s, sel[0], sel[1], interval_trig(cfg, &s, sel[0], sel[1]), F[0], Fw[0]);
  __syncthreads();
  for (int t = 0; t < intervals; ++t) {
    const int b = t & 1;
    if (tid < PROP_COV_THREADS) {
      for (int e = tid; e < D * D; e += PROP_COV_THREADS) {
        const int i = e / D, j = e - i * D;
        FP[e] = fp_element(F[b], s.cov, i, j, f_row_blocks(i / 3));
      }
      cov_warps_sync();
      for (int e = tid; e < D * D; e += PROP_COV_THREADS) {
        const int i = e / D, j = e - i * D;
        s.cov[e] = pn_element(cfg, FP, F[b], Fw[b], i, j, f_row_blocks(j / 3));
      }
    } else if (predictor && t + 1 < intervals) {
      const Trig g = interval_trig(cfg, &s, sel[t + 1], sel[t + 2]);
      predict_and_compute(cfg, &s, sel[t + 1], sel[t + 2], g, F[b ^ 1], Fw[b ^ 1]);
    }
    __syncthreads();
  }
  for (int e = tid; e < STATE_DOUBLES; e += PROP_THREADS) gd[e] = sd[e];
}

// uahn_ekf_prior_px -> float, as uahn_infer hands the prior to the forward
__device__ __forceinline__ float prior_component(const uahn_ekf_state& s, int i) {
  return (float)(s.offset[i >> 1][i & 1] * UAHN_FOCAL_PX);
}

// Start of a frame: the slot's frame counter counts the new frame, its failure flag clears, and the prior of
// iteration 0 is written.
__global__ void __launch_bounds__(BEGIN_THREADS)
filter_begin_kernel(const uahn_ekf_state* states, int* count, int* failed, float* prior, int n) {
  pdl_wait();
  const int slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n) return;
  if (count[slot] < (1 << 30)) count[slot] += 1;
  failed[slot] = 0;
  for (int i = 0; i < 8; ++i) prior[slot * 8 + i] = prior_component(states[slot], i);
}

// Iteration `it` of uahn_ekf_iekf_frame for one slot per CTA, after the forward wrote mean / cov (float rows of this
// iteration): the gates, uahn_ekf_update on the outputs widened to double, the offset reset after the last iteration,
// and the prior of the next iteration (next_prior != nullptr).  A failed inversion stops the slot for the rest of the
// frame, as the host loop's return does.
__global__ void __launch_bounds__(UPD_THREADS)
filter_update_kernel(uahn_ekf_state* states, const int* count, int* failed, int* status, const float* mean,
                     const float* cov, const uint8_t* use, int min_images, int update_offset, int last, double K_net_Cov,
                     float* next_prior) {
  __shared__ double Sinv[64], work[64], K[D * 8], HP[8 * D], cov_px[64], mean_px[8], propagated[8], inno[8], dx[D];
  __shared__ int inverted;
  pdl_wait();
  const int slot = blockIdx.x, tid = threadIdx.x;
  uahn_ekf_state* s = states + slot;
  double* P = s->cov;
  bool stopped = failed[slot] != 0;
  const int frames = count[slot];
  // frames < 2: "Only has one image", the forward's outputs are not used (uahn_infer returns UAHN_ERR_STATE)
  if (!stopped && frames >= 2 && (!use || use[slot]) && frames > min_images) {
    for (int e = tid; e < 64; e += UPD_THREADS) cov_px[e] = (double)cov[(size_t)slot * 64 + e];
    if (tid < 8) {
      mean_px[tid] = (double)mean[(size_t)slot * 8 + tid];
      propagated[tid] = s->offset[tid >> 1][tid & 1];
    }
    for (int e = tid; e < 8 * D; e += UPD_THREADS) HP[e] = P[meas_row(e / D) * D + e % D];
    __syncthreads();
    if (tid < 64) Sinv[tid] = innovation_cov_element(P, cov_px, K_net_Cov, tid >> 3, tid & 7);
    __syncthreads();
    if (tid == 0) inverted = invert8(Sinv, work);
    __syncthreads();
    if (!inverted) {
      stopped = true;
      if (tid == 0) { failed[slot] = 1; status[slot] = UAHN_ERR_INVALID; }
    } else {
      for (int e = tid; e < D * 8; e += UPD_THREADS) K[e] = gain_element(P, Sinv, e >> 3, e & 7);
      if (tid < 8) inno[tid] = innovation_element(mean_px, propagated, tid);
      __syncthreads();
      for (int e = tid; e < D * D; e += UPD_THREADS) P[e] -= cov_update_element(K, HP, e / D, e % D);
      const int rows = update_offset ? D : 15;
      for (int r = tid; r < rows; r += UPD_THREADS) dx[r] = increment_element(K, inno, r);
      __syncthreads();
      if (tid == 0) apply_increment(s, dx, update_offset);
    }
    __syncthreads();
  }
  if (last && !stopped) {                                      // uahn_ekf_reset_offsets
    if (tid < 12) s->offset[tid / 3][tid % 3] = 0.0;
    for (int e = tid; e < D * D; e += UPD_THREADS)
      if (!reset_keeps(e / D, e % D)) P[e] = 0.0;
  }
  if (next_prior) {
    __syncthreads();
    if (tid < 8) next_prior[(size_t)slot * 8 + tid] = prior_component(*s, tid);
  }
}

}  // namespace

struct uahn_filter {
  uahn_handle* h = nullptr;
  int n = 0, device = 0;
  Cfg cfg{};
  uahn_ekf_state* d_state = nullptr;
  int *d_count = nullptr, *d_failed = nullptr, *d_status = nullptr;
  uint8_t* d_frames = nullptr;   // [2][n] frames: the half `ring` holds the latest frame of every slot, the other its prev
  int ring = 0;
  uint8_t* d_use = nullptr;
  float *d_prior = nullptr, *d_mean = nullptr, *d_cov = nullptr;   // [iter_cap][n] rows
  int iter_cap = 0;
  // propagation staging: the selected readings of all slots (CSR) and {offsets[n + 1], codes[n]}, pinned + device
  uahn_imu_sample *h_sel = nullptr, *d_sel = nullptr;
  size_t sel_cap = 0;
  int *h_csr = nullptr, *d_csr = nullptr;
  int* h_status = nullptr;
  cudaEvent_t ev_staged = nullptr;                       // the last propagation's uploads have left h_sel / h_csr
  cudaEvent_t ev_to_iter = nullptr, ev_from_iter = nullptr;
  uint64_t auto_pair = 0;                                // pair index of frames called with rng == NULL
  // raw frames (uahn_filter_frame_raw): the undistort maps, two staging buffers of n packed raw frames, and a copy stream
  // on which the upload of frame k + 1 runs under frame k's forward.  Frame k stages in buffer k % 2: its copy waits for
  // ev_consumed (the remap of frame k - 2), the bank stream's remap waits for ev_filled.
  float *d_map1 = nullptr, *d_map2 = nullptr;
  int raw_rows = 0, raw_cols = 0;                        // 0: no maps
  uint8_t* d_raw[2] = {nullptr, nullptr};
  size_t raw_cap = 0;                                    // bytes of each staging buffer
  cudaStream_t copy_st = nullptr;
  cudaEvent_t ev_filled[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};
  uint64_t raw_frames = 0;
};

namespace {

int failf(uahn_handle* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  return handle_fail(h, code, buf);
}

#define FCK(expr)                                                                                               \
  do {                                                                                                          \
    cudaError_t e__ = (expr);                                                                                   \
    if (e__ != cudaSuccess)                                                                                     \
      return failf(f->h, UAHN_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

cudaStream_t stream_of(uahn_handle* h) { return (cudaStream_t)uahn_stream(h); }

void release(uahn_filter* f) {
  void* dev[] = {f->d_state, f->d_count, f->d_failed, f->d_status, f->d_frames, f->d_use, f->d_prior, f->d_mean, f->d_cov,
                 f->d_sel, f->d_csr, f->d_map1, f->d_map2, f->d_raw[0], f->d_raw[1]};
  for (void* p : dev) if (p) cudaFree(p);
  void* host[] = {f->h_sel, f->h_csr, f->h_status};
  for (void* p : host) if (p) cudaFreeHost(p);
  for (cudaEvent_t e : {f->ev_staged, f->ev_to_iter, f->ev_from_iter, f->ev_filled[0], f->ev_filled[1], f->ev_consumed[0],
                        f->ev_consumed[1]})
    if (e) cudaEventDestroy(e);
  if (f->copy_st) cudaStreamDestroy(f->copy_st);
  delete f;
}

// prior / mean / cov rows for max_iter iterations
int ensure_iterations(uahn_filter* f, int max_iter) {
  if (max_iter <= f->iter_cap) return UAHN_OK;
  FCK(cudaStreamSynchronize(stream_of(f->h)));               // the old buffers may still be read by enqueued work
  for (float** p : {&f->d_prior, &f->d_mean, &f->d_cov}) { if (*p) cudaFree(*p); *p = nullptr; }
  f->iter_cap = 0;
  const size_t rows = (size_t)max_iter * f->n;
  FCK(cudaMalloc(&f->d_prior, rows * 8 * sizeof(float)));
  FCK(cudaMalloc(&f->d_mean, rows * 8 * sizeof(float)));
  FCK(cudaMalloc(&f->d_cov, rows * 64 * sizeof(float)));
  f->iter_cap = max_iter;
  return UAHN_OK;
}

int ensure_samples(uahn_filter* f, size_t count) {
  if (count <= f->sel_cap) return UAHN_OK;
  FCK(cudaStreamSynchronize(stream_of(f->h)));
  if (f->h_sel) cudaFreeHost(f->h_sel);
  if (f->d_sel) cudaFree(f->d_sel);
  f->h_sel = nullptr;
  f->d_sel = nullptr;
  f->sel_cap = 0;
  const size_t cap = count + count / 2 + 64;
  FCK(cudaMallocHost(&f->h_sel, cap * sizeof(uahn_imu_sample)));
  FCK(cudaMalloc(&f->d_sel, cap * sizeof(uahn_imu_sample)));
  f->sel_cap = cap;
  return UAHN_OK;
}

// Checks shared by the two frame entries; nothing is enqueued.  h_iter == the bank's own handle becomes NULL.
int check_frame(uahn_filter* f, const char* who, uahn_handle*& h_iter, int max_iter, const uahn_rng* rng) {
  uahn_handle* h = f->h;
  if (max_iter < 1) return failf(h, UAHN_ERR_INVALID, "%s: max_iter=%d < 1", who, max_iter);
  if (rng && rng->keep_masks)
    return failf(h, UAHN_ERR_UNSUPPORTED, "%s: explicit masks are not supported (Philox masks only)", who);
  if (h_iter == h) h_iter = nullptr;
  if (h_iter && handle_device(h_iter) != f->device)
    return failf(h, UAHN_ERR_INVALID, "%s: h_iter is on device %d, the bank on device %d", who, handle_device(h_iter),
                 f->device);
  if (h_iter && handle_max_batch(h_iter) < f->n)
    return failf(h, UAHN_ERR_INVALID, "%s: h_iter has max_batch=%d < n=%d", who, handle_max_batch(h_iter), f->n);
  return UAHN_OK;
}

// One IEKF frame of every slot: ring flip, fill(curr) enqueues what writes the n new frames into the new current half
// on the bank's stream, then the begin kernel, max_iter forwards and updates, and the outputs.
template <typename Fill>
int run_frame(uahn_filter* f, const char* who, uahn_handle* h_iter, Fill fill, int max_iter, double K_net_Cov,
              int min_images, const uint8_t* use_measurement, const uahn_rng* rng, float* prior_out, float* mean_out,
              float* cov_out, double* imu_out) {
  uahn_handle* h = f->h;
  const int n = f->n;
  FCK(cudaSetDevice(f->device));
  int rc = ensure_iterations(f, max_iter);
  if (rc) return rc;
  cudaStream_t st = stream_of(h);
  f->ring ^= 1;
  uint8_t* curr = f->d_frames + (size_t)f->ring * n * UAHN_IMG_PIXELS;
  const uint8_t* prev = f->d_frames + (size_t)(f->ring ^ 1) * n * UAHN_IMG_PIXELS;
  if ((rc = fill(curr))) return rc;
  if (use_measurement) FCK(cudaMemcpyAsync(f->d_use, use_measurement, (size_t)n, cudaMemcpyHostToDevice, st));
  FCK(launch_pdl(filter_begin_kernel, dim3((n + BEGIN_THREADS - 1) / BEGIN_THREADS), dim3(BEGIN_THREADS), 0, st,
                 f->d_state, f->d_count, f->d_failed, f->d_prior, n));
  const uint64_t seed = rng ? rng->seed : 0, first = rng ? rng->first_pair_index : f->auto_pair;
  for (int it = 0; it < max_iter; ++it) {
    uahn_handle* net = (it > 0 && h_iter) ? h_iter : h;                   // HomographyNet.cpp:209
    const uahn_rng r{seed, first + (uint64_t)it * n, nullptr};
    float* prior = f->d_prior + (size_t)it * n * 8;
    float* mean = f->d_mean + (size_t)it * n * 8;
    float* cov = f->d_cov + (size_t)it * n * 64;
    cudaStream_t nst = stream_of(net);
    if (nst != st) {
      FCK(cudaEventRecord(f->ev_to_iter, st));
      FCK(cudaStreamWaitEvent(nst, f->ev_to_iter, 0));
    }
    if ((rc = uahn_infer_batch_device(net, n, prev, curr, prior, &r, mean, cov, nullptr))) {
      if (net != h) failf(h, rc, "%s: forward on h_iter: %s", who, uahn_last_error(net));
      return rc;
    }
    if (nst != st) {
      FCK(cudaEventRecord(f->ev_from_iter, nst));
      FCK(cudaStreamWaitEvent(st, f->ev_from_iter, 0));
    }
    FCK(launch_pdl(filter_update_kernel, dim3(n), dim3(UPD_THREADS), 0, st, f->d_state, (const int*)f->d_count, f->d_failed,
                   f->d_status, (const float*)mean, (const float*)cov, use_measurement ? (const uint8_t*)f->d_use : nullptr,
                   min_images, it != max_iter - 1 ? 1 : 0, it == max_iter - 1 ? 1 : 0, K_net_Cov,
                   it + 1 < max_iter ? f->d_prior + (size_t)(it + 1) * n * 8 : nullptr));
  }
  if (!rng) f->auto_pair += (uint64_t)max_iter * n;
  const size_t rows = (size_t)max_iter * n;
  if (prior_out) FCK(cudaMemcpyAsync(prior_out, f->d_prior, rows * 8 * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (mean_out) FCK(cudaMemcpyAsync(mean_out, f->d_mean, rows * 8 * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (cov_out) FCK(cudaMemcpyAsync(cov_out, f->d_cov, rows * 64 * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (imu_out)
    FCK(cudaMemcpy2DAsync(imu_out, 16 * sizeof(double), f->d_state, sizeof(uahn_ekf_state), 16 * sizeof(double), n,
                          cudaMemcpyDeviceToHost, st));
  return UAHN_OK;
}

// Checks of the raw-frame entries; nothing is enqueued.
int check_raw(uahn_filter* f, const char* who, const uint8_t* raw, size_t stride) {
  if (!f->raw_rows) return failf(f->h, UAHN_ERR_STATE, "%s: uahn_filter_set_undistort_maps has not been called", who);
  if (!raw) return failf(f->h, UAHN_ERR_INVALID, "%s: null raw frames", who);
  if (stride < (size_t)f->raw_cols || stride > (size_t)INT32_MAX)
    return failf(f->h, UAHN_ERR_INVALID, "%s: row stride %zu outside [raw_cols=%d, 2^31)", who, stride, f->raw_cols);
  return UAHN_OK;
}

// The n raw frames of one call: upload into staging buffer raw_frames % 2 on the copy stream (after the remap that last
// read that buffer), then the batched remap into dst on the bank's stream.
int enqueue_raw(uahn_filter* f, const uint8_t* raw, size_t stride, uint8_t* dst) {
  const int b = (int)(f->raw_frames & 1);
  const int rows = f->raw_rows, cols = f->raw_cols;
  cudaStream_t st = stream_of(f->h);
  FCK(cudaStreamWaitEvent(f->copy_st, f->ev_consumed[b], 0));
  FCK(cudaMemcpy2DAsync(f->d_raw[b], (size_t)cols, raw, stride, (size_t)cols, (size_t)f->n * rows, cudaMemcpyHostToDevice,
                        f->copy_st));
  FCK(cudaEventRecord(f->ev_filled[b], f->copy_st));
  FCK(cudaStreamWaitEvent(st, f->ev_filled[b], 0));
  FCK(launch_remap_u8(f->d_raw[b], rows, cols, (size_t)cols, f->n, f->d_map1, f->d_map2, dst, st));
  FCK(cudaEventRecord(f->ev_consumed[b], st));
  ++f->raw_frames;
  return UAHN_OK;
}

}  // namespace

extern "C" {

int uahn_filter_create(uahn_handle* h, int n, const uahn_propagator_config* cfg, uahn_filter** out) {
  if (!h) return UAHN_ERR_INVALID;
  if (!cfg || !out) return handle_fail(h, UAHN_ERR_INVALID, "uahn_filter_create: null config / output");
  if (n < 1 || n > handle_max_batch(h))
    return failf(h, UAHN_ERR_INVALID, "uahn_filter_create: n=%d outside [1, max_batch=%d]", n, handle_max_batch(h));
  uahn_filter* f = new uahn_filter();
  f->h = h;
  f->n = n;
  f->device = handle_device(h);
  f->cfg = resolve_config(cfg);
  auto step = [&]() -> int {
    FCK(cudaSetDevice(f->device));
    FCK(cudaMalloc(&f->d_state, (size_t)n * sizeof(uahn_ekf_state)));
    FCK(cudaMemset(f->d_state, 0, (size_t)n * sizeof(uahn_ekf_state)));
    for (int** p : {&f->d_count, &f->d_failed, &f->d_status}) {
      FCK(cudaMalloc(p, (size_t)n * sizeof(int)));
      FCK(cudaMemset(*p, 0, (size_t)n * sizeof(int)));
    }
    FCK(cudaMalloc(&f->d_frames, (size_t)2 * n * UAHN_IMG_PIXELS));
    FCK(cudaMemset(f->d_frames, 0, (size_t)2 * n * UAHN_IMG_PIXELS));
    FCK(cudaMalloc(&f->d_use, (size_t)n));
    FCK(cudaMalloc(&f->d_csr, (size_t)(2 * n + 1) * sizeof(int)));
    FCK(cudaMallocHost(&f->h_csr, (size_t)(2 * n + 1) * sizeof(int)));
    FCK(cudaMallocHost(&f->h_status, (size_t)n * sizeof(int)));
    for (cudaEvent_t* e : {&f->ev_staged, &f->ev_to_iter, &f->ev_from_iter}) FCK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    FCK(cudaDeviceSynchronize());
    return ensure_iterations(f, 1);
  };
  const int rc = step();
  if (rc) { release(f); return rc; }
  *out = f;
  return UAHN_OK;
}

void uahn_filter_destroy(uahn_filter* f) {
  if (!f) return;
  int prev_dev = -1;
  cudaGetDevice(&prev_dev);
  cudaSetDevice(f->device);
  cudaStreamSynchronize(stream_of(f->h));
  if (f->copy_st) cudaStreamSynchronize(f->copy_st);
  release(f);
  if (prev_dev >= 0) cudaSetDevice(prev_dev);
}

int uahn_filter_set_states(uahn_filter* f, int first, int count, const uahn_ekf_state* states) {
  if (!f) return UAHN_ERR_INVALID;
  if (!states) return handle_fail(f->h, UAHN_ERR_INVALID, "uahn_filter_set_states: null states");
  if (first < 0 || count < 0 || first + count > f->n)
    return failf(f->h, UAHN_ERR_INVALID, "uahn_filter_set_states: slots [%d, %d) outside [0, %d)", first, first + count, f->n);
  FCK(cudaSetDevice(f->device));
  cudaStream_t st = stream_of(f->h);
  FCK(cudaMemcpyAsync(f->d_state + first, states, (size_t)count * sizeof(uahn_ekf_state), cudaMemcpyHostToDevice, st));
  FCK(cudaMemsetAsync(f->d_count + first, 0, (size_t)count * sizeof(int), st));
  FCK(cudaStreamSynchronize(st));
  return UAHN_OK;
}

int uahn_filter_get_states(uahn_filter* f, int first, int count, uahn_ekf_state* states) {
  if (!f) return UAHN_ERR_INVALID;
  if (!states) return handle_fail(f->h, UAHN_ERR_INVALID, "uahn_filter_get_states: null states");
  if (first < 0 || count < 0 || first + count > f->n)
    return failf(f->h, UAHN_ERR_INVALID, "uahn_filter_get_states: slots [%d, %d) outside [0, %d)", first, first + count, f->n);
  FCK(cudaSetDevice(f->device));
  cudaStream_t st = stream_of(f->h);
  FCK(cudaMemcpyAsync(states, f->d_state + first, (size_t)count * sizeof(uahn_ekf_state), cudaMemcpyDeviceToHost, st));
  FCK(cudaStreamSynchronize(st));
  return UAHN_OK;
}

int uahn_filter_propagate(uahn_filter* f, const uahn_imu_sample* imu, const int* offsets, const double* t0, const double* t1) {
  if (!f) return UAHN_ERR_INVALID;
  const int n = f->n;
  if (!imu || !offsets || !t0 || !t1) return handle_fail(f->h, UAHN_ERR_INVALID, "uahn_filter_propagate: null argument");
  size_t bound = 0;
  for (int i = 0; i < n; ++i) {
    if (offsets[i] < 0 || offsets[i + 1] < offsets[i])
      return failf(f->h, UAHN_ERR_INVALID, "uahn_filter_propagate: offsets[%d..%d] = %d, %d", i, i + 1, offsets[i], offsets[i + 1]);
    bound += (size_t)(offsets[i + 1] - offsets[i]) + 2;   // select_imu_readings adds at most one interpolated reading
  }
  FCK(cudaSetDevice(f->device));
  FCK(cudaEventSynchronize(f->ev_staged));                   // the previous propagation's uploads have left the staging
  int rc = ensure_samples(f, bound);
  if (rc) return rc;
  // select_imu_readings stays on the host (it is a scan with data-dependent output): CSR of the selected readings
  int* off = f->h_csr;
  int* code = f->h_csr + n + 1;
  int total = 0;
  for (int i = 0; i < n; ++i) {
    off[i] = total;
    code[i] = UAHN_OK;
    if (!(t1[i] > t0[i])) { code[i] = UAHN_ERR_STATE; continue; }   // Propagator.cpp:32-42 (uahn_imu_propagate)
    const int cnt = offsets[i + 1] - offsets[i];
    int got = 0;
    if (uahn_imu_select_readings(imu + offsets[i], cnt, t0[i], t1[i], f->h_sel + total, cnt + 2, &got))
      return failf(f->h, UAHN_ERR_INVALID, "uahn_filter_propagate: reading selection of slot %d failed", i);
    total += got;
  }
  off[n] = total;
  cudaStream_t st = stream_of(f->h);
  FCK(cudaMemcpyAsync(f->d_csr, f->h_csr, (size_t)(2 * n + 1) * sizeof(int), cudaMemcpyHostToDevice, st));
  if (total) FCK(cudaMemcpyAsync(f->d_sel, f->h_sel, (size_t)total * sizeof(uahn_imu_sample), cudaMemcpyHostToDevice, st));
  FCK(cudaEventRecord(f->ev_staged, st));
  FCK(launch_pdl(filter_propagate_kernel, dim3(n), dim3(PROP_THREADS), 0, st, f->d_state, f->d_sel, f->d_csr, f->cfg, n,
                 f->d_status));
  return UAHN_OK;
}

int uahn_filter_frame(uahn_filter* f, uahn_handle* h_iter, const uint8_t* frames, int max_iter, double K_net_Cov,
                      int min_images, const uint8_t* use_measurement, const uahn_rng* rng, float* prior_out,
                      float* mean_out, float* cov_out, double* imu_out) {
  if (!f) return UAHN_ERR_INVALID;
  if (!frames) return handle_fail(f->h, UAHN_ERR_INVALID, "uahn_filter_frame: null frames");
  int rc = check_frame(f, "uahn_filter_frame", h_iter, max_iter, rng);
  if (rc) return rc;
  auto upload = [&](uint8_t* curr) -> int {
    FCK(cudaMemcpyAsync(curr, frames, (size_t)f->n * UAHN_IMG_PIXELS, cudaMemcpyHostToDevice, stream_of(f->h)));
    return UAHN_OK;
  };
  return run_frame(f, "uahn_filter_frame", h_iter, upload, max_iter, K_net_Cov, min_images, use_measurement, rng, prior_out,
                   mean_out, cov_out, imu_out);
}

int uahn_filter_set_undistort_maps(uahn_filter* f, int raw_rows, int raw_cols, const float* map1, const float* map2) {
  if (!f) return UAHN_ERR_INVALID;
  if (!map1 || !map2 || raw_rows < 2 || raw_cols < 2 || raw_rows > 32767 || raw_cols > 32767)
    return failf(f->h, UAHN_ERR_INVALID, "uahn_filter_set_undistort_maps: bad maps / raw size %dx%d", raw_rows, raw_cols);
  FCK(cudaSetDevice(f->device));
  cudaStream_t st = stream_of(f->h);
  FCK(cudaStreamSynchronize(st));                 // enqueued remaps still read the maps and the staging
  if (f->copy_st) FCK(cudaStreamSynchronize(f->copy_st));
  f->raw_rows = f->raw_cols = 0;                  // no maps unless this call succeeds
  for (cudaEvent_t* e : {&f->ev_filled[0], &f->ev_filled[1], &f->ev_consumed[0], &f->ev_consumed[1]})
    if (!*e) FCK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  if (!f->copy_st) FCK(cudaStreamCreateWithFlags(&f->copy_st, cudaStreamNonBlocking));
  for (float** m : {&f->d_map1, &f->d_map2})
    if (!*m) FCK(cudaMalloc(m, (size_t)UAHN_IMG_PIXELS * sizeof(float)));
  const size_t bytes = (size_t)f->n * raw_rows * raw_cols;
  if (bytes > f->raw_cap) {
    for (uint8_t*& p : f->d_raw) { if (p) cudaFree(p); p = nullptr; }
    f->raw_cap = 0;
    FCK(cudaMalloc(&f->d_raw[0], bytes));
    FCK(cudaMalloc(&f->d_raw[1], bytes));
    f->raw_cap = bytes;
  }
  FCK(cudaMemcpyAsync(f->d_map1, map1, (size_t)UAHN_IMG_PIXELS * sizeof(float), cudaMemcpyHostToDevice, st));
  FCK(cudaMemcpyAsync(f->d_map2, map2, (size_t)UAHN_IMG_PIXELS * sizeof(float), cudaMemcpyHostToDevice, st));
  FCK(cudaStreamSynchronize(st));
  f->raw_rows = raw_rows;
  f->raw_cols = raw_cols;
  return UAHN_OK;
}

int uahn_filter_frame_raw(uahn_filter* f, uahn_handle* h_iter, const uint8_t* raw, size_t stride, int max_iter,
                          double K_net_Cov, int min_images, const uint8_t* use_measurement, const uahn_rng* rng,
                          float* prior_out, float* mean_out, float* cov_out, double* imu_out) {
  if (!f) return UAHN_ERR_INVALID;
  int rc = check_raw(f, "uahn_filter_frame_raw", raw, stride);
  if (rc || (rc = check_frame(f, "uahn_filter_frame_raw", h_iter, max_iter, rng))) return rc;
  auto remap = [&](uint8_t* curr) { return enqueue_raw(f, raw, stride, curr); };
  return run_frame(f, "uahn_filter_frame_raw", h_iter, remap, max_iter, K_net_Cov, min_images, use_measurement, rng,
                   prior_out, mean_out, cov_out, imu_out);
}

int uahn_filter_stage_undistort(uahn_filter* f, const uint8_t* raw, size_t stride, uint8_t* out) {
  if (!f) return UAHN_ERR_INVALID;
  int rc = check_raw(f, "uahn_filter_stage_undistort", raw, stride);
  if (rc) return rc;
  if (!out) return handle_fail(f->h, UAHN_ERR_INVALID, "uahn_filter_stage_undistort: null out");
  FCK(cudaSetDevice(f->device));
  cudaStream_t st = stream_of(f->h);
  const size_t bytes = (size_t)f->n * UAHN_IMG_PIXELS;
  uint8_t* d_out = nullptr;
  FCK(cudaMalloc(&d_out, bytes));
  auto step = [&]() -> int {
    int r = enqueue_raw(f, raw, stride, d_out);
    if (r) return r;
    FCK(cudaMemcpyAsync(out, d_out, bytes, cudaMemcpyDeviceToHost, st));
    FCK(cudaStreamSynchronize(st));
    return UAHN_OK;
  };
  rc = step();
  if (rc) cudaStreamSynchronize(st);              // whatever was enqueued may still write d_out
  cudaFree(d_out);
  return rc;
}

int uahn_filter_wait(uahn_filter* f, int* status) {
  if (!f) return UAHN_ERR_INVALID;
  FCK(cudaSetDevice(f->device));
  cudaStream_t st = stream_of(f->h);
  FCK(cudaMemcpyAsync(f->h_status, f->d_status, (size_t)f->n * sizeof(int), cudaMemcpyDeviceToHost, st));
  FCK(cudaMemsetAsync(f->d_status, 0, (size_t)f->n * sizeof(int), st));
  FCK(cudaStreamSynchronize(st));
  if (status) memcpy(status, f->h_status, (size_t)f->n * sizeof(int));
  for (int i = 0; i < f->n; ++i)
    if (f->h_status[i]) return f->h_status[i];
  return UAHN_OK;
}

}  // extern "C"
