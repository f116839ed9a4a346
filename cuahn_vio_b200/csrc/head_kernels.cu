// Regression / uncertainty head kernels of the UAHN cascade:
//   * 4-point DLT solve (model_to_trace.py:42-61) in closed form, fp64, every lane of a pair's warp redundantly
//   * Linear(5120->8) + DLT + homography composition H <- H·H_b (model_to_trace.py:143-150,163-168,183-188)
//   * MC-dropout expansion of the block-4 feature (model_to_trace.py:222-235,272-273)
//   * second head layer, 16-sample ensemble (model_to_trace.py:274-281), covariance transfer
//     (model_to_trace.py:18-38), output packing and the showError homography (model_to_trace.py:311-323)
#include "common.cuh"
#include "kernels.h"
#include "tc_ptx.cuh"

namespace uahn {
namespace {

__device__ __forceinline__ void corner(int i, float& x, float& y) {   // model_to_trace.py:78-83: UL, BL, BR, UR
  x = (i == 2 || i == 3) ? (float)(IMG_W - 1) : 0.f;
  y = (i == 1 || i == 2) ? (float)(IMG_H - 1) : 0.f;
}

// The DLT solve.  The four source points are always the corners of the 320 x 224 frame
// (model_to_trace.py:78-83), so the 8x8 system is the square-to-quadrilateral mapping (Heckbert, "Fundamentals of Texture
// Mapping and Image Warping", 1989, sec. 2.2.3) composed with the frame's scaling: with (u, v) = (x / (W-1), y / (H-1)) and
// the unit square's corners (0,0), (1,0), (1,1), (0,1) going to q0, q1, q2, q3,
//   g = | S  d2 | / | d1 d2 |,  h = | d1 S | / | d1 d2 |   (d1 = q1 - q2, d2 = q3 - q2, S = q0 - q1 + q2 - q3),
//   X = (a u + b v + c) / (g u + h v + 1) with a = q1.x - q0.x + g q1.x, b = q3.x - q0.x + h q3.x, c = q0.x (Y alike).
// ~40 fp64 operations per lane and no shuffles: a warp-shuffle Gauss-Jordan elimination of the general system spends ~3 us
// more per DLT launch on the batch-1 chain.  Same exact solution, far inside the fp32 noise of the reference's torch.inverse
// (tests/test_gpu_parity.py::test_stage_dlt_matches_reference).
__device__ __forceinline__ void dlt_rect(const float* dst, double* h) {
  // corner order of the model: UL, BL, BR, UR  ->  q0 = UL, q1 = UR, q2 = BR, q3 = BL
  const double x0 = dst[0], y0 = dst[1], x3 = dst[2], y3 = dst[3], x2 = dst[4], y2 = dst[5], x1 = dst[6], y1 = dst[7];
  const double dx1 = x1 - x2, dx2 = x3 - x2, dy1 = y1 - y2, dy2 = y3 - y2;
  const double sx = (x0 - x1) + (x2 - x3), sy = (y0 - y1) + (y2 - y3);
  const double inv = 1.0 / (dx1 * dy2 - dy1 * dx2);
  const double g = (sx * dy2 - sy * dx2) * inv, k = (dx1 * sy - dy1 * sx) * inv;
  constexpr double IW = 1.0 / (IMG_W - 1), IH = 1.0 / (IMG_H - 1);
  h[0] = ((x1 - x0) + g * x1) * IW; h[1] = ((x3 - x0) + k * x3) * IH; h[2] = x0;
  h[3] = ((y1 - y0) + g * y1) * IW; h[4] = ((y3 - y0) + k * y3) * IH; h[5] = y0;
  h[6] = g * IW; h[7] = k * IH; h[8] = 1.0;
}

// fp32 3x3 product, k accumulated sequentially with FMA (torch.bmm on CPU)
__device__ __forceinline__ void mat3_mul(const float* A, const float* B, float* C) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      C[i * 3 + j] = __fmaf_rn(A[i * 3 + 2], B[6 + j], __fmaf_rn(A[i * 3 + 1], B[3 + j], __fmul_rn(A[i * 3], B[j])));
}

// The tail of every DLT-bearing stage, for the 8 offsets d of one pair: H_b = DLT(pts0, pts0 + d), then
// Hout[pair] = Hprev ? Hprev[pair]·H_b : H_b.  Called by a whole warp: every lane solves, lane 0 stores.
__device__ __forceinline__ void dlt_compose_store(const float* d, int pair, const float* Hprev, float* Hout) {
  float dst[8];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float x, y;
    corner(i, x, y);
    dst[2 * i] = __fadd_rn(x, d[2 * i]);
    dst[2 * i + 1] = __fadd_rn(y, d[2 * i + 1]);
  }
  double h[9];
  dlt_rect(dst, h);
  if ((threadIdx.x & 31) == 0) {
    float hb[9], out[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) hb[i] = (float)h[i];
    if (Hprev) {
      float hp[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) hp[i] = Hprev[pair * 9 + i];
      mat3_mul(hp, hb, out);
    } else {
#pragma unroll
      for (int i = 0; i < 9; ++i) out[i] = hb[i];
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) Hout[pair * 9 + i] = out[i];
  }
}

// H = DLT(pts0, pts0 + off); optional left-multiplication by Hprev.  One warp per pair.
__global__ void dlt_kernel(int n, const float* __restrict__ off, const float* __restrict__ Hprev, float* __restrict__ Hout) {
  pdl_wait();
  pdl_launch_dependents();
  const int pair = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (pair >= n) return;
  dlt_compose_store(off + pair * 8, pair, Hprev, Hout);
}

// d = W8·feat + b8 ; H_b = DLT(pts0, pts0 + d) ; Hout = Hprev ? Hprev·H_b : H_b.
// feat is the last conv output in NHWC order ((h*5+w)*256 + c); W8 was permuted to that order at load.
// Batch path (round 2): eight pairs per CTA.  A thread owns five 4-element slices of k (k = 4 (t + 256 i)): per slice eight
// 16-byte weight loads serve 8 pairs x 8 outputs x 4 k = 256 FMAs, so the L2 -> SM weight traffic per pair is half that of
// 4 pairs per CTA with scalar loads, and a thread waits for 5 batches of 16 wide loads instead of 20 trips of 12
// scalar ones — the stage is a chain of L2 round trips, nothing else (16 us per launch at 1024 pairs, issue slots 23 % busy).
// The 64 partial sums of a thread meet in shared memory ([output][thread], conflict-free) and are added in a fixed order.
constexpr int FC8W_PAIRS = 8;
constexpr size_t FC8W_SMEM = (size_t)FC8W_PAIRS * 8 * 257 * sizeof(float);
template <typename T>
__global__ void __launch_bounds__(256, 1) fc8_dlt_wide_kernel(int n, const T* __restrict__ feat, const float* __restrict__ W8,
                                                             const float* __restrict__ b8, const float* __restrict__ Hprev,
                                                             float* __restrict__ Hout, float* __restrict__ dout) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ __align__(16) float red_w[];              // [64][257]
  __shared__ float d_s[FC8W_PAIRS][8];
  const int pair0 = blockIdx.x * FC8W_PAIRS, tid = threadIdx.x, wid = tid >> 5;
  const int np = min(FC8W_PAIRS, n - pair0);
  float acc[FC8W_PAIRS][8];
#pragma unroll
  for (int p = 0; p < FC8W_PAIRS; ++p)
#pragma unroll
    for (int o = 0; o < 8; ++o) acc[p][o] = 0.f;
#pragma unroll
  for (int i = 0; i < FC_IN / (4 * 256); ++i) {
    const int k = 4 * (tid + 256 * i);
    float4 w[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) w[o] = __ldg(reinterpret_cast<const float4*>(W8 + o * FC_IN + k));
    float x[FC8W_PAIRS][4];
#pragma unroll
    for (int p = 0; p < FC8W_PAIRS; ++p) {
      const T* f = feat + (size_t)(pair0 + (p < np ? p : 0)) * FC_IN + k;      // (pairs past n re-read pair0; results dropped)
      if constexpr (sizeof(T) == 2) {
        const uint2 v = *reinterpret_cast<const uint2*>(f);
        x[p][0] = __uint_as_float(v.x << 16); x[p][1] = __uint_as_float(v.x & 0xffff0000u);
        x[p][2] = __uint_as_float(v.y << 16); x[p][3] = __uint_as_float(v.y & 0xffff0000u);
      } else {
        const float4 v = *reinterpret_cast<const float4*>(f);
        x[p][0] = v.x; x[p][1] = v.y; x[p][2] = v.z; x[p][3] = v.w;
      }
    }
#pragma unroll
    for (int p = 0; p < FC8W_PAIRS; ++p)
#pragma unroll
      for (int o = 0; o < 8; ++o) {
        acc[p][o] = fmaf(x[p][0], w[o].x, acc[p][o]);
        acc[p][o] = fmaf(x[p][1], w[o].y, acc[p][o]);
        acc[p][o] = fmaf(x[p][2], w[o].z, acc[p][o]);
        acc[p][o] = fmaf(x[p][3], w[o].w, acc[p][o]);
      }
  }
#pragma unroll
  for (int p = 0; p < FC8W_PAIRS; ++p)
#pragma unroll
    for (int o = 0; o < 8; ++o) red_w[(p * 8 + o) * 257 + tid] = acc[p][o];
  __syncthreads();
  {   // output tid / 4, quarter tid % 4 of the 256 partial sums, then the four quarters in lane order
    const int po = tid >> 2, qt = tid & 3;
    float v = 0.f;
#pragma unroll 8
    for (int j = 0; j < 64; ++j) v += red_w[po * 257 + qt * 64 + j];
    const float v1 = __shfl_down_sync(0xffffffffu, v, 1), v2 = __shfl_down_sync(0xffffffffu, v, 2), v3 = __shfl_down_sync(0xffffffffu, v, 3);
    if (qt == 0) {
      const float sum = ((v + v1) + v2) + v3 + b8[po & 7];
      d_s[po >> 3][po & 7] = sum;
      if (dout && (po >> 3) < np) dout[(pair0 + (po >> 3)) * 8 + (po & 7)] = sum;
    }
  }
  __syncthreads();
  if (wid < np) dlt_compose_store(d_s[wid], pair0 + wid, Hprev, Hout);   // one warp per pair
}

// Latency path (<= FC8_SMALL_MAX pairs): the same stage with the 5120-long dot products split over a cluster of 8 CTAs per
// pair (640 k each, 8 x fewer dependent L2 round trips per thread), partial sums reduced through distributed shared
// memory into rank 0, which adds the bias and runs the DLT + composition.  (One CTA per 4 pairs takes 20 us at batch 1.)
constexpr int FC8_SMALL_MAX = 8;
constexpr int FC8_CLUSTER = 8;
template <typename T>
__global__ void __cluster_dims__(FC8_CLUSTER, 1, 1) __launch_bounds__(256)
    fc8_dlt_cluster_kernel(int n, const T* __restrict__ feat, const float* __restrict__ W8, const float* __restrict__ b8,
                           const float* __restrict__ Hprev, float* __restrict__ Hout, float* __restrict__ dout) {
  __shared__ float part[8][8];
  __shared__ float red[FC8_CLUSTER][8];     // rank 0's copy collects every rank's partial sums
  __shared__ float d_s[8];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x / FC8_CLUSTER;
  constexpr int KPER = FC_IN / FC8_CLUSTER;   // 640
  constexpr int TRIPS = (KPER + 255) / 256;
  const int k0 = (int)rank * KPER;
  // this thread's 8 x 3 weights are requested before griddepcontrol.wait: only the feature comes from the previous kernel
  float w[TRIPS][8];
#pragma unroll
  for (int i = 0; i < TRIPS; ++i) {
    const int k = k0 + min(tid + 256 * i, KPER - 1);
#pragma unroll
    for (int o = 0; o < 8; ++o) w[i][o] = __ldg(W8 + o * FC_IN + k);
  }
  pdl_wait();
  pdl_launch_dependents();
  float acc[8];
#pragma unroll
  for (int o = 0; o < 8; ++o) acc[o] = 0.f;
#pragma unroll
  for (int i = 0; i < TRIPS; ++i) {
    const int kk = tid + 256 * i;
    if (kk < KPER) {
      const int k = k0 + kk;
      const float x = to_f32<T>(feat[(size_t)pair * FC_IN + k]);
#pragma unroll
      for (int o = 0; o < 8; ++o) acc[o] = fmaf(x, w[i][o], acc[o]);
    }
  }
#pragma unroll
  for (int o = 0; o < 8; ++o) {
#pragma unroll
    for (int sft = 16; sft >= 1; sft >>= 1) acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], sft);
    if (lane == 0) part[wid][o] = acc[o];
  }
  __syncthreads();
  if (tid < 8) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += part[w][tid];
    // red[rank][tid] in the shared memory of cluster rank 0
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(&red[rank][tid])), "r"(0u));
    asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(remote), "f"(v) : "memory");
  }
  cluster_sync_all();                        // release / acquire: the remote stores are visible to rank 0
  if (rank != 0) return;
  if (tid < 8) {
    float v = 0.f;
#pragma unroll
    for (int c = 0; c < FC8_CLUSTER; ++c) v += red[c][tid];
    v += b8[tid];
    d_s[tid] = v;
    if (dout) dout[pair * 8 + tid] = v;
  }
  __syncthreads();
  if (wid == 0) dlt_compose_store(d_s, pair, Hprev, Hout);   // one warp
}

// A'[head][pair][s][k'] = keep ? feat[k'] * (1/0.95) : 0     (Dropout(0.05) on the repeated feature)
// k' = NHWC index (hw*256 + c); explicit masks are indexed in the reference order kref = c*20 + hw.
// alias table of the keep-byte generator (common.cuh: alias_keep_byte), uploaded once per device by
// init_keep_alias_table()
__device__ uint32_t g_keep_alias[256];

template <typename T>
__global__ void __launch_bounds__(256) mc_expand_kernel(const T* __restrict__ feat, T* __restrict__ A, int n,
                                                         const uint8_t* __restrict__ keep_masks, uint64_t seed,
                                                         uint64_t first_pair, const uint64_t* __restrict__ rng_dev) {
  pdl_wait();
  pdl_launch_dependents();
  if (rng_dev) { seed = rng_dev[0]; first_pair = rng_dev[1]; }   // graph replay: values live in device memory
  const int pair = blockIdx.x, head = blockIdx.y;
  const T* f = feat + (size_t)pair * FC_IN;
  T* a = A + ((size_t)head * n + pair) * MC * FC_IN;
  for (int i = threadIdx.x; i < MC * (FC_IN / 8); i += blockDim.x) {
    const int s = i / (FC_IN / 8), k8 = i - s * (FC_IN / 8);
    uint32_t bits;
    if (keep_masks) {
      const uint8_t* m = keep_masks + ((size_t)(pair * 2 + head) * MC + s) * MASK_ROW;
      bits = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int kp = k8 * 8 + j, hw = kp >> 8, c = kp & 255;
        bits |= (m[c * 20 + hw] ? 1u : 0u) << j;
      }
    } else {
      bits = philox_keep8(seed, first_pair + pair, head, 0, s, k8, g_keep_alias);
    }
    T v[8];
    if constexpr (sizeof(T) == 2) {
      *reinterpret_cast<uint4*>(v) = *reinterpret_cast<const uint4*>(f + k8 * 8);     // 8 bf16 features
    } else {
      *reinterpret_cast<float4*>(v) = *reinterpret_cast<const float4*>(f + k8 * 8);
      *reinterpret_cast<float4*>(v + 4) = *reinterpret_cast<const float4*>(f + k8 * 8 + 4);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
      v[j] = from_f32<T>((bits >> j) & 1u ? __fmul_rn(to_f32<T>(v[j]), KEEP_SCALE) : 0.f);
    T* dstp = a + (size_t)s * FC_IN + k8 * 8;
    if constexpr (sizeof(T) == 2) {
      *reinterpret_cast<uint4*>(dstp) = *reinterpret_cast<const uint4*>(v);
    } else {
      *reinterpret_cast<float4*>(dstp) = *reinterpret_cast<const float4*>(v);
      *reinterpret_cast<float4*>(dstp + 4) = *reinterpret_cast<const float4*>(v + 4);
    }
  }
}

// First MC-head layer for the batch-1 latency path: hid[pair][s][j] = LeakyReLU(sum_k A[pair][s][k] * W[j][k] + b[j]) on
// CUDA cores.  With one or a few pairs the tensor-core GEMM is a handful of CTAs each walking all 80 K stages in
// sequence (25 us per head at batch 1); here 64 CTAs per pair and head each take 4 output columns, read the 16 masked
// sample rows once, and reduce across the block.  A: [n][16][5120] bf16 (mc_expand), W: [256][5120] bf16 in the same
// (NHWC) k order, out: [n][16][256] bf16 with the tensor path's epilogue arithmetic (bf16 round, LeakyReLU on bf16).
constexpr int FC1S_JT = 4;
__global__ void __launch_bounds__(256) mc_fc1_small_kernel(const __nv_bfloat16* __restrict__ A, const __nv_bfloat16* __restrict__ W,
                                                            const float* __restrict__ bias, __nv_bfloat16* __restrict__ out) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ float part[8][MC][FC1S_JT];
  const int j0 = blockIdx.x * FC1S_JT, pair = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const uint4* a4 = reinterpret_cast<const uint4*>(A + (size_t)pair * MC * FC_IN);
  const uint4* w4 = reinterpret_cast<const uint4*>(W + (size_t)j0 * FC_IN);
  float acc[MC][FC1S_JT];
#pragma unroll
  for (int s = 0; s < MC; ++s)
#pragma unroll
    for (int j = 0; j < FC1S_JT; ++j) acc[s][j] = 0.f;
  auto lo = [](uint32_t v) { return __uint_as_float(v << 16); };
  auto hi = [](uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); };
  for (int g = tid; g < FC_IN / 8; g += 256) {
    float wf[FC1S_JT][8];
#pragma unroll
    for (int j = 0; j < FC1S_JT; ++j) {
      const uint4 w = __ldg(w4 + (size_t)j * (FC_IN / 8) + g);
      wf[j][0] = lo(w.x); wf[j][1] = hi(w.x); wf[j][2] = lo(w.y); wf[j][3] = hi(w.y);
      wf[j][4] = lo(w.z); wf[j][5] = hi(w.z); wf[j][6] = lo(w.w); wf[j][7] = hi(w.w);
    }
#pragma unroll
    for (int s = 0; s < MC; ++s) {
      const uint4 a = __ldg(a4 + (size_t)s * (FC_IN / 8) + g);
      const float af[8] = {lo(a.x), hi(a.x), lo(a.y), hi(a.y), lo(a.z), hi(a.z), lo(a.w), hi(a.w)};
#pragma unroll
      for (int j = 0; j < FC1S_JT; ++j)
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[s][j] = fmaf(af[e], wf[j][e], acc[s][j]);
    }
  }
#pragma unroll
  for (int s = 0; s < MC; ++s)
#pragma unroll
    for (int j = 0; j < FC1S_JT; ++j) {
      float v = acc[s][j];
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) part[wid][s][j] = v;
    }
  __syncthreads();
  if (tid < MC * FC1S_JT / 2) {            // one thread per pair of adjacent output columns
    const int s = tid / (FC1S_JT / 2), jp = (tid % (FC1S_JT / 2)) * 2;
    float v0 = bias[j0 + jp], v1 = bias[j0 + jp + 1];
#pragma unroll
    for (int w = 0; w < 8; ++w) { v0 += part[w][s][jp]; v1 += part[w][s][jp + 1]; }
    reinterpret_cast<uint32_t*>(out + ((size_t)pair * MC + s) * FC_HID + j0 + jp)[0] = pack_lrelu_bf16x2(v0, v1);
  }
}

// The same layer with the MC-dropout expansion fused in and both heads in one launch (the latency path's 3 launches ->
// 1): every CTA first builds the keep bytes of its (pair, head) in shared memory — [k8][sample], bit j = keep(8*k8 + j),
// from the Philox generator or the explicit masks, exactly the bytes mc_maskbits_kernel / mc_expand_kernel use — then runs
// the dot products on feat directly: a = keep ? bf16(feat * 1/0.95) : 0, the value mc_expand_kernel would have stored.
__global__ void __launch_bounds__(256) mc_fc1_small_fused_kernel(const __nv_bfloat16* __restrict__ feat, int n,
                                                                  const __nv_bfloat16* __restrict__ Wm,
                                                                  const __nv_bfloat16* __restrict__ Wu,
                                                                  const float* __restrict__ bm, const float* __restrict__ bu,
                                                                  __nv_bfloat16* __restrict__ hid,
                                                                  const uint8_t* __restrict__ keep_masks, uint64_t seed,
                                                                  uint64_t first_pair, const uint64_t* __restrict__ rng_dev) {
  // the keep bytes depend on (seed, pair) only — uploaded in front of the whole chain — so the whole mask phase runs BEFORE
  // griddepcontrol.wait, next to the last conv layer; only the feature needs the previous kernel
  if (rng_dev) { seed = rng_dev[0]; first_pair = rng_dev[1]; }
  __shared__ float part[8][MC][FC1S_JT];
  __shared__ __align__(16) uint8_t s_bits[(FC_IN / 8) * MC];      // 10 KB
  __shared__ uint32_t s_tab[256];
  const int j0 = blockIdx.x * FC1S_JT, pair = blockIdx.y, head = blockIdx.z, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (keep_masks) {
    for (int i = tid; i < MC * (FC_IN / 8); i += 256) {
      const int k8 = i / MC, smp = i - k8 * MC;
      const uint8_t* m = keep_masks + ((size_t)(pair * 2 + head) * MC + smp) * MASK_ROW;
      uint32_t bits = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int kp = k8 * 8 + j, hw = kp >> 8, c = kp & 255;   // kernel order -> reference order c*20 + hw
        bits |= (m[c * 20 + hw] ? 1u : 0u) << j;
      }
      s_bits[i] = (uint8_t)bits;
    }
  } else {
    s_tab[tid] = g_keep_alias[tid];
    __syncthreads();
#pragma unroll 2
    for (int i = tid; i < MC * (FC_IN / 32); i += 256) {
      const int k32 = i / MC, smp = i - k32 * MC;
      uint32_t b[4];
      philox_keep32(seed, first_pair + pair, head, 0, smp, k32, s_tab, b);
#pragma unroll
      for (int qd = 0; qd < 4; ++qd) s_bits[(k32 * 4 + qd) * MC + smp] = (uint8_t)b[qd];
    }
  }
  pdl_wait();
  pdl_launch_dependents();
  __syncthreads();
  const uint4* f4 = reinterpret_cast<const uint4*>(feat + (size_t)pair * FC_IN);
  const uint4* w4 = reinterpret_cast<const uint4*>((head ? Wu : Wm) + (size_t)j0 * FC_IN);
  float acc[MC][FC1S_JT];
#pragma unroll
  for (int s_ = 0; s_ < MC; ++s_)
#pragma unroll
    for (int j = 0; j < FC1S_JT; ++j) acc[s_][j] = 0.f;
  auto lo = [](uint32_t v) { return __uint_as_float(v << 16); };
  auto hi = [](uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); };
  for (int g = tid; g < FC_IN / 8; g += 256) {
    float wf[FC1S_JT][8];
#pragma unroll
    for (int j = 0; j < FC1S_JT; ++j) {
      const uint4 w = __ldg(w4 + (size_t)j * (FC_IN / 8) + g);
      wf[j][0] = lo(w.x); wf[j][1] = hi(w.x); wf[j][2] = lo(w.y); wf[j][3] = hi(w.y);
      wf[j][4] = lo(w.z); wf[j][5] = hi(w.z); wf[j][6] = lo(w.w); wf[j][7] = hi(w.w);
    }
    const uint4 fv = __ldg(f4 + g);
    const float fr[8] = {lo(fv.x), hi(fv.x), lo(fv.y), hi(fv.y), lo(fv.z), hi(fv.z), lo(fv.w), hi(fv.w)};
    float kept[8];                                     // the bf16 value mc_expand_kernel stores for a kept unit
#pragma unroll
    for (int e = 0; e < 8; ++e) kept[e] = __bfloat162float(__float2bfloat16_rn(__fmul_rn(fr[e], KEEP_SCALE)));
    const uint4 bw = *reinterpret_cast<const uint4*>(s_bits + g * MC);   // this granule's keep bytes of the 16 samples
    const uint32_t bword[4] = {bw.x, bw.y, bw.z, bw.w};
#pragma unroll
    for (int s_ = 0; s_ < MC; ++s_) {
      const uint32_t bits = (bword[s_ >> 2] >> (8 * (s_ & 3))) & 0xFFu;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float a = (bits >> e) & 1u ? kept[e] : 0.f;
#pragma unroll
        for (int j = 0; j < FC1S_JT; ++j) acc[s_][j] = fmaf(a, wf[j][e], acc[s_][j]);
      }
    }
  }
#pragma unroll
  for (int s_ = 0; s_ < MC; ++s_)
#pragma unroll
    for (int j = 0; j < FC1S_JT; ++j) {
      float v = acc[s_][j];
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) part[wid][s_][j] = v;
    }
  __syncthreads();
  if (tid < MC * FC1S_JT / 2) {            // one thread per pair of adjacent output columns
    const int s_ = tid / (FC1S_JT / 2), jp = (tid % (FC1S_JT / 2)) * 2;
    const float* bias = head ? bu : bm;
    float v0 = bias[j0 + jp], v1 = bias[j0 + jp + 1];
#pragma unroll
    for (int w = 0; w < 8; ++w) { v0 += part[w][s_][jp]; v1 += part[w][s_][jp + 1]; }
    __nv_bfloat16* out = hid + (size_t)head * n * MC * FC_HID;
    reinterpret_cast<uint32_t*>(out + ((size_t)pair * MC + s_) * FC_HID + j0 + jp)[0] = pack_lrelu_bf16x2(v0, v1);
  }
}

// Keep-mask BITS of the first MC dropout, consumed by the masked-A producer of the fused 5120->256 GEMMs
// (conv_bf16.cu): bits[head][pair][k8][sample] bytes, bit j of a byte = keep(k' = 8*k8 + j).  20 KB per pair instead
// of the 327 KB of materialised, masked features mc_expand_kernel writes.
__global__ void __launch_bounds__(256) mc_maskbits_kernel(uint8_t* __restrict__ bits_out, int n,
                                                           const uint8_t* __restrict__ keep_masks, uint64_t seed,
                                                           uint64_t first_pair, const uint64_t* __restrict__ rng_dev) {
  pdl_wait();
  pdl_launch_dependents();
  if (rng_dev) { seed = rng_dev[0]; first_pair = rng_dev[1]; }
  const int pair = blockIdx.x, head = blockIdx.y;
  uint8_t* o = bits_out + ((size_t)head * n + pair) * (FC_IN / 8) * MC;
  if (keep_masks) {
    for (int i = threadIdx.x; i < MC * (FC_IN / 8); i += blockDim.x) {
      const int k8 = i / MC, smp = i - k8 * MC;            // consecutive threads -> consecutive bytes
      const uint8_t* m = keep_masks + ((size_t)(pair * 2 + head) * MC + smp) * MASK_ROW;
      uint32_t bits = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int kp = k8 * 8 + j, hw = kp >> 8, c = kp & 255;   // kernel order -> reference order c*20 + hw
        bits |= (m[c * 20 + hw] ? 1u : 0u) << j;
      }
      o[i] = (uint8_t)bits;
    }
    return;
  }
  // One Philox block -> four keep bytes (32 units) of one sample through the alias table (shared-memory copy: the
  // look-up index is random).  Thread -> (block k32, sample): its bytes k8 = 4*k32 .. +3 land 16 bytes apart, the 16
  // samples of a k8 in consecutive bytes.
  __shared__ uint32_t s_tab[256];
  s_tab[threadIdx.x] = g_keep_alias[threadIdx.x];
  __syncthreads();
#pragma unroll 2      // independent Philox chains per thread: 7 dependent multiply rounds each
  for (int i = threadIdx.x; i < MC * (FC_IN / 32); i += blockDim.x) {
    const int k32 = i / MC, smp = i - k32 * MC;
    uint32_t b[4];
    philox_keep32(seed, first_pair + pair, head, 0, smp, k32, s_tab, b);
#pragma unroll
    for (int q = 0; q < 4; ++q) o[(k32 * 4 + q) * MC + smp] = (uint8_t)b[q];
  }
}

// transfer_mean_var_single for corner i (model_to_trace.py:18-38) + output packing (:311-317): projects the block-4 point
// (u, v) through the part-1 homography Hp, writes flow[2i..2i+1] = p/s - corner and rows 2i, 2i+1 of the block-diagonal
// 8x8 covariance, Cov_i = ((Hp/s) diag(vu, vv, 0) (Hp/s)^T)[0:2, 0:2], in the reference's fp32 operation order.
__device__ __forceinline__ void transfer_point(int i, const float* Hp, float u, float v, float vu, float vv, float* mean8,
                                               float* cov64) {
  float p[3];
#pragma unroll
  for (int r = 0; r < 3; ++r)
    p[r] = __fmaf_rn(Hp[r * 3 + 2], 1.f, __fmaf_rn(Hp[r * 3 + 1], v, __fmul_rn(Hp[r * 3], u)));
  const float sc = p[2];
  float x0, y0;
  corner(i, x0, y0);
  mean8[2 * i] = __fsub_rn(__fdiv_rn(p[0], sc), x0);          // model_to_trace.py:311
  mean8[2 * i + 1] = __fsub_rn(__fdiv_rn(p[1], sc), y0);
  float Hs[9];
#pragma unroll
  for (int r = 0; r < 9; ++r) Hs[r] = __fdiv_rn(Hp[r], sc);   // model_to_trace.py:30
  float c2[2][2];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      const float t0 = __fmul_rn(Hs[a * 3], vu), t1 = __fmul_rn(Hs[a * 3 + 1], vv);
      c2[a][b] = __fmaf_rn(t1, Hs[b * 3 + 1], __fmul_rn(t0, Hs[b * 3]));   // third term is exactly 0
    }
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) cov64[(2 * i + a) * 8 + b] = (b >> 1) == i ? c2[a][b & 1] : 0.f;
}

// stage entry point (parity tests): the covariance transfer alone, one thread per (pair, corner)
__global__ void transfer_kernel(int n, const float* __restrict__ var, const float* __restrict__ Hp, const float* __restrict__ pts_w,
                                float* __restrict__ mean, float* __restrict__ cov) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x, pair = t >> 2, i = t & 3;
  if (pair >= n) return;
  float H[9];
#pragma unroll
  for (int r = 0; r < 9; ++r) H[r] = Hp[pair * 9 + r];
  transfer_point(i, H, pts_w[pair * 8 + 2 * i], pts_w[pair * 8 + 2 * i + 1], var[pair * 8 + 2 * i], var[pair * 8 + 2 * i + 1],
                 mean + pair * 8, cov + (size_t)pair * 64);
}

struct HeadOut {
  float* mean;     // [n][8]
  float* cov;      // [n][64]
  float* Htot;     // [n][9] or null (showError)
  float* mc_mean;  // [n][16][8] or null (debug tap)
  float* mc_logvar;
};

// hid: [head][pair][s][256] = LeakyReLU(Linear(5120->256)(dropped feature)).  One CTA (256 threads) per pair:
// thread (head, s, o) does the second dropout + Linear(256->8); then ensemble, transfer, packing.
template <typename T>
__global__ void __launch_bounds__(256) mc_final_kernel(const T* __restrict__ hid, int n, const float* __restrict__ W2m,
                                                        const float* __restrict__ b2m, const float* __restrict__ W2u,
                                                        const float* __restrict__ b2u, const float* __restrict__ Hpart1,
                                                        const uint8_t* __restrict__ keep_masks, uint64_t seed,
                                                        uint64_t first_pair, const uint64_t* __restrict__ rng_dev,
                                                        HeadOut o) {
  // before griddepcontrol.wait: everything that does not come from the previous kernel (the second-layer weights; the rng
  // block was uploaded in front of the whole chain, and every kernel of the chain has waited on its predecessor)
  if (rng_dev) { seed = rng_dev[0]; first_pair = rng_dev[1]; }
  __shared__ __align__(16) float w2[2][8][FC_HID + 4];   // +4 floats: the 8 output rows hit 8 different bank groups
  __shared__ float outv[2][MC][8];
  __shared__ float mu_s[8], var_s[8];
  const int pair = blockIdx.x, tid = threadIdx.x;
  for (int i = tid; i < 8 * FC_HID; i += 256) {
    w2[0][i / FC_HID][i % FC_HID] = W2m[i];
    w2[1][i / FC_HID][i % FC_HID] = W2u[i];
  }
  pdl_wait();
  pdl_launch_dependents();
  __syncthreads();
  {
    const int head = tid >> 7, s = (tid >> 3) & 15, oo = tid & 7;
    const T* hrow = hid + (((size_t)head * n + pair) * MC + s) * FC_HID;
    const uint8_t* m = keep_masks ? keep_masks + ((size_t)(pair * 2 + head) * MC + s) * MASK_ROW + FC_IN : nullptr;
    float acc = 0.f;
    // the 8 lanes of one (head, sample) share the hidden-layer keep bits: lane oo owns bytes 4*oo .. 4*oo+3, the four
    // keep bytes of ONE Philox block
    uint32_t mybits[4];
    if (m) {
#pragma unroll
      for (int jo = 0; jo < 4; ++jo) {
        const int j8 = 4 * oo + jo;
        mybits[jo] = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) mybits[jo] |= (m[j8 * 8 + j] ? 1u : 0u) << j;
      }
    } else {
      philox_keep32(seed, first_pair + pair, head, 1, s, oo, g_keep_alias, mybits);
    }
    const int lane_base = (tid & 31) & ~7;
#pragma unroll
    for (int j8 = 0; j8 < FC_HID / 8; ++j8) {
      const uint32_t bits = __shfl_sync(0xffffffffu, mybits[j8 & 3], lane_base | (j8 >> 2));
      T hv[8];
      if constexpr (sizeof(T) == 2) {
        *reinterpret_cast<uint4*>(hv) = *reinterpret_cast<const uint4*>(hrow + j8 * 8);
      } else {
        *reinterpret_cast<float4*>(hv) = *reinterpret_cast<const float4*>(hrow + j8 * 8);
        *reinterpret_cast<float4*>(hv + 4) = *reinterpret_cast<const float4*>(hrow + j8 * 8 + 4);
      }
      const float4 wa = *reinterpret_cast<const float4*>(&w2[head][oo][j8 * 8]);
      const float4 wb = *reinterpret_cast<const float4*>(&w2[head][oo][j8 * 8 + 4]);
      const float wv[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float x = (bits >> j) & 1u ? __fmul_rn(to_f32<T>(hv[j]), KEEP_SCALE) : 0.f;
        acc = fmaf(x, wv[j], acc);
      }
    }
    acc += head ? b2u[oo] : b2m[oo];
    if (head) acc = __fmul_rn(acc, 1e-03f);      // model_to_trace.py:256
    outv[head][s][oo] = acc;
    if (o.mc_mean && !head) o.mc_mean[((size_t)pair * MC + s) * 8 + oo] = acc;
    if (o.mc_logvar && head) o.mc_logvar[((size_t)pair * MC + s) * 8 + oo] = acc;
  }
  __syncthreads();
  if (tid < 8) {                                 // model_to_trace.py:274-280
    float sm = 0.f, sv = 0.f;
#pragma unroll
    for (int s = 0; s < MC; ++s) {
      sm += outv[0][s][tid];
      sv += expf(outv[1][s][tid]);
    }
    const float mu = sm / (float)MC, avg_pred = sv / (float)MC;
    float se = 0.f;
#pragma unroll
    for (int s = 0; s < MC; ++s) {
      const float d = mu - outv[0][s][tid];
      se += d * d;
    }
    mu_s[tid] = mu;
    var_s[tid] = se / (float)MC + avg_pred;
  }
  __syncthreads();
  if (tid < 32) {
    const int lane = tid;
    float Hp[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) Hp[i] = Hpart1[pair * 9 + i];
    float ptsw[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float x, y;
      corner(i, x, y);
      ptsw[2 * i] = __fadd_rn(x, mu_s[2 * i]);          // model_to_trace.py:281
      ptsw[2 * i + 1] = __fadd_rn(y, mu_s[2 * i + 1]);
    }
    if (lane < 4) transfer_point(lane, Hp, ptsw[2 * lane], ptsw[2 * lane + 1], var_s[2 * lane], var_s[2 * lane + 1],
                                 o.mean + pair * 8, o.cov + (size_t)pair * 64);
    if (o.Htot) {                                       // model_to_trace.py:321-323
      double h4[9];
      dlt_rect(ptsw, h4);
      if (lane == 0) {
        float hb[9], out[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) hb[i] = (float)h4[i];
        mat3_mul(Hp, hb, out);
#pragma unroll
        for (int i = 0; i < 9; ++i) o.Htot[pair * 9 + i] = out[i];
      }
    }
  }
}

}  // namespace

cudaError_t launch_transfer(int n, const float* var, const float* Hp, const float* pts_w, float* mean, float* cov,
                            cudaStream_t st) {
  transfer_kernel<<<(4 * n + 127) / 128, 128, 0, st>>>(n, var, Hp, pts_w, mean, cov);
  return cudaGetLastError();
}

cudaError_t launch_dlt(int n, const float* off, const float* Hprev, float* Hout, cudaStream_t st) {
  const int threads = 128, pairs_per_block = threads / 32;
  return launch_pdl(dlt_kernel, dim3((n + pairs_per_block - 1) / pairs_per_block), dim3(threads), 0, st, n, off, Hprev, Hout);
}

template <typename T>
cudaError_t launch_fc8_dlt(int n, const T* feat, const float* W8, const float* b8, const float* Hprev, float* Hout,
                           float* dout, cudaStream_t st) {
  if (n <= FC8_SMALL_MAX)   // latency path: a cluster of 8 CTAs per pair (compile-time cluster dimensions)
    return launch_pdl(fc8_dlt_cluster_kernel<T>, dim3(FC8_CLUSTER * n), dim3(256), 0, st, n, feat, W8, b8, Hprev, Hout, dout);
  static SmemOptIn optin;   // per device (common.cuh)
  if (cudaError_t e = optin.ensure(fc8_dlt_wide_kernel<T>, FC8W_SMEM); e != cudaSuccess) return e;
  return launch_pdl(fc8_dlt_wide_kernel<T>, dim3((n + FC8W_PAIRS - 1) / FC8W_PAIRS), dim3(256), FC8W_SMEM, st, n, feat, W8, b8, Hprev, Hout, dout);
}
template cudaError_t launch_fc8_dlt<float>(int, const float*, const float*, const float*, const float*, float*, float*,
                                           cudaStream_t);
template cudaError_t launch_fc8_dlt<__nv_bfloat16>(int, const __nv_bfloat16*, const float*, const float*, const float*,
                                                   float*, float*, cudaStream_t);

template <typename T>
cudaError_t launch_mc_expand(int n, const T* feat, T* A, const uint8_t* keep_masks, uint64_t seed, uint64_t first_pair,
                             const uint64_t* rng_dev, cudaStream_t st) {
  return launch_pdl(mc_expand_kernel<T>, dim3(n, 2), dim3(256), 0, st, feat, A, n, keep_masks, seed, first_pair, rng_dev);
}
template cudaError_t launch_mc_expand<float>(int, const float*, float*, const uint8_t*, uint64_t, uint64_t,
                                             const uint64_t*, cudaStream_t);
template cudaError_t launch_mc_expand<__nv_bfloat16>(int, const __nv_bfloat16*, __nv_bfloat16*, const uint8_t*,
                                                     uint64_t, uint64_t, const uint64_t*, cudaStream_t);

cudaError_t launch_mc_fc1_small(int n, const void* A, const void* W, const float* bias, void* out, cudaStream_t st) {
  return launch_pdl(mc_fc1_small_kernel, dim3(FC_HID / FC1S_JT, n), dim3(256), 0, st, (const __nv_bfloat16*)A,
                    (const __nv_bfloat16*)W, bias, (__nv_bfloat16*)out);
}

cudaError_t launch_mc_fc1_small_fused(int n, const void* feat, const void* Wm, const void* Wu, const float* bm, const float* bu,
                                      void* hid, const uint8_t* keep_masks, uint64_t seed, uint64_t first_pair,
                                      const uint64_t* rng_dev, cudaStream_t st) {
  return launch_pdl(mc_fc1_small_fused_kernel, dim3(FC_HID / FC1S_JT, n, 2), dim3(256), 0, st, (const __nv_bfloat16*)feat, n,
                    (const __nv_bfloat16*)Wm, (const __nv_bfloat16*)Wu, bm, bu, (__nv_bfloat16*)hid, keep_masks, seed,
                    first_pair, rng_dev);
}

// host side: build the alias table and upload it to the current device (idempotent; called by uahn_create)
cudaError_t init_keep_alias_table() {
  uint32_t tab[256];
  build_keep_alias_table(tab);
  return cudaMemcpyToSymbol(g_keep_alias, tab, sizeof(tab));
}

cudaError_t launch_mc_maskbits(int n, uint8_t* bits, const uint8_t* keep_masks, uint64_t seed, uint64_t first_pair,
                               const uint64_t* rng_dev, cudaStream_t st) {
  return launch_pdl(mc_maskbits_kernel, dim3(n, 2), dim3(256), 0, st, bits, n, keep_masks, seed, first_pair, rng_dev);
}

template <typename T>
cudaError_t launch_mc_final(int n, const T* hid, const float* W2m, const float* b2m, const float* W2u,
                            const float* b2u, const float* Hpart1, const uint8_t* keep_masks, uint64_t seed,
                            uint64_t first_pair, const uint64_t* rng_dev, float* mean, float* cov, float* Htot,
                            float* mc_mean, float* mc_logvar, cudaStream_t st) {
  HeadOut o{mean, cov, Htot, mc_mean, mc_logvar};
  return launch_pdl(mc_final_kernel<T>, dim3(n), dim3(256), 0, st, hid, n, W2m, b2m, W2u, b2u, Hpart1, keep_masks, seed, first_pair, rng_dev, o);
}
template cudaError_t launch_mc_final<float>(int, const float*, const float*, const float*, const float*, const float*,
                                            const float*, const uint8_t*, uint64_t, uint64_t, const uint64_t*, float*,
                                            float*, float*, float*, float*, cudaStream_t);
template cudaError_t launch_mc_final<__nv_bfloat16>(int, const __nv_bfloat16*, const float*, const float*,
                                                    const float*, const float*, const float*, const uint8_t*, uint64_t,
                                                    uint64_t, const uint64_t*, float*, float*, float*, float*, float*,
                                                    cudaStream_t);

}  // namespace uahn
