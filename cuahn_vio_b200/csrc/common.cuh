// Shared definitions for the UAHN sm_100a kernels and the host engine.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#ifdef __CUDACC__
#include <atomic>
#endif

namespace uahn {

constexpr int IMG_H = 224;
constexpr int IMG_W = 320;
constexpr int IMG_PIXELS = IMG_H * IMG_W;
constexpr int MC = 16;          // MC-dropout samples (model_to_trace.py:202)
constexpr int FC_IN = 5120;     // 256 x 4 x 5  (model_to_trace.py:89)
constexpr int FC_HID = 256;     // model_to_trace.py:224
constexpr float LRELU_SLOPE = 0.1f;
constexpr float KEEP_SCALE = 1.0f / 0.95f;  // nn.Dropout(p=0.05) in train mode
constexpr int MASK_ROW = FC_IN + FC_HID;    // explicit keep-mask bytes per (head, sample)

// Activation tensors are zero-haloed NHWC ("padded NHWC"): [n][ph + H + ph][pwl + W + pwr][C].
// The halo is the consuming convolution's zero padding, materialised once (cudaMemset at
// allocation; kernels only ever write the interior), so conv producers need no bounds checks.
struct Tensor {
  void* p = nullptr;
  int N = 0, H = 0, W = 0, C = 0;
  int ph = 0, pwl = 0, pwr = 0;
  int Hp = 0, Wp = 0;        // padded extents
  long long pitch_n = 0;     // elements between consecutive images
  __host__ __device__ long long pitch_y() const { return (long long)Wp * C; }
  __host__ __device__ long long off(int n, int y, int x, int c = 0) const {
    return (long long)n * pitch_n + ((long long)(y + ph) * Wp + (x + pwl)) * C + c;
  }
};

// One convolution (or dense layer seen as a 1x1 convolution over a 1x1 image).
struct ConvGeom {
  int M;                 // output pixels over the whole batch = N * Ho * Wo
  int Ho, Wo;
  int Cin, Cout;
  int KH, KW, stride;
  int K;                 // KH * KW * Cin, ordered (ky, kx, c) — c fastest
  long long in_pitch_n, in_pitch_y;    // elements
  long long in_origin;   // element offset of tap (ky=0,kx=0,c=0) of output pixel (0,0) in image 0
  long long out_pitch_n, out_pitch_y;  // elements
  long long out_origin;  // element offset of output pixel (0,0), channel 0 in image 0
  int act;               // 1: LeakyReLU(0.1), 0: identity
};

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------------
// Every kernel of the forward is launched with cudaLaunchAttributeProgrammaticStreamSerialization: the next
// kernel's CTAs may become resident and run their prologue (barrier init, TMEM allocation, weight loads) while the
// previous kernel drains, and block in pdl_wait() until its memory is visible.  Nothing produced by an earlier
// kernel may be read, and nothing may be written to global memory, before pdl_wait() — and EVERY kernel of the chain calls it,
// even one that reads nothing from its predecessor: a grid that never waits could complete before the grid in front of it and
// release its own dependents too early.  Used at every batch size (engine.cu: pdl_enabled); UAHN_NO_PDL=1 disables it.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// Grids that fit the machine in one wave (the latency path: 28-CTA warp bands, 32-CTA split-K clusters) let their dependents
// start right away — the next kernel's prologue (barrier init, TMEM allocation, weight prefetch) then overlaps this grid
// instead of starting when its last CTA exits.  Many-wave grids keep the implicit trigger at exit: early dependents would hold
// SM resources that their own later CTAs still need.
__device__ __forceinline__ void pdl_launch_dependents_if_single_wave() {
  if (gridDim.x * gridDim.y * gridDim.z <= 128) pdl_launch_dependents();
}

#ifdef __CUDACC__
// ---- per-device host-side caches ----------------------------------------------------------------------------
// cudaFuncAttributeMaxDynamicSharedMemorySize and the SM count belong to a DEVICE, and one process may hold handles on
// several GPUs (uahn_config.device), so the caches are indexed by the current device.  Plain relaxed atomics: a racing
// second cudaFuncSetAttribute / attribute query is harmless.
constexpr int UAHN_MAX_DEVICES = 64;
inline int current_device() {
  int d = 0;
  cudaGetDevice(&d);
  return (d >= 0 && d < UAHN_MAX_DEVICES) ? d : 0;
}
inline int device_num_sms() {
  static std::atomic<int> sms[UAHN_MAX_DEVICES];
  int dev = 0;
  cudaGetDevice(&dev);
  int v = (dev >= 0 && dev < UAHN_MAX_DEVICES) ? sms[dev].load(std::memory_order_relaxed) : 0;
  if (!v) {
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    if (dev >= 0 && dev < UAHN_MAX_DEVICES) sms[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}
struct SmemOptIn {   // one (function-local static) per kernel instantiation
  std::atomic<size_t> bytes[UAHN_MAX_DEVICES];
  template <typename K>
  cudaError_t ensure(K kern, size_t smem) {
    int dev = 0;
    cudaGetDevice(&dev);
    const bool cached = dev >= 0 && dev < UAHN_MAX_DEVICES;
    if (cached && smem <= bytes[dev].load(std::memory_order_relaxed)) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess && cached) bytes[dev].store(smem, std::memory_order_relaxed);
    return e;
  }
};

bool pdl_enabled();   // engine.cu: on for a thread once it has run a forward(), unless UAHN_NO_PDL is set
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
#endif

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ float lrelu(float v) { return v > 0.f ? v : v * LRELU_SLOPE; }

// ---- Philox4x32-7 (host + device): the in-kernel MC-dropout mask source ---------------------------------
// 7 rounds is the smallest Crush-resistant Philox4x32 (Salmon et al., SC'11; 10 is the library default's safety
// margin).  The masks cost 5 120 Philox blocks per pair and head.
constexpr int PHILOX_ROUNDS = 7;
struct Philox {
  static constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
  __host__ __device__ static inline void mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
    unsigned long long p = (unsigned long long)a * b;
    hi = (uint32_t)(p >> 32);
    lo = (uint32_t)p;
  }
  __host__ __device__ static inline void gen(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                             uint32_t out[4]) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < PHILOX_ROUNDS; ++r) {
      uint32_t h0, l0, h1, l1;
      mulhilo(M0, c0, h0, l0);
      mulhilo(M1, c2, h1, l1);
      uint32_t n0 = h1 ^ c1 ^ k0, n1 = l1, n2 = h0 ^ c3 ^ k1, n3 = l0;
      c0 = n0; c1 = n1; c2 = n2; c3 = n3;
      k0 += W0; k1 += W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
  }
};
// The keep byte of 8 consecutive units comes from ONE 32-bit uniform through a Walker/Vose alias table over the 256
// byte patterns: P(byte = b) = 19^popcount(b) / 20^8, i.e. every unit is kept independently with probability 0.95
// (nn.Dropout(p = 0.05)), exact up to the 24-bit column threshold.  One Philox block therefore serves 32 units instead
// of 8 (the rounds are the run time of mc_maskbits_kernel) and the decode is branch-free: no per-unit compare.
//   tab[c] = threshold(24 bits) << 8 | alias(8 bits);  byte = (u & 0xFFFFFF) < threshold ? c : alias,  c = u >> 24.
__host__ __device__ inline uint32_t alias_keep_byte(uint32_t u, const uint32_t* tab) {
  const uint32_t c = u >> 24, e = tab[c];
  return (u & 0xFFFFFFu) < (e >> 8) ? c : (e & 0xFFu);
}
// Exact integer construction (Vose): pattern weights 256 * 19^popcount against a column capacity of 20^8, so the table
// is the same on every host that builds it.
inline void build_keep_alias_table(uint32_t tab[256]) {
  const unsigned long long W = 25600000000ull;            // 20^8
  unsigned long long pow19[9], w[256];
  pow19[0] = 1;
  for (int i = 1; i <= 8; ++i) pow19[i] = pow19[i - 1] * 19ull;
  int small[256], large[256], ns = 0, nl = 0;
  unsigned long long thr[256];
  int alias[256];
  for (int b = 0; b < 256; ++b) {
    int pop = 0;
    for (int j = 0; j < 8; ++j) pop += (b >> j) & 1;
    w[b] = 256ull * pow19[pop];
    thr[b] = W;
    alias[b] = b;
    if (w[b] < W) small[ns++] = b; else large[nl++] = b;
  }
  while (ns > 0 && nl > 0) {
    const int l = small[--ns], g = large[--nl];
    thr[l] = w[l];
    alias[l] = g;
    w[g] = w[g] + w[l] - W;
    if (w[g] < W) small[ns++] = g; else large[nl++] = g;
  }
  for (int b = 0; b < 256; ++b) {
    unsigned long long t24 = thr[b] >= W ? 0xFFFFFFull : (thr[b] << 24) / W;   // floor(thr * 2^24 / 20^8), thr < 2^35
    tab[b] = (uint32_t)(t24 << 8) | (uint32_t)alias[b];
  }
}
// keep byte for (pair, head, layer, sample, index / 8): Philox block idx8 / 4, word idx8 % 4.  bit j = keep(idx8*8 + j).
__host__ __device__ inline uint32_t philox_keep8(uint64_t seed, uint64_t pair, int head, int layer, int sample, int idx8,
                                                 const uint32_t* alias_tab) {
  uint32_t r[4];
  Philox::gen(seed, (uint32_t)(idx8 >> 2), (uint32_t)(sample | (head << 8) | (layer << 16)), (uint32_t)pair,
              (uint32_t)(pair >> 32), r);
  const uint32_t u = (idx8 & 2) ? ((idx8 & 1) ? r[3] : r[2]) : ((idx8 & 1) ? r[1] : r[0]);
  return alias_keep_byte(u, alias_tab);
}
// the four keep bytes of Philox block idx32 (units idx32*32 ... +31) from one block
__host__ __device__ inline void philox_keep32(uint64_t seed, uint64_t pair, int head, int layer, int sample, int idx32,
                                              const uint32_t* alias_tab, uint32_t out[4]) {
  uint32_t r[4];
  Philox::gen(seed, (uint32_t)idx32, (uint32_t)(sample | (head << 8) | (layer << 16)), (uint32_t)pair,
              (uint32_t)(pair >> 32), r);
#pragma unroll
  for (int i = 0; i < 4; ++i) out[i] = alias_keep_byte(r[i], alias_tab);
}

}  // namespace uahn
