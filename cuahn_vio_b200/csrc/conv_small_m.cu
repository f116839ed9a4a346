// Latency path of the deep bf16 convolutions (model_to_trace.py:94-95,102-103,112-113,215-216 at batch 1-2): split-K over a
// cluster of 8 CTAs.
//
// At batch 1 the layers from 14x20 down have 20 or 70 GEMM rows against K = 1152 ... 3200: through the tcgen05 kernel they are
// 2-4 CTAs, each streaming 150-400 KB of weights through one SM while 140 SMs idle (8-14 us per layer, the longest links of
// the 27-kernel chain).  Here the work is cut the other way: CTA (n-slab j, rank r) of cluster j takes 64 output channels and
// one eighth of the (tap, 64-channel chunk) K stages, so 16-32 SMs each pull 18-50 KB of weights; the fp32 partial tiles meet in
// distributed shared memory and every rank reduces, in rank order, one eighth of the rows (bias, LeakyReLU, bf16).  The K split
// depends on the layer only — never on the batch — so a 2-pair call is bit for bit two 1-pair calls.
//
// Operands: A rows are gathered from the haloed NHWC input with cp.async (one K stage of an output pixel = 128 contiguous
// bytes), B stages are copied verbatim from the pre-swizzled tcgen05 operand image ([stage][N][128 B], 16-byte granules XOR-ed
// with n & 7 — which is also conflict-free for ldmatrix), math is mma.sync.m16n8k16 bf16 with fp32 accumulation: 20-160 rows
// cannot fill a 128-row UMMA tile, and the legacy path needs no TMEM allocation or descriptor set-up on a 4 us kernel.
// The weight copies are issued BEFORE griddepcontrol.wait: they do not depend on the previous layer and overlap its tail.

#include "common.cuh"
#include "conv_bf16.h"
#include "tc_ptx.cuh"

namespace uahn {

namespace {

constexpr int SMM_THREADS = 128, SMM_CLUSTER = 8, SMM_MAXCH = 7, SMM_NSLAB = 64;

struct SmallMParams {
  const uint8_t* in;
  const uint8_t* b_image;
  const float* bias;
  uint8_t* out;
  int M, HoWo, Wo, stride, KW, cin_chunks, k_stages, n_total, act;
  long long in_pitch_n_b, in_origin_b, out_pitch_n_b, out_origin_b;
  int in_pitch_y_b, cin_b, out_pitch_y_b, cout_b;
};

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void ldmatrix_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// MT: 16-row tiles of the GEMM (M <= 16 MT).  Shared memory: SMM_MAXCH x (A stage 16 MT x 128 B + B stage 64 x 128 B); the
// fp32 partial tile [16 MT][64] re-uses the front of it after the last MMA.
template <int MT>
__global__ void __cluster_dims__(SMM_CLUSTER, 1, 1) __launch_bounds__(SMM_THREADS) conv_small_m_kernel(const __grid_constant__ SmallMParams p) {
  extern __shared__ __align__(128) uint8_t smem[];
  constexpr int ROWS = MT * 16, A_BYTES = ROWS * 128, B_BYTES = SMM_NSLAB * 128, ST_BYTES = A_BYTES + B_BYTES;
  __shared__ uint32_t rowoff[ROWS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t rank = cluster_ctarank();
  const int n0 = (blockIdx.x / SMM_CLUSTER) * SMM_NSLAB;
  const int c_lo = (int)(rank * p.k_stages) / SMM_CLUSTER, c_hi = (int)((rank + 1) * p.k_stages) / SMM_CLUSTER;
  const int nch = c_hi - c_lo;                                  // <= SMM_MAXCH (host-checked)
  const uint32_t s0 = smem_u32(smem);

  // ---- weights of this CTA's K stages: independent of the previous kernel ----
  for (int i = 0; i < nch; ++i) {
    const uint8_t* src = p.b_image + ((size_t)(c_lo + i) * p.n_total + n0) * 128;
    const uint32_t dst = s0 + i * ST_BYTES + A_BYTES;
    for (int q = tid; q < B_BYTES / 16; q += SMM_THREADS) cp_async16(dst + q * 16, src + q * 16);
  }
  cp_async_commit();
  // ---- input rows ----
  for (int r = tid; r < ROWS; r += SMM_THREADS) {
    const int m = r < p.M ? r : 0;                              // rows past M re-read row 0; their results are dropped
    const int img = m / p.HoWo, rem = m - img * p.HoWo, oy = rem / p.Wo, ox = rem - oy * p.Wo;
    rowoff[r] = (uint32_t)(img * p.in_pitch_n_b + (long long)(oy * p.stride) * p.in_pitch_y_b + (long long)(ox * p.stride) * p.cin_b);
  }
  pdl_wait();                                                   // the input comes from the previous layer
  pdl_launch_dependents();                                      // 16-32 CTAs: the next kernel's prologue overlaps this one
  __syncthreads();
  const uint8_t* in0 = p.in + p.in_origin_b;
#pragma unroll
  for (int i = 0; i < SMM_MAXCH; ++i) {
    if (i < nch) {
      const int s = c_lo + i, tap = s / p.cin_chunks, cc = s - tap * p.cin_chunks, ky = tap / p.KW, kx = tap - ky * p.KW;
      const long long toff = (long long)ky * p.in_pitch_y_b + (long long)kx * p.cin_b + cc * 128;
      const uint32_t dst = s0 + i * ST_BYTES;
      for (int q = tid; q < ROWS * 8; q += SMM_THREADS) {
        const int r = q >> 3, g = q & 7;
        cp_async16(dst + r * 128 + ((g ^ (r & 7)) << 4), in0 + rowoff[r] + toff + g * 16);
      }
    }
    cp_async_commit();                                          // always SMM_MAXCH groups: the waits below are compile-time
  }

  // ---- MMAs: warp w owns columns 16 w ... 16 w + 15 of the slab ----
  float acc[MT][2][4];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;
  const int a_row = lane & 15, a_kh = lane >> 4;                         // ldmatrix.x4 of A: rows 0-15, k halves 0 / 1
  const int b_row = warp * 16 + ((lane >> 4) << 3) + (lane & 7), b_kh = (lane >> 3) & 1;   // of B: n tile lane/16, k half
  auto stage_mma = [&](int i) {
    const uint32_t sa = s0 + i * ST_BYTES, sb = sa + A_BYTES;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t b[4];
      ldmatrix_x4(sb + b_row * 128 + (((ks * 2 + b_kh) ^ (b_row & 7)) << 4), b[0], b[1], b[2], b[3]);
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        uint32_t a[4];
        const int r = mt * 16 + a_row;
        ldmatrix_x4(sa + r * 128 + (((ks * 2 + a_kh) ^ (r & 7)) << 4), a[0], a[1], a[2], a[3]);
        mma_bf16(acc[mt][0], a, b[0], b[1]);
        mma_bf16(acc[mt][1], a, b[2], b[3]);
      }
    }
  };
#define SMM_STAGE(I)                    \
  if (I < nch) {                        \
    cp_async_wait<SMM_MAXCH - 1 - I>(); \
    __syncthreads();                    \
    stage_mma(I);                       \
  }
  SMM_STAGE(0) SMM_STAGE(1) SMM_STAGE(2) SMM_STAGE(3) SMM_STAGE(4) SMM_STAGE(5) SMM_STAGE(6)
#undef SMM_STAGE
  cp_async_wait<0>();
  __syncthreads();                                              // every warp is done with the stages: the partial tile re-uses them

  // ---- partial tile -> own shared memory; reduce one eighth of the rows over the cluster in rank order ----
  float* part = reinterpret_cast<float*>(smem);
  {
    const int g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        const int c = warp * 16 + nt * 8 + 2 * t;
        *reinterpret_cast<float2*>(part + (mt * 16 + g) * SMM_NSLAB + c) = make_float2(acc[mt][nt][0], acc[mt][nt][1]);
        *reinterpret_cast<float2*>(part + (mt * 16 + g + 8) * SMM_NSLAB + c) = make_float2(acc[mt][nt][2], acc[mt][nt][3]);
      }
  }
  cluster_sync_all();
  uint32_t remote[SMM_CLUSTER];
#pragma unroll
  for (int j = 0; j < SMM_CLUSTER; ++j) asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote[j]) : "r"(s0), "r"(j));
  const int my_rows = (p.M - (int)rank + SMM_CLUSTER - 1) / SMM_CLUSTER;       // rows rank, rank + 8, ...
  // every remote load of this thread is issued before the first sum: one DSMEM round trip per thread instead of one per item
  constexpr int ITEMS = (2 * MT * (SMM_NSLAB / 2) + SMM_THREADS - 1) / SMM_THREADS;     // ceil(rows per rank * column pairs / threads)
  float2 part2[ITEMS][SMM_CLUSTER];
#pragma unroll
  for (int it = 0; it < ITEMS; ++it) {
    const int idx = tid + it * SMM_THREADS;
    const bool on = idx < my_rows * (SMM_NSLAB / 2);
    const int m = (int)rank + SMM_CLUSTER * (idx / (SMM_NSLAB / 2)), c = (idx % (SMM_NSLAB / 2)) * 2;
#pragma unroll
    for (int j = 0; j < SMM_CLUSTER; ++j) {
      part2[it][j] = make_float2(0.f, 0.f);
      if (on)
        asm volatile("ld.shared::cluster.v2.f32 {%0, %1}, [%2];"
                     : "=f"(part2[it][j].x), "=f"(part2[it][j].y)
                     : "r"(remote[j] + (uint32_t)(m * SMM_NSLAB + c) * 4));
    }
  }
#pragma unroll
  for (int it = 0; it < ITEMS; ++it) {
    const int idx = tid + it * SMM_THREADS;
    if (idx >= my_rows * (SMM_NSLAB / 2)) break;
    const int m = (int)rank + SMM_CLUSTER * (idx / (SMM_NSLAB / 2)), c = (idx % (SMM_NSLAB / 2)) * 2;
    float v0 = 0.f, v1 = 0.f;
#pragma unroll
    for (int j = 0; j < SMM_CLUSTER; ++j) {
      v0 += part2[it][j].x;
      v1 += part2[it][j].y;
    }
    v0 += __ldg(p.bias + n0 + c);
    v1 += __ldg(p.bias + n0 + c + 1);
    if (p.act) { v0 = lrelu(v0); v1 = lrelu(v1); }
    const int img = m / p.HoWo, rem = m - img * p.HoWo, oy = rem / p.Wo, ox = rem - oy * p.Wo;
    uint8_t* o = p.out + p.out_origin_b + img * p.out_pitch_n_b + (long long)oy * p.out_pitch_y_b + (long long)ox * p.cout_b + (n0 + c) * 2;
    *reinterpret_cast<__nv_bfloat162*>(o) = __floats2bfloat162_rn(v0, v1);
  }
  cluster_sync_all();                                           // nobody leaves while a peer still reads its partial tile
}

template <int MT>
cudaError_t launch_mt(const SmallMParams& p, cudaStream_t st) {
  constexpr size_t SMEM = (size_t)SMM_MAXCH * (MT * 16 * 128 + SMM_NSLAB * 128);
  static SmemOptIn optin;   // per device (common.cuh)
  if (cudaError_t e = optin.ensure(conv_small_m_kernel<MT>, SMEM); e != cudaSuccess) return e;
  return launch_pdl(conv_small_m_kernel<MT>, dim3((p.n_total / SMM_NSLAB) * SMM_CLUSTER), dim3(SMM_THREADS), SMEM, st, p);
}

}  // namespace

// 1: this layer at this batch takes the split-K latency kernel
int conv_small_m_ok(const ConvBf16Weights& wb, const ConvGeom& g) {
  if (!wb.ready || wb.xb != 1 || g.Cin % 64 || g.Cout % SMM_NSLAB || g.KH != g.KW || wb.n_total != g.Cout) return 0;
  const int k_stages = g.KH * g.KW * (g.Cin / 64);
  if (wb.k_total != k_stages * 64 || (k_stages + SMM_CLUSTER - 1) / SMM_CLUSTER > SMM_MAXCH) return 0;
  // worth it where the tcgen05 kernel would be a handful of CTAs walking a long K loop
  return g.M <= 160 && k_stages >= 16;
}

cudaError_t launch_conv_small_m(const ConvBf16Weights& wb, const void* in, const float* bias, void* out, const ConvGeom& g,
                                cudaStream_t st) {
  SmallMParams p{};
  p.in = (const uint8_t*)in;
  p.b_image = (const uint8_t*)wb.b_image;
  p.bias = bias;
  p.out = (uint8_t*)out;
  p.M = g.M; p.HoWo = g.Ho * g.Wo; p.Wo = g.Wo; p.stride = g.stride; p.KW = g.KW;
  p.cin_chunks = g.Cin / 64;
  p.k_stages = g.KH * g.KW * p.cin_chunks;
  p.n_total = g.Cout;
  p.act = g.act;
  p.in_pitch_n_b = g.in_pitch_n * 2; p.in_origin_b = g.in_origin * 2; p.in_pitch_y_b = (int)(g.in_pitch_y * 2); p.cin_b = g.Cin * 2;
  p.out_pitch_n_b = g.out_pitch_n * 2; p.out_origin_b = g.out_origin * 2; p.out_pitch_y_b = (int)(g.out_pitch_y * 2); p.cout_b = g.Cout * 2;
  const long long n_img = (g.M + (long long)p.HoWo - 1) / p.HoWo;
  if (n_img * p.in_pitch_n_b >= (1ll << 32)) return cudaErrorInvalidValue;   // 32-bit row offsets
  if (g.M <= 32) return launch_mt<2>(p, st);
  if (g.M <= 80) return launch_mt<5>(p, st);
  if (g.M <= 160) return launch_mt<10>(p, st);
  return cudaErrorInvalidValue;
}

}  // namespace uahn
