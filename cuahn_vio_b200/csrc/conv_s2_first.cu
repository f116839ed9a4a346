// block_2_1: conv 7x7 stride 2 (2 -> 64) + LeakyReLU on the 4x-pooled 2-channel block input, as a TMA-staged tcgen05
// kernel.  (The cp.async gather of conv_bf16.cu spends 2688 LDGSTS per 128-row tile on this layer — 4-byte pixels, 16-byte
// granules — and was bound by exactly that: 71 us at 1024 pairs with the tensor pipe 16 % busy.)
//
// Same operand trick as conv 1 of the fused fronts (conv_fused_front.cu): one 4-D TMA box {32 el, 8 groups, 38 rows} of
// the input with overlapping x windows (group = 2 output pixels = a window start every 4 input pixels = 16 B; 9 pixels x 2
// channels = 18 of the 32 elements are used), 64-byte rows, SWIZZLE_64B.  GEMM row (y, g) = output row y, group g; the conv
// stride in y lives in the A descriptor — its 8-row atoms are TWO image rows apart (SBO = 1024 B) — and tap ky is the same
// plane shifted by ky rows, so A comes straight from the box.  The stride in x and the 7 taps in x live in the banded B
// operand: N = 2 pixels x 64 channels = 128, K = 7 taps x 32; two taps share one 128-byte B row.  14 MMAs of N = 128 per
// 16 x 8 tile of groups.
//
// Warp roles: warp 0 TMA producer (input double-buffered), warp 1 MMA issuer (accumulator double-buffered in TMEM, pre-loaded
// with the bias), warps 2..17 epilogue: TMEM -> bf16 -> LeakyReLU on the packed pair -> per-quadrant staging in shared
// memory -> every warp writes one patch row of its quadrant (8 groups x 256 B = 2 KB contiguous) with coalesced 512-byte
// stores.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include <cudaTypedefs.h>

#include "conv_bf16.h"
#include "tc_ptx.cuh"

namespace uahn {
namespace {

constexpr int S2_EPI_WARPS = 16;
constexpr int S2_THREADS = 64 + 32 * S2_EPI_WARPS;
constexpr int S2_IN_ROWS = 38;                       // 2 * 15 + 7 input rows of a 16-row output tile (+1)
constexpr int S2_IN_ROW_BYTES = 8 * 64;              // 8 groups x 64 B
constexpr int S2_IN_BYTES = S2_IN_ROWS * S2_IN_ROW_BYTES;   // 19 456
constexpr int S2_B_STAGES = 4, S2_B_STAGE = 128 * 128;      // 7 taps in pairs; N = 128 rows x 128 B
constexpr int S2_EPI_ROW = 256 + 16;                 // staged row: 128 bf16 + pad
constexpr int S2_EPI_BYTES = 2 * 4 * 32 * S2_EPI_ROW;       // 2 buffers x 4 quadrants x 32 rows
constexpr int S2_NBUF = 4;                           // input boxes in flight: one box (304 rows of 64 B) takes the TMA unit
                                                     // about as long as two tiles of MMAs, so the producer runs three tiles ahead
constexpr int S2_SMEM = 1024 + S2_NBUF * S2_IN_BYTES + S2_B_STAGES * S2_B_STAGE + S2_EPI_BYTES + 128 * 4 + 16 * 8 + 16;

struct S2Params {
  const uint8_t* b_image;
  const float* bias_x;      // [128]: bias[n % 64]
  uint8_t* out;
  int n_img, TX, TY, Ho, Wog;      // Wog: output groups (of 2 pixels) per row
  long long out_pitch_n_b;
  int out_pitch_y_b;
  long long out_origin_b;
  unsigned long long magic_tiles, magic_tx;
};

__global__ void __launch_bounds__(S2_THREADS, 1) conv_s2_first_kernel(const __grid_constant__ CUtensorMap tmap,
                                                                       const __grid_constant__ S2Params p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sIn = smem;                                             // [S2_NBUF][S2_IN_BYTES]
  uint8_t* sB = sIn + S2_NBUF * S2_IN_BYTES;                             // resident B: [4][128][128 B]
  uint8_t* sStage = sB + S2_B_STAGES * S2_B_STAGE;                 // epilogue staging
  float* sBias = reinterpret_cast<float*>(sStage + S2_EPI_BYTES);  // [128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sBias + 128);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  // bars: 0-3 in_full, 4-7 in_empty, 8-9 d_full, 10-11 d_empty, 12 b resident
  constexpr int B_IN_FULL = 0, B_IN_EMPTY = S2_NBUF, B_D_FULL = 2 * S2_NBUF, B_D_EMPTY = 2 * S2_NBUF + 2, B_RES = 2 * S2_NBUF + 4;
  constexpr uint32_t TMEM_COLS = 256;                              // 2 accumulators x 128 columns

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tiles_per_img = p.TX * p.TY;
  const int total_tiles = p.n_img * tiles_per_img;
  const int my_tiles = (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < S2_NBUF; ++i) { mbar_init(BAR(B_IN_FULL + i), 1); mbar_init(BAR(B_IN_EMPTY + i), 1); }
      for (int i = 0; i < 2; ++i) { mbar_init(BAR(B_D_FULL + i), 1); mbar_init(BAR(B_D_EMPTY + i), S2_EPI_WARPS); }
      mbar_init(BAR(B_RES), 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  for (int i = tid; i < 128; i += S2_THREADS) sBias[i] = p.bias_x[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int q = warp & 3, cg = (warp - 2) >> 2;                    // TMEM lane quadrant (hardware rule), 32-column group
  const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(cg * 32);
  uint32_t biasu[32];
  if (warp >= 2) {
#pragma unroll
    for (int c = 0; c < 32; ++c) biasu[c] = __float_as_uint(sBias[cg * 32 + c]);
#pragma unroll
    for (int ab = 0; ab < 2; ++ab) { tmem_st16(t_lane + (uint32_t)(ab * 128), biasu); tmem_st16(t_lane + (uint32_t)(ab * 128 + 16), biasu + 16); }
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();                 // everything above touched only shared memory, TMEM and weights
  pdl_launch_dependents();

  if (warp == 0) {
    // ===================== TMA producer (warp-uniform loop, one elected lane issues) =====================
    const bool leader = elect_one();
    if (leader) {
      tma_prefetch_desc(&tmap);
      mbar_arrive_expect_tx(BAR(B_RES), (uint32_t)(S2_B_STAGES * S2_B_STAGE));
      for (int s = 0; s < S2_B_STAGES; ++s)
        bulk_g2s(smem_u32(sB + s * S2_B_STAGE), p.b_image + (size_t)s * S2_B_STAGE, S2_B_STAGE, BAR(B_RES));
    }
    __syncwarp();
    for (int k = 0; k < my_tiles; ++k) {
      const int tile = blockIdx.x + k * gridDim.x;
      const int img = fast_div(tile, p.magic_tiles), rem = tile - img * tiles_per_img;
      const int ty = fast_div(rem, p.magic_tx), tx = rem - ty * p.TX;
      const int ib = k % S2_NBUF;
      mbar_wait(BAR(B_IN_EMPTY + ib), ((k / S2_NBUF) & 1) ^ 1);
      if (leader) {
        mbar_arrive_expect_tx(BAR(B_IN_FULL + ib), S2_IN_BYTES);
        tma_load_4d(smem_u32(sIn + ib * S2_IN_BYTES), &tmap, 0, 8 * tx, 32 * ty, img, BAR(B_IN_FULL + ib));
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = umma_idesc_bf16(128, 128);
    // A: K-major SWIZZLE_64B (layout 4), 8-row atoms (one image row of the plane: 512 B) two image rows apart
    constexpr uint64_t DESC_A = (1ull << 16) | (1ull << 46) | (4ull << 61) | ((uint64_t)((2 * S2_IN_ROW_BYTES) >> 4) << 32);
    constexpr uint64_t DESC_B = (1ull << 16) | (1ull << 46) | (2ull << 61) | ((uint64_t)(1024 >> 4) << 32);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t in16 = (smem_u32(sIn) & 0x3FFFFu) >> 4, b16 = (smem_u32(sB) & 0x3FFFFu) >> 4;
    const bool leader = elect_one();
    mbar_wait(BAR(B_RES), 0);
    for (int k = 0; k < my_tiles; ++k) {
      const int ib = k % S2_NBUF, buf = k & 1;                 // input buffer, accumulator
      mbar_wait(BAR(B_IN_FULL + ib), (k / S2_NBUF) & 1);
      mbar_wait(BAR(B_D_EMPTY + buf), ((k >> 1) & 1) ^ 1);
      tc_fence_after();
      if (leader) {
#pragma unroll
        for (int ky = 0; ky < 7; ++ky)
#pragma unroll
          for (int kk = 0; kk < 2; ++kk) {
            const uint32_t alo = in16 + (uint32_t)(ib * (S2_IN_BYTES / 16) + ky * (S2_IN_ROW_BYTES / 16) + kk * 2);
            const uint32_t blo = b16 + (uint32_t)((ky >> 1) * (S2_B_STAGE / 16) + (ky & 1) * 4 + kk * 2);
            tc_mma_bf16(tmem_u + (uint32_t)(buf * 128), DESC_A | (uint64_t)alo, DESC_B | (uint64_t)blo, idesc, 1u);
          }
        tc_commit(BAR(B_D_FULL + buf));
        tc_commit(BAR(B_IN_EMPTY + ib));
      }
      __syncwarp();
    }
    tc_fence_before();
  } else {
    // ===================== epilogue (warps 2..17) =====================
    const int step_img = (int)gridDim.x / tiles_per_img, step_rem = (int)gridDim.x - step_img * tiles_per_img;
    int img = (int)blockIdx.x / tiles_per_img, rem = (int)blockIdx.x - img * tiles_per_img;
    const uint32_t mtx = (uint32_t)((65536 + p.TX - 1) / p.TX);
    const uint32_t stage_s = smem_u32(sStage);
    for (int k = 0; k < my_tiles; ++k) {
      const int ty = (int)(((uint32_t)rem * mtx) >> 16), tx = rem - ty * p.TX;
      const int ab = k & 1;
      mbar_wait(BAR(B_D_FULL + ab), (k >> 1) & 1);
      tc_fence_after();
      uint32_t acc[32];
      tmem_ld32(t_lane + (uint32_t)(ab * 128), acc);
      tmem_ld_wait();
      tmem_st16(t_lane + (uint32_t)(ab * 128), biasu);
      tmem_st16(t_lane + (uint32_t)(ab * 128 + 16), biasu + 16);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(BAR(B_D_EMPTY + ab));      // this warp's slice is in registers and re-armed
      uint32_t packed[16];
#pragma unroll
      for (int e = 0; e < 16; ++e) packed[e] = pack_lrelu_bf16x2(__uint_as_float(acc[2 * e]), __uint_as_float(acc[2 * e + 1]));
      // stage the quadrant's 32 rows x 256 B (four warps, 64 B per lane each); then every warp writes ONE patch row of the
      // quadrant — 8 groups x 256 B = 2 KB contiguous in global memory — with four coalesced 512-byte stores
      const uint32_t sbuf = stage_s + (uint32_t)(((k & 1) * 4 + q) * (32 * S2_EPI_ROW));
#pragma unroll
      for (int c = 0; c < 4; ++c)
        st_shared_v4(sbuf + (uint32_t)(lane * S2_EPI_ROW + cg * 64 + c * 16), packed[4 * c], packed[4 * c + 1], packed[4 * c + 2],
                     packed[4 * c + 3]);
      asm volatile("bar.sync %0, 128;" ::"r"(1 + q) : "memory");
      const int prow = 4 * q + cg, oy = 16 * ty + prow;               // this warp's patch row
      if (oy < p.Ho) {
        uint8_t* orow = p.out + (p.out_origin_b + (long long)img * p.out_pitch_n_b + (long long)oy * p.out_pitch_y_b +
                                 (long long)(8 * tx) * 256);
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int g = (lane >> 4) + 2 * it, c = lane & 15;          // group of the patch row, 16-byte chunk of its 256 B
          const uint4 v = ld_shared_v4(sbuf + (uint32_t)((cg * 8 + g) * S2_EPI_ROW + c * 16));
          if (8 * tx + g < p.Wog) st_global_v4(orow + g * 256 + c * 16, v.x, v.y, v.z, v.w);
        }
      }
      rem += step_rem; img += step_img;
      if (rem >= tiles_per_img) { rem -= tiles_per_img; ++img; }
    }
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

PFN_cuTensorMapEncodeTiled_v12000 get_encode_s2() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
  }
  return fn;
}

}  // namespace

// g: the 7x7 s2 conv with Cin 2, Cout 64; x: its haloed (pad 3) 2-channel input.  Returns 0 (plan.enabled says whether
// the layer qualifies) or < 0 on a CUDA error.
int conv_s2first_prepare(S2Plan& plan, const std::vector<float>& wk, const std::vector<float>& bias, const ConvGeom& g,
                         const Tensor& x, std::vector<void*>& allocs, std::string& err) {
  plan.enabled = 0;
  if (!(g.KH == 7 && g.KW == 7 && g.stride == 2 && g.Cin == 2 && g.Cout == 64)) return 0;
  if (x.ph != 3 || x.pwl != 3 || x.C != 2 || g.Wo % 2) return 0;
  plan.Wog = g.Wo / 2;
  plan.Ho = g.Ho;
  plan.TX = (plan.Wog + 7) / 8;
  plan.TY = (g.Ho + 15) / 16;
  // the last tile's box may start inside the image and run past it: rows / groups beyond the tensor are zero-filled by TMA
  PFN_cuTensorMapEncodeTiled_v12000 encode = get_encode_s2();
  if (!encode) { err = "cuTensorMapEncodeTiled entry point not found"; return -2; }
  // dims: {32-element window, group (window start every 4 input pixels = 16 B), padded input row, image}
  const int groups_total = (x.Wp * 2 - 32) / 8 + 1;      // windows that fit in a padded row
  const cuuint64_t gdim[4] = {32, (cuuint64_t)std::max(groups_total, 1), (cuuint64_t)x.Hp, (cuuint64_t)x.N};
  const cuuint64_t gstr[3] = {16, (cuuint64_t)x.pitch_y() * 2, (cuuint64_t)x.pitch_n * 2};
  const cuuint32_t box[4] = {32, 8, S2_IN_ROWS, 1}, estr[4] = {1, 1, 1, 1};
  if (encode(reinterpret_cast<CUtensorMap*>(plan.tmap), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, x.p, gdim, gstr, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return 0;
  // B: taps ky in pairs per 128-byte row; element (n = i*64 + co, k = (ky&1)*32 + xi*2 + c) of stage ky>>1 =
  //    W[co][c][ky][kx = xi - 2i]   (i = 0, 1: the group's two output pixels; xi = 0..8: the window's input pixels)
  std::vector<uint16_t> b((size_t)S2_B_STAGES * 128 * 64, 0);
  for (int ky = 0; ky < 7; ++ky)
    for (int xi = 0; xi < 9; ++xi)
      for (int c = 0; c < 2; ++c)
        for (int i = 0; i < 2; ++i) {
          const int kx = xi - 2 * i;
          if (kx < 0 || kx >= 7) continue;
          for (int co = 0; co < 64; ++co) {
            const float w = wk[(size_t)((ky * 7 + kx) * 2 + c) * 64 + co];
            const int n = i * 64 + co, kk = (ky & 1) * 32 + xi * 2 + c;
            const size_t byte = ((size_t)(ky >> 1) * 128 + n) * 128 + (size_t)((((kk >> 3) ^ (n & 7)) << 4) + (kk & 7) * 2);
            b[byte / 2] = f32_to_bf16_host(w);
          }
        }
  std::vector<float> bx(128);
  for (int n = 0; n < 128; ++n) bx[n] = bias[n % 64];
  void *db = nullptr, *dbias = nullptr;
  if (cudaMalloc(&db, b.size() * 2) != cudaSuccess) { err = "cudaMalloc(B image)"; return -2; }
  allocs.push_back(db);
  if (cudaMalloc(&dbias, 512) != cudaSuccess) { err = "cudaMalloc(bias)"; return -2; }
  allocs.push_back(dbias);
  if (cudaMemcpy(db, b.data(), b.size() * 2, cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(dbias, bx.data(), 512, cudaMemcpyHostToDevice) != cudaSuccess) { err = "memcpy(s2 first operands)"; return -2; }
  plan.b_image = db;
  plan.bias_x = (float*)dbias;
  plan.enabled = 1;
  if (getenv("UAHN_DEBUG"))
    fprintf(stderr, "[uahn] s2-first plan: 7x7 s2 2->64 out=%dx%d tiles %dx%d per image, smem %d B\n", g.Ho, g.Wo, plan.TX, plan.TY, S2_SMEM);
  return 0;
}

cudaError_t launch_conv_s2first(const S2Plan& plan, void* out, const ConvGeom& g, int num_sms, cudaStream_t st) {
  S2Params p{};
  p.b_image = (const uint8_t*)plan.b_image;
  p.bias_x = plan.bias_x;
  p.out = (uint8_t*)out;
  p.n_img = g.M / (g.Ho * g.Wo);
  p.TX = plan.TX; p.TY = plan.TY; p.Ho = plan.Ho; p.Wog = plan.Wog;
  p.out_pitch_n_b = g.out_pitch_n * 2;
  p.out_pitch_y_b = (int)(g.out_pitch_y * 2);
  p.out_origin_b = g.out_origin * 2;
  p.magic_tiles = ((1ull << 40) + p.TX * p.TY - 1) / (p.TX * p.TY);
  p.magic_tx = ((1ull << 40) + p.TX - 1) / p.TX;
  const int tiles = p.n_img * p.TX * p.TY;
  static SmemOptIn optin;   // per device (common.cuh)
  if (cudaError_t e = optin.ensure(conv_s2_first_kernel, S2_SMEM); e != cudaSuccess) return e;
  return launch_pdl(conv_s2_first_kernel, dim3(std::min(tiles, num_sms)), dim3(S2_THREADS), S2_SMEM, st,
                    *reinterpret_cast<const CUtensorMap*>(plan.tmap), p);
}

}  // namespace uahn
