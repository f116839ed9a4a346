// Shifted-window implicit GEMM for the large-spatial convolutions (block_4_0..3, block_3_0..2): TMA-staged A.
//
// The cp.async gather of conv_bf16.cu tops out at one 128-byte line per ~8 cycles per SM (measured: 14-15 B/clk/SM
// of A fill on every layer) and re-reads every input row KH times from L2.  Here the tile is a BW x BR patch of
// output pixel groups of ONE image, ordered row = rr*BW + w, and each input row segment is brought to shared
// memory exactly once per tile by a 4-D tiled TMA load (cp.async.bulk.tensor, SWIZZLE_128B):
//
//   tensor map dims  d0 = 64 bf16 of the K run (128 B)   stride 2 B
//                    d1 = pixel group oxb                 stride xb*stride*Cin*2 B   (windows OVERLAP in x)
//                    d2 = input row y                     stride pitch_y, traversed with elementStride = conv stride
//                    d3 = image                           stride pitch_n
//   one "plane" = box {64, BW, R, 1} for a row parity rho (y = s*t + rho) and a 64-element chunk c of the run.
//
// Kernel row ky = rho + s*a then needs patch rows t = rr + a of plane (rho, c): the A operand of that tap is the
// SAME shared-memory plane with its UMMA descriptor start advanced by a*BW*128 B — a whole number of 1024-byte
// swizzle atoms because BW is a multiple of 8 — so the KH-fold im2col amplification never leaves the SM.
// x-direction taps and the conv stride in x live in the banded ("Toeplitz") B operand, which is small enough
// to stay resident in shared memory for the lifetime of the persistent CTA.
//
// Warp roles: warp 0 = TMA producer, warp 1 = tcgen05.mma issuer, warps 2-17 = epilogue (TMEM -> bf16 -> LeakyReLU on
// the packed pair -> each thread stores its 32 contiguous output bytes; the accumulators are pre-loaded with the bias
// and re-armed by every drain).  Planes flow through a ring of n_slots shared-memory slots guarded by full/empty
// mbarriers; two TMEM accumulators overlap the epilogue of tile i with the MMAs of tile i+1.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <cudaTypedefs.h>

#include "conv_bf16.h"
#include "tc_ptx.cuh"

namespace uahn {
namespace {

constexpr int EPI_WARPS = 16;             // 4 per TMEM lane quadrant; each takes BN/4 accumulator columns
constexpr int TM_THREADS = 64 + 32 * EPI_WARPS;
// epilogue staging: [2 buffers][4 TMEM lane quadrants][32 rows][128 B of bf16 + 16 B pad]
constexpr int EPI_ROW = 144, EPI_STAGE_BYTES = 2 * 4 * 32 * EPI_ROW;
constexpr int MAX_SLOTS = 12;
constexpr int MAX_OPS = 128;              // tcgen05.mma instructions per tile (KH taps x chunks x k-steps)
constexpr int SMEM_LIMIT = 227 * 1024;

// Per-role cycle accounting (UAHN_TMA_DEBUG=1 prints it): compiled in only with -DUAHN_TMA_PROFILE=1.
#ifndef UAHN_TMA_PROFILE
#define UAHN_TMA_PROFILE 0
#endif
__device__ __forceinline__ long long prof_clock() { return UAHN_TMA_PROFILE ? clock64() : 0ll; }

struct TmaConvParams {
  const uint8_t* b_image;
  const float* bias_x;
  uint8_t* out;
  int n_img, PX, PY, BW, BR, Ho, Wox;
  int stride, KH, chunks, run_elems;
  int n_planes, n_slots, slot_bytes, b_stages;
  int plane_rows[8], plane_taps[8], plane_rho[8], plane_chunk[8];
  long long out_pitch_n_b;
  int out_pitch_y_b, out_col_step_b;
  long long out_origin_b;
  int n_total, act;
  unsigned long long magic_tiles, magic_px;   // ceil(2^40 / tiles_per_img), ceil(2^40 / PX)
  unsigned long long* dbg;   // optional [grid][8] cycle counters (UAHN_TMA_DEBUG)
};

// Compile-time layer shape: kernel rows KH, conv stride ST, 64-element chunks of the K run and the k-steps (of 16)
// in chunk 0 / chunk 1.  With these fixed, every tcgen05.mma of a tile has immediate descriptor offsets, so the
// single issuing lane spends a couple of uniform-datapath adds per MMA instead of table look-ups.
template <int BN, int KH, int ST, int CHUNKS, int KS0, int KS1>
__global__ void __launch_bounds__(TM_THREADS, 1) conv_tma_bf16_kernel(const __grid_constant__ CUtensorMap tmap,
                                                                       const __grid_constant__ TmaConvParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr int B_STAGE_BYTES = BN * 128;
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                                               // [n_slots][slot_bytes]
  uint8_t* sB = sA + (size_t)p.n_slots * p.slot_bytes;             // [b_stages][BN][128 B], resident
  float* sBias = reinterpret_cast<float*>(sB + (size_t)p.b_stages * B_STAGE_BYTES);   // [BN]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sBias + 256);
  // bars: [0,S) full, [S,2S) empty, 2S..2S+1 accumulator full, 2S+2..2S+3 accumulator empty, 2S+4 B resident
  const int S = p.n_slots;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * MAX_SLOTS + 5);
  uint8_t* sStage = reinterpret_cast<uint8_t*>(bars + 2 * MAX_SLOTS + 8) + 16 * 4;   // epilogue staging (16-byte aligned)

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + MAX_SLOTS);
  const uint32_t tfull0 = smem_u32(bars + 2 * MAX_SLOTS), tempty0 = smem_u32(bars + 2 * MAX_SLOTS + 2);
  const uint32_t bres = smem_u32(bars + 2 * MAX_SLOTS + 4);
  const int tiles_per_img = p.PX * p.PY;
  const int total_tiles = p.n_img * tiles_per_img;

  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < S; ++s) {
        mbar_init(full0 + 8 * s, 1);    // producer's expect_tx arrive; TMA completes the bytes
        mbar_init(empty0 + 8 * s, 1);   // one tcgen05.commit
      }
      for (int b = 0; b < 2; ++b) {
        mbar_init(tfull0 + 8 * b, 1);
        mbar_init(tempty0 + 8 * b, EPI_WARPS);
      }
      mbar_init(bres, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)(2 * BN))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  for (int i = tid; i < BN; i += TM_THREADS) sBias[i] = p.bias_x[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Both accumulators start out holding the bias (tcgen05.st by the epilogue warps), every MMA accumulates and each
  // epilogue drain re-arms its columns: no bias add in the epilogue.
  constexpr int COLS = BN / (EPI_WARPS / 4);            // accumulator columns per epilogue warp (16 for BN = 64)
  static_assert(COLS == 16, "epilogue is written for 16 accumulator columns per warp");
  const int q = warp & 3, cg = (warp - 2) >> 2;         // TMEM lane quadrant (hardware rule), column group
  const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(cg * COLS);
  const uint32_t stage_s = smem_u32(sStage);
  uint32_t biasu[COLS];
  if (warp >= 2) {
#pragma unroll
    for (int c = 0; c < COLS; ++c) biasu[c] = __float_as_uint(sBias[cg * COLS + c]);
    tmem_st16(t_lane, biasu);
    tmem_st16(t_lane + (uint32_t)BN, biasu);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();                 // everything above touched only shared memory, TMEM and weights
  pdl_launch_dependents();

  if (warp == 0) {
    // ===================== TMA producer =====================
    // warp-uniform loop, the TMA / barrier instructions predicated on one elected lane: coordinates and barrier
    // addresses stay in uniform registers (a single-lane loop pays an ELECT / R2UR.BROADCAST round trip per operand —
    // several hundred cycles per load, more than the 18 MMAs of a tile take)
    const bool leader = elect_one();
    if (leader) {
      tma_prefetch_desc(&tmap);
      mbar_arrive_expect_tx(bres, (uint32_t)(p.b_stages * B_STAGE_BYTES));
      for (int s = 0; s < p.b_stages; ++s)
        bulk_g2s(smem_u32(sB + s * B_STAGE_BYTES), p.b_image + (size_t)s * B_STAGE_BYTES, B_STAGE_BYTES, bres);
    }
    __syncwarp();
    int slot = 0;
    uint32_t par = 1;
    const int step_img = (int)gridDim.x / tiles_per_img, step_rem = (int)gridDim.x - step_img * tiles_per_img;
    int img = (int)blockIdx.x / tiles_per_img, rem = (int)blockIdx.x - img * tiles_per_img;
    long long w_empty = 0, t_begin = prof_clock();
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int py = rem / p.PX, px = rem - py * p.PX;
      for (int pl = 0; pl < p.n_planes; ++pl) {
        const long long t0 = prof_clock();
        mbar_wait(empty0 + 8 * slot, par);
        w_empty += prof_clock() - t0;
        if (leader) {
          mbar_arrive_expect_tx(full0 + 8 * slot, (uint32_t)(p.plane_rows[pl] * p.BW * 128));
          tma_load_4d(smem_u32(sA + (size_t)slot * p.slot_bytes), &tmap, p.plane_chunk[pl] * 64, px * p.BW,
                      p.stride * (py * p.BR) + p.plane_rho[pl], img, full0 + 8 * slot);
        }
        __syncwarp();
        if (++slot == S) { slot = 0; par ^= 1u; }
      }
      rem += step_rem; img += step_img;
      if (rem >= tiles_per_img) { rem -= tiles_per_img; ++img; }
    }
    if (p.dbg && lane == 0) { p.dbg[blockIdx.x * 8 + 0] = w_empty; p.dbg[blockIdx.x * 8 + 1] = prof_clock() - t_begin; }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = umma_idesc_bf16(128, BN);
    // descriptor bits above the address: LBO = 1, SBO = 1024 B, version 1, SWIZZLE_128B (see umma_desc_sw128)
    constexpr uint64_t DESC_HI = (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
    const int slot_bytes = p.slot_bytes;
    const uint32_t sA0 = smem_u32(sA);
    const uint32_t b16 = (smem_u32(sB) & 0x3FFFFu) >> 4;
    int it = 0, tcount = 0;
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    mbar_wait(bres, 0);
    long long w_tempty = 0, w_full = 0, t_begin = prof_clock();
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tcount) {
      const int ab = tcount & 1;
      long long t0 = prof_clock();
      mbar_wait(tempty0 + 8 * ab, ((tcount >> 1) & 1) ^ 1);
      w_tempty += prof_clock() - t0;
      tc_fence_after();
      const uint32_t d_tmem = tmem_u + (uint32_t)(ab * BN);
      const bool leader = elect_one();
#pragma unroll
      for (int pl = 0; pl < ST * CHUNKS; ++pl, ++it) {        // planes: parity-major, chunk inner
        constexpr int dummy = 0; (void)dummy;
        const int rho = pl / CHUNKS, c = pl % CHUNKS;
        const int slot = it % S;
        t0 = prof_clock();
        mbar_wait(full0 + 8 * slot, (it / S) & 1);
        w_full += prof_clock() - t0;
        tc_fence_after();
        const uint32_t a16 = ((sA0 + (uint32_t)slot * slot_bytes) & 0x3FFFFu) >> 4;
        if (leader) {
          const int taps = (KH - rho + ST - 1) / ST;
          const int ks = c == 0 ? KS0 : KS1;
#pragma unroll
          for (int a = 0; a < taps; ++a) {
#pragma unroll
            for (int kk = 0; kk < ks; ++kk) {
              // A: the plane shifted by `a` patch rows (a * 8 groups * 128 B) ; B: resident stage (ky, c)
              const uint32_t alo = a16 + (uint32_t)(a * 8 * 128 / 16 + kk * 2);
              const uint32_t blo = b16 + (uint32_t)(((rho + ST * a) * CHUNKS + c) * (BN * 128 / 16) + kk * 2);
              tc_mma_bf16(d_tmem, DESC_HI | (uint64_t)alo, DESC_HI | (uint64_t)blo, idesc, 1u);
            }
          }
          tc_commit(empty0 + 8 * slot);
          if (pl == ST * CHUNKS - 1) tc_commit(tfull0 + 8 * ab);
        }
        __syncwarp();
      }
    }
    if (p.dbg && lane == 0) {
      p.dbg[blockIdx.x * 8 + 2] = w_tempty; p.dbg[blockIdx.x * 8 + 3] = w_full; p.dbg[blockIdx.x * 8 + 4] = prof_clock() - t_begin;
    }
    tc_fence_before();
  } else {
    // ===================== epilogue (warps 2..17) =====================
    // TMEM -> registers -> (LeakyReLU on packed bf16x2) -> per-quadrant staging -> coalesced global stores.
    // TMEM lane r = q*32 + lane is pixel group (patch row r / 8, column r % 8): BW = 8, N = 64 -> 128 B per group.
    const int step_img = (int)gridDim.x / tiles_per_img, step_rem = (int)gridDim.x - step_img * tiles_per_img;
    int img = (int)blockIdx.x / tiles_per_img, rem = (int)blockIdx.x - img * tiles_per_img;
    const uint32_t mpx = (uint32_t)((65536 + p.PX - 1) / p.PX);                 // rem < 65536 / PX
    int tcount = 0;
    long long w_tfull = 0, w_tmem = 0, t_begin = prof_clock();
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tcount) {
      const int ab = tcount & 1;
      const int py = (int)(((uint32_t)rem * mpx) >> 16), px = rem - py * p.PX;
      const long long t0 = prof_clock();
      mbar_wait(tfull0 + 8 * ab, (tcount >> 1) & 1);
      const long long t1 = prof_clock();
      w_tfull += t1 - t0;
      tc_fence_after();
      uint32_t acc[COLS];
      tmem_ld16(t_lane + (uint32_t)(ab * BN), acc);
      tmem_ld_wait();
      tmem_st16(t_lane + (uint32_t)(ab * BN), biasu);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty0 + 8 * ab);       // this warp's slice is in registers and re-armed
      const long long t2 = prof_clock();
      w_tmem += t2 - t1;
      uint32_t packed[8];
#pragma unroll
      for (int e = 0; e < 8; ++e)
        packed[e] = p.act ? pack_lrelu_bf16x2(__uint_as_float(acc[2 * e]), __uint_as_float(acc[2 * e + 1]))
                          : pack_bf16x2(__uint_as_float(acc[2 * e]), __uint_as_float(acc[2 * e + 1]));
      // Stage the quadrant's 32 rows x 128 B (four warps, 32 B per lane each), then every warp writes ONE patch row of
      // the quadrant — 8 pixel groups x 128 B = 1 KB contiguous in global memory — with two fully coalesced 512-byte
      // stores.  (Storing each lane's 32 bytes directly costs 32 line requests per instruction: the kernel was bound
      // by exactly that, 1800 of 2000 cycles per tile in the store phase.)  Two buffers: the barrier of tile t+1
      // orders the copy-out of tile t before the staging writes of tile t+2.
      const uint32_t sbuf = stage_s + (uint32_t)(((tcount & 1) * 4 + q) * (32 * EPI_ROW));
      st_shared_v4(sbuf + (uint32_t)(lane * EPI_ROW + cg * 32), packed[0], packed[1], packed[2], packed[3]);
      st_shared_v4(sbuf + (uint32_t)(lane * EPI_ROW + cg * 32 + 16), packed[4], packed[5], packed[6], packed[7]);
      asm volatile("bar.sync %0, 128;" ::"r"(1 + q) : "memory");
      const int prow = 4 * q + cg, oy = py * p.BR + prow;             // this warp's patch row
      if (prow < p.BR && oy < p.Ho) {
        uint8_t* orow = p.out + (p.out_origin_b + (long long)img * p.out_pitch_n_b + (long long)oy * p.out_pitch_y_b +
                                 (long long)(px * p.BW) * p.out_col_step_b);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const int g = (lane >> 3) + 4 * k, c = lane & 7;
          const uint4 v = ld_shared_v4(sbuf + (uint32_t)((cg * 8 + g) * EPI_ROW + c * 16));
          if (px * p.BW + g < p.Wox) st_global_v4(orow + g * 128 + c * 16, v.x, v.y, v.z, v.w);
        }
      }
      rem += step_rem; img += step_img;
      if (rem >= tiles_per_img) { rem -= tiles_per_img; ++img; }
    }
    if (p.dbg && warp == 2 && lane == 0) {
      p.dbg[blockIdx.x * 8 + 5] = w_tfull; p.dbg[blockIdx.x * 8 + 6] = prof_clock() - t_begin; p.dbg[blockIdx.x * 8 + 7] = w_tmem;
    }
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * BN))
                 : "memory");
  }
}

template <int BN>
size_t tma_smem_bytes(int n_slots, int slot_bytes, int b_stages) {
  return 1024 + (size_t)n_slots * slot_bytes + (size_t)b_stages * BN * 128 + 256 * 4 + (2 * MAX_SLOTS + 8) * 8 + 16 * 4 +
         EPI_STAGE_BYTES;
}

PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

}  // namespace

int conv_tma_prepare(TmaPlan& plan, const std::vector<float>& wk, const std::vector<float>& bias, const ConvGeom& g,
                     const Tensor& in, std::vector<void*>& allocs, std::string& err) {
  plan.enabled = 0;
  if (g.KH == 1) return 0;
  const int s = g.stride;
  if (s > 2) return 0;
  // ---- choose the Toeplitz factor: N = xb*Cout must be 64 here, patch width BW = 8 groups ----
  int best_xb = 0;
  double best_cost = 1e30;
  for (int xb = 1; xb <= 32; xb *= 2) {
    if (g.Wo % xb) continue;
    if ((xb * s * g.Cin * 2) % 16) continue;
    const int n = xb * g.Cout;
    if (n != 64) continue;
    const int wox = g.Wo / xb;
    if (wox % 8) continue;
    const int run = (s * (xb - 1) + g.KW) * g.Cin;
    const int chunks = (run + 63) / 64;
    if (chunks > 4) continue;
    if ((size_t)g.KH * chunks * n * 128 > 100 * 1024) continue;
    int ksteps = 0;
    for (int c = 0; c < chunks; ++c) ksteps += std::min(4, (run - c * 64 + 15) / 16);
    const double mma = (double)g.KH * ksteps * (n / 2.0), epi = 8.0 * n;
    const double cost = std::max(mma, epi) / (128.0 * xb);   // cycles per output pixel
    if (cost < best_cost) { best_cost = cost; best_xb = xb; }
  }
  if (!best_xb) return 0;
  if (g.Ho < 16 || g.Ho * (g.Wo / best_xb) < 512) return 0;   // small images: the consecutive-row gather kernel
  const int xb = best_xb, n_total = xb * g.Cout, wox = g.Wo / xb;
  const int run = (s * (xb - 1) + g.KW) * g.Cin, chunks = (run + 63) / 64;
  {   // only the instantiated (KH, stride, chunks, k-steps) shapes
    const int k0 = std::min(4, (run + 15) / 16), k1 = chunks > 1 ? std::min(4, (run - 64 + 15) / 16) : 0;
    const int sig = g.KH * 10000 + s * 1000 + chunks * 100 + k0 * 10 + k1;
    if (sig != 71120 && sig != 52242 && sig != 52243 && sig != 32241 && sig != 32242) return 0;
  }
  plan.xb = xb; plan.BW = 8; plan.chunks = chunks; plan.run_elems = run; plan.n_total = n_total;
  int bestbr = 16, bestpy = 1 << 30;
  for (int br = 16; br >= 8; --br) {
    const int py = (g.Ho + br - 1) / br;
    if (py < bestpy) { bestpy = py; bestbr = br; }
  }
  plan.BR = bestbr; plan.PY = bestpy; plan.PX = wox / plan.BW;
  // planes: parity-major, chunk inner
  plan.n_planes = 0;
  int max_rows = 0;
  for (int rho = 0; rho < s && rho < g.KH; ++rho) {
    const int taps = (g.KH - rho + s - 1) / s;
    for (int c = 0; c < chunks; ++c) {
      const int i = plan.n_planes++;
      plan.plane_rho[i] = rho; plan.plane_chunk[i] = c; plan.plane_taps[i] = taps;
      plan.plane_rows[i] = plan.BR + taps - 1;
      max_rows = std::max(max_rows, plan.plane_rows[i]);
    }
  }
  // a tap reads 128 rows starting at a*BW even when BR*BW < 128: the slot must cover them
  plan.slot_bytes = std::max(max_rows * plan.BW, 128 + (max_rows - plan.BR) * plan.BW) * 128;
  plan.slot_bytes = (plan.slot_bytes + 1023) / 1024 * 1024;
  const int b_stages = g.KH * chunks;
  const size_t fixed = (n_total == 64 ? tma_smem_bytes<64>(0, 0, b_stages) : tma_smem_bytes<128>(0, 0, b_stages));
  int slots = (int)((SMEM_LIMIT - (int)fixed) / plan.slot_bytes);
  slots = std::min(slots, std::min(MAX_SLOTS, 3 * plan.n_planes));
  if (slots < plan.n_planes + 1 && slots < 2) return 0;
  plan.n_slots = slots;

  // ---- tensor map over the haloed NHWC input ----
  PFN_cuTensorMapEncodeTiled_v12000 encode = get_encode();
  if (!encode) { err = "cuTensorMapEncodeTiled entry point not found"; return -2; }
  const cuuint64_t gdim[4] = {(cuuint64_t)chunks * 64, (cuuint64_t)wox, (cuuint64_t)in.Hp, (cuuint64_t)in.N};
  const cuuint64_t gstr[3] = {(cuuint64_t)xb * s * g.Cin * 2, (cuuint64_t)g.in_pitch_y * 2, (cuuint64_t)g.in_pitch_n * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)plan.BW, 0, 1};
  const cuuint32_t estr[4] = {1, 1, (cuuint32_t)s, 1};
  // all planes use the same box height (the largest); shorter planes simply load one row more than they need
  box[2] = (cuuint32_t)(max_rows * s);
  for (int i = 0; i < plan.n_planes; ++i) plan.plane_rows[i] = max_rows;
  void* base = (uint8_t*)in.p + g.in_origin * 2;
  CUresult r = encode(reinterpret_cast<CUtensorMap*>(plan.tmap), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, gdim, gstr,
                      box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    if (getenv("UAHN_DEBUG")) fprintf(stderr, "[uahn] cuTensorMapEncodeTiled failed (%d): falling back to cp.async gather\n", (int)r);
    return 0;
  }

  // ---- B operand image: stage (ky, c) = [N][64 K-elements] SW128 K-major; K element e of chunk c <-> run element c*64+e
  std::vector<uint16_t> img((size_t)b_stages * n_total * 64, 0);
  for (int ky = 0; ky < g.KH; ++ky)
    for (int qel = 0; qel < chunks * 64; ++qel) {
      const int xi = qel / g.Cin, c = qel % g.Cin;
      const int st = ky * chunks + qel / 64, kk = qel % 64;
      for (int xo = 0; xo < xb; ++xo) {
        const int kx = xi - xo * s;
        if (kx < 0 || kx >= g.KW) continue;
        for (int co = 0; co < g.Cout; ++co) {
          const int n = xo * g.Cout + co;
          const float w = wk[(size_t)((ky * g.KW + kx) * g.Cin + c) * g.Cout + co];
          const size_t byte = ((size_t)st * n_total + n) * 128 + (size_t)((((kk >> 3) ^ (n & 7)) << 4) + (kk & 7) * 2);
          img[byte / 2] = f32_to_bf16_host(w);
        }
      }
    }
  void* d = nullptr;
  if (cudaMalloc(&d, img.size() * 2) != cudaSuccess) { err = "cudaMalloc(B image)"; return -2; }
  allocs.push_back(d);
  if (cudaMemcpy(d, img.data(), img.size() * 2, cudaMemcpyHostToDevice) != cudaSuccess) { err = "memcpy(B image)"; return -2; }
  std::vector<float> bx((size_t)n_total);
  for (int xo = 0; xo < xb; ++xo)
    for (int co = 0; co < g.Cout; ++co) bx[(size_t)xo * g.Cout + co] = bias[co];
  void* db = nullptr;
  if (cudaMalloc(&db, bx.size() * 4) != cudaSuccess) { err = "cudaMalloc(bias)"; return -2; }
  allocs.push_back(db);
  if (cudaMemcpy(db, bx.data(), bx.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess) { err = "memcpy(bias)"; return -2; }
  plan.b_image = d;
  plan.bias_x = (float*)db;
  plan.enabled = 1;
  if (getenv("UAHN_DEBUG"))
    fprintf(stderr, "[uahn] TMA plan: Cin=%d Cout=%d k=%d s=%d out=%dx%d  xb=%d N=%d patch=%dx%d (PX=%d PY=%d) chunks=%d planes=%d slots=%d x %d B\n",
            g.Cin, g.Cout, g.KH, s, g.Ho, g.Wo, xb, n_total, plan.BW, plan.BR, plan.PX, plan.PY, chunks, plan.n_planes,
            plan.n_slots, plan.slot_bytes);
  return 0;
}

cudaError_t launch_conv_tma(const TmaPlan& plan, const float* bias, void* out, const ConvGeom& g, int num_sms,
                            cudaStream_t st) {
  (void)bias;
  TmaConvParams p{};
  p.b_image = (const uint8_t*)plan.b_image;
  p.bias_x = plan.bias_x;
  p.out = (uint8_t*)out;
  p.n_img = g.M / (g.Ho * g.Wo);
  p.PX = plan.PX; p.PY = plan.PY; p.BW = plan.BW; p.BR = plan.BR;
  p.Ho = g.Ho; p.Wox = g.Wo / plan.xb;
  p.stride = g.stride; p.KH = g.KH; p.chunks = plan.chunks; p.run_elems = plan.run_elems;
  p.n_planes = plan.n_planes; p.n_slots = plan.n_slots; p.slot_bytes = plan.slot_bytes;
  p.b_stages = g.KH * plan.chunks;
  for (int i = 0; i < 8; ++i) {
    p.plane_rows[i] = plan.plane_rows[i]; p.plane_taps[i] = plan.plane_taps[i];
    p.plane_rho[i] = plan.plane_rho[i]; p.plane_chunk[i] = plan.plane_chunk[i];
  }
  p.out_pitch_n_b = g.out_pitch_n * 2;
  p.out_pitch_y_b = (int)(g.out_pitch_y * 2);
  p.out_col_step_b = plan.xb * g.Cout * 2;
  p.out_origin_b = g.out_origin * 2;
  p.n_total = plan.n_total;
  p.act = g.act;
  const int tiles = p.n_img * p.PX * p.PY;
  const int grid = std::min(tiles, num_sms);
  p.magic_tiles = ((1ull << 40) + p.PX * p.PY - 1) / (p.PX * p.PY);
  p.magic_px = ((1ull << 40) + p.PX - 1) / p.PX;
  static unsigned long long* d_dbg = nullptr;
  const bool debug = UAHN_TMA_PROFILE && getenv("UAHN_TMA_DEBUG") != nullptr;
  if (debug && !d_dbg) cudaMalloc(&d_dbg, 2 * 8 * 8 * 1024);
  p.dbg = debug ? d_dbg : nullptr;
  if (debug) cudaMemsetAsync(d_dbg, 0, 2 * 8 * 8 * 1024, st);
  const CUtensorMap* tm = reinterpret_cast<const CUtensorMap*>(plan.tmap);
  const int ks0 = std::min(4, (plan.run_elems + 15) / 16);
  const int ks1 = plan.chunks > 1 ? std::min(4, (plan.run_elems - 64 + 15) / 16) : 0;
  const size_t smem = tma_smem_bytes<64>(p.n_slots, p.slot_bytes, p.b_stages);
  cudaError_t lerr = cudaErrorInvalidConfiguration;
#define UAHN_TMA_CASE(KH_, ST_, CH_, K0_, K1_)                                                                     \
  if (g.KH == KH_ && g.stride == ST_ && plan.chunks == CH_ && ks0 == K0_ && ks1 == K1_) {                          \
    auto kern = conv_tma_bf16_kernel<64, KH_, ST_, CH_, K0_, K1_>;                                                 \
    static SmemOptIn optin;                                                                                         \
    if (cudaError_t e = optin.ensure(kern, smem); e != cudaSuccess) return e;                                       \
    lerr = launch_pdl(kern, dim3(grid), dim3(TM_THREADS), smem, st, *tm, p);                                        \
  }
  UAHN_TMA_CASE(7, 1, 1, 2, 0)   // block_4_0 / block_3_0 : 7x7 s1, Cin 2
  UAHN_TMA_CASE(5, 2, 2, 4, 2)   // block_4_1            : 5x5 s2, Cin 8  (run 88)
  UAHN_TMA_CASE(5, 2, 2, 4, 3)   // block_3_1            : 5x5 s2, Cin 16 (run 112)
  UAHN_TMA_CASE(3, 2, 2, 4, 1)   // block_4_2            : 3x3 s2, Cin 16 (run 80)
  UAHN_TMA_CASE(3, 2, 2, 4, 2)   // block_4_3 / block_3_2: 3x3 s2, Cin 32 (run 96)
#undef UAHN_TMA_CASE
  if (lerr != cudaSuccess) return lerr;
  if (debug) {
    std::vector<unsigned long long> h(8 * grid);
    cudaStreamSynchronize(st);
    cudaMemcpy(h.data(), d_dbg, h.size() * 8, cudaMemcpyDeviceToHost);
    double a[8] = {0};
    for (int i = 0; i < grid; ++i) for (int j = 0; j < 8; ++j) a[j] += (double)h[i * 8 + j] / grid;
    fprintf(stderr, "[uahn-tma] Cin=%d Cout=%d out=%dx%d tiles/CTA=%.1f planes=%d | producer: wait_empty %.0f of %.0f | mma: wait_tempty %.0f wait_full %.0f of %.0f | epi(w2): wait_tfull %.0f tmem ld/st+arrive %.0f of %.0f  (cycles, mean over CTAs)\n",
            g.Cin, g.Cout, g.Ho, g.Wo, (double)tiles / grid, p.n_planes, a[0], a[1], a[2], a[3], a[4], a[5], a[7], a[6]);
  }
  return cudaSuccess;
}

}  // namespace uahn
