// bf16 implicit-GEMM convolution on the sm_100a tensor cores (tcgen05.mma, accumulators in TMEM).
//
//   D[m][n] = sum_k A[m][k] * B[n][k]      M = output pixel groups, N = XB * Cout, K = KH * run
//
// * A (activations) is never materialised: zero-haloed NHWC makes the im2col row of an output pixel a set of
//   KH contiguous byte runs (one per kernel row), so the producer warps gather 16-byte granules with
//   cp.async (zero-fill for tail rows) straight into the 128B-swizzled K-major shared-memory layout the
//   UMMA descriptor expects.
// * "Toeplitz" expansion along x: one GEMM row can cover XB consecutive output pixels; its K run is the union
//   of their receptive fields and B holds the correspondingly shifted (banded) filter copies.  This is what
//   lets the 2-channel 7x7 first layers (Cin*2 B = 4 B per pixel, far below a 16 B granule) and the thin
//   Cout = 8/16/32 layers fill a 128 x N tensor-core tile: N = XB*Cout.
// * B (weights) is prepared once on the host as the exact shared-memory image of every K stage, so a stage
//   is one cp.async.bulk (TMA bulk copy, UBLKCP) completing on the stage's mbarrier.
// * Warp roles: warps 0-3 produce A — cp.async gather; or (AM_IM2COL) warp 0 issues one im2col-mode TMA load per stage
//   and warp 1 the B stage; or (AM_MC) each warp builds every 4th stage of the MC-dropout expansion of the block-4
//   feature on the fly.  Warp 4 issues tcgen05.mma from one elected lane, warp 5 streams B (gather / MC modes), warps
//   6-9 run the epilogue (tcgen05.ld -> bias -> bf16 -> LeakyReLU -> 64-column staging -> coalesced global).
//   Full/empty mbarriers per stage; tcgen05.commit releases a stage when the MMAs that read it retire.
// * PAIR: clusters of two CTAs share every UMMA (cta_group::2, M = 256) and split each B stage between them.
// * All TMA / bulk-copy issue loops are warp-uniform with the copy predicated on an elected lane (a single-lane loop
//   costs ~500 cycles per stage in ELECT / R2UR.BROADCAST round trips).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <cstring>

#include <cudaTypedefs.h>

#include "conv_bf16.h"
#include "tc_ptx.cuh"

namespace uahn {
namespace {

constexpr int BM = 128;                 // UMMA M
constexpr int A_STAGE_BYTES = BM * 128; // 128 rows x 64 bf16 (one 128 B swizzle row each)
constexpr int IG_THREADS = 320;         // warps 0-3 gather A, 4 MMA, 5 B loader, 6-9 epilogue
constexpr int SMEM_LIMIT = 227 * 1024;

struct IgemmParams {
  const uint8_t* in;        // activation base
  const uint8_t* b_image;   // [k_stages][N_total][128 B], SW128 K-major
  const float* bias_x;      // [N_total]
  uint8_t* out;
  int M_rows, rows_per_img, Wox;
  unsigned long long magic_rows, magic_wox;   // ceil(2^40 / d): exact m / d for m < 2^40 / d
  long long in_pitch_n_b;
  int in_pitch_y_b, in_row_step_b, in_col_step_b;
  long long in_origin_b;
  int run_granules, total_granules, k_stages, k_steps;
  long long out_pitch_n_b;
  int out_pitch_y_b, out_col_step_b;
  long long out_origin_b;
  int n_total, n_tiles, m_tiles;
  int act;
  const uint8_t* mc_bits;   // MC_A mode: keep bits [pair][k8][16 samples] of this head (head_kernels.cu)
  // AM_IM2COL mode
  int Ho, stride, KW, cin_chunks;
  unsigned long long* dbg;  // optional [grid][16] cycle counters (UAHN_IG_PROFILE)
};
constexpr int AM_GATHER = 0, AM_MC = 1, AM_IM2COL = 2;
// the MC-dropout producer gets four more warps (10-13): two warps share a stage, four stages are under construction
constexpr int ig_threads(int am) { return am == AM_MC ? IG_THREADS + 128 : IG_THREADS; }

// -DUAHN_IG_PROFILE=1 + UAHN_IG_DEBUG=1: per-role cycle counters of the im2col-mode kernels (printed per launch)
#ifndef UAHN_IG_PROFILE
#define UAHN_IG_PROFILE 0
#endif
__device__ __forceinline__ long long ig_clock() { return UAHN_IG_PROFILE ? clock64() : 0ll; }

template <int BN>
constexpr int tmem_cols() { return 2 * BN < 32 ? 32 : 2 * BN; }   // two accumulator buffers
// epilogue staging: the accumulator is drained in chunks of EPI_CHUNK columns, so the staging buffer is 18 KB for every
// BN and the shared memory it used to take (67 KB at BN = 256) goes to a deeper A/B ring — the cp.async A fill is
// latency-bound, its throughput is (stages in flight) x 16 KB / L2 latency
template <int BN>
constexpr int epi_chunk() { return BN < 64 ? BN : 64; }
template <int BN>
constexpr int stage_row_bytes() { return epi_chunk<BN>() * 2 + 16; }   // staging row (+16 B: conflict-free)

// Persistent, warp-specialised implicit GEMM.  B_RES: the whole B operand (k_stages x BN x 128 B) stays in
// shared memory for the lifetime of the CTA (shallow-K layers); otherwise B streams through the stage ring.
// MC_A: the A operand is the MC-dropout expansion of the block-4 feature, built on the fly (model_to_trace.py:222-224,
// 272-273): GEMM row (pair, sample) = keep-mask(pair, sample) * feature(pair) / 0.95.  The producer reads each 16-byte
// feature granule once per pair, scales it, and writes 16 masked copies straight into the swizzled stage; the masked
// features (327 KB per pair and head) never exist in HBM.
// AM_IM2COL: the A stage of (filter tap, 64-channel chunk) is ONE im2col-mode TMA load of 128 consecutive output
// positions x 64 channels, written by the TMA unit straight into the 128B-swizzled stage (layers with Cin % 64 == 0:
// a K stage is exactly one tap and channel chunk).  One elected thread issues it together with the stage's B copy.
// PAIR: launched as clusters of two CTAs that share every UMMA (tcgen05.mma.cta_group::2, M = 256).  The two CTAs work
// on consecutive M tiles of the same N tile; each keeps its own A ring, accumulators and epilogue but holds only HALF of
// each B stage (BN/2 rows, loaded through a tiled tensor map over the pre-swizzled B image), so the B bytes an SM pulls
// from L2 per tile halve — the deep layers are bound by exactly that ingest (64 B/clk per SM).  All loads of a stage
// complete on the leader's full barrier; the leader's tcgen05.commit multicasts to the empty / accumulator-full
// barriers of both CTAs; the peer's epilogue warps release the accumulator on the leader's barrier.
template <int BN, int STAGES, bool B_RES, int AM = AM_GATHER, bool PAIR = false>
__global__ void __launch_bounds__(ig_threads(AM), 1) conv_igemm_bf16_kernel(const __grid_constant__ IgemmParams p,
                                                                         const __grid_constant__ CUtensorMap amap,
                                                                         const __grid_constant__ CUtensorMap bmap) {
  static_assert(!PAIR || (AM != AM_GATHER && !B_RES), "CTA pairs: im2col or MC producer, streamed B");
  constexpr bool MC_A = AM == AM_MC;
  constexpr int NCTA = PAIR ? 2 : 1;
  const long long k_entry = ig_clock();
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr int B_STAGE_BYTES = BN * 128 / NCTA;     // bytes of one B stage in THIS CTA
  constexpr int SROW = stage_row_bytes<BN>();
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * A_STAGE_BYTES;
  const int b_slots = B_RES ? p.k_stages : STAGES;
  uint8_t* sOut = sB + (size_t)b_slots * B_STAGE_BYTES;               // [4 warps][32 rows][SROW]
  float* sBias = reinterpret_cast<float*>(sOut + 128 * SROW);          // [n_total]
  long long* sRowOff = reinterpret_cast<long long*>(sBias + 256);      // [128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sRowOff + 128);
  // bars: [0,S) full, [S,2S) empty, 2S..2S+1 accumulator full, 2S+2..2S+3 accumulator empty, 2S+4 B resident
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 5);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + STAGES);
  const uint32_t tfull0 = smem_u32(bars + 2 * STAGES), tempty0 = smem_u32(bars + 2 * STAGES + 2);
  const uint32_t bres = smem_u32(bars + 2 * STAGES + 4);
  // work unit: one N tile of NCTA consecutive M tiles (one per CTA of the cluster)
  const int total_tiles = ((p.m_tiles + NCTA - 1) / NCTA) * p.n_tiles;
  const uint32_t crank = PAIR ? cluster_ctarank() : 0u;
  const bool cta_leader = crank == 0;
  const int cid = (int)blockIdx.x / NCTA, ncl = (int)gridDim.x / NCTA;
  auto tile_m0 = [&](int tile) { return ((tile / p.n_tiles) * NCTA + (int)crank) * BM; };

  if (warp == 4) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) {
        // im2col: one arrive.expect_tx for A and B together; MC: the stage's producer warp (of each CTA) + the B
        // loader's expect_tx; gather: 128 producer threads (+ the B loader)
        mbar_init(full0 + 8 * s, AM == AM_IM2COL ? 1 : MC_A ? 2 * NCTA + 1 : (B_RES ? 128 : 129));
        mbar_init(empty0 + 8 * s, 1);                  // one tcgen05.commit
      }
      for (int b = 0; b < 2; ++b) {
        mbar_init(tfull0 + 8 * b, 1);                  // tcgen05.commit after the tile's last MMA
        mbar_init(tempty0 + 8 * b, 4 * NCTA);          // one elected lane per epilogue warp (of both CTAs)
      }
      mbar_init(bres, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                   "r"((uint32_t)tmem_cols<BN>())
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                   "r"((uint32_t)tmem_cols<BN>())
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  for (int i = tid; i < p.n_total; i += ig_threads(AM)) sBias[i] = p.bias_x[i];
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();   // the peer's barriers are initialised before anything arrives on them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                 // everything above touched only shared memory, TMEM and weights
  pdl_launch_dependents();    // persistent grid: all CTAs are resident, the next kernel may start its prologue
  const long long k_roles = ig_clock();

  if (AM == AM_IM2COL && warp < 4) {
    // ===================== im2col TMA producers: warp 0 issues the A tile (TMA im2col), warp 1 the B stage ============
    // Whole warps run the (warp-uniform) loops and only the TMA / barrier instructions are predicated on an elected
    // lane: operands stay in uniform registers.  (A single-lane loop pays an ELECT + R2UR round trip per operand and
    // ~500 cycles per stage, more than the MMAs of a stage take.)
    if (warp == 0) {
      if (lane == 0) tma_prefetch_desc(&amap);
      const bool leader = elect_one();
      int slot = 0;
      uint32_t par = 1;                                   // parity to wait for on the empty barrier of `slot`
      long long pw = 0;
      int it = 0;
      const long long pbeg = ig_clock();
      for (int tile = cid; tile < total_tiles; tile += ncl) {
        const int m0 = tile_m0(tile);
        const int img = fast_div(m0, p.magic_rows), rem = m0 - img * p.rows_per_img;
        const int oy = fast_div(rem, p.magic_wox), ox = rem - oy * p.Wox;
        const int w = ox * p.stride, h = oy * p.stride;
        int ky = 0, kx = 0, cc = 0;
        for (int s = 0; s < p.k_stages; ++s, ++it) {
          const long long t0 = ig_clock();
          mbar_wait(empty0 + 8 * slot, par);
          pw += ig_clock() - t0;
          if (leader) {
            if (PAIR) {
              // both CTAs' A tiles and B halves complete on the leader's barrier, which the leader arms for all four
              if (cta_leader) mbar_arrive_expect_tx(full0 + 8 * slot, (uint32_t)(2 * (A_STAGE_BYTES + B_STAGE_BYTES)));
              tma_load_im2col_4d_pair(smem_u32(sA + slot * A_STAGE_BYTES), &amap, cc * 64, w, h, img, (uint16_t)kx, (uint16_t)ky,
                                      full0 + 8 * slot);
            } else {
              mbar_arrive_expect_tx(full0 + 8 * slot, (uint32_t)(A_STAGE_BYTES + (B_RES ? 0 : B_STAGE_BYTES)));
              tma_load_im2col_4d(smem_u32(sA + slot * A_STAGE_BYTES), &amap, cc * 64, w, h, img, (uint16_t)kx, (uint16_t)ky,
                                 full0 + 8 * slot);
            }
          }
          __syncwarp();
          if (++cc == p.cin_chunks) { cc = 0; if (++kx == p.KW) { kx = 0; ++ky; } }
          if (++slot == STAGES) { slot = 0; par ^= 1u; }
        }
      }
      if (UAHN_IG_PROFILE && p.dbg && lane == 0) { p.dbg[blockIdx.x * 16 + 0] = pw; p.dbg[blockIdx.x * 16 + 1] = ig_clock() - pbeg; p.dbg[blockIdx.x * 16 + 10] = it; }
    } else if (warp == 1 && !B_RES) {
      if (PAIR && lane == 0) tma_prefetch_desc(&bmap);
      const bool leader = elect_one();
      int slot = 0;
      uint32_t par = 1;
      for (int tile = cid; tile < total_tiles; tile += ncl) {
        const int n0 = (tile % p.n_tiles) * BN;
        for (int s = 0; s < p.k_stages; ++s) {
          mbar_wait(empty0 + 8 * slot, par);
          if (leader) {
            if (PAIR)
              tma_load_2d_pair(smem_u32(sB + slot * B_STAGE_BYTES), &bmap, 0, s * p.n_total + n0 + (int)crank * (BN / 2),
                               full0 + 8 * slot);
            else
              bulk_g2s(smem_u32(sB + slot * B_STAGE_BYTES), p.b_image + ((size_t)s * p.n_total + n0) * 128, B_STAGE_BYTES,
                       full0 + 8 * slot);
          }
          __syncwarp();
          if (++slot == STAGES) { slot = 0; par ^= 1u; }
        }
      }
    }
  } else if (MC_A && (warp < 4 || warp >= 10)) {
    // ===================== masked-feature producer (MC-dropout GEMM) =====================
    // Producer warps w and w + 10 build every 4th stage (global stage counter it = w mod 4) between them, so four
    // stages are under construction at once: the per-stage chain wait(empty) -> stores -> fence.proxy.async -> arrive
    // is latency-, not issue-bound, and four warps working on the SAME stage ran it once per ~800 cycles.
    // lane -> (granule j of the stage, pair pg + 4 * hw of the tile's 8), all 16 samples: 16 stores per stage.
    const int j = lane & 7, pg = (lane >> 3) + (warp < 4 ? 0 : 4), pwarp = warp < 4 ? warp : warp - 10;
    const int my_tiles = total_tiles > cid ? (total_tiles - cid + ncl - 1) / ncl : 0;
    const int n_it = my_tiles * p.k_stages;
    long long pw = 0;
    const long long pbeg = ig_clock();
    auto src = [&](int it, int pp, const uint8_t*& f, const uint8_t*& mb) -> bool {
      const int tl = it / p.k_stages, st = it - tl * p.k_stages;
      const int pair = (tile_m0(cid + tl * ncl) >> 4) + pg;
      f = p.in + (size_t)pair * (FC_IN * 2) + (size_t)st * 128 + j * 16;
      mb = p.mc_bits + ((size_t)pair * (FC_IN / 8) + (size_t)st * 8 + j) * MC;
      return pair * MC < p.M_rows;
    };
    uint4 gq[1], mq[1];                                   // this warp's next stage, fetched one round (4 stages) ahead
#pragma unroll
    for (int pp = 0; pp < 1; ++pp) {
      gq[pp] = mq[pp] = make_uint4(0u, 0u, 0u, 0u);
      const uint8_t *f, *mb;
      if (pwarp < n_it && src(pwarp, pp, f, mb)) {
        gq[pp] = __ldg(reinterpret_cast<const uint4*>(f));
        mq[pp] = __ldg(reinterpret_cast<const uint4*>(mb));
      }
    }
    for (int it = pwarp; it < n_it; it += 4) {
      const int slot = it % STAGES;
      uint4 g[1] = {gq[0]}, mk[1] = {mq[0]};
#pragma unroll
      for (int pp = 0; pp < 1; ++pp) {
        gq[pp] = mq[pp] = make_uint4(0u, 0u, 0u, 0u);
        const uint8_t *f, *mb;
        if (it + 4 < n_it && src(it + 4, pp, f, mb)) {
          gq[pp] = __ldg(reinterpret_cast<const uint4*>(f));
          mq[pp] = __ldg(reinterpret_cast<const uint4*>(mb));
        }
      }
      // kept values are scaled by 1/0.95 in fp32 and rounded to bf16 once per pair (same rounding as mc_expand)
      uint32_t sc[1][4];
#pragma unroll
      for (int pp = 0; pp < 1; ++pp) {
        const uint32_t w[4] = {g[pp].x, g[pp].y, g[pp].z, g[pp].w};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float lo = __uint_as_float(w[c] << 16) * KEEP_SCALE, hi = __uint_as_float(w[c] & 0xFFFF0000u) * KEEP_SCALE;
          sc[pp][c] = pack_bf16x2(lo, hi);
        }
      }
      const long long t0 = ig_clock();
      mbar_wait(empty0 + 8 * slot, ((it / STAGES) & 1) ^ 1);
      pw += ig_clock() - t0;
      const uint32_t stage = smem_u32(sA + slot * A_STAGE_BYTES);
#pragma unroll
      for (int pp = 0; pp < 1; ++pp) {
        const uint32_t mw[4] = {mk[pp].x, mk[pp].y, mk[pp].z, mk[pp].w};
#pragma unroll
        for (int si = 0; si < MC; ++si) {
          const uint32_t bits = (mw[si >> 2] >> (8 * (si & 3))) & 0xFFu;
          uint32_t o[4];
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const uint32_t b2 = bits >> (2 * c);
            o[c] = sc[pp][c] & (((b2 & 1u) ? 0x0000FFFFu : 0u) | ((b2 & 2u) ? 0xFFFF0000u : 0u));
          }
          const int r = pg * MC + si;
          st_shared_v4(stage + (uint32_t)(r * 128 + ((j ^ (r & 7)) << 4)), o[0], o[1], o[2], o[3]);
        }
      }
      fence_proxy_async();                          // generic-proxy writes -> visible to the UMMA reads
      __syncwarp();
      if (lane == 0) { if (PAIR) mbar_arrive_leader(full0 + 8 * slot); else mbar_arrive(full0 + 8 * slot); }
    }
    if (UAHN_IG_PROFILE && p.dbg && tid == 0) { p.dbg[blockIdx.x * 16 + 0] = pw; p.dbg[blockIdx.x * 16 + 1] = ig_clock() - pbeg; p.dbg[blockIdx.x * 16 + 10] = n_it; }
  } else if (warp < 4) {
    // ===================== A gather: 128 threads, 8 rows x 1 granule column each per stage ==============
    const int j = tid & 7, rb = tid >> 3;
    const uint32_t dst_off = (uint32_t)rb * 128 + (uint32_t)((j ^ (rb & 7)) << 4);
    int it = 0;                                        // global stage counter (ring position)
    for (int tile = cid; tile < total_tiles; tile += ncl) {
      const int m0 = tile_m0(tile);
      uint32_t rowoff[8];
      uint32_t rowok = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int m = m0 + rb + 16 * i;
        rowoff[i] = 0;
        if (m < p.M_rows) {
          const int img = fast_div(m, p.magic_rows), rem = m - img * p.rows_per_img;
          const int oy = fast_div(rem, p.magic_wox), oxb = rem - oy * p.Wox;
          rowoff[i] = (uint32_t)(p.in_origin_b + (long long)img * p.in_pitch_n_b + (long long)oy * p.in_row_step_b +
                                 (long long)oxb * p.in_col_step_b);
          rowok |= 1u << i;
        }
      }
      int ky = 0, jj = j;                              // granule (s*8 + j) = ky * run_granules + jj
      while (jj >= p.run_granules) { jj -= p.run_granules; ++ky; }
      for (int s = 0; s < p.k_stages; ++s, ++it) {
        const int slot = it % STAGES;
        mbar_wait(empty0 + 8 * slot, ((it / STAGES) & 1) ^ 1);
        const int g = s * 8 + j;
        if (g < p.total_granules + (p.total_granules & 1)) {   // granules past K are never read by an MMA
          const bool gvalid = g < p.total_granules;            // the odd partner granule must be zero
          const uint8_t* src = p.in + (long long)ky * p.in_pitch_y_b + jj * 16;
          const uint32_t dst = smem_u32(sA + slot * A_STAGE_BYTES) + dst_off;
          // rows past M (tail tile, batch-1 latency path) are never stored: leave their smem rows stale
#pragma unroll
          for (int i = 0; i < 8; ++i)
            if ((rowok >> i) & 1u) cp_async16(dst + i * 16 * 128, gvalid ? src + rowoff[i] : p.in, gvalid ? 16u : 0u);
        }
        // the hardware arrives on the stage's full barrier when this thread's copies have landed (no wait here,
        // same producer protocol as CUTLASS's sm100 cp.async + UMMA mainloop)
        cp_async_mbar_arrive_noinc(full0 + 8 * slot);
        jj += 8;
        while (jj >= p.run_granules) { jj -= p.run_granules; ++ky; }
      }
    }
    cp_async_wait_all();
  } else if (warp == 4) {
    // ===================== MMA issuer =====================
    // The whole warp runs the (warp-uniform) loop control; only the tcgen05 instructions are predicated on the
    // elected lane, so descriptors stay in uniform registers and MMAs issue back to back.
    constexpr uint32_t idesc = umma_idesc_bf16(BM * NCTA, BN);
    constexpr uint64_t DESC_HI = (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t a16_0 = (smem_u32(sA) & 0x3FFFFu) >> 4, b16_0 = (smem_u32(sB) & 0x3FFFFu) >> 4;
    const int k_stages = p.k_stages, k_steps = p.k_steps;
    int it = 0, tcount = 0;
    long long mw_full = 0, mw_te = 0;
    const long long mbeg = ig_clock();
    if (B_RES) mbar_wait(bres, 0);
    for (int tile = cid; tile < (cta_leader ? total_tiles : 0); tile += ncl, ++tcount) {   // the leader issues for the pair
      const int ab = tcount & 1;
      long long tq = ig_clock();
      mbar_wait(tempty0 + 8 * ab, ((tcount >> 1) & 1) ^ 1);      // epilogue has drained this accumulator
      mw_te += ig_clock() - tq;
      tc_fence_after();
      const uint32_t d_tmem = tmem_u + (uint32_t)(ab * BN);
      const bool leader = elect_one();
      for (int s = 0; s < k_stages; ++s, ++it) {
        const int slot = it % STAGES;
        tq = ig_clock();
        mbar_wait(full0 + 8 * slot, (it / STAGES) & 1);
        mw_full += ig_clock() - tq;
        tc_fence_after();
        const uint32_t alo = a16_0 + (uint32_t)(slot * (A_STAGE_BYTES / 16));
        const uint32_t blo = b16_0 + (uint32_t)((B_RES ? s : slot) * (B_STAGE_BYTES / 16));
        const int ksteps = min(4, k_steps - s * 4);
        if (leader) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)      // +32 B along K inside the swizzle row = +2 in descriptor units
            if (kk < ksteps) {
              if (PAIR)
                tc_mma_bf16_pair(d_tmem, DESC_HI | (uint64_t)(alo + 2 * kk), DESC_HI | (uint64_t)(blo + 2 * kk), idesc,
                                 (s | kk) != 0 ? 1u : 0u);
              else
                tc_mma_bf16(d_tmem, DESC_HI | (uint64_t)(alo + 2 * kk), DESC_HI | (uint64_t)(blo + 2 * kk), idesc,
                            (s | kk) != 0 ? 1u : 0u);
            }
          if (PAIR) tc_commit_pair(empty0 + 8 * slot); else tc_commit(empty0 + 8 * slot);
          if (s == k_stages - 1) { if (PAIR) tc_commit_pair(tfull0 + 8 * ab); else tc_commit(tfull0 + 8 * ab); }
        }
        __syncwarp();
      }
    }
    tc_fence_before();
    if (UAHN_IG_PROFILE && p.dbg && lane == 0) {
      unsigned long long* d = p.dbg + blockIdx.x * 16;
      d[2] = mw_full; d[3] = mw_te; d[4] = ig_clock() - mbeg; d[9] = tcount;
    }
  } else if (warp == 5) {
    // ===================== B loader (gather / MC modes; the im2col mode loads B from warp 1) =====================
    // warp-uniform loop, the copies predicated on one elected lane (see the im2col producers)
    const bool leader = elect_one();
    if (PAIR && lane == 0) tma_prefetch_desc(&bmap);
    if (B_RES) {
      const int n0 = (blockIdx.x % p.n_tiles) * BN;   // resident mode is launched with n_tiles == 1
      if (leader) {
        mbar_arrive_expect_tx(bres, (uint32_t)(p.k_stages * B_STAGE_BYTES));
        for (int s = 0; s < p.k_stages; ++s)
          bulk_g2s(smem_u32(sB + s * B_STAGE_BYTES), p.b_image + ((size_t)s * p.n_total + n0) * 128, B_STAGE_BYTES, bres);
      }
    } else if (AM != AM_IM2COL) {
      int slot = 0;
      uint32_t par = 1;
      long long bw = 0;
      const long long bbeg = ig_clock();
      for (int tile = cid; tile < total_tiles; tile += ncl) {
        const int n0 = (tile % p.n_tiles) * BN;
        for (int s = 0; s < p.k_stages; ++s) {
          const long long t0 = ig_clock();
          mbar_wait(empty0 + 8 * slot, par);
          bw += ig_clock() - t0;
          if (leader) {
            if (PAIR) {   // both halves complete on the leader CTA's barrier
              if (cta_leader) mbar_arrive_expect_tx(full0 + 8 * slot, 2 * B_STAGE_BYTES);
              tma_load_2d_pair(smem_u32(sB + slot * B_STAGE_BYTES), &bmap, 0, s * p.n_total + n0 + (int)crank * (BN / 2),
                               full0 + 8 * slot);
            } else {
              mbar_arrive_expect_tx(full0 + 8 * slot, B_STAGE_BYTES);
              bulk_g2s(smem_u32(sB + slot * B_STAGE_BYTES), p.b_image + ((size_t)s * p.n_total + n0) * 128, B_STAGE_BYTES,
                       full0 + 8 * slot);
            }
          }
          __syncwarp();
          if (++slot == STAGES) { slot = 0; par ^= 1u; }
        }
      }
      if (UAHN_IG_PROFILE && p.dbg && lane == 0) { p.dbg[blockIdx.x * 16 + 11] = bw; p.dbg[blockIdx.x * 16 + 12] = ig_clock() - bbeg; }
    }
  } else {
    // ===================== epilogue (warps 6-9): TMEM -> bias/LeakyReLU -> bf16 -> smem -> coalesced global ====
    const int q = warp & 3;                             // TMEM lane quadrant this warp may read
    const uint32_t out_s = smem_u32(sOut + q * 32 * SROW), row_s = smem_u32(sRowOff + q * 32), bias_s = smem_u32(sBias);
    constexpr int CH = epi_chunk<BN>();                 // accumulator columns per staging pass
    constexpr int CPR = CH / 8;                         // 16-byte chunks per staged row
    constexpr int RPI = 32 / CPR;                       // rows covered by one warp-wide store
    int tcount = 0;
    long long ew = 0, e_ld = 0, e_st = 0;
    const long long ebeg = ig_clock();
    for (int tile = cid; tile < total_tiles; tile += ncl, ++tcount) {
      const int ab = tcount & 1;
      const int m0 = tile_m0(tile), n0 = (tile % p.n_tiles) * BN;
      {
        const int m = m0 + q * 32 + lane;
        long long off = -1;
        if (m < p.M_rows) {
          const int img = fast_div(m, p.magic_rows), rem = m - img * p.rows_per_img;
          const int oy = fast_div(rem, p.magic_wox), oxb = rem - oy * p.Wox;
          off = p.out_origin_b + (long long)img * p.out_pitch_n_b + (long long)oy * p.out_pitch_y_b +
                (long long)oxb * p.out_col_step_b + (long long)n0 * 2;
        }
        st_shared_b64(row_s + (uint32_t)lane * 8, off);
      }
      long long tq = ig_clock();
      mbar_wait(tfull0 + 8 * ab, (tcount >> 1) & 1);
      ew += ig_clock() - tq;
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * BN);
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += CH) {
        tq = ig_clock();
#pragma unroll
        for (int c = 0; c < CH / 16; ++c) {
          uint32_t r[16];
          tmem_ld16(taddr + c0 + c * 16, r);
          tmem_ld_wait();
          uint32_t packed[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float2 b2 = ld_shared_f32x2(bias_s + (uint32_t)(n0 + c0 + c * 16 + 2 * e) * 4);
            const float v0 = __uint_as_float(r[2 * e]) + b2.x, v1 = __uint_as_float(r[2 * e + 1]) + b2.y;
            // LeakyReLU on the packed bf16 pair: the same epilogue arithmetic as the TMA and fused-front kernels
            packed[e] = p.act ? pack_lrelu_bf16x2(v0, v1) : pack_bf16x2(v0, v1);
          }
          st_shared_v4(out_s + (uint32_t)(lane * SROW + c * 32), packed[0], packed[1], packed[2], packed[3]);
          st_shared_v4(out_s + (uint32_t)(lane * SROW + c * 32 + 16), packed[4], packed[5], packed[6], packed[7]);
        }
        if (c0 + CH >= BN) {                              // the whole accumulator is in registers / staged
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { if (PAIR) mbar_arrive_leader(tempty0 + 8 * ab); else mbar_arrive(tempty0 + 8 * ab); }   // the next tile's MMAs may start
        } else {
          __syncwarp();
        }
        e_ld += ig_clock() - tq;
        tq = ig_clock();
        const int rsub = lane / CPR, ch = lane % CPR;
#pragma unroll 4
        for (int r0 = 0; r0 < 32; r0 += RPI) {
          const int row = r0 + rsub;
          const long long off = ld_shared_b64(row_s + (uint32_t)row * 8);
          const uint4 v = ld_shared_v4(out_s + (uint32_t)(row * SROW + ch * 16));
          if (off >= 0) st_global_v4(p.out + off + c0 * 2 + ch * 16, v.x, v.y, v.z, v.w);
        }
        __syncwarp();
        e_st += ig_clock() - tq;
      }
    }
    if (UAHN_IG_PROFILE && p.dbg && warp == 6 && lane == 0) {
      unsigned long long* d = p.dbg + blockIdx.x * 16;
      d[5] = ew; d[6] = e_ld; d[7] = e_st; d[8] = ig_clock() - ebeg;
    }
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();   // the peer's shared memory and TMEM are in use until the leader's last MMA has retired
  if (UAHN_IG_PROFILE && p.dbg && tid == 0) { p.dbg[blockIdx.x * 16 + 13] = k_roles - k_entry; p.dbg[blockIdx.x * 16 + 14] = ig_clock() - k_entry; }
  if (warp == 4) {
    tc_fence_after();
    if (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)tmem_cols<BN>())
                   : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)tmem_cols<BN>())
                   : "memory");
  }
}

template <int BN>
constexpr size_t fixed_smem() { return 1024 + 128 * (size_t)stage_row_bytes<BN>() + 256 * 4 + 128 * 8 + 64 * 8; }

template <int BN, int STAGES, bool B_RES, int AM = AM_GATHER, bool PAIR = false>
cudaError_t launch_t(const IgemmParams& p, int num_sms, cudaStream_t st, const CUtensorMap* amap = nullptr,
                     const CUtensorMap* bmap = nullptr) {
  constexpr int NCTA = PAIR ? 2 : 1;
  const size_t smem =
      fixed_smem<BN>() + (size_t)STAGES * A_STAGE_BYTES + (size_t)(B_RES ? p.k_stages : STAGES) * (BN * 128 / NCTA);
  if (smem > SMEM_LIMIT) return cudaErrorInvalidConfiguration;
  auto kern = conv_igemm_bf16_kernel<BN, STAGES, B_RES, AM, PAIR>;
  static SmemOptIn optin;   // per device (common.cuh)
  if (cudaError_t e = optin.ensure(kern, smem); e != cudaSuccess) return e;
  static const CUtensorMap no_map{};
  if (PAIR && (!bmap || (AM == AM_IM2COL && !amap))) return cudaErrorInvalidValue;
#if UAHN_IG_PROFILE
  static unsigned long long* d_dbg = nullptr;
  const bool debug = getenv("UAHN_IG_DEBUG") != nullptr;
  if (debug && !d_dbg) cudaMalloc(&d_dbg, 16 * 8 * 256);
  if (debug) cudaMemsetAsync(d_dbg, 0, 16 * 8 * 256, st);
  IgemmParams pd = p;
  pd.dbg = debug ? d_dbg : nullptr;
#else
  const IgemmParams& pd = p;
#endif
  // PAIR: one unit = two consecutive M tiles of one N tile, one cluster of two CTAs per unit
  const int units = ((p.m_tiles + NCTA - 1) / NCTA) * p.n_tiles;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(NCTA * std::min(units, num_sms / NCTA));
  cfg.blockDim = dim3(ig_threads(AM));
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = NCTA;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  cudaError_t le = cudaLaunchKernelEx(&cfg, kern, pd, amap ? *amap : no_map, bmap ? *bmap : no_map);
#if UAHN_IG_PROFILE
  if (debug && le == cudaSuccess) {
    const int grid = (int)cfg.gridDim.x;
    std::vector<unsigned long long> h(16 * grid);
    cudaStreamSynchronize(st);
    cudaMemcpy(h.data(), d_dbg, h.size() * 8, cudaMemcpyDeviceToHost);
    for (int par = 0; par < NCTA; ++par) {
      double a[16] = {0};
      int cnt = 0;
      for (int i = par; i < grid; i += NCTA, ++cnt) for (int j = 0; j < 16; ++j) a[j] += (double)h[i * 16 + j];
      for (int j = 0; j < 16; ++j) a[j] /= cnt;
      fprintf(stderr, "[uahn-ig] BN=%d S=%d AM=%d k_stages=%d m_tiles=%d %s: stages/CTA %.1f tiles/CTA %.1f | producer wait_empty %.0f of %.0f | B loader wait_empty %.0f of %.0f | mma wait_full %.0f wait_tempty %.0f of %.0f | epi wait_tfull %.0f ld+pack %.0f store %.0f of %.0f (cycles per CTA) | prologue %.0f kernel %.0f\n",
              BN, STAGES, AM, p.k_stages, p.m_tiles, !PAIR ? "" : par ? "peer  " : "leader", a[10], a[9], a[0], a[1], a[11], a[12], a[2], a[3], a[4], a[5],
              a[6], a[7], a[8], a[13], a[14]);
    }
  }
#endif
  return le;
}

}  // namespace

uint16_t f32_to_bf16_host(float f) {   // round-to-nearest-even, like __float2bfloat16_rn
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
static inline uint16_t f2bf(float f) { return f32_to_bf16_host(f); }

// Choose XB (output pixels per GEMM row) for a layer.  Constraints: XB divides Wo; the run start must be
// 16-byte aligned (XB*stride*Cin*2 % 16 == 0); N = XB*Cout in [16, 256], multiple of 16.
static int choose_xb(const ConvGeom& g) {
  if (g.KH == 1 && g.KW == 1) return 1;
  int best = 0;
  double best_cost = 1e30;
  for (int xb = 1; xb <= 16; xb *= 2) {
    if (g.Wo % xb) continue;
    if ((xb * g.stride * g.Cin * 2) % 16) continue;
    const int n = xb * g.Cout;
    if (n < 16 || n > 256 || n % 16) continue;
    const int run_elems = (g.stride * (xb - 1) + g.KW) * g.Cin;
    const int rlg = (run_elems + 7) / 8;
    const int stages = (g.KH * rlg + 7) / 8;
    const double rows = (double)g.Ho * g.Wo / xb;
    // per 128-row tile and K stage: gather ~256 cycles (LDGSTS issue), MMA 2N cycles (SURVEY/DESIGN cost model)
    const double cost = rows / 128.0 * stages * std::max(256.0, 2.0 * n);
    if (cost < best_cost) { best_cost = cost; best = xb; }
  }
  return best;
}

int conv_bf16_prepare(ConvBf16Weights& wb, const std::vector<float>& wk, const std::vector<float>& bias,
                      const ConvGeom& g, const Tensor& in, const Tensor& out, std::vector<void*>& allocs,
                      std::string& err) {
  (void)out;
  if (in.p) {
    // block_2_1: the dedicated TMA-staged stride-2 first-layer kernel; other convolutions: the shifted-window TMA kernels
    std::string serr;
    int rc = conv_s2first_prepare(wb.s2, wk, bias, g, in, allocs, serr);
    if (rc < 0) { err = serr; return rc; }
    if (wb.s2.enabled) { wb.ready = 1; return 0; }
    rc = conv_tma_prepare(wb.tma, wk, bias, g, in, allocs, serr);
    if (rc < 0) { err = serr; return rc; }
    if (wb.tma.enabled) { wb.ready = 1; return 0; }
  }
  // im2col TMA A producer: layers whose K stage is exactly one (tap, 64-channel chunk)
  const bool im2col_ok = in.p && g.Cin % 64 == 0 && g.KH == g.KW && g.KH > 1;
  const int xb = im2col_ok ? 1 : choose_xb(g);
  if (!xb) { err = "no valid Toeplitz factor"; return -1; }
  if (g.Cin % 8 && !(g.Cin == 2 && (xb * g.stride) % 4 == 0)) { err = "unsupported Cin"; return -1; }
  const int n_total = xb * g.Cout;
  const int run_elems = (g.stride * (xb - 1) + g.KW) * g.Cin;
  const int rlg = (run_elems + 7) / 8;
  const int total_granules = g.KH * rlg;
  const int k_steps = (total_granules + 1) / 2;
  const int k_stages = (k_steps + 3) / 4;
  std::vector<uint16_t> img((size_t)k_stages * n_total * 64, 0);
  for (int ky = 0; ky < g.KH; ++ky)
    for (int q = 0; q < rlg * 8; ++q) {
      const int xi = q / g.Cin, c = q % g.Cin;
      const int kidx = (ky * rlg) * 8 + q;              // K index inside the GEMM
      const int s = kidx / 64, kk = kidx % 64;
      for (int xo = 0; xo < xb; ++xo) {
        const int kx = xi - xo * g.stride;
        if (kx < 0 || kx >= g.KW) continue;
        for (int co = 0; co < g.Cout; ++co) {
          const int n = xo * g.Cout + co;
          const float w = wk[(size_t)((ky * g.KW + kx) * g.Cin + c) * g.Cout + co];
          const size_t byte = ((size_t)s * n_total + n) * 128 + (size_t)((((kk >> 3) ^ (n & 7)) << 4) + (kk & 7) * 2);
          img[byte / 2] = f2bf(w);
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
  if (im2col_ok) {
    static PFN_cuTensorMapEncodeIm2col_v12000 encode = nullptr;
    if (!encode) {
      void* fp = nullptr;
      cudaDriverEntryPointQueryResult qres;
      if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fp, cudaEnableDefault, &qres) == cudaSuccess &&
          qres == cudaDriverEntryPointSuccess)
        encode = reinterpret_cast<PFN_cuTensorMapEncodeIm2col_v12000>(fp);
    }
    if (encode) {
      const int p_ = (g.KH - 1) / 2, s_ = g.stride;
      const int Wt = in.Wp - (in.pwl - p_), Ht = in.Hp - (in.ph - p_);     // extents seen from the window origin
      const cuuint64_t gdim[4] = {(cuuint64_t)g.Cin, (cuuint64_t)Wt, (cuuint64_t)Ht, (cuuint64_t)in.N};
      const cuuint64_t gstr[3] = {(cuuint64_t)g.Cin * 2, (cuuint64_t)g.in_pitch_y * 2, (cuuint64_t)g.in_pitch_n * 2};
      // base pixels (window origins) run over [0, W + upper): exactly Wo x Ho positions per image at the conv stride
      const int lower[2] = {0, 0};
      const int upper[2] = {s_ * (g.Wo - 1) + 1 - Wt, s_ * (g.Ho - 1) + 1 - Ht};
      const cuuint32_t estr[4] = {1, (cuuint32_t)s_, (cuuint32_t)s_, 1};
      void* base = (uint8_t*)in.p + g.in_origin * 2;
      const CUresult r = encode(reinterpret_cast<CUtensorMap*>(wb.im2col_map), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, gdim,
                                gstr, lower, upper, 64, BM, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      wb.im2col = r == CUDA_SUCCESS;
      if (getenv("UAHN_DEBUG"))
        fprintf(stderr, "[uahn] im2col TMA map Cin=%d k=%d s=%d out=%dx%d: W'=%d H'=%d upper=(%d,%d) -> %s\n", g.Cin, g.KH, s_,
                g.Ho, g.Wo, Wt, Ht, upper[0], upper[1], wb.im2col ? "ok" : "encode failed, cp.async gather");
    }
  }
  // CTA-pair mode streams each CTA's half of a B stage through a plain 2-D tiled map over the pre-swizzled image
  // (rows of 128 bytes, copied verbatim: no swizzle in the map)
  {
    static PFN_cuTensorMapEncodeTiled_v12000 encode_tiled = nullptr;
    if (!encode_tiled) {
      void* fp2 = nullptr;
      cudaDriverEntryPointQueryResult q2;
      if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp2, cudaEnableDefault, &q2) == cudaSuccess &&
          q2 == cudaDriverEntryPointSuccess)
        encode_tiled = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fp2);
    }
    wb.pair_ok = encode_tiled && n_total >= 64 && !getenv("UAHN_NO_IGEMM_PAIR");
    for (int i = 0; i < 3 && wb.pair_ok; ++i) {
      const int rows = 128 >> i;
      if (rows * 2 > n_total) { memset(wb.b_half_map[i], 0, 128); continue; }
      const cuuint64_t bdim[2] = {64, (cuuint64_t)k_stages * n_total};
      const cuuint64_t bstr[1] = {128};
      const cuuint32_t bbox[2] = {64, (cuuint32_t)rows};
      const cuuint32_t bes[2] = {1, 1};
      const CUresult rb = encode_tiled(reinterpret_cast<CUtensorMap*>(wb.b_half_map[i]), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, d,
                                       bdim, bstr, bbox, bes, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                       CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (rb != CUDA_SUCCESS) wb.pair_ok = 0;
    }
  }
  wb.b_image = d;
  wb.bias_x = (float*)db;
  wb.xb = xb;
  wb.n_total = n_total;
  wb.k_total = k_stages * 64;
  wb.runs = g.KH;
  wb.run_granules = rlg;
  wb.ready = 1;
  return 0;
}

// The two 5120 -> 256 linears of the MC-dropout heads with the dropout expansion fused into the A producer.
// feat: [n][5120] bf16 (NHWC feature order); mc_bits: this head's keep bits; out: [n*16][256] bf16 hidden activations.
cudaError_t launch_mc_gemm_bf16(const ConvBf16Weights& wb, const void* feat, const uint8_t* mc_bits, void* out, int n,
                                cudaStream_t st) {
  if (!wb.ready || wb.n_total != FC_HID || wb.k_total != FC_IN) return cudaErrorInvalidValue;
  const int num_sms = device_num_sms();
  IgemmParams p{};
  p.in = (const uint8_t*)feat;
  p.b_image = (const uint8_t*)wb.b_image;
  p.bias_x = wb.bias_x;
  p.out = (uint8_t*)out;
  p.mc_bits = mc_bits;
  p.Wox = 1; p.rows_per_img = 1;
  p.M_rows = n * MC;
  p.magic_rows = (1ull << 40); p.magic_wox = (1ull << 40);
  p.total_granules = FC_IN / 8; p.run_granules = FC_IN / 8;
  p.k_steps = FC_IN / 16; p.k_stages = FC_IN / 64;
  p.out_pitch_n_b = FC_HID * 2; p.out_pitch_y_b = FC_HID * 2; p.out_col_step_b = FC_HID * 2; p.out_origin_b = 0;
  p.n_total = FC_HID;
  p.act = 1;
  p.m_tiles = (p.M_rows + BM - 1) / BM;
  p.n_tiles = 1;
  // CTA pairs (two consecutive 8-pair M tiles share every UMMA, half of each weight stage per CTA) once there are
  // enough tiles: the one-CTA kernel is bound by shared-memory bandwidth (16 KB of A + 32 KB of B written and 48 KB read
  // by the tensor core per stage), the pair moves a third less
  if (wb.pair_ok && p.m_tiles >= 32)
    return launch_t<256, 6, false, AM_MC, true>(p, num_sms, st, nullptr, reinterpret_cast<const CUtensorMap*>(wb.b_half_map[0]));
  return launch_t<256, 4, false, AM_MC>(p, num_sms, st);
}

cudaError_t launch_conv_bf16(const ConvBf16Weights& wb, const void* in, const float* bias, void* out,
                             const ConvGeom& g, cudaStream_t st) {
  if (!wb.ready) return cudaErrorInvalidValue;
  const int num_sms = device_num_sms();
  if (wb.s2.enabled) return launch_conv_s2first(wb.s2, out, g, num_sms, st);
  if (wb.tma.enabled) return launch_conv_tma(wb.tma, bias, out, g, num_sms, st);
  if (conv_small_m_ok(wb, g)) return launch_conv_small_m(wb, in, wb.bias_x, out, g, st);   // batch 1-2: split-K over a cluster
  IgemmParams p{};
  const int xb = wb.xb;
  p.in = (const uint8_t*)in;
  p.b_image = (const uint8_t*)wb.b_image;
  p.bias_x = wb.bias_x;
  p.out = (uint8_t*)out;
  p.Wox = g.Wo / xb;
  p.rows_per_img = g.Ho * p.Wox;
  p.M_rows = g.M / xb;
  p.magic_rows = ((1ull << 40) + p.rows_per_img - 1) / p.rows_per_img;
  p.magic_wox = ((1ull << 40) + p.Wox - 1) / p.Wox;
  p.in_pitch_n_b = g.in_pitch_n * 2;
  p.in_pitch_y_b = (int)(g.in_pitch_y * 2);
  p.in_row_step_b = (int)(g.stride * g.in_pitch_y * 2);
  p.in_col_step_b = xb * g.stride * g.Cin * 2;
  p.in_origin_b = g.in_origin * 2;
  p.run_granules = wb.run_granules;
  p.total_granules = wb.runs * wb.run_granules;
  p.k_steps = (p.total_granules + 1) / 2;
  p.k_stages = (p.k_steps + 3) / 4;
  p.out_pitch_n_b = g.out_pitch_n * 2;
  p.out_pitch_y_b = (int)(g.out_pitch_y * 2);
  p.out_col_step_b = xb * g.Cout * 2;
  p.out_origin_b = g.out_origin * 2;
  p.n_total = wb.n_total;
  p.act = g.act;
  const long long n_img = (g.M + (long long)g.Ho * g.Wo - 1) / ((long long)g.Ho * g.Wo);
  if (n_img * p.in_pitch_n_b >= (1ll << 32) || (long long)p.M_rows * p.rows_per_img >= (1ll << 40))
    return cudaErrorInvalidValue;   // 32-bit gather offsets / fast_div range
  p.m_tiles = (p.M_rows + BM - 1) / BM;
  // N tile: all of N when there are enough M tiles to fill the machine; narrower for the small-M tail layers
  int bn = std::min(p.n_total, 256);
  while (bn > 64 && (long long)p.m_tiles * (p.n_total / bn) < num_sms) bn /= 2;
  p.n_tiles = p.n_total / bn;
  // B resident in shared memory when the whole operand of this N tile fits next to a 4-stage A ring
  const bool res = p.n_tiles == 1 && (size_t)p.k_stages * bn * 128 <= 112 * 1024;
  if (wb.im2col) {
    p.Ho = g.Ho; p.stride = g.stride; p.KW = g.KW; p.cin_chunks = g.Cin / 64;
    const CUtensorMap* am = reinterpret_cast<const CUtensorMap*>(wb.im2col_map);
    // enough tiles to fill the machine: CTA pairs (half the B bytes per SM and tile)
    if (wb.im2col && wb.pair_ok && (long long)p.m_tiles * p.n_tiles >= num_sms) {
      switch (bn) {
        case 256: return launch_t<256, 6, false, AM_IM2COL, true>(p, num_sms, st, am, reinterpret_cast<const CUtensorMap*>(wb.b_half_map[0]));
        case 128: return launch_t<128, 8, false, AM_IM2COL, true>(p, num_sms, st, am, reinterpret_cast<const CUtensorMap*>(wb.b_half_map[1]));
        case 64: return launch_t<64, 8, false, AM_IM2COL, true>(p, num_sms, st, am, reinterpret_cast<const CUtensorMap*>(wb.b_half_map[2]));
        default: break;
      }
    }
    switch (bn) {
      case 256: return launch_t<256, 4, false, AM_IM2COL>(p, num_sms, st, am);
      case 128: return res ? launch_t<128, 5, true, AM_IM2COL>(p, num_sms, st, am) : launch_t<128, 6, false, AM_IM2COL>(p, num_sms, st, am);
      case 64: return res ? launch_t<64, 5, true, AM_IM2COL>(p, num_sms, st, am) : launch_t<64, 8, false, AM_IM2COL>(p, num_sms, st, am);
      default: break;   // narrower tiles: the gather path below
    }
  }
  switch (bn) {
    case 256: return launch_t<256, 4, false>(p, num_sms, st);
    case 128: return res ? launch_t<128, 5, true>(p, num_sms, st) : launch_t<128, 6, false>(p, num_sms, st);
    case 64: return res ? launch_t<64, 5, true>(p, num_sms, st) : launch_t<64, 8, false>(p, num_sms, st);
    case 32: return res ? launch_t<32, 5, true>(p, num_sms, st) : launch_t<32, 8, false>(p, num_sms, st);
    case 16: return res ? launch_t<16, 5, true>(p, num_sms, st) : launch_t<16, 8, false>(p, num_sms, st);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace uahn
