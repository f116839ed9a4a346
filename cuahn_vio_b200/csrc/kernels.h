// Launch wrappers of the UAHN kernels (definitions in the .cu files next to this header).
#pragma once
#include "common.cuh"

struct uahn_handle;

namespace uahn {

// engine.cu: what the filter bank (filter_bank.cu) needs of a handle; handle_fail records `msg` for uahn_last_error
int handle_device(const uahn_handle* h);
int handle_max_batch(const uahn_handle* h);
int handle_fail(uahn_handle* h, int code, const char* msg);

// image_kernels.cu
// The current frames of one call as zero-separated cells of a 2-D CUDA array: the source of the texture-gather warp kernel
// (bf16 path, batches above the latency path).  fill: linear u8 frames [n][224][320] -> cells.
struct WarpCells {
  cudaArray_t arr = nullptr;
  cudaTextureObject_t tex = 0;
  cudaSurfaceObject_t surf = 0;
  int cap = 0;
};
int warp_cells_capacity();      // images one array can hold (texture-gather arrays are limited to 32768 x 32768 texels)
cudaError_t warp_cells_create(WarpCells& c, int cap, cudaStream_t st);
void warp_cells_destroy(WarpCells& c);
cudaError_t launch_warp_cells_fill(const WarpCells& c, const uint8_t* frames, int n, cudaStream_t st);
// cells != nullptr (bf16 only): curr has been copied into the cell array by launch_warp_cells_fill
template <typename T>
cudaError_t launch_warp_concat_pool(const uint8_t* prev, const uint8_t* curr, const float* Hmat, const Tensor& out,
                                    int pool, int n, cudaStream_t st, const WarpCells* cells = nullptr);
// out (float) or out_u8 (error map clamped to [0,255] and truncated, HomographyNet.cpp:201) — exactly one is non-null
// allow_fast: the bf16 product path's coordinate mode (image_kernels.cu CM_FAST: fast coordinates, exact fallback near
// integer boundaries — indices stay bit-exact); 0 = the exact chain everywhere (fp32 validation mode)
cudaError_t launch_warp_plain(const uint8_t* prev, const uint8_t* curr, const float* Hmat, float* out, uint8_t* out_u8,
                              int16_t* ix, int16_t* iy, int error_map, int n, cudaStream_t st, int allow_fast);

// cv::remap(INTER_LINEAR, constant-0 border) of n raw u8 frames through one pair of float maps (224x320 each) into n
// 224x320 u8 images.  Raw frame i's row y starts at raw + (i * rows + y) * pitch; out is [n][224][320].
cudaError_t launch_remap_u8(const uint8_t* raw, int rows, int cols, size_t pitch, int n, const float* map1,
                            const float* map2, uint8_t* out, cudaStream_t st);

// conv_f32.cu
// ws: optional split-K workspace (ws_floats floats) for the small-M deep layers of the latency path; rows_per_pair: GEMM rows
// one pair contributes (Ho * Wo, or 16 for the MC-head linears) — the split is chosen from it, not from the batch
cudaError_t launch_conv_f32(const float* in, const float* wk, const float* bias, float* out, const ConvGeom& g,
                            cudaStream_t st, float* ws = nullptr, size_t ws_floats = 0, int rows_per_pair = 0);
int conv_f32_extra_launches();   // kernels beyond the first that this thread's last launch_conv_f32 call enqueued (split-K reduce)

// head_kernels.cu
// transfer_mean_var_single + packing for n pairs: var, pts_w [n][8], Hp [n][9] -> flow [n][8], cov [n][64]
cudaError_t launch_transfer(int n, const float* var, const float* Hp, const float* pts_w, float* mean, float* cov,
                            cudaStream_t st);
cudaError_t launch_dlt(int n, const float* off, const float* Hprev, float* Hout, cudaStream_t st);
template <typename T>
cudaError_t launch_fc8_dlt(int n, const T* feat, const float* W8, const float* b8, const float* Hprev, float* Hout,
                           float* dout, cudaStream_t st);
template <typename T>
cudaError_t launch_mc_expand(int n, const T* feat, T* A, const uint8_t* keep_masks, uint64_t seed, uint64_t first_pair,
                             const uint64_t* rng_dev, cudaStream_t st);
// first MC-head layer on CUDA cores for the batch-1 latency path (bf16): A [n][16][5120], W [256][5120], out [n][16][256]
cudaError_t launch_mc_fc1_small(int n, const void* A, const void* W, const float* bias, void* out, cudaStream_t st);
// the same with the dropout expansion fused in and both heads in one launch: feat [n][5120] bf16 -> hid [2][n][16][256]
cudaError_t launch_mc_fc1_small_fused(int n, const void* feat, const void* Wm, const void* Wu, const float* bm, const float* bu,
                                      void* hid, const uint8_t* keep_masks, uint64_t seed, uint64_t first_pair,
                                      const uint64_t* rng_dev, cudaStream_t st);
// bits[head][pair][k8][sample]: keep bits of the first MC dropout for the fused masked GEMM (bf16 path)
cudaError_t init_keep_alias_table();   // uploads the keep-byte alias table (common.cuh) to the current device
cudaError_t launch_mc_maskbits(int n, uint8_t* bits, const uint8_t* keep_masks, uint64_t seed, uint64_t first_pair,
                               const uint64_t* rng_dev, cudaStream_t st);
template <typename T>
cudaError_t launch_mc_final(int n, const T* hid, const float* W2m, const float* b2m, const float* W2u,
                            const float* b2u, const float* Hpart1, const uint8_t* keep_masks, uint64_t seed,
                            uint64_t first_pair, const uint64_t* rng_dev, float* mean, float* cov, float* Htot,
                            float* mc_mean, float* mc_logvar, cudaStream_t st);

}  // namespace uahn
