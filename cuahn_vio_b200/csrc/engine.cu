// Host engine + C ABI (include/uahn.h) of the B200-native UAHN forward.
// Stage schedule follows combined_stu_model.forward / Down_Net_3blocks.forward / HomoNet_last_block.forward
// (reference model_to_trace.py:124-193, 258-282, 299-330); see DESIGN.md for the kernel map.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/uahn.h"
#include "../../include/uahn_preproc.h"
#include "common.cuh"
#include "conv_bf16.h"
#include "kernels.h"

using namespace uahn;

namespace uahn {
// Programmatic dependent launch at every batch size: with the next grid already resident in the launch queue its CTAs
// start as SMs drain, which is worth 2-3 us per dependent kernel — 9 % of the batch-1 p50 (27 dependent kernels of a few
// microseconds each), 10 % of a 256-pair call (0.748 -> 0.671 ms), 2 % of a 1024-pair call (same-box A/B on B200).
// The flag is per thread and set by the first forward() on it: the stage entry points and the preprocessing launches of
// a thread that has not run a forward yet go without.  UAHN_NO_PDL=1 disables it.
static thread_local bool g_pdl_on = false;
bool pdl_enabled() {
  static const bool allowed = getenv("UAHN_NO_PDL") == nullptr;
  return allowed && g_pdl_on;
}
}  // namespace uahn

namespace {

thread_local std::string g_create_error;

struct HostTensor {
  std::vector<int> dims;
  std::vector<float> data;
  size_t numel() const {
    size_t n = 1;
    for (int d : dims) n *= d;
    return n;
  }
};

// A truncated or corrupt file must come back as UAHN_ERR_WEIGHTS, never as an exception across the C ABI: every dim is
// bounded, the payload is checked against the bytes left in the file before anything is allocated, and the caller wraps
// the whole load in try/catch.
bool load_weight_file(const char* path, std::map<std::string, HostTensor>& out, std::string& err) {
  FILE* f = fopen(path, "rb");
  if (!f) { err = std::string("cannot open weights file: ") + path; return false; }
  struct Closer { FILE* f; ~Closer() { fclose(f); } } closer{f};
  if (fseek(f, 0, SEEK_END) != 0) { err = "cannot seek in weights file"; return false; }
  const long file_size = ftell(f);
  rewind(f);
  char magic[8];
  uint32_t count = 0;
  if (fread(magic, 1, 8, f) != 8 || memcmp(magic, "UAHNWTS1", 8) != 0 || fread(&count, 4, 1, f) != 1 || count > 4096) {
    err = "bad weights file header"; return false;
  }
  for (uint32_t i = 0; i < count; ++i) {
    uint32_t nl = 0, nd = 0;
    if (fread(&nl, 4, 1, f) != 1 || nl == 0 || nl > 256) { err = "bad tensor name"; return false; }
    std::string name(nl, '\0');
    if (fread(&name[0], 1, nl, f) != nl || fread(&nd, 4, 1, f) != 1 || nd > 4) { err = "bad tensor header"; return false; }
    HostTensor t;
    t.dims.resize(nd);
    size_t numel = 1;
    for (uint32_t d = 0; d < nd; ++d) {
      uint32_t v;
      if (fread(&v, 4, 1, f) != 1 || v == 0 || v > (1u << 20)) { err = "bad dims of tensor " + name; return false; }
      t.dims[d] = (int)v;
      numel *= v;
      if (numel > (size_t(1) << 28)) { err = "tensor " + name + " is implausibly large"; return false; }
    }
    const long pos = ftell(f);
    if (pos < 0 || file_size < pos || (size_t)(file_size - pos) < numel * 4) { err = "truncated tensor " + name; return false; }
    t.data.resize(numel);
    if (fread(t.data.data(), 4, numel, f) != numel) { err = "truncated tensor " + name; return false; }
    out[name] = std::move(t);
  }
  return true;
}

struct LayerSpec { const char* name; int cout, cin, k, stride; };
// model_to_trace.py:93-95,100-103,108-113,210-216
const LayerSpec B1[] = {{"block_1_1", 128, 2, 7, 2}, {"block_1_2", 128, 128, 5, 2}, {"block_1_3", 256, 128, 3, 2}};
const LayerSpec B2[] = {{"block_2_1", 64, 2, 7, 2}, {"block_2_2", 128, 64, 5, 2}, {"block_2_3", 256, 128, 3, 2}, {"block_2_4", 256, 256, 3, 2}};
const LayerSpec B3[] = {{"block_3_0", 16, 2, 7, 1}, {"block_3_1", 32, 16, 5, 2}, {"block_3_2", 64, 32, 3, 2}, {"block_3_3", 128, 64, 3, 2}, {"block_3_4", 256, 128, 3, 2}, {"block_3_5", 256, 256, 3, 2}};
const LayerSpec B4[] = {{"block_4_0", 8, 2, 7, 1}, {"block_4_1", 16, 8, 5, 2}, {"block_4_2", 32, 16, 3, 2}, {"block_4_3", 64, 32, 3, 2}, {"block_4_4", 128, 64, 3, 2}, {"block_4_5", 256, 128, 3, 2}, {"block_4_6", 256, 256, 3, 2}};
constexpr int F32_SPLITK_MAX_PAIRS = 8; // fp32: up to here the deep SIMT layers split K over the idle SMs (latency path)
constexpr int WARP_TEX_MIN_PAIRS = 8;    // bf16: above this the warp takes its taps by texture gather (image_kernels.cu SMALL_BATCH)
constexpr int MC_SMALL_MAX_PAIRS = 8;    // bf16: up to here the first MC-head layer runs on CUDA cores (latency path)
constexpr int MC_FUSED_MIN_PAIRS = 64;   // bf16: batches from this size on use the fused masked-A MC GEMM
const char* P1 = "model_part1.";
const char* P4 = "model_last_block_list.0.";

struct Layer {
  LayerSpec spec;
  int Hin, Win, Ho, Wo;
  Tensor in, out;
  float* w_f32 = nullptr;   // [K][Cout], k = (ky*KW + kx)*Cin + c
  float* bias = nullptr;
  ConvBf16Weights wb;       // bf16 tcgen05 operand image (precision BF16 only)
};

struct Block {
  int id = 0, pool = 1;
  bool active = false;
  FusedPlan fused;          // blocks 3/4 in bf16: conv 0 + conv 1 fused, conv 0's output never reaches HBM
  Tensor x_unfused;         // small halo-3 input used only by the per-layer stage entry point in fused mode
  Tensor x;                 // 2-channel conv input
  std::vector<Layer> layers;
  float* W8 = nullptr;      // [8][5120] permuted to NHWC feature order (blocks 1-3)
  float* b8 = nullptr;
};

}  // namespace

struct uahn_handle {
  uahn_config cfg{};
  std::string last_error;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  bool bf16 = false;
  size_t es = 4;
  int cap = 0;
  int num_sms = 0;          // of cfg.device
  uint64_t launches = 0;
  std::vector<void*> allocs;
  Block blocks[5];
  // block-4 head
  float *W1m = nullptr, *b1m = nullptr, *W1u = nullptr, *b1u = nullptr;       // [5120][256] fp32 (k' order)
  ConvBf16Weights W1m_b, W1u_b;
  void *W1m_plain = nullptr, *W1u_plain = nullptr;   // [256][5120] bf16, NHWC k order: the batch-1 CUDA-core first layer
  float *W2m = nullptr, *b2m = nullptr, *W2u = nullptr, *b2u = nullptr;
  void* mcA = nullptr;    // [2][n][16][5120] masked features (fp32, small bf16 batches) or keep bits [2][n][640][16] bytes
  void* hid = nullptr;    // [2][cap][16][256] T
  float* Hb[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // cumulative H after prior(0)/block1..3 ; [4] unused
  float* Htot = nullptr;
  float* f32_ws = nullptr;        // fp32 mode: split-K workspace of the SIMT convolutions (latency path)
  size_t f32_ws_floats = 0;
  float* dblk[4] = {nullptr, nullptr, nullptr, nullptr};          // regressed offsets of blocks 1..3
  float *mc_mean = nullptr, *mc_logvar = nullptr;
  // staging for the host-pointer entry points
  uint8_t *d_prev = nullptr, *d_curr = nullptr, *d_masks = nullptr;
  WarpCells cells;          // bf16, batches above the latency path: the current frames as a texture-gather array (image_kernels.cu)
  float *d_prior = nullptr, *d_mean = nullptr, *d_cov = nullptr, *d_err = nullptr;
  // streaming (load_image / infer) state: 2-slot ring
  uint8_t* d_ring = nullptr;
  uint8_t* h_img = nullptr;   // pinned
  float* h_out = nullptr;     // pinned 72 floats (+ err map)
  // undistort + resize in front of the ring (uahn_preproc.h)
  float *d_map1 = nullptr, *d_map2 = nullptr;
  uint8_t *d_raw = nullptr, *h_raw = nullptr;   // h_raw pinned
  int raw_rows = 0, raw_cols = 0;
  int ring_curr = 0;
  int img_counter = 0;
  double latest_time = -1.0;
  int last_n = 0;
  // batch-1 latency path: the whole uahn_infer (H2D prior/rng, ~27 kernels, D2H results) is one CUDA graph per
  // (ring slot, explicit masks?, error map?) combination, captured on the second call and replayed afterwards
  cudaGraphExec_t graphs[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  uint64_t graph_launches[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  // batch-1 inputs travel as ONE 48-byte H2D copy and the results as ONE 288-byte D2H copy (every copy is a graph node
  // of its own on the latency path): {seed, first_pair, prior[8]} pinned + device, {mean[8], cov[64]} device
  uint64_t* d_rng = nullptr;    // device block: {seed, first_pair} read by the MC kernels during graph replay, then prior[8]
  uint64_t* h_rng = nullptr;    // pinned block, same layout
  float* h_prior = nullptr;     // = (float*)(h_rng + 2)
  float* d_in1_prior = nullptr; // = (float*)(d_rng + 2)
  float* d_out1 = nullptr;      // device {mean[8], cov[64]} of uahn_infer
  uint64_t infer_calls = 0;
  bool use_graph = true;
  // pipelined submissions (uahn_submit_batch): copy stream + second staging set
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
  uint8_t *s_prev[2] = {nullptr, nullptr}, *s_curr[2] = {nullptr, nullptr}, *s_frames[2] = {nullptr, nullptr};
  float *s_prior[2] = {nullptr, nullptr}, *s_mean[2] = {nullptr, nullptr}, *s_cov[2] = {nullptr, nullptr};
  uint64_t submit_count = 0;
  bool pipeline_ready = false;
  uint64_t auto_pair = 0;   // MC-dropout pair index of calls made with rng == NULL: fresh masks on every forward
  // per-category device timing (uahn_profile_*)
  struct ProfSpan { cudaEvent_t a, b; int cat; uint64_t launches; };
  bool prof_on = false;
  std::vector<ProfSpan> prof_spans;
  std::vector<cudaEvent_t> prof_pool;
  double prof_ms[4] = {0, 0, 0, 0};
  uint64_t prof_launches[4] = {0, 0, 0, 0};
  int prof_open = -1;
  uint64_t prof_l0 = 0;
  cudaEvent_t prof_event() {
    if (!prof_pool.empty()) { cudaEvent_t e = prof_pool.back(); prof_pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
  }
  void prof_begin(int cat) {
    if (!prof_on) return;
    ProfSpan s{prof_event(), prof_event(), cat, 0};
    cudaEventRecord(s.a, stream);
    prof_spans.push_back(s);
    prof_open = (int)prof_spans.size() - 1;
    prof_l0 = launches;
  }
  void prof_end() {
    if (!prof_on || prof_open < 0) return;
    cudaEventRecord(prof_spans[prof_open].b, stream);
    prof_spans[prof_open].launches = launches - prof_l0;
    prof_open = -1;
  }

  int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    last_error = buf;
    return code;
  }
};

#define CK(expr)                                                                                          \
  do {                                                                                                    \
    cudaError_t e__ = (expr);                                                                             \
    if (e__ != cudaSuccess) return h->fail(UAHN_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)
#define LAUNCH(expr)  \
  do {                \
    CK(expr);         \
    ++h->launches;    \
  } while (0)

namespace {

template <typename T>
int dev_alloc(uahn_handle* h, T** p, size_t count, bool zero = true) {
  void* q = nullptr;
  CK(cudaMalloc(&q, count * sizeof(T) + 4096));
  if (zero) CK(cudaMemset(q, 0, count * sizeof(T) + 4096));
  h->allocs.push_back(q);
  *p = reinterpret_cast<T*>(q);
  return UAHN_OK;
}

int upload(uahn_handle* h, float** dst, const std::vector<float>& v) {
  int rc = dev_alloc(h, dst, v.size(), false);
  if (rc) return rc;
  CK(cudaMemcpy(*dst, v.data(), v.size() * 4, cudaMemcpyHostToDevice));
  return UAHN_OK;
}

int make_tensor(uahn_handle* h, Tensor& t, int N, int H, int W, int C, int pad) {
  t.N = N; t.H = H; t.W = W; t.C = C;
  t.ph = pad; t.pwl = pad; t.pwr = pad ? pad + 8 : 0;
  t.Hp = H + 2 * pad;
  t.Wp = W + t.pwl + t.pwr;
  if (pad) t.Wp = (t.Wp + 7) / 8 * 8;
  t.pitch_n = ((long long)t.Hp * t.Wp * C + 63) / 64 * 64;
  uint8_t* p = nullptr;
  int rc = dev_alloc(h, &p, (size_t)N * t.pitch_n * h->es);
  t.p = p;
  return rc;
}

ConvGeom make_geom(const Layer& L, int n) {
  ConvGeom g{};
  const int p = (L.spec.k - 1) / 2;
  g.Ho = L.Ho; g.Wo = L.Wo; g.M = n * L.Ho * L.Wo;
  g.Cin = L.spec.cin; g.Cout = L.spec.cout; g.KH = g.KW = L.spec.k; g.stride = L.spec.stride;
  g.K = L.spec.k * L.spec.k * L.spec.cin;
  g.in_pitch_n = L.in.pitch_n; g.in_pitch_y = L.in.pitch_y();
  g.in_origin = L.in.off(0, -p, -p, 0);
  g.out_pitch_n = L.out.pitch_n; g.out_pitch_y = L.out.pitch_y();
  g.out_origin = L.out.off(0, 0, 0, 0);
  g.act = 1;
  return g;
}

ConvGeom dense_geom(int rows, int K, int N, int act) {   // Linear as a 1x1 conv over 1x1 images
  ConvGeom g{};
  g.Ho = g.Wo = 1; g.M = rows; g.Cin = K; g.Cout = N; g.KH = g.KW = 1; g.stride = 1; g.K = K;
  g.in_pitch_n = K; g.in_pitch_y = K; g.in_origin = 0;
  g.out_pitch_n = N; g.out_pitch_y = N; g.out_origin = 0;
  g.act = act;
  return g;
}

const HostTensor* find(const std::map<std::string, HostTensor>& w, const std::string& key, std::vector<int> dims,
                       std::string& err) {
  auto it = w.find(key);
  if (it == w.end()) { err = "missing tensor " + key; return nullptr; }
  if (it->second.dims != dims) { err = "shape mismatch for " + key; return nullptr; }
  return &it->second;
}

// [8][5120] or [256][5120] with the 5120 axis in NCHW order (c*20+hw) -> NHWC order (hw*256+c)
std::vector<float> permute_fc_in(const HostTensor& t) {
  const int rows = t.dims[0];
  std::vector<float> o((size_t)rows * FC_IN);
  for (int r = 0; r < rows; ++r)
    for (int c = 0; c < 256; ++c)
      for (int hw = 0; hw < 20; ++hw) o[(size_t)r * FC_IN + hw * 256 + c] = t.data[(size_t)r * FC_IN + c * 20 + hw];
  return o;
}

int build_block(uahn_handle* h, const std::map<std::string, HostTensor>& w, int id, const LayerSpec* specs, int nl,
                int pool) {
  Block& B = h->blocks[id];
  B.id = id; B.pool = pool; B.active = true;
  const char* pre = id == 4 ? P4 : P1;
  int H = IMG_H / pool, W = IMG_W / pool;
  const bool try_fuse = h->bf16 && id >= 3 && !getenv("UAHN_NO_FUSE");
  int rc = make_tensor(h, B.x, h->cap, H, W, 2, try_fuse ? 5 : (specs[0].k - 1) / 2);
  if (rc) return rc;
  const int small_cap = std::min(h->cap, 4);
  if (try_fuse && (rc = make_tensor(h, B.x_unfused, small_cap, H, W, 2, (specs[0].k - 1) / 2))) return rc;
  Tensor cur = try_fuse ? B.x_unfused : B.x;
  std::string err;
  std::vector<float> wk_keep[2], bias_keep[2];
  for (int i = 0; i < nl; ++i) {
    Layer L;
    L.spec = specs[i];
    const int p = (L.spec.k - 1) / 2;
    L.Hin = H; L.Win = W;
    L.Ho = (H + 2 * p - L.spec.k) / L.spec.stride + 1;
    L.Wo = (W + 2 * p - L.spec.k) / L.spec.stride + 1;
    L.in = cur;
    const int next_pad = i + 1 < nl ? (specs[i + 1].k - 1) / 2 : 0;
    rc = make_tensor(h, L.out, i == 0 && try_fuse ? small_cap : h->cap, L.Ho, L.Wo, L.spec.cout, next_pad);
    if (rc) return rc;
    const std::string key = std::string(pre) + L.spec.name + ".0.";
    const HostTensor* wt = find(w, key + "weight", {L.spec.cout, L.spec.cin, L.spec.k, L.spec.k}, err);
    const HostTensor* bt = wt ? find(w, key + "bias", {L.spec.cout}, err) : nullptr;
    if (!bt) return h->fail(UAHN_ERR_WEIGHTS, "%s", err.c_str());
    const int K = L.spec.k * L.spec.k * L.spec.cin, kk = L.spec.k;
    std::vector<float> wk((size_t)K * L.spec.cout);
    for (int co = 0; co < L.spec.cout; ++co)
      for (int c = 0; c < L.spec.cin; ++c)
        for (int ky = 0; ky < kk; ++ky)
          for (int kx = 0; kx < kk; ++kx)
            wk[(size_t)((ky * kk + kx) * L.spec.cin + c) * L.spec.cout + co] =
                wt->data[(((size_t)co * L.spec.cin + c) * kk + ky) * kk + kx];
    if (h->bf16) {
      if (conv_bf16_prepare(L.wb, wk, bt->data, make_geom(L, 1), L.in, L.out, h->allocs, err))
        return h->fail(UAHN_ERR_UNSUPPORTED, "%s: %s", L.spec.name, err.c_str());
    } else {
      if ((rc = upload(h, &L.w_f32, wk))) return rc;
    }
    if ((rc = upload(h, &L.bias, bt->data))) return rc;
    if (try_fuse && i < 2) { wk_keep[i] = wk; bias_keep[i] = bt->data; }
    B.layers.push_back(L);
    cur = L.out;
    H = L.Ho; W = L.Wo;
  }
  if (try_fuse) {
    if (conv_fused_prepare(B.fused, wk_keep[0], bias_keep[0], wk_keep[1], bias_keep[1], make_geom(B.layers[0], 1),
                           make_geom(B.layers[1], 1), B.x, h->allocs, err) < 0)
      return h->fail(UAHN_ERR_CUDA, "fused front of block %d: %s", id, err.c_str());
    if (!B.fused.enabled) return h->fail(UAHN_ERR_UNSUPPORTED, "fused front of block %d not available", id);
  }
  if (H != 4 || W != 5 || specs[nl - 1].cout != 256) return h->fail(UAHN_ERR_INVALID, "block %d does not end at 256x4x5", id);
  if (id != 4) {
    const std::string key = std::string(P1) + "fc_block_" + std::to_string(id) + ".";
    const HostTensor* wt = find(w, key + "weight", {8, FC_IN}, err);
    const HostTensor* bt = wt ? find(w, key + "bias", {8}, err) : nullptr;
    if (!bt) return h->fail(UAHN_ERR_WEIGHTS, "%s", err.c_str());
    if ((rc = upload(h, &B.W8, permute_fc_in(*wt)))) return rc;
    if ((rc = upload(h, &B.b8, bt->data))) return rc;
  }
  return UAHN_OK;
}

int build_head(uahn_handle* h, const std::map<std::string, HostTensor>& w) {
  std::string err;
  int rc;
  struct { const char* name; float** W1; float** b1; float** W2; float** b2; ConvBf16Weights* wb; void** plain; } heads[2] = {
      {"fc_block_4_mean", &h->W1m, &h->b1m, &h->W2m, &h->b2m, &h->W1m_b, &h->W1m_plain},
      {"fc_block_4_uncertainty", &h->W1u, &h->b1u, &h->W2u, &h->b2u, &h->W1u_b, &h->W1u_plain}};
  for (auto& hd : heads) {
    const std::string key = std::string(P4) + hd.name;
    const HostTensor* w1 = find(w, key + ".1.weight", {FC_HID, FC_IN}, err);
    const HostTensor* b1 = w1 ? find(w, key + ".1.bias", {FC_HID}, err) : nullptr;
    const HostTensor* w2 = b1 ? find(w, key + ".4.weight", {8, FC_HID}, err) : nullptr;
    const HostTensor* b2 = w2 ? find(w, key + ".4.bias", {8}, err) : nullptr;
    if (!b2) return h->fail(UAHN_ERR_WEIGHTS, "%s", err.c_str());
    std::vector<float> perm = permute_fc_in(*w1);           // [256][5120 NHWC]
    std::vector<float> wk((size_t)FC_IN * FC_HID);          // [K][Cout]
    for (int j = 0; j < FC_HID; ++j)
      for (int k = 0; k < FC_IN; ++k) wk[(size_t)k * FC_HID + j] = perm[(size_t)j * FC_IN + k];
    if (h->bf16) {
      Tensor tin{}, tout{};
      if (conv_bf16_prepare(*hd.wb, wk, b1->data, dense_geom(1, FC_IN, FC_HID, 1), tin, tout, h->allocs, err))
        return h->fail(UAHN_ERR_UNSUPPORTED, "%s: %s", hd.name, err.c_str());
      std::vector<uint16_t> plain(perm.size());
      for (size_t i = 0; i < perm.size(); ++i) plain[i] = f32_to_bf16_host(perm[i]);
      uint16_t* dp = nullptr;
      if ((rc = dev_alloc(h, &dp, plain.size(), false))) return rc;
      CK(cudaMemcpy(dp, plain.data(), plain.size() * 2, cudaMemcpyHostToDevice));
      *hd.plain = dp;
    } else {
      if ((rc = upload(h, hd.W1, wk))) return rc;
    }
    if ((rc = upload(h, hd.b1, b1->data))) return rc;
    if ((rc = upload(h, hd.W2, w2->data))) return rc;
    if ((rc = upload(h, hd.b2, b2->data))) return rc;
  }
  return UAHN_OK;
}

template <typename T>
int run_conv(uahn_handle* h, Layer& L, int n) {
  ConvGeom g = make_geom(L, n);
  if constexpr (sizeof(T) == 4) {
    LAUNCH(launch_conv_f32((const float*)L.in.p, L.w_f32, L.bias, (float*)L.out.p, g, h->stream, n <= F32_SPLITK_MAX_PAIRS ? h->f32_ws : nullptr,
                           h->f32_ws_floats, L.Ho * L.Wo));
    h->launches += conv_f32_extra_launches();
  } else {
    LAUNCH(launch_conv_bf16(L.wb, L.in.p, L.bias, L.out.p, g, h->stream));
  }
  return UAHN_OK;
}

// warp + concat + pool -> conv stack of one cascade block: the warp, then either the fused front (convs 0 and 1) and
// layers 2.. or every layer in order.
template <typename T>
int run_block(uahn_handle* h, Block& B, int n, const uint8_t* prev, const uint8_t* curr, const float* Hcur,
              const WarpCells* cells = nullptr) {
  cudaStream_t st = h->stream;
  int rc;
  const size_t nl = B.layers.size();
  h->prof_begin(0);
  LAUNCH(launch_warp_concat_pool<T>(prev, curr, Hcur, B.x, B.pool, n, st, cells));
  h->prof_end();
  h->prof_begin(1);
  size_t first = 0;
  if constexpr (sizeof(T) == 2) {
    if (B.fused.enabled) {
      LAUNCH(launch_conv_fused(B.fused, B.layers[1].out.p, make_geom(B.layers[1], n), n, h->num_sms, st));
      first = 2;
    }
  }
  for (size_t i = first; i < nl; ++i)
    if ((rc = run_conv<T>(h, B.layers[i], n))) return rc;
  h->prof_end();
  return UAHN_OK;
}

template <typename T>
int forward(uahn_handle* h, int n, const uint8_t* prev, const uint8_t* curr, const float* prior, const uahn_rng* rng,
            const uint8_t* d_masks, float* mean, float* cov, float* err, const uint64_t* rng_dev = nullptr,
            uint8_t* err_u8 = nullptr) {
  cudaStream_t st = h->stream;
  const int variant = h->cfg.variant;
  const float* Hcur = nullptr;
  int rc;
  g_pdl_on = true;
  if (variant != UAHN_VARIANT_FULL) {
    if (!prior) return h->fail(UAHN_ERR_INVALID, "this variant needs a prior");
    h->prof_begin(3);
    LAUNCH(launch_dlt(n, prior, nullptr, h->Hb[0], st));                   // model_to_trace.py:129-130
    h->prof_end();
    Hcur = h->Hb[0];
  }
  // bf16, above the latency path: the warps gather their taps through the texture unit from a cell array of the current
  // frames (image_kernels.cu), filled here once per call; charged to the warp stage
  const WarpCells* cells = nullptr;
  if (sizeof(T) == 2 && h->cells.arr && n > WARP_TEX_MIN_PAIRS && n <= h->cells.cap) {
    h->prof_begin(0);
    LAUNCH(launch_warp_cells_fill(h->cells, curr, n, st));
    h->prof_end();
    cells = &h->cells;
  }
  for (int b = 1; b <= 3; ++b) {
    Block& B = h->blocks[b];
    if (!B.active) continue;
    // block 1 sees the raw current image (model_to_trace.py:138-139); blocks 2,3 the warped one (:154,172)
    if ((rc = run_block<T>(h, B, n, prev, curr, b == 1 ? nullptr : Hcur, cells))) return rc;
    h->prof_begin(3);
    LAUNCH(launch_fc8_dlt<T>(n, (const T*)B.layers.back().out.p, B.W8, B.b8, b == 1 ? nullptr : Hcur, h->Hb[b],
                             h->dblk[b], st));
    h->prof_end();
    Hcur = h->Hb[b];
  }
  Block& B4 = h->blocks[4];
  if ((rc = run_block<T>(h, B4, n, prev, curr, Hcur, cells))) return rc;      // model_to_trace.py:261-263
  const T* feat = (const T*)B4.layers.back().out.p;
  const uint64_t seed = rng ? rng->seed : 0, first = rng ? rng->first_pair_index : 0;
  // bf16, large batches: the dropout expansion is fused into the GEMM's A producer and only the keep BITS (20 KB per
  // pair) are staged.  Small batches (the batch-1 latency path) and fp32 mode materialise the masked features: with one
  // or two M tiles the fused producer is a serial latency chain (80 K-stages per tile) and the plain GEMM, split over N
  // tiles, finishes sooner.
  const bool fused_mc = sizeof(T) == 2 && n >= MC_FUSED_MIN_PAIRS;
  if (sizeof(T) == 2 && n <= MC_SMALL_MAX_PAIRS && !getenv("UAHN_NO_MC_SMALL_FUSED")) {
    // latency path: dropout expansion + first layer of both heads in ONE CUDA-core kernel (was expand + 2 launches)
    h->prof_begin(2);
    LAUNCH(launch_mc_fc1_small_fused(n, feat, h->W1m_plain, h->W1u_plain, h->b1m, h->b1u, h->hid, d_masks, seed, first, rng_dev, st));
    h->prof_end();
  } else if (!fused_mc) {
    h->prof_begin(3);
    LAUNCH(launch_mc_expand<T>(n, feat, (T*)h->mcA, d_masks, seed, first, rng_dev, st));
    h->prof_end();
    h->prof_begin(2);
    for (int head = 0; head < 2; ++head) {
      ConvGeom g = dense_geom(n * MC, FC_IN, FC_HID, 1);
      const T* a = (const T*)h->mcA + (size_t)head * n * MC * FC_IN;
      T* o = (T*)h->hid + (size_t)head * n * MC * FC_HID;
      if constexpr (sizeof(T) == 4) {
        LAUNCH(launch_conv_f32((const float*)a, head ? h->W1u : h->W1m, head ? h->b1u : h->b1m, (float*)o, g, st,
                               n <= F32_SPLITK_MAX_PAIRS ? h->f32_ws : nullptr, h->f32_ws_floats, MC));
        h->launches += conv_f32_extra_launches();
      } else if (n <= MC_SMALL_MAX_PAIRS) {     // latency path: CUDA-core kernel, 64 CTAs per pair and head
        LAUNCH(launch_mc_fc1_small(n, a, head ? h->W1u_plain : h->W1m_plain, head ? h->b1u : h->b1m, o, st));
      } else {
        LAUNCH(launch_conv_bf16(head ? h->W1u_b : h->W1m_b, a, head ? h->b1u : h->b1m, o, g, st));
      }
    }
    h->prof_end();
  } else {
    h->prof_begin(3);
    LAUNCH(launch_mc_maskbits(n, (uint8_t*)h->mcA, d_masks, seed, first, rng_dev, st));
    h->prof_end();
    h->prof_begin(2);
    for (int head = 0; head < 2; ++head) {
      const uint8_t* bits = (const uint8_t*)h->mcA + (size_t)head * n * (FC_IN / 8) * MC;
      T* o = (T*)h->hid + (size_t)head * n * MC * FC_HID;
      LAUNCH(launch_mc_gemm_bf16(head ? h->W1u_b : h->W1m_b, feat, bits, o, n, st));
    }
    h->prof_end();
  }
  const bool want_err = h->cfg.show_error && (err || err_u8);
  h->prof_begin(3);
  LAUNCH(launch_mc_final<T>(n, (const T*)h->hid, h->W2m, h->b2m, h->W2u, h->b2u, Hcur, d_masks, seed, first, rng_dev, mean, cov,
                            h->cfg.show_error ? h->Htot : nullptr, h->mc_mean, h->mc_logvar, st));
  h->prof_end();
  if (want_err) {
    h->prof_begin(0);
    LAUNCH(launch_warp_plain(prev, curr, h->Htot, err_u8 ? nullptr : err, err_u8, nullptr, nullptr, 1, n, st, sizeof(T) == 2));
    h->prof_end();
  }
  h->last_n = n;
  return UAHN_OK;
}

int forward_any(uahn_handle* h, int n, const uint8_t* prev, const uint8_t* curr, const float* prior,
                const uahn_rng* rng, const uint8_t* d_masks, float* mean, float* cov, float* err,
                const uint64_t* rng_dev = nullptr, uint8_t* err_u8 = nullptr) {
  if (n <= 0 || n > h->cap) return h->fail(UAHN_ERR_INVALID, "n=%d outside [1, max_batch=%d]", n, h->cap);
  return h->bf16 ? forward<__nv_bfloat16>(h, n, prev, curr, prior, rng, d_masks, mean, cov, err, rng_dev, err_u8)
                 : forward<float>(h, n, prev, curr, prior, rng, d_masks, mean, cov, err, rng_dev, err_u8);
}

}  // namespace

// ------------------------------------------------------------------------------------------------------
extern "C" {

int uahn_create(const uahn_config* cfg, uahn_handle** out) {
  if (!cfg || !out || !cfg->weights_path) { g_create_error = "null config / weights_path"; return UAHN_ERR_INVALID; }
  if (cfg->variant < UAHN_VARIANT_AUTO || cfg->variant > 3 || cfg->precision < 0 || cfg->precision > 1 || cfg->max_batch < 1) {
    g_create_error = "invalid variant / precision / max_batch";
    return UAHN_ERR_INVALID;
  }
  uahn_handle* h = new uahn_handle();
  h->cfg = *cfg;
  h->cap = cfg->max_batch;
  h->bf16 = cfg->precision == UAHN_PRECISION_BF16;
  h->es = h->bf16 ? 2 : 4;
  auto bail = [&](int rc) {
    g_create_error = h->last_error;
    uahn_destroy(h);
    return rc;
  };
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    h->fail(UAHN_ERR_CUDA, "no CUDA device: %s — this library has no CPU fallback", cudaGetErrorString(e));
    return bail(UAHN_ERR_CUDA);
  }
  if ((e = cudaSetDevice(cfg->device)) != cudaSuccess) {
    h->fail(UAHN_ERR_CUDA, "cudaSetDevice(%d): %s", cfg->device, cudaGetErrorString(e));
    return bail(UAHN_ERR_CUDA);
  }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, cfg->device);
  h->num_sms = prop.multiProcessorCount;
  if (prop.major != 10) {
    h->fail(UAHN_ERR_UNSUPPORTED, "device sm_%d%d: kernels are built for sm_100a only", prop.major, prop.minor);
    return bail(UAHN_ERR_UNSUPPORTED);
  }
  if (cfg->stream) {
    h->stream = (cudaStream_t)cfg->stream;
  } else {
    if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) {
      h->fail(UAHN_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
      return bail(UAHN_ERR_CUDA);
    }
    h->own_stream = true;
  }
  if ((e = init_keep_alias_table()) != cudaSuccess) {
    h->fail(UAHN_ERR_CUDA, "keep-byte alias table upload: %s", cudaGetErrorString(e));
    return bail(UAHN_ERR_CUDA);
  }
  std::map<std::string, HostTensor> w;
  std::string err;
  bool loaded = false;
  try {
    loaded = load_weight_file(cfg->weights_path, w, err);
  } catch (const std::exception& ex) {
    err = std::string("weights file: ") + ex.what();
  }
  if (!loaded) {
    h->fail(UAHN_ERR_WEIGHTS, "%s", err.c_str());
    return bail(UAHN_ERR_WEIGHTS);
  }
  // UAHN_VARIANT_AUTO: the exporter recorded which traced graph the file came from (weights.export_torchscript)
  if (h->cfg.variant == UAHN_VARIANT_AUTO) {
    auto it = w.find("__meta__.variant");
    if (it == w.end() || it->second.data.size() != 1 || it->second.data[0] < 0 || it->second.data[0] > 3) {
      h->fail(UAHN_ERR_WEIGHTS, "UAHN_VARIANT_AUTO: the weights file carries no variant record");
      return bail(UAHN_ERR_WEIGHTS);
    }
    h->cfg.variant = (int)it->second.data[0];
  }
  if (h->cfg.show_error == UAHN_SHOW_ERROR_AUTO) {
    auto it = w.find("__meta__.show_error");
    h->cfg.show_error = (it != w.end() && it->second.data.size() == 1 && it->second.data[0] != 0.f) ? 1 : 0;
  }
  int rc = UAHN_OK;
  const int v = h->cfg.variant;
  if (v == UAHN_VARIANT_FULL && (rc = build_block(h, w, 1, B1, 3, 8))) return bail(rc);
  if ((v == UAHN_VARIANT_FULL || v == UAHN_VARIANT_PRIOR3) && (rc = build_block(h, w, 2, B2, 4, 4))) return bail(rc);
  if (v != UAHN_VARIANT_PRIOR1 && (rc = build_block(h, w, 3, B3, 6, 2))) return bail(rc);
  if ((rc = build_block(h, w, 4, B4, 7, 1))) return bail(rc);
  if ((rc = build_head(h, w))) return bail(rc);
  const size_t cap = h->cap;
  uint8_t* p8 = nullptr;
  {
    const size_t expand_pairs = h->bf16 ? std::min<size_t>(cap, MC_FUSED_MIN_PAIRS - 1) : cap;   // pairs on the expand path
    const size_t bytes = std::max<size_t>(2 * expand_pairs * MC * FC_IN * h->es, h->bf16 ? 2 * cap * (FC_IN / 8) * MC : 0);
    if ((rc = dev_alloc(h, &p8, bytes))) return bail(rc);
  }
  h->mcA = p8;
  if ((rc = dev_alloc(h, &p8, 2 * cap * MC * FC_HID * h->es))) return bail(rc);
  h->hid = p8;
  for (int i = 0; i < 4; ++i) {
    if ((rc = dev_alloc(h, &h->Hb[i], cap * 9))) return bail(rc);
    if ((rc = dev_alloc(h, &h->dblk[i], cap * 8))) return bail(rc);
  }
  if ((rc = dev_alloc(h, &h->Htot, cap * 9))) return bail(rc);
  if (!h->bf16) {   // splits * M * Cout <= num_sms * 64 * 64 * pairs by construction (conv_f32.cu)
    h->f32_ws_floats = (size_t)h->num_sms * 64 * 64 * F32_SPLITK_MAX_PAIRS;
    if ((rc = dev_alloc(h, &h->f32_ws, h->f32_ws_floats, false))) return bail(rc);
  }
  if ((rc = dev_alloc(h, &h->mc_mean, cap * MC * 8))) return bail(rc);
  if ((rc = dev_alloc(h, &h->mc_logvar, cap * MC * 8))) return bail(rc);
  if ((rc = dev_alloc(h, &h->d_prev, cap * IMG_PIXELS))) return bail(rc);
  if ((rc = dev_alloc(h, &h->d_curr, cap * IMG_PIXELS))) return bail(rc);
  if (h->bf16 && h->cap > WARP_TEX_MIN_PAIRS && h->cap <= warp_cells_capacity() && !getenv("UAHN_NO_TEX_WARP")) {
    if ((e = warp_cells_create(h->cells, h->cap, h->stream)) != cudaSuccess) {
      h->fail(UAHN_ERR_CUDA, "cell array of the texture-gather warp (%d images): %s", h->cap, cudaGetErrorString(e));
      return bail(UAHN_ERR_CUDA);
    }
  }
  if ((rc = dev_alloc(h, &h->d_prior, cap * 8))) return bail(rc);
  if ((rc = dev_alloc(h, &h->d_mean, cap * 8))) return bail(rc);
  if ((rc = dev_alloc(h, &h->d_cov, cap * 64))) return bail(rc);
  if (h->cfg.show_error && (rc = dev_alloc(h, &h->d_err, cap * IMG_PIXELS))) return bail(rc);
  if ((rc = dev_alloc(h, &h->d_ring, (size_t)2 * IMG_PIXELS))) return bail(rc);
  if ((rc = dev_alloc(h, &h->d_rng, 2 + 4))) return bail(rc);
  h->d_in1_prior = reinterpret_cast<float*>(h->d_rng + 2);
  if ((rc = dev_alloc(h, &h->d_out1, 72))) return bail(rc);
  h->use_graph = getenv("UAHN_NO_GRAPH") == nullptr;
  if ((e = cudaMallocHost((void**)&h->h_rng, 48)) != cudaSuccess ||
      (e = cudaMallocHost((void**)&h->h_img, IMG_PIXELS)) != cudaSuccess ||
      (e = cudaMallocHost((void**)&h->h_out, (72 + IMG_PIXELS) * sizeof(float))) != cudaSuccess) {
    h->fail(UAHN_ERR_CUDA, "cudaMallocHost: %s", cudaGetErrorString(e));
    return bail(UAHN_ERR_CUDA);
  }
  h->h_prior = reinterpret_cast<float*>(h->h_rng + 2);
  if ((e = cudaDeviceSynchronize()) != cudaSuccess) {
    h->fail(UAHN_ERR_CUDA, "setup: %s", cudaGetErrorString(e));
    return bail(UAHN_ERR_CUDA);
  }
  *out = h;
  return UAHN_OK;
}

void uahn_destroy(uahn_handle* h) {
  if (!h) return;
  int prev_dev = -1;                       // the array / texture / surface objects belong to the handle's device
  cudaGetDevice(&prev_dev);
  cudaSetDevice(h->cfg.device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (void* p : h->allocs) cudaFree(p);
  warp_cells_destroy(h->cells);
  for (auto& sp : h->prof_spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
  for (cudaEvent_t e : h->prof_pool) cudaEventDestroy(e);
  if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
  for (int i = 0; i < 2; ++i) { if (h->ev_in[i]) cudaEventDestroy(h->ev_in[i]); if (h->ev_done[i]) cudaEventDestroy(h->ev_done[i]); }
  for (cudaGraphExec_t g : h->graphs) if (g) cudaGraphExecDestroy(g);
  if (h->h_rng) cudaFreeHost(h->h_rng);
  if (h->h_img) cudaFreeHost(h->h_img);
  if (h->h_raw) cudaFreeHost(h->h_raw);
  if (h->h_out) cudaFreeHost(h->h_out);
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  delete h;
  if (prev_dev >= 0) cudaSetDevice(prev_dev);
}

const char* uahn_last_error(const uahn_handle* h) { return h ? h->last_error.c_str() : g_create_error.c_str(); }
int uahn_synchronize(uahn_handle* h) {
  if (!h) return UAHN_ERR_INVALID;
  CK(cudaStreamSynchronize(h->stream));
  return UAHN_OK;
}
void* uahn_stream(uahn_handle* h) { return h ? (void*)h->stream : nullptr; }
uint64_t uahn_launch_count(const uahn_handle* h) { return h ? h->launches : 0; }
double uahn_latest_inference_time(const uahn_handle* h) { return h ? h->latest_time : -1.0; }
int uahn_image_count(const uahn_handle* h) { return h ? h->img_counter : 0; }

int uahn_infer_batch_device(uahn_handle* h, int n, const uint8_t* prev, const uint8_t* curr, const float* prior,
                            const uahn_rng* rng, float* mean, float* cov, float* err) {
  if (!h) return UAHN_ERR_INVALID;
  if (!prev || !curr || !mean || !cov) return h->fail(UAHN_ERR_INVALID, "null buffer");
  if (err && !h->cfg.show_error) return h->fail(UAHN_ERR_INVALID, "err requested but handle created with show_error=0");
  CK(cudaSetDevice(h->cfg.device));
  return forward_any(h, n, prev, curr, prior, rng, rng ? rng->keep_masks : nullptr, mean, cov, err);
}

int uahn_infer_batch(uahn_handle* h, int n, const uint8_t* prev, const uint8_t* curr, const float* prior,
                     const uahn_rng* rng, float* mean, float* cov, float* err) {
  if (!h) return UAHN_ERR_INVALID;
  if (!prev || !curr || !mean || !cov) return h->fail(UAHN_ERR_INVALID, "null buffer");
  if (n <= 0 || n > h->cap) return h->fail(UAHN_ERR_INVALID, "n=%d outside [1, max_batch=%d]", n, h->cap);
  if (err && !h->cfg.show_error) return h->fail(UAHN_ERR_INVALID, "err requested but handle created with show_error=0");
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = h->stream;
  CK(cudaMemcpyAsync(h->d_prev, prev, (size_t)n * IMG_PIXELS, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(h->d_curr, curr, (size_t)n * IMG_PIXELS, cudaMemcpyHostToDevice, st));
  if (prior) CK(cudaMemcpyAsync(h->d_prior, prior, (size_t)n * 8 * 4, cudaMemcpyHostToDevice, st));
  const uint8_t* dm = nullptr;
  if (rng && rng->keep_masks) {
    if (!h->d_masks) {
      int rc = dev_alloc(h, &h->d_masks, (size_t)h->cap * UAHN_MASK_BYTES_PER_PAIR, false);
      if (rc) return rc;
    }
    CK(cudaMemcpyAsync(h->d_masks, rng->keep_masks, (size_t)n * UAHN_MASK_BYTES_PER_PAIR, cudaMemcpyHostToDevice, st));
    dm = h->d_masks;
  }
  int rc = forward_any(h, n, h->d_prev, h->d_curr, prior ? h->d_prior : nullptr, rng, dm, h->d_mean, h->d_cov,
                       err ? h->d_err : nullptr);
  if (rc) return rc;
  CK(cudaMemcpyAsync(mean, h->d_mean, (size_t)n * 8 * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(cov, h->d_cov, (size_t)n * 64 * 4, cudaMemcpyDeviceToHost, st));
  if (err) CK(cudaMemcpyAsync(err, h->d_err, (size_t)n * IMG_PIXELS * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return UAHN_OK;
}

namespace {
// copy stream, events and the second staging set of the pipelined entry points
int ensure_pipeline(uahn_handle* h) {
  if (h->pipeline_ready) return UAHN_OK;
  // a failure part-way leaves pipeline_ready false: the next submission retries only what is still missing
  if (!h->copy_stream) CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    if (!h->ev_in[i]) CK(cudaEventCreateWithFlags(&h->ev_in[i], cudaEventDisableTiming));
    if (!h->ev_done[i]) CK(cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming));
  }
  h->s_prev[0] = h->d_prev; h->s_curr[0] = h->d_curr; h->s_prior[0] = h->d_prior;
  h->s_mean[0] = h->d_mean; h->s_cov[0] = h->d_cov;
  int rc;
  if (!h->s_prev[1] && (rc = dev_alloc(h, &h->s_prev[1], (size_t)h->cap * IMG_PIXELS))) return rc;
  if (!h->s_curr[1] && (rc = dev_alloc(h, &h->s_curr[1], (size_t)h->cap * IMG_PIXELS))) return rc;
  if (!h->s_prior[1] && (rc = dev_alloc(h, &h->s_prior[1], (size_t)h->cap * 8))) return rc;
  if (!h->s_mean[1] && (rc = dev_alloc(h, &h->s_mean[1], (size_t)h->cap * 8))) return rc;
  if (!h->s_cov[1] && (rc = dev_alloc(h, &h->s_cov[1], (size_t)h->cap * 64))) return rc;
  h->pipeline_ready = true;
  return UAHN_OK;
}

// One pipelined submission.  frames == nullptr: n independent pairs from prev / curr.  frames != nullptr: n + 1
// consecutive frames, pair i = (frames[i], frames[i+1]) — each frame crosses PCIe once.
int submit(uahn_handle* h, int n, const uint8_t* prev, const uint8_t* curr, const uint8_t* frames, const float* prior,
           const uahn_rng* rng, float* mean, float* cov) {
  if (n <= 0 || n > h->cap) return h->fail(UAHN_ERR_INVALID, "n=%d outside [1, max_batch=%d]", n, h->cap);
  if (rng && rng->keep_masks) return h->fail(UAHN_ERR_UNSUPPORTED, "explicit masks are not supported by the pipelined entry points");
  if (h->cfg.variant != UAHN_VARIANT_FULL && !prior) return h->fail(UAHN_ERR_INVALID, "this variant needs a prior");
  CK(cudaSetDevice(h->cfg.device));
  int rc = ensure_pipeline(h);
  if (rc) return rc;
  if (frames && !h->s_frames[0])
    for (int i = 0; i < 2; ++i)
      if ((rc = dev_alloc(h, &h->s_frames[i], (size_t)(h->cap + 1) * IMG_PIXELS))) return rc;
  const int k = (int)(h->submit_count & 1);
  cudaStream_t cs = h->copy_stream, st = h->stream;
  CK(cudaStreamWaitEvent(cs, h->ev_done[k], 0));   // staging set k is free again (never-recorded events are complete)
  const uint8_t *dp, *dc;
  if (frames) {
    CK(cudaMemcpyAsync(h->s_frames[k], frames, (size_t)(n + 1) * IMG_PIXELS, cudaMemcpyHostToDevice, cs));
    dp = h->s_frames[k];
    dc = h->s_frames[k] + IMG_PIXELS;
  } else {
    CK(cudaMemcpyAsync(h->s_prev[k], prev, (size_t)n * IMG_PIXELS, cudaMemcpyHostToDevice, cs));
    CK(cudaMemcpyAsync(h->s_curr[k], curr, (size_t)n * IMG_PIXELS, cudaMemcpyHostToDevice, cs));
    dp = h->s_prev[k];
    dc = h->s_curr[k];
  }
  if (prior) CK(cudaMemcpyAsync(h->s_prior[k], prior, (size_t)n * 8 * 4, cudaMemcpyHostToDevice, cs));
  CK(cudaEventRecord(h->ev_in[k], cs));
  CK(cudaStreamWaitEvent(st, h->ev_in[k], 0));
  rc = forward_any(h, n, dp, dc, prior ? h->s_prior[k] : nullptr, rng, nullptr, h->s_mean[k], h->s_cov[k], nullptr);
  if (rc) return rc;
  CK(cudaMemcpyAsync(mean, h->s_mean[k], (size_t)n * 8 * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(cov, h->s_cov[k], (size_t)n * 64 * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaEventRecord(h->ev_done[k], st));
  ++h->submit_count;
  return UAHN_OK;
}
}  // namespace

int uahn_submit_batch(uahn_handle* h, int n, const uint8_t* prev, const uint8_t* curr, const float* prior,
                      const uahn_rng* rng, float* mean, float* cov) {
  if (!h) return UAHN_ERR_INVALID;
  if (!prev || !curr || !mean || !cov) return h->fail(UAHN_ERR_INVALID, "null buffer");
  return submit(h, n, prev, curr, nullptr, prior, rng, mean, cov);
}

int uahn_submit_sequence(uahn_handle* h, int n_frames, const uint8_t* frames, const float* prior, const uahn_rng* rng,
                         float* mean, float* cov) {
  if (!h) return UAHN_ERR_INVALID;
  if (!frames || !mean || !cov) return h->fail(UAHN_ERR_INVALID, "null buffer");
  if (n_frames < 2) return h->fail(UAHN_ERR_STATE, "HNet cannot inference! Only has one image!");   // HomographyNet.cpp:155-158
  return submit(h, n_frames - 1, nullptr, nullptr, frames, prior, rng, mean, cov);
}

int uahn_wait(uahn_handle* h) {
  if (!h) return UAHN_ERR_INVALID;
  if (h->copy_stream) CK(cudaStreamSynchronize(h->copy_stream));
  CK(cudaStreamSynchronize(h->stream));
  return UAHN_OK;
}

int uahn_load_image(uahn_handle* h, const uint8_t* gray, int rows, int cols, size_t stride, double time_stamp) {
  if (!h) return UAHN_ERR_INVALID;
  if (!gray || rows != IMG_H || cols != IMG_W || stride < (size_t)IMG_W)
    return h->fail(UAHN_ERR_INVALID, "image must be CV_8UC1 %dx%d (got %dx%d, stride %zu)", IMG_H, IMG_W, rows, cols, stride);
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaStreamSynchronize(h->stream));   // h_img may still be in flight from the previous frame
  for (int y = 0; y < IMG_H; ++y) memcpy(h->h_img + (size_t)y * IMG_W, gray + (size_t)y * stride, IMG_W);
  h->img_counter++;
  // prev <- curr is a slot flip, not a copy (HomographyNet.cpp:143 clones the tensor)
  h->ring_curr ^= 1;
  CK(cudaMemcpyAsync(h->d_ring + (size_t)h->ring_curr * IMG_PIXELS, h->h_img, IMG_PIXELS, cudaMemcpyHostToDevice, h->stream));
  if (h->img_counter >= 2) h->latest_time = time_stamp;   // HomographyNet.cpp:148
  return UAHN_OK;
}

int uahn_infer(uahn_handle* h, const double* prior_px, const uahn_rng* rng, double* mean8, double* cov64,
               uint8_t* err_map) {
  if (!h) return UAHN_ERR_INVALID;
  if (h->img_counter < 2) return h->fail(UAHN_ERR_STATE, "HNet cannot inference! Only has one image!");
  if (!mean8 || !cov64) return h->fail(UAHN_ERR_INVALID, "null output");
  if (err_map && !h->cfg.show_error) return h->fail(UAHN_ERR_INVALID, "err_map requested but show_error=0");
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = h->stream;
  const bool need_prior = h->cfg.variant != UAHN_VARIANT_FULL;
  if (need_prior) {
    if (!prior_px) return h->fail(UAHN_ERR_INVALID, "this variant needs a prior");
    for (int i = 0; i < 8; ++i) h->h_prior[i] = (float)prior_px[i];        // HomographyNet.cpp:160-165 (.toType(kFloat))
  }
  // rng == NULL: like the reference, which draws fresh masks on every forward (model_to_trace.py:266-273), every call
  // gets its own Philox pair index from a per-handle counter
  h->h_rng[0] = rng ? rng->seed : 0;
  h->h_rng[1] = rng ? rng->first_pair_index : h->auto_pair++;
  const uint8_t* dm = nullptr;
  if (rng && rng->keep_masks) {
    if (!h->d_masks) {
      int rc = dev_alloc(h, &h->d_masks, (size_t)h->cap * UAHN_MASK_BYTES_PER_PAIR, false);
      if (rc) return rc;
    }
    CK(cudaMemcpyAsync(h->d_masks, rng->keep_masks, UAHN_MASK_BYTES_PER_PAIR, cudaMemcpyHostToDevice, st));
    dm = h->d_masks;
  }
  const uint8_t* curr = h->d_ring + (size_t)h->ring_curr * IMG_PIXELS;
  const uint8_t* prev = h->d_ring + (size_t)(h->ring_curr ^ 1) * IMG_PIXELS;
  // everything between the host buffers: prior + rng H2D, the forward, results D2H
  auto enqueue = [&]() -> int {
    CK(cudaMemcpyAsync(h->d_rng, h->h_rng, need_prior ? 48 : 16, cudaMemcpyHostToDevice, st));
    // the error map leaves the device already clamped and truncated to u8 (HomographyNet.cpp:201): 71 680 B of D2H
    // instead of 286 720 B of floats plus a host conversion loop
    int rc = forward_any(h, 1, prev, curr, need_prior ? h->d_in1_prior : nullptr, rng, dm, h->d_out1, h->d_out1 + 8, nullptr,
                         h->d_rng, err_map ? reinterpret_cast<uint8_t*>(h->d_err) : nullptr);
    if (rc) return rc;
    CK(cudaMemcpyAsync(h->h_out, h->d_out1, 72 * 4, cudaMemcpyDeviceToHost, st));
    if (err_map) CK(cudaMemcpyAsync(h->h_out + 72, h->d_err, (size_t)IMG_PIXELS, cudaMemcpyDeviceToHost, st));
    return UAHN_OK;
  };
  const int key = h->ring_curr | (dm ? 2 : 0) | (err_map ? 4 : 0);
  const bool graphable = h->use_graph && !h->prof_on && h->infer_calls >= 2;   // first calls run eagerly (lazy attributes)
  ++h->infer_calls;
  if (graphable && !h->graphs[key]) {
    const uint64_t l0 = h->launches;
    cudaGraph_t graph = nullptr;
    CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    int rc = enqueue();
    cudaError_t ce = cudaStreamEndCapture(st, &graph);
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (ce != cudaSuccess) return h->fail(UAHN_ERR_CUDA, "graph capture: %s", cudaGetErrorString(ce));
    ce = cudaGraphInstantiate(&h->graphs[key], graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) { h->graphs[key] = nullptr; return h->fail(UAHN_ERR_CUDA, "graph instantiate: %s", cudaGetErrorString(ce)); }
    h->graph_launches[key] = h->launches - l0;
    h->launches = l0;       // capture enqueued nothing; replays are counted below
  }
  if (graphable) {
    CK(cudaGraphLaunch(h->graphs[key], st));
    h->launches += h->graph_launches[key];
    h->last_n = 1;
  } else {
    int rc = enqueue();
    if (rc) return rc;
  }
  CK(cudaStreamSynchronize(st));
  for (int i = 0; i < 8; ++i) mean8[i] = h->h_out[i];
  for (int i = 0; i < 64; ++i) cov64[i] = h->h_out[8 + i];
  if (err_map) memcpy(err_map, h->h_out + 72, IMG_PIXELS);
  return UAHN_OK;
}

int uahn_set_undistort_maps(uahn_handle* h, int raw_rows, int raw_cols, const float* map1, const float* map2) {
  if (!h) return UAHN_ERR_INVALID;
  if (!map1 || !map2 || raw_rows < 2 || raw_cols < 2 || raw_rows > 32767 || raw_cols > 32767)
    return h->fail(UAHN_ERR_INVALID, "bad undistort maps / raw size %dx%d", raw_rows, raw_cols);
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaStreamSynchronize(h->stream));
  int rc;
  if (!h->d_map1) {
    if ((rc = dev_alloc(h, &h->d_map1, (size_t)IMG_PIXELS, false))) return rc;
    if ((rc = dev_alloc(h, &h->d_map2, (size_t)IMG_PIXELS, false))) return rc;
  }
  if ((size_t)raw_rows * raw_cols > (size_t)h->raw_rows * h->raw_cols) {
    if (h->h_raw) { cudaFreeHost(h->h_raw); h->h_raw = nullptr; }
    if ((rc = dev_alloc(h, &h->d_raw, (size_t)raw_rows * raw_cols, false))) return rc;
    CK(cudaMallocHost((void**)&h->h_raw, (size_t)raw_rows * raw_cols));
  }
  h->raw_rows = raw_rows; h->raw_cols = raw_cols;
  CK(cudaMemcpy(h->d_map1, map1, (size_t)IMG_PIXELS * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->d_map2, map2, (size_t)IMG_PIXELS * 4, cudaMemcpyHostToDevice));
  return UAHN_OK;
}

namespace {
int stage_raw(uahn_handle* h, const uint8_t* raw, int rows, int cols, size_t stride, uint8_t* d_out) {
  if (!h->d_map1) return h->fail(UAHN_ERR_STATE, "uahn_set_undistort_maps has not been called");
  if (!raw || rows != h->raw_rows || cols != h->raw_cols || stride < (size_t)cols)
    return h->fail(UAHN_ERR_INVALID, "raw image must be CV_8UC1 %dx%d (got %dx%d, stride %zu)", h->raw_rows, h->raw_cols, rows,
                   cols, stride);
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaStreamSynchronize(h->stream));   // h_raw may still be in flight from the previous frame
  for (int y = 0; y < rows; ++y) memcpy(h->h_raw + (size_t)y * cols, raw + (size_t)y * stride, cols);
  CK(cudaMemcpyAsync(h->d_raw, h->h_raw, (size_t)rows * cols, cudaMemcpyHostToDevice, h->stream));
  LAUNCH(launch_remap_u8(h->d_raw, rows, cols, (size_t)cols, 1, h->d_map1, h->d_map2, d_out, h->stream));
  return UAHN_OK;
}
}  // namespace

int uahn_load_raw_image(uahn_handle* h, const uint8_t* raw, int rows, int cols, size_t stride, double time_stamp) {
  if (!h) return UAHN_ERR_INVALID;
  // prev <- curr is a slot flip (HomographyNet.cpp:143); the remap writes straight into the new curr slot
  int rc = stage_raw(h, raw, rows, cols, stride, h->d_ring + (size_t)(h->ring_curr ^ 1) * IMG_PIXELS);
  if (rc) return rc;
  h->ring_curr ^= 1;
  h->img_counter++;
  if (h->img_counter >= 2) h->latest_time = time_stamp;   // HomographyNet.cpp:148
  return UAHN_OK;
}

int uahn_stage_undistort(uahn_handle* h, const uint8_t* raw, int rows, int cols, size_t stride, uint8_t* out) {
  if (!h || !out) return UAHN_ERR_INVALID;
  int rc = stage_raw(h, raw, rows, cols, stride, h->d_prev);
  if (rc) return rc;
  CK(cudaMemcpyAsync(out, h->d_prev, IMG_PIXELS, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return UAHN_OK;
}

int uahn_profile_enable(uahn_handle* h, int on) {
  if (!h) return UAHN_ERR_INVALID;
  CK(cudaStreamSynchronize(h->stream));
  for (auto& sp : h->prof_spans) { h->prof_pool.push_back(sp.a); h->prof_pool.push_back(sp.b); }
  h->prof_spans.clear();
  for (int i = 0; i < 4; ++i) { h->prof_ms[i] = 0; h->prof_launches[i] = 0; }
  h->prof_on = on != 0;
  return UAHN_OK;
}

int uahn_profile_read(uahn_handle* h, double* ms4, uint64_t* launches4) {
  if (!h || !ms4) return UAHN_ERR_INVALID;
  CK(cudaStreamSynchronize(h->stream));
  for (auto& sp : h->prof_spans) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, sp.a, sp.b));
    h->prof_ms[sp.cat] += ms;
    h->prof_launches[sp.cat] += sp.launches;
    h->prof_pool.push_back(sp.a);
    h->prof_pool.push_back(sp.b);
  }
  h->prof_spans.clear();
  for (int i = 0; i < 4; ++i) {
    ms4[i] = h->prof_ms[i];
    if (launches4) launches4[i] = h->prof_launches[i];
  }
  return UAHN_OK;
}

int uahn_philox_keep_masks(uint64_t seed, uint64_t pair_index, uint8_t* out) {
  if (!out) return UAHN_ERR_INVALID;
  static uint32_t tab[256];
  static const bool tab_ready = (build_keep_alias_table(tab), true);
  (void)tab_ready;
  for (int head = 0; head < 2; ++head)
    for (int s = 0; s < MC; ++s) {
      uint8_t* row = out + ((size_t)head * MC + s) * MASK_ROW;
      for (int k8 = 0; k8 < FC_IN / 8; ++k8) {
        const uint32_t bits = philox_keep8(seed, pair_index, head, 0, s, k8, tab);
        for (int j = 0; j < 8; ++j) {
          const int kp = k8 * 8 + j, hw = kp >> 8, c = kp & 255;   // kernel order -> reference order
          row[c * 20 + hw] = (bits >> j) & 1u;
        }
      }
      for (int j8 = 0; j8 < FC_HID / 8; ++j8) {
        const uint32_t bits = philox_keep8(seed, pair_index, head, 1, s, j8, tab);
        for (int j = 0; j < 8; ++j) row[FC_IN + j8 * 8 + j] = (bits >> j) & 1u;
      }
    }
  return UAHN_OK;
}

int uahn_stage_dlt(uahn_handle* h, int n, const float* offsets, float* Hout) {
  if (!h || !offsets || !Hout) return UAHN_ERR_INVALID;
  if (n <= 0 || n > h->cap) return h->fail(UAHN_ERR_INVALID, "n outside [1, max_batch]");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemcpyAsync(h->d_prior, offsets, (size_t)n * 32, cudaMemcpyHostToDevice, h->stream));
  LAUNCH(launch_dlt(n, h->d_prior, nullptr, h->Hb[0], h->stream));
  CK(cudaMemcpyAsync(Hout, h->Hb[0], (size_t)n * 36, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return UAHN_OK;
}

int uahn_stage_warp(uahn_handle* h, int n, const uint8_t* img, const float* Hm, float* out, int16_t* ix_nw,
                    int16_t* iy_nw) {
  if (!h || !img || !Hm || !out) return UAHN_ERR_INVALID;
  if (n <= 0 || n > h->cap) return h->fail(UAHN_ERR_INVALID, "n outside [1, max_batch]");
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = h->stream;
  struct Scratch {   // freed on every exit path
    float* out = nullptr; int16_t *ix = nullptr, *iy = nullptr;
    ~Scratch() { cudaFree(out); cudaFree(ix); cudaFree(iy); }
  } d;
  CK(cudaMalloc(&d.out, (size_t)n * IMG_PIXELS * 4));
  CK(cudaMalloc(&d.ix, (size_t)n * IMG_PIXELS * 2));
  CK(cudaMalloc(&d.iy, (size_t)n * IMG_PIXELS * 2));
  CK(cudaMemcpyAsync(h->d_curr, img, (size_t)n * IMG_PIXELS, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(h->Hb[0], Hm, (size_t)n * 36, cudaMemcpyHostToDevice, st));
  LAUNCH(launch_warp_plain(h->d_curr, h->d_curr, h->Hb[0], d.out, nullptr, d.ix, d.iy, 0, n, st, h->bf16));   // the handle's own coordinate mode
  CK(cudaMemcpyAsync(out, d.out, (size_t)n * IMG_PIXELS * 4, cudaMemcpyDeviceToHost, st));
  if (ix_nw) CK(cudaMemcpyAsync(ix_nw, d.ix, (size_t)n * IMG_PIXELS * 2, cudaMemcpyDeviceToHost, st));
  if (iy_nw) CK(cudaMemcpyAsync(iy_nw, d.iy, (size_t)n * IMG_PIXELS * 2, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return UAHN_OK;
}

// model_to_trace.py:18-38 + :311-317 alone: var, pts_w n x 8, Hp n x 9 (HOST) -> flow n x 8, cov n x 64
int uahn_stage_transfer(uahn_handle* h, int n, const float* var, const float* Hp, const float* pts_w, float* flow,
                        float* cov) {
  if (!h || !var || !Hp || !pts_w || !flow || !cov) return UAHN_ERR_INVALID;
  if (n <= 0 || n > h->cap) return h->fail(UAHN_ERR_INVALID, "n outside [1, max_batch]");
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = h->stream;
  // scratch: var -> dblk[1], pts_w -> dblk[2], Hp -> Hb[0]; results in the regular output staging
  CK(cudaMemcpyAsync(h->dblk[1], var, (size_t)n * 32, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(h->dblk[2], pts_w, (size_t)n * 32, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(h->Hb[0], Hp, (size_t)n * 36, cudaMemcpyHostToDevice, st));
  LAUNCH(launch_transfer(n, h->dblk[1], h->Hb[0], h->dblk[2], h->d_mean, h->d_cov, st));
  CK(cudaMemcpyAsync(flow, h->d_mean, (size_t)n * 32, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(cov, h->d_cov, (size_t)n * 256, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return UAHN_OK;
}

int uahn_variant(const uahn_handle* h) { return h ? h->cfg.variant : UAHN_ERR_INVALID; }
int uahn_show_error(const uahn_handle* h) { return h ? h->cfg.show_error : UAHN_ERR_INVALID; }

int uahn_stage_conv(uahn_handle* h, const char* layer, int n, const float* in_nchw) {
  if (!h || !layer || !in_nchw) return UAHN_ERR_INVALID;
  if (n <= 0 || n > h->cap) return h->fail(UAHN_ERR_INVALID, "n outside [1, max_batch]");
  CK(cudaSetDevice(h->cfg.device));
  Layer* L = nullptr;
  for (int b = 1; b <= 4 && !L; ++b)
    for (auto& l : h->blocks[b].layers)
      if (h->blocks[b].active && !strcmp(layer, l.spec.name)) L = &l;
  if (!L) return h->fail(UAHN_ERR_INVALID, "layer '%s' not in this variant", layer);
  const Tensor& t = L->in;
  if (n > t.N) return h->fail(UAHN_ERR_INVALID, "layer '%s' accepts at most %d images through this entry point", layer, t.N);
  std::vector<uint8_t> raw((size_t)n * t.pitch_n * h->es, 0);
  for (int i = 0; i < n; ++i)
    for (int c = 0; c < t.C; ++c)
      for (int y = 0; y < t.H; ++y)
        for (int x = 0; x < t.W; ++x) {
          const float v = in_nchw[(((size_t)i * t.C + c) * t.H + y) * t.W + x];
          const size_t dst = (size_t)t.off(i, y, x, c);
          if (h->bf16) {
            uint32_t u; memcpy(&u, &v, 4);
            u += 0x7fffu + ((u >> 16) & 1u);
            reinterpret_cast<uint16_t*>(raw.data())[dst] = (uint16_t)(u >> 16);
          } else {
            reinterpret_cast<float*>(raw.data())[dst] = v;
          }
        }
  CK(cudaMemcpyAsync(t.p, raw.data(), raw.size(), cudaMemcpyHostToDevice, h->stream));
  int rc = h->bf16 ? run_conv<__nv_bfloat16>(h, *L, n) : run_conv<float>(h, *L, n);
  if (rc) return rc;
  CK(cudaStreamSynchronize(h->stream));
  h->last_n = n;
  return UAHN_OK;
}

long uahn_debug_read(uahn_handle* h, const char* what, float* out, size_t capacity) {
  if (!h || !what || !out) return UAHN_ERR_INVALID;
  const int n = h->last_n;
  if (n <= 0) return h->fail(UAHN_ERR_STATE, "no batch has been run");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaStreamSynchronize(h->stream));
  const std::string w(what);
  auto copy_f32 = [&](const float* d, size_t count) -> long {
    if (count > capacity) return h->fail(UAHN_ERR_INVALID, "capacity too small (%zu needed)", count);
    if (cudaMemcpy(out, d, count * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return h->fail(UAHN_ERR_CUDA, "memcpy");
    return (long)count;
  };
  if (w.size() == 2 && w[0] == 'H' && w[1] >= '0' && w[1] <= '3') return copy_f32(h->Hb[w[1] - '0'], (size_t)n * 9);
  if (w == "Htot") return copy_f32(h->Htot, (size_t)n * 9);
  if (w.size() == 2 && w[0] == 'd' && w[1] >= '1' && w[1] <= '3') return copy_f32(h->dblk[w[1] - '0'], (size_t)n * 8);
  if (w == "mcmean") return copy_f32(h->mc_mean, (size_t)n * MC * 8);
  if (w == "mclogvar") return copy_f32(h->mc_logvar, (size_t)n * MC * 8);
  // tensors stored in the activation dtype: "feat<b>", "x<b>", "act:<layer name>"
  const Tensor* t = nullptr;
  bool nchw_flat = false;
  if (w.rfind("feat", 0) == 0 && w.size() == 5) {
    const int b = w[4] - '0';
    if (b < 1 || b > 4 || !h->blocks[b].active) return h->fail(UAHN_ERR_INVALID, "block not active");
    t = &h->blocks[b].layers.back().out;
    nchw_flat = true;
  } else if (w.rfind("x", 0) == 0 && w.size() == 2) {
    const int b = w[1] - '0';
    if (b < 1 || b > 4 || !h->blocks[b].active) return h->fail(UAHN_ERR_INVALID, "block not active");
    t = &h->blocks[b].x;
  } else if (w.rfind("act:", 0) == 0) {
    for (int b = 1; b <= 4 && !t; ++b)
      for (auto& L : h->blocks[b].layers)
        if (h->blocks[b].active && w.substr(4) == L.spec.name) t = &L.out;
  }
  if (!t) return h->fail(UAHN_ERR_INVALID, "unknown debug tensor '%s'", what);
  // the fused fronts of blocks 3 and 4 never write conv 0's output: its buffer holds only what uahn_stage_conv put there
  if (n > t->N) return h->fail(UAHN_ERR_STATE, "'%s' holds %d pairs; rerun with n <= %d to read it", what, t->N, t->N);
  const size_t count = (size_t)n * t->C * t->H * t->W;
  if (count > capacity) return h->fail(UAHN_ERR_INVALID, "capacity too small (%zu needed)", count);
  std::vector<uint8_t> raw((size_t)n * t->pitch_n * h->es);
  if (cudaMemcpy(raw.data(), t->p, raw.size(), cudaMemcpyDeviceToHost) != cudaSuccess) return h->fail(UAHN_ERR_CUDA, "memcpy");
  (void)nchw_flat;   // all activation reads are returned NCHW: [n][C][H][W]
  for (int i = 0; i < n; ++i)
    for (int c = 0; c < t->C; ++c)
      for (int y = 0; y < t->H; ++y)
        for (int x = 0; x < t->W; ++x) {
          const size_t src = (size_t)t->off(i, y, x, c);
          float v;
          if (h->bf16) {
            uint32_t bits = (uint32_t)reinterpret_cast<const uint16_t*>(raw.data())[src] << 16;
            memcpy(&v, &bits, 4);
          } else {
            v = reinterpret_cast<const float*>(raw.data())[src];
          }
          out[(((size_t)i * t->C + c) * t->H + y) * t->W + x] = v;
        }
  return (long)count;
}

}  // extern "C"

// what the filter bank (filter_bank.cu) needs of a handle
namespace uahn {
int handle_device(const uahn_handle* h) { return h->cfg.device; }
int handle_max_batch(const uahn_handle* h) { return h->cap; }
int handle_fail(uahn_handle* h, int code, const char* msg) { return h->fail(code, "%s", msg); }
}  // namespace uahn
