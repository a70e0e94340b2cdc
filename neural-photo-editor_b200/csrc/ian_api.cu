// ian_api.cu -- C-ABI of libian_b200.so (include/ian_b200.h): handle, weight preparation, per-batch
// plans (activation buffers in HBM + tap-GEMM descriptors + TMA maps) and the layer schedules of the three
// graphs -- IAN_simple (reference IAN_simple.py:56-241), IANv1.py and IAN.py -- for encode, decode, brush
// gradient, edit loop, paint stroke and the multi-GPU gather.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include <cuda.h>

#include "../../include/ian_b200.h"
#include "edge.h"
#include "tapgemm.h"

using namespace ian;

namespace {

thread_local std::string g_create_error;

// ------------------------------------------------------------------------------------------------
// host-side bf16 helpers (round-to-nearest-even), independent of device headers
// ------------------------------------------------------------------------------------------------
inline uint16_t f2bf(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);  // NaN
  const uint32_t r = 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)((u + r) >> 16);
}
inline float bf2f(uint16_t h) {
  uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

struct HostParam {
  std::vector<int64_t> shape;
  std::vector<float> data;
};

struct ParamSpec {
  const char* name;
  int ndim;
  int64_t shape[4];
};

// reference checkpoint names / shapes (IAN_simple.py layer names; SURVEY Appendix A)
const ParamSpec kSimpleWeights[] = {
    {"enc_conv1.W", 4, {128, 3, 5, 5}},    {"enc_conv1.b", 1, {128}},
    {"enc_conv2.W", 4, {256, 128, 5, 5}},  {"enc_conv3.W", 4, {512, 256, 5, 5}},
    {"enc_conv4.W", 4, {1024, 512, 5, 5}}, {"enc_fc1.W", 2, {16384, 1000}},
    {"enc_mu.W", 2, {1000, 100}},          {"enc_logsigma.W", 2, {1000, 100}},
    {"l_dec_fc2.W", 2, {100, 16384}},      {"dec_conv1.W", 4, {1024, 512, 5, 5}},
    {"dec_conv2.W", 4, {512, 256, 5, 5}},  {"dec_conv3.W", 4, {256, 128, 5, 5}},
    {"dec_out.W", 4, {128, 3, 5, 5}},
};
struct BnSpec { const char* name; int64_t c; };
const BnSpec kSimpleBn[] = {{"bnorm2", 256},       {"bnorm3", 512},     {"bnorm4", 1024},  {"bnorm_enc_fc1", 1000},
                            {"mu_bnorm", 100},     {"ls_bnorm", 100},   {"bnorm_dec_fc2", 16384},
                            {"bnorm_dc1", 512},    {"bnorm_dc2", 256},  {"bnorm_dc3", 128}};
const char* kBnFields[] = {"beta", "gamma", "mean", "inv_std"};

struct Spec { std::string name; std::vector<int64_t> shape; };

void add_bn(std::vector<Spec>& v, const std::string& name, int64_t c) {
  for (const char* f : kBnFields) v.push_back({name + "." + f, {c}});
}
void add_mdcl(std::vector<Spec>& v, const std::string& name, int64_t F, int64_t C, std::initializer_list<int> scales) {
  v.push_back({name + "W", {F, C, 3, 3}});
  v.push_back({name + "_coeff_base", {F}});
  for (int s : scales) v.push_back({name + (s == 0 ? std::string("_coeff_1x1") : "_coeff_" + std::to_string(s)), {F}});
}
void add_mdblock(std::vector<Spec>& v, const std::string& name, int64_t F, std::initializer_list<int> scales) {
  add_mdcl(v, name, F, F, scales);
  add_mdcl(v, name + "2", F, F, scales);
  add_bn(v, name + "bnorm0", F); add_bn(v, name + "bnorm1", F); add_bn(v, name + "bnorm2", F);
}

// parameter names / shapes of a model kind, in the reference's checkpoint naming (GANcheckpoints.py:11-30)
std::vector<Spec> spec_list(int kind) {
  std::vector<Spec> v;
  if (kind == IAN_MODEL_SIMPLE) {
    for (const auto& s : kSimpleWeights) v.push_back({s.name, std::vector<int64_t>(s.shape, s.shape + s.ndim)});
    for (const auto& b : kSimpleBn) add_bn(v, b.name, b.c);
    return v;
  }
  // IAN.py:67-207
  for (const auto& s : kSimpleWeights) {
    const std::string n = s.name;
    if (n.rfind("enc_", 0) == 0) v.push_back({n, std::vector<int64_t>(s.shape, s.shape + s.ndim)});
  }
  for (const char* b : {"bnorm2", "bnorm3", "bnorm4"}) add_bn(v, b, b[5] == '2' ? 256 : b[5] == '3' ? 512 : 1024);
  add_bn(v, "bnorm_enc_fc1", 1000); add_bn(v, "mu_bnorm", 100); add_bn(v, "ls_bnorm", 100);
  for (const char* m : {"l_IAF_mu", "l_IAF_ls"})
    for (const char* sub : {"_input", "_output_W", "_output_D"}) {
      v.push_back({std::string(m) + sub + ".W", {100, 100}});
      v.push_back({std::string(m) + sub + ".b", {100}});
    }
  if (kind == IAN_MODEL_V1) {                             // IANv1.py:125-201
    v.push_back({"l_dec_fc2.W", {100, 16384}}); v.push_back({"l_dec_fc2.b", {16384}});
    v.push_back({"dec_conv1.W", {1024, 512, 5, 5}}); add_bn(v, "bnorm_dc1", 512);
    v.push_back({"dec_conv2.W", {512, 256, 5, 5}}); add_bn(v, "bnorm_dc2", 256);
    v.push_back({"dec_conv3.W", {256, 128, 5, 5}}); add_bn(v, "bnorm_dc3", 128);
    v.push_back({"dec_conv4.W", {128, 64, 5, 5}}); add_bn(v, "bnorm_dc4", 64);
    add_mdcl(v, "R", 2, 64, {2, 3, 4}); add_mdcl(v, "G_a", 2, 64, {2, 3, 4}); add_mdcl(v, "G_b", 2, 2, {2, 3, 4});
    add_mdcl(v, "B_a", 2, 64, {2, 3, 4}); add_mdcl(v, "B_b", 2, 4, {2, 3, 4});
    return v;
  }
  v.push_back({"l_dec_fc2.W", {100, 8192}}); v.push_back({"l_dec_fc2.b", {8192}});
  v.push_back({"dec_conv1.W", {512, 512, 5, 5}});
  add_mdblock(v, "dec_conv2a", 512, {0, 2});
  v.push_back({"dec_conv2.W", {512, 256, 5, 5}});
  add_mdblock(v, "dec_conv3a", 256, {0, 2, 3});
  v.push_back({"dec_conv3.W", {256, 128, 5, 5}});
  add_mdblock(v, "dec_conv4a", 128, {0, 2, 3});
  v.push_back({"dec_conv4.W", {128, 128, 5, 5}});
  add_bn(v, "bnorm_dc4", 128);
  add_mdcl(v, "R", 2, 128, {2, 3, 4}); add_mdcl(v, "G_a", 2, 128, {2, 3, 4}); add_mdcl(v, "G_b", 2, 2, {2, 3, 4});
  add_mdcl(v, "B_a", 2, 128, {2, 3, 4}); add_mdcl(v, "B_b", 2, 4, {2, 3, 4});
  return v;
}

enum LayerId {
  L_ENC_CONV2 = 0, L_ENC_CONV3, L_ENC_CONV4, L_ENC_FC1, L_ENC_HEAD, L_DEC_FC2, L_DEC_CONV1, L_DEC_CONV2, L_DEC_CONV3,
  L_BWD_CONV3, L_BWD_CONV2, L_BWD_CONV1, L_BWD_FC2,
  // full IAN decoder (reference IAN.py:129-207)
  F_DEC_FC2, F_DEC_CONV1, F_MD1A, F_MD1B, F_DEC_CONV2, F_MD2A, F_MD2B, F_DEC_CONV3, F_MD3A, F_MD3B, F_DEC_CONV4, F_HEAD,
  // brush gradient through the IAN.py / IANv1.py decoders (T.grad at API.py:59,64 on those graphs)
  F_BWD_HEAD, F_BWD_CONV4, F_BWD_MD3B, F_BWD_MD3A, F_BWD_CONV3, F_BWD_MD2B, F_BWD_MD2A, F_BWD_CONV2, F_BWD_MD1B, F_BWD_MD1A,
  F_BWD_CONV1, F_BWD_FC2,
  L_COUNT,
  T_CONV1 = L_COUNT, T_DEC_OUT, T_COUNT   // timing-only slots of the two edge kernels
};
const char* kLayerNames[T_COUNT] = {"enc_conv2", "enc_conv3", "enc_conv4", "enc_fc1", "enc_head", "l_dec_fc2", "dec_conv1",
                                    "dec_conv2", "dec_conv3", "bwd_dec_conv3", "bwd_dec_conv2", "bwd_dec_conv1", "bwd_l_dec_fc2",
                                    "full_dec_fc2", "full_dec_conv1", "dec_conv2a", "dec_conv2a2", "full_dec_conv2", "dec_conv3a", "dec_conv3a2",
                                    "full_dec_conv3", "dec_conv4a", "dec_conv4a2", "full_dec_conv4", "rgb_head",
                                    "bwd_rgb_head", "bwd_full_dec_conv4", "bwd_dec_conv4a2", "bwd_dec_conv4a", "bwd_full_dec_conv3",
                                    "bwd_dec_conv3a2", "bwd_dec_conv3a", "bwd_full_dec_conv2", "bwd_dec_conv2a2", "bwd_dec_conv2a",
                                    "bwd_full_dec_conv1", "bwd_full_dec_fc2",
                                    "enc_conv1", "dec_out"};

struct DevWeights {           // one GEMM layer's B operand + epilogue vectors
  __nv_bfloat16* b = nullptr;
  long long plane = 0;
  int ntiles = 0, Cout = 0, Cin = 0;
  float* scale = nullptr;
  float* shift = nullptr;
};

struct Plan;

}  // namespace

struct ian_handle {
  int device = 0;
  int model_kind = 0;
  int path = IAN_PATH_TC;
  int passes = 3;              // 3: float32 semantics (bf16 hi|lo split); 1: plain bf16 tensor-core math
  float* sk_ws = nullptr;      // stream-K partial-sum slots + arrival flags (shared by all layers of the handle)
  int* sk_flags = nullptr;
  int sk_epoch = 0;
  bool streamk = true;
  bool splitk = true;          // split-K for small-M layers (IAN_SPLITK=0: whole tiles everywhere; used by tests)
  bool tc2 = true;             // CTA-pair tap-GEMM for layers with enough whole tiles (IAN_TC2=0 turns it off)
  bool coop_finalize = true;   // deep split-K layers: cooperative finalize kernel (IAN_FINALIZE8=0: one thread per output everywhere)
  bool pdl = true;             // programmatic dependent launch along the kernel chains (tapgemm.h; IAN_PDL=0 turns it off)
  int tc2_min_tiles = 37;      // pair-tiles needed before a layer moves to the pair kernel (IAN_TC2_MIN); half a wave: stream-K fills it
  bool graphs = true;          // replay small-batch host calls as CUDA graphs (IAN_GRAPHS=0 turns it off)
  bool capturing = false;
  bool finalized = false;
  cudaStream_t stream = nullptr;
  cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;   // copy streams of the pipelined host API
  std::vector<void*> host_allocs;
  // fused all-gather over NVLink peer memory (ian_gather_*): this rank's double gather buffer + flags, peers' views
  int gw = 0, grank = 0, gn = 0, gcur = 0, gepoch = 0;
  float* gbuf = nullptr;                       // [2][world][n_local][3][64][64] + flags (int[8]) at the end
  float* gpeer_buf[8] = {nullptr};             // base of every rank's allocation (peer-mapped)
  bool gconnected = false;
  float** gather_dsts = nullptr;               // non-null only inside ian_reconstruct_gather_dev
  int gather_ndst = 0;
  // pipelined gather (ian_reconstruct_gather_async_dev): side stream + per-half events
  cudaStream_t push_stream = nullptr;
  cudaEvent_t g_comp[2] = {nullptr, nullptr}, g_done[2] = {nullptr, nullptr};
  bool g_done_valid[2] = {false, false};
  int g_last = -1;                             // buffer half of the most recent async step
  int push_ctas = 32;
  int push_mode = 0;                           // 0: copy engines + stream memory ops (no SM is touched); 1: the copy kernel
  void* train_ws = nullptr;                    // workspace of the training-mode ops (grown on demand)
  size_t train_ws_bytes = 0;
  long long tickets = 0;
  struct Ticket { int id = -1, n = 0, slot = 0; };
  Ticket inflight[2];          // the two most recent pipelined requests (ian_reconstruct_submit)
  std::string err;
  int64_t launches = 0;
  std::map<std::string, HostParam> params;
  DevWeights w[L_COUNT];
  float* conv1_wt = nullptr;   // [75][128]
  float* conv1_b = nullptr;    // [128]
  __nv_bfloat16* conv1_tc_wt = nullptr;    // [3][128 cout][64 k] bf16 blocks (hi | lo | tail), k = c*25+i*5+j (75 used)
  Conv1Maps* conv1_maps = nullptr;
  float* decout_wt = nullptr;  // [25][128][4] fp32 (SIMT forward + brush backward)
  __nv_bfloat16* decout_tc_wt = nullptr;   // [2][80][128] bf16 planes, row = tap*3+co (tensor-core forward)
  // full IAN extras
  std::vector<int32_t> made_ordering;       // MADE input ordering (mask_generator.py:35-38); set by ian_set_made_ordering
  float *made_w = nullptr, *made_b = nullptr;   // [2][3][100][100] masked weights (in,out), [2][3][100] biases
  int* head_taps = nullptr;                 // [33][2] (dy,dx) of the scales-[2,3,4] MDC
  float *head_wgb = nullptr, *head_wbb = nullptr;   // composite G_b [33][2][2], B_b [33][2][4]
  int head_ntaps = 0;
  __nv_bfloat16* head_tc_wt = nullptr;      // fused head (head_tc.cu): [2 planes][3 convs x 80 rows][128] bf16, row = sorted tap*2 + filter
  int head_dy_start[10] = {0};              // taps sorted by row offset: taps with dy = -4 + i are [dy_start[i], dy_start[i+1])
  int head_dx[33] = {0};
  std::map<int, Plan*> plans;
  int max_chunk = 512;
  bool timing = false;
  struct Timed { cudaEvent_t e0, e1; };
  std::vector<Timed> timed[T_COUNT];
  double time_ms[T_COUNT] = {0};
  long long time_cnt[T_COUNT] = {0};
};

namespace {

inline bool has_flow(const ian_handle* h) { return h->model_kind != IAN_MODEL_SIMPLE; }   // MADE/IAF latent + RGB-Beta head

int fail(ian_handle* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf; else g_create_error = buf;
  return code;
}

#define CUDA_TRY(h, expr)                                                                            \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    if (_e != cudaSuccess) return fail(h, IAN_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define LAUNCH_TRY(h, expr)                                                                          \
  do {                                                                                               \
    ian::pdl_flag() = (h)->pdl && !(h)->capturing && !(h)->timing;   /* tapgemm.h: PDL */              \
    ian::coop_finalize_flag() = (h)->coop_finalize;                                                  \
    int _n = (expr);                                                                                 \
    if (_n < 0) return fail(h, IAN_ERR_CUDA, "%s: launch failed: %s", #expr, cudaGetErrorString(cudaGetLastError())); \
    (h)->launches += _n;                                                                             \
  } while (0)

struct Planes {               // NHWC split-plane activation tensor
  __nv_bfloat16* p = nullptr;
  long long plane = 0;
};

struct Plan {
  int n = 0;
  Planes a1, a2, a3, a4, f1, zp, h0, h1, h2, h3, d3, d2, d1, d0;
  float *x = nullptr, *head = nullptr, *z = nullptr, *xhat = nullptr, *gpad = nullptr, *eps = nullptr;
  float* target = nullptr;
  int32_t* boxes = nullptr;
  // full IAN activations (NHWC split planes): block input x, pre-activated t0, mid t2, block output y per scale
  Planes fh0, fx1, ft1, fu1, fy1, fx2, ft2, fu2, fy2, fx3, ft3, fu3, fy3, fh4;
  uint8_t* stroke = nullptr;     // ian_paint_stroke_host staging (allocated on first use)
  float *z0 = nullptr, *ha = nullptr, *rg = nullptr, *tt = nullptr;   // tt: head tap table [n][198][4096]
  // brush backward of the flow models: saved B, head gradient, its im2col operand, and the per-stage gradients
  float *bsave = nullptr, *dpre = nullptr;
  Planes dha2, d4, ds3, du3, dx3, ds2, du2, dx2, ds1, du1, dx1, dfh0;
  TapGemm g[L_COUNT];
  TcMaps* maps[L_COUNT] = {nullptr};
  Tc2Maps* maps2[L_COUNT] = {nullptr};   // CTA-pair kernel (only for layers that run on it; see choose_kernels)
  struct Kernel { bool pair = false; int ksplit = 1; };
  Kernel kernel[L_COUNT][2];             // per precision ([0] float32, [1] bf16): pair or one-CTA kernel, and its K split
  DecOutMaps* decout_maps = nullptr;
  Conv1OutMap* conv1_out = nullptr;       // TMA-store view of a1 (conv1_tc.cu)
  HeadMaps* head_maps = nullptr;
  // pipelined host API: double-buffered boundary tensors + events (allocated on first use)
  float *sx[2] = {nullptr, nullptr}, *sz[2] = {nullptr, nullptr}, *sxh[2] = {nullptr, nullptr};
  cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
  // CUDA graphs of the kernel sequences behind the host entry points (small batches only; see run_graphed)
  struct GraphSlot { cudaGraphExec_t exec = nullptr; int64_t launches = 0; uint64_t key = 0; };
  enum { G_ENCODE, G_ENCODE_EPS, G_DECODE, G_RECON, G_GRAD, G_EDIT_STEP, G_STROKE, G_COUNT };
  GraphSlot graph[G_COUNT];
  std::vector<void*> allocs;
};

int alloc_planes(ian_handle* h, Plan* pl, Planes& t, long long elems) {
  void* p = nullptr;
  CUDA_TRY(h, cudaMalloc(&p, (size_t)elems * 2 * sizeof(__nv_bfloat16)));
  CUDA_TRY(h, cudaMemsetAsync(p, 0, (size_t)elems * 2 * sizeof(__nv_bfloat16), h->stream));
  pl->allocs.push_back(p);
  t.p = (__nv_bfloat16*)p;
  t.plane = elems;
  return IAN_OK;
}
template <typename T>
int alloc_buf(ian_handle* h, Plan* pl, T*& out, long long elems) {
  void* p = nullptr;
  CUDA_TRY(h, cudaMalloc(&p, (size_t)elems * sizeof(T)));
  CUDA_TRY(h, cudaMemsetAsync(p, 0, (size_t)elems * sizeof(T), h->stream));
  pl->allocs.push_back(p);
  out = (T*)p;
  return IAN_OK;
}

// ---- tap tables --------------------------------------------------------------------------------
void taps_conv_s2(TapGemm& g) {           // enc_conv: y[p] = sum_i x[2p+i-2] W[i]   (IAN_simple.py:73-116)
  g.nphase = 1;
  g.phase[0] = {0, 25, 0, 0};
  int t = 0;
  for (int i = 0; i < 5; ++i)
    for (int j = 0; j < 5; ++j) {
      const int a = (i - 2) >> 1, r = (i - 2) & 1, b = (j - 2) >> 1, s = (j - 2) & 1;
      g.taps[t++] = {(int16_t)(r * 2 + s), (int16_t)a, (int16_t)b, (int16_t)(i * 5 + j)};
    }
  g.sh = g.sw = 2;
  g.osh = g.osw = 1;
}
void taps_deconv_s2(TapGemm& g) {         // dec_conv: y[2p+r] = sum_d x[p+d] W[2+2d-r]   (layers.py:436-483)
  g.nphase = 4;
  int t = 0;
  for (int r = 0; r < 2; ++r)
    for (int s = 0; s < 2; ++s) {
      Phase& ph = g.phase[r * 2 + s];
      ph.tap_begin = t;
      ph.oh0 = r;
      ph.ow0 = s;
      for (int d = (r ? 0 : -1); d <= 1; ++d)
        for (int e = (s ? 0 : -1); e <= 1; ++e) {
          const int ki = 2 + 2 * d - r, kj = 2 + 2 * e - s;
          g.taps[t++] = {0, (int16_t)d, (int16_t)e, (int16_t)(ki * 5 + kj)};
        }
      ph.ntaps = t - ph.tap_begin;
    }
  g.sh = g.sw = 1;
  g.osh = g.osw = 2;
}
void taps_deconv_bwd(TapGemm& g) {        // dx[a] = sum_ki dy[2+2a-ki] W[ki]   (T.grad of the above, API.py:59,64)
  g.nphase = 1;
  g.phase[0] = {0, 25, 0, 0};
  int t = 0;
  for (int ki = 0; ki < 5; ++ki)
    for (int kj = 0; kj < 5; ++kj) {
      const int e = 2 - ki, f = 2 - kj;
      g.taps[t++] = {(int16_t)((e & 1) * 2 + (f & 1)), (int16_t)(e >> 1), (int16_t)(f >> 1), (int16_t)(ki * 5 + kj)};
    }
  g.sh = g.sw = 2;
  g.osh = g.osw = 1;
}
void taps_dense(TapGemm& g) {
  g.nphase = 1;
  g.phase[0] = {0, 1, 0, 0};
  g.taps[0] = {0, 0, 0, 0};
  g.sh = g.sw = 1;
  g.osh = g.osw = 1;
}

// distinct tap offsets of an MDC layer (reference layers.py:207-258): 3x3 base, then 3x3 dilated by each s > 0
// (0 in scales = the 1x1 mean filter, which lands on the centre tap).  17 / 25 / 33 offsets for [0,2] / [0,2,3] / [2,3,4].
std::vector<std::pair<int, int>> mdc_offsets(const std::vector<int>& scales) {
  std::vector<std::pair<int, int>> off;
  auto add = [&](int dy, int dx) {
    for (auto& o : off) if (o.first == dy && o.second == dx) return;
    off.push_back({dy, dx});
  };
  for (int i = -1; i <= 1; ++i) for (int j = -1; j <= 1; ++j) add(i, j);
  for (int s : scales) if (s > 0) for (int i = -1; i <= 1; ++i) for (int j = -1; j <= 1; ++j) add(i * s, j * s);
  return off;
}
void taps_mdc(TapGemm& g, const std::vector<int>& scales) {
  const auto off = mdc_offsets(scales);
  g.nphase = 1;
  g.phase[0] = {0, (int)off.size(), 0, 0};
  for (size_t t = 0; t < off.size(); ++t) g.taps[t] = {0, (int16_t)off[t].first, (int16_t)off[t].second, (int16_t)t};
  g.sh = g.sw = 1;
  g.osh = g.osw = 1;
}

void taps_mdc_bwd(TapGemm& g, const std::vector<int>& scales) {   // din[q] = sum_t dout[q - off_t] * comp_t^T
  const auto off = mdc_offsets(scales);
  g.nphase = 1;
  g.phase[0] = {0, (int)off.size(), 0, 0};
  for (size_t t = 0; t < off.size(); ++t) g.taps[t] = {0, (int16_t)(-off[t].first), (int16_t)(-off[t].second), (int16_t)t};
  g.sh = g.sw = 1;
  g.osh = g.osw = 1;
}

// ---- layer tables --------------------------------------------------------------------------------
// Every tap-GEMM layer of a graph is one row: its taps, the plan buffers it reads and writes, its input size and its
// epilogue.  Cin comes from the layer's weights, the M grid and the output size from the taps (wire_layer).
enum TapKind { CONV_S2, DECONV_S2, DECONV_BWD, DENSE, MDC, MDC_BWD };
enum Seq { ENCODE, DECODE, BRUSH, HEAD };   // the sequence a layer runs in; HEAD: the RGB-Beta head's GEMM (run_head)

struct LayerRow {
  int id, seq, tap;
  Planes Plan::*in;
  int Hin, act;                                   // Hin: input height = width
  Planes Plan::*out = nullptr;                    // NHWC split-plane output (nullptr: a float32 output, set below)
  Planes Plan::*mask = nullptr;                   // ACT_MASK: the forward activation whose sign gates the gradient, and
  float mask_slope = 0.f;                         // the factor where it is not positive (0: rectify, 0.2: LeakyRectify)
  // set by the few layers that need them
  std::vector<int> scales;                        // MDC / MDC_BWD: the dilations (0 = the 1x1 mean filter)
  Planes Plan::*res = nullptr;                    // MDBLOCK residual (TapGemm::res / res_after)
  int res_after = 0;
  Planes Plan::*out_raw = nullptr;                // the un-normalised sum: an MDBLOCK's input x
  float* Plan::*out_f32 = nullptr;                // float32 NHWC output
  float* Plan::*out_f32_t = nullptr;              // channel-major float32 output, cout_real columns (the head's tap table)
  int cout_real = 0;
  int scale_pix_stride = 0;
  bool always_split = false;                      // choose a K split whatever the tile count (the deep dense layers)

  LayerRow& mdc(std::vector<int> s) { scales = std::move(s); return *this; }
  LayerRow& residual(Planes Plan::*r, int after) { res = r; res_after = after; return *this; }
  LayerRow& raw(Planes Plan::*r) { out_raw = r; return *this; }
  LayerRow& f32(float* Plan::*o) { out_f32 = o; return *this; }
  LayerRow& f32_t(float* Plan::*o, int c) { out_f32_t = o; cout_real = c; return *this; }
  LayerRow& pix_stride(int s) { scale_pix_stride = s; return *this; }
  LayerRow& split() { always_split = true; return *this; }
};

// The rows of one model kind: the encoder, then the decoder with its RGB output layer, then the brush backward, each in
// run order.
std::vector<LayerRow> make_layer_table(int kind) {
  using R = LayerRow;
  const int fc1_act = kind == IAN_MODEL_SIMPLE ? ACT_ELU : ACT_RELU;   // IAN_simple.py:121 elu; IAN.py:118 / IANv1.py:109 rectify
  std::vector<R> t = {                                                 // encoder (IAN_simple.py:84-126)
      {L_ENC_CONV2, ENCODE, CONV_S2, &Plan::a1, 32, ACT_LRELU, &Plan::a2},
      {L_ENC_CONV3, ENCODE, CONV_S2, &Plan::a2, 16, ACT_LRELU, &Plan::a3},
      {L_ENC_CONV4, ENCODE, CONV_S2, &Plan::a3, 8, ACT_LRELU, &Plan::a4},
      R{L_ENC_FC1, ENCODE, DENSE, &Plan::a4, 1, fc1_act, &Plan::f1}.split(),
      R{L_ENC_HEAD, ENCODE, DENSE, &Plan::f1, 1, ACT_NONE}.f32(&Plan::head)};
  std::vector<R> d;
  if (kind == IAN_MODEL_SIMPLE) {
    // decoder (IAN_simple.py:129-170), then its backward-data for the latent brush (T.grad at API.py:59,64)
    d = {{L_DEC_FC2, DECODE, DENSE, &Plan::zp, 1, ACT_RELU, &Plan::h0},
         {L_DEC_CONV1, DECODE, DECONV_S2, &Plan::h0, 4, ACT_RELU, &Plan::h1},
         {L_DEC_CONV2, DECODE, DECONV_S2, &Plan::h1, 8, ACT_RELU, &Plan::h2},
         {L_DEC_CONV3, DECODE, DECONV_S2, &Plan::h2, 16, ACT_RELU, &Plan::h3},
         {L_BWD_CONV3, BRUSH, DECONV_BWD, &Plan::d3, 32, ACT_MASK, &Plan::d2, &Plan::h2},
         {L_BWD_CONV2, BRUSH, DECONV_BWD, &Plan::d2, 16, ACT_MASK, &Plan::d1, &Plan::h1},
         R{L_BWD_CONV1, BRUSH, DECONV_BWD, &Plan::d1, 8, ACT_MASK, &Plan::d0, &Plan::h0}.pix_stride(1024),  // bnorm_dec_fc2 is per FEATURE (pixel, channel)
         R{L_BWD_FC2, BRUSH, DENSE, &Plan::d0, 1, ACT_NONE}.f32(&Plan::gpad).split()};
  } else if (kind == IAN_MODEL_V1) {
    // decoder of IANv1 (reference IANv1.py:125-201): dense (linear) -> 4 x [deconv, BN, relu] -> RGB-Beta head.  The last
    // deconv has 64 output channels; it is stored 128 wide (upper half zero weights) so the head GEMM keeps Cin % 64 == 0
    // tiles.  Brush backward (T.grad of API.py:59,64 on this graph): head GEMM, the four deconvs' backward-data, the dense.
    d = {{L_DEC_FC2, DECODE, DENSE, &Plan::zp, 1, ACT_NONE, &Plan::h0},
         {L_DEC_CONV1, DECODE, DECONV_S2, &Plan::h0, 4, ACT_RELU, &Plan::h1},
         {L_DEC_CONV2, DECODE, DECONV_S2, &Plan::h1, 8, ACT_RELU, &Plan::h2},
         {L_DEC_CONV3, DECODE, DECONV_S2, &Plan::h2, 16, ACT_RELU, &Plan::h3},
         {F_DEC_CONV4, DECODE, DECONV_S2, &Plan::h3, 32, ACT_RELU, &Plan::fh4},
         R{F_HEAD, HEAD, DENSE, &Plan::fh4, 64, ACT_NONE}.f32_t(&Plan::tt, 198),
         {F_BWD_HEAD, BRUSH, DENSE, &Plan::dha2, 64, ACT_MASK, &Plan::d4, &Plan::fh4},
         {F_BWD_CONV4, BRUSH, DECONV_BWD, &Plan::d4, 64, ACT_MASK, &Plan::d3, &Plan::h3},
         {L_BWD_CONV3, BRUSH, DECONV_BWD, &Plan::d3, 32, ACT_MASK, &Plan::d2, &Plan::h2},
         {L_BWD_CONV2, BRUSH, DECONV_BWD, &Plan::d2, 16, ACT_MASK, &Plan::d1, &Plan::h1},
         {L_BWD_CONV1, BRUSH, DECONV_BWD, &Plan::d1, 8, ACT_NONE, &Plan::d0},       // l_dec_fc2 is linear here (IANv1.py:125-130)
         R{L_BWD_FC2, BRUSH, DENSE, &Plan::d0, 1, ACT_NONE}.f32(&Plan::gpad).split()};
  } else {
    // decoder of the full IAN (reference IAN.py:129-207): dense -> 3 x (deconv, MDBLOCK) -> deconv -> RGB-Beta head.
    // Per block: the deconv's raw sum -> x (the block's residual), lrelu(BN0(x)) -> t (layers.py:413: BN(incoming) strips
    // the bias); MDCL 1: u = lrelu(BN1(M1(t))); MDCL 2: y = lrelu(BN2(x + M2(u))).  The RGB-Beta head is ONE dense
    // 128 -> 33 taps x 6 filters GEMM (the feature map is staged once, not 33 times), written channel-major; the dilated
    // taps are applied afterwards as coalesced shifted reads (head_gather).
    // Brush backward (T.grad of API.py:59,64 on this graph).  LeakyRectify(0.2) backward = mask slope 0.2 on the sign of
    // the stored forward activation; per block, after the backward-data of the deconv ABOVE it (its input gradient lives
    // at 2x the block's resolution):
    //   ds = dy * lrelu'(y) * s2 ;  du = M2^T(ds) * lrelu'(u) * s1 ;  dx = M1^T(du) * lrelu'(t) * s0 + ds
    d = {{F_DEC_FC2, DECODE, DENSE, &Plan::zp, 1, ACT_LRELU, &Plan::fh0},
         R{F_DEC_CONV1, DECODE, DECONV_S2, &Plan::fh0, 4, ACT_LRELU, &Plan::ft1}.raw(&Plan::fx1),
         R{F_MD1A, DECODE, MDC, &Plan::ft1, 8, ACT_LRELU, &Plan::fu1}.mdc({0, 2}),
         R{F_MD1B, DECODE, MDC, &Plan::fu1, 8, ACT_LRELU, &Plan::fy1}.mdc({0, 2}).residual(&Plan::fx1, 0),
         R{F_DEC_CONV2, DECODE, DECONV_S2, &Plan::fy1, 8, ACT_LRELU, &Plan::ft2}.raw(&Plan::fx2),
         R{F_MD2A, DECODE, MDC, &Plan::ft2, 16, ACT_LRELU, &Plan::fu2}.mdc({0, 2, 3}),
         R{F_MD2B, DECODE, MDC, &Plan::fu2, 16, ACT_LRELU, &Plan::fy2}.mdc({0, 2, 3}).residual(&Plan::fx2, 0),
         R{F_DEC_CONV3, DECODE, DECONV_S2, &Plan::fy2, 16, ACT_LRELU, &Plan::ft3}.raw(&Plan::fx3),
         R{F_MD3A, DECODE, MDC, &Plan::ft3, 32, ACT_LRELU, &Plan::fu3}.mdc({0, 2, 3}),
         R{F_MD3B, DECODE, MDC, &Plan::fu3, 32, ACT_LRELU, &Plan::fy3}.mdc({0, 2, 3}).residual(&Plan::fx3, 0),
         {F_DEC_CONV4, DECODE, DECONV_S2, &Plan::fy3, 32, ACT_LRELU, &Plan::fh4},
         R{F_HEAD, HEAD, DENSE, &Plan::fh4, 64, ACT_NONE}.f32_t(&Plan::tt, 198),
         {F_BWD_HEAD, BRUSH, DENSE, &Plan::dha2, 64, ACT_MASK, &Plan::d4, &Plan::fh4, 0.2f},
         {F_BWD_CONV4, BRUSH, DECONV_BWD, &Plan::d4, 64, ACT_MASK, &Plan::ds3, &Plan::fy3, 0.2f},
         R{F_BWD_MD3B, BRUSH, MDC_BWD, &Plan::ds3, 32, ACT_MASK, &Plan::du3, &Plan::fu3, 0.2f}.mdc({0, 2, 3}),
         R{F_BWD_MD3A, BRUSH, MDC_BWD, &Plan::du3, 32, ACT_MASK, &Plan::dx3, &Plan::ft3, 0.2f}.mdc({0, 2, 3}).residual(&Plan::ds3, 1),
         {F_BWD_CONV3, BRUSH, DECONV_BWD, &Plan::dx3, 32, ACT_MASK, &Plan::ds2, &Plan::fy2, 0.2f},
         R{F_BWD_MD2B, BRUSH, MDC_BWD, &Plan::ds2, 16, ACT_MASK, &Plan::du2, &Plan::fu2, 0.2f}.mdc({0, 2, 3}),
         R{F_BWD_MD2A, BRUSH, MDC_BWD, &Plan::du2, 16, ACT_MASK, &Plan::dx2, &Plan::ft2, 0.2f}.mdc({0, 2, 3}).residual(&Plan::ds2, 1),
         {F_BWD_CONV2, BRUSH, DECONV_BWD, &Plan::dx2, 16, ACT_MASK, &Plan::ds1, &Plan::fy1, 0.2f},
         R{F_BWD_MD1B, BRUSH, MDC_BWD, &Plan::ds1, 8, ACT_MASK, &Plan::du1, &Plan::fu1, 0.2f}.mdc({0, 2}),
         R{F_BWD_MD1A, BRUSH, MDC_BWD, &Plan::du1, 8, ACT_MASK, &Plan::dx1, &Plan::ft1, 0.2f}.mdc({0, 2}).residual(&Plan::ds1, 1),
         {F_BWD_CONV1, BRUSH, DECONV_BWD, &Plan::dx1, 8, ACT_MASK, &Plan::dfh0, &Plan::fh0, 0.2f},
         R{F_BWD_FC2, BRUSH, DENSE, &Plan::dfh0, 1, ACT_NONE}.f32(&Plan::gpad).split()};
  }
  t.insert(t.end(), d.begin(), d.end());
  return t;
}

const std::vector<LayerRow>& layer_table(int kind) {
  static const std::vector<LayerRow> tables[3] = {make_layer_table(IAN_MODEL_SIMPLE), make_layer_table(IAN_MODEL_FULL),
                                                  make_layer_table(IAN_MODEL_V1)};
  return tables[kind];
}

// the TapGemm of one row (g is zero-filled): Cin from the layer's weights, the M grid and output size from the taps
void wire_layer(TapGemm& g, const LayerRow& r, Plan* pl, const DevWeights& w) {
  switch (r.tap) {
    case CONV_S2: taps_conv_s2(g); break;
    case DECONV_S2: taps_deconv_s2(g); break;
    case DECONV_BWD: taps_deconv_bwd(g); break;
    case DENSE: taps_dense(g); break;
    case MDC: taps_mdc(g, r.scales); break;
    case MDC_BWD: taps_mdc_bwd(g, r.scales); break;
  }
  g.a = (pl->*r.in).p; g.a_plane = (pl->*r.in).plane;
  g.n_img = pl->n; g.Hin = g.Win = r.Hin; g.Cin = w.Cin;
  g.Hg = g.Wg = r.Hin / g.sh;                  // stride-2 conv and backward-data halve the size,
  g.Hout = g.Wout = g.Hg * g.osh;              // the stride-2 deconv doubles it
  g.b = w.b; g.b_plane = w.plane; g.Cout = w.Cout;
  g.scale = w.scale; g.shift = w.shift; g.scale_pix_stride = r.scale_pix_stride;
  g.act = r.act;
  g.ksplit = 1;
  if (r.out) { g.out = (pl->*r.out).p; g.out_plane = (pl->*r.out).plane; }
  if (r.mask) g.mask = (pl->*r.mask).p;
  g.mask_slope = r.mask_slope;
  if (r.res) { g.res = (pl->*r.res).p; g.res_plane = (pl->*r.res).plane; }
  g.res_after = r.res_after;
  if (r.out_raw) { g.out_raw = (pl->*r.out_raw).p; g.out_raw_plane = (pl->*r.out_raw).plane; }
  if (r.out_f32) g.out_f32 = pl->*r.out_f32;
  if (r.out_f32_t) g.out_f32_t = pl->*r.out_f32_t;
  g.cout_real = r.cout_real;
}

// output tiles of the one-CTA kernel
long long one_cta_tiles(const TapGemm& g) {
  const int bn = (g.Cout % 256 == 0) ? 256 : (g.Cout % 128 == 0) ? 128 : 16;
  return (long long)((g.n_img * g.Hg * g.Wg + 127) / 128) * (g.Cout / bn) * g.nphase;
}

int choose_ksplit(const TapGemm& g) {
  // fill ~one wave of 148 SMs when the output tile count is small; keep >= 4 K steps per CTA
  const int ctas = (int)one_cta_tiles(g);
  int min_it = 1 << 30;
  for (int p = 0; p < g.nphase; ++p) {
    const int it = g.phase[p].ntaps * (g.Cin / 64);
    if (it < min_it) min_it = it;
  }
  int ks = 148 / ctas;
  if (ks > min_it / 4) ks = min_it / 4;
  if (ks < 1) ks = 1;
  if (ks > 64) ks = 64;
  return ks;
}

// One workspace per plan, shared by its split-K layers (they run back to back on one stream):
// [ksplit][pixel][Cout] float32 slabs, sized for the largest user.
int alloc_splitk_workspace(ian_handle* h, Plan* pl) {
  long long need = 0;
  for (int l = 0; l < L_COUNT; ++l) {
    TapGemm& g = pl->g[l];
    if (g.ksplit <= 1) continue;
    g.ws_slab = (long long)g.n_img * g.Hout * g.Wout * g.Cout;
    need = std::max(need, g.ws_slab * g.ksplit);
  }
  if (need == 0) return IAN_OK;
  float* ws = nullptr;
  int rc = alloc_buf(h, pl, ws, need);
  if (rc != IAN_OK) return rc;
  for (int l = 0; l < L_COUNT; ++l)
    if (pl->g[l].ksplit > 1) pl->g[l].ws = ws;
  return IAN_OK;
}

// The kernel each precision runs layer l on.  A layer moves to the CTA-pair kernel when it has no channel-major output, its
// channel counts fit the 256 x 128 pair tile and it has at least tc2_min_tiles pair-tiles (half of the SM pairs).  A split-K
// factor that choose_ksplit() picked to fill the one-CTA kernel's wave (37..74 tiles: e.g. the decoder's backward-data layers
// of the batch-128 edit loop) does not hold a layer back: in float32 mode the pair kernel runs it un-split, balanced by
// stream-K, without the workspace round trip and the finalize launch; bf16 mode keeps the split one-CTA form.
int choose_kernels(ian_handle* h, Plan* pl, int l) {
  const TapGemm& g = pl->g[l];
  Plan::Kernel* k = pl->kernel[l];
  k[0] = k[1] = {false, g.ksplit};
  if (!h->tc2 || g.out_f32_t || g.Cout % 128 || g.Cin % 64) return IAN_OK;
  char err[256] = {0};
  Tc2Maps* m = tc2_build_maps(g, err, sizeof(err));
  if (!m) return fail(h, IAN_ERR_CUDA, "layer %s (pair kernel): %s", kLayerNames[l], err);
  const long long pt = tc2_pair_tiles(g, m);
  int pks = pt >= h->tc2_min_tiles ? 1 : 0;
  // Few tiles but a deep K (enc_fc1 at batch 256: 8 pair-tiles x 256 K steps): split K over the SM pairs in the pair kernel
  // too.  The one-CTA kernel's 256-wide float32 tiles leave room for only 2 x 96 KB stages -- the TMA ring covers half of the
  // load latency and enc_fc1 ran at 35 % tensor activity; the pair kernel's 48 KB stages are four deep.  Same slab /
  // finalize protocol (the plan's workspace is sized for the one-CTA split, which is never smaller).  Batches above the
  // graph-replayed sizes only, so the single-image latency path keeps one schedule.
  if (!pks && g.ksplit > 1 && g.n_img > 32 && (long long)g.n_img * g.Hg * g.Wg >= 256) {
    int min_it = 1 << 30;
    for (int p = 0; p < g.nphase; ++p) min_it = std::min(min_it, g.phase[p].ntaps * (g.Cin / 64));
    int ks = (int)((tc_num_sms() / 2) / pt);
    ks = std::min(ks, std::min(min_it / 8, g.ksplit));
    if (ks >= 2 && pt * ks >= h->tc2_min_tiles) pks = ks;
  }
  if (!pks) {
    tc2_free_maps(m);
    return IAN_OK;
  }
  pl->maps2[l] = m;
  k[0] = {true, pks};
  // bf16 mode: the un-split Cout % 256 == 0 layers run on 256 x 256 pair tiles (32 KB per 512-clock stage instead of 48 KB:
  // the 192 KB ring then covers ~3 k clocks of TMA latency instead of ~2 k; measured +5 % on enc_conv2-4).  Cout = 128
  // single-pass layers stay on the one-CTA kernel's paired-M tiles (256 x 128 pair tiles: 24 KB stages, measured slower).
  if (pks == 1 && g.ksplit == 1 && g.Cout % 256 == 0 && pt / 2 >= h->tc2_min_tiles) k[1] = {true, 1};
  return IAN_OK;
}

// Per row of the plan: TMA maps, the K split and the kernel of each precision.  Small batches (NPE runs batch 1): a layer
// with fewer tiles than SMs would stream its weights through a handful of SMs, so it gets the K split choose_ksplit()
// sizes to spread K over the chip.
int finish_layer(ian_handle* h, Plan* pl, int l, bool always_split) {
  TapGemm& g = pl->g[l];
  char err[256] = {0};
  pl->maps[l] = tc_build_maps(g, err, sizeof(err));
  if (!pl->maps[l]) return fail(h, IAN_ERR_CUDA, "layer %s: %s", kLayerNames[l], err);
  if (always_split || (!g.out_f32_t && one_cta_tiles(g) <= 74)) g.ksplit = h->splitk ? choose_ksplit(g) : 1;
  return choose_kernels(h, pl, l);
}

int build_plan(ian_handle* h, int n, Plan** out) {
  Plan* pl = new Plan();
  pl->n = n;
  const long long N = n;
  int rc;
#define AP(t, e) if ((rc = alloc_planes(h, pl, pl->t, (e))) != IAN_OK) return rc;
#define AB(t, e) if ((rc = alloc_buf(h, pl, pl->t, (e))) != IAN_OK) return rc;
  const bool full = h->model_kind == IAN_MODEL_FULL, v1 = h->model_kind == IAN_MODEL_V1;
  AP(a1, N * 32 * 32 * 128) AP(a2, N * 16 * 16 * 256) AP(a3, N * 8 * 8 * 512) AP(a4, N * 4 * 4 * 1024)
  AP(f1, N * 1024) AP(zp, N * 128)
  AB(x, N * 3 * 4096) AB(head, N * 256) AB(z, N * 100) AB(xhat, N * 3 * 4096) AB(eps, N * 100)
  if (!full) {
    AP(h0, N * 16384) AP(h1, N * 8 * 8 * 512) AP(h2, N * 16 * 16 * 256) AP(h3, N * 32 * 32 * 128)
  }
  if (v1) {
    AP(fh4, N * 4096 * 128)
    AB(z0, N * 100) AB(ha, N * 4096 * 16) AB(rg, N * 4096 * 4) AB(tt, N * 198 * 4096)
    AB(bsave, N * 4096 * 2) AB(dpre, N * 4096 * 8) AP(dha2, N * 4096 * 256) AP(d4, N * 4096 * 128)
    AP(d3, N * 32 * 32 * 128) AP(d2, N * 16 * 16 * 256) AP(d1, N * 8 * 8 * 512) AP(d0, N * 16384)
    AB(gpad, N * 128) AB(target, N * 3 * 4096) AB(boxes, N * 4)
  } else if (!full) {
    AP(d3, N * 32 * 32 * 128) AP(d2, N * 16 * 16 * 256) AP(d1, N * 8 * 8 * 512) AP(d0, N * 16384)
    AB(gpad, N * 128) AB(target, N * 3 * 4096) AB(boxes, N * 4)
  } else {
    AP(fh0, N * 8192)
    AP(fx1, N * 64 * 512) AP(ft1, N * 64 * 512) AP(fu1, N * 64 * 512) AP(fy1, N * 64 * 512)
    AP(fx2, N * 256 * 256) AP(ft2, N * 256 * 256) AP(fu2, N * 256 * 256) AP(fy2, N * 256 * 256)
    AP(fx3, N * 1024 * 128) AP(ft3, N * 1024 * 128) AP(fu3, N * 1024 * 128) AP(fy3, N * 1024 * 128)
    AP(fh4, N * 4096 * 128)
    AB(z0, N * 100) AB(ha, N * 4096 * 16) AB(rg, N * 4096 * 4) AB(tt, N * 198 * 4096)
    AB(bsave, N * 4096 * 2) AB(dpre, N * 4096 * 8) AP(dha2, N * 4096 * 256) AP(d4, N * 4096 * 128)
    AP(ds3, N * 1024 * 128) AP(du3, N * 1024 * 128) AP(dx3, N * 1024 * 128)
    AP(ds2, N * 256 * 256) AP(du2, N * 256 * 256) AP(dx2, N * 256 * 256)
    AP(ds1, N * 64 * 512) AP(du1, N * 64 * 512) AP(dx1, N * 64 * 512)
    AP(dfh0, N * 8192)
    AB(gpad, N * 128) AB(target, N * 3 * 4096) AB(boxes, N * 4)
  }
#undef AP
#undef AB

  memset(pl->g, 0, sizeof(TapGemm) * L_COUNT);
  for (const LayerRow& r : layer_table(h->model_kind)) {
    wire_layer(pl->g[r.id], r, pl, h->w[r.id]);
    if ((rc = finish_layer(h, pl, r.id, r.always_split)) != IAN_OK) return rc;
  }
  if ((rc = alloc_splitk_workspace(h, pl)) != IAN_OK) return rc;
  char err[256] = {0};
  pl->conv1_out = conv1_build_out_map(pl->a1.p, pl->a1.plane, n, err, sizeof(err));   // both paths: ian_set_path may
  if (!pl->conv1_out) return fail(h, IAN_ERR_CUDA, "enc_conv1: %s", err);               // switch a live handle
  if (has_flow(h)) {
    pl->head_maps = head_build_maps(pl->fh4.p, pl->fh4.plane, n, h->head_tc_wt, 3 * 80 * 128, err, sizeof(err));
    if (!pl->head_maps) return fail(h, IAN_ERR_CUDA, "rgb head: %s", err);
  } else {
    pl->decout_maps = decout_build_maps(pl->h3.p, pl->h3.plane, n, h->decout_tc_wt, 80 * 128, err, sizeof(err));
    if (!pl->decout_maps) return fail(h, IAN_ERR_CUDA, "dec_out: %s", err);
  }
  *out = pl;
  return IAN_OK;
}

void free_plan(Plan* pl) {
  for (void* p : pl->allocs) cudaFree(p);
  for (int s = 0; s < 2; ++s) {
    if (pl->ev_h2d[s]) cudaEventDestroy(pl->ev_h2d[s]);
    if (pl->ev_comp[s]) cudaEventDestroy(pl->ev_comp[s]);
    if (pl->ev_d2h[s]) cudaEventDestroy(pl->ev_d2h[s]);
  }
  for (int l = 0; l < L_COUNT; ++l) if (pl->maps[l]) tc_free_maps(pl->maps[l]);
  for (int l = 0; l < L_COUNT; ++l) if (pl->maps2[l]) tc2_free_maps(pl->maps2[l]);
  if (pl->decout_maps) decout_free_maps(pl->decout_maps);
  if (pl->conv1_out) conv1_free_out_map(pl->conv1_out);
  if (pl->head_maps) head_free_maps(pl->head_maps);
  for (auto& gs : pl->graph) if (gs.exec) cudaGraphExecDestroy(gs.exec);
  delete pl;
}

int get_plan(ian_handle* h, int n, Plan** out) {
  auto it = h->plans.find(n);
  if (it != h->plans.end()) { *out = it->second; return IAN_OK; }
  Plan* pl = nullptr;
  int rc = build_plan(h, n, &pl);
  if (rc != IAN_OK) { if (pl) free_plan(pl); return rc; }
  h->plans[n] = pl;
  *out = pl;
  return IAN_OK;
}

// ---- one tap-GEMM layer -------------------------------------------------------------------------
// CUDA-event pair around one kernel when layer timing is on; err: why the events could not be created or recorded
struct ScopedTimer {
  ian_handle* h; int slot; cudaStream_t st; ian_handle::Timed tm{}; bool on; cudaError_t err = cudaSuccess;
  ScopedTimer(ian_handle* h_, int slot_, cudaStream_t st_) : h(h_), slot(slot_), st(st_), on(h_->timing) {
    if (!on) return;
    if ((err = cudaEventCreate(&tm.e0)) == cudaSuccess && (err = cudaEventCreate(&tm.e1)) == cudaSuccess)
      err = cudaEventRecord(tm.e0, st);
    on = err == cudaSuccess;
  }
  ~ScopedTimer() {
    if (on) { cudaEventRecord(tm.e1, st); h->timed[slot].push_back(tm); }
  }
};

int run_gemm(ian_handle* h, Plan* pl, int l, cudaStream_t st) {
  TapGemm g = pl->g[l];
  if (g.ksplit < 1) return fail(h, IAN_ERR_INVALID, "layer %s is not part of this plan", kLayerNames[l]);
  g.passes = h->passes;
  g.out_t_bf16 = (g.out_f32_t && h->passes == 1) ? 1 : 0;   // bf16 mode: the head's tap table travels as bf16
  g.sk_ws = (h->streamk && !h->capturing) ? h->sk_ws : nullptr;   // the stream-K epoch is a kernel argument: not replayable
  g.sk_flags = h->sk_flags;
  g.sk_epoch = ++h->sk_epoch;
  // the verification path runs every layer un-split; the tensor-core path runs the kernel the plan chose for this precision
  const bool simt = h->path == IAN_PATH_SIMT;
  const Plan::Kernel k = simt ? Plan::Kernel{} : pl->kernel[l][h->passes == 1 ? 1 : 0];
  g.ksplit = k.ksplit;
  if (k.ksplit == 1) g.ws = nullptr;
  {
    ScopedTimer tm(h, l, st);                              // the layer's time ends before the split-K finalize
    CUDA_TRY(h, tm.err);
    if (simt)
      LAUNCH_TRY(h, launch_tapgemm_simt(g, st));
    else if (k.pair)
      LAUNCH_TRY(h, launch_tapgemm_tc2(g, pl->maps2[l], st));
    else
      LAUNCH_TRY(h, launch_tapgemm_tc(g, pl->maps[l], st));
  }
  if (g.ksplit > 1) LAUNCH_TRY(h, launch_splitk_finalize(g, st));
  return IAN_OK;
}

// the tap-GEMM layers of one sequence of the handle's graph, in table order
int run_layers(ian_handle* h, Plan* pl, int seq, cudaStream_t st) {
  for (const LayerRow& r : layer_table(h->model_kind)) {
    if (r.seq != seq) continue;
    int rc = run_gemm(h, pl, r.id, st);
    if (rc != IAN_OK) return rc;
  }
  return IAN_OK;
}

// z_pre (nullable): the pre-flow latent l_Z_IAF (= z itself for IAN_simple)
int run_encode(ian_handle* h, Plan* pl, const float* x, const float* eps, float* z, cudaStream_t st, float* z_pre = nullptr) {
  const int n = pl->n;
  {
    ScopedTimer tm(h, T_CONV1, st);
    if (h->path == IAN_PATH_TC)
      LAUNCH_TRY(h, launch_conv1_tc(h->conv1_maps, pl->conv1_out, x, h->conv1_b, n, st));
    else
      LAUNCH_TRY(h, launch_conv1(x, h->conv1_wt, h->conv1_b, pl->a1.p, pl->a1.plane, n, st));
  }
  int rc = run_layers(h, pl, ENCODE, st);
  if (rc != IAN_OK) return rc;
  if (has_flow(h)) {
    // l_Z_IAF = mu (+ exp(ls) eps), then l_Z = IAF(l_Z_IAF; MADE_mu, MADE_ls)   (IAN.py:126-128)
    LAUNCH_TRY(h, launch_sample(pl->head, eps, z_pre ? z_pre : pl->z0, nullptr, 0, n, st));
    LAUNCH_TRY(h, launch_made_iaf(z_pre ? z_pre : pl->z0, h->made_w, h->made_b, z, pl->zp.p, pl->zp.plane, n, st));
    return IAN_OK;
  }
  LAUNCH_TRY(h, launch_sample(pl->head, eps, z, pl->zp.p, pl->zp.plane, n, st));
  if (z_pre) CUDA_TRY(h, cudaMemcpyAsync(z_pre, z, (size_t)n * 400, cudaMemcpyDeviceToDevice, st));
  return IAN_OK;
}

// RGB-Beta head (IAN.py:183-207) from the feature map fh4.  Tensor-core path: head_tc.cu (dense GEMM + on-chip tap gather,
// then the autoregressive part in one kernel).  Verification path: the dense GEMM into the HBM tap table + gather + the
// three per-pixel kernels of round 1 -- a second, independent formulation.  The last of those kernels stores x_hat, or,
// inside ian_reconstruct_gather*_dev, into the gather destinations (as dec_out does for IAN_simple).
int run_head(ian_handle* h, Plan* pl, float* xhat, cudaStream_t st) {
  float* one[1] = {xhat};
  float* const* dsts = h->gather_dsts ? h->gather_dsts : one;
  const int ndst = h->gather_dsts ? h->gather_ndst : 1;
  if (h->path == IAN_PATH_TC) {
    {
      ScopedTimer tm(h, F_HEAD, st);
      LAUNCH_TRY(h, launch_head_tc(pl->head_maps, h->passes, pl->ha, pl->n, st));
    }
    LAUNCH_TRY(h, launch_rgb_beta_head(pl->ha, 1, pl->rg, h->head_taps, h->head_wgb, h->head_wbb, h->head_ntaps, dsts, ndst, pl->bsave, pl->n, st));
    return IAN_OK;
  }
  int rc;
  if ((rc = run_gemm(h, pl, F_HEAD, st)) != IAN_OK) return rc;
  LAUNCH_TRY(h, launch_head_gather(pl->tt, h->passes == 1 ? 1 : 0, h->head_taps, h->head_ntaps, pl->ha, pl->n, st));
  LAUNCH_TRY(h, launch_rgb_beta_head(pl->ha, 0, pl->rg, h->head_taps, h->head_wgb, h->head_wbb, h->head_ntaps, dsts, ndst, pl->bsave, pl->n, st));
  return IAN_OK;
}

// zp must already hold the latent planes
int run_decode_from_planes(ian_handle* h, Plan* pl, float* xhat, cudaStream_t st) {
  int rc = run_layers(h, pl, DECODE, st);
  if (rc != IAN_OK) return rc;
  if (has_flow(h)) return run_head(h, pl, xhat, st);
  ScopedTimer tm(h, T_DEC_OUT, st);
  if (h->path == IAN_PATH_TC) {
    float* one[1] = {xhat};
    LAUNCH_TRY(h, launch_dec_out_tc(pl->decout_maps, h->gather_dsts ? h->gather_dsts : one, h->gather_dsts ? h->gather_ndst : 1, pl->n, st));
  }
  else
    LAUNCH_TRY(h, launch_dec_out(pl->h3.p, pl->h3.plane, h->decout_wt, xhat, pl->n, st));
  return IAN_OK;
}

int run_decode(ian_handle* h, Plan* pl, const float* z, float* xhat, cudaStream_t st) {
  LAUNCH_TRY(h, launch_z_to_planes(z, pl->zp.p, pl->zp.plane, pl->n, st));
  return run_decode_from_planes(h, pl, xhat, st);
}

// decoder forward (from zp) + backward; leaves g (n,128 padded) in pl->gpad
int run_grad_core(ian_handle* h, Plan* pl, const int32_t* boxes, const float* target, int target_is_frame,
                  cudaStream_t st) {
  int rc;
  if ((rc = run_decode_from_planes(h, pl, pl->xhat, st)) != IAN_OK) return rc;
  if (has_flow(h)) {
    // the gradient is w.r.t. l_Z, the decoder's input (API.py:46: X_hat = get_output(l_out, {l_Z: Z})): no MADE/IAF backward
    LAUNCH_TRY(h, launch_head_bwd(pl->xhat, pl->rg, pl->bsave, boxes, target, target_is_frame, h->head_taps, h->head_wgb,
                                  h->head_wbb, h->head_ntaps, pl->dpre, pl->dha2.p, pl->dha2.plane, pl->n, st));
  } else {
    LAUNCH_TRY(h, launch_brush_seed_bwd(pl->xhat, boxes, target, target_is_frame, h->decout_wt, h->w[L_DEC_CONV3].scale,
                                        pl->h3.p, pl->d3.p, pl->d3.plane, pl->n, st));
  }
  return run_layers(h, pl, BRUSH, st);
}

int check_ready(ian_handle* h, int n, const void* a, const void* b) {
  if (!h) return IAN_ERR_INVALID;
  if (!h->finalized) return fail(h, IAN_ERR_STATE, "ian_finalize() has not been called");
  if (n <= 0) return fail(h, IAN_ERR_INVALID, "batch size must be positive (got %d)", n);
  if (!a || !b) return fail(h, IAN_ERR_INVALID, "NULL tensor pointer");
  return IAN_OK;
}

int validate_boxes(ian_handle* h, const int32_t* bx, int n) {
  for (int k = 0; k < n; ++k) {
    const int c1 = bx[4 * k], r1 = bx[4 * k + 1], c2 = bx[4 * k + 2], r2 = bx[4 * k + 3];
    if (c1 < 0 || r1 < 0 || c2 > 64 || r2 > 64 || c1 >= c2 || r1 >= r2)
      return fail(h, IAN_ERR_INVALID, "box %d = [c1=%d,r1=%d,c2=%d,r2=%d] is empty or outside the 64x64 frame", k, c1, r1, c2, r2);
  }
  return IAN_OK;
}

// ---- weight preparation --------------------------------------------------------------------------
const HostParam& P(ian_handle* h, const char* name) { return h->params[name]; }

// float32 v in the split-plane operand format (tapgemm.h): hi = bf16(v) at dst[i], lo = bf16(v - hi) at dst[i + lo_off]
inline void store_split(std::vector<uint16_t>& dst, size_t i, size_t lo_off, float v) {
  const uint16_t hi = f2bf(v);
  dst[i] = hi;
  dst[i + lo_off] = f2bf(v - bf2f(hi));
}

// our NHWC index hw*C + c of the reference's flatten(NCHW) index j = c*16 + hw of a (C, 4, 4) map
inline int nhwc_index(int j, int C) { return (j % 16) * C + j / 16; }

int upload_gemm_weights(ian_handle* h, int l, const std::vector<float>& B, int ntiles, int Cout, int Cin,
                        const std::vector<float>& scale, const std::vector<float>& shift) {
  DevWeights& w = h->w[l];
  const long long elems = (long long)ntiles * Cout * Cin;
  std::vector<uint16_t> planes((size_t)elems * 2);
  for (long long i = 0; i < elems; ++i) store_split(planes, i, elems, B[i]);
  CUDA_TRY(h, cudaMalloc((void**)&w.b, planes.size() * 2));
  CUDA_TRY(h, cudaMemcpy(w.b, planes.data(), planes.size() * 2, cudaMemcpyHostToDevice));
  w.plane = elems; w.ntiles = ntiles; w.Cout = Cout; w.Cin = Cin;
  CUDA_TRY(h, cudaMalloc((void**)&w.scale, scale.size() * 4));
  CUDA_TRY(h, cudaMemcpy(w.scale, scale.data(), scale.size() * 4, cudaMemcpyHostToDevice));
  if (!shift.empty()) {
    CUDA_TRY(h, cudaMalloc((void**)&w.shift, shift.size() * 4));
    CUDA_TRY(h, cudaMemcpy(w.shift, shift.data(), shift.size() * 4, cudaMemcpyHostToDevice));
  }
  return IAN_OK;
}

// inference BatchNorm folded to y = x*scale + shift (lasagne batch_norm, IAN_simple.py:84-170)
void fold_bn(ian_handle* h, const std::string& name, int c, std::vector<float>& scale, std::vector<float>& shift) {
  const auto& be = P(h, (name + ".beta").c_str()).data;
  const auto& ga = P(h, (name + ".gamma").c_str()).data;
  const auto& me = P(h, (name + ".mean").c_str()).data;
  const auto& is = P(h, (name + ".inv_std").c_str()).data;
  scale.resize(c);
  shift.resize(c);
  for (int i = 0; i < c; ++i) {
    scale[i] = ga[i] * is[i];
    shift[i] = be[i] - me[i] * scale[i];
  }
}

int prepare_encoder(ian_handle* h) {
  int rc;
  std::vector<float> B, sc, sf;
  // enc_conv2..4: B[i*5+j][o][c] = W[o][c][i][j]
  struct CS { int l; const char* w; const char* bn; int Cout, Cin; } convs[] = {
      {L_ENC_CONV2, "enc_conv2.W", "bnorm2", 256, 128}, {L_ENC_CONV3, "enc_conv3.W", "bnorm3", 512, 256},
      {L_ENC_CONV4, "enc_conv4.W", "bnorm4", 1024, 512}};
  for (auto& c : convs) {
    const auto& W = P(h, c.w).data;
    B.assign((size_t)25 * c.Cout * c.Cin, 0.f);
    for (int o = 0; o < c.Cout; ++o)
      for (int ci = 0; ci < c.Cin; ++ci)
        for (int t = 0; t < 25; ++t) B[((size_t)t * c.Cout + o) * c.Cin + ci] = W[((size_t)o * c.Cin + ci) * 25 + t];
    fold_bn(h, c.bn, c.Cout, sc, sf);
    if ((rc = upload_gemm_weights(h, c.l, B, 25, c.Cout, c.Cin, sc, sf)) != IAN_OK) return rc;
  }
  // enc_fc1: rows of W are flatten(NCHW) = c*16 + hw; our A is NHWC = hw*1024 + c.  Cout 1000 -> 1024.
  {
    const auto& W = P(h, "enc_fc1.W").data;
    B.assign((size_t)1024 * 16384, 0.f);
    for (int j = 0; j < 16384; ++j)
      for (int o = 0; o < 1000; ++o) B[(size_t)o * 16384 + nhwc_index(j, 1024)] = W[(size_t)j * 1000 + o];
    fold_bn(h, "bnorm_enc_fc1", 1000, sc, sf);
    sc.resize(1024, 0.f);
    sf.resize(1024, 0.f);
    if ((rc = upload_gemm_weights(h, L_ENC_FC1, B, 1, 1024, 16384, sc, sf)) != IAN_OK) return rc;
  }
  // head: mu (cols 0..99) | logsigma (cols 100..199), Cout 200 -> 256, Cin 1000 -> 1024
  {
    const auto& Wm = P(h, "enc_mu.W").data;
    const auto& Wl = P(h, "enc_logsigma.W").data;
    B.assign((size_t)256 * 1024, 0.f);
    for (int k = 0; k < 1000; ++k)
      for (int o = 0; o < 100; ++o) {
        B[(size_t)o * 1024 + k] = Wm[(size_t)k * 100 + o];
        B[(size_t)(100 + o) * 1024 + k] = Wl[(size_t)k * 100 + o];
      }
    std::vector<float> s1, f1, s2, f2;
    fold_bn(h, "mu_bnorm", 100, s1, f1);
    fold_bn(h, "ls_bnorm", 100, s2, f2);
    sc.assign(256, 0.f);
    sf.assign(256, 0.f);
    for (int o = 0; o < 100; ++o) { sc[o] = s1[o]; sf[o] = f1[o]; sc[100 + o] = s2[o]; sf[100 + o] = f2[o]; }
    if ((rc = upload_gemm_weights(h, L_ENC_HEAD, B, 1, 256, 1024, sc, sf)) != IAN_OK) return rc;
  }
  // conv1: wt[(c*5+i)*5+j][o] = W[o][c][i][j]
  {
    const auto& W = P(h, "enc_conv1.W").data;
    std::vector<float> wt(75 * 128);
    for (int o = 0; o < 128; ++o)
      for (int k = 0; k < 75; ++k) wt[k * 128 + o] = W[o * 75 + k];
    CUDA_TRY(h, cudaMalloc((void**)&h->conv1_wt, wt.size() * 4));
    CUDA_TRY(h, cudaMemcpy(h->conv1_wt, wt.data(), wt.size() * 4, cudaMemcpyHostToDevice));
    const auto& b = P(h, "enc_conv1.b").data;
    CUDA_TRY(h, cudaMalloc((void**)&h->conv1_b, 128 * 4));
    CUDA_TRY(h, cudaMemcpy(h->conv1_b, b.data(), 128 * 4, cudaMemcpyHostToDevice));
    // tensor-core form: B[co][k] = W[co][c][i][j] (the reference layout flattened), K padded 75 -> 80, as three
    // [128 cout][64 k] blocks: hi of k < 64 | lo of k < 64 | tail (hi of k 64..79 at columns 0..15, lo at 16..31)
    std::vector<uint16_t> planes(3 * 128 * 64, 0);
    for (int o = 0; o < 128; ++o)
      for (int k = 0; k < 75; ++k) {
        if (k < 64)
          store_split(planes, o * 64 + k, 128 * 64, W[o * 75 + k]);
        else
          store_split(planes, 2 * 128 * 64 + o * 64 + (k - 64), 16, W[o * 75 + k]);
      }
    CUDA_TRY(h, cudaMalloc((void**)&h->conv1_tc_wt, planes.size() * 2));
    CUDA_TRY(h, cudaMemcpy(h->conv1_tc_wt, planes.data(), planes.size() * 2, cudaMemcpyHostToDevice));
    char err[256] = {0};
    h->conv1_maps = conv1_build_maps(h->conv1_tc_wt, err, sizeof(err));
    if (!h->conv1_maps) return fail(h, IAN_ERR_CUDA, "enc_conv1: %s", err);
  }
  return IAN_OK;
}

// 5x5 stride-2 transposed conv weights W (Cin,Cout,5,5) -> forward tiles B[k][co][ci] = W[ci][co][k] (Cout padded to CoutPad)
void deconv_fwd_tiles(const std::vector<float>& W, int Cin, int Cout, int CoutPad, std::vector<float>& B) {
  B.assign((size_t)25 * CoutPad * Cin, 0.f);
  for (int ci = 0; ci < Cin; ++ci)
    for (int co = 0; co < Cout; ++co)
      for (int t = 0; t < 25; ++t) B[((size_t)t * CoutPad + co) * Cin + ci] = W[((size_t)ci * Cout + co) * 25 + t];
}

// backward-data of the same layer: the gradient w.r.t. the deconv's INPUT is a stride-2 convolution of the output gradient
// with tiles B[k][ci][co] = W[ci][co][k] (GEMM Cout = the deconv's Cin, GEMM Cin = the deconv's Cout, padded to CoutPad)
void deconv_bwd_tiles(const std::vector<float>& W, int Cin, int Cout, int CoutPad, std::vector<float>& B) {
  B.assign((size_t)25 * Cin * CoutPad, 0.f);
  for (int ci = 0; ci < Cin; ++ci)
    for (int co = 0; co < Cout; ++co)
      for (int t = 0; t < 25; ++t) B[((size_t)t * Cin + ci) * CoutPad + co] = W[((size_t)ci * Cout + co) * 25 + t];
}
// transposed composite MDC tiles: comp [nt][F][C] -> [nt][C][F]
void transpose_tiles(const std::vector<float>& comp, int nt, int F, int C, std::vector<float>& out) {
  out.assign((size_t)nt * C * F, 0.f);
  for (int t = 0; t < nt; ++t)
    for (int f = 0; f < F; ++f)
      for (int c = 0; c < C; ++c) out[((size_t)t * C + c) * F + f] = comp[((size_t)t * F + f) * C + c];
}

// l_dec_fc2 (W: (100, 16 C); reference column j = c*16 + hw, ours hw*C + c) as the forward GEMM (Cin 100 -> 128) and the
// brush backward dz[k] = sum_col d[col] * W[k][col] (Cout 100 -> 128).  The forward epilogue's scale and shift come per
// reference column and are returned in our column order.
int prepare_dec_fc2(ian_handle* h, int lf, int lb, int C, std::vector<float>& scale, std::vector<float>& shift) {
  const auto& W = P(h, "l_dec_fc2.W").data;
  const int N = 16 * C;
  std::vector<float> B((size_t)N * 128, 0.f), Bt((size_t)128 * N, 0.f), sc(N), sf(N);
  for (int j = 0; j < N; ++j) {
    const int col = nhwc_index(j, C);
    sc[col] = scale[j];
    sf[col] = shift[j];
    for (int k = 0; k < 100; ++k) B[(size_t)col * 128 + k] = Bt[(size_t)k * N + col] = W[(size_t)k * N + j];
  }
  scale.swap(sc);
  shift.swap(sf);
  int rc = upload_gemm_weights(h, lf, B, 1, N, 128, scale, shift);
  if (rc != IAN_OK) return rc;
  return upload_gemm_weights(h, lb, Bt, 1, 128, N, std::vector<float>(128, 1.f), {});
}

// dec_conv1..3 of IAN_simple and IANv1 (W: (Cin, Cout, 5, 5)): the forward GEMMs with their BN folded in, and the brush's
// backward-data GEMMs.  A backward GEMM produces the gradient w.r.t. its layer's INPUT activation, so its epilogue applies
// the BN scale of the layer below: `below` (l_dec_fc2's) for dec_conv1, then the previous deconv's.
int prepare_dec_convs(ian_handle* h, std::vector<float> below) {
  struct DS { int lf, lb; const char* w; const char* bn; int Cin, Cout; } decs[] = {
      {L_DEC_CONV1, L_BWD_CONV1, "dec_conv1.W", "bnorm_dc1", 1024, 512},
      {L_DEC_CONV2, L_BWD_CONV2, "dec_conv2.W", "bnorm_dc2", 512, 256},
      {L_DEC_CONV3, L_BWD_CONV3, "dec_conv3.W", "bnorm_dc3", 256, 128}};
  std::vector<float> B, sc, sf;
  for (const DS& d : decs) {
    const auto& W = P(h, d.w).data;
    deconv_fwd_tiles(W, d.Cin, d.Cout, d.Cout, B);
    fold_bn(h, d.bn, d.Cout, sc, sf);
    int rc = upload_gemm_weights(h, d.lf, B, 25, d.Cout, d.Cin, sc, sf);
    if (rc != IAN_OK) return rc;
    deconv_bwd_tiles(W, d.Cin, d.Cout, d.Cout, B);
    if ((rc = upload_gemm_weights(h, d.lb, B, 25, d.Cin, d.Cout, below, {})) != IAN_OK) return rc;
    below = sc;
  }
  return IAN_OK;
}

int prepare_simple_decoder(ian_handle* h) {
  int rc;
  std::vector<float> s, f;
  fold_bn(h, "bnorm_dec_fc2", 16384, s, f);
  if ((rc = prepare_dec_fc2(h, L_DEC_FC2, L_BWD_FC2, 1024, s, f)) != IAN_OK) return rc;
  if ((rc = prepare_dec_convs(h, s)) != IAN_OK) return rc;   // per feature: bwd_dec_conv1 has scale_pix_stride 1024
  // dec_out: wt[ki*5+kj][ci][co(4)] = W[ci][co][ki][kj]
  {
    const auto& W = P(h, "dec_out.W").data;
    // tensor-core form (decout_tc.cu): rows j = tap*3+co (75, padded to 80), K-major over ci; bf16 hi|lo planes
    {
      std::vector<uint16_t> planes(2 * 80 * 128, 0);
      for (int ci = 0; ci < 128; ++ci)
        for (int co = 0; co < 3; ++co)
          for (int t = 0; t < 25; ++t) store_split(planes, (t * 3 + co) * 128 + ci, 80 * 128, W[(ci * 3 + co) * 25 + t]);
      CUDA_TRY(h, cudaMalloc((void**)&h->decout_tc_wt, planes.size() * 2));
      CUDA_TRY(h, cudaMemcpy(h->decout_tc_wt, planes.data(), planes.size() * 2, cudaMemcpyHostToDevice));
    }
    std::vector<float> wt(25 * 128 * 4, 0.f);
    for (int ci = 0; ci < 128; ++ci)
      for (int co = 0; co < 3; ++co)
        for (int t = 0; t < 25; ++t) wt[(t * 128 + ci) * 4 + co] = W[(ci * 3 + co) * 25 + t];
    CUDA_TRY(h, cudaMalloc((void**)&h->decout_wt, wt.size() * 4));
    CUDA_TRY(h, cudaMemcpy(h->decout_wt, wt.data(), wt.size() * 4, cudaMemcpyHostToDevice));
  }
  return IAN_OK;
}

// composite MDC weights (reference layers.py:207-258): per distinct offset one [F][C] matrix
//   base 3x3: W[f,c,i,j]*coeff_base[f] at (i-1, j-1);  scale 0: mean_ij(W)*coeff_1x1[f] at (0,0);
//   scale s: W[f,c,i,j]*coeff_s[f] at ((i-1)s, (j-1)s)
void mdc_composite(ian_handle* h, const std::string& name, int F, int C, const std::vector<int>& scales,
                   std::vector<float>& comp /*[ntaps][F][C]*/) {
  const auto off = mdc_offsets(scales);
  const auto& W = P(h, (name + "W").c_str()).data;
  comp.assign(off.size() * (size_t)F * C, 0.f);
  auto tile_of = [&](int dy, int dx) { for (size_t t = 0; t < off.size(); ++t) if (off[t].first == dy && off[t].second == dx) return (int)t; return -1; };
  auto put = [&](int s, const std::vector<float>& coeff) {
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) {
        const int t = tile_of((i - 1) * s, (j - 1) * s);
        for (int f = 0; f < F; ++f)
          for (int c = 0; c < C; ++c) comp[((size_t)t * F + f) * C + c] += W[(((size_t)f * C + c) * 3 + i) * 3 + j] * coeff[f];
      }
  };
  put(1, P(h, (name + "_coeff_base").c_str()).data);
  for (int s : scales) {
    if (s == 0) {
      const auto& coeff = P(h, (name + "_coeff_1x1").c_str()).data;
      const int t = tile_of(0, 0);
      for (int f = 0; f < F; ++f)
        for (int c = 0; c < C; ++c) {
          float m = 0.f;
          for (int k = 0; k < 9; ++k) m += W[((size_t)f * C + c) * 9 + k];
          comp[((size_t)t * F + f) * C + c] += (m / 9.f) * coeff[f];
        }
    } else {
      put(s, P(h, (name + "_coeff_" + std::to_string(s)).c_str()).data);
    }
  }
}

// MADE connectivity (reference mask_generator.py:29-38,93-94 as API.IAN leaves it after reset("Once")): with ordering o,
// layer connectivities are input = o + 1, hidden = 1, output = o and a weight (i -> j) survives iff
// conn_in[i] <= conn_out[j].  which: 0 = `_input` (input -> hidden), 1 = `_output_W` (hidden -> output),
// 2 = `_output_D` (input -> output, direct).  Integer comparisons only: W * M is bit-exact.
inline bool made_keep(const int32_t* o, int which, int i, int j) {
  return which == 0 ? (o[i] + 1 <= 1) : which == 1 ? (1 <= o[j]) : (o[i] + 1 <= o[j]);
}

int prepare_made(ian_handle* h) {
  // ---- MADE (layers.py:653-853): masks from the ordering (mask_generator.py:93-94; SURVEY Appendix D), integer
  // comparisons, multiplied into the float32 weights here on the host (bit-exact W*M)
  {
    if (h->made_ordering.size() != 100) return fail(h, IAN_ERR_STATE, "ian_set_made_ordering() must precede ian_finalize() for the full IAN");
    const auto& o = h->made_ordering;
    std::vector<float> mw(2 * 3 * 10000), mb(2 * 3 * 100);
    const char* nets[2] = {"l_IAF_mu", "l_IAF_ls"};
    const char* subs[3] = {"_input", "_output_W", "_output_D"};
    for (int net = 0; net < 2; ++net)
      for (int m = 0; m < 3; ++m) {
        const auto& W = P(h, (std::string(nets[net]) + subs[m] + ".W").c_str()).data;
        const auto& b = P(h, (std::string(nets[net]) + subs[m] + ".b").c_str()).data;
        for (int i = 0; i < 100; ++i)
          for (int j = 0; j < 100; ++j) {
            const bool keep = made_keep(o.data(), m, i, j);
            mw[((net * 3 + m) * 100 + i) * 100 + j] = keep ? W[i * 100 + j] : 0.f;
          }
        for (int j = 0; j < 100; ++j) mb[(net * 3 + m) * 100 + j] = b[j];
      }
    CUDA_TRY(h, cudaMalloc((void**)&h->made_w, mw.size() * 4));
    CUDA_TRY(h, cudaMemcpy(h->made_w, mw.data(), mw.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMalloc((void**)&h->made_b, mb.size() * 4));
    CUDA_TRY(h, cudaMemcpy(h->made_b, mb.data(), mb.size() * 4, cudaMemcpyHostToDevice));
  }
  return IAN_OK;
}

// RGB-Beta head weights for a feature map with C real channels (128 for IAN.py, 64 for IANv1.py) stored 128 wide
int prepare_head(ian_handle* h, int C, const std::vector<float>& scale_below /*BN scale of the feature map (128 wide)*/) {
  int rc;
  std::vector<float> B, sc, comp;
  // ---- RGB-Beta head (IAN.py:183-207): the three 128->2 MDC convs as one 16-row tile [R | G_a | B_a | 0...]
  {
    const std::vector<int> hs = {2, 3, 4};
    const auto off = mdc_offsets(hs);
    const int nt = (int)off.size();
    if (nt * 6 != 198) return fail(h, IAN_ERR_STATE, "unexpected head tap count %d", nt);
    // one weight tile [256 rows][128]: row t*6 + (2k+f) = composite tap t of filter f of conv k in {R, G_a, B_a}
    B.assign((size_t)256 * 128, 0.f);
    const char* names[3] = {"R", "G_a", "B_a"};
    for (int k = 0; k < 3; ++k) {
      mdc_composite(h, names[k], 2, C, hs, comp);
      for (int t = 0; t < nt; ++t)
        for (int f = 0; f < 2; ++f)
          for (int c = 0; c < C; ++c) B[((size_t)(t * 6 + 2 * k + f)) * 128 + c] = comp[((size_t)t * 2 + f) * C + c];
    }
    sc.assign(256, 1.f);
    if ((rc = upload_gemm_weights(h, F_HEAD, B, 1, 256, 128, sc, {})) != IAN_OK) return rc;
    // backward: dh[c] = sum_k A2[k] * B[k][c], k = t*6 + (2 conv + filter): the transposed tile, GEMM Cout = 128, Cin = 256
    std::vector<float> Bt((size_t)128 * 256, 0.f);
    for (int k = 0; k < 256; ++k)
      for (int c = 0; c < 128; ++c) Bt[(size_t)c * 256 + k] = B[(size_t)k * 128 + c];
    if ((rc = upload_gemm_weights(h, F_BWD_HEAD, Bt, 1, 128, 256, scale_below, {})) != IAN_OK) return rc;
    std::vector<int> taps(nt * 2);
    for (int t = 0; t < nt; ++t) { taps[2 * t] = off[t].first; taps[2 * t + 1] = off[t].second; }
    CUDA_TRY(h, cudaMalloc((void**)&h->head_taps, taps.size() * 4));
    CUDA_TRY(h, cudaMemcpy(h->head_taps, taps.data(), taps.size() * 4, cudaMemcpyHostToDevice));
    h->head_ntaps = nt;
    // fused head (head_tc.cu): taps sorted by row offset (stable), per conv k one 80-row tile: row = sorted tap * 2 + filter
    {
      std::vector<int> order;
      int pos = 0;
      for (int dy = -4; dy <= 4; ++dy) {
        h->head_dy_start[dy + 4] = pos;
        for (int t = 0; t < nt; ++t)
          if (off[t].first == dy) { order.push_back(t); h->head_dx[pos++] = off[t].second; }
      }
      h->head_dy_start[9] = pos;
      if (pos != 33) return fail(h, IAN_ERR_STATE, "head taps do not fit the [-4,4] row-offset window");
      // head_tc.cu's gather uses the analytic form of this table: dy != 0 -> dx in {-|dy|, 0, |dy|}; dy = 0 -> the nine offsets
      // in the order base 3x3, then dilations 2, 3, 4 (mdc_offsets' insertion order).  Refuse anything else.
      const int dx0[9] = {-1, 0, 1, -2, 2, -3, 3, -4, 4};
      for (int dy = -4; dy <= 4; ++dy) {
        const int j0 = h->head_dy_start[dy + 4], cnt = h->head_dy_start[dy + 5] - j0;
        bool ok = cnt == (dy == 0 ? 9 : 3) && j0 == (dy < 0 ? 3 * (dy + 4) : dy == 0 ? 12 : 21 + 3 * (dy - 1));
        for (int e = 0; ok && e < cnt; ++e) {
          const int a = dy < 0 ? -dy : dy;
          ok = h->head_dx[j0 + e] == (dy == 0 ? dx0[e] : (e - 1) * a);
        }
        if (!ok) return fail(h, IAN_ERR_STATE, "RGB-head tap set differs from the scales-[2,3,4] MDC layout head_tc.cu assumes");
      }
      std::vector<uint16_t> planes((size_t)2 * 3 * 80 * 128, 0);
      const size_t plane = (size_t)3 * 80 * 128;
      for (int k = 0; k < 3; ++k)
        for (int j = 0; j < 33; ++j)
          for (int f = 0; f < 2; ++f)
            for (int c = 0; c < 128; ++c)
              store_split(planes, ((size_t)k * 80 + j * 2 + f) * 128 + c, plane, B[((size_t)(order[j] * 6 + 2 * k + f)) * 128 + c]);
      CUDA_TRY(h, cudaMalloc((void**)&h->head_tc_wt, planes.size() * 2));
      CUDA_TRY(h, cudaMemcpy(h->head_tc_wt, planes.data(), planes.size() * 2, cudaMemcpyHostToDevice));
    }
    mdc_composite(h, "G_b", 2, 2, hs, comp);             // [nt][2 out][2 in]
    CUDA_TRY(h, cudaMalloc((void**)&h->head_wgb, comp.size() * 4));
    CUDA_TRY(h, cudaMemcpy(h->head_wgb, comp.data(), comp.size() * 4, cudaMemcpyHostToDevice));
    mdc_composite(h, "B_b", 2, 4, hs, comp);             // [nt][2 out][4 in]
    CUDA_TRY(h, cudaMalloc((void**)&h->head_wbb, comp.size() * 4));
    CUDA_TRY(h, cudaMemcpy(h->head_wbb, comp.data(), comp.size() * 4, cudaMemcpyHostToDevice));
  }
  return IAN_OK;
}

// IANv1 decoder weights (IANv1.py:125-175)
int prepare_v1_decoder(ian_handle* h) {
  int rc;
  if ((rc = prepare_made(h)) != IAN_OK) return rc;
  // l_dec_fc2: dense 100 -> 16384 + bias, NO nonlinearity
  std::vector<float> sc(16384, 1.f), sf = P(h, "l_dec_fc2.b").data;
  if ((rc = prepare_dec_fc2(h, L_DEC_FC2, L_BWD_FC2, 1024, sc, sf)) != IAN_OK) return rc;
  if ((rc = prepare_dec_convs(h, std::vector<float>(1024, 1.f))) != IAN_OK) return rc;
  // dec_conv4: 128 -> 64 channels, stored 128 wide: channels 64..127 have zero weights, scale and shift (relu(0) = 0)
  const auto& W = P(h, "dec_conv4.W").data;
  std::vector<float> B;
  deconv_fwd_tiles(W, 128, 64, 128, B);
  fold_bn(h, "bnorm_dc4", 64, sc, sf);
  sc.resize(128, 0.f);
  sf.resize(128, 0.f);
  if ((rc = upload_gemm_weights(h, F_DEC_CONV4, B, 25, 128, 128, sc, sf)) != IAN_OK) return rc;
  // its backward-data lands on dec_conv3's output: bnorm_dc3's scale
  std::vector<float> s3, f3;
  fold_bn(h, "bnorm_dc3", 128, s3, f3);
  deconv_bwd_tiles(W, 128, 64, 128, B);
  if ((rc = upload_gemm_weights(h, F_BWD_CONV4, B, 25, 128, 128, s3, {})) != IAN_OK) return rc;
  return prepare_head(h, 64, sc);                          // sc: bnorm_dc4's scale (64 real channels, padded with zeros)
}

int prepare_full_decoder(ian_handle* h) {
  int rc;
  if ((rc = prepare_made(h)) != IAN_OK) return rc;
  // ---- l_dec_fc2: dense 100 -> 8192 + bias, lrelu (IAN.py:129-134)
  std::vector<float> B, sc(8192, 1.f), sf = P(h, "l_dec_fc2.b").data, comp;
  if ((rc = prepare_dec_fc2(h, F_DEC_FC2, F_BWD_FC2, 512, sc, sf)) != IAN_OK) return rc;
  // ---- deconvs + MDBLOCKs (IAN.py:139-171)
  struct St { int dconv, mda, mdb; const char* w; const char* blk; int Cin, Cout; std::vector<int> scales; };
  const St sts[3] = {{F_DEC_CONV1, F_MD1A, F_MD1B, "dec_conv1.W", "dec_conv2a", 512, 512, {0, 2}},
                     {F_DEC_CONV2, F_MD2A, F_MD2B, "dec_conv2.W", "dec_conv3a", 512, 256, {0, 2, 3}},
                     {F_DEC_CONV3, F_MD3A, F_MD3B, "dec_conv3.W", "dec_conv4a", 256, 128, {0, 2, 3}}};
  for (const St& s : sts) {
    deconv_fwd_tiles(P(h, s.w).data, s.Cin, s.Cout, s.Cout, B);
    fold_bn(h, std::string(s.blk) + "bnorm0", s.Cout, sc, sf);
    if ((rc = upload_gemm_weights(h, s.dconv, B, 25, s.Cout, s.Cin, sc, sf)) != IAN_OK) return rc;
    const int nt = (int)mdc_offsets(s.scales).size();
    mdc_composite(h, s.blk, s.Cout, s.Cout, s.scales, comp);
    fold_bn(h, std::string(s.blk) + "bnorm1", s.Cout, sc, sf);
    if ((rc = upload_gemm_weights(h, s.mda, comp, nt, s.Cout, s.Cout, sc, sf)) != IAN_OK) return rc;
    mdc_composite(h, std::string(s.blk) + "2", s.Cout, s.Cout, s.scales, comp);
    fold_bn(h, std::string(s.blk) + "bnorm2", s.Cout, sc, sf);
    if ((rc = upload_gemm_weights(h, s.mdb, comp, nt, s.Cout, s.Cout, sc, sf)) != IAN_OK) return rc;
  }
  deconv_fwd_tiles(P(h, "dec_conv4.W").data, 128, 128, 128, B);
  fold_bn(h, "bnorm_dc4", 128, sc, sf);
  if ((rc = upload_gemm_weights(h, F_DEC_CONV4, B, 25, 128, 128, sc, sf)) != IAN_OK) return rc;
  if ((rc = prepare_head(h, 128, sc)) != IAN_OK) return rc;
  // ---- brush backward (see the IAN.py rows of make_layer_table): every backward GEMM's epilogue applies the BN scale of the activation it lands on
  struct Bk { int dconv, mdb, mda; const char* w_above; int Cin_above, Cout_above; const char* blk; int C; std::vector<int> scales; };
  // dconv = backward-data of the deconv ABOVE block `blk` (w_above: (Cin_above = this block's C, Cout_above))
  const Bk bks[3] = {{F_BWD_CONV4, F_BWD_MD3B, F_BWD_MD3A, "dec_conv4.W", 128, 128, "dec_conv4a", 128, {0, 2, 3}},
                     {F_BWD_CONV3, F_BWD_MD2B, F_BWD_MD2A, "dec_conv3.W", 256, 128, "dec_conv3a", 256, {0, 2, 3}},
                     {F_BWD_CONV2, F_BWD_MD1B, F_BWD_MD1A, "dec_conv2.W", 512, 256, "dec_conv2a", 512, {0, 2}}};
  std::vector<float> s0, s1, s2, f_, Bt;
  for (const Bk& b : bks) {
    fold_bn(h, std::string(b.blk) + "bnorm0", b.C, s0, f_);
    fold_bn(h, std::string(b.blk) + "bnorm1", b.C, s1, f_);
    fold_bn(h, std::string(b.blk) + "bnorm2", b.C, s2, f_);
    deconv_bwd_tiles(P(h, b.w_above).data, b.Cin_above, b.Cout_above, b.Cout_above, B);
    if ((rc = upload_gemm_weights(h, b.dconv, B, 25, b.Cin_above, b.Cout_above, s2, {})) != IAN_OK) return rc;
    const int nt = (int)mdc_offsets(b.scales).size();
    mdc_composite(h, std::string(b.blk) + "2", b.C, b.C, b.scales, comp);
    transpose_tiles(comp, nt, b.C, b.C, Bt);
    if ((rc = upload_gemm_weights(h, b.mdb, Bt, nt, b.C, b.C, s1, {})) != IAN_OK) return rc;
    mdc_composite(h, b.blk, b.C, b.C, b.scales, comp);
    transpose_tiles(comp, nt, b.C, b.C, Bt);
    if ((rc = upload_gemm_weights(h, b.mda, Bt, nt, b.C, b.C, s0, {})) != IAN_OK) return rc;
  }
  deconv_bwd_tiles(P(h, "dec_conv1.W").data, 512, 512, 512, B);
  return upload_gemm_weights(h, F_BWD_CONV1, B, 25, 512, 512, std::vector<float>(512, 1.f), {});
}

// stream memory operations (driver API, fetched through the runtime): the free / pushed flag handshake of the pipelined
// all-gather runs as cuStreamWriteValue32 / cuStreamWaitValue32 on peer-mapped memory -- no kernel, hence no SM slot
typedef CUresult (*StreamWrite32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
typedef CUresult (*StreamWait32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
struct MemOps { StreamWrite32Fn write = nullptr; StreamWait32Fn wait = nullptr; };
inline const MemOps& memops() {
  static MemOps m;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void *pw = nullptr, *pq = nullptr;
    cudaDriverEntryPointQueryResult q1, q2;
    if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &pw, cudaEnableDefault, &q1) == cudaSuccess && q1 == cudaDriverEntryPointSuccess &&
        cudaGetDriverEntryPoint("cuStreamWaitValue32", &pq, cudaEnableDefault, &q2) == cudaSuccess && q2 == cudaDriverEntryPointSuccess) {
      m.write = reinterpret_cast<StreamWrite32Fn>(pw);
      m.wait = reinterpret_cast<StreamWait32Fn>(pq);
    }
  }
  return m;
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

template <typename F>
int for_chunks(ian_handle* h, int n, F&& f) {
  for (int off = 0; off < n; off += h->max_chunk) {
    const int cn = (n - off < h->max_chunk) ? n - off : h->max_chunk;
    Plan* pl = nullptr;
    int rc = get_plan(h, cn, &pl);
    if (rc != IAN_OK) return rc;
    if ((rc = f(pl, off, cn)) != IAN_OK) return rc;
  }
  return IAN_OK;
}

// The interactive calls (NPE: batch 1) are launch-bound: ~20-40 kernels of a few microseconds each.  The kernel
// sequence of a host entry point depends only on the plan (fixed buffers, fixed tensor maps) and a few scalars, so it is
// captured once per (plan, entry point, key) and replayed with one cudaGraphLaunch; the H2D/D2H copies of the
// caller's buffers stay outside the graph.  Large batches are not launch-bound (and may schedule stream-K, whose
// epoch is a kernel argument): they keep plain launches.
constexpr int kGraphMaxBatch = 32;

template <typename F>
int run_graphed(ian_handle* h, Plan* pl, int slot, uint64_t key, cudaStream_t st, F&& body) {
  if (!h->graphs || h->timing || h->path != IAN_PATH_TC || pl->n > kGraphMaxBatch || st != h->stream || h->gather_dsts)
    return body();
  Plan::GraphSlot& gs = pl->graph[slot];
  key = key * 4 + (uint64_t)(h->passes == 1 ? 1 : 0) + 2;      // +2: a valid key is never 0
  if (gs.exec && gs.key != key) {
    cudaGraphExecDestroy(gs.exec);
    gs.exec = nullptr;
  }
  if (!gs.exec) {
    const int64_t l0 = h->launches;
    CUDA_TRY(h, cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
    h->capturing = true;
    const int r = body();
    h->capturing = false;
    cudaGraph_t graph = nullptr;
    const cudaError_t e = cudaStreamEndCapture(st, &graph);
    gs.launches = h->launches - l0;
    h->launches = l0;
    if (r != IAN_OK) { if (graph) cudaGraphDestroy(graph); return r; }
    if (e != cudaSuccess) return fail(h, IAN_ERR_CUDA, "cudaStreamEndCapture failed: %s", cudaGetErrorString(e));
    const cudaError_t ei = cudaGraphInstantiate(&gs.exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ei != cudaSuccess) { gs.exec = nullptr; return fail(h, IAN_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ei)); }
    gs.key = key;
  }
  CUDA_TRY(h, cudaGraphLaunch(gs.exec, st));
  h->launches += gs.launches;
  return IAN_OK;
}

inline uint64_t float_bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

}  // namespace

// ================================================================================================
// C-ABI
// ================================================================================================
extern "C" {

int ian_create(int model_kind, int device, ian_handle** out) {
  if (!out) return fail(nullptr, IAN_ERR_INVALID, "out is NULL");
  if (model_kind != IAN_MODEL_SIMPLE && model_kind != IAN_MODEL_FULL && model_kind != IAN_MODEL_V1)
    return fail(nullptr, IAN_ERR_UNSUPPORTED, "unknown model kind %d", model_kind);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, IAN_ERR_CUDA, "no CUDA device: %s (this library has no CPU path)", cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(nullptr, IAN_ERR_INVALID, "device %d out of range [0,%d)", device, ndev);
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10)
    return fail(nullptr, IAN_ERR_UNSUPPORTED, "device %d is sm_%d%d; libian_b200 is built for sm_100a only", device, prop.major, prop.minor);
  ian_handle* h = new ian_handle();
  h->device = device;
  h->model_kind = model_kind;
  DeviceGuard dg(device);
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&h->h2d_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete h;
    return fail(nullptr, IAN_ERR_CUDA, "cudaStreamCreate failed");
  }
  if (const char* c = getenv("IAN_CHUNK")) { int v = atoi(c); if (v > 0) h->max_chunk = v > 4096 ? 4096 : v; }
  if (const char* c = getenv("IAN_PATH")) { if (!strcmp(c, "simt")) h->path = IAN_PATH_SIMT; }
  if (const char* c = getenv("IAN_STREAMK")) h->streamk = atoi(c) != 0;
  if (const char* c = getenv("IAN_SPLITK")) h->splitk = atoi(c) != 0;
  if (const char* c = getenv("IAN_TC2")) h->tc2 = atoi(c) != 0;
  if (const char* c = getenv("IAN_PDL")) h->pdl = atoi(c) != 0;
  if (const char* c = getenv("IAN_FINALIZE8")) h->coop_finalize = atoi(c) != 0;
  if (const char* c = getenv("IAN_TC2_MIN")) { int v = atoi(c); if (v > 0) h->tc2_min_tiles = v; }
  if (const char* c = getenv("IAN_GRAPHS")) h->graphs = atoi(c) != 0;
  *out = h;
  return IAN_OK;
}

int ian_set_param(ian_handle* h, const char* name, const float* data, const int64_t* shape, int ndim) {
  if (!h || !name || !data || !shape) return fail(h, IAN_ERR_INVALID, "NULL argument");
  if (h->finalized) return fail(h, IAN_ERR_STATE, "model already finalized");
  const std::vector<Spec> specs = spec_list(h->model_kind);
  const Spec* spec = nullptr;
  for (const auto& sp : specs)
    if (sp.name == name) spec = &sp;
  if (!spec) return fail(h, IAN_ERR_INVALID, "unknown parameter name '%s'", name);
  if (ndim != (int)spec->shape.size()) return fail(h, IAN_ERR_INVALID, "parameter %s: expected %d dims, got %d", name, (int)spec->shape.size(), ndim);
  int64_t elems = 1;
  for (int i = 0; i < ndim; ++i) {
    if (shape[i] != spec->shape[i])
      return fail(h, IAN_ERR_INVALID, "parameter %s: shape mismatch at dim %d (expected %lld, got %lld)", name, i,
                  (long long)spec->shape[i], (long long)shape[i]);
    elems *= shape[i];
  }
  HostParam& p = h->params[name];
  p.shape.assign(shape, shape + ndim);
  p.data.assign(data, data + elems);
  return IAN_OK;
}

int ian_set_made_ordering(ian_handle* h, const int32_t* ordering, int n) {
  if (!h || !ordering) return fail(h, IAN_ERR_INVALID, "NULL argument");
  if (h->finalized) return fail(h, IAN_ERR_STATE, "model already finalized");
  if (n != 100) return fail(h, IAN_ERR_INVALID, "ordering must have 100 entries (got %d)", n);
  std::vector<char> seen(100, 0);
  for (int i = 0; i < n; ++i) {
    if (ordering[i] < 0 || ordering[i] >= 100 || seen[ordering[i]]) return fail(h, IAN_ERR_INVALID, "ordering is not a permutation of 0..99");
    seen[ordering[i]] = 1;
  }
  h->made_ordering.assign(ordering, ordering + n);
  return IAN_OK;
}

// The model's OWN parameter list: what `lasagne.layers.get_all_params(...)` hands GANcheckpoints.load_weights in the
// reference (API.py:23-30).  A loader iterates these names and looks each one up in the checkpoint, so that extra keys
// of the file (log_sigma_theta, discriminator weights, metadata ...) are ignored exactly as the reference does.
static const std::vector<Spec>& cached_specs(int kind) {
  static std::vector<Spec> cache[3];
  static bool built[3] = {false, false, false};
  if (!built[kind]) { cache[kind] = spec_list(kind); built[kind] = true; }
  return cache[kind];
}

int ian_model_param_count(int model_kind) {
  if (model_kind < 0 || model_kind > 2) return IAN_ERR_INVALID;
  return (int)cached_specs(model_kind).size();
}

int ian_model_param_spec(int model_kind, int index, const char** name, int64_t* shape /*[4]*/, int* ndim) {
  if (model_kind < 0 || model_kind > 2 || !name || !shape || !ndim) return IAN_ERR_INVALID;
  const auto& v = cached_specs(model_kind);
  if (index < 0 || index >= (int)v.size()) return IAN_ERR_INVALID;
  *name = v[index].name.c_str();
  *ndim = (int)v[index].shape.size();
  for (int i = 0; i < 4; ++i) shape[i] = i < *ndim ? v[index].shape[i] : 1;
  return IAN_OK;
}

int ian_made_mask(const int32_t* ordering, int n, int which, uint8_t* mask_out /*[100][100], (in,out)*/) {
  if (!ordering || !mask_out || n != 100 || which < 0 || which > 2) return IAN_ERR_INVALID;
  for (int i = 0; i < 100; ++i)
    for (int j = 0; j < 100; ++j) mask_out[i * 100 + j] = made_keep(ordering, which, i, j) ? 1 : 0;
  return IAN_OK;
}

int ian_debug_made_weights(ian_handle* h, float* out /*[2][3][100][100]*/) {
  if (!h || !out) return IAN_ERR_INVALID;
  if (!h->finalized || !h->made_w) return fail(h, IAN_ERR_STATE, "no MADE weights on this handle (IAN_simple, or not finalized)");
  DeviceGuard dg(h->device);
  CUDA_TRY(h, cudaMemcpy(out, h->made_w, (size_t)2 * 3 * 10000 * sizeof(float), cudaMemcpyDeviceToHost));
  return IAN_OK;
}

int ian_finalize(ian_handle* h) {
  if (!h) return IAN_ERR_INVALID;
  if (h->finalized) return IAN_OK;
  for (const auto& sp : spec_list(h->model_kind))
    if (!h->params.count(sp.name)) return fail(h, IAN_ERR_STATE, "missing parameter '%s'", sp.name.c_str());
  DeviceGuard dg(h->device);
  int rc = prepare_encoder(h);
  if (rc != IAN_OK) return rc;
  rc = h->model_kind == IAN_MODEL_FULL ? prepare_full_decoder(h)
       : h->model_kind == IAN_MODEL_V1 ? prepare_v1_decoder(h) : prepare_simple_decoder(h);
  if (rc != IAN_OK) return rc;
  CUDA_TRY(h, cudaMalloc((void**)&h->sk_ws, tc_sk_workspace_floats() * sizeof(float)));
  CUDA_TRY(h, cudaMalloc((void**)&h->sk_flags, tc_sk_flag_ints() * sizeof(int)));
  CUDA_TRY(h, cudaMemset(h->sk_flags, 0, tc_sk_flag_ints() * sizeof(int)));
  h->params.clear();
  h->finalized = true;
  return IAN_OK;
}

int ian_destroy(ian_handle* h) {
  if (!h) return IAN_OK;
  DeviceGuard dg(h->device);
  cudaStreamSynchronize(h->stream);
  cudaStreamSynchronize(h->h2d_stream);
  cudaStreamSynchronize(h->d2h_stream);
  for (auto& kv : h->plans) free_plan(kv.second);
  for (auto& w : h->w) { cudaFree(w.b); cudaFree(w.scale); cudaFree(w.shift); }
  cudaFree(h->conv1_wt); cudaFree(h->conv1_b); cudaFree(h->decout_wt); cudaFree(h->decout_tc_wt);
  cudaFree(h->sk_ws); cudaFree(h->sk_flags);
  cudaFree(h->conv1_tc_wt); if (h->conv1_maps) conv1_free_maps(h->conv1_maps);
  cudaFree(h->made_w); cudaFree(h->made_b); cudaFree(h->head_taps); cudaFree(h->head_wgb); cudaFree(h->head_wbb);
  cudaFree(h->head_tc_wt);
  cudaFree(h->train_ws);
  for (auto& v : h->timed) for (auto& t : v) { cudaEventDestroy(t.e0); cudaEventDestroy(t.e1); }
  if (h->push_stream) { cudaStreamSynchronize(h->push_stream); cudaStreamDestroy(h->push_stream); }
  for (int b = 0; b < 2; ++b) { if (h->g_comp[b]) cudaEventDestroy(h->g_comp[b]); if (h->g_done[b]) cudaEventDestroy(h->g_done[b]); }
  for (int r = 0; r < h->gw; ++r) if (r != h->grank && h->gpeer_buf[r]) cudaIpcCloseMemHandle(h->gpeer_buf[r]);
  cudaFree(h->gbuf);
  for (void* p : h->host_allocs) cudaFreeHost(p);
  cudaStreamDestroy(h->stream);
  cudaStreamDestroy(h->h2d_stream);
  cudaStreamDestroy(h->d2h_stream);
  delete h;
  return IAN_OK;
}

const char* ian_last_error(const ian_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }
int ian_get_zdim(const ian_handle*) { return 100; }
int64_t ian_launch_count(const ian_handle* h) { return h ? h->launches : 0; }

int ian_set_path(ian_handle* h, int path) {
  if (!h) return IAN_ERR_INVALID;
  if (path != IAN_PATH_TC && path != IAN_PATH_SIMT) return fail(h, IAN_ERR_INVALID, "unknown path %d", path);
  h->path = path;
  return IAN_OK;
}

int ian_set_precision(ian_handle* h, int precision) {
  if (!h) return IAN_ERR_INVALID;
  if (precision != IAN_PRECISION_FP32 && precision != IAN_PRECISION_BF16) return fail(h, IAN_ERR_INVALID, "unknown precision %d", precision);
  if (precision == IAN_PRECISION_BF16 && h->model_kind == IAN_MODEL_SIMPLE)
    return fail(h, IAN_ERR_UNSUPPORTED, "bf16 mode is built for the IAN.py / IANv1.py graphs (BASELINE configs[2]); IAN_simple runs in float32");
  h->passes = precision == IAN_PRECISION_BF16 ? 1 : 3;
  return IAN_OK;
}

int ian_set_layer_timing(ian_handle* h, int enable) {
  if (!h) return IAN_ERR_INVALID;
  h->timing = enable != 0;
  return IAN_OK;
}

double ian_layer_time_ms(ian_handle* h, const char* layer_name, int reset) {
  if (!h || !layer_name) return -1.0;
  DeviceGuard dg(h->device);
  for (int l = 0; l < T_COUNT; ++l) {
    if (strcmp(kLayerNames[l], layer_name)) continue;
    for (auto& t : h->timed[l]) {
      float ms = 0.f;
      if (cudaEventSynchronize(t.e1) == cudaSuccess && cudaEventElapsedTime(&ms, t.e0, t.e1) == cudaSuccess) {
        h->time_ms[l] += ms;
        h->time_cnt[l] += 1;
      }
      cudaEventDestroy(t.e0);
      cudaEventDestroy(t.e1);
    }
    h->timed[l].clear();
    const double r = h->time_cnt[l] ? h->time_ms[l] / (double)h->time_cnt[l] : -1.0;
    if (reset) { h->time_ms[l] = 0; h->time_cnt[l] = 0; }
    return r;
  }
  return -1.0;
}

// ---- encode ---------------------------------------------------------------------------------------
int ian_encode_dev(ian_handle* h, const float* x, int n, const float* eps, float* z, void* stream) {
  int rc = check_ready(h, n, x, z);
  if (rc != IAN_OK) return rc;
  DeviceGuard dg(h->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  return for_chunks(h, n, [&](Plan* pl, int off, int) {
    return run_encode(h, pl, x + (size_t)off * 12288, eps ? eps + (size_t)off * 100 : nullptr, z + (size_t)off * 100, st);
  });
}

int ian_encode_host(ian_handle* h, const float* x, int n, const float* eps, float* z) {
  int rc = check_ready(h, n, x, z);
  if (rc != IAN_OK) return rc;
  DeviceGuard dg(h->device);
  cudaStream_t st = h->stream;
  rc = for_chunks(h, n, [&](Plan* pl, int off, int cn) {
    CUDA_TRY(h, cudaMemcpyAsync(pl->x, x + (size_t)off * 12288, (size_t)cn * 12288 * 4, cudaMemcpyHostToDevice, st));
    if (eps) CUDA_TRY(h, cudaMemcpyAsync(pl->eps, eps + (size_t)off * 100, (size_t)cn * 400, cudaMemcpyHostToDevice, st));
    int r = run_graphed(h, pl, eps ? Plan::G_ENCODE_EPS : Plan::G_ENCODE, 0, st,
                        [&] { return run_encode(h, pl, pl->x, eps ? pl->eps : nullptr, pl->z, st); });
    if (r != IAN_OK) return r;
    CUDA_TRY(h, cudaMemcpyAsync(z + (size_t)off * 100, pl->z, (size_t)cn * 400, cudaMemcpyDeviceToHost, st));
    return (int)IAN_OK;
  });
  if (rc != IAN_OK) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return IAN_OK;
}

// ---- decode ---------------------------------------------------------------------------------------
int ian_decode_dev(ian_handle* h, const float* z, int n, float* x, void* stream) {
  int rc = check_ready(h, n, z, x);
  if (rc != IAN_OK) return rc;
  DeviceGuard dg(h->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  return for_chunks(h, n, [&](Plan* pl, int off, int) {
    return run_decode(h, pl, z + (size_t)off * 100, x + (size_t)off * 12288, st);
  });
}

int ian_decode_host(ian_handle* h, const float* z, int n, float* x) {
  int rc = check_ready(h, n, z, x);
  if (rc != IAN_OK) return rc;
  DeviceGuard dg(h->device);
  cudaStream_t st = h->stream;
  rc = for_chunks(h, n, [&](Plan* pl, int off, int cn) {
    CUDA_TRY(h, cudaMemcpyAsync(pl->z, z + (size_t)off * 100, (size_t)cn * 400, cudaMemcpyHostToDevice, st));
    int r = run_graphed(h, pl, Plan::G_DECODE, 0, st, [&] { return run_decode(h, pl, pl->z, pl->xhat, st); });
    if (r != IAN_OK) return r;
    CUDA_TRY(h, cudaMemcpyAsync(x + (size_t)off * 12288, pl->xhat, (size_t)cn * 12288 * 4, cudaMemcpyDeviceToHost, st));
    return (int)IAN_OK;
  });
  if (rc != IAN_OK) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return IAN_OK;
}

// ---- encode -> decode -----------------------------------------------------------------------------
int ian_reconstruct_dev(ian_handle* h, const float* x, int n, float* z_out, float* x_hat, void* stream) {
  int rc = check_ready(h, n, x, x_hat);
  if (rc != IAN_OK) return rc;
  DeviceGuard dg(h->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  return for_chunks(h, n, [&](Plan* pl, int off, int) {
    int r = run_encode(h, pl, x + (size_t)off * 12288, nullptr, z_out ? z_out + (size_t)off * 100 : nullptr, st);
    if (r != IAN_OK) return r;
    return run_decode_from_planes(h, pl, x_hat + (size_t)off * 12288, st);
  });
}

int ian_reconstruct_host(ian_handle* h, const float* x, int n, float* z_out, float* x_hat) {
  int rc = check_ready(h, n, x, x_hat);
  if (rc != IAN_OK) return rc;
  DeviceGuard dg(h->device);
  cudaStream_t st = h->stream;
  rc = for_chunks(h, n, [&](Plan* pl, int off, int cn) {
    CUDA_TRY(h, cudaMemcpyAsync(pl->x, x + (size_t)off * 12288, (size_t)cn * 12288 * 4, cudaMemcpyHostToDevice, st));
    int r = run_graphed(h, pl, Plan::G_RECON, 0, st, [&] {
      int q = run_encode(h, pl, pl->x, nullptr, pl->z, st);
      return q != IAN_OK ? q : run_decode_from_planes(h, pl, pl->xhat, st);
    });
    if (r != IAN_OK) return r;
    if (z_out) CUDA_TRY(h, cudaMemcpyAsync(z_out + (size_t)off * 100, pl->z, (size_t)cn * 400, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaMemcpyAsync(x_hat + (size_t)off * 12288, pl->xhat, (size_t)cn * 12288 * 4, cudaMemcpyDeviceToHost, st));
    return (int)IAN_OK;
  });
  if (rc != IAN_OK) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return IAN_OK;
}

// ---- brush gradient -------------------------------------------------------------------------------
int ian_grad_dev(ian_handle* h, const float* z, const int32_t* boxes, const float* target, int target_is_frame, int n,
                 float* g, void* stream) {
  int rc = check_ready(h, n, z, g);
  if (rc != IAN_OK) return rc;
  if (!boxes) return fail(h, IAN_ERR_INVALID, "boxes is NULL");
  DeviceGuard dg(h->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  const size_t tstride = target_is_frame ? 12288 : 3;
  return for_chunks(h, n, [&](Plan* pl, int off, int cn) {
    LAUNCH_TRY(h, launch_z_to_planes(z + (size_t)off * 100, pl->zp.p, pl->zp.plane, cn, st));
    int r = run_grad_core(h, pl, boxes + (size_t)off * 4, target ? target + off * tstride : nullptr, target_is_frame, st);
    if (r != IAN_OK) return r;
    LAUNCH_TRY(h, launch_brush_update(pl->gpad, boxes + (size_t)off * 4, 0.f, g + (size_t)off * 100, nullptr, nullptr, 0, cn, st));
    return (int)IAN_OK;
  });
}

int ian_grad_host(ian_handle* h, const float* z, const int32_t* boxes, const float* target, int target_is_frame, int n,
                  float* g) {
  int rc = check_ready(h, n, z, g);
  if (rc != IAN_OK) return rc;
  if (!boxes) return fail(h, IAN_ERR_INVALID, "boxes is NULL");
  if ((rc = validate_boxes(h, boxes, n)) != IAN_OK) return rc;
  DeviceGuard dg(h->device);
  cudaStream_t st = h->stream;
  const size_t tstride = target_is_frame ? 12288 : 3;
  rc = for_chunks(h, n, [&](Plan* pl, int off, int cn) {
    CUDA_TRY(h, cudaMemcpyAsync(pl->z, z + (size_t)off * 100, (size_t)cn * 400, cudaMemcpyHostToDevice, st));
    CUDA_TRY(h, cudaMemcpyAsync(pl->boxes, boxes + (size_t)off * 4, (size_t)cn * 16, cudaMemcpyHostToDevice, st));
    if (target) CUDA_TRY(h, cudaMemcpyAsync(pl->target, target + off * tstride, cn * tstride * 4, cudaMemcpyHostToDevice, st));
    int r = run_graphed(h, pl, Plan::G_GRAD, (target ? 1 : 0) + (target_is_frame ? 2 : 0), st, [&] {
      LAUNCH_TRY(h, launch_z_to_planes(pl->z, pl->zp.p, pl->zp.plane, cn, st));
      int q = run_grad_core(h, pl, pl->boxes, target ? pl->target : nullptr, target_is_frame, st);
      if (q != IAN_OK) return q;
      LAUNCH_TRY(h, launch_brush_update(pl->gpad, pl->boxes, 0.f, pl->z /*reuse as g staging*/, nullptr, nullptr, 0, cn, st));
      return (int)IAN_OK;
    });
    if (r != IAN_OK) return r;
    CUDA_TRY(h, cudaMemcpyAsync(g + (size_t)off * 100, pl->z, (size_t)cn * 400, cudaMemcpyDeviceToHost, st));
    return (int)IAN_OK;
  });
  if (rc != IAN_OK) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return IAN_OK;
}

// ---- edit loop ------------------------------------------------------------------------------------
int ian_edit_loop_dev(ian_handle* h, float* z, const int32_t* boxes, const float* target, int target_is_frame, int n,
                      int n_steps, float weight, void* stream) {
  int rc = check_ready(h, n, z, z);
  if (rc != IAN_OK) return rc;
  if (!boxes) return fail(h, IAN_ERR_INVALID, "boxes is NULL");
  if (n_steps < 0) return fail(h, IAN_ERR_INVALID, "n_steps < 0");
  DeviceGuard dg(h->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  const size_t tstride = target_is_frame ? 12288 : 3;
  return for_chunks(h, n, [&](Plan* pl, int off, int cn) {
    float* zc = z + (size_t)off * 100;
    LAUNCH_TRY(h, launch_z_to_planes(zc, pl->zp.p, pl->zp.plane, cn, st));
    for (int s = 0; s < n_steps; ++s) {
      int r = run_grad_core(h, pl, boxes + (size_t)off * 4, target ? target + off * tstride : nullptr, target_is_frame, st);
      if (r != IAN_OK) return r;
      LAUNCH_TRY(h, launch_brush_update(pl->gpad, boxes + (size_t)off * 4, weight, nullptr, zc, pl->zp.p, pl->zp.plane, cn, st));
    }
    return (int)IAN_OK;
  });
}

int ian_edit_loop_host(ian_handle* h, float* z, const int32_t* boxes, const float* target, int target_is_frame, int n,
                       int n_steps, float weight) {
  int rc = check_ready(h, n, z, z);
  if (rc != IAN_OK) return rc;
  if (!boxes) return fail(h, IAN_ERR_INVALID, "boxes is NULL");
  if ((rc = validate_boxes(h, boxes, n)) != IAN_OK) return rc;
  DeviceGuard dg(h->device);
  cudaStream_t st = h->stream;
  const size_t tstride = target_is_frame ? 12288 : 3;
  rc = for_chunks(h, n, [&](Plan* pl, int off, int cn) {
    CUDA_TRY(h, cudaMemcpyAsync(pl->z, z + (size_t)off * 100, (size_t)cn * 400, cudaMemcpyHostToDevice, st));
    CUDA_TRY(h, cudaMemcpyAsync(pl->boxes, boxes + (size_t)off * 4, (size_t)cn * 16, cudaMemcpyHostToDevice, st));
    if (target) CUDA_TRY(h, cudaMemcpyAsync(pl->target, target + off * tstride, cn * tstride * 4, cudaMemcpyHostToDevice, st));
    LAUNCH_TRY(h, launch_z_to_planes(pl->z, pl->zp.p, pl->zp.plane, cn, st));
    const uint64_t key = float_bits(weight) * 4 + (target ? 1 : 0) + (target_is_frame ? 2 : 0);
    for (int s = 0; s < n_steps; ++s) {                    // one graph = one paint step, replayed n_steps times
      int r = run_graphed(h, pl, Plan::G_EDIT_STEP, key, st, [&] {
        int q = run_grad_core(h, pl, pl->boxes, target ? pl->target : nullptr, target_is_frame, st);
        if (q != IAN_OK) return q;
        LAUNCH_TRY(h, launch_brush_update(pl->gpad, pl->boxes, weight, nullptr, pl->z, pl->zp.p, pl->zp.plane, cn, st));
        return (int)IAN_OK;
      });
      if (r != IAN_OK) return r;
    }
    CUDA_TRY(h, cudaMemcpyAsync(z + (size_t)off * 100, pl->z, (size_t)cn * 400, cudaMemcpyDeviceToHost, st));
    return (int)IAN_OK;
  });
  if (rc != IAN_OK) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return IAN_OK;
}


// ---- pipelined host API -----------------------------------------------------------------------------
int ian_host_alloc(ian_handle* h, size_t bytes, void** out) {
  if (!h || !out || bytes == 0) return fail(h, IAN_ERR_INVALID, "bad argument");
  DeviceGuard dg(h->device);
  void* p = nullptr;
  CUDA_TRY(h, cudaHostAlloc(&p, bytes, cudaHostAllocDefault));
  h->host_allocs.push_back(p);
  *out = p;
  return IAN_OK;
}

int ian_host_free(ian_handle* h, void* p) {
  if (!h || !p) return IAN_ERR_INVALID;
  for (size_t i = 0; i < h->host_allocs.size(); ++i)
    if (h->host_allocs[i] == p) {
      h->host_allocs.erase(h->host_allocs.begin() + i);
      DeviceGuard dg(h->device);
      CUDA_TRY(h, cudaFreeHost(p));
      return IAN_OK;
    }
  return fail(h, IAN_ERR_INVALID, "pointer was not allocated by ian_host_alloc");
}

int ian_reconstruct_submit(ian_handle* h, const float* x, int n, float* z_out, float* x_hat, int* ticket) {
  int rc = check_ready(h, n, x, x_hat);
  if (rc != IAN_OK) return rc;
  if (!ticket) return fail(h, IAN_ERR_INVALID, "ticket is NULL");
  if (n > h->max_chunk) return fail(h, IAN_ERR_INVALID, "pipelined calls take at most %d images (got %d)", h->max_chunk, n);
  DeviceGuard dg(h->device);
  Plan* pl = nullptr;
  if ((rc = get_plan(h, n, &pl)) != IAN_OK) return rc;
  const int s = (int)(h->tickets & 1);
  if (h->inflight[s].id >= 0) {                          // the request that used this slot two submits ago (any plan) is done
    auto prev = h->plans.find(h->inflight[s].n);
    if (prev != h->plans.end() && prev->second->ev_d2h[s]) CUDA_TRY(h, cudaEventSynchronize(prev->second->ev_d2h[s]));
  }
  if (!pl->sx[s]) {
    for (int b = 0; b < 2; ++b) {
      if ((rc = alloc_buf(h, pl, pl->sx[b], (long long)n * 12288)) != IAN_OK) return rc;
      if ((rc = alloc_buf(h, pl, pl->sz[b], (long long)n * 100)) != IAN_OK) return rc;
      if ((rc = alloc_buf(h, pl, pl->sxh[b], (long long)n * 12288)) != IAN_OK) return rc;
      CUDA_TRY(h, cudaEventCreateWithFlags(&pl->ev_h2d[b], cudaEventDisableTiming));
      CUDA_TRY(h, cudaEventCreateWithFlags(&pl->ev_comp[b], cudaEventDisableTiming));
      CUDA_TRY(h, cudaEventCreateWithFlags(&pl->ev_d2h[b], cudaEventDisableTiming));
    }
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));     // the memsets of the new buffers
  }
  CUDA_TRY(h, cudaMemcpyAsync(pl->sx[s], x, (size_t)n * 12288 * 4, cudaMemcpyHostToDevice, h->h2d_stream));
  CUDA_TRY(h, cudaEventRecord(pl->ev_h2d[s], h->h2d_stream));
  CUDA_TRY(h, cudaStreamWaitEvent(h->stream, pl->ev_h2d[s], 0));
  if ((rc = run_encode(h, pl, pl->sx[s], nullptr, pl->sz[s], h->stream)) != IAN_OK) return rc;
  if ((rc = run_decode_from_planes(h, pl, pl->sxh[s], h->stream)) != IAN_OK) return rc;
  CUDA_TRY(h, cudaEventRecord(pl->ev_comp[s], h->stream));
  CUDA_TRY(h, cudaStreamWaitEvent(h->d2h_stream, pl->ev_comp[s], 0));
  CUDA_TRY(h, cudaMemcpyAsync(x_hat, pl->sxh[s], (size_t)n * 12288 * 4, cudaMemcpyDeviceToHost, h->d2h_stream));
  if (z_out) CUDA_TRY(h, cudaMemcpyAsync(z_out, pl->sz[s], (size_t)n * 400, cudaMemcpyDeviceToHost, h->d2h_stream));
  CUDA_TRY(h, cudaEventRecord(pl->ev_d2h[s], h->d2h_stream));
  const int id = (int)(h->tickets & 0x7fffffff);             // monotonically increasing; mapped to (plan, slot) below
  h->inflight[s].id = id; h->inflight[s].n = n; h->inflight[s].slot = s;
  *ticket = id;
  h->tickets += 1;
  return IAN_OK;
}

int ian_reconstruct_wait(ian_handle* h, int ticket) {
  if (!h) return IAN_ERR_INVALID;
  if (ticket < 0 || (long long)ticket >= h->tickets) return fail(h, IAN_ERR_INVALID, "unknown ticket %d", ticket);
  const ian_handle::Ticket* tk = nullptr;
  for (const auto& t : h->inflight) if (t.id == ticket) tk = &t;
  if (!tk) return IAN_OK;      // older than the two requests in flight: its slot was reused, i.e. it completed (submit waited)
  auto it = h->plans.find(tk->n);
  if (it == h->plans.end() || !it->second->ev_d2h[tk->slot]) return fail(h, IAN_ERR_INVALID, "unknown ticket %d", ticket);
  DeviceGuard dg(h->device);
  CUDA_TRY(h, cudaEventSynchronize(it->second->ev_d2h[tk->slot]));
  return IAN_OK;
}

// ---- sample_IAN.py function set (reference sample_IAN.py:86-94) ----------------------------------------
// Zfn: X -> l_Z_IAF (deterministic: mu).  For IAN_simple there is no flow and this equals ian_encode_host.
int ian_encode_pre_host(ian_handle* h, const float* x, int n, float* z_iaf) {
  int rc = check_ready(h, n, x, z_iaf);
  if (rc != IAN_OK) return rc;
  DeviceGuard dg(h->device);
  cudaStream_t st = h->stream;
  rc = for_chunks(h, n, [&](Plan* pl, int off, int cn) {
    CUDA_TRY(h, cudaMemcpyAsync(pl->x, x + (size_t)off * 12288, (size_t)cn * 12288 * 4, cudaMemcpyHostToDevice, st));
    int r = run_encode(h, pl, pl->x, nullptr, pl->z, st, pl->eps /*staging for l_Z_IAF*/);
    if (r != IAN_OK) return r;
    CUDA_TRY(h, cudaMemcpyAsync(z_iaf + (size_t)off * 100, pl->eps, (size_t)cn * 400, cudaMemcpyDeviceToHost, st));
    return (int)IAN_OK;
  });
  if (rc != IAN_OK) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return IAN_OK;
}

// Z_IAF_fn: l_Z_IAF -> l_Z = (z - MADE_mu(z)) / exp(MADE_ls(z)); identity for IAN_simple.
// x_out != NULL additionally decodes: `sample` of sample_IAN.py:86 (l_Z_IAF -> X).
int ian_flow_host(ian_handle* h, const float* z_iaf, int n, float* z_out /*nullable*/, float* x_out /*nullable*/) {
  int rc = check_ready(h, n, z_iaf, z_iaf);
  if (rc != IAN_OK) return rc;
  if (!z_out && !x_out) return fail(h, IAN_ERR_INVALID, "both outputs are NULL");
  DeviceGuard dg(h->device);
  cudaStream_t st = h->stream;
  rc = for_chunks(h, n, [&](Plan* pl, int off, int cn) {
    CUDA_TRY(h, cudaMemcpyAsync(pl->eps, z_iaf + (size_t)off * 100, (size_t)cn * 400, cudaMemcpyHostToDevice, st));
    if (has_flow(h))
      LAUNCH_TRY(h, launch_made_iaf(pl->eps, h->made_w, h->made_b, pl->z, pl->zp.p, pl->zp.plane, cn, st));
    else {
      CUDA_TRY(h, cudaMemcpyAsync(pl->z, pl->eps, (size_t)cn * 400, cudaMemcpyDeviceToDevice, st));
      LAUNCH_TRY(h, launch_z_to_planes(pl->z, pl->zp.p, pl->zp.plane, cn, st));
    }
    if (z_out) CUDA_TRY(h, cudaMemcpyAsync(z_out + (size_t)off * 100, pl->z, (size_t)cn * 400, cudaMemcpyDeviceToHost, st));
    if (x_out) {
      int r = run_decode_from_planes(h, pl, pl->xhat, st);
      if (r != IAN_OK) return r;
      CUDA_TRY(h, cudaMemcpyAsync(x_out + (size_t)off * 12288, pl->xhat, (size_t)cn * 12288 * 4, cudaMemcpyDeviceToHost, st));
    }
    return (int)IAN_OK;
  });
  if (rc != IAN_OK) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return IAN_OK;
}

// ---- fused all-gather of decoded images over NVLink peer memory ---------------------------------------------
static size_t gather_bytes(int world, int n_local) { return (size_t)2 * world * n_local * 12288 * sizeof(float) + 256; }

int ian_gather_create(ian_handle* h, int world, int rank, int n_local, void* ipc_handle_out) {
  if (!h || !ipc_handle_out) return fail(h, IAN_ERR_INVALID, "NULL argument");
  if (!h->finalized) return fail(h, IAN_ERR_STATE, "ian_finalize() has not been called");
  if (world < 1 || world > 8 || rank < 0 || rank >= world || n_local < 1 || n_local > 65536)
    return fail(h, IAN_ERR_INVALID, "bad world/rank/n_local (%d,%d,%d)", world, rank, n_local);
  if (h->gbuf) return fail(h, IAN_ERR_STATE, "gather buffers already created");
  DeviceGuard dg(h->device);
  CUDA_TRY(h, cudaMalloc((void**)&h->gbuf, gather_bytes(world, n_local)));
  CUDA_TRY(h, cudaMemset(h->gbuf, 0, gather_bytes(world, n_local)));
  cudaIpcMemHandle_t ipc;
  CUDA_TRY(h, cudaIpcGetMemHandle(&ipc, h->gbuf));
  memcpy(ipc_handle_out, &ipc, sizeof(ipc));
  h->gw = world; h->grank = rank; h->gn = n_local;
  return IAN_OK;
}

int ian_gather_connect(ian_handle* h, const void* all_handles) {
  if (!h || !all_handles || !h->gbuf) return fail(h, IAN_ERR_STATE, "ian_gather_create() first");
  DeviceGuard dg(h->device);
  for (int r = 0; r < h->gw; ++r) {
    if (r == h->grank) { h->gpeer_buf[r] = h->gbuf; continue; }
    cudaIpcMemHandle_t ipc;
    memcpy(&ipc, (const char*)all_handles + (size_t)r * sizeof(ipc), sizeof(ipc));
    void* p = nullptr;
    CUDA_TRY(h, cudaIpcOpenMemHandle(&p, ipc, cudaIpcMemLazyEnablePeerAccess));
    h->gpeer_buf[r] = (float*)p;
  }
  h->gconnected = true;
  return IAN_OK;
}

namespace {
struct GatherSlots { float* dsts[8]; float* flags[8]; size_t half, mine; };
GatherSlots gather_slots(const ian_handle* h) {
  GatherSlots g;
  g.half = (size_t)h->gw * h->gn * 12288;                         // floats per gather buffer
  g.mine = (size_t)h->grank * h->gn * 12288;
  for (int r = 0; r < h->gw; ++r) {
    g.dsts[r] = h->gpeer_buf[r] + (size_t)h->gcur * g.half + g.mine;   // my shard's slot in rank r's current buffer
    g.flags[r] = h->gpeer_buf[r] + 2 * g.half;                    // rank r's flag block (64 ints) after its buffers
  }
  return g;
}

int check_gather_ready(ian_handle* h, const float* x, int n_local) {
  int rc = check_ready(h, n_local, x, x);
  if (rc != IAN_OK) return rc;
  if (!h->gconnected) return fail(h, IAN_ERR_STATE, "ian_gather_connect() has not been called");
  if (n_local != h->gn) return fail(h, IAN_ERR_INVALID, "n_local %d differs from the %d the gather buffers were sized for", n_local, h->gn);
  if (h->path != IAN_PATH_TC) return fail(h, IAN_ERR_UNSUPPORTED, "fused gather runs on the tensor-core path");
  return IAN_OK;
}

// encode -> decode of the local shard (in <= 512-image chunks), the decoder's last kernel (dec_out, or the RGB-Beta head
// of the flow graphs) storing into `ndst` destination bases
int run_shard_into(ian_handle* h, const float* x, int n_local, float* z_out, float* const* bases, int ndst, cudaStream_t st) {
  return for_chunks(h, n_local, [&](Plan* pl, int off, int) {
    float* dsts[8];
    for (int r = 0; r < ndst; ++r) dsts[r] = bases[r] + (size_t)off * 12288;
    int rc = run_encode(h, pl, x + (size_t)off * 12288, nullptr, z_out ? z_out + (size_t)off * 100 : pl->z, st);
    if (rc != IAN_OK) return rc;
    h->gather_dsts = dsts; h->gather_ndst = ndst;
    rc = run_decode_from_planes(h, pl, nullptr, st);
    h->gather_dsts = nullptr; h->gather_ndst = 0;
    return rc;
  });
}
}  // namespace

int ian_reconstruct_gather_dev(ian_handle* h, const float* x, int n_local, float* z_out, float** gathered_out, void* stream) {
  if (!gathered_out) return fail(h, IAN_ERR_INVALID, "gathered_out is NULL");
  int rc = check_gather_ready(h, x, n_local);
  if (rc != IAN_OK) return rc;
  DeviceGuard dg(h->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  if (h->g_done_valid[h->gcur]) {                                  // an earlier pipelined step still owns this half
    CUDA_TRY(h, cudaStreamWaitEvent(st, h->g_done[h->gcur], 0));
    h->g_done_valid[h->gcur] = false;
  }
  GatherSlots g = gather_slots(h);
  if ((rc = run_shard_into(h, x, n_local, z_out, g.dsts, h->gw, st)) != IAN_OK) return rc;   // peer stores from the decoder's last kernel
  h->gepoch += 1;
  LAUNCH_TRY(h, launch_peer_barrier(g.flags, h->gw, h->grank, h->gepoch, st));
  *gathered_out = h->gbuf + (size_t)h->gcur * g.half;
  h->gcur ^= 1;
  h->g_last = -1;
  return IAN_OK;
}

// Pipelined form: the shard is decoded into this rank's own buffer on `stream`; a small copy kernel on a side stream
// then pushes it to every peer while the caller's NEXT step computes.  ian_gather_wait_dev makes `stream` wait for the
// most recent step's gather and returns its buffer.
int ian_reconstruct_gather_async_dev(ian_handle* h, const float* x, int n_local, float* z_out, void* stream) {
  int rc = check_gather_ready(h, x, n_local);
  if (rc != IAN_OK) return rc;
  DeviceGuard dg(h->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  if (!h->push_stream) {
    CUDA_TRY(h, cudaStreamCreateWithFlags(&h->push_stream, cudaStreamNonBlocking));
    for (int b = 0; b < 2; ++b) {
      CUDA_TRY(h, cudaEventCreateWithFlags(&h->g_comp[b], cudaEventDisableTiming));
      CUDA_TRY(h, cudaEventCreateWithFlags(&h->g_done[b], cudaEventDisableTiming));
    }
    if (const char* c = getenv("IAN_PUSH_CTAS")) { int v = atoi(c); if (v >= 1 && v <= 148) h->push_ctas = v; }
    if (const char* c = getenv("IAN_PUSH")) h->push_mode = !strcmp(c, "kernel") ? 1 : 0;
  }
  const int half_id = h->gcur;
  if (h->g_done_valid[half_id]) CUDA_TRY(h, cudaStreamWaitEvent(st, h->g_done[half_id], 0));   // push of step t-2 has read this half
  GatherSlots g = gather_slots(h);
  float* local[1] = {g.dsts[h->grank]};
  if ((rc = run_shard_into(h, x, n_local, z_out, local, 1, st)) != IAN_OK) return rc;
  CUDA_TRY(h, cudaEventRecord(h->g_comp[half_id], st));
  CUDA_TRY(h, cudaStreamWaitEvent(h->push_stream, h->g_comp[half_id], 0));
  h->gepoch += 1;
  const MemOps& mo = memops();
  if (h->push_mode == 0 && mo.write && mo.wait) {
    // copy engines + stream memory operations: nothing of the push occupies an SM, so the next step's persistent tensor
    // kernels keep all 148 (a co-resident copy KERNEL held its SMs' shared-memory configuration and cost the first three
    // tap-GEMMs of the next step +60 % at 8 GPUs).  Order on the side stream: publish free[t] to every peer; per peer wait
    // for ITS free[t], then DMA the shard into its buffer; publish pushed[t]; wait for everybody's pushed[t].
    CUstream ps = (CUstream)h->push_stream;
    const size_t bytes = (size_t)n_local * 12288 * sizeof(float);
    auto flag = [&](int r, int idx) { return (CUdeviceptr)(uintptr_t)(reinterpret_cast<int*>(g.flags[r]) + idx); };
    for (int k = 1; k < h->gw; ++k) {
      const int p = (h->grank + k) % h->gw;
      if (mo.write(ps, flag(p, 8 + h->grank), (cuuint32_t)h->gepoch, CU_STREAM_WRITE_VALUE_DEFAULT) != CUDA_SUCCESS)
        return fail(h, IAN_ERR_CUDA, "cuStreamWriteValue32(free) failed");
    }
    for (int k = 1; k < h->gw; ++k) {
      const int p = (h->grank + k) % h->gw;
      if (mo.wait(ps, flag(h->grank, 8 + p), (cuuint32_t)h->gepoch, CU_STREAM_WAIT_VALUE_GEQ) != CUDA_SUCCESS)
        return fail(h, IAN_ERR_CUDA, "cuStreamWaitValue32(free) failed");
      CUDA_TRY(h, cudaMemcpyAsync(g.dsts[p], g.dsts[h->grank], bytes, cudaMemcpyDeviceToDevice, h->push_stream));
    }
    for (int p = 0; p < h->gw; ++p)
      if (mo.write(ps, flag(p, 16 + h->grank), (cuuint32_t)h->gepoch, CU_STREAM_WRITE_VALUE_DEFAULT) != CUDA_SUCCESS)
        return fail(h, IAN_ERR_CUDA, "cuStreamWriteValue32(pushed) failed");
    for (int p = 0; p < h->gw; ++p)
      if (mo.wait(ps, flag(h->grank, 16 + p), (cuuint32_t)h->gepoch, CU_STREAM_WAIT_VALUE_GEQ) != CUDA_SUCCESS)
        return fail(h, IAN_ERR_CUDA, "cuStreamWaitValue32(pushed) failed");
  } else {
    LAUNCH_TRY(h, launch_peer_push(g.dsts[h->grank], g.dsts, g.flags, (long long)n_local * 12288, h->gw, h->grank, h->gepoch,
                                   h->push_ctas, h->push_stream));
  }
  CUDA_TRY(h, cudaEventRecord(h->g_done[half_id], h->push_stream));
  h->g_done_valid[half_id] = true;
  h->g_last = half_id;
  h->gcur ^= 1;
  return IAN_OK;
}

int ian_gather_wait_dev(ian_handle* h, float** gathered_out, void* stream) {
  if (!h || !gathered_out) return fail(h, IAN_ERR_INVALID, "NULL argument");
  if (h->g_last < 0) return fail(h, IAN_ERR_STATE, "no pipelined gather step is outstanding");
  DeviceGuard dg(h->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  CUDA_TRY(h, cudaStreamWaitEvent(st, h->g_done[h->g_last], 0));
  *gathered_out = h->gbuf + (size_t)h->g_last * ((size_t)h->gw * h->gn * 12288);
  return IAN_OK;
}

// ---- training-mode pieces (SURVEY 8f rank 4; the trainers themselves stay the reference's) ------------------------------
static int ensure_train_ws(ian_handle* h, size_t bytes) {
  if (bytes <= h->train_ws_bytes) return IAN_OK;
  if (h->train_ws) { CUDA_TRY(h, cudaDeviceSynchronize()); CUDA_TRY(h, cudaFree(h->train_ws)); h->train_ws = nullptr; h->train_ws_bytes = 0; }
  CUDA_TRY(h, cudaMalloc(&h->train_ws, bytes));
  h->train_ws_bytes = bytes;
  return IAN_OK;
}

int ian_bn_batch_stats_dev(ian_handle* h, const float* x, int n, int c, int hw, double* sum, double* sumsq, void* stream) {
  if (!h) return IAN_ERR_INVALID;
  if (!x || !sum || !sumsq || n < 1 || c < 1 || hw < 1) return fail(h, IAN_ERR_INVALID, "bad argument (n=%d c=%d hw=%d)", n, c, hw);
  DeviceGuard dg(h->device);
  int rc = ensure_train_ws(h, bn_workspace_bytes(c));
  if (rc != IAN_OK) return rc;
  LAUNCH_TRY(h, launch_bn_batch_stats(x, n, c, hw, sum, sumsq, h->train_ws, stream ? (cudaStream_t)stream : h->stream));
  return IAN_OK;
}

int ian_bn_train_normalize_dev(ian_handle* h, const float* x, int n, int c, int hw, const double* sum, const double* sumsq,
                               double count, const float* gamma, const float* beta, float eps, float alpha, float* running_mean,
                               float* running_inv_std, float* y, void* stream) {
  if (!h) return IAN_ERR_INVALID;
  if (!x || !y || !sum || !sumsq || n < 1 || c < 1 || hw < 1 || !(count >= 1.0))
    return fail(h, IAN_ERR_INVALID, "bad argument (n=%d c=%d hw=%d count=%g)", n, c, hw, count);
  DeviceGuard dg(h->device);
  int rc = ensure_train_ws(h, bn_workspace_bytes(c));
  if (rc != IAN_OK) return rc;
  LAUNCH_TRY(h, launch_bn_train_normalize(x, n, c, hw, sum, sumsq, count, gamma, beta, eps, alpha, running_mean, running_inv_std, y,
                                          h->train_ws, stream ? (cudaStream_t)stream : h->stream));
  return IAN_OK;
}

int ian_minibatch_discrim_dev(ian_handle* h, const float* x, int n, int d, const float* theta, const float* log_weight_scale,
                              const float* b, int num_kernels, int dim_per_kernel, float* out, void* stream) {
  if (!h) return IAN_ERR_INVALID;
  if (!x || !theta || !log_weight_scale || !b || !out || n < 1 || d < 1 || num_kernels < 1 || dim_per_kernel < 1)
    return fail(h, IAN_ERR_INVALID, "bad argument");
  DeviceGuard dg(h->device);
  int rc = ensure_train_ws(h, mb_workspace_bytes(n, num_kernels, dim_per_kernel));
  if (rc != IAN_OK) return rc;
  LAUNCH_TRY(h, launch_minibatch_discrim(x, n, d, theta, log_weight_scale, b, num_kernels, dim_per_kernel, out, h->train_ws,
                                         stream ? (cudaStream_t)stream : h->stream));
  return IAN_OK;
}

// ---- one NPE paint stroke in one call (reference NPE.py:192-235, photo mode) ---------------------------------
int ian_paint_stroke_host(ian_handle* h, float* z, const int32_t* box, const float* rgb_frame, float weight,
                          const uint8_t* recon_u8, const float* error, uint8_t* im_u8, uint8_t* display_u8) {
  int rc = check_ready(h, 1, z, rgb_frame);
  if (rc != IAN_OK) return rc;
  if (!box || !recon_u8 || !error || !im_u8) return fail(h, IAN_ERR_INVALID, "NULL argument");
  if ((rc = validate_boxes(h, box, 1)) != IAN_OK) return rc;
  DeviceGuard dg(h->device);
  cudaStream_t st = h->stream;
  Plan* pl = nullptr;
  if ((rc = get_plan(h, 1, &pl)) != IAN_OK) return rc;
  // staging buffer of the stroke: error (float32) | recon (u8) | IM (u8) | display (u8 HWC)
  if (!pl->stroke) {
    uint8_t* p = nullptr;
    if ((rc = alloc_buf(h, pl, p, 49152 + 12288 + 12288 + 256 * 256 * 3)) != IAN_OK) return rc;
    pl->stroke = p;
  }
  float* d_error = reinterpret_cast<float*>(pl->stroke);
  uint8_t* d_recon = pl->stroke + 49152;
  uint8_t* d_im = d_recon + 12288;
  uint8_t* d_disp = d_im + 12288;
  CUDA_TRY(h, cudaMemcpyAsync(pl->z, z, 400, cudaMemcpyHostToDevice, st));
  CUDA_TRY(h, cudaMemcpyAsync(pl->boxes, box, 16, cudaMemcpyHostToDevice, st));
  CUDA_TRY(h, cudaMemcpyAsync(pl->target, rgb_frame, 12288 * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(h, cudaMemcpyAsync(d_recon, recon_u8, 12288, cudaMemcpyHostToDevice, st));
  CUDA_TRY(h, cudaMemcpyAsync(d_error, error, 12288 * 4, cudaMemcpyHostToDevice, st));
  rc = run_graphed(h, pl, Plan::G_STROKE, float_bits(weight), st, [&] {
    LAUNCH_TRY(h, launch_z_to_planes(pl->z, pl->zp.p, pl->zp.plane, 1, st));
    int q = run_grad_core(h, pl, pl->boxes, pl->target, 1, st);                                    // NPE.py:205
    if (q != IAN_OK) return q;
    LAUNCH_TRY(h, launch_brush_update(pl->gpad, pl->boxes, weight, nullptr, pl->z, pl->zp.p, pl->zp.plane, 1, st));  // :206-209
    if ((q = run_decode_from_planes(h, pl, pl->xhat, st)) != IAN_OK) return q;                     // NPE.py:218 sample_at
    LAUNCH_TRY(h, launch_npe_blend(pl->xhat, d_recon, d_error, d_im, d_disp, st));                  // NPE.py:218-231
    return (int)IAN_OK;
  });
  if (rc != IAN_OK) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(z, pl->z, 400, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaMemcpyAsync(im_u8, d_im, 12288, cudaMemcpyDeviceToHost, st));
  if (display_u8) CUDA_TRY(h, cudaMemcpyAsync(display_u8, d_disp, 256 * 256 * 3, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return IAN_OK;
}

}  // extern "C"
