// libb200tts.so -- C-ABI entry points (include/b200tts.h), weight packing and launch logic.
#include "../../include/b200tts.h"

#include <cooperative_groups.h>
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"
#include "wavernn_upsample.cuh"
#include "wavernn_utt.cuh"
#include "wavernn_grid.cuh"
#include "wavernn_push.cuh"
#include "wavernn_pushmg.cuh"
#include "wavernn_tc.cuh"
#include "taco_decoder.cuh"
#include "taco_encpost.cuh"
#include "taco_grid.cuh"

using namespace b200tts;

static thread_local std::string g_err;

#define API_BEGIN try {
#define API_END                                       \
  }                                                   \
  catch (const ::b200tts::Error& e) {                 \
    g_err = e.what();                                 \
    return e.code;                                    \
  }                                                   \
  catch (const std::bad_alloc&) {                     \
    g_err = "host allocation failed";                 \
    return B200TTS_ENOMEM;                            \
  }                                                   \
  catch (const std::exception& e) {                   \
    g_err = e.what();                                 \
    return B200TTS_EINVAL;                            \
  }                                                   \
  return B200TTS_OK;

#define REQUIRE(cond, code, msg)                                 \
  do {                                                           \
    if (!(cond)) throw ::b200tts::Error((code), std::string(msg)); \
  } while (0)

namespace {

struct DeviceBuf {
  void* p = nullptr;
  size_t bytes = 0;
  void ensure(size_t n) {
    if (n <= bytes) return;
    if (p) B200_CUDA(cudaFree(p));
    p = nullptr;
    bytes = 0;
    cudaError_t e = cudaMalloc(&p, n);
    if (e != cudaSuccess) {
      p = nullptr;
      throw Error(B200TTS_ENOMEM, std::string("cudaMalloc(") + std::to_string(n) + "): " + cudaGetErrorString(e));
    }
    bytes = n;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

struct HostPinned {
  void* p = nullptr;
  size_t bytes = 0;
  void ensure(size_t n) {
    if (n <= bytes) return;
    if (p) cudaFreeHost(p);
    p = nullptr;
    bytes = 0;
    cudaError_t e = cudaMallocHost(&p, n);
    if (e != cudaSuccess) {
      p = nullptr;
      throw Error(B200TTS_ENOMEM, std::string("cudaMallocHost: ") + cudaGetErrorString(e));
    }
    bytes = n;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    bytes = 0;
  }
};

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    B200_CUDA(cudaGetDevice(&prev));
    if (prev != dev) B200_CUDA(cudaSetDevice(dev));
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

using TensorMap = std::map<std::string, const b200tts_tensor*>;

const b200tts_tensor* need(const TensorMap& m, const std::string& name, std::initializer_list<int64_t> shape) {
  auto it = m.find(name);
  if (it == m.end()) throw Error(B200TTS_EMISSING, "missing weight tensor '" + name + "'");
  const b200tts_tensor* t = it->second;
  size_t nd = shape.size();
  bool ok = (size_t)t->ndim == nd && t->data != nullptr;
  size_t i = 0;
  for (int64_t s : shape) {
    if (ok && t->shape[i] != s) ok = false;
    ++i;
  }
  if (!ok) {
    std::string got = "[";
    for (int k = 0; k < t->ndim && k < 4; ++k) got += (k ? "," : "") + std::to_string(t->shape[k]);
    got += "]";
    std::string want = "[";
    i = 0;
    for (int64_t s : shape) want += (i++ ? "," : "") + std::to_string(s);
    want += "]";
    throw Error(B200TTS_ESHAPE, "weight '" + name + "' has shape " + got + ", expected " + want);
  }
  return t;
}

// Host-side staging of one packed fp32 blob; every sub-array starts 16-byte aligned.
struct Packer {
  std::vector<float> h;
  size_t add(size_t n) {
    size_t off = (h.size() + 3) & ~size_t(3);
    h.resize(off + n, 0.f);
    return off;
  }
};

inline int round4(int x) { return (x + 3) & ~3; }

}  // namespace

struct b200tts_wavernn {
  int device = 0;
  b200tts_wavernn_cfg cfg{};
  int aux = 0, NC = 0, NT = 0, sm_count = 0;
  DeviceBuf weights;          // packed blob
  StepWeights sw{};
  ResnetParams rp{};
  const float* d_fir = nullptr;   // [hop][NT]
  GridModel gm{};                 // per-CTA weight blobs of the grid kernel
  DeviceBuf grid_blob, mels_T, aux_T, grid_sync, grid_prof, fold_mels, fold_aux;
  PushModel pm{};                 // small-batch push kernel (wavernn_push.cuh): per-CTA blobs + conditioning-projection weights
  PushCondW pcw{};
  DeviceBuf push_blob, push_condw, push_tab, push_vec, push_best, push_prof;
  DeviceBuf tc_wimg, tc_prm, tc_vec, tc_x1f, tc_win, tc_cnt, tc_cond;     // tensor-core pipeline (wavernn_tc.cuh)
  bool tc_ok = false;
  int last_kernel = 0;            // 1 utterance, 2 wide grid, 3 push, 4 multi-group push, 5 tensor-core pipeline
  int last_push_ncta = 0;
  int* d_grid_error = nullptr;    // set by the grid kernel when a barrier wait timed out (a peer CTA vanished)
  int last_grid_ncta = 0;
  int coop = 0;
  // scratch
  DeviceBuf mels_up, aux_frames, labels, mel_in, wave, grid_scratch;
  HostPinned h_stage;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool ev_valid = false;
  int64_t launches = 0;
  bool warned_fallback = false;
};

// ------------------------------------------------------------------------------------------------
extern "C" int b200tts_abi_version(void) { return B200TTS_ABI_VERSION; }
extern "C" const char* b200tts_last_error(void) { return g_err.c_str(); }
extern "C" int b200tts_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    g_err = std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e);
    cudaGetLastError();
    return B200TTS_ECUDA;
  }
  return n;
}

// Composite polyphase FIR of the Stretch2d/Conv2d chain (see wavernn_upsample.cuh).  Returns [hop][NT] doubles.
static std::vector<double> composite_fir(const b200tts_wavernn_cfg& c, const std::vector<std::vector<double>>& taps,
                                         int* NT_out) {
  const int hop = c.hop_length;
  // reach of the composite response beyond the frame's own box, in output samples
  int reach = 0, rate = hop;
  for (int j = 0; j < c.n_upsample; ++j) {
    rate /= c.upsample_factors[j];
    reach += c.upsample_factors[j] * rate;
  }
  int side = (reach + hop - 1) / hop;            // frames on each side that can contribute
  int NT = 2 * side + 1;
  REQUIRE(NT <= kMaxTaps, B200TTS_EINVAL, "upsample factors give a composite FIR wider than kMaxTaps frames");
  const int nf = 2 * side + 5, f0 = nf / 2;      // impulse in the middle, far from both ends
  std::vector<double> x(nf, 0.0);
  x[f0] = 1.0;
  for (int j = 0; j < c.n_upsample; ++j) {
    const int s = c.upsample_factors[j];
    std::vector<double> r(x.size() * s);
    for (size_t i = 0; i < r.size(); ++i) r[i] = x[i / s];
    std::vector<double> y(r.size(), 0.0);
    for (long i = 0; i < (long)r.size(); ++i) {
      double a = 0.0;
      for (int k = 0; k < 2 * s + 1; ++k) {
        long idx = i + k - s;
        if (idx >= 0 && idx < (long)r.size()) a += taps[j][k] * r[idx];
      }
      y[i] = a;
    }
    x.swap(y);
  }
  // out[n] = sum_f melpad[f] * Rsp[n - hop*f];  with n = hop*fr + ph and f = fr + (j - side):  Rsp[ph - hop*(j-side)]
  std::vector<double> fir((size_t)hop * NT);
  for (int ph = 0; ph < hop; ++ph)
    for (int j = 0; j < NT; ++j) {
      long idx = (long)hop * f0 + ph - (long)hop * (j - side);
      fir[(size_t)ph * NT + j] = (idx >= 0 && idx < (long)x.size()) ? x[idx] : 0.0;
    }
  *NT_out = NT;
  return fir;
}

extern "C" int b200tts_wavernn_create(b200tts_wavernn** out, int device, const b200tts_wavernn_cfg* cfg,
                                      const b200tts_tensor* weights, int n_weights) {
  API_BEGIN
  REQUIRE(out && cfg && weights && n_weights > 0, B200TTS_EINVAL, "null argument");
  *out = nullptr;
  const b200tts_wavernn_cfg& c = *cfg;
  REQUIRE(c.n_upsample >= 1 && c.n_upsample <= 4, B200TTS_EINVAL, "n_upsample must be 1..4");
  int prod = 1;
  for (int j = 0; j < c.n_upsample; ++j) {
    REQUIRE(c.upsample_factors[j] >= 1, B200TTS_EINVAL, "bad upsample factor");
    prod *= c.upsample_factors[j];
  }
  REQUIRE(prod == c.hop_length, B200TTS_EINVAL, "prod(upsample_factors) != hop_length (wavernn_train.py:67 asserts the same)");
  REQUIRE(c.res_out_dims % 4 == 0, B200TTS_EINVAL, "res_out_dims must be divisible by 4");
  REQUIRE(c.rnn_dims % 128 == 0 && c.fc_dims % 128 == 0, B200TTS_EINVAL, "rnn_dims / fc_dims must be multiples of 128");
  REQUIRE(c.bits >= 2 && c.bits <= 15, B200TTS_EINVAL, "bits must be 2..15 (labels are int16)");
  REQUIRE(c.compute_dims <= 1024 && c.res_out_dims <= 1024, B200TTS_EINVAL, "compute/res_out dims too large");
  const int R = c.rnn_dims, F = c.fc_dims, AUX = c.res_out_dims / 4, FEAT = c.feat_dims, NC = 1 << c.bits;
  const int C = c.compute_dims, O = c.res_out_dims, K = 2 * c.pad + 1;
  REQUIRE(AUX % 4 == 0, B200TTS_EINVAL, "aux dims (res_out_dims/4) must be a multiple of 4");
  int ndev = 0;
  B200_CUDA(cudaGetDeviceCount(&ndev));
  REQUIRE(device >= 0 && device < ndev, B200TTS_EINVAL, "no such CUDA device");
  DeviceGuard dg(device);

  TensorMap tm;
  for (int i = 0; i < n_weights; ++i)
    if (weights[i].name) tm[weights[i].name] = &weights[i];

  auto ctx = new b200tts_wavernn();
  struct Cleanup {
    b200tts_wavernn* c;
    ~Cleanup() {
      if (c) b200tts_wavernn_destroy(c);
    }
  } cleanup{ctx};
  ctx->device = device;
  ctx->cfg = c;
  ctx->aux = AUX;
  ctx->NC = NC;
  B200_CUDA(cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device));

  Packer pk;
  // ---- step weights, original layouts ----
  const int nin = 1 + FEAT + AUX, ldI = round4(nin);
  const float* Iw = need(tm, "I.weight", {R, nin})->data;
  size_t oI = pk.add((size_t)R * ldI);
  for (int r = 0; r < R; ++r) std::memcpy(&pk.h[oI + (size_t)r * ldI], Iw + (size_t)r * nin, sizeof(float) * nin);
  auto copy = [&](const std::string& name, std::initializer_list<int64_t> shape) {
    const b200tts_tensor* t = need(tm, name, shape);
    size_t n = 1;
    for (int64_t s : shape) n *= (size_t)s;
    size_t off = pk.add(n);
    std::memcpy(&pk.h[off], t->data, n * sizeof(float));
    return off;
  };
  size_t oIb = copy("I.bias", {R});
  size_t o_ih1 = copy("rnn1.weight_ih_l0", {3 * R, R}), o_hh1 = copy("rnn1.weight_hh_l0", {3 * R, R});
  size_t o_bih1 = copy("rnn1.bias_ih_l0", {3 * R}), o_bhh1 = copy("rnn1.bias_hh_l0", {3 * R});
  size_t o_ih2 = copy("rnn2.weight_ih_l0", {3 * R, R + AUX}), o_hh2 = copy("rnn2.weight_hh_l0", {3 * R, R});
  size_t o_bih2 = copy("rnn2.bias_ih_l0", {3 * R}), o_bhh2 = copy("rnn2.bias_hh_l0", {3 * R});
  size_t o_fc1 = copy("fc1.weight", {F, R + AUX}), o_fc1b = copy("fc1.bias", {F});
  size_t o_fc2 = copy("fc2.weight", {F, F + AUX}), o_fc2b = copy("fc2.bias", {F});
  size_t o_fc3 = copy("fc3.weight", {NC, F}), o_fc3b = copy("fc3.bias", {NC});

  // ---- MelResNet, transposed to [in][out]; BatchNorm (eval, eps 1e-5) folded to scale/shift in double ----
  const float* cin = need(tm, "upsample.resnet.conv_in.weight", {C, FEAT, K})->data;
  size_t o_cin = pk.add((size_t)FEAT * K * C);
  for (int cc = 0; cc < C; ++cc)
    for (int i = 0; i < FEAT; ++i)
      for (int j = 0; j < K; ++j) pk.h[o_cin + ((size_t)i * K + j) * C + cc] = cin[((size_t)cc * FEAT + i) * K + j];
  const int nbn = 1 + 2 * c.res_blocks;
  size_t o_bns = pk.add((size_t)nbn * C), o_bnh = pk.add((size_t)nbn * C);
  auto fold_bn = [&](const std::string& prefix, int slot) {
    const float* g = need(tm, prefix + ".weight", {C})->data;
    const float* b = need(tm, prefix + ".bias", {C})->data;
    const float* m = need(tm, prefix + ".running_mean", {C})->data;
    const float* v = need(tm, prefix + ".running_var", {C})->data;
    for (int cc = 0; cc < C; ++cc) {
      double sc = (double)g[cc] / std::sqrt((double)v[cc] + 1e-5);
      pk.h[o_bns + (size_t)slot * C + cc] = (float)sc;
      pk.h[o_bnh + (size_t)slot * C + cc] = (float)((double)b[cc] - (double)m[cc] * sc);
    }
  };
  fold_bn("upsample.resnet.batch_norm", 0);
  size_t o_res = pk.add((size_t)c.res_blocks * 2 * C * C);
  for (int blk = 0; blk < c.res_blocks; ++blk) {
    std::string p = "upsample.resnet.layers." + std::to_string(blk);
    for (int h = 0; h < 2; ++h) {
      const float* w = need(tm, p + (h ? ".conv2.weight" : ".conv1.weight"), {C, C, 1})->data;
      size_t base = o_res + ((size_t)blk * 2 + h) * C * C;
      for (int co = 0; co < C; ++co)
        for (int ci = 0; ci < C; ++ci) pk.h[base + (size_t)ci * C + co] = w[(size_t)co * C + ci];
    }
    fold_bn(p + ".batch_norm1", 1 + 2 * blk);
    fold_bn(p + ".batch_norm2", 2 + 2 * blk);
  }
  const float* cow = need(tm, "upsample.resnet.conv_out.weight", {O, C, 1})->data;
  size_t o_cout = pk.add((size_t)C * O);
  for (int o = 0; o < O; ++o)
    for (int ci = 0; ci < C; ++ci) pk.h[o_cout + (size_t)ci * O + o] = cow[(size_t)o * C + ci];
  size_t o_coutb = copy("upsample.resnet.conv_out.bias", {O});

  // ---- composite FIR ----
  std::vector<std::vector<double>> taps(c.n_upsample);
  for (int j = 0; j < c.n_upsample; ++j) {
    int s = c.upsample_factors[j];
    const float* w = need(tm, "upsample.up_layers." + std::to_string(2 * j + 1) + ".weight", {1, 1, 1, 2 * s + 1})->data;
    taps[j].assign(w, w + 2 * s + 1);
  }
  int NT = 0;
  std::vector<double> fir = composite_fir(c, taps, &NT);
  ctx->NT = NT;
  size_t o_fir = pk.add(fir.size());
  for (size_t i = 0; i < fir.size(); ++i) pk.h[o_fir + i] = (float)fir[i];

  ctx->weights.ensure(pk.h.size() * sizeof(float));
  B200_CUDA(cudaMemcpy(ctx->weights.p, pk.h.data(), pk.h.size() * sizeof(float), cudaMemcpyHostToDevice));
  const float* base = ctx->weights.as<float>();
  StepWeights& sw = ctx->sw;
  sw.I_w = base + oI; sw.I_b = base + oIb;
  sw.ih1_w = base + o_ih1; sw.hh1_w = base + o_hh1; sw.ih1_b = base + o_bih1; sw.hh1_b = base + o_bhh1;
  sw.ih2_w = base + o_ih2; sw.hh2_w = base + o_hh2; sw.ih2_b = base + o_bih2; sw.hh2_b = base + o_bhh2;
  sw.fc1_w = base + o_fc1; sw.fc1_b = base + o_fc1b; sw.fc2_w = base + o_fc2; sw.fc2_b = base + o_fc2b;
  sw.fc3_w = base + o_fc3; sw.fc3_b = base + o_fc3b;
  sw.R = R; sw.F = F; sw.aux = AUX; sw.feat = FEAT; sw.NC = NC; sw.ldI = ldI;
  ResnetParams& rp = ctx->rp;
  rp.conv_in_t = base + o_cin; rp.bn_scale = base + o_bns; rp.bn_shift = base + o_bnh; rp.res_w_t = base + o_res;
  rp.conv_out_t = base + o_cout; rp.conv_out_b = base + o_coutb;
  rp.feat = FEAT; rp.k = K; rp.C = C; rp.O = O; rp.blocks = c.res_blocks; rp.pad = c.pad;
  ctx->d_fir = base + o_fir;

  // ---- weight-stationary per-CTA blobs for the grid kernel (wavernn_grid.cuh) ----
  {
    GridModel& g = ctx->gm;
    g.R = R; g.F = F; g.AUX = AUX; g.FEAT = FEAT; g.NC = NC;
    g.ldC = FEAT + AUX; g.ldX = R + AUX; g.ldF = F + AUX;
    g.ncta = R / kUPC;
    g.ok = (R == F) && (R % kUPC == 0) && (NC == g.ncta * kCPC) && (FEAT % 4 == 0) && (g.ncta <= ctx->sm_count);
    // the narrow mapping stages [x1|aux], [f1|aux], [mel|aux] in a 640*G-float area and h in a 512*G-float area
    if (R + AUX > 640 || F + AUX > 640 || FEAT + AUX > 640 || R > 512) g.ok = 0;
    int off = 0;
    auto take = [&](int n) { int o = off; off += (n + 3) & ~3; return o; };
    g.oA_w = take(16 * g.ldC); g.oA_x = take(16); g.oA_b = take(16);
    g.ohh1 = take(3 * kUPC * R); g.oih2 = take(3 * kUPC * g.ldX); g.ohh2 = take(3 * kUPC * R);
    g.ofc1 = take(kUPC * g.ldX); g.ofc2 = take(kUPC * g.ldF); g.ofc3 = take(kCPC * F);
    g.obhh1 = take(3 * kUPC); g.obih2 = take(3 * kUPC); g.obhh2 = take(3 * kUPC);
    g.obfc1 = take(kUPC); g.obfc2 = take(kUPC); g.obfc3 = take(kCPC);
    g.blob = off;
    constexpr int kMaxScratch = std::max({MapTraits<0, 4, 1>::kScratchFloats, MapTraits<0, 8, 1>::kScratchFloats,
                                          MapTraits<1, 1, 1>::kScratchFloats, MapTraits<2, 1, 1>::kScratchFloats,
                                          MapTraits<4, 1, 1>::kScratchFloats, MapTraits<1, 1, 2>::kScratchFloats,
                                          MapTraits<2, 1, 2>::kScratchFloats, MapTraits<4, 1, 2>::kScratchFloats,
                                          MapTraits<2, 2, 2>::kScratchFloats});   // every variant launch_grid can dispatch
    size_t smem_need = ((size_t)g.blob + (size_t)kMaxScratch) * sizeof(float) + 2048;
    if (smem_need > 227 * 1024) g.ok = 0;
    B200_CUDA(cudaDeviceGetAttribute(&ctx->coop, cudaDevAttrCooperativeLaunch, device));
    if (!ctx->coop) g.ok = 0;
    if (g.ok) {
      std::vector<float> hb((size_t)g.ncta * g.blob, 0.f);
      std::vector<double> fold_acc(1 + g.ldC);
      const float* P = pk.h.data();
      for (int cta = 0; cta < g.ncta; ++cta) {
        float* b = &hb[(size_t)cta * g.blob];
        for (int j = 0; j < kUPC; ++j) {
          const int row = cta * kUPC + j;
          const float* src = P + oI + (size_t)row * ldI;          // [x | feat | aux] padded
          b[g.oA_x + j] = src[0];
          std::memcpy(b + g.oA_w + (size_t)j * g.ldC, src + 1, sizeof(float) * g.ldC);
          b[g.oA_b + j] = P[oIb + row];
          std::memcpy(b + g.ofc1 + (size_t)j * g.ldX, P + o_fc1 + (size_t)row * g.ldX, sizeof(float) * g.ldX);
          std::memcpy(b + g.ofc2 + (size_t)j * g.ldF, P + o_fc2 + (size_t)row * g.ldF, sizeof(float) * g.ldF);
          b[g.obfc1 + j] = P[o_fc1b + row];
          b[g.obfc2 + j] = P[o_fc2b + row];
          for (int gate = 0; gate < 3; ++gate) {
            const int srow = gate * R + row, drow = gate * kUPC + j;
            // folded input projection of GRU 1: row srow of W_ih1.W_I (x column | cond columns) and W_ih1.b_I + b_ih1, in double
            {
              const float* wr = P + o_ih1 + (size_t)srow * R;
              double bacc = (double)P[o_bih1 + srow];
              std::vector<double>& accv = fold_acc;
              std::fill(accv.begin(), accv.end(), 0.0);
              for (int k = 0; k < R; ++k) {
                const double wk = (double)wr[k];
                const float* irow = P + oI + (size_t)k * ldI;
                for (int col = 0; col < 1 + g.ldC; ++col) accv[col] += wk * (double)irow[col];
                bacc += wk * (double)P[oIb + k];
              }
              b[g.oA_x + 4 + drow] = (float)accv[0];
              for (int col = 0; col < g.ldC; ++col) b[g.oA_w + (size_t)(4 + drow) * g.ldC + col] = (float)accv[1 + col];
              b[g.oA_b + 4 + drow] = (float)bacc;
            }
            std::memcpy(b + g.ohh1 + (size_t)drow * R, P + o_hh1 + (size_t)srow * R, sizeof(float) * R);
            std::memcpy(b + g.oih2 + (size_t)drow * g.ldX, P + o_ih2 + (size_t)srow * g.ldX, sizeof(float) * g.ldX);
            std::memcpy(b + g.ohh2 + (size_t)drow * R, P + o_hh2 + (size_t)srow * R, sizeof(float) * R);
            b[g.obhh1 + drow] = P[o_bhh1 + srow];
            b[g.obih2 + drow] = P[o_bih2 + srow]; b[g.obhh2 + drow] = P[o_bhh2 + srow];
          }
        }
        for (int r = 0; r < kCPC; ++r) {
          const int row = cta * kCPC + r;
          std::memcpy(b + g.ofc3 + (size_t)r * F, P + o_fc3 + (size_t)row * F, sizeof(float) * F);
          b[g.obfc3 + r] = P[o_fc3b + row];
        }
      }
      ctx->grid_blob.ensure(hb.size() * sizeof(float));
      B200_CUDA(cudaMemcpy(ctx->grid_blob.p, hb.data(), hb.size() * sizeof(float), cudaMemcpyHostToDevice));

      // ---- push kernel (wavernn_push.cuh): recurrent / feed-forward rows only; the conditioned columns become tables ----
      PushModel& pm = ctx->pm;
      pm.ncta = g.ncta; pm.R = R; pm.F = F; pm.NC = NC;
      int poff = 0;
      auto ptake = [&](int n) { int o = poff; poff += (n + 3) & ~3; return o; };
      // W_ih2 (12 rows) | fc1 (4 rows) | W_hh2 (12 rows) are contiguous: x1 is multiplied by the first 16 rows in one pass, h2 by the
      // last 16 (fc1, then W_hh2) from one set of registers
      pm.ohh1 = ptake(12 * R); pm.oih2 = ptake(12 * R); pm.ofc1 = ptake(4 * R); pm.ohh2 = ptake(12 * R);
      pm.ofc2 = ptake(4 * F); pm.ofc3 = ptake(8 * F);
      pm.oAx = ptake(16); pm.obhh1 = ptake(12); pm.obhh2 = ptake(12); pm.obfc3 = ptake(8);
      pm.blob = poff;
      const size_t push_smem = ((size_t)pm.blob + (size_t)PushTraits<32>::scratch_floats(c.hop_length, NT)) * sizeof(float) + 1024;
      pm.ok = (R == 512 && F == 512 && g.ncta == 128 && NC <= 1024 && push_smem <= 227 * 1024) ? 1 : 0;
      if (pm.ok) {
        std::vector<float> pb((size_t)g.ncta * pm.blob, 0.f);
        std::vector<float> cw((size_t)g.ncta * (16 * FEAT + 36 * AUX + 36), 0.f);
        float* wm = cw.data();
        float* wa = wm + (size_t)g.ncta * 16 * FEAT;
        float* cb = wa + (size_t)g.ncta * 36 * AUX;
        for (int cta = 0; cta < g.ncta; ++cta) {
          const float* b = &hb[(size_t)cta * g.blob];
          float* d = &pb[(size_t)cta * pm.blob];
          for (int r = 0; r < 12; ++r) {
            std::memcpy(d + pm.ohh1 + (size_t)r * R, b + g.ohh1 + (size_t)r * R, sizeof(float) * R);
            std::memcpy(d + pm.oih2 + (size_t)r * R, b + g.oih2 + (size_t)r * g.ldX, sizeof(float) * R);
            std::memcpy(d + pm.ohh2 + (size_t)r * R, b + g.ohh2 + (size_t)r * R, sizeof(float) * R);
            d[pm.obhh1 + r] = b[g.obhh1 + r];
            d[pm.obhh2 + r] = b[g.obhh2 + r];
            std::memcpy(wa + ((size_t)cta * 36 + 16 + r) * AUX, b + g.oih2 + (size_t)r * g.ldX + R, sizeof(float) * AUX);
            cb[(size_t)cta * 36 + 16 + r] = b[g.obih2 + r];
          }
          for (int j = 0; j < 4; ++j) {
            std::memcpy(d + pm.ofc1 + (size_t)j * R, b + g.ofc1 + (size_t)j * g.ldX, sizeof(float) * R);
            std::memcpy(d + pm.ofc2 + (size_t)j * F, b + g.ofc2 + (size_t)j * g.ldF, sizeof(float) * F);
            std::memcpy(wa + ((size_t)cta * 36 + 28 + j) * AUX, b + g.ofc1 + (size_t)j * g.ldX + R, sizeof(float) * AUX);
            std::memcpy(wa + ((size_t)cta * 36 + 32 + j) * AUX, b + g.ofc2 + (size_t)j * g.ldF + F, sizeof(float) * AUX);
            cb[(size_t)cta * 36 + 28 + j] = b[g.obfc1 + j];
            cb[(size_t)cta * 36 + 32 + j] = b[g.obfc2 + j];
          }
          for (int r = 0; r < 8; ++r) {
            std::memcpy(d + pm.ofc3 + (size_t)r * F, b + g.ofc3 + (size_t)r * F, sizeof(float) * F);
            d[pm.obfc3 + r] = b[g.obfc3 + r];
          }
          for (int r = 0; r < 16; ++r) {          // I rows 0-3, folded GRU-1 rows 4-15: [mel | a1] columns, x coefficient, bias
            d[pm.oAx + r] = b[g.oA_x + r];
            std::memcpy(wm + ((size_t)cta * 16 + r) * FEAT, b + g.oA_w + (size_t)r * g.ldC, sizeof(float) * FEAT);
            std::memcpy(wa + ((size_t)cta * 36 + r) * AUX, b + g.oA_w + (size_t)r * g.ldC + FEAT, sizeof(float) * AUX);
            cb[(size_t)cta * 36 + r] = b[g.oA_b + r];
          }
        }
        ctx->push_blob.ensure(pb.size() * sizeof(float));
        B200_CUDA(cudaMemcpy(ctx->push_blob.p, pb.data(), pb.size() * sizeof(float), cudaMemcpyHostToDevice));
        ctx->push_condw.ensure(cw.size() * sizeof(float));
        B200_CUDA(cudaMemcpy(ctx->push_condw.p, cw.data(), cw.size() * sizeof(float), cudaMemcpyHostToDevice));
        const float* cwd = ctx->push_condw.as<float>();
        ctx->pcw.wm = cwd;
        ctx->pcw.wa = cwd + (size_t)g.ncta * 16 * FEAT;
        ctx->pcw.bias = ctx->pcw.wa + (size_t)g.ncta * 36 * AUX;
        ctx->pcw.ncta = g.ncta; ctx->pcw.feat = FEAT; ctx->pcw.aux = AUX;

        // ---- tensor-core pipeline (wavernn_tc.cuh): per-CTA B-operand images, every weight split into two fp16 planes
        //      (hi, lo' = (w - hi) * 2048) in the UMMA K-major no-swizzle layout [plane][k-step 32][k half 2][N/8][8 cols][8 halves]
        if (NC == 1024 && ctx->sm_count >= kTcCtas) {
          std::vector<uint16_t> img((size_t)kTcCtas * kTcWimgBytes / 2, 0);
          std::vector<float> prm((size_t)kTcCtas * kTcPrm, 0.f);
          auto put = [&](uint16_t* base, int N, int col, const float* wrow) {     // one weight row (K = 512) -> column `col` of an image
            for (int k = 0; k < 512; ++k) {
              const float w = wrow[k];
              const __half hi = __float2half_rn(w);
              const __half lo = __float2half_rn((w - __half2float(hi)) * 2048.0f);
              const size_t off = ((size_t)(k >> 4) * 2 + ((k >> 3) & 1)) * ((size_t)N * 8) + (size_t)(col >> 3) * 64 + (size_t)(col & 7) * 8 + (k & 7);
              base[off] = __half_as_ushort(hi);
              base[(size_t)32 * N * 16 + off] = __half_as_ushort(lo);
            }
          };
          auto unit_blob = [&](int unit) { return &pb[(size_t)(unit >> 2) * pm.blob]; };
          for (int cta = 0; cta < kTcCtas; ++cta) {
            uint16_t* wi = &img[(size_t)cta * kTcWimgBytes / 2];
            float* pr = &prm[(size_t)cta * kTcPrm];
            if (cta < 32) {                                   // GRU-1: 16 units, columns gate*16 + i
              for (int i = 0; i < 16; ++i) {
                const int unit = 16 * cta + i, j = unit & 3;
                const float* b = unit_blob(unit);
                for (int gate = 0; gate < 3; ++gate) {
                  put(wi, 48, gate * 16 + i, b + pm.ohh1 + (size_t)(gate * 4 + j) * R);
                  pr[64 + gate * 16 + i] = b[pm.obhh1 + gate * 4 + j];
                }
                for (int kind = 0; kind < 4; ++kind) pr[kind * 16 + i] = b[pm.oAx + kind * 4 + j];
              }
            } else if (cta < 96) {                            // GRU-2: 8 units, W_ih2 image then W_hh2 image, columns gate*8 + i (24-31 zero)
              const int ci = cta - 32;
              for (int i = 0; i < 8; ++i) {
                const int unit = 8 * ci + i, j = unit & 3;
                const float* b = unit_blob(unit);
                for (int gate = 0; gate < 3; ++gate) {
                  put(wi, 32, gate * 8 + i, b + pm.oih2 + (size_t)(gate * 4 + j) * R);
                  put(wi + 32768, 32, gate * 8 + i, b + pm.ohh2 + (size_t)(gate * 4 + j) * R);
                  pr[gate * 8 + i] = b[pm.obhh2 + gate * 4 + j];
                }
              }
            } else if (cta < 128) {                           // fc1 / fc2: 32 units
              const bool first = cta < 112;
              const int ci = first ? cta - 96 : cta - 112;
              for (int i = 0; i < 32; ++i) {
                const int unit = 32 * ci + i, j = unit & 3;
                const float* b = unit_blob(unit);
                put(wi, 32, i, b + (first ? pm.ofc1 : pm.ofc2) + (size_t)j * R);
              }
            } else {                                          // fc3: 64 classes
              const int ci = cta - 128;
              for (int i = 0; i < 64; ++i) {
                const int cls = 64 * ci + i;
                const float* b = &pb[(size_t)(cls >> 3) * pm.blob];
                put(wi, 64, i, b + pm.ofc3 + (size_t)(cls & 7) * F);
                pr[i] = b[pm.obfc3 + (cls & 7)];
              }
            }
          }
          ctx->tc_wimg.ensure(img.size() * sizeof(uint16_t));
          B200_CUDA(cudaMemcpy(ctx->tc_wimg.p, img.data(), img.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
          ctx->tc_prm.ensure(prm.size() * sizeof(float));
          B200_CUDA(cudaMemcpy(ctx->tc_prm.p, prm.data(), prm.size() * sizeof(float), cudaMemcpyHostToDevice));
          ctx->tc_ok = true;
        }
      }
    }
  }
  B200_CUDA(cudaEventCreate(&ctx->ev0));
  B200_CUDA(cudaEventCreate(&ctx->ev1));
  cleanup.c = nullptr;
  *out = ctx;
  API_END
}

extern "C" void b200tts_wavernn_destroy(b200tts_wavernn* ctx) {
  if (!ctx) return;
  int prev = -1;
  cudaGetDevice(&prev);
  cudaSetDevice(ctx->device);
  ctx->weights.release();
  ctx->mels_up.release();
  ctx->aux_frames.release();
  ctx->labels.release();
  ctx->mel_in.release();
  ctx->wave.release();
  ctx->grid_scratch.release();
  ctx->grid_blob.release();
  ctx->mels_T.release();
  ctx->aux_T.release();
  ctx->grid_sync.release();
  ctx->grid_prof.release();
  ctx->fold_mels.release();
  ctx->fold_aux.release();
  ctx->push_blob.release();
  ctx->push_condw.release();
  ctx->push_tab.release();
  ctx->push_vec.release();
  ctx->push_best.release();
  ctx->push_prof.release();
  ctx->tc_wimg.release(); ctx->tc_prm.release(); ctx->tc_vec.release(); ctx->tc_x1f.release(); ctx->tc_win.release(); ctx->tc_cnt.release(); ctx->tc_cond.release();
  ctx->h_stage.release();
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (prev >= 0) cudaSetDevice(prev);
  delete ctx;
}

extern "C" int64_t b200tts_wavernn_launch_count(const b200tts_wavernn* ctx) { return ctx ? ctx->launches : -1; }

extern "C" int b200tts_wavernn_last_kernel(const b200tts_wavernn* ctx) { return ctx ? ctx->last_kernel : 0; }

extern "C" double b200tts_wavernn_last_kernel_ms(b200tts_wavernn* ctx) {
  if (!ctx || !ctx->ev_valid) {
    g_err = "no generate call has been timed on this context";
    return -1.0;
  }
  float ms = 0.f;
  cudaError_t e = cudaEventSynchronize(ctx->ev1);
  if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  if (e != cudaSuccess) {
    g_err = std::string("cudaEventElapsedTime: ") + cudaGetErrorString(e);
    return -1.0;
  }
  if (ctx->d_grid_error) {
    int flag = 0;
    if (cudaMemcpy(&flag, ctx->d_grid_error, sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess && flag) {
      g_err = "grid kernel: a grid-barrier wait timed out (co-resident CTA missing); results are invalid";
      return -1.0;
    }
  }
  return (double)ms;
}

// ---- conditioning ---------------------------------------------------------------------------------
static void run_upsample(b200tts_wavernn* ctx, const float* d_mel, int B, int T, float* d_mels_up, float* d_aux_frames,
                         float* d_aux_full, cudaStream_t st) {
  const b200tts_wavernn_cfg& c = ctx->cfg;
  const int hop = c.hop_length, O = c.res_out_dims;
  float* auxf = d_aux_frames;
  if (!auxf && d_aux_full) {
    ctx->aux_frames.ensure((size_t)B * T * O * sizeof(float));
    auxf = ctx->aux_frames.as<float>();
  }
  if (auxf) {
    constexpr int FT = 8;
    int threads = ((std::max(c.compute_dims, 32) + 31) / 32) * 32;
    size_t smem = ((size_t)c.feat_dims * (2 * c.pad + 1) * FT + 2 * (size_t)c.compute_dims * FT) * sizeof(float);
    if (smem > 48 * 1024)
      B200_CUDA(cudaFuncSetAttribute(melresnet_kernel<FT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((T + FT - 1) / FT, B);
    melresnet_kernel<FT><<<grid, threads, smem, st>>>(ctx->rp, d_mel, T, auxf);
    B200_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  if (d_mels_up) {
    size_t n = (size_t)T * hop * c.feat_dims;
    dim3 grid((unsigned)std::min<size_t>((n + 255) / 256, 4096), B);
    mel_fir_kernel<<<grid, 256, 0, st>>>(d_mel, ctx->d_fir, T, c.feat_dims, hop, c.pad, ctx->NT, d_mels_up);
    B200_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  if (d_aux_full) {
    size_t n = (size_t)T * hop * O;
    dim3 grid((unsigned)std::min<size_t>((n + 255) / 256, 4096), B);
    aux_repeat_kernel<<<grid, 256, 0, st>>>(auxf, T, hop, O, d_aux_full);
    B200_CUDA(cudaGetLastError());
    ctx->launches++;
  }
}

extern "C" int b200tts_wavernn_upsample(b200tts_wavernn* ctx, const float* d_mel, int B, int T, float* d_mels_up,
                                        float* d_aux_frames, float* d_aux_full, void* stream) {
  API_BEGIN
  REQUIRE(ctx && d_mel, B200TTS_EINVAL, "null argument");
  REQUIRE(B >= 1 && T >= 1, B200TTS_EINVAL, "B and T must be positive");
  REQUIRE(B <= 65535, B200TTS_EINVAL, "B must be <= 65535");
  DeviceGuard dg(ctx->device);
  run_upsample(ctx, d_mel, B, T, d_mels_up, d_aux_frames, d_aux_full, (cudaStream_t)stream);
  API_END
}

// ---- generation -----------------------------------------------------------------------------------
template <int G>
static void launch_utt(b200tts_wavernn* ctx, const GenArgs& a, cudaStream_t st) {
  const StepWeights& w = ctx->sw;
  size_t fl = (size_t)G * (w.ldI + w.R + 4 * w.R + 2 * (w.R + w.aux) + (w.F + w.aux) + w.F + w.NC);
  size_t smem = fl * sizeof(float);
  REQUIRE(smem <= 227 * 1024, B200TTS_EINVAL, "model too large for the utterance kernel's shared memory");
  B200_CUDA(cudaFuncSetAttribute(wavernn_utt_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int grid = (a.B + G - 1) / G;
  wavernn_utt_kernel<G><<<grid, kUttThreads, smem, st>>>(w, a);
  B200_CUDA(cudaGetLastError());
  ctx->launches++;
}

template <int U, int UW, int GROUPS>
static void launch_grid_t(b200tts_wavernn* ctx, GridArgs& a, cudaStream_t st) {
  const GridModel& g = ctx->gm;
  using MT = MapTraits<U, UW, GROUPS>;
  constexpr int kThreads = MT::NW * 32;
  size_t smem = ((size_t)g.blob + (size_t)MT::kScratchFloats) * sizeof(float);
  auto kern = wavernn_grid_kernel<U, UW, GROUPS>;
  B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, smem));
  REQUIRE(per_sm * ctx->sm_count >= g.ncta, B200TTS_EINVAL, "grid kernel cannot be made co-resident on this device");
  GridModel gm = g;
  void* args[] = {(void*)&gm, (void*)&a};
  B200_CUDA(cudaLaunchCooperativeKernel((const void*)kern, dim3(g.ncta), dim3(kThreads), args, smem, st));
  ctx->launches++;
}

// Mapping for B utterances: returns the padded batch; variant = index into the dispatch table below.
enum { GV_N4, GV_N8, GV_W1, GV_W1x2, GV_W2x2, GV_W4x2, GV_W2, GV_W4, GV_W2_2x2 };
static int grid_variant(int B, int* variant) {
  if (B <= 4) { *variant = GV_N4; return 4; }
  static const bool narrow8 = getenv("B200TTS_GRID_NARROW8") != nullptr;       // A/B switch: measured 30.7 us/step against 29.4 us
  if (B <= 8 && narrow8) { *variant = GV_N8; return 8; }                       // for the 32-wide mapping, so 5..8 utterances go wide
  if (B <= 32) { *variant = GV_W1; return 32; }
  static const bool mid_dual = getenv("B200TTS_GRID_MID_DUAL") != nullptr;       // A/B switch: old mid-batch mapping
  if (B <= 64) { *variant = mid_dual ? GV_W1x2 : GV_W2; return 64; }
  if (B <= 128) { *variant = mid_dual ? GV_W2x2 : GV_W4; return 128; }
  static const bool big22 = getenv("B200TTS_GRID_BIG_2X2") != nullptr;         // A/B switch: 2 utt x 12 rows per thread, no row slices
  *variant = big22 ? GV_W2_2x2 : GV_W4x2;
  return (B + 255) / 256 * 256;
}

struct FoldGeom {           // fold_with_overlap geometry (fatchord_version.py:319-330)
  int nfold, L, stride, total_len;
};
static FoldGeom fold_geometry(int S, int target, int overlap) {
  FoldGeom g{};
  g.stride = target + overlap;
  g.L = target + 2 * overlap;
  int num_folds = (S - overlap) / g.stride;
  int extended = num_folds * g.stride + overlap;
  if (S - extended != 0) num_folds += 1;
  g.nfold = num_folds;
  g.total_len = num_folds * g.stride + overlap;
  return g;
}

// `fold` != null: `ua` already describes the folded problem (B = nfold, S = T = L, hop = 1) and the conditioning of the
// single source utterance is in ctx->mels_up [S0][feat] / ctx->aux_frames [T0][O].
static void launch_grid(b200tts_wavernn* ctx, const float* d_mel, GenArgs& ua, cudaStream_t st, const FoldGeom* fold = nullptr,
                        int S0 = 0) {
  const b200tts_wavernn_cfg& c = ctx->cfg;
  const GridModel& g = ctx->gm;
  REQUIRE(g.ok, B200TTS_EINVAL, "this model/device cannot run the grid kernel (use B200TTS_KERNEL_UTTERANCE)");
  int variant = 0;
  const int B = ua.B, T = ua.T, S = ua.S, O = c.res_out_dims;
  const int Bp = grid_variant(B, &variant);
  // conditioning in K-major layout
  ctx->mels_T.ensure((size_t)S * c.feat_dims * Bp * sizeof(float));
  ctx->aux_T.ensure((size_t)T * O * Bp * sizeof(float));
  if (fold) {
    size_t n = (size_t)S * (c.feat_dims + O) * Bp;
    unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx->sm_count * 32);
    fold_cond_T_kernel<<<grid, 256, 0, st>>>(ctx->mels_up.as<float>(), ctx->aux_frames.as<float>(), S0, c.hop_length, c.feat_dims, O,
                                             fold->L, fold->stride, fold->nfold, Bp, ctx->mels_T.as<float>(), ctx->aux_T.as<float>());
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
  } else {
    size_t n = (size_t)S * c.feat_dims * Bp;
    unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx->sm_count * 32);
    mel_fir_T_kernel<<<grid, 256, 0, st>>>(d_mel, ctx->d_fir, B, Bp, T, c.feat_dims, c.hop_length, c.pad, ctx->NT,
                                           ctx->mels_T.as<float>());
    B200_CUDA(cudaGetLastError());
    n = (size_t)T * O * Bp;
    grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx->sm_count * 32);
    aux_T_kernel<<<grid, 256, 0, st>>>(ua.aux_frames, B, Bp, T, O, ctx->aux_T.as<float>());
    B200_CUDA(cudaGetLastError());
    ctx->launches += 2;
  }
  // activations + sync words, zero-initialised (h1 = h2 = 0, fatchord_version.py:194-195)
  const size_t RB = (size_t)g.R * Bp;
  const size_t act_floats = 8 * RB;
  const size_t sync_bytes = 2 * (size_t)Bp * sizeof(unsigned long long) + 512;
  ctx->grid_scratch.ensure(act_floats * sizeof(float));
  ctx->grid_sync.ensure(sync_bytes);
  B200_CUDA(cudaMemsetAsync(ctx->grid_scratch.p, 0, act_floats * sizeof(float), st));
  B200_CUDA(cudaMemsetAsync(ctx->grid_sync.p, 0, sync_bytes, st));
  float* base = ctx->grid_scratch.as<float>();
  GridArgs a{};
  a.wblob = ctx->grid_blob.as<float>();
  a.h1 = base; a.h2 = base + 2 * RB; a.x1 = base + 4 * RB; a.x2 = base + 5 * RB;
  a.f1 = base + 6 * RB; a.f2 = base + 7 * RB;
  a.best = ctx->grid_sync.as<unsigned long long>();
  a.barrier = reinterpret_cast<unsigned int*>(ctx->grid_sync.as<char>() + 2 * (size_t)Bp * sizeof(unsigned long long));
  a.error = reinterpret_cast<int*>(a.barrier + 96);
  ctx->d_grid_error = a.error;
  a.mels_T = ctx->mels_T.as<float>();
  a.aux_T = ctx->aux_T.as<float>();
  a.B = B; a.Bp = Bp; a.S = S; a.T = T; a.hop = ua.hop; a.steps = ua.steps;
  a.rng_mode = ua.rng_mode; a.seed = ua.seed; a.utt_offset = ua.utt_offset; a.utt_ids = ua.utt_ids; a.q = ua.q;
  a.teacher = ua.teacher; a.logits_out = ua.logits_out; a.labels = ua.labels;
  a.prof = nullptr;
  if (getenv("B200TTS_GRID_PROF")) {
    ctx->grid_prof.ensure((size_t)g.ncta * 12 * sizeof(long long));
    B200_CUDA(cudaMemsetAsync(ctx->grid_prof.p, 0, (size_t)g.ncta * 12 * sizeof(long long), st));
    a.prof = ctx->grid_prof.as<long long>();
    ctx->last_grid_ncta = g.ncta;
  }
  B200_CUDA(cudaEventRecord(ctx->ev0, st));
  switch (variant) {
    case GV_N4: launch_grid_t<0, 4, 1>(ctx, a, st); break;
    case GV_N8: launch_grid_t<0, 8, 1>(ctx, a, st); break;
    case GV_W1: launch_grid_t<1, 1, 1>(ctx, a, st); break;
    case GV_W1x2: launch_grid_t<1, 1, 2>(ctx, a, st); break;
    case GV_W2x2: launch_grid_t<2, 1, 2>(ctx, a, st); break;
    case GV_W4x2: launch_grid_t<4, 1, 2>(ctx, a, st); break;
    case GV_W2: launch_grid_t<2, 1, 1>(ctx, a, st); break;
    case GV_W4: launch_grid_t<4, 1, 1>(ctx, a, st); break;
    case GV_W2_2x2: launch_grid_t<2, 2, 2>(ctx, a, st); break;
    default: REQUIRE(false, B200TTS_EINVAL, "internal: unknown grid variant");
  }
  B200_CUDA(cudaEventRecord(ctx->ev1, st));
}

// ---- small-batch push kernel (wavernn_push.cuh) --------------------------------------------------------------------------
template <int G, bool STREAM>
static void launch_push_t(b200tts_wavernn* ctx, PushArgs& a, cudaStream_t st) {
  const PushModel& pm = ctx->pm;
  using PT = PushTraits<G>;
  size_t smem = ((size_t)pm.blob + (size_t)PT::scratch_floats(a.hop, a.NT)) * sizeof(float);
  auto kern = wavernn_push_kernel<G, STREAM>;
  B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kPushThreads, smem));
  REQUIRE(per_sm * ctx->sm_count >= pm.ncta, B200TTS_EINVAL, "push kernel cannot be made co-resident on this device");
  PushModel m = pm;
  void* args[] = {(void*)&m, (void*)&a};
  B200_CUDA(cudaLaunchCooperativeKernel((const void*)kern, dim3(pm.ncta), dim3(kPushThreads), args, smem, st));
  ctx->launches++;
}

// rows per group of the push kernels.  Measured (profiles/r02_push_v3_phase_cycles.txt): 8 rows 9.2 us per step, 4 rows 14.5 us
// (64 hot L2 lines polled by 65 536 threads) -- so up to 8 rows run the 8-row variant; env B200TTS_PUSH_MIN_G is an A/B switch.
static inline int push_rows(int B) {
  static const int min_g = getenv("B200TTS_PUSH_MIN_G") ? atoi(getenv("B200TTS_PUSH_MIN_G")) : 8;
  const int g = B <= 4 ? 4 : (B <= 8 ? 8 : (B <= 16 ? 16 : 32));
  return g < min_g ? (min_g <= 8 ? 8 : (min_g <= 16 ? 16 : 32)) : g;
}

// Can this call take the push kernel?  (env B200TTS_PUSH=0 keeps the round-1 mappings for A/B timing.)
static bool push_eligible(const b200tts_wavernn* ctx, int rows) {
  static const bool off = getenv("B200TTS_PUSH") != nullptr && getenv("B200TTS_PUSH")[0] == '0';
  // Default 32: the multi-group form (wavernn_pushmg.cuh, 33 ... 256 rows) is parity-green but MEASURED SLOWER than the round-1 wide
  // mapping (144 vs 68 us per lock-step at 256 rows, profiles/r02_pushmg_time.txt), so it only runs when asked for.
  static const int max_rows = getenv("B200TTS_PUSH_MAX_ROWS") ? atoi(getenv("B200TTS_PUSH_MAX_ROWS")) : kMgG;
  return ctx->pm.ok && ctx->gm.ok && rows <= max_rows && rows <= kMgG * kMgMaxGroups && !off;
}

// `fold` != null: rows are the folds of ONE source utterance of T0 frames (conditioning tables of utterance 0, row u
// starts at sample u * stride); otherwise row u is utterance u.
struct PackInfo {            // gen_opts.d_pack_*: kernel rows run queues of utterances
  const int* utt;
  const int* start;
  int rows, segs, steps, n_utt;
};
// b200tts_wavernn_generate_stream: the kernel also hands every final wave sample to pinned host memory (device aliases here)
struct StreamWave {
  double* h_wave;
  long long* h_progress;
  int chunk_steps;
  const int* utt_frames;
  int fade_len, mu_law;
};
static void launch_push(b200tts_wavernn* ctx, const float* d_mel, GenArgs& ua, cudaStream_t st, const FoldGeom* fold, int T0,
                        const PackInfo* pack = nullptr, const StreamWave* sw = nullptr) {
  const b200tts_wavernn_cfg& c = ctx->cfg;
  const PushModel& pm = ctx->pm;
  const int rows = pack ? pack->rows : ua.B;
  const int ng = rows > kMgG ? (rows + kMgG - 1) / kMgG : 1;          // > 32 rows: multi-group kernel, groups of 32
  const int G = ng > 1 ? kMgG : push_rows(rows);
  const int T = fold ? T0 : ua.T, hop = c.hop_length;
  const int tab_rows = fold ? 1 : (pack ? pack->n_utt : ng * G), src_rows = fold ? 1 : (pack ? pack->n_utt : rows);
  // conditioning tables [tab_rows][T+1][ncta][52]
  ctx->push_tab.ensure((size_t)tab_rows * (T + 1) * pm.ncta * kPushCondRows * sizeof(float));
  {
    constexpr int FT = 8;
    dim3 grid((T + 1 + FT - 1) / FT, tab_rows);
    size_t smem = (size_t)(c.feat_dims + c.res_out_dims) * FT * sizeof(float);
    push_cond_table_kernel<FT><<<grid, 256, smem, st>>>(ctx->pcw, d_mel, ua.aux_frames, src_rows, T, ctx->push_tab.as<float>());
    B200_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  const size_t nvec = (size_t)ng * kPushVecs * 2 * pm.ncta * G * 4, nbest = (size_t)ng * pm.ncta * G;
  ctx->push_vec.ensure(nvec * sizeof(float));
  ctx->push_best.ensure(nbest * sizeof(unsigned long long) + 64);
  int* d_err = reinterpret_cast<int*>(ctx->push_best.as<unsigned long long>() + nbest);
  push_init_kernel<<<ctx->sm_count, 256, 0, st>>>(ctx->push_vec.as<uint32_t>(), nvec, ctx->push_best.as<unsigned long long>(), nbest, d_err);
  B200_CUDA(cudaGetLastError());
  ctx->launches++;
  ctx->d_grid_error = d_err;
  PushArgs a{};
  a.wblob = ctx->push_blob.as<float>();
  a.vec = ctx->push_vec.as<float>();
  a.best = ctx->push_best.as<unsigned long long>();
  a.error = d_err;
  a.tab = ctx->push_tab.as<float>();
  a.fir = ctx->d_fir;
  a.NT = ctx->NT;
  a.B = pack ? pack->n_utt : rows; a.S = ua.S; a.T = T; a.hop = hop; a.steps = pack ? pack->steps : ua.steps;
  a.ng = ng;
  if (pack) { a.pack_utt = pack->utt; a.pack_start = pack->start; a.pack_segs = pack->segs; a.pack_rows = pack->rows; }
  a.row_stride = fold ? fold->stride : 0;
  a.S_src = T * hop;
  a.rng_mode = ua.rng_mode; a.seed = ua.seed; a.utt_offset = ua.utt_offset; a.utt_ids = ua.utt_ids; a.q = ua.q;
  a.teacher = ua.teacher; a.logits_out = ua.logits_out; a.labels = ua.labels;
  if (sw) {
    REQUIRE(ng == 1 && !fold && !pack, B200TTS_EINVAL, "internal: streaming needs a plain batch of <= 32 rows");
    a.h_wave = sw->h_wave; a.h_progress = sw->h_progress; a.chunk_steps = sw->chunk_steps;
    a.d_utt_frames = sw->utt_frames; a.fade_len = sw->fade_len; a.mu_law = sw->mu_law;
  }
  a.prof = nullptr;
  if (getenv("B200TTS_GRID_PROF")) {
    ctx->push_prof.ensure((size_t)pm.ncta * 12 * sizeof(long long));
    B200_CUDA(cudaMemsetAsync(ctx->push_prof.p, 0, (size_t)pm.ncta * 12 * sizeof(long long), st));
    a.prof = ctx->push_prof.as<long long>();
    ctx->last_push_ncta = pm.ncta;
    ctx->last_grid_ncta = 0;
  }
  B200_CUDA(cudaEventRecord(ctx->ev0, st));
  if (ng > 1) {
    const MgLayout L(ng);
    size_t smem = ((size_t)pm.blob + (size_t)L.total) * sizeof(float);
    REQUIRE(smem + 2048 <= 227 * 1024, B200TTS_EINVAL, "multi-group push kernel: shared memory budget exceeded");
    B200_CUDA(cudaFuncSetAttribute(wavernn_pushmg_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wavernn_pushmg_kernel, kPushThreads, smem));
    REQUIRE(per_sm * ctx->sm_count >= pm.ncta, B200TTS_EINVAL, "multi-group push kernel cannot be made co-resident on this device");
    PushModel m = pm;
    void* args[] = {(void*)&m, (void*)&a};
    B200_CUDA(cudaLaunchCooperativeKernel((const void*)wavernn_pushmg_kernel, dim3(pm.ncta), dim3(kPushThreads), args, smem, st));
    ctx->launches++;
  } else if (sw) switch (G) {
    case 4: launch_push_t<4, true>(ctx, a, st); break;
    case 8: launch_push_t<8, true>(ctx, a, st); break;
    case 16: launch_push_t<16, true>(ctx, a, st); break;
    default: launch_push_t<32, true>(ctx, a, st); break;
  } else switch (G) {
    case 4: launch_push_t<4, false>(ctx, a, st); break;
    case 8: launch_push_t<8, false>(ctx, a, st); break;
    case 16: launch_push_t<16, false>(ctx, a, st); break;
    default: launch_push_t<32, false>(ctx, a, st); break;
  }
  B200_CUDA(cudaEventRecord(ctx->ev1, st));
}

// ---- tensor-core pipeline (wavernn_tc.cuh): 33 ... 256 rows, plain batches ----------------------------------------------
static bool tc_eligible(const b200tts_wavernn* ctx, int rows, bool folding, bool packing) {
  return ctx->tc_ok && ctx->pm.ok && !folding && !packing && rows >= 1 && rows <= kTcRows * kTcMaxGroups;
}
static void launch_tc(b200tts_wavernn* ctx, const float* d_mel, GenArgs& ua, cudaStream_t st) {
  const b200tts_wavernn_cfg& c = ctx->cfg;
  const PushModel& pm = ctx->pm;
  const int rows = ua.B, T = ua.T, hop = c.hop_length;
  const int ng = (rows + kTcRows - 1) / kTcRows;
  ctx->push_tab.ensure((size_t)rows * (T + 1) * pm.ncta * kPushCondRows * sizeof(float));
  {
    constexpr int FT = 8;
    dim3 grid((T + 1 + FT - 1) / FT, rows);
    size_t smem = (size_t)(c.feat_dims + c.res_out_dims) * FT * sizeof(float);
    push_cond_table_kernel<FT><<<grid, 256, smem, st>>>(ctx->pcw, d_mel, ua.aux_frames, rows, T, ctx->push_tab.as<float>());
    B200_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  ctx->tc_vec.ensure((size_t)TV_COUNT * ng * 2 * kTcVecBytes);
  ctx->tc_x1f.ensure((size_t)ng * 2 * kTcRows * 512 * sizeof(float));
  ctx->tc_win.ensure((size_t)ng * 2 * kTcWinCopies * kTcRows * 16 * sizeof(unsigned long long));
  ctx->tc_cond.ensure((size_t)32 * 2 * ng * kTcCondBlk * kTcCondSlot * sizeof(float));
  REQUIRE((size_t)hop * ctx->NT * sizeof(float) <= (size_t)kTcFirMaxBytes, B200TTS_EINVAL, "tensor-core kernel: FIR table does not fit its shared-memory slot");
  const size_t ncnt = (size_t)ng * TCN_COUNT * 32;
  ctx->tc_cnt.ensure((ncnt + 32) * sizeof(unsigned));
  B200_CUDA(cudaMemsetAsync(ctx->tc_cnt.p, 0, (ncnt + 32) * sizeof(unsigned), st));
  int* d_err = reinterpret_cast<int*>(ctx->tc_cnt.as<unsigned>() + ncnt);
  ctx->d_grid_error = d_err;
  TcArgs a{};
  a.wimg = ctx->tc_wimg.as<uint8_t>();
  a.prm = ctx->tc_prm.as<float>();
  a.vec = ctx->tc_vec.as<uint8_t>();
  a.x1f = ctx->tc_x1f.as<float>();
  a.winners = ctx->tc_win.as<unsigned long long>();
  a.cnt = ctx->tc_cnt.as<unsigned>();
  a.condg = ctx->tc_cond.as<float>();
  a.error = d_err;
  a.tab = ctx->push_tab.as<float>();
  a.fir = ctx->d_fir;
  a.NT = ctx->NT; a.B = rows; a.S = ua.S; a.T = T; a.hop = hop; a.steps = ua.steps; a.ng = ng; a.NC = ctx->NC;
  a.rng_mode = ua.rng_mode; a.seed = ua.seed; a.utt_offset = ua.utt_offset; a.utt_ids = ua.utt_ids; a.q = ua.q;
  a.teacher = ua.teacher; a.logits_out = ua.logits_out; a.labels = ua.labels;
  a.prof = nullptr;
  const bool prof = getenv("B200TTS_TC_PROF") != nullptr;
  a.prof_mode = prof ? atoi(getenv("B200TTS_TC_PROF")) : 0;
#ifndef B200TTS_TC_CHAIN_PROF
  if (a.prof_mode == 2) {      // the chain-event probe is a compile-time option (wavernn_tc.cuh): fall back to the cycle accounting
    fprintf(stderr, "libb200tts: B200TTS_TC_PROF=2 needs a build with -DB200TTS_TC_CHAIN_PROF; printing the cycle accounting instead\n");
    a.prof_mode = 1;
  }
#endif
  if (prof) {
    ctx->push_prof.ensure((size_t)kTcCtas * 12 * sizeof(long long));
    B200_CUDA(cudaMemsetAsync(ctx->push_prof.p, 0, (size_t)kTcCtas * 12 * sizeof(long long), st));
    a.prof = ctx->push_prof.as<long long>();
  }
  ctx->last_push_ncta = 0;
  ctx->last_grid_ncta = 0;
  B200_CUDA(cudaFuncSetAttribute(wavernn_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBytes));
  int per_sm = 0;
  B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wavernn_tc_kernel, kTcThreads, (size_t)kTcSmemBytes));
  REQUIRE(per_sm * ctx->sm_count >= kTcCtas, B200TTS_EINVAL, "tensor-core kernel cannot be made co-resident on this device");
  B200_CUDA(cudaEventRecord(ctx->ev0, st));
  void* args[] = {(void*)&a};
  B200_CUDA(cudaLaunchCooperativeKernel((const void*)wavernn_tc_kernel, dim3(kTcCtas), dim3(kTcThreads), args, (size_t)kTcSmemBytes, st));
  ctx->launches++;
  B200_CUDA(cudaEventRecord(ctx->ev1, st));
  if (prof) {      // development aid: mean cycles per lock-step and role, to stderr
    B200_CUDA(cudaStreamSynchronize(st));
    std::vector<long long> h((size_t)kTcCtas * 12);
    B200_CUDA(cudaMemcpy(h.data(), ctx->push_prof.p, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    static const char* names[12] = {"ld:cnt", "ld:empty+issue", "mma:accfree", "mma:full", "mma:issue", "epi:wait-main", "epi:wait-other",
                                    "epi:tmem", "epi:math+store", "epi:publish", "cond:wait", "cond:compute"};
    static const char* roles[5] = {"GRU1", "GRU2", "fc1", "fc2", "fc3"};
    const int lo[6] = {0, 32, 96, 112, 128, 144};
    if (a.prof_mode == 2 && ua.steps > 2) {    // chain events of group 0 (first CTA of every role), mean ns between consecutive events
      const double n = (double)(ua.steps - 1);
      auto ev = [&](int cta, int slot) { return (double)h[(size_t)cta * 12 + slot] / n; };
      const double a0 = ev(0, 5), b0 = ev(0, 6), a2 = ev(0, 7);
      double prev = b0;
      fprintf(stderr, "tc chain (ns, group 0): GRU1 winners->published %.0f", b0 - a0);
      for (int r = 1; r < 5; ++r) {
        const double c0 = ev(lo[r], 0), d0 = ev(lo[r], 5), e0 = ev(lo[r], 6);
        fprintf(stderr, " | hop %.0f  %s GEMM %.0f (first stage %.0f, last stage %.0f, last MMA issued %.0f, accumulator seen %.0f) epilogue %.0f", c0 - prev,
                roles[r], d0 - c0, ev(lo[r], 2) - c0, ev(lo[r], 3) - c0, ev(lo[r], 4) - c0, d0 - c0, e0 - d0);
        prev = e0;
      }
      fprintf(stderr, " | hop %.0f  (step %.0f)\n", a2 - prev, a2 - a0);
    } else
    for (int r = 0; r < 5; ++r) {
      fprintf(stderr, "tc prof %-4s (cycles per lock-step):", roles[r]);
      for (int i = 0; i < 12; ++i) {
        double s = 0;
        for (int cta = lo[r]; cta < lo[r + 1]; ++cta) s += (double)h[(size_t)cta * 12 + i];
        fprintf(stderr, " %s=%.0f", names[i], s / (lo[r + 1] - lo[r]) / ua.steps);
      }
      fprintf(stderr, "\n");
    }
  }
}

// After the stream has been synchronised: did the last grid launch abandon a barrier?
static void check_grid_error(b200tts_wavernn* ctx) {
  if (!ctx->d_grid_error) return;
  int flag = 0;
  B200_CUDA(cudaMemcpy(&flag, ctx->d_grid_error, sizeof(int), cudaMemcpyDeviceToHost));
  REQUIRE(flag == 0, B200TTS_ECUDA, "grid kernel: a grid-barrier wait timed out (co-resident CTA missing); results are invalid");
}

static void run_generate_rows(b200tts_wavernn* ctx, const float* d_mel, int B, int T, const b200tts_rng* rng,
                              const b200tts_gen_opts* opts, int16_t* d_labels, double* d_wave, cudaStream_t st,
                              StreamWave* sw = nullptr);

// The wide mapping streams a sample-rate mel buffer [S][feat][Bp] (1.8 GB at 256 rows x 80 frames, 22.5 GB at 256 x 1000): long
// utterances x large batches would run out of memory before anything else.  Such a call is cut into row ranges whose buffers stay
// under a budget (default 8 GB, env B200TTS_MAX_COND_BYTES); the noise is keyed by the global row, so the result is unchanged.
// (Not for the debug modes whose buffers are indexed [step][row]: external noise, logits.)
static bool tc_eligible(const b200tts_wavernn* ctx, int rows, bool folding, bool packing);
static void run_generate(b200tts_wavernn* ctx, const float* d_mel, int B, int T, const b200tts_rng* rng,
                         const b200tts_gen_opts* opts, int16_t* d_labels, double* d_wave, cudaStream_t st) {
  const double budget = getenv("B200TTS_MAX_COND_BYTES") ? atof(getenv("B200TTS_MAX_COND_BYTES")) : 8e9;   // read per call
  const b200tts_wavernn_cfg& c = ctx->cfg;
  const double per_row = (double)T * c.hop_length * c.feat_dims * sizeof(float);
  const bool debug_bufs = (rng && rng->mode == B200TTS_RNG_EXT_EXPONENTIAL) || (opts && opts->d_logits);
  const bool folding = opts && opts->fold_target > 0;
  const bool packing = opts && opts->d_pack_utt;
  // kernel=auto and more than 256 rows: launches of 256 rows through the tensor-core pipeline (50 us per lock-step each) beat the
  // wide mapping on the whole batch (68 us per 256 rows); the noise is keyed by the global row, so the result does not change
  const bool tc_off = getenv("B200TTS_TC") != nullptr && getenv("B200TTS_TC")[0] == '0';
  const bool tc_slices = B > kTcRows * kTcMaxGroups && !tc_off && (!opts || opts->kernel == B200TTS_KERNEL_AUTO) && !debug_bufs && d_labels &&
                         tc_eligible(ctx, kTcRows * kTcMaxGroups, folding, packing);
  const bool sliceable = tc_slices || B > 256 || per_row * 256 > budget;
  if (!sliceable || debug_bufs || folding || packing || (!tc_slices && per_row * ((B + 255) / 256 * 256) <= budget) || !d_labels) {
    run_generate_rows(ctx, d_mel, B, T, rng, opts, d_labels, d_wave, st);
    return;
  }
  int rows = tc_slices ? kTcRows * kTcMaxGroups : (int)(budget / per_row);
  if (!tc_slices) rows = rows >= 256 ? rows / 256 * 256 : (rows >= 32 ? 32 : std::max(rows, 1));
  const size_t S = (size_t)T * c.hop_length, wave_len = (size_t)(T - 1) * c.hop_length;
  for (int r0 = 0; r0 < B; r0 += rows) {
    const int nb = std::min(rows, B - r0);
    b200tts_rng r{};
    if (rng) r = *rng;
    if (r.d_utterance_ids) r.d_utterance_ids += r0;
    else r.utterance_offset += (uint64_t)r0;
    b200tts_gen_opts o{};
    if (opts) o = *opts;
    else o.mu_law = 1;
    if (o.d_teacher) o.d_teacher += (size_t)r0 * S;
    if (o.d_utt_frames) o.d_utt_frames += r0;
    run_generate_rows(ctx, d_mel + (size_t)r0 * c.feat_dims * T, nb, T, &r, &o, d_labels + (size_t)r0 * S,
                      d_wave ? d_wave + (size_t)r0 * wave_len : nullptr, st);
  }
}

static void run_generate_rows(b200tts_wavernn* ctx, const float* d_mel, int B, int T, const b200tts_rng* rng,
                              const b200tts_gen_opts* opts, int16_t* d_labels, double* d_wave, cudaStream_t st,
                              StreamWave* sw) {
  const b200tts_wavernn_cfg& c = ctx->cfg;
  const int hop = c.hop_length, S = T * hop, O = c.res_out_dims;
  b200tts_gen_opts o{};
  if (opts) o = *opts;
  else o.mu_law = 1;
  b200tts_rng r{};
  if (rng) r = *rng;
  REQUIRE(r.mode == B200TTS_RNG_PHILOX || r.mode == B200TTS_RNG_EXT_EXPONENTIAL, B200TTS_EINVAL, "unknown rng mode");
  REQUIRE(r.mode != B200TTS_RNG_EXT_EXPONENTIAL || r.d_q, B200TTS_EINVAL, "EXT_EXPONENTIAL needs d_q");
  REQUIRE(o.max_steps >= 0 && o.max_steps <= S, B200TTS_EINVAL, "max_steps out of range");
  const int steps = o.max_steps ? o.max_steps : S;
  const int fade_len = 20 * hop;                      // fatchord_version.py:256
  const int wave_len = (T - 1) * hop;                 // :184
  if (d_wave || sw) {
    REQUIRE(steps == S, B200TTS_EINVAL, "a wave needs all steps (max_steps must be 0)");
    REQUIRE(wave_len >= fade_len, B200TTS_EINVAL,
            "T must be >= 21 frames: the reference's 20-hop fade-out (fatchord_version.py:256-258) fails below that");
  }
  int kernel = o.kernel;
  if (kernel == B200TTS_KERNEL_AUTO) {
    kernel = ctx->gm.ok ? B200TTS_KERNEL_GRID : B200TTS_KERNEL_UTTERANCE;
    if (!ctx->gm.ok && !ctx->warned_fallback) {      // never silently: this path is ~4x slower
      ctx->warned_fallback = true;
      fprintf(stderr, "libb200tts: these hparams / this device cannot run the weight-stationary grid kernel; kernel=auto falls "
                      "back to the L2-streaming utterance kernel (about 4x slower at large batch)\n");
    }
  }
  REQUIRE(kernel == B200TTS_KERNEL_UTTERANCE || kernel == B200TTS_KERNEL_GRID || kernel == B200TTS_KERNEL_TC, B200TTS_EINVAL,
          "unknown kernel selector");
  const bool folding = o.fold_target > 0;
  FoldGeom fg{};
  if (folding) {
    REQUIRE(B == 1, B200TTS_EINVAL, "fold-with-overlap generation takes exactly one utterance (the reference folds x[0] only)");
    REQUIRE(o.fold_overlap >= 2 && o.fold_target >= 1, B200TTS_EINVAL, "fold target/overlap out of range");
    REQUIRE(steps == S, B200TTS_EINVAL, "max_steps is not supported together with folding");
    REQUIRE(S > o.fold_overlap, B200TTS_EINVAL, "utterance shorter than the fold overlap");
    fg = fold_geometry(S, o.fold_target, o.fold_overlap);
    REQUIRE(fg.nfold >= 1 && fg.nfold <= 65535, B200TTS_EINVAL, "fold count out of range");
  }
  const bool packing = o.d_pack_utt != nullptr;
  if (packing) {
    REQUIRE(!folding && o.d_pack_start && o.pack_rows >= 1 && o.pack_rows <= 32 && o.pack_segs >= 1 && o.pack_steps >= 1, B200TTS_EINVAL,
            "bad packed-row schedule (pack_rows 1..32, pack_segs >= 1, pack_steps >= 1, not together with folding)");
    REQUIRE(o.max_steps == 0 && !o.d_logits && !o.d_teacher && r.mode == B200TTS_RNG_PHILOX && d_labels, B200TTS_EINVAL,
            "packed generation takes PHILOX noise, all steps, caller-owned labels and no debug buffers");
  }
  const int GB = folding ? fg.nfold : B;            // rows the generation kernels see
  const int GS = folding ? fg.L : S;                // steps per row
  ctx->aux_frames.ensure((size_t)B * T * O * sizeof(float));
  int16_t* labels = d_labels;
  if (!labels) {
    ctx->labels.ensure((size_t)GB * GS * sizeof(int16_t));
    labels = ctx->labels.as<int16_t>();
  }
  bool use_tc = false;
  // kernel=auto: the tensor-core pipeline costs ~50 us per lock-step whatever the row count (1 or 2 groups of 128 rows in flight),
  // the wide CUDA-core mapping 33.8 / 41.4 / 68.0 us at 64 / 128 / 256 rows -> the crossover is near 160 rows (env
  // B200TTS_TC_MIN_ROWS; B200TTS_TC=0 keeps the CUDA-core mappings).  Fold mode and packed rows stay on the other kernels.
  static const int tc_min_rows = getenv("B200TTS_TC_MIN_ROWS") ? atoi(getenv("B200TTS_TC_MIN_ROWS")) : 161;
  static const bool tc_off = getenv("B200TTS_TC") != nullptr && getenv("B200TTS_TC")[0] == '0';
  if (o.kernel == B200TTS_KERNEL_AUTO && kernel == B200TTS_KERNEL_GRID && !tc_off && GB >= tc_min_rows && tc_eligible(ctx, GB, folding, packing))
    kernel = B200TTS_KERNEL_TC;
  if (kernel == B200TTS_KERNEL_TC) {
    REQUIRE(tc_eligible(ctx, GB, folding, packing), B200TTS_EINVAL,
            "kernel=tc needs rnn_dims = fc_dims = 512, 10-bit classes, >= 144 SMs, 1..256 rows, no folding / packing");
    use_tc = true;
    kernel = B200TTS_KERNEL_GRID;
  }
  const bool use_push = !use_tc && kernel == B200TTS_KERNEL_GRID && push_eligible(ctx, packing ? o.pack_rows : GB);
  REQUIRE(!packing || use_push, B200TTS_EINVAL, "packed generation needs the push kernel (kernel=auto/grid, rnn_dims = fc_dims = 512)");
  REQUIRE(!sw || (use_push && GB <= kMgG), B200TTS_EINVAL,
          "streaming needs the push kernel (kernel=auto/grid, 1..32 rows, rnn_dims = fc_dims = 512)");
  if (kernel == B200TTS_KERNEL_GRID && !ctx->gm.ok)
    throw Error(B200TTS_EINVAL, "kernel=grid was requested but this model/device cannot run the weight-stationary grid kernel "
                                "(needs rnn_dims == fc_dims, n_classes == 2*rnn_dims, cooperative launch, R/4 <= SM count)");
  float* mels_up = nullptr;
  if (kernel == B200TTS_KERNEL_UTTERANCE || (folding && !use_push)) {
    ctx->mels_up.ensure((size_t)B * S * c.feat_dims * sizeof(float));
    mels_up = ctx->mels_up.as<float>();
  }
  run_upsample(ctx, d_mel, B, T, mels_up, ctx->aux_frames.as<float>(), nullptr, st);

  GenArgs a{};
  a.mels_up = ctx->mels_up.as<float>();
  a.aux_frames = ctx->aux_frames.as<float>();
  a.B = GB; a.S = GS; a.T = folding ? GS : T; a.hop = folding ? 1 : hop; a.steps = folding ? GS : steps;
  a.rng_mode = r.mode; a.seed = r.seed; a.utt_offset = r.utterance_offset; a.q = r.d_q;
  a.utt_ids = reinterpret_cast<const unsigned long long*>(r.d_utterance_ids);
  REQUIRE(!(folding && r.d_utterance_ids), B200TTS_EINVAL, "d_utterance_ids cannot be combined with fold-with-overlap generation");
  a.teacher = o.d_teacher; a.logits_out = o.d_logits; a.labels = labels;

  ctx->last_kernel = kernel == B200TTS_KERNEL_UTTERANCE ? 1 : (use_tc ? 5 : (use_push ? (GB > kMgG && !packing ? 4 : 3) : 2));
  if (kernel == B200TTS_KERNEL_UTTERANCE) {
    if (folding) {   // per-fold conditioning in the row-major layout this kernel reads, aux per sample (hop = 1)
      ctx->fold_mels.ensure((size_t)GB * GS * c.feat_dims * sizeof(float));
      ctx->fold_aux.ensure((size_t)GB * GS * O * sizeof(float));
      size_t n = (size_t)GB * GS * (c.feat_dims + O);
      unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx->sm_count * 32);
      fold_cond_kernel<<<grid, 256, 0, st>>>(ctx->mels_up.as<float>(), ctx->aux_frames.as<float>(), S, hop, c.feat_dims, O, fg.L,
                                             fg.stride, fg.nfold, ctx->fold_mels.as<float>(), ctx->fold_aux.as<float>());
      B200_CUDA(cudaGetLastError());
      ctx->launches++;
      a.mels_up = ctx->fold_mels.as<float>();
      a.aux_frames = ctx->fold_aux.as<float>();
    }
    ctx->d_grid_error = nullptr;
    B200_CUDA(cudaEventRecord(ctx->ev0, st));
    // utterances per CTA: enough CTAs to cover the SMs first, then amortise the L2 weight stream over more rows
    int per = (GB + ctx->sm_count - 1) / ctx->sm_count;
    if (per <= 1) launch_utt<1>(ctx, a, st);
    else if (per <= 2) launch_utt<2>(ctx, a, st);
    else if (per <= 4) launch_utt<4>(ctx, a, st);
    else launch_utt<8>(ctx, a, st);
    B200_CUDA(cudaEventRecord(ctx->ev1, st));
  } else if (use_tc) {
    launch_tc(ctx, d_mel, a, st);
  } else if (use_push) {
    PackInfo pi{o.d_pack_utt, o.d_pack_start, o.pack_rows, o.pack_segs, o.pack_steps, B};
    if (sw) { sw->utt_frames = o.d_utt_frames; sw->fade_len = fade_len; sw->mu_law = o.mu_law; }
    launch_push(ctx, d_mel, a, st, folding ? &fg : nullptr, T, packing ? &pi : nullptr, sw);
  } else {
    launch_grid(ctx, d_mel, a, st, folding ? &fg : nullptr, S);
  }
  ctx->ev_valid = true;
  if (d_wave) {
    if (folding) {
      xfade_unfold_kernel<<<(wave_len + 255) / 256, 256, 0, st>>>(labels, fg.nfold, fg.L, o.fold_target, o.fold_overlap, wave_len,
                                                                  fade_len, ctx->NC, o.mu_law, ctx->d_grid_error, d_wave);
    } else {
      dim3 grid((wave_len + 255) / 256, B);
      finish_wave_kernel<<<grid, 256, 0, st>>>(labels, S, wave_len, fade_len, ctx->NC, o.mu_law, o.d_utt_frames, hop, ctx->d_grid_error,
                                               d_wave);
    }
    B200_CUDA(cudaGetLastError());
    ctx->launches++;
  }
}

extern "C" int b200tts_wavernn_fold_geometry(int T, int hop, int target, int overlap, int* n_folds, int* fold_len) {
  API_BEGIN
  REQUIRE(T >= 1 && hop >= 1 && target >= 1 && overlap >= 2 && n_folds && fold_len, B200TTS_EINVAL, "bad argument");
  REQUIRE(T * hop > overlap, B200TTS_EINVAL, "utterance shorter than the fold overlap");
  FoldGeom g = fold_geometry(T * hop, target, overlap);
  *n_folds = g.nfold;
  *fold_len = g.L;
  API_END
}

extern "C" int b200tts_wavernn_generate(b200tts_wavernn* ctx, const float* d_mel, int B, int T, const b200tts_rng* rng,
                                        const b200tts_gen_opts* opts, int16_t* d_labels, double* d_wave, void* stream) {
  API_BEGIN
  REQUIRE(ctx && d_mel, B200TTS_EINVAL, "null argument");
  REQUIRE(B >= 1 && T >= 1 && B <= 65535, B200TTS_EINVAL, "B must be 1..65535 and T positive");
  DeviceGuard dg(ctx->device);
  run_generate(ctx, d_mel, B, T, rng, opts, d_labels, d_wave, (cudaStream_t)stream);
  API_END
}

// Pinned host memory the device can write: the device alias of [p, p + bytes).  Pageable memory cannot be written by a running
// kernel (it would need a copy, i.e. the end of the kernel) -> EINVAL.
static void* host_alias(void* p, size_t bytes, const char* name) {
  for (const char* q : {(const char*)p, (const char*)p + bytes - 1}) {
    cudaPointerAttributes at{};
    B200_CUDA(cudaPointerGetAttributes(&at, q));
    REQUIRE(at.type == cudaMemoryTypeHost, B200TTS_EINVAL,
            std::string(name) + " must be PINNED host memory the device can write (cudaHostAlloc / torch pin_memory), not pageable "
            "or device memory");
  }
  void* d = nullptr;
  const cudaError_t e = cudaHostGetDevicePointer(&d, p, 0);
  if (e != cudaSuccess) {
    cudaGetLastError();
    throw Error(B200TTS_EINVAL, std::string(name) + ": pinned memory not mapped into the device address space: " + cudaGetErrorString(e));
  }
  return d;
}

extern "C" int b200tts_wavernn_generate_stream(b200tts_wavernn* ctx, const float* d_mel, int B, int T, const b200tts_rng* rng,
                                               const b200tts_gen_opts* opts, int chunk_steps, double* h_wave, int64_t* h_progress,
                                               int16_t* d_labels, double* d_wave, void* stream) {
  API_BEGIN
  REQUIRE(ctx && d_mel && h_wave && h_progress, B200TTS_EINVAL, "null argument");
  REQUIRE(chunk_steps >= 1, B200TTS_EINVAL, "chunk_steps must be >= 1");
  REQUIRE(B >= 1 && B <= 32 && T >= 1, B200TTS_EINVAL, "streaming takes 1..32 rows (the push kernel) and T positive");
  REQUIRE(((uintptr_t)h_progress & 7) == 0, B200TTS_EINVAL, "h_progress must be 8-byte aligned");
  if (opts) {
    REQUIRE(opts->fold_target == 0, B200TTS_EINVAL, "streaming does not take fold-with-overlap generation (its output crosses folds)");
    REQUIRE(!opts->d_pack_utt, B200TTS_EINVAL, "streaming does not take packed rows (an utterance would start mid-launch)");
    REQUIRE(opts->max_steps == 0, B200TTS_EINVAL, "streaming produces the whole wave (max_steps must be 0)");
    REQUIRE(opts->kernel == B200TTS_KERNEL_AUTO || opts->kernel == B200TTS_KERNEL_GRID, B200TTS_EINVAL,
            "streaming runs the push kernel only (kernel=auto or grid)");
  }
  REQUIRE(T >= 21, B200TTS_EINVAL, "T must be >= 21 frames: the reference's 20-hop fade-out (fatchord_version.py:256-258) fails below that");
  // the kernel choice (push kernel only) is made by run_generate_rows, like for b200tts_wavernn_generate
  void* dp = host_alias(h_progress, sizeof(int64_t), "h_progress");        // first CUDA call: ECUDA without a device
  DeviceGuard dg(ctx->device);
  const size_t wl = (size_t)(T - 1) * ctx->cfg.hop_length;
  void* dw = host_alias(h_wave, (size_t)B * wl * sizeof(double), "h_wave");
  __atomic_store_n(h_progress, (int64_t)0, __ATOMIC_RELEASE);
  StreamWave sw{reinterpret_cast<double*>(dw), reinterpret_cast<long long*>(dp), chunk_steps, nullptr, 0, 0};
  run_generate_rows(ctx, d_mel, B, T, rng, opts, d_labels, d_wave, (cudaStream_t)stream, &sw);
  API_END
}

extern "C" int b200tts_wavernn_stream_wait(const int64_t* h_progress, int64_t at_least, int timeout_ms, int64_t* progress) {
  API_BEGIN
  REQUIRE(h_progress && progress, B200TTS_EINVAL, "null argument");
  REQUIRE(timeout_ms >= 0, B200TTS_EINVAL, "timeout_ms must be >= 0");
  const auto t0 = std::chrono::steady_clock::now();
  const auto limit = t0 + std::chrono::milliseconds(timeout_ms);
  int64_t v = __atomic_load_n(h_progress, __ATOMIC_ACQUIRE);
  // spin for the first 200 us (a chunk of 275 steps takes 2.5-5.6 ms, the first one is what time-to-audio measures), then sleep
  // in 50-us naps: a waiting thread costs no core while the kernel runs for seconds
  for (unsigned it = 0; v < at_least && v >= 0; ++it) {
    const auto now = std::chrono::steady_clock::now();
    if (now >= limit) break;
    if (now - t0 > std::chrono::microseconds(200)) std::this_thread::sleep_for(std::chrono::microseconds(50));
    v = __atomic_load_n(h_progress, __ATOMIC_ACQUIRE);
  }
  *progress = v;
  API_END
}

extern "C" int b200tts_wavernn_generate_host(b200tts_wavernn* ctx, const float* h_mel, int B, int T, const b200tts_rng* rng,
                                             const b200tts_gen_opts* opts, int16_t* h_labels, double* h_wave) {
  API_BEGIN
  REQUIRE(ctx && h_mel, B200TTS_EINVAL, "null argument");
  REQUIRE(B >= 1 && T >= 1 && B <= 65535, B200TTS_EINVAL, "B must be 1..65535 and T positive");
  REQUIRE(!opts || (!opts->d_teacher && !opts->d_logits), B200TTS_EINVAL, "device-side debug buffers need the device entry point");
  REQUIRE(!rng || rng->mode == B200TTS_RNG_PHILOX, B200TTS_EINVAL, "the host entry point only takes the PHILOX mode");
  REQUIRE(!opts || opts->fold_target == 0 || !h_labels, B200TTS_EINVAL, "folded generation returns only the wave through the host entry point");
  DeviceGuard dg(ctx->device);
  const b200tts_wavernn_cfg& c = ctx->cfg;
  const size_t S = (size_t)T * c.hop_length, wave_len = (size_t)(T - 1) * c.hop_length;
  const size_t mel_bytes = (size_t)B * c.feat_dims * T * sizeof(float);
  const size_t lab_bytes = (size_t)B * S * sizeof(int16_t), wav_bytes = (size_t)B * wave_len * sizeof(double);
  cudaStream_t st = nullptr;   // legacy default stream: ordered with everything else the caller enqueued
  ctx->mel_in.ensure(mel_bytes);
  ctx->h_stage.ensure(std::max(mel_bytes, std::max(lab_bytes, wav_bytes)));
  std::memcpy(ctx->h_stage.p, h_mel, mel_bytes);
  B200_CUDA(cudaMemcpyAsync(ctx->mel_in.p, ctx->h_stage.p, mel_bytes, cudaMemcpyHostToDevice, st));
  ctx->labels.ensure(lab_bytes);
  double* d_wave = nullptr;
  if (h_wave) {
    ctx->wave.ensure(wav_bytes);
    d_wave = ctx->wave.as<double>();
  }
  run_generate(ctx, ctx->mel_in.as<float>(), B, T, rng, opts, ctx->labels.as<int16_t>(), d_wave, st);
  if (h_labels) {
    B200_CUDA(cudaMemcpyAsync(ctx->h_stage.p, ctx->labels.p, lab_bytes, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    std::memcpy(h_labels, ctx->h_stage.p, lab_bytes);
  }
  if (h_wave) {
    B200_CUDA(cudaMemcpyAsync(ctx->h_stage.p, ctx->wave.p, wav_bytes, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    std::memcpy(h_wave, ctx->h_stage.p, wav_bytes);
  }
  B200_CUDA(cudaStreamSynchronize(st));
  check_grid_error(ctx);
  API_END
}

extern "C" int b200tts_wavernn_check(b200tts_wavernn* ctx) {
  API_BEGIN
  REQUIRE(ctx, B200TTS_EINVAL, "null argument");
  DeviceGuard dg(ctx->device);
  B200_CUDA(cudaDeviceSynchronize());
  check_grid_error(ctx);
  API_END
}

// Register-only packed-fp32 FMA loop on every SM: the measured fp32 CUDA-core ceiling bench.py quotes the FLOP form against.
__global__ void fp32_peak_kernel(float* out, int iters) {
  float2 a[8], x = make_float2(1.0001f + threadIdx.x * 1e-7f, 0.9999f), y = make_float2(1e-3f, -1e-3f);
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = make_float2((float)i, (float)(i + 1));
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = __ffma2_rn(a[i], x, y);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += a[i].x + a[i].y;
  if (s == 123.456f) out[0] = s;
}
extern "C" int b200tts_debug_fp32_peak(int device, double* tflops) {
  API_BEGIN
  REQUIRE(tflops, B200TTS_EINVAL, "null argument");
  DeviceGuard dg(device);
  int sms = 0;
  B200_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  float* d = nullptr;
  B200_CUDA(cudaMalloc(&d, 16));
  cudaEvent_t e0, e1;
  B200_CUDA(cudaEventCreate(&e0));
  B200_CUDA(cudaEventCreate(&e1));
  const int iters = 20000, threads = 512, blocks = sms * 2;
  fp32_peak_kernel<<<blocks, threads>>>(d, 2000);       // warm-up
  double best = 0.0;
  for (int rep = 0; rep < 3; ++rep) {
    B200_CUDA(cudaEventRecord(e0));
    fp32_peak_kernel<<<blocks, threads>>>(d, iters);
    B200_CUDA(cudaEventRecord(e1));
    B200_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    B200_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double flop = 2.0 * 2.0 * 32.0 * (double)iters * blocks * threads;   // 32 FFMA2 per iteration, 2 FMAs each
    best = std::max(best, flop / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  *tflops = best;
  API_END
}

// Debug: per-phase cycle counters of the last grid-kernel launch (needs env B200TTS_GRID_PROF=1 at generate time).
// out[12] = mean over CTAs of {P0 compute, P0 barrier, P1 compute, P1 barrier, ...} in SM cycles.
extern "C" int b200tts_wavernn_debug_phase_cycles(b200tts_wavernn* ctx, double* out12) {
  API_BEGIN
  REQUIRE(ctx && out12, B200TTS_EINVAL, "null argument");
  const bool push = ctx->last_grid_ncta == 0 && ctx->last_push_ncta > 0 && ctx->push_prof.p;
  REQUIRE(push || (ctx->grid_prof.p && ctx->last_grid_ncta > 0), B200TTS_EINVAL, "no phase profile recorded");
  DeviceGuard dg(ctx->device);
  const int n = push ? ctx->last_push_ncta : ctx->last_grid_ncta;
  std::vector<long long> h((size_t)n * 12);
  B200_CUDA(cudaDeviceSynchronize());
  B200_CUDA(cudaMemcpy(h.data(), push ? ctx->push_prof.p : ctx->grid_prof.p, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
  for (int i = 0; i < 12; ++i) {
    double s = 0;
    for (int c = 0; c < n; ++c) s += (double)h[(size_t)c * 12 + i];
    out12[i] = s / n;
  }
  API_END
}

// ---- PHILOX noise dump ------------------------------------------------------------------------------
__global__ void philox_dump_kernel(unsigned long long seed, unsigned long long utt0, int B, int step0, int n_steps, int NC,
                                   float* __restrict__ q) {
  size_t total = (size_t)n_steps * B * (NC / 4);
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    int c4 = (int)(e % (NC / 4));
    size_t sb = e / (NC / 4);
    int b = (int)(sb % B), s = (int)(sb / B);
    float v[4];
    philox_exp4(seed, utt0 + (unsigned long long)b, (uint32_t)(step0 + s), (uint32_t)c4, v);
    *reinterpret_cast<float4*>(q + sb * NC + (size_t)c4 * 4) = make_float4(v[0], v[1], v[2], v[3]);
  }
}

extern "C" int b200tts_philox_exponential(int device, uint64_t seed, uint64_t utterance_offset, int B, int step0, int n_steps,
                                          int n_classes, float* d_q, void* stream) {
  API_BEGIN
  REQUIRE(d_q && B >= 1 && n_steps >= 1 && n_classes >= 4 && n_classes % 4 == 0 && step0 >= 0, B200TTS_EINVAL, "bad argument");
  DeviceGuard dg(device);
  size_t total = (size_t)n_steps * B * (n_classes / 4);
  unsigned grid = (unsigned)std::min<size_t>((total + 255) / 256, 148 * 16);
  philox_dump_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(seed, utterance_offset, B, step0, n_steps, n_classes, d_q);
  B200_CUDA(cudaGetLastError());
  API_END
}

// ================================================================================================================
// Tacotron-2 decoder
// ================================================================================================================
struct TacoConvW {          // one conv1d + folded BatchNorm
  const float *K, *bias, *scale, *shift;
  int k, Cin, Cout;
};
struct b200tts_taco {
  int device = 0;
  b200tts_taco_cfg cfg{};
  DeviceBuf weights, keys, act_a, act_b;
  TacoWeights tw{};
  // run-once neighbours (present when the weight list carried them)
  bool has_encoder = false, has_postnet = false;
  const float* embedding = nullptr;
  int vocab = 0, emb_dim = 0, enc_units = 0;
  TacoConvW enc_conv[3]{}, post_conv[5]{};
  const float *enc_kfw = nullptr, *enc_bfw = nullptr, *enc_kbw = nullptr, *enc_bbw = nullptr;
  const float *post_pk = nullptr, *post_pb = nullptr;
  int post_channels = 0;
  int64_t launches = 0;
  // weight-stationary single-sentence decoder (taco_grid.cuh)
  TacoGridModel tgm{};
  DeviceBuf tg_blob, tg_vec;
  bool tg_ok = false;
  int sm_count = 0;
};

extern "C" int b200tts_taco_create(b200tts_taco** out, int device, const b200tts_taco_cfg* cfg, const b200tts_tensor* weights,
                                   int n_weights) {
  API_BEGIN
  REQUIRE(out && cfg && weights && n_weights > 0, B200TTS_EINVAL, "null argument");
  *out = nullptr;
  const b200tts_taco_cfg& c = *cfg;
  const int M = c.num_mels, P = c.prenet_units, U = c.lstm_units, E = c.enc_dim, AD = c.attn_dim, NF = c.attn_filters, KW = c.attn_kernel;
  REQUIRE(M % 4 == 0 && P % 4 == 0 && U % 4 == 0 && E % 4 == 0 && AD % 4 == 0, B200TTS_EINVAL, "dims must be multiples of 4");
  REQUIRE(M <= 96 && P == 256 && 4 * U == 1024 && E <= 1024 && AD <= 256 && KW % 2 == 1 && KW * NF <= 992 && NF * AD <= 4096,
          B200TTS_EINVAL, "decoder dims outside what taco_decoder_kernel is laid out for");
  int ndev = 0;
  B200_CUDA(cudaGetDeviceCount(&ndev));
  REQUIRE(device >= 0 && device < ndev, B200TTS_EINVAL, "no such CUDA device");
  DeviceGuard dg(device);
  TensorMap tm;
  for (int i = 0; i < n_weights; ++i)
    if (weights[i].name) tm[weights[i].name] = &weights[i];
  auto ctx = new b200tts_taco();
  struct Cleanup { b200tts_taco* c; ~Cleanup() { if (c) b200tts_taco_destroy(c); } } cleanup{ctx};
  ctx->device = device;
  ctx->cfg = c;
  Packer pk;
  auto copy = [&](const std::string& name, std::initializer_list<int64_t> shape) {
    const b200tts_tensor* t = need(tm, name, shape);
    size_t n = 1;
    for (int64_t s : shape) n *= (size_t)s;
    size_t off = pk.add(n);
    std::memcpy(&pk.h[off], t->data, n * sizeof(float));
    return off;
  };
  const std::string D = "decoder/", L = D + "Location_Sensitive_Attention/";
  size_t o[21];
  o[0] = copy(D + "decoder_prenet/dense_1/kernel", {M, P}); o[1] = copy(D + "decoder_prenet/dense_1/bias", {P});
  o[2] = copy(D + "decoder_prenet/dense_2/kernel", {P, P}); o[3] = copy(D + "decoder_prenet/dense_2/bias", {P});
  o[4] = copy(D + "decoder_LSTM/multi_rnn_cell/cell_0/decoder_LSTM_1/kernel", {P + E + U, 4 * U});
  o[5] = copy(D + "decoder_LSTM/multi_rnn_cell/cell_0/decoder_LSTM_1/bias", {4 * U});
  o[6] = copy(D + "decoder_LSTM/multi_rnn_cell/cell_1/decoder_LSTM_2/kernel", {2 * U, 4 * U});
  o[7] = copy(D + "decoder_LSTM/multi_rnn_cell/cell_1/decoder_LSTM_2/bias", {4 * U});
  o[8] = copy(L + "query_layer/kernel", {U, AD});
  o[9] = copy(L + "location_features_convolution/kernel", {KW, 1, NF}); o[10] = copy(L + "location_features_convolution/bias", {NF});
  o[11] = copy(L + "location_features_layer/kernel", {NF, AD});
  o[12] = copy(L + "attention_variable_projection", {AD}); o[13] = copy(L + "attention_bias", {AD});
  o[14] = copy(D + "dense/kernel", {E + U, 1}); o[15] = copy(D + "dense/bias", {1});
  o[16] = copy(D + "linear_transform_projection/projection_linear_transform_projection/kernel", {U + E, M});
  o[17] = copy(D + "linear_transform_projection/projection_linear_transform_projection/bias", {M});
  o[18] = copy(D + "stop_token_projection/projection_stop_token_projection/kernel", {U + E, 1});
  o[19] = copy(D + "stop_token_projection/projection_stop_token_projection/bias", {1});
  o[20] = copy("memory_layer/kernel", {E, AD});
  // ---- optional run-once neighbours: encoder and postnet ----
  struct ConvOff { size_t K, bias, scale, shift; int k, Cin, Cout; };
  auto pack_conv = [&](const std::string& scope) {
    auto it = tm.find(scope + "/conv1d/kernel");
    REQUIRE(it != tm.end() && it->second->ndim == 3, B200TTS_EMISSING, "missing weight tensor '" + scope + "/conv1d/kernel'");
    const b200tts_tensor* kt = it->second;
    ConvOff c{};
    c.k = (int)kt->shape[0]; c.Cin = (int)kt->shape[1]; c.Cout = (int)kt->shape[2];
    c.K = copy(scope + "/conv1d/kernel", {c.k, c.Cin, c.Cout});
    c.bias = copy(scope + "/conv1d/bias", {c.Cout});
    const float* g = need(tm, scope + "/batch_normalization/gamma", {c.Cout})->data;
    const float* be = need(tm, scope + "/batch_normalization/beta", {c.Cout})->data;
    const float* mu = need(tm, scope + "/batch_normalization/moving_mean", {c.Cout})->data;
    const float* var = need(tm, scope + "/batch_normalization/moving_variance", {c.Cout})->data;
    c.scale = pk.add(c.Cout); c.shift = pk.add(c.Cout);
    for (int i = 0; i < c.Cout; ++i) {                 // tf.layers.batch_normalization, moving stats, epsilon 1e-3
      double sc = (double)g[i] / std::sqrt((double)var[i] + 1e-3);
      pk.h[c.scale + i] = (float)sc;
      pk.h[c.shift + i] = (float)((double)be[i] - (double)mu[i] * sc);
    }
    return c;
  };
  ConvOff encc[3]{}, postc[5]{};
  size_t o_emb = 0, o_kfw = 0, o_bfw = 0, o_kbw = 0, o_bbw = 0, o_pk = 0, o_pb = 0;
  if (tm.count("inputs_embedding") && tm.count("encoder_convolutions/conv_layer_1_encoder_convolutions/conv1d/kernel")) {
    const b200tts_tensor* et = tm["inputs_embedding"];
    REQUIRE(et->ndim == 2, B200TTS_ESHAPE, "inputs_embedding must be 2-D");
    ctx->vocab = (int)et->shape[0]; ctx->emb_dim = (int)et->shape[1];
    o_emb = copy("inputs_embedding", {ctx->vocab, ctx->emb_dim});
    for (int i = 0; i < 3; ++i) encc[i] = pack_conv("encoder_convolutions/conv_layer_" + std::to_string(i + 1) + "_encoder_convolutions");
    REQUIRE(encc[0].Cin == ctx->emb_dim && encc[2].Cout % 4 == 0 && E % 2 == 0, B200TTS_ESHAPE, "encoder conv shapes");
    const int EU = E / 2, CI = encc[2].Cout;
    REQUIRE(4 * EU == 1024, B200TTS_EINVAL, "encoder LSTM units must be 256");
    const std::string LS = "encoder_LSTM/bidirectional_rnn/";
    o_kfw = copy(LS + "fw/encoder_fw_LSTM/kernel", {CI + EU, 4 * EU}); o_bfw = copy(LS + "fw/encoder_fw_LSTM/bias", {4 * EU});
    o_kbw = copy(LS + "bw/encoder_bw_LSTM/kernel", {CI + EU, 4 * EU}); o_bbw = copy(LS + "bw/encoder_bw_LSTM/bias", {4 * EU});
    ctx->enc_units = EU;
    ctx->has_encoder = true;
  }
  if (tm.count("postnet_projection/projection_postnet_projection/kernel")) {
    for (int i = 0; i < 5; ++i) postc[i] = pack_conv("postnet_convolutions/conv_layer_" + std::to_string(i + 1) + "_postnet_convolutions");
    REQUIRE(postc[0].Cin == M, B200TTS_ESHAPE, "postnet conv 1 must take num_mels channels");
    ctx->post_channels = postc[4].Cout;
    o_pk = copy("postnet_projection/projection_postnet_projection/kernel", {ctx->post_channels, M});
    o_pb = copy("postnet_projection/projection_postnet_projection/bias", {M});
    ctx->has_postnet = true;
  }
  ctx->weights.ensure(pk.h.size() * sizeof(float));
  B200_CUDA(cudaMemcpy(ctx->weights.p, pk.h.data(), pk.h.size() * sizeof(float), cudaMemcpyHostToDevice));
  const float* b = ctx->weights.as<float>();
  TacoWeights& w = ctx->tw;
  w.pre1_k = b + o[0]; w.pre1_b = b + o[1]; w.pre2_k = b + o[2]; w.pre2_b = b + o[3];
  w.l1_k = b + o[4]; w.l1_b = b + o[5]; w.l2_k = b + o[6]; w.l2_b = b + o[7];
  w.q_k = b + o[8]; w.loc_k = b + o[9]; w.loc_b = b + o[10]; w.locl_k = b + o[11]; w.v_a = b + o[12]; w.b_a = b + o[13];
  w.mu_k = b + o[14]; w.mu_b = b + o[15]; w.fr_k = b + o[16]; w.fr_b = b + o[17]; w.st_k = b + o[18]; w.st_b = b + o[19];
  w.mem_k = b + o[20];
  w.mels = M; w.P = P; w.U = U; w.E = E; w.A = AD; w.NF = NF; w.KW = KW; w.zoneout = c.zoneout;
  auto bind = [&](const ConvOff& c0) { return TacoConvW{b + c0.K, b + c0.bias, b + c0.scale, b + c0.shift, c0.k, c0.Cin, c0.Cout}; };
  if (ctx->has_encoder) {
    ctx->embedding = b + o_emb;
    for (int i = 0; i < 3; ++i) ctx->enc_conv[i] = bind(encc[i]);
    ctx->enc_kfw = b + o_kfw; ctx->enc_bfw = b + o_bfw; ctx->enc_kbw = b + o_kbw; ctx->enc_bbw = b + o_bbw;
  }
  if (ctx->has_postnet) {
    for (int i = 0; i < 5; ++i) ctx->post_conv[i] = bind(postc[i]);
    ctx->post_pk = b + o_pk; ctx->post_pb = b + o_pb;
  }
  // ---- per-block weight blobs of the weight-stationary single-sentence decoder (taco_grid.cuh) ----
  {
    int coop = 0;
    B200_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
    B200_CUDA(cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device));
    if (coop && ctx->sm_count >= kTgCtas && P == 256 && U == 256 && E == 512 && AD == 128 && M <= 96 && KW <= 64) {
      TacoGridModel& g = ctx->tgm;
      g.M = M; g.P = P; g.U = U; g.E = E; g.KW = KW;
      int off = 0;
      auto take = [&](int n) { int o0 = off; off += (n + 3) & ~3; return o0; };
      g.oW1 = take(M * 2); g.oB1 = take(2);
      g.oWfold = take((U + E) * 2); g.oBfold = take(2);
      g.oW2 = take(P * 2); g.oB2 = take(2);
      g.oK1 = take((P + E + U) * 8); g.oBk1 = take(8);
      g.oK2 = take(2 * U * 8); g.oBk2 = take(8);
      g.oWq = take(U);
      g.oFloc = take(KW + 4);
      g.oProj = take((U + E) * 4 + 4);
      g.blob = off;
      const float* H = pk.h.data();
      const float *W1 = H + o[0], *b1 = H + o[1], *W2 = H + o[2], *b2 = H + o[3], *K1 = H + o[4], *bk1 = H + o[5], *K2 = H + o[6],
                  *bk2 = H + o[7], *Wq = H + o[8], *lock = H + o[9], *locb = H + o[10], *locl = H + o[11], *va = H + o[12], *ba = H + o[13],
                  *muk = H + o[14], *mub = H + o[15], *frk = H + o[16], *frb = H + o[17], *stk = H + o[18], *stb = H + o[19];
      // W_f . W_1 and b_f . W_1 + b_1 in float64
      std::vector<double> fold((size_t)(U + E) * P), bfold(P);
      for (int i = 0; i < U + E; ++i)
        for (int p2 = 0; p2 < P; ++p2) {
          double a = 0;
          for (int m = 0; m < M; ++m) a += (double)frk[(size_t)i * M + m] * (double)W1[(size_t)m * P + p2];
          fold[(size_t)i * P + p2] = a;
        }
      for (int p2 = 0; p2 < P; ++p2) {
        double a = b1[p2];
        for (int m = 0; m < M; ++m) a += (double)frb[m] * (double)W1[(size_t)m * P + p2];
        bfold[p2] = a;
      }
      std::vector<float> hb((size_t)kTgCtas * g.blob, 0.f);
      for (int c2 = 0; c2 < kTgCtas; ++c2) {
        float* d = &hb[(size_t)c2 * g.blob];
        for (int j = 0; j < 2; ++j) {
          const int col = 2 * c2 + j;
          for (int m = 0; m < M; ++m) d[g.oW1 + m * 2 + j] = W1[(size_t)m * P + col];
          d[g.oB1 + j] = b1[col];
          for (int i = 0; i < U + E; ++i) d[g.oWfold + i * 2 + j] = (float)fold[(size_t)i * P + col];
          d[g.oBfold + j] = (float)bfold[col];
          for (int k = 0; k < P; ++k) d[g.oW2 + k * 2 + j] = W2[(size_t)k * P + col];
          d[g.oB2 + j] = b2[col];
          for (int gate = 0; gate < 4; ++gate) {
            const int src = gate * U + col, dst = gate * 2 + j;
            for (int k = 0; k < P + E + U; ++k) d[g.oK1 + k * 8 + dst] = K1[(size_t)k * 4 * U + src];
            d[g.oBk1 + dst] = bk1[src];
            for (int k = 0; k < 2 * U; ++k) d[g.oK2 + k * 8 + dst] = K2[(size_t)k * 4 * U + src];
            d[g.oBk2 + dst] = bk2[src];
          }
        }
        for (int u = 0; u < U; ++u) d[g.oWq + u] = Wq[(size_t)u * AD + c2];
        double bl = ba[c2];
        for (int f = 0; f < NF; ++f) bl += (double)locb[f] * (double)locl[(size_t)f * AD + c2];
        for (int k = 0; k < KW; ++k) {
          double a = 0;
          for (int f = 0; f < NF; ++f) a += (double)lock[(size_t)k * NF + f] * (double)locl[(size_t)f * AD + c2];
          d[g.oFloc + k] = (float)a;
        }
        d[g.oFloc + KW] = (float)bl;
        d[g.oFloc + KW + 1] = va[c2];
        d[g.oFloc + KW + 2] = 1.0f - c.zoneout;
        d[g.oFloc + KW + 3] = c.zoneout;
        for (int i = 0; i < U + E; ++i) {
          d[g.oProj + i * 4 + 0] = muk[i < U ? E + i : i - U];          // attention.py:229 concatenates [context, query]
          d[g.oProj + i * 4 + 1] = stk[i];
          d[g.oProj + i * 4 + 2] = c2 < M ? frk[(size_t)i * M + c2] : 0.f;
        }
        d[g.oProj + (U + E) * 4 + 0] = mub[0];
        d[g.oProj + (U + E) * 4 + 1] = stb[0];
        d[g.oProj + (U + E) * 4 + 2] = c2 < M ? frb[c2] : 0.f;
      }
      ctx->tg_blob.ensure(hb.size() * sizeof(float));
      B200_CUDA(cudaMemcpy(ctx->tg_blob.p, hb.data(), hb.size() * sizeof(float), cudaMemcpyHostToDevice));
      ctx->tg_ok = true;
    }
  }
  cleanup.c = nullptr;
  *out = ctx;
  API_END
}

extern "C" void b200tts_taco_destroy(b200tts_taco* ctx) {
  if (!ctx) return;
  int prev = -1;
  cudaGetDevice(&prev);
  cudaSetDevice(ctx->device);
  ctx->weights.release();
  ctx->keys.release();
  ctx->act_a.release();
  ctx->act_b.release();
  ctx->tg_blob.release();
  ctx->tg_vec.release();
  if (prev >= 0) cudaSetDevice(prev);
  delete ctx;
}

static int taco_decode_impl(b200tts_taco* ctx, const float* d_memory, const int32_t* d_lengths, int B, int Tx_max,
                            const b200tts_taco_dropout* dropout, int max_steps, int window, const float* d_forced, float* d_frames,
                            float* d_stop, float* d_align, int32_t* d_nsteps, void* stream) {
  API_BEGIN
  REQUIRE(ctx && d_memory && d_lengths && d_frames && d_stop && d_nsteps, B200TTS_EINVAL, "null argument");
  REQUIRE(B >= 1 && Tx_max >= 1 && Tx_max <= kTacoMaxTx && max_steps >= 1, B200TTS_EINVAL, "B, Tx_max (<= 512), max_steps out of range");
  b200tts_taco_dropout d{};
  if (dropout) d = *dropout;
  REQUIRE(d.mode == B200TTS_TACO_DROPOUT_PHILOX || (d.mode == B200TTS_TACO_DROPOUT_EXT && d.d_masks), B200TTS_EINVAL,
          "bad dropout descriptor");
  DeviceGuard dg(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  const TacoWeights& w = ctx->tw;
  ctx->keys.ensure((size_t)B * Tx_max * w.A * sizeof(float));
  taco_keys_kernel<<<B * Tx_max, 128, w.E * sizeof(float), st>>>(d_memory, w.mem_k, B * Tx_max, w.E, w.A, ctx->keys.as<float>());
  B200_CUDA(cudaGetLastError());
  TacoArgs a{};
  a.memory = d_memory; a.keys = ctx->keys.as<float>(); a.lengths = d_lengths;
  a.B = B; a.Tx_max = Tx_max; a.max_steps = max_steps; a.window = window;
  a.rng_mode = d.mode; a.seed = d.seed; a.utt_offset = d.utterance_offset; a.masks = d.d_masks;
  a.frames = d_frames; a.stop = d_stop; a.align = d_align; a.nsteps = d_nsteps;
  a.forced = d_forced;
  static const bool tg_off = getenv("B200TTS_TACO_GRID") != nullptr && getenv("B200TTS_TACO_GRID")[0] == '0';
  if (B == 1 && ctx->tg_ok && !tg_off) {
    // ONE sentence: the weight-stationary 128-block decoder (taco_grid.cuh).  The sentence length is needed on the host to size
    // the exchange buffers; d_lengths is a device pointer, so Tx_max (the caller's padded length) bounds it and the kernel
    // reads the true length itself.
    const TacoGridModel& g = ctx->tgm;
    const int Txp = (Tx_max + 3) & ~3;
    const size_t copy = (size_t)2048 + (size_t)kTgCtas * Txp;
    ctx->tg_vec.ensure(2 * copy * sizeof(float) + 64);
    int* d_err = reinterpret_cast<int*>(ctx->tg_vec.as<float>() + 2 * copy);
    push_init_kernel<<<ctx->sm_count, 256, 0, st>>>(ctx->tg_vec.as<uint32_t>(), 2 * copy, nullptr, 0, d_err);
    B200_CUDA(cudaGetLastError());
    TacoGridArgs ga{};
    ga.wblob = ctx->tg_blob.as<float>();
    ga.vec = ctx->tg_vec.as<float>();
    ga.error = d_err;
    ga.memory = d_memory; ga.keys = ctx->keys.as<float>();
    ga.lengths = d_lengths;
    ga.Tx = Tx_max; ga.Txp = Txp; ga.max_steps = max_steps; ga.window = window;
    ga.rng_mode = d.mode; ga.seed = d.seed; ga.utt = d.utterance_offset; ga.masks = d.d_masks;
    ga.forced = d_forced; ga.Tx_alloc = Tx_max;
    ga.frames = d_frames; ga.stop = d_stop; ga.align = d_align; ga.nsteps = d_nsteps;
    const size_t fl = (size_t)g.blob + (size_t)(w.P + w.E + w.U) + 2 * w.U + (w.U + w.E) + w.P + 128 + 24 * (size_t)Txp + 176;
    const size_t smem = fl * sizeof(float);
    REQUIRE(smem <= 227 * 1024, B200TTS_EINVAL, "taco_grid_kernel: shared memory budget exceeded");
    B200_CUDA(cudaFuncSetAttribute(taco_grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    TacoGridModel gm = g;
    void* args[] = {(void*)&gm, (void*)&ga};
    B200_CUDA(cudaLaunchCooperativeKernel((const void*)taco_grid_kernel, dim3(kTgCtas), dim3(kTgThreads), args, smem, st));
    taco_grid_finish_kernel<<<1, 1, 0, st>>>(d_err, d_nsteps);
    B200_CUDA(cudaGetLastError());
    ctx->launches += 4;
    return B200TTS_OK;
  }
  size_t fl = 128 + w.P + (w.P + w.E + w.U) + 2 * w.U + 4 * w.U + 2 * w.U + (w.U + w.E) + w.A + 3 * kTacoMaxTx + 96 + 64 +
              (size_t)w.KW * w.NF + (size_t)w.NF * w.A + 16384;
  size_t smem = fl * sizeof(float);
  B200_CUDA(cudaFuncSetAttribute(taco_decoder_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  taco_decoder_kernel<<<B, kTacoThreads, smem, st>>>(w, a);
  B200_CUDA(cudaGetLastError());
  ctx->launches += 2;
  API_END
}

extern "C" int b200tts_taco_decode(b200tts_taco* ctx, const float* d_memory, const int32_t* d_lengths, int B, int Tx_max,
                                   const b200tts_taco_dropout* dropout, int max_steps, int window, float* d_frames, float* d_stop,
                                   float* d_align, int32_t* d_nsteps, void* stream) {
  return taco_decode_impl(ctx, d_memory, d_lengths, B, Tx_max, dropout, max_steps, window, nullptr, d_frames, d_stop, d_align, d_nsteps,
                          stream);
}

extern "C" int b200tts_taco_state_floats(const b200tts_taco* ctx, int Tx_max) {
  if (!ctx || Tx_max < 1) return B200TTS_EINVAL;
  return taco_state_floats(ctx->cfg.num_mels, ctx->cfg.enc_dim, ctx->cfg.lstm_units, Tx_max);
}

extern "C" int b200tts_taco_decode_forced(b200tts_taco* ctx, const float* d_memory, const int32_t* d_lengths, int B, int Tx_max,
                                          const b200tts_taco_dropout* dropout, int n_steps, int window, const float* d_states,
                                          float* d_frames, float* d_stop, float* d_align, int32_t* d_nsteps, void* stream) {
  if (!d_states) {
    g_err = "b200tts_taco_decode_forced needs d_states";
    return B200TTS_EINVAL;
  }
  return taco_decode_impl(ctx, d_memory, d_lengths, B, Tx_max, dropout, n_steps, window, d_states, d_frames, d_stop, d_align, d_nsteps,
                          stream);
}

extern "C" int b200tts_taco_philox_masks(int device, uint64_t seed, uint64_t utterance_offset, int B, int steps, int prenet_units,
                                         uint8_t* d_masks, void* stream) {
  API_BEGIN
  REQUIRE(d_masks && B >= 1 && steps >= 1 && prenet_units >= 4, B200TTS_EINVAL, "bad argument");
  DeviceGuard dg(device);
  size_t total = (size_t)B * steps * 2 * prenet_units;
  unsigned grid = (unsigned)std::min<size_t>((total + 255) / 256, 148 * 16);
  taco_philox_masks_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(seed, utterance_offset, B, steps, prenet_units, d_masks);
  B200_CUDA(cudaGetLastError());
  API_END
}

static void taco_launch_conv(b200tts_taco* ctx, const TacoConvW& cw, const float* x, const int* ids, const int* lengths, int B, int Tmax,
                             int act, bool clip_in, float lo, float hi, float* y, cudaStream_t st) {
  ConvArgs a{};
  a.x = x; a.ids = ids; a.table = ctx->embedding; a.lengths = lengths;
  a.K = cw.K; a.bias = cw.bias; a.bn_scale = cw.scale; a.bn_shift = cw.shift; a.y = y;
  a.Tmax = Tmax; a.Cin = cw.Cin; a.Cout = cw.Cout; a.k = cw.k; a.act = act; a.clip_in = clip_in ? 1 : 0; a.lo = lo; a.hi = hi;
  size_t smem = (size_t)(kConvTile + cw.k - 1) * cw.Cin * sizeof(float);
  dim3 grid((Tmax + kConvTile - 1) / kConvTile, B);
  taco_conv_bn_kernel<<<grid, 256, smem, st>>>(a);
  B200_CUDA(cudaGetLastError());
  ctx->launches++;
}

extern "C" int b200tts_taco_encode(b200tts_taco* ctx, const int32_t* d_ids, const int32_t* d_lengths, int B, int Tx_max, float* d_memory,
                                   void* stream) {
  API_BEGIN
  REQUIRE(ctx && d_ids && d_lengths && d_memory, B200TTS_EINVAL, "null argument");
  REQUIRE(ctx->has_encoder, B200TTS_EMISSING, "this context was created without the encoder variables");
  REQUIRE(B >= 1 && Tx_max >= 1 && Tx_max <= kTacoMaxTx, B200TTS_EINVAL, "B / Tx_max out of range");
  DeviceGuard dg(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  const int C = ctx->enc_conv[0].Cout;
  ctx->act_a.ensure((size_t)B * Tx_max * C * sizeof(float));
  ctx->act_b.ensure((size_t)B * Tx_max * C * sizeof(float));
  float* a = ctx->act_a.as<float>();
  float* bb = ctx->act_b.as<float>();
  taco_launch_conv(ctx, ctx->enc_conv[0], nullptr, d_ids, d_lengths, B, Tx_max, 1, false, 0.f, 0.f, a, st);
  taco_launch_conv(ctx, ctx->enc_conv[1], a, nullptr, d_lengths, B, Tx_max, 1, false, 0.f, 0.f, bb, st);
  taco_launch_conv(ctx, ctx->enc_conv[2], bb, nullptr, d_lengths, B, Tx_max, 1, false, 0.f, 0.f, a, st);
  const int U = ctx->enc_units, Cin = ctx->enc_conv[2].Cout;
  size_t smem = ((size_t)(Cin + U) + 4 * U + U + 4 * 4 * U) * sizeof(float);
  B200_CUDA(cudaFuncSetAttribute(taco_bilstm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  taco_bilstm_kernel<<<dim3(B, 2), kTacoThreads, smem, st>>>(a, d_lengths, Tx_max, Cin, U, ctx->enc_kfw, ctx->enc_bfw, ctx->enc_kbw,
                                                              ctx->enc_bbw, ctx->cfg.zoneout, d_memory);
  B200_CUDA(cudaGetLastError());
  ctx->launches++;
  API_END
}

extern "C" int b200tts_taco_postnet(b200tts_taco* ctx, const float* d_frames, const int32_t* d_nsteps, int B, int max_steps, float* d_mel,
                                    void* stream) {
  API_BEGIN
  REQUIRE(ctx && d_frames && d_nsteps && d_mel, B200TTS_EINVAL, "null argument");
  REQUIRE(ctx->has_postnet, B200TTS_EMISSING, "this context was created without the postnet variables");
  REQUIRE(B >= 1 && max_steps >= 1, B200TTS_EINVAL, "B / max_steps out of range");
  DeviceGuard dg(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  const int C = ctx->post_channels, M = ctx->cfg.num_mels;
  const float lo = -4.0f - 0.1f, hi = 4.0f;       // T2_output_range[0] - lower_bound_decay, T2_output_range[1] (tacotron.py:33,111-112)
  ctx->act_a.ensure((size_t)B * max_steps * C * sizeof(float));
  ctx->act_b.ensure((size_t)B * max_steps * C * sizeof(float));
  float* a = ctx->act_a.as<float>();
  float* bb = ctx->act_b.as<float>();
  taco_launch_conv(ctx, ctx->post_conv[0], d_frames, nullptr, d_nsteps, B, max_steps, 2, true, lo, hi, a, st);
  taco_launch_conv(ctx, ctx->post_conv[1], a, nullptr, d_nsteps, B, max_steps, 2, false, 0.f, 0.f, bb, st);
  taco_launch_conv(ctx, ctx->post_conv[2], bb, nullptr, d_nsteps, B, max_steps, 2, false, 0.f, 0.f, a, st);
  taco_launch_conv(ctx, ctx->post_conv[3], a, nullptr, d_nsteps, B, max_steps, 2, false, 0.f, 0.f, bb, st);
  taco_launch_conv(ctx, ctx->post_conv[4], bb, nullptr, d_nsteps, B, max_steps, 0, false, 0.f, 0.f, a, st);
  taco_postnet_proj_kernel<<<dim3(max_steps, B), 128, C * sizeof(float), st>>>(d_frames, a, d_nsteps, max_steps, C, M, ctx->post_pk,
                                                                                 ctx->post_pb, lo, hi, d_mel);
  B200_CUDA(cudaGetLastError());
  ctx->launches++;
  API_END
}
