// ovc_lib.cu -- host side of libovc_b200.so: context, checkpoint ingestion (weight-norm folding,
// Flip absorption, kernel-layout packing), workspace arena, the launch sequence of
// SynthesizerTrn.voice_conversion (openvoice/models.py:492-499) and the C ABI of include/ovc.h.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <optional>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/ovc.h"
#include "ovc_small.cuh"
#include "ovc_tcconv.cuh"
#include "ovc_tcpair.cuh"
#include "ovc_tts.cuh"
#include "ovc_refenc.cuh"
#include "ovc_variants.h"

namespace ovc {

static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

// every ABI entry point runs on its context's device and puts the caller's current device back on exit (PyTorch
// reads the current device through cudaGetDevice: a converter on cuda:N must not move the caller's default)
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};
#define ON_DEVICE(c)                                                                              \
  DeviceGuard dev_guard_((c)->device);                                                            \
  if (!dev_guard_.ok) return fail(OVC_ERR_CUDA, "cudaSetDevice(%d) failed", (c)->device)

#define CK(expr)                                                                                  \
  do {                                                                                            \
    cudaError_t e_ = (expr);                                                                      \
    if (e_ != cudaSuccess)                                                                        \
      return fail(OVC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, \
                  __LINE__);                                                                      \
  } while (0)

#define TRY(expr)                   \
  do {                              \
    int rc_ = (expr);               \
    if (rc_ != OVC_OK) return rc_;  \
  } while (0)

// cuTensorMapEncodeTiled, resolved through the runtime (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
      p = nullptr;
    cudaGetLastError();
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

static const VariantInfo kInfo[V_COUNT] = {
#define X(name, K, D, WM, WN, CI, EPI, NG, XA)                                                    \
  {#name, K, D, 32 * WM, 64 * WN, CI, EPI, 32 * WM * WN, ConvCfg<K, D, WM, WN, CI, EPI, NG, XA>::SMEM_BYTES},
    OVC_VARIANTS_ALL(X)
#undef X
};
static const LaunchFn kLaunch[V_COUNT] = {
#define X(name, K, D, WM, WN, CI, EPI, NG, XA) launch_##name,
    OVC_VARIANTS_ALL(X)
#undef X
};
static const PrepareFn kPrepare[V_COUNT] = {
#define X(name, K, D, WM, WN, CI, EPI, NG, XA) prepare_##name,
    OVC_VARIANTS_ALL(X)
#undef X
};

// The tensor-core conv instantiations, each with its dynamic shared memory.  launch_tc and launch_pair take their kernel
// from these tables and finalize sets every kernel's shared-memory limit from them, so whatever can be launched has its
// limit set.  A new instantiation is one more entry here.
struct TcConvKernel {
  int TN; bool in16, out16;   // output columns per CTA; fp16 input / output activations (precision 3)
  void (*fn)(TcConvArgs, int, int, CUtensorMap);
  size_t smem;
};
template <int TN, bool IN16 = false, bool OUT16 = false>
static TcConvKernel tcconv_entry() { return {TN, IN16, OUT16, tcconv_kernel<TN, IN16, OUT16>, TcnCfg<TN>::SMEM_BYTES}; }
static const TcConvKernel kTcConv[] = {
    tcconv_entry<128>(), tcconv_entry<64>(), tcconv_entry<32>(),
    tcconv_entry<128, false, true>(),   // conv_pre of precision 3: fp32 z_hat in, fp16 out
    tcconv_entry<128, true, true>(), tcconv_entry<64, true, true>(), tcconv_entry<32, true, true>()};

struct TcPairKernel {
  int TN;   // = the pair's channel count
  void (*fn)(TcPairArgs, int, int, CUtensorMap);
  size_t smem;
};
template <int TN>
static TcPairKernel tcpair_entry() { return {TN, tcpair_kernel<TN>, TcpCfg<TN>::SMEM_BYTES}; }
static const TcPairKernel kTcPair[] = {tcpair_entry<64>(), tcpair_entry<32>()};

static const TcConvKernel* find_tcconv(int TN, bool in16, bool out16) {
  for (const TcConvKernel& k : kTcConv)
    if (k.TN == TN && k.in16 == in16 && k.out16 == out16) return &k;
  return nullptr;
}
static const TcPairKernel* find_tcpair(int TN) {
  for (const TcPairKernel& k : kTcPair)
    if (k.TN == TN) return &k;
  return nullptr;
}

struct HostTensor {
  std::vector<int64_t> shape;
  std::vector<float> data;
  int64_t numel() const {
    int64_t n = 1;
    for (auto s : shape) n *= s;
    return n;
  }
};

// one convolution as the kernels see it
struct ConvLayer {
  int variant = -1;
  int rows = 0;        // packed output rows (multiple of CO_T)
  int row_tiles = 0;
  int cin = 0;         // real input channels
  int n_chunks = 0;
  size_t w_off = 0;    // float offsets into the device weight arena
  size_t b_off = 0;
  int K = 1;           // true taps / channels, for FLOP accounting
  int cout = 0;
  int out_mul = 1;     // outputs per input step (transposed convs: stride)
};

// one ResBlock conv as the tensor-core kernel sees it (pre-split hi/lo weights in operand layout)
struct TcLayer {
  size_t w_off = 0;   // float offsets into the tc weight arena
  size_t b_off = 0;
  int Cin = 0, Ntot = 0, K = 0, DIL = 1, TN = 0;
};

struct WNLayers {
  std::vector<ConvLayer> in, rs;
  std::vector<TcLayer> tc_in, tc_rs;   // tensor-core twins (channels-last)
};

// V1 TTS front half (TextEncoder / DurationPredictor / StochasticDurationPredictor, models.py:16-180): dense convs
// as tensor-core layers, small fp32 parameters as offsets into the fp32 arena.  Hyper-parameters are read off the
// checkpoint shapes (the reference takes them from config.json: api.py:26-31, models.py:451-465).
// k = 3 convs and the whole duration chain stay on the CUDA cores in plain fp32: the FFMA2 conv kernel on a [C][T]
// copy when the shape fits a variant (k 3, N % 64 == 0: every released checkpoint), else the one-thread-per-output
// kernel (sequential fmaf chain over w [K][Cin][N])
struct Fp32Dense { size_t w = 0, b = 0; int Cin = 0, K = 0, N = 0; bool fast = false; ConvLayer cl; };
struct DdsLayers {            // DDSConv, modules.py:84-113
  size_t sep_w[3] = {0}, sep_b[3] = {0}, n1g[3] = {0}, n1b[3] = {0}, n2g[3] = {0}, n2b[3] = {0};
  Fp32Dense c1x1[3];          // fp32: the spline inverses downstream amplify conditioning errors up to 1e3 x
};
struct TtsLayers {
  bool ready = false;
  int n_vocab = 0, n_speakers = 0, H = 0, C = 0, Fc = 0, heads = 0, n_layers = 0, window = 0, D = 0;
  size_t emb = 0, emb_g = 0;
  std::vector<TcLayer> qkv, o;
  std::vector<Fp32Dense> ffn1, ffn2;
  std::vector<size_t> relk, relv, ln1g, ln1b, ln2g, ln2b;
  TcLayer proj;
  Fp32Dense dp_c1, dp_c2, sdp_pre, sdp_proj;
  size_t dp_n1g = 0, dp_n1b = 0, dp_n2g = 0, dp_n2b = 0, dp_pw = 0, dp_pb = 0, dp_cw = 0, dp_cb = 0, sdp_cw = 0, sdp_cb = 0,
         ea = 0;               // ea: {m[0], logs[0]} of sdp.flows.0
  DdsLayers dds[4];            // 0: sdp.convs, j = 1..3: sdp.flows.{2j+1}.convs (flows.1 is never run in reverse, models.py:172)
  size_t cf_pre_w[4] = {0}, cf_pre_b[4] = {0}, cf_pw[4] = {0}, cf_pb[4] = {0};
};

// one profiled launch: kernel variant, family (1 = MRF conv: the roofline total of ovc_profile_read), algorithmic work
struct ProfRec {
  int variant = 0, family = 0;
  double flops = 0, bytes = 0;
  int tag = 0;   // (Cin << 16 | K << 8 | dilation) of a tensor-core launch, else 0
};

struct DebugBuf {
  float* d = nullptr;
  int64_t shape[4] = {0, 0, 0, 0};
  size_t floats = 0;
};

}  // namespace ovc

using namespace ovc;

struct ovc_ctx {
  ovc_hparams hp{};
  int device = 0;
  int sm_count = 0;
  std::map<std::string, HostTensor> sd;
  bool finalized = false;

  // device weights
  float* d_w = nullptr;
  size_t w_floats = 0;
  std::vector<float> h_w;   // staging while packing

  // layers
  ConvLayer enc_pre, enc_pre16, enc_proj;
  WNLayers enc_wn;
  ConvLayer flow_pre[4], flow_post[4];
  WNLayers flow_wn[4];
  ConvLayer dec_pre, dec_ups[4];
  ConvLayer rb_c1[12][3], rb_c2[12][3];
  TcLayer tc_c1[12][3], tc_c2[12][3], tc_ups[4], tc_pre;
  float* d_tcw = nullptr;      // tensor-core weight arena (hi/lo split)
  std::vector<float> h_tcw;
  int precision = 0;           // 0: fp32 FFMA everywhere; 1: 3xFP16 split-precision tcgen05 convs; 2: single-pass fp16;
                               // 3: as 1, but the generator stores fp16 activations and runs one fp16 pass per conv
  int wide_variant = 3;        // kernel of the 128-column tensor-core layers (see launch_tc); 3 = chosen per layer
  bool tts_simple = false;     // OVC_OPT_TTS_SIMPLE
  bool use_graph = true;       // OVC_OPT_GRAPH
  int use_pdl = 2;             // OVC_OPT_PDL: 0 off, 1 every tensor-core conv, 2 (default) the WaveNet stacks only -- short kernels
                               // whose fill / drain dominates (measured: 2 gives -0.5 .. -0.8 % at batch 32 and -2.4 % at
                               // batch 1; 1 gives +3 % at batch 32)
  // small calls: the three ResBlock branches of an MRF stage run concurrently on three streams, each kernel on a third
  // of the SMs (OVC_OPT_BRANCHES; taken when B * Tmax <= par_frames = 512 frames: measured -8 % at 258 frames, +2 % at 861)
  bool use_branches = true;
  int par_frames = 512;
  bool use_pair = true;        // OVC_OPT_PAIR: the HBM-bound ResBlock conv pairs (C <= 64, k = 3) as ONE kernel (ovc_tcpair.cuh)
  cudaStream_t br_stream[2] = {nullptr, nullptr};
  cudaEvent_t br_ev[4] = {nullptr, nullptr, nullptr, nullptr};
  size_t post_w_off = 0;
  // cond mat-vec
  size_t cond_w_off = 0, cond_b_off = 0;
  int* d_cond_wrow = nullptr;
  int* d_cond_sel = nullptr;
  int cond_rows_out = 0;
  int cond_off_enc = 0, cond_off_fsrc = 0, cond_off_ftgt = 0, cond_off_dec = 0;
  int cond_off_enc_tc = 0, cond_off_fsrc_tc = 0, cond_off_ftgt_tc = 0;   // same vectors in the tc kernel's column order

  // STFT tables (twiddles exp(-2 pi i m / 1024), periodic hann window)
  float2* d_tw = nullptr;
  float* d_win = nullptr;

  // ReferenceEncoder (extract_se): offsets into d_w, own scratch
  bool has_refenc = false;
  size_t re_conv_w[6] = {0}, re_conv_b[6] = {0}, re_wih = 0, re_whh = 0, re_bih = 0, re_bhh = 0, re_pw = 0, re_pb = 0,
         re_lng = 0, re_lnb = 0;
  int re_gru_in = 0;           // columns of ref_enc.gru.weight_ih_l0
  float* d_re = nullptr;
  size_t re_floats = 0;

  // workspace
  float* d_ws = nullptr;
  size_t ws_floats = 0;

  // TTS front half: layers, text-side workspace, and what ovc_tts_encode leaves for ovc_tts_decode
  TtsLayers tts;
  float* d_tts = nullptr;
  size_t tts_floats = 0;
  int tts_B = 0, tts_T = 0;

  // profiling: launch k of prof_log is bracketed by events ev[2k], ev[2k + 1]
  bool prof = false;
  std::vector<cudaEvent_t> ev;
  std::vector<ovc::ProfRec> prof_log;

  // debug taps
  bool debug = false;
  std::map<std::string, DebugBuf> taps;

  int launches = 0;

  // CUDA-graph replay of a repeated call (OVC_OPT_GRAPH): the launch sequence of a (entry point, shapes, buffers,
  // options) signature is captured on an internal stream the second time it is seen and replayed from then on; the
  // per-call scalars (noise seed, tau) reach the kernels through d_callp
  struct GraphEntry {
    std::vector<uintptr_t> key;
    cudaGraphExec_t exec = nullptr;
    int launches = 0;
    int seen = 0;
    uint64_t stamp = 0;
  };
  std::vector<GraphEntry> graphs;
  uint64_t graph_clock = 0;
  cudaStream_t cap_stream = nullptr;
  ovc::CallParams* d_callp = nullptr;
  int graph_replays = 0;       // diagnostics: calls served by a replay since creation
};

namespace ovc {

static size_t round_up(size_t v, size_t m) { return (v + m - 1) / m * m; }
static void drop_graphs(ovc_ctx* c);

static const HostTensor* find(const ovc_ctx* c, const std::string& k) {
  auto it = c->sd.find(k);
  return it == c->sd.end() ? nullptr : &it->second;
}

// Checkpoint tensors by key and expected shape (-1: any extent; an empty shape: not checked).  The first error is kept
// -- a missing key is OVC_ERR_MISSING, a mis-shaped one OVC_ERR_INVALID, both naming the key -- and a failed read
// returns null / an empty tensor, so a packing step checks ok() once after its reads.
struct Reader {
  ovc_ctx* c;
  int code = OVC_OK;
  std::string msg;

  bool ok() const { return code == OVC_OK; }
  int status() const { return ok() ? OVC_OK : fail(code, "%s", msg.c_str()); }
  void error(int cd, const std::string& k, const std::string& what) {
    if (ok()) { code = cd; msg = "checkpoint tensor '" + k + "' " + what; }
  }
  const HostTensor* get(const std::string& k, std::initializer_list<int64_t> shape) {
    const HostTensor* t = find(c, k);
    if (!t) { error(OVC_ERR_MISSING, k, "is missing"); return nullptr; }
    bool good = !shape.size() || t->shape.size() == shape.size();
    size_t i = 0;
    for (int64_t d : shape) { if (good && d >= 0 && t->shape[i] != d) good = false; ++i; }
    if (!good) { error(OVC_ERR_INVALID, k, "has shape " + dims(t->shape) + ", expected " + dims(shape)); return nullptr; }
    return t;
  }
  // effective weight of a (possibly weight-normed) conv: g * v / ||v|| over dims != 0
  // (torch.nn.utils.weight_norm dim=0; modules.py:160,172,182, models.py:247)
  HostTensor weff(const std::string& prefix, std::initializer_list<int64_t> shape) {
    if (find(c, prefix + ".weight")) {
      const HostTensor* w = get(prefix + ".weight", shape);
      return w ? *w : HostTensor();
    }
    const HostTensor* v = get(prefix + ".weight_v", shape);
    const HostTensor* g = v ? get(prefix + ".weight_g", {}) : nullptr;
    if (!g) return HostTensor();
    const int64_t d0 = v->shape[0];
    const int64_t inner = v->numel() / d0;
    if (g->numel() != d0) {
      error(OVC_ERR_INVALID, prefix + ".weight_g", "has " + std::to_string(g->numel()) + " elements, expected " + std::to_string(d0));
      return HostTensor();
    }
    HostTensor out = *v;
    for (int64_t i = 0; i < d0; ++i) {
      double ss = 0;
      for (int64_t j = 0; j < inner; ++j) { const double q = v->data[i * inner + j]; ss += q * q; }
      const float scale = g->data[i] / (float)std::sqrt(ss);
      for (int64_t j = 0; j < inner; ++j) out.data[i * inner + j] = v->data[i * inner + j] * scale;
    }
    return out;
  }
  // append to the fp32 parameter arena (256-byte aligned blobs); 0 for a failed read
  size_t put(const std::vector<float>& v) {
    const size_t o = round_up(c->h_w.size(), 64);
    c->h_w.resize(o + v.size());
    std::copy(v.begin(), v.end(), c->h_w.begin() + o);
    return o;
  }
  size_t put(const HostTensor* t) { return t ? put(t->data) : 0; }

  template <class S>
  static std::string dims(const S& s) {
    std::string r;
    for (int64_t d : s) r += (r.empty() ? "(" : ", ") + (d < 0 ? std::string("*") : std::to_string(d));
    return r + ")";
  }
};

// append a packed conv to the staging arena.  wfun(row_packed, ci, k) -> weight; bfun(row) -> bias
template <class WF, class BF>
static ConvLayer pack_conv(ovc_ctx* c, int variant, int rows, int cin, WF wfun, BF bfun, int bias_rows,
                           int trueK, int cout) {
  const VariantInfo& vi = kInfo[variant];
  ConvLayer L;
  L.variant = variant;
  L.rows = rows;
  L.row_tiles = rows / vi.CO_T;
  L.cin = cin;
  L.n_chunks = (cin + vi.CI_CH - 1) / vi.CI_CH;
  L.K = trueK;
  L.cout = cout;
  const int cin_pad = L.n_chunks * vi.CI_CH;
  L.w_off = round_up(c->h_w.size(), 64);   // 256-byte aligned blobs (TMA bulk needs 16)
  c->h_w.resize(L.w_off + (size_t)L.row_tiles * cin_pad * vi.K * vi.CO_T, 0.f);
  float* dst = c->h_w.data() + L.w_off;
  for (int rt = 0; rt < L.row_tiles; ++rt)
    for (int ci = 0; ci < cin_pad; ++ci)
      for (int k = 0; k < vi.K; ++k)
        for (int r = 0; r < vi.CO_T; ++r)
          dst[(((size_t)rt * cin_pad + ci) * vi.K + k) * vi.CO_T + r] =
              ci < cin ? wfun(rt * vi.CO_T + r, ci, k) : 0.f;
  L.b_off = round_up(c->h_w.size(), 64);
  c->h_w.resize(L.b_off + bias_rows, 0.f);
  for (int r = 0; r < bias_rows; ++r) c->h_w[L.b_off + r] = bfun(r);
  return L;
}

// packed row -> original row for the paired (tanh|sigmoid, m|logs) layouts: a thread's 8 rows
// are 4 channels of the first half followed by the same 4 channels of the second half
static inline int paired_row(int p, int half) {
  const int q = p / 8, r = p % 8;
  return r < 4 ? 4 * q + r : half + 4 * q + (r - 4);
}

// column order of the tensor-core WN gate: every 32-column group = 16 tanh rows then their 16 sigmoid partners
static inline int paired_row32(int p, int half) {
  const int g = p / 32, r = p % 32;
  return r < 16 ? 16 * g + r : half + 16 * g + (r - 16);
}

static int dec_variant(int C, int K, int D) {
  const int cls = C >= 128 ? 0 : (C == 64 ? 1 : 2);
  static const int tab[3][3][3] = {
      {{V_A_K3D1, V_A_K3D3, V_A_K3D5}, {V_A_K7D1, V_A_K7D3, V_A_K7D5}, {V_A_K11D1, V_A_K11D3, V_A_K11D5}},
      {{V_B_K3D1, V_B_K3D3, V_B_K3D5}, {V_B_K7D1, V_B_K7D3, V_B_K7D5}, {V_B_K11D1, V_B_K11D3, V_B_K11D5}},
      {{V_C_K3D1, V_C_K3D3, V_C_K3D5}, {V_C_K7D1, V_C_K7D3, V_C_K7D5}, {V_C_K11D1, V_C_K11D3, V_C_K11D5}}};
  const int ki = K == 3 ? 0 : (K == 7 ? 1 : 2);
  const int di = D == 1 ? 0 : (D == 3 ? 1 : 2);
  return tab[cls][ki][di];
}

static int validate_hparams(const ovc_hparams* hp) {
  if (hp->inter_channels != 192 || hp->hidden_channels != 192)
    return fail(OVC_ERR_INVALID, "kernels are specialised for inter_channels = hidden_channels = 192 (got %d, %d)",
                hp->inter_channels, hp->hidden_channels);
  if (hp->spec_channels < 1 || hp->spec_channels > 4096) return fail(OVC_ERR_INVALID, "bad spec_channels %d", hp->spec_channels);
  if (hp->gin_channels < 1 || hp->gin_channels > 4096) return fail(OVC_ERR_INVALID, "bad gin_channels %d", hp->gin_channels);
  if (hp->resblock != 1) return fail(OVC_ERR_INVALID, "only resblock \"1\" (ResBlock1) is supported, got %d", hp->resblock);
  if (hp->n_resblock_kernels != 3 || hp->resblock_kernel_sizes[0] != 3 || hp->resblock_kernel_sizes[1] != 7 ||
      hp->resblock_kernel_sizes[2] != 11)
    return fail(OVC_ERR_INVALID, "resblock_kernel_sizes must be [3,7,11]");
  for (int j = 0; j < 3; ++j)
    if (hp->resblock_dilations[j][0] != 1 || hp->resblock_dilations[j][1] != 3 || hp->resblock_dilations[j][2] != 5)
      return fail(OVC_ERR_INVALID, "resblock_dilation_sizes must be [[1,3,5]]*3");
  static const int ur[4] = {8, 8, 2, 2}, uk[4] = {16, 16, 4, 4};
  if (hp->n_upsamples != 4) return fail(OVC_ERR_INVALID, "need 4 upsample stages");
  for (int i = 0; i < 4; ++i)
    if (hp->upsample_rates[i] != ur[i] || hp->upsample_kernel_sizes[i] != uk[i])
      return fail(OVC_ERR_INVALID, "upsample_rates/kernel_sizes must be [8,8,2,2]/[16,16,4,4]");
  if (hp->upsample_initial_channel != 512) return fail(OVC_ERR_INVALID, "upsample_initial_channel must be 512");
  if (hp->hop_length != 256) return fail(OVC_ERR_INVALID, "hop_length must be 256");
  return OVC_OK;
}

static bool key_is_hot(const std::string& k) {
  if (k.rfind("sdp.post_", 0) == 0) return false;   // training-only half of the SDP (models.py:118-125)
  return k.rfind("enc_q.", 0) == 0 || k.rfind("flow.", 0) == 0 || k.rfind("dec.", 0) == 0 || k.rfind("ref_enc.", 0) == 0 ||
         k.rfind("enc_p.", 0) == 0 || k.rfind("dp.", 0) == 0 || k.rfind("sdp.", 0) == 0 || k.rfind("emb_g.", 0) == 0;
}

// tensor-core copy of a conv: fp16 [n_tile][Cin/16][K][column block][hi|lo][TN][8]: hi = fp16(w), lo = fp16((w - hi) * 2^11)
// (ovc_tc.cuh), laid out exactly as the kernel's shared-memory operand slots (one TMA bulk copy per slot)
template <class WF, class BF>
static TcLayer pack_tc(ovc_ctx* c, int Ntot, int Cin, int K, int DIL, WF wfun, BF bfun) {
  TcLayer T;
  T.Cin = Cin; T.Ntot = Ntot; T.K = K; T.DIL = DIL;
  T.TN = Ntot % 128 == 0 ? 128 : (Ntot % 64 == 0 ? 64 : 32);   // widest column tile that divides the row
  // the kernels stage 32 input channels at a time (128-byte rows for the activation TMA); halo tile = 2 * 25 rows at most
  if (Ntot % 32 || Cin % 32 || (K - 1) / 2 * DIL > 25) { T.TN = 0; return T; }
  T.w_off = round_up(c->h_tcw.size(), 64);
  const int slot = 16 * T.TN;   // floats: 2 (hi|lo) x 2 (column blocks) x TN x 8 halfs
  c->h_tcw.resize(T.w_off + (size_t)(Ntot / T.TN) * (Cin / 16) * K * slot, 0.f);
  uint16_t* dst = reinterpret_cast<uint16_t*>(c->h_tcw.data() + T.w_off);
  for (int nt = 0; nt < Ntot / T.TN; ++nt)
    for (int k16 = 0; k16 < Cin / 16; ++k16)
      for (int tap = 0; tap < K; ++tap) {
        uint16_t* sl = dst + (((size_t)nt * (Cin / 16) + k16) * K + tap) * (2 * slot);
        for (int kc = 0; kc < 2; ++kc)
          for (int n = 0; n < T.TN; ++n)
            for (int e = 0; e < 8; ++e) {
              const float w = wfun(nt * T.TN + n, k16 * 16 + kc * 8 + e, tap);
              const __half hi = __float2half_rn(w);
              const __half lo = __float2half_rn((w - __half2float(hi)) * 2048.f);
              sl[((kc * 2 + 0) * T.TN + n) * 8 + e] = __half_as_ushort(hi);   // rows [0, TN) of the 2*TN-row operand
              sl[((kc * 2 + 1) * T.TN + n) * 8 + e] = __half_as_ushort(lo);   // rows [TN, 2*TN)
            }
      }
  T.b_off = round_up(c->h_tcw.size(), 64);
  c->h_tcw.resize(T.b_off + Ntot, 0.f);
  for (int n = 0; n < Ntot; ++n) c->h_tcw[T.b_off + n] = bfun(n);
  return T;
}

// one WN stack (modules.py:160-182), both packed forms: FFMA [C][T] layers and their tensor-core twins
static void pack_wn(ovc_ctx* c, Reader& rd, const std::string& prefix, int n_layers, WNLayers* out) {
  const int H = 192;
  *out = WNLayers();
  for (int i = 0; i < n_layers && rd.ok(); ++i) {
    const std::string pin = prefix + ".in_layers." + std::to_string(i);
    const HostTensor w = rd.weff(pin, {2 * H, H, 5});
    const std::string prs = prefix + ".res_skip_layers." + std::to_string(i);
    const int rows = (i < n_layers - 1) ? 2 * H : H;
    const HostTensor r = rd.weff(prs, {rows, H, -1});
    const HostTensor* rb = rd.get(prs + ".bias", {});
    if (!rd.ok()) return;
    // bias of the in_layer is folded into the per-batch conditioning vector (cond kernel)
    out->in.push_back(pack_conv(
        c, V_WN_IN, 2 * H, H,
        [&](int p, int ci, int k) { return w.data[((size_t)paired_row(p, H) * H + ci) * 5 + k]; },
        [&](int) { return 0.f; }, 0, 5, 2 * H));
    out->rs.push_back(pack_conv(
        c, V_WN_RS, rows, H, [&](int p, int ci, int) { return r.data[(size_t)p * H + ci]; },
        [&](int p) { return rb->data[p]; }, rows, 1, rows));
    out->tc_in.push_back(pack_tc(
        c, 2 * H, H, 5, 1, [&](int p, int ci, int k) { return w.data[((size_t)paired_row32(p, H) * H + ci) * 5 + k]; },
        [&](int) { return 0.f; }));
    out->tc_rs.push_back(pack_tc(
        c, rows, H, 1, 1, [&](int p, int ci, int) { return r.data[(size_t)p * H + ci]; },
        [&](int p) { return rb->data[p]; }));
  }
}

#include "ovc_tts_pack.inc"   // pack_tts(): V1 TTS front-half weights (text encoder, duration predictors, emb_g)

static int finalize(ovc_ctx* c) {
  const ovc_hparams& hp = c->hp;
  const int H = 192, S = hp.spec_channels, G = hp.gin_channels;
  Reader rd{c};
  drop_graphs(c);               // captured launches point at the old weight arenas
  c->h_w.clear();
  c->h_tcw.clear();

  // ---- posterior encoder (models.py:182-221)
  {
    const HostTensor* w = rd.get("enc_q.pre.weight", {H, S, -1});
    const HostTensor* b = rd.get("enc_q.pre.bias", {});
    if (!rd.ok()) return rd.status();
    c->enc_pre = pack_conv(c, V_ENC_PRE, H, S, [&](int p, int ci, int) { return w->data[(size_t)p * S + ci]; },
                           [&](int p) { return b->data[p]; }, H, 1, H);
    c->enc_pre16 = c->enc_pre;            // same packing, 16-byte cp.async when the spectrogram pitch allows it
    c->enc_pre16.variant = V_FLOW_PRE;
    pack_wn(c, rd, "enc_q.enc", 16, &c->enc_wn);
    const HostTensor* pw = rd.get("enc_q.proj.weight", {2 * H, H, -1});
    const HostTensor* pb = rd.get("enc_q.proj.bias", {});
    if (!rd.ok()) return rd.status();
    c->enc_proj = pack_conv(c, V_ENC_PROJ, 2 * H, H,
                            [&](int p, int ci, int) { return pw->data[(size_t)paired_row(p, H) * H + ci]; },
                            [&](int p) { return pb->data[paired_row(p, H)]; }, 2 * H, 1, 2 * H);
  }
  // ---- flow: 4 x (coupling, Flip) (models.py:385-388).  The Flips are absorbed: coupling f sees
  // the channel-reversed tensor iff f is odd, in both directions, so its `pre` reads the physical
  // upper half with reversed columns and its `post` writes the physical lower half with reversed rows.
  for (int f = 0; f < 4; ++f) {
    const std::string p = "flow.flows." + std::to_string(2 * f);
    const bool flipped = f & 1;
    const HostTensor* w = rd.get(p + ".pre.weight", {H, 96, -1});
    const HostTensor* b = rd.get(p + ".pre.bias", {});
    if (!rd.ok()) return rd.status();
    c->flow_pre[f] = pack_conv(
        c, V_FLOW_PRE, H, 96,
        [&](int r, int ci, int) { return w->data[(size_t)r * 96 + (flipped ? 95 - ci : ci)]; },
        [&](int r) { return b->data[r]; }, H, 1, H);
    pack_wn(c, rd, p + ".enc", 4, &c->flow_wn[f]);
    const HostTensor* pw = rd.get(p + ".post.weight", {96, H, -1});   // mean_only couplings only
    const HostTensor* pb = rd.get(p + ".post.bias", {});
    if (!rd.ok()) return rd.status();
    c->flow_post[f] = pack_conv(
        c, V_FLOW_POST, 96, H,
        [&](int r, int ci, int) { return pw->data[(size_t)(flipped ? 95 - r : r) * H + ci]; },
        [&](int r) { return pb->data[flipped ? 95 - r : r]; }, 96, 1, 96);
  }
  // ---- generator (models.py:224-291)
  const HostTensor* cpb = rd.get("dec.conv_pre.bias", {});
  {
    const HostTensor* w = rd.get("dec.conv_pre.weight", {512, H, 7});
    if (!rd.ok()) return rd.status();
    // bias comes per batch item from the cond kernel (conv_pre.bias + cond(g))
    c->dec_pre = pack_conv(c, V_A_K7D1, 512, H, [&](int r, int ci, int k) { return w->data[((size_t)r * H + ci) * 7 + k]; },
                           [&](int) { return 0.f; }, 0, 7, 512);
    c->tc_pre = pack_tc(c, 512, H, 7, 1, [&](int r, int ci, int k) { return w->data[((size_t)r * H + ci) * 7 + k]; },
                        [&](int) { return 0.f; });
  }
  int ch = 512;
  for (int i = 0; i < 4; ++i) {
    const int s = hp.upsample_rates[i], kk = hp.upsample_kernel_sizes[i], pad = (kk - s) / 2;
    const int cin = ch, cout = ch / 2;
    const std::string p = "dec.ups." + std::to_string(i);
    const HostTensor w = rd.weff(p, {cin, cout, kk});   // [cin][cout][kk], weight-norm over dim 0 = cin (SURVEY appendix C.12)
    const HostTensor* b = rd.get(p + ".bias", {});
    if (!rd.ok()) return rd.status();
    const int variant = s == 8 ? V_UPS8_A : (cout * s >= 128 ? V_UPS2_A : V_UPS2_B);
    // polyphase: out[co, s*n+ph] = sum_ci sum_m x[ci, n-m] * W[ci, co, s*m + ph + pad];
    // packed row = co*s + ph, tap 0/1/2 <-> x[n-1], x[n], x[n+1] <-> m = 1, 0, -1
    c->dec_ups[i] = pack_conv(
        c, variant, cout * s, cin,
        [&](int row, int ci, int tap) {
          const int co = row / s, ph = row % s;
          const int kidx = s * (1 - tap) + ph + pad;
          return (kidx >= 0 && kidx < kk) ? w.data[((size_t)ci * cout + co) * kk + kidx] : 0.f;
        },
        [&](int co) { return b->data[co]; }, cout, 2, cout);
    c->dec_ups[i].out_mul = s;
    // tensor-core form: channels-last, row = ph * cout + co, so input step n yields the s output rows s*n .. s*n+s-1
    c->tc_ups[i] = pack_tc(
        c, s * cout, cin, 3, 1,
        [&](int row, int ci, int tap) {
          const int ph = row / cout, co = row % cout;
          const int kidx = s * (1 - tap) + ph + pad;
          return (kidx >= 0 && kidx < kk) ? w.data[((size_t)ci * cout + co) * kk + kidx] : 0.f;
        },
        [&](int row) { return b->data[row % cout]; });
    ch = cout;
    for (int j = 0; j < 3; ++j) {
      const int K = hp.resblock_kernel_sizes[j];
      const int rbi = i * 3 + j;
      for (int d = 0; d < 3; ++d) {
        for (int which = 0; which < 2; ++which) {
          const std::string q = "dec.resblocks." + std::to_string(rbi) + (which ? ".convs2." : ".convs1.") + std::to_string(d);
          const HostTensor rw = rd.weff(q, {ch, ch, K});
          const HostTensor* rbias = rd.get(q + ".bias", {});
          if (!rd.ok()) return rd.status();
          const int dil = which ? 1 : hp.resblock_dilations[j][d];
          ConvLayer L = pack_conv(c, dec_variant(ch, K, dil), ch, ch,
                                  [&](int r, int ci, int k) { return rw.data[((size_t)r * ch + ci) * K + k]; },
                                  [&](int r) { return rbias->data[r]; }, ch, K, ch);
          (which ? c->rb_c2 : c->rb_c1)[rbi][d] = L;
          (which ? c->tc_c2 : c->tc_c1)[rbi][d] =
              pack_tc(c, ch, ch, K, dil, [&](int r, int ci, int k) { return rw.data[((size_t)r * ch + ci) * K + k]; },
                      [&](int r) { return rbias->data[r]; });
        }
      }
    }
  }
  c->post_w_off = rd.put(rd.get("dec.conv_post.weight", {1, 32, 7}));
  if (!rd.ok()) return rd.status();
  // ---- speaker conditioning mat-vec: stack cond_layer of enc_q, of the 4 couplings and dec.cond
  std::vector<int> wrow, sel;
  std::vector<float> cbias;
  {
    std::vector<float> cw;
    auto add_wn = [&](const std::string& prefix, int n_layers, int first_row, int selv, bool add_matrix, bool tc_order) {
      const HostTensor w = rd.weff(prefix + ".cond_layer", {2 * H * n_layers, G, -1});
      const HostTensor* cb = rd.get(prefix + ".cond_layer.bias", {});
      if (!rd.ok()) return;
      if (add_matrix) cw.insert(cw.end(), w.data.begin(), w.data.end());
      for (int l = 0; l < n_layers; ++l) {
        const HostTensor* ib = rd.get(prefix + ".in_layers." + std::to_string(l) + ".bias", {});
        if (!ib) return;
        for (int p = 0; p < 2 * H; ++p) {
          const int o = tc_order ? paired_row32(p, H) : paired_row(p, H);
          wrow.push_back(first_row + l * 2 * H + o);
          sel.push_back(selv);
          cbias.push_back(cb->data[l * 2 * H + o] + ib->data[o]);
        }
      }
    };
    auto flows = [&](int selv, bool add_matrix, bool tc_order) {
      for (int f = 0; f < 4; ++f)
        add_wn("flow.flows." + std::to_string(2 * f) + ".enc", 4, 16 * 2 * H + f * 4 * 2 * H, selv, add_matrix, tc_order);
    };
    c->cond_off_enc = 0;
    add_wn("enc_q.enc", 16, 0, hp.zero_g ? 0 : 1, true, false);
    c->cond_off_fsrc = (int)wrow.size();
    flows(1, true, false);
    c->cond_off_ftgt = (int)wrow.size();
    flows(2, false, false);
    // the same conditioning vectors once more in the tensor-core kernel's column order
    c->cond_off_enc_tc = (int)wrow.size();
    add_wn("enc_q.enc", 16, 0, hp.zero_g ? 0 : 1, false, true);
    c->cond_off_fsrc_tc = (int)wrow.size();
    flows(1, false, true);
    c->cond_off_ftgt_tc = (int)wrow.size();
    flows(2, false, true);
    c->cond_off_dec = (int)wrow.size();
    const HostTensor* dw = rd.get("dec.cond.weight", {512, G, -1});
    const HostTensor* db = rd.get("dec.cond.bias", {});
    if (!rd.ok()) return rd.status();
    const int dec_first = (int)(cw.size() / G);
    cw.insert(cw.end(), dw->data.begin(), dw->data.end());
    for (int r = 0; r < 512; ++r) {
      wrow.push_back(dec_first + r);
      sel.push_back(hp.zero_g ? 0 : 2);
      cbias.push_back(db->data[r] + cpb->data[r]);
    }
    c->cond_rows_out = (int)wrow.size();
    c->cond_w_off = rd.put(cw);
    c->cond_b_off = rd.put(cbias);
  }
  // ---- ReferenceEncoder (optional: only extract_se needs it; models.py:301-338)
  c->has_refenc = false;
  if (find(c, "ref_enc.proj.weight")) {
    static const int filt[7] = {1, 32, 32, 64, 64, 128, 128};
    for (int i = 0; i < 6; ++i) {
      const std::string q = "ref_enc.convs." + std::to_string(i);
      const HostTensor cw = rd.weff(q, {filt[i + 1], filt[i], 3, 3});
      const HostTensor* cb = rd.get(q + ".bias", {});
      if (!rd.ok()) return rd.status();
      c->re_conv_w[i] = rd.put(cw.data);
      c->re_conv_b[i] = rd.put(cb);
    }
    int w6 = S;   // width after the six stride-2 convs (models.py:330-337)
    for (int i = 0; i < 6; ++i) w6 = (w6 - 1) / 2 + 1;
    c->re_gru_in = 128 * w6;
    c->re_wih = rd.put(rd.get("ref_enc.gru.weight_ih_l0", {384, 128 * w6}));
    c->re_whh = rd.put(rd.get("ref_enc.gru.weight_hh_l0", {384, 128}));
    c->re_bih = rd.put(rd.get("ref_enc.gru.bias_ih_l0", {384}));
    c->re_bhh = rd.put(rd.get("ref_enc.gru.bias_hh_l0", {384}));
    c->re_pw = rd.put(rd.get("ref_enc.proj.weight", {G, 128}));
    c->re_pb = rd.put(rd.get("ref_enc.proj.bias", {G}));
    c->re_lng = rd.put(rd.get("ref_enc.layernorm.weight", {S}));
    c->re_lnb = rd.put(rd.get("ref_enc.layernorm.bias", {S}));
    if (!rd.ok()) return rd.status();
    c->has_refenc = true;
  }
  // ---- V1 TTS front half (optional: base-speaker checkpoints only, models.py:451-465)
  c->tts = TtsLayers();
  if (find(c, "enc_p.emb.weight")) TRY(pack_tts(c, rd));
  // ---- upload
  ON_DEVICE(c);
  if (c->d_w) { cudaFree(c->d_w); c->d_w = nullptr; }
  c->w_floats = c->h_w.size();
  CK(cudaMalloc(&c->d_w, c->w_floats * sizeof(float)));
  CK(cudaMemcpy(c->d_w, c->h_w.data(), c->w_floats * sizeof(float), cudaMemcpyHostToDevice));
  if (c->d_tcw) { cudaFree(c->d_tcw); c->d_tcw = nullptr; }
  CK(cudaMalloc(&c->d_tcw, c->h_tcw.size() * sizeof(float)));
  CK(cudaMemcpy(c->d_tcw, c->h_tcw.data(), c->h_tcw.size() * sizeof(float), cudaMemcpyHostToDevice));
  c->h_tcw.clear();
  c->h_tcw.shrink_to_fit();
  CK(cudaFuncSetAttribute(tcconv_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TcwCfg::SMEM_BYTES));
  for (const TcConvKernel& k : kTcConv) CK(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem));
  for (const TcPairKernel& k : kTcPair) CK(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem));
  if (c->d_cond_wrow) cudaFree(c->d_cond_wrow);
  if (c->d_cond_sel) cudaFree(c->d_cond_sel);
  CK(cudaMalloc(&c->d_cond_wrow, wrow.size() * sizeof(int)));
  CK(cudaMalloc(&c->d_cond_sel, sel.size() * sizeof(int)));
  CK(cudaMemcpy(c->d_cond_wrow, wrow.data(), wrow.size() * sizeof(int), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(c->d_cond_sel, sel.data(), sel.size() * sizeof(int), cudaMemcpyHostToDevice));
  if (!c->d_tw) {
    std::vector<float2> tw(STFT_N);
    std::vector<float> win(STFT_N);
    const double PI = 3.14159265358979323846;
    for (int m = 0; m < STFT_N; ++m) {
      tw[m] = make_float2((float)std::cos(2.0 * PI * m / STFT_N), (float)(-std::sin(2.0 * PI * m / STFT_N)));
      win[m] = (float)(0.5 - 0.5 * std::cos(2.0 * PI * m / STFT_N));   // torch.hann_window(periodic=True)
    }
    CK(cudaMalloc(&c->d_tw, STFT_N * sizeof(float2)));
    CK(cudaMalloc(&c->d_win, STFT_N * sizeof(float)));
    CK(cudaMemcpy(c->d_tw, tw.data(), STFT_N * sizeof(float2), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(c->d_win, win.data(), STFT_N * sizeof(float), cudaMemcpyHostToDevice));
  }
  c->h_w.clear();
  c->h_w.shrink_to_fit();
  c->sd.clear();
  for (int v = 0; v < V_COUNT; ++v) CK(kPrepare[v]());
  c->finalized = true;
  return OVC_OK;
}

// ---------------------------------------------------------------------------------------------
// workspace layout
// ---------------------------------------------------------------------------------------------
struct WsLayout {
  int P;   // frame pitch (multiple of 4)
  size_t cond, x, skip, acts, z, dpre, bufA, bufB, bufC, bufD, bufE, bufF, spec, frames, total;
  size_t brB[2], brC[2];   // per-branch ResBlock buffers of the concurrent-branch mode (small calls only)
  bool branches;
};
static WsLayout ws_layout(const ovc_ctx* c, int B, int Tmax) {
  WsLayout L;
  L.P = (int)round_up((size_t)Tmax, 4);
  size_t o = 0;
  auto take = [&](size_t n) { size_t r = o; o = round_up(o + n, 64); return r; };
  L.cond = take((size_t)B * c->cond_rows_out);
  L.x = take((size_t)B * 192 * L.P);
  L.skip = take((size_t)B * 192 * L.P);
  L.acts = take((size_t)B * 192 * L.P);
  L.z = take((size_t)B * 192 * L.P);
  L.dpre = take((size_t)B * 512 * L.P);
  const size_t big = (size_t)B * 8192 * L.P;
  // precision 3: the generator's activations are fp16, two per float of these buffers.  bufA still holds the fp32
  // channels-last z_hat of conv_pre (192 * P floats per utterance) and, earlier in the call, the WN stacks' fp32
  // scratch; both fit in half.
  const size_t gen = c->precision == 3 ? big / 2 : big;
  L.bufA = take(gen);
  L.bufB = take(gen);
  L.bufC = take(gen);
  L.bufD = take(gen);
  L.bufE = c->precision ? take((size_t)B * (c->precision == 3 ? 256 : 512) * L.P) : 0;   // conv_pre output, channels-last
  L.bufF = (c->precision && c->debug) ? take(big) : 0;        // fp32 [C][T] scratch of the debug taps only
  L.branches = c->precision && c->use_branches && (long long)B * Tmax <= c->par_frames;
  for (int j = 0; j < 2; ++j) {
    L.brB[j] = L.branches ? take(gen) : 0;
    L.brC[j] = L.branches ? take(gen) : 0;
  }
  L.spec = take((size_t)B * c->hp.spec_channels * L.P);
  L.frames = take((size_t)2 * B + 4);   // B int64
  L.total = o;
  return L;
}

struct Run {
  ovc_ctx* c;
  cudaStream_t st;
  int B, Tmax, P;
  const long long* lens;
  const long long* glens;   // generator lengths: lens when ragged, NULL (= Tmax) otherwise
};

enum { V_TCH128 = -14, V_TCH64 = -15, V_TCH32 = -16, V_TCPAIR64 = -12, V_TCPAIR32 = -13, V_TC128 = -1, V_TC64 = -2, V_TC32 = -3, V_TRANSPOSE = -4, V_TTS_DENSE = -5, V_TTS_LN = -6, V_TTS_SCORES = -7,
       V_TTS_ATTN = -8, V_TTS_DW = -9, V_TTS_SPLINE = -10, V_TTS_MISC = -11 };
static const char* variant_name(int v) {
  if (v >= 0) return kInfo[v].name;
  switch (v) {
    case V_TCPAIR64: return "PAIR_N64";
    case V_TCPAIR32: return "PAIR_N32";
    case V_TC128: return "TC3_N128";
    case V_TC64: return "TC3_N64";
    case V_TC32: return "TC3_N32";
    case V_TCH128: return "TC1H_N128";
    case V_TCH64: return "TC1H_N64";
    case V_TCH32: return "TC1H_N32";
    case V_TTS_DENSE: return "TTS_DENSE32";
    case V_TTS_LN: return "TTS_LAYERNORM";
    case V_TTS_SCORES: return "TTS_SCORES";
    case V_TTS_ATTN: return "TTS_ATTN_OUT";
    case V_TTS_DW: return "TTS_DWCONV";
    case V_TTS_SPLINE: return "TTS_SPLINE";
    case V_TTS_MISC: return "TTS_MISC";
    default: return "TRANSPOSE";
  }
}

// Every counted kernel launch: `enqueue` puts one kernel on r.st (a <<<>>> launch, or a call that returns its
// cudaError_t).  With profiling on and a record given, two events bracket the launch and the record is kept.
template <class F>
static int launch_kernel(Run& r, const std::optional<ProfRec>& rec, F enqueue) {
  ovc_ctx* c = r.c;
  const bool prof = c->prof && rec;
  const size_t e = 2 * c->prof_log.size();
  if (prof) {
    if (e + 2 > c->ev.size()) {
      const size_t old = c->ev.size();
      c->ev.resize(old + 512);
      for (size_t i = old; i < c->ev.size(); ++i) CK(cudaEventCreate(&c->ev[i]));
    }
    CK(cudaEventRecord(c->ev[e], r.st));
  }
  if constexpr (std::is_void<decltype(enqueue())>::value) enqueue();
  else CK(enqueue());
  CK(cudaGetLastError());
  c->launches++;
  if (prof) {
    CK(cudaEventRecord(c->ev[e + 1], r.st));
    c->prof_log.push_back(*rec);
  }
  return OVC_OK;
}

// ConvArgs of one FFMA conv: x [B][x_C][x_pitch] -> y [B][y_C][y_pitch] over the frame limits `lens` (time axis in
// units of `mul` samples), leaky-relu `slope` on the input; the layer's own bias unless the caller sets one
static ConvArgs conv_args(const float* x, int x_C, int x_pitch, float* y, int y_C, int y_pitch, const long long* lens, int mul,
                          float slope) {
  ConvArgs a{};
  a.x = x; a.x_bs = (long long)x_C * x_pitch; a.x_pitch = x_pitch;
  a.y = y; a.y_bs = (long long)y_C * y_pitch; a.y_pitch = y_pitch;
  a.lens_in = lens; a.lens_out = lens; a.mul_in = mul; a.mul_out = mul;
  a.slope = slope; a.scale = 1.f;
  return a;
}

static int launch(Run& r, const ConvLayer& L, ConvArgs a, int t_len, bool mrf = false) {
  a.w = r.c->d_w + L.w_off;
  if (!a.bias) a.bias = r.c->d_w + L.b_off;
  a.n_chunks = L.n_chunks;
  a.cin = L.cin;
  a.tmax = r.Tmax;
  // algorithmic work of this launch over all B * t_len positions (upper bound for ragged batches)
  const double units = (double)r.B * t_len;
  const ProfRec rec{L.variant, mrf ? 1 : 0, 2.0 * L.cout * L.cin * L.K * units * L.out_mul,
                    4.0 * units * ((double)L.cin + (double)L.cout * L.out_mul)};
  return launch_kernel(r, rec, [&] { return kLaunch[L.variant](a, t_len, L.row_tiles, r.B, r.st); });
}

static int tap(Run& r, const char* name, const float* src, int C, int T, int pitch) {
  ovc_ctx* c = r.c;
  if (!c->debug) return OVC_OK;
  DebugBuf& d = c->taps[name];
  const size_t n = (size_t)r.B * C * pitch;
  if (d.floats < n) {
    if (d.d) cudaFree(d.d);
    CK(cudaMalloc(&d.d, n * sizeof(float)));
    d.floats = n;
  }
  d.shape[0] = r.B; d.shape[1] = C; d.shape[2] = T; d.shape[3] = pitch;
  CK(cudaMemcpyAsync(d.d, src, n * sizeof(float), cudaMemcpyDeviceToDevice, r.st));
  return OVC_OK;
}

// how one conv runs on the tensor cores; a call sets only what differs from these defaults
struct TcOpt {
  float slope = 1.f;              // leaky_relu slope on the input (1 = identity)
  float scale = 1.f;              // epilogue multiplier (1/3 for the last MRF accumulation)
  int accumulate = 0;             // y += result
  int family = 0;                 // profile family: 1 MRF conv, 2 polyphase transposed conv, 0 other
  int epi = 0;                    // 0 linear, 1 WN gate, 2 WN res/skip
  const float* bias = nullptr;    // override (per-utterance conditioning vector), with stride
  long long bias_bs = 0;
  float* s = nullptr;             // skip accumulator (EPI 2)
  int split = 0, first = 0;
  int y_ld = 0;                   // output row width when it differs from Ntot
  bool use_lens_frames = false;   // limits are the frame lengths (enc/flow) instead of the generator lengths
  const long long* lens_x = nullptr; bool has_lens_x = false;   // the input's own limit (TcConvArgs.lens_x)
  int grid_div = 1;               // persistent kernel: use 1 / grid_div of the SMs (concurrent ResBlock branches)
  bool in16 = false, out16 = false;   // fp16 input / output activations (precision 3, generator only): one fp16 pass
};
// kernel launch with (optionally) the programmatic-stream-serialization attribute: the kernel may begin while its
// predecessor in the stream drains; it calls griddepcontrol.wait before it touches dependent data (ovc_tcconv.cuh)
template <class... KArgs, class... Args>
static cudaError_t launch_ex(void (*kernel)(KArgs...), dim3 grid, int block, size_t smem, cudaStream_t st, bool pdl, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = dim3((unsigned)block, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// activation chunks by tensor-map TMA: the channels-last input as a [B][P * mul][C] tensor, one box = box_rows x 32
// channels; rows outside the tensor are zero-filled by the copy engine.  fp32: 128-byte rows, 128-byte swizzle (the
// converter reads them row-strided).  fp16 (f16 = true): 64-byte rows, no swizzle (the converter reads them whole,
// tc_convert_raw16).
static CUresult encode_act_map(CUtensorMap* tmap, const Run& r, const float* x, int C, int mul, int box_rows, bool f16 = false) {
  memset(tmap, 0, sizeof *tmap);
  const cuuint64_t es = f16 ? 2 : 4;
  const cuuint64_t gdim[3] = {(cuuint64_t)C, (cuuint64_t)r.P * mul, (cuuint64_t)r.B};
  const cuuint64_t gstr[2] = {(cuuint64_t)C * es, (cuuint64_t)((long long)C * r.P * mul) * es};
  const cuuint32_t box[3] = {32, (cuuint32_t)box_rows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  return encode_tiled_fn()(tmap, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(x), gdim,
                           gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, f16 ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

// one conv on the tensor cores (3xFP16 split precision / single-pass fp16), channels-last in/out.  t_len / mul are in INPUT steps.
static int launch_tc(Run& r, const TcLayer& T, const float* x, float* y, const float* res, int t_len, int mul,
                     const TcOpt& o = TcOpt()) {
  TcConvArgs a{};
  const int y_ld = o.y_ld ? o.y_ld : T.Ntot;
  a.x = x; a.x_bs = (long long)T.Cin * r.P * mul;
  a.w = reinterpret_cast<const uint16_t*>(r.c->d_tcw + T.w_off);
  a.bias = o.bias ? o.bias : r.c->d_tcw + T.b_off; a.bias_bs = o.bias_bs;
  a.y = y; a.y_bs = (long long)y_ld * r.P * mul; a.y_ld = y_ld;
  a.r = res;
  a.s = o.s; a.s_bs = a.y_bs;
  a.epi = o.epi; a.split = o.split; a.first = o.first;
  a.lens = o.use_lens_frames ? r.lens : r.glens; a.tmax = r.Tmax; a.mul = mul;
  a.lens_x = o.lens_x; a.has_lens_x = o.has_lens_x ? 1 : 0;
  a.Cin = T.Cin; a.Ntot = T.Ntot; a.K = T.K; a.DIL = T.DIL;
  a.slope = o.slope; a.scale = o.scale; a.accumulate = o.accumulate;
  const bool f16s = o.in16 || o.out16;   // fp16 storage: one pass, the persistent kernel, the linear epilogue
  a.passes = (r.c->precision == 2 || f16s) ? 1 : 3;
  if (T.TN == 0) return fail(OVC_ERR_INVALID, "conv %d -> %d (k %d, dilation %d) does not fit the tensor-core kernels", T.Cin, T.Ntot, T.K, T.DIL);
  if (!(o.slope >= 0.f && o.slope <= 1.f)) return fail(OVC_ERR_INVALID, "leaky_relu slope %g outside [0, 1]", (double)o.slope);
  // the fp16-storage instantiations have the linear epilogue only
  const TcConvKernel* kern = find_tcconv(T.TN, o.in16, o.out16);
  if (!kern || (f16s && o.epi != 0))
    return fail(OVC_ERR_INVALID, "no tensor-core kernel for conv %d -> %d (fp16 in %d, fp16 out %d, epilogue %d)", T.Cin, T.Ntot,
                (int)o.in16, (int)o.out16, o.epi);
  const double units = (double)r.B * t_len;
  const int eff_k = o.family == 2 ? 2 : T.K;   // polyphase transposed conv: 2 of the 3 packed taps are non-zero per row
  const double in_b = o.in16 ? 2.0 : 4.0, out_b = o.out16 ? 2.0 : 4.0;   // bytes per element
  const int var = f16s ? (T.TN == 128 ? V_TCH128 : T.TN == 64 ? V_TCH64 : V_TCH32) : (T.TN == 128 ? V_TC128 : T.TN == 64 ? V_TC64 : V_TC32);
  const ProfRec rec{var, o.family == 1 ? 1 : 0, 2.0 * T.Cin * T.Ntot * eff_k * units,
                    (in_b * T.Cin + out_b * T.Ntot * (1 + (res ? 1 : 0) + (o.accumulate ? 1 : 0))) * units, (T.Cin << 16) | (T.K << 8) | T.DIL};
  const bool pdl = r.c->use_pdl == 1 || (r.c->use_pdl == 2 && o.epi != 0);
  // 3 (default): the generator's first stage (k >= 7 at C = 256: few, long tiles) on the two-CTAs-per-SM kernel, whose
  // second CTA fills the tensor pipe while the first waits on a barrier; everything else on the persistent kernel.
  // fp16 storage always runs on the persistent kernel (the wide kernel is fp32-only).
  int wv = r.c->wide_variant;
  if (wv == 3) wv = (T.K >= 7 && T.Cin >= 256) ? 2 : 0;
  if (T.TN == 128 && wv == 2 && !f16s) {
    // 128-step tiles, two CTAs per SM
    dim3 grid((t_len + 127) / 128, T.Ntot / 128, r.B);
    return launch_kernel(r, rec, [&] { return launch_ex(tcconv_wide_kernel, grid, TcwCfg::THREADS, TcwCfg::SMEM_BYTES, r.st, pdl, a); });
  }
  // persistent: one CTA per SM walks the (utterance, tile) list; column tiles (if any) on grid.y
  const int MT = T.TN == 128 ? TcnCfg<128>::MT : TcnCfg<64>::MT;
  const int steps = MT * 128;
  const int n_tt = (t_len + steps - 1) / steps, total = n_tt * r.B;
  if (!encode_tiled_fn()) return fail(OVC_ERR_CUDA, "cuTensorMapEncodeTiled is not available");
  const int rows = tcn_rows(MT, (T.K - 1) / 2 * T.DIL);
  a.n_box = rows > 256 ? 2 : 1;
  a.box_rows = rows / a.n_box;
  CUtensorMap tmap;
  const CUresult cr = encode_act_map(&tmap, r, x, T.Cin, mul, a.box_rows, o.in16);
  if (cr != CUDA_SUCCESS) return fail(OVC_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for a [%d][%d][%d] activation tensor", (int)cr,
                                      r.B, r.P * mul, T.Cin);
  const int ncol = T.Ntot / T.TN;
  const int per_col = std::max(1, r.c->sm_count / ncol / std::max(1, o.grid_div));
  dim3 pg((unsigned)std::min(total, per_col), ncol, 1);
  return launch_kernel(r, rec, [&] { return launch_ex(kern->fn, pg, TCN_THREADS, kern->smem, r.st, pdl, a, n_tt, total, tmap); });
}

// one ResBlock conv pair (c1 dilated, c2 dilation 1, residual = the pair's input) as ONE kernel: C = 64 / 32 stages
// Only where BOTH convs' weights stay resident in shared memory next to the operand tiles, and only the HBM-bound pairs:
// C = 32 and C = 64 at k <= 5 / k = 3.  Measured (C = 32, per pair, 32 x 10 s): k = 3 -25 %, k = 7 equal, k = 11 +8 % (those are
// bound by shared-memory operand reads, not HBM, and pay for the 118 / 128 tile efficiency).
static bool pair_fits(const TcLayer& T1, const TcLayer& T2) {
  if (!(T1.TN == 32 || T1.TN == 64)) return false;
  const int ring = T1.TN == 32 ? TcpCfg<32>::RING : TcpCfg<64>::RING, hmax = T1.TN == 32 ? TcpCfg<32>::HMAX : TcpCfg<64>::HMAX;
  return T1.Ntot == T1.TN && T1.Cin == T1.TN && T2.Ntot == T1.TN && T2.Cin == T1.TN && T2.TN == T1.TN && T2.K == T1.K &&
         T2.DIL == 1 && (T1.K - 1) / 2 * T1.DIL <= hmax && 2 * (T1.Cin / 16) * T1.K <= ring && T1.K <= 5;
}
// slope, scale and accumulate of `o` apply (family: always MRF)
static int launch_pair(Run& r, const TcLayer& T1, const TcLayer& T2, const float* x, float* y, int t_len, int mul, const TcOpt& o) {
  TcPairArgs a{};
  const int C = T1.TN;
  const TcPairKernel* kern = find_tcpair(C);
  if (!kern) return fail(OVC_ERR_INVALID, "no conv-pair kernel for C = %d", C);
  a.x = x; a.x_bs = (long long)C * r.P * mul;
  a.w1 = reinterpret_cast<const uint16_t*>(r.c->d_tcw + T1.w_off);
  a.w2 = reinterpret_cast<const uint16_t*>(r.c->d_tcw + T2.w_off);
  a.bias1 = r.c->d_tcw + T1.b_off; a.bias2 = r.c->d_tcw + T2.b_off;
  a.y = y; a.y_bs = a.x_bs;
  a.lens = r.glens; a.tmax = r.Tmax; a.mul = mul;
  a.C = C; a.K = T1.K; a.DIL1 = T1.DIL;
  a.slope = o.slope; a.scale = o.scale; a.accumulate = o.accumulate;
  a.passes = r.c->precision == 2 ? 1 : 3;
  if (!encode_tiled_fn()) return fail(OVC_ERR_CUDA, "cuTensorMapEncodeTiled is not available");
  const int H1 = (T1.K - 1) / 2 * T1.DIL, H2 = (T1.K - 1) / 2;
  const int R = 128 - 2 * H2, rows8 = (128 + 2 * H1 + 7) & ~7;
  const int n_tt = (t_len + R - 1) / R, total = n_tt * r.B;
  CUtensorMap tmap;
  const CUresult cr = encode_act_map(&tmap, r, x, C, mul, rows8);
  if (cr != CUDA_SUCCESS) return fail(OVC_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for a conv pair", (int)cr);
  const double units = (double)r.B * t_len;
  const ProfRec rec{C == 64 ? V_TCPAIR64 : V_TCPAIR32, 1, 2.0 * 2.0 * C * C * T1.K * units,
                    4.0 * C * (2 + (o.accumulate ? 1 : 0)) * units, (C << 16) | (T1.K << 8) | T1.DIL};
  dim3 pg((unsigned)std::min(total, r.c->sm_count), 1, 1);
  return launch_kernel(r, rec, [&] { return launch_ex(kern->fn, pg, TCN_THREADS, kern->smem, r.st, false, a, n_tt, total, tmap); });
}

// src16: the source is fp16 (read through the same pointer type as the fp32 workspace buffers), dst is always fp32
static int launch_transpose(Run& r, const float* src, float* dst, int rows, int cols, bool src16 = false) {
  dim3 grid((cols + 31) / 32, (rows + 31) / 32, r.B);
  return launch_kernel(r, ProfRec{V_TRANSPOSE, 0, 0.0, (src16 ? 6.0 : 8.0) * rows * cols * r.B}, [&] {
    if (src16)
      transpose_kernel<<<grid, 256, 0, r.st>>>(reinterpret_cast<const __half*>(src), dst, rows, cols, (long long)rows * cols);
    else
      transpose_kernel<<<grid, 256, 0, r.st>>>(src, dst, rows, cols, (long long)rows * cols);
  });
}

// every speaker-conditioning 1x1 conv of a call in one launch (rows of the cond section of the workspace)
static int launch_cond(Run& r, const float* g_src, const float* g_tgt, float* out) {
  ovc_ctx* c = r.c;
  CondArgs a;
  a.w = c->d_w + c->cond_w_off; a.bias = c->d_w + c->cond_b_off;
  a.w_row = c->d_cond_wrow; a.sel = c->d_cond_sel;
  a.g_src = g_src; a.g_tgt = g_tgt; a.out = out;
  a.rows_out = c->cond_rows_out; a.gin = c->hp.gin_channels;
  dim3 grid((c->cond_rows_out + 7) / 8, r.B);
  return launch_kernel(r, std::nullopt, [&] { cond_kernel<<<grid, 256, 0, r.st>>>(a); });
}

// one WN stack (modules.py:185-210): x <- in place, skip <- output
static int run_wn(Run& r, const WNLayers& wn, float* x, float* skip, float* acts, const float* cond, int cond_bs) {
  const int P = r.P, T = r.Tmax;
  const int n = (int)wn.in.size();
  for (int i = 0; i < n; ++i) {
    ConvArgs a = conv_args(x, 192, P, acts, 192, P, r.lens, 1, 1.f);
    a.bias = cond + (size_t)i * 384; a.bias_bs = cond_bs;
    TRY(launch(r, wn.in[i], a, T));
    ConvArgs b = conv_args(acts, 192, P, x, 192, P, r.lens, 1, 1.f);
    b.s = skip; b.s_bs = 192LL * P; b.s_pitch = P;
    b.split = (i < n - 1) ? 192 : 0;
    b.flags = (i == 0) ? F_FIRST : 0;
    TRY(launch(r, wn.rs[i], b, T));
  }
  return OVC_OK;
}

// the same stack on the tensor cores: x, acts, skip live channels-last inside the stack; h comes in and the
// output leaves in the [C][T] layout of the small FFMA kernels around it (pre / proj / post)
static int run_wn_tc(Run& r, const WNLayers& wn, float* x, float* skip, float* acts, float* x_cl, float* skip_cl,
                     const float* cond_tc, int cond_bs) {
  const int P = r.P, T = r.Tmax;
  const int n = (int)wn.tc_in.size();
  TRY(launch_transpose(r, x, x_cl, 192, P));
  for (int i = 0; i < n; ++i) {
    TcOpt g;
    g.epi = 1; g.bias = cond_tc + (size_t)i * 384; g.bias_bs = cond_bs; g.y_ld = 192; g.use_lens_frames = true;
    TRY(launch_tc(r, wn.tc_in[i], x_cl, acts, nullptr, T, 1, g));
    TcOpt q;
    q.epi = 2; q.s = skip_cl; q.split = (i < n - 1) ? 192 : 0; q.first = (i == 0); q.y_ld = 192; q.use_lens_frames = true;
    TRY(launch_tc(r, wn.tc_rs[i], acts, x_cl, nullptr, T, 1, q));
  }
  TRY(launch_transpose(r, skip_cl, skip, P, 192));
  return OVC_OK;
}

static int run_flow(Run& r, const WsLayout& W, float* ws, bool reverse, const float* cond_all) {
  ovc_ctx* c = r.c;
  const int P = r.P, T = r.Tmax;
  float* z = ws + W.z;
  float* x = ws + W.x;
  float* skip = ws + W.skip;
  float* acts = ws + W.acts;
  const int sect = reverse ? c->cond_off_ftgt : c->cond_off_fsrc;
  for (int step = 0; step < 4; ++step) {
    const int f = reverse ? 3 - step : step;
    const bool flipped = f & 1;
    // pre: x0 (physical lower half, or upper half when flipped) -> h     (modules.py:438-439)
    TRY(launch(r, c->flow_pre[f], conv_args(z + (flipped ? 96 * (size_t)P : 0), 192, P, x, 192, P, r.lens, 1, 1.f), T));
    if (c->precision >= 1) {
      const int sect_tc = reverse ? c->cond_off_ftgt_tc : c->cond_off_fsrc_tc;
      TRY(run_wn_tc(r, c->flow_wn[f], x, skip, acts, ws + W.bufA, ws + W.bufB, cond_all + sect_tc + f * 4 * 384, c->cond_rows_out));
    } else {
      TRY(run_wn(r, c->flow_wn[f], x, skip, acts, cond_all + sect + f * 4 * 384, c->cond_rows_out));
    }
    // post + coupling update of x1 in place                                (modules.py:441-454)
    ConvArgs b = conv_args(skip, 192, P, z + (flipped ? 0 : 96 * (size_t)P), 192, P, r.lens, 1, 1.f);
    b.sign = reverse ? -1.f : 1.f;
    TRY(launch(r, c->flow_post[f], b, T));
  }
  return OVC_OK;
}

static void drop_graphs(ovc_ctx* c) {
  for (auto& g : c->graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  c->graphs.clear();
}

__global__ void set_call_params_kernel(CallParams* p, unsigned long long seed, float tau) {
  p->seed = seed;
  p->tau = tau;
}

// Run `body(stream)` -- a pure launch sequence -- directly, or replay it from a CUDA graph when the same signature `key`
// has been seen before (captured on the second sighting: a one-off call never pays for an instantiation).  Capture
// happens on an internal stream (the caller's may be the legacy default stream, which cannot be captured); the graph is
// launched into the caller's stream.
template <class Body>
static int run_graphed(ovc_ctx* c, const std::vector<uintptr_t>& key, cudaStream_t st, Body body) {
  if (!c->use_graph || c->prof || c->debug) return body(st);
  ovc_ctx::GraphEntry* e = nullptr;
  for (auto& g : c->graphs)
    if (g.key == key) { e = &g; break; }
  if (!e) {
    if (c->graphs.size() >= 16) {   // evict the least recently used signature
      size_t lru = 0;
      for (size_t i = 1; i < c->graphs.size(); ++i)
        if (c->graphs[i].stamp < c->graphs[lru].stamp) lru = i;
      if (c->graphs[lru].exec) cudaGraphExecDestroy(c->graphs[lru].exec);
      c->graphs.erase(c->graphs.begin() + lru);
    }
    c->graphs.emplace_back();
    e = &c->graphs.back();
    e->key = key;
  }
  e->stamp = ++c->graph_clock;
  e->seen++;
  if (e->exec) {
    CK(cudaGraphLaunch(e->exec, st));
    c->launches = e->launches;
    c->graph_replays++;
    return OVC_OK;
  }
  if (e->seen < 2) return body(st);
  if (!c->cap_stream) CK(cudaStreamCreateWithFlags(&c->cap_stream, cudaStreamNonBlocking));
  CK(cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeThreadLocal));
  const int rc = body(c->cap_stream);
  cudaGraph_t graph = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(c->cap_stream, &graph);
  if (rc != OVC_OK || ce != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    e->seen = -1000000;           // never try this signature again
    if (rc != OVC_OK) return rc;
    return body(st);
  }
  const cudaError_t ie = cudaGraphInstantiate(&e->exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ie != cudaSuccess) {
    cudaGetLastError();
    e->exec = nullptr;
    e->seen = -1000000;
    return body(st);
  }
  e->launches = c->launches;
  CK(cudaGraphLaunch(e->exec, st));
  c->graph_replays++;
  return OVC_OK;
}

static int set_call_params(ovc_ctx* c, uint64_t seed, float tau, cudaStream_t st) {
  if (!c->d_callp) CK(cudaMalloc(&c->d_callp, sizeof(CallParams)));
  set_call_params_kernel<<<1, 1, 0, st>>>(c->d_callp, seed, tau);
  CK(cudaGetLastError());
  return OVC_OK;
}
static uintptr_t option_bits(const ovc_ctx* c) {
  return (uintptr_t)c->precision | ((uintptr_t)c->wide_variant << 4) | ((uintptr_t)c->use_branches << 14) | ((uintptr_t)c->use_pdl << 15) |
         ((uintptr_t)c->use_pair << 17);
}

// Grow a device arena to `need` floats.  Work queued on `st` may still use the old one, so the stream drains first.  A
// failed allocation leaves the arena empty and no CUDA error pending, and returns OVC_ERR_NOMEM.
static int grow_arena(float*& d, size_t& floats, size_t need, cudaStream_t st, const char* what) {
  if (need <= floats) return OVC_OK;
  CK(cudaStreamSynchronize(st));
  if (d) CK(cudaFree(d));
  d = nullptr;
  floats = 0;
  const cudaError_t e = cudaMalloc(&d, need * sizeof(float));
  if (e != cudaSuccess) {
    d = nullptr;
    cudaGetLastError();
    return fail(OVC_ERR_NOMEM, "%s of %.2f GB does not fit: %s", what, need * 4e-9, cudaGetErrorString(e));
  }
  floats = need;
  return OVC_OK;
}

static int ensure_ws(ovc_ctx* c, const WsLayout& W, cudaStream_t st) {
  if (W.total > c->ws_floats) drop_graphs(c);   // captured launches point into the old workspace
  return grow_arena(c->d_ws, c->ws_floats, W.total, st, "workspace");
}

// z (workspace, [B][192][P]) -> a caller tensor [B][192][Tmax], zero past each length
static int copy_latent_out(Run& r, const WsLayout& W, float* ws, float* dst) {
  if (!dst) return OVC_OK;
  dim3 grid((r.Tmax + 255) / 256, 192, r.B);
  return launch_kernel(r, std::nullopt, [&] { copy_latent_kernel<<<grid, 256, 0, r.st>>>(ws + W.z, W.P, dst, r.Tmax, 192, r.lens); });
}

// the MRF of upsampling stage i on the tensor cores (models.py:280-286): xs = sum_j ResBlock1_j(bufA) / 3 -> bufD.
// `par`: a latency-bound call runs the three ResBlock branches side by side -- branch 0 on the caller's stream, 1 and 2
// on side streams with their own B / C buffers, every kernel on a third of the SMs.  The MRF sum keeps its order (the
// last conv of branch j waits for that of branch j - 1), so the result is bit-identical to the sequential schedule.
static int run_mrf_tc(Run& r, const WsLayout& W, float* ws, int i, int Tlen, int up_out, bool par) {
  ovc_ctx* c = r.c;
  float* bufA = ws + W.bufA; float* bufD = ws + W.bufD;
  if (par) CK(cudaEventRecord(c->br_ev[3], r.st));
  for (int j = 0; j < 3; ++j) {
    const TcLayer* c1 = c->tc_c1[i * 3 + j];
    const TcLayer* c2 = c->tc_c2[i * 3 + j];
    Run rj = r;
    float* Bj = ws + W.bufB; float* Cj = ws + W.bufC;
    TcOpt o;
    o.slope = 0.1f; o.family = 1;
    o.in16 = o.out16 = c->precision == 3;
    if (par) {
      o.grid_div = 3;
      if (j > 0) {
        rj.st = c->br_stream[j - 1];
        CK(cudaStreamWaitEvent(rj.st, c->br_ev[3], 0));
        Bj = ws + W.brB[j - 1]; Cj = ws + W.brC[j - 1];
      }
    }
    bool fused = !par && c->use_pair && c->precision != 3;   // the pair kernel is fp32-only
    for (int d = 0; d < 3; ++d) fused = fused && pair_fits(c1[d], c2[d]);
    for (int d = 0; d < 3; ++d) {
      TcOpt o2 = o;
      o2.scale = (d == 2 && j == 2) ? 1.0f / 3.0f : 1.f;   // xs / num_kernels (models.py:286), as a multiply
      o2.accumulate = (d == 2 && j > 0) ? 1 : 0;
      if (fused) {
        // one kernel per conv pair; a pair never runs in place (its tiles read x with a halo), so the running
        // activation ping-pongs bufA -> bufB -> bufC -> bufD (bufC is free: the intermediate stays on chip)
        const float* xs[3] = {bufA, Bj, Cj};
        float* ys[3] = {Bj, Cj, bufD};
        TRY(launch_pair(rj, c1[d], c2[d], xs[d], ys[d], Tlen, up_out, o2));
        continue;
      }
      const float* xin = d == 0 ? bufA : Bj;
      TRY(launch_tc(rj, c1[d], xin, Cj, nullptr, Tlen, up_out, o));
      if (par && d == 2 && j > 0) CK(cudaStreamWaitEvent(rj.st, c->br_ev[j - 1], 0));   // xs so far is complete
      TRY(launch_tc(rj, c2[d], Cj, d < 2 ? Bj : bufD, xin, Tlen, up_out, o2));
    }
    if (par) CK(cudaEventRecord(c->br_ev[j], rj.st));
  }
  if (par) CK(cudaStreamWaitEvent(r.st, c->br_ev[2], 0));   // join (branch 1 is joined through branch 2's wait)
  return OVC_OK;
}

// HiFi-GAN generator on the latent in ws.z (models.py:272-291): shared by voice_conversion and the TTS decode
static int run_dec(Run& r, const WsLayout& W, float* ws, const float* cond, const long long* lens, float* o_hat) {
  ovc_ctx* c = r.c;
  const int B = r.B, Tmax = r.Tmax, P = W.P;
  // ---- generator (models.py:272-291).  Lengths: frames * cumulative upsampling.
  float* bufA = ws + W.bufA; float* bufB = ws + W.bufB; float* bufC = ws + W.bufC; float* bufD = ws + W.bufD;
  if (c->precision >= 1) {
    // ---- tensor-core generator: channels-last [t][C] from conv_pre's output to conv_post's input.
    // ConvTranspose1d = polyphase conv Cin -> s*Cout whose row n IS output rows s*n .. s*n+s-1 of the
    // channels-last result; ResBlock convs = tcconv with fused lrelu / bias / residual / MRF average.
    const bool f16s = c->precision == 3;   // fp16 activations from conv_pre's output to conv_post's input
    float* bufE = ws + W.bufE;
    float* bufF = ws + W.bufF;   // fp32 [C][T] scratch for debug taps
    auto tap_cl = [&](const char* nm, const float* cl, int C, int T_, int pitch) -> int {
      if (!c->debug) return OVC_OK;
      TRY(launch_transpose(r, cl, bufF, pitch, C, f16s));
      return tap(r, nm, bufF, C, T_, pitch);
    };
    // conv_pre (192 -> 512, k 7) + cond(g) on the tensor cores too: z channels-last through bufA, result straight into
    // bufE; the input is cut at the frame lengths (z_hat * y_mask), the output runs over the generator's own limit
    TRY(launch_transpose(r, ws + W.z, bufA, 192, P));
    TcOpt e;
    e.bias = cond + c->cond_off_dec; e.bias_bs = c->cond_rows_out;
    e.lens_x = lens; e.has_lens_x = lens != nullptr;
    e.out16 = f16s;
    TRY(launch_tc(r, c->tc_pre, bufA, bufE, nullptr, Tmax, 1, e));
    TRY(tap_cl("dec.pre", bufE, 512, Tmax, P));
    const float* stage_in = bufE;
    int cin = 512, up = 1;
    const bool par = W.branches && !c->prof && !c->debug;
    if (par && !c->br_stream[0]) {
      for (int j = 0; j < 2; ++j) CK(cudaStreamCreateWithFlags(&c->br_stream[j], cudaStreamNonBlocking));
      for (int j = 0; j < 4; ++j) CK(cudaEventCreateWithFlags(&c->br_ev[j], cudaEventDisableTiming));
    }
    for (int i = 0; i < 4; ++i) {
      const int s = c->hp.upsample_rates[i];
      const int cout = cin / 2, up_out = up * s;
      const int Tlen = Tmax * up_out, pitch_out = P * up_out;
      char nm[32];
      TcOpt u;
      u.slope = 0.1f; u.family = 2;
      u.in16 = u.out16 = f16s;
      TRY(launch_tc(r, c->tc_ups[i], stage_in, bufA, nullptr, Tmax * up, up, u));
      snprintf(nm, sizeof nm, "dec.ups%d", i);
      TRY(tap_cl(nm, bufA, cout, Tlen, pitch_out));
      TRY(run_mrf_tc(r, W, ws, i, Tlen, up_out, par));
      snprintf(nm, sizeof nm, "dec.stage%d", i);
      TRY(tap_cl(nm, bufD, cout, Tlen, pitch_out));
      stage_in = bufD;   // the next upsampling consumes xs before that stage's MRF rewrites bufD (stream order)
      cin = cout; up = up_out;
    }
    const int y_len = Tmax * up;
    dim3 grid((y_len + 255) / 256, B);
    return launch_kernel(r, std::nullopt, [&] {
      if (f16s)
        conv_post_cl_kernel<32, __half><<<grid, 256, 0, r.st>>>(reinterpret_cast<const __half*>(stage_in), 32LL * P * up, c->d_w + c->post_w_off,
                                                        o_hat, (long long)y_len, y_len, r.glens, Tmax, up);
      else
        conv_post_cl_kernel<32><<<grid, 256, 0, r.st>>>(stage_in, 32LL * P * up, c->d_w + c->post_w_off, o_hat, (long long)y_len,
                                                        y_len, r.glens, Tmax, up);
    });
  }
  // ---- fp32 generator: [C][T] activations, every conv on the FFMA kernels
  ConvArgs a = conv_args(ws + W.z, 192, P, ws + W.dpre, 512, P, r.glens, 1, 1.f);
  a.bias = cond + c->cond_off_dec; a.bias_bs = c->cond_rows_out;
  a.lens_in = lens;          // z_hat * y_mask
  TRY(launch(r, c->dec_pre, a, Tmax));
  TRY(tap(r, "dec.pre", ws + W.dpre, 512, Tmax, P));
  const float* stage_in = ws + W.dpre;
  int cin = 512, up = 1;
  for (int i = 0; i < 4; ++i) {
    const int s = c->hp.upsample_rates[i];
    const int cout = cin / 2;
    const int up_out = up * s;
    const int pitch_in = P * up, pitch_out = P * up_out;
    // leaky_relu(0.1) + ConvTranspose1d (models.py:278-279), polyphase; kernel time axis = input samples
    TRY(launch(r, c->dec_ups[i], conv_args(stage_in, cin, pitch_in, bufA, cout, pitch_out, r.glens, up, 0.1f), Tmax * up));
    char nm[32]; snprintf(nm, sizeof nm, "dec.ups%d", i);
    TRY(tap(r, nm, bufA, cout, Tmax * up_out, pitch_out));
    // MRF: xs = sum_j ResBlock1_j(x) / 3 (models.py:280-286; ResBlock1 = modules.py:296-309)
    const int Tlen = Tmax * up_out;
    for (int j = 0; j < 3; ++j) {
      for (int d = 0; d < 3; ++d) {
        const float* xin = d == 0 ? bufA : bufB;
        TRY(launch(r, c->rb_c1[i * 3 + j][d], conv_args(xin, cout, pitch_out, bufC, cout, pitch_out, r.glens, up_out, 0.1f), Tlen, true));
        ConvArgs b = conv_args(bufC, cout, pitch_out, d < 2 ? bufB : bufD, cout, pitch_out, r.glens, up_out, 0.1f);
        b.r = xin; b.r_bs = b.x_bs; b.r_pitch = pitch_out;
        if (d == 2 && j > 0) b.flags = F_ACCUM;
        if (d == 2 && j == 2) b.scale = 1.0f / 3.0f;   // xs / num_kernels (models.py:286), as a multiply
        TRY(launch(r, c->rb_c2[i * 3 + j][d], b, Tlen, true));
      }
    }
    snprintf(nm, sizeof nm, "dec.stage%d", i);
    TRY(tap(r, nm, bufD, cout, Tlen, pitch_out));
    stage_in = bufD;
    cin = cout; up = up_out;
  }
  // leaky_relu(0.01) + conv_post + tanh (models.py:287-289)
  const int y_len = Tmax * up;   // 256 * Tmax
  dim3 grid((y_len / 4 + 255) / 256, B);
  return launch_kernel(r, std::nullopt, [&] {
    conv_post_kernel<32><<<grid, 256, 0, r.st>>>(stage_in, 32LL * P * up, P * up, c->d_w + c->post_w_off, o_hat,
                                                 (long long)y_len, y_len, r.glens, Tmax, up);
  });
}

static int run_vc(ovc_ctx* c, const float* spec, int spec_pitch, const long long* lens, const float* g_src, const float* g_tgt,
                  const float* noise, uint64_t seed, float tau, int B, int Tmax, int ragged, float* o_hat,
                  float* z_out, float* zp_out, float* zh_out, cudaStream_t st) {
  const WsLayout W = ws_layout(c, B, Tmax);
  TRY(ensure_ws(c, W, st));
  float* ws = c->d_ws;
  Run r{c, st, B, Tmax, W.P, lens, ragged ? lens : nullptr};
  c->launches = 0;
  const int P = W.P;

  TRY(launch_cond(r, g_src, g_tgt, ws + W.cond));
  const float* cond = ws + W.cond;
  TRY(tap(r, "cond", cond, 1, c->cond_rows_out, c->cond_rows_out));

  // ---- posterior encoder (models.py:212-221)
  const bool aligned = (spec_pitch % 4 == 0) && ((reinterpret_cast<uintptr_t>(spec) & 15) == 0);
  TRY(launch(r, aligned ? c->enc_pre16 : c->enc_pre, conv_args(spec, c->hp.spec_channels, spec_pitch, ws + W.x, 192, P, lens, 1, 1.f), Tmax));
  TRY(tap(r, "enc.pre", ws + W.x, 192, Tmax, P));
  if (c->precision >= 1) {
    TRY(run_wn_tc(r, c->enc_wn, ws + W.x, ws + W.skip, ws + W.acts, ws + W.bufA, ws + W.bufB, cond + c->cond_off_enc_tc,
                  c->cond_rows_out));
  } else {
    TRY(run_wn(r, c->enc_wn, ws + W.x, ws + W.skip, ws + W.acts, cond + c->cond_off_enc, c->cond_rows_out));
  }
  TRY(tap(r, "enc.wn", ws + W.skip, 192, Tmax, P));
  ConvArgs p = conv_args(ws + W.skip, 192, P, ws + W.z, 192, P, lens, 1, 1.f);
  p.r = noise; p.r_bs = 192LL * Tmax; p.r_pitch = Tmax;
  p.tau = tau; p.seed = seed;
  p.callp = c->d_callp;       // set_call_params_kernel wrote (seed, tau) there earlier on this stream
  TRY(launch(r, c->enc_proj, p, Tmax));
  TRY(copy_latent_out(r, W, ws, z_out));
  // ---- flow forward with g_src, reverse with g_tgt (models.py:496-497)
  TRY(run_flow(r, W, ws, false, cond));
  TRY(copy_latent_out(r, W, ws, zp_out));
  TRY(run_flow(r, W, ws, true, cond));
  TRY(copy_latent_out(r, W, ws, zh_out));

  return run_dec(r, W, ws, cond, lens, o_hat);
}

#include "ovc_tts_run.inc"    // run_tts_encode() / run_tts_decode(): SynthesizerTrn.infer on the device

// what every call entry point checks first: a context with finalized weights, and its tensor arguments
static int check_call(const ovc_ctx* c, std::initializer_list<const void*> tensors) {
  if (!c) return fail(OVC_ERR_INVALID, "null context");
  if (!c->finalized) return fail(OVC_ERR_STATE, "ovc_finalize_weights has not been called");
  for (const void* t : tensors)
    if (!t) return fail(OVC_ERR_INVALID, "null tensor argument");
  return OVC_OK;
}
// the generator's widest layer (64 channels x 256 samples per frame) must stay inside 32-bit indexing
static bool too_many_frames(long long T) { return T * 256 * 64 > 2000000000LL; }

static void prof_reset(ovc_ctx* c) { c->prof_log.clear(); }

}  // namespace ovc

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int ovc_abi_version(void) { return OVC_ABI_VERSION; }

const char* ovc_last_error(void) { return ovc::g_err.c_str(); }

int ovc_create(const ovc_hparams* hp, int device, ovc_ctx** out) {
  if (!hp || !out) return fail(OVC_ERR_INVALID, "null argument");
  *out = nullptr;
  int rc = validate_hparams(hp);
  if (rc != OVC_OK) return rc;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    return fail(OVC_ERR_CUDA, "no CUDA device available (%s); this library has no CPU path",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  }
  if (device < 0 || device >= n) return fail(OVC_ERR_INVALID, "device %d out of range (0..%d)", device, n - 1);
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(OVC_ERR_CUDA, "device %d is sm_%d%d; this library contains sm_100a code only", device, prop.major, prop.minor);
  ovc_ctx* c = new ovc_ctx();
  c->hp = *hp;
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  *out = c;
  return OVC_OK;
}

void ovc_destroy(ovc_ctx* c) {
  if (!c) return;
  DeviceGuard dev_guard_(c->device);
  if (c->d_w) cudaFree(c->d_w);
  if (c->d_ws) cudaFree(c->d_ws);
  if (c->d_tts) cudaFree(c->d_tts);
  if (c->d_cond_wrow) cudaFree(c->d_cond_wrow);
  if (c->d_cond_sel) cudaFree(c->d_cond_sel);
  if (c->d_tcw) cudaFree(c->d_tcw);
  if (c->d_re) cudaFree(c->d_re);
  if (c->d_tw) cudaFree(c->d_tw);
  if (c->d_win) cudaFree(c->d_win);
  drop_graphs(c);
  for (auto& q : c->br_stream)
    if (q) cudaStreamDestroy(q);
  for (auto& q : c->br_ev)
    if (q) cudaEventDestroy(q);
  if (c->cap_stream) cudaStreamDestroy(c->cap_stream);
  if (c->d_callp) cudaFree(c->d_callp);
  for (auto& e : c->ev) cudaEventDestroy(e);
  for (auto& kv : c->taps)
    if (kv.second.d) cudaFree(kv.second.d);
  delete c;
}

int ovc_load_tensor(ovc_ctx* c, const char* key, const float* data, const int64_t* shape, int ndim) {
  if (!c || !key || !data || !shape || ndim < 1 || ndim > 4) return fail(OVC_ERR_INVALID, "bad argument to ovc_load_tensor");
  const std::string k(key);
  if (!key_is_hot(k)) return 1;
  HostTensor t;
  t.shape.assign(shape, shape + ndim);
  const int64_t n = t.numel();
  if (n <= 0) return fail(OVC_ERR_INVALID, "tensor '%s' is empty", key);
  t.data.assign(data, data + n);
  c->sd[k] = std::move(t);
  c->finalized = false;
  return OVC_OK;
}

int ovc_finalize_weights(ovc_ctx* c) {
  if (!c) return fail(OVC_ERR_INVALID, "null context");
  return finalize(c);
}

size_t ovc_workspace_floats(const ovc_ctx* c, int B, int Tmax) {
  if (!c || B < 1 || Tmax < 1 || !c->finalized) return 0;
  return ws_layout(c, B, Tmax).total;
}

int ovc_voice_conversion(ovc_ctx* c, const float* spec, const int64_t* lengths, const float* g_src, const float* g_tgt,
                         const float* noise, uint64_t seed, float tau, int B, int Tmax, int ragged, float* o_hat, float* z,
                         float* z_p, float* z_hat, void* stream) {
  TRY(check_call(c, {spec, lengths, g_src, g_tgt, o_hat}));
  if (B < 1 || Tmax < 1) return fail(OVC_ERR_INVALID, "B and Tmax must be positive (got %d, %d)", B, Tmax);
  if (too_many_frames(Tmax)) return fail(OVC_ERR_INVALID, "Tmax %d too large for 32-bit indexing", Tmax);
  if (B > 65535) return fail(OVC_ERR_INVALID, "B %d exceeds the grid limit", B);
  ON_DEVICE(c);
  cudaStream_t st = (cudaStream_t)stream;
  TRY(ensure_ws(c, ws_layout(c, B, Tmax), st));
  TRY(set_call_params(c, seed, tau, st));
  const std::vector<uintptr_t> key = {1, (uintptr_t)spec, (uintptr_t)lengths, (uintptr_t)g_src, (uintptr_t)g_tgt, (uintptr_t)noise,
                                      (uintptr_t)o_hat, (uintptr_t)z, (uintptr_t)z_p, (uintptr_t)z_hat, (uintptr_t)B, (uintptr_t)Tmax,
                                      (uintptr_t)ragged, option_bits(c)};
  return run_graphed(c, key, st, [&](cudaStream_t s) {
    return run_vc(c, spec, Tmax, (const long long*)lengths, g_src, g_tgt, noise, seed, tau, B, Tmax, ragged, o_hat, z, z_p, z_hat, s);
  });
}

static int launch_stft(ovc_ctx* c, const float* wav, const int64_t* wav_lengths, int B, int Lmax, int Tmax, float* spec,
                       int spec_pitch, long long* frames, cudaStream_t st) {
  if (c->hp.spec_channels != STFT_N / 2 + 1 || c->hp.hop_length != 256)
    return fail(OVC_ERR_INVALID, "the STFT kernel is specialised for n_fft = win_length = 1024, hop 256");
  dim3 grid((Tmax + STFT_FR - 1) / STFT_FR, B);
  stft_mag_kernel<<<grid, 256, 0, st>>>(wav, (long long)Lmax, (const long long*)wav_lengths, c->hp.hop_length, spec,
                                        (long long)c->hp.spec_channels * spec_pitch, spec_pitch, Tmax, c->d_tw, c->d_win,
                                        frames);
  CK(cudaGetLastError());
  return OVC_OK;
}

int ovc_spectrogram(ovc_ctx* c, const float* wav, const int64_t* wav_lengths, int B, int Lmax, int Tmax, float* spec,
                    int64_t* frames, void* stream) {
  TRY(check_call(c, {wav, wav_lengths, spec}));
  if (B < 1 || Lmax < 1 || Tmax < 1 || B > 65535) return fail(OVC_ERR_INVALID, "bad sizes B=%d Lmax=%d Tmax=%d", B, Lmax, Tmax);
  ON_DEVICE(c);
  return launch_stft(c, wav, wav_lengths, B, Lmax, Tmax, spec, Tmax, (long long*)frames, (cudaStream_t)stream);
}

int ovc_convert_waveform(ovc_ctx* c, const float* wav, const int64_t* wav_lengths, int B, int Lmax, const float* g_src,
                         const float* g_tgt, const float* noise, uint64_t seed, float tau, float* o_hat, int64_t* frames,
                         void* stream) {
  TRY(check_call(c, {wav, wav_lengths, g_src, g_tgt, o_hat}));
  const int Tmax = Lmax / c->hp.hop_length;
  if (B < 1 || Tmax < 1 || B > 65535) return fail(OVC_ERR_INVALID, "bad sizes B=%d Lmax=%d", B, Lmax);
  if (too_many_frames(Tmax)) return fail(OVC_ERR_INVALID, "Lmax %d too large for 32-bit indexing", Lmax);
  ON_DEVICE(c);
  cudaStream_t st = (cudaStream_t)stream;
  const WsLayout W = ws_layout(c, B, Tmax);
  TRY(ensure_ws(c, W, st));
  TRY(set_call_params(c, seed, tau, st));
  const std::vector<uintptr_t> key = {2, (uintptr_t)wav, (uintptr_t)wav_lengths, (uintptr_t)g_src, (uintptr_t)g_tgt, (uintptr_t)noise,
                                      (uintptr_t)o_hat, (uintptr_t)frames, (uintptr_t)B, (uintptr_t)Lmax, option_bits(c)};
  return run_graphed(c, key, st, [&](cudaStream_t s) {
    float* spec = c->d_ws + W.spec;
    long long* fr = reinterpret_cast<long long*>(c->d_ws + W.frames);
    TRY(launch_stft(c, wav, wav_lengths, B, Lmax, Tmax, spec, W.P, fr, s));
    if (frames) CK(cudaMemcpyAsync(frames, fr, (size_t)B * sizeof(long long), cudaMemcpyDeviceToDevice, s));
    const int rc = run_vc(c, spec, W.P, fr, g_src, g_tgt, noise, seed, tau, B, Tmax, 1, o_hat, nullptr, nullptr, nullptr, s);
    c->launches += 1;
    return rc;
  });
}

int ovc_reference_encoder(ovc_ctx* c, const float* spec, int N, int T, float* out, void* stream) {
  TRY(check_call(c, {}));
  if (!c->has_refenc) return fail(OVC_ERR_MISSING, "the checkpoint had no ref_enc.* tensors");
  if (!spec || !out || N < 1 || T < 1) return fail(OVC_ERR_INVALID, "bad argument to ovc_reference_encoder");
  ON_DEVICE(c);
  cudaStream_t st = (cudaStream_t)stream;
  const int F = c->hp.spec_channels, G = c->hp.gin_channels;
  static const int filt[7] = {1, 32, 32, 64, 64, 128, 128};
  int H[7], W[7];
  H[0] = T; W[0] = F;
  size_t maxact = (size_t)N * T * F;
  for (int i = 0; i < 6; ++i) {
    H[i + 1] = (H[i] - 1) / 2 + 1; W[i + 1] = (W[i] - 1) / 2 + 1;
    maxact = std::max(maxact, (size_t)N * filt[i + 1] * H[i + 1] * W[i + 1]);
  }
  if (128 * W[6] != c->re_gru_in)
    return fail(OVC_ERR_INVALID, "ref_enc.gru.weight_ih_l0 takes %d inputs but spec_channels %d gives %d", c->re_gru_in, F, 128 * W[6]);
  const size_t gi_floats = (size_t)N * H[6] * 384;
  const size_t need = 2 * round_up(maxact, 64) + round_up(gi_floats, 64);
  TRY(grow_arena(c->d_re, c->re_floats, need, st, "reference-encoder scratch"));
  float* a0 = c->d_re;
  float* a1 = a0 + round_up(maxact, 64);
  float* gi = a1 + round_up(maxact, 64);
  {
    const int warps = N * T;
    refenc_layernorm_kernel<<<(warps * 32 + 255) / 256, 256, 0, st>>>(spec, c->d_w + c->re_lng, c->d_w + c->re_lnb, a0, N, F, T);
    CK(cudaGetLastError());
  }
  float* cur = a0; float* nxt = a1;
  for (int i = 0; i < 6; ++i) {
    const long long total = (long long)N * filt[i + 1] * H[i + 1] * W[i + 1];
    refenc_conv_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(cur, c->d_w + c->re_conv_w[i], c->d_w + c->re_conv_b[i], nxt, N,
                                                                        filt[i], H[i], W[i], filt[i + 1], H[i + 1], W[i + 1]);
    CK(cudaGetLastError());
    std::swap(cur, nxt);
  }
  {
    const long long warps = (long long)N * H[6] * 384;
    refenc_gru_in_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(cur, c->d_w + c->re_wih, c->d_w + c->re_bih, gi, N, 128,
                                                                              H[6], W[6], 384);
    CK(cudaGetLastError());
    refenc_gru_kernel<<<N, 128, 0, st>>>(gi, c->d_w + c->re_whh, c->d_w + c->re_bhh, c->d_w + c->re_pw, c->d_w + c->re_pb, out, H[6], G);
    CK(cudaGetLastError());
  }
  return OVC_OK;
}

int ovc_tts_info(const ovc_ctx* c, int32_t* out8) {
  if (!c || !out8) return fail(OVC_ERR_INVALID, "null argument");
  if (!c->finalized) return fail(OVC_ERR_STATE, "ovc_finalize_weights has not been called");
  const TtsLayers& L = c->tts;
  const int32_t v[8] = {L.ready ? 1 : 0, L.n_vocab, L.n_speakers, L.heads, L.n_layers, L.window, L.Fc, L.D};
  for (int i = 0; i < 8; ++i) out8[i] = v[i];
  return OVC_OK;
}

int ovc_tts_encode(ovc_ctx* c, const int64_t* tokens, const int64_t* x_lengths, const int64_t* sid, const float* noise_w,
                   uint64_t seed, float noise_scale_w, float length_scale, float sdp_ratio, int B, int T, int64_t* y_lengths,
                   float* w_ceil, float* logw, void* stream) {
  TRY(check_call(c, {}));
  if (!c->tts.ready) return fail(OVC_ERR_STATE, "the checkpoint has no TTS members (enc_p / dp / sdp / emb_g): not a V1 base speaker");
  if (!tokens || !x_lengths || !sid || !y_lengths) return fail(OVC_ERR_INVALID, "null tensor argument");
  if (B < 1 || T < 1) return fail(OVC_ERR_INVALID, "B and T must be positive (got %d, %d)", B, T);
  if (B > 65535 || (long long)T * T > 2000000000LL / 256) return fail(OVC_ERR_INVALID, "B %d / T %d exceed the grid limits", B, T);
  if (!(length_scale > 0.f)) return fail(OVC_ERR_INVALID, "length_scale must be positive");
  ON_DEVICE(c);
  return run_tts_encode(c, (const long long*)tokens, (const long long*)x_lengths, (const long long*)sid, noise_w, seed,
                        noise_scale_w, length_scale, sdp_ratio, B, T, (long long*)y_lengths, w_ceil, logw, (cudaStream_t)stream);
}

int ovc_tts_decode(ovc_ctx* c, const float* noise, uint64_t seed, float noise_scale, int B, int Ymax, int max_len, int ragged,
                   float* o, float* z, float* z_p, void* stream) {
  if (!c) return fail(OVC_ERR_INVALID, "null context");
  if (!c->finalized || !c->tts.ready) return fail(OVC_ERR_STATE, "no finalized TTS checkpoint");
  if (c->tts_B < 1) return fail(OVC_ERR_STATE, "ovc_tts_decode needs a preceding ovc_tts_encode");
  if (B != c->tts_B) return fail(OVC_ERR_INVALID, "B = %d but the pending ovc_tts_encode had B = %d", B, c->tts_B);
  if (!o) return fail(OVC_ERR_INVALID, "null tensor argument");
  if (Ymax < 1) return fail(OVC_ERR_INVALID, "Ymax must be positive");
  if (too_many_frames(Ymax)) return fail(OVC_ERR_INVALID, "Ymax %d too large for 32-bit indexing", Ymax);
  ON_DEVICE(c);
  if (max_len < 0) return fail(OVC_ERR_INVALID, "max_len must be >= 0 (0 = no limit)");
  return run_tts_decode(c, noise, seed, noise_scale, B, Ymax, max_len, ragged, o, z, z_p, (cudaStream_t)stream);
}

int ovc_set_precision(ovc_ctx* c, int mode) {
  if (!c) return fail(OVC_ERR_INVALID, "null context");
  if (mode < 0 || mode > 3)
    return fail(OVC_ERR_INVALID, "precision mode must be 0 (fp32 FFMA2), 1 (3xFP16 tensor cores), 2 (single-pass fp16) or 3 (fp16 generator "
                                 "storage)");
  c->precision = mode;
  return OVC_OK;
}

int ovc_set_option(ovc_ctx* c, int key, int value) {
  if (!c) return fail(OVC_ERR_INVALID, "null context");
  switch (key) {
    case OVC_OPT_WIDE_VARIANT:
      if (value != 0 && value != 2 && value != 3) return fail(OVC_ERR_INVALID, "wide variant must be 0, 2 or 3 (1 is retired)");
      c->wide_variant = value;
      return OVC_OK;
    case OVC_OPT_TTS_SIMPLE: c->tts_simple = value != 0; return OVC_OK;
    case OVC_OPT_GRAPH: c->use_graph = value != 0; return OVC_OK;
    case OVC_OPT_PDL:
      if (value < 0 || value > 2) return fail(OVC_ERR_INVALID, "pdl must be 0, 1 or 2");
      c->use_pdl = value;
      return OVC_OK;
    case 4:   // activation loads by the converter warps (OVC_OPT_ACT_TMA = 0): retired
    case 6:   // A/B switches of the persistent conv kernel (OVC_OPT_TUNE): retired
      return fail(OVC_ERR_INVALID, "option %d is retired", key);
    case OVC_OPT_BRANCHES: c->use_branches = value != 0; return OVC_OK;
    case OVC_OPT_PAIR: c->use_pair = value != 0; return OVC_OK;
    default: return fail(OVC_ERR_INVALID, "unknown option %d", key);
  }
}

int ovc_last_launch_count(const ovc_ctx* c) { return c ? c->launches : 0; }

int ovc_graph_replays(const ovc_ctx* c) { return c ? c->graph_replays : 0; }

int ovc_profile_enable(ovc_ctx* c, int enable) {
  if (!c) return fail(OVC_ERR_INVALID, "null context");
  c->prof = enable != 0;
  prof_reset(c);
  return OVC_OK;
}

int ovc_profile_read(ovc_ctx* c, double* ms, int64_t* launches, double* flops, double* bytes) {
  if (!c) return fail(OVC_ERR_INVALID, "null context");
  double tms = 0, tf = 0, tb = 0;
  int64_t n = 0;
  for (size_t k = 0; k < c->prof_log.size(); ++k) {
    const ProfRec& p = c->prof_log[k];
    if (!p.family) continue;
    float m = 0;
    CK(cudaEventElapsedTime(&m, c->ev[2 * k], c->ev[2 * k + 1]));
    tms += m;
    tf += p.flops;
    tb += p.bytes;
    ++n;
  }
  if (ms) *ms = tms;
  if (launches) *launches = n;
  if (flops) *flops = tf;
  if (bytes) *bytes = tb;
  prof_reset(c);
  return OVC_OK;
}

int ovc_profile_detail(ovc_ctx* c, int max, char* names /* max x 16 */, double* ms, double* flops, double* bytes, int* family) {
  if (!c) return fail(OVC_ERR_INVALID, "null context");
  int n = 0;
  for (; n < (int)c->prof_log.size() && n < max; ++n) {
    const ProfRec& p = c->prof_log[n];
    float m = 0;
    CK(cudaEventElapsedTime(&m, c->ev[2 * n], c->ev[2 * n + 1]));
    if (names) {
      const int tag = p.tag, v = p.variant;
      if (tag && (v == V_TCPAIR64 || v == V_TCPAIR32)) snprintf(names + 16 * n, 16, "P%dk%dd%d", tag >> 16, (tag >> 8) & 255, tag & 255);
      else if (tag) {
        const bool h = v == V_TCH128 || v == V_TCH64 || v == V_TCH32;   // fp16-storage launch: "H..." instead of "T..."
        snprintf(names + 16 * n, 16, "%c%dc%dk%dd%d", h ? 'H' : 'T', v == V_TC128 || v == V_TCH128 ? 128 : v == V_TC64 || v == V_TCH64 ? 64 : 32,
                 tag >> 16, (tag >> 8) & 255, tag & 255);
      }
      else { strncpy(names + 16 * n, variant_name(v), 15); names[16 * n + 15] = 0; }
    }
    if (ms) ms[n] = m;
    if (flops) flops[n] = p.flops;
    if (bytes) bytes[n] = p.bytes;
    if (family) family[n] = p.family;
  }
  return n;
}

int ovc_debug_enable(ovc_ctx* c, int enable) {
  if (!c) return fail(OVC_ERR_INVALID, "null context");
  c->debug = enable != 0;
  return OVC_OK;
}

int ovc_debug_fetch(ovc_ctx* c, const char* name, float* host_out, size_t max_floats, int64_t* shape4) {
  if (!c || !name) return fail(OVC_ERR_INVALID, "null argument");
  auto it = c->taps.find(name);
  if (it == c->taps.end()) return fail(OVC_ERR_INVALID, "no debug tap named '%s' (enable debug and run a call first)", name);
  const DebugBuf& d = it->second;
  const size_t n = (size_t)d.shape[0] * d.shape[1] * d.shape[3];
  if (shape4) memcpy(shape4, d.shape, sizeof d.shape);
  if (host_out) {
    if (max_floats < n) return fail(OVC_ERR_INVALID, "buffer too small for tap '%s': need %zu floats", name, n);
    ON_DEVICE(c);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(host_out, d.d, n * sizeof(float), cudaMemcpyDeviceToHost));
  }
  return OVC_OK;
}

}  // extern "C"
