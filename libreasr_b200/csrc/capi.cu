// C-ABI layer: handle, weight ingestion / repack, workspaces, and the entry points declared
// in include/rnnt_b200.h.  Host orchestration only -- all arithmetic is in the kernels.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/rnnt_b200.h"
#include "kernels.h"
#include "tc_common.cuh"

using namespace rnnt;

namespace {

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  cudaError_t ensure(size_t need) {
    if (need <= bytes) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
    size_t sz = need + need / 8;
    cudaError_t e = cudaMalloc(&p, sz);
    if (e != cudaSuccess) return e;
    bytes = sz;
    return cudaMemset(p, 0, sz);
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
};

struct EncLayer {
  int in = 0;
  float *Wih_r = nullptr, *bias_r = nullptr, *Whh_t = nullptr, *h0 = nullptr, *c0 = nullptr, *bn_scale = nullptr,
        *bn_shift = nullptr;
};

}  // namespace

struct rnnt_b200_handle_s {
  rnnt_b200_config cfg;
  std::string err;
  std::map<std::string, std::vector<float>> raw;
  bool finalized = false;
  int sm_count = 0, coop_blocks = 0;
  int64_t launches = 0;
  int open_streams = 0;
  int64_t fp32_decode_launches = 0;    // launches of the fp32 cooperative decode kernel (the slow twin of the tcgen05 kernels)                // streaming sessions that reference this handle (destroy refuses while > 0)
  std::vector<void*> weight_allocs;
  // frontend
  float* window = nullptr;
  float2* tw = nullptr;
  int *mel_start = nullptr, *mel_count = nullptr, *mel_off = nullptr;
  float* mel_w = nullptr;
  // encoder
  float *ln_g = nullptr, *ln_b = nullptr;
  std::vector<EncLayer> enc;
  // predictor + joint
  DecodeWeights dw;
  float* W1 = nullptr;  // [J][2H] as loaded; enc half = W1 + H with ld 2H
  uint8_t* W1e_img = nullptr;          // TC modes: operand image of the enc half
  std::vector<uint8_t*> Wih_img;       // TC modes: operand images of the interleaved W_ih
  std::vector<uint8_t*> Whh_img;       // TC modes: operand images (TR = NC) of the interleaved W_hh
  bool lstm_tc_ok = false;             // persistent tcgen05 LSTM layer usable for this H / SM count
  std::vector<uint8_t*> Whh_img2;      // ... (TR = 128) for the cluster split-K kernel (lstm_tc2.cu)
  bool lstm_tc2_ok = false;            // cluster split-K LSTM layer usable (H % 256 == 0, H <= 1024, clusters co-resident)
  bool dec_tc_ok = false;              // tcgen05 decode kernel usable
  uint8_t *W1p_img = nullptr, *W2_img = nullptr;
  // decode_tc2.cu (cluster split-K decode): row tiles of one cluster, TR = 32 / V/32 / 96
  uint8_t *W1p_img2 = nullptr, *W2_img2 = nullptr, *K1_img2 = nullptr, *R_img2[2] = {nullptr, nullptr};
  bool dec_tc2_ok = false;
  // beam search (beam.cu): 256-row-tile weight images for gemm_tc.cu, built at the first call; workspaces
  uint8_t *bm_w1p = nullptr, *bm_w2 = nullptr, *bm_k1 = nullptr, *bm_r[2] = {nullptr, nullptr};
  DevBuf bm_state, bm_meta, bm_aimg, bm_f32;
  DevBuf lt_f32, lt_i32, lt_enc;       // lattice.cu workspaces (training-time forward + loss)
  uint8_t* R_img[kMaxPredLayers] = {nullptr, nullptr, nullptr, nullptr};
  uint8_t* K_img[kMaxPredLayers] = {nullptr, nullptr, nullptr, nullptr};
  DevBuf dimg;                         // decode activation operand images
  DevBuf dkeys;                        // decode arg-max keys + evaluation counts
  DevBuf x_img[2], gbar;               // TC modes: h operand images (ping-pong), grid step counter
  DevBuf a_img;                        // TC modes: activation operand image (workspace)
  // workspaces
  DevBuf feats, lnx, xp, ya, yb, ep, ehT[2], ecT, dhT, dxT, dgT, deT, dppT, dzT, dpart, dlse;
  DevBuf t_audio, t_lens, t_tokens, t_ntok, t_nlp, t_iters, t_enc;
  // fused language model (lm.py): fp32 layouts + per-call fuser workspace / registered stream blob
  LmWeights lmw;
  DevBuf lm_ws, lm_logitT, lm_part, lm_jpart, lm_fpart;
  bool lm_tc_ok = false;      // LM phases available in the tcgen05 decode kernel for this shape
  uint8_t* lmR_img[kTcLmLayers] = {};   // operand images of the LM weight slices (TR = NC_L / NC_B)
  uint8_t* lmW_img[kTcLmLayers] = {};
  uint8_t* lmWo_img = nullptr;
  DevBuf lm_himg, lm_stat;
  float* lm_blob = nullptr;   // caller-owned fuser state (rnnt_b200_set_lm_state); nullptr = fresh fuser per call
  int lm_blob_B = 0;
  // resampler filter banks per source rate (built on first use)
  struct ResampleTab { int o = 0, n = 0, width = 0, K = 0; float* dev = nullptr; };
  std::map<int, ResampleTab> resample_tabs;
  // transcribe_host: copy engine stream + events so that the H2D of utterance block i+1 overlaps the front end of block i
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t copy_ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  // two-deep pipeline over the whole path (rnnt_b200_pipeline_submit / _collect): the front half of batch i+1 (host->device
  // copy, front end) runs on a low-priority stream under the persistent recurrent kernels of batch i, which leave 20 SMs idle
  struct PipeSlot {
    DevBuf audio, feats, lens, tokens, ntok, nlp;
    cudaEvent_t in_ready = nullptr, front_done = nullptr, back_done = nullptr;
    bool busy = false;
  };
  PipeSlot pipe[2];
  cudaStream_t pipe_front = nullptr, pipe_back = nullptr;
  // profiling
  bool profiling = false;
  std::vector<cudaEvent_t*> evsets;  // one set of events per profiled transcribe() call: 6 stage marks + 2 per encoder layer
  int ev_used = 0;                   // sets holding a complete recording
  cudaEvent_t* ev = nullptr;         // set being recorded
};

namespace {

constexpr int kEvPerSet = 6 + 2 * 16;

thread_local std::string g_create_err;

int fail(rnnt_b200_handle h, int code, const std::string& msg) {
  if (h) h->err = msg; else g_create_err = msg;
  return code;
}
int fail_cuda(rnnt_b200_handle h, cudaError_t e, const char* what) {
  return fail(h, RNNT_B200_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define CK(expr)                                                   \
  do {                                                             \
    cudaError_t e_ = (expr);                                       \
    if (e_ != cudaSuccess) return fail_cuda(h, e_, #expr);         \
  } while (0)
// kernel launch through a launcher returning cudaError_t; counts launches
#define LAUNCH(n, expr)                                            \
  do {                                                             \
    cudaError_t e_ = (expr);                                       \
    if (e_ != cudaSuccess) return fail_cuda(h, e_, #expr);         \
    h->launches += (n);                                            \
  } while (0)

int64_t num_frames(const rnnt_b200_config& c, int64_t n) { return n / c.hop_length + 1; }
int64_t num_steps(const rnnt_b200_config& c, int64_t n) {
  const int64_t F = num_frames(c, n);
  return F >= c.n_stack ? (F - c.n_stack) / c.downsample + 1 : 0;
}

template <class T>
cudaError_t upload(rnnt_b200_handle h, const std::vector<T>& v, T** out) {
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, std::max<size_t>(v.size(), 1) * sizeof(T));
  if (e != cudaSuccess) return e;
  h->weight_allocs.push_back(p);
  *out = reinterpret_cast<T*>(p);
  return cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
}
cudaError_t dalloc(rnnt_b200_handle h, size_t n_floats, float** out) {
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, std::max<size_t>(n_floats, 1) * sizeof(float));
  if (e != cudaSuccess) return e;
  h->weight_allocs.push_back(p);
  *out = reinterpret_cast<float*>(p);
  return cudaSuccess;
}

int64_t expected_numel(const rnnt_b200_config& c, const std::string& name, bool* known) {
  const int64_t H = c.hidden_sz, X = (int64_t)c.n_mels * c.n_stack, E = c.embed_sz, J = c.joint_sz, V = c.vocab_sz;
  *known = true;
  if (name == "frontend.window") return c.win_length;
  if (name == "frontend.mel_fb") return (int64_t)(c.n_fft / 2 + 1) * c.n_mels;
  if (name == "encoder.input_norm.weight" || name == "encoder.input_norm.bias") return X;
  if (name == "predictor.embed.weight") return V * E;
  if (name == "predictor.ffn.weight") return H * E;
  if (name == "predictor.ffn.bias") return H;
  if (name == "joint.joint.0.weight") return J * 2 * H;
  if (name == "joint.joint.0.bias") return J;
  if (name == "joint.joint.2.weight") return V * J;
  if (name == "joint.joint.2.bias") return V;
  if (c.lm_layers > 0 && name.compare(0, 3, "lm.") == 0) {   // LM.state_dict() keys (lm.py:20-29)
    const int64_t Hl = c.lm_hidden_sz, El = c.lm_embed_sz;
    const std::string rest = name.substr(3);
    if (rest == "embed.weight") return V * El;
    if (rest == "linear.weight") return V * Hl;
    if (rest == "linear.bias") return V;
    const size_t pos = rest.rfind("_l");
    if (rest.compare(0, 4, "rnn.") == 0 && pos != std::string::npos && pos > 4 && pos + 2 < rest.size()) {
      const std::string f = rest.substr(4, pos - 4), num = rest.substr(pos + 2);
      int idx = 0;
      bool digits = true;
      for (char ch : num) { digits = digits && ch >= '0' && ch <= '9'; idx = idx * 10 + (ch - '0'); }
      if (digits && num.size() <= 2 && idx < c.lm_layers) {
        if (f == "weight_ih") return 4 * Hl * (idx == 0 ? El : Hl);
        if (f == "weight_hh") return 4 * Hl * Hl;
        if (f == "bias_ih" || f == "bias_hh") return 4 * Hl;
      }
    }
  }
  for (int side = 0; side < 2; ++side) {
    const std::string pre = side == 0 ? "encoder.rnn_stack." : "predictor.rnn_stack.";
    if (name.compare(0, pre.size(), pre) != 0) continue;
    const std::string rest = name.substr(pre.size());
    const int L = side == 0 ? c.enc_layers : c.pred_layers;
    int idx = -1, used = 0;
    if (sscanf(rest.c_str(), "hs.%d%n", &idx, &used) == 1 && (size_t)used == rest.size() && idx >= 0 && idx < L)
      return side == 0 ? 2 * H : H;
    char field[64];
    if (sscanf(rest.c_str(), "bns.%d.%63s", &idx, field) == 2 && idx >= 0 && idx < L) {
      const std::string f(field);
      if (f == "weight" || f == "bias" || f == "running_mean" || f == "running_var") return H;
    }
    if (sscanf(rest.c_str(), "rnns.%d.%63s", &idx, field) == 2 && idx >= 0 && idx < L) {
      const std::string f(field);
      if (side == 0) {
        const int64_t in = idx == 0 ? X : H;
        if (f == "weight_ih_l0") return 4 * H * in;
        if (f == "weight_hh_l0") return 4 * H * H;
        if (f == "bias_ih_l0" || f == "bias_hh_l0") return 4 * H;
      } else {
        if (f == "kernel" || f == "recurrent_kernel") return H * 3 * H;
        if (f == "bias" || f == "recurrent_bias") return 3 * H;
      }
    }
  }
  *known = false;
  return 0;
}

int validate_config(const rnnt_b200_config& c, std::string* why) {
  auto bad = [&](const char* m) { *why = m; return 1; };
  if (c.n_fft != 1024) return bad("only n_fft == 1024 is implemented (melkwargs.n_fft, config/testing.yaml:133)");
  if (c.win_length < 2 || c.win_length > 1024 || (c.win_length & 1)) return bad("win_length must be even and <= n_fft");
  if (c.hop_length < 1) return bad("hop_length must be >= 1");
  if (c.n_mels < 1 || c.n_mels > 256) return bad("n_mels must be in [1, 256]");
  if (c.n_stack < 1 || c.n_stack > kFrontendMaxWarps) return bad("n_stack must be in [1, 16]");
  if (c.downsample < 1) return bad("downsample must be >= 1");
  if (c.hidden_sz < 64 || c.hidden_sz % 64) return bad("hidden_sz must be a positive multiple of 64");
  if (c.joint_sz < 64 || c.joint_sz % 64) return bad("joint_sz must be a positive multiple of 64");
  if (c.vocab_sz < 32 || c.vocab_sz % 32) return bad("vocab_sz must be a positive multiple of 32");
  if ((c.n_mels * c.n_stack) % 4) return bad("n_mels*n_stack must be a multiple of 4");
  if (c.embed_sz < 4 || c.embed_sz % 4) return bad("embed_sz must be a positive multiple of 4");
  if (c.enc_layers < 1 || c.enc_layers > 16) return bad("enc_layers must be in [1, 16]");
  if (c.pred_layers < 1 || c.pred_layers > kMaxPredLayers) return bad("pred_layers must be in [1, 4]");
  if (c.blank < 0 || c.blank >= c.vocab_sz || c.bos < 0 || c.bos >= c.vocab_sz) return bad("blank/bos out of range");
  if (c.lm_layers < 0 || c.lm_layers > kMaxLmLayers) return bad("lm_layers must be in [0, 8]");
  if (c.lm_layers > 0) {
    if (c.lm_hidden_sz < 64 || c.lm_hidden_sz % 64) return bad("lm_hidden_sz must be a positive multiple of 64");
    if (c.lm_embed_sz < 4 || c.lm_embed_sz % 4) return bad("lm_embed_sz must be a positive multiple of 4");
  }
  if (c.gemm_mode != RNNT_B200_GEMM_FP32_SIMT && c.gemm_mode != RNNT_B200_GEMM_TC_FP16X3)
    return bad("gemm_mode not available in this build (0 = fp32 CUDA cores, 1 = tcgen05 3xFP16)");
  return 0;
}

int bp_of(int B) { return (int)round_up(B, kBatchTile); }

}  // namespace

extern "C" {

int32_t rnnt_b200_abi_version(void) { return RNNT_B200_ABI_VERSION; }

int32_t rnnt_b200_default_config(rnnt_b200_config* c) {
  if (!c) return RNNT_B200_ERR_INVALID;
  memset(c, 0, sizeof(*c));
  c->sample_rate = 16000; c->n_fft = 1024; c->win_length = 400; c->hop_length = 160;
  c->n_mels = 128; c->n_stack = 10; c->downsample = 8;
  c->enc_layers = 6; c->pred_layers = 2; c->hidden_sz = 1024; c->embed_sz = 512; c->joint_sz = 1024; c->vocab_sz = 2048;
  c->blank = 0; c->bos = 2; c->device = 0; c->gemm_mode = RNNT_B200_GEMM_TC_FP16X3;
  c->log_offset = 1e-6f; c->ln_eps = 1e-5f; c->bn_eps = 1e-5f;
  c->lm_layers = 0; c->lm_hidden_sz = 768; c->lm_embed_sz = 768;   // LM off; shapes of the shipped override (testing.yaml:306-313)
  c->lm_alpha = 0.1f; c->lm_theta = 1.0f;                           // lm.py:13-14
  return RNNT_B200_OK;
}

const char* rnnt_b200_last_error(rnnt_b200_handle h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int32_t rnnt_b200_create(const rnnt_b200_config* cfg, rnnt_b200_handle* out) {
  rnnt_b200_handle h = nullptr;
  if (!cfg || !out) return fail(nullptr, RNNT_B200_ERR_INVALID, "null argument");
  *out = nullptr;
  std::string why;
  if (validate_config(*cfg, &why)) return fail(nullptr, RNNT_B200_ERR_INVALID, why);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, RNNT_B200_ERR_CUDA,
                std::string("no CUDA device available (this library has no CPU fallback): ") + cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, RNNT_B200_ERR_INVALID, "device ordinal out of range");
  if ((e = cudaSetDevice(cfg->device)) != cudaSuccess) return fail_cuda(nullptr, e, "cudaSetDevice");
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, cfg->device)) != cudaSuccess) return fail_cuda(nullptr, e, "cudaGetDeviceProperties");
  if (prop.major != 10)
    return fail(nullptr, RNNT_B200_ERR_UNSUPPORTED, "kernels are built for sm_100a (B200) only; found sm_" +
                                                        std::to_string(prop.major) + std::to_string(prop.minor));
  h = new rnnt_b200_handle_s();
  h->cfg = *cfg;
  h->sm_count = prop.multiProcessorCount;
  if ((e = configure_lstm()) != cudaSuccess || (e = configure_gemm_tc()) != cudaSuccess ||
      (e = configure_lstm_tc()) != cudaSuccess || (e = configure_lstm_tc2()) != cudaSuccess || (e = configure_decode_tc()) != cudaSuccess || (e = configure_decode_tc2()) != cudaSuccess || (e = configure_decode(cfg->device, &h->coop_blocks)) != cudaSuccess) {
    delete h;
    return fail_cuda(nullptr, e, "kernel configuration");
  }
  *out = h;
  return RNNT_B200_OK;
}

int32_t rnnt_b200_destroy(rnnt_b200_handle h) {
  if (!h) return RNNT_B200_OK;
  if (h->open_streams > 0)
    return fail(h, RNNT_B200_ERR_STATE, "destroy: " + std::to_string(h->open_streams) + " streaming session(s) still reference this handle; close them first");
  cudaSetDevice(h->cfg.device);
  cudaDeviceSynchronize();
  for (void* p : h->weight_allocs) cudaFree(p);
  DevBuf* bufs[] = {&h->feats, &h->lnx, &h->xp, &h->ya, &h->yb, &h->ep, &h->ehT[0], &h->ehT[1], &h->ecT, &h->dhT, &h->dxT,
                    &h->dgT, &h->deT, &h->dppT, &h->dzT, &h->dpart, &h->dlse, &h->t_audio, &h->t_lens, &h->t_tokens,
                    &h->t_ntok, &h->t_nlp, &h->t_iters, &h->t_enc, &h->a_img, &h->x_img[0], &h->x_img[1], &h->gbar, &h->dimg, &h->dkeys,
                    &h->lm_ws, &h->lm_logitT, &h->lm_part, &h->lm_jpart, &h->lm_fpart, &h->lm_himg, &h->lm_stat};
  for (DevBuf* b : bufs) b->release();
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  for (cudaEvent_t e : h->copy_ev)
    if (e) cudaEventDestroy(e);
  for (auto& ps : h->pipe) {
    for (DevBuf* b : {&ps.audio, &ps.feats, &ps.lens, &ps.tokens, &ps.ntok, &ps.nlp}) b->release();
    for (cudaEvent_t e : {ps.in_ready, ps.front_done, ps.back_done})
      if (e) cudaEventDestroy(e);
  }
  if (h->pipe_front) cudaStreamDestroy(h->pipe_front);
  if (h->pipe_back) cudaStreamDestroy(h->pipe_back);
  for (cudaEvent_t* set : h->evsets) {
    for (int i = 0; i < kEvPerSet; ++i) cudaEventDestroy(set[i]);
    delete[] set;
  }
  delete h;
  return RNNT_B200_OK;
}

int32_t rnnt_b200_set_weight(rnnt_b200_handle h, const char* name, const float* data, int64_t numel) {
  if (!h || !name || !data) return fail(h, RNNT_B200_ERR_INVALID, "null argument");
  if (h->finalized) return fail(h, RNNT_B200_ERR_STATE, "weights are frozen after finalize()");
  const std::string nm(name);
  if (nm.size() > 19 && nm.compare(nm.size() - 19, 19, "num_batches_tracked") == 0) return RNNT_B200_OK;
  bool known = false;
  const int64_t want = expected_numel(h->cfg, nm, &known);
  if (!known) return fail(h, RNNT_B200_ERR_INVALID, "unknown weight name: " + nm);
  if (want != numel)
    return fail(h, RNNT_B200_ERR_INVALID,
                "size mismatch for " + nm + ": expected " + std::to_string(want) + " elements, got " + std::to_string(numel));
  h->raw[nm].assign(data, data + numel);
  return RNNT_B200_OK;
}

int32_t rnnt_b200_finalize(rnnt_b200_handle h, void* stream) {
  if (!h) return RNNT_B200_ERR_INVALID;
  if (h->finalized) return RNNT_B200_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const rnnt_b200_config& c = h->cfg;
  const int H = c.hidden_sz, X = c.n_mels * c.n_stack, E = c.embed_sz, J = c.joint_sz, V = c.vocab_sz;
  CK(cudaSetDevice(c.device));
  auto need = [&](const std::string& n) -> const std::vector<float>* {
    auto it = h->raw.find(n);
    return it == h->raw.end() ? nullptr : &it->second;
  };
#define NEED(var, name)                                                                    \
  const std::vector<float>* var = need(name);                                              \
  if (!var) return fail(h, RNNT_B200_ERR_STATE, std::string("missing weight: ") + (name));

  // ---- frontend constants ----
  NEED(win, "frontend.window");
  NEED(fb, "frontend.mel_fb");
  CK(upload(h, *win, &h->window));
  {
    std::vector<float2> tw(512);
    for (int j = 0; j < 512; ++j) {
      const double a = -2.0 * M_PI * (double)j / 1024.0;
      tw[j] = make_float2((float)cos(a), (float)sin(a));
    }
    CK(upload(h, tw, &h->tw));
    const int nf = c.n_fft / 2 + 1;
    std::vector<int> ms(c.n_mels), mc(c.n_mels), mo(c.n_mels);
    std::vector<float> mw;
    for (int m = 0; m < c.n_mels; ++m) {
      int lo = -1, hi = -1;
      for (int k = 0; k < nf; ++k)
        if ((*fb)[(size_t)k * c.n_mels + m] != 0.f) {
          if (lo < 0) lo = k;
          hi = k;
        }
      ms[m] = lo < 0 ? 0 : lo;
      mc[m] = lo < 0 ? 0 : hi - lo + 1;
      mo[m] = (int)mw.size();
      for (int k = 0; k < mc[m]; ++k) mw.push_back((*fb)[(size_t)(ms[m] + k) * c.n_mels + m]);
    }
    CK(upload(h, ms, &h->mel_start));
    CK(upload(h, mc, &h->mel_count));
    CK(upload(h, mo, &h->mel_off));
    CK(upload(h, mw, &h->mel_w));
  }

  auto bn_fold = [&](const std::string& pre, float** scale, float** shift) -> int {
    NEED(g, pre + ".weight");
    NEED(b, pre + ".bias");
    NEED(mu, pre + ".running_mean");
    NEED(var, pre + ".running_var");
    std::vector<float> sc(H), sh(H);
    for (int i = 0; i < H; ++i) {
      sc[i] = (*g)[i] / sqrtf((*var)[i] + c.bn_eps);
      sh[i] = (*b)[i] - (*mu)[i] * sc[i];
    }
    CK(upload(h, sc, scale));
    CK(upload(h, sh, shift));
    return 0;
  };

  // scratch for device-side repacks (freed at the end)
  std::vector<void*> tmp;
  auto tmp_upload = [&](const std::vector<float>& v, float** out) -> cudaError_t {
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, v.size() * sizeof(float));
    if (e != cudaSuccess) return e;
    tmp.push_back(p);
    *out = (float*)p;
    return cudaMemcpyAsync(p, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice, st);
  };
  auto tmp_alloc = [&](size_t n, float** out) -> cudaError_t {
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, n * sizeof(float));
    if (e != cudaSuccess) return e;
    tmp.push_back(p);
    *out = (float*)p;
    return cudaSuccess;
  };
  int* perm4 = nullptr;  // interleaved row (unit*4+gate) <- native row (gate*H+unit)
  int* perm3 = nullptr;
  {
    std::vector<int> p4(4 * H), p3(3 * H);
    for (int u = 0; u < H; ++u) {
      for (int g = 0; g < 4; ++g) p4[u * 4 + g] = g * H + u;
      for (int g = 0; g < 3; ++g) p3[u * 3 + g] = g * H + u;
    }
    CK(upload(h, p4, &perm4));
    CK(upload(h, p3, &perm3));
  }
  auto interleave = [&](const std::vector<float>& v, int G) {
    std::vector<float> o(v.size());
    for (int u = 0; u < H; ++u)
      for (int g = 0; g < G; ++g) o[u * G + g] = v[g * H + u];
    return o;
  };

  // ---- encoder (models.py:68-100; custom_rnn.py:113-126,259-269) ----
  {
    NEED(lg, "encoder.input_norm.weight");
    NEED(lb, "encoder.input_norm.bias");
    CK(upload(h, *lg, &h->ln_g));
    CK(upload(h, *lb, &h->ln_b));
  }
  h->enc.resize(c.enc_layers);
  for (int l = 0; l < c.enc_layers; ++l) {
    EncLayer& L = h->enc[l];
    L.in = l == 0 ? X : H;
    const std::string p = "encoder.rnn_stack.rnns." + std::to_string(l) + ".";
    NEED(wih, p + "weight_ih_l0");
    NEED(whh, p + "weight_hh_l0");
    NEED(bih, p + "bias_ih_l0");
    NEED(bhh, p + "bias_hh_l0");
    NEED(hs, "encoder.rnn_stack.hs." + std::to_string(l));
    std::vector<float> bsum(4 * H);
    for (int i = 0; i < 4 * H; ++i) bsum[i] = (*bih)[i] + (*bhh)[i];
    CK(upload(h, interleave(bsum, 4), &L.bias_r));
    CK(upload(h, std::vector<float>(hs->begin(), hs->begin() + H), &L.h0));
    CK(upload(h, std::vector<float>(hs->begin() + H, hs->end()), &L.c0));
    if (bn_fold("encoder.rnn_stack.bns." + std::to_string(l), &L.bn_scale, &L.bn_shift)) return RNNT_B200_ERR_STATE;
    float *d_wih, *d_whh, *d_whh_r;
    CK(tmp_upload(*wih, &d_wih));
    CK(tmp_upload(*whh, &d_whh));
    CK(tmp_alloc((size_t)4 * H * H, &d_whh_r));
    CK(dalloc(h, (size_t)4 * H * L.in, &L.Wih_r));
    CK(dalloc(h, (size_t)4 * H * H, &L.Whh_t));
    LAUNCH(1, launch_gather_rows(d_wih, L.Wih_r, perm4, 4 * H, L.in, st));
    LAUNCH(1, launch_gather_rows(d_whh, d_whh_r, perm4, 4 * H, H, st));
    LAUNCH(1, launch_transpose(d_whh_r, H, L.Whh_t, 4 * H, H, st));  // -> [H][4H]
    if (c.gemm_mode == RNNT_B200_GEMM_TC_FP16X3) {
      void* img = nullptr;
      CK(cudaMalloc(&img, gemm_tc_w_image_bytes(4 * H, L.in)));
      h->weight_allocs.push_back(img);
      h->Wih_img.push_back((uint8_t*)img);
      LAUNCH(1, launch_to_image(L.Wih_r, L.in, 4 * H, L.in, 256, (uint8_t*)img, st));
      LstmTcPlan pl;
      h->lstm_tc_ok = lstm_tc_plan(H, 1, h->sm_count, &pl);
      if (h->lstm_tc_ok) {
        void* wimg = nullptr;
        CK(cudaMalloc(&wimg, img_bytes(4 * H, H, pl.NC)));
        h->weight_allocs.push_back(wimg);
        h->Whh_img.push_back((uint8_t*)wimg);
        LAUNCH(1, launch_to_image(d_whh_r, H, 4 * H, H, pl.NC, (uint8_t*)wimg, st));
      }
      LstmTc2Plan pl2;
      h->lstm_tc2_ok = lstm_tc2_plan(H, 1, h->sm_count, &pl2);
      if (h->lstm_tc2_ok) {
        void* wimg = nullptr;
        CK(cudaMalloc(&wimg, img_bytes(4 * H, H, 128)));
        h->weight_allocs.push_back(wimg);
        h->Whh_img2.push_back((uint8_t*)wimg);
        LAUNCH(1, launch_to_image(d_whh_r, H, 4 * H, H, 128, (uint8_t*)wimg, st));
      }
    }
  }

  // ---- predictor (models.py:143-187; haste/nbrc.py:134-138) ----
  DecodeWeights& dw = h->dw;
  memset(&dw, 0, sizeof(dw));
  dw.H = H; dw.J = J; dw.V = V; dw.Lp = c.pred_layers; dw.blank = c.blank; dw.bos = c.bos;
  for (int l = 0; l < c.pred_layers; ++l) {
    const std::string p = "predictor.rnn_stack.rnns." + std::to_string(l) + ".";
    NEED(kern, p + "kernel");
    NEED(rk, p + "recurrent_kernel");
    NEED(kb, p + "bias");
    NEED(rb, p + "recurrent_bias");
    NEED(hs, "predictor.rnn_stack.hs." + std::to_string(l));
    float *t_h0, *t_rb, *bs, *bh;
    CK(upload(h, *hs, &t_h0));
    CK(upload(h, interleave(*rb, 3), &t_rb));
    if (bn_fold("predictor.rnn_stack.bns." + std::to_string(l), &bs, &bh)) return RNNT_B200_ERR_STATE;
    dw.h0[l] = t_h0; dw.rbias[l] = t_rb; dw.bn_scale[l] = bs; dw.bn_shift[l] = bh;
    // recurrent_kernel [H(k)][3H gate-major] -> [H(k)][unit*3+gate]
    float *d_rk, *d_t1, *d_t2, *Rt;
    CK(tmp_upload(*rk, &d_rk));
    CK(tmp_alloc((size_t)3 * H * H, &d_t1));
    CK(tmp_alloc((size_t)3 * H * H, &d_t2));
    CK(dalloc(h, (size_t)3 * H * H, &Rt));
    LAUNCH(1, launch_transpose(d_rk, 3 * H, d_t1, H, 3 * H, st));   // [3H][H]
    LAUNCH(1, launch_gather_rows(d_t1, d_t2, perm3, 3 * H, H, st));  // rows interleaved
    LAUNCH(1, launch_transpose(d_t2, H, Rt, 3 * H, H, st));          // [H][3H interleaved]
    dw.Rt[l] = Rt;
    DecodeTcPlan dpl;
    const bool dtc = c.gemm_mode == RNNT_B200_GEMM_TC_FP16X3 && decode_tc_wplan(H, J, V, h->sm_count, &dpl);
    h->dec_tc_ok = dtc;
    if (dtc) {
      void* img = nullptr;
      CK(cudaMalloc(&img, img_bytes((int64_t)dpl.G * dpl.NC_C, H, dpl.NC_C)));
      h->weight_allocs.push_back(img);
      h->R_img[l] = (uint8_t*)img;
      LAUNCH(1, launch_to_image(d_t2, H, 3 * H, H, dpl.NC_C, (uint8_t*)img, st));   // d_t2: [3H interleaved][H]
    }
    h->dec_tc2_ok = c.gemm_mode == RNNT_B200_GEMM_TC_FP16X3 && decode_tc2_plan(H, J, V, c.pred_layers, 1, h->sm_count, c.lm_layers);
    if (h->dec_tc2_ok && l < 2) {
      void* img = nullptr;
      CK(cudaMalloc(&img, img_bytes(3 * H, H, 96)));
      h->weight_allocs.push_back(img);
      h->R_img2[l] = (uint8_t*)img;
      LAUNCH(1, launch_to_image(d_t2, H, 3 * H, H, 96, (uint8_t*)img, st));
    }
    float* d_k;
    CK(tmp_upload(*kern, &d_k));
    if (l == 0) {
      // table0 = (embed * ffn^T + ffn.b) * kernel_0 + bias_0  -> [V][3H] gate-major
      NEED(emb, "predictor.embed.weight");
      float *d_emb, *d_e1 = nullptr, *d_k0t, *d_kb, *table;
      CK(tmp_upload(*emb, &d_emb));
      const std::vector<float>* fw = need("predictor.ffn.weight");
      const std::vector<float>* fbias = need("predictor.ffn.bias");
      if (fw) {
        if (!fbias) return fail(h, RNNT_B200_ERR_STATE, "missing weight: predictor.ffn.bias");
        float *d_fw, *d_fb;
        CK(tmp_upload(*fw, &d_fw));
        CK(tmp_upload(*fbias, &d_fb));
        CK(tmp_alloc((size_t)V * H, &d_e1));
        LAUNCH(1, launch_gemm_nt_f32(d_emb, E, d_fw, E, d_fb, d_e1, H, V, H, E, st));
      } else {
        if (E != H) return fail(h, RNNT_B200_ERR_STATE, "missing weight: predictor.ffn.weight (required when embed_sz != hidden_sz, models.py:160-163)");
        d_e1 = d_emb;
      }
      CK(tmp_alloc((size_t)3 * H * H, &d_k0t));
      CK(tmp_upload(*kb, &d_kb));
      CK(dalloc(h, (size_t)V * 3 * H, &table));
      LAUNCH(1, launch_transpose(d_k, 3 * H, d_k0t, H, 3 * H, st));  // [3H][H]
      LAUNCH(1, launch_gemm_nt_f32(d_e1, H, d_k0t, H, d_kb, table, 3 * H, V, 3 * H, H, st));
      dw.table0 = table;
    } else {
      float *d_a, *d_b, *Kt, *t_kb;
      CK(tmp_alloc((size_t)3 * H * H, &d_a));
      CK(tmp_alloc((size_t)3 * H * H, &d_b));
      CK(dalloc(h, (size_t)3 * H * H, &Kt));
      LAUNCH(1, launch_transpose(d_k, 3 * H, d_a, H, 3 * H, st));
      LAUNCH(1, launch_gather_rows(d_a, d_b, perm3, 3 * H, H, st));
      LAUNCH(1, launch_transpose(d_b, H, Kt, 3 * H, H, st));
      if (dtc) {
        void* img = nullptr;
        CK(cudaMalloc(&img, img_bytes((int64_t)dpl.G * dpl.NC_C, H, dpl.NC_C)));
        h->weight_allocs.push_back(img);
        h->K_img[l] = (uint8_t*)img;
        LAUNCH(1, launch_to_image(d_b, H, 3 * H, H, dpl.NC_C, (uint8_t*)img, st));   // d_b: [3H interleaved][H]
      }
      if (h->dec_tc2_ok && l == 1) {
        void* img = nullptr;
        CK(cudaMalloc(&img, img_bytes(3 * H, H, 96)));
        h->weight_allocs.push_back(img);
        h->K1_img2 = (uint8_t*)img;
        LAUNCH(1, launch_to_image(d_b, H, 3 * H, H, 96, (uint8_t*)img, st));
      }
      CK(upload(h, interleave(*kb, 3), &t_kb));
      dw.Kt[l] = Kt; dw.kbias[l] = t_kb;
    }
  }

  // ---- joint (models.py:116-140, concat) ----
  {
    NEED(w1, "joint.joint.0.weight");
    NEED(b1, "joint.joint.0.bias");
    NEED(w2, "joint.joint.2.weight");
    NEED(b2, "joint.joint.2.bias");
    float *t_b1, *t_b2, *d_w2, *W1p_t, *W1e_t, *W2_t;
    CK(upload(h, *w1, &h->W1));
    CK(upload(h, *b1, &t_b1));
    CK(upload(h, *b2, &t_b2));
    CK(tmp_upload(*w2, &d_w2));
    CK(dalloc(h, (size_t)H * J, &W1p_t));
    CK(dalloc(h, (size_t)H * J, &W1e_t));
    CK(dalloc(h, (size_t)J * V, &W2_t));
    LAUNCH(1, launch_transpose(h->W1, 2 * H, W1p_t, J, H, st));      // pred half: cat((h_pred, h_enc)) -> first H columns
    LAUNCH(1, launch_transpose(h->W1 + H, 2 * H, W1e_t, J, H, st));  // enc half
    LAUNCH(1, launch_transpose(d_w2, J, W2_t, V, J, st));
    dw.W1p_t = W1p_t; dw.W1e_t = W1e_t; dw.b1 = t_b1; dw.W2_t = W2_t; dw.b2 = t_b2;
    if (c.gemm_mode == RNNT_B200_GEMM_TC_FP16X3) {
      void* img = nullptr;
      CK(cudaMalloc(&img, gemm_tc_w_image_bytes(J, H)));
      h->weight_allocs.push_back(img);
      h->W1e_img = (uint8_t*)img;
      LAUNCH(1, launch_to_image(h->W1 + H, 2 * H, J, H, 256, h->W1e_img, st));
      DecodeTcPlan dpl;
      if (h->dec_tc_ok && decode_tc_wplan(H, J, V, h->sm_count, &dpl)) {
        void *ia = nullptr, *ib = nullptr;
        CK(cudaMalloc(&ia, img_bytes((int64_t)dpl.G * dpl.NC_A, H, dpl.NC_A)));
        CK(cudaMalloc(&ib, img_bytes((int64_t)dpl.G * dpl.NC_B, J, dpl.NC_B)));
        h->weight_allocs.push_back(ia);
        h->weight_allocs.push_back(ib);
        h->W1p_img = (uint8_t*)ia;
        h->W2_img = (uint8_t*)ib;
        LAUNCH(1, launch_to_image(h->W1, 2 * H, J, H, dpl.NC_A, h->W1p_img, st));   // pred half: first H columns
        LAUNCH(1, launch_to_image(d_w2, J, V, J, dpl.NC_B, h->W2_img, st));
      }
      if (h->dec_tc2_ok) {
        void *ia = nullptr, *ib = nullptr;
        CK(cudaMalloc(&ia, img_bytes(J, H, 32)));
        CK(cudaMalloc(&ib, img_bytes(V, J, V / 32)));
        h->weight_allocs.push_back(ia);
        h->weight_allocs.push_back(ib);
        h->W1p_img2 = (uint8_t*)ia;
        h->W2_img2 = (uint8_t*)ib;
        LAUNCH(1, launch_to_image(h->W1, 2 * H, J, H, 32, h->W1p_img2, st));
        LAUNCH(1, launch_to_image(d_w2, J, V, J, V / 32, h->W2_img2, st));
      }
    }
  }
  // ---- fused language model (lm.py:20-41): fp32 k-major layouts for the decode loop's tile GEMMs ----
  memset(&h->lmw, 0, sizeof(h->lmw));
  if (c.lm_layers > 0) {
    const int Hl = c.lm_hidden_sz, El = c.lm_embed_sz, Ll = c.lm_layers;
    LmWeights& lw = h->lmw;
    lw.L = Ll; lw.Hl = Hl; lw.alpha = c.lm_alpha; lw.theta = c.lm_theta;
    DecodeTcPlan lpl;
    const bool lm_tc = h->dec_tc_ok && decode_tc_wplan(H, J, V, h->sm_count, &lpl, Ll, Hl);
    h->lm_tc_ok = lm_tc;
    int* lperm4 = nullptr;
    {
      std::vector<int> p4(4 * Hl);
      for (int u = 0; u < Hl; ++u)
        for (int g = 0; g < 4; ++g) p4[u * 4 + g] = g * Hl + u;
      CK(upload(h, p4, &lperm4));
    }
    NEED(lemb, "lm.embed.weight");
    NEED(lwo, "lm.linear.weight");
    NEED(lbo, "lm.linear.bias");
    for (int l = 0; l < Ll; ++l) {
      const std::string sl = std::to_string(l);
      NEED(wih, "lm.rnn.weight_ih_l" + sl);
      NEED(whh, "lm.rnn.weight_hh_l" + sl);
      NEED(bih, "lm.rnn.bias_ih_l" + sl);
      NEED(bhh, "lm.rnn.bias_hh_l" + sl);
      std::vector<float> bsum(4 * Hl);
      for (int i = 0; i < 4 * Hl; ++i) bsum[i] = (*bih)[i] + (*bhh)[i];
      float *d_whh, *d_r, *Rt;
      CK(tmp_upload(*whh, &d_whh));
      CK(tmp_alloc((size_t)4 * Hl * Hl, &d_r));
      CK(dalloc(h, (size_t)4 * Hl * Hl, &Rt));
      LAUNCH(1, launch_gather_rows(d_whh, d_r, lperm4, 4 * Hl, Hl, st));   // rows unit*4+gate
      LAUNCH(1, launch_transpose(d_r, Hl, Rt, 4 * Hl, Hl, st));            // [Hl][4Hl interleaved]
      lw.Rt[l] = Rt;
      if (lm_tc) {
        void* img = nullptr;
        CK(cudaMalloc(&img, img_bytes((int64_t)lpl.G_l * lpl.NC_L, Hl, lpl.NC_L)));
        h->weight_allocs.push_back(img);
        h->lmR_img[l] = (uint8_t*)img;
        LAUNCH(1, launch_to_image(d_r, Hl, 4 * Hl, Hl, lpl.NC_L, (uint8_t*)img, st));   // d_r: [4Hl interleaved][Hl]
      }
      float* d_wih;
      CK(tmp_upload(*wih, &d_wih));
      if (l == 0) {
        // table0 = embed * W_ih0^T + (b_ih0 + b_hh0)  -> [V][4Hl] gate-major (i|f|g|o)
        float *d_emb, *d_b, *table;
        CK(tmp_upload(*lemb, &d_emb));
        CK(tmp_upload(bsum, &d_b));
        CK(dalloc(h, (size_t)V * 4 * Hl, &table));
        LAUNCH(1, launch_gemm_nt_f32(d_emb, El, d_wih, El, d_b, table, 4 * Hl, V, 4 * Hl, El, st));
        lw.table0 = table;
      } else {
        float *d_a, *Wt, *t_b;
        CK(tmp_alloc((size_t)4 * Hl * Hl, &d_a));
        CK(dalloc(h, (size_t)4 * Hl * Hl, &Wt));
        LAUNCH(1, launch_gather_rows(d_wih, d_a, lperm4, 4 * Hl, Hl, st));
        LAUNCH(1, launch_transpose(d_a, Hl, Wt, 4 * Hl, Hl, st));
        if (lm_tc) {
          void* img = nullptr;
          CK(cudaMalloc(&img, img_bytes((int64_t)lpl.G_l * lpl.NC_L, Hl, lpl.NC_L)));
          h->weight_allocs.push_back(img);
          h->lmW_img[l] = (uint8_t*)img;
          LAUNCH(1, launch_to_image(d_a, Hl, 4 * Hl, Hl, lpl.NC_L, (uint8_t*)img, st));
        }
        std::vector<float> bi(4 * Hl);
        for (int u = 0; u < Hl; ++u)
          for (int g = 0; g < 4; ++g) bi[u * 4 + g] = bsum[g * Hl + u];
        CK(upload(h, bi, &t_b));
        lw.Wt[l] = Wt; lw.bias[l] = t_b;
      }
    }
    float *d_wo, *Wo_t, *t_bo;
    CK(tmp_upload(*lwo, &d_wo));
    CK(dalloc(h, (size_t)Hl * V, &Wo_t));
    LAUNCH(1, launch_transpose(d_wo, Hl, Wo_t, V, Hl, st));   // [V][Hl] -> [Hl][V]
    if (lm_tc) {
      void* img = nullptr;
      CK(cudaMalloc(&img, img_bytes((int64_t)lpl.G * lpl.NC_B, Hl, lpl.NC_B)));
      h->weight_allocs.push_back(img);
      h->lmWo_img = (uint8_t*)img;
      LAUNCH(1, launch_to_image(d_wo, Hl, V, Hl, lpl.NC_B, (uint8_t*)img, st));
    }
    CK(upload(h, *lbo, &t_bo));
    lw.Wo_t = Wo_t; lw.bo = t_bo;
  }
#undef NEED
  CK(cudaStreamSynchronize(st));
  for (void* p : tmp) cudaFree(p);
  h->raw.clear();
  h->finalized = true;
  return RNNT_B200_OK;
}

int64_t rnnt_b200_num_frames(rnnt_b200_handle h, int64_t n) { return h ? num_frames(h->cfg, n) : -1; }
int64_t rnnt_b200_num_steps(rnnt_b200_handle h, int64_t n) { return h ? num_steps(h->cfg, n) : -1; }

static int ensure_encode_ws(rnnt_b200_handle h, int B, int T) {
  const rnnt_b200_config& c = h->cfg;
  const size_t M = (size_t)B * T, H = c.hidden_sz, X = (size_t)c.n_mels * c.n_stack, Bp = bp_of(B);
  CK(h->lnx.ensure(M * X * 4));
  CK(h->xp.ensure(M * 4 * H * 4));
  CK(h->ya.ensure(M * H * 4));
  CK(h->yb.ensure(M * H * 4));
  CK(h->ehT[0].ensure(H * Bp * 4));
  CK(h->ehT[1].ensure(H * Bp * 4));
  CK(h->ecT.ensure(H * Bp * 4));
  return 0;
}
static int ensure_decode_ws(rnnt_b200_handle h, int B, int T, int trace_cap) {
  const rnnt_b200_config& c = h->cfg;
  const size_t M = (size_t)B * T, H = c.hidden_sz, J = c.joint_sz, V = c.vocab_sz, Bp = bp_of(B);
  CK(h->ep.ensure(M * J * 4));
  CK(h->dhT.ensure((size_t)c.pred_layers * 2 * H * Bp * 4));
  CK(h->dxT.ensure(2 * H * Bp * 4));
  CK(h->dgT.ensure(H * Bp * 4));
  CK(h->deT.ensure(H * Bp * 4));
  CK(h->dppT.ensure(J * Bp * 4));
  CK(h->dzT.ensure(J * Bp * 4));
  CK(h->dpart.ensure((V / 32) * Bp * 4 * 4));
  CK(h->dlse.ensure(std::max<size_t>((size_t)B * trace_cap, 1) * 4));
  return 0;
}

int32_t rnnt_b200_reserve(rnnt_b200_handle h, int32_t max_batch, int64_t max_samples) {
  if (!h || max_batch < 1 || max_samples < 1) return fail(h, RNNT_B200_ERR_INVALID, "bad reserve() arguments");
  CK(cudaSetDevice(h->cfg.device));
  const rnnt_b200_config& c = h->cfg;
  const int64_t T = std::max<int64_t>(num_steps(c, max_samples), 1);
  const size_t X = (size_t)c.n_mels * c.n_stack;
  CK(h->feats.ensure((size_t)max_batch * T * X * 4));
  if (int r = ensure_encode_ws(h, max_batch, (int)T)) return r;
  if (int r = ensure_decode_ws(h, max_batch, (int)T, 0)) return r;
  CK(h->t_enc.ensure((size_t)max_batch * T * c.hidden_sz * 4));
  CK(h->t_audio.ensure((size_t)max_batch * max_samples * 4));
  CK(h->t_lens.ensure((size_t)max_batch * 4 * 2));
  return RNNT_B200_OK;
}

static int check_ready(rnnt_b200_handle h) {
  if (!h) return RNNT_B200_ERR_INVALID;
  if (!h->finalized) return fail(h, RNNT_B200_ERR_STATE, "finalize() has not been called");
  cudaError_t e = cudaSetDevice(h->cfg.device);
  if (e != cudaSuccess) return fail_cuda(h, e, "cudaSetDevice");
  return 0;
}

int32_t rnnt_b200_features(rnnt_b200_handle h, const float* audio, const int32_t* lens, int32_t B, int64_t n, float* feats,
                           void* stream) {
  if (int r = check_ready(h)) return r;
  const rnnt_b200_config& c = h->cfg;
  if (!audio || !feats || B < 1 || B > 65535) return fail(h, RNNT_B200_ERR_INVALID, "features: bad arguments");
  if (n <= c.n_fft / 2) return fail(h, RNNT_B200_ERR_INVALID, "features: need more than n_fft/2 samples (reflect padding, torch.stft)");
  const int64_t T = num_steps(c, n);
  if (T < 1) return fail(h, RNNT_B200_ERR_INVALID, "features: input shorter than one stacked row");
  FrontendArgs a;
  a.audio = audio; a.n = n; a.lens = lens; a.out = feats; a.T_out = (int)T; a.frame0 = 0; a.is_stream = 0;
  a.n_mels = c.n_mels; a.n_stack = c.n_stack; a.D = c.downsample; a.hop = c.hop_length; a.win = c.win_length;
  a.window = h->window; a.tw = h->tw; a.mel_start = h->mel_start; a.mel_count = h->mel_count; a.mel_off = h->mel_off;
  a.mel_w = h->mel_w; a.log_offset = c.log_offset;
  LAUNCH(1, launch_mel_stack(a, B, (cudaStream_t)stream));
  return RNNT_B200_OK;
}

int32_t rnnt_b200_logmel(rnnt_b200_handle h, const float* audio, const int32_t* lens, int32_t B, int64_t n, float* out,
                         void* stream) {
  if (int r = check_ready(h)) return r;
  const rnnt_b200_config& c = h->cfg;
  if (!audio || !out || B < 1 || B > 65535) return fail(h, RNNT_B200_ERR_INVALID, "logmel: bad arguments");
  if (n <= c.n_fft / 2) return fail(h, RNNT_B200_ERR_INVALID, "logmel: need more than n_fft/2 samples (reflect padding, torch.stft)");
  FrontendArgs a;
  a.audio = audio; a.n = n; a.lens = lens; a.out = out; a.T_out = (int)num_frames(c, n); a.frame0 = 0; a.is_stream = 0;
  a.n_mels = c.n_mels; a.n_stack = 1; a.D = 1; a.hop = c.hop_length; a.win = c.win_length;
  a.window = h->window; a.tw = h->tw; a.mel_start = h->mel_start; a.mel_count = h->mel_count; a.mel_off = h->mel_off;
  a.mel_w = h->mel_w; a.log_offset = c.log_offset;
  LAUNCH(1, launch_mel_stack(a, B, (cudaStream_t)stream));
  return RNNT_B200_OK;
}

int32_t rnnt_b200_features_stream(rnnt_b200_handle h, const float* window, int32_t B, int64_t W, float* feats, void* stream) {
  if (int r = check_ready(h)) return r;
  const rnnt_b200_config& c = h->cfg;
  if (!window || !feats || B < 1 || B > 65535) return fail(h, RNNT_B200_ERR_INVALID, "features_stream: bad arguments");
  const int64_t F = num_frames(c, W);
  const int64_t a0 = F / 3 + 1;  // StreamPostprocess, transforms.py:338-341
  if (W <= c.n_fft / 2 || a0 + c.n_stack > F)
    return fail(h, RNNT_B200_ERR_INVALID, "features_stream: window too short for n_stack frames after the middle-third crop");
  FrontendArgs a;
  a.audio = window; a.n = W; a.lens = nullptr; a.out = feats; a.T_out = 1; a.frame0 = (int)a0; a.is_stream = 1;
  a.n_mels = c.n_mels; a.n_stack = c.n_stack; a.D = c.downsample; a.hop = c.hop_length; a.win = c.win_length;
  a.window = h->window; a.tw = h->tw; a.mel_start = h->mel_start; a.mel_count = h->mel_count; a.mel_off = h->mel_off;
  a.mel_w = h->mel_w; a.log_offset = c.log_offset;
  LAUNCH(1, launch_mel_stack(a, B, (cudaStream_t)stream));
  return RNNT_B200_OK;
}

namespace {
int64_t gcd64(int64_t a, int64_t b) { while (b) { const int64_t t = a % b; a = b; b = t; } return a; }
}

int64_t rnnt_b200_resample_len(rnnt_b200_handle h, int64_t n, int32_t orig_sr) {
  if (!h || n < 0 || orig_sr < 1) return -1;
  const int64_t g = gcd64(orig_sr, h->cfg.sample_rate), o = orig_sr / g, nn = h->cfg.sample_rate / g;
  return (nn * n + o - 1) / o;   // ceil(new * n / orig)
}

int32_t rnnt_b200_resample(rnnt_b200_handle h, const float* audio, int32_t B, int64_t n, int32_t orig_sr, float* out, void* stream) {
  if (!h) return RNNT_B200_ERR_INVALID;
  if (!audio || !out || B < 1 || B > 65535 || n < 1 || orig_sr < 1) return fail(h, RNNT_B200_ERR_INVALID, "resample: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const rnnt_b200_config& c = h->cfg;
  CK(cudaSetDevice(c.device));
  if (orig_sr == c.sample_rate) {
    CK(cudaMemcpyAsync(out, audio, (size_t)B * n * 4, cudaMemcpyDeviceToDevice, st));
    return RNNT_B200_OK;
  }
  auto it = h->resample_tabs.find(orig_sr);
  if (it == h->resample_tabs.end()) {
    // torchaudio.functional._get_sinc_resample_kernel (sinc_interp_hann, lowpass_filter_width = 6, rolloff = 0.99):
    // float64 grid, the phase term -p / new formed in float32, result rounded to float32
    const int64_t g = gcd64(orig_sr, c.sample_rate);
    rnnt_b200_handle_s::ResampleTab t;
    t.o = (int)(orig_sr / g); t.n = (int)(c.sample_rate / g);
    const double lpw = 6.0, base = (double)std::min(t.o, t.n) * 0.99;
    t.width = (int)std::ceil(lpw * t.o / base);
    t.K = 2 * t.width + t.o;
    if ((int64_t)t.n * t.K > (int64_t)64 << 20) return fail(h, RNNT_B200_ERR_UNSUPPORTED, "resample: rate ratio needs an unreasonably large filter bank");
    std::vector<float> tab((size_t)t.n * t.K);
    const double pi = 3.14159265358979323846;
    for (int p = 0; p < t.n; ++p) {
      const double phase = (double)((float)(-p) / (float)t.n);
      for (int k = 0; k < t.K; ++k) {
        double x = (phase + (double)(k - t.width) / (double)t.o) * base;
        x = std::min(std::max(x, -lpw), lpw);
        const double cw = std::cos(x * pi / lpw / 2.0), window = cw * cw;
        x *= pi;
        const double sinc = (x == 0.0) ? 1.0 : std::sin(x) / x;
        tab[(size_t)p * t.K + k] = (float)(sinc * window * (base / (double)t.o));
      }
    }
    CK(upload(h, tab, &t.dev));
    it = h->resample_tabs.emplace(orig_sr, t).first;
  }
  const auto& t = it->second;
  const int64_t L = rnnt_b200_resample_len(h, n, orig_sr);
  LAUNCH(1, launch_resample(audio, B, n, t.dev, t.o, t.n, t.width, t.K, out, L, st));
  return RNNT_B200_OK;
}

// Recurrent kernels of the encoder and the decode loop: the fp32 kernels (lstm.cu / decode.cu), the round-1 persistent
// tcgen05 kernels (lstm_tc.cu / decode_tc.cu) and the cluster split-K kernels (lstm_tc2.cu / decode_tc2.cu).
enum class RecKernel { Fp32, Tc, Tc2 };

struct EncoderRoute {
  RecKernel kernel;
  int rows;          // rows per launch: a call with more rows runs as consecutive sub-batches
  LstmTcPlan tc;     // plan of a launch of `rows` rows (kernel Tc)
  LstmTc2Plan tc2;   // ... (kernel Tc2)
};

// The encoder's kernel for a call of B rows.  Stateless batches beyond 32 rows run as 32-row sub-batches of the cluster
// kernel (measured on a B200: 64 utterances 50.0k x real time vs 44.6k in one 64-row launch of the round-1 kernel, 256
// utterances equal); streaming ticks (T = 2, carried state) are faster in one wide launch of the round-1 kernel (8.7k vs 8.0k x).
static EncoderRoute route_encoder(rnnt_b200_handle h, int B, bool stateful) {
  EncoderRoute r = {};
  r.kernel = RecKernel::Fp32;
  r.rows = B;
  if (h->cfg.gemm_mode != RNNT_B200_GEMM_TC_FP16X3) return r;
  const int H = h->cfg.hidden_sz;
  const int cap = (!stateful && h->lstm_tc2_ok) ? 32 : 128;
  if (h->lstm_tc_ok && B > cap) r.rows = cap;   // (without the round-1 kernel a call is never split: one launch of the fp32 kernel)
  if (h->lstm_tc2_ok && lstm_tc2_plan(H, r.rows, h->sm_count, &r.tc2)) r.kernel = RecKernel::Tc2;
  else if (h->lstm_tc_ok && lstm_tc_plan(H, r.rows, h->sm_count, &r.tc)) r.kernel = RecKernel::Tc;
  return r;
}

// RNNT_LSTM_DBG: per-step phase times of CTA 0, the publish skew over all CTAs and CTA 0's cycle breakdown of one
// cluster-kernel layer, on stderr (tuning aid: synchronises the stream; frees the stamp buffers)
static int32_t report_lstm_stamps(rnnt_b200_handle h, const LstmTc2Args& a, int grid, cudaStream_t st) {
  const int B = a.B, T = a.T;
  std::vector<unsigned long long> ha((size_t)grid * T * 2), hb((size_t)T * 4 + 16);
  CK(cudaStreamSynchronize(st));
  CK(cudaMemcpy(ha.data(), a.dbg_all, ha.size() * 8, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hb.data(), a.dbg, (size_t)T * 32 + 128, cudaMemcpyDeviceToHost));
  cudaFree(a.dbg_all);
  cudaFree(a.dbg);
  double sp_pub = 0, sp_red = 0, first_to_last = 0;
  for (int t = 1; t < T; ++t) {
    unsigned long long mn = ~0ull, mx = 0, mn2 = ~0ull, mx2 = 0;
    for (int c2 = 0; c2 < grid; ++c2) {
      const unsigned long long a0 = ha[((size_t)c2 * T + t) * 2], a1 = ha[((size_t)c2 * T + t) * 2 + 1];
      mn = std::min(mn, a0); mx = std::max(mx, a0); mn2 = std::min(mn2, a1); mx2 = std::max(mx2, a1);
    }
    sp_pub += (double)(mx - mn); sp_red += (double)(mx2 - mn2);
    unsigned long long pm = 0;
    for (int c2 = 0; c2 < grid; ++c2) pm = std::max(pm, ha[((size_t)c2 * T + t - 1) * 2]);
    first_to_last += (double)(mn2 - pm);   // last publish of step t-1 -> first CTA with complete tiles at step t
  }
  fprintf(stderr, "[lstm_tc2 skew] avg ns over %d CTAs: spread of publish times %.0f | spread of tiles-complete times %.0f | last publish(t-1) -> first tiles-complete(t) %.0f\n",
          grid, sp_pub / (T - 1), sp_red / (T - 1), first_to_last / (T - 1));
  fprintf(stderr, "[lstm_tc2 epilogue cycles/step, CTA 0 thread 0] wait accumulators %.0f | TMEM drain %.0f | scatter issue %.0f | wait tiles %.0f | tile sums %.0f | cell %.0f | publish %.0f | BN outputs %.0f\n",
          (double)hb[(size_t)T * 4 + 0] / T, (double)hb[(size_t)T * 4 + 1] / T, (double)hb[(size_t)T * 4 + 2] / T, (double)hb[(size_t)T * 4 + 3] / T,
          (double)hb[(size_t)T * 4 + 4] / T, (double)hb[(size_t)T * 4 + 5] / T, (double)hb[(size_t)T * 4 + 6] / T, (double)hb[(size_t)T * 4 + 7] / T);
  fprintf(stderr, "[lstm_tc2 loader cycles/step, CTA 0 thread 0] first chunk visible %.0f | k-block 0 valid %.0f | k-blocks 1-3 valid %.0f | stores+fence+arrive %.0f\n",
          (double)hb[(size_t)T * 4 + 8] / T, (double)hb[(size_t)T * 4 + 9] / T, (double)hb[(size_t)T * 4 + 10] / T, (double)hb[(size_t)T * 4 + 11] / T);
  double ld = 0, mma = 0, red = 0, fin = 0;
  for (int t = 1; t < T; ++t) {
    ld += (double)(hb[t * 4 + 0] - hb[(t - 1) * 4 + 3]);   // previous publish -> K slice of h landed in smem
    mma += (double)(hb[t * 4 + 1] - hb[t * 4 + 0]);        // -> accumulators ready
    red += (double)(hb[t * 4 + 2] - hb[t * 4 + 1]);        // TMEM drain + DSMEM scatter + partial tiles complete
    fin += (double)(hb[t * 4 + 3] - hb[t * 4 + 2]);        // cell + publish
  }
  fprintf(stderr, "[lstm_tc2 dbg] B=%d T=%d steps avg ns: publish->h landed %.0f | ->tmem_full %.0f | drain+reduce %.0f | cell+publish %.0f | total/step %.0f\n",
          B, T, ld / (T - 1), mma / (T - 1), red / (T - 1), fin / (T - 1), (double)(hb[(T - 1) * 4 + 3] - hb[3]) / (T - 1));
  return RNNT_B200_OK;
}

static int32_t encode_impl(rnnt_b200_handle h, const float* feats, const int32_t* lens_T, int32_t B, int32_t T, float* state_h,
                           float* state_c, int32_t use_state_in, float* enc_out, void* stream, int state_ld);

int32_t rnnt_b200_encode(rnnt_b200_handle h, const float* feats, const int32_t* lens_T, int32_t B, int32_t T, float* state_h,
                         float* state_c, int32_t use_state_in, float* enc_out, void* stream) {
  return encode_impl(h, feats, lens_T, B, T, state_h, state_c, use_state_in, enc_out, stream, B);
}

// state_ld: batch stride of state_h / state_c per layer ([L][state_ld][H]); = B for a whole call, the full stream count for a
// sub-batch of a stateful call (whose rows come first from the pointers passed)
static int32_t encode_impl(rnnt_b200_handle h, const float* feats, const int32_t* lens_T, int32_t B, int32_t T, float* state_h,
                           float* state_c, int32_t use_state_in, float* enc_out, void* stream, int state_ld) {
  if (int r = check_ready(h)) return r;
  const rnnt_b200_config& c = h->cfg;
  if (!feats || !enc_out || B < 1 || T < 1) return fail(h, RNNT_B200_ERR_INVALID, "encode: bad arguments");
  if (use_state_in && (!state_h || !state_c)) return fail(h, RNNT_B200_ERR_INVALID, "encode: use_state_in needs state_h and state_c");
  if ((state_h == nullptr) != (state_c == nullptr)) return fail(h, RNNT_B200_ERR_INVALID, "encode: state_h and state_c must both be given");
  cudaStream_t st = (cudaStream_t)stream;
  const int H = c.hidden_sz, X = c.n_mels * c.n_stack, Bp = bp_of(B);
  const EncoderRoute rt = route_encoder(h, B, state_h != nullptr);
  if (B > rt.rows) {
    // independent utterances / streams: the state [L][state_ld][H] is sliced by rows (every layer passes its own base pointer
    // to the kernel).  Each sub-batch routes again at its own size, so a short last one may take another kernel.
    for (int b0 = 0; b0 < B; b0 += rt.rows) {
      const int nb = std::min(rt.rows, B - b0);
      const int r = encode_impl(h, feats + (size_t)b0 * T * X, lens_T ? lens_T + b0 : nullptr, nb, T,
                                state_h ? state_h + (size_t)b0 * H : nullptr, state_c ? state_c + (size_t)b0 * H : nullptr, use_state_in,
                                enc_out + (size_t)b0 * T * H, stream, state_ld);
      if (r) return r;
    }
    return RNNT_B200_OK;
  }
  const int64_t M = (int64_t)B * T;
  if (int r = ensure_encode_ws(h, B, T)) return r;
  if (h->ev) cudaEventRecord(h->ev[0], st);
  LAUNCH(1, launch_layernorm(feats, h->lnx.as<float>(), h->ln_g, h->ln_b, M, X, c.ln_eps, st));
  for (int l = 0; l < c.enc_layers; ++l) {
    const EncLayer& L = h->enc[l];
    const float* A = l == 0 ? h->lnx.as<float>() : ((l - 1) & 1 ? h->yb.as<float>() : h->ya.as<float>());
    float* y = (l == c.enc_layers - 1) ? enc_out : (l & 1 ? h->yb.as<float>() : h->ya.as<float>());
    if (h->ev) cudaEventRecord(h->ev[6 + 2 * l], st);
    if (c.gemm_mode == RNNT_B200_GEMM_TC_FP16X3) {
      CK(h->a_img.ensure(gemm_tc_a_image_bytes(M, std::max(L.in, H))));
      // layer 0 reads the LayerNorm output; deeper layers find their operand image already written
      // by the previous layer's recurrent kernel (when that ran on the tensor-core path)
      if (l == 0 || rt.kernel == RecKernel::Fp32) LAUNCH(1, launch_to_image(A, L.in, M, L.in, 128, h->a_img.as<uint8_t>(), st));
      LAUNCH(1, launch_gemm_tc(h->a_img.as<uint8_t>(), h->Wih_img[l], L.bias_r, h->xp.as<float>(), 4 * H, M, 4 * H, L.in, st));
    } else {
      LAUNCH(1, launch_gemm_nt_f32(A, L.in, L.Wih_r, L.in, L.bias_r, h->xp.as<float>(), 4 * H, M, 4 * H, L.in, st));
    }
    if (h->ev) cudaEventRecord(h->ev[7 + 2 * l], st);
    if (rt.kernel == RecKernel::Tc2) {
      // cluster split-K kernel (lstm_tc2.cu): 4x less operand ingest per step, tagged h exchange
      CK(h->x_img[0].ensure(img_bytes(128, H, 128)));
      CK(h->x_img[1].ensure(img_bytes(128, H, 128)));
      CK(h->gbar.ensure(1024));
      CK(cudaMemsetAsync(h->gbar.p, 0, 4, st));
      LstmTc2Args a;
      memset(&a, 0, sizeof(a));
      a.w_img = h->Whh_img2[l];
      a.x_img[0] = h->x_img[0].as<uint8_t>(); a.x_img[1] = h->x_img[1].as<uint8_t>();
      a.xp = h->xp.as<float>(); a.bn_scale = L.bn_scale; a.bn_shift = L.bn_shift;
      a.y = y; a.y_img = (l == c.enc_layers - 1) ? nullptr : h->a_img.as<uint8_t>();
      a.lens_T = lens_T; a.h_init_vec = L.h0; a.c_init_vec = L.c0;
      a.state_h_in = use_state_in ? state_h + (size_t)l * state_ld * H : nullptr;
      a.state_c_in = use_state_in ? state_c + (size_t)l * state_ld * H : nullptr;
      a.state_h_out = state_h ? state_h + (size_t)l * state_ld * H : nullptr;
      a.state_c_out = state_c ? state_c + (size_t)l * state_ld * H : nullptr;
      a.barrier = h->gbar.as<unsigned int>();
      a.T = T; a.B = B; a.H = H;
      static const bool stamps = getenv("RNNT_LSTM_DBG") != nullptr;
      if (stamps && l == 0) {
        CK(cudaMalloc((void**)&a.dbg, (size_t)T * 32 + 128));
        CK(cudaMemset(a.dbg, 0, (size_t)T * 32 + 128));
        CK(cudaMalloc((void**)&a.dbg_all, (size_t)rt.tc2.grid * T * 16));
        CK(cudaMemset(a.dbg_all, 0, (size_t)rt.tc2.grid * T * 16));
      }
      LAUNCH(1, launch_lstm_layer_tc2(a, rt.tc2, st));
      if (a.dbg)
        if (int r = report_lstm_stamps(h, a, rt.tc2.grid, st)) return r;
      continue;
    }
    if (rt.kernel == RecKernel::Tc) {
      const size_t ximg = img_bytes(128, H, 128);
      CK(h->x_img[0].ensure(ximg));
      CK(h->x_img[1].ensure(ximg));
      CK(h->gbar.ensure(1024));
      CK(cudaMemsetAsync(h->gbar.p, 0, (size_t)(H / 64) * 4, st));
      LstmTcArgs a;
      memset(&a, 0, sizeof(a));
      a.w_img = h->Whh_img[l];
      a.x_img[0] = h->x_img[0].as<uint8_t>(); a.x_img[1] = h->x_img[1].as<uint8_t>();
      a.xp = h->xp.as<float>(); a.bn_scale = L.bn_scale; a.bn_shift = L.bn_shift;
      a.y = y; a.y_img = (l == c.enc_layers - 1) ? nullptr : h->a_img.as<uint8_t>();
      a.lens_T = lens_T; a.h_init_vec = L.h0; a.c_init_vec = L.c0;
      a.state_h_in = use_state_in ? state_h + (size_t)l * state_ld * H : nullptr;
      a.state_c_in = use_state_in ? state_c + (size_t)l * state_ld * H : nullptr;
      a.state_h_out = state_h ? state_h + (size_t)l * state_ld * H : nullptr;
      a.state_c_out = state_c ? state_c + (size_t)l * state_ld * H : nullptr;
      a.barrier = h->gbar.as<unsigned int>();
      a.T = T; a.B = B; a.H = H;
      LAUNCH(1, launch_lstm_layer_tc(a, rt.tc, st));
      continue;
    }
    if (use_state_in) {
      LAUNCH(1, launch_state_to_T(state_h + (size_t)l * state_ld * H, h->ehT[0].as<float>(), B, Bp, H, st));
      LAUNCH(1, launch_state_to_T(state_c + (size_t)l * state_ld * H, h->ecT.as<float>(), B, Bp, H, st));
    } else {
      LAUNCH(1, launch_state_broadcast_T(L.h0, h->ehT[0].as<float>(), B, Bp, H, st));
      LAUNCH(1, launch_state_broadcast_T(L.c0, h->ecT.as<float>(), B, Bp, H, st));
    }
    LstmStepArgs a;
    a.Whh_t = L.Whh_t; a.cT = h->ecT.as<float>(); a.xp = h->xp.as<float>(); a.bn_scale = L.bn_scale; a.bn_shift = L.bn_shift;
    a.y = y; a.lens_T = lens_T; a.T = T; a.B = B; a.Bp = Bp; a.H = H;
    for (int t = 0; t < T; ++t) {
      a.t = t;
      a.hT_in = h->ehT[t & 1].as<float>();
      a.hT_out = h->ehT[(t + 1) & 1].as<float>();
      LAUNCH(1, launch_lstm_step(a, st));
    }
    if (state_h) {
      LAUNCH(1, launch_state_from_T(h->ehT[T & 1].as<float>(), state_h + (size_t)l * state_ld * H, B, Bp, H, st));
      LAUNCH(1, launch_state_from_T(h->ecT.as<float>(), state_c + (size_t)l * state_ld * H, B, Bp, H, st));
    }
  }
  if (h->ev) cudaEventRecord(h->ev[1], st);
  return RNNT_B200_OK;
}

int32_t rnnt_b200_predict(rnnt_b200_handle h, const int32_t* tokens, int32_t B, float* state_h, int32_t use_state_in,
                          float* out, void* stream) {
  if (int r = check_ready(h)) return r;
  const rnnt_b200_config& c = h->cfg;
  if (!tokens || !state_h || !out || B < 1 || B > kDecodeMaxBatch)
    return fail(h, RNNT_B200_ERR_INVALID, "predict: bad arguments (1 <= B <= 256, state_h and out required)");
  cudaStream_t st = (cudaStream_t)stream;
  const int H = c.hidden_sz, Bp = bp_of(B);
  if (int r = ensure_decode_ws(h, B, 1, 0)) return r;
  const size_t hb = (size_t)H * Bp;
  float* dh = h->dhT.as<float>();
  for (int l = 0; l < c.pred_layers; ++l) {
    float* in = dh + (size_t)(2 * l) * hb;
    float* outb = dh + (size_t)(2 * l + 1) * hb;
    if (use_state_in) LAUNCH(1, launch_state_to_T(state_h + (size_t)l * B * H, in, B, Bp, H, st));
    else LAUNCH(1, launch_state_broadcast_T(h->dw.h0[l], in, B, Bp, H, st));
    PredictArgs a;
    a.w = h->dw; a.tokens = tokens; a.B = B; a.Bp = Bp; a.layer = l; a.hT_in = in; a.hT_out = outb;
    a.xT_in = l == 0 ? nullptr : h->dxT.as<float>() + (size_t)((l - 1) & 1) * hb;
    a.xT_out = (l == c.pred_layers - 1) ? h->dgT.as<float>() : h->dxT.as<float>() + (size_t)(l & 1) * hb;
    LAUNCH(1, launch_gru_layer(a, st));
    LAUNCH(1, launch_state_from_T(outb, state_h + (size_t)l * B * H, B, Bp, H, st));
  }
  LAUNCH(1, launch_state_from_T(h->dgT.as<float>(), out, B, Bp, H, st));
  return RNNT_B200_OK;
}

int32_t rnnt_b200_joint(rnnt_b200_handle h, const float* h_pred, const float* h_enc, int32_t B, float* logits, void* stream) {
  if (int r = check_ready(h)) return r;
  const rnnt_b200_config& c = h->cfg;
  if (!h_pred || !h_enc || !logits || B < 1) return fail(h, RNNT_B200_ERR_INVALID, "joint: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int H = c.hidden_sz, Bp = bp_of(B);
  if (int r = ensure_decode_ws(h, B, 1, 0)) return r;
  LAUNCH(1, launch_state_to_T(h_pred, h->dgT.as<float>(), B, Bp, H, st));
  LAUNCH(1, launch_state_to_T(h_enc, h->deT.as<float>(), B, Bp, H, st));
  JointArgs a;
  a.w = h->dw; a.B = B; a.Bp = Bp; a.gT = h->dgT.as<float>(); a.eT = h->deT.as<float>(); a.zT = h->dzT.as<float>();
  a.logits = logits;
  LAUNCH(2, launch_joint(a, st));
  return RNNT_B200_OK;
}

struct DecoderRoute {
  RecKernel kernel;
  int rows;          // rows per launch: a call with more rows runs as consecutive sub-batches
  DecodeTcPlan tc;   // plan of a launch of min(B, rows) rows (kernel Tc)
};

// The decode loop's kernel for a call of B rows; stateful: the call carries predictor state or a registered LM state.  The
// round-1 kernel takes up to 64 utterances; the cluster kernel 32, and stateless calls beyond that run as 32-row sub-batches
// of it (same policy as the encoder, see route_encoder).  With a fused language model the loop runs in the round-1 kernel
// where its LM phases fit the shape, else in the fp32 cooperative kernel (decode.cu), whatever gemm_mode says.
static DecoderRoute route_decoder(rnnt_b200_handle h, int B, bool stateful) {
  const rnnt_b200_config& c = h->cfg;
  DecoderRoute r = {};
  r.kernel = RecKernel::Fp32;
  r.rows = kDecodeMaxBatch;
  const bool tc = c.gemm_mode == RNNT_B200_GEMM_TC_FP16X3 && h->dec_tc_ok && (c.lm_layers == 0 || h->lm_tc_ok);
  if (tc) {
    r.rows = 64;
    if (!stateful && h->dec_tc2_ok) r.rows = 32;   // (only where the round-1 kernel is usable too)
  }
  // The predictor state [Lp][state_ld][H] / [B][H] is sliceable by rows (the kernels take the layer stride), the fused LM's
  // feature-major state blob is not: with a registered LM blob the call runs in one launch, whatever its size.
  if (h->lm_blob) r.rows = std::max(r.rows, B);
  const int n = std::min(B, r.rows);
  if (h->dec_tc2_ok && !h->lm_blob && decode_tc2_plan(c.hidden_sz, c.joint_sz, c.vocab_sz, c.pred_layers, n, h->sm_count, c.lm_layers)) {
    r.kernel = RecKernel::Tc2;
  } else if (tc) {
    if (decode_tc_plan(c.hidden_sz, c.joint_sz, c.vocab_sz, c.pred_layers, n, h->sm_count, &r.tc, c.lm_layers, c.lm_hidden_sz)) {
      r.kernel = RecKernel::Tc;
    } else if (!stateful && n > 32 &&
               decode_tc_plan(c.hidden_sz, c.joint_sz, c.vocab_sz, c.pred_layers, 32, h->sm_count, &r.tc, c.lm_layers, c.lm_hidden_sz)) {
      // some shapes (e.g. H = 1536: 12 vocabulary rows per epilogue thread at 64) only plan for 32, which still beats the
      // fp32 kernel
      r.kernel = RecKernel::Tc;
      r.rows = 32;
    }
  }
  return r;
}

// RNNT_DEC_DBG: mean time of each segment of the cluster decode kernel's lock-step, from CTA 0's (time, tag) trail, on
// stderr (tuning aid: synchronises the stream; frees the trail)
static int32_t report_decode_stamps(rnnt_b200_handle h, const DecodeTc2Args& t, cudaStream_t st) {
  const int dcap = t.dbg_cap;
  std::vector<unsigned long long> hb((size_t)dcap * 2);
  CK(cudaStreamSynchronize(st));
  CK(cudaMemcpy(hb.data(), t.dbg, (size_t)dcap * 16, cudaMemcpyDeviceToHost));
  cudaFree(t.dbg);
  double sum[8] = {0}; int cnt[8] = {0}; int n = 0;
  for (int i = 1; i < dcap && hb[2 * i]; ++i, ++n) {
    const int tag = (int)hb[2 * i + 1];
    if (tag < 8) { sum[tag] += (double)(hb[2 * i] - hb[2 * i - 2]); cnt[tag]++; }
  }
  fprintf(stderr, "[decode_tc2 dbg] B=%d stamps=%d avg ns per segment: ->z published %.0f (n=%d) | ->keys published %.0f | ->table reduced %.0f | rule %.0f | C0 %.0f (n=%d) | C1 %.0f | total %.0f us over %d steps\n",
          t.B, n, cnt[0] ? sum[0] / cnt[0] : 0, cnt[0], cnt[1] ? sum[1] / cnt[1] : 0, cnt[2] ? sum[2] / cnt[2] : 0,
          cnt[3] ? sum[3] / cnt[3] : 0, cnt[4] ? sum[4] / cnt[4] : 0, cnt[4], cnt[5] ? sum[5] / cnt[5] : 0,
          n > 1 ? (double)(hb[2 * n] - hb[2]) / 1e3 : 0.0, cnt[3]);
  return RNNT_B200_OK;
}

static int32_t decode_greedy_impl(rnnt_b200_handle h, const float* enc, const int32_t* lens_T, int32_t B, int32_t T,
                                  int32_t max_iters, float* pred_state_h, float* pred_out, int32_t use_state_in,
                                  int32_t* tokens_out, int32_t U_cap, int32_t* ntok_out, double* neg_logp_out,
                                  uint8_t* iters_out, float* trace_logp, int32_t trace_cap, void* stream, int state_ld);

int32_t rnnt_b200_decode_greedy(rnnt_b200_handle h, const float* enc, const int32_t* lens_T, int32_t B, int32_t T,
                                int32_t max_iters, float* pred_state_h, float* pred_out, int32_t use_state_in,
                                int32_t* tokens_out, int32_t U_cap, int32_t* ntok_out, double* neg_logp_out,
                                uint8_t* iters_out, float* trace_logp, int32_t trace_cap, void* stream) {
  return decode_greedy_impl(h, enc, lens_T, B, T, max_iters, pred_state_h, pred_out, use_state_in, tokens_out, U_cap, ntok_out, neg_logp_out,
                            iters_out, trace_logp, trace_cap, stream, B);
}

// state_ld: batch stride of pred_state_h per layer ([Lp][state_ld][H]); = B for a whole call, the full stream count when this call
// is a sub-batch of a stateful call (the rows of the sub-batch come first from the pointer passed)
static int32_t decode_greedy_impl(rnnt_b200_handle h, const float* enc, const int32_t* lens_T, int32_t B, int32_t T,
                                  int32_t max_iters, float* pred_state_h, float* pred_out, int32_t use_state_in,
                                  int32_t* tokens_out, int32_t U_cap, int32_t* ntok_out, double* neg_logp_out,
                                  uint8_t* iters_out, float* trace_logp, int32_t trace_cap, void* stream, int state_ld) {
  if (int r = check_ready(h)) return r;
  const rnnt_b200_config& c = h->cfg;
  if (!enc || !tokens_out || !ntok_out || B < 1 || T < 1 || max_iters < 1 || max_iters > 255)
    return fail(h, RNNT_B200_ERR_INVALID, "decode_greedy: bad arguments");
  if ((int64_t)U_cap < (int64_t)max_iters * T) return fail(h, RNNT_B200_ERR_INVALID, "decode_greedy: U_cap < max_iters*T");
  const bool stateful = pred_state_h || pred_out || use_state_in || h->lm_blob;
  if (stateful && B > kDecodeMaxBatch)
    return fail(h, RNNT_B200_ERR_INVALID, "decode_greedy: stateful calls are limited to " + std::to_string(kDecodeMaxBatch) + " streams per call");
  const DecoderRoute rt = route_decoder(h, B, stateful);
  if (B > rt.rows) {
    // utterances / streams are independent; each sub-batch routes again at its own size
    const int H0 = c.hidden_sz;
    for (int b0 = 0; b0 < B; b0 += rt.rows) {
      const int nb = std::min(rt.rows, B - b0);
      const int r = decode_greedy_impl(h, enc + (size_t)b0 * T * H0, lens_T ? lens_T + b0 : nullptr, nb, T, max_iters,
                                       pred_state_h ? pred_state_h + (size_t)b0 * H0 : nullptr, pred_out ? pred_out + (size_t)b0 * H0 : nullptr,
                                       use_state_in, tokens_out + (size_t)b0 * U_cap, U_cap, ntok_out + b0,
                                       neg_logp_out ? neg_logp_out + b0 : nullptr, iters_out ? iters_out + (size_t)b0 * T : nullptr,
                                       trace_logp ? trace_logp + (size_t)b0 * trace_cap * c.vocab_sz : nullptr, trace_cap, stream, state_ld);
      if (r) return r;
    }
    return RNNT_B200_OK;
  }
  if (use_state_in && (!pred_state_h || !pred_out)) return fail(h, RNNT_B200_ERR_INVALID, "decode_greedy: use_state_in needs pred_state_h and pred_out");
  if (trace_logp && trace_cap < 1) return fail(h, RNNT_B200_ERR_INVALID, "decode_greedy: trace_cap < 1");
  cudaStream_t st = (cudaStream_t)stream;
  const int H = c.hidden_sz, J = c.joint_sz, Bp = bp_of(B);
  const int64_t M = (int64_t)B * T;
  if (int r = ensure_decode_ws(h, B, T, trace_logp ? trace_cap : 0)) return r;
  if (h->ev) cudaEventRecord(h->ev[2], st);
  // hoisted encoder half of the joint's first Linear (incl. its bias): ep = enc * W1[:, H:]^T + b1
  if (c.gemm_mode == RNNT_B200_GEMM_TC_FP16X3) {
    CK(h->a_img.ensure(gemm_tc_a_image_bytes(M, H)));
    LAUNCH(1, launch_to_image(enc, H, M, H, 128, h->a_img.as<uint8_t>(), st));
    LAUNCH(1, launch_gemm_tc(h->a_img.as<uint8_t>(), h->W1e_img, h->dw.b1, h->ep.as<float>(), J, M, J, H, st));
  } else {
    LAUNCH(1, launch_gemm_nt_f32(enc, H, h->W1 + H, 2 * H, h->dw.b1, h->ep.as<float>(), J, M, J, H, st));
  }
  if (h->ev) cudaEventRecord(h->ev[3], st);
  if (rt.kernel == RecKernel::Tc2) {
    // cluster split-K decode (decode_tc2.cu): up to 32 utterances per launch
    const size_t one = decode_tc2_image_bytes();
    const int nimg = decode_tc2_images();
    CK(h->dimg.ensure(one * 2 * nimg));
    const int max_steps = max_iters * T + 2;
    const int nBp = decode_tc2_part_ctas();
    CK(h->dpart.ensure((size_t)max_steps * nBp * 32 * 8));
    CK(h->dkeys.ensure(decode_tc2_keys_bytes() + (size_t)B * 4 + 64));
    CK(h->dlse.ensure(std::max<size_t>((size_t)B * (trace_logp ? trace_cap : 1), 1) * 4));
    CK(h->gbar.ensure(1024));
    CK(cudaMemsetAsync(h->gbar.p, 0, 4, st));
    if (trace_logp) {
      CK(cudaMemsetAsync(h->dlse.p, 0, (size_t)B * trace_cap * 4, st));
      CK(cudaMemsetAsync(trace_logp, 0, (size_t)B * trace_cap * c.vocab_sz * 4, st));
    }
    if (iters_out) CK(cudaMemsetAsync(iters_out, 0, (size_t)B * T, st));
    DecodeTc2Args t;
    memset(&t, 0, sizeof(t));
    t.w = h->dw;
    t.w1p_img = h->W1p_img2; t.w2_img = h->W2_img2; t.k1_img = h->K1_img2; t.r_img[0] = h->R_img2[0]; t.r_img[1] = h->R_img2[1];
    for (int i = 0; i < nimg; ++i) t.img[i] = h->dimg.as<uint8_t>() + (size_t)(2 * i) * one;
    t.img_stride = one;
    t.keys = h->dkeys.as<unsigned long long>();
    t.n_eval = reinterpret_cast<int*>(h->dkeys.as<uint8_t>() + decode_tc2_keys_bytes());
    t.ep = h->ep.as<float>(); t.lens_T = lens_T; t.B = B; t.T = T; t.max_iters = max_iters; t.use_state_in = use_state_in;
    t.part = h->dpart.as<float>(); t.trace_lse = h->dlse.as<float>(); t.max_steps = max_steps;
    t.state_h = pred_state_h; t.pred_out = pred_out; t.state_ld = state_ld;
    t.tokens = tokens_out; t.U_cap = U_cap; t.ntok = ntok_out; t.neg_logp = neg_logp_out; t.iters = iters_out;
    t.trace = trace_logp; t.trace_cap = trace_logp ? trace_cap : 0;
    t.barrier = h->gbar.as<unsigned int>();
    static const bool stamps = getenv("RNNT_DEC_DBG") != nullptr;
    if (stamps) {
      t.dbg_cap = 8192;
      CK(cudaMalloc((void**)&t.dbg, (size_t)t.dbg_cap * 16));
      CK(cudaMemset(t.dbg, 0, (size_t)t.dbg_cap * 16));
    }
    LAUNCH(trace_logp ? 3 : 2, launch_decode_tc2(t, st));
    if (t.dbg)
      if (int r = report_decode_stamps(h, t, st)) return r;
    if (h->ev) cudaEventRecord(h->ev[4], st);
    return RNNT_B200_OK;
  }
  if (rt.kernel == RecKernel::Tc) {
    const DecodeTcPlan& dpl = rt.tc;
    const size_t one = (size_t)(std::max(H, J) / 64) * 2 * dpl.Bpad8 * 128;
    const int nimg = 4 + 2 * c.pred_layers;
    CK(h->dimg.ensure(one * nimg));
    const int max_steps = max_iters * T + 2;
    const int nBp = (int)ceil_div(c.vocab_sz, dpl.NC_B);
    CK(h->dpart.ensure((size_t)max_steps * nBp * dpl.Bq * 8));
    CK(h->dkeys.ensure((size_t)max_steps * dpl.Bq * 8 + (size_t)B * 4 + 64));
    CK(cudaMemsetAsync(h->dkeys.p, 0, (size_t)max_steps * dpl.Bq * 8, st));
    CK(h->dlse.ensure(std::max<size_t>((size_t)B * (trace_logp ? trace_cap : 1), 1) * 4));
    CK(h->gbar.ensure(1024));
    CK(cudaMemsetAsync(h->gbar.p, 0, 4, st));
    if (trace_logp) {
      CK(cudaMemsetAsync(h->dlse.p, 0, (size_t)B * trace_cap * 4, st));
      CK(cudaMemsetAsync(trace_logp, 0, (size_t)B * trace_cap * c.vocab_sz * 4, st));
    }
    if (iters_out) CK(cudaMemsetAsync(iters_out, 0, (size_t)B * T, st));
    DecodeTcArgs t;
    memset(&t, 0, sizeof(t));
    t.w = h->dw;
    t.w1p_img = h->W1p_img; t.w2_img = h->W2_img;
    uint8_t* ib = h->dimg.as<uint8_t>();
    t.g_img = ib; t.z_img = ib + one; t.x_img[0] = ib + 2 * one; t.x_img[1] = ib + 3 * one;
    for (int l = 0; l < c.pred_layers; ++l) {
      t.r_img[l] = h->R_img[l]; t.k_img[l] = h->K_img[l];
      t.h_img[l][0] = ib + (4 + 2 * l) * one; t.h_img[l][1] = ib + (5 + 2 * l) * one;
    }
    t.ep = h->ep.as<float>(); t.lens_T = lens_T; t.B = B; t.T = T; t.max_iters = max_iters; t.use_state_in = use_state_in;
    t.part = h->dpart.as<float>(); t.trace_lse = h->dlse.as<float>();
    t.keys = h->dkeys.as<unsigned long long>();
    t.n_eval = reinterpret_cast<int*>(h->dkeys.as<uint8_t>() + (size_t)max_steps * dpl.Bq * 8);
    t.max_steps = max_steps;
    t.state_h = pred_state_h; t.pred_out = pred_out; t.state_ld = state_ld;
    t.tokens = tokens_out; t.U_cap = U_cap; t.ntok = ntok_out; t.neg_logp = neg_logp_out; t.iters = iters_out;
    t.trace = trace_logp; t.trace_cap = trace_logp ? trace_cap : 0;
    t.barrier = h->gbar.as<unsigned int>();
    if (c.lm_layers > 0) {   // LMFuser (lm.py:43-83) inside the tcgen05 loop
      const int V = c.vocab_sz, Ll = c.lm_layers, Hl = c.lm_hidden_sz;
      const size_t nfl = lm_state_floats(Ll, Hl, V, Bp);
      float* blob = h->lm_blob;
      if (blob) {
        if (h->lm_blob_B != B) return fail(h, RNNT_B200_ERR_INVALID, "decode_greedy: the registered LM state was sized for " +
                                                                        std::to_string(h->lm_blob_B) + " streams, call has " + std::to_string(B));
      } else {
        CK(h->lm_ws.ensure(nfl * 4));
        CK(cudaMemsetAsync(h->lm_ws.p, 0, nfl * 4, st));
        blob = h->lm_ws.as<float>();
      }
      const size_t lone = (size_t)(Hl / 64) * 2 * dpl.Bpad8 * 128;
      CK(h->lm_himg.ensure(lone * 2 * Ll));
      const size_t stat_bytes = (size_t)max_steps * dpl.Bq * 16;   // jstat | lmstat | fkeys (8 B each)
      CK(h->lm_stat.ensure(stat_bytes * 2 + (size_t)max_steps * dpl.Bq * 8));
      CK(cudaMemsetAsync(h->lm_stat.p, 0, stat_bytes * 2 + (size_t)max_steps * dpl.Bq * 8, st));
      DecodeTcLm& L = t.lm;
      L.L = Ll; L.Hl = Hl; L.alpha = c.lm_alpha; L.theta = c.lm_theta;
      L.table0 = h->lmw.table0; L.bo = h->lmw.bo;
      for (int l = 0; l < Ll; ++l) {
        L.bias[l] = h->lmw.bias[l];
        L.r_img[l] = h->lmR_img[l]; L.w_img[l] = h->lmW_img[l];
        L.h_img[l][0] = h->lm_himg.as<uint8_t>() + (size_t)(2 * l) * lone;
        L.h_img[l][1] = h->lm_himg.as<uint8_t>() + (size_t)(2 * l + 1) * lone;
      }
      L.wo_img = h->lmWo_img;
      L.st = lm_state_view(blob, Ll, Hl, V, Bp);
      L.Bp = Bp;
      L.jstat = h->lm_stat.as<double>();
      L.lmstat = reinterpret_cast<double*>(h->lm_stat.as<uint8_t>() + stat_bytes);
      L.fkeys = reinterpret_cast<unsigned long long*>(h->lm_stat.as<uint8_t>() + 2 * stat_bytes);
    }
    LAUNCH(trace_logp ? 3 : 2, launch_decode_tc(t, dpl, st));
    if (h->ev) cudaEventRecord(h->ev[4], st);
    return RNNT_B200_OK;
  }
  const size_t hb = (size_t)H * Bp;
  float* dh = h->dhT.as<float>();
  DecodeArgs a;
  memset(&a, 0, sizeof(a));
  a.w = h->dw;
  for (int l = 0; l < c.pred_layers; ++l) {
    a.hT[l][0] = dh + (size_t)(2 * l) * hb;
    a.hT[l][1] = dh + (size_t)(2 * l + 1) * hb;
    if (use_state_in) LAUNCH(1, launch_state_to_T(pred_state_h + (size_t)l * B * H, a.hT[l][0], B, Bp, H, st));
    else LAUNCH(1, launch_state_broadcast_T(h->dw.h0[l], a.hT[l][0], B, Bp, H, st));
  }
  if (use_state_in) LAUNCH(1, launch_state_to_T(pred_out, h->dgT.as<float>(), B, Bp, H, st));
  if (iters_out) CK(cudaMemsetAsync(iters_out, 0, (size_t)B * T, st));
  a.ep = h->ep.as<float>(); a.lens_T = lens_T; a.B = B; a.Bp = Bp; a.T = T; a.max_iters = max_iters; a.use_state_in = use_state_in;
  a.xT = h->dxT.as<float>(); a.gT = h->dgT.as<float>(); a.ppT = h->dppT.as<float>(); a.zT = h->dzT.as<float>();
  a.part = h->dpart.as<float>(); a.trace_lse = h->dlse.as<float>();
  a.tokens = tokens_out; a.U_cap = U_cap; a.ntok = ntok_out; a.neg_logp = neg_logp_out; a.iters = iters_out;
  a.trace = trace_logp; a.trace_cap = trace_logp ? trace_cap : 0;
  if (c.lm_layers > 0) {   // LMFuser (lm.py:43-83): a fresh fuser per call unless the caller registered stream state
    const int V = c.vocab_sz, Ll = c.lm_layers, Hl = c.lm_hidden_sz;
    const size_t nfl = lm_state_floats(Ll, Hl, V, Bp);
    float* blob = h->lm_blob;
    if (blob) {
      if (h->lm_blob_B != B) return fail(h, RNNT_B200_ERR_INVALID, "decode_greedy: the registered LM state was sized for " +
                                                                      std::to_string(h->lm_blob_B) + " streams, call has " + std::to_string(B));
    } else {
      CK(h->lm_ws.ensure(nfl * 4));
      CK(cudaMemsetAsync(h->lm_ws.p, 0, nfl * 4, st));
      blob = h->lm_ws.as<float>();
    }
    const size_t ntile = (size_t)(V / 32) * Bp;
    CK(h->lm_logitT.ensure((size_t)V * Bp * 4));
    CK(h->lm_part.ensure(ntile * 2 * 8));
    CK(h->lm_jpart.ensure(ntile * 2 * 8));
    CK(h->lm_fpart.ensure(ntile * 2 * 4));
    a.lm = h->lmw;
    a.lms = lm_state_view(blob, Ll, Hl, V, Bp);
    a.logitT = h->lm_logitT.as<float>();
    a.lmpart = h->lm_part.as<double>();
    a.jpart = h->lm_jpart.as<double>();
    a.fpart = h->lm_fpart.as<float>();
  }
  LAUNCH(1, launch_decode(a, h->coop_blocks, st));
  h->fp32_decode_launches += 1;
  if (pred_state_h)
    for (int l = 0; l < c.pred_layers; ++l)
      LAUNCH(1, launch_state_from_T(a.hT[l][0], pred_state_h + (size_t)l * B * H, B, Bp, H, st));
  if (pred_out) LAUNCH(1, launch_state_from_T(h->dgT.as<float>(), pred_out, B, Bp, H, st));
  if (h->ev) cudaEventRecord(h->ev[4], st);
  return RNNT_B200_OK;
}

int32_t rnnt_b200_lm_state_bytes(rnnt_b200_handle h, int32_t B, int64_t* bytes_out) {
  if (!h || !bytes_out) return fail(h, RNNT_B200_ERR_INVALID, "lm_state_bytes: null argument");
  const rnnt_b200_config& c = h->cfg;
  if (c.lm_layers < 1) return fail(h, RNNT_B200_ERR_STATE, "lm_state_bytes: the handle has no language model (cfg.lm_layers == 0)");
  if (B < 1 || B > kDecodeMaxBatch) return fail(h, RNNT_B200_ERR_INVALID, "lm_state_bytes: B must be in [1, 256]");
  *bytes_out = (int64_t)lm_state_floats(c.lm_layers, c.lm_hidden_sz, c.vocab_sz, bp_of(B)) * 4;
  return RNNT_B200_OK;
}

int32_t rnnt_b200_set_lm_state(rnnt_b200_handle h, void* blob_dev, int32_t B) {
  if (!h) return RNNT_B200_ERR_INVALID;
  if (!blob_dev) { h->lm_blob = nullptr; h->lm_blob_B = 0; return RNNT_B200_OK; }
  if (h->cfg.lm_layers < 1) return fail(h, RNNT_B200_ERR_STATE, "set_lm_state: the handle has no language model (cfg.lm_layers == 0)");
  if (B < 1 || B > kDecodeMaxBatch) return fail(h, RNNT_B200_ERR_INVALID, "set_lm_state: B must be in [1, 256]");
  h->lm_blob = static_cast<float*>(blob_dev);
  h->lm_blob_B = B;
  return RNNT_B200_OK;
}

// audio_host != nullptr: `audio` is the device staging buffer and the samples still have to come from the host; the copy is
// issued in utterance blocks on the copy stream so that block i+1 transfers while the front end works on block i.
static int32_t transcribe_impl(rnnt_b200_handle h, const float* audio, const float* audio_host, const int32_t* lens, int32_t B, int64_t n,
                               int32_t max_iters, int32_t* tokens_out, int32_t U_cap, int32_t* ntok_out, double* neg_logp_out,
                               uint8_t* iters_out, void* stream) {
  if (int r = check_ready(h)) return r;
  if (h->pipe[0].busy || h->pipe[1].busy)
    return fail(h, RNNT_B200_ERR_STATE, "transcribe: a pipelined batch is in flight on this handle (shared workspaces); collect it first");
  const rnnt_b200_config& c = h->cfg;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t T = num_steps(c, n);
  if (T < 1) return fail(h, RNNT_B200_ERR_INVALID, "transcribe: input shorter than one stacked row");
  const size_t X = (size_t)c.n_mels * c.n_stack;
  CK(h->feats.ensure((size_t)B * T * X * 4));
  CK(h->t_enc.ensure((size_t)B * T * c.hidden_sz * 4));
  const int32_t* lens_T = nullptr;
  if (lens) {
    // lens_T[b] = num_steps(lens[b]); computed on the host would need a sync, so the feature
    // kernel's own rule is replayed by a tiny device pass stored behind t_lens
    CK(h->t_lens.ensure((size_t)B * 4 * 2));
  }
  if (h->profiling) {
    if (h->ev_used >= (int)h->evsets.size()) {
      cudaEvent_t* set = new cudaEvent_t[kEvPerSet];
      for (int i = 0; i < kEvPerSet; ++i) cudaEventCreate(&set[i]);
      h->evsets.push_back(set);
    }
    h->ev = h->evsets[h->ev_used++];
    cudaEventRecord(h->ev[5], st);
  } else {
    h->ev = nullptr;
  }
  if (audio_host) {
    if (!h->copy_stream) {
      CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
      for (cudaEvent_t& e : h->copy_ev) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    CK(cudaEventRecord(h->copy_ev[4], st));                 // the staging buffer may still be read by earlier work on `st`
    CK(cudaStreamWaitEvent(h->copy_stream, h->copy_ev[4], 0));
    const int nblk = B < 4 ? B : 4, per = (B + nblk - 1) / nblk;
    float* stage = const_cast<float*>(audio);
    for (int i = 0, b0 = 0; b0 < B; ++i, b0 += per) {
      const int nb = std::min(per, B - b0);
      CK(cudaMemcpyAsync(stage + (size_t)b0 * n, audio_host + (size_t)b0 * n, (size_t)nb * n * 4, cudaMemcpyHostToDevice, h->copy_stream));
      CK(cudaEventRecord(h->copy_ev[i], h->copy_stream));
      CK(cudaStreamWaitEvent(st, h->copy_ev[i], 0));
      if (int r = rnnt_b200_features(h, audio + (size_t)b0 * n, lens ? lens + b0 : nullptr, nb, n, h->feats.as<float>() + (size_t)b0 * T * X, stream))
        return r;
    }
  } else if (int r = rnnt_b200_features(h, audio, lens, B, n, h->feats.as<float>(), stream)) {
    return r;
  }
  if (lens) {
    int32_t* lt = h->t_lens.as<int32_t>() + B;
    LAUNCH(1, launch_lens_to_steps(lens, lt, B, c.hop_length, c.n_stack, c.downsample, (int)T, st));
    lens_T = lt;
  }
  if (int r = rnnt_b200_encode(h, h->feats.as<float>(), lens_T, B, (int)T, nullptr, nullptr, 0, h->t_enc.as<float>(), stream)) return r;
  return rnnt_b200_decode_greedy(h, h->t_enc.as<float>(), lens_T, B, (int)T, max_iters, nullptr, nullptr, 0, tokens_out, U_cap,
                                 ntok_out, neg_logp_out, iters_out, nullptr, 0, stream);
}

int32_t rnnt_b200_transcribe(rnnt_b200_handle h, const float* audio, const int32_t* lens, int32_t B, int64_t n, int32_t max_iters,
                             int32_t* tokens_out, int32_t U_cap, int32_t* ntok_out, double* neg_logp_out, uint8_t* iters_out,
                             void* stream) {
  if (!audio) return fail(h, RNNT_B200_ERR_INVALID, "transcribe: null audio");
  return transcribe_impl(h, audio, nullptr, lens, B, n, max_iters, tokens_out, U_cap, ntok_out, neg_logp_out, iters_out, stream);
}

int32_t rnnt_b200_transcribe_host(rnnt_b200_handle h, const float* audio_host, const int32_t* lens_host, int32_t B, int64_t n,
                                  int32_t max_iters, int32_t* tokens_host, int32_t U_cap, int32_t* ntok_host,
                                  double* neg_logp_host, void* stream) {
  if (int r = check_ready(h)) return r;
  if (!audio_host || !tokens_host || !ntok_host || B < 1 || n < 1) return fail(h, RNNT_B200_ERR_INVALID, "transcribe_host: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  CK(h->t_audio.ensure((size_t)B * n * 4));
  CK(h->t_lens.ensure((size_t)B * 4 * 2));
  CK(h->t_tokens.ensure((size_t)B * U_cap * 4));
  CK(h->t_ntok.ensure((size_t)B * 4));
  CK(h->t_nlp.ensure((size_t)B * 8));
  if (lens_host) CK(cudaMemcpyAsync(h->t_lens.p, lens_host, (size_t)B * 4, cudaMemcpyHostToDevice, st));
  if (int r = transcribe_impl(h, h->t_audio.as<float>(), audio_host, lens_host ? h->t_lens.as<int32_t>() : nullptr, B, n, max_iters,
                              h->t_tokens.as<int32_t>(), U_cap, h->t_ntok.as<int32_t>(), h->t_nlp.as<double>(), nullptr, stream))
    return r;
  CK(cudaMemcpyAsync(tokens_host, h->t_tokens.p, (size_t)B * U_cap * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(ntok_host, h->t_ntok.p, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
  if (neg_logp_host) CK(cudaMemcpyAsync(neg_logp_host, h->t_nlp.p, (size_t)B * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return RNNT_B200_OK;
}

// ---------------- two-deep pipeline over the whole path ----------------
// The persistent recurrent kernels (4 LSTM layers + the decode loop: ~90 % of a batch) occupy 128 of the 148 SMs with one CTA
// each and all of their shared memory; the copy engines and the other 20 SMs idle meanwhile.  submit() therefore queues the
// front half of a batch (host->device copy, STFT / mel / stack) on a low-priority stream, where it runs under the recurrent
// kernels of the batch submitted before it, and the back half (encoder, decode, results to the host) on a high-priority
// stream in submission order.  The serving analogue in the reference is its request thread pool (api-server.py:138-139).
int32_t rnnt_b200_pipeline_submit(rnnt_b200_handle h, const float* audio, int32_t on_host, const int32_t* lens, int32_t B, int64_t n,
                                  int32_t max_iters, int32_t slot, int32_t* tokens_host, int32_t U_cap, int32_t* ntok_host,
                                  double* neg_logp_host, void* stream) {
  if (int r = check_ready(h)) return r;
  if (!audio || !tokens_host || !ntok_host || B < 1 || n < 1 || U_cap < 1 || slot < 0 || slot > 1)
    return fail(h, RNNT_B200_ERR_INVALID, "pipeline_submit: bad arguments");
  rnnt_b200_handle_s::PipeSlot& s = h->pipe[slot];
  if (s.busy) return fail(h, RNNT_B200_ERR_STATE, "pipeline_submit: slot still in flight; collect it first");
  const rnnt_b200_config& c = h->cfg;
  const int64_t T = num_steps(c, n);
  if (T < 1) return fail(h, RNNT_B200_ERR_INVALID, "pipeline_submit: input shorter than one stacked row");
  if (!h->pipe_front) {
    int lo = 0, hi = 0;
    CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));   // lo = least urgent (numerically greatest), hi = most urgent
    CK(cudaStreamCreateWithPriority(&h->pipe_front, cudaStreamNonBlocking, lo));
    CK(cudaStreamCreateWithPriority(&h->pipe_back, cudaStreamNonBlocking, hi));
    for (auto& ps : h->pipe)
      for (cudaEvent_t* e : {&ps.in_ready, &ps.front_done, &ps.back_done}) CK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  }
  const size_t X = (size_t)c.n_mels * c.n_stack;
  if (on_host) CK(s.audio.ensure((size_t)B * n * 4));
  CK(s.feats.ensure((size_t)B * T * X * 4));
  CK(s.lens.ensure((size_t)B * 4 * 2));
  CK(s.tokens.ensure((size_t)B * U_cap * 4));
  CK(s.ntok.ensure((size_t)B * 4));
  CK(s.nlp.ensure((size_t)B * 8));
  CK(h->t_enc.ensure((size_t)B * T * c.hidden_sz * 4));
  cudaStream_t st = (cudaStream_t)stream, fs = h->pipe_front, bs = h->pipe_back;
  CK(cudaEventRecord(s.in_ready, st));   // the caller's inputs are complete in `stream` order
  CK(cudaStreamWaitEvent(fs, s.in_ready, 0));
  const float* a_dev = audio;
  const int32_t* lens_dev = lens;
  if (on_host) {
    CK(cudaMemcpyAsync(s.audio.p, audio, (size_t)B * n * 4, cudaMemcpyHostToDevice, fs));
    a_dev = s.audio.as<float>();
    if (lens) {
      CK(cudaMemcpyAsync(s.lens.p, lens, (size_t)B * 4, cudaMemcpyHostToDevice, fs));
      lens_dev = s.lens.as<int32_t>();
    }
  }
  if (int r = rnnt_b200_features(h, a_dev, lens_dev, B, n, s.feats.as<float>(), fs)) return r;
  const int32_t* lens_T = nullptr;
  if (lens) {
    int32_t* lt = s.lens.as<int32_t>() + B;
    LAUNCH(1, launch_lens_to_steps(lens_dev, lt, B, c.hop_length, c.n_stack, c.downsample, (int)T, fs));
    lens_T = lt;
  }
  CK(cudaEventRecord(s.front_done, fs));
  CK(cudaStreamWaitEvent(bs, s.front_done, 0));
  h->ev = nullptr;   // no stage events on the pipelined path (stages of consecutive batches overlap)
  struct CoopOff {   // plain launches for the persistent kernels while the front end of the next batch may be resident (kernels.h)
    bool prev;
    CoopOff() : prev(coop_launch_enabled()) { set_coop_launch(false); }
    ~CoopOff() { set_coop_launch(prev); }
  } coop_off;
  if (int r = rnnt_b200_encode(h, s.feats.as<float>(), lens_T, B, (int)T, nullptr, nullptr, 0, h->t_enc.as<float>(), bs)) return r;
  if (int r = rnnt_b200_decode_greedy(h, h->t_enc.as<float>(), lens_T, B, (int)T, max_iters, nullptr, nullptr, 0, s.tokens.as<int32_t>(), U_cap,
                                      s.ntok.as<int32_t>(), s.nlp.as<double>(), nullptr, nullptr, 0, bs))
    return r;
  CK(cudaMemcpyAsync(tokens_host, s.tokens.p, (size_t)B * U_cap * 4, cudaMemcpyDeviceToHost, bs));
  CK(cudaMemcpyAsync(ntok_host, s.ntok.p, (size_t)B * 4, cudaMemcpyDeviceToHost, bs));
  if (neg_logp_host) CK(cudaMemcpyAsync(neg_logp_host, s.nlp.p, (size_t)B * 8, cudaMemcpyDeviceToHost, bs));
  CK(cudaEventRecord(s.back_done, bs));
  s.busy = true;
  return RNNT_B200_OK;
}

/* Non-blocking progress probe of a slot: *front_done / *back_done = 1 when that half has finished on the device. */
int32_t rnnt_b200_pipeline_query(rnnt_b200_handle h, int32_t slot, int32_t* front_done, int32_t* back_done) {
  if (!h || slot < 0 || slot > 1 || !front_done || !back_done) return fail(h, RNNT_B200_ERR_INVALID, "pipeline_query: bad arguments");
  rnnt_b200_handle_s::PipeSlot& s = h->pipe[slot];
  *front_done = *back_done = 0;
  if (!s.front_done) return RNNT_B200_OK;
  *front_done = cudaEventQuery(s.front_done) == cudaSuccess;
  *back_done = cudaEventQuery(s.back_done) == cudaSuccess;
  cudaGetLastError();
  return RNNT_B200_OK;
}

int32_t rnnt_b200_pipeline_collect(rnnt_b200_handle h, int32_t slot) {
  if (!h || slot < 0 || slot > 1) return fail(h, RNNT_B200_ERR_INVALID, "pipeline_collect: bad arguments");
  rnnt_b200_handle_s::PipeSlot& s = h->pipe[slot];
  if (!s.busy) return fail(h, RNNT_B200_ERR_STATE, "pipeline_collect: nothing was submitted on this slot");
  CK(cudaSetDevice(h->cfg.device));
  s.busy = false;
  CK(cudaEventSynchronize(s.back_done));
  return RNNT_B200_OK;
}


// ---------------- beam search (beam.cu) ----------------
namespace {
int ensure_beam_weights(rnnt_b200_handle h, cudaStream_t st) {
  if (h->bm_w1p) return RNNT_B200_OK;
  const rnnt_b200_config& c = h->cfg;
  const int H = c.hidden_sz, J = c.joint_sz, V = c.vocab_sz;
  auto mk = [&](uint8_t** out, size_t bytes) -> cudaError_t {
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return e;
    h->weight_allocs.push_back(p);
    *out = (uint8_t*)p;
    return cudaSuccess;
  };
  float* tmp = nullptr;
  CK(cudaMalloc((void**)&tmp, (size_t)std::max(3 * H, V) * std::max(H, J) * 4));
  CK(mk(&h->bm_w1p, gemm_tc_w_image_bytes(J, H)));
  LAUNCH(1, launch_to_image(h->W1, 2 * H, J, H, 256, h->bm_w1p, st));                       // pred half of joint.0: first H columns
  CK(mk(&h->bm_w2, gemm_tc_w_image_bytes(V, J)));
  LAUNCH(1, launch_transpose(h->dw.W2_t, V, tmp, J, V, st));                                 // [J][V] -> [V][J]
  LAUNCH(1, launch_to_image(tmp, J, V, J, 256, h->bm_w2, st));
  for (int l = 0; l < 2; ++l) {
    CK(mk(&h->bm_r[l], gemm_tc_w_image_bytes(3 * H, H)));
    LAUNCH(1, launch_transpose(h->dw.Rt[l], 3 * H, tmp, H, 3 * H, st));                      // [H][3H] -> [3H interleaved][H]
    LAUNCH(1, launch_to_image(tmp, H, 3 * H, H, 256, h->bm_r[l], st));
  }
  CK(mk(&h->bm_k1, gemm_tc_w_image_bytes(3 * H, H)));
  LAUNCH(1, launch_transpose(h->dw.Kt[1], 3 * H, tmp, H, 3 * H, st));
  LAUNCH(1, launch_to_image(tmp, H, 3 * H, H, 256, h->bm_k1, st));
  CK(cudaStreamSynchronize(st));
  cudaFree(tmp);
  return RNNT_B200_OK;
}
}  // namespace

int32_t rnnt_b200_decode_beam(rnnt_b200_handle h, const float* enc, const int32_t* lens_T, int32_t B, int32_t T, int32_t width,
                              int32_t max_iters, int32_t* tokens_out, int32_t U_cap, int32_t* ntok_out, double* score_out,
                              void* stream) {
  if (int r = check_ready(h)) return r;
  const rnnt_b200_config& c = h->cfg;
  if (!enc || !tokens_out || !ntok_out || B < 1 || T < 1) return fail(h, RNNT_B200_ERR_INVALID, "decode_beam: bad arguments");
  if (width < 1 || width > 8 || max_iters < 1 || max_iters > 16) return fail(h, RNNT_B200_ERR_INVALID, "decode_beam: width must be in [1, 8], max_iters in [1, 16]");
  if ((int64_t)U_cap < (int64_t)max_iters * T) return fail(h, RNNT_B200_ERR_INVALID, "decode_beam: U_cap < max_iters*T");
  if (c.gemm_mode != RNNT_B200_GEMM_TC_FP16X3) return fail(h, RNNT_B200_ERR_INVALID, "decode_beam: needs gemm_mode 1 (tcgen05)");
  if (c.pred_layers != 2 || c.vocab_sz > 4096 || (c.hidden_sz % 64) || (c.joint_sz % 64))
    return fail(h, RNNT_B200_ERR_INVALID, "decode_beam: unsupported shape (two predictor layers, vocab <= 4096, H and J multiples of 64)");
  if (c.lm_layers > 0) return fail(h, RNNT_B200_ERR_INVALID, "decode_beam: LM fusion is not part of the beam search");
  cudaStream_t st = (cudaStream_t)stream;
  const int H = c.hidden_sz, J = c.joint_sz, V = c.vocab_sz, W = width;
  {   // utterances are independent: bound the rows per pass
    const int cap = std::max(1, 1024 / W);
    if (B > cap) {
      for (int b0 = 0; b0 < B; b0 += cap) {
        const int nb = std::min(cap, B - b0);
        if (int r = rnnt_b200_decode_beam(h, enc + (size_t)b0 * T * H, lens_T ? lens_T + b0 : nullptr, nb, T, width, max_iters,
                                          tokens_out + (size_t)b0 * U_cap, U_cap, ntok_out + b0, score_out ? score_out + b0 : nullptr, stream))
          return r;
      }
      return RNNT_B200_OK;
    }
  }
  if (int r = ensure_beam_weights(h, st)) return r;
  const int R = B * W, NG = max_iters + 2;
  const int64_t M = (int64_t)B * T;
  if (int r = ensure_decode_ws(h, B, T, 0)) return r;
  // hoisted encoder half of the joint's first Linear (as decode_greedy)
  CK(h->a_img.ensure(gemm_tc_a_image_bytes(M, H)));
  LAUNCH(1, launch_to_image(enc, H, M, H, 128, h->a_img.as<uint8_t>(), st));
  LAUNCH(1, launch_gemm_tc(h->a_img.as<uint8_t>(), h->W1e_img, h->dw.b1, h->ep.as<float>(), J, M, J, H, st));
  // workspaces
  const int leave_cap = W * (max_iters + 1), node_cap = 1 + T * max_iters * W + W;
  CK(h->bm_state.ensure((size_t)3 * NG * R * H * 4));
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
  const size_t o_hyp = take((size_t)NG * R * sizeof(BeamHyp)), o_leave = take((size_t)B * leave_cap * sizeof(BeamLeave)), o_nl = take((size_t)B * 4),
               o_np = take((size_t)B * node_cap * 4), o_nt = take((size_t)B * node_cap * 4), o_nn = take((size_t)B * 4), o_cv = take((size_t)R * W * 4),
               o_ci = take((size_t)R * W * 4), o_lb = take((size_t)R * 4), o_sr = take((size_t)R * 4), o_stok = take((size_t)R * 4), o_cs = take((size_t)R * 4);
  CK(h->bm_meta.ensure(off));
  uint8_t* mb = h->bm_meta.as<uint8_t>();
  CK(h->bm_aimg.ensure(gemm_tc_a_image_bytes(R, std::max(H, J))));
  size_t fo = 0;
  auto takef = [&](size_t n) { const size_t o = fo; fo += (n + 63) & ~(size_t)63; return o; };
  const size_t f_pp = takef((size_t)R * J), f_lg = takef((size_t)R * V), f_rec = takef((size_t)R * 3 * H), f_kin = takef((size_t)R * 3 * H), f_x1 = takef((size_t)R * H);
  CK(h->bm_f32.ensure(fo * 4));
  float* fb = h->bm_f32.as<float>();
  BeamArgs a;
  memset(&a, 0, sizeof(a));
  a.w = h->dw; a.ep = h->ep.as<float>(); a.lens_T = lens_T; a.B = B; a.T = T; a.W = W; a.n_gen = NG;
  a.state = h->bm_state.as<float>();
  a.hyp = reinterpret_cast<BeamHyp*>(mb + o_hyp);
  a.leave = reinterpret_cast<BeamLeave*>(mb + o_leave); a.leave_cap = leave_cap; a.n_leave = reinterpret_cast<int*>(mb + o_nl);
  a.node_parent = reinterpret_cast<int*>(mb + o_np); a.node_token = reinterpret_cast<int*>(mb + o_nt); a.node_cap = node_cap;
  a.n_nodes = reinterpret_cast<int*>(mb + o_nn);
  a.cand_val = reinterpret_cast<float*>(mb + o_cv); a.cand_idx = reinterpret_cast<int*>(mb + o_ci); a.lp_blank = reinterpret_cast<float*>(mb + o_lb);
  a.sel_row = reinterpret_cast<int*>(mb + o_sr); a.sel_tok = reinterpret_cast<int*>(mb + o_stok); a.copy_src = reinterpret_cast<int*>(mb + o_cs);
  BeamBuffers bf;
  bf.a_img = h->bm_aimg.as<uint8_t>();
  bf.w1p_img = h->bm_w1p; bf.w2_img = h->bm_w2; bf.k1_img = h->bm_k1; bf.r_img[0] = h->bm_r[0]; bf.r_img[1] = h->bm_r[1];
  bf.pp = fb + f_pp; bf.logits = fb + f_lg; bf.rec = fb + f_rec; bf.kin = fb + f_kin; bf.x1 = fb + f_x1;
  int launches = 0;
  cudaError_t e = launch_beam_search(a, bf, max_iters, tokens_out, U_cap, ntok_out, score_out, &launches, st);
  if (e != cudaSuccess) return fail_cuda(h, e, "decode_beam");
  h->launches += launches;
  return RNNT_B200_OK;
}

// ---------------- training-time forward: joint lattice + RNN-T loss (lattice.cu) ----------------
int32_t rnnt_b200_rnnt_loss(rnnt_b200_handle h, const float* lattice, const int32_t* lens_T, const int32_t* labels,
                            const int32_t* label_lens, int32_t N, int32_t T, int32_t U, double* loss_out, void* stream) {
  if (int r = check_ready(h)) return r;
  if (!lattice || !labels || !label_lens || !loss_out || N < 1 || T < 1 || U < 1) return fail(h, RNNT_B200_ERR_INVALID, "rnnt_loss: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t rows = (int64_t)N * T * U;
  CK(h->lt_f32.ensure((size_t)rows * 2 * 4));
  float* lpb = h->lt_f32.as<float>();
  float* lpl = lpb + rows;
  LAUNCH(1, launch_lattice_gather(lattice, rows, h->cfg.vocab_sz, labels, T, U, U - 1, h->cfg.blank, lpb, lpl, st));
  LAUNCH(1, launch_rnnt_alpha(lpb, lpl, lens_T, label_lens, N, T, U, loss_out, st));
  return RNNT_B200_OK;
}

int32_t rnnt_b200_forward_loss(rnnt_b200_handle h, const float* feats, const int32_t* lens_T, const int32_t* labels,
                               const int32_t* label_lens, int32_t N, int32_t T, int32_t Umax, float* lattice_out,
                               double* loss_out, void* stream) {
  if (int r = check_ready(h)) return r;
  const rnnt_b200_config& c = h->cfg;
  if (!feats || !labels || !label_lens || !loss_out || N < 1 || N > kDecodeMaxBatch || T < 1 || Umax < 1)
    return fail(h, RNNT_B200_ERR_INVALID, "forward_loss: bad arguments (1 <= N <= 256)");
  if (c.gemm_mode != RNNT_B200_GEMM_TC_FP16X3) return fail(h, RNNT_B200_ERR_INVALID, "forward_loss: needs gemm_mode 1 (tcgen05)");
  if ((c.hidden_sz % 64) || (c.joint_sz % 64)) return fail(h, RNNT_B200_ERR_INVALID, "forward_loss: H and J must be multiples of 64");
  cudaStream_t st = (cudaStream_t)stream;
  const int H = c.hidden_sz, J = c.joint_sz, V = c.vocab_sz, U = Umax + 1;
  if (int r = ensure_beam_weights(h, st)) return r;     // 256-row-tile images of W1p / W2 for gemm_tc.cu
  // encoder (models.py:318-320), then the encoder half of the joint's first Linear for all frames
  CK(h->lt_enc.ensure((size_t)N * T * H * 4));
  float* enc = h->lt_enc.as<float>();
  if (int r = rnnt_b200_encode(h, feats, lens_T, N, T, nullptr, nullptr, 0, enc, stream)) return r;
  const int64_t M = (int64_t)N * T;
  if (int r = ensure_decode_ws(h, N, T, 0)) return r;
  CK(h->a_img.ensure(gemm_tc_a_image_bytes(M, H)));
  LAUNCH(1, launch_to_image(enc, H, M, H, 128, h->a_img.as<uint8_t>(), st));
  LAUNCH(1, launch_gemm_tc(h->a_img.as<uint8_t>(), h->W1e_img, h->dw.b1, h->ep.as<float>(), J, M, J, H, st));
  // workspaces: g_all [N*U][H] | pp_all [N*U][J] | lpb, lpl [N*T*U] | logits chunk [CH][V] | predictor state, step output
  const int64_t rows = (int64_t)N * T * U;
  const int CH = 8192;
  size_t fo = 0;
  auto takef = [&](size_t n) { const size_t o = fo; fo += (n + 63) & ~(size_t)63; return o; };
  const size_t f_g = takef((size_t)N * U * H), f_pp = takef((size_t)N * U * J), f_lpb = takef((size_t)rows), f_lpl = takef((size_t)rows),
               f_lg = takef((size_t)CH * V), f_st = takef((size_t)c.pred_layers * N * H), f_out = takef((size_t)N * H);
  CK(h->lt_f32.ensure(fo * 4));
  float* fb = h->lt_f32.as<float>();
  CK(h->lt_i32.ensure((size_t)N * 4));
  int32_t* toks = h->lt_i32.as<int32_t>();
  // predictor, teacher-forced over cat(bos, y) (models.py:326-336): one step per label position, state carried
  for (int u = 0; u < U; ++u) {
    LAUNCH(1, launch_lattice_tokens(labels, N, Umax, u, c.bos, toks, st));
    if (int r = rnnt_b200_predict(h, toks, N, fb + f_st, u > 0 ? 1 : 0, fb + f_out, stream)) return r;
    CK(cudaMemcpy2DAsync(fb + f_g + (size_t)u * H, (size_t)U * H * 4, fb + f_out, (size_t)H * 4, (size_t)H * 4, N, cudaMemcpyDeviceToDevice, st));
  }
  // pred half of the joint's first Linear for every label position
  CK(h->bm_aimg.ensure(gemm_tc_a_image_bytes(std::max<int64_t>((int64_t)N * U, CH), std::max(H, J))));
  LAUNCH(1, launch_to_image(fb + f_g, H, (int64_t)N * U, H, 128, h->bm_aimg.as<uint8_t>(), st));
  LAUNCH(1, launch_gemm_tc(h->bm_aimg.as<uint8_t>(), h->bm_w1p, nullptr, fb + f_pp, J, (int64_t)N * U, J, H, st));
  // the lattice in L2-sized chunks of rows (n, t, u): z image -> logits -> (log p(blank), log p(label)) [+ log_softmax rows]
  for (int64_t r0 = 0; r0 < rows; r0 += CH) {
    const int nr = (int)std::min<int64_t>(CH, rows - r0);
    LAUNCH(1, launch_lattice_z_image(fb + f_pp, h->ep.as<float>(), T, U, r0, nr, J, h->bm_aimg.as<uint8_t>(), st));
    LAUNCH(1, launch_gemm_tc(h->bm_aimg.as<uint8_t>(), h->bm_w2, h->dw.b2, fb + f_lg, V, nr, V, J, st));
    LAUNCH(1, launch_lattice_lse(fb + f_lg, nr, V, r0, labels, T, U, Umax, c.blank, fb + f_lpb, fb + f_lpl, lattice_out, st));
  }
  LAUNCH(1, launch_rnnt_alpha(fb + f_lpb, fb + f_lpl, lens_T, label_lens, N, T, U, loss_out, st));
  return RNNT_B200_OK;
}

// ---------------- streaming sessions ----------------
struct rnnt_b200_stream_s {
  rnnt_b200_handle h = nullptr;
  int B = 0, chunk = 0, n_window = 0, n_buffer = 0, max_iters = 0;
  // per-stream phase of the serving loop: chunks seen since the stream (re)started, rows waiting in its Buffer
  std::vector<int64_t> n_chunks;
  std::vector<int> n_rows;
  int cur = 0;            // which window buffer is current
  DevBuf win[2], stage, row, rows, enc_h, enc_c, pred_h, pred_out, enc_out, tokens, ntok, lm;
  DevBuf bos_h, bos_out;  // predictor state / output after feeding BOS from the learnable state (reset_predictor, models.py:484-489)
  DevBuf ctl;             // device copy of the per-tick control words: pos[B] | lens_T[B]
  int32_t* ctl_host = nullptr;   // pinned staging for `ctl`
  bool counted = false;          // registered in h->open_streams
};

namespace {
// stream `slot` back to the state of a fresh connection; keep_audio: only what the reference's reset_fn resets
// (encoder state, predictor -> BOS, LM fuser; models.py:480-500) -- the 3-chunk audio window and the Buffer live in the
// serving loop (api-server.py:83-115, transforms.py:455-471) and survive it
int stream_reset_slot_impl(rnnt_b200_stream s, int slot, cudaStream_t st, bool keep_audio = false) {
  rnnt_b200_handle h = s->h;
  const rnnt_b200_config& c = h->cfg;
  const size_t H = c.hidden_sz, W = (size_t)s->n_window * s->chunk;
  const int B = s->B;
  if (!keep_audio)
    for (int i = 0; i < 2; ++i) CK(cudaMemsetAsync(s->win[i].as<float>() + (size_t)slot * W, 0, W * 4, st));
  for (int l = 0; l < c.enc_layers; ++l) {   // state None -> the learnable hs[i] (custom_rnn.py:152-158)
    CK(cudaMemcpyAsync(s->enc_h.as<float>() + ((size_t)l * B + slot) * H, h->enc[l].h0, H * 4, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(s->enc_c.as<float>() + ((size_t)l * B + slot) * H, h->enc[l].c0, H * 4, cudaMemcpyDeviceToDevice, st));
  }
  for (int l = 0; l < c.pred_layers; ++l)
    CK(cudaMemcpyAsync(s->pred_h.as<float>() + ((size_t)l * B + slot) * H, s->bos_h.as<float>() + (size_t)l * H, H * 4,
                       cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(s->pred_out.as<float>() + (size_t)slot * H, s->bos_out.p, H * 4, cudaMemcpyDeviceToDevice, st));
  if (c.lm_layers > 0) {   // LMFuser.reset (lm.py:81-83): column `slot` of the feature-major blob
    const int Bp = bp_of(B);
    const size_t rows = lm_state_floats(c.lm_layers, c.lm_hidden_sz, c.vocab_sz, Bp) / Bp;
    CK(cudaMemset2DAsync(s->lm.as<float>() + slot, (size_t)Bp * 4, 0, 4, rows, st));
  }
  if (!keep_audio) {
    s->n_chunks[slot] = 0;
    s->n_rows[slot] = 0;
  }
  return RNNT_B200_OK;
}
}  // namespace

int32_t rnnt_b200_stream_open(rnnt_b200_handle h, int32_t B, int32_t chunk, int32_t n_window, int32_t n_buffer,
                              int32_t max_iters, rnnt_b200_stream* out) {
  if (int r = check_ready(h)) return r;
  if (!out) return fail(h, RNNT_B200_ERR_INVALID, "stream_open: null argument");
  *out = nullptr;
  const rnnt_b200_config& c = h->cfg;
  const int cap = kDecodeMaxBatch;   // beyond the tcgen05 kernel's 64 streams the fp32 kernel takes over
  if (B < 1 || B > cap) return fail(h, RNNT_B200_ERR_INVALID, "stream_open: n_streams must be in [1, " + std::to_string(cap) + "]");
  if (chunk < 1 || n_window < 1 || n_buffer < 1 || n_buffer > 64 || max_iters < 1 || max_iters > 255)
    return fail(h, RNNT_B200_ERR_INVALID, "stream_open: bad arguments");
  const int64_t W = (int64_t)n_window * chunk, F = num_frames(c, W);
  if (W <= c.n_fft / 2 || F / 3 + 1 + c.n_stack > F)
    return fail(h, RNNT_B200_ERR_INVALID, "stream_open: window too short for n_stack frames after the middle-third crop");
  CK(cudaSetDevice(c.device));
  rnnt_b200_stream s = new rnnt_b200_stream_s();
  s->h = h; s->B = B; s->chunk = chunk; s->n_window = n_window; s->n_buffer = n_buffer; s->max_iters = max_iters;
  s->n_chunks.assign(B, 0); s->n_rows.assign(B, 0);
  const size_t X = (size_t)c.n_mels * c.n_stack, H = c.hidden_sz;
  cudaError_t e = cudaSuccess;
  auto need = [&](DevBuf& b, size_t bytes) { if (e == cudaSuccess) e = b.ensure(bytes); };
  need(s->win[0], (size_t)B * W * 4); need(s->win[1], (size_t)B * W * 4);
  need(s->stage, (size_t)B * chunk * 4);
  need(s->row, (size_t)B * X * 4); need(s->rows, (size_t)B * n_buffer * X * 4);
  need(s->enc_h, (size_t)c.enc_layers * B * H * 4); need(s->enc_c, (size_t)c.enc_layers * B * H * 4);
  need(s->pred_h, (size_t)c.pred_layers * B * H * 4); need(s->pred_out, (size_t)B * H * 4);
  need(s->enc_out, (size_t)B * n_buffer * H * 4);
  need(s->tokens, (size_t)B * max_iters * n_buffer * 4); need(s->ntok, (size_t)B * 4);
  need(s->bos_h, (size_t)c.pred_layers * H * 4); need(s->bos_out, H * 4);
  need(s->ctl, (size_t)2 * B * 4);
  if (c.lm_layers > 0) need(s->lm, lm_state_floats(c.lm_layers, c.lm_hidden_sz, c.vocab_sz, bp_of(B)) * 4);
  if (e == cudaSuccess) e = cudaMallocHost((void**)&s->ctl_host, (size_t)2 * B * 4);
  if (e != cudaSuccess) { rnnt_b200_stream_close(s); return fail_cuda(h, e, "stream_open: allocation"); }
  // The predictor state of a fresh stream = the decode loop's own BOS step (models.py:484-489): run the decode kernel on
  // one stream with zero frames -- it feeds BOS from the learnable state, finds nothing to decode and hands the state back.
  {
    void* prev_blob = h->lm_blob; const int prev_B = h->lm_blob_B;
    h->lm_blob = nullptr; h->lm_blob_B = 0;
    int32_t* zero_len = s->ctl.as<int32_t>();   // ensure() zero-fills: lens_T = 0
    const int r = rnnt_b200_decode_greedy(h, s->enc_out.as<float>(), zero_len, 1, 1, max_iters, s->bos_h.as<float>(), s->bos_out.as<float>(), 0,
                                          s->tokens.as<int32_t>(), max_iters * n_buffer, s->ntok.as<int32_t>(), nullptr, nullptr, nullptr, 0,
                                          nullptr);
    h->lm_blob = static_cast<float*>(prev_blob); h->lm_blob_B = prev_B;
    if (r) { rnnt_b200_stream_close(s); return r; }
  }
  for (int b = 0; b < B; ++b)
    if (int r = stream_reset_slot_impl(s, b, nullptr)) { rnnt_b200_stream_close(s); return r; }
  CK(cudaStreamSynchronize(nullptr));
  h->open_streams += 1;
  s->counted = true;
  *out = s;
  return RNNT_B200_OK;
}

static int32_t stream_reset_common(rnnt_b200_stream s, int32_t slot, bool keep_audio) {
  if (!s) return RNNT_B200_ERR_INVALID;
  rnnt_b200_handle h = s->h;
  if (slot < -1 || slot >= s->B) return fail(h, RNNT_B200_ERR_INVALID, "stream_reset: slot out of range (-1 = all streams)");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  for (int b = (slot < 0 ? 0 : slot); b < (slot < 0 ? s->B : slot + 1); ++b)
    if (int r = stream_reset_slot_impl(s, b, nullptr, keep_audio)) return r;
  CK(cudaStreamSynchronize(nullptr));
  return RNNT_B200_OK;
}
int32_t rnnt_b200_stream_reset(rnnt_b200_stream s, int32_t slot) { return stream_reset_common(s, slot, false); }
int32_t rnnt_b200_stream_reset_state(rnnt_b200_stream s, int32_t slot) { return stream_reset_common(s, slot, true); }

int32_t rnnt_b200_stream_close(rnnt_b200_stream s) {
  if (!s) return RNNT_B200_OK;
  cudaSetDevice(s->h->cfg.device);
  cudaDeviceSynchronize();
  if (s->h->lm_blob == s->lm.p) { s->h->lm_blob = nullptr; s->h->lm_blob_B = 0; }
  for (DevBuf* b : {&s->win[0], &s->win[1], &s->stage, &s->row, &s->rows, &s->enc_h, &s->enc_c, &s->pred_h, &s->pred_out,
                    &s->enc_out, &s->tokens, &s->ntok, &s->lm, &s->bos_h, &s->bos_out, &s->ctl})
    b->release();
  if (s->ctl_host) cudaFreeHost(s->ctl_host);
  if (s->counted) s->h->open_streams -= 1;
  delete s;
  return RNNT_B200_OK;
}

int32_t rnnt_b200_stream_push(rnnt_b200_stream s, const float* chunks, int32_t on_host, const uint8_t* active_host,
                              int32_t* tokens_host, int32_t U_cap, int32_t* ntok_host, int32_t* advanced, void* stream) {
  if (!s) return RNNT_B200_ERR_INVALID;
  rnnt_b200_handle h = s->h;
  const rnnt_b200_config& c = h->cfg;
  if (!chunks || !advanced) return fail(h, RNNT_B200_ERR_INVALID, "stream_push: null argument");
  if (h->pipe[0].busy || h->pipe[1].busy)
    return fail(h, RNNT_B200_ERR_STATE, "stream_push: a pipelined batch is in flight on this handle (shared workspaces); collect it first");
  *advanced = 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int B = s->B, ck = s->chunk;
  const size_t W = (size_t)s->n_window * ck, X = (size_t)c.n_mels * c.n_stack;
  const int U = s->max_iters * s->n_buffer;
  // per-stream phase (api-server.py:95-115 + Buffer, transforms.py:463-471), advanced on the host; the kernels get it as words
  StreamMask mask;
  memset(&mask, 0, sizeof(mask));
  int32_t* pos = s->ctl_host;
  int32_t* lens = s->ctl_host + B;
  bool any_row = false, any_ready = false;
  CK(cudaStreamSynchronize(st));   // the staging words of the previous tick have been consumed
  for (int b = 0; b < B; ++b) {
    pos[b] = -1; lens[b] = 0;
    if (active_host && !active_host[b]) continue;
    mask.bits[b >> 5] |= 1u << (b & 31);
    s->n_chunks[b] += 1;
    if (s->n_chunks[b] < s->n_window) continue;       // server: `continue` until the window is full
    pos[b] = s->n_rows[b];
    any_row = true;
    if (++s->n_rows[b] == s->n_buffer) { s->n_rows[b] = 0; lens[b] = s->n_buffer; any_ready = true; }
  }
  const float* chunks_dev = chunks;
  if (on_host) {
    CK(cudaMemcpyAsync(s->stage.p, chunks, (size_t)B * ck * 4, cudaMemcpyHostToDevice, st));
    chunks_dev = s->stage.as<float>();
  }
  float* wold = s->win[s->cur].as<float>();
  float* wnew = s->win[s->cur ^ 1].as<float>();
  LAUNCH(1, launch_slide_window(wold, wnew, chunks_dev, B, (int)W, ck, mask, st));
  s->cur ^= 1;
  // a host chunk buffer may be reused by the caller as soon as this call returns: on the paths that do not end in the
  // stream synchronisation below, wait for the copy out of it here
  if (!any_row) { if (on_host) CK(cudaStreamSynchronize(st)); return RNNT_B200_OK; }
  CK(cudaMemcpyAsync(s->ctl.p, s->ctl_host, (size_t)2 * B * 4, cudaMemcpyHostToDevice, st));
  // stream transforms -> one stacked row per stream, appended to its Buffer (transforms.py:326-342,463-471)
  if (int r = rnnt_b200_features_stream(h, wnew, B, (int64_t)W, s->row.as<float>(), stream)) return r;
  LAUNCH(1, launch_store_rows(s->row.as<float>(), s->rows.as<float>(), s->ctl.as<int32_t>(), B, (int)X, s->n_buffer, st));
  if (!any_ready) { if (on_host) CK(cudaStreamSynchronize(st)); return RNNT_B200_OK; }
  if (!tokens_host || !ntok_host || U_cap < U) return fail(h, RNNT_B200_ERR_INVALID, "stream_push: token outputs missing or U_cap < max_iters * n_buffer");
  // Transducer.transcribe_stream, one chunk of n_buffer encoder steps for the streams whose Buffer filled (models.py:503-571);
  // the others take part with zero frames (state untouched)
  const int32_t* lens_dev = s->ctl.as<int32_t>() + B;
  if (int r = rnnt_b200_encode(h, s->rows.as<float>(), lens_dev, B, s->n_buffer, s->enc_h.as<float>(), s->enc_c.as<float>(), 1,
                               s->enc_out.as<float>(), stream))
    return r;
  void* prev_blob = h->lm_blob;
  const int prev_B = h->lm_blob_B;
  if (c.lm_layers > 0) { h->lm_blob = s->lm.as<float>(); h->lm_blob_B = B; }
  const int r = rnnt_b200_decode_greedy(h, s->enc_out.as<float>(), lens_dev, B, s->n_buffer, s->max_iters, s->pred_h.as<float>(),
                                        s->pred_out.as<float>(), 1, s->tokens.as<int32_t>(), U, s->ntok.as<int32_t>(), nullptr,
                                        nullptr, nullptr, 0, stream);
  h->lm_blob = static_cast<float*>(prev_blob); h->lm_blob_B = prev_B;
  if (r) return r;
  CK(cudaMemcpy2DAsync(tokens_host, (size_t)U_cap * 4, s->tokens.p, (size_t)U * 4, (size_t)U * 4, B, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(ntok_host, s->ntok.p, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (int b = 0; b < B; ++b)
    if (lens[b] == 0) ntok_host[b] = -1;   // this stream did not run the model in this tick
  *advanced = 1;
  return RNNT_B200_OK;
}

int32_t rnnt_b200_selftest_gemm(rnnt_b200_handle h, const float* A, const float* W, const float* bias, float* C, int64_t M,
                                int32_t N, int32_t K, int32_t gemm_mode, void* stream) {
  if (!h || !A || !W || !C || M < 1 || N < 1 || K < 1 || (K & 3) || (N & 3)) return fail(h, RNNT_B200_ERR_INVALID, "selftest_gemm: bad arguments");
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  if (gemm_mode == RNNT_B200_GEMM_FP32_SIMT) {
    LAUNCH(1, launch_gemm_nt_f32(A, K, W, K, bias, C, N, M, N, K, st));
    return RNNT_B200_OK;
  }
  if (gemm_mode != RNNT_B200_GEMM_TC_FP16X3) return fail(h, RNNT_B200_ERR_INVALID, "selftest_gemm: unknown gemm_mode");
  void *ai = nullptr, *wi = nullptr;
  CK(cudaMalloc(&ai, gemm_tc_a_image_bytes(M, K)));
  CK(cudaMalloc(&wi, gemm_tc_w_image_bytes(N, K)));
  cudaError_t e = launch_to_image(A, K, M, K, 128, (uint8_t*)ai, st);
  if (e == cudaSuccess) e = launch_to_image(W, K, N, K, 256, (uint8_t*)wi, st);
  if (e == cudaSuccess) e = launch_gemm_tc((uint8_t*)ai, (uint8_t*)wi, bias, C, N, M, N, K, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(ai);
  cudaFree(wi);
  if (e != cudaSuccess) return fail_cuda(h, e, "selftest_gemm");
  h->launches += 3;
  return RNNT_B200_OK;
}

int64_t rnnt_b200_kernel_launches(rnnt_b200_handle h) { return h ? h->launches : -1; }
int64_t rnnt_b200_fp32_decode_launches(rnnt_b200_handle h) { return h ? h->fp32_decode_launches : -1; }

int32_t rnnt_b200_set_profiling(rnnt_b200_handle h, int32_t enable) {
  if (!h) return RNNT_B200_ERR_INVALID;
  h->profiling = enable != 0;
  h->ev_used = 0;
  h->ev = nullptr;
  return RNNT_B200_OK;
}

int32_t rnnt_b200_stage_times_ms(rnnt_b200_handle h, float* out) {
  if (!h || !out) return RNNT_B200_ERR_INVALID;
  if (!h->profiling || h->ev_used < 1) return fail(h, RNNT_B200_ERR_STATE, "no profiled transcribe() call recorded");
  CK(cudaSetDevice(h->cfg.device));
  // ev5 -> ev0: features ; ev0 -> ev1: encoder ; ev2 -> ev3: ep GEMM ; ev3 -> ev4: decode
  double acc[5] = {0, 0, 0, 0, 0};
  for (int s = 0; s < h->ev_used; ++s) {
    cudaEvent_t* ev = h->evsets[s];
    CK(cudaEventSynchronize(ev[4]));
    float f = 0, e = 0, j = 0, d = 0;
    for (int l = 0; l < h->cfg.enc_layers; ++l) {
      float gl = 0;
      CK(cudaEventElapsedTime(&gl, ev[6 + 2 * l], ev[7 + 2 * l]));
      acc[2] += gl;
    }
    CK(cudaEventElapsedTime(&f, ev[5], ev[0]));
    CK(cudaEventElapsedTime(&e, ev[0], ev[1]));
    CK(cudaEventElapsedTime(&j, ev[2], ev[3]));
    CK(cudaEventElapsedTime(&d, ev[3], ev[4]));
    acc[0] += f; acc[1] += e; acc[3] += j; acc[4] += d;
  }
  for (int i = 0; i < 5; ++i) out[i] = (float)(acc[i] / h->ev_used);
  h->ev_used = 0;
  h->ev = nullptr;
  return RNNT_B200_OK;
}

}  // extern "C"
