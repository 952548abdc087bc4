// Internal launcher interface between the C-ABI layer (capi.cu) and the kernels.
#pragma once
#include "common.cuh"

namespace rnnt {

// The persistent kernels need their whole grid co-resident (they synchronise across CTAs).  The plans verify that against
// the occupancy of an empty GPU; the launches normally also carry the cooperative attribute.  The two-deep pipeline
// (capi.cu: rnnt_b200_pipeline_submit) launches them WITHOUT it: a cooperative launch from a high-priority stream next
// to a running lower-priority kernel (the front end of the next batch) was measured 4x slower per batch, while a plain
// launch just fills the SMs as the front-end blocks -- which never wait on anything -- retire.
// Thread-local: set by the calling thread around its launches.
bool coop_launch_enabled();
void set_coop_launch(bool on);
cudaError_t launch_persistent(const void* fn, dim3 grid, dim3 block, void** kargs, size_t smem, cudaStream_t st);

constexpr int kDecodeMaxBatchWords = 8;   // 256 streams / 32

// ---------------- frontend.cu ----------------
constexpr int kFrontendMaxWarps = 16;

struct FrontendArgs {
  const float* audio;      // [B, n]
  int64_t n;               // row stride (samples)
  const int32_t* lens;     // [B] valid samples or nullptr
  float* out;              // [B, T_out, n_mels*n_stack]
  int T_out;               // rows per utterance
  int frame0;              // first frame of row t is t*D + frame0
  int is_stream;           // 1: every row valid (serving window), 0: rows >= T_b are zero-filled
  int n_mels, n_stack, D, hop, win;
  const float* window;     // [win]
  const float2* tw;        // [512] exp(-2 pi i j / 1024)
  const int* mel_start;    // [n_mels] first non-zero FFT bin
  const int* mel_count;    // [n_mels] number of taps
  const int* mel_off;      // [n_mels] offset into mel_w
  const float* mel_w;      // taps
  float log_offset;
};
size_t frontend_smem_bytes(int n_stack, int n_mels);
cudaError_t launch_mel_stack(const FrontendArgs& a, int B, cudaStream_t st);
cudaError_t launch_resample(const float* x, int B, int64_t n, const float* tab, int n_orig, int n_new, int width, int K, float* out,
                            int64_t L, cudaStream_t st);
cudaError_t launch_layernorm(const float* in, float* out, const float* gamma, const float* beta, int64_t rows, int X,
                             float eps, cudaStream_t st);

// ---------------- gemm_simt.cu ----------------
// C[M,N] = A[M,K] * W[N,K]^T + bias[N]   (fp32 FMA; lda/ldw/ldc in elements, K % 4 == 0)
cudaError_t launch_gemm_nt_f32(const float* A, int lda, const float* W, int ldw, const float* bias, float* C, int ldc,
                               int64_t M, int N, int K, cudaStream_t st);
// out[c][r] = in[r*ld_in + c]   (out is dense [cols][rows])
cudaError_t launch_transpose(const float* in, int ld_in, float* out, int rows, int cols, cudaStream_t st);
// out[r][perm(c)] row/column permutations used by the weight repack (see capi.cu)
cudaError_t launch_gather_rows(const float* in, float* out, const int* src_row, int rows_out, int cols, cudaStream_t st);

// ---------------- gemm_tc.cu (tcgen05, 3xFP16 split) ----------------
cudaError_t configure_gemm_tc();
size_t gemm_tc_a_image_bytes(int64_t M, int K);   // activation operand image, 128-row tiles
size_t gemm_tc_w_image_bytes(int N, int K);       // weight operand image, 256-row tiles
// fp32 row-major [R][ld] -> hi/lo fp16 operand image with TR-row tiles (tc_common.cuh)
cudaError_t launch_to_image(const float* src, int ld, int64_t R, int K, int TR, uint8_t* img, cudaStream_t st);
// C[M,N] = A * W^T + bias from operand images (A: TR=128, W: TR=256)
cudaError_t launch_gemm_tc(const uint8_t* a_img, const uint8_t* w_img, const float* bias, float* C, int ldc, int64_t M, int N,
                           int K, cudaStream_t st);

// ---------------- lstm_tc.cu (persistent tcgen05 LSTM layer) ----------------
struct LstmTcPlan {
  int U, NC, grid, KB, Bpad8, stages, w_resident, bar_offset, smem_bytes, tmem_cols;
  int kps;         // k-blocks (64 k) per pipeline stage / TMA bulk copy
  int mma_m;       // MMA M: 64 when hi+lo rows of the batch fit (B <= 32), else 128
  int fused;       // B <= 64: [A_hi;A_lo] stacked in one A tile -> one tcgen05.mma per 16-deep k slice
  int pre_offset;  // smem offset of the accumulator exchange buffers (fused mode)
};
struct LstmTcArgs {
  const uint8_t* w_img;      // operand image (TR = NC) of the interleaved W_hh [4H][H]
  uint8_t* x_img[2];         // h_{t-1} / h_t operand images (TR = Bpad8 rows: [kb][part] contiguous), ping-pong
  const float* xp;           // [B*T][4H] hoisted input projection incl. biases
  const float* bn_scale; const float* bn_shift;
  float* y;                  // [B*T][H] BatchNorm(h_t) fp32, or nullptr
  uint8_t* y_img;            // operand image (TR = 128) of the same rows, or nullptr
  const int32_t* lens_T;
  const float* h_init_vec; const float* c_init_vec;   // [H] learnable initial state
  const float* state_h_in; const float* state_c_in;   // [B][H] or nullptr
  float* state_h_out; float* state_c_out;             // [B][H] or nullptr
  unsigned int* barrier;     // [H/64] per-k-block readiness counters, zero at launch
  int T, B, H;
  // filled from the plan by the launcher
  int U, NC, KB, Bpad8, stages, w_resident, bar_offset, tmem_cols, kps, mma_m, fused, pre_offset;
};
cudaError_t configure_lstm_tc();
bool lstm_tc_plan(int H, int B, int sms, LstmTcPlan* pl);
cudaError_t launch_lstm_layer_tc(const LstmTcArgs& a, const LstmTcPlan& pl, cudaStream_t st);

// ---------------- lstm_tc2.cu (persistent tcgen05 LSTM layer, cluster split-K over DSMEM) ----------------
struct LstmTc2Plan {
  int KS;          // k-blocks (64 k) of the K slice one CTA keeps resident (H / 256)
  int KB;          // H / 64
  int grid;        // H / 8 CTAs = H / 32 clusters of 4
  int smem_bytes;
};
struct LstmTc2Args {
  const uint8_t* w_img;      // operand image (TR = 128) of the interleaved W_hh [4H][H]
  uint8_t* x_img[2];         // h images: [H/64][hi|lo][32 rows x 128 B], tagged 16-byte chunks (see lstm_tc2.cu)
  const float* xp;           // [B*T][4H] hoisted input projection incl. biases, interleaved gate columns
  const float* bn_scale; const float* bn_shift;
  float* y;                  // [B*T][H] BatchNorm(h_t) fp32, or nullptr
  uint8_t* y_img;            // operand image (TR = 128) of the same rows, or nullptr
  const int32_t* lens_T;
  const float* h_init_vec; const float* c_init_vec;
  const float* state_h_in; const float* state_c_in;
  float* state_h_out; float* state_c_out;
  unsigned int* barrier;     // one launch-start counter, zero at launch
  unsigned long long* dbg;   // optional [T][4] globaltimer stamps of CTA 0, or nullptr
  unsigned long long* dbg_all;   // optional [grid][T][2] (publish, tiles complete) stamps of every CTA: skew diagnosis
  int T, B, H;
  int KS, KB;                // filled from the plan by the launcher
};
cudaError_t configure_lstm_tc2();
bool lstm_tc2_plan(int H, int B, int sms, LstmTc2Plan* pl);
cudaError_t launch_lstm_layer_tc2(const LstmTc2Args& a, const LstmTc2Plan& pl, cudaStream_t st);

// ---------------- lstm.cu ----------------
struct LstmStepArgs {
  const float* Whh_t;   // [H][4H] k-major, columns interleaved unit*4 + gate(i,f,g,o)
  const float* hT_in;   // [H][Bp]
  float* hT_out;        // [H][Bp]
  float* cT;            // [H][Bp] in/out
  const float* xp;      // [B*T][4H] hoisted input projection incl. both biases, interleaved columns
  const float* bn_scale;  // [H]
  const float* bn_shift;  // [H]
  float* y;             // [B*T][H] BatchNorm(h_t)
  const int32_t* lens_T;  // [B] or nullptr
  int t, T, B, Bp, H;
};
cudaError_t configure_lstm();
cudaError_t launch_lstm_step(const LstmStepArgs& a, cudaStream_t st);
// state layout helpers: [B,H] row-major <-> [H][Bp] feature-major
cudaError_t launch_state_to_T(const float* in_BH, float* out_HB, int B, int Bp, int H, cudaStream_t st);
cudaError_t launch_state_from_T(const float* in_HB, float* out_BH, int B, int Bp, int H, cudaStream_t st);
cudaError_t launch_state_broadcast_T(const float* vec_H, float* out_HB, int B, int Bp, int H, cudaStream_t st);
// steps[b] = min(T_max, encoder steps of an utterance with lens[b] samples)
cudaError_t launch_lens_to_steps(const int32_t* lens, int32_t* steps, int B, int hop, int n_stack, int D, int T_max,
                                 cudaStream_t st);

// ---------------- stream.cu (streaming session helpers) ----------------
struct StreamMask { uint32_t bits[kDecodeMaxBatchWords]; };   // one bit per stream
cudaError_t launch_slide_window(const float* w_old, float* w_new, const float* chunks, int B, int W, int ck, const StreamMask& active,
                                cudaStream_t st);
cudaError_t launch_store_rows(const float* row, float* rows, const int32_t* pos, int B, int X, int n_buffer, cudaStream_t st);

// ---------------- decode.cu ----------------
constexpr int kMaxPredLayers = 4;
constexpr int kDecodeMaxBatch = 256;

struct DecodeWeights {
  int H, J, V, Lp, blank, bos;
  const float* table0;          // [V][3H] gate-major (z|r|g): (embed*ffn)*kernel_0 + bias_0
  const float* Rt[kMaxPredLayers];     // [H][3H] k-major, columns unit*3 + gate
  const float* rbias[kMaxPredLayers];  // [3H] interleaved
  const float* Kt[kMaxPredLayers];     // layers >= 1: [H][3H] k-major interleaved
  const float* kbias[kMaxPredLayers];  // layers >= 1: [3H] interleaved
  const float* h0[kMaxPredLayers];     // [H] learnable initial state
  const float* bn_scale[kMaxPredLayers];
  const float* bn_shift[kMaxPredLayers];
  const float* W1p_t;           // [H][J]  pred half of joint.0, k-major
  const float* W1e_t;           // [H][J]  enc half of joint.0, k-major (standalone joint only)
  const float* b1;              // [J]
  const float* W2_t;            // [J][V]  k-major
  const float* b2;              // [V]
};

// Fused language model (reference libreasr/lib/lm.py:20-83); L == 0 means no LM.
constexpr int kMaxLmLayers = 8;
struct LmWeights {
  int L, Hl;
  float alpha, theta;
  const float* table0;              // [V][4Hl] gate-major (i|f|g|o): embed * W_ih0^T + b_ih0 + b_hh0
  const float* Wt[kMaxLmLayers];    // layers >= 1: [Hl][4Hl] k-major, columns unit*4 + gate
  const float* Rt[kMaxLmLayers];    // [Hl][4Hl] k-major interleaved
  const float* bias[kMaxLmLayers];  // layers >= 1: [4Hl] interleaved (b_ih + b_hh)
  const float* rbias0;              // unused (layer 0's biases live in table0)
  const float* Wo_t;                // [Hl][V] k-major output projection
  const float* bo;                  // [V]
};
// Per-stream fuser state, feature-major like the predictor state; all zero = fresh fuser (lm.py:81-83).
// Layout of the blob (floats): h [L][2][Hl][Bp] | c [L][Hl][Bp] | logits [V][Bp] | stats [2][Bp] | valid [Bp]
struct LmState {
  float* h; float* c; float* logits; float* stats; float* valid;
};
inline size_t lm_state_floats(int L, int Hl, int V, int Bp) { return ((size_t)3 * L * Hl + V + 3) * Bp; }
inline LmState lm_state_view(float* blob, int L, int Hl, int V, int Bp) {
  LmState s;
  s.h = blob;
  s.c = s.h + (size_t)2 * L * Hl * Bp;
  s.logits = s.c + (size_t)L * Hl * Bp;
  s.stats = s.logits + (size_t)V * Bp;
  s.valid = s.stats + (size_t)2 * Bp;
  return s;
}

struct DecodeArgs {
  DecodeWeights w;
  LmWeights lm;
  LmState lms;            // fuser state (workspace zeroed by the caller, or the registered stream blob)
  float* logitT;          // [V][Bp] joint logits of the current evaluation (LM fusion only)
  double* lmpart;         // [V/32][Bp][2] per-tile (sum, sum of squares) of the LM logits
  double* jpart;          // [V/32][Bp][2] ... of the joint logits of the current evaluation
  float* fpart;           // [V/32][Bp][2] per-tile (max, argmax) of the fused scores
  const float* ep;        // [B][T][J] enc half projection incl. b1
  const int32_t* lens_T;  // [B] or nullptr
  int B, Bp, T, max_iters, use_state_in;
  // feature-major state, ping-pong where a phase reads and writes the same vector
  float* hT[kMaxPredLayers][2];  // [H][Bp]
  float* xT;      // [2][H][Bp] BatchNorm output of the layer below (input of layers >= 1), ping-pong by layer parity
  float* gT;      // [H][Bp] predictor output (h_t_pred)
  float* ppT;     // [J][Bp] W1p * g
  float* zT;      // [J][Bp] tanh(pp + ep[t_b])
  float* part;    // [V/32][Bp][4] per-tile (max, argmax, sumexp, -) partials
  float* trace_lse;  // [B][trace_cap] log-sum-exp of every traced evaluation (workspace)
  // outputs
  int32_t* tokens; int U_cap; int32_t* ntok; double* neg_logp; uint8_t* iters; float* trace; int trace_cap;
};
size_t decode_smem_bytes();
cudaError_t configure_decode(int device, int* max_coop_blocks);
cudaError_t launch_decode(const DecodeArgs& a, int grid_blocks, cudaStream_t st);

// ---------------- decode_tc.cu (tcgen05 greedy decode) ----------------
struct DecodeTcPlan {
  int G, Uc, NC_A, NC_B, NC_C, NC_max;                 // weight-side plan (batch independent)
  int Bpad8, Bq, mma_m, kps, stages, pre_offset, ctl_offset, bar_offset, smem_bytes, tmem_cols, rec_col0, rec_cols;
  // fused language model (0 layers = none): G_l CTAs own Ul LM units (NC_L = 4*Ul gate rows) each
  int Ul, NC_L, G_l, lm_col0, lm_offset;
};
// LM side of the tcgen05 decode kernel (lm.py:20-83); L == 0: no LM
constexpr int kTcLmLayers = 6;
struct DecodeTcLm {
  int L, Hl;
  float alpha, theta;
  const float* table0;                 // [V][4Hl] gate-major: embed * W_ih0^T + b_ih0 + b_hh0
  const float* bias[kTcLmLayers];      // layers >= 1: [4Hl] interleaved (b_ih + b_hh)
  const float* bo;                     // [V]
  const uint8_t* r_img[kTcLmLayers];   // operand images (TR = NC_L) of the interleaved W_hh
  const uint8_t* w_img[kTcLmLayers];   // layers >= 1: ... of the interleaved W_ih
  const uint8_t* wo_img;               // output projection [V][Hl] (TR = NC_B)
  uint8_t* h_img[kTcLmLayers][2];      // activation images of the LM hidden state (ping-pong), TR = Bpad8
  LmState st;                          // fuser state blob (feature-major, ld = Bp); zero = fresh fuser
  int Bp;
  double* jstat;                       // [max_steps][Bq][2] (sum, sum of squares) of the joint logits per evaluation, zero at launch
  double* lmstat;                      // [max_steps][Bq][2] ... of the LM logits per LM run, zero at launch
  unsigned long long* fkeys;           // [max_steps][Bq] packed arg-max keys of the fused scores, zero at launch
};
struct DecodeTcArgs {
  DecodeTcLm lm;
  DecodeWeights w;                 // fp32 vectors / tables (table0, biases, h0, BatchNorm, b2)
  const uint8_t* w1p_img;          // operand images of the weight slices (TR = NC_A / NC_B / NC_C rows per CTA)
  const uint8_t* w2_img;
  const uint8_t* r_img[kMaxPredLayers];
  const uint8_t* k_img[kMaxPredLayers];
  const float* ep;                 // [B][T][J] encoder half of the joint incl. b1
  const int32_t* lens_T;
  int B, T, max_iters, use_state_in;
  uint8_t* g_img; uint8_t* z_img; uint8_t* x_img[2]; uint8_t* h_img[kMaxPredLayers][2];   // activation images (TR = Bpad8)
  float* part;                     // [max_steps][nB][Bq][2] per-step (max, sum exp) of every CTA's vocabulary slice
  unsigned long long* keys;        // [max_steps][Bq] packed arg-max keys (atomicMax), zero at launch
  int* n_eval;                     // [B] evaluations per utterance (out)
  int max_steps;
  float* trace_lse;
  float* state_h; float* pred_out; // [Lp][state_ld][H] (rows of this launch first), [B][H] in/out (nullable unless use_state_in)
  int state_ld;                    // batch stride of state_h per layer (= B unless the launch is a slice of a larger state)
  int32_t* tokens; int U_cap; int32_t* ntok; double* neg_logp; uint8_t* iters; float* trace; int trace_cap;
  unsigned int* barrier;           // grid phase counter, zero at launch
  // filled from the plan by the launcher
  int Uc, NC_A, NC_B, NC_C, NC_max, Bpad8, Bq, mma_m, kps, stages, pre_offset, ctl_offset, bar_offset, tmem_cols, rec_col0, rec_cols;
  int Ul, NC_L, G_l, lm_col0, lm_offset;
};
cudaError_t configure_decode_tc();
bool decode_tc_wplan(int H, int J, int V, int sms, DecodeTcPlan* pl, int lm_layers = 0, int lm_hidden = 0);
bool decode_tc_plan(int H, int J, int V, int Lp, int B, int sms, DecodeTcPlan* pl, int lm_layers = 0, int lm_hidden = 0);
cudaError_t launch_decode_tc(const DecodeTcArgs& a, const DecodeTcPlan& pl, cudaStream_t st);

// ---------------- decode_tc2.cu (tcgen05 greedy decode, cluster split-K over DSMEM, tagged exchange) ----------------
struct DecodeTc2Args {
  DecodeWeights w;                 // fp32 vectors / tables (table0, biases, h0, BatchNorm, b2)
  const uint8_t* w1p_img;          // operand images, row tiles of one cluster: TR = 32 (W1p), V/32 (W2), 96 (K1, R0, R1)
  const uint8_t* w2_img;
  const uint8_t* k1_img;
  const uint8_t* r_img[2];
  uint8_t* img[8];                 // tagged activation images g, BN(h0'), h0', h1', z of look-ahead frame 0, 1, ..: 2 buffers of img_stride bytes each
  int n_spec;                      // joint evaluations per utterance and lock-step (1 = none speculative); set by the launcher
  size_t img_stride;
  unsigned long long* keys;        // [2][128 CTAs][32] packed (logit, index, tag) arg-max keys
  const float* ep;                 // [B][T][J] encoder half of the joint incl. b1
  const int32_t* lens_T;
  int B, T, max_iters, use_state_in;
  float* part;                     // [max_steps][128][32][2] per-step (max, sum exp) of every CTA's vocabulary rows
  int* n_eval;                     // [B]
  int max_steps;
  float* trace_lse;
  float* state_h; float* pred_out; // [2][state_ld][H] (rows of this launch first), [B][H] in/out (nullable unless use_state_in)
  int state_ld;                    // batch stride of state_h per layer
  int32_t* tokens; int U_cap; int32_t* ntok; double* neg_logp; uint8_t* iters; float* trace; int trace_cap;
  unsigned int* barrier;           // launch-start counter, zero at launch
  unsigned long long* dbg; int dbg_cap;   // optional (time, tag) trail of CTA 0 (tuning aid)
};
cudaError_t configure_decode_tc2();
bool decode_tc2_plan(int H, int J, int V, int Lp, int B, int sms, int lm_layers);
size_t decode_tc2_image_bytes();   // one buffer of one activation image
size_t decode_tc2_keys_bytes();
int decode_tc2_part_ctas();
int decode_tc2_images();
cudaError_t launch_decode_tc2(const DecodeTc2Args& a, cudaStream_t st);

// ---------------- beam.cu (batched RNN-T beam search; algorithm defined by oracle/beam.py) ----------------
struct BeamHyp { double score; unsigned long long hash; int node; int valid; };
struct BeamLeave { double score; unsigned long long hash; int node; int gen; int slot; };
struct BeamArgs {
  DecodeWeights w;
  const float* ep;             // [B][T][J] encoder half of the joint incl. b1
  const int32_t* lens_T;
  int B, T, W, n_gen;          // n_gen = max_iters + 2 generation buffers
  float* state;                // [3 (h0, h1, g)][n_gen][B*W][H]
  BeamHyp* hyp;                // [n_gen][B*W]
  BeamLeave* leave; int leave_cap; int* n_leave;        // [B][leave_cap], [B]
  int* node_parent; int* node_token; int node_cap; int* n_nodes;   // per-utterance token trie
  float* cand_val; int* cand_idx; float* lp_blank;      // [B*W][W], [B*W][W], [B*W]
  int* sel_row; int* sel_tok;  // [B*W] parent row / token of the rows of the generation being built
  int* copy_src;               // [B*W]
};
struct BeamBuffers {
  uint8_t* a_img;              // activation operand image (128-row tiles) for up to B*W rows x max(H, J)
  const uint8_t *w1p_img, *w2_img, *k1_img, *r_img[2];   // 256-row-tile weight images (gemm_tc.cu)
  float *pp, *logits, *rec, *kin, *x1;
};
cudaError_t launch_beam_search(const BeamArgs& a, const BeamBuffers& bf, int max_iters, int32_t* tokens, int U_cap, int32_t* ntok, double* score,
                               int* launches, cudaStream_t st);

// ---------------- lattice.cu (training-time forward: joint lattice + RNN-T loss, eval mode) ----------------
cudaError_t launch_lattice_tokens(const int32_t* labels, int N, int Umax, int u, int bos, int32_t* out, cudaStream_t st);
cudaError_t launch_lattice_z_image(const float* pp, const float* ep, int T, int U, int64_t row0, int rows, int J, uint8_t* img, cudaStream_t st);
cudaError_t launch_lattice_lse(const float* logits, int rows, int V, int64_t row0, const int32_t* labels, int T, int U, int Umax, int blank,
                               float* lp_blank, float* lp_label, float* lattice_out, cudaStream_t st);
cudaError_t launch_lattice_gather(const float* lat, int64_t rows, int V, const int32_t* labels, int T, int U, int Umax, int blank, float* lp_blank,
                                  float* lp_label, cudaStream_t st);
cudaError_t launch_rnnt_alpha(const float* lp_blank, const float* lp_label, const int32_t* xl, const int32_t* yl, int N, int T, int U, double* loss,
                              cudaStream_t st);

// standalone predictor step / joint (same phase code, one launch per phase)
struct PredictArgs {
  DecodeWeights w;
  const int32_t* tokens;  // [B]
  int B, Bp, layer;
  const float* hT_in; float* hT_out;   // [H][Bp]
  const float* xT_in;     // layers >= 1
  float* xT_out;          // BN(h_new)
};
cudaError_t launch_gru_layer(const PredictArgs& a, cudaStream_t st);
struct JointArgs {
  DecodeWeights w;
  int B, Bp;
  const float* gT; const float* eT;   // [H][Bp]
  float* zT;                           // [J][Bp]
  float* logits;                       // [B][V]
};
cudaError_t launch_joint(const JointArgs& a, cudaStream_t st);

}  // namespace rnnt
