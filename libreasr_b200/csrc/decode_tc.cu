// Device-resident batched greedy RNN-T decode on the tcgen05 tensor cores (gemm_mode 1).
//
// Same loop as decode.cu (reference libreasr/lib/models.py:403-443 / 528-571): per lock-step
//   A  pp = W1p * g (utterances whose predictor output changed), z = tanh(pp + ep[b, t_b])
//   B  logits slice = W2 * z + b2 -> per-CTA (max, argmax, sum exp) partials
//   R  every CTA folds the partials and applies the blank / max_iters rule to its own copy
//      of the control state
//   C..  one phase per predictor layer (GRU cell + BatchNorm eval; layer 0 input = table lookup)
// but every contraction is a skinny tcgen05 GEMM in the formulation of lstm_tc.cu: the BATCH is
// on the MMA M axis with the hi rows stacked on the lo rows of the 3xFP16 split, the CTA's slice
// of weight rows [hi;lo] on N -- ONE tcgen05.mma per 16-deep k slice gives all four split
// products -- and both operands stream from their operand images (tc_common.cuh) with TMA bulk
// copies through one mbarrier ring.  All G = H / Uc CTAs take a slice of every phase.
//   warp 0     producer (TMA bulk copies; waits on the grid phase counter before touching an
//              activation image another CTA wrote)
//   warp 1     MMA issuer (one elected lane per stage)
//   warps 2-5  epilogue: TMEM -> smem exchange -> thread (b, rows) math; predictor state h, the
//              joint pre-activation pp and the control state live in registers / smem for the
//              whole decode; results are written straight into the next phase's operand image
// Grid-wide synchronisation = one release-add on a phase counter per phase.
#include <algorithm>

#include "kernels.h"
#include "tc_common.cuh"

namespace rnnt {
namespace {

constexpr int DT_THREADS = 224;   // warp 0 activation producer, 1 MMA, 2-5 epilogue, 6 weight producer
constexpr int DT_MAXB = 64;
constexpr int DT_MAX_RPT = 8;   // rows (or units) per epilogue thread

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_add(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

struct Ctrl {
  double nlp[DT_MAXB];
  int t[DT_MAXB], it[DT_MAXB], ntok[DT_MAXB], tok[DT_MAXB], n_eval[DT_MAXB], len[DT_MAXB];
  float red[4][DT_MAXB][4];   // partial (max, argmax, sumexp) exchange between the threads of one batch row
  unsigned char active[DT_MAXB], emit[DT_MAXB];
  int flags[3];               // any_emit, any_active of the current step; any pending fused arg max
  // LM fusion
  float j_mean[DT_MAXB], j_rstd[DT_MAXB], lm_mean[DT_MAXB], lm_rstd[DT_MAXB];   // standardisation constants (utils.py:162-164)
  int am[DT_MAXB];
  unsigned char pend[DT_MAXB], lm_valid[DT_MAXB];
};
constexpr float kLmMinVal = -10.0f;  // lm.py:15
constexpr float kLmStdEps = 1e-5f;   // utils.py:162
constexpr int DT_LM_UPT = 4;         // LM units per epilogue thread
__device__ __forceinline__ void standardize_consts(double s, double q, int n, float* mean, float* rstd) {
  const double m = s / n;
  double var = (q - s * m) / (n - 1);   // unbiased, torch.Tensor.std
  if (var < 0.0) var = 0.0;
  *mean = (float)m;
  *rstd = 1.0f / ((float)sqrt(var) + kLmStdEps);
}
__device__ __forceinline__ unsigned long long pack_key(float m, int idx) {   // orderable (value, lowest index wins ties)
  unsigned u = __float_as_uint(m);
  u ^= (u & 0x80000000u) ? 0xFFFFFFFFu : 0x80000000u;
  return ((unsigned long long)u << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)idx);
}

// n (1, 2 or 4) consecutive k of one image row as hi / lo halves
__device__ __forceinline__ void store_split(uint8_t* hi_tile, uint8_t* lo_tile, int r, int k, int n, const float* v) {
  __align__(8) __half hi[4];
  __align__(8) __half lo[4];
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (j < n) split_f16x3(v[j], hi[j], lo[j]);
  const uint32_t off = img_elem_offset(r, k);
  if (n == 4) {
    *reinterpret_cast<uint2*>(hi_tile + off) = *reinterpret_cast<const uint2*>(hi);
    *reinterpret_cast<uint2*>(lo_tile + off) = *reinterpret_cast<const uint2*>(lo);
  } else if (n == 2) {
    *reinterpret_cast<uint32_t*>(hi_tile + off) = *reinterpret_cast<const uint32_t*>(hi);
    *reinterpret_cast<uint32_t*>(lo_tile + off) = *reinterpret_cast<const uint32_t*>(lo);
  } else {
    *reinterpret_cast<__half*>(hi_tile + off) = hi[0];
    *reinterpret_cast<__half*>(lo_tile + off) = lo[0];
  }
}

// One GEMM of a phase: activation image x weight-slice image -> TMEM columns [col, col + 2*NC)
struct Gemm {
  const uint8_t* act;   // activation image (TR = Bpad8 tiles, [kb][part] contiguous)
  const uint8_t* w;     // this CTA's weight tiles ([kb][part] contiguous, NC rows each)
  int KB, NC, col;
  int gated;            // 1: the activation image was written in the phase just before (wait for the grid counter);
                        // 0: it is older (the recurrent state h of a predictor layer) and can stream immediately
};

// LM = true instantiates the LM shallow-fusion phases (LMFuser, reference libreasr/lib/lm.py:43-83): see the block
// comment at `lm_phase` below.  The LM = false instantiation is the plain greedy loop.
template <bool LM>
__global__ void __launch_bounds__(DT_THREADS, 1) decode_tc_kernel(DecodeTcArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024 - (smem_u32(smem_raw) & 1023)) & 1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cta = blockIdx.x, G = gridDim.x;
  const DecodeWeights& w = p.w;
  const int H = w.H, J = w.J, V = w.V, Lp = w.Lp;
  const int S = p.stages, KPS = p.kps, MM = p.mma_m, Bq = p.Bq, B = p.B, T = p.T;
  const uint32_t xr = (uint32_t)p.Bpad8 * 128;
  const uint32_t xkb = 2 * xr;                                  // activation bytes per k-block (hi | lo rows)
  const uint32_t wmax = (uint32_t)p.NC_max * 256;               // weight bytes per k-block reserved in a stage
  const uint32_t stage_bytes = (uint32_t)KPS * (xkb + wmax);
  uint8_t* ring = base;
  float* pre_hi = reinterpret_cast<float*>(base + p.pre_offset);
  const int prs = 4 * p.NC_max + 1;                             // exchange row stride (two GEMMs of 2*NC_max columns)
  float* pre_lo = pre_hi + Bq * prs;
  Ctrl& c = *reinterpret_cast<Ctrl*>(base + p.ctl_offset);
  uint64_t* full = reinterpret_cast<uint64_t*>(base + p.bar_offset);   // activation part of a stage landed
  uint64_t* fullw = full + S;                                          // weight part of a stage landed
  uint64_t* empty = fullw + S;
  uint64_t* tfull = empty + S;
  uint64_t* tempty = tfull + 1;
  uint64_t* ctlbar = tempty + 1;
  uint64_t* tfull_r = ctlbar + 1;    // speculative recurrent products (all predictor layers) complete
  uint64_t* tempty_r = tfull_r + 1;  // ... and drained by the predictor phases that consumed them
  uint64_t* tfull_l = tempty_r + 1;  // LM accumulators (layer products / output projection) complete
  uint64_t* tempty_l = tfull_l + 1;  // ... and drained
  uint64_t* ctlack = tempty_l + 1;   // the three GEMM-side warps have read the control flags of a step
  uint32_t* tptr = reinterpret_cast<uint32_t*>(ctlack + 1);
  const int nB = (V + p.NC_B - 1) / p.NC_B;                     // CTAs that produce a softmax partial

  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&fullw[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tfull, 1);
    mbar_init(tempty, 128);
    mbar_init(ctlbar, 1);
    mbar_init(tfull_r, 1);
    mbar_init(tempty_r, 128);
    mbar_init(tfull_l, 1);
    mbar_init(tempty_l, 128);
    mbar_init(ctlack, 3);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tptr, p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tptr;

  // ---- per-phase slices of this CTA (CTAs beyond the slice count sit a phase out but keep the barriers) ----
  const int KBH = H / 64, KBJ = J / 64;
  const bool in_A = cta * p.NC_A < J, in_B = cta * p.NC_B < V;   // GRU phases: every CTA owns Uc units
  const uint8_t* wA = p.w1p_img + img_tile_offset(cta, 0, 0, KBH, p.NC_A);
  const uint8_t* wB = p.w2_img + img_tile_offset(cta, 0, 0, KBJ, p.NC_B);

  // The three roles walk the same phase sequence; `phase_gemms` describes the GEMMs of a phase.
  //   phase 0 = A (pp), 1 = B (logits), 2 + l = predictor layer l.  par = parity of the h images.
  auto phase_gemms = [&](int phase, int par, Gemm (&gm)[2]) -> int {
    if (phase == 0) {
      if (!in_A) return 0;
      gm[0] = Gemm{p.g_img, wA, KBH, p.NC_A, 0, 1};
      return 1;
    }
    if (phase == 1) {
      if (!in_B) return 0;
      gm[0] = Gemm{p.z_img, wB, KBJ, p.NC_B, 0, 1};
      return 1;
    }
    // predictor layer l: only the input product x * K_l (l > 0), which needs BatchNorm(h_{l-1}) of this run; layer 0's
    // input is a table row.  The recurrent products are speculative (rec_gemm below).
    const int l = phase - 2;
    if (l == 0) return 0;
    gm[0] = Gemm{p.x_img[(l - 1) & 1], p.k_img[l] + img_tile_offset(cta, 0, 0, KBH, p.NC_C), KBH, p.NC_C, 0, 1};
    return 1;
  };
  // The recurrent product h_l * R_l of every predictor layer depends only on state written by the PREVIOUS predictor
  // run, so it is issued speculatively right after phase B's operands -- before the greedy rule of this step is known --
  // into its own TMEM columns.  It overlaps B's epilogue, the barrier and the rule; when no utterance emits, the
  // products stay valid (h unchanged) and are consumed by the next predictor run.
  auto rec_gemm = [&](int l, int par) -> Gemm {
    return Gemm{p.h_img[l][par], p.r_img[l] + img_tile_offset(cta, 0, 0, KBH, p.NC_C), KBH, p.NC_C, p.rec_col0 + l * p.rec_cols, 0};
  };
  // ---- LM (lm.py:20-41): G_l CTAs own Ul units (NC_L = 4 Ul gate rows) of every LSTM layer; the output projection is
  // sliced over the vocabulary exactly like phase B.  LM accumulators live in their own TMEM block [lm_col0, ...):
  // input product at +0, recurrent product at +2 NC_L; the output projection reuses +0.
  const DecodeTcLm& lm = p.lm;
  const int Ll = LM ? lm.L : 0, KBL = LM ? lm.Hl / 64 : 0;
  const bool in_L = LM && cta < p.G_l;
  auto lm_rec_gemm = [&](int l, int lpar) -> Gemm {   // h_l of the previous LM run: not gated
    return Gemm{lm.h_img[l][lpar], lm.r_img[l] + img_tile_offset(cta, 0, 0, KBL, p.NC_L), KBL, p.NC_L, p.lm_col0 + 2 * p.NC_L, 0};
  };
  auto lm_in_gemm = [&](int l, int lpar) -> Gemm {    // h_{l-1} of THIS run (written one phase ago): gated
    return Gemm{lm.h_img[l - 1][lpar ^ 1], lm.w_img[l] + img_tile_offset(cta, 0, 0, KBL, p.NC_L), KBL, p.NC_L, p.lm_col0, 1};
  };
  auto lm_out_gemm = [&](int lpar) -> Gemm {          // top layer's h of the run just finished: gated
    return Gemm{lm.h_img[Ll - 1][lpar], lm.wo_img + img_tile_offset(cta, 0, 0, KBL, p.NC_B), KBL, p.NC_B, p.lm_col0, 1};
  };

  if (warp == 0 || warp == 6) {
    // =========================== producers ===========================
    // warp 0 streams ACTIVATION tiles (gated by the grid phase counter: another CTA wrote them);
    // warp 6 streams WEIGHT tiles of the same stages and is never gated, so at a phase boundary the
    // next phase's weight slices (up to S stages) are already landing while the barrier propagates.
    const bool acts = warp == 0;
    uint32_t g = 0;
    unsigned nbar = 1;   // grid barriers to wait for before a phase reads activations (1 = initial images)
    unsigned seen = 0;   // highest grid-barrier count this warp has observed
    auto gate = [&](unsigned n) {
      if (acts && seen < n) {
        while (ld_acquire_u32(p.barrier) < n * (unsigned)G) {
        }
        fence_proxy_async_global();
        seen = n;
      }
    };
    auto run_gemm = [&](const Gemm& gq) {
      const uint32_t wkb = (uint32_t)gq.NC * 256;
      for (int kb0 = 0; kb0 < gq.KB; kb0 += KPS, ++g) {
        const int s = g % S;
        const uint32_t ph = (g / S) & 1;
        mbar_wait(&empty[s], ph ^ 1);
        if (elect_one()) {
          const int nkb = min(KPS, gq.KB - kb0);
          uint8_t* dst = ring + (size_t)s * stage_bytes;
          if (acts) {
            mbar_arrive_expect_tx(&full[s], (uint32_t)nkb * xkb);
            tma_bulk_g2s(dst, gq.act + (size_t)kb0 * xkb, (uint32_t)nkb * xkb, &full[s]);
          } else {
            mbar_arrive_expect_tx(&fullw[s], (uint32_t)nkb * wkb);
            tma_bulk_g2s(dst + KPS * xkb, gq.w + (size_t)kb0 * wkb, (uint32_t)nkb * wkb, &fullw[s]);
          }
        }
        __syncwarp();
      }
    };
    auto run_phase = [&](int phase, int par) {
      Gemm gm[2];
      const int ng = phase_gemms(phase, par, gm);
      for (int q = 0; q < ng; ++q) {
        if (gm[q].gated) gate(nbar);
        run_gemm(gm[q]);
      }
      ++nbar;
    };
    unsigned hgate = 1;   // barrier count after which the current h images are complete
    auto run_spec = [&](int par) {
      gate(hgate);
      for (int l = 0; l < Lp; ++l) run_gemm(rec_gemm(l, par));
    };
    int par = 0, lpar = 0;
    bool lm_pending = false;   // an LM run finished; its output projection rides on the next phase A
    gate(1);   // the initial operand images (written by every CTA's epilogue warps) precede even the ungated GEMMs
    // one grid phase of a predictor (+ LM) run: layer i of both
    auto run_layer_phase = [&](int i, bool with_lm) {
      Gemm gm[2];
      if (i < Lp) {
        const int ng = phase_gemms(2 + i, par, gm);
        for (int q = 0; q < ng; ++q) { gate(nbar); run_gemm(gm[q]); }
      }
      if (LM && with_lm && i < Ll && in_L) {
        gate(hgate);
        run_gemm(lm_rec_gemm(i, lpar));
        if (i > 0) { gate(nbar); run_gemm(lm_in_gemm(i, lpar)); }
      }
      ++nbar;
    };
    if (!p.use_state_in) {
      run_spec(par);
      for (int l = 0; l < Lp; ++l) run_layer_phase(l, false);
      par ^= 1;
      hgate = nbar;
    }
    bool any_upd = true, spec_valid = false;
    for (int step = 0;; ++step) {
      if (any_upd) {
        Gemm gm[2];
        const int ng = phase_gemms(0, par, gm);
        for (int q = 0; q < ng; ++q) { gate(nbar); run_gemm(gm[q]); }
        if (LM && lm_pending && in_B) { gate(nbar); run_gemm(lm_out_gemm(lpar)); }
        lm_pending = false;
      }
      ++nbar;
      run_phase(1, par);
      if (!spec_valid) { run_spec(par); spec_valid = true; }
      mbar_wait(ctlbar, step & 1);
      const bool any_emit = c.flags[0] != 0, any_active = c.flags[1] != 0;
      const bool any_pend = LM && c.flags[2] != 0;
      __syncwarp();
      if (lane == 0) mbar_arrive(ctlack);   // the epilogue may now publish the next step's flags
      if (any_pend) ++nbar;   // the fused-arg-max barrier of this step (no GEMM)
      if (any_emit) {
        const int nph = (LM && Ll > Lp) ? Ll : Lp;
        for (int i = 0; i < nph; ++i) run_layer_phase(i, true);
        par ^= 1;
        hgate = nbar;
        spec_valid = false;
        if (LM) { lpar ^= 1; lm_pending = true; }
      }
      any_upd = any_emit;
      if (!any_active) break;
    }
    if (LM && lm_pending) {   // the fuser must hold the row of the last emitted token (lm.py:50-54)
      if (in_B) { gate(nbar); run_gemm(lm_out_gemm(lpar)); }
      ++nbar;
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===========================
    const uint64_t a_desc0 = umma_desc_sw128(smem_u32(ring));
    const uint64_t b_desc0 = umma_desc_sw128(smem_u32(ring) + KPS * xkb);
    const uint32_t stage_u = stage_bytes >> 4, xkb_u = xkb >> 4;
    uint32_t g = 0, nacc = 0, nspec = 0;
    // issue one GEMM into its TMEM columns; `done` (nullable) is committed with the last stage
    auto run_gemm = [&](const Gemm& gq, uint64_t* done) {
      const uint32_t idesc = umma_idesc_f16(MM, 2 * gq.NC);
      const uint32_t wkb_u = ((uint32_t)gq.NC * 256) >> 4;
      const uint32_t dcol = tmem + (uint32_t)gq.col;
      for (int kb0 = 0; kb0 < gq.KB; kb0 += KPS, ++g) {
        const int s = g % S;
        const uint32_t ph = (g / S) & 1;
        mbar_wait(&fullw[s], ph);
        mbar_wait(&full[s], ph);
        tc_fence_after();
        if (elect_one()) {
          const int nkb = min(KPS, gq.KB - kb0);
          uint64_t ad = a_desc0 + (uint64_t)(s * stage_u);
          uint64_t bd = b_desc0 + (uint64_t)(s * stage_u);
          uint32_t accumulate = kb0 == 0 ? 0u : 1u;
          for (int i = 0; i < nkb; ++i) {
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4) {
              tc_mma_f16(dcol, ad + 2 * k4, bd + 2 * k4, idesc, accumulate);
              accumulate = 1u;
            }
            ad += xkb_u;
            bd += wkb_u;
          }
          tc_commit(&empty[s]);
          if (done && kb0 + KPS >= gq.KB) tc_commit(done);
        }
        __syncwarp();
      }
    };
    auto run_phase = [&](int phase, int par) {
      Gemm gm[2];
      const int ng = phase_gemms(phase, par, gm);
      if (ng == 0) return;
      // the previous phase's accumulators must be drained before they are overwritten
      if (nacc > 0) mbar_wait(tempty, (nacc - 1) & 1);
      tc_fence_after();
      for (int q = 0; q < ng; ++q) run_gemm(gm[q], q == ng - 1 ? tfull : nullptr);
      ++nacc;
    };
    auto run_spec = [&](int par) {   // the recurrent columns are free once the predictor run that read them has drained
      if (nspec > 0) mbar_wait(tempty_r, (nspec - 1) & 1);
      tc_fence_after();
      for (int l = 0; l < Lp; ++l) run_gemm(rec_gemm(l, par), l == Lp - 1 ? tfull_r : nullptr);
      ++nspec;
    };
    uint32_t nacc_l = 0;
    // LM accumulators: one (tfull_l, tempty_l) hand-over per LM layer phase / output projection
    auto lm_begin = [&]() {
      if (nacc_l > 0) mbar_wait(tempty_l, (nacc_l - 1) & 1);
      tc_fence_after();
      ++nacc_l;
    };
    int par = 0, lpar = 0;
    bool lm_pending = false;
    auto run_layer_phase = [&](int i, bool with_lm) {
      if (i < Lp) run_phase(2 + i, par);
      if (LM && with_lm && i < Ll && in_L) {
        lm_begin();
        run_gemm(lm_rec_gemm(i, lpar), i == 0 ? tfull_l : nullptr);
        if (i > 0) run_gemm(lm_in_gemm(i, lpar), tfull_l);
      }
    };
    if (!p.use_state_in) {
      run_spec(par);
      for (int l = 0; l < Lp; ++l) run_layer_phase(l, false);
      par ^= 1;
    }
    bool any_upd = true, spec_valid = false;
    for (int step = 0;; ++step) {
      if (any_upd) {
        run_phase(0, par);
        if (LM && lm_pending && in_B) { lm_begin(); run_gemm(lm_out_gemm(lpar), tfull_l); }
        lm_pending = false;
      }
      run_phase(1, par);
      if (!spec_valid) { run_spec(par); spec_valid = true; }
      mbar_wait(ctlbar, step & 1);
      const bool any_emit = c.flags[0] != 0, any_active = c.flags[1] != 0;
      __syncwarp();
      if (lane == 0) mbar_arrive(ctlack);
      if (any_emit) {
        const int nph = (LM && Ll > Lp) ? Ll : Lp;
        for (int i = 0; i < nph; ++i) run_layer_phase(i, true);
        par ^= 1;
        spec_valid = false;
        if (LM) { lpar ^= 1; lm_pending = true; }
      }
      any_upd = any_emit;
      if (!any_active) break;
    }
    if (LM && lm_pending && in_B) { lm_begin(); run_gemm(lm_out_gemm(lpar), tfull_l); }
  } else {
    // =========================== epilogue ===========================
    const int q = warp & 3;
    const int et = (warp - 2) * 32 + lane;               // 0..127
    const int tpr = 128 / Bq;                            // threads per batch row (4 or 2)
    const int b = et % Bq, sub = et / Bq;
    const bool bvalid = b < B;
    const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);
    const int rows_per_warp = MM == 64 ? 16 : 32;
    uint32_t nacc = 0;

    // control state (identical in every CTA)
    for (int i = et; i < DT_MAXB; i += 128) {
      const int len = (i < B) ? (p.lens_T ? min(p.lens_T[i], T) : T) : 0;
      c.len[i] = len; c.t[i] = 0; c.it[i] = 0; c.ntok[i] = 0; c.n_eval[i] = 0; c.nlp[i] = 0.0;
      c.tok[i] = w.bos; c.active[i] = len > 0; c.emit[i] = i < B;
    }

    // TMEM accumulator rows -> exchange buffers (row r < Bpad8: hi row of batch r, else lo row of batch r - Bpad8).
    // A GEMM with NC rows occupies 2*NC columns: [0,NC) x*hi, [NC,2NC) x*lo.
    auto copy_cols = [&](int tcol, int ncols /*multiple of 8*/, int dstoff) {
      const int r = q * rows_per_warp + lane;
      if (q * rows_per_warp < 2 * p.Bpad8) {
        const bool mine = lane < rows_per_warp && r < 2 * p.Bpad8;
        const bool is_lo = r >= p.Bpad8;
        float* dstrow = (is_lo ? pre_lo + (r - p.Bpad8) * prs : pre_hi + r * prs) + dstoff;
        const float sc = is_lo ? kLoInv : 1.0f;
        for (int c0 = 0; c0 < ncols; c0 += 16) {
          float d[16];
          tmem_ld16(tlane + (uint32_t)(tcol + c0), d);
          tmem_ld_wait();
          if (mine) {
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (c0 + i < ncols) dstrow[c0 + i] = sc * d[i];
          }
        }
      }
    };
    auto drain = [&](int ncols) {   // the phase GEMM at column 0
      mbar_wait(tfull, nacc & 1);
      tc_fence_after();
      copy_cols(0, ncols, 0);
      tc_fence_before();
      mbar_arrive(tempty);
      ++nacc;
      named_bar_sync(1, 128);
    };
    uint32_t nspec = 0;
    // predictor layer l: input product (l > 0, column 0 -> exchange [0, 2NC)) and the speculative recurrent product
    // (its own columns -> exchange [2NC, 4NC))
    auto drain_pred = [&](int l) {
      const int NC = p.NC_C;
      if (l == 0) mbar_wait(tfull_r, nspec & 1);
      if (l > 0) mbar_wait(tfull, nacc & 1);
      tc_fence_after();
      if (l > 0) copy_cols(0, 2 * NC, 0);
      copy_cols(p.rec_col0 + l * p.rec_cols, 2 * NC, 2 * NC);
      tc_fence_before();
      if (l > 0) { mbar_arrive(tempty); ++nacc; }
      if (l == Lp - 1) { mbar_arrive(tempty_r); ++nspec; }
      named_bar_sync(1, 128);
    };
    // value of GEMM `gi` (NC rows at TMEM column base gi*2*NC), row `rr`, batch b:  hi-row and lo-row pieces summed
    auto pre_val = [&](int gbase, int NC, int rr) -> float {
      const float* ph = pre_hi + b * prs + gbase;
      const float* pl = pre_lo + b * prs + gbase;
      return (ph[rr] + kLoInv * ph[NC + rr]) + (pl[rr] + kLoInv * pl[NC + rr]);
    };
    unsigned ebar = 0;   // grid arrivals so far (same count in every CTA)
    // The phase counter only ever grows, and "barrier k complete" is tested as counter >= k * G.  That is only sound
    // if no CTA makes its (k+1)-th arrival before barrier k is complete -- otherwise early arrivals stand in for late
    // ones.  A CTA that consumed a gated operand in this phase has waited by data dependence; a CTA that SAT THE PHASE
    // OUT (no slice of it, e.g. cta * NC_A >= J) has not, and must check the previous barrier itself (`waited` false).
    auto grid_arrive = [&](bool waited = true) {
      named_bar_sync(1, 128);
      if (et == 0) {
        if (!waited)
          while (ld_acquire_u32(p.barrier) < ebar * (unsigned)G) {
          }
        red_release_add(p.barrier, 1u);
      }
      ++ebar;
    };
    auto grid_wait = [&]() {   // every CTA has made its ebar-th arrival
      if (et == 0) {
        while (ld_acquire_u32(p.barrier) < ebar * (unsigned)G) {
        }
      }
      named_bar_sync(1, 128);
    };

    // ---- persistent per-thread state ----
    const int rptA = p.NC_A * Bq / 128, rptB = p.NC_B * Bq / 128, upt = p.Uc * Bq / 128;
    const int jA0 = cta * p.NC_A + sub * rptA, vB0 = cta * p.NC_B + sub * rptB, unit0 = cta * p.Uc + sub * upt;
    float ppv[DT_MAX_RPT];
    float hst[kMaxPredLayers][DT_MAX_RPT];
    float gval[DT_MAX_RPT];
#pragma unroll
    for (int i = 0; i < DT_MAX_RPT; ++i) { ppv[i] = 0.f; gval[i] = 0.f; }
#pragma unroll
    for (int l = 0; l < kMaxPredLayers; ++l)
#pragma unroll
      for (int i = 0; i < DT_MAX_RPT; ++i)
        hst[l][i] = (l < Lp && i < upt && bvalid)
                        ? (p.use_state_in ? p.state_h[((size_t)l * p.state_ld + b) * H + unit0 + i] : w.h0[l][unit0 + i]) : 0.f;
    auto store_act = [&](uint8_t* img, int k0, int n, const float* v) {   // n consecutive k of batch row b
#pragma unroll
      for (int j0 = 0; j0 < DT_MAX_RPT; j0 += 4) {
        if (j0 < n) {
          const int k = k0 + j0;
          uint8_t* hi = img + (size_t)((k >> 6) * 2) * xr;
          store_split(hi, hi + xr, b, k & 63, (n - j0) < 4 ? (n - j0) : 4, v + j0);
        }
      }
    };
    int par = 0;
    // initial operand images: h of every layer (and g when the caller supplied the state)
    if (bvalid) {
      for (int l = 0; l < Lp; ++l) store_act(p.h_img[l][0], unit0, upt, hst[l]);
      if (p.use_state_in) {
#pragma unroll
        for (int i = 0; i < DT_MAX_RPT; ++i)
          if (i < upt) gval[i] = p.pred_out[(size_t)b * H + unit0 + i];
        store_act(p.g_img, unit0, upt, gval);
      }
    }
    // ---- LM fuser state (lm.py:43-48): per-thread slices kept in shared memory, column et of each array ----
    //   lmh / lmc [Ll][upt_l][128]   hidden / cell state of this thread's (b, units)
    //   lmv / lvj [rptB][128]        LM logits / joint logits of this thread's (b, vocabulary rows)
    //   dred [4][DT_MAXB][2]         double exchange between the threads of one batch row
    const int upt_l = LM ? p.Ul * Bq / 128 : 0;
    const int lunit0 = cta * p.Ul + sub * upt_l;
    float* lmh = reinterpret_cast<float*>(base + p.lm_offset);
    float* lmc = lmh + Ll * upt_l * 128;
    float* lmv = lmc + Ll * upt_l * 128;
    float* lvj = lmv + rptB * 128;
    double* dred = reinterpret_cast<double*>(lvj + rptB * 128);
    uint32_t nacc_l = 0;
    int lpar = 0, lm_runs = 0;   // LM runs whose output projection has been folded into lmv / lmstat
    bool lm_pending = false;
    if constexpr (LM) {
      const int Bp = lm.Bp, Hl = lm.Hl;
      for (int i = et; i < DT_MAXB; i += 128) {
        const bool v = i < B && lm.st.valid[i] != 0.f;
        c.lm_valid[i] = v;
        c.lm_mean[i] = v ? lm.st.stats[i] : 0.f;
        c.lm_rstd[i] = v ? lm.st.stats[Bp + i] : 0.f;
        c.pend[i] = 0;
      }
      if (in_L) {
        for (int l = 0; l < Ll; ++l) {
          float hv[DT_LM_UPT];
#pragma unroll
          for (int i = 0; i < DT_LM_UPT; ++i) {
            if (i < upt_l) {
              const size_t si = (size_t)(lunit0 + i) * Bp + b;
              hv[i] = bvalid ? lm.st.h[(size_t)l * 2 * Hl * Bp + si] : 0.f;
              lmh[(l * upt_l + i) * 128 + et] = hv[i];
              lmc[(l * upt_l + i) * 128 + et] = bvalid ? lm.st.c[(size_t)l * Hl * Bp + si] : 0.f;
            }
          }
          if (bvalid) store_act(lm.h_img[l][0], lunit0, upt_l, hv);
        }
      }
      if (in_B)
        for (int i = 0; i < rptB; ++i)
          lmv[i * 128 + et] = (bvalid && vB0 + i < V) ? lm.st.logits[(size_t)(vB0 + i) * Bp + b] : 0.f;
    }
    grid_arrive();

    // ---- predictor layer l (GRU cell + BatchNorm), haste/nbrc.py:46-56 ----
    auto predictor_phase = [&](int l) {
      const int NC = p.NC_C;
      // operands that do not depend on the accumulators are fetched before they are awaited
      const bool em = bvalid && c.emit[b] != 0;
      float vxin[DT_MAX_RPT][3], rbv[DT_MAX_RPT][3];
      if (em) {
#pragma unroll
        for (int i = 0; i < DT_MAX_RPT; ++i) {
          if (i < upt) {
            const int unit = unit0 + i;
            if (l == 0) {   // Embedding -> Linear -> kernel_0 folded into a [V][3H] table (models.py:182-183)
              const float* row = w.table0 + (size_t)c.tok[b] * (3 * H);
              vxin[i][0] = row[unit]; vxin[i][1] = row[H + unit]; vxin[i][2] = row[2 * H + unit];
            } else {
#pragma unroll
              for (int gg = 0; gg < 3; ++gg) vxin[i][gg] = w.kbias[l][unit * 3 + gg];
            }
#pragma unroll
            for (int gg = 0; gg < 3; ++gg) rbv[i][gg] = w.rbias[l][unit * 3 + gg];
          }
        }
      }
      drain_pred(l);
      const int gh = 2 * NC;   // exchange column base of the recurrent product
      float xo[DT_MAX_RPT];
      if (bvalid) {
#pragma unroll
        for (int i = 0; i < DT_MAX_RPT; ++i) {
          if (i < upt) {
            const int unit = unit0 + i, lr = (sub * upt + i) * 3;
            if (em) {
              float vx[3];
#pragma unroll
              for (int gg = 0; gg < 3; ++gg) vx[gg] = (l == 0) ? vxin[i][gg] : pre_val(0, NC, lr + gg) + vxin[i][gg];
              const float* rb = rbv[i];
              const float z = sigmoidf_acc(vx[0] + (pre_val(gh, NC, lr + 0) + rb[0]));
              const float r = sigmoidf_acc(vx[1] + (pre_val(gh, NC, lr + 1) + rb[1]));
              const float gg_ = tanhf(vx[2] + r * (pre_val(gh, NC, lr + 2) + rb[2]));
              hst[l][i] = z * hst[l][i] + (1.0f - z) * gg_;
            }
            xo[i] = hst[l][i] * w.bn_scale[l][unit] + w.bn_shift[l][unit];
          }
        }
        store_act(p.h_img[l][par ^ 1], unit0, upt, hst[l]);
        if (l == Lp - 1) {
#pragma unroll
          for (int i = 0; i < DT_MAX_RPT; ++i) gval[i] = xo[i];
          store_act(p.g_img, unit0, upt, xo);
        } else {
          store_act(p.x_img[l & 1], unit0, upt, xo);
        }
      }
    };
    // ---- LM layer l (torch.nn.LSTM cell, gate order i,f,g,o; lm.py:23,33-36), sharing a grid phase with predictor
    // layer l.  Only streams that emitted a token this step advance (LMFuser.advance, lm.py:50-54); layer 0's input
    // projection is a row of the Embedding * W_ih0 table. ----
    auto lm_phase = [&](int l, bool after_pred) {
      if (!in_L) return;
      const int NC = p.NC_L, Hl = lm.Hl;
      const bool em = bvalid && c.emit[b] != 0;
      float vxin[DT_LM_UPT][4];
      if (em) {
#pragma unroll
        for (int i = 0; i < DT_LM_UPT; ++i) {
          if (i < upt_l) {
            const int unit = lunit0 + i;
            if (l == 0) {
              const float* row = lm.table0 + (size_t)c.tok[b] * (4 * Hl);
#pragma unroll
              for (int gg = 0; gg < 4; ++gg) vxin[i][gg] = row[gg * Hl + unit];
            } else {
#pragma unroll
              for (int gg = 0; gg < 4; ++gg) vxin[i][gg] = lm.bias[l][unit * 4 + gg];
            }
          }
        }
      }
      if (after_pred) named_bar_sync(1, 128);   // the predictor part has finished reading the exchange buffers
      mbar_wait(tfull_l, nacc_l & 1);
      tc_fence_after();
      if (l > 0) copy_cols(p.lm_col0, 2 * NC, 0);
      copy_cols(p.lm_col0 + 2 * NC, 2 * NC, 2 * NC);
      tc_fence_before();
      mbar_arrive(tempty_l);
      ++nacc_l;
      named_bar_sync(1, 128);
      if (bvalid) {
        float hv[DT_LM_UPT];
#pragma unroll
        for (int i = 0; i < DT_LM_UPT; ++i) {
          if (i < upt_l) {
            const int lr = (sub * upt_l + i) * 4, si = (l * upt_l + i) * 128 + et;
            float h = lmh[si];
            if (em) {
              float v[4];
#pragma unroll
              for (int gg = 0; gg < 4; ++gg)
                v[gg] = ((l == 0) ? vxin[i][gg] : pre_val(0, NC, lr + gg) + vxin[i][gg]) + pre_val(2 * NC, NC, lr + gg);
              const float ig = sigmoidf_acc(v[0]), fg = sigmoidf_acc(v[1]), gg_ = tanhf(v[2]), og = sigmoidf_acc(v[3]);
              const float cn = fg * lmc[si] + ig * gg_;
              lmc[si] = cn;
              h = og * tanhf(cn);
              lmh[si] = h;
            }
            hv[i] = h;
          }
        }
        store_act(lm.h_img[l][lpar ^ 1], lunit0, upt_l, hv);
      }
    };
    // LM output projection (lm.py:37-40) for this CTA's vocabulary rows: raw logits (log_softmax is a per-row shift
    // that standardisation removes) + the (sum, sum of squares) the fuser standardises with (utils.py:162-164)
    auto lm_out_epilogue = [&](bool after_other) {
      if (!in_B) return;
      if (after_other) named_bar_sync(1, 128);
      mbar_wait(tfull_l, nacc_l & 1);
      tc_fence_after();
      copy_cols(p.lm_col0, 2 * p.NC_B, 0);
      tc_fence_before();
      mbar_arrive(tempty_l);
      ++nacc_l;
      named_bar_sync(1, 128);
      double sd = 0.0, qd = 0.0;
      if (bvalid) {
        for (int i = 0; i < rptB; ++i) {
          const int v = vB0 + i;
          if (v < V) {
            const float x = pre_val(0, p.NC_B, sub * rptB + i) + lm.bo[v];
            lmv[i * 128 + et] = x;
            sd += (double)x; qd += (double)x * (double)x;
          }
        }
        dred[(sub * DT_MAXB + b) * 2] = sd; dred[(sub * DT_MAXB + b) * 2 + 1] = qd;
      }
      named_bar_sync(1, 128);
      if (bvalid && sub == 0) {
        for (int k = 1; k < tpr; ++k) { sd += dred[(k * DT_MAXB + b) * 2]; qd += dred[(k * DT_MAXB + b) * 2 + 1]; }
        atomicAdd(lm.lmstat + ((size_t)lm_runs * Bq + b) * 2, sd);
        atomicAdd(lm.lmstat + ((size_t)lm_runs * Bq + b) * 2 + 1, qd);
      }
    };
    auto layer_phase = [&](int i, bool with_lm) {
      if (i < Lp) predictor_phase(i);
      if (LM && with_lm && i < Ll) lm_phase(i, i < Lp);
      // layer 0 follows an explicit grid wait (the rule R) or, for the BOS run, consumes operands gated on the initial
      // images; deeper layers wait through their gated input product -- unless this CTA has none in this phase
      grid_arrive(i == 0 || i < Lp || (LM && with_lm && i < Ll && in_L));
    };

    if (!p.use_state_in) {   // feed BOS from the learnable initial state (models.py:397-398); the LM only sees emitted tokens
      for (int l = 0; l < Lp; ++l) layer_phase(l, false);
      par ^= 1;
    }

    bool any_upd = true;
    for (int step = 0;; ++step) {
      // ---------------- phase A: pp and z ----------------
      float epv[DT_MAX_RPT];
      const bool actA = in_A && bvalid && c.active[b] != 0;
      if (actA) {   // issued before the accumulators are awaited
        const float* epr = p.ep + ((size_t)b * T + c.t[b]) * J + jA0;
#pragma unroll
        for (int i = 0; i < DT_MAX_RPT; ++i)
          if (i < rptA) epv[i] = epr[i];
      }
      if (any_upd && in_A) drain(2 * p.NC_A);
      if (in_A && bvalid) {
        float zv[DT_MAX_RPT];
        const bool act = actA;
#pragma unroll
        for (int i = 0; i < DT_MAX_RPT; ++i) {
          if (i < rptA) {
            if (any_upd && c.emit[b]) ppv[i] = pre_val(0, p.NC_A, sub * rptA + i);
            zv[i] = act ? tanhf(ppv[i] + epv[i]) : 0.f;
          }
        }
        if (act) store_act(p.z_img, jA0, rptA, zv);
      }
      const bool waited_A = !any_upd /* the rule's grid wait was the last barrier */ || in_A || (LM && lm_pending && in_B);
      if (LM && lm_pending) {   // rides on phase A: the row the fuser holds for the tokens emitted last step
        lm_out_epilogue(any_upd && in_A);
        ++lm_runs;
        lm_pending = false;
      }
      grid_arrive(waited_A);

      // ---------------- phase B: logits slice + softmax partials ----------------
      if (in_B) {
        drain(2 * p.NC_B);
        float m = -INFINITY, s = 0.f;
        int am = 0;
        if (bvalid) {
          float lv[DT_MAX_RPT];
#pragma unroll
          for (int i = 0; i < DT_MAX_RPT; ++i) {
            if (i < rptB) {
              const int v = vB0 + i;
              lv[i] = (v < V) ? pre_val(0, p.NC_B, sub * rptB + i) + w.b2[v] : -INFINITY;
              if (lv[i] > m) { m = lv[i]; am = v; }
            }
          }
#pragma unroll
          for (int i = 0; i < DT_MAX_RPT; ++i)
            if (i < rptB && vB0 + i < V) s += expf(lv[i] - m);
          if (p.trace && c.active[b] && c.n_eval[b] < p.trace_cap) {
            float* tr = p.trace + ((size_t)b * p.trace_cap + c.n_eval[b]) * V + vB0;
#pragma unroll
            for (int i = 0; i < DT_MAX_RPT; ++i)
              if (i < rptB && vB0 + i < V) tr[i] = lv[i];
          }
          c.red[sub][b][0] = m; c.red[sub][b][1] = __int_as_float(am); c.red[sub][b][2] = s;
          if constexpr (LM) {   // the fuser standardises the joint row too (lm.py:59-61)
            double sd = 0.0, qd = 0.0;
            for (int i = 0; i < rptB; ++i) {
              if (vB0 + i < V) {
                lvj[i * 128 + et] = lv[i];
                sd += (double)lv[i]; qd += (double)lv[i] * (double)lv[i];
              }
            }
            dred[(sub * DT_MAXB + b) * 2] = sd; dred[(sub * DT_MAXB + b) * 2 + 1] = qd;
          }
        }
        named_bar_sync(1, 128);
        if (LM && bvalid && sub == 0 && c.active[b] && step < p.max_steps) {
          double sd = 0.0, qd = 0.0;
          for (int k = 0; k < tpr; ++k) { sd += dred[(k * DT_MAXB + b) * 2]; qd += dred[(k * DT_MAXB + b) * 2 + 1]; }
          atomicAdd(lm.jstat + ((size_t)step * Bq + b) * 2, sd);
          atomicAdd(lm.jstat + ((size_t)step * Bq + b) * 2 + 1, qd);
        }
        if (bvalid && sub == 0) {
          for (int k = 1; k < tpr; ++k) {   // ascending vocabulary order, strict > keeps the first maximum
            const float m2 = c.red[k][b][0], s2 = c.red[k][b][2];
            if (m2 > m) { s = s * expf(m - m2) + s2; m = m2; am = __float_as_int(c.red[k][b][1]); }
            else s += s2 * expf(m2 - m);
          }
          // (max, sum exp) of this CTA's slice goes to the per-step log (log-probabilities are finished by a
          // post-pass, off the critical path); the arg max -- all the control flow needs -- is one 64-bit
          // atomicMax on a packed (orderable logit, ~index) key: lowest index wins ties like torch.max
          if (c.active[b] && step < p.max_steps) {
            *reinterpret_cast<float2*>(p.part + (((size_t)step * nB + cta) * Bq + b) * 2) = make_float2(m, s);
            unsigned u = __float_as_uint(m);
            u ^= (u & 0x80000000u) ? 0xFFFFFFFFu : 0x80000000u;
            atomicMax(p.keys + (size_t)step * Bq + b, ((unsigned long long)u << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)am));
          }
        }
      }
      grid_arrive(in_B);
      grid_wait();   // every CTA's atomicMax has landed

      // ---------------- R: greedy rule (models.py:408-437), identical in every CTA ----------------
      {
        const int kstep = min(step, p.max_steps - 1);
        // the flags are a single-slot mailbox: the GEMM-side warps must have read the previous step's before they
        // are overwritten (and before ctlbar can complete another phase)
        if (step > 0) mbar_wait(ctlack, (step - 1) & 1);
        if (et < B) {
          const int bb = et;
          c.pend[bb] = 0;
          if (c.active[bb]) {
            const unsigned long long key = __ldcg(p.keys + (size_t)kstep * Bq + bb);
            const int am2 = (int)(0xFFFFFFFFu - (unsigned)(key & 0xFFFFFFFFull));
            c.am[bb] = am2;
            if constexpr (LM) {
              // LMFuser.fuse applies to a non-blank decision once the fuser holds an LM row (models.py:427-431, lm.py:58)
              if (am2 != w.blank && c.lm_valid[bb]) {
                const double* js = lm.jstat + ((size_t)kstep * Bq + bb) * 2;
                standardize_consts(__ldcg(js), __ldcg(js + 1), V, &c.j_mean[bb], &c.j_rstd[bb]);
                if (lm_runs > 0) {   // else: the row carried in by the stream state, constants already in c.lm_mean / c.lm_rstd
                  const double* ls = lm.lmstat + ((size_t)(lm_runs - 1) * Bq + bb) * 2;
                  standardize_consts(__ldcg(ls), __ldcg(ls + 1), V, &c.lm_mean[bb], &c.lm_rstd[bb]);
                }
                c.pend[bb] = 1;
              }
            }
          }
        }
        if constexpr (LM) {
          named_bar_sync(1, 128);
          if (et == 0) {
            int ap = 0;
            for (int i = 0; i < B; ++i) ap |= c.pend[i];
            c.flags[2] = ap;
          }
          named_bar_sync(1, 128);
          if (c.flags[2]) {
            // ---- F: arg max of alpha * std(lm row) + theta * std(joint row), entry 0 of both rows pinned to -10
            //      (lm.py:54,59-77); this thread's vocabulary rows, then one packed atomicMax per stream ----
            if (in_B) {
              const bool on = bvalid && c.pend[b];
              float m = -INFINITY;
              int am = 0;
              if (on) {
                const float lmean = c.lm_mean[b], lrstd = c.lm_rstd[b], jmean = c.j_mean[b], jrstd = c.j_rstd[b];
                for (int i = 0; i < rptB; ++i) {
                  const int v = vB0 + i;
                  if (v < V) {
                    float a = (lmv[i * 128 + et] - lmean) * lrstd;
                    float j = (lvj[i * 128 + et] - jmean) * jrstd;
                    if (v == 0) { a = kLmMinVal; j = kLmMinVal; }
                    const float f = __fadd_rn(__fmul_rn(lm.alpha, a), __fmul_rn(lm.theta, j));
                    if (f > m) { m = f; am = v; }
                  }
                }
                c.red[sub][b][0] = m; c.red[sub][b][1] = __int_as_float(am);
              }
              named_bar_sync(1, 128);
              if (on && sub == 0) {
                for (int k = 1; k < tpr; ++k) {
                  const float m2 = c.red[k][b][0];
                  if (m2 > m) { m = m2; am = __float_as_int(c.red[k][b][1]); }
                }
                atomicMax(lm.fkeys + (size_t)kstep * Bq + b, pack_key(m, am));
              }
            }
            grid_arrive();
            grid_wait();
            if (et < B && c.pend[et]) {
              const unsigned long long key = __ldcg(lm.fkeys + (size_t)kstep * Bq + et);
              c.am[et] = (int)(0xFFFFFFFFu - (unsigned)(key & 0xFFFFFFFFull));
            }
            named_bar_sync(1, 128);
          }
        }
        if (et < B) {
          const int bb = et;
          unsigned char emit = 0;
          if (c.active[bb]) {
            const int am2 = c.am[bb], t = c.t[bb];
            c.n_eval[bb] += 1;
            const int it = c.it[bb] + 1;
            bool advance;
            if (am2 == w.blank && !c.pend[bb]) {
              advance = true;
            } else {
              const int n = c.ntok[bb];
              if (cta == 0 && n < p.U_cap) p.tokens[(size_t)bb * p.U_cap + n] = am2;
              c.ntok[bb] = n + 1;
              c.tok[bb] = am2;
              emit = 1;
              if (LM) c.lm_valid[bb] = 1;   // the LM advances on this token (lm.py:50-54)
              advance = it >= p.max_iters;
            }
            if (advance) {
              if (cta == 0 && p.iters) p.iters[(size_t)bb * T + t] = (uint8_t)it;
              c.t[bb] = t + 1;
              c.it[bb] = 0;
              if (t + 1 >= c.len[bb]) c.active[bb] = 0;
            } else {
              c.it[bb] = it;
            }
          }
          c.emit[bb] = emit;
        }
        named_bar_sync(1, 128);
        if (et == 0) {
          int ae = 0, aa = 0;
          for (int i = 0; i < B; ++i) { ae |= c.emit[i]; aa |= c.active[i]; }
          c.flags[0] = ae; c.flags[1] = aa;
          if (!LM) c.flags[2] = 0;
          mbar_arrive(ctlbar);
        }
        named_bar_sync(1, 128);
      }
      const bool any_emit = c.flags[0] != 0, any_active = c.flags[1] != 0;
      if (any_emit) {
        const int nph = (LM && Ll > Lp) ? Ll : Lp;
        for (int i = 0; i < nph; ++i) layer_phase(i, true);
        par ^= 1;
        if (LM) { lpar ^= 1; lm_pending = true; }
      }
      any_upd = any_emit;
      if (!any_active) break;
    }
    if (LM && lm_pending) {   // the fuser must hold the row of the last emitted token (lm.py:50-54)
      lm_out_epilogue(false);
      ++lm_runs;
      grid_arrive(in_B);
      grid_wait();
    }

    // ---- results and state ----
    if (cta == 0 && et < B) {
      p.ntok[et] = c.ntok[et];
      p.n_eval[et] = c.n_eval[et];
    }
    if (bvalid) {
      if (p.state_h)
        for (int l = 0; l < Lp; ++l)
#pragma unroll
          for (int i = 0; i < DT_MAX_RPT; ++i)
            if (i < upt) p.state_h[((size_t)l * p.state_ld + b) * H + unit0 + i] = hst[l][i];
      if (p.pred_out)
#pragma unroll
        for (int i = 0; i < DT_MAX_RPT; ++i)
          if (i < upt) p.pred_out[(size_t)b * H + unit0 + i] = gval[i];
    }
    if constexpr (LM) {   // fuser state back into the blob (buffer 0 of h), same layout as the fp32 kernel's
      const int Bp = lm.Bp, Hl = lm.Hl;
      if (in_L && bvalid)
        for (int l = 0; l < Ll; ++l)
          for (int i = 0; i < upt_l; ++i) {
            const size_t si = (size_t)(lunit0 + i) * Bp + b;
            lm.st.h[(size_t)l * 2 * Hl * Bp + si] = lmh[(l * upt_l + i) * 128 + et];
            lm.st.c[(size_t)l * Hl * Bp + si] = lmc[(l * upt_l + i) * 128 + et];
          }
      if (in_B && bvalid)
        for (int i = 0; i < rptB; ++i)
          if (vB0 + i < V) lm.st.logits[(size_t)(vB0 + i) * Bp + b] = lmv[i * 128 + et];
      if (cta == 0 && et < B) {
        lm.st.valid[et] = c.lm_valid[et] ? 1.f : 0.f;
        if (lm_runs > 0) {
          const double* ls = lm.lmstat + ((size_t)(lm_runs - 1) * Bq + et) * 2;
          standardize_consts(__ldcg(ls), __ldcg(ls + 1), V, &c.lm_mean[et], &c.lm_rstd[et]);
        }
        lm.st.stats[et] = c.lm_mean[et];
        lm.st.stats[Bp + et] = c.lm_rstd[et];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, p.tmem_cols);
}

// Post-pass, off the decode loop's critical path: fold the per-step softmax partials into the
// log-sum-exp of every evaluation (ascending vocabulary order, as the fp32 kernel does), accumulate
// -sum(log p(arg max)) per utterance (models.py:422,455) and turn the traced raw logits into log_softmax rows.
__global__ void __launch_bounds__(1024) decode_finish_kernel(const float* __restrict__ part, const int* __restrict__ n_eval,
                                                            int nB, int Bq, int max_steps, double* __restrict__ neg_logp,
                                                            float* __restrict__ lse_out, int lse_cap) {
  // one block (32 warps) per utterance, one warp per evaluation; lanes fold contiguous runs of the vocabulary partials and are
  // combined in a fixed shuffle tree (deterministic)
  const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ne = min(n_eval[b], max_steps);
  const int per = (nB + 31) / 32;
  double acc = 0.0;
  const int nwarps = blockDim.x >> 5;
  for (int e = warp; e < ne; e += nwarps) {
    float M = -INFINITY, S = 0.f;
    for (int k = lane * per; k < min(nB, (lane + 1) * per); ++k) {
      const float2 q = *reinterpret_cast<const float2*>(part + (((size_t)e * nB + k) * Bq + b) * 2);
      if (q.x > M) { S = S * expf(M - q.x) + q.y; M = q.x; }
      else S += q.y * expf(q.x - M);
    }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {   // lane l absorbs lane l + o
      const float M2 = __shfl_down_sync(0xffffffffu, M, o), S2 = __shfl_down_sync(0xffffffffu, S, o);
      if ((lane & (2 * o - 1)) == 0 && lane + o < 32) {
        if (M2 > M) { S = (M == -INFINITY ? 0.f : S * expf(M - M2)) + S2; M = M2; }
        else if (M2 != -INFINITY) S += S2 * expf(M2 - M);
      }
    }
    if (lane == 0) {
      const float lse = M + logf(S);
      acc += (double)(M - lse);
      if (lse_out && e < lse_cap) lse_out[(size_t)b * lse_cap + e] = lse;
    }
  }
  __shared__ double red[32];
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0 && neg_logp) {
    double t = 0.0;
    for (int w = 0; w < nwarps; ++w) t += red[w];
    neg_logp[b] = -t;
  }
}

__global__ void trace_normalize_kernel(float* trace, const float* lse, int B, int cap, int V) {
  const size_t n = (size_t)B * cap * V;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    trace[i] -= lse[i / V];   // rows never evaluated hold 0 - 0
}

}  // namespace

cudaError_t configure_decode_tc() {
  cudaError_t e = cudaFuncSetAttribute(decode_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(decode_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

// weight-side plan (independent of the batch): slices per CTA
bool decode_tc_wplan(int H, int J, int V, int sms, DecodeTcPlan* pl, int lm_layers, int lm_hidden) {
  if (H % 64 || J % 64) return false;
  int Uc = 0;
  for (int u : {8, 16, 32})
    if (H % u == 0 && H / u <= sms) { Uc = u; break; }
  if (!Uc) return false;
  pl->Uc = Uc;
  pl->G = H / Uc;
  pl->NC_C = 3 * Uc;
  pl->NC_A = (int)round_up(ceil_div(J, pl->G), 8);
  pl->NC_B = (int)round_up(ceil_div(V, pl->G), 8);
  pl->NC_max = std::max(pl->NC_C, std::max(pl->NC_A, pl->NC_B));
  pl->Ul = pl->NC_L = pl->G_l = 0;
  if (lm_layers > 0) {   // LM units per CTA: a multiple of 4 (whole units per epilogue thread at 2 or 4 threads per stream)
    if (lm_layers > kTcLmLayers || lm_hidden % 64) return false;
    for (int u = 4; u <= 16; u += 4)
      if (lm_hidden % u == 0 && lm_hidden / u <= pl->G) { pl->Ul = u; break; }
    if (!pl->Ul) return false;
    pl->NC_L = 4 * pl->Ul;
    pl->G_l = lm_hidden / pl->Ul;
    pl->NC_max = std::max(pl->NC_max, pl->NC_L);
  }
  return 2 * pl->NC_max <= 256;
}

bool decode_tc_plan(int H, int J, int V, int Lp, int B, int sms, DecodeTcPlan* pl, int lm_layers, int lm_hidden) {
  if (B < 1 || B > DT_MAXB) return false;
  if (!decode_tc_wplan(H, J, V, sms, pl, lm_layers, lm_hidden)) return false;
  pl->Bpad8 = (int)round_up(B, 8);
  pl->Bq = pl->Bpad8 <= 32 ? 32 : 64;
  pl->mma_m = 2 * pl->Bpad8 <= 64 ? 64 : 128;
  // rows per epilogue thread must be whole and small
  for (int n : {pl->NC_A, pl->NC_B, pl->Uc}) {
    if ((n * pl->Bq) % 128) return false;
    if (n * pl->Bq / 128 > DT_MAX_RPT) return false;
  }
  // TMEM columns: [0, rec_col0) the phase GEMM (A, B or a predictor layer's input product), then one block of
  // rec_cols per predictor layer for the speculative recurrent products
  pl->rec_col0 = (int)round_up(2 * pl->NC_max, 16);
  pl->rec_cols = (int)round_up(2 * pl->NC_C, 16);
  pl->lm_col0 = pl->rec_col0 + Lp * pl->rec_cols;
  const int lm_cols = lm_layers > 0 ? (int)round_up(std::max(4 * pl->NC_L, 2 * pl->NC_B), 16) : 0;
  if (lm_layers > 0 && pl->Ul * pl->Bq / 128 > DT_LM_UPT) return false;
  int cols = 32;
  while (cols < pl->lm_col0 + lm_cols) cols *= 2;
  if (Lp < 1 || Lp > kMaxPredLayers || cols > 512) return false;
  pl->tmem_cols = cols;
  const size_t xkb = (size_t)2 * pl->Bpad8 * 128, wmax = (size_t)pl->NC_max * 256;
  const size_t guard = (size_t)pl->mma_m * 128;
  const size_t pre_bytes = round_up((size_t)2 * pl->Bq * (4 * pl->NC_max + 1) * 4, 1024);
  const size_t ctl_bytes = round_up(sizeof(Ctrl), 1024);
  // LM per-thread state: lmh, lmc [Ll][upt_l][128], lmv, lvj [rptB][128] floats, dred [4][DT_MAXB][2] doubles
  const size_t lm_bytes = lm_layers > 0 ? round_up(((size_t)2 * lm_layers * (pl->Ul * pl->Bq / 128) + 2 * (pl->NC_B * pl->Bq / 128)) * 128 * 4 +
                                                       (size_t)4 * DT_MAXB * 2 * 8, 1024) : 0;
  const size_t budget = 227 * 1024 - 2048 - guard - pre_bytes - ctl_bytes - lm_bytes;
  for (int kps : {4, 2, 1}) {
    const size_t stage = kps * (xkb + wmax);
    int S = (int)(budget / stage);
    if (S > 8) S = 8;
    if (S < 3 && !(kps == 1 && S >= 2)) continue;
    pl->kps = kps;
    pl->stages = S;
    const size_t used = (size_t)S * stage + guard;
    pl->pre_offset = (int)round_up(used, 1024);
    pl->ctl_offset = pl->pre_offset + (int)pre_bytes;
    pl->lm_offset = pl->ctl_offset + (int)ctl_bytes;
    pl->bar_offset = pl->lm_offset + (int)lm_bytes;
    pl->smem_bytes = pl->bar_offset + 1024 + 1024;
    return pl->smem_bytes <= 227 * 1024;
  }
  return false;
}

// post-pass shared with decode_tc2.cu
cudaError_t launch_decode_finish(const float* part, const int* n_eval, int B, int nB, int Bq, int max_steps, double* neg_logp, float* trace,
                                 float* trace_lse, int trace_cap, int V, cudaStream_t st) {
  decode_finish_kernel<<<B, 1024, 0, st>>>(part, n_eval, nB, Bq, max_steps, neg_logp, trace ? trace_lse : nullptr, trace_cap);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if (trace) {
    trace_normalize_kernel<<<148, 256, 0, st>>>(trace, trace_lse, B, trace_cap, V);
    return cudaGetLastError();
  }
  return cudaSuccess;
}

cudaError_t launch_decode_tc(const DecodeTcArgs& a, const DecodeTcPlan& pl, cudaStream_t st) {
  DecodeTcArgs args = a;
  args.Uc = pl.Uc; args.NC_A = pl.NC_A; args.NC_B = pl.NC_B; args.NC_C = pl.NC_C; args.NC_max = pl.NC_max;
  args.Bpad8 = pl.Bpad8; args.Bq = pl.Bq; args.mma_m = pl.mma_m; args.kps = pl.kps; args.stages = pl.stages;
  args.pre_offset = pl.pre_offset; args.ctl_offset = pl.ctl_offset; args.bar_offset = pl.bar_offset; args.tmem_cols = pl.tmem_cols;
  args.rec_col0 = pl.rec_col0; args.rec_cols = pl.rec_cols;
  args.Ul = pl.Ul; args.NC_L = pl.NC_L; args.G_l = pl.G_l; args.lm_col0 = pl.lm_col0; args.lm_offset = pl.lm_offset;
  void* kargs[] = {&args};
  cudaError_t e = launch_persistent(a.lm.L > 0 ? (const void*)decode_tc_kernel<true> : (const void*)decode_tc_kernel<false>, dim3(pl.G), dim3(DT_THREADS), kargs, pl.smem_bytes, st);
  if (e != cudaSuccess) return e;
  const int nB = (int)ceil_div(a.w.V, pl.NC_B);
  decode_finish_kernel<<<a.B, 1024, 0, st>>>(a.part, a.n_eval, nB, pl.Bq, a.max_steps, a.neg_logp, a.trace ? a.trace_lse : nullptr, a.trace_cap);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if (a.trace) {
    trace_normalize_kernel<<<148, 256, 0, st>>>(a.trace, a.trace_lse, a.B, a.trace_cap, a.w.V);
    return cudaGetLastError();
  }
  return cudaSuccess;
}

}  // namespace rnnt
