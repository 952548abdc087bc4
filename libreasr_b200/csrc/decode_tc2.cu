// Device-resident batched greedy RNN-T decode, cluster split-K formulation (gemm_mode 1, up to 32 utterances,
// H = J = 1024, two predictor layers, no fused LM; every other case keeps decode_tc.cu).
//
// Same loop as decode_tc.cu / decode.cu (reference libreasr/lib/models.py:403-443 / 528-571; predictor
// haste/nbrc.py:46-56; joint models.py:132-140) with the dependent GEMMs of a lock-step
//      A   pp = W1p g            z = tanh(pp + ep[b, t_b])
//      B   logits = W2 z + b2    -> arg max over the vocabulary -> greedy rule R
//      C0  GRU layer 0 (input = table row of the token, recurrent product R0 h0 speculative)
//      C1  GRU layer 1 (input product K1 BN(h0'), recurrent product R1 h1 speculative) -> g = BN(h1')
// re-partitioned like lstm_tc2.cu instead of "every CTA takes a slice of the rows and ingests the whole activation":
//   * 32 clusters of 4 CTAs.  Cluster c owns a block of output rows of every matrix (32 rows of W1p, V/32 of W2,
//     32 units = 96 interleaved gate rows of K1 / R0 / R1); CTA `rank` of the cluster holds the K-slice
//     [256 rank, 256 rank + 256) of those rows.  Weight rows sit on the MMA M axis (M = 64 / 128), the batch on N
//     ([h_hi ; h_lo] x W_hi, h_hi x W_lo: the 3xFP16 split of tc_common.cuh), so a GEMM job costs 32 tcgen05.mma and a
//     CTA ingests 32 KB of activations per job instead of 128 KB.
//   * Split-K reduction through distributed shared memory: every epilogue warp folds its TMEM lanes and writes the
//     32-batch partial rows into the owner CTA's shared memory (st.async, whose bytes complete a transaction count on
//     the owner's mbarrier); the owner (rank r owns rows [r R/4, (r+1) R/4) of the cluster's block) sums the four partial
//     tiles and finalises.
//   * Activations (g, z, BN(h0'), h0', h1') travel as tagged 16-byte chunks (tc2_common.cuh): published with one
//     st.relaxed.gpu.v4 by the finalising thread group, polled as data by the consumers' loader warps.  The per-step
//     arg max is exchanged the same way: every CTA publishes one packed (logit, index, tag) key per utterance, every CTA
//     reads the 128 x 32 table and reduces it: no atomics, no grid barrier anywhere in the loop.
//   * W2 (needed by every lock-step) stays resident in shared memory; W1p, K1, R0, R1 stream through a 3-stage TMA ring
//     ahead of their jobs.  The recurrent products R0 h0', R1 h1' are issued speculatively right after the predictor
//     run that produced h0' / h1' (jobs JR0 / JR1), their reduced rows wait in registers for the next emission.
//
//   warps 0-3  epilogue / finalise (TMEM -> fold -> DSMEM scatter -> sum -> cell / softmax partials / rule -> publish)
//   warps 4-7  loaders (tagged activation chunks -> 8 KB k-block stages of a 6-stage ring)
//   warp  8    MMA issuer (accumulators double-buffered in TMEM, 2 x 128 columns)
//   warp  9    weight streamer (TMA bulk copies, 24 KB k-block stages)
#include <algorithm>

#include <cstdlib>

#include "kernels.h"
#include "tc_common.cuh"
#include "tc2_common.cuh"

namespace rnnt {
namespace {

constexpr int D2_THREADS = 320;
constexpr int D2_CL = 4;          // CTAs per cluster = K slices
constexpr int D2_NCL = 32;        // clusters
constexpr int D2_G = D2_CL * D2_NCL;
constexpr int D2_NB = 32;         // batch rows (N tile: 32 hi + 32 lo)
constexpr int D2_KS = 4;          // k-blocks per K slice (K = 1024)
constexpr int D2_AST = 6;         // activation ring stages (8 KB each)
constexpr int D2_WST = 3;         // streamed-weight ring stages (24 KB each)
constexpr int D2_WSTAGE = 24576;
constexpr int D2_RP = 24;         // row stride of a partial tile (max rows finalised per CTA)
constexpr int D2_K = 1024;        // H = J

constexpr int D2_MAXS = 2;        // joint evaluations per utterance and lock-step (speculative look-ahead frames)
// Look-ahead frames evaluated per lock-step (<= D2_MAXS; measured on a B200: three frames are slower, 7.12 ms per batch).
constexpr int D2_SPEC = 2;
// Producers (of 8) of the polled line whose chunk must carry the new tag before a loader warp issues the loads of a
// K slice (fewer stale chunks to re-read).  Measured on a B200, ms per batch: 6.52 at 1, 6.36-6.39 at 5-7, 6.42 at 8.
constexpr int D2_TRIG = 6;
enum { IMG_G = 0, IMG_X = 1, IMG_H0 = 2, IMG_H1 = 3, IMG_Z0 = 4, IMG_N = 4 + D2_MAXS };
enum { JOB_A = 0, JOB_B = 1, JOB_K1 = 2, JOB_R0 = 3, JOB_R1 = 4 };

struct Ctrl2 {
  int t[D2_NB], it[D2_NB], ntok[D2_NB], tok[D2_NB], n_eval[D2_NB], len[D2_NB], am[D2_NB];
  unsigned char active[D2_NB], emit[D2_NB];
  int flags[2];                                  // any_emit, any_active of the current step
  unsigned long long kred[D2_MAXS][8][D2_NB];    // partial maxima of the key table, per look-ahead frame
  unsigned long long kbuf[D2_CL][D2_MAXS][D2_NB]; // cluster leader: the four CTAs' keys of a step (written through DSMEM)
};

__global__ void __launch_bounds__(D2_THREADS, 1) decode_tc2_kernel(DecodeTc2Args p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024 - (smem_u32(smem_raw) & 1023)) & 1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const int cta = blockIdx.x, cl = cta / D2_CL;
  const DecodeWeights& w = p.w;
  const int H = w.H, J = w.J, V = w.V, B = p.B, T = p.T;
  const int RB = V / D2_NCL;                      // W2 rows per cluster (<= 64)
  const int rpB = RB / D2_CL;                     // ... finalised per CTA (<= 16)
  // ---- shared memory ----
  uint8_t* W2s = base;                                             // [KS][hi RB x 128 B | lo RB x 128 B]
  const uint32_t w2kb = (uint32_t)RB * 256u;
  uint8_t* wring = W2s + 65536;                                    // D2_WST x 24 KB
  uint8_t* aring = wring + D2_WST * D2_WSTAGE + 4096;              // D2_AST x 8 KB (4 KB guard: an M=128 lo tile is read 16 KB deep)
  float* P = reinterpret_cast<float*>(aring + D2_AST * 8192);     // [2][4 src][32 b][24] fp32
  Ctrl2& c = *reinterpret_cast<Ctrl2*>(reinterpret_cast<uint8_t*>(P) + 2 * D2_CL * D2_NB * D2_RP * 4);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(&c) + ((sizeof(Ctrl2) + 15) & ~15));
  uint64_t* afull = bars;                 // [AST] loaders -> MMA (one arrive per loader warp)
  uint64_t* aempty = afull + D2_AST;      // [AST] MMA -> loaders
  uint64_t* wfull = aempty + D2_AST;      // [WST] TMA -> MMA
  uint64_t* wempty = wfull + D2_WST;      // [WST] MMA -> streamer
  uint64_t* tfull = wempty + D2_WST;      // [2]
  uint64_t* tempty = tfull + 2;           // [2] 128 arrivals
  uint64_t* pbar = tempty + 2;            // [2] partial tiles of a job complete: 16 warp arrivals (4 CTAs x 4 warps)
  uint64_t* pfree = pbar + 2;             // [2] partial tiles of a job consumed by their 4 owners: 16 warp arrivals
  uint64_t* w2full = pfree + 2;
  uint64_t* ctlbar = w2full + 1;          // flags of a step published
  uint64_t* ctlack = ctlbar + 1;          // ... and read by the 6 GEMM-side warps
  uint64_t* kbar = ctlack + 1;            // cluster leader: the keys of a step have arrived (transaction bytes)
  uint32_t* tptr = reinterpret_cast<uint32_t*>(kbar + 1);

  if (threadIdx.x == 0) {
    for (int i = 0; i < D2_AST; ++i) { mbar_init(&afull[i], 4); mbar_init(&aempty[i], 1); }
    for (int i = 0; i < D2_WST; ++i) { mbar_init(&wfull[i], 1); mbar_init(&wempty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 128);
      mbar_init(&pbar[i], 4);    // one arming arrive per epilogue warp
      mbar_init(&pfree[i], 16);
    }
    mbar_init(w2full, 1);
    mbar_init(ctlbar, 1);
    mbar_init(ctlack, 6);
    mbar_init(kbar, 4);   // armed by the four epilogue warps of the leader
    fence_mbar_init();
  }
  if (warp == 8) tmem_alloc(tptr, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  cluster_sync_all();
  const uint32_t tmem = *tptr;
  const size_t slice_off = (size_t)rank * D2_KS * 8192;   // this CTA's K slice inside an activation image

  // image `i`, write number n (0-based) lives in buffer n & 1 and carries tag (n >> 1) & 1
  auto img_ptr = [&](int i, unsigned n) -> uint8_t* { return p.img[i] + (size_t)(n & 1u) * p.img_stride; };

  // The four roles walk the same job sequence; these helpers keep the shared bookkeeping identical.
  //   job j: accumulators / partial tiles in buffer j & 1
  if (warp < 4) {
    // ======================================= epilogue / finalise =======================================
    const int q = warp;
    const uint32_t tl = tmem + ((uint32_t)(q * 32) << 16);
    const int et = warp * 32 + lane;
    const int fb = warp * 8 + (lane >> 2);      // batch row finalised by this thread
    const int fw = lane & 3;
    const bool bvalid = fb < B;
    const int u0 = cl * 32 + rank * 8;          // first unit / joint row finalised by this CTA
    const int unit = u0 + 2 * fw;
    const int vB0 = cl * RB + rank * rpB;       // first vocabulary row finalised by this CTA
    const int rptB = rpB / 4;                   // vocabulary rows per thread (1..4)
    const uint32_t off_hi = (uint32_t)((u0 >> 6) * 2) * 4096u + (uint32_t)fb * 128u + (uint32_t)((((u0 & 63) >> 3) ^ (fb & 7)) << 4);
    const uint32_t P_u32 = smem_u32(P);

    for (int i = et; i < D2_NB; i += 128) {
      const int len = (i < B) ? (p.lens_T ? min(p.lens_T[i], T) : T) : 0;
      c.len[i] = len; c.t[i] = 0; c.it[i] = 0; c.ntok[i] = 0; c.n_eval[i] = 0; c.am[i] = 0;
      c.tok[i] = w.bos; c.active[i] = len > 0; c.emit[i] = i < B;
    }
    // ---- persistent per-thread state ----
    float pp[2] = {0.f, 0.f}, gval[2] = {0.f, 0.f}, hst[2][2], rec[2][6];
    float bsc[2][2], bsh[2][2];
#pragma unroll
    for (int l = 0; l < 2; ++l)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        hst[l][i] = (bvalid && p.use_state_in) ? p.state_h[((size_t)l * p.state_ld + fb) * H + unit + i] : w.h0[l][unit + i];
        bsc[l][i] = w.bn_scale[l][unit + i];
        bsh[l][i] = w.bn_shift[l][unit + i];
      }
#pragma unroll
    for (int l = 0; l < 2; ++l)
#pragma unroll
      for (int i = 0; i < 6; ++i) rec[l][i] = 0.f;
    if (bvalid && p.use_state_in) {
      gval[0] = p.pred_out[(size_t)fb * H + unit];
      gval[1] = p.pred_out[(size_t)fb * H + unit + 1];
    }
    unsigned nw[IMG_N];                     // writes issued so far per image
#pragma unroll
    for (int i = 0; i < IMG_N; ++i) nw[i] = 0;
    const int NS = p.n_spec;
    unsigned nkeys = 0;                     // key-table writes so far
    // 8 consecutive k (the two values of the 4 lanes of a batch row) -> one hi and one lo 16-byte chunk, tagged
    auto publish = [&](int img, float v0, float v1) {
      const unsigned n = nw[img]++;
      uint8_t* dst = img_ptr(img, n);
      const uint32_t tag = (n >> 1) & 1u;
      uint32_t h0, l0, h1, l1;
      split_tag(v0, false, 0u, h0, l0);
      split_tag(v1, fw == 3, tag, h1, l1);
      const uint32_t hp = h0 | (h1 << 16), lp = l0 | (l1 << 16);
      const int g0 = lane & ~3;
      const uint32_t a0 = __shfl_sync(0xffffffffu, hp, g0), a1 = __shfl_sync(0xffffffffu, hp, g0 + 1);
      const uint32_t a2 = __shfl_sync(0xffffffffu, hp, g0 + 2), a3 = __shfl_sync(0xffffffffu, hp, g0 + 3);
      const uint32_t b0 = __shfl_sync(0xffffffffu, lp, g0), b1 = __shfl_sync(0xffffffffu, lp, g0 + 1);
      const uint32_t b2 = __shfl_sync(0xffffffffu, lp, g0 + 2), b3 = __shfl_sync(0xffffffffu, lp, g0 + 3);
      if (fw == 0) st_relaxed_v4(dst + off_hi, a0, a1, a2, a3);
      else if (fw == 1) st_relaxed_v4(dst + off_hi + 4096u, b0, b1, b2, b3);
    };
    // ---- launch start: every image buffer gets a defined tag (stale chunks of an earlier launch must not validate) ----
    {
      // write #0 of g / h0 / h1 = the initial state (tag 0 in buffer 0); buffer 1 and both buffers of z / x: tag 1
      publish(IMG_G, gval[0], gval[1]);
      publish(IMG_H0, hst[0][0], hst[0][1]);
      publish(IMG_H1, hst[1][0], hst[1][1]);
      const uint4 one = make_uint4(0u, 0u, 0u, 0x00010000u);
      if (fw < 2) {
        const uint32_t off = off_hi + (fw == 1 ? 4096u : 0u);
        st_relaxed_v4(p.img[IMG_G] + p.img_stride + off, one.x, one.y, one.z, one.w);
        st_relaxed_v4(p.img[IMG_H0] + p.img_stride + off, one.x, one.y, one.z, one.w);
        st_relaxed_v4(p.img[IMG_H1] + p.img_stride + off, one.x, one.y, one.z, one.w);
        for (int bf = 0; bf < 2; ++bf) {
          st_relaxed_v4(p.img[IMG_X] + (size_t)bf * p.img_stride + off, one.x, one.y, one.z, one.w);
#pragma unroll
          for (int zs = 0; zs < D2_MAXS; ++zs)
            if (zs < NS) st_relaxed_v4(p.img[IMG_Z0 + zs] + (size_t)bf * p.img_stride + off, one.x, one.y, one.z, one.w);
        }
      }
      // key table [2][NS][32 clusters][32 b] u64 (written by the cluster leaders): tag 1 (bit 0) everywhere
      if (et < 32 && rank == 0)
        for (int i = 0; i < 2 * NS; ++i) p.keys[((size_t)i * D2_NCL + cl) * D2_NB + et] = 1ull;
      __threadfence();
      named_bar_sync(1, 128);
      if (et == 0) {
        red_release_add(p.barrier, 1u);
        while (ld_acquire_u32(p.barrier) < (unsigned)D2_G) {
        }
      }
      named_bar_sync(1, 128);
    }

    unsigned job = 0;
    int ndbg = 0;
    auto stamp = [&](int tag) {
      if (p.dbg && cta == 0 && et == 0 && ndbg < p.dbg_cap) { p.dbg[2 * ndbg] = gtimer(); p.dbg[2 * ndbg + 1] = (unsigned long long)tag; ++ndbg; }
    };
    // Drain the accumulators of the current job, scatter this warp's rows to their owner CTAs, wait for the four
    // partial tiles of the rows this CTA owns.  M: MMA M of the job, rows: valid rows of the cluster, rp: rows per owner.
    // A GEMM job's epilogue in two halves so that consecutive jobs can overlap their waits:
    //   send_job: drain the accumulators of the next job, scatter this warp's rows to their owner CTAs      -> job index j
    //   wait_job: the four partial tiles of the rows this CTA owns have arrived                              -> this thread's batch row
    //   release_job: all reads of those tiles are done, hand the buffer back to the senders
    // M: MMA M of the job, rows: valid rows of the cluster, rp: rows per owner.
    auto send_job = [&](int M, int rows, int rp) -> unsigned {
      const unsigned j = job++;
      const int ab = (int)(j & 1u);
      const unsigned n = j >> 1;
      // every epilogue warp arms a quarter of the job's bytes (4 sources x rp rows x 32 x 4 B in total): the phase cannot
      // complete before all four warps have entered the job, so no warp can be lapped by the barrier
      if (lane == 0) mbar_arrive_expect_tx(&pbar[ab], (uint32_t)(D2_NB * rp * 4));
      mbar_wait(&tfull[ab], n & 1u);
      tc_fence_after();
      const int r = (M == 64) ? q * 16 + lane : q * 32 + lane;
      const bool mine = (M == 64 ? lane < 16 : true) && r < rows;
      const int dst_rank = mine ? r / rp : 0, lrow = mine ? r % rp : 0;
      const uint32_t dst = mapa(P_u32 + (uint32_t)((((ab * D2_CL + rank) * D2_NB) * D2_RP + lrow) * 4), (uint32_t)dst_rank);
      const uint32_t rbar = mapa(smem_u32(&pbar[ab]), (uint32_t)dst_rank);
      mbar_wait_cluster_relaxed(&pfree[ab], (n & 1u) ^ 1u);   // the owners have consumed the tiles of job j - 2
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        float d0[16], d1[16], d2[16];
        const uint32_t tc = tl + (uint32_t)(ab * 128 + hf * 16);
        tmem_ld16(tc, d0);          // W_hi * h_hi
        tmem_ld16(tc + 32, d1);     // W_hi * h_lo (x 2^11)
        tmem_ld16(tc + 64, d2);     // W_lo * h_hi (x 2^11)
        tmem_ld_wait();
        if (mine) {
#pragma unroll
          for (int b = 0; b < 16; ++b) st_async_f32(dst + (uint32_t)((hf * 16 + b) * D2_RP * 4), fmaf(d1[b] + d2[b], kLoInv, d0[b]), rbar);
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty[ab]);
      return j;
    };
    auto wait_job = [&](unsigned j) -> const float* {
      const int ab = (int)(j & 1u);
      mbar_wait(&pbar[ab], (j >> 1) & 1u);
      return P + (size_t)((ab * D2_CL) * D2_NB + fb) * D2_RP;   // + src * 32 * 24 ; this thread's batch row
    };
    auto release_job = [&](unsigned j) {
      const int ab = (int)(j & 1u);
      __syncwarp();
      if (lane < D2_CL) mbar_arrive_cluster_relaxed(mapa(smem_u32(&pfree[ab]), (uint32_t)lane));   // (the values read are already consumed: program order suffices)
    };
    auto sum2 = [&](const float* pr, int off, float* o, int nfl) {   // o[i] = sum over the 4 sources, nfl in {2, 4, 6}
#pragma unroll
      for (int s = 0; s < D2_CL; ++s) {
        const float* ps = pr + (size_t)s * D2_NB * D2_RP + off;
#pragma unroll
        for (int i = 0; i < 6; i += 2) {
          if (i < nfl) {
            const float2 v = *reinterpret_cast<const float2*>(ps + i);
            if (s == 0) { o[i] = v.x; o[i + 1] = v.y; } else { o[i] += v.x; o[i + 1] += v.y; }
          }
        }
      }
    };
    // speculative recurrent product of predictor layer l -> registers
    auto epi_rec = [&](int l) {
      const unsigned j = send_job(128, 96, 24);
      sum2(wait_job(j), fw * 6, rec[l], 6);
      release_job(j);
    };
    // predictor layer l (GRU cell + BatchNorm eval, haste/nbrc.py:46-56); vx = input pre-activations incl. bias
    auto gru_cell = [&](int l, const float (&vx)[6]) {
      const bool em = bvalid && c.emit[fb] != 0;
      if (em) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const float* rb = w.rbias[l] + (size_t)(unit + i) * 3;
          const float z = sigmoid_fast(vx[3 * i + 0] + (rec[l][3 * i + 0] + rb[0]));
          const float r = sigmoid_fast(vx[3 * i + 1] + (rec[l][3 * i + 1] + rb[1]));
          const float gg = tanh_fast(vx[3 * i + 2] + r * (rec[l][3 * i + 2] + rb[2]));
          hst[l][i] = z * hst[l][i] + (1.0f - z) * gg;
        }
      }
    };
    float vpre[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // table row of the token this thread's utterance is about to emit, fetched ahead of the rule
    auto load_table0 = [&](int tok, float (&vx)[6]) {   // Embedding -> Linear -> kernel_0 folded into a [V][3H] table (models.py:182-183)
      const float* row = w.table0 + (size_t)tok * (3 * H);
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        vx[3 * i + 0] = row[unit + i]; vx[3 * i + 1] = row[H + unit + i]; vx[3 * i + 2] = row[2 * H + unit + i];
      }
    };
    // tok_pre: the token whose row sits in vpre (-1: none).  The replay that produced it reads the control state without a
    // barrier against the rule, so it is only a hint: the row is used iff it is the row of the token the rule has recorded.
    auto phase_c0 = [&](int tok_pre) {
      float vx[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (bvalid && c.emit[fb]) {
        if (tok_pre == c.tok[fb]) {
#pragma unroll
          for (int i = 0; i < 6; ++i) vx[i] = vpre[i];
        } else {
          load_table0(c.tok[fb], vx);
        }
      }
      gru_cell(0, vx);
      // BN(h0') feeds JK1 on the dependent chain; h0' itself only the speculative recurrent product of the NEXT emission
      publish(IMG_X, hst[0][0] * bsc[0][0] + bsh[0][0], hst[0][1] * bsc[0][1] + bsh[0][1]);
      publish(IMG_H0, hst[0][0], hst[0][1]);
    };
    auto phase_c1 = [&]() {
      float kb[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) kb[i] = w.kbias[1][(size_t)unit * 3 + i];
      const unsigned j = send_job(128, 96, 24);
      float vx[6];
      sum2(wait_job(j), fw * 6, vx, 6);
      release_job(j);
#pragma unroll
      for (int i = 0; i < 6; ++i) vx[i] += kb[i];
      gru_cell(1, vx);
      gval[0] = hst[1][0] * bsc[1][0] + bsh[1][0];
      gval[1] = hst[1][1] * bsc[1][1] + bsh[1][1];
      publish(IMG_G, gval[0], gval[1]);       // g feeds JA on the dependent chain, h1' only the speculative JR1
      publish(IMG_H1, hst[1][0], hst[1][1]);
    };

    if (!p.use_state_in) {   // feed BOS from the learnable initial state (models.py:397-398)
      epi_rec(0);
      epi_rec(1);
      phase_c0(-1);
      phase_c1();
    }
    bool pending = true, any_upd = true;
    for (int step = 0;; ++step) {
      if (pending) epi_rec(0);
      // ---------------- phase A: pp and z ----------------
      // Look-ahead: z is formed for the current frame AND the next NS - 1 frames of every utterance (same predictor
      // state: valid as long as the earlier evaluations of this step come out blank, which ~75 % do), so the rule below can
      // consume up to NS joint evaluations per lock-step.  Every evaluation is the one the sequential loop would make.
      {
        const bool act = bvalid && c.active[fb] != 0;
        float2 epv[D2_MAXS];
        bool vs[D2_MAXS];
#pragma unroll
        for (int zs = 0; zs < D2_MAXS; ++zs) {
          vs[zs] = zs < NS && act && c.t[fb] + zs < c.len[fb];
          epv[zs] = make_float2(0.f, 0.f);
          if (vs[zs]) epv[zs] = *reinterpret_cast<const float2*>(p.ep + ((size_t)fb * T + c.t[fb] + zs) * J + unit);
        }
        if (any_upd) {
          const unsigned j = send_job(64, 32, 8);
          sum2(wait_job(j), fw * 2, pp, 2);
          release_job(j);
        }
#pragma unroll
        for (int zs = 0; zs < D2_MAXS; ++zs)
          if (zs < NS) publish(IMG_Z0 + zs, vs[zs] ? tanh_fast(pp[0] + epv[zs].x) : 0.f, vs[zs] ? tanh_fast(pp[1] + epv[zs].y) : 0.f);
      }
      stamp(0);
      if (pending) { epi_rec(1); pending = false; }
      // ---------------- phase B: logits of this CTA's vocabulary rows (one job per look-ahead frame), arg max exchange ----------------
      {
        float b2v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) b2v[i] = (i < rptB) ? w.b2[vB0 + fw * rptB + i] : 0.f;
        unsigned long long keys[D2_MAXS];
        const unsigned nk = nkeys++;
        const uint32_t ktag = (nk >> 1) & 1u;
        // two look-ahead frames: both scatters go out before either wait (the two jobs use the two tile buffers)
        unsigned jb[D2_MAXS];
#pragma unroll
        for (int zs = 0; zs < D2_MAXS; ++zs)
          if (zs < NS && zs < 2) jb[zs] = send_job(64, RB, rpB);
        // first pass, on the dependent chain: the logits of my rows and their (max, arg max) -> key
        float lv[D2_MAXS][4];
#pragma unroll
        for (int zs = 0; zs < D2_MAXS; ++zs) {
          keys[zs] = (unsigned long long)ktag;
#pragma unroll
          for (int i = 0; i < 4; ++i) lv[zs][i] = -INFINITY;
          if (zs < NS) {
            if (zs >= 2) jb[zs] = send_job(64, RB, rpB);   // a third frame reuses the first frame's buffer: only after its release
            const float* pr = wait_job(jb[zs]);
#pragma unroll
            for (int sr = 0; sr < D2_CL; ++sr) {
              const float* ps = pr + (size_t)sr * D2_NB * D2_RP + fw * rptB;
#pragma unroll
              for (int i = 0; i < 4; ++i)
                if (i < rptB) lv[zs][i] = (sr == 0 ? b2v[i] : lv[zs][i]) + ps[i];
            }
            release_job(jb[zs]);
            const bool vz = bvalid && c.active[fb] != 0 && c.t[fb] + zs < c.len[fb];
            const int e = c.n_eval[fb] + zs;     // index of this evaluation in the utterance's sequence
            float m = -INFINITY;
            int am = 0;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (i < rptB && lv[zs][i] > m) { m = lv[zs][i]; am = vB0 + fw * rptB + i; }
            // the 4 lanes of a batch row hold ascending vocabulary slices: strict > keeps the first maximum (torch.max)
#pragma unroll
            for (int o = 1; o < 4; o <<= 1) {
              const float m2 = __shfl_down_sync(0xffffffffu, m, o);
              const int am2 = __shfl_down_sync(0xffffffffu, am, o);
              if ((fw & (2 * o - 1)) == 0 && m2 > m) { m = m2; am = am2; }
            }
            if (vz && e < p.max_steps) {
              unsigned u = __float_as_uint(m);
              u ^= (u & 0x80000000u) ? 0xFFFFFFFFu : 0x80000000u;
              keys[zs] = ((unsigned long long)u << 32) | (unsigned long long)(((0x7FFFFFFFu - (unsigned)am) << 1) | ktag);
            }
          }
        }
        // second pass, off the chain: softmax partials (max, sum exp) of my vocabulary rows for the log-probability
        // post-pass, optional logit trace
        auto second_pass = [&]() {
#pragma unroll
        for (int zs = 0; zs < D2_MAXS; ++zs) {
          if (zs < NS) {
            const bool vz = bvalid && c.active[fb] != 0 && c.t[fb] + zs < c.len[fb];
            const int e = c.n_eval[fb] + zs;
            float m = -INFINITY, sx = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (i < rptB && lv[zs][i] > m) m = lv[zs][i];
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (i < rptB) sx += expf(lv[zs][i] - m);
            if (p.trace && vz && e < p.trace_cap) {
              float* tr = p.trace + ((size_t)fb * p.trace_cap + e) * V + vB0 + fw * rptB;
#pragma unroll
              for (int i = 0; i < 4; ++i)
                if (i < rptB) tr[i] = lv[zs][i];
            }
#pragma unroll
            for (int o = 1; o < 4; o <<= 1) {
              const float m2 = __shfl_down_sync(0xffffffffu, m, o), s2 = __shfl_down_sync(0xffffffffu, sx, o);
              if ((fw & (2 * o - 1)) == 0) {
                if (m2 > m) { sx = sx * expf(m - m2) + s2; m = m2; }
                else sx += s2 * expf(m2 - m);
              }
            }
            if (vz && e < p.max_steps && fw == 0)
              *reinterpret_cast<float2*>(p.part + (((size_t)e * D2_G + cta) * D2_NB + fb) * 2) = make_float2(m, sx);
          }
        }
        };
        // Arg-max exchange in two hops: every CTA hands its keys to the cluster leader through DSMEM (st.async, 117 ns), the
        // leader folds the four and publishes ONE tagged entry per (frame, utterance pair); every CTA then reads the 32-cluster
        // table of all look-ahead frames in a single pass (8 chunks per thread at two frames).
        unsigned long long* ktab = p.keys + (size_t)(nk & 1u) * NS * D2_NCL * D2_NB;
        if (rank == 0 && lane == 0) mbar_arrive_expect_tx(kbar, (uint32_t)(D2_NB * NS * 8));   // a quarter of 4 CTAs x 32 x NS keys
        {
          const uint32_t kb_remote = mapa(smem_u32(&c.kbuf[rank][0][fb]), 0u), kbar_remote = mapa(smem_u32(kbar), 0u);
#pragma unroll
          for (int zs = 0; zs < D2_MAXS; ++zs)
            if (zs < NS && fw == 0) st_async_b64(kb_remote + (uint32_t)(zs * D2_NB * 8), keys[zs], kbar_remote);
        }
        if (rank == 0) {
          mbar_wait(kbar, nk & 1u);
          const int kb_b = et & 31, kb_z = et >> 5;
          unsigned long long kk = (unsigned long long)ktag;
          if (kb_z < NS) {
#pragma unroll
            for (int sr = 0; sr < D2_CL; ++sr) kk = c.kbuf[sr][kb_z][kb_b] > kk ? c.kbuf[sr][kb_z][kb_b] : kk;
          }
          const unsigned long long kk2 = __shfl_down_sync(0xffffffffu, kk, 1);
          if (kb_z < NS && (kb_b & 1) == 0)
            st_relaxed_v4(ktab + ((size_t)kb_z * D2_NCL + cl) * D2_NB + kb_b, (uint32_t)kk, (uint32_t)(kk >> 32), (uint32_t)kk2, (uint32_t)(kk2 >> 32));
        }
        stamp(1);
        // thread -> batch pair et % 16, clusters {et / 16 + 8 i}; all frames requested before the first is validated
        {
          const int bp = et & 15, g = et >> 4;
          const unsigned long long* src = ktab + (size_t)g * D2_NB + 2 * bp;
          uint4 r[D2_MAXS][4];
#pragma unroll
          for (int zs = 0; zs < D2_MAXS; ++zs)
            if (zs < NS) {
#pragma unroll
              for (int i = 0; i < 4; ++i) r[zs][i] = ld_relaxed_v4(src + ((size_t)zs * D2_NCL + 8 * i) * D2_NB);
            }
          second_pass();   // while the table loads are in flight
          for (;;) {
            uint32_t bad = 0;
#pragma unroll
            for (int zs = 0; zs < D2_MAXS; ++zs)
              if (zs < NS) {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                  if ((r[zs][i].x & 1u) != ktag || (r[zs][i].z & 1u) != ktag) bad |= 1u << (zs * 4 + i);
              }
            if (!__any_sync(0xffffffffu, bad != 0u)) break;
#pragma unroll
            for (int zs = 0; zs < D2_MAXS; ++zs)
              if (zs < NS) {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                  if ((bad >> (zs * 4 + i)) & 1u) r[zs][i] = ld_relaxed_v4(src + ((size_t)zs * D2_NCL + 8 * i) * D2_NB);
              }
          }
#pragma unroll
          for (int zs = 0; zs < D2_MAXS; ++zs)
            if (zs < NS) {
              unsigned long long k0 = 0ull, k1 = 0ull;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const unsigned long long a = ((unsigned long long)r[zs][i].y << 32) | r[zs][i].x, b = ((unsigned long long)r[zs][i].w << 32) | r[zs][i].z;
                k0 = a > k0 ? a : k0;
                k1 = b > k1 ? b : k1;
              }
              c.kred[zs][g][2 * bp] = k0;
              c.kred[zs][g][2 * bp + 1] = k1;
            }
        }
        named_bar_sync(1, 128);
        stamp(2);
      }
      // ---------------- R: greedy rule (models.py:408-437), identical in every CTA ----------------
      // consumes the look-ahead evaluations in order: a blank moves on to the next frame (whose evaluation is already there),
      // the first non-blank ends the step for the utterance (its predictor state changes)
      int tok_pre = -1;
      {
        // every thread replays the rule for ITS utterance on the reduced keys (read-only) to learn the token it will emit, and
        // requests that token's table row now: the L2 round trip overlaps warp 0's rule and the barrier behind it
        if (bvalid && c.active[fb] != 0) {
          int tl = c.t[fb];
          const int ln = c.len[fb];
#pragma unroll
          for (int zs = 0; zs < D2_MAXS; ++zs) {
            if (zs < NS && tok_pre < 0 && tl < ln) {
              unsigned long long key = 0ull;
#pragma unroll
              for (int g = 0; g < 8; ++g) key = c.kred[zs][g][fb] > key ? c.kred[zs][g][fb] : key;
              const int am2 = (int)(0x7FFFFFFFu - (unsigned)((key & 0xFFFFFFFFull) >> 1));
              if (am2 == w.blank) ++tl; else tok_pre = am2;
            }
          }
        }
        if (tok_pre >= 0) load_table0(tok_pre, vpre);
        if (et < B) {
          const int bb = et;
          unsigned char emit = 0;
          for (int zs = 0; zs < NS && c.active[bb] && !emit; ++zs) {
            unsigned long long key = 0ull;
#pragma unroll
            for (int g = 0; g < 8; ++g) key = c.kred[zs][g][bb] > key ? c.kred[zs][g][bb] : key;
            const int am2 = (int)(0x7FFFFFFFu - (unsigned)((key & 0xFFFFFFFFull) >> 1));
            const int t = c.t[bb];
            c.n_eval[bb] += 1;
            const int it = c.it[bb] + 1;
            bool advance;
            if (am2 == w.blank) {
              advance = true;
            } else {
              const int n = c.ntok[bb];
              if (cta == 0 && n < p.U_cap) p.tokens[(size_t)bb * p.U_cap + n] = am2;
              c.ntok[bb] = n + 1;
              c.tok[bb] = am2;
              emit = 1;
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
        if (warp == 0) {   // B <= 32: the whole control state lives in warp 0's lanes
          const unsigned ae = __ballot_sync(0xffffffffu, et < B && c.emit[et] != 0);
          const unsigned aa = __ballot_sync(0xffffffffu, et < B && c.active[et] != 0);
          if (lane == 0) {
            // The six GEMM-side warps have read the previous flags.  ONLY this thread waits on ctlack: it is also the one whose
            // ctlbar arrive lets the next ctlack phase begin, so it cannot be lapped.  (All 128 epilogue threads used to wait here;
            // a warp that reached the wait late -- after this thread had already published the step and the six acks had come in --
            // saw the parity of the NEXT completed phase and spun forever: a hang about once in 100 full-size calls once other
            // work was placed in front of the wait.  Phase-lapping rule, DESIGN.md section 4.)
            if (step > 0) mbar_wait(ctlack, (step - 1) & 1);
            c.flags[0] = ae != 0u; c.flags[1] = aa != 0u;
            mbar_arrive(ctlbar);
          }
          __syncwarp();
        }
        named_bar_sync(1, 128);
      }
      const bool any_emit = c.flags[0] != 0, any_active = c.flags[1] != 0;
      stamp(3);
      if (any_emit) {
        phase_c0(tok_pre);
        stamp(4);
        phase_c1();
        stamp(5);
        pending = true;
      }
      any_upd = any_emit;
      if (!any_active) break;
    }
    // ---- results and state ----
    if (cta == 0 && et < B) {
      p.ntok[et] = c.ntok[et];
      p.n_eval[et] = c.n_eval[et];
    }
    if (bvalid) {
      if (p.state_h)
#pragma unroll
        for (int l = 0; l < 2; ++l)
          *reinterpret_cast<float2*>(p.state_h + ((size_t)l * p.state_ld + fb) * H + unit) = make_float2(hst[l][0], hst[l][1]);
      if (p.pred_out) *reinterpret_cast<float2*>(p.pred_out + (size_t)fb * H + unit) = make_float2(gval[0], gval[1]);
    }
  } else if (warp < 8) {
    // ======================================= loaders =======================================
    const int lt = (warp - 4) * 32 + lane;
    unsigned nw[IMG_N];                     // writes that precede the point reached in the job sequence
#pragma unroll
    for (int i = 0; i < IMG_N; ++i) nw[i] = (i == IMG_G || i == IMG_H0 || i == IMG_H1) ? 1u : 0u;
    const int NS = p.n_spec;
    unsigned ga = 0;                        // k-block stages filled so far
    if (lane == 0) {
      while (ld_acquire_u32(p.barrier) < (unsigned)D2_G) {
      }
    }
    __syncwarp();
    // K slice of the latest write of image `img` -> 4 ring stages
    auto fetch = [&](int img) {
      const unsigned n = nw[img] - 1;
      const uint32_t tag = (n >> 1) & 1u;
      const uint8_t* src = img_ptr(img, n) + slice_off + (size_t)lt * 16;
      uint4 r[16];
      poll_issue<16>(src, 16, tag, r, D2_TRIG);
#pragma unroll
      for (int kb = 0; kb < D2_KS; ++kb, ++ga) {
        poll_validate_kb<16>(src, kb, tag, r);
        const int s = (int)(ga % D2_AST);
        mbar_wait(&aempty[s], ((ga / D2_AST) & 1u) ^ 1u);
        uint8_t* dst = aring + (size_t)s * 8192 + (size_t)lt * 16;
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          chunk_strip_tag(r[kb * 4 + jj]);
          *reinterpret_cast<uint4*>(dst + (size_t)jj * 2048) = r[kb * 4 + jj];
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&afull[s]);
      }
    };
    if (!p.use_state_in) {
      fetch(IMG_H0);
      fetch(IMG_H1);
      nw[IMG_H0]++; nw[IMG_X]++;
      fetch(IMG_X);
      nw[IMG_H1]++; nw[IMG_G]++;
    }
    bool pending = true, any_upd = true;
    for (int step = 0;; ++step) {
      if (pending) fetch(IMG_H0);
      if (any_upd) fetch(IMG_G);
#pragma unroll
      for (int zs = 0; zs < D2_MAXS; ++zs)
        if (zs < NS) nw[IMG_Z0 + zs]++;
      if (pending) { fetch(IMG_H1); pending = false; }
#pragma unroll
      for (int zs = 0; zs < D2_MAXS; ++zs)
        if (zs < NS) fetch(IMG_Z0 + zs);
      mbar_wait(ctlbar, step & 1);
      const bool any_emit = c.flags[0] != 0, any_active = c.flags[1] != 0;
      __syncwarp();
      if (lane == 0) mbar_arrive(ctlack);
      if (any_emit) {
        nw[IMG_H0]++; nw[IMG_X]++;
        fetch(IMG_X);
        nw[IMG_H1]++; nw[IMG_G]++;
        pending = true;
      }
      any_upd = any_emit;
      if (!any_active) break;
    }
  } else if (warp == 8) {
    // ======================================= MMA issuer =======================================
    if (elect_one()) {
      mbar_arrive_expect_tx(w2full, (uint32_t)D2_KS * w2kb);
      tma_bulk_g2s(W2s, p.w2_img + img_tile_offset(cl, rank * D2_KS, 0, D2_K / 64, RB), (uint32_t)D2_KS * w2kb, w2full);
    }
    __syncwarp();
    const uint64_t a_ring0 = umma_desc_sw128(smem_u32(aring));
    const uint64_t w_ring0 = umma_desc_sw128(smem_u32(wring));
    const uint64_t w2_0 = umma_desc_sw128(smem_u32(W2s));
    unsigned job = 0, ga = 0, gw = 0;
    // one GEMM job: weights either resident (W2) or from the ring; hi part of a k-block = `rows` x 128 B
    auto run_job = [&](int M, int rows, bool resident) {
      const unsigned j = job++;
      const int ab = (int)(j & 1u);
      mbar_wait(&tempty[ab], ((j >> 1) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t idesc1 = umma_idesc_f16(M, 64), idesc2 = umma_idesc_f16(M, 32);
      const uint32_t dcol = tmem + (uint32_t)(ab * 128);
      const uint32_t lo_u = ((uint32_t)rows * 128u) >> 4;
      for (int kb = 0; kb < D2_KS; ++kb, ++ga) {
        const int sa = (int)(ga % D2_AST);
        uint64_t wd;
        int sw = 0;
        if (resident) {
          wd = w2_0 + (uint64_t)((uint32_t)kb * (w2kb >> 4));
        } else {
          sw = (int)(gw % D2_WST);
          mbar_wait(&wfull[sw], (gw / D2_WST) & 1u);
          wd = w_ring0 + (uint64_t)((uint32_t)sw * (D2_WSTAGE >> 4));
        }
        mbar_wait(&afull[sa], (ga / D2_AST) & 1u);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t bd = a_ring0 + (uint64_t)((uint32_t)sa * (8192 >> 4));
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4) {
            const uint32_t accumulate = (kb | k4) ? 1u : 0u;
            tc_mma_f16(dcol, wd + 2 * k4, bd + 2 * k4, idesc1, accumulate);
            tc_mma_f16(dcol + 64, wd + lo_u + 2 * k4, bd + 2 * k4, idesc2, accumulate);
          }
          tc_commit(&aempty[sa]);
          if (!resident) tc_commit(&wempty[sw]);
          if (kb == D2_KS - 1) tc_commit(&tfull[ab]);
        }
        __syncwarp();
        if (!resident) ++gw;
      }
    };
    mbar_wait(w2full, 0);
    if (!p.use_state_in) {
      run_job(128, 96, false);   // R0 h0
      run_job(128, 96, false);   // R1 h1
      run_job(128, 96, false);   // K1 BN(h0')
    }
    bool pending = true, any_upd = true;
    for (int step = 0;; ++step) {
      if (pending) run_job(128, 96, false);
      if (any_upd) run_job(64, 32, false);
      if (pending) { run_job(128, 96, false); pending = false; }
      for (int zs = 0; zs < p.n_spec; ++zs) run_job(64, RB, true);
      mbar_wait(ctlbar, step & 1);
      const bool any_emit = c.flags[0] != 0, any_active = c.flags[1] != 0;
      __syncwarp();
      if (lane == 0) mbar_arrive(ctlack);
      if (any_emit) {
        run_job(128, 96, false);
        pending = true;
      }
      any_upd = any_emit;
      if (!any_active) break;
    }
  } else {
    // ======================================= weight streamer =======================================
    // The streamed matrices are consumed in a fixed cyclic order whatever the emission pattern is -- (BOS run: R0, R1, K1,)
    // then R0, W1p, R1, K1, R0, W1p, ... -- so the streamer never waits for the flags of a step to know WHAT comes next:
    // it keeps the 3-stage ring full (K1's first 72 KB are resident before the rule that needs them has even run) and
    // only watches the control barrier to learn when the loop ends.
    unsigned gw = 0;
    int seq = p.use_state_in ? 3 : 0;   // position in  R0 R1 K1 | R0 W1p R1 K1 | R0 W1p R1 K1 ...
    int kb = 0, step = 0;
    bool done = false, finishing = false;   // finishing: the loop has ended with an emission, the last K1 still has to be delivered
    int k1_needed = p.use_state_in ? 0 : 1, k1_issued = 0;   // K1 matrices the MMA warp will consume in total / fully streamed so far
    while (!done) {
      const int s = (int)(gw % D2_WST);
      if (mbar_try_wait(&wempty[s], ((gw / D2_WST) & 1u) ^ 1u)) {
        const int m = seq < 3 ? seq : (seq - 3) % 4;                 // which matrix
        const uint8_t* wimg;
        int TR;
        if (seq < 3) { wimg = m == 0 ? p.r_img[0] : (m == 1 ? p.r_img[1] : p.k1_img); TR = 96; }
        else if (m == 0) { wimg = p.r_img[0]; TR = 96; }
        else if (m == 1) { wimg = p.w1p_img; TR = 32; }
        else if (m == 2) { wimg = p.r_img[1]; TR = 96; }
        else { wimg = p.k1_img; TR = 96; }
        const uint32_t kbb = (uint32_t)TR * 256u;
        if (elect_one()) {
          mbar_arrive_expect_tx(&wfull[s], kbb);
          tma_bulk_g2s(wring + (size_t)s * D2_WSTAGE, wimg + img_tile_offset(cl, rank * D2_KS + kb, 0, D2_K / 64, TR), kbb, &wfull[s]);
        }
        __syncwarp();
        ++gw;
        if (++kb == D2_KS) {
          kb = 0;
          const bool was_k1 = seq == 2 || seq == 6;
          ++seq;
          if (seq >= 7) seq = 3;
          if (was_k1) ++k1_issued;
          if (finishing && k1_issued >= k1_needed) done = true;
        }
      } else if (!finishing && mbar_try_wait(ctlbar, step & 1)) {
        const bool any_emit = c.flags[0] != 0, any_active = c.flags[1] != 0;
        __syncwarp();
        if (lane == 0) mbar_arrive(ctlack);
        ++step;
        if (any_emit) ++k1_needed;
        if (!any_active) {
          // the other roles still run the predictor of a final emission (JK1): its K1 must be delivered in full
          if (k1_issued >= k1_needed) done = true;
          else finishing = true;
        }
      }
    }
    // every copy that was issued has to land before the CTA may go (stages fetched ahead of a loop that ended)
    for (unsigned g = gw > D2_WST ? gw - D2_WST : 0; g < gw; ++g) mbar_wait(&wfull[g % D2_WST], (g / D2_WST) & 1u);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 8) tmem_dealloc(tmem, 256);
}

int g_dec2_max_clusters = -1;

}  // namespace

// defined in decode_tc.cu: post-pass that folds the per-step softmax partials into log-probabilities
cudaError_t launch_decode_finish(const float* part, const int* n_eval, int B, int nB, int Bq, int max_steps, double* neg_logp, float* trace,
                                 float* trace_lse, int trace_cap, int V, cudaStream_t st);

static size_t decode_tc2_smem() {
  return 65536 + (size_t)D2_WST * D2_WSTAGE + 4096 + (size_t)D2_AST * 8192 + (size_t)2 * D2_CL * D2_NB * D2_RP * 4 + ((sizeof(Ctrl2) + 15) & ~15) + 512 + 1024;
}

cudaError_t configure_decode_tc2() {
  return cudaFuncSetAttribute(decode_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

bool decode_tc2_plan(int H, int J, int V, int Lp, int B, int sms, int lm_layers) {
  if (lm_layers > 0 || Lp != 2 || H != D2_K || J != D2_K || V % 512 || V < 512 || V > 2048 || B < 1 || B > D2_NB || sms < D2_G) return false;
  if (decode_tc2_smem() > 227 * 1024) return false;
  if (g_dec2_max_clusters < 0) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(D2_G);
    cfg.blockDim = dim3(D2_THREADS);
    cfg.dynamicSmemBytes = decode_tc2_smem();
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = D2_CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, decode_tc2_kernel, &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
    g_dec2_max_clusters = n;
  }
  return g_dec2_max_clusters >= D2_NCL;
}

size_t decode_tc2_image_bytes() { return (size_t)(D2_K / 64) * 8192; }        // one buffer of one activation image
size_t decode_tc2_keys_bytes() { return (size_t)2 * D2_MAXS * D2_NCL * D2_NB * 8; }
int decode_tc2_images() { return IMG_N; }
int decode_tc2_part_ctas() { return D2_G; }

cudaError_t launch_decode_tc2(const DecodeTc2Args& a, cudaStream_t st) {
  DecodeTc2Args args = a;
  args.n_spec = D2_SPEC;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(D2_G);
  cfg.blockDim = dim3(D2_THREADS);
  cfg.dynamicSmemBytes = decode_tc2_smem();
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = D2_CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeCooperative;
  at[1].val.cooperative = 1;
  cfg.attrs = at;
  // cooperative unless switched off (kernels.h: coop_launch_enabled; the plan has verified with
  // cudaOccupancyMaxActiveClusters that all clusters fit)
  cfg.numAttrs = coop_launch_enabled() ? 2 : 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, decode_tc2_kernel, args);
  if (e != cudaSuccess) return e;
  return launch_decode_finish(a.part, a.n_eval, a.B, D2_G, D2_NB, a.max_steps, a.neg_logp, a.trace, a.trace_lse, a.trace_cap, a.w.V, st);
}

}  // namespace rnnt
