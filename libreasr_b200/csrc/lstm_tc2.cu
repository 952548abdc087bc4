// Persistent tcgen05 LSTM layer, 2-D (gate rows x K) partition with a cluster-local split-K
// reduction over distributed shared memory.  Same contract as lstm_tc.cu (reference
// libreasr/lib/layers/custom_rnn.py:140-175 driving torch.nn.LSTM, arithmetic haste/lstm.py:51-60,
// gate order i,f,g,o, + BatchNorm1d eval custom_rnn.py:210-213), different decomposition:
//
//   * A cluster of 4 CTAs owns 32 hidden units = 128 interleaved gate rows (unit*4 + gate) of W_hh.
//     CTA `rank` of the cluster keeps the K-slice [rank*H/4, (rank+1)*H/4) of those rows RESIDENT in
//     shared memory (hi + lo fp16 operand image, 128 KB at H = 1024) for the whole layer.
//   * The gate rows sit on the MMA M axis (M = 128: full tensor rate, lane = gate row), the batch on N:
//         D1[128 x 64] += W_hi[128 x 16] * [h_hi ; h_lo][64 x 16]^T      (hi*hi | hi*lo)
//         D2[128 x 32] += W_lo[128 x 16] *  h_hi       [32 x 16]^T       (lo*hi)
//     so a step costs H/4/16 * 2 tcgen05.mma per CTA instead of H/16, and a CTA ingests only ITS K-slice of
//     h_{t-1}: 32 KB instead of 128 KB per step (the grid-wide all-gather of lstm_tc.cu shrinks 4x).
//   * Split-K reduction: epilogue warp q (TMEM lanes 32q..32q+31 = the gate rows of the 8 units CTA q
//     finalises) folds the three split products and writes its 32 x 32 fp32 partial tile straight into CTA q's
//     shared memory with st.async, whose bytes complete a transaction count on CTA q's mbarrier (no fence on
//     either side).  Every CTA sums the 4 partial tiles of its 8 units, adds the hoisted input projection,
//     applies the cell with c (and h) in registers, and publishes h_t.
//   * h exchange without a flag round trip: h_t is published as 16-byte chunks (8 consecutive units of one
//     batch row, hi or lo halves, already in the swizzled operand-image order) whose last half carries a
//     1-bit sequence tag in its LSB (the hi half is tagged BEFORE lo is derived from it, so the pair still
//     represents the value).  Consumers poll the DATA (ld.relaxed.gpu v4, one chunk = one aligned 16-byte
//     store) and copy validated chunks into the UMMA tile: publish -> consume is one store + one load
//     latency; no release fence, no counter, no TMA issue on the dependent chain.
//
//   warps 0-3  epilogue: TMEM -> fold -> DSMEM scatter; then finalise 8 units x 32 rows; publish h_t; y outputs
//   warps 4-7  loaders: poll/validate the K-slice of h_{t-1} (32 KB), store to smem, fence.proxy.async, arrive
//   warp  8    MMA issuer (one elected lane), accumulators double-buffered in TMEM
#include <cstdlib>

#include "kernels.h"
#include "tc_common.cuh"
#include "tc2_common.cuh"

namespace rnnt {
namespace {

constexpr int L2_THREADS = 288;
constexpr int L2_CL = 4;          // CTAs per cluster = K slices
constexpr int L2_UPC = 8;         // units finalised per CTA
constexpr int L2_NB = 32;         // batch rows per launch (N tile: 32 hi + 32 lo)
constexpr int L2_MAX_KS = 4;      // k-blocks (64 k) per K slice
// Producers (of 8) of the polled line whose chunk must carry the new tag before a loader warp issues the loads of its
// K slice (measured on a B200: 5 and 6 change nothing against 3).
constexpr int L2_TRIG = 3;

__global__ void __launch_bounds__(L2_THREADS, 1) lstm_layer_tc2_kernel(LstmTc2Args p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024 - (smem_u32(smem_raw) & 1023)) & 1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const int cl = blockIdx.x / L2_CL;          // cluster index = 32-unit group
  const int KS = p.KS, H = p.H, T = p.T;
  // shared memory: W slice [KS][hi 16 KB | lo 16 KB] | h slice [KS][hi 4 KB | lo 4 KB] | partial tiles [2][4][32 b][32 rows] f32 | barriers
  uint8_t* Wsm = base;
  uint8_t* hs = Wsm + (size_t)KS * 32768;
  float* P = reinterpret_cast<float*>(hs + (size_t)KS * 8192);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(P) + 32768);
  uint64_t* hfull = bars;                     // [KS] loaders -> MMA
  uint64_t* hempty = hfull + L2_MAX_KS;       // [KS] MMA -> loaders
  uint64_t* tfull = hempty + L2_MAX_KS;       // [2] accumulators ready
  uint64_t* tempty = tfull + 2;               // [2] accumulators drained
  uint64_t* pbar = tempty + 2;                // [2] partial tiles of a step complete (4 remote warp arrivals)
  uint64_t* wfull = pbar + 2;
  uint32_t* tptr = reinterpret_cast<uint32_t*>(wfull + 1);

  if (threadIdx.x == 0) {
    for (int i = 0; i < L2_MAX_KS; ++i) {
      mbar_init(&hfull[i], 4);   // one arrive per loader warp
      mbar_init(&hempty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 128);
      mbar_init(&pbar[i], 4);   // one arming arrive per epilogue warp
    }
    mbar_init(wfull, 1);
    fence_mbar_init();
  }
  if (warp == 8) tmem_alloc(tptr, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  cluster_sync_all();   // peers' barriers are initialised before anyone arrives on them remotely
  const uint32_t tmem = *tptr;
  const size_t slice_off = (size_t)rank * KS * 8192;   // this CTA's K-slice inside an h image

  if (warp < 4) {
    // =========================== epilogue / finalise ===========================
    const int q = warp;                                  // TMEM lane quarter = destination CTA of this warp's rows
    const uint32_t tl = tmem + ((uint32_t)(q * 32) << 16);
    const int et = warp * 32 + lane;
    const int fb = warp * 8 + (lane >> 2);               // batch row finalised by this thread
    const int fw = lane & 3;                             // unit pair
    const int ucta = cl * 32 + rank * L2_UPC;            // first unit finalised by this CTA
    const int unit = ucta + 2 * fw;
    const bool valid = fb < p.B;
    const int len = valid ? (p.lens_T ? min(p.lens_T[fb], T) : T) : 0;
    float h[2], c[2], bsc[2], bsh[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      h[j] = (valid && p.state_h_in) ? p.state_h_in[(size_t)fb * H + unit + j] : p.h_init_vec[unit + j];
      c[j] = (valid && p.state_c_in) ? p.state_c_in[(size_t)fb * H + unit + j] : p.c_init_vec[unit + j];
      bsc[j] = p.bn_scale[unit + j];
      bsh[j] = p.bn_shift[unit + j];
    }
    // chunk (fb, units ucta..ucta+7) inside an h image: [kb][part][32 rows x 128 B, 16-byte chunks swizzled by row]
    const uint32_t off_hi = (uint32_t)((ucta >> 6) * 2) * 4096u + (uint32_t)fb * 128u + (uint32_t)((((ucta & 63) >> 3) ^ (fb & 7)) << 4);
    auto publish = [&](uint8_t* img, float v0, float v1, uint32_t tag) {
      uint32_t h0, l0, h1, l1;
      split_tag(v0, false, 0u, h0, l0);
      split_tag(v1, fw == 3, tag, h1, l1);
      const uint32_t hp = h0 | (h1 << 16), lp = l0 | (l1 << 16);
      const int g0 = lane & ~3;
      const uint32_t a0 = __shfl_sync(0xffffffffu, hp, g0), a1 = __shfl_sync(0xffffffffu, hp, g0 + 1);
      const uint32_t a2 = __shfl_sync(0xffffffffu, hp, g0 + 2), a3 = __shfl_sync(0xffffffffu, hp, g0 + 3);
      const uint32_t b0 = __shfl_sync(0xffffffffu, lp, g0), b1 = __shfl_sync(0xffffffffu, lp, g0 + 1);
      const uint32_t b2 = __shfl_sync(0xffffffffu, lp, g0 + 2), b3 = __shfl_sync(0xffffffffu, lp, g0 + 3);
      if (fw == 0) st_relaxed_v4(img + off_hi, a0, a1, a2, a3);
      else if (fw == 1) st_relaxed_v4(img + off_hi + 4096u, b0, b1, b2, b3);
    };
    // h_{-1} -> image 0 (tag 0); image 1 gets the tag its first real write (after step 0, tag 0) will flip
    publish(p.x_img[0], h[0], h[1], 0u);
    publish(p.x_img[1], 0.f, 0.f, 1u);
    __threadfence();
    named_bar_sync(1, 128);
    if (et == 0) red_release_add(p.barrier, 1u);   // once per launch: stale chunks of an earlier launch cannot be mistaken for h_{-1}

    const uint32_t P_u32 = smem_u32(P);
    long long cyc[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // tuning aid (CTA 0, thread 0): cycles per epilogue segment, summed over the steps
    const bool prof = p.dbg != nullptr && blockIdx.x == 0 && et == 0;
    for (int t = 0; t < T; ++t) {
      long long c0 = prof ? clock64() : 0;
      const int ab = t & 1;
      const int64_t row = (int64_t)fb * T + t;
      const bool upd = valid && t < len;
      float4 xv0 = make_float4(0.f, 0.f, 0.f, 0.f), xv1 = xv0;
      if (upd) {   // hoisted input projection of my two units (interleaved gate columns): issued before the accumulators are awaited
        const float4* xr = reinterpret_cast<const float4*>(p.xp + row * (size_t)(4 * H) + (size_t)unit * 4);
        xv0 = xr[0];
        xv1 = xr[1];
      }
      // every epilogue warp arms a quarter of the step's bytes, so the phase cannot complete (and the barrier cannot run a
      // phase ahead of a lagging warp) before all four warps have entered the step
      if (lane == 0) mbar_arrive_expect_tx(&pbar[ab], (uint32_t)(L2_NB * 32 * 4));
      mbar_wait(&tfull[ab], (t >> 1) & 1);
      tc_fence_after();
      if (p.dbg && blockIdx.x == 0 && et == 0) p.dbg[t * 4 + 1] = gtimer();
      if (prof) { const long long c1 = clock64(); cyc[0] += c1 - c0; c0 = c1; }   // waiting for the accumulators
      {
        float d0[32], d1[32], d2[32];
        const uint32_t tc = tl + (uint32_t)(ab * 128);
        tmem_ld32(tc, d0);          // W_hi * h_hi
        tmem_ld32(tc + 32, d1);     // W_hi * h_lo  (x 2^11)
        tmem_ld32(tc + 64, d2);     // W_lo * h_hi  (x 2^11)
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&tempty[ab]);
        if (prof) { const long long c1 = clock64(); cyc[1] += c1 - c0; c0 = c1; }   // TMEM drain
        // my gate row's 32 batch values -> CTA q's partial tile [ab][src = rank][b][row = lane]
        // (the bytes are counted on the owner's mbarrier: no fence on either side)
        const uint32_t dst = mapa(P_u32 + (uint32_t)(((ab * L2_CL + rank) * L2_NB) * 128 + lane * 4), (uint32_t)q);
        const uint32_t rbar = mapa(smem_u32(&pbar[ab]), (uint32_t)q);
#pragma unroll
        for (int b = 0; b < 32; ++b) st_async_f32(dst + (uint32_t)b * 128u, fmaf(d1[b] + d2[b], kLoInv, d0[b]), rbar);
      }
      if (prof) { const long long c1 = clock64(); cyc[2] += c1 - c0; c0 = c1; }   // scatter issue
      mbar_wait(&pbar[ab], (t >> 1) & 1);
      if (p.dbg && blockIdx.x == 0 && et == 0) p.dbg[t * 4 + 2] = gtimer();
      if (p.dbg_all && et == 0) p.dbg_all[((size_t)blockIdx.x * T + t) * 2 + 1] = gtimer();
      if (prof) { const long long c1 = clock64(); cyc[3] += c1 - c0; c0 = c1; }   // waiting for the four partial tiles
      {
        float acc[8];
        const float* pr = P + (size_t)((ab * L2_CL) * L2_NB + fb) * 32 + fw * 8;
#pragma unroll
        for (int s = 0; s < L2_CL; ++s) {
          const float4 u0 = *reinterpret_cast<const float4*>(pr + (size_t)s * L2_NB * 32);
          const float4 u1 = *reinterpret_cast<const float4*>(pr + (size_t)s * L2_NB * 32 + 4);
          if (s == 0) {
            acc[0] = u0.x; acc[1] = u0.y; acc[2] = u0.z; acc[3] = u0.w; acc[4] = u1.x; acc[5] = u1.y; acc[6] = u1.z; acc[7] = u1.w;
          } else {
            acc[0] += u0.x; acc[1] += u0.y; acc[2] += u0.z; acc[3] += u0.w; acc[4] += u1.x; acc[5] += u1.y; acc[6] += u1.z; acc[7] += u1.w;
          }
        }
        if (prof) { const long long c1 = clock64(); cyc[4] += c1 - c0; c0 = c1; }   // tile sums (LDS)
        if (upd) {
          {
            const float vi = acc[0] + xv0.x, vf = acc[1] + xv0.y, vg = acc[2] + xv0.z, vo = acc[3] + xv0.w;
            const float cn = sigmoid_fast(vf) * c[0] + sigmoid_fast(vi) * tanh_fast(vg);
            c[0] = cn;
            h[0] = sigmoid_fast(vo) * tanh_fast(cn);
          }
          {
            const float vi = acc[4] + xv1.x, vf = acc[5] + xv1.y, vg = acc[6] + xv1.z, vo = acc[7] + xv1.w;
            const float cn = sigmoid_fast(vf) * c[1] + sigmoid_fast(vi) * tanh_fast(vg);
            c[1] = cn;
            h[1] = sigmoid_fast(vo) * tanh_fast(cn);
          }
        }
      }
      if (prof) { const long long c1 = clock64(); cyc[5] += c1 - c0; c0 = c1; }   // cell
      // h_t gates the next step: publish first; the BatchNorm(h_t) outputs follow off the critical path
      publish(p.x_img[(t + 1) & 1], h[0], h[1], (uint32_t)(((t + 1) >> 1) & 1));
      if (prof) { const long long c1 = clock64(); cyc[6] += c1 - c0; c0 = c1; }   // publish
      if (p.dbg && blockIdx.x == 0 && et == 0) p.dbg[t * 4 + 3] = gtimer();
      if (p.dbg_all && et == 0) p.dbg_all[((size_t)blockIdx.x * T + t) * 2] = gtimer();
      if (valid) {
        const float y0 = h[0] * bsc[0] + bsh[0], y1 = h[1] * bsc[1] + bsh[1];
        if (p.y) *reinterpret_cast<float2*>(p.y + row * H + unit) = make_float2(y0, y1);
        if (p.y_img) {
          uint32_t h0, l0, h1, l1;
          split_tag(y0, false, 0u, h0, l0);
          split_tag(y1, false, 0u, h1, l1);
          uint8_t* hi = p.y_img + img_tile_offset(row >> 7, unit >> 6, 0, p.KB, 128) + img_elem_offset((int)(row & 127), unit & 63);
          *reinterpret_cast<uint32_t*>(hi) = h0 | (h1 << 16);
          *reinterpret_cast<uint32_t*>(hi + 128 * 128) = l0 | (l1 << 16);
        }
      }
      if (prof) { const long long c1 = clock64(); cyc[7] += c1 - c0; }   // BatchNorm outputs
    }
    if (prof)
      for (int i = 0; i < 8; ++i) p.dbg[(size_t)T * 4 + i] = (unsigned long long)cyc[i];
    if (valid) {
      if (p.state_h_out) *reinterpret_cast<float2*>(p.state_h_out + (size_t)fb * H + unit) = make_float2(h[0], h[1]);
      if (p.state_c_out) *reinterpret_cast<float2*>(p.state_c_out + (size_t)fb * H + unit) = make_float2(c[0], c[1]);
    }
  } else if (warp < 8) {
    // =========================== loaders ===========================
    const int lt = (warp - 4) * 32 + lane;
    const int NL = KS * 4;   // 16-byte chunks per thread per step (KS * 8 KB / 128 threads)
    if (lane == 0) {
      while (ld_acquire_u32(p.barrier) < gridDim.x) {
      }
    }
    __syncwarp();
    long long lcyc[4] = {0, 0, 0, 0};
    const bool lprof = p.dbg != nullptr && blockIdx.x == 0 && lt == 0;
    for (int t = 0; t < T; ++t) {
      const uint32_t tag = (uint32_t)((t >> 1) & 1);
      const uint8_t* src = p.x_img[t & 1] + slice_off + (size_t)lt * 16;
      uint4 r[L2_MAX_KS * 4];
      long long lc0 = lprof ? clock64() : 0;
      poll_issue<L2_MAX_KS * 4>(src, NL, tag, r, L2_TRIG);
      if (lprof) { const long long c1 = clock64(); lcyc[0] += c1 - lc0; lc0 = c1; }   // until the first chunk of h_{t-1} shows up
#pragma unroll
      for (int kb = 0; kb < L2_MAX_KS; ++kb) {
        if (kb < KS) {
          poll_validate_kb<L2_MAX_KS * 4>(src, kb, tag, r);
          if (lprof) { const long long c1 = clock64(); lcyc[1 + (kb > 0)] += c1 - lc0; lc0 = c1; }   // k-block 0 complete | the others
          if (t > 0) mbar_wait(&hempty[kb], (t - 1) & 1);   // the MMAs of step t-1 have finished reading this k-block
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int i = kb * 4 + j;
            chunk_strip_tag(r[i]);
            *reinterpret_cast<uint4*>(hs + (size_t)i * 2048 + (size_t)lt * 16) = r[i];
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(&hfull[kb]);
          if (lprof) { const long long c1 = clock64(); lcyc[3] += c1 - lc0; lc0 = c1; }   // stores + fence + arrive
        }
      }
      if (p.dbg && blockIdx.x == 0 && lt == 0) p.dbg[t * 4 + 0] = gtimer();
    }
    if (lprof)
      for (int i = 0; i < 4; ++i) p.dbg[(size_t)T * 4 + 8 + i] = (unsigned long long)lcyc[i];
  } else {
    // =========================== MMA issuer ===========================
    if (elect_one()) {
      mbar_arrive_expect_tx(wfull, (uint32_t)KS * 32768u);
      tma_bulk_g2s(Wsm, p.w_img + img_tile_offset(cl, rank * KS, 0, p.KB, 128), (uint32_t)KS * 32768u, wfull);
    }
    __syncwarp();
    const uint32_t idesc1 = umma_idesc_f16(128, 64), idesc2 = umma_idesc_f16(128, 32);
    const uint64_t a_desc0 = umma_desc_sw128(smem_u32(Wsm));
    const uint64_t b_desc0 = umma_desc_sw128(smem_u32(hs));
    mbar_wait(wfull, 0);
    for (int t = 0; t < T; ++t) {
      const int ab = t & 1;
      if (t >= 2) mbar_wait(&tempty[ab], ((t >> 1) + 1) & 1);
      tc_fence_after();
      const uint32_t dcol = tmem + (uint32_t)(ab * 128);
      for (int kb = 0; kb < KS; ++kb) {
        mbar_wait(&hfull[kb], t & 1);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t ah = a_desc0 + (uint64_t)(kb * (32768 >> 4)), al = ah + (uint64_t)(16384 >> 4);
          const uint64_t bd = b_desc0 + (uint64_t)(kb * (8192 >> 4));
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4) {
            const uint32_t accumulate = (kb | k4) ? 1u : 0u;
            tc_mma_f16(dcol, ah + 2 * k4, bd + 2 * k4, idesc1, accumulate);
            tc_mma_f16(dcol + 64, al + 2 * k4, bd + 2 * k4, idesc2, accumulate);
          }
          tc_commit(&hempty[kb]);
          if (kb == KS - 1) tc_commit(&tfull[ab]);
        }
        __syncwarp();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // no CTA leaves while a peer may still address its shared memory
  if (warp == 8) tmem_dealloc(tmem, 256);
}

int g_lstm_tc2_max_clusters = -1;

}  // namespace

cudaError_t configure_lstm_tc2() {
  return cudaFuncSetAttribute(lstm_layer_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

static size_t lstm_tc2_smem(int KS) { return (size_t)KS * (32768 + 8192) + 32768 + 1024 + 1024; }

// Cluster split-K plan: H/32 clusters of 4 CTAs, K slice of H/4 per CTA; B <= 32 rows per launch.
bool lstm_tc2_plan(int H, int B, int sms, LstmTc2Plan* pl) {
  if (B < 1 || B > L2_NB || H % 256 || H > 256 * L2_MAX_KS) return false;
  pl->KS = H / 256;
  pl->KB = H / 64;
  pl->grid = H / 8;
  pl->smem_bytes = (int)lstm_tc2_smem(pl->KS);
  if (pl->grid > sms || pl->smem_bytes > 227 * 1024) return false;
  if (g_lstm_tc2_max_clusters < 0) {   // all clusters must be co-resident (the kernel synchronises across the grid)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(pl->grid);
    cfg.blockDim = dim3(L2_THREADS);
    cfg.dynamicSmemBytes = (size_t)227 * 1024 - 2048;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = L2_CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, lstm_layer_tc2_kernel, &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
    g_lstm_tc2_max_clusters = n;
  }
  return g_lstm_tc2_max_clusters >= pl->grid / L2_CL;
}

cudaError_t launch_lstm_layer_tc2(const LstmTc2Args& a, const LstmTc2Plan& pl, cudaStream_t st) {
  LstmTc2Args args = a;
  args.KS = pl.KS;
  args.KB = pl.KB;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(pl.grid);
  cfg.blockDim = dim3(L2_THREADS);
  cfg.dynamicSmemBytes = (size_t)pl.smem_bytes;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = L2_CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeCooperative;
  at[1].val.cooperative = 1;
  cfg.attrs = at;
  // cooperative unless switched off (kernels.h: coop_launch_enabled; the plan has verified with
  // cudaOccupancyMaxActiveClusters that all clusters fit)
  cfg.numAttrs = coop_launch_enabled() ? 2 : 1;
  return cudaLaunchKernelEx(&cfg, lstm_layer_tc2_kernel, args);
}

}  // namespace rnnt
