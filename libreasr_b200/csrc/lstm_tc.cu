// Persistent tcgen05 LSTM layer: the recurrent half of the LSTM gate GEMMs on the 5th-gen
// tensor cores, one launch per layer for ALL time steps.
// Replaces torch.nn.LSTM as driven by CustomRNN.forward_one_rnn (reference
// libreasr/lib/layers/custom_rnn.py:140-175, arithmetic haste/lstm.py:51-60, gate order
// i,f,g,o) + the per-layer BatchNorm1d eval (custom_rnn.py:210-213).
//
// Decomposition.  CTA c owns U hidden units = NC = 4U interleaved gate rows of W_hh and
// keeps that slice (hi+lo fp16 operand image, NC x H x 4 bytes) RESIDENT in shared memory
// for the whole layer when it fits (H = 1024: 128 KB); otherwise it is streamed per step.
// Each step is one skinny GEMM with the BATCH on the MMA M axis and the CTA's gate rows on
// N, so all H/U CTAs (128 of the 148 SMs at H = 1024) share every step.  The 3xFP16 split
// (gemm_tc.cu) is folded into ONE instruction per 16-deep k slice: the A tile stacks the hi
// rows of the batch on top of its lo rows, the B tile the hi rows of the weight slice on top
// of its lo rows, so  [A_hi;A_lo] x [B_hi;B_lo]^T  yields hi*hi, hi*lo, lo*hi (and lo*lo) in
// four quadrants of one M64/M128 x 2NC accumulator (measured: a tcgen05.mma costs >= ~25-50
// cycles however small it is, so instruction count is what matters at batch 32).
//   warp 0     producer: waits for the grid-wide "h_{t-1} complete" counter, then streams the
//              h_{t-1} operand image (B rows x 64 k, hi|lo) per k-block with TMA bulk copies
//   warp 1     one thread issues 12 tcgen05.mma (M128 x NC x K16) per k-block into TMEM
//   warps 2-5  epilogue: thread (q, lane) owns batch row 32q+lane: tcgen05.ld its NC gate
//              pre-activations, adds the hoisted input projection xp, applies the cell with
//              c (and h) kept in REGISTERS across steps, writes h_t straight into the next
//              step's operand image (fp16 hi/lo, swizzled) and BatchNorm(h_t) both as fp32
//              and as the operand image of the next layer's input GEMM; then arrives on the
//              readiness counter of its 64-unit k-block (release) that the producers poll (acquire).
// There is no grid-wide rendezvous: a k-block of h_t is consumable as soon as its 64/U owner CTAs published it.
#include "kernels.h"
#include "tc_common.cuh"

namespace rnnt {
namespace {

constexpr int LT_THREADS = 192;
constexpr int LT_MAX_U = 16;

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

struct Smem {
  uint8_t* ring;
  uint8_t* wres;
  float* pre_hi;
  float* pre_lo;
  uint64_t *full, *empty, *tfull, *tempty, *wfull;
  uint32_t* tptr;
};

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

template <bool FUSED>
__global__ void __launch_bounds__(LT_THREADS, 1) lstm_layer_tc_kernel(LstmTcArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024 - (smem_u32(smem_raw) & 1023)) & 1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cta = blockIdx.x;
  const int NC = p.NC, U = p.U, KB = p.KB, S = p.stages, KPS = p.kps, MM = p.mma_m;
  constexpr bool fused = FUSED;                          // hi and lo rows of the batch share one A tile
  const uint32_t xr = (uint32_t)p.Bpad8 * 128;          // valid rows of one part of an h tile
  const uint32_t wtile = (uint32_t)NC * 256;            // hi + lo weight tile of one k-block
  const uint32_t xstage = (uint32_t)KPS * 2 * xr;
  const uint32_t stage_bytes = xstage + (p.w_resident ? 0 : KPS * wtile);
  const int n_groups = KB / KPS;                        // stage fills per time step
  Smem sm;
  sm.ring = base;
  sm.wres = base + (size_t)S * stage_bytes;
  sm.pre_hi = reinterpret_cast<float*>(base + p.pre_offset);
  sm.pre_lo = sm.pre_hi + 64 * (NC + 1);
  uint8_t* bars = base + p.bar_offset;
  sm.full = reinterpret_cast<uint64_t*>(bars);
  sm.empty = sm.full + S;
  sm.tfull = sm.empty + S;
  sm.tempty = sm.tfull + 1;
  sm.wfull = sm.tempty + 1;
  sm.tptr = reinterpret_cast<uint32_t*>(sm.wfull + 1);

  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&sm.full[s], 1);
      mbar_init(&sm.empty[s], 1);
    }
    mbar_init(sm.tfull, 1);
    mbar_init(sm.tempty, 128);
    mbar_init(sm.wfull, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(sm.tptr, p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *sm.tptr;

  if (warp == 0) {
    // =========================== producer (warp-uniform, one elected lane issues) ===========================
    if (p.w_resident && elect_one()) {
      mbar_arrive_expect_tx(sm.wfull, (uint32_t)KB * wtile);
      tma_bulk_g2s(sm.wres, p.w_img + img_tile_offset(cta, 0, 0, KB, NC), (uint32_t)KB * wtile, sm.wfull);
    }
    uint32_t g = 0;
    for (int t = 0; t < p.T; ++t) {
      // h_{t-1} is published per 64-unit k-block: p.barrier[kb] counts the (64 / U) CTAs that own its units, so the
      // first k-blocks stream in while slower CTAs are still in their epilogue (no single grid-wide rendezvous)
      const unsigned target = (unsigned)(t + 1) * (unsigned)(64 / U);
      const uint8_t* ximg = p.x_img[t & 1];
      uint32_t ready = 0;   // k-blocks of h_{t-1} known to be published (lane i polls counter i: one L2 round trip per poll)
      for (int gi = 0; gi < n_groups; ++gi, ++g) {
        const uint32_t need = ((KPS >= 32 ? 0u : (1u << KPS)) - 1u) << (gi * KPS);
        while ((ready & need) != need) {
          const bool ok = lane < KB ? (ld_acquire_u32(p.barrier + lane) >= target) : true;
          ready = __ballot_sync(0xffffffffu, ok);
        }
        fence_proxy_async_global();
        const int s = g % S;
        const uint32_t ph = (g / S) & 1;
        mbar_wait(&sm.empty[s], ph ^ 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(&sm.full[s], stage_bytes);
          uint8_t* dst = sm.ring + (size_t)s * stage_bytes;
          tma_bulk_g2s(dst, ximg + (size_t)gi * xstage, xstage, &sm.full[s]);
          if (!p.w_resident)
            tma_bulk_g2s(dst + xstage, p.w_img + img_tile_offset(cta, gi * KPS, 0, KB, NC), KPS * wtile, &sm.full[s]);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===========================
    // Warp-uniform control flow; ONE elected lane per pipeline stage issues all of the stage's
    // tcgen05.mma.  Descriptors are a loop-invariant base plus small 16-byte-unit offsets (+2 per
    // 16-deep k slice) so that the per-instruction overhead stays near the ~35-50 cycle issue floor.
    const uint32_t idesc = umma_idesc_f16(MM, 2 * NC);   // [A_hi;A_lo] (or A_hi / A_lo) x [B_hi ; B_lo]
    const uint64_t a_desc0 = umma_desc_sw128(smem_u32(sm.ring));
    const uint64_t b_desc0 = umma_desc_sw128(p.w_resident ? smem_u32(sm.wres) : smem_u32(sm.ring) + xstage);
    const uint32_t stage_u = stage_bytes >> 4, kb_u = (2 * xr) >> 4, lo_u = xr >> 4, wt_u = wtile >> 4;
    const bool wres = p.w_resident != 0;
    if (wres) mbar_wait(sm.wfull, 0);
    uint32_t g = 0;
    for (int t = 0; t < p.T; ++t) {
      if (t > 0) mbar_wait(sm.tempty, (t - 1) & 1);
      tc_fence_after();
      for (int gi = 0; gi < n_groups; ++gi, ++g) {
        const int s = g % S;
        const uint32_t ph = (g / S) & 1;
        mbar_wait(&sm.full[s], ph);
        tc_fence_after();
        if (elect_one()) {
          uint64_t ad = a_desc0 + (uint64_t)(s * stage_u);
          uint64_t bd = b_desc0 + (uint64_t)(wres ? (uint32_t)(gi * KPS) * wt_u : s * stage_u);
          uint32_t accumulate = gi == 0 ? 0u : 1u;
          for (int i = 0; i < KPS; ++i) {
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4) {
              tc_mma_f16(tmem, ad + 2 * k4, bd + 2 * k4, idesc, accumulate);
              if (!FUSED) tc_mma_f16(tmem + 2 * NC, ad + lo_u + 2 * k4, bd + 2 * k4, idesc, accumulate);
              accumulate = 1u;
            }
            ad += kb_u;
            bd += wt_u;
          }
          tc_commit(&sm.empty[s]);
          if (gi == n_groups - 1) tc_commit(sm.tfull);
        }
        __syncwarp();
      }
    }
  } else {
    // =========================== epilogue ===========================
    const int q = warp & 3;
    const int et = (warp - 2) * 32 + lane;  // 0..127
    const int H = p.H;
    const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);
    // ownership.  fused (B <= 64): accumulator rows are redistributed through smem and thread et owns
    // batch row et % Bq and U*Bq/128 units (Bq = 32 or 64); else (B > 64): thread = TMEM lane = batch row, all U units
    const int Bq = fused ? (p.Bpad8 <= 32 ? 32 : 64) : 128;
    const int upt = fused ? U * Bq / 128 : U;             // units per thread
    const int b = fused ? (et % Bq) : q * 32 + lane;
    const int unit0 = cta * U + (fused ? (et / Bq) * upt : 0);
    const bool valid = b < p.B && upt > 0;
    float c[LT_MAX_U], h[LT_MAX_U], bsc[LT_MAX_U], bsh[LT_MAX_U];
    const int len = valid ? (p.lens_T ? min(p.lens_T[b], p.T) : p.T) : 0;
#pragma unroll
    for (int j = 0; j < LT_MAX_U; ++j) {
      if (j < upt && valid) {
        h[j] = p.state_h_in ? p.state_h_in[(size_t)b * H + unit0 + j] : p.h_init_vec[unit0 + j];
        c[j] = p.state_c_in ? p.state_c_in[(size_t)b * H + unit0 + j] : p.c_init_vec[unit0 + j];
        bsc[j] = p.bn_scale[unit0 + j];
        bsh[j] = p.bn_shift[unit0 + j];
      } else {
        h[j] = 0.f; c[j] = 0.f; bsc[j] = 0.f; bsh[j] = 0.f;
      }
    }
    // h_t of this thread's units -> h operand image (TR = Bpad8 row tiles, [kb][part] contiguous)
    auto store_h = [&](uint8_t* img, const float* v) {
      const int n = upt < 4 ? upt : 4;
#pragma unroll
      for (int j0 = 0; j0 < LT_MAX_U; j0 += 4) {
        if (j0 < upt) {
          const int k = unit0 + j0;
          uint8_t* hi = img + (size_t)((k >> 6) * 2) * xr;
          store_split(hi, hi + xr, b, k & 63, n, v + j0);
        }
      }
    };
    // BatchNorm(h_t) -> operand image (TR = 128 row tiles) of the next layer's input GEMM
    auto store_yimg = [&](int64_t row, const float* v) {
      const int n = upt < 4 ? upt : 4;
#pragma unroll
      for (int j0 = 0; j0 < LT_MAX_U; j0 += 4) {
        if (j0 < upt) {
          const int k = unit0 + j0;
          uint8_t* hi = p.y_img + img_tile_offset(row >> 7, k >> 6, 0, KB, 128);
          store_split(hi, hi + 128 * 128, (int)(row & 127), k & 63, n, v + j0);
        }
      }
    };
    unsigned* my_flag = p.barrier + (cta * U) / 64;   // readiness counter of the k-block holding this CTA's units
    if (valid) store_h(p.x_img[0], h);
    named_bar_sync(1, 128);
    if (et == 0) red_release_add(my_flag, 1u);

    const int prs = NC + 1;  // row stride of the exchange buffers
    for (int t = 0; t < p.T; ++t) {
      const int64_t row = (int64_t)b * p.T + t;
      // hoisted input projection of this thread's units for step t: issued before the accumulators are ready
      float4 xv[LT_MAX_U];
#pragma unroll
      for (int j = 0; j < LT_MAX_U; ++j)
        if (j < upt && valid) xv[j] = *reinterpret_cast<const float4*>(p.xp + row * (size_t)(4 * H) + (size_t)(unit0 + j) * 4);
      mbar_wait(sm.tfull, t & 1);
      tc_fence_after();
      float hy[LT_MAX_U];
      if (fused) {
        // accumulator row r: r < Bpad8 -> hi row of batch r; else lo row of batch r - Bpad8.
        // M = 64: row r sits in TMEM lane (r % 16) + 32 * (r / 16); M = 128: lane r.
        const int rows_per_warp = MM == 64 ? 16 : 32;
        const int r = q * rows_per_warp + lane;
        if (q * rows_per_warp < 2 * p.Bpad8) {
          const bool mine = lane < rows_per_warp && r < 2 * p.Bpad8;
          const bool is_lo = r >= p.Bpad8;
          float* dstrow = (is_lo ? sm.pre_lo + (r - p.Bpad8) * prs : sm.pre_hi + r * prs);
          const float sc = is_lo ? kLoInv : 1.0f;
          for (int c0 = 0; c0 < NC; c0 += 16) {
            float d0[16], d1[16];
            tmem_ld16(tlane + c0, d0);
            tmem_ld16(tlane + NC + c0, d1);
            tmem_ld_wait();
            if (mine) {
#pragma unroll
              for (int i = 0; i < 16; ++i) dstrow[c0 + i] = sc * fmaf(d1[i], kLoInv, d0[i]);
            }
          }
        }
        tc_fence_before();
        mbar_arrive(sm.tempty);
        named_bar_sync(1, 128);
        if (valid) {
          const int lc = (unit0 - cta * U) * 4;
          const float* ph = sm.pre_hi + b * prs + lc;
          const float* pl = sm.pre_lo + b * prs + lc;
#pragma unroll
          for (int j = 0; j < LT_MAX_U; ++j) {
            if (j < upt) {
              if (t < len) {
                const float vi = (ph[4 * j + 0] + pl[4 * j + 0]) + xv[j].x, vf = (ph[4 * j + 1] + pl[4 * j + 1]) + xv[j].y;
                const float vg = (ph[4 * j + 2] + pl[4 * j + 2]) + xv[j].z, vo = (ph[4 * j + 3] + pl[4 * j + 3]) + xv[j].w;
                const float cn = sigmoidf_acc(vf) * c[j] + sigmoidf_acc(vi) * tanhf(vg);
                c[j] = cn;
                h[j] = sigmoidf_acc(vo) * tanhf(cn);
              }
              hy[j] = h[j] * bsc[j] + bsh[j];
            }
          }
        }
      } else {
#pragma unroll
        for (int j0 = 0; j0 < LT_MAX_U; j0 += 4) {  // 16 gate columns = 4 units per chunk
          if (j0 < U) {
            float d0[16], d1[16], e0[16], e1[16];
            tmem_ld16(tlane + j0 * 4, d0);                 // hi*hi
            tmem_ld16(tlane + NC + j0 * 4, d1);            // hi*lo
            tmem_ld16(tlane + 2 * NC + j0 * 4, e0);        // lo*hi
            tmem_ld16(tlane + 3 * NC + j0 * 4, e1);        // lo*lo
            tmem_ld_wait();
            if (valid) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                if (t < len) {
                  float pre[4];
#pragma unroll
                  for (int gg = 0; gg < 4; ++gg) {
                    const int i = 4 * j + gg;
                    pre[gg] = fmaf(d1[i], kLoInv, d0[i]) + kLoInv * fmaf(e1[i], kLoInv, e0[i]);
                  }
                  const float vi = pre[0] + xv[j0 + j].x, vf = pre[1] + xv[j0 + j].y;
                  const float vg = pre[2] + xv[j0 + j].z, vo = pre[3] + xv[j0 + j].w;
                  const float cn = sigmoidf_acc(vf) * c[j0 + j] + sigmoidf_acc(vi) * tanhf(vg);
                  c[j0 + j] = cn;
                  h[j0 + j] = sigmoidf_acc(vo) * tanhf(cn);
                }
                hy[j0 + j] = h[j0 + j] * bsc[j0 + j] + bsh[j0 + j];
              }
            }
          }
        }
        tc_fence_before();
        mbar_arrive(sm.tempty);
      }
      // Only h_t gates the next step: publish it first (stores -> CTA barrier -> one gpu-scope release on the
      // step counter, paired with the consumers' ld.acquire + fence.proxy.async before their TMA reads);
      // the BatchNorm(h_t) outputs for the next layer are written after the release, off the critical path.
      if (valid) store_h(p.x_img[(t + 1) & 1], h);
      named_bar_sync(1, 128);
      if (et == 0) red_release_add(my_flag, 1u);
      if (valid) {
        if (p.y) {
          float* yo = p.y + row * H + unit0;
          if (upt >= 4) {
#pragma unroll
            for (int j0 = 0; j0 < LT_MAX_U; j0 += 4)
              if (j0 < upt) *reinterpret_cast<float4*>(yo + j0) = make_float4(hy[j0], hy[j0 + 1], hy[j0 + 2], hy[j0 + 3]);
          } else if (upt == 2) {
            *reinterpret_cast<float2*>(yo) = make_float2(hy[0], hy[1]);
          } else {
            yo[0] = hy[0];
          }
        }
        if (p.y_img) store_yimg(row, hy);
      }
    }
    if (valid) {
#pragma unroll
      for (int j = 0; j < LT_MAX_U; ++j) {
        if (j < upt) {
          if (p.state_h_out) p.state_h_out[(size_t)b * H + unit0 + j] = h[j];
          if (p.state_c_out) p.state_c_out[(size_t)b * H + unit0 + j] = c[j];
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, p.tmem_cols);
}

}  // namespace

cudaError_t configure_lstm_tc() {
  cudaError_t e = cudaFuncSetAttribute(lstm_layer_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(lstm_layer_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

// Chooses the decomposition for hidden size H, batch B on a device with `sms` SMs; false if none fits.
bool lstm_tc_plan(int H, int B, int sms, LstmTcPlan* pl) {
  if (B < 1 || B > 128 || H % 64 || H > 2048) return false;   // H / 64 <= 32: one polling lane per k-block counter
  int U = 0;
  for (int u : {4, 8, 16})
    if (H % u == 0 && H / u <= sms) { U = u; break; }
  if (!U) return false;
  pl->U = U;
  pl->NC = 4 * U;
  pl->grid = H / U;
  pl->KB = H / 64;
  pl->Bpad8 = (int)round_up(B, 8);
  pl->fused = pl->Bpad8 <= 64 ? 1 : 0;                     // hi + lo rows of the batch fit one MMA M tile
  pl->mma_m = (pl->fused && 2 * pl->Bpad8 <= 64) ? 64 : 128;
  if (pl->fused && (U * (pl->Bpad8 <= 32 ? 32 : 64)) % 128) return false;
  int cols = 32;
  while (cols < (pl->fused ? 2 : 4) * pl->NC) cols *= 2;
  if (cols > 512) return false;
  pl->tmem_cols = cols;
  const size_t xr = (size_t)pl->Bpad8 * 128, wtile = (size_t)pl->NC * 256;
  const size_t guard = (size_t)pl->mma_m * 128;   // an A tile is read as mma_m rows; rows beyond the valid ones alias what follows
  const size_t pre_bytes = pl->fused ? round_up((size_t)2 * 64 * (pl->NC + 1) * 4, 1024) : 0;
  const size_t budget = 227 * 1024 - 2048 /*alignment slack + barriers*/ - guard - pre_bytes;
  const size_t wall = (size_t)pl->KB * wtile;
  for (int want_res = 1; want_res >= 0; --want_res) {   // prefer the W-resident layout
    for (int kps : {4, 2, 1}) {
      if (pl->KB % kps) continue;
      const size_t xstage = (size_t)kps * 2 * xr;
      const bool res = wall + 3 * xstage <= budget;
      if (res != (want_res != 0)) continue;
      const size_t stage = xstage + (res ? 0 : kps * wtile);
      const size_t avail = budget - (res ? wall : 0);
      int S = (int)(avail / stage);
      if (S > 8) S = 8;
      if (S < 3 && !(kps == 1 && S >= 2)) continue;
      pl->kps = kps;
      pl->w_resident = res ? 1 : 0;
      pl->stages = S;
      const size_t used = (size_t)S * stage + (res ? wall : 0) + guard;
      pl->pre_offset = (int)round_up(used, 1024);
      pl->bar_offset = pl->pre_offset + (int)pre_bytes;
      pl->smem_bytes = pl->bar_offset + 1024 + 1024;
      return pl->smem_bytes <= 227 * 1024;
    }
  }
  return false;
}

cudaError_t launch_lstm_layer_tc(const LstmTcArgs& a, const LstmTcPlan& pl, cudaStream_t st) {
  LstmTcArgs args = a;
  args.U = pl.U; args.NC = pl.NC; args.KB = pl.KB; args.Bpad8 = pl.Bpad8; args.stages = pl.stages;
  args.w_resident = pl.w_resident; args.bar_offset = pl.bar_offset; args.tmem_cols = pl.tmem_cols;
  args.kps = pl.kps; args.mma_m = pl.mma_m; args.fused = pl.fused; args.pre_offset = pl.pre_offset;
  void* kargs[] = {&args};
  void* fn = pl.fused ? (void*)lstm_layer_tc_kernel<true> : (void*)lstm_layer_tc_kernel<false>;
  return launch_persistent(fn, dim3(pl.grid), dim3(LT_THREADS), kargs, pl.smem_bytes, st);
}

}  // namespace rnnt
