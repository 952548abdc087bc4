// tcgen05 GEMM with 3xFP16 split operands (fp32-grade accuracy on the tensor cores):
//     C[M,N] = A[M,K] * W[N,K]^T + bias[N]
// used for the hoisted LSTM input projections (x_t * W_ih^T for all t at once -- half of the
// LSTM gate FLOPs) and the encoder half of the joint's first Linear.
//
// Each operand element is x ~= hi + lo * 2^-11 with hi, lo fp16 (tc_common.cuh), so the fp32
// product needs three fp16 MMAs with fp32 accumulation in TMEM:
//     D0 += A_hi * B_hi        D1 += A_hi * B_lo + A_lo * B_hi        C = D0 + D1 * 2^-11
// (the dropped lo*lo term is 2^-22 relative).  fp16 x fp16 products are exact in fp32.
//
// One CTA = one 128 x 256 output tile: warp 0 streams [A hi|lo 32 KB][B hi|lo 64 KB] per
// 64-deep k-block from the operand images with two TMA bulk copies into a 2-stage ring,
// one thread of warp 1 issues 12 tcgen05.mma (M128 N256 K16) per k-block into 512 TMEM
// columns (D0 | D1), warps 2-5 drain TMEM (tcgen05.ld 32x32b) and write C with the bias.
#include "kernels.h"
#include "tc_common.cuh"

namespace rnnt {
namespace {

constexpr int GT_BM = 128, GT_BN = 256, GT_STAGES = 2;
constexpr int GT_A_BYTES = 2 * GT_BM * 128;   // hi + lo
constexpr int GT_B_BYTES = 2 * GT_BN * 128;
constexpr int GT_STAGE_BYTES = GT_A_BYTES + GT_B_BYTES;
constexpr int GT_SMEM_BYTES = GT_STAGES * GT_STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
constexpr int GT_THREADS = 192;
#ifndef GT_CHUNK
#define GT_CHUNK 8192
#endif

struct GemmTcArgs {
  const uint8_t* a_img;  // image(TR=128) of A
  const uint8_t* b_img;  // image(TR=256) of W
  const float* bias;     // [N] or nullptr
  float* C;
  int ldc;
  int64_t M;
  int N, KB;
};

__global__ void __launch_bounds__(GT_THREADS, 1) gemm_tc_f16x3_kernel(GemmTcArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024 - (smem_u32(smem_raw) & 1023)) & 1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + GT_STAGES * GT_STAGE_BYTES);
  uint64_t* empty = full + GT_STAGES;
  uint64_t* tfull = empty + GT_STAGES;
  uint32_t* tptr = reinterpret_cast<uint32_t*>(tfull + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nt = blockIdx.x;
  const int64_t mt = blockIdx.y;

  if (threadIdx.x == 0) {
    for (int s = 0; s < GT_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tfull, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tptr, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tptr;

  if (warp == 0) {
    // producer: warp-uniform loop, one elected lane issues the TMA bulk copies
    for (int kb = 0; kb < p.KB; ++kb) {
      const int s = kb % GT_STAGES;
      const uint32_t ph = (kb / GT_STAGES) & 1;
      mbar_wait(&empty[s], ph ^ 1);
      if (elect_one()) {
        mbar_arrive_expect_tx(&full[s], GT_STAGE_BYTES);
        uint8_t* dst = smem + s * GT_STAGE_BYTES;
        // several medium-sized bulk copies in flight instead of two large ones (GT_CHUNK bytes each)
        const uint8_t* asrc = p.a_img + img_tile_offset(mt, kb, 0, p.KB, GT_BM);
        const uint8_t* bsrc = p.b_img + img_tile_offset(nt, kb, 0, p.KB, GT_BN);
#pragma unroll
        for (int o = 0; o < GT_A_BYTES; o += GT_CHUNK) tma_bulk_g2s(dst + o, asrc + o, GT_CHUNK, &full[s]);
#pragma unroll
        for (int o = 0; o < GT_B_BYTES; o += GT_CHUNK) tma_bulk_g2s(dst + GT_A_BYTES + o, bsrc + o, GT_CHUNK, &full[s]);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // MMA issuer: warp-uniform so that the descriptors stay in uniform registers
    const uint32_t idesc = umma_idesc_f16(GT_BM, GT_BN);
    for (int kb = 0; kb < p.KB; ++kb) {
      const int s = kb % GT_STAGES;
      const uint32_t ph = (kb / GT_STAGES) & 1;
      mbar_wait(&full[s], ph);
      tc_fence_after();
      const uint32_t a_base = smem_u32(smem + s * GT_STAGE_BYTES);
      const uint32_t b_base = a_base + GT_A_BYTES;
      const uint64_t a_hi = umma_desc_sw128(a_base), a_lo = umma_desc_sw128(a_base + GT_BM * 128);
      const uint64_t b_hi = umma_desc_sw128(b_base), b_lo = umma_desc_sw128(b_base + GT_BN * 128);
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        const uint32_t acc = (kb > 0 || k4 > 0) ? 1u : 0u;
        if (elect_one()) {  // descriptor start addresses are in 16-byte units: +2 per 16-deep k slice
          tc_mma_f16(tmem, a_hi + 2 * k4, b_hi + 2 * k4, idesc, acc);
          tc_mma_f16(tmem + GT_BN, a_hi + 2 * k4, b_lo + 2 * k4, idesc, acc);
          tc_mma_f16(tmem + GT_BN, a_lo + 2 * k4, b_hi + 2 * k4, idesc, 1u);
        }
      }
      if (elect_one()) tc_commit(&empty[s]);
      __syncwarp();
    }
    if (elect_one()) tc_commit(tfull);
    __syncwarp();
  } else {
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int64_t row = mt * GT_BM + q * 32 + lane;
    mbar_wait(tfull, 0);
    tc_fence_after();
    const uint32_t tbase = tmem + ((uint32_t)(q * 32) << 16);
    for (int c0 = 0; c0 < GT_BN; c0 += 16) {
      float d0[16], d1[16];
      tmem_ld16(tbase + c0, d0);
      tmem_ld16(tbase + GT_BN + c0, d1);
      tmem_ld_wait();
      const int col = nt * GT_BN + c0;
      if (row < p.M && col < p.N) {
        float* out = p.C + row * p.ldc + col;
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          float4 v;
          v.x = fmaf(d1[j + 0], kLoInv, d0[j + 0]);
          v.y = fmaf(d1[j + 1], kLoInv, d0[j + 1]);
          v.z = fmaf(d1[j + 2], kLoInv, d0[j + 2]);
          v.w = fmaf(d1[j + 3], kLoInv, d0[j + 3]);
          if (col + j + 3 < p.N) {
            if (p.bias) {
              const float4 b = *reinterpret_cast<const float4*>(p.bias + col + j);
              v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
            }
            *reinterpret_cast<float4*>(out + j) = v;
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// fp32 row-major [R][ld] -> operand image(TR): one 16-byte chunk (8 halves) of hi and lo per thread
__global__ void __launch_bounds__(256) to_image_kernel(const float* __restrict__ src, int ld, int64_t R, int K, int TR,
                                                       uint8_t* __restrict__ img) {
  const int KB = (K + kImgK - 1) / kImgK;
  const int64_t rt = blockIdx.y;
  const int kb = blockIdx.x;
  uint8_t* hi_t = img + img_tile_offset(rt, kb, 0, KB, TR);
  uint8_t* lo_t = img + img_tile_offset(rt, kb, 1, KB, TR);
  for (int i = threadIdx.x; i < TR * 8; i += blockDim.x) {
    const int r = i >> 3, c = i & 7;
    const int64_t row = rt * TR + r;
    const int k0 = kb * kImgK + c * 8;
    float x[8];
    if (row < R && k0 + 7 < K) {
      const float4 a = *reinterpret_cast<const float4*>(src + row * ld + k0);
      const float4 b = *reinterpret_cast<const float4*>(src + row * ld + k0 + 4);
      x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j] = (row < R && k0 + j < K) ? src[row * ld + k0 + j] : 0.f;
    }
    __align__(16) __half h[8];
    __align__(16) __half l[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) split_f16x3(x[j], h[j], l[j]);
    const uint32_t off = img_elem_offset(r, c * 8);
    *reinterpret_cast<uint4*>(hi_t + off) = *reinterpret_cast<const uint4*>(h);
    *reinterpret_cast<uint4*>(lo_t + off) = *reinterpret_cast<const uint4*>(l);
  }
}

}  // namespace

cudaError_t configure_gemm_tc() {
  return cudaFuncSetAttribute(gemm_tc_f16x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GT_SMEM_BYTES);
}

// rounded to an even number of 128-row tiles: the recurrent kernels write their outputs into this image too
size_t gemm_tc_a_image_bytes(int64_t M, int K) { return img_bytes(round_up(M, 2 * GT_BM), K, GT_BM); }
size_t gemm_tc_w_image_bytes(int N, int K) { return img_bytes(N, K, GT_BN); }

cudaError_t launch_to_image(const float* src, int ld, int64_t R, int K, int TR, uint8_t* img, cudaStream_t st) {
  if ((ld & 3) || (K & 3)) return cudaErrorInvalidValue;
  dim3 grid((unsigned)ceil_div(K, kImgK), (unsigned)ceil_div(R, TR));
  to_image_kernel<<<grid, 256, 0, st>>>(src, ld, R, K, TR, img);
  return cudaGetLastError();
}

cudaError_t launch_gemm_tc(const uint8_t* a_img, const uint8_t* w_img, const float* bias, float* C, int ldc, int64_t M, int N,
                           int K, cudaStream_t st) {
  if ((ldc & 3) || (N & 3)) return cudaErrorInvalidValue;
  GemmTcArgs a;
  a.a_img = a_img; a.b_img = w_img; a.bias = bias; a.C = C; a.ldc = ldc; a.M = M; a.N = N; a.KB = (int)ceil_div(K, kImgK);
  dim3 grid((unsigned)ceil_div(N, GT_BN), (unsigned)ceil_div(M, GT_BM));
  gemm_tc_f16x3_kernel<<<grid, GT_THREADS, GT_SMEM_BYTES, st>>>(a);
  return cudaGetLastError();
}

}  // namespace rnnt
