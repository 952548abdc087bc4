// Feature front-end: framed STFT (hann(400) in a 1024-point frame, hop 160, reflect
// padding) -> power -> HTK mel filterbank -> log(x + 1e-6) -> 10-frame stack / 8-frame
// hop, written directly in the reference's (mel-major, stack-minor) feature layout.
// Replaces TransformTime.encodes + StackDownsample.encodes (+ StreamPostprocess for the
// serving window): reference libreasr/lib/transforms.py:301-323, 335-342, 436-441.
//
// One CTA per output row (b, t): warp s computes frame t*D + frame0 + s (real 1024-point FFT
// as a 512-point complex radix-8 Stockham FFT in registers + untangle; only the 400 windowed
// samples are non-zero), the CTA then writes the X = n_mels*n_stack floats of the row with
// one coalesced pass.  Audio is read once per frame (25% of frames are
// shared by two rows and recomputed: the kernel is FFT-, not HBM-bound; see DESIGN.md).
#include "kernels.h"

namespace rnnt {

namespace {

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

// MINB = CTAs per SM the register allocation must allow (1: ~125 registers, one 10-warp CTA per SM = 16 % of the warp slots;
// 2: <= 102 registers so that two CTAs share an SM and hide each other's FFT latency)
template <int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB)
mel_stack_kernel(FrontendArgs p) {
  extern __shared__ __align__(16) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = blockIdx.x, b = blockIdx.y;

  float2* tw = reinterpret_cast<float2*>(smem);                 // [512] exp(-2 pi i j / 1024)
  float* lm = smem + 1024;                                      // [n_stack][n_mels]
  float* wbase = lm + p.n_stack * p.n_mels;
  wbase += (4 - ((p.n_stack * p.n_mels) & 3)) & 3;              // keep float2/float4 alignment
  float2* z = reinterpret_cast<float2*>(wbase + warp * (1152 + 520));  // [512 (+64 pad)] complex, phys(i) = i + i/8
  float* P = wbase + warp * (1152 + 520) + 1152;                // [513] power spectrum

  for (int i = threadIdx.x; i < 512; i += blockDim.x) tw[i] = p.tw[i];

  const int len = p.lens ? p.lens[b] : (int)p.n;
  const int F = len / p.hop + 1;
  const int Tb = (F >= p.n_stack) ? (F - p.n_stack) / p.D + 1 : 0;
  float* orow = p.out + ((size_t)b * p.T_out + t) * (size_t)(p.n_mels * p.n_stack);
  const bool valid = p.is_stream ? true : (t < Tb);
  if (!valid) {  // uniform per CTA
    for (int i = threadIdx.x; i < p.n_mels * p.n_stack; i += blockDim.x) orow[i] = 0.f;
    return;
  }
  __syncthreads();

  // ---- 512-point complex FFT of z[m] = x[2m] + i x[2m+1] (windowed frame, zero beyond win/2) ----
  // Radix-8 Stockham autosort, 3 passes (Ns = 1, 8, 64); every lane owns butterflies j = lane and lane + 32.
  // Pass 1 takes its inputs straight from global memory (window applied on the fly); between passes the warp
  // exchanges through its private smem buffer, indexed with phys(i) = i + i/8 so that the stride-8 stores of
  // pass 1 spread over the banks.  (The radix-2 version this replaces spent 87 % of smem bandwidth.)
  const float* x = p.audio + (size_t)b * p.n;
  const int f = t * p.D + p.frame0 + warp;
  const int start = f * p.hop - p.win / 2;
  const int half_win = p.win / 2;
  auto load_in = [&](int m) -> float2 {
    float2 v = make_float2(0.f, 0.f);
    if (m < half_win) {
      int i0 = start + 2 * m, i1 = i0 + 1;
      if (i0 < 0) i0 = -i0;
      if (i1 < 0) i1 = -i1;
      if (i0 >= len) i0 = 2 * (len - 1) - i0;
      if (i1 >= len) i1 = 2 * (len - 1) - i1;
      i0 = min(max(i0, 0), len - 1);
      i1 = min(max(i1, 0), len - 1);
      v.x = __ldg(x + i0) * __ldg(p.window + 2 * m);
      v.y = __ldg(x + i1) * __ldg(p.window + 2 * m + 1);
    }
    return v;
  };
  auto tw512 = [&](int n) -> float2 {   // exp(-2 pi i n / 512), n in [0, 512): table holds angles below pi
    const float2 w = tw[(n & 255) * 2];
    return (n & 256) ? make_float2(-w.x, -w.y) : w;
  };
  auto phys = [](int i) { return i + (i >> 3); };
  // in-register 8-point DFT (natural order out): three radix-2 layers
  auto dft8 = [](float2 (&v)[8]) {
    const float r = 0.70710678118654752440f;
    auto bf = [](float2& a, float2& bb) { const float2 t = a; a = make_float2(t.x + bb.x, t.y + bb.y); bb = make_float2(t.x - bb.x, t.y - bb.y); };
    bf(v[0], v[4]); bf(v[1], v[5]); bf(v[2], v[6]); bf(v[3], v[7]);
    v[5] = make_float2(r * (v[5].x + v[5].y), r * (v[5].y - v[5].x));    // * exp(-i pi/4)
    v[6] = make_float2(v[6].y, -v[6].x);                                   // * (-i)
    v[7] = make_float2(r * (v[7].y - v[7].x), -r * (v[7].x + v[7].y));   // * exp(-3 i pi/4)
    bf(v[0], v[2]); bf(v[1], v[3]); bf(v[4], v[6]); bf(v[5], v[7]);
    v[3] = make_float2(v[3].y, -v[3].x);
    v[7] = make_float2(v[7].y, -v[7].x);
    bf(v[0], v[1]); bf(v[2], v[3]); bf(v[4], v[5]); bf(v[6], v[7]);
    // bit-reversed -> natural: (0,4,2,6,1,5,3,7)
    float2 t1 = v[1]; v[1] = v[4]; v[4] = t1;
    float2 t3 = v[3]; v[3] = v[6]; v[6] = t3;
  };
#pragma unroll 1
  for (int pass = 0; pass < 3; ++pass) {
    const int Ns = pass == 0 ? 1 : (pass == 1 ? 8 : 64);
    float2 v[2][8];
#pragma unroll
    for (int h2 = 0; h2 < 2; ++h2) {
      const int j = lane + 32 * h2;
      const int k = j & (Ns - 1);
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        float2 a = pass == 0 ? load_in(j + 64 * r) : z[phys(j + 64 * r)];
        if (pass > 0 && r > 0) a = cmul(a, tw512(k * r * (64 / Ns)));
        v[h2][r] = a;
      }
      dft8(v[h2]);
    }
    __syncwarp();
#pragma unroll
    for (int h2 = 0; h2 < 2; ++h2) {
      const int j = lane + 32 * h2;
      const int k = j & (Ns - 1);
      const int j0 = ((j - k) << 3) + k;   // (j / Ns) * Ns * 8 + k
#pragma unroll
      for (int r = 0; r < 8; ++r) z[phys(j0 + r * Ns)] = v[h2][r];
    }
    __syncwarp();
  }

  // ---- untangle the real FFT and take the power: P[k], P[512-k] for k = 0..256 ----
  for (int k = lane; k <= 256; k += 32) {
    const float2 zk = z[k + (k >> 3)];
    const int kn = (512 - k) & 511;
    const float2 zn = z[kn + (kn >> 3)];
    const float2 xe = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
    const float2 xo = make_float2(0.5f * (zk.y + zn.y), -0.5f * (zk.x - zn.x));
    const float2 wx = cmul(tw[k], xo);
    const float ar = xe.x + wx.x, ai = xe.y + wx.y;
    const float br = xe.x - wx.x, bi = xe.y - wx.y;
    P[k] = ar * ar + ai * ai;
    P[512 - k] = br * br + bi * bi;
  }
  __syncwarp();

  // ---- sparse triangular mel filterbank + log ----
  for (int m = lane; m < p.n_mels; m += 32) {
    const int k0 = p.mel_start[m], cnt = p.mel_count[m];
    const float* w = p.mel_w + p.mel_off[m];
    float s = 0.f;
    for (int i = 0; i < cnt; ++i) s = fmaf(w[i], P[k0 + i], s);
    lm[warp * p.n_mels + m] = logf(s + p.log_offset);
  }
  __syncthreads();

  // ---- stacked row: feature index = m * n_stack + s (transforms.py:439-440) ----
  const int X = p.n_mels * p.n_stack;
  for (int i = threadIdx.x; i < X; i += blockDim.x) {
    const int m = i / p.n_stack, s = i - m * p.n_stack;
    orow[i] = lm[s * p.n_mels + m];
  }
}

// LayerNorm over the feature axis (Encoder.input_norm, models.py:84,107): one warp per row.
__global__ void __launch_bounds__(256) layernorm_rows_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                             const float* __restrict__ gamma, const float* __restrict__ beta,
                                                             int64_t rows, int X, float eps) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const float* r = in + (size_t)warp * X;
  float s = 0.f;
  for (int i = lane; i < X; i += 32) s += r[i];
  const float mean = warp_sum(s) / (float)X;
  float v = 0.f;
  for (int i = lane; i < X; i += 32) {
    const float d = r[i] - mean;
    v = fmaf(d, d, v);
  }
  const float inv = 1.0f / sqrtf(warp_sum(v) / (float)X + eps);
  float* o = out + (size_t)warp * X;
  for (int i = lane; i < X; i += 32) o[i] = (r[i] - mean) * inv * gamma[i] + beta[i];
}

// Polyphase windowed-sinc resampler (torchaudio.transforms.Resample as the reference calls it, transforms.py:135-144):
// out[b][j * n_new + p] = sum_k tab[p][k] * x[b][j * n_orig + k - width]   (zero outside the utterance)
__global__ void __launch_bounds__(256) resample_kernel(const float* __restrict__ x, int64_t n, const float* __restrict__ tab,
                                                       int n_orig, int n_new, int width, int K, float* __restrict__ out, int64_t L) {
  const int b = blockIdx.y;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L) return;
  const int64_t j = i / n_new;
  const int p = (int)(i - j * n_new);
  const float* xb = x + (size_t)b * n;
  const float* t = tab + (size_t)p * K;
  const int64_t s0 = j * n_orig - width;
  float acc = 0.f;
  for (int k = 0; k < K; ++k) {
    const int64_t s = s0 + k;
    if (s >= 0 && s < n) acc = fmaf(t[k], xb[s], acc);
  }
  out[(size_t)b * L + i] = acc;
}

}  // namespace

size_t frontend_smem_bytes(int n_stack, int n_mels) {
  size_t fl = 1024 + (size_t)n_stack * n_mels + 4 + (size_t)n_stack * (1152 + 520);
  return fl * sizeof(float);
}

cudaError_t launch_mel_stack(const FrontendArgs& a, int B, cudaStream_t st) {
  if (a.n_stack > kFrontendMaxWarps) return cudaErrorInvalidValue;
  const size_t smem = frontend_smem_bytes(a.n_stack, a.n_mels);
  dim3 grid(a.T_out, B);
  cudaError_t e;
  if (a.n_stack * 32 <= 320) {   // two CTAs per SM
    e = cudaFuncSetAttribute(mel_stack_kernel<320, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    mel_stack_kernel<320, 2><<<grid, a.n_stack * 32, smem, st>>>(a);
  } else {
    e = cudaFuncSetAttribute(mel_stack_kernel<kFrontendMaxWarps * 32, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    mel_stack_kernel<kFrontendMaxWarps * 32, 1><<<grid, a.n_stack * 32, smem, st>>>(a);
  }
  return cudaGetLastError();
}

cudaError_t launch_layernorm(const float* in, float* out, const float* gamma, const float* beta, int64_t rows, int X,
                             float eps, cudaStream_t st) {
  const int64_t blocks = ceil_div(rows, 8);
  layernorm_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(in, out, gamma, beta, rows, X, eps);
  return cudaGetLastError();
}

cudaError_t launch_resample(const float* x, int B, int64_t n, const float* tab, int n_orig, int n_new, int width, int K, float* out,
                            int64_t L, cudaStream_t st) {
  dim3 grid((unsigned)ceil_div(L, 256), (unsigned)B);
  resample_kernel<<<grid, 256, 0, st>>>(x, n, tab, n_orig, n_new, width, K, out, L);
  return cudaGetLastError();
}

}  // namespace rnnt
