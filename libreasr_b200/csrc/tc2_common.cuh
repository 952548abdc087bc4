// Building blocks shared by the cluster split-K kernels (lstm_tc2.cu, decode_tc2.cu): gpu-scope relaxed vector
// loads / stores for the tagged-chunk exchange, distributed-shared-memory stores and remote mbarrier arrives,
// cluster barriers, 32-column TMEM loads, the hi/lo split with an embedded sequence tag.
#pragma once
#include <cuda_fp16.h>

#include "tc_common.cuh"

namespace rnnt {
namespace {

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_add(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ uint4 ld_relaxed_v4(const void* p) {
  uint4 v;
  asm volatile("ld.relaxed.gpu.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
// 32 lanes x 32 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// x ~= hi + lo * 2^-11.  With `tagged`, the LSB of both halves is a 1-bit sequence tag on the wire: the VALUE uses
// LSB = 0 (hi is truncated to an even code before lo is derived from it, so the pair still represents x to ~2^-21
// relative), the consumer clears the bit again (`chunk_strip_tag`) -- the operand never depends on the tag.
__device__ __forceinline__ void split_tag(float x, bool tagged, uint32_t tag, uint32_t& hi, uint32_t& lo) {
  __half h = __float2half_rn(x);
  uint32_t hb = __half_as_ushort(h);
  if (tagged) {
    hb &= 0xFFFEu;
    h = __ushort_as_half((unsigned short)hb);
  }
  const __half l = __float2half_rn((x - __half2float(h)) * kLoScale);
  uint32_t lb = __half_as_ushort(l);
  if (tagged) lb &= 0xFFFEu;
  hi = hb | (tagged ? tag : 0u);
  lo = lb | (tagged ? tag : 0u);
}
// a 16-byte chunk carries its tag in the LSB of its last half (bit 16 of word 3)
__device__ __forceinline__ bool chunk_tag_ok(const uint4& r, uint32_t tag) { return ((r.w >> 16) & 1u) == tag; }
__device__ __forceinline__ void chunk_strip_tag(uint4& r) { r.w &= 0xFFFEFFFFu; }

// Tagged-chunk fetch of NKB k-blocks x 4 chunks per thread (chunk i at src + i * 2048).  The warp spins, converged, on
// chunk 0 until ANY lane sees the new tag (one coalesced request per round trip: nothing is worth loading earlier), then
// issues every load back to back; `poll_validate_kb` afterwards re-reads only the stale chunks of one k-block, in
// parallel rounds, so the first k-blocks can be handed to the MMA while the stragglers of the later ones are in flight.
template <int N>
__device__ __forceinline__ void poll_issue(const uint8_t* src, int n, uint32_t tag, uint4 (&r)[N], int min_valid = 1) {
  // lanes 0-7 = the eight chunks (eight producer CTAs) of one 128-byte line: one sector request per producer and round trip
  const bool poller = (threadIdx.x & 31) < 8;
  r[0] = make_uint4(0u, 0u, 0u, (tag ^ 1u) << 16);
  for (;;) {
    if (poller) r[0] = ld_relaxed_v4(src);
    if (__popc(__ballot_sync(0xffffffffu, poller && chunk_tag_ok(r[0], tag))) >= min_valid) break;   // min_valid of the 8 producers have published
  }
  if (!poller) r[0] = ld_relaxed_v4(src);
#pragma unroll
  for (int i = 1; i < N; ++i)
    if (i < n) r[i] = ld_relaxed_v4(src + (size_t)i * 2048);
}
template <int N>
__device__ __forceinline__ void poll_validate_kb(const uint8_t* src, int kb, uint32_t tag, uint4 (&r)[N]) {
  for (;;) {
    uint32_t bad = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (!chunk_tag_ok(r[kb * 4 + j], tag)) bad |= 1u << j;
    if (!__any_sync(0xffffffffu, bad != 0u)) break;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if ((bad >> j) & 1u) r[kb * 4 + j] = ld_relaxed_v4(src + (size_t)(kb * 4 + j) * 2048);
  }
}

// Gate non-linearities of the cluster kernels' cells: one ex2.approx and one rcp.approx each.  Absolute error ~1e-7
// (the outputs live in (-1, 1): that is fp32 epsilon), against ~250 dependent instructions for the libm versions on the
// single warp per scheduler that sits on the recurrent chain.
__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_fast(float x) { return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * x)); }

// ---- distributed-shared-memory partial tiles without fences ----
// st.async delivers the value and counts its bytes on the RECEIVER's mbarrier (complete_tx), like a TMA copy: the
// receiver arms the barrier with the byte count of a job (arrive.expect_tx) and waits for the phase -- no release fence
// on the sender (mbarrier.arrive.release.cluster lowers to MEMBAR.ALL.GPU), no acquire + L1 invalidate on the receiver.
__device__ __forceinline__ void st_async_f32(uint32_t remote_addr, float v, uint32_t remote_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.f32 [%0], %1, [%2];" ::"r"(remote_addr), "f"(v), "r"(remote_mbar) : "memory");
}
__device__ __forceinline__ void st_async_b64(uint32_t remote_addr, unsigned long long v, uint32_t remote_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];" ::"r"(remote_addr), "l"(v), "r"(remote_mbar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster_relaxed(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.relaxed.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!ok);
}

}  // namespace
}  // namespace rnnt
