// Device helpers shared by the single-agent kernels (cx_agent_kernels.cu, cx_agent_obs_kernels.cu).
#pragma once
#include "cx_episode.cuh"

namespace {

template <bool VEC>
__device__ __forceinline__ uint32_t ld_u8x4(const uint8_t* p, int64_t i, int64_t end, uint32_t fill) {
  if (VEC) return __ldcs(reinterpret_cast<const unsigned int*>(p + i));
  uint32_t v = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) v |= (uint32_t)(i + k < end ? p[i + k] : (uint8_t)fill) << (8 * k);
  return v;
}

template <bool VEC>
__device__ __forceinline__ void st_u8x4(uint8_t* p, int64_t i, int64_t end, uint32_t v) {
  if (VEC) {
    __stcs(reinterpret_cast<unsigned int*>(p + i), v);
    return;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (i + k < end) p[i + k] = (uint8_t)(v >> (8 * k));
}

template <bool VEC>
__device__ __forceinline__ void st_f32x4(float* p, int64_t i, int64_t end, const float (&v)[4]) {
  if (VEC) {
    __stcs(reinterpret_cast<float4*>(p + i), make_float4(v[0], v[1], v[2], v[3]));
    return;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (i + k < end) p[i + k] = v[k];
}

// GW-wide variants (GW = 4: the quad helpers above; GW = 2: half quads, for the 64-envs-per-warp build)
template <bool VEC, int GW>
__device__ __forceinline__ uint32_t ld_u8xg(const uint8_t* p, int64_t i, int64_t end, uint32_t fill) {
  if (GW == 4) return ld_u8x4<VEC>(p, i, end, fill);
  if (VEC) return (uint32_t)__ldcs(reinterpret_cast<const unsigned short*>(p + i));
  uint32_t v = 0;
#pragma unroll
  for (int k = 0; k < GW; ++k) v |= (uint32_t)(i + k < end ? p[i + k] : (uint8_t)fill) << (8 * k);
  return v;
}
template <bool VEC, int GW>
__device__ __forceinline__ void st_u8xg(uint8_t* p, int64_t i, int64_t end, uint32_t v) {
  if (GW == 4) {
    st_u8x4<VEC>(p, i, end, v);
    return;
  }
  if (VEC) {
    __stcs(reinterpret_cast<unsigned short*>(p + i), (unsigned short)v);
    return;
  }
#pragma unroll
  for (int k = 0; k < GW; ++k)
    if (i + k < end) p[i + k] = (uint8_t)(v >> (8 * k));
}
template <bool VEC, int GW>
__device__ __forceinline__ void st_f32xg(float* p, int64_t i, int64_t end, const float (&v)[4]) {
  if (GW == 4) {
    st_f32x4<VEC>(p, i, end, v);
    return;
  }
  if (VEC) {
    __stcs(reinterpret_cast<float2*>(p + i), make_float2(v[0], v[1]));
    return;
  }
#pragma unroll
  for (int k = 0; k < GW; ++k)
    if (i + k < end) p[i + k] = v[k];
}

// ---- bulk asynchronous copy shared -> global (TMA engine, no tensor map: the tile is a flat byte range) ----
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_store_s2g(void* gdst, const void* ssrc, uint32_t bytes, uint64_t pol) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(gdst),
               "r"((uint32_t)__cvta_generic_to_shared(ssrc)), "r"(bytes), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the source bytes of every committed bulk store have been read: the tile may be modified again
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... of all but the N most recently committed groups (a ring of N + 1 tiles)
template <int N>
__device__ __forceinline__ void bulk_wait_read_pending() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// make this thread's generic-proxy shared-memory writes visible to the async proxy (the TMA engine)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

}  // namespace
