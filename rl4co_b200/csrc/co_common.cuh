// Shared helpers for libcorollout (sm_100a). See include/corollout.h for the ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "corollout.h"

namespace co {

constexpr int E = CO_EMBED_DIM;   // 128
constexpr int H = CO_NUM_HEADS;   // 8
constexpr int D = E / H;          // 16
constexpr unsigned FULL = 0xffffffffu;

extern thread_local char g_err[512];

inline int fail(int code, const char* fmt, const char* a = "", long long x = 0, long long y = 0) {
  snprintf(g_err, sizeof(g_err), fmt, a, x, y);
  return code;
}

inline int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return CO_ERR_CUDA;
  }
  return CO_OK;
}

struct DeviceInfo {
  int sm_count;
  int max_smem_optin;
};
const DeviceInfo& device_info();

// Function attributes (opt-in dynamic shared memory) are per device: remember them per device id so a
// process that drives several GPUs configures each of them once.
struct PerDeviceOnce {
  bool done[64] = {};
  bool& flag() {
    int dev = 0;
    cudaGetDevice(&dev);
    return done[dev & 63];
  }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL, v, o));
  return v;
}
// argmax with "first index wins on ties" (torch.argmax semantics)
__device__ __forceinline__ void warp_argmax(float& v, int& idx) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float ov = __shfl_xor_sync(FULL, v, o);
    int oi = __shfl_xor_sync(FULL, idx, o);
    if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
  }
}

// Euclidean distance as sqrt(fma(dy, dy, dx * dx)): what torch's CPU reduction produces for the 2-norm of a
// two-element difference (torch.norm, rl4co/utils/ops.py:93-100), so recorded reference distances are met bit for
// bit.  Symmetric exactly: dist2(a, b) == dist2(b, a).
__device__ __forceinline__ float dist2(float2 a, float2 b) {
  const float dx = a.x - b.x, dy = a.y - b.y;
  return sqrtf(fmaf(dy, dy, dx * dx));
}

// Philox4x32-10 (Salmon et al. 2011), used for CO_SELECT_SAMPLE_PHILOX.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0; key.y += W1;
  }
  return ctr;
}
// Exp(1) draw for (trajectory, decode step, node): q = -log(u), u in (0,1)
__device__ __forceinline__ float philox_exp1(uint64_t seed, uint64_t offset, uint32_t traj, uint32_t step, uint32_t node) {
  uint4 c = make_uint4(traj, step, node, (uint32_t)offset);
  uint2 k = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ (uint32_t)(offset >> 32));
  uint4 r = philox4x32_10(c, k);
  // 23 random bits + 0.5: every value is exactly representable in fp32, so u in [2^-24, 1 - 2^-24]
  // and q = -log(u) is finite and > 0 (with 24 bits, 16777215.5 would round up to 2^24 -> u = 1 -> q = 0)
  float u = ((float)(r.x >> 9) + 0.5f) * (1.0f / 8388608.0f);
  return -logf(u);
}

}  // namespace co
