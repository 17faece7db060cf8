// Orienteering problem (sibling env, SURVEY.md 8f-4): step / action mask / reward of rl4co.envs.OPEnv as one kernel each.
//   co_op_step        <- rl4co/envs/routing/op/env.py:72-105 (_step incl. the trailing get_action_mask)
//   co_op_action_mask <- op/env.py:140-155
//   co_op_reward      <- op/env.py:157-165 (sum of the collected prizes)
// One warp per instance row.  Distances are co::dist2 (co_common.cuh), so the recorded tour lengths and masks are
// reproduced bit for bit.
#include "co_common.cuh"

namespace co {

constexpr int OP_ROWS_PER_CTA = 8;

// get_action_mask: visited | depot re-entered | tour_length + dist(cur, n) > max_length[n]; the depot is always feasible
__device__ __forceinline__ void op_mask_row(const float2* __restrict__ locs, const float* __restrict__ max_length,
                                            const uint8_t* visited, float tour_length, int cur, uint8_t* mask_out, int N,
                                            int lane) {
  const float2 pc = locs[cur];
  const bool depot_seen = visited[0] != 0;
  for (int n = lane; n < N; n += 32) {
    const bool exceeds = (tour_length + dist2(locs[n], pc)) > max_length[n];
    const bool masked = (visited[n] != 0) || depot_seen || exceeds;
    mask_out[n] = (n == 0 || !masked) ? 1 : 0;
  }
}

__global__ void __launch_bounds__(256) op_mask_kernel(const float2* __restrict__ locs, const float* __restrict__ max_length,
                                                      const uint8_t* __restrict__ visited,
                                                      const float* __restrict__ tour_length,
                                                      const int64_t* __restrict__ current_node, uint8_t* mask_out, int B,
                                                      int N) {
  const int row = blockIdx.x * OP_ROWS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= B) return;
  op_mask_row(locs + (size_t)row * N, max_length + (size_t)row * N, visited + (size_t)row * N, tour_length[row],
              (int)current_node[row], mask_out + (size_t)row * N, N, lane);
}

__global__ void __launch_bounds__(256) op_step_kernel(const int64_t* __restrict__ action, const float2* __restrict__ locs,
                                                      const float* __restrict__ prize, const float* __restrict__ max_length,
                                                      const uint8_t* visited_in, uint8_t* visited_out, float* tour_length,
                                                      float* total_prize, int64_t* current_node, int64_t* i, uint8_t* done,
                                                      uint8_t* mask_out, int B, int N) {
  const int row = blockIdx.x * OP_ROWS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= B) return;
  const int a = (int)action[row], prev = (int)current_node[row];
  const float2* lr = locs + (size_t)row * N;
  const float tl = tour_length[row] + dist2(lr[a], lr[prev]);  // op/env.py:75-77
  const uint8_t* vin = visited_in + (size_t)row * N;
  uint8_t* vout = visited_out + (size_t)row * N;
  for (int n = lane; n < N; n += 32) vout[n] = (n == a) ? 1 : vin[n];  // visited.scatter(-1, action, 1)
  __syncwarp();
  op_mask_row(lr, max_length + (size_t)row * N, vout, tl, a, mask_out + (size_t)row * N, N, lane);
  if (lane == 0) {
    const int64_t iv = i[row];
    tour_length[row] = tl;
    total_prize[row] += prize[(size_t)row * N + a];
    done[row] = (a == 0) && (iv > 0);  // back at the depot after the first step
    current_node[row] = a;
    i[row] = iv + 1;
  }
}

__global__ void __launch_bounds__(256) op_reward_kernel(const float* __restrict__ prize, const int64_t* __restrict__ actions,
                                                        float* reward, int B, int N, int T) {
  const int row = blockIdx.x * OP_ROWS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= B) return;
  float s = 0.f;
  for (int t = lane; t < T; t += 32) {
    const int a = (int)actions[(size_t)row * T + t];
    s += (a >= 0 && a < N) ? prize[(size_t)row * N + a] : 0.f;
  }
  s = warp_sum(s);
  if (lane == 0) reward[row] = s;
}

}  // namespace co

using namespace co;

extern "C" int co_op_action_mask(const float* locs, const float* max_length, const uint8_t* visited, const float* tour_length,
                                 const int64_t* current_node, uint8_t* mask_out, int B, int N, void* stream) {
  if (!locs || !max_length || !visited || !tour_length || !current_node || !mask_out)
    return fail(CO_ERR_BAD_ARG, "co_op_action_mask: null pointer%s");
  if (B < 0 || N < 2) return fail(CO_ERR_BAD_ARG, "co_op_action_mask: bad shape%s B=%lld N=%lld", "", B, N);
  if (B == 0) return CO_OK;
  op_mask_kernel<<<(B + OP_ROWS_PER_CTA - 1) / OP_ROWS_PER_CTA, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float2*>(locs), max_length, visited, tour_length, current_node, mask_out, B, N);
  return check_launch("co_op_action_mask");
}

extern "C" int co_op_step(const int64_t* action, const float* locs, const float* prize, const float* max_length,
                          const uint8_t* visited_in, uint8_t* visited_out, float* tour_length, float* current_total_prize,
                          int64_t* current_node, int64_t* i, uint8_t* done, uint8_t* mask_out, int B, int N, void* stream) {
  if (!action || !locs || !prize || !max_length || !visited_in || !visited_out || !tour_length || !current_total_prize ||
      !current_node || !i || !done || !mask_out)
    return fail(CO_ERR_BAD_ARG, "co_op_step: null pointer%s");
  if (B < 0 || N < 2) return fail(CO_ERR_BAD_ARG, "co_op_step: bad shape%s B=%lld N=%lld", "", B, N);
  if (B == 0) return CO_OK;
  op_step_kernel<<<(B + OP_ROWS_PER_CTA - 1) / OP_ROWS_PER_CTA, 256, 0, (cudaStream_t)stream>>>(
      action, reinterpret_cast<const float2*>(locs), prize, max_length, visited_in, visited_out, tour_length,
      current_total_prize, current_node, i, done, mask_out, B, N);
  return check_launch("co_op_step");
}

extern "C" int co_op_reward(const float* prize, const int64_t* actions, float* reward, int B, int N, int T, void* stream) {
  if (!prize || !actions || !reward) return fail(CO_ERR_BAD_ARG, "co_op_reward: null pointer%s");
  if (B < 0 || N < 1 || T < 1) return fail(CO_ERR_BAD_ARG, "co_op_reward: bad shape%s");
  if (B == 0) return CO_OK;
  op_reward_kernel<<<(B + OP_ROWS_PER_CTA - 1) / OP_ROWS_PER_CTA, 256, 0, (cudaStream_t)stream>>>(prize, actions, reward, B, N, T);
  return check_launch("co_op_reward");
}

// ---------------------------------------------------------------------------------------------------------------------
// Prize-collecting TSP (third sibling env): rl4co/envs/routing/pctsp/env.py
//   co_pctsp_step        <- _step :62-93 + get_action_mask :143-151
//   co_pctsp_action_mask <- get_action_mask: customers masked once visited or once the depot was re-entered; the depot is
//                           infeasible while the collected prize is below 1.0 and unvisited customers remain
// (reward = co_op_reward over the penalties + co_tour_length, see FusedPCTSPEnv._get_reward)
namespace co {

__device__ __forceinline__ void pctsp_mask_row(const uint8_t* visited, float prize, uint8_t* mask_out, int N, int lane) {
  const bool depot_seen = visited[0] != 0;
  int unvisited = 0;
  for (int n = 1 + lane; n < N; n += 32) {
    const bool v = visited[n] != 0;
    mask_out[n] = (v || depot_seen) ? 0 : 1;
    unvisited += v ? 0 : 1;
  }
  unvisited = __reduce_add_sync(FULL, unvisited);
  if (lane == 0) mask_out[0] = ((prize < 1.0f) && (unvisited > 0)) ? 0 : 1;
}

__global__ void __launch_bounds__(256) pctsp_mask_kernel(const uint8_t* __restrict__ visited, const float* __restrict__ prize,
                                                         uint8_t* mask_out, int B, int N) {
  const int row = blockIdx.x * OP_ROWS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= B) return;
  pctsp_mask_row(visited + (size_t)row * N, prize[row], mask_out + (size_t)row * N, N, lane);
}

__global__ void __launch_bounds__(256) pctsp_step_kernel(const int64_t* __restrict__ action, const float* __restrict__ real_prize,
                                                         const float* __restrict__ penalty, const uint8_t* visited_in,
                                                         uint8_t* visited_out, float* total_prize, float* total_penalty,
                                                         int64_t* current_node, int64_t* i, uint8_t* done, uint8_t* mask_out,
                                                         int B, int N) {
  const int row = blockIdx.x * OP_ROWS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= B) return;
  const int a = (int)action[row];
  const float p = total_prize[row] + real_prize[(size_t)row * N + a];
  const uint8_t* vin = visited_in + (size_t)row * N;
  uint8_t* vout = visited_out + (size_t)row * N;
  for (int n = lane; n < N; n += 32) vout[n] = (n == a) ? 1 : vin[n];
  __syncwarp();
  pctsp_mask_row(vout, p, mask_out + (size_t)row * N, N, lane);
  if (lane == 0) {
    const int64_t iv = i[row];
    total_prize[row] = p;
    total_penalty[row] += penalty[(size_t)row * N + a];
    done[row] = (iv > 0) && (a == 0);
    current_node[row] = a;
    i[row] = iv + 1;
  }
}

}  // namespace co

extern "C" int co_pctsp_action_mask(const uint8_t* visited, const float* cur_total_prize, uint8_t* mask_out, int B, int N,
                                    void* stream) {
  if (!visited || !cur_total_prize || !mask_out) return fail(CO_ERR_BAD_ARG, "co_pctsp_action_mask: null pointer%s");
  if (B < 0 || N < 2) return fail(CO_ERR_BAD_ARG, "co_pctsp_action_mask: bad shape%s B=%lld N=%lld", "", B, N);
  if (B == 0) return CO_OK;
  pctsp_mask_kernel<<<(B + OP_ROWS_PER_CTA - 1) / OP_ROWS_PER_CTA, 256, 0, (cudaStream_t)stream>>>(visited, cur_total_prize,
                                                                                                   mask_out, B, N);
  return check_launch("co_pctsp_action_mask");
}

extern "C" int co_pctsp_step(const int64_t* action, const float* real_prize, const float* penalty, const uint8_t* visited_in,
                             uint8_t* visited_out, float* cur_total_prize, float* cur_total_penalty, int64_t* current_node,
                             int64_t* i, uint8_t* done, uint8_t* mask_out, int B, int N, void* stream) {
  if (!action || !real_prize || !penalty || !visited_in || !visited_out || !cur_total_prize || !cur_total_penalty ||
      !current_node || !i || !done || !mask_out)
    return fail(CO_ERR_BAD_ARG, "co_pctsp_step: null pointer%s");
  if (B < 0 || N < 2) return fail(CO_ERR_BAD_ARG, "co_pctsp_step: bad shape%s B=%lld N=%lld", "", B, N);
  if (B == 0) return CO_OK;
  pctsp_step_kernel<<<(B + OP_ROWS_PER_CTA - 1) / OP_ROWS_PER_CTA, 256, 0, (cudaStream_t)stream>>>(
      action, real_prize, penalty, visited_in, visited_out, cur_total_prize, cur_total_penalty, current_node, i, done, mask_out,
      B, N);
  return check_launch("co_pctsp_step");
}
