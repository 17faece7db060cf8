// 2-opt local search for TSP tours: rl4co/envs/routing/tsp/local_search.py (local_search :16-44, two_opt_once :47-70,
// _two_opt_python :73-81), reproduced bit for bit.
//
// One CTA owns one instance at a time (persistent grid striding over the batch).  Shared memory holds the tour, the
// coordinates in tour order and the length of every tour edge: 16 B per node, no N x N distance matrix.  A scan is the
// reference's double loop over positions i = 1..N-2, j = i+1..N-1; each thread walks a contiguous run of those pairs in
// loop order, so the coordinates and node of position j+1 carry over to the next pair.  Per pair:
//     change = ((D[prev, j] + D[i, next]) - D[prev, i]) - D[j, next]        (fp32, the reference's order)
// with the two new distances from coordinates (co::dist2 == the reference's get_distance_matrix entry) and the two old
// ones from the edge array (bit-identical: the distance is exactly symmetric).  The reference keeps the first pair in
// loop order with the strictly smallest change < 0; here every thread keeps its own first minimum and the block takes
// the minimum of the 64-bit keys (order-preserving bits of change, then i * N + j), which gives the same pair whatever
// the thread mapping.  The move is applied only if delta < -1e-6 in double, as a cooperative reversal of positions
// p..q followed by a recompute of edges p-1..q.  The loop ends after a scan that applies no move or after
// max_iterations scans.
//
// The reference adds 1e9 to the diagonal of D.  For a permutation no diagonal entry is ever read; for a tour that
// repeats a node, the skip rule keeps the new distances off the diagonal and tour_edge() returns 1e9 for an edge
// between equal nodes, so such rows follow the reference too.  A row with a node index outside [0, N) is copied
// unchanged and reports -1 moves.
#include "co_common.cuh"

namespace co {

constexpr int TWO_OPT_MAX_THREADS = 512;
constexpr float TWO_OPT_DIAGONAL = 1e9f;  // local_search.py:38: distances + 1e9 * eye
constexpr unsigned long long NO_MOVE = ~0ull;

// edge k joins positions k and k+1 (mod n): D[tour[k], tour[k+1]]
__device__ __forceinline__ float tour_edge(const float2* pos, const int* node, int k, int n) {
  const int k1 = (k + 1 == n) ? 0 : k + 1;
  return node[k] == node[k1] ? TWO_OPT_DIAGONAL : dist2(pos[k], pos[k1]);
}

// change < 0 only: the complemented bits of a negative float ascend with the value
__device__ __forceinline__ unsigned long long move_key(float change, int flat) {
  return ((unsigned long long)(~__float_as_uint(change)) << 32) | (unsigned)flat;
}

__global__ void __launch_bounds__(TWO_OPT_MAX_THREADS) two_opt_kernel(const float2* __restrict__ locs,
                                                                      const int64_t* tours_in, int64_t* tours_out,
                                                                      int32_t* moves_out, int B, int N,
                                                                      int max_iterations) {
  extern __shared__ __align__(16) unsigned char smem[];
  float2* pos = reinterpret_cast<float2*>(smem);   // [N] coordinates of the node at each tour position
  float* edge = reinterpret_cast<float*>(pos + N);  // [N] edge lengths
  int* node = reinterpret_cast<int*>(edge + N);     // [N] the tour
  __shared__ unsigned long long best_key[2];        // alternating per scan, so one barrier per scan resets it

  const int tid = threadIdx.x, T = blockDim.x;
  // this thread's share of the P = (N-1)(N-2)/2 pairs: flat indices [first, first + count) in loop order; row i holds
  // N-1-i pairs.  The split depends on N only, so it is found once.
  const long long P = N >= 3 ? (long long)(N - 1) * (N - 2) / 2 : 0;
  const long long chunk = (P + T - 1) / T;
  const long long first = min(P, (long long)tid * chunk);
  const long long count = min(P, first + chunk) - first;
  int i0 = 1;
  long long rem = first;
  while (count > 0 && rem >= N - 1 - i0) rem -= N - 1 - i0++;
  const int j0 = i0 + 1 + (int)rem;

  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const int64_t* tin = tours_in + (size_t)b * N;
    int64_t* tout = tours_out + (size_t)b * N;
    __syncthreads();  // the previous instance is fully written out
    int bad = 0;
    for (int k = tid; k < N; k += T) {
      const int64_t v = tin[k];
      bad |= (v < 0 || v >= N);
      node[k] = (int)v;
    }
    if (__syncthreads_or(bad)) {
      for (int k = tid; k < N; k += T) tout[k] = tin[k];
      if (moves_out && tid == 0) moves_out[b] = -1;
      continue;
    }
    const float2* lb = locs + (size_t)b * N;
    for (int k = tid; k < N; k += T) pos[k] = lb[node[k]];
    if (tid == 0) best_key[0] = best_key[1] = NO_MOVE;
    __syncthreads();
    for (int k = tid; k < N; k += T) edge[k] = tour_edge(pos, node, k, N);
    __syncthreads();

    int moves = 0;
    for (int it = 0; it < max_iterations; ++it) {
      float best = 0.f;  // two_opt_once :51 starts from delta = 0: only improving pairs count
      int best_flat = 0;
      if (count > 0) {
        int i = i0, j = j0;
        float2 p_prev = pos[i - 1], p_i = pos[i], p_j = pos[j];
        int n_prev = node[i - 1], n_i = node[i], n_j = node[j];
        float e_prev = edge[i - 1];
        for (long long s = 0; s < count; ++s) {
          const int jn = (j + 1 == N) ? 0 : j + 1;
          const float2 p_next = pos[jn];
          const int n_next = node[jn];
          if (n_prev != n_j && n_next != n_i) {  // :56-57
            const float change = ((dist2(p_prev, p_j) + dist2(p_i, p_next)) - e_prev) - edge[j];
            if (change < best) {
              best = change;
              best_flat = i * N + j;
            }
          }
          if (jn != 0) {
            j = jn;
            p_j = p_next;
            n_j = n_next;
          } else if (s + 1 < count) {  // end of row i: the next pair is (i+1, i+2)
            ++i;
            j = i + 1;
            p_prev = pos[i - 1];
            p_i = pos[i];
            p_j = pos[j];
            n_prev = node[i - 1];
            n_i = node[i];
            n_j = node[j];
            e_prev = edge[i - 1];
          }
        }
      }
      unsigned long long key = best < 0.f ? move_key(best, best_flat) : NO_MOVE;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) key = min(key, __shfl_xor_sync(FULL, key, o));
      if ((tid & 31) == 0 && key != NO_MOVE) atomicMin(&best_key[it & 1], key);
      __syncthreads();
      key = best_key[it & 1];
      if (tid == 0) best_key[(it + 1) & 1] = NO_MOVE;
      if (key == NO_MOVE) break;
      const float delta = __uint_as_float(~(unsigned)(key >> 32));
      if (!((double)delta < -1e-6)) break;  // :66, then _two_opt_python's loop test :78
      const int flat = (int)(key & 0xffffffffu), p = flat / N, q = flat - p * N;
      for (int k = tid; k < (q - p + 1) / 2; k += T) {  // tour[p:q+1] = flip(tour[p:q+1])
        const float2 pa = pos[p + k];
        const int na = node[p + k];
        pos[p + k] = pos[q - k];
        node[p + k] = node[q - k];
        pos[q - k] = pa;
        node[q - k] = na;
      }
      __syncthreads();
      for (int k = p - 1 + tid; k <= q; k += T) edge[k] = tour_edge(pos, node, k, N);
      __syncthreads();
      ++moves;
    }
    for (int k = tid; k < N; k += T) tout[k] = node[k];
    if (moves_out && tid == 0) moves_out[b] = moves;
  }
}

// threads per instance: about one per node, so small instances pack many CTAs onto an SM
int two_opt_threads(int N) { return N <= 32 ? 32 : N <= 64 ? 64 : N <= 128 ? 128 : N <= 256 ? 256 : TWO_OPT_MAX_THREADS; }

}  // namespace co

using namespace co;

extern "C" int co_tsp_two_opt(const float* locs, const int64_t* tours_in, int64_t* tours_out, int32_t* moves_out, int B,
                              int N, int max_iterations, void* stream) {
  if (!locs || !tours_in || !tours_out) return fail(CO_ERR_BAD_ARG, "co_tsp_two_opt: null pointer%s");
  if (B < 0 || N < 0 || max_iterations < 0)
    return fail(CO_ERR_BAD_ARG, "co_tsp_two_opt: negative argument%s B=%lld N=%lld", "", B, N);
  if (N > CO_TWO_OPT_MAX_NODES)
    return fail(CO_ERR_UNSUPPORTED, "co_tsp_two_opt: N=%s%lld above CO_TWO_OPT_MAX_NODES=%lld", "", N,
                CO_TWO_OPT_MAX_NODES);
  if (B == 0) return CO_OK;
  const int threads = two_opt_threads(N);
  const size_t smem = (size_t)N * (sizeof(float2) + sizeof(float) + sizeof(int));
  int per_sm = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, two_opt_kernel, threads, smem);
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "co_tsp_two_opt: %s", cudaGetErrorString(e));
    return CO_ERR_CUDA;
  }
  const long long slots = (long long)device_info().sm_count * (per_sm > 0 ? per_sm : 1);
  const int grid = (int)(slots < B ? slots : B);
  two_opt_kernel<<<grid, threads, smem, (cudaStream_t)stream>>>(reinterpret_cast<const float2*>(locs), tours_in,
                                                                tours_out, moves_out, B, N, max_iterations);
  return check_launch("co_tsp_two_opt");
}
